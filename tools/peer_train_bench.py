"""One GraphNCF training step on the peer-partitioned graph (forward_peer with grad + a collective backward) against the single-GPU eager
step, on the config 3 graph (bench.build_graph: 162,541 users x 62,423 items x 25 M interactions; GraphNCF(L = 2, d = 128, hetero,
mlp = [256, 128]); a batch of 512 pairs; sum-MSE and Adam(fused=True)).

    python tools/peer_train_bench.py [--steps K] [--warmup W] [--out FILE.json]                                 # one GPU: P = 1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/peer_train_bench.py ...

Dropout is off (dropout_rate = 0), so that the two paths compute the same step: before the timed steps, both compute the gradient of the
same loss at the same parameters and the max-norm relative difference over all parameters is reported.  Then the single-GPU and the
partitioned steps alternate (each on its own copy of the model and its own optimizer), each timed with CUDA events from zero_grad to the end
of optimizer.step().  Reported: the median of each over the timed steps, their ratio, min / max.  Rank 0 prints one JSON line with the
card's name and power limit read in the same run."""
import argparse
import copy
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                                                    # noqa: E402
from deeprecommendation_b200 import synth                                                       # noqa: E402
from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF                # noqa: E402
from deeprecommendation_b200.parallel import partition_graph                                    # noqa: E402
from deeprecommendation_b200.peer import forward_peer, grad_floats                              # noqa: E402


def gpu_info(index):
    r = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(',')]
    return {'name': name, 'power_limit': power, 'max_sm_clock': clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--out', default=None)
    args = ap.parse_args()
    multi = 'WORLD_SIZE' in os.environ
    local = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if multi:
        dist.init_process_group('nccl', device_id=dev)
    else:
        dist.init_process_group('gloo', init_method='tcp://127.0.0.1:29733', rank=0, world_size=1)       # P = 1: one real rank
    rank, world = dist.get_rank(), dist.get_world_size()
    info = gpu_info(local)
    w = bench.build_graph(dev)
    graph, E, L_, d = w['graph'], w['E'], w['L'], w['d']
    kw = dict(w['kw'], dropout_rate=0.0)
    single = GraphNCF(**kw).to(dev).train()
    single.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=2, **kw)))
    peer = copy.deepcopy(single)
    pg = partition_graph(graph, scheme='peer', d_max=d, batch_max=bench.BATCH, grad_floats=grad_floats(peer))
    u2i = graph.user2item_edge_index
    batches = [(u2i[0][w['pick'][k]].contiguous(), u2i[1][w['pick'][k]].contiguous()) for k in range(w['pick'].shape[0])]
    gen = torch.Generator(device=dev).manual_seed(11)
    ys = [torch.randn((bench.BATCH, 1), device=dev, generator=gen) for _ in batches]

    def run(model, fwd, k):
        uid, iid = batches[k % len(batches)]
        model.zero_grad(set_to_none=True)
        ((fwd(model, uid, iid) - ys[k % len(ys)]) ** 2).sum().backward()

    fwd_single = lambda m, a, b: m(graph, a, b)            # training mode: GraphNCF.forward takes the single-GPU path
    fwd_peer = lambda m, a, b: forward_peer(m, pg, a, b)
    run(single, fwd_single, 0)
    run(peer, fwd_peer, 0)
    ps = dict(single.named_parameters())
    grad_err = {n: float((p.grad - ps[n].grad).abs().max() / ps[n].grad.abs().max()) for n, p in peer.named_parameters()}
    opts = {id(m): torch.optim.Adam(m.parameters(), lr=1e-3, fused=True) for m in (single, peer)}

    def step(model, fwd, k):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        run(model, fwd, k)
        opts[id(model)].step()
        b.record()
        b.synchronize()
        return a.elapsed_time(b)

    t_single, t_peer = [], []
    for k in range(args.warmup + args.steps):
        ts, tp = step(single, fwd_single, k), step(peer, fwd_peer, k)
        if k >= args.warmup:
            t_single.append(ts)
            t_peer.append(tp)
    pg.check()
    res = {'single_gpu_step_ms': statistics.median(t_single), 'peer_step_ms': statistics.median(t_peer),
           'peer_over_single': statistics.median(t_peer) / statistics.median(t_single),
           'single_gpu_ms_minmax': [min(t_single), max(t_single)], 'peer_ms_minmax': [min(t_peer), max(t_peer)],
           'max_grad_rel_err_vs_single_gpu': max(grad_err.values()), 'grad_rel_err': grad_err}
    per_rank = [None] * world
    dist.all_gather_object(per_rank, {'gpu': info, 'results': res})
    if rank == 0:
        rec = {'tool': 'tools/peer_train_bench.py', 'world': world, 'graph': {'users': w['nU'], 'items': w['nI'], 'interactions': E, 'd': d, 'L': L_},
               'model': kw, 'batch': bench.BATCH, 'steps': args.steps, 'warmup': args.warmup, 'gpu': info, 'results': res,
               'peer_step_ms_per_rank': [r['results']['peer_step_ms'] for r in per_rank], 'gpus': [r['gpu'] for r in per_rank]}
        print(json.dumps(rec), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, 'w') as f:
                json.dump(rec, f, indent=1)
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
