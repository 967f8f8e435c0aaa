"""Partitioned GraphNCF forward (scheme 'peer') with LightGAT and with the concat combine, against the single-GPU forward, on the config 3
graph (bench.build_graph: 162,541 users x 62,423 items x 25 M interactions, d = 128, L = 2, a batch of 512 pairs).

    python tools/peer_gat_bench.py [--steps K] [--warmup W] [--out FILE.json]                                   # one GPU: P = 1
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P tools/peer_gat_bench.py ...

Models: LightGCN with mean combine (the existing exchange, for reference), LightGAT with mean combine, LightGCN with concat combine.  Each
forward is captured once as a CUDA graph and replayed; a step is one replay timed with CUDA events, and the single-GPU and partitioned
replays alternate step by step.  Reported per model: the median step of each, their ratio, and the max-norm relative difference of the
partitioned scores against the single-GPU ones.  Rank 0 prints one JSON line with the card's name and power limit read in the same run."""
import argparse
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
from deeprecommendation_b200.graphed import GraphedForward                                      # noqa: E402
from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF                # noqa: E402
from deeprecommendation_b200.parallel import partition_graph                                    # noqa: E402

MODELS = (('LightGCN', False), ('LightGAT', False), ('LightGCN', True))


def gpu_info(index):
    r = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(',')]
    return {'name': name, 'power_limit': power, 'max_sm_clock': clock}


def step_ms(fn, *args):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn(*args)
    b.record()
    b.synchronize()
    return a.elapsed_time(b), out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--steps', type=int, default=50)
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
        dist.init_process_group('gloo', init_method='tcp://127.0.0.1:29731', rank=0, world_size=1)       # P = 1: one real rank
    rank, world = dist.get_rank(), dist.get_world_size()
    info = gpu_info(local)
    w = bench.build_graph(dev)
    graph, E, L_, d = w['graph'], w['E'], w['L'], w['d']
    u2i = graph.user2item_edge_index
    pick = w['pick'][0]
    uid, iid = u2i[0][pick].contiguous(), u2i[1][pick].contiguous()
    pg = partition_graph(graph, scheme='peer', d_max=d, batch_max=bench.BATCH * (L_ + 1))      # rows buffer: 512 pairs of (L + 1)·d floats
    res = {}
    for conv, concat in MODELS:
        kw = dict(w['kw'], convType=conv, concat=concat)
        model = GraphNCF(**kw).to(dev).eval()
        model.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=2, **kw)))
        fn = lambda a, b: model(graph, a, b, dev)
        object.__setattr__(graph, '_b200rec_partition', None)                # single-GPU forward over the whole graph
        single = GraphedForward(fn, uid, iid)
        object.__setattr__(graph, '_b200rec_partition', pg)
        peer = GraphedForward(fn, uid, iid)
        t_single, t_peer = [], []
        for k in range(args.warmup + args.steps):
            ts, out_single = step_ms(single, uid, iid)
            tp, out_peer = step_ms(peer, uid, iid)
            if k >= args.warmup:
                t_single.append(ts)
                t_peer.append(tp)
        pg.check()
        err = float((out_peer - out_single).abs().max() / out_single.abs().max())
        name = f'{conv}_{"concat" if concat else "mean"}'
        res[name] = {'single_gpu_ms': statistics.median(t_single), 'peer_ms': statistics.median(t_peer),
                     'peer_over_single': statistics.median(t_peer) / statistics.median(t_single), 'rel_err_vs_single_gpu': err,
                     'single_gpu_ms_minmax': [min(t_single), max(t_single)], 'peer_ms_minmax': [min(t_peer), max(t_peer)]}
        del single, peer, model
        dist.barrier()
    per_rank = [None] * world
    dist.all_gather_object(per_rank, {'gpu': info, 'results': res})
    if rank == 0:
        rec = {'tool': 'tools/peer_gat_bench.py', 'world': world, 'graph': {'users': w['nU'], 'items': w['nI'], 'interactions': E, 'd': d, 'L': L_},
               'batch': bench.BATCH, 'steps': args.steps, 'warmup': args.warmup, 'gpu': info, 'results': res,
               'peer_ms_per_rank': {k: [r['results'][k]['peer_ms'] for r in per_rank] for k in res},
               'gpus': [r['gpu'] for r in per_rank]}
        print(json.dumps(rec), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, 'w') as f:
                json.dump(rec, f, indent=1)
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
