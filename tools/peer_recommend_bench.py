"""Whole-catalogue top-k on the peer-partitioned graph (peer.recommend_peer) against the single-GPU GraphNCF.recommend.

    python tools/peer_recommend_bench.py [--calls K] [--users N] [--out FILE.json]                 # one GPU: P = 1, config 3 graph
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... tools/peer_recommend_bench.py ...         # P = N
    python -m torch.distributed.run --nnodes=1 --nproc-per-node 8 ... tools/peer_recommend_bench.py --graph5 --users-frac 0.01

Config 3 graph (bench.build_graph: 162,541 users x 62,423 items x 25 M interactions, d = 128, L = 2), models: bench.py's MLP [256, 128]
(K5 on tcgen05) and a dot-product model of the same size (the exact dot kernel).  `--users` sampled users (the same on every rank) are
served; single-GPU and partitioned calls alternate, each timed between device synchronisations, median of `--calls`.  A traced pass splits
a partitioned call into propagation, catalogue push and scoring (%globaltimer markers, peer.TRACE).  Parity as in
tests/test_peer_recommend_gpu.py: value error, the reference score of the returned items, and the share of users with equal index sets.
On one GPU the dot kernel is also timed against GEMM + topk_rows on the same (users x items) slab.

--graph5: BASELINE configs[4] built per rank (bench.g5_shard_edges + sharded.build_shard, d = 64, L = 3, MLP [128] = relu_dot), a
`--users-frac` sample of every rank's users against the full catalogue; time per call, per 10^9 pairs, and the catalogue push.
Rank 0 prints one JSON line with the card's name, power limit and max SM clock read in the same run."""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

import torch
import torch.distributed as dist

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench                                                                                    # noqa: E402
from deeprecommendation_b200 import ops, peer, synth                                            # noqa: E402
from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF                # noqa: E402


def gpu_info(index):
    r = subprocess.run(['nvidia-smi', '-i', str(index), '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [x.strip() for x in r.stdout.strip().splitlines()[0].split(',')]
    return {'name': name, 'power_limit': power, 'max_sm_clock': clock}


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) * 1e3, out


def phases(sh, fn, n=3):
    """median device-side split of a partitioned call (ms)"""
    peer.TRACE = True
    try:
        rows = []
        for _ in range(n):
            fn()
            torch.cuda.synchronize()
            t = dict(sh.trace())
            rows.append((t['layers joined'] - t['start'], t['catalogue arrived'] - t['layers joined'], t['scored'] - t['catalogue arrived']))
    finally:
        peer.TRACE = False
    med = [statistics.median(r[i] for r in rows) / 1e3 for i in range(3)]
    return {'propagation_ms': med[0], 'catalogue_push_ms': med[1], 'scoring_ms': med[2]}


def parity(mine, ref, k, tol=1e-5):
    nodes, val, idx = mine
    rv, ri, rs = ref
    S = rs.double()
    scale = float(S.nan_to_num(0.0).abs().max())
    pad = idx < 0
    e_val = float((val[~pad].double() - rv[~pad].double()).abs().max()) / scale
    e_hit = float((S.gather(1, idx.clamp_min(0))[~pad] - val[~pad].double()).abs().max()) / scale
    same = sum(torch.equal(a.sort().values, b.sort().values) for a, b in zip(idx, ri)) / max(len(idx), 1)
    return {'val_err': e_val, 'hit_err': e_hit, 'share_equal_index_sets': same, 'within_tol': e_val < tol and e_hit < tol}


def config3(args, dev, rank, world):
    from deeprecommendation_b200.parallel import partition_graph
    w = bench.build_graph(dev)
    graph, d, L_ = w['graph'], w['d'], w['L']
    nI, nU = w['nI'], w['nU']
    g = torch.Generator(device=dev).manual_seed(3)
    users = torch.randperm(nU, device=dev, generator=g)[:args.users] + nI
    res = {}
    for name, dot in (('mlp_256_128', False), ('dot', True)):
        kw = dict(w['kw'], use_dot_product=dot)
        model = GraphNCF(**kw).to(dev).eval()
        model.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=2, **kw)))
        pg = partition_graph(graph, scheme='peer', d_max=d, batch_max=bench.BATCH, catalogue_width=peer.catalogue_width(model))
        object.__setattr__(graph, '_b200rec_partition', None)
        with torch.no_grad():
            part = lambda: peer.recommend_peer(model, pg, k=args.k, users=users)
            mine = part()
            single = lambda: model.recommend(graph, args.k, user_nodes=mine[0])
            ts, tp = [], []
            for c in range(args.warmup + args.calls):
                a, _ = timed(single)
                b, mine = timed(part)
                if c >= args.warmup:
                    ts.append(a)
                    tp.append(b)
            pg.check()
            ref = model.recommend(graph, args.k, user_nodes=mine[0], return_scores=True)
            split = phases(pg, part)
        n_pairs = int(mine[0].numel()) * nI
        res[name] = {'users_served': int(mine[0].numel()), 'single_gpu_ms': statistics.median(ts) if world == 1 else None,
                     'peer_ms': statistics.median(tp), 'peer_ms_minmax': [min(tp), max(tp)], 'single_gpu_ms_minmax': [min(ts), max(ts)],
                     'peer_ms_per_1e9_pairs': statistics.median(tp) / n_pairs * 1e9, **split, 'parity': parity(mine, ref, args.k)}
        del pg, model
        dist.barrier()
    if world == 1:                                     # the dot kernel alone vs GEMM + topk_rows on one (users x items) slab
        A = torch.randn(args.users, d, device=dev, generator=g)
        B = torch.randn(nI, d, device=dev, generator=g)
        kern = lambda: ops.allpairs_dot_topk_raw(A, B, args.k)
        gemm = lambda: ops.topk_rows(ops.linear_raw(A, B, None), args.k)
        tk, tg = [], []
        for c in range(args.warmup + args.calls):
            a, outk = timed(kern)
            b, outg = timed(gemm)
            if c >= args.warmup:
                tk.append(a)
                tg.append(b)
        res['dot_kernel_vs_gemm_topk'] = {'users': args.users, 'items': nI, 'd': d, 'dot_kernel_ms': statistics.median(tk),
                                          'gemm_topk_ms': statistics.median(tg), 'value_err': float((outk[0] - outg[0]).abs().max() / outg[0].abs().max()),
                                          'score_matrix_bytes': args.users * nI * 4}
    return {'graph': {'users': nU, 'items': nI, 'interactions': w['E'], 'd': d, 'L': L_}, 'sampled_users': args.users, 'results': res}


def graph5(args, dev, rank, world):
    from deeprecommendation_b200.sharded import build_shard
    V = bench.G5_VSHARDS
    nU, nI, E, d, L_ = bench.G5_USERS, bench.G5_ITEMS, bench.G5_EDGES, bench.G5_D, bench.G5_LAYERS
    nU_v, E_v = nU // V, E // V
    mine = list(range(rank * (V // world), (rank + 1) * (V // world)))
    us, its, rs = [], [], []
    for j, v in enumerate(mine):
        u, i, r = bench.g5_shard_edges(v, nU_v, nI, E_v, dev)
        us.append(u + j * nU_v)
        its.append(i)
        rs.append(r)
    u_local, items, ratings = torch.cat(us), torch.cat(its), torch.cat(rs)
    del us, its, rs
    n_local, users_r0 = nU_v * len(mine), mine[0] * nU_v
    item_features = torch.randn(nI, d, device=dev, generator=torch.Generator(device=dev).manual_seed(77))
    user_features = torch.cat([torch.randn(nU_v, d, device=dev, generator=torch.Generator(device=dev).manual_seed(500 + v)) for v in mine])
    kw = dict(item_dim=d, user_dim=d, num_gnn_layers=L_, hetero=True, node_emb=d, mlp_dense_layers=[128], dropout_rate=0.2)
    model = GraphNCF(**kw).to(dev).eval()
    model.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=2, **kw)))
    sh = build_shard(u_local, items, ratings, nI=nI, nU=nU, users_r0=users_r0, n_local_users=n_local, item_features=item_features,
                     user_features_local=user_features, d_max=d, batch_max=bench.BATCH, edges_total=2 * E, catalogue_width=peer.catalogue_width(model))
    del u_local, items, ratings
    g = torch.Generator(device=dev).manual_seed(9)
    users = torch.nonzero(torch.rand(nU, device=dev, generator=g) < args.users_frac).view(-1) + nI     # the same sample on every rank
    with torch.no_grad():
        part = lambda: peer.recommend_peer(model, sh, k=args.k, users=users)
        t, out = [], None
        for c in range(1 + args.calls):
            ms, out = timed(part)
            if c >= 1:
                t.append(ms)
        sh.check()
        split = phases(sh, part, n=1)
    pairs = int(out[0].numel()) * nI
    return {'graph': {'users': nU, 'items': nI, 'interactions': E, 'd': d, 'L': L_, 'mlp': [128]}, 'users_frac': args.users_frac,
            'results': {'users_served': int(out[0].numel()), 'call_ms': statistics.median(t), 'call_ms_minmax': [min(t), max(t)],
                        'ms_per_1e9_pairs': statistics.median(t) / pairs * 1e9, **split}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--calls', type=int, default=7)
    ap.add_argument('--warmup', type=int, default=2)
    ap.add_argument('--users', type=int, default=16384)
    ap.add_argument('--k', type=int, default=10)
    ap.add_argument('--graph5', action='store_true')
    ap.add_argument('--users-frac', type=float, default=0.01)
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
    rec = graph5(args, dev, rank, world) if args.graph5 else config3(args, dev, rank, world)
    per_rank = [None] * world
    dist.all_gather_object(per_rank, {'gpu': info, 'results': rec['results']})
    if rank == 0:
        out = {'tool': 'tools/peer_recommend_bench.py', 'world': world, 'calls': args.calls, 'k': args.k, 'gpu': info, **rec,
               'per_rank': [r['results'] for r in per_rank], 'gpus': [r['gpu'] for r in per_rank]}
        print(json.dumps(out), flush=True)
        if args.out:
            os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
            with open(args.out, 'w') as f:
                json.dump(out, f, indent=1)
    dist.destroy_process_group()


if __name__ == '__main__':
    main()
