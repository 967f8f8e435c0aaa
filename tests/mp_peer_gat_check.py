"""Multi-process check of scheme 'peer' with LightGAT and the concat combine (run under torchrun; not collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29512 tests/mp_peer_gat_check.py

Every rank builds the same graph, maps the peers' arenas (CUDA IPC), runs the partitioned GraphNCF forward of a LightGAT / concat model —
eagerly and replayed from a captured CUDA graph — and compares with the single-GPU forward computed locally.  With B200REC_PEER_CHECK_SAME_GPU=1 all
ranks use cuda:0 and rendezvous over gloo (the single-GPU test-suite runs it that way); otherwise one GPU per rank over NCCL.
Rank 0 prints one JSON line."""
import json
import os
import sys

import numpy as np
import torch
import torch.distributed as dist

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))


def main():
    from deeprecommendation_b200 import synth
    from deeprecommendation_b200.graph import IdTable, create_graph
    from deeprecommendation_b200.graphed import GraphedForward
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.parallel import partition_graph
    same = os.environ.get('B200REC_PEER_CHECK_SAME_GPU') == '1'
    local = 0 if same else int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if same:
        dist.init_process_group('gloo')
    else:
        dist.init_process_group('nccl', device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    small = same or os.environ.get('B200REC_PEER_CHECK_SMALL') == '1'
    n_users, n_items, n, F, d = (3000, 1200, 100_000, 48, 64) if small else (20000, 8000, 1_500_000, 64, 128)
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=21)
    rng = np.random.default_rng(4)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    info, err = {}, 0.0
    for conv, concat, L_, msg in (('LightGAT', False, 2, 'fp32'), ('LightGAT', True, 2, 'fp32'), ('LightGCN', True, 3, 'fp32'),
                                  ('LightGAT', False, 2, 'bf16')):
        kw = dict(item_dim=F, user_dim=F, num_gnn_layers=L_, hetero=True, node_emb=d, mlp_dense_layers=[256, 128], dropout_rate=0.2,
                  convType=conv, concat=concat)
        sd = synth.to_torch(synth.graph_ncf_weights(seed=5, **kw))
        g = create_graph(torch.from_numpy(users).to(dev), torch.from_numpy(items).to(dev), torch.from_numpy(ratings).to(dev),
                         torch.from_numpy(fi).to(dev), torch.from_numpy(fu).to(dev),
                         IdTable(torch.arange(n_users, device=dev)), IdTable(torch.arange(n_items, device=dev)))
        m = GraphNCF(**kw).to(dev).eval()
        m.load_state_dict(sd)
        pick = rng.permutation(n)[:1000]
        uid, iid = g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()
        with torch.no_grad():
            ref = m(g, uid, iid, dev)
            m.message_dtype = msg
            pg = partition_graph(g, scheme='peer', d_max=d, batch_max=4096)       # room for 1000 rows of (L + 1)·d floats
            outs = [m(g, uid, iid, dev) for _ in range(3)]                    # eager, three epochs of the flags
            torch.cuda.synchronize()
            pg.check()
            e = max(float((o - ref).abs().max() / ref.abs().max()) for o in outs)
            if not same:                                                     # replayed from a captured CUDA graph (bench.py's mode)
                gf = GraphedForward(lambda a, b: m(g, a, b, dev), uid, iid)
                for _ in range(3):
                    og = gf(uid, iid)
                torch.cuda.synchronize()
                pg.check()
                e = max(e, float((og - ref).abs().max() / ref.abs().max()))
            m.message_dtype = 'fp32'
        tol = 1e-2 if msg == 'bf16' else 1e-5
        info[f'{conv}{"_concat" if concat else ""}_L{L_}_{msg}'] = e
        err = max(err, e / tol)
        dist.barrier()
        del pg, g
    errs = [None] * world
    dist.all_gather_object(errs, (err, info))
    if rank == 0:
        print(json.dumps({'world': world, 'same_gpu': same, 'worst_err_over_tol_per_rank': [e[0] for e in errs], 'rel_err': errs[0][1],
                          'ok': all(e[0] < 1.0 for e in errs)}), flush=True)
    dist.destroy_process_group()
    if err >= 1.0:
        sys.exit(1)


if __name__ == '__main__':
    main()
