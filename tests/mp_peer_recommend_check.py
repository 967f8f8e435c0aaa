"""Multi-process check of peer.recommend_peer (run under torchrun; not collected by pytest):

    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port 29514 tests/mp_peer_recommend_check.py

Every rank builds the same graph, maps the peers' arenas (CUDA IPC) with a catalogue section, serves its users' whole-catalogue top-k for a
K5 MLP, a one-hidden-layer MLP and a dot-product model (a forward in between, so both kinds of call share the epoch counters) and compares
with the single-GPU GraphNCF.recommend for the same users computed locally.  With B200REC_PEER_CHECK_SAME_GPU=1 all ranks use cuda:0 and
rendezvous over gloo (the single-GPU test-suite runs it that way); otherwise one GPU per rank over NCCL.  Rank 0 prints one JSON line."""
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
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.parallel import partition_graph
    from deeprecommendation_b200.peer import catalogue_width, recommend_peer
    same = os.environ.get('B200REC_PEER_CHECK_SAME_GPU') == '1'
    local = 0 if same else int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if same:
        dist.init_process_group('gloo')
    else:
        dist.init_process_group('nccl', device_id=dev)
    rank, world = dist.get_rank(), dist.get_world_size()
    n_users, n_items, n, F, d = (3000, 1200, 100_000, 48, 64) if same else (20000, 8000, 1_500_000, 64, 128)
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=21)
    rng = np.random.default_rng(4)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    info, ok = {}, True
    for name, mlp, conv, concat in (('k5', [256, 128], 'LightGCN', False), ('relu_dot_gat_concat', [128], 'LightGAT', True),
                                    ('dot', None, 'LightGCN', False)):
        kw = dict(item_dim=F, user_dim=F, num_gnn_layers=2, hetero=True, node_emb=d, mlp_dense_layers=mlp or [8], dropout_rate=0.2,
                  convType=conv, concat=concat, use_dot_product=mlp is None)
        g = create_graph(torch.from_numpy(users).to(dev), torch.from_numpy(items).to(dev), torch.from_numpy(ratings).to(dev),
                         torch.from_numpy(fi).to(dev), torch.from_numpy(fu).to(dev),
                         IdTable(torch.arange(n_users, device=dev)), IdTable(torch.arange(n_items, device=dev)))
        m = GraphNCF(**kw).to(dev).eval()
        m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=5, **kw)))
        pick = rng.permutation(n)[:500]
        uid, iid = g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()
        with torch.no_grad():
            fwd_ref = m(g, uid, iid, dev)
            pg = partition_graph(g, scheme='peer', d_max=d, batch_max=2048, catalogue_width=catalogue_width(m))
            res = [recommend_peer(m, pg, k=10)]
            fwd = m(g, uid, iid, dev)
            res.append(recommend_peer(m, pg, k=10))
            torch.cuda.synchronize()
            pg.check()
            nodes = res[0][0]
            rv, ri, rs = m.recommend(g, 10, user_nodes=nodes, return_scores=True)
        scale = float(rs.nan_to_num(0.0).abs().max())
        e_val = max(float((r[1] - rv).abs().max()) / scale for r in res)
        e_hit = max(float((rs.gather(1, r[2]) - r[1]).abs().max()) / scale for r in res)    # the reference's score of every returned item
        e_fwd = float((fwd - fwd_ref).abs().max() / fwd_ref.abs().max())
        counts = [None] * world
        dist.all_gather_object(counts, int(nodes.numel()))
        info[name] = {'served': counts, 'val_err': e_val, 'hit_err': e_hit, 'forward_err': e_fwd}
        ok = ok and e_val < 1e-5 and e_hit < 1e-5 and e_fwd < 1e-5 and sum(counts) == n_users and torch.equal(res[0][2], res[1][2])
        dist.barrier()
        del pg, g
    oks = [None] * world
    dist.all_gather_object(oks, (ok, info))
    if rank == 0:
        print(json.dumps({'world': world, 'same_gpu': same, 'ok': all(o[0] for o in oks), 'per_rank': [o[1] for o in oks]}), flush=True)
    dist.destroy_process_group()
    if not ok:
        sys.exit(1)


if __name__ == '__main__':
    main()
