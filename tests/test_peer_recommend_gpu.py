"""peer.recommend_peer: whole-catalogue top-k on the peer-partitioned graph (propagation, catalogue broadcast into the `cat` arena section,
K5 / relu_dot / the dot kernel per rank).  Reference = the single-GPU GraphNCF.recommend on the same graph for the users a rank serves.
The partitioned propagation differs from the single-GPU one in the last bits, so the check is (per rank, tolerance `tol` max-norm relative):
values within tol; the reference score of every returned item equals the returned value; the index sets equal wherever the reference's
gap between rank k and k + 1 exceeds 2 tol; the served node lists of all ranks together are the request, each node once."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import synth
from tests._golden import maxnorm_rel

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MLPS = {'k5': (256, 128), 'relu_dot': (128,), 'dot': None}


def _graph(n_users=1500, n_items=900, n=60_000, F=48, d_emb=64, L_=2, mlp=(128,), hetero=True, conv='LightGCN', concat=False, seed=13):
    from deeprecommendation_b200.graph import IdTable, create_graph
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=seed)
    rng = np.random.default_rng(2)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=L_, hetero=hetero, node_emb=d_emb, mlp_dense_layers=list(mlp or (8,)), dropout_rate=0.2,
              use_dot_product=mlp is None, convType=conv, concat=concat)
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV),
                     IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV)))
    m = GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=3, **kw)))
    return m, g


def _check_rank(m, g, res, k, tol, precision='fp32', ignore_seen=True, return_scores=False):
    """one rank's result against GraphNCF.recommend for the nodes it served"""
    from deeprecommendation_b200.graph import get_index
    nodes, val, idx = res[:3]
    n, nI = nodes.numel(), g.item_features.shape[0]
    assert val.shape == (n, k) and idx.shape == (n, k) and idx.dtype == torch.int64
    if n == 0:
        return
    with torch.no_grad():
        rv, ri, rs = m.recommend(g, k, user_nodes=nodes, precision=precision, ignore_seen=ignore_seen, return_scores=True)
    S = rs.double().clone()
    if ignore_seen:                                         # the MLP path's scores include seen items; the dot path's hold NaN there
        ptr, items = get_index(g).seen_items(nodes)
        rows = torch.repeat_interleave(torch.arange(n, device=DEV), (ptr[1:] - ptr[:-1]).long())
        S[rows, items.long()] = float('nan')
    scale = float(S.nan_to_num(0.0).abs().max())
    pad = idx < 0
    assert torch.equal(pad, ri < 0) and torch.isinf(val[pad]).all() and (val[pad] < 0).all()
    if bool(pad.all()):
        return
    assert float((val[~pad].double() - rv[~pad].double()).abs().max()) <= tol * scale
    got = S.gather(1, idx.clamp_min(0))
    assert not torch.isnan(got[~pad]).any()                 # never a seen item
    assert float((got[~pad] - val[~pad].double()).abs().max()) <= tol * scale
    srt = S.nan_to_num(float('-inf')).sort(dim=1, descending=True).values
    if nI > k:
        clear = (srt[:, k - 1] - srt[:, k] > 2 * tol * scale) & torch.isfinite(srt[:, k])
        for u in clear.nonzero().view(-1).tolist():
            assert set(idx[u].tolist()) == set(ri[u].tolist()), u
    if return_scores:
        sc = res[3].double()
        ok = ~torch.isnan(rs)
        assert sc.shape == (n, nI) and float((sc[ok] - rs.double()[ok]).abs().max()) <= tol * scale


def _run(m, g, P, k=10, users=None, tol=1e-5, shards=None, **kw):
    from deeprecommendation_b200.peer import catalogue_width, emulated_shards, recommend_emulated
    shards = shards or emulated_shards(g, P, d_max=128, batch_max=512, catalogue_width=catalogue_width(m))
    with torch.no_grad():
        outs = recommend_emulated(m, shards, k=k, users=users, **kw)
    torch.cuda.synchronize()
    for sh in shards:
        sh.check()
    nI, N = g.item_features.shape[0], g.item_features.shape[0] + g.user_features.shape[0]
    req = torch.arange(nI, N, device=DEV) if users is None else users
    served = torch.cat([o[0] for o in outs])
    assert sorted(served.tolist()) == sorted(req.tolist())
    for o in outs:
        if users is not None and o[0].numel():              # request order kept within a rank
            pos = {v: i for i, v in enumerate(users.tolist())}
            assert [pos[v] for v in o[0].tolist()] == sorted(pos[v] for v in o[0].tolist())
        _check_rank(m, g, o, k, tol, precision=kw.get('precision', 'fp32'), ignore_seen=kw.get('ignore_seen', True),
                    return_scores=kw.get('return_scores', False))
    return shards, outs


@pytest.mark.parametrize('P', [1, 2, 3, 8])
@pytest.mark.parametrize('scorer', sorted(MLPS))
def test_recommend_emulated_ranks_match_single_gpu(P, scorer):
    m, g = _graph(mlp=MLPS[scorer])
    _run(m, g, P, return_scores=True)


@pytest.mark.parametrize('conv,concat,d_emb,L_,scorer,hetero', [
    ('LightGAT', False, 64, 2, 'k5', True),
    ('LightGCN', True, 32, 2, 'dot', True),           # width 96 -> the dot kernel pads to 128
    ('LightGAT', True, 48, 2, 'relu_dot', True),
    ('LightGAT', True, 32, 3, 'dot', True),
    ('LightGCN', False, 64, 0, 'dot', True),
    ('LightGAT', False, 48, 0, 'k5', True),
    ('LightGCN', False, 128, 3, 'k5', True),
    ('LightGCN', False, 64, 2, 'relu_dot', False),     # homogeneous: one W for both edge types
    ('LightGAT', False, 64, 2, 'dot', False),
])
def test_recommend_models(conv, concat, d_emb, L_, scorer, hetero):
    m, g = _graph(n_users=1200, n_items=700, n=45_000, d_emb=d_emb, L_=L_, mlp=MLPS[scorer], hetero=hetero, conv=conv, concat=concat, seed=5)
    _run(m, g, 3, k=10)


def test_recommend_bf16_messages_and_bf16_precision():
    m, g = _graph(mlp=MLPS['k5'])
    m.message_dtype = 'bf16'
    try:
        _run(m, g, 4, tol=1e-2)
    finally:
        m.message_dtype = 'fp32'
    _run(m, g, 4, tol=1e-2, precision='bf16')
    m, g = _graph(mlp=None)
    _run(m, g, 2, tol=1e-2, precision='bf16')          # the exact dot kernel serves a bf16 request too


@pytest.mark.parametrize('k', [1, 10, 64])
@pytest.mark.parametrize('scorer', ['k5', 'dot'])
def test_recommend_users_subset_ignore_seen_and_chunks(k, scorer):
    m, g = _graph(mlp=MLPS[scorer])
    nI = g.item_features.shape[0]
    gen = torch.Generator().manual_seed(k)
    users = (torch.randperm(1500, generator=gen)[:400] + nI).to(DEV)      # every rank's range, shuffled
    _run(m, g, 3, k=k, users=users, ignore_seen=False, return_scores=True)
    _run(m, g, 3, k=k, users=users, chunk_users=37)
    _run(m, g, 2, k=k, chunk_users=100)


@pytest.mark.parametrize('scorer', sorted(MLPS))
def test_recommend_tiny_catalogue_pads_rows(scorer):
    """12 items, users who have seen nearly all of them: k = 10 leaves padded rows (-inf, -1) like the single-GPU call"""
    m, g = _graph(n_users=300, n_items=12, n=1500, mlp=MLPS[scorer], seed=9)
    _, outs = _run(m, g, 3, k=10)
    assert any(bool((o[2] < 0).any()) for o in outs)


@pytest.mark.parametrize('scorer', ['relu_dot', 'dot'])
def test_recommend_more_ranks_than_item_rows(scorer):
    m, g = _graph(n_users=400, n_items=5, n=800, mlp=MLPS[scorer], seed=7)       # 5 items over 8 ranks: ranks without items push nothing
    shards, _ = _run(m, g, 8, k=3)
    assert sum(sh.it_rows == 0 for sh in shards) == 3


def test_recommend_rank_without_users():
    """more ranks than users with edges: a rank that serves nobody still pushes its items and joins both barriers"""
    from deeprecommendation_b200.peer import catalogue_width, emulated_shards, recommend_emulated
    m, g = _graph(n_users=2, n_items=300, n=200, mlp=MLPS['relu_dot'], seed=4)
    shards = emulated_shards(g, 3, d_max=64, batch_max=64, catalogue_width=catalogue_width(m))
    assert any(sh.users_rows == 0 for sh in shards)
    _run(m, g, 3, k=5, shards=shards)


def test_recommend_forward_recommend_with_changed_weights():
    """the epoch counters are shared by forwards and recommends; new weights reach the composites and the catalogue"""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.peer import catalogue_width, emulated_shards, forward_emulated
    m, g = _graph(mlp=MLPS['k5'])
    shards = emulated_shards(g, 3, d_max=64, batch_max=512, catalogue_width=catalogue_width(m))
    _, first = _run(m, g, 3, shards=shards)
    pick = torch.arange(0, 60_000, 200, device=DEV)
    uid, iid = g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()
    with torch.no_grad():
        ref = m(g, uid, iid, DEV)
        outs = forward_emulated(m, shards, uid, iid)
    torch.cuda.synchronize()
    assert all(maxnorm_rel(o, ref) < 1e-6 for o in outs)
    kw = dict(item_dim=48, user_dim=48, num_gnn_layers=2, hetero=True, node_emb=64, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=11, **kw)))
    ops.invalidate_caches()
    _, second = _run(m, g, 3, shards=shards)
    assert any(not torch.equal(a[1], b[1]) for a, b in zip(first, second) if a[0].numel())


def test_recommend_refuses_missing_or_narrow_catalogue_and_wide_dot_rows():
    from deeprecommendation_b200.peer import emulated_shards, recommend_peer
    m, g = _graph(mlp=MLPS['dot'], d_emb=32, L_=2, concat=True)                   # needs 128 (96 padded)
    with torch.no_grad():
        for width in (0, 96):
            sh = emulated_shards(g, 1, d_max=64, batch_max=64, catalogue_width=width)[0]
            with pytest.raises(ValueError, match='catalogue_width=128'):
                recommend_peer(m, sh)
        m, g = _graph(mlp=MLPS['dot'], d_emb=128, L_=2, concat=True)              # 384 floats per row
        sh = emulated_shards(g, 1, d_max=128, batch_max=64, catalogue_width=384)[0]
        with pytest.raises(NotImplementedError, match='256'):
            recommend_peer(m, sh)
        m.train()
        with pytest.raises(NotImplementedError, match='eval'):
            recommend_peer(m, sh)
    m.eval()
    with pytest.raises(NotImplementedError, match='inference'):
        recommend_peer(m, sh)


def test_recommend_per_rank_build_equals_shard_cut_from_full_index():
    """sharded.create_graph_local + shard_from_local (a rank sees only its users' interactions; its seen lists come from its local
    index, whose item ids exceed the number of owned users) recommends what shard_from_full does"""
    from deeprecommendation_b200.graph import IdTable, create_graph, get_index
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.peer import PeerArena, PeerShard, _rows_per_part, catalogue_width, emulated_shards, recommend_emulated
    from deeprecommendation_b200.sharded import create_graph_local, shard_from_local
    n_users, n_items, n, F, d, P = 2000, 700, 80_000, 64, 64, 4
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=17)
    order = np.argsort(users, kind='stable')
    users, items, ratings = users[order], items[order], ratings[order]
    rng = np.random.default_rng(3)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    tu, ti, tr = torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV)
    g = create_graph(tu, ti, tr, torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV), IdTable(torch.arange(n_users, device=DEV)),
                     IdTable(torch.arange(n_items, device=DEV)))
    full = get_index(g)
    for scorer in ('relu_dot', 'dot'):
        kw = dict(item_dim=F, user_dim=F, num_gnn_layers=3, hetero=True, node_emb=d, mlp_dense_layers=list(MLPS[scorer] or (8,)), dropout_rate=0.2,
                  use_dot_product=MLPS[scorer] is None)
        m = GraphNCF(**kw).to(DEV).eval()
        m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=3, **kw)))
        cw = catalogue_width(m)
        ref_shards = emulated_shards(g, P, d_max=d, batch_max=512, catalogue_width=cw)
        glob = {'cnt': torch.bincount(ti, minlength=n_items).int(), 'sum': torch.zeros(n_items, dtype=torch.float64, device=DEV).index_add_(0, ti, tr.double()),
                'deg': full.deg[:n_items].clone()}
        reduce_items = lambda t, what: t.copy_(glob[what])
        arenas = PeerArena.emulated(PeerShard.layout(P, _rows_per_part(n_items, P), d, 512, cw)['total'], P, DEV)
        shards = []
        for q, ref in enumerate(ref_shards):
            mine = (tu >= ref.users_r0) & (tu < ref.users_r0 + ref.users_rows)
            gl = create_graph_local(tu[mine] - ref.users_r0, ti[mine], tr[mine], ref.users_rows, n_items, g.item_features,
                                    g.user_features[ref.users_r0: ref.users_r0 + ref.users_rows], reduce_items)
            shards.append(shard_from_local(gl, rank=q, world=P, nI=n_items, nU=n_users, users_r0=ref.users_r0, arena=arenas[q], d_max=d,
                                           batch_max=512, reduce_items=reduce_items, edges_total=full.e1 + full.e2, catalogue_width=cw))
        assert any(sh.users_rows < n_items for sh in shards)
        with torch.no_grad():
            a = recommend_emulated(m, ref_shards, k=10)
            b = recommend_emulated(m, shards, k=10)
        torch.cuda.synchronize()
        for x, y in zip(a, b):
            assert torch.equal(x[0], y[0]) and torch.equal(x[2], y[2]) and maxnorm_rel(x[1], y[1]) < 1e-6
        _run(m, g, P, shards=shards)


def test_recommend_two_processes_share_one_gpu_over_cuda_ipc():
    """two real ranks (gloo rendezvous, both on cuda:0): the catalogue crosses process boundaries through the mapped arenas"""
    env = dict(os.environ, MASTER_ADDR='127.0.0.1', MASTER_PORT=str(29900 + os.getpid() % 300), B200REC_PEER_CHECK_SAME_GPU='1')
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
                        '--master-port', env['MASTER_PORT'], os.path.join(ROOT, 'tests', 'mp_peer_recommend_check.py')],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert r.returncode == 0 and lines, (r.returncode, r.stdout[-2000:], r.stderr[-3000:])
    res = json.loads(lines[-1])
    assert res['ok'] and res['world'] == 2, res
