"""Scheme 'peer' with LightGAT and the concat combine (deeprecommendation_b200/peer.py, csrc/spmm.cu, csrc/peer.cu): K3 pushes unnormalised
partial item rows with their softmax state (m, l), the owner merges the P slots (b200rec_peer_reduce_softmax), the owners publish their
item scores into every rank's score table, and every rank keeps its owned rows of comb = [x0 | ... | xL].  Same harness as
tests/test_peer_gpu.py: P emulated ranks inside one process, and two real processes on cuda:0 (tests/mp_peer_gat_check.py).
Reference = the single-GPU forward (pinned to the reference goldens in tests/test_models_gpu.py), plus the stored goldens themselves."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import synth
from tests._golden import load, maxnorm_rel

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _graph(n_users=1500, n_items=900, n=60_000, F=48, d_emb=64, L_=2, mlp=(128,), dot=False, seed=13, conv='LightGAT', hetero=True,
           concat=False):
    from deeprecommendation_b200.graph import IdTable, create_graph
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=seed)
    rng = np.random.default_rng(2)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=L_, hetero=hetero, node_emb=d_emb, mlp_dense_layers=list(mlp), dropout_rate=0.2,
              use_dot_product=dot, convType=conv, concat=concat)
    sd = synth.to_torch(synth.graph_ncf_weights(seed=3, **kw))
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV),
                     IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV)))
    m = GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    pick = rng.permutation(n)[:300]
    return m, g, g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()


def _check_world(m, g, uid, iid, P, tol=1e-5, d_max=128, batch_max=512):
    from deeprecommendation_b200.graph import get_index
    from deeprecommendation_b200.peer import emulated_shards, forward_emulated
    full = get_index(g)
    nI = g.item_features.shape[0]
    with torch.no_grad():
        ref = m(g, uid, iid, DEV)
        comb = m._encode(g, full, None, full.dinv, False)
        shards = emulated_shards(g, P, d_max=d_max, batch_max=batch_max)
        assert sum(sh.edges_own for sh in shards) == full.e1 + full.e2
        assert sum(sh.users_rows for sh in shards) == full.num_nodes - nI and sum(sh.it_rows for sh in shards) == nI
        for rep in range(2):                         # second pass: the device-side epoch counters advance (CUDA-graph replay contract)
            keep = [dict() for _ in range(P)]
            outs = forward_emulated(m, shards, uid, iid, keep)
            torch.cuda.synchronize()
            for sh, out, k in zip(shards, outs, keep):
                sh.check()
                assert maxnorm_rel(out, ref) < tol, (P, sh.rank, rep)
                assert k['items'].shape[1] == comb.shape[1] and k['users'].shape[1] == comb.shape[1]
                assert maxnorm_rel(k['items'], comb[sh.it_r0: sh.it_r0 + sh.it_rows]) < tol if sh.it_rows else True
                assert maxnorm_rel(k['users'], comb[nI + sh.users_r0: nI + sh.users_r0 + sh.users_rows]) < tol if sh.users_rows else True
            assert all(torch.equal(outs[0], o) for o in outs[1:])       # every rank ends with the same bits
    return outs[0], ref


@pytest.mark.parametrize('P', [1, 2, 3, 8])
def test_gat_emulated_ranks_match_single_gpu(P):
    m, g, uid, iid = _graph()
    _check_world(m, g, uid, iid, P)


@pytest.mark.parametrize('P', [2, 3])
def test_gat_homogeneous(P):
    m, g, uid, iid = _graph(hetero=False, seed=9)
    _check_world(m, g, uid, iid, P)


@pytest.mark.parametrize('d_emb,L_,mlp', [(128, 2, (256, 128)), (64, 3, (128,)), (32, 1, (64,)), (64, 0, (128,)), (48, 2, (64,))])
def test_gat_emulated_shapes(d_emb, L_, mlp):
    """d = 48 is not a shape of K1c: the transform takes the plain GEMM + the copy kernel to the peers"""
    m, g, uid, iid = _graph(n_users=2500, n_items=1200, n=90_000, d_emb=d_emb, L_=L_, mlp=mlp, seed=5)
    _check_world(m, g, uid, iid, 3)


@pytest.mark.parametrize('P', [1, 2, 3, 8])
@pytest.mark.parametrize('conv', ['LightGCN', 'LightGAT'])
def test_concat_emulated_ranks_match_single_gpu(conv, P):
    m, g, uid, iid = _graph(conv=conv, concat=True, L_=2, mlp=(128,))
    _check_world(m, g, uid, iid, P)


@pytest.mark.parametrize('conv,concat,L_', [('LightGAT', False, 2), ('LightGAT', True, 3), ('LightGCN', True, 1)])
def test_dot_product_and_more_ranks_than_item_rows(conv, concat, L_):
    """11 items over 8 ranks: empty item shards; the dot-product head reads the (L+1)·d-wide rows under concat"""
    m, g, uid, iid = _graph(n_users=400, n_items=11, n=2500, d_emb=64, L_=L_, dot=True, seed=7, conv=conv, concat=concat)
    _check_world(m, g, uid, iid, 8, batch_max=1024)


@pytest.mark.parametrize('concat', [False, True])
def test_gat_bf16_messages(concat):
    m, g, uid, iid = _graph(d_emb=128, L_=2, mlp=(256, 128), concat=concat)
    with torch.no_grad():
        ref = m(g, uid, iid, DEV)
    m.message_dtype = 'bf16'
    try:
        out, _ = _check_world(m, g, uid, iid, 4, tol=1e-2, batch_max=1024)
    finally:
        m.message_dtype = 'fp32'
    assert maxnorm_rel(out, ref) < 1e-2 and not torch.equal(out, ref)


def test_gat_push_and_softmax_merge_equal_single_gpu_rows():
    """K3 LightGAT with `push`: every rank pushes its unnormalised partial item rows + (m, l); b200rec_peer_reduce_softmax merges the P slots.
    The merged rows equal the single-GPU K3 LightGAT x_next.  16-edge chunks, so that rows span several chunks and some rows have more than
    FIX_LONG = 64 chunk slots on one rank (the fix-up kernel's CTA-cooperative phase)."""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.graph import get_index
    from deeprecommendation_b200.parallel import _LocalIndex
    from deeprecommendation_b200.peer import emulated_shards
    m, g, uid, iid = _graph(n_users=6000, n_items=500, n=200_000, d_emb=64, seed=11)
    P, d, nI = 3, 64, 500
    full = get_index(g)
    shards = emulated_shards(g, P, d_max=d, batch_max=64)
    gen = torch.Generator(device=DEV).manual_seed(5)
    t = torch.randn(6000, d, device=DEV, generator=gen)
    ps = 2.0 * torch.randn(6000, device=DEV, generator=gen)
    t_full = torch.cat((torch.zeros(nI, d, device=DEV), t))
    ps_full = torch.cat((torch.zeros(nI, device=DEV), ps))
    ref = torch.zeros(full.num_nodes, d, device=DEV)
    ops.spmm_raw(full, t_full, w=full.w, dinv=None, x_next=ref, att_src=ps_full)
    multi, long_rows = False, False
    for par in (0, 1):
        for sh in shards:
            ix = sh.index_items
            ix16 = _LocalIndex(ix.row_ptr, ix.col, ix.w, ix.pos, ix.dinv, 16)
            multi |= ix16.n_multi > 0
            long_rows |= bool(ix16.n_multi > 0 and int(ix16.multi_n_slots.max()) > 64)
            r0, n = sh.users_r0, sh.users_rows
            ops.spmm_raw(ix16, t[r0: r0 + n].contiguous(), w=ix16.w, dinv=None, att_src=ps[r0: r0 + n].contiguous(), push=sh.push_spec(par, d),
                         push_stats=sh.stats_offset(par))
        for sh in shards:
            out = torch.full((sh.it_rows, d), float('nan'), device=DEV)
            sh.reduce(par, d, x_next=out, acc_in=None, acc_out=None, acc_scale=1.0, softmax=True)
            torch.cuda.synchronize()
            want = ref[sh.it_r0: sh.it_r0 + sh.it_rows]
            assert maxnorm_rel(out, want) < 1e-5, (par, sh.rank)
            no_edges = full.row_ptr[sh.it_r0 + 1: sh.it_r0 + sh.it_rows + 1] == full.row_ptr[sh.it_r0: sh.it_r0 + sh.it_rows]
            assert torch.all(out[no_edges] == 0)                       # a row without edges merges to 0, as on one GPU
    assert multi and long_rows


def test_gat_push_needs_the_statistics_destination():
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.peer import emulated_shards
    m, g, uid, iid = _graph(n_users=300, n_items=80, n=3000)
    sh = emulated_shards(g, 2, d_max=64, batch_max=16)[0]
    tu = torch.randn(sh.users_rows, 64, device=DEV)
    ps = torch.randn(sh.users_rows, device=DEV)
    with pytest.raises(ValueError, match='push_stats'):
        ops.spmm_raw(sh.index_items, tu, w=sh.index_items.w, att_src=ps, push=sh.push_spec(0, 64))


def _graph_from_golden(build, d):
    from deeprecommendation_b200.graph import GraphData
    g = GraphData(item_features=torch.from_numpy(d['item_features']), user_features=torch.from_numpy(d['user_features']),
                  user2item_edge_index=torch.from_numpy(build['user2item_edge_index']),
                  item2user_edge_index=torch.from_numpy(build['item2user_edge_index']),
                  user2item_edge_attr=torch.from_numpy(build['user2item_edge_attr']) if 'user2item_edge_attr' in build else None,
                  item2user_edge_attr=torch.from_numpy(build['item2user_edge_attr']) if 'item2user_edge_attr' in build else None)
    return g.to(DEV)


@pytest.mark.parametrize('P', [2, 3])
@pytest.mark.parametrize('name', ['graph_ncf_gat', 'graph_ncf_concat'])
def test_partitioned_forward_on_reference_goldens(name, P):
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.peer import emulated_shards, forward_emulated
    d, sd, kw = load(name)
    build, _, _ = load('graph_build_binary0')
    g = _graph_from_golden(build, d)
    m = GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    uid, iid = torch.from_numpy(d['userIds']).to(DEV), torch.from_numpy(d['itemIds']).to(DEV)
    with torch.no_grad():
        shards = emulated_shards(g, P, d_max=64, batch_max=64)
        outs = forward_emulated(m, shards, uid, iid)
    torch.cuda.synchronize()
    for sh, o in zip(shards, outs):
        sh.check()
        assert maxnorm_rel(o, d['out']) < 1e-5, (name, P, sh.rank)


def test_sharded_build_with_lightgat_equals_cut_out_shards():
    """sharded.create_graph_local / shard_from_local (a rank sees only its users' interactions) against peer.shard_from_full, with a LightGAT
    model: the same forward"""
    from deeprecommendation_b200.graph import IdTable, create_graph, get_index
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.peer import PeerArena, PeerShard, _rows_per_part, emulated_shards, forward_emulated
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
    ref_shards = emulated_shards(g, P, d_max=d, batch_max=512)
    glob = {'cnt': torch.bincount(ti, minlength=n_items).int(), 'sum': torch.zeros(n_items, dtype=torch.float64, device=DEV).index_add_(0, ti, tr.double()),
            'deg': full.deg[:n_items].clone()}
    reduce_items = lambda t, what: t.copy_(glob[what])
    arenas = PeerArena.emulated(PeerShard.layout(P, _rows_per_part(n_items, P), d, 512)['total'], P, DEV)
    shards = []
    for q, ref in enumerate(ref_shards):
        mine = (tu >= ref.users_r0) & (tu < ref.users_r0 + ref.users_rows)
        gl = create_graph_local(tu[mine] - ref.users_r0, ti[mine], tr[mine], ref.users_rows, n_items, g.item_features,
                                g.user_features[ref.users_r0: ref.users_r0 + ref.users_rows], reduce_items)
        shards.append(shard_from_local(gl, rank=q, world=P, nI=n_items, nU=n_users, users_r0=ref.users_r0, arena=arenas[q], d_max=d, batch_max=512,
                                       reduce_items=reduce_items, edges_total=full.e1 + full.e2))
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=3, hetero=True, node_emb=d, mlp_dense_layers=[128], dropout_rate=0.2, convType='LightGAT')
    m = GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=3, **kw)))
    pick = rng.permutation(n)[:300]
    uid, iid = g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()
    with torch.no_grad():
        ref_out = m(g, uid, iid, DEV)
        cut = forward_emulated(m, ref_shards, uid, iid)
        outs = forward_emulated(m, shards, uid, iid)
    torch.cuda.synchronize()
    for sh, o, c in zip(shards, outs, cut):
        sh.check()
        assert torch.equal(o, c)
        assert maxnorm_rel(o, ref_out) < 1e-5


def test_gat_two_processes_share_one_gpu_over_cuda_ipc():
    """two real ranks (gloo rendezvous, both on cuda:0): LightGAT, concat and bf16 messages across process boundaries"""
    env = dict(os.environ, MASTER_ADDR='127.0.0.1', MASTER_PORT=str(29300 + os.getpid() % 300), B200REC_PEER_CHECK_SAME_GPU='1')
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
                        '--master-port', env['MASTER_PORT'], os.path.join(ROOT, 'tests', 'mp_peer_gat_check.py')],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert r.returncode == 0 and lines, (r.returncode, r.stdout[-2000:], r.stderr[-3000:])
    res = json.loads(lines[-1])
    assert res['ok'] and res['world'] == 2, res


@pytest.mark.parametrize('kw', [dict(convType='LightGAT'), dict(concat=True)])
def test_nccl_schemes_still_refuse_gat_and_concat(kw):
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    from deeprecommendation_b200.parallel import encode_partitioned, forward_user_partitioned
    m = GraphNCF(item_dim=16, user_dim=16, num_gnn_layers=2, hetero=True, node_emb=16, mlp_dense_layers=[16], **kw).eval()
    ids = torch.zeros(4, dtype=torch.int64)
    with torch.no_grad():
        with pytest.raises(NotImplementedError, match='concat / LightGAT'):
            forward_user_partitioned(m, None, ids, ids)                 # scheme 'reduce'
        with pytest.raises(NotImplementedError, match='concat / LightGAT'):
            encode_partitioned(m, None)                                 # scheme 'gather'


def test_concat_batch_over_the_rows_capacity_raises():
    from deeprecommendation_b200.peer import emulated_shards, forward_emulated
    m, g, uid, iid = _graph(n_users=300, n_items=80, n=3000, d_emb=64, L_=2, conv='LightGCN', concat=True)
    shards = emulated_shards(g, 2, d_max=64, batch_max=64)
    ids = torch.arange(64, device=DEV)                 # 64 pairs fit batch_max, but not 64 rows of 3 x 64 floats in a 64 x 64 buffer
    with torch.no_grad(), pytest.raises(ValueError, match='concatenated rows'):
        forward_emulated(m, shards, g.user2item_edge_index[0][ids].contiguous(), g.user2item_edge_index[1][ids].contiguous())
