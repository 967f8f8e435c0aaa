"""Partitioned GraphNCF training on the peer scheme (peer.train_emulated / forward_peer with grad): emulated ranks against the single-GPU
training path (GraphNCF.forward under autograd) and, with dropout, against a float64 restatement in this file that uses the masks the ranks
drew.  Scores and gradients must agree to 1e-5 (max-norm relative), and the gradients of all ranks must be bit-identical."""
import copy
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
TOL = 1e-5
# Parameters after Adam steps of an MLP model: Adam divides each gradient element by its own running magnitude, so elements whose gradient
# is near zero turn rounding-level differences into visible ones, and a ReLU input within rounding of 0 switches a unit on in one run and
# off in the other.  Two single-GPU runs of the same 3 steps of an MLP model (its backward sums rows with index_add_) were measured 1.2e-4
# apart in one MLP weight on a B200; a dot-product model stays within 1e-5 (tests/mp_peer_train_check.py).
PARAM_TOL = 1e-3


def _data(n_users=1200, n_items=700, n=40_000, F=40, seed=13, extra=None):
    """(users, items, ratings) numpy + graph; `extra` = interactions appended as they are (degree edge cases)"""
    from deeprecommendation_b200.graph import IdTable, create_graph
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=seed)
    if extra is not None:
        users, items, ratings = (np.concatenate((a, np.asarray(b, dtype=a.dtype))) for a, b in zip((users, items, ratings), extra))
        n_users, n_items = int(users.max()) + 1, int(items.max()) + 1
    rng = np.random.default_rng(2)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV),
                     IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV)))
    return g


def _model(g, d=64, L_=2, mlp=(128,), hetero=True, dropout=0.0, seed=3, **extra):
    from deeprecommendation_b200.neural_collaborative_filtering.models import GraphNCF
    F = g.item_features.shape[1]
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=L_, hetero=hetero, node_emb=d, mlp_dense_layers=list(mlp or (8,)), dropout_rate=dropout,
              use_dot_product=mlp is None, **{k: v for k, v in extra.items() if k in ('convType', 'concat')})
    m = GraphNCF(**kw, **{k: v for k, v in extra.items() if k not in kw}).to(DEV).train()
    m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=seed, **kw)))
    return m


def _batch(g, B, seed=5):
    pick = torch.from_numpy(np.random.default_rng(seed).permutation(g.user2item_edge_index.shape[1])[:B]).to(DEV)
    return g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()


def _loss(y):
    return lambda out: ((out - y) ** 2).sum()                        # sum-MSE


def _single(m, g, uid, iid, loss_fn, mask_targets=True):
    """single-GPU training step: (scores, {name: grad}).  Dot-product models: GraphNCF's propagation under autograd, then the row dot in torch."""
    from deeprecommendation_b200.graph import get_index
    m.zero_grad(set_to_none=True)
    if m.MLP is None:
        index = get_index(g)
        skip, dinv = None, index.dinv
        if m.training and mask_targets:
            skip, dinv = index.masked(index.positions(uid, iid))
        comb = m._encode(g, index, skip, dinv, m.training)
        out = (comb[uid] * comb[iid]).sum(1, keepdim=True)
    else:
        out = m(g, uid, iid, mask_targets=mask_targets)
    loss_fn(out).backward()
    return out.detach(), {n: p.grad.clone() for n, p in m.named_parameters() if p.grad is not None}


def _shards(g, P, m, batch_max=512, d_max=128, **kw):
    from deeprecommendation_b200.peer import emulated_shards, grad_floats
    return emulated_shards(g, P, d_max=d_max, batch_max=batch_max, grad_floats=grad_floats(m), **kw)


def _check(res, ref_out, ref_grads, tol=TOL):
    """every rank: scores and gradients within tol of the reference; gradients and scores bit-identical across ranks"""
    out0, g0 = res[0]
    assert maxnorm_rel(out0, ref_out.detach()) <= tol
    assert sorted(g0) == sorted(ref_grads)
    for n, r in ref_grads.items():
        assert maxnorm_rel(g0[n], r) <= tol, (n, maxnorm_rel(g0[n], r))
    for out, gr in res[1:]:
        assert torch.equal(out, out0)
        for n in g0:
            assert torch.equal(gr[n], g0[n]), n


def _parity(g, m, P, uid, iid, mask_targets=True, shards=None, steps=1, tol=TOL):
    from deeprecommendation_b200.peer import train_emulated
    shards = shards or _shards(g, P, m)
    y = torch.randn((uid.numel(), 1), generator=torch.Generator().manual_seed(7)).to(DEV)
    ref_m, probe = copy.deepcopy(m), copy.deepcopy(m)
    opt, ref_opt = (torch.optim.Adam(x.parameters(), lr=1e-3, fused=True) for x in (m, ref_m))
    for _ in range(steps):
        res = train_emulated(m, shards, uid, iid, _loss(y), mask_targets=mask_targets)
        torch.cuda.synchronize()
        for sh in shards:
            sh.check()
        probe.load_state_dict(m.state_dict())                  # the single-GPU step at the same parameters
        _check(res, *_single(probe, g, uid, iid, _loss(y), mask_targets), tol)
        for n, p in m.named_parameters():
            p.grad = res[0][1].get(n)
        opt.step()
        if steps > 1:                                          # and the single-GPU trajectory of its own
            _single(ref_m, g, uid, iid, _loss(y), mask_targets)
            ref_opt.step()
    if steps > 1:
        ref_p = dict(ref_m.named_parameters())
        for n, p in m.named_parameters():
            assert maxnorm_rel(p.detach(), ref_p[n].detach()) <= PARAM_TOL, n
    return shards


CASES = [  # (P, hetero, L, d, mlp, mask_targets)
    (1, True, 2, 64, (256, 128), True), (2, True, 2, 64, (256, 128), True), (3, False, 2, 32, (128,), True), (8, True, 2, 128, None, True),
    (1, False, 0, 64, (128,), True), (2, True, 0, 128, None, False), (3, True, 1, 64, (256, 128), False), (8, False, 1, 32, (128,), True),
    (1, True, 3, 32, None, True), (2, False, 3, 128, (128,), True), (3, True, 3, 64, None, True), (8, True, 3, 64, (256, 128), False),
    (2, True, 1, 128, (256, 128), True), (3, False, 0, 32, (256, 128), True), (8, False, 2, 64, None, False), (1, True, 1, 128, (128,), False),
]


@pytest.mark.parametrize('P, hetero, L_, d, mlp, mask', CASES)
def test_train_emulated_matches_single_gpu(P, hetero, L_, d, mlp, mask):
    g = _data()
    m = _model(g, d=d, L_=L_, mlp=mlp, hetero=hetero)
    uid, iid = _batch(g, 256)
    _parity(g, m, P, uid, iid, mask_targets=mask)


@pytest.mark.parametrize('P', [1, 2, 3, 8])
def test_three_adam_steps_follow_single_gpu(P):
    g = _data()
    m = _model(g, d=64, L_=2, mlp=(256, 128))
    uid, iid = _batch(g, 256)
    _parity(g, m, P, uid, iid, steps=3)


def test_duplicate_pairs_and_degrees_dropping_to_zero():
    """identical pairs count once; user 'lonely' and item 'rare' have one interaction each, so masking it leaves them without edges"""
    g = _data(extra=([1200, 5, 1200], [3, 700, 700], [4.0, 2.5, 3.0]))       # user 1200: items 3 and 700; item 700: users 5 and 1200
    g2 = _data(extra=([1200], [700], [4.0]))                                  # user 1200 and item 700: one edge, each other's only one
    for graph, pairs in ((g, [(1200, 3), (1200, 3), (5, 700), (1200, 700)]), (g2, [(1200, 700), (1200, 700)])):
        nI = graph.item_features.shape[0]
        uid, iid = _batch(graph, 200)
        extra_u = torch.tensor([nI + u for u, _ in pairs], device=DEV)
        extra_i = torch.tensor([i for _, i in pairs], device=DEV)
        uid, iid = torch.cat((uid, extra_u, uid[:20])), torch.cat((iid, extra_i, iid[:20]))      # and repeats of ordinary pairs
        for P in (1, 3, 8):
            _parity(graph, _model(graph, d=64, L_=2, mlp=(128,)), P, uid, iid)


def test_more_ranks_than_item_rows_and_rank_without_users():
    g = _data(n_users=400, n_items=5, n=800, F=16, seed=7)              # 5 items over 8 ranks
    shards = _shards(g, 8, _model(g))
    assert any(sh.it_rows == 0 for sh in shards)
    g2 = _data(n_users=2, n_items=300, n=200, F=16, seed=4)              # 2 users over 8 ranks
    shards2 = _shards(g2, 8, _model(g2))
    assert any(sh.users_rows == 0 for sh in shards2)
    for graph, sh in ((g, shards), (g2, shards2)):
        u, i = _batch(graph, 64)
        for mlp in ((128,), None):
            _parity(graph, _model(graph, d=32, L_=2, mlp=mlp), 8, u, i, shards=sh)


def test_batch_at_batch_max():
    g = _data()
    m = _model(g, d=64, L_=2, mlp=(256, 128))
    uid, iid = _batch(g, 512)
    _parity(g, m, 3, uid, iid, shards=_shards(g, 3, m, batch_max=512))


# ---- dropout: float64 restatement with the masks the ranks drew ------------------------------------------------------------
def _restate(m, g, uid, iid, conv_masks, mlp_masks, mask_targets=True):
    """GraphNCF's training forward in float64 (gnn_ncf.py:298-367 with transform-before-gather): returns the scores and a float64 copy of
    the parameters (leaves) the loss can be differentiated by"""
    from deeprecommendation_b200.neural_collaborative_filtering.util import mlp_parameters
    P = {n: p.detach().double().clone().requires_grad_() for n, p in m.named_parameters()}
    nI = g.item_features.shape[0]
    N = nI + g.user_features.shape[0]
    u2i, i2u = g.user2item_edge_index, g.item2user_edge_index
    wu, wi = g.user2item_edge_attr.double(), g.item2user_edge_attr.double()
    alive = torch.ones(u2i.shape[1], dtype=torch.bool, device=DEV)
    if mask_targets:
        key = {(int(a), int(b)): k for k, (a, b) in reversed(list(enumerate(zip(u2i[0].tolist(), u2i[1].tolist()))))}
        for a, b in zip(uid.tolist(), iid.tolist()):
            alive[key[(a, b)]] = False
    deg = torch.zeros(N, dtype=torch.float64, device=DEV)
    deg.index_add_(0, u2i[1][alive], torch.ones(int(alive.sum()), dtype=torch.float64, device=DEV))
    deg.index_add_(0, i2u[1][alive], torch.ones(int(alive.sum()), dtype=torch.float64, device=DEV))
    dinv = torch.where(deg > 0, deg.clamp_min(1).rsqrt(), torch.zeros_like(deg))
    lin = lambda x, pre: x @ P[pre + '.weight'].t() + P[pre + '.bias']
    x = torch.cat((lin(g.item_features.double(), 'item_embeddings.0'), lin(g.user_features.double(), 'user_embeddings.0')))
    hs = [x]
    conv = 'gnn_convs.0.' + ('{}2{}_W.0' if m.gnn_convs[0].hetero else 'W.0') if len(m.gnn_convs) else None
    for l in range(len(m.gnn_convs)):
        t = torch.cat((lin(x[:nI], conv.format('item', 'user')), lin(x[nI:], conv.format('user', 'item')))) * dinv[:, None]
        if conv_masks is not None:
            t = t * conv_masks[l]
        src = torch.cat((u2i[0][alive], i2u[0][alive]))
        dst = torch.cat((u2i[1][alive], i2u[1][alive]))
        w = torch.cat((wu[alive], wi[alive]))
        x = torch.zeros((N, t.shape[1]), dtype=torch.float64, device=DEV).index_add(0, dst, t[src] * w[:, None]) * dinv[:, None]
        hs.append(x)
    comb = torch.stack(hs).mean(0)
    a, b = comb[iid], comb[uid]
    if m.MLP is None:
        return (a * b).sum(1, keepdim=True), P
    weights, biases, _ = mlp_parameters(m.MLP)
    names = {id(p): n for n, p in m.named_parameters()}
    h = torch.cat((a, b), 1)
    for k, (wt, bs) in enumerate(zip(weights, biases)):
        h = h @ P[names[id(wt)]].t() + P[names[id(bs)]]
        if k < len(weights) - 1:
            h = torch.relu(h)
            if mlp_masks is not None:
                h = h * mlp_masks[k]
    return h, P


@pytest.mark.parametrize('P', [1, 3, 8])
@pytest.mark.parametrize('mlp', [(256, 128), None])
def test_dropout_matches_float64_restatement_with_the_drawn_masks(P, mlp):
    from deeprecommendation_b200.neural_collaborative_filtering.util import mlp_parameters
    from deeprecommendation_b200.peer import MLP_DROPOUT_SEED, train_emulated
    g = _data()
    m = _model(g, d=64, L_=2, mlp=mlp, dropout=0.3)
    uid, iid = _batch(g, 256)
    shards = _shards(g, P, m)
    keep = [{} for _ in shards]
    y = torch.randn((256, 1), generator=torch.Generator().manual_seed(7)).to(DEV)
    res = train_emulated(m, shards, uid, iid, _loss(y), keep=keep)
    torch.cuda.synchronize()
    conv_masks = []
    for l in range(2):
        mi = [k['masks_items'][l] for k in keep if k['masks_items'][l] is not None]
        mu = [k['masks_users'][l] for k in keep if k['masks_users'][l] is not None]
        conv_masks.append(torch.cat(mi + mu).double())
    assert float((conv_masks[0] == 0).double().mean()) == pytest.approx(0.15, abs=0.02)
    mlp_masks = None
    if mlp is not None:                            # what every shard's generator drew: the same stream, replayed here
        gen = torch.Generator(device=DEV)
        gen.manual_seed(MLP_DROPOUT_SEED)
        weights, _, p = mlp_parameters(m.MLP)
        mlp_masks = [torch.empty((256, w.shape[0]), device=DEV).bernoulli_(1 - p, generator=gen).div_(1 - p).double() for w in weights[:-1]]
    out, params = _restate(m, g, uid, iid, conv_masks, mlp_masks)
    ((out - y.double()) ** 2).sum().backward()
    ref_grads = {n: p.grad for n, p in params.items() if p.grad is not None}
    _check(res, out, ref_grads)


# ---- interleaving, per-rank build, two processes ------------------------------------------------------------------------
def test_inference_after_training_steps_equals_single_gpu_eval():
    from deeprecommendation_b200.peer import catalogue_width, forward_emulated, recommend_emulated
    g = _data()
    m = _model(g, d=64, L_=2, mlp=(256, 128))
    uid, iid = _batch(g, 256)
    shards = _parity(g, m, 3, uid, iid, shards=_shards(g, 3, m, catalogue_width=catalogue_width(m)), steps=2)
    m.eval()
    with torch.no_grad():
        ref = m(g, uid, iid)
        outs = forward_emulated(m, shards, uid, iid)
        recs = recommend_emulated(m, shards, k=10)
        rv, ri = m.recommend(g, 10, user_nodes=recs[1][0])
    for o in outs:
        assert maxnorm_rel(o, ref) <= TOL
    assert maxnorm_rel(recs[1][1], rv) <= TOL
    m.train()
    _parity(g, m, 3, uid, iid, shards=shards)          # and training again on the same epoch counters


def test_inference_forward_enqueues_the_same_kernels_with_grad_off():
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.peer import forward_peer
    g = _data()
    m = _model(g).eval()
    uid, iid = _batch(g, 128)
    sh = _shards(g, 1, m)[0]
    with torch.no_grad():
        forward_peer(m, sh, uid, iid)                  # one-time work (cached weight forms) out of the count
        n0 = ops.launch_count()
        forward_peer(m, sh, uid, iid)
        n1 = ops.launch_count()
        m.train()
        forward_peer(m, sh, uid, iid)                  # grad off: the inference forward, whatever the mode
        n2 = ops.launch_count()
    assert n1 - n0 == n2 - n1


def test_per_rank_build_gives_the_gradients_of_the_full_cut():
    from deeprecommendation_b200.graph import IdTable, create_graph, get_index
    from deeprecommendation_b200.peer import PeerArena, PeerShard, _rows_per_part, grad_floats, train_emulated
    from deeprecommendation_b200.sharded import create_graph_local, shard_from_local
    n_users, n_items, n, F, d, P = 1500, 600, 50_000, 32, 64, 4
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=17)
    order = np.argsort(users, kind='stable')
    users, items, ratings = users[order], items[order], ratings[order]
    rng = np.random.default_rng(3)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    tu, ti, tr = torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV)
    g = create_graph(tu, ti, tr, torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV), IdTable(torch.arange(n_users, device=DEV)),
                     IdTable(torch.arange(n_items, device=DEV)))
    full = get_index(g)
    m = _model(g, d=d, L_=3, mlp=(256, 128))
    gf = grad_floats(m)
    ref_shards = _shards(g, P, m, d_max=d)
    glob = {'cnt': torch.bincount(ti, minlength=n_items).int(), 'sum': torch.zeros(n_items, dtype=torch.float64, device=DEV).index_add_(0, ti, tr.double()),
            'deg': full.deg[:n_items].clone()}
    reduce_items = lambda t, what: t.copy_(glob[what])
    arenas = PeerArena.emulated(PeerShard.layout(P, _rows_per_part(n_items, P), d, 512, 0, gf)['total'], P, DEV)
    shards = []
    for q, ref in enumerate(ref_shards):
        mine = (tu >= ref.users_r0) & (tu < ref.users_r0 + ref.users_rows)
        gl = create_graph_local(tu[mine] - ref.users_r0, ti[mine], tr[mine], ref.users_rows, n_items, g.item_features,
                                g.user_features[ref.users_r0: ref.users_r0 + ref.users_rows], reduce_items)
        shards.append(shard_from_local(gl, rank=q, world=P, nI=n_items, nU=n_users, users_r0=ref.users_r0, arena=arenas[q], d_max=d,
                                       batch_max=512, reduce_items=reduce_items, edges_total=full.e1 + full.e2, grad_floats=gf))
    uid, iid = _batch(g, 300)
    y = torch.randn((300, 1), generator=torch.Generator().manual_seed(7)).to(DEV)
    a = train_emulated(m, ref_shards, uid, iid, _loss(y))
    b = train_emulated(m, shards, uid, iid, _loss(y))
    torch.cuda.synchronize()
    for (oa, ga), (ob, gb) in zip(a, b):
        assert maxnorm_rel(ob, oa) < 1e-6
        for n in ga:
            assert maxnorm_rel(gb[n], ga[n]) < 1e-6, n
    _parity(g, m, P, uid, iid, shards=shards)


# ---- errors ---------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('opt', ['gat', 'concat', 'node_dropout', 'message_dropout'])
def test_refused_options_raise_before_any_rank_signals(opt):
    from deeprecommendation_b200.peer import train_emulated
    g = _data(n_users=300, n_items=200, n=5000, F=16)
    extra = {'gat': dict(convType='LightGAT'), 'concat': dict(concat=True), 'node_dropout': dict(node_dropout=0.1),
             'message_dropout': dict(message_dropout=0.1)}[opt]
    m = _model(g, d=32, **extra)
    shards = _shards(g, 2, m)
    uid, iid = _batch(g, 32)
    counters = [sh.arena.buf[1024:1024 + 128].clone() for sh in shards]
    with pytest.raises(NotImplementedError):
        train_emulated(m, shards, uid, iid, lambda o: o.sum())
    assert all(torch.equal(sh.arena.buf[1024:1024 + 128], c) for sh, c in zip(shards, counters))


def test_binary_graph_and_nccl_schemes_are_refused():
    from deeprecommendation_b200.graph import IdTable, create_graph
    from deeprecommendation_b200.parallel import UserPartitionedGraph, forward_partitioned
    from deeprecommendation_b200.peer import train_emulated
    users, items, ratings = synth.interactions_zipf(300, 200, 5000, seed=3)
    rng = np.random.default_rng(1)
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(rng.standard_normal((200, 16)).astype(np.float32)).to(DEV),
                     torch.from_numpy(rng.standard_normal((300, 16)).astype(np.float32)).to(DEV),
                     IdTable(torch.arange(300, device=DEV)), IdTable(torch.arange(200, device=DEV)), binary=True)
    m = _model(g, d=32)
    uid, iid = _batch(g, 16)
    with pytest.raises(NotImplementedError, match='binary'):
        train_emulated(m, _shards(g, 2, m), uid, iid, lambda o: o.sum())
    g2 = _data(n_users=300, n_items=200, n=5000, F=16)
    pg = UserPartitionedGraph(g2, rank=0, world=1)
    with pytest.raises(NotImplementedError):
        forward_partitioned(m, pg, *_batch(g2, 16))


def test_missing_or_small_grad_section_raises_value_error():
    from deeprecommendation_b200.peer import emulated_shards, grad_floats, train_emulated
    g = _data(n_users=300, n_items=200, n=5000, F=16)
    m = _model(g, d=32)
    uid, iid = _batch(g, 32)
    for gf in (0, grad_floats(m) - 4):
        with pytest.raises(ValueError, match='grad_floats='):
            train_emulated(m, emulated_shards(g, 2, d_max=64, batch_max=64, grad_floats=gf), uid, iid, lambda o: o.sum())


@pytest.mark.parametrize('P', [1, 3])
def test_non_edge_pair_raises_key_error_on_every_rank(P):
    from deeprecommendation_b200.peer import train_emulated
    g = _data(n_users=300, n_items=200, n=5000, F=16)
    m = _model(g, d=32)
    shards = _shards(g, P, m)
    uid, iid = _batch(g, 32)
    nI = g.item_features.shape[0]
    edges = set(zip(g.user2item_edge_index[0].tolist(), g.user2item_edge_index[1].tolist()))
    bad = next((u, i) for u in range(nI + 299, nI, -1) for i in range(200) if (u, i) not in edges)
    uid[5], iid[5] = bad
    with pytest.raises(KeyError):
        train_emulated(m, shards, uid, iid, lambda o: o.sum())
    torch.cuda.synchronize()
    assert all(int(sh._err.item()) == 0 for sh in shards)
    uid, iid = _batch(g, 32)
    _parity(g, m, P, uid, iid, shards=shards)                # the counters stay in step: the next step runs


def test_two_processes_train_three_steps_over_cuda_ipc():
    env = dict(os.environ, B200REC_PEER_CHECK_SAME_GPU='1', MASTER_PORT='29517', PYTHONPATH=ROOT)
    r = subprocess.run([sys.executable, '-m', 'torch.distributed.run', '--nnodes=1', '--nproc-per-node', '2', '--master-addr', '127.0.0.1',
                        '--master-port', env['MASTER_PORT'], os.path.join(ROOT, 'tests', 'mp_peer_train_check.py')],
                       capture_output=True, text=True, timeout=600, env=env, cwd=ROOT)
    lines = [l for l in r.stdout.splitlines() if l.startswith('{')]
    assert r.returncode == 0 and lines, (r.returncode, r.stdout[-2000:], r.stderr[-3000:])
    res = json.loads(lines[-1])
    assert res['ok'] and res['world'] == 2, res
