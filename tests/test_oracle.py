"""The oracle's restatement vs golden outputs of the UNMODIFIED reference (CPU; no GPU needed).

tests/golden/*.npz were produced by oracle/make_golden.py running the original project's own classes.
A restatement that disagrees with them is not an oracle.
"""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from oracle import synth, ref_loader
from tests._golden import load, maxnorm_rel

TOL = 2e-6      # fp32 CPU vs fp32 CPU, same op order; only BLAS blocking may differ


@pytest.mark.parametrize('name', ['basic_small_a', 'basic_small_b', 'basic_small_c'])
def test_basic_small(name):
    d, sd, kw = load(name)
    out = R.basic_ncf_forward(sd, torch.from_numpy(d['X_user']), torch.from_numpy(d['X_item']))
    assert out.shape == d['out'].shape
    assert maxnorm_rel(out, d['out']) < TOL


@pytest.mark.parametrize('name', ['basic_full_256', 'basic_full_256_128'])
def test_basic_full(name):
    d, _, kw = load(name)
    sd = synth.to_torch(synth.basic_ncf_weights(seed=int(d['weight_seed']), **kw))
    B = int(d['B'])
    xi = torch.from_numpy(synth.item_profiles(B, seed=int(d['item_seed'])))
    xu = torch.from_numpy((synth.item_profiles(B, seed=int(d['user_seed'])) - 0.25) * 0.125)
    assert maxnorm_rel(R.basic_ncf_forward(sd, xu, xi), d['out']) < TOL


@pytest.mark.parametrize('name', ['attention_small_net', 'attention_small_lin', 'attention_small_cos'])
def test_attention_small(name):
    d, sd, kw = load(name)
    t = [torch.from_numpy(d[k]) for k in ('candidate_items', 'rated_items', 'user_matrix')]
    out, att = R.attention_ncf_forward(sd, *t, use_cos_sim_instead=kw['use_cos_sim_instead'], return_attention_weights=True)
    assert maxnorm_rel(out, d['out']) < TOL and maxnorm_rel(att, d['att']) < TOL
    assert torch.all(att[1] == 0)            # user with no rated item -> all weights 0 (attention_ncf.py:208-209)
    out_tr, att_tr = R.attention_ncf_forward(sd, *t, use_cos_sim_instead=kw['use_cos_sim_instead'], training=True,
                                             return_attention_weights=True)
    assert maxnorm_rel(out_tr, d['out_train']) < TOL and maxnorm_rel(att_tr, d['att_train']) < TOL
    assert att_tr[0, 3] == 0 and d['att'][0, 3] > 0     # the candidate's own rated entry is masked only in training
    # blocking over candidate rows does not change any value
    out_b = R.attention_ncf_forward_blocked(sd, *t, block=4, use_cos_sim_instead=kw['use_cos_sim_instead'])
    assert torch.equal(out_b, out) or maxnorm_rel(out_b, out) < 1e-6


def attention_full_inputs(d):
    B, I = int(d['B']), int(d['I'])
    prof = synth.item_profiles(I + B, seed=int(d['profile_seed']))
    rated = prof[:I]
    cand = prof[I:I + B].copy()
    cand[0] = rated[3]
    cand[5] = rated[0]
    return cand, rated, d['user_matrix']


def test_attention_full():
    d, _, kw = load('attention_full')
    wkw = {k: v for k, v in kw.items() if k not in ('use_cos_sim_instead', 'message_dropout')}
    sd = synth.to_torch(synth.attention_ncf_weights(seed=int(d['weight_seed']), **wkw))
    cand, rated, um = attention_full_inputs(d)
    out, att = R.attention_ncf_forward(sd, torch.from_numpy(cand), torch.from_numpy(rated), torch.from_numpy(um),
                                       return_attention_weights=True)
    assert maxnorm_rel(out, d['out']) < TOL and maxnorm_rel(att, d['att']) < TOL


@pytest.mark.parametrize('binary', [0, 1])
def test_create_graph_bit_exact(binary):
    d, _, _ = load(f'graph_build_binary{binary}')
    users_sorted, items_sorted = R.node_ids(d['all_users'], d['all_items'])
    g = R.create_graph(d['user_raw'], d['item_raw'], d['rating'], users_sorted, items_sorted, binary=bool(binary))
    assert np.array_equal(g['user2item_edge_index'], d['user2item_edge_index'])
    assert np.array_equal(g['item2user_edge_index'], d['item2user_edge_index'])
    if not binary:
        # bit-exact fp32 (view as int32 so that -0.0 / NaN could not hide)
        assert np.array_equal(g['user2item_edge_attr'].view(np.int32), d['user2item_edge_attr'].view(np.int32))
        assert np.array_equal(g['item2user_edge_attr'].view(np.int32), d['item2user_edge_attr'].view(np.int32))
    else:
        assert g['user2item_edge_attr'] is None and 'user2item_edge_attr' not in d
    # pos_df rows alternate u2i / i2u as the loop appends them (graph_providers.py:37,46); compare as a map
    ref_pos = {(int(a), int(b)): int(p) for a, b, p in zip(d['pos_Id1'], d['pos_Id2'], d['pos_pos'])}
    mine = {}
    for (s, t), p in zip(g['user2item_edge_index'].T.tolist(), g['pos_user2item'].tolist()):
        mine[(s, t)] = p
    for (s, t), p in zip(g['item2user_edge_index'].T.tolist(), g['pos_item2user'].tolist()):
        mine[(s, t)] = p
    assert mine == ref_pos


def _graph_dict(build, feats):
    g = {k: torch.from_numpy(build[k]) for k in ('user2item_edge_index', 'item2user_edge_index')}
    for k in ('user2item_edge_attr', 'item2user_edge_attr'):
        if k in build:
            g[k] = torch.from_numpy(build[k])
    g['item_features'] = torch.from_numpy(feats['item_features'])
    g['user_features'] = torch.from_numpy(feats['user_features'])
    return g


GRAPH_CASES = ['graph_ncf_hetero_mean', 'graph_ncf_hetero_l3', 'graph_ncf_concat', 'graph_ncf_dot', 'graph_ncf_homo',
               'graph_ncf_gat', 'graph_ncf_binary']


@pytest.mark.parametrize('name', GRAPH_CASES)
def test_graph_ncf(name):
    d, sd, kw = load(name)
    build, _, _ = load('graph_build_binary1' if name == 'graph_ncf_binary' else 'graph_build_binary0')
    g = _graph_dict(build, d)
    args = dict(hetero=kw['hetero'], concat=kw.get('concat', False), use_dot_product=kw.get('use_dot_product', False),
                convType=kw.get('convType', 'LightGCN'))
    uid, iid = torch.from_numpy(d['userIds']), torch.from_numpy(d['itemIds'])
    out = R.graph_ncf_forward(sd, g, uid, iid, kw['num_gnn_layers'], **args)
    assert maxnorm_rel(out, d['out']) < TOL
    if 'out_train_masked' in d:
        # look the batch's (user, item) pairs up in pos_df exactly as gnn_ncf.py:316-320,370 does
        pos = {(int(a), int(b)): int(p) for a, b, p in zip(build['pos_Id1'], build['pos_Id2'], build['pos_pos'])}
        positions = torch.tensor([pos[(int(u), int(i))] for u, i in zip(uid, iid)])
        out_m = R.graph_ncf_forward(sd, g, uid, iid, kw['num_gnn_layers'], masked_positions=positions, **args)
        assert maxnorm_rel(out_m, d['out_train_masked']) < TOL
        assert maxnorm_rel(out, d['out_train_unmasked']) < TOL
        assert maxnorm_rel(d['out_train_masked'], d['out_train_unmasked']) > 1e-4   # the mask does something


def test_collate():
    d, _, _ = load('collate')
    rated_ids, cand, rated, um = R.collate_interacted_items(
        d['batch_users'], d['batch_items'], d['row_ptr'], d['rated_idx'], d['rated_rating'], d['mean_rating'],
        d['profiles'])
    assert np.array_equal(rated_ids, d['rated_items_idx'])
    assert np.array_equal(cand.view(np.int32), d['candidate_items'].view(np.int32))
    assert np.array_equal(rated.view(np.int32), d['rated_items'].view(np.int32))
    assert np.array_equal(um.view(np.int32), d['user_matrix'].view(np.int32))
    assert np.all(um[2] == 0)     # user 4: every centred rating is exactly 0.0 -> "unrated" everywhere


def test_csr_by_destination_is_stable():
    build, _, _ = load('graph_build_binary0')
    ei = build['user2item_edge_index']
    n = int(max(ei.max(), build['item2user_edge_index'].max())) + 1
    row_ptr, src, perm = R.csr_by_destination(ei, n)
    assert row_ptr[-1] == ei.shape[1]
    for r in range(n):
        seg = perm[row_ptr[r]:row_ptr[r + 1]]
        assert np.all(ei[1][seg] == r) and np.all(np.diff(seg) > 0)
    assert np.array_equal(src, ei[0][perm])


@pytest.mark.reference
@pytest.mark.skipif(not ref_loader.available(), reason='B200REC_REFERENCE_ROOT does not name a checkout of the original project')
def test_restatement_vs_live_reference_shipped_checkpoint():
    """Shipped AttentionNCF checkpoint (real trained weights) through the live reference and the restatement."""
    import os
    ref = ref_loader.load()
    path = os.path.join(ref.checkpoint_dir, 'AttentionNCF_with_features_attNet128.pt')
    state, kwargs = torch.load(path, map_location='cpu', weights_only=False)
    m = ref.AttentionNCF(**kwargs).eval()
    m.load_state_dict(state)
    rng = np.random.default_rng(0)
    prof = synth.item_profiles(260, seed=5)
    cand, rated = torch.from_numpy(prof[:40]), torch.from_numpy(prof[40:])
    um = torch.from_numpy(((rng.integers(1, 11, (40, 220)) * 0.5 - 2.75) * (rng.random((40, 220)) < 0.3)).astype(np.float32))
    with torch.no_grad():
        out, att = m(cand, rated, um, return_attention_weights=True)
    o2, a2 = R.attention_ncf_forward(state, cand, rated, um, return_attention_weights=True)
    assert maxnorm_rel(o2, out) < TOL and maxnorm_rel(a2, att) < TOL


@pytest.mark.parametrize('net', [True, False])
def test_attention_pool_backward_closed_form_vs_autograd(net):
    """the per-non-zero gradient formulas the K2 backward kernel evaluates (oracle.attention_pool_backward) == autograd of the
    factorised forward, in float64: empty rows, a full row, masked pairs, score_scale != 1"""
    g = torch.Generator().manual_seed(5)
    B, I, H, U = 9, 40, 12, 8
    Pc, Pr, Q = (torch.randn(n, w, generator=g, dtype=torch.float64) for n, w in ((B, H), (I, H), (I, U)))
    a2, a20, bU = (torch.randn(n, generator=g, dtype=torch.float64) for n in (H, 1, U))
    um = (torch.randint(1, 11, (B, I), generator=g).double() * 0.5 - 2.75) * (torch.rand(B, I, generator=g) < 0.3)
    um[0] = 0.0
    um[1] = torch.randint(1, 11, (I,), generator=g).double() * 0.5 - 2.75
    keep = (um != 0) & (torch.rand(B, I, generator=g) < 0.9)            # some rated pairs masked out (target mask / dropped scores)
    gout = torch.randn(B, U, generator=g, dtype=torch.float64)
    leaves = [t.clone().requires_grad_(True) for t in (Pc, Pr, Q, a2, a20, bU)]
    out, alpha = R.attention_pool_factorised(*leaves, um, keep, net=net, scale=1.25)
    auto = torch.autograd.grad(out, leaves, gout, allow_unused=True)
    got = R.attention_pool_backward(Pc, Pr, Q, a2, bU, um, alpha.detach(), out.detach(), gout, net=net, scale=1.25)
    for name, ref in zip(('Pc', 'Pr', 'Q', 'a2', 'a20', 'bU'), auto):
        if not net and name in ('a2', 'a20'):
            assert got[name] is None
            continue
        assert torch.allclose(got[name].reshape(ref.shape), ref, rtol=1e-10, atol=1e-12), name
