"""Independent pin of the PyG boundary (SURVEY.md §8c: GraphNCF's arithmetic runs inside torch_geometric 2.0.4, which is absent here).

Everything graph-side in this repo is checked against the unmodified `gnn_ncf.py` running on `oracle/pyg_shim` — a chain that
would not notice a mistake in the shim itself.  This file closes that loop with CLOSED FORMS written from the published PyG 2.0.4
definitions, in float64, with plain Python loops over nodes and edges (no index_add / scatter / gather shared with the shim):

    degree(index, N)[n]          = #{e : index[e] = n}
    softmax(src, index)[e]       = exp(src[e] - max_{e' : index[e'] = index[e]} src[e']) / (sum_{e'} exp(...) + 1e-16)
    subgraph(S, edges)           = edges whose BOTH endpoints are in S, in order, not relabelled
    propagate (aggr='add',       out[i] = sum_{e : dst[e] = i} message_e;   x_j = x[src[e]], x_i = x[dst[e]]
      flow source_to_target)
    LightGCNConv (gnn_ncf.py:39-94)    out = D^-1/2 A_u2i D^-1/2 (X W_u2i^T + b) + D^-1/2 A_i2u D^-1/2 (X W_i2u^T + b'),
                                       D = in-degree over BOTH lists (duplicates and zero-weight edges count), 0 where deg = 0
    LightGATConv (gnn_ncf.py:128-177)  out[i] = sum_e w_e * softmax_i(a·[x_j; x_i] + a0)_e * (W x_j + b), softmax per list

Tiny graphs cover a node without in-edges, an isolated node, a duplicated edge, a zero-weight edge, a self-contained hub; the shim
and the restatement (oracle/restatement.py) are compared with the closed forms on them.  The UNMODIFIED reference layers on the shim
are compared with the closed forms through their stored outputs (tests/golden/graph_ncf_*.npz), so no reference checkout is needed."""
import math

import numpy as np
import pytest
import torch

from oracle import restatement as R

TOL = 1e-5      # fp32 implementation vs float64 closed form, max-norm relative


def _shim():
    import importlib
    import os
    import sys
    p = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'oracle', 'pyg_shim')
    if p not in sys.path:
        sys.path.insert(0, p)
    return importlib.import_module('torch_geometric.utils'), importlib.import_module('torch_geometric.nn')


# ---- tiny hetero graphs: items are nodes 0..nI-1, users nI.. (graph_providers.py:76-80) -------------------------------------
def tiny_graphs():
    gs = []
    # A: 3 items, 4 users; item 2 has no rating (zero in-degree), user 6 is isolated, (u3,i0) rated twice, one zero weight
    nI, nU = 3, 4
    pairs = [(3, 0, 0.75), (4, 0, -1.25), (3, 1, 0.0), (5, 1, 2.0), (3, 0, -0.5), (4, 1, 1.5)]
    gs.append(('dup_zero_isolated', nI, nU, pairs))
    # B: one hub item rated by every user, one user rating everything
    nI, nU = 4, 5
    pairs = [(4 + u, 0, 0.5 * (u + 1) - 1.5) for u in range(nU)] + [(4, i, 0.25 * i - 0.5) for i in range(1, nI)]
    gs.append(('hub', nI, nU, pairs))
    # C: a single edge
    gs.append(('single_edge', 2, 2, [(3, 1, -2.25)]))
    return gs


def _lists(pairs, binary=False):
    u2i = torch.tensor([[u for u, _, _ in pairs], [i for _, i, _ in pairs]], dtype=torch.int64)
    i2u = torch.tensor([[i for _, i, _ in pairs], [u for u, _, _ in pairs]], dtype=torch.int64)
    wu = None if binary else torch.tensor([w for _, _, w in pairs], dtype=torch.float32)
    wi = None if binary else torch.tensor([0.5 * w + 0.125 for _, _, w in pairs], dtype=torch.float32)     # the two directions carry different attrs
    return u2i, i2u, wu, wi


def _weights(d, seed, gat=False):
    g = torch.Generator().manual_seed(seed)
    sd = {}
    for name in ('user2item_W', 'item2user_W'):
        sd[f'{name}.0.weight'] = torch.randn(d, d, generator=g) * 0.5
        sd[f'{name}.0.bias'] = torch.randn(d, generator=g) * 0.1
    if gat:
        for name in ('user2item_AttNet', 'item2user_AttNet'):
            sd[f'{name}.0.weight'] = torch.randn(1, 2 * d, generator=g) * 0.7
            sd[f'{name}.0.bias'] = torch.randn(1, generator=g) * 0.1
    return sd


# ---- closed forms (float64, explicit loops) -------------------------------------------------------------------------------
def closed_degree(index, n):
    deg = [0.0] * n
    for v in index.tolist():
        deg[v] += 1.0
    return deg


def closed_lightgcn(x, u2i, i2u, wu, wi, sd):
    N, d = x.shape
    X = x.double().numpy()
    deg = closed_degree(torch.cat([u2i[1], i2u[1]]), N)
    dinv = [0.0 if v == 0 else v ** -0.5 for v in deg]
    out = np.zeros((N, d))
    for (ei, w, name) in ((u2i, wu, 'user2item_W'), (i2u, wi, 'item2user_W')):
        W, b = sd[f'{name}.0.weight'].double().numpy(), sd[f'{name}.0.bias'].double().numpy()
        T = X @ W.T + b                                        # transform per NODE: the Linear commutes with the gather
        A = np.zeros((N, N))                                    # dense adjacency, duplicates add up
        for e in range(ei.shape[1]):
            s, t = int(ei[0, e]), int(ei[1, e])
            A[t, s] += 1.0 if w is None else float(w[e])
        Dm = np.diag(dinv)
        out += Dm @ A @ Dm @ T
    return out


def closed_lightgat(x, u2i, i2u, wu, wi, sd):
    N, d = x.shape
    X = x.double().numpy()
    out = np.zeros((N, d))
    for (ei, w, name, att) in ((u2i, wu, 'user2item_W', 'user2item_AttNet'), (i2u, wi, 'item2user_W', 'item2user_AttNet')):
        W, b = sd[f'{name}.0.weight'].double().numpy(), sd[f'{name}.0.bias'].double().numpy()
        a, a0 = sd[f'{att}.0.weight'].double().numpy()[0], float(sd[f'{att}.0.bias'][0])
        E = ei.shape[1]
        score = [float(a @ np.concatenate([X[int(ei[0, e])], X[int(ei[1, e])]]) + a0) for e in range(E)]
        for i in range(N):
            es = [e for e in range(E) if int(ei[1, e]) == i]
            if not es:
                continue
            m = max(score[e] for e in es)
            den = sum(math.exp(score[e] - m) for e in es) + 1e-16
            for e in es:
                alpha = math.exp(score[e] - m) / den
                out[i] += (1.0 if w is None else float(w[e])) * alpha * (W @ X[int(ei[0, e])] + b)
    return out


def rel(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


# ---- the shim's five symbols --------------------------------------------------------------------------------------------
def test_shim_degree_counts_duplicates_and_leaves_absent_nodes_zero():
    U, _ = _shim()
    idx = torch.tensor([2, 0, 2, 2, 5], dtype=torch.int64)
    got = U.degree(idx, 7, dtype=torch.float32)
    assert got.tolist() == closed_degree(idx, 7) == [1.0, 0.0, 3.0, 0.0, 0.0, 1.0, 0.0]
    assert U.degree(idx).shape[0] == 6                                   # num_nodes defaults to max + 1


def test_shim_softmax_matches_definition_including_the_1e16_denominator():
    U, _ = _shim()
    g = torch.Generator().manual_seed(0)
    src = torch.randn(9, 1, generator=g) * 3
    index = torch.tensor([0, 3, 3, 0, 3, 5, 0, 3, 5])
    got = U.softmax(src, index=index).double().view(-1).tolist()
    for e in range(9):
        grp = [k for k in range(9) if int(index[k]) == int(index[e])]
        m = max(float(src[k]) for k in grp)
        want = math.exp(float(src[e]) - m) / (sum(math.exp(float(src[k]) - m) for k in grp) + 1e-16)
        assert abs(got[e] - want) < 1e-6
    one = U.softmax(torch.tensor([[4.0]]), index=torch.tensor([2]))      # a group of one: 1 / (1 + 1e-16)
    assert float(one) == pytest.approx(1.0)


def test_shim_subgraph_keeps_edges_with_both_endpoints_no_relabel():
    U, _ = _shim()
    ei = torch.tensor([[0, 1, 2, 3, 4, 1], [1, 2, 3, 4, 0, 4]])
    attr = torch.arange(6, dtype=torch.float32)
    sub, sattr = U.subgraph(torch.tensor([1, 2, 4]), ei, attr, num_nodes=5)
    assert sub.tolist() == [[1, 1], [2, 4]] and sattr.tolist() == [1.0, 5.0]


def test_shim_propagate_adds_messages_at_the_destination():
    _, NN = _shim()

    class Scale(NN.MessagePassing):
        def __init__(self):
            super().__init__(aggr='add')

        def message(self, x_j, x_i, gain):
            return gain.view(-1, 1) * (x_j - 0.5 * x_i)

    x = torch.arange(12, dtype=torch.float32).view(4, 3)
    ei = torch.tensor([[0, 1, 1, 3], [2, 2, 0, 2]])
    gain = torch.tensor([1.0, -2.0, 0.5, 3.0])
    got = Scale().propagate(ei, x=(x, x), gain=gain)
    want = torch.zeros(4, 3)
    for e in range(4):
        s, t = int(ei[0, e]), int(ei[1, e])
        want[t] += gain[e] * (x[s] - 0.5 * x[t])
    assert torch.allclose(got, want) and torch.all(got[1] == 0) and torch.all(got[3] == 0)


# ---- restatement and the unmodified reference layers vs the closed forms ------------------------------------------------
CASES = [(name, nI, nU, pairs, binary) for (name, nI, nU, pairs) in tiny_graphs() for binary in (False, True)]


@pytest.mark.parametrize('name,nI,nU,pairs,binary', CASES, ids=[f'{c[0]}{"_binary" if c[4] else ""}' for c in CASES])
def test_restatement_lightgcn_and_lightgat_match_closed_forms(name, nI, nU, pairs, binary):
    d = 6
    x = torch.randn(nI + nU, d, generator=torch.Generator().manual_seed(3))
    u2i, i2u, wu, wi = _lists(pairs, binary)
    sd = _weights(d, 5, gat=True)
    psd = {f'c.{k}': v for k, v in sd.items()}
    got = R.lightgcn_conv(x, u2i, i2u, wu, wi, psd, 'c.')
    assert rel(got, closed_lightgcn(x, u2i, i2u, wu, wi, sd)) < TOL
    got = R.lightgat_conv(x, u2i, i2u, wu, wi, psd, 'c.')
    assert rel(got, closed_lightgat(x, u2i, i2u, wu, wi, sd)) < TOL
    if name == 'dup_zero_isolated':
        assert torch.all(got[2] == 0) and torch.all(got[nI + 3] == 0)       # no in-edge -> zero row


GOLDEN_GRAPH_CASES = ['graph_ncf_hetero_mean', 'graph_ncf_hetero_l3', 'graph_ncf_concat', 'graph_ncf_dot', 'graph_ncf_homo', 'graph_ncf_gat',
                      'graph_ncf_binary']


def closed_graph_ncf(d, build, kw, sd, masked=None):
    """GraphNCF.forward (gnn_ncf.py:298-367), dropouts inert, recomputed in float64 from the definitions: node embed, L layers of the ONE
    shared conv (gnn_convs.0, gnn_ncf.py:227), mean (or concat) of the L + 1 embeddings, item-first MLP or dot product.  `masked` = pos_df
    positions removed from both edge lists (the training target mask, gnn_ncf.py:314-320)."""
    u2i, i2u = (torch.from_numpy(build[k]) for k in ('user2item_edge_index', 'item2user_edge_index'))
    wu, wi = (torch.from_numpy(build[k]) if k in build else None for k in ('user2item_edge_attr', 'item2user_edge_attr'))
    if masked is not None:
        keep_u, keep_i = (np.setdiff1d(np.arange(ei.shape[1]), masked) for ei in (u2i, i2u))
        u2i, i2u = u2i[:, keep_u], i2u[:, keep_i]
        wu, wi = (None if w is None else w[k] for w, k in ((wu, keep_u), (wi, keep_i)))
    lin = lambda x, w, b: x @ sd[w].double().numpy().T + sd[b].double().numpy()
    x = np.vstack([lin(d['item_features'].astype(np.float64), 'item_embeddings.0.weight', 'item_embeddings.0.bias'),
                   lin(d['user_features'].astype(np.float64), 'user_embeddings.0.weight', 'user_embeddings.0.bias')])
    csd = {k[len('gnn_convs.0.'):]: v for k, v in sd.items() if k.startswith('gnn_convs.0.')}
    if not kw['hetero']:            # one transform over the union of both lists = the hetero form with the same W on each list
        csd = {f'{side}_W.0.{p}': csd[f'W.0.{p}'] for side in ('user2item', 'item2user') for p in ('weight', 'bias')}
    conv = closed_lightgat if kw.get('convType', 'LightGCN') == 'LightGAT' else closed_lightgcn
    hs = [x]
    for _ in range(kw['num_gnn_layers']):
        hs.append(conv(torch.from_numpy(hs[-1]), u2i, i2u, wu, wi, csd))
    emb = np.concatenate(hs, axis=1) if kw.get('concat') else sum(hs) / len(hs)
    item, user = emb[d['itemIds']], emb[d['userIds']]
    if kw.get('use_dot_product'):
        return (item * user).sum(axis=1, keepdims=True)
    h = np.concatenate([item, user], axis=1)
    keys = sorted({int(k.split('.')[1]) for k in sd if k.startswith('MLP.')})
    for q, k in enumerate(keys):
        h = lin(h, f'MLP.{k}.weight', f'MLP.{k}.bias')
        h = np.maximum(h, 0.0) if q < len(keys) - 1 else h
    return h


@pytest.mark.parametrize('name', GOLDEN_GRAPH_CASES)
def test_unmodified_reference_graphncf_golden_equals_stacked_closed_form(name):
    """tests/golden/graph_ncf_*.npz hold outputs of the UNMODIFIED reference GraphNCF executed on oracle/pyg_shim (oracle/make_golden.py),
    with its weights: LightGCN hetero / homogeneous / binary edges / 3 layers / concat / dot product, and LightGAT.  The stored reference
    outputs must equal the stacked closed forms — the reference on the shim checked against the definitions without the reference present."""
    from tests._golden import load
    d, sd, kw = load(name)
    build, _, _ = load('graph_build_binary1' if name == 'graph_ncf_binary' else 'graph_build_binary0')
    assert rel(d['out'], closed_graph_ncf(d, build, kw, sd)) < TOL
    if 'out_train_masked' in d:
        pos = {(int(a), int(b)): int(p) for a, b, p in zip(build['pos_Id1'], build['pos_Id2'], build['pos_pos'])}
        masked = np.array([pos[(int(u), int(i))] for u, i in zip(d['userIds'], d['itemIds'])])
        assert rel(d['out_train_masked'], closed_graph_ncf(d, build, kw, sd, masked)) < TOL
