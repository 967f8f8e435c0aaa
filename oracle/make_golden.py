"""Generate tests/golden/*.npz by running the UNMODIFIED reference (container only).

TEST INFRASTRUCTURE (oracle/__init__.py).  Usage:  python -m oracle.make_golden
Requires a checkout of the original project (B200REC_REFERENCE_ROOT).  The reference ships no golden vectors of its own (SURVEY.md §4), so these
fixtures — outputs of the reference's own classes on seeded inputs — are what pins the restatement
(oracle/restatement.py) and, through it, the CUDA path.  GraphNCF cases execute the reference's
gnn_ncf.py on top of oracle/pyg_shim (PyG 2.0.4 itself is not installable): "parity unpinned" at that
boundary, see oracle/__init__.py.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import pandas as pd
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

from oracle import ref_loader, synth  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden')


def _save(name, **arrays):
    os.makedirs(OUT, exist_ok=True)
    clean = {k: (v.detach().cpu().numpy() if torch.is_tensor(v) else np.asarray(v)) for k, v in arrays.items()
             if v is not None}
    np.savez_compressed(os.path.join(OUT, name + '.npz'), **clean)
    print(f'{name}: ' + ', '.join(f'{k}{list(v.shape)}' for k, v in clean.items()))


def _sd_arrays(sd, prefix='w::'):
    return {prefix + k: v for k, v in sd.items()}


# --------------------------------------------------------------------------------------------------
def golden_basic(ref):
    rng = np.random.default_rng(7)
    for tag, kw in {
        'basic_small_a': dict(item_dim=48, user_dim=40, item_emb=24, user_emb=16, mlp_dense_layers=[32, 16], dropout_rate=0.2),
        'basic_small_b': dict(item_dim=33, user_dim=33, item_emb=8, user_emb=8, mlp_dense_layers=[20], dropout_rate=None),
        'basic_small_c': dict(item_dim=70, user_dim=5, item_emb=12, user_emb=4, mlp_dense_layers=[24, 12, 6], dropout_rate=0.5),
    }.items():
        sd = synth.basic_ncf_weights(seed=3, **kw)
        m = ref.BasicNCF(**kw).eval()
        m.load_state_dict(synth.to_torch(sd))
        B = 37
        xu = rng.standard_normal((B, kw['user_dim'])).astype(np.float32)
        xi = rng.standard_normal((B, kw['item_dim'])).astype(np.float32)
        with torch.no_grad():
            out = m(torch.from_numpy(xu), torch.from_numpy(xi))
        _save(tag, X_user=xu, X_item=xi, out=out, kwargs=np.array(repr(kw)), **_sd_arrays(sd))
    # full reference shape (train_model.py:38-42 and the class default), outputs only
    for tag, layers in {'basic_full_256': [256], 'basic_full_256_128': [256, 128]}.items():
        kw = dict(item_dim=2094, user_dim=2094, item_emb=128, user_emb=128, mlp_dense_layers=layers, dropout_rate=0.2)
        sd = synth.basic_ncf_weights(seed=11, **kw)
        m = ref.BasicNCF(**kw).eval()
        m.load_state_dict(synth.to_torch(sd))
        xi = synth.item_profiles(96, seed=101)
        xu = (synth.item_profiles(96, seed=102) - 0.25) * 0.125
        with torch.no_grad():
            out = m(torch.from_numpy(xu), torch.from_numpy(xi))
        _save(tag, out=out, kwargs=np.array(repr(kw)), weight_seed=11, item_seed=101, user_seed=102, B=96)


def _attention_inputs(rng, B, I, F, density, profiles=None):
    rated = rng.random((I, F)).astype(np.float32) if profiles is None else profiles[:I]
    cand = rng.random((B, F)).astype(np.float32) if profiles is None else profiles[I:I + B].copy()
    cand[0] = rated[min(3, I - 1)]                # a candidate that IS one of the rated items (training mask :199)
    if B > 5:
        cand[5] = rated[0]
    um = (rng.integers(1, 11, size=(B, I)) * 0.5 - 2.75).astype(np.float32)
    um *= rng.random((B, I)) < density
    um[1, :] = 0.0                                # a user with no rated item -> all -inf row (:208-209)
    um[0, min(3, I - 1)] = 1.25                   # make sure the candidate's own rated entry is non-zero
    um[2, :min(4, I)] = 0.0                       # exact zeros = "unrated"
    return cand, rated, um


def golden_attention(ref):
    rng = np.random.default_rng(9)
    cases = {
        'attention_small_net': dict(item_dim=48, item_emb=16, user_emb=12, att_dense=16, mlp_dense_layers=[32, 16],
                                    dropout_rate=0.0, use_cos_sim_instead=False, message_dropout=None),
        'attention_small_lin': dict(item_dim=40, item_emb=8, user_emb=8, att_dense=None, mlp_dense_layers=[16],
                                    dropout_rate=0.0, use_cos_sim_instead=False, message_dropout=None),
        'attention_small_cos': dict(item_dim=40, item_emb=8, user_emb=8, att_dense=None, mlp_dense_layers=[16, 8],
                                    dropout_rate=0.0, use_cos_sim_instead=True, message_dropout=None),
    }
    for tag, kw in cases.items():
        wkw = {k: v for k, v in kw.items() if k not in ('use_cos_sim_instead', 'message_dropout')}
        sd = synth.attention_ncf_weights(seed=5, **wkw)
        m = ref.AttentionNCF(**kw)
        if kw['use_cos_sim_instead']:
            sd = {k: v for k, v in sd.items() if not k.startswith('AttentionNet')}
        m.load_state_dict(synth.to_torch(sd))
        cand, rated, um = _attention_inputs(rng, 21, 33, kw['item_dim'], 0.4)
        t = [torch.from_numpy(a) for a in (cand, rated, um)]
        with torch.no_grad():
            m.eval()
            out, att = m(*t, return_attention_weights=True)
            m.train()          # dropout_rate=0.0 / message_dropout=None: only the candidate mask differs
            out_tr, att_tr = m(*t, return_attention_weights=True)
        _save(tag, candidate_items=cand, rated_items=rated, user_matrix=um, out=out, att=att,
              out_train=out_tr, att_train=att_tr, kwargs=np.array(repr(kw)), **_sd_arrays(sd))
    # shipped-checkpoint shape (models/runs/*.pt kwargs), outputs only
    kw = dict(item_dim=2094, item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[256, 128],
              dropout_rate=0.2, use_cos_sim_instead=False, message_dropout=None)
    wkw = {k: v for k, v in kw.items() if k not in ('use_cos_sim_instead', 'message_dropout')}
    sd = synth.attention_ncf_weights(seed=13, **wkw)
    m = ref.AttentionNCF(**kw).eval()
    m.load_state_dict(synth.to_torch(sd))
    prof = synth.item_profiles(300 + 48, seed=201)
    cand, rated, um = _attention_inputs(np.random.default_rng(202), 48, 300, 2094, 0.25, profiles=prof)
    with torch.no_grad():
        out, att = m(torch.from_numpy(cand), torch.from_numpy(rated), torch.from_numpy(um), return_attention_weights=True)
    _save('attention_full', out=out, att=att, user_matrix=um, kwargs=np.array(repr(kw)),
          weight_seed=13, profile_seed=201, B=48, I=300)


# --------------------------------------------------------------------------------------------------
def _small_interactions(seed, n_users=40, n_items=60, n=700):
    rng = np.random.default_rng(seed)
    keys = rng.permutation(n_users * n_items)[:n]
    u = keys // n_items
    i = keys % n_items
    # raw ids: sparse and unsorted, so that the sorted-unique node-id map matters (graph_providers.py:76-80)
    user_raw = (u * 3 + 11).astype(np.int64)
    item_raw = (i * 5 + 2).astype(np.int64)
    r = rng.integers(1, 11, size=n) * 0.5
    return user_raw, item_raw, r


def golden_graph(ref):
    user_raw, item_raw, r = _small_interactions(21)
    # "all interactions" = these plus a few users/items that only exist outside the graph's file
    all_users = np.concatenate([user_raw, np.array([5, 500])])
    all_items = np.concatenate([item_raw, np.array([1, 999])])
    items_sorted = sorted(np.unique(all_items).tolist())
    users_sorted = sorted(np.unique(all_users).tolist())
    item_to_node = {i: k for k, i in enumerate(items_sorted)}
    user_to_node = {u: len(items_sorted) + k for k, u in enumerate(users_sorted)}
    nI, nU = len(items_sorted), len(users_sorted)
    df = pd.DataFrame({'userId': user_raw, 'movieId': item_raw, 'rating': r})
    rng = np.random.default_rng(22)
    Fi, Fu = 20, 24
    item_feat = rng.standard_normal((nI, Fi)).astype(np.float32)
    user_feat = rng.standard_normal((nU, Fu)).astype(np.float32)
    graphs = {}
    for binary in (False, True):
        g = ref.create_graph(df, torch.from_numpy(item_feat), torch.from_numpy(user_feat), item_to_node, user_to_node, binary)
        graphs[binary] = g
        pos = g.pos_df.reset_index()
        _save(f'graph_build_binary{int(binary)}', user_raw=user_raw, item_raw=item_raw, rating=r,
              all_users=all_users, all_items=all_items,
              user2item_edge_index=g.user2item_edge_index, item2user_edge_index=g.item2user_edge_index,
              user2item_edge_attr=g.user2item_edge_attr, item2user_edge_attr=g.item2user_edge_attr,
              pos_Id1=pos['Id1'].values, pos_Id2=pos['Id2'].values, pos_pos=pos['pos'].values)

    B = 50
    pick = rng.permutation(len(df))[:B]
    userIds = torch.tensor([user_to_node[u] for u in user_raw[pick]], dtype=torch.long)
    itemIds = torch.tensor([item_to_node[i] for i in item_raw[pick]], dtype=torch.long)
    variants = {
        'graph_ncf_hetero_mean': dict(num_gnn_layers=2, hetero=True, node_emb=16, mlp_dense_layers=[32, 16], concat=False),
        'graph_ncf_hetero_l3': dict(num_gnn_layers=3, hetero=True, node_emb=8, mlp_dense_layers=[16], concat=False),
        'graph_ncf_concat': dict(num_gnn_layers=2, hetero=True, node_emb=16, mlp_dense_layers=[32], concat=True),
        'graph_ncf_dot': dict(num_gnn_layers=2, hetero=True, node_emb=16, use_dot_product=True),
        'graph_ncf_homo': dict(num_gnn_layers=2, hetero=False, node_emb=16, mlp_dense_layers=[32, 16]),
        'graph_ncf_gat': dict(num_gnn_layers=2, hetero=True, node_emb=16, mlp_dense_layers=[32, 16], convType='LightGAT'),
        'graph_ncf_binary': dict(num_gnn_layers=2, hetero=True, node_emb=16, mlp_dense_layers=[32, 16]),
    }
    for tag, kw in variants.items():
        full = dict(item_dim=Fi, user_dim=Fu, dropout_rate=0.0, message_dropout=None, node_dropout=None, **kw)
        wkw = {k: v for k, v in full.items() if k not in ('message_dropout', 'node_dropout')}
        sd = synth.graph_ncf_weights(seed=31, **wkw)
        m = ref.GraphNCF(**full)
        m.load_state_dict(synth.to_torch(sd))
        g = graphs[tag == 'graph_ncf_binary']
        with torch.no_grad():
            m.eval()
            out = m(g, userIds, itemIds, 'cpu')
            extra = {}
            if tag != 'graph_ncf_binary':
                m.train()      # dropout 0 everywhere: only the target-edge masking (:314-320) differs
                extra['out_train_masked'] = m(g, userIds, itemIds, 'cpu', mask_targets=True)
                extra['out_train_unmasked'] = m(g, userIds, itemIds, 'cpu', mask_targets=False)
        _save(tag, out=out, userIds=userIds, itemIds=itemIds, item_features=item_feat, user_features=user_feat,
              kwargs=np.array(repr(full)), **extra, **_sd_arrays(sd))


# --------------------------------------------------------------------------------------------------
def golden_collate(ref):
    """DynamicProfilesProvider.collate_interacted_items on hand-built frames (its __init__ only reads .h5)."""
    rng = np.random.default_rng(41)
    n_items, n_users, F = 30, 12, 10
    item_ids = np.array([f'tt{1000 + 7 * k:07d}' for k in range(n_items)])
    metadata = pd.DataFrame(rng.random((n_items, F)), index=item_ids)
    rows = {}
    csr_ptr, csr_idx, csr_r, means = [0], [], [], []
    for u in range(n_users):
        k = int(rng.integers(2, 9))
        idx = np.sort(rng.permutation(n_items)[:k])
        rr = rng.integers(1, 11, size=k) * 0.5
        if u == 3:
            rr[:] = 3.0                   # mean 3.0 -> centre 2.75; no exact zero
        if u == 4:
            rr[:] = 2.5                   # mean 2.5 -> centre 2.5 -> every centred rating is exactly 0.0
        rows[100 + u] = {'rating': rr, 'movieId': item_ids[idx], 'meanRating': rr.mean(), 'numRatings': k}
        csr_idx += idx.tolist(); csr_r += rr.tolist(); csr_ptr.append(len(csr_idx)); means.append(rr.mean())
    user_ratings = pd.DataFrame.from_dict(rows, orient='index')
    prov = object.__new__(ref.DynamicProfilesProvider)
    prov.metadata, prov.user_ratings = metadata, user_ratings
    bu = np.array([0, 3, 4, 7, 7, 11, 2])
    bi = np.array([5, 0, 29, 12, 13, 1, 5])
    batch = [(100 + int(u), item_ids[int(i)], 3.5) for u, i in zip(bu, bi)]
    cand_ids, rated_ids, cand, rated, um, tgt = prov.collate_interacted_items(batch, for_ranking=False)
    rated_idx = np.array([int(np.where(item_ids == s)[0][0]) for s in rated_ids])
    _save('collate', profiles=metadata.values, row_ptr=np.array(csr_ptr), rated_idx=np.array(csr_idx),
          rated_rating=np.array(csr_r), mean_rating=np.array(means), batch_users=bu, batch_items=bi,
          rated_items_idx=rated_idx, candidate_items=cand, rated_items=rated, user_matrix=um)


def golden_ranking(ref):
    """RankingDataset.__getitem__ (datasets/base.py:57-78: np.random.choice with the 'sum_dynamic' weights) and BPR_loss (:97-98) of the
    unmodified reference on a hand-built frame (its __init__ only reads .h5).  Per access the legacy generator is seeded, the uniform it would
    produce next is recorded, it is re-seeded and the reference draws: the fixture holds (uniform, drawn negative) pairs."""
    import importlib
    base = importlib.import_module('neural_collaborative_filtering.datasets.base')
    rng = np.random.default_rng(77)
    n = 40
    rows = []
    for k in range(n):
        m = int(rng.integers(1, 80))
        ids = rng.choice(50_000, size=m, replace=False)
        r = rng.integers(0 if k % 6 == 0 else 1, 11, m) * 0.5
        if not r.any():
            r[0] = 2.0
        rows.append({'userId': int(rng.integers(0, 300)), 'positive_movieId': int(rng.integers(0, 50_000)),
                     'negative_movieIds': ids, 'negative_ratings': r})
    frame = pd.DataFrame(rows)
    ds = object.__new__(base.RankingDataset)
    ds.samples, ds.loss_fn = frame, base.BPR_loss
    ptr = np.concatenate([[0], np.cumsum([len(x) for x in frame['negative_movieIds']])])
    access = rng.integers(0, n, 600)
    out = {}
    for w in (0.0, 1.0, 2.5):
        ds.w = w
        us, negs = [], []
        for t, item in enumerate(access):
            np.random.seed(1000 + t)
            us.append(np.random.random_sample())
            np.random.seed(1000 + t)
            user, pos, neg = ds[int(item)]
            assert user == frame['userId'][int(item)] and pos == frame['positive_movieId'][int(item)]
            negs.append(int(neg))
        tag = str(w).replace('.', '_')
        out[f'uniform_w{tag}'], out[f'negative_w{tag}'] = np.array(us), np.array(negs, dtype=np.int64)
    a, b = torch.randn(50, 1), torch.randn(50, 1)
    _save('ranking_sampling', neg_ptr=ptr, neg_item=np.concatenate(list(frame['negative_movieIds'])).astype(np.int64),
          neg_rating=np.concatenate(list(frame['negative_ratings'])).astype(np.float64), user=frame['userId'].to_numpy(),
          positive=frame['positive_movieId'].to_numpy(), access=access, bpr_pos=a, bpr_neg=b, bpr_loss=ds.calculate_loss(a, b), **out)


def main():
    torch.manual_seed(0)
    torch.set_num_threads(1)      # deterministic reduction order for the stored fp32 outputs
    ref = ref_loader.load()
    only = sys.argv[1:]           # e.g. `python -m oracle.make_golden ranking`: regenerate one family, leave the other fixtures untouched
    for name, fn in (('basic', golden_basic), ('attention', golden_attention), ('graph', golden_graph), ('collate', golden_collate),
                     ('ranking', golden_ranking)):
        if not only or name in only:
            fn(ref)


if __name__ == '__main__':
    main()
