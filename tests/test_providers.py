"""Host-side logic that needs no GPU: the dynamic collate (a-8) against the reference's golden output, the datasets'
collate / do_forward contract, and checkpoint round trips with the reference's key names."""
import io

import numpy as np
import pandas as pd
import torch

from deeprecommendation_b200.content_providers import ArrayDynamicProvider, ArrayProfilesProvider
from deeprecommendation_b200.neural_collaborative_filtering.datasets.dynamic_datasets import DynamicPointwiseDataset
from deeprecommendation_b200.neural_collaborative_filtering.datasets.fixed_datasets import FixedPointwiseDataset
from deeprecommendation_b200.neural_collaborative_filtering.models import AttentionNCF, BasicNCF, GraphNCF
from deeprecommendation_b200.neural_collaborative_filtering.util import load_model
from tests._golden import load


def _provider(d):
    n_items, n_users = d['profiles'].shape[0], len(d['mean_rating'])
    return ArrayDynamicProvider(np.arange(n_items), d['profiles'], np.arange(n_users), d['row_ptr'], d['rated_idx'], d['rated_rating'])


def test_collate_bit_exact_vs_reference():
    d, _, _ = load('collate')
    p = _provider(d)
    assert np.array_equal(p.mean_rating, d['mean_rating'])
    batch = [(int(u), int(i), 3.5) for u, i in zip(d['batch_users'], d['batch_items'])]
    cand_ids, rated_ids, cand, rated, um, tgt = p.collate_interacted_items(batch, for_ranking=False)
    assert np.array_equal(rated_ids, d['rated_items_idx']) and np.array_equal(cand_ids, d['batch_items'])
    for got, key in ((cand, 'candidate_items'), (rated, 'rated_items'), (um, 'user_matrix')):
        assert got.dtype == torch.float32
        assert np.array_equal(got.numpy().view(np.int32), d[key].view(np.int32)), key
    assert tgt.tolist() == [3.5] * len(batch)
    # ranking form: the third element becomes the second candidate's profiles
    out = p.collate_interacted_items([(0, 1, 2), (3, 4, 5)], for_ranking=True)
    assert out[5].shape == (2, d['profiles'].shape[1])


def test_dataset_contract_with_dataloader():
    d, _, _ = load('collate')
    p = _provider(d)
    frame = pd.DataFrame({'userId': d['batch_users'], 'movieId': d['batch_items'], 'rating': np.linspace(1, 4, len(d['batch_users']))})
    ds = DynamicPointwiseDataset(frame, p)
    loader = torch.utils.data.DataLoader(ds, batch_size=4, collate_fn=ds.use_collate())
    batches = list(loader)
    assert len(batches) == 2 and len(batches[0]) == 6 and batches[0][4].shape[0] == 4
    calls = []

    class Probe(torch.nn.Module):
        def forward(self, cand, rated, um, return_attention_weights=False):
            calls.append((cand.dtype, cand.shape, rated.shape, um.shape))
            out = torch.zeros(cand.shape[0], 1)
            return (out, torch.zeros_like(um)) if return_attention_weights else out
    out, y = DynamicPointwiseDataset.do_forward(Probe(), batches[0], 'cpu')
    assert out.shape == (4, 1) and y.shape == (4,) and calls[0][0] == torch.float32
    res = DynamicPointwiseDataset.do_forward(Probe(), batches[0], 'cpu', return_attention_weights=True)
    assert len(res) == 6
    assert float(ds.calculate_loss(torch.ones(4, 1), torch.tensor([1., 2., 3., 4.]))) == 14.0    # MSE, reduction='sum'

    fp = ArrayProfilesProvider(np.arange(30), d['profiles'], np.arange(12), np.ones((12, 5)))
    fds = FixedPointwiseDataset(frame, fp)
    b = next(iter(torch.utils.data.DataLoader(fds, batch_size=3, collate_fn=fds.use_collate())))
    assert b[0].shape == (3, 5) and b[1].shape == (3, d['profiles'].shape[1]) and b[2].shape == (3,)


def test_compatibility_checks_and_hyperparams():
    from deeprecommendation_b200.neural_collaborative_filtering.datasets import fixed_datasets, dynamic_datasets, gnn_datasets
    b = BasicNCF(8, 8, item_emb=4, user_emb=4, mlp_dense_layers=[8])
    a = AttentionNCF(8, 4, 4, att_dense=4, mlp_dense_layers=[8])
    g = GraphNCF(8, 8, 2, True, node_emb=4, mlp_dense_layers=[8])
    assert b.is_dataset_compatible(fixed_datasets.FixedPointwiseDataset) and not b.is_dataset_compatible(dynamic_datasets.DynamicPointwiseDataset)
    assert a.is_dataset_compatible(dynamic_datasets.DynamicRankingDataset) and not a.is_dataset_compatible(gnn_datasets.GraphPointwiseDataset)
    assert g.is_dataset_compatible(gnn_datasets.GraphPointwiseDataset) and not g.is_dataset_compatible(fixed_datasets.FixedRankingDataset)
    assert a.important_hypeparams() == '_attNet4' and g.important_hypeparams() == '_LightGCN'
    assert AttentionNCF(8, 4, 4, use_cos_sim_instead=True).important_hypeparams() == '_cosine'
    assert g.gnn_convs[0] is g.gnn_convs[1]                    # one conv aliased L times (gnn_ncf.py:227)
    assert set(b.kwargs) == {'item_dim', 'user_dim', 'item_emb', 'user_emb', 'mlp_dense_layers', 'dropout_rate'}


def test_checkpoint_round_trip_and_reference_keys():
    _, sd, kw = load('attention_small_net')
    m = AttentionNCF(**kw)
    m.load_state_dict(sd)                                      # the reference's own key names
    buf = io.BytesIO()
    m.save_model(buf)
    buf.seek(0)
    m2 = load_model(buf, AttentionNCF, map_location='cpu')
    assert m2.kwargs == m.kwargs
    for (k1, v1), (k2, v2) in zip(m.state_dict().items(), m2.state_dict().items()):
        assert k1 == k2 and torch.equal(v1, v2)
    _, gsd, gkw = load('graph_ncf_hetero_l3')
    g = GraphNCF(**gkw)
    assert set(g.state_dict().keys()) == set(gsd.keys())
    g.load_state_dict(gsd)


def test_resident_provider_collate_equals_dense_collate():
    """device-resident form of the collate (row numbers + CSR) carries exactly the dense 6-tuple's information"""
    from deeprecommendation_b200.content_providers import ResidentDynamicProvider
    d, _, _ = load('collate')
    n_items, n_users = d['profiles'].shape[0], len(d['mean_rating'])
    args = (np.arange(n_items), d['profiles'], np.arange(n_users), d['row_ptr'], d['rated_idx'], d['rated_rating'])
    dense, res = ArrayDynamicProvider(*args), ResidentDynamicProvider(*args, device='cpu')
    batch = [(int(u), int(i), 3.5) for u, i in zip(d['batch_users'], d['batch_items'])]
    a = dense.collate_interacted_items(batch, for_ranking=False)
    b = res.collate_interacted_items(batch, for_ranking=False)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) and torch.equal(a[5], b[5])
    assert torch.equal(b[2].dense(), a[2]) and torch.equal(b[3].dense(), a[3])
    assert torch.equal(b[4].to_dense(), a[4])
    assert int((a[4] != 0).sum()) == b[4].col.numel()                     # exact zeros are absent from the CSR
    # the dataset hands the resident form to model.forward_resident
    seen = {}

    class Probe(torch.nn.Module):
        def forward_resident(self, cand, rated, um, return_attention_weights=False):
            seen['shapes'] = (len(cand), len(rated), um.shape)
            return torch.zeros(len(cand), 1)
    out, y = DynamicPointwiseDataset.do_forward(Probe(), b, 'cpu')
    assert out.shape == (len(batch), 1) and seen['shapes'] == (len(batch), a[3].shape[0], tuple(a[4].shape))


def test_sparse_row_containers_round_trip_and_take():
    """OneHotRows / MixedRows (the sparse forms of the fixed-profile collate contract) reproduce the dense rows they stand for"""
    from deeprecommendation_b200.content_providers import MixedProfilesProvider, MixedRows, OneHotArrayProvider, OneHotRows
    rng = np.random.default_rng(0)
    rows = np.concatenate([(rng.random((40, 30)) < 0.1).astype(np.float32), rng.random((40, 12)).astype(np.float32)], axis=1)
    rows[3, :30] = 0.0
    m = MixedRows.from_dense(rows, 30)
    assert m.val is None and m.shape == (40, 42) and np.array_equal(m.dense_rows().numpy(), rows)
    pick = np.array([5, 3, 39, 5])
    assert np.array_equal(m.take(pick).dense_rows().numpy(), rows[pick])
    weighted = rows.copy()
    weighted[:, :30] *= 2.5
    mw = MixedRows.from_dense(weighted, 30)
    assert mw.val is not None and np.array_equal(mw.dense_rows().numpy(), weighted)
    item_ids, user_ids = np.array([3, 8, 20, 41]), np.array([7, 9])
    sp, de = OneHotArrayProvider(item_ids, user_ids, sparse=True), OneHotArrayProvider(item_ids, user_ids, sparse=False)
    got = sp.get_item_profile(np.array([20, 3]))
    assert isinstance(got, OneHotRows) and got.float() is got and np.array_equal(got.dense().numpy(), de.get_item_profile(np.array([20, 3])))
    assert sp.get_item_feature_dim() == 4 and sp.get_num_users() == 2
    cp = MixedProfilesProvider(np.arange(40) * 3, rows, np.arange(5), rng.random((5, 42)).astype(np.float32), 30)
    assert np.array_equal(cp.get_item_profile(np.array([9, 0])).dense_rows().numpy(), rows[[3, 0]])


def test_model_hooks_empty_the_derived_stores():
    """load_state_dict / .to() / invalidate_caches() drop the derived copies of the weights (packed tiles, composites, cached embeddings) that are
    reused while the source tensor keeps its address and _version — an edit through `.data` changes neither"""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.neural_collaborative_filtering.models import AttentionNCF, GraphNCF
    ops_stores = (ops._pack_cache, ops._wt_cache, ops._ap_cache)

    def fill_ops_stores(w):
        ops._transposed_weight(w, 0, 4)
        ops._pack_cache.get((w,), lambda: torch.zeros(1), w.shape[1], 0)
        ops._ap_cache.get((w, None, None, None), lambda: torch.zeros(1), 64, 0)
        assert all(len(s) == 1 for s in ops_stores)

    a = AttentionNCF(8, 4, 4, att_dense=4, mlp_dense_layers=[8]).eval()
    with torch.no_grad():
        comp = a._composite_projection()
        assert a._composite_projection() is comp and len(a._comp_cache) == 1 and len(a._att_cache) == 1
        fill_ops_stores(a.ItemEmbeddings[0].weight)
    a.load_state_dict(a.state_dict())
    assert len(a._comp_cache) == 0 and len(a._att_cache) == 0 and all(len(s) == 0 for s in ops_stores)
    g = GraphNCF(8, 8, 2, True, node_emb=4, mlp_dense_layers=[8], cache_eval_embeddings=True)
    for drop in (g.double, g.invalidate_caches):
        with torch.no_grad():
            g._cache.get(tuple(g.parameters()), lambda: torch.zeros(1), g.message_dtype)
            fill_ops_stores(g.item_embeddings[0].weight)
        assert len(g._cache) == 1
        drop()
        assert len(g._cache) == 0 and all(len(s) == 0 for s in ops_stores)
