"""End-to-end parity of the three model classes (the drop-in seam, SURVEY.md §8b) on a B200: CUDA path through the
C ABI vs (1) golden outputs of the UNMODIFIED reference (tests/golden, made by oracle/make_golden.py) and (2) the CPU
oracle restatement on larger seeded inputs.  fp32 tolerance: max-norm relative error <= 1e-5 (north_star)."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from oracle import synth
from tests._golden import load, maxnorm_rel
from tests.test_oracle import GRAPH_CASES, attention_full_inputs

pytestmark = pytest.mark.gpu
TOL = 1e-5
DEV = 'cuda:0'


def _models():
    from deeprecommendation_b200.neural_collaborative_filtering import models
    return models


def _cuda(sd):
    return {k: v.to(DEV) for k, v in sd.items()}


# ---- BasicNCF -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['basic_small_a', 'basic_small_b', 'basic_small_c'])
def test_basic_small_vs_reference(name):
    d, sd, kw = load(name)
    m = _models().BasicNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)                       # reference key names load unchanged
    with torch.no_grad():
        out = m(torch.from_numpy(d['X_user']).to(DEV), torch.from_numpy(d['X_item']).to(DEV))
    assert out.shape == (37, 1) and out.device.type == 'cuda'
    assert maxnorm_rel(out, d['out']) < TOL


@pytest.mark.parametrize('name', ['basic_full_256', 'basic_full_256_128'])
def test_basic_full_vs_reference(name):
    d, _, kw = load(name)
    sd = synth.to_torch(synth.basic_ncf_weights(seed=int(d['weight_seed']), **kw))
    m = _models().BasicNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    B = int(d['B'])
    xi = torch.from_numpy(synth.item_profiles(B, seed=int(d['item_seed']))).to(DEV)
    xu = torch.from_numpy((synth.item_profiles(B, seed=int(d['user_seed'])) - 0.25) * 0.125).to(DEV)
    with torch.no_grad():
        out = m(xu, xi)
    assert maxnorm_rel(out, d['out']) < TOL


def test_basic_cfg1_batches_vs_oracle():
    """BASELINE config 1 shape: F=2094 dense profiles, emb 128, batches of 512 (train_model.py:38-42)."""
    kw = dict(item_dim=2094, user_dim=2094, item_emb=128, user_emb=128, mlp_dense_layers=[256], dropout_rate=0.2)
    sd = synth.to_torch(synth.basic_ncf_weights(seed=1, **kw))
    m = _models().BasicNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    items = synth.item_profiles(2048, seed=7)
    users = (synth.item_profiles(2048, seed=8) - 0.3) * 0.1
    for B in (1, 127, 512, 2048):
        xu, xi = torch.from_numpy(users[:B]), torch.from_numpy(items[:B])
        ref = R.basic_ncf_forward(sd, xu, xi)
        with torch.no_grad():
            out = m(xu.to(DEV), xi.to(DEV))
        assert maxnorm_rel(out, ref) < TOL


def test_basic_resident_profiles_through_the_dataset_contract_and_embedding_store():
    """ResidentProfilesProvider (both profile tables in HBM, batches = row numbers) through FixedPointwiseDataset / FixedRankingDataset:
    identical bits to the dense contract; with cached per-row embeddings within 1e-5 of the oracle; training falls back to dense rows."""
    import pandas as pd
    from deeprecommendation_b200.content_providers import ArrayProfilesProvider, ResidentProfilesProvider
    from deeprecommendation_b200.neural_collaborative_filtering.datasets.fixed_datasets import FixedPointwiseDataset, FixedRankingDataset
    kw = dict(item_dim=2094, user_dim=2094, item_emb=128, user_emb=128, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    sd = synth.to_torch(synth.basic_ncf_weights(seed=3, **kw))
    m = _models().BasicNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    nI, nU, B = 700, 90, 300
    items = synth.item_profiles(nI, seed=11)
    users = ((synth.item_profiles(nU, seed=12) - 0.3) * 0.1).astype(np.float32)
    item_ids, user_ids = np.arange(nI) * 3 + 5, np.arange(nU) * 7 + 1
    rng = np.random.default_rng(0)
    pu, pi, pj = rng.integers(0, nU, B), rng.integers(0, nI, B), rng.integers(0, nI, B)
    frame = pd.DataFrame({'userId': user_ids[pu], 'movieId': item_ids[pi], 'rating': rng.integers(1, 11, B) * 0.5})
    dense_p, res_p = ArrayProfilesProvider(item_ids, items, user_ids, users), ResidentProfilesProvider(item_ids, items, user_ids, users, device=DEV)
    outs = {}
    for name, prov in (('dense', dense_p), ('resident', res_p)):
        ds = FixedPointwiseDataset(frame, prov)
        batch = next(iter(torch.utils.data.DataLoader(ds, batch_size=B, collate_fn=ds.use_collate())))
        with torch.no_grad():
            outs[name], y = FixedPointwiseDataset.do_forward(m, batch, DEV)
        assert y.shape == (B,)
    assert torch.equal(outs['dense'], outs['resident'])
    ref = R.basic_ncf_forward(sd, torch.from_numpy(users[pu]), torch.from_numpy(items[pi]))
    assert maxnorm_rel(outs['resident'], ref) < TOL
    m.cache_eval_embeddings = True
    ds = FixedPointwiseDataset(frame, res_p)
    batch = next(iter(torch.utils.data.DataLoader(ds, batch_size=B, collate_fn=ds.use_collate())))
    with torch.no_grad():
        cached, _ = FixedPointwiseDataset.do_forward(m, batch, DEV)
        assert maxnorm_rel(cached, ref) < TOL
        (first,) = m._emb_cache.values()
        assert first[0].shape == (nU, 128) and first[1].shape == (nI, 128)
        FixedPointwiseDataset.do_forward(m, batch, DEV)
        assert m._emb_cache.values()[0] is first                       # reused while the weights are unchanged
        m.load_state_dict(sd)
        assert len(m._emb_cache) == 0                                  # dropped with the weights
        # ranking form: (user, positive, negative) rows, two scores per sample
        trip = (res_p.get_user_profile(user_ids[pu]), res_p.get_item_profile(item_ids[pi]), res_p.get_item_profile(item_ids[pj]))
        pos, neg = FixedRankingDataset.do_forward(m, trip, DEV)
        assert maxnorm_rel(pos, ref) < TOL
        assert maxnorm_rel(neg, R.basic_ncf_forward(sd, torch.from_numpy(users[pu]), torch.from_numpy(items[pj]))) < TOL
    m.train()
    out = FixedPointwiseDataset.do_forward(m, batch, DEV)[0]
    out.sum().backward()
    assert torch.isfinite(m.user_embeddings[0].weight.grad).all()


def test_basic_cached_embeddings_of_a_new_provider_at_the_old_addresses():
    """cache_eval_embeddings: a provider dropped and rebuilt with other tables of the same size, which the caching allocator places at the
    freed addresses (with `_version` 0 again), gets its own embeddings and not the old tables' cached ones"""
    from deeprecommendation_b200.content_providers import ResidentProfilesProvider
    kw = dict(item_dim=2094, user_dim=2094, item_emb=128, user_emb=128, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    m = _models().BasicNCF(**kw).to(DEV).eval()
    m.load_state_dict(synth.to_torch(synth.basic_ncf_weights(seed=3, **kw)))
    nI, nU, B = 700, 90, 300
    rng = np.random.default_rng(1)
    pu, pi = rng.integers(0, nU, B), rng.integers(0, nI, B)

    def provider(seed):
        users = ((synth.item_profiles(nU, seed=seed) - 0.3) * 0.1).astype(np.float32)
        return ResidentProfilesProvider(np.arange(nI), synth.item_profiles(nI, seed=seed + 1), np.arange(nU), users, device=DEV)

    def run(prov, cached):
        m.cache_eval_embeddings = cached
        with torch.no_grad():
            return m(prov.get_user_profile(pu), prov.get_item_profile(pi))
    prov = provider(11)
    addresses = (prov.user_table.data_ptr(), prov.item_table.data_ptr())
    run(prov, True)
    del prov
    prov = provider(21)
    if (prov.user_table.data_ptr(), prov.item_table.data_ptr()) != addresses:
        pytest.skip('the caching allocator placed the new tables elsewhere')
    assert prov.user_table._version == prov.item_table._version == 0
    cached = run(prov, True)
    assert maxnorm_rel(cached, run(prov, False)) < TOL


def test_graph_cached_embeddings_of_a_new_graph():
    """cache_eval_embeddings=True: graph A freed, then a graph object of other edges with the same sizes built (CPython tends to give it and its
    index the freed objects' `id`s) gets its own propagated embeddings"""
    from deeprecommendation_b200.graph import GraphData, IdTable, create_graph, get_index
    n_users, n_items, n, F = 400, 300, 8000, 32
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=2, hetero=True, node_emb=64, mlp_dense_layers=[128], dropout_rate=0.2)
    m = _models().GraphNCF(**kw, cache_eval_embeddings=True).to(DEV).eval()
    m.load_state_dict(synth.to_torch(synth.graph_ncf_weights(seed=8, **kw)))
    rng = np.random.default_rng(3)
    fi, fu = (torch.from_numpy(rng.standard_normal((k, F)).astype(np.float32)).to(DEV) for k in (n_items, n_users))
    ut, it = IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV))
    iid = torch.from_numpy(rng.integers(0, n_items, 128)).to(DEV)
    uid = torch.from_numpy(rng.integers(0, n_users, 128) + n_items).to(DEV)

    def graph(seed):
        users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=seed)
        return create_graph(*(torch.from_numpy(a).to(DEV) for a in (users, items, ratings)), fi, fu, ut, it)
    g = graph(7)
    with torch.no_grad():
        m(g, uid, iid, DEV)
    index_id = id(get_index(g))
    edges_b = vars(graph(17))
    del g
    g = GraphData(**edges_b)
    with torch.no_grad():
        cached = m(g, uid, iid, DEV)
        print(f'the new graph index took the freed one\'s id: {id(get_index(g)) == index_id}')
        m.cache_eval_embeddings = False
        assert torch.equal(cached, m(g, uid, iid, DEV))


# ---- AttentionNCF ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('name', ['attention_small_net', 'attention_small_lin', 'attention_small_cos'])
def test_attention_small_vs_reference(name):
    d, sd, kw = load(name)
    m = _models().AttentionNCF(**kw).to(DEV)
    m.load_state_dict(sd)
    t = [torch.from_numpy(d[k]).to(DEV) for k in ('candidate_items', 'rated_items', 'user_matrix')]
    with torch.no_grad():
        m.eval()
        out, att = m(*t, return_attention_weights=True)
        out_only = m(*t)
        m.train()                 # dropout_rate=0.0, message_dropout=None: only the isclose() candidate mask differs
        out_tr, att_tr = m(*t, return_attention_weights=True)
    assert maxnorm_rel(out, d['out']) < TOL and maxnorm_rel(att, d['att']) < TOL
    assert torch.equal(out_only, out)
    assert torch.all(att[1] == 0) and torch.all(att[d['user_matrix'] == 0] == 0)
    assert maxnorm_rel(out_tr, d['out_train']) < TOL and maxnorm_rel(att_tr, d['att_train']) < TOL
    assert att_tr[0, 3] == 0 and att[0, 3] > 0


def test_attention_full_vs_reference():
    d, _, kw = load('attention_full')
    wkw = {k: v for k, v in kw.items() if k not in ('use_cos_sim_instead', 'message_dropout')}
    sd = synth.to_torch(synth.attention_ncf_weights(seed=int(d['weight_seed']), **wkw))
    m = _models().AttentionNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    cand, rated, um = attention_full_inputs(d)
    with torch.no_grad():
        out, att = m(torch.from_numpy(cand).to(DEV), torch.from_numpy(rated).to(DEV), torch.from_numpy(um).to(DEV),
                     return_attention_weights=True)
    assert maxnorm_rel(out, d['out']) < TOL and maxnorm_rel(att, d['att']) < TOL
    rows = torch.from_numpy((um != 0).any(1))
    assert torch.allclose(att.sum(1).cpu()[rows], torch.ones(int(rows.sum())), atol=1e-5)


def _cfg2_batch(B, n_items, seed, max_len=2698):
    """ragged rated lists, mean ~165 / heavy tail, as a dense (B, I) user_matrix over the batch's item union"""
    rng = np.random.default_rng(seed)
    lens = np.clip(rng.lognormal(4.6, 1.0, size=B).astype(int), 1, min(max_len, n_items))
    lens[0], lens[1] = min(max_len, n_items), 0          # the longest list and an empty one
    um = np.zeros((B, n_items), dtype=np.float32)
    for b in range(B):
        cols = rng.choice(n_items, size=lens[b], replace=False)
        um[b, cols] = rng.integers(1, 11, size=lens[b]) * 0.5 - 2.75
    used = np.flatnonzero((um != 0).any(0))
    return um[:, used], used


def test_attention_cfg2_ragged_vs_oracle():
    """BASELINE config 2 shape (F=2094, 128/128/128, [256,128]); ragged lists up to ~2.7k, dense and CSR front-ends"""
    from deeprecommendation_b200 import ops
    kw = dict(item_dim=2094, item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    sd = synth.to_torch(synth.attention_ncf_weights(seed=3, **kw))
    m = _models().AttentionNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    B, n_items = 96, 3000
    um, used = _cfg2_batch(B, n_items, seed=11)
    prof = synth.item_profiles(n_items + B, seed=12)
    rated, cand = torch.from_numpy(prof[used]), torch.from_numpy(prof[n_items:])
    umt = torch.from_numpy(um)
    ref_out, ref_att = R.attention_ncf_forward_blocked(sd, cand, rated, umt, block=16, return_attention_weights=True)
    with torch.no_grad():
        out, att = m(cand.to(DEV), rated.to(DEV), umt.to(DEV), return_attention_weights=True)
    assert maxnorm_rel(out, ref_out) < TOL and maxnorm_rel(att, ref_att) < TOL
    # the ragged-native (CSR) entry gives the same user embeddings as the dense drop-in entry
    E = 128
    with torch.no_grad():
        Ec = ops.linear_raw(cand.to(DEV), m.ItemEmbeddings[0].weight, m.ItemEmbeddings[0].bias)
        Er = ops.linear_raw(rated.to(DEV), m.ItemEmbeddings[0].weight, m.ItemEmbeddings[0].bias)
        Q = ops.linear_raw(rated.to(DEV), m.UserEmbeddings[0].weight, None)
        A1 = m.AttentionNet[0].weight
        Pc = ops.linear_raw(Ec, A1[:, :E], m.AttentionNet[0].bias)
        Pr = ops.linear_raw(Er, A1[:, E:], None)
        common = dict(mode=0, a2=m.AttentionNet[3].weight, a20=m.AttentionNet[3].bias, bU=m.UserEmbeddings[0].bias)
        dense = ops.attention_pool_raw(Pc, Pr, Q, user_matrix=umt.to(DEV), **common)
        nz = umt != 0
        row_ptr = torch.cat((torch.zeros(1, dtype=torch.int64), nz.sum(1).cumsum(0))).int()
        col = nz.nonzero()[:, 1].int()
        csr = ops.attention_pool_raw(Pc, Pr, Q, csr=(row_ptr.to(DEV), col.to(DEV), umt[nz].to(DEV)), **common)
        assert maxnorm_rel(csr, dense) < 1e-6      # same core; the warps slice the row by column (dense) vs by non-zero count (CSR)
        # single fused kernel (no workspace) vs segment-parallel path (compaction + one CTA per 512 non-zeros + merge)
        fused_d = ops.attention_pool_raw(Pc, Pr, Q, user_matrix=umt.to(DEV), use_workspace=False, **common)
        fused_c = ops.attention_pool_raw(Pc, Pr, Q, csr=(row_ptr.to(DEV), col.to(DEV), umt[nz].to(DEV)), use_workspace=False, **common)
        assert maxnorm_rel(fused_d, dense) < 1e-6 and maxnorm_rel(fused_c, dense) < 1e-6
        o1, a1 = ops.attention_pool_raw(Pc, Pr, Q, user_matrix=umt.to(DEV), return_attention_weights=True, use_workspace=False, **common)
        o2, a2 = ops.attention_pool_raw(Pc, Pr, Q, csr=(row_ptr.to(DEV), col.to(DEV), umt[nz].to(DEV)), return_attention_weights=True, **common)
        assert maxnorm_rel(a1, att) < 1e-5 and maxnorm_rel(a2, att) < 1e-5
        bf = ops.attention_pool_raw(Pc, Pr.bfloat16(), Q.bfloat16(), user_matrix=umt.to(DEV), **common)
        assert maxnorm_rel(bf, dense) < 1e-2                                  # bf16 tables, fp32 accumulate
        # the same segments with the rows staged by TMA bulk copies (the path big tables take): same arithmetic, same order
        csr_args = (row_ptr.to(DEV), col.to(DEV), umt[nz].to(DEV))
        ops.set_attention_path('tma')
        try:
            t_dense = ops.attention_pool_raw(Pc, Pr, Q, user_matrix=umt.to(DEV), **common)
            t_csr, t_att = ops.attention_pool_raw(Pc, Pr, Q, csr=csr_args, return_attention_weights=True,
                                                  max_row_nnz=int(nz.sum(1).max()), **common)
            t_bf = ops.attention_pool_raw(Pc, Pr.bfloat16(), Q.bfloat16(), csr=csr_args, **common)
            t_hint = ops.attention_pool_raw(Pc, Pr, Q, csr=csr_args, max_row_nnz=7, **common)          # nnz is known from the CSR: a wrong hint is ignored
        finally:
            ops.set_attention_path('auto')
        assert torch.equal(t_dense, dense) and torch.equal(t_csr, csr) and torch.equal(t_hint, csr)
        assert maxnorm_rel(t_att, att) < 1e-5 and maxnorm_rel(t_bf, dense) < 1e-2


def test_attention_webapp_pattern_vs_oracle():
    """webapp/backend.py:78-99: one user, every candidate shares the same rated list"""
    kw = dict(item_dim=256, item_emb=64, user_emb=64, att_dense=64, mlp_dense_layers=[128, 64], dropout_rate=0.2)
    sd = synth.to_torch(synth.attention_ncf_weights(seed=4, **kw))
    m = _models().AttentionNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    prof = synth.item_profiles(1200, seed=5, f_binary=128, f_dense=128)
    rated, cand = torch.from_numpy(prof[:40]), torch.from_numpy(prof[40:])
    row = np.random.default_rng(6).integers(1, 11, size=40) * 0.5 - 2.9
    um = torch.from_numpy(np.repeat(row[None, :], cand.shape[0], 0).astype(np.float32))
    ref, ref_att = R.attention_ncf_forward_blocked(sd, cand, rated, um, block=128, return_attention_weights=True)
    with torch.no_grad():
        out, att = m(cand.to(DEV), rated.to(DEV), um.to(DEV), return_attention_weights=True)
    assert maxnorm_rel(out, ref) < TOL and maxnorm_rel(att, ref_att) < TOL


# ---- GraphNCF ------------------------------------------------------------------------------------------------------------
def _graph_from_golden(build, d):
    from deeprecommendation_b200.graph import GraphData
    g = GraphData(item_features=torch.from_numpy(d['item_features']), user_features=torch.from_numpy(d['user_features']),
                  user2item_edge_index=torch.from_numpy(build['user2item_edge_index']),
                  item2user_edge_index=torch.from_numpy(build['item2user_edge_index']),
                  user2item_edge_attr=torch.from_numpy(build['user2item_edge_attr']) if 'user2item_edge_attr' in build else None,
                  item2user_edge_attr=torch.from_numpy(build['item2user_edge_attr']) if 'item2user_edge_attr' in build else None)
    return g.to(DEV)


@pytest.mark.parametrize('name', GRAPH_CASES)
def test_graph_ncf_vs_reference(name):
    d, sd, kw = load(name)
    build, _, _ = load('graph_build_binary1' if name == 'graph_ncf_binary' else 'graph_build_binary0')
    g = _graph_from_golden(build, d)
    m = _models().GraphNCF(**kw).to(DEV)
    m.load_state_dict(sd)                       # aliased gnn_convs.{k}.* keys load as in the reference
    uid, iid = torch.from_numpy(d['userIds']).to(DEV), torch.from_numpy(d['itemIds']).to(DEV)
    with torch.no_grad():
        m.eval()
        out = m(g, uid, iid, DEV)
        assert maxnorm_rel(out, d['out']) < TOL
        if 'out_train_masked' in d:
            m.train()             # every dropout is 0: only the target-edge masking differs (gnn_ncf.py:314-320)
            assert maxnorm_rel(m(g, uid, iid, DEV, mask_targets=True), d['out_train_masked']) < TOL
            assert maxnorm_rel(m(g, uid, iid, DEV, mask_targets=False), d['out_train_unmasked']) < TOL
    if 'out_train_masked' in d and name != 'graph_ncf_gat':   # the autograd path runs the same kernels (LightGAT: forward only)
        m.train()
        assert maxnorm_rel(m(g, uid, iid, DEV, mask_targets=True), d['out_train_masked']) < TOL


def test_graph_ncf_gat_medium_vs_oracle():
    """LightGAT edge softmax over rows far longer than one SpMM chunk (multi-chunk merge of the softmax state)"""
    from deeprecommendation_b200.graph import IdTable, create_graph
    n_users, n_items, n, F, d_emb = 800, 300, 60_000, 32, 64
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=5)
    rng = np.random.default_rng(3)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=2, hetero=True, node_emb=d_emb, mlp_dense_layers=[64], dropout_rate=0.2, convType='LightGAT')
    sd = synth.to_torch(synth.graph_ncf_weights(seed=4, **kw))
    ref_g = R.create_graph(users, items, ratings, np.arange(n_users), np.arange(n_items))
    gd = {k: (torch.from_numpy(v) if v is not None else None) for k, v in ref_g.items()}
    gd['item_features'], gd['user_features'] = torch.from_numpy(fi), torch.from_numpy(fu)
    pick = rng.permutation(n)[:256]
    uid, iid = torch.from_numpy(ref_g['user2item_edge_index'][0][pick]), torch.from_numpy(ref_g['user2item_edge_index'][1][pick])
    ref = R.graph_ncf_forward(sd, gd, uid, iid, 2, convType='LightGAT')
    ref_masked = R.graph_ncf_forward(sd, gd, uid, iid, 2, convType='LightGAT', masked_positions=torch.from_numpy(pick))
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV),
                     IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV)))
    m = _models().GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    with torch.no_grad():
        assert maxnorm_rel(m(g, uid.to(DEV), iid.to(DEV), DEV), ref) < TOL
        m.train()
        for mod in m.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
        assert maxnorm_rel(m(g, uid.to(DEV), iid.to(DEV), DEV, mask_targets=True), ref_masked) < TOL


@pytest.mark.parametrize('conv', ['LightGCN', 'LightGAT'])
def test_graph_ncf_long_rows_cta_fixup_on_a_16_edge_chunk_index_vs_oracle(conv):
    """rows cut into MORE than 64 chunks (the CTA-cooperative branch of spmm_fixup_kernel): index built with 16-edge chunks, so
    that the hot items of a small Zipf graph own hundreds of partial slots"""
    from deeprecommendation_b200.derived import Derived
    from deeprecommendation_b200.graph import GraphIndex, IdTable, create_graph, get_index
    n_users, n_items, n, F, d_emb = 2500, 120, 60_000, 24, 64
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=15)
    rng = np.random.default_rng(8)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=2, hetero=True, node_emb=d_emb, mlp_dense_layers=[64], dropout_rate=0.2, convType=conv)
    sd = synth.to_torch(synth.graph_ncf_weights(seed=14, **kw))
    ref_g = R.create_graph(users, items, ratings, np.arange(n_users), np.arange(n_items))
    gd = {k: (torch.from_numpy(v) if v is not None else None) for k, v in ref_g.items()}
    gd['item_features'], gd['user_features'] = torch.from_numpy(fi), torch.from_numpy(fu)
    pick = rng.permutation(n)[:128]
    uid, iid = torch.from_numpy(ref_g['user2item_edge_index'][0][pick]), torch.from_numpy(ref_g['user2item_edge_index'][1][pick])
    ref = R.graph_ncf_forward(sd, gd, uid, iid, 2, convType=conv)
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV),
                     IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV)))
    idx = GraphIndex(g.user2item_edge_index, g.item2user_edge_index, g.user2item_edge_attr, g.item2user_edge_attr, n_users + n_items, chunk=16)
    assert int(idx.row_ptr.diff().max()) > 64 * 16                      # some row really takes the long-row branch
    store = Derived(1)                                                  # what get_index caches on the graph
    store.get((g.user2item_edge_index, g.item2user_edge_index, g.user2item_edge_attr, g.item2user_edge_attr), lambda: idx, n_users + n_items)
    object.__setattr__(g, '_b200rec_index', store)
    assert get_index(g) is idx
    m = _models().GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    with torch.no_grad():
        out = m(g, uid.to(DEV), iid.to(DEV), DEV)
        assert maxnorm_rel(out, ref) < TOL
        assert torch.equal(out, m(g, uid.to(DEV), iid.to(DEV), DEV))


def test_graph_ncf_missing_target_edge_raises_keyerror():
    d, sd, kw = load('graph_ncf_hetero_mean')
    build, _, _ = load('graph_build_binary0')
    g = _graph_from_golden(build, d)
    m = _models().GraphNCF(**kw).to(DEV).train()
    m.load_state_dict(sd)
    u2i = set(zip(build['user2item_edge_index'][0].tolist(), build['user2item_edge_index'][1].tolist()))
    nI = d['item_features'].shape[0]
    u, i = next((u, i) for u in range(nI, nI + 5) for i in range(nI) if (u, i) not in u2i)
    with pytest.raises(KeyError):
        m(g, torch.tensor([u], device=DEV), torch.tensor([i], device=DEV), DEV)


@pytest.mark.parametrize('d_emb,L_,n_users,n_items,n', [(128, 2, 3000, 1500, 150_000), (64, 3, 2000, 4000, 120_000)])
def test_graph_ncf_medium_vs_oracle(d_emb, L_, n_users, n_items, n):
    """heavy-tailed degrees (rows far longer than one SpMM chunk), zero-degree items, both reference hyper-parameter sets"""
    from deeprecommendation_b200.graph import IdTable, create_graph
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=9)
    F = 96
    rng = np.random.default_rng(1)
    item_feat = rng.standard_normal((n_items, F)).astype(np.float32)
    user_feat = rng.standard_normal((n_users, F)).astype(np.float32)
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=L_, hetero=True, node_emb=d_emb, mlp_dense_layers=[256, 128] if d_emb == 128 else [128],
              dropout_rate=0.2)
    sd = synth.to_torch(synth.graph_ncf_weights(seed=2, **kw))
    all_u, all_i = np.arange(n_users), np.arange(n_items)
    ref_g = R.create_graph(users, items, ratings, all_u, all_i)
    gd = {k: (torch.from_numpy(v) if v is not None else None) for k, v in ref_g.items()}
    gd['item_features'], gd['user_features'] = torch.from_numpy(item_feat), torch.from_numpy(user_feat)
    pick = rng.permutation(n)[:512]
    uid = torch.from_numpy(ref_g['user2item_edge_index'][0][pick])
    iid = torch.from_numpy(ref_g['user2item_edge_index'][1][pick])
    ref = R.graph_ncf_forward(sd, gd, uid, iid, L_)
    ref_masked = R.graph_ncf_forward(sd, gd, uid, iid, L_, masked_positions=torch.from_numpy(pick))
    ut, it = IdTable(torch.from_numpy(all_u).to(DEV)), IdTable(torch.from_numpy(all_i).to(DEV))
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(item_feat).to(DEV), torch.from_numpy(user_feat).to(DEV), ut, it)
    m = _models().GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    with torch.no_grad():
        out = m(g, uid.to(DEV), iid.to(DEV), DEV)
        assert maxnorm_rel(out, ref) < TOL
        assert torch.equal(out, m(g, uid.to(DEV), iid.to(DEV), DEV))            # deterministic: no atomics in K3
        m.message_dtype = 'bf16'                                                # bf16 message table, fp32 accumulate: rel <= 1e-2
        out_bf = m(g, uid.to(DEV), iid.to(DEV), DEV)
        assert maxnorm_rel(out_bf, ref) < 1e-2 and not torch.equal(out_bf, out)
        m.message_dtype = 'fp32'
        m.train()
        for mod in m.modules():
            if isinstance(mod, torch.nn.Dropout):
                mod.p = 0.0
        assert maxnorm_rel(m(g, uid.to(DEV), iid.to(DEV), DEV, mask_targets=True), ref_masked) < TOL


# ---- backward (interim torch recompute + CUDA SpMM transpose) ------------------------------------------------------------------
def test_gradients_vs_oracle_autograd():
    d, sd, kw = load('graph_ncf_hetero_mean')
    build, _, _ = load('graph_build_binary0')
    g = _graph_from_golden(build, d)
    m = _models().GraphNCF(**kw).to(DEV).train()
    m.load_state_dict(sd)
    uid, iid = torch.from_numpy(d['userIds']), torch.from_numpy(d['itemIds'])
    m(g, uid.to(DEV), iid.to(DEV), DEV, mask_targets=False).square().sum().backward()
    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    # aliases of the shared conv must be ONE leaf, as in the reference (gnn_ncf.py:227)
    for k in list(ref_sd):
        if k.startswith('gnn_convs.1.'):
            ref_sd[k] = ref_sd[k.replace('gnn_convs.1.', 'gnn_convs.0.')]
    gd = {k: torch.from_numpy(build[k]) for k in ('user2item_edge_index', 'item2user_edge_index', 'user2item_edge_attr', 'item2user_edge_attr')}
    gd['item_features'], gd['user_features'] = torch.from_numpy(d['item_features']), torch.from_numpy(d['user_features'])
    R.graph_ncf_forward(ref_sd, gd, uid, iid, kw['num_gnn_layers']).square().sum().backward()
    got = dict(m.named_parameters())
    for k in ('item_embeddings.0.weight', 'user_embeddings.0.bias', 'gnn_convs.0.user2item_W.0.weight', 'gnn_convs.0.item2user_W.0.bias',
              'MLP.0.weight', 'MLP.6.bias'):
        assert maxnorm_rel(got[k].grad, ref_sd[k].grad) < 1e-4, k

    da, sda, kwa = load('attention_small_net')
    ma = _models().AttentionNCF(**kwa).to(DEV).train()
    ma.load_state_dict(sda)
    t = [torch.from_numpy(da[k]) for k in ('candidate_items', 'rated_items', 'user_matrix')]
    ma(*[x.to(DEV) for x in t]).square().sum().backward()
    ref_a = {k: v.clone().requires_grad_(True) for k, v in sda.items()}
    R.attention_ncf_forward(ref_a, *t, training=True).square().sum().backward()
    scale = max(float(v.grad.abs().max()) for v in ref_a.values())
    for k, p in ma.named_parameters():
        # AttentionNet.3.bias shifts every score of a row equally: its true gradient is 0 (softmax shift invariance)
        assert float((p.grad.cpu() - ref_a[k].grad).abs().max()) < 1e-4 * max(float(ref_a[k].grad.abs().max()), 1e-4 * scale), k


# ---- multi-GPU partition, exercised on one GPU ---------------------------------------------------------------------------------
def _medium_graph(n_users=1500, n_items=900, n=60_000, F=48, d_emb=64, L_=2):
    from deeprecommendation_b200.graph import IdTable, create_graph
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=13)
    rng = np.random.default_rng(2)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=L_, hetero=True, node_emb=d_emb, mlp_dense_layers=[128], dropout_rate=0.2)
    sd = synth.to_torch(synth.graph_ncf_weights(seed=3, **kw))
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV),
                     IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV)))
    m = _models().GraphNCF(**kw).to(DEV).eval()
    m.load_state_dict(sd)
    pick = rng.permutation(n)[:300]
    return m, g, g.user2item_edge_index[0][pick].contiguous(), g.user2item_edge_index[1][pick].contiguous()


def test_partitioned_world1_equals_single():
    from deeprecommendation_b200.parallel import PartitionedGraph, UserPartitionedGraph, forward_partitioned
    m, g, uid, iid = _medium_graph()
    with torch.no_grad():
        ref = m(g, uid, iid, DEV)
        for cls in (PartitionedGraph, UserPartitionedGraph):
            out = forward_partitioned(m, cls(g, rank=0, world=1), uid, iid)
            assert maxnorm_rel(out, ref) < 1e-6


@pytest.mark.parametrize('P', [2, 3, 8])
def test_partition_emulated_ranks_on_one_gpu(P):
    """P emulated ranks share one GPU and one pair of gather buffers (so the all-gathers are the identity): checks the
    per-type nnz-balanced split, the slot addressing of `col`, the per-rank chunk plans and `locate` with the real kernels."""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.graph import get_index
    from deeprecommendation_b200.parallel import PartitionedGraph
    m, g, uid, iid = _medium_graph()
    full = get_index(g)
    L_, d = len(m.gnn_convs), 64
    ranks = [PartitionedGraph(g, rank=r, world=P) for r in range(P)]
    assert sum(pg.edges_own for pg in ranks) == full.e1 + full.e2
    assert max(pg.edges_own for pg in ranks) <= (full.e1 + full.e2) / P + 2 * int(full.deg.max())
    ie, ue = m.item_embeddings[0], m.user_embeddings[0]
    lin_u, lin_i, _ = m.gnn_convs[0].typed()
    TI, TU = ranks[0].gather_buffers(d, DEV)
    mi, mu = ranks[0].items.max_rows, ranks[0].users.max_rows
    with torch.no_grad():
        xs, accs = [], []
        for pg in ranks:
            ni, nu = pg.items.rows, pg.users.rows
            x0 = torch.empty((ni + nu, d), device=DEV)
            if ni:
                ops.linear_raw(pg.item_features, ie.weight, ie.bias, out=x0[:ni])
            if nu:
                ops.linear_raw(pg.user_features, ue.weight, ue.bias, out=x0[ni:])
            xs.append(x0)
            accs.append(torch.empty_like(x0))
        x0s = list(xs)
        for l in range(L_):
            for pg, x in zip(ranks, xs):
                ni, nu = pg.items.rows, pg.users.rows
                if ni:
                    ops.linear_raw(x[:ni], lin_i.weight, lin_i.bias, row_scale=pg.dinv_items, out=TI[pg.rank * mi: pg.rank * mi + ni])
                if nu:
                    ops.linear_raw(x[ni:], lin_u.weight, lin_u.bias, row_scale=pg.dinv_users, out=TU[pg.rank * mu: pg.rank * mu + nu])
            nxt = []
            for k, pg in enumerate(ranks):
                ni, nu = pg.items.rows, pg.users.rows
                xn = torch.empty_like(xs[k])
                src = x0s[k] if l == 0 else accs[k]
                scale = 1.0 / (L_ + 1) if l == L_ - 1 else 1.0
                if nu:
                    ops.spmm_raw(pg.index_users, TI, w=pg.index_users.w, dinv=pg.dinv_users, x_next=xn[ni:], acc_in=src[ni:],
                                 acc_out=accs[k][ni:], acc_scale=scale)
                if ni:
                    ops.spmm_raw(pg.index_items, TU, w=pg.index_items.w, dinv=pg.dinv_items, x_next=xn[:ni], acc_in=src[:ni],
                                 acc_out=accs[k][:ni], acc_scale=scale)
                nxt.append(xn)
            xs = nxt
        ref = m._encode(g, full, None, full.dinv, False)
        nI = ranks[0].nI
        comb = torch.empty_like(ref)
        ids = torch.arange(ref.shape[0], device=DEV)
        seen = torch.zeros(ref.shape[0], dtype=torch.int32, device=DEV)
        for k, pg in enumerate(ranks):
            mine, local = pg.locate(ids)
            comb[mine] = accs[k][local[mine]]
            seen += mine.int()
        assert torch.all(seen == 1)                     # every node has exactly one owner
    assert maxnorm_rel(comb, ref) < 1e-6


@pytest.mark.parametrize('P', [2, 3, 8])
def test_user_partition_reduce_scheme_emulated_ranks(P):
    """scheme 'reduce' with P emulated ranks on one GPU: the all-reduce of the item partials is a sum over the ranks'
    buffers.  Checks the column-sliced item CSRs, the owned user-row CSRs and their chunk plans with the real kernels."""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.graph import get_index
    from deeprecommendation_b200.parallel import UserPartitionedGraph
    m, g, uid, iid = _medium_graph()
    full = get_index(g)
    L_, d = len(m.gnn_convs), 64
    ranks = [UserPartitionedGraph(g, rank=r, world=P) for r in range(P)]
    nI = ranks[0].nI
    assert sum(pg.edges_own for pg in ranks) == full.e1 + full.e2
    assert sum(pg.users.rows for pg in ranks) == full.num_nodes - nI
    ie, ue = m.item_embeddings[0], m.user_embeddings[0]
    lin_u, lin_i, _ = m.gnn_convs[0].typed()
    with torch.no_grad():
        ref = m._encode(g, full, None, full.dinv, False)
        x_items = ops.linear_raw(g.item_features, ie.weight, ie.bias)
        x_users = [ops.linear_raw(pg.user_features, ue.weight, ue.bias) for pg in ranks]
        acc_items = x_items.clone()
        acc_users = [x.clone() for x in x_users]
        for l in range(L_):
            t_items = ops.linear_raw(x_items, lin_i.weight, lin_i.bias, row_scale=ranks[0].dinv_items)
            total = torch.zeros((nI, d), device=DEV)
            nxt = []
            for k, pg in enumerate(ranks):
                nu = pg.users.rows
                part = torch.zeros((nI, d), device=DEV)
                xn = torch.empty((nu, d), device=DEV)
                if nu:
                    t_users = ops.linear_raw(x_users[k], lin_u.weight, lin_u.bias, row_scale=pg.dinv_users)
                    ops.spmm_raw(pg.index_items, t_users, w=pg.index_items.w, dinv=pg.dinv_items, x_next=part)
                    ops.spmm_raw(pg.index_users, t_items, w=pg.index_users.w, dinv=pg.dinv_users, x_next=xn)
                total += part                                        # the all-reduce
                nxt.append(xn)
                acc_users[k] = acc_users[k] + xn
            x_items, x_users = total, nxt
            acc_items = acc_items + x_items
        comb = torch.cat([acc_items] + acc_users) / (L_ + 1)
    assert maxnorm_rel(comb, ref) < 1e-6


def test_attention_forward_resident_equals_dense_forward():
    """ResidentDynamicProvider + forward_resident (ids + CSR in, gather fused into the GEMM) == the dense contract, bit for bit"""
    from deeprecommendation_b200 import ops
    from deeprecommendation_b200.content_providers import ArrayDynamicProvider, ResidentDynamicProvider
    from deeprecommendation_b200.neural_collaborative_filtering.datasets.dynamic_datasets import DynamicPointwiseDataset
    users_raw, items_raw, ratings = synth.interactions_small(200, 3000, 60_000, seed=3)
    _, u = synth.dense_ids(users_raw)
    item_ids, it = synth.dense_ids(items_raw)
    n_items = len(item_ids)
    profiles = synth.item_profiles(n_items, seed=4, f_binary=300, f_dense=300)
    row_ptr, idx, rr, _ = synth.user_rating_lists(u, it, ratings, 200)
    args = (np.arange(n_items), profiles, np.arange(200), row_ptr, idx, rr)
    dense, res = ArrayDynamicProvider(*args), ResidentDynamicProvider(*args, device=DEV)
    kw = dict(item_dim=600, item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[256, 128], dropout_rate=0.2)
    m = _models().AttentionNCF(**kw).to(DEV).eval()
    m.load_state_dict(synth.to_torch(synth.attention_ncf_weights(seed=9, **kw)))
    pick = np.random.default_rng(0).permutation(len(u))[:256]
    batch = [(int(a), int(b), 3.0) for a, b in zip(u[pick], it[pick])]
    for engine in ('simt', 'tf32x3', 'bf16x3'):
        prev = ops.set_gemm_engine(engine)
        try:
            with torch.no_grad():
                out_d, _, _, _, att_d, _ = DynamicPointwiseDataset.do_forward(m, dense.collate_interacted_items(batch, False), DEV, True)
                out_r, _, _, _, att_r, _ = DynamicPointwiseDataset.do_forward(m, res.collate_interacted_items(batch, False), DEV, True)
        finally:
            ops.set_gemm_engine(prev)
        assert torch.equal(out_d, out_r), engine
        assert torch.equal(att_d, att_r), engine


@pytest.mark.parametrize('masked', [False, True])
def test_lightgat_gradients_vs_oracle_autograd(masked):
    """LightGATConv training step (gnn_ncf.py:97-177 under train.py:99-105): forward on K3's edge-softmax kernel, closed-form backward
    (ops._GatPropagateFn: dt on K3 over the reversed index, softmax gradient per edge) against torch autograd through the oracle restatement."""
    from deeprecommendation_b200.graph import IdTable, create_graph
    n_users, n_items, n, F, d_emb = 300, 120, 6000, 24, 32
    users, items, ratings = synth.interactions_zipf(n_users, n_items, n, seed=15)
    rng = np.random.default_rng(13)
    fi, fu = rng.standard_normal((n_items, F)).astype(np.float32), rng.standard_normal((n_users, F)).astype(np.float32)
    kw = dict(item_dim=F, user_dim=F, num_gnn_layers=2, hetero=True, node_emb=d_emb, mlp_dense_layers=[32], dropout_rate=0.2, convType='LightGAT')
    sd = synth.to_torch(synth.graph_ncf_weights(seed=14, **kw))
    ref_g = R.create_graph(users, items, ratings, np.arange(n_users), np.arange(n_items))
    gd = {k: (torch.from_numpy(v) if v is not None else None) for k, v in ref_g.items()}
    gd['item_features'], gd['user_features'] = torch.from_numpy(fi), torch.from_numpy(fu)
    pick = rng.permutation(n)[:96]
    uid, iid = torch.from_numpy(ref_g['user2item_edge_index'][0][pick]), torch.from_numpy(ref_g['user2item_edge_index'][1][pick])
    g = create_graph(torch.from_numpy(users).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(ratings).to(DEV),
                     torch.from_numpy(fi).to(DEV), torch.from_numpy(fu).to(DEV),
                     IdTable(torch.arange(n_users, device=DEV)), IdTable(torch.arange(n_items, device=DEV)))
    m = _models().GraphNCF(**kw).to(DEV).train()
    m.load_state_dict(sd)
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    out = m(g, uid.to(DEV), iid.to(DEV), DEV, mask_targets=masked)
    out.square().sum().backward()
    ref_sd = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    for k in list(ref_sd):
        if k.startswith('gnn_convs.1.'):
            ref_sd[k] = ref_sd[k.replace('gnn_convs.1.', 'gnn_convs.0.')]
    ref = R.graph_ncf_forward(ref_sd, gd, uid, iid, 2, convType='LightGAT', masked_positions=torch.from_numpy(pick) if masked else None)
    assert maxnorm_rel(out.detach(), ref.detach()) < TOL
    ref.square().sum().backward()
    got = dict(m.named_parameters())
    scale = max(float(v.grad.abs().max()) for v in ref_sd.values() if v.grad is not None)
    for k in ('item_embeddings.0.weight', 'user_embeddings.0.bias', 'gnn_convs.0.user2item_W.0.weight', 'gnn_convs.0.item2user_W.0.bias',
              'gnn_convs.0.user2item_AttNet.0.weight', 'gnn_convs.0.item2user_AttNet.0.weight', 'MLP.0.weight'):
        gk = got[k].grad
        rk = ref_sd[k].grad
        if 'AttNet' in k:                       # the destination half cancels in the row softmax: exactly 0 here, ~1e-17·scale in autograd
            assert float((gk[:, :d_emb].cpu() - rk[:, :d_emb]).abs().max()) < 1e-4 * max(float(rk[:, :d_emb].abs().max()), 1e-6 * scale), k
            assert float(gk[:, d_emb:].abs().max()) == 0.0 and float(rk[:, d_emb:].abs().max()) < 1e-5 * scale, k
        else:
            assert maxnorm_rel(gk, rk) < 1e-4, k


def test_pipelined_scoring_equals_sequential_replays():
    """graphed.PipelinedScoring: H2D copies of batch k + 1 under the kernels of batch k, per-graph events against a graph's own previous replay.
    Three batch shapes, two calls with different inputs: every result equals the plain captured forward on the same inputs."""
    from deeprecommendation_b200.graphed import GraphedForward, PipelinedScoring
    kw = dict(item_dim=96, item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[64], dropout_rate=0.2)
    m = _models().AttentionNCF(**kw).to(DEV).eval()
    m.load_state_dict(synth.to_torch(synth.attention_ncf_weights(seed=4, **kw)))
    rng = np.random.default_rng(8)

    def batch(B, I, seed):
        prof = synth.item_profiles(I + B, seed=seed, f_binary=48, f_dense=48)
        um = ((rng.integers(1, 11, (B, I)) * 0.5 - 2.75) * (rng.random((B, I)) < 0.3)).astype(np.float32)
        return tuple(torch.from_numpy(a).pin_memory() for a in (prof[I:], prof[:I], um))

    shapes = [(64, 300), (64, 517), (32, 1200)]
    first = [batch(B, I, 10 + k) for k, (B, I) in enumerate(shapes)]
    second = [batch(B, I, 20 + k) for k, (B, I) in enumerate(shapes)]
    graphs = [GraphedForward(lambda c, r, u: m(c, r, u), *(t.to(DEV) for t in b)) for b in first]
    pipe = PipelinedScoring(graphs)
    for batches in (first, second, first):
        got = [t.clone() for t in pipe(batches)]
        for k, b in enumerate(batches):
            want = graphs[k](*b).cpu()
            assert torch.equal(got[k], want), k
            with torch.no_grad():
                assert maxnorm_rel(got[k], m(*(t.to(DEV) for t in b)).cpu()) < 1e-6
