"""AttentionNCF.recommend(precision='bf16') (K8b, csrc/attention_recommend.cu): the pooling on bf16 tensor cores and the hidden layers after the
first on K1a's bf16 engine, held to the project's bf16 tolerance (max-norm relative error <= 1e-2) against the fp32 call and the CPU oracle;
K8b alone against a float64 restatement; the top-k, determinism, caches and `explain` after a bf16 call."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from oracle import synth
from tests._golden import maxnorm_rel

pytestmark = pytest.mark.gpu
TOL = 1e-2
DEV = 'cuda:0'


def _AttentionNCF():
    from deeprecommendation_b200.neural_collaborative_filtering.models import AttentionNCF
    return AttentionNCF


def _model(F, seed=1, **kw):
    kw = dict(dict(item_emb=32, user_emb=32, att_dense=64, mlp_dense_layers=[256, 128], dropout_rate=0.2), **kw)
    cos = kw.pop('use_cos_sim_instead', False)
    sd = synth.to_torch(synth.attention_ncf_weights(F, seed=seed, **kw))
    if cos:                                                               # the cosine variant has no AttentionNet
        sd = {k: v for k, v in sd.items() if not k.startswith('AttentionNet')}
    m = _AttentionNCF()(item_dim=F, use_cos_sim_instead=cos, **kw).to(DEV).eval()
    m.load_state_dict(sd)
    return m, sd


def _lists(rng, nU, nI, max_len, zero_frac=0.1):
    """K6-format rating lists: ascending unique items per user, centred ratings with some exact zeros; user 0 is empty, user 1 has only
    zero-centred entries, user 2 has one entry"""
    ptr, items, vals = [0], [], []
    for u in range(nU):
        n = 0 if u == 0 else 1 if u == 2 else int(rng.integers(1, max_len + 1))
        it = np.sort(rng.choice(nI, n, replace=False))
        v = rng.choice([-1.75, -1.25, -0.75, -0.25, 0.25, 0.75, 1.25], n).astype(np.float32)
        v[rng.random(n) < zero_frac] = 0.0
        if u == 1:
            v[:] = 0.0
        items.append(it); vals.append(v); ptr.append(ptr[-1] + n)
    return np.array(ptr, np.int64), np.concatenate(items).astype(np.int32), np.concatenate(vals).astype(np.float32)


def _dev(ptr, items, vals):
    return torch.from_numpy(ptr).to(DEV), torch.from_numpy(items).to(DEV), torch.from_numpy(vals).to(DEV)


def _seen(ptr, items, users):
    return [items[ptr[u]:ptr[u + 1]].astype(np.int64) for u in users]


def _profiles(rng, nI, F):
    return torch.from_numpy(rng.uniform(-1, 1, (nI, F)).astype(np.float32))


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _equal(a, b):
    """bit equality of recommend() outputs (the seen pairs of the score matrix are NaN)"""
    assert len(a) == len(b)
    for x, y in zip(a, b):
        assert torch.equal(_bits(x), _bits(y))


# ---- 1. accuracy: bf16 against the fp32 call and the CPU oracle -----------------------------------------------------------------------
VARIANTS = [
    dict(att_dense=64, mlp_dense_layers=[256, 128]),
    dict(att_dense=6, mlp_dense_layers=[128]),
    dict(att_dense=None, mlp_dense_layers=[256]),
    dict(att_dense=None, use_cos_sim_instead=True, mlp_dense_layers=[256, 128]),
    dict(att_dense=64, mlp_dense_layers=[128], item_emb=32, user_emb=30),
]


def _check_vs_fp32_and_oracle(m, sd, prof, ptr, items, vals, cos):
    nI, nU = prof.shape[0], len(ptr) - 1
    lists = _dev(ptr, items, vals)
    _, _, s32 = m.recommend(prof.to(DEV), *lists, k=5, return_scores=True)
    _, _, s16 = m.recommend(prof.to(DEV), *lists, k=5, return_scores=True, precision='bf16')
    s32, s16 = s32.cpu(), s16.cpu()
    worst = 0.0
    for u in range(nU):
        rated = items[ptr[u]:ptr[u + 1]].astype(np.int64)
        seen = np.zeros(nI, bool)
        seen[rated] = True
        keep = torch.from_numpy(~seen)
        assert torch.isnan(s16[u, torch.from_numpy(seen)]).all() and not torch.isnan(s16[u, keep]).any()
        if rated.size == 0:                      # the oracle cannot take I = 0: an empty list is one zero-centred entry
            rated, um = np.array([0]), np.zeros(1, np.float32)
        else:
            um = vals[ptr[u]:ptr[u + 1]]
        um_t = torch.from_numpy(um).view(1, -1).expand(nI, -1).contiguous()
        ref = R.attention_ncf_forward_blocked(sd, prof, prof[torch.from_numpy(rated)], um_t, use_cos_sim_instead=cos).view(-1)
        e32, eref = maxnorm_rel(s16[u, keep], s32[u, keep]), maxnorm_rel(s16[u, keep], ref[keep])
        assert e32 <= TOL and eref <= TOL, (u, e32, eref)
        worst = max(worst, e32, eref)
    return worst


@pytest.mark.parametrize('variant', VARIANTS, ids=['att64', 'att6', 'attNone', 'cosine', 'emb32_30'])
def test_scores_vs_fp32_and_oracle(variant):
    rng = np.random.default_rng(11)
    nI, F, nU = 150, 40, 9
    m, sd = _model(F, **variant)
    prof = _profiles(rng, nI, F)
    ptr, items, vals = _lists(rng, nU, nI, 90)
    worst = _check_vs_fp32_and_oracle(m, sd, prof, ptr, items, vals, variant.get('use_cos_sim_instead', False))
    print(f'bf16 {variant}: max-norm rel err {worst:.2e}')


@pytest.mark.parametrize('tail', [[], [128], [64, 32]], ids=['depth1', 'depth2', 'depth3'])
@pytest.mark.parametrize('H1', [32, 48, 128, 256])
def test_widths_and_depths(H1, tail):
    """first-layer widths of every H1P (48 pads to 64) and MLPs with 0, 1 and 2 hidden layers after the first"""
    rng = np.random.default_rng(H1 + len(tail))
    nI, F, nU = 131, 24, 6
    m, sd = _model(F, mlp_dense_layers=[H1] + tail)
    prof = _profiles(rng, nI, F)
    ptr, items, vals = _lists(rng, nU, nI, 100)
    worst = _check_vs_fp32_and_oracle(m, sd, prof, ptr, items, vals, False)
    print(f'bf16 MLP {[H1] + tail}: max-norm rel err {worst:.2e}')


# ---- 2. K8b alone against a float64 restatement on the same tables ------------------------------------------------------------------
def _h1_reference(tables, Qb, ptr, items, vals, u):
    """ReLU(Ai + Σ_i softmax_i(s)·um_i·bf16(Q')[i]) in float64 on the CPU (zero-centred entries get no attention; none -> α = 0)"""
    from deeprecommendation_b200 import _lib as L
    Pc, Pr, mode, a2, a20, Ai = tables[:6]
    Pc, Pr, Ai, Q = (t.detach().double().cpu() for t in (Pc, Pr, Ai, Qb.float()))
    rows = torch.from_numpy(items[ptr[u]:ptr[u + 1]].astype(np.int64))
    um = torch.from_numpy(vals[ptr[u]:ptr[u + 1]]).double()
    if rows.numel() == 0:
        return torch.relu(Ai)
    if mode == L.ATT_NET:
        s = torch.relu(Pc[:, None, :] + Pr[rows][None, :, :]) @ a2.detach().double().cpu()
        if a20 is not None:
            s = s + float(a20.detach().double().cpu().view(-1)[0])
    else:
        s = Pc @ Pr[rows].T
    s = s.masked_fill((um == 0).view(1, -1), float('-inf'))
    alpha = torch.nan_to_num(torch.softmax(s, dim=1), nan=0.0)
    return torch.relu(Ai + (alpha * um) @ Q[rows])


K8B_CASES = [(dict(att_dense=64), H1) for H1 in (32, 48, 128, 256)] + \
            [(dict(att_dense=None, use_cos_sim_instead=True), H1) for H1 in (32, 48, 128, 256)] + \
            [(dict(att_dense=256, item_emb=64, user_emb=64), 256)]


@pytest.mark.parametrize('variant,H1', K8B_CASES, ids=[f'{"cos" if v.get("use_cos_sim_instead") else "net"}{v.get("att_dense") or ""}_h{h}'
                                                        for v, h in K8B_CASES])
def test_kernel_vs_float64(variant, H1):
    from deeprecommendation_b200 import ops
    rng = np.random.default_rng(H1)
    nI, F, nU = 150, 40, 7                                               # 150 candidates: the last tile is partial
    m, _ = _model(F, mlp_dense_layers=[H1, 16], **variant)
    prof = _profiles(rng, nI, F).to(DEV)
    ptr, items, vals = _lists(rng, nU, nI, 120)
    tables = m._recommend_tables(prof)
    Pc, Pr, mode, a2, a20, Ai, Qp, _ = tables
    Qb = Qp.to(torch.bfloat16, memory_format=torch.contiguous_format)
    users = torch.arange(nU, device=DEV)
    h1 = ops.attention_recommend_raw(Pc, Pr, Ai, Qb, mode=mode, a2=a2, a20=a20, list_ptr=torch.from_numpy(ptr).to(DEV),
                                     list_item=torch.from_numpy(items).to(DEV), list_val=torch.from_numpy(vals).to(DEV), users=users)
    h1 = h1.view(nU, nI, -1).cpu()
    assert h1.shape[2] == Ai.shape[1]
    worst = 0.0
    for u in range(nU):
        ref = _h1_reference(tables, Qb, ptr, items, vals, u)
        if u in (0, 1):                                                   # empty and all-zero-centred lists: α = 0, h1 = ReLU(Ai) exactly
            assert torch.equal(h1[u], torch.relu(Ai.cpu()))
        err = maxnorm_rel(h1[u], ref)
        assert err <= TOL, (u, err)
        worst = max(worst, err)
    print(f'K8b {variant} H1={H1}: max-norm rel err vs float64 {worst:.2e}')


# ---- 3. selection ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nI', [1, 70, 131])
@pytest.mark.parametrize('k', [1, 10, 64])
def test_topk(nI, k):
    rng = np.random.default_rng(nI * 100 + k)
    F = 24
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    nU = 6
    ptr, items, vals = _lists(rng, nU, nI, max(1, nI - 8))            # long lists: some users have fewer than k unseen items
    lists = _dev(ptr, items, vals)
    for ignore_seen in (True, False):
        val, idx, scores = m.recommend(prof, *lists, k=k, ignore_seen=ignore_seen, return_scores=True, precision='bf16')
        seen = _seen(ptr, items, range(nU)) if ignore_seen else None
        rv, ri = R.topk_stable(scores.cpu(), k, seen=seen)             # a stable sort of the call's own bf16 scores
        assert torch.equal(idx.cpu(), ri) and torch.equal(val.cpu(), rv)
        v32, i32, s32 = m.recommend(prof, *lists, k=k, ignore_seen=ignore_seen, return_scores=True)
        s32 = s32.cpu()
        for u in range(nU):
            got = idx[u].cpu()
            if ignore_seen:
                assert not np.isin(got.numpy(), seen[u]).any()
                unseen = nI - len(seen[u])
                if unseen < k:
                    assert (got[unseen:] == -1).all() and torch.isinf(val[u, unseen:]).all() and (val[u, unseen:] < 0).all()
            pad = got < 0
            assert torch.equal(pad, i32[u].cpu() < 0)
            if (~pad).any():
                # near-ties may swap, larger differences may not: the fp32 score of bf16's j-th item against fp32's j-th value
                scale = float(s32[u][~torch.isnan(s32[u])].abs().max())
                d = (s32[u, got[~pad]] - v32[u].cpu()[~pad]).abs().max()
                assert float(d) <= TOL * scale, (u, float(d), scale)


# ---- 4. config-2 scale ----------------------------------------------------------------------------------------------------------------
def test_config2_all_users():
    from deeprecommendation_b200.content_providers import DeviceCollateProvider
    users_raw, items_raw, ratings = synth.interactions_small(610, 9724, 100_836, seed=42)
    _, u = synth.dense_ids(users_raw)
    item_ids, it = synth.dense_ids(items_raw)
    n_items = len(item_ids)
    profiles = synth.item_profiles(n_items, seed=43)
    row_ptr, idx, rr, _ = synth.user_rating_lists(u, it, ratings, 610)
    prov = DeviceCollateProvider(np.arange(n_items), profiles, np.arange(610), row_ptr, idx, rr, device=DEV)
    m, _ = _model(profiles.shape[1], item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[256, 128])
    lists = (prov.table, prov.d_list_ptr, prov.d_list_item, prov.d_list_val)
    _, i32, s32 = m.recommend(*lists, k=10, return_scores=True)
    _, i16, s16 = m.recommend(*lists, k=10, return_scores=True, precision='bf16')
    assert torch.equal(torch.isnan(s16), torch.isnan(s32))
    worst = 0.0
    for row in range(610):
        keep = ~torch.isnan(s32[row])
        worst = max(worst, maxnorm_rel(s16[row, keep], s32[row, keep]))
    assert worst <= TOL, worst
    same = sum(int(set(a.tolist()) == set(b.tolist())) for a, b in zip(i16.cpu(), i32.cpu()))
    print(f'config 2, all 610 users: bf16 vs fp32 max-norm rel err {worst:.2e}; identical top-10 sets for {same} of 610 users')


# ---- 5. determinism -------------------------------------------------------------------------------------------------------------------
def test_deterministic_and_chunking_on_the_cached_bf16_copy():
    from deeprecommendation_b200 import ops
    rng = np.random.default_rng(4)
    nI, F = 4200, 32
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    nU = 6
    lists = _dev(*_lists(rng, nU, nI, 200))
    a = m.recommend(prof, *lists, k=10, return_scores=True, precision='bf16')
    _equal(a, m.recommend(prof, *lists, k=10, return_scores=True, precision='bf16'))
    m.invalidate_caches()
    _equal(a, m.recommend(prof, *lists, k=10, return_scores=True, precision='bf16'))
    # K8b's h1 rows of a user do not depend on which users share the launch: bit for bit
    Pc, Pr, mode, a2, a20, Ai, Qp = m._recommend_tables(prof)[:7]
    kw = dict(mode=mode, a2=a2, a20=a20, list_ptr=lists[0], list_item=lists[1], list_val=lists[2])
    (Qb,) = m._rec_bf16.values()                                         # the cached bf16 copy of the cached Q'
    assert Qb.is_contiguous() and torch.equal(Qb, Qp.to(torch.bfloat16))
    h_all = ops.attention_recommend_raw(Pc, Pr, Ai, Qb, users=torch.arange(nU, device=DEV), **kw)
    h_one = torch.cat([ops.attention_recommend_raw(Pc, Pr, Ai, Qb, users=torch.tensor([u], device=DEV), **kw) for u in range(nU)])
    assert torch.equal(h_all, h_one)
    # the whole call per chunk size: K1a's layer-2 GEMM rounds a row differently when the number of rows changes (~1e-8, the fp32 path too)
    c = m.recommend(prof, *lists, k=10, return_scores=True, precision='bf16', chunk_users=1)
    assert torch.equal(torch.isnan(c[2]), torch.isnan(a[2])) and maxnorm_rel(c[2].nan_to_num(0.0), a[2].nan_to_num(0.0)) < 1e-6
    # duplicated users, in any order, against users=None
    users = torch.tensor([3, 0, 3, 5, 1], device=DEV)
    d = m.recommend(prof, *lists, k=10, users=users, return_scores=True, precision='bf16', chunk_users=2)
    _equal([x[0] for x in d], [x[2] for x in d])                     # the same user twice in one call
    for row, uu in enumerate(users.tolist()):
        assert maxnorm_rel(d[2][row].nan_to_num(0.0), a[2][uu].nan_to_num(0.0)) < 1e-6
    # no users
    val, idx, sc = m.recommend(prof, *lists, k=10, users=torch.zeros(0, dtype=torch.int64, device=DEV), return_scores=True, precision='bf16')
    assert val.shape == (0, 10) and idx.shape == (0, 10) and sc.shape == (0, nI)


# ---- 6. caches ------------------------------------------------------------------------------------------------------------------------
def _fresh(m, prof, lists, precision):
    f = _AttentionNCF()(**m.kwargs).to(DEV).eval()
    f.load_state_dict({k: v.clone() for k, v in m.state_dict().items()})
    return f.recommend(prof, *lists, k=10, return_scores=True, precision=precision)


def test_caches_and_the_bf16_store_follow_changes():
    rng = np.random.default_rng(8)
    nI, F = 200, 32
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    lists = _dev(*_lists(rng, 8, nI, 80))
    fp32 = m.recommend(prof, *lists, k=10, return_scores=True)
    assert len(m._rec_cache) == 1 and len(m._rec_bf16) == 0             # an fp32 call makes no bf16 copy
    base = m.recommend(prof, *lists, k=10, return_scores=True, precision='bf16')
    assert len(m._rec_bf16) == 1
    _equal(fp32, m.recommend(prof, *lists, k=10, return_scores=True))   # fp32 after bf16: untouched
    _equal(fp32, _fresh(m, prof, lists, 'fp32'))
    # an optimizer step (in place, bumps _version)
    opt = torch.optim.SGD(m.parameters(), lr=0.5)
    loss = sum((p * torch.randn_like(p)).sum() for p in m.parameters())
    loss.backward()
    opt.step()
    after = m.recommend(prof, *lists, k=10, return_scores=True, precision='bf16')
    assert not torch.equal(after[2].nan_to_num(0.0), base[2].nan_to_num(0.0))
    _equal(after, _fresh(m, prof, lists, 'bf16'))
    # load_state_dict
    _, sd2 = _model(F, seed=9)
    m.load_state_dict(sd2)
    assert len(m._rec_cache) == 0 and len(m._rec_bf16) == 0
    _equal(m.recommend(prof, *lists, k=10, return_scores=True, precision='bf16'), _fresh(m, prof, lists, 'bf16'))
    _equal(m.recommend(prof, *lists, k=10, return_scores=True), _fresh(m, prof, lists, 'fp32'))


# ---- 7. explain after a bf16 recommend ------------------------------------------------------------------------------------------------
def test_explain_after_bf16_recommend():
    rng = np.random.default_rng(17)
    nI, F = 300, 40
    m, _ = _model(F, att_dense=32, mlp_dense_layers=[64, 32])
    prof = _profiles(rng, nI, F).to(DEV)
    lists = _dev(*_lists(rng, 12, nI, 60, zero_frac=0.2))
    _, items = m.recommend(prof, *lists, k=10, precision='bf16')
    e16 = m.explain(prof, *lists, items, explain_factor=0.5)
    f = _AttentionNCF()(**m.kwargs).to(DEV).eval()
    f.load_state_dict({k: v.clone() for k, v in m.state_dict().items()})
    f.recommend(prof, *lists, k=10)
    e32 = f.explain(prof, *lists, items, explain_factor=0.5)
    assert int(e16[0][-1]) > 0
    _equal(e16, e32)


# ---- 8. errors ------------------------------------------------------------------------------------------------------------------------
def test_errors():
    from deeprecommendation_b200 import _lib as L
    from deeprecommendation_b200 import ops
    rng = np.random.default_rng(2)
    nI, F = 40, 16
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    ptr, items, vals = _lists(rng, 4, nI, 10)
    lists = _dev(ptr, items, vals)
    for p in ('fp16', 'FP32', None):
        with pytest.raises(ValueError, match='precision'):
            m.recommend(prof, *lists, precision=p)
    m.train()
    with pytest.raises(RuntimeError, match='eval'):
        m.recommend(prof, *lists, precision='bf16')
    m.eval()
    Pc, Pr, mode, a2, a20, Ai, Qp, _ = m._recommend_tables(prof)
    kw = dict(mode=mode, a2=a2, a20=a20, list_ptr=lists[0], list_item=lists[1], list_val=lists[2], users=torch.arange(4, device=DEV))
    for dt in (torch.float16, torch.float64):
        with pytest.raises(ValueError, match='Qp'):
            ops.attention_recommend_raw(Pc, Pr, Ai, Qp.to(dt), **kw)
    # the C entry's host-side checks, before any launch: NULL operands and a bf16 pitch that is not 16 bytes
    lib = L.lib()
    Qb = Qp.to(torch.bfloat16, memory_format=torch.contiguous_format)
    H, H1P = Pc.shape[1], Ai.shape[1]
    out = torch.empty((4 * nI, H1P), device=DEV)
    args = [Pc.data_ptr(), Pc.stride(0), Pr.data_ptr(), Pr.stride(0), H, int(mode), a2.data_ptr(), a20.data_ptr(), Ai.data_ptr(), Ai.stride(0),
            Qb.data_ptr(), H1P, H1P, nI, lists[0].data_ptr(), lists[1].data_ptr(), lists[2].data_ptr(), kw['users'].data_ptr(), 4, out.data_ptr(),
            H1P, None]
    for i in (0, 2, 8, 10, 14, 15, 16, 17, 19):
        bad = list(args)
        bad[i] = None
        with pytest.raises(ValueError, match='null'):
            L.check(lib.b200rec_attention_recommend_bf16(*bad), 'attention_recommend_bf16')
    bad = list(args)
    bad[11] = H1P + 4
    with pytest.raises(ValueError, match='multiple of 8'):
        L.check(lib.b200rec_attention_recommend_bf16(*bad), 'attention_recommend_bf16')
    L.check(lib.b200rec_attention_recommend_bf16(*args), 'attention_recommend_bf16')
    torch.cuda.synchronize()
    ref = ops.attention_recommend_raw(Pc, Pr, Ai, Qb, **kw)
    assert torch.equal(out, ref)
