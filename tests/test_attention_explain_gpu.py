"""AttentionNCF.explain (K9, csrc/attention_explain.cu): attention-threshold explanations of many users' recommendations against the CPU
oracle, `recommend_for_user`, and the GPU `forward` (K2) at config-2 scale; shapes and edges, determinism, caches and input errors.

α tolerance rtol=1e-4, atol=1e-6 (as for recommend_for_user's explanations).  Kept sets must be equal, except that an entry whose reference
α lies within 1e-6 of the threshold may go either way: the reference and the kernel sum in different orders."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from tests.test_attention_recommend_gpu import VARIANTS, _dev, _lists, _model, _profiles, config2  # noqa: F401 (config2 is a fixture)

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'
NEAR = 1e-6


def _thr(factor, constant, n):
    return np.float32(factor * (1.0 / max(n, 1)) + constant)          # recommend_for_user's threshold, compared in fp32


def _check_row(because, attention, rated, att_ref, thr, what):
    """one output row against the reference weights `att_ref` (R,) of the list `rated` (R,) ascending"""
    because, attention = because.cpu().numpy(), attention.cpu().numpy()
    near = np.abs(att_ref.astype(np.float64) - float(thr)) <= NEAR
    must = set(rated[(att_ref > thr) & ~near].tolist())
    may = set(rated[near].tolist())
    got = set(because.tolist())
    assert must <= got <= must | may, (what, sorted(must ^ got))
    assert len(got) == because.size and np.all(np.diff(because) > 0), what                  # list order, no duplicates
    ref = att_ref[np.searchsorted(rated, because)]
    assert np.allclose(attention, ref, rtol=1e-4, atol=1e-6), (what, np.abs(attention - ref).max())


def _rows(out, r):
    ptr, b, a = out
    return b[ptr[r]:ptr[r + 1]], a[ptr[r]:ptr[r + 1]]


def _check_vs_oracle(sd, prof, ptr, items, vals, top, out, factor, constant, cos):
    """every row of `explain`'s output against R.attention_ncf_forward(..., return_attention_weights=True) with the threshold applied"""
    nU, k = top.shape
    assert out[0].shape == (nU * k + 1,) and int(out[0][0]) == 0
    for u in range(nU):
        rated = items[ptr[u]:ptr[u + 1]].astype(np.int64)
        um = vals[ptr[u]:ptr[u + 1]]
        cand = top[u].cpu().numpy()
        real = cand >= 0
        att = np.zeros((k, rated.size), np.float32)
        if rated.size and real.any():
            um_t = torch.from_numpy(um).view(1, -1).expand(int(real.sum()), -1).contiguous()
            with torch.no_grad():
                _, a = R.attention_ncf_forward(sd, prof[torch.from_numpy(cand[real])], prof[torch.from_numpy(rated)], um_t,
                                               use_cos_sim_instead=cos, return_attention_weights=True)
            att[real] = a.numpy()
        thr = _thr(factor, constant, rated.size)
        for j in range(k):
            b, a = _rows(out, u * k + j)
            if not real[j] or rated.size == 0:
                assert b.numel() == 0 and a.numel() == 0, (u, j)
            else:
                _check_row(b, a, rated, att[j], thr, (u, j))


# ---- 1. against the CPU oracle ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('variant', VARIANTS, ids=['att64', 'att6', 'attNone', 'cosine', 'emb32_30'])
def test_vs_oracle(variant):
    rng = np.random.default_rng(12)
    nI, F, nU = 150, 40, 9
    m, sd = _model(F, **variant)
    prof = _profiles(rng, nI, F)
    ptr, items, vals = _lists(rng, nU, nI, 90)                                # user 0 empty, 1 only zero-centred, 2 one entry
    vals[ptr[2]] = 0.75                                                         # (which is not zero-centred)
    lists = _dev(ptr, items, vals)
    _, top = m.recommend(prof.to(DEV), *lists, k=10)
    cos = variant.get('use_cos_sim_instead', False)
    for factor, constant in ((1.5, 0.025), (0.0, 0.025)):
        out = m.explain(prof.to(DEV), *lists, top, explain_factor=factor, explain_constant=constant)
        _check_vs_oracle(sd, prof, ptr, items, vals, top, out, factor, constant, cos)
        ptr_o = out[0].cpu()
        assert (ptr_o[1:21] == 0).all()                                                      # the empty and the all-zero-centred list
        one = ptr_o[21:31] - ptr_o[20:30]                                                    # the one-entry list: thr 1.525 > α = 1
        assert (one == (1 if factor == 0.0 else 0)).all(), one
    assert out[0][-1] > 0


# ---- 2. against recommend_for_user -----------------------------------------------------------------------------------------------
def test_agrees_with_recommend_for_user():
    rng = np.random.default_rng(21)
    nI, F = 300, 48
    m, _ = _model(F, att_dense=32, mlp_dense_layers=[64, 32])
    prof = _profiles(rng, nI, F).to(DEV)
    ptr, items, vals, raw = [0], [], [], []
    for u in range(5):
        n = int(rng.integers(2, 60))
        it = np.sort(rng.choice(nI, n, replace=False))
        r = rng.choice([0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 3.5, 4.0, 4.5, 5.0], n)
        centred = (r - (r.mean() + 2.5) / 2).astype(np.float32)            # recommend_for_user's centring (backend.py:93)
        items.append(it); vals.append(centred); raw.append((it, r)); ptr.append(ptr[-1] + n)
    lists = _dev(np.array(ptr, np.int64), np.concatenate(items).astype(np.int32), np.concatenate(vals))
    _, top = m.recommend(prof, *lists, k=10)
    out = m.explain(prof, *lists, top)
    assert out[0][-1] > 0
    for u, (it, r) in enumerate(raw):
        perm = rng.permutation(len(it))
        rec = m.recommend_for_user(prof, torch.from_numpy(it[perm]).to(DEV), torch.from_numpy(r[perm]).to(DEV), k=10)
        assert torch.equal(top[u], rec['items'])
        for j in range(10):
            b, a = _rows(out, u * 10 + j)
            assert torch.equal(b, rec['because'][j]), (u, j)
            assert torch.allclose(a, rec['attention'][j], rtol=1e-4, atol=1e-6), (u, j)


# ---- 3. config-2 scale against the GPU forward (K2) ------------------------------------------------------------------------------
def test_config2_vs_forward(config2):  # noqa: F811
    c = config2
    m, table, ptr, items, vals, users = c['model'], c['table'], c['ptr'], c['items'], c['vals'], c['users']
    assert np.diff(ptr)[users].max() > 2000
    lists = _dev(ptr, items, vals)
    u_dev = torch.from_numpy(users).to(DEV)
    _, top = m.recommend(table, *lists, k=10, users=u_dev)
    out = m.explain(table, *lists, top, users=u_dev)
    assert out[0][-1] > 0
    for row, u in enumerate(users):
        rated = items[ptr[u]:ptr[u + 1]].astype(np.int64)
        um = vals[ptr[u]:ptr[u + 1]]
        if rated.size == 0:
            assert int(out[0][row * 10 + 10] - out[0][row * 10]) == 0
            continue
        um_t = torch.from_numpy(um).to(DEV).view(1, -1).expand(10, -1).contiguous()
        with torch.no_grad():
            _, att = m(table[top[row]], table[torch.from_numpy(rated).to(DEV)], um_t, return_attention_weights=True)
        att = att.cpu().numpy()
        thr = _thr(1.5, 0.025, rated.size)
        for j in range(10):
            b, a = _rows(out, row * 10 + j)
            _check_row(b, a, rated, att[j], thr, (row, int(u), j))
        if u in (611, 612):                                                    # only zero-centred entries / one entry: nothing
            assert int(out[0][row * 10 + 10] - out[0][row * 10]) == 0
    first, last = 0, len(users) - 1                                            # the longest list, also the duplicate at the end
    assert users[first] == users[last]
    for j in range(10):
        for x, y in zip(_rows(out, first * 10 + j), _rows(out, last * 10 + j)):
            assert torch.equal(x, y)


# ---- 4. shapes and edges ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('k', [1, 64])
def test_shapes_and_edges(k):
    rng = np.random.default_rng(30 + k)
    nI, F, nU = 200, 32, 7
    m, sd = _model(F)
    prof = _profiles(rng, nI, F)
    ptr, items, vals = _lists(rng, nU, nI, 150)
    lists = _dev(ptr, items, vals)
    _, top = m.recommend(prof.to(DEV), *lists, k=k, ignore_seen=False)     # a user's own list items are candidates too
    top = top.clone()
    top[3, k // 2] = -1                                                         # padding rows
    top[5, :] = -1
    top[4, -1] = int(items[ptr[4]])                                             # (at least one candidate from the user's own list)
    for factor, constant in ((1.5, 0.025), (0.0, 0.0)):                        # 0, 0: every α > 0 explains (the capacity path)
        out = m.explain(prof.to(DEV), *lists, top, explain_factor=factor, explain_constant=constant)
        _check_vs_oracle(sd, prof, ptr, items, vals, top, out, factor, constant, False)
        pad = out[0][1:] - out[0][:-1]
        assert pad[3 * k + k // 2] == 0 and (pad[5 * k:6 * k] == 0).all()
    assert out[0][-1] > 0
    ptr_o, b, a = m.explain(prof.to(DEV), *lists, top, explain_constant=2.0)   # α <= 1 < 2: nothing, n = 0
    assert (ptr_o == 0).all() and b.shape == (0,) and a.shape == (0,) and b.dtype == torch.int64 and a.dtype == torch.float32


def test_no_users():
    rng = np.random.default_rng(3)
    m, _ = _model(16)
    prof = _profiles(rng, 30, 16).to(DEV)
    lists = _dev(*_lists(rng, 4, 30, 10))
    ptr, b, a = m.explain(prof, *lists, torch.empty((0, 5), dtype=torch.int64, device=DEV), users=torch.empty(0, dtype=torch.int64, device=DEV))
    assert ptr.tolist() == [0] and b.numel() == 0 and a.numel() == 0


# ---- 5. determinism --------------------------------------------------------------------------------------------------------------
def test_deterministic():
    rng = np.random.default_rng(4)
    nI, F = 500, 64
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    lists = _dev(*_lists(rng, 20, nI, 400))
    _, top = m.recommend(prof, *lists, k=16)
    a = m.explain(prof, *lists, top, explain_factor=0.5)
    m.invalidate_caches()
    b = m.explain(prof, *lists, top, explain_factor=0.5)
    assert a[0][-1] > 0
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32) if x.is_floating_point() else x, y.view(torch.int32) if y.is_floating_point() else y)


# ---- 6. caches follow changes ----------------------------------------------------------------------------------------------------
def _fresh(m, prof, lists, top):
    from deeprecommendation_b200.neural_collaborative_filtering.models import AttentionNCF
    f = AttentionNCF(**m.kwargs).to(DEV).eval()
    f.load_state_dict({k: v.clone() for k, v in m.state_dict().items()})
    return f.explain(prof, *lists, top, explain_factor=0.5)


def _same(x, y):
    assert torch.equal(x[0], y[0]) and torch.equal(x[1], y[1])
    assert torch.allclose(x[2], y[2], rtol=1e-6, atol=0)


def test_caches_follow_changes():
    rng = np.random.default_rng(8)
    nI, F = 200, 32
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    lists = _dev(*_lists(rng, 8, nI, 80))
    _, top = m.recommend(prof, *lists, k=10)
    base = m.explain(prof, *lists, top, explain_factor=0.5)
    opt = torch.optim.SGD(m.parameters(), lr=0.5)                              # an optimizer step (in place, bumps _version)
    loss = sum((p * torch.randn_like(p)).sum() for p in m.parameters())
    loss.backward()
    opt.step()
    after = m.explain(prof, *lists, top, explain_factor=0.5)
    assert not (torch.equal(after[1], base[1]) and torch.equal(after[2], base[2]))
    _same(after, _fresh(m, prof, lists, top))
    _, sd2 = _model(F, seed=9)                                                 # load_state_dict
    m.load_state_dict(sd2)
    _same(m.explain(prof, *lists, top, explain_factor=0.5), _fresh(m, prof, lists, top))


# ---- 7. errors -------------------------------------------------------------------------------------------------------------------
def test_errors():
    rng = np.random.default_rng(2)
    nI, F = 40, 16
    m, _ = _model(F)
    prof = _profiles(rng, nI, F)
    ptr, items, vals = _lists(rng, 4, nI, 10)
    lists = _dev(ptr, items, vals)
    p = prof.to(DEV)
    top = torch.zeros((4, 3), dtype=torch.int64, device=DEV)
    m.train()
    with pytest.raises(RuntimeError, match='eval'):
        m.explain(p, *lists, top)
    m.eval()
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m.explain(prof, *lists, top)
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m.explain(p, *lists, top.cpu())
    with pytest.raises(ValueError):
        m.explain(p, lists[0], lists[1].long(), lists[2], top)
    with pytest.raises(ValueError):
        m.explain(p, lists[0].int(), lists[1], lists[2], top)
    with pytest.raises(ValueError):
        m.explain(p, lists[0], lists[1], lists[2].double(), top)
    with pytest.raises(ValueError, match='int64'):
        m.explain(p, *lists, top.int())
    for bad in (nI, -2):
        t = top.clone()
        t[1, 2] = bad
        with pytest.raises(ValueError, match='items'):
            m.explain(p, *lists, t)
    with pytest.raises(ValueError, match='rows'):
        m.explain(p, *lists, top[:3])
    with pytest.raises(ValueError, match='rows'):
        m.explain(p, *lists, top, users=torch.tensor([0, 1], device=DEV))
    for kk in (0, 65):
        with pytest.raises(ValueError, match='k'):
            m.explain(p, *lists, torch.zeros((4, kk), dtype=torch.int64, device=DEV))
    with pytest.raises(ValueError, match='users'):
        m.explain(p, *lists, top[:2], users=torch.tensor([0, 4], device=DEV))
    with pytest.raises(ValueError, match='users'):
        m.explain(p, *lists, top[:1], users=torch.tensor([-1], device=DEV))
    bad_item = lists[1].clone()
    bad_item[-1] = nI
    with pytest.raises(ValueError, match='list_item'):
        m.explain(p, lists[0], bad_item, lists[2], top)
    bad_ptr = lists[0].clone()
    bad_ptr[-1] += 1
    with pytest.raises(ValueError, match='list_ptr'):
        m.explain(p, bad_ptr, lists[1], lists[2], top)
    for kw in (dict(mlp_dense_layers=[512]), dict(mlp_dense_layers=[]), dict(att_dense=260),
               dict(att_dense=None, use_cos_sim_instead=True, item_emb=260)):
        wide, _ = _model(F, **kw)
        with pytest.raises(NotImplementedError):
            wide.explain(p, *lists, top)
