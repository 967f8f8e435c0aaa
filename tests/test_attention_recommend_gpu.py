"""AttentionNCF.recommend (K8, csrc/attention_recommend.cu): whole-catalogue top-k for many users against the CPU oracle, the GPU
`forward` (K2 path) at config-2 scale, `recommend_for_user`, the stable top-k, and its caches.  fp32 tolerance: max-norm relative
error <= 1e-5."""
import numpy as np
import pytest
import torch

from oracle import restatement as R
from oracle import synth
from tests._golden import maxnorm_rel

pytestmark = pytest.mark.gpu
TOL = 1e-5
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


# ---- 1. against the CPU oracle ------------------------------------------------------------------------------------------
VARIANTS = [
    dict(att_dense=64, mlp_dense_layers=[256, 128]),
    dict(att_dense=6, mlp_dense_layers=[128]),
    dict(att_dense=None, mlp_dense_layers=[256]),
    dict(att_dense=None, use_cos_sim_instead=True, mlp_dense_layers=[256, 128]),
    dict(att_dense=64, mlp_dense_layers=[128], item_emb=32, user_emb=30),
]


@pytest.mark.parametrize('variant', VARIANTS, ids=['att64', 'att6', 'attNone', 'cosine', 'emb32_30'])
def test_scores_vs_oracle(variant):
    rng = np.random.default_rng(11)
    nI, F, nU = 150, 40, 9
    m, sd = _model(F, **variant)
    prof = _profiles(rng, nI, F)
    ptr, items, vals = _lists(rng, nU, nI, 90)
    _, _, scores = m.recommend(prof.to(DEV), *_dev(ptr, items, vals), k=5, return_scores=True)
    scores = scores.cpu()
    cos = variant.get('use_cos_sim_instead', False)
    for u in range(nU):
        rated = items[ptr[u]:ptr[u + 1]].astype(np.int64)
        seen = np.zeros(nI, bool)
        seen[rated] = True
        assert torch.isnan(scores[u, torch.from_numpy(seen)]).all()
        if rated.size == 0:                      # the oracle cannot take I = 0: an empty list is one zero-centred entry
            rated, um = np.array([0]), np.zeros(1, np.float32)
        else:
            um = vals[ptr[u]:ptr[u + 1]]
        um_t = torch.from_numpy(um).view(1, -1).expand(nI, -1).contiguous()
        ref = R.attention_ncf_forward_blocked(sd, prof, prof[torch.from_numpy(rated)], um_t, use_cos_sim_instead=cos).view(-1)
        keep = torch.from_numpy(~seen)
        assert maxnorm_rel(scores[u, keep], ref[keep]) < TOL, u


# ---- 2. against the GPU forward (K2) at config-2 scale ---------------------------------------------------------------------
@pytest.fixture(scope='module')
def config2():
    from deeprecommendation_b200.content_providers import DeviceCollateProvider
    users_raw, items_raw, ratings = synth.interactions_small(610, 9724, 100_836, seed=42)
    _, u = synth.dense_ids(users_raw)
    item_ids, it = synth.dense_ids(items_raw)
    n_items = len(item_ids)
    profiles = synth.item_profiles(n_items, seed=43)
    row_ptr, idx, rr, _ = synth.user_rating_lists(u, it, ratings, 610)
    prov = DeviceCollateProvider(np.arange(n_items), profiles, np.arange(610), row_ptr, idx, rr, device=DEV)
    kw = dict(item_emb=128, user_emb=128, att_dense=128, mlp_dense_layers=[256, 128])
    m, _ = _model(profiles.shape[1], **kw)
    ptr, items, vals = prov.d_list_ptr.cpu().numpy(), prov.d_list_item.cpu().numpy(), prov.d_list_val.cpu().numpy()
    lens = np.diff(ptr)
    pick = list(np.random.default_rng(5).choice(610, 44, replace=False))
    pick[0] = int(np.argmax(lens))                                    # the longest list
    # three extra list rows: empty, only zero-centred entries, one entry
    ex_items = [np.zeros(0, np.int32), np.array([3, 17, 400], np.int32), np.array([1234], np.int32)]
    ex_vals = [np.zeros(0, np.float32), np.zeros(3, np.float32), np.array([0.75], np.float32)]
    ptr2 = np.concatenate([ptr, ptr[-1] + np.cumsum([len(x) for x in ex_items])]).astype(np.int64)
    items2 = np.concatenate([items] + ex_items).astype(np.int32)
    vals2 = np.concatenate([vals] + ex_vals).astype(np.float32)
    users = np.array(pick + [610, 611, 612, int(np.argmax(lens))], np.int64)      # (a duplicate of the longest list at the end)
    return dict(model=m, table=prov.table, ptr=ptr2, items=items2, vals=vals2, users=users, prov=prov)


def _forward_row(m, table, rated, um):
    nI = table.shape[0]
    keep = torch.ones(nI, dtype=torch.bool, device=DEV)
    if rated.size:
        keep[torch.from_numpy(rated.astype(np.int64)).to(DEV)] = False
    else:
        rated, um = np.array([0]), np.zeros(1, np.float32)          # empty list == one zero-centred entry
    cand = keep.nonzero().view(-1)
    r = torch.from_numpy(rated.astype(np.int64)).to(DEV)
    um_t = torch.from_numpy(um).to(DEV).view(1, -1).expand(cand.numel(), -1).contiguous()
    with torch.no_grad():
        y = m(table[cand], table[r], um_t).view(-1)
    return cand, y


@pytest.mark.parametrize('chunk', [1, 7, None])
def test_config2_vs_forward(config2, chunk):
    c = config2
    m, table, ptr, items, vals, users = c['model'], c['table'], c['ptr'], c['items'], c['vals'], c['users']
    assert np.diff(ptr)[users].max() > 2000
    _, _, scores = m.recommend(table, *_dev(ptr, items, vals), k=10, users=torch.from_numpy(users).to(DEV), return_scores=True,
                               chunk_users=chunk)
    for row, u in enumerate(users):
        rated, um = items[ptr[u]:ptr[u + 1]], vals[ptr[u]:ptr[u + 1]]
        cand, y = _forward_row(m, table, rated, um)
        got = scores[row, cand]
        assert not torch.isnan(got).any()
        assert maxnorm_rel(got, y) < TOL, (row, int(u))
        if rated.size:
            assert torch.isnan(scores[row, torch.from_numpy(rated.astype(np.int64)).to(DEV)]).all()


def test_config2_provider_lists_default_users(config2):
    """a DeviceCollateProvider's resident lists feed the method directly; users=None = every list row"""
    c = config2
    prov, m = c['prov'], c['model']
    val, idx = m.recommend(prov.table, prov.d_list_ptr, prov.d_list_item, prov.d_list_val, k=10)
    assert val.shape == (610, 10) and idx.shape == (610, 10) and idx.dtype == torch.int64
    assert (idx >= 0).all() and torch.isfinite(val).all()
    assert (val[:, :-1] >= val[:, 1:]).all()


# ---- 3. top-k ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('nI', [1, 70, 131])
@pytest.mark.parametrize('k', [1, 10, 64])
def test_topk_bit_exact(nI, k):
    rng = np.random.default_rng(nI * 100 + k)
    F = 24
    m, _ = _model(F)
    prof = _profiles(rng, nI, F)
    if nI > 1:
        prof[1::2] = prof[0:nI - 1:2]                                  # duplicate profiles: tied scores, the lower item must win
    nU = 6
    ptr, items, vals = _lists(rng, nU, nI, max(1, nI - 8))            # long lists: some users have fewer than k unseen items
    users = list(range(nU))
    for ignore_seen in (True, False):
        val, idx, scores = m.recommend(prof.to(DEV), *_dev(ptr, items, vals), k=k, ignore_seen=ignore_seen, return_scores=True)
        rv, ri = R.topk_stable(scores.cpu(), k, seen=_seen(ptr, items, users) if ignore_seen else None)
        assert torch.equal(idx.cpu(), ri)
        assert torch.equal(val.cpu(), rv)
        if ignore_seen:
            unseen = nI - np.diff(ptr)
            for u in range(nU):
                if unseen[u] < k:
                    assert (idx[u, unseen[u]:] == -1).all() and torch.isinf(val[u, unseen[u]:]).all()
    if nI > 1:                                                           # the duplicates really tie
        s, n2 = scores.cpu(), nI // 2
        assert torch.equal(s[:, 1:2 * n2:2], s[:, 0:2 * n2:2])


# ---- 4. agreement with recommend_for_user -----------------------------------------------------------------------------------
def test_agrees_with_recommend_for_user():
    rng = np.random.default_rng(21)
    nI, F = 300, 48
    m, _ = _model(F, att_dense=32, mlp_dense_layers=[64, 32])
    prof = _profiles(rng, nI, F).to(DEV)
    ptr, items, vals = [0], [], []
    raw = []
    for u in range(5):
        n = int(rng.integers(2, 60))
        it = np.sort(rng.choice(nI, n, replace=False))
        r = rng.choice([0.5, 1.0, 1.5, 2.0, 2.5, 3.0, 3.5, 4.0, 4.5, 5.0], n)
        centred = (r - (r.mean() + 2.5) / 2).astype(np.float32)        # recommend_for_user's centring (backend.py:93)
        items.append(it); vals.append(centred); raw.append((it, r)); ptr.append(ptr[-1] + n)
    lists = _dev(np.array(ptr, np.int64), np.concatenate(items).astype(np.int32), np.concatenate(vals))
    val, idx = m.recommend(prof, *lists, k=10)
    for u, (it, r) in enumerate(raw):
        perm = rng.permutation(len(it))                                 # recommend_for_user takes any order
        rec = m.recommend_for_user(prof, torch.from_numpy(it[perm]).to(DEV), torch.from_numpy(r[perm]).to(DEV), k=10)
        assert torch.equal(idx[u], rec['items'])
        assert maxnorm_rel(val[u], rec['scores']) < TOL


# ---- 5. determinism --------------------------------------------------------------------------------------------------------
def test_deterministic():
    rng = np.random.default_rng(4)
    nI, F = 500, 64
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    lists = _dev(*_lists(rng, 20, nI, 200))
    a = m.recommend(prof, *lists, k=10, return_scores=True)
    m.invalidate_caches()
    b = m.recommend(prof, *lists, k=10, return_scores=True)
    for x, y in zip(a, b):                                               # bit patterns: the seen pairs are NaN
        assert torch.equal(x.view(torch.int32) if x.is_floating_point() else x, y.view(torch.int32) if y.is_floating_point() else y)


# ---- 6. caches ---------------------------------------------------------------------------------------------------------------
def _fresh(m, F, prof, lists):
    f = _AttentionNCF()(**m.kwargs).to(DEV).eval()
    f.load_state_dict({k: v.clone() for k, v in m.state_dict().items()})
    return f.recommend(prof, *lists, k=10, return_scores=True)


def _same(a, b):
    assert torch.equal(a[1], b[1])
    assert maxnorm_rel(a[2].nan_to_num(0.0), b[2].nan_to_num(0.0)) < 1e-6


def test_caches_follow_changes():
    rng = np.random.default_rng(8)
    nI, F = 200, 32
    m, _ = _model(F)
    prof = _profiles(rng, nI, F).to(DEV)
    lists = _dev(*_lists(rng, 8, nI, 80))
    base = m.recommend(prof, *lists, k=10, return_scores=True)
    # an optimizer step (in place, bumps _version)
    opt = torch.optim.SGD(m.parameters(), lr=0.5)
    loss = sum((p * torch.randn_like(p)).sum() for p in m.parameters())
    loss.backward()
    opt.step()
    after = m.recommend(prof, *lists, k=10, return_scores=True)
    assert not torch.equal(after[2], base[2])
    _same(after, _fresh(m, F, prof, lists))
    # load_state_dict
    _, sd2 = _model(F, seed=9)
    m.load_state_dict(sd2)
    _same(m.recommend(prof, *lists, k=10, return_scores=True), _fresh(m, F, prof, lists))
    # an edit through .data (no _version bump) + invalidate_caches()
    with torch.no_grad():
        m.MLP[0].weight.data.mul_(-1.0)
    m.invalidate_caches()
    _same(m.recommend(prof, *lists, k=10, return_scores=True), _fresh(m, F, prof, lists))
    # a new profile table, then an in-place edit of it
    prof2 = _profiles(rng, nI, F).to(DEV)
    _same(m.recommend(prof2, *lists, k=10, return_scores=True), _fresh(m, F, prof2, lists))
    prof2.mul_(0.5)
    _same(m.recommend(prof2, *lists, k=10, return_scores=True), _fresh(m, F, prof2, lists))


# ---- 7. errors ---------------------------------------------------------------------------------------------------------------
def test_errors():
    rng = np.random.default_rng(2)
    nI, F = 40, 16
    m, _ = _model(F)
    prof = _profiles(rng, nI, F)
    ptr, items, vals = _lists(rng, 4, nI, 10)
    lists = _dev(ptr, items, vals)
    m.train()
    with pytest.raises(RuntimeError, match='eval'):
        m.recommend(prof.to(DEV), *lists)
    m.eval()
    with pytest.raises(RuntimeError, match='no CPU fallback'):
        m.recommend(prof, *lists)
    with pytest.raises(ValueError):
        m.recommend(prof.to(DEV), lists[0], lists[1].long(), lists[2])
    with pytest.raises(ValueError):
        m.recommend(prof.to(DEV), lists[0].int(), lists[1], lists[2])
    for layers in ([512], []):
        big, _ = _model(F, mlp_dense_layers=layers)
        with pytest.raises(NotImplementedError):
            big.recommend(prof.to(DEV), *lists)
    for kw in (dict(att_dense=260), dict(att_dense=None, use_cos_sim_instead=True, item_emb=260)):     # score tables wider than K8 stages
        wide, _ = _model(F, **kw)
        with pytest.raises(NotImplementedError):
            wide.recommend(prof.to(DEV), *lists)
    # row numbers out of range are caught on the host, before the kernel reads with them
    with pytest.raises(ValueError, match='users'):
        m.recommend(prof.to(DEV), *lists, users=torch.tensor([0, 4], device=DEV))
    with pytest.raises(ValueError, match='users'):
        m.recommend(prof.to(DEV), *lists, users=torch.tensor([-1], device=DEV))
    bad_item = lists[1].clone()
    bad_item[-1] = nI
    with pytest.raises(ValueError, match='list_item'):
        m.recommend(prof.to(DEV), lists[0], bad_item, lists[2])
    bad_ptr = lists[0].clone()
    bad_ptr[-1] += 1
    with pytest.raises(ValueError, match='list_ptr'):
        m.recommend(prof.to(DEV), bad_ptr, lists[1], lists[2])


# ---- 8. memory: without return_scores nothing of size (nU, nI) is allocated ---------------------------------------------------------------
def test_memory_bounded_without_scores():
    rng = np.random.default_rng(13)
    nI, F, nU = 2000, 32, 300
    m, _ = _model(F, mlp_dense_layers=[32, 16])
    prof = _profiles(rng, nI, F).to(DEV)
    lists = _dev(*_lists(rng, nU, nI, 40))
    ref = m.recommend(prof, *lists, k=10, chunk_users=1, return_scores=True)          # (also builds the cached catalogue tables)
    torch.cuda.synchronize()
    base = torch.cuda.memory_allocated()
    torch.cuda.reset_peak_memory_stats()
    val, idx = m.recommend(prof, *lists, k=10, chunk_users=1)
    torch.cuda.synchronize()
    peak = torch.cuda.max_memory_allocated() - base
    assert peak < nU * nI * 4 // 2, peak
    assert torch.equal(val, ref[0]) and torch.equal(idx, ref[1])
