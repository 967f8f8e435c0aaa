"""The dot form of the exact all-pairs kernel (csrc/allpairs.cu, allpairs_relu_dot_kernel<DOT = true>, ops.allpairs_dot_topk_raw):
score(u, i) = A[u]·B[i] against float64 A @ Bᵀ, and its top-k against a stable sort of the kernel's own scores (ties to the lower item,
NaN and `seen` items never selected, short rows padded with (-inf, -1))."""
import numpy as np
import pytest
import torch

from deeprecommendation_b200 import ops
from tests._golden import maxnorm_rel

pytestmark = pytest.mark.gpu
DEV = 'cuda:0'


def _select(S, k, seen=None):
    """reference top-k of a (nU, nI) float tensor: descending, stable (lower index first), NaN / -inf / seen excluded, padded"""
    S = S.double().cpu().numpy()
    val = np.full((S.shape[0], k), -np.inf)
    idx = np.full((S.shape[0], k), -1, dtype=np.int64)
    for u in range(S.shape[0]):
        ok = ~np.isnan(S[u]) & (S[u] > -np.inf)
        if seen is not None:
            ok[seen[u]] = False
        cand = np.nonzero(ok)[0]
        order = cand[np.lexsort((cand, -S[u, cand]))][:k]
        val[u, :len(order)], idx[u, :len(order)] = S[u, order], order
    return val, idx


@pytest.mark.parametrize('nU,nI,H,k,splits', [(5, 70, 32, 10, 0), (67, 1000, 48, 10, 3), (33, 1000, 64, 64, 17), (100, 257, 128, 20, 1),
                                               (1, 3001, 192, 10, 0), (130, 515, 256, 1, 3)])
def test_dot_kernel_against_float64(nU, nI, H, k, splits):
    g = torch.Generator().manual_seed(nU * 7 + H)
    A, B = torch.randn(nU, H, generator=g), torch.randn(nI, H, generator=g)
    val, idx, sc = ops.allpairs_dot_topk_raw(A.to(DEV), B.to(DEV), k, return_scores=True, n_splits=splits)
    ref = A.double() @ B.double().T
    assert maxnorm_rel(sc, ref) < 1e-6
    rv, ri = _select(sc, k)
    assert np.array_equal(idx.cpu().numpy(), ri) and np.array_equal(val.double().cpu().numpy(), rv)
    # top-k alone (no score matrix) selects the same
    v2, i2, none = ops.allpairs_dot_topk_raw(A.to(DEV), B.to(DEV), k, n_splits=splits)
    assert none is None and torch.equal(i2, idx) and torch.equal(v2, val)


@pytest.mark.parametrize('splits', [1, 3, 17])
def test_dot_kernel_seen_ties_nan(splits):
    g = torch.Generator().manual_seed(splits)
    nU, nI, H, k = 45, 2300, 64, 12
    A, B = torch.randn(nU, H, generator=g), torch.randn(nI, H, generator=g)
    B[1500] = B[7]                                      # duplicated rows: equal scores, the lower item first
    B[2200] = B[7]
    B[300] = float('nan')                               # a NaN row: never selected
    A[3] = 0.0                                          # a user whose every score is 0: ties across the whole catalogue
    rng = np.random.default_rng(splits)
    seen = [np.sort(rng.choice(nI, size=rng.integers(0, 40), replace=False)) for _ in range(nU)]
    ptr = torch.tensor(np.concatenate([[0], np.cumsum([len(s) for s in seen])]), dtype=torch.int32)
    items = torch.tensor(np.concatenate(seen), dtype=torch.int32)
    val, idx, sc = ops.allpairs_dot_topk_raw(A.to(DEV), B.to(DEV), k, return_scores=True, seen=(ptr.to(DEV), items.to(DEV)), n_splits=splits)
    rv, ri = _select(sc, k, seen)
    assert np.array_equal(idx.cpu().numpy(), ri) and np.array_equal(val.double().cpu().numpy(), rv)
    assert not (idx == 300).any()
    assert torch.isnan(sc[:, 300]).all()
    assert idx[3].tolist() == [i for i in range(nI) if i not in set(seen[3].tolist()) and i != 300][:k]
    assert torch.equal(sc[:, 1500], sc[:, 7]) and torch.equal(sc[:, 2200], sc[:, 7])


def test_dot_kernel_k0_scores_only_and_padding():
    g = torch.Generator().manual_seed(1)
    A, B = torch.randn(9, 40, generator=g), torch.randn(5, 40, generator=g)
    val, idx, sc = ops.allpairs_dot_topk_raw(A.to(DEV), B.to(DEV), 0, return_scores=True)
    assert val is None and idx is None and maxnorm_rel(sc, A.double() @ B.double().T) < 1e-6
    val, idx, _ = ops.allpairs_dot_topk_raw(A.to(DEV), B.to(DEV), 8)          # 5 items for k = 8: three padding entries per row
    assert (idx[:, 5:] == -1).all() and torch.isinf(val[:, 5:]).all() and (idx[:, :5] >= 0).all()


def test_dot_kernel_rejects_wide_rows():
    with pytest.raises(NotImplementedError, match='256'):
        ops.allpairs_dot_topk_raw(torch.zeros(2, 320, device=DEV), torch.zeros(3, 320, device=DEV), 4)
