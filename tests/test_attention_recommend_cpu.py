"""The folded algebra of AttentionNCF.recommend (models/attention_ncf.py `_recommend_tables`, csrc/attention_recommend.cu), restated in
float64 torch on the CPU and held against the reference's op order:

    h1[b] = ReLU(Ai[b] + Σ_i α_bi·um_i·Q'[i]),   Ai = Ec·W1eᵀ + b1 + W1u·b_U,   Q' = R·(W1u·W_U)ᵀ

then the rest of the MLP.  The oracle rounds its (B, I) score matrix to fp32 (attention_ncf.py:182); here it is evaluated with that
dtype mapped to float64, so the two sides differ only by float64 reassociation and the algebra is pinned to 1e-12."""
import types

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import restatement as R
from oracle import synth


def _float64_oracle(monkeypatch):
    shim = types.SimpleNamespace(**{k: getattr(torch, k) for k in dir(torch) if not k.startswith('__')})
    shim.float32 = torch.float64
    monkeypatch.setattr(R, 'torch', shim)


def _folded(sd, profiles, rated_rows, um_row, *, cos):
    """scores of every catalogue row against ONE rated list, through the folded tables (pooling in H1 space)"""
    WI, bI = sd['ItemEmbeddings.0.weight'], sd['ItemEmbeddings.0.bias']
    WU, bU = sd['UserEmbeddings.0.weight'], sd['UserEmbeddings.0.bias']
    E = WI.shape[0]
    ks = R.mlp_linear_indices(sd)
    W1, b1 = sd[f'MLP.{ks[0]}.weight'], sd[f'MLP.{ks[0]}.bias']
    W1e, W1u = W1[:, :E], W1[:, E:]
    Ec = profiles @ WI.T + bI
    Er = Ec[rated_rows]
    if cos:
        s = F.normalize(Ec, dim=1) @ F.normalize(Er, dim=1).T
    elif 'AttentionNet.3.weight' in sd:
        A, a = sd['AttentionNet.0.weight'], sd['AttentionNet.0.bias']
        Pc, Pr = Ec @ A[:, :E].T + a, Er @ A[:, E:].T
        s = torch.relu(Pc[:, None, :] + Pr[None, :, :]) @ sd['AttentionNet.3.weight'].view(-1) + sd['AttentionNet.3.bias']
    else:
        A, a = sd['AttentionNet.0.weight'], sd['AttentionNet.0.bias']
        s = (Ec @ A[:, :E].T + a) + (Er @ A[:, E:].T).T
    keep = (um_row != 0).expand_as(s)
    alpha = torch.nan_to_num(torch.softmax(s.masked_fill(~keep, float('-inf')), dim=1), nan=0.0)
    Ai = Ec @ W1e.T + b1 + W1u @ bU
    Qp = profiles[rated_rows] @ (W1u @ WU).T
    x = torch.relu(Ai + (alpha * um_row) @ Qp)
    for n, k in enumerate(ks[1:]):
        if n:
            x = torch.relu(x)
        x = F.linear(x, sd[f'MLP.{k}.weight'], sd[f'MLP.{k}.bias'])
    return x


CASES = [
    dict(att_dense=8, mlp=[16, 8], cos=False, E=8, U=8),
    dict(att_dense=6, mlp=[16], cos=False, E=8, U=6),
    dict(att_dense=None, mlp=[12, 8], cos=False, E=4, U=4),
    dict(att_dense=None, mlp=[16], cos=True, E=6, U=10),
]


@pytest.mark.parametrize('case', CASES, ids=lambda c: f"att{c['att_dense']}_cos{int(c['cos'])}_mlp{'x'.join(map(str, c['mlp']))}")
def test_folded_algebra_matches_reference_order(case, monkeypatch):
    nI, Fdim = 23, 11
    sd = {k: v.double() for k, v in synth.to_torch(synth.attention_ncf_weights(Fdim, item_emb=case['E'], user_emb=case['U'], att_dense=case['att_dense'],
                                                                               mlp_dense_layers=case['mlp'], seed=5)).items()}
    rng = np.random.default_rng(3)
    profiles = torch.from_numpy(rng.uniform(-1, 1, (nI, Fdim)))
    _float64_oracle(monkeypatch)
    for n_rated, n_zero in ((7, 2), (1, 0), (3, 3), (nI, 5)):
        rated = torch.from_numpy(np.sort(rng.choice(nI, n_rated, replace=False))) if n_rated else torch.zeros(0, dtype=torch.int64)
        um = torch.from_numpy(rng.uniform(-2, 2, n_rated))
        um[:n_zero] = 0.0                                            # zero-centred entries: no attention
        got = _folded(sd, profiles, rated, um.view(1, -1), cos=case['cos'])
        ref = R.attention_ncf_forward(sd, profiles, profiles[rated], um.view(1, -1).expand(nI, -1).contiguous(), use_cos_sim_instead=case['cos'])
        assert ref.dtype == torch.float64
        err = (got - ref).abs().max() / ref.abs().max()
        assert err < 1e-12, (n_rated, n_zero, float(err))
