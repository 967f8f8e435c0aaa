"""BasicNCF on the B200 path (reference: neural_collaborative_filtering/models/basic_ncf.py:9-48)."""
from __future__ import annotations

import torch
from torch import nn

from ... import ops
from ...derived import Derived
from ..util import build_MLP_layers, mlp_parameters, run_mlp
from .base import NCF, _named_like


class BasicNCF(NCF):
    """out = MLP([user_embeddings(X_user), item_embeddings(X_item)])  — user first (basic_ncf.py:40).

    Two CUDA projection GEMMs (K1a) feed the fused MLP tower (K1b); the concatenation is never materialised."""

    def __init__(self, item_dim, user_dim, dropout_rate=0.2, item_emb=256, user_emb=256, mlp_dense_layers=None):
        super().__init__()
        mlp_dense_layers = [256, 128] if mlp_dense_layers is None else mlp_dense_layers
        self.kwargs = dict(item_dim=item_dim, user_dim=user_dim, item_emb=item_emb, user_emb=user_emb,
                           mlp_dense_layers=mlp_dense_layers, dropout_rate=dropout_rate)
        self.item_embeddings = nn.Sequential(nn.Linear(item_dim, item_emb))
        self.user_embeddings = nn.Sequential(nn.Linear(user_dim, user_emb))
        self.MLP = build_MLP_layers(item_emb + user_emb, mlp_dense_layers, dropout_rate=dropout_rate)
        self._emb_cache = Derived(1)         # (user table, item table) embeddings of forward_resident

    cache_eval_embeddings = False        # forward_resident: project every row of the resident tables once per weight version (inference)

    def forward_resident(self, X_user, X_item):
        """`forward` fed by `content_providers.ResidentProfilesProvider`: both arguments are `ResidentRows` (row numbers into profile tables
        that live in HBM).  Default: the rows are gathered on the device and take the same kernels as the dense contract (identical bits).
        With `cache_eval_embeddings` (inference only) every row of both tables is projected ONCE per weight version and a batch is one
        launch of the MLP tower over gathered embedding rows — the per-unique-row form SURVEY.md §8d names for config 4, and what the
        reference's serving loop would want (src/webapp/backend.py:96-99 re-projects every candidate on every request)."""
        dev = X_user.table.device
        if self.training or (torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())):
            return self.forward(X_user.dense(), X_item.dense())
        pu, pi = X_user.pos.to(dev, non_blocking=True), X_item.pos.to(dev, non_blocking=True)
        if not self.cache_eval_embeddings:
            return self.forward(X_user.table.index_select(0, pu), X_item.table.index_select(0, pi))
        ue, ie = self.user_embeddings[0], self.item_embeddings[0]
        user_emb, item_emb = self._emb_cache.get(
            (X_user.table, X_item.table, ue.weight, ue.bias, ie.weight, ie.bias),
            lambda: (ops.linear_raw(X_user.table, ue.weight, ue.bias), ops.linear_raw(X_item.table, ie.weight, ie.bias)))
        return run_mlp(self.MLP, user_emb, item_emb, idx0=pu, idx1=pi, training=False)

    def forward(self, X_user, X_item):
        if hasattr(X_user, 'table') and hasattr(X_item, 'table'):
            return self.forward_resident(X_user, X_item)
        ue, ie = self.user_embeddings[0], self.item_embeddings[0]
        if not (torch.is_tensor(X_user) and torch.is_tensor(X_item)):
            # one-hot / multi-hot rows (content_providers.OneHotRows / MixedRows): gather-sum projection K1s, dense columns on K1a
            user_emb = ops.linear_rows(X_user, ue.weight, ue.bias)
            item_emb = ops.linear_rows(X_item, ie.weight, ie.bias)
        elif not (torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())):
            # inference: both projections of the batch in one launch when they are short-M / long-K (split-K over one wave)
            user_emb, item_emb = ops.linear_pair(X_user, ue.weight, ue.bias, X_item, ie.weight, ie.bias)
        else:
            user_emb = ops.linear(X_user, ue.weight, ue.bias)
            item_emb = ops.linear(X_item, ie.weight, ie.bias)
        return run_mlp(self.MLP, user_emb, item_emb, training=self.training)

    def recommend(self, X_users, X_items, k=10, precision='fp32', seen=None, return_scores=False):
        """Top-k items for every user over ALL (user, item) pairs — BASELINE configs[3]; the batched form of the reference's
        serving loop (src/webapp/backend.py:78-121: score every candidate for a user, sort, keep k).  X_users (nU, user_dim),
        X_items (nI, item_dim).  Returns (scores (nU, k), item positions (nU, k) int64[, all scores (nU, nI)]).
        Same arithmetic as `forward` on every pair, with the first MLP Linear split per side (exact) and the rest in the fused
        tcgen05 kernel (csrc/allpairs.cu); `seen` = CSR (ptr, idx) of pairs to leave out (`ignore_seen`, backend.py:85)."""
        if self.training:
            raise RuntimeError('recommend() is an inference call: model.eval() first')
        ue, ie = self.user_embeddings[0], self.item_embeddings[0]
        with torch.no_grad():
            user_emb = ops.linear_raw(X_users, ue.weight, ue.bias)
            item_emb = ops.linear_raw(X_items, ie.weight, ie.bias)
            weights, biases, _ = mlp_parameters(self.MLP)
            val, idx, scores = ops.mlp_allpairs_topk(user_emb, item_emb, weights, biases, k, rows_first=True, precision=precision,
                                                     seen=seen, return_scores=return_scores)
        return (val, idx, scores) if return_scores else (val, idx)

    def is_dataset_compatible(self, dataset_class):
        return _named_like(dataset_class, 'FixedPointwiseDataset', 'FixedRankingDataset')
