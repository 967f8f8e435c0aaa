"""GraphNCF on the B200 path (reference: neural_collaborative_filtering/models/gnn_ncf.py:13-94,180-378)."""
from __future__ import annotations

import os

import numpy as np
import torch
from torch import nn

from ... import ops
from ...derived import Derived
from ...graph import get_index
from ..util import build_MLP_layers, mlp_parameters, run_mlp
from .base import GNN_NCF, _named_like


class _TypedLinear(nn.Sequential):
    """`Sequential(Linear, Dropout)` — the parameter container of one edge type (gnn_ncf.py:22-29), Xavier-initialised
    like the reference (:30-31,37)."""

    def __init__(self, channels_in, channels_out, dropout):
        super().__init__(nn.Linear(channels_in, channels_out), nn.Dropout(dropout))
        nn.init.xavier_uniform_(self[0].weight)


class LightGCNConv(nn.Module):
    """Parameter holder for one LightGCN-style layer (gnn_ncf.py:13-37).  The arithmetic of its forward/message
    (:39-94) is executed by GraphNCF through the transform GEMM (K1a) + CSR SpMM (K3); there is no PyG here."""

    def __init__(self, in_channels, out_channels, hetero, dropout=0.1):
        super().__init__()
        self.hetero = hetero
        if hetero:
            self.user2item_W = _TypedLinear(in_channels, out_channels, dropout)
            self.item2user_W = _TypedLinear(in_channels, out_channels, dropout)
        else:
            self.W = _TypedLinear(in_channels, out_channels, dropout)

    def typed(self):
        """(linear for user sources, linear for item sources, dropout p)."""
        if self.hetero:
            return self.user2item_W[0], self.item2user_W[0], self.user2item_W[1].p
        return self.W[0], self.W[0], self.W[1].p


class LightGATConv(nn.Module):
    """Parameter holder for the GAT-style layer (gnn_ncf.py:97-177): per edge type a Linear(d, d) and an attention
    Linear(2d, 1) over [x_source, x_destination].  Executed by K3 with an edge softmax: the destination half of the
    attention Linear is constant over the incoming edges of a node, so it cancels in the softmax (PyG's `+1e-16`
    denominator included) and only the source half is evaluated — one scalar per NODE instead of one 2d-dot per EDGE."""

    def __init__(self, in_channels, out_channels, hetero, dropout=0.1):
        super().__init__()
        self.hetero = hetero
        if hetero:
            self.user2item_W = _TypedLinear(in_channels, out_channels, dropout)
            self.item2user_W = _TypedLinear(in_channels, out_channels, dropout)
            self.user2item_AttNet = nn.Sequential(nn.Linear(in_channels * 2, 1))
            self.item2user_AttNet = nn.Sequential(nn.Linear(in_channels * 2, 1))
        else:
            self.W = _TypedLinear(in_channels, out_channels, dropout)
            self.AttNet = nn.Sequential(nn.Linear(in_channels * 2, 1))

    def typed(self):
        if self.hetero:
            return self.user2item_W[0], self.item2user_W[0], self.user2item_W[1].p
        return self.W[0], self.W[0], self.W[1].p

    def attention(self):
        """(attention Linear for user sources, for item sources)"""
        if self.hetero:
            return self.user2item_AttNet[0], self.item2user_AttNet[0]
        return self.AttNet[0], self.AttNet[0]


class GraphNCF(GNN_NCF):
    """Node embed -> L shared-weight propagation layers over the whole bipartite graph -> mean (or concat) of the L+1
    embeddings -> gather the batch rows -> MLP (item first) or dot product  (gnn_ncf.py:298-367).

    Per layer:  t[s] = deg[s]^-1/2 · (W_type x[s] + b_type)   one GEMM per node type (the reference runs this Linear per EDGE)
                x'[r] = deg[r]^-1/2 · Σ_{s->r} w_sr · t[s]     deterministic edge-balanced CSR SpMM, running mean fused in

    `cache_eval_embeddings=True` (new, default off) keeps the propagated embeddings between eval-mode calls while neither
    the graph nor the parameters change; the reference recomputes them for every mini-batch (:298-351).

    `message_dtype = 'bf16'` (attribute, default 'fp32'; inference only): the per-node messages `t` are rounded ONCE to bf16 by
    the transform GEMM's epilogue and K3 gathers 2-byte features (half the bytes through L1 / L2 / HBM); accumulation, the
    running mean and everything else stay fp32.  Tolerance of this mode: max-norm relative error <= 1e-2 (north_star)."""

    message_dtype = os.environ.get('B200REC_GRAPH_MESSAGE_DTYPE', 'fp32')

    def __init__(self, item_dim, user_dim, num_gnn_layers: int, hetero, node_emb=64, mlp_dense_layers=None, dropout_rate=0.2,
                 use_dot_product=False, concat=False, message_dropout=None, node_dropout=None, convType='LightGCN',
                 cache_eval_embeddings=False):
        super().__init__()
        mlp_dense_layers = [256, 128] if mlp_dense_layers is None else mlp_dense_layers
        self.kwargs = dict(item_dim=item_dim, user_dim=user_dim, node_emb=node_emb, num_gnn_layers=num_gnn_layers,
                           mlp_dense_layers=mlp_dense_layers, use_dot_product=use_dot_product, dropout_rate=dropout_rate,
                           message_dropout=message_dropout, node_dropout=node_dropout, hetero=hetero, concat=concat,
                           convType=convType)
        self.concat, self.message_dropout, self.node_dropout, self.convType = concat, message_dropout, node_dropout, convType
        self.cache_eval_embeddings = cache_eval_embeddings
        self._cache = Derived(1)                  # propagated embeddings (cache_eval_embeddings)
        self._peer_layer0 = Derived(1)            # layer-0 composite weights of the peer-partitioned forward (peer.py)
        self.item_embeddings = nn.Sequential(nn.Linear(item_dim, node_emb))
        self.user_embeddings = nn.Sequential(nn.Linear(user_dim, node_emb))
        if convType == 'LightGCN':
            conv = LightGCNConv(node_emb, node_emb, hetero=hetero, dropout=dropout_rate / 2)
        elif convType == 'LightGAT':
            conv = LightGATConv(node_emb, node_emb, hetero=hetero, dropout=dropout_rate / 2)
        else:
            raise ValueError('Invalid convType.')
        self.gnn_convs = nn.ModuleList([conv] * num_gnn_layers)        # ONE module aliased L times (gnn_ncf.py:227)
        width = node_emb * (num_gnn_layers + 1) if concat else node_emb
        self.MLP = None if use_dot_product else build_MLP_layers(2 * width, mlp_dense_layers, dropout_rate=dropout_rate)

    def important_hypeparams(self) -> str:
        return '_' + self.convType

    def is_dataset_compatible(self, dataset_class):
        return _named_like(dataset_class, 'GraphPointwiseDataset', 'GraphRankingDataset')

    # ------------------------------------------------------------------------------------------------------------------
    def _training_mask(self, index, userIds, itemIds, mask_targets):
        """Positions (in the interaction list) of the edges removed for this step: batch targets (:314-320), node dropout
        (:281-296) and message dropout (:246-279).  Returns None when nothing is removed."""
        removed = []
        if mask_targets:
            removed.append(index.positions(userIds, itemIds))
        dev = index.u2i.device
        if self.node_dropout is not None and self.node_dropout > 0.0:
            n = index.num_nodes
            in_batch = torch.zeros(n, dtype=torch.bool, device=dev)
            in_batch[itemIds] = True
            in_batch[userIds] = True
            others = (~in_batch).nonzero().view(-1)
            n_keep = int((1.0 - self.node_dropout) * others.numel())
            kept = others[torch.randperm(others.numel(), device=dev)[:n_keep]]
            alive = in_batch.clone()
            alive[kept] = True
            removed.append((~(alive[index.u2i[0]] & alive[index.u2i[1]])).nonzero().view(-1))
        if self.message_dropout is not None and self.message_dropout > 0.0:
            removed.append((torch.rand(index.e1, device=dev) < self.message_dropout).nonzero().view(-1))
        if not removed:
            return None
        return torch.cat(removed)

    def _encode(self, graph, index, skip, dinv, training):
        nI = graph.item_features.shape[0]
        N, L_ = index.num_nodes, len(self.gnn_convs)
        d = self.item_embeddings[0].weight.shape[0]
        ie, ue = self.item_embeddings[0], self.user_embeddings[0]
        lin_u, lin_i, p_conv = self.gnn_convs[0].typed() if L_ else (None, None, 0.0)
        need_grad = torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())
        dev = graph.item_features.device
        if not need_grad:
            # inference path: every layer writes straight into preallocated buffers, the running mean is fused into K3
            width = d * (L_ + 1) if self.concat else d
            comb = torch.empty((N, width), dtype=torch.float32, device=dev)
            x0 = comb[:, :d] if self.concat else torch.empty((N, d), dtype=torch.float32, device=dev)
            ops.linear_raw(graph.item_features, ie.weight, ie.bias, out=x0[:nI])          # :300
            ops.linear_raw(graph.user_features, ue.weight, ue.bias, out=x0[nI:])          # :301, items first (:304)
            if L_ == 0:
                return x0
            if self.message_dtype not in ('fp32', 'bf16'):
                raise ValueError("message_dtype must be 'fp32' or 'bf16'")
            t_dtype = torch.bfloat16 if (self.message_dtype == 'bf16' and d % 8 == 0) else torch.float32
            x, t = x0, torch.empty((N, d), dtype=t_dtype, device=dev)
            spare = torch.empty((N, d), dtype=torch.float32, device=dev) if (L_ > 1 and not self.concat) else None
            gat = self.convType == 'LightGAT'
            if gat:
                att_u, att_i = self.gnn_convs[0].attention()
                ps = torch.empty((N, 1), dtype=torch.float32, device=dev)
            for l in range(L_):
                if gat:      # no degree normalisation; per-source attention score from the source half of Linear(2d, 1)
                    ops.linear_raw(x[:nI], lin_i.weight, lin_i.bias, out=t[:nI])
                    ops.linear_raw(x[nI:], lin_u.weight, lin_u.bias, out=t[nI:])
                    ops.linear_raw(x[:nI], att_i.weight[:, :d], None, out=ps[:nI], engine='simt')
                    ops.linear_raw(x[nI:], att_u.weight[:, :d], None, out=ps[nI:], engine='simt')
                else:
                    ops.linear_raw(x[:nI], lin_i.weight, lin_i.bias, row_scale=dinv[:nI], out=t[:nI])     # item sources: item2user_W
                    ops.linear_raw(x[nI:], lin_u.weight, lin_u.bias, row_scale=dinv[nI:], out=t[nI:])     # user sources: user2item_W
                last = l == L_ - 1
                if self.concat:
                    xn = comb[:, d * (l + 1): d * (l + 2)]
                    ops.propagate_step(index, t, dinv=None if gat else dinv, x_next=xn, skip_bits=skip, att_src=ps if gat else None)
                else:
                    # x is dead once t has been formed (same stream), so one spare buffer serves every layer; it must not
                    # alias x0, which layer 0 still reads as acc_in
                    xn = None if last else spare
                    ops.propagate_step(index, t, dinv=None if gat else dinv, x_next=xn, acc_in=x0 if l == 0 else comb, acc_out=comb,
                                       acc_scale=1.0 / (L_ + 1) if last else 1.0, skip_bits=skip, att_src=ps if gat else None)
                x = xn
            return comb
        # training path: same kernels through autograd Functions (backward of K3 = K3 on the reverse weights)
        x = torch.cat((ops.linear(graph.item_features, ie.weight, ie.bias), ops.linear(graph.user_features, ue.weight, ue.bias)), 0)
        hs = [x]
        if self.convType == 'LightGAT':
            # gnn_ncf.py:128-177 with gradients: W(x_j) per node, the source half of the attention Linear per node, K3 with the edge softmax forward,
            # closed-form backward (ops._GatPropagateFn).  The destination half of AttNet and its bias cancel inside the row softmax: their gradient is 0.
            att_u, att_i = self.gnn_convs[0].attention()
            d_ = x.shape[1]
            for _ in range(L_):
                t = torch.cat((ops.linear(x[:nI], lin_i.weight, lin_i.bias), ops.linear(x[nI:], lin_u.weight, lin_u.bias)), 0)
                if training and p_conv > 0.0:
                    t = torch.nn.functional.dropout(t, p_conv, training=True)
                ps = torch.cat((ops.linear(x[:nI], att_i.weight[:, :d_], None), ops.linear(x[nI:], att_u.weight[:, :d_], None)), 0)
                x = ops.propagate_gat(t, ps, index, skip)
                hs.append(x)
            return torch.cat(hs, dim=1) if self.concat else torch.mean(torch.stack(hs, dim=0), dim=0)
        for _ in range(L_):
            t = torch.cat((ops.linear(x[:nI], lin_i.weight, lin_i.bias, row_scale=dinv[:nI]),
                           ops.linear(x[nI:], lin_u.weight, lin_u.bias, row_scale=dinv[nI:])), 0)
            if training and p_conv > 0.0:
                # the reference drops entries of W(x_j) per EDGE (:22-29,:91); after transform-before-gather the mask is per
                # source NODE and layer — same expectation, documented in DESIGN.md
                t = torch.nn.functional.dropout(t, p_conv, training=True)
            x = ops.propagate(t, index, index.w, index.w_bwd, dinv, skip)
            hs.append(x)
        return torch.cat(hs, dim=1) if self.concat else torch.mean(torch.stack(hs, dim=0), dim=0)     # :348-351

    def recommend(self, graph, k=10, user_nodes=None, precision='fp32', ignore_seen=True, return_scores=False):
        """Top-k item NODE ids for the given user nodes (default: every user) over ALL items — the whole-catalogue form of
        `forward` (gnn_ncf.py:298-367: propagate, gather the pair's rows, MLP item-first or dot product), with the selection of
        the reference's serving loop (src/webapp/backend.py:85,113-121).  One propagation (K1a + K3), then the fused all-pairs
        kernel K5 over (users x items); `ignore_seen` leaves out the items a user is connected to in the graph."""
        if self.training:
            raise RuntimeError('recommend() is an inference call: model.eval() first')
        index = get_index(graph)
        nI = graph.item_features.shape[0]
        with torch.no_grad():
            comb = self._encode(graph, index, None, index.dinv, False)
            users = torch.arange(nI, index.num_nodes, device=comb.device) if user_nodes is None else user_nodes.long()
            user_emb, item_emb = comb[users].contiguous(), comb[:nI]
            seen = index.seen_items(users) if ignore_seen else None
            if self.MLP is None:                                      # dot product (:365): one GEMM + row-wise top-k
                scores = ops.linear_raw(user_emb, item_emb, None)
                if seen is not None:
                    ptr, idx = seen
                    rows = torch.repeat_interleave(torch.arange(users.numel(), device=comb.device), (ptr[1:] - ptr[:-1]).long())
                    scores[rows, idx.long()] = float('nan')           # never selected by the top-k kernel
                val, idx = ops.topk_rows(scores, k)
                return (val, idx, scores) if return_scores else (val, idx)
            weights, biases, _ = mlp_parameters(self.MLP)
            val, idx, scores = ops.mlp_allpairs_topk(user_emb, item_emb, weights, biases, k, rows_first=False, precision=precision,
                                                     seen=seen, return_scores=return_scores)
        return (val, idx, scores) if return_scores else (val, idx)

    def forward(self, graph, userIds, itemIds, device=None, mask_targets=True):
        pg = getattr(graph, '_b200rec_partition', None)
        if pg is not None and not self.training:      # 1-D row-partitioned multi-GPU propagation (parallel.py)
            from ...parallel import forward_partitioned
            return forward_partitioned(self, pg, userIds, itemIds)
        index = get_index(graph)
        skip, dinv = None, index.dinv
        if self.training:
            removed = self._training_mask(index, userIds, itemIds, mask_targets)
            if removed is not None:
                skip, dinv = index.masked(removed)
        if self.cache_eval_embeddings and not self.training and not torch.is_grad_enabled():
            comb = self._cache.get((index, *self.parameters()), lambda: self._encode(graph, index, skip, dinv, False), self.message_dtype)
        else:
            self._cache.clear()
            comb = self._encode(graph, index, skip, dinv, self.training)
        if self.MLP is None:
            return ops.rowdot(comb, comb, userIds, itemIds)                               # :365
        return run_mlp(self.MLP, comb, comb, idx0=itemIds, idx1=userIds, training=self.training)   # item first (:361)
