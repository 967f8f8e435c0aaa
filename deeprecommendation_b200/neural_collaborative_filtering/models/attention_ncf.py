"""AttentionNCF on the B200 path (reference: neural_collaborative_filtering/models/attention_ncf.py:64-224)."""
from __future__ import annotations

import torch
from torch import nn

from ... import _lib as L
from ... import ops
from ...derived import Derived
from ..util import build_MLP_layers, mlp_parameters, run_mlp
from .base import NCF, _named_like


RECOMMEND_SLAB_BYTES = 1 << 30      # default budget of one chunk's h1 slab in `AttentionNCF.recommend` (users per chunk = budget / (nI·H1P·4))


def _pad_rows(w, b, mult=4):
    """Zero-pads the output rows of a Linear to a multiple of `mult` (the pooling kernel loads 128-bit rows)."""
    n = w.shape[0]
    extra = (-n) % mult
    if extra == 0:
        return w, b
    w = torch.cat((w, w.new_zeros(extra, w.shape[1])), 0)
    if b is not None:
        b = torch.cat((b, b.new_zeros(extra)), 0)
    return w, b


class AttentionNCF(NCF):
    """The user profile is built on the fly from the user's rated items with item-item attention against the candidate
    (attention_ncf.py:136-224).  Device pipeline per call:

      K1a  Ec = ItemEmb(candidate)                         (B, E)
      K1a  [Er | Q] = rated_items · [W_I ; W_U]ᵀ           one pass over the (I, F) profiles feeds both the item
                                                           embedding and the pooled-profile projection Q = R·W_Uᵀ
      K1a  Pc = Ec·A1cᵀ + a1,  Pr = Er·A1rᵀ                AttentionNet.0 split into candidate / rated halves
           (inference: the last two lines collapse into [Ec | Pc] and [Pr | Q] straight from the profiles, `_composite_projection`)
      K2   user_emb = Σ_i softmax_i(a2·ReLU(Pc+Pr_i)+a20)·um_bi·Q_i + b_U     ragged, one warp per candidate
      K1b  out = MLP([Ec, user_emb])                       item first (attention_ncf.py:219)

    Nothing of shape (B·I, E) or (B, I, ·) is ever materialised (the reference builds two of them, :154-155)."""

    def __init__(self, item_dim, item_emb=128, user_emb=128, att_dense=None, mlp_dense_layers=None, use_cos_sim_instead=False,
                 dropout_rate=0.2, message_dropout=None):
        super().__init__()
        mlp_dense_layers = [256, 128] if mlp_dense_layers is None else mlp_dense_layers
        self.kwargs = dict(item_dim=item_dim, item_emb=item_emb, user_emb=user_emb, att_dense=att_dense,
                           mlp_dense_layers=mlp_dense_layers, dropout_rate=dropout_rate,
                           use_cos_sim_instead=use_cos_sim_instead, message_dropout=message_dropout)
        self.use_cos_sim_instead, self.message_dropout = use_cos_sim_instead, message_dropout
        self.ItemEmbeddings = nn.Sequential(nn.Linear(item_dim, item_emb))
        self.UserEmbeddings = nn.Sequential(nn.Linear(item_dim, user_emb))
        if not use_cos_sim_instead:
            self.att_dense = att_dense if att_dense is not None else 0
            if att_dense is not None:
                self.AttentionNet = nn.Sequential(nn.Linear(2 * item_emb, att_dense), nn.ReLU(), nn.Dropout(dropout_rate),
                                                  nn.Linear(att_dense, 1))
            else:
                self.AttentionNet = nn.Sequential(nn.Linear(2 * item_emb, 1))
        self.MLP = build_MLP_layers(item_emb + user_emb, mlp_dense_layers, dropout_rate=dropout_rate)
        self._proj_cache = Derived(1)        # _stacked_projection
        self._comp_cache = Derived(1)        # _composite_projection
        self._att_cache = Derived(1)         # _attention_halves
        self._rec_cache = Derived(1)         # _recommend_tables
        self._rec_bf16 = Derived(1)          # bf16 copy of the cached Q' table (recommend(precision='bf16'))

    def important_hypeparams(self) -> str:
        return '_cosine' if self.use_cos_sim_instead else f'_attNet{self.att_dense}'

    def is_dataset_compatible(self, dataset_class):
        return _named_like(dataset_class, 'DynamicPointwiseDataset', 'DynamicRankingDataset')

    # ------------------------------------------------------------------------------------------------------------------
    def _score_tables(self, Ec, Er):
        """(Pc, Pr, mode, a2, a20) for the three scoring variants (attention_ncf.py:162-179)."""
        E = Ec.shape[1]
        if self.use_cos_sim_instead:                               # <normalize(Ec_b), normalize(Er_i)>  (:163-173)
            Pc = torch.nn.functional.normalize(Ec, p=2, dim=1)
            Pr = torch.nn.functional.normalize(Er, p=2, dim=1)
            pad = (-E) % 4
            if pad:
                Pc, Pr = torch.nn.functional.pad(Pc, (0, pad)), torch.nn.functional.pad(Pr, (0, pad))
            return Pc, Pr.contiguous(), L.ATT_DOT, None, None
        first = self.AttentionNet[0]
        if len(self.AttentionNet) > 1:                             # Linear(2E,H) ReLU Dropout Linear(H,1)  (:112-117)
            head = self.AttentionNet[3]
            A1, a1 = _pad_rows(first.weight, first.bias)
            a2 = head.weight.view(-1)
            if a2.shape[0] != A1.shape[0]:
                a2 = torch.cat((a2, a2.new_zeros(A1.shape[0] - a2.shape[0])))
            Pc = ops.linear(Ec, A1[:, :E], a1)                     # candidate half first (:176)
            Pr = ops.linear(Er, A1[:, E:], None)
            return Pc, Pr, L.ATT_NET, a2, head.bias
        # att_dense=None: a single Linear(2E, 1): s = A_c·Ec_b + A_r·Er_i + a0 = <[sc,1,0,0], [1,sr,0,0]>  (:120-122)
        sc = ops.linear(Ec, first.weight[:, :E], first.bias)       # (B, 1)
        sr = ops.linear(Er, first.weight[:, E:], None)             # (I, 1)
        Pc = torch.cat((sc, torch.ones_like(sc), torch.zeros_like(sc), torch.zeros_like(sc)), 1)
        Pr = torch.cat((torch.ones_like(sr), sr, torch.zeros_like(sr), torch.zeros_like(sr)), 1)
        return Pc, Pr, L.ATT_DOT, None, None

    def _stacked_projection(self):
        """[W_I ; W_U] and [b_I ; 0] for the single sweep over rated_items.  Under no_grad the stacked copies are cached
        until a parameter changes (its `_version` moves with every optimizer step / load_state_dict)."""
        item, user = self.ItemEmbeddings[0], self.UserEmbeddings[0]

        def stack():
            WU, bU = _pad_rows(user.weight, user.bias)
            return torch.cat((item.weight, WU), 0), torch.cat((item.bias, torch.zeros_like(bU)), 0), bU
        return self._proj_cache.get((item.weight, item.bias, user.weight, user.bias), stack)

    def _composite_projection(self):
        """Inference-only algebra: AttentionNet.0's halves are folded into the profile projections, so that the attention
        pre-activations come straight out of the two sweeps over the F-wide profiles and the (I, E) x (E, H) GEMMs disappear:

            Pr = (R·W_Iᵀ + b_I)·A1rᵀ       = R·(A1r·W_I)ᵀ + A1r·b_I              rated side:      [Pr | Q]  = R·[A1r·W_I ; W_U]ᵀ + [A1r·b_I ; 0]
            Pc = (C·W_Iᵀ + b_I)·A1cᵀ + a1  = C·(A1c·W_I)ᵀ + (A1c·b_I + a1)        candidate side:  [Ec | Pc] = C·[W_I ; A1c·W_I]ᵀ + [b_I ; A1c·b_I + a1]

        (Er itself is only needed by the training-mode isclose() mask, attention_ncf.py:199.)  The composites are formed in
        float64 and rounded once; the results differ from the two-step order by ~1e-7 relative, inside the fp32 tolerance.
        Returns (Wr, br, Wc, bc, bU, a2, a20, H) or None when the variant does not apply; cached per parameter version."""
        halves = self._attention_halves()
        if halves is None:
            return None
        item, user, first = self.ItemEmbeddings[0], self.UserEmbeddings[0], self.AttentionNet[0]
        params = (item.weight, item.bias, user.weight, user.bias, first.weight, first.bias, self.AttentionNet[3].weight)

        def compose():
            with torch.no_grad():
                A1c, A1r, a1, a2, a20 = halves
                WI, bI = item.weight.double(), item.bias.double()
                WU, bU = _pad_rows(user.weight.detach(), user.bias.detach())
                Wr = torch.cat(((A1r.double() @ WI).float(), WU), 0).contiguous()
                br = torch.cat(((A1r.double() @ bI).float(), torch.zeros_like(bU)), 0).contiguous()
                Wc = torch.cat((item.weight.detach(), (A1c.double() @ WI).float()), 0).contiguous()
                bc = torch.cat((item.bias.detach(), (A1c.double() @ bI + a1.double()).float()), 0).contiguous()
            return Wr, br, Wc, bc, bU, a2, a20, A1r.shape[0]
        return self._comp_cache.get(params, compose)

    def _attention_halves(self):
        """(A1c, A1r, a1, a2, head bias) of AttentionNet as STABLE view objects (so their MMA-ready packed copies stay cached)
        — only for the Linear-ReLU-Linear variant with att_dense % 4 == 0; None otherwise."""
        if self.use_cos_sim_instead or len(self.AttentionNet) == 1 or self.AttentionNet[0].weight.shape[0] % 4:
            return None
        first, head = self.AttentionNet[0], self.AttentionNet[3]
        w, E = first.weight, first.weight.shape[1] // 2
        return self._att_cache.get((w, first.bias, head.weight, head.bias), lambda: (
            w.detach()[:, :E], w.detach()[:, E:], first.bias.detach(), head.weight.detach().view(-1), head.bias.detach()))

    def forward(self, candidate_items, rated_items, user_matrix, return_attention_weights=False):
        item, user = self.ItemEmbeddings[0], self.UserEmbeddings[0]
        E, U = item.weight.shape[0], user.weight.shape[0]
        no_grad = not (torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters()))
        comp = self._composite_projection() if (no_grad and not self.training) else None
        if comp is not None:
            # inference: two sweeps over the F-wide profiles give everything K2 and the MLP need (see _composite_projection).
            # The rated-item sweep fills the device exactly at config 2 (74 x 2 tiles on 148 SMs — adding the candidates' 4
            # row tiles to that launch costs a second wave, measured 132 vs 71 us), so the candidates keep their own GEMM.
            Wr, br, Wc, bc, bU, a2, a20, H = comp
            EcPc = ops.linear_raw(candidate_items, Wc, bc)                              # :150 (+ candidate half of :176)
            PrQ = ops.linear_raw(rated_items, Wr, br)                                   # :151 folded with :176, + Q = R·W_Uᵀ
            Ec, Pc = EcPc[:, :E], EcPc[:, E:]
            Pr, Q = PrQ[:, :H], PrQ[:, H:]
            mode = L.ATT_NET
        else:
            Wcat, bcat, bU = self._stacked_projection()
            Ec = ops.linear(candidate_items, item.weight, item.bias)                    # :150
            # one sweep over rated_items: item embedding (:151) and Q = rated_items·W_Uᵀ (pooling moved into embedding
            # space: W_U(Σ α·um·R_i) = Σ α·um·(W_U R_i), :213+:216)
            ErQ = ops.linear(rated_items, Wcat, bcat)
            Er, Q = ErQ[:, :E], ErQ[:, E:]
            Pc, Pr, mode, a2, a20 = self._score_tables(Ec, Er)

        um, scale, drop_zero, train_mask = user_matrix, 1.0, False, None
        if self.training:
            if self.message_dropout is not None:                                        # :185-189
                drop_zero = True
                if self.message_dropout > 0.0:
                    keep = torch.rand_like(um) >= self.message_dropout
                    um = um * keep                   # a dropped pair gets -inf, i.e. behaves like "unrated"
                    scale = 1.0 / (1.0 - self.message_dropout)
            train_mask = (Ec, Er, 1e-5, 1e-5)                                           # isclose(atol=1e-5) (:199)
        inner = None
        if self.training and mode == L.ATT_NET and len(self.AttentionNet) > 1:
            p_inner = float(self.AttentionNet[2].p)                                     # Linear -> ReLU -> Dropout(p) -> Linear (:112-117)
            if p_inner > 0.0:
                # the mask is a Philox stream keyed by a seed drawn from torch's default generator (reproducible under torch.manual_seed); it
                # cannot be bit-matched to torch's own dropout stream, like every other dropout of the reference (DESIGN.md §5)
                # drawn ON the device (no host round trip, and a captured training step gets a new mask on every replay)
                inner = (p_inner, torch.randint(0, 2 ** 62, (1,), dtype=torch.int64, device=Pc.device))
        res = ops.attention_pool(Pc, Pr, Q, mode=mode, a2=a2, a20=a20,
                                 bU=bU, user_matrix=um, return_attention_weights=return_attention_weights,
                                 train_mask=train_mask, drop_zero_scores=drop_zero, score_scale=scale, inner_dropout=inner)
        user_emb, att = res if return_attention_weights else (res, None)
        if user_emb.shape[1] != U:
            user_emb = user_emb[:, :U]
        out = run_mlp(self.MLP, Ec, user_emb, training=self.training)                   # :219-222
        return (out, att.detach()) if return_attention_weights else out

    def forward_resident(self, candidate_items, rated_items, user_matrix, return_attention_weights=False):
        """`forward` fed by a device-resident provider (content_providers.ResidentDynamicProvider): `candidate_items` /
        `rated_items` are `ResidentRows` (row numbers into the profile table in HBM), `user_matrix` a `SparseUserMatrix` (CSR).
        Per call ~2.4 MB cross PCIe instead of 103 MB; the gather of the rated rows is fused into the projection GEMM
        (`row_index`), K2 reads the CSR directly.  Same kernels, same order of operations -> identical results."""
        table = rated_items.table
        dev = table.device
        if self.training or (torch.is_grad_enabled() and any(p.requires_grad for p in self.parameters())):
            # training keeps the reference's dense contract (embedding mask, dropout): materialise on the device
            return self.forward(candidate_items.dense(), rated_items.dense(), user_matrix.to_dense().to(dev),
                                return_attention_weights=return_attention_weights)
        item, user = self.ItemEmbeddings[0], self.UserEmbeddings[0]
        E, U = item.weight.shape[0], user.weight.shape[0]
        cand_pos = candidate_items.pos.to(dev, non_blocking=True)
        rated_pos = rated_items.pos.to(dev, non_blocking=True)
        csr = tuple(t.to(dev, non_blocking=True) for t in (user_matrix.row_ptr, user_matrix.col, user_matrix.val))
        comp = self._composite_projection()
        if comp is not None:
            Wr, br, Wc, bc, bU, a2, a20, H = comp
            EcPc = ops.linear_raw(table.index_select(0, cand_pos), Wc, bc)
            PrQ = ops.linear_raw(table, Wr, br, row_index=rated_pos)
            Ec, Pc = EcPc[:, :E], EcPc[:, E:]
            Pr, Q = PrQ[:, :H], PrQ[:, H:]
            mode = L.ATT_NET
        else:
            Wcat, bcat, bU = self._stacked_projection()
            Ec = ops.linear_raw(table.index_select(0, cand_pos), item.weight, item.bias)
            ErQ = ops.linear_raw(table, Wcat, bcat, row_index=rated_pos)
            Er, Q = ErQ[:, :E], ErQ[:, E:]
            Pc, Pr, mode, a2, a20 = self._score_tables(Ec, Er)
        res = ops.attention_pool_raw(Pc, Pr, Q, mode=mode, a2=a2, a20=a20, bU=bU, csr=csr,
                                     return_attention_weights=return_attention_weights, max_row_nnz=getattr(user_matrix, 'max_row_nnz', 0))
        user_emb, att = res if return_attention_weights else (res, None)
        if user_emb.shape[1] != U:
            user_emb = user_emb[:, :U]
        out = run_mlp(self.MLP, Ec, user_emb, training=False)
        return (out, att) if return_attention_weights else out

    def recommend_for_user(self, item_profiles, rated_positions, rated_ratings, k=10, ignore_seen=True, explain_factor=1.5,
                           explain_constant=0.025):
        """The reference's serving call (src/webapp/backend.py:78-121 `recommend_for_user`) on the device: every item of the
        catalogue is a candidate for ONE user described by the items they rated.

        item_profiles (nI, F) CUDA fp32; rated_positions (R,) int64 rows of `item_profiles` the user rated (any order, unique);
        rated_ratings (R,) raw ratings.  Returns a dict: `items` (k,) catalogue rows sorted by score, `scores` (k,), and per
        recommended item the rated items whose attention weight exceeds `explain_factor / R + explain_constant` (:105-110):
        `because` (list of k int64 tensors of catalogue rows) and `attention` (their weights)."""
        if self.training:
            raise RuntimeError('recommend_for_user() is an inference call: model.eval() first')
        dev = item_profiles.device
        rated_positions = rated_positions.to(dev).long()
        order = torch.argsort(rated_positions)                                          # np.sort(np.unique(...)) (:89)
        rated_sorted = rated_positions[order]
        ratings = rated_ratings.to(dev).double()[order]
        centred = (ratings - (ratings.mean() + 2.5) / 2).float()                        # (:93)
        if ignore_seen:                                                                 # item_features.drop(...) (:85)
            keep = torch.ones(item_profiles.shape[0], dtype=torch.bool, device=dev)
            keep[rated_sorted] = False
            cand_rows = keep.nonzero().view(-1)
        else:
            cand_rows = torch.arange(item_profiles.shape[0], device=dev)
        with torch.no_grad():
            um = centred.view(1, -1).expand(cand_rows.numel(), -1).contiguous()        # the same row B times (:93)
            y, att = self.forward(item_profiles[cand_rows], item_profiles[rated_sorted], um, return_attention_weights=True)
            val, top = ops.topk_rows(y.view(1, -1), min(k, cand_rows.numel()))
        top = top.view(-1)
        thr = explain_factor * (1.0 / max(rated_sorted.numel(), 1)) + explain_constant  # (:102)
        att_top = att[top]
        mask = att_top > thr
        return {'items': cand_rows[top], 'scores': val.view(-1),
                'because': [rated_sorted[m] for m in mask], 'attention': [a[m] for a, m in zip(att_top, mask)]}

    # ------------------------------------------------------------------------------------------------------------------
    def _recommend_tables(self, item_profiles):
        """Catalogue tables of `recommend`, one GEMM over the (nI, F) profiles per weight version.  The candidate and rated sides are the
        same catalogue, and the user-embedding half of the first MLP Linear is folded into the pooled table (W1 = [W1e | W1u], item first,
        attention_ncf.py:219; user_emb = Σ α·um·Q + b_U):

            h1_pre[b] = Ai[b] + Σ_i α_bi·um_i·Q'[i],   Ai = Ec·W1eᵀ + (b1 + W1u·b_U),   Q' = Q·W1uᵀ = R·(W1u·W_U)ᵀ

        so no per-pair (U x H1) GEMM is left.  Composites are formed in float64 and rounded once, like `_composite_projection`.
        Returns (Pc, Pr, mode, a2, a20, Ai, Qp, H1) with Ai / Qp zero-padded to H1P in {32, 64, 128, 256} columns; cached on the profile
        tensor (identity, `_version`, shape) and the parameter versions."""
        weights, biases, _ = mlp_parameters(self.MLP)
        if len(weights) < 2:
            raise NotImplementedError('recommend(): the MLP needs at least one hidden layer (the kernel ends at the first hidden ReLU)')
        H1 = weights[0].shape[0]
        if H1 > 256:
            raise NotImplementedError(f'recommend(): first MLP layer of width {H1} > 256 is not supported')
        H1P = max(32, 1 << (H1 - 1).bit_length())
        E = self.ItemEmbeddings[0].weight.shape[0]
        if self.use_cos_sim_instead:                                   # width of the score tables K8 stages in shared memory
            H = (E + 3) // 4 * 4
        else:
            H = (self.AttentionNet[0].weight.shape[0] + 3) // 4 * 4 if len(self.AttentionNet) > 1 else 4
        if H > 256:
            raise NotImplementedError(f'recommend(): attention width {H} > 256 is not supported')
        item, user = self.ItemEmbeddings[0], self.UserEmbeddings[0]

        def build():
            self._rec_bf16.clear()                                                         # the bf16 copy of Q' goes with the old tables
            R = item_profiles if item_profiles.dtype == torch.float32 else item_profiles.float()
            WI, bI, WU, bU = (t.detach().double() for t in (item.weight, item.bias, user.weight, user.bias))
            W1, b1 = weights[0].detach().double(), biases[0].detach().double()
            W1e, W1u = W1[:, :E], W1[:, E:]
            pad = H1P - H1
            Wa = torch.nn.functional.pad(W1e @ WI, (0, 0, 0, pad))                         # (H1P, F)
            ba = torch.nn.functional.pad(W1e @ bI + b1 + W1u @ bU, (0, pad))
            Wq = torch.nn.functional.pad(W1u @ WU, (0, 0, 0, pad))
            bq = torch.zeros(H1P, dtype=torch.float64, device=Wq.device)
            halves = self._attention_halves()
            if halves is not None:                                                         # AttentionNet, att_dense % 4 == 0: composites
                A1c, A1r, a1, a2, a20 = halves
                H = A1r.shape[0]
                A1c, A1r = A1c.double(), A1r.double()
                W = torch.cat((Wa, A1c @ WI, A1r @ WI, Wq), 0)
                b = torch.cat((ba, A1c @ bI + a1.double(), A1r @ bI, bq), 0)
                T = ops.linear_raw(R, W.float().contiguous(), b.float().contiguous())
                Ai, Pc, Pr, Qp = T[:, :H1P], T[:, H1P:H1P + H], T[:, H1P + H:H1P + 2 * H], T[:, H1P + 2 * H:]
                mode = L.ATT_NET
            else:                                                                          # cosine, att_dense=None, att_dense % 4 != 0
                Ep = (E + 3) // 4 * 4
                W = torch.cat((torch.nn.functional.pad(WI, (0, 0, 0, Ep - E)), Wa, Wq), 0)
                b = torch.cat((torch.nn.functional.pad(bI, (0, Ep - E)), ba, bq), 0)
                T = ops.linear_raw(R, W.float().contiguous(), b.float().contiguous())
                Ec, Ai, Qp = T[:, :E], T[:, Ep:Ep + H1P], T[:, Ep + H1P:]
                Pc, Pr, mode, a2, a20 = self._score_tables(Ec, Ec)
                Pc, Pr = Pc.detach().contiguous(), Pr.detach().contiguous()
            return Pc, Pr, mode, a2, a20, Ai, Qp, H1
        with torch.no_grad():                          # constants of the catalogue and the weights: cached in any grad mode, like the forward's
            return self._rec_cache.get((item_profiles, *self.parameters()), build)

    def recommend(self, item_profiles, list_ptr, list_item, list_val, k=10, users=None, ignore_seen=True, return_scores=False, chunk_users=None,
                  precision='fp32'):
        """Top-k catalogue items for many users at once: the reference's serving call (src/webapp/backend.py:78-121, one user x every
        catalogue item, attention_ncf.py:136-224) batched over users.

        item_profiles (nI, F) CUDA fp32 — the catalogue, every row a candidate.  The rating lists use K6's resident format (a
        `DeviceCollateProvider` feeds it directly: `prov.table, prov.d_list_ptr, prov.d_list_item, prov.d_list_val`): list_ptr int64
        (rows+1), list_item int32 catalogue rows ascending per user, list_val fp32 ALREADY centred (an entry of exactly 0.0 gets no
        attention).  `users` int64 list rows (default: every row; duplicates allowed).  `ignore_seen` leaves a user's own list items out.
        Users are processed `chunk_users` at a time (default: an h1 slab of about RECOMMEND_SLAB_BYTES): the working memory is bounded by
        the chunk, whatever the number of users; the whole (nU, nI) score matrix is only allocated with `return_scores=True`.

        Pipeline per chunk: K8 (csrc/attention_recommend.cu: attention pooling over the shared list, h1 slab) on the cached catalogue tables
        (`_recommend_tables`), the remaining MLP layers on the slab (K1a), seen pairs set to NaN, `ops.topk_rows`.
        precision 'fp32' (default, max-norm relative error <= 1e-5) or 'bf16' (<= 1e-2): the attention scores, the softmax and α are the fp32 ones,
        bit for bit (so `explain` of a bf16 call's items is that of an fp32 call), the pooling runs on bf16 tensor cores (K8b: Q' and the
        weights α·um rounded to bf16, fp32 accumulation) and the hidden layers after the first on K1a's bf16 engine; the output layer is the
        fp32 path's.  The bf16 copy of Q' is made on the first bf16 call and cached with the catalogue tables.
        Returns (top_scores (nU, k) fp32, top_items (nU, k) int64 catalogue rows, padded with (-inf, -1)[, scores (nU, nI)])."""
        if self.training:
            raise RuntimeError('recommend() is an inference call: model.eval() first')
        if precision not in ('fp32', 'bf16'):
            raise ValueError(f"recommend(): precision must be 'fp32' or 'bf16', not {precision!r}")
        ops._require_cuda(item_profiles, list_ptr, list_item, list_val, users)
        if list_ptr.dtype != torch.int64 or list_item.dtype != torch.int32 or list_val.dtype != torch.float32:
            raise ValueError('recommend(): list_ptr must be int64, list_item int32 and list_val float32')
        if not 1 <= k <= 64:
            raise ValueError('recommend(): need 1 <= k <= 64')
        dev = item_profiles.device
        nI = item_profiles.shape[0]
        n_rows = list_ptr.numel() - 1
        users = torch.arange(max(n_rows, 0), device=dev) if users is None else users.to(dev).long().contiguous()
        nU = users.numel()
        self._check_lists(list_ptr, list_item, list_val, users, nI)
        weights, biases, _ = mlp_parameters(self.MLP)
        with torch.no_grad():
            Pc, Pr, mode, a2, a20, Ai, Qp, H1 = self._recommend_tables(item_profiles)
            hidden = None
            if precision == 'bf16':
                Qp = self._rec_bf16.get((Qp,), lambda: Qp.to(torch.bfloat16, memory_format=torch.contiguous_format))
                # K = H1 <= 256 is below ops.TC_MIN_K, where the default routing picks the FFMA GEMM: force the bf16 tensor cores
                hidden = 'bf16!'
            H1P = Ai.shape[1]
            if chunk_users is None:
                chunk_users = max(1, RECOMMEND_SLAB_BYTES // max(1, nI * H1P * 4))
            chunk_users = int(max(1, min(chunk_users, 65535)))
            val = torch.full((nU, k), float('-inf'), dtype=torch.float32, device=dev)
            idx = torch.full((nU, k), -1, dtype=torch.int64, device=dev)
            scores = torch.empty((nU, nI), dtype=torch.float32, device=dev) if return_scores else None
            last = len(weights) - 1
            for s in range(0, nU if nI > 0 else 0, chunk_users):
                uc = users[s:s + chunk_users]
                n = uc.numel()
                sc = scores[s:s + n] if scores is not None else torch.empty((n, nI), dtype=torch.float32, device=dev)
                x = ops.attention_recommend_raw(Pc, Pr, Ai, Qp, mode=mode, a2=a2, a20=a20, list_ptr=list_ptr, list_item=list_item,
                                                list_val=list_val, users=uc)[:, :H1]
                for li in range(1, last):
                    x = ops.linear_raw(x, weights[li], biases[li], relu=True, engine=hidden)
                ops.linear_raw(x, weights[last], biases[last], out=sc.view(n * nI, 1))
                del x
                if ignore_seen:                                        # item_features.drop(...) (backend.py:85): never selected by the top-k
                    self._mask_seen(sc, uc, list_ptr, list_item)
                val[s:s + n], idx[s:s + n] = ops.topk_rows(sc, k)
        return (val, idx, scores) if return_scores else (val, idx)

    def explain(self, item_profiles, list_ptr, list_item, list_val, items, users=None, explain_factor=1.5, explain_constant=0.025):
        """Explanations of many users' recommendations: the reference's "because you liked ..." (src/webapp/backend.py:102-110) for the output
        of `recommend`, in one call.  `val, idx = m.recommend(...)` followed by `m.explain(..., idx, users=...)` covers the whole serving call.

        item_profiles, list_ptr, list_item, list_val and `users` as for `recommend`.  `items` (len(users), k) int64 catalogue rows, 1 <= k <= 64,
        -1 = padding (exactly `recommend`'s top_items; any catalogue row is accepted, also a user's own list items).  Entry i of user u's list
        explains candidate b when α_bi > explain_factor / max(R_u, 1) + explain_constant — `recommend_for_user`'s rule: R_u = length of u's list,
        zero-centred entries included; α_bi = the eval-mode attention weight `forward(..., return_attention_weights=True)` reports.
        Zero-centred entries have α = 0 and never explain; an empty list explains nothing.

        K9 (csrc/attention_explain.cu) on `recommend`'s cached catalogue tables: after a `recommend` call on the same profiles and weights no
        projection GEMM runs.  Returns (ptr (nU·k + 1,) int64, because (n,) int64 catalogue rows, attention (n,) fp32): row u·k + j explains
        items[u, j] with because[ptr[r]:ptr[r+1]], in list order (ascending catalogue row); padding rows are empty."""
        if self.training:
            raise RuntimeError('explain() is an inference call: model.eval() first')
        ops._require_cuda(item_profiles, list_ptr, list_item, list_val, users, items)
        if list_ptr.dtype != torch.int64 or list_item.dtype != torch.int32 or list_val.dtype != torch.float32:
            raise ValueError('explain(): list_ptr must be int64, list_item int32 and list_val float32')
        if items.dtype != torch.int64 or items.dim() != 2:
            raise ValueError('explain(): items must be a (len(users), k) int64 tensor')
        if not 1 <= items.shape[1] <= 64:
            raise ValueError('explain(): need 1 <= k <= 64')
        dev = item_profiles.device
        nI = item_profiles.shape[0]
        users = torch.arange(max(list_ptr.numel() - 1, 0), device=dev) if users is None else users.to(dev).long().contiguous()
        if items.shape[0] != users.numel():
            raise ValueError(f'explain(): items has {items.shape[0]} rows for {users.numel()} users')
        self._check_lists(list_ptr, list_item, list_val, users, nI, 'explain')
        if items.numel() and bool(((items < -1) | (items >= nI)).any()):
            raise ValueError(f'explain(): items must hold catalogue rows in [0, {nI}) or -1')
        with torch.no_grad():
            Pc, Pr, mode, a2, a20 = self._recommend_tables(item_profiles)[:5]
            return ops.attention_explain_raw(Pc, Pr, mode=mode, a2=a2, a20=a20, list_ptr=list_ptr, list_item=list_item, list_val=list_val,
                                             users=users, items=items, explain_factor=explain_factor, explain_constant=explain_constant)

    @staticmethod
    def _check_lists(list_ptr, list_item, list_val, users, nI, what='recommend'):
        """Host-side range checks of the rating lists and user rows (one device read-back): K8 and K9 read `list_ptr[users]` and the table rows
        `list_item[...]` without bounds checks."""
        n_rows = list_ptr.numel() - 1
        if n_rows < 0:
            raise ValueError(f'{what}(): list_ptr needs at least one element')
        z = torch.zeros((), dtype=torch.bool, device=list_ptr.device)
        flags = torch.stack((
            ((users < 0) | (users >= n_rows)).any() if users.numel() else z,
            (list_ptr[0] != 0) | (list_ptr[-1] > min(list_item.numel(), list_val.numel())) | ((list_ptr[1:] < list_ptr[:-1]).any() if n_rows else z),
            ((list_item < 0) | (list_item >= nI)).any() if list_item.numel() else z)).tolist()
        if flags[0]:
            raise ValueError(f'{what}(): `users` must be list rows in [0, {n_rows})')
        if flags[1]:
            raise ValueError(f'{what}(): list_ptr must start at 0, be non-decreasing and end within list_item / list_val')
        if flags[2]:
            raise ValueError(f'{what}(): list_item must hold catalogue rows in [0, {nI})')

    @staticmethod
    def _mask_seen(scores, users, list_ptr, list_item):
        """scores[r, list_item of users[r]] = NaN for every list entry of every row r"""
        start, lens = list_ptr[users], list_ptr[users + 1] - list_ptr[users]
        total = int(lens.sum())
        if total:
            dev = scores.device
            rows = torch.repeat_interleave(torch.arange(users.numel(), device=dev), lens, output_size=total)
            first = torch.repeat_interleave(start - (torch.cumsum(lens, 0) - lens), lens, output_size=total)
            scores[rows, list_item[first + torch.arange(total, device=dev)].long()] = float('nan')
