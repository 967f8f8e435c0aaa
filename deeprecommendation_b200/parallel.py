"""Multi-GPU GraphNCF propagation (SURVEY.md §8e).  Two schemes over the same nnz-balanced 1-D partition:

  'reduce' (default)  users are partitioned, the (much smaller) item side is replicated.  Rank r owns a range of user
                      rows; per layer it computes  (a) the partial item update from ITS users' edges and (b) its own user
                      rows from the replicated item table, and ONE all-reduce of the (nI, d) item partials replaces the
                      all-gather of all N rows — 32 MB instead of 115 MB per layer on the MovieLens-25M shape, and it
                      overlaps with (b).  After the last layer only the 2B batch rows are exchanged.
  'gather'            both node types partitioned, per-layer all-gather of the transformed features (below).

1-D row partition of the node embeddings with a per-layer all-gather:

One process per GPU (torch.distributed, NCCL over NVLink/NVSwitch).  Destination rows of the neighbour index are split
into P contiguous ranges with (nearly) equal numbers of EDGES — degrees are heavy-tailed, equal row counts would not
balance.  Rank r owns rows [splits[r], splits[r+1]) of x, of the CSR and of every output.  Per layer:

    t_own   = dinv ∘ (W_type x_own + b_type)          K1a, written straight into rank r's slot of the gather buffer
    T       = all_gather(t_own)                        (P, max_rows, d) padded slots; NCCL, in place, one per node type
    x'_own  = dinv ∘ (A_own · T)                       K3 over the local rows; `col` was remapped once to slot addressing

BasicNCF / AttentionNCF need no collective: pairs are sharded across ranks (bench.py).

The partition arithmetic (`split_rows`, `RowPartition`) is pure torch so that world_size-2 gloo tests cover it on CPU
(tests/test_parallel_cpu.py); the propagation itself only runs on CUDA.
"""
from __future__ import annotations

import torch

from . import ops
from .graph import GraphIndex, get_index


def split_rows(row_ptr: torch.Tensor, parts: int) -> list:
    """P+1 row boundaries such that every part holds ~nnz/P entries (ties broken towards more rows on the left)."""
    n_rows = int(row_ptr.numel() - 1)
    nnz = int(row_ptr[-1])
    targets = torch.tensor([(nnz * k) // parts for k in range(1, parts)], dtype=row_ptr.dtype, device=row_ptr.device)
    cuts = torch.searchsorted(row_ptr[1:].contiguous(), targets, right=False) + 1 if parts > 1 else targets
    splits = [0] + [min(int(c), n_rows) for c in cuts.tolist()] + [n_rows]
    for k in range(1, len(splits)):                      # monotone even for degenerate graphs
        splits[k] = max(splits[k], splits[k - 1])
    return splits


class RowPartition:
    """Ownership map of the N node rows and the slot addressing of the gathered feature buffer."""

    def __init__(self, splits, rank: int):
        self.splits, self.rank, self.parts = list(splits), rank, len(splits) - 1
        self.r0, self.r1 = self.splits[rank], self.splits[rank + 1]
        self.rows = self.r1 - self.r0
        self.max_rows = max(b - a for a, b in zip(self.splits[:-1], self.splits[1:]))
        self.max_rows = max(1, (self.max_rows + 3) // 4 * 4)

    def slot_index(self, ids: torch.Tensor) -> torch.Tensor:
        """global node id -> row of the (P * max_rows, d) gathered buffer"""
        bounds = torch.tensor(self.splits[1:-1], dtype=ids.dtype, device=ids.device)
        owner = torch.searchsorted(bounds, ids, right=True) if self.parts > 1 else torch.zeros_like(ids)
        starts = torch.tensor(self.splits[:-1], dtype=ids.dtype, device=ids.device)
        return owner * self.max_rows + (ids - starts[owner])

    def local_csr(self, row_ptr, col, *per_edge):
        """slices of a full CSR for the owned rows; `col` comes back in slot addressing"""
        k0, k1 = int(row_ptr[self.r0]), int(row_ptr[self.r1])
        lrp = (row_ptr[self.r0:self.r1 + 1] - k0).contiguous()
        lcol = self.slot_index(col[k0:k1].long()).to(col.dtype).contiguous()
        return (lrp, lcol) + tuple(None if a is None else a[k0:k1].contiguous() for a in per_edge)


class _LocalIndex(GraphIndex):
    """GraphIndex over a set of owned rows only (no edge lists).  `w_bwd` = weight of the reverse edge of every entry (the backward of
    the partitioned training, peer.py); `pair_hash` is built on first use."""

    def __init__(self, row_ptr, col, w, pos, dinv_own, chunk, w_bwd=None):
        self.row_ptr, self.col, self.w, self.pos = row_ptr, col, w, pos
        self.dinv = dinv_own
        self.num_nodes = int(row_ptr.numel() - 1)
        self.e1, self.e2 = int(col.numel()), 0
        self.chunk_size = chunk
        self.symmetric, self.w_bwd, self._hash = False, w_bwd, None
        if self.num_nodes == 0:                      # a rank without rows of this type (more ranks than users): no SpMM ever runs on it
            empty = torch.zeros(0, dtype=torch.int32, device=row_ptr.device)
            self.n_chunks = self.n_multi = self.n_slots = 0
            self.chunk_row = self.chunk_start = self.chunk_slot = self.multi_row = self.multi_first_slot = self.multi_n_slots = empty
            return
        self._build_plan()

    def pair_hash(self, node0):
        """(keys int64, vals int32, capacity) of the pair hash (source row node0 + r, column) -> CSR entry of this index's entries (the
        `b200rec_pairhash_build` format; a shard's user index: user node -> item).  Identical pairs keep their first entry, which is
        their first interaction position: a row's entries are in position order.  Built on first use."""
        if self._hash is None:
            from . import _lib as L
            from .ops import _ptr, _stream
            dev, n = self.row_ptr.device, int(self.col.numel())
            rows = torch.repeat_interleave(torch.arange(self.num_nodes, device=dev), (self.row_ptr[1:] - self.row_ptr[:-1]).long()) + int(node0)
            edges = torch.stack((rows, self.col.long()))
            cap = 1 << max(4, (2 * n - 1).bit_length())
            keys, vals = torch.empty(cap, dtype=torch.int64, device=dev), torch.empty(cap, dtype=torch.int32, device=dev)
            with torch.cuda.device(dev):
                L.check(L.lib().b200rec_pairhash_build(_ptr(edges), n, _ptr(keys), _ptr(vals), cap, _stream()), 'pairhash_build')
            self._hash = (keys, vals, cap)
        return self._hash


class PartitionedGraph:
    """What rank `rank` keeps of a graph.  Build with `partition_graph`.

    Ownership is per node TYPE: rank r owns an nnz-balanced range of the item rows AND an nnz-balanced range of the user
    rows.  Item rows only gather user features and vice versa (the graph is bipartite), so a layer needs two all-gathers
    — T_items (consumed by the user rows) and T_users (consumed by the item rows) — and the second one is hidden behind
    the first SpMM (see `encode_partitioned`)."""

    def __init__(self, graph, group=None, rank=None, world=None):
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        full = get_index(graph)                      # every rank builds the (cheap, ~10 ms at 50M edges) full index, keeps slices
        nI, N = int(graph.item_features.shape[0]), full.num_nodes
        self.nI, self.N = nI, N
        rp = full.row_ptr
        k_items = int(rp[nI])                        # CSR entries of the item rows come first
        self.items = RowPartition(split_rows(rp[:nI + 1], self.world), self.rank)
        self.users = RowPartition(split_rows(rp[nI:] - k_items, self.world), self.rank)
        it, us = self.items, self.users
        # item rows [it.r0, it.r1): sources are USERS -> slot addressing of T_users (ids shifted by nI)
        k0, k1 = int(rp[it.r0]), int(rp[it.r1])
        cut = lambda a: None if a is None else a[k0:k1].contiguous()
        col_i = us.slot_index(full.col[k0:k1].long() - nI).to(full.col.dtype).contiguous()
        self.dinv_items = full.dinv[it.r0:it.r1].contiguous()
        self.index_items = _LocalIndex((rp[it.r0:it.r1 + 1] - k0).contiguous(), col_i, cut(full.w), cut(full.pos), self.dinv_items,
                                       full.chunk_size)
        # user rows [nI + us.r0, nI + us.r1): sources are ITEMS -> slot addressing of T_items
        k0, k1 = int(rp[nI + us.r0]), int(rp[nI + us.r1])
        col_u = it.slot_index(full.col[k0:k1].long()).to(full.col.dtype).contiguous()
        self.dinv_users = full.dinv[nI + us.r0: nI + us.r1].contiguous()
        self.index_users = _LocalIndex((rp[nI + us.r0: nI + us.r1 + 1] - k0).contiguous(), col_u, cut(full.w), cut(full.pos),
                                       self.dinv_users, full.chunk_size)
        self.edges_total = full.e1 + full.e2
        self.edges_own = int(col_i.numel() + col_u.numel())
        self.item_features = graph.item_features[it.r0:it.r1]
        self.user_features = graph.user_features[us.r0:us.r1]
        self._bufs = None

    def gather_buffers(self, d, device):
        if self._bufs is None or self._bufs[0].shape[1] != d:
            self._bufs = (torch.zeros((self.world * self.items.max_rows, d), dtype=torch.float32, device=device),
                          torch.zeros((self.world * self.users.max_rows, d), dtype=torch.float32, device=device))
        return self._bufs

    def locate(self, ids: torch.Tensor):
        """(owned-by-me mask, local row in my [items | users] block) for global node ids"""
        is_item = ids < self.nI
        it, us = self.items, self.users
        local_item = ids - it.r0
        local_user = ids - self.nI - us.r0
        mine = torch.where(is_item, (local_item >= 0) & (local_item < it.rows), (local_user >= 0) & (local_user < us.rows))
        return mine, torch.where(is_item, local_item, local_user + it.rows)


def column_slice_csr(row_ptr, col, c0: int, c1: int, *per_edge):
    """CSR restricted to the entries whose column lies in [c0, c1), columns renumbered from 0; entry order inside a row is
    kept.  Pure torch (covered by the gloo tests on CPU)."""
    keep = (col >= c0) & (col < c1)
    csum = torch.zeros(col.numel() + 1, dtype=torch.int64, device=col.device)
    csum[1:] = torch.cumsum(keep, 0)
    new_rp = csum[row_ptr.long()].to(row_ptr.dtype).contiguous()
    idx = keep.nonzero().view(-1)
    return (new_rp, (col[idx] - c0).to(col.dtype).contiguous()) + tuple(None if a is None else a[idx].contiguous() for a in per_edge)


class UserPartitionedGraph:
    """Scheme 'reduce': what rank `rank` keeps when users are partitioned and items replicated.

    index_users  CSR of the OWNED user rows; sources are item nodes 0..nI-1, gathered from the replicated (nI, d) table.
    index_items  CSR of ALL item rows restricted to the edges that come from owned users (columns = local user index):
                 its SpMM yields this rank's partial sums of every item row; the all-reduce over ranks completes them
                 (deg^-1/2 of the destination is a per-row factor, so it is applied to the partials)."""

    def __init__(self, graph, group=None, rank=None, world=None):
        import torch.distributed as dist
        self.group = group
        self.rank = dist.get_rank(group) if rank is None else rank
        self.world = dist.get_world_size(group) if world is None else world
        full = get_index(graph)
        nI, N = int(graph.item_features.shape[0]), full.num_nodes
        self.nI, self.N = nI, N
        rp = full.row_ptr
        k_items = int(rp[nI])
        self.users = RowPartition(split_rows(rp[nI:] - k_items, self.world), self.rank)
        us = self.users
        k0, k1 = int(rp[nI + us.r0]), int(rp[nI + us.r1])
        cut = lambda a: None if a is None else a[k0:k1].contiguous()
        self.dinv_users = full.dinv[nI + us.r0: nI + us.r1].contiguous()
        self.dinv_items = full.dinv[:nI].contiguous()
        self.index_users = _LocalIndex((rp[nI + us.r0: nI + us.r1 + 1] - k0).contiguous(), full.col[k0:k1].contiguous(), cut(full.w),
                                       cut(full.pos), self.dinv_users, full.chunk_size)
        head = lambda a: None if a is None else a[:k_items]
        lrp, lcol, lw, lpos = column_slice_csr(rp[:nI + 1], full.col[:k_items], nI + us.r0, nI + us.r1, head(full.w), head(full.pos))
        self.index_items = _LocalIndex(lrp, lcol, lw, lpos, self.dinv_items, full.chunk_size)
        self.edges_total = full.e1 + full.e2
        self.edges_own = int(self.index_users.col.numel() + lcol.numel())
        self.item_features = graph.item_features
        self.user_features = graph.user_features[us.r0:us.r1]

    def locate_users(self, user_nodes: torch.Tensor):
        local = user_nodes - self.nI - self.users.r0
        return (local >= 0) & (local < self.users.rows), local


def partition_graph(graph, group=None, scheme: str = 'peer', d_max: int = 128, batch_max: int = 8192, catalogue_width: int = 0,
                    grad_floats: int = 0):
    """'peer' (default): users partitioned, the exchange written as this library's own kernels over peer-mapped memory (peer.py);
    'reduce' / 'gather': the same partitions with NCCL collectives issued from Python (kept as the comparison baseline).
    `catalogue_width` (scheme 'peer' only): floats per item row of the catalogue section of `peer.recommend_peer`.
    `grad_floats` (scheme 'peer' only): floats per rank of the gradient section of partitioned training (`peer.grad_floats(model)`)."""
    if scheme not in ('peer', 'reduce', 'gather'):
        raise ValueError(scheme)
    if catalogue_width and scheme != 'peer':
        raise ValueError("catalogue_width: only scheme 'peer' serves recommend_peer")
    if grad_floats and scheme != 'peer':
        raise ValueError("grad_floats: only scheme 'peer' trains on a partitioned graph")
    get_index(graph)                                   # (resets a stale partition of an edited graph)
    if scheme == 'peer':
        from .peer import partition_graph_peer
        pg = partition_graph_peer(graph, group, d_max=d_max, batch_max=batch_max, catalogue_width=catalogue_width, grad_floats=grad_floats)
    else:
        pg = UserPartitionedGraph(graph, group) if scheme == 'reduce' else PartitionedGraph(graph, group)
    try:
        object.__setattr__(graph, '_b200rec_partition', pg)
    except Exception:
        pass
    return pg


def encode_partitioned(model, pg: PartitionedGraph):
    """Propagated + combined embeddings of the OWNED rows, ([items_own | users_own], d).  Inference only.

    Per layer (main stream; NCCL runs the gathers on its own stream, `async_op=True`):
        GEMM t_items_own -> T_items slot,  GEMM t_users_own -> T_users slot
        all_gather(T_items) | all_gather(T_users)          issued back to back
        wait(T_items);  SpMM(user rows <- T_items)          overlaps the (larger) T_users gather
        wait(T_users);  SpMM(item rows <- T_users)
    """
    import torch.distributed as dist
    if torch.is_grad_enabled() and any(p.requires_grad for p in model.parameters()):
        raise NotImplementedError('partitioned GraphNCF propagation is inference-only; wrap the call in torch.no_grad()')
    if model.concat or model.convType != 'LightGCN':
        raise NotImplementedError('the partitioned path covers LightGCN with mean combine (concat / LightGAT: single GPU)')
    it, us = pg.items, pg.users
    dev = pg.dinv_items.device
    L_ = len(model.gnn_convs)
    d = model.item_embeddings[0].weight.shape[0]
    ie, ue = model.item_embeddings[0], model.user_embeddings[0]
    ni, nu = it.rows, us.rows
    x0 = torch.empty((ni + nu, d), dtype=torch.float32, device=dev)
    if ni:
        ops.linear_raw(pg.item_features, ie.weight, ie.bias, out=x0[:ni])
    if nu:
        ops.linear_raw(pg.user_features, ue.weight, ue.bias, out=x0[ni:])
    if L_ == 0:
        return x0
    TI, TU = pg.gather_buffers(d, dev)
    slot_i = TI[it.rank * it.max_rows: (it.rank + 1) * it.max_rows]
    slot_u = TU[us.rank * us.max_rows: (us.rank + 1) * us.max_rows]
    acc = torch.empty((ni + nu, d), dtype=torch.float32, device=dev)
    spare = torch.empty((ni + nu, d), dtype=torch.float32, device=dev) if L_ > 1 else None
    lin_u, lin_i, _ = model.gnn_convs[0].typed()
    x = x0
    for l in range(L_):
        if ni:
            ops.linear_raw(x[:ni], lin_i.weight, lin_i.bias, row_scale=pg.dinv_items, out=slot_i[:ni])
        if nu:
            ops.linear_raw(x[ni:], lin_u.weight, lin_u.bias, row_scale=pg.dinv_users, out=slot_u[:nu])
        w_i = w_u = None
        if pg.world > 1:                              # in place: this rank's slot already sits at its position
            w_i = dist.all_gather_into_tensor(TI, slot_i, group=pg.group, async_op=True)
            w_u = dist.all_gather_into_tensor(TU, slot_u, group=pg.group, async_op=True)
        last = l == L_ - 1
        scale = 1.0 / (L_ + 1) if last else 1.0
        src = x0 if l == 0 else acc
        xn = None if last else spare
        if w_i is not None:
            w_i.wait()
        if nu:
            ops.spmm_raw(pg.index_users, TI, w=pg.index_users.w, dinv=pg.dinv_users, x_next=None if xn is None else xn[ni:],
                         acc_in=src[ni:], acc_out=acc[ni:], acc_scale=scale)
        if w_u is not None:
            w_u.wait()
        if ni:
            ops.spmm_raw(pg.index_items, TU, w=pg.index_items.w, dinv=pg.dinv_items, x_next=None if xn is None else xn[:ni],
                         acc_in=src[:ni], acc_out=acc[:ni], acc_scale=scale)
        x = xn
    return acc


def forward_user_partitioned(model, pg: UserPartitionedGraph, userIds, itemIds):
    """GraphNCF.forward under scheme 'reduce' (inference).  Per layer l (main stream; the all-reduce runs on NCCL's stream):

        t_items = dinv ∘ (W_i2u x_items + b)      all items, computed redundantly on every rank (nI x d x d GEMM)
        t_users = dinv ∘ (W_u2i x_users + b)      owned users
        part    = dinv_items ∘ (A[:, owned users] · t_users)        SpMM over ALL item rows, this rank's edges only
        all_reduce(part)  ||  x_users' = dinv_users ∘ (A[owned users, :] · t_items)  (+ running mean, fused)
        x_items' = part

    After the last layer only the batch rows cross NVLink: one all-reduce of a (2B, d) buffer holding the partial item rows
    (sum = the full rows) and the owned user rows (exactly one non-zero contributor each)."""
    import torch.distributed as dist
    from .neural_collaborative_filtering.util import run_mlp
    if torch.is_grad_enabled() and any(p.requires_grad for p in model.parameters()):
        raise NotImplementedError('partitioned GraphNCF propagation is inference-only; wrap the call in torch.no_grad()')
    if model.concat or model.convType != 'LightGCN':
        raise NotImplementedError('the partitioned path covers LightGCN with mean combine (concat / LightGAT: single GPU)')
    dev = pg.dinv_items.device
    L_ = len(model.gnn_convs)
    d = model.item_embeddings[0].weight.shape[0]
    ie, ue = model.item_embeddings[0], model.user_embeddings[0]
    nI, nu = pg.nI, pg.users.rows
    B = userIds.shape[0]
    iid, uid = itemIds.long(), userIds.long()
    x_items = ops.linear_raw(pg.item_features, ie.weight, ie.bias)
    x_users = ops.linear_raw(pg.user_features, ue.weight, ue.bias) if nu else torch.empty((0, d), dtype=torch.float32, device=dev)
    mine, local = pg.locate_users(uid)
    local = local.clamp(0, max(nu - 1, 0))
    rows = torch.zeros((2 * B, d), dtype=torch.float32, device=dev)
    item_sum = x_items[iid]                                        # Σ_l x_l[item] of the layers that are replicated in full
    if L_ == 0:
        if nu:
            rows[B:] = x_users[local] * mine[:, None].to(torch.float32)
        inv = 1.0
    else:
        lin_u, lin_i, _ = model.gnn_convs[0].typed()
        acc_users = torch.empty((nu, d), dtype=torch.float32, device=dev)
        spare = torch.empty((nu, d), dtype=torch.float32, device=dev) if L_ > 1 else None
        t_users = torch.empty((max(nu, 1), d), dtype=torch.float32, device=dev)
        x0_users = x_users
        for l in range(L_):
            last = l == L_ - 1
            t_items = ops.linear_raw(x_items, lin_i.weight, lin_i.bias, row_scale=pg.dinv_items)
            part = torch.zeros((nI, d), dtype=torch.float32, device=dev)          # rows without an owned in-edge stay 0
            if nu:
                ops.linear_raw(x_users, lin_u.weight, lin_u.bias, row_scale=pg.dinv_users, out=t_users[:nu])
                ops.spmm_raw(pg.index_items, t_users, w=pg.index_items.w, dinv=pg.dinv_items, x_next=part)
            work = None
            if last:
                rows[:B] = part[iid]
            elif pg.world > 1:
                work = dist.all_reduce(part, group=pg.group, async_op=True)
            if nu:
                ops.spmm_raw(pg.index_users, t_items, w=pg.index_users.w, dinv=pg.dinv_users, x_next=None if last else spare,
                             acc_in=x0_users if l == 0 else acc_users, acc_out=acc_users, acc_scale=1.0 / (L_ + 1) if last else 1.0)
            if work is not None:
                work.wait()
            if not last:
                x_items, x_users = part, spare
                item_sum = item_sum + x_items[iid]
        if nu:
            rows[B:] = acc_users[local] * mine[:, None].to(torch.float32)
        inv = 1.0 / (L_ + 1)
    if pg.world > 1:
        dist.all_reduce(rows, group=pg.group)
    item_rows = (item_sum + rows[:B]) * inv if L_ > 0 else item_sum
    user_rows = rows[B:]
    if model.MLP is None:
        return ops.rowdot(user_rows, item_rows)
    return run_mlp(model.MLP, item_rows, user_rows, training=False)               # item first (gnn_ncf.py:361)


def forward_partitioned(model, pg, userIds, itemIds):
    """GraphNCF.forward on a partitioned graph (dispatches on the scheme).  After the propagation only the 2B batch rows are exchanged: every rank
    drops the rows it owns into a zero (2B, d) buffer and one all-reduce (exactly one non-zero contributor per row, so
    the sum is exact) gives every rank the batch embeddings; the MLP on B pairs is then computed on every rank."""
    from .peer import PeerShard, forward_peer
    if isinstance(pg, PeerShard):
        return forward_peer(model, pg, userIds, itemIds)
    if isinstance(pg, UserPartitionedGraph):
        return forward_user_partitioned(model, pg, userIds, itemIds)
    import torch.distributed as dist
    from .neural_collaborative_filtering.util import run_mlp
    comb = encode_partitioned(model, pg)
    B = userIds.shape[0]
    ids = torch.cat((itemIds.long(), userIds.long()))
    mine, local = pg.locate(ids)
    # no boolean-mask indexing here: it would force a device->host sync in the middle of every step
    rows = comb[local.clamp(0, comb.shape[0] - 1)] * mine[:, None].to(comb.dtype)
    if pg.world > 1:
        dist.all_reduce(rows, group=pg.group)
    if model.MLP is None:
        return ops.rowdot(rows[B:], rows[:B])
    return run_mlp(model.MLP, rows[:B], rows[B:], training=False)              # item first (gnn_ncf.py:361)
