"""Device-side graph build (K4) and the neighbour index GraphNCF propagates over.

`create_graph` mirrors src/content_providers/graph_providers.py:10-66 (+ the node-id assignment of :76-80) of the
reference, but runs as CUDA kernels over HBM-resident arrays instead of a Python `iterrows()` loop, and is bit-exact
against it (tests/test_graph_build.py).  `GraphData` is the attribute bag the reference gets from
`torch_geometric.data.Data` (only `.to(device)` and attribute access are used, gnn_datasets.py:19-20, gnn_ncf.py:300-311);
GraphNCF accepts either.  `GraphIndex` (CSR by destination + SpMM chunk plan + (src,dst)->position hash) is derived
from the two edge lists once per graph and cached on the graph object.
"""
from __future__ import annotations

import ctypes as C

import torch

from . import _lib as L
from .derived import Derived
from .ops import _ptr, _stream, _require_cuda

SPMM_CHUNK = 256


class GraphData:
    """Attribute bag with `.to(device)` moving tensor attributes only (what the reference uses of PyG's Data)."""

    def __init__(self, **kwargs):
        for k, v in kwargs.items():
            setattr(self, k, v)

    def to(self, device, *args, **kwargs):
        dev = torch.device(device)
        moved = False
        for k, v in list(self.__dict__.items()):
            if torch.is_tensor(v) and v.device != dev:
                setattr(self, k, v.to(dev, *args, **kwargs))
                moved = True
        if moved:                                   # derived structures live on the old device
            for k in ('_b200rec_index', '_b200rec_partition'):
                self.__dict__.pop(k, None)
        return self

    def __repr__(self):
        parts = [f'{k}={list(v.shape)}' if torch.is_tensor(v) else f'{k}={type(v).__name__}'
                 for k, v in self.__dict__.items() if not k.startswith('_')]
        return 'GraphData(' + ', '.join(parts) + ')'


def _i32(n, device, zero=False):
    return (torch.zeros if zero else torch.empty)(int(n), dtype=torch.int32, device=device)


def _ws(nbytes, device):
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


# ----------------------------------------------------------------------------------------------------------------------
# node ids (graph_providers.py:76-80)
# ----------------------------------------------------------------------------------------------------------------------
class IdTable:
    """sorted-unique raw integer id -> rank, as device arrays (`sorted(unique(ids))` + `{id: index}` of the reference)."""

    def __init__(self, all_ids: torch.Tensor):
        _require_cuda(all_ids)
        ids = all_ids.contiguous().long()
        dev = ids.device
        self.bound = int(ids.max().item()) + 1 if ids.numel() else 1
        if ids.numel() and int(ids.min().item()) < 0:
            raise ValueError('ids must be non-negative integers (factorise other id types on the host first)')
        self.flags = _i32(self.bound, dev)
        self.rank = _i32(self.bound + 1, dev)
        err = _i32(1, dev, zero=True)
        lib = L.lib()
        wsb = lib.b200rec_scan_workspace(self.bound)
        ws = _ws(wsb, dev)
        # first pass without the sorted list (its length is only known after the scan)
        with torch.cuda.device(dev):
            L.check(lib.b200rec_id_rank_table(_ptr(ids), ids.numel(), self.bound, _ptr(self.flags), _ptr(self.rank), None, _ptr(err),
                                              _ptr(ws), ws.numel(), _stream()), 'id_rank_table')
        self.count = int(self.rank[self.bound].item())
        self._ids, self._dev, self._sorted = ids, dev, None

    def sorted(self) -> torch.Tensor:
        """The sorted unique ids (node order), materialised on first use by a second pass of the same kernel."""
        if self._sorted is None:
            out = torch.empty(self.count, dtype=torch.int64, device=self._dev)
            err = _i32(1, self._dev, zero=True)
            lib = L.lib()
            ws = _ws(lib.b200rec_scan_workspace(self.bound), self._dev)
            with torch.cuda.device(self._dev):
                L.check(lib.b200rec_id_rank_table(_ptr(self._ids), self._ids.numel(), self.bound, _ptr(self.flags), _ptr(self.rank),
                                                  _ptr(out), _ptr(err), _ptr(ws), ws.numel(), _stream()), 'id_rank_table')
            self._sorted = out
        return self._sorted

    def lookup(self, ids: torch.Tensor, offset: int = 0) -> torch.Tensor:
        ids = ids.contiguous().long()
        out = torch.empty_like(ids)
        err = _i32(1, ids.device, zero=True)
        with torch.cuda.device(ids.device):
            L.check(L.lib().b200rec_id_lookup(_ptr(ids), ids.numel(), self.bound, _ptr(self.flags), _ptr(self.rank), offset, _ptr(out),
                                              _ptr(err), _stream()), 'id_lookup')
        if int(err.item()):
            bad = ids[out < 0][:4].tolist()
            raise KeyError(f'unknown id(s) {bad} (the reference raises KeyError from its id dict)')
        return out


# ----------------------------------------------------------------------------------------------------------------------
# create_graph (graph_providers.py:10-66)
# ----------------------------------------------------------------------------------------------------------------------
def create_graph(user_ids, item_ids, ratings, item_features, user_features, user_table: IdTable, item_table: IdTable,
                 binary: bool = False) -> GraphData:
    """Edge lists + centred-rating attrs of the interaction list, in file order, on the device.

    user_ids / item_ids: raw integer ids (int64) per interaction; ratings: float64 (float32 is widened).
    Returns GraphData(item_features, user_features, user2item_edge_index (2,E1) int64, item2user_edge_index (2,E2) int64,
    user2item_edge_attr / item2user_edge_attr fp32 or None when `binary`)."""
    _require_cuda(user_ids, item_ids, ratings)
    dev = user_ids.device
    lib = L.lib()
    n = int(user_ids.numel())
    nI, nU = item_table.count, user_table.count
    u_node = user_table.lookup(user_ids, offset=nI)            # users after the items (:80)
    i_node = item_table.lookup(item_ids, offset=0)
    r = ratings.contiguous().double()
    cnt_u, cnt_i = _i32(nU, dev, zero=True), _i32(nI, dev, zero=True)
    sum_u = torch.zeros(nU, dtype=torch.float64, device=dev)
    sum_i = torch.zeros(nI, dtype=torch.float64, device=dev)
    attr_u = torch.empty(n, dtype=torch.float32, device=dev)
    attr_i = torch.empty(n, dtype=torch.float32, device=dev)
    keep_u = _i32(n, dev) if binary else None
    keep_i = _i32(n, dev) if binary else None
    with torch.cuda.device(dev):
        st = _stream()
        L.check(lib.b200rec_group_stats(_ptr(u_node), _ptr(r), n, nI, _ptr(cnt_u), _ptr(sum_u), st), 'group_stats')
        L.check(lib.b200rec_group_stats(_ptr(i_node), _ptr(r), n, 0, _ptr(cnt_i), _ptr(sum_i), st), 'group_stats')
        L.check(lib.b200rec_edge_attrs(_ptr(u_node), _ptr(i_node), _ptr(r), n, nI, _ptr(cnt_u), _ptr(sum_u), _ptr(cnt_i), _ptr(sum_i),
                                       _ptr(attr_u), _ptr(attr_i), _ptr(keep_u), _ptr(keep_i), st), 'edge_attrs')
        if not binary:
            u2i = torch.empty((2, n), dtype=torch.int64, device=dev)
            i2u = torch.empty((2, n), dtype=torch.int64, device=dev)
            L.check(lib.b200rec_edge_scatter(_ptr(u_node), _ptr(i_node), n, None, None, n, _ptr(u2i), st), 'edge_scatter')
            L.check(lib.b200rec_edge_scatter(_ptr(i_node), _ptr(u_node), n, None, None, n, _ptr(i2u), st), 'edge_scatter')
        else:
            wsb = lib.b200rec_scan_workspace(n)
            ws = _ws(wsb, dev)
            pos_u, pos_i = _i32(n + 1, dev), _i32(n + 1, dev)
            L.check(lib.b200rec_exclusive_scan_i32(_ptr(keep_u), n, _ptr(pos_u), _ptr(ws), ws.numel(), st), 'scan')
            L.check(lib.b200rec_exclusive_scan_i32(_ptr(keep_i), n, _ptr(pos_i), _ptr(ws), ws.numel(), st), 'scan')
            e1, e2 = int(pos_u[n].item()), int(pos_i[n].item())
            u2i = torch.empty((2, e1), dtype=torch.int64, device=dev)
            i2u = torch.empty((2, e2), dtype=torch.int64, device=dev)
            L.check(lib.b200rec_edge_scatter(_ptr(u_node), _ptr(i_node), n, _ptr(keep_u), _ptr(pos_u), e1, _ptr(u2i), st), 'edge_scatter')
            L.check(lib.b200rec_edge_scatter(_ptr(i_node), _ptr(u_node), n, _ptr(keep_i), _ptr(pos_i), e2, _ptr(i2u), st), 'edge_scatter')
    return GraphData(item_features=item_features, user_features=user_features,
                     user2item_edge_index=u2i, item2user_edge_index=i2u,
                     user2item_edge_attr=None if binary else attr_u, item2user_edge_attr=None if binary else attr_i)


# ----------------------------------------------------------------------------------------------------------------------
# neighbour index
# ----------------------------------------------------------------------------------------------------------------------
class GraphIndex:
    """CSR by destination of cat(user2item, item2user) (stable: ties in file order), deg^-1/2, the SpMM chunk plan and
    the reverse-direction weights for the backward pass."""

    def __init__(self, u2i: torch.Tensor, i2u: torch.Tensor, attr_u2i, attr_i2u, num_nodes: int, chunk: int = SPMM_CHUNK):
        _require_cuda(u2i, i2u)
        dev = u2i.device
        lib = L.lib()
        u2i, i2u = u2i.contiguous().long(), i2u.contiguous().long()
        self.u2i, self.i2u = u2i, i2u
        e1, e2 = int(u2i.shape[1]), int(i2u.shape[1])
        n = e1 + e2
        self.e1, self.e2, self.num_nodes, self.chunk_size = e1, e2, int(num_nodes), int(chunk)
        has_w = attr_u2i is not None and attr_i2u is not None
        if has_w:
            attr_u2i, attr_i2u = attr_u2i.contiguous().float(), attr_i2u.contiguous().float()
        self.row_ptr = _i32(num_nodes + 1, dev)
        self.col = _i32(n, dev)
        self.pos = _i32(n, dev)
        self.w = torch.empty(n, dtype=torch.float32, device=dev) if has_w else None
        self.deg = _i32(num_nodes, dev)
        self.dinv = torch.empty(num_nodes, dtype=torch.float32, device=dev)
        ws = _ws(lib.b200rec_csr_workspace(n, num_nodes), dev)
        with torch.cuda.device(dev):
            st = _stream()
            L.check(lib.b200rec_csr_build(_ptr(u2i), e1, _ptr(i2u), e2, _ptr(attr_u2i) if has_w else None,
                                          _ptr(attr_i2u) if has_w else None, num_nodes, _ptr(self.row_ptr), _ptr(self.col),
                                          _ptr(self.w), _ptr(self.pos), _ptr(self.deg), _ptr(self.dinv), _ptr(ws), ws.numel(), st),
                    'csr_build')
        self._build_plan()
        # the two lists mirror each other position by position when nothing was filtered (binary=False)
        self.symmetric = has_w and e1 == e2
        if self.symmetric:
            p = self.pos.long()
            self.w_bwd = torch.cat((attr_i2u[p[:e1]], attr_u2i[p[e1:]]))     # weight of the reverse edge of every CSR entry
        else:
            self.w_bwd = None
        self._hash = None
        self._attrs = (attr_u2i, attr_i2u) if has_w else None
        self._transposed = None

    def transposed(self) -> 'GraphIndex':
        """Index of the REVERSED edges (CSR by source of this graph): what the backward of a propagation step over a
        non-symmetric graph multiplies by.  Built on first use."""
        if self._transposed is None:
            a = self._attrs or (None, None)
            self._transposed = GraphIndex(self.u2i.flip(0), self.i2u.flip(0), a[0], a[1], self.num_nodes, self.chunk_size)
        return self._transposed

    def _build_plan(self):
        """SpMM chunk plan (chunk_row / chunk_start / chunk_slot + the multi-chunk row lists) for self.row_ptr."""
        lib = L.lib()
        dev = self.row_ptr.device
        n_rows, chunk = int(self.row_ptr.numel() - 1), self.chunk_size
        with torch.cuda.device(dev):
            st = _stream()
            chunk_off, multi_off, slot_off = (_i32(n_rows + 1, dev) for _ in range(3))
            pws = _ws(lib.b200rec_spmm_plan_workspace(n_rows), dev)
            L.check(lib.b200rec_spmm_plan_count(_ptr(self.row_ptr), n_rows, chunk, _ptr(chunk_off), _ptr(multi_off), _ptr(slot_off),
                                                _ptr(pws), pws.numel(), st), 'spmm_plan_count')
            totals = torch.stack([chunk_off[-1], multi_off[-1], slot_off[-1]]).tolist()     # one D2H sync per graph build
            self.n_chunks, self.n_multi, self.n_slots = (int(x) for x in totals)
            self.chunk_row, self.chunk_start, self.chunk_slot = (_i32(self.n_chunks, dev) for _ in range(3))
            self.multi_row, self.multi_first_slot, self.multi_n_slots = (_i32(max(self.n_multi, 1), dev) for _ in range(3))
            L.check(lib.b200rec_spmm_plan_fill(_ptr(self.row_ptr), n_rows, chunk, _ptr(chunk_off), _ptr(multi_off), _ptr(slot_off),
                                               _ptr(self.chunk_row), _ptr(self.chunk_start), _ptr(self.chunk_slot),
                                               _ptr(self.multi_row), _ptr(self.multi_first_slot), _ptr(self.multi_n_slots), st),
                    'spmm_plan_fill')

    # (src,dst) -> position in the user2item list: the reference's `pos_df` (graph_providers.py:54)
    def positions(self, user_nodes: torch.Tensor, item_nodes: torch.Tensor) -> torch.Tensor:
        dev = self.u2i.device
        lib = L.lib()
        if self._hash is None:
            cap = 1 << max(4, (2 * self.e1 - 1).bit_length())
            keys = torch.empty(cap, dtype=torch.int64, device=dev)
            vals = _i32(cap, dev)
            with torch.cuda.device(dev):
                L.check(lib.b200rec_pairhash_build(_ptr(self.u2i), self.e1, _ptr(keys), _ptr(vals), cap, _stream()), 'pairhash_build')
            self._hash = (keys, vals, cap)
        keys, vals, cap = self._hash
        src, dst = user_nodes.contiguous().long(), item_nodes.contiguous().long()
        out = torch.empty_like(src)
        missing = _i32(1, dev, zero=True)
        with torch.cuda.device(dev):
            L.check(lib.b200rec_pairhash_lookup(_ptr(src), _ptr(dst), src.numel(), _ptr(keys), _ptr(vals), cap, _ptr(out), _ptr(missing),
                                                _stream()), 'pairhash_lookup')
        if int(missing.item()):
            bad = torch.stack([src, dst], 1)[out < 0][:3].tolist()
            raise KeyError(f'{bad}: not edges of the graph (pos_df.loc raises KeyError in the reference, gnn_ncf.py:370)')
        return out

    def masked(self, positions: torch.Tensor):
        """skip bitmap + adjusted deg^-1/2 for a set of interaction positions removed from BOTH lists (gnn_ncf.py:314-320)."""
        if not (self.e1 == self.e2):
            raise NotImplementedError('edge masking needs binary=False graphs (same restriction as the reference, graph_providers.py:13)')
        dev = self.u2i.device
        lib = L.lib()
        skip = _i32((self.e1 + 31) // 32 + 1, dev, zero=True)
        deg = self.deg.clone()
        dinv = torch.empty_like(self.dinv)
        positions = positions.contiguous().long()
        with torch.cuda.device(dev):
            st = _stream()
            L.check(lib.b200rec_mask_targets(_ptr(positions), positions.numel(), self.e1, _ptr(self.u2i), _ptr(self.i2u), _ptr(skip),
                                             _ptr(deg), st), 'mask_targets')
            L.check(lib.b200rec_dinv(_ptr(deg), self.num_nodes, _ptr(dinv), st), 'dinv')
        return skip, dinv

    def seen_items(self, user_nodes: torch.Tensor):
        """CSR (ptr int32 (n+1), idx int32 sorted ascending) of the item nodes each given user node is connected to — the
        `ignore_seen` set of the serving path (src/webapp/backend.py:85).  Rows of the neighbour index are ordered by
        interaction position, so the sources of a user row are sorted here once per call."""
        users = user_nodes.contiguous().long()
        dev = users.device
        start, end = self.row_ptr[users].long(), self.row_ptr[users + 1].long()
        cnt = end - start
        ptr = torch.zeros(users.numel() + 1, dtype=torch.int64, device=dev)
        ptr[1:] = torch.cumsum(cnt, 0)
        total = int(ptr[-1])
        rows = torch.repeat_interleave(torch.arange(users.numel(), device=dev), cnt)
        within = torch.arange(total, device=dev) - ptr[:-1][rows]
        items = self.col[start[rows] + within].long()
        key = torch.sort(rows * self.num_nodes + items).values
        return ptr.int(), (key % self.num_nodes).int()


class StreamPlan:
    """Edge-balanced work plan of the inference SpMM (csrc/spmm_stream.cu) for one CSR + one deg^-1/2 vector: entry stream with the
    last-entry-of-row flag, destination normalisation folded into the entry values, `seg` entries per warp, the partial slots of rows cut
    by segment boundaries.  Built once per (index, dinv, seg) with torch ops — index-build time, not on the propagation path."""

    def __init__(self, row_ptr, col, w, dinv, seg: int):
        dev = row_ptr.device
        n_rows, nnz = int(row_ptr.numel() - 1), int(col.numel())
        self.seg, self.nnz, self.n_rows = int(seg), nnz, n_rows
        rp = row_ptr.long()
        deg = rp[1:] - rp[:-1]
        ne = deg > 0
        self.rows_ne = ne.nonzero().view(-1).int()
        self.rows_empty = (~ne).nonzero().view(-1).int()
        self.n_ne, self.n_empty = int(self.rows_ne.numel()), int(self.rows_empty.numel())
        self.n_segs = (nnz + seg - 1) // seg
        i32 = lambda n: torch.zeros(max(int(n), 1), dtype=torch.int32, device=dev)
        if nnz == 0:
            self.colf, self.wd = i32(1), torch.zeros(1, dtype=torch.float32, device=dev)
            self.seg_first_j = self.seg_head_slot = self.seg_tail_slot = i32(1)
            self.multi_row = self.multi_first_slot = self.multi_n_slots = i32(1)
            self.n_multi = self.n_slots = 0
            return
        start, end = rp[:-1][ne], rp[1:][ne]
        colf = col.int().clone()
        colf[end - 1] += -2 ** 31                                    # bit 31 = last entry of its row (column numbers are < 2^31)
        self.colf = colf
        dst = torch.repeat_interleave(torch.arange(n_rows, device=dev), deg)
        wd = dinv.float()[dst] if dinv is not None else torch.ones(nnz, dtype=torch.float32, device=dev)
        self.wd = (wd * w.float()) if w is not None else wd
        del dst
        first_seg, last_seg = start // seg, (end - 1) // seg
        n_pieces = last_seg - first_seg + 1
        multi = n_pieces > 1
        self.multi_row = self.rows_ne[multi].contiguous()
        mn = n_pieces[multi]
        self.n_multi = int(mn.numel())
        mfirst = torch.cumsum(mn, 0) - mn
        self.multi_n_slots, self.multi_first_slot = mn.int(), mfirst.int()
        self.n_slots = int(mn.sum()) if self.n_multi else 0
        if self.n_multi == 0:
            self.multi_row = self.multi_first_slot = self.multi_n_slots = i32(1)
        slot_base = torch.full((self.n_ne,), -1, dtype=torch.int64, device=dev)
        slot_base[multi] = mfirst
        s_idx = torch.arange(self.n_segs, device=dev)
        s_start = s_idx * seg
        j0 = torch.searchsorted(start, s_start, right=True) - 1       # row holding the segment's first entry
        self.seg_first_j = j0.int()
        head = start[j0] < s_start
        self.seg_head_slot = torch.where(head, slot_base[j0] + (s_idx - first_seg[j0]), torch.full_like(j0, -1)).int()
        e_next = torch.clamp(s_start + seg, max=nnz)                  # one past the segment's last entry
        jl = torch.searchsorted(start, e_next - 1, right=True) - 1
        still_open = end[jl] > e_next
        self.seg_tail_slot = torch.where(still_open, slot_base[jl] + (s_idx - first_seg[jl]), torch.full_like(jl, -1)).int()


def default_stream_seg(nnz: int) -> int:
    """entries per warp: long segments amortise the set-up, but a launch should still be >= ~8 warps per resident warp slot of the GPU"""
    return 256 if nnz >= 24_000_000 else (128 if nnz >= 2_000_000 else 64)


def stream_plan(index, dinv=None, seg=None) -> StreamPlan:
    """cached StreamPlan of a GraphIndex / local index for its own (or the given) deg^-1/2"""
    dinv = index.dinv if dinv is None else dinv
    seg = default_stream_seg(int(index.col.numel())) if seg is None else seg
    plans = index.__dict__.setdefault('_stream_plans', Derived(5))
    return plans.get((dinv, index.w), lambda: StreamPlan(index.row_ptr, index.col, index.w, dinv, seg), seg)


def get_index(graph) -> GraphIndex:
    """GraphIndex of a graph object (ours or the reference's PyG `Data`), built once and cached on it.  Replacing or editing an edge
    list or an attr tensor, or changing the node counts, rebuilds it (and drops a partition of the old graph)."""
    store = graph.__dict__.setdefault('_b200rec_index', Derived(1))
    u2i, i2u = graph.user2item_edge_index, graph.item2user_edge_index
    au, ai = getattr(graph, 'user2item_edge_attr', None), getattr(graph, 'item2user_edge_attr', None)
    n_nodes = int(graph.item_features.shape[0] + graph.user_features.shape[0])

    def build():
        graph.__dict__['_b200rec_partition'] = None
        return GraphIndex(u2i, i2u, au, ai, n_nodes)
    return store.get((u2i, i2u, au, ai), build, n_nodes)
