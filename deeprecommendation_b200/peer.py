"""Partitioned GraphNCF propagation over peer-mapped memory (scheme 'peer'; SURVEY.md §8e, csrc/peer.cu).

Replaces, on the P GPUs of one NVSwitch box, the whole-graph loop of the reference (models/gnn_ncf.py:336-345, recomputed for
every batch) WITHOUT a library collective on the data path.  Ownership (same as scheme 'reduce' of parallel.py):

    users   nnz-balanced contiguous ranges; a rank holds x / acc / t of ITS users only
    items   equal contiguous ranges of `rpp` rows; a rank holds x / acc of its items, and a copy T of the transformed features
            t_items of ALL items (the table its user rows gather from)

Per layer l on rank r (one stream, `par = l & 1` selects one of two copies of every exchange buffer):

    A_l   K3 over ALL item rows restricted to the edges from r's users (sources: local t_users).  Its epilogue stores each
          partial row straight into the OWNER's receive slot recv[par][r] over NVLink  — reduce-scatter fused into the SpMM.
          signal(A)
    B_l   wait(T);  K3 over r's user rows from the table T[par]  (+ the fused running mean)    — hides A_l's stores in flight
    C_l   wait(A);  x_items' = sum of the P receive slots in rank order (deterministic), running mean;
          K1c transform of x_items' whose epilogue writes t_items into T[1-par] of EVERY rank  — all-gather fused into the GEMM.
          signal(T);  t_users for the next layer (local)

After the last layer the owners push the 2B batch rows into every rank's `rows` buffer (peer_gather_rows) and every rank runs the
MLP on the batch.

LightGAT (convType='LightGAT'): the transforms carry no degree scaling and K3 runs the edge softmax over the source scores
ps[s] = a_src·x[s].  In A_l a rank sees only its own users' edges of an item row, so K3 pushes that partial row UNNORMALISED (relative
to its own max m) together with its softmax state (m, l) into the owner's statistics slot; C_l merges the P slots with PyG's rule
(peer_reduce_softmax: M = max m_s, x = Σ acc_s e^(m_s - M) / (Σ l_s e^(m_s - M) + 1e-16)).  B_l needs the score of every item: the owners
publish theirs into the score table S[par] of every rank next to T[par], under the same flag.  User scores stay local.

concat=True: every rank keeps its owned rows of comb = [x0 | x1 | ... | xL]; each layer writes its column block (x_next with a leading
dimension) and the batch rows travel (L+1)·d wide.  signal / wait are epoch flags inside the arenas (release / acquire at system scope; waits time out into an
error flag instead of hanging the GPU), counted on the device so that a captured CUDA graph can be replayed.

Whole-catalogue top-k (`recommend_peer`): the same propagation (`_propagate`, shared with the forward), then

    cat   every owner pushes its final item rows into the section `cat` of EVERY rank (itself included) at rows it_r0 ..;  signal(C)
    score wait(C);  the owned users' rows against cat[:nI] — K5 / relu_dot through ops.mlp_allpairs_topk, or the dot form of relu_dot
    close signal(D);  wait(D)

C orders the pushes before any rank reads the table.  D orders every rank's scoring before the next call of any rank writes `cat` again:
without it a fast rank's next push would overwrite rows a slow rank is still scoring from, and with L = 0 there are no layer flags in
between that could order it.  The propagation sections are ordered exactly as for the forward (a recommend ends with all ranks past D, a
stronger state than the end of a forward), so forwards and recommends can follow each other in any order on the same epoch counters.

Training (`forward_peer` with grad, `train_emulated`; LightGCN, mean combine): the forward above on one stream with per-shard target masking
and dropout (`_train_forward`), then a collective backward (`_train_backward`) that runs the same exchanges in reverse on the reverse-edge weights
`w_bwd` — C' pushes dinv ∘ G of the owned items into T[par] (the all-gather), A' pushes partial item gradients into the owners' recv[par] (the
reduce-scatter) — and ends with the partial parameter gradients pushed into every rank's `grad` section and summed there in rank order (channel G),
so every rank gets the same bits.  A missing-pair count crosses channel M before any data moves.  DESIGN.md §7 has the exchange table.

The arenas are cudaMalloc'd by libb200rec and exchanged as CUDA IPC handles through torch.distributed (plumbing).
`emulated_shards` builds all P shards inside ONE process (plain device buffers, the same kernels and addresses) so that the
exchange logic is covered by the single-GPU test-suite; there the ranks advance in lock step, segment by segment.
"""
from __future__ import annotations

import ctypes as C
import os
import weakref

import torch

from . import _lib as L
from . import ops
from .derived import Derived
from .graph import get_index
from .ops import _ptr, _stream

CH_T0, CH_T1, CH_A0, CH_A1, CH_R, CH_E, CH_C, CH_D, CH_M, CH_G = 0, 1, 2, 3, 4, 5, 6, 7, 8, 9
_CTRL_BYTES = 4096                 # flags uint32[16][16] (1 KB) | counters uint32[32] | err int32 | ... | missing int32[16] at 2 KB
_OFF_COUNTERS = L.PEER_CHANNELS * L.PEER_MAX * 4
_OFF_ERR = _OFF_COUNTERS + 2 * L.PEER_CHANNELS * 4
_OFF_MISSING = 2048                # training: slot q = the number of batch pairs rank q could not find among its edges
MLP_DROPOUT_SEED = 0x5eed          # initial state of every shard's MLP dropout generator (the same on every rank)
WAIT_TIMEOUT_NS = 10_000_000_000
TRACE = os.environ.get('B200REC_PEER_TRACE', '0') == '1'


class _Raw:
    def __init__(self, ptr, nbytes):
        self.__cuda_array_interface__ = {'shape': (int(nbytes),), 'typestr': '|u1', 'data': (int(ptr), False), 'version': 3, 'strides': None}


def _align(n, a=256):
    return (int(n) + a - 1) // a * a


def _round4(n):
    return (int(n) + 3) // 4 * 4


class PeerArena:
    """`nbytes` of device memory on this rank, addressable from every rank of the group.  bases[q] = address of rank q's arena in
    THIS process (bases[rank] is the local one); `buf` is a uint8 torch view of the local arena."""

    def __init__(self, rank, world, bases, buf, owner=None):
        self.rank, self.world, self.bases, self.buf = rank, world, [int(b) for b in bases], buf
        self._owner = owner                                            # keeps the memory alive (emulation) / frees it (IPC)

    @classmethod
    def ipc(cls, nbytes, group=None, device=None):
        import torch.distributed as dist
        rank, world = dist.get_rank(group), dist.get_world_size(group)
        if world > L.PEER_MAX:
            raise NotImplementedError(f'peer exchange addresses at most {L.PEER_MAX} GPUs of one box')
        dev = torch.device('cuda', torch.cuda.current_device()) if device is None else torch.device(device)
        lib = L.lib()
        ptr = C.c_void_p()
        handle = C.create_string_buffer(L.PEER_HANDLE_BYTES)
        with torch.cuda.device(dev):
            L.check(lib.b200rec_peer_alloc(nbytes, C.byref(ptr), handle), 'peer_alloc')
        handles = [None] * world
        dist.all_gather_object(handles, bytes(handle.raw), group=group)
        bases, opened = [], []
        with torch.cuda.device(dev):
            for q in range(world):
                if q == rank:
                    bases.append(ptr.value)
                    continue
                p = C.c_void_p()
                L.check(lib.b200rec_peer_open(handles[q], C.byref(p)), 'peer_open')
                bases.append(p.value)
                opened.append(p.value)
        buf = torch.as_tensor(_Raw(ptr.value, nbytes), device=dev)

        class _Owner:
            pass
        owner = _Owner()

        def _release(local=ptr.value, opened=tuple(opened), dev=dev):
            try:
                with torch.cuda.device(dev):
                    for p in opened:
                        lib.b200rec_peer_close(C.c_void_p(p))
                    lib.b200rec_peer_free(C.c_void_p(local))
            except Exception:
                pass
        weakref.finalize(owner, _release)
        dist.barrier(group=group)                                      # nobody frees or writes before every rank has mapped everything
        return cls(rank, world, bases, buf, owner)

    @classmethod
    def emulated(cls, nbytes, world, device):
        """`world` arenas inside one process (tests): ordinary device buffers, every 'rank' sees every base address"""
        bufs = [torch.zeros(int(nbytes), dtype=torch.uint8, device=device) for _ in range(world)]
        bases = [b.data_ptr() for b in bufs]
        return [cls(q, world, bases, bufs[q], owner=bufs) for q in range(world)]

    def view(self, offset, shape, dtype=torch.float32):
        n = 1
        for s in shape:
            n *= int(s)
        nb = n * torch.empty((), dtype=dtype).element_size()
        return self.buf[offset: offset + nb].view(dtype).view(*shape)

    def ptrs(self, offset=0, first=None):
        """host array of the P addresses `base[q] + offset` (optionally rotated so that rank `first` comes first)"""
        order = list(range(self.world))
        if first is not None:
            order = [first] + [q for q in order if q != first]
        arr = (C.c_void_p * self.world)()
        for k, q in enumerate(order):
            arr[k] = self.bases[q] + offset
        return arr


class PeerShard:
    """What rank `rank` keeps of a user-partitioned graph + the arena layout (identical on every rank)."""

    def __init__(self, *, rank, world, nI, nU, d_max, rpp, users_r0, users_rows, index_users, index_items, dinv_users, dinv_items_all,
                 item_features_own, user_features_own, arena, batch_max, edges_total, edges_own, catalogue_width=0, grad_floats=0,
                 deg_users=None, deg_items_all=None, n_positions=0, symmetric=False):
        self.rank, self.world, self.nI, self.nU, self.rpp = rank, world, int(nI), int(nU), int(rpp)
        self.N = self.nI + self.nU
        self.users_r0, self.users_rows = int(users_r0), int(users_rows)
        self.it_r0 = min(rank * self.rpp, self.nI)
        self.it_rows = min(self.it_r0 + self.rpp, self.nI) - self.it_r0
        self.index_users, self.index_items = index_users, index_items
        self.dinv_users, self.dinv_items_all = dinv_users, dinv_items_all
        self.dinv_items_own = dinv_items_all[self.it_r0: self.it_r0 + self.it_rows]
        self.item_features_own, self.user_features_own = item_features_own, user_features_own
        self.arena, self.d_max, self.batch_max = arena, int(d_max), int(batch_max)
        self.edges_total, self.edges_own = int(edges_total), int(edges_own)
        self.catalogue_width = int(catalogue_width)
        self.grad_floats = int(grad_floats)
        # training (_train_forward / _train_backward): unmasked in-degrees of the owned users and of ALL items, the number of interaction positions the local
        # indexes' `pos` refer to (skip bitmap size), and whether the reverse weights w_bwd describe the same edges (binary=False graphs)
        self.deg_users, self.deg_items_all = deg_users, deg_items_all
        self.n_positions, self.symmetric = int(n_positions), bool(symmetric)
        self._mlp_generator = None
        self.off = self.layout(world, self.rpp, self.d_max, self.batch_max, self.catalogue_width, self.grad_floats)
        self.device = arena.buf.device
        self._flag_ptrs = arena.ptrs(0)
        self._counters = arena.buf[_OFF_COUNTERS:].data_ptr()
        self._err = arena.view(_OFF_ERR, (1,), torch.int32)
        self.table_rows = world * self.rpp
        self._seen = Derived(1)                                        # seen CSR of every owned user (recommend_peer, users=None)

    @staticmethod
    def layout(world, rpp, d_max, batch_max, catalogue_width=0, grad_floats=0):
        off, cur = {}, _CTRL_BYTES
        slab = _align(world * rpp * d_max * 4)
        for name in ('recv0', 'recv1', 'T0', 'T1'):
            off[name] = cur
            cur += slab
        off['rows'] = cur
        cur += _align(2 * batch_max * d_max * 4)
        # LightGAT: item score tables (P * rpp fp32) and the (m, l) softmax state of every receive slot (P * rpp, 2) fp32
        for name, nbytes in (('S0', world * rpp * 4), ('S1', world * rpp * 4), ('stats0', world * rpp * 8), ('stats1', world * rpp * 8)):
            off[name] = cur
            cur += _align(nbytes)
        if catalogue_width:                 # recommend_peer: the final item rows of ALL items, (P * rpp, catalogue_width) fp32
            off['cat'] = cur
            cur += _align(world * rpp * catalogue_width * 4)
        if grad_floats:                     # training: one slot of grad_floats fp32 (rounded up to 4) per rank, summed in rank order
            off['grad'] = cur
            cur += _align(world * _round4(grad_floats) * 4)
        off['total'] = cur
        return off

    @property
    def mlp_generator(self):
        """generator of the MLP dropout masks in training: seeded with MLP_DROPOUT_SEED on every rank and advanced by the same draws, so
        that every rank drops the same units of the (identical) batch MLP"""
        if self._mlp_generator is None:
            self._mlp_generator = torch.Generator(device=self.device)
            self._mlp_generator.manual_seed(MLP_DROPOUT_SEED)
        return self._mlp_generator

    # ---- exchange primitives ---------------------------------------------------------------------------------------------
    def signal(self, channel):
        with torch.cuda.device(self.device):
            L.check(L.lib().b200rec_peer_signal(self._flag_ptrs, self.world, self.rank, channel, C.c_void_p(self._counters), _stream()), 'peer_signal')

    def wait(self, channel):
        with torch.cuda.device(self.device):
            L.check(L.lib().b200rec_peer_wait(C.c_void_p(self.arena.bases[self.rank]), self.world, channel, C.c_void_p(self._counters),
                                              WAIT_TIMEOUT_NS, _ptr(self._err), _stream()), 'peer_wait')

    def check(self):
        """raises if a wait of this rank ever timed out (call after a synchronize)"""
        e = int(self._err.item())
        if e:
            raise L.B200RecError(f'peer exchange: rank {self.rank} timed out waiting for rank {e - 1}')

    def table(self, par, d, dtype):
        """local copy of the transformed item features of ALL items: (P * rpp, d)"""
        return self.arena.view(self.off[f'T{par}'], (self.table_rows, d), dtype)

    def scores(self, par):
        """local copy of the LightGAT source scores of ALL items: (P * rpp,) fp32"""
        return self.arena.view(self.off[f'S{par}'], (self.table_rows,))

    def push_spec(self, par, d):
        """(destination arenas, parts, rows per part, element offset of MY receive slot, leading dimension) for K3's epilogue"""
        return (self.arena.ptrs(self.off[f'recv{par}']), self.world, self.rpp, self.rank * self.rpp * d, d)

    def stats_offset(self, par):
        """element offset of MY (m, l) statistics slot from the push destinations of `push_spec(par, ...)`, which point at the receive
        sections `recv{par}` of the arenas (LightGAT pushes)"""
        return (self.off[f'stats{par}'] - self.off[f'recv{par}']) // 4 + self.rank * self.rpp * 2

    def reduce(self, par, d, *, x_next, acc_in, acc_out, acc_scale, softmax=False):
        """owned item rows from the P receive slots: a sum (LightGCN) or the softmax merge by the slots' (m, l) (LightGAT)"""
        if self.it_rows == 0:
            return
        recv = self.arena.view(self.off[f'recv{par}'], (self.world * self.rpp, d))
        ld_x = x_next.stride(0) if x_next is not None else 0
        ld_acc = acc_out.stride(0) if acc_out is not None else d
        lib = L.lib()
        with torch.cuda.device(self.device), ops._timed('peer_reduce', (self.it_rows, d, self.world)):
            if softmax:
                stats = self.arena.view(self.off[f'stats{par}'], (self.world * self.rpp, 2))
                L.check(lib.b200rec_peer_reduce_softmax(_ptr(recv), _ptr(stats), self.world, self.rpp * d, d, 2 * self.rpp, self.it_rows, d, _ptr(x_next),
                                                        ld_x, _ptr(acc_in), _ptr(acc_out), ld_acc, float(acc_scale), _stream()), 'peer_reduce_softmax')
            else:
                L.check(lib.b200rec_peer_reduce(_ptr(recv), self.world, self.rpp * d, d, self.it_rows, d, _ptr(x_next), ld_x,
                                                _ptr(acc_in), _ptr(acc_out), ld_acc, float(acc_scale), _stream()), 'peer_reduce')

    def push_scores(self, x, lin, par):
        """S[par][it_r0 : it_r0 + rows] = w·x + b (fp32) on EVERY rank: the LightGAT source scores of the owned items.
        `lin` = a (weight (1, K), bias (1,) or None) pair."""
        M = x.shape[0]
        if M == 0:
            return
        local = self.scores(par)[self.it_r0: self.it_r0 + M].view(M, 1)
        ops.linear_raw(x, lin[0], lin[1], out=local, engine='simt')
        if self.world > 1:
            others = (C.c_void_p * (self.world - 1))(*[self.arena.bases[q] + self.off[f'S{par}'] for q in range(self.world) if q != self.rank])
            with torch.cuda.device(self.device):
                L.check(L.lib().b200rec_peer_push_floats(_ptr(local), M, others, self.world - 1, self.it_r0, _stream()), 'peer_push_floats')

    def push_transform(self, x, lin, par, t_dtype, scaled=True):
        """T[par][it_r0 : it_r0 + rows] = dinv ∘ (W x + b) on EVERY rank — K1c with the all-gather in its epilogue.
        `lin` = a Linear module or a (weight, bias) pair; `scaled=False` leaves out dinv (LightGAT)."""
        M, K = x.shape
        if M == 0:
            return
        w, b = lin if isinstance(lin, tuple) else (lin.weight, lin.bias)
        N = w.shape[0]
        esz = 2 if t_dtype == torch.bfloat16 else 4
        row_scale = self.dinv_items_own if scaled else None
        dst = self.arena.ptrs(self.off[f'T{par}'], first=self.rank)
        y_off = self.it_r0 * N
        if K <= 128 and K % 32 == 0 and N <= 128 and x.stride(0) % 4 == 0 and x.data_ptr() % 16 == 0 and x.stride(1) == 1:
            wc, ldw = ops._row_major(w)
            packed = ops._packed_weight(wc, ldw, L.TC_TF32X3)
            bias = None if b is None else b.detach().contiguous().float()
            with torch.cuda.device(self.device), ops._timed('linear_shortk_push', (M, K, N, self.world)):
                L.check(L.lib().b200rec_linear_shortk_push(_ptr(x), M, K, x.stride(0), _ptr(packed), N, _ptr(bias), _ptr(row_scale), 0,
                                                          dst, self.world, y_off, N, ops._dtype_code(t_dtype), _stream()), 'linear_shortk_push')
            return
        # widths the persistent kernel does not take: plain GEMM into the local table, then a copy kernel to the peers
        local = self.table(par, N, t_dtype)[self.it_r0: self.it_r0 + M]
        ops.linear_raw(x, w, b, row_scale=row_scale, out=local)
        if self.world > 1:
            if (N * esz) % 16:
                raise NotImplementedError('the peer path needs rows of the message table that are multiples of 16 bytes')
            n32 = N * esz // 4                          # the copy kernel moves 128-bit words: a bf16 row is N/2 32-bit columns
            others = (C.c_void_p * (self.world - 1))(*[self.arena.bases[q] + self.off[f'T{par}'] for q in range(self.world) if q != self.rank])
            with torch.cuda.device(self.device):
                L.check(L.lib().b200rec_peer_push_rows(_ptr(local), n32, M, n32, others, self.world - 1, self.it_r0 * n32, n32, _stream()), 'peer_push_rows')

    def gather_rows(self, table, row0, rows, ids, dst_row, d, scale=1.0):
        dst = self.arena.ptrs(self.off['rows'])
        with torch.cuda.device(self.device):
            L.check(L.lib().b200rec_peer_gather_rows(_ptr(table) if rows else None, d, row0, rows, _ptr(ids), ids.numel(), d, float(scale), dst,
                                                    self.world, dst_row * d, d, _stream()), 'peer_gather_rows')

    # ---- device-side trace (B200REC_PEER_TRACE=1): %globaltimer markers between the kernels of a forward, readable after a graph replay
    def stamp(self, tag):
        if not TRACE:
            return
        if getattr(self, '_trace_buf', None) is None:
            self._trace_buf = torch.zeros(256, dtype=torch.int64, device=self.device)
            self._trace_tags = []
        if self._trace_reset:
            self._trace_tags, self._trace_reset = [], False
        k = len(self._trace_tags)
        if k >= 256:
            return
        self._trace_tags.append(tag)
        with torch.cuda.device(self.device):
            L.check(L.lib().b200rec_device_timestamp(C.c_void_p(self._trace_buf.data_ptr() + 8 * k), _stream()), 'device_timestamp')

    _trace_reset = True

    def trace(self):
        """[(tag, microseconds since the first marker)] of the last forward (after a synchronize)"""
        if getattr(self, '_trace_buf', None) is None:
            return []
        t = self._trace_buf[:len(self._trace_tags)].cpu().tolist()
        return [(tag, round((x - t[0]) / 1e3, 1)) for tag, x in zip(self._trace_tags, t)]

    def side_stream(self):
        if getattr(self, '_side', None) is None:
            self._side = torch.cuda.Stream(device=self.device)
        return self._side

    def rows_view(self, n, d):
        return self.arena.view(self.off['rows'], (n, d))


def _rows_per_part(nI, world):
    return max(1, (int(nI) + world - 1) // world)


def shard_from_full(graph, rank, world, arena, d_max, batch_max=8192, catalogue_width=0, grad_floats=0):
    """Shard of rank `rank` cut out of the full neighbour index (every rank builds the ~10 ms full index and keeps its slices;
    graphs that do not fit one GPU are built per rank instead: `bench.py --workload graph5`)."""
    from .parallel import RowPartition, _LocalIndex, column_slice_csr, split_rows
    full = get_index(graph)
    nI, N = int(graph.item_features.shape[0]), full.num_nodes
    rp = full.row_ptr
    k_items = int(rp[nI])
    users = RowPartition(split_rows(rp[nI:] - k_items, world), rank)
    k0, k1 = int(rp[nI + users.r0]), int(rp[nI + users.r1])
    cut = lambda a: None if a is None else a[k0:k1].contiguous()
    dinv_users = full.dinv[nI + users.r0: nI + users.r1].contiguous()
    dinv_items = full.dinv[:nI].contiguous()
    index_users = _LocalIndex((rp[nI + users.r0: nI + users.r1 + 1] - k0).contiguous(), full.col[k0:k1].contiguous(), cut(full.w), cut(full.pos),
                              dinv_users, full.chunk_size, w_bwd=cut(full.w_bwd))
    head = lambda a: None if a is None else a[:k_items]
    lrp, lcol, lw, lpos, lwb = column_slice_csr(rp[:nI + 1], full.col[:k_items], nI + users.r0, nI + users.r1, head(full.w), head(full.pos),
                                                head(full.w_bwd))
    index_items = _LocalIndex(lrp, lcol, lw, lpos, dinv_items, full.chunk_size, w_bwd=lwb)
    rpp = _rows_per_part(nI, world)
    i0 = min(rank * rpp, nI)
    return PeerShard(rank=rank, world=world, nI=nI, nU=N - nI, d_max=d_max, rpp=rpp, users_r0=users.r0, users_rows=users.rows,
                     index_users=index_users, index_items=index_items, dinv_users=dinv_users, dinv_items_all=dinv_items,
                     item_features_own=graph.item_features[i0: min(i0 + rpp, nI)], user_features_own=graph.user_features[users.r0:users.r1],
                     arena=arena, batch_max=batch_max, edges_total=full.e1 + full.e2, edges_own=int(index_users.col.numel() + lcol.numel()),
                     catalogue_width=catalogue_width, grad_floats=grad_floats, deg_users=full.deg[nI + users.r0: nI + users.r1].contiguous(),
                     deg_items_all=full.deg[:nI].contiguous(), n_positions=full.e1, symmetric=full.symmetric)


def partition_graph_peer(graph, group=None, d_max=128, batch_max=8192, catalogue_width=0, grad_floats=0):
    """One process per GPU: allocates + exchanges the arenas and cuts this rank's shard.  `d_max` = largest node_emb served;
    `catalogue_width` = floats per item row of the catalogue section that `recommend_peer` needs (`catalogue_width(model)`; 0 = none);
    `grad_floats` = floats per rank of the gradient section that training needs (`grad_floats(model)`; 0 = none)."""
    import torch.distributed as dist
    world = dist.get_world_size(group)
    nI = int(graph.item_features.shape[0])
    nbytes = PeerShard.layout(world, _rows_per_part(nI, world), d_max, batch_max, catalogue_width, grad_floats)['total']
    arena = PeerArena.ipc(nbytes, group, device=graph.item_features.device)
    return shard_from_full(graph, dist.get_rank(group), world, arena, d_max, batch_max, catalogue_width, grad_floats)


def emulated_shards(graph, world, d_max=128, batch_max=8192, catalogue_width=0, grad_floats=0):
    """all P shards in ONE process (single-GPU tests of the exchange logic; run with `forward_emulated` / `recommend_emulated` /
    `train_emulated`)"""
    nI = int(graph.item_features.shape[0])
    nbytes = PeerShard.layout(world, _rows_per_part(nI, world), d_max, batch_max, catalogue_width, grad_floats)['total']
    arenas = PeerArena.emulated(nbytes, world, graph.item_features.device)
    return [shard_from_full(graph, q, world, arenas[q], d_max, batch_max, catalogue_width, grad_floats) for q in range(world)]


# ----------------------------------------------------------------------------------------------------------------------
def _widths(model, sh: PeerShard):
    """(node_emb d, width of a combined row) after the checks every partitioned call makes"""
    if torch.is_grad_enabled() and any(p.requires_grad for p in model.parameters()):
        raise NotImplementedError('partitioned GraphNCF propagation is inference-only; wrap the call in torch.no_grad()')
    d = model.item_embeddings[0].weight.shape[0]
    if d > sh.d_max or d % 4:
        raise ValueError(f'node_emb {d} does not fit the arena of this partition (d_max {sh.d_max}) or is not a multiple of 4')
    return d, (d * (len(model.gnn_convs) + 1) if model.concat else d)             # combined embedding [x0 | ... | xL] or their mean


def _steps(model, sh: PeerShard, userIds, itemIds, keep=None):
    """Generator: GraphNCF.forward on shard `sh` (inference).  It yields right before every cross-rank wait, so that an emulation can
    advance all ranks in lock step; a real rank just runs it to the end.  Returns the (B, 1) scores."""
    from .neural_collaborative_filtering.util import run_mlp
    d, width = _widths(model, sh)
    B = int(userIds.shape[0])
    if 2 * B > 2 * sh.batch_max:
        raise ValueError(f'batch of {B} pairs exceeds the partition\'s batch_max {sh.batch_max}')
    if B * width > sh.batch_max * sh.d_max:
        raise ValueError(f'batch of {B} pairs of {width}-wide concatenated rows exceeds the partition\'s rows buffer (batch_max {sh.batch_max} '
                         f'x d_max {sh.d_max} floats per side)')
    nu, ni = sh.users_rows, sh.it_rows
    iid, uid = itemIds.long().contiguous(), userIds.long().contiguous()
    acc_items, acc_users = yield from _propagate(model, sh, d, width)
    if keep is not None:                        # tests: the owned rows of the combined embedding
        keep['items'], keep['users'] = acc_items, acc_users
    sh.gather_rows(acc_items, sh.it_r0, ni, iid, 0, width)
    sh.gather_rows(acc_users, sh.nI + sh.users_r0, nu, uid, B, width)
    sh.signal(CH_R)
    yield
    sh.wait(CH_R)
    sh.stamp('batch rows arrived')
    rows = sh.rows_view(2 * B, width)
    if model.MLP is None:
        out = ops.rowdot(rows[B:], rows[:B])
    else:
        out = run_mlp(model.MLP, rows[:B], rows[B:], training=False)               # item first (gnn_ncf.py:361)
    sh.stamp('end')
    if len(model.gnn_convs) == 0:               # no layer barrier protected `rows` against the next call's writers
        sh.signal(CH_E)
        yield
        sh.wait(CH_E)
    return out


def _propagate(model, sh: PeerShard, d, width):
    """Generator (part of `_steps` / `_recommend_steps`, same yields): the L layers on shard `sh`.  Returns the owned rows of the combined
    embedding, (items (it_rows, width), users (users_rows, width)): the running mean, or comb = [x0 | ... | xL] with concat."""
    dev = sh.device
    L_ = len(model.gnn_convs)
    concat, gat = model.concat, model.convType == 'LightGAT'
    ie, ue = model.item_embeddings[0], model.user_embeddings[0]
    nu, ni = sh.users_rows, sh.it_rows
    empty = lambda n: torch.empty((n, d), dtype=torch.float32, device=dev)
    sh._trace_reset = True
    sh.stamp('start')
    if concat:                                                                       # owned rows of comb; x_l is its column block l
        comb_items, comb_users = (torch.empty((n, width), dtype=torch.float32, device=dev) for n in (ni, nu))
        x0_items, x0_users = comb_items[:, :d], comb_users[:, :d]
        block = lambda comb, l: comb[:, d * l: d * (l + 1)]
    else:
        x0_items, x0_users = empty(ni), empty(nu)

    def embed():                                                                     # x0 = node embeddings of the owned rows (:300-301)
        if ni:
            ops.linear_raw(sh.item_features_own, ie.weight, ie.bias, out=x0_items)
        if nu:
            ops.linear_raw(sh.user_features_own, ue.weight, ue.bias, out=x0_users)

    acc_items, acc_users = x0_items, x0_users
    if L_ == 0:
        embed()
    if L_ > 0:
        conv = model.gnn_convs[0]
        lin_u, lin_i, _ = conv.typed()
        if model.message_dtype not in ('fp32', 'bf16'):
            raise ValueError("message_dtype must be 'fp32' or 'bf16'")
        t_dtype = torch.bfloat16 if (model.message_dtype == 'bf16' and d % 32 == 0 and d <= 128) else torch.float32
        t_users = torch.empty((max(nu, 1), d), dtype=t_dtype, device=dev)
        if not concat:
            acc_users, acc_items = empty(nu), empty(ni)
            spare_u = empty(nu) if L_ > 1 else None
            xi_next = empty(ni) if L_ > 1 else None
        if gat:                                                                      # LightGAT: source scores, no degree normalisation
            att_u, att_i = conv.attention()
            a_u, a_i = (att_u.weight[:, :d], None), (att_i.weight[:, :d], None)
            ps_u = torch.empty((max(nu, 1), 1), dtype=torch.float32, device=dev)
        dinv_users, dinv_items = (None, None) if gat else (sh.dinv_users, sh.dinv_items_all)
        main = torch.cuda.current_stream(dev)
        side = sh.side_stream()
        # Layer 0's messages straight from the node features: t0 = dinv ∘ (W_t (W_e f + b_e) + b_t) = dinv ∘ ((W_t W_e) f + (W_t b_e + b_t)) — composite
        # weights formed once per weight version in float64 (LightGAT: also the scores a·x0 = (a W_e) f + a b_e).  So the first SpMM waits for ONE
        # transform only; the embeddings x0 (needed from the first running-mean update on) and the broadcast of the item messages run on the side
        # stream underneath it.
        (Wci, bci), (Wcu, bcu), sc_i, sc_u = _layer0_composites(model, ie, ue, lin_i, lin_u, *((att_i, att_u) if gat else ()))
        if nu:
            ops.linear_raw(sh.user_features_own, Wcu, bcu, row_scale=dinv_users, out=t_users[:nu])
            if gat:
                ops.linear_raw(sh.user_features_own, *sc_u, out=ps_u[:nu], engine='simt')

        def layer0_side():
            sh.push_transform(sh.item_features_own, (Wci, bci), 0, t_dtype, scaled=not gat)
            if gat:
                sh.push_scores(sh.item_features_own, sc_i, 0)
            sh.signal(CH_T0)
            embed()

        start = torch.cuda.Event()
        start.record(main)
        side.wait_event(start)
        with torch.cuda.stream(side):
            layer0_side()
            x0_ready = torch.cuda.Event()
            x0_ready.record(side)

        def item_side(l, par, last, scale):                                          # C_l: needs every rank's A_l, nothing of B_l
            sh.stamp(f'C{l} begin')
            sh.wait(CH_A0 + par)
            sh.stamp(f'C{l} partials arrived')
            if concat:
                xi = block(comb_items, l + 1)
                sh.reduce(par, d, x_next=xi, acc_in=None, acc_out=None, acc_scale=1.0, softmax=gat)
            else:
                xi = None if last else xi_next
                sh.reduce(par, d, x_next=xi, acc_in=x0_items if l == 0 else acc_items, acc_out=acc_items, acc_scale=scale, softmax=gat)
            if not last:
                sh.push_transform(xi, lin_i, 1 - par, t_dtype, scaled=not gat)
                if gat:
                    sh.push_scores(xi, a_i, 1 - par)
                sh.signal(CH_T0 + (1 - par))
            sh.stamp(f'C{l} end')

        for l in range(L_):
            par, last = l & 1, l == L_ - 1
            scale = 1.0 / (L_ + 1) if last else 1.0
            sh.stamp(f'A{l} begin')
            if nu:                                                                   # A_l: partial item rows -> owners' receive slots
                ops.propagate_step(sh.index_items, t_users, dinv=dinv_items, push=sh.push_spec(par, d), att_src=ps_u if gat else None,
                                   push_stats=sh.stats_offset(par) if gat else None)
            sh.signal(CH_A0 + par)
            sh.stamp(f'A{l} end')
            forked = torch.cuda.Event()
            forked.record(main)
            yield
            side.wait_event(forked)                                                  # C_l on the side stream, under B_l
            with torch.cuda.stream(side):
                item_side(l, par, last, scale)
                joined = torch.cuda.Event()
                joined.record(side)
            sh.wait(CH_T0 + par)
            if l == 0:
                main.wait_event(x0_ready)                                            # x0_users is B_0's running-mean input
            sh.stamp(f'B{l} table arrived')
            xu = block(comb_users, l + 1) if concat else (None if last else spare_u)
            if nu:                                                                   # B_l: own user rows from the gathered table
                acc = {} if concat else dict(acc_in=x0_users if l == 0 else acc_users, acc_out=acc_users, acc_scale=scale)
                ops.propagate_step(sh.index_users, sh.table(par, d, t_dtype), dinv=dinv_users, x_next=xu, att_src=sh.scores(par) if gat else None,
                                   **acc)
            sh.stamp(f'B{l} end')
            if not last and nu:
                ops.linear_raw(xu, lin_u.weight, lin_u.bias, row_scale=dinv_users, out=t_users[:nu])
                if gat:
                    ops.linear_raw(xu, *a_u, out=ps_u[:nu], engine='simt')
        main.wait_event(joined)
        sh.stamp('layers joined')
    if concat:
        acc_items, acc_users = comb_items, comb_users
    return acc_items, acc_users


def _layer0_composites(model, ie, ue, lin_i, lin_u, att_i=None, att_u=None):
    """((W_i2u·W_item, W_i2u·b_item + b_i2u), (W_u2i·W_user, W_u2i·b_user + b_u2i), item score pair, user score pair) as cached fp32 tensors
    (float64 products, rounded once).  With the LightGAT attention Linears a score pair is (a·W_emb, a·b_emb), a = the source half of the
    attention weight (the scores a·x0 of layer 0); None otherwise."""
    d = ie.weight.shape[0]

    def comp(w_out, b_out, emb):
        w = (w_out.detach().double() @ emb.weight.detach().double()).float().contiguous()
        eb = emb.bias.detach().double() if emb.bias is not None else torch.zeros(emb.weight.shape[0], dtype=torch.float64, device=w.device)
        b = w_out.detach().double() @ eb
        if b_out is not None:
            b = b + b_out.detach().double()
        return w, b.float().contiguous()

    def build():
        out = (comp(lin_i.weight, lin_i.bias, ie), comp(lin_u.weight, lin_u.bias, ue))
        if att_i is None:
            return out + (None, None)
        return out + (comp(att_i.weight[:, :d], None, ie), comp(att_u.weight[:, :d], None, ue))

    att = (None, None) if att_i is None else (att_i.weight, att_u.weight)
    return model._peer_layer0.get((ie.weight, ie.bias, ue.weight, ue.bias, lin_i.weight, lin_i.bias, lin_u.weight, lin_u.bias) + att, build)


def forward_peer(model, sh: PeerShard, userIds, itemIds, keep=None, mask_targets=True):
    """GraphNCF.forward on a partitioned graph; every rank of the group calls it with the same batch and gets the same (B, 1) scores.

    With grad off this is the inference forward (`model.training` is not looked at).  With grad on it is the training forward: the
    scores carry a grad_fn, and `loss.backward()`, called by every rank, leaves the gradient of that loss in every parameter's `.grad`,
    bit-identical on all ranks.  `model.training` then switches on target masking (`mask_targets`) and dropout, as on one GPU.  The
    partition needs a gradient section of `grad_floats(model)` floats (ValueError otherwise)."""
    if torch.is_grad_enabled() and any(p.requires_grad for p in model.parameters()):
        return _head(model, sh, _PeerTrainFn.apply(model, sh, userIds, itemIds, mask_targets, keep, *_train_params(model).values()))
    return _run(_steps(model, sh, userIds, itemIds, keep))


def forward_emulated(model, shards, userIds, itemIds, keep=None):
    """all ranks of `emulated_shards` in lock step on one stream; returns the list of per-rank outputs"""
    keep = keep if keep is not None else [None] * len(shards)
    gens = [_steps(model, sh, userIds, itemIds, keep[q]) for q, sh in enumerate(shards)]
    outs = [None] * len(shards)
    live = list(range(len(shards)))
    while live:
        for q in list(live):
            try:
                next(gens[q])
            except StopIteration as stop:
                outs[q] = stop.value
                live.remove(q)
    return outs


# ----------------------------------------------------------------------------------------------------------------------
# whole-catalogue top-k on the partitioned graph
# ----------------------------------------------------------------------------------------------------------------------
def _dot_width(width):
    return max(64, (int(width) + 63) // 64 * 64)


def catalogue_width(model):
    """Floats per item row of the catalogue section (`catalogue_width=` of the partition builders) that `recommend_peer` needs for `model`:
    the combined width (L+1)·d with concat, else d; for a dot-product model padded to a multiple of 64, the operand width of the dot kernel."""
    d = model.item_embeddings[0].weight.shape[0]
    width = d * (len(model.gnn_convs) + 1) if model.concat else d
    return _dot_width(width) if model.MLP is None else width


def served_rows(users, nI, users_r0, users_rows):
    """(node ids int64, local rows int64) of the entries of `users` (global user NODE ids) that fall in the range [nI + users_r0,
    nI + users_r0 + users_rows) of a rank, in request order"""
    users = users.long()
    local = users - (nI + users_r0)
    mine = (local >= 0) & (local < users_rows)
    return users[mine], local[mine]


def seen_csr(row_ptr, col, rows, n_items):
    """CSR (ptr int32 (n+1), idx int32 ascending per row) of the sources of `rows` of a CSR whose sources are item ids < `n_items`: the
    `ignore_seen` sets of a shard's users (rows of `index_users`; neighbour rows are in interaction order, so they are sorted here).
    The sort key is row · n_items + item.  (GraphIndex.seen_items multiplies by `num_nodes`, which on a shard's local user index is the
    number of OWNED users: item ids can exceed it, and then the keys of neighbouring rows overlap.)"""
    rows = rows.long()
    dev = rows.device
    start, end = row_ptr[rows].long(), row_ptr[rows + 1].long()
    cnt = end - start
    ptr = torch.zeros(rows.numel() + 1, dtype=torch.int64, device=dev)
    ptr[1:] = torch.cumsum(cnt, 0)
    total = int(ptr[-1])
    r = torch.repeat_interleave(torch.arange(rows.numel(), device=dev), cnt)
    within = torch.arange(total, device=dev) - ptr[:-1][r]
    key = torch.sort(r * int(n_items) + col[start[r] + within].long()).values
    return ptr.int(), (key - r * int(n_items)).int()


def _recommend_steps(model, sh: PeerShard, k=10, users=None, precision='fp32', ignore_seen=True, return_scores=False, chunk_users=None):
    """Generator (yields like `_steps`): `recommend_peer` on shard `sh`."""
    from .neural_collaborative_filtering.util import mlp_parameters
    if model.training:
        raise NotImplementedError('recommend_peer is an inference call: model.eval() first')
    d, width = _widths(model, sh)
    if precision not in ('fp32', 'bf16'):
        raise ValueError("precision must be 'fp32' or 'bf16'")
    if not 1 <= int(k) <= 64:
        raise ValueError(f'k = {k}: the all-pairs kernels keep 1 to 64 items per user')
    dot = model.MLP is None
    if dot and width > 256:
        raise NotImplementedError(f'dot-product scoring of {width}-wide combined rows: the all-pairs dot kernel takes at most 256 floats per row')
    if not dot:                                    # the all-pairs limits, checked before any rank signals
        weights, biases, _ = mlp_parameters(model.MLP)
        if len(weights) not in (2, 3) or weights[0].shape[0] > 256 or (len(weights) == 3 and weights[1].shape[0] > 128):
            raise NotImplementedError('all-pairs scoring supports MLPs of 1 or 2 hidden layers, the first at most 256 and the second at most 128 wide')
    cw = catalogue_width(model)
    if sh.catalogue_width < cw:
        raise ValueError(f'recommend_peer needs a catalogue section of {cw} floats per item row; this partition has {sh.catalogue_width} '
                         f'(build it with catalogue_width={cw})')
    dev, nI = sh.device, sh.nI
    if users is None:
        nodes = torch.arange(nI + sh.users_r0, nI + sh.users_r0 + sh.users_rows, device=dev)
        local = None
    else:
        nodes, local = served_rows(users.to(dev), nI, sh.users_r0, sh.users_rows)
    n = int(nodes.numel())
    seen = None
    if ignore_seen:
        rp, col = sh.index_users.row_ptr, sh.index_users.col
        if local is None:
            seen = sh._seen.get((rp, col), lambda: seen_csr(rp, col, torch.arange(sh.users_rows, device=dev), nI))
        else:
            seen = seen_csr(rp, col, local, nI)
        if seen[1].numel() == 0:                   # nobody has seen anything (an empty idx array would reach the kernels as NULL)
            seen = None

    acc_items, acc_users = yield from _propagate(model, sh, d, width)

    # the final item rows of every owner -> the catalogue section of every rank (itself included), rows it_r0 ..
    cat = sh.arena.view(sh.off['cat'], (sh.table_rows, cw))
    if cw > width:                                 # the dot kernel's zero padding: only this rank writes these columns
        cat[:, width:].zero_()
    if sh.it_rows:
        with torch.cuda.device(dev):
            L.check(L.lib().b200rec_peer_push_rows(_ptr(acc_items), acc_items.stride(0), sh.it_rows, width, sh.arena.ptrs(sh.off['cat']), sh.world,
                                                   sh.it_r0 * cw, cw, _stream()), 'peer_push_rows')
    sh.signal(CH_C)
    sh.stamp('catalogue pushed')
    yield
    sh.wait(CH_C)
    sh.stamp('catalogue arrived')

    items = cat[:nI]
    val = torch.full((n, k), float('-inf'), dtype=torch.float32, device=dev)
    idx = torch.full((n, k), -1, dtype=torch.int64, device=dev)
    scores = torch.empty((n, nI), dtype=torch.float32, device=dev) if return_scores else None
    step = n if not chunk_users else int(chunk_users)
    for s in range(0, n, max(step, 1)):
        e = min(s + step, n)
        rows = acc_users[s:e] if local is None else acc_users[local[s:e]]
        sc = None if seen is None else (seen[0][s:e + 1], seen[1])     # absolute offsets into the shard's idx array
        if dot:
            v, i, sc_out = ops.allpairs_dot_topk_raw(rows if cw == width else torch.nn.functional.pad(rows, (0, cw - width)), items, k,
                                                     return_scores=return_scores, seen=sc)
        else:
            v, i, sc_out = ops.mlp_allpairs_topk(rows, items, weights, biases, k, rows_first=False, precision=precision, seen=sc,
                                                 return_scores=return_scores)
        val[s:e], idx[s:e] = v, i
        if return_scores:
            scores[s:e] = sc_out
    sh.stamp('scored')

    # closing barrier: the next call's catalogue push must not overwrite a table a slower rank still scores from
    sh.signal(CH_D)
    yield
    sh.wait(CH_D)
    return (nodes, val, idx, scores) if return_scores else (nodes, val, idx)


def recommend_peer(model, sh: PeerShard, k=10, users=None, precision='fp32', ignore_seen=True, return_scores=False, chunk_users=None):
    """Top-k items over the WHOLE catalogue for the users this rank owns — `GraphNCF.recommend` on a partitioned graph.  Every rank of the
    group calls it (with the same arguments); the propagation runs again on every call.

    users          global user NODE ids (nI .. N-1) or None = every owned user.  A rank serves the ids of its range, in request order.
    precision      'fp32' / 'bf16' as in GraphNCF.recommend (two-hidden-layer MLPs: the tensor-core operand split; the exact kernels of
                   one-hidden-layer MLPs and of dot-product models ignore it).
    ignore_seen    leave out the items a user is connected to in the graph.
    chunk_users    score at most this many users per kernel call (bounds the per-user tables and workspace on large shards).

    Returns (user_nodes int64 (n,), val (n, k) fp32, idx (n, k) int64 item node ids[, scores (n, nI)]), rows padded with (-inf, -1).  Nothing
    is gathered across ranks: the union of the ranks' `user_nodes` is the request.  The partition needs a catalogue section of
    `catalogue_width(model)` floats per item row (ValueError otherwise)."""
    gen = _recommend_steps(model, sh, k, users, precision, ignore_seen, return_scores, chunk_users)
    try:
        while True:
            next(gen)
    except StopIteration as stop:
        return stop.value


def recommend_emulated(model, shards, **kw):
    """`recommend_peer` on all ranks of `emulated_shards` in lock step on one stream; returns the list of per-rank results"""
    gens = [_recommend_steps(model, sh, **kw) for sh in shards]
    outs = [None] * len(shards)
    live = list(range(len(shards)))
    while live:
        for q in list(live):
            try:
                next(gens[q])
            except StopIteration as stop:
                outs[q] = stop.value
                live.remove(q)
    return outs


# ----------------------------------------------------------------------------------------------------------------------
# training on the partitioned graph (LightGCN, mean combine)
# ----------------------------------------------------------------------------------------------------------------------
def _train_params(model):
    """{name: parameter} of the embedding and conv parameters, in the order of the flat gradient vector.  The MLP is not among them: every
    rank runs it on the same batch rows under ordinary autograd, so its gradients are already the same on every rank."""
    return {n: p for n, p in model.named_parameters() if n.startswith(('item_embeddings.', 'user_embeddings.', 'gnn_convs.'))}


def _slot(p):
    return _round4(p.numel())                       # every parameter starts 16-byte aligned in the flat vector


def grad_floats(model):
    """Floats per rank of the gradient section (`grad_floats=` of the partition builders) that training `model` needs: the embedding and
    conv parameters, each padded to a multiple of 4"""
    return sum(_slot(p) for p in _train_params(model).values())


def _train_check(model, sh: PeerShard, B):
    """node_emb d after the checks of a training call (all made before any rank signals)"""
    if model.convType != 'LightGCN':
        raise NotImplementedError(f"partitioned training covers convType='LightGCN', not convType={model.convType!r} (train it on one GPU)")
    if model.concat:
        raise NotImplementedError('partitioned training covers the mean combine, not concat=True (train it on one GPU)')
    for name in ('node_dropout', 'message_dropout'):
        if getattr(model, name) is not None and getattr(model, name) > 0.0:
            raise NotImplementedError(f'partitioned training does not support {name} (train it on one GPU)')
    if not sh.symmetric:
        raise NotImplementedError('partitioned training needs a binary=False graph: its backward multiplies by the reverse-edge weights of the same '
                                  'index, and edge masking has the same restriction on one GPU')
    d = model.item_embeddings[0].weight.shape[0]
    if d > sh.d_max or d % 4:
        raise ValueError(f'node_emb {d} does not fit the arena of this partition (d_max {sh.d_max}) or is not a multiple of 4')
    if B > sh.batch_max:
        raise ValueError(f'batch of {B} pairs exceeds the partition\'s batch_max {sh.batch_max}')
    need = grad_floats(model)
    if sh.grad_floats < need:
        raise ValueError(f'training needs a gradient section of {need} floats per rank; this partition has {sh.grad_floats} '
                         f'(build it with grad_floats={need})')
    return d


def _mask_batch(sh: PeerShard, uid, iid):
    """(skip bitmap, masked dinv of the owned users, masked dinv of ALL items, count of pairs this rank could not find) for the batch targets.
    Identical pairs of the batch count once (GraphIndex.masked: one interaction position each).  Every rank takes the item degrees down
    from the batch alone; the owner of a pair's user finds its position in its local pair hash and masks it in both local indexes."""
    dev, B, lib = sh.device, int(uid.numel()), L.lib()
    skip = torch.zeros((sh.n_positions + 31) // 32 + 1, dtype=torch.int32, device=dev)
    deg_u, deg_i = sh.deg_users.clone(), sh.deg_items_all.clone()
    dinv_u, dinv_i = torch.empty(sh.users_rows, dtype=torch.float32, device=dev), torch.empty(sh.nI, dtype=torch.float32, device=dev)
    cap = 1 << max(4, (2 * B - 1).bit_length())
    keys, vals = torch.empty(cap, dtype=torch.int64, device=dev), torch.empty(cap, dtype=torch.int32, device=dev)
    first = torch.empty(B, dtype=torch.int64, device=dev)
    missing = torch.zeros(1, dtype=torch.int32, device=dev)
    pairs = torch.stack((uid, iid))
    hk, hv, hcap = sh.index_users.pair_hash(sh.nI + sh.users_r0)
    with torch.cuda.device(dev):
        st = _stream()
        # first[j] = the first batch entry holding the pair of entry j (a batch-local hash; every pair is found)
        L.check(lib.b200rec_pairhash_build(_ptr(pairs), B, _ptr(keys), _ptr(vals), cap, st), 'pairhash_build')
        L.check(lib.b200rec_pairhash_lookup(_ptr(uid), _ptr(iid), B, _ptr(keys), _ptr(vals), cap, _ptr(first), _ptr(missing), st), 'pairhash_lookup')
        L.check(lib.b200rec_peer_mask_targets(_ptr(uid), _ptr(iid), B, _ptr(first), sh.nI, sh.N, sh.nI + sh.users_r0, sh.users_rows, _ptr(hk), _ptr(hv),
                                              hcap, _ptr(sh.index_users.pos), _ptr(skip), _ptr(deg_u), _ptr(deg_i), _ptr(missing), st), 'peer_mask_targets')
        if sh.users_rows:
            L.check(lib.b200rec_dinv(_ptr(deg_u), sh.users_rows, _ptr(dinv_u), st), 'dinv')
        L.check(lib.b200rec_dinv(_ptr(deg_i), sh.nI, _ptr(dinv_i), st), 'dinv')
    return skip, dinv_u, dinv_i, missing


def _train_forward(model, sh: PeerShard, userIds, itemIds, mask_targets, keep=None):
    """Generator (yields like `_steps`): the training forward of GraphNCF on shard `sh` up to the batch rows.  Returns ((2B, d) batch rows,
    item rows first, the same on every rank; what the backward needs).  Layer 0 runs as two steps, x0 = W_e f + b_e and
    t0 = drop(dinv ∘ (W_t x0 + b_t)), like the single-GPU training path; each row's conv-dropout mask is drawn by its owner."""
    B = int(userIds.shape[0])
    d = _train_check(model, sh, B)
    dev, nI = sh.device, sh.nI
    uid, iid = userIds.to(dev).long().contiguous(), itemIds.to(dev).long().contiguous()
    L_ = len(model.gnn_convs)
    ie, ue = model.item_embeddings[0], model.user_embeddings[0]
    nu, ni = sh.users_rows, sh.it_rows
    empty = lambda n: torch.empty((n, d), dtype=torch.float32, device=dev)
    skip, dinv_u, dinv_i = None, sh.dinv_users, sh.dinv_items_all
    if model.training and mask_targets:
        skip, dinv_u, dinv_i, missing = _mask_batch(sh, uid, iid)
        # every rank learns every rank's count before any data moves, so that a batch with a non-edge fails on all ranks alike
        with torch.cuda.device(dev):
            L.check(L.lib().b200rec_peer_push_floats(_ptr(missing), 1, sh.arena.ptrs(0), sh.world, _OFF_MISSING // 4 + sh.rank, _stream()),
                    'peer_push_floats')
        sh.signal(CH_M)
        yield
        sh.wait(CH_M)
        if sum(sh.arena.view(_OFF_MISSING, (sh.world,), torch.int32).tolist()):
            raise KeyError('batch pairs that are not edges of the graph (pos_df.loc raises KeyError in the reference, gnn_ncf.py:370)')
    dinv_i_own = dinv_i[sh.it_r0: sh.it_r0 + ni]
    x0_i, x0_u = empty(ni), empty(nu)
    if ni:
        ops.linear_raw(sh.item_features_own, ie.weight, ie.bias, out=x0_i)
    if nu:
        ops.linear_raw(sh.user_features_own, ue.weight, ue.bias, out=x0_u)
    xs_i, xs_u, masks_i, masks_u = [], [], [], []
    acc_i, acc_u = x0_i, x0_u
    if L_ > 0:
        lin_u, lin_i, p = model.gnn_convs[0].typed()
        p = p if model.training else 0.0
        acc_i, acc_u = empty(ni), empty(nu)
        t_u = empty(max(nu, 1))

        def transform(x, lin, rs, out):              # out = drop(rs ∘ (W x + b)); returns the dropout multipliers (0 or 1/(1-p)) or None
            if x.shape[0] == 0:
                return None
            ops.linear_raw(x, lin.weight, lin.bias, row_scale=rs, out=out)
            if p <= 0.0:
                return None
            m = torch.empty_like(out).bernoulli_(1.0 - p).div_(1.0 - p)
            ops.scale_rows_raw(out, mask=m, out=out)
            return m

        def publish(x, par):                         # the owned item messages into T[par] of every rank
            local = sh.table(par, d, torch.float32)[sh.it_r0: sh.it_r0 + ni]
            m = transform(x, lin_i, dinv_i_own, local)
            _push_table_rows(sh, local, par, d)
            return m

        x_i, x_u = x0_i, x0_u
        masks_u.append(transform(x_u, lin_u, dinv_u, t_u[:nu]))
        masks_i.append(publish(x_i, 0))
        sh.signal(CH_T0)
        for l in range(L_):
            par, last = l & 1, l == L_ - 1
            scale = 1.0 / (L_ + 1) if last else 1.0
            xs_i.append(x_i)
            xs_u.append(x_u)
            if nu:                                   # A_l: partial item rows -> owners' receive slots
                ops.spmm_raw(sh.index_items, t_u, w=sh.index_items.w, dinv=dinv_i, skip_bits=skip, push=sh.push_spec(par, d))
            sh.signal(CH_A0 + par)
            yield
            sh.wait(CH_A0 + par)                     # C_l: owned item rows, then their messages for the next layer
            xi_next = None if last else empty(ni)
            sh.reduce(par, d, x_next=xi_next, acc_in=x0_i if l == 0 else acc_i, acc_out=acc_i, acc_scale=scale)
            if not last:
                masks_i.append(publish(xi_next, 1 - par))
                sh.signal(CH_T0 + (1 - par))
            sh.wait(CH_T0 + par)                     # B_l: owned user rows from the gathered table
            xu_next = None if last else empty(nu)
            if nu:
                ops.spmm_raw(sh.index_users, sh.table(par, d, torch.float32), w=sh.index_users.w, dinv=dinv_u, skip_bits=skip, x_next=xu_next,
                             acc_in=x0_u if l == 0 else acc_u, acc_out=acc_u, acc_scale=scale)
            if not last:
                masks_u.append(transform(xu_next, lin_u, dinv_u, t_u[:nu]))
            x_i, x_u = xi_next, xu_next
    sh.gather_rows(acc_i, sh.it_r0, ni, iid, 0, d)
    sh.gather_rows(acc_u, nI + sh.users_r0, nu, uid, B, d)
    sh.signal(CH_R)
    yield
    sh.wait(CH_R)
    rows = sh.rows_view(2 * B, d).clone()
    if L_ == 0:                                      # no layer barrier protects `rows` against the next call's writers
        sh.signal(CH_E)
        yield
        sh.wait(CH_E)
    if keep is not None:                             # tests: the owned combined rows and the conv-dropout multipliers of every layer
        keep.update(items=acc_i, users=acc_u, masks_items=masks_i, masks_users=masks_u)
    return rows, dict(uid=uid, iid=iid, d=d, skip=skip, dinv_u=dinv_u, dinv_i_own=dinv_i_own, xs_i=xs_i, xs_u=xs_u, masks_i=masks_i,
                      masks_u=masks_u)


def _push_table_rows(sh: PeerShard, local, par, d):
    """rows it_r0 .. of the local T[par] into T[par] of every other rank"""
    if local.shape[0] == 0 or sh.world == 1:
        return
    others = (C.c_void_p * (sh.world - 1))(*[sh.arena.bases[q] + sh.off[f'T{par}'] for q in range(sh.world) if q != sh.rank])
    with torch.cuda.device(sh.device):
        L.check(L.lib().b200rec_peer_push_rows(_ptr(local), d, local.shape[0], d, others, sh.world - 1, sh.it_r0 * d, d, _stream()), 'peer_push_rows')


def _train_backward(model, sh: PeerShard, saved, g_rows):
    """Generator (yields like `_steps`): the backward of `_train_forward` on shard `sh` for the gradient `g_rows` of its batch rows (the same
    on every rank).  Returns {name: gradient} of the embedding and conv parameters, summed over the ranks in rank order (bit-identical on
    every rank).  Per layer l = L-1 .. 0, with G_l the gradient of the owned rows x_l and par = l & 1:

        C'  s_i = dinv_i ∘ G_{l+1,i} of the owned items -> T[par] of every rank;  g_t_u = K3(index_users, w_bwd, T[par])
        A'  K3(index_items, w_bwd, dinv_u ∘ G_{l+1,u}) -> the owners' recv[par];  g_t_i = the P slots summed in rank order
        G_l = G_L + (dinv ∘ mask ∘ g_t) W;   partial dW += (dinv ∘ mask ∘ g_t)ᵀ x_l,  db += its column sums

    It starts after the forward's CH_R barrier, when every exchange section is free, and ends with the gradient exchange on CH_G."""
    d, uid, iid = saved['d'], saved['uid'], saved['iid']
    B = int(uid.numel())
    dev = sh.device
    L_ = len(model.gnn_convs)
    nu, ni = sh.users_rows, sh.it_rows
    params = _train_params(model)
    need = grad_floats(model)
    flat = torch.zeros(need, dtype=torch.float32, device=dev)
    views, o = {}, 0
    for name, p in params.items():
        views[id(p)] = flat[o: o + p.numel()].view((1, -1) if p.dim() == 1 else p.shape)
        o += _slot(p)
    ones = torch.ones((1, max(nu, ni, 1)), dtype=torch.float32, device=dev)

    def add_grad(p, g):                              # slot of p += g
        v = views[id(p)]
        ops.scale_rows_raw(g.view(v.shape), add=v, out=v)

    def transform_backward(gt, m, rs, lin, x, base):
        if gt.shape[0] == 0:
            return base
        g_lin = torch.empty_like(gt)
        ops.scale_rows_raw(gt, mask=m, row_scale=rs, out=g_lin)
        add_grad(lin.weight, ops.linear_raw(g_lin.t(), x.t()))
        if lin.bias is not None:
            add_grad(lin.bias, ops.linear_raw(ones[:, :gt.shape[0]], g_lin.t()))
        out = ops.linear_raw(g_lin, lin.weight.t())
        ops.scale_rows_raw(out, add=base, out=out)
        return out

    g = g_rows.contiguous().float()
    G_i, G_u = torch.zeros((ni, d), dtype=torch.float32, device=dev), torch.zeros((nu, d), dtype=torch.float32, device=dev)
    ops.rows_to_owned_raw(g[:B], iid, sh.it_r0, ni, 1.0 / (L_ + 1), G_i)
    ops.rows_to_owned_raw(g[B:], uid, sh.nI + sh.users_r0, nu, 1.0 / (L_ + 1), G_u)
    if L_ > 0:
        lin_u, lin_i, _ = model.gnn_convs[0].typed()
        skip, dinv_u, dinv_i_own = saved['skip'], saved['dinv_u'], saved['dinv_i_own']
        base_i, base_u = G_i, G_u                    # what every x_l receives from the mean
        s_u = torch.empty((max(nu, 1), d), dtype=torch.float32, device=dev)
        for l in reversed(range(L_)):
            par = l & 1
            local = sh.table(par, d, torch.float32)[sh.it_r0: sh.it_r0 + ni]
            if ni:
                ops.scale_rows_raw(G_i, row_scale=dinv_i_own, out=local)
            _push_table_rows(sh, local, par, d)
            sh.signal(CH_T0 + par)
            if nu:
                ops.scale_rows_raw(G_u, row_scale=dinv_u, out=s_u[:nu])
                ops.spmm_raw(sh.index_items, s_u, w=sh.index_items.w_bwd, dinv=None, skip_bits=skip, push=sh.push_spec(par, d))
            sh.signal(CH_A0 + par)
            yield
            sh.wait(CH_T0 + par)
            gt_u = torch.empty((nu, d), dtype=torch.float32, device=dev)
            if nu:
                ops.spmm_raw(sh.index_users, sh.table(par, d, torch.float32), w=sh.index_users.w_bwd, dinv=None, skip_bits=skip, x_next=gt_u)
            sh.wait(CH_A0 + par)
            gt_i = torch.empty((ni, d), dtype=torch.float32, device=dev)
            sh.reduce(par, d, x_next=gt_i, acc_in=None, acc_out=None, acc_scale=1.0)
            G_u = transform_backward(gt_u, saved['masks_u'][l], dinv_u, lin_u, saved['xs_u'][l], base_u)
            G_i = transform_backward(gt_i, saved['masks_i'][l], dinv_i_own, lin_i, saved['xs_i'][l], base_i)
    for n, G, f, emb in ((ni, G_i, sh.item_features_own, model.item_embeddings[0]), (nu, G_u, sh.user_features_own, model.user_embeddings[0])):
        if n:
            ops.linear_raw(G.t(), f.t(), out=views[id(emb.weight)])
            if emb.bias is not None:
                ops.linear_raw(ones[:, :n], G.t(), out=views[id(emb.bias)])
    # the partial gradients -> slot `rank` of every rank's gradient section; every rank sums the P slots in rank order
    stride = _round4(sh.grad_floats)
    with torch.cuda.device(dev):
        L.check(L.lib().b200rec_peer_push_rows(_ptr(flat), need, 1, need, sh.arena.ptrs(sh.off['grad']), sh.world, sh.rank * stride, need, _stream()),
                'peer_push_rows')
    sh.signal(CH_G)
    yield
    sh.wait(CH_G)
    total = torch.empty(need, dtype=torch.float32, device=dev)
    slots = sh.arena.view(sh.off['grad'], (sh.world * stride,))
    with torch.cuda.device(dev):
        L.check(L.lib().b200rec_peer_reduce(_ptr(slots), sh.world, stride, need, 1, need, _ptr(total), need, None, None, need, 1.0, _stream()),
                'peer_reduce')
    out, o = {}, 0
    for name, p in params.items():
        out[name] = total[o: o + p.numel()].view(p.shape)
        o += _slot(p)
    return out


class _RowDotFn(torch.autograd.Function):
    """(B, 1) row-wise dot products of the batch rows (the dot-product head, gnn_ncf.py:365) with a gradient"""

    @staticmethod
    def forward(ctx, a, b):
        ctx.save_for_backward(a, b)
        return ops.rowdot(a, b)

    @staticmethod
    def backward(ctx, g):
        a, b = ctx.saved_tensors
        return g * b, g * a


def _head(model, sh: PeerShard, rows):
    """scores of the (2B, d) batch rows (items first) under autograd; the MLP's dropout masks come from the shard's generator"""
    from .neural_collaborative_filtering.util import run_mlp
    B = rows.shape[0] // 2
    if model.MLP is None:
        return _RowDotFn.apply(rows[B:], rows[:B])
    return run_mlp(model.MLP, rows[:B], rows[B:], training=model.training, generator=sh.mlp_generator)


def _run(gen):
    try:
        while True:
            next(gen)
    except StopIteration as stop:
        return stop.value


class _PeerTrainFn(torch.autograd.Function):
    """(embedding and conv parameters) -> the (2B, d) batch rows of a partitioned propagation.  backward is collective: every rank runs it."""

    @staticmethod
    def forward(ctx, model, sh, userIds, itemIds, mask_targets, keep, *params):
        rows, saved = _run(_train_forward(model, sh, userIds, itemIds, mask_targets, keep))
        ctx.state = (model, sh, saved)
        return rows

    @staticmethod
    def backward(ctx, g):
        model, sh, saved = ctx.state
        ctx.state = None
        grads = _run(_train_backward(model, sh, saved, g))
        return (None,) * 6 + tuple(grads.values())


def _lockstep(gens):
    """runs the generators of all emulated ranks segment by segment; when one rank raises, the others still run to their end (or their own
    error), and the error is raised when every rank raised the same kind"""
    outs, errs = [None] * len(gens), [None] * len(gens)
    live = list(range(len(gens)))
    with torch.no_grad():
        while live:
            for q in list(live):
                try:
                    next(gens[q])
                except StopIteration as stop:
                    outs[q] = stop.value
                    live.remove(q)
                except Exception as e:              # noqa: BLE001 (re-raised below)
                    errs[q] = e
                    live.remove(q)
    failed = [e for e in errs if e is not None]
    if failed:
        if len(failed) == len(errs) and all(type(e) is type(failed[0]) for e in failed):
            raise failed[0]
        raise RuntimeError(f'emulated ranks failed differently: {errs}') from failed[0]
    return outs


def train_emulated(model, shards, userIds, itemIds, loss_fn, mask_targets=True, keep=None):
    """One training step's forward and backward on all ranks of `emulated_shards` in lock step.  `loss_fn(out)` maps a rank's (B, 1) scores
    to its scalar loss.  Returns, per rank, (scores, {parameter name: gradient}); nothing is written to `.grad`."""
    keep = keep if keep is not None else [None] * len(shards)
    fwd = _lockstep([_train_forward(model, sh, userIds, itemIds, mask_targets, keep[q]) for q, sh in enumerate(shards)])
    own = _train_params(model)
    head = {n: p for n, p in model.named_parameters() if n not in own and p.requires_grad}
    outs, g_rows, head_grads = [], [], []
    for q, sh in enumerate(shards):
        rows = fwd[q][0].requires_grad_()
        with torch.enable_grad():
            out = _head(model, sh, rows)
            gs = torch.autograd.grad(loss_fn(out), [rows] + list(head.values()), allow_unused=True)
        outs.append(out.detach())
        g_rows.append(gs[0])
        head_grads.append({n: g for n, g in zip(head, gs[1:]) if g is not None})
    bwd = _lockstep([_train_backward(model, sh, fwd[q][1], g_rows[q]) for q, sh in enumerate(shards)])
    return [(outs[q], {**bwd[q], **head_grads[q]}) for q in range(len(shards))]
