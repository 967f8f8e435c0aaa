"""Tensor-level wrappers over the C ABI (include/b200rec.h) + autograd glue.

PyTorch is plumbing here: device memory, streams and autograd bookkeeping.  Every forward op launches
hand-written sm_100a kernels from libb200rec.so on the caller's current CUDA stream.  There is no CPU
path: tensors must live on a CUDA device.

Backward passes (training is row (f)-1 "next" in SURVEY.md §8): the SpMM backward runs the same CUDA
kernel on the transposed weights; Linear / MLP-tower / attention-pool backward recompute with torch
CUDA ops for now (documented in DESIGN.md §7).
"""
from __future__ import annotations

import ctypes as C
import os

import torch

from . import _lib as L
from .derived import Derived


class OpTimer:
    """Optional per-op CUDA-event timing on the launching stream (bench.py's roofline leg).  Off by default."""

    def __init__(self):
        self.records = []          # (name, meta, start_event, end_event)

    def summary(self):
        """{(name, meta): [ms, ...]} — call after a synchronize."""
        out = {}
        for name, meta, a, b in self.records:
            out.setdefault((name, meta), []).append(a.elapsed_time(b))
        return out


_timer = None


def set_timer(timer):
    """Install (or remove with None) an OpTimer; returns the previous one."""
    global _timer
    prev, _timer = _timer, timer
    return prev


class _timed:
    def __init__(self, name, meta=()):
        self.name, self.meta = name, meta

    def __enter__(self):
        if _timer is not None:
            self.a = torch.cuda.Event(enable_timing=True)
            self.a.record()
        return self

    def __exit__(self, *exc):
        if _timer is not None:
            b = torch.cuda.Event(enable_timing=True)
            b.record()
            _timer.records.append((self.name, self.meta, self.a, b))
        return False


def launch_count() -> int:
    """Kernels launched by libb200rec in this process so far."""
    return int(L.lib().b200rec_launch_count())


def _require_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError('deeprecommendation_b200 runs on CUDA (sm_100a) only; got a CPU tensor and there is no CPU fallback')


def _ptr(t):
    return None if t is None else C.c_void_p(t.data_ptr())


_raw_stream = getattr(torch._C, '_cuda_getCurrentRawStream', None)
_raw_device = getattr(torch._C, '_cuda_getDevice', None)


def _stream():
    """the current stream of the current device as a `cudaStream_t` (the raw getters are ~20x cheaper than building a torch Stream object:
    an eager forward makes a dozen of these calls — tools/host_profile.py)"""
    if _raw_stream is not None and _raw_device is not None:
        return C.c_void_p(_raw_stream(_raw_device()))
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


class _on:
    """`torch.cuda.device(dev)` that costs nothing when `dev` already is the current device (one process per GPU: always)."""
    __slots__ = ('idx', 'prev')

    def __init__(self, dev):
        self.idx = dev.index if isinstance(dev, torch.device) else torch.device(dev).index
        self.prev = -1

    def __enter__(self):
        if self.idx is not None:
            cur = _raw_device() if _raw_device is not None else torch.cuda.current_device()
            if cur != self.idx:
                self.prev = cur
                torch.cuda.set_device(self.idx)
        return self

    def __exit__(self, *exc):
        if self.prev >= 0:
            torch.cuda.set_device(self.prev)
            self.prev = -1
        return False


def _row_major(t: torch.Tensor):
    """Returns (tensor, leading dimension) for a 2-D fp32 tensor usable without a copy when rows are contiguous."""
    if t.dim() != 2:
        raise ValueError('expected a 2-D tensor')
    if t.dtype != torch.float32:
        t = t.float()
    if t.stride(1) != 1 or (t.size(0) > 1 and t.stride(0) < t.size(1)):
        t = t.contiguous()
    ld = t.stride(0) if t.size(0) > 1 else max(t.size(1), t.stride(0))
    return t, ld


def _dtype_code(dt):
    if dt == torch.float32:
        return L.F32
    if dt == torch.bfloat16:
        return L.BF16
    raise ValueError(f'unsupported dtype {dt}')


# ------------------------------------------------------------------------------------------------------------------
# K1a linear
# ------------------------------------------------------------------------------------------------------------------
# GEMM engine for K1a: 'simt' = fp32 FFMA everywhere; 'tf32x3' / 'bf16' = tcgen05 tensor-core kernel (csrc/gemm_tc.cu) for
# large M, FFMA for the small ones (a 128-row tile per CTA cannot fill 148 SMs below ~2k rows).
# fp32-parity tensor-core engines: 'tf32x3' (3xTF32 everywhere) and 'bf16x3' (default: the same, except that the wide form — large M, 128 < N, long K —
# runs the three products on a bf16 hi/lo split at twice the MMA rate: ~4e-6 instead of ~6e-7 of the largest output, budget 1e-5; the whole GPU suite
# passes under either)
_gemm_engine = os.environ.get('B200REC_GEMM_ENGINE', 'bf16x3')
TC_MIN_ROWS = 2048
TC_SPLITK_MIN_ROWS = 128      # below TC_MIN_ROWS the tensor-core GEMM runs split-K (if K is long enough to be dealt out)
SHORTK_MIN_ROWS = 4096  # below this a handful of 64x64 FFMA tiles is as fast as the persistent kernel's set-up
TC_MIN_K = 512          # short-K GEMMs (the d x d GraphNCF transforms) are epilogue/latency-bound: FFMA is as fast there


_pack_cache = Derived(64)     # MMA-ready packed weights: a handful of weight matrices at most
_wt_cache = Derived(64)       # transposed K1s tables
_ap_cache = Derived(32)       # all-pairs second-layer packs


def _packed_weight(w, ldw, mode):
    """MMA-ready copy of a weight matrix (b200rec_pack_weights_tc), cached until the tensor changes (`_version`)."""
    def pack():
        lib = L.lib()
        N, K = w.shape
        nbytes = lib.b200rec_packed_weight_bytes(N, K, mode)
        buf = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
        with _on(w.device):
            L.check(lib.b200rec_pack_weights_tc(_ptr(w), N, K, ldw, mode, _ptr(buf), nbytes, _stream()), 'pack_weights_tc')
        return buf
    return _pack_cache.get((w,), pack, ldw, mode)


def invalidate_caches():
    """Drops every derived copy of a weight kept by this module (MMA-ready packed weights, transposed tables, all-pairs packs).  An entry
    is reused only while its source is the same live tensor at the same address with the same `_version` (`derived.Derived`): an in-place
    edit THROUGH `.data` (`p.data.copy_()`, some EMA / weight-averaging utilities) does not bump `_version`, so such code must call this
    (the model classes do it from `load_state_dict` / `_apply` / `invalidate_caches()`)."""
    _pack_cache.clear()
    _wt_cache.clear()
    _ap_cache.clear()


def _tc_mode(engine):
    """MMA mode of an engine name: 'bf16' -> bf16 operands; 'tf32x3' and 'bf16x3' -> 3xTF32 (bf16x3 only differs in the wide form)"""
    return L.TC_BF16 if engine.startswith('bf16') and not engine.startswith('bf16x3') else L.TC_TF32X3


def set_gemm_engine(name: str):
    global _gemm_engine
    if name not in ('simt', 'tf32x3', 'bf16', 'bf16x3'):
        raise ValueError(name)
    prev, _gemm_engine = _gemm_engine, name
    return prev


def linear_raw(x, weight, bias=None, row_scale=None, relu=False, out=None, out_dtype=torch.float32, engine=None, row_index=None):
    """out = act((x @ weight.T + bias) * row_scale[:, None]) — b200rec_linear / b200rec_linear_tc.
    `row_index` (int64, M): use rows x[row_index] without materialising them (tensor-core engine; gathered first otherwise)."""
    _require_cuda(x, weight, bias, row_scale, out, row_index)
    x, ldx = _row_major(x)
    w, ldw = _row_major(weight)
    x_rows = x.shape[0]
    if row_index is not None:
        row_index = row_index.contiguous().long()
        eng = engine or _gemm_engine
        if eng == 'simt' or not ((row_index.numel() >= TC_MIN_ROWS and x.shape[1] >= TC_MIN_K) or eng.endswith('!')) or x_rows * ldx >= 2 ** 32:
            x, row_index = x.index_select(0, row_index), None
            x, ldx = _row_major(x)
    M, K = (x.shape if row_index is None else (row_index.numel(), x.shape[1]))
    N = w.shape[0]
    if w.shape[1] != K:
        raise ValueError(f'linear: weight is {tuple(w.shape)}, input is {tuple(x.shape)}')
    if bias is not None and (bias.dtype != torch.float32 or not bias.is_contiguous()):
        bias = bias.contiguous().float()
    if row_scale is not None and (row_scale.dtype != torch.float32 or not row_scale.is_contiguous()):
        row_scale = row_scale.contiguous().float()
    if out is None:
        out = torch.empty((M, N), dtype=out_dtype, device=x.device)
    elif out.shape != (M, N) or out.stride(1) != 1:
        raise ValueError('linear: bad `out`')
    ldy = out.stride(0) if M > 1 else max(N, out.stride(0))
    if M == 0:
        return out                                   # empty batch: nothing to launch (nn.Linear returns an empty (0, N) too)
    lib = L.lib()
    engine = engine or _gemm_engine
    if (engine in ('tf32x3', 'bf16x3', 'shortk!') and row_index is None and K <= 128 and K % 32 == 0 and N <= 128 and (M >= SHORTK_MIN_ROWS or engine == 'shortk!')
            and ldx % 4 == 0 and x.data_ptr() % 16 == 0 and out.dtype in (torch.float32, torch.bfloat16)):
        # per-node d x d transforms (GraphNCF): persistent streaming kernel, W resident in shared memory
        packed = _packed_weight(w, ldw, L.TC_TF32X3)
        with _on(x.device), _timed('linear_shortk', (M, K, N)):
            L.check(lib.b200rec_linear_shortk(_ptr(x), M, K, ldx, _ptr(packed), N, _ptr(bias), _ptr(row_scale), int(relu), _ptr(out), ldy,
                                              _dtype_code(out.dtype), _stream()), 'linear_shortk')
        return out
    if engine == 'shortk!':
        raise ValueError('linear: shape not supported by the short-K kernel')
    if engine != 'simt' and ((M >= TC_MIN_ROWS and K >= TC_MIN_K) or engine.endswith('!')) and (x_rows if row_index is not None else M) * ldx < 2 ** 32:
        mode = _tc_mode(engine)
        if mode == L.TC_TF32X3 and N > 128 and ((N + 127) // 128) % 2 == 0 and K >= 256:
            # 128 x 256 tiles: every X block converted and staged once for both halves of W, k range split over the CTAs
            if engine.startswith('bf16x3'):              # the same three products on a bf16 hi/lo split (2x MMA rate, ~4e-6)
                mode = L.TC_BF16X3
            packed = _packed_weight(w, ldw, mode)
            wsb = lib.b200rec_linear_tc_wide_workspace(M, N, K, mode)
            ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device=x.device)
            with _on(x.device), _timed('linear_tc', (M, K, N)):
                L.check(lib.b200rec_linear_tc_wide(_ptr(x), M, K, ldx, N, _ptr(bias), _ptr(row_scale), int(relu), _ptr(out), ldy, _dtype_code(out.dtype),
                                                   mode, _ptr(packed), _ptr(row_index), x_rows, _ptr(ws), wsb, _stream()), 'linear_tc_wide')
            return out
        packed = _packed_weight(w, ldw, mode)
        with _on(x.device), _timed('linear_tc', (M, K, N)):
            L.check(lib.b200rec_linear_tc(_ptr(x), M, K, ldx, _ptr(w), N, ldw, _ptr(bias), _ptr(row_scale), int(relu), _ptr(out), ldy,
                                          _dtype_code(out.dtype), mode, _ptr(packed), _ptr(row_index), x_rows, _stream()), 'linear_tc')
        return out
    if engine != 'simt' and row_index is None and TC_SPLITK_MIN_ROWS <= M < TC_MIN_ROWS and K >= TC_MIN_K and M * ldx < 2 ** 32:
        # short-M, long-K (a batch of pairs against the F-wide profiles): split-K on the tensor cores
        mode = _tc_mode(engine)
        ws_bytes = lib.b200rec_linear_tc_splitk_workspace(M, N, K, mode)
        if ws_bytes:
            packed = _packed_weight(w, ldw, mode)
            ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device)
            with _on(x.device), _timed('linear_tc_splitk', (M, K, N)):
                L.check(lib.b200rec_linear_tc_splitk(_ptr(x), M, K, ldx, _ptr(w), N, ldw, _ptr(bias), _ptr(row_scale), int(relu), _ptr(out), ldy,
                                                     _dtype_code(out.dtype), mode, _ptr(packed), _ptr(ws), ws_bytes, _stream()), 'linear_tc_splitk')
            return out
    ws_bytes = lib.b200rec_linear_workspace(M, N, K)
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=x.device) if ws_bytes else None
    with _on(x.device), _timed('linear', (M, K, N)):
        L.check(lib.b200rec_linear(_ptr(x), M, K, ldx, _ptr(w), N, ldw, _ptr(bias), _ptr(row_scale), int(relu), _ptr(out), ldy,
                                   _dtype_code(out.dtype), _ptr(ws), ws_bytes, _stream()), 'linear')
    return out


def tc_batch_available(engine=None):
    return (engine or _gemm_engine) != 'simt'


def linear_tc_batch(problems, engine=None):
    """Up to four `out = x @ weight.T + bias` GEMMs of the same K in ONE tensor-core launch (b200rec_linear_tc_batch).
    problems: list of (x, weight, bias | None, out | None); returns the outputs.  Inference only."""
    engine = engine or _gemm_engine
    if engine == 'simt':
        raise RuntimeError('linear_tc_batch needs a tensor-core engine (set_gemm_engine)')
    mode = _tc_mode(engine)
    arr = (L.LinearProblem * len(problems))()
    keep, outs, K, dev, meta = [], [], None, None, []
    for q, (x, weight, bias, out) in enumerate(problems):
        _require_cuda(x, weight, bias, out)
        x, ldx = _row_major(x)
        w, ldw = _row_major(weight)
        M, Kq = x.shape
        N = w.shape[0]
        if w.shape[1] != Kq or (K is not None and Kq != K):
            raise ValueError('linear_tc_batch: the problems must share K')
        K, dev = Kq, x.device
        if M * ldx >= 2 ** 32:
            raise NotImplementedError('linear_tc_batch: operand larger than 2^32 elements')
        if bias is not None and (bias.dtype != torch.float32 or not bias.is_contiguous()):
            bias = bias.contiguous().float()
        if out is None:
            out = torch.empty((M, N), dtype=torch.float32, device=dev)
        elif out.shape != (M, N) or out.stride(1) != 1:
            raise ValueError('linear_tc_batch: bad `out`')
        packed = _packed_weight(weight if weight is w else w, ldw, mode)
        p = arr[q]
        p.X, p.M, p.ldx = x.data_ptr(), M, ldx
        p.W, p.N, p.ldw = w.data_ptr(), N, ldw
        p.packed_w = packed.data_ptr()
        p.bias = bias.data_ptr() if bias is not None else None
        p.row_scale, p.relu = None, 0
        p.Y, p.ldy, p.y_dtype = out.data_ptr(), (out.stride(0) if M > 1 else max(N, out.stride(0))), _dtype_code(out.dtype)
        keep += [x, w, bias, packed, out]
        outs.append(out)
        meta.append((M, N))
    with _on(dev), _timed('linear_tc_batch', (sum(m for m, _ in meta), K, max(n for _, n in meta))):
        L.check(L.lib().b200rec_linear_tc_batch(arr, len(problems), K, mode, _stream()), 'linear_tc_batch')
    return outs


def linear_pair(xa, wa, ba, xb, wb, bb):
    """(xa @ wa.T + ba, xb @ wb.T + bb) — the two projections of one NCF batch (basic_ncf.py:38-39).  When both are short-M / long-K
    problems of the same K on a tensor-core engine they share ONE split-K launch (b200rec_linear_tc_splitk_batch); otherwise two
    `linear_raw` calls.  Inference only."""
    engine = _gemm_engine
    Ma, Mb, K = xa.shape[0], xb.shape[0], xa.shape[1]
    ok = (engine != 'simt' and xb.shape[1] == K and K >= TC_MIN_K and TC_SPLITK_MIN_ROWS <= Ma < TC_MIN_ROWS and
          TC_SPLITK_MIN_ROWS <= Mb < TC_MIN_ROWS)
    if not ok:
        return linear_raw(xa, wa, ba), linear_raw(xb, wb, bb)
    _require_cuda(xa, wa, ba, xb, wb, bb)
    mode = _tc_mode(engine)
    arr = (L.LinearProblem * 2)()
    keep, outs = [], []
    for q, (x, weight, bias) in enumerate(((xa, wa, ba), (xb, wb, bb))):
        x, ldx = _row_major(x)
        w, ldw = _row_major(weight)
        M, N = x.shape[0], w.shape[0]
        if w.shape[1] != K:
            raise ValueError(f'linear_pair: weight is {tuple(w.shape)}, input is {tuple(x.shape)}')
        if M * ldx >= 2 ** 32:
            return linear_raw(xa, wa, ba), linear_raw(xb, wb, bb)
        if bias is not None and (bias.dtype != torch.float32 or not bias.is_contiguous()):
            bias = bias.contiguous().float()
        out = torch.empty((M, N), dtype=torch.float32, device=x.device)
        packed = _packed_weight(weight if weight is w else w, ldw, mode)
        pr = arr[q]
        pr.X, pr.M, pr.ldx = x.data_ptr(), M, ldx
        pr.W, pr.N, pr.ldw = w.data_ptr(), N, ldw
        pr.packed_w = packed.data_ptr()
        pr.bias = bias.data_ptr() if bias is not None else None
        pr.row_scale, pr.relu = None, 0
        pr.Y, pr.ldy, pr.y_dtype = out.data_ptr(), N, L.F32
        keep += [x, w, bias, packed]
        outs.append(out)
    lib = L.lib()
    ws_bytes = lib.b200rec_linear_tc_splitk_batch_workspace(arr, 2, K, mode)
    ws = torch.empty(max(ws_bytes, 16), dtype=torch.uint8, device=outs[0].device)
    with _on(outs[0].device), _timed('linear_tc_splitk_batch', (Ma + Mb, K, max(wa.shape[0], wb.shape[0]))):
        L.check(lib.b200rec_linear_tc_splitk_batch(arr, 2, K, mode, _ptr(ws), ws_bytes, _stream()), 'linear_tc_splitk_batch')
    return outs[0], outs[1]


# ------------------------------------------------------------------------------------------------------------------
# K1s sparse projection (one-hot / multi-hot profile rows)
# ------------------------------------------------------------------------------------------------------------------
def _transposed_weight(weight, c0, c1, dtype=torch.float32):
    """W[:, c0:c1]^T as a contiguous (c1 - c0, N) table (the "embedding table" K1s gathers from), cached per weight version."""
    return _wt_cache.get((weight,), lambda: weight.detach()[:, c0:c1].t().to(dtype).contiguous(), c0, c1, dtype)


def linear_sparse_raw(weight, bias, *, csr=None, ids=None, cols=None, out=None, accumulate=False, table_dtype=torch.float32):
    """out (+)= bias + sum_k val[k] * weight[:, c0 + col[k]]  — b200rec_linear_sparse.  `csr` = (row_ptr int32 (M+1), col int32, val fp32 | None)
    or `ids` (M int64: one-hot rows); `cols` = (c0, c1): the weight columns the indices refer to (default: all)."""
    _require_cuda(weight, bias, out)
    c0, c1 = (0, weight.shape[1]) if cols is None else cols
    N = weight.shape[0]
    if N % 4:
        raise NotImplementedError('linear_sparse: output width must be a multiple of 4')
    wt = _transposed_weight(weight, c0, c1, table_dtype)
    if csr is not None:
        rp, col, val = csr
        rp, col = rp.contiguous().int(), col.contiguous().int()
        val = None if val is None else val.contiguous().float()
        M = rp.numel() - 1
        _require_cuda(rp, col, val)
    else:
        ids = ids.contiguous().long()
        _require_cuda(ids)
        rp = col = val = None
        M = ids.numel()
    if out is None:
        if accumulate:
            raise ValueError('linear_sparse: accumulate needs `out`')
        out = torch.empty((M, N), dtype=torch.float32, device=weight.device)
    elif out.shape != (M, N) or out.stride(1) != 1 or out.dtype != torch.float32:
        raise ValueError('linear_sparse: bad `out`')
    if bias is not None and (bias.dtype != torch.float32 or not bias.is_contiguous()):
        bias = bias.detach().contiguous().float()
    ldy = out.stride(0) if M > 1 else max(N, out.stride(0))
    nnz = int(col.numel()) if col is not None else M
    with _on(weight.device), _timed('linear_sparse', (M, nnz, c1 - c0, N)):
        L.check(L.lib().b200rec_linear_sparse(_ptr(rp), _ptr(col), _ptr(val), _ptr(ids), M, _ptr(wt), c1 - c0, N, N, _dtype_code(table_dtype),
                                              None if accumulate else _ptr(bias), _ptr(out), ldy, int(accumulate), _stream()), 'linear_sparse')
    return out


def dense_to_csr(x, c0, c1):
    """(row_ptr int32, col int32, val fp32) of the non-zero entries of x[:, c0:c1] (b200rec_dense_nnz_count / _fill + the library scan)"""
    _require_cuda(x)
    x, ldx = _row_major(x)
    M = x.shape[0]
    lib = L.lib()
    cnt = torch.empty(M, dtype=torch.int32, device=x.device)
    rp = torch.empty(M + 1, dtype=torch.int32, device=x.device)
    ws = torch.empty(max(int(lib.b200rec_scan_workspace(M)), 16), dtype=torch.uint8, device=x.device)
    with _on(x.device):
        L.check(lib.b200rec_dense_nnz_count(_ptr(x), M, ldx, c0, c1, _ptr(cnt), _stream()), 'dense_nnz_count')
        L.check(lib.b200rec_exclusive_scan_i32(_ptr(cnt), M, _ptr(rp), _ptr(ws), ws.numel(), _stream()), 'scan')
        nnz = int(rp[-1].item())
        col = torch.empty(max(nnz, 1), dtype=torch.int32, device=x.device)
        val = torch.empty(max(nnz, 1), dtype=torch.float32, device=x.device)
        L.check(lib.b200rec_dense_nnz_fill(_ptr(x), M, ldx, c0, c1, _ptr(rp), _ptr(col), _ptr(val), _stream()), 'dense_nnz_fill')
    return rp, col[:nnz], val[:nnz]


class _SparseLinearFn(torch.autograd.Function):
    """forward: K1s.  backward: dW^T[col] += val * g[row] (torch index_add_, hardware order like the reference's GEMM-free scatter)."""

    @staticmethod
    def forward(ctx, weight, bias, rp, col, val, ids, c0, c1):
        ctx.save_for_backward(weight, rp, col, val, ids)
        ctx.cols, ctx.has_bias = (c0, c1), bias is not None
        return linear_sparse_raw(weight, bias, csr=None if rp is None else (rp, col, val), ids=ids, cols=(c0, c1))

    @staticmethod
    def backward(ctx, g):
        weight, rp, col, val, ids = ctx.saved_tensors
        c0, c1 = ctx.cols
        g = g.contiguous().float()
        gwt = torch.zeros((c1 - c0, weight.shape[0]), dtype=torch.float32, device=g.device)
        if ids is not None:
            ok = ids >= 0
            gwt.index_add_(0, ids[ok], g[ok])
        else:
            rows = torch.repeat_interleave(torch.arange(g.shape[0], device=g.device), (rp[1:] - rp[:-1]).long())
            contrib = g[rows] if val is None else g[rows] * val[:, None]
            gwt.index_add_(0, col.long(), contrib)
        gw = torch.zeros_like(weight, dtype=torch.float32)
        gw[:, c0:c1] = gwt.t()
        return gw, (g.sum(0) if ctx.has_bias else None), None, None, None, None, None, None


def linear_rows(x, weight, bias=None, out=None):
    """`nn.Linear` over profile rows in whichever form the provider delivers them (content_providers.py): a dense tensor (K1a), `OneHotRows`
    (K1s: one table row per output row) or `MixedRows` (K1a over the dense columns, then K1s accumulates the non-zeros of the sparse ones)."""
    if torch.is_tensor(x):
        if out is not None:
            return linear_raw(x, weight, bias, out=out)
        return linear(x, weight, bias)
    needs = torch.is_grad_enabled() and (weight.requires_grad or (bias is not None and bias.requires_grad))
    kind = getattr(x, 'kind', None)
    if kind == 'onehot':
        if x.num_classes != weight.shape[1]:
            raise ValueError(f'one-hot rows over {x.num_classes} classes against a weight with {weight.shape[1]} inputs')
        if needs:
            y = _SparseLinearFn.apply(weight, bias, None, None, None, x.ids, 0, weight.shape[1])
            return y if out is None else out.copy_(y)
        return linear_sparse_raw(weight, bias, ids=x.ids, out=out)
    if kind == 'mixed':
        ns, K = x.n_sparse, weight.shape[1]
        if x.width != K:
            raise ValueError(f'mixed rows of width {x.width} against a weight with {K} inputs')
        if needs:
            y = _SparseLinearFn.apply(weight, bias if x.dense is None else None, x.row_ptr, x.col, x.val, None, 0, ns)
            if x.dense is not None:
                y = y + linear(x.dense, weight[:, ns:], bias)
            return y if out is None else out.copy_(y)
        if x.dense is None:
            return linear_sparse_raw(weight, bias, csr=(x.row_ptr, x.col, x.val), cols=(0, ns), out=out)
        y = linear_raw(x.dense, weight[:, ns:], bias, out=out)
        return linear_sparse_raw(weight, None, csr=(x.row_ptr, x.col, x.val), cols=(0, ns), out=y, accumulate=True)
    raise TypeError(f'cannot project {type(x).__name__}')


class _LinearFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, row_scale, relu):
        y = linear_raw(x, weight, bias, row_scale, relu)
        ctx.save_for_backward(x, weight, row_scale, y if relu else None)
        ctx.has_bias = bias is not None
        return y

    @staticmethod
    def backward(ctx, g):
        x, w, rs, y = ctx.saved_tensors
        g = g.contiguous()
        if y is not None:
            g = g * (y > 0)
        if rs is not None:
            g = g * rs[:, None]
        # both gradient GEMMs on the library's own kernels (K1a): gx = g·W, gW = gᵀ·x
        gx = linear_raw(g, w.t()) if ctx.needs_input_grad[0] else None
        gw = linear_raw(g.t(), x.t()) if ctx.needs_input_grad[1] else None
        gb = g.sum(0) if (ctx.has_bias and ctx.needs_input_grad[2]) else None
        return gx, gw, gb, None, None


def linear(x, weight, bias=None, row_scale=None, relu=False):
    if torch.is_grad_enabled() and (x.requires_grad or weight.requires_grad or (bias is not None and bias.requires_grad)):
        return _LinearFn.apply(x, weight, bias, row_scale, relu)
    return linear_raw(x, weight, bias, row_scale, relu)


# ------------------------------------------------------------------------------------------------------------------
# K1b MLP tower
# ------------------------------------------------------------------------------------------------------------------
def mlp_tower_raw(in0, in1, weights, biases, idx0=None, idx1=None):
    _require_cuda(in0, in1, idx0, idx1, *weights)
    n = len(weights)
    if n < 1 or n > L.MLP_MAX_LAYERS:
        raise NotImplementedError(f'MLP tower supports 1..{L.MLP_MAX_LAYERS} Linear layers, got {n}')
    in0, ld0 = _row_major(in0)
    E0 = in0.shape[1]
    if in1 is not None:
        in1, ld1 = _row_major(in1)
        E1 = in1.shape[1]
    else:
        ld1, E1 = 0, 0
    B = idx0.shape[0] if idx0 is not None else in0.shape[0]
    keep = []
    d = L.MlpDesc()
    d.n_layers = n
    prev = E0 + E1
    for l, (w, b) in enumerate(zip(weights, biases)):
        if w.dtype != torch.float32 or not w.is_contiguous():
            w = w.detach().contiguous().float()
        if w.shape[1] != prev:
            raise ValueError(f'MLP layer {l}: weight {tuple(w.shape)} does not take {prev} inputs')
        keep.append(w)
        d.W[l] = w.data_ptr()
        if b is not None:
            if b.dtype != torch.float32 or not b.is_contiguous():
                b = b.detach().contiguous().float()
            keep.append(b)
            d.b[l] = b.data_ptr()
        else:
            d.b[l] = None
        d.out_dim[l] = w.shape[0]
        prev = w.shape[0]
    if idx0 is not None:
        idx0 = idx0.contiguous().long()
    if idx1 is not None:
        idx1 = idx1.contiguous().long()
    out = torch.empty((B, prev), dtype=torch.float32, device=in0.device)
    if B == 0:
        return out
    with _on(in0.device), _timed('mlp_tower', (B, E0 + E1)):
        L.check(L.lib().b200rec_mlp_tower(_ptr(in0), ld0, _ptr(idx0), E0, _ptr(in1), ld1, _ptr(idx1), E1, B, C.byref(d), _ptr(out),
                                         prev, _stream()), 'mlp_tower')
    return out


class _MlpTowerFn(torch.autograd.Function):
    """forward: fused CUDA tower (K1b).  backward: the layer activations are recomputed with K1a (bias + ReLU fused) and
    every gradient GEMM (g·W, gᵀ·h) runs on K1a too; only masks, bias sums and the row scatter are torch elementwise ops."""

    @staticmethod
    def forward(ctx, in0, in1, idx0, idx1, n_layers, *params):
        weights, biases = params[:n_layers], params[n_layers:]
        ctx.n_layers = n_layers
        ctx.save_for_backward(in0, in1, idx0, idx1, *params)
        return mlp_tower_raw(in0, in1, weights, biases, idx0, idx1)

    @staticmethod
    def backward(ctx, g):
        in0, in1, idx0, idx1, *params = ctx.saved_tensors
        n = ctx.n_layers
        weights, biases = params[:n], params[n:]
        xa = in0[idx0] if idx0 is not None else in0
        if in1 is not None:
            x = torch.cat((xa, in1[idx1] if idx1 is not None else in1), dim=1)
        else:
            x = xa
        acts = [x.float().contiguous()]
        for l in range(n - 1):                                         # the last layer's output is not needed
            acts.append(linear_raw(acts[-1], weights[l], biases[l], relu=True))
        g = g.contiguous().float()
        gws, gbs = [None] * n, [None] * n
        for l in range(n - 1, -1, -1):
            if l < n - 1:
                g = g * (acts[l + 1] > 0)
            gws[l] = linear_raw(g.t(), acts[l].t())
            if biases[l] is not None:
                gbs[l] = g.sum(0)
            g = linear_raw(g, weights[l].t())
        E0 = in0.shape[1]
        ga_rows, gb_rows = g[:, :E0], (g[:, E0:] if in1 is not None else None)
        ga = torch.zeros_like(in0, dtype=torch.float32).index_add_(0, idx0, ga_rows) if idx0 is not None else ga_rows
        gb = None
        if in1 is not None:
            gb = torch.zeros_like(in1, dtype=torch.float32).index_add_(0, idx1, gb_rows) if idx1 is not None else gb_rows
        return (ga, gb, None, None, None, *gws, *gbs)


def mlp_tower(in0, in1, weights, biases, idx0=None, idx1=None):
    params = list(weights) + list(biases)
    needs = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in [in0, in1] + params)
    if needs:
        return _MlpTowerFn.apply(in0, in1, idx0, idx1, len(weights), *params)
    return mlp_tower_raw(in0, in1, weights, biases, idx0, idx1)


def rowdot(in0, in1, idx0=None, idx1=None):
    _require_cuda(in0, in1)
    in0, ld0 = _row_major(in0)
    in1, ld1 = _row_major(in1)
    B = idx0.shape[0] if idx0 is not None else in0.shape[0]
    if idx0 is not None:
        idx0 = idx0.contiguous().long()
    if idx1 is not None:
        idx1 = idx1.contiguous().long()
    out = torch.empty((B, 1), dtype=torch.float32, device=in0.device)
    with _on(in0.device):
        L.check(L.lib().b200rec_rowdot(_ptr(in0), ld0, _ptr(idx0), _ptr(in1), ld1, _ptr(idx1), in0.shape[1], B, _ptr(out), _stream()),
                'rowdot')
    return out


def scale_rows_raw(x, *, mask=None, row_scale=None, scale=1.0, add=None, out=None):
    """out = scale · x ∘ mask ∘ row_scale[:, None] (+ add) on (rows, d) fp32 blocks — b200rec_peer_scale_rows (partitioned training).
    `out` may be `x` or `add`."""
    _require_cuda(x, mask, row_scale, add, out)
    rows, d = x.shape
    if out is None:
        out = torch.empty((rows, d), dtype=torch.float32, device=x.device)
    for t in (x, mask, add, out):
        if t is not None and (t.shape != (rows, d) or t.dtype != torch.float32 or t.stride(1) != 1):
            raise ValueError('scale_rows: operands must be (rows, d) fp32 blocks with unit column stride')
    if row_scale is not None:
        row_scale = row_scale.contiguous().float()
    ld = lambda t: (t.stride(0) if rows > 1 else d) if t is not None else 0
    with _on(x.device):
        L.check(L.lib().b200rec_peer_scale_rows(_ptr(x), ld(x), rows, d, _ptr(mask), ld(mask), _ptr(row_scale), float(scale), _ptr(add), ld(add),
                                                _ptr(out), ld(out), _stream()), 'peer_scale_rows')
    return out


def rows_to_owned_raw(g, ids, row0, rows, scale, out):
    """out[ids[j] - row0] = scale · Σ_j g[j] for the ids in [row0, row0 + rows), duplicates summed in batch order (no atomics) —
    b200rec_peer_rows_to_owned.  Rows no id names are left as they are."""
    _require_cuda(g, ids, out)
    sorted_ids, perm = torch.sort(ids.long(), stable=True)
    with _on(g.device):
        L.check(L.lib().b200rec_peer_rows_to_owned(_ptr(g), g.stride(0), _ptr(sorted_ids), _ptr(perm), ids.numel(), int(row0), int(rows), g.shape[1],
                                                   float(scale), _ptr(out), out.stride(0) if rows > 1 else out.shape[1], _stream()), 'peer_rows_to_owned')
    return out


# ------------------------------------------------------------------------------------------------------------------
# K2 attention pooling
# ------------------------------------------------------------------------------------------------------------------
def set_attention_path(path: str):
    """'auto' | 'registers' | 'tma' — how K2's segment-parallel path gathers table rows (b200rec_attention_pool_set_path)"""
    L.check(L.lib().b200rec_attention_pool_set_path({'auto': 0, 'registers': 1, 'tma': 2}[path]), 'attention_pool_set_path')


def _set_dropout_seed(d, seed, device):
    """`seed`: a Python int (baked into the launch), or a one-element int64 CUDA tensor the kernels read at run time — what a captured CUDA graph
    needs, since a replay must draw a new mask (the tensor is produced by torch's graph-safe generator inside the capture)."""
    if torch.is_tensor(seed):
        if seed.device != torch.device(device) or seed.dtype != torch.int64 or seed.numel() != 1:
            raise ValueError('inner dropout: the seed tensor must be one int64 on the device of the tables')
        d.dropout_seed, d.dropout_seed_dev = 0, seed.data_ptr()
    else:
        d.dropout_seed, d.dropout_seed_dev = int(seed) & (2 ** 64 - 1), None


def attention_pool_raw(Pc, Pr, Q, *, mode=L.ATT_NET, a2=None, a20=None, bU=None, user_matrix=None, csr=None,
                       return_attention_weights=False, train_mask=None, drop_zero_scores=False, score_scale=1.0, use_workspace=True, max_row_nnz=0,
                       inner_dropout=None):
    """out (B,U) [, att (B,I)] — b200rec_attention_pool.  `csr` = (row_ptr int32, col int32, val fp32); `max_row_nnz` (CSR only,
    optional) = a host-known bound of the row lengths, so that the segment grid is not sized by I."""
    _require_cuda(Pc, Pr, Q, user_matrix)
    if Pc.dtype != torch.float32 or Pc.stride(1) != 1 or Pc.stride(0) % 4 or Pc.data_ptr() % 16:
        Pc = Pc.contiguous().float()
    if Pr.dtype != Q.dtype:
        raise ValueError('Pr and Q must share a dtype')
    if Pr.stride(1) != 1 or Pr.stride(0) % 4 or Pr.data_ptr() % 16:
        Pr = Pr.clone(memory_format=torch.contiguous_format)
    if Q.stride(1) != 1 or Q.stride(0) % 4 or Q.data_ptr() % 16:
        Q = Q.clone(memory_format=torch.contiguous_format)
    B, H = Pc.shape
    I, U = Q.shape
    if Pr.shape != (I, H):
        raise ValueError('attention_pool: table shapes disagree')
    d = L.AttentionDesc()
    keep = [Pc, Pr, Q]
    d.Pc, d.Pr, d.Q = Pc.data_ptr(), Pr.data_ptr(), Q.data_ptr()
    d.table_dtype = _dtype_code(Pr.dtype)
    d.mode = mode
    for name, t in (('a2', a2), ('a20', a20), ('bU', bU)):
        if t is not None:
            t = t.detach().contiguous().float().view(-1)
            keep.append(t)
            setattr(d, name, t.data_ptr())
    if user_matrix is not None:
        um, ld = _row_major(user_matrix)
        if um.shape != (B, I):
            raise ValueError('attention_pool: user_matrix must be (B, I)')
        keep.append(um)
        d.user_matrix, d.ld_user_matrix = um.data_ptr(), ld
    elif csr is not None:
        rp, col, val = csr
        rp, col, val = rp.contiguous().int(), col.contiguous().int(), val.contiguous().float()
        keep += [rp, col, val]
        d.row_ptr, d.col, d.val = rp.data_ptr(), col.data_ptr(), val.data_ptr()
    else:
        raise ValueError('attention_pool: need user_matrix or csr')
    d.B, d.I, d.H, d.U = B, I, H, U
    if user_matrix is None:
        d.max_row_nnz, d.nnz = max(0, int(max_row_nnz)), int(csr[1].numel())
        wsb = L.lib().b200rec_attention_pool_workspace_csr(B, I, U, d.max_row_nnz, d.nnz) if use_workspace else 0
    else:
        wsb = L.lib().b200rec_attention_pool_workspace(B, I, U, 1) if use_workspace else 0
    if wsb:
        ws = torch.empty(wsb, dtype=torch.uint8, device=Pc.device)
        keep.append(ws)
        d.workspace, d.workspace_bytes = ws.data_ptr(), wsb
    d.ld_pr, d.ld_q = (Pr.stride(0) if I > 1 else H), (Q.stride(0) if I > 1 else U)
    d.ld_pc = Pc.stride(0) if B > 1 else H
    out = torch.empty((B, U), dtype=torch.float32, device=Pc.device)
    d.out, d.ldo = out.data_ptr(), U
    att = None
    if return_attention_weights:
        att = torch.zeros((B, I), dtype=torch.float32, device=Pc.device)
        d.att_weights = att.data_ptr()
    if train_mask is not None:
        Ec, Er, atol, rtol = train_mask
        Ec, Er = Ec.detach().contiguous().float(), Er.detach().contiguous().float()
        keep += [Ec, Er]
        d.train_cand_emb, d.train_rated_emb, d.E, d.atol, d.rtol = Ec.data_ptr(), Er.data_ptr(), Ec.shape[1], atol, rtol
    d.drop_zero_scores = int(drop_zero_scores)
    d.score_scale = float(score_scale)
    if B == 0:
        return (out, att) if return_attention_weights else out
    entry = L.lib().b200rec_attention_pool
    if inner_dropout is not None and inner_dropout[0] > 0.0:
        # training: AttentionNet's Dropout between ReLU and the head Linear (attention_ncf.py:112-117), mask = Philox keyed by `seed`
        if mode != L.ATT_NET or Pr.dtype != torch.float32:
            raise ValueError('inner dropout belongs to the AttentionNet variant with fp32 tables')
        d.dropout_p = float(inner_dropout[0])
        _set_dropout_seed(d, inner_dropout[1], Pc.device)
        entry = L.lib().b200rec_attention_pool_dropout
    with _on(Pc.device), _timed('attention_pool', (B, I, H, U)):
        L.check(entry(C.byref(d), _stream()), 'attention_pool')
    return (out, att) if return_attention_weights else out


# ------------------------------------------------------------------------------------------------------------------
# K3 SpMM
# ------------------------------------------------------------------------------------------------------------------
def spmm_raw(index, t, *, w, dinv=None, x_next=None, acc_in=None, acc_out=None, acc_scale=1.0, skip_bits=None, att_src=None, push=None,
             push_stats=None):
    """One propagation step over a `GraphIndex` (graph.py): b200rec_spmm.  Returns nothing; writes x_next / acc_out.
    `push` = (host array of arena addresses, parts, rows per part, element offset, leading dimension): finished rows go to the
    receive slot of their owner rank instead (peer.py: reduce-scatter fused into the epilogue).  With `att_src` (LightGAT) the
    pushed rows are unnormalised and `push_stats` = element offset of this rank's (m, l) slot in the arenas is required."""
    _require_cuda(t)
    if t.stride(1) != 1:
        t = t.contiguous()
    d = L.SpmmDesc()
    d.chunk_row, d.chunk_start, d.chunk_slot = index.chunk_row.data_ptr(), index.chunk_start.data_ptr(), index.chunk_slot.data_ptr()
    d.n_chunks, d.chunk_size = index.n_chunks, index.chunk_size
    d.row_ptr, d.col = index.row_ptr.data_ptr(), index.col.data_ptr()
    d.w = w.data_ptr() if w is not None else None
    d.perm = index.pos.data_ptr()
    d.skip_bits = skip_bits.data_ptr() if skip_bits is not None else None
    d.t, d.t_dtype, d.ld_t, d.d = t.data_ptr(), _dtype_code(t.dtype), t.stride(0), t.shape[1]
    d.dinv = dinv.data_ptr() if dinv is not None else None
    partials = None
    if index.n_multi > 0:
        partials = torch.empty((index.n_slots, t.shape[1]), dtype=torch.float32, device=t.device)
        d.partials = partials.data_ptr()
    if x_next is not None:
        d.x_next, d.ld_x = x_next.data_ptr(), x_next.stride(0)
    if acc_out is not None:
        d.acc_out, d.ld_acc = acc_out.data_ptr(), acc_out.stride(0)
        if acc_in is not None:
            if acc_in.stride(0) != acc_out.stride(0):
                raise ValueError('spmm: acc_in and acc_out must share a leading dimension')
            d.acc_in = acc_in.data_ptr()
    d.acc_scale = acc_scale
    if index.n_multi > 0:
        d.multi_row, d.multi_first_slot, d.multi_n_slots = (index.multi_row.data_ptr(), index.multi_first_slot.data_ptr(),
                                                            index.multi_n_slots.data_ptr())
    d.n_multi = index.n_multi
    if push is not None:
        dst, parts, rpp, off, ld = push
        if x_next is not None or acc_out is not None:
            raise ValueError('spmm: `push` replaces x_next / acc_out')
        if att_src is not None and push_stats is None:
            raise ValueError('spmm: LightGAT with `push` needs `push_stats` (the softmax state travels with the rows)')
        for q in range(parts):
            d.push_dst[q] = dst[q]
        d.push_parts, d.push_rows_per_part, d.push_offset, d.push_ld = parts, rpp, off, ld
        d.push_stats_offset = push_stats or 0
    ml = None
    if att_src is not None:
        att_src = att_src.contiguous().float().view(-1)
        d.att_src = att_src.data_ptr()
        if index.n_multi > 0:
            ml = torch.empty((index.n_slots, 2), dtype=torch.float32, device=t.device)
            d.partials_ml = ml.data_ptr()
    with _on(t.device), _timed('spmm', (index.e1 + index.e2, t.shape[1])):
        L.check(L.lib().b200rec_spmm(C.byref(d), _stream()), 'spmm')


STREAM_MAX_NNZ = 16_000_000


def stream_applicable(t, nnz, *, skip_bits=None, att_src=None):
    """the stream kernel covers LightGCN inference with 64 < node_emb <= 128 (a lane owns 4 columns) on indices of up to STREAM_MAX_NNZ
    entries — the shards of a partitioned graph, where it is 5-15 % faster (profiles/r02); narrower rows and the whole 50 M-entry graph
    (1.43 vs 1.42 ms per layer) keep the row-owner kernel"""
    return (skip_bits is None and att_src is None and 64 < t.shape[1] <= 128 and t.shape[1] % 4 == 0 and 0 < nnz <= STREAM_MAX_NNZ)


def spmm_stream_raw(plan, t, *, x_next=None, acc_in=None, acc_out=None, acc_scale=1.0, push=None):
    """One propagation step over a `graph.StreamPlan`: b200rec_spmm_stream (the destination normalisation lives in the plan's entry values)."""
    _require_cuda(t)
    if t.stride(1) != 1:
        t = t.contiguous()
    d = L.SpmmStreamDesc()
    d.colf, d.wd, d.nnz, d.seg, d.n_segs = plan.colf.data_ptr(), plan.wd.data_ptr(), plan.nnz, plan.seg, plan.n_segs
    d.seg_first_j, d.seg_head_slot, d.seg_tail_slot = plan.seg_first_j.data_ptr(), plan.seg_head_slot.data_ptr(), plan.seg_tail_slot.data_ptr()
    d.rows_ne, d.n_ne = plan.rows_ne.data_ptr() if plan.n_ne else None, plan.n_ne
    d.rows_empty, d.n_empty = plan.rows_empty.data_ptr() if plan.n_empty else None, plan.n_empty
    d.t, d.t_dtype, d.ld_t, d.d = t.data_ptr(), _dtype_code(t.dtype), t.stride(0), t.shape[1]
    partials = None
    if plan.n_multi > 0:
        partials = torch.empty((plan.n_slots, t.shape[1]), dtype=torch.float32, device=t.device)
        d.partials = partials.data_ptr()
        d.multi_row, d.multi_first_slot, d.multi_n_slots = plan.multi_row.data_ptr(), plan.multi_first_slot.data_ptr(), plan.multi_n_slots.data_ptr()
    d.n_multi = plan.n_multi
    if x_next is not None:
        d.x_next, d.ld_x = x_next.data_ptr(), x_next.stride(0)
    if acc_out is not None:
        d.acc_out, d.ld_acc = acc_out.data_ptr(), acc_out.stride(0)
        if acc_in is not None:
            if acc_in.stride(0) != acc_out.stride(0):
                raise ValueError('spmm: acc_in and acc_out must share a leading dimension')
            d.acc_in = acc_in.data_ptr()
    d.acc_scale = acc_scale
    if push is not None:
        dst, parts, rpp, off, ld = push
        if x_next is not None or acc_out is not None:
            raise ValueError('spmm: `push` replaces x_next / acc_out')
        for q in range(parts):
            d.push_dst[q] = dst[q]
        d.push_parts, d.push_rows_per_part, d.push_offset, d.push_ld = parts, rpp, off, ld
    with _on(t.device), _timed('spmm', (plan.nnz, t.shape[1])):
        L.check(L.lib().b200rec_spmm_stream(C.byref(d), _stream()), 'spmm_stream')


def propagate_step(index, t, *, dinv, x_next=None, acc_in=None, acc_out=None, acc_scale=1.0, skip_bits=None, att_src=None, push=None,
                   push_stats=None):
    """x' = dinv ∘ (A_w · t) (+ the fused running mean / the push epilogue) on whichever K3 form applies: the edge-balanced stream kernel for
    LightGCN inference at 64 < d <= 128, else the row-owner chunk kernel."""
    if stream_applicable(t, int(index.col.numel()), skip_bits=skip_bits, att_src=att_src):
        from .graph import stream_plan
        return spmm_stream_raw(stream_plan(index, dinv), t, x_next=x_next, acc_in=acc_in, acc_out=acc_out, acc_scale=acc_scale, push=push)
    return spmm_raw(index, t, w=index.w, dinv=dinv, x_next=x_next, acc_in=acc_in, acc_out=acc_out, acc_scale=acc_scale, skip_bits=skip_bits,
                    att_src=att_src, push=push, push_stats=push_stats)


class _PropagateFn(torch.autograd.Function):
    """x_next = dinv ∘ (A_w · t).  backward = the same kernel on the reverse-direction weights (graph.py: w_bwd)."""

    @staticmethod
    def forward(ctx, t, index, w, w_bwd, dinv, skip_bits):
        x_next = torch.empty((index.num_nodes, t.shape[1]), dtype=torch.float32, device=t.device)
        spmm_raw(index, t, w=w, dinv=dinv, x_next=x_next, skip_bits=skip_bits)
        ctx.index, ctx.w_bwd, ctx.dinv, ctx.skip_bits, ctx.has_w = index, w_bwd, dinv, skip_bits, w is not None
        return x_next

    @staticmethod
    def backward(ctx, g):
        index = ctx.index
        gs = (g * ctx.dinv[:, None]).contiguous() if ctx.dinv is not None else g.contiguous()
        gt = torch.empty_like(gs)
        if getattr(index, 'symmetric', False) and ctx.w_bwd is not None:
            # both lists hold the same pairs position by position (binary=False): A^T has the sparsity of A, only the weights differ
            spmm_raw(index, gs, w=ctx.w_bwd, dinv=None, x_next=gt, skip_bits=ctx.skip_bits)
        else:
            # binary graphs (graph_providers.py:33,42 filter the two lists by different thresholds) are NOT symmetric: gt = A^T·gs needs
            # the index of the reversed edges
            if ctx.skip_bits is not None:
                raise NotImplementedError('edge masking on a non-symmetric graph (the reference has the same restriction, graph_providers.py:13)')
            tr = index.transposed()
            spmm_raw(tr, gs, w=tr.w, dinv=None, x_next=gt)
        return gt, None, None, None, None, None


def propagate(t, index, w, w_bwd, dinv, skip_bits=None):
    return _PropagateFn.apply(t, index, w, w_bwd, dinv, skip_bits)


class _GatPropagateFn(torch.autograd.Function):
    """LightGATConv step (gnn_ncf.py:128-177): x'[r] = Σ_{k in row r} w_k·α_k·t[s_k],  α = softmax over the row of the SOURCE scores ps[s_k] with PyG's
    `+1e-16` denominator (the destination half of the Linear(2d, 1) and its bias are constant within a row and cancel).
    forward: K3 with the online edge softmax.  backward (closed form, per edge k of row r):
        dα_k = w_k·<g[r], t[s_k]>        da_k = α_k·(dα_k − Σ_j α_j dα_j)        dps[s] = Σ_{k: s_k = s} da_k        dt[s] = Σ_{k: s_k = s} w_k α_k g[r_k]
    dt runs on K3 over the index of the reversed edges with the per-edge weights w·α carried over; the per-edge dot products are formed in chunks of
    2^20 edges with torch CUDA ops (training-side glue, like the other backward passes of this file)."""

    @staticmethod
    def forward(ctx, t, ps, index, skip_bits):
        x_next = torch.empty((index.num_nodes, t.shape[1]), dtype=torch.float32, device=t.device)
        spmm_raw(index, t, w=index.w, dinv=None, x_next=x_next, skip_bits=skip_bits, att_src=ps)
        ctx.index, ctx.skip_bits = index, skip_bits
        ctx.save_for_backward(t, ps)
        return x_next

    @staticmethod
    def backward(ctx, g):
        t, ps = ctx.saved_tensors
        index, skip = ctx.index, ctx.skip_bits
        dev = t.device
        g = g.contiguous().float()
        rp, col = index.row_ptr.long(), index.col.long()
        n, nnz = index.num_nodes, col.numel()
        rows = torch.repeat_interleave(torch.arange(n, device=dev), rp[1:] - rp[:-1])
        a = ps.detach().float().view(-1)[col]
        alive = torch.ones(nnz, dtype=torch.bool, device=dev)
        if skip is not None:                                                    # target edges of the batch take no part in the softmax
            pos = index.pos.long()
            alive = ((skip.long()[pos >> 5] >> (pos & 31)) & 1) == 0
            a = torch.where(alive, a, torch.full_like(a, float('-inf')))
        amax = torch.full((n,), float('-inf'), device=dev).scatter_reduce(0, rows, a, reduce='amax', include_self=True)
        e = torch.where(alive, (a - amax[rows]).exp(), torch.zeros_like(a))
        den = torch.zeros(n, device=dev).index_add_(0, rows, e) + 1e-16
        alpha = e / den[rows]
        w = index.w if index.w is not None else torch.ones(nnz, device=dev)
        d_alpha = torch.empty(nnz, device=dev)
        for k0 in range(0, nnz, 1 << 20):
            k1 = min(nnz, k0 + (1 << 20))
            d_alpha[k0:k1] = (g[rows[k0:k1]] * t.detach().float()[col[k0:k1]]).sum(1)
        d_alpha = d_alpha * w
        row_dot = torch.zeros(n, device=dev).index_add_(0, rows, alpha * d_alpha)
        d_a = alpha * (d_alpha - row_dot[rows])
        d_ps = torch.zeros(n, device=dev).index_add_(0, col, d_a).view(ps.shape)
        # dt = A_{w·α}^T g on K3 over the reversed index; its entries find their forward entry through (edge list, position)
        tr = index.transposed()
        k_items = index.e1                                                      # item rows come first and hold exactly the u2i list (destination = item)
        inv_u2i = torch.empty(index.e1, dtype=torch.long, device=dev)
        inv_i2u = torch.empty(index.e2, dtype=torch.long, device=dev)
        fpos = index.pos.long()
        inv_u2i[fpos[:k_items]] = torch.arange(k_items, device=dev)            # forward entries of item rows hold the u2i list (destination = item)
        inv_i2u[fpos[k_items:]] = torch.arange(k_items, nnz, device=dev)
        tpos = tr.pos.long()
        kt = tr.e2                                                              # transposed item rows hold the flipped i2u list (e2 entries), then user rows the flipped u2i list
        fwd = torch.cat((inv_i2u[tpos[:kt]], inv_u2i[tpos[kt:]]))
        wt = (w * alpha)[fwd].contiguous()
        gt = torch.empty_like(g)
        spmm_raw(tr, g, w=wt, dinv=None, x_next=gt)
        return gt, d_ps, None, None


def propagate_gat(t, ps, index, skip_bits=None):
    return _GatPropagateFn.apply(t, ps, index, skip_bits)


# ------------------------------------------------------------------------------------------------------------------
# K2 autograd wrapper
# ------------------------------------------------------------------------------------------------------------------
ATT_BWD_SLICES = 4   # CTAs per candidate row in K2's backward: 0.170 ms (1) / 0.116 (4) / 0.114 (8) at config 2


def _f32_rows(t):
    """fp32, unit column stride, 16-byte aligned rows (what the 128-bit loads of K2 need); copies only when it must"""
    if t.dtype != torch.float32 or t.stride(1) != 1 or t.stride(0) % 4 or t.data_ptr() % 16:
        t = t.contiguous().float()
    return t


def attention_pool_backward_raw(Pc, Pr, Q, a2, bU, um, att, out, grad_out, mode, score_scale=1.0, inner_dropout=None):
    """(dPc, dPr, dQ, da2, da20) — b200rec_attention_pool_backward (csrc/attention_pool_bwd.cu).  `att` / `out` are the forward's
    attention weights and output; da2 / da20 are None in mode DOT."""
    _require_cuda(Pc, Pr, Q, um, att, out, grad_out)
    Pc, Pr, Q, out, grad_out = (_f32_rows(t.detach()) for t in (Pc, Pr, Q, out, grad_out))
    um, ld_um = _row_major(um.detach())
    att = att.detach().contiguous().float()
    B, H = Pc.shape
    I, U = Q.shape
    dev = Pc.device
    S = ATT_BWD_SLICES if I >= 1024 else 1              # CTAs per candidate row (long rows would otherwise set the tail)
    dPc = torch.empty((S * B, H), dtype=torch.float32, device=dev)
    dPr = torch.zeros((I, H), dtype=torch.float32, device=dev)
    dQ = torch.zeros((I, U), dtype=torch.float32, device=dev)
    net = mode == L.ATT_NET
    da2_rows = torch.empty((S * B, H), dtype=torch.float32, device=dev) if net else None
    da20_rows = torch.empty((S * B,), dtype=torch.float32, device=dev) if net else None
    if B == 0 or I == 0:
        dPc.zero_()
        return dPc, dPr, dQ, (torch.zeros(H, device=dev) if net else None), (torch.zeros((), device=dev) if net else None)
    d = L.AttentionBwdDesc()
    d.Pc, d.Pr, d.Q, d.mode = Pc.data_ptr(), Pr.data_ptr(), Q.data_ptr(), mode
    keep = []
    if net:
        a2c = a2.detach().contiguous().float().view(-1)
        keep.append(a2c)
        d.a2 = a2c.data_ptr()
    if bU is not None:
        buc = bU.detach().contiguous().float().view(-1)
        keep.append(buc)
        d.bU = buc.data_ptr()
    d.user_matrix, d.ld_user_matrix = um.data_ptr(), ld_um
    d.att_weights, d.out, d.ldo = att.data_ptr(), out.data_ptr(), (out.stride(0) if B > 1 else U)
    d.grad_out, d.ld_grad_out = grad_out.data_ptr(), (grad_out.stride(0) if B > 1 else U)
    d.B, d.I, d.H, d.U, d.score_scale, d.n_slices = B, I, H, U, float(score_scale), S
    d.ld_pc, d.ld_pr, d.ld_q = (Pc.stride(0) if B > 1 else H), (Pr.stride(0) if I > 1 else H), (Q.stride(0) if I > 1 else U)
    d.dPc, d.dPr, d.dQ = dPc.data_ptr(), dPr.data_ptr(), dQ.data_ptr()
    if net:
        d.da2_rows, d.da20_rows = da2_rows.data_ptr(), da20_rows.data_ptr()
    if inner_dropout is not None and inner_dropout[0] > 0.0:
        d.dropout_p = float(inner_dropout[0])
        _set_dropout_seed(d, inner_dropout[1], dev)
    with _on(dev), _timed('attention_pool_backward', (B, I, H, U)):
        L.check(L.lib().b200rec_attention_pool_backward(C.byref(d), _stream()), 'attention_pool_backward')
    if S > 1:
        dPc = dPc.view(S, B, H).sum(0)
    return dPc, dPr, dQ, (da2_rows.sum(0) if net else None), (da20_rows.sum() if net else None)


class _AttentionPoolFn(torch.autograd.Function):
    """forward: K2 (always with the attention weights, which the backward kernel consumes).  backward: csrc/attention_pool_bwd.cu;
    only the column sums of the per-row a2 / a20 parts and of grad_out (dbU) are torch reductions."""

    @staticmethod
    def forward(ctx, Pc, Pr, Q, a2, a20, bU, um, mode, want_att, train_mask, drop_zero_scores, score_scale, inner_dropout=None):
        out, att = attention_pool_raw(Pc, Pr, Q, mode=mode, a2=a2, a20=a20, bU=bU, user_matrix=um, return_attention_weights=True,
                                      train_mask=train_mask, drop_zero_scores=drop_zero_scores, score_scale=score_scale, inner_dropout=inner_dropout)
        ctx.mode, ctx.scale, ctx.inner_dropout = mode, score_scale, inner_dropout
        ctx.shapes = (None if a2 is None else a2.shape, None if a20 is None else a20.shape, None if bU is None else bU.shape)
        ctx.save_for_backward(Pc, Pr, Q, a2, bU, um, att, out)
        ctx.mark_non_differentiable(att)
        return out, att

    @staticmethod
    def backward(ctx, g, _g_att=None):
        Pc, Pr, Q, a2, bU, um, att, out = ctx.saved_tensors
        dPc, dPr, dQ, da2, da20 = attention_pool_backward_raw(Pc, Pr, Q, a2, bU, um, att, out, g, ctx.mode, ctx.scale, ctx.inner_dropout)
        s_a2, s_a20, s_bU = ctx.shapes
        d_a2 = da2.view(s_a2) if (s_a2 is not None and da2 is not None) else None
        d_a20 = da20.view(s_a20) if (s_a20 is not None and da20 is not None) else None
        d_bU = g.sum(0).view(s_bU) if s_bU is not None else None
        return (dPc, dPr, dQ, d_a2, d_a20, d_bU, None, None, None, None, None, None, None)


def attention_pool(Pc, Pr, Q, *, mode, a2, a20, bU, user_matrix, return_attention_weights=False, train_mask=None,
                   drop_zero_scores=False, score_scale=1.0, inner_dropout=None):
    """`inner_dropout` = (p, seed): AttentionNet's Dropout on ReLU(Pc + Pr) in training mode (fused, regenerated by the backward kernel)."""
    needs = torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in (Pc, Pr, Q, a2, a20, bU))
    if needs:
        out, att = _AttentionPoolFn.apply(Pc, Pr, Q, a2, a20, bU, user_matrix, mode, return_attention_weights, train_mask,
                                          drop_zero_scores, score_scale, inner_dropout)
        return (out, att) if return_attention_weights else out
    return attention_pool_raw(Pc, Pr, Q, mode=mode, a2=a2, a20=a20, bU=bU, user_matrix=user_matrix,
                              return_attention_weights=return_attention_weights, train_mask=train_mask,
                              drop_zero_scores=drop_zero_scores, score_scale=score_scale, inner_dropout=inner_dropout)


# ------------------------------------------------------------------------------------------------------------------
# K8 whole-catalogue attention pooling (attention_ncf.py:136-224 for every catalogue item of many users, backend.py:78-121)
# ------------------------------------------------------------------------------------------------------------------
def _check_rows(t, what):
    if t.dim() != 2 or t.dtype != torch.float32 or t.stride(1) != 1 or t.stride(0) % 4 or t.data_ptr() % 16:
        raise ValueError(f'attention_recommend: {what} must be a 2-D fp32 table with unit column stride, 16-byte aligned rows')
    return t.stride(0) if t.shape[0] > 1 else max(t.stride(0), (t.shape[1] + 3) // 4 * 4)


def attention_recommend_raw(Pc, Pr, Ai, Qp, *, mode, a2, a20, list_ptr, list_item, list_val, users, out=None):
    """h1 = ReLU(Ai[b] + Σ_i softmax_i(s_bi)·val_i·Qp[i]) for every (user of `users`, catalogue row b) — b200rec_attention_recommend.
    Pc / Pr (nI, H) score tables (mode ATT_NET: s = a2·ReLU(Pc[b] + Pr[i]) + a20; ATT_DOT: s = <Pc[b], Pr[i]>); Ai / Qp (nI, H1P) with
    H1P in {32, 64, 128, 256}; the rating lists in K6's resident format (list_ptr int64, list_item int32, list_val fp32 centred); `users`
    int64 list rows.  Returns (len(users)·nI, H1P) fp32, row u·nI + b (or fills `out` of that shape).
    The dtype of Qp picks the kernel: fp32 runs K8; bf16 runs K8b (b200rec_attention_recommend_bf16: the same scores and α, the pooling
    on bf16 tensor cores with the weights α·val rounded to bf16, fp32 accumulation)."""
    _require_cuda(Pc, Pr, Ai, Qp, a2, a20, list_ptr, list_item, list_val, users, out)
    if list_ptr.dtype != torch.int64 or users.dtype != torch.int64:
        raise ValueError('attention_recommend: list_ptr and users must be int64')
    if list_item.dtype != torch.int32:
        raise ValueError('attention_recommend: list_item must be int32')
    if list_val.dtype != torch.float32:
        raise ValueError('attention_recommend: list_val must be float32')
    nI, H = Pc.shape
    H1P = Ai.shape[1]
    if Pr.shape != (nI, H) or Ai.shape[0] != nI or Qp.shape != (nI, H1P):
        raise ValueError('attention_recommend: table shapes disagree')
    ld_pc, ld_pr, ld_ai = _check_rows(Pc, 'Pc'), _check_rows(Pr, 'Pr'), _check_rows(Ai, 'Ai')
    lib = L.lib()
    if Qp.dtype == torch.float32:
        ld_q, entry, name = _check_rows(Qp, 'Qp'), lib.b200rec_attention_recommend, 'attention_recommend'
    elif Qp.dtype == torch.bfloat16:
        if Qp.dim() != 2 or Qp.stride(1) != 1 or Qp.stride(0) % 8 or Qp.data_ptr() % 16:
            raise ValueError('attention_recommend: a bf16 Qp must be a 2-D table with unit column stride, 16-byte aligned rows')
        ld_q = Qp.stride(0) if Qp.shape[0] > 1 else max(Qp.stride(0), (H1P + 7) // 8 * 8)
        entry, name = lib.b200rec_attention_recommend_bf16, 'attention_recommend_bf16'
    else:
        raise ValueError(f'attention_recommend: Qp must be float32 (K8) or bfloat16 (K8b), not {Qp.dtype}')
    list_ptr, list_item, list_val, users = list_ptr.contiguous(), list_item.contiguous(), list_val.contiguous(), users.contiguous()
    if a2 is not None:
        a2 = a2.detach().contiguous().float()
    if a20 is not None:
        a20 = a20.detach().contiguous().float()
    nU = users.numel()
    if out is None:
        out = torch.empty((nU * nI, H1P), dtype=torch.float32, device=Pc.device)
    elif out.shape != (nU * nI, H1P) or out.dtype != torch.float32 or out.stride(1) != 1:
        raise ValueError('attention_recommend: bad `out`')
    ldo = out.stride(0) if out.shape[0] > 1 else H1P
    with _on(Pc.device), _timed(name, (nU, nI, H, H1P)):
        L.check(entry(_ptr(Pc), ld_pc, _ptr(Pr), ld_pr, H, int(mode), _ptr(a2), _ptr(a20), _ptr(Ai), ld_ai, _ptr(Qp), ld_q, H1P, nI, _ptr(list_ptr),
                      _ptr(list_item), _ptr(list_val), _ptr(users), nU, _ptr(out), ldo, _stream()), name)
    return out


def attention_explain_raw(Pc, Pr, *, mode, a2, a20, list_ptr, list_item, list_val, users, items, explain_factor=1.5, explain_constant=0.025):
    """The list entries i of user `users[u]` with α_bi > explain_factor · (1 / max(R_u, 1)) + explain_constant for every candidate b = items[u, j]
    (src/webapp/backend.py:102-110) — b200rec_attention_explain_count, one read-back of the total, b200rec_attention_explain_fill.
    Pc / Pr / mode / a2 / a20 and the rating lists as for `attention_recommend_raw`; `items` (nU, k) int64 catalogue rows, 1 <= k <= 64, rows
    outside [0, nI) are padding.  Returns (ptr (nU·k + 1,) int64, because (n,) int64 catalogue rows, attention (n,) fp32): row u·k + j explains
    items[u, j], its entries in list order."""
    _require_cuda(Pc, Pr, a2, a20, list_ptr, list_item, list_val, users, items)
    if list_ptr.dtype != torch.int64 or users.dtype != torch.int64 or items.dtype != torch.int64:
        raise ValueError('attention_explain: list_ptr, users and items must be int64')
    if list_item.dtype != torch.int32:
        raise ValueError('attention_explain: list_item must be int32')
    if list_val.dtype != torch.float32:
        raise ValueError('attention_explain: list_val must be float32')
    nI, H = Pc.shape
    if Pr.shape != (nI, H):
        raise ValueError('attention_explain: table shapes disagree')
    if items.dim() != 2 or items.shape[0] != users.numel():
        raise ValueError('attention_explain: items must be (len(users), k)')
    ld_pc, ld_pr = _check_rows(Pc, 'Pc'), _check_rows(Pr, 'Pr')
    list_ptr, list_item, list_val, users, items = (t.contiguous() for t in (list_ptr, list_item, list_val, users, items))
    if a2 is not None:
        a2 = a2.detach().contiguous().float()
    if a20 is not None:
        a20 = a20.detach().contiguous().float()
    nU, k = items.shape
    dev = Pc.device
    lib = L.lib()
    ptr = torch.empty(nU * k + 1, dtype=torch.int64, device=dev)
    wsb = int(lib.b200rec_attention_explain_workspace(nU, k))
    ws = torch.empty(max(wsb, 16), dtype=torch.uint8, device=dev)
    args = (_ptr(Pc), ld_pc, _ptr(Pr), ld_pr, H, int(mode), _ptr(a2), _ptr(a20), nI, _ptr(list_ptr), _ptr(list_item), _ptr(list_val), _ptr(users),
            nU, _ptr(items), k)
    with _on(dev):
        with _timed('attention_explain_count', (nU, k, H)):
            L.check(lib.b200rec_attention_explain_count(*args, float(explain_factor), float(explain_constant), _ptr(ptr), _ptr(ws), ws.numel(),
                                                        _stream()), 'attention_explain_count')
        n = int(ptr[-1].item())
        because = torch.empty(n, dtype=torch.int64, device=dev)
        attention = torch.empty(n, dtype=torch.float32, device=dev)
        if n:
            with _timed('attention_explain_fill', (nU, k, H)):
                L.check(lib.b200rec_attention_explain_fill(*args, _ptr(ptr), _ptr(ws), ws.numel(), _ptr(because), _ptr(attention), _stream()),
                        'attention_explain_fill')
    return ptr, because, attention


# ------------------------------------------------------------------------------------------------------------------
# top-k
# ------------------------------------------------------------------------------------------------------------------
def topk_rows(scores, k):
    """(values (R,k), indices (R,k) int64) of the k largest entries of every row, descending — b200rec_topk_rows."""
    _require_cuda(scores)
    squeeze = scores.dim() == 1
    s2 = scores.view(1, -1) if squeeze else scores
    s2, ld = _row_major(s2)
    R, Cc = s2.shape
    val = torch.empty((R, k), dtype=torch.float32, device=s2.device)
    idx = torch.empty((R, k), dtype=torch.int64, device=s2.device)
    with _on(s2.device), _timed('topk', (R, Cc, k)):
        L.check(L.lib().b200rec_topk_rows(_ptr(s2), R, Cc, ld, k, _ptr(val), _ptr(idx), _stream()), 'topk_rows')
    return (val[0], idx[0]) if squeeze else (val, idx)


# ------------------------------------------------------------------------------------------------------------------
# K6 device-side collate (dynamic_profiles_provider.py:30-73)
# ------------------------------------------------------------------------------------------------------------------
def collate_interacted_raw(user_rows, list_ptr, list_item, list_val, n_items, *, rated_capacity, nnz_capacity):
    """(rated int64 (rated_capacity,), um_row_ptr int32 (B+1,), um_col int32, um_val fp32 (nnz_capacity,), counts int32 (2,) = [I, nnz])
    — b200rec_collate_interacted.  `user_rows` int64 (B,) device; the rating lists (`list_ptr` int64, `list_item` int32, `list_val`
    fp32 or None) are the provider's resident CSR.  Nothing is read back here: the caller decides when to learn I."""
    _require_cuda(user_rows, list_ptr, list_item, list_val)
    if user_rows.dtype != torch.int64 or list_ptr.dtype != torch.int64 or list_item.dtype != torch.int32:
        raise ValueError('collate_interacted: user_rows / list_ptr must be int64, list_item int32')
    if list_val is not None and list_val.dtype != torch.float32:
        raise ValueError('collate_interacted: list_val must be float32')
    user_rows = user_rows.contiguous()
    dev = user_rows.device
    B = int(user_rows.numel())
    rated = torch.empty(max(int(rated_capacity), 1), dtype=torch.int64, device=dev)
    rp = torch.empty(B + 1, dtype=torch.int32, device=dev)
    col = torch.empty(max(int(nnz_capacity), 1), dtype=torch.int32, device=dev)
    val = torch.empty(max(int(nnz_capacity), 1), dtype=torch.float32, device=dev)
    counts = torch.empty(2, dtype=torch.int32, device=dev)
    wsb = L.lib().b200rec_collate_workspace(B, int(n_items))
    ws = torch.empty(max(wsb, 1), dtype=torch.uint8, device=dev)
    with _on(dev), _timed('collate', (B, int(n_items))):
        L.check(L.lib().b200rec_collate_interacted(_ptr(user_rows), B, _ptr(list_ptr), _ptr(list_item), _ptr(list_val), int(n_items), _ptr(rated),
                                                   _ptr(rp), _ptr(col), _ptr(val), _ptr(counts), _ptr(ws), wsb, _stream()), 'collate_interacted')
    return rated, rp, col, val, counts


# ------------------------------------------------------------------------------------------------------------------
# K7 negative sampling (datasets/base.py:57-78)
# ------------------------------------------------------------------------------------------------------------------
def sample_negatives_raw(sample_rows, neg_ptr, neg_item, neg_rating, *, w, seed, offset, return_uniforms=False):
    """(negative item ids int64 (B,), position inside the list int32 (B,)[, uniforms float64 (B,)]) — b200rec_sample_negatives."""
    _require_cuda(sample_rows, neg_ptr, neg_item, neg_rating)
    if sample_rows.dtype != torch.int64 or neg_ptr.dtype != torch.int64 or neg_item.dtype != torch.int64:
        raise ValueError('sample_negatives: sample_rows / neg_ptr / neg_item must be int64')
    if neg_rating is not None and neg_rating.dtype != torch.float32:
        raise ValueError('sample_negatives: neg_rating must be float32')
    sample_rows = sample_rows.contiguous()
    dev, B = sample_rows.device, int(sample_rows.numel())
    out = torch.empty(B, dtype=torch.int64, device=dev)
    pos = torch.empty(B, dtype=torch.int32, device=dev)
    u = torch.empty(B, dtype=torch.float64, device=dev) if return_uniforms else None
    with _on(dev), _timed('sample_negatives', (B,)):
        L.check(L.lib().b200rec_sample_negatives(_ptr(sample_rows), B, _ptr(neg_ptr), _ptr(neg_item), _ptr(neg_rating), float(w),
                                                 int(seed) & (2 ** 64 - 1), int(offset) & (2 ** 64 - 1), _ptr(out), _ptr(pos), _ptr(u), _stream()),
                'sample_negatives')
    return (out, pos, u) if return_uniforms else (out, pos)


# ------------------------------------------------------------------------------------------------------------------
# K5 all-pairs scoring + top-k (tcgen05)
# ------------------------------------------------------------------------------------------------------------------
class AllPairsWeights:
    """second MLP layer in MMA-ready form (device) + the epilogue constants b2 | w3 | b3 as a HOST array (they travel in
    the kernel's parameter block)"""

    def __init__(self, buf, epi, H2):
        self.buf, self.epi, self.H2 = buf, epi, H2


def allpairs_pack(W2, b2, w3, b3, H1p, mode):
    """`AllPairsWeights` for `allpairs_topk_raw`; cached until a tensor changes (one device->host read of 2*H2+1 floats
    per weight version)."""
    _require_cuda(W2, b2, w3, b3)
    return _ap_cache.get((W2, b2, w3, b3), lambda: _allpairs_pack(W2, b2, w3, b3, H1p, mode), H1p, mode)


def _allpairs_pack(W2, b2, w3, b3, H1p, mode):
    lib = L.lib()
    H2, H1 = W2.shape
    w2p = W2.detach().float()
    if H1 != H1p or not w2p.is_contiguous():                 # zero-pad K to a multiple of 64
        w2p = torch.nn.functional.pad(w2p, (0, H1p - H1)).contiguous()
    b3c = b3.detach().float().view(-1)[:1] if b3 is not None else torch.zeros(1, device=W2.device)
    epi = torch.cat((b2.detach().float().view(-1), w3.detach().float().view(-1), b3c)).cpu().contiguous()
    nbytes = lib.b200rec_allpairs_packed_bytes(H1p, mode)
    if nbytes == 0:
        raise NotImplementedError(f'all-pairs kernel: first hidden width {H1} > 256')
    buf = torch.empty(nbytes, dtype=torch.uint8, device=W2.device)
    with _on(W2.device):
        L.check(lib.b200rec_allpairs_pack(_ptr(w2p), H1p, H2, H1p, mode, _ptr(buf), nbytes, _stream()), 'allpairs_pack')
    return AllPairsWeights(buf, epi, H2)


def allpairs_topk_raw(A, B, packed, mode, k, *, return_scores=False, seen=None, n_splits=0):
    """A (nU, H1p), B (nI, H1p) contiguous fp32 with H1p % 64 == 0.  Returns (top_val (nU,k), top_idx (nU,k) int64, scores|None)
    — b200rec_allpairs_topk.  `seen` = (ptr int32 (nU+1), idx int32 sorted per user): pairs never recommended."""
    _require_cuda(A, B, packed.buf)
    if A.dtype != torch.float32 or B.dtype != torch.float32 or not A.is_contiguous() or not B.is_contiguous():
        raise ValueError('allpairs: A and B must be contiguous fp32')
    nU, H1p = A.shape
    nI = B.shape[0]
    if B.shape[1] != H1p:
        raise ValueError('allpairs: A and B disagree on the hidden width')
    lib = L.lib()
    dev = A.device
    if n_splits <= 0:
        n_splits = lib.b200rec_allpairs_splits(nU, nI, mode)
    val = torch.empty((nU, k), dtype=torch.float32, device=dev) if k > 0 else None
    idx = torch.empty((nU, k), dtype=torch.int64, device=dev) if k > 0 else None
    scores = torch.empty((nU, nI), dtype=torch.float32, device=dev) if return_scores else None
    wsb = lib.b200rec_allpairs_workspace(nU, k, n_splits) if k > 0 else 0
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev) if wsb else None
    sp = si = None
    if seen is not None:
        sp, si = seen[0].contiguous().int(), seen[1].contiguous().int()
        if sp.numel() != nU + 1:
            raise ValueError('allpairs: seen_ptr must have nU + 1 entries')
    with _on(dev), _timed('allpairs', (nU, nI, H1p, k, mode)):
        L.check(lib.b200rec_allpairs_topk(_ptr(A), _ptr(B), nU, nI, H1p, _ptr(packed.buf), _ptr(packed.epi), packed.H2, mode, k, n_splits, _ptr(sp), _ptr(si),
                                          _ptr(scores), nI, _ptr(val), _ptr(idx), _ptr(ws), wsb, _stream()), 'allpairs_topk')
    return val, idx, scores


def allpairs_relu_dot_raw(A, B, w2, b2, k, *, return_scores=False, seen=None, n_splits=0):
    """score(u, i) = b2 + w2·ReLU(A[u] + B[i]) for every pair + the k best columns per row — b200rec_allpairs_relu_dot_topk (exact fp32)."""
    _require_cuda(A, B, w2)
    nU, H1p = A.shape
    nI = B.shape[0]
    lib = L.lib()
    dev = A.device
    w2p = torch.zeros(H1p, dtype=torch.float32, device=dev)
    w2p[:w2.numel()] = w2.float().view(-1)
    b2v = float(b2.detach().float().view(-1)[0].item()) if b2 is not None else 0.0
    if n_splits <= 0:
        n_splits = lib.b200rec_allpairs_relu_dot_splits(nU, nI)
    val = torch.empty((nU, k), dtype=torch.float32, device=dev) if k > 0 else None
    idx = torch.empty((nU, k), dtype=torch.int64, device=dev) if k > 0 else None
    scores = torch.empty((nU, nI), dtype=torch.float32, device=dev) if return_scores else None
    wsb = lib.b200rec_allpairs_workspace(nU, k, n_splits) if k > 0 else 0
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev) if wsb else None
    sp = si = None
    if seen is not None:
        sp, si = seen[0].contiguous().int(), seen[1].contiguous().int()
        if sp.numel() != nU + 1:
            raise ValueError('allpairs: seen_ptr must have nU + 1 entries')
    with _on(dev), _timed('allpairs_relu_dot', (nU, nI, H1p, k)):
        L.check(lib.b200rec_allpairs_relu_dot_topk(_ptr(A), _ptr(B), nU, nI, H1p, _ptr(w2p), b2v, k, n_splits, _ptr(sp), _ptr(si), _ptr(scores), nI,
                                                   _ptr(val), _ptr(idx), _ptr(ws), wsb, _stream()), 'allpairs_relu_dot_topk')
    return val, idx, scores


def allpairs_dot_topk_raw(A, B, k, *, return_scores=False, seen=None, n_splits=0):
    """score(u, i) = A[u]·B[i] for every pair + the k best columns per row — b200rec_allpairs_dot_topk (exact fp32, the dot form of the
    relu_dot kernel).  A (nU, H), B (nI, H) fp32 with H <= 256; widths that are not a multiple of 64 are zero-padded here.  Returns
    (top_val (nU, k), top_idx (nU, k) int64, scores (nU, nI) | None); `seen` as for `allpairs_topk_raw`."""
    _require_cuda(A, B)
    nU, H = A.shape
    nI = B.shape[0]
    if B.shape[1] != H:
        raise ValueError('allpairs_dot: A and B disagree on the width')
    Hp = max(64, (H + 63) // 64 * 64)
    if Hp > 256:
        raise NotImplementedError(f'all-pairs dot kernel: embedding width {H} > 256')
    dev = A.device
    pad = lambda t: t.float().contiguous() if H == Hp else torch.nn.functional.pad(t.float(), (0, Hp - H)).contiguous()
    A, B = pad(A), pad(B)
    lib = L.lib()
    if n_splits <= 0:
        n_splits = lib.b200rec_allpairs_relu_dot_splits(nU, nI)            # same tiling as relu_dot
    val = torch.empty((nU, k), dtype=torch.float32, device=dev) if k > 0 else None
    idx = torch.empty((nU, k), dtype=torch.int64, device=dev) if k > 0 else None
    scores = torch.empty((nU, nI), dtype=torch.float32, device=dev) if return_scores else None
    wsb = lib.b200rec_allpairs_workspace(nU, k, n_splits) if k > 0 else 0
    ws = torch.empty(wsb, dtype=torch.uint8, device=dev) if wsb else None
    sp = si = None
    if seen is not None:
        sp, si = seen[0].contiguous().int(), seen[1].contiguous().int()
        if sp.numel() != nU + 1:
            raise ValueError('allpairs: seen_ptr must have nU + 1 entries')
    with _on(dev), _timed('allpairs_dot', (nU, nI, Hp, k)):
        L.check(lib.b200rec_allpairs_dot_topk(_ptr(A), _ptr(B), nU, nI, Hp, k, n_splits, _ptr(sp), _ptr(si), _ptr(scores), nI, _ptr(val), _ptr(idx),
                                              _ptr(ws), wsb, _stream()), 'allpairs_dot_topk')
    return val, idx, scores


def mlp_allpairs_topk(row_emb, col_emb, weights, biases, k, *, rows_first=True, precision='fp32', seen=None, return_scores=False,
                      n_splits=0):
    """Scores `MLP(cat(row_emb[u], col_emb[i]))` (rows_first) or `MLP(cat(col_emb[i], row_emb[u]))` for EVERY (u, i) and keeps
    the k best columns per row.  The first Linear is split into its two halves (two K1a GEMMs over nU resp. nI rows), the rest
    runs in the fused tensor-core kernel.  precision 'fp32' = bf16 hi/lo split operands (rel <= 1e-5), 'bf16' = plain bf16."""
    n = len(weights)
    if n not in (2, 3):
        raise NotImplementedError(f'all-pairs scoring supports MLPs with 1 or 2 hidden layers (the reference uses [256], [128], '
                                  f'[256,128]); got {n - 1}')
    mode = {'fp32': L.AP_BF16X2, 'bf16': L.AP_BF16}[precision]
    W1, b1 = weights[0], biases[0]
    Er, Ec = row_emb.shape[1], col_emb.shape[1]
    H1 = W1.shape[0]
    if W1.shape[1] != Er + Ec:
        raise ValueError('all-pairs: first MLP layer does not take cat(row_emb, col_emb)')
    H1p = (H1 + 63) // 64 * 64
    if H1p > 256:
        raise NotImplementedError(f'all-pairs kernel: first hidden width {H1} > 256')
    W1r, W1c = (W1[:, :Er], W1[:, Er:]) if rows_first else (W1[:, Ec:], W1[:, :Ec])
    dev = row_emb.device
    A = torch.zeros((row_emb.shape[0], H1p), dtype=torch.float32, device=dev) if H1p != H1 else \
        torch.empty((row_emb.shape[0], H1p), dtype=torch.float32, device=dev)
    Bm = torch.zeros((col_emb.shape[0], H1p), dtype=torch.float32, device=dev) if H1p != H1 else \
        torch.empty((col_emb.shape[0], H1p), dtype=torch.float32, device=dev)
    linear_raw(row_emb, W1r, b1, out=A[:, :H1])
    linear_raw(col_emb, W1c, None, out=Bm[:, :H1])
    if n == 3:
        W2, b2, w3, b3 = weights[1], biases[1], weights[2], biases[2]
        if W2.shape[0] > 128:
            raise NotImplementedError(f'all-pairs kernel: second hidden width {W2.shape[0]} > 128')
    else:
        # one hidden layer: score = b2 + w2·ReLU(a_u + b_i) has no GEMM left — exact FP32 kernel (csrc/allpairs.cu, relu_dot).  It is also FASTER
        # than running it as two rows of the tensor-core kernel's second layer (0.47 s vs 0.83 s per 1.25e10 pairs), so the bf16 request takes it
        # too (exact is within 1e-2).
        return allpairs_relu_dot_raw(A, Bm, weights[1].detach(), biases[1], k, return_scores=return_scores, seen=seen, n_splits=n_splits)
    packed = allpairs_pack(W2, b2, w3, b3, H1p, mode)
    return allpairs_topk_raw(A, Bm, packed, mode, k, return_scores=return_scores, seen=seen, n_splits=n_splits)
