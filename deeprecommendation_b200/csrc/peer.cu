// Peer-memory exchange for the partitioned GraphNCF propagation (SURVEY.md §8e; replaces the whole-graph loop of
// gnn_ncf.py:336-345 on the GPUs of one NVSwitch box).
//
// One process per GPU.  Every rank allocates one ARENA with cudaMalloc, exports it with a CUDA IPC handle and maps the arenas
// of its peers (b200rec_peer_alloc / _open; the handles travel through torch.distributed, which is plumbing).  After that the
// data path has no library collective in it:
//
//   * K3's epilogue (csrc/spmm.cu, `push_*` fields) stores the partial item rows of a rank straight into the OWNER's receive
//     slot over NVLink (reduce-scatter fused into the SpMM);
//   * peer_reduce_kernel adds the P slots of the owned rows in rank order (deterministic) and folds the running mean in;
//     for LightGAT, peer_reduce_softmax_kernel merges the slots' unnormalised rows by their softmax state (m, l) instead;
//   * peer_push_floats_kernel copies the owners' LightGAT source scores (one float per item) into every rank's score table;
//   * K1c's epilogue (csrc/node_gemm.cu, b200rec_linear_shortk_push) writes the transformed rows into the feature table of
//     EVERY rank (all-gather fused into the transform GEMM);
//   * peer_signal_kernel / peer_wait_kernel are the cross-GPU ordering: a release store of an epoch number into every peer's
//     flag word after the producing kernel, an acquire spin (bounded by a timeout that raises an error flag instead of hanging
//     the GPU) before the consuming kernel.  Epochs are counted on the device, so a captured CUDA graph can be replayed.
//   * peer_gather_rows_kernel pushes the batch rows a rank owns into every rank's (2B, d) buffer (replaces an all-reduce).
//   * training (peer.py): peer_rows_to_owned_kernel sums the batch rows' gradient onto the owned rows in batch order and
//     peer_scale_rows_kernel applies dropout multipliers / degree scaling and accumulates partial gradients; the backward's exchanges
//     are the forward's kernels on the reverse-edge weights.
#include <math.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"

namespace b200rec {

constexpr int PEER_MAX = B200REC_PEER_MAX;

struct PeerPtrs {
  void* p[PEER_MAX];
};

__device__ __forceinline__ void st_release_sys(uint32_t* p, uint32_t v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_acquire_sys(const uint32_t* p) {
  uint32_t v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ unsigned long long globaltimer_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
  return t;
}

// flags layout (per rank, inside its arena): flags[channel * PEER_MAX + source rank]; counters (local only):
// counters[channel] = signals sent, counters[PEER_MAX_CH + channel] = waits passed.
__global__ void peer_signal_kernel(PeerPtrs flags, int n_peers, int rank, int channel, uint32_t* counters) {
  __shared__ uint32_t epoch;
  if (threadIdx.x == 0) {
    epoch = counters[channel] + 1u;
    counters[channel] = epoch;
  }
  __syncthreads();
  __threadfence_system();                       // every earlier write of this stream (incl. the remote stores) before the flag
  if ((int)threadIdx.x < n_peers)
    st_release_sys(reinterpret_cast<uint32_t*>(flags.p[threadIdx.x]) + channel * PEER_MAX + rank, epoch);
}

__global__ void peer_wait_kernel(const uint32_t* flags, int n_peers, int channel, uint32_t* counters, long long timeout_ns, int* err_flag) {
  __shared__ uint32_t epoch;
  if (threadIdx.x == 0) {
    epoch = counters[B200REC_PEER_CHANNELS + channel] + 1u;
    counters[B200REC_PEER_CHANNELS + channel] = epoch;
  }
  __syncthreads();
  if ((int)threadIdx.x < n_peers) {
    const uint32_t* f = flags + channel * PEER_MAX + threadIdx.x;
    const unsigned long long t0 = globaltimer_ns();
    while ((int)(ld_acquire_sys(f) - epoch) < 0) {
      if ((long long)(globaltimer_ns() - t0) > timeout_ns) {    // never hang the GPU: report and fall through
        atomicExch(err_flag, 1 + (int)threadIdx.x);
        break;
      }
      __nanosleep(64);
    }
  }
  __syncthreads();
  __threadfence_system();
}

// out rows = sum over the P receive slots in slot order; optional running-mean fold (same formula as K3's epilogue)
__global__ void __launch_bounds__(256) peer_reduce_kernel(const float* __restrict__ recv, int n_slots, long long slot_stride, long long ld_recv,
                                                          int rows, int d4, float* __restrict__ x_next, long long ld_x,
                                                          const float* __restrict__ acc_in, float* __restrict__ acc_out, long long ld_acc,
                                                          float acc_scale) {
  const long long total = (long long)rows * d4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / d4), c = (int)(i - (long long)r * d4) * 4;
    const float* src = recv + (long long)r * ld_recv + c;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    float4 t[8];
    for (int s0 = 0; s0 < n_slots; s0 += 8) {
#pragma unroll
      for (int k = 0; k < 8; ++k)
        t[k] = (s0 + k < n_slots) ? __ldcs(reinterpret_cast<const float4*>(src + (long long)(s0 + k) * slot_stride)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int k = 0; k < 8; ++k) { v.x += t[k].x; v.y += t[k].y; v.z += t[k].z; v.w += t[k].w; }
    }
    if (x_next) *reinterpret_cast<float4*>(x_next + (long long)r * ld_x + c) = v;
    if (acc_out) {
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if (acc_in) a = *reinterpret_cast<const float4*>(acc_in + (long long)r * ld_acc + c);
      *reinterpret_cast<float4*>(acc_out + (long long)r * ld_acc + c) =
          make_float4((a.x + v.x) * acc_scale, (a.y + v.y) * acc_scale, (a.z + v.z) * acc_scale, (a.w + v.w) * acc_scale);
    }
  }
}

// LightGAT: the P slots are unnormalised rows relative to their own softmax max; merged with PyG's rule as K3's fix-up merges chunks.
// A slot with l == 0 (nobody wrote it: the zero-initialised arena, or no edges from that rank) takes part neither in the max nor in the sums.
__global__ void __launch_bounds__(256) peer_reduce_softmax_kernel(const float* __restrict__ recv, const float* __restrict__ stats, int n_slots,
                                                                  long long slot_stride, long long ld_recv, long long stats_stride, int rows, int d4,
                                                                  float* __restrict__ x_next, long long ld_x, const float* __restrict__ acc_in,
                                                                  float* __restrict__ acc_out, long long ld_acc, float acc_scale) {
  const long long total = (long long)rows * d4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / d4), c = (int)(i - (long long)r * d4) * 4;
    const float* src = recv + (long long)r * ld_recv + c;
    const float* ml = stats + 2ll * r;
    float M = -INFINITY;
    for (int s = 0; s < n_slots; ++s) {
      const float2 v = __ldg(reinterpret_cast<const float2*>(ml + s * stats_stride));
      if (v.y > 0.f) M = fmaxf(M, v.x);
    }
    float L = 0.f;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = 0; s < n_slots; ++s) {
      const float2 st = __ldg(reinterpret_cast<const float2*>(ml + s * stats_stride));
      if (!(st.y > 0.f)) continue;
      const float e = __expf(st.x - M);
      L = fmaf(st.y, e, L);
      const float4 t = __ldcs(reinterpret_cast<const float4*>(src + (long long)s * slot_stride));
      v = make_float4(fmaf(t.x, e, v.x), fmaf(t.y, e, v.y), fmaf(t.z, e, v.z), fmaf(t.w, e, v.w));
    }
    const float inv = 1.f / (L + 1e-16f);
    v = make_float4(v.x * inv, v.y * inv, v.z * inv, v.w * inv);
    if (x_next) *reinterpret_cast<float4*>(x_next + (long long)r * ld_x + c) = v;
    if (acc_out) {
      float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
      if (acc_in) a = *reinterpret_cast<const float4*>(acc_in + (long long)r * ld_acc + c);
      *reinterpret_cast<float4*>(acc_out + (long long)r * ld_acc + c) =
          make_float4((a.x + v.x) * acc_scale, (a.y + v.y) * acc_scale, (a.z + v.z) * acc_scale, (a.w + v.w) * acc_scale);
    }
  }
}

// n floats into the same place of n_dst buffers
__global__ void __launch_bounds__(256) peer_push_floats_kernel(const float* __restrict__ src, long long n, PeerPtrs dst, int n_dst, long long dst_offset) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = src[i];
    for (int q = 0; q < n_dst; ++q) reinterpret_cast<float*>(dst.p[q])[dst_offset + i] = v;
  }
}

// copies a (rows, d) block into the same place of n_dst buffers (the local one may be among them)
__global__ void __launch_bounds__(256) peer_push_rows_kernel(const float* __restrict__ src, long long ld_src, int rows, int d4, PeerPtrs dst, int n_dst,
                                                             long long dst_offset, long long ld_dst) {
  const long long total = (long long)rows * d4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / d4), c = (int)(i - (long long)r * d4) * 4;
    const float4 v = *reinterpret_cast<const float4*>(src + (long long)r * ld_src + c);
    for (int q = 0; q < n_dst; ++q)
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(dst.p[q]) + dst_offset + (long long)r * ld_dst + c) = v;
  }
}

// batch rows: ids[j] is a global node id; the rank owning it (row0 <= id < row0 + rows) writes table[id - row0] * scale into row
// (dst_row0 + j) of every destination.  One warp per batch entry.
__global__ void __launch_bounds__(256) peer_gather_rows_kernel(const float* __restrict__ table, long long ld, long long row0, long long rows,
                                                               const long long* __restrict__ ids, int n_ids, int d4, float scale, PeerPtrs dst,
                                                               int n_dst, long long dst_offset, long long ld_dst) {
  const int w = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (w >= n_ids) return;
  const long long local = ids[w] - row0;
  if (local < 0 || local >= rows) return;
  for (int c4 = lane; c4 < d4; c4 += 32) {
    float4 v = *reinterpret_cast<const float4*>(table + local * ld + 4 * c4);
    v = make_float4(v.x * scale, v.y * scale, v.z * scale, v.w * scale);
    for (int q = 0; q < n_dst; ++q)
      *reinterpret_cast<float4*>(reinterpret_cast<float*>(dst.p[q]) + dst_offset + (long long)w * ld_dst + 4 * c4) = v;
  }
}

// training (peer.py, _train_backward): out = scale · x ∘ mask ∘ row_scale[r] (+ add) elementwise over a (rows, d) block; mask / row_scale /
// add may be null.  The conv-dropout multipliers, the degree scaling of a gradient and the accumulation of partial gradients.  out may alias
// x or add.
__global__ void __launch_bounds__(256) peer_scale_rows_kernel(const float* x, long long ld_x, int rows, int d4, const float* mask, long long ld_m,
                                                              const float* row_scale, float scale, const float* add, long long ld_add, float* out,
                                                              long long ld_out) {
  const long long total = (long long)rows * d4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(i / d4), c = (int)(i - (long long)r * d4) * 4;
    float4 v = *reinterpret_cast<const float4*>(x + (long long)r * ld_x + c);
    if (mask) {
      const float4 m = *reinterpret_cast<const float4*>(mask + (long long)r * ld_m + c);
      v = make_float4(v.x * m.x, v.y * m.y, v.z * m.z, v.w * m.w);
    }
    const float s = row_scale ? scale * row_scale[r] : scale;
    v = make_float4(v.x * s, v.y * s, v.z * s, v.w * s);
    if (add) {
      const float4 a = *reinterpret_cast<const float4*>(add + (long long)r * ld_add + c);
      v = make_float4(v.x + a.x, v.y + a.y, v.z + a.z, v.w + a.w);
    }
    *reinterpret_cast<float4*>(out + (long long)r * ld_out + c) = v;
  }
}

// training: the gradient of the batch rows onto the owned rows they were gathered from, without atomics.  sorted / perm = the batch ids
// sorted stably and their batch positions, so that the entries of one id are adjacent and in batch order.  One warp per sorted entry; the
// first entry of an id this rank owns (row0 <= id < row0 + rows) writes out[id - row0] = scale · Σ g[j] over that id's entries, in batch
// order.  Rows no entry names are not written.
__global__ void __launch_bounds__(256) peer_rows_to_owned_kernel(const float* __restrict__ g, long long ld_g, const long long* __restrict__ sorted,
                                                                 const long long* __restrict__ perm, int n, long long row0, long long rows, int d4,
                                                                 float scale, float* __restrict__ out, long long ld_out) {
  const int w = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5), lane = threadIdx.x & 31;
  if (w >= n) return;
  const long long id = sorted[w], local = id - row0;
  if (local < 0 || local >= rows || (w > 0 && sorted[w - 1] == id)) return;
  for (int c4 = lane; c4 < d4; c4 += 32) {
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s = w; s < n && sorted[s] == id; ++s) {
      const float4 v = *reinterpret_cast<const float4*>(g + perm[s] * ld_g + 4 * c4);
      acc = make_float4(acc.x + v.x, acc.y + v.y, acc.z + v.z, acc.w + v.w);
    }
    *reinterpret_cast<float4*>(out + local * ld_out + 4 * c4) = make_float4(acc.x * scale, acc.y * scale, acc.z * scale, acc.w * scale);
  }
}

// device-side tracing: one thread writes %globaltimer (ns) — a marker between the kernels of a captured forward, so that the phases of a
// rank (and the time it spends waiting for its peers) can be read back after a CUDA-graph replay
__global__ void device_timestamp_kernel(unsigned long long* slot) { *slot = globaltimer_ns(); }

static int fill_ptrs(PeerPtrs& out, void* const* in, int n, const char* what) {
  if (n <= 0 || n > PEER_MAX || !in) return b200rec_fail(B200REC_ERR_BAD_ARG, what);
  for (int q = 0; q < PEER_MAX; ++q) out.p[q] = q < n ? in[q] : nullptr;
  for (int q = 0; q < n; ++q)
    if (!out.p[q] || ((uintptr_t)out.p[q] % 16)) return b200rec_fail(B200REC_ERR_BAD_ARG, what);
  return B200REC_OK;
}

}  // namespace b200rec

using namespace b200rec;

extern "C" int b200rec_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle) {
  if (!dev_ptr || !handle || bytes == 0) return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_alloc: null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == B200REC_PEER_HANDLE_BYTES, "IPC handle size");
  void* p = nullptr;
  B200REC_CUDA(cudaMalloc(&p, bytes));
  cudaError_t e = cudaMemset(p, 0, bytes);
  if (e == cudaSuccess) e = cudaDeviceSynchronize();
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    cudaFree(p);
    return b200rec_set_cuda_error(e);
  }
  memcpy(handle, &h, sizeof(h));
  *dev_ptr = p;
  return B200REC_OK;
}

extern "C" int b200rec_peer_open(const unsigned char* handle, void** dev_ptr) {
  if (!dev_ptr || !handle) return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_open: null argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle, sizeof(h));
  void* p = nullptr;
  B200REC_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
  *dev_ptr = p;
  return B200REC_OK;
}

extern "C" int b200rec_peer_close(void* dev_ptr) {
  if (dev_ptr) B200REC_CUDA(cudaIpcCloseMemHandle(dev_ptr));
  return B200REC_OK;
}

extern "C" int b200rec_peer_free(void* dev_ptr) {
  if (dev_ptr) B200REC_CUDA(cudaFree(dev_ptr));
  return B200REC_OK;
}

extern "C" int b200rec_peer_signal(void* const* peer_flags, int n_peers, int rank, int channel, uint32_t* counters, b200rec_stream_t stream) {
  PeerPtrs f;
  if (int rc = fill_ptrs(f, peer_flags, n_peers, "peer_signal: bad flag pointers")) return rc;
  if (rank < 0 || rank >= n_peers || channel < 0 || channel >= B200REC_PEER_CHANNELS || !counters)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_signal: bad rank / channel");
  peer_signal_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(f, n_peers, rank, channel, counters);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_wait(const uint32_t* flags, int n_peers, int channel, uint32_t* counters, int64_t timeout_ns, int* err_flag,
                                 b200rec_stream_t stream) {
  if (!flags || !counters || !err_flag || n_peers <= 0 || n_peers > PEER_MAX || channel < 0 || channel >= B200REC_PEER_CHANNELS)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_wait: bad argument");
  peer_wait_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(flags, n_peers, channel, counters, timeout_ns > 0 ? timeout_ns : 2000000000ll, err_flag);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_reduce(const float* recv, int n_slots, int64_t slot_stride, int64_t ld_recv, int64_t rows, int d, float* x_next,
                                   int64_t ld_x, const float* acc_in, float* acc_out, int64_t ld_acc, float acc_scale, b200rec_stream_t stream) {
  if (rows == 0) return B200REC_OK;
  if (!recv || n_slots <= 0 || rows < 0 || d <= 0 || (d % 4) || (ld_recv % 4) || (slot_stride % 4) || ((uintptr_t)recv % 16) ||
      (x_next && (((uintptr_t)x_next % 16) || (ld_x % 4))) || (acc_out && (((uintptr_t)acc_out % 16) || (ld_acc % 4))) ||
      (acc_in && ((uintptr_t)acc_in % 16)) || rows > INT32_MAX)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_reduce: operands must allow 128-bit access (d, leading dims multiples of 4)");
  const long long total = rows * (long long)(d / 4);
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)b200rec_num_sms() * 8);
  peer_reduce_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(recv, n_slots, slot_stride, ld_recv, (int)rows, d / 4, x_next, ld_x, acc_in, acc_out,
                                                             ld_acc, acc_scale);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_reduce_softmax(const float* recv, const float* stats, int n_slots, int64_t slot_stride, int64_t ld_recv,
                                           int64_t stats_stride, int64_t rows, int d, float* x_next, int64_t ld_x, const float* acc_in, float* acc_out,
                                           int64_t ld_acc, float acc_scale, b200rec_stream_t stream) {
  if (rows == 0) return B200REC_OK;
  if (!recv || !stats || n_slots <= 0 || rows < 0 || d <= 0 || (d % 4) || (ld_recv % 4) || (slot_stride % 4) || ((uintptr_t)recv % 16) ||
      (stats_stride % 2) || ((uintptr_t)stats % 8) || (x_next && (((uintptr_t)x_next % 16) || (ld_x % 4))) ||
      (acc_out && (((uintptr_t)acc_out % 16) || (ld_acc % 4))) || (acc_in && ((uintptr_t)acc_in % 16)) || rows > INT32_MAX)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_reduce_softmax: operands must allow 128-bit access (d, leading dims multiples of 4; stats 8-byte pairs)");
  const long long total = rows * (long long)(d / 4);
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)b200rec_num_sms() * 8);
  peer_reduce_softmax_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(recv, stats, n_slots, slot_stride, ld_recv, stats_stride, (int)rows, d / 4, x_next,
                                                                     ld_x, acc_in, acc_out, ld_acc, acc_scale);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_push_floats(const float* src, int64_t n, void* const* dst, int n_dst, int64_t dst_offset, b200rec_stream_t stream) {
  if (n == 0) return B200REC_OK;
  PeerPtrs pp;
  if (int rc = fill_ptrs(pp, dst, n_dst, "peer_push_floats: bad destination pointers")) return rc;
  if (!src || n < 0 || dst_offset < 0) return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_push_floats: bad source / size / offset");
  const int grid = (int)std::min<long long>((n + 255) / 256, (long long)b200rec_num_sms() * 8);
  peer_push_floats_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, n, pp, n_dst, dst_offset);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_push_rows(const float* src, int64_t ld_src, int64_t rows, int d, void* const* dst, int n_dst, int64_t dst_offset,
                                      int64_t ld_dst, b200rec_stream_t stream) {
  if (rows == 0) return B200REC_OK;
  PeerPtrs pp;
  if (int rc = fill_ptrs(pp, dst, n_dst, "peer_push_rows: bad destination pointers")) return rc;
  if (!src || rows < 0 || rows > INT32_MAX || d <= 0 || (d % 4) || (ld_src % 4) || (ld_dst % 4) || (dst_offset % 4) || ((uintptr_t)src % 16))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_push_rows: operands must allow 128-bit access");
  const long long total = rows * (long long)(d / 4);
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)b200rec_num_sms() * 8);
  peer_push_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, ld_src, (int)rows, d / 4, pp, n_dst, dst_offset, ld_dst);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_gather_rows(const float* table, int64_t ld, int64_t row0, int64_t rows, const int64_t* ids, int64_t n_ids, int d,
                                        float scale, void* const* dst, int n_dst, int64_t dst_offset, int64_t ld_dst, b200rec_stream_t stream) {
  if (n_ids == 0) return B200REC_OK;
  PeerPtrs pp;
  if (int rc = fill_ptrs(pp, dst, n_dst, "peer_gather_rows: bad destination pointers")) return rc;
  if ((rows > 0 && !table) || !ids || n_ids < 0 || n_ids > INT32_MAX / 32 || d <= 0 || (d % 4) || (ld % 4) || (ld_dst % 4) || (dst_offset % 4) ||
      ((uintptr_t)table % 16))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_gather_rows: operands must allow 128-bit access");
  const int grid = (int)((n_ids * 32 + 255) / 256);
  peer_gather_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(table, ld, row0, rows, reinterpret_cast<const long long*>(ids), (int)n_ids, d / 4,
                                                                  scale, pp, n_dst, dst_offset, ld_dst);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_scale_rows(const float* x, int64_t ld_x, int64_t rows, int d, const float* mask, int64_t ld_m, const float* row_scale,
                                       float scale, const float* add, int64_t ld_add, float* out, int64_t ld_out, b200rec_stream_t stream) {
  if (rows == 0) return B200REC_OK;
  auto a16 = [](const void* p) { return ((uintptr_t)p % 16) == 0; };
  if (!x || !out || rows < 0 || rows > INT32_MAX || d <= 0 || (d % 4) || (ld_x % 4) || (ld_out % 4) || !a16(x) || !a16(out) ||
      (mask && (!a16(mask) || (ld_m % 4))) || (add && (!a16(add) || (ld_add % 4))))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_scale_rows: operands must allow 128-bit access (d, leading dims multiples of 4)");
  const long long total = rows * (long long)(d / 4);
  const int grid = (int)std::min<long long>((total + 255) / 256, (long long)b200rec_num_sms() * 8);
  peer_scale_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(x, ld_x, (int)rows, d / 4, mask, ld_m, row_scale, scale, add, ld_add, out, ld_out);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_rows_to_owned(const float* g, int64_t ld_g, const int64_t* sorted, const int64_t* perm, int64_t n, int64_t row0,
                                          int64_t rows, int d, float scale, float* out, int64_t ld_out, b200rec_stream_t stream) {
  if (n == 0 || rows == 0) return B200REC_OK;
  if (!g || !sorted || !perm || !out || n < 0 || n > INT32_MAX / 32 || rows < 0 || d <= 0 || (d % 4) || (ld_g % 4) || (ld_out % 4) ||
      ((uintptr_t)g % 16) || ((uintptr_t)out % 16))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_rows_to_owned: operands must allow 128-bit access");
  const int grid = (int)((n * 32 + 255) / 256);
  peer_rows_to_owned_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(g, ld_g, reinterpret_cast<const long long*>(sorted),
                                                                    reinterpret_cast<const long long*>(perm), (int)n, row0, rows, d / 4, scale, out, ld_out);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_device_timestamp(uint64_t* slot, b200rec_stream_t stream) {
  if (!slot) return b200rec_fail(B200REC_ERR_BAD_ARG, "device_timestamp: null slot");
  device_timestamp_kernel<<<1, 1, 0, (cudaStream_t)stream>>>(reinterpret_cast<unsigned long long*>(slot));
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}
