// K1b — fused NCF MLP tower (fp32 parity mode).
//
// Replaces `torch.cat((a, b), dim=1)` + `build_MLP_layers` (NCF/util.py:5-18; call sites basic_ncf.py:40-41,
// attention_ncf.py:219-222, gnn_ncf.py:354-362): Linear, then (ReLU, [Dropout: inert in eval], Linear)*.
// One CTA owns TM pairs.  The concatenation is never materialised — the two halves are read (optionally
// through a row gather, which is GraphNCF's `combined[itemIds]` / `combined[userIds]`) straight into the
// first activation buffer in shared memory, and every intermediate activation ping-pongs between two
// shared-memory buffers; only the final (B, out) scores are written to HBM.
#include "common.cuh"

namespace b200rec {

constexpr int MLP_THREADS = 256;
constexpr int MLP_KC = 32;             // k extent of a staged W tile
constexpr int MLP_WS = MLP_KC + 4;     // padded row stride (floats) of the tile
// W tiles in flight = template parameter MLP_NSTG: 4 for small batches (a CTA of a 512-pair batch is a chain of ~20 dependent
// 36 KB tile loads out of L2 — 64 CTAs, each streaming all the weights), 2 when there are CTAs enough to overlap each other.

template <int TM, int MLP_NSTG>
__global__ void __launch_bounds__(MLP_THREADS)
mlp_tower_kernel(const float* __restrict__ in0, long long ld0, const int64_t* __restrict__ idx0, int E0,
                 const float* __restrict__ in1, long long ld1, const int64_t* __restrict__ idx1, int E1, long long B,
                 b200rec_mlp_t d, float* __restrict__ out, long long ldo, int stride, int w_vec_ok) {
  extern __shared__ __align__(16) float smem[];
  float* buf0 = smem;
  float* buf1 = smem + (size_t)TM * stride;
  float* wtile = smem + (size_t)2 * TM * stride;      // MLP_NSTG x [256 x 36] floats
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long row0 = (long long)blockIdx.x * TM;

  // ---- stage the (virtually concatenated) input rows --------------------------------------------------
  const int E = E0 + E1;
  for (int r = warp; r < TM; r += MLP_THREADS / 32) {
    long long row = row0 + r;
    float* dst = buf0 + (size_t)r * stride;
    if (row < B) {
      long long s0 = idx0 ? idx0[row] : row;
      const float* p0 = in0 + s0 * ld0;
      for (int c = lane; c < E0; c += 32) dst[c] = __ldg(p0 + c);
      if (E1 > 0) {
        long long s1 = idx1 ? idx1[row] : row;
        const float* p1 = in1 + s1 * ld1;
        for (int c = lane; c < E1; c += 32) dst[E0 + c] = __ldg(p1 + c);
      }
    } else {
      for (int c = lane; c < E; c += 32) dst[c] = 0.f;
    }
  }
  __syncthreads();

  float* cur = buf0;
  float* nxt = buf1;
  int Kd = E;
  for (int l = 0; l < d.n_layers; ++l) {
    const int H = d.out_dim[l];
    const float* __restrict__ W = d.W[l];
    const float* __restrict__ bias = d.b[l];
    const bool last = (l == d.n_layers - 1);
    if (H >= 32 && w_vec_ok && (Kd % 4 == 0)) {
      // Wide layer.  Thread c owns output column c for all TM rows.  W is streamed through shared memory in
      // [256 columns x 32 k] tiles with cp.async (coalesced 128-byte row segments, double buffered, rows padded to 36
      // floats so that the per-thread float4 reads are conflict-free); activations are shared-memory broadcasts.
      // (v1 let every thread walk its own W row in global memory: 32 different sectors per load, 34 us at B = 512.)
      const int n_kc = (Kd + MLP_KC - 1) / MLP_KC;
      for (int c0 = 0; c0 < H; c0 += MLP_THREADS) {
        const int c = c0 + tid;
        float acc[TM];
        const float b0 = (bias && c < H) ? __ldg(bias + c) : 0.f;
#pragma unroll
        for (int r = 0; r < TM; ++r) acc[r] = b0;
        auto stage = [&](int kc, int buf) {
          float* dst = wtile + (size_t)buf * MLP_THREADS * MLP_WS;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const int idx = tid + j * MLP_THREADS;
            const int rr = idx >> 3, ch = idx & 7;              // 8 x 16-byte chunks per 128-byte row segment
            const int col = c0 + rr, k = kc * MLP_KC + ch * 4;
            float* d = dst + (size_t)rr * MLP_WS + ch * 4;
            if (col < H && k < Kd) {
              const unsigned sa = (unsigned)__cvta_generic_to_shared(d);
              asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(sa), "l"(W + (size_t)col * Kd + k) : "memory");
            } else {
              *reinterpret_cast<float4*>(d) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
          asm volatile("cp.async.commit_group;\n" ::: "memory");
        };
#pragma unroll
        for (int s0 = 0; s0 < MLP_NSTG - 1; ++s0) {
          if (s0 < n_kc) stage(s0, s0);
          else asm volatile("cp.async.commit_group;\n" ::: "memory");      // empty group: keeps the count uniform
        }
        for (int kc = 0; kc < n_kc; ++kc) {
          if (kc + MLP_NSTG - 1 < n_kc) stage(kc + MLP_NSTG - 1, (kc + MLP_NSTG - 1) % MLP_NSTG);
          else asm volatile("cp.async.commit_group;\n" ::: "memory");
          asm volatile("cp.async.wait_group %0;\n" ::"n"(MLP_NSTG - 1) : "memory");      // tile kc has landed
          __syncthreads();
          const float* wt = wtile + (size_t)(kc % MLP_NSTG) * MLP_THREADS * MLP_WS + (size_t)tid * MLP_WS;
          const int kbase = kc * MLP_KC;
          const int kn = min(MLP_KC, Kd - kbase);
#pragma unroll 4
          for (int k = 0; k < kn; k += 4) {
            const float4 w = *reinterpret_cast<const float4*>(wt + k);
#pragma unroll
            for (int r = 0; r < TM; ++r) {
              const float4 a = *reinterpret_cast<const float4*>(cur + (size_t)r * stride + kbase + k);
              acc[r] = fmaf(a.x, w.x, acc[r]);
              acc[r] = fmaf(a.y, w.y, acc[r]);
              acc[r] = fmaf(a.z, w.z, acc[r]);
              acc[r] = fmaf(a.w, w.w, acc[r]);
            }
          }
          __syncthreads();                                      // the tile is free for the stage after next
        }
        if (c < H) {
#pragma unroll
          for (int r = 0; r < TM; ++r) {
            if (last) {
              if (row0 + r < B) out[(row0 + r) * ldo + c] = acc[r];
            } else {
              nxt[(size_t)r * stride + c] = fmaxf(acc[r], 0.f);
            }
          }
        }
      }
    } else if (H >= 32) {
      // wide layer, unaligned weights: thread-per-output-column straight from global memory
      for (int c = tid; c < H; c += MLP_THREADS) {
        float acc[TM];
        const float b0 = bias ? __ldg(bias + c) : 0.f;
#pragma unroll
        for (int r = 0; r < TM; ++r) acc[r] = b0;
        const float* wrow = W + (size_t)c * Kd;
        for (int k = 0; k < Kd; ++k) {
          const float w = __ldg(wrow + k);
#pragma unroll
          for (int r = 0; r < TM; ++r) acc[r] = fmaf(cur[(size_t)r * stride + k], w, acc[r]);
        }
#pragma unroll
        for (int r = 0; r < TM; ++r) {
          float v = last ? acc[r] : fmaxf(acc[r], 0.f);
          if (last) {
            if (row0 + r < B) out[(row0 + r) * ldo + c] = v;
          } else {
            nxt[(size_t)r * stride + c] = v;
          }
        }
      }
    } else {
      // narrow layer (the score head, H = 1): one warp per (row, column) dot product
      for (int p = warp; p < TM * H; p += MLP_THREADS / 32) {
        const int r = p / H, c = p % H;
        const float* wrow = W + (size_t)c * Kd;
        const float* a = cur + (size_t)r * stride;
        float s = 0.f;
        for (int k = lane; k < Kd; k += 32) s = fmaf(a[k], __ldg(wrow + k), s);
        s = warp_sum(s);
        if (lane == 0) {
          s += bias ? __ldg(bias + c) : 0.f;
          if (last) {
            if (row0 + r < B) out[(row0 + r) * ldo + c] = s;
          } else {
            nxt[(size_t)r * stride + c] = fmaxf(s, 0.f);
          }
        }
      }
    }
    __syncthreads();
    float* t = cur; cur = nxt; nxt = t;
    Kd = H;
  }
}

// GraphNCF(use_dot_product=True): out[b] = <in0[idx0[b]], in1[idx1[b]]>   (gnn_ncf.py:365)
__global__ void rowdot_kernel(const float* __restrict__ in0, long long ld0, const int64_t* __restrict__ idx0,
                              const float* __restrict__ in1, long long ld1, const int64_t* __restrict__ idx1, int E,
                              long long B, float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B) return;
  const float* a = in0 + (idx0 ? idx0[row] : row) * ld0;
  const float* b = in1 + (idx1 ? idx1[row] : row) * ld1;
  float s = 0.f;
  for (int k = lane; k < E; k += 32) s = fmaf(__ldg(a + k), __ldg(b + k), s);
  s = warp_sum(s);
  if (lane == 0) out[row] = s;
}

}  // namespace b200rec

using namespace b200rec;

extern "C" int b200rec_mlp_tower(const float* in0, int64_t ld0, const int64_t* idx0, int E0, const float* in1, int64_t ld1,
                                 const int64_t* idx1, int E1, int64_t B, const b200rec_mlp_t* mlp, float* out, int64_t ldo,
                                 b200rec_stream_t stream) {
  if (!mlp || mlp->n_layers < 1 || mlp->n_layers > B200REC_MLP_MAX_LAYERS || E0 <= 0 || E1 < 0 || !in0 || (E1 > 0 && !in1) || !out)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "mlp_tower: bad argument");
  if (B == 0) return B200REC_OK;
  int maxw = E0 + E1;
  bool vec_ok = true;
  for (int l = 0; l < mlp->n_layers; ++l) {
    if (!mlp->W[l] || mlp->out_dim[l] <= 0) return b200rec_fail(B200REC_ERR_BAD_ARG, "mlp_tower: bad layer");
    if (l + 1 < mlp->n_layers && mlp->out_dim[l] > maxw) maxw = mlp->out_dim[l];
    if ((uintptr_t)mlp->W[l] % 16 != 0) vec_ok = false;
  }
  if (ldo < mlp->out_dim[mlp->n_layers - 1]) return b200rec_fail(B200REC_ERR_BAD_ARG, "mlp_tower: ldo too small");
  const int stride = (maxw + 3) & ~3;
  cudaStream_t st = (cudaStream_t)stream;
  const int sms = b200rec_num_sms();
  // small batches: fewer rows per CTA so that more SMs take part
  const bool small = B < (long long)16 * sms * 2;
  // a batch that 4-row CTAs still fit into one wave (512 pairs -> 128 CTAs): the tower is a latency chain per CTA, more and shorter
  // chains finish sooner
  const bool tiny = B <= (long long)4 * sms;
  const int TM = tiny ? 4 : (small ? 8 : 16);
  size_t smem = ((size_t)2 * TM * stride + (size_t)(small ? 4 : 2) * MLP_THREADS * MLP_WS) * sizeof(float);
  if (smem > 200 * 1024) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "mlp_tower: layer too wide for shared memory");
  long long grid = (B + TM - 1) / TM;
  if (grid > INT32_MAX) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "mlp_tower: batch too large");
  if (tiny) {
    B200REC_CUDA(cudaFuncSetAttribute(mlp_tower_kernel<4, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    mlp_tower_kernel<4, 4><<<(unsigned)grid, MLP_THREADS, smem, st>>>(in0, ld0, idx0, E0, in1, ld1, idx1, E1, B, *mlp, out, ldo,
                                                                  stride, vec_ok);
  } else if (small) {
    B200REC_CUDA(cudaFuncSetAttribute(mlp_tower_kernel<8, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    mlp_tower_kernel<8, 4><<<(unsigned)grid, MLP_THREADS, smem, st>>>(in0, ld0, idx0, E0, in1, ld1, idx1, E1, B, *mlp, out, ldo,
                                                                  stride, vec_ok);
  } else {
    B200REC_CUDA(cudaFuncSetAttribute(mlp_tower_kernel<16, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    mlp_tower_kernel<16, 2><<<(unsigned)grid, MLP_THREADS, smem, st>>>(in0, ld0, idx0, E0, in1, ld1, idx1, E1, B, *mlp, out, ldo,
                                                                   stride, vec_ok);
  }
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_rowdot(const float* in0, int64_t ld0, const int64_t* idx0, const float* in1, int64_t ld1,
                              const int64_t* idx1, int E, int64_t B, float* out, b200rec_stream_t stream) {
  if (!in0 || !in1 || !out || E <= 0) return b200rec_fail(B200REC_ERR_BAD_ARG, "rowdot: bad argument");
  if (B == 0) return B200REC_OK;
  long long grid = (B + 7) / 8;
  rowdot_kernel<<<(unsigned)grid, 256, 0, (cudaStream_t)stream>>>(in0, ld0, idx0, in1, ld1, idx1, E, B, out);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}
