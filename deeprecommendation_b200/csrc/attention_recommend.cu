// K8 — AttentionNCF whole-catalogue recommendation: attention pooling over ONE shared rated list per user.
//
// The reference's serving call (src/webapp/backend.py:78-121) scores every catalogue item b for a user whose rated list
// {(i, um_i)} is the same for all candidates.  In the inference algebra of attention_ncf.py:136-224 (see K2):
//
//   s_bi   = a2 · ReLU(Pc[b] + Pr[i]) + a20        (MODE_NET)   or   <Pc[b], Pr[i]>   (MODE_DOT: cosine / att_dense=None)
//   α_bi   = softmax_i(s_b·) over the entries with um_i != 0    (exact 0.0 = "unrated", :158,192; nothing rated -> α = 0, :208-209)
//   h1[b]  = ReLU(Ai[b] + Σ_i α_bi·um_i·Q'[i])
//
// where the user-embedding half of the MLP's first Linear is folded into the pooled table (item first, :219):
//   W1 = [W1e | W1u],  Ai = Ec·W1eᵀ + b1 + W1u·b_U,  Q' = Q·W1uᵀ  — no per-pair (U x H1) GEMM is left, the pooling runs in H1 space.
//
// One CTA = (user, tile of 64 candidates).  The candidates' Pc rows are staged once, h-major; the user's list streams through
// shared memory 32 entries at a time (Pr rows h-major, Q' rows as they are).  Per chunk:
//   scores   thread = 4 candidates x 2 entries, ~3·H FP32 operations per (candidate, entry) on the FP32 pipes;
//   softmax  online per candidate (running max / denominator, rescale), 4 threads per candidate;
//   pooling  thread = CPT candidates x 8 columns of H1, accumulators in registers for the whole list.
// Per (user, candidate) pair nothing touches HBM except the h1 row it writes.  No atomics: results are bit-identical run to run.
#include <math.h>

#include "common.cuh"

namespace b200rec {

constexpr int AR_TB = 64;          // candidates per CTA
constexpr int AR_RC = 32;          // list entries per shared-memory chunk
constexpr int AR_THREADS = 256;
constexpr int AR_SS = 72;          // row stride of the (entry, candidate) score tile: 16-byte rows, conflict-free softmax reads
constexpr int AR_HMAX = 256;       // largest score width H
enum { AR_NET = 0, AR_DOT = 1 };

struct ArParams {
  const float* Pc; long long ld_pc;     // (nI, H) candidate score table
  const float* Pr; long long ld_pr;     // (nI, H) rated score table
  const float* Ai; long long ld_ai;     // (nI, H1P)
  const float* Qp; long long ld_q;      // (nI, H1P)
  const float* a2; const float* a20;    // MODE_NET: (H) and a device scalar (or null)
  const long long* list_ptr; const int* list_item; const float* list_val;
  const long long* users;
  int nI, H;
  float* out; long long ld_out;         // row (user slot u, candidate b) = u·nI + b, H1P columns
};

static size_t ar_smem_bytes(int H, int H1P) {
  return (size_t)(H * AR_TB + H * AR_RC + AR_RC * H1P + AR_RC * AR_SS + 2 * AR_TB + AR_RC + H) * 4;
}

template <int MODE, int H1P>
__global__ void __launch_bounds__(AR_THREADS, 2)
attention_recommend_kernel(const ArParams p) {
  constexpr int TH = H1P / 8;                       // threads across the H1 columns (8 columns each)
  constexpr int CPT = AR_TB * TH / AR_THREADS;      // candidates per pooling thread
  static_assert(CPT >= 1 && AR_TB % CPT == 0, "H1P in {32, 64, 128, 256}");
  extern __shared__ __align__(16) float ar_smem[];
  const int H = p.H;
  float* sPc = ar_smem;                       // [H][AR_TB]
  float* sPr = sPc + H * AR_TB;               // [H][AR_RC]
  float* sQ = sPr + H * AR_RC;                // [AR_RC][H1P]
  float* sS = sQ + AR_RC * H1P;               // [AR_RC][AR_SS]  scores, then pooling weights α·um (unnormalised)
  float* sScale = sS + AR_RC * AR_SS;         // [AR_TB]  rescale of the pooled accumulator for this chunk
  float* sInv = sScale + AR_TB;               // [AR_TB]  1 / softmax denominator
  float* sVal = sInv + AR_TB;                 // [AR_RC]
  float* sA2 = sVal + AR_RC;                  // [H]

  const int tid = threadIdx.x;
  const int b0 = blockIdx.x * AR_TB;
  const long long urow = __ldg(p.users + blockIdx.y);
  const long long e_begin = __ldg(p.list_ptr + urow), e_end = __ldg(p.list_ptr + urow + 1);
  const float a20 = (MODE == AR_NET && p.a20 != nullptr) ? __ldg(p.a20) : 0.f;
  const int H4 = H >> 2;

  // candidate tile, h-major (rows past the catalogue repeat its last row and are never stored)
  for (int idx = tid; idx < AR_TB * H4; idx += AR_THREADS) {
    const int r = idx % AR_TB, h = (idx / AR_TB) * 4;
    const float4 v = ld4(p.Pc + (long long)min(b0 + r, p.nI - 1) * p.ld_pc + h);
    sPc[(h + 0) * AR_TB + r] = v.x; sPc[(h + 1) * AR_TB + r] = v.y;
    sPc[(h + 2) * AR_TB + r] = v.z; sPc[(h + 3) * AR_TB + r] = v.w;
  }
  if (MODE == AR_NET)
    for (int h = tid; h < H; h += AR_THREADS) sA2[h] = __ldg(p.a2 + h);

  // score thread: candidates 4 ci .. 4 ci + 3, entries 2 rj, 2 rj + 1
  const int ci = tid & 15, rj = tid >> 4;
  // softmax thread: candidate sb, entries qq + 4 e
  const int sb = tid >> 2, qq = tid & 3;
  float m_run = -INFINITY, l_run = 0.f;
  // pooling thread: candidates cg·CPT .. + CPT, columns 8 tc .. 8 tc + 7
  const int tc = tid % TH, cg = tid / TH;
  float acc[CPT][8];
#pragma unroll
  for (int c = 0; c < CPT; ++c)
#pragma unroll
    for (int e = 0; e < 8; ++e) acc[c][e] = 0.f;

  for (long long c0 = e_begin; c0 < e_end; c0 += AR_RC) {
    const int cnt = (int)min((long long)AR_RC, e_end - c0);
    __syncthreads();                                              // the previous chunk's pooling is done with sQ / sS / sVal
    // ---- stage the chunk: Pr rows h-major, Q' rows, centred ratings (entries past `cnt`: zero rows, um = 0) ----
    for (int idx = tid; idx < AR_RC * H4; idx += AR_THREADS) {
      const int j = idx % AR_RC, h = (idx / AR_RC) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j < cnt) v = ld4(p.Pr + (long long)__ldg(p.list_item + c0 + j) * p.ld_pr + h);
      sPr[(h + 0) * AR_RC + j] = v.x; sPr[(h + 1) * AR_RC + j] = v.y;
      sPr[(h + 2) * AR_RC + j] = v.z; sPr[(h + 3) * AR_RC + j] = v.w;
    }
    for (int idx = tid; idx < AR_RC * (H1P / 4); idx += AR_THREADS) {
      const int j = idx / (H1P / 4), c = (idx % (H1P / 4)) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j < cnt) v = ld4(p.Qp + (long long)__ldg(p.list_item + c0 + j) * p.ld_q + c);
      st4(sQ + j * H1P + c, v);
    }
    if (tid < AR_RC) sVal[tid] = tid < cnt ? __ldg(p.list_val + c0 + tid) : 0.f;
    __syncthreads();

    // ---- scores of the (64 candidates x 32 entries) tile ----
    {
      float s[4][2];
#pragma unroll
      for (int q = 0; q < 4; ++q) { s[q][0] = 0.f; s[q][1] = 0.f; }
      const float* pc = sPc + 4 * ci;
      const float* pr = sPr + 2 * rj;
#pragma unroll 4
      for (int h = 0; h < H; ++h) {
        const float4 a = *reinterpret_cast<const float4*>(pc + h * AR_TB);
        const float2 r = *reinterpret_cast<const float2*>(pr + h * AR_RC);
        const float av[4] = {a.x, a.y, a.z, a.w};
        if (MODE == AR_NET) {
          const float w = sA2[h];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            s[q][0] = fmaf(w, fmaxf(av[q] + r.x, 0.f), s[q][0]);
            s[q][1] = fmaf(w, fmaxf(av[q] + r.y, 0.f), s[q][1]);
          }
        } else {
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            s[q][0] = fmaf(av[q], r.x, s[q][0]);
            s[q][1] = fmaf(av[q], r.y, s[q][1]);
          }
        }
      }
#pragma unroll
      for (int t = 0; t < 2; ++t)
        *reinterpret_cast<float4*>(sS + (2 * rj + t) * AR_SS + 4 * ci) = make_float4(s[0][t] + a20, s[1][t] + a20, s[2][t] + a20, s[3][t] + a20);
    }
    __syncthreads();

    // ---- online softmax: 4 threads per candidate, 8 entries each ----
    // __expf (ex2.approx, ~2 ulp) for the rescale and the weights, deliberately, as in K2 (csrc/attention_pool.cu): the error it adds to
    // α is far below the fp32 1e-5 budget of the scores (parity against `forward` is measured in tools/attention_recommend_bench.py).
    {
      float sv[8], mx = -INFINITY;
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int j = qq + 4 * e;
        const float v = sVal[j] != 0.f ? sS[j * AR_SS + sb] : -INFINITY;     // zero-centred entries are "unrated"
        sv[e] = v;
        mx = fmaxf(mx, v);
      }
      mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 1));
      mx = fmaxf(mx, __shfl_xor_sync(FULL, mx, 2));
      const float m_new = fmaxf(m_run, mx);
      float scale = 1.f;
      if (m_new != -INFINITY) {
        scale = __expf(m_run - m_new);                                        // m_run == -inf -> 0
        float ps = 0.f;
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const int j = qq + 4 * e;
          const float pj = sv[e] == -INFINITY ? 0.f : __expf(sv[e] - m_new);
          ps += pj;
          sS[j * AR_SS + sb] = pj * sVal[j];
        }
        ps += __shfl_xor_sync(FULL, ps, 1);
        ps += __shfl_xor_sync(FULL, ps, 2);
        l_run = l_run * scale + ps;
        m_run = m_new;
      } else {
#pragma unroll
        for (int e = 0; e < 8; ++e) sS[(qq + 4 * e) * AR_SS + sb] = 0.f;
      }
      if (qq == 0) sScale[sb] = scale;
    }
    __syncthreads();

    // ---- pooling in H1 space: acc[c][:] = acc[c][:]·scale + Σ_j w_cj · Q'[j][:] ----
    {
#pragma unroll
      for (int c = 0; c < CPT; ++c) {
        const float sc = sScale[cg * CPT + c];
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[c][e] *= sc;
      }
      const float* wq = sS + cg * CPT;
      const float* qq8 = sQ + tc * 8;
#pragma unroll 2
      for (int j = 0; j < cnt; ++j) {
        float w[CPT];
        if constexpr (CPT % 4 == 0) {
#pragma unroll
          for (int c = 0; c < CPT; c += 4) {
            const float4 t = *reinterpret_cast<const float4*>(wq + j * AR_SS + c);
            w[c] = t.x; w[c + 1] = t.y; w[c + 2] = t.z; w[c + 3] = t.w;
          }
        } else {
#pragma unroll
          for (int c = 0; c < CPT; ++c) w[c] = wq[j * AR_SS + c];
        }
        const float4 q0 = *reinterpret_cast<const float4*>(qq8 + j * H1P);
        const float4 q1 = *reinterpret_cast<const float4*>(qq8 + j * H1P + 4);
        const float qv[8] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w};
#pragma unroll
        for (int c = 0; c < CPT; ++c)
#pragma unroll
          for (int e = 0; e < 8; ++e) acc[c][e] = fmaf(w[c], qv[e], acc[c][e]);
      }
    }
  }

  // ---- h1 = ReLU(Ai + pooled / denominator) ----
  if (qq == 0) sInv[sb] = l_run > 0.f ? 1.f / l_run : 0.f;                    // nothing rated -> α = 0 -> user_emb = b_U (:208-209)
  __syncthreads();
#pragma unroll
  for (int c = 0; c < CPT; ++c) {
    const int bl = cg * CPT + c, b = b0 + bl;
    if (b >= p.nI) continue;
    const float inv = sInv[bl];
    const float* ai = p.Ai + (long long)b * p.ld_ai + tc * 8;
    const float4 x0 = ld4(ai), x1 = ld4(ai + 4);
    float* o = p.out + ((long long)blockIdx.y * p.nI + b) * p.ld_out + tc * 8;
    st4(o, make_float4(fmaxf(fmaf(acc[c][0], inv, x0.x), 0.f), fmaxf(fmaf(acc[c][1], inv, x0.y), 0.f),
                       fmaxf(fmaf(acc[c][2], inv, x0.z), 0.f), fmaxf(fmaf(acc[c][3], inv, x0.w), 0.f)));
    st4(o + 4, make_float4(fmaxf(fmaf(acc[c][4], inv, x1.x), 0.f), fmaxf(fmaf(acc[c][5], inv, x1.y), 0.f),
                           fmaxf(fmaf(acc[c][6], inv, x1.z), 0.f), fmaxf(fmaf(acc[c][7], inv, x1.w), 0.f)));
  }
}

template <int MODE, int H1P>
static int ar_launch(const ArParams& p, dim3 grid, cudaStream_t st) {
  static B200recSmemOptIn opted;
  B200REC_CUDA(b200rec_opt_in_smem(opted, attention_recommend_kernel<MODE, H1P>, (int)ar_smem_bytes(AR_HMAX, H1P)));
  attention_recommend_kernel<MODE, H1P><<<grid, AR_THREADS, ar_smem_bytes(p.H, H1P), st>>>(p);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

template <int MODE>
static int ar_dispatch(const ArParams& p, int H1P, dim3 grid, cudaStream_t st) {
  switch (H1P) {
    case 32: return ar_launch<MODE, 32>(p, grid, st);
    case 64: return ar_launch<MODE, 64>(p, grid, st);
    case 128: return ar_launch<MODE, 128>(p, grid, st);
    case 256: return ar_launch<MODE, 256>(p, grid, st);
  }
  return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_recommend: H1P must be 32, 64, 128 or 256");
}

}  // namespace b200rec

using namespace b200rec;

extern "C" size_t b200rec_attention_recommend_workspace(int64_t n_users, int64_t n_items, int H1P) {
  if (n_users <= 0 || n_items <= 0 || H1P <= 0) return 0;
  return (size_t)n_users * (size_t)n_items * (size_t)H1P * sizeof(float);
}

extern "C" int b200rec_attention_recommend(const float* Pc, int64_t ld_pc, const float* Pr, int64_t ld_pr, int H, int mode, const float* a2,
                                           const float* a20, const float* Ai, int64_t ld_ai, const float* Qp, int64_t ld_q, int H1P,
                                           int64_t n_items, const int64_t* list_ptr, const int32_t* list_item, const float* list_val,
                                           const int64_t* users, int64_t n_users, float* h1, int64_t ld_h1, b200rec_stream_t stream) {
  if (n_users < 0 || n_items < 0) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_recommend: negative size");
  if (n_users == 0 || n_items == 0) return B200REC_OK;
  if (!Pc || !Pr || !Ai || !Qp || !list_ptr || !list_item || !list_val || !users || !h1)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_recommend: null operand");
  if (mode != B200REC_ATT_NET && mode != B200REC_ATT_DOT) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_recommend: bad mode");
  if (mode == B200REC_ATT_NET && !a2) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_recommend: mode NET needs a2");
  if (H <= 0 || (H & 3) || H > AR_HMAX) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_recommend: H must be a multiple of 4, <= 256");
  if (H1P != 32 && H1P != 64 && H1P != 128 && H1P != 256)
    return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_recommend: H1P must be 32, 64, 128 or 256 (zero-pad H1)");
  if (ld_pc < H || ld_pr < H || ld_ai < H1P || ld_q < H1P || ld_h1 < H1P || ((ld_pc | ld_pr | ld_ai | ld_q | ld_h1) & 3))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_recommend: leading dimensions must cover the rows and be multiples of 4");
  if (((uintptr_t)Pc | (uintptr_t)Pr | (uintptr_t)Ai | (uintptr_t)Qp | (uintptr_t)h1) & 15)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_recommend: tables and h1 must be 16-byte aligned");
  if (n_items > INT32_MAX / 2 || n_users > 65535) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_recommend: n_items < 2^30 and n_users <= 65535 per call");
  ArParams p;
  p.Pc = Pc; p.ld_pc = ld_pc; p.Pr = Pr; p.ld_pr = ld_pr; p.Ai = Ai; p.ld_ai = ld_ai; p.Qp = Qp; p.ld_q = ld_q;
  p.a2 = a2; p.a20 = a20;
  p.list_ptr = reinterpret_cast<const long long*>(list_ptr); p.list_item = list_item; p.list_val = list_val;
  p.users = reinterpret_cast<const long long*>(users);
  p.nI = (int)n_items; p.H = H; p.out = h1; p.ld_out = ld_h1;
  const dim3 grid((unsigned)((n_items + AR_TB - 1) / AR_TB), (unsigned)n_users);
  cudaStream_t st = (cudaStream_t)stream;
  return mode == B200REC_ATT_NET ? ar_dispatch<AR_NET>(p, H1P, grid, st) : ar_dispatch<AR_DOT>(p, H1P, grid, st);
}
