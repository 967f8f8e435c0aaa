// K2 — AttentionNCF dynamic user profile: ragged item-item attention + segmented softmax + weighted pooling.
//
// Replaces attention_ncf.py:154-216 of the reference (the (B*I, E) repeat_interleave/repeat materialisation, the
// boolean-mask gather, AttentionNet on the valid pairs, the -inf filled (B, I) softmax, `scores * user_matrix`,
// the (B,I)x(I,F) pooling GEMM and the user-embedding Linear) by ONE memory-bound kernel over the non-zeros of
// `user_matrix`, using the exact algebraic factorisation (SURVEY.md §8a-3 / §8d):
//
//   AttentionNet.0 = [A1c | A1r]           P_c = Ec·A1cᵀ + a1   (B, H)      P_r = Er·A1rᵀ   (I, H)
//   s_bi = a2 · ReLU(P_c[b] + P_r[i]) + a20                      (score; MODE_NET)
//   Q    = R · W_Uᵀ                                              (I, U)   pooling in embedding space
//   user_emb[b] = Σ_i softmax_i(s_b·)·um_bi · Q[i] + b_U
//
// (cosine variant / att_dense=None variant: s_bi = <P_c[b], P_r[i]>, MODE_DOT, with the host passing
// normalised embeddings resp. 4-wide [sc,1,0,0]/[1,sr,0,0] rows.)
//
// One CTA owns one candidate row b and each of its 8 warps a contiguous slice of the row (round 1 used one warp per
// row: 4.6 % warps active, 560 us at B=512 — profiles/r01).  Per warp, non-zeros are consumed 32 at a time: for each of the 32 the warp loads the
// P_r row with one coalesced 128-bit load per lane, every lane forms its partial dot product, and a 31-shuffle
// butterfly reduce-scatter leaves lane j with the full score of non-zero j (1 shuffle per score instead of 5).
// The softmax is online (running max / denominator, FlashAttention-style rescale), so each segment is read once;
// pooling re-walks the 32 non-zeros with one coalesced Q-row load each; the per-warp (max, denominator, pooled vector)
// states are merged through shared memory at the end.  Nothing of size (B, I, *) exists.
// Two front-ends feed the same core: a CSR reader (ragged-native entry) and a dense-row scanner that compacts
// the reference's dense (B, I) `user_matrix` on the fly through a per-warp shared-memory queue (drop-in entry;
// exact 0.0 means "unrated", attention_ncf.py:158,192).
#include <math.h>

#include <algorithm>

#include "common.cuh"

// Compiled twice: as is (the scoring path) and, through csrc/attention_pool_drop.cu, with B200REC_ATT_DROPOUT defined — the training-mode
// variant that applies AttentionNet's inner Dropout (attention_ncf.py:112-117) to ReLU(Pc + Pr) with a regenerable Philox mask.  The second copy
// lives in its own namespace and exports ONE entry point (b200rec_attention_pool_dropout), so the scoring kernels stay byte-identical.
namespace b200rec {
#ifdef B200REC_ATT_DROPOUT
namespace attdrop {
#endif

static int g_att_path = 0;       // b200rec_attention_pool_set_path: 0 auto, 1 register-staged gathers, 2 TMA-staged gathers
constexpr int ATT_WARPS = 8;      // one CTA per candidate row; the row's non-zeros are split over the warps
enum { MODE_NET = 0, MODE_DOT = 1 };

struct AttParams {
  const float* Pc;     // (B, H) fp32, bias a1 folded in
  const void* Pr;      // (I, H) table
  const void* Q;       // (I, U) table
  const float* a2;     // (H) fp32 (MODE_NET)
  const float* a20;    // device scalar (MODE_NET) or null
  const float* bU;     // (U) or null
  float* out;          // (B, U)
  long long ldo;
  float* att;          // (B, I) or null; must be zero-filled by the caller
  int B, I, H, U;
  // training-mode extras (attention_ncf.py:185-203)
  const float* Ec;     // (B, E) or null: candidate embeddings for the isclose() target mask
  const float* Er;     // (I, E)
  int E;
  float atol, rtol;
  int drop_zero_scores;   // message_dropout is not None: scores == 0.0 -> -inf (:189)
  float score_scale;      // message dropout: kept scores are scaled by 1/(1-p) (:187)
  long long ldPr, ldQ, ldPc;
  unsigned drop_key, drop_thr16;   // inner dropout (B200REC_ATT_DROPOUT build only): Philox key, keep threshold on 16 bits
  float drop_scale;
  const unsigned long long* drop_seed_dev;   // optional: the 64-bit seed lives in device memory (CUDA-graph replays draw a new one each time)
};


// ---- TMA / mbarrier helpers (bulk-copy row gathers of the warp-segment kernel) -----------------------------------
__device__ __forceinline__ uint32_t att_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void att_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(att_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void att_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(att_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void att_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "ATT_WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra ATT_DONE_%=;\n\t"
      "bra ATT_WAIT_%=;\n\t"
      "ATT_DONE_%=:\n\t}" ::"r"(att_smem_u32(bar)), "r"(parity) : "memory");
}
// 1-D bulk copy global -> shared; completion = transaction bytes on the mbarrier.  16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void att_bulk_g2s(void* dst_smem, const void* src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(att_smem_u32(dst_smem)),
               "l"(src), "r"(bytes), "r"(att_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void att_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// 4 consecutive table elements from SHARED memory as fp32
__device__ __forceinline__ float4 lds4(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 lds4(const __nv_bfloat16* p) {
  const uint2 r = *reinterpret_cast<const uint2*>(p);
  return make_float4(__uint_as_float(r.x << 16), __uint_as_float(r.x & 0xffff0000u), __uint_as_float(r.y << 16), __uint_as_float(r.y & 0xffff0000u));
}

template <int HV, int UV, int MODE, typename T>
struct RowCore {
  const AttParams& p;
  const int lane;
  const int b;
  float pc[HV][4], a2[HV][4];
  float acc[UV][4];
  float m, l, a20;
  unsigned dkey;          // Philox key of the inner dropout (dropout build)
  unsigned hcol[HV], ucol[UV];   // this lane's column vector of a Pr / Q row (float4 units, clamped to the last one in range)
  int ldPr, ldQ;

  __device__ RowCore(const AttParams& p_, int lane_, int b_) : p(p_), lane(lane_), b(b_) {
#pragma unroll
    for (int hv = 0; hv < HV; ++hv) {
      const int h = lane * 4 + hv * 128;
      float4 c = make_float4(0.f, 0.f, 0.f, 0.f), w = c;
      if (h < p.H) {
        c = ld4(p.Pc + (long long)b * p.ldPc + h);
        if (MODE == MODE_NET) w = ld4(p.a2 + h);
      }
      pc[hv][0] = c.x; pc[hv][1] = c.y; pc[hv][2] = c.z; pc[hv][3] = c.w;
      a2[hv][0] = w.x; a2[hv][1] = w.y; a2[hv][2] = w.z; a2[hv][3] = w.w;
    }
#pragma unroll
    for (int uv = 0; uv < UV; ++uv)
#pragma unroll
      for (int e = 0; e < 4; ++e) acc[uv][e] = 0.f;
    m = -INFINITY;
    l = 0.f;
    a20 = (MODE == MODE_NET && p.a20) ? __ldg(p.a20) : 0.f;
    ldPr = (int)p.ldPr; ldQ = (int)p.ldQ;
#pragma unroll
    for (int hv = 0; hv < HV; ++hv) hcol[hv] = (unsigned)min(lane * 4 + hv * 128, p.H - 4) >> 2;
#pragma unroll
    for (int uv = 0; uv < UV; ++uv) ucol[uv] = (unsigned)min(lane * 4 + uv * 128, p.U - 4) >> 2;
    dkey = p.drop_key;
#ifdef B200REC_ATT_DROPOUT
    if (p.drop_seed_dev != nullptr) {
      const unsigned long long sd = __ldg(p.drop_seed_dev);
      dkey = (unsigned)(sd ^ (sd >> 32));
    }
#endif
  }

  // scores of one batch (lane-partial dot products in v[0..31]) -> online-softmax state update; returns this lane's
  // pooling weight = attention numerator x centred rating (:212)
  __device__ __forceinline__ float softmax_update(float (&v)[32], int my_col, float my_val, int count) {
    // butterfly reduce-scatter: after the last step lane j holds sum over lanes of v[j]
#pragma unroll
    for (int k = 16; k >= 1; k >>= 1) {
      const bool up = (lane & k) != 0;
#pragma unroll
      for (int i = 0; i < k; ++i) {
        const float send = up ? v[i] : v[i + k];
        const float keep = up ? v[i + k] : v[i];
        v[i] = keep + __shfl_xor_sync(FULL, send, k);
      }
    }
    float s = (v[0] + a20) * p.score_scale;
    if (my_col < 0) s = -INFINITY;                    // beyond `count`, or an explicit zero in a CSR
    if (p.drop_zero_scores && s == 0.f) s = -INFINITY;
    if (p.Ec != nullptr) {     // training: mask rated items whose EMBEDDING is close to the candidate's (:199)
      unsigned masked = 0u;
      if (p.E <= 128 && (p.E & 3) == 0 && ((((uintptr_t)p.Ec | (uintptr_t)p.Er) & 15) == 0)) {
        // the usual shape (item_emb <= 128): a lane owns 4 consecutive embedding columns; the candidate's are read once per batch, the rated
        // rows as ONE 128-bit gather per pair, eight pairs in flight (the scalar loop below was 4x the cost of the whole pooling in train mode)
        const int e0 = min(lane * 4, p.E - 4);
        const bool mine = lane * 4 < p.E;
        const float4 x = ld4(p.Ec + (long long)b * p.E + e0);
        const unsigned fill = (unsigned)max(__shfl_sync(FULL, my_col, __ffs(__ballot_sync(FULL, my_col >= 0)) - 1), 0);
#pragma unroll 1
        for (int j0 = 0; j0 < count; j0 += 8) {
          float4 y[8];
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {
            const int c = __shfl_sync(FULL, my_col, (j0 + jj) & 31);
            y[jj] = ld4(p.Er + (long long)(c >= 0 ? (unsigned)c : fill) * p.E + e0);
          }
#pragma unroll
          for (int jj = 0; jj < 8; ++jj) {
            const bool ok = !mine || (fabsf(x.x - y[jj].x) <= p.atol + p.rtol * fabsf(y[jj].x) && fabsf(x.y - y[jj].y) <= p.atol + p.rtol * fabsf(y[jj].y) &&
                                      fabsf(x.z - y[jj].z) <= p.atol + p.rtol * fabsf(y[jj].z) && fabsf(x.w - y[jj].w) <= p.atol + p.rtol * fabsf(y[jj].w));
            const bool close = __all_sync(FULL, ok);
            const int c = __shfl_sync(FULL, my_col, (j0 + jj) & 31);
            if (close && j0 + jj < count && c >= 0) masked |= (1u << (j0 + jj));
          }
        }
      } else {
        for (int j = 0; j < count; ++j) {
          const int c = __shfl_sync(FULL, my_col, j);
          if (c < 0) continue;
          bool ok = true;
          for (int e = lane; e < p.E; e += 32) {
            const float x = __ldg(p.Ec + (long long)b * p.E + e), y = __ldg(p.Er + (long long)c * p.E + e);
            ok = ok && (fabsf(x - y) <= p.atol + p.rtol * fabsf(y));
          }
          if (__all_sync(FULL, ok)) masked |= (1u << j);
        }
      }
      if ((masked >> lane) & 1u) s = -INFINITY;
    }
    if (p.att != nullptr && my_col >= 0) p.att[(long long)b * p.I + my_col] = s;    // raw score; normalised in finish()

    const float m_new = fmaxf(m, warp_max(s));
    float pj = 0.f;
    if (m_new != -INFINITY) {
      const float scale = __expf(m - m_new);          // m == -inf -> 0
      pj = (s == -INFINITY) ? 0.f : __expf(s - m_new);
      l = l * scale + warp_sum(pj);
#pragma unroll
      for (int uv = 0; uv < UV; ++uv)
#pragma unroll
        for (int e = 0; e < 4; ++e) acc[uv][e] *= scale;
      m = m_new;
    }
    return pj * my_val;
  }

  // lane j holds non-zero j of this batch (col < 0 beyond `count`).
  // Round 2 (ncu source page: 67 instructions per (candidate, rated item) pair and lane, 63 % of them overhead — 64-bit address products per
  // gathered row, kernel parameters re-read from the constant bank, zero-fill and selects around predicated loads): every lane computes the row
  // offsets of ITS entry once per batch, in units of one 4-element vector (32 bits: tables below 2^34 elements, checked on the host), and the
  // inner loops broadcast that one word.  The gathers are unconditional: a lane without an entry (beyond `count`, or an explicit zero of a CSR)
  // points at the row of the batch's first valid entry — a row this candidate uses anyway, so no new inf / NaN can enter — its score is forced to
  // -inf and its pooling weight is 0.  Columns past H / U read the last in-range vector: Pc and a2 are zero there, and pooled lanes past U are
  // never stored.
  __device__ void batch(int my_col, float my_val, int count) {
    const T* __restrict__ Pr = reinterpret_cast<const T*>(p.Pr);
    const T* __restrict__ Q = reinterpret_cast<const T*>(p.Q);
    const unsigned valid = __ballot_sync(FULL, my_col >= 0);
    if (valid == 0u) return;                               // nothing rated in this batch: state unchanged
    const int c_fill = __shfl_sync(FULL, my_col, __ffs(valid) - 1);
    const unsigned row = (unsigned)(my_col >= 0 ? my_col : c_fill);
    const unsigned offPr = row * (unsigned)(ldPr >> 2), offQ = row * (unsigned)(ldQ >> 2);     // float4 / 4 x bf16 units
    float v[32];
    constexpr int LB = (HV == 1 && UV == 1) ? 16 : 8;     // row gathers in flight per warp
#pragma unroll
    for (int j0 = 0; j0 < 32; j0 += LB) {
      if (j0 < count) {
        float4 pr[LB][HV];
#pragma unroll
        for (int jj = 0; jj < LB; ++jj) {
          const unsigned o = __shfl_sync(FULL, offPr, j0 + jj);
#pragma unroll
          for (int hv = 0; hv < HV; ++hv) pr[jj][hv] = ld4(Pr + ((size_t)(o + hcol[hv]) << 2));
        }
#pragma unroll
        for (int jj = 0; jj < LB; ++jj) {
          float s = 0.f;
#ifdef B200REC_ATT_DROPOUT
          const int cdrop = __shfl_sync(FULL, my_col, j0 + jj);
#endif
#pragma unroll
          for (int hv = 0; hv < HV; ++hv) {
            const float r[4] = {pr[jj][hv].x, pr[jj][hv].y, pr[jj][hv].z, pr[jj][hv].w};
#ifdef B200REC_ATT_DROPOUT
            float dm[4] = {1.f, 1.f, 1.f, 1.f};
            if (MODE == MODE_NET && p.drop_thr16 < 65536u) att_dropout_mult(dkey, p.drop_thr16, p.drop_scale, b, cdrop, lane + 32 * hv, dm);
#endif
#pragma unroll
            for (int e = 0; e < 4; ++e) {
#ifdef B200REC_ATT_DROPOUT
              if (MODE == MODE_NET) s = fmaf(a2[hv][e] * dm[e], fmaxf(pc[hv][e] + r[e], 0.f), s);
#else
              if (MODE == MODE_NET) s = fmaf(a2[hv][e], fmaxf(pc[hv][e] + r[e], 0.f), s);
#endif
              else s = fmaf(pc[hv][e], r[e], s);
            }
          }
          v[j0 + jj] = s;
        }
      } else {
#pragma unroll
        for (int jj = 0; jj < LB; ++jj) v[j0 + jj] = 0.f;
      }
    }
    const float wgt = softmax_update(v, my_col, my_val, count);
#pragma unroll
    for (int j0 = 0; j0 < 32; j0 += LB) {
      if (j0 < count) {
        float4 q[LB][UV];
        float w[LB];
#pragma unroll
        for (int jj = 0; jj < LB; ++jj) {
          const unsigned o = __shfl_sync(FULL, offQ, j0 + jj);
          w[jj] = __shfl_sync(FULL, wgt, j0 + jj);
#pragma unroll
          for (int uv = 0; uv < UV; ++uv) q[jj][uv] = ld4(Q + ((size_t)(o + ucol[uv]) << 2));
        }
#pragma unroll
        for (int jj = 0; jj < LB; ++jj)
#pragma unroll
          for (int uv = 0; uv < UV; ++uv) {
            acc[uv][0] = fmaf(w[jj], q[jj][uv].x, acc[uv][0]);
            acc[uv][1] = fmaf(w[jj], q[jj][uv].y, acc[uv][1]);
            acc[uv][2] = fmaf(w[jj], q[jj][uv].z, acc[uv][2]);
            acc[uv][3] = fmaf(w[jj], q[jj][uv].w, acc[uv][3]);
          }
      }
    }
  }

  // The same batch with the 32 Pr rows and 32 Q rows already in shared memory (landed there by TMA bulk copies: one
  // memory latency per batch instead of four register-staged gather rounds).  HV == UV == 1 only; sPr / sQ rows are 128
  // elements apart; `valid` = ballot of (my_col >= 0): rows of invalid lanes were not copied and are never read.
  __device__ void batch_smem(int my_col, float my_val, int count, const T* sPr, const T* sQ, unsigned valid) {
    static_assert(HV == 1 && UV == 1, "shared-memory batches are for H, U <= 128");
    float v[32];
    const int h = lane * 4;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      float s = 0.f;
      if (((valid >> j) & 1u) && h < p.H) {
        const float4 r4 = lds4(sPr + j * 128 + h);
        const float r[4] = {r4.x, r4.y, r4.z, r4.w};
#ifdef B200REC_ATT_DROPOUT
        float dm[4] = {1.f, 1.f, 1.f, 1.f};
        if (MODE == MODE_NET && p.drop_thr16 < 65536u) att_dropout_mult(dkey, p.drop_thr16, p.drop_scale, b, __shfl_sync(FULL, my_col, j), lane, dm);
#endif
#pragma unroll
        for (int e = 0; e < 4; ++e) {
#ifdef B200REC_ATT_DROPOUT
          if (MODE == MODE_NET) s = fmaf(a2[0][e] * dm[e], fmaxf(pc[0][e] + r[e], 0.f), s);
#else
          if (MODE == MODE_NET) s = fmaf(a2[0][e], fmaxf(pc[0][e] + r[e], 0.f), s);
#endif
          else s = fmaf(pc[0][e], r[e], s);
        }
      }
      v[j] = s;
    }
    const float wgt = softmax_update(v, my_col, my_val, count);
    const int u = lane * 4;
#pragma unroll
    for (int j = 0; j < 32; ++j) {
      const float wj = __shfl_sync(FULL, wgt, j);
      if (((valid >> j) & 1u) && u < p.U) {
        const float4 q = lds4(sQ + j * 128 + u);
        acc[0][0] = fmaf(wj, q.x, acc[0][0]); acc[0][1] = fmaf(wj, q.y, acc[0][1]);
        acc[0][2] = fmaf(wj, q.z, acc[0][2]); acc[0][3] = fmaf(wj, q.w, acc[0][3]);
      }
    }
  }

  // ---- cross-warp merge (one CTA = one candidate row, every warp owns a slice of the row's non-zeros) ----------
  __device__ void export_state(float* s_m, float* s_l, float* s_acc, int warp) const {
    if (lane == 0) { s_m[warp] = m; s_l[warp] = l; }
#pragma unroll
    for (int uv = 0; uv < UV; ++uv)
      *reinterpret_cast<float4*>(s_acc + (size_t)warp * (UV * 128) + lane * 4 + uv * 128) =
          make_float4(acc[uv][0], acc[uv][1], acc[uv][2], acc[uv][3]);
  }
};

// after __syncthreads(): global running max / denominator of the row and the pooled output
template <int UV>
__device__ __forceinline__ void merge_and_write(const AttParams& p, int b, const float* s_m, const float* s_l, const float* s_acc,
                                                float& M, float& Lsum) {
  M = -INFINITY;
#pragma unroll
  for (int w = 0; w < ATT_WARPS; ++w) M = fmaxf(M, s_m[w]);
  float scale[ATT_WARPS];
  Lsum = 0.f;
#pragma unroll
  for (int w = 0; w < ATT_WARPS; ++w) {
    scale[w] = (s_m[w] == -INFINITY) ? 0.f : __expf(s_m[w] - M);
    Lsum += s_l[w] * scale[w];
  }
  const float inv = Lsum > 0.f ? 1.f / Lsum : 0.f;      // no valid rated item -> weights 0 -> user_emb = b_U (:208-209)
  for (int u = threadIdx.x; u < p.U; u += ATT_WARPS * 32) {
    float a = 0.f;
#pragma unroll
    for (int w = 0; w < ATT_WARPS; ++w) a = fmaf(s_acc[(size_t)w * (UV * 128) + u], scale[w], a);
    p.out[(long long)b * p.ldo + u] = fmaf(a, inv, p.bU ? __ldg(p.bU + u) : 0.f);
  }
}

__device__ __forceinline__ float normalise_score(float s, float M, float Lsum) {
  return (Lsum > 0.f && s != -INFINITY) ? __expf(s - M) / Lsum : 0.f;
}

// ---- ragged-native front-end: CSR of user_matrix ------------------------------------------------------------
template <int HV, int UV, int MODE, typename T>
__global__ void __launch_bounds__(ATT_WARPS * 32, (HV == 1 && UV == 1) ? 2 : 1)
attention_pool_csr_kernel(AttParams p, const int* __restrict__ row_ptr, const int* __restrict__ col,
                          const float* __restrict__ val, const int* __restrict__ row_nnz, long long padded_stride) {
  __shared__ float s_m[ATT_WARPS], s_l[ATT_WARPS];
  __shared__ __align__(16) float s_acc[ATT_WARPS * UV * 128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x;
  RowCore<HV, UV, MODE, T> core(p, lane, b);
  // either a true CSR (row_ptr) or the row-padded form written by um_compact_kernel (row b starts at b*stride)
  const long long start = row_nnz ? (long long)b * padded_stride : (long long)__ldg(row_ptr + b);
  const long long end = row_nnz ? start + __ldg(row_nnz + b) : (long long)__ldg(row_ptr + b + 1);
  const int blocks = (int)((end - start + 31) >> 5);
  const int bpw = (blocks + ATT_WARPS - 1) / ATT_WARPS;
  const long long my_start = start + (long long)warp * bpw * 32, my_end = min(end, my_start + (long long)bpw * 32);
  for (long long k0 = my_start; k0 < my_end; k0 += 32) {
    const long long k = k0 + lane;
    int c = -1;
    float v = 0.f;
    if (k < my_end) { c = __ldg(col + k); v = __ldg(val + k); }
    const bool valid = (k < my_end) && (v != 0.f);     // an explicit 0.0 in the CSR is "unrated", like the dense form
    core.batch(valid ? c : -1, valid ? v : 0.f, (int)min(32LL, my_end - k0));
  }
  core.export_state(s_m, s_l, s_acc, warp);
  __syncthreads();
  float M, Lsum;
  merge_and_write<UV>(p, b, s_m, s_l, s_acc, M, Lsum);
  if (p.att != nullptr) {
    for (long long k = my_start + lane; k < my_end; k += 32) {
      if (__ldg(val + k) != 0.f) {
        float* a = p.att + (long long)b * p.I + __ldg(col + k);
        *a = normalise_score(*a, M, Lsum);
      }
    }
  }
}

// ---- segment-parallel ragged kernel -------------------------------------------------------------------------
// Rows are heavy-tailed (config 2: mean ~550 non-zeros per candidate, max ~2.7k; a big catalogue: mean ~160), so neither a CTA
// per row (lasts as long as its longest row) nor a CTA per 512-non-zero segment (v3: 5 of 8 warps idle at a barrier on the typical
// short row — ncu on the HBM-regime shape: 15 resident warps per SM of which ~6 live, 0.375 of the HBM roofline) keeps the
// memory system busy.  Here the unit is ONE WARP per segment of <= ATT_WSEG non-zeros: a tiny kernel (or the tail of the
// compaction kernel) writes a dense work list of (row, segment) items — list positions come from an atomic counter, which only
// orders the list, never a value — and a persistent grid of warps strides over it.  Every resident warp is live, there is no
// block-level barrier and no shared memory; each item leaves a (max, denominator, pooled vector) partial, and the merge kernel
// combines a row's partials in segment order (bit-reproducible), adds b_U and normalises the attention weights.
constexpr int ATT_WSEG = 64;

// Round 2 — a two-ended list.  Config 2 has ~4,900 items for 2,368 resident warps: with one list 7 % of the warps took a third full-length item while
// the rest idled (ncu: issue slots 53 % busy on the active cycles, 23 % of the warp slots).  A row's last segment is SHORT when it holds <= 32 entries
// (one batch of gathers instead of two); short items are appended from the END of the list (counter[1]), everything else from the front
// (counter[0]), and the warps walk front-then-back: whatever spills into a last round is a single batch.  A partial lives in the slot of its item's
// list position; seg_base[b] is the first front slot of row b, tail_pos[b] the slot of its short last segment (or -1).
struct AttWork {
  int* counter;        // [0] = items at the front of the list, [1] = short items at its end
  int* tail_pos;       // (B): list position of the row's short last segment, -1 if it has none
  int* seg_base;       // (B): first partial slot of the row
  int2* items;         // (row, segment)
  float* partials;     // (n_items, U + 4): m, l, -, -, acc[U]
  int max_items;       // capacity of items / partials (a max_row_nnz hint that is not a true bound must not overrun them)
};

// segments of a row of `len` entries, and how many of them go to the front of the list (all but a short last one)
__device__ __forceinline__ int att_nseg(long long len) { return (int)((len + ATT_WSEG - 1) / ATT_WSEG); }
__device__ __forceinline__ int att_nfront(long long len) {
  const int rem = (int)(len % ATT_WSEG);
  return att_nseg(len) - ((rem >= 1 && rem <= 32) ? 1 : 0);
}
// one thread: reserve the row's list positions (front block + short tail), record them, write the tail item; returns the front base
__device__ __forceinline__ int att_reserve_row(const AttWork& w, int b, long long len) {
  const int n = att_nseg(len), nf = att_nfront(len);
  const int base = nf > 0 ? atomicAdd(w.counter, nf) : 0;
  w.seg_base[b] = base;
  int tail = -1;
  if (n > nf) {
    tail = w.max_items - 1 - atomicAdd(w.counter + 1, 1);
    if (tail >= 0) w.items[tail] = make_int2(b, n - 1);
  }
  w.tail_pos[b] = tail;
  return base;
}
// Both ends grow towards each other inside `max_items` slots; with a true bound on the number of items they never meet.  If a caller's hint was
// too small, front writes stop at the capacity (as before) and the counters are clamped by the readers (att_list_counts).
__device__ __forceinline__ void att_list_counts(const AttWork& w, int& front, int& back) {
  front = min(__ldg(w.counter), w.max_items);
  back = min(__ldg(w.counter + 1), w.max_items - front);
}

__device__ __forceinline__ void att_emit_items(const AttWork& w, int b, int len, int tid, int nthreads, int* s_base) {
  if (tid == 0) *s_base = att_reserve_row(w, b, len);
  __syncthreads();
  const int base = *s_base, nf = att_nfront(len);
  for (int j = tid; j < nf; j += nthreads)
    if (base + j < w.max_items) w.items[base + j] = make_int2(b, j);
}

__global__ void __launch_bounds__(128)
att_worklist_kernel(const int* __restrict__ row_ptr, int B, AttWork w) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int len = __ldg(row_ptr + b + 1) - __ldg(row_ptr + b);
  const int base = att_reserve_row(w, b, len), nf = att_nfront(len);
  for (int j = 0; j < nf; ++j)
    if (base + j < w.max_items) w.items[base + j] = make_int2(b, j);
}

template <int HV, int UV, int MODE, typename T>
__global__ void __launch_bounds__(ATT_WARPS * 32, (HV == 1 && UV == 1) ? 2 : 1)
attention_wseg_kernel(AttParams p, const int* __restrict__ row_ptr, const int* __restrict__ col, const float* __restrict__ val,
                      const int* __restrict__ row_nnz, long long padded_stride, AttWork w) {
  const int lane = threadIdx.x & 31;
  const int n_warps = gridDim.x * ATT_WARPS;
  int front, back;
  att_list_counts(w, front, back);
  for (int v = blockIdx.x * ATT_WARPS + (threadIdx.x >> 5); v < front + back; v += n_warps) {
    const int it = v < front ? v : w.max_items - 1 - (v - front);          // list position = partial slot
    const int2 item = __ldg(w.items + it);
    const int b = item.x, seg = item.y;
    const long long start = row_nnz ? (long long)b * padded_stride : (long long)__ldg(row_ptr + b);
    const long long end = row_nnz ? start + __ldg(row_nnz + b) : (long long)__ldg(row_ptr + b + 1);
    const long long seg_start = start + (long long)seg * ATT_WSEG;
    const long long seg_end = min(end, seg_start + ATT_WSEG);
    // index stream of the whole segment (<= 64 entries = two batches) is fetched up front: one latency instead of one per batch
    int c0 = -1, c1 = -1;
    float v0 = 0.f, v1 = 0.f;
    if (seg_start + lane < seg_end) { c0 = __ldg(col + seg_start + lane); v0 = __ldg(val + seg_start + lane); }
    if (seg_start + 32 + lane < seg_end) { c1 = __ldg(col + seg_start + 32 + lane); v1 = __ldg(val + seg_start + 32 + lane); }
    const int slot_idx = it;
    RowCore<HV, UV, MODE, T> core(p, lane, b);
    const int n0 = (int)min(32LL, seg_end - seg_start);
    core.batch(v0 != 0.f ? c0 : -1, v0, n0);                      // an explicit 0.0 is "unrated", like the dense form
    if (seg_start + 32 < seg_end) core.batch(v1 != 0.f ? c1 : -1, v1, (int)(seg_end - seg_start - 32));
    float* slot = w.partials + (long long)slot_idx * (p.U + 4);
    if (lane == 0) { slot[0] = core.m; slot[1] = core.l; }
#pragma unroll
    for (int uv = 0; uv < UV; ++uv) {
      const int u = lane * 4 + uv * 128;
      if (u < p.U) st4(slot + 4 + u, make_float4(core.acc[uv][0], core.acc[uv][1], core.acc[uv][2], core.acc[uv][3]));
    }
  }
}

// The same persistent warp-per-segment loop with the row gathers done by the TMA engine: every lane issues ONE 1-D bulk copy
// for "its" Pr row and one for its Q row (2 x 32 rows x 512 B = 32 KB per warp in flight, no registers held), the warp waits on
// its own mbarrier and then reads the rows from shared memory.  Bytes in flight per SM are bounded by shared memory (6 warps x
// 32 KB fp32, 12 x 16 KB bf16) instead of by registers (v4: 16 warps x 8 KB, and four dependent gather rounds per batch).
template <int MODE, typename T>
__global__ void __launch_bounds__(512, 1)
attention_wseg_tma_kernel(AttParams p, const int* __restrict__ row_ptr, const int* __restrict__ col, const float* __restrict__ val,
                          const int* __restrict__ row_nnz, long long padded_stride, AttWork w) {
  extern __shared__ __align__(128) unsigned char att_smem[];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, warps = blockDim.x >> 5;
  constexpr int ROW = 128 * (int)sizeof(T);                     // shared-memory pitch of one staged row
  T* sPr = reinterpret_cast<T*>(att_smem + (size_t)warp * 64 * ROW);
  T* sQ = sPr + 32 * 128;
  uint64_t* bar = reinterpret_cast<uint64_t*>(att_smem + (size_t)warps * 64 * ROW) + warp;
  if (lane == 0) {
    att_mbar_init(bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncwarp();
  unsigned phase = 0;
  const uint32_t pr_bytes = (uint32_t)p.H * sizeof(T), q_bytes = (uint32_t)p.U * sizeof(T);
  const T* __restrict__ Pr = reinterpret_cast<const T*>(p.Pr);
  const T* __restrict__ Q = reinterpret_cast<const T*>(p.Q);
  const int n_warps = gridDim.x * warps;
  int front, back;
  att_list_counts(w, front, back);
  for (int v = blockIdx.x * warps + warp; v < front + back; v += n_warps) {
    const int it = v < front ? v : w.max_items - 1 - (v - front);          // list position = partial slot
    const int2 item = __ldg(w.items + it);
    const int b = item.x, seg = item.y;
    const long long start = row_nnz ? (long long)b * padded_stride : (long long)__ldg(row_ptr + b);
    const long long end = row_nnz ? start + __ldg(row_nnz + b) : (long long)__ldg(row_ptr + b + 1);
    const long long seg_start = start + (long long)seg * ATT_WSEG;
    const long long seg_end = min(end, seg_start + ATT_WSEG);
    int cc[ATT_WSEG / 32];
    float vv[ATT_WSEG / 32];
#pragma unroll
    for (int t = 0; t < ATT_WSEG / 32; ++t) {
      cc[t] = -1; vv[t] = 0.f;
      const long long k = seg_start + 32 * t + lane;
      if (k < seg_end) { cc[t] = __ldg(col + k); vv[t] = __ldg(val + k); }
      if (vv[t] == 0.f) cc[t] = -1;                               // an explicit 0.0 is "unrated", like the dense form
    }
    const int slot_idx = it;
    RowCore<1, 1, MODE, T> core(p, lane, b);
#pragma unroll
    for (int t = 0; t < ATT_WSEG / 32; ++t) {
      const int cnt = (int)min(32LL, seg_end - seg_start - 32 * t);
      if (cnt <= 0) break;
      const unsigned valid = __ballot_sync(FULL, cc[t] >= 0);
      if (valid) {
        att_fence_async();                                         // this warp's earlier shared-memory reads before the async writes
        __syncwarp();
        if (lane == 0) att_mbar_expect_tx(bar, (uint32_t)__popc(valid) * (pr_bytes + q_bytes));
        __syncwarp();
        if (cc[t] >= 0) {
          att_bulk_g2s(sPr + lane * 128, Pr + (long long)cc[t] * p.ldPr, pr_bytes, bar);
          att_bulk_g2s(sQ + lane * 128, Q + (long long)cc[t] * p.ldQ, q_bytes, bar);
        }
        att_mbar_wait(bar, phase);
        phase ^= 1u;
      }
      core.batch_smem(cc[t], vv[t], cnt, sPr, sQ, valid);
    }
    float* slot = w.partials + (long long)slot_idx * (p.U + 4);
    if (lane == 0) { slot[0] = core.m; slot[1] = core.l; }
    if (lane * 4 < p.U) st4(slot + 4 + lane * 4, make_float4(core.acc[0][0], core.acc[0][1], core.acc[0][2], core.acc[0][3]));
  }
}

// One WARP per candidate row: lanes take the segments' (max, denominator) pairs in parallel, then every lane owns 4 output columns
// and adds the partial vectors in segment order with independent 128-bit loads (v4 used a CTA per row whose threads walked the
// segments with three dependent scalar loops: 35 us at 8192 rows, 10 % of the K2 call).
constexpr int MERGE_WARPS = 2;      // 512 rows -> 256 CTAs: every SM takes part (8 warps per CTA left 84 of 148 SMs idle at config 2)
constexpr int MERGE_LD = 16;        // partial vectors in flight per lane: a typical row (~10 segments) is one round of loads
__global__ void __launch_bounds__(MERGE_WARPS * 32)
attention_merge_kernel(AttParams p, const int* __restrict__ row_ptr, const int* __restrict__ col, const float* __restrict__ val,
                       const int* __restrict__ row_nnz, long long padded_stride, AttWork w) {
  const int lane = threadIdx.x & 31;
  const int b = blockIdx.x * MERGE_WARPS + (threadIdx.x >> 5);
  if (b >= p.B) return;
  const long long start = row_nnz ? (long long)b * padded_stride : (long long)__ldg(row_ptr + b);
  const long long end = row_nnz ? start + __ldg(row_nnz + b) : (long long)__ldg(row_ptr + b + 1);
  const int first = __ldg(w.seg_base + b);
  const int nf = max(0, min(att_nfront(end - start), w.max_items - first));          // segments at the front of the list: slots first, first + 1, ...
  const int tail = att_nseg(end - start) > att_nfront(end - start) ? __ldg(w.tail_pos + b) : -1;      // + the short last segment, if any
  const int nseg = nf + (tail >= 0 ? 1 : 0);
  const long long stride = p.U + 4;
  auto slot = [&](int sidx) -> const float* { return w.partials + (long long)(sidx < nf ? first + sidx : tail) * stride; };
  float M = -INFINITY;
  for (int s0 = 0; s0 < nseg; s0 += 32) M = fmaxf(M, (s0 + lane < nseg) ? *slot(s0 + lane) : -INFINITY);
  M = warp_max(M);
  float Lsum = 0.f;
  for (int s0 = 0; s0 < nseg; s0 += 32) {
    if (s0 + lane < nseg) {
      const float2 ml = *reinterpret_cast<const float2*>(slot(s0 + lane));
      Lsum += ml.y * ((ml.x == -INFINITY) ? 0.f : __expf(ml.x - M));
    }
  }
  Lsum = warp_sum(Lsum);          // (the summation order over segments is fixed by the lane layout -> reproducible)
  const float inv = Lsum > 0.f ? 1.f / Lsum : 0.f;      // no valid rated item -> weights 0 -> user_emb = b_U (:208-209)
  for (int u = lane * 4; u < p.U; u += 128) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int s0 = 0; s0 < nseg; s0 += MERGE_LD) {
      float4 v[MERGE_LD];
      float f[MERGE_LD];
#pragma unroll
      for (int k = 0; k < MERGE_LD; ++k) {
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        f[k] = 0.f;
        if (s0 + k < nseg) {
          const float* sp = slot(s0 + k);
          const float ms = sp[0];
          f[k] = (ms == -INFINITY) ? 0.f : __expf(ms - M);
          v[k] = *reinterpret_cast<const float4*>(sp + 4 + u);
        }
      }
#pragma unroll
      for (int k = 0; k < MERGE_LD; ++k) {
        a.x = fmaf(v[k].x, f[k], a.x); a.y = fmaf(v[k].y, f[k], a.y); a.z = fmaf(v[k].z, f[k], a.z); a.w = fmaf(v[k].w, f[k], a.w);
      }
    }
    const float4 bu = p.bU ? ld4(p.bU + u) : make_float4(0.f, 0.f, 0.f, 0.f);
    st4(p.out + (long long)b * p.ldo + u, make_float4(fmaf(a.x, inv, bu.x), fmaf(a.y, inv, bu.y), fmaf(a.z, inv, bu.z), fmaf(a.w, inv, bu.w)));
  }
  if (p.att != nullptr) {
    for (long long k = start + lane; k < end; k += 32) {
      if (__ldg(val + k) != 0.f) {
        float* a = p.att + (long long)b * p.I + __ldg(col + k);
        *a = normalise_score(*a, M, Lsum);
      }
    }
  }
}

// ---- dense (B, I) user_matrix -> row-padded (col, val) lists + per-row counts ---------------------------------
// One CTA per row; pure streaming (four independent coalesced loads per thread and iteration, no dependent work), so
// the dense scan costs a few microseconds instead of sitting on the critical path of the pooling kernel, and the
// pooling kernel can split every row's non-zeros EVENLY over its warps.
// This streaming form reads the row from global memory twice; it serves rows wider than the shared memory of um_compact_vec_kernel below.
__global__ void __launch_bounds__(ATT_WARPS * 32)
um_compact_kernel(const float* __restrict__ um, long long ld_um, int I, int* __restrict__ col, float* __restrict__ val,
                  int* __restrict__ row_nnz, AttWork w) {
  __shared__ int s_cnt[ATT_WARPS];
  __shared__ int s_base;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x;
  const float* __restrict__ row = um + (long long)b * ld_um;
  const int chunks = (I + 31) >> 5;
  const int cpw = (chunks + ATT_WARPS - 1) / ATT_WARPS;
  const int i_begin = warp * cpw * 32, i_end = min(I, i_begin + cpw * 32);
  int cnt = 0;
  for (int i0 = i_begin; i0 < i_end; i0 += 128) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 32 + lane;
      v[u] = (i < i_end) ? __ldg(row + i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) cnt += __popc(__ballot_sync(FULL, v[u] != 0.f));
  }
  if (lane == 0) s_cnt[warp] = cnt;
  __syncthreads();
  int base = 0, total = 0;
#pragma unroll
  for (int w = 0; w < ATT_WARPS; ++w) {
    if (w < warp) base += s_cnt[w];
    total += s_cnt[w];
  }
  if (threadIdx.x == 0) row_nnz[b] = total;
  att_emit_items(w, b, total, threadIdx.x, ATT_WARPS * 32, &s_base);      // this row's (row, segment) work items
  long long out = (long long)b * I + base;
  for (int i0 = i_begin; i0 < i_end; i0 += 128) {
    float v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int i = i0 + u * 32 + lane;
      v[u] = (i < i_end) ? __ldg(row + i) : 0.f;
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const bool nz = v[u] != 0.f;
      const unsigned mask = __ballot_sync(FULL, nz);
      if (nz) {
        const long long pos = out + __popc(mask & ((1u << lane) - 1u));
        col[pos] = i0 + u * 32 + lane;
        val[pos] = v[u];
      }
      out += __popc(mask);
    }
  }
}

// The compaction staged through shared memory with 128-bit accesses (round 2: the scalar form above issued ~1,700 instructions per warp and row —
// 60 % issue-slot utilisation, 14 us for the 19 MB matrix of config 2).  A row starts on a 4-byte boundary only, so it is staged into shared
// memory SHIFTED by its phase (`shift` = words past a 16-byte boundary): padded element e = column e - shift, elements [0, shift) and the tail
// pad are zeros and drop out of the compaction like any other zero.  Interior vectors move as LDG.128 -> STS.128 (all of a thread's loads in
// flight at once, clamped rather than predicated), the <= 6 edge elements as scalars.  The scans read one float4 per lane: four ballots per
// 128 elements give the lane-major (= column) order.
__global__ void __launch_bounds__(ATT_WARPS * 32)
um_compact_vec_kernel(const float* __restrict__ um, long long ld_um, int I, int* __restrict__ col, float* __restrict__ val,
                      int* __restrict__ row_nnz, AttWork w) {
  extern __shared__ __align__(16) float um_vec_smem[];
  __shared__ int s_cnt[ATT_WARPS];
  __shared__ int s_base;
  constexpr int NT = ATT_WARPS * 32;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int b = blockIdx.x;
  const float* __restrict__ grow = um + (long long)b * ld_um;
  const int shift = (int)(((uintptr_t)grow >> 2) & 3);
  const int n = I + shift, n4 = (n + 3) >> 2;
  const int q_lo = shift ? 1 : 0, q_hi = n >> 2;                          // vectors entirely inside the row
  const float4* __restrict__ g4 = reinterpret_cast<const float4*>(grow - shift);
  float4* s4 = reinterpret_cast<float4*>(um_vec_smem);
  constexpr int NLD = 10;                                                 // 256 threads x 10 vectors = 10,240 columns per round
  for (int q0 = q_lo; q0 < q_hi; q0 += NT * NLD) {
    float4 v[NLD];
#pragma unroll
    for (int u = 0; u < NLD; ++u) v[u] = __ldcs(g4 + min(q0 + u * NT + tid, q_hi - 1));
#pragma unroll
    for (int u = 0; u < NLD; ++u) {
      const int q = q0 + u * NT + tid;
      if (q < q_hi) s4[q] = v[u];
    }
  }
  if (tid < 8) {                                                          // edges: first vector (tid 0-3), last vector (tid 4-7), pads = 0
    const int e = (tid < 4) ? tid : 4 * (n4 - 1) + (tid - 4);
    const bool edge_vec = (tid < 4) ? (q_lo == 1 || q_hi == 0) : (q_hi < n4);
    if (edge_vec && e < 4 * n4) {
      const int c = e - shift;
      um_vec_smem[e] = (c >= 0 && c < I) ? __ldcs(grow + c) : 0.f;
    }
  }
  __syncthreads();
  const int vpw = (((n4 + ATT_WARPS - 1) / ATT_WARPS) + 31) & ~31;       // vectors per warp, whole iterations of 32
  const int q_begin = warp * vpw, q_end = min(n4, q_begin + vpw);
  int cnt = 0;
  for (int q0 = q_begin; q0 < q_end; q0 += 32) {
    const int q = q0 + lane;
    const float4 t = (q < q_end) ? s4[q] : make_float4(0.f, 0.f, 0.f, 0.f);
    cnt += (t.x != 0.f) + (t.y != 0.f) + (t.z != 0.f) + (t.w != 0.f);
  }
  cnt = __reduce_add_sync(FULL, cnt);
  if (lane == 0) s_cnt[warp] = cnt;
  __syncthreads();
  int base = 0, total = 0;
#pragma unroll
  for (int x = 0; x < ATT_WARPS; ++x) {
    if (x < warp) base += s_cnt[x];
    total += s_cnt[x];
  }
  if (tid == 0) row_nnz[b] = total;
  att_emit_items(w, b, total, tid, NT, &s_base);                          // this row's (row, segment) work items
  long long out = (long long)b * I + base;
  const unsigned lt = (1u << lane) - 1u;
  for (int q0 = q_begin; q0 < q_end; q0 += 32) {
    const int q = q0 + lane;
    const float4 t = (q < q_end) ? s4[q] : make_float4(0.f, 0.f, 0.f, 0.f);
    const float x[4] = {t.x, t.y, t.z, t.w};
    unsigned m[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) m[k] = __ballot_sync(FULL, x[k] != 0.f);
    long long pos = out + __popc(m[0] & lt) + __popc(m[1] & lt) + __popc(m[2] & lt) + __popc(m[3] & lt);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (x[k] != 0.f) {
        col[pos] = 4 * q + k - shift;
        val[pos] = x[k];
        ++pos;
      }
    }
    out += __popc(m[0]) + __popc(m[1]) + __popc(m[2]) + __popc(m[3]);
  }
}

// ---- drop-in front-end: the reference's dense (B, I) user_matrix --------------------------------------------
template <int HV, int UV, int MODE, typename T>
__global__ void __launch_bounds__(ATT_WARPS * 32)
attention_pool_dense_kernel(AttParams p, const float* __restrict__ um, long long ld_um) {
  __shared__ int qcol[ATT_WARPS][64];
  __shared__ float qval[ATT_WARPS][64];
  __shared__ float s_m[ATT_WARPS], s_l[ATT_WARPS];
  __shared__ __align__(16) float s_acc[ATT_WARPS * UV * 128];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int b = blockIdx.x;
  RowCore<HV, UV, MODE, T> core(p, lane, b);
  const float* __restrict__ row = um + (long long)b * ld_um;
  // every warp scans a contiguous slice of the row (multiples of 32 columns) and compacts its non-zeros on the fly
  const int chunks = (p.I + 31) >> 5;
  const int cpw = (chunks + ATT_WARPS - 1) / ATT_WARPS;
  const int i_begin = warp * cpw * 32, i_end = min(p.I, i_begin + cpw * 32);
  int qn = 0;
  for (int i0 = i_begin; i0 < i_end; i0 += 32) {
    const int i = i0 + lane;
    const float v = (i < i_end) ? __ldg(row + i) : 0.f;
    const bool nz = v != 0.f;
    const unsigned mask = __ballot_sync(FULL, nz);
    if (nz) {
      const int pos = qn + __popc(mask & ((1u << lane) - 1u));
      qcol[warp][pos] = i;
      qval[warp][pos] = v;
    }
    qn += __popc(mask);
    __syncwarp();
    if (qn >= 32) {
      core.batch(qcol[warp][lane], qval[warp][lane], 32);
      const int rem = qn - 32;
      int tc = 0; float tv = 0.f;
      if (lane < rem) { tc = qcol[warp][32 + lane]; tv = qval[warp][32 + lane]; }
      __syncwarp();
      if (lane < rem) { qcol[warp][lane] = tc; qval[warp][lane] = tv; }
      qn = rem;
      __syncwarp();
    }
  }
  if (qn > 0) core.batch(lane < qn ? qcol[warp][lane] : -1, lane < qn ? qval[warp][lane] : 0.f, qn);
  core.export_state(s_m, s_l, s_acc, warp);
  __syncthreads();
  float M, Lsum;
  merge_and_write<UV>(p, b, s_m, s_l, s_acc, M, Lsum);
  if (p.att != nullptr) {
    __syncwarp();
    for (int i = i_begin + lane; i < i_end; i += 32) {
      if (__ldg(row + i) != 0.f) {
        float* a = p.att + (long long)b * p.I + i;
        *a = normalise_score(*a, M, Lsum);
      }
    }
  }
}

struct AttInputs {
  const float* um; long long ld_um;
  const int* row_ptr; const int* col; const float* val;
  void* ws; size_t ws_bytes;
  long long max_row_nnz;     // CSR form: upper bound of a row's length (0 = unknown -> I); sizes the work list and the partial slots
  long long nnz;             // CSR form: number of stored entries (0 = unknown); tightens the same bound
};

static size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }
// upper bound of the number of (row, segment) work items: every row ends with at most one partial segment
static long long att_max_items(long long B, long long I, long long max_row_nnz, long long nnz) {
  const long long full = B * std::max(1LL, (I + ATT_WSEG - 1) / ATT_WSEG);
  if (nnz > 0) return std::min(full, nnz / ATT_WSEG + B);                 // exact knowledge wins over the hint
  if (max_row_nnz > 0) return std::min(full, B * ((max_row_nnz + ATT_WSEG - 1) / ATT_WSEG));
  return full;
}
struct AttLayout { size_t counter, tail_pos, seg_base, items, partials, compact, total; };
// workspace = counters (2) | tail_pos (B) | seg_base (B) | items | partials | [dense: col, val, row_nnz lists]
static AttLayout att_layout(long long B, long long I, int U, bool dense, long long max_row_nnz, long long nnz) {
  const long long items = att_max_items(B, I, dense ? 0 : max_row_nnz, dense ? 0 : nnz);
  AttLayout l;
  l.counter = 0;
  l.tail_pos = 256;
  l.seg_base = l.tail_pos + align256((size_t)B * sizeof(int));
  l.items = l.seg_base + align256((size_t)B * sizeof(int));
  l.partials = l.items + align256((size_t)items * sizeof(int2));
  l.compact = l.partials + align256((size_t)items * (size_t)(U + 4) * sizeof(float));
  l.total = l.compact + (dense ? (size_t)(B * I) * (sizeof(int) + sizeof(float)) + (size_t)B * sizeof(int) + 64 : 0);
  return l;
}

struct AttLists { const int* col; const float* val; const int* row_nnz; const int* row_ptr; long long stride; };

// First phase of the segment-parallel path: zero the counter, compact a dense matrix (or read the CSR's row lengths) and write
// the work list.
static int att_prepare(int B, int I, int U, const AttInputs& in, cudaStream_t st, AttWork& w, AttLists& lists) {
  const bool dense = in.um != nullptr;
  const AttLayout lay = att_layout(B, I, U, dense, in.max_row_nnz, in.nnz);
  unsigned char* ws = reinterpret_cast<unsigned char*>(in.ws);
  w.counter = reinterpret_cast<int*>(ws + lay.counter);
  w.tail_pos = reinterpret_cast<int*>(ws + lay.tail_pos);
  w.seg_base = reinterpret_cast<int*>(ws + lay.seg_base);
  w.items = reinterpret_cast<int2*>(ws + lay.items);
  w.partials = reinterpret_cast<float*>(ws + lay.partials);
  const long long max_items = att_max_items(B, I, dense ? 0 : in.max_row_nnz, dense ? 0 : in.nnz);
  if (max_items > 0x7fffffffLL) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_pool: more than 2^31 segments");
  w.max_items = (int)max_items;
  B200REC_CUDA(cudaMemsetAsync(w.counter, 0, 2 * sizeof(int), st));
  lists.col = in.col; lists.val = in.val; lists.row_nnz = nullptr; lists.row_ptr = in.row_ptr; lists.stride = 0;
  if (dense) {                         // streaming compaction of the dense matrix into row-padded lists (+ the work list)
    int* wcol = reinterpret_cast<int*>(ws + lay.compact);
    float* wval = reinterpret_cast<float*>(wcol + (size_t)B * I);
    int* wnnz = reinterpret_cast<int*>(wval + (size_t)B * I);
    const size_t row_bytes = (size_t)I * sizeof(float);
    if (row_bytes + 32 <= 96 * 1024) {
      static B200recSmemOptIn opted;
      B200REC_CUDA(b200rec_opt_in_smem(opted, um_compact_vec_kernel, 96 * 1024));
      um_compact_vec_kernel<<<B, ATT_WARPS * 32, row_bytes + 32, st>>>(in.um, in.ld_um, I, wcol, wval, wnnz, w);
    } else {
      um_compact_kernel<<<B, ATT_WARPS * 32, 0, st>>>(in.um, in.ld_um, I, wcol, wval, wnnz, w);
    }
    B200REC_CHECK_LAUNCH();
    lists.col = wcol; lists.val = wval; lists.row_nnz = wnnz; lists.row_ptr = nullptr; lists.stride = I;
  } else {
    att_worklist_kernel<<<ceil_div_i(B, 128), 128, 0, st>>>(in.row_ptr, B, w);
    B200REC_CHECK_LAUNCH();
  }
  return B200REC_OK;
}

template <int HV, int UV, int MODE, typename T>
static int launch_att(const AttParams& p, const AttInputs& in, cudaStream_t st) {
  const bool dense = in.um != nullptr;
  const AttLayout lay = att_layout(p.B, p.I, p.U, dense, in.max_row_nnz, in.nnz);
  const bool have_ws = in.ws && in.ws_bytes >= lay.total;
  if (!have_ws) {                      // no workspace: single fused kernel, one CTA per row
    if (dense) attention_pool_dense_kernel<HV, UV, MODE, T><<<p.B, ATT_WARPS * 32, 0, st>>>(p, in.um, in.ld_um);
    else attention_pool_csr_kernel<HV, UV, MODE, T><<<p.B, ATT_WARPS * 32, 0, st>>>(p, in.row_ptr, in.col, in.val, nullptr, 0);
    B200REC_CHECK_LAUNCH();
    return B200REC_OK;
  }
  AttWork w;
  AttLists lists;
  {
    const int rc = att_prepare(p.B, p.I, p.U, in, st, w, lists);
    if (rc) return rc;
  }
  const int* ccol = lists.col; const float* cval = lists.val; const int* cnnz = lists.row_nnz; const int* rp = lists.row_ptr;
  const long long stride = lists.stride;
  const long long max_items = w.max_items;
  // rows as TMA bulk copies need 16-byte aligned rows whose length is a multiple of 16 bytes
  const bool no_tma = g_att_path == 1, force_tma = g_att_path == 2;
  // tables that stay in L2 (config 2: 10 MB) are served faster by the register-staged gathers with 16 warps per SM (72 vs 98 us);
  // the TMA staging pays when the rows come from HBM
  const bool big_tables = (double)p.I * (p.H + p.U) * sizeof(T) > 0.5 * b200rec_l2_bytes();
  const bool tma_ok = HV == 1 && UV == 1 && !no_tma && (big_tables || force_tma) && (p.H * sizeof(T)) % 16 == 0 && (p.U * sizeof(T)) % 16 == 0 &&
                      (p.ldPr * sizeof(T)) % 16 == 0 && (p.ldQ * sizeof(T)) % 16 == 0 && (uintptr_t)p.Pr % 16 == 0 && (uintptr_t)p.Q % 16 == 0;
  if constexpr (HV == 1 && UV == 1) {
    if (tma_ok) {
      const int warps = sizeof(T) == 4 ? 7 : 14;      // 7 x 32 KB (fp32) of rows in flight per SM: 224 KB of the 227
      const size_t smem = (size_t)warps * 64 * 128 * sizeof(T) + (size_t)warps * sizeof(uint64_t);
      static B200recSmemOptIn opted;       // per template instantiation, one bit per device
      B200REC_CUDA(b200rec_opt_in_smem(opted, attention_wseg_tma_kernel<MODE, T>, (int)smem));
      const int grid = (int)std::max(1LL, std::min((max_items + warps - 1) / warps, (long long)b200rec_num_sms()));
      attention_wseg_tma_kernel<MODE, T><<<grid, warps * 32, smem, st>>>(p, rp, ccol, cval, cnnz, stride, w);
      B200REC_CHECK_LAUNCH();
    }
  }
  if (!tma_ok) {
    const int ctas_per_sm = (HV == 1 && UV == 1) ? 2 : 1;
    const int grid = (int)std::max(1LL, std::min((max_items + ATT_WARPS - 1) / ATT_WARPS, (long long)b200rec_num_sms() * ctas_per_sm));
    attention_wseg_kernel<HV, UV, MODE, T><<<grid, ATT_WARPS * 32, 0, st>>>(p, rp, ccol, cval, cnnz, stride, w);
    B200REC_CHECK_LAUNCH();
  }
  attention_merge_kernel<<<ceil_div_i(p.B, MERGE_WARPS), MERGE_WARPS * 32, 0, st>>>(p, rp, ccol, cval, cnnz, stride, w);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

template <int MODE, typename T>
static int dispatch_att(const AttParams& p, const AttInputs& in, cudaStream_t st) {
  const int w = p.H > p.U ? p.H : p.U;
  if (w <= 128) return launch_att<1, 1, MODE, T>(p, in, st);
  if (w <= 256) return launch_att<2, 2, MODE, T>(p, in, st);
  if (w <= 512) return launch_att<4, 4, MODE, T>(p, in, st);
  return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_pool: att_dense / user_emb wider than 512");
}

#ifdef B200REC_ATT_DROPOUT
}  // namespace attdrop
#endif
}  // namespace b200rec

using namespace b200rec;
#ifdef B200REC_ATT_DROPOUT
using namespace b200rec::attdrop;
#define B200REC_ATT_ENTRY b200rec_attention_pool_dropout
#else
#define B200REC_ATT_ENTRY b200rec_attention_pool

extern "C" int b200rec_attention_pool_set_path(int path) {
  if (path < 0 || path > 2) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool_set_path: 0 auto, 1 registers, 2 TMA");
  g_att_path = path;
  return B200REC_OK;
}
extern "C" size_t b200rec_attention_pool_workspace(int64_t B, int64_t I, int U, int dense) {
  return (B > 0 && I > 0 && U > 0) ? att_layout(B, I, U, dense != 0, 0, 0).total : 0;
}
extern "C" size_t b200rec_attention_pool_workspace_csr(int64_t B, int64_t I, int U, int64_t max_row_nnz, int64_t nnz) {
  return (B > 0 && I > 0 && U > 0) ? att_layout(B, I, U, false, max_row_nnz, nnz).total : 0;
}

#endif  // !B200REC_ATT_DROPOUT

extern "C" int B200REC_ATT_ENTRY(const b200rec_attention_t* a, b200rec_stream_t stream) {
  if (!a) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: null descriptor");
  if (a->B < 0 || a->I < 0 || a->H <= 0 || a->U <= 0 || (a->H % 4) || (a->U % 4))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: H and U must be positive multiples of 4");
  if (a->B == 0) return B200REC_OK;
  if (!a->Pc || !a->out || (a->I > 0 && (!a->Pr || !a->Q))) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: null table");
  if (!a->user_matrix && !(a->row_ptr && (a->col || a->I == 0)))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: need user_matrix or CSR");
  if (a->mode == MODE_NET && !a->a2) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: a2 missing");
  if (a->ldo < a->U) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: ldo too small");
  if ((uintptr_t)a->Pc % 16 || (uintptr_t)a->Pr % 8 || (uintptr_t)a->Q % 8 || (uintptr_t)a->out % 16 || (a->ldo % 4) ||
      (a->table_dtype == B200REC_F32 && ((uintptr_t)a->Pr % 16 || (uintptr_t)a->Q % 16)) || (a->bU && (uintptr_t)a->bU % 16) ||
      (a->a2 && (uintptr_t)a->a2 % 16))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: pointers must be 16-byte aligned");
  AttParams p;
  p.Pc = a->Pc; p.Pr = a->Pr; p.Q = a->Q; p.a2 = a->a2; p.a20 = a->a20; p.bU = a->bU;
  p.out = a->out; p.ldo = a->ldo; p.att = a->att_weights;
  p.B = (int)a->B; p.I = (int)a->I; p.H = a->H; p.U = a->U;
  p.Ec = a->train_cand_emb; p.Er = a->train_rated_emb; p.E = a->E; p.atol = a->atol; p.rtol = a->rtol;
  p.drop_zero_scores = a->drop_zero_scores;
  p.score_scale = a->score_scale == 0.f ? 1.f : a->score_scale;
  p.ldPr = a->ld_pr ? a->ld_pr : a->H;
  p.ldQ = a->ld_q ? a->ld_q : a->U;
  p.ldPc = a->ld_pc ? a->ld_pc : a->H;
  p.drop_key = 0u; p.drop_thr16 = 65536u; p.drop_scale = 1.f; p.drop_seed_dev = nullptr;
#ifdef B200REC_ATT_DROPOUT
  if (!(a->dropout_p >= 0.f && a->dropout_p < 1.f)) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool_dropout: need 0 <= dropout_p < 1");
  if (a->B >= (1 << 26)) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_pool_dropout: more than 2^26 candidate rows");
  {
    unsigned thr = (unsigned)((1.0 - (double)a->dropout_p) * 65536.0 + 0.5);
    if (thr < 1u) thr = 1u;
    if (thr > 65536u) thr = 65536u;
    p.drop_thr16 = thr;
    p.drop_scale = 65536.f / (float)thr;
    p.drop_key = (unsigned)(a->dropout_seed ^ (a->dropout_seed >> 32));
    p.drop_seed_dev = reinterpret_cast<const unsigned long long*>(a->dropout_seed_dev);
  }
#else
  if (a->dropout_p != 0.f) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: inner dropout is applied by b200rec_attention_pool_dropout");
#endif
  if (p.ldPc < a->H || (p.ldPc % 4)) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: bad Pc leading dimension");
  if (p.ldPr < a->H || p.ldQ < a->U || (p.ldPr % 4) || (p.ldQ % 4)) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: bad table leading dimension");
  // the kernels address a gathered row by a 32-bit count of 4-element vectors
  if (p.ldPr > 0x7fffffffLL || p.ldQ > 0x7fffffffLL || (double)a->I * (double)(p.ldPr / 4) >= 4294967296.0 || (double)a->I * (double)(p.ldQ / 4) >= 4294967296.0)
    return b200rec_fail(B200REC_ERR_UNSUPPORTED, "attention_pool: table larger than 2^34 elements");
  if (p.Ec && (!p.Er || p.E <= 0)) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: training mask needs both embeddings");
  cudaStream_t st = (cudaStream_t)stream;
  const long long ld_um = a->user_matrix ? (a->ld_user_matrix ? a->ld_user_matrix : a->I) : 0;
  AttInputs in{a->user_matrix, ld_um, a->row_ptr, a->col, a->val, a->workspace, a->workspace_bytes, a->max_row_nnz, a->nnz};
  if (a->table_dtype == B200REC_F32) {
    if (a->mode == MODE_NET) return dispatch_att<MODE_NET, float>(p, in, st);
    if (a->mode == MODE_DOT) return dispatch_att<MODE_DOT, float>(p, in, st);
  } else if (a->table_dtype == B200REC_BF16) {
    if (a->mode == MODE_NET) return dispatch_att<MODE_NET, __nv_bfloat16>(p, in, st);
    if (a->mode == MODE_DOT) return dispatch_att<MODE_DOT, __nv_bfloat16>(p, in, st);
  }
  return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_pool: bad mode / table_dtype");
}
