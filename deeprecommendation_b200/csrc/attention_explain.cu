// K9 — AttentionNCF explanations for many users' recommendations: the rated items whose attention weight is above a threshold.
//
// The reference's serving call explains every recommended item b of a user by the rated items i with (src/webapp/backend.py:102-110)
//
//   α_bi > explain_factor / R_u + explain_constant,      R_u = length of u's list (zero-centred entries included)
//
// where α_bi is the eval-mode attention weight of attention_ncf.py:136-209 (K8's algebra, csrc/attention_recommend.cu):
//   s_bi = a2 · ReLU(Pc[b] + Pr[i]) + a20  (MODE_NET)   or   <Pc[b], Pr[i]>  (MODE_DOT);   α_bi = softmax_i(s_b·) over the entries with um_i != 0.
//
// All k (<= 64) candidates of a user share one list, so one CTA takes one user: the candidates' Pc rows are staged once, the list streams
// through shared memory 32 entries at a time (Pr rows h-major), and warp w scores candidates w, w + 8, ... against the chunk, lane j = entry j.
// A candidate's scores of one chunk are thus one warp's registers: softmax sums, counts and the compaction are warp reductions / ballots.
// The scores are K8's, operation for operation (fmaf over h = 0 .. H-1, then + a20).
//
//   count  pass 1: running max and denominator per candidate (online softmax);  pass 2: entries with α > thr.
//          Writes counts and (max, 1/denominator, thr) per (user, candidate) row into the workspace; a one-CTA scan turns the counts into ptr.
//   fill   one pass recomputes α from the stored (max, 1/denominator) and writes the kept (item, α) pairs; a ballot per chunk keeps list order.
// Both kernels compute α with the same code from the same inputs, so the fill writes exactly the counted entries.  No atomics, fixed
// reduction orders: bit-identical output run to run.
#include <math.h>
#include <stdio.h>

#include "common.cuh"

namespace b200rec {

constexpr int AE_THREADS = 256;
constexpr int AE_WARPS = AE_THREADS / 32;
constexpr int AE_RC = 32;                   // list entries per shared-memory chunk (one per lane)
constexpr int AE_KMAX = 64;                 // candidates per user
constexpr int AE_SLOTS = AE_KMAX / AE_WARPS;  // candidates per warp
constexpr int AE_HMAX = 256;
enum { AE_NET = 0, AE_DOT = 1 };

struct AeParams {
  const float* Pc; long long ld_pc;         // (nI, H) candidate score table
  const float* Pr; long long ld_pr;         // (nI, H) rated score table
  const float* a2; const float* a20;        // MODE_NET: (H) and a device scalar (or null)
  const long long* list_ptr; const int* list_item; const float* list_val;
  const long long* users;
  const long long* items;                   // (n_users, k) catalogue rows; outside [0, nI): padding, an empty row
  int nI, H, k, KT;                         // KT = k rounded up to a multiple of AE_WARPS
  double factor, constant;                  // (count) threshold = factor · (1 / max(R_u, 1)) + constant
  int* counts; float4* stats;               // workspace: per row (user slot u, candidate j) = u·k + j
  const long long* ptr; long long* because; float* attention;   // (fill)
};

static size_t ae_smem_bytes(int H, int KT) { return (size_t)(H * KT + H * AE_RC + H) * 4; }

// s of (candidate row pc, entry column pr of the h-major chunk) — K8's arithmetic
template <int MODE>
__device__ __forceinline__ float ae_score(const float* pc, const float* pr, const float* sA2, int H, float a20) {
  float s = 0.f;
#pragma unroll 2
  for (int h = 0; h < H; h += 4) {
    const float4 a = *reinterpret_cast<const float4*>(pc + h);
    const float av[4] = {a.x, a.y, a.z, a.w};
    if (MODE == AE_NET) {
      const float4 w = *reinterpret_cast<const float4*>(sA2 + h);
      const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int q = 0; q < 4; ++q) s = fmaf(wv[q], fmaxf(av[q] + pr[(h + q) * AE_RC], 0.f), s);
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) s = fmaf(av[q], pr[(h + q) * AE_RC], s);
    }
  }
  return s + a20;
}

// α of a score (-inf: zero-centred or past the list's end) and whether it explains; the count and the fill both decide through here
__device__ __forceinline__ bool ae_keep(float s, float4 st, float& alpha) {
  alpha = s == -INFINITY ? 0.f : __expf(s - st.x) * st.y;
  return s != -INFINITY && alpha > st.z;
}

// Streams the user's list [e_begin, e_end) through shared memory and calls f(t, s, item) for every live candidate slot t of this warp
// (candidate warp + 8 t), s = this lane's score against entry c0 + lane of the chunk.  Every thread of the CTA must call it.
template <int MODE, typename F>
__device__ __forceinline__ void ae_stream(const AeParams& p, long long e_begin, long long e_end, const float* sPc, float* sPr, const float* sA2,
                                          float a20, unsigned live, F&& f) {
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, H = p.H, H4 = H >> 2;
  for (long long c0 = e_begin; c0 < e_end; c0 += AE_RC) {
    const int cnt = (int)min((long long)AE_RC, e_end - c0);
    const bool in = lane < cnt;
    const int item = in ? __ldg(p.list_item + c0 + lane) : 0;
    const float val = in ? __ldg(p.list_val + c0 + lane) : 0.f;
    __syncthreads();                                                   // the previous chunk's scores are done with sPr
    for (int idx = tid; idx < AE_RC * H4; idx += AE_THREADS) {
      const int j = idx % AE_RC, h = (idx / AE_RC) * 4;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (j < cnt) v = ld4(p.Pr + (long long)__ldg(p.list_item + c0 + j) * p.ld_pr + h);
      sPr[(h + 0) * AE_RC + j] = v.x; sPr[(h + 1) * AE_RC + j] = v.y;
      sPr[(h + 2) * AE_RC + j] = v.z; sPr[(h + 3) * AE_RC + j] = v.w;
    }
    __syncthreads();
#pragma unroll
    for (int t = 0; t < AE_SLOTS; ++t) {
      if (!(live >> t & 1u)) continue;
      const float s = ae_score<MODE>(sPc + (warp + AE_WARPS * t) * H, sPr + lane, sA2, H, a20);
      f(t, val != 0.f ? s : -INFINITY, item);                         // zero-centred entries are "unrated" (attention_ncf.py:158,192)
    }
  }
}

// stages the k candidates' Pc rows (row-major, padding rows zero) and a2; returns this warp's mask of real candidates
template <int MODE>
__device__ __forceinline__ unsigned ae_stage_candidates(const AeParams& p, float* sPc, float* sA2) {
  const int tid = threadIdx.x, warp = tid >> 5, H = p.H, H4 = H >> 2;
  const long long* it = p.items + (long long)blockIdx.x * p.k;
  for (int idx = tid; idx < p.KT * H4; idx += AE_THREADS) {
    const int c = idx / H4, h = (idx % H4) * 4;
    const long long b = c < p.k ? __ldg(it + c) : -1;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (b >= 0 && b < p.nI) v = ld4(p.Pc + b * p.ld_pc + h);
    st4(sPc + c * H + h, v);
  }
  if (MODE == AE_NET)
    for (int h = tid; h < H; h += AE_THREADS) sA2[h] = __ldg(p.a2 + h);
  unsigned valid = 0u;
#pragma unroll
  for (int t = 0; t < AE_SLOTS; ++t) {
    const int c = warp + AE_WARPS * t;
    const long long b = c < p.k ? __ldg(it + c) : -1;
    if (b >= 0 && b < p.nI) valid |= 1u << t;
  }
  return valid;
}

template <int MODE>
__global__ void __launch_bounds__(AE_THREADS, 2)
attention_explain_count_kernel(const AeParams p) {
  extern __shared__ __align__(16) float ae_smem[];
  float* sPc = ae_smem;                        // [KT][H]
  float* sPr = sPc + p.KT * p.H;               // [H][AE_RC]
  float* sA2 = sPr + p.H * AE_RC;              // [H]
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long urow = __ldg(p.users + blockIdx.x);
  const long long e_begin = __ldg(p.list_ptr + urow), e_end = __ldg(p.list_ptr + urow + 1);
  const float a20 = (MODE == AE_NET && p.a20 != nullptr) ? __ldg(p.a20) : 0.f;
  const float thr = (float)(p.factor * (1.0 / (double)max(e_end - e_begin, 1ll)) + p.constant);   // backend.py:102, as recommend_for_user
                                                                                                      // forms it; compared in fp32
  const unsigned valid = ae_stage_candidates<MODE>(p, sPc, sA2);
  __syncthreads();

  float m[AE_SLOTS], l[AE_SLOTS];                                   // l: the denominator, then its inverse
  int n[AE_SLOTS];
#pragma unroll
  for (int t = 0; t < AE_SLOTS; ++t) { m[t] = -INFINITY; l[t] = 0.f; n[t] = 0; }
  // pass 1: online softmax denominators (the warp butterflies leave the same value in every lane)
  ae_stream<MODE>(p, e_begin, e_end, sPc, sPr, sA2, a20, valid, [&](int t, float s, int) {
    const float m_new = fmaxf(m[t], warp_max(s));
    if (m_new != -INFINITY) {
      const float scale = __expf(m[t] - m_new);                       // m == -inf -> 0
      l[t] = l[t] * scale + warp_sum(s == -INFINITY ? 0.f : __expf(s - m_new));
      m[t] = m_new;
    }
  });
  unsigned live = 0u;
#pragma unroll
  for (int t = 0; t < AE_SLOTS; ++t) {
    if (l[t] > 0.f) live |= 1u << t;                                  // a candidate with nothing rated explains nothing
    l[t] = l[t] > 0.f ? 1.f / l[t] : 0.f;
  }
  // pass 2: count the entries that explain
  ae_stream<MODE>(p, e_begin, e_end, sPc, sPr, sA2, a20, live, [&](int t, float s, int) {
    float a;
    n[t] += __popc(__ballot_sync(FULL, ae_keep(s, make_float4(m[t], l[t], thr, 0.f), a)));
  });
  if (lane == 0) {
#pragma unroll
    for (int t = 0; t < AE_SLOTS; ++t) {
      const int c = warp + AE_WARPS * t;
      if (c >= p.k) break;
      const long long row = (long long)blockIdx.x * p.k + c;
      p.counts[row] = n[t];
      p.stats[row] = make_float4(m[t], l[t], thr, 0.f);
    }
  }
}

template <int MODE>
__global__ void __launch_bounds__(AE_THREADS, 2)
attention_explain_fill_kernel(const AeParams p) {
  extern __shared__ __align__(16) float ae_smem[];
  float* sPc = ae_smem;
  float* sPr = sPc + p.KT * p.H;
  float* sA2 = sPr + p.H * AE_RC;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long row0 = (long long)blockIdx.x * p.k;
  if (__ldg(p.ptr + row0) == __ldg(p.ptr + row0 + p.k)) return;        // nothing to write for this user (uniform over the CTA)
  const long long urow = __ldg(p.users + blockIdx.x);
  const long long e_begin = __ldg(p.list_ptr + urow), e_end = __ldg(p.list_ptr + urow + 1);
  const float a20 = (MODE == AE_NET && p.a20 != nullptr) ? __ldg(p.a20) : 0.f;
  const unsigned valid = ae_stage_candidates<MODE>(p, sPc, sA2);
  __syncthreads();

  float4 st[AE_SLOTS];
  long long pos[AE_SLOTS], end[AE_SLOTS];
  unsigned live = 0u;
#pragma unroll
  for (int t = 0; t < AE_SLOTS; ++t) {
    const int c = warp + AE_WARPS * t;
    const bool row = c < p.k;
    st[t] = row ? p.stats[row0 + c] : make_float4(0.f, 0.f, 0.f, 0.f);
    pos[t] = row ? __ldg(p.ptr + row0 + c) : 0;
    end[t] = row ? __ldg(p.ptr + row0 + c + 1) : 0;
    if ((valid >> t & 1u) && end[t] > pos[t]) live |= 1u << t;
  }
  const unsigned below = (1u << lane) - 1u;
  ae_stream<MODE>(p, e_begin, e_end, sPc, sPr, sA2, a20, live, [&](int t, float s, int item) {
    float a;
    const bool keep = ae_keep(s, st[t], a);
    const unsigned mask = __ballot_sync(FULL, keep);
    const long long o = pos[t] + __popc(mask & below);
    if (keep && o < end[t]) {                                          // (bounded by ptr: a ptr from another call cannot write past a row)
      p.because[o] = item;
      p.attention[o] = a;
    }
    pos[t] += __popc(mask);
  });
}

// ptr[0] = 0, ptr[r + 1] = counts[0] + ... + counts[r]  (one CTA, int64 sums)
constexpr int AE_SCAN_THREADS = 1024;
__global__ void __launch_bounds__(AE_SCAN_THREADS)
attention_explain_scan_kernel(const int* __restrict__ counts, long long n, long long* __restrict__ ptr) {
  __shared__ long long s_warp[AE_SCAN_THREADS / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  long long carry = 0;
  if (threadIdx.x == 0) ptr[0] = 0;
  for (long long base = 0; base < n; base += AE_SCAN_THREADS) {
    const long long i = base + threadIdx.x;
    long long inc = i < n ? counts[i] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long v = __shfl_up_sync(FULL, inc, o);
      if (lane >= o) inc += v;
    }
    __syncthreads();                                                   // s_warp of the previous round has been read
    if (lane == 31) s_warp[warp] = inc;
    __syncthreads();
    long long wsum = s_warp[lane], winc = wsum;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const long long v = __shfl_up_sync(FULL, winc, o);
      if (lane >= o) winc += v;
    }
    const long long wbase = __shfl_sync(FULL, winc - wsum, warp);
    if (i < n) ptr[i + 1] = carry + wbase + inc;
    carry += __shfl_sync(FULL, winc, 31);
  }
}

static inline size_t ae_align(size_t n) { return (n + 255) & ~(size_t)255; }

template <int MODE, bool FILL>
static int ae_launch(const AeParams& p, int n_users, cudaStream_t st) {
  static B200recSmemOptIn opted;
  auto kernel = FILL ? attention_explain_fill_kernel<MODE> : attention_explain_count_kernel<MODE>;
  B200REC_CUDA(b200rec_opt_in_smem(opted, kernel, (int)ae_smem_bytes(AE_HMAX, AE_KMAX)));
  kernel<<<n_users, AE_THREADS, ae_smem_bytes(p.H, p.KT), st>>>(p);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

// argument checks shared by the two entry points; fills the common part of `p`
static int ae_setup(AeParams& p, const char* who, const float* Pc, int64_t ld_pc, const float* Pr, int64_t ld_pr, int H, int mode, const float* a2,
                    const float* a20, int64_t n_items, const int64_t* list_ptr, const int32_t* list_item, const float* list_val, const int64_t* users,
                    int64_t n_users, const int64_t* items, int k, const void* workspace, size_t workspace_bytes) {
  static thread_local char msg[160];
  auto fail = [&](int code, const char* what) {
    snprintf(msg, sizeof(msg), "%s: %s", who, what);
    return b200rec_fail(code, msg);
  };
  if (n_users < 0 || n_items < 0) return fail(B200REC_ERR_BAD_ARG, "negative size");
  if (k < 1 || k > AE_KMAX) return fail(B200REC_ERR_BAD_ARG, "k must be in 1..64");
  if (n_users > INT32_MAX || n_items > INT32_MAX / 2) return fail(B200REC_ERR_UNSUPPORTED, "n_users < 2^31 and n_items < 2^30");
  if (n_users > 0 && (!Pc || !Pr || !list_ptr || !list_item || !list_val || !users || !items))
    return fail(B200REC_ERR_BAD_ARG, "null operand");
  if (mode != B200REC_ATT_NET && mode != B200REC_ATT_DOT) return fail(B200REC_ERR_BAD_ARG, "bad mode");
  if (mode == B200REC_ATT_NET && !a2) return fail(B200REC_ERR_BAD_ARG, "mode NET needs a2");
  if (H <= 0 || (H & 3) || H > AE_HMAX) return fail(B200REC_ERR_UNSUPPORTED, "H must be a multiple of 4, <= 256");
  if (ld_pc < H || ld_pr < H || ((ld_pc | ld_pr) & 3)) return fail(B200REC_ERR_BAD_ARG, "leading dimensions must cover the rows and be multiples of 4");
  if (((uintptr_t)Pc | (uintptr_t)Pr) & 15) return fail(B200REC_ERR_BAD_ARG, "tables must be 16-byte aligned");
  if (workspace_bytes < b200rec_attention_explain_workspace(n_users, k) || (n_users > 0 && !workspace))
    return fail(B200REC_ERR_WORKSPACE, "workspace too small (b200rec_attention_explain_workspace)");
  p.Pc = Pc; p.ld_pc = ld_pc; p.Pr = Pr; p.ld_pr = ld_pr; p.a2 = a2; p.a20 = a20;
  p.list_ptr = reinterpret_cast<const long long*>(list_ptr); p.list_item = list_item; p.list_val = list_val;
  p.users = reinterpret_cast<const long long*>(users); p.items = reinterpret_cast<const long long*>(items);
  p.nI = (int)n_items; p.H = H; p.k = k; p.KT = (k + AE_WARPS - 1) / AE_WARPS * AE_WARPS;
  unsigned char* ws = reinterpret_cast<unsigned char*>(const_cast<void*>(workspace));
  p.counts = reinterpret_cast<int*>(ws);
  p.stats = reinterpret_cast<float4*>(ws + ae_align((size_t)n_users * k * sizeof(int)));
  p.ptr = nullptr; p.because = nullptr; p.attention = nullptr;
  return B200REC_OK;
}

}  // namespace b200rec

using namespace b200rec;

extern "C" size_t b200rec_attention_explain_workspace(int64_t n_users, int k) {
  if (n_users <= 0 || k <= 0) return 0;
  const size_t rows = (size_t)n_users * (size_t)k;
  return ae_align(rows * sizeof(int)) + rows * sizeof(float4);
}

extern "C" int b200rec_attention_explain_count(const float* Pc, int64_t ld_pc, const float* Pr, int64_t ld_pr, int H, int mode, const float* a2,
                                               const float* a20, int64_t n_items, const int64_t* list_ptr, const int32_t* list_item,
                                               const float* list_val, const int64_t* users, int64_t n_users, const int64_t* items, int k,
                                               double explain_factor, double explain_constant, int64_t* ptr, void* workspace,
                                               size_t workspace_bytes, b200rec_stream_t stream) {
  AeParams p;
  const int rc = ae_setup(p, "attention_explain_count", Pc, ld_pc, Pr, ld_pr, H, mode, a2, a20, n_items, list_ptr, list_item, list_val, users,
                          n_users, items, k, workspace, workspace_bytes);
  if (rc != B200REC_OK) return rc;
  if (!ptr) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_explain_count: null ptr");
  p.factor = explain_factor; p.constant = explain_constant;
  cudaStream_t st = (cudaStream_t)stream;
  if (n_users > 0) {
    const int r = mode == B200REC_ATT_NET ? ae_launch<AE_NET, false>(p, (int)n_users, st) : ae_launch<AE_DOT, false>(p, (int)n_users, st);
    if (r != B200REC_OK) return r;
  }
  attention_explain_scan_kernel<<<1, AE_SCAN_THREADS, 0, st>>>(p.counts, n_users * k, reinterpret_cast<long long*>(ptr));
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_attention_explain_fill(const float* Pc, int64_t ld_pc, const float* Pr, int64_t ld_pr, int H, int mode, const float* a2,
                                              const float* a20, int64_t n_items, const int64_t* list_ptr, const int32_t* list_item,
                                              const float* list_val, const int64_t* users, int64_t n_users, const int64_t* items, int k,
                                              const int64_t* ptr, const void* workspace, size_t workspace_bytes, int64_t* because, float* attention,
                                              b200rec_stream_t stream) {
  AeParams p;
  const int rc = ae_setup(p, "attention_explain_fill", Pc, ld_pc, Pr, ld_pr, H, mode, a2, a20, n_items, list_ptr, list_item, list_val, users,
                          n_users, items, k, workspace, workspace_bytes);
  if (rc != B200REC_OK) return rc;
  if (n_users > 0 && (!ptr || !because || !attention)) return b200rec_fail(B200REC_ERR_BAD_ARG, "attention_explain_fill: null output");
  if (n_users == 0) return B200REC_OK;
  p.ptr = reinterpret_cast<const long long*>(ptr);
  p.because = reinterpret_cast<long long*>(because);
  p.attention = attention;
  cudaStream_t st = (cudaStream_t)stream;
  return mode == B200REC_ATT_NET ? ae_launch<AE_NET, true>(p, (int)n_users, st) : ae_launch<AE_DOT, true>(p, (int)n_users, st);
}
