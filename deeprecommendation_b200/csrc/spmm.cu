// K3 — GraphNCF bipartite message passing as a row-owner CSR SpMM with symmetric degree normalisation and a
// fused per-layer combine.
//
// Replaces PyG `propagate` + `message` + scatter-add of gnn_ncf.py:39-94 and the `stack`+`mean` of :351.
// The reference transforms every EDGE (`W(x_j)` on an (E, d) tensor, :91-93) and scatter-adds with atomics;
// here the Linear is applied once per NODE beforehand (K1a with row_scale = deg^-1/2 of the source), so a layer is
//
//   x_next[r] = dinv[r] * sum_{k in row r}  w[k] * t[col[k]]            t[s] = dinv[s] * (W_type x[s] + b_type)
//   acc_out[r] = (acc_in[r] + x_next[r]) * acc_scale                    (running sum of hs; 1/(L+1) on the last layer)
//
// over the neighbour index built by K4 (edges stably sorted by destination, 8 bytes per edge: int32 source +
// fp32 weight).  Rows are cut into chunks of <= CHUNK edges at graph-build time; one warp owns one chunk, so the
// heavy-tailed MovieLens degrees (max ~81k) are edge-balanced.  Single-chunk rows are finished in the same
// kernel; multi-chunk rows write per-chunk partials that a second tiny kernel adds IN CHUNK ORDER — no atomics,
// bit-reproducible run to run (the reference's GPU scatter-add is not).  Each edge costs one coalesced 128-bit
// load per lane of the source row (d=128 fp32: 512 B per edge; d=64: two edges per warp step), 8 row gathers in
// flight per warp.  (A cp.async/LDGSTS shared-memory ring was tried and measured 1.5x SLOWER — 3.4 vs 2.25 ms per
// layer on the MovieLens-25M shape — and was dropped; see DESIGN.md §6.)
#include <math.h>

#include "common.cuh"

namespace b200rec {

constexpr int SPMM_WARPS = 8;
#ifndef SPMM_MIN_CTAS
#define SPMM_MIN_CTAS 4      // 4 CTAs x 8 warps at 64 registers (a few spilled index registers) beat 3 CTAs without spills: 10.7 vs 12.1 ms
#endif                      // per HBM-regime layer — resident warps, not per-warp latency, carry the gathers

constexpr int FIX_WARPS = 8;

struct SpmmParams {
  const int* chunk_row;
  const int* chunk_start;
  const int* chunk_slot;     // -1: the row has a single chunk (direct epilogue); else index into `partials`
  int n_chunks;
  int chunk_size;
  const int* row_ptr;
  const int* col;
  const float* w;            // per CSR entry, or null (binary graph: weight 1)
  const int* perm;           // CSR entry -> position in the interactions file (for the skip bitmap)
  const unsigned* skip_bits; // training: bit p set = interaction p is a target edge of this batch (masked out)
  const void* t;             // (N, d) source features, fp32 or bf16
  long long ld_t;
  int d;
  const float* dinv;         // per destination row, or null
  float* partials;
  float* x_next;             // nullable
  long long ld_x;
  const float* acc_in;       // nullable
  float* acc_out;            // nullable
  long long ld_acc;
  float acc_scale;
  // fix-up pass
  const int* multi_row;
  const int* multi_first_slot;
  const int* multi_n_slots;
  int n_multi;
  // LightGAT (gnn_ncf.py:97-177): edge weight = w * softmax over the row of att_src[col]; no degree normalisation
  const float* att_src;      // per SOURCE node score A[:, :d]·x[s]; null = LightGCN
  float* partials_ml;        // (n_slots, 2): running max and denominator of multi-chunk rows
  // partitioned propagation: finished rows go to the receive slot of their owner rank (peer-mapped arenas, csrc/peer.cu)
  void* push_dst[B200REC_PEER_MAX];
  int push_parts;
  int push_rpp;              // rows per owner
  long long push_off;        // element offset of this rank's slot inside an arena
  long long push_ld;
  long long push_ml_off;     // LightGAT + push: element offset of this rank's (m, l) statistics slot inside an arena
};

// writes 4 consecutive columns [c, c+4) of one finished row
template <bool PUSH = false>
__device__ __forceinline__ void row_epilogue4(const SpmmParams& p, int row, int c, float s, float4 v) {
  if (c >= p.d) return;
  v = make_float4(v.x * s, v.y * s, v.z * s, v.w * s);
  if constexpr (PUSH) {                 // reduce-scatter fused into the epilogue: one 512-byte remote store per warp and row
    const int o = row / p.push_rpp;
    st4(reinterpret_cast<float*>(p.push_dst[o]) + p.push_off + (long long)(row - o * p.push_rpp) * p.push_ld + c, v);
    return;
  }
  if (p.x_next) st4(p.x_next + (long long)row * p.ld_x + c, v);
  if (p.acc_out) {
    float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
    if (p.acc_in) a = *reinterpret_cast<const float4*>(p.acc_in + (long long)row * p.ld_acc + c);
    st4(p.acc_out + (long long)row * p.ld_acc + c,
        make_float4((a.x + v.x) * p.acc_scale, (a.y + v.y) * p.acc_scale, (a.z + v.z) * p.acc_scale, (a.w + v.w) * p.acc_scale));
  }
}

// LightGAT + push: a finished row travels unnormalised (relative to its own max m) with its softmax state (m, l); the owner merges the
// P slots (b200rec_peer_reduce_softmax) and divides by the merged denominator
__device__ __forceinline__ void push_softmax_state(const SpmmParams& p, int row, float m, float l) {
  const int o = row / p.push_rpp;
  *reinterpret_cast<float2*>(reinterpret_cast<float*>(p.push_dst[o]) + p.push_ml_off + 2ll * (row - o * p.push_rpp)) = make_float2(m, l);
}

template <typename T> struct Lane16;
template <> struct Lane16<float> {
  static constexpr int VPL = 4;
  static __device__ __forceinline__ void fma(float (&acc)[4], float w, const uint4& raw) {
    acc[0] = fmaf(w, __uint_as_float(raw.x), acc[0]); acc[1] = fmaf(w, __uint_as_float(raw.y), acc[1]);
    acc[2] = fmaf(w, __uint_as_float(raw.z), acc[2]); acc[3] = fmaf(w, __uint_as_float(raw.w), acc[3]);
  }
};
template <> struct Lane16<__nv_bfloat16> {
  static constexpr int VPL = 8;
  static __device__ __forceinline__ void fma(float (&acc)[8], float w, const uint4& raw) {
    const unsigned r[4] = {raw.x, raw.y, raw.z, raw.w};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      acc[2 * i] = fmaf(w, __uint_as_float(r[i] << 16), acc[2 * i]);
      acc[2 * i + 1] = fmaf(w, __uint_as_float(r[i] & 0xffff0000u), acc[2 * i + 1]);
    }
  }
};

__device__ __forceinline__ uint4 ldg16(const unsigned char* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

// G lanes cooperate on one edge (each lane owns 16 bytes of the source row; G*16*NV >= row bytes), so 32/G edges
// advance per warp step.  The inner loop is branch- and predicate-free: padding / masked edges carry (source 0,
// weight 0) and lanes beyond the row width read column 0, so every load is valid and the per-edge cost is
// 2 SHFL + 1 IMAD.WIDE.U32 + 1 LDG.128 + 4 FFMA (the first version spent ~26 instructions per edge on predicated
// 64-bit address arithmetic and zero-fill moves — profiles/r01).
template <int G, int NV, typename T, bool GAT, bool PUSH = false>
__global__ void __launch_bounds__(SPMM_WARPS * 32, (NV == 1 && !GAT) ? SPMM_MIN_CTAS : 1)
spmm_chunk_kernel(const __grid_constant__ SpmmParams p) {
  constexpr int EPW = 32 / G;                       // edges per warp step
  constexpr int UN = 8;                             // warp steps whose row loads are in flight together
  constexpr int VPL = Lane16<T>::VPL;
  constexpr int STEPS = 32 / EPW;                   // warp steps per 32-edge block (= G)
  const int lane = threadIdx.x & 31;
  const int chunk = blockIdx.x * SPMM_WARPS + (threadIdx.x >> 5);
  if (chunk >= p.n_chunks) return;
  const int g = lane / G, sl = lane % G;
  const int row = __ldg(p.chunk_row + chunk);
  const int s = __ldg(p.chunk_start + chunk);
  const int slot = __ldg(p.chunk_slot + chunk);                  // (epilogue operands are fetched up front, off the critical path:
  const float dinv_row = p.dinv ? __ldg(p.dinv + row) : 1.f;     //  ncu showed the final FMUL waiting on dinv[row])
  const int e = min(s + p.chunk_size, __ldg(p.row_ptr + row + 1));
  const unsigned stride_bytes = (unsigned)(p.ld_t * (long long)sizeof(T));
  const unsigned char* base[NV];
  bool active[NV];
#pragma unroll
  for (int nv = 0; nv < NV; ++nv) {
    const int cidx = (sl + nv * G) * VPL;
    active[nv] = cidx < p.d;
    base[nv] = reinterpret_cast<const unsigned char*>(p.t) + (size_t)(active[nv] ? cidx : 0) * sizeof(T);
  }

  float acc[NV][VPL];
#pragma unroll
  for (int nv = 0; nv < NV; ++nv)
#pragma unroll
    for (int q = 0; q < VPL; ++q) acc[nv][q] = 0.f;
  float gat_m = -INFINITY, gat_l = 0.f;             // GAT: online softmax state of this chunk (warp-uniform)

  // the index stream of the NEXT 32-edge block is fetched while the rows of the current one are gathered, so the
  // (col -> row address) dependency costs one memory latency per chunk instead of one per block
  unsigned c_nx = 0u;
  float w_nx = 0.f;
  int pos_nx = 0;
  if (s + lane < e) {
    c_nx = (unsigned)__ldcs(p.col + s + lane);
    w_nx = p.w ? __ldcs(p.w + s + lane) : 1.f;
    if (p.skip_bits) pos_nx = __ldcs(p.perm + s + lane);
  }
  for (int k0 = s; k0 < e; k0 += 32) {
    const int cnt = min(32, e - k0);
    unsigned c = c_nx;
    float wv = w_nx;
    const int pos = pos_nx;
    c_nx = 0u; w_nx = 0.f;
    if (k0 + 32 + lane < e) {
      c_nx = (unsigned)__ldcs(p.col + k0 + 32 + lane);
      w_nx = p.w ? __ldcs(p.w + k0 + 32 + lane) : 1.f;
      if (p.skip_bits) pos_nx = __ldcs(p.perm + k0 + 32 + lane);
    }
    bool masked = false;
    if (p.skip_bits != nullptr && lane < cnt) masked = ((__ldg(p.skip_bits + (pos >> 5)) >> (pos & 31)) & 1u) != 0u;
    const unsigned c_raw = c;
    if (masked) { wv = 0.f; c = 0u; }
    if constexpr (GAT) {
      // softmax over the incoming edges of the row of the source scores (the destination half of the reference's
      // Linear(2d -> 1) is constant within a row and cancels in the softmax).  Masked edges (training) do not take part.
      float sc = -INFINITY;
      if (lane < cnt && !masked) sc = __ldg(p.att_src + c_raw);
      const float m_new = fmaxf(gat_m, warp_max(sc));
      float ex = 0.f;
      if (m_new != -INFINITY) {
        const float rescale = __expf(gat_m - m_new);           // gat_m == -inf -> 0
        ex = (sc == -INFINITY) ? 0.f : __expf(sc - m_new);
        gat_l = gat_l * rescale + warp_sum(ex);
#pragma unroll
        for (int nv = 0; nv < NV; ++nv)
#pragma unroll
          for (int q = 0; q < VPL; ++q) acc[nv][q] *= rescale;
        gat_m = m_new;
      }
      wv *= ex;
    }
#pragma unroll
    for (int st0 = 0; st0 < STEPS; st0 += UN) {
      if (st0 * EPW < cnt) {                                       // warp-uniform: at most UN steps of padding per chunk
        uint4 x[UN][NV];
        float ww[UN];
#pragma unroll
        for (int u = 0; u < UN; ++u) {
          const int src_lane = (st0 + u) * EPW + g;
          const unsigned cc = __shfl_sync(FULL, c, src_lane);
          ww[u] = __shfl_sync(FULL, wv, src_lane);
#pragma unroll
          for (int nv = 0; nv < NV; ++nv) {
            const unsigned char* src = base[nv] + (unsigned long long)cc * stride_bytes;
            x[u][nv] = ldg16(src);
          }
        }
#pragma unroll
        for (int u = 0; u < UN; ++u)
#pragma unroll
          for (int nv = 0; nv < NV; ++nv) Lane16<T>::fma(acc[nv], ww[u], x[u][nv]);
      }
    }
  }
  // fold the 32/G edge lanes together (fixed order)
#pragma unroll
  for (int o = G; o < 32; o <<= 1)
#pragma unroll
    for (int nv = 0; nv < NV; ++nv)
#pragma unroll
      for (int q = 0; q < VPL; ++q) acc[nv][q] += __shfl_xor_sync(FULL, acc[nv][q], o);

  if (g == 0) {
    float sc = (slot < 0 && p.dinv) ? dinv_row : 1.f;
    if constexpr (GAT && PUSH) {
      if (slot < 0) {
        sc = 1.f;
        if (sl == 0) push_softmax_state(p, row, gat_m, gat_l);
      } else if (sl == 0) { p.partials_ml[2 * slot] = gat_m; p.partials_ml[2 * slot + 1] = gat_l; }
    } else if constexpr (GAT) {
      if (slot < 0) sc = 1.f / (gat_l + 1e-16f);               // PyG softmax: exp(s - max) / (sum + 1e-16)
      else if (sl == 0) { p.partials_ml[2 * slot] = gat_m; p.partials_ml[2 * slot + 1] = gat_l; }
    }
#pragma unroll
    for (int nv = 0; nv < NV; ++nv) {
      if (!active[nv]) continue;
#pragma unroll
      for (int h = 0; h < VPL / 4; ++h) {
        const int c4 = (sl + nv * G) * VPL + 4 * h;
        const float4 v = make_float4(acc[nv][4 * h], acc[nv][4 * h + 1], acc[nv][4 * h + 2], acc[nv][4 * h + 3]);
        if (slot < 0) row_epilogue4<PUSH>(p, row, c4, sc, v);
        else if (c4 < p.d) st4(p.partials + (long long)slot * p.d + c4, v);
      }
    }
  }
}

// rows that were cut into several chunks: add the partials in a fixed order, then the same epilogue.
// One warp per row while the row has <= FIX_LONG partial slots (slots added in chunk order, 8 independent loads at a time).
// Longer rows — the few hottest items of a Zipf catalogue own thousands of chunks; one warp walking 9,800 slots was 2.0 ms of a
// 12.4 ms layer in the HBM regime — are handled by the whole CTA afterwards: warp w adds slots w, w+8, ..., the eight sums are
// combined in warp order.  Either way the order depends only on the index structure: bit-reproducible run to run.
constexpr int FIX_LONG = 64;

template <int NV, bool GAT>
__device__ __forceinline__ void fixup_accumulate(const SpmmParams& p, int first, int begin, int step, int n, int lane, float M,
                                                 float (&acc)[NV][4], float& Lsum) {
  for (int s0 = begin; s0 < n; s0 += 8 * step) {
    float4 v[8][NV];
    float f[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int sidx = s0 + k * step;
      const bool ok = sidx < n;
      f[k] = ok ? 1.f : 0.f;
      if constexpr (GAT) {
        if (ok) {
          const float ms = p.partials_ml[2 * (first + sidx)];
          const float e = (ms == -INFINITY) ? 0.f : __expf(ms - M);
          Lsum += p.partials_ml[2 * (first + sidx) + 1] * e;
          f[k] = e;
        }
      }
#pragma unroll
      for (int nv = 0; nv < NV; ++nv) {
        const int cidx = lane * 4 + nv * 128;
        v[k][nv] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cidx < p.d && ok) v[k][nv] = *reinterpret_cast<const float4*>(p.partials + (long long)(first + sidx) * p.d + cidx);
      }
    }
#pragma unroll
    for (int k = 0; k < 8; ++k)
#pragma unroll
      for (int nv = 0; nv < NV; ++nv) {
        acc[nv][0] = fmaf(v[k][nv].x, f[k], acc[nv][0]); acc[nv][1] = fmaf(v[k][nv].y, f[k], acc[nv][1]);
        acc[nv][2] = fmaf(v[k][nv].z, f[k], acc[nv][2]); acc[nv][3] = fmaf(v[k][nv].w, f[k], acc[nv][3]);
      }
  }
}

template <int NV, bool GAT, bool PUSH = false>
__global__ void __launch_bounds__(FIX_WARPS * 32)
spmm_fixup_kernel(const __grid_constant__ SpmmParams p) {
  __shared__ __align__(16) float s_acc[FIX_WARPS][NV * 128];
  __shared__ float s_red[FIX_WARPS];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  // ---- phase 1: one warp per short row ----
  {
    const int m = blockIdx.x * FIX_WARPS + warp;
    const int n = m < p.n_multi ? __ldg(p.multi_n_slots + m) : 0;
    if (n > 0 && n <= FIX_LONG) {
      const int row = __ldg(p.multi_row + m), first = __ldg(p.multi_first_slot + m);
      float acc[NV][4] = {};
      float M = -INFINITY, Lsum = 0.f;
      if constexpr (GAT) {
        for (int sidx = 0; sidx < n; ++sidx) M = fmaxf(M, p.partials_ml[2 * (first + sidx)]);
      }
      fixup_accumulate<NV, GAT>(p, first, 0, 1, n, lane, M, acc, Lsum);
      float sc;
      if constexpr (GAT && PUSH) {
        sc = 1.f;
        if (lane == 0) push_softmax_state(p, row, M, Lsum);
      } else {
        sc = GAT ? 1.f / (Lsum + 1e-16f) : (p.dinv ? __ldg(p.dinv + row) : 1.f);
      }
#pragma unroll
      for (int nv = 0; nv < NV; ++nv)
        row_epilogue4<PUSH>(p, row, lane * 4 + nv * 128, sc, make_float4(acc[nv][0], acc[nv][1], acc[nv][2], acc[nv][3]));
    }
  }
  // ---- phase 2: the CTA's long rows, one after the other, all warps on each (CTA-uniform control flow) ----
  for (int r = 0; r < FIX_WARPS; ++r) {
    const int m = blockIdx.x * FIX_WARPS + r;
    if (m >= p.n_multi) break;
    const int n = __ldg(p.multi_n_slots + m);
    if (n <= FIX_LONG) continue;
    const int row = __ldg(p.multi_row + m), first = __ldg(p.multi_first_slot + m);
    float M = -INFINITY;
    if constexpr (GAT) {
      for (int sidx = threadIdx.x; sidx < n; sidx += FIX_WARPS * 32) M = fmaxf(M, p.partials_ml[2 * (first + sidx)]);
      M = warp_max(M);
      if (lane == 0) s_red[warp] = M;
      __syncthreads();
      M = s_red[0];
#pragma unroll
      for (int w = 1; w < FIX_WARPS; ++w) M = fmaxf(M, s_red[w]);
      __syncthreads();
    }
    float acc[NV][4] = {};
    float Lsum = 0.f;
    fixup_accumulate<NV, GAT>(p, first, warp, FIX_WARPS, n, lane, M, acc, Lsum);
#pragma unroll
    for (int nv = 0; nv < NV; ++nv)
      *reinterpret_cast<float4*>(&s_acc[warp][nv * 128 + lane * 4]) = make_float4(acc[nv][0], acc[nv][1], acc[nv][2], acc[nv][3]);
    if (GAT && lane == 0) s_red[warp] = Lsum;
    __syncthreads();
    if (warp == 0) {
      float L = 0.f;
      float4 t[NV];
#pragma unroll
      for (int nv = 0; nv < NV; ++nv) t[nv] = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
      for (int w = 0; w < FIX_WARPS; ++w) {
        if (GAT) L += s_red[w];
#pragma unroll
        for (int nv = 0; nv < NV; ++nv) {
          const float4 x = *reinterpret_cast<const float4*>(&s_acc[w][nv * 128 + lane * 4]);
          t[nv].x += x.x; t[nv].y += x.y; t[nv].z += x.z; t[nv].w += x.w;
        }
      }
      float sc;
      if constexpr (GAT && PUSH) {
        sc = 1.f;
        if (lane == 0) push_softmax_state(p, row, M, L);
      } else {
        sc = GAT ? 1.f / (L + 1e-16f) : (p.dinv ? __ldg(p.dinv + row) : 1.f);
      }
#pragma unroll
      for (int nv = 0; nv < NV; ++nv) row_epilogue4<PUSH>(p, row, lane * 4 + nv * 128, sc, t[nv]);
    }
    __syncthreads();
  }
}

template <int G, int NV, typename T>
static int launch_chunks(const SpmmParams& p, cudaStream_t st) {
  const int grid = ceil_div_i(p.n_chunks, SPMM_WARPS);
  if (p.push_parts > 0 && p.att_src) spmm_chunk_kernel<G, NV, T, true, true><<<grid, SPMM_WARPS * 32, 0, st>>>(p);
  else if (p.push_parts > 0) spmm_chunk_kernel<G, NV, T, false, true><<<grid, SPMM_WARPS * 32, 0, st>>>(p);
  else if (p.att_src) spmm_chunk_kernel<G, NV, T, true><<<grid, SPMM_WARPS * 32, 0, st>>>(p);
  else spmm_chunk_kernel<G, NV, T, false><<<grid, SPMM_WARPS * 32, 0, st>>>(p);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

template <typename T>
static int launch_spmm(const SpmmParams& p, cudaStream_t st) {
  const int row_bytes = p.d * (int)sizeof(T);
  if (p.n_chunks > 0) {
    int rc;
    if (row_bytes <= 128) rc = launch_chunks<8, 1, T>(p, st);
    else if (row_bytes <= 256) rc = launch_chunks<16, 1, T>(p, st);
    else if (row_bytes <= 512) rc = launch_chunks<32, 1, T>(p, st);
    else if (row_bytes <= 1024) rc = launch_chunks<32, 2, T>(p, st);
    else if (row_bytes <= 2048 && sizeof(T) == 4) rc = launch_chunks<32, 4, T>(p, st);
    else return b200rec_fail(B200REC_ERR_UNSUPPORTED, "spmm: node_emb wider than 512");
    if (rc) return rc;
  }
  if (p.n_multi > 0) {
    const int g2 = ceil_div_i(p.n_multi, FIX_WARPS);
    if (p.push_parts > 0 && p.att_src) {
      if (p.d <= 128) spmm_fixup_kernel<1, true, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else if (p.d <= 256) spmm_fixup_kernel<2, true, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else spmm_fixup_kernel<4, true, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
    } else if (p.push_parts > 0) {
      if (p.d <= 128) spmm_fixup_kernel<1, false, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else if (p.d <= 256) spmm_fixup_kernel<2, false, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else spmm_fixup_kernel<4, false, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
    } else if (p.att_src) {
      if (p.d <= 128) spmm_fixup_kernel<1, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else if (p.d <= 256) spmm_fixup_kernel<2, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else spmm_fixup_kernel<4, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
    } else {
      if (p.d <= 128) spmm_fixup_kernel<1, false><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else if (p.d <= 256) spmm_fixup_kernel<2, false><<<g2, FIX_WARPS * 32, 0, st>>>(p);
      else spmm_fixup_kernel<4, false><<<g2, FIX_WARPS * 32, 0, st>>>(p);
    }
    B200REC_CHECK_LAUNCH();
  }
  return B200REC_OK;
}

}  // namespace b200rec

using namespace b200rec;

// the fix-up pass alone, for csrc/spmm_stream.cu (rows cut by segment boundaries; normalisation already folded into the entries)
int b200rec_spmm_fixup_launch(const float* partials, int d, const int* multi_row, const int* multi_first_slot, const int* multi_n_slots, int n_multi,
                              float* x_next, long long ld_x, const float* acc_in, float* acc_out, long long ld_acc, float acc_scale,
                              void* const* push_dst, int push_parts, int push_rpp, long long push_off, long long push_ld, cudaStream_t st) {
  if (n_multi <= 0) return B200REC_OK;
  SpmmParams p = {};
  p.d = d; p.partials = const_cast<float*>(partials); p.dinv = nullptr;
  p.multi_row = multi_row; p.multi_first_slot = multi_first_slot; p.multi_n_slots = multi_n_slots; p.n_multi = n_multi;
  p.x_next = x_next; p.ld_x = ld_x; p.acc_in = acc_in; p.acc_out = acc_out; p.ld_acc = ld_acc; p.acc_scale = acc_scale;
  p.push_parts = push_parts; p.push_rpp = push_rpp; p.push_off = push_off; p.push_ld = push_ld;
  for (int q = 0; q < B200REC_PEER_MAX; ++q) p.push_dst[q] = push_dst ? push_dst[q] : nullptr;
  const int g2 = ceil_div_i(n_multi, FIX_WARPS);
  if (push_parts > 0) spmm_fixup_kernel<1, false, true><<<g2, FIX_WARPS * 32, 0, st>>>(p);
  else spmm_fixup_kernel<1, false, false><<<g2, FIX_WARPS * 32, 0, st>>>(p);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_spmm(const b200rec_spmm_t* a, b200rec_stream_t stream) {
  if (!a) return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: null descriptor");
  if (a->d <= 0 || (a->d % 4) || a->n_chunks < 0 || a->n_multi < 0 || a->chunk_size <= 0 || (a->t_dtype == B200REC_BF16 && (a->d % 8)))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: d must be a positive multiple of 4 (fp32) / 8 (bf16)");
  if (a->n_chunks == 0) return B200REC_OK;
  if (!a->chunk_row || !a->chunk_start || !a->chunk_slot || !a->row_ptr || !a->col || !a->t)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: null index / feature pointer");
  if (a->n_multi > 0 && (!a->partials || !a->multi_row || !a->multi_first_slot || !a->multi_n_slots))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: multi-chunk rows need partials + lists");
  if (a->skip_bits && !a->perm) return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: skip bitmap needs perm");
  const int esz = a->t_dtype == B200REC_BF16 ? 2 : 4;
  if ((uintptr_t)a->t % 16 || ((a->ld_t * esz) % 16) || (a->ld_t % 4) || (a->x_next && ((uintptr_t)a->x_next % 16 || a->ld_x % 4)) ||
      (a->acc_out && ((uintptr_t)a->acc_out % 16 || a->ld_acc % 4)) || (a->acc_in && (uintptr_t)a->acc_in % 16) ||
      (a->partials && (uintptr_t)a->partials % 16))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: feature pointers / leading dims must allow 128-bit access");
  SpmmParams p;
  p.chunk_row = a->chunk_row; p.chunk_start = a->chunk_start; p.chunk_slot = a->chunk_slot;
  p.n_chunks = a->n_chunks; p.chunk_size = a->chunk_size;
  p.row_ptr = a->row_ptr; p.col = a->col; p.w = a->w; p.perm = a->perm; p.skip_bits = a->skip_bits;
  p.t = a->t; p.ld_t = a->ld_t; p.d = a->d; p.dinv = a->dinv; p.partials = a->partials;
  p.x_next = a->x_next; p.ld_x = a->ld_x; p.acc_in = a->acc_in; p.acc_out = a->acc_out; p.ld_acc = a->ld_acc;
  p.acc_scale = a->acc_scale;
  p.multi_row = a->multi_row; p.multi_first_slot = a->multi_first_slot; p.multi_n_slots = a->multi_n_slots;
  p.n_multi = a->n_multi;
  p.att_src = a->att_src; p.partials_ml = a->partials_ml;
  p.push_parts = a->push_parts; p.push_rpp = a->push_rows_per_part; p.push_off = a->push_offset; p.push_ld = a->push_ld;
  p.push_ml_off = a->push_stats_offset;
  for (int q = 0; q < B200REC_PEER_MAX; ++q) p.push_dst[q] = a->push_dst[q];
  if (p.push_parts < 0 || p.push_parts > B200REC_PEER_MAX) return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: push_parts out of range");
  if (p.push_parts > 0) {
    if (p.push_rpp <= 0 || (p.push_ld % 4) || (p.push_off % 4) || p.push_ld < p.d)
      return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: bad push arguments (offsets / leading dimension multiples of 4)");
    if (p.att_src && (p.push_ml_off <= 0 || (p.push_ml_off % 2)))
      return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: LightGAT with push needs push_stats_offset (a positive multiple of 2)");
    for (int q = 0; q < p.push_parts; ++q)
      if (!p.push_dst[q] || ((uintptr_t)p.push_dst[q] % 16)) return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: null / misaligned push destination");
  }
  if (p.att_src && p.n_multi > 0 && !p.partials_ml) return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: LightGAT needs partials_ml for multi-chunk rows");
  cudaStream_t st = (cudaStream_t)stream;
  if (a->t_dtype == B200REC_F32) return launch_spmm<float>(p, st);
  if (a->t_dtype == B200REC_BF16) return launch_spmm<__nv_bfloat16>(p, st);
  return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm: bad t_dtype");
}
