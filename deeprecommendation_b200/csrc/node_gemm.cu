// K1c — persistent short-K GEMM for the per-node transforms of GraphNCF:  Y = act((X · Wᵀ + bias) ∘ row_scale),  K <= 128, N <= 128.
//
// GraphNCF applies a d x d Linear to every node once per layer (gnn_ncf.py:91-93 applies it per EDGE; transform-before-
// gather, csrc/spmm.cu) — with d = 64/128 these GEMMs are pure streaming: 2·d·4 bytes per node against 2·d² FLOP.  The
// general tensor-core kernel (csrc/gemm_tc.cu) spends one CTA per 128-row tile: TMEM allocation, barrier set-up, a 4-k-block
// main loop and a serial epilogue — ~1 TB/s.  Here the CTA is PERSISTENT: W (TF32 hi + lo planes, the packed format of
// b200rec_pack_weights_tc) stays in shared memory, row tiles are walked with stride gridDim.x, and three roles overlap
// through mbarriers: 8 producer warps (global fp32 -> TF32 hi/lo -> swizzled smem ring), one MMA warp (3xTF32: hi·hi into a
// main accumulator, hi·lo + lo·hi into a second one), 4 epilogue warps draining the previous tile's accumulators from TMEM
// (two accumulator pairs = all 512 columns) while the next tile is produced.  fp32 parity: the same split as gemm_tc.cu.
#include "common.cuh"

namespace b200rec {

constexpr int NT_PRODUCERS = 256, NT_EPI = 128, NT_THREADS = NT_PRODUCERS + NT_EPI + 32;
constexpr int NT_TILE = 128 * 128;          // 128 rows x 128 bytes (32 TF32 of K)
constexpr int NT_STAGE = 2 * NT_TILE;       // hi + lo planes
constexpr int NT_NS = 2;                    // ring stages
constexpr int NT_STG_LD = 36;               // staging row pitch in floats (144 B: conflict-free 128-bit accesses)

__device__ __forceinline__ uint32_t nt_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void nt_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(nt_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void nt_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(nt_u32(bar)) : "memory");
}
__device__ __forceinline__ void nt_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(nt_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void nt_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "NT_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra NT_DONE;\n\t"
      "bra NT_WAIT;\n\t"
      "NT_DONE:\n\t"
      "}" ::"r"(nt_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void nt_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(nt_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(nt_u32(bar))
               : "memory");
}
__device__ __forceinline__ void nt_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void nt_tc_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void nt_tc_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void nt_umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void nt_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(nt_u32(bar)) : "memory");
}
__device__ __forceinline__ uint64_t nt_desc(uint32_t smem_addr) {      // K-major SWIZZLE_128B, as in gemm_tc.cu
  return (uint64_t)((smem_addr & 0x3ffff) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
__device__ __forceinline__ uint32_t nt_idesc() {                        // F32 accumulate, TF32 x TF32, N = 128, M = 128
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(128 >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
__device__ __forceinline__ float nt_tf32_round(float x) { return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u); }

struct NodeGemmParams {
  const float* X; long long ldx;
  int M, N, K;                         // K in {32, 64, 96, 128}, N <= 128
  const unsigned char* Wp;             // b200rec_pack_weights_tc(TF32X3) of W (N, K): [k-block][hi | lo] tiles of 16 KB
  const float* bias; const float* row_scale; int relu;
  void* Y; long long ldy; int y_bf16;   // Y: fp32, or bf16 (GraphNCF's bf16 message mode: K3 gathers half the bytes)
  // all-gather fused into the epilogue (partitioned propagation): every tile is also stored to Yx[q], q < n_extra — the same
  // place of the peer ranks' feature tables, mapped over NVLink (csrc/peer.cu)
  void* Yx[B200REC_PEER_MAX]; int n_extra;
};

template <int NKB, bool PUSH>
__global__ void __launch_bounds__(NT_THREADS, 1)
node_gemm_kernel(const __grid_constant__ NodeGemmParams p) {
  extern __shared__ unsigned char nt_smem_raw[];
  unsigned char* sm = reinterpret_cast<unsigned char*>(((uintptr_t)nt_smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned char* sm_w = sm;                                   // NKB * 32 KB
  unsigned char* sm_ring = sm + NKB * NT_STAGE;               // NT_NS * 32 KB
  float* sm_bias = reinterpret_cast<float*>(sm_ring + NT_NS * NT_STAGE);   // 128 floats
  float* sm_stage = sm_bias + 128;                                         // 4 warps x 32 rows x NT_STG_LD floats
  __shared__ __align__(8) uint64_t w_bar, a_full[NT_NS], a_empty[NT_NS], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_base_smem;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int n_tiles = (p.M + 127) >> 7;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < NT_NS; ++s) { nt_mbar_init(&a_full[s], NT_PRODUCERS); nt_mbar_init(&a_empty[s], 1); }
#pragma unroll
    for (int s = 0; s < 2; ++s) { nt_mbar_init(&acc_full[s], 1); nt_mbar_init(&acc_empty[s], NT_EPI); }
    nt_mbar_init(&w_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 12) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(nt_u32(&tmem_base_smem)), "r"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid < 128) sm_bias[tid] = (p.bias != nullptr && tid < p.N) ? __ldg(p.bias + tid) : 0.f;
  nt_tc_before();
  __syncthreads();
  nt_tc_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (tid == 0) {
    nt_mbar_expect_tx(&w_bar, NKB * NT_STAGE);
#pragma unroll
    for (int t = 0; t < NKB * 2; ++t) nt_bulk_g2s(sm_w + t * NT_TILE, p.Wp + (size_t)t * NT_TILE, NT_TILE, &w_bar);
  }

  if (warp < 8) {
    // ===================== producers =====================
    // thread = (16-byte chunk c of the 128-byte k-block row, row r0 + 32 it): coalesced 128-bit loads, 4 rows per thread
    const int c = tid & 7, r0 = tid >> 3;
    uint32_t soff[4];
#pragma unroll
    for (int it = 0; it < 4; ++it) {
      const int r = r0 + 32 * it;
      soff[it] = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + (uint32_t)((c ^ (r & 7)) << 4);
    }
    // register buffer k holds k-block k of the current tile and is refilled with the NEXT tile's k-block k right after it
    // has been converted: a whole tile (64 KB at K = 128) of loads is always in flight per CTA with 16 registers per k-block
    float4 cur[NKB][4];
    auto load_kb = [&](float4 (&dst)[4], int tile, int kb) {
#pragma unroll
      for (int it = 0; it < 4; ++it) {
        const int row = min(tile * 128 + r0 + 32 * it, p.M - 1);
        dst[it] = __ldg(reinterpret_cast<const float4*>(p.X + (long long)row * p.ldx + kb * 32 + c * 4));
      }
    };
    int tile = blockIdx.x;
    if (tile < n_tiles) {
#pragma unroll
      for (int kb = 0; kb < NKB; ++kb) load_kb(cur[kb], tile, kb);
    }
    uint32_t cnt = 0;
    for (; tile < n_tiles; tile += gridDim.x) {
      const int next = tile + gridDim.x;
#pragma unroll
      for (int kb = 0; kb < NKB; ++kb) {
        const uint32_t s = cnt % NT_NS, ph = (cnt / NT_NS) & 1u;
        nt_mbar_wait(&a_empty[s], ph ^ 1u);
        unsigned char* st = sm_ring + (size_t)s * NT_STAGE;
#pragma unroll
        for (int it = 0; it < 4; ++it) {
          const float4 x = cur[kb][it];
          const float4 hi = make_float4(nt_tf32_round(x.x), nt_tf32_round(x.y), nt_tf32_round(x.z), nt_tf32_round(x.w));
          *reinterpret_cast<float4*>(st + soff[it]) = hi;
          *reinterpret_cast<float4*>(st + NT_TILE + soff[it]) = make_float4(x.x - hi.x, x.y - hi.y, x.z - hi.z, x.w - hi.w);
        }
        nt_fence_async();
        nt_mbar_arrive(&a_full[s]);
        ++cnt;
        if (next < n_tiles) load_kb(cur[kb], next, kb);
      }
    }
  } else if (warp < 12) {
    // ===================== epilogue: (main + cross + bias) * row_scale, ReLU, store =====================
    const int e = warp - 8;
    uint32_t t = 0;
    for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
      const uint32_t acc = t & 1u;
      nt_mbar_wait(&acc_full[acc], (t >> 1) & 1u);
      nt_tc_after();
      const int row = tile * 128 + e * 32 + lane;
      const float rs = (p.row_scale != nullptr && row < p.M) ? __ldg(p.row_scale + row) : 1.f;
#pragma unroll
      for (int cg = 0; cg < 4; ++cg) {
        uint32_t a[32], b[32];
        const uint32_t taddr = tmem_base + ((uint32_t)(e * 32) << 16) + acc * 256 + cg * 32;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(a[0]), "=r"(a[1]), "=r"(a[2]), "=r"(a[3]), "=r"(a[4]), "=r"(a[5]), "=r"(a[6]), "=r"(a[7]), "=r"(a[8]), "=r"(a[9]),
              "=r"(a[10]), "=r"(a[11]), "=r"(a[12]), "=r"(a[13]), "=r"(a[14]), "=r"(a[15]), "=r"(a[16]), "=r"(a[17]), "=r"(a[18]),
              "=r"(a[19]), "=r"(a[20]), "=r"(a[21]), "=r"(a[22]), "=r"(a[23]), "=r"(a[24]), "=r"(a[25]), "=r"(a[26]), "=r"(a[27]),
              "=r"(a[28]), "=r"(a[29]), "=r"(a[30]), "=r"(a[31])
            : "r"(taddr)
            : "memory");
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
            "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
            "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
            : "=r"(b[0]), "=r"(b[1]), "=r"(b[2]), "=r"(b[3]), "=r"(b[4]), "=r"(b[5]), "=r"(b[6]), "=r"(b[7]), "=r"(b[8]), "=r"(b[9]),
              "=r"(b[10]), "=r"(b[11]), "=r"(b[12]), "=r"(b[13]), "=r"(b[14]), "=r"(b[15]), "=r"(b[16]), "=r"(b[17]), "=r"(b[18]),
              "=r"(b[19]), "=r"(b[20]), "=r"(b[21]), "=r"(b[22]), "=r"(b[23]), "=r"(b[24]), "=r"(b[25]), "=r"(b[26]), "=r"(b[27]),
              "=r"(b[28]), "=r"(b[29]), "=r"(b[30]), "=r"(b[31])
            : "r"(taddr + 128)
            : "memory");
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
        if (cg == 3) {                                           // both accumulators read: hand the pair back
          nt_tc_before();
          nt_mbar_arrive(&acc_empty[acc]);
        }
        // through a per-warp staging tile so that the global stores are full 128-byte lines: a warp instruction writes
        // 4 rows x 32 columns instead of 32 rows x 4 columns (measured: 58 -> 36 us without the 16-byte-per-row stores)
        float* stg = sm_stage + e * (32 * NT_STG_LD);
#pragma unroll
        for (int j = 0; j < 32; j += 4) {
          const int n = cg * 32 + j;
          float o[4];
#pragma unroll
          for (int q = 0; q < 4; ++q) {
            const float v = (__uint_as_float(a[j + q]) + __uint_as_float(b[j + q]) + sm_bias[n + q]) * rs;
            o[q] = p.relu ? fmaxf(v, 0.f) : v;
          }
          *reinterpret_cast<float4*>(stg + lane * NT_STG_LD + j) = make_float4(o[0], o[1], o[2], o[3]);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int r = i * 4 + (lane >> 3), cc = (lane & 7) * 4;
          const int grow = tile * 128 + e * 32 + r, n = cg * 32 + cc;
          if (grow < p.M && n < p.N) {
            const float4 v = *reinterpret_cast<const float4*>(stg + r * NT_STG_LD + cc);
            const int n_dst = PUSH ? p.n_extra + 1 : 1;           // PUSH: the peers' copies of the table (NVLink stores) after the local one
#pragma unroll 1
            for (int dq = 0; dq < n_dst; ++dq) {
              void* const Yq = (!PUSH || dq == 0) ? p.Y : p.Yx[dq - 1];
              if (p.y_bf16) {                                      // 4 rows x 64 bytes per warp instruction
                __nv_bfloat16* d = reinterpret_cast<__nv_bfloat16*>(Yq) + (long long)grow * p.ldy + n;
                if (n + 3 < p.N && (((uintptr_t)d & 7) == 0)) {
                  const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
                  *reinterpret_cast<uint2*>(d) = make_uint2(*reinterpret_cast<const unsigned*>(&lo), *reinterpret_cast<const unsigned*>(&hi));
                } else {
                  const float o[4] = {v.x, v.y, v.z, v.w};
                  for (int q = 0; q < 4 && n + q < p.N; ++q) d[q] = __float2bfloat16_rn(o[q]);
                }
                continue;
              }
              float* d = reinterpret_cast<float*>(Yq) + (long long)grow * p.ldy + n;
              if (n + 3 < p.N && (((uintptr_t)d & 15) == 0)) *reinterpret_cast<float4*>(d) = v;
              else {
                const float o[4] = {v.x, v.y, v.z, v.w};
                for (int q = 0; q < 4 && n + q < p.N; ++q) d[q] = o[q];
              }
            }
          }
        }
        __syncwarp();
      }
    }
  } else {
    // ===================== MMA issuer =====================
    if (lane == 0) {
      const uint32_t idesc = nt_idesc();
      nt_mbar_wait(&w_bar, 0);
      uint32_t cnt = 0, t = 0;
      for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x, ++t) {
        const uint32_t acc = t & 1u;
        nt_mbar_wait(&acc_empty[acc], ((t >> 1) & 1u) ^ 1u);
        nt_tc_after();
        const uint32_t d_main = tmem_base + acc * 256, d_cross = d_main + 128;
#pragma unroll
        for (int kb = 0; kb < NKB; ++kb) {
          const uint32_t s = cnt % NT_NS, ph = (cnt / NT_NS) & 1u;
          nt_mbar_wait(&a_full[s], ph);
          nt_tc_after();
          const uint32_t a_hi = nt_u32(sm_ring + (size_t)s * NT_STAGE), a_lo = a_hi + NT_TILE;
          const uint32_t w_hi = nt_u32(sm_w + (size_t)kb * NT_STAGE), w_lo = w_hi + NT_TILE;
#pragma unroll
          for (int ks = 0; ks < 4; ++ks) {                       // 8 TF32 (32 bytes) of K per MMA
            const uint32_t off = (uint32_t)ks * 32u;
            const uint32_t first = (kb > 0 || ks > 0) ? 1u : 0u;
            nt_umma_tf32(d_main, nt_desc(a_hi + off), nt_desc(w_hi + off), idesc, first);     // hi · hi
            nt_umma_tf32(d_cross, nt_desc(a_hi + off), nt_desc(w_lo + off), idesc, first);    // hi · lo
            nt_umma_tf32(d_cross, nt_desc(a_lo + off), nt_desc(w_hi + off), idesc, 1u);       // lo · hi
          }
          nt_commit(&a_empty[s]);
          ++cnt;
        }
        nt_commit(&acc_full[acc]);
      }
    }
    __syncwarp();
  }
  nt_tc_before();
  __syncthreads();
  if (warp == 12) {
    nt_tc_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

template <int NKB, bool PUSH>
static int nt_launch(const NodeGemmParams& p, cudaStream_t st) {
  const size_t smem = (size_t)NKB * NT_STAGE + NT_NS * NT_STAGE + 512 + 4 * 32 * NT_STG_LD * 4 + 1024;
  static B200recSmemOptIn opted;
  B200REC_CUDA(b200rec_opt_in_smem(opted, node_gemm_kernel<NKB, PUSH>, (int)smem));
  const int n_tiles = (p.M + 127) / 128;
  const int sms = b200rec_num_sms();
  // persistent grid: every CTA gets the same number of tiles where possible (waves of `sms`)
  const int waves = (n_tiles + sms - 1) / sms;
  const int grid = (n_tiles + waves - 1) / waves;
  node_gemm_kernel<NKB, PUSH><<<grid, NT_THREADS, smem, st>>>(p);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

}  // namespace b200rec

using namespace b200rec;

static int shortk_run(const float* X, int64_t M, int64_t K, int64_t ldx, const void* packed_w, int64_t N, const float* bias,
                      const float* row_scale, int relu, void* Y, void* const* extra, int n_extra, int64_t ldy, int y_dtype,
                      b200rec_stream_t stream) {
  if (M < 0 || !packed_w || !Y || (M > 0 && !X)) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_shortk: null operand");
  if (K <= 0 || K > 128 || (K % 32) || N <= 0 || N > 128) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "linear_shortk: needs K in {32,64,96,128}, N <= 128");
  if (ldx < K || ldy < N || (ldx % 4) || ((uintptr_t)X % 16) || ((uintptr_t)packed_w % 128))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_shortk: X rows must be 16-byte aligned (ldx % 4 == 0), packed W 128-byte aligned");
  if (M > INT32_MAX) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "linear_shortk: M > int32");
  if (y_dtype != B200REC_F32 && y_dtype != B200REC_BF16) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_shortk: bad y_dtype");
  if (M == 0) return B200REC_OK;
  NodeGemmParams p;
  p.X = X; p.ldx = ldx; p.M = (int)M; p.N = (int)N; p.K = (int)K; p.Wp = (const unsigned char*)packed_w;
  p.bias = bias; p.row_scale = row_scale; p.relu = relu; p.Y = Y; p.ldy = ldy; p.y_bf16 = y_dtype == B200REC_BF16;
  p.n_extra = n_extra;
  for (int q = 0; q < B200REC_PEER_MAX; ++q) p.Yx[q] = q < n_extra ? extra[q] : nullptr;
  cudaStream_t st = (cudaStream_t)stream;
  if (n_extra > 0) {
    switch (K / 32) {
      case 1: return nt_launch<1, true>(p, st);
      case 2: return nt_launch<2, true>(p, st);
      case 3: return nt_launch<3, true>(p, st);
      default: return nt_launch<4, true>(p, st);
    }
  }
  switch (K / 32) {
    case 1: return nt_launch<1, false>(p, st);
    case 2: return nt_launch<2, false>(p, st);
    case 3: return nt_launch<3, false>(p, st);
    default: return nt_launch<4, false>(p, st);
  }
}

extern "C" int b200rec_linear_shortk(const float* X, int64_t M, int64_t K, int64_t ldx, const void* packed_w, int64_t N, const float* bias,
                                     const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, b200rec_stream_t stream) {
  return shortk_run(X, M, K, ldx, packed_w, N, bias, row_scale, relu, Y, nullptr, 0, ldy, y_dtype, stream);
}

extern "C" int b200rec_linear_shortk_push(const float* X, int64_t M, int64_t K, int64_t ldx, const void* packed_w, int64_t N, const float* bias,
                                          const float* row_scale, int relu, void* const* dst, int n_dst, int64_t y_offset, int64_t ldy,
                                          int y_dtype, b200rec_stream_t stream) {
  if (!dst || n_dst <= 0 || n_dst > B200REC_PEER_MAX) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_shortk_push: 1..B200REC_PEER_MAX destinations");
  const int64_t esz = y_dtype == B200REC_BF16 ? 2 : 4;
  void* d[B200REC_PEER_MAX];
  for (int q = 0; q < n_dst; ++q) {
    if (!dst[q]) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_shortk_push: null destination");
    d[q] = static_cast<unsigned char*>(dst[q]) + y_offset * esz;
  }
  return shortk_run(X, M, K, ldx, packed_w, N, bias, row_scale, relu, d[0], d + 1, n_dst - 1, ldy, y_dtype, stream);
}
