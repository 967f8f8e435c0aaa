// K1a on the 5th-generation tensor cores:  Y = act((X · Wᵀ + bias) ∘ row_scale)  with tcgen05.mma + TMEM accumulators.
//
// Why X is NOT moved by a TMA tensor map: the reference's profile width F = 2094 makes row pitches of 8376 bytes — not a
// multiple of 16, which cuTensorMapEncodeTiled requires — and X arrives as fp32 while the MMA wants bf16 or a
// TF32 hi/lo split.  So eight producer warps read X with 64-bit loads, convert in registers and write the tiles
// straight into the canonical K-major SWIZZLE_128B shared-memory layout (16-byte chunk c of row r lives at chunk c^(r&7)
// of its 128-byte row; 8-row groups are 1024 B apart), publish them to the async proxy with fence.proxy.async and an
// mbarrier, and one elected thread of a ninth warp issues the MMAs.  W is converted once into that layout
// (b200rec_pack_weights_tc) and moved by TMA bulk copies.  Every X byte is read once as fp32.
//
// Two arithmetic modes on the same skeleton:
//   TC_TF32X3 (fp32 parity, default): x = hi + lo with hi = round-to-TF32(x); D += A_hi·B_hi + A_hi·B_lo + A_lo·B_hi
//             (kind::tf32, fp32 accumulate in TMEM).  The dropped lo·lo term and the truncation of lo are ~2^-21
//             relative, i.e. inside the reference tolerance rel <= 1e-5.
//   TC_BF16   (bf16 mode, rel <= 1e-2): one kind::f16 MMA per k-step on bf16-rounded operands.
//   TC_BF16X3 (wide form only): x = hi + lo with hi = bf16(x), lo = bf16(x - hi); the same three products in kind::f16.  Twice the MMA rate
//             of TF32 and half the operand bytes per k, at 16 instead of 21 mantissa bits per operand: ~4e-6 relative to the largest
//             output at K = 2094 (measured), still inside the 1e-5 budget.  Opt-in (`engine='bf16x3'`).
//
// CTA = 128 (M) x 128 (N) output tile, accumulator = 128 TMEM columns x 128 lanes (fp32), NSTAGE-deep smem ring.
// Warp roles: warps 0-7 producers, then epilogue (tcgen05.ld 32x32b: warp w reads TMEM lanes 32*(w%4).., columns
// 64*(w/4)..); warp 8 allocates TMEM and issues tcgen05.mma / tcgen05.commit.
#include "common.cuh"

namespace b200rec {

enum { TC_TF32X3 = 0, TC_BF16 = 1, TC_BF16X3 = 2 };
// element width and number of operand planes of a mode
template <int MODE> struct TcMode {
  static constexpr bool E16 = MODE != TC_TF32X3;            // bf16 elements (64 per 128-byte swizzle row), kind::f16
  static constexpr int KB = E16 ? 64 : 32;                  // source elements per k-block
  static constexpr int PLANES = MODE == TC_BF16 ? 1 : 2;    // hi [, lo]
};
static inline int tc_kb(int mode) { return mode == TC_TF32X3 ? 32 : 64; }
static inline int tc_planes(int mode) { return mode == TC_BF16 ? 1 : 2; }

constexpr int TC_BM = 128, TC_BN = 128;
#ifndef TC_PF16
#define TC_PF16 1                                   // k-blocks of 64 in flight ahead of the store in the bf16 modes
#endif
constexpr int TC_PRODUCERS = 256;                 // 8 warps
constexpr int TC_THREADS = TC_PRODUCERS + 32;     // + MMA warp
constexpr int TILE_BYTES = 128 * 128;             // one operand tile: 128 rows x 128 bytes

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "LAB_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra LAB_DONE;\n\t"
      "bra LAB_WAIT;\n\t"
      "LAB_DONE:\n\t"
      "}" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// TMA bulk copy global -> shared (1-D, UBLKCP); completion is signalled on the mbarrier as transaction bytes
__device__ __forceinline__ void tma_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

template <int MODE>
__device__ __forceinline__ void umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  if constexpr (TcMode<MODE>::E16) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  } else {
    asm volatile(
        "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
  }
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address >> 4 in [0,14),
// LBO (unused for swizzled K-major) = 1 in [16,30), SBO = 1024 B >> 4 in [32,46), version = 1 in [46,48),
// layout_type = 2 (SWIZZLE_128B) in [61,64).
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3ffff) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (1) at [4,6), a/b format at [7,10)/[10,13)
// (BF16 = 1, TF32 = 2), both K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29).
template <int MODE, int BN = TC_BN>
__device__ __forceinline__ uint32_t make_idesc() {
  const uint32_t fmt = TcMode<MODE>::E16 ? 1u : 2u;
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(TC_BM >> 4) << 24);
}

__device__ __forceinline__ float tf32_round(float x) {
  // round-to-nearest (ties away) on the 13 dropped mantissa bits; inf/nan pass through unchanged enough for our inputs
  return __uint_as_float((__float_as_uint(x) + 0x1000u) & 0xffffe000u);
}

struct TcParams {
  const float* X; long long ldx;
  int M, N, K;
  void* Y; long long ldy; int y_bf16;
  const float* bias; const float* row_scale; int relu;
  const unsigned char* Wp;   // W pre-packed by pack_weights_kernel (swizzled tiles), moved by TMA bulk copies
  const long long* row_index;   // optional: row m of the GEMM is row row_index[m] of X (resident profile table + ids)
  // split-K (b200rec_linear_tc_splitk): CTA z = blockIdx.z owns k-blocks [z*kb_per_split, ...) and writes its raw fp32 tile to
  // partial[z] (M x N, ld N); bias / scale / activation are applied by tc_splitk_reduce_kernel.  0 = the whole K in one CTA.
  int kb_per_split;
  float* partial;
};

// Several GEMMs of the same K and mode in ONE launch (b200rec_linear_tc_batch): problem q owns the m-tiles
// [tile_start[q], tile_start[q+1]) of grid.y.  The scoring path is a chain of short GEMMs (candidate and rated-item
// projections share their weights; the two halves of AttentionNet.0 share their shape): one launch instead of four.
constexpr int TC_MAX_BATCH = 4;
struct TcBatch {
  TcParams prob[TC_MAX_BATCH];
  int tile_start[TC_MAX_BATCH + 1];
  int n;
};

// One operand tile (128 rows x KB fp32 source elements) -> smem by the 256 producer threads, COALESCED: a warp owns 16
// consecutive rows; in one load instruction its lanes cover 32/LPR rows x KB contiguous floats (EPL = 2 or 4 floats per
// lane, LPR = KB/EPL lanes per row).  Everything that does not depend on the k-block — clamped global row offsets, the
// swizzled shared-memory offsets, the row-validity bits — is computed ONCE per thread (TileAddr); per k-block a load costs
// IADD + IMAD.WIDE + LDG and a store LOP/FADD + STS.  History (profiles/r01/gemm_tc_notes.md): half-row-per-thread loads
// sat on the L1 tag stage; per-load bounds branches made ptxas wrap every LDG in BSSY/BSYNC; recomputing addresses in the
// loop cost ~1200 instructions per thread and k-block.
// (x0, x1) -> packed bf16 pairs hi = bf16(x), lo = bf16(x - hi): 2 F2FP + 2 bit ops + 2 FADD (the __nv_bfloat162 helpers cost a re-pack per pair)
__device__ __forceinline__ void bf16_split2(float x0, float x1, uint32_t& hi, uint32_t& lo) {
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(hi) : "f"(x1), "f"(x0));          // upper half = x1, lower half = x0
  const float h0 = __uint_as_float(hi << 16), h1 = __uint_as_float(hi & 0xffff0000u);
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(lo) : "f"(x1 - h1), "f"(x0 - h0));
}
__device__ __forceinline__ void sts32(uint32_t a, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts64(uint32_t a, uint32_t v0, uint32_t v1) {
  asm volatile("st.shared.v2.b32 [%0], {%1, %2};" ::"r"(a), "r"(v0), "r"(v1) : "memory");
}
__device__ __forceinline__ void sts128(uint32_t a, uint32_t v0, uint32_t v1, uint32_t v2, uint32_t v3) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v0), "r"(v1), "r"(v2), "r"(v3) : "memory");
}

// Round 2 (profiles/r02/ncu_full_gemm_bf16x3_v1.txt): the producers, not the loads, set the pace — ~35 instructions per (row, lane) and
// k-block, two warps per scheduler.  Three changes took that to ~12: (1) shared-memory stores are `st.shared` on 32-bit addresses (the generic
// 64-bit `ST` form kept a pointer pair per row and plane in registers); the swizzled offset of row `it` is a compile-time constant plus one of
// 8 / RPI run-time XOR terms (`xk`), because row r = 16·warp + it·RPI + sub has r & 7 = ((it·RPI) & 7) | sub with disjoint bits; (2) no row
// mask: rows past M are clamped at load time and only ever reach accumulator rows that are never written; (3) the k mask runs in the one
// k-block that crosses K (`store<true>`), every other block stores unmasked.
template <int MODE, int EPL>
struct TileAddr {
  static constexpr int KB = TcMode<MODE>::KB;
  static constexpr int LPR = KB / EPL, RPI = 32 / LPR, ITER = 16 / RPI;
  static constexpr int NX = (8 / RPI) > 0 ? (8 / RPI) : 1;   // distinct (it·RPI) & 7 values
  unsigned goff[ITER];        // element offset of (clamped row, this lane's first column at k = 0)
  unsigned xk[NX];            // tile-relative byte offset of this lane's chunk for every XOR term, + the lane's fixed part
  int kcol;                   // this lane's first column inside a k-block

  __device__ __forceinline__ void init(long long ld, int row0, int rows_total, int warp, int lane, const long long* row_index = nullptr) {
    kcol = (lane % LPR) * EPL;
    const unsigned byte = (unsigned)kcol * (TcMode<MODE>::E16 ? 2u : 4u);
    const unsigned sub = (unsigned)(lane / LPR);
#pragma unroll
    for (int it = 0; it < ITER; ++it) {
      const int grow = row0 + warp * 16 + it * RPI + (int)sub;
      const int crow = min(grow, rows_total - 1);
      const long long srow = row_index ? __ldg(row_index + crow) : (long long)crow;
      goff[it] = (unsigned)(srow * ld) + (unsigned)kcol;
    }
    const unsigned fixed = (unsigned)warp * 2048u + sub * 128u + (byte & 15u);
#pragma unroll
    for (int x = 0; x < NX; ++x) xk[x] = fixed + ((((byte >> 4) ^ sub) ^ (unsigned)((x * RPI) & 7)) << 4);
  }
  // byte offset of row `it` of this lane inside a 128 x 128-byte swizzled tile (`it` is a compile-time constant after unrolling)
  __device__ __forceinline__ unsigned soff(int it) const {
    return xk[it % NX] + (unsigned)(((it * RPI) >> 3) * 1024 + ((it * RPI) & 7) * 128);
  }
};

template <int MODE, int EPL>
struct TileRegs {
  using Addr = TileAddr<MODE, EPL>;
  static constexpr int ITER = Addr::ITER;
  float v[ITER][EPL];
  bool k_ok;

  // vector path: K % EPL == 0 (launcher), so a vector is entirely inside or outside [0, K)
  template <bool VEC>
  __device__ __forceinline__ void load(const float* __restrict__ src, const Addr& a, int k0, int K) {
    const int k = k0 + a.kcol;
    k_ok = k < K;
    if constexpr (VEC) {
      const float* srck = src + (k_ok ? (unsigned)k0 : 0u);   // out-of-range columns re-read k-block 0 and are zeroed at store time
#pragma unroll
      for (int it = 0; it < ITER; ++it) {
        const float* p = srck + a.goff[it];
        if constexpr (EPL == 4) {
          const float4 t = __ldg(reinterpret_cast<const float4*>(p));
          v[it][0] = t.x; v[it][1] = t.y; v[it][2] = t.z; v[it][3] = t.w;
        } else {
          const float2 t = __ldg(reinterpret_cast<const float2*>(p));
          v[it][0] = t.x; v[it][1] = t.y;
        }
      }
    } else {
#pragma unroll
      for (int it = 0; it < ITER; ++it) {
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
          const bool ok = k + e < K;
          const float t = __ldg(src + (a.goff[it] + (ok ? (unsigned)(k0 + e) : 0u)));
          v[it][e] = ok ? t : 0.f;
        }
      }
      k_ok = true;
    }
  }

  // MASK: this k-block crosses K — lanes past the end store zeros (uniform per CTA and k-block; false everywhere else)
  template <bool MASK>
  __device__ __forceinline__ void store(uint32_t tile_hi, uint32_t tile_lo, const Addr& a) const {
#pragma unroll
    for (int it = 0; it < ITER; ++it) {
      float x[EPL];
#pragma unroll
      for (int e = 0; e < EPL; ++e) x[e] = (!MASK || k_ok) ? v[it][e] : 0.f;
      const uint32_t so = a.soff(it);
      if constexpr (MODE == TC_BF16) {
        __nv_bfloat162 b0 = __floats2bfloat162_rn(x[0], x[1]);
        if constexpr (EPL == 4) {
          __nv_bfloat162 b1 = __floats2bfloat162_rn(x[2], x[3]);
          sts64(tile_hi + so, *reinterpret_cast<uint32_t*>(&b0), *reinterpret_cast<uint32_t*>(&b1));
        } else {
          sts32(tile_hi + so, *reinterpret_cast<uint32_t*>(&b0));
        }
      } else if constexpr (MODE == TC_BF16X3) {
        uint32_t h[EPL / 2], l[EPL / 2];
#pragma unroll
        for (int e = 0; e < EPL; e += 2) bf16_split2(x[e], x[e + 1], h[e / 2], l[e / 2]);
        if constexpr (EPL == 4) {
          sts64(tile_hi + so, h[0], h[1]);
          sts64(tile_lo + so, l[0], l[1]);
        } else {
          sts32(tile_hi + so, h[0]);
          sts32(tile_lo + so, l[0]);
        }
      } else {
        float hi[EPL], lo[EPL];
#pragma unroll
        for (int e = 0; e < EPL; ++e) {
          hi[e] = tf32_round(x[e]);
          lo[e] = x[e] - hi[e];
        }
        if constexpr (EPL == 4) {
          sts128(tile_hi + so, __float_as_uint(hi[0]), __float_as_uint(hi[1]), __float_as_uint(hi[2]), __float_as_uint(hi[3]));
          sts128(tile_lo + so, __float_as_uint(lo[0]), __float_as_uint(lo[1]), __float_as_uint(lo[2]), __float_as_uint(lo[3]));
        } else {
          sts64(tile_hi + so, __float_as_uint(hi[0]), __float_as_uint(hi[1]));
          sts64(tile_lo + so, __float_as_uint(lo[0]), __float_as_uint(lo[1]));
        }
      }
    }
  }
};

// BN = 256 ("wide" form, b200rec_linear_tc_wide): one CTA owns 128 rows x 256 columns, so every X block is loaded, split into TF32
// hi / lo and written to shared memory ONCE for both halves of W (the BN = 128 grid does that work twice, and the producers — not
// the tensor pipe — set the pace of a k-block: profiles/r01/gemm_tc_notes.md).  A stage is X (32 KB) + two packed W tiles (64 KB);
// two stages fit.  TMEM holds two 256-column accumulators (hi·hi | cross terms); the wide form always runs split-K, which keeps the
// accumulate chains short (see NACC below) and fills the device when M / 128 alone does not.
// Measured and dropped (round 2, profiles/r02/gemm_pair_ncu_v1.log): launching the two k-splits of a tile as a thread-block cluster so that split 0
// can wait for split 1's tile and finish the output itself (no second slab, no reduction kernel).  Both ways of handing the tile over lost:
// through distributed shared memory (~21 B/clk: +7 us), and through L2 with only the cluster barrier as the signal — the cluster launch of
// these 193 KB CTAs takes the kernel from 30 us to 49 us.  A third form without clusters — tickets from a per-tile semaphore, the first split
// to finish leaves its tile in one slab, the second adds it from L2 and completes the output — measured 46 us: only half of the CTAs take part in
// that tail, eight warps each, whereas tc_splitk_reduce_kernel streams the two slabs with every SM (8 us).  The separate reduction stays.
template <int MODE, int NSTAGE, int EPL, bool VEC, int BN = TC_BN>
__global__ void __launch_bounds__(TC_THREADS, 1)
gemm_tc_kernel(const __grid_constant__ TcBatch batch) {
  int q = 0;
#pragma unroll
  for (int t = 1; t < TC_MAX_BATCH; ++t)
    if (t < batch.n && (int)blockIdx.y >= batch.tile_start[t]) q = t;
  const TcParams& p = batch.prob[q];
  if ((int)blockIdx.x * BN >= p.N) return;                      // this problem has fewer n-tiles than the widest of the batch
  constexpr int KB = TcMode<MODE>::KB;
  constexpr int PLANES = TcMode<MODE>::PLANES;
  constexpr int NT = BN / 128;                                  // packed 128-row W tiles per stage
  constexpr int A_BYTES = PLANES * TILE_BYTES;
  constexpr int STAGE_BYTES = A_BYTES + NT * PLANES * TILE_BYTES;   // A (hi[,lo]) + B (hi[,lo]) x NT
  constexpr int UMMA_K_BYTES = 32;                              // 16 bf16 or 8 tf32 per MMA
  // The tensor core adds into the fp32 accumulator with truncation; over K = 2094 (786 accumulate steps in TF32x3) that
  // alone costs 1.3e-5 (measured).  TF32x3 therefore spreads the work over FOUR TMEM accumulators — hi·hi alternates
  // between two per k-block, the small cross terms go to two more — and the epilogue adds them in registers.  The wide form has
  // room for two (512 TMEM columns): hi·hi | cross terms; its k range is split over CTAs, ~130 accumulate steps per chain.
  constexpr int NACC = (MODE == TC_BF16) ? 1 : (BN == 256 ? 2 : 4);
  constexpr int TMEM_COLS = BN * NACC;
  extern __shared__ unsigned char smem_dyn[];
  // SWIZZLE_128B needs 1024-byte aligned tiles
  unsigned char* tiles = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
  __shared__ __align__(8) uint64_t full_bar[NSTAGE], empty_bar[NSTAGE], accum_bar;
  __shared__ uint32_t tmem_base_smem;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int m0 = ((int)blockIdx.y - batch.tile_start[q]) * TC_BM, n0 = blockIdx.x * BN;
  const int num_kb_total = (p.K + KB - 1) / KB;
  const int kb_base = p.kb_per_split ? (int)blockIdx.z * p.kb_per_split : 0;
  const int num_kb = p.kb_per_split ? min(p.kb_per_split, num_kb_total - kb_base) : num_kb_total;
  const int kb_shift = (int)((blockIdx.y * 7u + blockIdx.x * 3u + blockIdx.z) % (unsigned)num_kb);

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < NSTAGE; ++s) {
      mbar_init(&full_bar[s], TC_PRODUCERS / 32 + 1);   // one arrive per producer warp + the expect_tx arrive of the W bulk copy
      mbar_init(&empty_bar[s], 1);
    }
    mbar_init(&accum_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 8) {   // TMEM: 128 columns per fp32 accumulator (128 lanes x 128 columns)
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_base_smem)), "r"(TMEM_COLS) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (warp < 8) {
    // ===================== producers =====================
    // k-blocks are walked from a per-CTA offset (wrapping around): all CTAs of a wave would otherwise ask L2 for the
    // SAME W tile at the same moment.  The set of products accumulated is unchanged.
    // k-blocks of global loads in flight ahead of the store.  ncu (profiles/r01/ncu_full_gemm_tc_v3.txt, source page): 27 % of the
    // stall samples sat on the first use of the loaded registers (long scoreboard) with 2 k-blocks ahead.
    constexpr int PF = (MODE == TC_TF32X3) ? 2 : TC_PF16;    // (TF32: 3 and 4 were measured: register spills, 5-100 % slower)
    TileAddr<MODE, EPL> aa;
    aa.init(p.ldx, m0, p.M, warp, lane, p.row_index);
    // packed W: tile (n-tile, k-block) = PLANES x 16 KB, already converted and swizzled (pack_weights_kernel)
    const unsigned char* wp_tiles = p.Wp + ((size_t)blockIdx.x * NT * num_kb_total + kb_base) * (PLANES * TILE_BYTES);
    int kstore = kb_shift;                                    // k-block index of the stage being stored
    TileRegs<MODE, EPL> xa[PF + 1];
    int kload = kb_shift;                                     // k-block index of the next load
    int kcur = kb_shift;                                      // k-block index of the register buffer being stored
#pragma unroll
    for (int d = 0; d < PF; ++d) {
      if (d < num_kb) {
        xa[d].template load<VEC>(p.X, aa, (kb_base + kload) * KB, p.K);
        kload = (kload + 1 == num_kb) ? 0 : kload + 1;
      }
    }
    // The k-loop is unrolled by PF+1 so that the register buffers rotate by NAME: copying them (xa[d] = xa[d+1]) would
    // make every iteration wait for the loads it has just issued.
    for (int kb0 = 0; kb0 < num_kb; kb0 += PF + 1) {
#pragma unroll
      for (int j = 0; j <= PF; ++j) {
        const int kb = kb0 + j;
        if (kb < num_kb) {
          const int s = kb % NSTAGE;
          const uint32_t ph = (uint32_t)(kb / NSTAGE) & 1u;
          if (kb + PF < num_kb) {                             // loads of k-block kb+PF fly while kb is converted
            xa[(j + PF) % (PF + 1)].template load<VEC>(p.X, aa, (kb_base + kload) * KB, p.K);
            kload = (kload + 1 == num_kb) ? 0 : kload + 1;
          }
          mbar_wait(&empty_bar[s], ph ^ 1u);                  // first pass through the ring: returns immediately
          unsigned char* st = tiles + (size_t)s * STAGE_BYTES;
          if (tid == 0) {                                     // W tile(s): TMA bulk copies, no thread touches the data
            mbar_arrive_expect_tx(&full_bar[s], NT * PLANES * TILE_BYTES);
            if constexpr (NT == 1) {
              tma_bulk_g2s(st + A_BYTES, wp_tiles + (size_t)kstore * (PLANES * TILE_BYTES), PLANES * TILE_BYTES, &full_bar[s]);
            } else {
              // two packed tiles [hi | lo] each -> stage layout [hi 0][hi 1][lo 0][lo 1]: the MMA sees one 256-row K-major operand per plane
#pragma unroll
              for (int nt = 0; nt < NT; ++nt)
#pragma unroll
                for (int pl = 0; pl < PLANES; ++pl)
                  tma_bulk_g2s(st + A_BYTES + (pl * NT + nt) * TILE_BYTES,
                               wp_tiles + ((size_t)nt * num_kb_total + kstore) * (PLANES * TILE_BYTES) + (size_t)pl * TILE_BYTES, TILE_BYTES,
                               &full_bar[s]);
            }
          }
          kstore = (kstore + 1 == num_kb) ? 0 : kstore + 1;
          const uint32_t st_u = smem_u32(st);
          if ((kb_base + kcur + 1) * KB > p.K) xa[j].template store<true>(st_u, st_u + TILE_BYTES, aa);   // the one k-block that crosses K: masked stores (uniform branch)
          else xa[j].template store<false>(st_u, st_u + TILE_BYTES, aa);
          kcur = (kcur + 1 == num_kb) ? 0 : kcur + 1;
          fence_proxy_async();                                // generic-proxy smem writes -> visible to the tensor core
          __syncwarp();                                       // one arrive per warp: 256 arrives on one mbarrier serialise in the shared-memory atomic unit
          if (lane == 0) mbar_arrive(&full_bar[s]);
        }
      }
    }
    // ===================== epilogue =====================
    // tcgen05.ld hands a thread one accumulator ROW (32 columns at a time).  Stored straight to global memory that is 32 rows x 16 bytes per
    // instruction — 32 cache lines, 8 K L1 wavefronts per CTA, ~4 us of a 36 us kernel (round 2, ncu).  So the tile goes through the (now idle)
    // stage memory first: thread = row into a padded [128][BN] fp32 tile (pitch BN*4 + 16: eight 16-byte stores cover all 32 banks), then every
    // warp walks whole rows, 512 contiguous bytes per instruction, for the slab / the final arithmetic / the partner's partial.
    mbar_wait(&accum_bar, 0);
    tc_fence_after();
    constexpr int XPITCH = BN * 4 + 16;
    const uint32_t xbase = smem_u32(tiles);
    {
      const int quad = warp & 3, chalf = warp >> 2;
      const uint32_t xrow = xbase + (uint32_t)(quad * 32 + lane) * XPITCH;
#pragma unroll 1
      for (int cc = 0; cc < BN / 64; ++cc) {
        const int col0 = chalf * (BN / 2) + cc * 32;
        float acc[32];
#pragma unroll
        for (int a = 0; a < NACC; ++a) {
          uint32_t r[32];
          const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(a * BN + col0);
          asm volatile(
              "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
              "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
              "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
              : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
                "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]),
                "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
                "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
              : "r"(taddr)
              : "memory");
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          const bool written = NACC != 4 || (a & 1) == 0 || num_kb > 1;      // (4 accumulators) with a single k-block the odd ones stay untouched
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float x = written ? __uint_as_float(r[j]) : 0.f;
            acc[j] = (a == 0) ? x : acc[j] + x;
          }
        }
#pragma unroll
        for (int j = 0; j < 32; j += 4)
          sts128(xrow + (uint32_t)(col0 + j) * 4u, __float_as_uint(acc[j]), __float_as_uint(acc[j + 1]), __float_as_uint(acc[j + 2]),
                 __float_as_uint(acc[j + 3]));
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(TC_PRODUCERS) : "memory");       // the eight epilogue warps (a row is written by two of them)
    // row pass: warp w owns rows w, w + 8, ...; a lane owns 4 consecutive columns of every 128-column group
    const bool split = p.kb_per_split > 0;                                // raw tile to this split's slab; arithmetic after the reduction
    const long long e_np = ((long long)p.N + 3) & ~3LL;                   // slab rows are padded to 4 floats
    if (split) {
      float* slab = p.partial + (size_t)blockIdx.z * (size_t)p.M * (size_t)e_np;
#pragma unroll 1
      for (int r = warp; r < TC_BM; r += TC_PRODUCERS / 32) {
        const int row = m0 + r;
        if (row >= p.M) break;
        const float4* src = reinterpret_cast<const float4*>(tiles + (size_t)r * XPITCH);
        float* dst = slab + (long long)row * e_np + n0;
#pragma unroll
        for (int g = 0; g < BN / 128; ++g) {
          const int c = g * 128 + lane * 4;
          if (n0 + c < e_np) *reinterpret_cast<float4*>(dst + c) = src[c / 4];     // (pad columns carry zeros of the zero-padded W)
        }
      }
    } else {
#pragma unroll 1
      for (int r = warp; r < TC_BM; r += TC_PRODUCERS / 32) {
        const int row = m0 + r;
        if (row >= p.M) break;
        const float4* src = reinterpret_cast<const float4*>(tiles + (size_t)r * XPITCH);
        const float rs = p.row_scale ? __ldg(p.row_scale + row) : 1.f;
#pragma unroll
        for (int g = 0; g < BN / 128; ++g) {
          const int c = g * 128 + lane * 4, gc = n0 + c;
          if (gc >= p.N) continue;
          float4 t = src[c / 4];
          float o[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            if (gc + e < p.N) {
              if (p.bias) o[e] += __ldg(p.bias + gc + e);
              o[e] *= rs;
              if (p.relu) o[e] = fmaxf(o[e], 0.f);
            }
          }
          if (p.y_bf16) {
            __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(p.Y) + (long long)row * p.ldy + gc;
            if (gc + 3 < p.N && ((((uintptr_t)dst) & 7) == 0)) {
              const __nv_bfloat162 b0 = __floats2bfloat162_rn(o[0], o[1]), b1 = __floats2bfloat162_rn(o[2], o[3]);
              *reinterpret_cast<uint2*>(dst) = make_uint2(*reinterpret_cast<const uint32_t*>(&b0), *reinterpret_cast<const uint32_t*>(&b1));
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (gc + e < p.N) dst[e] = __float2bfloat16_rn(o[e]);
            }
          } else {
            float* dst = reinterpret_cast<float*>(p.Y) + (long long)row * p.ldy + gc;
            if (gc + 3 < p.N && ((((uintptr_t)dst) & 15) == 0)) {
              *reinterpret_cast<float4*>(dst) = make_float4(o[0], o[1], o[2], o[3]);
            } else {
#pragma unroll
              for (int e = 0; e < 4; ++e)
                if (gc + e < p.N) dst[e] = o[e];
            }
          }
        }
      }
    }
    tc_fence_before();
  } else {
    // ===================== MMA issuer (one elected lane) =====================
    if (lane == 0) {
      const uint32_t idesc = make_idesc<MODE, BN>();
      for (int kb = 0; kb < num_kb; ++kb) {
        const int s = kb % NSTAGE;
        const uint32_t ph = (uint32_t)(kb / NSTAGE) & 1u;
        mbar_wait(&full_bar[s], ph);
        tc_fence_after();
        const uint32_t a_hi = smem_u32(tiles + (size_t)s * STAGE_BYTES);
        const uint32_t b_hi = a_hi + A_BYTES;
#pragma unroll
        for (int ks = 0; ks < 128 / UMMA_K_BYTES; ++ks) {
          const uint32_t off = (uint32_t)ks * UMMA_K_BYTES;
          if constexpr (MODE == TC_BF16) {
            umma<MODE>(tmem_base, make_desc(a_hi + off), make_desc(b_hi + off), idesc, (kb > 0 || ks > 0) ? 1u : 0u);
          } else {
            const uint32_t a_lo = a_hi + TILE_BYTES, b_lo = b_hi + NT * TILE_BYTES;
            const uint32_t d_main = tmem_base + (uint32_t)(NACC == 4 ? (kb & 1) * 128 : 0);            // accumulators 0 / 1
            const uint32_t d_cross = tmem_base + (uint32_t)(NACC == 4 ? 256 + (kb & 1) * 128 : BN);    // accumulators 2 / 3
            const uint32_t first = (kb > (NACC == 4 ? 1 : 0) || ks > 0) ? 1u : 0u;   // the first k-block(s) start their accumulators
            umma<MODE>(d_main, make_desc(a_hi + off), make_desc(b_hi + off), idesc, first);    // hi·hi
            umma<MODE>(d_cross, make_desc(a_hi + off), make_desc(b_lo + off), idesc, first);   // hi·lo
            umma<MODE>(d_cross, make_desc(a_lo + off), make_desc(b_hi + off), idesc, 1u);      // lo·hi
          }
        }
        umma_commit(&empty_bar[s]);          // frees the smem stage once these MMAs have read it
      }
      umma_commit(&accum_bar);               // accumulator complete
    }
    __syncwarp();
    tc_fence_before();
  }
  __syncthreads();
  if (warp == 8) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(TMEM_COLS) : "memory");
  }
}

// W (N, K) fp32 -> tiles [n-tile][k-block][plane][128 rows x 128 B], converted (bf16 / TF32 hi,lo) and laid out exactly as
// the MMA wants them (K-major SWIZZLE_128B), zero-padded in N and K.  One thread per (row, 16-byte chunk).
template <int MODE>
__global__ void pack_weights_kernel(const float* __restrict__ W, long long ldw, int N, int K, unsigned char* __restrict__ out) {
  constexpr int KB = TcMode<MODE>::KB;
  constexpr int PLANES = TcMode<MODE>::PLANES;
  constexpr int EPC = TcMode<MODE>::E16 ? 8 : 4;                  // source elements per 16-byte chunk
  const int num_kb = (K + KB - 1) / KB;
  const int n_tiles = (N + 127) / 128;
  const long long total = (long long)n_tiles * num_kb * 128 * 8;  // 8 chunks per 128-byte row
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= total) return;
  const int ch = (int)(idx & 7);
  const int r = (int)((idx >> 3) & 127);
  const long long tile = idx >> 10;
  const int kb = (int)(tile % num_kb), nt = (int)(tile / num_kb);
  const int row = nt * 128 + r, k0 = kb * KB + ch * EPC;
  float v[EPC];
#pragma unroll
  for (int e = 0; e < EPC; ++e) v[e] = (row < N && k0 + e < K) ? __ldg(W + (long long)row * ldw + k0 + e) : 0.f;
  unsigned char* base = out + (size_t)tile * (PLANES * TILE_BYTES);
  const uint32_t off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + (uint32_t)((ch ^ (r & 7)) << 4);
  if constexpr (MODE == TC_BF16) {
    uint4 q;
    __nv_bfloat162 b0 = __floats2bfloat162_rn(v[0], v[1]), b1 = __floats2bfloat162_rn(v[2], v[3]);
    __nv_bfloat162 b2 = __floats2bfloat162_rn(v[4], v[5]), b3 = __floats2bfloat162_rn(v[6], v[7]);
    q.x = *reinterpret_cast<uint32_t*>(&b0); q.y = *reinterpret_cast<uint32_t*>(&b1);
    q.z = *reinterpret_cast<uint32_t*>(&b2); q.w = *reinterpret_cast<uint32_t*>(&b3);
    *reinterpret_cast<uint4*>(base + off) = q;
  } else if constexpr (MODE == TC_BF16X3) {
    uint32_t h[4], l[4];
#pragma unroll
    for (int e = 0; e < 8; e += 2) bf16_split2(v[e], v[e + 1], h[e / 2], l[e / 2]);
    *reinterpret_cast<uint4*>(base + off) = make_uint4(h[0], h[1], h[2], h[3]);
    *reinterpret_cast<uint4*>(base + TILE_BYTES + off) = make_uint4(l[0], l[1], l[2], l[3]);
  } else {
    float hi[4], lo[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) { hi[e] = tf32_round(v[e]); lo[e] = v[e] - hi[e]; }
    *reinterpret_cast<float4*>(base + off) = make_float4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<float4*>(base + TILE_BYTES + off) = make_float4(lo[0], lo[1], lo[2], lo[3]);
  }
}

static size_t packed_weight_bytes(long long N, long long K, int mode) {
  const int KB = tc_kb(mode), PL = tc_planes(mode);
  return (size_t)((N + 127) / 128) * (size_t)((K + KB - 1) / KB) * PL * TILE_BYTES;
}

// split-K: partial[z] (M x Np, Np = N rounded up to 4; the pad columns are never written nor used) summed in split order
// (deterministic), then bias, row scale, activation
__global__ void __launch_bounds__(256)
tc_splitk_reduce_kernel(const float* __restrict__ partial, int splits, int M, int N, void* __restrict__ Y, long long ldy, int y_bf16,
                        const float* __restrict__ bias, const float* __restrict__ row_scale, int relu) {
  const int Np = (N + 3) & ~3;
  const long long slab = (long long)M * Np;
  const long long i4 = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i4 >= slab / 4) return;
  const long long idx = i4 * 4;
  const int row = (int)(idx / Np), col = (int)(idx % Np);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int z0 = 0; z0 < splits; z0 += 8) {
    float4 v[8];
#pragma unroll
    for (int k = 0; k < 8; ++k)
      v[k] = (z0 + k < splits) ? __ldcs(reinterpret_cast<const float4*>(partial + (long long)(z0 + k) * slab + idx)) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int k = 0; k < 8; ++k) { s.x += v[k].x; s.y += v[k].y; s.z += v[k].z; s.w += v[k].w; }
  }
  float o[4] = {s.x, s.y, s.z, s.w};
  const float rs = row_scale ? __ldg(row_scale + row) : 1.f;
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if (bias && col + e < N) o[e] += __ldg(bias + col + e);
    o[e] *= rs;
    if (relu) o[e] = fmaxf(o[e], 0.f);
  }
  if (y_bf16) {
    __nv_bfloat16* dst = reinterpret_cast<__nv_bfloat16*>(Y) + (long long)row * ldy + col;
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (col + e < N) dst[e] = __float2bfloat16_rn(o[e]);
  } else {
    float* dst = reinterpret_cast<float*>(Y) + (long long)row * ldy + col;
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (col + e < N) dst[e] = o[e];
  }
}

// number of K splits for a GEMM whose output tiles alone leave most SMs idle (0 = do not split)
static int tc_splits_tiles(long long tiles, bool n_ok, long long K, int mode, int* kb_per_split) {
  const int KB = tc_kb(mode);
  const int num_kb = (int)((K + KB - 1) / KB);
  const int sms = b200rec_num_sms();
  *kb_per_split = 0;
  (void)n_ok;                                                  // (slab rows are padded: any N splits)
  if (tiles * 2 > sms || num_kb < 8) return 0;
  int want = (int)(sms / tiles);
  if (want > num_kb / 3) want = num_kb / 3;                    // at least 3 k-blocks per CTA
  if (want < 2) return 0;
  const int kbps = (num_kb + want - 1) / want;
  *kb_per_split = kbps;
  return (num_kb + kbps - 1) / kbps;
}
static int tc_splits(long long M, long long N, long long K, int mode, int* kb_per_split) {
  return tc_splits_tiles(((M + 127) / 128) * ((N + 127) / 128), (N % 4) == 0, K, mode, kb_per_split);
}

template <int MODE, int EPL, bool VEC, int BN = TC_BN>
static int launch_tc_epl(const TcBatch& b, cudaStream_t st) {
  constexpr int PLANES = TcMode<MODE>::PLANES;
  constexpr int NSTAGE = BN == 256 ? ((MODE == TC_BF16) ? 4 : 2) : ((MODE == TC_BF16) ? 4 : 3);
  const size_t smem = (size_t)NSTAGE * (1 + BN / 128) * PLANES * TILE_BYTES + 1024;
  static B200recSmemOptIn opted;                     // per template instantiation, one bit per device
  B200REC_CUDA(b200rec_opt_in_smem(opted, gemm_tc_kernel<MODE, NSTAGE, EPL, VEC, BN>, (int)smem));
  int nmax = 0;
  for (int q = 0; q < b.n; ++q) nmax = b.prob[q].N > nmax ? b.prob[q].N : nmax;
  const TcParams& p0 = b.prob[0];
  const int nsplit = p0.kb_per_split ? ceil_div_i(ceil_div_i(p0.K, TcMode<MODE>::KB), p0.kb_per_split) : 1;
  dim3 grid(ceil_div_i(nmax, BN), b.tile_start[b.n], nsplit);
  gemm_tc_kernel<MODE, NSTAGE, EPL, VEC, BN><<<grid, TC_THREADS, smem, st>>>(b);
  B200REC_CHECK_LAUNCH();
  if (p0.kb_per_split) {
    for (int q = 0; q < b.n; ++q) {                  // (a batch shares K and kb_per_split: b200rec_linear_tc_splitk_batch)
      const TcParams& pq = b.prob[q];
      const long long total4 = (long long)pq.M * (((long long)pq.N + 3) / 4);
      tc_splitk_reduce_kernel<<<ceil_div_i(total4, 256), 256, 0, st>>>(pq.partial, nsplit, pq.M, pq.N, pq.Y, pq.ldy, pq.y_bf16, pq.bias,
                                                                       pq.row_scale, pq.relu);
      B200REC_CHECK_LAUNCH();
    }
  }
  return B200REC_OK;
}

template <int MODE, int BN = TC_BN>
static int launch_tc(const TcBatch& b, cudaStream_t st) {
  auto aligned = [&](int n) {
    for (int q = 0; q < b.n; ++q) {
      const TcParams& p = b.prob[q];
      if (!((p.K % n) == 0 && (p.ldx % n) == 0 && ((uintptr_t)p.X % (4 * n)) == 0)) return false;
    }
    return true;
  };
  if (aligned(4)) return launch_tc_epl<MODE, 4, true, BN>(b, st);        // 128-bit loads (e.g. K = 128 transforms)
  if (aligned(2)) return launch_tc_epl<MODE, 2, true, BN>(b, st);        // 64-bit loads (F = 2094)
  return launch_tc_epl<MODE, 2, false, BN>(b, st);                       // odd K / pitch: scalar loads
}

}  // namespace b200rec

using namespace b200rec;

extern "C" size_t b200rec_packed_weight_bytes(int64_t N, int64_t K, int mode) {
  return (N > 0 && K > 0 && mode >= 0 && mode <= TC_BF16X3) ? packed_weight_bytes(N, K, mode) : 0;
}

extern "C" int b200rec_pack_weights_tc(const float* W, int64_t N, int64_t K, int64_t ldw, int mode, void* packed, size_t packed_bytes,
                                       b200rec_stream_t stream) {
  if (!W || !packed || N <= 0 || K <= 0 || ldw < K) return b200rec_fail(B200REC_ERR_BAD_ARG, "pack_weights_tc: bad argument");
  if (mode < 0 || mode > TC_BF16X3) return b200rec_fail(B200REC_ERR_BAD_ARG, "pack_weights_tc: bad mode");
  if (packed_bytes < packed_weight_bytes(N, K, mode) || ((uintptr_t)packed % 128))
    return b200rec_fail(B200REC_ERR_WORKSPACE, "pack_weights_tc: buffer too small or not 128-byte aligned");
  const int KB = tc_kb(mode);
  const long long total = ((N + 127) / 128) * ((K + KB - 1) / KB) * 128LL * 8;
  const unsigned grid = (unsigned)((total + 255) / 256);
  if (mode == TC_BF16) pack_weights_kernel<TC_BF16><<<grid, 256, 0, (cudaStream_t)stream>>>(W, ldw, (int)N, (int)K, (unsigned char*)packed);
  else if (mode == TC_TF32X3) pack_weights_kernel<TC_TF32X3><<<grid, 256, 0, (cudaStream_t)stream>>>(W, ldw, (int)N, (int)K, (unsigned char*)packed);
  else pack_weights_kernel<TC_BF16X3><<<grid, 256, 0, (cudaStream_t)stream>>>(W, ldw, (int)N, (int)K, (unsigned char*)packed);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

// W and ldw of the entry points are not read: the GEMM takes the weights from `packed_w`
static int tc_fill(TcParams& p, const float* X, int64_t M, int64_t K, int64_t ldx, int64_t N, const float* bias,
                   const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, const void* packed_w,
                   const int64_t* row_index = nullptr, int64_t x_rows = 0) {
  if (M < 0 || N <= 0 || K <= 0 || (M > 0 && (!X || !Y))) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc: bad argument");
  if (!packed_w) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc: needs the packed weights (b200rec_pack_weights_tc, same mode)");
  if (M > INT32_MAX || N > INT32_MAX || K > INT32_MAX) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "linear_tc: dim > int32");
  if (ldx < K || ldy < N) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc: leading dimension too small");
  if ((row_index ? x_rows : M) * ldx >= (1LL << 32)) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "linear_tc: operand larger than 2^32 elements");
  if (row_index && x_rows <= 0) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc: row_index needs the row count of X");
  if (y_dtype != B200REC_F32 && y_dtype != B200REC_BF16) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc: bad y_dtype");
  p.row_index = reinterpret_cast<const long long*>(row_index);
  p.X = X; p.ldx = ldx; p.M = (int)M; p.N = (int)N; p.K = (int)K;
  p.Wp = (const unsigned char*)packed_w;
  p.Y = Y; p.ldy = ldy; p.y_bf16 = y_dtype == B200REC_BF16; p.bias = bias; p.row_scale = row_scale; p.relu = relu;
  p.kb_per_split = 0;
  p.partial = nullptr;
  return B200REC_OK;
}

extern "C" int b200rec_linear_tc(const float* X, int64_t M, int64_t K, int64_t ldx, const float* W, int64_t N, int64_t ldw,
                                 const float* bias, const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, int mode,
                                 const void* packed_w, const int64_t* row_index, int64_t x_rows, b200rec_stream_t stream) {
  TcBatch b;
  b.n = 1;
  const int rc = tc_fill(b.prob[0], X, M, K, ldx, N, bias, row_scale, relu, Y, ldy, y_dtype, packed_w, row_index, x_rows);
  if (rc) return rc;
  if (M == 0) return B200REC_OK;
  b.tile_start[0] = 0;
  b.tile_start[1] = ceil_div_i(M, TC_BM);
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == B200REC_TC_TF32X3) return launch_tc<TC_TF32X3>(b, st);
  if (mode == B200REC_TC_BF16) return launch_tc<TC_BF16>(b, st);
  return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc: bad mode");
}

extern "C" size_t b200rec_linear_tc_splitk_workspace(int64_t M, int64_t N, int64_t K, int mode) {
  if (M <= 0 || N <= 0 || K <= 0) return 0;
  int kbps = 0;
  const int splits = tc_splits(M, N, K, mode == B200REC_TC_BF16 ? TC_BF16 : TC_TF32X3, &kbps);
  return splits > 1 ? (size_t)splits * (size_t)M * (size_t)((N + 3) & ~3LL) * sizeof(float) : 0;
}

extern "C" int b200rec_linear_tc_splitk(const float* X, int64_t M, int64_t K, int64_t ldx, const float* W, int64_t N, int64_t ldw,
                                        const float* bias, const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, int mode,
                                        const void* packed_w, void* workspace, size_t workspace_bytes, b200rec_stream_t stream) {
  TcBatch b;
  b.n = 1;
  const int rc = tc_fill(b.prob[0], X, M, K, ldx, N, bias, row_scale, relu, Y, ldy, y_dtype, packed_w, nullptr, 0);
  if (rc) return rc;
  if (M == 0) return B200REC_OK;
  if (mode != B200REC_TC_TF32X3 && mode != B200REC_TC_BF16) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc_splitk: bad mode");
  int kbps = 0;
  const int splits = tc_splits(M, N, K, mode == B200REC_TC_BF16 ? TC_BF16 : TC_TF32X3, &kbps);
  if (splits > 1) {
    const size_t need = (size_t)splits * (size_t)M * (size_t)((N + 3) & ~3LL) * sizeof(float);
    if (!workspace || workspace_bytes < need || ((uintptr_t)workspace % 16)) return b200rec_fail(B200REC_ERR_WORKSPACE, "linear_tc_splitk: workspace too small");
    b.prob[0].kb_per_split = kbps;
    b.prob[0].partial = (float*)workspace;
  }
  b.tile_start[0] = 0;
  b.tile_start[1] = ceil_div_i(M, TC_BM);
  for (int q = 1; q < TC_MAX_BATCH; ++q) b.tile_start[q + 1] = b.tile_start[1];
  cudaStream_t st = (cudaStream_t)stream;
  return mode == B200REC_TC_TF32X3 ? launch_tc<TC_TF32X3>(b, st) : launch_tc<TC_BF16>(b, st);
}

// wide form: 128 x 256 tiles, k range split so that (row tiles) x (column pairs) x splits fills the device once
static int tc_wide_splits(long long M, long long N, long long K, int mode, int* kb_per_split) {
  const long long tiles = ((M + 127) / 128) * ((N + 255) / 256);
  const int KB = tc_kb(mode);
  const int num_kb = (int)((K + KB - 1) / KB);
  const int sms = b200rec_num_sms();
  int want = (int)(sms / tiles);
  if (want < 2) want = 2;                                       // always split: the two TMEM accumulators want short chains
  if (want > num_kb * KB / 128) want = num_kb * KB / 128;         // at least 128 columns of k per CTA
  if (want < 1) want = 1;
  const int kbps = (num_kb + want - 1) / want;
  *kb_per_split = kbps;
  return (num_kb + kbps - 1) / kbps;
}

extern "C" size_t b200rec_linear_tc_wide_workspace(int64_t M, int64_t N, int64_t K, int mode) {
  if (M <= 0 || N <= 0 || K <= 0 || (mode != B200REC_TC_TF32X3 && mode != B200REC_TC_BF16X3)) return 0;
  int kbps = 0;
  const int splits = tc_wide_splits(M, N, K, mode, &kbps);
  return (size_t)splits * (size_t)M * (size_t)((N + 3) & ~3LL) * sizeof(float);
}

extern "C" int b200rec_linear_tc_wide(const float* X, int64_t M, int64_t K, int64_t ldx, int64_t N, const float* bias, const float* row_scale,
                                      int relu, void* Y, int64_t ldy, int y_dtype, int mode, const void* packed_w, const int64_t* row_index,
                                      int64_t x_rows, void* workspace, size_t workspace_bytes, b200rec_stream_t stream) {
  TcBatch b;
  b.n = 1;
  if (mode != B200REC_TC_TF32X3 && mode != B200REC_TC_BF16X3) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc_wide: mode is TF32X3 or BF16X3");
  if (N <= 128 || ((N + 127) / 128) % 2) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "linear_tc_wide: N must cover an even number of 128-column tiles");
  const int rc = tc_fill(b.prob[0], X, M, K, ldx, N, bias, row_scale, relu, Y, ldy, y_dtype, packed_w, row_index, x_rows);
  if (rc) return rc;
  if (M == 0) return B200REC_OK;
  int kbps = 0;
  const int splits = tc_wide_splits(M, N, K, mode, &kbps);
  const size_t need = (size_t)splits * (size_t)M * (size_t)((N + 3) & ~3LL) * sizeof(float);
  if (!workspace || workspace_bytes < need || ((uintptr_t)workspace % 16)) return b200rec_fail(B200REC_ERR_WORKSPACE, "linear_tc_wide: workspace too small");
  b.prob[0].kb_per_split = kbps;
  b.prob[0].partial = (float*)workspace;
  b.tile_start[0] = 0;
  b.tile_start[1] = ceil_div_i(M, TC_BM);
  for (int q = 1; q < TC_MAX_BATCH; ++q) b.tile_start[q + 1] = b.tile_start[1];
  return mode == B200REC_TC_TF32X3 ? launch_tc<TC_TF32X3, 256>(b, (cudaStream_t)stream) : launch_tc<TC_BF16X3, 256>(b, (cudaStream_t)stream);
}

extern "C" int b200rec_linear_tc_batch(const b200rec_linear_problem_t* problems, int n_problems, int64_t K, int mode,
                                       b200rec_stream_t stream) {
  if (!problems || n_problems < 1 || n_problems > TC_MAX_BATCH) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc_batch: 1..4 problems");
  TcBatch b;
  b.n = 0;
  b.tile_start[0] = 0;
  for (int q = 0; q < n_problems; ++q) {
    const b200rec_linear_problem_t& r = problems[q];
    if (r.M == 0) continue;
    const int rc = tc_fill(b.prob[b.n], r.X, r.M, K, r.ldx, r.N, r.bias, r.row_scale, r.relu, r.Y, r.ldy, r.y_dtype, r.packed_w);
    if (rc) return rc;
    b.tile_start[b.n + 1] = b.tile_start[b.n] + ceil_div_i(r.M, TC_BM);
    ++b.n;
  }
  if (b.n == 0) return B200REC_OK;
  for (int q = b.n; q < TC_MAX_BATCH; ++q) b.tile_start[q + 1] = b.tile_start[b.n];
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == B200REC_TC_TF32X3) return launch_tc<TC_TF32X3>(b, st);
  if (mode == B200REC_TC_BF16) return launch_tc<TC_BF16>(b, st);
  return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc_batch: bad mode");
}

// Several short-M / long-K GEMMs of one K in ONE split-K launch (BasicNCF's user and item projections: 2 x 4 row tiles dealt out over
// ~17 k-splits each fill the device in a single wave instead of two 88-CTA launches).  Workspace = splits x sum(M_q x N_q) floats.
static int tc_batch_splits(const b200rec_linear_problem_t* problems, int n, int64_t K, int mode, int* kbps, size_t* floats) {
  long long tiles = 0, total = 0;
  bool n_ok = true;
  for (int q = 0; q < n; ++q) {
    if (problems[q].M <= 0) continue;
    tiles += ((problems[q].M + 127) / 128) * ((problems[q].N + 127) / 128);
    total += problems[q].M * ((problems[q].N + 3) & ~3LL);
    n_ok = n_ok && (problems[q].N % 4) == 0;
  }
  *floats = (size_t)total;
  if (tiles == 0) return 0;
  return tc_splits_tiles(tiles, n_ok, K, mode == B200REC_TC_BF16 ? TC_BF16 : TC_TF32X3, kbps);
}

extern "C" size_t b200rec_linear_tc_splitk_batch_workspace(const b200rec_linear_problem_t* problems, int n_problems, int64_t K, int mode) {
  if (!problems || n_problems < 1 || n_problems > TC_MAX_BATCH || K <= 0) return 0;
  int kbps = 0;
  size_t floats = 0;
  const int splits = tc_batch_splits(problems, n_problems, K, mode, &kbps, &floats);
  return splits > 1 ? (size_t)splits * floats * sizeof(float) : 0;
}

extern "C" int b200rec_linear_tc_splitk_batch(const b200rec_linear_problem_t* problems, int n_problems, int64_t K, int mode, void* workspace,
                                              size_t workspace_bytes, b200rec_stream_t stream) {
  if (!problems || n_problems < 1 || n_problems > TC_MAX_BATCH) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc_splitk_batch: 1..4 problems");
  if (mode != B200REC_TC_TF32X3 && mode != B200REC_TC_BF16) return b200rec_fail(B200REC_ERR_BAD_ARG, "linear_tc_splitk_batch: bad mode");
  int kbps = 0;
  size_t floats = 0;
  const int splits = tc_batch_splits(problems, n_problems, K, mode, &kbps, &floats);
  if (splits > 1 && (!workspace || workspace_bytes < (size_t)splits * floats * sizeof(float) || ((uintptr_t)workspace % 16)))
    return b200rec_fail(B200REC_ERR_WORKSPACE, "linear_tc_splitk_batch: workspace too small");
  TcBatch b;
  b.n = 0;
  b.tile_start[0] = 0;
  float* part = (float*)workspace;
  for (int q = 0; q < n_problems; ++q) {
    const b200rec_linear_problem_t& r = problems[q];
    if (r.M == 0) continue;
    const int rc = tc_fill(b.prob[b.n], r.X, r.M, K, r.ldx, r.N, r.bias, r.row_scale, r.relu, r.Y, r.ldy, r.y_dtype, r.packed_w);
    if (rc) return rc;
    if (splits > 1) {
      b.prob[b.n].kb_per_split = kbps;
      b.prob[b.n].partial = part;
      part += (size_t)splits * (size_t)r.M * (size_t)((r.N + 3) & ~3LL);        // 16-byte aligned: padded rows
    }
    b.tile_start[b.n + 1] = b.tile_start[b.n] + ceil_div_i(r.M, TC_BM);
    ++b.n;
  }
  if (b.n == 0) return B200REC_OK;
  for (int q = b.n; q < TC_MAX_BATCH; ++q) b.tile_start[q + 1] = b.tile_start[b.n];
  cudaStream_t st = (cudaStream_t)stream;
  return mode == B200REC_TC_TF32X3 ? launch_tc<TC_TF32X3>(b, st) : launch_tc<TC_BF16>(b, st);
}
