// K5 — all-pairs NCF scoring with a per-user top-k, fused:  for every (user u, item i)
//
//     h1 = ReLU(A[u] + B[i])                       A = user_emb·W1[:, :Eu]ᵀ + b1   (nU, H1)   layer 1 of the MLP split
//     h2 = ReLU(W2·h1 + b2)                        B = item_emb·W1[:, Eu:]ᵀ        (nI, H1)   into its two halves
//     score(u, i) = w3·h2 + b3                     and per user the k best items.
//
// This is BASELINE configs[3] ("BasicNCF batch inference over all user×item pairs for top-K", 10^11 pairs) and the
// reference's only serving pattern (src/webapp/backend.py:78-121: score every candidate, `sort_values(...).iloc[:k]`).
// The reference evaluates `MLP(cat(user_emb, item_emb))` per pair (basic_ncf.py:40-41, util.py:5-18); splitting the first
// Linear is exact algebra and leaves 2·H1·H2 + 2·H2 FLOP per pair (65,792 for [256,128]) — the only dense contraction per
// pair, so it runs on the 5th-generation tensor cores:
//
//   * MMA tile = 128 pairs (4 users x 32 items) x N = H2 (<=128) x K = H1 (<=256), bf16 operands, fp32 accumulate in TMEM.
//   * The A operand (h1) never exists in HBM: 8 producer warps form ReLU(a_u + b_i) in registers (item rows live in
//     registers for the 4..8 user quads of the CTA, user rows in shared memory), convert and write the K-major
//     SWIZZLE_128B tile straight into a shared-memory ring; W2 sits in shared memory for the life of the CTA (TMA bulk).
//   * warp 12 issues tcgen05.mma into one of two TMEM accumulators; 4 epilogue warps read the other one (tcgen05.ld),
//     apply b2 / ReLU / w3 / b3 and keep each user's k best (score, item) in shared memory — warp e owns the users
//     e, 4+e, ... of the CTA, so the insertion needs no atomics.  Scores are never written unless asked for.
//   * modes: AP_BF16 (one MMA per k-step, rel <= 1e-2) and AP_BF16X2 (h1 and W2 split into bf16 hi + lo, three MMAs
//     hi·hi + hi·lo + lo·hi: measured 4e-6 max-norm relative error on the pre-activations, inside the fp32 tolerance).
//
// Grid = (user blocks of 32 resp. 16 users) x (item splits); every CTA walks its item range once for its users, so an
// item row is fetched from L2 once per 32 (16) users.  Partial top-k lists of the splits are merged by a second kernel.
#include <math.h>

#include "common.cuh"

namespace b200rec {

enum { AP_BF16 = 0, AP_BF16X2 = 1 };

constexpr int AP_PRODUCERS = 256;                       // warps 0-7
constexpr int AP_EPI = 128;                             // warps 8-11 (TMEM lane quadrant = warp % 4)
constexpr int AP_THREADS = AP_PRODUCERS + AP_EPI + 32;  // warp 12: MMA issuer
constexpr int AP_TILE = 128 * 128;                      // one operand tile: 128 rows x 128 bytes (64 bf16 of K)
constexpr int AP_IT = 32;                               // items per MMA tile (x 4 users = 128 rows)
constexpr int AP_KMAX = 64;                             // largest k
constexpr int AP_NPAD = 128;                            // W2 rows padded to 128 (MMA N)

__device__ __forceinline__ uint32_t ap_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void ap_mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(ap_smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void ap_mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(ap_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void ap_mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(ap_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void ap_mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "AP_WAIT:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra AP_DONE;\n\t"
      "bra AP_WAIT;\n\t"
      "AP_DONE:\n\t"
      "}" ::"r"(ap_smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void ap_bulk_g2s(void* dst_smem, const void* src_gmem, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(ap_smem_u32(dst_smem)),
               "l"(src_gmem), "r"(bytes), "r"(ap_smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void ap_fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void ap_tc_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void ap_tc_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void ap_umma(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void ap_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(ap_smem_u32(bar)) : "memory");
}
// K-major SWIZZLE_128B shared-memory matrix descriptor (same encoding as csrc/gemm_tc.cu)
__device__ __forceinline__ uint64_t ap_desc(uint32_t smem_addr) {
  return (uint64_t)((smem_addr & 0x3ffff) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// c_format F32, A/B bf16, both K-major, N = 128, M = 128
__device__ __forceinline__ uint32_t ap_idesc() {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(AP_NPAD >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
}
// two fp32 -> packed bf16x2 (x0 in the low half), round to nearest even, optional ReLU in the conversion
__device__ __forceinline__ uint32_t ap_pack_relu(float x0, float x1) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(x1), "f"(x0));
  return d;
}
__device__ __forceinline__ uint32_t ap_pack(float x0, float x1) {
  uint32_t d;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(x1), "f"(x0));
  return d;
}

// relu(a * 1 + b) on two packed bf16 pairs (HFMA2.BF16 with the ReLU folded in)
__device__ __forceinline__ uint32_t ap_add_relu_bf16x2(uint32_t a, uint32_t b) {
  uint32_t d;
  asm("fma.rn.relu.bf16x2 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(0x3F803F80u), "r"(b));
  return d;
}

struct AllPairsParams {
  const float* A;             // (nU, H1) contiguous
  const float* B;             // (nI, H1) contiguous
  int nU, nI, H1;             // H1 in {64, 128, 192, 256}
  const unsigned char* Wp;    // packed by allpairs_pack_kernel: [kb][plane][128 x 128 B] tiles
  int k;                      // 0 = no top-k
  int n_splits, items_per_split;
  float* part_val;            // (nU, n_splits, k)
  int* part_idx;
  float* scores;              // optional (nU, nI) ld = lds
  long long lds;
  const int* seen_ptr;        // optional CSR (nU+1) / sorted item ids: pairs the user has already interacted with are skipped
  const int* seen_idx;
  // epilogue constants travel in the kernel parameter block (constant bank): FADD / FFMA read them as c[0][..] operands.
  // As shared-memory broadcasts they cost one wavefront per quarter-warp and instruction — 1,024 wavefronts per tile, more
  // than the MMA's own operand fetch (profiles/r01/ncu_allpairs_v2.txt).
  float b2[AP_NPAD], w3[AP_NPAD], b3;
};

// shared-memory layout (byte offsets from the 1024-aligned base); NKB = H1 / 64
template <int MODE, int UQ>
struct ApLayout {
  static constexpr int PLANES = MODE == AP_BF16 ? 1 : 2;
  static constexpr int NS = MODE == AP_BF16 ? 4 : 2;            // ring stages (one stage = one 64-wide k-block, all planes)
  static constexpr int UT = 4 * UQ;                             // users per CTA
  static constexpr int STAGE = PLANES * AP_TILE;
  __host__ __device__ static constexpr int w2(int) { return 0; }
  __host__ __device__ static constexpr int ring(int nkb) { return nkb * PLANES * AP_TILE; }
  __host__ __device__ static constexpr int users(int nkb) { return ring(nkb) + NS * STAGE; }
  static constexpr int UBYTES = MODE == AP_BF16 ? 2 : 4;      // user rows: bf16 (AP_BF16) or permuted fp32 (AP_BF16X2)
  __host__ __device__ static constexpr int list_val(int nkb) { return users(nkb) + UT * nkb * 64 * UBYTES; }
  __host__ __device__ static constexpr int list_idx(int nkb) { return list_val(nkb) + UT * AP_KMAX * 4; }
  __host__ __device__ static constexpr int thr(int nkb) { return list_idx(nkb) + UT * AP_KMAX * 4; }
  __host__ __device__ static constexpr int total(int nkb) { return thr(nkb) + UT * 4 + 1024; }           // + alignment slack
};

// one warp inserts (cs, ci) into the descending list of user `ul` (ties: the earlier = lower item index stays in front)
__device__ __forceinline__ void ap_insert(float* lv, int* li, float* thr, int k, float cs, int ci, int lane) {
  const float v0 = lane < k ? lv[lane] : -INFINITY;
  const float v1 = lane + 32 < k ? lv[lane + 32] : -INFINITY;
  const int p = __popc(__ballot_sync(FULL, lane < k && v0 >= cs)) + __popc(__ballot_sync(FULL, lane + 32 < k && v1 >= cs));
  if (p >= k) return;                                             // warp-uniform
  const float pv0 = (lane > 0 && lane - 1 < k) ? lv[lane - 1] : 0.f, pv1 = lane + 31 < k ? lv[lane + 31] : 0.f;
  const int pi0 = (lane > 0 && lane - 1 < k) ? li[lane - 1] : -1, pi1 = lane + 31 < k ? li[lane + 31] : -1;
  __syncwarp();
  if (lane < k && lane >= p) { lv[lane] = lane == p ? cs : pv0; li[lane] = lane == p ? ci : pi0; }
  if (lane + 32 < k && lane + 32 >= p) { lv[lane + 32] = lane + 32 == p ? cs : pv1; li[lane + 32] = lane + 32 == p ? ci : pi1; }
  __syncwarp();
  if (lane == 0) *thr = lv[k - 1];
  __syncwarp();
}

template <int MODE, int UQ, int NKB>
__global__ void __launch_bounds__(AP_THREADS, 1)
allpairs_topk_kernel(AllPairsParams p) {
  using LY = ApLayout<MODE, UQ>;
  constexpr int PLANES = LY::PLANES, NS = LY::NS, UT = LY::UT, STAGE = LY::STAGE;
  constexpr int H1 = NKB * 64;
  extern __shared__ unsigned char ap_smem_raw[];
  unsigned char* sm = reinterpret_cast<unsigned char*>(((uintptr_t)ap_smem_raw + 1023) & ~(uintptr_t)1023);
  unsigned char* sm_w2 = sm + LY::w2(NKB);
  unsigned char* sm_ring = sm + LY::ring(NKB);
  float* sm_users = reinterpret_cast<float*>(sm + LY::users(NKB));
  float* sm_lv = reinterpret_cast<float*>(sm + LY::list_val(NKB));
  int* sm_li = reinterpret_cast<int*>(sm + LY::list_idx(NKB));
  float* sm_thr = reinterpret_cast<float*>(sm + LY::thr(NKB));
  __shared__ __align__(8) uint64_t w_bar, u_bar, a_full[NS], a_empty[NS], acc_full[2], acc_empty[2];
  __shared__ uint32_t tmem_base_smem;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int u0 = blockIdx.x * UT;
  const int users_here = min(UT, p.nU - u0);
  const int uq_count = (users_here + 3) >> 2;
  const int i_begin = blockIdx.y * p.items_per_split;
  const int i_end = min(p.nI, i_begin + p.items_per_split);
  const int n_it = (i_end - i_begin + AP_IT - 1) / AP_IT;

  if (tid == 0) {
#pragma unroll
    for (int s = 0; s < NS; ++s) { ap_mbar_init(&a_full[s], AP_PRODUCERS); ap_mbar_init(&a_empty[s], 1); }
#pragma unroll
    for (int s = 0; s < 2; ++s) { ap_mbar_init(&acc_full[s], 1); ap_mbar_init(&acc_empty[s], AP_EPI); }
    ap_mbar_init(&w_bar, 1);
    ap_mbar_init(&u_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 12) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(ap_smem_u32(&tmem_base_smem)), "r"(256) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  ap_tc_before();
  __syncthreads();
  ap_tc_after();
  const uint32_t tmem_base = tmem_base_smem;

  if (tid == 0) {                        // resident operands: W2 tiles; the CTA's user rows + b2 / w3 / b3
    constexpr uint32_t W2_BYTES = NKB * PLANES * AP_TILE;
    ap_mbar_expect_tx(&w_bar, W2_BYTES);
#pragma unroll
    for (int t = 0; t < NKB * PLANES; ++t) ap_bulk_g2s(sm_w2 + t * AP_TILE, p.Wp + (size_t)t * AP_TILE, AP_TILE, &w_bar);
    const uint32_t ub = (uint32_t)users_here * H1 * 4u;
    ap_mbar_expect_tx(&u_bar, ub);
    ap_bulk_g2s(sm_ring, p.A + (size_t)u0 * H1, ub, &u_bar);       // raw fp32 rows, re-laid out by the producers below
  }

  if (warp < 8) {
    // ===================== producers: A-operand tiles ReLU(a_u + b_i) =====================
    // (0) user rows: raw fp32 (TMA, parked in the ring) -> the layout the inner loop reads without bank conflicts
    ap_mbar_wait(&u_bar, 0);
    {
      const float4* raw = reinterpret_cast<const float4*>(sm_ring);
      if constexpr (MODE == AP_BF16) {                           // bf16 rows: one 16-byte chunk = 8 consecutive k
        uint4* dst = reinterpret_cast<uint4*>(sm_users);
        for (int idx = tid; idx < UT * H1 / 8; idx += AP_PRODUCERS) {
          uint4 q = make_uint4(0u, 0u, 0u, 0u);
          if (idx / (H1 / 8) < users_here) {
            const float4 x = raw[2 * idx], y = raw[2 * idx + 1];
            q = make_uint4(ap_pack(x.x, x.y), ap_pack(x.z, x.w), ap_pack(y.x, y.y), ap_pack(y.z, y.w));
          }
          dst[idx] = q;
        }
      } else {                                                   // fp32 rows, 16-byte pieces of a k-block stored as [half][chunk]
        float4* dst = reinterpret_cast<float4*>(sm_users);
        for (int idx = tid; idx < UT * H1 / 4; idx += AP_PRODUCERS) {
          const int row = idx / (H1 / 4), pq = idx % (H1 / 4), kb = pq >> 4, cc = (pq & 15) >> 1, half = pq & 1;
          dst[row * (H1 / 4) + kb * 16 + half * 8 + cc] = row < users_here ? raw[idx] : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    }
    asm volatile("bar.sync 1, %0;" ::"n"(AP_PRODUCERS) : "memory");   // the ring is free for operand tiles from here on
    uint32_t cnt = 0;
    if constexpr (MODE == AP_BF16) {
      // thread = (16-byte chunk c, item pair ip / ip+16, user half uh): 2 items x 2 users = 4 rows of every tile.  Item rows
      // live in registers as packed bf16 (prefetched one item tile ahead), user rows come from shared memory as bf16; one
      // HFMA2.BF16 with ReLU per two elements.  Shared-memory cost per tile: 256 wavefronts of loads + 512 of stores.
      const int c = tid & 7, ip = (tid >> 3) & 15, uh = tid >> 7;
      const uint32_t soff = (uint32_t)(ip >> 3) * 1024u + (uint32_t)(ip & 7) * 128u + (uint32_t)((c ^ (ip & 7)) << 4);
      uint4 bq[2][NKB], bnext[2][NKB];
      auto load_items = [&](uint4 (&dst)[2][NKB], int it) {
#pragma unroll
        for (int m = 0; m < 2; ++m) {
          const int item = min(i_begin + it * AP_IT + ip + 16 * m, p.nI - 1);
          const float* src = p.B + (size_t)item * H1 + c * 8;
#pragma unroll
          for (int kb = 0; kb < NKB; ++kb) {
            const float4 x = __ldg(reinterpret_cast<const float4*>(src + kb * 64));
            const float4 y = __ldg(reinterpret_cast<const float4*>(src + kb * 64 + 4));
            dst[m][kb] = make_uint4(ap_pack(x.x, x.y), ap_pack(x.z, x.w), ap_pack(y.x, y.y), ap_pack(y.z, y.w));
          }
        }
      };
      if (n_it > 0) load_items(bq, 0);
      const uint4* ua = reinterpret_cast<const uint4*>(sm_users);
      for (int it = 0; it < n_it; ++it) {
        if (it + 1 < n_it) load_items(bnext, it + 1);
        for (int uq = 0; uq < uq_count; ++uq) {
#pragma unroll
          for (int kb = 0; kb < NKB; ++kb) {
            const uint32_t s = cnt % NS, ph = (cnt / NS) & 1u;
            ap_mbar_wait(&a_empty[s], ph ^ 1u);
            unsigned char* st = sm_ring + (size_t)s * STAGE;
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
              const int j = 2 * uh + jj;
              const uint4 av = ua[(size_t)(uq * 4 + j) * (H1 / 8) + kb * 8 + c];
#pragma unroll
              for (int m = 0; m < 2; ++m) {
                uint4 q;
                q.x = ap_add_relu_bf16x2(av.x, bq[m][kb].x); q.y = ap_add_relu_bf16x2(av.y, bq[m][kb].y);
                q.z = ap_add_relu_bf16x2(av.z, bq[m][kb].z); q.w = ap_add_relu_bf16x2(av.w, bq[m][kb].w);
                *reinterpret_cast<uint4*>(st + soff + m * 2048 + j * 4096) = q;
              }
            }
            ap_fence_async();
            ap_mbar_arrive(&a_full[s]);
            ++cnt;
          }
        }
        if (it + 1 < n_it) {
#pragma unroll
          for (int m = 0; m < 2; ++m)
#pragma unroll
            for (int kb = 0; kb < NKB; ++kb) bq[m][kb] = bnext[m][kb];
        }
      }
    } else {
      // thread = (chunk c, item il): the 4 users of the quad x 1 item; fp32 sum, hi/lo bf16 split
      const int c = tid & 7, il = tid >> 3;
      const uint32_t soff = (uint32_t)(il >> 3) * 1024u + (uint32_t)(il & 7) * 128u + (uint32_t)((c ^ (il & 7)) << 4);
      float breg[NKB][8], bnext[NKB][8];
      auto load_items = [&](float (&dst)[NKB][8], int it) {
        const int item = min(i_begin + it * AP_IT + il, p.nI - 1);
        const float* src = p.B + (size_t)item * H1 + c * 8;
#pragma unroll
        for (int kb = 0; kb < NKB; ++kb) {
          const float4 lo = __ldg(reinterpret_cast<const float4*>(src + kb * 64));
          const float4 hi = __ldg(reinterpret_cast<const float4*>(src + kb * 64 + 4));
          dst[kb][0] = lo.x; dst[kb][1] = lo.y; dst[kb][2] = lo.z; dst[kb][3] = lo.w;
          dst[kb][4] = hi.x; dst[kb][5] = hi.y; dst[kb][6] = hi.z; dst[kb][7] = hi.w;
        }
      };
      if (n_it > 0) load_items(breg, 0);
      const float4* ua = reinterpret_cast<const float4*>(sm_users);
      for (int it = 0; it < n_it; ++it) {
        if (it + 1 < n_it) load_items(bnext, it + 1);             // in flight while this item tile is expanded
        for (int uq = 0; uq < uq_count; ++uq) {
#pragma unroll
          for (int kb = 0; kb < NKB; ++kb) {
            const uint32_t s = cnt % NS, ph = (cnt / NS) & 1u;
            ap_mbar_wait(&a_empty[s], ph ^ 1u);
            unsigned char* st = sm_ring + (size_t)s * STAGE;
#pragma unroll
            for (int j = 0; j < 4; ++j) {                          // the 4 users of the quad: rows 32 j + il
              const float4* a = ua + (size_t)(uq * 4 + j) * (H1 / 4) + kb * 16 + c;
              const float4 a0 = a[0], a1 = a[8];
              const float h[8] = {a0.x + breg[kb][0], a0.y + breg[kb][1], a0.z + breg[kb][2], a0.w + breg[kb][3],
                                  a1.x + breg[kb][4], a1.y + breg[kb][5], a1.z + breg[kb][6], a1.w + breg[kb][7]};
              uint4 q;
              q.x = ap_pack_relu(h[0], h[1]); q.y = ap_pack_relu(h[2], h[3]);
              q.z = ap_pack_relu(h[4], h[5]); q.w = ap_pack_relu(h[6], h[7]);
              *reinterpret_cast<uint4*>(st + soff + j * 4096) = q;
              const uint32_t qq[4] = {q.x, q.y, q.z, q.w};         // lo plane: bf16(relu(h) - hi)
              uint32_t r[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const float l0 = fmaxf(h[2 * e], 0.f) - __uint_as_float(qq[e] << 16);
                const float l1 = fmaxf(h[2 * e + 1], 0.f) - __uint_as_float(qq[e] & 0xffff0000u);
                r[e] = ap_pack(l0, l1);
              }
              *reinterpret_cast<uint4*>(st + AP_TILE + soff + j * 4096) = make_uint4(r[0], r[1], r[2], r[3]);
            }
            ap_fence_async();
            ap_mbar_arrive(&a_full[s]);
            ++cnt;
          }
        }
        if (it + 1 < n_it) {
#pragma unroll
          for (int kb = 0; kb < NKB; ++kb)
#pragma unroll
            for (int e = 0; e < 8; ++e) breg[kb][e] = bnext[kb][e];
        }
      }
    }
  } else if (warp < 12) {
    // ===================== epilogue: b2 / ReLU / w3 / b3, per-user top-k =====================
    const int e = warp - 8;                                       // TMEM lanes 32 e .. 32 e + 31 = user e of every quad
    for (int ul = e; ul < UT; ul += 4) {
      sm_lv[ul * AP_KMAX + lane] = -INFINITY; sm_lv[ul * AP_KMAX + lane + 32] = -INFINITY;
      sm_li[ul * AP_KMAX + lane] = -1; sm_li[ul * AP_KMAX + lane + 32] = -1;
      if (lane == 0) sm_thr[ul] = -INFINITY;
    }
    __syncwarp();
    uint32_t t = 0;
    for (int it = 0; it < n_it; ++it) {
      const int item = i_begin + it * AP_IT + lane;
      for (int uq = 0; uq < uq_count; ++uq, ++t) {
        const uint32_t acc = t & 1u;
        ap_mbar_wait(&acc_full[acc], (t >> 1) & 1u);
        ap_tc_after();
        float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
        for (int cg = 0; cg < AP_NPAD / 32; ++cg) {
          uint32_t r[32];
          const uint32_t taddr = tmem_base + ((uint32_t)(e * 32) << 16) + acc * AP_NPAD + cg * 32;
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
          if (cg == AP_NPAD / 32 - 1) {                            // accumulator fully read: hand it back to the MMA warp
            ap_tc_before();
            ap_mbar_arrive(&acc_empty[acc]);
          }
#pragma unroll
          for (int j = 0; j < 32; j += 4) {
            const int n = cg * 32 + j;
            s0 = fmaf(fmaxf(__uint_as_float(r[j]) + p.b2[n], 0.f), p.w3[n], s0);
            s1 = fmaf(fmaxf(__uint_as_float(r[j + 1]) + p.b2[n + 1], 0.f), p.w3[n + 1], s1);
            s2 = fmaf(fmaxf(__uint_as_float(r[j + 2]) + p.b2[n + 2], 0.f), p.w3[n + 2], s2);
            s3 = fmaf(fmaxf(__uint_as_float(r[j + 3]) + p.b2[n + 3], 0.f), p.w3[n + 3], s3);
          }
        }
        const float s = ((s0 + s1) + (s2 + s3)) + p.b3;
        const int ul = uq * 4 + e, u = u0 + ul;
        const bool valid = ul < users_here && item < i_end;
        if (p.scores != nullptr && valid) p.scores[(long long)u * p.lds + item] = s;
        if (p.k > 0) {
          unsigned mask = __ballot_sync(FULL, valid && s > sm_thr[ul]);
          while (mask) {                                           // rare after the first few tiles: ~k ln(n/k) inserts per user
            const int b = __ffs(mask) - 1;
            mask &= mask - 1;
            const float cs = __shfl_sync(FULL, s, b);
            const int ci = i_begin + it * AP_IT + b;
            if (!(cs > sm_thr[ul])) continue;
            if (p.seen_ptr != nullptr) {                           // already-interacted items are not recommended
              int lo = __ldg(p.seen_ptr + u), hi = __ldg(p.seen_ptr + u + 1);
              while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldg(p.seen_idx + mid) < ci) lo = mid + 1; else hi = mid;
              }
              if (lo < __ldg(p.seen_ptr + u + 1) && __ldg(p.seen_idx + lo) == ci) continue;
            }
            ap_insert(sm_lv + ul * AP_KMAX, sm_li + ul * AP_KMAX, sm_thr + ul, p.k, cs, ci, lane);
          }
        }
      }
    }
    if (p.k > 0) {
      __syncwarp();
      for (int ul = e; ul < users_here; ul += 4) {
        const long long o = ((long long)(u0 + ul) * p.n_splits + blockIdx.y) * p.k;
        for (int j = lane; j < p.k; j += 32) { p.part_val[o + j] = sm_lv[ul * AP_KMAX + j]; p.part_idx[o + j] = sm_li[ul * AP_KMAX + j]; }
      }
    }
  } else {
    // ===================== MMA issuer (one elected lane) =====================
    if (lane == 0) {
      const uint32_t idesc = ap_idesc();
      ap_mbar_wait(&w_bar, 0);
      uint32_t cnt = 0, t = 0;
      for (int it = 0; it < n_it; ++it) {
        for (int uq = 0; uq < uq_count; ++uq, ++t) {
          const uint32_t acc = t & 1u;
          ap_mbar_wait(&acc_empty[acc], ((t >> 1) & 1u) ^ 1u);     // first use of each accumulator: returns at once
          ap_tc_after();
          const uint32_t d = tmem_base + acc * AP_NPAD;
#pragma unroll
          for (int kb = 0; kb < NKB; ++kb) {
            const uint32_t s = cnt % NS, ph = (cnt / NS) & 1u;
            ap_mbar_wait(&a_full[s], ph);
            ap_tc_after();
            const uint32_t a_hi = ap_smem_u32(sm_ring + (size_t)s * STAGE);
            const uint32_t w_hi = ap_smem_u32(sm_w2 + (size_t)kb * PLANES * AP_TILE);
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {                       // 16 bf16 (32 bytes) of K per MMA
              const uint32_t off = (uint32_t)ks * 32u;
              ap_umma(d, ap_desc(a_hi + off), ap_desc(w_hi + off), idesc, (kb > 0 || ks > 0) ? 1u : 0u);
              if constexpr (MODE == AP_BF16X2) {
                ap_umma(d, ap_desc(a_hi + off), ap_desc(w_hi + AP_TILE + off), idesc, 1u);      // hi · lo
                ap_umma(d, ap_desc(a_hi + AP_TILE + off), ap_desc(w_hi + off), idesc, 1u);      // lo · hi
              }
            }
            ap_commit(&a_empty[s]);
            ++cnt;
          }
          ap_commit(&acc_full[acc]);
        }
      }
    }
    __syncwarp();
  }
  ap_tc_before();
  __syncthreads();
  if (warp == 12) {
    ap_tc_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(256) : "memory");
  }
}

// W2 (H2, H1) fp32 -> [kb][plane] swizzled bf16 tiles (rows >= H2 zero)
template <int MODE>
__global__ void allpairs_pack_kernel(const float* __restrict__ W2, long long ldw, int H2, int H1, unsigned char* __restrict__ out) {
  constexpr int PLANES = MODE == AP_BF16 ? 1 : 2;
  const int nkb = H1 / 64;
  const int total = nkb * 128 * 8;                               // (k-block, row, 16-byte chunk)
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < total) {
    const int ch = idx & 7, r = (idx >> 3) & 127, kb = idx >> 10;
    float v[8];
#pragma unroll
    for (int e = 0; e < 8; ++e) v[e] = r < H2 ? __ldg(W2 + (long long)r * ldw + kb * 64 + ch * 8 + e) : 0.f;
    unsigned char* base = out + (size_t)kb * PLANES * AP_TILE;
    const uint32_t off = (uint32_t)(r >> 3) * 1024u + (uint32_t)(r & 7) * 128u + (uint32_t)((ch ^ (r & 7)) << 4);
    uint32_t hi[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) hi[e] = ap_pack(v[2 * e], v[2 * e + 1]);
    *reinterpret_cast<uint4*>(base + off) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    if constexpr (MODE == AP_BF16X2) {
      uint32_t lo[4];
#pragma unroll
      for (int e = 0; e < 4; ++e)
        lo[e] = ap_pack(v[2 * e] - __uint_as_float(hi[e] << 16), v[2 * e + 1] - __uint_as_float(hi[e] & 0xffff0000u));
      *reinterpret_cast<uint4*>(base + AP_TILE + off) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
  }
}

// merges the per-split partial lists of one user (each sorted descending) into the final top-k; one warp per user
__global__ void __launch_bounds__(128)
allpairs_merge_kernel(const float* __restrict__ part_val, const int* __restrict__ part_idx, int nU, int n_splits, int k,
                      float* __restrict__ out_val, int64_t* __restrict__ out_idx) {
  const int lane = threadIdx.x & 31;
  const int u = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (u >= nU) return;
  const float* pv = part_val + (long long)u * n_splits * k;
  const int* pi = part_idx + (long long)u * n_splits * k;
  // lane owns the splits lane, lane+32, ...; `head` = how many entries of each owned list have been consumed (<= 4 lists/lane)
  int head[4] = {0, 0, 0, 0};
  for (int round = 0; round < k; ++round) {
    float bv = -INFINITY;
    int bi = -1, bs = -1;
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int s = lane + 32 * q;
      if (s < n_splits && head[q] < k) {
        const float v = pv[(long long)s * k + head[q]];
        const int i = pi[(long long)s * k + head[q]];
        if (i >= 0 && (bi < 0 || v > bv || (v == bv && i < bi))) { bv = v; bi = i; bs = q; }
      }
    }
    float wv = bv; int wi = bi, wl = lane;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(FULL, wv, o);
      const int oi = __shfl_xor_sync(FULL, wi, o), ol = __shfl_xor_sync(FULL, wl, o);
      if (oi >= 0 && (wi < 0 || ov > wv || (ov == wv && oi < wi))) { wv = ov; wi = oi; wl = ol; }
    }
    if (wl == lane && bs >= 0 && wi >= 0) {
#pragma unroll
      for (int q = 0; q < 4; ++q) if (q == bs) ++head[q];
    }
    if (lane == 0) {
      out_val[(long long)u * k + round] = wi >= 0 ? wv : -INFINITY;
      out_idx[(long long)u * k + round] = wi;
    }
  }
}

// ---------------------------------------------------------------------------------------------------------------------------------
// One-hidden-layer MLPs ([256] — train_model.py:41, the reference's fixed-profile experiments) in all-pairs mode degenerate to
//     score(u, i) = b2 + sum_h w2[h] * ReLU(a_u[h] + b_i[h])                     (SURVEY.md §8d: ~3·H1 FP32 operations per pair, NO GEMM)
// Through the tensor-core kernel above this costs a 2-row MMA per tile and the bf16 hi/lo split of BOTH operands of the only dot
// product there is (measured 1.1e-5 at F = 2094: over the fp32 budget).  Here it runs where it belongs, on the FP32 pipes, exactly:
// CTA = 64 users x 128-item tiles, a thread owns 4 users x 8 items = 32 accumulators and walks h through shared memory
// (user rows resident, item tile transposed to h-major so that a warp's 16 item columns are conflict-free); per h and pair one FADD,
// one FMNMX, one FFMA.  Same top-k epilogue / split lists / merge kernel as the tensor-core path.
//
// DOT = true is the dot-product model's form of the same kernel, score(u, i) = A[u]·B[i] (GraphNCF(use_dot_product=True) over a
// partitioned graph, peer.recommend_peer): one FFMA per h and pair and no w2 / b2.  The top-k never needs the (nU x nI) score matrix,
// which a GEMM + row-wise top-k would have to write (5 TB for one rank of BASELINE configs[4]).
constexpr int RD_UT = 64, RD_IT = 128, RD_HC = 64, RD_THREADS = 256;

struct ReluDotParams {
  const float* A; const float* B; const float* w2; float b2;
  int nU, nI, H1;
  int k, n_splits, items_per_split;
  float* part_val; int* part_idx;
  float* scores; long long lds;
  const int* seen_ptr; const int* seen_idx;
};

template <bool DOT>
__global__ void __launch_bounds__(RD_THREADS, 1)
allpairs_relu_dot_kernel(const ReluDotParams p) {
  extern __shared__ __align__(16) unsigned char rd_smem[];
  float* sA = reinterpret_cast<float*>(rd_smem);                       // [RD_UT][H1]
  float* sW = sA + RD_UT * p.H1;                                        // [H1]
  float* sB = sW + p.H1;                                                // [2][RD_HC][RD_IT]  (h-major)
  float* sS = sB + 2 * RD_HC * RD_IT;                                   // [RD_UT][RD_IT] scores of the current tile
  float* sm_lv = sS + RD_UT * RD_IT;                                    // [RD_UT][AP_KMAX]
  int* sm_li = reinterpret_cast<int*>(sm_lv + RD_UT * AP_KMAX);
  float* sm_thr = reinterpret_cast<float*>(sm_li + RD_UT * AP_KMAX);    // [RD_UT]
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int ty = tid >> 4, tx = tid & 15;                               // users ty + 16 q, items tx + 16 j
  const int u0 = blockIdx.x * RD_UT;
  const int users_here = min(RD_UT, p.nU - u0);
  const int i_begin = blockIdx.y * p.items_per_split, i_end = min(p.nI, i_begin + p.items_per_split);
  const int H1 = p.H1, n_hc = H1 / RD_HC;
  for (int i = tid; i < RD_UT * H1 / 4; i += RD_THREADS) {              // user rows (zero rows beyond the last user)
    const int r = (i * 4) / H1, c = (i * 4) % H1;
    reinterpret_cast<float4*>(sA)[i] = r < users_here ? __ldg(reinterpret_cast<const float4*>(p.A + (long long)(u0 + r) * H1 + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  if constexpr (!DOT)
    for (int i = tid; i < H1; i += RD_THREADS) sW[i] = __ldg(p.w2 + i);
  for (int i = tid; i < RD_UT * AP_KMAX; i += RD_THREADS) { sm_lv[i] = -INFINITY; sm_li[i] = -1; }
  if (tid < RD_UT) sm_thr[tid] = -INFINITY;
  __syncthreads();
  const int n_it = (i_end - i_begin + RD_IT - 1) / RD_IT;
  // item-tile chunk (RD_IT items x RD_HC h) global -> registers -> transposed shared memory: thread = (item = tid / 2 [+0], 32 h)
  const int l_item = tid >> 1, l_h0 = (tid & 1) * 32;
  float4 pre[8];
  auto load_chunk = [&](int it, int hc) {
    const int item = min(i_begin + it * RD_IT + l_item, p.nI - 1);
    const float* src = p.B + (long long)item * H1 + hc * RD_HC + l_h0;
#pragma unroll
    for (int q = 0; q < 8; ++q) pre[q] = __ldg(reinterpret_cast<const float4*>(src) + q);
  };
  auto store_chunk = [&](int buf) {
    float* dst = sB + buf * RD_HC * RD_IT;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
      const int h = l_h0 + 4 * q;
      dst[(h + 0) * RD_IT + l_item] = pre[q].x; dst[(h + 1) * RD_IT + l_item] = pre[q].y;
      dst[(h + 2) * RD_IT + l_item] = pre[q].z; dst[(h + 3) * RD_IT + l_item] = pre[q].w;
    }
  };
  if (n_it > 0) load_chunk(0, 0);
  int step = 0;
  for (int it = 0; it < n_it; ++it) {
    float acc[4][8];
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[q][j] = 0.f;
    for (int hc = 0; hc < n_hc; ++hc, ++step) {
      const int buf = step & 1;
      store_chunk(buf);                                                 // (buffer `buf` was last read two chunks ago: a barrier has passed since)
      __syncthreads();
      const int nhc = hc + 1 < n_hc ? hc + 1 : 0, nit = hc + 1 < n_hc ? it : it + 1;
      if (nit < n_it) load_chunk(nit, nhc);                             // next chunk's global loads fly under this chunk's arithmetic
      const float* bt = sB + buf * RD_HC * RD_IT + tx;
      const float* at = sA + ty * H1 + hc * RD_HC;
      const float* wt = sW + hc * RD_HC;
#pragma unroll 4
      for (int h = 0; h < RD_HC; ++h) {
        [[maybe_unused]] const float w = DOT ? 0.f : wt[h];
        float a[4], b[8];
#pragma unroll
        for (int q = 0; q < 4; ++q) a[q] = at[q * 16 * H1 + h];
#pragma unroll
        for (int j = 0; j < 8; ++j) b[j] = bt[h * RD_IT + 16 * j];
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if constexpr (DOT) acc[q][j] = fmaf(a[q], b[j], acc[q][j]);
            else acc[q][j] = fmaf(w, fmaxf(a[q] + b[j], 0.f), acc[q][j]);
          }
      }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
#pragma unroll
      for (int j = 0; j < 8; ++j) sS[(ty + 16 * q) * RD_IT + tx + 16 * j] = DOT ? acc[q][j] : acc[q][j] + p.b2;
    __syncthreads();
    // ---- tile epilogue: warp w owns users w, w + 8, ... ----
    for (int ul = warp; ul < users_here; ul += RD_THREADS / 32) {
      const int u = u0 + ul;
#pragma unroll 1
      for (int q = 0; q < RD_IT / 32; ++q) {
        const int item = i_begin + it * RD_IT + q * 32 + lane;
        const float sc = sS[ul * RD_IT + q * 32 + lane];
        const bool valid = item < i_end;
        if (p.scores != nullptr && valid) p.scores[(long long)u * p.lds + item] = sc;
        if (p.k > 0) {
          unsigned mask = __ballot_sync(FULL, valid && sc > sm_thr[ul]);
          while (mask) {
            const int b = __ffs(mask) - 1;
            mask &= mask - 1;
            const float cs = __shfl_sync(FULL, sc, b);
            const int ci = i_begin + it * RD_IT + q * 32 + b;
            if (!(cs > sm_thr[ul])) continue;
            if (p.seen_ptr != nullptr) {
              int lo = __ldg(p.seen_ptr + u), hi = __ldg(p.seen_ptr + u + 1);
              while (lo < hi) {
                const int mid = (lo + hi) >> 1;
                if (__ldg(p.seen_idx + mid) < ci) lo = mid + 1; else hi = mid;
              }
              if (lo < __ldg(p.seen_ptr + u + 1) && __ldg(p.seen_idx + lo) == ci) continue;
            }
            ap_insert(sm_lv + ul * AP_KMAX, sm_li + ul * AP_KMAX, sm_thr + ul, p.k, cs, ci, lane);
          }
        }
      }
    }
    __syncthreads();
  }
  if (p.k > 0) {
    for (int ul = warp; ul < users_here; ul += RD_THREADS / 32) {
      const long long o = ((long long)(u0 + ul) * p.n_splits + blockIdx.y) * p.k;
      for (int j = lane; j < p.k; j += 32) { p.part_val[o + j] = sm_lv[ul * AP_KMAX + j]; p.part_idx[o + j] = sm_li[ul * AP_KMAX + j]; }
    }
  }
}

static size_t rd_smem_bytes(int H1) {
  return (size_t)(RD_UT * H1 + H1 + 2 * RD_HC * RD_IT + RD_UT * RD_IT + 2 * RD_UT * AP_KMAX + RD_UT) * 4 + 16;
}

static size_t ap_packed_bytes(int H1, int mode) {
  return (size_t)(H1 / 64) * (mode == AP_BF16 ? 1 : 2) * AP_TILE;
}

template <int MODE, int UQ, int NKB>
static int ap_launch(const AllPairsParams& p, dim3 grid, cudaStream_t st) {
  const size_t smem = ApLayout<MODE, UQ>::total(NKB);
  static B200recSmemOptIn opted;
  B200REC_CUDA(b200rec_opt_in_smem(opted, allpairs_topk_kernel<MODE, UQ, NKB>, (int)smem));
  allpairs_topk_kernel<MODE, UQ, NKB><<<grid, AP_THREADS, smem, st>>>(p);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

template <int MODE, int UQ>
static int ap_dispatch(const AllPairsParams& p, dim3 grid, cudaStream_t st) {
  switch (p.H1 / 64) {
    case 1: return ap_launch<MODE, UQ, 1>(p, grid, st);
    case 2: return ap_launch<MODE, UQ, 2>(p, grid, st);
    case 3: return ap_launch<MODE, UQ, 3>(p, grid, st);
    case 4: return ap_launch<MODE, UQ, 4>(p, grid, st);
  }
  return b200rec_fail(B200REC_ERR_UNSUPPORTED, "allpairs: H1 must be 64, 128, 192 or 256");
}

constexpr int AP_UQ_BF16 = 8, AP_UQ_X2 = 4;

static int ap_users_per_cta(int mode) { return 4 * (mode == AP_BF16 ? AP_UQ_BF16 : AP_UQ_X2); }

// item splits: at least one CTA per SM where the items allow it (>= 256 items per split, <= 128 splits), and among the
// candidates up to four waves the count that leaves the smallest idle tail in the last wave
static int ap_auto_splits(int64_t nU, int64_t nI, int mode) {
  const int64_t ublocks = (nU + ap_users_per_cta(mode) - 1) / ap_users_per_cta(mode);
  const int64_t sms = b200rec_num_sms();
  int64_t smax = (nI + 255) / 256;
  if (smax > 128) smax = 128;
  if (smax < 1) smax = 1;
  if (ublocks >= 8 * sms) return 1;
  int best = 1;
  double best_eff = 0.0;
  for (int64_t s = 1; s <= smax; ++s) {
    const int64_t ctas = ublocks * s, waves = (ctas + sms - 1) / sms;
    const double eff = (double)ctas / (double)(waves * sms);
    if (eff > best_eff + 0.02) { best_eff = eff; best = (int)s; }
    if (waves > 4) break;
  }
  return best;
}

}  // namespace b200rec

using namespace b200rec;

extern "C" size_t b200rec_allpairs_packed_bytes(int H1, int mode) {
  if (H1 <= 0 || H1 > 256 || (H1 % 64) || (mode != AP_BF16 && mode != AP_BF16X2)) return 0;
  return ap_packed_bytes(H1, mode);
}

extern "C" int b200rec_allpairs_pack(const float* W2, int64_t ldw2, int H2, int H1, int mode, void* packed, size_t packed_bytes,
                                     b200rec_stream_t stream) {
  if (!W2 || !packed || H2 <= 0 || H2 > AP_NPAD || H1 <= 0 || H1 > 256 || (H1 % 64) || ldw2 < H1)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_pack: need H2 <= 128, H1 in {64,128,192,256} (zero-pad the inputs), ldw2 >= H1");
  if (mode != AP_BF16 && mode != AP_BF16X2) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_pack: bad mode");
  if (packed_bytes < ap_packed_bytes(H1, mode) || ((uintptr_t)packed % 128))
    return b200rec_fail(B200REC_ERR_WORKSPACE, "allpairs_pack: buffer too small or not 128-byte aligned");
  const int total = (H1 / 64) * 128 * 8;
  const int grid = (total + 255) / 256;
  cudaStream_t st = (cudaStream_t)stream;
  if (mode == AP_BF16) allpairs_pack_kernel<AP_BF16><<<grid, 256, 0, st>>>(W2, ldw2, H2, H1, (unsigned char*)packed);
  else allpairs_pack_kernel<AP_BF16X2><<<grid, 256, 0, st>>>(W2, ldw2, H2, H1, (unsigned char*)packed);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_allpairs_splits(int64_t nU, int64_t nI, int mode) {
  if (nU <= 0 || nI <= 0) return 1;
  return ap_auto_splits(nU, nI, mode);
}

extern "C" size_t b200rec_allpairs_workspace(int64_t nU, int k, int n_splits) {
  if (nU <= 0 || k <= 0 || n_splits <= 0) return 0;
  return (size_t)nU * n_splits * k * (sizeof(float) + sizeof(int)) + 256;
}

extern "C" int b200rec_allpairs_topk(const float* A, const float* B, int64_t nU, int64_t nI, int H1, const void* packed,
                                     const float* epilogue_host, int H2, int mode, int k, int n_splits, const int32_t* seen_ptr, const int32_t* seen_idx, float* scores, int64_t lds,
                                     float* top_val, int64_t* top_idx, void* workspace, size_t workspace_bytes,
                                     b200rec_stream_t stream) {
  if (nU < 0 || nI < 0 || !packed || !epilogue_host || (nU > 0 && nI > 0 && (!A || !B))) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: null operand");
  if (H2 <= 0 || H2 > AP_NPAD) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "allpairs_topk: H2 must be in 1..128");
  if (H1 <= 0 || H1 > 256 || (H1 % 64)) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "allpairs_topk: H1 must be 64, 128, 192 or 256 (zero-pad)");
  if (mode != AP_BF16 && mode != AP_BF16X2) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: bad mode");
  if (k < 0 || k > AP_KMAX) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: need 0 <= k <= 64");
  if (k > 0 && (!top_val || !top_idx)) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: top-k outputs missing");
  if (k == 0 && !scores) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: nothing to compute (k = 0 and no score buffer)");
  if (scores && lds < nI) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: lds too small");
  if ((seen_ptr == nullptr) != (seen_idx == nullptr)) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: seen CSR needs both arrays");
  if (nU > INT32_MAX / 2 || nI > INT32_MAX / 2) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "allpairs_topk: dims > 2^30");
  if ((uintptr_t)A % 16 || (uintptr_t)B % 16 || (uintptr_t)packed % 128) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: operands must be 16-byte (packed: 128-byte) aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (nU == 0) return B200REC_OK;
  if (n_splits <= 0) n_splits = nI > 0 ? ap_auto_splits(nU, nI, mode) : 1;
  if (n_splits > 128) return b200rec_fail(B200REC_ERR_BAD_ARG, "allpairs_topk: at most 128 item splits");
  if (k > 0 && (!workspace || workspace_bytes < b200rec_allpairs_workspace(nU, k, n_splits) || (uintptr_t)workspace % 16))
    return b200rec_fail(B200REC_ERR_WORKSPACE, "allpairs_topk: workspace too small (b200rec_allpairs_workspace)");
  AllPairsParams p;
  p.A = A; p.B = B; p.nU = (int)nU; p.nI = (int)nI; p.H1 = H1; p.Wp = (const unsigned char*)packed; p.k = k;
  p.n_splits = n_splits;
  p.items_per_split = (int)(((nI + n_splits - 1) / n_splits + AP_IT - 1) / AP_IT * AP_IT);
  if (p.items_per_split < AP_IT) p.items_per_split = AP_IT;
  p.part_val = reinterpret_cast<float*>(workspace);
  p.part_idx = k > 0 ? reinterpret_cast<int*>(p.part_val + (size_t)nU * n_splits * k) : nullptr;
  p.scores = scores; p.lds = lds; p.seen_ptr = seen_ptr; p.seen_idx = seen_idx;
  for (int n = 0; n < AP_NPAD; ++n) {            // host block: b2[H2] | w3[H2] | b3; padded columns contribute ReLU(0 + 0) * 0
    p.b2[n] = n < H2 ? epilogue_host[n] : 0.f;
    p.w3[n] = n < H2 ? epilogue_host[H2 + n] : 0.f;
  }
  p.b3 = epilogue_host[2 * H2];
  const int ut = ap_users_per_cta(mode);
  dim3 grid((unsigned)((nU + ut - 1) / ut), (unsigned)n_splits);
  if (nI > 0) {
    const int rc = mode == AP_BF16 ? ap_dispatch<AP_BF16, AP_UQ_BF16>(p, grid, st) : ap_dispatch<AP_BF16X2, AP_UQ_X2>(p, grid, st);
    if (rc) return rc;
  } else if (k > 0) {
    B200REC_CUDA(cudaMemsetAsync(p.part_idx, 0xff, (size_t)nU * n_splits * k * sizeof(int), st));
  }
  if (k > 0) {
    allpairs_merge_kernel<<<(unsigned)((nU + 3) / 4), 128, 0, st>>>(p.part_val, p.part_idx, (int)nU, n_splits, k, top_val, top_idx);
    B200REC_CHECK_LAUNCH();
  }
  return B200REC_OK;
}

static int rd_auto_splits(int64_t nU, int64_t nI) {
  const int64_t ublocks = (nU + RD_UT - 1) / RD_UT;
  const int sms = b200rec_num_sms();
  int64_t splits = ublocks >= sms ? 1 : (2 * sms + ublocks - 1) / ublocks;
  const int64_t max_splits = (nI + RD_IT - 1) / RD_IT;
  if (splits > max_splits) splits = max_splits;
  if (splits > 128) splits = 128;
  return (int)(splits < 1 ? 1 : splits);
}

extern "C" int b200rec_allpairs_relu_dot_splits(int64_t nU, int64_t nI) { return (nU <= 0 || nI <= 0) ? 1 : rd_auto_splits(nU, nI); }

// the checks, split lists and merge of both instantiations; `what` names the entry point in the error messages
template <bool DOT>
static int rd_topk(const char* const (&what)[11], const float* A, const float* B, int64_t nU, int64_t nI, int H1, const float* w2, float b2, int k,
                   int n_splits, const int* seen_ptr, const int* seen_idx, float* scores, int64_t lds, float* top_val, int64_t* top_idx,
                   void* workspace, size_t workspace_bytes, cudaStream_t st) {
  if (nU < 0 || nI < 0 || (!DOT && !w2) || (nU > 0 && nI > 0 && (!A || !B))) return b200rec_fail(B200REC_ERR_BAD_ARG, what[0]);
  if (H1 <= 0 || H1 > 256 || (H1 % 64)) return b200rec_fail(B200REC_ERR_UNSUPPORTED, what[1]);
  if (k < 0 || k > AP_KMAX) return b200rec_fail(B200REC_ERR_BAD_ARG, what[2]);
  if (k > 0 && (!top_val || !top_idx)) return b200rec_fail(B200REC_ERR_BAD_ARG, what[3]);
  if (k == 0 && !scores) return b200rec_fail(B200REC_ERR_BAD_ARG, what[4]);
  if (scores && lds < nI) return b200rec_fail(B200REC_ERR_BAD_ARG, what[5]);
  if ((seen_ptr == nullptr) != (seen_idx == nullptr)) return b200rec_fail(B200REC_ERR_BAD_ARG, what[6]);
  if (nU > INT32_MAX / 2 || nI > INT32_MAX / 2) return b200rec_fail(B200REC_ERR_UNSUPPORTED, what[7]);
  if ((uintptr_t)A % 16 || (uintptr_t)B % 16) return b200rec_fail(B200REC_ERR_BAD_ARG, what[8]);
  if (nU == 0) return B200REC_OK;
  if (n_splits <= 0) n_splits = nI > 0 ? rd_auto_splits(nU, nI) : 1;
  if (n_splits > 128) return b200rec_fail(B200REC_ERR_BAD_ARG, what[9]);
  if (k > 0 && (!workspace || workspace_bytes < b200rec_allpairs_workspace(nU, k, n_splits) || (uintptr_t)workspace % 16))
    return b200rec_fail(B200REC_ERR_WORKSPACE, what[10]);
  ReluDotParams p;
  p.A = A; p.B = B; p.w2 = w2; p.b2 = b2; p.nU = (int)nU; p.nI = (int)nI; p.H1 = H1; p.k = k; p.n_splits = n_splits;
  p.items_per_split = (int)(((nI + n_splits - 1) / n_splits + RD_IT - 1) / RD_IT * RD_IT);
  if (p.items_per_split < RD_IT) p.items_per_split = RD_IT;
  p.part_val = reinterpret_cast<float*>(workspace);
  p.part_idx = k > 0 ? reinterpret_cast<int*>(p.part_val + (size_t)nU * n_splits * k) : nullptr;
  p.scores = scores; p.lds = lds; p.seen_ptr = seen_ptr; p.seen_idx = seen_idx;
  if (nI > 0) {
    const size_t smem = rd_smem_bytes(H1);
    static B200recSmemOptIn opted;
    B200REC_CUDA(b200rec_opt_in_smem(opted, allpairs_relu_dot_kernel<DOT>, (int)rd_smem_bytes(256)));
    dim3 grid((unsigned)((nU + RD_UT - 1) / RD_UT), (unsigned)n_splits);
    allpairs_relu_dot_kernel<DOT><<<grid, RD_THREADS, smem, st>>>(p);
    B200REC_CHECK_LAUNCH();
  } else if (k > 0) {
    B200REC_CUDA(cudaMemsetAsync(p.part_idx, 0xff, (size_t)nU * n_splits * k * sizeof(int), st));
  }
  if (k > 0) {
    allpairs_merge_kernel<<<(unsigned)((nU + 3) / 4), 128, 0, st>>>(p.part_val, p.part_idx, (int)nU, n_splits, k, top_val, top_idx);
    B200REC_CHECK_LAUNCH();
  }
  return B200REC_OK;
}

extern "C" int b200rec_allpairs_relu_dot_topk(const float* A, const float* B, int64_t nU, int64_t nI, int H1, const float* w2, float b2, int k,
                                              int n_splits, const int* seen_ptr, const int* seen_idx, float* scores, int64_t lds, float* top_val,
                                              int64_t* top_idx, void* workspace, size_t workspace_bytes, b200rec_stream_t stream) {
  static const char* const what[11] = {
      "allpairs_relu_dot: null operand", "allpairs_relu_dot: H1 must be 64, 128, 192 or 256 (zero-pad)", "allpairs_relu_dot: need 0 <= k <= 64",
      "allpairs_relu_dot: top-k outputs missing", "allpairs_relu_dot: nothing to compute", "allpairs_relu_dot: lds too small",
      "allpairs_relu_dot: seen CSR needs both arrays", "allpairs_relu_dot: dims > 2^30", "allpairs_relu_dot: A / B must be 16-byte aligned",
      "allpairs_relu_dot: at most 128 item splits", "allpairs_relu_dot: workspace too small (b200rec_allpairs_workspace)"};
  return rd_topk<false>(what, A, B, nU, nI, H1, w2, b2, k, n_splits, seen_ptr, seen_idx, scores, lds, top_val, top_idx, workspace, workspace_bytes,
                        (cudaStream_t)stream);
}

extern "C" int b200rec_allpairs_dot_topk(const float* A, const float* B, int64_t nU, int64_t nI, int H, int k, int n_splits, const int* seen_ptr,
                                         const int* seen_idx, float* scores, int64_t lds, float* top_val, int64_t* top_idx, void* workspace,
                                         size_t workspace_bytes, b200rec_stream_t stream) {
  static const char* const what[11] = {
      "allpairs_dot: null operand", "allpairs_dot: H must be 64, 128, 192 or 256 (zero-pad)", "allpairs_dot: need 0 <= k <= 64",
      "allpairs_dot: top-k outputs missing", "allpairs_dot: nothing to compute", "allpairs_dot: lds too small",
      "allpairs_dot: seen CSR needs both arrays", "allpairs_dot: dims > 2^30", "allpairs_dot: A / B must be 16-byte aligned",
      "allpairs_dot: at most 128 item splits", "allpairs_dot: workspace too small (b200rec_allpairs_workspace)"};
  return rd_topk<true>(what, A, B, nU, nI, H, nullptr, 0.f, k, n_splits, seen_ptr, seen_idx, scores, lds, top_val, top_idx, workspace, workspace_bytes,
                       (cudaStream_t)stream);
}
