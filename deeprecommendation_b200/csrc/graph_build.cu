// K4 — neighbour-index build, on device, bit-exact against the reference's `create_graph`
// (src/content_providers/graph_providers.py:10-66) and node-id assignment (:76-80).
//
// The reference walks the interactions with a Python `iterrows()` loop (minutes at 1e6 rows, infeasible at 2.5e7).
// Here every stage is a data-parallel kernel over HBM-resident arrays:
//   1. sorted-unique id -> node id      presence flags + exclusive scan (ids are bounded integers)
//   2. per-user / per-item mean rating  fp64 atomics — exact, hence order-independent, for ratings on the
//                                       half-star grid (all partial sums are representable); pandas' mean (:16-17)
//                                       is sum/count in fp64, reproduced bit for bit
//   3. the two COO edge lists + centred-rating attrs in file order (:26-47); `binary` = stable compaction
//   4. CSR by destination               stable LSD radix sort (8-bit digits) of (dst, position); ties keep file
//                                       order = the order the reference's CPU index_add_ accumulates in
//   5. chunk plan for the edge-balanced SpMM (K3), deg^-1/2, the (src,dst)->position hash (replaces `pos_df`)
//      and the per-batch target-edge skip bitmap (replaces gnn_ncf.py:369-378)
// All index arithmetic is integer and deterministic; tests compare every output array with == against the oracle.
#include "common.cuh"

namespace b200rec {

// ------------------------------------------------------------------------------------------------------------
// exclusive scan, int32, n+1 outputs (out[n] = total).  Recursive 3-phase (tile scan, scan of tile sums, add).
// ------------------------------------------------------------------------------------------------------------
constexpr int SCAN_THREADS = 256;
constexpr int SCAN_ITEMS = 8;
constexpr int SCAN_TILE = SCAN_THREADS * SCAN_ITEMS;

__global__ void __launch_bounds__(SCAN_THREADS)
scan_tile_kernel(const int* __restrict__ in, long long n_in, int* __restrict__ out, long long n_out, int* __restrict__ tile_sums) {
  __shared__ int warp_tot[SCAN_THREADS / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const long long base = (long long)blockIdx.x * SCAN_TILE + (long long)tid * SCAN_ITEMS;
  int v[SCAN_ITEMS];
  int sum = 0;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    const long long idx = base + i;
    v[i] = (idx < n_in) ? in[idx] : 0;
    sum += v[i];
  }
  int incl = sum;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    int t = __shfl_up_sync(FULL, incl, o);
    if (lane >= o) incl += t;
  }
  if (lane == 31) warp_tot[warp] = incl;
  __syncthreads();
  if (warp == 0) {
    int w = (lane < SCAN_THREADS / 32) ? warp_tot[lane] : 0;
    int wi = w;
#pragma unroll
    for (int o = 1; o < SCAN_THREADS / 32; o <<= 1) {
      int t = __shfl_up_sync(FULL, wi, o);
      if (lane >= o) wi += t;
    }
    if (lane < SCAN_THREADS / 32) warp_tot[lane] = wi - w;     // exclusive warp offsets
    if (lane == SCAN_THREADS / 32 - 1 && tile_sums) tile_sums[blockIdx.x] = wi;
  }
  __syncthreads();
  int run = warp_tot[warp] + incl - sum;
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    const long long idx = base + i;
    if (idx < n_out) out[idx] = run;
    run += v[i];
  }
}

__global__ void scan_add_kernel(int* __restrict__ out, long long n_out, const int* __restrict__ tile_offsets) {
  const long long idx = (long long)blockIdx.x * SCAN_TILE + threadIdx.x;
  const int off = tile_offsets[blockIdx.x];
#pragma unroll
  for (int i = 0; i < SCAN_ITEMS; ++i) {
    const long long j = idx + (long long)i * SCAN_THREADS;
    if (j < n_out) out[j] += off;
  }
}

static size_t scan_workspace_ints(long long n_out) {
  size_t total = 0;
  long long n = n_out;
  while (n > SCAN_TILE) {
    long long tiles = (n + SCAN_TILE - 1) / SCAN_TILE;
    total += (size_t)tiles + 1;
    n = tiles + 1;
  }
  return total + 2;
}

// out has n+1 entries; ws holds scan_workspace_ints(n+1) ints
static int exclusive_scan(const int* in, long long n, int* out, int* ws, cudaStream_t st) {
  const long long n_out = n + 1;
  const long long tiles = (n_out + SCAN_TILE - 1) / SCAN_TILE;
  if (tiles == 1) {
    scan_tile_kernel<<<1, SCAN_THREADS, 0, st>>>(in, n, out, n_out, nullptr);
    B200REC_CHECK_LAUNCH();
    return B200REC_OK;
  }
  int* sums = ws;                       // [tiles] then scanned in place into [tiles+1]
  scan_tile_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(in, n, out, n_out, sums);
  B200REC_CHECK_LAUNCH();
  int* sums_scanned = ws + tiles + 1;   // next level's output lives after this level's sums
  // scan the tile sums into a separate array of tiles+1 entries
  int rc = exclusive_scan(sums, tiles, sums_scanned, sums_scanned + tiles + 1, st);
  if (rc) return rc;
  scan_add_kernel<<<(unsigned)tiles, SCAN_THREADS, 0, st>>>(out, n_out, sums_scanned);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

static size_t scan_ws_bytes(long long n) {
  // conservative: each level needs sums[tiles] + scanned[tiles+1] (+ recursion)
  size_t total = 0;
  long long m = n + 1;
  while (m > SCAN_TILE) {
    long long tiles = (m + SCAN_TILE - 1) / SCAN_TILE;
    total += (size_t)(2 * tiles + 4);
    m = tiles + 1;
  }
  return (total + 16) * sizeof(int);
}

// ------------------------------------------------------------------------------------------------------------
// stable LSD radix sort of (key int32 >= 0, value int32), 8-bit digits
// ------------------------------------------------------------------------------------------------------------
constexpr int RS_THREADS = 256;
constexpr int RS_ITEMS = 16;                       // consecutive elements per thread-round layout: warp-contiguous
constexpr int RS_TILE = RS_THREADS * RS_ITEMS;     // 4096 keys per CTA
constexpr int RS_WARPS = RS_THREADS / 32;

__global__ void __launch_bounds__(RS_THREADS)
radix_hist_kernel(const int* __restrict__ keys, long long n, int shift, int* __restrict__ hist, int n_blocks) {
  __shared__ int h[256];
  for (int i = threadIdx.x; i < 256; i += RS_THREADS) h[i] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * RS_TILE;
  for (int i = threadIdx.x; i < RS_TILE; i += RS_THREADS) {
    const long long idx = base + i;
    if (idx < n) atomicAdd(&h[(keys[idx] >> shift) & 255], 1);
  }
  __syncthreads();
  // digit-major layout so that one flat exclusive scan yields the global offsets
  for (int i = threadIdx.x; i < 256; i += RS_THREADS) hist[(long long)i * n_blocks + blockIdx.x] = h[i];
}

__global__ void __launch_bounds__(RS_THREADS)
radix_scatter_kernel(const int* __restrict__ keys_in, const int* __restrict__ vals_in, long long n, int shift,
                     const int* __restrict__ offsets, int n_blocks, int* __restrict__ keys_out, int* __restrict__ vals_out) {
  __shared__ int wh[RS_WARPS][256];        // per-warp digit counts -> exclusive prefix over warps
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  for (int i = tid; i < RS_WARPS * 256; i += RS_THREADS) (&wh[0][0])[i] = 0;
  __syncthreads();
  // warp w owns the contiguous range [w*ITEMS*32, (w+1)*ITEMS*32) of the tile, walked 32 at a time: position order
  // inside the tile == (warp, round, lane) order, which keeps the sort stable.
  const long long wbase = (long long)blockIdx.x * RS_TILE + (long long)warp * RS_ITEMS * 32;
  int key[RS_ITEMS], val[RS_ITEMS], rank[RS_ITEMS];
#pragma unroll
  for (int r = 0; r < RS_ITEMS; ++r) {
    const long long idx = wbase + r * 32 + lane;
    const bool ok = idx < n;
    key[r] = ok ? keys_in[idx] : 0;
    val[r] = ok ? vals_in[idx] : 0;
    const int dg = ok ? ((key[r] >> shift) & 255) : 256;            // 256 = out of range, matches nobody valid
    const unsigned peers = __match_any_sync(FULL, dg);
    const int before = __popc(peers & ((1u << lane) - 1u));
    int prev = 0;
    if (ok) prev = wh[warp][dg];                                     // count from earlier rounds of this warp
    __syncwarp();
    if (ok && before == 0) wh[warp][dg] = prev + __popc(peers);      // one leader per digit updates
    __syncwarp();
    rank[r] = prev + before;
  }
  __syncthreads();
  // exclusive prefix over warps for every digit, plus the global offset of (digit, block)
  for (int dg = tid; dg < 256; dg += RS_THREADS) {
    int run = offsets[(long long)dg * n_blocks + blockIdx.x];
#pragma unroll
    for (int w = 0; w < RS_WARPS; ++w) {
      const int c = wh[w][dg];
      wh[w][dg] = run;
      run += c;
    }
  }
  __syncthreads();
#pragma unroll
  for (int r = 0; r < RS_ITEMS; ++r) {
    const long long idx = wbase + r * 32 + lane;
    if (idx < n) {
      const int dg = (key[r] >> shift) & 255;
      const int dst = wh[warp][dg] + rank[r];
      keys_out[dst] = key[r];
      vals_out[dst] = val[r];
    }
  }
}

__global__ void iota_kernel(int* __restrict__ v, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) v[i] = (int)i;
}

static int radix_blocks(long long n) { return (int)((n + RS_TILE - 1) / RS_TILE); }

// workspace layout (ints): keys_tmp[n] vals_tmp[n] hist[256*nb] offs[256*nb+1] scan_ws
static size_t radix_ws_bytes(long long n) {
  const long long nb = radix_blocks(n);
  return (size_t)(2 * n + 2 * 256 * nb + 8) * sizeof(int) + scan_ws_bytes(256 * nb);
}

// sorts (keys, vals) in place; key_bits = number of significant bits in the keys
static int radix_sort_pairs(int* keys, int* vals, long long n, int key_bits, void* ws, cudaStream_t st) {
  if (n == 0) return B200REC_OK;
  const int nb = radix_blocks(n);
  int* keys_tmp = (int*)ws;
  int* vals_tmp = keys_tmp + n;
  int* hist = vals_tmp + n;
  int* offs = hist + (long long)256 * nb;
  int* scan_ws = offs + (long long)256 * nb + 1;
  int* kin = keys; int* vin = vals; int* kout = keys_tmp; int* vout = vals_tmp;
  int passes = (key_bits + 7) / 8;
  if (passes < 1) passes = 1;
  if (passes & 1) {
    // odd number of passes would leave the result in the temporaries: add a pass on a zero digit (stable no-op)
    passes += 1;
  }
  for (int p = 0; p < passes; ++p) {
    const int shift = 8 * p;
    if (shift >= 32) {   // digits beyond bit 31 are all zero: the pass degenerates to a stable copy
      B200REC_CUDA(cudaMemcpyAsync(kout, kin, n * sizeof(int), cudaMemcpyDeviceToDevice, st));
      B200REC_CUDA(cudaMemcpyAsync(vout, vin, n * sizeof(int), cudaMemcpyDeviceToDevice, st));
    } else {
      radix_hist_kernel<<<nb, RS_THREADS, 0, st>>>(kin, n, shift, hist, nb);
      B200REC_CHECK_LAUNCH();
      int rc = exclusive_scan(hist, (long long)256 * nb, offs, scan_ws, st);
      if (rc) return rc;
      radix_scatter_kernel<<<nb, RS_THREADS, 0, st>>>(kin, vin, n, shift, offs, nb, kout, vout);
      B200REC_CHECK_LAUNCH();
    }
    int* t = kin; kin = kout; kout = t;
    t = vin; vin = vout; vout = t;
  }
  return B200REC_OK;
}

// ------------------------------------------------------------------------------------------------------------
// ids, means, edges
// ------------------------------------------------------------------------------------------------------------
__global__ void mark_ids_kernel(const int64_t* __restrict__ ids, long long n, long long bound, int* __restrict__ flags,
                                int* __restrict__ err) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t id = ids[i];
  if (id < 0 || id >= bound) { *err = 1; return; }
  flags[id] = 1;
}

__global__ void lookup_ids_kernel(const int64_t* __restrict__ ids, long long n, long long bound, const int* __restrict__ flags,
                                  const int* __restrict__ rank, int64_t offset, int64_t* __restrict__ out, int* __restrict__ err) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t id = ids[i];
  if (id < 0 || id >= bound || flags[id] == 0) { *err = 1; out[i] = -1; return; }   // KeyError in the reference's dict
  out[i] = (int64_t)rank[id] + offset;
}

__global__ void unique_ids_kernel(const int* __restrict__ flags, const int* __restrict__ rank, long long bound,
                                  int64_t* __restrict__ sorted_ids) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < bound && flags[i]) sorted_ids[rank[i]] = i;
}

__global__ void group_stats_kernel(const int64_t* __restrict__ idx, const double* __restrict__ rating, long long n,
                                   int64_t idx_offset, int* __restrict__ count, double* __restrict__ sum) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t g = idx[i] - idx_offset;
  atomicAdd(count + g, 1);
  atomicAdd(sum + g, rating[i]);
}

// per interaction p (file order): centred attrs in fp64 -> fp32 and the `binary` keep flags (graph_providers.py:32-46)
__global__ void edge_attr_kernel(const int64_t* __restrict__ u_node, const int64_t* __restrict__ i_node,
                                 const double* __restrict__ rating, long long n, int64_t n_items,
                                 const int* __restrict__ cnt_u, const double* __restrict__ sum_u,
                                 const int* __restrict__ cnt_i, const double* __restrict__ sum_i,
                                 float* __restrict__ attr_u2i, float* __restrict__ attr_i2u, int* __restrict__ keep_u,
                                 int* __restrict__ keep_i) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const int64_t u = u_node[p] - n_items, it = i_node[p];
  const double r = rating[p];
  const double mean_u = sum_u[u] / (double)cnt_u[u];
  const double mean_i = sum_i[it] / (double)cnt_i[it];
  const double user_avg = (mean_u + 2.5) / 2.0;          // :32
  const double item_avg = (mean_i + 2.5) / 2.0;          // :41
  if (attr_u2i) attr_u2i[p] = (float)(r - user_avg);     // :36 then torch.tensor(dtype=float) :63
  if (attr_i2u) attr_i2u[p] = (float)(r - item_avg);     // :45, :64
  if (keep_u) keep_u[p] = (r >= user_avg) ? 1 : 0;       // :33
  if (keep_i) keep_i[p] = (r >= item_avg) ? 1 : 0;       // :42
}

// writes edge [src,dst] of interaction p at its (compacted) position; edge_index is (2, n_out) row-major int64
__global__ void edge_scatter_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, long long n,
                                    const int* __restrict__ keep, const int* __restrict__ pos, long long n_out,
                                    int64_t* __restrict__ edge_index) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  if (keep && !keep[p]) return;
  const long long q = pos ? pos[p] : p;
  edge_index[q] = src[p];
  edge_index[n_out + q] = dst[p];
}

// ------------------------------------------------------------------------------------------------------------
// CSR by destination
// ------------------------------------------------------------------------------------------------------------
__global__ void csr_keys_kernel(const int64_t* __restrict__ u2i, long long e1, const int64_t* __restrict__ i2u, long long e2,
                                int* __restrict__ keys, int* __restrict__ deg) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= e1 + e2) return;
  const int64_t d = (k < e1) ? u2i[e1 + k] : i2u[e2 + (k - e1)];       // row 1 of the (2,E) edge_index = destination
  keys[k] = (int)d;
  atomicAdd(deg + d, 1);
}

__global__ void csr_gather_kernel(const int* __restrict__ perm_comb, long long n, const int64_t* __restrict__ u2i, long long e1,
                                  const int64_t* __restrict__ i2u, long long e2, const float* __restrict__ attr_u2i,
                                  const float* __restrict__ attr_i2u, int* __restrict__ col, float* __restrict__ w,
                                  int* __restrict__ pos) {
  const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  const int q = perm_comb[k];
  if (q < e1) {
    col[k] = (int)u2i[q];
    if (w) w[k] = attr_u2i[q];
    pos[k] = q;
  } else {
    const long long r = q - e1;
    col[k] = (int)i2u[r];
    if (w) w[k] = attr_i2u[r];
    pos[k] = (int)r;
  }
}

__global__ void dinv_kernel(const int* __restrict__ deg, long long n, float* __restrict__ dinv) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int d = deg[i];
  dinv[i] = d > 0 ? 1.0f / sqrtf((float)d) : 0.f;        // deg.pow(-0.5); inf -> 0   (gnn_ncf.py:49-50)
}

// ------------------------------------------------------------------------------------------------------------
// SpMM chunk plan
// ------------------------------------------------------------------------------------------------------------
__global__ void plan_count_kernel(const int* __restrict__ row_ptr, int n_rows, int chunk, int* __restrict__ n_chunks,
                                  int* __restrict__ is_multi, int* __restrict__ n_slots) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  const int deg = row_ptr[r + 1] - row_ptr[r];
  const int c = deg <= chunk ? 1 : (deg + chunk - 1) / chunk;
  n_chunks[r] = c;
  is_multi[r] = c > 1 ? 1 : 0;
  n_slots[r] = c > 1 ? c : 0;
}

__global__ void plan_fill_kernel(const int* __restrict__ row_ptr, int n_rows, int chunk, const int* __restrict__ chunk_off,
                                 const int* __restrict__ multi_off, const int* __restrict__ slot_off, int* __restrict__ chunk_row,
                                 int* __restrict__ chunk_start, int* __restrict__ chunk_slot, int* __restrict__ multi_row,
                                 int* __restrict__ multi_first, int* __restrict__ multi_n) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  const int c0 = chunk_off[r], nc = chunk_off[r + 1] - c0;
  const int s = row_ptr[r];
  if (nc == 1) {
    chunk_row[c0] = r; chunk_start[c0] = s; chunk_slot[c0] = -1;
  } else {
    const int slot0 = slot_off[r];
    for (int j = 0; j < nc; ++j) {
      chunk_row[c0 + j] = r; chunk_start[c0 + j] = s + j * chunk; chunk_slot[c0 + j] = slot0 + j;
    }
    const int m = multi_off[r];
    multi_row[m] = r; multi_first[m] = slot0; multi_n[m] = nc;
  }
}

// ------------------------------------------------------------------------------------------------------------
// (src, dst) -> position hash (replaces pos_df) and the per-batch target-edge mask
// ------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned long long mix64(unsigned long long x) {
  x ^= x >> 33; x *= 0xff51afd7ed558ccdULL; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53ULL; x ^= x >> 33;
  return x;
}
constexpr unsigned long long HASH_EMPTY = ~0ULL;

__global__ void pairhash_insert_kernel(const int64_t* __restrict__ edge_index, long long n, unsigned long long* __restrict__ keys,
                                       int* __restrict__ vals, unsigned long long cap_mask) {
  const long long p = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (p >= n) return;
  const unsigned long long key = ((unsigned long long)edge_index[p] << 32) | (unsigned long long)(edge_index[n + p] & 0xffffffffLL);
  unsigned long long h = mix64(key) & cap_mask;
  while (true) {
    const unsigned long long prev = atomicCAS(keys + h, HASH_EMPTY, key);
    if (prev == HASH_EMPTY || prev == key) { atomicMin(vals + h, (int)p); return; }   // duplicates keep the first position
    h = (h + 1) & cap_mask;
  }
}

__global__ void pairhash_lookup_kernel(const int64_t* __restrict__ src, const int64_t* __restrict__ dst, long long n,
                                       const unsigned long long* __restrict__ keys, const int* __restrict__ vals,
                                       unsigned long long cap_mask, int64_t* __restrict__ out, int* __restrict__ n_missing) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const unsigned long long key = ((unsigned long long)src[i] << 32) | (unsigned long long)(dst[i] & 0xffffffffLL);
  unsigned long long h = mix64(key) & cap_mask;
  while (true) {
    const unsigned long long k = keys[h];
    if (k == key) { out[i] = vals[h]; return; }
    if (k == HASH_EMPTY) { out[i] = -1; atomicAdd(n_missing, 1); return; }
    h = (h + 1) & cap_mask;
  }
}

// positions -> skip bitmap + degree adjustment (both endpoints lose one in-edge; duplicates count once)
__global__ void mask_targets_kernel(const int64_t* __restrict__ positions, long long n, long long n_edges,
                                    const int64_t* __restrict__ u2i, const int64_t* __restrict__ i2u,
                                    unsigned* __restrict__ skip_bits, int* __restrict__ deg) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t p = positions[i];
  if (p < 0 || p >= n_edges) return;
  const unsigned bit = 1u << (p & 31);
  const unsigned old = atomicOr(skip_bits + (p >> 5), bit);
  if (!(old & bit)) {
    atomicSub(deg + u2i[n_edges + p], 1);      // the item loses the user->item edge
    atomicSub(deg + i2u[n_edges + p], 1);      // the user loses the item->user edge
  }
}

// partitioned training (peer.py): the batch targets on one rank.  Entry i counts when first[i] == i (the first entry of its pair in the
// batch; GraphIndex.masked takes each position once).  Every rank takes one off the degree of item iid[i]; the rank that owns user uid[i]
// (node0 <= uid < node0 + rows) finds the pair in its local hash (vals = CSR entry, local_pos = the entry's interaction position), sets
// that position's skip bit and takes one off the user's degree.  Ids outside the graph and pairs the owner does not find are counted in
// *n_missing.
__global__ void peer_mask_targets_kernel(const int64_t* __restrict__ uid, const int64_t* __restrict__ iid, long long n, const int64_t* __restrict__ first,
                                         long long n_items, long long n_nodes, long long node0, long long rows,
                                         const unsigned long long* __restrict__ keys, const int* __restrict__ vals, unsigned long long cap_mask,
                                         const int* __restrict__ local_pos, unsigned* __restrict__ skip_bits, int* __restrict__ deg_users,
                                         int* __restrict__ deg_items, int* __restrict__ n_missing) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const int64_t u = uid[i], it = iid[i];
  if (u < n_items || u >= n_nodes || it < 0 || it >= n_items) { atomicAdd(n_missing, 1); return; }
  if (first[i] != i) return;
  atomicSub(deg_items + it, 1);
  const long long lu = u - node0;
  if (lu < 0 || lu >= rows) return;
  const unsigned long long key = ((unsigned long long)u << 32) | (unsigned long long)(it & 0xffffffffLL);
  unsigned long long h = mix64(key) & cap_mask;
  while (true) {
    const unsigned long long k = keys[h];
    if (k == key) break;
    if (k == HASH_EMPTY) { atomicAdd(n_missing, 1); return; }
    h = (h + 1) & cap_mask;
  }
  const int p = local_pos[vals[h]];
  atomicOr(skip_bits + (p >> 5), 1u << (p & 31));
  atomicSub(deg_users + lu, 1);
}

}  // namespace b200rec

using namespace b200rec;

static inline unsigned grid1d(long long n, int threads = 256) { return (unsigned)((n + threads - 1) / threads); }

// ---- scan / sort (exported for tests and for host-side composition) ------------------------------------------
extern "C" size_t b200rec_scan_workspace(int64_t n) { return scan_ws_bytes(n); }

extern "C" int b200rec_exclusive_scan_i32(const int* in, int64_t n, int* out, void* ws, size_t ws_bytes, b200rec_stream_t stream) {
  if (n < 0 || !out || (n > 0 && !in)) return b200rec_fail(B200REC_ERR_BAD_ARG, "scan: bad argument");
  if (ws_bytes < scan_ws_bytes(n) || (!ws && scan_ws_bytes(n) > 64)) return b200rec_fail(B200REC_ERR_WORKSPACE, "scan: workspace too small");
  return exclusive_scan(in, n, out, (int*)ws, (cudaStream_t)stream);
}

extern "C" size_t b200rec_sort_pairs_workspace(int64_t n) { return radix_ws_bytes(n); }

extern "C" int b200rec_sort_pairs_i32(int* keys, int* vals, int64_t n, int key_bits, void* ws, size_t ws_bytes,
                                      b200rec_stream_t stream) {
  if (n < 0 || (n > 0 && (!keys || !vals))) return b200rec_fail(B200REC_ERR_BAD_ARG, "sort: bad argument");
  if (n > 0x7fffffffLL) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "sort: n > int32");
  if (ws_bytes < radix_ws_bytes(n) || !ws) return b200rec_fail(B200REC_ERR_WORKSPACE, "sort: workspace too small");
  return radix_sort_pairs(keys, vals, n, key_bits, ws, (cudaStream_t)stream);
}

// ---- node ids --------------------------------------------------------------------------------------------------
extern "C" int b200rec_id_rank_table(const int64_t* ids, int64_t n, int64_t id_bound, int* flags, int* rank, int64_t* sorted_ids,
                                     int* err_flag, void* ws, size_t ws_bytes, b200rec_stream_t stream) {
  if (n < 0 || id_bound <= 0 || !flags || !rank || !err_flag) return b200rec_fail(B200REC_ERR_BAD_ARG, "id_rank_table: bad argument");
  if (ws_bytes < scan_ws_bytes(id_bound)) return b200rec_fail(B200REC_ERR_WORKSPACE, "id_rank_table: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  B200REC_CUDA(cudaMemsetAsync(flags, 0, id_bound * sizeof(int), st));
  if (n > 0) { mark_ids_kernel<<<grid1d(n), 256, 0, st>>>(ids, n, id_bound, flags, err_flag); B200REC_CHECK_LAUNCH(); }
  int rc = exclusive_scan(flags, id_bound, rank, (int*)ws, st);
  if (rc) return rc;
  if (sorted_ids) { unique_ids_kernel<<<grid1d(id_bound), 256, 0, st>>>(flags, rank, id_bound, sorted_ids); B200REC_CHECK_LAUNCH(); }
  return B200REC_OK;
}

extern "C" int b200rec_id_lookup(const int64_t* ids, int64_t n, int64_t id_bound, const int* flags, const int* rank, int64_t offset,
                                 int64_t* out, int* err_flag, b200rec_stream_t stream) {
  if (n < 0 || !flags || !rank || !out || !err_flag) return b200rec_fail(B200REC_ERR_BAD_ARG, "id_lookup: bad argument");
  if (n == 0) return B200REC_OK;
  lookup_ids_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(ids, n, id_bound, flags, rank, offset, out, err_flag);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

// ---- means + edges ---------------------------------------------------------------------------------------------
extern "C" int b200rec_group_stats(const int64_t* idx, const double* rating, int64_t n, int64_t idx_offset, int* count, double* sum,
                                   b200rec_stream_t stream) {
  if (n < 0 || !count || !sum) return b200rec_fail(B200REC_ERR_BAD_ARG, "group_stats: bad argument");
  if (n == 0) return B200REC_OK;
  group_stats_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(idx, rating, n, idx_offset, count, sum);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_edge_attrs(const int64_t* u_node, const int64_t* i_node, const double* rating, int64_t n, int64_t n_items,
                                  const int* cnt_u, const double* sum_u, const int* cnt_i, const double* sum_i, float* attr_u2i,
                                  float* attr_i2u, int* keep_u, int* keep_i, b200rec_stream_t stream) {
  if (n < 0 || !cnt_u || !sum_u || !cnt_i || !sum_i) return b200rec_fail(B200REC_ERR_BAD_ARG, "edge_attrs: bad argument");
  if (n == 0) return B200REC_OK;
  edge_attr_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(u_node, i_node, rating, n, n_items, cnt_u, sum_u, cnt_i, sum_i,
                                                               attr_u2i, attr_i2u, keep_u, keep_i);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_edge_scatter(const int64_t* src, const int64_t* dst, int64_t n, const int* keep, const int* pos, int64_t n_out,
                                    int64_t* edge_index, b200rec_stream_t stream) {
  if (n < 0 || n_out < 0 || (n_out > 0 && !edge_index)) return b200rec_fail(B200REC_ERR_BAD_ARG, "edge_scatter: bad argument");
  if (n == 0) return B200REC_OK;
  edge_scatter_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(src, dst, n, keep, pos, n_out, edge_index);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

// compaction of a float attribute array with the same keep/pos (binary graphs carry no attrs, used by tests only)
// ---- CSR -------------------------------------------------------------------------------------------------------
extern "C" size_t b200rec_csr_workspace(int64_t n_edges_total, int64_t num_nodes) {
  size_t sort_part = radix_ws_bytes(n_edges_total);
  size_t scan_part = scan_ws_bytes(num_nodes);
  return (sort_part > scan_part ? sort_part : scan_part) + (size_t)(2 * n_edges_total + 8) * sizeof(int);
}

extern "C" int b200rec_csr_build(const int64_t* u2i, int64_t e1, const int64_t* i2u, int64_t e2, const float* attr_u2i,
                                 const float* attr_i2u, int64_t num_nodes, int* row_ptr, int* col, float* w, int* pos, int* deg,
                                 float* dinv, void* ws, size_t ws_bytes, b200rec_stream_t stream) {
  const long long n = e1 + e2;
  if (e1 < 0 || e2 < 0 || num_nodes <= 0 || !row_ptr || !deg) return b200rec_fail(B200REC_ERR_BAD_ARG, "csr_build: bad argument");
  if (n > 0x7fffffffLL || num_nodes > 0x7fffffffLL) return b200rec_fail(B200REC_ERR_UNSUPPORTED, "csr_build: > int32 edges/nodes");
  if (!ws || ws_bytes < b200rec_csr_workspace(n, num_nodes)) return b200rec_fail(B200REC_ERR_WORKSPACE, "csr_build: workspace too small");
  if (n > 0 && (!col || !pos)) return b200rec_fail(B200REC_ERR_BAD_ARG, "csr_build: null output");
  if (w && (!attr_u2i || !attr_i2u) && n > 0) return b200rec_fail(B200REC_ERR_BAD_ARG, "csr_build: weights requested without attrs");
  cudaStream_t st = (cudaStream_t)stream;
  B200REC_CUDA(cudaMemsetAsync(deg, 0, num_nodes * sizeof(int), st));
  int* keys = (int*)ws;
  int* perm = keys + n;
  void* sort_ws = perm + n + 8;
  if (n > 0) {
    csr_keys_kernel<<<grid1d(n), 256, 0, st>>>(u2i, e1, i2u, e2, keys, deg);
    B200REC_CHECK_LAUNCH();
    iota_kernel<<<grid1d(n), 256, 0, st>>>(perm, n);
    B200REC_CHECK_LAUNCH();
    int bits = 1;
    while (bits < 31 && (1LL << bits) < num_nodes) ++bits;
    int rc = radix_sort_pairs(keys, perm, n, bits, sort_ws, st);
    if (rc) return rc;
    csr_gather_kernel<<<grid1d(n), 256, 0, st>>>(perm, n, u2i, e1, i2u, e2, attr_u2i, attr_i2u, col, w, pos);
    B200REC_CHECK_LAUNCH();
  }
  // row_ptr = exclusive scan of the in-degrees.  The scan scratch reuses the (now free) sort workspace.
  int rc = exclusive_scan(deg, num_nodes, row_ptr, (int*)sort_ws, st);
  if (rc) return rc;
  if (dinv) { dinv_kernel<<<grid1d(num_nodes), 256, 0, st>>>(deg, num_nodes, dinv); B200REC_CHECK_LAUNCH(); }
  return B200REC_OK;
}

extern "C" int b200rec_dinv(const int* deg, int64_t n, float* dinv, b200rec_stream_t stream) {
  if (n < 0 || !deg || !dinv) return b200rec_fail(B200REC_ERR_BAD_ARG, "dinv: bad argument");
  if (n == 0) return B200REC_OK;
  dinv_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(deg, n, dinv);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

// ---- SpMM plan ---------------------------------------------------------------------------------------------------
extern "C" size_t b200rec_spmm_plan_workspace(int64_t n_rows) { return (size_t)(3 * (n_rows + 1)) * sizeof(int) + scan_ws_bytes(n_rows); }

// phase 1: scratch = [n_chunks_row | is_multi | n_slots_row] each n_rows+1 ints; offsets are written to
// chunk_off/multi_off/slot_off (n_rows+1 each); the totals sit in their last entries (read by the host).
extern "C" int b200rec_spmm_plan_count(const int* row_ptr, int64_t n_rows, int chunk, int* chunk_off, int* multi_off, int* slot_off,
                                       void* ws, size_t ws_bytes, b200rec_stream_t stream) {
  if (n_rows <= 0 || chunk <= 0 || !row_ptr || !chunk_off || !multi_off || !slot_off)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm_plan_count: bad argument");
  if (!ws || ws_bytes < b200rec_spmm_plan_workspace(n_rows)) return b200rec_fail(B200REC_ERR_WORKSPACE, "spmm_plan_count: workspace too small");
  cudaStream_t st = (cudaStream_t)stream;
  int* a = (int*)ws;
  int* b = a + n_rows + 1;
  int* c = b + n_rows + 1;
  int* sws = c + n_rows + 1;
  plan_count_kernel<<<grid1d(n_rows), 256, 0, st>>>(row_ptr, (int)n_rows, chunk, a, b, c);
  B200REC_CHECK_LAUNCH();
  int rc;
  if ((rc = exclusive_scan(a, n_rows, chunk_off, sws, st))) return rc;
  if ((rc = exclusive_scan(b, n_rows, multi_off, sws, st))) return rc;
  if ((rc = exclusive_scan(c, n_rows, slot_off, sws, st))) return rc;
  return B200REC_OK;
}

extern "C" int b200rec_spmm_plan_fill(const int* row_ptr, int64_t n_rows, int chunk, const int* chunk_off, const int* multi_off,
                                      const int* slot_off, int* chunk_row, int* chunk_start, int* chunk_slot, int* multi_row,
                                      int* multi_first_slot, int* multi_n_slots, b200rec_stream_t stream) {
  if (n_rows <= 0 || !row_ptr || !chunk_off || !chunk_row || !chunk_start || !chunk_slot)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "spmm_plan_fill: bad argument");
  plan_fill_kernel<<<grid1d(n_rows), 256, 0, (cudaStream_t)stream>>>(row_ptr, (int)n_rows, chunk, chunk_off, multi_off, slot_off,
                                                                    chunk_row, chunk_start, chunk_slot, multi_row,
                                                                    multi_first_slot, multi_n_slots);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

// ---- pair hash + target mask ---------------------------------------------------------------------------------------
extern "C" int b200rec_pairhash_build(const int64_t* edge_index, int64_t n, uint64_t* keys, int* vals, int64_t capacity,
                                      b200rec_stream_t stream) {
  if (n < 0 || capacity <= 0 || (capacity & (capacity - 1)) || capacity < 2 * n || !keys || !vals)
    return b200rec_fail(B200REC_ERR_BAD_ARG, "pairhash_build: capacity must be a power of two >= 2n");
  cudaStream_t st = (cudaStream_t)stream;
  B200REC_CUDA(cudaMemsetAsync(keys, 0xff, capacity * sizeof(uint64_t), st));
  B200REC_CUDA(cudaMemsetAsync(vals, 0x7f, capacity * sizeof(int), st));
  if (n > 0) {
    pairhash_insert_kernel<<<grid1d(n), 256, 0, st>>>(edge_index, n, (unsigned long long*)keys, vals, (unsigned long long)capacity - 1);
    B200REC_CHECK_LAUNCH();
  }
  return B200REC_OK;
}

extern "C" int b200rec_pairhash_lookup(const int64_t* src, const int64_t* dst, int64_t n, const uint64_t* keys, const int* vals,
                                       int64_t capacity, int64_t* out, int* n_missing, b200rec_stream_t stream) {
  if (n < 0 || capacity <= 0 || !keys || !vals || !out || !n_missing) return b200rec_fail(B200REC_ERR_BAD_ARG, "pairhash_lookup: bad argument");
  if (n == 0) return B200REC_OK;
  pairhash_lookup_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(src, dst, n, (const unsigned long long*)keys, vals,
                                                                     (unsigned long long)capacity - 1, out, n_missing);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_mask_targets(const int64_t* positions, int64_t n, int64_t n_edges, const int64_t* u2i, const int64_t* i2u,
                                    uint32_t* skip_bits, int* deg, b200rec_stream_t stream) {
  if (n < 0 || n_edges < 0 || !skip_bits || !deg || !u2i || !i2u) return b200rec_fail(B200REC_ERR_BAD_ARG, "mask_targets: bad argument");
  if (n == 0) return B200REC_OK;
  mask_targets_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(positions, n, n_edges, u2i, i2u, skip_bits, deg);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}

extern "C" int b200rec_peer_mask_targets(const int64_t* uid, const int64_t* iid, int64_t n, const int64_t* first, int64_t n_items, int64_t n_nodes,
                                         int64_t node0, int64_t rows, const uint64_t* keys, const int* vals, int64_t capacity, const int* local_pos,
                                         uint32_t* skip_bits, int* deg_users, int* deg_items, int* n_missing, b200rec_stream_t stream) {
  if (n < 0 || !skip_bits || !deg_items || !n_missing || (n > 0 && (!uid || !iid || !first)) ||
      (rows > 0 && (!keys || !vals || !local_pos || !deg_users || capacity <= 0 || (capacity & (capacity - 1)))))
    return b200rec_fail(B200REC_ERR_BAD_ARG, "peer_mask_targets: bad argument");
  if (n == 0) return B200REC_OK;
  peer_mask_targets_kernel<<<grid1d(n), 256, 0, (cudaStream_t)stream>>>(uid, iid, n, first, n_items, n_nodes, node0, rows, (const unsigned long long*)keys,
                                                                       vals, (unsigned long long)capacity - 1, local_pos, skip_bits, deg_users, deg_items,
                                                                       n_missing);
  B200REC_CHECK_LAUNCH();
  return B200REC_OK;
}
