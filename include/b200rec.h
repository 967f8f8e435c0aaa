/* libb200rec — C ABI of the B200-native scoring hot path of DeepRecommendation (BasicNCF / AttentionNCF / GraphNCF).
 *
 * The reference (michaelbzms/DeepRecommendation) is 100 % Python: it has no FFI, operator or plugin layer, so the
 * drop-in seam is its Python class API (SURVEY.md §8b).  This header is the boundary BELOW that seam: the entry
 * points a maintainer binds (ctypes stub in INTEGRATION.md; `deeprecommendation_b200/_lib.py` is that binding) to
 * replace the device work of the reference functions cited on each declaration.  Paths are relative to
 * /root/reference/src/neural_collaborative_filtering/ unless they start with src/.
 *
 * Conventions
 *  - plain pointers and sizes only; every pointer is a DEVICE pointer unless it says "host";
 *  - the caller owns every buffer; entry points never allocate, never synchronise and launch on `stream`
 *    (a cudaStream_t passed as void*); workspaces are sized by the matching *_workspace() query;
 *  - matrices are row-major with an explicit leading dimension in ELEMENTS; weights keep nn.Linear's (out, in) layout;
 *  - return value: B200REC_OK or an error code; b200rec_last_error() gives the message (thread-local);
 *  - there is no CPU path: without a CUDA device every compute call returns B200REC_ERR_CUDA.
 */
#ifndef B200REC_H
#define B200REC_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200REC_VERSION 205

typedef void* b200rec_stream_t; /* cudaStream_t */

enum { B200REC_OK = 0, B200REC_ERR_CUDA = 1, B200REC_ERR_BAD_ARG = 2, B200REC_ERR_UNSUPPORTED = 3, B200REC_ERR_WORKSPACE = 4 };
enum { B200REC_F32 = 0, B200REC_BF16 = 1 };
enum { B200REC_ATT_NET = 0, B200REC_ATT_DOT = 1 };
enum { B200REC_TC_TF32X3 = 0, B200REC_TC_BF16 = 1, B200REC_TC_BF16X3 = 2 /* wide form only */ };
#define B200REC_PEER_MAX 16          /* GPUs of one NVSwitch box that one exchange can address */
#define B200REC_PEER_CHANNELS 16     /* independent flag channels per arena */
#define B200REC_PEER_HANDLE_BYTES 64 /* sizeof(cudaIpcMemHandle_t) */

const char* b200rec_last_error(void);
int b200rec_version(void);
int b200rec_sm_count(void);
int64_t b200rec_launch_count(void); /* kernels launched by this library in this process so far */

/* ---- K1a  linear layer:  Y = act((X · Wᵀ + bias) ∘ row_scale) ---------------------------------------------------
 * Replaces nn.Linear at models/basic_ncf.py:38-39, models/attention_ncf.py:150-151,216, models/gnn_ncf.py:300-301 and
 * (transform-before-gather) the per-edge Linear of models/gnn_ncf.py:91-93.  fp32 FFMA, fp32 accumulate.
 * X (M,K) ld=ldx; W (N,K) ld=ldw; bias (N) or NULL; row_scale (M) or NULL; Y (M,N) ld=ldy of y_dtype. */
size_t b200rec_linear_workspace(int64_t M, int64_t N, int64_t K);
int b200rec_linear(const float* X, int64_t M, int64_t K, int64_t ldx, const float* W, int64_t N, int64_t ldw, const float* bias,
                   const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, void* workspace, size_t workspace_bytes,
                   b200rec_stream_t stream);

/* Same contract on the tensor cores (tcgen05.mma, TMEM accumulators; csrc/gemm_tc.cu).  mode B200REC_TC_TF32X3: fp32-parity
 * 3xTF32 split (rel <= 1e-5); B200REC_TC_BF16: bf16 operands (rel <= 1e-2).  Meant for M >= ~1024.  The weights come from `packed_w`
 * (b200rec_pack_weights_tc of W, same mode), which is required: NULL returns B200REC_ERR_BAD_ARG.  W and ldw are not read.
 * `row_index` (M int64, or NULL): GEMM row m reads row row_index[m] of an X table of `x_rows` rows — the gather of
 * `item_profiles[rated_items_ids]` (src/content_providers/dynamic_profiles_provider.py:70) fused into the projection. */
int b200rec_linear_tc(const float* X, int64_t M, int64_t K, int64_t ldx, const float* W, int64_t N, int64_t ldw, const float* bias,
                      const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, int mode, const void* packed_w,
                      const int64_t* row_index, int64_t x_rows, b200rec_stream_t stream);
/* Split-K form for SHORT-M, long-K GEMMs (a 512-pair batch against the F = 2094 profiles: 4 x 2 output tiles would occupy 8 of 148
 * SMs): the k-blocks are dealt out over ~SMs / tiles CTAs per output tile, every CTA leaves a raw fp32 tile in `workspace`
 * (b200rec_linear_tc_splitk_workspace bytes; 0 = the shape is not split and none is needed) and a second kernel adds the slabs in
 * split order (deterministic) and applies bias / row_scale / ReLU. */
size_t b200rec_linear_tc_splitk_workspace(int64_t M, int64_t N, int64_t K, int mode);
int b200rec_linear_tc_splitk(const float* X, int64_t M, int64_t K, int64_t ldx, const float* W, int64_t N, int64_t ldw, const float* bias,
                             const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, int mode, const void* packed_w,
                             void* workspace, size_t workspace_bytes, b200rec_stream_t stream);
/* Wide form for 128 < N (an even number of 128-column tiles, e.g. the 256 outputs of AttentionNCF's composite projections,
 * attention_ncf.py:150-151,176,216): a CTA owns 128 rows x 256 columns, so each X block is read, split and staged once for both
 * halves of W; the k range is always split (workspace = b200rec_linear_tc_wide_workspace bytes, slabs added in split order by the
 * same reduction kernel as b200rec_linear_tc_splitk).  `packed_w` (same mode) is required.  mode B200REC_TC_TF32X3: fp32 parity by the
 * 3xTF32 split (~6e-7 at K = 2094); B200REC_TC_BF16X3: the same three products on a bf16 hi/lo split of both operands — twice the MMA rate, 16
 * mantissa bits per operand: ~4e-6 of the largest output at K = 2094, inside the 1e-5 budget with less margin (opt-in). */
size_t b200rec_linear_tc_wide_workspace(int64_t M, int64_t N, int64_t K, int mode);
int b200rec_linear_tc_wide(const float* X, int64_t M, int64_t K, int64_t ldx, int64_t N, const float* bias, const float* row_scale, int relu,
                           void* Y, int64_t ldy, int y_dtype, int mode, const void* packed_w, const int64_t* row_index, int64_t x_rows,
                           void* workspace, size_t workspace_bytes, b200rec_stream_t stream);
/* Persistent short-K variant for the per-node transforms of GraphNCF (K in {32,64,96,128}, N <= 128; csrc/node_gemm.cu):
 * W stays in shared memory (`packed_w` = b200rec_pack_weights_tc(..., B200REC_TC_TF32X3)), row tiles are streamed, fp32 parity
 * by the 3xTF32 split.  X rows 16-byte aligned (ldx % 4 == 0); Y fp32 or bf16 (`y_dtype`; bf16 = the message table of GraphNCF's
 * bf16 mode, rounded once from the fp32 accumulator). */
int b200rec_linear_shortk(const float* X, int64_t M, int64_t K, int64_t ldx, const void* packed_w, int64_t N, const float* bias,
                          const float* row_scale, int relu, void* Y, int64_t ldy, int y_dtype, b200rec_stream_t stream);
/* The same GEMM with the all-gather of the partitioned GraphNCF propagation fused into its epilogue: every output tile is stored
 * into the SAME place (element offset `y_offset`, leading dimension ldy) of `n_dst` buffers — `dst` is a HOST array of device
 * pointers, one per rank of the box (peer-mapped arenas, b200rec_peer_open; the local buffer is one of them) — so the transformed
 * rows travel over NVLink tile by tile while the next tile is computed.  Replaces the per-layer feature exchange that a
 * multi-GPU form of models/gnn_ncf.py:336-345 needs. */
int b200rec_linear_shortk_push(const float* X, int64_t M, int64_t K, int64_t ldx, const void* packed_w, int64_t N, const float* bias,
                               const float* row_scale, int relu, void* const* dst, int n_dst, int64_t y_offset, int64_t ldy, int y_dtype,
                               b200rec_stream_t stream);
/* ---- K1s  projection of SPARSE profile rows (csrc/gather_sum.cu) -----------------------------------------------------------
 * One-hot rows (src/content_providers/one_hot_provider.py:17-21, fixed_profiles_provider.py:49-50) and the ~1 %-dense multi-hot
 * columns of the item profiles go through the same nn.Linear as dense columns in the reference (models/basic_ncf.py:38-39,
 * attention_ncf.py:150-151, gnn_ncf.py:300-301).  Here:  Y[m] (+)= bias + sum_{k in row m} val[k] * Wt[col[k]]  with Wt = W^T,
 * (K, N) row-major fp32 / bf16 — a warp-vectorised gather-sum, 128-bit loads, list order (deterministic).
 * Rows are given as CSR (row_ptr int32 (M+1), col int32, val fp32 or NULL = 1) or, for one-hot rows, as `ids` (M int64, one
 * column per row, negative = empty row); exactly one of the two.  accumulate != 0 adds onto the Y a dense-column GEMM has
 * written (mixed profiles: K1a over the dense slice, then this over the non-zeros); bias is ignored then.  N % 4 == 0. */
int b200rec_linear_sparse(const int* row_ptr, const int* col, const float* val, const int64_t* ids, int64_t M, const void* Wt, int64_t K,
                          int64_t N, int64_t ldwt, int wt_dtype, const float* bias, float* Y, int64_t ldy, int accumulate,
                          b200rec_stream_t stream);
/* CSR of the non-zero entries of columns [c0, c1) of a dense (M, ldx) matrix, for callers that hold only the dense profile rows:
 * count -> b200rec_exclusive_scan_i32 -> fill (col relative to c0, column order). */
int b200rec_dense_nnz_count(const float* X, int64_t M, int64_t ldx, int64_t c0, int64_t c1, int* counts, b200rec_stream_t stream);
int b200rec_dense_nnz_fill(const float* X, int64_t M, int64_t ldx, int64_t c0, int64_t c1, const int* row_ptr, int* col, float* val,
                           b200rec_stream_t stream);
/* Up to four such GEMMs sharing K and mode in ONE launch (candidate + rated-item projections, the two halves of
 * AttentionNet.0 — attention_ncf.py:150-151,176): problem q covers its own rows; fields as in b200rec_linear_tc (`packed_w` required). */
typedef struct {
  const float* X; int64_t M; int64_t ldx;
  const float* W; int64_t N; int64_t ldw; const void* packed_w;
  const float* bias; const float* row_scale; int relu;
  void* Y; int64_t ldy; int y_dtype;
} b200rec_linear_problem_t;
int b200rec_linear_tc_batch(const b200rec_linear_problem_t* problems, int n_problems, int64_t K, int mode, b200rec_stream_t stream);
/* The same batch as split-K (short M, long K — BasicNCF's user and item projections, basic_ncf.py:38-39, in one wave): workspace from
 * b200rec_linear_tc_splitk_batch_workspace (0 = no split pays: the call then behaves like b200rec_linear_tc_batch). */
size_t b200rec_linear_tc_splitk_batch_workspace(const b200rec_linear_problem_t* problems, int n_problems, int64_t K, int mode);
int b200rec_linear_tc_splitk_batch(const b200rec_linear_problem_t* problems, int n_problems, int64_t K, int mode, void* workspace,
                                   size_t workspace_bytes, b200rec_stream_t stream);
/* W converted once into MMA-ready swizzled tiles (bf16, TF32 hi/lo or bf16 hi/lo, zero-padded): the `packed_w` of the tensor-core GEMMs,
 * which move it by TMA bulk copies (cp.async.bulk) while the producer warps convert X.  128-byte aligned buffer. */
size_t b200rec_packed_weight_bytes(int64_t N, int64_t K, int mode);
int b200rec_pack_weights_tc(const float* W, int64_t N, int64_t K, int64_t ldw, int mode, void* packed, size_t packed_bytes,
                            b200rec_stream_t stream);

/* ---- K1b  fused MLP tower ------------------------------------------------------------------------------------
 * Replaces torch.cat + build_MLP_layers (util.py:5-18; basic_ncf.py:40-41, attention_ncf.py:219-222, gnn_ncf.py:354-362):
 * out = MLP([in0[idx0], in1[idx1]]).  idx0/idx1 (int64, B) are optional row gathers (GraphNCF's combined[itemIds] /
 * combined[userIds]); NULL = identity.  Layer l: W[l] (out_dim[l], in) row-major, b[l] (out_dim[l]) or NULL; ReLU between
 * layers, none after the last.  Activations never leave shared memory. */
#define B200REC_MLP_MAX_LAYERS 8
typedef struct {
  const float* W[B200REC_MLP_MAX_LAYERS];
  const float* b[B200REC_MLP_MAX_LAYERS];
  int out_dim[B200REC_MLP_MAX_LAYERS];
  int n_layers;
} b200rec_mlp_t;
int b200rec_mlp_tower(const float* in0, int64_t ld0, const int64_t* idx0, int E0, const float* in1, int64_t ld1, const int64_t* idx1,
                      int E1, int64_t B, const b200rec_mlp_t* mlp, float* out, int64_t ldo, b200rec_stream_t stream);
/* GraphNCF(use_dot_product=True), gnn_ncf.py:365: out[b] = <in0[idx0[b]], in1[idx1[b]]> */
int b200rec_rowdot(const float* in0, int64_t ld0, const int64_t* idx0, const float* in1, int64_t ld1, const int64_t* idx1, int E,
                   int64_t B, float* out, b200rec_stream_t stream);

/* ---- row-wise top-k (k <= 64), descending, ties towards the lower column, NaN never selected; rows with fewer than k valid
 * scores are padded with (-inf, -1).  Replaces `sort_values(by='score', ascending=False).iloc[:k]` of src/webapp/backend.py:113-121
 * and the per-user top-K of BASELINE config 4.  scores (rows, cols) ld; out_val (rows, k) fp32; out_idx (rows, k) int64. */
/* One-hidden-layer MLPs in all-pairs mode: score(u,i) = b2 + sum_h w2[h]·ReLU(A[u,h] + B[i,h]) — ~3·H1 FP32 operations per pair and no GEMM
 * (SURVEY.md §8d), evaluated exactly on the FP32 pipes with the same top-k / `seen` / split-list semantics as b200rec_allpairs_topk
 * (whose workspace query it shares).  A (nU, H1), B (nI, H1) contiguous fp32, H1 in {64,128,192,256} (zero-pad), w2 (H1) device. */
int b200rec_allpairs_relu_dot_splits(int64_t nU, int64_t nI);
int b200rec_allpairs_relu_dot_topk(const float* A, const float* B, int64_t nU, int64_t nI, int H1, const float* w2, float b2, int k, int n_splits,
                                   const int* seen_ptr, const int* seen_idx, float* scores, int64_t lds, float* top_val, int64_t* top_idx,
                                   void* workspace, size_t workspace_bytes, b200rec_stream_t stream);
int b200rec_topk_rows(const float* scores, int64_t rows, int64_t cols, int64_t ld, int k, float* out_val, int64_t* out_idx,
                      b200rec_stream_t stream);

/* ---- K5  all-pairs scoring + per-user top-k (tcgen05 tensor cores; csrc/allpairs.cu) --------------------------------
 * Replaces, for every (user, item) pair of a user set x item set, `MLP(cat(user_emb, item_emb))` of models/basic_ncf.py:40-41
 * (util.py:5-18; item-first for models/gnn_ncf.py:361) followed by the `sort_values(by='score', ascending=False).iloc[:k]` of
 * src/webapp/backend.py:113-121 — BASELINE configs[3].  The first Linear of the MLP is split by the caller:
 *   A = user_emb · W1[:, :Eu]^T + b1  (nU, H1),   B = item_emb · W1[:, Eu:]^T  (nI, H1)      (K1a; contiguous rows, H1 % 64 == 0,
 *   H1 <= 256 — zero-pad the columns);  score(u, i) = w3 · ReLU(W2 · ReLU(A[u] + B[i]) + b2) + b3,  W2 (H2 <= 128, H1).
 * b200rec_allpairs_pack converts W2 once into MMA-ready bf16 tiles; `epilogue_host` is a HOST array b2[H2] | w3[H2] | b3
 * (2*H2+1 floats) that travels in the kernel's parameter block (constant bank).  mode B200REC_AP_BF16: bf16 operands
 * (rel <= 1e-2); B200REC_AP_BF16X2: operands split into bf16 hi + lo, 3 MMAs per k-step (fp32 tolerance, rel <= 1e-5).
 * Outputs: top_val (nU, k) fp32 / top_idx (nU, k) int64 item positions, descending, ties towards the lower item, fewer than k
 * valid items padded with (-inf, -1), NaN never selected; optional `scores` (nU, nI) ld = lds (NULL = never materialised);
 * optional CSR `seen_ptr` (nU+1) / `seen_idx` (sorted item positions per user): those pairs are not recommended
 * (`ignore_seen`, backend.py:85).  n_splits <= 0 = automatic (b200rec_allpairs_splits). */
enum { B200REC_AP_BF16 = 0, B200REC_AP_BF16X2 = 1 };
size_t b200rec_allpairs_packed_bytes(int H1, int mode);
int b200rec_allpairs_pack(const float* W2, int64_t ldw2, int H2, int H1, int mode, void* packed, size_t packed_bytes,
                          b200rec_stream_t stream);
int b200rec_allpairs_splits(int64_t nU, int64_t nI, int mode);
size_t b200rec_allpairs_workspace(int64_t nU, int k, int n_splits);
int b200rec_allpairs_topk(const float* A, const float* B, int64_t nU, int64_t nI, int H1, const void* packed,
                          const float* epilogue_host, int H2, int mode, int k, int n_splits, const int32_t* seen_ptr, const int32_t* seen_idx, float* scores, int64_t lds, float* top_val,
                          int64_t* top_idx, void* workspace, size_t workspace_bytes, b200rec_stream_t stream);

/* ---- K2  AttentionNCF ragged attention pooling ------------------------------------------------------------------
 * Replaces attention_ncf.py:154-216.  With AttentionNet.0 = [A1c | A1r]:  Pc = Ec·A1cᵀ + a1 (B,H), Pr = Er·A1rᵀ (I,H),
 * Q = rated_items·W_Uᵀ (I,U);  s_bi = a2·ReLU(Pc[b] + Pr[i]) + a20 (mode NET)  or  <Pc[b], Pr[i]> (mode DOT: cosine / att_dense=None);
 * out[b] = Σ_i softmax_i(s_b·)·um_bi·Q[i] + bU   over the i with um_bi != 0 (exact 0.0 = "unrated", :158,192).
 * Give either the reference's dense user_matrix (B,I) or its CSR (row_ptr int32 B+1, col int32, val fp32).
 * att_weights (B,I), if non-NULL, must be zero-filled; it receives the softmax weights (:224).
 * Training extras: train_cand_emb/train_rated_emb (+E, atol, rtol) reproduce the isclose() target mask (:199);
 * drop_zero_scores reproduces `attOut[attOut == 0] = -inf` (:189).  H, U: multiples of 4, <= 512. */
typedef struct {
  const float* Pc;
  const void* Pr;
  const void* Q;
  int table_dtype; /* dtype of Pr and Q */
  int mode;
  const float* a2;  /* (H), mode NET */
  const float* a20; /* device scalar or NULL */
  const float* bU;  /* (U) or NULL */
  const float* user_matrix; /* (B,I) dense, or NULL when CSR is given */
  int64_t ld_user_matrix;   /* 0 = I */
  const int* row_ptr;
  const int* col;
  const float* val;
  int64_t B, I;
  int H, U;
  float* out; /* (B,U) */
  int64_t ldo;
  float* att_weights;
  const float* train_cand_emb;
  const float* train_rated_emb;
  int E;
  float atol, rtol;
  int drop_zero_scores;
  float score_scale; /* 0 = 1.0; message dropout keeps scores / (1-p) (F.dropout, :187) */
  int64_t ld_pr, ld_q; /* leading dimensions of Pr / Q in elements; 0 = H / U */
  void* workspace;     /* b200rec_attention_pool_workspace(B, I, U, dense) bytes enable the segment-parallel path (streaming compaction */
  size_t workspace_bytes; /* of a dense matrix, work list of <=64-non-zero segments, one warp each, merge kernel); NULL = one fused kernel */
  int64_t max_row_nnz;    /* CSR form, optional: upper bound of a row's length (0 = unknown, I is used) and the number of stored entries */
  int64_t nnz;            /* (0 = unknown).  They only size the work list / partial slots: b200rec_attention_pool_workspace_csr(). */
  int64_t ld_pc;          /* leading dimension of Pc in elements (a column slice of the [Ec | Pc] projection is used in place); 0 = H */
  float dropout_p;        /* training only, b200rec_attention_pool_dropout: p of the Dropout between AttentionNet's ReLU and its head Linear */
  uint64_t dropout_seed;  /* (attention_ncf.py:112-117); mask = Philox2x32-10 keyed by the seed, regenerated by the backward kernel */
  const uint64_t* dropout_seed_dev;   /* optional: read the seed from DEVICE memory instead (a captured CUDA graph draws a new seed per replay) */
} b200rec_attention_t;
size_t b200rec_attention_pool_workspace(int64_t B, int64_t I, int U, int dense);
size_t b200rec_attention_pool_workspace_csr(int64_t B, int64_t I, int U, int64_t max_row_nnz, int64_t nnz);
int b200rec_attention_pool(const b200rec_attention_t* a, b200rec_stream_t stream);
/* ---- K8  AttentionNCF whole-catalogue recommendation: attention pooling over one shared rated list per user ------------------
 * Replaces, for every catalogue item b as a candidate of user u, attention_ncf.py:136-224 up to the first hidden layer of the MLP — the
 * per-user scoring loop of src/webapp/backend.py:78-121 run for many users at once (csrc/attention_recommend.cu).  With the user-embedding
 * half of the first MLP Linear folded into the pooled table (W1 = [W1e | W1u], item first, :219):
 *   s_bi = a2·ReLU(Pc[b] + Pr[i]) + a20 (mode NET) or <Pc[b], Pr[i]> (mode DOT);  α = softmax_i over the list entries with val != 0
 *   (exact 0.0 = "unrated", :158,192; none -> α = 0, :208-209);  h1[u, b] = ReLU(Ai[b] + Σ_i α_bi·val_i·Qp[i])
 *   where Ai = Ec·W1eᵀ + b1 + W1u·b_U (nI, H1P) and Qp = Q·W1uᵀ (nI, H1P), columns past H1 zero.
 * Tables: Pc, Pr (n_items, H) fp32, H % 4 == 0, H <= 256; a2 (H) and a20 (device scalar or NULL) for mode NET.  H1P in {32, 64, 128, 256}.
 * Rating lists (the resident format of b200rec_collate_interacted): list_ptr int64 (rows+1), list_item int32 catalogue rows, list_val fp32
 * centred ratings.  users (n_users int64, list rows; duplicates allowed, n_users <= 65535 per call).  h1 (n_users·n_items, ld_h1 >= H1P) fp32:
 * row u·n_items + b; b200rec_attention_recommend_workspace gives its size in bytes for ld_h1 = H1P.  All leading dimensions % 4 == 0,
 * tables and h1 16-byte aligned.  No atomics: bit-identical results run to run. */
size_t b200rec_attention_recommend_workspace(int64_t n_users, int64_t n_items, int H1P);
int b200rec_attention_recommend(const float* Pc, int64_t ld_pc, const float* Pr, int64_t ld_pr, int H, int mode, const float* a2, const float* a20,
                                const float* Ai, int64_t ld_ai, const float* Qp, int64_t ld_q, int H1P, int64_t n_items, const int64_t* list_ptr,
                                const int32_t* list_item, const float* list_val, const int64_t* users, int64_t n_users, float* h1, int64_t ld_h1,
                                b200rec_stream_t stream);
/* ---- K9  AttentionNCF explanations of many users' recommendations (csrc/attention_explain.cu) -----------------------------------------
 * Replaces the explanation step of src/webapp/backend.py:102-110 for k recommended items of each of many users: the entries i of user u's list
 * with α_bi > explain_factor · (1 / max(R_u, 1)) + explain_constant (computed in double, compared in fp32), R_u = length of u's list, zero-centred
 * entries included.  α_bi is K8's attention weight (same tables, same mode, same score arithmetic); zero-centred entries have α = 0 and never
 * explain, an empty list explains nothing.
 * items (n_users, k) int64 catalogue rows, 1 <= k <= 64; a row outside [0, n_items) (e.g. -1, K8's top-k padding) is padding and explains nothing.
 * Row r = u·k + j of the output explains items[u, j]; its entries are in list order.  The other operands are those of b200rec_attention_recommend.
 * Two calls on one stream, with the same operands and workspace (b200rec_attention_explain_workspace bytes):
 *   _count  writes ptr (n_users·k + 1) int64: ptr[0] = 0, ptr[r+1] - ptr[r] = entries of row r;  the caller reads n = ptr[n_users·k]
 *   _fill   writes because (n) int64 list items (catalogue rows) and attention (n) fp32 α at [ptr[r], ptr[r+1]).
 * No atomics: bit-identical results run to run. */
size_t b200rec_attention_explain_workspace(int64_t n_users, int k);
int b200rec_attention_explain_count(const float* Pc, int64_t ld_pc, const float* Pr, int64_t ld_pr, int H, int mode, const float* a2, const float* a20,
                                    int64_t n_items, const int64_t* list_ptr, const int32_t* list_item, const float* list_val, const int64_t* users,
                                    int64_t n_users, const int64_t* items, int k, double explain_factor, double explain_constant, int64_t* ptr,
                                    void* workspace, size_t workspace_bytes, b200rec_stream_t stream);
int b200rec_attention_explain_fill(const float* Pc, int64_t ld_pc, const float* Pr, int64_t ld_pr, int H, int mode, const float* a2, const float* a20,
                                   int64_t n_items, const int64_t* list_ptr, const int32_t* list_item, const float* list_val, const int64_t* users,
                                   int64_t n_users, const int64_t* items, int k, const int64_t* ptr, const void* workspace, size_t workspace_bytes,
                                   int64_t* because, float* attention, b200rec_stream_t stream);
/* The same op with AttentionNet's inner Dropout applied in training mode: hidden = ReLU(Pc[b] + Pr[i]) ∘ m / keep, m ~ Bernoulli(keep), keep =
 * round((1 - dropout_p)·65536) / 65536, one Philox2x32-10 call (counter = (i, b·64 + hidden group), key = seed) per 4 hidden units
 * (csrc/common.cuh).  A separately compiled copy of the kernels (csrc/attention_pool_drop.cu): the scoring build above is untouched. */
int b200rec_attention_pool_dropout(const b200rec_attention_t* a, b200rec_stream_t stream);
/* How the segment-parallel path gathers table rows: 0 = auto (TMA bulk copies into shared memory when the tables exceed half of L2,
 * register-staged 128-bit loads otherwise), 1 = always registers, 2 = TMA whenever the layout allows (H, U <= 128, 16-byte rows). */
int b200rec_attention_pool_set_path(int path);

/* Gradient of b200rec_attention_pool for the training step (NCF/train.py:99-105 through attention_ncf.py:154-216), dense user_matrix form,
 * fp32 tables.  Inputs: the forward's operands, its `out`, its `att_weights` (the softmax weights: every pair the forward masked out —
 * unrated, isclose() target mask :199, zero score under message dropout :189 — has weight 0 and receives no gradient) and grad_out =
 * dL/dout (B,U).  Writes dPc (B,H); ADDS into dPr (I,H) and dQ (I,U) (contiguous, zero-filled by the caller: many rows share an item,
 * 128-bit vector reductions); mode NET also writes per-row parts da2_rows (B,H) and da20_rows (B) whose column sums are the gradients
 * of a2 / a20 (dbU is the column sum of grad_out).  H, U: multiples of 4, <= 512. */
typedef struct {
  const float* Pc;
  const float* Pr;
  const float* Q;
  int mode;          /* as b200rec_attention_t */
  const float* a2;   /* (H), mode NET */
  const float* bU;   /* (U) or NULL */
  const float* user_matrix; /* (B,I) */
  int64_t ld_user_matrix;   /* 0 = I */
  const float* att_weights; /* (B,I) contiguous, from the forward */
  const float* out;         /* (B,U) forward output */
  int64_t ldo;              /* 0 = U */
  const float* grad_out;    /* (B,U) */
  int64_t ld_grad_out;      /* 0 = U */
  int64_t B, I;
  int H, U;
  float score_scale;        /* 0 = 1.0 */
  int64_t ld_pc, ld_pr, ld_q; /* 0 = H / H / U */
  float* dPc;
  float* dPr;
  float* dQ;
  float* da2_rows;
  float* da20_rows;
  int n_slices;             /* 0 / 1 = one CTA per row; n > 1 = the columns are dealt out over n CTAs per row and dPc, da2_rows, da20_rows
                             * hold n parts of B rows each (part-major), which the caller adds */
  float dropout_p;          /* the forward's inner dropout (b200rec_attention_pool_dropout): same p and seed regenerate the same mask; 0 = none */
  uint64_t dropout_seed;
  const uint64_t* dropout_seed_dev;   /* as in b200rec_attention_t: the same device word the forward read */
} b200rec_attention_bwd_t;
int b200rec_attention_pool_backward(const b200rec_attention_bwd_t* a, b200rec_stream_t stream);

/* ---- K3  GraphNCF propagation: edge-balanced CSR SpMM + degree normalisation + fused combine -----------------------
 * Replaces LightGCNConv.forward/message + PyG propagate (gnn_ncf.py:39-94) and the stack+mean of gnn_ncf.py:351:
 *   x_next[r] = dinv[r] · Σ_{k in row r} w[k]·t[col[k]];   acc_out[r] = (acc_in[r] + x_next[r])·acc_scale
 * t (N,d) are the per-NODE transformed features dinv[s]·(W_type x[s] + b_type) produced by b200rec_linear.
 * chunk_* / multi_* come from b200rec_spmm_plan_*; skip_bits (+perm) is the training-time target-edge mask. */
typedef struct {
  const int* chunk_row;
  const int* chunk_start;
  const int* chunk_slot;
  int n_chunks;
  int chunk_size;
  const int* row_ptr;
  const int* col;
  const float* w; /* NULL = 1 (binary graph) */
  const int* perm;
  const uint32_t* skip_bits;
  const void* t;
  int t_dtype;
  int64_t ld_t;
  int d;
  const float* dinv;
  float* partials; /* (n_slots, d) */
  float* x_next;   /* may be NULL */
  int64_t ld_x;
  const float* acc_in; /* may be NULL */
  float* acc_out;      /* may be NULL */
  int64_t ld_acc;
  float acc_scale;
  const int* multi_row;
  const int* multi_first_slot;
  const int* multi_n_slots;
  int n_multi;
  const float* att_src; /* LightGAT (gnn_ncf.py:97-177): per-source score; edge weight = w * softmax_row(att_src[col]); NULL = LightGCN */
  float* partials_ml;   /* (n_slots, 2) scratch for the softmax state of multi-chunk rows */
  /* reduce-scatter fused into the epilogue (partitioned propagation): when push_parts > 0 a finished row r is not written to
   * x_next / acc_out but into the receive slot of its OWNER rank o = r / push_rows_per_part, i.e. to
   * (float*)push_dst[o] + push_offset + (r - o * push_rows_per_part) * push_ld — push_dst are the peer-mapped arenas */
  void* push_dst[B200REC_PEER_MAX];
  int push_parts;
  int push_rows_per_part;
  int64_t push_offset;
  int64_t push_ld;
} b200rec_spmm_t;
int b200rec_spmm(const b200rec_spmm_t* a, b200rec_stream_t stream);

/* Edge-balanced ("stream") form of the same propagation step for inference (csrc/spmm_stream.cu): a warp owns `seg` consecutive CSR
 * entries whatever rows they belong to, so short rows (a rank's slice of an item row on a partitioned graph) cost no per-row set-up.
 *   colf[k]  = source node | (k is the LAST entry of its row) << 31        wd[k] = deg[dst]^-1/2 * w[k]   (gnn_ncf.py:54,91)
 *   seg_first_j[s]   index into rows_ne of the row holding entry s*seg;   seg_head_slot[s] = partial slot of that row when it began in an
 *   earlier segment (else -1);   seg_tail_slot[s] = partial slot of the row still open after the segment's last entry (else -1)
 *   rows_ne / rows_empty = rows with / without entries (ascending);   multi_* = rows cut by a segment boundary and their slot runs,
 *   added in segment order by the fix-up pass (deterministic).   t (N, d <= 128) fp32 or bf16.   Outputs / push_* as in b200rec_spmm_t. */
typedef struct {
  const int* colf;
  const float* wd;
  int64_t nnz;
  int seg;
  int n_segs;
  const int* seg_first_j;
  const int* seg_head_slot;
  const int* seg_tail_slot;
  const int* rows_ne;
  int n_ne;
  const int* rows_empty;
  int n_empty;
  const void* t;
  int t_dtype;
  int64_t ld_t;
  int d;
  float* partials; /* (n_slots, d) */
  const int* multi_row;
  const int* multi_first_slot;
  const int* multi_n_slots;
  int n_multi;
  float* x_next;   /* may be NULL */
  int64_t ld_x;
  const float* acc_in; /* may be NULL */
  float* acc_out;      /* may be NULL */
  int64_t ld_acc;
  float acc_scale;
  void* push_dst[B200REC_PEER_MAX];
  int push_parts;
  int push_rows_per_part;
  int64_t push_offset;
  int64_t push_ld;
} b200rec_spmm_stream_t;
int b200rec_spmm_stream(const b200rec_spmm_stream_t* a, b200rec_stream_t stream);

/* ---- K4  neighbour-index build (bit-exact vs src/content_providers/graph_providers.py:10-66,76-80) ---------------- */
size_t b200rec_scan_workspace(int64_t n);
int b200rec_exclusive_scan_i32(const int* in, int64_t n, int* out /* n+1 */, void* ws, size_t ws_bytes, b200rec_stream_t stream);
size_t b200rec_sort_pairs_workspace(int64_t n);
int b200rec_sort_pairs_i32(int* keys, int* vals, int64_t n, int key_bits, void* ws, size_t ws_bytes, b200rec_stream_t stream);

/* sorted-unique raw id -> rank (graph_providers.py:76-80).  flags (id_bound), rank (id_bound+1; rank[id_bound] = #unique),
 * sorted_ids (#unique, may be NULL); *err_flag is set to 1 if an id is outside [0, id_bound). */
int b200rec_id_rank_table(const int64_t* ids, int64_t n, int64_t id_bound, int* flags, int* rank, int64_t* sorted_ids, int* err_flag,
                          void* ws, size_t ws_bytes, b200rec_stream_t stream);
int b200rec_id_lookup(const int64_t* ids, int64_t n, int64_t id_bound, const int* flags, const int* rank, int64_t offset, int64_t* out,
                      int* err_flag, b200rec_stream_t stream);
/* per-group rating count and fp64 sum (pandas groupby.mean, graph_providers.py:16-17); count/sum must be zeroed */
int b200rec_group_stats(const int64_t* idx, const double* rating, int64_t n, int64_t idx_offset, int* count, double* sum,
                        b200rec_stream_t stream);
/* centred edge attrs (fp64 -> fp32) and the `binary` keep flags per interaction, file order (graph_providers.py:32-46) */
int b200rec_edge_attrs(const int64_t* u_node, const int64_t* i_node, const double* rating, int64_t n, int64_t n_items, const int* cnt_u,
                       const double* sum_u, const int* cnt_i, const double* sum_i, float* attr_u2i, float* attr_i2u, int* keep_u,
                       int* keep_i, b200rec_stream_t stream);
/* edge_index (2, n_out) int64 from (src, dst) per interaction; keep/pos (exclusive scan of keep) compact when binary */
int b200rec_edge_scatter(const int64_t* src, const int64_t* dst, int64_t n, const int* keep, const int* pos, int64_t n_out,
                         int64_t* edge_index, b200rec_stream_t stream);
/* CSR by destination of cat(u2i, i2u): stable radix sort.  row_ptr (N+1), col/w/pos (e1+e2), deg (N), dinv (N, may be NULL);
 * pos[k] = position of CSR entry k inside its own edge list (the pos_df value). */
size_t b200rec_csr_workspace(int64_t n_edges_total, int64_t num_nodes);
int b200rec_csr_build(const int64_t* u2i, int64_t e1, const int64_t* i2u, int64_t e2, const float* attr_u2i, const float* attr_i2u,
                      int64_t num_nodes, int* row_ptr, int* col, float* w, int* pos, int* deg, float* dinv, void* ws, size_t ws_bytes,
                      b200rec_stream_t stream);
int b200rec_dinv(const int* deg, int64_t n, float* dinv, b200rec_stream_t stream);
/* chunk plan for b200rec_spmm: count (offset arrays of n_rows+1 ints; totals in their last entry), then fill */
size_t b200rec_spmm_plan_workspace(int64_t n_rows);
int b200rec_spmm_plan_count(const int* row_ptr, int64_t n_rows, int chunk, int* chunk_off, int* multi_off, int* slot_off, void* ws,
                            size_t ws_bytes, b200rec_stream_t stream);
int b200rec_spmm_plan_fill(const int* row_ptr, int64_t n_rows, int chunk, const int* chunk_off, const int* multi_off, const int* slot_off,
                           int* chunk_row, int* chunk_start, int* chunk_slot, int* multi_row, int* multi_first_slot, int* multi_n_slots,
                           b200rec_stream_t stream);
/* (src,dst) -> position hash = pos_df (graph_providers.py:54) and its lookup (gnn_ncf.py:370); missing pairs give -1 and bump
 * *n_missing (the reference raises KeyError).  capacity: power of two >= 2n. */
int b200rec_pairhash_build(const int64_t* edge_index, int64_t n, uint64_t* keys, int* vals, int64_t capacity, b200rec_stream_t stream);
int b200rec_pairhash_lookup(const int64_t* src, const int64_t* dst, int64_t n, const uint64_t* keys, const int* vals, int64_t capacity,
                            int64_t* out, int* n_missing, b200rec_stream_t stream);
/* training-time target-edge mask (gnn_ncf.py:314-320,369-378): sets skip bits and decrements both endpoints' in-degree */
int b200rec_mask_targets(const int64_t* positions, int64_t n, int64_t n_edges, const int64_t* u2i, const int64_t* i2u,
                         uint32_t* skip_bits, int* deg, b200rec_stream_t stream);

/* ---- K6  device-side collate of the dynamic-profile batches (csrc/collate.cu) -----------------------------------------
 * Replaces DynamicProfilesProvider.collate_interacted_items (src/content_providers/dynamic_profiles_provider.py:30-73; sklearn
 * MultiLabelBinarizer + pandas `.loc` per batch on the host) for a provider whose rating lists are resident in HBM:
 *   list_ptr  (n_users + 1) int64   CSR over ALL users of the provider
 *   list_item int32                 item numbers (rows of the profile table), ascending inside a user (the reference relies on the same order, :64)
 *   list_val  fp32 or NULL          rating - (meanRating + 2.5) / 2, computed in float64 and rounded once (:66); NULL = ignore_ratings (ones)
 * For the B users `user_rows` of a batch (repeats allowed):
 *   rated      (>= I) int64         ascending item numbers of the union of their lists  = rated_items_ids (:59)
 *   um_row_ptr (B + 1), um_col, um_val   CSR of user_matrix (B, I): col = position of the item in `rated`, list order inside a row; entries
 *                                   whose value is exactly 0.0 are absent (the dense matrix uses 0.0 for "unrated", attention_ncf.py:158-159)
 *   counts     int32[2]             { I, nnz }  (device memory)
 * Capacities are the caller's: `rated` holds min(n_items, total list length of the batch) entries, um_col / um_val the batch's non-zero
 * count (host-known from per-user counts).  Integer work, bit-exact against the host collate. */
size_t b200rec_collate_workspace(int64_t B, int64_t n_items);
int b200rec_collate_interacted(const int64_t* user_rows, int64_t B, const int64_t* list_ptr, const int* list_item, const float* list_val,
                               int64_t n_items, int64_t* rated, int* um_row_ptr, int* um_col, float* um_val, int* counts,
                               void* workspace, size_t workspace_bytes, b200rec_stream_t stream);

/* ---- K7  negative sampling of the ranking datasets (csrc/neg_sample.cu) -----------------------------------------------
 * Replaces RankingDataset.__getitem__'s per-sample np.random.choice (src/neural_collaborative_filtering/datasets/base.py:57-78,
 * 'sum_dynamic': p_k = r_k^w / sum_j r_j^w, w = 0 -> uniform) for datasets whose negative lists are resident in HBM as CSR over
 * samples (neg_ptr int64 (n_samples + 1), neg_item int64, neg_rating fp32 or NULL = uniform).  For every row b of the batch:
 * u_b = 53-bit uniform from Philox2x32-10 (counter = offset + b, key = seed), out_item[b] = the first list element whose cumulative
 * weight exceeds u_b * total (np.random.choice's inverse-CDF rule, float64); -1 for an empty list.  out_pos (position inside the
 * list) and out_u (the uniforms, for parity tests) are optional.  The caller advances `offset` by B per batch. */
int b200rec_sample_negatives(const int64_t* sample_rows, int64_t B, const int64_t* neg_ptr, const int64_t* neg_item, const float* neg_rating,
                             double w, uint64_t seed, uint64_t offset, int64_t* out_item, int* out_pos, double* out_u,
                             b200rec_stream_t stream);

/* ---- peer-memory exchange of the partitioned GraphNCF propagation (csrc/peer.cu) --------------------------------------
 * One process per GPU of an NVSwitch box.  Each rank allocates ONE arena, exports it as a CUDA IPC handle (64 opaque bytes,
 * exchanged by the host code), and maps the arenas of its peers.  The data path then consists of this library's kernels
 * only: K3 pushes partial rows to their owner (b200rec_spmm_t.push_*), b200rec_peer_reduce adds the receive slots in rank
 * order, b200rec_linear_shortk_push broadcasts the transformed rows, b200rec_peer_signal / _wait order the ranks (epoch
 * flags in the arenas; release/acquire at system scope; the wait gives up after timeout_ns and sets *err_flag instead of
 * hanging the GPU).  Replaces what a multi-GPU form of models/gnn_ncf.py:336-345 would do with all-gather / all-reduce. */
int b200rec_peer_alloc(size_t bytes, void** dev_ptr, unsigned char* handle /* host, B200REC_PEER_HANDLE_BYTES */);
int b200rec_peer_open(const unsigned char* handle /* host */, void** dev_ptr);
int b200rec_peer_close(void* dev_ptr);
int b200rec_peer_free(void* dev_ptr);
/* peer_flags: HOST array of n_peers device pointers to every rank's flag block (uint32 [B200REC_PEER_CHANNELS][B200REC_PEER_MAX]);
 * counters: LOCAL uint32 [2 * B200REC_PEER_CHANNELS] (signals sent | waits passed), zero-initialised once */
int b200rec_peer_signal(void* const* peer_flags, int n_peers, int rank, int channel, uint32_t* counters, b200rec_stream_t stream);
int b200rec_peer_wait(const uint32_t* flags, int n_peers, int channel, uint32_t* counters, int64_t timeout_ns, int* err_flag,
                      b200rec_stream_t stream);
/* x_next[r] = sum_{s < n_slots} recv[s * slot_stride + r * ld_recv ..] (slot order);  acc_out = (acc_in + x_next) * acc_scale */
int b200rec_peer_reduce(const float* recv, int n_slots, int64_t slot_stride, int64_t ld_recv, int64_t rows, int d, float* x_next,
                        int64_t ld_x, const float* acc_in, float* acc_out, int64_t ld_acc, float acc_scale, b200rec_stream_t stream);
/* copies src (rows, d) to (float*)dst[q] + dst_offset for every q < n_dst (dst: HOST array of device pointers) */
int b200rec_peer_push_rows(const float* src, int64_t ld_src, int64_t rows, int d, void* const* dst, int n_dst, int64_t dst_offset,
                           int64_t ld_dst, b200rec_stream_t stream);
/* batch rows (models/gnn_ncf.py:354-357 on a partitioned embedding): for every j < n_ids with row0 <= ids[j] < row0 + rows,
 * row (dst_offset / ld_dst + j) of every destination receives table[ids[j] - row0] * scale */
int b200rec_peer_gather_rows(const float* table, int64_t ld, int64_t row0, int64_t rows, const int64_t* ids, int64_t n_ids, int d,
                             float scale, void* const* dst, int n_dst, int64_t dst_offset, int64_t ld_dst, b200rec_stream_t stream);

/* tracing aid: *slot = %globaltimer (ns) when the stream reaches this point (one 1-thread kernel; usable inside a captured graph) */
int b200rec_device_timestamp(uint64_t* slot, b200rec_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* B200REC_H */
