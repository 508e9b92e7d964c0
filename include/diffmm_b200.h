/* diffmm_b200 — C ABI of the B200 (sm_100a) DiffMM hot-path library.
 *
 * The reference (sun2ot/DiffMM) is pure Python/PyTorch and has no FFI layer; its hot path is
 * the set of ATen/cuBLAS/cuSPARSE calls listed in SURVEY.md §2.1.  Each entry point below
 * replaces one of those call sites (cited as reference file:line) and is what a maintainer
 * binds from Python with ctypes (see INTEGRATION.md for the stub).
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless named h_*;
 *   - nothing is allocated inside: the caller passes outputs and workspaces
 *     (dmm_*_workspace_bytes tells how much);
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*), touches only
 *     the current device of `ctx`, and returns 0 or a negative dmm_status; the message of the
 *     last failure on the calling thread is dmm_last_error();
 *   - "bf16" buffers are raw uint16_t bit patterns (round-to-nearest-even);
 *   - leading dimensions (ld*) are in ELEMENTS.
 */
#ifndef DIFFMM_B200_H_
#define DIFFMM_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct dmm_ctx dmm_ctx;

enum dmm_status {
  DMM_OK = 0,
  DMM_ERR_INVALID = -1,   /* bad argument (shape, alignment, null)   */
  DMM_ERR_CUDA = -2,      /* CUDA runtime / driver error             */
  DMM_ERR_UNSUPPORTED = -3,
  DMM_ERR_WORKSPACE = -4  /* workspace too small                     */
};

/* ---- library / context ------------------------------------------------------------------ */
int dmm_version(void);
const char* dmm_last_error(void);
/* Context for CUDA device `device` (must be sm_100); resolves cuTensorMapEncodeTiled.  Does not change the calling
 * thread's current device: every later call launches on the current device, which must be `device`. */
int dmm_init(int device, dmm_ctx** out);
void dmm_destroy(dmm_ctx* ctx);
int dmm_num_sms(const dmm_ctx* ctx);

/* ---- operand packing --------------------------------------------------------------------
 * fp32 [rows, cols] (ld_src) -> bf16 hi (and optionally lo = bf16(x - hi)) [rows, ld_dst].
 * With transpose != 0 the destination is [cols, ld_dst] (dst[c, r] = src[r, c]).
 * Replaces the implicit fp32 operand read of F.linear (Model.py:212,215).                  */
int dmm_pack_bf16(dmm_ctx* ctx, const float* src, int64_t rows, int64_t cols, int64_t ld_src,
                  uint16_t* dst_hi, uint16_t* dst_lo, int64_t ld_dst, int transpose, void* stream);

/* Both orientations of one fp32 matrix from a single read: nat = bf16 hi (+ lo) [rows, ld_nat] (zero padded,
 * cols <= ld_nat <= pad64(cols)) and tr = its transpose [cols, ld_tr] (ld_tr >= rows).  For weights that feed a
 * contraction both ways (nn.Linear forward and input gradient; gather table and operand of the reverse chain). */
int dmm_pack_bf16_pair(dmm_ctx* ctx, const float* src, int64_t rows, int64_t cols, int64_t ld_src,
                       uint16_t* nat_hi, uint16_t* nat_lo, int64_t ld_nat, uint16_t* tr_hi, uint16_t* tr_lo,
                       int64_t ld_tr, void* stream);

/* Binary CSR user rows -> dense GEMM operand.  For r in [0, n_rows): row_ids[r] (or row0 + r
 * when row_ids == NULL) selects the CSR row; writes x_f32[r, :] (ld_x, fp32 0/1, optional) and
 * a_bf16[r, :] (ld_a, bf16 0/1, optional), zero filling both up to n_cols.
 * Replaces DiffusionData.__getitem__ + default collate (DataHandler.py:217-225) over the dense
 * U x I matrix (DataHandler.py:128).                                                        */
int dmm_csr_rows_to_dense(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices,
                          const int64_t* row_ids, int64_t row0, int64_t n_rows, int64_t n_cols,
                          float* x_f32, int64_t ld_x, uint16_t* a_bf16, int64_t ld_a, void* stream);

/* Time embedding columns (Model.py:196-202): temb = [cos(t f), sin(t f)] W_e^T + b_e written as
 * bf16 hi/lo into columns [col0, col0+d) of a_hi/a_lo (ld_a) and optionally fp32 into temb_f32
 * [n_rows, d].  `t` int64 per row, or NULL with `t_all` for every row (Model.py:319).        */
int dmm_time_embedding(dmm_ctx* ctx, const int64_t* t, int64_t t_all, int64_t n_rows, int d_emb,
                       const float* emb_w, const float* emb_b, uint16_t* a_hi, uint16_t* a_lo,
                       int64_t ld_a, int64_t col0, float* temb_f32, void* stream);

/* Time embedding folded into a bias (reverse chain: every row of a step shares t, Model.py:319):
 * bias_eff[i, h] = b[h] + sum_j w[h, col0 + j] * temb_j(t0 + i) for i in [0, n_t), temb as in
 * dmm_time_embedding, fp32 [n_t, n_out] (all steps of the chain in one launch).
 * Replaces the 10 extra operand columns of cat([x_t, temb]) (Model.py:202-203,212) for constant t. */
int dmm_time_bias(dmm_ctx* ctx, int64_t t0, int64_t n_t, int d_emb, const float* emb_w, const float* emb_b,
                  const float* w, int64_t ld_w, int64_t col0, const float* b, int64_t n_out,
                  float* bias_eff, void* stream);

/* First Denoise layer on binary CSR rows (x_t = x0 at the start of the reverse chain, Model.py:300-304):
 * h[r, :] = act(bias + sum_{c in row r} wt[c, :]), wt = W^T packed bf16 hi (+ lo) [n_cols, ld_w],
 * written as bf16 hi (+ lo) [n_rows, ld_h].  The dense contraction of Model.py:212 degenerates to a
 * gather-sum for 0/1 rows; rows are selected like in dmm_csr_rows_to_dense.  z_f32 (optional,
 * [n_rows, ld_z]) receives the plain sums x0 . W^T without bias: the fp32 state of the hidden-space
 * reverse chain.  `order` (optional, int32 [n_rows], a permutation of 0..n_rows-1) is the order in which
 * the rows are SCHEDULED (results do not depend on it): with the users of hundreds of interactions first,
 * their long gather chains overlap the rest of the grid instead of forming its tail.  `vals` (optional, fp32,
 * indexed like `indices`): entry values of a non-binary sparse row (dmm_csr_qsample_values), h = act(bias +
 * sum_c vals[c] wt[c, :]); NULL = binary rows.                                                  */
int dmm_csr_gather_act(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const float* vals,
                       const int64_t* row_ids, const int32_t* order, int64_t row0, int64_t n_rows, int64_t n_cols, const uint16_t* wt_hi,
                       const uint16_t* wt_lo, int64_t ld_w, const float* bias, int act, int64_t n_out,
                       uint16_t* h_hi, uint16_t* h_lo, int64_t ld_h, float* z_f32, int64_t ld_z, void* stream);

/* q_sample with the default noise (Model.py:324-341) restricted to BINARY CSR rows: sign(x0) zeroes the noise
 * wherever x0 is zero, so x_t keeps the row's sparsity pattern and only its entry values are needed:
 * vals[e] = coef_a + coef_b * noise[r, indices[e]] / max(||noise[r, :n_cols]||_2, 1e-12) for every entry e of the
 * selected rows (vals is indexed like `indices`; noise is the full fp32 randn block [n_rows, ld_noise], read once).
 * Keeps the first layer of a sampling_step > 0 rebuild (conf/baby.toml: 5) a gather-sum.            */
int dmm_csr_qsample_values(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                           int64_t row0, int64_t n_rows, int64_t n_cols, const float* noise, int64_t ld_noise,
                           float coef_a, float coef_b, float* vals, void* stream);

/* The same values with the standard-normal rows GENERATED in the kernel (Philox4x32-10 keyed by the 64-bit *seed, a
 * DEVICE scalar drawn from the framework's generator; counter = (row id, column / 4); Box-Muller): no randn block is
 * written to or read from HBM.  Element (r, c) is a pure function of (seed, r, c): deterministic per seed, independent of
 * blocking and launch geometry.  i.i.d. N(0, 1) like Model.py:337; not torch's stream.
 * full_rows != 0: all n_cols normals of every row are generated (norm pass + per-entry lookups).
 * full_rows == 0: only the row's support normals (the same elements (seed, r, c)) plus ONE chi-square(n_cols - k) variate
 * for the squared norm of the rest (Marsaglia-Tsang): the outputs depend on the row only through n_S and ||n||^2, and
 * (n_S, ||n||^2 - ||n_S||^2) ~ N(0, I_k) x chi^2(n_cols - k) independent, so the joint distribution of the outputs is
 * exactly the reference's at O(k) instead of O(n_cols) work per row.                                           */
int dmm_csr_qsample_values_rng(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                               int64_t row0, int64_t n_rows, int64_t n_cols, const int64_t* seed, float coef_a,
                               float coef_b, float* vals, int full_rows, void* stream);

/* dmm_csr_gather_act with the rows divided by length inside one launch.  `order` and `n_long` come from
 * dmm_rows_long_first (order: the rows of more than `threshold` entries first; n_long = its counters[0], a DEVICE scalar:
 * how many they are; no host sync) and max_long is any host-side upper bound of *n_long (e.g. nnz / (threshold + 1)).
 * The long rows take one warp per (row, 256-column slice) like dmm_csr_gather_act, every other row ONE warp for all its
 * columns (item ids and values broadcast once per entry, ceil(n_out / 256) independent gathers per entry and lane, the
 * per-row overhead paid once).  n_out <= 1024.  Results are bit-identical to dmm_csr_gather_act (same order of
 * summation).  Model.py:212 on the CSR rows, like dmm_csr_gather_act.                                        */
int dmm_csr_gather_act_split(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const float* vals,
                             const int64_t* row_ids, const int32_t* order, const int32_t* n_long, int64_t max_long,
                             int64_t row0, int64_t n_rows, int64_t n_cols, const uint16_t* wt_hi, const uint16_t* wt_lo,
                             int64_t ld_w, const float* bias, int act, int64_t n_out, uint16_t* h_hi, uint16_t* h_lo,
                             int64_t ld_h, float* z_f32, int64_t ld_z, void* stream);

/* Scheduling order for dmm_csr_gather_act: order[] (int32 [n_rows]) becomes a permutation of 0..n_rows-1 with every
 * row of the block [row0, row0 + n_rows) that has more than `threshold` entries in front (arbitrary order among
 * equals; `counters` is 2 int32 of device scratch).  No host sync.                                         */
int dmm_rows_long_first(dmm_ctx* ctx, const int64_t* indptr, int64_t row0, int64_t n_rows, int64_t threshold,
                        int32_t* order, int32_t* counters, void* stream);

/* y[r] = sum_k w[r, k] x[k], k < K (fp32): q = W1[:, :I] b2 of the hidden-space reverse chain (the image of
 * the second layer's bias, Model.py:215, under the first layer, Model.py:212).                          */
int dmm_gemv_f32(dmm_ctx* ctx, const float* w, int64_t ld_w, int64_t n_rows, int64_t K, const float* x,
                 float* y, void* stream);

/* h = act(z + bias) packed to bf16 hi (+ lo): the hidden layer tanh(z_t + b1'(t)) of the hidden-space
 * reverse chain, where z_t = x_t W1^T is carried in fp32 (Model.py:212-213 applied to the chain's state). */
int dmm_bias_act_pack(dmm_ctx* ctx, const float* z, int64_t ld_z, const float* bias, int64_t n_rows,
                      int64_t n_cols, int act, uint16_t* h_hi, uint16_t* h_lo, int64_t ld_h, void* stream);

/* x[r, c] += beta for every CSR entry (r, c) of the selected rows, x given as bf16 hi (+ lo):
 * the c2 * x0 term of the posterior mean (Model.py:375) for binary x0.                        */
int dmm_csr_axpy_bf16(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                      int64_t row0, int64_t n_rows, int64_t n_cols, float beta, uint16_t* x_hi,
                      uint16_t* x_lo, int64_t ld_x, void* stream);

/* q_sample (Model.py:324-341): x_t = a[r] x0 + b[r] noise with fp32 per-row coefficients
 * (the fp64->fp32 cast of Model.py:352 is done by the caller).  mode 0: `noise` is used as is.
 * mode 1: the default noise sign(x0) * normalize_row(noise) (Model.py:337, eps 1e-12).
 * Writes x_t fp32 (ld_x) and optionally bf16 hi/lo (ld_a).                                   */
int dmm_q_sample(dmm_ctx* ctx, const float* x0, int64_t ld_x0, const float* noise, int64_t ld_noise,
                 const float* coef_a, const float* coef_b, int64_t n_rows, int64_t n_cols, int mode,
                 float* x_t, int64_t ld_x, uint16_t* a_hi, uint16_t* a_lo, int64_t ld_a, void* stream);

/* ---- dense contraction on tcgen05 / TMEM / TMA -------------------------------------------
 * C[M,N] = epilogue( A[M,K] . B[N,K]^T ), both operands K-major bf16, fp32 accumulation in TMEM.
 * a_lo / b_lo (nullable) add the split-bf16 correction passes A_lo.B_hi and A_hi.B_lo, which
 * make the product fp32-faithful (rel ~1e-5) on the bf16 tensor pipe.
 * Replaces cuBLAS SGEMM behind nn.Linear / torch.mm (Model.py:205,208,212,215,416-417).
 * Output rows leave through 16-byte TMA units: the padding columns N .. round_up(N, 4 fp32 / 8 bf16)
 * of an output row (inside ld_out / ld_out16 by the rules above) may be overwritten.            */
typedef struct dmm_gemm_epilogue {
  const float* bias;      /* [N] added per column, or NULL                                   */
  int32_t act;            /* 0 none, 1 tanh (Model.py:213)                                   */
  float alpha;            /* v = alpha * v (+ beta * residual)  — posterior mean, Model.py:375 */
  float beta;
  const float* residual;  /* fp32 [M,N] ld_res, or NULL                                      */
  int64_t ld_res;
  float* out_f32;         /* optional fp32 [M,N]                                             */
  int64_t ld_out;
  uint16_t* out_hi;       /* optional bf16 [M,N] (operand of the next contraction)           */
  uint16_t* out_lo;       /* optional bf16 residual part                                     */
  int64_t ld_out16;
  const uint16_t* res_hi; /* residual given as bf16 hi (+ lo) instead of fp32 (exclusive with */
  const uint16_t* res_lo; /* `residual`); may alias out_hi/out_lo: each element is read, then  */
  int64_t ld_res16;       /* written, by the same thread                                      */
  int32_t res_pre_act;    /* != 0: v = alpha * act(acc + bias + beta * R) — the residual is a partial  */
                          /* sum of the same contraction (K processed in chunks), added before act    */
  int32_t post_act;       /* second stage on the bf16 output only: out_hi/lo = post_act(v + post_bias) */
  const float* post_bias; /* while out_f32 keeps v (hidden-space chain: z_t and h_{t-1} in one pass)    */
  float* cmax;            /* optional fp32 [M, ld_cmax]: cmax[r, c] = max(v[r, 32c .. 32c+31]) over the columns < N,  */
  int64_t ld_cmax;        /* NaN if any of them is NaN (max.NaN); ld_cmax >= ceil(N / 32).  The pruning side array   */
                          /* of dmm_topk_edges_pruned: 1/32 of the output bytes, written from the accumulator          */
                          /* registers, so the top-k never has to re-read the rows the contraction just wrote          */
} dmm_gemm_epilogue;

int dmm_gemm_bf16_tn(dmm_ctx* ctx, const uint16_t* a_hi, const uint16_t* a_lo, int64_t lda,
                     const uint16_t* b_hi, const uint16_t* b_lo, int64_t ldb,
                     int64_t M, int64_t N, int64_t K, const dmm_gemm_epilogue* ep, void* stream);

/* Split-K form for contractions with few output tiles and a long K (P = W1[:, :I] . W2 of the hidden-space chain,
 * [H, H] over I items: 16 pair tiles on 74 tile slots): C = A[M,K] . B[N,K]^T, single-pass bf16, no epilogue terms.  The k
 * blocks of every tile are divided over up to 8 work items of the same persistent launch; their fp32 partial products go to
 * slabs of `workspace` (dmm_gemm_splitk_workspace_bytes; 0 when the shape does not split) and a second launch adds the slabs
 * in a fixed order (deterministic) into out_f32 and / or the bf16 operand copies out_hi (+ out_lo = bf16(c - hi)).      */
int64_t dmm_gemm_splitk_workspace_bytes(dmm_ctx* ctx, int64_t M, int64_t N, int64_t K);
int dmm_gemm_bf16_tn_splitk(dmm_ctx* ctx, const uint16_t* a_hi, int64_t lda, const uint16_t* b_hi, int64_t ldb,
                            int64_t M, int64_t N, int64_t K, float* out_f32, int64_t ld_out, uint16_t* out_hi,
                            uint16_t* out_lo, int64_t ld_out16, void* workspace, int64_t workspace_bytes, void* stream);

/* Same contract on the fp32 CUDA-core pipe from fp32 operands (verification mode; no tensor cores). */
int dmm_gemm_f32_tn(dmm_ctx* ctx, const float* a, int64_t lda, const float* b, int64_t ldb,
                    int64_t M, int64_t N, int64_t K, const dmm_gemm_epilogue* ep, void* stream);

/* ---- per-user variable-k top-k -> edge list ------------------------------------------------
 * For row r of scores [n_rows, n_cols] (ld) emits the k_r = out_ptr[r+1]-out_ptr[r] largest
 * entries' column indices into out_items[out_ptr[r] .. out_ptr[r+1]) sorted ascending by column,
 * and row_base + r into out_users.  Tie-break: value descending, then column ascending.
 * k_r > n_cols is an error flagged by OR-ing bit 0 into *status (device int, optional; never cleared here).  `order` (optional, int32
 * permutation of 0..n_rows-1, e.g. from dmm_rows_long_first) is the order in which rows are scheduled;
 * results do not depend on it.  Rows wider than 8192 columns go through a column-segment pass plus a merge
 * when a `workspace` of dmm_topk_workspace_bytes(n_cols, n_edges) bytes is given (n_edges >= the number of
 * entries this call emits, out_ptr[n_rows] - out_ptr[0]); workspace == NULL keeps one CTA per whole row.
 * Replaces the per-user torch.topk loop + int(indices[j]) syncs of Main.py:224-230.          */
int64_t dmm_topk_workspace_bytes(int64_t n_cols, int64_t n_edges);
int dmm_topk_edges(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, int64_t n_cols,
                   const int64_t* out_ptr, int64_t row_base, int32_t* out_users, int32_t* out_items,
                   int32_t* status, const int32_t* order, void* workspace, int64_t workspace_bytes,
                   int64_t n_edges, void* stream);

/* Same contract and bit-identical output, for scores whose producer also wrote the chunk maxima
 * cmax[r, c] = max(scores[r, 32c .. 32c+31]) (dmm_gemm_epilogue.cmax; fp32 [n_rows, ld_cmax], ld_cmax % 4 == 0,
 * NaN-propagating): a row's k largest scores lie in the k chunks with the largest maxima, so the kernel reads
 * 4 * n_cols / 32 + 128 * k bytes per row instead of 4 * n_cols.  Rows that do not qualify (k > 64, k chunks more than
 * a quarter of the row, NaN scores, crowded ties) are collected on the device and finished in the same call by a small
 * persistent grid: two-level exact radix select (top-k of the chunk maxima, then top-k of those chunks' scores) or, for
 * rows with NaN / k chunks above half of the row, the whole-row generic path.
 * `workspace` (required): dmm_topk_pruned_workspace_bytes(n_rows, n_cols, n_edges).                              */
int64_t dmm_topk_pruned_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t n_edges);
int dmm_topk_edges_pruned(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, int64_t n_cols,
                          const float* cmax, int64_t ld_cmax, const int64_t* out_ptr, int64_t row_base,
                          int32_t* out_users, int32_t* out_items, int32_t* status, const int32_t* order,
                          void* workspace, int64_t workspace_bytes, int64_t n_edges, void* stream);

/* ---- normalised bipartite adjacency ---------------------------------------------------------
 * From a user->item edge list in CSR form (row_ptr int64 [U+1], items int32 sorted ascending and
 * unique within a row) builds A = D^-1/2 ([[0,R],[R^T,0]] + I) D^-1/2 as CSR over N = U + I nodes:
 * adj_ptr int64 [N+1], adj_idx int32 [2E+N] (sorted within rows), adj_val fp32 with the
 * reference's fp64 arithmetic (d_r^-1/2 * 1) * d_c^-1/2 rounded to fp32.
 * An item id outside [0, n_items) is an error flagged by OR-ing bit 1 into *status (device int, optional; the
 * arrays written for such a list are unspecified and must not be used).
 * Replaces Coach.makeTorchAdj (Main.py:113-116) -> DataHandler.makeTorchAdj / normalizeAdj
 * (DataHandler.py:53-93), which run on the host in scipy.                                    */
int64_t dmm_build_adj_workspace_bytes(int64_t n_users, int64_t n_items, int64_t n_edges);
int dmm_build_norm_adj_csr(dmm_ctx* ctx, const int64_t* row_ptr, const int32_t* items,
                           int64_t n_users, int64_t n_items, int64_t n_edges,
                           int64_t* adj_ptr, int32_t* adj_idx, float* adj_val,
                           void* workspace, int64_t workspace_bytes, int32_t* status, void* stream);

/* ---- CSR SpMM ------------------------------------------------------------------------------
 * Y[r0:r1, :] = alpha * A[r0:r1, :] . X (+ beta * Z[r0:r1, :]),  X fp32 [N_cols, D] (ld_x).
 * `row0,row1` select a row block (row-partitioned propagation); Y/Z are indexed by absolute row.
 * D must be a multiple of 4 and <= 256.  A symmetric => the backward is the same call.
 * Replaces torch.sparse.mm (Model.py:90,93,105,111,114,123,130; Main.py:319).
 *
 * Item popularity is heavy tailed, so for D == 64 a `plan` (built once per adjacency by
 * dmm_spmm_plan; device-resident, no host sync; at most 2^25 rows) lists the rows with more than 64
 * neighbours; they are cut into 64-neighbour chunks whose partial rows go through `workspace`
 * (dmm_spmm_workspace_bytes) and are added in a fixed order (deterministic), and lists the other rows
 * sorted by length, so that the lanes of a warp run equal trip counts.  plan == NULL keeps the
 * one-CTA-per-long-row path.  `nnz` is the number of stored entries of A (sizes the plan).      */
int64_t dmm_spmm_plan_bytes(int64_t n_rows, int64_t nnz);
int dmm_spmm_plan(dmm_ctx* ctx, const int64_t* adj_ptr, int64_t n_rows, int64_t nnz, void* plan,
                  int64_t plan_bytes, void* stream);
int64_t dmm_spmm_workspace_bytes(int64_t nnz, int64_t D);
int dmm_spmm_csr(dmm_ctx* ctx, const int64_t* adj_ptr, const int32_t* adj_idx, const float* adj_val,
                 int64_t row0, int64_t row1, const float* x, int64_t ld_x, int64_t D,
                 float alpha, float beta, const float* z, int64_t ld_z,
                 float* y, int64_t ld_y, const void* plan, int64_t nnz, void* workspace,
                 int64_t workspace_bytes, void* stream);

/* Propagation in the single-pass "bf16" precision for adjacencies whose values are SEPARABLE, val = d_r^-1/2 d_c^-1/2
 * with d_r = the number of stored entries of row r (what dmm_build_norm_adj_csr and DataHandler.normalizeAdj produce:
 * D^-1/2 (A + I) D^-1/2; SURVEY App. D.7).  dmm_spmm_table_bf16 writes the gather table T = bf16(d^-1/2 X) [n_rows, 64]
 * (X = [x ; x2] split at row n_first: the reference's torch.cat([u_embs, i_embs]) is never materialised; x2 may be NULL
 * when n_first >= n_rows) and dmm_spmm_norm_bf16 computes Y[r] = alpha d_r^-1/2 sum_{c in row r} T[c] (+ beta Z[r]): no
 * value stream, 128-byte rows through the L2, fp32 accumulation (FHADD.BF16).  d^-1/2 comes from the plan (dmm_spmm_plan
 * of the same adjacency; its row pointers define d).  Same plan / workspace / determinism as dmm_spmm_csr.      */
int dmm_spmm_table_bf16(dmm_ctx* ctx, const float* x, int64_t ld_x, int64_t n_first, const float* x2, int64_t ld_x2,
                        int64_t n_rows, const void* plan, int64_t nnz, uint16_t* t, void* stream);
int dmm_spmm_norm_bf16(dmm_ctx* ctx, const int32_t* adj_idx, int64_t row0, int64_t row1, int64_t n_rows, const uint16_t* t,
                       float alpha, float beta, const float* z, int64_t ld_z, float* y, int64_t ld_y, const void* plan,
                       int64_t nnz, void* workspace, int64_t workspace_bytes, void* stream);

/* Cross-layer CL perturbation (Main.py:320-321) fused with nothing else:
 * e[r,:] += sign(e[r,:]) * rnd[r,:] / max(||rnd[r,:]||, 1e-12) * noise_degree, in place. */
int dmm_sign_noise_(dmm_ctx* ctx, float* e, int64_t ld_e, const float* rnd, int64_t ld_r,
                    int64_t n_rows, int64_t D, float noise_degree, void* stream);

/* ---- element-wise glue of Model.gcn_MM between its SpMM products (Model.py:60-134), forward and backward ----------
 * F.normalize of the projected modality features (Model.py:89-93,104-105): y[r,:] = x[r,:] / max(||x[r,:]||_2, eps);
 * inv[r] = +-1 / max(||x||, eps), negative when the row was clamped at eps (flag for the backward).
 * Backward: gx = (g - y (y . g)) |inv| for an unclamped row, g |inv| for a clamped one.                             */
int dmm_rownorm_fwd(dmm_ctx* ctx, const float* x, int64_t ld_x, int64_t n_rows, int64_t D, float eps, float* y, int64_t ld_y,
                    float* inv, void* stream);
int dmm_rownorm_bwd(dmm_ctx* ctx, const float* y, int64_t ld_y, const float* inv, const float* g, int64_t ld_g, int64_t n_rows,
                    int64_t D, float* gx, int64_t ld_gx, void* stream);
/* The modality mix (Model.py:116-119,125-127): out = sum_m w[m] (y + lam z[m]) over dense fp32 arrays of n_elems elements
 * (multiple of 4, 16-byte aligned), w = softmax(modal_weight) on the DEVICE (no host sync), 1 <= n_modal <= 4, evaluated
 * in the reference's order of operations.  Backward: gy = sum_m w[m] g, gz[m] = lam w[m] g (gz[m] may be NULL), and
 * partial[b, m] = sum over CTA b of g . (y + lam z[m]) for b < dmm_modal_mix_partial_rows(n_elems): the caller adds the
 * rows in a fixed order to get d/dw[m] (deterministic, no atomics).                                               */
int dmm_modal_mix_fwd(dmm_ctx* ctx, const float* y, const float* const* z, const float* w, int32_t n_modal, float lam,
                      int64_t n_elems, float* out, void* stream);
int64_t dmm_modal_mix_partial_rows(int64_t n_elems);
int dmm_modal_mix_bwd(dmm_ctx* ctx, const float* g, const float* y, const float* const* z, const float* w, int32_t n_modal,
                      float lam, int64_t n_elems, float* gy, float* const* gz, float* partial, void* stream);

/* ---- optimiser step (Main.py:92-110,189-192,375-377; SURVEY 8(f3)) ------------------------------------------------
 * One launch for the Adam update of ALL tensors of an optimiser (weight_decay 0, no amsgrad): p, g, m, v read once, p, m, v
 * written once, the operation sequence of torch.optim.Adam's capturable foreach implementation evaluated in its own order
 * (bit-identical update).  `step` (already incremented) and `lr` are fp32 DEVICE scalars: capturable in a CUDA graph.
 * params / grads / exp_avg / exp_avg_sq: host arrays of n_tensors device pointers (dense fp32), numel their lengths.     */
int dmm_adam_step(dmm_ctx* ctx, int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                  float* const* exp_avg_sq, const int64_t* numel, const float* step, const float* lr, double beta1,
                  double beta2, double eps, void* stream);

/* Same launch for torch's NON-capturable foreach sequence (eager trainer): step_size = -lr / (1 - beta1^t) and
 * bias_correction2_sqrt = sqrt(1 - beta2^t) are the python doubles of torch.optim.adam._multi_tensor_adam, cast to fp32
 * where torch's kernels cast them; p = p + step_size (m / ((sqrt(v) / bc2_sqrt) + eps)).                              */
int dmm_adam_step_host(dmm_ctx* ctx, int32_t n_tensors, float* const* params, const float* const* grads, float* const* exp_avg,
                       float* const* exp_avg_sq, const int64_t* numel, double step_size, double bias_correction2_sqrt,
                       double beta1, double beta2, double eps, void* stream);

/* ---- fused losses ---------------------------------------------------------------------------
 * BPR (Utils/Utils.py:78-98): loss = mean_b -log(1e-5 + sigmoid(u.p - u.n)) over gathered rows
 * users[b] of U_emb and pos[b]/neg[b] of I_emb; also writes d(loss)/d(rows) scaled by
 * `grad_scale` into g_u/g_p/g_n [B, D] (optional).                                           */
int dmm_bpr_fwd_bwd(dmm_ctx* ctx, const float* u_emb, int64_t ld_u, const float* i_emb, int64_t ld_i,
                    const int64_t* users, const int64_t* pos, const int64_t* neg, int64_t B, int64_t D,
                    float grad_scale, float* row_loss /* [B] scratch */, float* loss,
                    float* g_u, float* g_p, float* g_n, void* stream);

/* InfoNCE (Utils/Utils.py:57-75) on gathered rows idx[b] of v1/v2: row-L2 normalise, logits/temp,
 * -mean diag log-softmax, never materialising the B x B matrix in HBM.  Forward writes loss and
 * saves per-row log-sum-exp (lse, [B]) and inverse norms (inv1, inv2, [B]); backward writes
 * d(loss)/d(gathered rows) [B, D] for both views (caller scatter-adds by idx).
 * `workspace` holds dmm_infonce_workspace_floats(B, D, backward) floats (the normalised gathers
 * plus, for D == 64, the per-column-split partial results of the tiled kernels).             */
int64_t dmm_infonce_workspace_floats(int64_t B, int64_t D, int backward);
int dmm_infonce_fwd(dmm_ctx* ctx, const float* v1, int64_t ld1, const float* v2, int64_t ld2,
                    const int64_t* idx, int64_t B, int64_t D, float temperature,
                    float* workspace, float* row_loss /* [B] scratch */, float* loss,
                    float* lse, float* inv1, float* inv2, void* stream);
int dmm_infonce_bwd(dmm_ctx* ctx, const float* v1, int64_t ld1, const float* v2, int64_t ld2,
                    const int64_t* idx, int64_t B, int64_t D, float temperature,
                    const float* lse, const float* inv1, const float* inv2, float grad_scale,
                    float* workspace, float* g1, float* g2, void* stream);

/* ---- every loss of a joint-training step in one call (Main.py:309,333,345-367) -----------------------------------
 * BPR on the final embeddings plus up to 12 InfoNCE terms (2 cross-layer + 2 M or 2 C(M, 2) modality terms), D = 64.
 * A view is a whole node table [N, ld >= 64] (fp32); a term compares rows row_offset + idx[b] of v1 and v2 (row_offset
 * 0 for the user rows, n_users for the item rows) at `temperature` and enters the contrastive total with `weight`.
 * Forward (3 launches): losses[0 .. P) = the InfoNCE means, losses[P] = BPR, losses[P + 1] = sum_p weight_p losses[p];
 *   lse [P, B] and inv [P, 2, B] are kept for the backward.
 * Backward (3 launches): d(g_bpr * BPR + g_cl * contrastive total) is scatter-ADDED (atomicAdd) into the caller-zeroed
 *   gradient tables: grad_tables[2 p] / [2 p + 1] (HOST array of device pointers, leading dimensions grad_ld) receive
 *   the rows of v1 / v2 of term p, grad_tables[2 P] the three BPR row blocks; NULL entries are skipped.  g_cl / g_bpr
 *   are DEVICE scalars (the upstream gradients), so no host sync is needed.
 * `problems` and `bpr` are HOST structs (copied into the kernel parameters).
 * Replaces one bpr_loss and 4-8 InfoNCE calls of Utils/Utils.py:57-98 per step.                                  */
typedef struct dmm_nce_problem {
  const float* v1; int64_t ld1;
  const float* v2; int64_t ld2;
  const int64_t* idx;     /* [B] device */
  int64_t row_offset;
  float temperature, weight;
} dmm_nce_problem;
typedef struct dmm_bpr_problem {
  const float* emb; int64_t ld_emb;      /* final embeddings [N, ld]: users first, items from item_offset */
  int64_t item_offset;
  const int64_t *users, *pos, *neg;      /* [B] device */
} dmm_bpr_problem;
int64_t dmm_bpr_infonce_workspace_floats(int64_t B, int n_problems, int backward);
int dmm_bpr_infonce_fwd(dmm_ctx* ctx, const dmm_nce_problem* problems, int n_problems, const dmm_bpr_problem* bpr, int64_t B,
                        float* workspace, float* losses, float* lse, float* inv, void* stream);
int dmm_bpr_infonce_bwd(dmm_ctx* ctx, const dmm_nce_problem* problems, int n_problems, const dmm_bpr_problem* bpr, int64_t B,
                        const float* lse, const float* inv, const float* g_cl, const float* g_bpr, float* workspace,
                        float* const* grad_tables, const int64_t* grad_ld, void* stream);

/* Scatter-add of per-batch row gradients into a table gradient: dst[idx[b], :] += src[b, :]. */
int dmm_scatter_add_rows(dmm_ctx* ctx, const float* src, int64_t ld_s, const int64_t* idx, int64_t B,
                         int64_t D, float* dst, int64_t ld_d, void* stream);

/* ---- fused Denoise training step (Model.py:385-428 + :183-220; driver Main.py:145-192) -----------------------------
 * The step is scheduled by the host layer as twelve dmm_gemm_bf16_tn contractions per modality and batch plus the
 * kernels below; together they replace the per-op autograd chain (q_sample -> fp32 x_t -> torch.cat -> pack, sigmoid
 * gate, mse / cosine tails, tanh', bias-gradient sums, operand transposes).
 *
 * dmm_train_prep: x_t = tab_a[t_r] x0 + tab_b[t_r] noise (Model.py:338-341; tables = sqrt(abar), sqrt(1 - abar) as fp32)
 *   written directly as the bf16 operand a_hi (+ a_lo) [n_rows, ld_a] of the first layer, columns [0, n_cols); the time
 *   embedding (Model.py:196-202) goes to columns [n_cols, n_cols + d_emb); x0_hi (optional) receives x0 as a bf16
 *   operand; te_raw (optional, fp32 [n_rows, d_emb]) the raw [cos, sin] features for the emb_layer gradient.       */
int dmm_train_prep(dmm_ctx* ctx, const float* x0, int64_t ld_x0, const float* noise, int64_t ld_noise, const int64_t* t,
                   const float* tab_a, const float* tab_b, int64_t n_rows, int64_t n_cols, int d_emb, const float* emb_w,
                   const float* emb_b, uint16_t* a_hi, uint16_t* a_lo, int64_t ld_a, uint16_t* x0_hi, int64_t ld_x0h,
                   float* te_raw, void* stream);
/* Gate (Model.py:205-207, latdim 64): sig = sigmoid(p Wg^T + bg) (fp32 [n_rows, 64]), G = p * sig as bf16 operand.
 * dmm_gate_bwd_pre: dpre = dG * p * sig (1 - sig), the gradient at the gate's pre-activation.                     */
int dmm_gate_fwd(dmm_ctx* ctx, const float* p, int64_t ld_p, int64_t n_rows, const float* gate_w, const float* gate_b,
                 float* sig, uint16_t* g_hi, uint16_t* g_lo, int64_t ld_g, void* stream);
int dmm_gate_bwd_pre(dmm_ctx* ctx, const float* dg, int64_t ld_dg, const float* p, int64_t ld_p, const float* sig,
                     int64_t n_rows, float* dpre, void* stream);
/* Loss tail (Model.py:407-425).  diff = out - x0 (fp32, from the second layer's epilogue), umd = diff F, x0f = x0 F,
 * ui = x0 i_embs (all [n_rows, 64]): loss[r] = w_tab[t_r] * mean(diff_r^2) + sim_weight * (1 - cos(umd + x0f, ui)) in
 * float64 (the reference's dtypes); um = umd + x0f and stats = (dot, |um|, |ui|) are kept for the backward.
 * Backward: cm[r] = g_r w_r 2 / n_cols, dumc = (d loss / d um) / cm as a bf16 operand (the backward contractions work
 * on d_out' = diff + dumc F^T and apply the row scale cm afterwards), d_ui (optional) = d loss / d ui.            */
int dmm_diff_loss_fwd(dmm_ctx* ctx, const float* diff, int64_t ld_d, int64_t n_rows, int64_t n_cols, const float* umd,
                      int64_t ld_umd, const float* x0f, int64_t ld_x0f, const float* ui, int64_t ld_ui, const int64_t* t,
                      const double* w_tab, float sim_weight, double* loss, float* mse, float* um, float* stats, void* stream);
int dmm_diff_loss_bwd(dmm_ctx* ctx, const double* g_loss, const float* um, const float* ui, int64_t ld_ui, const float* stats,
                      const int64_t* t, const double* w_tab, float sim_weight, int64_t n_rows, int64_t n_cols, float* cm,
                      uint16_t* dumc_hi, uint16_t* dumc_lo, int64_t ld_dumc, float* d_ui, void* stream);
/* Hidden layer backward: dz = cm[r] dh (1 - h^2) as fp32, as bf16 operand [n_rows, ld_dz16], and transposed [H, ld_t]
 * together with (cm h)^T [H, ld_t]: the K = batch operands of the weight-gradient contractions.  h comes from h_f32
 * (fp32 [n_rows, ld_hf]) when given, else from h_hi (+ h_lo): tanh' of a saturated unit needs more than bf16's 8 bits.
 * cm NULL means no row scale: dz = dh (1 - h^2) and the transposed activation is h^T itself (the inner layers of a
 * deeper Denoise, whose dh already carries the scale).                                                               */
int dmm_hidden_bwd(dmm_ctx* ctx, const float* dh, int64_t ld_dh, const float* h_f32, int64_t ld_hf, const uint16_t* h_hi,
                   const uint16_t* h_lo, int64_t ld_h,
                   const float* cm, int64_t n_rows, int64_t H, float* dz_f32, int64_t ld_dz, uint16_t* dz_hi, uint16_t* dz_lo,
                   int64_t ld_dz16, uint16_t* dzt_hi, uint16_t* dzt_lo, uint16_t* hct_hi, uint16_t* hct_lo, int64_t ld_t,
                   void* stream);
/* dst[c, r] = src[r, c] for bf16 operands (hi and optionally lo); dst columns up to ld_dst are written (zero padded). */
int dmm_transpose_bf16(dmm_ctx* ctx, const uint16_t* src_hi, const uint16_t* src_lo, int64_t ld_src, int64_t rows,
                       int64_t cols, uint16_t* dst_hi, uint16_t* dst_lo, int64_t ld_dst, void* stream);
/* out[c] = sum_r row_scale[r] * src[r, c] (row_scale NULL = 1): bias gradients, rows added in order (deterministic).
   rows = 0 writes zeros; src may then be NULL. */
int dmm_colsum(dmm_ctx* ctx, const float* src, int64_t ld, int64_t rows, int64_t cols, const float* row_scale, float* out,
               void* stream);
/* out[m, n] = x^T y for skinny fp32 x [rows, m], y [rows, n] (m, n <= 64): gate / time-embedding weight gradients.
   rows = 0 writes zeros; x and y may then be NULL. */
int64_t dmm_atb_small_workspace_floats(int64_t m, int64_t n);
int dmm_atb_small(dmm_ctx* ctx, const float* x, int64_t ld_x, int64_t m, const float* y, int64_t ld_y, int64_t n, int64_t rows,
                  float* workspace, float* out, void* stream);

/* ---- evaluation tail (Main.py:390-448) ------------------------------------------------------------
 * dmm_eval_mask_scores: scores[r, c] = fill for every train item c of user row_ids[r] (CSR indptr / indices): the
 * `predict * (1 - trainMask) - trainMask * 1e8` of Main.py:410 with fill = -1e8, without the dense mask rows.
 * dmm_eval_metrics: for row r (user row_ids[r]) the K columns top_items[r*K .. r*K+K) (from dmm_topk_edges with k = K on
 * the masked scores) are ranked by (score desc, column asc) and compared with the user's test items
 * test_items[test_ptr[u] .. test_ptr[u+1]) in stored order: out[3r + 0/1/2] = recall, ndcg, precision in float64 with
 * calcRes' arithmetic (Main.py:422-448).  inv_log2[p] = 1 / log2(p + 2) (p < K) and max_dcg[t] (t <= K) are HOST-computed
 * float64 tables passed on the device so that every term equals numpy's.  K <= 32.                    */
int dmm_eval_mask_scores(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                         int64_t n_rows, int64_t n_cols, float* scores, int64_t ld, float fill, void* stream);
int dmm_eval_metrics(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, const int32_t* top_items, int64_t K,
                     const int64_t* row_ids, const int64_t* test_ptr, const int32_t* test_items,
                     const double* inv_log2, const double* max_dcg, double* out, void* stream);

/* ---- ranked recommendation lists and metrics at several cutoffs (Main.py:410-411, Main.py:422-448) -----------------
 * dmm_eval_mask_scores_cmax: dmm_eval_mask_scores (Main.py:410), then, for every 32-column chunk of row r that holds a
 * filled column, cmax[r * ld_cmax + c] is recomputed from the row as it now stands, exactly as dmm_gemm_epilogue.cmax
 * builds it (max over the columns < n_cols, NaN-propagating); other chunks are left unchanged.  The chunk maxima written by
 * the contraction stay valid upper bounds for dmm_topk_edges_pruned after the mask.  ld_cmax >= ceil(n_cols / 32).    */
int dmm_eval_mask_scores_cmax(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                              int64_t n_rows, int64_t n_cols, float* scores, int64_t ld, float fill, float* cmax,
                              int64_t ld_cmax, void* stream);
/* dmm_topn_rank: the torch.topk(predict, N) ranking of Main.py:411.  Row r's N columns sel[r * ld_sel + 0 .. N) (as
 * dmm_topk_edges[_pruned] emits them, ascending) are put into rank order: score descending, then column ascending, in the
 * top-k kernels' total order (-0.0 ties with +0.0, +NaN above +inf, -NaN below -inf), so the first k ranked entries are
 * dmm_topk_edges' k-set for every k <= N.  items[r * ld_items + i] = the i-th column, or -1 where its score is -inf;
 * out_scores[r * ld_out + i] = its score.  1 <= N <= 1024.                                                          */
int dmm_topn_rank(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, const int32_t* sel, int64_t ld_sel, int64_t N,
                  int32_t* items, int64_t ld_items, float* out_scores, int64_t ld_out, void* stream);
/* dmm_eval_metrics_cutoffs: calcRes (Main.py:422-448) at every cutoff of the HOST array cutoffs[0 .. n_cutoffs)
 * (strictly increasing, in 1..N) from one ranked list ranked[r * ld_ranked + 0 .. N) of user row_ids[r] (dmm_topn_rank's
 * items).  The user's test items test_items[test_ptr[u] .. test_ptr[u+1]) are walked once in stored order; one at position
 * p < c of the list is a hit at cutoff c and adds inv_log2[p].  out[(r * n_cutoffs + j) * 3 + 0/1/2] = recall = hits / tst,
 * ndcg = dcg / max_dcg[min(tst, c)], precision = hits / c in float64 (recall = ndcg = 0 for a user without test items).
 * inv_log2[p] = 1 / log2(p + 2) (p < N) and max_dcg[t] (t <= N) are host-computed float64 tables on the device.  N <= 1024.
 * For all three, n_rows = 0 is a no-op (the device pointers may then be NULL).                                             */
int dmm_eval_metrics_cutoffs(dmm_ctx* ctx, const int32_t* ranked, int64_t ld_ranked, int64_t n_rows, int64_t N,
                             const int32_t* cutoffs, int64_t n_cutoffs, const int64_t* row_ids, const int64_t* test_ptr,
                             const int32_t* test_items, const double* inv_log2, const double* max_dcg, double* out,
                             void* stream);

/* ---- scores of given pairs, rankings of given candidates (the user . item score of Main.py:410) --------------------
 * Both score a (user row, item row) pair of fp32 rows (D = 1..1024, leading dimensions ld_u, ld_i >= D) the same way:
 * each value is split in registers into hi = bf16_rn(x) and lo = bf16_rn(x - hi) (the operands of dmm_pack_bf16), and
 * score = sum over d of hi_u hi_i + hi_u lo_i + lo_u hi_i (x3 = 1, bf16x3) or of hi_u hi_i (x3 = 0, bf16), accumulated
 * in fp32 in a fixed order, so a pair gets the same bits from either function; a zero score is +0.0.  These are the
 * terms of the tensor-pipe contraction (dmm_gemm_bf16_tn), but not its bits: the summation order differs.
 * dmm_score_pairs: out[p] = score(user[u_idx[p]], item[i_idx[p]]) for p < P; a pair with u_idx outside [0, n_users) or
 * i_idx outside [0, n_items) gets NaN and reads no row.
 * dmm_rank_candidates: row r (< n_rows) ranks the candidates cand[r * ld_c + 0 .. C) for user row r in one launch, in
 * the top-k kernels' total order (score descending, then item ascending; -0.0 ties with +0.0, +NaN above +inf, -NaN
 * below -inf).  -1 or any id outside [0, n_items) is an empty slot; an item listed several times is ranked once.  The
 * first N ranked items go to out_items[r * ld_oi + i] with their scores in out_scores[r * ld_os + i], a score of -inf
 * included; only the slots past the row's distinct valid candidates hold (-1, -inf).  1 <= C <= 4096,
 * 1 <= N <= min(1024, C).  No score but the N emitted reaches global memory.
 * For both, zero pairs / rows is a no-op (the device pointers may then be NULL).                                      */
int dmm_score_pairs(dmm_ctx* ctx, const float* user, int64_t ld_u, int64_t n_users, const float* item, int64_t ld_i,
                    int64_t n_items, int64_t D, const int64_t* u_idx, const int32_t* i_idx, int64_t P, int x3, float* out,
                    void* stream);
int dmm_rank_candidates(dmm_ctx* ctx, const float* user, int64_t ld_u, const float* item, int64_t ld_i, int64_t n_items,
                        int64_t D, const int32_t* cand, int64_t ld_c, int64_t n_rows, int64_t C, int64_t N, int x3,
                        int32_t* out_items, int64_t ld_oi, float* out_scores, int64_t ld_os, void* stream);

/* ---- host helper (no device work) --------------------------------------------------------------
 * Replays the reference's rejection-sampling loop (TrainData.negSampling, DataHandler.py:159-169)
 * over `n_draws` values pre-drawn by the caller from the same numpy generator: interaction i
 * (user rows[i]) consumes draws until one is not in the user's sorted CSR row.  All pointers are
 * HOST pointers.  *consumed = draws used; DMM_ERR_WORKSPACE if the stream ran out.              */
int dmm_host_neg_sampling(const int64_t* h_indptr, const int32_t* h_indices, const int32_t* h_rows, int64_t n,
                          const int64_t* h_draws, int64_t n_draws, int32_t* h_negs, int64_t* consumed);

#ifdef __cplusplus
}
#endif
#endif /* DIFFMM_B200_H_ */
