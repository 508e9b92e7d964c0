// Evaluation tail on the device (reference Main.py:390-448): train-mask, top-K ranking and Recall / NDCG / Precision per
// test user without a host round trip per batch.
//
//   predict = score * (1 - mask) - mask * 1e8      (Main.py:410)  -> dmm_eval_mask_scores: the train items of each test
//                                                      user (CSR row) are overwritten with -1e8 in the score block
//   torch.topk(predict, K)                          (Main.py:411)  -> dmm_topk_edges with k = K for every row
//   calcRes                                         (Main.py:422-448) -> dmm_eval_metrics: one warp per user ranks its K
//                                                      selected columns by (score desc, column asc) and walks the user's
//                                                      test items in their stored order with the reference's float64
//                                                      arithmetic (the 1 / log2(pos + 2) and max-DCG tables come from
//                                                      the host's numpy, so every term is bit-identical to calcRes).
//
// Ranked recommendation lists and metrics at several cutoffs from one ranked list (diffmm_b200.recommend):
//   dmm_eval_mask_scores_cmax   the mask above, then the chunk maxima of the pruned top-k refreshed for every chunk it wrote
//   dmm_topn_rank               the N selected columns of a row put into rank order (bitonic sort in shared memory)
//   dmm_eval_metrics_cutoffs    calcRes at every cutoff c_1 < ... < c_m of one ranked list, one pass over the test items
#include "common.cuh"

namespace {

// NaN-propagating maximum (max.NaN.f32), the instruction the contraction's epilogue builds the chunk maxima with
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

// the top-k kernels' total order: -0.0 ties with +0.0, +NaN above +inf, -NaN below -inf
__device__ __forceinline__ uint32_t order_key(float f) {
  uint32_t u = __float_as_uint(f);
  if (u == 0x80000000u) u = 0u;
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// One warp per row.  CMAX: after the fills, every chunk that holds a filled column gets its maximum recomputed from the
// row as it now stands, in the epilogue's order (columns ascending from -inf, max.NaN); chunks holding several filled
// columns are recomputed once per column, to the same value.
template <bool CMAX>
__global__ void __launch_bounds__(256) eval_mask_kernel(const int64_t* __restrict__ indptr,
                                                        const int32_t* __restrict__ indices,
                                                        const int64_t* __restrict__ row_ids, int64_t n_rows,
                                                        int64_t n_cols, float* __restrict__ scores, int64_t ld,
                                                        float fill, float* __restrict__ cmax, int64_t ld_cmax) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  const int64_t u = row_ids[r];
  const int64_t b = indptr[u], e = indptr[u + 1];
  for (int64_t k = b + lane; k < e; k += 32) {
    const int32_t c = indices[k];
    if (c >= 0 && c < n_cols) scores[r * ld + c] = fill;
  }
  if (CMAX) {
    __syncwarp();   // the warp's fills are visible to all its lanes
    const float* row = scores + r * ld;
    for (int64_t k = b + lane; k < e; k += 32) {
      const int32_t c = indices[k];
      if (c < 0 || c >= n_cols) continue;
      const int64_t c0 = (int64_t)(c & ~31);
      float m = __uint_as_float(0xFF800000u);
      for (int j = 0; j < 32 && c0 + j < n_cols; ++j) m = fmax_nan(m, row[c0 + j]);
      cmax[r * ld_cmax + (c >> 5)] = m;
    }
  }
}

// One CTA of max(P / 2, 32) threads per row, P = the power of two >= N: the N (key, column) pairs are sorted ascending
// as the 64-bit words (~order_key(score) << 32 | column), i.e. score descending then column ascending, by a bitonic
// network in shared memory; pad words (all ones) sort last.
template <int P>
__global__ void __launch_bounds__(P / 2 < 32 ? 32 : P / 2) topn_rank_kernel(
    const float* __restrict__ scores, int64_t ld, const int32_t* __restrict__ sel, int64_t ld_sel, int N,
    int32_t* __restrict__ items, int64_t ld_items, float* __restrict__ out_scores, int64_t ld_out) {
  constexpr int NT = P / 2 < 32 ? 32 : P / 2;
  __shared__ uint64_t w[P];
  const int64_t r = blockIdx.x;
  const float* row = scores + r * ld;
  for (int i = threadIdx.x; i < P; i += NT) {
    uint64_t v = ~0ull;
    if (i < N) {
      const uint32_t c = (uint32_t)sel[r * ld_sel + i];
      v = ((uint64_t)~order_key(row[c]) << 32) | c;
    }
    w[i] = v;
  }
  __syncthreads();
#pragma unroll 1
  for (int k = 2; k <= P; k <<= 1) {
#pragma unroll 1
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int i = threadIdx.x; i < P / 2; i += NT) {
        const int lo = 2 * i - (i & (j - 1));   // element with bit j clear; its partner is lo + j
        const uint64_t a = w[lo], bb = w[lo + j];
        if ((a > bb) == ((lo & k) == 0)) {
          w[lo] = bb;
          w[lo + j] = a;
        }
      }
      __syncthreads();
    }
  }
  for (int i = threadIdx.x; i < N; i += NT) {
    const int32_t c = (int32_t)(uint32_t)w[i];
    const float v = row[c];
    items[r * ld_items + i] = __float_as_uint(v) == 0xFF800000u ? -1 : c;
    out_scores[r * ld_out + i] = v;
  }
}

constexpr int CUT_NT = 128;
constexpr int CUT_MAX = 1024;
constexpr int CUT_PER = CUT_MAX / CUT_NT;   // cutoffs per thread

struct Cutoffs {
  int32_t c[CUT_MAX];
};

// One CTA per row.  The first c_m ranked items go to shared memory; the user's test items are taken CUT_NT at a time in
// stored order, each thread finds one of them there (its position, or none), and every thread then walks those positions
// in stored order for its own cutoffs: per cutoff the same float64 additions in the same order as calcRes.
__global__ void __launch_bounds__(CUT_NT) eval_metrics_cutoffs_kernel(
    const int32_t* __restrict__ ranked, int64_t ld_ranked, const __grid_constant__ Cutoffs cut, int m,
    const int64_t* __restrict__ row_ids, const int64_t* __restrict__ test_ptr, const int32_t* __restrict__ test_items,
    const double* __restrict__ inv_log2, const double* __restrict__ max_dcg, double* __restrict__ out) {
  __shared__ int32_t s_items[CUT_MAX];
  __shared__ int s_pos[CUT_NT];
  const int64_t r = blockIdx.x;
  const int tid = threadIdx.x;
  const int L = cut.c[m - 1];
  for (int i = tid; i < L; i += CUT_NT) s_items[i] = ranked[r * ld_ranked + i];
  int c[CUT_PER];
  double dcg[CUT_PER];
  int64_t hits[CUT_PER];
#pragma unroll
  for (int j = 0; j < CUT_PER; ++j) {
    c[j] = j * CUT_NT + tid < m ? cut.c[j * CUT_NT + tid] : 0;
    dcg[j] = 0.0;
    hits[j] = 0;
  }
  const int64_t u = row_ids[r];
  const int64_t b = test_ptr[u], e = test_ptr[u + 1];
  __syncthreads();
  for (int64_t k0 = b; k0 < e; k0 += CUT_NT) {
    int p = L;
    if (k0 + tid < e) {
      const int32_t item = test_items[k0 + tid];
      for (int q = 0; q < L; ++q)
        if (s_items[q] == item) {   // list.index: the first occurrence
          p = q;
          break;
        }
    }
    s_pos[tid] = p;
    __syncthreads();
    const int nb = e - k0 < CUT_NT ? (int)(e - k0) : CUT_NT;
    for (int t = 0; t < nb; ++t) {
      const int pos = s_pos[t];
      if (pos >= L) continue;
      const double g = inv_log2[pos];
#pragma unroll
      for (int j = 0; j < CUT_PER; ++j)
        if (pos < c[j]) {
          dcg[j] += g;
          ++hits[j];
        }
    }
    __syncthreads();
  }
  const int64_t tst = e - b;
#pragma unroll
  for (int j = 0; j < CUT_PER; ++j) {
    const int idx = j * CUT_NT + tid;
    if (idx >= m) break;
    const double h = (double)hits[j];
    double* o = out + 3 * (r * m + idx);
    o[0] = tst > 0 ? h / (double)tst : 0.0;
    o[1] = tst > 0 ? dcg[j] / max_dcg[tst < c[j] ? tst : c[j]] : 0.0;
    o[2] = h / (double)c[j];
  }
}

__global__ void __launch_bounds__(256) eval_metrics_kernel(const float* __restrict__ scores, int64_t ld, int64_t n_rows,
                                                           const int32_t* __restrict__ top_items, int K,
                                                           const int64_t* __restrict__ row_ids,
                                                           const int64_t* __restrict__ test_ptr,
                                                           const int32_t* __restrict__ test_items,
                                                           const double* __restrict__ inv_log2,
                                                           const double* __restrict__ max_dcg,
                                                           double* __restrict__ out) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  // lane j < K holds the j-th selected column (ascending) and its score; rank = position in (score desc, column asc)
  const int col = lane < K ? top_items[r * K + lane] : 0x7FFFFFFF;
  const float s = lane < K ? scores[r * ld + col] : 0.f;
  int rank = 0;
  for (int j = 0; j < K; ++j) {
    const float sj = __shfl_sync(0xffffffffu, s, j);
    const int cj = __shfl_sync(0xffffffffu, col, j);
    rank += (sj > s || (sj == s && cj < col)) ? 1 : 0;
  }
  const int64_t u = row_ids[r];
  const int64_t b = test_ptr[u], e = test_ptr[u + 1];
  const int64_t tst = e - b;
  double dcg = 0.0;
  int64_t hits = 0;
  for (int64_t k = b; k < e; ++k) {           // the user's test items in their stored order (calcRes' loop order)
    const int32_t item = test_items[k];
    const uint32_t m = __ballot_sync(0xffffffffu, lane < K && col == item);
    if (m) {
      const int pos = __shfl_sync(0xffffffffu, rank, __ffs(m) - 1);
      dcg += inv_log2[pos];
      ++hits;
    }
  }
  if (lane == 0) {
    const double h = (double)hits;
    out[3 * r + 0] = tst > 0 ? h / (double)tst : 0.0;
    out[3 * r + 1] = tst > 0 ? dcg / max_dcg[tst < K ? tst : K] : 0.0;
    out[3 * r + 2] = h / (double)K;
  }
}

}  // namespace

extern "C" int dmm_eval_mask_scores(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                                    int64_t n_rows, int64_t n_cols, float* scores, int64_t ld, float fill, void* stream) {
  DMM_CHECK_ARG(ctx && indptr && indices && row_ids && scores, "dmm_eval_mask_scores: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_cols > 0 && ld >= n_cols, "dmm_eval_mask_scores: bad shape");
  if (n_rows == 0) return DMM_OK;
  eval_mask_kernel<false><<<(unsigned)dmm_ceil_div(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      indptr, indices, row_ids, n_rows, n_cols, scores, ld, fill, nullptr, 0);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_eval_mask_scores_cmax(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                                         int64_t n_rows, int64_t n_cols, float* scores, int64_t ld, float fill, float* cmax,
                                         int64_t ld_cmax, void* stream) {
  DMM_CHECK_ARG(ctx, "dmm_eval_mask_scores_cmax: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_cols > 0 && ld >= n_cols, "dmm_eval_mask_scores_cmax: bad shape");
  DMM_CHECK_ARG(ld_cmax >= dmm_ceil_div(n_cols, 32), "dmm_eval_mask_scores_cmax: ld_cmax must be >= ceil(n_cols / 32)");
  if (n_rows == 0) return DMM_OK;   // before the pointer checks: empty tensors may have no storage
  DMM_CHECK_ARG(indptr && indices && row_ids && scores && cmax, "dmm_eval_mask_scores_cmax: null argument");
  eval_mask_kernel<true><<<(unsigned)dmm_ceil_div(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      indptr, indices, row_ids, n_rows, n_cols, scores, ld, fill, cmax, ld_cmax);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_topn_rank(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, const int32_t* sel, int64_t ld_sel,
                             int64_t N, int32_t* items, int64_t ld_items, float* out_scores, int64_t ld_out, void* stream) {
  DMM_CHECK_ARG(ctx, "dmm_topn_rank: null argument");
  DMM_CHECK_ARG(N >= 1 && N <= 1024, "dmm_topn_rank: N must be 1..1024 (got %lld)", (long long)N);
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31) && ld_sel >= N && ld_items >= N && ld_out >= N && ld >= 1,
                "dmm_topn_rank: bad shape");
  if (n_rows == 0) return DMM_OK;
  DMM_CHECK_ARG(scores && sel && items && out_scores, "dmm_topn_rank: null argument");
  cudaStream_t st = (cudaStream_t)stream;
  const unsigned g = (unsigned)n_rows;
  const int n = (int)N;
#define DMM_RANK_LAUNCH(P) \
  topn_rank_kernel<P><<<g, (P / 2 < 32 ? 32 : P / 2), 0, st>>>(scores, ld, sel, ld_sel, n, items, ld_items, out_scores, ld_out)
  if (n <= 32) DMM_RANK_LAUNCH(32);
  else if (n <= 64) DMM_RANK_LAUNCH(64);
  else if (n <= 128) DMM_RANK_LAUNCH(128);
  else if (n <= 256) DMM_RANK_LAUNCH(256);
  else if (n <= 512) DMM_RANK_LAUNCH(512);
  else DMM_RANK_LAUNCH(1024);
#undef DMM_RANK_LAUNCH
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_eval_metrics_cutoffs(dmm_ctx* ctx, const int32_t* ranked, int64_t ld_ranked, int64_t n_rows, int64_t N,
                                        const int32_t* cutoffs, int64_t n_cutoffs, const int64_t* row_ids,
                                        const int64_t* test_ptr, const int32_t* test_items, const double* inv_log2,
                                        const double* max_dcg, double* out, void* stream) {
  DMM_CHECK_ARG(ctx && cutoffs, "dmm_eval_metrics_cutoffs: null argument");
  DMM_CHECK_ARG(N >= 1 && N <= CUT_MAX, "dmm_eval_metrics_cutoffs: N must be 1..%d (got %lld)", CUT_MAX, (long long)N);
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31) && ld_ranked >= N, "dmm_eval_metrics_cutoffs: bad shape");
  DMM_CHECK_ARG(n_cutoffs >= 1 && n_cutoffs <= N, "dmm_eval_metrics_cutoffs: need 1..N cutoffs (got %lld)",
                (long long)n_cutoffs);
  Cutoffs cut;
  for (int64_t j = 0; j < n_cutoffs; ++j) {
    DMM_CHECK_ARG(cutoffs[j] >= 1 && cutoffs[j] <= N && (j == 0 || cutoffs[j] > cutoffs[j - 1]),
                  "dmm_eval_metrics_cutoffs: cutoffs must be strictly increasing in 1..N (N = %lld)", (long long)N);
    cut.c[j] = cutoffs[j];
  }
  if (n_rows == 0) return DMM_OK;
  DMM_CHECK_ARG(ranked && row_ids && test_ptr && test_items && inv_log2 && max_dcg && out,
                "dmm_eval_metrics_cutoffs: null argument");
  eval_metrics_cutoffs_kernel<<<(unsigned)n_rows, CUT_NT, 0, (cudaStream_t)stream>>>(
      ranked, ld_ranked, cut, (int)n_cutoffs, row_ids, test_ptr, test_items, inv_log2, max_dcg, out);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_eval_metrics(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, const int32_t* top_items,
                                int64_t K, const int64_t* row_ids, const int64_t* test_ptr, const int32_t* test_items,
                                const double* inv_log2, const double* max_dcg, double* out, void* stream) {
  DMM_CHECK_ARG(ctx && scores && top_items && row_ids && test_ptr && test_items && inv_log2 && max_dcg && out,
                "dmm_eval_metrics: null argument");
  DMM_CHECK_ARG(K >= 1 && K <= 32, "dmm_eval_metrics: top-K must be 1..32 (got %lld)", (long long)K);
  DMM_CHECK_ARG(n_rows >= 0, "dmm_eval_metrics: bad n_rows");
  if (n_rows == 0) return DMM_OK;
  eval_metrics_kernel<<<(unsigned)dmm_ceil_div(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      scores, ld, n_rows, top_items, (int)K, row_ids, test_ptr, test_items, inv_log2, max_dcg, out);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
