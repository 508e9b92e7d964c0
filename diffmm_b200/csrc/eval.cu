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
//
// Scores of given pairs and rankings of given candidate lists (user . item of Main.py:410 without the full contraction):
//   dmm_score_pairs             score(user[u_idx[p]], item[i_idx[p]]) for every pair p
//   dmm_rank_candidates         row r's candidates scored, deduplicated and ranked in one CTA, the first N emitted
// Both compute the score with pair_score: the same split-bf16 terms as the tensor-pipe contraction (bf16x3 or bf16),
// added by fp32 FMAs in a fixed lane layout.  A pair gets the same bits from either kernel, but not dmm_topn_rank's
// (contraction) bits: the summation order differs.
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

// Rank word of (score, item): ascending words are score descending, then item ascending, in order_key's total order.
// All ones (the pad word) sorts after every real word, since an item id is below 2^31.
__device__ __forceinline__ uint64_t rank_word(float s, uint32_t item) {
  return ((uint64_t)~order_key(s) << 32) | item;
}

// Inverse of rank_word's score half.  order_key maps -0.0 onto +0.0; pair_score never returns -0.0 (see there), so
// the scores of dmm_rank_candidates come back bit for bit.
__device__ __forceinline__ float rank_word_score(uint64_t w) {
  const uint32_t k = ~(uint32_t)(w >> 32);
  return __uint_as_float((k & 0x80000000u) ? (k & 0x7FFFFFFFu) : ~k);
}

// Sorts the P words of w ascending with a bitonic network, NT threads of the CTA taking part; P a power of two.
// Starts and ends with the CTA synchronised.
template <int P, int NT>
__device__ __forceinline__ void bitonic_sort_smem(uint64_t* w) {
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
      v = rank_word(row[c], c);
    }
    w[i] = v;
  }
  bitonic_sort_smem<P, NT>(w);
  for (int i = threadIdx.x; i < N; i += NT) {
    const int32_t c = (int32_t)(uint32_t)w[i];
    const float v = row[c];
    items[r * ld_items + i] = __float_as_uint(v) == 0xFF800000u ? -1 : c;
    out_scores[r * ld_out + i] = v;
  }
}

// ---- scores of given (user, item) pairs --------------------------------------------------------------------------
constexpr int PAIR_LANES = 8;   // lanes per (user, item) pair

// One d of the score: both values split in registers (hi = bf16_rn(x), lo = bf16_rn(x - hi), the operands of
// dmm_pack_bf16), then hi_u hi_i, hi_u lo_i, lo_u hi_i (X3) or hi_u hi_i alone, added in that order by fp32 FMAs
// (each bf16 product is exact in fp32).
template <bool X3>
__device__ __forceinline__ float score_term(float acc, float x, float y) {
  uint16_t xh, xl, yh, yl;
  dmm_split_bf16(x, xh, xl);
  dmm_split_bf16(y, yh, yl);
  const float hx = dmm_bf16_to_f32(xh), hy = dmm_bf16_to_f32(yh);
  acc = fmaf(hx, hy, acc);
  if (X3) {
    acc = fmaf(hx, dmm_bf16_to_f32(yl), acc);
    acc = fmaf(dmm_bf16_to_f32(xl), hy, acc);
  }
  return acc;
}

template <bool X3>
__device__ __forceinline__ float score_quad(float acc, float4 a, float4 b) {
  acc = score_term<X3>(acc, a.x, b.x);
  acc = score_term<X3>(acc, a.y, b.y);
  acc = score_term<X3>(acc, a.z, b.z);
  return score_term<X3>(acc, a.w, b.w);
}

template <bool VEC>
__device__ __forceinline__ float4 load_quad(const float* __restrict__ p) {
  if (VEC) return __ldg(reinterpret_cast<const float4*>(p));
  return make_float4(__ldg(p), __ldg(p + 1), __ldg(p + 2), __ldg(p + 3));
}

// score(u, v) of one pair on a group of PAIR_LANES aligned lanes; lane = the lane's index in its group.  Quad q (the
// elements 4q .. 4q + 3, the last one possibly partial) belongs to lane q % PAIR_LANES; each lane adds its quads in
// ascending q, elements ascending, into one fp32 sum from +0.0, and the lane sums are added by an xor butterfly (4, 2,
// 1), so every lane returns the same value.  VEC (16-byte aligned rows) only changes how the quads are loaded, not the
// order of the additions: a pair gets the same bits from every caller.  The result is returned as sum + (+0.0), so a
// zero score is always +0.0 (an underflowing product can make the sum -0.0), which rank_word_score relies on.
// Every lane of the warp must call it (full-warp shuffles); a lane with active = false reads nothing.
template <bool X3, bool VEC>
__device__ __forceinline__ float pair_score(const float* __restrict__ u, const float* __restrict__ v, int D, int lane,
                                            bool active) {
  float acc = 0.f;
  if (active) {
    const int Q = D >> 2;
    int q = lane;
    for (; q + PAIR_LANES < Q; q += 2 * PAIR_LANES) {   // two quads per step: four loads in flight per lane
      const float4 a0 = load_quad<VEC>(u + 4 * q), b0 = load_quad<VEC>(v + 4 * q);
      const float4 a1 = load_quad<VEC>(u + 4 * (q + PAIR_LANES)), b1 = load_quad<VEC>(v + 4 * (q + PAIR_LANES));
      acc = score_quad<X3>(acc, a0, b0);
      acc = score_quad<X3>(acc, a1, b1);
    }
    if (q < Q) acc = score_quad<X3>(acc, load_quad<VEC>(u + 4 * q), load_quad<VEC>(v + 4 * q));
    if (lane == Q % PAIR_LANES)
      for (int d = 4 * Q; d < D; ++d) acc = score_term<X3>(acc, __ldg(u + d), __ldg(v + d));
  }
#pragma unroll
  for (int o = PAIR_LANES / 2; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o, PAIR_LANES);
  return __fadd_rn(acc, 0.f);
}

// PAIR_LANES lanes per pair, grid-stride over the pairs (the loop bound is uniform across each warp).
template <bool X3, bool VEC>
__global__ void __launch_bounds__(256) score_pairs_kernel(const float* __restrict__ user, int64_t ld_u, int64_t n_users,
                                                          const float* __restrict__ item, int64_t ld_i, int64_t n_items,
                                                          int D, const int64_t* __restrict__ u_idx,
                                                          const int32_t* __restrict__ i_idx, int64_t P,
                                                          float* __restrict__ out) {
  constexpr int PER_WARP = 32 / PAIR_LANES;
  const int lane = threadIdx.x & (PAIR_LANES - 1);
  const int sub = (threadIdx.x & 31) / PAIR_LANES;
  const int64_t warp = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int64_t stride = (((int64_t)gridDim.x * blockDim.x) >> 5) * PER_WARP;
  for (int64_t p0 = warp * PER_WARP; p0 < P; p0 += stride) {
    const int64_t p = p0 + sub;
    int64_t u = -1, i = -1;
    if (p < P) {
      u = u_idx[p];
      i = i_idx[p];
    }
    const bool ok = p < P && u >= 0 && u < n_users && i >= 0 && i < n_items;
    const float s = pair_score<X3, VEC>(user + (ok ? u * ld_u : 0), item + (ok ? i * ld_i : 0), D, lane, ok);
    if (p < P && lane == 0) out[p] = ok ? s : __uint_as_float(0x7FC00000u);
  }
}

// ---- ranking of caller-supplied candidates --------------------------------------------------------------------------
__host__ __device__ constexpr int rank_cand_threads(int P) { return P / 2 < 64 ? 64 : (P / 2 > 512 ? 512 : P / 2); }

// One CTA per row, P = the power of two >= C.  Groups of PAIR_LANES lanes score the row's candidates (each item row read
// once, the scores kept in shared memory as rank words; an empty slot, -1 or an id outside [0, n_items), is the pad
// word), bitonic_sort_smem ranks them, and the distinct words are compacted: equal (row, item) pairs have equal words,
// adjacent after the sort, and only the first of a run is kept.  The first N go out; slots past the row's distinct valid
// candidates get (-1, -inf).
template <int P, bool X3, bool VEC>
__global__ void __launch_bounds__(rank_cand_threads(P)) rank_candidates_kernel(
    const float* __restrict__ user, int64_t ld_u, const float* __restrict__ item, int64_t ld_i, int64_t n_items, int D,
    const int32_t* __restrict__ cand, int64_t ld_c, int C, int N, int32_t* __restrict__ out_items, int64_t ld_oi,
    float* __restrict__ out_scores, int64_t ld_os) {
  constexpr int NT = rank_cand_threads(P);
  constexpr int G = NT / PAIR_LANES;
  constexpr int E = (P + NT - 1) / NT;   // words per thread in the compaction
  constexpr int NW = NT / 32;
  __shared__ uint64_t w[P];
  __shared__ int s_warp[NW];
  const int64_t r = blockIdx.x;
  const int t = threadIdx.x;
  const int lane = t & (PAIR_LANES - 1);
  const int g = t / PAIR_LANES;
  const float* urow = user + r * ld_u;
  const int32_t* crow = cand + r * ld_c;
  for (int c0 = 0; c0 < C; c0 += G) {
    const int c = c0 + g;
    const int32_t it = c < C ? crow[c] : -1;
    const bool ok = it >= 0 && it < n_items;
    const float s = pair_score<X3, VEC>(urow, item + (ok ? (int64_t)it * ld_i : 0), D, lane, ok);
    if (c < C && lane == 0) w[c] = ok ? rank_word(s, (uint32_t)it) : ~0ull;
  }
  for (int i = C + t; i < P; i += NT) w[i] = ~0ull;
  bitonic_sort_smem<P, NT>(w);

  // thread t owns the words [b0, b1); a word is kept if it is real and differs from the word before it
  const int b0 = t * E < P ? t * E : P, b1 = b0 + E < P ? b0 + E : P;
  int cnt = 0;
  uint64_t prev = b0 > 0 ? w[b0 - 1] : ~0ull;
  for (int i = b0; i < b1; ++i) {
    const uint64_t x = w[i];
    cnt += (x != ~0ull && x != prev) ? 1 : 0;
    prev = x;
  }
  int inc = cnt;   // inclusive scan of the counts: in the warp, then over the warp totals
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, inc, o);
    if ((t & 31) >= o) inc += y;
  }
  if ((t & 31) == 31) s_warp[t >> 5] = inc;
  __syncthreads();
  if (t < 32) {
    int v = t < NW ? s_warp[t] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, v, o);
      if (t >= o) v += y;
    }
    if (t < NW) s_warp[t] = v;
  }
  __syncthreads();
  int pos = inc - cnt + ((t >> 5) ? s_warp[(t >> 5) - 1] : 0);
  const int total = s_warp[NW - 1];
  prev = b0 > 0 ? w[b0 - 1] : ~0ull;
  for (int i = b0; i < b1 && pos < N; ++i) {
    const uint64_t x = w[i];
    if (x != ~0ull && x != prev) {
      out_items[r * ld_oi + pos] = (int32_t)(uint32_t)x;
      out_scores[r * ld_os + pos] = rank_word_score(x);
      ++pos;
    }
    prev = x;
  }
  for (int i = total + t; i < N; i += NT) {
    out_items[r * ld_oi + i] = -1;
    out_scores[r * ld_os + i] = __uint_as_float(0xFF800000u);
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

// float4 loads need both row bases and every row start 16-byte aligned
static bool pair_rows_aligned(const float* user, int64_t ld_u, const float* item, int64_t ld_i) {
  return (((uintptr_t)user | (uintptr_t)item) & 15) == 0 && ld_u % 4 == 0 && ld_i % 4 == 0;
}

extern "C" int dmm_score_pairs(dmm_ctx* ctx, const float* user, int64_t ld_u, int64_t n_users, const float* item,
                               int64_t ld_i, int64_t n_items, int64_t D, const int64_t* u_idx, const int32_t* i_idx,
                               int64_t P, int x3, float* out, void* stream) {
  DMM_CHECK_ARG(ctx, "dmm_score_pairs: null argument");
  DMM_CHECK_ARG(D >= 1 && D <= 1024, "dmm_score_pairs: D must be 1..1024 (got %lld)", (long long)D);
  DMM_CHECK_ARG(n_users >= 0 && n_items >= 0 && ld_u >= D && ld_i >= D && P >= 0 && (x3 == 0 || x3 == 1),
                "dmm_score_pairs: bad shape");
  if (P == 0) return DMM_OK;
  DMM_CHECK_ARG(u_idx && i_idx && out && (user || n_users == 0) && (item || n_items == 0),
                "dmm_score_pairs: null argument");
  const int64_t pairs_per_block = 256 / PAIR_LANES;
  const int64_t max_blocks = (int64_t)ctx->num_sms * 32;
  const int64_t need = dmm_ceil_div(P, pairs_per_block);
  const unsigned grid = (unsigned)(need < max_blocks ? need : max_blocks);
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = pair_rows_aligned(user, ld_u, item, ld_i);
#define DMM_PAIRS_LAUNCH(X3, VEC) \
  score_pairs_kernel<X3, VEC><<<grid, 256, 0, st>>>(user, ld_u, n_users, item, ld_i, n_items, (int)D, u_idx, i_idx, P, out)
  if (x3) {
    if (vec) DMM_PAIRS_LAUNCH(true, true);
    else DMM_PAIRS_LAUNCH(true, false);
  } else {
    if (vec) DMM_PAIRS_LAUNCH(false, true);
    else DMM_PAIRS_LAUNCH(false, false);
  }
#undef DMM_PAIRS_LAUNCH
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

template <int P>
static void launch_rank_candidates(bool x3, bool vec, unsigned grid, cudaStream_t st, const float* user, int64_t ld_u,
                                   const float* item, int64_t ld_i, int64_t n_items, int D, const int32_t* cand,
                                   int64_t ld_c, int C, int N, int32_t* out_items, int64_t ld_oi, float* out_scores,
                                   int64_t ld_os) {
  constexpr int NT = rank_cand_threads(P);
#define DMM_RANKC_LAUNCH(X3, VEC)                                                                                  \
  rank_candidates_kernel<P, X3, VEC><<<grid, NT, 0, st>>>(user, ld_u, item, ld_i, n_items, D, cand, ld_c, C, N, \
                                                          out_items, ld_oi, out_scores, ld_os)
  if (x3) {
    if (vec) DMM_RANKC_LAUNCH(true, true);
    else DMM_RANKC_LAUNCH(true, false);
  } else {
    if (vec) DMM_RANKC_LAUNCH(false, true);
    else DMM_RANKC_LAUNCH(false, false);
  }
#undef DMM_RANKC_LAUNCH
}

extern "C" int dmm_rank_candidates(dmm_ctx* ctx, const float* user, int64_t ld_u, const float* item, int64_t ld_i,
                                   int64_t n_items, int64_t D, const int32_t* cand, int64_t ld_c, int64_t n_rows,
                                   int64_t C, int64_t N, int x3, int32_t* out_items, int64_t ld_oi, float* out_scores,
                                   int64_t ld_os, void* stream) {
  DMM_CHECK_ARG(ctx, "dmm_rank_candidates: null argument");
  DMM_CHECK_ARG(C >= 1 && C <= 4096, "dmm_rank_candidates: C must be 1..4096 (got %lld)", (long long)C);
  DMM_CHECK_ARG(N >= 1 && N <= 1024 && N <= C, "dmm_rank_candidates: N must be 1..min(1024, C) (got %lld, C = %lld)",
                (long long)N, (long long)C);
  DMM_CHECK_ARG(D >= 1 && D <= 1024, "dmm_rank_candidates: D must be 1..1024 (got %lld)", (long long)D);
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31) && n_items >= 0 && ld_u >= D && ld_i >= D && ld_c >= C &&
                    ld_oi >= N && ld_os >= N && (x3 == 0 || x3 == 1),
                "dmm_rank_candidates: bad shape");
  if (n_rows == 0) return DMM_OK;
  DMM_CHECK_ARG(user && cand && out_items && out_scores && (item || n_items == 0), "dmm_rank_candidates: null argument");
  const unsigned g = (unsigned)n_rows;
  const bool vec = pair_rows_aligned(user, ld_u, item, ld_i);
  const int c = (int)C;
#define DMM_RANKC(P)                                                                                               \
  launch_rank_candidates<P>(x3 != 0, vec, g, (cudaStream_t)stream, user, ld_u, item, ld_i, n_items, (int)D, cand, \
                            ld_c, c, (int)N, out_items, ld_oi, out_scores, ld_os)
  if (c <= 32) DMM_RANKC(32);
  else if (c <= 64) DMM_RANKC(64);
  else if (c <= 128) DMM_RANKC(128);
  else if (c <= 256) DMM_RANKC(256);
  else if (c <= 512) DMM_RANKC(512);
  else if (c <= 1024) DMM_RANKC(1024);
  else if (c <= 2048) DMM_RANKC(2048);
  else DMM_RANKC(4096);
#undef DMM_RANKC
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
