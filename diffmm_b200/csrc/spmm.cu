// CSR SpMM for the LightGCN-style propagation over the normalised user-item graph.
//
// Replaces torch.sparse.mm on an uncoalesced COO (Model.py:90,93,105,111,114,123,130; Main.py:319),
// which coalesces (sorts) the operand on every call before cuSPARSE runs.  The adjacency is
// symmetric, so the backward pass is the same call on the incoming gradient.
//
// D = 64 with a plan (the product path): see "v3: degree-sorted units" below -- one persistent launch over equal-length
// units + a fixed-order reduce of the chunked long rows (deterministic, no atomics on Y); fp32 gather table with A's
// values, or bf16 gather table with the separable normalisation.  Without a plan: one warp per row, rows longer than
// LONG_ROW finished by their CTA alone.  Generic D: one warp per row.
// Compulsory traffic of one fp32 product: 8*nnz + 8*(N+1) + 2*N*D*4 bytes (SURVEY 8d).
#include "common.cuh"

#include <stdlib.h>

namespace {

constexpr int SPMM_THREADS = 256;
constexpr int SPMM_WARPS = SPMM_THREADS / 32;
constexpr int LONG_ROW = 1024;
constexpr int PLAN_LONG_ROW = 64;    // rows with more neighbours go through the plan
constexpr int PLAN_CHUNK = 64;       // neighbours per chunk of a planned row (one warp each)
constexpr int REDUCE_SMALL = 16;     // planned rows with more chunks are reduced by a whole CTA (listed in the plan)
constexpr int V3_HDR_WORDS = 128;    // int32 header of the v3 plan sections; [200] = number of listed big rows

// plan buffer (int64 words): [0] n_long, [1] n_chunks, [2, 2+cap) long row ids, [2+cap, 3+2cap) chunk_ptr,
// then (16-byte aligned) one descriptor per chunk, int4 {row, neighbours, first entry lo, first entry hi}
__host__ __device__ inline int64_t plan_cap(int64_t nnz) { return nnz / PLAN_LONG_ROW + 1; }
__host__ __device__ inline int64_t plan_max_chunks(int64_t nnz) { return nnz / PLAN_CHUNK + plan_cap(nnz) + 1; }

// v3 plan sections behind the chunk descriptors (int64 words): header, int32 big_row[cap] (positions in the long-row list of
// the rows with more than REDUCE_SMALL chunks), int2 unit[max_chunks + n_rows], float dinv[n_rows]
__host__ __device__ inline int64_t plan_desc_word(int64_t cap) { return (3 + 2 * cap + 1) & ~(int64_t)1; }
__host__ __device__ inline int64_t plan_v3_word(int64_t nnz) { return plan_desc_word(plan_cap(nnz)) + 2 * plan_max_chunks(nnz); }
__host__ __device__ inline int64_t plan_v3_unit_word(int64_t nnz) { return plan_v3_word(nnz) + V3_HDR_WORDS + (plan_cap(nnz) + 1) / 2; }
__host__ __device__ inline int64_t plan_v3_dinv_word(int64_t nnz, int64_t n_rows) {
  return plan_v3_unit_word(nnz) + plan_max_chunks(nnz) + n_rows;
}

struct Epi {
  float alpha, beta;
  const float* z;
  int64_t ld_z;
  const float* rscale;   // optional per-row factor applied with alpha (d_r^-1/2 of the separable normalisation), or null
};

// ---- D == 64 fast path --------------------------------------------------------------------
__device__ __forceinline__ float4 fma4(float a, const float4& x, const float4& acc) {
  return make_float4(fmaf(a, x.x, acc.x), fmaf(a, x.y, acc.y), fmaf(a, x.z, acc.z), fmaf(a, x.w, acc.w));
}
__device__ __forceinline__ float4 add4(const float4& a, const float4& b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

// accumulates A[r, beg:end) . X over neighbours j = beg + h, beg + h + stride, ... for this half warp
__device__ __forceinline__ float4 gather64(const int32_t* __restrict__ idx, const float* __restrict__ val,
                                           const float* __restrict__ x, int64_t ld_x, int64_t beg, int64_t end,
                                           int stride, int l16) {
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  int64_t j = beg;
  for (; j + 3 * stride < end; j += 4 * stride) {
    const int32_t c0 = __ldg(idx + j), c1 = __ldg(idx + j + stride), c2 = __ldg(idx + j + 2 * stride),
                  c3 = __ldg(idx + j + 3 * stride);
    const float v0 = __ldg(val + j), v1 = __ldg(val + j + stride), v2 = __ldg(val + j + 2 * stride),
                v3 = __ldg(val + j + 3 * stride);
    const float4 x0 = __ldg(reinterpret_cast<const float4*>(x + (int64_t)c0 * ld_x) + l16);
    const float4 x1 = __ldg(reinterpret_cast<const float4*>(x + (int64_t)c1 * ld_x) + l16);
    const float4 x2 = __ldg(reinterpret_cast<const float4*>(x + (int64_t)c2 * ld_x) + l16);
    const float4 x3 = __ldg(reinterpret_cast<const float4*>(x + (int64_t)c3 * ld_x) + l16);
    acc = fma4(v0, x0, acc);
    acc = fma4(v1, x1, acc);
    acc = fma4(v2, x2, acc);
    acc = fma4(v3, x3, acc);
  }
  for (; j < end; j += stride) {
    const int32_t c = __ldg(idx + j);
    const float v = __ldg(val + j);
    acc = fma4(v, __ldg(reinterpret_cast<const float4*>(x + (int64_t)c * ld_x) + l16), acc);
  }
  return acc;
}

__global__ void __launch_bounds__(SPMM_THREADS) spmm64_kernel(const int64_t* __restrict__ ptr,
                                                              const int32_t* __restrict__ idx,
                                                              const float* __restrict__ val, int64_t row0, int64_t row1,
                                                              const float* __restrict__ x, int64_t ld_x, Epi ep,
                                                              float* __restrict__ y, int64_t ld_y, int planned) {
  __shared__ int64_t long_rows[SPMM_WARPS];
  __shared__ int n_long;
  __shared__ float4 part[SPMM_WARPS * 2][16];
  if (threadIdx.x == 0) n_long = 0;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int half = lane >> 4, l16 = lane & 15;
  const int64_t r = row0 + (int64_t)blockIdx.x * SPMM_WARPS + warp;
  if (r < row1) {
    const int64_t b = ptr[r], e = ptr[r + 1];
    if (planned && e - b > PLAN_LONG_ROW) {
      // handled by the chunk kernels
    } else if (e - b > LONG_ROW) {
      if (lane == 0) long_rows[atomicAdd(&n_long, 1)] = r;
    } else {
      float4 acc = gather64(idx, val, x, ld_x, b + half, e, 2, l16);
      acc.x += __shfl_xor_sync(0xffffffffu, acc.x, 16);
      acc.y += __shfl_xor_sync(0xffffffffu, acc.y, 16);
      acc.z += __shfl_xor_sync(0xffffffffu, acc.z, 16);
      acc.w += __shfl_xor_sync(0xffffffffu, acc.w, 16);
      if (half == 0) {
        float4 o = make_float4(ep.alpha * acc.x, ep.alpha * acc.y, ep.alpha * acc.z, ep.alpha * acc.w);
        if (ep.z) {
          const float4 zz = __ldg(reinterpret_cast<const float4*>(ep.z + r * ep.ld_z) + l16);
          o = make_float4(fmaf(ep.beta, zz.x, o.x), fmaf(ep.beta, zz.y, o.y), fmaf(ep.beta, zz.z, o.z),
                          fmaf(ep.beta, zz.w, o.w));
        }
        reinterpret_cast<float4*>(y + r * ld_y)[l16] = o;
      }
    }
  }
  __syncthreads();
  const int nl = n_long;
  // long rows: all 16 half warps stride the neighbour list; fixed-order reduction
  for (int q = 0; q < nl; ++q) {
    // sort order of long_rows is irrelevant for determinism: each row's result is independent
    const int64_t rr = long_rows[q];
    const int64_t b = ptr[rr], e = ptr[rr + 1];
    const int hw = warp * 2 + half;
    part[hw][l16] = gather64(idx, val, x, ld_x, b + hw, e, SPMM_WARPS * 2, l16);
    __syncthreads();
    if (threadIdx.x < 16) {
      float4 acc = part[0][threadIdx.x];
      for (int k = 1; k < SPMM_WARPS * 2; ++k) acc = add4(acc, part[k][threadIdx.x]);
      float4 o = make_float4(ep.alpha * acc.x, ep.alpha * acc.y, ep.alpha * acc.z, ep.alpha * acc.w);
      if (ep.z) {
        const float4 zz = __ldg(reinterpret_cast<const float4*>(ep.z + rr * ep.ld_z) + threadIdx.x);
        o = make_float4(fmaf(ep.beta, zz.x, o.x), fmaf(ep.beta, zz.y, o.y), fmaf(ep.beta, zz.z, o.z),
                        fmaf(ep.beta, zz.w, o.w));
      }
      reinterpret_cast<float4*>(y + rr * ld_y)[threadIdx.x] = o;
    }
    __syncthreads();
  }
}

// ---- planned long rows ---------------------------------------------------------------------------
__global__ void __launch_bounds__(256) plan_collect_kernel(const int64_t* __restrict__ ptr, int64_t n_rows,
                                                           int64_t cap, int64_t* __restrict__ plan) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  if (ptr[r + 1] - ptr[r] > PLAN_LONG_ROW) {
    const unsigned long long i = atomicAdd(reinterpret_cast<unsigned long long*>(plan), 1ULL);
    if ((int64_t)i < cap) plan[2 + i] = r;
  }
}

// single block: chunk_ptr = exclusive scan of ceil(nnz_r / PLAN_CHUNK) over the listed rows
__global__ void __launch_bounds__(1024) plan_scan_kernel(const int64_t* __restrict__ ptr, int64_t cap,
                                                         int64_t* __restrict__ plan, int32_t* __restrict__ h,
                                                         int32_t* __restrict__ big_row) {
  __shared__ int64_t warp_sums[32];
  __shared__ int64_t carry;
  const int64_t n = plan[0] < cap ? plan[0] : cap;
  int64_t* chunk_ptr = plan + 2 + cap;
  if (threadIdx.x == 0) carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  for (int64_t base = 0; base < n; base += 1024) {
    const int64_t i = base + threadIdx.x;
    int64_t v = 0;
    if (i < n) {
      const int64_t r = plan[2 + i];
      v = (ptr[r + 1] - ptr[r] + PLAN_CHUNK - 1) / PLAN_CHUNK;
      if (v > REDUCE_SMALL) big_row[atomicAdd(&h[200], 1)] = (int32_t)i;      // any order: every row is reduced on its own
    }
    int64_t incl = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int64_t t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) warp_sums[w] = incl;
    __syncthreads();
    int64_t wbase = 0;
    for (int k = 0; k < w; ++k) wbase += warp_sums[k];
    const int64_t c = carry;
    if (i < n) chunk_ptr[i] = c + wbase + incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) carry = c + wbase + incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) {
    chunk_ptr[n] = carry;
    plan[1] = carry;
  }
}


// descriptor of every chunk c of planned row i: {row, neighbours in the chunk, first entry} (one warp per planned row)
__global__ void __launch_bounds__(256) plan_desc_kernel(const int64_t* __restrict__ ptr, int64_t cap, int64_t* __restrict__ plan,
                                                        int2* __restrict__ unit) {
  const int64_t n = plan[0] < cap ? plan[0] : cap;
  const int64_t* long_rows = plan + 2;
  const int64_t* chunk_ptr = plan + 2 + cap;
  int4* desc = reinterpret_cast<int4*>(plan + plan_desc_word(cap));
  const int lane = threadIdx.x & 31;
  for (int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5; i < n; i += ((int64_t)gridDim.x * blockDim.x) >> 5) {
    const int64_t r = long_rows[i];
    const int64_t rb = ptr[r], re = ptr[r + 1];
    const int64_t c0 = chunk_ptr[i], c1 = chunk_ptr[i + 1];
    for (int64_t c = c0 + lane; c < c1; c += 32) {
      const int64_t b = rb + (c - c0) * PLAN_CHUNK;
      const int nn = (int)(re - b < PLAN_CHUNK ? re - b : PLAN_CHUNK);
      desc[c] = make_int4((int)r, nn, (int)(uint32_t)(b & 0xFFFFFFFFll), (int)(b >> 32));
      unit[c] = make_int2((int)((uint32_t)r | ((uint32_t)nn << 25)), (int)(uint32_t)b);      // the same chunk as a v3 unit
    }
  }
}

// Y[row] = epilogue(sum of the row's partials), deterministic.  Pass A: rows with at most REDUCE_SMALL chunks,
// one half warp per row, all loads in flight.  Pass B: the few big rows, one CTA per row: the 16 half warps
// stride the partials (4 loads in flight each) and one half warp adds the 16 sums in a fixed order.
constexpr int REDUCE_THREADS = 1024;     // pass B: 64 half warps x 8 partial rows in flight per big row (the 1600-chunk row is 4 round trips)
__global__ void __launch_bounds__(REDUCE_THREADS) spmm64_reduce_kernel(int64_t row0, int64_t row1,
                                                                     const int64_t* __restrict__ plan, int64_t cap,
                                                                     const float* __restrict__ partial, Epi ep,
                                                                     float* __restrict__ y, int64_t ld_y,
                                                                     const int32_t* __restrict__ v3_hdr) {
  __shared__ float4 part[REDUCE_THREADS / 16][16];
  const int32_t* big_row = v3_hdr + 2 * V3_HDR_WORDS;
  const int l16 = threadIdx.x & 15, hw = threadIdx.x >> 4;
  constexpr int NHW = REDUCE_THREADS / 16;
  const int64_t n_long = plan[0] < cap ? plan[0] : cap;
  const int64_t* long_rows = plan + 2;
  const int64_t* chunk_ptr = plan + 2 + cap;
  auto finish = [&](int64_t r, const float4& sum) {
    const float a = ep.rscale ? ep.alpha * __ldg(ep.rscale + r) : ep.alpha;
    float4 o = make_float4(a * sum.x, a * sum.y, a * sum.z, a * sum.w);
    if (ep.z) {
      const float4 zz = __ldg(reinterpret_cast<const float4*>(ep.z + r * ep.ld_z) + l16);
      o = make_float4(fmaf(ep.beta, zz.x, o.x), fmaf(ep.beta, zz.y, o.y), fmaf(ep.beta, zz.z, o.z), fmaf(ep.beta, zz.w, o.w));
    }
    reinterpret_cast<float4*>(y + r * ld_y)[l16] = o;
  };
  // pass A
  for (int64_t i = (int64_t)blockIdx.x * NHW + hw; i < n_long; i += (int64_t)gridDim.x * NHW) {
    const int64_t r = long_rows[i];
    const int64_t cb = chunk_ptr[i];
    const int nc = (int)(chunk_ptr[i + 1] - cb);
    if (nc > REDUCE_SMALL || r < row0 || r >= row1) continue;
    float4 p[REDUCE_SMALL];
#pragma unroll
    for (int t = 0; t < REDUCE_SMALL; ++t) {
      p[t] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (t < nc) p[t] = __ldg(reinterpret_cast<const float4*>(partial + (cb + t) * 64) + l16);
    }
    float4 sum = p[0];
#pragma unroll
    for (int t = 1; t < REDUCE_SMALL; ++t) sum = add4(sum, p[t]);
    finish(r, sum);
  }
  // pass B: the rows listed by the plan as big
  const int n_big = v3_hdr[200];
  for (int j = blockIdx.x; j < n_big; j += gridDim.x) {
    const int64_t i = big_row[j];
    const int64_t r = long_rows[i];
    const int64_t cb = chunk_ptr[i], ce = chunk_ptr[i + 1];
    if (r < row0 || r >= row1) continue;     // block-uniform
    float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
    int64_t c = cb + hw;
    for (; c + 7 * NHW < ce; c += 8 * NHW) {      // 8 partial rows in flight per half warp (the longest row sets the tail)
      float4 p[8];
#pragma unroll
      for (int t = 0; t < 8; ++t) p[t] = __ldg(reinterpret_cast<const float4*>(partial + (c + t * NHW) * 64) + l16);
#pragma unroll
      for (int t = 0; t < 8; ++t) acc = add4(acc, p[t]);
    }
    for (; c < ce; c += NHW) acc = add4(acc, __ldg(reinterpret_cast<const float4*>(partial + c * 64) + l16));
    part[hw][l16] = acc;
    __syncthreads();
    if (hw == 0) {
      float4 sum = part[0][l16];
#pragma unroll
      for (int k = 1; k < NHW; ++k) sum = add4(sum, part[k][l16]);
      finish(r, sum);
    }
    __syncthreads();
  }
}

// streaming store of one finished row (fp32 path: 16 lanes x float4)
__device__ __forceinline__ void store_row_cs(float* __restrict__ y, int64_t ld_y, int64_t r, int l16, const float4& acc,
                                             const Epi& ep) {
  float4 o = make_float4(ep.alpha * acc.x, ep.alpha * acc.y, ep.alpha * acc.z, ep.alpha * acc.w);
  if (ep.z) {
    const float4 zz = __ldg(reinterpret_cast<const float4*>(ep.z + r * ep.ld_z) + l16);
    o = make_float4(fmaf(ep.beta, zz.x, o.x), fmaf(ep.beta, zz.y, o.y), fmaf(ep.beta, zz.z, o.z), fmaf(ep.beta, zz.w, o.w));
  }
  __stcs(reinterpret_cast<float4*>(y + r * ld_y) + l16, o);
}

// ---- D == 64, v3: degree-sorted units ------------------------------------------------------------------------------
// What bounded the lean kernels (profiles/r02_prof_spmm_v2.txt): 13 warp instructions per stored entry at IPC 1.4 -- the
// two half warps of a warp walk rows of DIFFERENT lengths (every loop trip is paid by both), each row pays its own
// pointer / index / store set-up for ~8 entries, and only 4 gathers per half warp are in flight.  v3 removes all three:
//   * the plan lists every row of at most 64 entries as a UNIT {row, length, first entry} sorted by length (longest
//     first: counting sort over 65 bins), so the groups of a warp run the same trip counts, and the chunks of the long
//     rows (all 64 entries) are units of the same kind: ONE persistent launch + the fixed-order reduce;
//   * a unit is one 8-byte descriptor away from its indices (no row-pointer round trip) and 8 gathers per group are in
//     flight;
//   * bf16 table mode (dmm_spmm_norm_bf16): the adjacency values are separable, val = d_r^-1/2 d_c^-1/2 (SURVEY App. D.7),
//     so the table is T = bf16(d^-1/2 X) (one streaming pass, dmm_spmm_table_bf16), a row of T is 128 B = 8 lanes x
//     16 B, an entry costs one LDG.128 + 8 FHADD.BF16 (sm_100's mixed-precision add: fp32 accumulator += bf16 half
//     register, no unpack) per 8 lanes and no value stream, and Y = alpha d_r^-1/2 sum (+ beta Z) in the epilogue.
// plan sections behind the chunk descriptors (int64 words): 128 words of int32 header {[0] n_short, [1 + b] running
// cursor and [80 + b] start of bin b = 64 - length}, int2 unit[max_chunks + n_rows] = {row | length << 25, first entry}
// (the chunks of the long rows, then the short rows by falling length), float dinv[n_rows].
constexpr int V3_ROW_BITS = 25;

__global__ void __launch_bounds__(1024) v3_hist_kernel(const int64_t* __restrict__ ptr, int64_t n_rows, int32_t* __restrict__ h,
                                                       float* __restrict__ dinv) {
  __shared__ int sh[65];
  if (threadIdx.x < 65) sh[threadIdx.x] = 0;
  __syncthreads();
  const int64_t r = (int64_t)blockIdx.x * 1024 + threadIdx.x;
  if (r < n_rows) {
    const int64_t len = ptr[r + 1] - ptr[r];
    dinv[r] = len > 0 ? (float)(1.0 / sqrt((double)len)) : 0.f;
    if (len <= PLAN_LONG_ROW) atomicAdd(&sh[PLAN_LONG_ROW - (int)len], 1);
  }
  __syncthreads();
  if (threadIdx.x < 65 && sh[threadIdx.x]) atomicAdd(&h[1 + threadIdx.x], sh[threadIdx.x]);
}

__global__ void v3_scan_kernel(int32_t* __restrict__ h) {
  if (threadIdx.x != 0) return;
  int start = 0;
  for (int b = 0; b < 65; ++b) {
    const int c = h[1 + b];
    h[1 + b] = start;
    h[80 + b] = start;
    start += c;
  }
  h[0] = start;
}

__global__ void __launch_bounds__(1024) v3_scatter_kernel(const int64_t* __restrict__ ptr, int64_t n_rows, int32_t* __restrict__ h,
                                                          int2* __restrict__ unit, const int64_t* __restrict__ n_chunks_ptr,
                                                          int64_t max_chunks) {
  __shared__ int cnt[65], base[65];
  if (threadIdx.x < 65) cnt[threadIdx.x] = 0;
  __syncthreads();
  unit += n_chunks_ptr[0] < max_chunks ? n_chunks_ptr[0] : max_chunks;      // the short rows follow the chunks
  const int64_t r = (int64_t)blockIdx.x * 1024 + threadIdx.x;
  int bin = -1, rank = 0;
  int64_t b = 0;
  if (r < n_rows) {
    b = ptr[r];
    const int64_t len = ptr[r + 1] - b;
    if (len <= PLAN_LONG_ROW) {
      bin = PLAN_LONG_ROW - (int)len;
      rank = atomicAdd(&cnt[bin], 1);
    }
  }
  __syncthreads();
  if (threadIdx.x < 65) base[threadIdx.x] = cnt[threadIdx.x] ? atomicAdd(&h[1 + threadIdx.x], cnt[threadIdx.x]) : 0;
  __syncthreads();
  if (bin >= 0) unit[base[bin] + rank] = make_int2((int)((uint32_t)r | ((uint32_t)(PLAN_LONG_ROW - bin) << V3_ROW_BITS)), (int)(uint32_t)b);
}

// acc[0..8) += the 8 bf16 of q (element 2j in the low half of word j)
__device__ __forceinline__ void add_bf16x8(float (&acc)[8], const uint4& q) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const uint16_t lo = (uint16_t)(w[j] & 0xFFFFu), hi = (uint16_t)(w[j] >> 16);
    asm("add.rn.f32.bf16 %0, %1, %0;" : "+f"(acc[2 * j]) : "h"(lo));
    asm("add.rn.f32.bf16 %0, %1, %0;" : "+f"(acc[2 * j + 1]) : "h"(hi));
  }
}

// B16: table rows are 64 bf16 (8 lanes x uint4, ld16 = row stride in 16-byte units), sum of the rows, scaled per row in the
// epilogue.  fp32: table rows are 64 floats (16 lanes x float4), A's values multiply.
template <bool B16>
__global__ void __launch_bounds__(256, B16 ? 4 : 3) spmm64_units_kernel(const int32_t* __restrict__ idx, const float* __restrict__ val,
                                                                      const void* __restrict__ tab, uint32_t row_bytes,
                                                                      const int64_t* __restrict__ plan, int64_t nnz, int64_t row0,
                                                                      int64_t row1, Epi ep, float* __restrict__ y, int64_t ld_y,
                                                                      float* __restrict__ partial) {
  constexpr int G = B16 ? 8 : 16;          // lanes per unit
  constexpr int GPW = 32 / G;              // units per warp
  constexpr uint32_t FULL = 0xffffffffu;
  constexpr uint32_t DEAD = 0xffffffffu;   // descriptor of "no unit" (length 127 does not exist)
  const int lane = threadIdx.x & 31;
  const int lg = lane & (G - 1);
  const int e8 = lg & 7;                   // entry of an 8-entry block this lane fetches (fp32: lanes 8-15 fetch the values)
  const int stride = (int)gridDim.x * 8 * GPW;
  const int64_t max_chunks = plan_max_chunks(nnz);
  const int n_chunks = (int)(plan[1] < max_chunks ? plan[1] : max_chunks);
  const int64_t v3w = plan_v3_word(nnz);
  const int n_units = n_chunks + reinterpret_cast<const int32_t*>(plan + v3w)[0];
  const int2* unit = reinterpret_cast<const int2*>(plan + plan_v3_unit_word(nnz));
  const char* tl = reinterpret_cast<const char*>(tab) + lg * 16;
  const uint32_t r_lo = (uint32_t)row0, r_hi = (uint32_t)row1;       // rows < 2^25

  // Software pipeline over this group's units u, u + stride, ...: while unit k is gathered, the first index block (and the
  // row scale) of unit k + 1 and the descriptor of unit k + 2 are in flight, so a unit exposes ONE memory round trip (its
  // gathers) instead of three.  All trip counts are warp-uniform (the units of a warp have equal lengths up to bin
  // borders): the shuffles use the full mask and only the final stores diverge.
  auto fetch = [&](int uu) { return uu < n_units ? __ldg(unit + uu) : make_int2((int)DEAD, 0); };
  auto first_block = [&](const int2& d, int len) -> uint32_t {
    if (e8 >= len) return 0u;
    if (!B16 && lg >= 8) return __float_as_uint(__ldcs(val + (uint32_t)d.y + e8));
    return (uint32_t)__ldcs(idx + (uint32_t)d.y + e8);
  };
  auto decode_len = [&](const int2& d) -> int {       // 0 for no unit / a row outside [row0, row1)
    const uint32_t r = (uint32_t)d.x & ((1u << V3_ROW_BITS) - 1);
    return ((uint32_t)d.x != DEAD && r >= r_lo && r < r_hi) ? (int)((uint32_t)d.x >> V3_ROW_BITS) : -1;
  };
  int u = ((int)blockIdx.x * 8 + (threadIdx.x >> 5)) * GPW + lane / G;
  int2 d_cur = fetch(u), d_nxt = fetch(u + stride);
  int len_cur = decode_len(d_cur);                     // -1: dead
  uint32_t my = first_block(d_cur, len_cur);
  float sc_cur = (len_cur >= 0 && ep.rscale) ? __ldg(ep.rscale + ((uint32_t)d_cur.x & ((1u << V3_ROW_BITS) - 1))) : 1.f;
  for (; __any_sync(FULL, u < n_units); u += stride) {
    const int2 d_nn = fetch(u + 2 * stride);
    const int len_nxt = decode_len(d_nxt);
    const uint32_t my_nxt = first_block(d_nxt, len_nxt);
    const float sc_nxt = (len_nxt >= 0 && ep.rscale) ? __ldg(ep.rscale + ((uint32_t)d_nxt.x & ((1u << V3_ROW_BITS) - 1))) : 1.f;
    const int len = len_cur < 0 ? 0 : len_cur;
    const uint32_t start = (uint32_t)d_cur.y;
    const int lenw = __reduce_max_sync(FULL, len);
    float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};      // fp32 path: acc[0..4)
#pragma unroll 1
    for (int base = 0; base < lenw; base += 8) {
      const int n = len - base;          // this unit's entries left (may be <= 0 in a mixed warp)
      const int nw = lenw - base;        // the warp's
      uint32_t my_nb = 0u;               // the next block's (column, value) pairs: in flight behind this block's gathers
      if (n > 8 && e8 < n - 8)
        my_nb = (!B16 && lg >= 8) ? __float_as_uint(__ldcs(val + start + base + 8 + e8)) : (uint32_t)__ldcs(idx + start + base + 8 + e8);
      if constexpr (B16) {
        uint4 q[8];
        if (nw >= 8) {
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const uint32_t c = __shfl_sync(FULL, my, t, 8);
            q[t] = __ldg(reinterpret_cast<const uint4*>(tl + (size_t)c * row_bytes));
          }
#pragma unroll
          for (int t = 0; t < 8; ++t)
            if (t < n) add_bf16x8(acc, q[t]);
        } else {
#pragma unroll
          for (int t = 0; t < 7; ++t)
            if (t < nw) {
              const uint32_t c = __shfl_sync(FULL, my, t, 8);
              q[t] = __ldg(reinterpret_cast<const uint4*>(tl + (size_t)c * row_bytes));
            }
#pragma unroll
          for (int t = 0; t < 7; ++t)
            if (t < nw && t < n) add_bf16x8(acc, q[t]);
        }
      } else {
        float4 q[8];
        float v[8];
        float4 a4 = make_float4(acc[0], acc[1], acc[2], acc[3]);
        if (nw >= 8) {
#pragma unroll
          for (int t = 0; t < 8; ++t) {
            const uint32_t c = __shfl_sync(FULL, my, t, 16);
            v[t] = __uint_as_float(__shfl_sync(FULL, my, 8 + t, 16));
            q[t] = __ldg(reinterpret_cast<const float4*>(tl + (size_t)c * row_bytes));
          }
#pragma unroll
          for (int t = 0; t < 8; ++t)
            if (t < n) a4 = fma4(v[t], q[t], a4);      // beyond this unit's entries: column 0 with value 0 (0 * inf = NaN)
        } else {
#pragma unroll
          for (int t = 0; t < 7; ++t)
            if (t < nw) {
              const uint32_t c = __shfl_sync(FULL, my, t, 16);
              v[t] = __uint_as_float(__shfl_sync(FULL, my, 8 + t, 16));
              q[t] = __ldg(reinterpret_cast<const float4*>(tl + (size_t)c * row_bytes));
            }
#pragma unroll
          for (int t = 0; t < 7; ++t)
            if (t < nw && t < n) a4 = fma4(v[t], q[t], a4);
        }
        acc[0] = a4.x, acc[1] = a4.y, acc[2] = a4.z, acc[3] = a4.w;
      }
      my = my_nb;
    }
    if (len_cur >= 0) {
      const int64_t row = (uint32_t)d_cur.x & ((1u << V3_ROW_BITS) - 1);
      if constexpr (B16) {
        float4 o0 = make_float4(acc[0], acc[1], acc[2], acc[3]), o1 = make_float4(acc[4], acc[5], acc[6], acc[7]);
        if (u < n_chunks) {
          float4* dst = reinterpret_cast<float4*>(partial + (int64_t)u * 64) + 2 * lg;
          dst[0] = o0, dst[1] = o1;
        } else {
          const float a = ep.alpha * sc_cur;
          o0 = make_float4(a * o0.x, a * o0.y, a * o0.z, a * o0.w), o1 = make_float4(a * o1.x, a * o1.y, a * o1.z, a * o1.w);
          if (ep.z) {
            const float4* zp = reinterpret_cast<const float4*>(ep.z + row * ep.ld_z) + 2 * lg;
            const float4 z0 = __ldg(zp), z1 = __ldg(zp + 1);
            o0 = make_float4(fmaf(ep.beta, z0.x, o0.x), fmaf(ep.beta, z0.y, o0.y), fmaf(ep.beta, z0.z, o0.z), fmaf(ep.beta, z0.w, o0.w));
            o1 = make_float4(fmaf(ep.beta, z1.x, o1.x), fmaf(ep.beta, z1.y, o1.y), fmaf(ep.beta, z1.z, o1.z), fmaf(ep.beta, z1.w, o1.w));
          }
          float4* dst = reinterpret_cast<float4*>(y + row * ld_y) + 2 * lg;
          __stcs(dst, o0);
          __stcs(dst + 1, o1);
        }
      } else {
        const float4 a4 = make_float4(acc[0], acc[1], acc[2], acc[3]);
        if (u < n_chunks) {
          reinterpret_cast<float4*>(partial + (int64_t)u * 64)[lg] = a4;
        } else {
          store_row_cs(y, ld_y, row, lg, a4, ep);
        }
      }
    }
    d_cur = d_nxt, d_nxt = d_nn, len_cur = len_nxt, my = my_nxt, sc_cur = sc_nxt;
  }
}

// T[r, :] = bf16(dinv[r] * X[r, :]) with X = [x (rows < n_first) ; x2 (the rest)]: the gather table of dmm_spmm_norm_bf16
__global__ void __launch_bounds__(256) spmm_table_bf16_kernel(const float* __restrict__ x, int64_t ld_x, int64_t n_first,
                                                              const float* __restrict__ x2, int64_t ld_x2, int64_t n_rows,
                                                              const float* __restrict__ dinv, uint4* __restrict__ t) {
  const int64_t r = ((int64_t)blockIdx.x * 256 + threadIdx.x) >> 3;
  if (r >= n_rows) return;
  const int lg = threadIdx.x & 7;
  const float* src = r < n_first ? x + r * ld_x : x2 + (r - n_first) * ld_x2;
  const float4 a = __ldcs(reinterpret_cast<const float4*>(src) + 2 * lg), b = __ldcs(reinterpret_cast<const float4*>(src) + 2 * lg + 1);
  const float s = __ldg(dinv + r);
  uint4 o;
  o.x = (uint32_t)dmm_bf16_bits(s * a.x) | ((uint32_t)dmm_bf16_bits(s * a.y) << 16);
  o.y = (uint32_t)dmm_bf16_bits(s * a.z) | ((uint32_t)dmm_bf16_bits(s * a.w) << 16);
  o.z = (uint32_t)dmm_bf16_bits(s * b.x) | ((uint32_t)dmm_bf16_bits(s * b.y) << 16);
  o.w = (uint32_t)dmm_bf16_bits(s * b.z) | ((uint32_t)dmm_bf16_bits(s * b.w) << 16);
  t[r * 8 + lg] = o;
}

// ---- generic D (multiple of 4, <= 256): one warp per row, lanes stride the float4 columns ----------
__global__ void __launch_bounds__(SPMM_THREADS) spmm_generic_kernel(const int64_t* __restrict__ ptr,
                                                                    const int32_t* __restrict__ idx,
                                                                    const float* __restrict__ val, int64_t row0,
                                                                    int64_t row1, const float* __restrict__ x,
                                                                    int64_t ld_x, int D4, Epi ep, float* __restrict__ y,
                                                                    int64_t ld_y) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t r = row0 + (int64_t)blockIdx.x * SPMM_WARPS + warp;
  if (r >= row1) return;
  const int64_t b = ptr[r], e = ptr[r + 1];
  float4 acc0 = make_float4(0.f, 0.f, 0.f, 0.f), acc1 = acc0;  // columns lane and lane + 32 (D4 <= 64)
  for (int64_t j = b; j < e; ++j) {
    const int32_t c = __ldg(idx + j);
    const float v = __ldg(val + j);
    const float4* xr = reinterpret_cast<const float4*>(x + (int64_t)c * ld_x);
    if (lane < D4) acc0 = fma4(v, __ldg(xr + lane), acc0);
    if (lane + 32 < D4) acc1 = fma4(v, __ldg(xr + lane + 32), acc1);
  }
  for (int k = 0; k < 2; ++k) {
    const int col = lane + 32 * k;
    if (col >= D4) break;
    const float4 a = k ? acc1 : acc0;
    float4 o = make_float4(ep.alpha * a.x, ep.alpha * a.y, ep.alpha * a.z, ep.alpha * a.w);
    if (ep.z) {
      const float4 zz = __ldg(reinterpret_cast<const float4*>(ep.z + r * ep.ld_z) + col);
      o = make_float4(fmaf(ep.beta, zz.x, o.x), fmaf(ep.beta, zz.y, o.y), fmaf(ep.beta, zz.z, o.z), fmaf(ep.beta, zz.w, o.w));
    }
    reinterpret_cast<float4*>(y + r * ld_y)[col] = o;
  }
}

// ---- cross-layer CL perturbation (Main.py:320-321), one warp per row --------------------------------
__global__ void __launch_bounds__(256) sign_noise_kernel(float* __restrict__ e, int64_t ld_e,
                                                         const float* __restrict__ rnd, int64_t ld_r, int64_t n_rows,
                                                         int D, float noise_degree) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  float ss = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float v = __ldg(rnd + r * ld_r + c);
    ss = fmaf(v, v, ss);
  }
  ss = dmm_warp_sum(ss);
  const float inv = noise_degree / fmaxf(sqrtf(ss), 1e-12f);
  for (int c = lane; c < D; c += 32) {
    const float v = e[r * ld_e + c];
    const float sg = (v > 0.f) ? 1.f : ((v < 0.f) ? -1.f : 0.f);
    e[r * ld_e + c] = v + sg * __ldg(rnd + r * ld_r + c) * inv;
  }
}

}  // namespace

extern "C" int64_t dmm_spmm_plan_bytes(int64_t n_rows, int64_t nnz) {
  // long-row list + chunk descriptors, then the v3 sections: header, one unit per row, d^-1/2 per row
  return (int64_t)sizeof(int64_t) * (plan_v3_dinv_word(nnz, n_rows) + (n_rows + 1) / 2 + 2);
}

extern "C" int dmm_spmm_plan(dmm_ctx* ctx, const int64_t* adj_ptr, int64_t n_rows, int64_t nnz, void* plan,
                             int64_t plan_bytes, void* stream) {
  DMM_CHECK_ARG(ctx && adj_ptr && plan, "dmm_spmm_plan: null argument");
  DMM_CHECK_ARG(n_rows > 0 && nnz >= 0, "dmm_spmm_plan: bad sizes");
  DMM_CHECK_ARG(n_rows < (1LL << V3_ROW_BITS) && nnz < (1LL << 31),
                "dmm_spmm_plan: at most 2^25 rows and 2^31 entries (call dmm_spmm_csr with plan = NULL beyond that)");
  DMM_CHECK_ARG(plan_bytes >= dmm_spmm_plan_bytes(n_rows, nnz), "dmm_spmm_plan: plan buffer too small");
  cudaStream_t st = (cudaStream_t)stream;
  const int64_t cap = plan_cap(nnz);
  DMM_CUDA(cudaMemsetAsync(plan, 0, 2 * sizeof(int64_t), st));
  int64_t* v3 = (int64_t*)plan + plan_v3_word(nnz);
  int32_t* h = (int32_t*)v3;
  DMM_CUDA(cudaMemsetAsync(h, 0, V3_HDR_WORDS * sizeof(int64_t), st));
  plan_collect_kernel<<<(unsigned)dmm_ceil_div(n_rows, 256), 256, 0, st>>>(adj_ptr, n_rows, cap, (int64_t*)plan);
  DMM_LAUNCH_CHECK();
  plan_scan_kernel<<<1, 1024, 0, st>>>(adj_ptr, cap, (int64_t*)plan, h, (int32_t*)(v3 + V3_HDR_WORDS));
  DMM_LAUNCH_CHECK();
  // v3: the chunks and the rows of at most PLAN_LONG_ROW entries as units sorted by length, and d^-1/2 per row
  int2* unit = (int2*)((int64_t*)plan + plan_v3_unit_word(nnz));
  float* dinv = (float*)((int64_t*)plan + plan_v3_dinv_word(nnz, n_rows));
  plan_desc_kernel<<<(unsigned)(ctx->num_sms * 4), 256, 0, st>>>(adj_ptr, cap, (int64_t*)plan, unit);
  DMM_LAUNCH_CHECK();
  v3_hist_kernel<<<(unsigned)dmm_ceil_div(n_rows, 1024), 1024, 0, st>>>(adj_ptr, n_rows, h, dinv);
  DMM_LAUNCH_CHECK();
  v3_scan_kernel<<<1, 32, 0, st>>>(h);
  DMM_LAUNCH_CHECK();
  v3_scatter_kernel<<<(unsigned)dmm_ceil_div(n_rows, 1024), 1024, 0, st>>>(adj_ptr, n_rows, h, unit, (const int64_t*)plan + 1,
                                                                          plan_max_chunks(nnz));
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

namespace {
// v3: one persistent launch over the units (chunks of the long rows + length-sorted short rows), then the fixed-order reduce
template <bool B16>
int launch_units(dmm_ctx* ctx, const int32_t* adj_idx, const float* adj_val, int64_t row0, int64_t row1, const void* tab,
                 uint32_t row_bytes, const Epi& ep, float* y, int64_t ld_y, const void* plan, int64_t nnz, void* workspace,
                 cudaStream_t st) {
  const int64_t cap = plan_cap(nnz);
  spmm64_units_kernel<B16><<<(unsigned)(ctx->num_sms * (B16 ? 4 : 3)), 256, 0, st>>>(adj_idx, adj_val, tab, row_bytes, (const int64_t*)plan, nnz,
                                                                        row0, row1, ep, y, ld_y, (float*)workspace);
  DMM_LAUNCH_CHECK();
  spmm64_reduce_kernel<<<(unsigned)(ctx->num_sms * 2), REDUCE_THREADS, 0, st>>>(row0, row1, (const int64_t*)plan, cap,
                                                                       (const float*)workspace, ep, y, ld_y,
                                                                       (const int32_t*)((const int64_t*)plan + plan_v3_word(nnz)));
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
}  // namespace

extern "C" int dmm_spmm_table_bf16(dmm_ctx* ctx, const float* x, int64_t ld_x, int64_t n_first, const float* x2, int64_t ld_x2,
                                   int64_t n_rows, const void* plan, int64_t nnz, uint16_t* t, void* stream) {
  DMM_CHECK_ARG(ctx && x && plan && t, "dmm_spmm_table_bf16: null argument");
  DMM_CHECK_ARG(n_rows > 0 && n_first >= 0 && (n_first >= n_rows || x2), "dmm_spmm_table_bf16: bad row split");
  DMM_CHECK_ARG(ld_x % 4 == 0 && ld_x >= 64 && (!x2 || (ld_x2 % 4 == 0 && ld_x2 >= 64)),
                "dmm_spmm_table_bf16: D is 64; leading dimensions must be multiples of 4");
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(x) && al16(x2) && al16(t), "dmm_spmm_table_bf16: X and T must be 16-byte aligned");
  const float* dinv = (const float*)((const int64_t*)plan + plan_v3_dinv_word(nnz, n_rows));
  spmm_table_bf16_kernel<<<(unsigned)dmm_ceil_div(n_rows * 8, 256), 256, 0, (cudaStream_t)stream>>>(
      x, ld_x, n_first < n_rows ? n_first : n_rows, x2, ld_x2, n_rows, dinv, (uint4*)t);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_spmm_norm_bf16(dmm_ctx* ctx, const int32_t* adj_idx, int64_t row0, int64_t row1, int64_t n_rows,
                                  const uint16_t* t, float alpha, float beta, const float* z, int64_t ld_z, float* y,
                                  int64_t ld_y, const void* plan, int64_t nnz, void* workspace, int64_t workspace_bytes,
                                  void* stream) {
  DMM_CHECK_ARG(ctx && adj_idx && t && y && plan && workspace, "dmm_spmm_norm_bf16: null argument");
  DMM_CHECK_ARG(ld_y % 4 == 0 && ld_y >= 64 && (!z || (ld_z % 4 == 0 && ld_z >= 64)),
                "dmm_spmm_norm_bf16: D is 64; leading dimensions must be multiples of 4");
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(t) && al16(y) && al16(z) && al16(workspace), "dmm_spmm_norm_bf16: T/Y/Z/workspace must be 16-byte aligned");
  DMM_CHECK_ARG(row0 >= 0 && row1 >= row0 && row1 <= n_rows && nnz < (1LL << 31), "dmm_spmm_norm_bf16: bad row range / nnz");
  DMM_CHECK_ARG(workspace_bytes >= dmm_spmm_workspace_bytes(nnz, 64), "dmm_spmm_norm_bf16: workspace too small");
  if (row1 == row0) return DMM_OK;
  const float* dinv = (const float*)((const int64_t*)plan + plan_v3_dinv_word(nnz, n_rows));
  const Epi ep{alpha, z ? beta : 0.f, z, ld_z, dinv};
  return launch_units<true>(ctx, adj_idx, nullptr, row0, row1, t, 128u, ep, y, ld_y, plan, nnz, workspace, (cudaStream_t)stream);
}

extern "C" int64_t dmm_spmm_workspace_bytes(int64_t nnz, int64_t D) {
  if (D != 64) return 0;
  // chunks <= nnz / PLAN_CHUNK + (#planned rows <= nnz / PLAN_LONG_ROW + 1)
  return (nnz / PLAN_CHUNK + plan_cap(nnz) + 1) * 64 * (int64_t)sizeof(float);
}

extern "C" int dmm_spmm_csr(dmm_ctx* ctx, const int64_t* adj_ptr, const int32_t* adj_idx, const float* adj_val,
                            int64_t row0, int64_t row1, const float* x, int64_t ld_x, int64_t D, float alpha,
                            float beta, const float* z, int64_t ld_z, float* y, int64_t ld_y, const void* plan,
                            int64_t nnz, void* workspace, int64_t workspace_bytes, void* stream) {
  DMM_CHECK_ARG(ctx && adj_ptr && adj_idx && adj_val && x && y, "dmm_spmm_csr: null argument");
  DMM_CHECK_ARG(D > 0 && D % 4 == 0 && D <= 256, "dmm_spmm_csr: D must be a multiple of 4 and <= 256 (got %lld)", (long long)D);
  DMM_CHECK_ARG(ld_x % 4 == 0 && ld_y % 4 == 0 && ld_x >= D && ld_y >= D && (!z || (ld_z % 4 == 0 && ld_z >= D)),
                "dmm_spmm_csr: leading dimensions must be >= D and multiples of 4");
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(x) && al16(y) && al16(z) && al16(workspace), "dmm_spmm_csr: X/Y/Z/workspace must be 16-byte aligned");
  DMM_CHECK_ARG(row0 >= 0 && row1 >= row0, "dmm_spmm_csr: bad row range");
  const bool planned = plan != nullptr && D == 64;
  DMM_CHECK_ARG(!planned || (workspace && workspace_bytes >= dmm_spmm_workspace_bytes(nnz, D)),
                "dmm_spmm_csr: a plan needs a workspace of dmm_spmm_workspace_bytes(nnz, D) bytes");
  if (row1 == row0) return DMM_OK;
  const Epi ep{alpha, z ? beta : 0.f, z, ld_z};
  const unsigned grid = (unsigned)dmm_ceil_div(row1 - row0, SPMM_WARPS);
  cudaStream_t st = (cudaStream_t)stream;
  if (D == 64) {
    if (!planned) {
      spmm64_kernel<<<grid, SPMM_THREADS, 0, st>>>(adj_ptr, adj_idx, adj_val, row0, row1, x, ld_x, ep, y, ld_y, 0);
    } else {
      DMM_CHECK_ARG(nnz < (1LL << 31) && ld_x < (1LL << 28), "dmm_spmm_csr: a planned product needs nnz < 2^31 and ld_x < 2^28");
      return launch_units<false>(ctx, adj_idx, adj_val, row0, row1, x, (uint32_t)(ld_x * 4), ep, y, ld_y, plan, nnz, workspace, st);
    }
  } else {
    spmm_generic_kernel<<<grid, SPMM_THREADS, 0, st>>>(adj_ptr, adj_idx, adj_val, row0, row1, x, ld_x, (int)(D / 4), ep, y, ld_y);
  }
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_sign_noise_(dmm_ctx* ctx, float* e, int64_t ld_e, const float* rnd, int64_t ld_r, int64_t n_rows,
                               int64_t D, float noise_degree, void* stream) {
  DMM_CHECK_ARG(ctx && e && rnd, "dmm_sign_noise_: null argument");
  DMM_CHECK_ARG(D > 0 && ld_e >= D && ld_r >= D, "dmm_sign_noise_: bad shape");
  if (n_rows <= 0) return DMM_OK;
  sign_noise_kernel<<<(unsigned)dmm_ceil_div(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(e, ld_e, rnd, ld_r, n_rows,
                                                                                              (int)D, noise_degree);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
