// Per-user variable-k top-k -> edge list (rebuild of the modality-aware user-item graph).
//
// Replaces the Python loop of Main.py:224-230 (one torch.topk launch per user and one
// int(tensor) host sync per emitted edge).  One CTA per user row; the output slot of row r is
// out_ptr[r] .. out_ptr[r+1] (k_r = deg(u), so the offsets are the train CSR indptr: no atomics
// on the output, no host sync, deterministic).  Tie-break: value descending, then column
// ascending (-0.0 == +0.0); the emitted columns are ascending.  HBM-bound by design: 4*I bytes
// read and 4*k bytes written per user and modality.
//
// Fast path (rows of up to 32 keys per thread, k <= block size: every shipped config):
//   1. the fp32 row is read ONCE (float4, streaming) into REGISTERS as order-preserving keys;
//   2. a lower bound L of the k-th largest key comes from the per-thread maxima: every warp sorts
//      its 32 maxima (shuffle bitonic network) and publishes its q-th largest, q = ceil(k / warps);
//      L = the smallest of those, so at least q keys per warp, i.e. >= k keys, are >= L;
//   3. the keys >= L (a few more than k for continuous scores) are compacted with warp-aggregated
//      atomics into shared memory and ranked exactly against each other (value desc, column asc);
//      the k best are written in ascending column order.  No per-key atomics, no pass over the row
//      after the load except the register compare of step 3.
// Generic path (huge k, crowded ties, very wide or unaligned rows; also the in-kernel fallback):
//   range-adapted bucket histogram -> exact MSB radix select of the threshold -> ordered block scan.
#include "common.cuh"

#include <stdlib.h>

namespace {

constexpr int TOPK_NB_LOG2 = 11;
constexpr int TOPK_NB = 1 << TOPK_NB_LOG2;   // range-adapted buckets of the generic path's first pass
constexpr int TOPK_CAND = 1024;              // candidate keys held in shared memory
constexpr int TOPK_V4 = 8;                   // float4 loads per thread on the register path (32 keys)
constexpr int TOPK_SEG_COLS = 8192;          // widest column segment of the segmented path (the 256-thread register kernel)
constexpr int TOPK_MERGE_CAP = 2048;         // candidates (segments x k) the merge kernel ranks per row

// Rows wider than TOPK_SEG_COLS.  One CTA of 512 / 1024 threads per row keeps only one or two rows per SM in flight and
// pays 16 / 32-warp barriers between the select phases (measured 1.1 TB/s at 18357 columns, 17 % of HBM).  Instead the
// row is cut into S column segments that the 256-thread register kernel treats as independent rows (mode 1: the k best
// of every segment go to a temporary list - the row's k best are among them), a small merge kernel ranks the S * k
// candidates of a row exactly (value desc, column asc) and emits the k best in ascending column order, and the rows
// that do not qualify (k > 256, k longer than the last segment, S * k > TOPK_MERGE_CAP, k = 0) take the whole-row
// kernels as before (mode 2).
struct SegCfg {
  int mode;       // 0: plain, 1: segment pass, 2: whole-row pass over the rows the segment pass skipped
  int S;          // segments per row
  int seg_cols;   // columns per segment (multiple of 4)
  int last_len;   // columns of the last segment
};
__device__ __forceinline__ bool seg_eligible(const SegCfg& sg, int k) {
  return k > 0 && k <= 256 && k <= sg.last_len && (int64_t)sg.S * k <= TOPK_MERGE_CAP;
}

// NaN-propagating maximum (max.NaN.f32): a NaN score surfaces in the piece / thread maximum instead of vanishing
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

__device__ __forceinline__ uint32_t order_key(float f) {
  uint32_t u = __float_as_uint(f);
  if (u == 0x80000000u) u = 0u;  // -0.0 ties with +0.0
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

template <int NT>
struct alignas(16) TopkSmem {
  int bucket[TOPK_NB];        // generic: bucket histogram; fast: selected-column scratch
  uint32_t cand[TOPK_CAND];   // candidate keys
  int cand_col[TOPK_CAND];    // candidate columns (fast path)
  int hist[256];
  int warp_sums[NT / 32];
  uint32_t red[2 * (NT / 32)];
  uint32_t prefix;
  int kk, bin, above, ncand;
};

// block-wide exclusive scan of one int per thread; returns the exclusive prefix, total in *total
template <int NT>
__device__ __forceinline__ int block_excl_scan(int v, int* warp_sums, int* total) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  int incl = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int t = __shfl_up_sync(0xffffffffu, incl, o);
    if (lane >= o) incl += t;
  }
  const int warp_total = __shfl_sync(0xffffffffu, incl, 31);
  if (lane == 0) warp_sums[w] = warp_total;
  __syncthreads();
  int base = 0, tot = 0;
#pragma unroll
  for (int i = 0; i < NT / 32; ++i) {
    const int s = warp_sums[i];
    if (i < w) base += s;
    tot += s;
  }
  __syncthreads();
  *total = tot;
  return base + incl - v;
}

// MSB-first radix select (4 passes x 8 bits, warp-aggregated shared-memory histograms) of the
// `want`-th largest of `count` keys read through `key_at`.  Returns the threshold key and, in
// *need_eq, how many keys equal to it belong to the top `want`.  Uniform across the block.
template <int NT, typename KeyAt>
__device__ __forceinline__ uint32_t radix_select(KeyAt key_at, int count, int want, TopkSmem<NT>& sm, int* need_eq) {
  const int tid = threadIdx.x;
  uint32_t prefix = 0u, mask = 0u;
  int kk = want;
#pragma unroll 1
  for (int shift = 24; shift >= 0; shift -= 8) {
    if (tid < 256) sm.hist[tid] = 0;
    __syncthreads();
    for (int i0 = 0; i0 < count; i0 += NT) {
      const int i = i0 + tid;
      const bool in = i < count;
      const uint32_t key = in ? key_at(i) : 0u;
      const bool cand = in && ((key & mask) == prefix);
      const uint32_t digit = (key >> shift) & 0xFFu;
      // one shared-memory atomic per distinct digit per warp
      const uint32_t active = __ballot_sync(0xffffffffu, cand);
      if (cand) {
        const uint32_t peers = __match_any_sync(active, digit);
        if ((int)(__ffs(peers) - 1) == (tid & 31)) atomicAdd(&sm.hist[digit], __popc(peers));
      }
    }
    __syncthreads();
    if (tid < 32) {
      // descending scan: lane l owns bins 255-8l .. 248-8l
      int loc[8], sum = 0;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        loc[j] = sm.hist[255 - 8 * tid - j];
        sum += loc[j];
      }
      int incl = sum;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (tid >= o) incl += t;
      }
      const int excl = incl - sum;
      if (excl < kk && kk <= incl) {
        int cum = excl;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          if (cum < kk && kk <= cum + loc[j]) {
            sm.prefix = prefix | ((uint32_t)(255 - 8 * tid - j) << shift);
            sm.kk = kk - cum;
          }
          cum += loc[j];
        }
      }
    }
    __syncthreads();
    prefix = sm.prefix;
    kk = sm.kk;
    mask |= 0xFFu << shift;
  }
  *need_eq = kk;
  return prefix;
}

// Exact selection + emission over `n` keys read through key_at(i) (value desc, index asc; the emitted entries leave in
// ascending index order as col_of(i)).  kmin / kmax: this thread's partial key range when `scanned`, else the function
// scans the keys itself.  Uniform across the block; every barrier is reached by every thread.
template <int NT, typename KeyAt, typename ColOf>
__device__ __forceinline__ void topk_select_emit(TopkSmem<NT>& sm, KeyAt key_at, ColOf col_of, int n_cols, int k,
                                                 bool scanned, uint32_t kmin, uint32_t kmax, int64_t o0, int32_t user,
                                                 int32_t* __restrict__ out_users, int32_t* __restrict__ out_items) {
  static_assert(NT >= 256, "the bucket scan and the radix histograms are laid out for at least 256 threads");
  const int tid = threadIdx.x;
  const bool take_all = !(k < n_cols);
  if (!scanned && !take_all) {
    kmin = 0xFFFFFFFFu;
    kmax = 0u;
    for (int i = tid; i < n_cols; i += NT) {
      const uint32_t key = key_at(i);
      kmin = min(kmin, key);
      kmax = max(kmax, key);
    }
  }
  uint32_t T = 0u;
  int need_eq = 0;
  if (!take_all) {
    for (int j = tid; j < TOPK_NB; j += NT) sm.bucket[j] = 0;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      kmin = min(kmin, __shfl_xor_sync(0xffffffffu, kmin, o));
      kmax = max(kmax, __shfl_xor_sync(0xffffffffu, kmax, o));
    }
    if ((tid & 31) == 0) {
      sm.red[tid >> 5] = kmin;
      sm.red[NT / 32 + (tid >> 5)] = kmax;
    }
    if (tid == 0) sm.ncand = 0;
    __syncthreads();
#pragma unroll
    for (int i = 0; i < NT / 32; ++i) {
      kmin = min(kmin, sm.red[i]);
      kmax = max(kmax, sm.red[NT / 32 + i]);
    }
    // (kmax - kmin) >> sh < TOPK_NB
    const uint32_t range = kmax - kmin;
    const int bits = 32 - __clz(range);               // range == 0 -> 0
    const int sh = bits > TOPK_NB_LOG2 ? bits - TOPK_NB_LOG2 : 0;
    for (int i = tid; i < n_cols; i += NT) atomicAdd(&sm.bucket[(key_at(i) - kmin) >> sh], 1);
    __syncthreads();
    {
      // descending scan over the buckets: thread t < 256 owns buckets NB-1-PER*t .. NB-PER*(t+1)
      constexpr int PER = TOPK_NB / 256;
      int loc[PER], sum = 0;
      if (tid < 256) {
#pragma unroll
        for (int j = 0; j < PER; ++j) {
          loc[j] = sm.bucket[TOPK_NB - 1 - PER * tid - j];
          sum += loc[j];
        }
      }
      int tot;
      const int excl = block_excl_scan<NT>(sum, sm.warp_sums, &tot);
      if (tid < 256 && excl < k && k <= excl + sum) {
        int cum = excl;
#pragma unroll
        for (int j = 0; j < PER; ++j) {
          if (cum < k && k <= cum + loc[j]) {
            sm.bin = TOPK_NB - 1 - PER * tid - j;
            sm.above = cum;
          }
          cum += loc[j];
        }
      }
    }
    __syncthreads();
    const int bin = sm.bin;
    const int want = k - sm.above;          // >= 1: rank of the threshold inside its bucket
    const int m = sm.bucket[bin];
    if (m <= TOPK_CAND) {
      for (int i = tid; i < n_cols; i += NT) {
        const uint32_t key = key_at(i);
        if ((int)((key - kmin) >> sh) == bin) sm.cand[atomicAdd(&sm.ncand, 1)] = key;
      }
      __syncthreads();
      T = radix_select<NT>([&](int i) -> uint32_t { return sm.cand[i]; }, m, want, sm, &need_eq);
    } else {
      T = radix_select<NT>(key_at, n_cols, k, sm, &need_eq);
    }
  }

  // take every key > T and the first need_eq keys == T (ascending column)
  // contiguous segment per thread, odd length => conflict-free strided shared-memory reads
  int seg = (n_cols + NT - 1) / NT;
  seg |= 1;
  const int b = min(tid * seg, n_cols), e = min(b + seg, n_cols);
  int c_gt = 0, c_eq = 0;
  for (int i = b; i < e; ++i) {
    const uint32_t key = key_at(i);
    c_gt += (take_all || key > T) ? 1 : 0;
    c_eq += (!take_all && key == T) ? 1 : 0;
  }
  int tot;
  const int eq_before = block_excl_scan<NT>(c_eq, sm.warp_sums, &tot);
  int eq_take = need_eq - eq_before;
  eq_take = eq_take < 0 ? 0 : (eq_take > c_eq ? c_eq : eq_take);
  const int pos0 = block_excl_scan<NT>(c_gt + eq_take, sm.warp_sums, &tot);
  if (c_gt + eq_take == 0) return;        // no barrier follows
  int64_t w = o0 + pos0;
  for (int i = b; i < e; ++i) {
    const uint32_t key = key_at(i);
    bool sel = take_all || key > T;
    if (!sel && key == T && eq_take > 0) {
      sel = true;
      --eq_take;
    }
    if (sel) {
      out_items[w] = col_of(i);
      if (out_users) out_users[w] = user;
      ++w;
    }
  }
}

// Generic row: exact for any k, any score distribution, any row width.  The leading radix digits of fp32
// scores (sign + exponent) barely discriminate, so ONE histogram pass over range-adapted buckets
// ((key - kmin) >> sh, monotone in the key) isolates the bucket holding the k-th largest key; only that
// bucket's keys go through the exact radix select.  Rows whose threshold bucket is crowded (heavy ties)
// select over the whole row.  s_keys: the row's keys in shared memory when IN_SMEM, else the row is
// (re-)read from global memory / L2 on every pass.
template <int NT, bool IN_SMEM>
__device__ __forceinline__ void topk_row_generic(TopkSmem<NT>& sm, uint32_t* s_keys, const float* __restrict__ row,
                                                 int n_cols, int k, int64_t o0, int32_t user,
                                                 int32_t* __restrict__ out_users, int32_t* __restrict__ out_items,
                                                 int col_off = 0) {
  const int tid = threadIdx.x;
  uint32_t kmin = 0xFFFFFFFFu, kmax = 0u;
  auto track = [&](uint32_t key) {
    kmin = min(kmin, key);
    kmax = max(kmax, key);
  };
  if (IN_SMEM) {
    // single HBM read of the row; float4 when the row start is 16 B aligned
    const bool vec = ((reinterpret_cast<uintptr_t>(row) & 15u) == 0);
    if (vec) {
      const int n4 = n_cols >> 2;
      const float4* row4 = reinterpret_cast<const float4*>(row);
      for (int i = tid; i < n4; i += NT) {
        const float4 v = __ldcs(row4 + i);
        const uint4 q = make_uint4(order_key(v.x), order_key(v.y), order_key(v.z), order_key(v.w));
        reinterpret_cast<uint4*>(s_keys)[i] = q;
        track(q.x); track(q.y); track(q.z); track(q.w);
      }
      for (int i = (n4 << 2) + tid; i < n_cols; i += NT) {
        const uint32_t q = order_key(__ldcs(row + i));
        s_keys[i] = q;
        track(q);
      }
    } else {
      for (int i = tid; i < n_cols; i += NT) {
        const uint32_t q = order_key(__ldcs(row + i));
        s_keys[i] = q;
        track(q);
      }
    }
  }
  auto key_at = [&](int i) -> uint32_t { return IN_SMEM ? s_keys[i] : order_key(__ldg(row + i)); };
  auto col_of = [&](int i) -> int { return i + col_off; };
  topk_select_emit<NT>(sm, key_at, col_of, n_cols, k, IN_SMEM, kmin, kmax, o0, user, out_users, out_items);
}

// ------------------------------------------------------------------------------------------ generic kernel
template <bool IN_SMEM>
__global__ void __launch_bounds__(256) topk_edges_kernel(const float* __restrict__ scores, int64_t ld, int64_t n_rows,
                                                         int n_cols, const int64_t* __restrict__ out_ptr,
                                                         int64_t row_base, int32_t* __restrict__ out_users,
                                                         int32_t* __restrict__ out_items, int32_t* __restrict__ status,
                                                         const int32_t* __restrict__ order, SegCfg sg,
                                                         const int32_t* __restrict__ live) {
  extern __shared__ uint32_t s_keys[];  // n_cols keys when IN_SMEM
  __shared__ TopkSmem<256> sm;
  if ((int64_t)blockIdx.x >= n_rows) return;
  if (live && (int64_t)blockIdx.x >= (int64_t)*live) return;   // `order` is a device-built list of *live rows
  const int64_t r = order ? (int64_t)order[blockIdx.x] : (int64_t)blockIdx.x;   // scheduling order only
  const int64_t o0 = out_ptr[r], o1 = out_ptr[r + 1];
  int k = (int)(o1 - o0);
  if (k <= 0) return;
  if (sg.mode == 2 && seg_eligible(sg, k)) return;      // done by the segment pass
  if (k > n_cols) {
    if (status && threadIdx.x == 0) atomicOr(status, 1);
    k = n_cols;
  }
  topk_row_generic<256, IN_SMEM>(sm, s_keys, scores + r * ld, n_cols, k, o0, (int32_t)(row_base + r), out_users,
                                 out_items);
}

// ------------------------------------------------------------------------------------------ register kernel
template <int NT>
__global__ void __launch_bounds__(NT, NT == 256 ? 5 : 1) topk_rows_reg_kernel(const float* __restrict__ scores, int64_t ld, int64_t n_rows,
                                                           int n_cols_arg, const int64_t* __restrict__ out_ptr,
                                                           int64_t row_base, int32_t* __restrict__ out_users,
                                                           int32_t* __restrict__ out_items_arg, int32_t* __restrict__ status,
                                                           const int32_t* __restrict__ order, SegCfg sg,
                                                           int32_t* __restrict__ seg_tmp, const int32_t* __restrict__ live) {
  __shared__ TopkSmem<NT> sm;
  constexpr int NW = NT / 32;
  // segment pass (sg.mode == 1): block b is segment b % S of the row scheduled in slot b / S
  const int seg = sg.mode == 1 ? (int)(blockIdx.x % (unsigned)sg.S) : 0;
  const int64_t slot = sg.mode == 1 ? (int64_t)(blockIdx.x / (unsigned)sg.S) : (int64_t)blockIdx.x;
  if (slot >= n_rows) return;
  if (live && slot >= (int64_t)*live) return;
  // scheduling order only (rows with a large k take the slower exact paths: started first, they overlap the rest)
  const int64_t r = order ? (int64_t)order[slot] : slot;
  const int col_off = seg * sg.seg_cols;
  const int n_cols = sg.mode == 1 ? (n_cols_arg - col_off < sg.seg_cols ? n_cols_arg - col_off : sg.seg_cols) : n_cols_arg;
  const float* row = scores + r * ld + col_off;
  int32_t* __restrict__ out_items = sg.mode == 1 ? seg_tmp : out_items_arg;
  if (sg.mode == 1) out_users = nullptr;
  if (sg.mode != 0) {
    // each row belongs to exactly one of the two passes: decided before the row is touched (block-uniform)
    const int kk = (int)(out_ptr[r + 1] - out_ptr[r]);
    if ((sg.mode == 1) != seg_eligible(sg, kk)) return;
  }
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const bool aligned = (reinterpret_cast<uintptr_t>(row) & 15u) == 0;

  // 1. the row -> registers, issued before anything depends on out_ptr so that both latencies overlap.
  //    Thread t owns the float4 pieces t, t + NT, ... (all TOPK_V4 loads in flight at once); the <= 3 columns
  //    past the last whole piece are one extra key each on threads 0..2.
  const int n4 = aligned ? (n_cols >> 2) : 0;
  const float4* row4 = reinterpret_cast<const float4*>(row);
  float4 v[TOPK_V4];
#pragma unroll
  for (int j = 0; j < TOPK_V4; ++j) {
    v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid + NT * j < n4) v[j] = __ldcs(row4 + tid + NT * j);
  }
  const int tail_col = (n4 << 2) + tid;
  const bool has_tail = aligned && tid < (n_cols & 3);
  float tail_v = 0.f;
  if (has_tail) tail_v = __ldcs(row + tail_col);

  int64_t o0 = out_ptr[r];
  const int64_t o1 = out_ptr[r + 1];
  int k = (int)(o1 - o0);
  if (k <= 0) return;
  if (sg.mode == 1) o0 = (int64_t)sg.S * (o0 - out_ptr[0]) + (int64_t)seg * k;   // this segment's slot of the temporary list
  if (k > n_cols) {
    if (status && threadIdx.x == 0) atomicOr(status, 1);
    k = n_cols;
  }
  const int32_t user = (int32_t)(row_base + r);
  if (k > NT || k >= n_cols || !aligned) {  // block-uniform
    topk_row_generic<NT, false>(sm, nullptr, row, n_cols, k, o0, user, out_users, out_items, col_off);
    return;
  }

  // pieces j < jfull are whole for every thread, piece jfull only for tid < jrem, later ones are empty.
  // The scan of the row stays in the float domain (one FMNMX per score); order-preserving keys, which carry
  // the exact tie semantics (-0.0 == +0.0, NaN order), are formed only for the thread maximum and the few
  // candidates.  The maxima propagate NaN, so a NaN score reaches the thread maximum and the row is handed to the
  // exact generic path (NaN keys have a total order the float comparisons cannot reproduce).
  const int jfull = n4 / NT, jrem = n4 - jfull * NT;
  const float NEG_INF = __uint_as_float(0xFF800000u);
  float pmax[TOPK_V4];                         // per-piece maximum: most pieces hold no candidate at all
  float tmaxf = has_tail ? fmax_nan(tail_v, NEG_INF) : NEG_INF;
#pragma unroll
  for (int j = 0; j < TOPK_V4; ++j) {
    pmax[j] = NEG_INF;
    if (j < jfull || (j == jfull && tid < jrem)) {
      pmax[j] = fmax_nan(fmax_nan(v[j].x, v[j].y), fmax_nan(v[j].z, v[j].w));
      tmaxf = fmax_nan(tmaxf, pmax[j]);
    }
  }
  // threads without a (non-NaN) score publish key 0, below every real key
  const uint32_t tmax = (tmaxf == NEG_INF) ? 0u : order_key(tmaxf);

  // 2. lower bound L of the k-th largest key from the per-thread maxima: this warp's q-th largest
  const int q = (k + NW - 1) / NW;             // 1 .. 32
  uint32_t wq;
  if (q <= 8) {
    // q rounds of warp max, retiring one holder of the maximum per round
    uint32_t sv = tmax;
    bool alive = true;
    wq = 0u;
    for (int i = 0; i < q; ++i) {
      wq = __reduce_max_sync(0xffffffffu, alive ? sv : 0u);
      const uint32_t holders = __ballot_sync(0xffffffffu, alive && sv == wq);
      if (holders == 0u) break;                // only retired lanes left: wq == 0
      if (lane == __ffs(holders) - 1) alive = false;
    }
  } else {
    uint32_t sv = tmax;
#pragma unroll
    for (int k2 = 2; k2 <= 32; k2 <<= 1) {
#pragma unroll
      for (int j = k2 >> 1; j > 0; j >>= 1) {
        const uint32_t other = __shfl_xor_sync(0xffffffffu, sv, j);
        const bool desc = (lane & k2) == 0;    // k2 == 32: the whole warp, descending
        const bool lower = (lane & j) == 0;
        sv = (lower == desc) ? max(sv, other) : min(sv, other);
      }
    }
    wq = __shfl_sync(0xffffffffu, sv, q - 1);
  }
  if (lane == 0) sm.red[wid] = wq;
  if (tid == 0) sm.ncand = 0;
  // the barrier doubles as the NaN vote: the bound below counts real scores, so a row with any NaN (whose key
  // order the float scan cannot see) takes the exact generic path
  if (__syncthreads_or(tmaxf != tmaxf)) {
    topk_row_generic<NT, false>(sm, nullptr, row, n_cols, k, o0, user, out_users, out_items, col_off);
    return;
  }
  uint32_t L = 0xFFFFFFFFu;
#pragma unroll
  for (int i = 0; i < NW; ++i) L = min(L, sm.red[i]);

  // 3. compact the candidates (key, column) into shared memory: one atomic per warp per hit group.
  //    L back in the float domain (L == 0: some warp lacks q real maxima, every score is a candidate)
  const float Lf = (L == 0u) ? NEG_INF : __uint_as_float((L & 0x80000000u) ? (L ^ 0x80000000u) : ~L);
  auto push = [&](bool c, float x, int col) {
    const uint32_t bal = __ballot_sync(0xffffffffu, c);
    if (bal) {
      int base = 0;
      if (lane == 0) base = atomicAdd(&sm.ncand, __popc(bal));
      base = __shfl_sync(0xffffffffu, base, 0);
      const int pos = base + __popc(bal & ((1u << lane) - 1u));
      if (c && pos < TOPK_CAND) {
        sm.cand[pos] = order_key(x);
        sm.cand_col[pos] = col;
      }
    }
  };
#pragma unroll
  for (int j = 0; j < TOPK_V4; ++j) {
    if (j > jfull) break;                      // block-uniform
    const bool have = j < jfull || tid < jrem;
    const bool open = have && !(pmax[j] < Lf);   // also true when the piece holds a NaN (pmax is NaN)
    if (__any_sync(0xffffffffu, open)) {
      const float xs[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) push(open && !(xs[e] < Lf), xs[e], 4 * (tid + NT * j) + e);
    }
  }
  if (n_cols & 3) push(has_tail && !(tail_v < Lf), tail_v, tail_col);   // block-uniform condition
  __syncthreads();
  const int m = sm.ncand;                      // >= k by construction of L (except for rows with NaN-only threads)
  constexpr int RANK_MAX = 512;                // candidates ranked against each other (m^2 / NT compares per thread)
  if (m > RANK_MAX || m < k) {                 // crowded threshold (ties) or loose bound: exact generic path
    __syncthreads();
    topk_row_generic<NT, false>(sm, nullptr, row, n_cols, k, o0, user, out_users, out_items, col_off);
    return;
  }
  // exact rank of every candidate among the m candidates by (value desc, column asc); the k best are marked
  // (one thread per candidate: a warp-cooperative variant executed more instructions in total and measured slower)
  for (int c = tid; c < m; c += NT) {
    const uint32_t my_key = sm.cand[c];
    const int my_col = sm.cand_col[c];
    int before = 0;
    if (m > k) {
      for (int j = 0; j < m; ++j) {
        const uint32_t kj = sm.cand[j];
        const int cj = sm.cand_col[j];
        before += (kj > my_key || (kj == my_key && cj < my_col)) ? 1 : 0;
      }
    }
    sm.bucket[c] = before < k ? my_col : 0x7FFFFFFF;
  }
  __syncthreads();
  // output position = number of selected columns below mine (ascending column order)
  for (int c = tid; c < m; c += NT) {
    const int my_col = sm.bucket[c];
    if (my_col == 0x7FFFFFFF) continue;
    int pos = 0;
    for (int j = 0; j < m; ++j) pos += (sm.bucket[j] < my_col) ? 1 : 0;
    out_items[o0 + pos] = my_col + col_off;
    if (out_users) out_users[o0 + pos] = user;
  }
}

// ------------------------------------------------------------------------------------------ merge of the segment lists
// One CTA per row that went through the segment pass: its S * k candidate columns (k per segment, read from the temporary
// list) are ranked exactly by (score desc, column asc) on the order-preserving keys of the scores they point at, and
// the k best leave in ascending column order.
__global__ void __launch_bounds__(128) topk_merge_kernel(const float* __restrict__ scores, int64_t ld, int64_t n_rows,
                                                         const int64_t* __restrict__ out_ptr, int64_t row_base,
                                                         int32_t* __restrict__ out_users, int32_t* __restrict__ out_items,
                                                         const int32_t* __restrict__ order, SegCfg sg,
                                                         const int32_t* __restrict__ seg_tmp, const int32_t* __restrict__ live) {
  __shared__ uint32_t key[TOPK_MERGE_CAP];
  __shared__ int col[TOPK_MERGE_CAP];
  __shared__ int sel[TOPK_MERGE_CAP];
  if ((int64_t)blockIdx.x >= n_rows) return;
  if (live && (int64_t)blockIdx.x >= (int64_t)*live) return;
  const int64_t r = order ? (int64_t)order[blockIdx.x] : (int64_t)blockIdx.x;
  const int64_t o0 = out_ptr[r];
  const int k = (int)(out_ptr[r + 1] - o0);
  if (!seg_eligible(sg, k)) return;
  const int m = sg.S * k;
  const int32_t* list = seg_tmp + (int64_t)sg.S * (o0 - out_ptr[0]);
  const float* row = scores + r * ld;
  for (int c = threadIdx.x; c < m; c += 128) {
    const int cc = list[c];
    col[c] = cc;
    key[c] = order_key(__ldg(row + cc));
  }
  __syncthreads();
  for (int c = threadIdx.x; c < m; c += 128) {
    const uint32_t my_key = key[c];
    const int my_col = col[c];
    int before = 0;
    for (int j = 0; j < m; ++j) before += (key[j] > my_key || (key[j] == my_key && col[j] < my_col)) ? 1 : 0;
    sel[c] = before < k ? my_col : 0x7FFFFFFF;
  }
  __syncthreads();
  const int32_t user = (int32_t)(row_base + r);
  for (int c = threadIdx.x; c < m; c += 128) {
    const int my_col = sel[c];
    if (my_col == 0x7FFFFFFF) continue;
    int pos = 0;
    for (int j = 0; j < m; ++j) pos += (sel[j] < my_col) ? 1 : 0;
    out_items[o0 + pos] = my_col;
    if (out_users) out_users[o0 + pos] = user;
  }
}

template <int NT>
void launch_reg(const float* scores, int64_t ld, int64_t n_rows, int n_cols, const int64_t* out_ptr, int64_t row_base,
                int32_t* out_users, int32_t* out_items, int32_t* status, const int32_t* order, SegCfg sg, int32_t* seg_tmp,
                const int32_t* live, cudaStream_t st) {
  const int64_t blocks = sg.mode == 1 ? n_rows * sg.S : n_rows;
  topk_rows_reg_kernel<NT><<<(unsigned)blocks, NT, 0, st>>>(scores, ld, n_rows, n_cols, out_ptr, row_base, out_users,
                                                           out_items, status, order, sg, seg_tmp, live);
}

// ------------------------------------------------------------------------------------------ pruned top-k
// The contraction that writes the scores also writes cmax[r, c] = max of the 32-column chunk c of row r (1/32 of the
// bytes, dmm_gemm_epilogue.cmax).  The k largest scores of a row lie in the k chunks with the largest maxima (ties:
// lower chunk first): each of those chunks holds a score >= the k-th largest maximum Lk, so the k-th largest score T
// is >= Lk, every chunk holding a score > Lk is among them, and a score == T in any other chunk sorts behind k scores
// that are >= T with lower columns.  So one CTA per row
//   1. reads the row of chunk maxima (n_chunks floats) into registers and selects its k largest exactly with the
//      same bound -> compaction -> all-pairs ranking scheme as the register kernel (columns = chunk ids);
//   2. reads ONLY those k chunks of the score row (128 B each), keeps the scores >= Lk and ranks them exactly by
//      (score desc, column asc); the k best leave in ascending column order.
// Per row that is 4 * I / 32 + 128 * k bytes instead of 4 * I (median k is 2-4).  Rows that do not qualify (k above
// PRUNE_KMAX or more than n_chunks / PRUNE_RATIO, a NaN maximum, crowded ties) are appended to a device list that
// the whole-row / segmented kernels process afterwards: every row is emitted by exactly one path, bit-identically.
constexpr int PRUNE_KMAX = 64;
constexpr int PRUNE_RATIO = 4;   // diffmm_b200/recommend.py PRUNE_RATIO selects this path by the same ratio
constexpr int PRUNE_CAND = 512;

struct PruneArgs {
  const float* scores;
  int64_t ld;
  const float* cmax;
  int64_t ld_cmax;
  int n_chunks, n_cols;
  int64_t n_rows;
  const int64_t* out_ptr;
  int64_t row_base;
  int32_t* out_users;
  int32_t* out_items;
  int32_t* status;
  const int32_t* order;
  int32_t* left_count;
  int32_t* left_rows;
};

// The k rule of the pruned path (block-uniform)
__host__ __device__ __forceinline__ int prune_kmax(int n_chunks) {
  const int nw = n_chunks <= 64 * 4 * TOPK_V4 ? 2 : (n_chunks <= 256 * 4 * TOPK_V4 ? 8 : 16);
  return PRUNE_KMAX < 32 * nw ? PRUNE_KMAX : 32 * nw;
}
__host__ __device__ __forceinline__ bool prune_k_ok(int64_t k, int n_chunks, int64_t n_cols) {
  return k <= prune_kmax(n_chunks) && k * PRUNE_RATIO <= n_chunks && k <= n_cols;
}

struct alignas(16) PruneSmem {
  uint32_t key[PRUNE_CAND];
  int col[PRUNE_CAND];
  int sel[PRUNE_CAND];
  uint32_t red[32];
  int ncand, nsel, ncand2;
  uint32_t lk;
};

__device__ __forceinline__ float key_to_float(uint32_t L) {   // inverse of order_key (L == 0: below every score)
  return (L == 0u) ? __uint_as_float(0xFF800000u) : __uint_as_float((L & 0x80000000u) ? (L ^ 0x80000000u) : ~L);
}

template <int NT>
__global__ void __launch_bounds__(NT) topk_pruned_kernel(const PruneArgs a) {
  __shared__ PruneSmem sm;
  constexpr int NW = NT / 32;
  if ((int64_t)blockIdx.x >= a.n_rows) return;
  const int64_t r = a.order ? (int64_t)a.order[blockIdx.x] : (int64_t)blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n_chunks = a.n_chunks;

  // 1a. the row of chunk maxima -> registers (issued before anything depends on out_ptr)
  const float* crow = a.cmax + r * a.ld_cmax;
  const int n4 = n_chunks >> 2;
  const float4* crow4 = reinterpret_cast<const float4*>(crow);
  float4 v[TOPK_V4];
#pragma unroll
  for (int j = 0; j < TOPK_V4; ++j) {
    v[j] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (tid + NT * j < n4) v[j] = __ldg(crow4 + tid + NT * j);
  }
  const int tail_col = (n4 << 2) + tid;
  const bool has_tail = tid < (n_chunks & 3);
  float tail_v = 0.f;
  if (has_tail) tail_v = __ldg(crow + tail_col);

  const int64_t o0 = a.out_ptr[r];
  const int k = (int)(a.out_ptr[r + 1] - o0);
  if (k <= 0) return;
  auto defer = [&]() {
    if (tid == 0) a.left_rows[atomicAdd(a.left_count, 1)] = (int32_t)r;
  };
  if (!prune_k_ok(k, n_chunks, a.n_cols)) {   // block-uniform
    defer();
    return;
  }
  const float NEG_INF = __uint_as_float(0xFF800000u);
  const int jfull = n4 / NT, jrem = n4 - jfull * NT;
  float pmax[TOPK_V4];
  float tmaxf = has_tail ? fmax_nan(tail_v, NEG_INF) : NEG_INF;
#pragma unroll
  for (int j = 0; j < TOPK_V4; ++j) {
    pmax[j] = NEG_INF;
    if (j < jfull || (j == jfull && tid < jrem)) {
      pmax[j] = fmax_nan(fmax_nan(v[j].x, v[j].y), fmax_nan(v[j].z, v[j].w));
      tmaxf = fmax_nan(tmaxf, pmax[j]);
    }
  }
  const uint32_t tmax = (tmaxf == NEG_INF) ? 0u : order_key(tmaxf);

  // 1b. lower bound L of the k-th largest chunk maximum: this warp's q-th largest thread maximum, q = ceil(k / warps)
  const int q = (k + NW - 1) / NW;
  uint32_t wq;
  {
    uint32_t sv = tmax;
#pragma unroll
    for (int k2 = 2; k2 <= 32; k2 <<= 1) {
#pragma unroll
      for (int j = k2 >> 1; j > 0; j >>= 1) {
        const uint32_t other = __shfl_xor_sync(0xffffffffu, sv, j);
        const bool desc = (lane & k2) == 0;
        const bool lower = (lane & j) == 0;
        sv = (lower == desc) ? max(sv, other) : min(sv, other);
      }
    }
    wq = __shfl_sync(0xffffffffu, sv, q - 1);
  }
  if (lane == 0) sm.red[wid] = wq;
  if (tid == 0) {
    sm.ncand = 0;
    sm.nsel = 0;
    sm.ncand2 = 0;
    sm.lk = 0xFFFFFFFFu;
  }
  if (__syncthreads_or(tmaxf != tmaxf)) {   // a NaN score somewhere in the row: exact whole-row path
    defer();
    return;
  }
  uint32_t L = 0xFFFFFFFFu;
#pragma unroll
  for (int i = 0; i < NW; ++i) L = min(L, sm.red[i]);
  const float Lf = key_to_float(L);

  // 1c. chunk candidates (maximum >= L) -> shared memory, one atomic per warp per hit group
  auto push = [&](int* counter, bool c, float x, int col) {
    const uint32_t bal = __ballot_sync(0xffffffffu, c);
    if (bal) {
      int base = 0;
      if (lane == 0) base = atomicAdd(counter, __popc(bal));
      base = __shfl_sync(0xffffffffu, base, 0);
      const int pos = base + __popc(bal & ((1u << lane) - 1u));
      if (c && pos < PRUNE_CAND) {
        sm.key[pos] = order_key(x);
        sm.col[pos] = col;
      }
    }
  };
#pragma unroll
  for (int j = 0; j < TOPK_V4; ++j) {
    if (j > jfull) break;                      // block-uniform
    const bool have = j < jfull || tid < jrem;
    const bool open = have && !(pmax[j] < Lf);
    if (__any_sync(0xffffffffu, open)) {
      const float xs[4] = {v[j].x, v[j].y, v[j].z, v[j].w};
#pragma unroll
      for (int e = 0; e < 4; ++e) push(&sm.ncand, open && !(xs[e] < Lf), xs[e], 4 * (tid + NT * j) + e);
    }
  }
  if (n_chunks & 3) push(&sm.ncand, has_tail && !(tail_v < Lf), tail_v, tail_col);
  __syncthreads();
  const int m = sm.ncand;
  if (m > PRUNE_CAND || m < k) {
    defer();
    return;
  }
  // 1d. the k best chunks by (maximum desc, chunk asc); Lk = the smallest maximum among them
  for (int c = tid; c < m; c += NT) {
    const uint32_t my_key = sm.key[c];
    const int my_col = sm.col[c];
    int before = 0;
    if (m > k) {
      for (int j = 0; j < m; ++j) {
        const uint32_t kj = sm.key[j];
        const int cj = sm.col[j];
        before += (kj > my_key || (kj == my_key && cj < my_col)) ? 1 : 0;
      }
    }
    if (before < k) {
      sm.sel[atomicAdd(&sm.nsel, 1)] = my_col;
      atomicMin(&sm.lk, my_key);
    }
  }
  __syncthreads();   // sm.key / sm.col are free again from here on
  const float Lkf = key_to_float(sm.lk);

  // 2a. the k selected chunks of the score row: one coalesced 128-byte read each, scores >= Lk are the candidates
  const float* row = a.scores + r * a.ld;
  constexpr int GB = 8;                       // chunk reads in flight per warp (a row with k = 64 is 4 rounds, not 32)
  for (int i0 = wid; i0 < k; i0 += NW * GB) {
    float xs[GB];
    int cols[GB];
#pragma unroll
    for (int t = 0; t < GB; ++t) {
      const int i = i0 + t * NW;
      cols[t] = i < k ? sm.sel[i] * 32 + lane : 0x7FFFFFFF;
      xs[t] = cols[t] < a.n_cols ? __ldg(row + cols[t]) : NEG_INF;
    }
#pragma unroll
    for (int t = 0; t < GB; ++t) {
      if (i0 + t * NW >= k) break;            // warp-uniform
      push(&sm.ncand2, cols[t] < a.n_cols && !(xs[t] < Lkf), xs[t], cols[t]);
    }
  }
  __syncthreads();
  const int m2 = sm.ncand2;          // >= k: every selected chunk holds its maximum >= Lk
  if (m2 > PRUNE_CAND || m2 < k) {   // crowded ties at the bound (or a maximum that matches no score: impossible by contract)
    defer();
    return;
  }
  // 2b. exact rank among the candidates by (score desc, column asc); the k best leave in ascending column order
  for (int c = tid; c < m2; c += NT) {
    const uint32_t my_key = sm.key[c];
    const int my_col = sm.col[c];
    int before = 0;
    if (m2 > k) {
      for (int j = 0; j < m2; ++j) {
        const uint32_t kj = sm.key[j];
        const int cj = sm.col[j];
        before += (kj > my_key || (kj == my_key && cj < my_col)) ? 1 : 0;
      }
    }
    sm.sel[c] = before < k ? my_col : 0x7FFFFFFF;
  }
  __syncthreads();
  const int32_t user = (int32_t)(a.row_base + r);
  for (int c = tid; c < m2; c += NT) {
    const int my_col = sm.sel[c];
    if (my_col == 0x7FFFFFFF) continue;
    int pos = 0;
    for (int j = 0; j < m2; ++j) pos += (sm.sel[j] < my_col) ? 1 : 0;
    a.out_items[o0 + pos] = my_col;
    if (a.out_users) a.out_users[o0 + pos] = user;
  }
}

// The rows the pruned kernel deferred (k above its limits: the 1 % of users with hundreds of interactions; NaN maxima;
// crowded ties): a small persistent grid walks the device-built list.  A row without NaN whose k chunks are at most half
// of the row takes the same two-level route with the exact radix select instead of the all-pairs ranking:
//   A. top-k of the row's chunk maxima (keys staged in shared memory when they fit) -> k chunk ids, ascending, into the
//      row's slot of `chunk_list`;
//   B. top-k of the k * 32 scores of those chunks (a virtual row: index i -> column chunk_list[i / 32] * 32 + i % 32, so
//      index order is column order; columns >= n_cols get key 0, below every real score) -> the row's edges.
// That is 4 * n_chunks + 128 * k bytes per row instead of several passes over 4 * n_cols (a 500 000-column row with
// k = 600: 140 KB instead of 8 MB).  Everything else takes the exact whole-row generic path.
__global__ void __launch_bounds__(256) topk_deferred_kernel(const float* __restrict__ scores, int64_t ld, int n_cols,
                                                            const float* __restrict__ cmax, int64_t ld_cmax, int n_chunks,
                                                            const int64_t* __restrict__ out_ptr, int64_t row_base,
                                                            int32_t* __restrict__ out_users, int32_t* __restrict__ out_items,
                                                            int32_t* __restrict__ status, const int32_t* __restrict__ rows,
                                                            const int32_t* __restrict__ live,
                                                            int32_t* __restrict__ chunk_list, int smem_keys) {
  extern __shared__ uint32_t s_keys[];       // smem_keys staged keys
  __shared__ TopkSmem<256> sm;
  const int tid = threadIdx.x;
  const int n = *live;
  const int64_t e0 = out_ptr[0];
  for (int slot = blockIdx.x; slot < n; slot += gridDim.x) {
    const int64_t r = rows[slot];
    const int64_t o0 = out_ptr[r];
    int k = (int)(out_ptr[r + 1] - o0);
    if (k > n_cols) {
      if (status && tid == 0) atomicOr(status, 1);
      k = n_cols;
    }
    if (k <= 0) continue;                     // block-uniform
    const float* row = scores + r * ld;
    const float* crow = cmax + r * ld_cmax;
    bool two_level = (int64_t)k * 2 <= n_chunks;
    if (two_level) {
      bool nan = false;
      for (int i = tid; i < n_chunks; i += 256) {
        const float c = __ldg(crow + i);
        nan |= c != c;
      }
      two_level = !__syncthreads_or(nan);
    }
    if (two_level) {
      int32_t* list = chunk_list + (o0 - e0);
      // A. the k chunks with the largest maxima
      if (n_chunks <= smem_keys) {
        uint32_t kmin = 0xFFFFFFFFu, kmax = 0u;
        for (int i = tid; i < n_chunks; i += 256) {
          const uint32_t q = order_key(__ldg(crow + i));
          s_keys[i] = q;
          kmin = min(kmin, q);
          kmax = max(kmax, q);
        }
        topk_select_emit<256>(sm, [&](int i) -> uint32_t { return s_keys[i]; }, [](int i) -> int { return i; }, n_chunks, k,
                              true, kmin, kmax, 0, 0, nullptr, list);
      } else {
        topk_select_emit<256>(sm, [&](int i) -> uint32_t { return order_key(__ldg(crow + i)); }, [](int i) -> int { return i; },
                              n_chunks, k, false, 0u, 0u, 0, 0, nullptr, list);
      }
      __syncthreads();                        // the chunk list (global) is complete and visible to the block
      // B. the k best of the k * 32 scores of those chunks
      const int nv = k * 32;
      auto vcol = [&](int i) -> int { return list[i >> 5] * 32 + (i & 31); };
      auto vkey = [&](int i) -> uint32_t {
        const int c = vcol(i);
        return c < n_cols ? order_key(__ldg(row + c)) : 0u;
      };
      if (nv <= smem_keys) {
        uint32_t kmin = 0xFFFFFFFFu, kmax = 0u;
#pragma unroll 4
        for (int i = tid; i < nv; i += 256) {
          const uint32_t q = vkey(i);
          s_keys[i] = q;
          kmin = min(kmin, q);
          kmax = max(kmax, q);
        }
        topk_select_emit<256>(sm, [&](int i) -> uint32_t { return s_keys[i]; }, vcol, nv, k, true, kmin, kmax, o0,
                              (int32_t)(row_base + r), out_users, out_items);
      } else {
        topk_select_emit<256>(sm, vkey, vcol, nv, k, false, 0u, 0u, o0, (int32_t)(row_base + r), out_users, out_items);
      }
    } else {
      topk_row_generic<256, false>(sm, nullptr, row, n_cols, k, o0, (int32_t)(row_base + r), out_users, out_items);
    }
    __syncthreads();
  }
}

SegCfg make_seg(int64_t n_cols) {
  SegCfg sg{0, 0, 0, 0};
  if (n_cols > TOPK_SEG_COLS) {
    sg.S = (int)dmm_ceil_div(n_cols, TOPK_SEG_COLS);
    sg.seg_cols = (int)((dmm_ceil_div(n_cols, sg.S) + 3) / 4 * 4);
    sg.last_len = (int)(n_cols - (int64_t)(sg.S - 1) * sg.seg_cols);
    if (sg.last_len <= 0) sg.S = 0;          // cannot happen for n_cols > 8192; guards the arithmetic
  }
  return sg;
}

}  // namespace

extern "C" int64_t dmm_topk_workspace_bytes(int64_t n_cols, int64_t n_edges) {
  const SegCfg sg = make_seg(n_cols);
  return sg.S > 0 ? (int64_t)sg.S * (n_edges > 0 ? n_edges : 0) * (int64_t)sizeof(int32_t) : 0;
}

// Whole-row / segmented dispatch shared by dmm_topk_edges and the leftover pass of dmm_topk_edges_pruned.
// `live` (device int32, optional): number of valid entries of `order` when that list was built on the device.
static int topk_dispatch(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, int64_t n_cols,
                         const int64_t* out_ptr, int64_t row_base, int32_t* out_users, int32_t* out_items, int32_t* status,
                         const int32_t* order, const int32_t* live, void* workspace, int64_t workspace_bytes,
                         int64_t n_edges, cudaStream_t st) {
  constexpr int PER_THREAD = 4 * TOPK_V4;
  static const bool force_generic = getenv("DMM_TOPK_GENERIC") != nullptr;   // test hook: exercise the generic kernels
  static const bool seg_ok = []() { const char* e = getenv("DMM_TOPK_SEG"); return !(e && e[0] == '0'); }();   // A/B switch

  // wide rows: segment pass + merge for the rows that qualify, whole-row kernels for the rest (see SegCfg)
  SegCfg sg = make_seg(n_cols);
  const bool rows_aligned = (reinterpret_cast<uintptr_t>(scores) & 15u) == 0 && ld % 4 == 0;
  const bool segmented = seg_ok && !force_generic && sg.S > 0 && rows_aligned && workspace != nullptr && n_edges >= 0 &&
                         workspace_bytes >= dmm_topk_workspace_bytes(n_cols, n_edges) && n_rows * (int64_t)sg.S < (1LL << 31);
  if (segmented) {
    sg.mode = 1;
    launch_reg<256>(scores, ld, n_rows, (int)n_cols, out_ptr, row_base, nullptr, nullptr, status, order, sg, (int32_t*)workspace,
                    live, st);
    DMM_LAUNCH_CHECK();
    topk_merge_kernel<<<(unsigned)n_rows, 128, 0, st>>>(scores, ld, n_rows, out_ptr, row_base, out_users, out_items, order, sg,
                                                       (const int32_t*)workspace, live);
    DMM_LAUNCH_CHECK();
    // the few rows the segment pass skipped: the 256-thread generic kernel (8 CTAs per SM; a 1024-thread CTA per row
    // that only reads two offsets and leaves would cost more in launch waves than the rows it really processes)
    sg.mode = 2;
    topk_edges_kernel<false><<<(unsigned)n_rows, 256, 0, st>>>(scores, ld, n_rows, (int)n_cols, out_ptr, row_base, out_users,
                                                              out_items, status, order, sg, live);
    DMM_LAUNCH_CHECK();
    return DMM_OK;
  }
  sg = SegCfg{0, 0, 0, 0};
  if (force_generic) {
    // fall through to the generic kernels below
  } else if (n_cols <= 256 * PER_THREAD) {
    launch_reg<256>(scores, ld, n_rows, (int)n_cols, out_ptr, row_base, out_users, out_items, status, order, sg, nullptr, live, st);
  } else if (n_cols <= 512 * PER_THREAD) {
    launch_reg<512>(scores, ld, n_rows, (int)n_cols, out_ptr, row_base, out_users, out_items, status, order, sg, nullptr, live, st);
  } else if (n_cols <= 1024 * PER_THREAD) {
    launch_reg<1024>(scores, ld, n_rows, (int)n_cols, out_ptr, row_base, out_users, out_items, status, order, sg, nullptr, live, st);
  }
  if (force_generic || n_cols > 1024 * PER_THREAD) {
    const size_t smem = (size_t)n_cols * sizeof(uint32_t);
    // static shared memory of the kernel (buckets, candidates, scratch) is ~18 KB
    const size_t cap = (size_t)ctx->max_smem_optin > 40960 ? (size_t)ctx->max_smem_optin - 20480 : 0;
    if (smem <= cap) {
      static DmmPerDeviceOnce smem_once;
      if (smem > 24 * 1024 && smem_once.need(ctx)) {
        DMM_CUDA(cudaFuncSetAttribute(topk_edges_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)cap));
        smem_once.mark(ctx);
      }
      topk_edges_kernel<true><<<(unsigned)n_rows, 256, smem, st>>>(scores, ld, n_rows, (int)n_cols, out_ptr, row_base,
                                                                  out_users, out_items, status, order, sg, live);
    } else {
      topk_edges_kernel<false><<<(unsigned)n_rows, 256, 0, st>>>(scores, ld, n_rows, (int)n_cols, out_ptr, row_base,
                                                                out_users, out_items, status, order, sg, live);
    }
  }
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_topk_edges(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, int64_t n_cols,
                              const int64_t* out_ptr, int64_t row_base, int32_t* out_users, int32_t* out_items,
                              int32_t* status, const int32_t* order, void* workspace, int64_t workspace_bytes,
                              int64_t n_edges, void* stream) {
  DMM_CHECK_ARG(ctx && scores && out_ptr && out_items, "dmm_topk_edges: null argument");
  DMM_CHECK_ARG(n_cols > 0 && n_cols < (1LL << 31) && ld >= n_cols, "dmm_topk_edges: bad shape n_cols=%lld ld=%lld",
                (long long)n_cols, (long long)ld);
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31), "dmm_topk_edges: bad n_rows");
  if (n_rows == 0) return DMM_OK;
  return topk_dispatch(ctx, scores, ld, n_rows, n_cols, out_ptr, row_base, out_users, out_items, status, order, nullptr,
                       workspace, workspace_bytes, n_edges, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------ pruned top-k
namespace {
inline size_t prune_align(size_t x) { return (x + 255) & ~(size_t)255; }
inline size_t prune_head_bytes(int64_t n_rows) { return 256 + prune_align((size_t)(n_rows > 0 ? n_rows : 1) * sizeof(int32_t)); }
}  // namespace

extern "C" int64_t dmm_topk_pruned_workspace_bytes(int64_t n_rows, int64_t n_cols, int64_t n_edges) {
  // [deferred-row count | deferred-row list | chunk lists of the deferred rows (one slot per emitted entry) | workspace of
  //  the segmented kernels (only used when pruning is switched off)]
  return (int64_t)prune_head_bytes(n_rows) + (int64_t)prune_align((size_t)(n_edges > 0 ? n_edges : 1) * sizeof(int32_t)) +
         dmm_topk_workspace_bytes(n_cols, n_edges);
}

extern "C" int dmm_topk_edges_pruned(dmm_ctx* ctx, const float* scores, int64_t ld, int64_t n_rows, int64_t n_cols,
                                     const float* cmax, int64_t ld_cmax, const int64_t* out_ptr, int64_t row_base,
                                     int32_t* out_users, int32_t* out_items, int32_t* status, const int32_t* order,
                                     void* workspace, int64_t workspace_bytes, int64_t n_edges, void* stream) {
  DMM_CHECK_ARG(ctx && scores && cmax && out_ptr && out_items && workspace, "dmm_topk_edges_pruned: null argument");
  DMM_CHECK_ARG(n_cols > 0 && n_cols < (1LL << 31) && ld >= n_cols, "dmm_topk_edges_pruned: bad shape n_cols=%lld ld=%lld",
                (long long)n_cols, (long long)ld);
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31) && n_edges >= 0, "dmm_topk_edges_pruned: bad n_rows / n_edges");
  const int64_t n_chunks = dmm_ceil_div(n_cols, 32);
  DMM_CHECK_ARG(ld_cmax >= n_chunks && ld_cmax % 4 == 0 && (reinterpret_cast<uintptr_t>(cmax) & 15u) == 0,
                "dmm_topk_edges_pruned: cmax rows must be 16-byte aligned with ld_cmax %% 4 == 0 and >= ceil(n_cols / 32)");
  DMM_CHECK_ARG(workspace_bytes >= dmm_topk_pruned_workspace_bytes(n_rows, n_cols, n_edges),
                "dmm_topk_edges_pruned: workspace smaller than dmm_topk_pruned_workspace_bytes");
  if (n_rows == 0) return DMM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const size_t list_bytes = prune_align((size_t)(n_edges > 0 ? n_edges : 1) * sizeof(int32_t));
  int32_t* const chunk_list = (int32_t*)((uint8_t*)workspace + prune_head_bytes(n_rows));
  uint8_t* const seg_ws = (uint8_t*)workspace + prune_head_bytes(n_rows) + list_bytes;
  const int64_t seg_ws_bytes = workspace_bytes - (int64_t)prune_head_bytes(n_rows) - (int64_t)list_bytes;
  static const bool prune_ok = []() { const char* e = getenv("DMM_TOPK_PRUNE"); return !(e && e[0] == '0'); }();   // A/B switch
  if (!prune_ok || n_chunks > 512 * 4 * TOPK_V4 || n_chunks < 8)
    return topk_dispatch(ctx, scores, ld, n_rows, n_cols, out_ptr, row_base, out_users, out_items, status, order, nullptr,
                         seg_ws, seg_ws_bytes, n_edges, st);
  int32_t* left_count = (int32_t*)workspace;
  int32_t* left_rows = (int32_t*)((uint8_t*)workspace + 256);
  DMM_CUDA(cudaMemsetAsync(left_count, 0, sizeof(int32_t), st));
  // 1. chunk maxima -> k chunks -> exact rank, one small CTA per row; rows it cannot take go to the device list
  const PruneArgs a{scores, ld, cmax, ld_cmax, (int)n_chunks, (int)n_cols, n_rows, out_ptr, row_base, out_users, out_items,
                    status, order, left_count, left_rows};
  if (n_chunks <= 64 * 4 * TOPK_V4) topk_pruned_kernel<64><<<(unsigned)n_rows, 64, 0, st>>>(a);
  else if (n_chunks <= 256 * 4 * TOPK_V4) topk_pruned_kernel<256><<<(unsigned)n_rows, 256, 0, st>>>(a);
  else topk_pruned_kernel<512><<<(unsigned)n_rows, 512, 0, st>>>(a);
  DMM_LAUNCH_CHECK();
  // 2. the deferred rows: persistent grid, two-level radix select (keys staged in up to 80 KB of shared memory)
  constexpr int SMEM_KEYS = 20480;
  static DmmPerDeviceOnce attr_once;
  if (attr_once.need(ctx)) {
    DMM_CUDA(cudaFuncSetAttribute(topk_deferred_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_KEYS * 4));
    attr_once.mark(ctx);
  }
  topk_deferred_kernel<<<(unsigned)(ctx->num_sms * 2), 256, SMEM_KEYS * 4, st>>>(
      scores, ld, (int)n_cols, cmax, ld_cmax, (int)n_chunks, out_ptr, row_base, out_users, out_items, status, left_rows,
      left_count, chunk_list, SMEM_KEYS);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
