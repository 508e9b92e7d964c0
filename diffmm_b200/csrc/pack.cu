// Operand staging kernels for the Denoise path: fp32 -> split-bf16 packing (optionally transposed),
// CSR user rows -> dense operand tiles, time-embedding columns, q_sample.  All HBM-bound,
// vectorised where alignment allows; grids are sized from the data, block = 256 threads.
#include "common.cuh"

namespace {

// ------------------------------------------------------------------ fp32 -> bf16 hi/lo (no transpose)
// one thread per 8 destination columns: two float4 loads, one 16-byte store per part (zero pad beyond cols);
// VEC = false is the scalar-load variant for sources whose rows are not 16-byte aligned
template <bool VEC>
__global__ void __launch_bounds__(256) pack_rows_kernel(const float* __restrict__ src, int64_t rows, int64_t cols,
                                                        int64_t ld_src, uint16_t* __restrict__ hi,
                                                        uint16_t* __restrict__ lo, int64_t ld_dst) {
  const int64_t n8 = ld_dst >> 3;                      // ld_dst % 8 == 0 (checked by the host)
  const int64_t total = rows * n8;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / n8, c = (t - r * n8) << 3;
    const float* s = src + r * ld_src + c;
    float v[8];
    if (VEC && c + 8 <= cols) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(s)), b4 = __ldg(reinterpret_cast<const float4*>(s) + 1);
      v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b4.x; v[5] = b4.y; v[6] = b4.z; v[7] = b4.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] = c + j < cols ? __ldg(s + j) : 0.f;
    }
    uint32_t ph[4], pl[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint16_t h0, l0, h1, l1;
      dmm_split_bf16(v[2 * j], h0, l0);
      dmm_split_bf16(v[2 * j + 1], h1, l1);
      ph[j] = (uint32_t)h0 | ((uint32_t)h1 << 16);
      pl[j] = (uint32_t)l0 | ((uint32_t)l1 << 16);
    }
    *reinterpret_cast<uint4*>(hi + r * ld_dst + c) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
    if (lo) *reinterpret_cast<uint4*>(lo + r * ld_dst + c) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
  }
}

// ------------------------------------------------------------------ fp32 -> bf16 hi/lo, transposed
// 64 source rows x 64 source columns per CTA through a padded fp32 tile in shared memory: float4 loads (256-byte row
// segments), and every thread converts one column run of 8 source rows into ONE 16-byte store per part (128-byte lines
// per destination row).  dst[c, r]: dst rows = src cols (only c < cols exist), dst cols = src rows, zero padded to ld_dst.
// nat_hi / nat_lo (optional): the same tile also leaves in the source orientation ([rows, ld_nat], zero padded to
// ld_nat), so a weight that is needed both ways (forward and input-gradient contraction; gather table and operand) is
// read from HBM once.
template <bool VEC>
__global__ void __launch_bounds__(256) pack_transpose_kernel(const float* __restrict__ src, int64_t rows, int64_t cols,
                                                             int64_t ld_src, uint16_t* __restrict__ hi,
                                                             uint16_t* __restrict__ lo, int64_t ld_dst,
                                                             uint16_t* __restrict__ nat_hi, uint16_t* __restrict__ nat_lo,
                                                             int64_t ld_nat) {
  __shared__ float tile[64][65];
  const int64_t r0 = (int64_t)blockIdx.y * 64, c0 = (int64_t)blockIdx.x * 64;
  const int tid = threadIdx.x;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int idx = tid + 256 * k;            // 64 rows x 16 float4
    const int rr = idx >> 4, q = idx & 15;
    const int64_t r = r0 + rr, c = c0 + 4 * q;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (r < rows) {
      if (VEC && c + 4 <= cols) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(src + r * ld_src + c));
        v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i) v[i] = c + i < cols ? __ldg(src + r * ld_src + c + i) : 0.f;
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) tile[rr][4 * q + i] = v[i];
  }
  __syncthreads();
#pragma unroll
  for (int k = 0; k < 2; ++k) {
    const int idx = tid + 256 * k;            // 64 destination rows x 8 pieces of 8 source rows
    const int cc = idx >> 3, pc = idx & 7;
    const int64_t c = c0 + cc, r = r0 + 8 * pc;
    if (c < cols && r < ld_dst) {             // ld_dst % 8 == 0: a piece that starts below ld_dst lies inside the row
      uint32_t ph[4], pl[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint16_t h0, l0, h1, l1;
        dmm_split_bf16(tile[8 * pc + 2 * j][cc], h0, l0);
        dmm_split_bf16(tile[8 * pc + 2 * j + 1][cc], h1, l1);
        ph[j] = (uint32_t)h0 | ((uint32_t)h1 << 16);
        pl[j] = (uint32_t)l0 | ((uint32_t)l1 << 16);
      }
      *reinterpret_cast<uint4*>(hi + c * ld_dst + r) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
      if (lo) *reinterpret_cast<uint4*>(lo + c * ld_dst + r) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
    }
  }
  if (nat_hi) {
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int idx = tid + 256 * k;          // 64 source rows x 8 pieces of 8 source columns
      const int rr = idx >> 3, pc = idx & 7;
      const int64_t r = r0 + rr, c = c0 + 8 * pc;
      if (r < rows && c < ld_nat) {           // ld_nat % 8 == 0; columns past `cols` are zero in the tile
        uint32_t ph[4], pl[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          uint16_t h0, l0, h1, l1;
          dmm_split_bf16(tile[rr][8 * pc + 2 * j], h0, l0);
          dmm_split_bf16(tile[rr][8 * pc + 2 * j + 1], h1, l1);
          ph[j] = (uint32_t)h0 | ((uint32_t)h1 << 16);
          pl[j] = (uint32_t)l0 | ((uint32_t)l1 << 16);
        }
        *reinterpret_cast<uint4*>(nat_hi + r * ld_nat + c) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
        if (nat_lo) *reinterpret_cast<uint4*>(nat_lo + r * ld_nat + c) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
      }
    }
  }
}

// ------------------------------------------------------------------ CSR rows -> dense 0/1 tiles
// One CTA per output row: zero fill with 16-byte stores (scalar head/tail where the row is not
// 16-byte aligned), then the row's interactions are scattered as 1.0.  HBM-bound: one write of the tile.
template <typename T>
__device__ __forceinline__ void zero_row(T* __restrict__ p, int64_t n) {
  constexpr int PER = 16 / (int)sizeof(T);
  const uintptr_t addr = reinterpret_cast<uintptr_t>(p);
  int64_t head = ((16 - (addr & 15)) & 15) / (int64_t)sizeof(T);
  if (head > n) head = n;
  for (int64_t c = threadIdx.x; c < head; c += blockDim.x) p[c] = T(0);
  const int64_t nvec = (n - head) / PER;
  uint4* v = reinterpret_cast<uint4*>(p + head);
  const uint4 z = make_uint4(0u, 0u, 0u, 0u);
  for (int64_t c = threadIdx.x; c < nvec; c += blockDim.x) v[c] = z;
  for (int64_t c = head + nvec * PER + threadIdx.x; c < n; c += blockDim.x) p[c] = T(0);
}

__global__ void __launch_bounds__(256) csr_rows_dense_kernel(const int64_t* __restrict__ indptr,
                                                             const int32_t* __restrict__ indices,
                                                             const int64_t* __restrict__ row_ids, int64_t row0,
                                                             int64_t n_rows, int64_t n_cols, float* __restrict__ x,
                                                             int64_t ld_x, uint16_t* __restrict__ a, int64_t ld_a) {
  for (int64_t r = blockIdx.x; r < n_rows; r += gridDim.x) {
    if (x) zero_row<float>(x + r * ld_x, n_cols);
    if (a) zero_row<uint16_t>(a + r * ld_a, n_cols);
    __syncthreads();   // the scatter below must land after this CTA's zero stores
    const int64_t u = row_ids ? row_ids[r] : row0 + r;
    const int64_t b = indptr[u], e = indptr[u + 1];
    for (int64_t j = b + threadIdx.x; j < e; j += blockDim.x) {
      const int32_t c = indices[j];
      if (c >= 0 && c < n_cols) {
        if (x) x[r * ld_x + c] = 1.f;
        if (a) a[r * ld_a + c] = 0x3F80;  // bf16(1.0)
      }
    }
    __syncthreads();
  }
}

// ------------------------------------------------------------------ time embedding columns
__global__ void __launch_bounds__(256) time_embedding_kernel(const int64_t* __restrict__ t, int64_t t_all,
                                                             int64_t n_rows, int d, const float* __restrict__ w,
                                                             const float* __restrict__ b, uint16_t* __restrict__ a_hi,
                                                             uint16_t* __restrict__ a_lo, int64_t ld_a, int64_t col0,
                                                             float* __restrict__ temb) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (r >= n_rows) return;
  const float ts = (float)(t ? t[r] : t_all);
  const int half = d / 2;
  float e[64];
  // Model.py:196-201: freqs = exp(-ln(1e4) * j / half); [cos, sin]; zero pad if d is odd
  for (int j = 0; j < half; ++j) {
    const float f = expf(-logf(10000.f) * (float)j / (float)half);
    const float ang = ts * f;
    e[j] = cosf(ang);
    e[half + j] = sinf(ang);
  }
  if (d & 1) e[d - 1] = 0.f;
  for (int o = 0; o < d; ++o) {
    float acc = b[o];
    for (int j = 0; j < d; ++j) acc = fmaf(e[j], w[o * d + j], acc);
    if (temb) temb[r * d + o] = acc;
    if (a_hi) {
      uint16_t h, l;
      dmm_split_bf16(acc, h, l);
      a_hi[r * ld_a + col0 + o] = h;
      if (a_lo) a_lo[r * ld_a + col0 + o] = l;
    }
  }
}

// ------------------------------------------------------------------ q_sample
__global__ void __launch_bounds__(256) q_sample_kernel(const float* __restrict__ x0, int64_t ld_x0,
                                                       const float* __restrict__ noise, int64_t ld_n,
                                                       const float* __restrict__ ca, const float* __restrict__ cb,
                                                       int64_t n_cols, int mode, float* __restrict__ xt, int64_t ld_x,
                                                       uint16_t* __restrict__ a_hi, uint16_t* __restrict__ a_lo,
                                                       int64_t ld_a) {
  // one block per row
  const int64_t r = blockIdx.x;
  const float* x = x0 + r * ld_x0;
  const float* g = noise + r * ld_n;
  __shared__ float red[8];
  __shared__ float s_inv;
  float inv = 1.f;
  if (mode == 1) {
    float ss = 0.f;
    for (int64_t c = threadIdx.x; c < n_cols; c += blockDim.x) {
      const float v = __ldg(g + c);
      ss = fmaf(v, v, ss);
    }
    ss = dmm_warp_sum(ss);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = ss;
    __syncthreads();
    if (threadIdx.x == 0) {
      float tot = 0.f;
      for (int i = 0; i < (int)(blockDim.x >> 5); ++i) tot += red[i];
      s_inv = 1.f / fmaxf(sqrtf(tot), 1e-12f);
    }
    __syncthreads();
    inv = s_inv;
  }
  const float a = ca[r], b = cb[r];
  for (int64_t c = threadIdx.x; c < n_cols; c += blockDim.x) {
    const float xv = __ldg(x + c);
    float nv = __ldg(g + c);
    if (mode == 1) {
      const float sg = (xv > 0.f) ? 1.f : ((xv < 0.f) ? -1.f : 0.f);
      nv = sg * (nv * inv);
    }
    const float v = a * xv + b * nv;
    if (xt) xt[r * ld_x + c] = v;
    if (a_hi) {
      uint16_t h, l;
      dmm_split_bf16(v, h, l);
      a_hi[r * ld_a + c] = h;
      if (a_lo) a_lo[r * ld_a + c] = l;
    }
  }
}

// ------------------------------------------------------------------ time embedding folded into the bias
// In the reverse chain every row of a step shares the timestep (Model.py:319), so the 10 time-embedding
// columns of cat([x_t, temb]) (Model.py:202-203,212) contribute the same vector to every row:
//   bias_eff[h] = b[h] + sum_j W[h, col0 + j] * temb_j(t)          (fp32, exact weights)
__global__ void __launch_bounds__(256) time_bias_kernel(int64_t t0, int d, const float* __restrict__ emb_w,
                                                        const float* __restrict__ emb_b, const float* __restrict__ w,
                                                        int64_t ld_w, int64_t col0, const float* __restrict__ b,
                                                        int64_t n_out, float* __restrict__ bias_eff) {
  __shared__ float temb[64];
  if (threadIdx.x < d) {
    const int o = threadIdx.x;
    const int half = d / 2;
    const float ts = (float)(t0 + blockIdx.y);   // one timestep per grid row
    float acc = emb_b[o];
    for (int j = 0; j < d; ++j) {
      float e = 0.f;
      if (j < half) {
        e = cosf(ts * expf(-logf(10000.f) * (float)j / (float)half));
      } else if (j < 2 * half) {
        e = sinf(ts * expf(-logf(10000.f) * (float)(j - half) / (float)half));
      }
      acc = fmaf(e, emb_w[o * d + j], acc);
    }
    temb[o] = acc;
  }
  __syncthreads();
  const int64_t h = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= n_out) return;
  float acc = b ? b[h] : 0.f;
  const float* wr = w + h * ld_w + col0;
  for (int j = 0; j < d; ++j) acc = fmaf(wr[j], temb[j], acc);
  bias_eff[(int64_t)blockIdx.y * n_out + h] = acc;
}

// ------------------------------------------------------------------ first layer on binary CSR rows
// h[r, :] = act(bias + sum_{c in row r} Wt[c, :]) for 0/1 rows (x0 of the reverse chain, Model.py:300-304 with
// sampling_step 0): the dense [B, I] x [I, H] contraction of Model.py:212 degenerates to a gather-sum of the
// rows of W^T.  One warp per user row; lane l owns the 16-byte pieces l, l+32, ... of the H columns, so every
// gathered weight row is read with full 512-byte warp transactions (the packed W^T is L2 resident).
template <bool LO, bool WT>
__global__ void __launch_bounds__(256) csr_gather_act_kernel(const int64_t* __restrict__ indptr,
                                                             const int32_t* __restrict__ indices,
                                                             const float* __restrict__ vals,
                                                             const int64_t* __restrict__ row_ids,
                                                             const int32_t* __restrict__ order, int64_t row0,
                                                             int64_t n_rows, int64_t n_cols,
                                                             const uint16_t* __restrict__ wt_hi,
                                                             const uint16_t* __restrict__ wt_lo, int64_t ld_w,
                                                             const float* __restrict__ bias, int act, int64_t n_out,
                                                             int slices, uint16_t* __restrict__ h_hi,
                                                             uint16_t* __restrict__ h_lo, int64_t ld_h,
                                                             float* __restrict__ z_f32, int64_t ld_z) {
  // one warp per (row, 256-column slice); lane l owns the 8 columns c0 .. c0+7 of the slice
  const int64_t wg = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const int64_t slot = wg / slices;
  if (slot >= n_rows) return;
  const int64_t r = order ? (int64_t)__ldg(order + slot) : slot;     // scheduling order only: outputs go to row r
  const int64_t c0 = (wg % slices) * 256 + 8 * lane;
  const bool col_ok = c0 < n_out;             // a piece that starts below n_out lies inside the padded row
  const int64_t u = row_ids ? row_ids[r] : row0 + r;
  const int64_t b = indptr[u], e = indptr[u + 1];
  float acc[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) acc[j] = 0.f;
  auto add = [&](const uint4& q, float w) {
    const uint32_t wv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      if constexpr (WT) {      // sparse rows with values (a q_sample'd start): x[c] * W^T[c, :]
        acc[2 * j] = fmaf(w, __uint_as_float(wv[j] << 16), acc[2 * j]);
        acc[2 * j + 1] = fmaf(w, __uint_as_float(wv[j] & 0xFFFF0000u), acc[2 * j + 1]);
      } else {
        acc[2 * j] += __uint_as_float(wv[j] << 16);
        acc[2 * j + 1] += __uint_as_float(wv[j] & 0xFFFF0000u);
      }
    }
  };
  const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
  constexpr int G = LO ? 4 : 8;     // gathered weight rows in flight per lane (16 bytes each, hi and lo)
  for (int64_t k = b; k < e; k += 32) {
    // the row's item ids: one coalesced load per 32 items, broadcast by shuffle; G gathers in flight per lane (the
    // 1 % of users with hundreds of interactions would otherwise set the length of the kernel's tail)
    int32_t mine = (k + lane < e) ? indices[k + lane] : -1;
    if (mine >= n_cols) mine = -1;
    float my_w = 1.f;
    if constexpr (WT) my_w = (k + lane < e) ? vals[k + lane] : 0.f;
    const int cnt = (int)((e - k) < 32 ? (e - k) : 32);
    for (int j = 0; j < cnt; j += G) {
      int32_t c[G];
      float w[G];
      uint4 qh[G], ql[LO ? G : 1];
#pragma unroll
      for (int t = 0; t < G; ++t) {
        c[t] = __shfl_sync(0xffffffffu, mine, (j + t) & 31);
        w[t] = WT ? __shfl_sync(0xffffffffu, my_w, (j + t) & 31) : 1.f;
      }
#pragma unroll
      for (int t = 0; t < G; ++t) {
        const bool ok = col_ok && j + t < cnt && c[t] >= 0;
        qh[t] = ok ? *reinterpret_cast<const uint4*>(wt_hi + (int64_t)c[t] * ld_w + c0) : zero;
        if constexpr (LO) ql[t] = ok ? *reinterpret_cast<const uint4*>(wt_lo + (int64_t)c[t] * ld_w + c0) : zero;
      }
#pragma unroll
      for (int t = 0; t < G; ++t) {
        add(qh[t], w[t]);
        if constexpr (LO) add(ql[t], w[t]);
      }
    }
  }
  if (!col_ok) return;
  if (z_f32) {
    // the plain gather-sum x0 . W^T (no bias): the hidden-space chain carries it as its fp32 state
    if (c0 + 8 <= n_out) {
      *reinterpret_cast<float4*>(z_f32 + r * ld_z + c0) = make_float4(acc[0], acc[1], acc[2], acc[3]);
      *reinterpret_cast<float4*>(z_f32 + r * ld_z + c0 + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
    } else {
      for (int j = 0; j < 8 && c0 + j < n_out; ++j) z_f32[r * ld_z + c0 + j] = acc[j];
    }
  }
  if (bias) {
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] += (c0 + j < n_out) ? bias[c0 + j] : 0.f;
  }
  uint32_t ph[4], pl[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float x0 = acc[2 * j], x1 = acc[2 * j + 1];
    if (act == 1) {
      x0 = 1.f - __fdividef(2.f, __expf(2.f * x0) + 1.f);
      x1 = 1.f - __fdividef(2.f, __expf(2.f * x1) + 1.f);
    }
    uint16_t a0, a1, l0, l1;
    dmm_split_bf16(x0, a0, l0);
    dmm_split_bf16(x1, a1, l1);
    ph[j] = (uint32_t)a0 | ((uint32_t)a1 << 16);
    pl[j] = (uint32_t)l0 | ((uint32_t)l1 << 16);
  }
  if (c0 + 8 <= n_out) {
    *reinterpret_cast<uint4*>(h_hi + r * ld_h + c0) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
    if (h_lo) *reinterpret_cast<uint4*>(h_lo + r * ld_h + c0) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
  } else {
    for (int j = 0; j < 8 && c0 + j < n_out; ++j) {
      h_hi[r * ld_h + c0 + j] = (uint16_t)(ph[j >> 1] >> (16 * (j & 1)));
      if (h_lo) h_lo[r * ld_h + c0 + j] = (uint16_t)(pl[j >> 1] >> (16 * (j & 1)));
    }
  }
}

// ------------------------------------------------------------------ first layer on CSR rows, rows scheduled by length
// What bounded the kernel above at the baby shape (ncu): 790 warp instructions per (row, slice) warp for a median row of
// 4-5 entries -- index arithmetic, item ids, shuffles, predicates and the bias / tanh / pack tail paid once per 256
// columns -- at 40 % occupancy.  Here ONE warp owns a whole short row: the item ids and entry values are loaded and
// broadcast once per entry, every entry issues NS independent 16-byte gathers per lane (all NS 256-column slices; two
// entries in flight), and the per-row overhead is paid once.  The rows of more than `threshold` entries (1 % of the users,
// 40 % of the entries) would be chains of hundreds of dependent gather rounds for a single warp, so they keep one warp per
// (row, slice): `order` lists them first (dmm_rows_long_first), `n_long_p` is their number (device scalar), and the first
// `long_blocks` CTAs of the same launch take them -- they start first and overlap the short rows.  The sums run over the
// entries in stored order in both roles: bit-identical to csr_gather_act_kernel.
template <bool LO, bool WT>
__device__ __forceinline__ void gather_tail(float (&acc)[8], const int64_t r, const int64_t c0, const float* __restrict__ bias,
                                            const int act, const int64_t n_out, uint16_t* __restrict__ h_hi,
                                            uint16_t* __restrict__ h_lo, const int64_t ld_h, float* __restrict__ z_f32,
                                            const int64_t ld_z) {
  if (c0 >= n_out) return;
  const bool full = c0 + 8 <= n_out;
  if (z_f32) {
    if (full) {
      *reinterpret_cast<float4*>(z_f32 + r * ld_z + c0) = make_float4(acc[0], acc[1], acc[2], acc[3]);
      *reinterpret_cast<float4*>(z_f32 + r * ld_z + c0 + 4) = make_float4(acc[4], acc[5], acc[6], acc[7]);
    } else {
      for (int j = 0; j < 8 && c0 + j < n_out; ++j) z_f32[r * ld_z + c0 + j] = acc[j];
    }
  }
  if (bias) {
    if (full && (reinterpret_cast<uintptr_t>(bias) & 15u) == 0) {
      const float4 b0 = *reinterpret_cast<const float4*>(bias + c0), b1 = *reinterpret_cast<const float4*>(bias + c0 + 4);
      acc[0] += b0.x; acc[1] += b0.y; acc[2] += b0.z; acc[3] += b0.w;
      acc[4] += b1.x; acc[5] += b1.y; acc[6] += b1.z; acc[7] += b1.w;
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] += (c0 + j < n_out) ? bias[c0 + j] : 0.f;
    }
  }
  uint32_t ph[4], pl[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float x0 = acc[2 * j], x1 = acc[2 * j + 1];
    if (act == 1) {
      x0 = 1.f - __fdividef(2.f, __expf(2.f * x0) + 1.f);
      x1 = 1.f - __fdividef(2.f, __expf(2.f * x1) + 1.f);
    }
    if constexpr (LO) {
      uint16_t a0, a1, l0, l1;
      dmm_split_bf16(x0, a0, l0);
      dmm_split_bf16(x1, a1, l1);
      ph[j] = (uint32_t)a0 | ((uint32_t)a1 << 16);
      pl[j] = (uint32_t)l0 | ((uint32_t)l1 << 16);
    } else {
      ph[j] = (uint32_t)dmm_bf16_bits(x0) | ((uint32_t)dmm_bf16_bits(x1) << 16);
      pl[j] = 0u;
    }
  }
  if (full) {
    *reinterpret_cast<uint4*>(h_hi + r * ld_h + c0) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
    if (LO && h_lo) *reinterpret_cast<uint4*>(h_lo + r * ld_h + c0) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
  } else {
    for (int j = 0; j < 8 && c0 + j < n_out; ++j) {
      h_hi[r * ld_h + c0 + j] = (uint16_t)(ph[j >> 1] >> (16 * (j & 1)));
      if (LO && h_lo) h_lo[r * ld_h + c0 + j] = (uint16_t)(pl[j >> 1] >> (16 * (j & 1)));
    }
  }
}

template <bool WT>
__device__ __forceinline__ void gather_add(float (&acc)[8], const uint4& q, const float w) {
  const uint32_t wv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if constexpr (WT) {      // sparse rows with values (a q_sample'd start): x[c] * W^T[c, :]
      acc[2 * j] = fmaf(w, __uint_as_float(wv[j] << 16), acc[2 * j]);
      acc[2 * j + 1] = fmaf(w, __uint_as_float(wv[j] & 0xFFFF0000u), acc[2 * j + 1]);
    } else {
      acc[2 * j] += __uint_as_float(wv[j] << 16);
      acc[2 * j + 1] += __uint_as_float(wv[j] & 0xFFFF0000u);
    }
  }
}

constexpr int GS_WARPS = 4;   // warps per CTA of the row-divided gather: 128 threads x 64 registers fit next to a resident contraction CTA
template <bool LO, bool WT, int NS>
__global__ void __launch_bounds__(32 * GS_WARPS, 32 / GS_WARPS) csr_gather_act_split_kernel(
    const int64_t* __restrict__ indptr, const int32_t* __restrict__ indices, const float* __restrict__ vals,
    const int64_t* __restrict__ row_ids, const int32_t* __restrict__ order, const int32_t* __restrict__ n_long_p,
    const int long_blocks, const int64_t max_long, int64_t row0, int64_t n_rows, int64_t n_cols,
    const uint16_t* __restrict__ wt_hi, const uint16_t* __restrict__ wt_lo, int64_t ld_w, const float* __restrict__ bias, int act,
    int64_t n_out, uint16_t* __restrict__ h_hi, uint16_t* __restrict__ h_lo, int64_t ld_h, float* __restrict__ z_f32,
    int64_t ld_z) {
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  int64_t n_long = (int64_t)__ldg(n_long_p);
  if (n_long > max_long) n_long = max_long;      // rows beyond the caller's bound take the short-row role (correct, slow)
  const uint4 zero = make_uint4(0u, 0u, 0u, 0u);
  if ((int)blockIdx.x < long_blocks) {
    // ---- long rows: one warp per (row, 256-column slice), 8 (LO: 4) entries in flight
    const int64_t wg = (int64_t)blockIdx.x * GS_WARPS + warp;
    const int64_t slot = wg / NS;
    if (slot >= n_long) return;
    const int64_t r = (int64_t)__ldg(order + slot);
    const int64_t c0 = (wg % NS) * 256 + 8 * lane;
    const bool col_ok = c0 < n_out;
    const int64_t u = row_ids ? row_ids[r] : row0 + r;
    const int64_t b = indptr[u], e = indptr[u + 1];
    float acc[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[j] = 0.f;
    constexpr int G = LO ? 4 : 8;
    for (int64_t k = b; k < e; k += 32) {
      int32_t mine = (k + lane < e) ? indices[k + lane] : -1;
      if (mine >= n_cols) mine = -1;
      float my_w = 1.f;
      if constexpr (WT) my_w = (k + lane < e) ? vals[k + lane] : 0.f;
      const int cnt = (int)((e - k) < 32 ? (e - k) : 32);
      for (int j = 0; j < cnt; j += G) {
        int32_t c[G];
        float w[G];
        uint4 qh[G], ql[LO ? G : 1];
#pragma unroll
        for (int t = 0; t < G; ++t) {
          c[t] = __shfl_sync(0xffffffffu, mine, (j + t) & 31);
          w[t] = WT ? __shfl_sync(0xffffffffu, my_w, (j + t) & 31) : 1.f;
        }
#pragma unroll
        for (int t = 0; t < G; ++t) {
          const bool ok = col_ok && j + t < cnt && c[t] >= 0;
          qh[t] = ok ? *reinterpret_cast<const uint4*>(wt_hi + (int64_t)c[t] * ld_w + c0) : zero;
          if constexpr (LO) ql[t] = ok ? *reinterpret_cast<const uint4*>(wt_lo + (int64_t)c[t] * ld_w + c0) : zero;
        }
#pragma unroll
        for (int t = 0; t < G; ++t) {
          gather_add<WT>(acc, qh[t], w[t]);
          if constexpr (LO) gather_add<WT>(acc, ql[t], w[t]);
        }
      }
    }
    gather_tail<LO, WT>(acc, r, c0, bias, act, n_out, h_hi, h_lo, ld_h, z_f32, ld_z);
    return;
  }
  // ---- short rows: one warp per row, all NS slices; 2 (LO: 1) entries x NS gathers in flight
  const int64_t s = (int64_t)((int)blockIdx.x - long_blocks) * GS_WARPS + warp;
  if (s >= n_rows - n_long) return;
  const int64_t r = (int64_t)__ldg(order + n_long + s);
  const int64_t u = row_ids ? row_ids[r] : row0 + r;
  const int64_t b = indptr[u], e = indptr[u + 1];
  const int64_t cl = 8 * lane;                    // this lane's first column inside every slice
  float acc[NS][8];
#pragma unroll
  for (int q = 0; q < NS; ++q)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[q][j] = 0.f;
  constexpr int G = LO ? 1 : 2;
  for (int64_t k = b; k < e; k += 32) {
    int32_t mine = (k + lane < e) ? indices[k + lane] : -1;
    if (mine >= n_cols) mine = -1;
    float my_w = 1.f;
    if constexpr (WT) my_w = (k + lane < e) ? vals[k + lane] : 0.f;
    const int cnt = (int)((e - k) < 32 ? (e - k) : 32);
    for (int j = 0; j < cnt; j += G) {
      int32_t c[G];
      float w[G];
      uint4 qh[G][NS], ql[LO ? G : 1][LO ? NS : 1];
#pragma unroll
      for (int t = 0; t < G; ++t) {
        c[t] = __shfl_sync(0xffffffffu, mine, (j + t) & 31);
        w[t] = WT ? __shfl_sync(0xffffffffu, my_w, (j + t) & 31) : 1.f;
      }
#pragma unroll
      for (int t = 0; t < G; ++t) {
        const bool ok = j + t < cnt && c[t] >= 0;
        const uint16_t* ph = wt_hi + (int64_t)(ok ? c[t] : 0) * ld_w + cl;
        const uint16_t* pl = LO ? wt_lo + (int64_t)(ok ? c[t] : 0) * ld_w + cl : nullptr;
#pragma unroll
        for (int q = 0; q < NS; ++q) {
          const bool okq = ok && q * 256 + cl < n_out;
          qh[t][q] = okq ? *reinterpret_cast<const uint4*>(ph + q * 256) : zero;
          if constexpr (LO) ql[t][q] = okq ? *reinterpret_cast<const uint4*>(pl + q * 256) : zero;
        }
      }
#pragma unroll
      for (int t = 0; t < G; ++t) {
        if (t > 0 && j + t >= cnt) break;        // warp-uniform: the padded slot of an odd row length adds zeros
#pragma unroll
        for (int q = 0; q < NS; ++q) {
          gather_add<WT>(acc[q], qh[t][q], w[t]);
          if constexpr (LO) gather_add<WT>(acc[q], ql[t][q], w[t]);
        }
      }
    }
  }
#pragma unroll
  for (int q = 0; q < NS; ++q) gather_tail<LO, WT>(acc[q], r, q * 256 + cl, bias, act, n_out, h_hi, h_lo, ld_h, z_f32, ld_z);
}

// ------------------------------------------------------------------ q_sample on binary CSR rows
// Default-noise q_sample (Model.py:324-341) of a BINARY row keeps the row's sparsity: noise = sign(x0) * normalize(n)
// vanishes wherever x0 does, so x_t = a x0 + b noise has the value a + b n_c / max(||n||_2, 1e-12) at the row's items
// and 0 elsewhere (n = the full randn row: its norm runs over all n_cols columns).  One CTA per row streams the noise
// row once for the norm and writes the values of the row's entries; the first Denoise layer then stays a (weighted)
// gather-sum instead of a dense contraction.  HBM-bound: 4 * n_cols bytes read per row.
__global__ void __launch_bounds__(256) csr_qsample_values_kernel(const int64_t* __restrict__ indptr,
                                                                 const int32_t* __restrict__ indices,
                                                                 const int64_t* __restrict__ row_ids, int64_t row0,
                                                                 int64_t n_cols, const float* __restrict__ noise,
                                                                 int64_t ld_noise, float coef_a, float coef_b,
                                                                 float* __restrict__ vals) {
  __shared__ float red[8];
  const int64_t r = blockIdx.x;
  const int tid = threadIdx.x;
  const int64_t u = row_ids ? row_ids[r] : row0 + r;
  const int64_t b = indptr[u], e = indptr[u + 1];
  if (b >= e) return;                                   // block-uniform: nothing to emit for an empty row
  const float* row = noise + r * ld_noise;
  float ss = 0.f;
  if ((reinterpret_cast<uintptr_t>(row) & 15u) == 0) {
    const int64_t n4 = n_cols >> 2;
    const float4* row4 = reinterpret_cast<const float4*>(row);
#pragma unroll 4
    for (int64_t i = tid; i < n4; i += 256) {
      const float4 q = __ldcs(row4 + i);
      ss = fmaf(q.x, q.x, ss);
      ss = fmaf(q.y, q.y, ss);
      ss = fmaf(q.z, q.z, ss);
      ss = fmaf(q.w, q.w, ss);
    }
    for (int64_t i = (n4 << 2) + tid; i < n_cols; i += 256) ss = fmaf(row[i], row[i], ss);
  } else {
    for (int64_t i = tid; i < n_cols; i += 256) ss = fmaf(row[i], row[i], ss);
  }
  ss = dmm_warp_sum(ss);
  if ((tid & 31) == 0) red[tid >> 5] = ss;
  __syncthreads();
  float tot = 0.f;
#pragma unroll
  for (int i = 0; i < 8; ++i) tot += red[i];
  const float inv = 1.f / fmaxf(sqrtf(tot), 1e-12f);
  for (int64_t k = b + tid; k < e; k += 256) {
    const int32_t c = indices[k];
    const float n = (c >= 0 && c < n_cols) ? row[c] : 0.f;
    vals[k] = __fadd_rn(coef_a, __fmul_rn(coef_b, __fmul_rn(n, inv)));
  }
}

// ------------------------------------------------------------------ q_sample on binary CSR rows, noise generated in place
// Same quantity as csr_qsample_values_kernel, but the standard-normal row n (Model.py:337: randn_like) is GENERATED inside
// the kernel instead of being written to and re-read from HBM by a separate generator launch (19445 x 7050 normals are
// 548 MB each way per modality: ncu showed generator + reader at 37 % of a conf/baby.toml rebuild step).  Counter-based
// Philox4x32-10 keyed by a 64-bit seed taken from torch's device generator, counter = (row, column / 4): element c of row r
// is a pure function of (seed, r, c), so any entry can be drawn on its own without storing the row; Box-Muller on the
// four 32-bit outputs.  The draw is i.i.d. N(0, 1) like the reference's; the stream is not torch's (no two GPU runs of
// the reference share a stream with each other either: its loader shuffles the users).
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(0xD2511F53u, ctr.x), lo0 = 0xD2511F53u * ctr.x;
    const uint32_t hi1 = __umulhi(0xCD9E8D57u, ctr.z), lo1 = 0xCD9E8D57u * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += 0x9E3779B9u;
    key.y += 0xBB67AE85u;
  }
  return ctr;
}
__device__ __forceinline__ float4 normal4(uint4 u) {
  // (0, 1] uniforms from the 32-bit words, Box-Muller pairs
  const float a0 = ((float)u.x + 1.0f) * 2.3283064365386963e-10f, a1 = (float)u.y * 2.3283064365386963e-10f;
  const float b0 = ((float)u.z + 1.0f) * 2.3283064365386963e-10f, b1 = (float)u.w * 2.3283064365386963e-10f;
  const float r0 = sqrtf(-2.0f * __logf(a0)), r1 = sqrtf(-2.0f * __logf(b0));
  float s0, c0, s1, c1;
  __sincosf(6.283185307179586f * a1, &s0, &c0);
  __sincosf(6.283185307179586f * b1, &s1, &c1);
  return make_float4(r0 * c0, r0 * s0, r1 * c1, r1 * s1);
}

// ------------------------------------------------------------------ q_sample on binary CSR rows, sufficient statistics only
// The entry values need only two things from the N(0, 1) row n: its entries on the row's support S (k = |S| normals) and
// its squared norm  ||n||^2 = sum_{c in S} n_c^2 + R,  R = sum_{c not in S} n_c^2 ~ chi^2(I - k), independent of n_S.
// So instead of I normals per row (137 M per modality at baby, ~0.18 ms of Philox + Box-Muller) the kernel draws the k
// support normals (the Philox elements (seed, row, c): the same normals a full row would have) and ONE chi-square variate:
// exactly the reference's joint distribution of the outputs (Model.py:337-341), O(k) work per row.
// chi^2(nu) = 2 Gamma(nu / 2) by Marsaglia-Tsang (exact rejection sampler, acceptance > 99.9 % at nu ~ 7000); nu <= 64:
// the sum of nu explicit normals.  One warp per row.
// `first`: the Philox block of attempt 0 when the caller already drew it (in lockstep with the support normals of the
// other lanes); the variate is the same either way.
__device__ __forceinline__ float chi2_sample(uint32_t nu, uint32_t row_lo, uint32_t row_hi, uint2 key,
                                             const uint4* first = nullptr) {
  if (nu == 0u) return 0.f;
  if (nu <= 64u) {
    float s = 0.f;
    for (uint32_t q = 0; 4u * q < nu; ++q) {
      const float4 n = normal4(philox4x32_10(make_uint4(q, row_lo, row_hi, 2u), key));
      s = fmaf(n.x, n.x, s);
      if (4u * q + 1u < nu) s = fmaf(n.y, n.y, s);
      if (4u * q + 2u < nu) s = fmaf(n.z, n.z, s);
      if (4u * q + 3u < nu) s = fmaf(n.w, n.w, s);
    }
    return s;
  }
  const float a = 0.5f * (float)nu;
  const float d = a - (1.0f / 3.0f);
  const float c = rsqrtf(9.0f * d);
  float v = 1.f;
  for (uint32_t attempt = 0; attempt < 64u; ++attempt) {
    const uint4 u4 = (attempt == 0u && first) ? *first : philox4x32_10(make_uint4(attempt, row_lo, row_hi, 1u), key);
    const float x = normal4(u4).x;
    const float t = fmaf(c, x, 1.0f);
    if (t <= 0.f) continue;
    v = t * t * t;
    const float u = ((float)u4.z + 1.0f) * 2.3283064365386963e-10f;
    const float x2 = x * x;
    if (u < 1.0f - 0.0331f * x2 * x2) break;
    if (logf(u) < 0.5f * x2 + d * (1.0f - v + log1pf(v - 1.0f))) break;
  }
  return 2.0f * d * v;
}

__global__ void __launch_bounds__(256) csr_qsample_values_chi2_kernel(const int64_t* __restrict__ indptr,
                                                                      const int32_t* __restrict__ indices,
                                                                      const int64_t* __restrict__ row_ids, int64_t row0,
                                                                      int64_t n_rows, int64_t n_cols,
                                                                      const int64_t* __restrict__ seed, float coef_a,
                                                                      float coef_b, float* __restrict__ vals) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  const int64_t u = row_ids ? row_ids[r] : row0 + r;
  const int64_t b = indptr[u], e = indptr[u + 1];
  if (b >= e) return;
  const uint64_t sd = (uint64_t)seed[0];
  const uint2 key = make_uint2((uint32_t)sd, (uint32_t)(sd >> 32));
  const uint32_t row_lo = (uint32_t)u, row_hi = (uint32_t)((uint64_t)u >> 32);
  auto pick = [](const float4& n, int w) -> float { return w == 0 ? n.x : (w == 1 ? n.y : (w == 2 ? n.z : n.w)); };
  if (e - b < 32) {
    // Short row (99 % of them): one entry per lane, ONE Philox + Box-Muller round for the whole row.  Lane 31 has no
    // entry: it draws attempt 0 of the chi-square variate in the same instructions (counter stream 1 instead of 0), and
    // every lane keeps its normal for the value pass.  Same Philox elements, same arithmetic, same values as the general
    // path below.
    const bool has = b + lane < e;
    const int32_t c = has ? indices[b + lane] : -1;
    const bool ok = c >= 0 && c < n_cols;
    const uint32_t valid = (uint32_t)__popc(__ballot_sync(0xffffffffu, ok));
    const uint4 ctr = lane == 31 ? make_uint4(0u, row_lo, row_hi, 1u) : make_uint4((uint32_t)(ok ? c >> 2 : 0), row_lo, row_hi, 0u);
    const uint4 blk = philox4x32_10(ctr, key);
    const float nv = ok ? pick(normal4(blk), c & 3) : 0.f;
    const float ss = dmm_warp_sum(ok ? fmaf(nv, nv, 0.f) : 0.f);
    float rest = 0.f;
    if (lane == 31) rest = chi2_sample((uint32_t)(n_cols - (int64_t)valid), row_lo, row_hi, key, &blk);
    rest = __shfl_sync(0xffffffffu, rest, 31);
    const float inv = 1.f / fmaxf(sqrtf(ss + rest), 1e-12f);
    if (has) vals[b + lane] = __fadd_rn(coef_a, __fmul_rn(coef_b, __fmul_rn(nv, inv)));
    return;
  }
  auto normal_at = [&](int32_t c) -> float {
    return pick(normal4(philox4x32_10(make_uint4((uint32_t)(c >> 2), row_lo, row_hi, 0u), key)), c & 3);
  };
  float ss = 0.f;
  uint32_t valid = 0;
  for (int64_t k = b + lane; k < e; k += 32) {
    const int32_t c = indices[k];
    if (c >= 0 && c < n_cols) {
      const float nv = normal_at(c);
      ss = fmaf(nv, nv, ss);
      ++valid;
    }
  }
  ss = dmm_warp_sum(ss);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) valid += __shfl_xor_sync(0xffffffffu, valid, o);
  float rest = 0.f;
  if (lane == 0) rest = chi2_sample((uint32_t)(n_cols - (int64_t)valid), row_lo, row_hi, key);
  rest = __shfl_sync(0xffffffffu, rest, 0);
  const float inv = 1.f / fmaxf(sqrtf(ss + rest), 1e-12f);
  for (int64_t k = b + lane; k < e; k += 32) {
    const int32_t c = indices[k];
    const float nv = (c >= 0 && c < n_cols) ? normal_at(c) : 0.f;
    vals[k] = __fadd_rn(coef_a, __fmul_rn(coef_b, __fmul_rn(nv, inv)));
  }
}

// ------------------------------------------------------------------ scheduling order: long rows first
// order[] = a permutation of 0..n_rows-1 with every row of more than `threshold` entries in front (slots taken from
// the front by the long rows, from the back by the others; warp-aggregated atomics on two counters).  The order
// among equals is arbitrary: it only decides WHEN dmm_csr_gather_act schedules a row, never what it computes.
__global__ void __launch_bounds__(256) rows_long_first_kernel(const int64_t* __restrict__ indptr, int64_t row0, int64_t n_rows,
                                                              int threshold, int32_t* __restrict__ order,
                                                              int32_t* __restrict__ counters) {
  const int64_t r = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int lane = threadIdx.x & 31;
  const bool in = r < n_rows;
  const bool heavy = in && (indptr[row0 + r + 1] - indptr[row0 + r] > threshold);
  const uint32_t mh = __ballot_sync(0xffffffffu, heavy), ml = __ballot_sync(0xffffffffu, in && !heavy);
  int bh = 0, bl = 0;
  if (lane == 0) {
    if (mh) bh = atomicAdd(counters, __popc(mh));
    if (ml) bl = atomicAdd(counters + 1, __popc(ml));
  }
  bh = __shfl_sync(0xffffffffu, bh, 0);
  bl = __shfl_sync(0xffffffffu, bl, 0);
  const uint32_t below = (1u << lane) - 1u;
  if (heavy) order[bh + __popc(mh & below)] = (int32_t)r;
  else if (in) order[n_rows - 1 - (bl + __popc(ml & below))] = (int32_t)r;
}

// ------------------------------------------------------------------ y = W[:, :K] x  (fp32, one warp per row)
// q = W1x b2 of the hidden-space chain: a 1024 x 7050 matrix-vector product is a bandwidth problem, not a GEMM.
__global__ void __launch_bounds__(128) gemv_rows_kernel(const float* __restrict__ w, int64_t ld_w, int64_t n_rows,
                                                        int64_t K, const float* __restrict__ x, float* __restrict__ y) {
  // one CTA (4 warps) per row: enough loads in flight to stream the matrix at HBM speed
  __shared__ float red[4];
  const int64_t r = blockIdx.x;
  const int tid = threadIdx.x;
  const float* row = w + r * ld_w;
  float acc = 0.f;
  if (((reinterpret_cast<uintptr_t>(row) | reinterpret_cast<uintptr_t>(x)) & 15u) == 0) {
    const int64_t k4 = K >> 2;
    const float4* row4 = reinterpret_cast<const float4*>(row);
    const float4* x4 = reinterpret_cast<const float4*>(x);
#pragma unroll 4
    for (int64_t k = tid; k < k4; k += 128) {
      const float4 a = __ldg(row4 + k), b = __ldg(x4 + k);
      acc = fmaf(a.x, b.x, acc);
      acc = fmaf(a.y, b.y, acc);
      acc = fmaf(a.z, b.z, acc);
      acc = fmaf(a.w, b.w, acc);
    }
    for (int64_t k = (k4 << 2) + tid; k < K; k += 128) acc = fmaf(__ldg(row + k), __ldg(x + k), acc);
  } else {
    for (int64_t k = tid; k < K; k += 128) acc = fmaf(__ldg(row + k), __ldg(x + k), acc);
  }
  acc = dmm_warp_sum(acc);
  if ((tid & 31) == 0) red[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) y[r] = (red[0] + red[1]) + (red[2] + red[3]);
}

// ------------------------------------------------------------------ h = act(z + bias) -> bf16 hi (+ lo)
// Hidden layer of the hidden-space reverse chain (rebuild.py): z is the fp32 pre-activation state [n_rows, n_cols].
__global__ void __launch_bounds__(256) bias_act_pack_kernel(const float* __restrict__ z, int64_t ld_z,
                                                            const float* __restrict__ bias, int64_t n_rows,
                                                            int64_t n_cols, int act, uint16_t* __restrict__ h_hi,
                                                            uint16_t* __restrict__ h_lo, int64_t ld_h) {
  const int64_t n4 = (n_cols + 3) >> 2;
  const int64_t total = n_rows * n4;
  for (int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (int64_t)gridDim.x * blockDim.x) {
    const int64_t r = t / n4, c = (t - r * n4) << 2;
    float v[4];
    if (c + 4 <= n_cols) {
      const float4 q = *reinterpret_cast<const float4*>(z + r * ld_z + c);
      v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
    } else {
      for (int j = 0; j < 4; ++j) v[j] = c + j < n_cols ? z[r * ld_z + c + j] : 0.f;
    }
    uint16_t hi[4], lo[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      float x = v[j] + ((bias && c + j < n_cols) ? __ldg(bias + c + j) : 0.f);
      if (act == 1) x = 1.f - __fdividef(2.f, __expf(2.f * x) + 1.f);
      dmm_split_bf16(x, hi[j], lo[j]);
    }
    if (c + 4 <= n_cols) {
      *reinterpret_cast<uint2*>(h_hi + r * ld_h + c) =
          make_uint2((uint32_t)hi[0] | ((uint32_t)hi[1] << 16), (uint32_t)hi[2] | ((uint32_t)hi[3] << 16));
      if (h_lo)
        *reinterpret_cast<uint2*>(h_lo + r * ld_h + c) =
            make_uint2((uint32_t)lo[0] | ((uint32_t)lo[1] << 16), (uint32_t)lo[2] | ((uint32_t)lo[3] << 16));
    } else {
      for (int j = 0; j < 4 && c + j < n_cols; ++j) {
        h_hi[r * ld_h + c + j] = hi[j];
        if (h_lo) h_lo[r * ld_h + c + j] = lo[j];
      }
    }
  }
}

// ------------------------------------------------------------------ x[r, c] += beta at the CSR positions
// Posterior mean of the first reverse step: x_{t-1} = c1 * pred + c2 * x0 with binary x0 (Model.py:375);
// the GEMM epilogue writes c1 * pred, this adds c2 where x0 is 1.  One warp per row.
__global__ void __launch_bounds__(256) csr_axpy_bf16_kernel(const int64_t* __restrict__ indptr,
                                                            const int32_t* __restrict__ indices,
                                                            const int64_t* __restrict__ row_ids, int64_t row0,
                                                            int64_t n_rows, int64_t n_cols, float beta,
                                                            uint16_t* __restrict__ x_hi, uint16_t* __restrict__ x_lo,
                                                            int64_t ld_x) {
  const int64_t r = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (r >= n_rows) return;
  const int64_t u = row_ids ? row_ids[r] : row0 + r;
  const int64_t b = indptr[u], e = indptr[u + 1];
  for (int64_t k = b + lane; k < e; k += 32) {
    const int32_t c = indices[k];
    if (c < 0 || c >= n_cols) continue;
    float v = dmm_bf16_to_f32(x_hi[r * ld_x + c]);
    if (x_lo) v += dmm_bf16_to_f32(x_lo[r * ld_x + c]);
    v += beta;
    uint16_t h, l;
    dmm_split_bf16(v, h, l);
    x_hi[r * ld_x + c] = h;
    if (x_lo) x_lo[r * ld_x + c] = l;
  }
}

}  // namespace

extern "C" int dmm_pack_bf16(dmm_ctx* ctx, const float* src, int64_t rows, int64_t cols, int64_t ld_src,
                             uint16_t* dst_hi, uint16_t* dst_lo, int64_t ld_dst, int transpose, void* stream) {
  DMM_CHECK_ARG(ctx && src && dst_hi, "dmm_pack_bf16: null argument");
  DMM_CHECK_ARG(rows > 0 && cols > 0 && ld_src >= cols, "dmm_pack_bf16: bad shape");
  DMM_CHECK_ARG(ld_dst % 8 == 0, "dmm_pack_bf16: ld_dst must be a multiple of 8 (got %lld)", (long long)ld_dst);
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(dst_hi) && al16(dst_lo), "dmm_pack_bf16: destinations must be 16-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (!transpose) {
    DMM_CHECK_ARG(ld_dst >= cols, "dmm_pack_bf16: ld_dst < cols");
    const int64_t total = rows * (ld_dst / 8);
    int64_t blocks = dmm_ceil_div(total, 256);
    const int64_t cap = (int64_t)ctx->num_sms * 32;
    if (blocks > cap) blocks = cap;
    if (al16(src) && ld_src % 4 == 0) {
      pack_rows_kernel<true><<<(unsigned)blocks, 256, 0, st>>>(src, rows, cols, ld_src, dst_hi, dst_lo, ld_dst);
    } else {
      pack_rows_kernel<false><<<(unsigned)blocks, 256, 0, st>>>(src, rows, cols, ld_src, dst_hi, dst_lo, ld_dst);
    }
  } else {
    DMM_CHECK_ARG(ld_dst >= rows, "dmm_pack_bf16: ld_dst < rows (transposed)");
    const int64_t gy = dmm_ceil_div(ld_dst, 64);
    DMM_CHECK_ARG(gy < 65536, "dmm_pack_bf16: too many rows for the transposed path");
    dim3 grid((unsigned)dmm_ceil_div(cols, 64), (unsigned)gy);
    if (al16(src) && ld_src % 4 == 0) {
      pack_transpose_kernel<true><<<grid, 256, 0, st>>>(src, rows, cols, ld_src, dst_hi, dst_lo, ld_dst, nullptr, nullptr, 0);
    } else {
      pack_transpose_kernel<false><<<grid, 256, 0, st>>>(src, rows, cols, ld_src, dst_hi, dst_lo, ld_dst, nullptr, nullptr, 0);
    }
  }
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_pack_bf16_pair(dmm_ctx* ctx, const float* src, int64_t rows, int64_t cols, int64_t ld_src,
                                  uint16_t* nat_hi, uint16_t* nat_lo, int64_t ld_nat, uint16_t* tr_hi, uint16_t* tr_lo,
                                  int64_t ld_tr, void* stream) {
  DMM_CHECK_ARG(ctx && src && nat_hi && tr_hi, "dmm_pack_bf16_pair: null argument");
  DMM_CHECK_ARG(rows > 0 && cols > 0 && ld_src >= cols, "dmm_pack_bf16_pair: bad shape");
  DMM_CHECK_ARG(ld_nat % 8 == 0 && ld_tr % 8 == 0 && ld_tr >= rows, "dmm_pack_bf16_pair: bad leading dimensions");
  DMM_CHECK_ARG(ld_nat >= cols && ld_nat <= (cols + 63) / 64 * 64, "dmm_pack_bf16_pair: ld_nat must lie in [cols, pad64(cols)]");
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(nat_hi) && al16(nat_lo) && al16(tr_hi) && al16(tr_lo), "dmm_pack_bf16_pair: destinations must be 16-byte aligned");
  DMM_CHECK_ARG((nat_lo == nullptr) == (tr_lo == nullptr), "dmm_pack_bf16_pair: lo parts are all-or-none");
  const int64_t gy = dmm_ceil_div(ld_tr, 64);
  DMM_CHECK_ARG(gy < 65536, "dmm_pack_bf16_pair: too many rows");
  dim3 grid((unsigned)dmm_ceil_div(cols, 64), (unsigned)gy);
  cudaStream_t st = (cudaStream_t)stream;
  if (al16(src) && ld_src % 4 == 0) {
    pack_transpose_kernel<true><<<grid, 256, 0, st>>>(src, rows, cols, ld_src, tr_hi, tr_lo, ld_tr, nat_hi, nat_lo, ld_nat);
  } else {
    pack_transpose_kernel<false><<<grid, 256, 0, st>>>(src, rows, cols, ld_src, tr_hi, tr_lo, ld_tr, nat_hi, nat_lo, ld_nat);
  }
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_csr_rows_to_dense(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices,
                                     const int64_t* row_ids, int64_t row0, int64_t n_rows, int64_t n_cols,
                                     float* x_f32, int64_t ld_x, uint16_t* a_bf16, int64_t ld_a, void* stream) {
  DMM_CHECK_ARG(ctx && indptr && indices, "dmm_csr_rows_to_dense: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_cols > 0, "dmm_csr_rows_to_dense: bad shape");
  DMM_CHECK_ARG((!x_f32 || ld_x >= n_cols) && (!a_bf16 || ld_a >= n_cols), "dmm_csr_rows_to_dense: ld too small");
  if (n_rows == 0) return DMM_OK;
  const unsigned grid = (unsigned)(n_rows < (int64_t)ctx->num_sms * 64 ? n_rows : (int64_t)ctx->num_sms * 64);
  csr_rows_dense_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(indptr, indices, row_ids, row0, n_rows, n_cols, x_f32, ld_x,
                                                               a_bf16, ld_a);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_time_embedding(dmm_ctx* ctx, const int64_t* t, int64_t t_all, int64_t n_rows, int d_emb,
                                  const float* emb_w, const float* emb_b, uint16_t* a_hi, uint16_t* a_lo,
                                  int64_t ld_a, int64_t col0, float* temb_f32, void* stream) {
  DMM_CHECK_ARG(ctx && emb_w && emb_b, "dmm_time_embedding: null argument");
  DMM_CHECK_ARG(d_emb >= 2 && d_emb <= 64, "dmm_time_embedding: d_emb must be in [2, 64]");
  DMM_CHECK_ARG(!a_hi || ld_a >= col0 + d_emb, "dmm_time_embedding: ld_a too small");
  if (n_rows <= 0) return DMM_OK;
  time_embedding_kernel<<<(unsigned)dmm_ceil_div(n_rows, 256), 256, 0, (cudaStream_t)stream>>>(
      t, t_all, n_rows, d_emb, emb_w, emb_b, a_hi, a_lo, ld_a, col0, temb_f32);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_q_sample(dmm_ctx* ctx, const float* x0, int64_t ld_x0, const float* noise, int64_t ld_noise,
                            const float* coef_a, const float* coef_b, int64_t n_rows, int64_t n_cols, int mode,
                            float* x_t, int64_t ld_x, uint16_t* a_hi, uint16_t* a_lo, int64_t ld_a, void* stream) {
  DMM_CHECK_ARG(ctx && x0 && noise && coef_a && coef_b, "dmm_q_sample: null argument");
  DMM_CHECK_ARG(mode == 0 || mode == 1, "dmm_q_sample: mode must be 0 or 1");
  DMM_CHECK_ARG(n_cols > 0 && ld_x0 >= n_cols && ld_noise >= n_cols, "dmm_q_sample: bad shape");
  if (n_rows <= 0) return DMM_OK;
  q_sample_kernel<<<(unsigned)n_rows, 256, 0, (cudaStream_t)stream>>>(x0, ld_x0, noise, ld_noise, coef_a, coef_b, n_cols,
                                                                      mode, x_t, ld_x, a_hi, a_lo, ld_a);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_time_bias(dmm_ctx* ctx, int64_t t0, int64_t n_t, int d_emb, const float* emb_w, const float* emb_b,
                             const float* w, int64_t ld_w, int64_t col0, const float* b, int64_t n_out,
                             float* bias_eff, void* stream) {
  DMM_CHECK_ARG(ctx && emb_w && emb_b && w && bias_eff, "dmm_time_bias: null argument");
  DMM_CHECK_ARG(d_emb >= 2 && d_emb <= 64, "dmm_time_bias: d_emb must be in [2, 64]");
  DMM_CHECK_ARG(n_out > 0 && col0 >= 0 && ld_w >= col0 + d_emb, "dmm_time_bias: bad shape");
  DMM_CHECK_ARG(n_t > 0 && n_t < 65536, "dmm_time_bias: n_t must be in [1, 65535]");
  dim3 grid((unsigned)dmm_ceil_div(n_out, 256), (unsigned)n_t);
  time_bias_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(t0, d_emb, emb_w, emb_b, w, ld_w, col0, b, n_out, bias_eff);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_csr_qsample_values(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                                      int64_t row0, int64_t n_rows, int64_t n_cols, const float* noise, int64_t ld_noise,
                                      float coef_a, float coef_b, float* vals, void* stream) {
  DMM_CHECK_ARG(ctx && indptr && indices && noise && vals, "dmm_csr_qsample_values: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31) && n_cols > 0 && ld_noise >= n_cols, "dmm_csr_qsample_values: bad shape");
  if (n_rows == 0) return DMM_OK;
  csr_qsample_values_kernel<<<(unsigned)n_rows, 256, 0, (cudaStream_t)stream>>>(indptr, indices, row_ids, row0, n_cols, noise,
                                                                               ld_noise, coef_a, coef_b, vals);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_csr_qsample_values_rng(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                                          int64_t row0, int64_t n_rows, int64_t n_cols, const int64_t* seed, float coef_a,
                                          float coef_b, float* vals, void* stream) {
  DMM_CHECK_ARG(ctx && indptr && indices && seed && vals, "dmm_csr_qsample_values_rng: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31) && n_cols > 0 && n_cols < (1LL << 31), "dmm_csr_qsample_values_rng: bad shape");
  if (n_rows == 0) return DMM_OK;
  csr_qsample_values_chi2_kernel<<<(unsigned)dmm_ceil_div(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      indptr, indices, row_ids, row0, n_rows, n_cols, seed, coef_a, coef_b, vals);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_csr_gather_act(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const float* vals,
                                  const int64_t* row_ids, const int32_t* order,
                                  int64_t row0, int64_t n_rows, int64_t n_cols, const uint16_t* wt_hi,
                                  const uint16_t* wt_lo, int64_t ld_w, const float* bias, int act, int64_t n_out,
                                  uint16_t* h_hi, uint16_t* h_lo, int64_t ld_h, float* z_f32, int64_t ld_z,
                                  void* stream) {
  DMM_CHECK_ARG(ctx && indptr && indices && wt_hi && h_hi, "dmm_csr_gather_act: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_cols > 0 && n_out > 0, "dmm_csr_gather_act: bad shape");
  DMM_CHECK_ARG(ld_w % 8 == 0 && ld_h % 8 == 0 && ld_w >= dmm_ceil_div(n_out, 8) * 8 && ld_h >= n_out,
                "dmm_csr_gather_act: ld_w / ld_h must be multiples of 8 covering n_out (got %lld, %lld)", (long long)ld_w,
                (long long)ld_h);
  DMM_CHECK_ARG(act == 0 || act == 1, "dmm_csr_gather_act: unknown activation %d", act);
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(wt_hi) && al16(wt_lo) && al16(h_hi) && al16(h_lo) && al16(z_f32),
                "dmm_csr_gather_act: buffers must be 16-byte aligned");
  DMM_CHECK_ARG(!z_f32 || (ld_z >= n_out && ld_z % 4 == 0), "dmm_csr_gather_act: ld_z must be >= n_out and a multiple of 4");
  if (n_rows == 0) return DMM_OK;
  const int slices = (int)dmm_ceil_div(n_out, 256);
  const int64_t blocks = dmm_ceil_div(n_rows * slices * 32, 256);
  DMM_CHECK_ARG(blocks < (1LL << 31), "dmm_csr_gather_act: too many rows");
  const unsigned grid = (unsigned)blocks;
  cudaStream_t st = (cudaStream_t)stream;
#define DMM_GATHER_ARGS indptr, indices, vals, row_ids, order, row0, n_rows, n_cols, wt_hi, wt_lo, ld_w, bias, act, n_out, slices, \
                        h_hi, h_lo, ld_h, z_f32, ld_z
  if (wt_lo) {
    if (vals) csr_gather_act_kernel<true, true><<<grid, 256, 0, st>>>(DMM_GATHER_ARGS);
    else csr_gather_act_kernel<true, false><<<grid, 256, 0, st>>>(DMM_GATHER_ARGS);
  } else {
    if (vals) csr_gather_act_kernel<false, true><<<grid, 256, 0, st>>>(DMM_GATHER_ARGS);
    else csr_gather_act_kernel<false, false><<<grid, 256, 0, st>>>(DMM_GATHER_ARGS);
  }
#undef DMM_GATHER_ARGS
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

template <bool LO, bool WT>
static void launch_gather_split(int ns, unsigned grid, cudaStream_t st, const int64_t* indptr, const int32_t* indices,
                                const float* vals, const int64_t* row_ids, const int32_t* order, const int32_t* n_long,
                                int long_blocks, int64_t max_long, int64_t row0, int64_t n_rows, int64_t n_cols,
                                const uint16_t* wt_hi, const uint16_t* wt_lo, int64_t ld_w, const float* bias, int act,
                                int64_t n_out, uint16_t* h_hi, uint16_t* h_lo, int64_t ld_h, float* z_f32, int64_t ld_z) {
#define DMM_GS_ARGS indptr, indices, vals, row_ids, order, n_long, long_blocks, max_long, row0, n_rows, n_cols, wt_hi, wt_lo, ld_w, \
                    bias, act, n_out, h_hi, h_lo, ld_h, z_f32, ld_z
  if (ns == 1) csr_gather_act_split_kernel<LO, WT, 1><<<grid, 32 * GS_WARPS, 0, st>>>(DMM_GS_ARGS);
  else if (ns == 2) csr_gather_act_split_kernel<LO, WT, 2><<<grid, 32 * GS_WARPS, 0, st>>>(DMM_GS_ARGS);
  else csr_gather_act_split_kernel<LO, WT, 4><<<grid, 32 * GS_WARPS, 0, st>>>(DMM_GS_ARGS);
#undef DMM_GS_ARGS
}

extern "C" int dmm_csr_gather_act_split(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const float* vals,
                                        const int64_t* row_ids, const int32_t* order, const int32_t* n_long,
                                        int64_t max_long, int64_t row0, int64_t n_rows, int64_t n_cols,
                                        const uint16_t* wt_hi, const uint16_t* wt_lo, int64_t ld_w, const float* bias,
                                        int act, int64_t n_out, uint16_t* h_hi, uint16_t* h_lo, int64_t ld_h,
                                        float* z_f32, int64_t ld_z, void* stream) {
  DMM_CHECK_ARG(ctx && indptr && indices && wt_hi && h_hi && order && n_long, "dmm_csr_gather_act_split: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_cols > 0 && n_out > 0 && max_long >= 0, "dmm_csr_gather_act_split: bad shape");
  DMM_CHECK_ARG(n_out <= 1024, "dmm_csr_gather_act_split: at most 1024 output columns (got %lld); use dmm_csr_gather_act",
                (long long)n_out);
  DMM_CHECK_ARG(ld_w % 8 == 0 && ld_h % 8 == 0 && ld_w >= dmm_ceil_div(n_out, 8) * 8 && ld_h >= n_out,
                "dmm_csr_gather_act_split: ld_w / ld_h must be multiples of 8 covering n_out (got %lld, %lld)", (long long)ld_w,
                (long long)ld_h);
  DMM_CHECK_ARG(act == 0 || act == 1, "dmm_csr_gather_act_split: unknown activation %d", act);
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(wt_hi) && al16(wt_lo) && al16(h_hi) && al16(h_lo) && al16(z_f32),
                "dmm_csr_gather_act_split: buffers must be 16-byte aligned");
  DMM_CHECK_ARG(!z_f32 || (ld_z >= n_out && ld_z % 4 == 0), "dmm_csr_gather_act_split: ld_z must be >= n_out and a multiple of 4");
  if (n_rows == 0) return DMM_OK;
  const int slices = (int)dmm_ceil_div(n_out, 256);
  const int ns = slices <= 1 ? 1 : (slices == 2 ? 2 : 4);
  if (max_long > n_rows) max_long = n_rows;
  const int64_t long_blocks = dmm_ceil_div(max_long * ns, GS_WARPS);
  const int64_t blocks = long_blocks + dmm_ceil_div(n_rows, GS_WARPS);
  DMM_CHECK_ARG(blocks < (1LL << 31), "dmm_csr_gather_act_split: too many rows");
  cudaStream_t st = (cudaStream_t)stream;
#define DMM_GS_CALL(LO, WT) launch_gather_split<LO, WT>(ns, (unsigned)blocks, st, indptr, indices, vals, row_ids, order, n_long, \
                              (int)long_blocks, max_long, row0, n_rows, n_cols, wt_hi, wt_lo, ld_w, bias, act, n_out, h_hi, h_lo, \
                              ld_h, z_f32, ld_z)
  if (wt_lo) {
    if (vals) DMM_GS_CALL(true, true); else DMM_GS_CALL(true, false);
  } else {
    if (vals) DMM_GS_CALL(false, true); else DMM_GS_CALL(false, false);
  }
#undef DMM_GS_CALL
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_csr_axpy_bf16(dmm_ctx* ctx, const int64_t* indptr, const int32_t* indices, const int64_t* row_ids,
                                 int64_t row0, int64_t n_rows, int64_t n_cols, float beta, uint16_t* x_hi,
                                 uint16_t* x_lo, int64_t ld_x, void* stream) {
  DMM_CHECK_ARG(ctx && indptr && indices && x_hi, "dmm_csr_axpy_bf16: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_cols > 0 && ld_x >= n_cols, "dmm_csr_axpy_bf16: bad shape");
  if (n_rows == 0) return DMM_OK;
  csr_axpy_bf16_kernel<<<(unsigned)dmm_ceil_div(n_rows * 32, 256), 256, 0, (cudaStream_t)stream>>>(
      indptr, indices, row_ids, row0, n_rows, n_cols, beta, x_hi, x_lo, ld_x);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_bias_act_pack(dmm_ctx* ctx, const float* z, int64_t ld_z, const float* bias, int64_t n_rows,
                                 int64_t n_cols, int act, uint16_t* h_hi, uint16_t* h_lo, int64_t ld_h, void* stream) {
  DMM_CHECK_ARG(ctx && z && h_hi, "dmm_bias_act_pack: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_cols > 0 && ld_z >= n_cols && ld_h >= n_cols, "dmm_bias_act_pack: bad shape");
  DMM_CHECK_ARG(ld_z % 4 == 0 && ld_h % 4 == 0, "dmm_bias_act_pack: leading dimensions must be multiples of 4");
  DMM_CHECK_ARG(act == 0 || act == 1, "dmm_bias_act_pack: unknown activation %d", act);
  auto al = [](const void* q, uintptr_t a) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & (a - 1)) == 0; };
  DMM_CHECK_ARG(al(z, 16) && al(h_hi, 8) && al(h_lo, 8), "dmm_bias_act_pack: z must be 16-byte, h 8-byte aligned");
  if (n_rows == 0) return DMM_OK;
  const int64_t total = n_rows * ((n_cols + 3) / 4);
  int64_t blocks = dmm_ceil_div(total, 256);
  const int64_t cap = (int64_t)ctx->num_sms * 16;
  if (blocks > cap) blocks = cap;
  bias_act_pack_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(z, ld_z, bias, n_rows, n_cols, act, h_hi, h_lo, ld_h);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_gemv_f32(dmm_ctx* ctx, const float* w, int64_t ld_w, int64_t n_rows, int64_t K, const float* x,
                            float* y, void* stream) {
  DMM_CHECK_ARG(ctx && w && x && y, "dmm_gemv_f32: null argument");
  DMM_CHECK_ARG(n_rows > 0 && K > 0 && ld_w >= K, "dmm_gemv_f32: bad shape");
  DMM_CHECK_ARG(n_rows < (1LL << 31), "dmm_gemv_f32: too many rows");
  gemv_rows_kernel<<<(unsigned)n_rows, 128, 0, (cudaStream_t)stream>>>(w, ld_w, n_rows, K, x, y);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_rows_long_first(dmm_ctx* ctx, const int64_t* indptr, int64_t row0, int64_t n_rows, int64_t threshold,
                                   int32_t* order, int32_t* counters, void* stream) {
  DMM_CHECK_ARG(ctx && indptr && order && counters, "dmm_rows_long_first: null argument");
  DMM_CHECK_ARG(n_rows >= 0 && n_rows < (1LL << 31) && threshold >= 0 && threshold < (1LL << 31), "dmm_rows_long_first: bad sizes");
  if (n_rows == 0) return DMM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  DMM_CUDA(cudaMemsetAsync(counters, 0, 2 * sizeof(int32_t), st));
  rows_long_first_kernel<<<(unsigned)dmm_ceil_div(n_rows, 256), 256, 0, st>>>(indptr, row0, n_rows, (int)threshold, order, counters);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
