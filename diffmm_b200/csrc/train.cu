// Non-GEMM pieces of the fused Denoise training step (reference Model.py:385-428 + :183-220, driver Main.py:145-192).
//
// The step is hand-scheduled by diffmm_b200/train_step.py: twelve tensor-pipe contractions per modality and batch
// (dmm_gemm_bf16_tn) and the kernels below, which replace the per-op autograd chain of ATen elementwise kernels
// (q_sample -> fp32 x_t -> cat -> pack, sigmoid gate, mse / cosine tails, tanh', bias-gradient sums, transposes):
//
//   forward   dmm_train_prep        x_t = a_t x0 + b_t noise (Model.py:338-341) and the time-embedding columns
//                                   (Model.py:196-202) written DIRECTLY as the bf16 operand of the first layer
//                                   (no fp32 x_t, no torch.cat, no pack pass), plus x0 as a bf16 operand
//             dmm_gate_fwd          G = P * sigmoid(P Wg^T + bg)                     (Model.py:205-207)
//             dmm_diff_loss_fwd     mse_b, cosine similarity, per-row loss in float64 (Model.py:407-425)
//   backward  dmm_diff_loss_bwd     per-row seeds of the backward contractions
//             dmm_hidden_bwd        dz = c_b dh (1 - h^2) as operand, transposed operand, and (c_b h)^T
//             dmm_transpose_bf16    operand transposes for the weight-gradient contractions
//             dmm_colsum            bias gradients (deterministic column sums, optional per-row scale)
//             dmm_gate_bwd_pre      d(pre-sigmoid) of the gate
//             dmm_atb_small         X^T Y for skinny matrices (gate / time-embedding weight gradients)
#include "common.cuh"

namespace {

__device__ __forceinline__ void split_store(float x, uint16_t* hi, uint16_t* lo, int64_t i) {
  uint16_t h, l;
  dmm_split_bf16(x, h, l);
  hi[i] = h;
  if (lo) lo[i] = l;
}

// ---------------------------------------------------------------------------------------------- forward prep
__global__ void __launch_bounds__(256) train_prep_kernel(const float* __restrict__ x0, int64_t ld_x0,
                                                         const float* __restrict__ noise, int64_t ld_noise,
                                                         const int64_t* __restrict__ t, const float* __restrict__ tab_a,
                                                         const float* __restrict__ tab_b, int64_t n_cols, int d,
                                                         const float* __restrict__ emb_w, const float* __restrict__ emb_b,
                                                         uint16_t* __restrict__ a_hi, uint16_t* __restrict__ a_lo, int64_t ld_a,
                                                         uint16_t* __restrict__ x0_hi, int64_t ld_x0h,
                                                         float* __restrict__ te_raw) {
  const int64_t r = blockIdx.x;
  const int tid = threadIdx.x;
  const int64_t tt = t[r];
  const float ca = tab_a[tt], cb = tab_b[tt];
  const float* xr = x0 + r * ld_x0;
  const float* nr = noise + r * ld_noise;
  // two columns per thread: the bf16 pair leaves as one 32-bit store (ld_a is even, c is even)
  for (int64_t c = 2 * tid; c < n_cols; c += 512) {
    const bool two = c + 1 < n_cols;
    const float xa = xr[c], xb = two ? xr[c + 1] : 0.f;
    // Model.py:341 `x0_coef * x_0 + noise_coef * noise`: two roundings and an add, no contraction
    const float va = __fadd_rn(__fmul_rn(ca, xa), __fmul_rn(cb, nr[c]));
    const float vb = two ? __fadd_rn(__fmul_rn(ca, xb), __fmul_rn(cb, nr[c + 1])) : 0.f;
    uint16_t ha, la, hb, lb;
    dmm_split_bf16(va, ha, la);
    dmm_split_bf16(vb, hb, lb);
    if (two) {
      *reinterpret_cast<uint32_t*>(a_hi + r * ld_a + c) = (uint32_t)ha | ((uint32_t)hb << 16);
      if (a_lo) *reinterpret_cast<uint32_t*>(a_lo + r * ld_a + c) = (uint32_t)la | ((uint32_t)lb << 16);
      if (x0_hi)
        *reinterpret_cast<uint32_t*>(x0_hi + r * ld_x0h + c) = (uint32_t)dmm_bf16_bits(xa) | ((uint32_t)dmm_bf16_bits(xb) << 16);
    } else {
      a_hi[r * ld_a + c] = ha;
      if (a_lo) a_lo[r * ld_a + c] = la;
      if (x0_hi) x0_hi[r * ld_x0h + c] = dmm_bf16_bits(xa);
    }
  }
  // time embedding (Model.py:196-202) into the operand columns [n_cols, n_cols + d)
  if (tid < d) {
    const float ts = (float)tt;
    const int half = d / 2;
    float acc = emb_b[tid];
    for (int j = 0; j < d; ++j) {
      float e = 0.f;
      if (j < 2 * half) {
        const int jj = j < half ? j : j - half;
        const float f = expf(-logf(10000.f) * (float)jj / (float)half);
        e = j < half ? cosf(ts * f) : sinf(ts * f);
      }
      if (tid == 0 && te_raw) te_raw[r * d + j] = e;
      acc = fmaf(e, emb_w[tid * d + j], acc);
    }
    split_store(acc, a_hi, a_lo, r * ld_a + n_cols + tid);
  }
}

// ---------------------------------------------------------------------------------------------- gate
// One warp per row: lane l owns outputs l and l + 32.  Wg^T lives in shared memory ([k][j]: conflict-free for
// consecutive j); the row of P is broadcast by shuffle.
__global__ void __launch_bounds__(256) gate_fwd_kernel(const float* __restrict__ p, int64_t ld_p, int64_t n_rows,
                                                       const float* __restrict__ gate_w, const float* __restrict__ gate_b,
                                                       float* __restrict__ sig, uint16_t* __restrict__ g_hi,
                                                       uint16_t* __restrict__ g_lo, int64_t ld_g) {
  __shared__ float wt[64 * 64];
  for (int i = threadIdx.x; i < 64 * 64; i += 256) wt[(i & 63) * 64 + (i >> 6)] = gate_w[i];   // wt[k][j] = Wg[j][k]
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const float p0 = p[r * ld_p + lane], p1 = p[r * ld_p + 32 + lane];
  float a0 = gate_b[lane], a1 = gate_b[32 + lane];
#pragma unroll 8
  for (int k = 0; k < 64; ++k) {
    const float pk = __shfl_sync(0xffffffffu, k < 32 ? p0 : p1, k & 31);
    a0 = fmaf(pk, wt[k * 64 + lane], a0);
    a1 = fmaf(pk, wt[k * 64 + 32 + lane], a1);
  }
  const float s0 = 1.f / (1.f + expf(-a0)), s1 = 1.f / (1.f + expf(-a1));
  sig[r * 64 + lane] = s0;
  sig[r * 64 + 32 + lane] = s1;
  split_store(p0 * s0, g_hi, g_lo, r * ld_g + lane);
  split_store(p1 * s1, g_hi, g_lo, r * ld_g + 32 + lane);
}

// d_pre[b, j] = dG[b, j] * P[b, j] * s (1 - s)      (G = P * sigmoid(pre); P carries no parameter gradient)
__global__ void __launch_bounds__(256) gate_bwd_pre_kernel(const float* __restrict__ dg, int64_t ld_dg,
                                                           const float* __restrict__ p, int64_t ld_p,
                                                           const float* __restrict__ sig, int64_t n_rows,
                                                           float* __restrict__ dpre) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_rows * 64) return;
  const int64_t r = i >> 6;
  const int j = (int)(i & 63);
  const float s = sig[i];
  dpre[i] = dg[r * ld_dg + j] * p[r * ld_p + j] * s * (1.f - s);
}

// ---------------------------------------------------------------------------------------------- loss tail
// One CTA of 128 threads per row.  diff = out - x0 (fp32, from the second layer's epilogue), um = diff F + x0 F.
__global__ void __launch_bounds__(128) diff_loss_fwd_kernel(const float* __restrict__ diff, int64_t ld_d, int64_t n_cols,
                                                            const float* __restrict__ umd, int64_t ld_umd,
                                                            const float* __restrict__ x0f, int64_t ld_x0f,
                                                            const float* __restrict__ ui, int64_t ld_ui,
                                                            const int64_t* __restrict__ t, const double* __restrict__ w_tab,
                                                            float sim_weight, double* __restrict__ loss,
                                                            float* __restrict__ mse_out, float* __restrict__ um_out,
                                                            float* __restrict__ stats) {
  __shared__ float red[4];
  __shared__ float red3[3][2];
  const int64_t r = blockIdx.x;
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const float* dr = diff + r * ld_d;
  float ss = 0.f;
  if ((reinterpret_cast<uintptr_t>(dr) & 15u) == 0) {
    const int64_t n4 = n_cols >> 2;
    const float4* d4 = reinterpret_cast<const float4*>(dr);
#pragma unroll 4
    for (int64_t i = tid; i < n4; i += 128) {
      const float4 q = d4[i];
      ss = fmaf(q.x, q.x, ss);
      ss = fmaf(q.y, q.y, ss);
      ss = fmaf(q.z, q.z, ss);
      ss = fmaf(q.w, q.w, ss);
    }
    for (int64_t i = (n4 << 2) + tid; i < n_cols; i += 128) ss = fmaf(dr[i], dr[i], ss);
  } else {
    for (int64_t i = tid; i < n_cols; i += 128) ss = fmaf(dr[i], dr[i], ss);
  }
  ss = dmm_warp_sum(ss);
  if (lane == 0) red[w] = ss;
  float dot = 0.f, nu = 0.f, ni = 0.f;
  if (tid < 64) {
    const float u = umd[r * ld_umd + tid] + x0f[r * ld_x0f + tid];
    const float v = ui[r * ld_ui + tid];
    um_out[r * 64 + tid] = u;
    dot = u * v;
    nu = u * u;
    ni = v * v;
  }
  if (w < 2) {
    dot = dmm_warp_sum(dot);
    nu = dmm_warp_sum(nu);
    ni = dmm_warp_sum(ni);
    if (lane == 0) {
      red3[0][w] = dot;
      red3[1][w] = nu;
      red3[2][w] = ni;
    }
  }
  __syncthreads();
  if (tid == 0) {
    const float mse = ((red[0] + red[1]) + (red[2] + red[3])) / (float)n_cols;
    const float d = red3[0][0] + red3[0][1];
    const float a = sqrtf(red3[1][0] + red3[1][1]), b = sqrtf(red3[2][0] + red3[2][1]);
    const float cosv = d / (fmaxf(a, 1e-8f) * fmaxf(b, 1e-8f));      // F.cosine_similarity, eps = 1e-8
    const float sim = 1.f - cosv;
    // Model.py:413,425: float64 weight times the fp32 mse, plus the fp32 product sim * sim_weight
    loss[r] = w_tab[t[r]] * (double)mse + (double)(sim * sim_weight);
    mse_out[r] = mse;
    stats[3 * r + 0] = d;
    stats[3 * r + 1] = a;
    stats[3 * r + 2] = b;
  }
}

// One warp per row (lane owns columns lane and lane + 32 of the 64-wide embeddings).
//   cm[b]   = g_b w_b 2 / I                       (d loss / d out = cm (out - x0) + d_um F^T)
//   dumc    = d_um / cm  as a bf16 operand        (d_out' = diff + dumc F^T, the row scale cm is applied downstream)
//   d_ui    = d loss / d ui (optional)
__global__ void __launch_bounds__(256) diff_loss_bwd_kernel(const double* __restrict__ g_loss, const float* __restrict__ um,
                                                            const float* __restrict__ ui, int64_t ld_ui,
                                                            const float* __restrict__ stats, const int64_t* __restrict__ t,
                                                            const double* __restrict__ w_tab, float sim_weight,
                                                            int64_t n_cols, int64_t n_rows, float* __restrict__ cm,
                                                            uint16_t* __restrict__ dumc_hi, uint16_t* __restrict__ dumc_lo,
                                                            int64_t ld_dumc, float* __restrict__ d_ui) {
  const int lane = threadIdx.x & 31;
  const int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= n_rows) return;
  const double g = g_loss[r];
  const float c = (float)(g * w_tab[t[r]] * 2.0 / (double)n_cols);
  const float gs = (float)g * sim_weight;                 // d loss / d sim
  const float d = stats[3 * r], a = stats[3 * r + 1], b = stats[3 * r + 2];
  const float ac = fmaxf(a, 1e-8f), bc = fmaxf(b, 1e-8f);
  const float cosv = d / (ac * bc);
  if (lane == 0) cm[r] = c;
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int k = lane + 32 * h;
    const float u = um[r * 64 + k], v = ui[r * ld_ui + k];
    // d cos / d um = ui / (ac bc) - cos um / (ac a)   (second term vanishes when the norm is clamped)
    float dcos_du = v / (ac * bc);
    if (a > 1e-8f) dcos_du -= cosv * u / (ac * a);
    float dcos_dv = u / (ac * bc);
    if (b > 1e-8f) dcos_dv -= cosv * v / (bc * b);
    const float dum = -gs * dcos_du;
    split_store(c != 0.f ? dum / c : 0.f, dumc_hi, dumc_lo, r * ld_dumc + k);
    if (d_ui) d_ui[r * 64 + k] = -gs * dcos_dv;
  }
}

// ---------------------------------------------------------------------------------------------- hidden layer backward
// 32 x 32 tiles: dz[b, h] = cm[b] dh[b, h] (1 - hv^2), hv = h_hi (+ h_lo).  Writes dz fp32 (bias gradient source), dz as
// the operand of the input-gradient contraction, and through a shared-memory transpose dz^T and (cm h)^T, the operands
// of the two weight-gradient contractions (K = batch).  cm == NULL: no row scale (cm = 1, so (cm h)^T is h^T).
__global__ void __launch_bounds__(256) hidden_bwd_kernel(const float* __restrict__ dh, int64_t ld_dh,
                                                         const float* __restrict__ h_f32, int64_t ld_hf,
                                                         const uint16_t* __restrict__ h_hi, const uint16_t* __restrict__ h_lo,
                                                         int64_t ld_h, const float* __restrict__ cm, int64_t n_rows, int64_t H,
                                                         float* __restrict__ dz_f32, int64_t ld_dz,
                                                         uint16_t* __restrict__ dz_hi, uint16_t* __restrict__ dz_lo, int64_t ld_dz16,
                                                         uint16_t* __restrict__ dzt_hi, uint16_t* __restrict__ dzt_lo,
                                                         uint16_t* __restrict__ hct_hi, uint16_t* __restrict__ hct_lo,
                                                         int64_t ld_t) {
  __shared__ float s_dz[32][33];
  __shared__ float s_hc[32][33];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;      // 32 x 8
  const int64_t b0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t b = b0 + ty + 8 * i, c = c0 + tx;
    float dz = 0.f, hc = 0.f;
    if (b < n_rows && c < H) {
      // tanh' = 1 - h^2 needs h at full precision: for a saturated unit (|h| -> 1) the bf16 rounding of h (2^-9) is as
      // large as 1 - h^2 itself
      float hv;
      if (h_f32) {
        hv = h_f32[b * ld_hf + c];
      } else {
        hv = dmm_bf16_to_f32(h_hi[b * ld_h + c]);
        if (h_lo) hv += dmm_bf16_to_f32(h_lo[b * ld_h + c]);
      }
      const float s = cm ? cm[b] : 1.f;
      dz = s * dh[b * ld_dh + c] * (1.f - hv * hv);
      hc = s * hv;
      dz_f32[b * ld_dz + c] = dz;
      split_store(dz, dz_hi, dz_lo, b * ld_dz16 + c);
    }
    s_dz[ty + 8 * i][tx] = dz;
    s_hc[ty + 8 * i][tx] = hc;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t c = c0 + ty + 8 * i, b = b0 + tx;      // transposed: row = hidden column, col = batch row
    if (c < H && b < ld_t) {                              // batch columns up to ld_t are written (zeros beyond n_rows)
      split_store(s_dz[tx][ty + 8 * i], dzt_hi, dzt_lo, c * ld_t + b);
      split_store(s_hc[tx][ty + 8 * i], hct_hi, hct_lo, c * ld_t + b);
    }
  }
}

// dst[c, r] = src[r, c] for 16-bit elements (hi and optionally lo), 32 x 32 tiles
__global__ void __launch_bounds__(256) transpose_bf16_kernel(const uint16_t* __restrict__ s_hi, const uint16_t* __restrict__ s_lo,
                                                             int64_t ld_s, int64_t R, int64_t C, uint16_t* __restrict__ d_hi,
                                                             uint16_t* __restrict__ d_lo, int64_t ld_d) {
  __shared__ uint16_t th[32][34];
  __shared__ uint16_t tl[32][34];
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
  const int64_t r0 = (int64_t)blockIdx.y * 32, c0 = (int64_t)blockIdx.x * 32;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t r = r0 + ty + 8 * i, c = c0 + tx;
    const bool in = r < R && c < C;
    th[ty + 8 * i][tx] = in ? s_hi[r * ld_s + c] : (uint16_t)0;
    if (s_lo) tl[ty + 8 * i][tx] = in ? s_lo[r * ld_s + c] : (uint16_t)0;
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int64_t c = c0 + ty + 8 * i, r = r0 + tx;
    if (c < C && r < ld_d) {
      d_hi[c * ld_d + r] = th[tx][ty + 8 * i];
      if (d_lo) d_lo[c * ld_d + r] = tl[tx][ty + 8 * i];
    }
  }
}

// out[c] = sum_r scale[r] * src[r, c]: one thread per column, rows in order (deterministic); R is a batch (~1024)
__global__ void __launch_bounds__(128) colsum_kernel(const float* __restrict__ src, int64_t ld, int64_t R, int64_t C,
                                                     const float* __restrict__ scale, float* __restrict__ out) {
  const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
  int64_t r = 0;
  for (; r + 3 < R; r += 4) {
    const float s0 = scale ? scale[r] : 1.f, s1 = scale ? scale[r + 1] : 1.f, s2 = scale ? scale[r + 2] : 1.f,
                s3 = scale ? scale[r + 3] : 1.f;
    a0 = fmaf(s0, src[r * ld + c], a0);
    a1 = fmaf(s1, src[(r + 1) * ld + c], a1);
    a2 = fmaf(s2, src[(r + 2) * ld + c], a2);
    a3 = fmaf(s3, src[(r + 3) * ld + c], a3);
  }
  for (; r < R; ++r) a0 = fmaf(scale ? scale[r] : 1.f, src[r * ld + c], a0);
  out[c] = (a0 + a1) + (a2 + a3);
}

// out[i, j] = sum_r x[r, i] y[r, j] for skinny x [R, m], y [R, n] (m, n <= 64): grid (m, S) partial sums over row
// slices, then a fixed-order sum of the S partials (deterministic, no atomics)
constexpr int ATB_SPLIT = 8;
__global__ void __launch_bounds__(256) atb_partial_kernel(const float* __restrict__ x, int64_t ld_x, const float* __restrict__ y,
                                                          int64_t ld_y, int64_t R, int m, int n, float* __restrict__ part) {
  __shared__ float red[4][64];
  const int i = blockIdx.x, s = blockIdx.y;
  const int j = threadIdx.x & 63, g = threadIdx.x >> 6;
  const int64_t per = (R + ATB_SPLIT - 1) / ATB_SPLIT;
  const int64_t r0 = s * per, r1 = (r0 + per < R) ? r0 + per : R;
  float acc = 0.f;
  if (j < n)
    for (int64_t r = r0 + g; r < r1; r += 4) acc = fmaf(x[r * ld_x + i], y[r * ld_y + j], acc);
  red[g][j] = acc;
  __syncthreads();
  if (g == 0 && j < n) part[((int64_t)s * m + i) * n + j] = (red[0][j] + red[1][j]) + (red[2][j] + red[3][j]);
}
__global__ void __launch_bounds__(256) atb_reduce_kernel(const float* __restrict__ part, int m, int n, float* __restrict__ out) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m * n) return;
  float acc = 0.f;
#pragma unroll
  for (int s = 0; s < ATB_SPLIT; ++s) acc += part[(int64_t)s * m * n + idx];
  out[idx] = acc;
}

}  // namespace

extern "C" int dmm_train_prep(dmm_ctx* ctx, const float* x0, int64_t ld_x0, const float* noise, int64_t ld_noise,
                              const int64_t* t, const float* tab_a, const float* tab_b, int64_t n_rows, int64_t n_cols,
                              int d_emb, const float* emb_w, const float* emb_b, uint16_t* a_hi, uint16_t* a_lo, int64_t ld_a,
                              uint16_t* x0_hi, int64_t ld_x0h, float* te_raw, void* stream) {
  DMM_CHECK_ARG(ctx && x0 && noise && t && tab_a && tab_b && emb_w && emb_b && a_hi, "dmm_train_prep: null argument");
  DMM_CHECK_ARG(n_cols > 0 && ld_x0 >= n_cols && ld_noise >= n_cols, "dmm_train_prep: bad shape");
  DMM_CHECK_ARG(d_emb >= 2 && d_emb <= 64, "dmm_train_prep: d_emb must be in [2, 64]");
  DMM_CHECK_ARG(ld_a >= n_cols + d_emb && ld_a % 2 == 0 && (!x0_hi || (ld_x0h >= n_cols && ld_x0h % 2 == 0)),
                "dmm_train_prep: operand leading dimensions must be even and cover the columns");
  if (n_rows <= 0) return DMM_OK;
  train_prep_kernel<<<(unsigned)n_rows, 256, 0, (cudaStream_t)stream>>>(x0, ld_x0, noise, ld_noise, t, tab_a, tab_b, n_cols, d_emb,
                                                                       emb_w, emb_b, a_hi, a_lo, ld_a, x0_hi, ld_x0h, te_raw);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_gate_fwd(dmm_ctx* ctx, const float* p, int64_t ld_p, int64_t n_rows, const float* gate_w, const float* gate_b,
                            float* sig, uint16_t* g_hi, uint16_t* g_lo, int64_t ld_g, void* stream) {
  DMM_CHECK_ARG(ctx && p && gate_w && gate_b && sig && g_hi, "dmm_gate_fwd: null argument");
  DMM_CHECK_ARG(ld_p >= 64 && ld_g >= 64, "dmm_gate_fwd: the gate is 64 wide (latdim)");
  if (n_rows <= 0) return DMM_OK;
  gate_fwd_kernel<<<(unsigned)dmm_ceil_div(n_rows, 8), 256, 0, (cudaStream_t)stream>>>(p, ld_p, n_rows, gate_w, gate_b, sig, g_hi,
                                                                                      g_lo, ld_g);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_gate_bwd_pre(dmm_ctx* ctx, const float* dg, int64_t ld_dg, const float* p, int64_t ld_p, const float* sig,
                                int64_t n_rows, float* dpre, void* stream) {
  DMM_CHECK_ARG(ctx && dg && p && sig && dpre, "dmm_gate_bwd_pre: null argument");
  if (n_rows <= 0) return DMM_OK;
  gate_bwd_pre_kernel<<<(unsigned)dmm_ceil_div(n_rows * 64, 256), 256, 0, (cudaStream_t)stream>>>(dg, ld_dg, p, ld_p, sig, n_rows,
                                                                                                 dpre);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_diff_loss_fwd(dmm_ctx* ctx, const float* diff, int64_t ld_d, int64_t n_rows, int64_t n_cols, const float* umd,
                                 int64_t ld_umd, const float* x0f, int64_t ld_x0f, const float* ui, int64_t ld_ui,
                                 const int64_t* t, const double* w_tab, float sim_weight, double* loss, float* mse, float* um,
                                 float* stats, void* stream) {
  DMM_CHECK_ARG(ctx && diff && umd && x0f && ui && t && w_tab && loss && mse && um && stats, "dmm_diff_loss_fwd: null argument");
  DMM_CHECK_ARG(n_cols > 0 && ld_d >= n_cols, "dmm_diff_loss_fwd: bad shape");
  if (n_rows <= 0) return DMM_OK;
  diff_loss_fwd_kernel<<<(unsigned)n_rows, 128, 0, (cudaStream_t)stream>>>(diff, ld_d, n_cols, umd, ld_umd, x0f, ld_x0f, ui, ld_ui,
                                                                          t, w_tab, sim_weight, loss, mse, um, stats);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_diff_loss_bwd(dmm_ctx* ctx, const double* g_loss, const float* um, const float* ui, int64_t ld_ui,
                                 const float* stats, const int64_t* t, const double* w_tab, float sim_weight, int64_t n_rows,
                                 int64_t n_cols, float* cm, uint16_t* dumc_hi, uint16_t* dumc_lo, int64_t ld_dumc, float* d_ui,
                                 void* stream) {
  DMM_CHECK_ARG(ctx && g_loss && um && ui && stats && t && w_tab && cm && dumc_hi, "dmm_diff_loss_bwd: null argument");
  DMM_CHECK_ARG(ld_dumc >= 64 && n_cols > 0, "dmm_diff_loss_bwd: bad shape");
  if (n_rows <= 0) return DMM_OK;
  diff_loss_bwd_kernel<<<(unsigned)dmm_ceil_div(n_rows, 8), 256, 0, (cudaStream_t)stream>>>(
      g_loss, um, ui, ld_ui, stats, t, w_tab, sim_weight, n_cols, n_rows, cm, dumc_hi, dumc_lo, ld_dumc, d_ui);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_hidden_bwd(dmm_ctx* ctx, const float* dh, int64_t ld_dh, const float* h_f32, int64_t ld_hf,
                              const uint16_t* h_hi, const uint16_t* h_lo,
                              int64_t ld_h, const float* cm, int64_t n_rows, int64_t H, float* dz_f32, int64_t ld_dz,
                              uint16_t* dz_hi, uint16_t* dz_lo, int64_t ld_dz16, uint16_t* dzt_hi, uint16_t* dzt_lo,
                              uint16_t* hct_hi, uint16_t* hct_lo, int64_t ld_t, void* stream) {
  DMM_CHECK_ARG(ctx && dh && (h_hi || h_f32) && dz_f32 && dz_hi && dzt_hi && hct_hi, "dmm_hidden_bwd: null argument");
  DMM_CHECK_ARG(H > 0 && ld_dh >= H && (!h_hi || ld_h >= H) && (!h_f32 || ld_hf >= H) && ld_dz >= H && ld_dz16 >= H && ld_t >= n_rows,
                "dmm_hidden_bwd: bad shape");
  DMM_CHECK_ARG(!!dz_lo == !!dzt_lo && !!dz_lo == !!hct_lo, "dmm_hidden_bwd: lo parts must be given together");
  if (n_rows <= 0) return DMM_OK;
  dim3 grid((unsigned)dmm_ceil_div(H, 32), (unsigned)dmm_ceil_div(ld_t, 32));
  hidden_bwd_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(dh, ld_dh, h_f32, ld_hf, h_hi, h_lo, ld_h, cm, n_rows, H, dz_f32, ld_dz, dz_hi, dz_lo,
                                                           ld_dz16, dzt_hi, dzt_lo, hct_hi, hct_lo, ld_t);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_transpose_bf16(dmm_ctx* ctx, const uint16_t* src_hi, const uint16_t* src_lo, int64_t ld_src, int64_t rows,
                                  int64_t cols, uint16_t* dst_hi, uint16_t* dst_lo, int64_t ld_dst, void* stream) {
  DMM_CHECK_ARG(ctx && src_hi && dst_hi, "dmm_transpose_bf16: null argument");
  DMM_CHECK_ARG(rows > 0 && cols > 0 && ld_src >= cols && ld_dst >= rows && (!src_lo == !dst_lo),
                "dmm_transpose_bf16: bad shape (lo parts must be given together)");
  dim3 grid((unsigned)dmm_ceil_div(cols, 32), (unsigned)dmm_ceil_div(ld_dst, 32));
  transpose_bf16_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src_hi, src_lo, ld_src, rows, cols, dst_hi, dst_lo, ld_dst);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_colsum(dmm_ctx* ctx, const float* src, int64_t ld, int64_t rows, int64_t cols, const float* row_scale,
                          float* out, void* stream) {
  // rows == 0 (an empty batch) is a valid call that writes zeros; an empty tensor has no storage, so src may be NULL then
  DMM_CHECK_ARG(ctx && (src || rows == 0) && out, "dmm_colsum: null argument");
  DMM_CHECK_ARG(rows >= 0 && cols > 0 && ld >= cols, "dmm_colsum: bad shape");
  colsum_kernel<<<(unsigned)dmm_ceil_div(cols, 128), 128, 0, (cudaStream_t)stream>>>(src, ld, rows, cols, row_scale, out);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int64_t dmm_atb_small_workspace_floats(int64_t m, int64_t n) { return (int64_t)ATB_SPLIT * m * n; }

extern "C" int dmm_atb_small(dmm_ctx* ctx, const float* x, int64_t ld_x, int64_t m, const float* y, int64_t ld_y, int64_t n,
                             int64_t rows, float* workspace, float* out, void* stream) {
  DMM_CHECK_ARG(ctx && ((x && y) || rows == 0) && workspace && out, "dmm_atb_small: null argument");   // as dmm_colsum
  DMM_CHECK_ARG(m >= 1 && m <= 64 && n >= 1 && n <= 64 && ld_x >= m && ld_y >= n && rows >= 0, "dmm_atb_small: m, n must be in [1, 64]");
  cudaStream_t st = (cudaStream_t)stream;
  atb_partial_kernel<<<dim3((unsigned)m, ATB_SPLIT), 256, 0, st>>>(x, ld_x, y, ld_y, rows, (int)m, (int)n, workspace);
  DMM_LAUNCH_CHECK();
  atb_reduce_kernel<<<(unsigned)dmm_ceil_div(m * n, 256), 256, 0, st>>>(workspace, (int)m, (int)n, out);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
