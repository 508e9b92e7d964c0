// Fused BPR and in-batch InfoNCE losses (forward + backward) with warp-shuffle reductions.
//
// Replaces Utils/Utils.py:57-98 (gathers, F.normalize, a B x B logits GEMM, log_softmax, diag, and
// the autograd graph behind them).  The B x B matrix is never written to HBM: every warp owns one
// anchor row, keeps its normalised vector in registers, streams the other view's normalised rows
// (B x D fp32 = 256 KB at B = 1024, L2/L1 resident) and folds them into an online log-sum-exp.
// Means are reduced in a fixed order (per-row scratch + single-CTA tree) so results are bitwise
// reproducible run to run.
#include "common.cuh"

namespace {

constexpr int MAX_D = 256;  // D <= 256: up to 8 elements per lane

__global__ void __launch_bounds__(1024) mean_reduce_kernel(const float* __restrict__ v, int64_t n, float scale,
                                                           float* __restrict__ out) {
  __shared__ float red[32];
  float s = 0.f;
  for (int64_t i = threadIdx.x; i < n; i += 1024) s += v[i];
  s = dmm_warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = red[threadIdx.x];
    t = dmm_warp_sum(t);
    if (threadIdx.x == 0) *out = t * scale;
  }
}

// ------------------------------------------------------------------------------------------ BPR
// Utils/Utils.py:92-98: loss_b = -log(1e-5 + sigmoid(u.p - u.n)); d loss_b/dx = -s(1-s)/(1e-5+s)
__global__ void __launch_bounds__(256) bpr_kernel(const float* __restrict__ ue, int64_t ld_u,
                                                  const float* __restrict__ ie, int64_t ld_i,
                                                  const int64_t* __restrict__ users, const int64_t* __restrict__ pos,
                                                  const int64_t* __restrict__ neg, int64_t B, int D, float gscale,
                                                  float* __restrict__ row_loss, float* __restrict__ g_u,
                                                  float* __restrict__ g_p, float* __restrict__ g_n) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* u = ue + users[b] * ld_u;
  const float* p = ie + pos[b] * ld_i;
  const float* n = ie + neg[b] * ld_i;
  float dp = 0.f, dn = 0.f;
  for (int c = lane; c < D; c += 32) {
    const float uv = __ldg(u + c);
    dp = fmaf(uv, __ldg(p + c), dp);
    dn = fmaf(uv, __ldg(n + c), dn);
  }
  dp = dmm_warp_sum(dp);
  dn = dmm_warp_sum(dn);
  const float x = dp - dn;
  const float s = 1.f / (1.f + expf(-x));
  if (lane == 0) row_loss[b] = -logf(10e-6f + s);
  if (g_u) {
    const float d = -(s * (1.f - s)) / (10e-6f + s) * gscale;  // gscale = upstream grad / B
    for (int c = lane; c < D; c += 32) {
      const float uv = __ldg(u + c), pv = __ldg(p + c), nv = __ldg(n + c);
      g_u[b * D + c] = d * (pv - nv);
      g_p[b * D + c] = d * uv;
      g_n[b * D + c] = -d * uv;
    }
  }
}

// ------------------------------------------------------------------------------------------ InfoNCE
// gathers rows idx[b] of both views, L2-normalises (eps 1e-12), writes n1/n2 [B, D] and inverse norms
__global__ void __launch_bounds__(256) nce_gather_norm_kernel(const float* __restrict__ v1, int64_t ld1,
                                                              const float* __restrict__ v2, int64_t ld2,
                                                              const int64_t* __restrict__ idx, int64_t B, int D,
                                                              float* __restrict__ n1, float* __restrict__ n2,
                                                              float* __restrict__ inv1, float* __restrict__ inv2) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const float* a = v1 + idx[b] * ld1;
  const float* c = v2 + idx[b] * ld2;
  float s1 = 0.f, s2 = 0.f;
  for (int k = lane; k < D; k += 32) {
    const float x = __ldg(a + k), y = __ldg(c + k);
    s1 = fmaf(x, x, s1);
    s2 = fmaf(y, y, s2);
  }
  s1 = dmm_warp_sum(s1);
  s2 = dmm_warp_sum(s2);
  const float i1 = 1.f / fmaxf(sqrtf(s1), 1e-12f), i2 = 1.f / fmaxf(sqrtf(s2), 1e-12f);
  for (int k = lane; k < D; k += 32) {
    n1[b * D + k] = __ldg(a + k) * i1;
    n2[b * D + k] = __ldg(c + k) * i2;
  }
  if (lane == 0 && inv1) {
    inv1[b] = i1;
    inv2[b] = i2;
  }
}

// One warp per anchor row i of `na` against all rows j of `nb` (both normalised [B, D]).
//   MODE 0 (forward):  lse_i = logsumexp_j(a_i.b_j / T);  row_loss_i = lse_i - a_i.b_i / T
//   MODE 1 (backward wrt a): ga_i = sum_j (p_ij - [i==j]) b_j * c,   p_ij = exp(a_i.b_j / T - lse_i)
//   MODE 2 (backward wrt b): gb_i = sum_j (p_ji - [i==j]) a_j * c,   p_ji = exp(a_j.b_i / T - lse_j)
//     (called with na/nb swapped: the anchor is b_i and the stream is a_j; lse is indexed by j)
// followed, for MODE 1/2, by the normalisation backward g_x = inv * (g - n (n.g)).
template <int MODE, int EPL /* elements per lane = D / 32 */>
__global__ void __launch_bounds__(256) nce_rows_kernel(const float* __restrict__ na, const float* __restrict__ nb,
                                                       int64_t B, float inv_temp, const float* __restrict__ lse_in,
                                                       const float* __restrict__ inv_norm, float coef,
                                                       float* __restrict__ out_lse, float* __restrict__ out_row_loss,
                                                       float* __restrict__ out_grad) {
  const int64_t i = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (i >= B) return;
  constexpr int D = EPL * 32;
  float a[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) a[e] = __ldg(na + i * D + lane + 32 * e);
  float m = -INFINITY, l = 0.f, diag = 0.f;
  float g[EPL];
#pragma unroll
  for (int e = 0; e < EPL; ++e) g[e] = 0.f;
  const float lse_i = (MODE == 1) ? lse_in[i] : 0.f;

  for (int64_t j0 = 0; j0 < B; j0 += 4) {
    float bv[4][EPL], s[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t j = j0 + q < B ? j0 + q : B - 1;
#pragma unroll
      for (int e = 0; e < EPL; ++e) bv[q][e] = __ldg(nb + j * D + lane + 32 * e);
      float d = 0.f;
#pragma unroll
      for (int e = 0; e < EPL; ++e) d = fmaf(a[e], bv[q][e], d);
      s[q] = d;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
#pragma unroll
      for (int q = 0; q < 4; ++q) s[q] += __shfl_xor_sync(0xffffffffu, s[q], o);
    }
#pragma unroll
    for (int q = 0; q < 4; ++q) {
      const int64_t j = j0 + q;
      if (j >= B) break;
      const float sc = s[q] * inv_temp;
      if (MODE == 0) {
        if (j == i) diag = sc;
        const float mn = fmaxf(m, sc);
        l = l * expf(m - mn) + expf(sc - mn);
        m = mn;
      } else {
        const float lse = (MODE == 1) ? lse_i : __ldg(lse_in + j);
        const float w = expf(sc - lse) - (j == i ? 1.f : 0.f);
#pragma unroll
        for (int e = 0; e < EPL; ++e) g[e] = fmaf(w, bv[q][e], g[e]);
      }
    }
  }
  if (MODE == 0) {
    if (lane == 0) {
      const float lse = m + logf(l);
      out_lse[i] = lse;
      out_row_loss[i] = lse - diag;
    }
  } else {
    // normalisation backward: x = raw row, n = x * inv;  g_x = inv * (g - n (n . g)) * coef
    float dot = 0.f;
#pragma unroll
    for (int e = 0; e < EPL; ++e) dot = fmaf(a[e], g[e], dot);
    dot = dmm_warp_sum(dot);
    const float sc = inv_norm[i] * coef;
#pragma unroll
    for (int e = 0; e < EPL; ++e) out_grad[i * D + lane + 32 * e] = sc * (g[e] - a[e] * dot);
  }
}

// ---- D == 64: register-tiled version ----------------------------------------------------------------
// The warp-per-anchor kernel above spends its time in shuffle reductions (one 5-step butterfly per logit).
// Here the B x B logit matrix is cut into CTA tiles of NT_I = 32 anchors x a range of stream rows: the grid is
// (B / 32 anchor tiles) x (JS column splits) so that ~128 CTAs are busy at B = 1024 instead of 64, and a CTA walks its
// range in tiles of NT_J = 64 stream rows staged in shared memory by cp.async (double buffered: the next tile lands
// while this one is consumed).  Thread (ty, tx) of 8 x 16 owns the 4 x 4 logits (4 ty + rr, tx + 16 q): 8 shared
// float4 reads feed 64 FMAs, i.e. the FP32 pipe, not shared-memory bandwidth, bounds the tile.
//   forward : per-split online log-sum-exp (m, l) and the diagonal logit of every anchor -> nce_fwd_combine_kernel
//             merges the splits, writes lse / row losses and reduces the mean in a fixed order;
//   backward: w_ij = exp(s_ij / T - lse) - [i == j] goes through shared memory (transposed, one float4 of 4 anchors per
//             stream row) into a second register-tiled product  g(4 anchors, 4 components) += w . B;  blockIdx.z picks
//             the side (1: d/d v1 with lse of the anchor; 2: d/d v2, anchors and stream swapped, lse of the stream row);
//             the per-split partial gradients are added in a fixed order by nce_bwd_combine_kernel, which also applies
//             the normalisation backward  g_x = inv (g - n (n . g)) coef.   Everything is deterministic.
constexpr int NT_I = 32, NT_J = 64, NT_LD = 68, NT_PLD = 36, NT_THREADS = 128, NCE_MAX_SPLIT = 4;
struct NceSmem {
  float As[NT_I][NT_LD];        // anchors, 68-float rows: 16-byte aligned, conflict-free float4 column walks
  float Bs[2][NT_J][NT_LD];     // stream tile, double buffered
  float Ps[NT_J][NT_PLD];       // backward: w transposed [stream row][anchor]
  float lse_s[2][NT_J];         // backward wrt v2: lse of the stream rows
};

__device__ __forceinline__ void cp_async16(void* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src),
               "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async4(void* dst, const void* src, int src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(dst)), "l"(src),
               "r"(src_bytes)
               : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// Batch of InfoNCE problems sharing one launch (blockIdx.z = problem, or 2 * problem + side in the backward): problem p
// keeps its normalised gathers at n_base + p * 2 B 64 (view 1, then view 2), its lse at lse_base + p B, its forward
// partials at part_base + p * B JS 3 and its backward partials at gpart_base + p * 2 JS B 64.
constexpr int NCE_MAX_PROBLEMS = 12;
struct NceBatch {
  float inv_temp[NCE_MAX_PROBLEMS];
};

template <bool FWD>
__global__ void __launch_bounds__(NT_THREADS) nce_tiles_kernel(const float* __restrict__ n_base, int64_t B, int64_t JR,
                                                               const NceBatch nb_par, const float* __restrict__ lse_base,
                                                               float* __restrict__ part_base, float* __restrict__ gpart_base) {
  extern __shared__ __align__(16) uint8_t nce_raw[];
  NceSmem& sm = *reinterpret_cast<NceSmem*>(nce_raw);
  const int prob = FWD ? (int)blockIdx.z : (int)(blockIdx.z >> 1);
  const int mode = FWD ? 0 : 1 + (int)(blockIdx.z & 1);
  const float inv_temp = nb_par.inv_temp[prob];
  const float* __restrict__ n1 = n_base + (int64_t)prob * 2 * B * 64;
  const float* __restrict__ n2 = n1 + B * 64;
  const float* __restrict__ lse = lse_base ? lse_base + (int64_t)prob * B : nullptr;
  float* __restrict__ part = part_base ? part_base + (int64_t)prob * B * gridDim.y * 3 : nullptr;
  float* __restrict__ gpart = gpart_base ? gpart_base + (int64_t)prob * 2 * gridDim.y * B * 64 : nullptr;
  const float* __restrict__ na = (mode == 2) ? n2 : n1;   // anchors
  const float* __restrict__ nb = (mode == 2) ? n1 : n2;   // stream
  const int tid = threadIdx.x, ty = tid >> 4, tx = tid & 15;
  const uint32_t hmask = 0xFFFFu << (tid & 16);           // the 16 threads of an anchor quad are one half warp
  const int64_t i0 = (int64_t)blockIdx.x * NT_I;
  const int split = blockIdx.y, JS = gridDim.y;
  const int64_t jbeg = (int64_t)split * JR;
  const int64_t jend = jbeg + JR < B ? jbeg + JR : B;
  const int ntiles = jbeg < jend ? (int)((jend - jbeg + NT_J - 1) / NT_J) : 0;

  auto issue = [&](int t) {
    const int st = t & 1;
    const int64_t j0 = jbeg + (int64_t)t * NT_J;
#pragma unroll
    for (int k = 0; k < NT_J * 16 / NT_THREADS; ++k) {
      const int idx = tid + NT_THREADS * k;
      const int row = idx >> 4, pc = idx & 15;
      const bool ok = j0 + row < jend;
      cp_async16(&sm.Bs[st][row][4 * pc], nb + (ok ? j0 + row : 0) * 64 + 4 * pc, ok ? 16 : 0);   // rows past the range: zeros
    }
    if (mode == 2 && tid < NT_J) {
      const bool ok = j0 + tid < jend;
      cp_async4(&sm.lse_s[st][tid], lse + (ok ? j0 + tid : 0), ok ? 4 : 0);
    }
  };
  if (ntiles > 0) issue(0);
  cp_async_commit();
#pragma unroll
  for (int k = 0; k < NT_I * 16 / NT_THREADS; ++k) {
    const int idx = tid + NT_THREADS * k;
    const int row = idx >> 4, pc = idx & 15;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (i0 + row < B) v = __ldg(reinterpret_cast<const float4*>(na + (i0 + row) * 64) + pc);
    *reinterpret_cast<float4*>(&sm.As[row][4 * pc]) = v;
  }

  float m[4], l[4], diag[4], lse_i[4];
  float g[4][4];
#pragma unroll
  for (int rr = 0; rr < 4; ++rr) {
    m[rr] = -INFINITY;
    l[rr] = 0.f;
    diag[rr] = -INFINITY;
    const int64_t i = i0 + 4 * ty + rr;
    lse_i[rr] = (mode == 1 && i < B) ? __ldg(lse + i) : 0.f;
#pragma unroll
    for (int e = 0; e < 4; ++e) g[rr][e] = 0.f;
  }

  for (int t = 0; t < ntiles; ++t) {
    if (t + 1 < ntiles) issue(t + 1);     // its buffer was released by the barrier that closed tile t - 1
    cp_async_commit();
    cp_async_wait<1>();
    __syncthreads();                      // tile t (and, on the first pass, the anchors) visible to every thread
    const int st = t & 1;
    const int64_t j0 = jbeg + (int64_t)t * NT_J;
    float s[4][4];
#pragma unroll
    for (int rr = 0; rr < 4; ++rr)
#pragma unroll
      for (int q = 0; q < 4; ++q) s[rr][q] = 0.f;
#pragma unroll 4
    for (int k4 = 0; k4 < 16; ++k4) {
      float4 a[4], b[4];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) a[rr] = *reinterpret_cast<const float4*>(&sm.As[4 * ty + rr][4 * k4]);
#pragma unroll
      for (int q = 0; q < 4; ++q) b[q] = *reinterpret_cast<const float4*>(&sm.Bs[st][tx + 16 * q][4 * k4]);
#pragma unroll
      for (int rr = 0; rr < 4; ++rr)
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          s[rr][q] = fmaf(a[rr].x, b[q].x, s[rr][q]);
          s[rr][q] = fmaf(a[rr].y, b[q].y, s[rr][q]);
          s[rr][q] = fmaf(a[rr].z, b[q].z, s[rr][q]);
          s[rr][q] = fmaf(a[rr].w, b[q].w, s[rr][q]);
        }
    }
    if (FWD) {
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const int64_t i = i0 + 4 * ty + rr;
        float tmax = -INFINITY;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int64_t j = j0 + tx + 16 * q;
          s[rr][q] = (j < jend) ? s[rr][q] * inv_temp : -INFINITY;
          if (j == i) diag[rr] = s[rr][q];
          tmax = fmaxf(tmax, s[rr][q]);
        }
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) tmax = fmaxf(tmax, __shfl_xor_sync(hmask, tmax, o, 16));
        const float mn = fmaxf(m[rr], tmax);      // finite: every tile holds at least one valid column
        float pt = 0.f;
#pragma unroll
        for (int q = 0; q < 4; ++q) pt += expf(s[rr][q] - mn);   // exp(-inf) = 0 for masked columns
#pragma unroll
        for (int o = 8; o > 0; o >>= 1) pt += __shfl_xor_sync(hmask, pt, o, 16);
        l[rr] = l[rr] * expf(m[rr] - mn) + pt;
        m[rr] = mn;
      }
    } else {
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int c = tx + 16 * q;
        const int64_t j = j0 + c;
        float w[4];
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          const int64_t i = i0 + 4 * ty + rr;
          const float ls = (mode == 1) ? lse_i[rr] : sm.lse_s[st][c];
          w[rr] = (j < jend && i < B) ? expf(s[rr][q] * inv_temp - ls) - (j == i ? 1.f : 0.f) : 0.f;
        }
        *reinterpret_cast<float4*>(&sm.Ps[c][4 * ty]) = make_float4(w[0], w[1], w[2], w[3]);
      }
      __syncthreads();
      // g(4 ty + rr, 4 tx + e) += sum_j w(rr, j) B(j, 4 tx + e)
#pragma unroll 8
      for (int j = 0; j < NT_J; ++j) {
        const float4 w = *reinterpret_cast<const float4*>(&sm.Ps[j][4 * ty]);
        const float4 b = *reinterpret_cast<const float4*>(&sm.Bs[st][j][4 * tx]);
        const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          g[rr][0] = fmaf(wv[rr], b.x, g[rr][0]);
          g[rr][1] = fmaf(wv[rr], b.y, g[rr][1]);
          g[rr][2] = fmaf(wv[rr], b.z, g[rr][2]);
          g[rr][3] = fmaf(wv[rr], b.w, g[rr][3]);
        }
      }
    }
    __syncthreads();   // tile t and Ps fully consumed
  }
  cp_async_wait<0>();

  if (FWD) {
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int64_t i = i0 + 4 * ty + rr;
      float dg = diag[rr];
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) dg = fmaxf(dg, __shfl_xor_sync(hmask, dg, o, 16));
      if (tx == 0 && i < B) {
        float* o3 = part + (i * JS + split) * 3;
        o3[0] = m[rr];
        o3[1] = l[rr];
        o3[2] = dg;
      }
    }
  } else {
    float* gp = gpart + ((int64_t)(mode - 1) * JS + split) * B * 64;
#pragma unroll
    for (int rr = 0; rr < 4; ++rr) {
      const int64_t i = i0 + 4 * ty + rr;
      if (i < B) *reinterpret_cast<float4*>(gp + i * 64 + 4 * tx) = make_float4(g[rr][0], g[rr][1], g[rr][2], g[rr][3]);
    }
  }
}

// merges the per-split (m, l, diag) of every anchor, writes lse and the row loss, reduces the mean (one CTA, fixed order)
__global__ void __launch_bounds__(1024) nce_fwd_combine_kernel(const float* __restrict__ part, int JS, int64_t B, float scale,
                                                               float* __restrict__ out_lse, float* __restrict__ row_loss,
                                                               float* __restrict__ out) {
  __shared__ float red[32];
  float acc = 0.f;
  for (int64_t i = threadIdx.x; i < B; i += 1024) {
    float M = -INFINITY, dg = -INFINITY;
    for (int k = 0; k < JS; ++k) {
      M = fmaxf(M, part[(i * JS + k) * 3]);
      dg = fmaxf(dg, part[(i * JS + k) * 3 + 2]);
    }
    float L = 0.f;
    for (int k = 0; k < JS; ++k) {
      const float mk = part[(i * JS + k) * 3], lk = part[(i * JS + k) * 3 + 1];
      if (lk > 0.f) L += lk * expf(mk - M);
    }
    const float lse = M + logf(L);
    out_lse[i] = lse;
    row_loss[i] = lse - dg;
    acc += lse - dg;
  }
  acc = dmm_warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    float t = red[threadIdx.x];
    t = dmm_warp_sum(t);
    if (threadIdx.x == 0) *out = t * scale;
  }
}

// adds the per-split partial gradients (fixed order) and applies the normalisation backward; one half warp per row,
// rows [0, B): d/d v1 (n1, inv1), rows [B, 2B): d/d v2 (n2, inv2)
__global__ void __launch_bounds__(256) nce_bwd_combine_kernel(const float* __restrict__ gpart, int JS, int64_t B,
                                                              const float* __restrict__ n1, const float* __restrict__ n2,
                                                              const float* __restrict__ inv1, const float* __restrict__ inv2,
                                                              float coef, float* __restrict__ g1, float* __restrict__ g2) {
  const int64_t x = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  const int l16 = threadIdx.x & 15;
  const uint32_t hmask = 0xFFFFu << (threadIdx.x & 16);
  if (x >= 2 * B) return;
  const int side = x >= B ? 1 : 0;
  const int64_t i = x - (int64_t)side * B;
  float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
  for (int k = 0; k < JS; ++k) {
    const float4 p = __ldg(reinterpret_cast<const float4*>(gpart + (((int64_t)side * JS + k) * B + i) * 64) + l16);
    g.x += p.x; g.y += p.y; g.z += p.z; g.w += p.w;
  }
  const float4 n = __ldg(reinterpret_cast<const float4*>((side ? n2 : n1) + i * 64) + l16);
  float dot = n.x * g.x + n.y * g.y + n.z * g.z + n.w * g.w;
#pragma unroll
  for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(hmask, dot, o, 16);
  const float sc = (side ? inv2 : inv1)[i] * coef;
  *reinterpret_cast<float4*>((side ? g2 : g1) + i * 64 + 4 * l16) =
      make_float4(sc * (g.x - n.x * dot), sc * (g.y - n.y * dot), sc * (g.z - n.z * dot), sc * (g.w - n.w * dot));
}

inline int nce_splits(int64_t B) {
  int64_t js = (B + 255) / 256;
  return (int)(js < 1 ? 1 : (js > NCE_MAX_SPLIT ? NCE_MAX_SPLIT : js));
}
inline int64_t nce_split_rows(int64_t B, int JS) { return ((B + JS - 1) / JS + NT_J - 1) / NT_J * NT_J; }

template <bool FWD>
int launch_nce_tiles(const dmm_ctx* ctx, int64_t B, const float* n_base, int n_problems, const NceBatch& batch, const float* lse,
                     float* part, float* gpart, cudaStream_t st) {
  static DmmPerDeviceOnce attr_once;
  if (attr_once.need(ctx)) {
    DMM_CUDA(cudaFuncSetAttribute(nce_tiles_kernel<FWD>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sizeof(NceSmem)));
    attr_once.mark(ctx);
  }
  const int JS = nce_splits(B);
  dim3 grid((unsigned)dmm_ceil_div(B, NT_I), (unsigned)JS, (unsigned)(FWD ? n_problems : 2 * n_problems));
  nce_tiles_kernel<FWD><<<grid, NT_THREADS, sizeof(NceSmem), st>>>(n_base, B, nce_split_rows(B, JS), batch, lse, part, gpart);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

__global__ void __launch_bounds__(256) scatter_add_rows_kernel(const float* __restrict__ src, int64_t ld_s,
                                                               const int64_t* __restrict__ idx, int64_t B, int D,
                                                               float* __restrict__ dst, int64_t ld_d) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const int64_t r = idx[b];
  for (int c = lane; c < D; c += 32) atomicAdd(dst + r * ld_d + c, __ldg(src + b * ld_s + c));
}

// the widths nce_rows_kernel is instantiated for (D / 32 picks the instance, so any other D must be refused up front:
// D = 48 would otherwise run the D = 32 kernel on rows of stride 48)
inline bool nce_supported_d(int64_t D) { return D == 32 || D == 64 || D == 128 || D == 256; }

template <int MODE>
int launch_nce(int64_t B, int64_t D, const float* na, const float* nb, float inv_temp, const float* lse_in,
               const float* inv_norm, float coef, float* out_lse, float* out_row_loss, float* out_grad,
               cudaStream_t st) {
  const unsigned grid = (unsigned)dmm_ceil_div(B * 32, 256);
  switch (D / 32) {
    case 1: nce_rows_kernel<MODE, 1><<<grid, 256, 0, st>>>(na, nb, B, inv_temp, lse_in, inv_norm, coef, out_lse, out_row_loss, out_grad); break;
    case 2: nce_rows_kernel<MODE, 2><<<grid, 256, 0, st>>>(na, nb, B, inv_temp, lse_in, inv_norm, coef, out_lse, out_row_loss, out_grad); break;
    case 4: nce_rows_kernel<MODE, 4><<<grid, 256, 0, st>>>(na, nb, B, inv_temp, lse_in, inv_norm, coef, out_lse, out_row_loss, out_grad); break;
    case 8: nce_rows_kernel<MODE, 8><<<grid, 256, 0, st>>>(na, nb, B, inv_temp, lse_in, inv_norm, coef, out_lse, out_row_loss, out_grad); break;
    default:
      dmm_set_error("InfoNCE: D must be 32, 64, 128 or 256 (got %lld)", (long long)D);
      return DMM_ERR_UNSUPPORTED;
  }
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

}  // namespace

extern "C" int dmm_bpr_fwd_bwd(dmm_ctx* ctx, const float* u_emb, int64_t ld_u, const float* i_emb, int64_t ld_i,
                               const int64_t* users, const int64_t* pos, const int64_t* neg, int64_t B, int64_t D,
                               float grad_scale, float* row_loss, float* loss, float* g_u, float* g_p, float* g_n,
                               void* stream) {
  DMM_CHECK_ARG(ctx && u_emb && i_emb && users && pos && neg && row_loss && loss, "dmm_bpr_fwd_bwd: null argument");
  DMM_CHECK_ARG(B > 0 && D > 0 && D <= MAX_D, "dmm_bpr_fwd_bwd: bad shape");
  DMM_CHECK_ARG((g_u && g_p && g_n) || (!g_u && !g_p && !g_n), "dmm_bpr_fwd_bwd: gradient outputs are all-or-none");
  cudaStream_t st = (cudaStream_t)stream;
  bpr_kernel<<<(unsigned)dmm_ceil_div(B * 32, 256), 256, 0, st>>>(u_emb, ld_u, i_emb, ld_i, users, pos, neg, B, (int)D,
                                                                 grad_scale / (float)B, row_loss, g_u, g_p, g_n);
  DMM_LAUNCH_CHECK();
  mean_reduce_kernel<<<1, 1024, 0, st>>>(row_loss, B, 1.f / (float)B, loss);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_infonce_fwd(dmm_ctx* ctx, const float* v1, int64_t ld1, const float* v2, int64_t ld2,
                               const int64_t* idx, int64_t B, int64_t D, float temperature, float* workspace,
                               float* row_loss, float* loss, float* lse, float* inv1, float* inv2, void* stream) {
  DMM_CHECK_ARG(ctx && v1 && v2 && idx && workspace && row_loss && loss && lse && inv1 && inv2,
                "dmm_infonce_fwd: null argument");
  DMM_CHECK_ARG(B > 0 && temperature > 0.f, "dmm_infonce_fwd: bad B or temperature");
  DMM_CHECK_ARG(nce_supported_d(D), "InfoNCE: D must be 32, 64, 128 or 256 (got %lld)", (long long)D);
  DMM_CHECK_ARG(ld1 >= D && ld2 >= D, "dmm_infonce_fwd: leading dimension < D");
  cudaStream_t st = (cudaStream_t)stream;
  float* n1 = workspace;
  float* n2 = workspace + B * D;
  nce_gather_norm_kernel<<<(unsigned)dmm_ceil_div(B * 32, 256), 256, 0, st>>>(v1, ld1, v2, ld2, idx, B, (int)D, n1, n2, inv1, inv2);
  DMM_LAUNCH_CHECK();
  if (D == 64) {
    float* part = workspace + 2 * B * D;     // [B][JS][3]
    NceBatch one;
    one.inv_temp[0] = 1.f / temperature;
    int rc = launch_nce_tiles<true>(ctx, B, n1, 1, one, nullptr, part, nullptr, st);
    if (rc) return rc;
    nce_fwd_combine_kernel<<<1, 1024, 0, st>>>(part, nce_splits(B), B, 1.f / (float)B, lse, row_loss, loss);
    DMM_LAUNCH_CHECK();
    return DMM_OK;
  }
  int rc = launch_nce<0>(B, D, n1, n2, 1.f / temperature, nullptr, nullptr, 0.f, lse, row_loss, nullptr, st);
  if (rc) return rc;
  mean_reduce_kernel<<<1, 1024, 0, st>>>(row_loss, B, 1.f / (float)B, loss);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int64_t dmm_infonce_workspace_floats(int64_t B, int64_t D, int backward) {
  int64_t n = 2 * B * D;                       // normalised gathers of both views
  if (D == 64) n += backward ? 2 * (int64_t)nce_splits(B) * B * D : 3 * (int64_t)nce_splits(B) * B;
  return n;
}

extern "C" int dmm_infonce_bwd(dmm_ctx* ctx, const float* v1, int64_t ld1, const float* v2, int64_t ld2,
                               const int64_t* idx, int64_t B, int64_t D, float temperature, const float* lse,
                               const float* inv1, const float* inv2, float grad_scale, float* workspace, float* g1,
                               float* g2, void* stream) {
  DMM_CHECK_ARG(ctx && v1 && v2 && idx && lse && inv1 && inv2 && workspace && g1 && g2, "dmm_infonce_bwd: null argument");
  DMM_CHECK_ARG(B > 0 && temperature > 0.f, "dmm_infonce_bwd: bad B or temperature");
  DMM_CHECK_ARG(nce_supported_d(D), "InfoNCE: D must be 32, 64, 128 or 256 (got %lld)", (long long)D);
  DMM_CHECK_ARG(ld1 >= D && ld2 >= D, "dmm_infonce_bwd: leading dimension < D");
  cudaStream_t st = (cudaStream_t)stream;
  float* n1 = workspace;
  float* n2 = workspace + B * D;
  // recompute the normalised gathers (cheaper than keeping 2*B*D floats alive across the whole step)
  nce_gather_norm_kernel<<<(unsigned)dmm_ceil_div(B * 32, 256), 256, 0, st>>>(v1, ld1, v2, ld2, idx, B, (int)D, n1, n2,
                                                                              nullptr, nullptr);
  DMM_LAUNCH_CHECK();
  const float coef = grad_scale / ((float)B * temperature);
  if (D == 64) {
    float* gpart = workspace + 2 * B * D;    // [2 sides][JS][B][64]
    NceBatch one;
    one.inv_temp[0] = 1.f / temperature;
    int rc = launch_nce_tiles<false>(ctx, B, n1, 1, one, lse, nullptr, gpart, st);
    if (rc) return rc;
    nce_bwd_combine_kernel<<<(unsigned)dmm_ceil_div(2 * B * 16, 256), 256, 0, st>>>(gpart, nce_splits(B), B, n1, n2, inv1, inv2,
                                                                                  coef, g1, g2);
    DMM_LAUNCH_CHECK();
    return DMM_OK;
  }
  int rc = launch_nce<1>(B, D, n1, n2, 1.f / temperature, lse, inv1, coef, nullptr, nullptr, g1, st);
  if (rc) return rc;
  return launch_nce<2>(B, D, n2, n1, 1.f / temperature, lse, inv2, coef, nullptr, nullptr, g2, st);
}

extern "C" int dmm_scatter_add_rows(dmm_ctx* ctx, const float* src, int64_t ld_s, const int64_t* idx, int64_t B,
                                    int64_t D, float* dst, int64_t ld_d, void* stream) {
  DMM_CHECK_ARG(ctx && src && idx && dst, "dmm_scatter_add_rows: null argument");
  DMM_CHECK_ARG(B >= 0 && D > 0 && ld_s >= D && ld_d >= D, "dmm_scatter_add_rows: bad shape");
  if (B == 0) return DMM_OK;
  scatter_add_rows_kernel<<<(unsigned)dmm_ceil_div(B * 32, 256), 256, 0, (cudaStream_t)stream>>>(src, ld_s, idx, B, (int)D, dst, ld_d);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

// ================================================================================================ fused BPR + InfoNCE
// One call for EVERY loss of a joint-training step (Main.py:309,333,345-367: BPR + 2 cross-layer + 2M or 2 C(M,2)
// modality InfoNCE terms): three launches forward and three backward in total instead of ~3 + 3 per term, plus one
// scatter of all row gradients.  Views are whole node tables [N, 64]; a problem addresses rows `row_off + idx[b]`.
namespace {

struct GradTabs {                         // destination tables of the backward scatter, by value in the kernel parameters
  float* tab[2 * NCE_MAX_PROBLEMS + 1];
  int64_t ld[2 * NCE_MAX_PROBLEMS + 1];
};

struct FusedSpec {
  int n_problems;
  const float* v1[NCE_MAX_PROBLEMS];
  const float* v2[NCE_MAX_PROBLEMS];
  int64_t ld1[NCE_MAX_PROBLEMS], ld2[NCE_MAX_PROBLEMS];
  int64_t off[NCE_MAX_PROBLEMS];          // row offset of the problem's rows inside both views (0 users, U items)
  const int64_t* idx[NCE_MAX_PROBLEMS];
  float weight[NCE_MAX_PROBLEMS];         // rate of the term in the contrastive total
  float temp[NCE_MAX_PROBLEMS];
  // BPR on the final embeddings: rows users[b], U + pos[b], U + neg[b] of `emb`
  const float* emb;
  int64_t ld_emb, item_off;
  const int64_t *users, *pos, *neg;
};

// blockIdx.y < n_problems: gather + L2-normalise both views of problem y (one warp per row); blockIdx.y == n_problems:
// the BPR rows (loss, and with g_bpr the row gradients scaled by *g_bpr / B)
__global__ void __launch_bounds__(256) fused_gather_kernel(const FusedSpec sp, int64_t B, float* __restrict__ n_base,
                                                           float* __restrict__ inv_base, float* __restrict__ bpr_row_loss,
                                                           const float* __restrict__ g_bpr, float* __restrict__ g_bpr_rows) {
  const int64_t b = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (b >= B) return;
  const int p = blockIdx.y;
  if (p < sp.n_problems) {
    const int64_t r = sp.off[p] + sp.idx[p][b];
    const float* a = sp.v1[p] + r * sp.ld1[p];
    const float* c = sp.v2[p] + r * sp.ld2[p];
    const float x0 = __ldg(a + lane), x1 = __ldg(a + 32 + lane), y0 = __ldg(c + lane), y1 = __ldg(c + 32 + lane);
    const float s1 = dmm_warp_sum(fmaf(x0, x0, x1 * x1)), s2 = dmm_warp_sum(fmaf(y0, y0, y1 * y1));
    const float i1 = 1.f / fmaxf(sqrtf(s1), 1e-12f), i2 = 1.f / fmaxf(sqrtf(s2), 1e-12f);
    float* n1 = n_base + (int64_t)p * 2 * B * 64 + b * 64;
    float* n2 = n1 + B * 64;
    n1[lane] = x0 * i1;
    n1[32 + lane] = x1 * i1;
    n2[lane] = y0 * i2;
    n2[32 + lane] = y1 * i2;
    if (lane == 0 && inv_base) {
      inv_base[(int64_t)p * 2 * B + b] = i1;
      inv_base[(int64_t)p * 2 * B + B + b] = i2;
    }
  } else {
    const float* u = sp.emb + sp.users[b] * sp.ld_emb;
    const float* q = sp.emb + (sp.item_off + sp.pos[b]) * sp.ld_emb;
    const float* n = sp.emb + (sp.item_off + sp.neg[b]) * sp.ld_emb;
    const float u0 = __ldg(u + lane), u1 = __ldg(u + 32 + lane), p0 = __ldg(q + lane), p1 = __ldg(q + 32 + lane),
                m0 = __ldg(n + lane), m1 = __ldg(n + 32 + lane);
    const float x = dmm_warp_sum(fmaf(u0, p0 - m0, u1 * (p1 - m1)));       // u.p - u.n
    const float s = 1.f / (1.f + expf(-x));
    if (bpr_row_loss && lane == 0) bpr_row_loss[b] = -logf(10e-6f + s);
    if (g_bpr_rows) {
      const float d = -(s * (1.f - s)) / (10e-6f + s) * (*g_bpr) / (float)B;
      float* gu = g_bpr_rows + b * 64;
      float* gp = g_bpr_rows + (B + b) * 64;
      float* gn = g_bpr_rows + (2 * B + b) * 64;
      gu[lane] = d * (p0 - m0);
      gu[32 + lane] = d * (p1 - m1);
      gp[lane] = d * u0;
      gp[32 + lane] = d * u1;
      gn[lane] = -d * u0;
      gn[32 + lane] = -d * u1;
    }
  }
}

// one CTA: per problem the split merge + mean (fixed order), then the BPR mean and the weighted contrastive total
// losses[0 .. P) = InfoNCE means, losses[P] = BPR, losses[P + 1] = sum_p weight_p * losses[p]
__global__ void __launch_bounds__(1024) fused_fwd_combine_kernel(const FusedSpec sp, const float* __restrict__ part_base, int JS,
                                                                 int64_t B, float* __restrict__ lse_base,
                                                                 const float* __restrict__ bpr_row_loss,
                                                                 float* __restrict__ losses) {
  __shared__ float red[32];
  __shared__ float total;
  if (threadIdx.x == 0) total = 0.f;
  for (int p = 0; p <= sp.n_problems; ++p) {
    float acc = 0.f;
    if (p < sp.n_problems) {
      const float* part = part_base + (int64_t)p * B * JS * 3;
      for (int64_t i = threadIdx.x; i < B; i += 1024) {
        float M = -INFINITY, dg = -INFINITY;
        for (int k = 0; k < JS; ++k) {
          M = fmaxf(M, part[(i * JS + k) * 3]);
          dg = fmaxf(dg, part[(i * JS + k) * 3 + 2]);
        }
        float L = 0.f;
        for (int k = 0; k < JS; ++k) {
          const float mk = part[(i * JS + k) * 3], lk = part[(i * JS + k) * 3 + 1];
          if (lk > 0.f) L += lk * expf(mk - M);
        }
        const float lse = M + logf(L);
        lse_base[(int64_t)p * B + i] = lse;
        acc += lse - dg;
      }
    } else {
      for (int64_t i = threadIdx.x; i < B; i += 1024) acc += bpr_row_loss[i];
    }
    acc = dmm_warp_sum(acc);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x < 32) {
      float t = dmm_warp_sum(red[threadIdx.x]);
      if (threadIdx.x == 0) {
        const float mean = t / (float)B;
        losses[p] = mean;
        if (p < sp.n_problems) total += sp.weight[p] * mean;
      }
    }
  }
  __syncthreads();
  if (threadIdx.x == 0) losses[sp.n_problems + 1] = total;
}

// partial gradients -> row gradients (normalisation backward, coef = weight_p g_cl / (B T_p)) scattered straight into the
// gradient tables of the views (atomicAdd: indices repeat inside a batch); z = 2 p + side.  The last z slot scatters the
// three BPR row-gradient blocks.  One half warp per row.
__global__ void __launch_bounds__(256) fused_bwd_scatter_kernel(const FusedSpec sp, const float* __restrict__ gpart_base, int JS,
                                                                int64_t B, const float* __restrict__ n_base,
                                                                const float* __restrict__ inv_base,
                                                                const float* __restrict__ g_cl,
                                                                const float* __restrict__ g_bpr_rows, const GradTabs gt) {
  const int64_t x = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 4;
  const int l16 = threadIdx.x & 15;
  const uint32_t hmask = 0xFFFFu << (threadIdx.x & 16);
  const int z = blockIdx.y;
  if (z < 2 * sp.n_problems) {
    if (x >= B) return;
    const int p = z >> 1, side = z & 1;
    float* dst = gt.tab[z];
    if (!dst) return;
    const float* gpart = gpart_base + (int64_t)p * 2 * JS * B * 64;
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int k = 0; k < JS; ++k) {
      const float4 q = __ldg(reinterpret_cast<const float4*>(gpart + (((int64_t)side * JS + k) * B + x) * 64) + l16);
      g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
    }
    const float4 n = __ldg(reinterpret_cast<const float4*>(n_base + (int64_t)p * 2 * B * 64 + (int64_t)side * B * 64 + x * 64) + l16);
    float dot = n.x * g.x + n.y * g.y + n.z * g.z + n.w * g.w;
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) dot += __shfl_xor_sync(hmask, dot, o, 16);
    const float sc = inv_base[(int64_t)p * 2 * B + (int64_t)side * B + x] * sp.weight[p] * (*g_cl) / ((float)B * sp.temp[p]);
    float* row = dst + (sp.off[p] + sp.idx[p][x]) * gt.ld[z] + 4 * l16;
    atomicAdd(row + 0, sc * (g.x - n.x * dot));
    atomicAdd(row + 1, sc * (g.y - n.y * dot));
    atomicAdd(row + 2, sc * (g.z - n.z * dot));
    atomicAdd(row + 3, sc * (g.w - n.w * dot));
  } else {
    if (x >= 3 * B) return;
    float* dst = gt.tab[z];
    if (!dst) return;
    const int kind = (int)(x / B);
    const int64_t b = x - (int64_t)kind * B;
    const int64_t r = kind == 0 ? sp.users[b] : sp.item_off + (kind == 1 ? sp.pos[b] : sp.neg[b]);
    const float4 q = __ldg(reinterpret_cast<const float4*>(g_bpr_rows + x * 64) + l16);
    float* row = dst + r * gt.ld[z] + 4 * l16;
    atomicAdd(row + 0, q.x);
    atomicAdd(row + 1, q.y);
    atomicAdd(row + 2, q.z);
    atomicAdd(row + 3, q.w);
  }
}

int fill_spec(FusedSpec& sp, const dmm_nce_problem* problems, int n_problems, const dmm_bpr_problem* bpr) {
  sp.n_problems = n_problems;
  for (int p = 0; p < n_problems; ++p) {
    const dmm_nce_problem& q = problems[p];
    DMM_CHECK_ARG(q.v1 && q.v2 && q.idx && q.ld1 >= 64 && q.ld2 >= 64 && q.temperature > 0.f && q.row_offset >= 0,
                  "dmm_bpr_infonce: bad problem %d", p);
    sp.v1[p] = q.v1; sp.v2[p] = q.v2; sp.ld1[p] = q.ld1; sp.ld2[p] = q.ld2; sp.off[p] = q.row_offset; sp.idx[p] = q.idx;
    sp.weight[p] = q.weight; sp.temp[p] = q.temperature;
  }
  DMM_CHECK_ARG(bpr && bpr->emb && bpr->users && bpr->pos && bpr->neg && bpr->ld_emb >= 64, "dmm_bpr_infonce: bad BPR problem");
  sp.emb = bpr->emb; sp.ld_emb = bpr->ld_emb; sp.item_off = bpr->item_offset;
  sp.users = bpr->users; sp.pos = bpr->pos; sp.neg = bpr->neg;
  return DMM_OK;
}

}  // namespace

extern "C" int64_t dmm_bpr_infonce_workspace_floats(int64_t B, int n_problems, int backward) {
  const int64_t P = n_problems;
  int64_t n = P * 2 * B * 64;                                   // normalised gathers
  if (backward) n += P * 2 * (int64_t)nce_splits(B) * B * 64 + 3 * B * 64;    // gradient partials + BPR row gradients
  else n += P * 3 * (int64_t)nce_splits(B) * B + B;            // forward partials + BPR row losses
  return n;
}

extern "C" int dmm_bpr_infonce_fwd(dmm_ctx* ctx, const dmm_nce_problem* problems, int n_problems, const dmm_bpr_problem* bpr,
                                   int64_t B, float* workspace, float* losses, float* lse, float* inv, void* stream) {
  DMM_CHECK_ARG(ctx && problems && workspace && losses && lse && inv, "dmm_bpr_infonce_fwd: null argument");
  DMM_CHECK_ARG(n_problems >= 1 && n_problems <= NCE_MAX_PROBLEMS && B > 0, "dmm_bpr_infonce_fwd: 1..%d problems", NCE_MAX_PROBLEMS);
  FusedSpec sp;
  int rc = fill_spec(sp, problems, n_problems, bpr);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  float* n_base = workspace;
  float* part = workspace + (int64_t)n_problems * 2 * B * 64;
  float* bpr_rows = part + (int64_t)n_problems * 3 * nce_splits(B) * B;
  fused_gather_kernel<<<dim3((unsigned)dmm_ceil_div(B * 32, 256), (unsigned)(n_problems + 1)), 256, 0, st>>>(
      sp, B, n_base, inv, bpr_rows, nullptr, nullptr);
  DMM_LAUNCH_CHECK();
  NceBatch batch;
  for (int p = 0; p < n_problems; ++p) batch.inv_temp[p] = 1.f / problems[p].temperature;
  rc = launch_nce_tiles<true>(ctx, B, n_base, n_problems, batch, nullptr, part, nullptr, st);
  if (rc) return rc;
  fused_fwd_combine_kernel<<<1, 1024, 0, st>>>(sp, part, nce_splits(B), B, lse, bpr_rows, losses);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

extern "C" int dmm_bpr_infonce_bwd(dmm_ctx* ctx, const dmm_nce_problem* problems, int n_problems, const dmm_bpr_problem* bpr,
                                   int64_t B, const float* lse, const float* inv, const float* g_cl, const float* g_bpr,
                                   float* workspace, float* const* grad_tables, const int64_t* grad_ld, void* stream) {
  DMM_CHECK_ARG(ctx && problems && lse && inv && g_cl && g_bpr && workspace && grad_tables && grad_ld,
                "dmm_bpr_infonce_bwd: null argument");
  DMM_CHECK_ARG(n_problems >= 1 && n_problems <= NCE_MAX_PROBLEMS && B > 0, "dmm_bpr_infonce_bwd: 1..%d problems", NCE_MAX_PROBLEMS);
  FusedSpec sp;
  int rc = fill_spec(sp, problems, n_problems, bpr);
  if (rc) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  float* n_base = workspace;
  float* gpart = workspace + (int64_t)n_problems * 2 * B * 64;
  float* g_bpr_rows = gpart + (int64_t)n_problems * 2 * nce_splits(B) * B * 64;
  // the normalised gathers are recomputed (cheaper than keeping them alive across the step); the BPR slot writes its
  // row gradients
  fused_gather_kernel<<<dim3((unsigned)dmm_ceil_div(B * 32, 256), (unsigned)(n_problems + 1)), 256, 0, st>>>(
      sp, B, n_base, nullptr, nullptr, g_bpr, g_bpr_rows);
  DMM_LAUNCH_CHECK();
  NceBatch batch;
  for (int p = 0; p < n_problems; ++p) batch.inv_temp[p] = 1.f / problems[p].temperature;
  rc = launch_nce_tiles<false>(ctx, B, n_base, n_problems, batch, lse, nullptr, gpart, st);
  if (rc) return rc;
  GradTabs gt;
  for (int i = 0; i < 2 * NCE_MAX_PROBLEMS + 1; ++i) {
    gt.tab[i] = nullptr;
    gt.ld[i] = 0;
  }
  for (int i = 0; i < 2 * n_problems; ++i) {
    gt.tab[i] = grad_tables[i];
    gt.ld[i] = grad_ld[i];
    DMM_CHECK_ARG(!gt.tab[i] || gt.ld[i] >= 64, "dmm_bpr_infonce_bwd: gradient table %d needs ld >= 64", i);
  }
  // the BPR slot of the kernel is z = 2 P; the caller passes it as entry 2 P of its arrays
  float* bpr_tab = grad_tables[2 * n_problems];
  const int64_t bpr_ld = grad_ld[2 * n_problems];
  fused_bwd_scatter_kernel<<<dim3((unsigned)dmm_ceil_div(3 * B * 16, 256), (unsigned)(2 * n_problems + 1)), 256, 0, st>>>(
      sp, gpart, nce_splits(B), B, n_base, inv, g_cl, g_bpr_rows, [&]() { gt.tab[2 * n_problems] = bpr_tab; gt.ld[2 * n_problems] = bpr_ld; return gt; }());
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
