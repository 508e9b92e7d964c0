// fp32 CUDA-core contraction with the same epilogue contract as gemm_tcgen05.cu.
// Verification mode only (checks the tensor-pipe kernel at sizes the CPU oracle cannot reach);
// the Denoise path runs on dmm_gemm_bf16_tn.
#include "common.cuh"

namespace {
constexpr int TM = 64, TN = 64, TK = 16;

__global__ void __launch_bounds__(256) gemm_f32_tn_kernel(const float* __restrict__ A, int64_t lda,
                                                           const float* __restrict__ B, int64_t ldb, int M, int N,
                                                           int K, dmm_gemm_epilogue ep) {
  __shared__ float sa[TK][TM + 1];
  __shared__ float sb[TK][TN + 1];
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  const int m0 = blockIdx.y * TM, n0 = blockIdx.x * TN;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += TK) {
    for (int i = threadIdx.x; i < TM * TK; i += 256) {
      const int r = i / TK, c = i % TK;
      const int gm = m0 + r, gn = n0 + r, gk = k0 + c;
      sa[c][r] = (gm < M && gk < K) ? A[(int64_t)gm * lda + gk] : 0.f;
      sb[c][r] = (gn < N && gk < K) ? B[(int64_t)gn * ldb + gk] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < TK; ++k) {
      float a[4], b[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = sa[k][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) b[j] = sb[k][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      float v = acc[i][j] + (ep.bias ? ep.bias[n] : 0.f);
      const bool has_res = ep.residual != nullptr || ep.res_hi != nullptr;
      float r = 0.f;
      if (ep.residual) {
        r = ep.residual[(int64_t)m * ep.ld_res + n];
      } else if (ep.res_hi) {
        r = dmm_bf16_to_f32(ep.res_hi[(int64_t)m * ep.ld_res16 + n]);
        if (ep.res_lo) r += dmm_bf16_to_f32(ep.res_lo[(int64_t)m * ep.ld_res16 + n]);
      }
      const bool pre = has_res && ep.res_pre_act != 0;
      if (pre) v += ep.beta * r;
      if (ep.act == 1) v = tanhf(v);
      if (has_res && !pre) {
        v = ep.alpha * v + ep.beta * r;
      } else {
        v *= ep.alpha;
      }
      if (ep.out_f32) ep.out_f32[(int64_t)m * ep.ld_out + n] = v;
      if (ep.out_hi) {
        if (ep.post_bias) v += ep.post_bias[n];
        if (ep.post_act == 1) v = tanhf(v);
        uint16_t h, l;
        dmm_split_bf16(v, h, l);
        ep.out_hi[(int64_t)m * ep.ld_out16 + n] = h;
        if (ep.out_lo) ep.out_lo[(int64_t)m * ep.ld_out16 + n] = l;
      }
    }
  }
}
}  // namespace

extern "C" int dmm_gemm_f32_tn(dmm_ctx* ctx, const float* a, int64_t lda, const float* b, int64_t ldb, int64_t M,
                               int64_t N, int64_t K, const dmm_gemm_epilogue* ep, void* stream) {
  DMM_CHECK_ARG(ctx && a && b && ep, "dmm_gemm_f32_tn: null argument");
  DMM_CHECK_ARG(!ep->cmax, "dmm_gemm_f32_tn: cmax is not supported");
  DMM_CHECK_ARG(M > 0 && N > 0 && K > 0 && lda >= K && ldb >= K, "dmm_gemm_f32_tn: bad shape");
  DMM_CHECK_ARG(dmm_ceil_div(M, TM) < 65536, "dmm_gemm_f32_tn: M too large for the verification kernel");
  dim3 grid((unsigned)dmm_ceil_div(N, TN), (unsigned)dmm_ceil_div(M, TM));
  gemm_f32_tn_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(a, lda, b, ldb, (int)M, (int)N, (int)K, *ep);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
