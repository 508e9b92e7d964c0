// Context, error reporting and version of the C ABI.
#include "common.cuh"

#include <string.h>

namespace {
thread_local char g_err[512] = "";
}

void dmm_set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

extern "C" int dmm_version(void) { return 102; }  // 0.1.2

extern "C" const char* dmm_last_error(void) { return g_err; }

extern "C" int dmm_init(int device, dmm_ctx** out) {
  DMM_CHECK_ARG(out, "dmm_init: null out pointer");
  *out = nullptr;
  int n = 0;
  DMM_CUDA(cudaGetDeviceCount(&n));
  DMM_CHECK_ARG(device >= 0 && device < n, "dmm_init: device %d out of range (%d visible)", device, n);
  // nothing here changes the calling thread's current device (cudaGetDeviceProperties and
  // cudaGetDriverEntryPoint do not need it)
  cudaDeviceProp prop;
  DMM_CUDA(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) {
    dmm_set_error("dmm_init: device %d is sm_%d%d; this library is built for sm_100a (B200) only", device, prop.major,
                  prop.minor);
    return DMM_ERR_UNSUPPORTED;
  }
  dmm_ctx* c = new dmm_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  c->max_smem_optin = (int)prop.sharedMemPerBlockOptin;
  c->encode_tiled = nullptr;
  cudaDriverEntryPointQueryResult q;
  void* fn = nullptr;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q);
  if (e != cudaSuccess || q != cudaDriverEntryPointSuccess || !fn) {
    delete c;
    dmm_set_error("dmm_init: cuTensorMapEncodeTiled not available from the driver (%s)", cudaGetErrorString(e));
    return DMM_ERR_CUDA;
  }
  c->encode_tiled = fn;
  *out = c;
  return DMM_OK;
}

extern "C" void dmm_destroy(dmm_ctx* ctx) { delete ctx; }

extern "C" int dmm_num_sms(const dmm_ctx* ctx) { return ctx ? ctx->num_sms : 0; }

// ---- host-side helper -------------------------------------------------------------------------
// The reference's negative sampler (DataHandler.py:159-169) is a Python loop of rejection sampling on
// the global numpy generator.  Its draws are a pure stream, so the caller pre-draws `n_draws` values
// with the same generator and this routine replays the loop over them: interaction i keeps consuming
// draws until one is not an item of its user (binary search in the user's sorted CSR row).  Returns
// DMM_ERR_WORKSPACE when the pre-drawn stream runs out (the caller draws more and calls again);
// *consumed is the number of draws the reference loop would have made.
extern "C" int dmm_host_neg_sampling(const int64_t* indptr, const int32_t* indices, const int32_t* rows, int64_t n,
                                     const int64_t* draws, int64_t n_draws, int32_t* negs, int64_t* consumed) {
  DMM_CHECK_ARG(indptr && indices && rows && draws && negs && consumed, "dmm_host_neg_sampling: null argument");
  int64_t j = 0;
  for (int64_t i = 0; i < n; ++i) {
    const int64_t b = indptr[rows[i]], e = indptr[rows[i] + 1];
    for (;;) {
      if (j >= n_draws) {
        *consumed = j;
        dmm_set_error("dmm_host_neg_sampling: %lld pre-drawn values exhausted at interaction %lld", (long long)n_draws,
                      (long long)i);
        return DMM_ERR_WORKSPACE;
      }
      const int32_t v = (int32_t)draws[j++];
      int64_t lo = b, hi = e;
      while (lo < hi) {
        const int64_t mid = (lo + hi) >> 1;
        if (indices[mid] < v) lo = mid + 1; else hi = mid;
      }
      if (!(lo < e && indices[lo] == v)) {
        negs[i] = v;
        break;
      }
    }
  }
  *consumed = j;
  return DMM_OK;
}
