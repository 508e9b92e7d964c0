// Device-side build of the normalised bipartite adjacency in CSR.
//
// Replaces Coach.makeTorchAdj (Main.py:113-116) -> DataHandler.makeTorchAdj / normalizeAdj
// (DataHandler.py:53-93): scipy vstack/hstack, binarise, + I, D^-1/2 A D^-1/2, then an H2D copy of an
// uncoalesced COO.  Here the edge list produced by dmm_topk_edges (CSR by user, items ascending)
// never leaves the device:
//   1. expand user ids per edge; stable LSD radix sort of (item, user) pairs by item gives R^T with
//      users ascending inside every item row  (CUB DeviceRadixSort: CCCL library plumbing, the only
//      non-hand-written device code of the library; candidate for a hand-written counting sort);
//   2. item row offsets from the boundaries of the sorted list (no atomics, no scan) and d^-1/2 per node, one kernel;
//   3. one thread per stored entry writes [self loop | neighbours] rows in ascending column order with
//      val = (d_r^-1/2 * 1) * d_c^-1/2 evaluated in fp64 and rounded to fp32 like the reference.
// HBM-bound: ~8E bytes in, 8(2E+N) + 8(N+1) bytes out.
#include "common.cuh"

#include <cub/device/device_radix_sort.cuh>

namespace {

__global__ void __launch_bounds__(256) expand_users_kernel(const int64_t* __restrict__ row_ptr, int64_t n_users,
                                                           int32_t* __restrict__ edge_user,
                                                           const int32_t* __restrict__ items, int64_t n_items,
                                                           int32_t* __restrict__ status) {
  const int64_t u = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (u >= n_users) return;
  const int64_t b = row_ptr[u], e = row_ptr[u + 1];
  for (int64_t j = b + lane; j < e; j += 32) {
    edge_user[j] = (int32_t)u;
    const int32_t it = items[j];
    if ((it < 0 || it >= n_items) && status) atomicOr(status, 2);
  }
}

// One thread per node: item row offsets from the item-sorted edge list -- item_ptr[it] = first position whose item is >= it
// (lower bound by binary search; no atomics: a popular item would serialise 10^5 of them) -- and d^-1/2 per node in fp64
// (degree counts the self loop), computed once per node instead of per entry.
__device__ __forceinline__ int64_t lower_bound_item(const int32_t* __restrict__ items_sorted, int64_t n_edges, int64_t it) {
  int64_t lo = 0, hi = n_edges;
  while (lo < hi) {
    const int64_t mid = (lo + hi) >> 1;
    if ((int64_t)__ldg(items_sorted + mid) < it) lo = mid + 1; else hi = mid;
  }
  return lo;
}
__global__ void __launch_bounds__(256) offsets_dinv_kernel(const int64_t* __restrict__ row_ptr,
                                                           const int32_t* __restrict__ items_sorted, int64_t n_users,
                                                           int64_t n_items, int64_t n_edges, int64_t* __restrict__ item_ptr,
                                                           double* __restrict__ dinv) {
  // blocks [0, user_blocks): one thread per user; the others: 255 items per block + one halo search, so that every thread
  // runs ONE binary search (17 dependent loads) and reads its row end from its neighbour
  __shared__ int64_t lb[256];
  const int64_t user_blocks = (n_users + 255) / 256;
  if ((int64_t)blockIdx.x < user_blocks) {
    const int64_t u = (int64_t)blockIdx.x * 256 + threadIdx.x;
    if (u < n_users) dinv[u] = 1.0 / sqrt((double)(row_ptr[u + 1] - row_ptr[u] + 1));
    return;
  }
  const int64_t it = ((int64_t)blockIdx.x - user_blocks) * 255 + threadIdx.x;      // threadIdx.x == 255: halo
  lb[threadIdx.x] = it < n_items ? lower_bound_item(items_sorted, n_edges, it) : n_edges;
  __syncthreads();
  if (threadIdx.x == 255 || it >= n_items) return;
  const int64_t b = lb[threadIdx.x], e = lb[threadIdx.x + 1];
  item_ptr[it] = b;
  if (it + 1 == n_items) item_ptr[n_items] = n_edges;
  dinv[n_users + it] = 1.0 / sqrt((double)(e - b + 1));
}

// Entry-parallel fill (no per-row walks, so popular items with thousands of users cost the same per
// entry as everything else).  Thread j < E writes the user-side entry of edge j (CSR by user) and the
// item-side entry of the j-th (item, user) pair of the transposed list; thread j < N writes node j's
// self loop and row pointer.  Row layout: users [self | items ascending], items [users ascending | self].
__global__ void __launch_bounds__(256) fill_adj_kernel(const int64_t* __restrict__ row_ptr,
                                                       const int32_t* __restrict__ items,
                                                       const int32_t* __restrict__ edge_user,
                                                       const int64_t* __restrict__ item_ptr,
                                                       const int32_t* __restrict__ items_sorted,
                                                       const int32_t* __restrict__ users_by_item,
                                                       const double* __restrict__ dinv, int64_t n_users,
                                                       int64_t n_items, int64_t n_edges, int64_t* __restrict__ adj_ptr,
                                                       int32_t* __restrict__ adj_idx, float* __restrict__ adj_val) {
  const int64_t j = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t N = n_users + n_items;
  if (j < n_edges) {
    // an item id outside [0, n_items) (flagged in status bit 1) indexes neither dinv nor an item-side slot: its user-side
    // entry becomes (the row's own node, NaN) and its item-side entry is not written, so nothing outside the arrays is
    // touched and no stored column is >= N
    {
      const int64_t u = edge_user[j];
      const int32_t it = items[j];
      const bool ok = it >= 0 && it < n_items;
      const int64_t o = j + u + 1;  // one self loop per user row up to and including u
      adj_idx[o] = ok ? (int32_t)(n_users + it) : (int32_t)u;
      adj_val[o] = ok ? (float)((dinv[u] * 1.0) * dinv[n_users + it]) : __int_as_float(0x7FC00000);
    }
    {
      const int64_t it = items_sorted[j];
      const int32_t u = users_by_item[j];
      if (it >= 0 && it < n_items) {
        const int64_t o = n_edges + n_users + j + it;  // user block, then one self loop per preceding item row
        adj_idx[o] = u;
        adj_val[o] = (float)((dinv[n_users + it] * 1.0) * dinv[u]);
      }
    }
  }
  if (j < N) {
    const double d = dinv[j];
    int64_t start, self;
    if (j < n_users) {
      start = row_ptr[j] + j;
      self = start;
    } else {
      const int64_t it = j - n_users;
      start = n_edges + n_users + item_ptr[it] + it;
      self = n_edges + n_users + item_ptr[it + 1] + it;
    }
    adj_ptr[j] = start;
    adj_idx[self] = (int32_t)j;
    adj_val[self] = (float)((d * 1.0) * d);
    if (j == N - 1) adj_ptr[N] = 2 * n_edges + N;
  }
}

struct Workspace {
  int32_t* edge_user;      // [E]
  int32_t* items_sorted;   // [E]
  int32_t* users_by_item;  // [E]
  int32_t* item_count;     // [I] (+1 status word)
  int64_t* item_ptr;       // [I+1]
  double* dinv;            // [U+I]
  void* cub_tmp;
  size_t cub_bytes;
};

inline size_t align256(size_t x) { return (x + 255) & ~(size_t)255; }

inline size_t carve(Workspace& w, void* base, int64_t U, int64_t I, int64_t E) {
  uint8_t* p = (uint8_t*)base;
  size_t off = 0;
  const size_t e4 = align256((size_t)(E > 0 ? E : 1) * 4);
  w.edge_user = (int32_t*)(p + off); off += e4;
  w.items_sorted = (int32_t*)(p + off); off += e4;
  w.users_by_item = (int32_t*)(p + off); off += e4;
  w.item_count = (int32_t*)(p + off); off += align256((size_t)(I + 1) * 4);
  w.item_ptr = (int64_t*)(p + off); off += align256((size_t)(I + 1) * 8);
  w.dinv = (double*)(p + off); off += align256((size_t)(U + I) * 8);
  w.cub_tmp = p + off;
  return off;
}

}  // namespace

extern "C" int64_t dmm_build_adj_workspace_bytes(int64_t n_users, int64_t n_items, int64_t n_edges) {
  Workspace w;
  const size_t fixed = carve(w, nullptr, n_users, n_items, n_edges);
  // CUB's SortPairs with separate input and output arrays allocates, besides its histograms and look-back tiles (< 32 MiB
  // + 1 byte per item for int32 keys), one more key and one more value array of E x 4 bytes each whenever the sort takes
  // more than one digit pass (dispatch_radix_sort.cuh, both the onesweep and the upsweep/downsweep paths)
  const size_t e = (size_t)(n_edges > 0 ? n_edges : 0);
  return (int64_t)(fixed + (size_t)(32u << 20) + e + 2 * align256(e * sizeof(int32_t)));
}

extern "C" int dmm_build_norm_adj_csr(dmm_ctx* ctx, const int64_t* row_ptr, const int32_t* items, int64_t n_users,
                                      int64_t n_items, int64_t n_edges, int64_t* adj_ptr, int32_t* adj_idx,
                                      float* adj_val, void* workspace, int64_t workspace_bytes, int32_t* status,
                                      void* stream) {
  DMM_CHECK_ARG(ctx && row_ptr && adj_ptr && adj_idx && adj_val && workspace, "dmm_build_norm_adj_csr: null argument");
  DMM_CHECK_ARG(n_users > 0 && n_items > 0 && n_edges >= 0, "dmm_build_norm_adj_csr: bad sizes");
  DMM_CHECK_ARG(n_users + n_items < (1LL << 31) && n_edges < (1LL << 31), "dmm_build_norm_adj_csr: int32 index overflow");
  DMM_CHECK_ARG(n_edges == 0 || items, "dmm_build_norm_adj_csr: null items");
  cudaStream_t st = (cudaStream_t)stream;
  Workspace w;
  const size_t fixed = carve(w, workspace, n_users, n_items, n_edges);
  DMM_CHECK_ARG((size_t)workspace_bytes > fixed, "dmm_build_norm_adj_csr: workspace too small");
  w.cub_bytes = (size_t)workspace_bytes - fixed;

  expand_users_kernel<<<(unsigned)dmm_ceil_div(n_users * 32, 256), 256, 0, st>>>(row_ptr, n_users, w.edge_user, items, n_items,
                                                                                status);
  DMM_LAUNCH_CHECK();
  if (n_edges > 0) {
    int end_bit = 1;
    while ((1LL << end_bit) < n_items) ++end_bit;
    size_t need = 0;
    DMM_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, need, items, w.items_sorted, w.edge_user, w.users_by_item,
                                             (int)n_edges, 0, end_bit, st));
    if (need > w.cub_bytes) {
      dmm_set_error("dmm_build_norm_adj_csr: sort scratch needs %zu bytes, %zu available", need, w.cub_bytes);
      return DMM_ERR_WORKSPACE;
    }
    DMM_CUDA(cub::DeviceRadixSort::SortPairs(w.cub_tmp, need, items, w.items_sorted, w.edge_user, w.users_by_item,
                                             (int)n_edges, 0, end_bit, st));
  }
  const int64_t N = n_users + n_items;
  offsets_dinv_kernel<<<(unsigned)(dmm_ceil_div(n_users, 256) + dmm_ceil_div(n_items, 255)), 256, 0, st>>>(
      row_ptr, w.items_sorted, n_users, n_items, n_edges, w.item_ptr, w.dinv);
  DMM_LAUNCH_CHECK();
  const int64_t work = n_edges > N ? n_edges : N;
  fill_adj_kernel<<<(unsigned)dmm_ceil_div(work, 256), 256, 0, st>>>(row_ptr, items, w.edge_user, w.item_ptr, w.items_sorted,
                                                                    w.users_by_item, w.dinv, n_users, n_items, n_edges,
                                                                    adj_ptr, adj_idx, adj_val);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}
