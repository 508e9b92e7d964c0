// Dense contraction for the Denoise MLP on the Blackwell tensor pipe (sm_100a).
//
//   C[M,N] = epilogue( sum_pass A_pass[M,K] . B_pass[N,K]^T )      bf16 operands, fp32 accum in TMEM
//
// Replaces cuBLAS SGEMM behind nn.Linear / torch.mm in the reference (Model.py:205,208,212,215,
// 416-417).  Design (one CTA per SM, persistent over output tiles, warp specialised):
//   warp 0  : TMA producer   — cp.async.bulk.tensor 2D tiles (SWIZZLE_128B) into a STAGES-deep ring
//   warp 1  : MMA issuer     — one lane issues tcgen05.mma (M=128, N=BN, K=16) into TMEM
//   warp 2  : TMEM allocator — 2 accumulator stages of BN fp32 columns (epilogue overlaps next tile)
//   warps 3-10: epilogue     — tcgen05.ld 32 lanes x 32 columns, bias/tanh/posterior-mean, fp32 and
//                              split-bf16 stores (the bf16 pair is the next contraction's operand);
//                              the bf16 residual of chunk c+1 is prefetched into registers while chunk c
//                              is drained, and the first chunk's before the accumulator barrier
// The optional lo operands add the passes A_lo.B_hi and A_hi.B_lo into the same accumulator
// ("bf16x3"), which restores fp32-level accuracy without leaving the bf16 tensor pipe.
#include "common.cuh"

namespace {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_K = 64;  // 64 bf16 = 128 B = one SWIZZLE_128B row
constexpr int UMMA_K = 16;
constexpr int EPI_WARP0 = 3;   // warps 0-2: TMA producer, MMA issuer, TMEM allocator
constexpr int EPI_WARPS = 8;   // any 8 consecutive warps cover each TMEM lane quarter (warp % 4) twice
constexpr int NUM_THREADS = 32 * (EPI_WARP0 + EPI_WARPS);
constexpr int EPI_STAGE_BYTES = 4096 + 128;  // per epilogue warp: one 32 x 32 fp32 chunk (or bf16 hi + lo chunks) + 32 bias values
constexpr int MAX_STAGES = 8;
constexpr int BAR_BYTES = 512;    // full[8], empty[8], tmem_full[2], tmem_empty[2], tmem_ptr, residual barriers [EPI_WARPS][3]
constexpr int SMEM_LIMIT = 232448;  // 227 KB opt-in shared memory of sm_100
constexpr int TEPI_MAX_BUF = 3;   // fp32 chunk buffers per epilogue warp of the TMA epilogue (residual ring)

// PAIR: two CTAs of a cluster (one TPC) run ONE tcgen05.mma.cta_group::2 tile of 256 rows x BN columns; each CTA
// stages its own 128 rows of A and HALF of the B rows, so a pipeline stage is 32 KB instead of 48 KB (6 stages
// instead of 4 at BN = 256) and the shared-memory / L2 operand traffic per flop drops by a third.
template <int BN, bool PAIR = false>
struct Cfg {
  static constexpr int CTAS = PAIR ? 2 : 1;
  static constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;
  static constexpr int B_ROWS = BN / CTAS;            // B rows staged by this CTA
  static constexpr int B_BYTES = B_ROWS * BLOCK_K * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = STAGE_BYTES >= 49152 ? 4 : (STAGE_BYTES >= 32768 ? 6 : 8);
  static constexpr int TMEM_COLS = 2 * BN;  // 128 / 256 / 512: powers of two >= 32
  static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + BAR_BYTES + EPI_WARPS * EPI_STAGE_BYTES + 1024;  // + alignment slack
  static_assert(SMEM_BYTES <= SMEM_LIMIT, "exceeds the 227 KB opt-in shared memory of sm_100");
  static_assert(STAGES <= MAX_STAGES, "barrier block holds MAX_STAGES ring barriers");
};

struct GemmParams {
  int M, N, K;
  int num_m_blocks, num_n_blocks, num_k_blocks;
  // Work items: the first `full_items` are whole BLOCK_M x BN tiles (a whole number of waves over the
  // grid); the tiles of the last, partly filled wave are cut into `split` column slices of `sub_bn`
  // columns each so that the tail keeps (almost) every SM busy for 1/split of a tile time.
  int full_items, total_items, split, sub_bn;
  // split-K (single-pass bf16, fp32 partial outputs only): work item w covers the k blocks [ks * kb_per, (ks + 1) * kb_per)
  // of tile w / ksplit with ks = w % ksplit, and writes its partial product to rows ks * ks_rows + [0, M) of out_f32
  int ksplit, kb_per, ks_rows;
  int n_pass;
  int pass_a[3];  // 0 = hi, 1 = lo
  int pass_b[3];
  // shared-memory layout (byte offsets from the 1024-aligned base), chosen per launch:
  //   [0, stages * STAGE_BYTES) operand ring | off_epi: epilogue staging | off_bar: barriers (BAR_BYTES)
  // TMA epilogue: off_epi holds EPI_WARPS x nbuf fp32 chunk buffers (4 KB, SWIZZLE_128B boxes), then at off_b16
  // EPI_WARPS bf16 chunk buffers (2 KB, SWIZZLE_64B boxes), then at off_bias EPI_WARPS x 256 B of bias slots
  int stages, nbuf;
  int off_epi, off_b16, off_bias, off_bar;
  dmm_gemm_epilogue ep;
};

// ------------------------------------------------------------------------------------------ PTX
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok;
}
// Bounded wait: a protocol bug must fault the launch (reported through cudaGetLastError) instead
// of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int tag) {
  if (mbar_try_wait(bar, parity)) return;
  long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 4000000000LL) {
      printf("diffmm_b200 gemm: mbarrier timeout tag=%d block=%d thread=%d parity=%u\n", tag, blockIdx.x,
             threadIdx.x, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// Epilogue-side TMA: a 32-row x 32-column box between a swizzled shared-memory chunk buffer and global memory.
// Stores go through bulk async-groups of the issuing thread (one lane per epilogue warp); boxes are clipped at the
// tensor bounds (loads zero-fill), so ragged M / N tails need no predicates.
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(map), "r"(src), "r"(c0),
               "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {
  asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// generic-proxy shared-memory writes -> visible to the async proxy (TMA store reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// cta_group::2 flavours.  `bar` is the shared::cluster address of the LEADER CTA's barrier (mapa_shared).
__device__ __forceinline__ void tma_load_2d_pair(uint32_t dst, const CUtensorMap* map, uint32_t bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(dst),
      "l"(map), "r"(bar), "r"(c0), "r"(c1)
      : "memory");
}
// Remote arrive on the leader's barrier.  Relaxed: the only thing the waiter (MMA issuer) depends on is that this
// warp's tcgen05.ld have completed, which tcgen05.wait::ld + tcgen05.fence::before_thread_sync already guarantee;
// a .release.cluster arrive would also drain this warp's outstanding global stores (MEMBAR + ERRBAR per tile).
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t bar) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ uint32_t mapa_shared(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void tcgen05_commit_pair(uint32_t bar) {
  asm volatile(
      "tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(bar),
      "h"((uint16_t)3)
      : "memory");
}
__device__ __forceinline__ void tcgen05_mma_bf16_pair(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                      uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tcgen05_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tcgen05_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void tcgen05_mma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}

// K-major SWIZZLE_128B shared-memory matrix descriptor (sm_100 format, version 1):
//   [0,14) addr>>4 | [16,30) LBO>>4 (=1, unused for swizzled K-major) | [32,46) SBO>>4 (8 rows x 128 B = 1024)
//   [46,48) version=1 | [61,64) layout=2 (SWIZZLE_128B)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFFu) >> 4);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at [17,23), M>>4 at [24,29)
__host__ __device__ constexpr uint32_t make_idesc(int bn, int m = BLOCK_M) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(bn >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ------------------------------------------------------------------------------------------ epilogue math
// tanh(x) = 1 - 2 / (exp(2x) + 1): absolute error ~1e-7 (the outputs are compared at the scale of 1),
// saturates correctly for |x| large (exp -> inf / 0)
__device__ __forceinline__ float fast_tanh(float x) {
  const float t = __expf(2.f * x);
  return 1.f - __fdividef(2.f, t + 1.f);
}

struct WorkItem {
  int m_blk;   // row block
  int col0;    // first output column
  int bn;      // columns of this item (BN, or sub_bn for a tail slice)
  int kb0, kb1;  // k blocks of this item (split-K; otherwise all of them)
  int ks;        // split index
};
// n fastest: the CTAs running together cover every column block of a few row blocks, so each A tile is
// fetched from HBM once and re-read from L2 by its neighbours
// MUFU.TANH (max abs error ~5e-4): used where the result is rounded to bf16 anyway (rounding error 2e-3),
// i.e. by the bf16-only instantiation; the split-bf16 (fp32-faithful) one keeps fast_tanh
__device__ __forceinline__ float approx_tanh(float x) {
  float y;
  asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
// NaN-propagating maximum: a NaN anywhere in a chunk surfaces in its maximum (the top-k then takes its exact path)
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
// maximum of the valid columns of one row of a 32-column chunk (the values exactly as they are written to out_f32)
template <bool FULL>
__device__ __forceinline__ float chunk_row_max(const float (&v)[32], int n0, int N) {
  float m = __uint_as_float(0xFF800000u);
#pragma unroll
  for (int j = 0; j < 32; ++j)
    if (FULL || n0 + j < N) m = fmax_nan(m, v[j]);
  return m;
}
template <bool X3>
__device__ __forceinline__ float epi_tanh(float x) {
  return X3 ? fast_tanh(x) : approx_tanh(x);
}

template <int BN>
__device__ __forceinline__ WorkItem decode_work(int w, const GemmParams& p) {
  WorkItem it;
  it.ks = 0, it.kb0 = 0, it.kb1 = p.num_k_blocks;
  if (p.ksplit > 1) {
    it.ks = w % p.ksplit;
    w /= p.ksplit;
    it.kb0 = it.ks * p.kb_per;
    it.kb1 = min(it.kb0 + p.kb_per, p.num_k_blocks);
    it.m_blk = w / p.num_n_blocks;
    it.col0 = (w % p.num_n_blocks) * BN;
    it.bn = BN;
    return it;
  }
  if (w < p.full_items) {
    it.m_blk = w / p.num_n_blocks;
    it.col0 = (w % p.num_n_blocks) * BN;
    it.bn = BN;
  } else {
    const int r = w - p.full_items;
    const int tile = p.full_items + r / p.split;
    it.m_blk = tile / p.num_n_blocks;
    it.col0 = (tile % p.num_n_blocks) * BN + (r % p.split) * p.sub_bn;
    it.bn = p.sub_bn;
  }
  return it;
}

// ------------------------------------------------------------------------------------------ epilogue
// One work item drained by one epilogue warp (TMEM lane quarter `ew`, chunk parity `chalf`).
//
// tcgen05.ld hands every thread one ROW of a 32-column chunk, and a row-per-thread global access touches
// 32 different 128-byte lines per instruction (the L1 tag stage, not DRAM, would bound the epilogue).  So
// every global access goes through a per-warp shared-memory staging tile, swizzled so that both views are
// bank-conflict free: the row view (thread = row) used with the accumulator, and the coalesced view (4 or
// 8 consecutive lanes cover one row segment) used against global memory.  The bf16 residual and the bias
// of the NEXT chunk are fetched (coalesced) into registers while this chunk is drained; the first chunk's
// before the accumulator barrier.  X3: lo (split-bf16) residual/output parts may be present.  INTERIOR:
// the item lies fully inside [0,M) x [0,N), no bounds predicates.
template <int BN, bool X3, bool INTERIOR>
__device__ __forceinline__ void epilogue_item(const GemmParams& p, const WorkItem wi, uint8_t* const stg,
                                              const uint32_t taddr, const uint32_t tfull, const uint32_t tphase,
                                              const int ew, const int chalf, const int lane) {
  const dmm_gemm_epilogue& ep = p.ep;
  const bool res16 = ep.res_hi != nullptr;
  const bool res16lo = X3 && ep.res_lo != nullptr;
  const bool out_lo = X3 && ep.out_lo != nullptr;
  const bool has_res = res16 || ep.residual != nullptr;
  const int rbase = wi.m_blk * BLOCK_M + ew * 32;
  const int nchunks = wi.bn >> 5;
  // bf16 chunk: 32 rows x 64 B; 16-byte piece pc of row r lives at r*64 + ((pc ^ ((r >> 1) & 3)) << 4)
  auto at16 = [&](int sub, int r, int pc) -> uint4* {
    return reinterpret_cast<uint4*>(stg + sub * 2048 + r * 64 + ((pc ^ ((r >> 1) & 3)) << 4));
  };
  // fp32 chunk: 32 rows x 128 B; piece pc of row r lives at r*128 + ((pc ^ (r & 7)) << 4)
  auto at32 = [&](int r, int pc) -> uint4* { return reinterpret_cast<uint4*>(stg + r * 128 + ((pc ^ (r & 7)) << 4)); };
  float* const stg_bias = reinterpret_cast<float*>(stg + 4096);
  const int cr16 = lane >> 2, cp16 = lane & 3;  // coalesced view, bf16: rows cr16 + 8 i, piece cp16
  const int cr32 = lane >> 3, cp32 = lane & 7;  // coalesced view, fp32: rows cr32 + 4 i, piece cp32
  auto chunk_ok = [&](int c) -> bool { return c < nchunks && (INTERIOR || wi.col0 + c * 32 < p.N); };

  uint4 nh[4], nl[4];
  float nb = 0.f, nb2 = 0.f;   // bias of the chunk being drained next / of the one after it (two chunks of lead)
  float npb = 0.f, npb2 = 0.f; // same for the post-stage bias
  auto fetch_bias = [&](int c) -> float {
    const int n0 = wi.col0 + c * 32;
    return (ep.bias && chunk_ok(c) && (INTERIOR || n0 + lane < p.N)) ? __ldg(ep.bias + n0 + lane) : 0.f;
  };
  auto fetch_post_bias = [&](int c) -> float {
    const int n0 = wi.col0 + c * 32;
    return (ep.post_bias && chunk_ok(c) && (INTERIOR || n0 + lane < p.N)) ? __ldg(ep.post_bias + n0 + lane) : 0.f;
  };
  // coalesced fetch of chunk c's raw residual, bf16 hi (+ lo) or fp32 (a 16-byte piece that starts below N always
  // lies inside the padded row because the leading dimension is a multiple of 8 / 4 elements)
  auto fetch = [&](int c) {
    const int n0 = wi.col0 + c * 32;
    if (res16) {
      const int col = n0 + 8 * cp16;
      const int64_t off = (int64_t)(rbase + cr16) * ep.ld_res16 + col;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (INTERIOR || (rbase + cr16 + 8 * i < p.M && col < p.N)) {
          nh[i] = *reinterpret_cast<const uint4*>(ep.res_hi + off + (int64_t)(8 * i) * ep.ld_res16);
          if (res16lo) nl[i] = *reinterpret_cast<const uint4*>(ep.res_lo + off + (int64_t)(8 * i) * ep.ld_res16);
        }
      }
    } else if (ep.residual) {
      // fp32 residual (the z state of the hidden-space chain): the same 8 x 16 bytes per thread, coalesced view
      // (rows cr32 + 4 i, piece cp32); a piece that starts below N lies inside the padded row (ld_res % 4 == 0)
      const int col = n0 + 4 * cp32;
      const float* base = ep.residual + (int64_t)(rbase + cr32) * ep.ld_res + col;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        uint4 t = make_uint4(0u, 0u, 0u, 0u);
        if (INTERIOR || (rbase + cr32 + 4 * i < p.M && col < p.N))
          t = *reinterpret_cast<const uint4*>(base + (int64_t)(4 * i) * ep.ld_res);
        if (i < 4) nh[i] = t; else nl[i - 4] = t;
      }
    }
  };
  if (chunk_ok(chalf)) fetch(chalf);
  nb = fetch_bias(chalf);
  nb2 = fetch_bias(chalf + EPI_WARPS / 4);
  npb = fetch_post_bias(chalf);
  npb2 = fetch_post_bias(chalf + EPI_WARPS / 4);
  mbar_wait(tfull, tphase, 4);
  tcgen05_fence_after();

#pragma unroll 1
  for (int c = chalf; chunk_ok(c); c += EPI_WARPS / 4) {
    const int n0 = wi.col0 + c * 32;
    // ---- residual + bias: registers (coalesced view) -> staging tile; read back per row below
    if (ep.bias) stg_bias[lane] = nb;
    if (res16) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        *at16(0, cr16 + 8 * i, cp16) = nh[i];
        if (res16lo) *at16(1, cr16 + 8 * i, cp16) = nl[i];
      }
    } else if (ep.residual) {
#pragma unroll
      for (int i = 0; i < 8; ++i) *at32(cr32 + 4 * i, cp32) = i < 4 ? nh[i] : nl[i - 4];
    }
    // next chunk's residual / bias: in flight while this chunk is combined and stored (it may alias only the
    // output of the NEXT chunk, which this warp writes later)
    if (chunk_ok(c + EPI_WARPS / 4)) fetch(c + EPI_WARPS / 4);
    nb = nb2;                                    // staged above; rotate the two-deep bias prefetch
    nb2 = fetch_bias(c + 2 * (EPI_WARPS / 4));
    const float pb_now = npb;
    npb = npb2;
    npb2 = fetch_post_bias(c + 2 * (EPI_WARPS / 4));
    // ---- accumulator chunk
    uint32_t r[32];
    __syncwarp();  // tcgen05.ld is .sync.aligned; also publishes the staging tile to the row view
    tmem_ld_32x32(taddr + (uint32_t)(c * 32), r);
    float v[32];
#pragma unroll
    for (int q = 0; q < 4; ++q) {  // 8 columns per step
      float t[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) t[j] = __uint_as_float(r[8 * q + j]);
      if (ep.bias) {
        const float4 b0 = *reinterpret_cast<const float4*>(stg_bias + 8 * q);
        const float4 b1 = *reinterpret_cast<const float4*>(stg_bias + 8 * q + 4);
        t[0] += b0.x; t[1] += b0.y; t[2] += b0.z; t[3] += b0.w;
        t[4] += b1.x; t[5] += b1.y; t[6] += b1.z; t[7] += b1.w;
      }
      float rs[8];
      if (has_res) {
        if (res16) {
          const uint4 h = *at16(0, lane, q);
          const uint32_t wv[4] = {h.x, h.y, h.z, h.w};
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            rs[2 * e] = __uint_as_float(wv[e] << 16);
            rs[2 * e + 1] = __uint_as_float(wv[e] & 0xFFFF0000u);
          }
          if (res16lo) {
            const uint4 l = *at16(1, lane, q);
            const uint32_t lv[4] = {l.x, l.y, l.z, l.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              rs[2 * e] += __uint_as_float(lv[e] << 16);
              rs[2 * e + 1] += __uint_as_float(lv[e] & 0xFFFF0000u);
            }
          }
        } else {
          const float4 r0 = *reinterpret_cast<const float4*>(at32(lane, 2 * q));
          const float4 r1 = *reinterpret_cast<const float4*>(at32(lane, 2 * q + 1));
          rs[0] = r0.x; rs[1] = r0.y; rs[2] = r0.z; rs[3] = r0.w;
          rs[4] = r1.x; rs[5] = r1.y; rs[6] = r1.z; rs[7] = r1.w;
        }
      }
      const bool pre = has_res && ep.res_pre_act != 0;   // residual enters before the activation (K-chunked sums)
      if (pre) {
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = fmaf(ep.beta, rs[j], t[j]);
      }
      if (ep.act == 1) {
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = fast_tanh(t[j]);
      }
      if (has_res && !pre) {
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] = fmaf(ep.alpha, t[j], ep.beta * rs[j]);
      } else if (ep.alpha != 1.f) {
#pragma unroll
        for (int j = 0; j < 8; ++j) t[j] *= ep.alpha;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) v[8 * q + j] = t[j];
    }
    if (ep.cmax) {   // pruning side array of the top-k: this thread's row maximum of the chunk, from registers
      const float m = (INTERIOR || n0 + 32 <= p.N) ? chunk_row_max<true>(v, n0, p.N) : chunk_row_max<false>(v, n0, p.N);
      if (INTERIOR || rbase + lane < p.M) ep.cmax[(int64_t)(rbase + lane) * ep.ld_cmax + (n0 >> 5)] = m;
    }
    __syncwarp();  // every row has consumed the staged residual / bias: the tile is reused for the outputs

    // ---- outputs: row view -> staging tile -> coalesced global stores
    if (ep.out_f32) {
#pragma unroll
      for (int q = 0; q < 8; ++q)
        *reinterpret_cast<float4*>(at32(lane, q)) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
      __syncwarp();
      const int col = n0 + 4 * cp32;
      float* const op0 = ep.out_f32 + (int64_t)(rbase + cr32) * ep.ld_out + col;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float4 t = *reinterpret_cast<const float4*>(at32(cr32 + 4 * i, cp32));
        float* const op = op0 + (int64_t)(4 * i) * ep.ld_out;
        if (INTERIOR) {
          *reinterpret_cast<float4*>(op) = t;
        } else if (rbase + cr32 + 4 * i < p.M) {
          if (col + 4 <= p.N) {
            *reinterpret_cast<float4*>(op) = t;
          } else {
            if (col + 0 < p.N) op[0] = t.x;
            if (col + 1 < p.N) op[1] = t.y;
            if (col + 2 < p.N) op[2] = t.z;
          }
        }
      }
      __syncwarp();
    }
    if (ep.out_hi) {
      if (ep.post_bias != nullptr || ep.post_act != 0) {
        // second stage on the bf16 output only: out_hi/lo = post_act(v + post_bias) while out_f32 keeps v
        // (hidden-space chain: z_t goes to out_f32, h_{t-1} = tanh(z_t + b1'(t-1)) to the next operand).
        // The prefetched post bias is broadcast through the (already consumed) bias slot of the staging tile.
        if (ep.post_bias) {
          stg_bias[lane] = pb_now;
          __syncwarp();
#pragma unroll
          for (int q = 0; q < 8; ++q) {
            const float4 t = *reinterpret_cast<const float4*>(stg_bias + 4 * q);
            v[4 * q] += t.x; v[4 * q + 1] += t.y; v[4 * q + 2] += t.z; v[4 * q + 3] += t.w;
          }
        }
        if (ep.post_act == 1) {
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = epi_tanh<X3>(v[j]);
        }
      }
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const float x0 = v[8 * q + 2 * e], x1 = v[8 * q + 2 * e + 1];
          const __nv_bfloat162 h2 = __floats2bfloat162_rn(x0, x1);  // .x (low half) = x0
          hi[e] = *reinterpret_cast<const uint32_t*>(&h2);
          if (out_lo) {
            const __nv_bfloat162 l2 = __floats2bfloat162_rn(x0 - __uint_as_float(hi[e] << 16),
                                                           x1 - __uint_as_float(hi[e] & 0xFFFF0000u));
            lo[e] = *reinterpret_cast<const uint32_t*>(&l2);
          }
        }
        *at16(0, lane, q) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        if (out_lo) *at16(1, lane, q) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
      __syncwarp();
      const int col = n0 + 8 * cp16;
      const int64_t off = (int64_t)(rbase + cr16) * ep.ld_out16 + col;
#pragma unroll
      for (int sub = 0; sub < (X3 ? 2 : 1); ++sub) {
        if (sub == 1 && !out_lo) break;
        uint16_t* const base = (sub ? ep.out_lo : ep.out_hi) + off;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint4 t = *at16(sub, cr16 + 8 * i, cp16);
          uint16_t* const op = base + (int64_t)(8 * i) * ep.ld_out16;
          if (INTERIOR) {
            *reinterpret_cast<uint4*>(op) = t;
          } else if (rbase + cr16 + 8 * i < p.M) {
            if (col + 8 <= p.N) {
              *reinterpret_cast<uint4*>(op) = t;
            } else {
              const uint32_t wv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
              for (int e = 0; e < 8; ++e)
                if (col + e < p.N) op[e] = (uint16_t)(wv[e >> 1] >> (16 * (e & 1)));
            }
          }
        }
      }
      __syncwarp();
    }
  }
}

// ------------------------------------------------------------------------------------------ TMA epilogue
// Whole epilogue loop of one warp (TMEM lane quarter `warp & 3`, chunk parity (warp - EPI_WARP0) / 4) for the
// single-pass bf16 outputs (no lo parts, no bf16 residual): every global access of the epilogue is a TMA box.
//   * fp32 residual (the z state of the hidden-space chain, or the partial sums of a K-chunked contraction): a ring of
//     `nbuf` swizzled 32 x 32 chunk buffers per warp, filled by cp.async.bulk.tensor loads that run up to nbuf - 1
//     chunks AHEAD of the consumer and across work items, so a chunk's DRAM latency is hidden behind the chunks before
//     it instead of being paid inside the warp's dependent chain;
//   * results are written back IN PLACE into the chunk buffer (row view, same thread) and leave through one
//     cp.async.bulk.tensor store per chunk (fp32) plus one for the bf16 operand copy; the buffer is reloaded once the
//     store has read it (bulk async-group of the issuing lane);
//   * boxes are clipped at the tensor bounds by the TMA unit: no interior / boundary instantiations.
// Row view <-> box layout: fp32 chunk rows are 128 B with the 16-byte piece index XOR (row & 7) (SWIZZLE_128B), bf16
// chunk rows are 64 B with the piece index XOR ((row >> 1) & 3) (SWIZZLE_64B): conflict-free for one row per thread.
template <int BN, bool PAIR>
__device__ __forceinline__ void epilogue_warp_tma(const GemmParams& p, const CUtensorMap* tm_res, const CUtensorMap* tm_o32,
                                                  const CUtensorMap* tm_o16, uint8_t* const smem_gen,
                                                  const uint32_t smem_base, const uint32_t tmem_base, const uint32_t tfull0,
                                                  const uint32_t tempty0, const uint32_t resbar0, const uint32_t cta_rank,
                                                  const int first_item, const int item_stride, const int warp,
                                                  const int lane) {
  constexpr int CTAS = PAIR ? 2 : 1;
  constexpr int CSTEP = EPI_WARPS / 4;
  const dmm_gemm_epilogue& ep = p.ep;
  const int wq = warp - EPI_WARP0;
  const int ew = warp & 3;
  const int chalf = wq >> 2;
  const bool has_res = ep.residual != nullptr;
  const bool o32 = ep.out_f32 != nullptr, o16 = ep.out_hi != nullptr;
  const bool both = o32 && o16;
  const bool pre = has_res && ep.res_pre_act != 0;   // residual enters before the activation (K-chunked sums)
  const bool post = ep.post_bias != nullptr || ep.post_act != 0;
  const int nbuf = p.nbuf;
  uint8_t* const fbuf = smem_gen + p.off_epi + wq * nbuf * 4096;
  const uint32_t fbuf_s = smem_base + (uint32_t)(p.off_epi + wq * nbuf * 4096);
  uint8_t* const hbuf = smem_gen + p.off_b16 + wq * 2048;
  const uint32_t hbuf_s = smem_base + (uint32_t)(p.off_b16 + wq * 2048);
  float* const stg_bias = reinterpret_cast<float*>(smem_gen + p.off_bias + wq * 256);   // [0,32) bias, [32,64) post bias
  const uint32_t resbar = resbar0 + 8u * TEPI_MAX_BUF * wq;
  auto at32 = [](uint8_t* b, int r, int pc) -> float4* {
    return reinterpret_cast<float4*>(b + r * 128 + ((pc ^ (r & 7)) << 4));
  };
  auto at16 = [](uint8_t* b, int r, int pc) -> uint4* {
    return reinterpret_cast<uint4*>(b + r * 64 + ((pc ^ ((r >> 1) & 3)) << 4));
  };

  // ---- loader cursor: the (item, chunk) sequence of this warp, up to nbuf - 1 chunks ahead of the consumer
  int lw = first_item, lc = 0, lseq = 0;
  WorkItem lwi;
  bool l_valid = false, l_more = has_res;
  auto l_next = [&]() -> bool {
    for (;;) {
      if (l_valid) {
        lc += CSTEP;
        if (lc < (lwi.bn >> 5) && lwi.col0 + lc * 32 < p.N) return true;
        lw += item_stride;
        l_valid = false;
      }
      if (lw >= p.total_items) return false;
      lwi = decode_work<BN>(lw, p);
      if (lwi.col0 >= p.N) {
        lw += item_stride;
        continue;
      }
      l_valid = true;
      lc = chalf - CSTEP;
    }
  };
  int seq = 0;   // chunks consumed so far by this warp; chunk s lives in buffer s % nbuf
  auto top_up = [&]() {
    while (l_more && lseq <= seq + nbuf - 1) {
      if (!l_next()) {
        l_more = false;
        break;
      }
      if (lane == 0) {
        // the buffer held chunk lseq - nbuf <= seq - 1: its fp32 store (followed by at most one bf16 store group) must
        // have read the buffer before the TMA load overwrites it
        if (lseq >= nbuf) {
          if (both) bulk_wait_read<1>(); else bulk_wait_read<0>();
        }
        const int j = lseq % nbuf;
        mbar_expect_tx(resbar + 8u * j, 4096u);
        tma_load_2d(fbuf_s + (uint32_t)(j * 4096), tm_res, resbar + 8u * j, lwi.col0 + lc * 32,
                    (lwi.m_blk * CTAS + (int)cta_rank) * BLOCK_M + ew * 32);
      }
      ++lseq;
    }
  };

  int it = 0;
  for (int w = first_item; w < p.total_items; w += item_stride) {
    WorkItem wi = decode_work<BN>(w, p);
    if (wi.col0 >= p.N) continue;
    wi.m_blk = wi.m_blk * CTAS + (int)cta_rank;     // this CTA's 128-row block of the (pair) tile
    const int acc = it & 1;
    const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
    ++it;
    const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN);
    const int row0 = wi.m_blk * BLOCK_M + ew * 32;
    const int nchunks = wi.bn >> 5;
    auto chunk_ok = [&](int c) -> bool { return c < nchunks && wi.col0 + c * 32 < p.N; };
    auto fetch_bias = [&](const float* b, int c) -> float {
      const int n = wi.col0 + c * 32 + lane;
      return (b && c < nchunks && n < p.N) ? __ldg(b + n) : 0.f;
    };
    float nb = fetch_bias(ep.bias, chalf), nb2 = fetch_bias(ep.bias, chalf + CSTEP);
    float npb = fetch_bias(ep.post_bias, chalf), npb2 = fetch_bias(ep.post_bias, chalf + CSTEP);
    top_up();
    mbar_wait(tfull0 + 8u * acc, acc_phase, 4);
    tcgen05_fence_after();

#pragma unroll 1
    for (int c = chalf; chunk_ok(c); c += CSTEP, ++seq) {
      const int n0 = wi.col0 + c * 32;
      const int j = seq % nbuf;
      uint8_t* const fb = fbuf + j * 4096;
      stg_bias[lane] = nb;
      stg_bias[32 + lane] = npb;
      nb = nb2;
      nb2 = fetch_bias(ep.bias, c + 2 * CSTEP);
      npb = npb2;
      npb2 = fetch_bias(ep.post_bias, c + 2 * CSTEP);
      if (has_res) {
        top_up();
        mbar_wait(resbar + 8u * j, (uint32_t)(seq / nbuf) & 1u, 5);
      } else if (o32 && lane == 0) {
        // staging buffer of chunk seq - nbuf: its store must have read it
        if (both) bulk_wait_read<1>(); else bulk_wait_read<0>();
      }
      __syncwarp();  // tcgen05.ld is .sync.aligned; publishes the bias slots and lane 0's buffer-free wait
      uint32_t r[32];
      tmem_ld_32x32(taddr + (uint32_t)(c * 32), r);
      float v[32];
#pragma unroll
      for (int q = 0; q < 4; ++q) {  // 8 columns per step
        float t[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) t[e] = __uint_as_float(r[8 * q + e]);
        if (ep.bias) {
          const float4 b0 = *reinterpret_cast<const float4*>(stg_bias + 8 * q);
          const float4 b1 = *reinterpret_cast<const float4*>(stg_bias + 8 * q + 4);
          t[0] += b0.x; t[1] += b0.y; t[2] += b0.z; t[3] += b0.w;
          t[4] += b1.x; t[5] += b1.y; t[6] += b1.z; t[7] += b1.w;
        }
        float rs[8];
        if (has_res) {
          const float4 r0 = *at32(fb, lane, 2 * q);
          const float4 r1 = *at32(fb, lane, 2 * q + 1);
          rs[0] = r0.x; rs[1] = r0.y; rs[2] = r0.z; rs[3] = r0.w;
          rs[4] = r1.x; rs[5] = r1.y; rs[6] = r1.z; rs[7] = r1.w;
        }
        if (pre) {
#pragma unroll
          for (int e = 0; e < 8; ++e) t[e] = fmaf(ep.beta, rs[e], t[e]);
        }
        if (ep.act == 1) {
#pragma unroll
          for (int e = 0; e < 8; ++e) t[e] = fast_tanh(t[e]);
        }
        if (has_res && !pre) {
#pragma unroll
          for (int e = 0; e < 8; ++e) t[e] = fmaf(ep.alpha, t[e], ep.beta * rs[e]);
        } else if (ep.alpha != 1.f) {
#pragma unroll
          for (int e = 0; e < 8; ++e) t[e] *= ep.alpha;
        }
#pragma unroll
        for (int e = 0; e < 8; ++e) v[8 * q + e] = t[e];
      }
      if (ep.cmax) {   // pruning side array of the top-k: this thread's row maximum of the chunk, from registers
        const float m = (n0 + 32 <= p.N) ? chunk_row_max<true>(v, n0, p.N) : chunk_row_max<false>(v, n0, p.N);
        if (row0 + lane < p.M) ep.cmax[(int64_t)(row0 + lane) * ep.ld_cmax + (n0 >> 5)] = m;
      }
      if (o32) {
        // in place: this thread read its row of the residual above and owns the same row of the result
#pragma unroll
        for (int q = 0; q < 8; ++q) *at32(fb, lane, q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(tm_o32, fbuf_s + (uint32_t)(j * 4096), n0, row0 + wi.ks * p.ks_rows);
          bulk_commit();
        }
      }
      if (o16) {
        if (post) {
          // second stage on the bf16 output only: out_hi = post_act(v + post_bias) while out_f32 keeps v
          if (ep.post_bias) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
              const float4 t = *reinterpret_cast<const float4*>(stg_bias + 32 + 4 * q);
              v[4 * q] += t.x; v[4 * q + 1] += t.y; v[4 * q + 2] += t.z; v[4 * q + 3] += t.w;
            }
          }
          if (ep.post_act == 1) {
#pragma unroll
            for (int e = 0; e < 32; ++e) v[e] = approx_tanh(v[e]);
          }
        }
        // the bf16 buffer still feeds the previous chunk's store (only this chunk's fp32 store group is newer)
        if (lane == 0) {
          if (o32) bulk_wait_read<1>(); else bulk_wait_read<0>();
        }
        __syncwarp();
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          uint32_t hi[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) {
            const __nv_bfloat162 h2 = __floats2bfloat162_rn(v[8 * q + 2 * e], v[8 * q + 2 * e + 1]);  // .x (low half) first
            hi[e] = *reinterpret_cast<const uint32_t*>(&h2);
          }
          *at16(hbuf, lane, q) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        }
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) {
          tma_store_2d(tm_o16, hbuf_s, n0, row0);
          bulk_commit();
        }
      }
    }
    tcgen05_fence_before();
    __syncwarp();
    if (lane == 0) {
      // the MMA issuer (leader CTA) reuses the accumulator stage once every epilogue warp of the pair has left it
      if (PAIR && cta_rank != 0) mbar_arrive_cluster(mapa_shared(tempty0 + 8u * acc, 0)); else mbar_arrive(tempty0 + 8u * acc);
    }
  }
  if (lane == 0) bulk_wait_all();   // every store has left shared memory and is performed before the CTA retires
}

// barrier block (byte offsets from smem_base + p.off_bar)
constexpr uint32_t BAR_FULL = 0, BAR_EMPTY = 8 * MAX_STAGES, BAR_TFULL = 16 * MAX_STAGES, BAR_TEMPTY = BAR_TFULL + 16,
                   BAR_TMEMPTR = BAR_TEMPTY + 16, BAR_RES = BAR_TMEMPTR + 8;
static_assert(BAR_RES + 8 * TEPI_MAX_BUF * EPI_WARPS <= BAR_BYTES, "barrier block too small");

template <int BN, bool X3, bool PAIR, bool TEPI>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_tn_kernel(const __grid_constant__ CUtensorMap tm_a_hi, const __grid_constant__ CUtensorMap tm_a_lo,
                    const __grid_constant__ CUtensorMap tm_b_hi, const __grid_constant__ CUtensorMap tm_b_lo,
                    const __grid_constant__ CUtensorMap tm_bs_hi, const __grid_constant__ CUtensorMap tm_bs_lo,
                    const __grid_constant__ CUtensorMap tm_res, const __grid_constant__ CUtensorMap tm_o32,
                    const __grid_constant__ CUtensorMap tm_o16, const GemmParams p) {
  using C = Cfg<BN, PAIR>;
  static_assert(!(TEPI && X3), "the TMA epilogue serves the single-pass bf16 outputs");
  // PAIR: CTA rank inside the 2-CTA cluster (0 = leader: issues the MMAs, owns the barriers the peer signals)
  const uint32_t cta_rank = PAIR ? cluster_ctarank() : 0u;
  const int first_item = PAIR ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
  const int item_stride = PAIR ? (int)(gridDim.x >> 1) : (int)gridDim.x;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t bar_base = smem_base + (uint32_t)p.off_bar;
  const int STAGES = p.stages;
  auto full_bar = [&](int s) { return bar_base + BAR_FULL + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + BAR_EMPTY + 8u * s; };
  auto tfull_bar = [&](int a) { return bar_base + BAR_TFULL + 8u * a; };
  auto tempty_bar = [&](int a) { return bar_base + BAR_TEMPTY + 8u * a; };
  const uint32_t tmem_ptr_addr = bar_base + BAR_TMEMPTR;
  volatile uint32_t* tmem_ptr_generic = reinterpret_cast<volatile uint32_t*>(smem_gen + p.off_bar + BAR_TMEMPTR);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;

  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    if (TEPI) {
      for (int i = 0; i < TEPI_MAX_BUF * EPI_WARPS; ++i) mbar_init(bar_base + BAR_RES + 8u * i, 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(tfull_bar(a), 1);
      mbar_init(tempty_bar(a), EPI_WARPS * C::CTAS);   // PAIR: the peer's epilogue warps arrive on the leader's barrier
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 2) {
    if (PAIR) {
      // collective over the CTA pair: one warp of each CTA, same columns in both SMs
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_ptr_addr),
                   "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tcgen05_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();   // PAIR: no remote arrive may hit an uninitialised barrier
  tcgen05_fence_after();
  const uint32_t tmem_base = *tmem_ptr_generic;

  // items whose first column lies beyond N (slices of a ragged last column block) are skipped by all roles

  if (warp == 0) {
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int w = first_item; w < p.total_items; w += item_stride) {
        const WorkItem wi = decode_work<BN>(w, p);
        if (wi.col0 >= p.N) continue;
        const bool sub = wi.bn != BN;
        // bytes landing on the (leader's) full barrier per stage: both CTAs' A tiles and B halves
        const uint32_t tx_bytes = (uint32_t)(C::CTAS * C::A_BYTES + wi.bn * BLOCK_K * 2);
        const int a_row = (wi.m_blk * C::CTAS + (int)cta_rank) * BLOCK_M;
        const int b_row = wi.col0 + (int)cta_rank * (wi.bn / C::CTAS);
        for (int ps = 0; ps < p.n_pass; ++ps) {
          const CUtensorMap* ma = p.pass_a[ps] ? &tm_a_lo : &tm_a_hi;
          const CUtensorMap* mb = p.pass_b[ps] ? (sub ? &tm_bs_lo : &tm_b_lo) : (sub ? &tm_bs_hi : &tm_b_hi);
          for (int kb = wi.kb0; kb < wi.kb1; ++kb) {
            mbar_wait(empty_bar(stage), phase ^ 1u, 1);
            const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
            if (PAIR) {
              // the leader arms its barrier for the whole pair; the peer's copies complete on the leader's barrier too
              if (cta_rank == 0) mbar_expect_tx(full_bar(stage), tx_bytes);
              const uint32_t lead_bar = mapa_shared(full_bar(stage), 0);
              tma_load_2d_pair(sa, ma, lead_bar, kb * BLOCK_K, a_row);
              tma_load_2d_pair(sa + C::A_BYTES, mb, lead_bar, kb * BLOCK_K, b_row);
            } else {
              mbar_expect_tx(full_bar(stage), tx_bytes);
              tma_load_2d(sa, ma, full_bar(stage), kb * BLOCK_K, a_row);
              tma_load_2d(sa + C::A_BYTES, mb, full_bar(stage), kb * BLOCK_K, b_row);
            }
            if (++stage == STAGES) {
              stage = 0;
              phase ^= 1u;
            }
          }
        }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    if (lane == 0 && cta_rank == 0) {   // PAIR: only the leader CTA issues the (pair-wide) MMAs
      int stage = 0;
      uint32_t phase = 0;
      int it = 0;
      for (int w = first_item; w < p.total_items; w += item_stride) {
        const WorkItem wi = decode_work<BN>(w, p);
        if (wi.col0 >= p.N) continue;
        const uint32_t idesc = make_idesc(wi.bn, BLOCK_M * C::CTAS);
        const int acc = it & 1;
        const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
        mbar_wait(tempty_bar(acc), acc_phase ^ 1u, 2);
        tcgen05_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BN);
        const int k_iters = p.n_pass * (wi.kb1 - wi.kb0);
        for (int j = 0; j < k_iters; ++j) {
          mbar_wait(full_bar(stage), phase, 3);
          tcgen05_fence_after();
          const uint32_t sa = smem_base + stage * C::STAGE_BYTES;
          const uint64_t adesc = make_smem_desc(sa);
          const uint64_t bdesc = make_smem_desc(sa + C::A_BYTES);
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            // +32 B per UMMA_K step inside the 128 B swizzle row => +2 in the (addr >> 4) field
            if (PAIR) {
              tcgen05_mma_bf16_pair(tmem_d, adesc + 2u * k, bdesc + 2u * k, idesc, (j > 0 || k > 0) ? 1u : 0u);
            } else {
              tcgen05_mma_bf16(tmem_d, adesc + 2u * k, bdesc + 2u * k, idesc, (j > 0 || k > 0) ? 1u : 0u);
            }
          }
          // smem slot is free once these MMAs retire (PAIR: in both CTAs, the commit multicasts to the same
          // barrier offset of the peer)
          if (PAIR) tcgen05_commit_pair(empty_bar(stage)); else tcgen05_commit(empty_bar(stage));
          if (++stage == STAGES) {
            stage = 0;
            phase ^= 1u;
          }
        }
        // accumulator ready for the epilogue (of both CTAs)
        if (PAIR) tcgen05_commit_pair(tfull_bar(acc)); else tcgen05_commit(tfull_bar(acc));
        ++it;
      }
    }
    __syncwarp();
  } else if (warp >= EPI_WARP0) {
    // 8 epilogue warps: warp % 4 selects the TMEM lane quarter (hardware rule), (warp - EPI_WARP0) / 4
    // the parity of the 32-column chunks this warp drains.
    if constexpr (TEPI) {
      epilogue_warp_tma<BN, PAIR>(p, &tm_res, &tm_o32, &tm_o16, smem_gen, smem_base, tmem_base, tfull_bar(0), tempty_bar(0),
                                  bar_base + BAR_RES, cta_rank, first_item, item_stride, warp, lane);
    } else {
    const int ew = warp & 3;
    const int chalf = (warp - EPI_WARP0) >> 2;
    uint8_t* const stg = smem_gen + p.off_epi + (warp - EPI_WARP0) * EPI_STAGE_BYTES;
    int it = 0;
    for (int w = first_item; w < p.total_items; w += item_stride) {
      WorkItem wi = decode_work<BN>(w, p);
      if (wi.col0 >= p.N) continue;
      wi.m_blk = wi.m_blk * C::CTAS + (int)cta_rank;     // this CTA's 128-row block of the (pair) tile
      const int acc = it & 1;
      const uint32_t acc_phase = (uint32_t)(it >> 1) & 1u;
      ++it;
      const uint32_t taddr = tmem_base + ((uint32_t)(ew * 32) << 16) + (uint32_t)(acc * BN);
      const bool interior = (wi.m_blk + 1) * BLOCK_M <= p.M && wi.col0 + wi.bn <= p.N;
      if (interior) {
        epilogue_item<BN, X3, true>(p, wi, stg, taddr, tfull_bar(acc), acc_phase, ew, chalf, lane);
      } else {
        epilogue_item<BN, X3, false>(p, wi, stg, taddr, tfull_bar(acc), acc_phase, ew, chalf, lane);
      }
      tcgen05_fence_before();
      __syncwarp();
      if (lane == 0) {
        // the MMA issuer (leader CTA) reuses the accumulator stage once every epilogue warp of the pair has left it
        if (PAIR && cta_rank != 0) mbar_arrive_cluster(mapa_shared(tempty_bar(acc), 0)); else mbar_arrive(tempty_bar(acc));
      }
    }
    }
  }

  tcgen05_fence_before();
  if (PAIR) cluster_sync_all(); else __syncthreads();   // PAIR: the peer may still be signalling this CTA's barriers
  if (warp == 2) {
    tcgen05_fence_after();
    if (PAIR) {
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
    } else {
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)C::TMEM_COLS)
                   : "memory");
    }
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

int make_map(dmm_ctx* ctx, CUtensorMap* map, const uint16_t* base, int64_t rows, int64_t k, int64_t ld, int box_rows) {
  cuuint64_t dims[2] = {(cuuint64_t)k, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)BLOCK_K, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ((EncodeTiledFn)ctx->encode_tiled)(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, (void*)base, dims, strides, box,
                                                  estr, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    dmm_set_error("cuTensorMapEncodeTiled failed (%d) rows=%lld k=%lld ld=%lld", (int)r, (long long)rows, (long long)k,
                  (long long)ld);
    return DMM_ERR_CUDA;
  }
  return DMM_OK;
}

// 32 x 32 element box of an epilogue tensor ([rows, cols] row-major, leading dimension ld): fp32 rows are 128 B
// (SWIZZLE_128B), bf16 rows 64 B (SWIZZLE_64B) -- the layouts of the epilogue's chunk buffers
int make_epi_map(dmm_ctx* ctx, CUtensorMap* map, const void* base, bool f32, int64_t rows, int64_t cols, int64_t ld) {
  cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * (f32 ? 4 : 2)};
  cuuint32_t box[2] = {32, 32};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = ((EncodeTiledFn)ctx->encode_tiled)(
      map, f32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides,
      box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, f32 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
      CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    dmm_set_error("cuTensorMapEncodeTiled (epilogue) failed (%d) rows=%lld cols=%lld ld=%lld", (int)r, (long long)rows,
                  (long long)cols, (long long)ld);
    return DMM_ERR_CUDA;
  }
  return DMM_OK;
}

// Shared-memory bytes of the TMA epilogue next to the operand ring: per epilogue warp nbuf fp32 chunk buffers (4 KB,
// SWIZZLE_128B boxes), a bf16 chunk buffer (2 KB, SWIZZLE_64B boxes) when there is a bf16 output, and 256 B of bias
// slots; then the barrier block.
int tepi_bytes(int nbuf, bool out_hi) { return EPI_WARPS * nbuf * 4096 + (out_hi ? EPI_WARPS * 2048 : 0) + EPI_WARPS * 256 + BAR_BYTES; }

// split-K work items per tile (1: the shape does not split)
int splitk_factor(int sms, int64_t M, int64_t N, int64_t K) {
  const int64_t tiles = dmm_ceil_div(M, 2 * BLOCK_M) * dmm_ceil_div(N, 256);
  const int64_t slots = sms / 2;
  const int64_t kblocks = dmm_ceil_div(K, BLOCK_K);
  int64_t ks = slots / (tiles > 0 ? tiles : 1);
  if (ks > 8) ks = 8;
  if (ks > kblocks / 8) ks = kblocks / 8;          // at least 8 k blocks (512 columns of K) per work item
  if (ks < 2 || N <= 128) return 1;
  const int64_t per = dmm_ceil_div(kblocks, ks);
  return (int)dmm_ceil_div(kblocks, per);          // no empty split
}

// The launch plan (dmm_gemm_plan): every decision of a launch that is not fixed by the arguments.  Host arithmetic
// only; the contraction launches exactly what this returns.
int plan_gemm(int sms, int64_t M, int64_t N, int64_t K, uint32_t flags, dmm_gemm_launch_plan* pl) {
  pl->ksplit = 1;
  if (flags & DMM_GEMM_SPLITK) {
    pl->ksplit = splitk_factor(sms, M, N, K);
    if (pl->ksplit > 1) flags = DMM_GEMM_OUT_F32;   // the work items write plain fp32 partial products to slabs
  }
  // Tile shape by a small cost model: waves over the SMs (or SM pairs) x work per SM and wave / measured relative
  // efficiency of the shape (256-wide pair tiles 1.0, single-CTA 256 / 128 / 64 columns 0.93 / 0.80 / 0.55).
  const int64_t m128 = dmm_ceil_div(M, BLOCK_M), m256 = dmm_ceil_div(M, 2 * BLOCK_M);
  auto waves = [](int64_t tiles, int64_t slots) { return (double)dmm_ceil_div(tiles, slots); };
  double best = 1e300;
  int bn = 64;
  bool pair = false;
  auto consider = [&](int cand_bn, bool cand_pair, double cost) {
    if (cost < best) { best = cost; bn = cand_bn; pair = cand_pair; }
  };
  consider(64, false, waves(m128 * dmm_ceil_div(N, 64), sms) * 64.0 / 0.55);
  if (N > 64) consider(128, false, waves(m128 * dmm_ceil_div(N, 128), sms) * 128.0 / 0.80);
  if (N > 128) {
    consider(256, false, waves(m128 * dmm_ceil_div(N, 256), sms) * 256.0 / 0.93);
    if (sms >= 2) consider(256, true, waves(m256 * dmm_ceil_div(N, 256), sms / 2) * 256.0 / 1.0);
  }
  if (pl->ksplit > 1) {
    bn = 256;
    pair = true;
  }
  pl->bn = bn;
  pl->ctas = pair ? 2 : 1;
  // work items are tiles of (BLOCK_M * CTAS) rows; one persistent CTA (or CTA pair) per SM (or TPC)
  const int64_t tiles = dmm_ceil_div(M, (int64_t)BLOCK_M * pl->ctas) * dmm_ceil_div(N, bn) * pl->ksplit;
  const int64_t slots = sms / pl->ctas;
  const int64_t grid = tiles < slots ? tiles : slots;
  pl->grid = (int)(grid * pl->ctas);
  // tail wave: when the last wave would fill at most half of the grid, cut its tiles into column slices
  const int64_t rem = tiles % grid;
  pl->split = 1;
  if (rem > 0 && tiles > grid && pl->ksplit == 1) {
    while (pl->split * 2 <= bn / 64 && rem * pl->split * 2 <= grid) pl->split *= 2;
  }
  pl->sub_bn = bn / pl->split;
  // TMA epilogue (residual prefetch ring + bulk tensor stores) for the single-pass bf16 configurations; the
  // register-staged epilogue serves the rest (split-bf16 operands, bf16 residual or lo output), in its split-bf16
  // (fp32-faithful) instantiation whenever ANY lo part takes part: it keeps the accurate tanh in the post stage
  const bool tepi = !(flags & (DMM_GEMM_A_LO | DMM_GEMM_B_LO | DMM_GEMM_RES_HI | DMM_GEMM_RES_LO | DMM_GEMM_OUT_LO)) &&
                    (flags & (DMM_GEMM_OUT_F32 | DMM_GEMM_OUT_HI));
  const bool x3 = flags & (DMM_GEMM_A_LO | DMM_GEMM_B_LO | DMM_GEMM_RES_LO | DMM_GEMM_OUT_LO);
  pl->epilogue = tepi ? DMM_GEMM_EPI_TMA : (x3 ? DMM_GEMM_EPI_REG_X3 : DMM_GEMM_EPI_REG);
  const int stage_bytes = BLOCK_M * BLOCK_K * 2 + (bn / pl->ctas) * BLOCK_K * 2;   // Cfg<bn, pair>::STAGE_BYTES
  const int max_stages = bn == 64 ? Cfg<64>::STAGES : bn == 128 ? Cfg<128>::STAGES
                         : pair ? Cfg<256, true>::STAGES : Cfg<256, false>::STAGES;
  pl->nbuf = 1;
  pl->stages = max_stages;
  if (tepi) {
    // with an fp32 residual every epilogue warp owns a ring of chunk buffers (prefetch depth nbuf - 1) and the
    // operand ring takes what is left
    pl->nbuf = (flags & DMM_GEMM_RESIDUAL) ? 2 : 1;   // measured: a 4-stage operand ring + 2 chunk buffers beats 3 stages + 3 buffers
    const int stages = (SMEM_LIMIT - 1024 - tepi_bytes(pl->nbuf, flags & DMM_GEMM_OUT_HI)) / stage_bytes;
    if (stages < 2) {
      dmm_set_error("dmm_gemm_bf16_tn: no room for the operand ring next to the TMA epilogue (BN=%d)", bn);
      return DMM_ERR_INVALID;
    }
    if (stages < pl->stages) pl->stages = stages;
  }
  return DMM_OK;
}

template <int BN, bool PAIR>
int launch(dmm_ctx* ctx, const uint16_t* a_hi, const uint16_t* a_lo, int64_t lda, const uint16_t* b_hi,
           const uint16_t* b_lo, int64_t ldb, GemmParams& p, const dmm_gemm_launch_plan& pl, cudaStream_t stream) {
  using C = Cfg<BN, PAIR>;
  static_assert(C::STAGE_BYTES == BLOCK_M * BLOCK_K * 2 + (BN / C::CTAS) * BLOCK_K * 2, "plan_gemm's ring arithmetic");
  CUtensorMap ma_hi, ma_lo, mb_hi, mb_lo, mbs_hi, mbs_lo, m_res, m_o32, m_o16;
  int rc;
  const bool tepi = pl.epilogue == DMM_GEMM_EPI_TMA;
  p.num_n_blocks = (int)dmm_ceil_div(p.N, BN);
  const int m_items = (int)dmm_ceil_div(p.M, (int64_t)BLOCK_M * C::CTAS);
  p.num_m_blocks = m_items;
  const int tiles = m_items * p.num_n_blocks * p.ksplit;      // split-K: every tile is ksplit work items
  const int grid = pl.grid / C::CTAS;
  const int rem = tiles % grid;
  p.split = pl.split;
  p.sub_bn = pl.sub_bn;
  p.full_items = p.split > 1 ? tiles - rem : tiles;
  p.total_items = p.full_items + (p.split > 1 ? rem * p.split : 0);
  p.stages = pl.stages;
  p.nbuf = pl.nbuf;
  if ((rc = make_map(ctx, &ma_hi, a_hi, p.M, p.K, lda, BLOCK_M))) return rc;
  if ((rc = make_map(ctx, &ma_lo, a_lo ? a_lo : a_hi, p.M, p.K, lda, BLOCK_M))) return rc;
  if ((rc = make_map(ctx, &mb_hi, b_hi, p.N, p.K, ldb, BN / C::CTAS))) return rc;
  if ((rc = make_map(ctx, &mb_lo, b_lo ? b_lo : b_hi, p.N, p.K, ldb, BN / C::CTAS))) return rc;
  if ((rc = make_map(ctx, &mbs_hi, b_hi, p.N, p.K, ldb, p.sub_bn / C::CTAS))) return rc;
  if ((rc = make_map(ctx, &mbs_lo, b_lo ? b_lo : b_hi, p.N, p.K, ldb, p.sub_bn / C::CTAS))) return rc;
  m_res = ma_hi;
  m_o32 = ma_hi;
  m_o16 = ma_hi;   // placeholders: never dereferenced unless the matching epilogue pointer is set
  int smem_bytes;
  if (tepi) {
    // shared-memory layout of the TMA epilogue (tepi_bytes)
    p.off_epi = p.stages * C::STAGE_BYTES;
    p.off_b16 = p.off_epi + EPI_WARPS * p.nbuf * 4096;
    p.off_bias = p.off_b16 + (p.ep.out_hi ? EPI_WARPS * 2048 : 0);
    p.off_bar = p.off_bias + EPI_WARPS * 256;
    smem_bytes = p.off_bar + BAR_BYTES + 1024;
    if (p.ep.residual && (rc = make_epi_map(ctx, &m_res, p.ep.residual, true, p.M, p.N, p.ep.ld_res))) return rc;
    // split-K: the partial products are slabs of ks_rows rows, one per split
    const int64_t o32_rows = p.ksplit > 1 ? (int64_t)p.ksplit * p.ks_rows : (int64_t)p.M;
    if (p.ep.out_f32 && (rc = make_epi_map(ctx, &m_o32, p.ep.out_f32, true, o32_rows, p.N, p.ep.ld_out))) return rc;
    if (p.ep.out_hi && (rc = make_epi_map(ctx, &m_o16, p.ep.out_hi, false, p.M, p.N, p.ep.ld_out16))) return rc;
  } else {
    p.off_bar = C::STAGES * C::STAGE_BYTES;
    p.off_epi = p.off_bar + BAR_BYTES;
    p.off_b16 = p.off_bias = 0;
    smem_bytes = C::SMEM_BYTES;
  }
  static DmmPerDeviceOnce attr_once;   // one per template instantiation; per device, thread-safe
  if (attr_once.need(ctx)) {
    DMM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_kernel<BN, false, PAIR, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    DMM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_kernel<BN, true, PAIR, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    DMM_CUDA(cudaFuncSetAttribute(gemm_bf16_tn_kernel<BN, false, PAIR, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_LIMIT));
    attr_once.mark(ctx);
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)pl.grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = (size_t)smem_bytes;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = C::CTAS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = PAIR ? 1 : 0;
  if (tepi) {
    DMM_CUDA(cudaLaunchKernelEx(&cfg, gemm_bf16_tn_kernel<BN, false, PAIR, true>, ma_hi, ma_lo, mb_hi, mb_lo, mbs_hi, mbs_lo,
                                m_res, m_o32, m_o16, p));
  } else if (pl.epilogue == DMM_GEMM_EPI_REG_X3) {
    DMM_CUDA(cudaLaunchKernelEx(&cfg, gemm_bf16_tn_kernel<BN, true, PAIR, false>, ma_hi, ma_lo, mb_hi, mb_lo, mbs_hi, mbs_lo,
                                m_res, m_o32, m_o16, p));
  } else {
    DMM_CUDA(cudaLaunchKernelEx(&cfg, gemm_bf16_tn_kernel<BN, false, PAIR, false>, ma_hi, ma_lo, mb_hi, mb_lo, mbs_hi, mbs_lo,
                                m_res, m_o32, m_o16, p));
  }
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

// fixed-order sum of the split-K partial slabs -> fp32 and / or bf16 hi (+ lo) operand copies
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ part, int ksplit, int64_t slab, int64_t ld_p,
                                                            int64_t M, int64_t N, float* __restrict__ out_f32, int64_t ld_out,
                                                            uint16_t* __restrict__ out_hi, uint16_t* __restrict__ out_lo,
                                                            int64_t ld16) {
  const int64_t n4 = (N + 3) >> 2;
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M * n4) return;
  const int64_t r = i / n4, c = (i % n4) * 4;
  float4 acc = __ldcs(reinterpret_cast<const float4*>(part + r * ld_p + c));
  for (int s = 1; s < ksplit; ++s) {
    const float4 v = __ldcs(reinterpret_cast<const float4*>(part + s * slab + r * ld_p + c));
    acc.x += v.x, acc.y += v.y, acc.z += v.z, acc.w += v.w;
  }
  const float v[4] = {acc.x, acc.y, acc.z, acc.w};
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    if (c + e >= N) break;
    if (out_f32) out_f32[r * ld_out + c + e] = v[e];
    if (out_hi) {
      uint16_t hi, lo;
      dmm_split_bf16(v[e], hi, lo);
      out_hi[r * ld16 + c + e] = hi;
      if (out_lo) out_lo[r * ld16 + c + e] = lo;
    }
  }
}

int run_gemm(dmm_ctx* ctx, const uint16_t* a_hi, const uint16_t* a_lo, int64_t lda, const uint16_t* b_hi, const uint16_t* b_lo,
             int64_t ldb, int64_t M, int64_t N, int64_t K, const dmm_gemm_epilogue* ep, bool splitk, int ks_rows, void* stream);

}  // namespace

extern "C" int dmm_gemm_bf16_tn(dmm_ctx* ctx, const uint16_t* a_hi, const uint16_t* a_lo, int64_t lda,
                                const uint16_t* b_hi, const uint16_t* b_lo, int64_t ldb, int64_t M, int64_t N,
                                int64_t K, const dmm_gemm_epilogue* ep, void* stream) {
  return run_gemm(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, M, N, K, ep, false, 0, stream);
}

// Split-K for contractions with few output tiles and a long K (P = W1x W2 of the hidden-space chain: 1024 x 1024 x I is 16
// pair tiles on 74 pair slots): each tile's k blocks are divided over up to 8 work items whose fp32 partial products go to
// slabs of the workspace; a second small launch adds the slabs in a fixed order (deterministic) and writes the fp32 result
// and / or its bf16 operand copies.  Falls back to the plain contraction when the tiles already fill the machine.
extern "C" int64_t dmm_gemm_splitk_workspace_bytes(dmm_ctx* ctx, int64_t M, int64_t N, int64_t K) {
  if (!ctx) return 0;
  const int ks = splitk_factor(ctx->num_sms, M, N, K);
  if (ks <= 1) return 0;
  const int64_t rows = dmm_ceil_div(M, 2 * BLOCK_M) * 2 * BLOCK_M, ld = (N + 3) & ~(int64_t)3;
  return (int64_t)ks * rows * ld * (int64_t)sizeof(float);
}

extern "C" int dmm_gemm_bf16_tn_splitk(dmm_ctx* ctx, const uint16_t* a_hi, int64_t lda, const uint16_t* b_hi, int64_t ldb,
                                       int64_t M, int64_t N, int64_t K, float* out_f32, int64_t ld_out, uint16_t* out_hi,
                                       uint16_t* out_lo, int64_t ld_out16, void* workspace, int64_t workspace_bytes,
                                       void* stream) {
  DMM_CHECK_ARG(ctx && a_hi && b_hi && (out_f32 || out_hi), "dmm_gemm_bf16_tn_splitk: null argument");
  DMM_CHECK_ARG(M > 0 && N > 0 && K > 0 && M < (1LL << 31) && N < (1LL << 31) && K < (1LL << 31), "dmm_gemm_bf16_tn_splitk: bad shape");
  DMM_CHECK_ARG(!out_f32 || ld_out >= N, "dmm_gemm_bf16_tn_splitk: ld_out must be >= N");
  DMM_CHECK_ARG(!out_hi || ld_out16 >= N, "dmm_gemm_bf16_tn_splitk: ld_out16 must be >= N");
  DMM_CHECK_ARG(!out_lo || out_hi, "dmm_gemm_bf16_tn_splitk: out_lo requires out_hi");
  uint32_t flags = DMM_GEMM_SPLITK | (out_f32 ? DMM_GEMM_OUT_F32 : 0) | (out_hi ? DMM_GEMM_OUT_HI : 0) | (out_lo ? DMM_GEMM_OUT_LO : 0);
  dmm_gemm_launch_plan pl;
  int rc = plan_gemm(ctx->num_sms, M, N, K, flags, &pl);
  if (rc) return rc;
  const int ks = pl.ksplit;
  if (ks <= 1) {
    // plain contraction; the bf16 lo part needs the fp32 result, which the split path has anyway
    DMM_CHECK_ARG(!out_lo || out_f32, "dmm_gemm_bf16_tn_splitk: out_lo without out_f32 needs a split (shape does not split)");
    dmm_gemm_epilogue ep = {};
    ep.alpha = 1.f;
    ep.out_f32 = out_f32, ep.ld_out = ld_out, ep.out_hi = out_hi, ep.out_lo = out_lo, ep.ld_out16 = ld_out16;
    return run_gemm(ctx, a_hi, nullptr, lda, b_hi, nullptr, ldb, M, N, K, &ep, false, 0, stream);
  }
  DMM_CHECK_ARG(workspace && workspace_bytes >= dmm_gemm_splitk_workspace_bytes(ctx, M, N, K) &&
                    (reinterpret_cast<uintptr_t>(workspace) & 15u) == 0,
                "dmm_gemm_bf16_tn_splitk: workspace of dmm_gemm_splitk_workspace_bytes bytes (16-byte aligned) required");
  const int64_t rows = dmm_ceil_div(M, 2 * BLOCK_M) * 2 * BLOCK_M, ld = (N + 3) & ~(int64_t)3;
  dmm_gemm_epilogue ep = {};
  ep.alpha = 1.f;
  ep.out_f32 = (float*)workspace;
  ep.ld_out = ld;
  rc = run_gemm(ctx, a_hi, nullptr, lda, b_hi, nullptr, ldb, M, N, K, &ep, true, (int)rows, stream);
  if (rc) return rc;
  const int64_t work = M * ((N + 3) >> 2);
  splitk_reduce_kernel<<<(unsigned)dmm_ceil_div(work, 256), 256, 0, (cudaStream_t)stream>>>(
      (const float*)workspace, ks, rows * ld, ld, M, N, out_f32, ld_out, out_hi, out_lo, ld_out16);
  DMM_LAUNCH_CHECK();
  return DMM_OK;
}

namespace {
int run_gemm(dmm_ctx* ctx, const uint16_t* a_hi, const uint16_t* a_lo, int64_t lda, const uint16_t* b_hi, const uint16_t* b_lo,
             int64_t ldb, int64_t M, int64_t N, int64_t K, const dmm_gemm_epilogue* ep, bool splitk, int ks_rows, void* stream) {
  DMM_CHECK_ARG(ctx && a_hi && b_hi && ep, "dmm_gemm_bf16_tn: null argument");
  DMM_CHECK_ARG(ctx->encode_tiled, "dmm_gemm_bf16_tn: cuTensorMapEncodeTiled unavailable");
  DMM_CHECK_ARG(M > 0 && N > 0 && K > 0, "dmm_gemm_bf16_tn: empty problem M=%lld N=%lld K=%lld", (long long)M,
                (long long)N, (long long)K);
  DMM_CHECK_ARG(M < (1LL << 31) && N < (1LL << 31) && K < (1LL << 31), "dmm_gemm_bf16_tn: dimension too large");
  DMM_CHECK_ARG(lda >= K && ldb >= K && lda % 8 == 0 && ldb % 8 == 0,
                "dmm_gemm_bf16_tn: lda/ldb must be >= K and multiples of 8 (got %lld, %lld, K=%lld)", (long long)lda,
                (long long)ldb, (long long)K);
  auto al16 = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15u) == 0; };
  DMM_CHECK_ARG(al16(a_hi) && al16(a_lo) && al16(b_hi) && al16(b_lo), "dmm_gemm_bf16_tn: operands must be 16-byte aligned");
  DMM_CHECK_ARG(al16(ep->residual) && al16(ep->out_f32) && al16(ep->out_hi) && al16(ep->out_lo),
                "dmm_gemm_bf16_tn: epilogue buffers must be 16-byte aligned");
  DMM_CHECK_ARG(!ep->residual || (ep->ld_res >= N && ep->ld_res % 4 == 0), "dmm_gemm_bf16_tn: ld_res must be >= N and %%4");
  DMM_CHECK_ARG(!(ep->residual && ep->res_hi), "dmm_gemm_bf16_tn: residual and res_hi are mutually exclusive");
  DMM_CHECK_ARG(!ep->res_hi || (ep->ld_res16 >= N && ep->ld_res16 % 8 == 0), "dmm_gemm_bf16_tn: ld_res16 must be >= N and %%8");
  DMM_CHECK_ARG(!ep->res_lo || ep->res_hi, "dmm_gemm_bf16_tn: res_lo requires res_hi");
  DMM_CHECK_ARG(al16(ep->res_hi) && al16(ep->res_lo), "dmm_gemm_bf16_tn: res_hi/res_lo must be 16-byte aligned");
  DMM_CHECK_ARG(!ep->out_f32 || (ep->ld_out >= N && ep->ld_out % 4 == 0), "dmm_gemm_bf16_tn: ld_out must be >= N and %%4");
  DMM_CHECK_ARG(!ep->out_hi || (ep->ld_out16 >= N && ep->ld_out16 % 8 == 0), "dmm_gemm_bf16_tn: ld_out16 must be >= N and %%8");
  DMM_CHECK_ARG(!ep->out_lo || ep->out_hi, "dmm_gemm_bf16_tn: out_lo requires out_hi");
  DMM_CHECK_ARG(ep->act == 0 || ep->act == 1, "dmm_gemm_bf16_tn: unknown activation %d", ep->act);
  DMM_CHECK_ARG(ep->post_act == 0 || ep->post_act == 1, "dmm_gemm_bf16_tn: unknown post activation %d", ep->post_act);
  DMM_CHECK_ARG((!ep->post_bias && !ep->post_act) || ep->out_hi, "dmm_gemm_bf16_tn: the post stage applies to out_hi/out_lo");
  DMM_CHECK_ARG(al16(ep->post_bias), "dmm_gemm_bf16_tn: post_bias must be 16-byte aligned");
  DMM_CHECK_ARG(!ep->cmax || ep->ld_cmax >= dmm_ceil_div(N, 32), "dmm_gemm_bf16_tn: ld_cmax must be >= ceil(N / 32)");

  const uint32_t flags = (a_lo ? DMM_GEMM_A_LO : 0) | (b_lo ? DMM_GEMM_B_LO : 0) | (ep->residual ? DMM_GEMM_RESIDUAL : 0) |
                         (ep->res_hi ? DMM_GEMM_RES_HI : 0) | (ep->res_lo ? DMM_GEMM_RES_LO : 0) |
                         (ep->out_f32 ? DMM_GEMM_OUT_F32 : 0) | (ep->out_hi ? DMM_GEMM_OUT_HI : 0) |
                         (ep->out_lo ? DMM_GEMM_OUT_LO : 0) | (splitk ? DMM_GEMM_SPLITK : 0);
  dmm_gemm_launch_plan pl;
  int rc = plan_gemm(ctx->num_sms, M, N, K, flags, &pl);
  if (rc) return rc;
  DMM_CHECK_ARG(pl.ksplit == 1 || (ep->out_f32 && !ep->out_hi && !ep->residual && !ep->bias && !ep->cmax && ep->act == 0),
                "dmm_gemm_bf16_tn: split-K writes plain fp32 partial products");

  GemmParams p;
  p.M = (int)M;
  p.N = (int)N;
  p.K = (int)K;
  p.num_m_blocks = (int)dmm_ceil_div(M, BLOCK_M);
  p.num_k_blocks = (int)dmm_ceil_div(K, BLOCK_K);
  p.ksplit = pl.ksplit;
  p.kb_per = (int)dmm_ceil_div(p.num_k_blocks, p.ksplit);
  p.ks_rows = ks_rows;
  p.n_pass = 0;
  // small correction passes first, the dominant hi.hi product last
  if (a_lo) { p.pass_a[p.n_pass] = 1; p.pass_b[p.n_pass] = 0; ++p.n_pass; }
  if (b_lo) { p.pass_a[p.n_pass] = 0; p.pass_b[p.n_pass] = 1; ++p.n_pass; }
  p.pass_a[p.n_pass] = 0; p.pass_b[p.n_pass] = 0; ++p.n_pass;
  for (int i = p.n_pass; i < 3; ++i) p.pass_a[i] = p.pass_b[i] = 0;
  p.ep = *ep;

  cudaStream_t st = (cudaStream_t)stream;
  switch (pl.bn) {
    case 64: return launch<64, false>(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, p, pl, st);
    case 128: return launch<128, false>(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, p, pl, st);
    default:
      return pl.ctas == 2 ? launch<256, true>(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, p, pl, st)
                          : launch<256, false>(ctx, a_hi, a_lo, lda, b_hi, b_lo, ldb, p, pl, st);
  }
}
}  // namespace

extern "C" int dmm_gemm_plan(int num_sms, int64_t M, int64_t N, int64_t K, uint32_t flags, dmm_gemm_launch_plan* plan) {
  DMM_CHECK_ARG(plan && num_sms > 0, "dmm_gemm_plan: null plan or num_sms < 1");
  DMM_CHECK_ARG(M > 0 && N > 0 && K > 0 && M < (1LL << 31) && N < (1LL << 31) && K < (1LL << 31), "dmm_gemm_plan: bad shape");
  DMM_CHECK_ARG((flags & ~0x1FFu) == 0, "dmm_gemm_plan: unknown flag bits 0x%x", flags);
  return plan_gemm(num_sms, M, N, K, flags, plan);
}
