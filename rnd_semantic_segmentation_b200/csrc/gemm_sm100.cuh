// Hand-written sm_100a GEMM core used by the fused ASPP head (fwd / dgrad / wgrad).
//
//   D[M x N] (fp32) = A[M x K] * B[N x K]^T     bf16 operands, fp32 accumulate in TMEM
//
// * operands staged by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) into a 4-stage
//   shared-memory ring guarded by mbarriers;
// * tcgen05.mma.cta_group::1.kind::f16, 128 x 256 x 16 per instruction, issued by one thread;
// * two 256-column fp32 accumulators in TMEM (512 columns) so the epilogue of tile i overlaps
//   the main loop of tile i+1; persistent CTAs, one per SM;
// * either operand may be K-major ([rows][K], K contiguous) or MN-major ([K][rows], rows
//   contiguous) -- the weight-gradient GEMM contracts over pixels and reads both operands
//   MN-major straight out of the layouts the forward pass already produced;
// * epilogue: tcgen05.ld -> registers -> padded smem transpose -> 128-byte coalesced stores,
//   with an optional "column = pixel index split by image" address map so the data-gradient
//   GEMM writes fp32 NCHW directly; optional split-K writes one partial slab per split.
#pragma once
#include <cuda.h>
#include "common.cuh"
#include "host_api.h"

namespace b200seg {
namespace gemm {

constexpr int BLOCK_M = 128;
constexpr int BLOCK_N = 256;
constexpr int BLOCK_K = 64;          // 64 bf16 = one 128-byte swizzle row
constexpr int UMMA_K = 16;
constexpr int STAGES = 4;
constexpr int A_BYTES = BLOCK_M * BLOCK_K * 2;   // 16 KB
constexpr int B_BYTES = BLOCK_N * BLOCK_K * 2;   // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;   // 48 KB
constexpr int MN_BOX_BYTES = 64 * BLOCK_K * 2;   // one MN-major TMA box: 64 k-rows x 128 B = 8 KB
constexpr int NUM_THREADS = 384;                 // warp0 TMA, warp1 MMA, warp2 TMEM alloc, warps 4-11 epilogue
constexpr int EPI_WARPS = 8;                     // two per TMEM lane quarter, each owning 128 accumulator columns
constexpr int EPI_PITCH = 20;                    // floats; 32 rows x 16 cols transpose tile, 16-byte aligned rows
constexpr int EPI_STAGE_FLOATS = 1024;           // per epilogue warp: the padded transpose tile (640 floats), or two dense
                                                 // 32 x 16 fp32 boxes (2 x 2 KB, 64-byte swizzle) for the TMA-store epilogue
constexpr int TMEM_COLS = 512;
constexpr int SMEM_BYTES = 1024 /*align slack*/ + STAGES * STAGE_BYTES + EPI_WARPS * EPI_STAGE_FLOATS * 4 + 256;

struct Params {
  int M, N, K;
  int m_tiles, n_tiles, splits, kb_per_split, kb_total;
  float* out;
  long long row_stride;     // elements between consecutive rows of D
  int col_hw;               // columns per image (INT_MAX => plain row-major)
  long long img_stride;     // elements between images (used when col_hw != INT_MAX)
  long long split_stride;   // elements between split-K partial slabs
  int vec_ok;               // output addressing allows 16-byte vector stores
  int out_bf16;             // D is written as bf16 (plain row-major [M][row_stride], 16-byte aligned rows) instead of fp32
  int n_fastest;            // tile order: consecutive work units walk along N (rows of D are written as long sequential runs)
  int row_hw_px;            // pixels per image for the row_hw mode
  int epi_sleep_ns;         // row_hw mode: pause after each 16-column chunk's stores (paces the epilogue's store bursts)
  int row_hw;               // > 0: ROWS of D are pixels of images with row_hw pixels each and D is fp32 NCHW: element (m, n)
                            // lives at out[(m / row_hw) * img_stride + n * row_hw + m % row_hw]; stored straight from registers
                            // (lane = pixel: a warp-level store is 32 consecutive pixels of one channel plane)
  // seam epilogue (SEAM kernels only): D[m, n] = bf16_rn(relu((acc * scale[n] + bias[n]) + identity[m, n])), identity fp32 NCHW
  // addressed as the row_hw map (row_hw_px pixels per image, img_stride elements between images), D bf16 row-major (out_bf16)
  const float* seam_identity;
  const float* seam_scale;
  const float* seam_bias;
  // statistics epilogue (gemm_bf16_stats_kernel only): for every 32-pixel TMEM lane group gi = m / 32 and column n < N,
  // stats[gi * N + n] = (mean, M2) of the fp32 D values the register-store epilogue writes for those pixels
  float2* stats;
};

// ------------------------------------------------------------------------------------------
// PTX wrappers
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n .reg .pred p;\n mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n selp.u32 %0, 1, 0, p;\n}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (kernel error) instead of hanging the GPU box.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const long long t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if (clock64() - t0 > 8000000000LL) __trap();
  }
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same with tf32 operands (fp32 in shared memory, the tensor core reads the top 19 bits): K = 8 per instruction
__device__ __forceinline__ void umma_tf32(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
// TMA bulk store of a {16 cols, 32 rows, 1 image} fp32 box from shared memory (3-D map: column-in-image, row, image)
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// Shared-memory matrix descriptor (sm_100 format): start>>4 [0,14), LBO>>4 [16,30),
// SBO>>4 [32,46), version=1 [46,48), layout type [61,64) (2 = SWIZZLE_128B; 1 = SWIZZLE_128B_BASE32B, 32-byte chunks swizzled
// over 4-row atoms: the only swizzled layout of MN-major 32-bit (tf32) operands).
constexpr uint32_t SMEM_SW128 = 2, SMEM_SW128_BASE32B = 1;
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes, uint32_t layout = SMEM_SW128) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)layout << 61;
  return d;
}
// Instruction descriptor: D=f32 [4,6)=1, A format [7,10), B format [10,13) (IDESC_BF16 = 1 for kind::f16, IDESC_TF32 = 2 for
// kind::tf32), a_major bit 15, b_major bit 16 (1 = MN-major), N>>3 [17,23), M>>4 [24,29).
constexpr uint32_t IDESC_BF16 = 1, IDESC_TF32 = 2;
__host__ __device__ constexpr uint32_t make_idesc(bool a_mn, bool b_mn, int m, int n, uint32_t fmt = IDESC_BF16) {
  return (1u << 4) | (fmt << 7) | (fmt << 10) | ((a_mn ? 1u : 0u) << 15) | ((b_mn ? 1u : 0u) << 16) |
         ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ------------------------------------------------------------------------------------------
// The kernel
// ------------------------------------------------------------------------------------------
// Operand sharing inside a 2-CTA cluster (the kernel is bound by SM<->L2 bandwidth, 48 KB per k-block per SM):
//   SHARE_NONE : plain launch, every CTA loads its whole A and B tiles.
//   SHARE_B    : the two CTAs of a cluster own M-tiles (2i, 2i+1) of the SAME N-tile; each loads its own A tile and
//                HALF of the shared B tile and multicasts that half into both CTAs' shared memory (32 KB per k-block).
//   SHARE_A    : the two CTAs own N-tiles (2i, 2i+1) of the SAME M-tile; each loads its own B tile and half of A (40 KB).
// Each CTA still issues its own cta_group::1 MMAs into its own TMEM.  A shared-memory stage is released to BOTH
// producers only when BOTH CTAs' MMAs have drained it (empty barriers count 2, tcgen05.commit multicast to both CTAs).
//   SHARE_PAIR : the two CTAs own M-tiles (2i, 2i+1) of the same N-tile and drive ONE tcgen05.mma.cta_group::2 (M = 256):
//                each stages its own A tile and HALF of the B tile (the tensor core reads the other half from the peer's
//                shared memory): 32 KB per k-block per SM, half the B operand reads per MMA, 6 stages instead of 4.  The
//                leader CTA issues; both CTAs' TMA bytes complete on the leader's full barrier; commits are multicast.
constexpr int SHARE_NONE = 0, SHARE_B = 1, SHARE_A = 2, SHARE_PAIR = 4;
constexpr int PAIR_STAGES = 6;
constexpr int PAIR_STAGE_BYTES = A_BYTES + B_BYTES / 2;          // 32 KB; 6 x 32 KB = 4 x 48 KB

__device__ __forceinline__ uint32_t mapa_u32(uint32_t addr, uint32_t rank) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(addr), "r"(rank));
  return r;
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// "accumulator drained" arrives of the epilogue warps.  RELAXED on purpose: what they order -- the tcgen05.ld reads of the
// accumulator before the next tcgen05.mma into it -- is already guaranteed by tcgen05.wait::ld + tcgen05.fence::before_thread_sync.
// A release arrive additionally waits (MEMBAR + ERRBAR in SASS) until every global store the warp has in flight is performed,
// i.e. it puts the drain of the epilogue's stores on the MMA's critical path once per tile (ncu: 11 % of the dgrad GEMM's warp
// samples sat on exactly that; profiles/README.md round-2 table).
__device__ __forceinline__ void mbar_arrive_relaxed(uint64_t* bar) {
  asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint32_t cluster_addr) {
  asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(cluster_addr) : "memory");
}
// 2-SM TMA load: the completion barrier is a shared::cluster address and may live in the peer (leader) CTA
__device__ __forceinline__ void tma_load_2d_2sm(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar_cluster, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_dst), "l"(m), "r"(bar_cluster), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tmem_alloc_2sm(uint32_t* dst_smem, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "r"(ncols) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_2sm(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_tf32_2sm(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n .reg .pred p;\n setp.ne.b32 p, %4, 0;\n tcgen05.mma.cta_group::2.kind::tf32 [%0], %1, %2, %3, p;\n}" ::"r"(tmem_d),
      "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}

__device__ __forceinline__ void tma_load_2d_mc(uint32_t smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1,
                                               uint16_t cta_mask) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster [%0], [%1, {%4, %5}], [%2], %3;"
      ::"r"(smem_dst), "l"(m), "r"(smem_u32(bar)), "h"(cta_mask), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t cta_mask) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
               "h"(cta_mask)
               : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_cta_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}

// work unit -> (split z, M-tile, N-tile) of this CTA
template <int SHARE>
struct TileSched {
  int units, worker, nworkers, rank, m_tiles, n_tiles, per_split, n_fastest;
  __device__ TileSched(const Params& p) {
    n_fastest = p.n_fastest;
    constexpr int CS = SHARE == SHARE_NONE ? 1 : 2;      // CTAs per cluster
    rank = SHARE != SHARE_NONE ? (int)cluster_cta_rank() : 0;
    worker = (int)blockIdx.x / CS;
    nworkers = (int)gridDim.x / CS;
    m_tiles = (SHARE == SHARE_B || SHARE == SHARE_PAIR) ? (p.m_tiles + 1) >> 1 : p.m_tiles;     // pairs along M
    n_tiles = SHARE == SHARE_A ? (p.n_tiles + 1) >> 1 : p.n_tiles;     // pairs along N
    per_split = m_tiles * n_tiles;
    units = per_split * p.splits;
  }
  __device__ void decode(int unit, int& z, int& mt, int& nt) const {
    z = unit / per_split;
    const int rem = unit - z * per_split;
    if (n_fastest) {
      mt = rem / n_tiles;                // N fastest: the CTAs running together write neighbouring column ranges of the same rows
      nt = rem - mt * n_tiles;
    } else {
      nt = rem / m_tiles;                // M fastest: tiles sharing the (large) B operand are adjacent in time
      mt = rem - nt * m_tiles;
    }
    if (SHARE == SHARE_B || SHARE == SHARE_PAIR) mt = mt * 2 + rank;
    if (SHARE == SHARE_A) nt = nt * 2 + rank;
  }
};

// Sum over the warp's 32 lanes of each of 16 values, by halving exchanges (8 + 4 + 2 + 1 + 1 shuffles, not 16 x 5): lane l
// returns the total of value l / 2 (lanes 2j and 2j + 1 get the same bits).  v is consumed.  A fixed order: deterministic.
__device__ __forceinline__ float warp_sum_scatter16(float (&v)[16], int lane) {
#pragma unroll
  for (int st = 0; st < 4; ++st) {
    const int w = 8 >> st, o = 16 >> st;
    const bool hi = (lane & o) != 0;
#pragma unroll
    for (int i = 0; i < w; ++i) {
      const float keep = hi ? v[i + w] : v[i], send = hi ? v[i] : v[i + w];
      v[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
    }
  }
  return v[0] + __shfl_xor_sync(0xffffffffu, v[0], 1);
}

// BN = accumulator columns per tile (256 by default).  A narrower tile (224 / 192) is picked by the host when it makes the
// tile count a near-multiple of the SM count: 5 M-tiles x 128 N-tiles of 256 on 148 SMs are 4.3 waves = 5 rounds; the same
// problem in 224-column tiles is 5 x 147 = 4.97 waves = 5 rounds of 12.5 % less work each.  K-major operands, fp32 output,
// SHARE_NONE / SHARE_A only.
// RS ("register stores"): the fp32 NCHW pixel-major epilogue only (Params::row_hw), which needs no shared-memory staging -- the
// 32 KB go to a seventh ring stage instead (PAIR mode): the operand loads of this store-heavy problem see their latency inflated
// by the epilogue's store bursts, and bytes in flight are what hides it.
// SEAM: the bf16 row-major epilogue with the backbone tail applied to the accumulator first (Params::seam_*): M = pixels, so a
// TMEM lane is a pixel and each identity column load is 32 consecutive pixels of one fp32 NCHW plane.  K-major operands only.
// STATS (gemm_bf16_stats_kernel): the RS epilogue also writes each lane group's per-column (mean, M2) (Params::stats).
template <bool A_MN, bool B_MN, int SHARE, int BN, bool RS, bool SEAM, bool STATS>
__device__ __forceinline__ void gemm_bf16_body(const CUtensorMap& tmap_a, const CUtensorMap& tmap_b, const CUtensorMap& tmap_out,
                                               const Params& p) {
  __builtin_assume(threadIdx.x < NUM_THREADS);      // what __launch_bounds__ tells the compiler in the kernel itself
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;                                   // 1024-byte aligned (128B swizzle atom)
  constexpr bool PAIR = SHARE == SHARE_PAIR;
  static_assert(BN == 256 || (!A_MN && !B_MN && (SHARE == SHARE_NONE || SHARE == SHARE_A)), "narrow tiles: K-major, unshared B only");
  static_assert(BN % 32 == 0 && BN <= 256, "epilogue halves are BN / 2 columns in chunks of 16");
  constexpr int BLOCK_N = BN;                                       // shadows gemm::BLOCK_N below
  constexpr int B_BYTES = BN * BLOCK_K * 2;
  static_assert(!RS || (PAIR && BN == 256), "register-store variant: cta_group::2 pairs only");
  static_assert(!SEAM || (!RS && !A_MN && !B_MN && BN == 256), "seam epilogue: K-major operands, 256-column tiles");
  static_assert(!STATS || (RS && !SEAM && !A_MN && !B_MN), "statistics epilogue: the register-store variant, K-major operands");
  constexpr int STAGES = PAIR ? (RS ? PAIR_STAGES + 1 : PAIR_STAGES) : gemm::STAGES;         // same total bytes either way
  constexpr int STAGE_BYTES = PAIR ? PAIR_STAGE_BYTES : gemm::STAGE_BYTES;     // ring stride (a narrow B tile leaves its tail unused)
  constexpr int STAGE_TX = PAIR ? PAIR_STAGE_BYTES : A_BYTES + B_BYTES;        // bytes that land in a stage per k-block
  static_assert(PAIR_STAGES * PAIR_STAGE_BYTES == gemm::STAGES * gemm::STAGE_BYTES, "epilogue staging / barriers sit behind the ring");
  static_assert(!RS || PAIR_STAGE_BYTES == EPI_WARPS * EPI_STAGE_FLOATS * 4, "the extra stage takes exactly the staging area");
  float* epi_stage = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);                   // (RS: not used)
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + (RS ? 0 : EPI_WARPS * EPI_STAGE_FLOATS * 4));
  uint64_t* full_bar = bars;                  // [STAGES]
  uint64_t* empty_bar = bars + STAGES;        // [STAGES]
  uint64_t* tfull_bar = bars + 2 * STAGES;    // [2]
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;  // [2]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr bool CLUSTER = SHARE != SHARE_NONE;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], PAIR ? 1 : (CLUSTER ? 2 : 1));   // multicast modes: both CTAs of the pair release the stage
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], PAIR ? 2 * EPI_WARPS : EPI_WARPS);   // one arrive per epilogue warp (PAIR: of both CTAs, on the leader)
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    if (PAIR) tmem_alloc_2sm(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  if (CLUSTER) cluster_sync_all();            // peer barriers are initialised before any remote arrive / multicast
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  const TileSched<SHARE> sched(p);

  if (warp == 0) {
    // ================= TMA producer (one thread) =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = sched.worker; unit < sched.units; unit += sched.nworkers) {
        int z, mt, nt;
        sched.decode(unit, z, mt, nt);
        const int m0 = mt * BLOCK_M, n0 = nt * BLOCK_N;
        const int kb0 = z * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
          const int k0 = kb * BLOCK_K;
          if (PAIR) {
            // own A tile + own half of B; both CTAs' bytes complete on the leader's full barrier
            // RS variant, last N-tile with <= 128 columns left: the MMA runs with N = 128 (half the cycles), of which each CTA
            // supplies 64 rows of B, fetched through a 64-row box (the tensor map in the otherwise unused tmap_out slot)
            const bool narrow = RS && !B_MN && (p.N - n0) <= BLOCK_N / 2;
            if (sched.rank == 0) mbar_arrive_expect_tx(&full_bar[stage], narrow ? 2 * (A_BYTES + B_BYTES / 4) : 2 * STAGE_TX);
            const uint32_t fb = mapa_u32(smem_u32(&full_bar[stage]), 0);
            if (!A_MN) tma_load_2d_2sm(sa, &tmap_a, fb, k0, m0);
            else {
#pragma unroll
              for (int b = 0; b < BLOCK_M / 64; ++b) tma_load_2d_2sm(sa + b * MN_BOX_BYTES, &tmap_a, fb, m0 + b * 64, k0);
            }
            const int nh = n0 + sched.rank * (narrow ? BLOCK_N / 4 : BLOCK_N / 2);
            if (narrow) tma_load_2d_2sm(sb, &tmap_out, fb, k0, nh);
            else if (!B_MN) tma_load_2d_2sm(sb, &tmap_b, fb, k0, nh);
            else {
#pragma unroll
              for (int b = 0; b < BLOCK_N / 2 / 64; ++b) tma_load_2d_2sm(sb + b * MN_BOX_BYTES, &tmap_b, fb, nh + b * 64, k0);
            }
            if (++stage == STAGES) { stage = 0; phase ^= 1u; }
            continue;
          }
          mbar_arrive_expect_tx(&full_bar[stage], STAGE_TX);      // own loads + the peer's multicast half
          // ---- A ----
          if (SHARE == SHARE_A) {
            // shared A tile: this CTA loads rows [64*ha, +64) and multicasts them to both CTAs of the pair
            const int ha = sched.rank;
            if (!A_MN) tma_load_2d_mc(sa + ha * (A_BYTES / 2), &tmap_a, &full_bar[stage], k0, m0 + ha * 64, 0x3);
            else tma_load_2d_mc(sa + ha * MN_BOX_BYTES, &tmap_a, &full_bar[stage], m0 + ha * 64, k0, 0x3);
          } else if (!A_MN) {
            tma_load_2d(sa, &tmap_a, &full_bar[stage], k0, m0);            // box {64 k, 128 rows}
          } else {
#pragma unroll
            for (int b = 0; b < BLOCK_M / 64; ++b)                          // box {64 m, 64 k}
              tma_load_2d(sa + b * MN_BOX_BYTES, &tmap_a, &full_bar[stage], m0 + b * 64, k0);
          }
          // ---- B ----
          if (SHARE == SHARE_B) {
            // shared B tile: this CTA loads rows [128*hb, +128) and multicasts them to both CTAs of the pair
            const int hb = sched.rank;
            if (!B_MN) {
              tma_load_2d_mc(sb + hb * (B_BYTES / 2), &tmap_b, &full_bar[stage], k0, n0 + hb * 128, 0x3);
            } else {
#pragma unroll
              for (int b = 0; b < 2; ++b)
                tma_load_2d_mc(sb + (hb * 2 + b) * MN_BOX_BYTES, &tmap_b, &full_bar[stage], n0 + (hb * 2 + b) * 64, k0, 0x3);
            }
          } else if (!B_MN) {
            tma_load_2d(sb, &tmap_b, &full_bar[stage], k0, n0);            // box {64 k, 256 rows}
          } else {
#pragma unroll
            for (int b = 0; b < BLOCK_N / 64; ++b)
              tma_load_2d(sb + b * MN_BOX_BYTES, &tmap_b, &full_bar[stage], n0 + b * 64, k0);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (one thread) =================
    if (lane == 0 && (!PAIR || sched.rank == 0)) {
      constexpr uint32_t idesc = make_idesc(A_MN, B_MN, PAIR ? 2 * BLOCK_M : BLOCK_M, BLOCK_N);
      constexpr uint32_t idesc_narrow = make_idesc(A_MN, B_MN, PAIR ? 2 * BLOCK_M : BLOCK_M, BLOCK_N / 2);   // RS: ragged last N-tile
      // K-major: 8-row groups 1024 B apart (SBO), LBO unused (1); +32 B per UMMA_K step.
      // MN-major: 64-element chunks one TMA box (8 KB) apart (LBO), 8-k-row groups 1024 B apart (SBO);
      //           +16 k-rows = 2048 B per UMMA_K step.
      constexpr uint32_t a_lbo = A_MN ? MN_BOX_BYTES : 16, a_sbo = 1024, a_step = A_MN ? 2048 : 32;
      constexpr uint32_t b_lbo = B_MN ? MN_BOX_BYTES : 16, b_sbo = 1024, b_step = B_MN ? 2048 : 32;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int unit = sched.worker; unit < sched.units; unit += sched.nworkers) {
        int z, mt, nt;
        sched.decode(unit, z, mt, nt);
        const int kb0 = z * p.kb_per_split;
        const int kb1 = min(p.kb_total, kb0 + p.kb_per_split);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * gemm::BLOCK_N);      // accumulators 256 columns apart for every BN
        for (int kb = kb0; kb < kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t adesc = make_smem_desc(sa + k * a_step, a_lbo, a_sbo);
            const uint64_t bdesc = make_smem_desc(sb + k * b_step, b_lbo, b_sbo);
            if (PAIR) umma_bf16_2sm(tmem_d, adesc, bdesc, (RS && !B_MN && (p.N - nt * BLOCK_N) <= BLOCK_N / 2) ? idesc_narrow : idesc,
                                    (kb > kb0 || k > 0) ? 1u : 0u);
            else umma_bf16(tmem_d, adesc, bdesc, idesc, (kb > kb0 || k > 0) ? 1u : 0u);
          }
          // frees the slot in every CTA that multicasts into this one (itself included) when these MMAs retire
          if (PAIR) umma_commit_2sm(&empty_bar[stage], 0x3);
          else if (CLUSTER) umma_commit_mc(&empty_bar[stage], 0x3);
          else umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (PAIR) umma_commit_2sm(&tfull_bar[acc], 0x3);
        else umma_commit(&tfull_bar[acc]);         // accumulator ready for the epilogue
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue (8 warps; warp w owns TMEM lanes [32*(w%4), +32) and columns [128*((w-4)/4), +128)) ====
    const int wq = warp & 3;
    const int half = (warp - 4) >> 2;
    float* stg = epi_stage + (warp - 4) * EPI_STAGE_FLOATS;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = sched.worker; unit < sched.units; unit += sched.nworkers) {
      int z, mt, nt;
      sched.decode(unit, z, mt, nt);
      const int row_base = mt * BLOCK_M + wq * 32;
      const int col_base = nt * BLOCK_N + half * (BLOCK_N / 2);
      float* out = p.out + (long long)z * p.split_stride;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(acc * gemm::BLOCK_N + half * (BLOCK_N / 2));
      const int rows = min(32, p.M - row_base);
      if (SEAM || (!RS && p.out_bf16)) {
        // bf16 row-major D (the NHWC feature gradient): 32 columns per pass, converted before the smem transpose, every
        // store instruction writes 8 rows x 64 contiguous bytes
        if (rows > 0 && col_base < p.N) {
          __nv_bfloat16* outb = reinterpret_cast<__nv_bfloat16*>(p.out) + (long long)z * p.split_stride;
          uint32_t* stw = reinterpret_cast<uint32_t*>(stg);
          const float* idp = nullptr;                  // SEAM: this lane's pixel in channel plane 0 of its image
          if (SEAM) {
            const int m = lane < rows ? row_base + lane : row_base;
            const int img = m / p.row_hw_px;
            idp = p.seam_identity + (long long)img * p.img_stride + (m - img * p.row_hw_px);
          }
#pragma unroll 1
          for (int c = 0; c < BLOCK_N / 2 / 32; ++c) {
            uint32_t r[32];
            tmem_ld16(taddr + (uint32_t)(c * 32), r);
            tmem_ld16(taddr + (uint32_t)(c * 32 + 16), r + 16);
            if (SEAM) {
              // the 32 identity loads are in flight with the TMEM loads; the tail in the stock order (mul, add, add, relu)
              const int cb = col_base + c * 32;
              float id[32];
#pragma unroll
              for (int k = 0; k < 32; ++k)
                id[k] = (lane < rows && cb + k < p.N) ? __ldcs(idp + (long long)(cb + k) * p.row_hw_px) : 0.f;
              tmem_ld_wait();
#pragma unroll
              for (int k = 0; k < 32; ++k) {
                const int n = min(cb + k, p.N - 1);
                const float v = __fadd_rn(__fadd_rn(__fmul_rn(__uint_as_float(r[k]), __ldg(p.seam_scale + n)), __ldg(p.seam_bias + n)), id[k]);
                r[k] = __float_as_uint(v <= 0.f ? 0.f : v);      // NaN passes through, as torch.relu
              }
            } else {
              tmem_ld_wait();
            }
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              uint32_t w4[4];
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const __nv_bfloat162 v = __floats2bfloat162_rn(__uint_as_float(r[8 * k + 2 * e]), __uint_as_float(r[8 * k + 2 * e + 1]));
                w4[e] = *reinterpret_cast<const uint32_t*>(&v);
              }
              *reinterpret_cast<uint4*>(stw + lane * EPI_PITCH + 4 * k) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
            }
            __syncwarp();
            const int col0 = col_base + c * 32 + (lane & 3) * 8;
            if (col0 < p.N) {                                  // N and row_stride are multiples of 8 on this path
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int rr = (lane >> 2) + 8 * i;
                if (rr < rows)
                  *reinterpret_cast<uint4*>(outb + (long long)(row_base + rr) * p.row_stride + col0) =
                      *reinterpret_cast<const uint4*>(stw + rr * EPI_PITCH + (lane & 3) * 4);
              }
            }
            __syncwarp();
          }
        }
      } else if (RS || p.row_hw > 0) {
        // fp32 NCHW D with the pixels along M: a TMEM lane is a pixel and a register column is a channel, so the 32 lanes of a
        // store instruction write 32 consecutive pixels of ONE channel plane = 128 contiguous bytes, straight from the registers
        // tcgen05.ld filled.  No shared-memory transpose (its STS + LDS traffic through L1 was what held the channel-major form
        // of this epilogue back: L1/TEX 76 % busy) and no dependence on the plane pitch being a multiple of 4 pixels.
        if (rows > 0 && col_base < p.N) {
          const int hw = p.row_hw_px;
          const bool ok = lane < rows;
          const int m = ok ? row_base + lane : row_base;
          const int img = m / hw;
          float* dst = out + (long long)img * p.img_stride + (m - img * hw) + (long long)col_base * hw;
          constexpr int NCH = BLOCK_N / 2 / 16;
          uint32_t rbuf[2][16];
          tmem_ld16(taddr, rbuf[0]);
#pragma unroll
          for (int c = 0; c < NCH; ++c) {
            tmem_ld_wait();
            const uint32_t* r = rbuf[c & 1];
            if (c + 1 < NCH) tmem_ld16(taddr + (uint32_t)((c + 1) * 16), rbuf[(c + 1) & 1]);
            const int ncols = p.N - (col_base + c * 16);
            if (ok) {
              float* d = dst + (long long)(c * 16) * hw;
              // (Code-generation note: with this two-way branch nvcc 12.9 keeps both TMEM register sets live -- 80 registers,
              //  147 us at the bench shape.  The same loop without the branch compiled to 71 registers and ran 248 us: check
              //  `cuobjdump --dump-resource-usage` and profiles/dgrad_modes.py after touching this block.)
              if (p.row_hw == 2) {                      // streaming (evict-first) stores: measured no better, kept as dgrad mode 2
#pragma unroll
                for (int k = 0; k < 16; ++k)
                  if (k < ncols) __stcs(d + (long long)k * hw, __uint_as_float(r[k]));
              } else {
#pragma unroll
                for (int k = 0; k < 16; ++k)
                  if (k < ncols) d[(long long)k * hw] = __uint_as_float(r[k]);
              }
            }
            if (STATS && ncols > 0) {
              // the chunk's 16 channels over this warp's `rows` pixels, corrected two-pass (no shift is available here to keep
              // |mean| >> sigma accurate): the group mean m, then M2 = sum (v - m)^2 - (sum (v - m))^2 / n about m + sum (v - m) / n;
              // lanes past the last pixel contribute nothing
              const float cnt = (float)rows;
              float v[16], sq[16];
#pragma unroll
              for (int k = 0; k < 16; ++k) v[k] = ok ? __uint_as_float(r[k]) : 0.f;
#pragma unroll
              for (int k = 0; k < 16; ++k) sq[k] = v[k];
              const float mean = warp_sum_scatter16(sq, lane) / cnt;            // of channel lane / 2
#pragma unroll
              for (int k = 0; k < 16; ++k) {
                const float mk = __shfl_sync(0xffffffffu, mean, 2 * k);
                v[k] = ok ? v[k] - mk : 0.f;
                sq[k] = v[k] * v[k];
              }
              const float sd = warp_sum_scatter16(v, lane);
              const float m2 = warp_sum_scatter16(sq, lane) - sd * sd / cnt;
              const int j = lane >> 1;
              if ((lane & 1) == 0 && j < ncols)                              // (the mean the corrected M2 is taken about)
                p.stats[(long long)(row_base >> 5) * p.N + col_base + c * 16 + j] = make_float2(mean + sd / cnt, m2);
            }
            if (p.epi_sleep_ns > 0) __nanosleep((unsigned)p.epi_sleep_ns);
          }
        }
      } else if (rows > 0 && col_base < p.N) {
        // per-lane (image, offset) of its first column, advanced by 16 columns per chunk (no division in the loop)
        const int lane_col = p.vec_ok ? (lane & 3) * 4 : (lane & 15);
        int img = (col_base + lane_col) / p.col_hw;
        int rem = (col_base + lane_col) - img * p.col_hw;
        // software pipeline: the TMEM load of chunk c + 1 is in flight while chunk c goes through the smem transpose and
        // out to global memory (two register sets, loop fully unrolled so both are statically indexed)
        constexpr int NCH = BLOCK_N / 2 / 16;
        uint32_t rbuf[2][16];
        tmem_ld16(taddr, rbuf[0]);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          tmem_ld_wait();
          const uint32_t* r = rbuf[c & 1];
          if (c + 1 < NCH) tmem_ld16(taddr + (uint32_t)((c + 1) * 16), rbuf[(c + 1) & 1]);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<float4*>(stg + lane * EPI_PITCH + 4 * k) =
                make_float4(__uint_as_float(r[4 * k]), __uint_as_float(r[4 * k + 1]), __uint_as_float(r[4 * k + 2]),
                            __uint_as_float(r[4 * k + 3]));
          __syncwarp();
          const int col0 = col_base + c * 16;
          float* dst = out + (long long)img * p.img_stride + rem + (long long)row_base * p.row_stride;
          if (p.vec_ok) {
            // lane -> (row lane/4 + 8i, 4 columns): every store instruction writes 8 rows x 64 contiguous bytes
            if (col0 + lane_col + 3 < p.N) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int rr = (lane >> 2) + 8 * i;
                if (rr < rows)
                  *reinterpret_cast<float4*>(dst + (long long)rr * p.row_stride) =
                      *reinterpret_cast<const float4*>(stg + rr * EPI_PITCH + lane_col);
              }
            } else {
              for (int e = 0; e < 4; ++e)
                if (col0 + lane_col + e < p.N)
                  for (int i = 0; i < 4; ++i) {
                    const int rr = (lane >> 2) + 8 * i;
                    if (rr < rows) dst[(long long)rr * p.row_stride + e] = stg[rr * EPI_PITCH + lane_col + e];
                  }
            }
          } else if (col0 + lane_col < p.N) {
            // scalar path (unaligned rows): lane -> (row lane/16 + 2i, column lane%16)
            for (int rr = (lane >> 4); rr < rows; rr += 2) dst[(long long)rr * p.row_stride] = stg[rr * EPI_PITCH + lane_col];
          }
          rem += 16;
          while (rem >= p.col_hw) { rem -= p.col_hw; ++img; }
          __syncwarp();
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        if (PAIR) mbar_arrive_cluster_relaxed(mapa_u32(smem_u32(&tempty_bar[acc]), 0));
        else mbar_arrive_relaxed(&tempty_bar[acc]);
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (CLUSTER) cluster_sync_all();            // the peer may still multicast into / arrive on this CTA until it is done too
  if (warp == 2) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

template <bool A_MN, bool B_MN, int SHARE, int BN = 256, bool RS = false, bool SEAM = false>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_bf16_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                 const __grid_constant__ CUtensorMap tmap_out, const Params p) {
  gemm_bf16_body<A_MN, B_MN, SHARE, BN, RS, SEAM, false>(tmap_a, tmap_b, tmap_out, p);
}

// ------------------------------------------------------------------------------------------
// Forward GEMM of the ASPP head that reads the features as the reference hands them over -- fp32 NCHW -- and converts them to
// the bf16 MMA operand INSIDE the kernel (no separate fp32 -> bf16 pack pass, no packed copy read back):
//
//   D[M x P] (fp32, row-major) = A[M x K] (bf16 K-major, TMA) * X[K x P]     X = fp32 NCHW features, K = channel, P = n*hw + pixel
//
// A cluster of 2 * MP CTAs owns ONE 256-pixel tile and ALL MP pairs of 128-row M-tiles (MP = 3 for the 19-class head: 640 packed
// weight rows).  CTAs (2q, 2q+1) form pair q and drive one tcgen05.mma.cta_group::2 exactly as SHARE_PAIR above: each CTA stages
// its own A tile by TMA and holds HALF r = rank & 1 of the B tile.  The B halves are PRODUCED by converter warps, once per cluster:
// k-block kb of half r is converted by CTA (2 (kb % MP) + r) -- lane l of a warp loads 16 bytes = 4 consecutive pixels of one
// channel row (a warp instruction = 512 contiguous bytes of x), rounds to bf16 (RN, as the pack kernel does) and stores 8 bytes
// into the MN-major, 128-byte-swizzled operand box of EVERY CTA holding half r (its own shared memory and the peers' through
// distributed shared memory) -- the NCHW layout IS the MN-major layout, so no transposition is involved.  x therefore crosses
// L2 -> SM once per pixel tile (fp32 in, 10.7 KB per k-block per SM) instead of three times, and each converter has MP k-blocks of
// lead.  A stage's full barrier (on each pair's leader) counts the leader's TMA arrive + one arrive per half from the converting
// CTA's signaller warp (the converter threads fence their generic-proxy writes to the async proxy and meet the signaller at a
// named barrier; the signaller's arrive carries the cluster-scope release); a stage is released to the cluster only when all MP
// pairs have consumed it (empty barriers count MP, commits multicast to the whole cluster).
// Optionally the bf16 values are also written out as NCHW (`xn`) for the weight-gradient GEMM of the backward pass.
// ------------------------------------------------------------------------------------------
constexpr int CONV_WARPS = 8;
constexpr int FWDX_EPI_WARPS = 4;              // one per TMEM lane quarter, all 256 columns each (the epilogue hides behind a 32-k-block main loop)
constexpr int FWDX_THREADS = (4 + FWDX_EPI_WARPS + CONV_WARPS) * 32;   // 512: warps 0-3 control, 4-7 epilogue, 8-15 convert -> 128 registers per thread,
                                                                        // so the converters' 16 loads in flight per lane stay in registers
constexpr int FWDX_MAX_MP = 3;               // 2 * MP <= ring stages (see the converters); 3 M-pairs = 768 packed weight rows = 23 classes

struct FwdXParams {
  int M, P, K;                       // rows of A / D, pixels (columns of D), channels
  int m_tiles, n_tiles, kb_total;
  float* out;                        // D [M][row_stride] fp32
  long long row_stride;
  const float* x;                    // fp32 NCHW [N][K][hw]
  int hw;
  __nv_bfloat16* xn;                 // optional bf16 NCHW copy of x (null: not written)
};

__device__ __forceinline__ void st_cluster_v2(uint32_t cluster_addr, uint32_t a, uint32_t b) {
  asm volatile("st.shared::cluster.v2.u32 [%0], {%1, %2};" ::"r"(cluster_addr), "r"(a), "r"(b) : "memory");
}
__device__ __forceinline__ void fence_proxy_async_all() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

template <int MP>
__global__ void __launch_bounds__(FWDX_THREADS, 1)
gemm_fwd_convert_kernel(const __grid_constant__ CUtensorMap tmap_a, const FwdXParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  constexpr int STAGES = PAIR_STAGES;
  constexpr int STAGE_BYTES = PAIR_STAGE_BYTES;                     // 16 KB A + 16 KB B half
  constexpr int CS = 2 * MP;                                        // CTAs per cluster
  float* epi_stage = reinterpret_cast<float*>(smem + STAGES * STAGE_BYTES);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES + EPI_WARPS * EPI_STAGE_FLOATS * 4);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tfull_bar = bars + 2 * STAGES;
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  const int rank = (int)cluster_cta_rank();
  const int q = rank >> 1, r = rank & 1;                            // pair (= M-pair) and pixel half of this CTA
  const uint32_t leader = (uint32_t)(rank & ~1);

  if (warp == 0 && lane == 0) tma_prefetch_desc(&tmap_a);
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1 + 2);                               // leader's TMA arrive + the signaller of each half's converting CTA
      mbar_init(&empty_bar[s], MP);                                 // every pair of the cluster has consumed the stage
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], 2 * FWDX_EPI_WARPS);
    }
    fence_mbar_init();
  }
  if (warp == 2) tmem_alloc_2sm(tmem_slot, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  // work unit = one 256-pixel tile; cluster c takes tiles c, c + nclusters, ...
  const int units = p.n_tiles;
  const int worker = (int)blockIdx.x / CS, nworkers = (int)gridDim.x / CS;
  const int my_units = worker < units ? (units - worker + nworkers - 1) / nworkers : 0;

  if (warp == 0) {
    // ================= TMA producer: the A tile of this CTA =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      const int m0 = (q * 2 + r) * BLOCK_M;
      const uint32_t fb0 = mapa_u32(smem_u32(&full_bar[0]), leader);
      for (int u = 0; u < my_units; ++u) {
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          if (r == 0) mbar_arrive_expect_tx(&full_bar[stage], 2 * A_BYTES);
          tma_load_2d_2sm(smem_u32(smem + stage * STAGE_BYTES), &tmap_a, fb0 + (uint32_t)stage * 8u, kb * BLOCK_K, m0);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer (the pair's leader CTA, one thread) =================
    if (lane == 0 && r == 0) {
      constexpr uint32_t idesc = make_idesc(false, true, 2 * BLOCK_M, BLOCK_N);
      constexpr uint16_t all_mask = (uint16_t)((1u << CS) - 1u);
      const uint16_t pair_mask = (uint16_t)(0x3u << (2 * q));
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int u = 0; u < my_units; ++u) {
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = 0; kb < p.kb_total; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
#pragma unroll
          for (int k = 0; k < BLOCK_K / UMMA_K; ++k) {
            const uint64_t adesc = make_smem_desc(sa + k * 32, 16, 1024);                    // K-major A
            const uint64_t bdesc = make_smem_desc(sb + k * 2048, MN_BOX_BYTES, 1024);        // MN-major B (two 64-pixel boxes)
            umma_bf16_2sm(tmem_d, adesc, bdesc, idesc, (kb > 0 || k > 0) ? 1u : 0u);
          }
          umma_commit_2sm(&empty_bar[stage], all_mask);             // this pair is done with the stage, in every CTA of the cluster
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        umma_commit_2sm(&tfull_bar[acc], pair_mask);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4 && warp < 4 + FWDX_EPI_WARPS) {
    // ================= epilogue: fp32 row-major D, 16-byte coalesced stores (as gemm_bf16_kernel's plain path) =================
    const int wq = warp & 3;
    float* stg = epi_stage + (warp - 4) * EPI_STAGE_FLOATS;
    const bool vec_ok = (p.row_stride % 4 == 0) && ((reinterpret_cast<uintptr_t>(p.out) & 15) == 0);
    const uint32_t te0 = mapa_u32(smem_u32(&tempty_bar[0]), leader);
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int u = 0; u < my_units; ++u) {
      const int nt = worker + u * nworkers;
      const int row_base = (q * 2 + r) * BLOCK_M + wq * 32;
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const int rows = min(32, p.M - row_base);
#pragma unroll 1
      for (int half = 0; half < 2; ++half) {
      const int col_base = nt * BLOCK_N + half * (BLOCK_N / 2);
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(acc * BLOCK_N + half * (BLOCK_N / 2));
      if (rows > 0 && col_base < p.P) {
        constexpr int NCH = BLOCK_N / 2 / 16;
        const int lane_col = vec_ok ? (lane & 3) * 4 : (lane & 15);
        uint32_t rbuf[2][16];
        tmem_ld16(taddr, rbuf[0]);
#pragma unroll
        for (int c = 0; c < NCH; ++c) {
          tmem_ld_wait();
          const uint32_t* rr_ = rbuf[c & 1];
          if (c + 1 < NCH) tmem_ld16(taddr + (uint32_t)((c + 1) * 16), rbuf[(c + 1) & 1]);
#pragma unroll
          for (int k = 0; k < 4; ++k)
            *reinterpret_cast<float4*>(stg + lane * EPI_PITCH + 4 * k) =
                make_float4(__uint_as_float(rr_[4 * k]), __uint_as_float(rr_[4 * k + 1]), __uint_as_float(rr_[4 * k + 2]),
                            __uint_as_float(rr_[4 * k + 3]));
          __syncwarp();
          const int col0 = col_base + c * 16;
          float* dst = p.out + (long long)row_base * p.row_stride + col0 + lane_col;
          if (vec_ok) {
            if (col0 + lane_col + 3 < p.P) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                const int rr = (lane >> 2) + 8 * i;
                if (rr < rows)
                  *reinterpret_cast<float4*>(dst + (long long)rr * p.row_stride) = *reinterpret_cast<const float4*>(stg + rr * EPI_PITCH + lane_col);
              }
            } else {
              for (int e = 0; e < 4; ++e)
                if (col0 + lane_col + e < p.P)
                  for (int i = 0; i < 4; ++i) {
                    const int rr = (lane >> 2) + 8 * i;
                    if (rr < rows) dst[(long long)rr * p.row_stride + e] = stg[rr * EPI_PITCH + lane_col + e];
                  }
            }
          } else if (col0 + lane_col < p.P) {
            for (int rr = (lane >> 4); rr < rows; rr += 2) dst[(long long)rr * p.row_stride] = stg[rr * EPI_PITCH + lane_col];
          }
          __syncwarp();
        }
      }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster_relaxed(te0 + (uint32_t)acc * 8u);
      if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
    }
  } else if (warp >= 4 + FWDX_EPI_WARPS) {
    // ================= converters: fp32 NCHW -> the bf16 MN-major half r of every pair, k-blocks kb % MP == q =================
    // Two groups of four warps take the CTA's owned k-blocks alternately (group g: owned blocks g, g + 2, ...).  Inside a group
    // warp cw owns channel rows [16 cw, 16 cw + 16) of the k-block and lane l pixels [4 l, 4 l + 4) of the 128-pixel half.  A
    // group's loads for its NEXT block are issued right after it has published the current one (the proxy fence before the
    // barrier arrive would otherwise wait for them), so every lane has 16 loads in flight for two owned blocks = 2 MP k-block
    // periods: 64 KB per SM, enough to cover the HBM latency at the rate the tensor core consumes.
    const int cwarp = warp - (4 + FWDX_EPI_WARPS);
    const int grp = cwarp >> 2, cw = cwarp & 3;
    // ownership by the cluster-wide k-block counter c = unit * kb_total + kb: CTA q converts c % MP == q, group (c / MP) % 2.
    // A group's consecutive blocks are therefore exactly 2 MP <= STAGES counters apart, so when it comes back to a stage the
    // use before the previous one has certainly been consumed and the parity wait below cannot be fooled (see static_assert).
    static_assert(2 * MP <= STAGES, "a converter group must revisit the ring within one lap (parity waits)");
    const int total_c = my_units * p.kb_total;
    const uint32_t box_off = (uint32_t)(lane >> 4) * MN_BOX_BYTES + (uint32_t)(lane & 1) * 8;   // 64-pixel box + half of the 16-byte chunk
    const uint32_t chunk = (uint32_t)((lane & 15) >> 1);
    const uint32_t smem_s = smem_u32(smem);
    uint32_t dst_base[MP];                                                     // the MP CTAs holding half r
#pragma unroll
    for (int d = 0; d < MP; ++d) dst_base[d] = mapa_u32(smem_s, (uint32_t)(2 * d + r));
    float4 buf[16];
    const float* src = nullptr;
    __nv_bfloat16* dstn = nullptr;
    // loads of the block with counter c (source address, by-product address)
    auto fetch_block = [&](int c) {
      const int u = c / p.kb_total;
      const int kb = c - u * p.kb_total;
      const int nt = worker + u * nworkers;
      const long long px = (long long)nt * BLOCK_N + r * (BLOCK_N / 2) + 4 * lane;
      src = nullptr; dstn = nullptr;
      if (px < p.P) {
        const int img = (int)(px / p.hw);
        const long long off = ((long long)img * p.K + kb * BLOCK_K + 16 * cw) * p.hw + (px - (long long)img * p.hw);
        src = p.x + off;
        if (p.xn != nullptr) dstn = p.xn + off;
      }
#pragma unroll
      for (int rr = 0; rr < 16; ++rr) buf[rr] = src ? ld_stream_f4(src + (long long)rr * p.hw) : make_float4(0.f, 0.f, 0.f, 0.f);
    };
    const int c_first = q + MP * grp;
    if (c_first < total_c) fetch_block(c_first);
#pragma unroll 1
    for (int c = c_first; c < total_c; c += 2 * MP) {
      const int stage = c % STAGES;
      const uint32_t phase = (uint32_t)(c / STAGES) & 1u;
      mbar_wait(&empty_bar[stage], phase ^ 1u);                     // all MP pairs have released this stage (in every CTA)
      const uint32_t so = (uint32_t)(stage * STAGE_BYTES + A_BYTES) + box_off;
#pragma unroll
      for (int rr = 0; rr < 16; ++rr) {
        const int row = 16 * cw + rr;
        const float4 v = buf[rr];
        const __nv_bfloat162 lo = __floats2bfloat162_rn(v.x, v.y), hi = __floats2bfloat162_rn(v.z, v.w);
        const uint32_t w0 = *reinterpret_cast<const uint32_t*>(&lo), w1 = *reinterpret_cast<const uint32_t*>(&hi);
        const uint32_t o = so + (uint32_t)row * 128u + ((chunk ^ (uint32_t)(row & 7)) << 4);
#pragma unroll
        for (int d = 0; d < MP; ++d) st_cluster_v2(dst_base[d] + o, w0, w1);
        if (dstn != nullptr) *reinterpret_cast<uint2*>(dstn + (long long)rr * p.hw) = make_uint2(w0, w1);
      }
      fence_proxy_async_all();                                      // this thread's generic-proxy writes -> visible to the async proxy
      named_bar_sync(1 + grp, 4 * 32 + 32);                         // the group's block is complete: hand it to the signaller warp
      if (c + 2 * MP < total_c) fetch_block(c + 2 * MP);            // in flight while the other group converts and the cluster advances
    }
  } else if (warp == 3) {
    // ================= signaller: publishes the converted blocks (release at cluster scope) =================
    // The barrier arrives carry release semantics over the whole cluster (a memory barrier each); keeping them off the converter
    // threads means those can put their next loads in flight immediately instead of draining them behind the barrier.
    const int total_c = my_units * p.kb_total;
    uint32_t dst_full[MP];
#pragma unroll
    for (int d = 0; d < MP; ++d) dst_full[d] = mapa_u32(smem_u32(&full_bar[0]), (uint32_t)(2 * d));
#pragma unroll 1
    for (int c = q; c < total_c; c += MP) {
      const int grp = (c / MP) & 1;
      named_bar_sync(1 + grp, 4 * 32 + 32);
      if (lane == 0) {
        const uint32_t stage = (uint32_t)(c % STAGES);
        asm volatile("fence.acq_rel.cluster;" ::: "memory");
#pragma unroll
        for (int d = 0; d < MP; ++d)
          asm volatile("mbarrier.arrive.relaxed.cluster.shared::cluster.b64 _, [%0];" ::"r"(dst_full[d] + stage * 8u) : "memory");
      }
      __syncwarp();
    }
  }

  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc_2sm(tmem_base, TMEM_COLS);
  }
}

// Host side (gemm_sm100.cu)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_fn();            // cuTensorMapEncodeTiled through the runtime's driver entry point (nullptr if unavailable)

struct Operand {
  const __nv_bfloat16* ptr;
  bool mn_major;        // false: [rows][K] K contiguous; true: [K][rows] rows contiguous
  long long pitch;      // elements between consecutive outer-dimension entries
};
// forward GEMM with in-kernel fp32 NCHW -> bf16 conversion of the pixel operand (see gemm_fwd_convert_kernel); returns
// B200SEG_ERR_UNSUPPORTED when the shape is not eligible (hw % 4, K % 64, alignment) -- the caller then packs and uses launch()
bool fwd_convert_eligible(const float* x, int K, int hw, int M);
int launch_fwd_convert(const __nv_bfloat16* a, long long a_pitch, const float* x, int n_img, int hw, int M, int K, float* out,
                       long long row_stride, __nv_bfloat16* xn, cudaStream_t stream, int prof_tag);
// What the GEMM writes: one layout and the fields that layout takes.  Build it with the functions below.
struct Out {
  enum Layout {
    F32,              // fp32 row-major: D[m, n] at ptr[m * row_stride + n]
    F32_NCHW_COLS,    // fp32 NCHW with the columns as pixels: D[m, n] at ptr[(n / hw) * img_stride + m * row_stride + n % hw]
    F32_NCHW_ROWS,    // fp32 NCHW with the rows as pixels, stored from registers: D[m, n] at ptr[(m / hw) * img_stride + n * hw + m % hw]
    BF16,             // bf16 row-major [M][row_stride]: N and row_stride multiples of 8, ptr 16-byte aligned
    SEAM,             // bf16 row-major [M][N] = bf16_rn(relu((D * scale[n] + bias[n]) + identity)), M = n_img * hw pixels,
                      // identity fp32 NCHW [n_img][N][hw]; K-major operands, N % 8 == 0, ptr 16-byte aligned
    F32_NCHW_ROWS_STATS,  // F32_NCHW_ROWS, and stats[(m / 32) * N + n] = (mean, M2) over the (up to) 32 pixels m of each lane
                          // group: always cta_group::2 pairs, K-major operands, no split-K
  } layout;
  void* ptr;
  long long row_stride, img_stride, split_stride;   // split_stride: elements between split-K slabs (F32, F32_NCHW_COLS, BF16)
  int hw;                                           // pixels per image (F32_NCHW_COLS, F32_NCHW_ROWS, SEAM, F32_NCHW_ROWS_STATS)
  const float *identity, *scale, *bias;             // SEAM
  float2* stats;                                    // F32_NCHW_ROWS_STATS: [ceil(M / 32)][N]
};
inline Out out_f32(float* d, long long row_stride, long long split_stride = 0) { return {Out::F32, d, row_stride, 0, split_stride}; }
inline Out out_f32_nchw_cols(float* d, int hw, long long row_stride, long long img_stride, long long split_stride = 0) {
  return {Out::F32_NCHW_COLS, d, row_stride, img_stride, split_stride, hw};
}
inline Out out_f32_nchw_rows(float* d, int hw, long long img_stride) { return {Out::F32_NCHW_ROWS, d, 0, img_stride, 0, hw}; }
inline Out out_bf16(__nv_bfloat16* d, long long row_stride, long long split_stride = 0) { return {Out::BF16, d, row_stride, 0, split_stride}; }
inline Out out_seam(__nv_bfloat16* d, const float* identity, const float* scale, const float* bias, int hw) {
  return {Out::SEAM, d, 0, 0, 0, hw, identity, scale, bias};
}
inline Out out_f32_nchw_rows_stats(float* d, int hw, long long img_stride, float2* stats) {
  return {Out::F32_NCHW_ROWS_STATS, d, 0, img_stride, 0, hw, nullptr, nullptr, nullptr, stats};
}

// D = A B^T, A [M][K] and B [N][K] (each K-major or MN-major), written as `out` says
struct Gemm {
  Operand a, b;
  int M, N, K;
  Out out;
  int splits = 1;                // split-K (clamped so that every split is non-empty); the count used goes to *splits_used
  int* splits_used = nullptr;
  int share = SHARE_NONE;        // the sharing geometry the caller asks for; b200seg_gemm_set_sharing() may veto or override it
  int pair_fallback = SHARE_B;   // what SHARE_PAIR becomes under sharing mode 5 (no cta_group::2)
  int sm_reserve = 0;            // SMs left free for a concurrent kernel
  int prof_tag = -1;
  int* variant_used = nullptr;   // the index of the kernel launched, in the table variant_info() reads
};
int launch(const Gemm& g, cudaStream_t stream);

}  // namespace gemm
}  // namespace b200seg
