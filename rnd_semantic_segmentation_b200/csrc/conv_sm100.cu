// 3x3 convolution layers as tcgen05 implicit GEMMs -- the PixelDiscriminator conv stack (SURVEY.md section 8f rank 1).
//
// Replaces (reference file:line): core/models/discriminator.py:34-41 (D = conv3x3(Cin,256)+LeakyReLU(0.2) ->
// conv3x3(256,128)+LeakyReLU(0.2); cls1 / cls2 = conv3x3(128,C)), applied at :45-47, and their autograd backward
// (call sites core/trainers/aspp_fada.py:110,119,123).
//
// Activations are bf16 NHWC ([N,h,w,C], channel pitch a multiple of 8) end to end, accumulation is fp32 in TMEM.
// There is NO im2col buffer: the "im2col" is done by TMA.  The activation tensor is described by a 4-D tensor map
// (c, x, y, n); the A tile of tap (dy, dx) is the box {64 channels, TW columns, TH rows, 1 image} fetched at the
// tile origin SHIFTED by (dx, dy).  Coordinates outside the image (including negative ones) are zero-filled by the
// TMA unit, which is exactly the convolution's zero padding -- no halo handling, no bounds tests in the kernel.
//
//   MODE_CONV  (forward, and data gradient = the same convolution with negated taps and transposed weights)
//       D[pixel, co] = sum_t sum_ck act[pixel + d_t, ck] * Wt[t][co][ck]
//       M = 128 pixels (a TH x TW rectangle of one image), N = 256 output channels, K = T * Ck (tap-major)
//       A: 4-D box, K-major;  B: 3-D map (ck, co, t), box {64, 256, 1}, K-major (rows >= Co are zero-filled)
//       epilogue (straight from TMEM, one pixel per thread): + bias, LeakyReLU, or * LeakyReLU'(saved activation),
//       then bf16 NHWC (the next layer's operand) or fp32 NCHW (the module's output / the feature gradient; for a
//       fixed channel a warp writes 32 consecutive pixels = 128 contiguous bytes, no transpose needed).
//   MODE_WGRAD
//       dW[t][co][ci] = sum_pixels G[pixel, co] * X[pixel + d_t, ci]
//       M = 128 co, N = 256 ci, K = pixels in chunks of 64 (a THk x TWk rectangle); both operands MN-major 4-D boxes
//       {64 channels, TWk, THk, 1}; X's box is shifted by the tap.  Work unit = (split, tap, M-tile, N-tile); fp32
//       partial slabs [split][t][Co][Ci] reduced and permuted to [Co][Ci][3][3] by conv_wgrad_reduce_kernel.
//
// Pipeline / roles are those of gemm_sm100.cuh (4-stage 48 KB TMA ring, one MMA-issuing thread, two 256-column TMEM
// accumulators, persistent CTAs, 8 epilogue warps).
//
// OP_TF32: the same GEMMs with fp32 operands read by tcgen05.mma.kind::tf32.  A 128-byte swizzle row then holds 32 channels, so a
// k-block is 32 channels (CONV) or 32 pixels (WGRAD), an MMA covers K = 8 (still 32 bytes of a K-major row, 8 k-rows of an
// MN-major box) and the stage sizes are those of bf16.  MN-major tf32 boxes use the 32-byte-chunk swizzle (SWIZZLE_128B_BASE32B),
// the one swizzled layout tcgen05 reads MN-major 32-bit operands from.  Activations and inter-layer gradients are fp32 NHWC (OUT_F32_NHWC) rounded
// to TF32 (nearest-even) when stored, so every operand the tensor core reads is exact; the fused column sums are taken from the
// unrounded values, and the LeakyReLU' mask is read as fp32.
#include <limits.h>
#include "common.cuh"
#include "gemm_sm100.cuh"

namespace b200seg {
namespace gemm {
namespace conv {

constexpr int MAX_T = 9;
constexpr int MODE_CONV = 0, MODE_WGRAD = 1;
constexpr int OUT_BF16_NHWC = 0, OUT_F32_NCHW = 1, OUT_F32_NHWC = 2;
constexpr int OP_BF16 = 0, OP_TF32 = 1;
// channels per 128-byte swizzle row = channels (CONV) or pixels (WGRAD) per k-block
__host__ __device__ constexpr int op_kb(int op) { return op == OP_TF32 ? 32 : 64; }
__host__ __device__ constexpr int op_bytes(int op) { return op == OP_TF32 ? 4 : 2; }
// the kernel's k-block geometry: KB channels or pixels per k-block, UK = the K of one MMA, MN_BOX = bytes of one MN-major box.
// MN-major tf32 operands take the 32-byte-chunk swizzle (TMA CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B), whose atom is 4 rows of 128 B:
// MN_SBO = the stride between 4-row k groups, MN_LAYOUT its descriptor layout type.
template <int OP> struct OpGeom {
  static constexpr int KB = op_kb(OP), UK = OP == OP_TF32 ? 8 : UMMA_K, MN_BOX = KB * 128;
  static constexpr uint32_t MN_SBO = OP == OP_TF32 ? 512 : 1024, MN_LAYOUT = OP == OP_TF32 ? SMEM_SW128_BASE32B : SMEM_SW128;
};
// BN = accumulator columns per tile: 256, or 128 for layers with <= 128 output channels (half the MMA work of a padded 256)
// PAIR = two CTAs of a cluster drive ONE tcgen05.mma.cta_group::2 (M = 256: 128 rows per CTA, N = BN): each CTA stages its own
// A tile and only HALF of the B tile (the tensor core reads the other half from the peer's shared memory), so the bytes a
// CTA pulls from L2 and the shared-memory operand reads per MMA drop by a third / a half.
template <int BN, bool PAIR> struct Cfg {
  static constexpr int B_ROWS = PAIR ? BN / 2 : BN;                 // B rows (output channels) staged per CTA
  static constexpr int B_BYTES_T = B_ROWS * BLOCK_K * 2;
  static constexpr int STAGE_T = A_BYTES + B_BYTES_T;
  static constexpr int NSTAGE = (200 * 1024) / STAGE_T > 8 ? 8 : (200 * 1024) / STAGE_T;     // 4 / 6 / 6 / 8
  static constexpr int SMEM = 1024 + NSTAGE * STAGE_T + 256;
};

// TMA loads whose completion is signalled on a barrier given as a shared::cluster address; with PAIR (.cta_group::2) that
// barrier may live in the peer CTA (the leader's full barrier collects the bytes of both CTAs)
template <bool PAIR>
__device__ __forceinline__ void tma_ld3(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2) {
  if (PAIR)
    asm volatile("cp.async.bulk.tensor.3d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
  else
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
                 ::"r"(smem_dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2) : "memory");
}
template <bool PAIR>
__device__ __forceinline__ void tma_ld4(uint32_t smem_dst, const CUtensorMap* m, uint32_t bar, int c0, int c1, int c2, int c3) {
  if (PAIR)
    asm volatile("cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(smem_dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
  else
    asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
                 ::"r"(smem_dst), "l"(m), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
struct ConvParams {
  int N, h, w;
  int tw_shift, TW, TH, tiles_x, tiles_y;   // pixel rectangle: M-tile (CONV, TW*TH = 128) or K-chunk (WGRAD, TW*TH = 64)
  int T;
  int dy[MAX_T], dx[MAX_T];
  int KC;                  // CONV: 64-channel chunks per tap
  int Co;                  // CONV: output channels (GEMM N);  WGRAD: gradient channels (GEMM M)
  int Ci;                  // WGRAD: input channels (GEMM N)
  int m_tiles, n_tiles, units;
  int splits, kb_per_split, kb_total;
  void* out;
  int out_mode;
  long long out_pitch;     // OUT_BF16_NHWC: elements between pixels (also the pitch of `mask`)
  const float* bias;       // [Co] or null
  int act;                 // apply LeakyReLU(slope) after the bias
  float slope;
  const __nv_bfloat16* mask;   // saved post-activation output of the layer below ([pixels][out_pitch]): multiply by LeakyReLU'
  long long split_stride;  // WGRAD: elements between split-K slabs
  float* colsum_part;      // CONV + NHWC output: per (M-tile, warp row quarter) column sums of the STORED (bf16-rounded) values,
  int m_tiles_real;        //   [m_tiles_real * 4][out_pitch] -> the bias gradient without another pass over the tensor
                           //   (OP_TF32 + OUT_F32_NHWC: of the values before their TF32 rounding)
};

__device__ __forceinline__ void tma_load_3d(uint32_t smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_dst), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(uint32_t smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_dst), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// pixel rectangle index -> (image, y0, x0)
__device__ __forceinline__ void rect_origin(const ConvParams& p, int idx, int& img, int& y0, int& x0) {
  const int per_img = p.tiles_x * p.tiles_y;
  img = idx / per_img;
  const int r = idx - img * per_img;
  const int ty = r / p.tiles_x;
  y0 = ty * p.TH;
  x0 = (r - ty * p.tiles_x) * p.TW;
}

struct Unit {
  int z, t, mt, nt, kb0, kb1;
};
// p.m_tiles counts PAIRS of M-tiles when the kernel runs as CTA pairs: CTA `rank` of the pair owns M-tile 2 * pm + rank
template <int MODE, bool PAIR>
__device__ __forceinline__ Unit decode_unit(const ConvParams& p, int unit, int rank) {
  Unit u;
  if (MODE == MODE_CONV) {
    u.z = 0; u.t = 0;
    u.nt = unit / p.m_tiles;                 // M fastest: CTAs running together share the weight slice
    u.mt = unit - u.nt * p.m_tiles;
    u.kb0 = 0; u.kb1 = p.kb_total;
  } else {
    const int per_tap = p.m_tiles * p.n_tiles;
    const int per_split = per_tap * p.T;
    u.z = unit / per_split;
    int rem = unit - u.z * per_split;
    u.t = rem / per_tap;
    rem -= u.t * per_tap;
    u.nt = rem / p.m_tiles;
    u.mt = rem - u.nt * p.m_tiles;
    u.kb0 = u.z * p.kb_per_split;
    u.kb1 = min(p.kb_total, u.kb0 + p.kb_per_split);
  }
  if (PAIR) u.mt = u.mt * 2 + rank;
  return u;
}

template <int MODE, int BN, bool PAIR, int OP>
__global__ void __launch_bounds__(NUM_THREADS, 1)
conv_gemm_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b, const ConvParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw_addr = smem_u32(smem_raw);
  const uint32_t pad = (1024u - (raw_addr & 1023u)) & 1023u;
  uint8_t* smem = smem_raw + pad;
  constexpr int STAGES = Cfg<BN, PAIR>::NSTAGE, STAGE_BYTES = Cfg<BN, PAIR>::STAGE_T;      // shadow the constants of gemm::
  constexpr int BLOCK_N = BN;
  constexpr int B_ROWS = Cfg<BN, PAIR>::B_ROWS;
  constexpr int NCTA = PAIR ? 2 : 1;
  const int rank = PAIR ? (int)cluster_cta_rank() : 0;
  const int worker = (int)blockIdx.x / NCTA, nworkers = (int)gridDim.x / NCTA;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + STAGES * STAGE_BYTES);
  uint64_t* full_bar = bars;
  uint64_t* empty_bar = bars + STAGES;
  uint64_t* tfull_bar = bars + 2 * STAGES;
  uint64_t* tempty_bar = bars + 2 * STAGES + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

  const int warp = threadIdx.x >> 5;
  const int lane = threadIdx.x & 31;
  constexpr bool MN = MODE == MODE_WGRAD;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmap_a);
    tma_prefetch_desc(&tmap_b);
  }
  if (warp == 1 && lane == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&full_bar[s], 1);
      mbar_init(&empty_bar[s], 1);
    }
    for (int a = 0; a < 2; ++a) {
      mbar_init(&tfull_bar[a], 1);
      mbar_init(&tempty_bar[a], EPI_WARPS * NCTA);        // the leader's MMA thread waits for the epilogue warps of BOTH CTAs
    }
    fence_mbar_init();
  }
  if (warp == 2) {
    if (PAIR) tmem_alloc_2sm(tmem_slot, TMEM_COLS);
    else tmem_alloc(tmem_slot, TMEM_COLS);
  }
  tc_fence_before();
  __syncthreads();
  if (PAIR) cluster_sync_all();              // the peer's barriers are initialised before any remote arrive / TMA completion
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ================= TMA producer =================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int unit = worker; unit < p.units; unit += nworkers) {
        const Unit u = decode_unit<MODE, PAIR>(p, unit, rank);
        int img = 0, y0 = 0, x0 = 0;
        if (MODE == MODE_CONV) rect_origin(p, u.mt, img, y0, x0);
        for (int kb = u.kb0; kb < u.kb1; ++kb) {
          mbar_wait(&empty_bar[stage], phase ^ 1u);
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
          // PAIR: both CTAs' loads complete on the LEADER's full barrier, which expects the bytes of both
          if (rank == 0) mbar_arrive_expect_tx(&full_bar[stage], STAGE_BYTES * NCTA);
          const uint32_t fb = PAIR ? mapa_u32(smem_u32(&full_bar[stage]), 0) : smem_u32(&full_bar[stage]);
          if (MODE == MODE_CONV) {
            const int t = kb / p.KC, kc = kb - t * p.KC;
            tma_ld4<PAIR>(sa, &tmap_a, fb, kc * OpGeom<OP>::KB, x0 + p.dx[t], y0 + p.dy[t], img);
            tma_ld3<PAIR>(sb, &tmap_b, fb, kc * OpGeom<OP>::KB, u.nt * BLOCK_N + rank * B_ROWS, t);
          } else {
            rect_origin(p, kb, img, y0, x0);
#pragma unroll
            for (int b = 0; b < BLOCK_M / OpGeom<OP>::KB; ++b)
              tma_ld4<PAIR>(sa + b * OpGeom<OP>::MN_BOX, &tmap_a, fb, u.mt * BLOCK_M + b * OpGeom<OP>::KB, x0, y0, img);
            const int xs = x0 + p.dx[u.t], ys = y0 + p.dy[u.t];
#pragma unroll
            for (int b = 0; b < B_ROWS / OpGeom<OP>::KB; ++b)
              tma_ld4<PAIR>(sb + b * OpGeom<OP>::MN_BOX, &tmap_b, fb, u.nt * BLOCK_N + rank * B_ROWS + b * OpGeom<OP>::KB, xs, ys, img);
          }
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    if (lane == 0 && rank == 0) {                                    // PAIR: the leader CTA issues for both
      constexpr uint32_t idesc = make_idesc(MN, MN, BLOCK_M * NCTA, BLOCK_N, OP == OP_TF32 ? IDESC_TF32 : IDESC_BF16);
      constexpr uint32_t lbo = MN ? OpGeom<OP>::MN_BOX : 16, sbo = MN ? OpGeom<OP>::MN_SBO : 1024, step = MN ? OpGeom<OP>::UK * 128 : 32;
      constexpr uint32_t layout = MN ? OpGeom<OP>::MN_LAYOUT : SMEM_SW128;
      int stage = 0;
      uint32_t phase = 0;
      int acc = 0;
      uint32_t acc_phase = 0;
      for (int unit = worker; unit < p.units; unit += nworkers) {
        const Unit u = decode_unit<MODE, PAIR>(p, unit, rank);
        mbar_wait(&tempty_bar[acc], acc_phase ^ 1u);
        tc_fence_after();
        const uint32_t tmem_d = tmem_base + (uint32_t)(acc * BLOCK_N);
        for (int kb = u.kb0; kb < u.kb1; ++kb) {
          mbar_wait(&full_bar[stage], phase);
          tc_fence_after();
          const uint32_t sa = smem_u32(smem + stage * STAGE_BYTES);
          const uint32_t sb = sa + A_BYTES;
#pragma unroll
          for (int k = 0; k < OpGeom<OP>::KB / OpGeom<OP>::UK; ++k) {
            const uint64_t adesc = make_smem_desc(sa + k * step, lbo, sbo, layout);
            const uint64_t bdesc = make_smem_desc(sb + k * step, lbo, sbo, layout);
            if constexpr (OP == OP_TF32) {
              if (PAIR) umma_tf32_2sm(tmem_d, adesc, bdesc, idesc, (kb > u.kb0 || k > 0) ? 1u : 0u);
              else umma_tf32(tmem_d, adesc, bdesc, idesc, (kb > u.kb0 || k > 0) ? 1u : 0u);
            } else {
              if (PAIR) umma_bf16_2sm(tmem_d, adesc, bdesc, idesc, (kb > u.kb0 || k > 0) ? 1u : 0u);
              else umma_bf16(tmem_d, adesc, bdesc, idesc, (kb > u.kb0 || k > 0) ? 1u : 0u);
            }
          }
          if (PAIR) umma_commit_2sm(&empty_bar[stage], 0x3);         // frees the stage in both CTAs
          else umma_commit(&empty_bar[stage]);
          if (++stage == STAGES) { stage = 0; phase ^= 1u; }
        }
        if (PAIR) umma_commit_2sm(&tfull_bar[acc], 0x3);
        else umma_commit(&tfull_bar[acc]);
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else if (warp >= 4) {
    // ================= epilogue: warp owns TMEM lanes [32*(warp%4), +32) and 128 of the 256 accumulator columns ========
    const int wq = warp & 3;
    const int half = (warp - 4) >> 2;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int unit = worker; unit < p.units; unit += nworkers) {
      const Unit u = decode_unit<MODE, PAIR>(p, unit, rank);
      mbar_wait(&tfull_bar[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(wq * 32) << 16) + (uint32_t)(acc * BLOCK_N + half * (BLOCK_N / 2));
      const int row = wq * 32 + lane;
      if (MODE == MODE_CONV) {
        int img, y0, x0;
        rect_origin(p, u.mt, img, y0, x0);
        const int yy = row >> p.tw_shift, xx = row & (p.TW - 1);
        const int y = y0 + yy, x = x0 + xx;
        const bool valid = y < p.h && x < p.w && img < p.N;      // img >= N: the odd M-tile of the last pair
        const long long pix = ((long long)img * p.h + y) * p.w + x;
#pragma unroll 1
        for (int c = 0; c < BLOCK_N / 2 / 32; ++c) {
          const int col0 = u.nt * BLOCK_N + half * (BLOCK_N / 2) + c * 32;
          if (col0 >= p.Co) break;                               // warp-uniform
          uint32_t r[32];
          tmem_ld32(taddr + (uint32_t)(c * 32), r);
          tmem_ld_wait();
          float v[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = __uint_as_float(r[j]);
          if (p.bias) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] += (col0 + j < p.Co) ? __ldg(p.bias + col0 + j) : 0.f;
          }
          if (p.act) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = v[j] > 0.f ? v[j] : v[j] * p.slope;
          }
          if constexpr (OP == OP_TF32) {
            if (p.mask && valid) {
              const float4* mp = reinterpret_cast<const float4*>(reinterpret_cast<const float*>(p.mask) + pix * p.out_pitch + col0);
#pragma unroll
              for (int k = 0; k < 8; ++k) {
                if (col0 + 4 * k < p.Co) {
                  const float4 m4 = __ldg(mp + k);
                  v[4 * k] *= m4.x > 0.f ? 1.f : p.slope;                 // ATen's x > 0 test: LeakyReLU'(0) = slope
                  v[4 * k + 1] *= m4.y > 0.f ? 1.f : p.slope;
                  v[4 * k + 2] *= m4.z > 0.f ? 1.f : p.slope;
                  v[4 * k + 3] *= m4.w > 0.f ? 1.f : p.slope;
                }
              }
            }
            if (p.out_mode == OUT_F32_NHWC) {
              if (valid) {
                float4* op = reinterpret_cast<float4*>(reinterpret_cast<float*>(p.out) + pix * p.out_pitch + col0);
#pragma unroll
                for (int k = 0; k < 8; ++k)
                  if (col0 + 4 * k < p.Co)
                    op[k] = make_float4(tf32_rn(v[4 * k]), tf32_rn(v[4 * k + 1]), tf32_rn(v[4 * k + 2]), tf32_rn(v[4 * k + 3]));
              }
              if (p.colsum_part) {                                 // the unrounded values (a bias gradient never passes through TF32)
#pragma unroll
                for (int j = 0; j < 32; ++j) v[j] = valid ? v[j] : 0.f;
#pragma unroll
                for (int sft = 16; sft >= 1; sft >>= 1) {          // the exchange of the bf16 path below
                  const bool up = (lane & sft) != 0;
#pragma unroll
                  for (int i = 0; i < sft; ++i) {
                    const float send = up ? v[i] : v[i + sft];
                    const float keep = up ? v[i + sft] : v[i];
                    v[i] = keep + __shfl_xor_sync(0xffffffffu, send, sft);
                  }
                }
                if (u.mt < p.m_tiles_real && col0 + lane < p.Co)
                  p.colsum_part[((long long)u.mt * 4 + wq) * p.out_pitch + col0 + lane] = v[0];
              }
              continue;
            }
          } else if (p.mask && valid) {
            const uint4* mp = reinterpret_cast<const uint4*>(p.mask + pix * p.out_pitch + col0);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if (col0 + 8 * k < p.Co) {
                const uint4 m4 = __ldg(mp + k);
                const uint32_t mw[4] = {m4.x, m4.y, m4.z, m4.w};
#pragma unroll
                for (int e = 0; e < 4; ++e) {
                  // bf16 > 0  <=>  sign bit clear and magnitude non-zero (LeakyReLU'(0) = slope, as ATen's x > 0 test)
                  const uint32_t lo = mw[e] & 0xFFFFu, hi = mw[e] >> 16;
                  const bool plo = lo != 0u && lo < 0x8000u, phi = hi != 0u && hi < 0x8000u;
                  v[8 * k + 2 * e] *= plo ? 1.f : p.slope;
                  v[8 * k + 2 * e + 1] *= phi ? 1.f : p.slope;
                }
              }
            }
          }
          if (p.out_mode == OUT_BF16_NHWC) {
            uint32_t w16[16];
#pragma unroll
            for (int e = 0; e < 16; ++e) {
              const __nv_bfloat162 b2 = __floats2bfloat162_rn(v[2 * e], v[2 * e + 1]);
              w16[e] = *reinterpret_cast<const uint32_t*>(&b2);
              if (p.colsum_part) {                                 // sum what is stored, so the result equals a pass over the tensor
                v[2 * e] = valid ? __low2float(b2) : 0.f;
                v[2 * e + 1] = valid ? __high2float(b2) : 0.f;
              }
            }
            if (valid) {
              uint4* op = reinterpret_cast<uint4*>(reinterpret_cast<__nv_bfloat16*>(p.out) + pix * p.out_pitch + col0);
#pragma unroll
              for (int k = 0; k < 4; ++k)
                if (col0 + 8 * k < p.Co) op[k] = make_uint4(w16[4 * k], w16[4 * k + 1], w16[4 * k + 2], w16[4 * k + 3]);
            }
            if (p.colsum_part) {
              // 32 rows (lanes) x 32 columns -> lane l ends up with the sum of column l over the warp's rows: five exchange
              // steps, each halving the values a lane carries (31 shuffles instead of 32 x 5); fixed order => deterministic
#pragma unroll
              for (int sft = 16; sft >= 1; sft >>= 1) {
                const bool up = (lane & sft) != 0;
#pragma unroll
                for (int i = 0; i < sft; ++i) {
                  const float send = up ? v[i] : v[i + sft];
                  const float keep = up ? v[i + sft] : v[i];
                  v[i] = keep + __shfl_xor_sync(0xffffffffu, send, sft);
                }
              }
              if (u.mt < p.m_tiles_real && col0 + lane < p.Co)
                p.colsum_part[((long long)u.mt * 4 + wq) * p.out_pitch + col0 + lane] = v[0];
            }
          } else if (valid) {
            {
              const long long hw = (long long)p.h * p.w;
              float* op = reinterpret_cast<float*>(p.out) + ((long long)img * p.Co + col0) * hw + (long long)y * p.w + x;
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (col0 + j < p.Co) op[j * hw] = v[j];
            }
          }
        }
      } else {
        const int grow = u.mt * BLOCK_M + row;                    // gradient channel co
        float* out = reinterpret_cast<float*>(p.out) + (long long)u.z * p.split_stride +
                     ((long long)u.t * p.Co + grow) * p.Ci;
#pragma unroll 1
        for (int c = 0; c < BLOCK_N / 2 / 32; ++c) {
          const int col0 = u.nt * BLOCK_N + half * (BLOCK_N / 2) + c * 32;
          if (col0 >= p.Ci) break;
          uint32_t r[32];
          tmem_ld32(taddr + (uint32_t)(c * 32), r);
          tmem_ld_wait();
          if (grow < p.Co) {
#pragma unroll
            for (int k = 0; k < 8; ++k)
              if (col0 + 4 * k < p.Ci)                            // Ci is a multiple of 4
                *reinterpret_cast<float4*>(out + col0 + 4 * k) =
                    make_float4(__uint_as_float(r[4 * k]), __uint_as_float(r[4 * k + 1]), __uint_as_float(r[4 * k + 2]),
                                __uint_as_float(r[4 * k + 3]));
          }
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
  if (PAIR) cluster_sync_all();              // the leader's MMAs read the peer's shared memory; remote arrives must have landed
  if (warp == 2) {
    tc_fence_after();
    if (PAIR) tmem_dealloc_2sm(tmem_base, TMEM_COLS);
    else tmem_dealloc(tmem_base, TMEM_COLS);
  }
}

// ------------------------------------------------------------------------------------------
// host: tensor maps
// ------------------------------------------------------------------------------------------
static int make_tmap_nd(CUtensorMap* m, const void* ptr, int rank, const cuuint64_t* gdim, const cuuint64_t* gstride_bytes,
                        const cuuint32_t* box, int op, bool mn = false) {
  EncodeTiledFn fn = encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point not available (driver too old or no GPU)");
    return B200SEG_ERR_CUDA;
  }
  B200SEG_CHECK_ARG((reinterpret_cast<uintptr_t>(ptr) & 15) == 0, "conv: TMA operand pointer must be 16-byte aligned");
  for (int i = 0; i < rank - 1; ++i)
    B200SEG_CHECK_ARG(gstride_bytes[i] % 16 == 0, "conv: TMA stride %d (%llu bytes) must be a multiple of 16", i,
                      (unsigned long long)gstride_bytes[i]);
  cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  CUresult r = fn(m, op == OP_TF32 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(ptr), gdim, gstride_bytes, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE,
                  (mn && op == OP_TF32) ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("conv: cuTensorMapEncodeTiled (rank %d) failed with CUresult %d", rank, (int)r);
    return B200SEG_ERR_CUDA;
  }
  return B200SEG_OK;
}

// activation map over NHWC [N][h][w][pitch] (bf16, or fp32 with OP_TF32) exposing `C` channels, box {64 | 32, TW, TH, 1};
// mn: the box is an MN-major operand (weight-gradient mode)
static int make_act_tmap(CUtensorMap* m, const void* ptr, int N, int h, int w, int C, long long pitch, int TW, int TH, int op,
                         bool mn = false) {
  const cuuint64_t es = (cuuint64_t)op_bytes(op);
  cuuint64_t gdim[4] = {(cuuint64_t)C, (cuuint64_t)w, (cuuint64_t)h, (cuuint64_t)N};
  cuuint64_t gstr[3] = {(cuuint64_t)pitch * es, (cuuint64_t)pitch * es * w, (cuuint64_t)pitch * es * w * h};
  cuuint32_t box[4] = {(cuuint32_t)op_kb(op), (cuuint32_t)TW, (cuuint32_t)TH, 1};
  return make_tmap_nd(m, ptr, 4, gdim, gstr, box, op, mn);
}

// pixel rectangle of `area` pixels (power of two) with the least padding over an h x w image; ties -> widest
static void pick_rect(int h, int w, int area, int* TW, int* TH) {
  long long best = LLONG_MAX;
  for (int tw = area; tw >= 8; tw >>= 1) {
    const int th = area / tw;
    const long long cover = (long long)ceil_div(w, tw) * ceil_div(h, th);
    if (cover < best) { best = cover; *TW = tw; *TH = th; }
  }
}

static void fill_taps(ConvParams& p, int dilation, int sign) {
  p.T = 9;
  for (int ky = 0; ky < 3; ++ky)
    for (int kx = 0; kx < 3; ++kx) {
      p.dy[ky * 3 + kx] = sign * (ky - 1) * dilation;
      p.dx[ky * 3 + kx] = sign * (kx - 1) * dilation;
    }
}

static int ilog2(int v) { int s = 0; while ((1 << s) < v) ++s; return s; }

static int g_pair = 1;                 // b200seg_conv_set_pair(): 0 = one CTA per tile, 1 = CTA pairs (cta_group::2) where two M-tiles exist
void set_pair(int on) { g_pair = on; }

template <int MODE, int BN, bool PAIR, int OP>
static int launch_conv_t(const CUtensorMap& ta, const CUtensorMap& tb, const ConvParams& p, cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    B200SEG_CUDA(cudaFuncSetAttribute(conv_gemm_kernel<MODE, BN, PAIR, OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<BN, PAIR>::SMEM));
    configured = true;
  }
  const int sms = num_sms();
  if (!PAIR) {
    const int grid = p.units < sms ? p.units : sms;
    conv_gemm_kernel<MODE, BN, PAIR, OP><<<grid, NUM_THREADS, Cfg<BN, PAIR>::SMEM, stream>>>(ta, tb, p);
  } else {
    const int pairs = p.units < sms / 2 ? p.units : sms / 2;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.dynamicSmemBytes = Cfg<BN, PAIR>::SMEM;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    B200SEG_CUDA(cudaLaunchKernelEx(&cfg, conv_gemm_kernel<MODE, BN, PAIR, OP>, ta, tb, p));
  }
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}
template <int MODE, int OP>
static int launch_conv_op(const CUtensorMap& ta, const CUtensorMap& tb, const ConvParams& p, int BN, bool pair, cudaStream_t stream) {
  if (BN == 128) return pair ? launch_conv_t<MODE, 128, true, OP>(ta, tb, p, stream) : launch_conv_t<MODE, 128, false, OP>(ta, tb, p, stream);
  return pair ? launch_conv_t<MODE, 256, true, OP>(ta, tb, p, stream) : launch_conv_t<MODE, 256, false, OP>(ta, tb, p, stream);
}
template <int MODE>
static int launch_conv(const CUtensorMap& ta, const CUtensorMap& tb, const ConvParams& p, int BN, bool pair, int op, cudaStream_t stream) {
  return op == OP_TF32 ? launch_conv_op<MODE, OP_TF32>(ta, tb, p, BN, pair, stream) : launch_conv_op<MODE, OP_BF16>(ta, tb, p, BN, pair, stream);
}

// D[pixel, co] = sum_t sum_ck act[pixel + sign*d_t, ck] * wt[t][co][ck]  (+ epilogue), see the header comment.  act, wt and
// mask are bf16 (OP_BF16) or fp32 holding TF32 values (OP_TF32)
static int conv3x3_run(const void* act, int N, int h, int w, int Ck, long long act_pitch, const void* wt, int Co, int dilation, int sign,
                       const float* bias, int lrelu, float slope, const void* mask, void* out, int out_mode, long long out_pitch,
                       cudaStream_t stream, int prof_tag, float* colsum_part, int op) {
  B200SEG_CHECK_ARG(act && wt && out, "conv3x3: null pointer");
  B200SEG_CHECK_ARG(out_mode != OUT_F32_NHWC || op == OP_TF32, "conv3x3: the fp32 NHWC output belongs to the TF32 layers");
  B200SEG_CHECK_ARG(!colsum_part || out_mode != OUT_F32_NCHW, "conv3x3: fused column sums need an NHWC output");
  B200SEG_CHECK_ARG(N > 0 && h > 0 && w > 0 && Ck > 0 && Co > 0 && dilation > 0, "conv3x3: bad geometry");
  B200SEG_CHECK_ARG(Ck % 8 == 0 && act_pitch % 8 == 0 && act_pitch >= Ck, "conv3x3: input channels (%d, pitch %lld) must be multiples of 8", Ck, act_pitch);
  B200SEG_CHECK_ARG((long long)N * h * w < (1LL << 31), "conv3x3: too many pixels");
  if (out_mode != OUT_F32_NCHW || mask)
    B200SEG_CHECK_ARG(Co % 8 == 0 && out_pitch % 8 == 0 && out_pitch >= Co && (reinterpret_cast<uintptr_t>(out) & 15) == 0 &&
                          (reinterpret_cast<uintptr_t>(mask) & 15) == 0,
                      "conv3x3: NHWC output / mask need channel counts that are multiples of 8 and 16-byte aligned bases");
  ConvParams p = {};
  p.N = N; p.h = h; p.w = w;
  pick_rect(h, w, BLOCK_M, &p.TW, &p.TH);
  p.tw_shift = ilog2(p.TW);
  p.tiles_x = ceil_div(w, p.TW);
  p.tiles_y = ceil_div(h, p.TH);
  fill_taps(p, dilation, sign);
  p.KC = ceil_div(Ck, op_kb(op));
  p.Co = Co; p.Ci = 0;
  const int BN = Co <= 128 ? 128 : 256;
  p.m_tiles = N * p.tiles_x * p.tiles_y;
  p.m_tiles_real = p.m_tiles;
  p.colsum_part = colsum_part;
  const bool pair = g_pair && p.m_tiles >= 2;
  if (pair) p.m_tiles = ceil_div(p.m_tiles, 2);       // pairs of M-tiles
  p.n_tiles = ceil_div(Co, BN);
  p.units = p.m_tiles * p.n_tiles;
  p.splits = 1;
  p.kb_total = p.T * p.KC;
  p.kb_per_split = p.kb_total;
  p.out = out; p.out_mode = out_mode; p.out_pitch = out_pitch;
  p.bias = bias; p.act = lrelu; p.slope = slope;
  p.mask = reinterpret_cast<const __nv_bfloat16*>(mask);
  p.split_stride = 0;
  CUtensorMap ta, tb;
  int rc = make_act_tmap(&ta, act, N, h, w, Ck, act_pitch, p.TW, p.TH, op);
  if (rc) return rc;
  {
    const cuuint64_t es = (cuuint64_t)op_bytes(op);
    cuuint64_t gdim[3] = {(cuuint64_t)Ck, (cuuint64_t)Co, (cuuint64_t)p.T};
    cuuint64_t gstr[2] = {(cuuint64_t)Ck * es, (cuuint64_t)Ck * es * Co};
    cuuint32_t box[3] = {(cuuint32_t)op_kb(op), (cuuint32_t)(pair ? BN / 2 : BN), 1};
    rc = make_tmap_nd(&tb, wt, 3, gdim, gstr, box, op);
    if (rc) return rc;
  }
  profile_begin(prof_tag, stream);
  rc = launch_conv<MODE_CONV>(ta, tb, p, BN, pair, op, stream);
  profile_end(prof_tag, stream);
  return rc;
}

// rows of the fused column-sum partials: one per (M-tile, epilogue warp quarter)
static int conv3x3_colsum_rows(int N, int h, int w) {
  int TW = 64, TH = 1;
  pick_rect(h, w, BLOCK_M, &TW, &TH);
  return N * ceil_div(w, TW) * ceil_div(h, TH) * 4;
}

static int conv3x3_wgrad_splits(int N, int h, int w, int Co, int Ci) {
  int TW = 64, TH = 1;
  pick_rect(h, w, BLOCK_K, &TW, &TH);
  const int kb_total = N * ceil_div(w, TW) * ceil_div(h, TH);
  int mt = ceil_div(Co, BLOCK_M);
  const bool pair = g_pair && mt >= 2;
  if (pair) mt = ceil_div(mt, 2);
  const int units = 9 * mt * ceil_div(Ci, Ci <= 128 ? 128 : 256);
  int s = (pair ? num_sms() / 2 : num_sms()) / units;
  if (s < 1) s = 1;
  if (s > kb_total) s = kb_total;
  return s;
}

// slabs[z][t][Co][Ci] = sum over the pixels of split z of g[pixel, co] * x[pixel + d_t, ci].  The split count is planned on 64-pixel
// chunks for both operand types (OP_TF32 runs 32-pixel k-blocks: the same splits, twice the k-blocks each)
static int conv3x3_wgrad_run(const void* g, int Co, long long g_pitch, const void* x, int Ci, long long x_pitch, int N, int h, int w,
                             int dilation, int splits, float* slabs, int* splits_used, cudaStream_t stream, int prof_tag, int op) {
  B200SEG_CHECK_ARG(g && x && slabs, "conv3x3_wgrad: null pointer");
  B200SEG_CHECK_ARG(N > 0 && h > 0 && w > 0 && Co > 0 && Ci > 0 && dilation > 0, "conv3x3_wgrad: bad geometry");
  B200SEG_CHECK_ARG(g_pitch % 8 == 0 && x_pitch % 8 == 0 && Ci % 4 == 0 && x_pitch >= Ci, "conv3x3_wgrad: channel pitches must be multiples of 8");
  B200SEG_CHECK_ARG((reinterpret_cast<uintptr_t>(slabs) & 15) == 0, "conv3x3_wgrad: slabs must be 16-byte aligned");
  ConvParams p = {};
  p.N = N; p.h = h; p.w = w;
  pick_rect(h, w, op_kb(op), &p.TW, &p.TH);
  p.tw_shift = ilog2(p.TW);
  p.tiles_x = ceil_div(w, p.TW);
  p.tiles_y = ceil_div(h, p.TH);
  fill_taps(p, dilation, 1);
  p.KC = 0;
  p.Co = Co; p.Ci = Ci;
  const int BN = Ci <= 128 ? 128 : 256;
  p.m_tiles = ceil_div(Co, BLOCK_M);
  const bool pair = g_pair && p.m_tiles >= 2;
  if (pair) p.m_tiles = ceil_div(p.m_tiles, 2);
  p.n_tiles = ceil_div(Ci, BN);
  p.kb_total = N * p.tiles_x * p.tiles_y;
  if (splits < 1) splits = 1;
  if (splits > p.kb_total) splits = p.kb_total;
  p.kb_per_split = ceil_div(p.kb_total, splits);
  p.splits = ceil_div(p.kb_total, p.kb_per_split);
  p.units = p.splits * p.T * p.m_tiles * p.n_tiles;
  p.out = slabs; p.out_mode = 0; p.out_pitch = 0;
  p.split_stride = (long long)p.T * Co * Ci;
  if (splits_used) *splits_used = p.splits;
  CUtensorMap ta, tb;
  // the gradient map exposes min(g_pitch, ...) channels: the zero padding of a padded gradient tensor is harmless, channels
  // beyond the pitch are zero-filled by TMA
  int rc = make_act_tmap(&ta, g, N, h, w, (int)g_pitch, g_pitch, p.TW, p.TH, op, true);
  if (rc) return rc;
  rc = make_act_tmap(&tb, x, N, h, w, Ci, x_pitch, p.TW, p.TH, op, true);
  if (rc) return rc;
  profile_begin(prof_tag, stream);
  rc = launch_conv<MODE_WGRAD>(ta, tb, p, BN, pair, op, stream);
  profile_end(prof_tag, stream);
  return rc;
}

}  // namespace conv
}  // namespace gemm

// ------------------------------------------------------------------------------------------
// helper kernels
// ------------------------------------------------------------------------------------------
// w fp32 [Co_part][Ci][3][3] -> Wf bf16 [9][Co_total][Ci] (rows co0 + co) and Wb bf16 [9][Ci][co_pitch] (columns co0 + co);
// with TF32 the same layouts in fp32, every value rounded to TF32.
// ONE launch packs every weight tensor of a layer -- or of the whole discriminator stack -- from a job table in the kernel
// parameters (training re-packs every step: four launches + three memsets + a concatenation cost ~70 us of device time, mostly
// dependency latency between tiny nodes).  A block owns 16 output x 64 input channels of one job: 16 contiguous runs of 576 floats
// in (coalesced), then Wf as 128-byte runs along ci and Wb as 32-byte runs along co -- full sectors, shift/mask indexing only.
// The block of the first output tile of a layer's last part also zero-fills the padding columns [Co_total, co_pitch) of Wb, and
// block 0 concatenates the bias vectors of the last layer's parts.
constexpr int CPW_CO = 16, CPW_CI = 64, CPW_PITCH = CPW_CI * 9 + 1;      // odd pitch: the co-fastest reads are conflict-free
constexpr int CPW_MAX_JOBS = 8, CPW_MAX_BIAS = 4;
struct PackJob {
  const float* w;
  void* Wf;                // __nv_bfloat16, or float with TF32
  void* Wb;
  int Co_part, Ci, co0, Co_total, co_pitch, tiles_ci, tile0, zero_pad;
};
struct PackTable {
  PackJob job[CPW_MAX_JOBS];
  int n, total_tiles;
  const float* bias_src[CPW_MAX_BIAS];
  int bias_len[CPW_MAX_BIAS];
  int n_bias;
  float* bias_dst;
};
template <bool TF32>
__device__ __forceinline__ void pack_store(void* base, long long i, float v) {
  if (TF32) reinterpret_cast<float*>(base)[i] = tf32_rn(v);
  else reinterpret_cast<__nv_bfloat16*>(base)[i] = __float2bfloat16(v);
}
template <bool TF32>
__global__ void __launch_bounds__(256) conv_pack_weights_kernel(const PackTable t) {
  __shared__ float sm[CPW_CO * CPW_PITCH];
  if (blockIdx.x == 0 && t.bias_dst) {
    int off = 0;
#pragma unroll
    for (int i = 0; i < CPW_MAX_BIAS; ++i) {
      if (i < t.n_bias) {
        for (int e = threadIdx.x; e < t.bias_len[i]; e += 256) t.bias_dst[off + e] = t.bias_src[i] ? __ldg(t.bias_src[i] + e) : 0.f;
        off += t.bias_len[i];
      }
    }
  }
  PackJob j = t.job[0];
#pragma unroll
  for (int k = 1; k < CPW_MAX_JOBS; ++k)
    if (k < t.n && (int)blockIdx.x >= t.job[k].tile0) j = t.job[k];
  const int local = (int)blockIdx.x - j.tile0;
  const int ci0 = (local % j.tiles_ci) * CPW_CI, cop0 = (local / j.tiles_ci) * CPW_CO;
  const int nci = min(CPW_CI, j.Ci - ci0), nco = min(CPW_CO, j.Co_part - cop0);
  for (int co_l = 0; co_l < nco; ++co_l) {
    const float* src = j.w + ((long long)(cop0 + co_l) * j.Ci + ci0) * 9;
    for (int off = threadIdx.x; off < nci * 9; off += 256) sm[co_l * CPW_PITCH + off] = __ldg(src + off);
  }
  __syncthreads();
  if (j.Wf) {
    for (int i = threadIdx.x; i < 9 * CPW_CO * CPW_CI; i += 256) {         // ci fastest
      const int ci_l = i & (CPW_CI - 1), co_l = (i >> 6) & (CPW_CO - 1), k = i >> 10;
      if (ci_l < nci && co_l < nco)
        pack_store<TF32>(j.Wf, ((long long)k * j.Co_total + j.co0 + cop0 + co_l) * j.Ci + ci0 + ci_l, sm[co_l * CPW_PITCH + ci_l * 9 + k]);
    }
  }
  if (j.Wb) {
    for (int i = threadIdx.x; i < 9 * CPW_CI * CPW_CO; i += 256) {         // co fastest
      const int co_l = i & (CPW_CO - 1), ci_l = (i >> 4) & (CPW_CI - 1), k = i >> 10;
      if (ci_l < nci && co_l < nco)
        pack_store<TF32>(j.Wb, ((long long)k * j.Ci + ci0 + ci_l) * j.co_pitch + j.co0 + cop0 + co_l, sm[co_l * CPW_PITCH + ci_l * 9 + k]);
    }
    const int npad = j.co_pitch - j.Co_total;
    if (j.zero_pad && cop0 == 0 && npad > 0) {
      for (int i = threadIdx.x; i < 9 * nci * npad; i += 256) {
        const int c = i % npad, kc = i / npad, ci_l = kc % nci, k = kc / nci;
        pack_store<TF32>(j.Wb, ((long long)k * j.Ci + ci0 + ci_l) * j.co_pitch + j.Co_total + c, 0.f);
      }
    }
  }
}

// deterministic column sums of bf16 [P][pitch]: per-block partials, then a fixed-order final sum (bias gradients)
constexpr int COLSUM_BLOCKS = 296;
__global__ void __launch_bounds__(256) colsum_partial_kernel(const __nv_bfloat16* __restrict__ g, long long P, int pitch,
                                                             float* __restrict__ part) {
  __shared__ float2 red[256];
  const int pairs = pitch >> 1;                       // <= 256
  const int rp = 256 / pairs;                         // rows in flight per block
  const int cp = threadIdx.x % pairs, rr = threadIdx.x / pairs;
  float2 acc = make_float2(0.f, 0.f);
  if (rr < rp) {
    const long long rows_per_block = ceil_div_ll(P, gridDim.x);
    const long long r0 = blockIdx.x * rows_per_block, r1 = min(P, r0 + rows_per_block);
    for (long long r = r0 + rr; r < r1; r += rp) {
      const float2 v = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(g + r * pitch + 2 * cp));
      acc.x += v.x; acc.y += v.y;
    }
  }
  red[threadIdx.x] = acc;
  __syncthreads();
  if (rr == 0) {
    for (int k = 1; k < rp; ++k) { acc.x += red[k * pairs + cp].x; acc.y += red[k * pairs + cp].y; }
    part[(long long)blockIdx.x * pitch + 2 * cp] = acc.x;
    part[(long long)blockIdx.x * pitch + 2 * cp + 1] = acc.y;
  }
}
__global__ void __launch_bounds__(256) colsum_final_kernel(const float* __restrict__ part, int blocks, int pitch, int C,
                                                          float* __restrict__ out) {
  // one warp per channel; lane l sums partials l, l+32, ... in order, then a fixed shuffle tree: run-to-run identical
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  double s = 0.0;
  for (int b = lane; b < blocks; b += 32) s += (double)part[(long long)b * pitch + c];
  s = warp_sum_d(s);
  if (lane == 0) out[c] = (float)s;
}

// out[c] = sum over n, s of src[n][c][s] (fp32 NCHW): the bias gradient of the TF32 cls1 | cls2 layer straight from the unrounded
// loss gradient.  One block per channel, fixed order (per-thread strided sums, then a double warp / block tree): deterministic
__global__ void __launch_bounds__(256) nchw_channel_sum_kernel(const float* __restrict__ src, int N, int C, int hw, float* __restrict__ out) {
  __shared__ double red[8];
  const int c = blockIdx.x;
  float acc = 0.f;
  for (int n = 0; n < N; ++n) {
    const float* row = src + ((long long)n * C + c) * hw;
    for (int s = threadIdx.x; s < hw; s += 256) acc += __ldg(row + s);
  }
  double d = warp_sum_d((double)acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = d;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i];
    out[c] = (float)t;
  }
}

// bf16 [n] -> fp32 [n] (exact; n a multiple of 8, 16-byte aligned): seam-format features as the TF32 layers' operand
__global__ void __launch_bounds__(256) widen_bf16_kernel(const uint4* __restrict__ src, long long n8, float4* __restrict__ dst) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n8; i += (long long)gridDim.x * 256) {
    const uint4 q = __ldcs(src + i);
    const uint32_t wv[4] = {q.x, q.y, q.z, q.w};
    float f[8];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      f[2 * e] = __uint_as_float(wv[e] << 16);
      f[2 * e + 1] = __uint_as_float(wv[e] & 0xFFFF0000u);
    }
    dst[2 * i] = make_float4(f[0], f[1], f[2], f[3]);
    dst[2 * i + 1] = make_float4(f[4], f[5], f[6], f[7]);
  }
}

// split-K slabs [S][9][Co_total][Ci] -> gw [Co_part][Ci][3][3] for rows co0 .. co0 + Co_part
__global__ void __launch_bounds__(256) conv_wgrad_reduce_kernel(const float* __restrict__ part, int S, long long slab, int Co_total,
                                                                int Ci, int co0, float* __restrict__ gw) {
  __shared__ __align__(16) float sm[256 * 9];
  const int ci0 = blockIdx.x * 256;
  const int ci = ci0 + threadIdx.x;
  const int co = blockIdx.y;
  if (ci < Ci) {
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const long long off = ((long long)k * Co_total + co0 + co) * Ci + ci;
      float acc = 0.f;
      for (int s = 0; s < S; ++s) acc += __ldcs(part + s * slab + off);
      sm[threadIdx.x * 9 + k] = acc;
    }
  }
  __syncthreads();
  const int nci = min(256, Ci - ci0);
  float* dst = gw + ((long long)co * Ci + ci0) * 9;
  if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0 && (nci * 9) % 4 == 0) {
    for (int i = threadIdx.x; i < nci * 9 / 4; i += 256)
      reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(sm)[i];
  } else {
    for (int i = threadIdx.x; i < nci * 9; i += 256) dst[i] = sm[i];
  }
}

// the same reduction for small layers (everything L2-resident): one thread per output element, so a [19][128][3][3] gradient
// is 86 blocks of independent loads instead of 19 blocks each walking 9 x S dependent ones
__global__ void __launch_bounds__(256) conv_wgrad_reduce_flat_kernel(const float* __restrict__ part, int S, long long slab, int Co_total,
                                                                     int Co_part, int Ci, int co0, float* __restrict__ gw) {
  const int idx = blockIdx.x * 256 + threadIdx.x;
  if (idx >= Co_part * Ci * 9) return;
  const int k = idx % 9, rem = idx / 9;
  const int ci = rem % Ci, co = rem / Ci;
  const float* src = part + ((long long)k * Co_total + co0 + co) * Ci + ci;
  float acc = 0.f;
#pragma unroll 4
  for (int s = 0; s < S; ++s) acc += __ldg(src + s * slab);
  gw[idx] = acc;
}

// ------------------------------------------------------------------------------------------
// host entry points (wrapped 1:1 by api.cu)
// ------------------------------------------------------------------------------------------
static int pack_add_layer(PackTable& t, const float* const* weights, const int* part_co, int n_parts, int Ci, void* Wf, void* Wb,
                          int co_pitch) {
  B200SEG_CHECK_ARG(weights && part_co && n_parts >= 1 && (Wf || Wb) && Ci > 0, "conv3x3_pack_weights: bad arguments");
  B200SEG_CHECK_ARG(t.n + n_parts <= CPW_MAX_JOBS, "conv3x3_pack_weights: more than %d weight tensors in one call", CPW_MAX_JOBS);
  int Co_total = 0;
  for (int i = 0; i < n_parts; ++i) {
    B200SEG_CHECK_ARG(weights[i] && part_co[i] > 0, "conv3x3_pack_weights: part %d is null or empty", i);
    Co_total += part_co[i];
  }
  B200SEG_CHECK_ARG(!Wb || co_pitch >= Co_total, "conv3x3_pack_weights: co_pitch %d < total output channels %d", co_pitch, Co_total);
  int co0 = 0;
  for (int i = 0; i < n_parts; ++i) {
    PackJob& j = t.job[t.n++];
    j.w = weights[i]; j.Wf = Wf; j.Wb = Wb;
    j.Co_part = part_co[i]; j.Ci = Ci; j.co0 = co0; j.Co_total = Co_total; j.co_pitch = co_pitch;
    j.tiles_ci = ceil_div(Ci, CPW_CI);
    j.tile0 = t.total_tiles;
    j.zero_pad = (i == n_parts - 1) ? 1 : 0;
    t.total_tiles += j.tiles_ci * ceil_div(part_co[i], CPW_CO);
    co0 += part_co[i];
  }
  return B200SEG_OK;
}

static int pack_launch(const PackTable& t, cudaStream_t stream, bool tf32 = false) {
  if (tf32) conv_pack_weights_kernel<true><<<t.total_tiles, 256, 0, stream>>>(t);
  else conv_pack_weights_kernel<false><<<t.total_tiles, 256, 0, stream>>>(t);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// one layer; the padding columns [sum part_co, co_pitch) of Wb are zero-filled by the kernel
int conv3x3_pack_weights(const float* const* weights, const int* part_co, int n_parts, int Ci, void* Wf, void* Wb, int co_pitch,
                         cudaStream_t stream) {
  PackTable t = {};
  int rc = pack_add_layer(t, weights, part_co, n_parts, Ci, Wf, Wb, co_pitch);
  if (rc) return rc;
  return pack_launch(t, stream);
}

// a whole stack of layers in one launch: layer l owns parts [first, first + parts_per_layer[l]) of the flattened weights / part_co
// arrays; bias_parts (optional, n_bias <= 4 device pointers, NULL = zeros) are concatenated into bias_out
static int pack_weights_stack(int n_layers, const float* const* weights, const int* part_co, const int* parts_per_layer, const int* Ci,
                              void* const* Wf, void* const* Wb, const int* co_pitch, const float* const* bias_parts, const int* bias_len,
                              int n_bias, float* bias_out, cudaStream_t stream, bool tf32) {
  B200SEG_CHECK_ARG(n_layers >= 1 && weights && part_co && parts_per_layer && Ci && Wf && Wb && co_pitch,
                    "conv3x3_pack_weights_stack: bad arguments");
  B200SEG_CHECK_ARG(n_bias >= 0 && n_bias <= CPW_MAX_BIAS && (n_bias == 0 || (bias_parts && bias_len && bias_out)),
                    "conv3x3_pack_weights_stack: 0..%d bias parts with an output buffer", CPW_MAX_BIAS);
  PackTable t = {};
  int first = 0;
  for (int l = 0; l < n_layers; ++l) {
    int rc = pack_add_layer(t, weights + first, part_co + first, parts_per_layer[l], Ci[l], Wf[l], Wb[l], co_pitch[l]);
    if (rc) return rc;
    first += parts_per_layer[l];
  }
  t.n_bias = n_bias;
  t.bias_dst = n_bias ? bias_out : nullptr;
  for (int i = 0; i < n_bias; ++i) { t.bias_src[i] = bias_parts[i]; t.bias_len[i] = bias_len[i]; }
  return pack_launch(t, stream, tf32);
}

int conv3x3_pack_weights_stack(int n_layers, const float* const* weights, const int* part_co, const int* parts_per_layer,
                               const int* Ci, void* const* Wf, void* const* Wb, const int* co_pitch, const float* const* bias_parts,
                               const int* bias_len, int n_bias, float* bias_out, cudaStream_t stream) {
  return pack_weights_stack(n_layers, weights, part_co, parts_per_layer, Ci, Wf, Wb, co_pitch, bias_parts, bias_len, n_bias, bias_out,
                            stream, false);
}

// the same layouts in fp32, rounded to TF32: the operands of the TF32 layers
int conv3x3_pack_weights_stack_tf32(int n_layers, const float* const* weights, const int* part_co, const int* parts_per_layer,
                                    const int* Ci, void* const* Wf, void* const* Wb, const int* co_pitch, const float* const* bias_parts,
                                    const int* bias_len, int n_bias, float* bias_out, cudaStream_t stream) {
  return pack_weights_stack(n_layers, weights, part_co, parts_per_layer, Ci, Wf, Wb, co_pitch, bias_parts, bias_len, n_bias, bias_out,
                            stream, true);
}

int nchw_channel_sum(const float* src, int N, int C, int hw, float* out, cudaStream_t stream) {
  B200SEG_CHECK_ARG(src && out && N > 0 && C > 0 && hw > 0, "nchw_channel_sum: bad arguments");
  nchw_channel_sum_kernel<<<C, 256, 0, stream>>>(src, N, C, hw, out);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int widen_bf16(const void* src, long long n, float* dst, cudaStream_t stream) {
  B200SEG_CHECK_ARG(src && dst && n > 0 && n % 8 == 0 && (reinterpret_cast<uintptr_t>(src) & 15) == 0 &&
                        (reinterpret_cast<uintptr_t>(dst) & 15) == 0,
                    "widen_bf16: bad arguments (n a multiple of 8, 16-byte aligned buffers)");
  const long long n8 = n / 8;
  const long long blocks = ceil_div_ll(n8, 256);
  widen_bf16_kernel<<<(int)(blocks < 4L * num_sms() ? blocks : 4L * num_sms()), 256, 0, stream>>>(
      reinterpret_cast<const uint4*>(src), n8, reinterpret_cast<float4*>(dst));
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}


long long nhwc_colsum_scratch_bytes(int pitch) { return (long long)COLSUM_BLOCKS * pitch * 4; }

int nhwc_bf16_colsum(const void* g, long long P, int C, int pitch, void* scratch, float* out, cudaStream_t stream) {
  B200SEG_CHECK_ARG(g && scratch && out && P > 0 && C > 0 && pitch % 2 == 0 && pitch >= C && pitch <= 512,
                    "nhwc_bf16_colsum: bad arguments (pitch must be even and <= 512)");
  colsum_partial_kernel<<<COLSUM_BLOCKS, 256, 0, stream>>>((const __nv_bfloat16*)g, P, pitch, (float*)scratch);
  B200SEG_LAUNCH_CHECK();
  colsum_final_kernel<<<ceil_div(C, 8), 256, 0, stream>>>((const float*)scratch, COLSUM_BLOCKS, pitch, C, out);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

long long conv3x3_wgrad_scratch_bytes(int N, int h, int w, int Co, int Ci, int splits) {
  if (splits < 1) splits = gemm::conv::conv3x3_wgrad_splits(N, h, w, Co, Ci);
  return (long long)splits * 9 * Co * Ci * 4 + 256;
}

int conv3x3_wgrad(const void* g, int Co, long long g_pitch, const void* x, int Ci, long long x_pitch, int N, int h, int w, int dilation,
                  int splits, void* scratch, long long scratch_bytes, float* const* grad_w, const int* part_co, int n_parts,
                  cudaStream_t stream, int tf32) {
  B200SEG_CHECK_ARG(grad_w && part_co && n_parts >= 1 && scratch, "conv3x3_wgrad: bad arguments");
  int Co_total = 0;
  for (int i = 0; i < n_parts; ++i) Co_total += part_co[i];
  B200SEG_CHECK_ARG(Co_total == Co, "conv3x3_wgrad: parts sum to %d output channels, expected %d", Co_total, Co);
  if (splits < 1) splits = gemm::conv::conv3x3_wgrad_splits(N, h, w, Co, Ci);
  B200SEG_CHECK_ARG(scratch_bytes >= (long long)splits * 9 * Co * Ci * 4, "conv3x3_wgrad: scratch too small");
  int used = 1;
  int rc = gemm::conv::conv3x3_wgrad_run(g, Co, g_pitch, x, Ci, x_pitch, N, h, w, dilation, splits, (float*)scratch, &used, stream, 14,
                                         tf32 ? gemm::conv::OP_TF32 : gemm::conv::OP_BF16);
  if (rc) return rc;
  int co0 = 0;
  for (int i = 0; i < n_parts; ++i) {
    if (grad_w[i]) {
      if ((long long)part_co[i] * Ci * 9 <= (1 << 20)) {
        conv_wgrad_reduce_flat_kernel<<<ceil_div(part_co[i] * Ci * 9, 256), 256, 0, stream>>>((const float*)scratch, used,
                                                                                              (long long)9 * Co * Ci, Co, part_co[i], Ci, co0, grad_w[i]);
      } else {
        dim3 grid(ceil_div(Ci, 256), part_co[i]);
        conv_wgrad_reduce_kernel<<<grid, 256, 0, stream>>>((const float*)scratch, used, (long long)9 * Co * Ci, Co, Ci, co0, grad_w[i]);
      }
      B200SEG_LAUNCH_CHECK();
    }
    co0 += part_co[i];
  }
  return B200SEG_OK;
}

int conv3x3_forward(const void* act, int N, int h, int w, int Ck, long long act_pitch, const void* Wf, int Co, int dilation,
                    const float* bias, int lrelu, float slope, void* out_nhwc, long long out_pitch, float* out_f32_nchw,
                    cudaStream_t stream, int tf32) {
  using namespace gemm::conv;
  B200SEG_CHECK_ARG((out_nhwc != nullptr) != (out_f32_nchw != nullptr), "conv3x3_forward: give exactly one output");
  const int op = tf32 ? OP_TF32 : OP_BF16;
  if (out_nhwc)
    return conv3x3_run(act, N, h, w, Ck, act_pitch, Wf, Co, dilation, 1, bias, lrelu, slope, nullptr, out_nhwc,
                       tf32 ? OUT_F32_NHWC : OUT_BF16_NHWC, out_pitch, stream, 12, nullptr, op);
  return conv3x3_run(act, N, h, w, Ck, act_pitch, Wf, Co, dilation, 1, bias, lrelu, slope, nullptr, out_f32_nchw, OUT_F32_NCHW, 0,
                     stream, 12, nullptr, op);
}

// data gradient: gin[pixel, ci] = (sum_t sum_co g[pixel - d_t, co] * Wb[t][ci][co]) * LeakyReLU'(mask[pixel, ci])
long long conv3x3_dgrad_colsum_scratch_bytes(int N, int h, int w, long long out_pitch) {
  return (long long)gemm::conv::conv3x3_colsum_rows(N, h, w) * out_pitch * 4;
}

// colsum_out (optional, with colsum_scratch): fp32 [Ci] column sums of the NHWC gradient = the bias gradient of the layer below,
// accumulated in the GEMM epilogue (per M-tile and warp quarter) and finished by one small fixed-order reduction: the sums of the
// stored bf16 values, or with tf32 of the fp32 values before their TF32 rounding.  With tf32 the NHWC output (out_nhwc, and the
// mask) is fp32, and out_bf16_nhwc is the bf16 NHWC output of the same fp32 result (no mask, no column sums).
int conv3x3_dgrad(const void* g, int N, int h, int w, int Cg, long long g_pitch, const void* Wb, int Ci, int dilation, const void* mask,
                  float slope, void* out_nhwc, long long out_pitch, float* out_f32_nchw, cudaStream_t stream,
                  void* colsum_scratch, long long colsum_scratch_bytes, float* colsum_out, int tf32, void* out_bf16_nhwc) {
  using namespace gemm::conv;
  B200SEG_CHECK_ARG((out_nhwc != nullptr) + (out_f32_nchw != nullptr) + (out_bf16_nhwc != nullptr) == 1,
                    "conv3x3_dgrad: give exactly one output");
  B200SEG_CHECK_ARG(!out_bf16_nhwc || (tf32 && !mask && !colsum_out), "conv3x3_dgrad: the bf16 output of the TF32 layers takes no mask or sums");
  B200SEG_CHECK_ARG(!mask || out_nhwc, "conv3x3_dgrad: the activation mask needs the NHWC output");
  const int op = tf32 ? OP_TF32 : OP_BF16;
  const int nhwc_mode = tf32 ? OUT_F32_NHWC : OUT_BF16_NHWC;
  if (colsum_out) {
    B200SEG_CHECK_ARG(out_nhwc && colsum_scratch, "conv3x3_dgrad: fused column sums need the NHWC output and a scratch buffer");
    B200SEG_CHECK_ARG(colsum_scratch_bytes >= conv3x3_dgrad_colsum_scratch_bytes(N, h, w, out_pitch), "conv3x3_dgrad: column-sum scratch too small");
    int rc = conv3x3_run(g, N, h, w, Cg, g_pitch, Wb, Ci, dilation, -1, nullptr, 0, slope, mask, out_nhwc, nhwc_mode, out_pitch, stream, 13,
                         (float*)colsum_scratch, op);
    if (rc) return rc;
    colsum_final_kernel<<<ceil_div(Ci, 8), 256, 0, stream>>>((const float*)colsum_scratch, conv3x3_colsum_rows(N, h, w), (int)out_pitch,
                                                            Ci, colsum_out);
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  if (out_nhwc)
    return conv3x3_run(g, N, h, w, Cg, g_pitch, Wb, Ci, dilation, -1, nullptr, 0, slope, mask, out_nhwc, nhwc_mode, out_pitch, stream, 13,
                       nullptr, op);
  if (out_bf16_nhwc)
    return conv3x3_run(g, N, h, w, Cg, g_pitch, Wb, Ci, dilation, -1, nullptr, 0, slope, nullptr, out_bf16_nhwc, OUT_BF16_NHWC, out_pitch,
                       stream, 13, nullptr, op);
  return conv3x3_run(g, N, h, w, Cg, g_pitch, Wb, Ci, dilation, -1, nullptr, 0, slope, nullptr, out_f32_nchw, OUT_F32_NCHW, 0, stream, 13,
                     nullptr, op);
}

}  // namespace b200seg
