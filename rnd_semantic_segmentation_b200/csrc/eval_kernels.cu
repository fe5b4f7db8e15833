// K4: align-corners bilinear upsample -> argmax of the softmax probabilities -> C x C confusion
// matrix, in ONE streaming pass that never materialises the full-resolution logits.
//
// Replaces, for one frame (reference file:line):
//   F.interpolate(..., bilinear, align_corners=True)      core/utils/utility.py:185
//   F.softmax(dim=1)                                      core/utils/utility.py:186
//   output.max(1)[1]                                      core/testers/aspp_tester.py:63
//   confusion_matrix(cfg, pd, gt)   (per-pixel Python loop) core/utils/utility.py:347-359
//   intersectionAndUnionGPU(...)    (3x CPU histc)         core/utils/utility.py:148-161  [= diag/row/col sums]
//
// Bit-exactness: the upsampled value uses ATen's expression form
//   h0*(w0*a + w1*b) + h1*(w0*c + w1*d)   (ATen/native/cuda/UpSampleBilinear2d.cu)
// as nvcc contracts it, fma(h0, t, h1*u), and argmax(softmax(v)) == first-max(v) unless another class is within
// ~1 ulp of the maximum after exp/divide; pixels where a second class lies within 1e-6 of the maximum re-run
// ATen's exact spatial-softmax sequence (max, sum of expf(v-max) in class order, expf(v-max)/sum, first maximum).
//
// Layout / mapping: one thread per output column, warps walk rows (row taps are warp-uniform); the horizontal
// lerps of all classes for the two source rows live in registers as class PAIRS and are reused for every output
// row of the same source-row pair.  The kernel is issue-bound (C classes per 8-byte label), so the per-pixel
// instruction count is what is optimised:
//   * interpolation on packed fp32x2 (FMUL2 + FFMA2: two classes per issue slot, each half IEEE-rounded),
//   * max over classes as a tree of 3-input FMNMX3,
//   * argmax + near-tie detection in one pass: bit c of a mask is set when v_c >= max - 1e-6 (FSETP + predicated
//     add, all independent); one bit set -> that is the argmax, several -> the exact path.
// Labels (int64, the only large stream) are staged by per-lane 8-byte cp.async into a per-warp shared-memory ring,
// one 8-row strip ahead (also across tiles), so no registers or issue slots are held by loads in flight.
// Histogram: each lane owns private uint8 counters hist[bin][lane] in shared memory (no atomics, no contention
// even for i.i.d. labels), folded with dp4a into an int32 CTA histogram before a counter could overflow and into
// the int64 global matrix once per frame per CTA.
#include "common.cuh"
#include "host_api.h"

namespace b200seg {

// build-time experiment knobs (profiles/build_variants.sh)
#ifndef K4_MIN_CTAS
#define K4_MIN_CTAS 3          // resident CTAs per SM the register allocation is bounded for
#endif
#ifndef K4_PAIR_ROWS
#define K4_PAIR_ROWS 1         // 1: two output rows per loop iteration (interleaved dependency chains)
#endif
#ifndef K4_FORCE_ATOMIC_HIST
#define K4_FORCE_ATOMIC_HIST 0 // 1: warp-aggregated shared-memory atomics instead of per-lane uint8 counters
#endif

constexpr int K4_THREADS = 128;
constexpr int K4_WARPS = K4_THREADS / 32;
constexpr int K4_TILE_W = 128;
constexpr int K4_STRIP = 8;                  // rows per label-ring stage
constexpr int K4_TILE_H_MAX = 32;            // rows per tile: 8, 16 or 32 (chosen per launch; one table row per lane)
constexpr int K4_SPAN = 8;                   // source columns a warp's 32 output columns may span on the staged path
constexpr float K4_NEAR_TIE = 1e-6f;
constexpr float K4_PAD = -1e30f;             // value of the padding classes (never wins, never NaN)
constexpr int K4_RING_BYTES = K4_WARPS * 2 * K4_STRIP * 32 * 8;
constexpr int K4_TAB_BYTES = K4_WARPS * K4_TILE_H_MAX * 16;
constexpr int K4_STAGE_FLOATS = 32 * K4_SPAN;   // per-warp staging buffer of one source row: [CT <= 32][K4_SPAN]
constexpr int K4_STAGE_BYTES = K4_WARPS * K4_STAGE_FLOATS * 4;
// per-lane uint8 counters need CT*CT*32 bytes per warp; above 48 KB per CTA fall back to warp-aggregated atomics
__host__ __device__ constexpr bool k4_use_u8(int CT) { return !K4_FORCE_ATOMIC_HIST && (CT * CT + 1) * 32 * K4_WARPS <= 48 * 1024; }

constexpr int K4_MAX_FRAMES = 16;            // frames per launch (each with its own logits / labels / pred pointers)
struct K4Params {
  const float* logits[K4_MAX_FRAMES];   // per frame [C, h, w]
  const void* labels[K4_MAX_FRAMES];    // per frame [H, W] int64 or uint8 (LU8), or all null
  void* pred[K4_MAX_FRAMES];            // per frame [H, W] int64 or uint8 (pred_u8), or all null
  long long* cm;            // [C, C] (+ frame * cm_frame_stride) or null
  int has_labels, has_pred, pred_u8;
  int N, C, h, w, H, W;
  int ignore_index;
  long long cm_frame_stride;
  float scale_h, scale_w;
  int tiles_x, tiles_y, total_tiles;
  int tile_h;               // rows per tile (multiple of K4_STRIP, <= K4_TILE_H_MAX)
};

// wa*a + wb*b with the rounding sequence selected by FMA:
//   0/1: fma(wa, a, wb*b)  -- what nvcc emits for ATen's source expression (bit-equal to F.interpolate on B200)
//   2:   fma(wb, b, wa*a)     3: (wa*a) + (wb*b) without contraction          (diagnostic variants)
template <int FMA>
__device__ __forceinline__ float lerp1(float wa, float a, float wb, float b) {
  if (FMA <= 1) return fmaf(wa, a, __fmul_rn(wb, b));
  if (FMA == 2) return fmaf(wb, b, __fmul_rn(wa, a));
  return __fadd_rn(__fmul_rn(wa, a), __fmul_rn(wb, b));
}
template <int FMA>
__device__ __forceinline__ float2 lerp2(float2 wa, float2 a, float2 wb, float2 b) {
  if (FMA <= 1) return fma2(wa, a, mul2(wb, b));
  if (FMA == 2) return fma2(wb, b, mul2(wa, a));
  return add2(mul2(wa, a), mul2(wb, b));
}

// Exact ATen spatial-softmax sequence for one pixel (rare path, recomputed from the L1/L2-resident low-res logits so
// the hot loop keeps no register array alive for it): sequential float sum of expf(v - max) in class order, IEEE
// divide, first maximum.
template <int FMA>
__device__ __noinline__ int k4_exact_softmax_argmax(const float* __restrict__ lg, int C, long long hw, int w, int row_top,
                                                    int row_bot, int i0, int i1, float l0, float l1, float h0, float h1) {
  const float* pt = lg + (long long)row_top * w;
  const float* pb = lg + (long long)row_bot * w;
  float m = -INFINITY;
  for (int c = 0; c < C; ++c) {
    const float t = lerp1<FMA>(l0, __ldg(pt + c * hw + i0), l1, __ldg(pt + c * hw + i1));
    const float u = lerp1<FMA>(l0, __ldg(pb + c * hw + i0), l1, __ldg(pb + c * hw + i1));
    m = fmaxf(m, lerp1<FMA>(h0, t, h1, u));
  }
  float s = 0.f;
  for (int c = 0; c < C; ++c) {
    const float t = lerp1<FMA>(l0, __ldg(pt + c * hw + i0), l1, __ldg(pt + c * hw + i1));
    const float u = lerp1<FMA>(l0, __ldg(pb + c * hw + i0), l1, __ldg(pb + c * hw + i1));
    s += expf(lerp1<FMA>(h0, t, h1, u) - m);
  }
  float pbest = -1.f;
  int idx = 0;
  for (int c = 0; c < C; ++c) {
    const float t = lerp1<FMA>(l0, __ldg(pt + c * hw + i0), l1, __ldg(pt + c * hw + i1));
    const float u = lerp1<FMA>(l0, __ldg(pb + c * hw + i0), l1, __ldg(pb + c * hw + i1));
    const float pc = expf(lerp1<FMA>(h0, t, h1, u) - m) / s;
    if (pc > pbest) { pbest = pc; idx = c; }
  }
  return idx;
}

// acc += K when v >= thr, as FSETP + one predicated add
template <int K>
__device__ __forceinline__ void add_if_ge(int& acc, float v, float thr) {
  asm("{ .reg .pred q; setp.ge.f32 q, %1, %2; @q add.s32 %0, %0, %3; }" : "+r"(acc) : "f"(v), "f"(thr), "n"(K));
}
template <int c, int CT, bool EXACT, int NF>
__device__ __forceinline__ void k4_candidates(int (&acc)[4], const float (&f)[NF], float thr, int C) {
  if constexpr (c < CT) {
    if (EXACT || c < C) add_if_ge<256 + c>(acc[c & 3], f[c], thr);
    k4_candidates<c + 1, CT, EXACT>(acc, f, thr, C);
  }
}

// Candidate accumulator of one pixel: adds (256 + c) for every class c whose interpolated logit is within 1e-6 of
// the maximum.  Exactly one candidate -> the result is argmax(softmax) in [0, C); none (NaN) or several (near tie)
// -> the result is outside [0, C) and the caller takes the exact path.  FSETP + predicated add per class, all
// independent except four short add chains; no transcendental-pipe (POPC/FLO) work.
template <int CT, int FMA, bool EXACT>
__device__ __forceinline__ int k4_pixel_candidate(const float2 (&top)[(CT + 1) / 2], const float2 (&bot)[(CT + 1) / 2], int C,
                                                  float h0, float h1) {
  constexpr int NP = (CT + 1) / 2;
  const float2 H0 = make_float2(h0, h0), H1 = make_float2(h1, h1);
  float f[2 * NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    const float2 v = lerp2<FMA>(H0, top[i], H1, bot[i]);
    f[2 * i] = v.x; f[2 * i + 1] = v.y;
  }
  const float thr = tree_max3<0, CT, 2 * NP>(f) - K4_NEAR_TIE;
  int acc[4] = {-256, 0, 0, 0};                      // four short predicated-add chains instead of two long ones
  k4_candidates<0, CT, EXACT>(acc, f, thr, C);
  return (acc[0] + acc[1]) + (acc[2] + acc[3]);
}

// ---- source rows --------------------------------------------------------------------------------------------
// Staged path (the warp's 32 columns span <= K4_SPAN source columns, i.e. any upsampling factor >= ~5.3): the warp
// copies the CT x K4_SPAN window of a source row into its shared-memory stage with <= CT*K4_SPAN/32 coalesced
// loads per lane (32-bit element offsets `soff`, fixed per tile) -- k4_row_fetch issues them (one segment ahead, so
// their latency hides behind a segment of compute), k4_row_commit parks them in the stage -- and every lane then
// reads its two taps per class with immediate-offset LDS: no per-load 64-bit address arithmetic.
template <int CT>
__device__ __forceinline__ void k4_row_fetch(float (&v)[(CT * K4_SPAN + 31) / 32], const float* __restrict__ rb,
                                             const int (&soff)[(CT * K4_SPAN + 31) / 32]) {
  constexpr int NS = (CT * K4_SPAN + 31) / 32;
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int q = 0; q < NS; ++q)
    if (q * 32 + lane < CT * K4_SPAN) v[q] = __ldg(rb + soff[q]);
}

template <int CT, int FMA, bool EXACT>
__device__ __forceinline__ void k4_row_commit(float2 (&dst)[(CT + 1) / 2], const float (&v)[(CT * K4_SPAN + 31) / 32], int C,
                                              unsigned stage_s, unsigned t0_s, unsigned t1_s, float l0, float l1) {
  constexpr int NP = (CT + 1) / 2;
  constexpr int NS = (CT * K4_SPAN + 31) / 32;
  const int lane = threadIdx.x & 31;
  __syncwarp();                                     // every lane has finished reading the previous row from the stage
#pragma unroll
  for (int q = 0; q < NS; ++q)
    if (q * 32 + lane < CT * K4_SPAN) sts_f32(stage_s + (q * 32 + lane) * 4, v[q]);
  __syncwarp();
  const float2 L0 = make_float2(l0, l0), L1 = make_float2(l1, l1);
#pragma unroll
  for (int i = 0; i < NP; ++i) {
    float2 a = make_float2(K4_PAD, K4_PAD), b = make_float2(K4_PAD, K4_PAD);
    if (EXACT || 2 * i < C) { a.x = lds_f32(t0_s + (2 * i) * K4_SPAN * 4); b.x = lds_f32(t1_s + (2 * i) * K4_SPAN * 4); }
    if (2 * i + 1 < CT && (EXACT || 2 * i + 1 < C)) {
      a.y = lds_f32(t0_s + (2 * i + 1) * K4_SPAN * 4); b.y = lds_f32(t1_s + (2 * i + 1) * K4_SPAN * 4);
    }
    dst[i] = lerp2<FMA>(L0, a, L1, b);
    if (!(EXACT || 2 * i < C)) dst[i].x = K4_PAD;
    if (!(2 * i + 1 < CT && (EXACT || 2 * i + 1 < C))) dst[i].y = K4_PAD;
  }
}

// Fallback for windows wider than K4_SPAN (mild or no upsampling): direct global loads.
template <int CT, int FMA, bool EXACT>
__device__ __forceinline__ void k4_row_direct(float2 (&dst)[(CT + 1) / 2], const float* __restrict__ rb, int C, long long hw,
                                              int i0, int i1, float l0, float l1) {
  constexpr int NP = (CT + 1) / 2;
  const char* p0 = reinterpret_cast<const char*>(rb + i0);
  const char* p1 = reinterpret_cast<const char*>(rb + i1);
  const long long step = hw * 4;
  const float2 L0 = make_float2(l0, l0), L1 = make_float2(l1, l1);
#pragma unroll 1
  for (int i = 0; i < NP; ++i) {
    float2 a = make_float2(K4_PAD, K4_PAD), b = make_float2(K4_PAD, K4_PAD);
    if (EXACT || 2 * i < C) { a.x = __ldg(reinterpret_cast<const float*>(p0)); b.x = __ldg(reinterpret_cast<const float*>(p1)); }
    p0 += step; p1 += step;
    if (2 * i + 1 < CT && (EXACT || 2 * i + 1 < C)) {
      a.y = __ldg(reinterpret_cast<const float*>(p0)); b.y = __ldg(reinterpret_cast<const float*>(p1));
    }
    p0 += step; p1 += step;
    float2 r = lerp2<FMA>(L0, a, L1, b);
    if (!(EXACT || 2 * i < C)) r.x = K4_PAD;
    if (!(2 * i + 1 < CT && (EXACT || 2 * i + 1 < C))) r.y = K4_PAD;
    // dynamic index into a register array would spill: select with an unrolled compare instead
#pragma unroll
    for (int j = 0; j < NP; ++j)
      if (j == i) dst[j] = r;
  }
}

struct K4RowCtx {
  const float* lg;          // frame base of the low-res logits
  char* pred;               // this lane's prediction column (row 0 of the frame; int64 or uint8 elements) or null
  int pred_u8;
  int* cta_hist;
  long long hw;
  unsigned tab_s;           // shared address of this warp's row table: {l0, l1, bits(i0), bits(segment end)} per tile row
  unsigned lab_s;           // shared address of this lane's label column in the current ring stage (row stride 256 B; 32 B for uint8)
  unsigned whist_s;         // shared address of this lane's uint8 counters (+ bin * 32)
  unsigned ign32;           // ignore_index when it fits a non-negative 32-bit value, else 0xffffffff (never a class)
  unsigned c_lim;           // number of classes for a lane inside the image, 0 for a lane right of it (never counts)
  int C, w, W, y_tile, y_strip;
  int i0x, i1x;
  float l0x, l1x;
  bool xvalid, do_cm;
};

// one output pixel: argmax class -> prediction store / histogram update (branch-free on the common path)
template <int CT, int FMA, bool EXACT, bool U8, bool LU8>
__device__ __forceinline__ void k4_finish_pixel(const K4RowCtx& k, int y, int cand, int i0y, int i1y, float h0, float h1) {
  const int C = EXACT ? CT : k.C;
  int idx = cand;
  if ((unsigned)cand >= (unsigned)C)                                 // near tie (or NaN): the exact sequence
    idx = k4_exact_softmax_argmax<FMA>(k.lg, C, k.hw, k.w, i0y, i1y, k.i0x, k.i1x, k.l0x, k.l1x, h0, h1);
  if (k.pred != nullptr) {                                           // uniform
    if (k.xvalid) {
      if (k.pred_u8) reinterpret_cast<uint8_t*>(k.pred)[(long long)y * k.W] = (uint8_t)idx;
      else reinterpret_cast<long long*>(k.pred)[(long long)y * k.W] = (long long)idx;
    }
  }
  if (k.do_cm) {                                                     // uniform
    uint2 g;
    if (LU8) g = make_uint2(lds_u8(k.lab_s + (y - k.y_strip) * 32), 0u);
    else g = lds_v2u32(k.lab_s + (y - k.y_strip) * 256);             // int64 label as {lo, hi}
    const bool count = (g.y == 0u) && (g.x < k.c_lim) && (g.x != k.ign32);
    if (U8) {
      const int bin = count ? (int)g.x * C + idx : C * C;            // pixels that do not count land in a spare bin
      smem_inc_u8(k.whist_s + bin * 32);
    } else {
      const int bin = count ? (int)g.x * C + idx : -1;
      const unsigned peers = __match_any_sync(__activemask(), bin);
      if (count && (threadIdx.x & 31) == (__ffs(peers) - 1)) atomicAdd(&k.cta_hist[bin], __popc(peers));
    }
  }
}

// rows [y, yend) of one source-row pair (top, bot), two rows per iteration so the two dependency chains interleave
template <int CT, int FMA, bool EXACT, bool U8, bool LU8>
__device__ __forceinline__ void k4_rows(const K4RowCtx& k, const float2 (&top)[(CT + 1) / 2], const float2 (&bot)[(CT + 1) / 2],
                                        int y, int yend, int i0y, int i1y) {
  unsigned ts = k.tab_s + (y - k.y_tile) * 16;
#pragma unroll 1
  for (; K4_PAIR_ROWS && y + 1 < yend; y += 2, ts += 32) {
    const float4 ta = lds_v4f32(ts), tb = lds_v4f32(ts + 16);
    const int ca = k4_pixel_candidate<CT, FMA, EXACT>(top, bot, k.C, ta.x, ta.y);
    const int cb = k4_pixel_candidate<CT, FMA, EXACT>(top, bot, k.C, tb.x, tb.y);
    k4_finish_pixel<CT, FMA, EXACT, U8, LU8>(k, y, ca, i0y, i1y, ta.x, ta.y);
    k4_finish_pixel<CT, FMA, EXACT, U8, LU8>(k, y + 1, cb, i0y, i1y, tb.x, tb.y);
  }
#pragma unroll 1
  for (; y < yend; ++y, ts += 16) {
    const float4 ta = lds_v4f32(ts);
    const int ca = k4_pixel_candidate<CT, FMA, EXACT>(top, bot, k.C, ta.x, ta.y);
    k4_finish_pixel<CT, FMA, EXACT, U8, LU8>(k, y, ca, i0y, i1y, ta.x, ta.y);
  }
}

// LU8: the labels are uint8 (what the dataloader holds, core/datasets/transform.py:31-33, before the tester's .long()):
// each lane loads its 8 label bytes of the NEXT strip into registers with plain 1-byte loads (a warp row is one 32-byte
// sector) and parks them in a lane-private shared-memory column at the start of that strip -- the dependent store is a whole
// strip of compute after the load, so the load latency is hidden exactly as the cp.async ring hides it for int64 labels.
template <int CT, int FMA, bool EXACT, bool LU8>
__global__ void __launch_bounds__(K4_THREADS, K4_MIN_CTAS) k4_upsample_argmax_confusion(const __grid_constant__ K4Params p) {
  constexpr int NP = (CT + 1) / 2;
  constexpr int NS = (CT * K4_SPAN + 31) / 32;
  constexpr bool U8 = k4_use_u8(CT);
  extern __shared__ __align__(16) uint8_t k4_smem[];
  const int C = EXACT ? CT : p.C, CC = C * C;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // smem: label ring [warps][2][STRIP][32] i64 | row table [warps][TILE_H_MAX] float4 | row stage [warps][32*SPAN] f32 |
  //       CTA histogram [CC] i32 | per-warp uint8 counters [CC + 1][32]   (bin CC = pixels that do not count)
  const unsigned ring_s = LU8 ? smem_u32(k4_smem) + warp * (K4_STRIP * 32) + lane
                              : smem_u32(k4_smem) + (warp * (2 * K4_STRIP * 32) + lane) * 8;
  float4* tab = reinterpret_cast<float4*>(k4_smem + K4_RING_BYTES) + warp * K4_TILE_H_MAX;
  const unsigned stage_s = smem_u32(k4_smem + K4_RING_BYTES + K4_TAB_BYTES) + warp * K4_STAGE_FLOATS * 4;
  int* cta_hist = reinterpret_cast<int*>(k4_smem + K4_RING_BYTES + K4_TAB_BYTES + K4_STAGE_BYTES);
  const int hist_off = K4_RING_BYTES + K4_TAB_BYTES + K4_STAGE_BYTES + ((CC * 4 + 15) / 16) * 16;
  const int warp_hist_bytes = (CC + 1) * 32;
  uint8_t* whist = k4_smem + hist_off + warp * warp_hist_bytes;           // [CC + 1][32] uint8, this warp's
  const bool do_cm = (p.cm != nullptr) && p.has_labels;

  if (do_cm) {
    for (int i = threadIdx.x; i < CC; i += K4_THREADS) cta_hist[i] = 0;
    if (U8) {
      int4* z = reinterpret_cast<int4*>(whist);
      for (int i = lane; i < warp_hist_bytes / 16; i += 32) z[i] = make_int4(0, 0, 0, 0);
    }
  }
  __syncthreads();

  const int tiles_per_frame = p.tiles_x * p.tiles_y;
  const int strips_per_tile = p.tile_h / K4_STRIP;
  const long long hw = (long long)p.h * p.w;
  const long long HW = (long long)p.H * p.W;
  const long long row_bytes = (long long)p.W * (LU8 ? 1 : 8);
  unsigned nb[LU8 ? K4_STRIP : 1];               // LU8: the label bytes of the strip in flight (one per row)

  // label staging, one strip (K4_STRIP rows of this lane's column) per commit group.  (pf_tile, pf_st) is the strip
  // that goes in flight next; pf_src its first label; pf_rows how many of its rows exist.
  int pf_tile = blockIdx.x, pf_st = 0, pf_stage = 0;
  const char* pf_src = nullptr;
  int pf_rows = 0;
  auto pf_setup_tile = [&]() {                   // first strip of tile pf_tile
    pf_rows = 0;
    if (do_cm && pf_tile < p.total_tiles) {
      const int n = pf_tile / tiles_per_frame;
      const int trem = pf_tile - n * tiles_per_frame;
      const int ty = trem / p.tiles_x;
      const int tx = trem - ty * p.tiles_x;
      const int x = tx * K4_TILE_W + threadIdx.x;
      const int y0 = ty * p.tile_h;
      pf_src = reinterpret_cast<const char*>(p.labels[n]) + ((long long)y0 * p.W + min(x, p.W - 1)) * (LU8 ? 1 : 8);
      pf_rows = (x < p.W) ? min(p.tile_h, p.H - y0) : 0;
    }
  };
  auto issue_strip = [&]() {
    const unsigned dst = ring_s + pf_stage * (K4_STRIP * 256);
    const char* src = pf_src;
#pragma unroll
    for (int r = 0; r < K4_STRIP; ++r) {
      if constexpr (LU8) {
        nb[r] = (r < pf_rows) ? (unsigned)__ldg(reinterpret_cast<const unsigned char*>(src)) : 0xffu;
      } else {
        if (r < pf_rows) cp_async_8s(dst + r * 256, src);
      }
      src += row_bytes;
    }
    if constexpr (!LU8) cp_async_commit();
    pf_src = src;
    pf_rows -= K4_STRIP;
    pf_stage ^= 1;
    if (++pf_st == strips_per_tile) { pf_st = 0; pf_tile += gridDim.x; pf_setup_tile(); }
  };

  // fold this warp's uint8 counters into the CTA histogram and clear them
  auto fold_warp_hist = [&]() {
    __syncwarp();
    uint4* wh = reinterpret_cast<uint4*>(whist);
    for (int b = lane; b < CC; b += 32) {
      const uint4 a = wh[b * 2], c4 = wh[b * 2 + 1];
      if ((a.x | a.y | a.z | a.w | c4.x | c4.y | c4.z | c4.w) != 0u) {
        unsigned sum = 0;
        sum = __dp4a(a.x, 0x01010101u, sum); sum = __dp4a(a.y, 0x01010101u, sum);
        sum = __dp4a(a.z, 0x01010101u, sum); sum = __dp4a(a.w, 0x01010101u, sum);
        sum = __dp4a(c4.x, 0x01010101u, sum); sum = __dp4a(c4.y, 0x01010101u, sum);
        sum = __dp4a(c4.z, 0x01010101u, sum); sum = __dp4a(c4.w, 0x01010101u, sum);
        atomicAdd(&cta_hist[b], (int)sum);
        wh[b * 2] = make_uint4(0, 0, 0, 0);
        wh[b * 2 + 1] = make_uint4(0, 0, 0, 0);
      }
    }
    __syncwarp();
  };

  K4RowCtx k;
  k.cta_hist = cta_hist;
  k.whist_s = smem_u32(whist) + lane;
  k.hw = hw;
  k.ign32 = (p.ignore_index >= 0) ? (unsigned)p.ignore_index : 0xffffffffu;
  k.C = C; k.w = p.w; k.W = p.W;
  k.pred_u8 = p.pred_u8;
  k.tab_s = smem_u32(tab);
  k.do_cm = do_cm;

  int cur_frame = -1;
  int rows_since_fold = 0;                       // rows counted into the uint8 counters since the last fold (<= 255)
  int cur_stage = 0;
  pf_setup_tile();
  issue_strip();

  for (int tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
    const int n = tile / tiles_per_frame;
    const int trem = tile - n * tiles_per_frame;
    const int ty = trem / p.tiles_x;
    const int tx = trem - ty * p.tiles_x;
    const int fkey = p.cm_frame_stride ? n : 0;   // one shared matrix: publish once, at the end

    if (do_cm && fkey != cur_frame) {        // frame boundary: publish this CTA's counts for the finished frame
      if (cur_frame >= 0) {
        if (U8) { fold_warp_hist(); rows_since_fold = 0; }
        __syncthreads();
        long long* dst = p.cm + (long long)cur_frame * p.cm_frame_stride;
        for (int i = threadIdx.x; i < CC; i += K4_THREADS) {
          const int v = cta_hist[i];
          if (v) atomicAdd(reinterpret_cast<unsigned long long*>(dst + i), (unsigned long long)v);
          cta_hist[i] = 0;
        }
        __syncthreads();
      }
      cur_frame = fkey;
    }

    const int x = tx * K4_TILE_W + threadIdx.x;
    const Tap tapx = ac_tap(p.scale_w, x < p.W ? x : p.W - 1, p.w);
    const int y_begin = ty * p.tile_h;
    const int y_tile_end = min(p.H, y_begin + p.tile_h);
    k.xvalid = x < p.W;
    k.c_lim = k.xvalid ? (unsigned)C : 0u;
    k.i0x = tapx.i0; k.i1x = tapx.i1; k.l0x = tapx.l0; k.l1x = tapx.l1;
    k.lg = p.logits[n];
    k.pred = p.has_pred ? reinterpret_cast<char*>(p.pred[n]) + (long long)x * (p.pred_u8 ? 1 : 8) : nullptr;
    k.y_tile = y_begin;

    // per-warp row table of the tile: vertical taps and, per row, the end of its run of rows sharing one source-row pair
    __syncwarp();
    {
      const int yy = min(y_begin + lane, p.H - 1);
      const Tap t = ac_tap(p.scale_h, yy, p.h);
      const int nxt = __shfl_down_sync(0xffffffffu, t.i0, 1);
      const bool last = (lane == 31) || (y_begin + lane >= y_tile_end - 1) || (nxt != t.i0);
      const unsigned ends = __ballot_sync(0xffffffffu, last);
      const int seg_end = y_begin + lane + __ffs(ends >> lane);            // one past the last row of this row's run
      tab[lane] = make_float4(t.l0, t.l1, __int_as_float(t.i0), __int_as_float(seg_end));
    }
    // staged row loads: window of K4_SPAN source columns starting at lane 0's left tap
    const int j_lo = __shfl_sync(0xffffffffu, tapx.i0, 0);
    const int j_hi = __shfl_sync(0xffffffffu, tapx.i1, 31);
    const bool staged = (j_hi - j_lo) < K4_SPAN;
    int soff[NS];
#pragma unroll
    for (int q = 0; q < NS; ++q) {
      const int e = q * 32 + lane;
      const int c = min(e / K4_SPAN, C - 1);
      soff[q] = c * (int)hw + min(j_lo + (e % K4_SPAN), p.w - 1);
    }
    const unsigned t0_s = stage_s + (tapx.i0 - j_lo) * 4, t1_s = stage_s + (tapx.i1 - j_lo) * 4;
    __syncwarp();

    // a0 / a1 hold the horizontally interpolated logits of two source rows; a0_top says which one is the upper row.
    float2 a0[NP], a1[NP];
    float pre[NS];                             // staged path: the window of source row `pre_row`, fetched one segment ahead
    int row_a0 = -1, row_a1 = -1, pre_row = -1;
    bool a0_top = true;

#pragma unroll 1
    for (int ys = y_begin; ys < y_begin + p.tile_h; ys += K4_STRIP) {
      if constexpr (LU8) {
#pragma unroll
        for (int r = 0; r < K4_STRIP; ++r) sts_u8(ring_s + r * 32, nb[r]);     // this strip's bytes (loaded a strip ago)
        issue_strip();                         // next strip's loads go in flight
        k.lab_s = ring_s;
      } else {
        issue_strip();                         // next strip (possibly of the next tile) goes in flight
        cp_async_wait<1>();                    // this strip has landed (each lane reads back only its own column)
        k.lab_s = ring_s + cur_stage * (K4_STRIP * 256);
        cur_stage ^= 1;
      }
      if (do_cm && U8 && rows_since_fold + K4_STRIP > 255) { fold_warp_hist(); rows_since_fold = 0; }
      rows_since_fold += K4_STRIP;
      const int ye = min(p.H, ys + K4_STRIP);
      k.y_strip = ys;
      int y = ys;
#pragma unroll 1
      while (y < ye) {
        const float4 t = lds_v4f32(k.tab_s + (y - y_begin) * 16);
        const int i0 = __float_as_int(t.z);
        const int i1 = i0 + ((i0 < p.h - 1) ? 1 : 0);
        const int yend = min(__float_as_int(t.w), ye);
        const int top = a0_top ? row_a0 : row_a1, bot = a0_top ? row_a1 : row_a0;
        if (i0 != top || i1 != bot) {                                    // new source-row pair (warp-uniform)
          bool need_top = false;
          if (i0 == bot && i0 != top) a0_top = !a0_top;                  // the old lower row becomes the upper row
          else if (i0 != top) need_top = true;                           // unrelated pair: load the upper row too
#pragma unroll 1
          for (int which = need_top ? 0 : 1; which < 2; ++which) {       // ONE inlined copy of the row loader
            const int row = which ? i1 : i0;
            const bool into_a0 = (which == 0) == a0_top;
            if ((into_a0 ? row_a0 : row_a1) == row) continue;
            const float* rb = k.lg + (long long)row * p.w;
            if (staged) {
              if (pre_row != row) k4_row_fetch<CT>(pre, rb, soff);
              pre_row = -1;
              if (into_a0) k4_row_commit<CT, FMA, EXACT>(a0, pre, C, stage_s, t0_s, t1_s, k.l0x, k.l1x);
              else         k4_row_commit<CT, FMA, EXACT>(a1, pre, C, stage_s, t0_s, t1_s, k.l0x, k.l1x);
            } else {
              if (into_a0) k4_row_direct<CT, FMA, EXACT>(a0, rb, C, hw, k.i0x, k.i1x, k.l0x, k.l1x);
              else         k4_row_direct<CT, FMA, EXACT>(a1, rb, C, hw, k.i0x, k.i1x, k.l0x, k.l1x);
            }
            if (into_a0) row_a0 = row; else row_a1 = row;
          }
          if (staged && i1 + 1 < p.h) {                                  // the next segment's lower row goes in flight now
            pre_row = i1 + 1;
            k4_row_fetch<CT>(pre, k.lg + (long long)pre_row * p.w, soff);
          }
        }
        if (a0_top) k4_rows<CT, FMA, EXACT, U8, LU8>(k, a0, a1, y, yend, i0, i1);
        else        k4_rows<CT, FMA, EXACT, U8, LU8>(k, a1, a0, y, yend, i0, i1);
        y = yend;
      }
    }
  }
  if constexpr (!LU8) cp_async_wait<0>();
  (void)HW;

  if (do_cm && cur_frame >= 0) {
    if (U8) fold_warp_hist();
    __syncthreads();
    long long* dst = p.cm + (long long)cur_frame * p.cm_frame_stride;
    for (int i = threadIdx.x; i < CC; i += K4_THREADS) {
      const int v = cta_hist[i];
      if (v) atomicAdd(reinterpret_cast<unsigned long long*>(dst + i), (unsigned long long)v);
    }
  }
}

template <int CT, int FMA, bool EXACT, bool LU8>
static int k4_launch_t(const K4Params& p, int grid, size_t smem, cudaStream_t stream) {
  static bool configured = false;
  if (!configured) {
    B200SEG_CUDA(cudaFuncSetAttribute(k4_upsample_argmax_confusion<CT, FMA, EXACT, LU8>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                      100 * 1024));
    configured = true;
  }
  profile_begin(7, stream);
  k4_upsample_argmax_confusion<CT, FMA, EXACT, LU8><<<grid, K4_THREADS, smem, stream>>>(p);
  profile_end(7, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

template <int CT, bool EXACT>
static int k4_launch_c(const K4Params& p, int fma_mode, bool lu8, int grid, size_t smem, cudaStream_t stream) {
  if (lu8) return k4_launch_t<CT, 1, EXACT, true>(p, grid, smem, stream);       // diagnostic FMA variants: int64 labels only
  switch (fma_mode) {
    case 0:
    case 1: return k4_launch_t<CT, 1, EXACT, false>(p, grid, smem, stream);
    case 2: return k4_launch_t<CT, 2, EXACT, false>(p, grid, smem, stream);
    default: return k4_launch_t<CT, 3, EXACT, false>(p, grid, smem, stream);
  }
}

// frames: n_frames low-res logit maps [C,h,w] (device pointers in a HOST array), each with its own label map [H,W]
// (int64 or uint8: label_bytes 8 / 1) and optional prediction map (pred_bytes 8 / 1).  More than K4_MAX_FRAMES frames are
// processed in consecutive launches of K4_MAX_FRAMES.
int k4_launch_frames(const float* const* logits, int n_frames, int C, int h, int w, const void* const* labels, int label_bytes,
                     int H, int W, int ignore_index, long long* cm, long long cm_frame_stride, void* const* pred, int pred_bytes,
                     int fma_mode, cudaStream_t stream) {
  B200SEG_CHECK_ARG(logits != nullptr, "upsample_argmax_confusion: logits is null");
  B200SEG_CHECK_ARG(n_frames > 0 && C > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_argmax_confusion: bad shape N=%d C=%d h=%d w=%d H=%d W=%d", n_frames, C, h, w, H, W);
  B200SEG_CHECK_ARG(C <= 32, "upsample_argmax_confusion: num_classes=%d > 32 is not supported", C);
  B200SEG_CHECK_ARG(cm == nullptr || labels != nullptr, "upsample_argmax_confusion: confusion matrix requested without labels");
  B200SEG_CHECK_ARG(cm != nullptr || pred != nullptr, "upsample_argmax_confusion: nothing to compute (cm and pred both null)");
  B200SEG_CHECK_ARG(labels == nullptr || label_bytes == 8 || label_bytes == 1, "upsample_argmax_confusion: labels must be int64 or uint8 (label_bytes=%d)", label_bytes);
  B200SEG_CHECK_ARG(pred == nullptr || pred_bytes == 8 || pred_bytes == 1, "upsample_argmax_confusion: pred must be int64 or uint8 (pred_bytes=%d)", pred_bytes);
  for (int f0 = 0; f0 < n_frames; f0 += K4_MAX_FRAMES) {
    const int N = (n_frames - f0 < K4_MAX_FRAMES) ? n_frames - f0 : K4_MAX_FRAMES;
    K4Params p;
    for (int i = 0; i < K4_MAX_FRAMES; ++i) {
      const int f = f0 + (i < N ? i : 0);
      p.logits[i] = logits[f];
      p.labels[i] = labels ? labels[f] : nullptr;
      p.pred[i] = pred ? pred[f] : nullptr;
      B200SEG_CHECK_ARG(p.logits[i] != nullptr && (!labels || p.labels[i]) && (!pred || p.pred[i]), "upsample_argmax_confusion: null frame pointer (frame %d)", f);
    }
    p.cm = cm ? cm + (long long)f0 * cm_frame_stride : nullptr;
    p.has_labels = labels != nullptr; p.has_pred = pred != nullptr; p.pred_u8 = (pred_bytes == 1);
    p.N = N; p.C = C; p.h = h; p.w = w; p.H = H; p.W = W;
    p.ignore_index = ignore_index;
    p.cm_frame_stride = cm_frame_stride;
    p.scale_h = ac_scale(h, H);
    p.scale_w = ac_scale(w, W);
    p.tiles_x = ceil_div(W, K4_TILE_W);
    // tile height: as tall as possible (fewer source-row loads per output row) while the launch still has >= 4 tiles per
    // resident CTA, so the static round-robin schedule stays balanced
    const int max_ctas = num_sms() * K4_MIN_CTAS;
    p.tile_h = K4_TILE_H_MAX;
    while (p.tile_h > K4_STRIP && (long long)N * p.tiles_x * ceil_div(H, p.tile_h) < 4LL * max_ctas) p.tile_h /= 2;
    p.tiles_y = ceil_div(H, p.tile_h);
    p.total_tiles = N * p.tiles_x * p.tiles_y;
    const int CC = C * C;
    const int CT = (C == 2) ? 2 : (C == 19) ? 19 : (C <= 8) ? 8 : 32;
    const size_t smem = (size_t)K4_RING_BYTES + K4_TAB_BYTES + K4_STAGE_BYTES + ((CC * 4 + 15) / 16) * 16 +
                        (k4_use_u8(CT) ? (size_t)K4_WARPS * ((CC + 1) * 32) : 0);
    const int grid = p.total_tiles < max_ctas ? p.total_tiles : max_ctas;
    const bool lu8 = labels != nullptr && label_bytes == 1;
    int rc;
    if (C == 2) rc = k4_launch_c<2, true>(p, fma_mode, lu8, grid, smem, stream);
    else if (C == 19) rc = k4_launch_c<19, true>(p, fma_mode, lu8, grid, smem, stream);
    else if (C <= 8) rc = k4_launch_c<8, false>(p, fma_mode, lu8, grid, smem, stream);
    else rc = k4_launch_c<32, false>(p, fma_mode, lu8, grid, smem, stream);
    if (rc) return rc;
  }
  return B200SEG_OK;
}

// contiguous batch [N,C,h,w] / [N,H,W]: the frame pointers are derived here
int k4_launch(const float* logits, int N, int C, int h, int w, const void* labels, int label_bytes, int H, int W, int ignore_index,
              long long* cm, long long cm_frame_stride, void* pred, int pred_bytes, int fma_mode, cudaStream_t stream) {
  B200SEG_CHECK_ARG(logits != nullptr, "upsample_argmax_confusion: logits is null");
  B200SEG_CHECK_ARG(N > 0 && C > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_argmax_confusion: bad shape N=%d C=%d h=%d w=%d H=%d W=%d", N, C, h, w, H, W);
  for (int f0 = 0; f0 < N; f0 += K4_MAX_FRAMES) {
    const int n = (N - f0 < K4_MAX_FRAMES) ? N - f0 : K4_MAX_FRAMES;
    const float* lg[K4_MAX_FRAMES];
    const void* lb[K4_MAX_FRAMES];
    void* pr[K4_MAX_FRAMES];
    for (int i = 0; i < n; ++i) {
      const long long f = f0 + i;
      lg[i] = logits + f * C * h * w;
      lb[i] = labels ? reinterpret_cast<const char*>(labels) + f * H * W * label_bytes : nullptr;
      pr[i] = pred ? reinterpret_cast<char*>(pred) + f * H * W * pred_bytes : nullptr;
    }
    const int rc = k4_launch_frames(lg, n, C, h, w, labels ? lb : nullptr, label_bytes, H, W, ignore_index,
                                    cm ? cm + f0 * cm_frame_stride : nullptr, cm_frame_stride, pred ? pr : nullptr, pred_bytes,
                                    fma_mode, stream);
    if (rc) return rc;
  }
  return B200SEG_OK;
}

// ---------------------------------------------------------------------------------------------
// API-compat: confusion matrix / IoU areas from an already-materialised prediction map
// (confusion_matrix(cfg, pd, gt) utility.py:347-359 and intersectionAndUnionGPU utility.py:148-161,
//  which also overwrites output[target == ignore] = ignore in place).
// ---------------------------------------------------------------------------------------------
template <typename PdT, typename GtT>
__global__ void __launch_bounds__(256) confusion_pairs_kernel(PdT* pd, const GtT* gt, long long n, int C,
                                                              int ignore_index, int mutate_pd, long long* cm) {
  extern __shared__ int cp_hist[];
  const int CC = C * C;
  for (int i = threadIdx.x; i < CC; i += blockDim.x) cp_hist[i] = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const long long stride = (long long)gridDim.x * blockDim.x;
  const long long n_round = ceil_div_ll(n, 32) * 32;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < n_round; i += stride) {
    int bin = -1;
    if (i < n) {
      const long long g = (long long)gt[i];
      const long long q = (long long)pd[i];
      if (g == ignore_index) {
        if (mutate_pd) pd[i] = (PdT)ignore_index;
      } else if (g >= 0 && g < C && q >= 0 && q < C) {
        bin = (int)g * C + (int)q;
      }
    }
    const unsigned peers = __match_any_sync(0xffffffffu, bin);
    if (bin >= 0 && lane == (__ffs(peers) - 1)) atomicAdd(&cp_hist[bin], __popc(peers));
  }
  __syncthreads();
  for (int i = threadIdx.x; i < CC; i += blockDim.x) {
    const int v = cp_hist[i];
    if (v) atomicAdd(reinterpret_cast<unsigned long long*>(cm + i), (unsigned long long)v);
  }
}

// Same histogram with K4's per-lane uint8 counters (no atomics, no match.any) and 16-byte loads (two int64 per load):
// used when the counters fit shared memory (C <= 19) and the maps are 16-byte aligned.
constexpr int CP_THREADS = 128;
__global__ void __launch_bounds__(CP_THREADS) confusion_pairs_u8_kernel(long long* pd, const long long* gt, long long n, int C,
                                                                        int ignore_index, int mutate_pd, long long* cm) {
  extern __shared__ __align__(16) uint8_t cp_smem[];
  const int CC = C * C;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* cta_hist = reinterpret_cast<int*>(cp_smem);
  const int hist_off = ((CC * 4 + 15) / 16) * 16;
  uint8_t* whist = cp_smem + hist_off + warp * ((CC + 1) * 32);
  for (int i = threadIdx.x; i < CC; i += CP_THREADS) cta_hist[i] = 0;
  {
    int4* z = reinterpret_cast<int4*>(whist);
    for (int i = lane; i < (CC + 1) * 2; i += 32) z[i] = make_int4(0, 0, 0, 0);
  }
  __syncthreads();
  const unsigned whist_s = smem_u32(whist) + lane;
  const unsigned ign32 = ignore_index >= 0 ? (unsigned)ignore_index : 0xffffffffu;
  const long long ign = ignore_index;

  auto fold = [&]() {
    __syncwarp();
    uint4* wh = reinterpret_cast<uint4*>(whist);
    for (int b = lane; b < CC; b += 32) {
      const uint4 a = wh[b * 2], c4 = wh[b * 2 + 1];
      if ((a.x | a.y | a.z | a.w | c4.x | c4.y | c4.z | c4.w) != 0u) {
        unsigned sum = 0;
        sum = __dp4a(a.x, 0x01010101u, sum); sum = __dp4a(a.y, 0x01010101u, sum);
        sum = __dp4a(a.z, 0x01010101u, sum); sum = __dp4a(a.w, 0x01010101u, sum);
        sum = __dp4a(c4.x, 0x01010101u, sum); sum = __dp4a(c4.y, 0x01010101u, sum);
        sum = __dp4a(c4.z, 0x01010101u, sum); sum = __dp4a(c4.w, 0x01010101u, sum);
        atomicAdd(&cta_hist[b], (int)sum);
        wh[b * 2] = make_uint4(0, 0, 0, 0);
        wh[b * 2 + 1] = make_uint4(0, 0, 0, 0);
      }
    }
    __syncwarp();
  };

  const long long pairs = n >> 1;
  int since_fold = 0;                                   // increments per lane since the last fold (<= 255)
  // block-uniform trip count (the in-loop fold synchronises the warp); CP_U pair-loads of each map in flight per thread
  constexpr int CP_U = 4;
  for (long long base = blockIdx.x * (long long)(CP_THREADS * CP_U); base < pairs + 1; base += (long long)gridDim.x * (CP_THREADS * CP_U)) {
    int4 qv[CP_U], gv[CP_U];
#pragma unroll
    for (int u = 0; u < CP_U; ++u) {
      const long long i2 = base + u * CP_THREADS + threadIdx.x;
      if (i2 < pairs) { qv[u] = ld_stream_v4(pd + 2 * i2); gv[u] = ld_stream_v4(gt + 2 * i2); }
    }
#pragma unroll
    for (int u = 0; u < CP_U; ++u) {
      const long long i2 = base + u * CP_THREADS + threadIdx.x;
      long long q[2] = {-1, -1}, g[2] = {-1, -1};
      int cnt = 0;
      if (i2 < pairs) {
        q[0] = ((long long)(unsigned)qv[u].x) | ((long long)qv[u].y << 32); q[1] = ((long long)(unsigned)qv[u].z) | ((long long)qv[u].w << 32);
        g[0] = ((long long)(unsigned)gv[u].x) | ((long long)gv[u].y << 32); g[1] = ((long long)(unsigned)gv[u].z) | ((long long)gv[u].w << 32);
        cnt = 2;
      } else if (i2 == pairs && (n & 1)) {               // odd tail element
        q[0] = pd[n - 1]; g[0] = gt[n - 1];
        cnt = 1;
      }
#pragma unroll
      for (int e = 0; e < 2; ++e)
        if (e < cnt) {
          const bool is_ign = g[e] == ign;
          if (is_ign && mutate_pd) pd[(i2 < pairs ? 2 * i2 : n - 1) + e] = ign;
          const bool valid = !is_ign && (unsigned long long)g[e] < (unsigned long long)C && (unsigned long long)q[e] < (unsigned long long)C;
          const int bin = valid ? (int)g[e] * C + (int)q[e] : CC;
          smem_inc_u8(whist_s + bin * 32);
        }
    }
    since_fold += 2 * CP_U;
    if (since_fold > 255 - 2 * CP_U) { fold(); since_fold = 0; }
  }
  fold();
  __syncthreads();
  for (int i = threadIdx.x; i < CC; i += CP_THREADS) {
    const int v = cta_hist[i];
    if (v) atomicAdd(reinterpret_cast<unsigned long long*>(cm + i), (unsigned long long)v);
  }
  (void)ign32;
}

// Mixed element widths (uint8 / int64 prediction and truth maps, SURVEY 8f rank 2: the label tensor the dataloader already has,
// core/datasets/transform.py:31-33, and uint8 pseudo-label maps): 8 consecutive elements per thread per step -- one 8-byte load
// of a uint8 map, four 16-byte loads of an int64 map -- and the same per-lane uint8 counters.
template <typename T>
__device__ __forceinline__ void cp_load8(const T* __restrict__ p, long long i, long long n, bool aligned, long long (&v)[8]) {
  if constexpr (sizeof(T) == 1) {
    if (aligned && i + 8 <= n) {
      const uint2 r = *reinterpret_cast<const uint2*>(p + i);
#pragma unroll
      for (int e = 0; e < 4; ++e) { v[e] = (r.x >> (8 * e)) & 0xffu; v[4 + e] = (r.y >> (8 * e)) & 0xffu; }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = (i + e < n) ? (long long)p[i + e] : -1;
    }
  } else {
    if (aligned && i + 8 <= n) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int4 r = ld_stream_v4(p + i + 2 * e);
        v[2 * e] = ((long long)(unsigned)r.x) | ((long long)r.y << 32);
        v[2 * e + 1] = ((long long)(unsigned)r.z) | ((long long)r.w << 32);
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) v[e] = (i + e < n) ? (long long)p[i + e] : -1;
    }
  }
}

template <typename PdT, typename GtT>
__global__ void __launch_bounds__(CP_THREADS) confusion_pairs_any_kernel(PdT* pd, const GtT* gt, long long n, int C, int ignore_index,
                                                                         int mutate_pd, long long* cm, int aligned) {
  extern __shared__ __align__(16) uint8_t cp_smem[];
  const int CC = C * C;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int* cta_hist = reinterpret_cast<int*>(cp_smem);
  const int hist_off = ((CC * 4 + 15) / 16) * 16;
  uint8_t* whist = cp_smem + hist_off + warp * ((CC + 1) * 32);
  for (int i = threadIdx.x; i < CC; i += CP_THREADS) cta_hist[i] = 0;
  {
    int4* z = reinterpret_cast<int4*>(whist);
    for (int i = lane; i < (CC + 1) * 2; i += 32) z[i] = make_int4(0, 0, 0, 0);
  }
  __syncthreads();
  const unsigned whist_s = smem_u32(whist) + lane;
  const long long ign = ignore_index;
  auto fold = [&]() {
    __syncwarp();
    uint4* wh = reinterpret_cast<uint4*>(whist);
    for (int b = lane; b < CC; b += 32) {
      const uint4 a = wh[b * 2], c4 = wh[b * 2 + 1];
      if ((a.x | a.y | a.z | a.w | c4.x | c4.y | c4.z | c4.w) != 0u) {
        unsigned sum = 0;
        sum = __dp4a(a.x, 0x01010101u, sum); sum = __dp4a(a.y, 0x01010101u, sum);
        sum = __dp4a(a.z, 0x01010101u, sum); sum = __dp4a(a.w, 0x01010101u, sum);
        sum = __dp4a(c4.x, 0x01010101u, sum); sum = __dp4a(c4.y, 0x01010101u, sum);
        sum = __dp4a(c4.z, 0x01010101u, sum); sum = __dp4a(c4.w, 0x01010101u, sum);
        atomicAdd(&cta_hist[b], (int)sum);
        wh[b * 2] = make_uint4(0, 0, 0, 0);
        wh[b * 2 + 1] = make_uint4(0, 0, 0, 0);
      }
    }
    __syncwarp();
  };
  const long long groups = ceil_div_ll(n, 8);
  int since_fold = 0;
  // block-uniform trip count (the in-loop fold synchronises the warp)
  for (long long gbase = blockIdx.x * (long long)CP_THREADS; gbase < groups; gbase += (long long)gridDim.x * CP_THREADS) {
    const long long i = (gbase + threadIdx.x) * 8;
    long long q[8], g[8];
    if (i < n) {
      cp_load8<PdT>(pd, i, n, aligned != 0, q);
      cp_load8<GtT>(gt, i, n, aligned != 0, g);
#pragma unroll
      for (int e = 0; e < 8; ++e)
        if (i + e < n) {
          const bool is_ign = g[e] == ign;
          if (is_ign && mutate_pd) pd[i + e] = (PdT)ign;
          const bool valid = !is_ign && (unsigned long long)g[e] < (unsigned long long)C && (unsigned long long)q[e] < (unsigned long long)C;
          const int bin = valid ? (int)g[e] * C + (int)q[e] : CC;
          smem_inc_u8(whist_s + bin * 32);
        }
    }
    since_fold += 8;
    if (since_fold > 255 - 8) { fold(); since_fold = 0; }
  }
  fold();
  __syncthreads();
  for (int i = threadIdx.x; i < CC; i += CP_THREADS) {
    const int v = cta_hist[i];
    if (v) atomicAdd(reinterpret_cast<unsigned long long*>(cm + i), (unsigned long long)v);
  }
}

template <typename PdT, typename GtT>
static int confusion_pairs_any_launch(PdT* pd, const GtT* gt, long long n, int C, int ignore_index, int mutate_pd, long long* cm,
                                      cudaStream_t stream) {
  const int CC = C * C;
  const size_t smem_u8 = ((CC * 4 + 15) / 16) * 16 + (size_t)(CP_THREADS / 32) * (CC + 1) * 32;
  if (smem_u8 > 48 * 1024) {                      // counters do not fit: warp-aggregated shared atomics
    B200SEG_CHECK_ARG(C <= 104, "confusion_from_pred: num_classes=%d unsupported (1..104)", C);
    long long blocks = ceil_div_ll(n, 256 * 8);
    const long long cap = (long long)num_sms() * 8;
    if (blocks > cap) blocks = cap;
    confusion_pairs_kernel<PdT, GtT><<<(unsigned)blocks, 256, CC * sizeof(int), stream>>>(pd, gt, n, C, ignore_index, mutate_pd, cm);
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  const int aligned = ((reinterpret_cast<uintptr_t>(pd) | reinterpret_cast<uintptr_t>(gt)) & 15) == 0;
  long long blocks = ceil_div_ll(ceil_div_ll(n, 8), CP_THREADS * 4);
  const long long capu = (long long)num_sms() * 4;
  if (blocks > capu) blocks = capu;
  if (blocks < 1) blocks = 1;
  confusion_pairs_any_kernel<PdT, GtT><<<(unsigned)blocks, CP_THREADS, smem_u8, stream>>>(pd, gt, n, C, ignore_index, mutate_pd, cm, aligned);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

static int confusion_pairs_launch(long long* pd, const long long* gt, long long n, int C, int ignore_index, int mutate_pd,
                           long long* cm, cudaStream_t stream) {
  B200SEG_CHECK_ARG(pd && gt && cm, "confusion_from_pred: null pointer");
  B200SEG_CHECK_ARG(C > 0 && C <= 104, "confusion_from_pred: num_classes=%d unsupported (1..104)", C);
  if (n <= 0) return B200SEG_OK;
  const int CC = C * C;
  const size_t smem_u8 = ((CC * 4 + 15) / 16) * 16 + (size_t)(CP_THREADS / 32) * (CC + 1) * 32;
  if (smem_u8 <= 48 * 1024 && ((reinterpret_cast<uintptr_t>(pd) | reinterpret_cast<uintptr_t>(gt)) & 15) == 0) {
    long long blocks = ceil_div_ll((n >> 1) + 1, CP_THREADS * 4 * 4);
    const long long capu = (long long)num_sms() * 4;
    if (blocks > capu) blocks = capu;
    confusion_pairs_u8_kernel<<<(unsigned)blocks, CP_THREADS, smem_u8, stream>>>(pd, gt, n, C, ignore_index, mutate_pd, cm);
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  long long blocks = ceil_div_ll(n, 256 * 8);
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  confusion_pairs_kernel<long long, long long><<<(unsigned)blocks, 256, C * C * sizeof(int), stream>>>(pd, gt, n, C, ignore_index, mutate_pd, cm);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int confusion_pairs_launch_ex(void* pd, int pd_bytes, const void* gt, int gt_bytes, long long n, int C, int ignore_index, int mutate_pd,
                              long long* cm, cudaStream_t stream) {
  B200SEG_CHECK_ARG(pd && gt && cm, "confusion_from_pred: null pointer");
  B200SEG_CHECK_ARG((pd_bytes == 1 || pd_bytes == 8) && (gt_bytes == 1 || gt_bytes == 8), "confusion_from_pred: maps must be int64 or uint8");
  B200SEG_CHECK_ARG(C > 0, "confusion_from_pred: bad num_classes");
  if (n <= 0) return B200SEG_OK;
  if (pd_bytes == 8 && gt_bytes == 8)
    return confusion_pairs_launch(reinterpret_cast<long long*>(pd), reinterpret_cast<const long long*>(gt), n, C, ignore_index, mutate_pd, cm, stream);
  if (pd_bytes == 1 && gt_bytes == 1)
    return confusion_pairs_any_launch(reinterpret_cast<uint8_t*>(pd), reinterpret_cast<const uint8_t*>(gt), n, C, ignore_index, mutate_pd, cm, stream);
  if (pd_bytes == 8)
    return confusion_pairs_any_launch(reinterpret_cast<long long*>(pd), reinterpret_cast<const uint8_t*>(gt), n, C, ignore_index, mutate_pd, cm, stream);
  return confusion_pairs_any_launch(reinterpret_cast<uint8_t*>(pd), reinterpret_cast<const long long*>(gt), n, C, ignore_index, mutate_pd, cm, stream);
}

}  // namespace b200seg
