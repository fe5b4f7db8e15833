// K7: test-time augmentation (horizontal flip and/or multi-scale) fused with the argmax and the confusion matrix.
//
// Replaces, for one frame (reference file:line):
//   inference(..., flip=True)          core/utils/utility.py:179-191   (output[0] + output[1].flip(2)) / 2
//   multi_scale_inference(...)         core/utils/utility.py:193-209   sum over scales (and flips) of inference(flip=False),
//                                                                      then / len(scales) [/ 2]
//   output.max(1)[1]                   core/testers/aspp_tester.py:63
//   output.argmax(0) (pseudo labels)   core/testers/aspp_tester.py:42  (save_distill)
//   confusion_matrix / intersectionAndUnionGPU                          utility.py:347-359, 148-161
//
// The reference materialises, per member of the ensemble, the upsampled logits and their softmax at label resolution
// (2 x 159 MB at 19 x 1024 x 2048) plus the flipped copy and the running sum.  Here every label pixel reads the (L1/L2
// resident) low-res logits of all members, computes each member's softmax probabilities in registers, sums them in the
// reference's order and scales them -- nothing at label resolution is written unless the caller asks for the probabilities.
//
// Bit-exactness: unlike K4 the argmax here depends on the probabilities themselves, so EVERY pixel runs ATen's sequences:
//   upsample   h0*(w0*a + w1*b) + h1*(w0*c + w1*d) as nvcc contracts it, fma(h0, t, h1*u)      (UpSampleBilinear2d.cu)
//   softmax    max over classes; fp32 sum of expf(v - max) in class order; expf(v - max) / sum (IEEE) (SoftMax.cu, spatial);
//              the 19 IEEE divisions by the same sum share one reciprocal (tta_div: identical results, 3 instructions each)
//   sum        fp32 adds in member order
//   division   tensor / python_scalar on CUDA multiplies by the fp32 reciprocal of the scalar     (BinaryDivTrueKernel.cu);
//              div_exact = 1 selects the IEEE division ATen's CPU kernel performs instead
//   argmax     first maximum
//
// Mapping: one thread per label pixel; a CTA owns a run of consecutive rows of one 128-column strip (consecutive rows share
// source rows, which stay in L1).  Confusion counts go to a shared-memory int32 histogram (atomics), published once per CTA.
#include "common.cuh"
#include "host_api.h"

namespace b200seg {

constexpr int TTA_MAX_MAPS = 8;
constexpr int TTA_THREADS = 128;

struct TtaMap {
  const float* logits;     // [C, h, w]
  int h, w, flip;
  float scale_h, scale_w;
};
struct TtaParams {
  TtaMap maps[TTA_MAX_MAPS];
  int n_maps, C, H, W, ignore_index;
  int n_div;               // 0, 1 or 2 scalar divisions after the sum
  int div_exact;           // 0: multiply by the fp32 reciprocal (ATen CUDA), 1: IEEE divide (ATen CPU)
  float div[2];
  const void* labels;      // [H, W] int64 (or uint8 when label_u8) or null
  long long* cm;           // [C, C] or null (accumulated into)
  void* pred;              // [H, W] int64 (or uint8 when pred_u8) or null
  int label_u8, pred_u8;
  float* probs;            // [C, H, W] or null
};

__device__ __forceinline__ float tta_lerp(float wa, float a, float wb, float b) { return fmaf(wa, a, __fmul_rn(wb, b)); }

// label / prediction maps in either element width (int64 as the reference passes them, or uint8 as the dataloader holds them)
__device__ __forceinline__ long long tta_label(const TtaParams& p, long long pix) {
  return p.label_u8 ? (long long)__ldg(reinterpret_cast<const unsigned char*>(p.labels) + pix)
                    : ld_stream_s64(reinterpret_cast<const long long*>(p.labels) + pix);
}
__device__ __forceinline__ void tta_store_pred(const TtaParams& p, long long pix, int idx) {
  if (p.pred_u8) reinterpret_cast<uint8_t*>(p.pred)[pix] = (uint8_t)idx;
  else reinterpret_cast<long long*>(p.pred)[pix] = idx;
}

// v / s for every class with ONE reciprocal: r = rn(1/s); q = rn(v*r); q' = fma(fma(-q, s, v), r, q) is the correctly rounded
// quotient (Markstein) as long as nothing is subnormal -- here s is in [1, 32] and v in (0, 1], so only a tiny v needs the generic
// IEEE division (checked against v / s on 4e8 random pairs, and bit for bit against torch on the GPU by the tests).
__device__ __forceinline__ float tta_div(float v, float s, float r) {
  const float q = __fmul_rn(v, r);
  return fmaf(fmaf(-q, s, v), r, q);
}
constexpr float TTA_SPREAD = 68.0f;      // expf(-68) = 2.9e-30: with a logit spread <= 68 no class is a non-zero value below 1e-30

__device__ __forceinline__ float fmin3(float a, float b, float c) {
  float d;
  asm("min.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
template <int LO, int HI, int CT>
__device__ __forceinline__ float tree_min3(const float (&f)[CT]) {
  constexpr int n = HI - LO;
  if constexpr (n == 1) return f[LO];
  else if constexpr (n == 2) return fminf(f[LO], f[LO + 1]);
  else if constexpr (n == 3) return fmin3(f[LO], f[LO + 1], f[LO + 2]);
  else {
    constexpr int a = (n + 2) / 3, b = (n - a + 1) / 2;
    return fmin3(tree_min3<LO, LO + a, CT>(f), tree_min3<LO + a, LO + a + b, CT>(f), tree_min3<LO + a + b, HI, CT>(f));
  }
}

// acc[c] += softmax(v)[c] with ATen's sequence (max; sequential fp32 sum of expf(v - max) in class order; IEEE division).
// Maximum and minimum are order-independent, so they are 3-input trees; the minimum only decides whether the shared-reciprocal
// division is safe (both division paths are correctly rounded, so the conservative test changes no result).
template <int CT, bool EXACT>
__device__ __forceinline__ void tta_softmax_add(float (&v)[CT], int C, float (&acc)[CT]) {
  float mx, mn;
  if (EXACT) {
    mx = tree_max3<0, CT, CT>(v);
    mn = tree_min3<0, CT, CT>(v);
  } else {
    mx = v[0];
    mn = v[0];
#pragma unroll
    for (int c = 1; c < CT; ++c)
      if (c < C) { mx = fmaxf(mx, v[c]); mn = fminf(mn, v[c]); }
  }
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < CT; ++c) {
    if (EXACT || c < C) {
      v[c] = expf(v[c] - mx);
      s += v[c];
    }
  }
  // acc starts at +0 and the probabilities are >= +0, so the first member's 0 + p is p itself
  if (!(mx - mn > TTA_SPREAD)) {
    const float r = __frcp_rn(s);
#pragma unroll
    for (int c = 0; c < CT; ++c)
      if (EXACT || c < C) acc[c] = __fadd_rn(acc[c], tta_div(v[c], s, r));
  } else {
#pragma unroll
    for (int c = 0; c < CT; ++c)                             // (unrolled as well: a dynamically indexed acc[] would live in local memory)
      if (EXACT || c < C) acc[c] = __fadd_rn(acc[c], __fdiv_rn(v[c], s));
  }
}

// scalar divisions, first-maximum argmax, outputs of one pixel
template <int CT, bool EXACT>
__device__ __forceinline__ void tta_finish(const TtaParams& p, float (&acc)[CT], int C, long long pix, long long plane, int* hist) {
#pragma unroll 1
  for (int k = 0; k < p.n_div; ++k) {
    const float d = p.div[k];
    if (!p.div_exact) {
      const float r = __fdiv_rn(1.0f, d);
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[c] = __fmul_rn(acc[c], r);
    } else {
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[c] = __fdiv_rn(acc[c], d);
    }
  }
  float best = acc[0];
  int idx = 0;
#pragma unroll
  for (int c = 1; c < CT; ++c) {
    if ((EXACT || c < C) && acc[c] > best) { best = acc[c]; idx = c; }
  }
  if (p.probs) {
#pragma unroll
    for (int c = 0; c < CT; ++c)
      if (EXACT || c < C) __stcs(p.probs + c * plane + pix, acc[c]);
  }
  if (p.pred) tta_store_pred(p, pix, idx);
  if (p.cm) {
    const long long lab = tta_label(p, pix);
    if (lab != p.ignore_index && lab >= 0 && lab < C) atomicAdd(&hist[(int)lab * C + idx], 1);
  }
}

// ---- labels-only fast path -----------------------------------------------------------------------------------------------
// When only the labels / the confusion matrix are wanted, the probabilities need not be ATen's bit for bit -- only their ORDER.
// acc[c] += e_c / s with e_c = ex2.approx((v_c - max) * log2 e) (one FFMA + one MUFU per class instead of expf's ~8 instructions)
// and one reciprocal; every class whose sum lies within TTA_FAST_EPS * members of the largest is a candidate, and a pixel with more
// than one candidate is recomputed by the exact sequence (tta_exact_pixel).  Error budget: |fast - exact| <= ~3.5e-6 per member and
// class (ex2.approx 2^-22, the rounded exponent, the fp32 sum, one reciprocal; the common factor exp2(-max * log2 e) cancels in
// e / s), so two classes whose fast sums differ by more than 7e-6 * members are ordered alike by the exact sequence; the scalar
// divisions are monotone and cannot reorder them either.  Exactness of the labels against torch is what the tests check.
constexpr float TTA_FAST_EPS = 2e-5f;
__device__ __forceinline__ float tta_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
template <int CT, bool EXACT>
__device__ __forceinline__ void tta_softmax_add_fast(const float (&v)[CT], int C, float (&acc)[CT]) {
  float mx;
  if (EXACT) {
    mx = tree_max3<0, CT, CT>(v);
  } else {
    mx = v[0];
#pragma unroll
    for (int c = 1; c < CT; ++c)
      if (c < C) mx = fmaxf(mx, v[c]);
  }
  const float k = 1.4426950408889634f, off = -mx * k;
  float e[CT];
  float s = 0.f;
#pragma unroll
  for (int c = 0; c < CT; ++c) {
    if (EXACT || c < C) {
      e[c] = tta_ex2(fmaf(v[c], k, off));                   // one FFMA + one MUFU.EX2
      s += e[c];
    }
  }
  const float r = __frcp_rn(s);
#pragma unroll
  for (int c = 0; c < CT; ++c)
    if (EXACT || c < C) acc[c] = fmaf(e[c], r, acc[c]);
}

// the exact sequence for ONE pixel, straight from the members' logits (the per-pixel kernel's body; rare path of the fast kernel)
template <int CT, bool EXACT>
__device__ __noinline__ int tta_exact_pixel(const TtaParams& p, int C, int x, int y) {
  float acc[CT];
#pragma unroll
  for (int c = 0; c < CT; ++c) acc[c] = 0.f;
#pragma unroll 1
  for (int m = 0; m < p.n_maps; ++m) {
    const TtaMap& mp = p.maps[m];
    const int xs = mp.flip ? p.W - 1 - x : x;
    const Tap ty = ac_tap(mp.scale_h, y, mp.h);
    const Tap tx = ac_tap(mp.scale_w, xs, mp.w);
    const unsigned hw = (unsigned)(mp.h * mp.w);
    unsigned o00 = (unsigned)(ty.i0 * mp.w + tx.i0), o01 = (unsigned)(ty.i0 * mp.w + tx.i1);
    unsigned o10 = (unsigned)(ty.i1 * mp.w + tx.i0), o11 = (unsigned)(ty.i1 * mp.w + tx.i1);
    const float* __restrict__ lg = mp.logits;
    float v[CT];
#pragma unroll
    for (int c = 0; c < CT; ++c) {
      if (EXACT || c < C) {
        const float t = tta_lerp(tx.l0, __ldg(lg + o00), tx.l1, __ldg(lg + o01));
        const float u = tta_lerp(tx.l0, __ldg(lg + o10), tx.l1, __ldg(lg + o11));
        v[c] = tta_lerp(ty.l0, t, ty.l1, u);
        o00 += hw; o01 += hw; o10 += hw; o11 += hw;
      }
    }
    tta_softmax_add<CT, EXACT>(v, C, acc);
  }
#pragma unroll 1
  for (int k = 0; k < p.n_div; ++k) {
    const float d = p.div[k];
    if (!p.div_exact) {
      const float r = __fdiv_rn(1.0f, d);
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[c] = __fmul_rn(acc[c], r);
    } else {
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[c] = __fdiv_rn(acc[c], d);
    }
  }
  float best = acc[0];
  int idx = 0;
#pragma unroll
  for (int c = 1; c < CT; ++c)
    if ((EXACT || c < C) && acc[c] > best) { best = acc[c]; idx = c; }
  return idx;
}

// labels-only epilogue: unique candidate -> it is the argmax; otherwise the exact sequence decides
template <int CT, bool EXACT>
__device__ __forceinline__ void tta_finish_fast(const TtaParams& p, const float (&acc)[CT], int C, int x, int y, int* hist) {
  float best;
  if (EXACT) {
    best = tree_max3<0, CT, CT>(acc);
  } else {
    best = acc[0];
#pragma unroll
    for (int c = 1; c < CT; ++c)
      if (c < C) best = fmaxf(best, acc[c]);
  }
  const float thr = best - TTA_FAST_EPS * (float)p.n_maps;
  int cand = 0;
#pragma unroll
  for (int c = 0; c < CT; ++c)
    if ((EXACT || c < C) && acc[c] >= thr) cand += 256 + c;       // exactly one candidate: cand - 256 is its index
  int idx = cand - 256;
  if (cand >= 512 || !(best == best)) idx = tta_exact_pixel<CT, EXACT>(p, C, x, y);       // near tie (or NaN): exact sequence
  const long long pix = (long long)y * p.W + x;
  if (p.pred) tta_store_pred(p, pix, idx);
  if (p.cm) {
    const long long lab = tta_label(p, pix);
    if (lab != p.ignore_index && lab >= 0 && lab < C) atomicAdd(&hist[(int)lab * C + idx], 1);
  }
}

// EXACT: the class count is the compile-time CT (no per-class predicates)
template <int CT, bool EXACT>
__global__ void __launch_bounds__(TTA_THREADS) tta_argmax_confusion_kernel(const TtaParams p) {
  extern __shared__ int tta_hist[];
  const int C = EXACT ? CT : p.C, CC = C * C;
  if (p.cm) {
    for (int i = threadIdx.x; i < CC; i += TTA_THREADS) tta_hist[i] = 0;
    __syncthreads();
  }
  const int tiles_x = ceil_div(p.W, TTA_THREADS);
  const long long units = (long long)tiles_x * p.H;
  const long long plane = (long long)p.H * p.W;
  const long long chunk = ceil_div_ll(units, gridDim.x);                 // a CTA walks DOWN one 128-column strip: 8 or so consecutive
  const long long u_end = min(units, (blockIdx.x + 1) * chunk);         // rows share their source-row pair, which stays in L1
  for (long long unit = blockIdx.x * chunk; unit < u_end; ++unit) {
    const int y = (int)(unit % p.H);
    const int x = (int)(unit / p.H) * TTA_THREADS + threadIdx.x;
    if (x >= p.W) continue;
    float acc[CT];
#pragma unroll
    for (int c = 0; c < CT; ++c) acc[c] = 0.f;
#pragma unroll 1
    for (int m = 0; m < p.n_maps; ++m) {
      const TtaMap& mp = p.maps[m];
      const int xs = mp.flip ? p.W - 1 - x : x;              // the member saw the mirrored image: un-mirror its probabilities
      const Tap ty = ac_tap(mp.scale_h, y, mp.h);
      const Tap tx = ac_tap(mp.scale_w, xs, mp.w);
      const unsigned hw = (unsigned)(mp.h * mp.w);           // C * h * w < 2^31 (checked by the launcher): 32-bit element offsets
      unsigned o00 = (unsigned)(ty.i0 * mp.w + tx.i0), o01 = (unsigned)(ty.i0 * mp.w + tx.i1);
      unsigned o10 = (unsigned)(ty.i1 * mp.w + tx.i0), o11 = (unsigned)(ty.i1 * mp.w + tx.i1);
      const float* __restrict__ lg = mp.logits;
      float v[CT];
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        if (EXACT || c < C) {
          const float t = tta_lerp(tx.l0, __ldg(lg + o00), tx.l1, __ldg(lg + o01));
          const float u = tta_lerp(tx.l0, __ldg(lg + o10), tx.l1, __ldg(lg + o11));
          v[c] = tta_lerp(ty.l0, t, ty.l1, u);
          o00 += hw; o01 += hw; o10 += hw; o11 += hw;
        }
      }
      tta_softmax_add<CT, EXACT>(v, C, acc);
    }
    tta_finish<CT, EXACT>(p, acc, C, (long long)y * p.W + x, plane, tta_hist);
  }
  if (p.cm) {
    __syncthreads();
    for (int i = threadIdx.x; i < CC; i += TTA_THREADS) {
      const int v = tta_hist[i];
      if (v) atomicAdd(reinterpret_cast<unsigned long long*>(p.cm + i), (unsigned long long)v);
    }
  }
}

// ---- row-walking variant for ensembles of up to four members (inference(flip=True) has two) --------------------------------
// The horizontal lerps of a source row do not depend on the output row: a thread (= one output column) keeps, per member and
// class, the pair {t, u} = horizontal lerps on the two source rows of the current output row in SHARED memory, laid out
// [member][class][thread] (8-byte accesses, conflict-free, private to the thread: no barriers), and refreshes it only when the
// source-row pair changes (every (H-1)/(h-1) ~ 8 rows; moving down by one source row re-uses u as the new t).  Per pixel and member
// that leaves one LDS.64 + the vertical lerp per class instead of four global loads and three lerps -- identical arithmetic,
// ~2x fewer instructions.  A unit is TTA_RB consecutive rows of one 128-column strip.  The cache costs 19.5 KB of shared memory per
// member and CTA, i.e. occupancy: measured at 1024 x 2048 against the per-pixel kernel 60 / 103 / 163 / 250 us vs 80 / 141 / 204 /
// 266 us for 1 / 2 / 3 / 4 members, so larger ensembles stay on the per-pixel kernel.
constexpr int TTA_RB = 8;
constexpr int TTA_ROWS_MAX_MAPS = 4;

template <int CT, bool EXACT>
__device__ __forceinline__ void tta_hrow(const TtaMap& mp, int C, int row, const Tap& tx, float (&out)[CT]) {
  const unsigned hw = (unsigned)(mp.h * mp.w);
  unsigned o0 = (unsigned)(row * mp.w + tx.i0), o1 = (unsigned)(row * mp.w + tx.i1);
  const float* __restrict__ lg = mp.logits;
#pragma unroll
  for (int c = 0; c < CT; ++c) {
    if (EXACT || c < C) {
      out[c] = tta_lerp(tx.l0, __ldg(lg + o0), tx.l1, __ldg(lg + o1));
      o0 += hw; o1 += hw;
    }
  }
}

template <int CT, bool EXACT, bool FAST>
__global__ void __launch_bounds__(TTA_THREADS, (FAST && EXACT) ? 5 : 1) tta_rows_kernel(const TtaParams p) {
  extern __shared__ __align__(16) unsigned char tta_smem_raw[];
  // [n_maps][CT][TTA_THREADS] float2 pairs, then the int32 histogram
  float2* pairs = reinterpret_cast<float2*>(tta_smem_raw);
  int* hist = reinterpret_cast<int*>(tta_smem_raw + (size_t)p.n_maps * CT * TTA_THREADS * sizeof(float2));
  const int C = EXACT ? CT : p.C, CC = C * C;
  if (p.cm) {
    for (int i = threadIdx.x; i < CC; i += TTA_THREADS) hist[i] = 0;
    __syncthreads();
  }
  const int tiles_x = ceil_div(p.W, TTA_THREADS), blocks_y = ceil_div(p.H, TTA_RB);
  const int units = tiles_x * blocks_y;
  const long long plane = (long long)p.H * p.W;
  for (int unit = blockIdx.x; unit < units; unit += gridDim.x) {
    const int x = (unit / blocks_y) * TTA_THREADS + threadIdx.x;        // consecutive units walk DOWN a strip
    const int y0 = (unit % blocks_y) * TTA_RB, y1 = min(p.H, y0 + TTA_RB);
    if (x >= p.W) continue;
    int cur0[TTA_ROWS_MAX_MAPS], cur1[TTA_ROWS_MAX_MAPS];
#pragma unroll
    for (int m = 0; m < TTA_ROWS_MAX_MAPS; ++m) cur0[m] = cur1[m] = -1;
    for (int y = y0; y < y1; ++y) {
      float acc[CT];
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[c] = 0.f;
#pragma unroll
      for (int m = 0; m < TTA_ROWS_MAX_MAPS; ++m) {
        if (m < p.n_maps) {
          const TtaMap& mp = p.maps[m];
          const Tap ty = ac_tap(mp.scale_h, y, mp.h);
          float2* mine = pairs + (size_t)m * CT * TTA_THREADS + threadIdx.x;
          if (ty.i0 != cur0[m] || ty.i1 != cur1[m]) {                   // CTA-uniform: depends on the row only
            const int xs = mp.flip ? p.W - 1 - x : x;                   // the member saw the mirrored image: un-mirror it
            const Tap tx = ac_tap(mp.scale_w, xs, mp.w);
            float u[CT];
            tta_hrow<CT, EXACT>(mp, C, ty.i1, tx, u);
            if (ty.i0 == cur1[m]) {                                     // one source row down: the old u is the new t
#pragma unroll
              for (int c = 0; c < CT; ++c)
                if (EXACT || c < C) mine[c * TTA_THREADS] = make_float2(mine[c * TTA_THREADS].y, u[c]);
            } else {
              float t[CT];
              tta_hrow<CT, EXACT>(mp, C, ty.i0, tx, t);
#pragma unroll
              for (int c = 0; c < CT; ++c)
                if (EXACT || c < C) mine[c * TTA_THREADS] = make_float2(t[c], u[c]);
            }
            cur0[m] = ty.i0;
            cur1[m] = ty.i1;
          }
          float v[CT];
#pragma unroll
          for (int c = 0; c < CT; ++c) {
            if (EXACT || c < C) {
              const float2 tu = mine[c * TTA_THREADS];
              v[c] = tta_lerp(ty.l0, tu.x, ty.l1, tu.y);
            }
          }
          if (FAST) tta_softmax_add_fast<CT, EXACT>(v, C, acc);
          else tta_softmax_add<CT, EXACT>(v, C, acc);
        }
      }
      if (FAST) tta_finish_fast<CT, EXACT>(p, acc, C, x, y, hist);
      else tta_finish<CT, EXACT>(p, acc, C, (long long)y * p.W + x, plane, hist);
    }
  }
  if (p.cm) {
    __syncthreads();
    for (int i = threadIdx.x; i < CC; i += TTA_THREADS) {
      const int v = hist[i];
      if (v) atomicAdd(reinterpret_cast<unsigned long long*>(p.cm + i), (unsigned long long)v);
    }
  }
}

static int g_tta_rows = 1;      // b200seg_tta_set_row_walk(): 0 = always the per-pixel kernel (A/B)
static int g_tta_fast = 1;      // bit 1 of the same knob: 0 = never the labels-only fast path (A/B)
void tta_set_row_walk(int on) { g_tta_rows = on & 1; g_tta_fast = (on & 2) ? 0 : 1; }

template <int CT, bool EXACT, bool FAST>
static int tta_rows_launch_t(const TtaParams& p, cudaStream_t stream) {
  const size_t smem = (size_t)p.n_maps * CT * TTA_THREADS * sizeof(float2) + (p.cm ? (size_t)p.C * p.C * 4 : 0);
  static size_t configured = 0;
  if (smem > configured) {
    B200SEG_CUDA(cudaFuncSetAttribute(tta_rows_kernel<CT, EXACT, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    configured = smem;
  }
  int per_sm = 1;
  B200SEG_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, tta_rows_kernel<CT, EXACT, FAST>, TTA_THREADS, smem));
  if (per_sm < 1) per_sm = 1;
  const int units = ceil_div(p.W, TTA_THREADS) * ceil_div(p.H, TTA_RB);
  const int cap = num_sms() * per_sm;
  tta_rows_kernel<CT, EXACT, FAST><<<units < cap ? units : cap, TTA_THREADS, smem, stream>>>(p);
  return B200SEG_OK;
}
template <int CT, bool EXACT>
static int tta_rows_launch(const TtaParams& p, cudaStream_t stream) {
  // probabilities requested: every value must be ATen's; labels / matrix only: the order suffices (fast path + exact fallback)
  // measured at 1024 x 2048 (us, fast / exact): 1 member 52 / 62, 2: 81 / 110, 3: 154 / 171, 4: 289 / 254 -> fast up to three members
  // (CT = 32 with four unrolled members would spill)
  if (g_tta_fast && p.probs == nullptr && CT <= 20 && p.n_maps <= 3) return tta_rows_launch_t<CT, EXACT, true>(p, stream);
  return tta_rows_launch_t<CT, EXACT, false>(p, stream);
}

// logits[m]: fp32 [C, h[m], w[m]] (device pointers in a HOST array); flip[m] != 0: the member saw the mirrored image
int tta_launch(const float* const* logits, const int* hs, const int* ws, const int* flips, int n_maps, int C, const void* labels,
               int label_bytes, int H, int W, int ignore_index, const float* divisors, int n_div, int div_exact, long long* cm,
               void* pred, int pred_bytes, float* probs, cudaStream_t stream) {
  B200SEG_CHECK_ARG(labels == nullptr || label_bytes == 8 || label_bytes == 1, "tta_argmax_confusion: labels must be int64 or uint8");
  B200SEG_CHECK_ARG(pred == nullptr || pred_bytes == 8 || pred_bytes == 1, "tta_argmax_confusion: pred must be int64 or uint8");
  B200SEG_CHECK_ARG(logits && hs && ws && flips, "tta_argmax_confusion: null member table");
  B200SEG_CHECK_ARG(n_maps >= 1 && n_maps <= TTA_MAX_MAPS, "tta_argmax_confusion: %d members (1..%d supported)", n_maps, TTA_MAX_MAPS);
  B200SEG_CHECK_ARG(C > 0 && C <= 32, "tta_argmax_confusion: num_classes=%d not in 1..32", C);
  B200SEG_CHECK_ARG(H > 0 && W > 0, "tta_argmax_confusion: bad label size %d x %d", H, W);
  B200SEG_CHECK_ARG(n_div >= 0 && n_div <= 2 && (n_div == 0 || divisors), "tta_argmax_confusion: 0..2 divisors");
  B200SEG_CHECK_ARG(cm == nullptr || labels != nullptr, "tta_argmax_confusion: confusion matrix requested without labels");
  B200SEG_CHECK_ARG(cm || pred || probs, "tta_argmax_confusion: nothing to compute (cm, pred and probs all null)");
  TtaParams p = {};
  for (int m = 0; m < n_maps; ++m) {
    B200SEG_CHECK_ARG(logits[m] && hs[m] > 0 && ws[m] > 0, "tta_argmax_confusion: member %d has a null pointer or an empty shape", m);
    B200SEG_CHECK_ARG((long long)C * hs[m] * ws[m] < (1LL << 31), "tta_argmax_confusion: member %d is too large", m);
    p.maps[m].logits = logits[m];
    p.maps[m].h = hs[m];
    p.maps[m].w = ws[m];
    p.maps[m].flip = flips[m] ? 1 : 0;
    p.maps[m].scale_h = ac_scale(hs[m], H);
    p.maps[m].scale_w = ac_scale(ws[m], W);
  }
  p.n_maps = n_maps; p.C = C; p.H = H; p.W = W; p.ignore_index = ignore_index;
  p.n_div = n_div; p.div_exact = div_exact ? 1 : 0;
  for (int k = 0; k < n_div; ++k) {
    B200SEG_CHECK_ARG(divisors[k] != 0.f, "tta_argmax_confusion: zero divisor");
    p.div[k] = divisors[k];
  }
  p.labels = labels; p.cm = cm; p.pred = pred; p.probs = probs;
  p.label_u8 = (label_bytes == 1); p.pred_u8 = (pred_bytes == 1);
  const long long units = (long long)ceil_div(W, TTA_THREADS) * H;
  const long long cap = (long long)num_sms() * 8;
  const int grid = (int)(units < cap ? units : cap);
  const size_t smem = cm ? (size_t)C * C * 4 : 0;
  if (g_tta_rows && n_maps <= TTA_ROWS_MAX_MAPS) {
    profile_begin(15, stream);
    int rc;
    if (C == 2) rc = tta_rows_launch<2, true>(p, stream);
    else if (C == 19) rc = tta_rows_launch<19, true>(p, stream);
    else if (C <= 8) rc = tta_rows_launch<8, false>(p, stream);
    else if (C <= 20) rc = tta_rows_launch<20, false>(p, stream);
    else rc = tta_rows_launch<32, false>(p, stream);
    profile_end(15, stream);
    if (rc) return rc;
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  profile_begin(15, stream);
  if (C == 2) tta_argmax_confusion_kernel<2, true><<<grid, TTA_THREADS, smem, stream>>>(p);
  else if (C == 19) tta_argmax_confusion_kernel<19, true><<<grid, TTA_THREADS, smem, stream>>>(p);
  else if (C <= 8) tta_argmax_confusion_kernel<8, false><<<grid, TTA_THREADS, smem, stream>>>(p);
  else if (C <= 20) tta_argmax_confusion_kernel<20, false><<<grid, TTA_THREADS, smem, stream>>>(p);
  else tta_argmax_confusion_kernel<32, false><<<grid, TTA_THREADS, smem, stream>>>(p);
  profile_end(15, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

}  // namespace b200seg
