// K2: align-corners bilinear upsample fused with softmax cross-entropy (ignore_index) forward
//     AND the gradient with respect to the LOW-RESOLUTION logits, in one pass over the labels.
//
// Replaces (reference file:line):
//   F.interpolate(out, size, 'bilinear', align_corners=True)     core/models/classifiers/aspp/classifier.py:30-31
//   src_pred.div(temperature)                                    core/combos/aspp_fada.py:93-94
//   torch.nn.CrossEntropyLoss(ignore_index=255)(output, label)   core/trainers/aspp_trainer.py:61,91
//   loss.backward() through both                                 core/trainers/aspp_trainer.py:92
//
// The full-resolution logits (76 B/px at C=19) are never written.  Per output pixel the kernel
// recomputes the C interpolated logits from register-resident horizontal lerps, does one
// max / exp / sum pass, accumulates the loss, and folds softmax(v) - onehot(label) back onto
// the two source rows (weights l0y, l1y) in registers.  At every change of source-row pair the
// 128 columns of the tile are reduced onto their source columns through shared memory, into a
// per-tile partial block [rows][cols][C] that is written to scratch WITHOUT atomics; a small
// finalize kernel sums the <= 4 partial blocks that touch each low-res logit in a fixed order
// and applies grad_out / (n_valid * T).  Results are therefore run-to-run deterministic (ATen's
// upsample backward scatters with atomicAdd).
//
// Also here: materialising align-corners upsample forward / backward (the API-compat path for
// callers that want the full-resolution tensor, e.g. PixelDiscriminator.forward(x, size)).
#include "ce_geom.cuh"
#include "host_api.h"

namespace b200seg {

constexpr int K2_THREADS = 128;
constexpr int K2_TILE_W = 128;
#ifndef K2_TILE_H_DEF
#define K2_TILE_H_DEF 32
#endif
constexpr int K2_TILE_H = K2_TILE_H_DEF;        // <= 32 (four label strips in flight)
constexpr int K2_STRIP = 8;

// CTA-tile geometry (128 x 32); the warp-tile kernel (ce_v2_kernels.cu) uses 32 x 32 tiles where the shape is eligible.  Forward
// and backward pick the same one from the shape alone.
static void k2_geometry(K2Geom& g, int N, int C, int h, int w, int H, int W) { k2_geometry_tiled(g, N, C, h, w, H, W, K2_TILE_W, K2_TILE_H); }

static int g_k2_variant = 1;
void k2_set_variant(int v) { g_k2_variant = v; }
// variant 0: always the CTA-tile kernel; 1 (default): the warp-tile kernel where it is eligible AND measured faster (19 classes);
// 2: the warp-tile kernel wherever it is eligible (tests / A-B)
static bool k2_pick_geometry(K2Geom& g, int N, int C, int h, int w, int H, int W) {
  if (g_k2_variant != 0 && (C == 19 || g_k2_variant == 2) && k2v2_eligible(N, C, h, w, H, W)) { k2v2_geometry(g, N, C, h, w, H, W); return true; }
  k2_geometry(g, N, C, h, w, H, W);
  return false;
}

long long k2_workspace_bytes(int N, int C, int h, int w, int H, int W) {
  K2Geom g;
  k2_geometry(g, N, C, h, w, H, W);
  long long b = k2_geom_bytes(g);
  if (k2v2_eligible(N, C, h, w, H, W)) {
    k2v2_geometry(g, N, C, h, w, H, W);
    if (k2_geom_bytes(g) > b) b = k2_geom_bytes(g);
  }
  return b;
}

constexpr int K2_PITCH = K2_THREADS + 1;      // stage row pitch (floats): conflict-free for both access patterns

// ---- K2 main kernel ------------------------------------------------------------------------------------------
// The kernel is issue-bound (C classes of arithmetic per 8-byte label), so the per-pixel instruction count is what
// is optimised (same recipe as K4, eval_kernels.cu):
//   * class PAIRS in registers, all per-pixel arithmetic on packed fp32x2 (FMUL2 / FFMA2 / FADD2), max as a tree of
//     3-input FMNMX3, exp as ex2.approx on a pre-scaled argument;
//   * source rows staged per warp through shared memory (coalesced 32-bit-offset loads, immediate-offset LDS) -- the
//     staged raw windows also serve the labelled-class logit, no dynamic register indexing and no global re-loads;
//   * labels (int64, the only large stream) brought in by per-lane 8-byte cp.async for the whole tile up front, one
//     commit group per 8-row strip, so no registers or issue slots are held by loads in flight;
//   * explicit 32-bit shared-memory addressing for the one-hot updates.
constexpr int K2_SPAN = 8;                       // source columns a warp's 32 output columns may span on the staged path
constexpr int K2_PITCH2 = K2_THREADS + 1;        // stage row pitch in float2 (class pair) units
constexpr float K2_PAD = -1e30f;                 // logit of the padding classes: exp() == 0, never the maximum

__host__ __device__ constexpr int k2_np(int CT) { return (CT + 1) / 2; }
__host__ __device__ constexpr int k2_ns(int CT) { return (CT * K2_SPAN + 31) / 32; }

// shared-memory carve-up of the main kernel, in bytes from the start of dynamic shared memory
struct K2Smem {
  int stage0, stage1, blk, wt, red_lo, red_n, colw0, colw1, colx0, colx1, red, raw, ring, total;
};
__host__ __device__ inline K2Smem k2_smem_layout(int CT, int C, int ispan, int jspan, int kmax, int nwarps) {
  K2Smem L;
  int o = 0;
  L.stage0 = o; o += k2_np(CT) * K2_PITCH2 * 8;
  L.stage1 = o; o += k2_np(CT) * K2_PITCH2 * 8;
  L.blk = o; o += ispan * jspan * C * 4;
  L.wt = o; o += jspan * kmax * 4;
  L.red_lo = o; o += jspan * 4;
  L.red_n = o; o += jspan * 4;
  L.colw0 = o; o += K2_THREADS * 4;
  L.colw1 = o; o += K2_THREADS * 4;
  L.colx0 = o; o += K2_THREADS * 4;
  L.colx1 = o; o += K2_THREADS * 4;
  L.red = o; o += 2 * 8 * 4;
  o = (o + 15) / 16 * 16;
  L.raw = o; o += nwarps * 2 * CT * K2_SPAN * 4;                   // [warps][2 rows][CT][SPAN] raw logit windows
  o = (o + 15) / 16 * 16;
  L.ring = o; o += K2_TILE_H * K2_THREADS * 8;                     // [TILE_H][128] int64 labels
  L.total = o;
  return L;
}

// Load source row `rb` (frame base + row * w): leave its raw CT x K2_SPAN window in this warp's stage `raw_s` (staged
// path) and fill `dst` with this thread's class pairs [pbase, pbase + NPH), horizontally interpolated and scaled by 1/T.
template <int CT, int NPH, bool EXACT>
__device__ __forceinline__ void k2_row_load(float2 (&dst)[NPH], int pbase, const float* __restrict__ rb, int C, long long hw, bool staged,
                                            unsigned raw_s, int wj_lo, int w, unsigned t0_off, unsigned t1_off, int i0, int i1,
                                            float w0, float w1) {
  constexpr int NS = (CT * K2_SPAN + 31) / 32;
  const float2 L0 = make_float2(w0, w0), L1 = make_float2(w1, w1);
  if (staged) {
    const int lane = threadIdx.x & 31;
    float v[NS];
#pragma unroll
    for (int q = 0; q < NS; ++q) {                  // element e of the window: class e / SPAN, column wj_lo + e % SPAN
      const int e = q * 32 + lane;
      const int c = min(e / K2_SPAN, C - 1);
      if (e < CT * K2_SPAN) v[q] = __ldg(rb + c * hw + min(wj_lo + (e % K2_SPAN), w - 1));
    }
    __syncwarp();                                   // every lane is done with the previous contents of this stage
#pragma unroll
    for (int q = 0; q < NS; ++q)
      if (q * 32 + lane < CT * K2_SPAN) sts_f32(raw_s + (q * 32 + lane) * 4, v[q]);
    __syncwarp();
    const unsigned base0 = raw_s + t0_off + (unsigned)(2 * pbase) * (K2_SPAN * 4);
    const unsigned base1 = raw_s + t1_off + (unsigned)(2 * pbase) * (K2_SPAN * 4);
#pragma unroll
    for (int i = 0; i < NPH; ++i) {
      const int c0 = 2 * (pbase + i), c1 = c0 + 1;
      float2 a = make_float2(0.f, 0.f), b = make_float2(0.f, 0.f);
      if (c0 < C) { a.x = lds_f32(base0 + (2 * i) * K2_SPAN * 4); b.x = lds_f32(base1 + (2 * i) * K2_SPAN * 4); }
      if (c1 < C) { a.y = lds_f32(base0 + (2 * i + 1) * K2_SPAN * 4); b.y = lds_f32(base1 + (2 * i + 1) * K2_SPAN * 4); }
      dst[i] = fma2(L0, a, mul2(L1, b));
      if (c0 >= C) dst[i].x = K2_PAD;
      if (c1 >= C) dst[i].y = K2_PAD;
    }
  } else {
    const long long step = hw * 4;
    const char* p0 = reinterpret_cast<const char*>(rb + i0) + step * (2 * pbase);
    const char* p1 = reinterpret_cast<const char*>(rb + i1) + step * (2 * pbase);
#pragma unroll
    for (int i = 0; i < NPH; ++i) {
      const int c0 = 2 * (pbase + i), c1 = c0 + 1;
      float2 a = make_float2(0.f, 0.f), b = make_float2(0.f, 0.f);
      if (c0 < C) { a.x = __ldg(reinterpret_cast<const float*>(p0)); b.x = __ldg(reinterpret_cast<const float*>(p1)); }
      p0 += step; p1 += step;
      if (c1 < C) { a.y = __ldg(reinterpret_cast<const float*>(p0)); b.y = __ldg(reinterpret_cast<const float*>(p1)); }
      p0 += step; p1 += step;
      dst[i] = fma2(L0, a, mul2(L1, b));
      if (c0 >= C) dst[i].x = K2_PAD;
      if (c1 >= C) dst[i].y = K2_PAD;
    }
  }
}

template <int N>
__device__ __forceinline__ float k2_sum(const float (&p)[N]) {      // pairwise tree on packed adds
  float2 t[N / 2];
#pragma unroll
  for (int i = 0; i < N / 2; ++i) t[i] = make_float2(p[2 * i], p[2 * i + 1]);
#pragma unroll
  for (int n = N / 2; n > 1; n = (n + 1) / 2) {
#pragma unroll
    for (int i = 0; i < n / 2; ++i) t[i] = add2(t[i], t[n - 1 - i]);
  }
  return t[0].x + t[0].y;
}

// SPLIT threads share one output column: thread `half` of a column owns class pairs [half * NPH, (half + 1) * NPH), the
// per-pixel max and sum are exchanged with one shuffle each.  SPLIT = 2 halves the register arrays (a0, a1, acc0, acc1),
// which is what bounds the resident warps of this latency-bound kernel; used for the larger class counts.
#ifndef K2_SPLIT_MINB
#define K2_SPLIT_MINB 2
#endif
template <int CT, bool GRAD, bool EXACT, int SPLIT>
__global__ void __launch_bounds__(K2_THREADS * SPLIT, SPLIT == 1 ? 3 : K2_SPLIT_MINB) k2_upsample_ce_main(const K2Params p) {
  constexpr int NP = (CT + 1) / 2;
  constexpr int NPH = (NP + SPLIT - 1) / SPLIT;
  constexpr int NT = K2_THREADS * SPLIT;
  constexpr int NWARPS = NT / 32;
  constexpr float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;
  extern __shared__ __align__(16) uint8_t k2_smem_raw[];
  const K2Geom& g = p.g;
  const int C = EXACT ? CT : g.C;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int col = tid / SPLIT, half = tid - col * SPLIT;
  const int pbase = half * NPH;
  // shared-memory regions are re-derived from the layout where they are used (setup / flush) instead of being kept
  // as live generic pointers across the row loop
#define K2_L k2_smem_layout(CT, C, g.ispan_max, g.jspan_max, g.kmax, NWARPS)
#define K2_STAGE0 reinterpret_cast<float2*>(k2_smem_raw + K2_L.stage0)   /* [NP][129] per-column sums toward a0's source row */
#define K2_STAGE1 reinterpret_cast<float2*>(k2_smem_raw + K2_L.stage1)   /* ... toward a1's source row (start as -onehot sums) */
#define K2_BLK reinterpret_cast<float*>(k2_smem_raw + K2_L.blk)          /* [ispan_max][jspan_max][C] */
#define K2_WT reinterpret_cast<float*>(k2_smem_raw + K2_L.wt)            /* [jspan_max][kmax] column -> source-column weights */
#define K2_RED_LO reinterpret_cast<int*>(k2_smem_raw + K2_L.red_lo)      /* [jspan_max] first contributing column */
#define K2_RED_N reinterpret_cast<int*>(k2_smem_raw + K2_L.red_n)        /* [jspan_max] number of contributing columns */
  const int blk_floats = g.ispan_max * g.jspan_max * C;
  const K2Smem L = K2_L;
  const unsigned smem_s = smem_u32(k2_smem_raw);
  const unsigned rawA_s = smem_s + L.raw + (warp * 2 + 0) * CT * K2_SPAN * 4;   // raw window of a0's source row
  const unsigned rawB_s = smem_s + L.raw + (warp * 2 + 1) * CT * K2_SPAN * 4;   // ... of a1's
  const unsigned ring_s = smem_s + L.ring + col * 8;                            // this column's labels, row stride 1 KB
  const unsigned st0_s = smem_s + L.stage0 + col * 8, st1_s = smem_s + L.stage1 + col * 8;

  const int tile = blockIdx.x;
  const int tiles_per_frame = g.tiles_x * g.tiles_y;
  const int n = tile / tiles_per_frame;
  const int trem = tile - n * tiles_per_frame;
  const int ty = trem / g.tiles_x;
  const int tx = trem - ty * g.tiles_x;
  const long long hw = (long long)g.h * g.w;

  const int x = tx * K2_TILE_W + col;
  const bool xvalid = x < g.W;
  const Tap tapx = ac_tap(g.scale_w, xvalid ? x : g.W - 1, g.w);
  const int j_lo = (int)(g.scale_w * (float)(tx * K2_TILE_W));
  const int y_begin = ty * K2_TILE_H;
  const int y_end = min(g.H, y_begin + K2_TILE_H);
  const int i_lo = (int)(g.scale_h * (float)y_begin);
  const int jspan = g.jspan_max;

  // labels of the whole tile go in flight first: one commit group per K2_STRIP rows (issued by thread 0 of each column).
  // uint8 labels (the tensor the dataloader holds, core/datasets/transform.py:31-33): plain byte loads, all rows of the column
  // in flight at once, parked in the same ring as zero-extended 64-bit entries so the row loop is unchanged.
  if (p.label_u8) {
    const unsigned char* src = reinterpret_cast<const unsigned char*>(p.labels) + (long long)n * g.H * g.W + (long long)y_begin * g.W + (xvalid ? x : 0);
    unsigned b[K2_TILE_H];
#pragma unroll
    for (int r = 0; r < K2_TILE_H; ++r) b[r] = (half == 0 && xvalid && y_begin + r < y_end) ? (unsigned)__ldg(src + (long long)r * g.W) : 0xffu;
#pragma unroll
    for (int r = 0; r < K2_TILE_H; ++r)
      if (half == 0) asm volatile("st.shared.v2.u32 [%0], {%1, %2};" ::"r"(ring_s + r * (K2_THREADS * 8)), "r"(b[r]), "r"(0u) : "memory");
#pragma unroll
    for (int st = 0; st < K2_TILE_H / K2_STRIP; ++st) cp_async_commit();       // keep the group accounting of the row loop
  } else {
    const char* src = reinterpret_cast<const char*>(reinterpret_cast<const long long*>(p.labels) + (long long)n * g.H * g.W + (long long)y_begin * g.W + (xvalid ? x : 0));
    const long long row_bytes = (long long)g.W * 8;
#pragma unroll
    for (int st = 0; st < K2_TILE_H / K2_STRIP; ++st) {
#pragma unroll
      for (int r = 0; r < K2_STRIP; ++r) {
        const int yy = y_begin + st * K2_STRIP + r;
        if (half == 0 && xvalid && yy < y_end) cp_async_8s(ring_s + (st * K2_STRIP + r) * (K2_THREADS * 8), src);
        src += row_bytes;
      }
      cp_async_commit();
    }
  }

  if (GRAD) {
    float* blk = K2_BLK;
    float2* stage0 = K2_STAGE0;
    float* wt = K2_WT;
    int* red_lo = K2_RED_LO;
    int* red_n = K2_RED_N;
    float* colw0 = reinterpret_cast<float*>(k2_smem_raw + L.colw0);
    float* colw1 = reinterpret_cast<float*>(k2_smem_raw + L.colw1);
    int* colx0 = reinterpret_cast<int*>(k2_smem_raw + L.colx0);
    int* colx1 = reinterpret_cast<int*>(k2_smem_raw + L.colx1);
    for (int i = tid; i < blk_floats; i += NT) blk[i] = 0.f;
    for (int i = tid; i < 2 * NP * K2_PITCH2; i += NT) stage0[i] = make_float2(0.f, 0.f);   // stage0 and stage1 are adjacent
    if (half == 0) {
      colw0[col] = xvalid ? tapx.l0 : 0.f;
      colw1[col] = xvalid ? tapx.l1 : 0.f;
      colx0[col] = tapx.i0 - j_lo;
      colx1[col] = tapx.i1 - j_lo;
    }
    __syncthreads();
    if (tid < jspan) {                               // reduce table of source column jj = tid
      const int jj = tid;
      int lo = 0, hi = K2_THREADS;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (colx0[mid] < jj - 1) lo = mid + 1; else hi = mid; }
      int k = 0;
      for (int cc = lo; cc < K2_THREADS && colx0[cc] <= jj && k < g.kmax; ++cc, ++k)
        wt[jj * g.kmax + k] = (colx0[cc] == jj ? colw0[cc] : 0.f) + (colx1[cc] == jj ? colw1[cc] : 0.f);
      red_lo[jj] = lo;
      red_n[jj] = k;
    }
    __syncthreads();
  }

  const float* lg = p.logits + (long long)n * C * hw;

  // staged row loads: window of K2_SPAN source columns starting at lane 0's left tap
  const int wj_lo = __shfl_sync(0xffffffffu, tapx.i0, 0);
  const int wj_hi = __shfl_sync(0xffffffffu, tapx.i1, 31);
  const bool staged = (wj_hi - wj_lo) < K2_SPAN;
  const unsigned t0_off = (unsigned)(tapx.i0 - wj_lo) * 4, t1_off = (unsigned)(tapx.i1 - wj_lo) * 4;
  const float wx0 = p.inv_T * tapx.l0, wx1 = p.inv_T * tapx.l1;

  float2 a0[NPH], a1[NPH];
  float2 acc0[GRAD ? NPH : 1], acc1[GRAD ? NPH : 1];     // d loss / d a0-row, d loss / d a1-row (softmax part)
  if constexpr (GRAD) {
#pragma unroll
    for (int i = 0; i < NPH; ++i) { acc0[i] = make_float2(0.f, 0.f); acc1[i] = make_float2(0.f, 0.f); }
  }
  int row0 = -1, row1 = -1;         // source rows held in a0 / a1
  bool swap = false;                // true: a1 is the upper row
  bool open_seg = false;
  float loss_acc = 0.f, cnt_acc = 0.f;

  // Reduce the open segment's per-column sums onto source columns and add them to blk.
  auto flush_segment = [&]() {
    if constexpr (GRAD) {
      float2* stage0 = K2_STAGE0;
      float2* stage1 = K2_STAGE1;
      float* blk = K2_BLK;
      const float* wt = K2_WT;
      const int* red_lo = K2_RED_LO;
      const int* red_n = K2_RED_N;
#pragma unroll
      for (int i = 0; i < NPH; ++i)
        if (pbase + i < NP) {
          stage0[(pbase + i) * K2_PITCH2 + col] = add2(stage0[(pbase + i) * K2_PITCH2 + col], acc0[i]);
          stage1[(pbase + i) * K2_PITCH2 + col] = add2(stage1[(pbase + i) * K2_PITCH2 + col], acc1[i]);
          acc0[i] = make_float2(0.f, 0.f); acc1[i] = make_float2(0.f, 0.f);
        }
      __syncthreads();
      const int r0 = row0 - i_lo, r1 = row1 - i_lo;
      for (int o = tid; o < NP * jspan; o += NT) {
        const int jj = o / NP;
        const int i = o - jj * NP;
        const int lo = red_lo[jj], cnt = red_n[jj];
        const float* wrow = wt + jj * g.kmax;
        const float2* s0 = stage0 + i * K2_PITCH2 + lo;
        const float2* s1 = stage1 + i * K2_PITCH2 + lo;
        float2 t0 = make_float2(0.f, 0.f), t1 = make_float2(0.f, 0.f);
        for (int k = 0; k < cnt; ++k) {
          const float wk = wrow[k];
          const float2 W = make_float2(wk, wk);
          t0 = fma2(W, s0[k], t0);
          t1 = fma2(W, s1[k], t1);
        }
        float* b0 = blk + (r0 * jspan + jj) * C + 2 * i;
        float* b1 = blk + (r1 * jspan + jj) * C + 2 * i;
        if (2 * i < C) { b0[0] += t0.x; b1[0] += t1.x; }
        if (2 * i + 1 < C) { b0[1] += t0.y; b1[1] += t1.y; }
      }
      __syncthreads();
#pragma unroll
      for (int i = 0; i < NPH; ++i)
        if (pbase + i < NP) {
          stage0[(pbase + i) * K2_PITCH2 + col] = make_float2(0.f, 0.f);
          stage1[(pbase + i) * K2_PITCH2 + col] = make_float2(0.f, 0.f);
        }
    }
  };

  const unsigned ign32 = (p.ignore_index >= 0) ? (unsigned)p.ignore_index : 0xffffffffu;
  const unsigned c_lim = xvalid ? (unsigned)C : 0u;

#pragma unroll 1
  for (int y = y_begin; y < y_end; ++y) {
    const int yr = y - y_begin;
    if ((yr & (K2_STRIP - 1)) == 0) {                        // this strip's labels have landed
      const int pending = K2_TILE_H / K2_STRIP - 1 - yr / K2_STRIP;      // commit groups that may still be in flight
      if (pending >= 3) cp_async_wait<3>();
      else if (pending == 2) cp_async_wait<2>();
      else if (pending == 1) cp_async_wait<1>();
      else cp_async_wait<0>();
      if (SPLIT > 1) __syncwarp();                           // the copies were issued by the column's thread 0
    }
    const Tap tapy = ac_tap(g.scale_h, y, g.h);              // CTA-uniform
    const int top = swap ? row1 : row0, bot = swap ? row0 : row1;
    if (!open_seg || tapy.i0 != top || tapy.i1 != bot) {      // new source-row pair (CTA-uniform branch)
      if (open_seg) flush_segment();
      open_seg = true;
      bool need_top = false;
      if (row0 == tapy.i0) swap = false;
      else if (row1 == tapy.i0) swap = true;
      else { swap = false; need_top = true; }
#pragma unroll 1
      for (int which = need_top ? 0 : 1; which < 2; ++which) {
        const int row = which ? tapy.i1 : tapy.i0;
        const bool into_a0 = (which == 0) != swap;
        if ((into_a0 ? row0 : row1) == row) continue;
        const float* rb = lg + (long long)row * g.w;
        if (into_a0) { k2_row_load<CT, NPH, EXACT>(a0, pbase, rb, C, hw, staged, rawA_s, wj_lo, g.w, t0_off, t1_off, tapx.i0, tapx.i1, wx0, wx1); row0 = row; }
        else         { k2_row_load<CT, NPH, EXACT>(a1, pbase, rb, C, hw, staged, rawB_s, wj_lo, g.w, t0_off, t1_off, tapx.i0, tapx.i1, wx0, wx1); row1 = row; }
      }
    }
    const uint2 gl = lds_v2u32(ring_s + yr * (K2_THREADS * 8));     // int64 label as {lo, hi}
    const bool valid = (gl.y == 0u) && (gl.x < c_lim) && (gl.x != ign32);
    // lanes of the warp that take the branch (both threads of a column always do together): the mask of the shuffles
    const unsigned vmask = SPLIT > 1 ? __ballot_sync(0xffffffffu, valid) : 0u;
    if (valid) {
      const int gi = (int)gl.x;
      const float w0 = swap ? tapy.l1 : tapy.l0;             // weight of a0's row, of a1's row
      const float w1 = swap ? tapy.l0 : tapy.l1;
      const float2 W0 = make_float2(w0, w0), W1 = make_float2(w1, w1);
      float f[2 * NPH];
#pragma unroll
      for (int i = 0; i < NPH; ++i) {
        const float2 v = fma2(W0, a0[i], mul2(W1, a1[i]));
        f[2 * i] = v.x; f[2 * i + 1] = v.y;
      }
      float m = tree_max3<0, 2 * NPH, 2 * NPH>(f);
      if (SPLIT > 1) m = fmaxf(m, __shfl_xor_sync(vmask, m, 1));
      // logit of the labelled class from the staged raw windows (or re-interpolated from global on the fallback path)
      float vA, vB;
      if (staged) {
        const unsigned ga = (unsigned)gi * (K2_SPAN * 4);
        vA = fmaf(tapx.l0, lds_f32(rawA_s + ga + t0_off), tapx.l1 * lds_f32(rawA_s + ga + t1_off));
        vB = fmaf(tapx.l0, lds_f32(rawB_s + ga + t0_off), tapx.l1 * lds_f32(rawB_s + ga + t1_off));
      } else {
        const float* u0 = lg + gi * hw + (long long)row0 * g.w;
        const float* u1 = lg + gi * hw + (long long)row1 * g.w;
        vA = fmaf(tapx.l0, __ldg(u0 + tapx.i0), tapx.l1 * __ldg(u0 + tapx.i1));
        vB = fmaf(tapx.l0, __ldg(u1 + tapx.i0), tapx.l1 * __ldg(u1 + tapx.i1));
      }
      const float vlab = p.inv_T * fmaf(w0, vA, w1 * vB);
      const float mneg = -m * LOG2E;
      const float2 K = make_float2(LOG2E, LOG2E), M = make_float2(mneg, mneg);
#pragma unroll
      for (int i = 0; i < NPH; ++i) {
        const float2 arg = fma2(make_float2(f[2 * i], f[2 * i + 1]), K, M);
        f[2 * i] = fast_exp2(arg.x); f[2 * i + 1] = fast_exp2(arg.y);
      }
      float s = k2_sum<2 * NPH>(f);
      if (SPLIT > 1) s += __shfl_xor_sync(vmask, s, 1);
      if (half == 0) {                                       // one thread per column carries the loss
        loss_acc += fmaf(__log2f(s), LN2, m) - vlab;
        cnt_acc += 1.f;
      }
      if constexpr (GRAD) {
        const float inv_s = __fdividef(1.f, s);
        const float c0 = w0 * inv_s, c1 = w1 * inv_s;
        const float2 C0 = make_float2(c0, c0), C1 = make_float2(c1, c1);
#pragma unroll
        for (int i = 0; i < NPH; ++i) {
          const float2 pr = make_float2(f[2 * i], f[2 * i + 1]);
          acc0[i] = fma2(C0, pr, acc0[i]);
          acc1[i] = fma2(C1, pr, acc1[i]);
        }
        // -onehot into the column's stage slot, by the thread that owns the labelled class
        if ((gi >> 1) / NPH == half) {
          const unsigned oh = (unsigned)(gi >> 1) * (K2_PITCH2 * 8) + (unsigned)(gi & 1) * 4;
          sts_f32(st0_s + oh, lds_f32(st0_s + oh) - w0);
          sts_f32(st1_s + oh, lds_f32(st1_s + oh) - w1);
        }
      }
    }
  }
  if (open_seg) flush_segment();

  // per-tile loss / count partials (fixed-order tree => deterministic)
  loss_acc = warp_sum(loss_acc);
  cnt_acc = warp_sum(cnt_acc);
  float* red = reinterpret_cast<float*>(k2_smem_raw + K2_L.red);
  if (lane == 0) { red[warp] = loss_acc; red[8 + warp] = cnt_acc; }
  __syncthreads();
  if (tid == 0) {
    float ls = 0.f, cs = 0.f;
#pragma unroll
    for (int q = 0; q < NWARPS; ++q) { ls += red[q]; cs += red[8 + q]; }
    p.loss_part[tile] = ls;
    p.cnt_part[tile] = cs;
  }
  if (GRAD) {
    const float* blk = K2_BLK;
    float* dst = p.blocks + (long long)tile * blk_floats;
    for (int i = tid; i < blk_floats; i += NT) dst[i] = blk[i];
  }
#undef K2_L
#undef K2_STAGE0
#undef K2_STAGE1
#undef K2_BLK
#undef K2_WT
#undef K2_RED_LO
#undef K2_RED_N
}

// loss = sum(loss_part) / sum(cnt_part)  (NaN when no valid pixel, like the reference); out = {loss, n_valid}
// (loss_copy: optional second home of the loss scalar -- the tensor handed back to autograd by the one-call train entry)
__global__ void __launch_bounds__(256) k2_finalize_loss(const float* loss_part, const float* cnt_part, int tiles, float* out2,
                                                        float* loss_copy) {
  __shared__ double sl[8], sc[8];
  double l = 0.0, c = 0.0;
  for (int i = threadIdx.x; i < tiles; i += 256) { l += (double)loss_part[i]; c += (double)cnt_part[i]; }
  l = warp_sum_d(l); c = warp_sum_d(c);
  if ((threadIdx.x & 31) == 0) { sl[threadIdx.x >> 5] = l; sc[threadIdx.x >> 5] = c; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double L = 0.0, Cn = 0.0;
    for (int i = 0; i < 8; ++i) { L += sl[i]; Cn += sc[i]; }
    out2[0] = (float)(L / Cn);
    out2[1] = (float)Cn;
    if (loss_copy) loss_copy[0] = (float)(L / Cn);
  }
}

// grad[n,c,i,j] = grad_out * inv_T / n_valid * sum over the tiles touching (i,j) of their partial block (0 when n_valid = 0).
// PACKED = false: fp32 NCHW grad_logits (the autograd contract of the stand-alone loss op).
// PACKED = true : bf16 class planes gOc[n][c][hw] (what the head's backward consumes) + per-block fp32 partial sums
//                 of the gradient per class (-> bias gradient), skipping the NCHW round trip.
template <bool PACKED>
__global__ void __launch_bounds__(128) k2_finalize_grad(const K2Geom g, const float* blocks, const float* loss_out2,
                                                        const float* grad_out, float inv_T, float* grad_logits,
                                                        __nv_bfloat16* gOt, float* bias_part) {
  __shared__ float wsum[4][32];
  const int j = blockIdx.x * 128 + threadIdx.x;
  const int i = blockIdx.y;
  const int n = blockIdx.z;
  const bool active = j < g.w;
  const float n_valid = loss_out2[1];
  // no valid label: every accumulator is 0 and so is the gradient (as in ATen); 1 / n_valid would make it 0 * inf = NaN
  const float scale = n_valid > 0.f ? (grad_out ? grad_out[0] : 1.f) * inv_T / n_valid : 0.f;
  float acc[32];
#pragma unroll
  for (int c = 0; c < 32; ++c) acc[c] = 0.f;
  const long long blk_floats = (long long)g.ispan_max * g.jspan_max * g.C;
  const long long hw = (long long)g.h * g.w;
  if (active) {
    // output rows / cols that interpolate from source row i / col j:  dst in [first(i-1), first(i+1))
    const int ya = ac_first_dst(g.scale_h, i - 1, g.h, g.H), yb = ac_first_dst(g.scale_h, i + 1, g.h, g.H);
    const int xa = ac_first_dst(g.scale_w, j - 1, g.w, g.W), xb = ac_first_dst(g.scale_w, j + 1, g.w, g.W);
    if (ya < yb && xa < xb) {
      const int ty0 = ya / g.tile_h, ty1 = (yb - 1) / g.tile_h;
      const int tx0 = xa / g.tile_w, tx1 = (xb - 1) / g.tile_w;
      for (int ty = ty0; ty <= ty1; ++ty) {
        const int li = i - (int)(g.scale_h * (float)(ty * g.tile_h));
        if (li < 0 || li >= g.ispan_max) continue;
        for (int tx = tx0; tx <= tx1; ++tx) {
          const int lj = j - (int)(g.scale_w * (float)(tx * g.tile_w));
          if (lj < 0 || lj >= g.jspan_max) continue;
          const long long tile = ((long long)n * g.tiles_y + ty) * g.tiles_x + tx;
          const float* src = blocks + tile * blk_floats + ((long long)li * g.jspan_max + lj) * g.C;
#pragma unroll
          for (int c = 0; c < 32; ++c)
            if (c < g.C) acc[c] += src[c];
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 32; ++c) acc[c] *= scale;
    if (!PACKED) {
      float* dst = grad_logits + (long long)n * g.C * hw + (long long)i * g.w + j;
#pragma unroll
      for (int c = 0; c < 32; ++c)
        if (c < g.C) dst[c * hw] = acc[c];
    } else {                           // bf16 class planes [N][C][hw], coalesced along x
      __nv_bfloat16* dst = gOt + (long long)n * g.C * hw + (long long)i * g.w + j;
#pragma unroll
      for (int c = 0; c < 32; ++c)
        if (c < g.C) dst[c * hw] = __float2bfloat16(acc[c]);
    }
  }
  if (PACKED) {                       // fixed-order block reduction of the fp32 gradient per class
#pragma unroll
    for (int c = 0; c < 32; ++c) {
      if (c < g.C) {                    // (uniform: classes beyond C are all-zero accumulators, no need to reduce them)
        const float v = warp_sum(acc[c]);
        if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5][c] = v;
      }
    }
    __syncthreads();
    if (threadIdx.x < 32) {
      const int c = threadIdx.x;
      const long long blk_id = ((long long)n * g.h + i) * gridDim.x + blockIdx.x;
      bias_part[blk_id * 32 + c] = c < g.C ? (wsum[0][c] + wsum[1][c]) + (wsum[2][c] + wsum[3][c]) : 0.f;
    }
  }
}

// bias_grad[c] = sum over finalize blocks of bias_part[blk][c]  (one block per class, fixed order), written to every one of the
// n destinations (the R branch biases of the head all receive the same gradient: classifier.py:27-29 sums the branches)
struct K2BiasOuts {
  float* p[8];
  int n;
};
__global__ void __launch_bounds__(256) k2_bias_from_partials(const float* bias_part, long long nblk, int C, const K2BiasOuts outs) {
  __shared__ double red[8];
  const int c = blockIdx.x;
  double acc = 0.0;
  for (long long b = threadIdx.x; b < nblk; b += 256) acc += (double)bias_part[b * 32 + c];
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int q = 0; q < 8; ++q) t += red[q];
    for (int q = 0; q < outs.n; ++q) outs.p[q][c] = (float)t;
  }
}

template <int CT, bool EXACT, int SPLIT>
static int k2_main_launch(const K2Params& p, bool grad, cudaStream_t stream) {
  const K2Geom& g = p.g;
  const size_t smem = (size_t)k2_smem_layout(CT, g.C, g.ispan_max, g.jspan_max, g.kmax, K2_THREADS * SPLIT / 32).total;
  B200SEG_CHECK_ARG(smem <= 200 * 1024, "upsample_ce: tile footprint %zu B exceeds shared memory (resize ratio too small)", smem);
  const int tiles = (int)k2_tiles(g);
  profile_begin(6, stream);
  if (grad) {
    static bool configured = false;
    if (!configured) {
      B200SEG_CUDA(cudaFuncSetAttribute(k2_upsample_ce_main<CT, true, EXACT, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      configured = true;
    }
    k2_upsample_ce_main<CT, true, EXACT, SPLIT><<<tiles, K2_THREADS * SPLIT, smem, stream>>>(p);
  } else {
    static bool configured = false;
    if (!configured) {
      B200SEG_CUDA(cudaFuncSetAttribute(k2_upsample_ce_main<CT, false, EXACT, SPLIT>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      configured = true;
    }
    k2_upsample_ce_main<CT, false, EXACT, SPLIT><<<tiles, K2_THREADS * SPLIT, smem, stream>>>(p);
  }
  profile_end(6, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int k2_forward(const float* logits, int N, int C, int h, int w, const void* labels, int label_bytes, int H, int W, int ignore_index,
               float inv_T, int need_grad, void* workspace, long long workspace_bytes, float* loss_out2, cudaStream_t stream,
               float* loss_copy) {
  B200SEG_CHECK_ARG(label_bytes == 8 || label_bytes == 1, "upsample_ce_forward: labels must be int64 or uint8 (label_bytes=%d)", label_bytes);
  B200SEG_CHECK_ARG(logits && labels && workspace && loss_out2, "upsample_ce_forward: null pointer");
  B200SEG_CHECK_ARG(N > 0 && C > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_ce_forward: bad shape");
  B200SEG_CHECK_ARG(C <= 32, "upsample_ce_forward: num_classes=%d > 32 is not supported", C);
  B200SEG_CHECK_ARG(workspace_bytes >= k2_workspace_bytes(N, C, h, w, H, W), "upsample_ce_forward: workspace too small (%lld < %lld)",
                    workspace_bytes, k2_workspace_bytes(N, C, h, w, H, W));
  K2Params p;
  const bool v2 = k2_pick_geometry(p.g, N, C, h, w, H, W);
  const long long tiles = k2_tiles(p.g);
  p.counter = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(workspace) + k2_geom_bytes(p.g) - 256);
  p.logits = logits; p.labels = labels; p.label_u8 = (label_bytes == 1); p.ignore_index = ignore_index; p.inv_T = inv_T;
  p.loss_part = reinterpret_cast<float*>(workspace);
  p.cnt_part = p.loss_part + tiles;
  p.blocks = p.cnt_part + tiles;
  int rc;
  if (v2) {
    rc = k2v2_main_launch(p, need_grad != 0, stream);
    if (rc) return rc;
    k2_finalize_loss<<<1, 256, 0, stream>>>(p.loss_part, p.cnt_part, (int)tiles, loss_out2, loss_copy);
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
#ifndef K2_SPLIT_DEF
#define K2_SPLIT_DEF 1   /* 2 = class dimension split over lane pairs: measured 135 us vs 108 us at C = 19 (profiles/README.md) */
#endif
  if (C == 2) rc = k2_main_launch<2, true, 1>(p, need_grad != 0, stream);
  else if (C == 19) rc = k2_main_launch<19, true, K2_SPLIT_DEF>(p, need_grad != 0, stream);
  else if (C <= 8) rc = k2_main_launch<8, false, 1>(p, need_grad != 0, stream);
  else rc = k2_main_launch<32, false, K2_SPLIT_DEF>(p, need_grad != 0, stream);
  if (rc) return rc;
  k2_finalize_loss<<<1, 256, 0, stream>>>(p.loss_part, p.cnt_part, (int)tiles, loss_out2, loss_copy);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int k2_backward(const void* workspace, int N, int C, int h, int w, int H, int W, float inv_T, const float* loss_out2,
                const float* grad_out, float* grad_logits, cudaStream_t stream) {
  B200SEG_CHECK_ARG(workspace && loss_out2 && grad_logits, "upsample_ce_backward: null pointer");
  K2Geom g;
  k2_pick_geometry(g, N, C, h, w, H, W);
  const long long tiles = k2_tiles(g);
  const float* blocks = reinterpret_cast<const float*>(workspace) + 2 * tiles;
  dim3 grid(ceil_div(w, 128), h, N);
  k2_finalize_grad<false><<<grid, 128, 0, stream>>>(g, blocks, loss_out2, grad_out, inv_T, grad_logits, nullptr, nullptr);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// Packed form for the fused head+loss path: bf16 pixel-major gradient + bias gradient, no fp32 NCHW tensor.
int k2_backward_packed_multi(void* workspace, int N, int C, int h, int w, int H, int W, float inv_T, const float* loss_out2,
                             const float* grad_out, void* gOt, float* const* bias_grads, int n_bias, cudaStream_t stream) {
  B200SEG_CHECK_ARG(workspace && loss_out2 && gOt, "upsample_ce_backward_packed: null pointer");
  B200SEG_CHECK_ARG(n_bias >= 0 && n_bias <= 8 && (n_bias == 0 || bias_grads), "upsample_ce_backward_packed: %d bias destinations", n_bias);
  B200SEG_CHECK_ARG(C <= 32, "upsample_ce_backward_packed: num_classes=%d > 32 is not supported", C);
  K2Geom g;
  k2_pick_geometry(g, N, C, h, w, H, W);
  const long long tiles = k2_tiles(g);
  float* base = reinterpret_cast<float*>(workspace);
  const float* blocks = base + 2 * tiles;
  float* bias_part = base + 2 * tiles + tiles * k2_block_floats(g);
  dim3 grid(ceil_div(w, 128), h, N);
  k2_finalize_grad<true><<<grid, 128, 0, stream>>>(g, blocks, loss_out2, grad_out, inv_T, nullptr, (__nv_bfloat16*)gOt, bias_part);
  B200SEG_LAUNCH_CHECK();
  K2BiasOuts outs = {};
  for (int q = 0; q < n_bias; ++q)
    if (bias_grads[q]) outs.p[outs.n++] = bias_grads[q];
  if (outs.n > 0) {
    k2_bias_from_partials<<<C, 256, 0, stream>>>(bias_part, (long long)grid.x * grid.y * grid.z, C, outs);
    B200SEG_LAUNCH_CHECK();
  }
  return B200SEG_OK;
}

int k2_backward_packed(void* workspace, int N, int C, int h, int w, int H, int W, float inv_T, const float* loss_out2,
                       const float* grad_out, void* gOt, float* bias_grad, cudaStream_t stream) {
  return k2_backward_packed_multi(workspace, N, C, h, w, H, W, inv_T, loss_out2, grad_out, gOt, &bias_grad, bias_grad ? 1 : 0, stream);
}

// =============================================================================================
// K5: the FADA PixelDiscriminator loss tail, fully fused on LOW-RESOLUTION tensors.
//
// Replaces, per call (reference file:line):
//   F.interpolate(cat(cls1, cls2), size, 'bilinear', align_corners=True)   core/models/discriminator.py:47-49
//   F.softmax(seg_pred / 1.8).detach(); soft[soft > 0.9] = 0.9              core/combos/aspp_fada.py:93-94,99-100,104-108
//   torch.cat((soft, zeros)) / torch.cat((zeros, soft))                     core/combos/aspp_fada.py:111,120,124
//   soft_label_cross_entropy(D_pred, soft_label) and its backward           core/utils/utility.py:172-177
// None of the five full-resolution [N,2C,H,W] / [N,C,H,W] tensors is materialised: per output pixel the kernel
// interpolates the 2C discriminator logits and the C segmentation logits from register-resident horizontal lerps,
// builds q = min(softmax(seg / T), clamp) on the fly, accumulates  lse(D) * sum(q) - sum_c q_c * D[slot*C + c]  and folds
// (softmax(D) * sum(q) - q) back onto the low-res discriminator logits with the same deterministic tile-partial scheme
// as K2.  Purely compute-bound (the only inputs are the low-res tensors).
// =============================================================================================
struct K5Params {
  K2Geom g;                  // geometry with g.C = 2*C (channels of the gradient blocks)
  const float* dlogits;      // [N, 2C, h, w]
  const float* slogits;      // [N,  C, h, w]
  float inv_T, clamp;
  float* loss_part;          // [tiles]
  float* blocks;             // [tiles][ispan_max][jspan_max][2C]
};

template <int NCH, bool EXACT>
__device__ __forceinline__ void k5_load_row(float (&dst)[NCH], const float* __restrict__ lg, int nch, long long hw, int row, int w,
                                            const Tap& tapx, float prescale) {
  const float* p0 = lg + (long long)row * w + tapx.i0;
  const float* p1 = lg + (long long)row * w + tapx.i1;
  const float w0 = prescale * tapx.l0, w1 = prescale * tapx.l1;
#pragma unroll
  for (int c = 0; c < NCH; ++c)
    if (EXACT || c < nch) {
      dst[c] = w0 * __ldg(p0) + w1 * __ldg(p1);
      p0 += hw; p1 += hw;
    }
}

template <int CT, bool GRAD, bool EXACT, int SLOT>
__global__ void __launch_bounds__(K2_THREADS, 2) k5_fada_softce_main(const K5Params p) {
  constexpr int KT = 2 * CT;
  constexpr float LOG2E = 1.4426950408889634f, LN2 = 0.6931471805599453f;
  extern __shared__ __align__(16) float k2_smem[];
  const K2Geom& g = p.g;
  const int C = EXACT ? CT : g.C / 2;
  const int K = 2 * C;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  float* stage0 = k2_smem;                           // [KT][129]
  float* stage1 = stage0 + KT * K2_PITCH;            // [KT][129]
  float* blk = stage1 + KT * K2_PITCH;               // [ispan_max][jspan_max][K]
  const int blk_floats = g.ispan_max * g.jspan_max * K;
  float* wt = blk + blk_floats;
  int* red_lo = reinterpret_cast<int*>(wt + g.jspan_max * g.kmax);
  int* red_n = red_lo + g.jspan_max;
  float* colw0 = reinterpret_cast<float*>(red_n + g.jspan_max);
  float* colw1 = colw0 + K2_THREADS;
  int* colx0 = reinterpret_cast<int*>(colw1 + K2_THREADS);
  int* colx1 = colx0 + K2_THREADS;
  float* red = reinterpret_cast<float*>(colx1 + K2_THREADS);

  const int tile = blockIdx.x;
  const int tiles_per_frame = g.tiles_x * g.tiles_y;
  const int n = tile / tiles_per_frame;
  const int trem = tile - n * tiles_per_frame;
  const int ty = trem / g.tiles_x;
  const int tx = trem - ty * g.tiles_x;
  const long long hw = (long long)g.h * g.w;
  const int x = tx * K2_TILE_W + tid;
  const bool xvalid = x < g.W;
  const Tap tapx = ac_tap(g.scale_w, xvalid ? x : g.W - 1, g.w);
  const int j_lo = (int)(g.scale_w * (float)(tx * K2_TILE_W));
  const int y_begin = ty * K2_TILE_H;
  const int y_end = min(g.H, y_begin + K2_TILE_H);
  const int i_lo = (int)(g.scale_h * (float)y_begin);
  const int jspan = g.jspan_max;

  if (GRAD) {
    for (int i = tid; i < blk_floats; i += K2_THREADS) blk[i] = 0.f;
    colw0[tid] = xvalid ? tapx.l0 : 0.f;
    colw1[tid] = xvalid ? tapx.l1 : 0.f;
    colx0[tid] = tapx.i0 - j_lo;
    colx1[tid] = tapx.i1 - j_lo;
    __syncthreads();
    if (tid < jspan) {
      const int jj = tid;
      int lo = 0, hi = K2_THREADS;
      while (lo < hi) { const int mid = (lo + hi) >> 1; if (colx0[mid] < jj - 1) lo = mid + 1; else hi = mid; }
      int k = 0;
      for (int col = lo; col < K2_THREADS && colx0[col] <= jj && k < g.kmax; ++col, ++k)
        wt[jj * g.kmax + k] = (colx0[col] == jj ? colw0[col] : 0.f) + (colx1[col] == jj ? colw1[col] : 0.f);
      red_lo[jj] = lo;
      red_n[jj] = k;
    }
    __syncthreads();
  }

  const float* dl = p.dlogits + (long long)n * K * hw;
  const float* sl = p.slogits + (long long)n * C * hw;

  // d*: discriminator logits * log2(e); s*: segmentation logits * log2(e) / T   (exp2 domain)
  float d0[KT], d1[KT], s0[CT], s1[CT];
  float acc0[GRAD ? KT : 1], acc1[GRAD ? KT : 1];
  if constexpr (GRAD) {
#pragma unroll
    for (int k = 0; k < KT; ++k) { acc0[k] = 0.f; acc1[k] = 0.f; }
  }
  int row0 = -1, row1 = -1;
  bool swap = false, open_seg = false;
  float loss_acc = 0.f;

  auto flush_segment = [&]() {
    if constexpr (GRAD) {
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (EXACT || k < K) {
          stage0[k * K2_PITCH + tid] = acc0[k];
          stage1[k * K2_PITCH + tid] = acc1[k];
          acc0[k] = 0.f; acc1[k] = 0.f;
        }
      __syncthreads();
      const int r0 = row0 - i_lo, r1 = row1 - i_lo;
      for (int o = tid; o < K * jspan; o += K2_THREADS) {
        const int jj = o / K;
        const int k = o - jj * K;
        const int lo = red_lo[jj], cnt = red_n[jj];
        const float* wrow = wt + jj * g.kmax;
        const float* q0 = stage0 + k * K2_PITCH + lo;
        const float* q1 = stage1 + k * K2_PITCH + lo;
        float t0 = 0.f, t1 = 0.f;
        for (int i = 0; i < cnt; ++i) {
          const float wk = wrow[i];
          t0 = fmaf(wk, q0[i], t0);
          t1 = fmaf(wk, q1[i], t1);
        }
        blk[(r0 * jspan + jj) * K + k] += t0;
        blk[(r1 * jspan + jj) * K + k] += t1;
      }
      __syncthreads();
    }
  };

#pragma unroll 1
  for (int y = y_begin; y < y_end; ++y) {
    const Tap tapy = ac_tap(g.scale_h, y, g.h);              // CTA-uniform
    const int top = swap ? row1 : row0, bot = swap ? row0 : row1;
    if (!open_seg || tapy.i0 != top || tapy.i1 != bot) {
      if (open_seg) flush_segment();
      open_seg = true;
      bool ld0 = false, ld1 = false;
      int nr0 = row0, nr1 = row1;
      if (row0 == tapy.i0) { swap = false; if (row1 != tapy.i1) { ld1 = true; nr1 = tapy.i1; } }
      else if (row1 == tapy.i0) { swap = true; if (row0 != tapy.i1) { ld0 = true; nr0 = tapy.i1; } }
      else { swap = false; ld0 = true; nr0 = tapy.i0; if (row1 != tapy.i1) { ld1 = true; nr1 = tapy.i1; } }
      if (ld0) {
        k5_load_row<KT, EXACT>(d0, dl, K, hw, nr0, g.w, tapx, LOG2E);
        k5_load_row<CT, EXACT>(s0, sl, C, hw, nr0, g.w, tapx, LOG2E * p.inv_T);
        row0 = nr0;
      }
      if (ld1) {
        k5_load_row<KT, EXACT>(d1, dl, K, hw, nr1, g.w, tapx, LOG2E);
        k5_load_row<CT, EXACT>(s1, sl, C, hw, nr1, g.w, tapx, LOG2E * p.inv_T);
        row1 = nr1;
      }
    }
    if (xvalid) {
      const float w0 = swap ? tapy.l1 : tapy.l0;
      const float w1 = swap ? tapy.l0 : tapy.l1;
      // soft label q = min(softmax(seg / T), clamp)
      float ms = -INFINITY;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) ms = fmaxf(ms, w0 * s0[c] + w1 * s1[c]);
      float q[CT];
      float ss = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          q[c] = fast_exp2((w0 * s0[c] + w1 * s1[c]) - ms);
          ss += q[c];
        }
      const float inv_ss = __fdividef(1.f, ss);
      float sq = 0.f;
#pragma unroll
      for (int c = 0; c < CT; ++c)
        if (EXACT || c < C) {
          q[c] = fminf(q[c] * inv_ss, p.clamp);
          sq += q[c];
        }
      // discriminator log-sum-exp (exp2 domain)
      float md = -INFINITY;
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (EXACT || k < K) md = fmaxf(md, w0 * d0[k] + w1 * d1[k]);
      float sd = 0.f, sqv = 0.f;
#pragma unroll
      for (int k = 0; k < KT; ++k)
        if (EXACT || k < K) {
          const float v = w0 * d0[k] + w1 * d1[k];
          sd += fast_exp2(v - md);
          // the soft label sits in channels [SLOT * C, SLOT * C + C) (a runtime offset for the padded instantiations: their q[]
          // is then indexed dynamically, i.e. lives in local memory -- the two class counts the reference trains are compile-time)
          const int cc = k - SLOT * C;
          if (cc >= 0 && cc < C) sqv = fmaf(q[cc], v, sqv);
        }
      loss_acc += LN2 * ((md + __log2f(sd)) * sq - sqv);
      if constexpr (GRAD) {
        const float scale = sq * __fdividef(1.f, sd);
#pragma unroll
        for (int k = 0; k < KT; ++k)
          if (EXACT || k < K) {
            float gk = fast_exp2((w0 * d0[k] + w1 * d1[k]) - md) * scale;
            const int cc = k - SLOT * C;
            if (cc >= 0 && cc < C) gk -= q[cc];
            acc0[k] = fmaf(w0, gk, acc0[k]);
            acc1[k] = fmaf(w1, gk, acc1[k]);
          }
      }
    }
  }
  if (open_seg) flush_segment();

  loss_acc = warp_sum(loss_acc);
  if (lane == 0) red[warp] = loss_acc;
  __syncthreads();
  if (tid == 0) p.loss_part[tile] = (red[0] + red[1]) + (red[2] + red[3]);
  if (GRAD) {
    float* dst = p.blocks + (long long)tile * blk_floats;
    for (int i = tid; i < blk_floats; i += K2_THREADS) dst[i] = blk[i];
  }
}

__global__ void __launch_bounds__(256) k5_finalize_loss(const float* loss_part, int tiles, double count, float* out2) {
  __shared__ double sl[8];
  double l = 0.0;
  for (int i = threadIdx.x; i < tiles; i += 256) l += (double)loss_part[i];
  l = warp_sum_d(l);
  if ((threadIdx.x & 31) == 0) sl[threadIdx.x >> 5] = l;
  __syncthreads();
  if (threadIdx.x == 0) {
    double L = 0.0;
    for (int i = 0; i < 8; ++i) L += sl[i];
    out2[0] = (float)(L / count);
    out2[1] = (float)count;
  }
}

// grad_d[n,k,i,j] = grad_out / (N*H*W) * sum over the tiles touching (i,j) of their partial block (any channel count).
// blockIdx.z = image * nchunk + channel chunk: a thread owns K5F_CC channels of one low-res pixel in registers, so the
// (strided) partial-block reads of a pixel are all in flight at once instead of one dependent load per channel.
constexpr int K5F_CC = 20;
__global__ void __launch_bounds__(128) k5_finalize_grad(const K2Geom g, const float* __restrict__ blocks, const float* loss_out2,
                                                        const float* grad_out, float* __restrict__ grad, int nchunk) {
  const int j = blockIdx.x * 128 + threadIdx.x;
  const int i = blockIdx.y;
  const int n = blockIdx.z / nchunk;
  const int c0 = (blockIdx.z - n * nchunk) * K5F_CC;
  if (j >= g.w) return;
  const int nc = min(K5F_CC, g.C - c0);
  const float scale = (grad_out ? grad_out[0] : 1.f) / loss_out2[1];
  const long long blk_floats = (long long)g.ispan_max * g.jspan_max * g.C;
  const long long hw = (long long)g.h * g.w;
  float acc[K5F_CC];
#pragma unroll
  for (int c = 0; c < K5F_CC; ++c) acc[c] = 0.f;
  const int ya = ac_first_dst(g.scale_h, i - 1, g.h, g.H), yb = ac_first_dst(g.scale_h, i + 1, g.h, g.H);
  const int xa = ac_first_dst(g.scale_w, j - 1, g.w, g.W), xb = ac_first_dst(g.scale_w, j + 1, g.w, g.W);
  if (ya < yb && xa < xb) {
    const int ty0 = ya / K2_TILE_H, ty1 = (yb - 1) / K2_TILE_H;
    const int tx0 = xa / K2_TILE_W, tx1 = (xb - 1) / K2_TILE_W;
    for (int ty = ty0; ty <= ty1; ++ty) {                         // same tile order as before: identical sums
      const int li = i - (int)(g.scale_h * (float)(ty * K2_TILE_H));
      if (li < 0 || li >= g.ispan_max) continue;
      for (int tx = tx0; tx <= tx1; ++tx) {
        const int lj = j - (int)(g.scale_w * (float)(tx * K2_TILE_W));
        if (lj < 0 || lj >= g.jspan_max) continue;
        const long long tile = ((long long)n * g.tiles_y + ty) * g.tiles_x + tx;
        const float* src = blocks + tile * blk_floats + ((long long)li * g.jspan_max + lj) * g.C + c0;
#pragma unroll
        for (int c = 0; c < K5F_CC; ++c)
          if (c < nc) acc[c] += src[c];
      }
    }
  }
  float* dst = grad + ((long long)n * g.C + c0) * hw + (long long)i * g.w + j;
#pragma unroll
  for (int c = 0; c < K5F_CC; ++c)
    if (c < nc) dst[c * hw] = acc[c] * scale;
}

long long k5_workspace_bytes(int N, int C, int h, int w, int H, int W) {
  K2Geom g;
  k2_geometry(g, N, 2 * C, h, w, H, W);
  return (k2_tiles(g) + k2_tiles(g) * k2_block_floats(g)) * 4 + 256;
}

template <int CT, bool EXACT>
static int k5_main_launch(const K5Params& p, bool grad, int slot, cudaStream_t stream) {
  const K2Geom& g = p.g;
  const size_t smem = ((size_t)2 * 2 * CT * K2_PITCH + (size_t)g.ispan_max * g.jspan_max * g.C + (size_t)g.jspan_max * (g.kmax + 2) +
                       4 * K2_THREADS + 8) * 4;
  B200SEG_CHECK_ARG(smem <= 200 * 1024, "fada_softce: tile footprint %zu B exceeds shared memory (resize ratio too small)", smem);
  const int tiles = (int)k2_tiles(g);
#define K5_LAUNCH(G, S)                                                                                                      \
  do {                                                                                                                       \
    static bool configured = false;                                                                                          \
    if (!configured) {                                                                                                       \
      B200SEG_CUDA(cudaFuncSetAttribute(k5_fada_softce_main<CT, G, EXACT, S>, cudaFuncAttributeMaxDynamicSharedMemorySize,   \
                                        200 * 1024));                                                                        \
      configured = true;                                                                                                     \
    }                                                                                                                        \
    k5_fada_softce_main<CT, G, EXACT, S><<<tiles, K2_THREADS, smem, stream>>>(p);                                             \
  } while (0)
  profile_begin(11, stream);
  if (grad) { if (slot == 0) K5_LAUNCH(true, 0); else K5_LAUNCH(true, 1); }
  else { if (slot == 0) K5_LAUNCH(false, 0); else K5_LAUNCH(false, 1); }
  profile_end(11, stream);
#undef K5_LAUNCH
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int k5_forward(const float* dlogits, const float* slogits, int N, int C, int h, int w, int H, int W, float inv_T, float clamp,
               int slot, int need_grad, void* workspace, long long workspace_bytes, float* loss_out2, cudaStream_t stream) {
  B200SEG_CHECK_ARG(dlogits && slogits && workspace && loss_out2, "fada_softce_forward: null pointer");
  B200SEG_CHECK_ARG(N > 0 && C > 0 && h > 0 && w > 0 && H > 0 && W > 0, "fada_softce_forward: bad shape");
  B200SEG_CHECK_ARG(slot == 0 || slot == 1, "fada_softce_forward: slot must be 0 (source) or 1 (target)");
  B200SEG_CHECK_ARG(C <= 32, "fada_softce_forward: num_classes=%d > 32 is not supported by the fused kernel (like K2 / K4); use the "
                    "materialised soft_ce path", C);
  B200SEG_CHECK_ARG(workspace_bytes >= k5_workspace_bytes(N, C, h, w, H, W), "fada_softce_forward: workspace too small");
  K5Params p;
  k2_geometry(p.g, N, 2 * C, h, w, H, W);
  const long long tiles = k2_tiles(p.g);
  p.dlogits = dlogits; p.slogits = slogits; p.inv_T = inv_T; p.clamp = clamp;
  p.loss_part = reinterpret_cast<float*>(workspace);
  p.blocks = p.loss_part + tiles;
  int rc;
  // compile-time class counts for the two the reference trains (19: Cityscapes / GTA5, 2: Kvasir / BLI); any other count up to 32
  // runs a padded instantiation with the count as a runtime bound (the widest ones trade registers for generality)
  if (C == 19) rc = k5_main_launch<19, true>(p, need_grad != 0, slot, stream);
  else if (C == 2) rc = k5_main_launch<2, true>(p, need_grad != 0, slot, stream);
  else if (C <= 8) rc = k5_main_launch<8, false>(p, need_grad != 0, slot, stream);
  else if (C <= 16) rc = k5_main_launch<16, false>(p, need_grad != 0, slot, stream);
  else if (C <= 24) rc = k5_main_launch<24, false>(p, need_grad != 0, slot, stream);
  else rc = k5_main_launch<32, false>(p, need_grad != 0, slot, stream);
  if (rc) return rc;
  k5_finalize_loss<<<1, 256, 0, stream>>>(p.loss_part, (int)tiles, (double)N * H * W, loss_out2);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int k5_backward(const void* workspace, int N, int C, int h, int w, int H, int W, const float* loss_out2, const float* grad_out,
                float* grad_d, cudaStream_t stream) {
  B200SEG_CHECK_ARG(workspace && loss_out2 && grad_d, "fada_softce_backward: null pointer");
  K2Geom g;
  k2_geometry(g, N, 2 * C, h, w, H, W);
  const long long tiles = k2_tiles(g);
  const float* blocks = reinterpret_cast<const float*>(workspace) + tiles;
  const int nchunk = ceil_div(g.C, K5F_CC);
  dim3 grid(ceil_div(w, 128), h, N * nchunk);
  k5_finalize_grad<<<grid, 128, 0, stream>>>(g, blocks, loss_out2, grad_out, grad_d, nchunk);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// ---------------------------------------------------------------------------------------------
// Materialising align-corners bilinear upsample (forward) and its adjoint (gather form, no atomics)
// ---------------------------------------------------------------------------------------------
template <int FMA>
__global__ void __launch_bounds__(256) upsample_fwd_kernel(const float* __restrict__ in, float* __restrict__ out, int NC,
                                                           int h, int w, int H, int W, float sh, float sw) {
  const int x = blockIdx.x * 256 + threadIdx.x;
  const int y = blockIdx.y;
  if (x >= W) return;
  const Tap ty = ac_tap(sh, y, h), tx = ac_tap(sw, x, w);
  for (int nc = blockIdx.z; nc < NC; nc += gridDim.z) {
    const float* src = in + (long long)nc * h * w;
    const float a = __ldg(src + (long long)ty.i0 * w + tx.i0), b = __ldg(src + (long long)ty.i0 * w + tx.i1);
    const float c = __ldg(src + (long long)ty.i1 * w + tx.i0), d = __ldg(src + (long long)ty.i1 * w + tx.i1);
    float v;
    if (FMA == 0) v = ty.l0 * (tx.l0 * a + tx.l1 * b) + ty.l1 * (tx.l0 * c + tx.l1 * d);
    else if (FMA == 1) v = fmaf(ty.l0, fmaf(tx.l0, a, tx.l1 * b), ty.l1 * fmaf(tx.l0, c, tx.l1 * d));
    else if (FMA == 2) v = fmaf(ty.l1, fmaf(tx.l1, d, tx.l0 * c), ty.l0 * fmaf(tx.l1, b, tx.l0 * a));
    else v = __fadd_rn(__fmul_rn(ty.l0, __fadd_rn(__fmul_rn(tx.l0, a), __fmul_rn(tx.l1, b))),
                       __fmul_rn(ty.l1, __fadd_rn(__fmul_rn(tx.l0, c), __fmul_rn(tx.l1, d))));
    out[((long long)nc * H + y) * W + x] = v;
  }
}

// Streaming form for W % 4 == 0 (the ATen-exact contraction, modes 0/1): one thread owns four adjacent output columns of
// one plane and walks UPS_ROWS output rows; the horizontal lerps of the two source rows live in registers and are reused
// for every output row between them, so an output float4 costs ~15 instructions and one 16-byte streaming store.
// 8 x 19 x 512 x 1024 (319 MB written): 50 us = 6.4 TB/s, the HBM write rate of a plain fill (47 us); the
// one-element-per-thread kernel it replaces took 197 us.
constexpr int UPS_ROWS = 16;
__global__ void __launch_bounds__(256) upsample_fwd_v4_kernel(const float* __restrict__ in, float* __restrict__ out, int h, int w,
                                                              int H, int W, float sh, float sw) {
  const int x0 = (blockIdx.x * 256 + threadIdx.x) * 4;
  if (x0 >= W) return;
  const long long nc = blockIdx.z;
  const float* src = in + nc * h * w;
  Tap tx[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) tx[e] = ac_tap(sw, x0 + e, w);
  const int y_begin = blockIdx.y * UPS_ROWS, y_end = min(H, y_begin + UPS_ROWS);
  float t[4], u[4];                          // horizontal lerps of source rows r0 (upper) / r1 (lower)
  int r0 = -1, r1 = -1;
  float* dst = out + (nc * H + y_begin) * W + x0;
  for (int y = y_begin; y < y_end; ++y, dst += W) {
    const Tap ty = ac_tap(sh, y, h);
    if (ty.i0 != r0 || ty.i1 != r1) {
      if (ty.i0 == r1) {
#pragma unroll
        for (int e = 0; e < 4; ++e) t[e] = u[e];
      } else {
        const float* p = src + (long long)ty.i0 * w;
#pragma unroll
        for (int e = 0; e < 4; ++e) t[e] = fmaf(tx[e].l0, __ldg(p + tx[e].i0), tx[e].l1 * __ldg(p + tx[e].i1));
      }
      if (ty.i1 == ty.i0) {
#pragma unroll
        for (int e = 0; e < 4; ++e) u[e] = t[e];
      } else {
        const float* p = src + (long long)ty.i1 * w;
#pragma unroll
        for (int e = 0; e < 4; ++e) u[e] = fmaf(tx[e].l0, __ldg(p + tx[e].i0), tx[e].l1 * __ldg(p + tx[e].i1));
      }
      r0 = ty.i0; r1 = ty.i1;
    }
    float4 v;
    v.x = fmaf(ty.l0, t[0], ty.l1 * u[0]);
    v.y = fmaf(ty.l0, t[1], ty.l1 * u[1]);
    v.z = fmaf(ty.l0, t[2], ty.l1 * u[2]);
    v.w = fmaf(ty.l0, t[3], ty.l1 * u[3]);
    st_stream_f4(dst, v);
  }
}

int upsample_fwd_launch(const float* in, float* out, int NC, int h, int w, int H, int W, int fma_mode, cudaStream_t stream) {
  B200SEG_CHECK_ARG(in && out && NC > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_bilinear_forward: bad arguments");
  const float sh = ac_scale(h, H), sw = ac_scale(w, W);
  if (fma_mode <= 1 && W % 4 == 0 && (reinterpret_cast<uintptr_t>(out) & 15) == 0 && NC <= 65535) {
    dim3 grid(ceil_div(W, 1024), ceil_div(H, UPS_ROWS), NC);
    upsample_fwd_v4_kernel<<<grid, 256, 0, stream>>>(in, out, h, w, H, W, sh, sw);
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  dim3 grid(ceil_div(W, 256), H, NC < 64 ? NC : 64);
  switch (fma_mode) {
    case 0: upsample_fwd_kernel<0><<<grid, 256, 0, stream>>>(in, out, NC, h, w, H, W, sh, sw); break;
    case 1: upsample_fwd_kernel<1><<<grid, 256, 0, stream>>>(in, out, NC, h, w, H, W, sh, sw); break;
    case 2: upsample_fwd_kernel<2><<<grid, 256, 0, stream>>>(in, out, NC, h, w, H, W, sh, sw); break;
    default: upsample_fwd_kernel<3><<<grid, 256, 0, stream>>>(in, out, NC, h, w, H, W, sh, sw); break;
  }
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

__global__ void __launch_bounds__(128) upsample_bwd_kernel(const float* __restrict__ gout, float* __restrict__ gin, int NC,
                                                           int h, int w, int H, int W, float sh, float sw) {
  const int j = blockIdx.x * 128 + threadIdx.x;
  const int i = blockIdx.y;
  if (j >= w) return;
  const int ya = ac_first_dst(sh, i - 1, h, H), yb = ac_first_dst(sh, i + 1, h, H);
  const int xa = ac_first_dst(sw, j - 1, w, W), xb = ac_first_dst(sw, j + 1, w, W);
  for (int nc = blockIdx.z; nc < NC; nc += gridDim.z) {
    const float* src = gout + (long long)nc * H * W;
    float acc = 0.f;
    for (int y = ya; y < yb; ++y) {
      const Tap ty = ac_tap(sh, y, h);
      const float wy = (ty.i0 == i ? ty.l0 : 0.f) + (ty.i1 == i ? ty.l1 : 0.f);
      if (wy == 0.f) continue;
      float racc = 0.f;
      for (int x = xa; x < xb; ++x) {
        const Tap tx = ac_tap(sw, x, w);
        const float wx = (tx.i0 == j ? tx.l0 : 0.f) + (tx.i1 == j ? tx.l1 : 0.f);
        racc = fmaf(wx, __ldg(src + (long long)y * W + x), racc);
      }
      acc = fmaf(wy, racc, acc);
    }
    gin[((long long)nc * h + i) * w + j] = acc;
  }
}

// Streaming adjoint for W % 4 == 0, W <= 1024 (one 256-thread block spans a whole output row).  A block owns UPB_ROWS
// low-res rows of one plane: its threads own four adjacent output columns each and walk the output rows that feed those
// low-res rows (16-byte streaming loads), reducing VERTICALLY in registers; each time a low-res row is complete the block
// parks the 4 KB row of vertical sums in shared memory and the first w threads reduce it HORIZONTALLY over their column
// windows.  Every low-res element is produced by exactly one thread in a fixed order: deterministic, no atomics.
constexpr int UPB_ROWS = 8;
__global__ void __launch_bounds__(256) upsample_bwd_v4_kernel(const float* __restrict__ gout, float* __restrict__ gin, int h, int w,
                                                              int H, int W, float sh, float sw) {
  __shared__ __align__(16) float vrow[1024];
  const int x0 = threadIdx.x * 4;
  const bool xin = x0 < W;
  const long long nc = blockIdx.z;
  const int ia = blockIdx.y * UPB_ROWS, ib = min(h, ia + UPB_ROWS);
  const int ya = ac_first_dst(sh, ia - 1, h, H), yb = ac_first_dst(sh, ib, h, H);     // output rows touching rows [ia, ib)
  // horizontal window of source column j = threadIdx.x
  const int j = threadIdx.x;
  int xa = 0, xb = 0;
  if (j < w) { xa = ac_first_dst(sw, j - 1, w, W); xb = ac_first_dst(sw, j + 1, w, W); }
  const float* src = gout + nc * H * W + x0;
  float* dstp = gin + nc * h * w;
  float accA[4] = {0.f, 0.f, 0.f, 0.f}, accB[4] = {0.f, 0.f, 0.f, 0.f};     // vertical sums of low-res rows r, r + 1
  int r = (ya < yb) ? (int)(sh * (float)ya) : ia;

  auto emit = [&](int row) {                // block-uniform: park row `row`'s vertical sums, reduce them horizontally
    __syncthreads();                        // previous readers of vrow are done
    if (xin) *reinterpret_cast<float4*>(&vrow[x0]) = make_float4(accA[0], accA[1], accA[2], accA[3]);
    __syncthreads();
    if (j < w && row >= ia && row < ib) {
      float a = 0.f;
      for (int x = xa; x < xb; ++x) {
        const Tap tx = ac_tap(sw, x, w);
        const float wx = (tx.i0 == j ? tx.l0 : 0.f) + (tx.i1 == j ? tx.l1 : 0.f);
        a = fmaf(wx, vrow[x], a);
      }
      dstp[(long long)row * w + j] = a;
    }
  };

  for (int y = ya; y < yb; ++y) {
    const Tap ty = ac_tap(sh, y, h);
    while (ty.i0 > r) {                     // row r is complete (block-uniform)
      emit(r);
#pragma unroll
      for (int e = 0; e < 4; ++e) { accA[e] = accB[e]; accB[e] = 0.f; }
      ++r;
    }
    float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
    if (xin) g = ld_stream_f4(src + (long long)y * W);
    const float wa = (ty.i1 == ty.i0) ? ty.l0 + ty.l1 : ty.l0;               // bottom border: both taps on row i0
    const float wb = (ty.i1 == ty.i0) ? 0.f : ty.l1;
    accA[0] = fmaf(wa, g.x, accA[0]); accA[1] = fmaf(wa, g.y, accA[1]); accA[2] = fmaf(wa, g.z, accA[2]); accA[3] = fmaf(wa, g.w, accA[3]);
    accB[0] = fmaf(wb, g.x, accB[0]); accB[1] = fmaf(wb, g.y, accB[1]); accB[2] = fmaf(wb, g.z, accB[2]); accB[3] = fmaf(wb, g.w, accB[3]);
  }
  // rows r and r + 1 are still open; rows of [ia, ib) that no output row touches (downsampling) are zero
  for (int row = r; row < ib; ++row) {
    emit(row);
#pragma unroll
    for (int e = 0; e < 4; ++e) { accA[e] = accB[e]; accB[e] = 0.f; }
  }
  if (ya >= yb || (int)(sh * (float)ya) > ia) {                              // leading rows without contributions
    const int first = (ya < yb) ? (int)(sh * (float)ya) : ib;
    for (int row = ia; row < min(first, ib); ++row)
      if (j < w) dstp[(long long)row * w + j] = 0.f;
  }
}

int upsample_bwd_launch(const float* gout, float* gin, int NC, int h, int w, int H, int W, cudaStream_t stream) {
  B200SEG_CHECK_ARG(gout && gin && NC > 0 && h > 0 && w > 0 && H > 0 && W > 0, "upsample_bilinear_backward: bad arguments");
  if (W % 4 == 0 && W <= 1024 && w <= 256 && NC <= 65535 && (reinterpret_cast<uintptr_t>(gout) & 15) == 0) {
    dim3 gridv(1, ceil_div(h, UPB_ROWS), NC);
    upsample_bwd_v4_kernel<<<gridv, 256, 0, stream>>>(gout, gin, h, w, H, W, ac_scale(h, H), ac_scale(w, W));
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  dim3 grid(ceil_div(w, 128), h, NC < 1024 ? NC : 1024);
  upsample_bwd_kernel<<<grid, 128, 0, stream>>>(gout, gin, NC, h, w, H, W, ac_scale(h, H), ac_scale(w, W));
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

}  // namespace b200seg
