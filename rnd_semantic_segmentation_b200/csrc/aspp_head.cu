// K1: the fused four-dilation ASPP classifier head (DeepLabV2), forward and backward.
//
// Replaces (reference file:line): ASPP_Classifier_V2.forward, core/models/classifiers/aspp/classifier.py:26-29
//   out = sum_r Conv2d(Cin, C, 3, padding=r, dilation=r)(x),  r in dilation_series (6/12/18/24)
// and its autograd backward (dgrad, wgrad, bias grad).
//
// Formulation ("tap-packed GEMM").  With T = 8R+1 distinct taps (the R centre taps hit the same
// pixel, so their weights are pre-summed) and offset d_t of tap t:
//     out[p, c] = bias[c] + sum_t sum_ci X[p + d_t, ci] * W[t, c, ci]
// Padding the class dimension to an MMA-friendly N (19 -> 32) would waste 41 % of the tensor
// pipe and leave it shared-memory-bound (a 128 x 32 x 16 MMA re-reads 4 KB of A for 16 cycles of
// math).  Instead (t, c) is packed into ONE GEMM dimension j = t*C + c  (33*19 = 627 -> 640):
//     fwd    Yt[j, p]   = sum_ci Wp[j, ci] * Xp[p, ci]          M=640  N=P     K=Cin   (K-major x K-major)
//            out[p, c]  = bias[c] + sum_t Yt[t*C+c, p + d_t]     shift-and-add gather, coalesced along p
//     G'[p, j]          = gO[p - d_t, c]                         bf16 "im2col of the output gradient"
//     dgrad  dX[ci, p]  = sum_j WpT[ci, j] * G'[p, j]            M=Cin  N=P     K=640   (writes fp32 NCHW directly)
//     wgrad  dWp[j, ci] = sum_p G'[p, j] * Xp[p, ci]             M=640  N=Cin   K=P     (MN-major x MN-major, split-K)
// All three GEMMs run on the tcgen05 core in gemm_sm100.cuh with 98 % useful MMA work at C=19.
// Operands are bf16 (features, packed weights, output gradient), accumulation is fp32 in TMEM.
#include <limits.h>
#include "common.cuh"
#include "gemm_sm100.cuh"

namespace b200seg {

constexpr int MAX_RATES = 8;
constexpr int MAX_TAPS = 8 * MAX_RATES + 1;

struct TapTable {
  int n_taps;              // 8R + 1 (last = merged centre)
  int dy[MAX_TAPS], dx[MAX_TAPS];
};

static void make_taps(TapTable& tt, const int* rates, int R) {
  int t = 0;
  for (int r = 0; r < R; ++r)
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx) {
        if (ky == 1 && kx == 1) continue;
        tt.dy[t] = (ky - 1) * rates[r];
        tt.dx[t] = (kx - 1) * rates[r];
        ++t;
      }
  tt.dy[t] = 0; tt.dx[t] = 0;
  tt.n_taps = t + 1;
}

int aspp_nj(int C, int R) { return ceil_div((8 * R + 1) * C, 128) * 128; }

struct PtrList {
  const float* p[MAX_RATES];
};
struct MutPtrList {
  float* p[MAX_RATES];
};

// ------------------------------------------------------------------------------------------
// pack weights: R x [C, Cin, 3, 3] fp32 -> Wp [NJ, Cin] bf16, WpT [Cin, NJ] bf16, bias_sum [C]
// ------------------------------------------------------------------------------------------
// A block owns 8 input channels x all classes x all branches: it reads, per (branch, class), the 72 contiguous floats
// w[r][c][ci0 .. ci0+8)[3][3] into shared memory (coalesced), then writes 8 full rows of WpT (contiguous along j) and one 16-byte
// segment of every Wp row -- no strided 2-byte scatter (the per-element version took ~30 us of every training step; the weights
// change every step).  Element values and the centre-tap summation order ((w0+w1)+w2)+w3 are those of the per-element version.
constexpr int PW_CI = 8;
// tab[j] >= 0: offset of w_s[r][c][0][k] for an off-centre row; -1 - c: centre row of class c (sum over branches); INT_MIN: padding
__device__ __forceinline__ float packed_weight(const float* __restrict__ w_s, const int* __restrict__ tab, int R, int C, int j, int ci_l) {
  const int e = tab[j];
  if (e >= 0) return w_s[e + ci_l * 9];
  float v = 0.f;
  if (e != INT_MIN) {
    const int c = -1 - e;
    for (int r = 0; r < R; ++r) v += w_s[((r * C + c) * PW_CI + ci_l) * 9 + 4];
  }
  return v;
}
__global__ void __launch_bounds__(256) pack_weights_kernel(PtrList w, PtrList b, int R, int C, int Cin, int NJ,
                                                           __nv_bfloat16* __restrict__ Wp, __nv_bfloat16* __restrict__ WpT,
                                                           float* __restrict__ bias_sum) {
  extern __shared__ float pw_s[];                                          // [R][C][PW_CI][9] floats, then the row table [NJ]
  int* tab = reinterpret_cast<int*>(pw_s + R * C * PW_CI * 9);
  const int ci0 = blockIdx.x * PW_CI;
  if (blockIdx.x == 0 && threadIdx.x < C) {
    const int idx = threadIdx.x;
    float s = b.p[0] ? b.p[0][idx] : 0.f;
    for (int r = 1; r < R; ++r) s += b.p[r] ? b.p[r][idx] : 0.f;          // ((b0+b1)+b2)+b3, the reference's order
    bias_sum[idx] = s;
  }
  for (int j = threadIdx.x; j < NJ; j += 256) {                            // the only integer divisions of the kernel
    const int t = j / C, c = j - t * C;
    int e = INT_MIN;
    if (t < 8 * R) {
      const int r = t >> 3, q = t & 7;
      e = ((r * C + c) * PW_CI) * 9 + (q < 4 ? q : q + 1);                 // skip the centre (k == 4)
    } else if (t == 8 * R) {
      e = -1 - c;
    }
    tab[j] = e;
  }
  constexpr int SEG = PW_CI * 9;
  for (int i = threadIdx.x; i < R * C * SEG; i += 256) {                   // independent loads: ~21 in flight per thread
    const int rc = i / SEG, off = i - rc * SEG;
    const int r = rc / C, c = rc - r * C;
    pw_s[i] = __ldg(w.p[r] + ((long long)c * Cin + ci0) * 9 + off);
  }
  __syncthreads();
  // WpT[ci][j]: pairs of j (NJ is a multiple of 128), contiguous along j
  const int half = NJ >> 1;
  for (int ci_l = 0; ci_l < PW_CI; ++ci_l) {
    for (int jp = threadIdx.x; jp < half; jp += 256) {
      const int j = 2 * jp;
      const __nv_bfloat162 v = __floats2bfloat162_rn(packed_weight(pw_s, tab, R, C, j, ci_l), packed_weight(pw_s, tab, R, C, j + 1, ci_l));
      *reinterpret_cast<__nv_bfloat162*>(WpT + (long long)(ci0 + ci_l) * NJ + j) = v;
    }
  }
  // Wp[j][ci0 .. ci0+8): one 16-byte store per row
  for (int j = threadIdx.x; j < NJ; j += 256) {
    uint32_t w4[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const __nv_bfloat162 v = __floats2bfloat162_rn(packed_weight(pw_s, tab, R, C, j, 2 * e), packed_weight(pw_s, tab, R, C, j, 2 * e + 1));
      w4[e] = *reinterpret_cast<const uint32_t*>(&v);
    }
    *reinterpret_cast<uint4*>(Wp + (long long)j * Cin + ci0) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
  }
}

// ------------------------------------------------------------------------------------------
// forward gather: logits[n,c,y,x] = bias[c] + sum_t Yt[t*C+c][p(n, y+dy_t, x+dx_t)]
// ------------------------------------------------------------------------------------------
// One thread per low-res pixel, all classes in registers: per tap one bounds test and C loads at a fixed stride
// (coalesced along x across the warp), so the kernel issues ~3 instructions per Yt element and runs at the HBM rate
// of the Yt read instead of being issue-bound on per-element address arithmetic.
constexpr int GATHER_THREADS = 64;
template <int CT>
__global__ void __launch_bounds__(GATHER_THREADS) head_gather_kernel(const float* __restrict__ Yt, long long ypitch, TapTable tt,
                                                                     const float* __restrict__ bias_sum, int C, int nchunk,
                                                                     int h, int w, float* __restrict__ logits) {
  // blockIdx.z = image * nchunk + class chunk; this thread owns classes [c0, c0 + nc) of one pixel (nc <= CT)
  const int n = blockIdx.z / nchunk;
  const int c0 = (blockIdx.z - n * nchunk) * CT;
  const int nc = min(CT, C - c0);
  const int xq = blockIdx.x * GATHER_THREADS + threadIdx.x;
  const int y = blockIdx.y;
  if (xq >= w) return;
  const long long pbase = (long long)n * h * w;
  const long long cstep = ypitch * 4;                         // bytes between classes of one tap
  float acc[CT];
#pragma unroll
  for (int c = 0; c < CT; ++c) acc[c] = (c < nc) ? bias_sum[c0 + c] : 0.f;
  const char* tap_base = reinterpret_cast<const char*>(Yt + pbase + (long long)y * w + xq) + cstep * c0;
  const long long tstep = cstep * C;                          // bytes between taps
  constexpr int TG = 3;                                        // taps per batch: TG * CT loads in flight per thread
#pragma unroll 1
  for (int t0 = 0; t0 < tt.n_taps; t0 += TG, tap_base += TG * tstep) {
    float v[TG][CT];
#pragma unroll
    for (int k = 0; k < TG; ++k) {
      const int t = min(t0 + k, tt.n_taps - 1);
      const int dy = tt.dy[t], dx = tt.dx[t];
      const int yy = y + dy, xx = xq + dx;
      const bool inb = (t0 + k < tt.n_taps) && yy >= 0 && yy < h && xx >= 0 && xx < w;
      const char* src = tap_base + k * tstep + ((long long)dy * w + dx) * 4;
#pragma unroll
      for (int c = 0; c < CT; ++c) {
        v[k][c] = 0.f;
        if (inb && c < nc) v[k][c] = __ldcs(reinterpret_cast<const float*>(src));
        src += cstep;
      }
    }
#pragma unroll
    for (int k = 0; k < TG; ++k)
#pragma unroll
      for (int c = 0; c < CT; ++c) acc[c] += v[k][c];
  }
  const long long hw = (long long)h * w;
  float* dst = logits + ((long long)n * C + c0) * hw + (long long)y * w + xq;
#pragma unroll
  for (int c = 0; c < CT; ++c)
    if (c < nc) dst[c * hw] = acc[c];
}

// ------------------------------------------------------------------------------------------
// backward prep: gO fp32 NCHW [N,C,hw] -> gOt bf16 [P][32]; bias grad; G' bf16 [P][NJ]
// ------------------------------------------------------------------------------------------
// gO fp32 NCHW -> gOc bf16 [N][C][hw] (same layout, half the bytes): the operand build_gprime_t_kernel shifts
__global__ void __launch_bounds__(256) grad_to_bf16_planes_kernel(const float* __restrict__ g, long long n,
                                                                  __nv_bfloat16* __restrict__ gOc) {
  const long long i = (blockIdx.x * 256LL + threadIdx.x) * 2;
  if (i + 1 < n) {
    *reinterpret_cast<__nv_bfloat162*>(gOc + i) = __floats2bfloat162_rn(g[i], g[i + 1]);
  } else if (i < n) {
    gOc[i] = __float2bfloat16(g[i]);
  }
}

// deterministic per-class sum over all pixels (bias gradient), one block per class
__global__ void __launch_bounds__(256) bias_grad_kernel(const float* __restrict__ g, int N, int C, int hw, MutPtrList gb, int R) {
  __shared__ double red[8];
  const int c = blockIdx.x;
  double acc = 0.0;
  for (int n = 0; n < N; ++n) {
    const float* src = g + ((long long)n * C + c) * hw;
    for (int s = threadIdx.x; s < hw; s += 256) acc += (double)src[s];
  }
  acc = warp_sum_d(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    double t = 0.0;
    for (int i = 0; i < 8; ++i) t += red[i];
    for (int r = 0; r < R; ++r)
      if (gb.p[r]) gb.p[r][c] = (float)t;
  }
}

// G't[j][p] = gO[c][p - d_t]  (j = t*C + c; zero outside the image and for j >= T*C), bf16 [NJ][Ppitch].
// In this (tap, class)-major layout every row is a SHIFTED COPY of one class plane of the output gradient with zero
// fill at the image borders, so the "im2col of the gradient" is a pure streaming copy: one thread per 4-byte word
// (two pixels), coalesced 128-byte loads and stores.  FAST: w even and every dx even (the DeepLab rates 6/12/18/24),
// so a word never straddles an image row and the shifted source word is 4-byte aligned; otherwise two 2-byte loads.
// dgrad consumes G't as the MN-major B operand, wgrad as the K-major A operand of the same tcgen05 kernel.
constexpr int GPT_ITERS = 8;                 // 4-byte words per thread; a block covers 256 * 2 * GPT_ITERS pixels of one row
template <bool FAST>
__global__ void __launch_bounds__(256) build_gprime_t_kernel(const __nv_bfloat16* __restrict__ gOc, TapTable tt, int C, int h, int w,
                                                             int N, long long Ppitch, __nv_bfloat16* __restrict__ Gp) {
  const int j = blockIdx.y;                                  // row of G't
  const int t = j / C, c = j - t * C;
  const int hw = h * w;
  const long long P = (long long)N * hw;
  long long p0 = (long long)blockIdx.x * (512 * GPT_ITERS) + threadIdx.x * 2;     // first of this thread's two pixels
  uint32_t* out = reinterpret_cast<uint32_t*>(Gp + (long long)j * Ppitch);          // Ppitch is even: words are aligned
  if (t >= tt.n_taps) {                                      // padding rows of the packed dimension
#pragma unroll
    for (int it = 0; it < GPT_ITERS; ++it, p0 += 512)
      if (p0 < P) out[p0 >> 1] = 0u;
    return;
  }
  const int dy = tt.dy[t], dx = tt.dx[t];
  const unsigned short* planes = reinterpret_cast<const unsigned short*>(gOc);
  if (FAST) {
    // (image, row, column) of p0, advanced by 512 pixels per iteration without divisions
    int n = (int)(p0 / hw);
    int sidx = (int)(p0 - (long long)n * hw);
    int y = sidx / w, x = sidx - y * w;
    const int step_y = 512 / w, step_x = 512 - step_y * w;
#pragma unroll
    for (int it = 0; it < GPT_ITERS; ++it, p0 += 512) {
      if (p0 < P) {
        const int ys = y - dy, xs = x - dx;
        uint32_t word = 0;
        if (ys >= 0 && ys < h && xs >= 0 && xs < w)
          word = __ldg(reinterpret_cast<const uint32_t*>(planes + ((long long)n * C + c) * hw + ys * w + xs));
        out[p0 >> 1] = word;
      }
      x += step_x; y += step_y;
      if (x >= w) { x -= w; ++y; }
      while (y >= h) { y -= h; ++n; }
    }
  } else {
#pragma unroll 1
    for (int it = 0; it < GPT_ITERS; ++it, p0 += 512) {
      if (p0 >= P) break;
      uint32_t word = 0;
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const long long pp = p0 + e;
        if (pp < P) {
          const int n = (int)(pp / hw);
          const int sidx = (int)(pp - (long long)n * hw);
          const int y = sidx / w, x = sidx - y * w;
          const int ys = y - dy, xs = x - dx;
          if (ys >= 0 && ys < h && xs >= 0 && xs < w)
            word |= (uint32_t)__ldg(planes + ((long long)n * C + c) * hw + (long long)ys * w + xs) << (16 * e);
        }
      }
      out[p0 >> 1] = word;                                   // may spill one element into the row padding
    }
  }
}

// Same copy with 16-byte stores: one thread per 8 pixels (requires w % 8 == 0 so a vector never straddles an image row,
// and even dx so the four shifted source words are 4-byte aligned).
constexpr int GPT8_ITERS = 4;                // 16-byte vectors per thread; a block covers 256 * 8 * GPT8_ITERS pixels
__global__ void __launch_bounds__(256) build_gprime_t8_kernel(const __nv_bfloat16* __restrict__ gOc, TapTable tt, int C, int h, int w,
                                                              int N, long long Ppitch, __nv_bfloat16* __restrict__ Gp) {
  const int j = blockIdx.y;
  const int t = j / C, c = j - t * C;
  const int hw = h * w;
  const int P = N * hw;                                  // (< 2^31: checked by the host)
  int p0 = (int)blockIdx.x * (2048 * GPT8_ITERS) + (int)threadIdx.x * 8;      // 32-bit index math: the per-thread set-up (three
  uint4* out = reinterpret_cast<uint4*>(Gp + (long long)j * Ppitch);          // divisions) was most of this kernel's instructions
  if (t >= tt.n_taps) {
#pragma unroll
    for (int it = 0; it < GPT8_ITERS; ++it, p0 += 2048)
      if (p0 < P) out[p0 >> 3] = make_uint4(0, 0, 0, 0);
    return;
  }
  const int dy = tt.dy[t], dx = tt.dx[t];
  const unsigned short* planes = reinterpret_cast<const unsigned short*>(gOc);
  int n = p0 / hw;
  int sidx = p0 - n * hw;
  int y = sidx / w, x = sidx - y * w;
  const int step_y = 2048 / w, step_x = 2048 - step_y * w;
#pragma unroll
  for (int it = 0; it < GPT8_ITERS; ++it, p0 += 2048) {
    if (p0 < P) {
      const int ys = y - dy, xs = x - dx;
      uint32_t wd[4] = {0u, 0u, 0u, 0u};
      if (ys >= 0 && ys < h) {
        const uint32_t* src = reinterpret_cast<const uint32_t*>(planes + ((long long)n * C + c) * hw + ys * w + xs);
#pragma unroll
        for (int k = 0; k < 4; ++k)
          if (xs + 2 * k >= 0 && xs + 2 * k < w) wd[k] = __ldg(src + k);
      }
      out[p0 >> 3] = make_uint4(wd[0], wd[1], wd[2], wd[3]);
    }
    x += step_x; y += step_y;
    if (x >= w) { x -= w; ++y; }
    while (y >= h) { y -= h; ++n; }
  }
}

// ------------------------------------------------------------------------------------------
// wgrad epilogue: sum split-K partials [S][NJ][Cin] and scatter to the R conv weight grads [C,Cin,3,3]
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) wgrad_reduce_kernel(const float* __restrict__ part, int S, long long slab, int R, int C,
                                                           int Cin, MutPtrList gw) {
  // reads: coalesced along ci for every (split, tap); writes: the block's [256 ci][9] outputs are contiguous in the
  // [C, Cin, 3, 3] gradient, so they are transposed through shared memory and stored as coalesced 16-byte vectors
  __shared__ __align__(16) float sm[256 * 9];
  const int ci0 = blockIdx.x * 256;
  const int ci = ci0 + threadIdx.x;
  const int c = blockIdx.y, r = blockIdx.z;
  if (!gw.p[r]) return;
  if (ci < Cin) {
    // nine independent loads per split in flight (two splits per trip): the kernel is latency-bound, not byte-bound (31 MB);
    // summation order per tap is still split 0, 1, 2, ... (deterministic)
    const float* src[9];
    float acc[9];
#pragma unroll
    for (int k = 0; k < 9; ++k) {
      const int t = (k == 4) ? 8 * R : r * 8 + (k < 4 ? k : k - 1);
      src[k] = part + (long long)(t * C + c) * Cin + ci;
      acc[k] = 0.f;
    }
#pragma unroll 2
    for (int s = 0; s < S; ++s) {
      float v[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) v[k] = __ldcs(src[k] + s * slab);
#pragma unroll
      for (int k = 0; k < 9; ++k) acc[k] += v[k];
    }
#pragma unroll
    for (int k = 0; k < 9; ++k) sm[threadIdx.x * 9 + k] = acc[k];
  }
  __syncthreads();
  const int nci = min(256, Cin - ci0);
  float* dst = gw.p[r] + ((long long)c * Cin + ci0) * 9;
  if ((reinterpret_cast<uintptr_t>(dst) & 15) == 0 && (nci * 9) % 4 == 0) {
    for (int i = threadIdx.x; i < nci * 9 / 4; i += 256)
      reinterpret_cast<float4*>(dst)[i] = reinterpret_cast<const float4*>(sm)[i];
  } else {
    for (int i = threadIdx.x; i < nci * 9; i += 256) dst[i] = sm[i];
  }
}

// The same reduction for the common case (Cin % 64 == 0, S <= 8 splits): a block owns 64 input channels of one (class, branch),
// a thread one tap and FOUR consecutive channels -- 16-byte loads, all S of them in flight at once, summed in split order
// (deterministic, same order as the kernel above).  Stand-alone timing (profiles/micro/wgrad_reduce_micro.cu, 6 splits,
// 4 x [19,2048,3,3]): 10.4 vs 15.8 us with the slabs in L2, 16.6 vs 25.1 us from HBM.
template <int S>
__global__ void __launch_bounds__(144) wgrad_reduce_vec_kernel(const float* __restrict__ part, long long slab, int R, int C, int Cin,
                                                               MutPtrList gw) {
  __shared__ __align__(16) float sm[64 * 9];
  const int ci0 = blockIdx.x * 64, c = blockIdx.y, r = blockIdx.z;
  if (!gw.p[r]) return;
  const int k = threadIdx.x / 16, q = threadIdx.x % 16;
  const int t = (k == 4) ? 8 * R : r * 8 + (k < 4 ? k : k - 1);
  const float4* src = reinterpret_cast<const float4*>(part + (long long)(t * C + c) * Cin + ci0) + q;
  float4 v[S];
#pragma unroll
  for (int s = 0; s < S; ++s) v[s] = __ldcs(src + s * (slab / 4));
  float4 a = v[0];
#pragma unroll
  for (int s = 1; s < S; ++s) { a.x += v[s].x; a.y += v[s].y; a.z += v[s].z; a.w += v[s].w; }
  sm[(4 * q + 0) * 9 + k] = a.x; sm[(4 * q + 1) * 9 + k] = a.y; sm[(4 * q + 2) * 9 + k] = a.z; sm[(4 * q + 3) * 9 + k] = a.w;
  __syncthreads();
  float* dst = gw.p[r] + ((long long)c * Cin + ci0) * 9;
  if (threadIdx.x < 64 * 9 / 4) reinterpret_cast<float4*>(dst)[threadIdx.x] = reinterpret_cast<const float4*>(sm)[threadIdx.x];
}

static bool wgrad_reduce_vec_launch(const float* part, int S, long long slab, int R, int C, int Cin, const MutPtrList& gw, cudaStream_t stream) {
  if (Cin % 64 != 0 || slab % 4 != 0 || S < 1 || S > 8 || (reinterpret_cast<uintptr_t>(part) & 15) != 0) return false;
  for (int r = 0; r < R; ++r)
    if (gw.p[r] && (reinterpret_cast<uintptr_t>(gw.p[r]) & 15) != 0) return false;
  dim3 grid(Cin / 64, C, R);
  switch (S) {
    case 1: wgrad_reduce_vec_kernel<1><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
    case 2: wgrad_reduce_vec_kernel<2><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
    case 3: wgrad_reduce_vec_kernel<3><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
    case 4: wgrad_reduce_vec_kernel<4><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
    case 5: wgrad_reduce_vec_kernel<5><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
    case 6: wgrad_reduce_vec_kernel<6><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
    case 7: wgrad_reduce_vec_kernel<7><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
    default: wgrad_reduce_vec_kernel<8><<<grid, 144, 0, stream>>>(part, slab, R, C, Cin, gw); break;
  }
  return true;
}

// ------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------
int aspp_pack_weights(const float* const* w, const float* const* b, int R, int C, int Cin, void* Wp, void* WpT,
                      float* bias_sum, cudaStream_t stream) {
  B200SEG_CHECK_ARG(R >= 1 && R <= MAX_RATES, "aspp: %d dilation branches unsupported (1..%d)", R, MAX_RATES);
  B200SEG_CHECK_ARG(w && Wp && WpT && bias_sum, "aspp_pack_weights: null pointer");
  B200SEG_CHECK_ARG(Cin % 8 == 0, "aspp: in_channels=%d must be a multiple of 8", Cin);
  PtrList pw, pb;
  for (int r = 0; r < MAX_RATES; ++r) { pw.p[r] = r < R ? w[r] : nullptr; pb.p[r] = (r < R && b) ? b[r] : nullptr; }
  const int NJ = aspp_nj(C, R);
  B200SEG_CHECK_ARG(C <= 256 && (reinterpret_cast<uintptr_t>(Wp) & 15) == 0 && (reinterpret_cast<uintptr_t>(WpT) & 3) == 0,
                    "aspp_pack_weights: at most 256 classes, Wp 16-byte aligned");
  const size_t smem = (size_t)R * C * PW_CI * 9 * sizeof(float) + (size_t)NJ * sizeof(int);
  B200SEG_CHECK_ARG(smem <= 200 * 1024, "aspp_pack_weights: %d branches x %d classes do not fit the staging buffer", R, C);
  if (smem > 48 * 1024)
    B200SEG_CUDA(cudaFuncSetAttribute(pack_weights_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  pack_weights_kernel<<<Cin / PW_CI, 256, smem, stream>>>(pw, pb, R, C, Cin, NJ, (__nv_bfloat16*)Wp, (__nv_bfloat16*)WpT, bias_sum);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int aspp_pack_features(const float* x, int N, int Cin, int h, int w, void* Xp, cudaStream_t stream) {
  B200SEG_CHECK_ARG(x && Xp && N > 0 && h > 0 && w > 0, "aspp_pack_features: bad arguments");
  B200SEG_CHECK_ARG(Cin % 8 == 0, "aspp: in_channels=%d must be a multiple of 8", Cin);
  profile_begin(3, stream);
  const int rc = nchw_to_nhwc_bf16(x, N, Cin, h * w, Xp, Cin, stream);      // Xp [N*hw, Cin] is NHWC with pitch Cin
  profile_end(3, stream);
  return rc;
}

long long aspp_yt_bytes(int N, int C, int h, int w, int R) {
  const long long P = (long long)N * h * w;
  return (long long)aspp_nj(C, R) * (ceil_div_ll(P, 4) * 4) * 4;
}

int aspp_forward(const void* Xp, const void* Wp, const float* bias_sum, const int* rates, int R, int N, int Cin, int C, int h,
                 int w, float* Yt, float* logits, cudaStream_t stream) {
  B200SEG_CHECK_ARG(Xp && Wp && bias_sum && rates && Yt && logits, "aspp_forward: null pointer");
  B200SEG_CHECK_ARG(R >= 1 && R <= MAX_RATES, "aspp: %d dilation branches unsupported", R);
  const long long P = (long long)N * h * w;
  B200SEG_CHECK_ARG(P < (1LL << 31), "aspp_forward: too many pixels");
  const int NJ = aspp_nj(C, R);
  const long long ypitch = ceil_div_ll(P, 4) * 4;
  gemm::Operand a{(const __nv_bfloat16*)Wp, false, Cin};
  gemm::Operand b{(const __nv_bfloat16*)Xp, false, Cin};
  // CTA pairs on one tcgen05.mma.cta_group::2 along M (NJ = 640 = 5 M-tiles -> 3 pairs, the last one half empty): each SM
  // pulls 32 KB per k-block instead of 48 KB -- 143 vs 154 us at the bench workload although a sixth of the pair slots idles
  int rc;
  if (gemm::fwd_mode() == 1 && P >= 2 * 128 && NJ > 256) {        // (one N-tile only, e.g. 2 classes: channel-major measured faster, 33 vs 37 us)
    // pixel-major: Yt[j, p] computed as D[p, j] with the PIXELS along M.  NJ = 640 is 2.5 N-tiles of 256: the last one runs at
    // MMA width 128 (half the cycles) instead of leaving half a CTA pair idle as the channel-major form does with its 5 M-tiles
    // on 3 pairs; the accumulator goes to Yt straight from registers (a lane is a pixel: 32 consecutive pixels of one row j per
    // store instruction)
    // (one plane of ypitch pixels: Yt[j][p] = D[p, j])
    gemm::Gemm g{b, a, (int)P, NJ, Cin, gemm::out_f32_nchw_rows(Yt, (int)ypitch, 0)};
    g.share = gemm::SHARE_PAIR;
    g.pair_fallback = gemm::SHARE_B;
    g.prof_tag = 0;
    rc = gemm::launch(g, stream);
  } else {
    gemm::Gemm g{a, b, NJ, (int)P, Cin, gemm::out_f32(Yt, ypitch)};
    g.share = gemm::SHARE_PAIR;
    g.pair_fallback = gemm::SHARE_A;
    g.prof_tag = 0;
    rc = gemm::launch(g, stream);
  }
  if (rc) return rc;
  TapTable tt;
  make_taps(tt, rates, R);
  // class chunks of CT per thread: enough threads in flight to cover the HBM latency of the strided Yt reads
  const int CT = (C == 19) ? 5 : (C <= 4 ? 4 : 8);
  const int nchunk = ceil_div(C, CT);
  dim3 grid(ceil_div(w, GATHER_THREADS), h, N * nchunk);
  profile_begin(4, stream);
  if (CT == 5) head_gather_kernel<5><<<grid, GATHER_THREADS, 0, stream>>>(Yt, ypitch, tt, bias_sum, C, nchunk, h, w, logits);
  else if (CT == 4) head_gather_kernel<4><<<grid, GATHER_THREADS, 0, stream>>>(Yt, ypitch, tt, bias_sum, C, nchunk, h, w, logits);
  else head_gather_kernel<8><<<grid, GATHER_THREADS, 0, stream>>>(Yt, ypitch, tt, bias_sum, C, nchunk, h, w, logits);
  profile_end(4, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// The same forward straight from the fp32 NCHW features the reference hands over (classifier.py:26-29): the fp32 -> bf16
// conversion of the pixel operand happens inside the GEMM's producer warps (gemm_fwd_convert_kernel), so there is no separate
// pack pass (146 us at the bench workload, 77 us per eval frame) and no packed copy to read back.  `xn` (optional): the bf16
// NCHW copy of x the weight-gradient GEMM of the backward pass consumes.  Returns B200SEG_ERR_UNSUPPORTED for shapes the fused
// kernel does not take (h*w % 4 != 0, Cin % 64 != 0, fewer than two M-tiles); aspp_forward_f32_supported() tells beforehand.
int aspp_forward_f32_supported(const float* x, int Cin, int C, int h, int w, int R) {
  return gemm::fwd_convert_eligible(x, Cin, h * w, aspp_nj(C, R)) ? 1 : 0;
}

int aspp_forward_f32(const float* x, const void* Wp, const float* bias_sum, const int* rates, int R, int N, int Cin, int C, int h,
                     int w, float* Yt, float* logits, void* xn, cudaStream_t stream) {
  B200SEG_CHECK_ARG(x && Wp && bias_sum && rates && Yt && logits, "aspp_forward_f32: null pointer");
  B200SEG_CHECK_ARG(R >= 1 && R <= MAX_RATES, "aspp: %d dilation branches unsupported", R);
  const long long P = (long long)N * h * w;
  B200SEG_CHECK_ARG(P < (1LL << 31), "aspp_forward: too many pixels");
  const int NJ = aspp_nj(C, R);
  if (!gemm::fwd_convert_eligible(x, Cin, h * w, NJ)) {
    set_error("aspp_forward_f32: shape not supported by the fused-conversion GEMM (h*w=%d, Cin=%d)", h * w, Cin);
    return B200SEG_ERR_UNSUPPORTED;
  }
  const long long ypitch = ceil_div_ll(P, 4) * 4;
  int rc = gemm::launch_fwd_convert((const __nv_bfloat16*)Wp, Cin, x, N, h * w, NJ, Cin, Yt, ypitch, (__nv_bfloat16*)xn, stream, 0);
  if (rc) return rc;
  TapTable tt;
  make_taps(tt, rates, R);
  const int CT = (C == 19) ? 5 : (C <= 4 ? 4 : 8);
  const int nchunk = ceil_div(C, CT);
  dim3 grid(ceil_div(w, GATHER_THREADS), h, N * nchunk);
  profile_begin(4, stream);
  if (CT == 5) head_gather_kernel<5><<<grid, GATHER_THREADS, 0, stream>>>(Yt, ypitch, tt, bias_sum, C, nchunk, h, w, logits);
  else if (CT == 4) head_gather_kernel<4><<<grid, GATHER_THREADS, 0, stream>>>(Yt, ypitch, tt, bias_sum, C, nchunk, h, w, logits);
  else head_gather_kernel<8><<<grid, GATHER_THREADS, 0, stream>>>(Yt, ypitch, tt, bias_sum, C, nchunk, h, w, logits);
  profile_end(4, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// scratch: gOc bf16 [N][C][hw] (P*32 elements reserved) | G't [NJ][Ppitch] bf16 | wpart [S][NJ][Cin] fp32
long long aspp_bwd_scratch_bytes(int N, int Cin, int C, int h, int w, int R, int splits) {
  const long long P = (long long)N * h * w;
  const int NJ = aspp_nj(C, R);
  const long long Ppitch = ceil_div_ll(P, 8) * 8;
  return P * 32 * 2 + 256 + Ppitch * NJ * 2 + 256 + (long long)splits * NJ * Cin * 4 + 256;
}

static void aspp_bwd_carve(void* scratch, long long P, int NJ, __nv_bfloat16** gOt, __nv_bfloat16** Gp, float** wpart) {
  uint8_t* sp = reinterpret_cast<uint8_t*>(scratch);
  *gOt = reinterpret_cast<__nv_bfloat16*>(sp);
  sp += (P * 32 * 2 + 255) / 256 * 256;
  *Gp = reinterpret_cast<__nv_bfloat16*>(sp);
  sp += (ceil_div_ll(P, 8) * 8 * NJ * 2 + 255) / 256 * 256;
  *wpart = reinterpret_cast<float*>(sp);
}

void* aspp_bwd_gOt_ptr(void* scratch) { return scratch; }

// backward GEMMs from the packed bf16 pixel-major output gradient gOt [P][32]
int aspp_backward_packed(const void* gOt_in, const void* Xp, const void* WpT, const int* rates, int R, int N, int Cin, int C,
                         int h, int w, void* scratch, long long scratch_bytes, int splits, float* grad_x, float* const* grad_w,
                         cudaStream_t stream, void* grad_x_nhwc_bf16, cudaEvent_t weights_ready) {
  B200SEG_CHECK_ARG(gOt_in && WpT && rates && scratch, "aspp_backward: null pointer");
  B200SEG_CHECK_ARG(Xp != nullptr || grad_w == nullptr, "aspp_backward: the weight gradient needs the packed features");
  B200SEG_CHECK_ARG(R >= 1 && R <= MAX_RATES, "aspp: %d dilation branches unsupported", R);
  B200SEG_CHECK_ARG(C <= 32, "aspp_backward: num_classes=%d > 32 is not supported", C);
  if (splits < 1) splits = 1;
  B200SEG_CHECK_ARG(scratch_bytes >= aspp_bwd_scratch_bytes(N, Cin, C, h, w, R, splits), "aspp_backward: scratch too small");
  const long long P = (long long)N * h * w;
  B200SEG_CHECK_ARG(P + 2048 * 16 < (1LL << 31), "aspp_backward: too many pixels");
  const int NJ = aspp_nj(C, R);
  const int hw = h * w;
  __nv_bfloat16 *gOt_own, *Gp;
  float* wpart;
  aspp_bwd_carve(scratch, P, NJ, &gOt_own, &Gp, &wpart);
  const __nv_bfloat16* gOt = reinterpret_cast<const __nv_bfloat16*>(gOt_in);
  TapTable tt;
  make_taps(tt, rates, R);
  const long long Ppitch = ceil_div_ll(P, 8) * 8;
  {
    bool fast = (w % 2 == 0);
    for (int t = 0; t < tt.n_taps; ++t) fast = fast && (tt.dx[t] % 2 == 0);
    profile_begin(5, stream);
    if (fast && w % 8 == 0) {
      dim3 grid((unsigned)ceil_div_ll(P, 2048 * GPT8_ITERS), (unsigned)NJ);
      build_gprime_t8_kernel<<<grid, 256, 0, stream>>>(gOt, tt, C, h, w, N, Ppitch, Gp);
    } else {
      dim3 grid((unsigned)ceil_div_ll(P, 512 * GPT_ITERS), (unsigned)NJ);
      if (fast) build_gprime_t_kernel<true><<<grid, 256, 0, stream>>>(gOt, tt, C, h, w, N, Ppitch, Gp);
      else build_gprime_t_kernel<false><<<grid, 256, 0, stream>>>(gOt, tt, C, h, w, N, Ppitch, Gp);
    }
    profile_end(5, stream);
    B200SEG_LAUNCH_CHECK();
  }
  if (grad_w) {
    MutPtrList gw;
    bool any = false;
    for (int r = 0; r < MAX_RATES; ++r) { gw.p[r] = r < R ? grad_w[r] : nullptr; any |= gw.p[r] != nullptr; }
    if (any) {
      // dWp[j, ci] = sum_p G't[j, p] * Xp[p, ci]   A K-major, B MN-major, split-K over pixels
      gemm::Operand a{Gp, false, Ppitch};
      gemm::Operand b{(const __nv_bfloat16*)Xp, true, Cin};
      int used = 1;
      const long long slab = (long long)NJ * Cin;
      gemm::Gemm g{a, b, NJ, Cin, (int)P, gemm::out_f32(wpart, Cin, slab)};
      g.splits = splits;
      g.splits_used = &used;
      g.share = gemm::SHARE_PAIR;                                 // cta_group::2 pairs: 138 vs 165 us
      g.pair_fallback = gemm::SHARE_A;
      g.prof_tag = 2;
      if (int rc = gemm::launch(g, stream)) return rc;
      dim3 grid(ceil_div(Cin, 256), C, R);
      profile_begin(10, stream);
      if (!wgrad_reduce_vec_launch(wpart, used, slab, R, C, Cin, gw, stream))
        wgrad_reduce_kernel<<<grid, 256, 0, stream>>>(wpart, used, slab, R, C, Cin, gw);
      profile_end(10, stream);
      B200SEG_LAUNCH_CHECK();
    }
  }
  // the weight gradients are complete here: a caller that all-reduces them on another stream can start while the
  // data-gradient GEMM below is still running
  if (weights_ready) {
    // inside a stream capture (the one-call entry's graph cache, or the caller's own graph) the record becomes an EXTERNAL event
    // node: every launch of the graph records the event when the weight gradients are complete, and a cudaStreamWaitEvent
    // issued on another stream after the graph launch orders behind it
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    B200SEG_CUDA(cudaStreamIsCapturing(stream, &cap));
    if (cap == cudaStreamCaptureStatusActive) B200SEG_CUDA(cudaEventRecordWithFlags(weights_ready, stream, cudaEventRecordExternal));
    else B200SEG_CUDA(cudaEventRecord(weights_ready, stream));
  }
  if (grad_x && gemm::dgrad_mode() == 0) {
    // dX[ci, p] = WpT[ci, :] . G't[:, p]   -> fp32 NCHW: column p = (image, pixel), row = channel
    gemm::Operand a{(const __nv_bfloat16*)WpT, false, NJ};
    gemm::Operand b{Gp, true, Ppitch};
    gemm::Gemm g{a, b, Cin, (int)P, NJ, gemm::out_f32_nchw_cols(grad_x, hw, hw, (long long)Cin * hw)};
    g.share = gemm::SHARE_B;
    g.sm_reserve = weights_ready ? gemm::overlap_sms() : 0;
    g.prof_tag = 1;
    if (int rc = gemm::launch(g, stream)) return rc;
  } else if (grad_x) {
    // dXt[p, ci] = G't[:, p] . WpT[ci, :] with the PIXELS along M, written as fp32 NCHW straight from the accumulator registers:
    // a TMEM lane is a pixel, so one store instruction covers 32 consecutive pixels of a channel plane (no smem transpose)
    gemm::Operand a{Gp, true, Ppitch};
    gemm::Operand b{(const __nv_bfloat16*)WpT, false, NJ};
    gemm::Gemm g{a, b, (int)P, Cin, NJ, gemm::out_f32_nchw_rows(grad_x, hw, (long long)Cin * hw)};
    g.share = gemm::SHARE_PAIR;
    g.pair_fallback = gemm::SHARE_B;
    g.sm_reserve = weights_ready ? gemm::overlap_sms() : 0;
    g.prof_tag = 1;
    if (int rc = gemm::launch(g, stream)) return rc;
  }
  if (grad_x_nhwc_bf16) {
    // seam format: dXt[p, ci] = G't[:, p] . WpT[ci, :]  written as bf16 pixel-major [P][Cin] (= channels_last NHWC),
    // half the bytes of the fp32 NCHW gradient, so the GEMM is MMA-bound instead of store-bound
    gemm::Operand a{Gp, true, Ppitch};
    gemm::Operand b{(const __nv_bfloat16*)WpT, false, NJ};
    // CTA pairs on one tcgen05.mma.cta_group::2 (M = 256 pixels): 164 vs 170 us with the multicast pairs.  (The fp32 NCHW
    // dgrad above is bound by its 537 MB store, where the 2-SM MMA measured 5 us SLOWER, so it keeps the multicast pairs.)
    gemm::Gemm g{a, b, (int)P, Cin, NJ, gemm::out_bf16(reinterpret_cast<__nv_bfloat16*>(grad_x_nhwc_bf16), Cin)};
    g.share = gemm::SHARE_PAIR;
    g.sm_reserve = weights_ready ? gemm::overlap_sms() : 0;
    g.prof_tag = 1;
    if (int rc = gemm::launch(g, stream)) return rc;
  }
  return B200SEG_OK;
}

// backward from the fp32 NCHW output gradient (generic autograd contract)
int aspp_backward(const float* grad_logits, const void* Xp, const void* WpT, const int* rates, int R, int N, int Cin, int C,
                  int h, int w, void* scratch, long long scratch_bytes, int splits, float* grad_x, float* const* grad_w,
                  float* const* grad_b, cudaStream_t stream) {
  B200SEG_CHECK_ARG(grad_logits && scratch, "aspp_backward: null pointer");
  B200SEG_CHECK_ARG(R >= 1 && R <= MAX_RATES, "aspp: %d dilation branches unsupported", R);
  B200SEG_CHECK_ARG(C <= 32, "aspp_backward: num_classes=%d > 32 is not supported", C);
  if (splits < 1) splits = 1;
  B200SEG_CHECK_ARG(scratch_bytes >= aspp_bwd_scratch_bytes(N, Cin, C, h, w, R, splits), "aspp_backward: scratch too small");
  const long long P = (long long)N * h * w;
  const int hw = h * w;
  __nv_bfloat16* gOt = reinterpret_cast<__nv_bfloat16*>(scratch);
  grad_to_bf16_planes_kernel<<<(unsigned)ceil_div_ll(P * C, 512), 256, 0, stream>>>(grad_logits, P * C, gOt);
  B200SEG_LAUNCH_CHECK();
  if (grad_b) {
    MutPtrList gb;
    bool any = false;
    for (int r = 0; r < MAX_RATES; ++r) { gb.p[r] = r < R ? grad_b[r] : nullptr; any |= gb.p[r] != nullptr; }
    if (any) {
      bias_grad_kernel<<<C, 256, 0, stream>>>(grad_logits, N, C, hw, gb, R);
      B200SEG_LAUNCH_CHECK();
    }
  }
  return aspp_backward_packed(gOt, Xp, WpT, rates, R, N, Cin, C, h, w, scratch, scratch_bytes, splits, grad_x, grad_w, stream, nullptr, nullptr);
}

}  // namespace b200seg
