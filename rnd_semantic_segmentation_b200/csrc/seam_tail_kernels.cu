// Fused tail of the backbone's last Bottleneck: the producer of the head's seam format (bf16 channels_last features).
//
// Replaces (reference file:line): the end of Bottleneck.forward, core/models/feature_extractor/resnet.py:106-113
//   out = self.bn3(out); out += identity; out = self.relu(out)
// with bn3 a FrozenBatchNorm2d (core/models/layers.py:17-23: x * scale + bias), followed by the bf16 channels_last cast that
// feeds the head without its feature pack:
//   forward   y  = bf16_rn(relu((c * scale + bias) + identity))     c, identity fp32 NCHW [N,C,hw] -> y bf16 NHWC [N,hw,C]
//   backward  g  = dy * (y > 0);  dc = g * scale;  didentity = g   dy, y bf16 NHWC -> dc, didentity fp32 NCHW
// Every step is rounded in fp32 in the stock order (mul, add, add, relu, one round-to-nearest cast; no FMA contraction), so
// y is bit-identical to the stock fp32 output converted with .to(torch.bfloat16).
//
// Both kernels are one memory-bound pass: a 32-channel x 128-pixel tile goes through shared memory between the NCHW side
// (one warp streams a 512-byte channel row with 16-byte accesses) and the NHWC side (one thread moves 8 channels = 16 bytes of
// one pixel; a warp covers 8 pixels x 64 contiguous bytes).  The tile's 4-pixel quads are XOR-swizzled with the channel's
// 8-group so that both the row-wise float4 accesses and the column-wise scalar accesses are free of bank conflicts.
//
// The forward pass with the identity prologue is also the library's fp32 NCHW -> bf16 NHWC conversion (nchw_to_nhwc_bf16):
// the head's feature pack (aspp_pack_features) and the discriminator's gradient layout, whose output pitch may exceed C (the
// pad channels are written as zeros).  At the 2:1 read/write mix of the pack this tile runs at 6.5 TB/s where the 64 x 64
// scalar-load tile it replaced ran at 5.6 (profiles/micro/nhwc_tile_micro.cu).
#include "common.cuh"

namespace b200seg {

constexpr int ST_CH = 32, ST_PX = 128, ST_THREADS = 256;

// float index of (channel ch, pixel s) in the [ST_CH][ST_PX] tile
__device__ __forceinline__ int st_idx(int ch, int s) {
  return ch * ST_PX + ((((s >> 2) ^ (((ch >> 3) & 3) << 1)) << 2) | (s & 3));
}

__device__ __forceinline__ float tail_value(float c, float sc, float bi, float id) {
  const float v = __fadd_rn(__fadd_rn(__fmul_rn(c, sc), bi), id);
  return v <= 0.f ? 0.f : v;                                       // NaN passes through, as torch.relu
}

// training-mode BatchNorm2d in its centred form (the fold c * scale + shift cancels when |mean| >> sigma), then residual + relu
__device__ __forceinline__ float bn_tail_value(float c, float mean, float invstd, float gamma, float beta, float id) {
  const float v = __fadd_rn(__fmaf_rn(__fmul_rn(__fsub_rn(c, mean), invstd), gamma, beta), id);
  return v <= 0.f ? 0.f : v;
}

// y[n, s, ch] = bf16_rn(f(c[n, ch, s])) for ch < pitch, with f the seam tail (TAIL) or the identity (then identity, scale and
// bias are not read); channels C <= ch < pitch are written as 0.
// BATCH (with TAIL): f is the batch-statistics tail bn_tail_value; scale / bias carry mean / invstd, and gamma / beta may be null
// (affine=False).  Without BATCH, gamma and beta are not read.
// VEC: hw % 4 == 0 and c / identity 16-byte aligned (float4 rows); otherwise scalar loads
template <bool TAIL, bool VEC, bool BATCH = false>
__global__ void __launch_bounds__(ST_THREADS) nchw_to_nhwc_tile_kernel(const float* __restrict__ c, const float* __restrict__ identity,
                                                                       const float* __restrict__ scale, const float* __restrict__ bias,
                                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                                       int C, int hw, int pitch, __nv_bfloat16* __restrict__ y) {
  __shared__ __align__(16) float tile[ST_CH * ST_PX];
  const int s0 = blockIdx.x * ST_PX, c0 = blockIdx.y * ST_CH, n = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int s = s0 + 4 * lane;
  float4 a[4], b[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {                                    // rows warp + 8 i: all eight loads in flight first
    const int cg = c0 + warp + 8 * i;
    a[i] = b[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (cg < C) {
      const long long off = ((long long)n * C + cg) * hw + s;
      if (VEC) {
        if (s < hw) {
          a[i] = __ldcs(reinterpret_cast<const float4*>(c + off));
          if (TAIL) b[i] = __ldcs(reinterpret_cast<const float4*>(identity + off));
        }
      } else {
        float* av = &a[i].x;
        float* bv = &b[i].x;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (s + j < hw) {
            av[j] = __ldcs(c + off + j);
            if (TAIL) bv[j] = __ldcs(identity + off + j);
          }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ch = warp + 8 * i, cg = c0 + ch;
    float4 v = a[i];
    if (TAIL && BATCH) {
      const float mu = cg < C ? __ldg(scale + cg) : 0.f, is = cg < C ? __ldg(bias + cg) : 0.f;
      const float ga = gamma && cg < C ? __ldg(gamma + cg) : 1.f, be = beta && cg < C ? __ldg(beta + cg) : 0.f;
      v = make_float4(bn_tail_value(a[i].x, mu, is, ga, be, b[i].x), bn_tail_value(a[i].y, mu, is, ga, be, b[i].y),
                      bn_tail_value(a[i].z, mu, is, ga, be, b[i].z), bn_tail_value(a[i].w, mu, is, ga, be, b[i].w));
    } else if (TAIL) {
      const float sc = cg < C ? __ldg(scale + cg) : 0.f, bi = cg < C ? __ldg(bias + cg) : 0.f;
      v = make_float4(tail_value(a[i].x, sc, bi, b[i].x), tail_value(a[i].y, sc, bi, b[i].y), tail_value(a[i].z, sc, bi, b[i].z),
                      tail_value(a[i].w, sc, bi, b[i].w));
    }
    *reinterpret_cast<float4*>(tile + st_idx(ch, 4 * lane)) = v;
  }
  __syncthreads();
  const int chunk = lane & 3, cc = c0 + 8 * chunk;
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int sl = (lane >> 2) + 8 * warp + 64 * it;
    if (s0 + sl < hw && cc < pitch) {
      uint32_t w4[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const __nv_bfloat162 v = __floats2bfloat162_rn(tile[st_idx(8 * chunk + 2 * e, sl)], tile[st_idx(8 * chunk + 2 * e + 1, sl)]);
        w4[e] = *reinterpret_cast<const uint32_t*>(&v);
      }
      *reinterpret_cast<uint4*>(y + ((long long)n * hw + s0 + sl) * pitch + cc) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
    }
  }
}

// Batch-statistics backward (BN != BN_FOLD): c, mean and invstd are read in both passes.
//   BN_REDUCE writes partial[ch * P + n * gridDim.x + blockIdx.x] = (sum g, sum g * (c - mean)) over the tile's 128 pixels
//             (P = N * gridDim.x) and nothing else;
//   BN_APPLY  writes dc = (g - sum_g / M - (c - mean) * invstd^2 * sum_gx / M) * invstd * gamma with the sums taken over the R
//             records of sums [R][2][C] in rank order and M = *count (gamma may be null), and didentity = g.
// BN_G (the fused conv3 tail, whose conv3 runs inside the tcgen05 GEMMs) writes g itself as bf16 NHWC (the GEMMs' operand; exact,
// no rounding) and didentity = g; c, scale and dc are not used.
// BN_APPLY_G (conv3 under batch statistics) computes dc as BN_APPLY does and writes it rounded once to bf16 NHWC into g (the operand
// of conv3's backward GEMMs) instead of fp32 NCHW dc; didentity = g as in BN_APPLY.
enum { BN_FOLD = 0, BN_REDUCE = 1, BN_APPLY = 2, BN_G = 3, BN_APPLY_G = 4 };
struct BnBackward {
  const float* c;
  const float* mean;
  const float* invstd;
  const float* gamma;
  const float* sums;
  int R;
  const double* count;
  float2* partial;
  __nv_bfloat16* g;
};

// VEC: hw % 4 == 0 and the requested outputs (and c) 16-byte aligned (float4 rows); otherwise scalar accesses.  dc / didentity may
// be null.
template <bool VEC, int BN = BN_FOLD>
__global__ void __launch_bounds__(ST_THREADS) seam_tail_backward_kernel(const __nv_bfloat16* __restrict__ dy,
                                                                        const __nv_bfloat16* __restrict__ y,
                                                                        const float* __restrict__ scale, int C, int hw,
                                                                        float* __restrict__ dc, float* __restrict__ didentity,
                                                                        BnBackward bn) {
  __shared__ __align__(16) float tile[ST_CH * ST_PX];
  const int s0 = blockIdx.x * ST_PX, c0 = blockIdx.y * ST_CH, n = blockIdx.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int chunk = lane & 3, cc = c0 + 8 * chunk;
  uint4 gv[2], yv[2];
#pragma unroll
  for (int it = 0; it < 2; ++it) {                                 // all four 16-byte loads in flight first
    const int sl = (lane >> 2) + 8 * warp + 64 * it;
    gv[it] = yv[it] = make_uint4(0u, 0u, 0u, 0u);
    if (s0 + sl < hw && cc < C) {
      const long long off = ((long long)n * hw + s0 + sl) * C + cc;
      gv[it] = __ldcs(reinterpret_cast<const uint4*>(dy + off));
      yv[it] = __ldcs(reinterpret_cast<const uint4*>(y + off));
    }
  }
  float4 cv[4];                                                    // the c rows this thread owns after the barrier, also in flight
  if (BN != BN_FOLD && BN != BN_G) {
    const int s = s0 + 4 * lane;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int cg = c0 + warp + 8 * i;
      cv[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (cg >= C) continue;
      const long long off = ((long long)n * C + cg) * hw + s;
      if (VEC) {
        if (s < hw) cv[i] = __ldcs(reinterpret_cast<const float4*>(bn.c + off));
      } else {
        float* p = &cv[i].x;
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (s + j < hw) p[j] = __ldcs(bn.c + off + j);
      }
    }
  }
#pragma unroll
  for (int it = 0; it < 2; ++it) {
    const int sl = (lane >> 2) + 8 * warp + 64 * it;
    const uint32_t* g32 = &gv[it].x;
    const uint32_t* y32 = &yv[it].x;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const float2 g2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(g32 + e));
      const float2 y2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(y32 + e));
      tile[st_idx(8 * chunk + 2 * e, sl)] = y2.x > 0.f ? g2.x : 0.f;
      tile[st_idx(8 * chunk + 2 * e + 1, sl)] = y2.y > 0.f ? g2.y : 0.f;
    }
    if (BN == BN_G && s0 + sl < hw && cc < C) {                    // the same values as bf16 NHWC: dy's bits where y > 0, else +0
      uint32_t w4[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const float2 y2 = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(y32 + e));
        w4[e] = (y2.x > 0.f ? (g32[e] & 0xffffu) : 0u) | (y2.y > 0.f ? (g32[e] & 0xffff0000u) : 0u);
      }
      *reinterpret_cast<uint4*>(bn.g + ((long long)n * hw + s0 + sl) * C + cc) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
    }
  }
  __syncthreads();
  const int s = s0 + 4 * lane;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ch = warp + 8 * i, cg = c0 + ch;
    if (cg >= C) continue;                                         // (warp-uniform)
    const float4 g = *reinterpret_cast<const float4*>(tile + st_idx(ch, 4 * lane));
    if (BN == BN_REDUCE) {                                         // pixels past hw have g = 0 and c = 0
      const float mu = __ldg(bn.mean + cg);
      float sg = (g.x + g.y) + (g.z + g.w);
      float sx = (g.x * (cv[i].x - mu) + g.y * (cv[i].y - mu)) + (g.z * (cv[i].z - mu) + g.w * (cv[i].w - mu));
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        sg += __shfl_down_sync(0xffffffffu, sg, o);
        sx += __shfl_down_sync(0xffffffffu, sx, o);
      }
      if (lane == 0) bn.partial[(long long)cg * gridDim.x * gridDim.z + (long long)n * gridDim.x + blockIdx.x] = make_float2(sg, sx);
      continue;
    }
    float4 d;
    if (BN == BN_APPLY || BN == BN_APPLY_G) {
      float sg = 0.f, sx = 0.f;
      for (int r = 0; r < bn.R; ++r) {                             // rank order: every rank computes the same sums
        sg += __ldg(bn.sums + (long long)r * 2 * C + cg);
        sx += __ldg(bn.sums + (long long)r * 2 * C + C + cg);
      }
      const float norm = (float)(1.0 / __ldg(bn.count));
      const float mu = __ldg(bn.mean + cg), is = __ldg(bn.invstd + cg);
      const float mdy = sg * norm, f1 = is * is * sx * norm, f2 = (bn.gamma ? __ldg(bn.gamma + cg) : 1.f) * is;
      d = make_float4((g.x - mdy - (cv[i].x - mu) * f1) * f2, (g.y - mdy - (cv[i].y - mu) * f1) * f2,
                      (g.z - mdy - (cv[i].z - mu) * f1) * f2, (g.w - mdy - (cv[i].w - mu) * f1) * f2);
    } else if (BN == BN_FOLD) {
      const float sc = __ldg(scale + cg);
      d = make_float4(__fmul_rn(g.x, sc), __fmul_rn(g.y, sc), __fmul_rn(g.z, sc), __fmul_rn(g.w, sc));
    } else {
      d = g;                                                       // (BN_G: dc is null)
    }
    if (BN == BN_APPLY_G) *reinterpret_cast<float4*>(tile + st_idx(ch, 4 * lane)) = d;    // (this thread's own slot)
    const long long off = ((long long)n * C + cg) * hw + s;
    if (VEC) {
      if (s < hw) {
        if (didentity) __stcs(reinterpret_cast<float4*>(didentity + off), g);
        if (dc) __stcs(reinterpret_cast<float4*>(dc + off), d);
      }
    } else {
      const float* gp = &g.x;
      const float* dp = &d.x;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (s + j >= hw) break;
        if (didentity) __stcs(didentity + off + j, gp[j]);
        if (dc) __stcs(dc + off + j, dp[j]);
      }
    }
  }
  if (BN == BN_APPLY_G) {                                          // dc through the tile to bf16 NHWC, as the forward's y
    __syncthreads();
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int sl = (lane >> 2) + 8 * warp + 64 * it;
      if (s0 + sl < hw && cc < C) {
        uint32_t w4[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const __nv_bfloat162 v = __floats2bfloat162_rn(tile[st_idx(8 * chunk + 2 * e, sl)], tile[st_idx(8 * chunk + 2 * e + 1, sl)]);
          w4[e] = *reinterpret_cast<const uint32_t*>(&v);
        }
        *reinterpret_cast<uint4*>(bn.g + ((long long)n * hw + s0 + sl) * C + cc) = make_uint4(w4[0], w4[1], w4[2], w4[3]);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------------------------------------
// Batch statistics (training-mode BatchNorm2d / SyncBatchNorm bn3).  No atomics: every reduction has a fixed order, so results are
// bit-identical run to run, and nothing synchronises with the host (the block can be captured in a CUDA graph).
//   bn_stats_partial_kernel  one CTA per (n, ch) plane: (mean, M2) of its hw values, shifted -> partial[ch][n]
//   bn_stats_record_kernel   per channel, the N planes (equal counts) in fp64 -> record [3][C] = (count, mean, M2)
//   bn_combine_kernel        per channel, R records in rank order (Chan's merge in fp64) -> mean, invstd, running stats
// Every value is first shifted by the first value of its plane, K = c[n, ch, 0] (x - K is exact in fp32 for x near K, so the
// fp32 arithmetic below works at the scale of sigma even when |mean| >> sigma; the record adds each K back in fp64).  Each thread then
// takes up to 32 values at a time and merges their two-pass (mean, M2) into its running one (Chan et al.), so no long sum cancels.
// ------------------------------------------------------------------------------------------------------------------------------
constexpr int BS_THREADS = 256, BS_GROUP = 8;

struct Moments {
  float n, mean, m2;
};

__device__ __forceinline__ Moments merge(Moments a, Moments b) {
  const float n = a.n + b.n;
  if (n == 0.f) return a;
  const float delta = b.mean - a.mean, fb = b.n / n;
  return {n, a.mean + delta * fb, a.m2 + b.m2 + delta * delta * (a.n * fb)};
}

// VEC: hw % 4 == 0 and c 16-byte aligned
template <bool VEC>
__global__ void __launch_bounds__(BS_THREADS) bn_stats_partial_kernel(const float* __restrict__ c, int C, int N, int hw,
                                                                      float2* __restrict__ partial) {
  const int plane = blockIdx.x, ch = plane % C, n = plane / C;
  const float* row = c + (long long)plane * hw;
  const float shift = __ldg(row);                                  // (the line of the row's first load)
  Moments acc = {0.f, 0.f, 0.f};
  float v[4 * BS_GROUP];
  const int span = VEC ? hw / 4 : hw;                              // float4s or floats in the row
  for (int base = threadIdx.x; base < span; base += BS_THREADS * BS_GROUP) {
    int k = 0;                                                     // valid loads: a prefix of the group
#pragma unroll
    for (int j = 0; j < BS_GROUP; ++j) {
      const int idx = base + j * BS_THREADS;
      if (idx < span) {
        if (VEC) {
          const float4 q = __ldcs(reinterpret_cast<const float4*>(row) + idx);
          v[4 * j] = q.x - shift; v[4 * j + 1] = q.y - shift; v[4 * j + 2] = q.z - shift; v[4 * j + 3] = q.w - shift;
        } else {
          v[j] = __ldcs(row + idx) - shift;
        }
        ++k;
      }
    }
    const int m = VEC ? 4 * k : k;
    float sum = 0.f;
#pragma unroll
    for (int j = 0; j < 4 * BS_GROUP; ++j)
      if (j < m && (VEC || j < BS_GROUP)) sum += v[j];
    const float gm = sum / (float)m;
    float m2 = 0.f;
#pragma unroll
    for (int j = 0; j < 4 * BS_GROUP; ++j)
      if (j < m && (VEC || j < BS_GROUP)) m2 += (v[j] - gm) * (v[j] - gm);
    acc = merge(acc, Moments{(float)m, gm, m2});
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const Moments other = {__shfl_down_sync(0xffffffffu, acc.n, o), __shfl_down_sync(0xffffffffu, acc.mean, o),
                           __shfl_down_sync(0xffffffffu, acc.m2, o)};
    acc = merge(acc, other);
  }
  __shared__ Moments warps[BS_THREADS / 32];
  if ((threadIdx.x & 31) == 0) warps[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    Moments t = warps[0];
    for (int w = 1; w < BS_THREADS / 32; ++w) t = merge(t, warps[w]);
    partial[(long long)ch * N + n] = make_float2(t.mean, t.m2);            // mean of x - row[0]
  }
}

__global__ void bn_stats_record_kernel(const float* __restrict__ c, const float2* __restrict__ partial, int C, int N, int hw,
                                       double* __restrict__ record) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= C) return;
  const float2* p = partial + (long long)ch * N;
  double mean = 0.0;                                               // each plane's mean: its shift c[n, ch, 0] added back
  for (int i = 0; i < N; ++i) mean += (double)c[((long long)i * C + ch) * hw] + (double)p[i].x;
  mean /= N;
  double m2 = 0.0, spread = 0.0;
  for (int i = 0; i < N; ++i) {
    const double d = ((double)c[((long long)i * C + ch) * hw] + (double)p[i].x) - mean;
    m2 += (double)p[i].y;
    spread += d * d;
  }
  record[ch] = (double)N * hw;
  record[C + ch] = mean;
  record[2 * C + ch] = m2 + spread * hw;
}

__global__ void bn_combine_kernel(const double* __restrict__ records, int R, int C, float eps, float momentum,
                                  const long long* __restrict__ num_batches_tracked, float* __restrict__ running_mean,
                                  float* __restrict__ running_var, float* __restrict__ mean_out, float* __restrict__ invstd_out,
                                  double* __restrict__ count_out) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= C) return;
  double n = 0.0, mean = 0.0, m2 = 0.0;
  for (int r = 0; r < R; ++r) {                                    // rank order
    const double* rec = records + (long long)r * 3 * C;
    const double nb = rec[ch], mb = rec[C + ch], m2b = rec[2 * C + ch];
    const double nn = n + nb;
    if (nn == 0.0) continue;
    const double delta = mb - mean, fb = nb / nn;
    mean += delta * fb;
    m2 += m2b + delta * delta * (n * fb);
    n = nn;
  }
  const double var = m2 / n;
  mean_out[ch] = (float)mean;
  invstd_out[ch] = (float)(1.0 / sqrt(var + (double)eps));
  if (count_out && ch == 0) *count_out = n;
  if (running_mean) {
    const double f = num_batches_tracked ? 1.0 / (double)*num_batches_tracked : (double)momentum;
    running_mean[ch] = (float)((1.0 - f) * running_mean[ch] + f * mean);
    running_var[ch] = (float)((1.0 - f) * running_var[ch] + f * var * n / (n - 1.0));
  }
}

// one warp per channel: the P partials of the reduce pass in fp64 -> sums [2][C] = (sum g, sum g (c - mean)), dbeta, dgamma
__global__ void bn_backward_finalize_kernel(const float2* __restrict__ partial, long long P, int C, const float* __restrict__ invstd,
                                            float* __restrict__ sums, float* __restrict__ dgamma, float* __restrict__ dbeta) {
  const int ch = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (ch >= C) return;
  const float2* p = partial + (long long)ch * P;
  double sg = 0.0, sx = 0.0;
  for (long long i = lane; i < P; i += 32) {
    const float2 q = p[i];
    sg += q.x;
    sx += q.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    sg += __shfl_down_sync(0xffffffffu, sg, o);
    sx += __shfl_down_sync(0xffffffffu, sx, o);
  }
  if (lane == 0) {
    sums[ch] = (float)sg;
    sums[C + ch] = (float)sx;
    if (dbeta) dbeta[ch] = (float)sg;
    if (dgamma) dgamma[ch] = (float)(sx * (double)invstd[ch]);
  }
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// identity may be null (TAIL = false); gamma / beta are read with BATCH only
template <bool TAIL, bool BATCH = false>
static int nchw_to_nhwc_launch(const float* c, const float* identity, const float* scale, const float* bias, const float* gamma,
                               const float* beta, int N, int C, int hw, int pitch, void* y, cudaStream_t stream) {
  const dim3 grid(ceil_div(hw, ST_PX), ceil_div(pitch, ST_CH), N);
  __nv_bfloat16* yb = reinterpret_cast<__nv_bfloat16*>(y);
  if (hw % 4 == 0 && aligned16(c) && aligned16(identity))         // (a null pointer counts as aligned)
    nchw_to_nhwc_tile_kernel<TAIL, true, BATCH><<<grid, ST_THREADS, 0, stream>>>(c, identity, scale, bias, gamma, beta, C, hw, pitch, yb);
  else
    nchw_to_nhwc_tile_kernel<TAIL, false, BATCH><<<grid, ST_THREADS, 0, stream>>>(c, identity, scale, bias, gamma, beta, C, hw, pitch, yb);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int seam_tail_forward(const float* c, const float* identity, const float* scale, const float* bias, int N, int C, int hw, void* y,
                      cudaStream_t stream) {
  B200SEG_CHECK_ARG(c && identity && scale && bias && y && N > 0 && C > 0 && hw > 0, "seam_tail_forward: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_forward: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_forward: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(y), "seam_tail_forward: y must be 16-byte aligned");
  return nchw_to_nhwc_launch<true>(c, identity, scale, bias, nullptr, nullptr, N, C, hw, C, y, stream);
}

// fp32 NCHW [N][C][hw] -> bf16 NHWC [N*hw][pitch], channels >= C zero
int nchw_to_nhwc_bf16(const float* src, int N, int C, int hw, void* dst, int pitch, cudaStream_t stream) {
  B200SEG_CHECK_ARG(src && dst && N > 0 && C > 0 && hw > 0 && pitch % 8 == 0 && pitch >= C, "nchw_to_nhwc_bf16: bad arguments");
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(pitch, ST_CH) <= 65535, "nchw_to_nhwc_bf16: N = %d / pitch = %d too large", N, pitch);
  B200SEG_CHECK_ARG(aligned16(dst), "nchw_to_nhwc_bf16: dst must be 16-byte aligned");
  return nchw_to_nhwc_launch<false>(src, nullptr, nullptr, nullptr, nullptr, nullptr, N, C, hw, pitch, dst, stream);
}

template <int BN>
static void backward_launch(const void* dy, const void* y, const float* scale, int N, int C, int hw, float* dc, float* didentity,
                            const BnBackward& bn, cudaStream_t stream) {
  const dim3 grid(ceil_div(hw, ST_PX), ceil_div(C, ST_CH), N);
  const __nv_bfloat16* g = reinterpret_cast<const __nv_bfloat16*>(dy);
  const __nv_bfloat16* yb = reinterpret_cast<const __nv_bfloat16*>(y);
  if (hw % 4 == 0 && aligned16(dc) && aligned16(didentity) && aligned16(bn.c))   // (a null pointer counts as aligned)
    seam_tail_backward_kernel<true, BN><<<grid, ST_THREADS, 0, stream>>>(g, yb, scale, C, hw, dc, didentity, bn);
  else
    seam_tail_backward_kernel<false, BN><<<grid, ST_THREADS, 0, stream>>>(g, yb, scale, C, hw, dc, didentity, bn);
}

int seam_tail_backward(const void* dy, const void* y, const float* scale, int N, int C, int hw, float* dc, float* didentity,
                       cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && scale && N > 0 && C > 0 && hw > 0, "seam_tail_backward: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_backward: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_backward: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(dy) && aligned16(y), "seam_tail_backward: dy and y must be 16-byte aligned");
  if (!dc && !didentity) return B200SEG_OK;
  backward_launch<BN_FOLD>(dy, y, scale, N, C, hw, dc, didentity, BnBackward{}, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// g = dy * (y > 0) as bf16 NHWC [N*hw][C] (the operand of the fused conv3's data- and weight-gradient GEMMs) and, when didentity is
// not null, didentity = g as fp32 NCHW
int seam_conv3_g(const void* dy, const void* y, int N, int C, int hw, void* g, float* didentity, cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && g && N > 0 && C > 0 && hw > 0, "seam_conv3_g: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_conv3_g: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_conv3_g: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(dy) && aligned16(y) && aligned16(g), "seam_conv3_g: dy, y and g must be 16-byte aligned");
  BnBackward bn{};
  bn.g = reinterpret_cast<__nv_bfloat16*>(g);
  backward_launch<BN_G>(dy, y, nullptr, N, C, hw, nullptr, didentity, bn, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// ---- batch-statistics tail -------------------------------------------------------------------------------------------------
long long bn_stats_scratch_bytes(int N, int C) { return (long long)N * C * (long long)sizeof(float2); }

int bn_stats(const float* c, int N, int C, int hw, void* scratch, long long scratch_bytes, double* record, cudaStream_t stream) {
  B200SEG_CHECK_ARG(c && record && N > 0 && C > 0 && hw > 0, "bn_stats: bad arguments");
  B200SEG_CHECK_ARG((long long)N * C <= 0x7fffffffLL, "bn_stats: N * C = %lld too large", (long long)N * C);
  B200SEG_CHECK_ARG(scratch && scratch_bytes >= bn_stats_scratch_bytes(N, C), "bn_stats: scratch too small");
  float2* partial = reinterpret_cast<float2*>(scratch);
  if (hw % 4 == 0 && aligned16(c))
    bn_stats_partial_kernel<true><<<N * C, BS_THREADS, 0, stream>>>(c, C, N, hw, partial);
  else
    bn_stats_partial_kernel<false><<<N * C, BS_THREADS, 0, stream>>>(c, C, N, hw, partial);
  bn_stats_record_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(c, partial, C, N, hw, record);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int bn_combine_stats(const double* records, int R, int C, float eps, float momentum, const long long* num_batches_tracked,
                     float* running_mean, float* running_var, float* mean, float* invstd, double* count, cudaStream_t stream) {
  B200SEG_CHECK_ARG(records && R > 0 && C > 0 && mean && invstd, "bn_combine_stats: bad arguments");
  B200SEG_CHECK_ARG((running_mean == nullptr) == (running_var == nullptr), "bn_combine_stats: give both running buffers or neither");
  bn_combine_kernel<<<ceil_div(C, 128), 128, 0, stream>>>(records, R, C, eps, momentum, num_batches_tracked, running_mean,
                                                          running_var, mean, invstd, count);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int seam_tail_bn_forward(const float* c, const float* identity, const float* mean, const float* invstd, const float* gamma,
                         const float* beta, int N, int C, int hw, void* y, cudaStream_t stream) {
  B200SEG_CHECK_ARG(c && identity && mean && invstd && y && N > 0 && C > 0 && hw > 0, "seam_tail_bn_forward: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_bn_forward: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_bn_forward: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(y), "seam_tail_bn_forward: y must be 16-byte aligned");
  return nchw_to_nhwc_launch<true, true>(c, identity, mean, invstd, gamma, beta, N, C, hw, C, y, stream);
}

long long seam_tail_bn_backward_reduce_scratch_bytes(int N, int C, int hw) {
  return (long long)C * N * ceil_div(hw, ST_PX) * (long long)sizeof(float2);
}

int seam_tail_bn_backward_reduce(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, int N, int C,
                                 int hw, void* scratch, long long scratch_bytes, float* sums, float* dgamma, float* dbeta,
                                 cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && c && mean && invstd && sums && N > 0 && C > 0 && hw > 0, "seam_tail_bn_backward_reduce: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_bn_backward_reduce: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_bn_backward_reduce: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(dy) && aligned16(y), "seam_tail_bn_backward_reduce: dy and y must be 16-byte aligned");
  B200SEG_CHECK_ARG(scratch && scratch_bytes >= seam_tail_bn_backward_reduce_scratch_bytes(N, C, hw),
                    "seam_tail_bn_backward_reduce: scratch too small");
  BnBackward bn{};
  bn.c = c;
  bn.mean = mean;
  bn.partial = reinterpret_cast<float2*>(scratch);
  backward_launch<BN_REDUCE>(dy, y, nullptr, N, C, hw, nullptr, nullptr, bn, stream);
  const long long P = (long long)N * ceil_div(hw, ST_PX);
  bn_backward_finalize_kernel<<<ceil_div(C, 8), 256, 0, stream>>>(bn.partial, P, C, invstd, sums, dgamma, dbeta);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int seam_tail_bn_backward(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, const float* gamma,
                          const float* sums, int R, const double* count, int N, int C, int hw, float* dc, float* didentity,
                          cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && c && mean && invstd && sums && count && R > 0 && N > 0 && C > 0 && hw > 0,
                    "seam_tail_bn_backward: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_bn_backward: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_bn_backward: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(dy) && aligned16(y), "seam_tail_bn_backward: dy and y must be 16-byte aligned");
  if (!dc && !didentity) return B200SEG_OK;
  BnBackward bn{c, mean, invstd, gamma, sums, R, count, nullptr};
  backward_launch<BN_APPLY>(dy, y, nullptr, N, C, hw, dc, didentity, bn, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

// conv3 under batch statistics: dc as seam_tail_bn_backward computes it, rounded once to bf16 NHWC [N*hw][C] (the operand of conv3's
// data- and weight-gradient GEMMs; fp32 dc is never written), and, when didentity is not null, didentity = g as fp32 NCHW
int seam_tail_bn_backward_g(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, const float* gamma,
                            const float* sums, int R, const double* count, int N, int C, int hw, void* g, float* didentity,
                            cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && c && mean && invstd && sums && count && g && R > 0 && N > 0 && C > 0 && hw > 0,
                    "seam_tail_bn_backward_g: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_bn_backward_g: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_bn_backward_g: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(dy) && aligned16(y) && aligned16(g), "seam_tail_bn_backward_g: dy, y and g must be 16-byte aligned");
  BnBackward bn{c, mean, invstd, gamma, sums, R, count, nullptr, reinterpret_cast<__nv_bfloat16*>(g)};
  backward_launch<BN_APPLY_G>(dy, y, nullptr, N, C, hw, nullptr, didentity, bn, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

}  // namespace b200seg
