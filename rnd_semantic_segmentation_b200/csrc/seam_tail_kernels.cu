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

// y[n, s, ch] = bf16_rn(f(c[n, ch, s])) for ch < pitch, with f the seam tail (TAIL) or the identity (then identity, scale and
// bias are not read); channels C <= ch < pitch are written as 0.
// VEC: hw % 4 == 0 and c / identity 16-byte aligned (float4 rows); otherwise scalar loads
template <bool TAIL, bool VEC>
__global__ void __launch_bounds__(ST_THREADS) nchw_to_nhwc_tile_kernel(const float* __restrict__ c, const float* __restrict__ identity,
                                                                       const float* __restrict__ scale, const float* __restrict__ bias,
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
    if (TAIL) {
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

// VEC: hw % 4 == 0 and the requested outputs 16-byte aligned (float4 rows); otherwise scalar stores.  dc / didentity may be null.
template <bool VEC>
__global__ void __launch_bounds__(ST_THREADS) seam_tail_backward_kernel(const __nv_bfloat16* __restrict__ dy,
                                                                        const __nv_bfloat16* __restrict__ y,
                                                                        const float* __restrict__ scale, int C, int hw,
                                                                        float* __restrict__ dc, float* __restrict__ didentity) {
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
  }
  __syncthreads();
  const int s = s0 + 4 * lane;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ch = warp + 8 * i, cg = c0 + ch;
    if (cg >= C) continue;
    const float4 g = *reinterpret_cast<const float4*>(tile + st_idx(ch, 4 * lane));
    const float sc = __ldg(scale + cg);
    const float4 d = make_float4(__fmul_rn(g.x, sc), __fmul_rn(g.y, sc), __fmul_rn(g.z, sc), __fmul_rn(g.w, sc));
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
}

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// identity may be null (TAIL = false)
template <bool TAIL>
static int nchw_to_nhwc_launch(const float* c, const float* identity, const float* scale, const float* bias, int N, int C, int hw,
                               int pitch, void* y, cudaStream_t stream) {
  const dim3 grid(ceil_div(hw, ST_PX), ceil_div(pitch, ST_CH), N);
  __nv_bfloat16* yb = reinterpret_cast<__nv_bfloat16*>(y);
  if (hw % 4 == 0 && aligned16(c) && aligned16(identity))         // (a null pointer counts as aligned)
    nchw_to_nhwc_tile_kernel<TAIL, true><<<grid, ST_THREADS, 0, stream>>>(c, identity, scale, bias, C, hw, pitch, yb);
  else
    nchw_to_nhwc_tile_kernel<TAIL, false><<<grid, ST_THREADS, 0, stream>>>(c, identity, scale, bias, C, hw, pitch, yb);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int seam_tail_forward(const float* c, const float* identity, const float* scale, const float* bias, int N, int C, int hw, void* y,
                      cudaStream_t stream) {
  B200SEG_CHECK_ARG(c && identity && scale && bias && y && N > 0 && C > 0 && hw > 0, "seam_tail_forward: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_forward: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_forward: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(y), "seam_tail_forward: y must be 16-byte aligned");
  return nchw_to_nhwc_launch<true>(c, identity, scale, bias, N, C, hw, C, y, stream);
}

// fp32 NCHW [N][C][hw] -> bf16 NHWC [N*hw][pitch], channels >= C zero
int nchw_to_nhwc_bf16(const float* src, int N, int C, int hw, void* dst, int pitch, cudaStream_t stream) {
  B200SEG_CHECK_ARG(src && dst && N > 0 && C > 0 && hw > 0 && pitch % 8 == 0 && pitch >= C, "nchw_to_nhwc_bf16: bad arguments");
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(pitch, ST_CH) <= 65535, "nchw_to_nhwc_bf16: N = %d / pitch = %d too large", N, pitch);
  B200SEG_CHECK_ARG(aligned16(dst), "nchw_to_nhwc_bf16: dst must be 16-byte aligned");
  return nchw_to_nhwc_launch<false>(src, nullptr, nullptr, nullptr, N, C, hw, pitch, dst, stream);
}

int seam_tail_backward(const void* dy, const void* y, const float* scale, int N, int C, int hw, float* dc, float* didentity,
                       cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && scale && N > 0 && C > 0 && hw > 0, "seam_tail_backward: bad arguments");
  B200SEG_CHECK_ARG(C % 8 == 0, "seam_tail_backward: C = %d is not a multiple of 8", C);
  B200SEG_CHECK_ARG(N <= 65535 && ceil_div(C, ST_CH) <= 65535, "seam_tail_backward: N = %d / C = %d too large", N, C);
  B200SEG_CHECK_ARG(aligned16(dy) && aligned16(y), "seam_tail_backward: dy and y must be 16-byte aligned");
  if (!dc && !didentity) return B200SEG_OK;
  const dim3 grid(ceil_div(hw, ST_PX), ceil_div(C, ST_CH), N);
  const __nv_bfloat16* g = reinterpret_cast<const __nv_bfloat16*>(dy);
  const __nv_bfloat16* yb = reinterpret_cast<const __nv_bfloat16*>(y);
  if (hw % 4 == 0 && aligned16(dc) && aligned16(didentity))       // (a null pointer counts as aligned)
    seam_tail_backward_kernel<true><<<grid, ST_THREADS, 0, stream>>>(g, yb, scale, C, hw, dc, didentity);
  else
    seam_tail_backward_kernel<false><<<grid, ST_THREADS, 0, stream>>>(g, yb, scale, C, hw, dc, didentity);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

}  // namespace b200seg
