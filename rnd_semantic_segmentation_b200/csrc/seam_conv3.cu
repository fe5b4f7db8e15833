// Fused backbone tail with conv3: the last Bottleneck's 1x1 conv3 runs as a tcgen05 GEMM whose epilogue applies the folded bn3,
// the residual add, the ReLU and the bf16 channels_last cast, so conv3's fp32 output c is never written nor read back.
//
// Replaces (reference file:line): core/models/feature_extractor/resnet.py:106-113
//   out = self.conv3(out); out = self.bn3(out); out += identity; out = self.relu(out)
// with conv3 a bias-free 1x1 stride-1 convolution (a plain GEMM over pixels) and bn3 folded to x * scale + bias:
//   forward   Xp = bf16(out2) NHWC [P][Cin];  W3b = bf16(W3) [Cout][Cin];  W't = bf16(scale * W3)^T [Cin][Cout]
//             y[p, co] = bf16_rn(relu((acc[p, co] * scale[co] + bias[co]) + identity[p, co])),  acc = sum_ci Xp[p, ci] W3b[co, ci]
//   backward  g = dy * (y > 0) (bf16 NHWC, exact);  didentity = g (fp32 NCHW)
//             d_out2[p, ci] = sum_co g[p, co] W'[co, ci]           (fp32 NCHW, register-store epilogue)
//             dW3[co, ci] = scale[co] * sum_p g[p, co] Xp[p, ci]    (split-K fp32 slabs summed in a fixed order: no atomics)
// bf16 operands, fp32 accumulation in TMEM: out2 and W3 are each rounded to bf16 once, the tail is applied to the fp32 accumulator
// in the fold path's __fmul_rn / __fadd_rn order, then one bf16 rounding.  No host synchronisation (capturable in a CUDA graph).
//
// conv3 under batch statistics (bn3 a training-mode BatchNorm2d / SyncBatchNorm, whose statistics need all of c before any feature):
//   forward   Xp = bf16(out2);  W3b = bf16(W3);  W't = bf16(W3)^T (unscaled)
//             c[p, co] = sum_ci Xp[p, ci] W3b[co, ci] written once as fp32 NCHW (register-store epilogue), and per 32-pixel group
//             the (mean, M2) of the stored values from the accumulator -> record [3][Cout] (count, mean, M2) in bn_stats' format;
//             the batch tail (bn_combine_stats, seam_tail_bn_forward) then runs unchanged on c
//   backward  dc as seam_tail_bn_backward computes it, rounded once to bf16 NHWC (the GEMM operand; fp32 dc is never written);
//             d_out2 = dc . W't (fp32 NCHW);  dW3 = dc^T . Xp (split-K slabs summed in a fixed order, no scale)
// The statistics are those of the stored fp32 c.  No atomics anywhere: every result is bit-identical run to run.
#include "gemm_sm100.cuh"

namespace b200seg {

// W3 fp32 [Cout][Cin] -> W3b bf16 [Cout][Cin] and W't bf16 [Cin][Cout] (W'[co, ci] = bf16_rn(scale[co] * W3[co, ci]); SCALE false:
// bf16_rn(W3[co, ci]), scale not read), through a 32 x 32 shared-memory tile
template <bool SCALE>
__device__ __forceinline__ void pack_weights(const float* __restrict__ w, const float* __restrict__ scale, int Cout, int Cin,
                                             __nv_bfloat16* __restrict__ wb, __nv_bfloat16* __restrict__ wt) {
  __shared__ float tile[32][33];
  const int ci0 = blockIdx.x * 32, co0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int co = co0 + ty + 8 * i, ci = ci0 + tx;
    if (co < Cout && ci < Cin) {
      const float v = w[(long long)co * Cin + ci];
      wb[(long long)co * Cin + ci] = __float2bfloat16_rn(v);
      tile[ty + 8 * i][tx] = SCALE ? __fmul_rn(__ldg(scale + co), v) : v;
    }
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int ci = ci0 + ty + 8 * i, co = co0 + tx;
    if (co < Cout && ci < Cin) wt[(long long)ci * Cout + co] = __float2bfloat16_rn(tile[tx][ty + 8 * i]);
  }
}

__global__ void __launch_bounds__(256) seam_conv3_pack_weights_kernel(const float* __restrict__ w, const float* __restrict__ scale,
                                                                      int Cout, int Cin, __nv_bfloat16* __restrict__ wb,
                                                                      __nv_bfloat16* __restrict__ wt) {
  pack_weights<true>(w, scale, Cout, Cin, wb, wt);
}

// the no-scale mode (conv3 under batch statistics): W't = bf16(W3)^T
__global__ void __launch_bounds__(256) seam_conv3_pack_weights_unscaled_kernel(const float* __restrict__ w, int Cout, int Cin,
                                                                               __nv_bfloat16* __restrict__ wb,
                                                                               __nv_bfloat16* __restrict__ wt) {
  pack_weights<false>(w, nullptr, Cout, Cin, wb, wt);
}

// dW[co, ci] = scale[co] * (part[0] + part[1] + ... + part[S-1])[co, ci] (SCALE false: the sum alone, scale not read), four
// consecutive ci per thread (Cin % 8 == 0)
template <bool SCALE>
__device__ __forceinline__ void wgrad_reduce(const float* __restrict__ part, int S, long long slab, const float* __restrict__ scale,
                                             int Cin, float* __restrict__ dw) {
  const long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 4;
  if (i >= slab) return;
  float4 a = __ldcs(reinterpret_cast<const float4*>(part + i));
  for (int s = 1; s < S; ++s) {
    const float4 v = __ldcs(reinterpret_cast<const float4*>(part + s * slab + i));
    a.x += v.x; a.y += v.y; a.z += v.z; a.w += v.w;
  }
  if (SCALE) {
    const float sc = __ldg(scale + i / Cin);
    a = make_float4(__fmul_rn(a.x, sc), __fmul_rn(a.y, sc), __fmul_rn(a.z, sc), __fmul_rn(a.w, sc));
  }
  reinterpret_cast<float4*>(dw)[i / 4] = a;
}

__global__ void __launch_bounds__(256) seam_conv3_wgrad_reduce_kernel(const float* __restrict__ part, int S, long long slab,
                                                                      const float* __restrict__ scale, int Cin, float* __restrict__ dw) {
  wgrad_reduce<true>(part, S, slab, scale, Cin, dw);
}

__global__ void __launch_bounds__(256) seam_conv3_wgrad_sum_kernel(const float* __restrict__ part, int S, long long slab, int Cin,
                                                                   float* __restrict__ dw) {
  wgrad_reduce<false>(part, S, slab, nullptr, Cin, dw);
}

// conv3 under batch statistics: the GEMM epilogue's (mean, M2) of every 32-pixel group gi and channel, stats [G][C], merged per
// channel in a fixed order in fp64 -> the record [3][C] = (count, mean, M2) in bn_stats' format.  Group gi holds min(32, P - 32 gi)
// pixels.  FIN_SPLIT threads per channel each merge a run of consecutive groups at once (Chan et al.'s combination of many sets:
// mean = sum n_g m_g / n, M2 = sum M2_g + n_g (m_g - mean)^2, two passes over the run, no division in the loop), then one thread
// merges the runs in order pairwise.
constexpr int FIN_CH = 32, FIN_SPLIT = 32;

__device__ __forceinline__ void chan_merge(double& n, double& mean, double& m2, double nb, double mb, double m2b) {
  const double nn = n + nb;
  const double delta = mb - mean, fb = nb / nn;
  mean += delta * fb;
  m2 += m2b + delta * delta * (n * fb);
  n = nn;
}

__global__ void __launch_bounds__(FIN_CH * FIN_SPLIT) seam_conv3_bn_record_kernel(const float2* __restrict__ stats, int G, long long P,
                                                                                  int C, double* __restrict__ record) {
  __shared__ double run[3][FIN_SPLIT][FIN_CH];
  const int ch = blockIdx.x * FIN_CH + threadIdx.x, part = threadIdx.y;
  const int per = ceil_div(G, FIN_SPLIT), g0 = part * per, g1 = min(G, g0 + per);
  double n = 0.0, mean = 0.0, m2 = 0.0;
  if (ch < C && g0 < g1) {
    double s = 0.0;
#pragma unroll 8
    for (int gi = g0; gi < g1; ++gi) s += (double)min(32LL, P - 32LL * gi) * (double)__ldg(stats + (long long)gi * C + ch).x;
    n = (double)(min(P, 32LL * g1) - 32LL * g0);
    mean = s / n;
#pragma unroll 8
    for (int gi = g0; gi < g1; ++gi) {
      const float2 q = __ldcs(stats + (long long)gi * C + ch);
      const double d = (double)q.x - mean;
      m2 += (double)q.y + (double)min(32LL, P - 32LL * gi) * d * d;
    }
  }
  run[0][part][threadIdx.x] = n;
  run[1][part][threadIdx.x] = mean;
  run[2][part][threadIdx.x] = m2;
  __syncthreads();
  if (part != 0 || ch >= C) return;
  for (int r = 1; r < FIN_SPLIT; ++r)
    if (run[0][r][threadIdx.x] > 0.0) chan_merge(n, mean, m2, run[0][r][threadIdx.x], run[1][r][threadIdx.x], run[2][r][threadIdx.x]);
  record[ch] = n;
  record[C + ch] = mean;
  record[2 * C + ch] = m2;
}

static long long align256(long long b) { return (b + 255) / 256 * 256; }
static bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15) == 0; }

// workspace (forward -> backward): Xp bf16 [P][Cin] | W't bf16 [Cin][Cout] | W3b bf16 [Cout][Cin]
long long seam_conv3_workspace_bytes(int N, int Cin, int Cout, int hw) {
  return align256((long long)N * hw * Cin * 2) + 2 * align256((long long)Cin * Cout * 2);
}

// split-K factor of the weight-gradient GEMM: one unit per CTA pair (Cout / 256 pairs of M-tiles x Cin / 256 N-tiles per split)
static int wgrad_splits(int Cin, int Cout, long long P) {
  const int units = ceil_div(ceil_div(Cout, gemm::BLOCK_M), 2) * ceil_div(Cin, gemm::BLOCK_N);
  const int kb = (int)ceil_div_ll(P, gemm::BLOCK_K);
  int s = (num_sms() / 2) / units;
  if (s > 8) s = 8;
  if (s > kb) s = kb;
  return s < 1 ? 1 : s;
}

// conv3 under batch statistics: also one split per 4096 pixels (up to 16), so that no fp32 accumulation chain in the tensor cores
// is longer than 4096 products: at the bench shape the four splits above put dW3 4.3e-5 (max-abs / max-abs) from fp64, sixteen
// bring it within 2e-5 for 50 MB more slabs
static int bn_wgrad_splits(int Cin, int Cout, long long P) {
  int s = (int)ceil_div_ll(P, 4096);
  if (s > 16) s = 16;
  const int base = wgrad_splits(Cin, Cout, P);
  return s > base ? s : base;
}

// scratch (backward only): g bf16 [P][Cout] | wgrad slabs fp32 [S][Cout][Cin]
long long seam_conv3_backward_scratch_bytes(int N, int Cin, int Cout, int hw) {
  const long long P = (long long)N * hw;
  return align256(P * Cout * 2) + (long long)wgrad_splits(Cin, Cout, P) * Cout * Cin * 4;
}

// the same layout with dc in place of g and bn_wgrad_splits slabs
long long seam_conv3_bn_backward_scratch_bytes(int N, int Cin, int Cout, int hw) {
  const long long P = (long long)N * hw;
  return align256(P * Cout * 2) + (long long)bn_wgrad_splits(Cin, Cout, P) * Cout * Cin * 4;
}

static int check_shape(const char* who, int N, int Cin, int Cout, int hw) {
  B200SEG_CHECK_ARG(N > 0 && Cin > 0 && Cout > 0 && hw > 0, "%s: bad shape", who);
  B200SEG_CHECK_ARG(Cin % 8 == 0 && Cout % 8 == 0, "%s: Cin = %d and Cout = %d must be multiples of 8", who, Cin, Cout);
  B200SEG_CHECK_ARG((long long)N * hw < (1LL << 31) - 256, "%s: too many pixels", who);
  return B200SEG_OK;
}

int seam_conv3_forward(const float* out2, const float* identity, const float* w3, const float* scale, const float* bias, int N, int Cin,
                       int Cout, int hw, void* ws, long long ws_bytes, void* y, cudaStream_t stream) {
  B200SEG_CHECK_ARG(out2 && identity && w3 && scale && bias && ws && y, "seam_conv3_forward: null pointer");
  if (int rc = check_shape("seam_conv3_forward", N, Cin, Cout, hw)) return rc;
  B200SEG_CHECK_ARG(ws_bytes >= seam_conv3_workspace_bytes(N, Cin, Cout, hw) && aligned16(ws) && aligned16(y),
                    "seam_conv3_forward: workspace too small, or workspace / y not 16-byte aligned");
  const long long P = (long long)N * hw;
  uint8_t* sp = reinterpret_cast<uint8_t*>(ws);
  __nv_bfloat16* Xp = reinterpret_cast<__nv_bfloat16*>(sp);
  __nv_bfloat16* Wt = reinterpret_cast<__nv_bfloat16*>(sp + align256(P * Cin * 2));
  __nv_bfloat16* Wb = reinterpret_cast<__nv_bfloat16*>(sp + align256(P * Cin * 2) + align256((long long)Cin * Cout * 2));
  int rc = nchw_to_nhwc_bf16(out2, N, Cin, hw, Xp, Cin, stream);
  if (rc) return rc;
  seam_conv3_pack_weights_kernel<<<dim3(ceil_div(Cin, 32), ceil_div(Cout, 32)), 256, 0, stream>>>(w3, scale, Cout, Cin, Wb, Wt);
  B200SEG_LAUNCH_CHECK();
  gemm::Operand a{Xp, false, Cin};
  gemm::Operand b{Wb, false, Cin};
  gemm::Gemm gm{a, b, (int)P, Cout, Cin, gemm::out_seam(reinterpret_cast<__nv_bfloat16*>(y), identity, scale, bias, hw)};
  gm.share = gemm::SHARE_PAIR;                // whenever sharing is on, under sharing mode 5 too: the pair is its own fallback
  gm.pair_fallback = gemm::SHARE_PAIR;
  return gemm::launch(gm, stream);
}

// conv3's two backward GEMMs from the bf16 NHWC gradient g [P][Cout] and the forward's workspace: dW3 (scaled by scale[co] over
// wgrad_splits; or, when scale is null, the plain sum over bn_wgrad_splits) and d_out2 = g . W't; either output may be null
static int conv3_backward_gemms(const __nv_bfloat16* g, const void* ws, const float* scale, int N, int Cin, int Cout, int hw, void* scratch,
                                float* d_out2, float* dw3, cudaStream_t stream) {
  const long long P = (long long)N * hw;
  const uint8_t* wp = reinterpret_cast<const uint8_t*>(ws);
  const __nv_bfloat16* Xp = reinterpret_cast<const __nv_bfloat16*>(wp);
  const __nv_bfloat16* Wt = reinterpret_cast<const __nv_bfloat16*>(wp + align256(P * Cin * 2));
  float* wpart = reinterpret_cast<float*>(reinterpret_cast<uint8_t*>(scratch) + align256(P * Cout * 2));
  int rc;
  if (dw3) {
    // dW3[co, ci] = sum_p g[p, co] Xp[p, ci]: both operands MN-major as the forward left them, split-K over pixels
    gemm::Operand a{g, true, Cout};
    gemm::Operand b{Xp, true, Cin};
    const long long slab = (long long)Cout * Cin;
    int used = 1;
    gemm::Gemm gm{a, b, Cout, Cin, (int)P, gemm::out_f32(wpart, Cin, slab)};
    gm.splits = scale ? wgrad_splits(Cin, Cout, P) : bn_wgrad_splits(Cin, Cout, P);
    gm.splits_used = &used;
    gm.share = gemm::SHARE_PAIR;
    gm.pair_fallback = gemm::SHARE_A;
    rc = gemm::launch(gm, stream);
    if (rc) return rc;
    const unsigned blocks = (unsigned)ceil_div_ll(slab / 4, 256);
    if (scale) seam_conv3_wgrad_reduce_kernel<<<blocks, 256, 0, stream>>>(wpart, used, slab, scale, Cin, dw3);
    else seam_conv3_wgrad_sum_kernel<<<blocks, 256, 0, stream>>>(wpart, used, slab, Cin, dw3);
    B200SEG_LAUNCH_CHECK();
  }
  if (d_out2) {
    // d_out2[p, ci] = sum_co g[p, co] W'[co, ci] with the pixels along M, fp32 NCHW straight from the accumulator registers
    gemm::Operand a{g, false, Cout};
    gemm::Operand b{Wt, false, Cout};
    gemm::Gemm gm{a, b, (int)P, Cin, Cout, gemm::out_f32_nchw_rows(d_out2, hw, (long long)Cin * hw)};
    gm.share = gemm::SHARE_PAIR;
    gm.pair_fallback = gemm::SHARE_B;
    rc = gemm::launch(gm, stream);
    if (rc) return rc;
  }
  return B200SEG_OK;
}

int seam_conv3_backward(const void* dy, const void* y, const void* ws, const float* scale, int N, int Cin, int Cout, int hw,
                        void* scratch, long long scratch_bytes, float* d_out2, float* dw3, float* didentity, cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && ws && scale && scratch, "seam_conv3_backward: null pointer");
  if (int rc = check_shape("seam_conv3_backward", N, Cin, Cout, hw)) return rc;
  B200SEG_CHECK_ARG(scratch_bytes >= seam_conv3_backward_scratch_bytes(N, Cin, Cout, hw) && aligned16(scratch) && aligned16(ws) &&
                        aligned16(dw3),
                    "seam_conv3_backward: scratch too small, or scratch / workspace / dW3 not 16-byte aligned");
  if (!d_out2 && !dw3 && !didentity) return B200SEG_OK;
  __nv_bfloat16* g = reinterpret_cast<__nv_bfloat16*>(scratch);
  int rc = seam_conv3_g(dy, y, N, Cout, hw, g, didentity, stream);
  if (rc) return rc;
  return conv3_backward_gemms(g, ws, scale, N, Cin, Cout, hw, scratch, d_out2, dw3, stream);
}

// ---- conv3 under batch statistics ----------------------------------------------------------------------------------------------
// forward scratch: the epilogue's (mean, M2) per 32-pixel group and channel, float2 [ceil(P / 32)][Cout]
long long seam_conv3_bn_forward_scratch_bytes(int N, int Cout, int hw) {
  return ceil_div_ll((long long)N * hw, 32) * Cout * (long long)sizeof(float2);
}

int seam_conv3_bn_forward(const float* out2, const float* w3, int N, int Cin, int Cout, int hw, void* ws, long long ws_bytes,
                          void* scratch, long long scratch_bytes, float* c, double* record, cudaStream_t stream) {
  B200SEG_CHECK_ARG(out2 && w3 && ws && scratch && c && record, "seam_conv3_bn_forward: null pointer");
  if (int rc = check_shape("seam_conv3_bn_forward", N, Cin, Cout, hw)) return rc;
  B200SEG_CHECK_ARG(ws_bytes >= seam_conv3_workspace_bytes(N, Cin, Cout, hw) && aligned16(ws),
                    "seam_conv3_bn_forward: workspace too small or not 16-byte aligned");
  B200SEG_CHECK_ARG(scratch_bytes >= seam_conv3_bn_forward_scratch_bytes(N, Cout, hw) && aligned16(scratch),
                    "seam_conv3_bn_forward: scratch too small or not 16-byte aligned");
  const long long P = (long long)N * hw;
  uint8_t* sp = reinterpret_cast<uint8_t*>(ws);
  __nv_bfloat16* Xp = reinterpret_cast<__nv_bfloat16*>(sp);
  __nv_bfloat16* Wt = reinterpret_cast<__nv_bfloat16*>(sp + align256(P * Cin * 2));
  __nv_bfloat16* Wb = reinterpret_cast<__nv_bfloat16*>(sp + align256(P * Cin * 2) + align256((long long)Cin * Cout * 2));
  float2* stats = reinterpret_cast<float2*>(scratch);
  int rc = nchw_to_nhwc_bf16(out2, N, Cin, hw, Xp, Cin, stream);
  if (rc) return rc;
  seam_conv3_pack_weights_unscaled_kernel<<<dim3(ceil_div(Cin, 32), ceil_div(Cout, 32)), 256, 0, stream>>>(w3, Cout, Cin, Wb, Wt);
  B200SEG_LAUNCH_CHECK();
  // c[p, co] = sum_ci Xp[p, ci] W3b[co, ci] as fp32 NCHW, with the pixels along M; the epilogue also writes the group statistics
  gemm::Operand a{Xp, false, Cin};
  gemm::Operand b{Wb, false, Cin};
  gemm::Gemm gm{a, b, (int)P, Cout, Cin, gemm::out_f32_nchw_rows_stats(c, hw, (long long)Cout * hw, stats)};
  rc = gemm::launch(gm, stream);
  if (rc) return rc;
  const int G = (int)ceil_div_ll(P, 32);
  seam_conv3_bn_record_kernel<<<ceil_div(Cout, FIN_CH), dim3(FIN_CH, FIN_SPLIT), 0, stream>>>(stats, G, P, Cout, record);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int seam_conv3_bn_backward(const void* dy, const void* y, const float* c, const float* mean, const float* invstd, const float* gamma,
                           const float* sums, int R, const double* count, const void* ws, int N, int Cin, int Cout, int hw, void* scratch,
                           long long scratch_bytes, float* d_out2, float* dw3, float* didentity, cudaStream_t stream) {
  B200SEG_CHECK_ARG(dy && y && c && mean && invstd && sums && count && R > 0 && ws && scratch, "seam_conv3_bn_backward: null pointer");
  if (int rc = check_shape("seam_conv3_bn_backward", N, Cin, Cout, hw)) return rc;
  B200SEG_CHECK_ARG(scratch_bytes >= seam_conv3_bn_backward_scratch_bytes(N, Cin, Cout, hw) && aligned16(scratch) && aligned16(ws) &&
                        aligned16(dw3),
                    "seam_conv3_bn_backward: scratch too small, or scratch / workspace / dW3 not 16-byte aligned");
  if (!d_out2 && !dw3) return didentity ? seam_tail_backward(dy, y, invstd, N, Cout, hw, nullptr, didentity, stream) : B200SEG_OK;
  __nv_bfloat16* dc = reinterpret_cast<__nv_bfloat16*>(scratch);
  int rc = seam_tail_bn_backward_g(dy, y, c, mean, invstd, gamma, sums, R, count, N, Cout, hw, dc, didentity, stream);
  if (rc) return rc;
  return conv3_backward_gemms(dc, ws, nullptr, N, Cin, Cout, hw, scratch, d_out2, dw3, stream);
}

}  // namespace b200seg
