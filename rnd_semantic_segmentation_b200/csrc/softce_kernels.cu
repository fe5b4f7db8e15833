// K3: soft-label cross-entropy on materialised operands (the reference's API-level contract).
//
// Replaces (reference file:line):
//   soft_label_cross_entropy(pred, soft_label, pixel_weights=None)   core/utils/utility.py:172-177
//     loss = mean_{N,H,W}( [w *] sum_c( -q_c * log_softmax(p)_c ) )
//          per pixel as  log(s) * sum_k q_k - sum_k q_k * (p_k - r),  s = sum_k exp(p_k - m),  with m the pixel's maximum and r
//          one of its own logits (m, or the first class on the online path): every term is a difference of logits, so a logit
//          offset common to all classes (which cancels in the loss) costs no precision
//     d loss / d p_c = ( softmax(p)_c * sum_k q_k - q_c ) * w / (N*H*W)
//   callers: core/combos/aspp_fada.py:111,120,124 on [N, 2C, H, W] fp32 operands.
//
// Pure HBM streaming: forward reads p and q once (8*K B/px), backward reads p and q and writes the
// gradient (12*K B/px).  One thread per pixel; the K class values of a pixel sit HW*4 bytes apart
// (NCHW), so every load/store instruction of a warp is one fully coalesced 128-byte line, and all K
// loads of a thread are issued before the first use (K independent requests in flight per thread).
#include "common.cuh"
#include "host_api.h"

namespace b200seg {

constexpr int K3_THREADS = 256;

template <int KT>
__global__ void __launch_bounds__(K3_THREADS) k3_softce_fwd(const float* __restrict__ pred, const float* __restrict__ soft,
                                                            const float* __restrict__ wts, int K, long long HW,
                                                            long long total_px, float* __restrict__ partial) {
  __shared__ float red[K3_THREADS / 32];
  float acc = 0.f;
  for (long long i = blockIdx.x * (long long)K3_THREADS + threadIdx.x; i < total_px; i += (long long)gridDim.x * K3_THREADS) {
    const long long n = i / HW;
    const long long base = n * K * HW + (i - n * HW);
    float p[KT];
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) p[k] = __ldcs(pred + base + k * HW);
    float m = -INFINITY;
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) m = fmaxf(m, p[k]);
    float s = 0.f, sq = 0.f, sqd = 0.f;
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) {
        const float q = __ldcs(soft + base + k * HW);
        const float d = p[k] - m;
        s += fast_exp2(d * 1.4426950408889634f);
        sq += q;
        sqd = fmaf(q, d, sqd);
      }
    float l = __logf(s) * sq - sqd;
    if (wts) l *= __ldcs(wts + i);
    acc += l;
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < K3_THREADS / 32; ++i) t += red[i];
    partial[blockIdx.x] = t;
  }
}

__global__ void __launch_bounds__(256) k3_finalize(const float* partial, int n, double inv_count, float* out) {
  __shared__ double sl[8];
  double l = 0.0;
  for (int i = threadIdx.x; i < n; i += 256) l += (double)partial[i];
  l = warp_sum_d(l);
  if ((threadIdx.x & 31) == 0) sl[threadIdx.x >> 5] = l;
  __syncthreads();
  if (threadIdx.x == 0) {
    double L = 0.0;
    for (int i = 0; i < 8; ++i) L += sl[i];
    out[0] = (float)(L * inv_count);
  }
}

template <int KT>
__global__ void __launch_bounds__(K3_THREADS) k3_softce_bwd(const float* __restrict__ pred, const float* __restrict__ soft,
                                                            const float* __restrict__ wts, const float* __restrict__ grad_out,
                                                            int K, long long HW, long long total_px, float inv_count,
                                                            float* __restrict__ grad) {
  const float go = (grad_out ? grad_out[0] : 1.f) * inv_count;
  for (long long i = blockIdx.x * (long long)K3_THREADS + threadIdx.x; i < total_px; i += (long long)gridDim.x * K3_THREADS) {
    const long long n = i / HW;
    const long long base = n * K * HW + (i - n * HW);
    float p[KT], q[KT];
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) p[k] = __ldcs(pred + base + k * HW);
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) q[k] = __ldcs(soft + base + k * HW);
    float m = -INFINITY, sq = 0.f;
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) { m = fmaxf(m, p[k]); sq += q[k]; }
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) {
        p[k] = fast_exp2((p[k] - m) * 1.4426950408889634f);
        s += p[k];
      }
    const float wgt = (wts ? __ldcs(wts + i) : 1.f) * go;
    const float a = wgt * sq * __fdividef(1.f, s);
#pragma unroll
    for (int k = 0; k < KT; ++k)
      if (k < K) __stcs(grad + base + k * HW, fmaf(a, p[k], -wgt * q[k]));
  }
}

// ---- 128-bit vectorised variants: one thread per 4 consecutive pixels (HW % 4 == 0, 16-byte aligned tensors) --------
// forward: online softmax over chunks of K3_CH class planes (2 * K3_CH independent 16-byte loads in flight per thread),
// optionally saving {m, sum_k q_k / s} per pixel (the maximum and the softmax scale of the soft-label mass) so that the backward
// is ONE streaming pass with no register arrays.
#ifndef K3_CH_DEF
#define K3_CH_DEF 4
#endif
#ifndef K3_MINB
#define K3_MINB 2
#endif
constexpr int K3_CH = K3_CH_DEF;
constexpr float K3_L2E = 1.4426950408889634f, K3_LN2 = 0.6931471805599453f;

__global__ void __launch_bounds__(K3_THREADS, K3_MINB) k3_softce_fwd_v4(const float* __restrict__ pred, const float* __restrict__ soft,
                                                               const float* __restrict__ wts, int K, long long HW,
                                                               long long total_px, float* __restrict__ stats,
                                                               float* __restrict__ partial) {
  __shared__ float red[K3_THREADS / 32];
  float acc = 0.f;
  const long long quads = total_px >> 2;
  for (long long qi = blockIdx.x * (long long)K3_THREADS + threadIdx.x; qi < quads; qi += (long long)gridDim.x * K3_THREADS) {
    const long long i = qi << 2;
    const long long n = i / HW;
    const float* pp = pred + n * K * HW + (i - n * HW);
    const float* qp = soft + n * K * HW + (i - n * HW);
    float m[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
    float sden[4] = {0.f, 0.f, 0.f, 0.f}, sq[4] = {0.f, 0.f, 0.f, 0.f}, sqd[4] = {0.f, 0.f, 0.f, 0.f};
    float r[4];                                      // reference logit of sqd = sum q * (p - r): the pixel's first class
    auto load_chunk = [&](float4 (&P)[K3_CH], float4 (&Q)[K3_CH], int k0) {
#pragma unroll
      for (int k = 0; k < K3_CH; ++k) {
        if (k0 + k < K) {
          P[k] = ld_stream_f4(pp + (long long)(k0 + k) * HW);
          Q[k] = ld_stream_f4(qp + (long long)(k0 + k) * HW);
        } else {
          P[k] = make_float4(-INFINITY, -INFINITY, -INFINITY, -INFINITY);
          Q[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
      }
    };
    auto fold_chunk = [&](const float4 (&P)[K3_CH], const float4 (&Q)[K3_CH], int k0) {
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float cm = -INFINITY;
#pragma unroll
        for (int k = 0; k < K3_CH; ++k) cm = fmaxf(cm, (&P[k].x)[e]);
        const float mn = fmaxf(m[e], cm);
        float sd = sden[e] * fast_exp2((m[e] - mn) * K3_L2E);             // m = -inf on the first chunk -> ex2(-inf) = 0
        if (k0 == 0) r[e] = (&P[0].x)[e];
#pragma unroll
        for (int k = 0; k < K3_CH; ++k) {
          const float pv = (&P[k].x)[e], qv = (&Q[k].x)[e];
          sd += fast_exp2((pv - mn) * K3_L2E);                             // padding planes: ex2(-inf) = 0
          sq[e] += qv;
          sqd[e] = fmaf(qv, (k0 + k < K) ? pv - r[e] : 0.f, sqd[e]);
        }
        sden[e] = sd;
        m[e] = mn;
      }
    };
    // two chunk buffers: the loads of chunk c+1 are in flight while chunk c is folded into the running statistics
    float4 PA[K3_CH], QA[K3_CH], PB[K3_CH], QB[K3_CH];
    load_chunk(PA, QA, 0);
    for (int k0 = 0; k0 < K; k0 += 2 * K3_CH) {
      if (k0 + K3_CH < K) load_chunk(PB, QB, k0 + K3_CH);
      fold_chunk(PA, QA, k0);
      if (k0 + 2 * K3_CH < K) load_chunk(PA, QA, k0 + 2 * K3_CH);
      if (k0 + K3_CH < K) fold_chunk(PB, QB, k0 + K3_CH);
    }
    float l[4];                                      // lse - r = (m - r) + log(s)
#pragma unroll
    for (int e = 0; e < 4; ++e) l[e] = (m[e] - r[e]) + __log2f(sden[e]) * K3_LN2;
    float4 wv = make_float4(1.f, 1.f, 1.f, 1.f);
    if (wts) wv = ld_stream_f4(wts + i);
    acc += (l[0] * sq[0] - sqd[0]) * wv.x + (l[1] * sq[1] - sqd[1]) * wv.y + (l[2] * sq[2] - sqd[2]) * wv.z +
           (l[3] * sq[3] - sqd[3]) * wv.w;
    if (stats) {
      st_stream_f4(stats + i, make_float4(m[0], m[1], m[2], m[3]));
      st_stream_f4(stats + total_px + i, make_float4(__fdividef(sq[0], sden[0]), __fdividef(sq[1], sden[1]),
                                                     __fdividef(sq[2], sden[2]), __fdividef(sq[3], sden[3])));
    }
  }
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < K3_THREADS / 32; ++i) t += red[i];
    partial[blockIdx.x] = t;
  }
}

// backward from the saved per-pixel {m, sum q / s}: grad_k = w * go / (NHW) * (exp(p_k - m) * sum_q / s - q_k), one streaming pass
__global__ void __launch_bounds__(K3_THREADS, K3_MINB) k3_softce_bwd_stats_v4(const float* __restrict__ pred, const float* __restrict__ soft,
                                                                     const float* __restrict__ wts, const float* __restrict__ stats,
                                                                     const float* __restrict__ grad_out, int K, long long HW,
                                                                     long long total_px, float inv_count, float* __restrict__ grad) {
  const float go = (grad_out ? grad_out[0] : 1.f) * inv_count;
  const long long quads = total_px >> 2;
  for (long long qi = blockIdx.x * (long long)K3_THREADS + threadIdx.x; qi < quads; qi += (long long)gridDim.x * K3_THREADS) {
    const long long i = qi << 2;
    const long long n = i / HW;
    const long long base = n * K * HW + (i - n * HW);
    const float4 m = ld_stream_f4(stats + i), sqs = ld_stream_f4(stats + total_px + i);
    float4 a = make_float4(go, go, go, go);
    if (wts) { const float4 wv = ld_stream_f4(wts + i); a = make_float4(go * wv.x, go * wv.y, go * wv.z, go * wv.w); }
    const float4 as = make_float4(a.x * sqs.x, a.y * sqs.y, a.z * sqs.z, a.w * sqs.w);
    for (int k0 = 0; k0 < K; k0 += K3_CH) {
      float4 P[K3_CH], Q[K3_CH];
#pragma unroll
      for (int k = 0; k < K3_CH; ++k)
        if (k0 + k < K) {
          P[k] = ld_stream_f4(pred + base + (long long)(k0 + k) * HW);
          Q[k] = ld_stream_f4(soft + base + (long long)(k0 + k) * HW);
        }
#pragma unroll
      for (int k = 0; k < K3_CH; ++k)
        if (k0 + k < K) {
          float4 gv;
          gv.x = fmaf(as.x, fast_exp2((P[k].x - m.x) * K3_L2E), -a.x * Q[k].x);
          gv.y = fmaf(as.y, fast_exp2((P[k].y - m.y) * K3_L2E), -a.y * Q[k].y);
          gv.z = fmaf(as.z, fast_exp2((P[k].z - m.z) * K3_L2E), -a.z * Q[k].z);
          gv.w = fmaf(as.w, fast_exp2((P[k].w - m.w) * K3_L2E), -a.w * Q[k].w);
          st_stream_f4(grad + base + (long long)(k0 + k) * HW, gv);
        }
    }
  }
}

long long k3_workspace_bytes() { return 4096 * 4 + 64; }
long long k3_stats_bytes(int N, int H, int W) { return 8LL * N * H * W + 64; }

static bool k3_vec_ok(const void* a, const void* b, const void* c, const void* d, long long HW) {
  return HW % 4 == 0 && ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) |
                          reinterpret_cast<uintptr_t>(d)) & 15) == 0;
}


static int k3_grid(long long total_px) {
  long long blocks = ceil_div_ll(total_px, K3_THREADS);
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  if (blocks > 4096) blocks = 4096;
  return (int)blocks;
}

int k3_forward(const float* pred, const float* soft, const float* wts, int N, int K, int H, int W, void* workspace,
               long long workspace_bytes, float* loss_out, cudaStream_t stream, float* stats) {
  B200SEG_CHECK_ARG(pred && soft && workspace && loss_out, "soft_ce_forward: null pointer");
  B200SEG_CHECK_ARG(N > 0 && K > 0 && H > 0 && W > 0, "soft_ce_forward: bad shape");
  B200SEG_CHECK_ARG(K <= 64, "soft_ce_forward: %d channels > 64 is not supported", K);
  B200SEG_CHECK_ARG(workspace_bytes >= k3_workspace_bytes(), "soft_ce_forward: workspace too small");
  const long long HW = (long long)H * W, total = HW * N;
  float* partial = reinterpret_cast<float*>(workspace);
  if (k3_vec_ok(pred, soft, wts, stats, HW)) {
    const int gridv = k3_grid(total >> 2);
    profile_begin(8, stream);
    k3_softce_fwd_v4<<<gridv, K3_THREADS, 0, stream>>>(pred, soft, wts, K, HW, total, stats, partial);
    profile_end(8, stream);
    B200SEG_LAUNCH_CHECK();
    k3_finalize<<<1, 256, 0, stream>>>(partial, gridv, 1.0 / (double)total, loss_out);
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  B200SEG_CHECK_ARG(stats == nullptr, "soft_ce_forward: per-pixel statistics need H*W %% 4 == 0 and 16-byte aligned tensors");
  const int grid = k3_grid(total);
  profile_begin(8, stream);
  if (K <= 4) k3_softce_fwd<4><<<grid, K3_THREADS, 0, stream>>>(pred, soft, wts, K, HW, total, partial);
  else if (K <= 38) k3_softce_fwd<38><<<grid, K3_THREADS, 0, stream>>>(pred, soft, wts, K, HW, total, partial);
  else k3_softce_fwd<64><<<grid, K3_THREADS, 0, stream>>>(pred, soft, wts, K, HW, total, partial);
  profile_end(8, stream);
  B200SEG_LAUNCH_CHECK();
  k3_finalize<<<1, 256, 0, stream>>>(partial, grid, 1.0 / (double)total, loss_out);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

int k3_backward(const float* pred, const float* soft, const float* wts, const float* grad_out, int N, int K, int H, int W,
                float* grad_pred, cudaStream_t stream, const float* stats) {
  B200SEG_CHECK_ARG(pred && soft && grad_pred, "soft_ce_backward: null pointer");
  B200SEG_CHECK_ARG(N > 0 && K > 0 && H > 0 && W > 0, "soft_ce_backward: bad shape");
  B200SEG_CHECK_ARG(K <= 64, "soft_ce_backward: %d channels > 64 is not supported", K);
  const long long HW = (long long)H * W, total = HW * N;
  const int grid = k3_grid(total);
  const float inv = (float)(1.0 / (double)total);
  if (stats) {
    B200SEG_CHECK_ARG(k3_vec_ok(pred, soft, wts, grad_pred, HW) && (reinterpret_cast<uintptr_t>(stats) & 15) == 0,
                      "soft_ce_backward: per-pixel statistics need H*W %% 4 == 0 and 16-byte aligned tensors");
    profile_begin(9, stream);
    k3_softce_bwd_stats_v4<<<k3_grid(total >> 2), K3_THREADS, 0, stream>>>(pred, soft, wts, stats, grad_out, K, HW, total, inv, grad_pred);
    profile_end(9, stream);
    B200SEG_LAUNCH_CHECK();
    return B200SEG_OK;
  }
  profile_begin(9, stream);
  if (K <= 4) k3_softce_bwd<4><<<grid, K3_THREADS, 0, stream>>>(pred, soft, wts, grad_out, K, HW, total, inv, grad_pred);
  else if (K <= 38) k3_softce_bwd<38><<<grid, K3_THREADS, 0, stream>>>(pred, soft, wts, grad_out, K, HW, total, inv, grad_pred);
  else k3_softce_bwd<64><<<grid, K3_THREADS, 0, stream>>>(pred, soft, wts, grad_out, K, HW, total, inv, grad_pred);
  profile_end(9, stream);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

}  // namespace b200seg
