// K8: multi-tensor optimizer steps for the head / discriminator parameters (SURVEY 8f rank 4).
//
// Replaces (reference file:line):
//   torch.optim.SGD(classifier.parameters(), lr=BASE_LR*10, momentum, weight_decay).step()     core/trainers/aspp_trainer.py:26,94-95
//   torch.optim.Adam(model_D.parameters(), lr=BASE_LR_D, betas=(0.9, 0.99)).step()             core/adapters/fada_adapter.py:24
// and, under data parallelism, the division of the all-reduced gradient by the world size (DDP's mean, train_distill.py:54-62):
// `grad_scale` is applied to the gradient as it is read, so the bucket can be all-reduced as a plain SUM and no separate
// averaging pass (or a second read of the 5.6 / 20.2 MB buckets) exists.
//
// One launch updates every tensor of a parameter group: the (pointer, length) table travels in the kernel parameters, a CTA
// finds its tensor by a linear scan of at most 16 prefix sums.  Pure HBM streaming: SGD reads p, g, buf and writes p, buf
// (20 B per element), Adam reads p, g, m, v and writes p, m, v (28 B per element); 128-bit accesses on the aligned body of each
// tensor, scalar head/tail.
//
// Arithmetic follows torch/optim/sgd.py::_single_tensor_sgd and torch/optim/adam.py::_single_tensor_adam op by op: every eager
// op rounds once, and ATen's `a + alpha * b` forms (add_/addcmul_/addcdiv_/lerp_ with a scalar) are single FMAs, as its CPU
// (vec::fmadd) and CUDA (contracted) kernels compute them:
//   SGD   g' = g*scale; g' = fma(wd, p, g'); buf = first ? g' : fma(1-damp, g', buf*mom); d = nesterov ? fma(mom, buf, g') : buf;
//         p = fma(-lr, d, p)
//   Adam  g' likewise; m = fma(1-b1, g'-m, m) [lerp_]; v = fma((1-b2)*g', g', v*b2) [mul_ + addcmul_];
//         p = fma(-lr/bc1, m / (sqrt(v)/sqrt(bc2) + eps), p),   bc_i = 1 - b_i^step (double, on the host, as Python computes it)
// Tests hold the result to 1e-6 relative of torch.optim on the same inputs (one-ulp differences where a backend of the reference
// rounds an intermediate the other way).
#include "common.cuh"
#include "host_api.h"

namespace b200seg {

constexpr int OPT_MAX_TENSORS = 16;
constexpr int OPT_THREADS = 256;
constexpr int OPT_CHUNK = OPT_THREADS * 4 * 4;      // elements per CTA step: four float4 per thread

struct OptTable {
  float* p[OPT_MAX_TENSORS];
  const float* g[OPT_MAX_TENSORS];
  float* s1[OPT_MAX_TENSORS];        // SGD: momentum buffer; Adam: exp_avg
  float* s2[OPT_MAX_TENSORS];        // Adam: exp_avg_sq
  long long chunk0[OPT_MAX_TENSORS + 1];   // prefix sums of ceil(numel / OPT_CHUNK)
  long long numel[OPT_MAX_TENSORS];
  int n;
};

struct SgdArgs {
  float lr, momentum, dampening_c, weight_decay, grad_scale;   // dampening_c = 1 - dampening
  int nesterov, first_step, use_scale;
};
struct AdamArgs {
  float lr, beta1_c, beta2, beta2_c, eps, weight_decay, grad_scale;   // beta1_c = 1 - beta1, beta2_c = 1 - beta2
  float step_size, bc2_sqrt;                                        // lr / bc1, sqrt(bc2)
  int use_scale;
};

__device__ __forceinline__ float sgd_one(float& p, float g, float& buf, const SgdArgs& a) {
  if (a.use_scale) g = __fmul_rn(g, a.grad_scale);
  if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
  float d = g;
  if (a.momentum != 0.f) {
    buf = a.first_step ? g : fmaf(a.dampening_c, g, __fmul_rn(buf, a.momentum));
    d = a.nesterov ? fmaf(a.momentum, buf, g) : buf;
  }
  p = fmaf(-a.lr, d, p);
  return p;
}

__device__ __forceinline__ float adam_one(float& p, float g, float& m, float& v, const AdamArgs& a) {
  if (a.use_scale) g = __fmul_rn(g, a.grad_scale);
  if (a.weight_decay != 0.f) g = fmaf(a.weight_decay, p, g);
  m = fmaf(a.beta1_c, __fsub_rn(g, m), m);                                       // exp_avg.lerp_(grad, 1 - beta1)
  v = fmaf(__fmul_rn(a.beta2_c, g), g, __fmul_rn(v, a.beta2));                   // mul_(beta2).addcmul_(grad, grad, value=1-beta2)
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), a.bc2_sqrt), a.eps);    // (sqrt / bias_correction2_sqrt).add_(eps)
  p = fmaf(-a.step_size, __fdiv_rn(m, denom), p);                                // addcdiv_(exp_avg, denom, value=-step_size)
  return p;
}

template <bool ADAM>
__global__ void __launch_bounds__(OPT_THREADS) optim_step_kernel(const OptTable t, const SgdArgs sa, const AdamArgs aa) {
  const long long total = t.chunk0[t.n];
  for (long long chunk = blockIdx.x; chunk < total; chunk += gridDim.x) {
    int k = 0;
    while (k + 1 < t.n && chunk >= t.chunk0[k + 1]) ++k;
    const long long base = (chunk - t.chunk0[k]) * OPT_CHUNK;
    const long long n = t.numel[k];
    float* __restrict__ P = t.p[k];
    const float* __restrict__ G = t.g[k];
    float* __restrict__ S1 = t.s1[k];
    float* __restrict__ S2 = t.s2[k];
    const bool need_s1 = ADAM || sa.momentum != 0.f;
    const bool aligned = ((reinterpret_cast<uintptr_t>(P) | reinterpret_cast<uintptr_t>(G) | reinterpret_cast<uintptr_t>(S1) |
                           reinterpret_cast<uintptr_t>(S2)) & 15) == 0;
    if (aligned && base + OPT_CHUNK <= n) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const long long i = base + ((long long)j * OPT_THREADS + threadIdx.x) * 4;
        float4 p4 = *reinterpret_cast<const float4*>(P + i);
        const float4 g4 = ld_stream_f4(G + i);
        float4 a4 = need_s1 && !(!ADAM && sa.first_step) ? *reinterpret_cast<const float4*>(S1 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        if (ADAM) {
          float4 b4 = *reinterpret_cast<const float4*>(S2 + i);
          adam_one(p4.x, g4.x, a4.x, b4.x, aa); adam_one(p4.y, g4.y, a4.y, b4.y, aa);
          adam_one(p4.z, g4.z, a4.z, b4.z, aa); adam_one(p4.w, g4.w, a4.w, b4.w, aa);
          *reinterpret_cast<float4*>(S2 + i) = b4;
        } else {
          sgd_one(p4.x, g4.x, a4.x, sa); sgd_one(p4.y, g4.y, a4.y, sa);
          sgd_one(p4.z, g4.z, a4.z, sa); sgd_one(p4.w, g4.w, a4.w, sa);
        }
        if (need_s1) *reinterpret_cast<float4*>(S1 + i) = a4;
        *reinterpret_cast<float4*>(P + i) = p4;
      }
    } else {
      const long long end = base + OPT_CHUNK < n ? base + OPT_CHUNK : n;
      for (long long i = base + threadIdx.x; i < end; i += OPT_THREADS) {
        float p1 = P[i];
        const float g1 = G[i];
        float a1 = need_s1 && !(!ADAM && sa.first_step) ? S1[i] : 0.f;
        if (ADAM) {
          float b1 = S2[i];
          adam_one(p1, g1, a1, b1, aa);
          S2[i] = b1;
        } else {
          sgd_one(p1, g1, a1, sa);
        }
        if (need_s1) S1[i] = a1;
        P[i] = p1;
      }
    }
  }
}

static int fill_table(OptTable& t, int n, float* const* params, const float* const* grads, float* const* s1, float* const* s2,
                      const long long* numels, bool need_s1, bool need_s2, const char* who) {
  t.n = n;
  long long c = 0;
  for (int k = 0; k < n; ++k) {
    B200SEG_CHECK_ARG(params[k] && grads[k] && numels[k] > 0, "%s: tensor %d has a null pointer or no elements", who, k);
    B200SEG_CHECK_ARG(!need_s1 || (s1 && s1[k]), "%s: tensor %d has no first state buffer", who, k);
    B200SEG_CHECK_ARG(!need_s2 || (s2 && s2[k]), "%s: tensor %d has no second state buffer", who, k);
    t.p[k] = params[k];
    t.g[k] = grads[k];
    t.s1[k] = need_s1 ? s1[k] : nullptr;
    t.s2[k] = need_s2 ? s2[k] : nullptr;
    t.numel[k] = numels[k];
    t.chunk0[k] = c;
    c += ceil_div_ll(numels[k], OPT_CHUNK);
  }
  t.chunk0[n] = c;
  return B200SEG_OK;
}

// the pointer arrays are HOST arrays of device pointers
int sgd_step(int n_tensors, float* const* params, const float* const* grads, float* const* momentum_bufs, const long long* numels,
             float lr, float momentum, float dampening, float weight_decay, int nesterov, int first_step, float grad_scale,
             cudaStream_t stream) {
  B200SEG_CHECK_ARG(n_tensors > 0 && params && grads && numels, "sgd_step: bad tensor table");
  B200SEG_CHECK_ARG(!nesterov || (momentum > 0.f && dampening == 0.f), "sgd_step: Nesterov momentum requires a momentum and zero dampening");
  SgdArgs a;
  a.lr = lr; a.momentum = momentum; a.dampening_c = 1.0f - dampening; a.weight_decay = weight_decay; a.grad_scale = grad_scale;
  a.nesterov = nesterov ? 1 : 0; a.first_step = first_step ? 1 : 0; a.use_scale = grad_scale != 1.0f;
  AdamArgs unused = {};
  for (int k0 = 0; k0 < n_tensors; k0 += OPT_MAX_TENSORS) {
    const int n = n_tensors - k0 < OPT_MAX_TENSORS ? n_tensors - k0 : OPT_MAX_TENSORS;
    OptTable t;
    int rc = fill_table(t, n, params + k0, grads + k0, momentum_bufs ? momentum_bufs + k0 : nullptr, nullptr, numels + k0,
                        momentum != 0.f, false, "sgd_step");
    if (rc) return rc;
    const long long cap = (long long)num_sms() * 8;
    const int grid = (int)(t.chunk0[n] < cap ? t.chunk0[n] : cap);
    optim_step_kernel<false><<<grid, OPT_THREADS, 0, stream>>>(t, a, unused);
    B200SEG_LAUNCH_CHECK();
  }
  return B200SEG_OK;
}

int adam_step(int n_tensors, float* const* params, const float* const* grads, float* const* exp_avg, float* const* exp_avg_sq,
              const long long* numels, float lr, float beta1, float beta2, float eps, float weight_decay, long long step,
              float grad_scale, cudaStream_t stream) {
  B200SEG_CHECK_ARG(n_tensors > 0 && params && grads && numels && exp_avg && exp_avg_sq, "adam_step: bad tensor table");
  B200SEG_CHECK_ARG(step >= 1, "adam_step: step must be >= 1 (the value AFTER this update, as torch counts it)");
  AdamArgs a;
  // python: bias_correction1 = 1 - beta1 ** step (double); step_size = lr / bias_correction1; bias_correction2_sqrt = sqrt(1 - beta2 ** step)
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  a.lr = lr; a.beta1_c = (float)(1.0 - (double)beta1); a.beta2 = beta2; a.beta2_c = (float)(1.0 - (double)beta2);
  a.eps = eps; a.weight_decay = weight_decay; a.grad_scale = grad_scale;
  a.step_size = (float)((double)lr / bc1); a.bc2_sqrt = (float)sqrt(bc2); a.use_scale = grad_scale != 1.0f;
  SgdArgs unused = {};
  for (int k0 = 0; k0 < n_tensors; k0 += OPT_MAX_TENSORS) {
    const int n = n_tensors - k0 < OPT_MAX_TENSORS ? n_tensors - k0 : OPT_MAX_TENSORS;
    OptTable t;
    int rc = fill_table(t, n, params + k0, grads + k0, exp_avg + k0, exp_avg_sq + k0, numels + k0, true, true, "adam_step");
    if (rc) return rc;
    const long long cap = (long long)num_sms() * 8;
    const int grid = (int)(t.chunk0[n] < cap ? t.chunk0[n] : cap);
    optim_step_kernel<true><<<grid, OPT_THREADS, 0, stream>>>(t, unused, a);
    B200SEG_LAUNCH_CHECK();
  }
  return B200SEG_OK;
}

}  // namespace b200seg
