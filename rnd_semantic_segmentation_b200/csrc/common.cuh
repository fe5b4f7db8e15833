// Shared helpers for the b200seg kernels (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>

#define B200SEG_OK 0
#define B200SEG_ERR_ARG 1
#define B200SEG_ERR_CUDA 2
#define B200SEG_ERR_UNSUPPORTED 3

namespace b200seg {

void set_error(const char* fmt, ...);           // api.cu
int num_sms();                                   // api.cu (cached per process)
void count_launch();                             // api.cu: kernels launched by this library (bench evidence)
// api.cu: when profiling is on, bracket a launch with CUDA events on its stream under `tag`
void profile_begin(int tag, cudaStream_t stream);
void profile_end(int tag, cudaStream_t stream);

#define B200SEG_CHECK_ARG(cond, ...)                                  \
  do {                                                                \
    if (!(cond)) {                                                    \
      ::b200seg::set_error(__VA_ARGS__);                              \
      return B200SEG_ERR_ARG;                                         \
    }                                                                 \
  } while (0)

#define B200SEG_CUDA(call)                                                              \
  do {                                                                                  \
    cudaError_t e__ = (call);                                                           \
    if (e__ != cudaSuccess) {                                                           \
      ::b200seg::set_error("%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__),     \
                           __FILE__, __LINE__);                                         \
      return B200SEG_ERR_CUDA;                                                          \
    }                                                                                   \
  } while (0)

#define B200SEG_LAUNCH_CHECK()             \
  do {                                     \
    ::b200seg::count_launch();             \
    B200SEG_CUDA(cudaGetLastError());      \
  } while (0)

__host__ __device__ __forceinline__ int ceil_div(int a, int b) { return (a + b - 1) / b; }
__host__ __device__ __forceinline__ long long ceil_div_ll(long long a, long long b) { return (a + b - 1) / b; }

// ---- align_corners=True bilinear taps, the ATen way -----------------------------------------
// (ATen/native/UpSample.h area_pixel_compute_scale / area_pixel_compute_source_index with
//  align_corners=true: scale = (float)(in-1)/(out-1) [0 when out<=1]; src = scale*dst;
//  i0 = (int)src; i1 = i0 + (i0 < in-1); l1 = src - i0; l0 = 1 - l1.)
__host__ __device__ __forceinline__ float ac_scale(int in_size, int out_size) {
  return out_size > 1 ? (float)(in_size - 1) / (float)(out_size - 1) : 0.0f;
}
struct Tap {
  int i0, i1;
  float l0, l1;
};
__device__ __forceinline__ Tap ac_tap(float scale, int dst, int in_size) {
  Tap t;
  const float src = scale * (float)dst;
  t.i0 = (int)src;
  t.i1 = t.i0 + ((t.i0 < in_size - 1) ? 1 : 0);
  t.l1 = src - (float)t.i0;
  t.l0 = 1.0f - t.l1;
  return t;
}
// First output index whose i0 is >= cell (monotone in dst); returns out_size if none.
__device__ __forceinline__ int ac_first_dst(float scale, int cell, int in_size, int out_size) {
  if (cell <= 0) return 0;
  if (scale <= 0.0f) return out_size;
  int d = (int)((float)cell / scale);
  if (d > out_size) d = out_size;
  if (d < 0) d = 0;
  while (d > 0 && (int)(scale * (float)(d - 1)) >= cell) --d;
  while (d < out_size && (int)(scale * (float)d) < cell) ++d;
  return d;
}

__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// ---- sm_100 packed fp32x2 arithmetic (FFMA2 / FMUL2 / FADD2: two IEEE fp32 results per issue slot) and the
//      3-input fp32 max (FMNMX3).  Each half is rounded exactly like the scalar instruction. ---------------------
__device__ __forceinline__ unsigned long long f2_bits(float2 v) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(v.x), "f"(v.y));
  return r;
}
__device__ __forceinline__ float2 bits_f2(unsigned long long r) {
  float2 v;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(v.x), "=f"(v.y) : "l"(r));
  return v;
}
__device__ __forceinline__ float2 fma2(float2 a, float2 b, float2 c) {
  unsigned long long d;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)), "l"(f2_bits(c)));
  return bits_f2(d);
}
__device__ __forceinline__ float2 mul2(float2 a, float2 b) {
  unsigned long long d;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)));
  return bits_f2(d);
}
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  unsigned long long d;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(f2_bits(a)), "l"(f2_bits(b)));
  return bits_f2(d);
}
__device__ __forceinline__ float fmax3(float a, float b, float c) {
  float d;
  asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}

// max of f[LO..HI) as a tree of 3-input maxima (depth log3 instead of a serial chain)
template <int LO, int HI, int CT>
__device__ __forceinline__ float tree_max3(const float (&f)[CT]) {
  constexpr int n = HI - LO;
  if constexpr (n == 1) return f[LO];
  else if constexpr (n == 2) return fmaxf(f[LO], f[LO + 1]);
  else if constexpr (n == 3) return fmax3(f[LO], f[LO + 1], f[LO + 2]);
  else {
    constexpr int a = (n + 2) / 3, b = (n - a + 1) / 2;
    return fmax3(tree_max3<LO, LO + a, CT>(f), tree_max3<LO + a, LO + a + b, CT>(f), tree_max3<LO + a + b, HI, CT>(f));
  }
}

// ---- per-thread asynchronous global->shared copies (LDGSTS) ----------------------------------
__device__ __forceinline__ void cp_async_8(void* smem_dst, const void* gmem_src) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(s), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() {
  asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory");
}

// ---- explicit shared-space accesses on 32-bit shared addresses (no generic->shared conversion per access) ----
__device__ __forceinline__ unsigned smem_u32(const void* p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ float lds_f32(unsigned a) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ float4 lds_v4f32(unsigned a) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint2 lds_v2u32(unsigned a) {
  uint2 v;
  asm volatile("ld.shared.v2.u32 {%0,%1}, [%2];" : "=r"(v.x), "=r"(v.y) : "r"(a));
  return v;
}
__device__ __forceinline__ unsigned lds_u8(unsigned a) {
  unsigned v;
  asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(a));
  return v;
}
__device__ __forceinline__ void sts_u8(unsigned a, unsigned v) { asm volatile("st.shared.u8 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void sts_f32(unsigned a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }
__device__ __forceinline__ void smem_inc_u8(unsigned a) {      // thread-private byte counter += 1
  asm volatile("{ .reg .u32 t; ld.shared.u8 t, [%0]; add.u32 t, t, 1; st.shared.u8 [%0], t; }" ::"r"(a) : "memory");
}
__device__ __forceinline__ void cp_async_8s(unsigned smem_dst, const void* gmem_src) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_dst), "l"(gmem_src) : "memory");
}

// fp32 -> the nearest TF32 value (10 explicit mantissa bits), ties to even: the low 13 mantissa bits cleared.  Values a tensor
// core reads as TF32 operands are stored this way, so the product does not depend on how the hardware treats the dropped bits.
// Inf / NaN pass unchanged.
__device__ __forceinline__ float tf32_rn(float x) {
  uint32_t u = __float_as_uint(x);
  if ((u & 0x7f800000u) != 0x7f800000u) u = (u + 0xfffu + ((u >> 13) & 1u)) & ~0x1fffu;
  return __uint_as_float(u);
}

// ---- warp / block reductions ----------------------------------------------------------------
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- streaming 128-bit loads/stores (read-once data: bypass L1 allocation) --------------------
__device__ __forceinline__ int4 ld_stream_v4(const void* p) {
  int4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.s32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ float4 ld_stream_f4(const void* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ long long ld_stream_s64(const void* p) {
  long long r;
  asm volatile("ld.global.nc.L1::no_allocate.s64 %0, [%1];" : "=l"(r) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream_f4(void* p, float4 v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

}  // namespace b200seg
