// Stand-alone timing of the library's fp32 NCHW -> bf16 NHWC tile pass (csrc/seam_tail_kernels.cu, 32 channels x 128 pixels)
// against the 64 x 64 scalar-load pack kernel it replaced:
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o /tmp/nt profiles/micro/nhwc_tile_micro.cu && /tmp/nt
// pack: 8 x 2048 x 64 x 128 (bench) and 1 x 2048 x 128 x 256 (eval frame); seam tail forward: 8 x 2048 x 64 x 128.
// Medians of 7 alternating rounds of 10 launches; every pass moves far more than the 126 MB L2.
#include <algorithm>
#include <cstdarg>
#include <vector>
#include "../../rnd_semantic_segmentation_b200/csrc/seam_tail_kernels.cu"

namespace b200seg {
void set_error(const char* fmt, ...) { va_list a; va_start(a, fmt); vfprintf(stderr, fmt, a); va_end(a); fputc('\n', stderr); }
void count_launch() {}
}  // namespace b200seg
using namespace b200seg;

__global__ void pack_64x64(const float* __restrict__ x, int Cin, int hw, __nv_bfloat16* __restrict__ Xp) {
  __shared__ float tile[64][65];
  const int s0 = blockIdx.x * 64, c0 = blockIdx.y * 64, n = blockIdx.z;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
  const float* src = x + ((long long)n * Cin + c0) * hw + s0;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const int ci = ty + i * 4;
    tile[ci][tx] = (c0 + ci < Cin && s0 + tx < hw) ? __ldcs(src + (long long)ci * hw + tx) : 0.f;
  }
  __syncthreads();
  const int cpair = threadIdx.x & 31, prow = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int s = prow + i * 8;
    if (s0 + s < hw && c0 + 2 * cpair < Cin)
      *reinterpret_cast<__nv_bfloat162*>(Xp + ((long long)n * hw + s0 + s) * Cin + c0 + 2 * cpair) =
          __floats2bfloat162_rn(tile[2 * cpair][s], tile[2 * cpair + 1][s]);
  }
}

__global__ void fill(float* p, long long n, unsigned seed) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n; i += (long long)gridDim.x * 256) {
    unsigned h = (unsigned)i * 2654435761u ^ seed;
    h ^= h >> 13; h *= 0x5bd1e995u; h ^= h >> 15;
    p[i] = (float)(h & 0xffffff) / 8388608.f - 1.f;
  }
}

template <bool TAIL>
static void tile(const float* x, const float* id, const float* sc, const float* bi, int N, int C, int hw, __nv_bfloat16* y) {
  nchw_to_nhwc_tile_kernel<TAIL, true><<<dim3(hw / ST_PX, C / ST_CH, N), ST_THREADS>>>(x, id, sc, bi, C, hw, C, y);
}

int main() {
  const int C = 2048;
  const long long big = 8LL * C * 8192;
  float *x, *id, *sc, *bi;
  __nv_bfloat16* y;
  cudaMalloc(&x, big * 4); cudaMalloc(&id, big * 4); cudaMalloc(&sc, C * 4); cudaMalloc(&bi, C * 4); cudaMalloc(&y, big * 2);
  fill<<<4096, 256>>>(x, big, 1u); fill<<<4096, 256>>>(id, big, 2u); fill<<<8, 256>>>(sc, C, 3u); fill<<<8, 256>>>(bi, C, 4u);
  cudaDeviceProp prop; cudaGetDeviceProperties(&prop, 0);
  printf("device %s\n", prop.name);
  struct V { const char* name; int N, hw; double mb; void (*f)(const float*, const float*, const float*, const float*, int, int, int, __nv_bfloat16*); };
  auto old = [](const float* x, const float*, const float*, const float*, int N, int C, int hw, __nv_bfloat16* y) {
    pack_64x64<<<dim3(hw / 64, C / 64, N), 256>>>(x, C, hw, y);
  };
  std::vector<V> vs;
  for (int shape = 0; shape < 2; ++shape) {
    const int N = shape ? 1 : 8, hw = shape ? 32768 : 8192;
    const double mb = (double)N * C * hw * 6 / 1e6;
    vs.push_back({shape ? "eval  pack 64x64 scalar (old)" : "bench pack 64x64 scalar (old)", N, hw, mb, old});
    vs.push_back({shape ? "eval  pack tile 32x128" : "bench pack tile 32x128", N, hw, mb, tile<false>});
  }
  vs.push_back({"bench tail tile 32x128", 8, 8192, 8.0 * C * 8192 * 10 / 1e6, tile<true>});
  std::vector<std::vector<float>> t(vs.size());
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  for (int round = 0; round < 8; ++round)
    for (size_t k = 0; k < vs.size(); ++k) {
      cudaEventRecord(e0);
      for (int it = 0; it < 10; ++it) vs[k].f(x, id, sc, bi, vs[k].N, C, vs[k].hw, y);
      cudaEventRecord(e1); cudaEventSynchronize(e1);
      float ms; cudaEventElapsedTime(&ms, e0, e1);
      if (round > 0) t[k].push_back(ms / 10);                      // round 0: warm-up
    }
  for (size_t k = 0; k < vs.size(); ++k) {
    std::sort(t[k].begin(), t[k].end());
    const double us = t[k][t[k].size() / 2] * 1e3;
    printf("%-32s %7.1f us  %6.0f MB  %5.2f TB/s  (min %.1f max %.1f)\n", vs[k].name, us, vs[k].mb, vs[k].mb / us,
           t[k].front() * 1e3, t[k].back() * 1e3);
  }
  printf("%s\n", cudaGetErrorString(cudaGetLastError()));
  return 0;
}
