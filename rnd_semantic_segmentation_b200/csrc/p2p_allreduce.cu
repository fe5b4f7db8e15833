// Mean all-reduce of a flat fp32 gradient bucket over NVLink / NVSwitch peer memory, as ONE small kernel per rank.
//
// Replaces the collective of DistributedDataParallel in train_distill.py:54-62 (mean of the per-rank gradients; the reference's
// train_adv.py shards the data but never synchronises, SURVEY.md section 2a) for the head's 5.6 MB and the discriminator's
// 20.2 MB buckets.  The bucket lives in symmetric memory (every rank maps every peer's buffer; torch's symmetric-memory
// rendezvous hands over the peer / multicast / signal-pad addresses -- plumbing only), and every rank runs this kernel:
//
//   1. cross-rank barrier per CTA through the signal pads (release / acquire at system scope): all ranks' gradients are written;
//   2. two-shot all-reduce in one pass: rank r owns slice r of the bucket.
//        NVSwitch multicast address available (NVLS):  v = multimem.ld_reduce.add(slice element)   -- summed IN THE SWITCH
//                                                     multimem.st(slice element, v / world)         -- broadcast by the switch
//        otherwise (plain P2P):                        v = sum over peers of peer[p][i];  store v / world into every peer's buffer
//      Nobody but rank r reads or writes slice r between the two barriers, so there is no hazard;
//   3. cross-rank barrier: every rank's stores have landed everywhere before anyone's next kernel reads the bucket.
//
// A ring all-reduce moves 2 (W-1)/W of the bucket through every link in 2 (W-1) latency-bound steps and wants 16-32 CTAs to do
// it inside the ~180 us data-gradient window (NCCL, measured: 178 / 104 / 57 us at 8 / 16 / 32 CTAs for 5.6 MB on 8 ranks).
// Here every byte crosses the switch once per direction in ONE step: a handful of CTAs suffice, so the persistent data-gradient
// GEMM cedes 4 SMs instead of 32.
#include "common.cuh"
#include "host_api.h"

namespace b200seg {

constexpr int P2P_MAX_WORLD = 16;
constexpr int P2P_THREADS = 512;

struct P2PParams {
  float* peer[P2P_MAX_WORLD];           // every rank's bucket (index = rank), mapped into this process
  unsigned* pad[P2P_MAX_WORLD];         // every rank's signal pad
  float* mc;                            // multicast address of the bucket (NVLS) or null
  int rank, world;
  long long n4;                         // bucket length in float4 (the buffer is padded to a multiple of 4 floats)
  float scale;                          // 1 / world
};

// put: flip the flag the peer waits on from 0 to 1 (spin while a previous signal is still unconsumed); wait: consume own flag.
// A peer that never arrives (crashed rank, mismatched call sequence) must not hang the GPU: after P2P_TIMEOUT_NS of spinning the
// kernel traps, which surfaces as a CUDA error on the host instead of a stuck device.
constexpr unsigned long long P2P_TIMEOUT_NS = 20ull * 1000ull * 1000ull * 1000ull;
__device__ __forceinline__ unsigned long long p2p_now_ns() {
  unsigned long long t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
__device__ __forceinline__ void p2p_put(unsigned* addr) {
  unsigned old;
  unsigned long long t0 = 0;
  unsigned spins = 0;
  do {
    asm volatile("atom.release.sys.global.cas.b32 %0, [%1], 0, 1;" : "=r"(old) : "l"(addr) : "memory");
    if (old != 0u && (++spins & 1023u) == 0u) {
      const unsigned long long t = p2p_now_ns();
      if (t0 == 0) t0 = t;
      else if (t - t0 > P2P_TIMEOUT_NS) __trap();
    }
  } while (old != 0u);
}
__device__ __forceinline__ void p2p_wait(unsigned* addr) {
  unsigned old;
  unsigned long long t0 = 0;
  unsigned spins = 0;
  do {
    asm volatile("atom.acquire.sys.global.cas.b32 %0, [%1], 1, 0;" : "=r"(old) : "l"(addr) : "memory");
    if (old != 1u && (++spins & 1023u) == 0u) {
      const unsigned long long t = p2p_now_ns();
      if (t0 == 0) t0 = t;
      else if (t - t0 > P2P_TIMEOUT_NS) __trap();
    }
  } while (old != 1u);
}
// every CTA b of every rank meets CTA b of every other rank
__device__ __forceinline__ void p2p_barrier(const P2PParams& p, int slot) {
  __syncthreads();
  if ((int)threadIdx.x < p.world && (int)threadIdx.x != p.rank) {
    const int peer = threadIdx.x;
    p2p_put(p.pad[peer] + (slot * p.world + p.rank));          // "rank is here" into the peer's pad
    p2p_wait(p.pad[p.rank] + (slot * p.world + peer));         // the peer is here too
  }
  __syncthreads();
}

__global__ void __launch_bounds__(P2P_THREADS) p2p_allreduce_mean_kernel(const __grid_constant__ P2PParams p, int pad_slot0) {
  const int slot = pad_slot0 + blockIdx.x;
  p2p_barrier(p, slot);
  // slice of this rank, then of this CTA
  const long long per = (p.n4 + p.world - 1) / p.world;
  const long long lo = per * p.rank, hi = min(p.n4, lo + per);
  const long long stride = (long long)gridDim.x * P2P_THREADS;
  // P2P_U elements per thread in flight: a trip through the switch is microseconds, so memory-level parallelism is what
  // gives a handful of CTAs their bandwidth
  constexpr int P2P_U = 8;
  const long long first = lo + (long long)blockIdx.x * P2P_THREADS + threadIdx.x;
  if (p.mc != nullptr) {
    for (long long i0 = first; i0 < hi; i0 += stride * P2P_U) {
      float4 v[P2P_U];
#pragma unroll
      for (int u = 0; u < P2P_U; ++u) {
        const long long i = i0 + u * stride;
        if (i < hi)
          asm volatile("multimem.ld_reduce.relaxed.sys.global.add.v4.f32 {%0, %1, %2, %3}, [%4];"
                       : "=f"(v[u].x), "=f"(v[u].y), "=f"(v[u].z), "=f"(v[u].w)
                       : "l"(p.mc + 4 * i)
                       : "memory");
      }
#pragma unroll
      for (int u = 0; u < P2P_U; ++u) {
        const long long i = i0 + u * stride;
        if (i < hi)
          asm volatile("multimem.st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p.mc + 4 * i), "f"(v[u].x * p.scale),
                       "f"(v[u].y * p.scale), "f"(v[u].z * p.scale), "f"(v[u].w * p.scale)
                       : "memory");
      }
    }
  } else {
    for (long long i0 = first; i0 < hi; i0 += stride * P2P_U) {
      float4 acc[P2P_U];
#pragma unroll
      for (int u = 0; u < P2P_U; ++u) acc[u] = make_float4(0.f, 0.f, 0.f, 0.f);
      for (int q = 0; q < p.world; ++q) {                       // fixed order: the result does not depend on which rank owns the slice
#pragma unroll
        for (int u = 0; u < P2P_U; ++u) {
          const long long i = i0 + u * stride;
          if (i < hi) {
            float4 v;
            asm volatile("ld.relaxed.sys.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p.peer[q] + 4 * i) : "memory");
            acc[u].x += v.x; acc[u].y += v.y; acc[u].z += v.z; acc[u].w += v.w;
          }
        }
      }
      for (int q = 0; q < p.world; ++q) {
#pragma unroll
        for (int u = 0; u < P2P_U; ++u) {
          const long long i = i0 + u * stride;
          if (i < hi)
            asm volatile("st.relaxed.sys.global.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p.peer[q] + 4 * i), "f"(acc[u].x * p.scale),
                         "f"(acc[u].y * p.scale), "f"(acc[u].z * p.scale), "f"(acc[u].w * p.scale)
                         : "memory");
        }
      }
    }
  }
  __threadfence_system();
  p2p_barrier(p, slot);
}

int p2p_allreduce_mean(void* const* peer_bufs, void* multicast_ptr, void* const* signal_pads, int rank, int world, long long numel,
                       int blocks, int pad_slot0, cudaStream_t stream) {
  B200SEG_CHECK_ARG(peer_bufs && signal_pads, "p2p_allreduce_mean: null pointer table");
  B200SEG_CHECK_ARG(world >= 1 && world <= P2P_MAX_WORLD && rank >= 0 && rank < world, "p2p_allreduce_mean: bad rank %d / world %d", rank, world);
  B200SEG_CHECK_ARG(numel > 0 && numel % 4 == 0, "p2p_allreduce_mean: the bucket length must be a positive multiple of 4 floats (%lld)", numel);
  B200SEG_CHECK_ARG(blocks >= 1 && blocks <= 64 && pad_slot0 >= 0 && (pad_slot0 + blocks) * world * 4 <= 8192,
                    "p2p_allreduce_mean: %d CTAs from pad slot %d do not fit the signal pad", blocks, pad_slot0);
  if (world == 1) return B200SEG_OK;
  P2PParams p = {};
  for (int q = 0; q < world; ++q) {
    B200SEG_CHECK_ARG(peer_bufs[q] && signal_pads[q], "p2p_allreduce_mean: null peer pointer (rank %d)", q);
    p.peer[q] = reinterpret_cast<float*>(peer_bufs[q]);
    p.pad[q] = reinterpret_cast<unsigned*>(signal_pads[q]);
  }
  p.mc = reinterpret_cast<float*>(multicast_ptr);
  p.rank = rank; p.world = world; p.n4 = numel / 4; p.scale = 1.0f / (float)world;
  p2p_allreduce_mean_kernel<<<blocks, P2P_THREADS, 0, stream>>>(p, pad_slot0);
  B200SEG_LAUNCH_CHECK();
  return B200SEG_OK;
}

}  // namespace b200seg
