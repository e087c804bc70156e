// Shared-weight gradient all-reduce FUSED with the Adam update, over NVLink / NVSwitch peer memory
// (NVFPCC.py:154,161,222 under data parallelism: every rank must apply the SUM of the ranks' weight gradients).
//
// The gradient is 52 219 / 200 915 floats, so the collective is latency-, not bandwidth-bound: a ring or tree over 8
// GPUs is a chain of dependent hops plus two more launches (partial reduction, Adam).  Here every rank owns one
// "symmetric" buffer (cudaMalloc + CUDA IPC, mapped by all peers of the node):
//     [64 x uint32 flags][gradient copy 0][gradient copy 1]
// and ONE kernel per step does, on every rank:
//   1. copy the rank's flat gradient into its own copy (seq & 1);
//   2. when the last CTA has finished copying: store.release.sys `seq` into flag[rank] of EVERY peer's buffer;
//   3. wait until all flags of the own buffer have reached `seq` (volatile polls + one acquire fence): every peer's
//      copy is complete;
//   4. read all W copies over NVLink (volatile 128-bit loads, 7 x 0.2 MB per rank), add them in rank order
//      0..W-1 - the same order on every rank, so the weights stay bit-identical across ranks - and apply Adam to
//      the rank's replica of the weights in the same pass.
// Two gradient copies alternate by step parity: a rank can only reach step s+1's copy phase after all peers have
// published step s (they had then finished reading step s-1), so no second barrier is needed.
// The step sequence number and the two tickets live in a small device-resident control block: graph replay safe.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "nvf_common.h"
#include "nvf_fast_latent.cuh"   // adam_update

namespace nvf {
namespace fast {

constexpr int kSymmMaxRanks = 16;
constexpr int kSymmHeaderBytes = 256;   // 64 flags

struct ArAdamParams {
  float* param; const float* grad; float* m; float* v;
  float* step; const float* lr;
  float beta1, beta2, eps;
  int32_t n;          // parameters
  int32_t n4;         // float4 per gradient copy (>= ceil(n / 4))
  int32_t rank, world;
  unsigned int* ctl;  // [0] last completed sequence number, [1] copy ticket, [2] done ticket
  char* peer[kSymmMaxRanks];   // every rank's symmetric buffer as mapped in THIS process (peer[rank] = own)
};

__device__ __forceinline__ void st_release_sys(unsigned int* p, unsigned int v) {
  asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ unsigned int ld_acquire_sys(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
__device__ __forceinline__ float4 ld_volatile_f4(const float4* p) {
  float4 v;
  asm volatile("ld.volatile.global.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "l"(p) : "memory");
  return v;
}

// grid <= 64 CTAs (all resident: the last CTA to finish its copy publishes for the whole grid)
__global__ void __launch_bounds__(256) k_allreduce_adam(ArAdamParams p) {
  const int tid = threadIdx.x;
  const unsigned int seq = *(volatile unsigned int*)p.ctl + 1u;
  const size_t boff = (size_t)(seq & 1u) * p.n4;
  __shared__ unsigned int s_last;
  float step_size, bc2s;            // evaluated (one thread) while the copies are in flight
  adam_bias_corrections(p.step, p.lr, p.beta1, p.beta2, step_size, bc2s);
  // 1. own gradient -> own symmetric copy (tail of the last float4 zero-filled)
  {
    float4* own = reinterpret_cast<float4*>(p.peer[p.rank] + kSymmHeaderBytes) + boff;
    for (int i = blockIdx.x * 256 + tid; i < p.n4; i += gridDim.x * 256) {
      float4 g = make_float4(0.f, 0.f, 0.f, 0.f);
      if (4 * i + 3 < p.n) {
        g = *reinterpret_cast<const float4*>(p.grad + 4 * i);
      } else {
        if (4 * i < p.n) g.x = p.grad[4 * i];
        if (4 * i + 1 < p.n) g.y = p.grad[4 * i + 1];
        if (4 * i + 2 < p.n) g.z = p.grad[4 * i + 2];
      }
      own[i] = g;
    }
  }
  __threadfence();
  __syncthreads();
  if (tid == 0) s_last = atomicAdd(&p.ctl[1], 1u) == gridDim.x - 1 ? 1u : 0u;
  __syncthreads();
  // 2. the last CTA publishes: flag[rank] = seq in every rank's buffer (own included)
  if (s_last) {
    if (tid < p.world) {
      __threadfence_system();
      st_release_sys(reinterpret_cast<unsigned int*>(p.peer[tid]) + p.rank, seq);
    }
    if (tid == 0) p.ctl[1] = 0u;
  }
  // 3. all peers have published this step
  // (the flags live in THIS rank's memory, so polling reads the local L2 - a relaxed volatile load per poll, one
  // system-scope acquire fence once the flag is there, instead of an acquire at system scope per poll)
  if (tid < p.world) {
    const volatile unsigned int* f = reinterpret_cast<const volatile unsigned int*>(p.peer[p.rank]) + tid;
    while ((int)(*f - seq) < 0) {
    }
    __threadfence_system();
  }
  __syncthreads();
  // 4. sum in rank order + Adam (same arithmetic as k_adam)
  for (int i = blockIdx.x * 256 + tid; i < p.n4; i += gridDim.x * 256) {
    float4 g = ld_volatile_f4(reinterpret_cast<const float4*>(p.peer[0] + kSymmHeaderBytes) + boff + i);
    for (int r = 1; r < p.world; ++r) {
      const float4 q = ld_volatile_f4(reinterpret_cast<const float4*>(p.peer[r] + kSymmHeaderBytes) + boff + i);
      g.x += q.x; g.y += q.y; g.z += q.z; g.w += q.w;
    }
    const float gv[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int e = 4 * i + j;
      if (e >= p.n) break;
      float m = p.m[e], v = p.v[e], w = p.param[e];
      adam_update(w, m, v, gv[j], p.beta1, p.beta2, p.eps, step_size, bc2s);
      p.m[e] = m; p.v[e] = v;
      p.param[e] = w;
    }
  }
  // 5. the last CTA to finish advances the sequence number and Adam's step counter
  __syncthreads();
  if (tid == 0 && atomicAdd(&p.ctl[2], 1u) == gridDim.x - 1) {
    p.ctl[2] = 0u;
    p.step[0] += 1.f;
    __threadfence();
    *(volatile unsigned int*)p.ctl = seq;
  }
}

}  // namespace fast
}  // namespace nvf
