// Parameter-side transforms of the training step as two fused kernels (+ their
// backward), replacing ~250 tiny framework launches per step:
//   W_eff = Q_q(kernel) + kernel_init, b_eff = b + b_init      utils/network.py:606-620, 669-686, 735-740
//   Q_1(k) = k + (U(0,1) - 1/2)/16, Q_2(k) = round(16 k)/16 (straight-through), IConv3d: identity
//   beta_eff = max(beta, bb)^2 - ped, gamma_eff = max(gamma, gb)^2 - ped   gdn_3d.py:143-150 (LowerBound backward :13-29)
//   net_bits[l] = sum_i -log2 max(Phi((r_i - mu + h)/s) - Phi((r_i - mu - h)/s), 1e-8),
//                 r = round(16 k)/16 (straight-through), h = 1/32, s = |sigma|  utils/network.py:287-305, 4777-4778
#pragma once
#include <cuda_runtime.h>
#include "../../include/nvf_b200.h"
#include "nvf_common.h"
#include "nvf_rng.cuh"

namespace nvf {
namespace fast {

// true on every thread of the LAST CTA of the grid to arrive (after its global writes are visible);
// the ticket word is zero on entry and left zero.
__device__ __forceinline__ bool last_cta(unsigned int* ticket) {
  __shared__ unsigned int s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned int t = atomicAdd(ticket, 1u);
    s_last = (t == gridDim.x * gridDim.y - 1) ? 1u : 0u;
    if (s_last) *ticket = 0u;
  }
  __syncthreads();
  if (s_last) __threadfence();
  return s_last != 0u;
}

constexpr int kParamChunk = 1024;   // elements per CTA (256 threads x 4)
constexpr int kNumConv = 9;         // up0 conv0 up1 conv1 up2 conv2 conv2_cls | conv1_cls conv0_cls
constexpr int kNumQuant = 7;

struct ParamJob {
  const float* kernel; const float* init; const float* b; const float* b_init;
  float* w_out; float* b_out;               // forward: effective tensors   | backward: gradient outputs
  const float* g_w; const float* g_b;       // backward: gradients w.r.t. the effective tensors
  int32_t n, nb, chunk0, nchunks, noise0;
  // optional: the packed layouts the conv kernels read (nvf_common.h PackMode), written in the same pass
  float* pk_fwd; float* pk_dg;              // dst[ci][k][co] and dst[co][k (flipped for conv)][ci], or null
  int32_t A, B, K3, convT;                  // source dims: convT (A=Ci,B=Co,K^3) | conv (A=Co,B=Ci,K^3)
};
struct ParamPrepParams {
  ParamJob job[kNumConv];
  const float* igdn_beta; const float* igdn_gamma;     // raw
  float* beta_out; float* gamma_out;                   // forward: effective | backward: gradients
  const float* g_beta; const float* g_gamma;           // backward inputs
  const float* lik_sigma; const float* lik_mu;
  const float* noise;                                  // U(0,1) per quantised element or null
  const float* g_bits;                                 // backward: [7]
  float* partial;                                      // [total_chunks][3]: bits | d sigma_abs | d mu
  float* net_bits;                                     // forward final: [7]
  float* g_sigma; float* g_mu;                         // backward final
  float beta_bound, gamma_bound, pedestal;
  int32_t q, c0, total_chunks;
  // fused-step extras: in-kernel noise (noise == null, rng_ctr != null), finalisation by the last CTA (ticket != null)
  unsigned long long seed; const unsigned long long* rng_ctr;
  unsigned int* ticket;
};

// net_bits (forward) / d sigma, d mu (backward) from the per-chunk partials, in chunk order (deterministic)
template <bool BWD>
__device__ __forceinline__ void param_finalise(const ParamPrepParams& p, int l) {
  if (!BWD) {
    if (l < kNumQuant) {
      float s = 0.f;
      for (int c = 0; c < p.job[l].nchunks; ++c) s += p.partial[(p.job[l].chunk0 + c) * 3];
      p.net_bits[l] = s;
    }
  } else if (l < 2) {
    float s = 0.f;
    for (int j = 0; j < kNumQuant; ++j)
      for (int c = 0; c < p.job[j].nchunks; ++c) s += p.partial[(p.job[j].chunk0 + c) * 3 + 1 + l];
    if (l == 0) p.g_sigma[0] = p.lik_sigma[0] > 0.f ? s : (p.lik_sigma[0] < 0.f ? -s : 0.f);
    else p.g_mu[0] = s;
  }
}

__device__ __forceinline__ float phi_cdf(float x) { return 0.5f * (1.f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float phi_pdf(float x) { return 0.39894228040143267794f * expf(-0.5f * x * x); }

// fixed-order CTA sum (256 threads); result valid on thread 0
__device__ __forceinline__ float cta_sum_256(float v, float* sm) {
  for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  float s = 0.f;
  if (threadIdx.x == 0)
    for (int i = 0; i < 8; ++i) s += sm[i];
  __syncthreads();
  return s;
}

template <bool BWD>
__global__ void __launch_bounds__(256) k_param_prep(ParamPrepParams p) {
  __shared__ float sm[8];
  const int tid = threadIdx.x;
  if ((int)blockIdx.x == p.total_chunks) {
    // ---- biases and the IGDN reparametrisation (one CTA)
    for (int l = 0; l < kNumConv; ++l) {
      const ParamJob& J = p.job[l];
      for (int i = tid; i < J.nb; i += 256) J.b_out[i] = BWD ? J.g_b[i] : J.b[i] + J.b_init[i];
    }
    const int c0 = p.c0;
    for (int i = tid; i < c0 + c0 * c0; i += 256) {
      const bool isb = i < c0;
      const float raw = isb ? p.igdn_beta[i] : p.igdn_gamma[i - c0];
      const float bound = isb ? p.beta_bound : p.gamma_bound;
      const float lb = fmaxf(raw, bound);
      float* out = isb ? p.beta_out + i : p.gamma_out + (i - c0);
      if (!BWD) {
        *out = lb * lb - p.pedestal;
      } else {
        const float g = (isb ? p.g_beta[i] : p.g_gamma[i - c0]) * 2.f * lb;
        *out = (raw >= bound || g < 0.f) ? g : 0.f;
      }
    }
    if (p.ticket && last_cta(p.ticket)) param_finalise<BWD>(p, tid);
    return;
  }
  int l = 0;
#pragma unroll
  for (int i = 1; i < kNumConv; ++i)
    if ((int)blockIdx.x >= p.job[i].chunk0) l = i;
  const ParamJob& J = p.job[l];
  const bool quant = l < kNumQuant;
  const float sigma = fabsf(p.lik_sigma[0]), mu = p.lik_mu[0];
  const float h = 1.f / 32.f;
  const float gbit = (BWD && quant) ? p.g_bits[l] : 0.f;
  const int base = ((int)blockIdx.x - J.chunk0) * kParamChunk;
  float s_bits = 0.f, s_dsig = 0.f, s_dmu = 0.f;
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const int i = base + k * 256 + tid;
    if (i >= J.n) continue;
    const float kv = J.kernel[i];
    const float r = rintf(kv * 16.f) / 16.f;
    if (!BWD) {
      float kq = kv;
      if (quant && p.q == 1) {
        const float u01 = p.noise ? p.noise[J.noise0 + i]
                                  : rng::uniform(p.seed, p.rng_ctr[0], rng::kKernelNoise, (uint64_t)(J.noise0 + i));
        kq = kv + (u01 - 0.5f) * (1.f / 16.f);
      } else if (quant && p.q == 2) {
        kq = r;
      }
      const float we = kq + J.init[i];
      J.w_out[i] = we;
      if (J.pk_fwd) {
        // source index i = (a * B + b) * K3 + k
        const int k = i % J.K3, ab = i / J.K3, bb = ab % J.B, aa = ab / J.B;
        const int ci = J.convT ? aa : bb, co = J.convT ? bb : aa, Ci = J.convT ? J.A : J.B, Co = J.convT ? J.B : J.A;
        J.pk_fwd[(ci * J.K3 + k) * Co + co] = we;
        if (J.pk_dg) J.pk_dg[(co * J.K3 + (J.convT ? k : J.K3 - 1 - k)) * Ci + ci] = we;
      }
      if (quant) {
        const float u = (r - mu + h) / sigma, lo = (r - mu - h) / sigma;
        const float L = fmaxf(phi_cdf(u) - phi_cdf(lo), 1e-8f);
        s_bits += -1.f * logf(L) / 0.69314718055994530942f;
      }
    } else {
      float g = J.g_w[i];
      if (quant) {
        const float u = (r - mu + h) / sigma, lo = (r - mu - h) / sigma;
        const float Lraw = phi_cdf(u) - phi_cdf(lo);
        const float Lc = fmaxf(Lraw, 1e-8f);
        const float gL = -gbit / (Lc * 0.69314718055994530942f);
        if (Lraw >= 1e-8f || gL < 0.f) {
          const float pu = phi_pdf(u), pl = phi_pdf(lo);
          g += gL * (pu - pl) / sigma;
          s_dmu += -gL * (pu - pl) / sigma;
          s_dsig += -gL * (u * pu - lo * pl) / sigma;
        }
      }
      J.w_out[i] = g;
    }
  }
  if (quant) {
    if (!BWD) {
      const float t = cta_sum_256(s_bits, sm);
      if (tid == 0) p.partial[blockIdx.x * 3] = t;
    } else {
      const float a = cta_sum_256(s_dsig, sm);
      const float b = cta_sum_256(s_dmu, sm);
      if (tid == 0) { p.partial[blockIdx.x * 3 + 1] = a; p.partial[blockIdx.x * 3 + 2] = b; }
    }
  }
  if (p.ticket && last_cta(p.ticket)) param_finalise<BWD>(p, tid);
}

template <bool BWD>
__global__ void __launch_bounds__(32) k_param_final(ParamPrepParams p) {
  param_finalise<BWD>(p, (int)threadIdx.x);
}

}  // namespace fast
}  // namespace nvf
