// Latent head of the NVF codec as ONE fused kernel per direction, plus the two other
// scalar-sized pieces of a training step (total loss, Adam), replacing ~200 tiny
// framework launches per step:
//
//   latent head  (SingleLayerLatentGen + QuantGaussianLikelihood, utils/network.py:4592-4612, 4490-4545)
//     h = W e + b               W = kernel + kernel_init (IConv3d, 1x1x1, :735-741), b = b + b_init
//     y_i = h_i / sqrt(beta_i + sum_j gamma_ij h_j^2)              GDN3d, gdn_3d.py:78-92
//     r = round(y)  (straight-through, :4519)                       -> decoder input
//     xt = y + (U - 1/2) * noise_scale (train) | r (eval)           :4516-4525
//     bits = sum -log2 max(Phi((xt-mu+1/2)/s) - Phi((xt-mu-1/2)/s), 1e-8),  s = |sigma|   :139-169
//   total loss   NVFPCC.py:161-164,196   loss = bce + ms0 + ms1 + lambda (w1 bits_latent/n_pts + w2 sum(net_bits)/N)
//   Adam         NVFPCC.py:116,222       torch.optim.Adam defaults (no weight decay, no amsgrad)
//
// One thread owns one latent position (block, voxel of the 2x2x2 grid) with all CH channels in
// registers.  Scalar results and parameter gradients are reduced CTA-wise in fixed order into
// per-CTA partials; the last CTA to finish (global ticket) folds the partials in CTA order, so
// results are deterministic without a second launch.
#pragma once
#include <cuda_runtime.h>
#include "../../include/nvf_b200.h"
#include "nvf_common.h"
#include "nvf_fast_params.cuh"

namespace nvf {
namespace fast {

constexpr int kLatentThreads = 128;
constexpr int kLatentMaxCtas = 256;

struct LatentKParams {
  const float* emb; const float* noise;             // [n][CH][8]; noise U(0,1) or null
  const float* kernel; const float* kernel_init; const float* b; const float* b_init;
  const float* beta; const float* gamma; const float* sigma; const float* mu;
  float beta_bound, gamma_bound, pedestal, noise_scale;
  int32_t n, train;
  // forward
  float* latent; float* bits_out;
  // backward
  const float* g_latent; const float* g_bits;
  float* g_emb;                                     // or null
  float *gk, *gb, *gbeta, *ggamma, *gsigma, *gmu;   // all null when parameter gradients are not wanted
  // scratch
  double* partial;                                  // [gridDim][NP]
  unsigned int* ticket;                             // zero on entry, zero on exit
  // fused-step extras (all optional): block b reads embedding row idx[b] of a resident dataset with n_rows rows
  // (out-of-range rows are clamped to 0 and reported by the caller's gather status); noise == null && rng_ctr:
  // in-kernel Philox noise; g_bits_scale != null: g_bits[0] is multiplied by it (lambda * w1, the caller passes 1/n_pts)
  const long long* idx; long long n_rows;
  unsigned long long seed; const unsigned long long* rng_ctr;
};

template <int CH>
struct LatentCfg {
  // partial layout (backward): dW[CH*CH] db[CH] dbeta_eff[CH] dgamma_eff[CH*CH] dsigma_abs[CH] dmu[CH]
  static constexpr int NP_BWD = 2 * CH * CH + 4 * CH;
};

// fixed-order CTA sum over kLatentThreads threads (double); result valid on thread 0
__device__ __forceinline__ double cta_sum_d(double v, double* sm) {
  for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
  if (threadIdx.x == 0)
    for (int i = 0; i < kLatentThreads / 32; ++i) s += sm[i];
  __syncthreads();
  return s;
}

template <int CH>
struct LatentPoint {
  float e[CH], h[CH], nrm[CH], y[CH], r[CH], xt[CH];
  bool valid;
};

template <int CH>
__device__ __forceinline__ void latent_point(const LatentKParams& p, const float (&W)[CH][CH], const float (&bias)[CH],
                                             const float (&beta)[CH], const float (&gamma)[CH][CH], int pos,
                                             LatentPoint<CH>& q) {
  q.valid = pos < p.n * 8;
  const int blk = q.valid ? pos >> 3 : 0, s = pos & 7;
  const size_t base = (size_t)blk * CH * 8 + s;
  size_t ebase = base;
  if (p.idx) {
    long long row = p.idx[blk];
    if (row < 0 || row >= p.n_rows) row = 0;
    ebase = (size_t)row * CH * 8 + s;
  }
#pragma unroll
  for (int j = 0; j < CH; ++j) q.e[j] = q.valid ? p.emb[ebase + j * 8] : 0.f;
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    float v = bias[i];
#pragma unroll
    for (int j = 0; j < CH; ++j) v = fmaf(W[i][j], q.e[j], v);
    q.h[i] = v;
  }
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    float v = beta[i];
#pragma unroll
    for (int j = 0; j < CH; ++j) v = fmaf(gamma[i][j], q.h[j] * q.h[j], v);
    q.nrm[i] = sqrtf(v);
    q.y[i] = q.h[i] / q.nrm[i];
    q.r[i] = rintf(q.y[i]);
    float nz = 0.f;
    if (p.noise && q.valid) nz = (p.noise[base + i * 8] - 0.5f) * p.noise_scale;
    else if (p.rng_ctr && q.valid && p.train)
      nz = (rng::uniform(p.seed, p.rng_ctr[0], rng::kLatentNoise, (uint64_t)(base + i * 8)) - 0.5f) * p.noise_scale;
    q.xt[i] = p.train ? q.y[i] + nz : q.r[i];
  }
}

template <int CH>
__device__ __forceinline__ void latent_load_params(const LatentKParams& p, float (&W)[CH][CH], float (&bias)[CH],
                                                   float (&beta)[CH], float (&gamma)[CH][CH]) {
#pragma unroll
  for (int i = 0; i < CH; ++i) {
    bias[i] = p.b[i] + p.b_init[i];
    const float lb = fmaxf(p.beta[i], p.beta_bound);
    beta[i] = lb * lb - p.pedestal;
#pragma unroll
    for (int j = 0; j < CH; ++j) {
      W[i][j] = p.kernel[i * CH + j] + p.kernel_init[i * CH + j];
      const float lg = fmaxf(p.gamma[i * CH + j], p.gamma_bound);
      gamma[i][j] = lg * lg - p.pedestal;
    }
  }
}

template <int CH>
__global__ void __launch_bounds__(kLatentThreads) k_latent_fwd(LatentKParams p) {
  __shared__ double sm[kLatentThreads / 32];
  float W[CH][CH], bias[CH], beta[CH], gamma[CH][CH];
  latent_load_params<CH>(p, W, bias, beta, gamma);
  double bits = 0.0;
  for (int pos = blockIdx.x * kLatentThreads + threadIdx.x; pos < p.n * 8; pos += gridDim.x * kLatentThreads) {
    LatentPoint<CH> q;
    latent_point<CH>(p, W, bias, beta, gamma, pos, q);
    const size_t base = (size_t)(pos >> 3) * CH * 8 + (pos & 7);
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      p.latent[base + i * 8] = q.r[i];
      const float s = fabsf(p.sigma[i]), m = p.mu[i];
      const float u = (q.xt[i] - m + 0.5f) / s, lo = (q.xt[i] - m - 0.5f) / s;
      const float L = fmaxf(phi_cdf(u) - phi_cdf(lo), 1e-8f);
      bits += (double)(-1.f * logf(L) / 0.69314718055994530942f);
    }
  }
  const double t = cta_sum_d(bits, sm);
  if (threadIdx.x == 0) p.partial[blockIdx.x] = t;
  if (last_cta(p.ticket) && threadIdx.x == 0) {
    double s = 0.0;
    for (unsigned int c = 0; c < gridDim.x; ++c) s += p.partial[c];
    p.bits_out[0] = (float)s;
  }
}

template <int CH>
__global__ void __launch_bounds__(kLatentThreads) k_latent_bwd(LatentKParams p) {
  constexpr int NP = LatentCfg<CH>::NP_BWD;
  float W[CH][CH], bias[CH], beta[CH], gamma[CH][CH];
  latent_load_params<CH>(p, W, bias, beta, gamma);
  const bool want_params = p.gk != nullptr;
  const float gbits = p.g_bits[0];
  float acc[NP];
#pragma unroll
  for (int i = 0; i < NP; ++i) acc[i] = 0.f;
  for (int pos = blockIdx.x * kLatentThreads + threadIdx.x; pos < p.n * 8; pos += gridDim.x * kLatentThreads) {
    LatentPoint<CH> q;
    latent_point<CH>(p, W, bias, beta, gamma, pos, q);
    const size_t base = (size_t)(pos >> 3) * CH * 8 + (pos & 7);
    float gy[CH];
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      // rate term (GaussianModel + LowerBound, utils/network.py:145-161)
      const float sraw = p.sigma[i], s = fabsf(sraw), m = p.mu[i];
      const float u = (q.xt[i] - m + 0.5f) / s, lo = (q.xt[i] - m - 0.5f) / s;
      const float Lraw = phi_cdf(u) - phi_cdf(lo);
      const float Lc = fmaxf(Lraw, 1e-8f);
      const float gL = -gbits / (Lc * 0.69314718055994530942f);
      float gx = 0.f;
      if (Lraw >= 1e-8f || gL < 0.f) {
        const float pu = phi_pdf(u), pl = phi_pdf(lo);
        gx = gL * (pu - pl) / s;
        acc[2 * CH * CH + 2 * CH + CH + i] += -gx;                         // d mu
        acc[2 * CH * CH + 2 * CH + i] += -gL * (u * pu - lo * pl) / s;     // d |sigma|
      }
      gy[i] = (p.g_latent ? p.g_latent[base + i * 8] : 0.f) + gx;         // round and +noise are identity in backward
    }
    // GDN backward: y_i = h_i / n_i
    float t[CH], gh[CH];
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      const float inv = 1.f / q.nrm[i];
      t[i] = gy[i] * q.h[i] * inv * inv * inv;                              // g_i h_i / n_i^3
      acc[CH * CH + CH + i] += -0.5f * t[i];                                // d beta_eff
#pragma unroll
      for (int j = 0; j < CH; ++j) acc[CH * CH + 2 * CH + i * CH + j] += -0.5f * t[i] * q.h[j] * q.h[j];  // d gamma_eff
    }
#pragma unroll
    for (int k = 0; k < CH; ++k) {
      float v = gy[k] / q.nrm[k];
#pragma unroll
      for (int i = 0; i < CH; ++i) v -= q.h[k] * t[i] * gamma[i][k];
      gh[k] = v;
    }
    // 1x1x1 conv backward
#pragma unroll
    for (int i = 0; i < CH; ++i) {
      acc[CH * CH + i] += gh[i];
#pragma unroll
      for (int j = 0; j < CH; ++j) acc[i * CH + j] += gh[i] * q.e[j];
    }
    if (p.g_emb) {
#pragma unroll
      for (int j = 0; j < CH; ++j) {
        float v = 0.f;
#pragma unroll
        for (int i = 0; i < CH; ++i) v = fmaf(W[i][j], gh[i], v);
        p.g_emb[base + j * 8] = v;
      }
    }
  }
  if (!want_params) return;
  {
    // fixed-order CTA sums of the NP partial gradients: warp shuffles, then one pass over the warps
    __shared__ double smp[NP][kLatentThreads / 32];
#pragma unroll
    for (int i = 0; i < NP; ++i) {
      double v = (double)acc[i];
      for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      if ((threadIdx.x & 31) == 0) smp[i][threadIdx.x >> 5] = v;
    }
    __syncthreads();
    if (threadIdx.x < NP) {
      double s = 0.0;
      for (int w = 0; w < kLatentThreads / 32; ++w) s += smp[threadIdx.x][w];
      p.partial[(size_t)blockIdx.x * NP + threadIdx.x] = s;
    }
  }
  if (!last_cta(p.ticket)) return;
  for (int i = threadIdx.x; i < NP; i += kLatentThreads) {
    double s = 0.0;
    for (unsigned int c = 0; c < gridDim.x; ++c) s += p.partial[(size_t)c * NP + i];
    const float v = (float)s;
    if (i < CH * CH) {
      p.gk[i] = v;
    } else if (i < CH * CH + CH) {
      p.gb[i - CH * CH] = v;
    } else if (i < CH * CH + 2 * CH) {             // beta: through max(beta, bound)^2 - pedestal (LowerBound, gdn_3d.py:13-29)
      const int k = i - (CH * CH + CH);
      const float raw = p.beta[k], g = v * 2.f * fmaxf(raw, p.beta_bound);
      p.gbeta[k] = (raw >= p.beta_bound || g < 0.f) ? g : 0.f;
    } else if (i < 2 * CH * CH + 2 * CH) {
      const int k = i - (CH * CH + 2 * CH);
      const float raw = p.gamma[k], g = v * 2.f * fmaxf(raw, p.gamma_bound);
      p.ggamma[k] = (raw >= p.gamma_bound || g < 0.f) ? g : 0.f;
    } else if (i < 2 * CH * CH + 3 * CH) {         // sigma: through abs()
      const int k = i - (2 * CH * CH + 2 * CH);
      const float raw = p.sigma[k];
      p.gsigma[k] = raw > 0.f ? v : (raw < 0.f ? -v : 0.f);
    } else {
      p.gmu[i - (2 * CH * CH + 3 * CH)] = v;
    }
  }
}

// ---------------------------------------------------------------------------
// total loss + logged scalars, forward and backward (one thread each)
// stats: loss bce ms0 ms1 b_latent b_net n_pts   (trainer.STAT_NAMES)
// ---------------------------------------------------------------------------
struct RdTotalParams {
  const double* sums;        // nvf_loss_seeds sums: [0] bce [1] ms0 [2] ms1
  const float* latent_bits;  // [1]
  const float* net_bits;     // [7]
  const float* n_pts;        // [1] batch-global number of occupied voxels
  float n_total, lmbda, w1, w2;
  float* loss;               // [1]
  float* stats;              // [7] or null
  // backward
  const float* g_loss;       // [1]
  float* g_dist;             // [3] gradients w.r.t. bce, ms0, ms1
  float* g_latent_bits;      // [1]
  float* g_net_bits;         // [7]
};

template <bool BWD>
__global__ void k_rd_total(RdTotalParams p) {
  if (threadIdx.x != 0 || blockIdx.x != 0) return;
  if (!BWD) {
    const float bce = (float)p.sums[0], ms0 = (float)p.sums[1], ms1 = (float)p.sums[2];
    const float npts = p.n_pts[0];
    float nb = 0.f;
    for (int i = 0; i < kNumQuant; ++i) nb += p.net_bits[i];
    const float b_latent = p.latent_bits[0] / npts;
    const float b_net = nb / p.n_total;
    const float loss = bce + ms0 + ms1 + p.lmbda * (b_latent * p.w1 + b_net * p.w2);
    p.loss[0] = loss;
    if (p.stats) {
      p.stats[0] = loss; p.stats[1] = bce; p.stats[2] = ms0; p.stats[3] = ms1;
      p.stats[4] = b_latent; p.stats[5] = b_net; p.stats[6] = npts;
    }
  } else {
    const float g = p.g_loss[0];
    p.g_dist[0] = g; p.g_dist[1] = g; p.g_dist[2] = g;
    p.g_latent_bits[0] = g * p.lmbda * p.w1 / p.n_pts[0];
    const float gn = g * p.lmbda * p.w2 / p.n_total;
    for (int i = 0; i < kNumQuant; ++i) p.g_net_bits[i] = gn;
  }
}

// ---------------------------------------------------------------------------
// Adam over one flat parameter buffer (torch.optim.Adam, default hyper-parameters):
//   m = m + (1-b1)(g - m); v = b2 v + (1-b2) g^2;
//   p -= lr / (1 - b1^t) * m / (sqrt(v) / sqrt(1 - b2^t) + eps)
// `step` is a device counter (float, like torch's capturable state) incremented by the kernel,
// `lr` a device scalar, so that a captured CUDA graph follows LR schedules.
// ---------------------------------------------------------------------------
// One element's update with every rounding spelled out (no compiler-chosen FMA contraction), so that k_adam and the
// fused all-reduce + Adam kernel (nvf_symm.cuh) produce bit-identical parameters from the same gradient.
__device__ __forceinline__ void adam_update(float& param, float& m, float& v, float g, float beta1, float beta2, float eps,
                                            float step_size, float bc2s) {
  m = __fmaf_rn(1.f - beta1, g - m, m);
  v = __fmaf_rn(1.f - beta2, __fmul_rn(g, g), __fmul_rn(v, beta2));
  const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(v), bc2s), eps);
  param = __fmaf_rn(-step_size, __fdiv_rn(m, denom), param);
}

// Bias corrections in double, like the Python scalars of torch's (non-capturable) Adam: step_size = lr / (1 - b1^t),
// bc2s = sqrt(1 - b2^t) with t = step + 1.  ONE thread of the CTA evaluates the two double-precision pow() calls (they
// were most of the kernel's time when every thread did) and hands the floats over through shared memory.
__device__ __forceinline__ void adam_bias_corrections(const float* step, const float* lr, float beta1, float beta2,
                                                      float& step_size, float& bc2s) {
  __shared__ float s_bc[2];
  if (threadIdx.x == 0) {
    const double t = (double)step[0] + 1.0;
    const double bc1 = 1.0 - pow((double)beta1, t), bc2 = 1.0 - pow((double)beta2, t);
    s_bc[0] = (float)((double)lr[0] / bc1);
    s_bc[1] = (float)sqrt(bc2);
  }
  __syncthreads();
  step_size = s_bc[0];
  bc2s = s_bc[1];
}

struct AdamParams {
  float* param; const float* grad; float* m; float* v;
  float* step; const float* lr;
  float beta1, beta2, eps;
  int64_t n;
};

__global__ void __launch_bounds__(256) k_adam(AdamParams p) {
  float step_size, bc2s;
  adam_bias_corrections(p.step, p.lr, p.beta1, p.beta2, step_size, bc2s);
  for (int64_t i = (int64_t)blockIdx.x * 256 + threadIdx.x; i < p.n; i += (int64_t)gridDim.x * 256) {
    float m = p.m[i], v = p.v[i], w = p.param[i];
    adam_update(w, m, v, p.grad[i], p.beta1, p.beta2, p.eps, step_size, bc2s);
    p.m[i] = m; p.v[i] = v;
    p.param[i] = w;
  }
}
// the counter is advanced by a separate one-thread launch so every CTA of k_adam sees the same t
__global__ void k_adam_tick(float* step) {
  step[0] += 1.f;
}

}  // namespace fast
}  // namespace nvf
