// Kernels that exist only in the fused training step (nvf_train_step): the loss of a weight-loop step as ONE
// launch.  NVFPCC.py:154-196 computes, per step,
//     n_pts, the GT pyramid (MultiscaleProcessor, :76-88), three focal losses (utils/loss.py:61-111), the logging
//     metrics (:74-84, :113-121), b_latent, b_net and loss = bce + ms0 + ms1 + lmbda (w1 b_latent + w2 b_net),
// and autograd then walks back through all of it.  Here one pass over (p, gt, dist) produces the per-CTA partial
// sums AND dL/dlogit of the three heads (d loss / d bce = d loss / d ms = 1, so the sigmoid derivative is folded
// in: g_logit = dF/dp * p (1 - p)); the last CTA to finish folds the partials in fixed order (deterministic) and
// writes the sums, the total loss, the logged scalars and the two scalar cotangents the parameter-side backward
// kernels need (d loss / d latent_bits, d loss / d net_bits).
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"
#include "nvf_layers.h"
#include "nvf_fast_params.cuh"

namespace nvf {
namespace fast {

struct LossStepParams {
  const float* out;   // [n][32768] probabilities of the main head
  const float* cls1;  // [n][4096]
  const float* cls0;  // [n][512]
  const float* gt;    // dataset rows [n_rows][32768] (or the batch itself when idx == null)
  const float* dist;
  const long long* idx; long long n_rows;
  int* status;        // optional sticky word: bit 0 = an index was outside [0, n_rows) (that block read row 0)
  float* gl2; float* gl1; float* gl0;   // dL/dlogit, or null (no backward wanted)
  double* partial;    // [n * kLossChunks][NVF_LOSS_SUMS]
  unsigned int* ticket;
  float alpha_main, alpha_aux, thh_metric;
  int32_t n;
  // finalisation (last CTA)
  const float* latent_bits;  // [1]
  const float* net_bits;     // [7]
  const float* n_pts;        // [1]
  float n_total, lmbda, w1, w2, w2_grad;
  double* sums;              // [NVF_LOSS_SUMS]
  float* stats;              // [7] loss bce ms0 ms1 b_latent b_net n_pts
  float* g_scal;             // [8]: d loss / d latent_bits, then d loss / d net_bits[0..6]
};

__global__ void __launch_bounds__(256) k_loss_step(LossStepParams p) {
  __shared__ double sm[8][NVF_LOSS_SUMS];
  const int tid = threadIdx.x;
  const int b = blockIdx.x / kLossChunks, chunk = blockIdx.x % kLossChunks;
  long long row = b;
  if (p.idx) {
    row = p.idx[b];
    if (row < 0 || row >= p.n_rows) {
      if (p.status && chunk == 0 && tid == 0) atomicOr(p.status, 1);
      row = 0;
    }
  }
  double s[NVF_LOSS_SUMS];
#pragma unroll
  for (int i = 0; i < NVF_LOSS_SUMS; ++i) s[i] = 0.0;
  const float a_occ = p.alpha_main, a_emp = 1.f - p.alpha_main;
  const float x_occ = p.alpha_aux, x_emp = 1.f - p.alpha_aux;
  const float* gt = p.gt + (size_t)row * kVox;
  const float* dist = p.dist + (size_t)row * kVox;
  const float* out = p.out + (size_t)b * kVox;
  // main head: chunk c covers slices 2c, 2c+1 (2048 voxels), four per thread per pass
  for (int v = chunk * (kVox / kLossChunks) + 4 * tid; v < (chunk + 1) * (kVox / kLossChunks); v += 4 * 256) {
    const float4 g4 = __ldg(reinterpret_cast<const float4*>(gt + v));
    const float4 d4 = __ldg(reinterpret_cast<const float4*>(dist + v));
    const float4 p4 = *reinterpret_cast<const float4*>(out + v);
    const float gv[4] = {g4.x, g4.y, g4.z, g4.w}, dv[4] = {d4.x, d4.y, d4.z, d4.w}, pv[4] = {p4.x, p4.y, p4.z, p4.w};
    float gl[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const bool occ = gv[j] != 0.f;
      const float pr = pv[j], d = dv[j];
      float l, g;
      focal_term(pr, occ, a_occ, a_emp, d + (occ ? 1.f : 0.f), l, g);
      s[0] += l;
      gl[j] = g * pr * (1.f - pr);
      if (pr > p.thh_metric) { s[3] += (double)(d * d); s[4] += 1.0; }
      if (occ) { s[6] += 1.0; if (pr > 0.5f) s[5] += 1.0; }
      else { s[8] += 1.0; if (!(pr > 0.5f)) s[7] += 1.0; }
    }
    if (p.gl2) *reinterpret_cast<float4*>(p.gl2 + (size_t)b * kVox + v) = make_float4(gl[0], gl[1], gl[2], gl[3]);
  }
  // 16^3 head (cls1): GT = max over 2x2x2
  for (int v = chunk * (4096 / kLossChunks) + tid; v < (chunk + 1) * (4096 / kLossChunks); v += 256) {
    const int z = v >> 8, y = (v >> 4) & 15, x = v & 15;
    bool occ = false;
#pragma unroll
    for (int dz = 0; dz < 2; ++dz)
#pragma unroll
      for (int dy = 0; dy < 2; ++dy) {
        const float2 t = __ldg(reinterpret_cast<const float2*>(gt + ((2 * z + dz) * 32 + 2 * y + dy) * 32 + 2 * x));
        occ = occ || t.x != 0.f || t.y != 0.f;
      }
    const float pr = p.cls1[(size_t)b * 4096 + v];
    float l, g;
    focal_term(pr, occ, x_occ, x_emp, 1.f, l, g);
    s[2] += l;
    if (p.gl1) p.gl1[(size_t)b * 4096 + v] = g * pr * (1.f - pr);
    if (occ) { s[14] += 1.0; if (pr > 0.5f) s[13] += 1.0; }
    else { s[16] += 1.0; if (!(pr > 0.5f)) s[15] += 1.0; }
  }
  // 8^3 head (cls0): GT = max over 4x4x4
  for (int v = chunk * (512 / kLossChunks) + tid; v < (chunk + 1) * (512 / kLossChunks); v += 256) {
    const int z = v >> 6, y = (v >> 3) & 7, x = v & 7;
    bool occ = false;
    for (int dz = 0; dz < 4; ++dz)
#pragma unroll
      for (int dy = 0; dy < 4; ++dy) {
        const float4 t = __ldg(reinterpret_cast<const float4*>(gt + ((4 * z + dz) * 32 + 4 * y + dy) * 32 + 4 * x));
        occ = occ || t.x != 0.f || t.y != 0.f || t.z != 0.f || t.w != 0.f;
      }
    const float pr = p.cls0[(size_t)b * 512 + v];
    float l, g;
    focal_term(pr, occ, x_occ, x_emp, 1.f, l, g);
    s[1] += l;
    if (p.gl0) p.gl0[(size_t)b * 512 + v] = g * pr * (1.f - pr);
    if (occ) { s[10] += 1.0; if (pr > 0.5f) s[9] += 1.0; }
    else { s[12] += 1.0; if (!(pr > 0.5f)) s[11] += 1.0; }
  }
  // CTA reduction in fixed order: shuffle tree inside each warp, then the 8 warps in order
#pragma unroll
  for (int i = 0; i < NVF_LOSS_SUMS; ++i) {
    double v = s[i];
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((tid & 31) == 0) sm[tid >> 5][i] = v;
  }
  __syncthreads();
  if (tid < NVF_LOSS_SUMS) {
    double t = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) t += sm[w][tid];
    p.partial[(size_t)blockIdx.x * NVF_LOSS_SUMS + tid] = t;
  }
  if (!last_cta(p.ticket)) return;
  // ---- last CTA: fold the partials (one warp per sum, lanes stride over the partials, fixed shuffle tree)
  __shared__ double tot[NVF_LOSS_SUMS];
  const int np = p.n * kLossChunks;
  for (int w = tid >> 5; w < NVF_LOSS_SUMS; w += 8) {
    double v = 0.0;
    for (int c = tid & 31; c < np; c += 32) v += p.partial[(size_t)c * NVF_LOSS_SUMS + w];
    for (int o = 16; o >= 1; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((tid & 31) == 0) {
      tot[w] = v;
      p.sums[w] = v;
    }
  }
  __syncthreads();
  if (tid == 0) {
    const float bce = (float)tot[0], ms0 = (float)tot[1], ms1 = (float)tot[2];
    const float npts = p.n_pts[0];
    float nb = 0.f;
    for (int i = 0; i < kNumQuant; ++i) nb += p.net_bits[i];
    const float b_latent = p.latent_bits[0] / npts;
    const float b_net = nb / p.n_total;
    const float loss = bce + ms0 + ms1 + p.lmbda * (b_latent * p.w1 + b_net * p.w2);
    if (p.stats) {
      p.stats[0] = loss; p.stats[1] = bce; p.stats[2] = ms0; p.stats[3] = ms1;
      p.stats[4] = b_latent; p.stats[5] = b_net; p.stats[6] = npts;
    }
    if (p.g_scal) {
      p.g_scal[0] = p.lmbda * p.w1 / npts;
      const float gn = p.lmbda * p.w2_grad / p.n_total;
      for (int i = 0; i < kNumQuant; ++i) p.g_scal[1 + i] = gn;
    }
  }
}

// advances the device-resident step counter of the in-kernel noise generators (one thread, end of the step)
__global__ void k_rng_tick(unsigned long long* ctr) {
  ctr[0] += 1ull;
}

}  // namespace fast
}  // namespace nvf
