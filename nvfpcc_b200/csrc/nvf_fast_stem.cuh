// The "stem" of the NVF decoder - everything at <= 8^3 resolution - as ONE CTA
// per leaf block, activations in shared memory:
//   forward   latent -> up0 (convT k5 s2 p2 op1) -> IGDN -> conv0 (convT k5 s2 p2 op1, ReLU) -> conv0_cls + sigmoid
//             (utils/network.py:4759-4761, gdn_3d.py:153-157)
//   backward  d(conv0 pre-activation) -> conv0 wgrad/bias/dgrad -> IGDN backward (dx, dbeta, dgamma)
//             -> up0 wgrad/bias -> d_latent                       (SURVEY.md 3.5)
// These layers hold < 0.5 % of the MACs; as separate grid-wide launches they were
// latency-bound (a handful of CTAs each).  Per-block weight-gradient partials are
// summed over blocks in fixed order by k_reduce_partials.
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"

namespace nvf {
namespace fast {

constexpr int kStemThreads = 512;

struct StemFwdParams {
  const float* latent;  // [n][CH][8]
  const float* up0_wp;  // PACK_CONVT_FWD [ci][k][co]  (CH x 125 x C0)
  const float* up0_b;
  const float* beta;    // [C0]
  const float* gamma;   // [C0][C0]
  const float* conv0_wp;// PACK_CONVT_FWD [ci][k][co]  (C0 x 125 x C1)
  const float* conv0_b;
  const float* cls0_wp; // [C1][27] or null (decode: no aux head)
  const float* cls0_b;
  float* x0;            // [n][C0][64]
  float* a0;            // [n][C0][64]
  float* a1;            // [n][C1][512]
  float* cls0;          // [n][512] or null
  float* cls0_copy;     // [n][512] or null
  int32_t n, CH, C0, C1;
};

// convT k5 s2 p2 op1 taps of output coordinate o along one axis: k = (o & 1) + 2t, input (o + 2 - k) / 2
__device__ __forceinline__ int stem_tap_lo(int o) { return o & 1; }

// PERSIST = false (training, few blocks): grid = n * 8, CTA (b, zs) recomputes the tiny up0 + IGDN and produces conv0's
// output slice zs: 8 short CTAs per block, everything latency-bound runs in parallel.
// PERSIST = true (decode of a whole cloud): grid = 2 * G, CTA (g, z parity) stages the conv0 taps of its parity ONCE
// (154 KB at 16,32 channels: re-staging them per slice was 1.9 GB of L2 traffic per 1247 leaves and 3.4 ms), then
// walks over the leaves g, g+G, ..: up0 + IGDN once per leaf, then the four slices of its parity.  Per output the
// arithmetic is the same in both modes, so a leaf's result does not depend on the mode.
// The conv0_cls head runs afterwards as a classifier kernel (nvf_fast_conv.cuh).
constexpr int kStemFwdThreads = 512;
template <bool PERSIST>
__global__ void __launch_bounds__(kStemFwdThreads) k_stem_fwd(StemFwdParams p) {
  extern __shared__ __align__(128) float smem[];
  const int CH = p.CH, C0 = p.C0, C1 = p.C1;
  float* s_lat = smem;                 // [CH][8]
  float* s_x0 = s_lat + CH * 8;        // [C0][64]
  float* s_a0 = s_x0 + C0 * 64;        // [C0][64]
  float* s_gam = s_a0 + C0 * 64;       // [C0][C0] gamma, then [C0] beta
  float* s_wu = s_gam + C0 * C0 + C0;  // up0 weights [CH][125][C0]
  float* s_wc = s_wu + ((CH * 125 * C0 + 3) & ~3);  // conv0 weights of this slice's kz parity [C0][3][25][C1]
  const int tid = threadIdx.x;
  const int pz = PERSIST ? (blockIdx.x & 1) : (blockIdx.x & 7) & 1, NT = pz ? 2 : 3;   // kz = pz + 2t
  for (int i = tid; i < C0 * C0 + C0; i += kStemFwdThreads) s_gam[i] = i < C0 * C0 ? p.gamma[i] : p.beta[i - C0 * C0];
  for (int i = tid; i < CH * 125 * C0; i += kStemFwdThreads) s_wu[i] = __ldg(p.up0_wp + i);
  {
    const int tapv = 25 * C1 / 4;   // float4 per (ci, kz)
    for (int i = tid; i < C0 * 3 * tapv; i += kStemFwdThreads) {
      const int v4 = i % tapv, t = (i / tapv) % 3, ci = i / (3 * tapv);
      if (t < NT)
        reinterpret_cast<float4*>(s_wc)[i] =
            __ldg(reinterpret_cast<const float4*>(p.conv0_wp + ((size_t)(ci * 5 + pz + 2 * t) * 25) * C1) + v4);
    }
  }
  const int b_step = PERSIST ? (int)(gridDim.x >> 1) : p.n;
#pragma unroll 1
  for (int b = PERSIST ? (int)(blockIdx.x >> 1) : (int)(blockIdx.x >> 3); b < p.n; b += b_step) {
  __syncthreads();                                       // weights staged / the previous leaf's activations are free
  if (tid < CH * 8) s_lat[tid] = p.latent[(size_t)b * CH * 8 + tid];
  __syncthreads();
  // up0: CH x 2^3 -> C0 x 4^3
  for (int idx = tid; idx < C0 * 64; idx += kStemFwdThreads) {
    const int co = idx >> 6, z = (idx >> 4) & 3, y = (idx >> 2) & 3, x = idx & 3;
    float v = p.up0_b[co];
    for (int ci = 0; ci < CH; ++ci)
      for (int kz = z & 1; kz < 5; kz += 2) {
        const int tz = z + 2 - kz;
        if (tz < 0 || tz >= 4) continue;
        for (int ky = y & 1; ky < 5; ky += 2) {
          const int ty = y + 2 - ky;
          if (ty < 0 || ty >= 4) continue;
          for (int kx = x & 1; kx < 5; kx += 2) {
            const int tx = x + 2 - kx;
            if (tx < 0 || tx >= 4) continue;
            v = fmaf(s_lat[ci * 8 + (tz >> 1) * 4 + (ty >> 1) * 2 + (tx >> 1)],
                     s_wu[(ci * 125 + kz * 25 + ky * 5 + kx) * C0 + co], v);
          }
        }
      }
    s_x0[idx] = v;
    if (PERSIST ? pz == 0 : (blockIdx.x & 7) == 0) p.x0[(size_t)b * C0 * 64 + idx] = v;
  }
  __syncthreads();
  // IGDN
  for (int idx = tid; idx < C0 * 64; idx += kStemFwdThreads) {
    const int c = idx >> 6, pos = idx & 63;
    float nn = s_gam[C0 * C0 + c];
    for (int j = 0; j < C0; ++j) {
      const float xj = s_x0[j * 64 + pos];
      nn = fmaf(s_gam[c * C0 + j], xj * xj, nn);
    }
    const float v = s_x0[idx] * sqrtf(nn);
    s_a0[idx] = v;
    if (PERSIST ? pz == 0 : (blockIdx.x & 7) == 0) p.a0[(size_t)b * C0 * 64 + idx] = v;
  }
  __syncthreads();
  // conv0 slice zs: C0 x 4^3 -> C1 x 8 x 8, ReLU.  item = (position in the slice, group of 4 output channels);
  // the input-channel sum of an item is split over the two threads of a lane pair (halves the serial chain of
  // this latency-bound kernel) and combined with one shuffle, always in the order (low half) + (high half).
  const int groups = C1 / 4;
  const int half = tid & 1, ci_lo = half * (C0 / 2), ci_hi = ci_lo + C0 / 2;
#pragma unroll 1
  for (int zs = PERSIST ? pz : (int)(blockIdx.x & 7); zs < (PERSIST ? 8 : (int)(blockIdx.x & 7) + 1); zs += 2)
  for (int item = tid >> 1; item < 64 * groups; item += kStemFwdThreads / 2) {
    const int pos = item & 63, cg = item >> 6;
    const int z = zs, y = pos >> 3, x = pos & 7;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < NT; ++t) {
      const int tz = z + 2 - (pz + 2 * t);
      if (tz < 0 || tz >= 8) continue;
      for (int ky = y & 1; ky < 5; ky += 2) {
        const int ty = y + 2 - ky;
        if (ty < 0 || ty >= 8) continue;
        for (int kx = x & 1; kx < 5; kx += 2) {
          const int tx = x + 2 - kx;
          if (tx < 0 || tx >= 8) continue;
          const int ipos = (tz >> 1) * 16 + (ty >> 1) * 4 + (tx >> 1);
          const float* wk = s_wc + (size_t)(t * 25 + ky * 5 + kx) * C1 + cg * 4;
#pragma unroll 4
          for (int ci = ci_lo; ci < ci_hi; ++ci) {
            const float a = s_a0[ci * 64 + ipos];
            const float4 w0 = *reinterpret_cast<const float4*>(wk + (size_t)ci * 75 * C1);
            acc[0] = fmaf(a, w0.x, acc[0]); acc[1] = fmaf(a, w0.y, acc[1]);
            acc[2] = fmaf(a, w0.z, acc[2]); acc[3] = fmaf(a, w0.w, acc[3]);
          }
        }
      }
    }
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const float other = __shfl_xor_sync(0xffffffffu, acc[c], 1);
      const float v = (half ? other + acc[c] : acc[c] + other) + p.conv0_b[cg * 4 + c];
      if (half == 0) p.a1[((size_t)b * C1 + cg * 4 + c) * 512 + zs * 64 + pos] = v > 0.f ? v : 0.f;
    }
  }
  }
}

struct StemBwdParams {
  const float* latent;   // [n][CH][8]
  const float* x0;       // [n][C0][64]
  const float* a0;       // [n][C0][64]
  const float* g1;       // [n][C1][512]  dL/d(conv0 pre-activation)
  const float* beta;     // [C0]
  const float* gamma;    // [C0][C0]
  const float* conv0_w;  // raw (C0, C1, 5,5,5)
  const float* up0_w;    // raw (CH, C0, 5,5,5)
  float* partial;        // [n][stem_partial_floats] or null (no weight gradients)
  float* g_latent;       // [n][CH][8] or null
  int32_t n, CH, C0, C1, need_w;
};
// per-block partial layout: conv0_w | conv0_b | igdn_gamma | igdn_beta | up0_w | up0_b
__host__ __device__ inline int stem_partial_floats(int CH, int C0, int C1) {
  return C0 * C1 * 125 + C1 + C0 * C0 + C0 + CH * C0 * 125 + C0;
}

// Kernel A, grid = n * C0: CTA (b, ci) holds g1[b] in shared memory and produces
//   conv0 wgrad rows dW[ci][:][:]  (per-block partial), the conv0 bias gradient (ci == 0),
//   conv0 dgrad gy[b][ci][64] -> p.gy (global).
constexpr int kStemBwdAThreads = 512;   // these kernels are latency-bound chains: more threads = shorter chains
__global__ void __launch_bounds__(kStemBwdAThreads) k_stem_bwd_a(StemBwdParams p, float* gy_out) {
  extern __shared__ __align__(128) float smem[];
  const int CH = p.CH, C0 = p.C0, C1 = p.C1;
  float* s_g1 = smem;                   // [C1][512]
  float* s_a0 = s_g1 + C1 * 512;        // [64]
  float* s_part = s_a0 + 64;            // [8][64]
  float* s_w = s_part + 512;            // conv0 W[ci][C1][125]
  const int b = blockIdx.x / C0, ci = blockIdx.x % C0, tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  {
    const float4* src = reinterpret_cast<const float4*>(p.g1 + (size_t)b * C1 * 512);
    for (int i = tid; i < C1 * 128; i += kStemBwdAThreads) reinterpret_cast<float4*>(s_g1)[i] = __ldg(src + i);
    if (tid < 64) s_a0[tid] = p.a0[((size_t)b * C0 + ci) * 64 + tid];
    for (int i = tid; i < C1 * 125; i += kStemBwdAThreads) s_w[i] = __ldg(p.conv0_w + (size_t)ci * C1 * 125 + i);
  }
  __syncthreads();
  float* part = p.partial ? p.partial + (size_t)b * stem_partial_floats(CH, C0, C1) : nullptr;
  if (p.need_w && part) {
    // conv0 wgrad: dW[ci][co][k] = sum_{i in 4^3} a0[ci][i] * g1[co][2i + k - 2]
    for (int e = tid; e < C1 * 125; e += kStemBwdAThreads) {
      int q = e;
      const int kx = q % 5; q /= 5;
      const int ky = q % 5; q /= 5;
      const int kz = q % 5; q /= 5;
      const int co = q;
      float s = 0.f;
      for (int iz = 0; iz < 4; ++iz) {
        const int oz = 2 * iz + kz - 2;
        if (oz < 0 || oz >= 8) continue;
        for (int iy = 0; iy < 4; ++iy) {
          const int oy = 2 * iy + ky - 2;
          if (oy < 0 || oy >= 8) continue;
#pragma unroll
          for (int ix = 0; ix < 4; ++ix) {
            const int ox = 2 * ix + kx - 2;
            if (ox < 0 || ox >= 8) continue;
            s = fmaf(s_a0[iz * 16 + iy * 4 + ix], s_g1[co * 512 + oz * 64 + oy * 8 + ox], s);
          }
        }
      }
      part[(size_t)ci * C1 * 125 + e] = s;
    }
    if (ci == 0) {
      // conv0 bias: one warp per channel, fixed-order shuffle tree
      for (int co = warp; co < C1; co += kStemBwdAThreads / 32) {
        float s = 0.f;
        for (int i = lane; i < 512; i += 32) s += s_g1[co * 512 + i];
        for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
        if (lane == 0) part[C0 * C1 * 125 + co] = s;
      }
    }
  }
  // conv0 dgrad: gy[ci][i] = sum_co sum_k g1[co][2i + k - 2] * W[ci][co][k]; co range split in 8 parts
  {
    const int h = tid >> 6, e = tid & 63;
    const int iz = (e >> 4) & 3, iy = (e >> 2) & 3, ix = e & 3;
    float s = 0.f;
    for (int co = h * (C1 / 8); co < (h + 1) * (C1 / 8); ++co) {
      const float* wk = s_w + co * 125;
      for (int kz = 0; kz < 5; ++kz) {
        const int oz = 2 * iz + kz - 2;
        if (oz < 0 || oz >= 8) continue;
        for (int ky = 0; ky < 5; ++ky) {
          const int oy = 2 * iy + ky - 2;
          if (oy < 0 || oy >= 8) continue;
#pragma unroll
          for (int kx = 0; kx < 5; ++kx) {
            const int ox = 2 * ix + kx - 2;
            if (ox < 0 || ox >= 8) continue;
            s = fmaf(s_g1[co * 512 + oz * 64 + oy * 8 + ox], wk[kz * 25 + ky * 5 + kx], s);
          }
        }
      }
    }
    s_part[h * 64 + e] = s;
  }
  __syncthreads();
  if (tid < 64)
    gy_out[((size_t)b * C0 + ci) * 64 + tid] = ((s_part[tid] + s_part[64 + tid]) + (s_part[128 + tid] + s_part[192 + tid])) +
                                               ((s_part[256 + tid] + s_part[320 + tid]) + (s_part[384 + tid] + s_part[448 + tid]));
}

// Kernel B, grid = n: IGDN backward (dx, dbeta, dgamma), up0 wgrad / bias, d_latent.
constexpr int kStemBwdBThreads = 1024;
__global__ void __launch_bounds__(kStemBwdBThreads) k_stem_bwd_b(StemBwdParams p, const float* gy_in) {
  extern __shared__ __align__(128) float smem[];
  const int CH = p.CH, C0 = p.C0, C1 = p.C1;
  float* s_x0 = smem;                   // [C0][64]
  float* s_gy = s_x0 + C0 * 64;         // [C0][64]  dL/d(IGDN out)
  float* s_gx = s_gy + C0 * 64;         // [C0][64]  dL/d(up0 out)
  float* s_n = s_gx + C0 * 64;          // [C0][64]  IGDN norm
  float* s_lat = s_n + C0 * 64;         // [CH][8]
  float* s_gam = s_lat + CH * 8;        // [C0][C0] gamma, then [C0] beta
  float* s_wu = s_gam + C0 * C0 + C0;   // up0 W (CH, C0, 125)
  const int b = blockIdx.x, tid = threadIdx.x;
  const int warp = tid >> 5, lane = tid & 31;
  for (int i = tid; i < C0 * 64; i += kStemBwdBThreads) {
    s_x0[i] = p.x0[(size_t)b * C0 * 64 + i];
    s_gy[i] = gy_in[(size_t)b * C0 * 64 + i];
  }
  if (tid < CH * 8) s_lat[tid] = p.latent[(size_t)b * CH * 8 + tid];
  for (int i = tid; i < C0 * C0 + C0; i += kStemBwdBThreads) s_gam[i] = i < C0 * C0 ? p.gamma[i] : p.beta[i - C0 * C0];
  if (p.g_latent)
    for (int i = tid; i < CH * C0 * 125; i += kStemBwdBThreads) s_wu[i] = __ldg(p.up0_w + i);
  __syncthreads();
  float* part = p.partial ? p.partial + (size_t)b * stem_partial_floats(CH, C0, C1) : nullptr;
  const int o_c0b = C0 * C1 * 125, o_gam = o_c0b + C1, o_bet = o_gam + C0 * C0, o_u0w = o_bet + C0,
            o_u0b = o_u0w + CH * C0 * 125;
  for (int e = tid; e < C0 * 64; e += kStemBwdBThreads) {
    const int c = e >> 6, pos = e & 63;
    float nn = s_gam[C0 * C0 + c];
    for (int j = 0; j < C0; ++j) {
      const float xj = s_x0[j * 64 + pos];
      nn = fmaf(s_gam[c * C0 + j], xj * xj, nn);
    }
    s_n[e] = sqrtf(nn);
  }
  __syncthreads();
  // IGDN backward: dx_k = g_k n_k + x_k sum_i g_i x_i gamma_ik / n_i
  for (int e = tid; e < C0 * 64; e += kStemBwdBThreads) {
    const int k = e >> 6, pos = e & 63;
    float acc = 0.f;
    for (int i = 0; i < C0; ++i)
      acc += s_gy[i * 64 + pos] * s_x0[i * 64 + pos] * s_gam[i * C0 + k] / s_n[i * 64 + pos];
    s_gx[e] = s_gy[e] * s_n[e] + s_x0[e] * acc;
  }
  if (p.need_w && part) {
    // dbeta_i = sum t_i, dgamma_ij = sum t_i x_j^2 with t_i = g_i x_i / (2 n_i)
    for (int e = tid; e < C0 * C0 + C0; e += kStemBwdBThreads) {
      float s = 0.f;
      if (e < C0 * C0) {
        const int i = e / C0, j = e % C0;
        for (int pos = 0; pos < 64; ++pos) {
          const float t = s_gy[i * 64 + pos] * s_x0[i * 64 + pos] / (2.f * s_n[i * 64 + pos]);
          const float xj = s_x0[j * 64 + pos];
          s = fmaf(t, xj * xj, s);
        }
        part[o_gam + e] = s;
      } else {
        const int i = e - C0 * C0;
        for (int pos = 0; pos < 64; ++pos) s += s_gy[i * 64 + pos] * s_x0[i * 64 + pos] / (2.f * s_n[i * 64 + pos]);
        part[o_bet + i] = s;
      }
    }
  }
  __syncthreads();
  if (p.need_w && part) {
    // up0 wgrad: dW[ci][co][k] = sum_{i in 2^3} lat[ci][i] * gx[co][2i + k - 2]
    for (int e = tid; e < CH * C0 * 125; e += kStemBwdBThreads) {
      int q = e;
      const int kx = q % 5; q /= 5;
      const int ky = q % 5; q /= 5;
      const int kz = q % 5; q /= 5;
      const int co = q % C0, ci = q / C0;
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int oz = 2 * (i >> 2) + kz - 2, oy = 2 * ((i >> 1) & 1) + ky - 2, ox = 2 * (i & 1) + kx - 2;
        if (oz < 0 || oz >= 4 || oy < 0 || oy >= 4 || ox < 0 || ox >= 4) continue;
        s = fmaf(s_lat[ci * 8 + i], s_gx[co * 64 + oz * 16 + oy * 4 + ox], s);
      }
      part[o_u0w + e] = s;
    }
    for (int co = warp; co < C0; co += kStemBwdBThreads / 32) {
      float s = s_gx[co * 64 + lane] + s_gx[co * 64 + 32 + lane];
      for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) part[o_u0b + co] = s;
    }
  }
  // d_latent[ci][i] = sum_co sum_k gx[co][2i + k - 2] * W[ci][co][k]: one warp per output, lanes over (co,k)
  if (p.g_latent) {
    for (int e = warp; e < CH * 8; e += kStemBwdBThreads / 32) {
      const int ci = e >> 3, i = e & 7;
      const int iz = i >> 2, iy = (i >> 1) & 1, ix = i & 1;
      float s = 0.f;
      for (int t = lane; t < C0 * 125; t += 32) {
        const int co = t / 125, k = t % 125;
        const int oz = 2 * iz + k / 25 - 2, oy = 2 * iy + (k / 5) % 5 - 2, ox = 2 * ix + k % 5 - 2;
        if (oz < 0 || oz >= 4 || oy < 0 || oy >= 4 || ox < 0 || ox >= 4) continue;
        s = fmaf(s_gx[co * 64 + oz * 16 + oy * 4 + ox], s_wu[(ci * C0 + co) * 125 + k], s);
      }
      for (int o = 16; o >= 1; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
      if (lane == 0) p.g_latent[(size_t)b * CH * 8 + e] = s;
    }
  }
}

}  // namespace fast
}  // namespace nvf
