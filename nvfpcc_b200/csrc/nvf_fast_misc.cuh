// Small-layer kernels of the training path: weight gradient of the three
// 3x3x3 classifier heads (conv2_cls / conv1_cls / conv0_cls, utils/network.py:
// 4731-4751) and the IGDN parameter gradients (gdn_3d.py:137-159 backward).
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"
#include "nvf_tma.cuh"

namespace nvf {
namespace fast {

// dW[ci][kz][ky][kx] = sum_{b,pos} gl[b][pos] * a[b][ci][pos + k - 1]   (zero padding 1)
// db                 = sum gl
// Thread = (ci, kz, ky) owns 3 outputs; NSET position sets share the rows of a band.
struct ClsWgradParams {
  const float* g;    // [n][D][D][D]      dL/dlogit
  const float* a;    // [n][C][D][D][D]   head input
  float* partial;    // [gridDim.x][C*27 + 1]
  int32_t n;
};

// One CTA = (block, row band, z segment): it streams along z with a ring of four staged input
// slices (each slice is fetched once per CTA instead of three times); slice z+2 and the g rows of
// z+1 stream in with cp.async while slice z is being consumed.
template <int C, int D, int TYB, int ZSEG>
struct ClsWgradCfg {
  static constexpr int SETT = C * 9;
  static constexpr int NSET = 256 / SETT;
  static constexpr int PI = D + 4;                 // tile col c <-> ix = c - 1
  static constexpr int RA = TYB + 2;
  static constexpr int SLOT = C * RA * PI;         // one staged slice
  static constexpr int A_FLOATS = 4 * SLOT;
  static constexpr int G_FLOATS = TYB * D;        // one of two g buffers
  static constexpr int NW = C * 27;
  static constexpr int OUT_FLOATS = NW + 1;
  static constexpr int RED_FLOATS = NSET * NW + 256;
  static constexpr int SMEM_FLOATS = (A_FLOATS + 2 * G_FLOATS) > RED_FLOATS ? (A_FLOATS + 2 * G_FLOATS) : RED_FLOATS;
  static constexpr int SMEM_BYTES = SMEM_FLOATS * 4;
  static constexpr int BANDS = D / TYB;
  static constexpr int SEGS = D / ZSEG;
  static_assert(SETT <= 256 && D % 8 == 0 && D % TYB == 0 && D % ZSEG == 0, "cls wgrad tiling");
};

template <int C, int D, int TYB, int ZSEG>
__global__ void __launch_bounds__(256) k_cls_wgrad(ClsWgradParams p) {
  using G = ClsWgradCfg<C, D, TYB, ZSEG>;
  extern __shared__ __align__(128) float smem[];
  float* s_a = smem;
  float* s_g = smem + G::A_FLOATS;
  const int tid = threadIdx.x;
  const bool active = tid < G::NSET * G::SETT;
  const int set = active ? tid / G::SETT : 0;
  int r = active ? tid % G::SETT : 0;
  const int ky = r % 3; r /= 3;
  const int kz = r % 3; r /= 3;
  const int ci = r;
  float acc[3] = {0.f, 0.f, 0.f};
  float dbacc = 0.f;

  int q = blockIdx.x;
  const int seg = q % G::SEGS; q /= G::SEGS;
  const int band = q % G::BANDS; q /= G::BANDS;
  const int b = q;
  const int y0 = band * TYB, z0 = seg * ZSEG;
  const float* ab = p.a + (size_t)b * C * D * D * D;

  // stage input slice iz into ring slot (iz + 4) % 4 (zero outside the block: padding 1), asynchronously
  auto stage = [&](int iz) {
    float* dst = s_a + ((iz + 4) & 3) * G::SLOT;
    constexpr int NV = D / 4;
    for (int i = tid; i < C * G::RA * NV; i += 256) {
      int t = i;
      const int xv = t % NV; t /= NV;
      const int rr = t % G::RA; t /= G::RA;
      const int ch = t;
      const int iy = y0 + rr - 1;
      const bool ok = iz >= 0 && iz < D && iy >= 0 && iy < D;
      const float* src = ok ? ab + (((size_t)ch * D + iz) * D + iy) * D + 4 * xv : ab;
      float* d = dst + (ch * G::RA + rr) * G::PI + 1 + 4 * xv;
      tma::cp_async4z(d, src, ok); tma::cp_async4z(d + 1, src + 1, ok);
      tma::cp_async4z(d + 2, src + 2, ok); tma::cp_async4z(d + 3, src + 3, ok);
    }
  };
  auto stage_g = [&](int z) {
    const float* gb = p.g + (((size_t)b * D + z) * D + y0) * D;
    float* dst = s_g + (z & 1) * G::G_FLOATS;
    for (int i = tid; i < G::G_FLOATS / 4; i += 256) tma::cp_async16(dst + 4 * i, gb + 4 * i);
  };
  // the two halo columns of every staged row stay zero for the whole kernel
  for (int i = tid; i < 4 * C * G::RA; i += 256) {
    s_a[i * G::PI] = 0.f;
    s_a[i * G::PI + D + 1] = 0.f;
  }
  stage(z0 - 1);
  stage(z0);
  stage(z0 + 1);
  stage_g(z0);
  for (int z = z0; z < z0 + ZSEG; ++z) {
    tma::cp_async_wait_all();
    __syncthreads();                 // slices z-1..z+1 and g(z) have landed; everyone is done with z-1
    if (z + 1 < z0 + ZSEG) {
      stage(z + 2);                  // overwrites the slot of slice z-2
      stage_g(z + 1);
    }
    const float* sg = s_g + (z & 1) * G::G_FLOATS;
    {
      float s = 0.f;
      for (int i = tid; i < G::G_FLOATS; i += 256) s += sg[i];
      dbacc += s;
    }
    if (active) {
      const float* a_base = s_a + ((z + kz - 1 + 4) & 3) * G::SLOT + (ci * G::RA + ky) * G::PI;
      for (int rr = set; rr < TYB; rr += G::NSET) {
#pragma unroll
        for (int xo = 0; xo < D / 8; ++xo) {
          const float* ar = a_base + rr * G::PI + 8 * xo;
          const float4 a0 = *reinterpret_cast<const float4*>(ar);
          const float4 a1 = *reinterpret_cast<const float4*>(ar + 4);
          const float2 a2 = *reinterpret_cast<const float2*>(ar + 8);
          const float av[10] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w, a2.x, a2.y};
          const float4 g0 = *reinterpret_cast<const float4*>(sg + rr * D + 8 * xo);
          const float4 g1 = *reinterpret_cast<const float4*>(sg + rr * D + 8 * xo + 4);
          const float gv[8] = {g0.x, g0.y, g0.z, g0.w, g1.x, g1.y, g1.z, g1.w};
#pragma unroll
          for (int j = 0; j < 8; ++j)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx) acc[kx] = fmaf(gv[j], av[j + kx], acc[kx]);
        }
      }
    }
  }
  __syncthreads();
  float* red = smem;
  if (active) {
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) red[set * G::NW + ci * 27 + kz * 9 + ky * 3 + kx] = acc[kx];
  }
  red[G::NSET * G::NW + tid] = dbacc;
  __syncthreads();
  float* out = p.partial + (size_t)blockIdx.x * G::OUT_FLOATS;
  for (int i = tid; i < G::NW; i += 256) {
    float s = 0.f;
#pragma unroll
    for (int t = 0; t < G::NSET; ++t) s += red[t * G::NW + i];
    out[i] = s;
  }
  if (tid == 0) {
    float s = 0.f;
    for (int i = 0; i < 256; ++i) s += red[G::NSET * G::NW + i];
    out[G::NW] = s;
  }
}

// IGDN parameter gradients, one CTA per block:
//   n_i = sqrt(beta_i + sum_j gamma_ij x_j^2),  t_i = g_i x_i / (2 n_i)
//   dbeta_i = sum_pos t_i,  dgamma_ij = sum_pos t_i x_j^2
// partial[b][C*C + C] = (dgamma, dbeta) of block b.
struct IgdnParamParams {
  const float* x;      // [n][C][64]
  const float* g;      // [n][C][64]  dL/dy
  const float* beta;   // [C]
  const float* gamma;  // [C][C]
  float* partial;      // [n][C*C + C]
  int32_t n, C;
};
__global__ void __launch_bounds__(256) k_igdn_param(IgdnParamParams p) {
  extern __shared__ __align__(128) float smem[];
  const int C = p.C;
  float* sx2 = smem;             // [C][64]  x^2
  float* st = smem + C * 64;     // [C][64]  t
  const int b = blockIdx.x, tid = threadIdx.x;
  const float* xb = p.x + (size_t)b * C * 64;
  const float* gb = p.g + (size_t)b * C * 64;
  for (int i = tid; i < C * 64; i += 256) {
    const float v = xb[i];
    sx2[i] = v * v;
  }
  __syncthreads();
  for (int i = tid; i < C * 64; i += 256) {
    const int c = i >> 6, pos = i & 63;
    float nn = p.beta[c];
    for (int j = 0; j < C; ++j) nn = fmaf(p.gamma[c * C + j], sx2[j * 64 + pos], nn);
    st[i] = gb[i] * xb[i] / (2.f * sqrtf(nn));
  }
  __syncthreads();
  float* out = p.partial + (size_t)b * (C * C + C);
  for (int e = tid; e < C * C + C; e += 256) {
    float s = 0.f;
    if (e < C * C) {
      const int i = e / C, j = e % C;
      for (int pos = 0; pos < 64; ++pos) s = fmaf(st[i * 64 + pos], sx2[j * 64 + pos], s);
    } else {
      const int i = e - C * C;
      for (int pos = 0; pos < 64; ++pos) s += st[i * 64 + pos];
    }
    out[e] = s;
  }
}

}  // namespace fast
}  // namespace nvf
