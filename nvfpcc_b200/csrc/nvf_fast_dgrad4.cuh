// Data gradient of the k=4 stride-1 convolutions of the training path (conv1, conv2), computed with only the
// algorithmic multiply-adds:
//
//   dX[ci][z][y][x] = (a[ci][z][y][x] > 0) ? sum_co sum_k W[co][ci][k] * g[co][z-kz][y-ky][x-kx] : 0
//
// g is D^3 (pitch D), dX and a are (D+3)^3 with the x pitch padded to D+4.  Every product is formed only where
// g is in range, so nothing multiplies a padding zero:
//   z, y: one warp owns one output row (z, y).  The kz and ky taps that reach inside g are a warp-uniform range
//         [max(0, z-D+1), min(3, z)]; the two tap loops run over exactly that range, outside the unrolled body.
//   x:    input-stationary.  Lane q of a channel group holds the R inputs x' = qR .. qR+R-1 of the row and adds
//         each of them into the R+3 outputs x' .. x'+3 it reaches (partial sums in registers).  The runs of
//         neighbouring lanes overlap by three outputs; the epilogue adds them with shuffles in a fixed order.
//   ci:   four channel groups per warp; a lane accumulates CPL = C/8 channel pairs in 64-bit registers (FFMA2),
//         pair P = k*4 + group, so the weight loads of the four groups hit distinct banks.
// Lane = group * 8 + q, QX = D / R = 8 lanes along x.  The unrolled body per (kz, ky) is, for each co, one
// g load (LDS.128 for R = 4, LDS.64 for R = 2, the same address for the four groups), 2*CPL weight LDS.128
// and R * 4 * CPL FFMA2.
//
// Work count.  Per (z, y, kz, ky, co) the 32 lanes issue R*4*CPL FFMA2 = 32*R*4*(C/8)*2 = 4*D*C multiply-adds,
// and the (kz, ky) ranges summed over the (D+3)^2 rows give (4D)^2 pairs, so a block executes
// (4D)^2 * C * 4*D*C = 64 * C^2 * D^3 multiply-adds: exactly the algorithmic count (ratio 1.00).  SASS: the
// unrolled (kz, ky) body holds C*R*4*CPL FFMA2 (conv2 C = 8: 128, C = 16: 512; conv1 C = 8: 64, C = 16: 256)
// and no other FFMA.
//
// CTA: TZ x TY warps (output rows), staged in shared memory once: the g rows the tile reaches
// ([C][TZ+3][TY+3][D], rows outside g are never read and not loaded) and all weights ([co][kz][ky][P][kx][2],
// repacked from PACK_CONV_DGRAD while staging).  ptxas (sm_100a, -Xptxas -v), no spills in any instantiation:
//   <8, 32, 1, 7>   69 registers, 56 KB smem, 224 threads: 4 CTAs (28 warps) per SM
//   <16, 32, 3, 7>  78 registers, 184 KB smem, 672 threads: 1 CTA (21 warps) per SM
//   <8, 16, 1, 5>   69 registers, 32 KB smem, 160 threads: 5 CTAs (25 warps) per SM
//   <16, 16, 2, 5>  87 registers, 104 KB smem, 320 threads: 2 CTAs (20 warps) per SM
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"
#include "nvf_tma.cuh"

namespace nvf {
namespace fast {

struct Dgrad4Params {
  const float* g;     // [n][C][D][D][D]
  float* out;         // [n][C][D+3][D+3][D+4]
  const float* Wp;    // PACK_CONV_DGRAD: [co][flipped k][ci]
  const float* mask;  // same layout as out: v = mask > 0 ? v : 0
  int32_t n;
};

template <int C, int D, int TZ, int TY>
struct Dgrad4Cfg {
  static constexpr int R = D / 8;                    // inputs per lane along x
  static constexpr int CPL = C / 8;                  // channel pairs per lane
  static constexpr int DO = D + 3, OP = D + 4;       // output edge and x pitch
  static constexpr int THREADS = 32 * TZ * TY;
  static constexpr int SZ = TZ + 3, SY = TY + 3;     // staged slices / rows
  static constexpr int CS = SZ * SY * D;             // staged floats per channel
  static constexpr int G_FLOATS = C * CS;
  static constexpr int W_FLOATS = C * C * 64;
  static constexpr int SMEM_BYTES = (G_FLOATS + W_FLOATS) * 4;
  static constexpr int TILES_Z = (DO + TZ - 1) / TZ, TILES_Y = (DO + TY - 1) / TY;
  static_assert(C % 8 == 0 && D % 8 == 0 && (R == 2 || R == 4), "dgrad4 lane layout");
};

template <int R>
__device__ __forceinline__ void ld_run(const float* p, float (&v)[R]) {
  if constexpr (R == 4) {
    const float4 t = *reinterpret_cast<const float4*>(p);
    v[0] = t.x; v[1] = t.y; v[2] = t.z; v[3] = t.w;
  } else {
    const float2 t = *reinterpret_cast<const float2*>(p);
    v[0] = t.x; v[1] = t.y;
  }
}
template <int R>
__device__ __forceinline__ void st_run(float* p, const float (&v)[R]) {
  if constexpr (R == 4) *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]);
  else *reinterpret_cast<float2*>(p) = make_float2(v[0], v[1]);
}

template <int C, int D, int TZ, int TY, int MINB>
__global__ void __launch_bounds__(Dgrad4Cfg<C, D, TZ, TY>::THREADS, MINB) k_conv4_dgrad(Dgrad4Params p) {
  using G = Dgrad4Cfg<C, D, TZ, TY>;
  constexpr int R = G::R, CPL = G::CPL, NX = R + 3;
  extern __shared__ __align__(128) float smem[];
  float* s_g = smem;
  float* s_w = smem + G::G_FLOATS;
  const int tid = threadIdx.x;
  int t = blockIdx.x;
  const int tyi = t % G::TILES_Y; t /= G::TILES_Y;
  const int tzi = t % G::TILES_Z; t /= G::TILES_Z;
  const int b = t;
  const int z0 = tzi * TZ, y0 = tyi * TY;

  // ---- stage the g rows of slices z0-3 .. z0+TZ-1, rows y0-3 .. y0+TY-1 that lie inside g
  {
    constexpr int NV = D / 4;
    const float* gb = p.g + (size_t)b * C * D * D * D;
    for (int i = tid; i < C * G::SZ * G::SY * NV; i += G::THREADS) {
      int q = i;
      const int xv = q % NV; q /= NV;
      const int sy = q % G::SY; q /= G::SY;
      const int sz = q % G::SZ; q /= G::SZ;
      const int co = q;
      const int iz = z0 - 3 + sz, iy = y0 - 3 + sy;
      if (iz >= 0 && iz < D && iy >= 0 && iy < D)
        tma::cp_async16(s_g + co * G::CS + (sz * G::SY + sy) * D + 4 * xv,
                        gb + (((size_t)co * D + iz) * D + iy) * D + 4 * xv);
    }
    // weights: s_w[co][kz][ky][P][kx][2] = W[co][2P..2P+1][kz][ky][kx] = Wp[co][(3-kz,3-ky,3-kx)][2P..2P+1]
    for (int i = tid; i < G::W_FLOATS / 2; i += G::THREADS) {
      int q = i;
      const int kx = q & 3; q >>= 2;
      const int pr = q % (C / 2); q /= C / 2;
      const int ky = q & 3; q >>= 2;
      const int kz = q & 3; q >>= 2;
      const int co = q;
      const float2 w = __ldg(reinterpret_cast<const float2*>(
          p.Wp + ((size_t)co * 64 + (3 - kz) * 16 + (3 - ky) * 4 + (3 - kx)) * C + 2 * pr));
      reinterpret_cast<float2*>(s_w)[i] = w;
    }
    tma::cp_async_wait_all();
  }
  __syncthreads();

  const int warp = tid >> 5, lane = tid & 31;
  const int tz = warp / TY, ty = warp % TY;
  const int z = z0 + tz, y = y0 + ty;
  if (z >= G::DO || y >= G::DO) return;
  const int grp = lane >> 3, q = lane & 7;

  p2 acc[CPL][NX];
#pragma unroll
  for (int k = 0; k < CPL; ++k)
#pragma unroll
    for (int j = 0; j < NX; ++j) acc[k][j] = p2_bcast(0.f);

  // taps that reach inside g: warp-uniform bounds
  const int kz_lo = z - (D - 1) > 0 ? z - (D - 1) : 0, kz_hi = z < 3 ? z : 3;
  const int ky_lo = y - (D - 1) > 0 ? y - (D - 1) : 0, ky_hi = y < 3 ? y : 3;
#pragma unroll 1
  for (int kz = kz_lo; kz <= kz_hi; ++kz) {
#pragma unroll 1
    for (int ky = ky_lo; ky <= ky_hi; ++ky) {
      const float* gr = s_g + ((tz + 3 - kz) * G::SY + (ty + 3 - ky)) * D + q * R;
      const float* wr = s_w + (kz * 4 + ky) * 4 * C + grp * 8;
#pragma unroll
      for (int co = 0; co < C; ++co) {
        float gv[R];
        ld_run<R>(gr + co * G::CS, gv);
        p2 w[CPL][4];
#pragma unroll
        for (int k = 0; k < CPL; ++k) {
          p2_ld2(wr + co * 64 * C + k * 32, w[k][0], w[k][1]);
          p2_ld2(wr + co * 64 * C + k * 32 + 4, w[k][2], w[k][3]);
        }
#pragma unroll
        for (int r = 0; r < R; ++r) {
          const p2 gg = p2_bcast(gv[r]);
#pragma unroll
          for (int kx = 0; kx < 4; ++kx)
#pragma unroll
            for (int k = 0; k < CPL; ++k) p2_fma(acc[k][r + kx], w[k][kx], gg);
        }
      }
    }
  }

  // ---- epilogue: output x = qR + j gets the partial sums of lanes q, q-1, q-2 (in that order) whose runs
  // reach it; lane q stores x = qR .. qR+R-1, lane 7 also the three outputs past the last input and the pad
  // column (zero)
  constexpr size_t out_cs = (size_t)G::DO * G::DO * G::OP;
  const size_t row = ((size_t)z * G::DO + y) * G::OP;
#pragma unroll
  for (int k = 0; k < CPL; ++k) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      float f[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) f[j] = h ? p2_hi(acc[k][j]) : p2_lo(acc[k][j]);
      float s[NX];
#pragma unroll
      for (int j = 0; j < NX; ++j) s[j] = f[j];
#pragma unroll
      for (int m = 1; m * R < NX; ++m)
#pragma unroll
        for (int j = 0; j + m * R < NX; ++j) {
          const float v = __shfl_up_sync(0xffffffffu, f[j + m * R], m, 8);
          if (q >= m) s[j] += v;
        }
      const int ci = 2 * (k * 4 + grp) + h;
      float* o = p.out + ((size_t)b * C + ci) * out_cs + row;
      const float* mk = p.mask + ((size_t)b * C + ci) * out_cs + row;
      float v[R], m[R];
#pragma unroll
      for (int j = 0; j < R; ++j) v[j] = s[j];
      ld_run<R>(mk + q * R, m);
#pragma unroll
      for (int j = 0; j < R; ++j) v[j] = m[j] > 0.f ? v[j] : 0.f;
      st_run<R>(o + q * R, v);
      if (q == 7) {
        const float4 mt = *reinterpret_cast<const float4*>(mk + D);
        *reinterpret_cast<float4*>(o + D) = make_float4(mt.x > 0.f ? s[R] : 0.f, mt.y > 0.f ? s[R + 1] : 0.f,
                                                        mt.z > 0.f ? s[R + 2] : 0.f, 0.f);
      }
    }
  }
}

}  // namespace fast
}  // namespace nvf
