// Shared-memory tiled FP32 kernels for the stride-2, k=5 transposed convolutions
// of the NVF decoder's training path (up1 / up2, padding 0; F.conv_transpose3d at
// utils/network.py:621), their data gradient and their weight gradient.
//
//   forward   y[co,o]  = b[co] + sum_ci sum_{k: (o-k) even, 0 <= (o-k)/2 < DIN} x[ci,(o-k)/2] W[ci,co,k]
//   dgrad     dx[ci,i] = sum_co sum_k g[co, 2i+k] W[ci,co,k]
//   wgrad     dW[ci,co,k] = sum_{b,i} x[b,ci,i] g[b,co,2i+k]
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"
#include "nvf_fast_conv.cuh"

namespace nvf {
namespace fast {

// ---------------------------------------------------------------------------
// forward: one CTA per (block, output z-slice).  Thread tile: 4 co x 8 x (4 even
// + 4 odd columns) x rows (y, y+2) = 64 accumulators; rows of equal parity share
// the weight taps, the four input rows they touch are fetched once per (ci, kz).
// ---------------------------------------------------------------------------
struct ConvTFwdParams {
  const float* in;    // [n][CI][DIN][DIN][IN_PITCH]
  float* out;         // [n][CO][DOUT][DOUT][OUT_PITCH]   relu(acc + bias)
  const float* Wp;    // PACK_CONVT_FWD [ci][kz][ky][kx][co]
  const float* bias;  // [CO]
  int32_t n;
};

// KS: split of the input-channel sum over KS thread groups (partial sums combined through shared memory in
// fixed order) - the small up1 layer has too few outputs to occupy the GPU otherwise.
template <int CI, int CO, int DIN, int KS = 1>
struct ConvTFwdCfg {
  static constexpr int DOUT = 2 * DIN + 3;
  static constexpr int IN_PITCH = (DIN + 3) / 4 * 4, OUT_PITCH = (DOUT + 3) / 4 * 4;
  static constexpr int QX = (DOUT + 7) / 8;   // column groups of 8 outputs
  static constexpr int RG = (DOUT + 3) / 4;   // row groups of 4 (two (y, y+2) pairs each)
  static constexpr int COG = CO / 4;
  static constexpr int THREADS_USED = QX * RG * 2 * COG;                 // per channel-split group
  static constexpr int THREADS = (THREADS_USED * KS + 31) / 32 * 32;
  static constexpr int TR = DIN + 4;          // tile rows: iy = r - 2
  static constexpr int IP = 4 * QX + 4;       // tile cols: ix = c - 4
  static constexpr int IN_FLOATS = CI * 3 * TR * IP;
  static constexpr int W_FLOATS = CI * 3 * 25 * CO;
  static constexpr int RED_FLOATS = (KS - 1) * THREADS_USED * 64;
  static constexpr int SMEM_FLOATS = (IN_FLOATS + W_FLOATS) > RED_FLOATS ? (IN_FLOATS + W_FLOATS) : RED_FLOATS;
  static constexpr int SMEM_BYTES = SMEM_FLOATS * 4;
  static_assert(CO % 4 == 0 && DIN % 4 == 0 && 2 * RG + 2 <= TR && DIN + 4 <= IP && CI % KS == 0, "convT fwd tiling");
};

template <int CI, int CO, int DIN, int MINB, int KS = 1>
__global__ void __launch_bounds__(ConvTFwdCfg<CI, CO, DIN, KS>::THREADS, MINB) k_convT5_fwd(ConvTFwdParams p) {
  using G = ConvTFwdCfg<CI, CO, DIN, KS>;
  extern __shared__ __align__(128) float smem[];
  float* s_in = smem;
  float* s_w = smem + G::IN_FLOATS;
  const int tid = threadIdx.x;
  // even output slices use three kz taps, odd ones two: schedule the heavy (even) slices of all blocks first
  constexpr int NEV = (G::DOUT + 1) / 2, NOD = G::DOUT / 2;
  int z, b;
  if ((int)blockIdx.x < p.n * NEV) {
    z = 2 * ((int)blockIdx.x % NEV);
    b = (int)blockIdx.x / NEV;
  } else {
    const int i = (int)blockIdx.x - p.n * NEV;
    z = 2 * (i % NOD) + 1;
    b = i / NOD;
  }
  const int pz = z & 1;
  const int NT = pz ? 2 : 3;  // kz = pz + 2t, input slice iz = (z - pz) / 2 - t

  // ---- stage: three input slices with a zero halo, and the weight taps of this z parity
  {
    const float* in_b = p.in + (size_t)b * CI * DIN * DIN * G::IN_PITCH;
    constexpr int NV = G::IP / 4;
    for (int i = tid; i < CI * 3 * G::TR * NV; i += G::THREADS) {
      int q = i;
      const int cv = q % NV; q /= NV;
      const int r = q % G::TR; q /= G::TR;
      const int t = q % 3; q /= 3;
      const int ci = q;
      const int iz = ((z - pz) >> 1) - t, iy = r - 2, ix = 4 * cv - 4;
      const bool ok = t < NT && iz >= 0 && iz < DIN && iy >= 0 && iy < DIN && ix >= 0 && ix < DIN;
      tma::cp_async16(s_in + ((ci * 3 + t) * G::TR + r) * G::IP + 4 * cv,
                      ok ? in_b + (((size_t)ci * DIN + iz) * DIN + iy) * G::IN_PITCH + ix : in_b, ok);
    }
    constexpr int TAPV = 25 * CO / 4;
    for (int i = tid; i < CI * 3 * TAPV; i += G::THREADS) {
      int q = i;
      const int v4 = q % TAPV; q /= TAPV;
      const int t = q % 3; q /= 3;
      const int ci = q;
      if (t < NT) tma::cp_async16(s_w + 4 * i, p.Wp + ((size_t)(ci * 5 + pz + 2 * t) * 25) * CO + 4 * v4);
    }
    tma::cp_async_wait_all();
  }
  __syncthreads();
  const bool active = tid < G::THREADS_USED * KS;
  if (KS == 1 && !active) return;
  const int kgrp = active ? tid / G::THREADS_USED : 0, local = tid - kgrp * G::THREADS_USED;
  int r = active ? local : 0;
  const int q = r % G::QX; r /= G::QX;
  const int pr = r % (2 * G::RG); r /= (2 * G::RG);
  const int cog = r;
  const int rg = pr >> 1, sub = pr & 1;
  const int y = 4 * rg + sub;      // rows y and y + 2 (parity `sub`)
  const int NKY = sub ? 2 : 3;     // ky = sub + 2u, input rows 2rg - u (row y) and 2rg - u + 1 (row y + 2)

  p2 acc2[2][2][8];   // [row of the pair][co pair][x]: fma.rn.f32x2 over output-channel pairs
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc2[a][c][j] = p2_bcast(0.f);

#pragma unroll 1
  for (int ci = kgrp * (CI / KS); ci < (active ? (kgrp + 1) * (CI / KS) : 0); ++ci) {
#pragma unroll 1
    for (int t = 0; t < NT; ++t) {
      // input slice of this tap outside the tensor (first / last output slices): all zeros, nothing to add (uniform)
      const int iz_t = ((z - pz) >> 1) - t;
      if (iz_t < 0 || iz_t >= DIN) continue;
      // tile rows 2rg .. 2rg+3  (iy = 2rg-2 .. 2rg+1), columns 4q+2 .. 4q+7  (ix = 4q-2 .. 4q+3)
      const float* base = s_in + ((ci * 3 + t) * G::TR + 2 * rg) * G::IP + 4 * q + 2;
      p2 R[4][6];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const float2 lo = *reinterpret_cast<const float2*>(base + k * G::IP);
        const float4 hi = *reinterpret_cast<const float4*>(base + k * G::IP + 2);
        R[k][0] = p2_bcast(lo.x); R[k][1] = p2_bcast(lo.y); R[k][2] = p2_bcast(hi.x);
        R[k][3] = p2_bcast(hi.y); R[k][4] = p2_bcast(hi.z); R[k][5] = p2_bcast(hi.w);
      }
      const float* wt = s_w + ((ci * 3 + t) * 25) * CO + cog * 4;
#pragma unroll
      for (int u = 0; u < 3; ++u) {
        if (u < NKY) {
          const int ky = sub + 2 * u;
#pragma unroll
          for (int kx = 0; kx < 5; ++kx) {
            p2 w[2];
            p2_ld2(wt + (ky * 5 + kx) * CO, w[0], w[1]);
            const int h = kx >> 1;
#pragma unroll
            for (int c = 0; c < 2; ++c) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                if ((kx & 1) == 0) {
                  p2_fma(acc2[0][c][2 * j], w[c], R[2 - u][j + 2 - h]);
                  p2_fma(acc2[1][c][2 * j], w[c], R[3 - u][j + 2 - h]);
                } else {
                  p2_fma(acc2[0][c][2 * j + 1], w[c], R[2 - u][j + 2 - h]);
                  p2_fma(acc2[1][c][2 * j + 1], w[c], R[3 - u][j + 2 - h]);
                }
              }
            }
          }
        }
      }
    }
  }
  float acc[2][4][8];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[a][c][j] = (c & 1) ? p2_hi(acc2[a][c >> 1][j]) : p2_lo(acc2[a][c >> 1][j]);
  if constexpr (KS > 1) {
    // combine the channel-split groups: groups 1.. hand their sums to group 0 (fixed order)
    __syncthreads();                       // every group is done reading the staged tile
    float* red = smem;
    if (active && kgrp > 0) {
#pragma unroll
      for (int a = 0; a < 2; ++a)
#pragma unroll
        for (int c = 0; c < 4; ++c)
#pragma unroll
          for (int j = 0; j < 8; ++j) red[((kgrp - 1) * 64 + (a * 4 + c) * 8 + j) * G::THREADS_USED + local] = acc[a][c][j];
    }
    __syncthreads();
    if (!active || kgrp > 0) return;
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          float sacc = acc[a][c][j];
#pragma unroll
          for (int g2 = 0; g2 < KS - 1; ++g2) sacc += red[(g2 * 64 + (a * 4 + c) * 8 + j) * G::THREADS_USED + local];
          acc[a][c][j] = sacc;
        }
  }
  // ---- epilogue: bias + ReLU, columns >= DOUT of a padded row are written as zero
  constexpr size_t out_cs = (size_t)G::DOUT * G::DOUT * G::OUT_PITCH;
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    const int oy = y + 2 * a;
    if (oy >= G::DOUT) continue;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      const int co = cog * 4 + c;
      const float bb = __ldg(p.bias + co);
      float v[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float t = acc[a][c][j] + bb;
        v[j] = (8 * q + j < G::DOUT && t > 0.f) ? t : 0.f;
      }
      float* o = p.out + ((size_t)b * CO + co) * out_cs + ((size_t)z * G::DOUT + oy) * G::OUT_PITCH + 8 * q;
      *reinterpret_cast<float4*>(o) = make_float4(v[0], v[1], v[2], v[3]);
      if (8 * q + 4 < G::OUT_PITCH) *reinterpret_cast<float4*>(o + 4) = make_float4(v[4], v[5], v[6], v[7]);
    }
  }
}

// ---------------------------------------------------------------------------
// data gradient (stride-2 correlation).  One CTA per (block, z, row band); the
// five kz taps are split over five thread groups whose partial sums are combined
// through shared memory (the layer has too few outputs to fill the GPU
// otherwise).  Thread tile: 8 ci x 4 x x rows (y, y+1) = 64 accumulators.
// ---------------------------------------------------------------------------
struct ConvTDgradParams {
  const float* g;     // [n][CG][DG][DG][GP]   DG = 2*DIN + 3
  float* dx;          // [n][CX][DIN][DIN][DIN]
  const float* Wp;    // PACK_CONVT_DGRAD [cg][kz][ky][kx][cx]
  const float* add;   // like dx or null
  const float* mask;  // like dx or null (dx = mask > 0 ? v : 0)
  int32_t n;
};

template <int CG, int CX, int DIN, int TY, int CGC>
struct ConvTDgradCfg {
  static constexpr int DG = 2 * DIN + 3, GP = (DG + 3) / 4 * 4;
  static constexpr int XG = DIN / 4, NYP = TY / 2, CXG = CX / 8;
  static constexpr int POS = XG * NYP * CXG;
  static constexpr int THREADS_USED = POS * 5;
  static constexpr int THREADS = (THREADS_USED + 31) / 32 * 32;
  static constexpr int GR = 2 * TY + 3;                     // staged g rows
  static constexpr int GPS = GP + 4;                        // staged pitch (cols .. 8*xg+11 readable)
  static constexpr int G_FLOATS = CGC * 5 * GR * GPS;
  static constexpr int W_FLOATS = CGC * 125 * CX;
  static constexpr int RED_FLOATS = 4 * POS * 64;           // kz groups 1..4 hand their sums to group 0
  static constexpr int STAGE = G_FLOATS + W_FLOATS;         // one of two cp.async stages
  static constexpr int SMEM_FLOATS = 2 * STAGE > RED_FLOATS ? 2 * STAGE : RED_FLOATS;
  static constexpr int SMEM_BYTES = SMEM_FLOATS * 4;
  static constexpr int BANDS = DIN / TY;
  static_assert(DIN % 4 == 0 && DIN % TY == 0 && TY % 2 == 0 && CX % 8 == 0 && CG % CGC == 0, "convT dgrad tiling");
};

template <int CG, int CX, int DIN, int TY, int CGC, int MINB>
__global__ void __launch_bounds__(ConvTDgradCfg<CG, CX, DIN, TY, CGC>::THREADS, MINB) k_convT5_dgrad(ConvTDgradParams p) {
  using G = ConvTDgradCfg<CG, CX, DIN, TY, CGC>;
  extern __shared__ __align__(128) float smem[];
  const int tid = threadIdx.x;
  int t = blockIdx.x;
  const int band = t % G::BANDS; t /= G::BANDS;
  const int z = t % DIN; t /= DIN;
  const int b = t;
  const int y0 = band * TY;
  const bool active = tid < G::THREADS_USED;
  int r = active ? tid : 0;
  const int pos = r % G::POS;
  const int kz = r / G::POS;
  r = pos;
  const int xg = r % G::XG; r /= G::XG;
  const int yp = r % G::NYP; r /= G::NYP;
  const int cxg = r;

  p2 acc2[2][4][4];   // [row][cx pair][x]: fma.rn.f32x2 over input-channel pairs
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc2[a][c][j] = p2_bcast(0.f);

  const float* g_b = p.g + (size_t)b * CG * G::DG * G::DG * G::GP;
  // two-stage cp.async pipeline over chunks of CGC gradient channels: chunk c+1 streams in while chunk c is consumed.
  // A thread copies the same tile positions for every chunk, so the (channel, slice, row, column) decomposition of
  // its copy indices is done once here; per chunk only the channel offset is added.
  constexpr int NV = G::GP / 4;
  constexpr int NCOPY = CGC * 5 * G::GR * NV;
  constexpr int PER_T = (NCOPY + G::THREADS - 1) / G::THREADS;
  int soff[PER_T], goff[PER_T];
#pragma unroll
  for (int u = 0; u < PER_T; ++u) {
    const int i = tid + u * G::THREADS;
    int q = i < NCOPY ? i : 0;
    const int cv = q % NV; q /= NV;
    const int rr = q % G::GR; q /= G::GR;
    const int s5 = q % 5; q /= 5;
    const int c = q;
    soff[u] = i < NCOPY ? ((c * 5 + s5) * G::GR + rr) * G::GPS + 4 * cv : -1;
    goff[u] = ((c * G::DG + 2 * z + s5) * G::DG + 2 * y0 + rr) * G::GP + 4 * cv;
  }
  auto stage = [&](int chunk) {
    float* sg = smem + (chunk & 1) * G::STAGE;
    float* sw = sg + G::G_FLOATS;
    const int c0 = chunk * CGC;
    const float* gc = g_b + (size_t)c0 * G::DG * G::DG * G::GP;
#pragma unroll
    for (int u = 0; u < PER_T; ++u)
      if (soff[u] >= 0) tma::cp_async16(sg + soff[u], gc + goff[u]);
    const float* src = p.Wp + (size_t)c0 * 125 * CX;
    for (int i = tid; i < G::W_FLOATS / 4; i += G::THREADS) tma::cp_async16(sw + 4 * i, src + 4 * i);
  };
  constexpr int NCHUNK = CG / CGC;
  stage(0);
  tma::cp_async_wait_all();
  __syncthreads();
#pragma unroll 1
  for (int chunk = 0; chunk < NCHUNK; ++chunk) {
    if (chunk + 1 < NCHUNK) stage(chunk + 1);
    const float* s_g = smem + (chunk & 1) * G::STAGE;
    const float* s_w = s_g + G::G_FLOATS;
    if (active) {
#pragma unroll 1
      for (int c = 0; c < CGC; ++c) {
#pragma unroll 1
        for (int ky = 0; ky < 5; ++ky) {
          const float* ra = s_g + ((c * 5 + kz) * G::GR + 4 * yp + ky) * G::GPS + 8 * xg;
          p2 A[2][12];
#pragma unroll
          for (int a = 0; a < 2; ++a) {
#pragma unroll
            for (int v = 0; v < 3; ++v) {
              const float4 f = *reinterpret_cast<const float4*>(ra + a * 2 * G::GPS + 4 * v);
              A[a][4 * v] = p2_bcast(f.x); A[a][4 * v + 1] = p2_bcast(f.y);
              A[a][4 * v + 2] = p2_bcast(f.z); A[a][4 * v + 3] = p2_bcast(f.w);
            }
          }
          const float* wk = s_w + ((c * 5 + kz) * 5 + ky) * 5 * CX + cxg * 8;
#pragma unroll
          for (int kx = 0; kx < 5; ++kx) {
            p2 w[4];
            p2_load_w8(wk + kx * CX, w);
#pragma unroll
            for (int cc = 0; cc < 4; ++cc)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                p2_fma(acc2[0][cc][j], w[cc], A[0][2 * j + kx]);
                p2_fma(acc2[1][cc][j], w[cc], A[1][2 * j + kx]);
              }
          }
        }
      }
    }
    tma::cp_async_wait_all();
    __syncthreads();   // next chunk has landed; everyone is done with this one
  }
  float acc[2][8][4];
#pragma unroll
  for (int a = 0; a < 2; ++a)
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[a][c][j] = (c & 1) ? p2_hi(acc2[a][c >> 1][j]) : p2_lo(acc2[a][c >> 1][j]);
  // ---- combine the five kz groups (fixed order), add / mask, store
  __syncthreads();
  float* red = smem;
  if (active && kz > 0) {
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int c = 0; c < 8; ++c)
#pragma unroll
        for (int j = 0; j < 4; ++j) red[((kz - 1) * 64 + (a * 8 + c) * 4 + j) * G::POS + pos] = acc[a][c][j];
  }
  __syncthreads();
  if (!active || kz != 0) return;
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    const int oy = y0 + 2 * yp + a;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float s = acc[a][c][j];
#pragma unroll
        for (int k = 0; k < 4; ++k) s += red[(k * 64 + (a * 8 + c) * 4 + j) * G::POS + pos];
        v[j] = s;
      }
      const size_t o = ((((size_t)b * CX + cxg * 8 + c) * DIN + z) * DIN + oy) * DIN + 4 * xg;
      if (p.add) {
        const float4 ad = *reinterpret_cast<const float4*>(p.add + o);
        v[0] += ad.x; v[1] += ad.y; v[2] += ad.z; v[3] += ad.w;
      }
      if (p.mask) {
        const float4 m = *reinterpret_cast<const float4*>(p.mask + o);
        v[0] = m.x > 0.f ? v[0] : 0.f; v[1] = m.y > 0.f ? v[1] : 0.f;
        v[2] = m.z > 0.f ? v[2] : 0.f; v[3] = m.w > 0.f ? v[3] : 0.f;
      }
      *reinterpret_cast<float4*>(p.dx + o) = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

// ---------------------------------------------------------------------------
// weight gradient.  Thread = (co, kz, ky) owns dW[CIB ci][co][kz][ky][5 kx] in
// registers for the whole kernel; persistent CTAs walk over items (block, z, row
// band); g rows are per-lane LDS.128 in a bank-conflict-free layout (consecutive
// (kz,ky) taps 16 bytes apart modulo 128), x rows are warp-broadcast.
// grid.y = (CO / 8) * (CI / CIB) channel groups.
// ---------------------------------------------------------------------------
struct ConvTWgradParams {
  const float* x;    // [n][CI][DIN][DIN][DIN]
  const float* g;    // [n][CO][DG][DG][GP]
  float* partial;    // [gridDim.y][gridDim.x][CIB*8*125]
  int32_t n;
};

template <int CI, int CO, int DIN, int TYB, int CIB>
struct ConvTWgradCfg {
  static constexpr int DG = 2 * DIN + 3, GP = (DG + 3) / 4 * 4;
  static constexpr int THREADS = 224;            // 200 used: (co 8, kz 5, ky 5)
  static constexpr int GR = 2 * TYB + 3;         // staged g rows per slice
  // tap (kz,ky) -> float offset T(kz,ky) with T = 4 (kz*5+ky) (mod 32); co stride = 4*25 (mod 32) = 4
  static constexpr int ROWP = (GP % 32 <= 4) ? GP / 32 * 32 + 4 : GP / 32 * 32 + 36;   // = 4 (mod 32), >= GP
  static constexpr int S0 = GR * ROWP;
  static constexpr int SLICE = S0 + ((20 - S0 % 32) + 32) % 32;                        // = 20 (mod 32)
  static constexpr int C0 = 5 * SLICE;
  static constexpr int CSTR = C0 + ((4 - C0 % 32) + 32) % 32;                          // = 4 (mod 32)
  static constexpr int G_FLOATS = 8 * CSTR;
  static constexpr int X_FLOATS = CIB * TYB * DIN;
  static constexpr int SMEM_BYTES = (G_FLOATS + X_FLOATS) * 4;
  static constexpr int BANDS = DIN / TYB;
  static constexpr int OUT_FLOATS = CIB * 8 * 125;
  static constexpr int GROUPS = (CO / 8) * (CI / CIB);
  static_assert(DIN % 4 == 0 && DIN % TYB == 0 && CO % 8 == 0 && CI % CIB == 0, "convT wgrad tiling");
};

template <int CI, int CO, int DIN, int TYB, int CIB, int MINB>
__global__ void __launch_bounds__(224, MINB) k_convT5_wgrad(ConvTWgradParams p) {
  using G = ConvTWgradCfg<CI, CO, DIN, TYB, CIB>;
  extern __shared__ __align__(128) float smem[];
  float* s_g = smem;
  float* s_x = smem + G::G_FLOATS;
  const int tid = threadIdx.x;
  const int cog = blockIdx.y % (CO / 8), cig = blockIdx.y / (CO / 8);
  const bool active = tid < 200;
  const int tt = active ? tid : 0;
  const int ky = tt % 5, kz = (tt / 5) % 5, co = tt / 25;

  static_assert(CIB % 2 == 0, "input channels are processed in pairs (fma.rn.f32x2)");
  p2 acc2[CIB / 2][5];   // [ci pair][kx]
#pragma unroll
  for (int c = 0; c < CIB / 2; ++c)
#pragma unroll
    for (int k = 0; k < 5; ++k) acc2[c][k] = p2_bcast(0.f);

  const int items = p.n * DIN * G::BANDS;
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    int q = item;
    const int band = q % G::BANDS; q /= G::BANDS;
    const int z = q % DIN; q /= DIN;
    const int b = q;
    const int y0 = band * TYB;
    __syncthreads();
    {
      constexpr int NV = G::GP / 4;
      const float* gb = p.g + ((size_t)b * CO + cog * 8) * G::DG * G::DG * G::GP;
      for (int i = tid; i < 8 * 5 * G::GR * NV; i += 224) {
        int t = i;
        const int cv = t % NV; t /= NV;
        const int rr = t % G::GR; t /= G::GR;
        const int s = t % 5; t /= 5;
        const int c = t;
        tma::cp_async16(s_g + c * G::CSTR + s * G::SLICE + rr * G::ROWP + 4 * cv,
                        gb + (((size_t)c * G::DG + 2 * z + s) * G::DG + 2 * y0 + rr) * G::GP + 4 * cv);
      }
      constexpr int XV = DIN / 4;
      const float* xb = p.x + ((size_t)b * CI + cig * CIB) * DIN * DIN * DIN;
      for (int i = tid; i < CIB * TYB * XV; i += 224) {
        int t = i;
        const int cv = t % XV; t /= XV;
        const int rr = t % TYB; t /= TYB;
        const int c = t;
        // s_x[c/2][rr][x][c&1]: channel pairs interleaved (one LDS.128 = the operand pairs of two x)
        const float* sx = xb + (((size_t)c * DIN + z) * DIN + y0 + rr) * DIN + 4 * cv;
        float* d = s_x + (((c >> 1) * TYB + rr) * DIN + 4 * cv) * 2 + (c & 1);
        tma::cp_async4(d, sx); tma::cp_async4(d + 2, sx + 1); tma::cp_async4(d + 4, sx + 2); tma::cp_async4(d + 6, sx + 3);
      }
      tma::cp_async_wait_all();
    }
    __syncthreads();
    if (active) {
      const float* gk = s_g + co * G::CSTR + kz * G::SLICE + ky * G::ROWP;
#pragma unroll 1
      for (int rr = 0; rr < TYB; ++rr) {
#pragma unroll 1
        for (int xq = 0; xq < DIN / 4; ++xq) {
          const float* gr = gk + 2 * rr * G::ROWP + 8 * xq;
          p2 gv[12];
#pragma unroll
          for (int v = 0; v < 3; ++v) {
            const float4 f = *reinterpret_cast<const float4*>(gr + 4 * v);
            gv[4 * v] = p2_bcast(f.x); gv[4 * v + 1] = p2_bcast(f.y);
            gv[4 * v + 2] = p2_bcast(f.z); gv[4 * v + 3] = p2_bcast(f.w);
          }
#pragma unroll
          for (int c = 0; c < CIB / 2; ++c) {
            p2 xv[4];
            const float* xr = s_x + ((c * TYB + rr) * DIN + 4 * xq) * 2;
            p2_ld2(xr, xv[0], xv[1]);
            p2_ld2(xr + 4, xv[2], xv[3]);
#pragma unroll
            for (int kx = 0; kx < 5; ++kx)
#pragma unroll
              for (int j = 0; j < 4; ++j) p2_fma(acc2[c][kx], xv[j], gv[2 * j + kx]);
          }
        }
      }
    }
  }
  if (!active) return;
  // partial in the layout [ci_local][co_local][kz][ky][kx]
  float* out = p.partial + ((size_t)blockIdx.y * gridDim.x + blockIdx.x) * G::OUT_FLOATS;
#pragma unroll
  for (int c = 0; c < CIB; ++c)
#pragma unroll
    for (int kx = 0; kx < 5; ++kx)
      out[((c * 8 + co) * 25 + kz * 5 + ky) * 5 + kx] = (c & 1) ? p2_hi(acc2[c >> 1][kx]) : p2_lo(acc2[c >> 1][kx]);
}

// ---------------------------------------------------------------------------
// per-channel sums (bias gradients): partial[blockIdx.x][c] = sum over one
// (block, z-slice chunk) of g[b][c][...]; summed in fixed order by k_reduce_partials.
// ---------------------------------------------------------------------------
struct ChanSumFastParams {
  const float* g;   // [n][C][D][D][P]
  float* partial;   // [n*ZCH][C]
  int32_t n, C, D, P, ZCH;  // ZCH chunks along z
};
__global__ void __launch_bounds__(256) k_chansum_fast(ChanSumFastParams p) {
  __shared__ float sm[256];
  const int c = blockIdx.x % p.C;
  const int zc = (blockIdx.x / p.C) % p.ZCH;
  const int b = blockIdx.x / (p.C * p.ZCH);
  const int zlo = (int)((int64_t)p.D * zc / p.ZCH), zhi = (int)((int64_t)p.D * (zc + 1) / p.ZCH);
  const float* base = p.g + (((size_t)b * p.C + c) * p.D + zlo) * p.D * p.P;
  const int rows = (zhi - zlo) * p.D;
  const int pv = p.P / 4;
  float s = 0.f;
  for (int i = threadIdx.x; i < rows * pv; i += 256) {
    const int row = i / pv, v = i - row * pv;
    const float4 f = __ldg(reinterpret_cast<const float4*>(base + (size_t)row * p.P) + v);
    const int x = 4 * v;
    s += (x < p.D ? f.x : 0.f) + (x + 1 < p.D ? f.y : 0.f) + (x + 2 < p.D ? f.z : 0.f) + (x + 3 < p.D ? f.w : 0.f);
  }
  sm[threadIdx.x] = s;
  __syncthreads();
  for (int st = 128; st >= 1; st >>= 1) {
    if (threadIdx.x < st) sm[threadIdx.x] += sm[threadIdx.x + st];
    __syncthreads();
  }
  if (threadIdx.x == 0) p.partial[(size_t)(b * p.ZCH + zc) * p.C + c] = sm[0];
}

}  // namespace fast
}  // namespace nvf
