// Shared-memory tiled, register-blocked FP32 kernels for the k=4 stride-1
// convolutions of the NVF decoder's training path (conv1 / conv2 and their
// data gradients; utils/network.py:4702-4729 via F.conv3d, :687).
//
//   y[co,z,y,x] = sum_ci sum_k in[ci, z+kz-P, y+ky-P, x+kx-P] * Wp[ci][k][co]
//   forward:  P = 0, Wp = PACK_CONV_FWD,   epilogue  relu(acc + bias)
//   dgrad:    P = 3, Wp = PACK_CONV_DGRAD, epilogue  acc masked by (act > 0)
//
// CTA tile: (2*NZP) z-slices x TY rows x 4*XG columns x C output channels.
// Thread tile: 8 output channels x 4 x x 2 z (64 accumulators).  The input tile
// (CIC input channels at a time, halo included, zero-filled outside the tensor)
// and the matching weight chunk are staged in shared memory; every activation
// row fetched from shared memory (2 x LDS.128) feeds 8 co x 4 kx x 4 x FMAs for
// each of up to two output slices, weights are warp-broadcast LDS.128.
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"
#include "nvf_tma.cuh"

namespace nvf {
namespace fast {

struct ConvS1Params {
  const float* in;    // [n][CI][DIN][DIN][IN_PITCH]
  float* out;         // [n][CO][DOUT][DOUT][OUT_PITCH]
  float* out2;        // optional second copy of the output (same layout) or null
  const float* Wp;    // packed [ci][kz][ky][kx][co]
  const float* bias;  // [CO] or null
  const float* mask;  // same layout as out or null: v = mask > 0 ? v : 0
  int32_t n, act;     // act: 0 none, 1 relu, 2 sigmoid
};

// XSH: extra left shift of the staged columns (tile column = ix + PAD + XSH).  The TMA unit needs the
// innermost start coordinate of a box to be 16-byte aligned (x0 = -(PAD + XSH) must be a multiple of 4:
// probed on B200, scripts/probe/tma_probe.cu), so the PAD = 3 data-gradient tiles use XSH = 1.
template <int K, int CI, int C, int DIN, int PAD, int XG, int TY, int NZP, int CIC, int XSH = 0, int COTP = 0>
struct ConvS1Cfg {
  // output channels per thread; COTP > 0 overrides (smaller tiles = more threads for the small layers)
  static constexpr int COT = COTP > 0 ? COTP : (C >= 8 ? 8 : C);
  static constexpr int DOUT = DIN + 2 * PAD - (K - 1);
  static constexpr int IN_PITCH = (DIN + 3) / 4 * 4, OUT_PITCH = (DOUT + 3) / 4 * 4;
  static constexpr int NV = IN_PITCH / 4;                 // float4 per global input row
  static constexpr int COG = C / COT;                     // output-channel groups
  static constexpr int THREADS_USED = XG * TY * NZP * COG;
  static constexpr int THREADS = (THREADS_USED + 31) / 32 * 32;
  static constexpr int TZ = 2 * NZP;                      // output slices per tile
  static constexpr int TZI = TZ + K - 1, TYI = TY + K - 1;
  static constexpr int PI = 4 * XG + 4 + (XSH ? 4 : 0);   // input row pitch (x0 .. x0+7(+XSH) readable)
  static constexpr int IN_FLOATS = CIC * TZI * TYI * PI;
  static constexpr int W_FLOATS = CIC * K * K * K * C;
  static constexpr int SMEM_BYTES = (IN_FLOATS + W_FLOATS) * 4;
  // TMA variant: two stages of {input tile, weight chunk}, each part 128-byte aligned, + two mbarriers
  static constexpr int IN_AL = (IN_FLOATS + 31) / 32 * 32, W_AL = (W_FLOATS + 31) / 32 * 32, STAGE = IN_AL + W_AL;
  static constexpr int SMEM_BYTES_TMA = 2 * STAGE * 4 + 16;
  static constexpr int TILES_Z = (DOUT + TZ - 1) / TZ, TILES_Y = (DOUT + TY - 1) / TY;
  static_assert(C % COT == 0 && CI % CIC == 0 && (K == 3 || K == 4), "channel blocking");
  static_assert(4 * XG >= DOUT && 4 * XG <= OUT_PITCH, "x groups cover one output row");
  static_assert(PAD % 4 != 0 || 4 * NV <= PI, "staged row fits the tile pitch");
};
// One staged chunk of CIC input channels: accumulate into the thread's register tile.
// s_in: [CIC][TZI][TYI][PI] input tile (halo included), s_w: [CIC][K][K][K][C] weights.
// eight consecutive tile columns starting at r[XSH] (r 16-byte aligned) as broadcast pairs
template <int XSH>
__device__ __forceinline__ void load_row8_p2(const float* r, p2 (&a)[8]) {
  const float4 lo = *reinterpret_cast<const float4*>(r);
  const float4 hi = *reinterpret_cast<const float4*>(r + 4);
  if constexpr (XSH == 0) {
    a[0] = p2_bcast(lo.x); a[1] = p2_bcast(lo.y); a[2] = p2_bcast(lo.z); a[3] = p2_bcast(lo.w);
    a[4] = p2_bcast(hi.x); a[5] = p2_bcast(hi.y); a[6] = p2_bcast(hi.z); a[7] = p2_bcast(hi.w);
  } else {
    static_assert(XSH == 0 || XSH == 1, "XSH");
    const float4 h2 = *reinterpret_cast<const float4*>(r + 8);
    a[0] = p2_bcast(lo.y); a[1] = p2_bcast(lo.z); a[2] = p2_bcast(lo.w); a[3] = p2_bcast(hi.x);
    a[4] = p2_bcast(hi.y); a[5] = p2_bcast(hi.z); a[6] = p2_bcast(hi.w); a[7] = p2_bcast(h2.x);
  }
}

template <class G, int K, int C, int CIC, int COT, int CP, bool PAIR, int XSH>
__device__ __forceinline__ void conv_s1_chunk(const float* __restrict__ s_in, const float* __restrict__ s_w, int zp, int ty,
                                              int xg, int cg, p2 (&acc2)[2][CP][4], float (&acc)[2][COT][4]) {
#pragma unroll 1
  for (int ci = 0; ci < CIC; ++ci) {
#pragma unroll 1
    for (int ky = 0; ky < K; ++ky) {
      const float* rowp = s_in + ((ci * G::TZI + 2 * zp) * G::TYI + ty + ky) * G::PI + 4 * xg;
      const float* wp = s_w + ((ci * K) * K + ky) * K * C + cg * COT;
      if constexpr (PAIR) {
        p2 a0[8], a1[8];
        load_row8_p2<XSH>(rowp, a0);
#pragma unroll
        for (int kz = 0; kz < K; ++kz) {
          load_row8_p2<XSH>(rowp + (kz + 1) * G::TYI * G::PI, a1);
#pragma unroll
          for (int kx = 0; kx < K; ++kx) {
            const float* wk = wp + (kz * K * K + kx) * C;
            p2 w[CP];
            if constexpr (COT == 8) {
              p2_ld2(wk, w[0], w[1]);
              p2_ld2(wk + 4, w[2 % CP], w[3 % CP]);
            } else if constexpr (COT == 4) {
              p2_ld2(wk, w[0], w[1 % CP]);
            } else {
#pragma unroll
              for (int c = 0; c < CP; ++c) w[c] = p2_make(wk[2 * c], wk[2 * c + 1]);
            }
#pragma unroll
            for (int c = 0; c < CP; ++c) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                p2_fma(acc2[0][c][j], w[c], a0[j + kx]);
                p2_fma(acc2[1][c][j], w[c], a1[j + kx]);
              }
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) a0[i] = a1[i];
        }
      } else {
        float a0[8], a1[8];
        {
          const float4 lo = *reinterpret_cast<const float4*>(rowp);
          const float4 hi = *reinterpret_cast<const float4*>(rowp + 4);
          a0[0] = lo.x; a0[1] = lo.y; a0[2] = lo.z; a0[3] = lo.w;
          a0[4] = hi.x; a0[5] = hi.y; a0[6] = hi.z; a0[7] = hi.w;
        }
#pragma unroll
        for (int kz = 0; kz < K; ++kz) {
          {
            const float* r1 = rowp + (kz + 1) * G::TYI * G::PI;
            const float4 lo = *reinterpret_cast<const float4*>(r1);
            const float4 hi = *reinterpret_cast<const float4*>(r1 + 4);
            a1[0] = lo.x; a1[1] = lo.y; a1[2] = lo.z; a1[3] = lo.w;
            a1[4] = hi.x; a1[5] = hi.y; a1[6] = hi.z; a1[7] = hi.w;
          }
#pragma unroll
          for (int kx = 0; kx < K; ++kx) {
            const float* wk = wp + (kz * K * K + kx) * C;
            float w[COT];
#pragma unroll
            for (int c = 0; c < COT; ++c) w[c] = wk[c];
#pragma unroll
            for (int c = 0; c < COT; ++c) {
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                acc[0][c][j] = fmaf(w[c], a0[j + kx], acc[0][c][j]);
                acc[1][c][j] = fmaf(w[c], a1[j + kx], acc[1][c][j]);
              }
            }
          }
#pragma unroll
          for (int i = 0; i < 8; ++i) a0[i] = a1[i];
        }
      }
    }
  }
}


// TMA = true: the input tile is fetched by the TMA unit (cp.async.bulk.tensor.5d, out-of-bounds = conv halo =
// zero fill) and the weight chunk by a 1-D bulk copy, double buffered behind two mbarriers, so chunk ch+1
// streams in while the CTA computes on chunk ch.  TMA = false: cooperative register-staged copy (tmap unused).
template <int K, int CI, int C, int DIN, int PAD, int XG, int TY, int NZP, int CIC, int MINB, bool TMA, int COTP = 0>
__global__ void __launch_bounds__(ConvS1Cfg<K, CI, C, DIN, PAD, XG, TY, NZP, CIC, 0, COTP>::THREADS, MINB)
    k_conv_s1(const __grid_constant__ CUtensorMap tmap, ConvS1Params p) {
  constexpr int XSH = TMA ? (4 - PAD % 4) % 4 : 0;
  using G = ConvS1Cfg<K, CI, C, DIN, PAD, XG, TY, NZP, CIC, XSH, COTP>;
  constexpr int COT = G::COT;
  extern __shared__ __align__(128) float smem[];
  float* s_in = smem;
  float* s_w = smem + G::IN_FLOATS;
  const int tid = threadIdx.x;
  int t = blockIdx.x;
  const int tyi = t % G::TILES_Y; t /= G::TILES_Y;
  const int tzi = t % G::TILES_Z; t /= G::TILES_Z;
  const int b = t;
  const int z0 = tzi * G::TZ, y0 = tyi * TY;

  const bool active = tid < G::THREADS_USED;
  int r = active ? tid : 0;
  const int xg = r % XG; r /= XG;
  const int ty = r % TY; r /= TY;
  const int zp = r % NZP; r /= NZP;
  const int cg = r;

  // accumulators: output-channel PAIRS in 64-bit registers (fma.rn.f32x2) when COT is even
  constexpr bool PAIR = (COT % 2 == 0);
  constexpr int CP = PAIR ? COT / 2 : COT;
  p2 acc2[2][CP][4];
  float acc[2][COT][4];
#pragma unroll
  for (int a = 0; a < 2; ++a) {
#pragma unroll
    for (int c = 0; c < CP; ++c)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc2[a][c][j] = p2_bcast(0.f);
#pragma unroll
    for (int c = 0; c < COT; ++c)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[a][c][j] = 0.f;
  }

  if constexpr (TMA) {
    static_assert((G::W_FLOATS * 4) % 16 == 0, "bulk copy granularity");
    constexpr int NCH = CI / CIC;
    constexpr uint32_t BYTES = (uint32_t)(G::IN_FLOATS + G::W_FLOATS) * 4u;
    uint64_t* bar = reinterpret_cast<uint64_t*>(smem + 2 * G::STAGE);
    if (tid == 0) {
      tma::mbar_init(bar, 1);
      tma::mbar_init(bar + 1, 1);
      tma::fence_barrier_init();
    }
    __syncthreads();
    auto issue = [&](int ch) {
      float* dst = smem + (ch & 1) * G::STAGE;
      tma::mbar_arrive_expect_tx(bar + (ch & 1), BYTES);
      tma::load_5d(dst, &tmap, bar + (ch & 1), -(PAD + XSH), y0 - PAD, z0 - PAD, ch * CIC, b);
      tma::load_1d(dst + G::IN_AL, p.Wp + (size_t)ch * G::W_FLOATS, (uint32_t)G::W_FLOATS * 4u, bar + (ch & 1));
    };
    if (tid == 0) {
      issue(0);
      if (NCH > 1) issue(1);
    }
#pragma unroll 1
    for (int ch = 0; ch < NCH; ++ch) {
      tma::mbar_wait(bar + (ch & 1), (uint32_t)(ch >> 1) & 1u);
      const float* st = smem + (ch & 1) * G::STAGE;
      if (active) conv_s1_chunk<G, K, C, CIC, COT, CP, PAIR, XSH>(st, st + G::IN_AL, zp, ty, xg, cg, acc2, acc);
      if (ch + 2 < NCH) {
        __syncthreads();               // every thread is done reading this stage
        if (tid == 0) issue(ch + 2);
      }
    }
  } else {
  const float* in_b = p.in + (size_t)b * CI * DIN * DIN * G::IN_PITCH;
  constexpr int plane = DIN * G::IN_PITCH;

  for (int c0 = 0; c0 < CI; c0 += CIC) {
    __syncthreads();
    // ---- stage the input tile (zero fill outside the tensor) and the weight chunk.
    // Global rows are read as aligned float4 and written at column PAD + ix of the tile row.
    constexpr int ROWS = CIC * G::TZI * G::TYI;
    for (int i = tid; i < ROWS * G::NV; i += G::THREADS) {
      const int row = i / G::NV, xv = i - row * G::NV;
      int q = row;
      const int ry = q % G::TYI; q /= G::TYI;
      const int sz = q % G::TZI; q /= G::TZI;
      const int ci = q;
      const int iy = y0 + ry - PAD, iz = z0 + sz - PAD;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (iy >= 0 && iy < DIN && iz >= 0 && iz < DIN)
        v = __ldg(reinterpret_cast<const float4*>(in_b + (size_t)(c0 + ci) * DIN * plane + (size_t)iz * plane +
                                                   iy * G::IN_PITCH) + xv);
      float* d = s_in + row * G::PI + PAD + 4 * xv;
      if (PAD % 4 == 0) {
        *reinterpret_cast<float4*>(d) = v;
      } else {
        const float e[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (PAD + 4 * xv + j < G::PI) d[j] = (4 * xv + j < DIN) ? e[j] : 0.f;
      }
    }
    // halo columns left of the data and right of it
    constexpr int RPAD = G::PI - (PAD + 4 * G::NV) > 0 ? G::PI - (PAD + 4 * G::NV) : 0;
    if constexpr (PAD + RPAD > 0) {
      for (int i = tid; i < ROWS * (PAD + RPAD); i += G::THREADS) {
        const int row = i / (PAD + RPAD), c = i - row * (PAD + RPAD);
        s_in[row * G::PI + (c < PAD ? c : 4 * G::NV + c)] = 0.f;
      }
    }
    {
      const float* src = p.Wp + (size_t)c0 * K * K * K * C;
      if (G::W_FLOATS % 4 == 0) {
        for (int i = tid; i < G::W_FLOATS / 4; i += G::THREADS)
          reinterpret_cast<float4*>(s_w)[i] = __ldg(reinterpret_cast<const float4*>(src) + i);
      } else {
        for (int i = tid; i < G::W_FLOATS; i += G::THREADS) s_w[i] = __ldg(src + i);
      }
    }
    __syncthreads();
    if (active) conv_s1_chunk<G, K, C, CIC, COT, CP, PAIR, XSH>(s_in, s_w, zp, ty, xg, cg, acc2, acc);
  }
  }
  if constexpr (PAIR) {
#pragma unroll
    for (int a = 0; a < 2; ++a)
#pragma unroll
      for (int c = 0; c < COT; ++c)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[a][c][j] = (c & 1) ? p2_hi(acc2[a][c >> 1][j]) : p2_lo(acc2[a][c >> 1][j]);
  }
  if (!active) return;
  // ---- epilogue
  const int oy = y0 + ty, ox = 4 * xg;
  if (oy >= G::DOUT) return;
  constexpr size_t out_cs = (size_t)G::DOUT * G::DOUT * G::OUT_PITCH;
#pragma unroll
  for (int a = 0; a < 2; ++a) {
    const int oz = z0 + 2 * zp + a;
    if (oz >= G::DOUT) continue;
#pragma unroll
    for (int c = 0; c < COT; ++c) {
      const int co = cg * COT + c;
      const size_t o = ((size_t)b * C + co) * out_cs + ((size_t)oz * G::DOUT + oy) * G::OUT_PITCH + ox;
      const float bb = p.bias ? __ldg(p.bias + co) : 0.f;
      float v[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[j] = acc[a][c][j] + bb;
        if (p.act == 1) v[j] = v[j] > 0.f ? v[j] : 0.f;
        else if (p.act == 2) v[j] = sigmoidf(v[j]);
      }
      if (p.mask) {
        const float4 m = *reinterpret_cast<const float4*>(p.mask + o);
        v[0] = m.x > 0.f ? v[0] : 0.f; v[1] = m.y > 0.f ? v[1] : 0.f;
        v[2] = m.z > 0.f ? v[2] : 0.f; v[3] = m.w > 0.f ? v[3] : 0.f;
      }
      // columns >= DOUT of a padded row are never consumed; keep them zero
#pragma unroll
      for (int j = 0; j < 4; ++j)
        if (ox + j >= G::DOUT) v[j] = 0.f;
      *reinterpret_cast<float4*>(p.out + o) = make_float4(v[0], v[1], v[2], v[3]);
      if (p.out2) *reinterpret_cast<float4*>(p.out2 + o) = make_float4(v[0], v[1], v[2], v[3]);
    }
  }
}

// ---------------------------------------------------------------------------
// Weight gradient of the k=4 stride-1 convolutions:
//   dW[co][ci][kz][ky][kx] = sum_{b,z,y,x} g[b][co][z][y][x] * a[b][ci][z+kz][y+ky][x+kx]
//   db[co]                 = sum g[b][co][...]
// Split-K over positions: persistent CTAs walk over items (block, z, row band),
// stage the g band and the four matching a bands in shared memory, and every
// thread OWNS 64 outputs dW[8 co][ci][kz][2 ky][4 kx] in registers for the whole
// kernel (thread = (co group, ci, kz, ky pair), NSET position sets per CTA share
// the rows of a band).  g rows are warp-broadcast LDS.128, a rows per-lane
// LDS.128 laid out bank-conflict free.  Each CTA writes ONE partial result;
// k_reduce_partials sums them in fixed order (deterministic, no atomics).
// ---------------------------------------------------------------------------
struct WgradS1Params {
  const float* g;    // [n][C][DG][DG][GP]
  const float* a;    // [n][C][DA][DA][APG]   DA = DG + 3
  float* partial;    // [gridDim.x][C*C*64 + C]
  int32_t n;
};

template <int C, int DG, int TYG>
struct WgradS1Cfg {
  static constexpr int DA = DG + 3;
  static constexpr int GP = (DG + 3) / 4 * 4, APG = (DA + 3) / 4 * 4;  // global pitches
  static constexpr int THREADS = 256;
  static constexpr int SET_THREADS = C * 8 * (C / 8);                  // (cog, ci, kz, kyp)
  static constexpr int NSET = THREADS / SET_THREADS;
  static constexpr int ROWS_PER_SET = TYG / NSET;
  static constexpr int XQ = DG / 4;
  // smem a tile [C][4][TYG+3][AP]: AP = 8 (mod 16), plane stride = 4 (mod 32) floats -> the 8 lanes
  // (kyp, kz) of a quarter warp hit 8 distinct 16-byte bank groups
  static constexpr int AP = (APG % 16 <= 8) ? APG / 16 * 16 + 8 : APG / 16 * 16 + 24;
  static constexpr int ZS0 = (TYG + 3) * AP;
  static constexpr int ZSA = ZS0 + ((4 - ZS0 % 32) + 32) % 32;
  static constexpr int A_FLOATS = C * 4 * ZSA;
  static constexpr int G_FLOATS = C * TYG * GP;
  static constexpr int NW = C * C * 64;
  static constexpr int OUT_FLOATS = NW + C;
  static constexpr int RED_FLOATS = NSET > 1 ? NSET * NW : 0;
  static constexpr int SMEM_FLOATS = (A_FLOATS + G_FLOATS) > RED_FLOATS ? (A_FLOATS + G_FLOATS) : RED_FLOATS;
  static constexpr int SMEM_BYTES = SMEM_FLOATS * 4;
  static constexpr int BANDS = DG / TYG;
  static_assert(DG % 4 == 0 && DG % TYG == 0 && TYG % NSET == 0 && NSET >= 1, "wgrad tiling");
  static_assert(THREADS % SET_THREADS == 0, "wgrad sets");
};

template <int C, int DG, int TYG, int MINB>
__global__ void __launch_bounds__(256, MINB) k_wgrad4_s1(WgradS1Params p) {
  using G = WgradS1Cfg<C, DG, TYG>;
  extern __shared__ __align__(128) float smem[];
  float* s_a = smem;
  float* s_g = smem + G::A_FLOATS;
  const int tid = threadIdx.x;
  const int set = tid / G::SET_THREADS;
  int r = tid % G::SET_THREADS;
  const int kyp = r & 1; r >>= 1;
  const int kz = r & 3; r >>= 2;
  const int ci = r % C; r /= C;
  const int cog = r;

  p2 acc2[4][2][4];   // [co pair][ky of the pair][kx]: lo = even co, hi = odd co (fma.rn.f32x2)
#pragma unroll
  for (int c = 0; c < 4; ++c)
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
      for (int x = 0; x < 4; ++x) acc2[c][k][x] = p2_bcast(0.f);
  float dbacc = 0.f;
  constexpr int DB_PARTS = 256 / C;  // threads per channel for the bias-gradient side sum
  const int db_c = tid / DB_PARTS, db_part = tid % DB_PARTS;

  const int items = p.n * DG * G::BANDS;
  for (int item = blockIdx.x; item < items; item += gridDim.x) {
    int q = item;
    const int band = q % G::BANDS; q /= G::BANDS;
    const int z = q % DG; q /= DG;
    const int b = q;
    const int y0 = band * TYG;
    __syncthreads();
    // ---- stage g band [C][TYG][GP] and a bands [C][4][TYG+3][AP]
    {
      constexpr int NVG = G::GP / 4;
      const float* gb = p.g + (((size_t)b * C) * DG + z) * DG * G::GP + (size_t)y0 * G::GP;
      // s_g[c/2][row][x][c&1]: the two channels of a pair are interleaved so that one LDS.128 yields
      // the (g_c, g_c+1) operand pairs of two x positions
      for (int i = tid; i < C * TYG * NVG; i += 256) {
        const int c = i / (TYG * NVG), rem = i - c * (TYG * NVG);
        const float* sg = gb + (size_t)c * DG * DG * G::GP + 4 * rem;
        float* d = s_g + ((c >> 1) * TYG * G::GP + rem * 4) * 2 + (c & 1);
        tma::cp_async4(d, sg); tma::cp_async4(d + 2, sg + 1); tma::cp_async4(d + 4, sg + 2); tma::cp_async4(d + 6, sg + 3);
      }
      constexpr int NVA = G::APG / 4;
      constexpr int RA = TYG + 3;
      const float* ab = p.a + (((size_t)b * C) * G::DA + z) * G::DA * G::APG + (size_t)y0 * G::APG;
      for (int i = tid; i < C * 4 * RA * NVA; i += 256) {
        int t = i;
        const int xv = t % NVA; t /= NVA;
        const int ry = t % RA; t /= RA;
        const int sz = t & 3; t >>= 2;
        const int c = t;
        tma::cp_async16(s_a + (c * 4 + sz) * G::ZSA + ry * G::AP + 4 * xv,
                        ab + ((size_t)c * G::DA + sz) * G::DA * G::APG + (size_t)ry * G::APG + 4 * xv);
      }
      tma::cp_async_wait_all();
    }
    __syncthreads();
    // ---- bias gradient side sum (all threads, C channels x DB_PARTS parts)
    {
      const float* gc = s_g + (db_c >> 1) * TYG * G::GP * 2 + (db_c & 1);
      float s = 0.f;
      for (int i = db_part; i < TYG * DG; i += DB_PARTS) s += gc[((i / DG) * G::GP + (i % DG)) * 2];
      dbacc += s;
    }
    // ---- main accumulation
    const float* a_base = s_a + (ci * 4 + kz) * G::ZSA + (2 * kyp) * G::AP;
    const float* g_base = s_g + (cog * 4) * TYG * G::GP * 2;
#pragma unroll 1
    for (int rr = 0; rr < G::ROWS_PER_SET; ++rr) {
      const int row = set * G::ROWS_PER_SET + rr;
#pragma unroll 2
      for (int xq = 0; xq < G::XQ; ++xq) {
        p2 av[2][8];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
          const float* ar = a_base + (row + k) * G::AP + 4 * xq;
          const float4 lo = *reinterpret_cast<const float4*>(ar);
          const float4 hi = *reinterpret_cast<const float4*>(ar + 4);
          av[k][0] = p2_bcast(lo.x); av[k][1] = p2_bcast(lo.y); av[k][2] = p2_bcast(lo.z); av[k][3] = p2_bcast(lo.w);
          av[k][4] = p2_bcast(hi.x); av[k][5] = p2_bcast(hi.y); av[k][6] = p2_bcast(hi.z); av[k][7] = p2_bcast(hi.w);
        }
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          p2 gv[4];
          const float* gr = g_base + ((c * TYG + row) * G::GP + 4 * xq) * 2;
          p2_ld2(gr, gv[0], gv[1]);
          p2_ld2(gr + 4, gv[2], gv[3]);
#pragma unroll
          for (int k = 0; k < 2; ++k)
#pragma unroll
            for (int kx = 0; kx < 4; ++kx)
#pragma unroll
              for (int j = 0; j < 4; ++j) p2_fma(acc2[c][k][kx], gv[j], av[k][j + kx]);
        }
      }
    }
  }
  // ---- CTA result: sum the position sets, write one partial in PyTorch layout (co,ci,kz,ky,kx)
  float acc[8][2][4];
#pragma unroll
  for (int c = 0; c < 8; ++c)
#pragma unroll
    for (int k = 0; k < 2; ++k)
#pragma unroll
      for (int x = 0; x < 4; ++x) acc[c][k][x] = (c & 1) ? p2_hi(acc2[c >> 1][k][x]) : p2_lo(acc2[c >> 1][k][x]);
  __syncthreads();
  float* out = p.partial + (size_t)blockIdx.x * G::OUT_FLOATS;
  if (G::NSET > 1) {
    float* red = smem;
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int kx = 0; kx < 4; ++kx)
          red[set * G::NW + (((cog * 8 + c) * C + ci) * 4 + kz) * 16 + (2 * kyp + k) * 4 + kx] = acc[c][k][kx];
    __syncthreads();
    for (int i = tid; i < G::NW; i += 256) {
      float s = 0.f;
#pragma unroll
      for (int t = 0; t < G::NSET; ++t) s += red[t * G::NW + i];
      out[i] = s;
    }
  } else {
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int k = 0; k < 2; ++k)
#pragma unroll
        for (int kx = 0; kx < 4; ++kx)
          out[(((cog * 8 + c) * C + ci) * 4 + kz) * 16 + (2 * kyp + k) * 4 + kx] = acc[c][k][kx];
  }
  // bias gradient: reduce the DB_PARTS partial sums of each channel (fixed order)
  __syncthreads();
  float* sdb = smem;
  sdb[tid] = dbacc;
  __syncthreads();
  if (tid < C) {
    float s = 0.f;
    for (int i = 0; i < DB_PARTS; ++i) s += sdb[tid * DB_PARTS + i];
    out[G::NW + tid] = s;
  }
}

// dst[map(i)] = sum_{c < count} partial[c * stride + i]   (fixed order => deterministic)
// map(i) = i for i < n_w when seg_len == 0, else (i / seg_len) * seg_stride + i % seg_len;
// the n_b values after the first n_w go to dst_b.
struct ReduceJob {
  const float* partial;
  float* dst_w;
  float* dst_b;   // may be null when n_b == 0
  int32_t count, stride, n_w, n_b, seg_len, seg_stride;
};
constexpr int kMaxReduceJobs = 28;
struct ReduceParams {
  ReduceJob job[kMaxReduceJobs];
  int32_t njobs;
};
// grid.y = job; 8 lanes along the partial index x 32 outputs per CTA
__global__ void __launch_bounds__(256) k_reduce_partials(ReduceParams p) {
  __shared__ float sm[8][33];
  const ReduceJob& J = p.job[blockIdx.y];
  const int n = J.n_w + J.n_b;
  const int lane = threadIdx.x & 31, part = threadIdx.x >> 5;
  for (int i0 = blockIdx.x * 32; i0 < n; i0 += gridDim.x * 32) {
    const int i = i0 + lane;
    float s = 0.f;
    if (i < n) {
      // four independent running sums keep four loads in flight (the loop is L2-latency bound); the order
      // of the additions is fixed, so the result is deterministic
      float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
      const float* src = J.partial + i;
      int c = part;
      for (; c + 24 < J.count; c += 32) {
        s0 += src[(size_t)c * J.stride];
        s1 += src[(size_t)(c + 8) * J.stride];
        s2 += src[(size_t)(c + 16) * J.stride];
        s3 += src[(size_t)(c + 24) * J.stride];
      }
      for (; c < J.count; c += 8) s0 += src[(size_t)c * J.stride];
      s = (s0 + s1) + (s2 + s3);
    }
    sm[part][lane] = s;
    __syncthreads();
    if (part == 0 && i < n) {
      float t = sm[0][lane];
#pragma unroll
      for (int k = 1; k < 8; ++k) t += sm[k][lane];
      if (i < J.n_w) {
        const int d = J.seg_len ? (i / J.seg_len) * J.seg_stride + i % J.seg_len : i;
        J.dst_w[d] = t;
      } else {
        J.dst_b[i - J.n_w] = t;
      }
    }
    __syncthreads();
  }
}

}  // namespace fast
}  // namespace nvf
