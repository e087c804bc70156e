// Row-register-tile kernels for the stride-2, k=5 transposed convolutions (up1 / up2, padding 0;
// F.conv_transpose3d at utils/network.py:621) of the training path.
//
// Why another formulation.  The tile kernels of nvf_fast_convt.cuh compute every output of a zero-padded tile with
// every tap: for a 16^3 -> 35^3 layer that is 1.98x the exact multiply-adds (zero halo in y and x, 40 columns for 35,
// row-parity divergence inside warps).  Here
//   * a THREAD owns one whole output row (all DOUT = 2 DIN + 3 columns) of one output-channel pair and walks over the
//     input rows that feed it.  In x the work is written in scatter form, acc[2 i + kx] += a[i] * w[kx], fully
//     unrolled: every one of the DIN x 5 products is a real one - no halo, no padding columns, decided at compile time;
//   * a WARP works on rows of one (z parity, y parity) class, so the tap counts (3 or 2 per dimension) are warp-uniform
//     and taps whose input slice / row lies outside the tensor for the whole warp are skipped;
//   * input rows are read straight from global memory through L1 (a 16-float row is four LDG.128; the layer's whole
//     input is 0.1-0.5 MB per block and the rows a warp needs are shared by its neighbours), so there is no staging
//     phase, no __syncthreads in the main loop and no CTA-sized work item: warps pull 32-row items from a global
//     queue, heaviest class first, which is what lets 16 blocks fill 148 SMs evenly;
//   * the input-channel sum is split over KS lane groups of a warp (item = 32 / KS rows), combined by shuffles, to
//     keep the items small against the 16-block step.
// Weights (the only data every thread needs) are staged once per CTA in shared memory, re-laid as
// [ci][kz][ky][lane group][co pair][kx] so that a row's five taps are three LDS.128 and the eight (group, pair)
// addresses of a warp fall into distinct banks.
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"
#include "nvf_tma.cuh"

namespace nvf {
namespace fast {

__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait_group() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

struct RowTFwdParams {
  const float* in;      // [n][CI][DIN][DIN][DIN]
  float* out;           // [n][CO][DOUT][DOUT][OP]   relu(acc + bias), columns >= DOUT written as zero
  const float* Wp;      // PACK_CONVT_FWD [ci][kz][ky][kx][co]
  const float* bias;    // [CO]
  unsigned int* queue;  // [2] work-queue words: zero on entry, left at zero
  int32_t n;
};

template <int CI, int CO, int DIN, int KS>
struct RowTFwdCfg {
  static constexpr int DOUT = 2 * DIN + 3, OP = (DOUT + 3) / 4 * 4;
  static constexpr int NCOP = CO / 2;
  static constexpr int TPW = 32 / KS;        // rows (tasks) per warp item
  static constexpr int CIK = CI / KS;        // input channels per lane group
  static constexpr int NE = DIN + 2, NO = DIN + 1;   // even / odd output positions per dimension
  static constexpr int WROW = 12;            // floats per (ci, kz, ky, group, pair): 5 kx pairs + one pad pair
  static constexpr int W_FLOATS = CI * 25 * NCOP * WROW;
  static constexpr int SMEM_BYTES = W_FLOATS * 4;
  // class c = 2 * (z parity) + (y parity); cost ~ taps_z * taps_y = 9, 6, 6, 4: heaviest first in the queue
  static constexpr int I0 = (NE * NE * NCOP + TPW - 1) / TPW, I1 = (NE * NO * NCOP + TPW - 1) / TPW, I2 = I1,
                       I3 = (NO * NO * NCOP + TPW - 1) / TPW;   // warp items per block and class
  static constexpr int ITEMS_PER_BLOCK = I0 + I1 + I2 + I3;
  static_assert(CI % KS == 0 && 32 % KS == 0 && CO % 2 == 0 && DIN % 4 == 0, "row-tile convT configuration");
};

// one step of a row task: DIN x 5 products of one input row (four floats per register quad) with the five taps
template <int DIN, int DOUT>
__device__ __forceinline__ void row_step(p2 (&acc)[DOUT], const float4 (&r)[DIN / 4], const p2 (&w)[6]) {
#pragma unroll
  for (int q4 = 0; q4 < DIN / 4; ++q4) {
    const p2 a[4] = {p2_bcast(r[q4].x), p2_bcast(r[q4].y), p2_bcast(r[q4].z), p2_bcast(r[q4].w)};
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int kx = 0; kx < 5; ++kx) p2_fma(acc[2 * (4 * q4 + j) + kx], w[kx], a[j]);
  }
}

// PIPE: software-pipeline the step loop in registers (needs ~40 more registers: 1 CTA of 384 threads per SM);
// CHUNK: a CTA pulls THREADS / 32 consecutive items at a time, one per warp, so that its warps work on neighbouring
// rows of one block and class and share their input rows in L1 (items of one class cost the same)
template <int CI, int CO, int DIN, int KS, int THREADS, int MINB, bool PIPE = false, bool CHUNK = true>
__global__ void __launch_bounds__(THREADS, MINB) k_convT5_fwd_rows(RowTFwdParams p) {
  using G = RowTFwdCfg<CI, CO, DIN, KS>;
  extern __shared__ __align__(128) float s_w[];
  const int tid = threadIdx.x, lane = tid & 31;
  // ---- weights -> shared memory, [cc][kz*5+ky][group][pair][kx][half]  (ci = group * CIK + cc)
  for (int i = tid; i < CI * 25 * G::NCOP * 10; i += THREADS) {
    int q = i;
    const int h = q & 1; q >>= 1;
    const int kx = q % 5; q /= 5;
    const int cop = q % G::NCOP; q /= G::NCOP;
    const int kk = q % 25; q /= 25;
    const int ci = q;
    const int grp = ci / G::CIK, cc = ci % G::CIK;
    s_w[(((cc * 25 + kk) * KS + grp) * G::NCOP + cop) * G::WROW + 2 * kx + h] =
        __ldg(p.Wp + ((size_t)(ci * 25 + kk) * 5 + kx) * CO + 2 * cop + h);
  }
  __syncthreads();
  const int tl = lane % G::TPW, grp = lane / G::TPW;
  const unsigned total = (unsigned)p.n * G::ITEMS_PER_BLOCK;
  constexpr size_t in_cs = (size_t)DIN * DIN * DIN;
  constexpr size_t out_cs = (size_t)G::DOUT * G::DOUT * G::OP;

  __shared__ unsigned s_base;
  for (;;) {
    unsigned item = 0;
    if constexpr (CHUNK) {
      __syncthreads();                       // every warp has read the previous base
      if (tid == 0) s_base = atomicAdd(p.queue, (unsigned)(THREADS / 32));
      __syncthreads();
      if (s_base >= total) break;            // uniform for the CTA
      item = s_base + (unsigned)(tid >> 5);
      if (item >= total) continue;           // ragged last chunk: this warp idles one round
    } else {
      if (lane == 0) item = atomicAdd(p.queue, 1u);
      item = __shfl_sync(0xffffffffu, item, 0);
      if (item >= total) break;
    }
    // ---- decode: class (heaviest first), block, row group
    int c = 0;
    unsigned rem = item;
    const unsigned n0 = (unsigned)p.n * G::I0, n1 = (unsigned)p.n * G::I1, n2 = (unsigned)p.n * G::I2;
    if (rem >= n0) {
      rem -= n0; c = 1;
      if (rem >= n1) {
        rem -= n1; c = 2;
        if (rem >= n2) { rem -= n2; c = 3; }
      }
    }
    const int ipb = c == 0 ? G::I0 : (c == 3 ? G::I3 : G::I1);
    const int b = (int)(rem / (unsigned)ipb), g = (int)(rem % (unsigned)ipb);
    const int pz = c >> 1, py = c & 1;
    const int rows = py ? G::NO : G::NE;
    const int npairs = (pz ? G::NO : G::NE) * rows;
    const int t = g * G::TPW + tl;
    const bool active = t < npairs * G::NCOP;
    const int cop = active ? t % G::NCOP : 0;
    const int pair = active ? t / G::NCOP : 0;
    const int sz = pair / rows, ry = pair - sz * rows;     // output z = 2 sz + pz, y = 2 ry + py
    const int NT = pz ? 2 : 3, NKY = py ? 2 : 3;

    p2 acc[G::DOUT];
#pragma unroll
    for (int j = 0; j < G::DOUT; ++j) acc[j] = p2_bcast(0.f);

    // ---- flat loop over the (input channel, kz tap, ky tap) steps, software-pipelined in registers: the input row
    // and the taps of step s + 1 are fetched (LDG through L1, LDS) before the products of step s are issued, so a
    // warp's own arithmetic covers its load latency; rows outside the tensor read as zero, steps whose rows lie
    // outside for the whole warp are skipped
    const float* in_b = p.in + ((size_t)b * CI + (size_t)grp * G::CIK) * in_cs;
    const int nky = NKY, nstep = G::CIK * NT * NKY;
    auto fetch = [&](int s, float4 (&r)[DIN / 4], p2 (&w)[6]) -> bool {
      const int cc = s / (NT * nky), rr = s - cc * (NT * nky), tz = rr / nky, u = rr - tz * nky;
      const int iz = sz - tz, iy = ry - u;
      const bool v = active && (unsigned)iz < (unsigned)DIN && (unsigned)iy < (unsigned)DIN;
      const bool any = __any_sync(0xffffffffu, v);
      if (any) {
        const float4* row = reinterpret_cast<const float4*>(in_b + (size_t)cc * in_cs + ((size_t)(v ? iz : 0) * DIN + (v ? iy : 0)) * DIN);
#pragma unroll
        for (int q4 = 0; q4 < DIN / 4; ++q4) r[q4] = v ? __ldg(row + q4) : make_float4(0.f, 0.f, 0.f, 0.f);
        const float* wr = s_w + ((((cc * 5 + pz + 2 * tz) * 5 + py + 2 * u) * KS + grp) * G::NCOP + cop) * G::WROW;
        p2_ld2(wr, w[0], w[1]);
        p2_ld2(wr + 4, w[2], w[3]);
        p2_ld2(wr + 8, w[4], w[5]);
      }
      return any;
    };
    if constexpr (PIPE) {
      float4 ra[DIN / 4], rb[DIN / 4];
      p2 wa[6], wb[6];
      bool any_a = fetch(0, ra, wa), any_b = false;
#pragma unroll 1
      for (int s = 0; s < nstep; s += 2) {
        if (s + 1 < nstep) any_b = fetch(s + 1, rb, wb);
        if (any_a) row_step<DIN, G::DOUT>(acc, ra, wa);
        if (s + 2 < nstep) any_a = fetch(s + 2, ra, wa);
        if (s + 1 < nstep && any_b) row_step<DIN, G::DOUT>(acc, rb, wb);
      }
    } else {
#pragma unroll 1
      for (int s = 0; s < nstep; ++s) {
        float4 ra[DIN / 4];
        p2 wa[6];
        if (fetch(s, ra, wa)) row_step<DIN, G::DOUT>(acc, ra, wa);
      }
    }
    // ---- combine the lane groups (fixed order: group 0 + group 1 [+ ...])
    if constexpr (KS > 1) {
#pragma unroll
      for (int off = G::TPW; off < 32; off <<= 1) {
#pragma unroll
        for (int j = 0; j < G::DOUT; ++j) {
          const float lo = __shfl_xor_sync(0xffffffffu, p2_lo(acc[j]), off);
          const float hi = __shfl_xor_sync(0xffffffffu, p2_hi(acc[j]), off);
          acc[j] = p2_make(p2_lo(acc[j]) + lo, p2_hi(acc[j]) + hi);
        }
      }
    }
    if (active && grp == 0) {
      const int oz = 2 * sz + pz, oy = 2 * ry + py;
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int co = 2 * cop + h;
        const float bb = __ldg(p.bias + co);
        float* o = p.out + ((size_t)b * CO + co) * out_cs + ((size_t)oz * G::DOUT + oy) * G::OP;
#pragma unroll
        for (int q4 = 0; q4 < G::OP / 4; ++q4) {
          float vv[4];
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const int x = 4 * q4 + j;
            float r = 0.f;
            if (x < G::DOUT) {
              r = (h ? p2_hi(acc[x < G::DOUT ? x : 0]) : p2_lo(acc[x < G::DOUT ? x : 0])) + bb;
              r = r > 0.f ? r : 0.f;
            }
            vv[j] = r;
          }
          *reinterpret_cast<float4*>(o + 4 * q4) = make_float4(vv[0], vv[1], vv[2], vv[3]);
        }
      }
    }
  }
  // ---- retire: the last warp / CTA of the grid to run dry rewinds the queue for the next launch
  if (CHUNK ? tid == 0 : lane == 0) {
    const unsigned d = atomicAdd(p.queue + 1, 1u);
    if (d == (CHUNK ? gridDim.x : gridDim.x * (THREADS / 32)) - 1) {
      p.queue[0] = 0u;
      p.queue[1] = 0u;
    }
  }
}

}  // namespace fast
}  // namespace nvf
