// Warp-specialised fused decode head:  up2 -> ReLU -> conv2 -> ReLU -> conv2_cls -> sigmoid -> threshold
// (utils/network.py:4765-4768, NVFPCC.py:631-633) for one leaf block per persistent CTA, 87 % of the decoder's
// multiply-adds.  Nothing of the up2 / conv2 activations (1.3 + 1.0 MB per leaf at 8,16,8,8; 2.8 + 2.1 MB at
// 16,32,16,16) leaves the SM; the input is the (zero-padded) conv1 output written by the batched stem kernels.
//
// One CTA = 8 consumer warps + 4 producer warps, register file re-split with setmaxnreg (consumers 184, producers
// 136 registers per thread):
//   * producers compute one up2 slice (z fixed, all rows of the pass, all output channels) at a time into a
//     double-buffered shared-memory slice: polyphase stride-2 transposed conv, 8 x (4 even + 4 odd) outputs x 8
//     channels per thread, even rows first then odd rows so every warp's tap count is uniform; input rows come
//     straight from global memory (L1 / L2 resident; all taps of an input channel are unrolled, so the loads of later
//     taps are issued under the FFMA2s of earlier ones).  For the wide configuration
//     the 128 KB of up2 weights do not fit next to the slices: they stream through a two-stage cp.async ring, one
//     input channel (8 KB) per step;
//   * consumers run conv2 "input-stationary" along z as the round-1 kernel did: slice z of up2 contributes to the
//     four output slices z-3..z whose partial sums live in registers (8 channels x 4 x per slice, FFMA2 over
//     channel pairs; the oldest slice is finished and written out before the other three are touched, so 96, not
//     128, accumulators are live at a time); a finished conv2 slice goes to shared memory once and is
//     consumed the same way by the 3x3x3 classifier; probabilities are thresholded into mask words with warp
//     shuffles (no shared-memory atomics).
//   Producer and consumer meet only at the full / empty mbarriers of the two slice buffers, so the transposed conv of
//   slice z+1 runs under the conv2 of slice z and the FMA pipe sees three warps per scheduler instead of one phase
//   with 175 busy threads followed by another with 256.
//   * 16 output channels x 32 x 32 positions x 4 slices of partial sums do not fit 256 threads' registers, so the
//     wide configuration walks a leaf in two y passes (16 rows of conv2 output each, 19 rows of up2).  The
//     classifier rows next to the cut (15 | 16) need the other pass's conv2 row: each pass leaves that row's partial
//     logits and its conv2 row in a global scratch (136 KB per leaf), and k_head_fixup adds the missing tap row,
//     applies sigmoid / threshold and writes those two rows.
//   * Work items are (leaf, pass) units, round-robin over the persistent CTAs.  The units of the last, partial round
//     are cut along z into 2, 4 or 8 chunks (each re-computing the few up2 / conv2 slices next to its cuts) so that
//     the round keeps all SMs busy and ends early; every output is still summed in exactly the same order, so a
//     leaf's result does not depend on its position in the batch or on the number of leaves / GPUs.
#pragma once
#include <cuda_runtime.h>
#include "nvf_common.h"
#include "nvf_tma.cuh"

namespace nvf {
namespace fast {

struct HeadParams {
  const float* sp;       // zero-padded conv1 output [n][C2][16][20][24] (data at rows 2..17, columns 4..19)
  const float* w_up2;    // [C2][5][5][5][C3]
  const float* w_c2;     // [C3][4][4][4][C3]
  const float* w_cls;    // [C3][3 ky][3 kz][4 (kx, pad)]
  const float* up2_b;    // [C3]
  const float* conv2_b;  // [C3]
  const float* cls2_b;   // [1]
  float* prob_out;       // [n][32768] or null
  uint32_t* mask_out;    // [n][1024]
  int32_t* counts_out;   // [n], ZERO on entry (rows add their point counts)
  float* brow;           // wide configuration: [n][2 passes][C3][32 z][32 x] conv2 rows next to the cut, else null
  float* pl;             // wide configuration: [n][2 passes][32 z][32 x] partial logits of those rows, else null
  float thh;
  int32_t n_blocks;
};

constexpr int kHeadConsumers = 256, kHeadProducers = 128, kHeadThreads = kHeadConsumers + kHeadProducers;
constexpr int kSpRows = 20, kSpPitch = 24, kSpPlane = kSpRows * kSpPitch;   // padded conv1 slice

template <int C2, int C3>
struct HeadCfg {
  static_assert(C3 == 8 || C3 == 16, "conv2 channel groups of 8: one or two y passes");
  static constexpr int COH = C3 / 8;            // output-channel groups of 8 = y passes per leaf
  static constexpr int RY = 32 / COH;           // conv2 / logit rows per pass
  static constexpr int UR = RY + 3;             // up2 rows per pass
  static constexpr int NE = (UR + 1) / 2, NO = UR / 2;   // even / odd up2 rows of a pass (the first row is even)
  static constexpr int U_PITCH = 36, U_PLANE = UR * U_PITCH, U_SIZE = C3 * U_PLANE;
  static constexpr int CR = RY + 2, C_PITCH = 36, C_PLANE = CR * C_PITCH, C_SIZE = C3 * C_PLANE + 4;
  static constexpr int W_UP2 = C2 * 125 * C3, W_C2 = C3 * 64 * C3, W_CLS = C3 * 36;
  static constexpr bool RING = (W_UP2 + W_C2) * 4 > 100 * 1024;
  static constexpr int STAGE = 125 * C3;        // up2 weights of one input channel
  static constexpr int OFF_W_C2 = 0;
  static constexpr int OFF_W_CLS = OFF_W_C2 + W_C2;
  static constexpr int OFF_BIAS = OFF_W_CLS + W_CLS;           // [C3] up2_b, [C3] conv2_b, [4] cls_b
  static constexpr int OFF_W_UP2 = OFF_BIAS + 2 * C3 + 4;
  static constexpr int OFF_U = OFF_W_UP2 + (RING ? 2 * STAGE : W_UP2);
  static constexpr int OFF_C = OFF_U + 2 * U_SIZE;
  static constexpr int OFF_EX = OFF_C + C_SIZE;                // [2][RY][32] partial logits of the second channel group
  static constexpr int OFF_BAR = OFF_EX + (COH == 2 ? 2 * RY * 32 : 0);
  static constexpr int SMEM_FLOATS = OFF_BAR + 8;
  static constexpr int SMEM_BYTES = SMEM_FLOATS * 4;
  static constexpr int BROW_FLOATS = COH == 2 ? 2 * C3 * 1024 : 0;   // per leaf
  static constexpr int PL_FLOATS = COH == 2 ? 2048 : 0;              // per leaf
  static_assert(OFF_W_CLS % 4 == 0 && OFF_BIAS % 4 == 0 && OFF_W_UP2 % 4 == 0 && OFF_U % 4 == 0 && OFF_C % 4 == 0 &&
                    OFF_EX % 4 == 0 && OFF_BAR % 2 == 0 && U_SIZE % 4 == 0 && STAGE % 4 == 0,
                "16-byte alignment of the shared-memory regions");
  static_assert(SMEM_BYTES <= 227 * 1024, "decode head shared memory");
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(tma::smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
template <int N>
__device__ __forceinline__ void reg_inc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(N)); }
template <int N>
__device__ __forceinline__ void reg_dec() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(N)); }

// Work items.  Units = (leaf, pass); the units of the last partial round are cut along z into k chunks.
struct HeadItems {
  int n_full, k, total;   // whole units, chunks per tail unit, number of items
  __device__ __forceinline__ HeadItems(int units, int ctas) {
    n_full = units / ctas * ctas;
    const int tail = units - n_full;
    k = 1;
    if (tail > 0) {
      const int f = ctas / tail;
      k = f >= 8 ? 8 : (f >= 4 ? 4 : (f >= 2 ? 2 : 1));
    }
    total = n_full + tail * k;
  }
  // item -> unit and logit slices [za, zb)
  __device__ __forceinline__ void get(int item, int& unit, int& za, int& zb) const {
    if (item < n_full) {
      unit = item; za = 0; zb = 32;
    } else {
      const int j = item - n_full;
      unit = n_full + j / k;
      const int len = 32 / k;
      za = (j % k) * len;
      zb = za + len;
    }
  }
};

// ------------------------------------------------------------------------------------------------- consumers
// conv2 partial sums of one up2 slice for the slots J0 .. J0+NJ-1 (slot j = output slice s-3+j, tap kz = 3-j)
template <int C2, int C3, int J0, int NJ, bool ALL>
__device__ __forceinline__ void head_conv2_accum(const float* U, const float* W, p2 (&acc)[4][4][4], int y, int x0,
                                                 int lo, int hi) {
  using G = HeadCfg<C2, C3>;
#pragma unroll 1
  for (int ci = 0; ci < C3; ++ci) {
#pragma unroll
    for (int ky = 0; ky < 4; ++ky) {
      const float* r = U + ci * G::U_PLANE + (y + ky) * G::U_PITCH + x0;
      const f4 v0 = ld4(r), v1 = ld4(r + 4);
      const p2 a[8] = {p2_bcast(v0.x), p2_bcast(v0.y), p2_bcast(v0.z), p2_bcast(v0.w),
                       p2_bcast(v1.x), p2_bcast(v1.y), p2_bcast(v1.z), p2_bcast(v1.w)};
#pragma unroll
      for (int j = J0; j < J0 + NJ; ++j) {
        if (!ALL && (j < lo || j > hi)) continue;
        const int kz = 3 - j;
        const float* wrow = W + (((ci * 4 + kz) * 4 + ky) * 4) * C3;
#pragma unroll
        for (int kx = 0; kx < 4; ++kx) {
          p2 w[4];
          p2_load_w8(wrow + kx * C3, w);
#pragma unroll
          for (int c = 0; c < 4; ++c) {
#pragma unroll
            for (int i = 0; i < 4; ++i) p2_fma(acc[j][c][i], w[c], a[i + kx]);
          }
        }
      }
    }
  }
}

template <int C2, int C3>
__device__ __forceinline__ void head_consumer(const HeadParams& p, float* sm, uint64_t* bars, const int tid) {
  using G = HeadCfg<C2, C3>;
  const int coh = tid / (G::RY * 8);             // warp-uniform: this thread's group of 8 output channels
  const int rem = tid - coh * (G::RY * 8);
  const int y = rem >> 3, x0 = (rem & 7) * 4;
  const int lane = tid & 31;
  const float* Wc2 = sm + G::OFF_W_C2 + coh * 8;
  const float* Wcls = sm + G::OFF_W_CLS;
  float* C = sm + G::OFF_C;
  const float cls_b = sm[G::OFF_BIAS + 2 * C3];
  uint32_t it = 0;                               // running slice number: buffer it & 1, phase (it >> 1) & 1
  const HeadItems items(p.n_blocks * G::COH, gridDim.x);

#pragma unroll 1
  for (int item = blockIdx.x; item < items.total; item += gridDim.x) {
    int unit, za, zb;                            // logit slices [za, zb) of this item
    items.get(item, unit, za, zb);
    const int b = unit / G::COH, yh = unit - b * G::COH;
    const int zc_lo = za > 0 ? za - 1 : 0, zc_hi = zb < 32 ? zb : 31;   // conv2 slices the classifier needs
    const bool is_brow = G::COH == 2 && y == (yh == 0 ? G::RY - 1 : 0);  // row next to the cut between the passes
    const int Y = yh * G::RY + y;                // row inside the leaf
    float* brow = G::COH == 2 ? p.brow + ((size_t)b * 2 + yh) * C3 * 1024 : nullptr;
    int cnt = 0;
    p2 acc[4][4][4];                             // [slot j: conv2 slice s-3+j][channel pair][x]
    p2 cacc[3][2];                               // [slot g: logit slice z1-1+g][x pair] (lo = even x)
#pragma unroll
    for (int j = 0; j < 4; ++j)
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[j][c][i] = p2_bcast(0.f);
#pragma unroll
    for (int g = 0; g < 3; ++g) cacc[g][0] = cacc[g][1] = p2_bcast(0.f);

#pragma unroll 1
    for (int s = zc_lo; s <= zc_hi + 3; ++s, ++it) {   // up2 slices of this item
      const float* U = sm + G::OFF_U + (it & 1) * G::U_SIZE;
      tma::mbar_wait(&bars[it & 1], (it >> 1) & 1);
      // The oldest slot (conv2 slice zo = s-3, tap kz = 3) is finished first and written out, so that only three
      // of the four slots of partial sums are live at any time (96 instead of 128 accumulator registers): the new
      // slot s starts from zero only in the second pass.  The order of additions per output is unchanged.
      const int zo = s - 3;                      // conv2 slice finished by this step
      const bool have = zo >= zc_lo;
      if (have) {
        head_conv2_accum<C2, C3, 0, 1, true>(U, Wc2, acc, y, x0, 0, 3);
        const float* bias = sm + G::OFF_BIAS + C3 + coh * 8;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const float bb = bias[c];
          float v[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) v[i] = relu(((c & 1) ? p2_hi(acc[0][c >> 1][i]) : p2_lo(acc[0][c >> 1][i])) + bb);
          st4(C + (coh * 8 + c) * G::C_PLANE + (y + 1) * G::C_PITCH + 4 + x0, v[0], v[1], v[2], v[3]);
          if (G::COH == 2 && is_brow)
            st4(brow + ((size_t)(coh * 8 + c) * 32 + zo) * 32 + x0, v[0], v[1], v[2], v[3]);
        }
      }
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < 4; ++i) acc[3][c][i] = p2_bcast(0.f);   // the new slot (conv2 slice s) starts here
      {
        // slot j holds conv2 slice s-3+j: accumulate the ones inside [zc_lo, zc_hi]
        const int lo = zc_lo + 3 - s > 1 ? zc_lo + 3 - s : 1;
        const int hi = zc_hi + 3 - s < 3 ? zc_hi + 3 - s : 3;
        if (lo == 1 && hi == 3) head_conv2_accum<C2, C3, 1, 3, true>(U, Wc2, acc, y, x0, lo, hi);
        else head_conv2_accum<C2, C3, 1, 3, false>(U, Wc2, acc, y, x0, lo, hi);
      }
      mbar_arrive(&bars[2 + (it & 1)]);          // this thread is done with the slice buffer
#pragma unroll
      for (int c = 0; c < 4; ++c)
#pragma unroll
        for (int i = 0; i < 4; ++i) {            // slot j+1 -> j (slot 3 is dead until the next step re-creates it)
          acc[0][c][i] = acc[1][c][i];
          acc[1][c][i] = acc[2][c][i];
          acc[2][c][i] = acc[3][c][i];
        }
      named_bar_sync(1, kHeadConsumers);         // conv2 slice zo complete in C
      const int z1 = zo;
      if (have) {
        // classifier, input-stationary: conv2 slice z1 contributes to logit slices z1-1+g (tap kz = 2-g) inside
        // [za, zb); each channel group sums over its own 8 channels
        const int lo = za - z1 + 1 > 0 ? za - z1 + 1 : 0;
        const int hi = zb - z1 < 2 ? zb - z1 : 2;
#pragma unroll 1
        for (int cc = 0; cc < 8; ++cc) {
          const int ci = coh * 8 + cc;
#pragma unroll
          for (int ky = 0; ky < 3; ++ky) {
            const float* r = C + ci * G::C_PLANE + (y + ky) * G::C_PITCH + x0 + 3;
            const f4 v = ld4(r + 1);
            // x pairs of the six-wide window: FFMA2 with the tap weight as the scalar operand; per output the
            // taps are still added in the order kx = 0, 1, 2
            const float a0 = r[0], a5 = r[5];
            const p2 A[5] = {p2_make(a0, v.x), p2_make(v.x, v.y), p2_make(v.y, v.z), p2_make(v.z, v.w), p2_make(v.w, a5)};
            const float* wr = Wcls + (ci * 3 + ky) * 12;
#pragma unroll
            for (int g = 0; g < 3; ++g) {
              if (g < lo || g > hi) continue;
              const f4 w = ld4(wr + (2 - g) * 4);
              const p2 wx = p2_bcast(w.x), wy = p2_bcast(w.y), wz = p2_bcast(w.z);
#pragma unroll
              for (int h = 0; h < 2; ++h) {
                p2_fma(cacc[g][h], A[2 * h], wx);
                p2_fma(cacc[g][h], A[2 * h + 1], wy);
                p2_fma(cacc[g][h], A[2 * h + 2], wz);
              }
            }
          }
        }
        if (G::COH == 2 && coh == 1) {           // hand the second group's finished partial logits to the first
          float* ex = sm + G::OFF_EX + y * 32 + x0;
          if (z1 - 1 >= za) st4(ex, p2_lo(cacc[0][0]), p2_hi(cacc[0][0]), p2_lo(cacc[0][1]), p2_hi(cacc[0][1]));
          if (z1 == 31) st4(ex + G::RY * 32, p2_lo(cacc[1][0]), p2_hi(cacc[1][0]), p2_lo(cacc[1][1]), p2_hi(cacc[1][1]));
        }
      }
      named_bar_sync(1, kHeadConsumers);         // C has been read by everyone; partial logits exchanged
      if (have) {
        if (coh == 0) {
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            if (e == 0 ? z1 - 1 < za : z1 != 31) continue;
            const int zl = e == 0 ? z1 - 1 : 31;   // logit slice that is complete now
            float v[4] = {p2_lo(cacc[e][0]), p2_hi(cacc[e][0]), p2_lo(cacc[e][1]), p2_hi(cacc[e][1])};
            if (G::COH == 2) {
              const f4 o = ld4(sm + G::OFF_EX + e * G::RY * 32 + y * 32 + x0);
              v[0] += o.x; v[1] += o.y; v[2] += o.z; v[3] += o.w;
            }
            uint32_t nib = 0;
            float pr[4];
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              pr[i] = sigmoidf(v[i] + cls_b);
              if (pr[i] > p.thh) nib |= 1u << i;
            }
            uint32_t word = nib << x0;
            word |= __shfl_xor_sync(0xffffffffu, word, 1);
            word |= __shfl_xor_sync(0xffffffffu, word, 2);
            word |= __shfl_xor_sync(0xffffffffu, word, 4);
            if (is_brow) {                       // finished by k_head_fixup
              st4(p.pl + (((size_t)b * 2 + yh) * 32 + zl) * 32 + x0, v[0], v[1], v[2], v[3]);
            } else {
              if (p.prob_out) st4(p.prob_out + (size_t)b * kVox + (zl * 32 + Y) * 32 + x0, pr[0], pr[1], pr[2], pr[3]);
              if ((lane & 7) == 0) {
                p.mask_out[(size_t)b * 1024 + zl * 32 + Y] = word;
                cnt += __popc(word);
              }
            }
          }
        }
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          cacc[0][h] = cacc[1][h];
          cacc[1][h] = cacc[2][h];
          cacc[2][h] = p2_bcast(0.f);
        }
      }
    }
    if (cnt) atomicAdd(p.counts_out + b, cnt);
  }
}

// ------------------------------------------------------------------------------------------------- producers
// All taps of one input channel for one thread tile (8 x = 4 even + 4 odd outputs, 8 output channels) of an up2 row
// of parity CY in a slice with NKZ valid kz taps: kz = kz0 + 2 jz reads the input slice jz before the first one,
// ky = CY + 2 jy the input row jy above - compile-time offsets, so the loop is branch-free and the compiler can
// issue the loads of later steps under the FFMA2s of earlier ones.
template <int C3, int CY, int NKZ, int PLANE = kSpPlane, int PITCH = kSpPitch>
__device__ __forceinline__ void head_up2_channel(p2 (&acc)[4][8], const float* in, const float* w) {
#pragma unroll
  for (int jz = 0; jz < NKZ; ++jz) {
#pragma unroll
    for (int jy = 0; jy < (CY ? 2 : 3); ++jy) {
      const float* r = in - jz * PLANE - jy * PITCH;
      float a0, a1;
      ld2(r, a0, a1);
      const f4 v = ld4(r + 2);
      const p2 a[6] = {p2_bcast(a0), p2_bcast(a1), p2_bcast(v.x), p2_bcast(v.y), p2_bcast(v.z), p2_bcast(v.w)};
      const float* wrow = w + ((2 * jz * 5 + 2 * jy) * 5) * C3;
#pragma unroll
      for (int kx = 0; kx < 5; ++kx) {
        p2 wv[4];
        p2_load_w8(wrow + kx * C3, wv);
        const int h = kx >> 1;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if ((kx & 1) == 0) p2_fma(acc[c][2 * j], wv[c], a[j + 2 - h]);
            else p2_fma(acc[c][2 * j + 1], wv[c], a[j + 2 - h]);
          }
        }
      }
    }
  }
}

// The same step with the kz taps in a run-time loop: a third of the code (the six fully unrolled variants of
// head_up2_channel are 86 KB of SASS, and warps of the stand-alone kernel that sit in different variants starve on
// instruction fetch: "no instruction" was its top stall), at the price of one load bubble per kz tap.  Inside the
// head kernel the unrolled variants win (measured: 9.03 vs 9.35 ms at 8,16,8,8; 36.6 vs 40.4 ms at 16,32,16,16).
template <int C3, int CY, int PLANE, int PITCH>
__device__ __forceinline__ void up2_channel_loop(p2 (&acc)[4][8], const float* in, const float* w, int nkz) {
#pragma unroll 1
  for (int jz = 0; jz < nkz; ++jz) {
#pragma unroll
    for (int jy = 0; jy < (CY ? 2 : 3); ++jy) {
      const float* r = in - jy * PITCH;
      float a0, a1;
      ld2(r, a0, a1);
      const f4 v = ld4(r + 2);
      const p2 a[6] = {p2_bcast(a0), p2_bcast(a1), p2_bcast(v.x), p2_bcast(v.y), p2_bcast(v.z), p2_bcast(v.w)};
      const float* wrow = w + (2 * jy * 5) * C3;
#pragma unroll
      for (int kx = 0; kx < 5; ++kx) {
        p2 wv[4];
        p2_load_w8(wrow + kx * C3, wv);
        const int h = kx >> 1;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            if ((kx & 1) == 0) p2_fma(acc[c][2 * j], wv[c], a[j + 2 - h]);
            else p2_fma(acc[c][2 * j + 1], wv[c], a[j + 2 - h]);
          }
        }
      }
    }
    in -= PLANE;
    w += 50 * C3;
  }
}

template <int C2, int C3>
__device__ __forceinline__ void head_producer(const HeadParams& p, float* sm, uint64_t* bars, const int pt) {
  using G = HeadCfg<C2, C3>;
  const float* Wres = sm + G::OFF_W_UP2;
  uint32_t it = 0;
  uint32_t ring_step = 0;                        // RING: number of stages consumed so far
  if (G::RING) {                                 // first stage: input channel 0
    for (int i = pt; i < G::STAGE / 4; i += kHeadProducers)
      tma::cp_async16(sm + G::OFF_W_UP2 + 4 * i, p.w_up2 + 4 * i);
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  const HeadItems items(p.n_blocks * G::COH, gridDim.x);
#pragma unroll 1
  for (int item = blockIdx.x; item < items.total; item += gridDim.x) {
    int unit, za, zb;
    items.get(item, unit, za, zb);
    const int b = unit / G::COH, yh = unit - b * G::COH;
    const int zc_lo = za > 0 ? za - 1 : 0, zc_hi = zb < 32 ? zb : 31;
    const float* in_b = p.sp + (size_t)b * C2 * 16 * kSpPlane;
    {
#pragma unroll 1
      for (int s = zc_lo; s <= zc_hi + 3; ++s, ++it) {
        float* U = sm + G::OFF_U + (it & 1) * G::U_SIZE;
        tma::mbar_wait(&bars[2 + (it & 1)], ((it >> 1) & 1) ^ 1);   // consumers have released this buffer
        // valid kz taps of this slice: kz = pz, pz+2, .. with 0 <= (s - kz) / 2 <= 15
        const int pz = s & 1;
        int kz0 = pz;
        while (s - kz0 > 30) kz0 += 2;
        int nkz = 0;
        for (int kz = kz0; kz < 5 && kz <= s; kz += 2) ++nkz;
#pragma unroll 1
        for (int cy = 0; cy < 2; ++cy) {         // even rows (3 ky taps), then odd rows (2 ky taps)
          const int nrows = cy ? G::NO : G::NE;
          const int ntile = nrows * 5 * G::COH;
          const bool active = pt < ntile;
          const int q = active ? pt % 5 : 0;
          const int rr = active ? (pt / 5) % nrows : 0;
          const int cohp = active ? pt / (5 * nrows) : 0;
          const int l = 2 * rr + cy;             // row inside the pass' up2 slice
          const int Y2 = yh * G::RY + l;         // up2 row inside the leaf (same parity as l)
          p2 acc[4][8];                          // [channel pair][x]
#pragma unroll
          for (int c = 0; c < 4; ++c)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[c][j] = p2_bcast(0.f);
          // first step's input address: slice (s - kz0) / 2, padded row (Y2 - cy) / 2 + 2, columns 4q+2 .. 4q+7;
          // the further taps of a channel lie whole slices / rows before it (head_up2_channel)
          const float* in_t = in_b + ((size_t)((s - kz0) >> 1) * kSpRows + (((Y2 - cy) >> 1) + 2)) * kSpPitch + 4 * q + 2;
          const int w_off = ((kz0 * 5 + cy) * 5) * C3 + cohp * 8;
#pragma unroll 1
          for (int ci = 0; ci < C2; ++ci) {
            const float* Wci;
            if (G::RING) {
              // stage ring_step & 1 holds channel ci: wait for my copies, meet the other producers (their copies have
              // landed, and everybody is done with the other stage), then refill that other stage with channel ci + 1
              asm volatile("cp.async.wait_group 0;" ::: "memory");
              named_bar_sync(2, kHeadProducers);
              const int nci = ci + 1 < C2 ? ci + 1 : 0;
              float* dst = sm + G::OFF_W_UP2 + ((ring_step + 1) & 1) * G::STAGE;
              const float* src = p.w_up2 + (size_t)nci * G::STAGE;
              for (int i = pt; i < G::STAGE / 4; i += kHeadProducers) tma::cp_async16(dst + 4 * i, src + 4 * i);
              asm volatile("cp.async.commit_group;" ::: "memory");
              Wci = sm + G::OFF_W_UP2 + (ring_step & 1) * G::STAGE;
              ++ring_step;
            } else {
              Wci = Wres + ci * G::STAGE;
            }
            if (!active) continue;
            const float* in_c = in_t + (size_t)ci * 16 * kSpPlane;
            const float* w_c = Wci + w_off;
            if (cy == 0) {
              if (nkz == 3) head_up2_channel<C3, 0, 3>(acc, in_c, w_c);
              else if (nkz == 2) head_up2_channel<C3, 0, 2>(acc, in_c, w_c);
              else head_up2_channel<C3, 0, 1>(acc, in_c, w_c);
            } else {
              if (nkz == 3) head_up2_channel<C3, 1, 3>(acc, in_c, w_c);
              else if (nkz == 2) head_up2_channel<C3, 1, 2>(acc, in_c, w_c);
              else head_up2_channel<C3, 1, 1>(acc, in_c, w_c);
            }
          }
          if (active) {
            const float* bias = sm + G::OFF_BIAS + cohp * 8;
#pragma unroll
            for (int c = 0; c < 8; ++c) {
              float* o = U + (cohp * 8 + c) * G::U_PLANE + l * G::U_PITCH + 8 * q;
              const float bb = bias[c];
              float v[8];
#pragma unroll
              for (int j = 0; j < 8; ++j) v[j] = relu(((c & 1) ? p2_hi(acc[c >> 1][j]) : p2_lo(acc[c >> 1][j])) + bb);
              st4(o, v[0], v[1], v[2], v[3]);
              if (q < 4) st4(o + 4, v[4], v[5], v[6], v[7]);
            }
          }
        }
        mbar_arrive(&bars[it & 1]);              // slice complete (release: the stores above are visible to the waiters)
      }
    }
  }
  if (G::RING) asm volatile("cp.async.wait_group 0;" ::: "memory");
}

template <int C2, int C3>
__global__ void __launch_bounds__(kHeadThreads, 1) k_decode_head(HeadParams p) {
  using G = HeadCfg<C2, C3>;
  extern __shared__ __align__(128) float sm[];
  const int tid = threadIdx.x;
  uint64_t* bars = reinterpret_cast<uint64_t*>(sm + G::OFF_BAR);   // full[0], full[1], empty[0], empty[1]
  for (int i = tid * 4; i < G::W_C2; i += kHeadThreads * 4) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p.w_c2 + i));
    *reinterpret_cast<float4*>(sm + G::OFF_W_C2 + i) = v;
  }
  for (int i = tid * 4; i < G::W_CLS; i += kHeadThreads * 4) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p.w_cls + i));
    *reinterpret_cast<float4*>(sm + G::OFF_W_CLS + i) = v;
  }
  if (!G::RING)
    for (int i = tid * 4; i < G::W_UP2; i += kHeadThreads * 4) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(p.w_up2 + i));
      *reinterpret_cast<float4*>(sm + G::OFF_W_UP2 + i) = v;
    }
  if (tid < C3) sm[G::OFF_BIAS + tid] = p.up2_b[tid];
  else if (tid < 2 * C3) sm[G::OFF_BIAS + tid] = p.conv2_b[tid - C3];
  else if (tid < 2 * C3 + 4) sm[G::OFF_BIAS + tid] = p.cls2_b[0];
  for (int i = tid; i < G::C_SIZE; i += kHeadThreads) sm[G::OFF_C + i] = 0.f;   // halo rows / columns stay zero
  if (tid == 0) {
    tma::mbar_init(&bars[0], kHeadProducers);
    tma::mbar_init(&bars[1], kHeadProducers);
    tma::mbar_init(&bars[2], kHeadConsumers);
    tma::mbar_init(&bars[3], kHeadConsumers);
    tma::fence_barrier_init();
  }
  __syncthreads();
  if (tid >= kHeadConsumers) {
    reg_dec<136>();
    head_producer<C2, C3>(p, sm, bars, tid - kHeadConsumers);
  } else {
    reg_inc<184>();
    head_consumer<C2, C3>(p, sm, bars, tid);
  }
}

// Wide configuration: the two logit rows next to the cut between the y passes (rows 15 and 16).  Each pass left the
// row's partial logits (its own two conv2 tap rows) in `pl` and its own conv2 row in `brow`; add the third tap row
// from the other pass's conv2 row, then sigmoid / threshold / mask word / point count as in the head kernel.
template <int C3>
__global__ void __launch_bounds__(256) k_head_fixup(HeadParams p) {
  constexpr int RY = 16;
  __shared__ float s_w[C3 * 36];
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  for (int i = tid; i < C3 * 36; i += 256) s_w[i] = p.w_cls[i];
  __syncthreads();
  const float cls_b = p.cls2_b[0];
  int cnt = 0;
  for (int idx = tid; idx < 2048; idx += 256) {
    const int x = idx & 31, zl = (idx >> 5) & 31, pp = idx >> 10;       // pp: pass that owns the row
    float v = p.pl[(size_t)b * 2048 + idx];
    const float* nb = p.brow + ((size_t)b * 2 + (1 - pp)) * C3 * 1024;   // the other pass's conv2 row [ci][z][x]
    const int ky = pp == 0 ? 2 : 0;
    for (int ci = 0; ci < C3; ++ci)
#pragma unroll
      for (int kz = 0; kz < 3; ++kz) {
        const int z1 = zl + kz - 1;
        if (z1 < 0 || z1 > 31) continue;
        const float* wr = s_w + (ci * 3 + ky) * 12 + kz * 4;
        const float* row = nb + ((size_t)ci * 32 + z1) * 32;
#pragma unroll
        for (int kx = 0; kx < 3; ++kx) {
          const int xx = x + kx - 1;
          if (xx >= 0 && xx < 32) v = fmaf(wr[kx], row[xx], v);
        }
      }
    const float pr = sigmoidf(v + cls_b);
    const uint32_t word = __ballot_sync(0xffffffffu, pr > p.thh);
    const int Yb = pp == 0 ? RY - 1 : RY;
    if (p.prob_out) p.prob_out[(size_t)b * kVox + (zl * 32 + Yb) * 32 + x] = pr;
    if (lane == 0) {
      p.mask_out[(size_t)b * 1024 + zl * 32 + Yb] = word;
      cnt += __popc(word);
    }
  }
  if (cnt) atomicAdd(p.counts_out + b, cnt);
}

// [planes][DIN][DIN] -> zero-padded [planes][DIN+4][DIN+8], data at rows 2.., columns 4.. (one float4 of the
// destination per thread): the layout the polyphase transposed-conv tiles read their 6-float windows from
template <int DIN>
__global__ void __launch_bounds__(256) k_pad_in(const float* __restrict__ src, float* __restrict__ dst, long long planes) {
  constexpr int ROWS = DIN + 4, P4 = (DIN + 8) / 4, PL4 = ROWS * P4;
  const long long total = planes * PL4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long pl = i / PL4;
    const int r4 = (int)(i - pl * PL4);
    const int row = r4 / P4, c4 = r4 - row * P4;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row >= 2 && row < DIN + 2 && c4 >= 1 && c4 <= DIN / 4)
      v = __ldg(reinterpret_cast<const float4*>(src + pl * (DIN * DIN) + (row - 2) * DIN + (c4 - 1) * 4));
    reinterpret_cast<float4*>(dst)[i] = v;
  }
}

// Stand-alone polyphase k=5 stride-2 transposed conv + ReLU (up1 of the decode stem): the head producer's thread tile (8 x = 4 even + 4 odd outputs, 8 output channels) with one
// WARP ITEM per (leaf, row parity, output slice, channel group, group of RPW rows): up to 32 tiles of equal tap count.
// Weights stay resident in shared memory when they fit 72 KB - the warps then pull items independently and never
// meet - else they stream through a two-stage cp.async ring, one input channel at a time, and the four warps of a CTA
// walk their four consecutive items channel by channel together.
template <int CI, int CO, int DIN>
struct PolyCfg {
  static_assert(CO == 8 || CO == 16, "channel groups of 8");
  static constexpr int DOUT = 2 * DIN + 3, OP = (DOUT + 3) / 4 * 4;
  static constexpr int PROWS = DIN + 4, PPITCH = DIN + 8, PPLANE = PROWS * PPITCH;
  static constexpr int COH = CO / 8;
  static constexpr int NE = (DOUT + 1) / 2, NO = DOUT / 2, XT = (DOUT + 7) / 8;
  static constexpr int RPW = 32 / XT;                      // rows of one warp item
  static constexpr int RG = (NE + RPW - 1) / RPW;          // row groups per (slice, parity)
  static_assert((NO + RPW - 1) / RPW == RG, "same number of row groups for both parities");
  static constexpr int WPL = 2 * DOUT * COH * RG;          // warp items per leaf, ordered [row parity][slice: even z, then odd z][channel group][row group]
  static constexpr int STAGE = 125 * CO;
  static constexpr bool RING = CI * STAGE * 4 > 72 * 1024;
  static constexpr int SMEM_BYTES = (RING ? 2 : CI) * STAGE * 4;
  // resident weights: 8 independent warps share one copy of the weights, two CTAs (16 warps, 128 registers) per SM;
  // ring: four lock-step warps per CTA, four CTAs per SM
  static constexpr int THREADS = RING ? 128 : 256, WARPS = THREADS / 32;
  static constexpr int MINB = RING ? 4 : 2;
};

struct PolyParams {
  const float* inp;    // padded input [n][CI][DIN][DIN+4][DIN+8]
  float* out;          // [n][CO][DOUT][DOUT][OP], columns >= DOUT written as zero
  const float* w;      // [CI][5][5][5][CO]
  const float* bias;   // [CO]
  int32_t n;
};

template <int CI, int CO, int DIN>
__global__ void __launch_bounds__((PolyCfg<CI, CO, DIN>::THREADS), (PolyCfg<CI, CO, DIN>::MINB)) k_convT5_poly(PolyParams p) {
  using G = PolyCfg<CI, CO, DIN>;
  extern __shared__ __align__(128) float sm[];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = lane % G::XT, rl = lane / G::XT;            // x tile and row inside the group
  uint32_t ring_step = 0;
  for (int i = tid; i < (G::RING ? 1 : CI) * G::STAGE / 4; i += G::THREADS) tma::cp_async16(sm + 4 * i, p.w + 4 * i);
  asm volatile("cp.async.commit_group;" ::: "memory");
  if (!G::RING) {
    asm volatile("cp.async.wait_group 0;" ::: "memory");
    __syncthreads();
  }
  const long long total = (long long)p.n * G::WPL;
  // RING: the CTA's warps take four consecutive items per round (same number of rounds for every warp of the CTA);
  // resident weights: every warp strides over the items on its own
  const long long first = (long long)blockIdx.x * G::WARPS + warp, stride = (long long)gridDim.x * G::WARPS;
  const long long rounds = (total + stride - 1) / stride;
#pragma unroll 1
  for (long long rd = 0; rd < rounds; ++rd) {
    const long long wi = first + rd * stride;
    const bool have = wi < total;
    if (!G::RING && !have) break;
    int b = 0, cy = 0, s = 0, coh = 0, rg = 0;
    if (have) {
      b = (int)(wi / G::WPL);
      int r = (int)(wi - (long long)b * G::WPL);
      rg = r % G::RG; r /= G::RG;
      coh = r % G::COH; r /= G::COH;
      const int j = r % G::DOUT;                            // slices of equal z parity (equal kz tap count) are neighbours,
      s = j < G::NE ? 2 * j : 2 * (j - G::NE) + 1;          // so the four items a CTA walks in step cost the same
      cy = r / G::DOUT;
    }
    const int nrows = cy ? G::NO : G::NE;
    const int rr = rg * G::RPW + rl;
    const bool active = have && rl < G::RPW && rr < nrows;
    const int l = 2 * rr + cy;                              // output row
    // valid kz taps: kz = kz0, kz0+2, .. with 0 <= (s - kz) / 2 <= DIN-1
    int kz0 = s & 1;
    while (s - kz0 > 2 * (DIN - 1)) kz0 += 2;
    int nkz = 0;
    for (int kz = kz0; kz < 5 && kz <= s; kz += 2) ++nkz;
    p2 acc[4][8];
#pragma unroll
    for (int c = 0; c < 4; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[c][j] = p2_bcast(0.f);
    const float* in_t = p.inp + (size_t)b * CI * DIN * G::PPLANE +
                        ((size_t)((s - kz0) >> 1) * G::PROWS + (active ? rr + 2 : 2)) * G::PPITCH + 4 * q + 2;
    const int w_off = ((kz0 * 5 + cy) * 5) * CO + coh * 8;
#pragma unroll 1
    for (int ci = 0; ci < CI; ++ci) {
      const float* w_c;
      if (G::RING) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();                                    // stage ring_step & 1 holds channel ci; the other is free
        const int nci = ci + 1 < CI ? ci + 1 : 0;
        float* dst = sm + ((ring_step + 1) & 1) * G::STAGE;
        const float* src = p.w + (size_t)nci * G::STAGE;
        for (int i = tid; i < G::STAGE / 4; i += G::THREADS) tma::cp_async16(dst + 4 * i, src + 4 * i);
        asm volatile("cp.async.commit_group;" ::: "memory");
        w_c = sm + (ring_step & 1) * G::STAGE + w_off;
        ++ring_step;
      } else {
        w_c = sm + ci * G::STAGE + w_off;
      }
      if (!active) continue;
      const float* in_c = in_t + (size_t)ci * DIN * G::PPLANE;
      if (cy == 0) up2_channel_loop<CO, 0, G::PPLANE, G::PPITCH>(acc, in_c, w_c, nkz);
      else up2_channel_loop<CO, 1, G::PPLANE, G::PPITCH>(acc, in_c, w_c, nkz);
    }
    if (active) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const int co = coh * 8 + c;
        const float bb = __ldg(p.bias + co);
        float* o = p.out + (((size_t)b * CO + co) * G::DOUT + s) * G::DOUT * G::OP + (size_t)l * G::OP + 8 * q;
        float v[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float r = relu(((c & 1) ? p2_hi(acc[c >> 1][j]) : p2_lo(acc[c >> 1][j])) + bb);
          v[j] = 8 * q + j < G::DOUT ? r : 0.f;
        }
        st4(o, v[0], v[1], v[2], v[3]);
        if (8 * q + 4 < G::OP) st4(o + 4, v[4], v[5], v[6], v[7]);
      }
    }
  }
  asm volatile("cp.async.wait_group 0;" ::: "memory");
}

// conv1 output [n][C][16][16][16] -> zero-padded [n][C][16][20][24] (one float4 of the destination per thread)
__global__ void __launch_bounds__(256) k_pad_conv1(const float* __restrict__ src, float* __restrict__ dst, long long planes) {
  const long long total = planes * (kSpPlane / 4);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const long long pl = i / (kSpPlane / 4);
    const int r4 = (int)(i - pl * (kSpPlane / 4));
    const int row = r4 / (kSpPitch / 4), c4 = r4 - row * (kSpPitch / 4);
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row >= 2 && row < 18 && c4 >= 1 && c4 < 5)
      v = __ldg(reinterpret_cast<const float4*>(src + pl * 256 + (row - 2) * 16 + (c4 - 1) * 4));
    reinterpret_cast<float4*>(dst)[i] = v;
  }
}

}  // namespace fast
}  // namespace nvf
