// Per-thread register-tile routines for the three convolution families of the
// NVF decoder.  Every routine computes COT output channels x 4 consecutive
// outputs along x for ONE (z,y) position, reading packed weights
// Wp[cin][kz][ky][kx][cout] (nvf_common.h) with 128-bit loads.
//
// Maths restated from the reference's library calls (SURVEY.md 3.4 / 3.5):
//   conv   (F.conv3d,            utils/network.py:687,741):
//       y[co,z] = b[co] + sum_ci sum_k x[ci, z + k - P] * W[co,ci,k]
//   convT  (F.conv_transpose3d,  utils/network.py:621), stride 2, k 5:
//       y[co,o] = b[co] + sum_ci sum_{k : (o+P-k) even, 0 <= (o+P-k)/2 < Din}
//                                   x[ci,(o+P-k)/2] * W[ci,co,k]
//   convT dgrad = stride-2 correlation:
//       dx[ci,i] = sum_co sum_k g[co, 2i - P + k] * W[ci,co,k]
#pragma once
#include "nvf_common.h"

namespace nvf {

// Input tensor view: element (c,z,y,x) at base[c*cs + z*zs + y*ys + x]; valid
// coordinates are [0,d) on every axis (out-of-range reads are zero padding).
struct View {
  const float* base;
  int cs, zs, ys, d;
};

template <int COT>
NVF_HD void zero_acc(float (&acc)[COT][4]) {
  NVF_UNROLL
  for (int c = 0; c < COT; ++c) {
    NVF_UNROLL
    for (int j = 0; j < 4; ++j) acc[c][j] = 0.f;
  }
}

template <int COT>
NVF_HD void load_w(const float* wp, float (&w)[COT]) {
  static_assert(COT % 4 == 0 || COT == 1, "COT");
  if (COT == 1) {
    w[0] = wp[0];
  } else {
    NVF_UNROLL
    for (int c = 0; c < COT; c += 4) {
      f4 v = ld4(wp + c);
      w[c] = v.x; w[c + 1] = v.y; w[c + 2] = v.z; w[c + 3] = v.w;
    }
  }
}

// Stride-1 correlation with zero padding P (bounds-checked scalar loads):
// acc[c][j] += sum_ci sum_k in[ci, oz+kz-P, oy+ky-P, ox0+j+kx-P] * Wp[ci][k][co0+c]
template <int K, int COT>
NVF_HD void corr_s1_tile(const View& in, int CI, int P, const float* Wp, int CO, int co0, int oz, int oy, int ox0,
                         float (&acc)[COT][4]) {
  NVF_NOUNROLL
  for (int ci = 0; ci < CI; ++ci) {
    NVF_NOUNROLL
    for (int kz = 0; kz < K; ++kz) {
      const int iz = oz + kz - P;
      if (iz < 0 || iz >= in.d) continue;
      NVF_NOUNROLL
      for (int ky = 0; ky < K; ++ky) {
        const int iy = oy + ky - P;
        if (iy < 0 || iy >= in.d) continue;
        const float* row = in.base + ci * in.cs + iz * in.zs + iy * in.ys;
        float a[K + 3];
        NVF_UNROLL
        for (int i = 0; i < K + 3; ++i) {
          const int ix = ox0 + i - P;
          a[i] = (ix >= 0 && ix < in.d) ? row[ix] : 0.f;
        }
        const float* wrow = Wp + (((ci * K + kz) * K + ky) * K) * CO + co0;
        NVF_UNROLL
        for (int kx = 0; kx < K; ++kx) {
          float w[COT];
          load_w<COT>(wrow + kx * CO, w);
          NVF_UNROLL
          for (int c = 0; c < COT; ++c) {
            NVF_UNROLL
            for (int j = 0; j < 4; ++j) acc[c][j] = fmaf(w[c], a[j + kx], acc[c][j]);
          }
        }
      }
    }
  }
}

// Transposed conv k5 s2, padding P in {0,2}: 4 consecutive outputs ox0..ox0+3
// (ox0 % 4 == 0, so outputs 0,2 use even kx and 1,3 odd kx).
template <int COT>
NVF_HD void convT5_tile(const View& in, int CI, int P, const float* Wp, int CO, int co0, int oz, int oy, int ox0,
                        float (&acc)[COT][4]) {
  const int m0 = (ox0 + P) >> 1;  // input index of output ox0 at kx = 0
  NVF_NOUNROLL
  for (int ci = 0; ci < CI; ++ci) {
    NVF_NOUNROLL
    for (int kz = (oz + P) & 1; kz < 5; kz += 2) {
      const int tz = oz + P - kz;
      if (tz < 0) break;
      const int iz = tz >> 1;
      if (iz >= in.d) continue;
      NVF_NOUNROLL
      for (int ky = (oy + P) & 1; ky < 5; ky += 2) {
        const int ty = oy + P - ky;
        if (ty < 0) break;
        const int iy = ty >> 1;
        if (iy >= in.d) continue;
        const float* row = in.base + ci * in.cs + iz * in.zs + iy * in.ys;
        float a[4];  // inputs m0-2 .. m0+1
        NVF_UNROLL
        for (int i = 0; i < 4; ++i) {
          const int ix = m0 - 2 + i;
          a[i] = (ix >= 0 && ix < in.d) ? row[ix] : 0.f;
        }
        const float* wrow = Wp + (((ci * 5 + kz) * 5 + ky) * 5) * CO + co0;
        NVF_UNROLL
        for (int kx = 0; kx < 5; ++kx) {
          float w[COT];
          load_w<COT>(wrow + kx * CO, w);
          const int h = kx >> 1;
          NVF_UNROLL
          for (int c = 0; c < COT; ++c) {
            if ((kx & 1) == 0) {
              acc[c][0] = fmaf(w[c], a[2 - h], acc[c][0]);
              acc[c][2] = fmaf(w[c], a[3 - h], acc[c][2]);
            } else {
              acc[c][1] = fmaf(w[c], a[2 - h], acc[c][1]);
              acc[c][3] = fmaf(w[c], a[3 - h], acc[c][3]);
            }
          }
        }
      }
    }
  }
}

// Stride-2 correlation k5 (dgrad of the transposed conv): for outputs i = ox0..ox0+3
// acc[c][j] += sum_ci sum_k in[ci, 2*oz-P+kz, 2*oy-P+ky, 2*(ox0+j)-P+kx] * Wp[ci][k][co0+c]
template <int COT>
NVF_HD void corr_s2_tile(const View& in, int CI, int P, const float* Wp, int CO, int co0, int oz, int oy, int ox0,
                         float (&acc)[COT][4]) {
  NVF_NOUNROLL
  for (int ci = 0; ci < CI; ++ci) {
    NVF_NOUNROLL
    for (int kz = 0; kz < 5; ++kz) {
      const int iz = 2 * oz - P + kz;
      if (iz < 0 || iz >= in.d) continue;
      NVF_NOUNROLL
      for (int ky = 0; ky < 5; ++ky) {
        const int iy = 2 * oy - P + ky;
        if (iy < 0 || iy >= in.d) continue;
        const float* row = in.base + ci * in.cs + iz * in.zs + iy * in.ys;
        float a[11];
        NVF_UNROLL
        for (int i = 0; i < 11; ++i) {
          const int ix = 2 * ox0 - P + i;
          a[i] = (ix >= 0 && ix < in.d) ? row[ix] : 0.f;
        }
        const float* wrow = Wp + (((ci * 5 + kz) * 5 + ky) * 5) * CO + co0;
        NVF_UNROLL
        for (int kx = 0; kx < 5; ++kx) {
          float w[COT];
          load_w<COT>(wrow + kx * CO, w);
          NVF_UNROLL
          for (int c = 0; c < COT; ++c) {
            NVF_UNROLL
            for (int j = 0; j < 4; ++j) acc[c][j] = fmaf(w[c], a[2 * j + kx], acc[c][j]);
          }
        }
      }
    }
  }
}

}  // namespace nvf
