// Shared definitions for the NVF B200 kernels.
//
// All kernel bodies are written as host/device templates so that the exact
// same index arithmetic can be executed (a) on the GPU by nvf_capi.cu and
// (b) sequentially on the CPU by the test-only emulator tests/emu/nvf_emu.cpp
// (used by the `-m "not gpu"` tests to check kernel logic before GPU time is
// spent; it is never part of the product library).
#pragma once

#include <stdint.h>
#include <math.h>

#if defined(__CUDACC__)
#define NVF_HD __host__ __device__ __forceinline__
#define NVF_D __device__ __forceinline__
#else
#define NVF_HD inline
#define NVF_D inline
#endif

#if defined(__CUDA_ARCH__)
#define NVF_UNROLL _Pragma("unroll")
#define NVF_NOUNROLL _Pragma("unroll 1")
#else
#define NVF_UNROLL
#define NVF_NOUNROLL
#endif

namespace nvf {

constexpr int kThreads = 256;   // CTA size of every kernel in this library
constexpr int kLeaf = 32;       // leaf block edge (get_octree.cpp:788, level-5 leaves of a 1024 root)
constexpr int kVox = kLeaf * kLeaf * kLeaf;

struct f4 {
  float x, y, z, w;
};

NVF_HD f4 ld4(const float* p) {
#if defined(__CUDA_ARCH__)
  float4 v = *reinterpret_cast<const float4*>(p);
  return f4{v.x, v.y, v.z, v.w};
#else
  return f4{p[0], p[1], p[2], p[3]};
#endif
}
NVF_HD void st4(float* p, float a, float b, float c, float d) {
#if defined(__CUDA_ARCH__)
  *reinterpret_cast<float4*>(p) = make_float4(a, b, c, d);
#else
  p[0] = a; p[1] = b; p[2] = c; p[3] = d;
#endif
}
NVF_HD void ld2(const float* p, float& a, float& b) {
#if defined(__CUDA_ARCH__)
  float2 v = *reinterpret_cast<const float2*>(p);
  a = v.x; b = v.y;
#else
  a = p[0]; b = p[1];
#endif
}


// ---------------------------------------------------------------------------
// Packed pair of fp32 values living in one aligned 64-bit register pair, and the
// Blackwell two-wide FMA (PTX fma.rn.f32x2 -> SASS FFMA2): each half is an IEEE
// fmaf, so results are bit-identical to two scalar fmaf calls, but one warp
// instruction feeds the FP32 pipe for two cycles - the issue slot freed every
// other cycle is what the LDS / address instructions of the conv loops need.
// On the host (CPU emulator) it is a plain struct.
// ---------------------------------------------------------------------------
#if defined(__CUDA_ARCH__)
typedef unsigned long long p2;
NVF_D p2 p2_make(float lo, float hi) {
  p2 r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
NVF_D p2 p2_bcast(float a) { return p2_make(a, a); }
NVF_D float p2_lo(p2 v) {
  [[maybe_unused]] float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
  (void)hi;
  return lo;
}
NVF_D float p2_hi(p2 v) {
  [[maybe_unused]] float lo, hi;
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
  (void)lo;
  return hi;
}
// acc = a * b + acc (per half)
NVF_D void p2_fma(p2& acc, p2 a, p2 b) { asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc) : "l"(a), "l"(b)); }
// four consecutive floats (16-byte aligned) -> pairs (p[0],p[1]) and (p[2],p[3]) with one 128-bit load
NVF_D void p2_ld2(const float* p, p2& a, p2& b) {
  const ulonglong2 v = *reinterpret_cast<const ulonglong2*>(p);
  a = v.x;
  b = v.y;
}
#else
struct p2 {
  [[maybe_unused]] float lo, hi;
};
NVF_HD p2 p2_make(float lo, float hi) { return p2{lo, hi}; }
NVF_HD p2 p2_bcast(float a) { return p2{a, a}; }
NVF_HD float p2_lo(p2 v) { return v.lo; }
NVF_HD float p2_hi(p2 v) { return v.hi; }
NVF_HD void p2_fma(p2& acc, p2 a, p2 b) {
  acc.lo = fmaf(a.lo, b.lo, acc.lo);
  acc.hi = fmaf(a.hi, b.hi, acc.hi);
}
NVF_HD void p2_ld2(const float* p, p2& a, p2& b) {
  a = p2{p[0], p[1]};
  b = p2{p[2], p[3]};
}
#endif
// eight consecutive output-channel weights -> four channel pairs
NVF_HD void p2_load_w8(const float* wp, p2 (&w)[4]) {
  p2_ld2(wp, w[0], w[1]);
  p2_ld2(wp + 4, w[2], w[3]);
}

NVF_HD float relu(float v) { return v > 0.f ? v : 0.f; }
// torch.sigmoid in fp32: 1/(1+exp(-x))
NVF_HD float sigmoidf(float v) { return 1.f / (1.f + expf(-v)); }

NVF_HD void atomic_add_f32(float* p, float v) {
#if defined(__CUDA_ARCH__)
  atomicAdd(p, v);
#else
  *p += v;
#endif
}
NVF_HD void atomic_add_f64(double* p, double v) {
#if defined(__CUDA_ARCH__)
  atomicAdd(p, v);
#else
  *p += v;
#endif
}
NVF_HD int popc32(uint32_t v) {
#if defined(__CUDA_ARCH__)
  return __popc(v);
#else
  return __builtin_popcount(v);
#endif
}

// ---------------------------------------------------------------------------
// Packed weight layouts.  Every convolution kernel is re-laid-out (once per
// call, 52k-201k floats) as  Wp[cin][kz][ky][kx][cout]  so that the inner loop
// fetches all output channels of one tap with broadcast 128-bit loads.
// ---------------------------------------------------------------------------
enum PackMode {
  PACK_CONV_FWD = 0,    // src (Co,Ci,K,K,K)  -> dst[ci][k][co]            (conv forward)
  PACK_CONVT_FWD = 1,   // src (Ci,Co,K,K,K)  -> dst[ci][k][co]            (convT forward)
  PACK_CONV_DGRAD = 2,  // src (Co,Ci,K,K,K)  -> dst[co][K-1-k][ci]        (dX = full corr of g with flipped W)
  PACK_CONVT_DGRAD = 3, // src (Ci,Co,K,K,K)  -> dst[co][k][ci]            (dX = stride-2 corr of g with W)
  PACK_CLS_IS = 4       // src (1,Ci,3,3,3)   -> dst[ci][ky][kz][4(kx,pad)]  (input-stationary cls head)
};

struct PackJob {
  const float* src;
  float* dst;
  int32_t mode, A, B, K;  // A,B = first two dims of src
};
constexpr int kMaxPackJobs = 24;
struct PackParams {
  PackJob job[kMaxPackJobs];
  int32_t njobs;
};

// only_job >= 0: this thread works on that job alone (the GPU launches one grid row per job, so the jobs'
// load -> store latencies overlap instead of adding up)
NVF_HD void pack_thread(const PackParams& p, int gtid, int gthreads, int only_job = -1) {
  for (int j = (only_job >= 0 ? only_job : 0); j < (only_job >= 0 ? only_job + 1 : p.njobs); ++j) {
    const PackJob& J = p.job[j];
    const int K3 = J.K * J.K * J.K;
    const int n = J.A * J.B * K3;
    if (J.mode == PACK_CLS_IS) {
      // dst[ci][ky][kz][4]
      const int nd = J.B * 3 * 3 * 4;
      for (int i = gtid; i < nd; i += gthreads) {
        int kx = i & 3, kz = (i >> 2) % 3, ky = (i / 12) % 3, ci = i / 36;
        J.dst[i] = (kx < 3) ? J.src[ci * 27 + kz * 9 + ky * 3 + kx] : 0.f;
      }
      continue;
    }
    for (int i = gtid; i < n; i += gthreads) {
      // i indexes dst
      float v;
      if (J.mode == PACK_CONV_FWD) {          // dst[ci][k][co], A=Co,B=Ci
        int co = i % J.A, k = (i / J.A) % K3, ci = i / (J.A * K3);
        v = J.src[(co * J.B + ci) * K3 + k];
      } else if (J.mode == PACK_CONVT_FWD) {  // dst[ci][k][co], A=Ci,B=Co
        int co = i % J.B, k = (i / J.B) % K3, ci = i / (J.B * K3);
        v = J.src[(ci * J.B + co) * K3 + k];
      } else if (J.mode == PACK_CONV_DGRAD) { // dst[co][kf][ci], A=Co,B=Ci
        int ci = i % J.B, kf = (i / J.B) % K3, co = i / (J.B * K3);
        int kz = kf / (J.K * J.K), ky = (kf / J.K) % J.K, kx = kf % J.K;
        int k = ((J.K - 1 - kz) * J.K + (J.K - 1 - ky)) * J.K + (J.K - 1 - kx);
        v = J.src[(co * J.B + ci) * K3 + k];
      } else {                                // PACK_CONVT_DGRAD dst[co][k][ci], A=Ci,B=Co
        int ci = i % J.A, k = (i / J.A) % K3, co = i / (J.A * K3);
        v = J.src[(ci * J.B + co) * K3 + k];
      }
      J.dst[i] = v;
    }
  }
}

}  // namespace nvf
