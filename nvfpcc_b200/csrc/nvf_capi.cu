// C ABI (include/nvf_b200.h) + CUDA launchers for sm_100a.
// Build: nvcc -gencode arch=compute_100a,code=sm_100a -lineinfo -O3 -shared -Xcompiler -fPIC
#include <cuda_runtime.h>
#include <stdio.h>
#include <string.h>
#include <stdlib.h>
#include <atomic>

#include "nvf_api_impl.h"
#include "nvf_fast_conv.cuh"
#include "nvf_fast_dgrad4.cuh"
#include "nvf_fast_convt.cuh"
#include "nvf_fast_misc.cuh"
#include "nvf_fast_stem.cuh"
#include "nvf_fast_params.cuh"
#include "nvf_fast_latent.cuh"
#include "nvf_step.cuh"
#include "nvf_rows_convt.cuh"
#include "nvf_decode_head.cuh"
#include "nvf_symm.cuh"

namespace nvf {
std::atomic<long long> g_launches{0};  // kernels launched by this library (bench.py: gpu_launches); shared with nvf_prep.cu
}

using namespace nvf;

namespace {

thread_local int g_last_cuda = 0;

// One auxiliary non-blocking stream + a ring of timing-free events per device, created lazily:
// independent kernels of one call (weight gradients vs. the data-gradient chain, the auxiliary
// heads) are forked onto it and joined back before the call returns, also under stream capture.
constexpr int kMaxDevices = 16, kEventRing = 64;
struct SidePool {
  cudaStream_t stream = nullptr;
  cudaEvent_t ev[kEventRing] = {};
  int next = 0;
  bool ready = false;
};
SidePool g_side[kMaxDevices];

template <class... KArgs, class... Args>
void nvf_launch(void (*k)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args&&... args) {
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchKernelEx(&cfg, k, KArgs(args)...);   // errors are picked up by the caller's cudaGetLastError()
}

template <class TS>
struct DevEnv {
  TS ts;
  template <class F>
  __device__ __forceinline__ void phase(F&& f) {
    f((int)threadIdx.x, ts);
    __syncthreads();
  }
};

// ------------------------------------------------------------------ kernels
__global__ void __launch_bounds__(kThreads) k_pack(PackParams p) {
  pack_thread(p, blockIdx.x * blockDim.x + threadIdx.x, gridDim.x * blockDim.x, (int)blockIdx.y);
}

__global__ void __launch_bounds__(kThreads) k_scan_counts(EmitParams p) {
  __shared__ int64_t sm[2 * kThreads];
  DevEnv<int> env;
  ScanBlock<DevEnv<int>>::run(env, p, sm);
}

__global__ void __launch_bounds__(kThreads) k_emit_coords(EmitParams p) {
  __shared__ int sm[2 * kThreads];
  DevEnv<int> env;
  EmitBlock<DevEnv<int>>::run(env, p, sm, blockIdx.x);
}

template <class K>
__global__ void __launch_bounds__(kThreads) k_generic(typename K::Params p) {
  K::thread(p, blockIdx.x, threadIdx.x, gridDim.x);
}

template <int COT, int K>
__global__ void __launch_bounds__(kThreads) k_wgrad(WgradParams p) {
  extern __shared__ __align__(128) float smem[];
  DevEnv<int> env;
  WgradBlock<COT, K>::run(env, p, smem, blockIdx.x);
}

__global__ void __launch_bounds__(kThreads) k_chansum(ChanSumParams p) {
  __shared__ float sm[kThreads];
  DevEnv<int> env;
  ChanSumBlock::run(env, p, sm, blockIdx.x);
}

__global__ void __launch_bounds__(kThreads) k_mask(MaskParams p) {
  __shared__ int sm[kThreads];
  DevEnv<int> env;
  MaskBlock::run(env, p, sm, blockIdx.x);
}

__global__ void __launch_bounds__(kThreads) k_loss(LossParams p) {
  __shared__ double sm[kThreads * NVF_LOSS_SUMS];
  DevEnv<int> env;
  LossBlock::run(env, p, sm, blockIdx.x);
}

// FFMA throughput probes.  variant 0: scalar FFMA, 8x8 register tile (the shape
// of the conv inner loops); variant 1: packed fma.rn.f32x2 on the same tile.
__global__ void __launch_bounds__(kThreads) k_ffma(int variant, long long iters, float* sink) {
  float w[8], a[8];
  for (int i = 0; i < 8; ++i) {
    w[i] = 1.0f + 1e-6f * (threadIdx.x + i);
    a[i] = 0.5f + 1e-6f * (blockIdx.x + i);
  }
  if (variant == 0) {
    float acc[8][8];
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[c][j] = 0.f;
    for (long long it = 0; it < iters; ++it) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
#pragma unroll
        for (int c = 0; c < 8; ++c)
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[c][j] = fmaf(w[c], a[(j + r) & 7], acc[c][j]);
      }
    }
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int j = 0; j < 8; ++j) s += acc[c][j];
    sink[blockIdx.x * blockDim.x + threadIdx.x] = s;
  } else {
    unsigned long long acc[8][4], ww[8], aa[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      asm("mov.b64 %0, {%1, %1};" : "=l"(ww[c]) : "f"(w[c]));
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[c][j] = 0ull;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) asm("mov.b64 %0, {%1, %2};" : "=l"(aa[j]) : "f"(a[j]), "f"(a[(j + 1) & 7]));
    for (long long it = 0; it < iters; ++it) {
#pragma unroll
      for (int r = 0; r < 4; ++r) {
#pragma unroll
        for (int c = 0; c < 8; ++c)
#pragma unroll
          for (int j = 0; j < 4; ++j)
            asm volatile("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(acc[c][j]) : "l"(ww[c]), "l"(aa[(2 * j + r) & 7]));
      }
    }
    float s = 0.f;
#pragma unroll
    for (int c = 0; c < 8; ++c)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        float lo, hi;
        asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(acc[c][j]));
        s += lo + hi;
      }
    sink[blockIdx.x * blockDim.x + threadIdx.x] = s;
  }
}

// ------------------------------------------------------------------ launcher
struct DevLauncher {
  cudaStream_t st;      // stream kernels are launched on (the caller's stream, or the side stream inside a fork)
  int n_sms = 0;
  int rc = NVF_OK;
  cudaStream_t main_st = nullptr;
  SidePool* pool = nullptr;
  bool forked = false;

  // ---- fork / join of independent work onto the auxiliary stream
  cudaEvent_t next_event() {
    cudaEvent_t e = pool->ev[pool->next];
    pool->next = (pool->next + 1) % kEventRing;
    return e;
  }
  void side_begin() {   // subsequent launches run on the side stream, after everything launched so far
    if (!pool || !pool->ready) return;
    cudaEvent_t e = next_event();
    if (!chk(cudaEventRecord(e, main_st)) || !chk(cudaStreamWaitEvent(pool->stream, e, 0))) return;
    st = pool->stream;
    forked = true;
  }
  void side_end() { st = main_st; }
  void join() {         // the caller's stream waits for all forked work
    if (!forked) return;
    cudaEvent_t e = next_event();
    if (chk(cudaEventRecord(e, pool->stream))) chk(cudaStreamWaitEvent(main_st, e, 0));
    forked = false;
  }

  int init() {
    int dev = 0, major = 0;
    main_st = st;
    if (!chk(cudaGetDevice(&dev))) return rc;
    if (dev >= 0 && dev < kMaxDevices) {
      SidePool& P = g_side[dev];
      if (!P.ready) {
        bool ok = cudaStreamCreateWithFlags(&P.stream, cudaStreamNonBlocking) == cudaSuccess;
        for (int i = 0; ok && i < kEventRing; ++i) ok = cudaEventCreateWithFlags(&P.ev[i], cudaEventDisableTiming) == cudaSuccess;
        P.ready = ok;
        if (!ok) cudaGetLastError();   // run without forking
      }
      pool = &P;
    }
    if (!chk(cudaDeviceGetAttribute(&n_sms, cudaDevAttrMultiProcessorCount, dev))) return rc;
    if (!chk(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev))) return rc;
    if (major != 10) rc = NVF_ERR_NO_DEVICE;
    return rc;
  }
  bool chk(cudaError_t e) {
    if (e != cudaSuccess) {
      g_last_cuda = (int)e;
      if (rc == NVF_OK) rc = (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? NVF_ERR_NO_DEVICE : NVF_ERR_CUDA;
      return false;
    }
    return true;
  }
  void post() {
    chk(cudaGetLastError());
    g_launches.fetch_add(1, std::memory_order_relaxed);
  }
  int sms() const { return n_sms; }
  int error() const { return rc; }

  void pack(const PackParams& p) {
    if (p.njobs <= 0) return;
    nvf_launch(k_pack, dim3(32, p.njobs), dim3(kThreads), (size_t)(0), st, p);   // one grid row per job
    post();
  }
  bool has_head(const NvfDesc& d) { return head_cfg(d); }
  void zero_ints(int32_t* p, int64_t n) { chk(cudaMemsetAsync(p, 0, sizeof(int32_t) * (size_t)n, st)); }
  void pad_conv1(const float* src, float* dst, int64_t planes) {
    int64_t grid = (planes * (fast::kSpPlane / 4) + 255) / 256;
    if (grid > (int64_t)n_sms * 16) grid = (int64_t)n_sms * 16;
    nvf_launch(fast::k_pad_conv1, dim3((unsigned)grid), dim3(256), (size_t)0, st, src, dst, (long long)planes);
    post();
  }
  template <int CI, int CO, int DIN>
  bool poly_t(const LayerParams& p, float* pad) {
    using G = fast::PolyCfg<CI, CO, DIN>;
    auto* k = fast::k_convT5_poly<CI, CO, DIN>;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    const long long planes = (long long)p.n * CI * DIN;
    long long g0 = (planes * (G::PPLANE / 4) + 255) / 256;
    if (g0 > (long long)n_sms * 16) g0 = (long long)n_sms * 16;
    nvf_launch(fast::k_pad_in<DIN>, dim3((unsigned)g0), dim3(256), (size_t)0, st, p.in, pad, planes);
    post();
    fast::PolyParams q{pad, p.out, p.Wp, p.bias, p.n};
    long long grid = ((long long)p.n * G::WPL + G::WARPS - 1) / G::WARPS;
    if (grid > (long long)n_sms * G::MINB) grid = (long long)n_sms * G::MINB;
    nvf_launch(k, dim3((unsigned)grid), dim3(G::THREADS), (size_t)G::SMEM_BYTES, st, q);
    post();
    return true;
  }
  // up1 of the decode stem: polyphase kernel on a zero-padded copy of the input; false = not instantiated for this
  // shape.  Decode uses it for EVERY batch size (a leaf's result must not depend on it).
  bool up_poly(const LayerParams& p, float* pad) {
    if (p.act != ACT_RELU || p.op != OP_CONVT || p.P != 0 || p.Din != 8) return false;
    // measured on B200, 1247 leaves, vs the tile kernel: 32 -> 16 channels 5.51 -> 3.73 ms, 16 -> 8 channels 1.28 -> 0.98 ms
    if (p.CI == 32 && p.CO == 16) return poly_t<32, 16, 8>(p, pad);
    if (p.CI == 16 && p.CO == 8) return poly_t<16, 8, 8>(p, pad);
    return false;
  }
  template <int C2, int C3>
  void head_t(const HeadArgs& a, int grid) {
    using G = fast::HeadCfg<C2, C3>;
    auto* k = fast::k_decode_head<C2, C3>;
    if (!smem_attr(k, G::SMEM_BYTES)) return;
    fast::HeadParams p{a.sp, a.w_up2, a.w_c2, a.w_cls, a.up2_b, a.conv2_b, a.cls2_b, a.prob_out, a.mask_out,
                       a.counts_out, G::COH == 2 ? a.brow : nullptr, G::COH == 2 ? a.pl : nullptr, a.thh, a.n_blocks};
    nvf_launch(k, dim3(grid), dim3(fast::kHeadThreads), (size_t)G::SMEM_BYTES, st, p);
    post();
    if (G::COH == 2) {
      nvf_launch(fast::k_head_fixup<C3>, dim3(a.n_blocks), dim3(256), (size_t)0, st, p);
      post();
    }
  }
  void head(const NvfDesc& d, const HeadArgs& a, int grid) {
    if (d.c3 == 8) head_t<8, 8>(a, grid);
    else head_t<16, 16>(a, grid);
  }
  void scan(const EmitParams& p) { nvf_launch(k_scan_counts, dim3(1), dim3(kThreads), (size_t)(0), st, p); post(); }
  void emit(const EmitParams& p, int grid) { nvf_launch(k_emit_coords, dim3(grid), dim3(kThreads), (size_t)(0), st, p); post(); }
  template <int COT>
  void layer(const LayerParams& p) {
    const int64_t XT = (p.Dout + 3) >> 2;
    const int64_t total = (int64_t)(p.CO / COT) * p.Dout * p.Dout * XT * p.n;
    int64_t grid = (total + kThreads - 1) / kThreads;
    const int64_t cap = (int64_t)n_sms * 32;
    if (grid > cap) grid = cap;
    if (grid < 1) grid = 1;
    nvf_launch(k_generic<LayerKernel<COT>>, dim3((unsigned)grid), dim3(kThreads), (size_t)(0), st, p);
    post();
  }
  template <int COT, int K>
  void wgrad(const WgradParams& p, int grid) {
    const int smem = kThreads * COT * K * (int)sizeof(float);
    nvf_launch(k_wgrad<COT, K>, dim3(grid), dim3(kThreads), (size_t)(smem), st, p);
    post();
  }
  void chansum(const ChanSumParams& p, int grid) { nvf_launch(k_chansum, dim3(grid), dim3(kThreads), (size_t)(0), st, p); post(); }
  template <class K>
  void generic(const typename K::Params& p, int grid) {
    nvf_launch(k_generic<K>, dim3(grid < 1 ? 1 : grid), dim3(kThreads), (size_t)(0), st, p);
    post();
  }
  void mask(const MaskParams& p, int grid) { nvf_launch(k_mask, dim3(grid), dim3(kThreads), (size_t)(0), st, p); post(); }
  void loss(const LossParams& p, int grid) { nvf_launch(k_loss, dim3(grid), dim3(kThreads), (size_t)(0), st, p); post(); }

  // ---- shared-memory tiled kernels of the training path (nvf_fast_*.cuh) --------------------
  float* part_base = nullptr;   // scratch for split-K partial results (bump allocated per call)
  size_t part_off = 0, part_cap = 0;
  fast::ReduceParams red{};     // pending fixed-order reductions, flushed by flush_reduce()

  // work-queue words of the queue-fed kernels: 16 bytes per launch, zero on entry (the kernels rewind them)
  unsigned int* queue_base = nullptr;
  int queue_next = 0;
  void set_queue(void* base) { queue_base = (unsigned int*)base; queue_next = 0; }
  void zero_queue(void* base, size_t bytes) { chk(cudaMemsetAsync(base, 0, bytes, st)); }
  unsigned int* take_queue() {
    if (!queue_base || queue_next >= kQueueSlots) return nullptr;
    return queue_base + 4 * (queue_next++);
  }
  void set_partial(float* base, size_t floats) { part_base = base; part_cap = floats; part_off = 0; }
  float* take_partial(size_t floats) {
    floats = (floats + 63) / 64 * 64;
    if (!part_base || part_off + floats > part_cap) return nullptr;
    float* r = part_base + part_off;
    part_off += floats;
    return r;
  }
  void add_reduce(const fast::ReduceJob& j) {
    if (red.njobs == fast::kMaxReduceJobs) flush_reduce();
    red.job[red.njobs++] = j;
  }
  void flush_reduce() {
    if (!red.njobs) return;
    int nmax = 0;
    for (int i = 0; i < red.njobs; ++i) nmax = red.job[i].n_w + red.job[i].n_b > nmax ? red.job[i].n_w + red.job[i].n_b : nmax;
    int gx = (nmax + 31) / 32;
    if (gx > 1024) gx = 1024;
    nvf_launch(fast::k_reduce_partials, dim3(dim3(gx, red.njobs)), dim3(256), (size_t)(0), st, red);
    post();
    red.njobs = 0;
  }
  template <class KernelT>
  bool smem_attr(KernelT* k, int bytes) {
    return chk(cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  }

  template <int K, int CI, int CO, int DIN, int PAD, int XG, int TY, int NZP, int CIC, int MINB, bool TMA = false, int COTP = 0>
  bool conv_s1(const LayerParams& p) {
    using G = fast::ConvS1Cfg<K, CI, CO, DIN, PAD, XG, TY, NZP, CIC, COTP>;
    constexpr int SMEM = TMA ? G::SMEM_BYTES_TMA : G::SMEM_BYTES;
    static_assert(SMEM <= 227 * 1024, "conv_s1 smem");
    auto* k = fast::k_conv_s1<K, CI, CO, DIN, PAD, XG, TY, NZP, CIC, MINB, TMA, COTP>;
    if (!smem_attr(k, SMEM)) return true;
    CUtensorMap map;
    memset(&map, 0, sizeof(map));
    if (TMA && !tma::make_map_5d(&map, p.in, p.n, CI, DIN, DIN, G::IN_PITCH, G::PI, G::TYI, G::TZI, CIC)) {
      if (rc == NVF_OK) rc = NVF_ERR_CUDA;    // no silent fallback: the TMA path is the product path
      return true;
    }
    fast::ConvS1Params q{p.in, p.out, p.out2, p.Wp, p.bias, p.mask, p.n, p.act};
    nvf_launch(k, dim3(p.n * G::TILES_Z * G::TILES_Y), dim3(G::THREADS), (size_t)(SMEM), st, map, q);
    post();
    return true;
  }
  template <int C, int D, int TZ, int TY, int MINB>
  bool conv4_dgrad(const LayerParams& p) {
    using G = fast::Dgrad4Cfg<C, D, TZ, TY>;
    static_assert(G::SMEM_BYTES <= 227 * 1024, "conv4 dgrad smem");
    auto* k = fast::k_conv4_dgrad<C, D, TZ, TY, MINB>;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    fast::Dgrad4Params q{p.in, p.out, p.Wp, p.mask, p.n};
    nvf_launch(k, dim3(p.n * G::TILES_Z * G::TILES_Y), dim3(G::THREADS), (size_t)(G::SMEM_BYTES), st, q);
    post();
    return true;
  }
  template <int CI, int CO, int DIN, int MINB, int KS = 1>
  bool convT_fwd(const LayerParams& p) {
    using G = fast::ConvTFwdCfg<CI, CO, DIN, KS>;
    static_assert(G::SMEM_BYTES <= 227 * 1024, "convT fwd smem");
    auto* k = fast::k_convT5_fwd<CI, CO, DIN, MINB, KS>;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    fast::ConvTFwdParams q{p.in, p.out, p.Wp, p.bias, p.n};
    nvf_launch(k, dim3(p.n * G::DOUT), dim3(G::THREADS), (size_t)(G::SMEM_BYTES), st, q);
    post();
    return true;
  }
  template <int CI, int CO, int DIN, int KS, int THREADS, int MINB, bool PIPE = false, bool CHUNK = true>
  bool convT_fwd_rows(const LayerParams& p) {
    using G = fast::RowTFwdCfg<CI, CO, DIN, KS>;
    static_assert(G::SMEM_BYTES <= 226 * 1024 / MINB, "row-tile convT weights");
    unsigned int* q = take_queue();
    if (!q) return false;
    auto* k = fast::k_convT5_fwd_rows<CI, CO, DIN, KS, THREADS, MINB, PIPE, CHUNK>;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    fast::RowTFwdParams a{p.in, p.out, p.Wp, p.bias, q, p.n};
    int grid = n_sms * MINB;
    const int need = (p.n * G::ITEMS_PER_BLOCK + THREADS / 32 - 1) / (THREADS / 32);
    if (grid > need) grid = need;
    nvf_launch(k, dim3(grid), dim3(THREADS), (size_t)(G::SMEM_BYTES), st, a);
    post();
    return true;
  }
  template <int CG, int CX, int DIN, int TY, int CGC, int MINB>
  bool convT_dgrad(const LayerParams& p) {
    using G = fast::ConvTDgradCfg<CG, CX, DIN, TY, CGC>;
    static_assert(G::SMEM_BYTES <= 227 * 1024, "convT dgrad smem");
    auto* k = fast::k_convT5_dgrad<CG, CX, DIN, TY, CGC, MINB>;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    fast::ConvTDgradParams q{p.in, p.out, p.Wp, p.add, p.mask, p.n};
    nvf_launch(k, dim3(p.n * DIN * G::BANDS), dim3(G::THREADS), (size_t)(G::SMEM_BYTES), st, q);
    post();
    return true;
  }
  // returns true when a tiled kernel handled the layer
  bool fast_layer(const LayerParams& p) {
    if (p.n <= 0) return false;
    if (p.op == OP_CORR4 && p.CI == p.CO && !p.add && !p.out2 && p.act != ACT_SIGMOID) {
      const bool fwd = p.P == 0 && !p.mask, dg = p.P == 3 && p.mask && !p.bias && p.act == ACT_NONE;
      if (p.CI == 8) {
        if (fwd && p.Din == 35) return conv_s1<4, 8, 8, 35, 0, 8, 16, 2, 2, 2, true>(p);
        if (dg && p.Din == 32) return conv4_dgrad<8, 32, 1, 7, 4>(p);
        if (fwd && p.Din == 19) return conv_s1<4, 8, 8, 19, 0, 4, 8, 1, 2, 6, true, 4>(p);
        if (dg && p.Din == 16) return conv4_dgrad<8, 16, 1, 5, 5>(p);
      } else if (p.CI == 16) {
        if (fwd && p.Din == 35) return conv_s1<4, 16, 16, 35, 0, 8, 16, 1, 4, 2>(p);
        if (dg && p.Din == 32) return conv4_dgrad<16, 32, 3, 7, 1>(p);
        if (fwd && p.Din == 19) return conv_s1<4, 16, 16, 19, 0, 4, 8, 2, 4, 2>(p);
        if (dg && p.Din == 16) return conv4_dgrad<16, 16, 2, 5, 2>(p);
      }
      return false;
    }
    if (p.op == OP_CORR3 && p.P == 1 && !p.add) {
      if (p.CI == 1 && !p.out2 && p.act == ACT_NONE) {           // classifier data gradient 1 -> C
        if (p.CO == 8 && p.Din == 32) return conv_s1<3, 1, 8, 32, 1, 8, 16, 2, 1, 2>(p);
        if (p.CO == 8 && p.Din == 16) return conv_s1<3, 1, 8, 16, 1, 4, 8, 2, 1, 4>(p);
        if (p.CO == 16 && p.Din == 8) return conv_s1<3, 1, 16, 8, 1, 2, 8, 1, 1, 4>(p);
        if (p.CO == 16 && p.Din == 32) return conv_s1<3, 1, 16, 32, 1, 8, 16, 1, 1, 2>(p);
        if (p.CO == 16 && p.Din == 16) return conv_s1<3, 1, 16, 16, 1, 4, 8, 2, 1, 4>(p);
        if (p.CO == 32 && p.Din == 8) return conv_s1<3, 1, 32, 8, 1, 2, 8, 1, 1, 4>(p);
      } else if (p.CO == 1 && !p.mask) {                          // classifier forward C -> 1
        if (p.CI == 8 && p.Din == 32) return conv_s1<3, 8, 1, 32, 1, 8, 16, 2, 4, 2>(p);
        if (p.CI == 8 && p.Din == 16) return conv_s1<3, 8, 1, 16, 1, 4, 8, 2, 4, 4>(p);
        if (p.CI == 16 && p.Din == 8) return conv_s1<3, 16, 1, 8, 1, 2, 8, 2, 8, 4>(p);
        if (p.CI == 16 && p.Din == 32) return conv_s1<3, 16, 1, 32, 1, 8, 16, 2, 4, 2>(p);
        if (p.CI == 16 && p.Din == 16) return conv_s1<3, 16, 1, 16, 1, 4, 8, 2, 4, 4>(p);
        if (p.CI == 32 && p.Din == 8) return conv_s1<3, 32, 1, 8, 1, 2, 8, 2, 8, 4>(p);
      }
      return false;
    }
    if (p.op == OP_CONVT && p.P == 0 && p.act == ACT_RELU && !p.add && !p.mask && !p.out2) {
      // up2 on the queue-fed row kernels (no queue slot: the generic kernel).  Measured on B200 (16-block step): up2
      // (8,8,16) 60 -> 54 us against the tile kernel; up1 (16,8,8) loses (25 -> 33 us: too little work per warp item
      // against the per-CTA weight staging), so it stays on the tile kernel
      if (p.CI == 8 && p.CO == 8 && p.Din == 16) return convT_fwd_rows<8, 8, 16, 2, 256, 2, false, false>(p);
      if (p.CI == 16 && p.CO == 16 && p.Din == 16) return convT_fwd_rows<16, 16, 16, 2, 256, 1>(p);
      if (p.CI == 16 && p.CO == 8 && p.Din == 8) return convT_fwd<16, 8, 8, 2, 4>(p);
      if (p.CI == 32 && p.CO == 16 && p.Din == 8) return convT_fwd<32, 16, 8, 1>(p);
      return false;
    }
    if (p.op == OP_CORR_S2 && p.P == 0 && p.act == ACT_NONE && !p.bias && !p.out2) {
      if (p.CI == 8 && p.CO == 8 && p.Dout == 16) return convT_dgrad<8, 8, 16, 16, 1, 2>(p);
      if (p.CI == 8 && p.CO == 16 && p.Dout == 8) return convT_dgrad<8, 16, 8, 8, 1, 2>(p);
      if (p.CI == 16 && p.CO == 16 && p.Dout == 16) return convT_dgrad<16, 16, 16, 16, 1, 1>(p);
      if (p.CI == 16 && p.CO == 32 && p.Dout == 8) return convT_dgrad<16, 32, 8, 8, 1, 1>(p);
      return false;
    }
    return false;
  }

  template <int C, int DG, int TYG, int MINB>
  bool wgrad4(const WgradParams& p, float* db) {
    using G = fast::WgradS1Cfg<C, DG, TYG>;
    auto* k = fast::k_wgrad4_s1<C, DG, TYG, MINB>;
    const int items = p.n * DG * G::BANDS;
    int grid = n_sms * MINB;
    if (grid > items) grid = items;
    float* partial = take_partial((size_t)grid * G::OUT_FLOATS);
    if (!partial) return false;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    fast::WgradS1Params q{p.A, p.Sft, partial, p.n};
    nvf_launch(k, dim3(grid), dim3(256), (size_t)(G::SMEM_BYTES), st, q);
    post();
    add_reduce(fast::ReduceJob{partial, p.dW, db, grid, G::OUT_FLOATS, G::NW, C, 0, 0});
    return true;
  }
  bool chansum_fast(const ChanSumParams& c) {
    if (c.pitch % 4) return false;
    const int zch = c.D >= 16 ? 4 : 1;
    float* partial = take_partial((size_t)c.n * zch * c.C);
    if (!partial) return false;
    fast::ChanSumFastParams q{c.g, partial, c.n, c.C, c.D, c.pitch, zch};
    nvf_launch(fast::k_chansum_fast, dim3(c.n * zch * c.C), dim3(256), (size_t)(0), st, q);
    post();
    add_reduce(fast::ReduceJob{partial, c.out, nullptr, c.n * zch, c.C, c.C, 0, 0, 0});
    return true;
  }
  template <int CI, int CO, int DIN, int TYB, int CIB, int MINB>
  bool convT_wgrad(const WgradParams& p, const ChanSumParams& c) {
    using G = fast::ConvTWgradCfg<CI, CO, DIN, TYB, CIB>;
    static_assert(G::SMEM_BYTES <= 227 * 1024, "convT wgrad smem");
    auto* k = fast::k_convT5_wgrad<CI, CO, DIN, TYB, CIB, MINB>;
    const int items = p.n * DIN * G::BANDS;
    int grid = (n_sms * MINB + G::GROUPS - 1) / G::GROUPS;
    if (grid > items) grid = items;
    if (grid * G::GROUPS > kMaxPartialCtas) grid = kMaxPartialCtas / G::GROUPS;
    // persistent CTAs: the same number on every SM (304 CTAs on 148 SMs would leave eight SMs with three CTAs
    // while the others hold two, and the kernel ends with those eight)
    if (grid * G::GROUPS > n_sms) grid = (grid * G::GROUPS / n_sms) * n_sms / G::GROUPS;
    float* partial = take_partial((size_t)grid * G::GROUPS * G::OUT_FLOATS);
    if (!partial) return false;
    if (!chansum_fast(c)) return false;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    fast::ConvTWgradParams q{p.A, p.Sft, partial, p.n};
    nvf_launch(k, dim3(dim3(grid, G::GROUPS)), dim3(224), (size_t)(G::SMEM_BYTES), st, q);
    post();
    for (int grp = 0; grp < G::GROUPS; ++grp) {
      const int cog = grp % (CO / 8), cig = grp / (CO / 8);
      // partial rows [ci_local][co_local 8][125] -> dW[(cig*CIB + ci)][cog*8 + co][125]
      add_reduce(fast::ReduceJob{partial + (size_t)grp * grid * G::OUT_FLOATS,
                                 p.dW + ((size_t)cig * CIB * CO + cog * 8) * 125, nullptr, grid, G::OUT_FLOATS,
                                 G::OUT_FLOATS, 0, 8 * 125, CO * 125});
    }
    return true;
  }
  template <int C, int D, int TYB, int ZSEG>
  bool cls_wgrad(const WgradParams& p, float* db) {
    using G = fast::ClsWgradCfg<C, D, TYB, ZSEG>;
    auto* k = fast::k_cls_wgrad<C, D, TYB, ZSEG>;
    const int grid = p.n * G::BANDS * G::SEGS;
    float* partial = take_partial((size_t)grid * G::OUT_FLOATS);
    if (!partial) return false;
    if (!smem_attr(k, G::SMEM_BYTES)) return true;
    fast::ClsWgradParams q{p.A, p.Sft, partial, p.n};
    nvf_launch(k, dim3(grid), dim3(256), (size_t)(G::SMEM_BYTES), st, q);
    post();
    add_reduce(fast::ReduceJob{partial, p.dW, db, grid, G::OUT_FLOATS, G::NW, 1, 0, 0});
    return true;
  }
  // weight + bias gradient of one layer; false = not handled (the generic kernels run instead)
  bool fast_wgrad(const WgradParams& p, const ChanSumParams& c) {
    if (p.n <= 0 || !c.out) return false;
    if (p.K == 4 && p.S == 1 && p.CA == p.CS && p.P == 0) {
      if (p.CA == 8 && p.Da == 32) return wgrad4<8, 32, 8, 2>(p, c.out);
      if (p.CA == 8 && p.Da == 16) return wgrad4<8, 16, 8, 2>(p, c.out);
      if (p.CA == 16 && p.Da == 32) return wgrad4<16, 32, 4, 2>(p, c.out);
      if (p.CA == 16 && p.Da == 16) return wgrad4<16, 16, 4, 2>(p, c.out);
      return false;
    }
    if (p.K == 5 && p.S == 2 && p.P == 0) {
      if (p.CA == 8 && p.CS == 8 && p.Da == 16) return convT_wgrad<8, 8, 16, 4, 8, 3>(p, c);
      if (p.CA == 16 && p.CS == 8 && p.Da == 8) return convT_wgrad<16, 8, 8, 4, 16, 2>(p, c);
      if (p.CA == 16 && p.CS == 16 && p.Da == 16) return convT_wgrad<16, 16, 16, 4, 16, 2>(p, c);
      if (p.CA == 32 && p.CS == 16 && p.Da == 8) return convT_wgrad<32, 16, 8, 4, 16, 2>(p, c);
      return false;
    }
    if (p.K == 3 && p.S == 1 && p.P == 1 && p.CA == 1) {
      if (p.CS == 8 && p.Da == 32) return cls_wgrad<8, 32, 16, 4>(p, c.out);
      if (p.CS == 8 && p.Da == 16) return cls_wgrad<8, 16, 16, 4>(p, c.out);
      if (p.CS == 16 && p.Da == 8) return cls_wgrad<16, 8, 8, 4>(p, c.out);
      if (p.CS == 16 && p.Da == 32) return cls_wgrad<16, 32, 16, 4>(p, c.out);
      if (p.CS == 16 && p.Da == 16) return cls_wgrad<16, 16, 16, 4>(p, c.out);
      return false;
    }
    return false;
  }
  // stem (everything at <= 8^3): one CTA per block, see nvf_fast_stem.cuh
  bool fast_stem_fwd(const NvfDesc& d, const NvfWeights& w, const float* up0_wp, const float* conv0_wp,
                     const float* cls0_wp, const float* latent, int n, float* x0, float* a0, float* a1, float* cls0,
                     float* cls0_copy) {
    if (n <= 0 || d.c1 % 8 || d.c0 > 32) return false;
    const int smem = (d.ch * 8 + 2 * d.c0 * 64 + d.c0 * d.c0 + d.c0 + ((d.ch * 125 * d.c0 + 3) & ~3) + d.c0 * 75 * d.c1) *
                     (int)sizeof(float);
    if (smem > 200 * 1024) return false;
    fast::StemFwdParams q{latent, up0_wp, w.up0_b, w.igdn_beta, w.igdn_gamma, conv0_wp, w.conv0_b,
                          nullptr, nullptr, x0, a0, a1, nullptr, nullptr, n, d.ch, d.c0, d.c1};
    const int per_sm = smem > 110 * 1024 ? 1 : (smem > 56 * 1024 ? 2 : 4);   // resident 512-thread CTAs per SM
    if (n * 8 > n_sms * per_sm * 2) {     // more slice CTAs than two waves: persistent CTAs, weights staged once
      if (!smem_attr(fast::k_stem_fwd<true>, smem)) return true;
      int ctas = n_sms * per_sm & ~1;
      nvf_launch(fast::k_stem_fwd<true>, dim3(ctas), dim3(fast::kStemFwdThreads), (size_t)(smem), st, q);
    } else {
      if (!smem_attr(fast::k_stem_fwd<false>, smem)) return true;
      nvf_launch(fast::k_stem_fwd<false>, dim3(n * 8), dim3(fast::kStemFwdThreads), (size_t)(smem), st, q);
    }
    post();
    if (cls0) {   // conv0_cls + sigmoid: auxiliary head, off the critical path
      LayerParams p{a1, cls0, cls0_wp, w.cls0_b, nullptr, nullptr, n, d.c1, 1, 8, 8, 8, 8, 1, ACT_SIGMOID, OP_CORR3};
      p.out2 = cls0_copy;
      side_begin();
      const bool ok = fast_layer(p);
      side_end();
      if (!ok) { nvf_launch(k_generic<LayerKernel<1>>, dim3((n * 128 + kThreads - 1) / kThreads), dim3(kThreads), (size_t)(0), st, p); post(); }
    }
    return true;
  }
  bool fast_stem_bwd(const NvfDesc& d, const NvfWeights& w, const float* latent, int n, const float* x0,
                     const float* a0, const float* g1, float* gy0, const NvfWeightGrads* gw, float* g_latent) {
    if (n <= 0 || d.c1 % 8 || d.c0 > 32) return false;
    const int pf = fast::stem_partial_floats(d.ch, d.c0, d.c1);
    float* partial = nullptr;
    if (gw) {
      partial = take_partial((size_t)n * pf);
      if (!partial) return false;
    }
    const int smem_a = (d.c1 * 512 + 64 + 512 + d.c1 * 125) * (int)sizeof(float);
    const int smem_b = (4 * d.c0 * 64 + d.ch * 8 + d.c0 * d.c0 + d.c0 + d.ch * d.c0 * 125) * (int)sizeof(float);
    if (smem_a > 200 * 1024 || smem_b > 200 * 1024) return false;
    if (!smem_attr(fast::k_stem_bwd_a, smem_a) || !smem_attr(fast::k_stem_bwd_b, smem_b)) return true;
    fast::StemBwdParams q{latent, x0, a0, g1, w.igdn_beta, w.igdn_gamma, w.conv0_w, w.up0_w, partial, g_latent,
                          n, d.ch, d.c0, d.c1, gw ? 1 : 0};
    nvf_launch(fast::k_stem_bwd_a, dim3(n * d.c0), dim3(fast::kStemBwdAThreads), (size_t)(smem_a), st, q, gy0);
    post();
    nvf_launch(fast::k_stem_bwd_b, dim3(n), dim3(fast::kStemBwdBThreads), (size_t)(smem_b), st, q, gy0);
    post();
    if (gw) {
      const int n0 = d.c0 * d.c1 * 125, ng = d.c0 * d.c0, nu = d.ch * d.c0 * 125;
      add_reduce(fast::ReduceJob{partial, gw->conv0_w, gw->conv0_b, n, pf, n0, d.c1, 0, 0});
      add_reduce(fast::ReduceJob{partial + n0 + d.c1, gw->igdn_gamma, gw->igdn_beta, n, pf, ng, d.c0, 0, 0});
      add_reduce(fast::ReduceJob{partial + n0 + d.c1 + ng + d.c0, gw->up0_w, gw->up0_b, n, pf, nu, d.c0, 0, 0});
    }
    return true;
  }
  bool fast_igdn_param(const IgdnParams& ip) {
    if (!ip.dbeta || !ip.dgamma || ip.C > 32) return false;
    float* partial = take_partial((size_t)ip.n * (ip.C * ip.C + ip.C));
    if (!partial) return false;
    fast::IgdnParamParams q{ip.x, ip.g, ip.beta, ip.gamma, partial, ip.n, ip.C};
    nvf_launch(fast::k_igdn_param, dim3(ip.n), dim3(256), (size_t)(ip.C * 64 * 2 * sizeof(float)), st, q);
    post();
    add_reduce(fast::ReduceJob{partial, ip.dgamma, ip.dbeta, ip.n, ip.C * ip.C + ip.C, ip.C * ip.C, ip.C, 0, 0});
    return true;
  }
};

}  // namespace

// ------------------------------------------------------------------ C ABI
namespace nvf {
void note_cuda_error(int e) { g_last_cuda = e; }   // used by nvf_prep.cu
}

extern "C" {

int nvf_abi_version(void) { return NVF_ABI_VERSION; }

const char* nvf_strerror(int code) {
  switch (code) {
    case NVF_OK: return "ok";
    case NVF_ERR_INVALID_ARG: return "invalid argument";
    case NVF_ERR_UNSUPPORTED: return "unsupported channel configuration";
    case NVF_ERR_WORKSPACE: return "workspace too small";
    case NVF_ERR_CUDA: return "CUDA runtime error";
    case NVF_ERR_NO_DEVICE: return "no sm_100 device";
    case NVF_ERR_BITSTREAM: return "corrupt entropy-coded stream";
    default: return "unknown error";
  }
}

int nvf_last_cuda_error(void) { return g_last_cuda; }

long long nvf_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int nvf_has_fused_decode(const NvfDesc* desc) { return desc && head_cfg(*desc) ? 1 : 0; }

int nvf_workspace_bytes(const NvfDesc* desc, int64_t n_blocks, int mode, size_t* bytes_out) {
  if (!desc || !bytes_out || n_blocks < 0) return NVF_ERR_INVALID_ARG;
  if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
  if (mode == NVF_MODE_DECODE) *bytes_out = DecodeWs::make(*desc, n_blocks, head_cfg(*desc)).total;
  else if (mode == NVF_MODE_TRAIN) *bytes_out = TrainWs::make(*desc, n_blocks).total;
  else return NVF_ERR_INVALID_ARG;
  return NVF_OK;
}

int nvf_decode(const NvfDesc* desc, const NvfWeights* w, const float* latent, const int32_t* origins,
               int64_t n_blocks, float thh, float* prob_out, uint32_t* mask_out, int32_t* counts_out,
               int32_t* coords_out, int64_t cap, int64_t* total_out, void* workspace, size_t workspace_bytes,
               void* stream) {
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  return Api<DevLauncher>::decode(l, desc, w, latent, origins, n_blocks, thh, prob_out, mask_out, counts_out,
                                  coords_out, cap, total_out, workspace, workspace_bytes);
}

int nvf_emit_points(const uint32_t* mask, const int32_t* counts, const int32_t* origins, int64_t n_blocks,
                    int32_t* coords_out, int64_t cap, int64_t* total_out, void* workspace, size_t workspace_bytes,
                    void* stream) {
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  return Api<DevLauncher>::emit_points(l, mask, counts, origins, n_blocks, coords_out, cap, total_out, workspace,
                              workspace_bytes);
}

int nvf_train_forward(const NvfDesc* desc, const NvfWeights* w, const float* latent, int64_t n_blocks, float* out,
                      float* cls1, float* cls0, void* workspace, size_t workspace_bytes, void* stream) {
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  return Api<DevLauncher>::train_forward(l, desc, w, latent, n_blocks, out, cls1, cls0, workspace, workspace_bytes);
}

int nvf_loss_seeds(const float* out, const float* cls1, const float* cls0, const float* gt, const float* dist,
                   int64_t n_blocks, float alpha_main, float alpha_aux, float thh_metric, double* sums_out,
                   float* g_out, float* g_cls1, float* g_cls0, void* workspace, size_t workspace_bytes,
                   void* stream) {
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  return Api<DevLauncher>::loss_seeds(l, out, cls1, cls0, gt, dist, n_blocks, alpha_main, alpha_aux, thh_metric,
                                      sums_out, g_out, g_cls1, g_cls0, workspace, workspace_bytes);
}

int nvf_train_backward(const NvfDesc* desc, const NvfWeights* w, const float* latent, int64_t n_blocks,
                       const float* g_out, const float* g_cls1, const float* g_cls0, int flags,
                       const NvfWeightGrads* gw, float* g_latent, void* workspace, size_t workspace_bytes,
                       void* stream) {
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  return Api<DevLauncher>::train_backward(l, desc, w, latent, n_blocks, g_out, g_cls1, g_cls0, flags, gw, g_latent,
                                          workspace, workspace_bytes);
}

namespace {
// The job of each layer from its geometry and raw tensors; the callers add the gradient inputs, the outputs and the
// packed layouts.
int fill_param_jobs(const NvfDesc& d, const NvfParamSet& ps, fast::ParamPrepParams& pp) {
  int chunk = 0, noise0 = 0;
  for (int l = 0; l < NVF_NUM_CONV; ++l) {
    const ConvGeom c = conv_geom(d, l);
    fast::ParamJob& J = pp.job[l];
    if (!ps.kernel[l] || !ps.kernel_init[l] || !ps.b[l] || !ps.b_init[l]) return NVF_ERR_INVALID_ARG;
    J.kernel = ps.kernel[l]; J.init = ps.kernel_init[l]; J.b = ps.b[l]; J.b_init = ps.b_init[l];
    J.n = (int32_t)c.n(); J.nb = c.nb;
    J.chunk0 = chunk;
    J.nchunks = (J.n + fast::kParamChunk - 1) / fast::kParamChunk;
    chunk += J.nchunks;
    J.noise0 = noise0;
    if (l < NVF_NUM_QUANT) noise0 += J.n;
    J.A = c.A; J.B = c.B; J.K3 = c.K3(); J.convT = c.convT;   // read only when the job also packs (pk_fwd)
  }
  pp.total_chunks = chunk;
  pp.igdn_beta = ps.igdn_beta; pp.igdn_gamma = ps.igdn_gamma;
  pp.lik_sigma = ps.lik_sigma; pp.lik_mu = ps.lik_mu;
  pp.c0 = d.c0;
  if (!ps.igdn_beta || !ps.igdn_gamma || !ps.lik_sigma || !ps.lik_mu) return NVF_ERR_INVALID_ARG;
  if ((size_t)chunk * 3 * sizeof(float) > NVF_PARAM_WS_BYTES) return NVF_ERR_UNSUPPORTED;
  return NVF_OK;
}
}  // namespace

int nvf_param_prep(const NvfDesc* desc, const NvfParamSet* params, int q, const float* noise, float beta_bound,
                   float gamma_bound, float pedestal, const NvfWeightGrads* eff, float* net_bits, void* workspace,
                   size_t workspace_bytes, void* stream) {
  if (!desc || !params || !eff || !net_bits || !workspace || q < 0 || q > 2) return NVF_ERR_INVALID_ARG;
  if (q == 1 && !noise) return NVF_ERR_INVALID_ARG;
  if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
  if (workspace_bytes < NVF_PARAM_WS_BYTES) return NVF_ERR_WORKSPACE;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  fast::ParamPrepParams pp{};
  int rc = fill_param_jobs(*desc, *params, pp);
  if (rc != NVF_OK) return rc;
  float* const* e = slots(*eff);
  for (int i = 0; i < NVF_NUM_CONV; ++i) {
    const int s = conv_geom(*desc, i).slot;
    if (!e[s] || !e[s + 1]) return NVF_ERR_INVALID_ARG;
    pp.job[i].w_out = e[s]; pp.job[i].b_out = e[s + 1];
  }
  if (!eff->igdn_beta || !eff->igdn_gamma) return NVF_ERR_INVALID_ARG;
  pp.beta_out = eff->igdn_beta; pp.gamma_out = eff->igdn_gamma;
  pp.noise = noise; pp.q = q;
  pp.partial = (float*)workspace; pp.net_bits = net_bits;
  pp.beta_bound = beta_bound; pp.gamma_bound = gamma_bound; pp.pedestal = pedestal;
  nvf_launch(fast::k_param_prep<false>, dim3(pp.total_chunks + 1), dim3(256), (size_t)(0), l.st, pp);
  l.post();
  nvf_launch(fast::k_param_final<false>, dim3(1), dim3(32), (size_t)(0), l.st, pp);
  l.post();
  return l.rc;
}

int nvf_param_prep_backward(const NvfDesc* desc, const NvfParamSet* params, float beta_bound, float gamma_bound,
                            const NvfWeights* g_eff, const float* g_net_bits, const NvfParamGrads* out,
                            void* workspace, size_t workspace_bytes, void* stream) {
  if (!desc || !params || !g_eff || !g_net_bits || !out || !workspace) return NVF_ERR_INVALID_ARG;
  if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
  if (workspace_bytes < NVF_PARAM_WS_BYTES) return NVF_ERR_WORKSPACE;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  fast::ParamPrepParams pp{};
  int rc = fill_param_jobs(*desc, *params, pp);
  if (rc != NVF_OK) return rc;
  const float* const* ge = slots(*g_eff);
  for (int i = 0; i < NVF_NUM_CONV; ++i) {
    const int s = conv_geom(*desc, i).slot;
    if (!ge[s] || !ge[s + 1] || !out->kernel[i] || !out->b[i]) return NVF_ERR_INVALID_ARG;
    pp.job[i].g_w = ge[s]; pp.job[i].g_b = ge[s + 1];
    pp.job[i].w_out = out->kernel[i]; pp.job[i].b_out = out->b[i];
  }
  if (!g_eff->igdn_beta || !g_eff->igdn_gamma || !out->igdn_beta || !out->igdn_gamma || !out->lik_sigma || !out->lik_mu)
    return NVF_ERR_INVALID_ARG;
  pp.g_beta = g_eff->igdn_beta; pp.g_gamma = g_eff->igdn_gamma;
  pp.beta_out = out->igdn_beta; pp.gamma_out = out->igdn_gamma;
  pp.g_bits = g_net_bits;
  pp.partial = (float*)workspace;
  pp.g_sigma = out->lik_sigma; pp.g_mu = out->lik_mu;
  pp.beta_bound = beta_bound; pp.gamma_bound = gamma_bound;
  nvf_launch(fast::k_param_prep<true>, dim3(pp.total_chunks + 1), dim3(256), (size_t)(0), l.st, pp);
  l.post();
  nvf_launch(fast::k_param_final<true>, dim3(1), dim3(32), (size_t)(0), l.st, pp);
  l.post();
  return l.rc;
}

}  // extern "C"

namespace {
template <int CH>
void launch_latent(DevLauncher& l, const fast::LatentKParams& kp, bool bwd) {
  int grid = (int)(((int64_t)kp.n * 8 + fast::kLatentThreads - 1) / fast::kLatentThreads);
  if (grid > fast::kLatentMaxCtas) grid = fast::kLatentMaxCtas;
  if (bwd) nvf_launch(fast::k_latent_bwd<CH>, dim3(grid), dim3(fast::kLatentThreads), (size_t)(0), l.st, kp);
  else nvf_launch(fast::k_latent_fwd<CH>, dim3(grid), dim3(fast::kLatentThreads), (size_t)(0), l.st, kp);
  l.post();
}
void launch_latent(DevLauncher& l, int ch, const fast::LatentKParams& kp, bool bwd) {
  switch (ch) {
    case 1: launch_latent<1>(l, kp, bwd); break;
    case 2: launch_latent<2>(l, kp, bwd); break;
    case 3: launch_latent<3>(l, kp, bwd); break;
    default: launch_latent<4>(l, kp, bwd); break;
  }
}
int latent_call(int ch, const NvfLatentParams* ps, const float* emb, const float* noise, float noise_scale, int train,
                int64_t n, float beta_bound, float gamma_bound, float pedestal, fast::LatentKParams& kp,
                void* workspace, size_t workspace_bytes, void* stream, bool bwd) {
  if (!ps || !emb || !workspace || n <= 0 || n > (1 << 24)) return NVF_ERR_INVALID_ARG;
  if (!ps->kernel || !ps->kernel_init || !ps->b || !ps->b_init || !ps->gdn_beta || !ps->gdn_gamma || !ps->sigma || !ps->mu)
    return NVF_ERR_INVALID_ARG;
  if (ch < 1 || ch > 4) return NVF_ERR_UNSUPPORTED;
  if (workspace_bytes < NVF_LATENT_WS_BYTES) return NVF_ERR_WORKSPACE;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  kp.emb = emb; kp.noise = noise;
  kp.kernel = ps->kernel; kp.kernel_init = ps->kernel_init; kp.b = ps->b; kp.b_init = ps->b_init;
  kp.beta = ps->gdn_beta; kp.gamma = ps->gdn_gamma; kp.sigma = ps->sigma; kp.mu = ps->mu;
  kp.beta_bound = beta_bound; kp.gamma_bound = gamma_bound; kp.pedestal = pedestal; kp.noise_scale = noise_scale;
  kp.n = (int32_t)n; kp.train = train ? 1 : 0;
  kp.ticket = (unsigned int*)workspace;
  kp.partial = (double*)((char*)workspace + 16);
  launch_latent(l, ch, kp, bwd);
  return l.rc;
}
}  // namespace

extern "C" {

int nvf_latent_forward(int ch, const NvfLatentParams* params, const float* emb, const float* noise, float noise_scale,
                       int train, int64_t n_blocks, float beta_bound, float gamma_bound, float pedestal,
                       float* latent_out, float* bits_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (!latent_out || !bits_out) return NVF_ERR_INVALID_ARG;
  fast::LatentKParams kp{};
  kp.latent = latent_out; kp.bits_out = bits_out;
  return latent_call(ch, params, emb, noise, noise_scale, train, n_blocks, beta_bound, gamma_bound, pedestal, kp,
                     workspace, workspace_bytes, stream, false);
}

int nvf_latent_backward(int ch, const NvfLatentParams* params, const float* emb, const float* noise,
                        float noise_scale, int train, int64_t n_blocks, float beta_bound, float gamma_bound,
                        float pedestal, const float* g_latent, const float* g_bits, const NvfLatentGrads* grads,
                        float* g_emb, void* workspace, size_t workspace_bytes, void* stream) {
  if (!g_bits || (!grads && !g_emb)) return NVF_ERR_INVALID_ARG;
  fast::LatentKParams kp{};
  kp.g_latent = g_latent; kp.g_bits = g_bits; kp.g_emb = g_emb;
  if (grads) {
    if (!grads->kernel || !grads->b || !grads->gdn_beta || !grads->gdn_gamma || !grads->sigma || !grads->mu)
      return NVF_ERR_INVALID_ARG;
    kp.gk = grads->kernel; kp.gb = grads->b; kp.gbeta = grads->gdn_beta; kp.ggamma = grads->gdn_gamma;
    kp.gsigma = grads->sigma; kp.gmu = grads->mu;
  }
  return latent_call(ch, params, emb, noise, noise_scale, train, n_blocks, beta_bound, gamma_bound, pedestal, kp,
                     workspace, workspace_bytes, stream, true);
}

int nvf_rd_total(const double* sums, const float* latent_bits, const float* net_bits, const float* n_pts,
                 float n_total, float lmbda, float w1, float w2, float* loss_out, float* stats_out, void* stream) {
  if (!sums || !latent_bits || !net_bits || !n_pts || !loss_out) return NVF_ERR_INVALID_ARG;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  fast::RdTotalParams p{};
  p.sums = sums; p.latent_bits = latent_bits; p.net_bits = net_bits; p.n_pts = n_pts;
  p.n_total = n_total; p.lmbda = lmbda; p.w1 = w1; p.w2 = w2;
  p.loss = loss_out; p.stats = stats_out;
  nvf_launch(fast::k_rd_total<false>, dim3(1), dim3(32), (size_t)(0), l.st, p);
  l.post();
  return l.rc;
}

int nvf_rd_total_backward(const float* g_loss, const float* n_pts, float n_total, float lmbda, float w1, float w2,
                          float* g_dist, float* g_latent_bits, float* g_net_bits, void* stream) {
  if (!g_loss || !n_pts || !g_dist || !g_latent_bits || !g_net_bits) return NVF_ERR_INVALID_ARG;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  fast::RdTotalParams p{};
  p.g_loss = g_loss; p.n_pts = n_pts; p.n_total = n_total; p.lmbda = lmbda; p.w1 = w1; p.w2 = w2;
  p.g_dist = g_dist; p.g_latent_bits = g_latent_bits; p.g_net_bits = g_net_bits;
  nvf_launch(fast::k_rd_total<true>, dim3(1), dim3(32), (size_t)(0), l.st, p);
  l.post();
  return l.rc;
}

int nvf_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float* step,
                  const float* lr, float beta1, float beta2, float eps, void* stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq || !step || !lr || n <= 0) return NVF_ERR_INVALID_ARG;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  fast::AdamParams p{param, grad, exp_avg, exp_avg_sq, step, lr, beta1, beta2, eps, n};
  int grid = (int)((n + 255) / 256);
  if (grid > l.n_sms * 4) grid = l.n_sms * 4;
  nvf_launch(fast::k_adam, dim3(grid), dim3(256), (size_t)(0), l.st, p);
  l.post();
  nvf_launch(fast::k_adam_tick, dim3(1), dim3(1), (size_t)(0), l.st, step);
  l.post();
  return l.rc;
}

size_t nvf_symm_bytes(int64_t n) {
  return (size_t)fast::kSymmHeaderBytes + 2 * sizeof(float) * 4 * (size_t)((n + 3) / 4);
}

int nvf_symm_alloc(size_t bytes, void** ptr_out, void* handle64_out) {
  if (!ptr_out || !handle64_out || bytes < (size_t)fast::kSymmHeaderBytes) return NVF_ERR_INVALID_ARG;
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
  void* p = nullptr;
  cudaError_t e = cudaMalloc(&p, bytes);
  if (e == cudaSuccess) e = cudaMemset(p, 0, bytes);
  cudaIpcMemHandle_t h;
  if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
  if (e != cudaSuccess) {
    g_last_cuda = (int)e;
    cudaGetLastError();
    if (p) cudaFree(p);
    return NVF_ERR_CUDA;
  }
  memcpy(handle64_out, &h, 64);
  *ptr_out = p;
  return NVF_OK;
}

int nvf_symm_open(const void* handle64, void** ptr_out) {
  if (!handle64 || !ptr_out) return NVF_ERR_INVALID_ARG;
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  void* p = nullptr;
  const cudaError_t e = cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess);
  if (e != cudaSuccess) {
    g_last_cuda = (int)e;
    cudaGetLastError();
    return NVF_ERR_CUDA;
  }
  *ptr_out = p;
  return NVF_OK;
}

int nvf_symm_close(void* ptr) {
  if (!ptr) return NVF_ERR_INVALID_ARG;
  const cudaError_t e = cudaIpcCloseMemHandle(ptr);
  if (e != cudaSuccess) { g_last_cuda = (int)e; cudaGetLastError(); return NVF_ERR_CUDA; }
  return NVF_OK;
}

int nvf_symm_free(void* ptr) {
  if (!ptr) return NVF_ERR_INVALID_ARG;
  const cudaError_t e = cudaFree(ptr);
  if (e != cudaSuccess) { g_last_cuda = (int)e; cudaGetLastError(); return NVF_ERR_CUDA; }
  return NVF_OK;
}

int nvf_adam_allreduce_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n, float* step,
                            const float* lr, float beta1, float beta2, float eps, void* const* peers, int rank,
                            int world, void* ctl, void* stream) {
  if (!param || !grad || !exp_avg || !exp_avg_sq || !step || !lr || !peers || !ctl || n <= 0 || n > (1 << 30))
    return NVF_ERR_INVALID_ARG;
  if (world < 1 || world > fast::kSymmMaxRanks || rank < 0 || rank >= world) return NVF_ERR_INVALID_ARG;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  fast::ArAdamParams p{};
  p.param = param; p.grad = grad; p.m = exp_avg; p.v = exp_avg_sq; p.step = step; p.lr = lr;
  p.beta1 = beta1; p.beta2 = beta2; p.eps = eps;
  p.n = (int32_t)n; p.n4 = (int32_t)((n + 3) / 4);
  p.rank = rank; p.world = world; p.ctl = (unsigned int*)ctl;
  for (int r = 0; r < world; ++r) {
    if (!peers[r]) return NVF_ERR_INVALID_ARG;
    p.peer[r] = (char*)peers[r];
  }
  int grid = (p.n4 + 255) / 256;
  if (grid > 64) grid = 64;                 // all CTAs resident: the last one to finish its copy publishes
  if (grid > l.n_sms) grid = l.n_sms;
  nvf_launch(fast::k_allreduce_adam, dim3(grid), dim3(256), (size_t)(0), l.st, p);
  l.post();
  return l.rc;
}

int nvf_ffma_microbench(int variant, int64_t iters, float* sink, double* flops_out, void* stream) {
  if (!sink || iters <= 0 || variant < 0 || variant > 1) return NVF_ERR_INVALID_ARG;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  const int grid = l.n_sms * 4;
  nvf_launch(k_ffma, dim3(grid), dim3(kThreads), (size_t)(0), l.st, variant, (long long)iters, sink);
  l.post();
  if (flops_out) *flops_out = 2.0 * 256.0 * (double)iters * (double)grid * kThreads;
  return l.rc;
}

}  // extern "C"


// ------------------------------------------------------------------ fused weight-loop step
namespace {

struct StepWs {
  size_t off_train, off_eff, off_geff, off_latent, off_glatent, off_scal, off_param, off_latws, off_tickets, off_losspart, total;
  int64_t eff_off[kEffTensors], eff_total;   // the effective tensors in NvfWeights field order
  static StepWs make(const NvfDesc& d, int64_t n) {
    StepWs L{};
    int64_t sz[kEffTensors];
    sz[offsetof(NvfWeights, igdn_beta) / sizeof(float*)] = d.c0;
    sz[offsetof(NvfWeights, igdn_gamma) / sizeof(float*)] = (int64_t)d.c0 * d.c0;
    for (int l = 0; l < NVF_NUM_CONV; ++l) {
      const ConvGeom c = conv_geom(d, l);
      sz[c.slot] = c.n();
      sz[c.slot + 1] = c.nb;
    }
    int64_t eo = 0;
    for (int i = 0; i < kEffTensors; ++i) { L.eff_off[i] = eo; eo += (sz[i] + 3) / 4 * 4; }
    L.eff_total = eo;
    size_t o = 0;
    auto take = [&](size_t bytes) { size_t r = o; o += align_up(bytes); return r; };
    L.off_train = take(TrainWs::make(d, n).total);
    L.off_eff = take(sizeof(float) * (size_t)eo);
    L.off_geff = take(sizeof(float) * (size_t)eo);
    L.off_latent = take(sizeof(float) * (size_t)n * d.ch * 8);
    L.off_glatent = take(sizeof(float) * (size_t)n * d.ch * 8);
    L.off_scal = take(sizeof(float) * 32);
    L.off_param = take(NVF_PARAM_WS_BYTES);
    L.off_latws = take(NVF_LATENT_WS_BYTES);
    L.off_tickets = take(64);
    L.off_losspart = take(sizeof(double) * NVF_LOSS_SUMS * (size_t)n * kLossChunks);
    L.total = o;
    return L;
  }
};

int train_step_impl(DevLauncher& l, const NvfStepArgs& a, void* workspace, size_t workspace_bytes) {
  const NvfDesc& d = a.desc;
  if (a.n <= 0 || a.n > (1 << 20) || a.q < 0 || a.q > 2 || !a.emb || !a.gt || !a.dist || !a.n_pts || !a.stats || !a.sums ||
      !workspace)
    return NVF_ERR_INVALID_ARG;
  if (!generic_supported(d)) return NVF_ERR_UNSUPPORTED;
  if (d.ch < 1 || d.ch > 4) return NVF_ERR_UNSUPPORTED;
  if (a.idx && a.n_rows < 1) return NVF_ERR_INVALID_ARG;
  const bool wg = (a.flags & NVF_BWD_WGRAD) != 0, demb = (a.flags & NVF_BWD_DLATENT) != 0;
  if (demb && !a.g_emb) return NVF_ERR_INVALID_ARG;
  const bool need_rng = (a.q == 1 && !a.noise_kernel) || (a.train_mode && !a.noise_latent && a.noise_scale != 0.f);
  if (need_rng && !a.rng_counter) return NVF_ERR_INVALID_ARG;
  const int n = a.n;
  const StepWs W = StepWs::make(d, n);
  if (workspace_bytes < W.total) return NVF_ERR_WORKSPACE;
  char* ws = (char*)workspace;
  char* tws = ws + W.off_train;
  const TrainWs T = TrainWs::make(d, n);
  float* eff = (float*)(ws + W.off_eff);
  float* geff = (float*)(ws + W.off_geff);
  float* latent = (float*)(ws + W.off_latent);
  float* g_latent = (float*)(ws + W.off_glatent);
  float* scal = (float*)(ws + W.off_scal);       // [0] latent_bits, [1..7] net_bits, [8] g latent_bits, [9..15] g net_bits
  unsigned int* tickets = (unsigned int*)(ws + W.off_tickets);
  const unsigned long long* ctr = (const unsigned long long*)a.rng_counter;

  NvfWeights w{};
  NvfWeightGrads gw{}, effw{};
  for (int i = 0; i < kEffTensors; ++i) {
    slots(w)[i] = slots(effw)[i] = eff + W.eff_off[i];
    slots(gw)[i] = geff + W.eff_off[i];
  }

  // ---- latent head on the auxiliary stream ...
  fast::LatentKParams lk{};
  lk.emb = a.emb; lk.noise = a.noise_latent;
  lk.kernel = a.latent.kernel; lk.kernel_init = a.latent.kernel_init; lk.b = a.latent.b; lk.b_init = a.latent.b_init;
  lk.beta = a.latent.gdn_beta; lk.gamma = a.latent.gdn_gamma; lk.sigma = a.latent.sigma; lk.mu = a.latent.mu;
  if (!lk.kernel || !lk.kernel_init || !lk.b || !lk.b_init || !lk.beta || !lk.gamma || !lk.sigma || !lk.mu)
    return NVF_ERR_INVALID_ARG;
  lk.beta_bound = a.latent_beta_bound; lk.gamma_bound = a.latent_gamma_bound; lk.pedestal = a.latent_pedestal;
  lk.noise_scale = a.noise_scale; lk.n = n; lk.train = a.train_mode ? 1 : 0;
  lk.ticket = (unsigned int*)(ws + W.off_latws);
  lk.partial = (double*)(ws + W.off_latws + 16);
  lk.idx = (const long long*)a.idx; lk.n_rows = a.n_rows;
  lk.seed = a.seed; lk.rng_ctr = (a.noise_latent || !a.train_mode) ? nullptr : ctr;
  lk.latent = latent; lk.bits_out = scal;
  l.side_begin();
  launch_latent(l, d.ch, lk, false);
  l.side_end();

  // ---- ... while the parameter kernel writes the effective tensors, their packed layouts and net_bits
  fast::ParamPrepParams pp{};
  int rc = fill_param_jobs(d, a.params, pp);
  if (rc != NVF_OK) return rc;
  const GenericPacked g = GenericPacked::make(d);
  float* packed = (float*)(tws + T.off_packed);
  for (int i = 0; i < NVF_NUM_CONV; ++i) {
    const int s = conv_geom(d, i).slot;
    fast::ParamJob& J = pp.job[i];
    J.w_out = slots(effw)[s]; J.b_out = slots(effw)[s + 1];
    J.pk_fwd = packed + g.fwd[i]; J.pk_dg = packed + g.dg[i];
  }
  pp.beta_out = effw.igdn_beta; pp.gamma_out = effw.igdn_gamma;
  pp.noise = a.noise_kernel; pp.q = a.q;
  pp.seed = a.seed; pp.rng_ctr = ctr;
  pp.partial = (float*)(ws + W.off_param); pp.net_bits = scal + 1;
  pp.beta_bound = a.igdn_beta_bound; pp.gamma_bound = a.igdn_gamma_bound; pp.pedestal = a.igdn_pedestal;
  pp.ticket = tickets;
  nvf_launch(fast::k_param_prep<false>, dim3(pp.total_chunks + 1), dim3(256), (size_t)(0), l.st, pp);
  l.post();
  l.join();

  // ---- decoder forward (probabilities of the three heads stay in the workspace)
  float* p2 = (float*)(tws + T.off_p2);
  float* p1 = (float*)(tws + T.off_p1);
  float* p0 = (float*)(tws + T.off_p0);
  l.set_queue(tws + T.off_queue);   // zero since the caller's one-time fill; every queue-fed kernel rewinds its words
  Api<DevLauncher>::forward_layers(l, d, w, (const float*)(tws + T.off_packed), latent, n, (float*)(tws + T.off_stash), p2, p1, p0,
                                   nullptr, nullptr, nullptr);

  // ---- loss, metrics, dL/dlogit, total loss and scalar cotangents: one launch
  const bool bwd = wg || demb;
  fast::LossStepParams lp{};
  lp.out = p2; lp.cls1 = p1; lp.cls0 = p0; lp.gt = a.gt; lp.dist = a.dist;
  lp.idx = (const long long*)a.idx; lp.n_rows = a.n_rows; lp.status = a.status;
  lp.gl2 = bwd ? (float*)(tws + T.off_gl2) : nullptr;
  lp.gl1 = bwd ? (float*)(tws + T.off_gl1) : nullptr;
  lp.gl0 = bwd ? (float*)(tws + T.off_gl0) : nullptr;
  lp.partial = (double*)(ws + W.off_losspart); lp.ticket = tickets + 2;
  lp.alpha_main = a.alpha_main; lp.alpha_aux = a.alpha_aux; lp.thh_metric = a.thh_metric; lp.n = n;
  lp.latent_bits = scal; lp.net_bits = scal + 1; lp.n_pts = a.n_pts;
  lp.n_total = a.n_total; lp.lmbda = a.lmbda; lp.w1 = a.w1; lp.w2 = a.w2; lp.w2_grad = a.w2_grad;
  lp.sums = a.sums; lp.stats = a.stats; lp.g_scal = scal + 8;
  nvf_launch(fast::k_loss_step, dim3(n * kLossChunks), dim3(256), (size_t)(0), l.st, lp);
  l.post();
  if (!bwd) return l.rc;

  // ---- decoder backward
  rc = Api<DevLauncher>::train_backward(l, &d, &w, latent, n, lp.gl2, lp.gl1, lp.gl0,
                                        (wg ? NVF_BWD_WGRAD : 0) | NVF_BWD_DLATENT | NVF_BWD_DLOGIT, wg ? &gw : nullptr,
                                        g_latent, tws, T.total);
  if (rc != NVF_OK) return rc;

  // ---- latent head backward on the auxiliary stream, parameter-side backward on the caller's
  lk.g_latent = g_latent; lk.g_bits = scal + 8; lk.g_emb = demb ? a.g_emb : nullptr;
  if (wg) {
    const NvfLatentGrads& G = a.g_latent;
    if (!G.kernel || !G.b || !G.gdn_beta || !G.gdn_gamma || !G.sigma || !G.mu) return NVF_ERR_INVALID_ARG;
    lk.gk = G.kernel; lk.gb = G.b; lk.gbeta = G.gdn_beta; lk.ggamma = G.gdn_gamma; lk.gsigma = G.sigma; lk.gmu = G.mu;
  }
  l.side_begin();
  launch_latent(l, d.ch, lk, true);
  if (need_rng) {
    nvf_launch(fast::k_rng_tick, dim3(1), dim3(1), (size_t)(0), l.st, (unsigned long long*)a.rng_counter);
    l.post();
  }
  l.side_end();
  if (wg) {
    const NvfParamGrads& O = a.g_params;
    for (int i = 0; i < NVF_NUM_CONV; ++i) {
      if (!O.kernel[i] || !O.b[i]) return NVF_ERR_INVALID_ARG;
      const int s = conv_geom(d, i).slot;
      fast::ParamJob& J = pp.job[i];
      J.g_w = slots(gw)[s]; J.g_b = slots(gw)[s + 1];
      J.w_out = O.kernel[i]; J.b_out = O.b[i];
      J.pk_fwd = nullptr; J.pk_dg = nullptr;
    }
    if (!O.igdn_beta || !O.igdn_gamma || !O.lik_sigma || !O.lik_mu) return NVF_ERR_INVALID_ARG;
    pp.g_beta = gw.igdn_beta; pp.g_gamma = gw.igdn_gamma;
    pp.beta_out = O.igdn_beta; pp.gamma_out = O.igdn_gamma;
    pp.g_bits = scal + 9;
    pp.g_sigma = O.lik_sigma; pp.g_mu = O.lik_mu;
    pp.ticket = tickets + 1;
    nvf_launch(fast::k_param_prep<true>, dim3(pp.total_chunks + 1), dim3(256), (size_t)(0), l.st, pp);
    l.post();
  }
  l.join();
  return l.rc;
}

__global__ void __launch_bounds__(256) k_rng_uniform(unsigned long long seed, unsigned long long step, unsigned int stream,
                                                     long long first, long long n, float* out) {
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < n; i += (long long)gridDim.x * 256)
    out[i] = rng::uniform(seed, step, stream, (uint64_t)(first + i));
}

}  // namespace

extern "C" {

int nvf_train_step_workspace_bytes(const NvfDesc* desc, int64_t n_blocks, size_t* bytes_out) {
  if (!desc || !bytes_out || n_blocks < 0) return NVF_ERR_INVALID_ARG;
  if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
  *bytes_out = StepWs::make(*desc, n_blocks).total;
  return NVF_OK;
}

int nvf_train_step(const NvfStepArgs* args, void* workspace, size_t workspace_bytes, void* stream) {
  if (!args) return NVF_ERR_INVALID_ARG;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  return train_step_impl(l, *args, workspace, workspace_bytes);
}

int nvf_rng_uniform(uint64_t seed, uint64_t step, int stream_id, int64_t first, int64_t n, float* out, void* stream) {
  if (!out || n < 0 || first < 0 || stream_id < 0 || stream_id > 255) return NVF_ERR_INVALID_ARG;
  if (n == 0) return NVF_OK;
  DevLauncher l{(cudaStream_t)stream};
  if (l.init() != NVF_OK) return l.rc;
  int grid = (int)((n + 255) / 256 < 1184 ? (n + 255) / 256 : 1184);
  nvf_launch(k_rng_uniform, dim3(grid), dim3(256), (size_t)(0), l.st, (unsigned long long)seed, (unsigned long long)step,
             (unsigned int)stream_id, (long long)first, (long long)n, out);
  l.post();
  return l.rc;
}

}  // extern "C"
