// TEST-ONLY CPU emulator of the NVF kernels.
//
// Compiles the SAME generic kernel bodies (nvf_layers.h, nvf_emit.h) and host
// orchestration (nvf_api_impl.h) as the CUDA library with g++, executing every
// CTA's threads sequentially phase by phase (a phase boundary is a
// __syncthreads()).  The fused decode head and the shared-memory tiled kernels
// are CUDA-only, so here decode and training run layer-wise for every
// configuration.  It lets the `-m "not gpu"` tests check index arithmetic,
// workspace layouts and sequencing against the oracle before GPU time is spent.
// It is NOT part of the product: nvfpcc_b200 never loads it and there is no CPU
// fallback in the package.
#include <stdlib.h>
#include <string.h>
#include <vector>

#include "../../nvfpcc_b200/csrc/nvf_api_impl.h"

using namespace nvf;

namespace {

template <class TS>
struct EmuEnv {
  std::vector<TS> ts;
  EmuEnv() : ts(kThreads) {}
  template <class F>
  void phase(F&& f) {
    for (int t = 0; t < kThreads; ++t) f(t, ts[t]);
  }
};

struct EmuLauncher {
  int n_sms = 3;  // few persistent CTAs so that the round-robin block loop is exercised
  int sms() const { return n_sms; }
  int error() const { return NVF_OK; }

  void pack(const PackParams& p) {
    const int g = 4 * kThreads;
    for (int t = 0; t < g; ++t) pack_thread(p, t, g);
  }
  void scan(const EmitParams& p) {
    std::vector<int64_t> sm(2 * kThreads);
    EmuEnv<int> env;
    ScanBlock<EmuEnv<int>>::run(env, p, sm.data());
  }
  void emit(const EmitParams& p, int grid) {
    std::vector<int> sm(2 * kThreads);
    for (int b = 0; b < grid; ++b) {
      EmuEnv<int> env;
      EmitBlock<EmuEnv<int>>::run(env, p, sm.data(), b);
    }
  }
  // the shared-memory tiled CUDA kernels have no emulated counterpart: the generic kernels run instead
  bool fast_layer(const LayerParams&) { return false; }
  bool fast_wgrad(const WgradParams&, const ChanSumParams&) { return false; }
  bool fast_igdn_param(const IgdnParams&) { return false; }
  bool fast_stem_fwd(const NvfDesc&, const NvfWeights&, const float*, const float*, const float*, const float*, int,
                     float*, float*, float*, float*, float*) { return false; }
  bool fast_stem_bwd(const NvfDesc&, const NvfWeights&, const float*, int, const float*, const float*, const float*,
                     float*, const NvfWeightGrads*, float*) { return false; }
  // the warp-specialised fused decode head is CUDA-only: the emulator decodes with the layer kernels
  bool has_head(const NvfDesc&) { return false; }
  void zero_ints(int32_t*, int64_t) {}
  void pad_conv1(const float*, float*, int64_t) {}
  bool up_poly(const LayerParams&, float*) { return false; }
  void head(const NvfDesc&, const HeadArgs&, int) {}
  void side_begin() {}
  void side_end() {}
  void join() {}
  void set_partial(float*, size_t) {}
  void set_queue(void*) {}
  void zero_queue(void*, size_t) {}
  void flush_reduce() {}
  template <int COT>
  void layer(const LayerParams& p) {
    const int grid = 7;
    for (int b = 0; b < grid; ++b)
      for (int t = 0; t < kThreads; ++t) LayerKernel<COT>::thread(p, b, t, grid);
  }
  template <int COT, int K>
  void wgrad(const WgradParams& p, int grid) {
    std::vector<float> sm((size_t)kThreads * COT * K);
    for (int b = 0; b < grid; ++b) {
      EmuEnv<int> env;
      WgradBlock<COT, K>::run(env, p, sm.data(), b);
    }
  }
  void chansum(const ChanSumParams& p, int grid) {
    std::vector<float> sm(kThreads);
    for (int b = 0; b < grid; ++b) {
      EmuEnv<int> env;
      ChanSumBlock::run(env, p, sm.data(), b);
    }
  }
  template <class K>
  void generic(const typename K::Params& p, int grid) {
    if (grid < 1) grid = 1;
    for (int b = 0; b < grid; ++b)
      for (int t = 0; t < kThreads; ++t) K::thread(p, b, t, grid);
  }
  void mask(const MaskParams& p, int grid) {
    std::vector<int> sm(kThreads);
    for (int b = 0; b < grid; ++b) {
      EmuEnv<int> env;
      MaskBlock::run(env, p, sm.data(), b);
    }
  }
  void loss(const LossParams& p, int grid) {
    std::vector<double> sm((size_t)kThreads * NVF_LOSS_SUMS);
    for (int b = 0; b < grid; ++b) {
      EmuEnv<int> env;
      LossBlock::run(env, p, sm.data(), b);
    }
  }
};

}  // namespace

extern "C" {

int nvf_abi_version(void) { return NVF_ABI_VERSION; }
const char* nvf_strerror(int code) { return code == NVF_OK ? "ok" : "error (emulator)"; }
int nvf_last_cuda_error(void) { return 0; }
long long nvf_launch_count(void) { return 0; }
int nvf_has_fused_decode(const NvfDesc*) { return 0; }

int nvf_workspace_bytes(const NvfDesc* desc, int64_t n_blocks, int mode, size_t* bytes_out) {
  if (!desc || !bytes_out || n_blocks < 0) return NVF_ERR_INVALID_ARG;
  if (!generic_supported(*desc)) return NVF_ERR_UNSUPPORTED;
  if (mode == NVF_MODE_DECODE) *bytes_out = DecodeWs::make(*desc, n_blocks, false).total;
  else if (mode == NVF_MODE_TRAIN) *bytes_out = TrainWs::make(*desc, n_blocks).total;
  else return NVF_ERR_INVALID_ARG;
  return NVF_OK;
}

int nvf_decode(const NvfDesc* desc, const NvfWeights* w, const float* latent, const int32_t* origins,
               int64_t n_blocks, float thh, float* prob_out, uint32_t* mask_out, int32_t* counts_out,
               int32_t* coords_out, int64_t cap, int64_t* total_out, void* workspace, size_t workspace_bytes,
               void*) {
  EmuLauncher l;
  return Api<EmuLauncher>::decode(l, desc, w, latent, origins, n_blocks, thh, prob_out, mask_out, counts_out,
                                  coords_out, cap, total_out, workspace, workspace_bytes);
}
int nvf_emit_points(const uint32_t* mask, const int32_t* counts, const int32_t* origins, int64_t n_blocks,
                    int32_t* coords_out, int64_t cap, int64_t* total_out, void* workspace, size_t workspace_bytes,
                    void*) {
  EmuLauncher l;
  return Api<EmuLauncher>::emit_points(l, mask, counts, origins, n_blocks, coords_out, cap, total_out, workspace,
                              workspace_bytes);
}

int nvf_train_forward(const NvfDesc* desc, const NvfWeights* w, const float* latent, int64_t n_blocks, float* out,
                      float* cls1, float* cls0, void* workspace, size_t workspace_bytes, void*) {
  EmuLauncher l;
  return Api<EmuLauncher>::train_forward(l, desc, w, latent, n_blocks, out, cls1, cls0, workspace, workspace_bytes);
}
int nvf_loss_seeds(const float* out, const float* cls1, const float* cls0, const float* gt, const float* dist,
                   int64_t n_blocks, float alpha_main, float alpha_aux, float thh_metric, double* sums_out,
                   float* g_out, float* g_cls1, float* g_cls0, void* workspace, size_t workspace_bytes, void*) {
  EmuLauncher l;
  return Api<EmuLauncher>::loss_seeds(l, out, cls1, cls0, gt, dist, n_blocks, alpha_main, alpha_aux, thh_metric,
                                      sums_out, g_out, g_cls1, g_cls0, workspace, workspace_bytes);
}
int nvf_train_backward(const NvfDesc* desc, const NvfWeights* w, const float* latent, int64_t n_blocks,
                       const float* g_out, const float* g_cls1, const float* g_cls0, int flags,
                       const NvfWeightGrads* gw, float* g_latent, void* workspace, size_t workspace_bytes, void*) {
  EmuLauncher l;
  return Api<EmuLauncher>::train_backward(l, desc, w, latent, n_blocks, g_out, g_cls1, g_cls0, flags, gw, g_latent,
                                          workspace, workspace_bytes);
}
int nvf_ffma_microbench(int, int64_t, float*, double*, void*) { return NVF_ERR_NO_DEVICE; }
// the fused step and its noise generator exist only in the CUDA library
int nvf_train_step_workspace_bytes(const NvfDesc*, int64_t, size_t*) { return NVF_ERR_UNSUPPORTED; }
int nvf_train_step(const NvfStepArgs*, void*, size_t, void*) { return NVF_ERR_UNSUPPORTED; }
int nvf_rng_uniform(uint64_t, uint64_t, int, int64_t, int64_t, float*, void*) { return NVF_ERR_UNSUPPORTED; }
size_t nvf_symm_bytes(int64_t) { return 0; }
int nvf_symm_alloc(size_t, void**, void*) { return NVF_ERR_UNSUPPORTED; }
int nvf_symm_open(const void*, void**) { return NVF_ERR_UNSUPPORTED; }
int nvf_symm_close(void*) { return NVF_ERR_UNSUPPORTED; }
int nvf_symm_free(void*) { return NVF_ERR_UNSUPPORTED; }
int nvf_adam_allreduce_step(float*, const float*, float*, float*, int64_t, float*, const float*, float, float, float,
                            void* const*, int, int, void*, void*) { return NVF_ERR_UNSUPPORTED; }


// parameter-side fused kernels exist only in the CUDA library (the torch ops they replace are the CPU reference)
int nvf_param_prep(const NvfDesc*, const NvfParamSet*, int, const float*, float, float, float, const NvfWeightGrads*,
                   float*, void*, size_t, void*) { return NVF_ERR_UNSUPPORTED; }
int nvf_param_prep_backward(const NvfDesc*, const NvfParamSet*, float, float, const NvfWeights*, const float*,
                            const NvfParamGrads*, void*, size_t, void*) { return NVF_ERR_UNSUPPORTED; }
// likewise the latent head, total loss and Adam kernels
int nvf_latent_forward(int, const NvfLatentParams*, const float*, const float*, float, int, int64_t, float, float, float,
                       float*, float*, void*, size_t, void*) { return NVF_ERR_UNSUPPORTED; }
int nvf_latent_backward(int, const NvfLatentParams*, const float*, const float*, float, int, int64_t, float, float,
                        float, const float*, const float*, const NvfLatentGrads*, float*, void*, size_t, void*) {
  return NVF_ERR_UNSUPPORTED;
}
int nvf_rd_total(const double*, const float*, const float*, const float*, float, float, float, float, float*, float*,
                 void*) { return NVF_ERR_UNSUPPORTED; }
int nvf_rd_total_backward(const float*, const float*, float, float, float, float, float*, float*, float*, void*) {
  return NVF_ERR_UNSUPPORTED;
}
int nvf_adam_step(float*, const float*, float*, float*, int64_t, float*, const float*, float, float, float, void*) {
  return NVF_ERR_UNSUPPORTED;
}
}  // extern "C"
