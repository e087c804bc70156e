// C ABI (include/nvf_prep_b200.h) + launchers of the preparation-side kernels for sm_100a.
#include <cuda_runtime.h>
#include <atomic>

#include "../../include/nvf_b200.h"
#include "../../include/nvf_prep_b200.h"
#include "nvf_grids.cuh"

namespace nvf {
extern std::atomic<long long> g_launches;   // nvf_capi.cu (nvf_launch_count)
void note_cuda_error(int e);                // nvf_capi.cu (nvf_last_cuda_error)
}

using namespace nvf;

namespace {

struct GridWs {
  size_t keys, vals, counter, masks, total;
  uint32_t cap;
  static GridWs make(int64_t max_cells) {
    GridWs w{};
    uint64_t cap = 64;
    while (cap < 2ull * (uint64_t)max_cells) cap <<= 1;
    w.cap = (uint32_t)cap;
    size_t off = 0;
    auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) / 256 * 256; return o; };
    w.keys = take(cap * 8);
    w.vals = take(cap * 4);
    w.counter = take(256);
    w.masks = take((size_t)max_cells * 4096);
    w.total = off;
    return w;
  }
};

struct Chk {
  int rc = NVF_OK;
  bool operator()(cudaError_t e) {
    if (e != cudaSuccess) {
      note_cuda_error((int)e);
      if (rc == NVF_OK) rc = (e == cudaErrorNoDevice || e == cudaErrorInsufficientDriver) ? NVF_ERR_NO_DEVICE : NVF_ERR_CUDA;
      return false;
    }
    return true;
  }
  void launched() {
    (*this)(cudaGetLastError());
    g_launches.fetch_add(1, std::memory_order_relaxed);
  }
};

// rows idx[b] of gt / dist (32768 floats each) and of emb -> static batch buffers; grid (n, 16).
// An index outside [0, n_rows) is clamped to row 0 and reported through the sticky status word.
__global__ void __launch_bounds__(256) k_gather_batch(const float* __restrict__ emb_all, const float4* __restrict__ gt_all,
                                                      const float4* __restrict__ dist_all, const int64_t* __restrict__ idx,
                                                      int64_t n_rows, int emb_floats, float* __restrict__ emb_out,
                                                      float4* __restrict__ gt_out, float4* __restrict__ dist_out,
                                                      int32_t* __restrict__ status) {
  const int b = blockIdx.x, part = blockIdx.y;
  int64_t row = idx[b];
  if (row < 0 || row >= n_rows) {
    if (status && part == 0 && threadIdx.x == 0) atomicOr(status, 1);
    row = 0;
  }
  const size_t src = (size_t)row * 8192, dst = (size_t)b * 8192;
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int i = part * 512 + u * 256 + threadIdx.x;
    gt_out[dst + i] = __ldg(gt_all + src + i);
    dist_out[dst + i] = __ldg(dist_all + src + i);
  }
  if (part == 0)
    for (int i = threadIdx.x; i < emb_floats; i += 256)
      emb_out[(size_t)b * emb_floats + i] = emb_all[(size_t)row * emb_floats + i];
}

}  // namespace

extern "C" {

int nvf_gather_batch(const float* emb_all, const float* gt_all, const float* dist_all, const int64_t* idx, int64_t n,
                     int64_t n_rows, int32_t emb_floats, float* emb_out, float* gt_out, float* dist_out,
                     int32_t* status, void* stream) {
  if (n < 0 || n > 0x7fffffff || n_rows < 1 || emb_floats < 1 || !emb_all || !gt_all || !dist_all || !idx || !emb_out ||
      !gt_out || !dist_out)
    return NVF_ERR_INVALID_ARG;
  if (n == 0) return NVF_OK;
  Chk chk;
  k_gather_batch<<<dim3((unsigned)n, 16), 256, 0, (cudaStream_t)stream>>>(
      emb_all, (const float4*)gt_all, (const float4*)dist_all, idx, n_rows, emb_floats, emb_out, (float4*)gt_out,
      (float4*)dist_out, status);
  chk.launched();
  return chk.rc;
}

int nvf_grids_workspace_bytes(int64_t max_cells, size_t* bytes_out) {
  if (!bytes_out || max_cells < 1 || max_cells > (1ll << 24)) return NVF_ERR_INVALID_ARG;
  *bytes_out = GridWs::make(max_cells).total;
  return NVF_OK;
}

int nvf_build_grids(const int32_t* points, int64_t n_points, const int32_t* origins, int64_t n_blocks,
                    int64_t max_cells, int32_t max_radius, uint8_t* gt_out, double* dist64_out, float* dist32_out,
                    uint16_t* d2_out, int32_t* status_out, void* workspace, size_t workspace_bytes, void* stream) {
  if (n_points < 0 || n_blocks < 0 || max_cells < 1 || max_cells > (1ll << 24) || max_radius < 0 || !status_out ||
      !workspace || (n_points > 0 && !points) || (n_blocks > 0 && !origins) || n_blocks > 0x7fffffffll)
    return NVF_ERR_INVALID_ARG;
  const GridWs W = GridWs::make(max_cells);
  if (workspace_bytes < W.total) return NVF_ERR_WORKSPACE;
  cudaStream_t st = (cudaStream_t)stream;
  Chk chk;
  int dev = 0, major = 0, sms = 0;
  if (!chk(cudaGetDevice(&dev)) || !chk(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev)) ||
      !chk(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)))
    return chk.rc;
  if (major != 10) return NVF_ERR_NO_DEVICE;
  char* ws = (char*)workspace;
  grids::CellTable T;
  T.keys = (unsigned long long*)(ws + W.keys);
  T.vals = (int32_t*)(ws + W.vals);
  T.counter = (int32_t*)(ws + W.counter);
  T.masks = (uint32_t*)(ws + W.masks);
  T.status = status_out;
  T.cap_mask = W.cap - 1;
  T.max_cells = (int32_t)max_cells;
  // keys = empty, vals = -1, counter = 0, masks = 0, status = 0
  if (!chk(cudaMemsetAsync(ws + W.keys, 0xFF, W.vals + (size_t)W.cap * 4 - W.keys, st)) ||
      !chk(cudaMemsetAsync(ws + W.counter, 0, W.total - W.counter, st)) ||
      !chk(cudaMemsetAsync(status_out, 0, sizeof(int32_t), st)))
    return chk.rc;
  if (n_points > 0) {
    const int grid = (int)((n_points + 255) / 256 < (int64_t)sms * 8 ? (n_points + 255) / 256 : (int64_t)sms * 8);
    grids::k_cells_insert<<<grid, 256, 0, st>>>(points, n_points, T);
    chk.launched();
    grids::k_points_scatter<<<grid, 256, 0, st>>>(points, n_points, T);
    chk.launched();
  }
  if (n_blocks > 0) {
    static_assert(sizeof(grids::EdtSmem) <= 113 * 1024, "two CTAs per SM");
    if (!chk(cudaFuncSetAttribute(grids::k_edt_blocks, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                  (int)sizeof(grids::EdtSmem))))
      return chk.rc;
    grids::EdtParams p;
    p.origins = origins;
    p.gt = gt_out;
    p.dist64 = dist64_out;
    p.dist32 = dist32_out;
    p.d2 = d2_out;
    p.max_radius = max_radius;
    p.T = T;
    grids::k_edt_blocks<<<(unsigned)n_blocks, kThreads, sizeof(grids::EdtSmem), st>>>(p);
    chk.launched();
  }
  return chk.rc;
}

}  // extern "C"
