// C ABI (include/nvf_prep_b200.h, include/nvf_metrics_b200.h) + launchers of the preparation-side and distortion
// metric kernels for sm_100a.
#include <cuda_runtime.h>
#include <atomic>

#include <cub/device/device_radix_sort.cuh>

#include "../../include/nvf_b200.h"
#include "../../include/nvf_prep_b200.h"
#include "../../include/nvf_metrics_b200.h"
#include "nvf_grids.cuh"
#include "nvf_metrics.cuh"

namespace nvf {
extern std::atomic<long long> g_launches;   // nvf_capi.cu (nvf_launch_count)
void note_cuda_error(int e);                // nvf_capi.cu (nvf_last_cuda_error)
}

using namespace nvf;
using namespace nvf::metrics;

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

// ----------------------------------------------------------------------------- distortion metrics
constexpr int kMortonBits = 63;   // three interleaved 21-bit fields

size_t round256(size_t b) { return (b + 255) / 256 * 256; }

// Upper bound of CUB's onesweep radix-sort scratch for n pairs with the caller owning both key / value buffers
// (DoubleBuffer): per-portion digit bins, one lookback row of 256 digits per tile of at least 256 items, counters.
// Computed without a device so that the workspace queries need none; the launch checks CUB's own figure against it.
size_t cub_sort_bound(int64_t n) { return 256 * 1024 + round256((size_t)n * 8 + 2048); }

uint32_t leaf_slots(int64_t n) {
  const uint64_t leaves = (uint64_t)((n + kNnLeaf - 1) / kNnLeaf);
  uint32_t P = 1;
  while (P < leaves) P <<= 1;
  return P;
}

// Workspace of one tree over n target points.  The Morton-ordered points reuse the key buffers once the sort is done.
struct TreeWs {
  size_t keys0, keys1, vals0, vals1, boxes, cub, cub_bytes;
  uint32_t P;
  static TreeWs make(int64_t n, size_t& off) {
    TreeWs w{};
    w.P = leaf_slots(n);
    auto take = [&](size_t bytes) { size_t o = off; off += round256(bytes); return o; };
    w.keys0 = take((size_t)n * 16);        // keys0 and keys1 are adjacent: 16 bytes per point for `sorted`
    w.keys1 = w.keys0 + (size_t)n * 8;
    w.vals0 = take((size_t)n * 4);
    w.vals1 = take((size_t)n * 4);
    w.boxes = take((size_t)w.P * 2 * sizeof(Box));
    w.cub_bytes = cub_sort_bound(n);
    w.cub = take(w.cub_bytes);
    return w;
  }
};

// Per-query results and first-stage partials of the distortion sums.
struct DistWs {
  TreeWs tree;
  size_t d2, plane, psum, pmax, pplane, total;
  int64_t n_part;
  static DistWs make(int64_t n_source, int64_t n_rec) {
    DistWs w{};
    const int64_t n = n_source > n_rec ? n_source : n_rec;
    size_t off = 0;
    w.tree = TreeWs::make(n, off);
    auto take = [&](size_t bytes) { size_t o = off; off += round256(bytes); return o; };
    w.n_part = (n + kRedChunk - 1) / kRedChunk;
    w.d2 = take((size_t)n * 8);
    w.plane = take((size_t)n * 8);
    w.psum = take((size_t)w.n_part * 8);
    w.pmax = take((size_t)w.n_part * 8);
    w.pplane = take((size_t)w.n_part * 8);
    w.total = off;
    return w;
  }
};

bool valid_count(int64_t n, int64_t lo) { return n >= lo && n <= 0x7fffffffll; }

int device_sms(Chk& chk, int& sms) {
  int dev = 0, major = 0;
  if (!chk(cudaGetDevice(&dev)) || !chk(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev)) ||
      !chk(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev)))
    return chk.rc;
  return major == 10 ? NVF_OK : NVF_ERR_NO_DEVICE;
}

unsigned stride_grid(int64_t n, int sms) {
  const int64_t g = (n + 255) / 256, cap = (int64_t)sms * 8;
  return (unsigned)(g < 1 ? 1 : (g < cap ? g : cap));
}

// Sort + boxes of the target cloud into W; returns the Morton-ordered points.
int build_tree(Chk& chk, const TreeWs& W, char* ws, const int32_t* target, int64_t n, int32_t* status, int sms,
               cudaStream_t st, const int4*& sorted) {
  unsigned long long* keys0 = (unsigned long long*)(ws + W.keys0);
  unsigned long long* keys1 = (unsigned long long*)(ws + W.keys1);
  int32_t* vals0 = (int32_t*)(ws + W.vals0);
  int32_t* vals1 = (int32_t*)(ws + W.vals1);
  k_morton_keys<<<stride_grid(n, sms), 256, 0, st>>>(target, n, keys0, vals0, status);
  chk.launched();
  cub::DoubleBuffer<unsigned long long> kb(keys0, keys1);
  cub::DoubleBuffer<int32_t> vb(vals0, vals1);
  size_t need = 0;
  if (!chk(cub::DeviceRadixSort::SortPairs(nullptr, need, kb, vb, (int)n, 0, kMortonBits, st))) return chk.rc;
  if (need > W.cub_bytes) return NVF_ERR_WORKSPACE;
  if (!chk(cub::DeviceRadixSort::SortPairs(ws + W.cub, need, kb, vb, (int)n, 0, kMortonBits, st))) return chk.rc;
  // (CUB's own launches are not counted by nvf_launch_count)
  int4* out = (int4*)(ws + W.keys0);
  k_gather_sorted<<<stride_grid(n, sms), 256, 0, st>>>(target, n, vb.Current(), out);
  chk.launched();
  Box* boxes = (Box*)(ws + W.boxes);
  k_leaf_boxes<<<stride_grid(W.P, sms), 256, 0, st>>>(out, n, W.P, boxes);
  chk.launched();
  for (uint32_t first = W.P / 2; first >= 1; first /= 2) {
    k_parent_boxes<<<stride_grid(first, sms), 256, 0, st>>>(first, boxes);
    chk.launched();
  }
  sorted = out;
  return chk.rc;
}

int run_query(Chk& chk, int mode, NnParams p, cudaStream_t st) {
  if (p.n_query == 0) return chk.rc;
  const unsigned grid = (unsigned)((p.n_query + 255) / 256);
  if (mode == kQueryNormals)
    k_nn_query<kQueryNormals><<<grid, 256, 0, st>>>(p);
  else if (mode == kTargetNormals)
    k_nn_query<kTargetNormals><<<grid, 256, 0, st>>>(p);
  else
    k_nn_query<kNoNormals><<<grid, 256, 0, st>>>(p);
  chk.launched();
  return chk.rc;
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


int nvf_nn_workspace_bytes(int64_t n_target, size_t* bytes_out) {
  if (!bytes_out || !valid_count(n_target, 1)) return NVF_ERR_INVALID_ARG;
  size_t off = 0;
  TreeWs::make(n_target, off);
  *bytes_out = off;
  return NVF_OK;
}

int nvf_nearest_points(const int32_t* target, int64_t n_target, const int32_t* query, int64_t n_query,
                       int32_t* index_out, int64_t* d2_out, int32_t* ties_out, int32_t* status_out, void* workspace,
                       size_t workspace_bytes, void* stream) {
  if (!valid_count(n_target, 1) || !valid_count(n_query, 0) || !target || (n_query > 0 && !query) || !status_out ||
      !workspace)
    return NVF_ERR_INVALID_ARG;
  size_t total = 0;
  const TreeWs W = TreeWs::make(n_target, total);
  if (workspace_bytes < total) return NVF_ERR_WORKSPACE;
  Chk chk;
  int sms = 0;
  if (int rc = device_sms(chk, sms)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  if (!chk(cudaMemsetAsync(status_out, 0, sizeof(int32_t), st))) return chk.rc;
  const int4* sorted = nullptr;
  if (int rc = build_tree(chk, W, ws, target, n_target, status_out, sms, st, sorted)) return rc;
  NnParams p{};
  p.sorted = sorted;
  p.boxes = (const Box*)(ws + W.boxes);
  p.n_target = n_target;
  p.P = W.P;
  p.query = query;
  p.n_query = n_query;
  p.index_out = index_out;
  p.d2_out = d2_out;
  p.ties_out = ties_out;
  p.status = status_out;
  return run_query(chk, kNoNormals, p, st);
}

int nvf_distortion_workspace_bytes(int64_t n_source, int64_t n_rec, size_t* bytes_out) {
  if (!bytes_out || !valid_count(n_source, 1) || !valid_count(n_rec, 1)) return NVF_ERR_INVALID_ARG;
  *bytes_out = DistWs::make(n_source, n_rec).total;
  return NVF_OK;
}

int nvf_pc_distortion(const int32_t* source, int64_t n_source, const double* source_normals, const int32_t* rec,
                      int64_t n_rec, NvfDistortion* out, int32_t* status_out, void* workspace,
                      size_t workspace_bytes, void* stream) {
  if (!valid_count(n_source, 1) || !valid_count(n_rec, 1) || !source || !rec || !out || !status_out || !workspace)
    return NVF_ERR_INVALID_ARG;
  const DistWs W = DistWs::make(n_source, n_rec);
  if (workspace_bytes < W.total) return NVF_ERR_WORKSPACE;
  Chk chk;
  int sms = 0;
  if (int rc = device_sms(chk, sms)) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  char* ws = (char*)workspace;
  if (!chk(cudaMemsetAsync(status_out, 0, sizeof(int32_t), st))) return chk.rc;
  int64_t* d2 = (int64_t*)(ws + W.d2);
  double* plane = (double*)(ws + W.plane);
  // direction 0: every source point queries the reconstruction; direction 1 the other way round.  Both reuse
  // the same tree and per-query buffers in stream order.
  for (int dir = 0; dir < 2; ++dir) {
    const int32_t* target = dir == 0 ? rec : source;
    const int32_t* query = dir == 0 ? source : rec;
    const int64_t n_t = dir == 0 ? n_rec : n_source, n_q = dir == 0 ? n_source : n_rec;
    const int4* sorted = nullptr;
    TreeWs T = W.tree;                   // sized for the larger cloud; only the leaf slots follow this target
    T.P = leaf_slots(n_t);
    if (int rc = build_tree(chk, T, ws, target, n_t, status_out, sms, st, sorted)) return rc;
    NnParams p{};
    p.sorted = sorted;
    p.boxes = (const Box*)(ws + T.boxes);
    p.n_target = n_t;
    p.P = T.P;
    p.query = query;
    p.n_query = n_q;
    p.normals = source_normals;
    p.d2_out = d2;
    p.plane_out = plane;
    p.status = status_out;
    if (int rc = run_query(chk, source_normals ? (dir == 0 ? kQueryNormals : kTargetNormals) : kNoNormals, p, st))
      return rc;
    const int64_t n_part = (n_q + kRedChunk - 1) / kRedChunk;
    k_reduce_partials<<<(unsigned)n_part, kRedThreads, 0, st>>>(d2, plane, n_q, (unsigned long long*)(ws + W.psum),
                                                                (unsigned long long*)(ws + W.pmax),
                                                                (double*)(ws + W.pplane));
    chk.launched();
    k_reduce_final<<<1, kFinalThreads, 0, st>>>((const unsigned long long*)(ws + W.psum),
                                                (const unsigned long long*)(ws + W.pmax), (const double*)(ws + W.pplane),
                                                n_part, n_q, dir, out, status_out);
    chk.launched();
    if (chk.rc) return chk.rc;
  }
  return chk.rc;
}

}  // extern "C"
