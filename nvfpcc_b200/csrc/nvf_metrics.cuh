// Exact nearest neighbours of integer lattice clouds and the D1 / D2 distortion sums built on them
// (include/nvf_metrics_b200.h).
//
//   1. k_morton_keys + CUB radix sort: the target points are ordered by the Morton code of their coordinates
//      (the 21-bit biased fields of grids::cell_key, interleaved), index as payload.  The sort is stable, so
//      duplicate points keep ascending index order.
//   2. k_leaf_boxes / k_parent_boxes: an implicit binary tree over the sorted points.  Leaf l holds sorted points
//      [l * kNnLeaf, (l + 1) * kNnLeaf); the leaf count is padded to a power of two P and node i (heap order, root 1)
//      has children 2i and 2i + 1.  Every node stores the integer bounding box of its points.
//   3. k_nn_query: one thread per query walks the tree depth first, nearer child first, and skips a node only when
//      the squared distance to its box is GREATER than the best squared distance found so far: every target point at
//      exactly the nearest distance is visited, so the tie count, the lowest tied index and the tie-averaged plane
//      error are exact.  There is no search radius: a query thousands of voxels from the cloud costs a root-to-leaf
//      walk, not a sweep over empty space.
//   4. k_reduce_partials + k_reduce_final: fixed-order two-stage sums of the per-query results (int64 for D1,
//      float64 for D2) into NvfDistortion.  No float atomics: two runs are bit-identical.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/nvf_metrics_b200.h"
#include "nvf_grids.cuh"

namespace nvf {
namespace metrics {

constexpr int kNnLeaf = 8;              // sorted points per tree leaf
constexpr int kNnStack = 32;            // > tree depth: log2(2^31 / kNnLeaf) + 1 levels
constexpr int kRedThreads = 256;
constexpr int kRedItems = 16;           // per thread: a first-stage block sums kRedThreads * kRedItems queries
constexpr int kRedChunk = kRedThreads * kRedItems;
constexpr int kFinalThreads = 1024;

struct Box {
  int4 lo;   // lo.w = 1 when the node holds at least one point
  int4 hi;
};

// 21 low bits of v spread to every third bit.
__device__ __forceinline__ unsigned long long spread3(unsigned long long v) {
  v &= 0x1fffffull;
  v = (v | v << 32) & 0x1f00000000ffffull;
  v = (v | v << 16) & 0x1f0000ff0000ffull;
  v = (v | v << 8) & 0x100f00f00f00f00full;
  v = (v | v << 4) & 0x10c30c30c30c30c3ull;
  v = (v | v << 2) & 0x1249249249249249ull;
  return v;
}

// true when (a0, a1, a2) lies in the range of the cell key; the key's biased fields give the Morton code
__device__ __forceinline__ bool morton_key(int a0, int a1, int a2, unsigned long long& code) {
  unsigned long long key;
  const bool ok = grids::cell_key(a0, a1, a2, key);
  if (!ok) {
    const int lo = -grids::COFF, hi = grids::COFF - 1;
    grids::cell_key(min(max(a0, lo), hi), min(max(a1, lo), hi), min(max(a2, lo), hi), key);
  }
  code = (spread3(key >> 42) << 2) | (spread3(key >> 21) << 1) | spread3(key);
  return ok;
}

__global__ void __launch_bounds__(256) k_morton_keys(const int32_t* __restrict__ pts, int64_t n,
                                                     unsigned long long* __restrict__ keys,
                                                     int32_t* __restrict__ vals, int32_t* __restrict__ status) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long code;
    if (!morton_key(pts[3 * i], pts[3 * i + 1], pts[3 * i + 2], code)) atomicOr(status, NVF_METRIC_STATUS_RANGE);
    keys[i] = code;
    vals[i] = (int32_t)i;
  }
}

// sorted[i] = {x, y, z, original index} of the i-th point in Morton order
__global__ void __launch_bounds__(256) k_gather_sorted(const int32_t* __restrict__ pts, int64_t n,
                                                       const int32_t* __restrict__ order, int4* __restrict__ sorted) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int32_t j = order[i];
    sorted[i] = make_int4(pts[3 * (int64_t)j], pts[3 * (int64_t)j + 1], pts[3 * (int64_t)j + 2], j);
  }
}

// boxes[P + l] for every leaf slot l < P (slots at or past the last point are empty)
__global__ void __launch_bounds__(256) k_leaf_boxes(const int4* __restrict__ sorted, int64_t n, uint32_t P,
                                                    Box* __restrict__ boxes) {
  for (int64_t l = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; l < P; l += (int64_t)gridDim.x * blockDim.x) {
    Box b;
    b.lo = make_int4(INT32_MAX, INT32_MAX, INT32_MAX, 0);
    b.hi = make_int4(INT32_MIN, INT32_MIN, INT32_MIN, 0);
    const int64_t s = l * kNnLeaf, e = min(s + kNnLeaf, n);
    for (int64_t i = s; i < e; ++i) {
      const int4 p = sorted[i];
      b.lo = make_int4(min(b.lo.x, p.x), min(b.lo.y, p.y), min(b.lo.z, p.z), 1);
      b.hi = make_int4(max(b.hi.x, p.x), max(b.hi.y, p.y), max(b.hi.z, p.z), 0);
    }
    boxes[P + l] = b;
  }
}

// boxes[i] = union of its children, for the nodes i in [first, 2 * first) of one tree level
__global__ void __launch_bounds__(256) k_parent_boxes(uint32_t first, Box* __restrict__ boxes) {
  for (uint32_t i = first + blockIdx.x * blockDim.x + threadIdx.x; i < 2 * first; i += gridDim.x * blockDim.x) {
    const Box a = boxes[2 * i], c = boxes[2 * i + 1];
    Box b;
    b.lo = make_int4(min(a.lo.x, c.lo.x), min(a.lo.y, c.lo.y), min(a.lo.z, c.lo.z), a.lo.w | c.lo.w);
    b.hi = make_int4(max(a.hi.x, c.hi.x), max(a.hi.y, c.hi.y), max(a.hi.z, c.hi.z), 0);
    boxes[i] = b;
  }
}

enum NormalMode { kNoNormals = 0, kQueryNormals = 1, kTargetNormals = 2 };

struct NnParams {
  const int4* sorted;       // [n_target] Morton-ordered target points {x, y, z, original index}
  const Box* boxes;         // [2P] heap-ordered node boxes, root at 1
  int64_t n_target;
  uint32_t P;               // leaf slots (power of two)
  const int32_t* query;     // [n_query][3]
  int64_t n_query;
  const double* normals;    // kQueryNormals: [n_query][3]; kTargetNormals: [n_target][3] by original index
  int32_t* index_out;       // [n_query] or null
  int64_t* d2_out;          // [n_query] or null
  int32_t* ties_out;        // [n_query] or null
  double* plane_out;        // [n_query] tie-averaged squared plane error, or null
  int32_t* status;
};

// squared distance from (qx, qy, qz) to the box (0 inside); coordinates are int32, so every term fits int64
__device__ __forceinline__ unsigned long long box_d2(const Box& b, long long qx, long long qy, long long qz) {
  const long long dx = max(max((long long)b.lo.x - qx, 0ll), qx - (long long)b.hi.x);
  const long long dy = max(max((long long)b.lo.y - qy, 0ll), qy - (long long)b.hi.y);
  const long long dz = max(max((long long)b.lo.z - qz, 0ll), qz - (long long)b.hi.z);
  return (unsigned long long)(dx * dx) + (unsigned long long)(dy * dy) + (unsigned long long)(dz * dz);
}

__device__ __forceinline__ Box load_box(const Box* boxes, uint32_t i) {
  Box b;
  b.lo = __ldg(&boxes[i].lo);
  b.hi = __ldg(&boxes[i].hi);
  return b;
}

template <int MODE>
__global__ void __launch_bounds__(256) k_nn_query(NnParams p) {
  const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= p.n_query) return;
  const int qx = p.query[3 * q], qy = p.query[3 * q + 1], qz = p.query[3 * q + 2];
  unsigned long long key;
  if (!grids::cell_key(qx, qy, qz, key)) atomicOr(p.status, NVF_METRIC_STATUS_RANGE);
  double n0 = 0.0, n1 = 0.0, n2 = 0.0;
  if (MODE == kQueryNormals) {
    n0 = p.normals[3 * q]; n1 = p.normals[3 * q + 1]; n2 = p.normals[3 * q + 2];
  }
  unsigned long long best = ~0ull;
  int32_t best_idx = INT32_MAX, ties = 0;
  double plane = 0.0;
  uint32_t stack_node[kNnStack];
  unsigned long long stack_lb[kNnStack];
  int sp = 0;
  uint32_t node = 1;
  while (true) {
    if (node >= p.P) {                                   // leaf: test its points
      const int64_t s = (int64_t)(node - p.P) * kNnLeaf, e = min(s + kNnLeaf, p.n_target);
      for (int64_t i = s; i < e; ++i) {
        const int4 t = __ldg(&p.sorted[i]);
        const long long dx = (long long)qx - t.x, dy = (long long)qy - t.y, dz = (long long)qz - t.z;
        const unsigned long long d = (unsigned long long)(dx * dx) + (unsigned long long)(dy * dy) +
                                     (unsigned long long)(dz * dz);
        if (d > best) continue;
        double e2 = 0.0;
        if (MODE == kQueryNormals) {
          const double pe = (double)dx * n0 + (double)dy * n1 + (double)dz * n2;
          e2 = pe * pe;
        } else if (MODE == kTargetNormals) {
          const double* nt = p.normals + 3 * (int64_t)t.w;
          const double pe = (double)dx * __ldg(nt) + (double)dy * __ldg(nt + 1) + (double)dz * __ldg(nt + 2);
          e2 = pe * pe;
        }
        if (d < best) {
          best = d; best_idx = t.w; ties = 1; plane = e2;
        } else {
          best_idx = min(best_idx, t.w); ++ties; plane += e2;
        }
      }
    } else {                                             // inner node: nearer child first, the other on the stack
      const uint32_t c0 = 2 * node, c1 = c0 + 1;
      const Box b0 = load_box(p.boxes, c0), b1 = load_box(p.boxes, c1);
      const unsigned long long l0 = b0.lo.w ? box_d2(b0, qx, qy, qz) : ~0ull;
      const unsigned long long l1 = b1.lo.w ? box_d2(b1, qx, qy, qz) : ~0ull;
      const bool v0 = b0.lo.w && l0 <= best, v1 = b1.lo.w && l1 <= best;
      if (v0 && v1) {
        const bool first0 = l0 <= l1;
        stack_node[sp] = first0 ? c1 : c0;
        stack_lb[sp] = first0 ? l1 : l0;
        ++sp;
        node = first0 ? c0 : c1;
        continue;
      }
      if (v0 || v1) {
        node = v0 ? c0 : c1;
        continue;
      }
    }
    // pop the next subtree that can still hold a point at distance <= best
    bool found = false;
    while (sp > 0) {
      --sp;
      if (stack_lb[sp] <= best) { node = stack_node[sp]; found = true; break; }
    }
    if (!found) break;
  }
  if (p.index_out) p.index_out[q] = best_idx;
  if (p.d2_out) p.d2_out[q] = (int64_t)best;
  if (p.ties_out) p.ties_out[q] = ties;
  if (p.plane_out) p.plane_out[q] = MODE == kNoNormals ? 0.0 : plane / (double)ties;
}

// Stage 1: block b sums queries [b * kRedChunk, (b + 1) * kRedChunk) in a fixed order (< 2^56 for in-range points).
__global__ void __launch_bounds__(kRedThreads) k_reduce_partials(const int64_t* __restrict__ d2,
                                                                 const double* __restrict__ plane, int64_t n,
                                                                 unsigned long long* __restrict__ part_sum,
                                                                 unsigned long long* __restrict__ part_max,
                                                                 double* __restrict__ part_plane) {
  __shared__ unsigned long long s_sum[kRedThreads], s_max[kRedThreads];
  __shared__ double s_plane[kRedThreads];
  const int tid = threadIdx.x;
  const int64_t base = (int64_t)blockIdx.x * kRedChunk;
  unsigned long long sum = 0, mx = 0;
  double ps = 0.0;
#pragma unroll
  for (int k = 0; k < kRedItems; ++k) {
    const int64_t i = base + k * kRedThreads + tid;
    if (i < n) {
      const unsigned long long v = (unsigned long long)d2[i];
      sum += v;
      mx = max(mx, v);
      if (plane) ps += plane[i];
    }
  }
  s_sum[tid] = sum; s_max[tid] = mx; s_plane[tid] = ps;
  __syncthreads();
  for (int s = kRedThreads / 2; s > 0; s >>= 1) {
    if (tid < s) {
      s_sum[tid] += s_sum[tid + s];
      s_max[tid] = max(s_max[tid], s_max[tid + s]);
      s_plane[tid] += s_plane[tid + s];
    }
    __syncthreads();
  }
  if (tid == 0) {
    part_sum[blockIdx.x] = s_sum[0];
    part_max[blockIdx.x] = s_max[0];
    part_plane[blockIdx.x] = s_plane[0];
  }
}

// Stage 2 (one block): the partials in a fixed order into NvfDistortion field [dir].  The int64 sum carries an
// overflow flag instead of wrapping.
__global__ void __launch_bounds__(kFinalThreads) k_reduce_final(const unsigned long long* __restrict__ part_sum,
                                                                const unsigned long long* __restrict__ part_max,
                                                                const double* __restrict__ part_plane, int64_t n_part,
                                                                int64_t n, int dir, NvfDistortion* out,
                                                                int32_t* status) {
  __shared__ unsigned long long s_sum[kFinalThreads], s_max[kFinalThreads];
  __shared__ double s_plane[kFinalThreads];
  __shared__ int s_ovf;
  const int tid = threadIdx.x;
  if (tid == 0) s_ovf = 0;
  unsigned long long sum = 0, mx = 0;
  double ps = 0.0;
  bool ovf = false;
  for (int64_t i = tid; i < n_part; i += kFinalThreads) {
    const unsigned long long v = part_sum[i];
    ovf |= sum + v < sum;
    sum += v;
    mx = max(mx, part_max[i]);
    ps += part_plane[i];
  }
  s_sum[tid] = sum; s_max[tid] = mx; s_plane[tid] = ps;
  __syncthreads();
  for (int s = kFinalThreads / 2; s > 0; s >>= 1) {
    if (tid < s) {
      const unsigned long long a = s_sum[tid], b = s_sum[tid + s];
      ovf |= a + b < a;
      s_sum[tid] = a + b;
      s_max[tid] = max(s_max[tid], s_max[tid + s]);
      s_plane[tid] += s_plane[tid + s];
    }
    __syncthreads();
  }
  if (ovf) s_ovf = 1;
  __syncthreads();
  if (tid == 0) {
    if (s_ovf || s_sum[0] > (unsigned long long)INT64_MAX) atomicOr(status, NVF_METRIC_STATUS_SUM_OVERFLOW);
    out->n[dir] = n;
    out->d1_sum[dir] = (int64_t)s_sum[0];
    out->d1_max[dir] = (int64_t)s_max[0];
    out->d2_sum[dir] = s_plane[0];
  }
}

}  // namespace metrics
}  // namespace nvf
