// Ground-truth occupancy grid + exact nearest-point distance field of the leaf
// blocks (the training targets of the NVF path).  Replaces util_get_grids.py:19-46,
// which asks an open3d KD-tree for the nearest cloud point of EVERY grid voxel
// of every 32^3 leaf (N_leaf * 32768 Python calls) and stores
//     dist[n,0,i,j,k]    = || nearest(p) - p ||,  p = origin[n] + (i,j,k)   (float64)
//     gt_grid[n,0,i,j,k] = (dist == 0)                                     (uint8)
//
// Voxelised clouds live on the integer lattice, so the nearest-point distance
// is an exact Euclidean distance transform of a binary volume:
//   1. k_cells_insert / k_points_scatter: the cloud becomes a sparse set of
//      32^3-bit occupancy cells (4 KB each, word (a0&31)*32+(a1&31), bit a2&31),
//      found through an open-addressing hash of the cell coordinates.
//   2. k_edt_blocks: one CTA per leaf block runs the separable squared-distance
//      transform plane by plane: per plane a0', every non-empty row a1' gives
//      g(a1',k) = distance along a2 to the nearest set bit (CLZ/FFS on a 64-bit
//      window), h(j,k) = min_a1' g^2 + (j-a1')^2, and the block's 32^3 squared
//      distances (16-bit halves in shared memory) take min(d2, h + (i-a0')^2); both
//      min-plus loops run two values per instruction on VIADDMNMX.S16x2 (DPX).
//      A leaf holds at least one point, so every distance is <= 31*sqrt(3) < 54:
//      the own 32 planes are swept first, then only the outer planes within
//      floor(sqrt(max d2)) of the block.  Everything is integer arithmetic;
//      dist = sqrt((double)d2) is correctly rounded, hence bit-identical to the
//      float64 result of the reference (ties between equidistant points do not matter).
//   No float atomics, no order dependence: results are deterministic.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "nvf_common.h"

namespace nvf {
namespace grids {

constexpr int L = 32;                    // leaf edge
constexpr int RMAX = 53;                 // floor(31 * sqrt(3)): farthest possible nearest point of a non-empty leaf
constexpr int EXT = L + 2 * RMAX;        // 138 rows / planes / bits of the search window
constexpr int NC = 6;                    // 32-cells per axis that can intersect the window (unaligned origins)
constexpr int ROWW = NC + 4;             // row words: 2 zero words, 6 data words, 2 zero words
constexpr int COFF = 1 << 20;            // cell coordinates are stored biased into 21 bits
constexpr unsigned long long kEmptyKey = ~0ull;
constexpr uint32_t D2_INF = 0xFFFFu;

enum { GRID_STATUS_CELL_OVERFLOW = 1, GRID_STATUS_NOT_FOUND = 2 };

struct CellTable {
  unsigned long long* keys;   // [cap] cell key or kEmptyKey
  int32_t* vals;              // [cap] cell id or -1
  uint32_t* masks;            // [max_cells][1024] occupancy words
  int32_t* counter;           // [1] number of cells
  int32_t* status;            // [1] GRID_STATUS_* bits
  uint32_t cap_mask;          // cap - 1 (cap is a power of two)
  int32_t max_cells;
};

__device__ __forceinline__ bool cell_key(int c0, int c1, int c2, unsigned long long& key) {
  const int b0 = c0 + COFF, b1 = c1 + COFF, b2 = c2 + COFF;
  if ((unsigned)b0 >= (2u * COFF) || (unsigned)b1 >= (2u * COFF) || (unsigned)b2 >= (2u * COFF)) return false;
  key = ((unsigned long long)b0 << 42) | ((unsigned long long)b1 << 21) | (unsigned long long)b2;
  return true;
}
__device__ __forceinline__ uint32_t cell_hash(unsigned long long k) {
  k ^= k >> 33; k *= 0xff51afd7ed558ccdull; k ^= k >> 33; k *= 0xc4ceb9fe1a85ec53ull; k ^= k >> 33;
  return (uint32_t)k;
}
__device__ __forceinline__ int cell_lookup(const CellTable& T, int c0, int c1, int c2) {
  unsigned long long key;
  if (!cell_key(c0, c1, c2, key)) return -1;
  uint32_t slot = cell_hash(key) & T.cap_mask;
  for (uint32_t probe = 0; probe <= T.cap_mask; ++probe) {
    const unsigned long long k = T.keys[slot];
    if (k == key) return T.vals[slot];
    if (k == kEmptyKey) return -1;
    slot = (slot + 1) & T.cap_mask;
  }
  return -1;
}

// Pass 1a: every point claims the hash slot of its cell; the first claimant numbers the cell.
__global__ void __launch_bounds__(256) k_cells_insert(const int32_t* __restrict__ pts, int64_t n, CellTable T) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    unsigned long long key;
    if (!cell_key(pts[3 * i] >> 5, pts[3 * i + 1] >> 5, pts[3 * i + 2] >> 5, key)) {
      atomicOr(T.status, GRID_STATUS_CELL_OVERFLOW);
      continue;
    }
    uint32_t slot = cell_hash(key) & T.cap_mask;
    for (uint32_t probe = 0; probe <= T.cap_mask; ++probe) {
      const unsigned long long prev = atomicCAS(T.keys + slot, kEmptyKey, key);
      if (prev == kEmptyKey) {
        const int id = atomicAdd(T.counter, 1);
        if (id < T.max_cells) {
          T.vals[slot] = id;
        } else {
          T.vals[slot] = -1;
          atomicOr(T.status, GRID_STATUS_CELL_OVERFLOW);
        }
        break;
      }
      if (prev == key) break;
      slot = (slot + 1) & T.cap_mask;
    }
  }
}

// Pass 1b: set the point's bit in its cell.
__global__ void __launch_bounds__(256) k_points_scatter(const int32_t* __restrict__ pts, int64_t n, CellTable T) {
  for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const int a0 = pts[3 * i], a1 = pts[3 * i + 1], a2 = pts[3 * i + 2];
    const int id = cell_lookup(T, a0 >> 5, a1 >> 5, a2 >> 5);
    if (id >= 0) atomicOr(T.masks + (size_t)id * 1024 + (a0 & 31) * 32 + (a1 & 31), 1u << (a2 & 31));
  }
}

struct EdtParams {
  const int32_t* origins;   // [n][3]
  uint8_t* gt;              // [n][32768] or null
  double* dist64;           // [n][32768] or null
  float* dist32;            // [n][32768] or null
  uint16_t* d2;             // [n][32768] or null  (squared distance, 0xFFFF = nothing within max_radius)
  int32_t max_radius;       // <= RMAX
  CellTable T;
};

// Squared distances live in shared memory as signed 16-bit halves of 32-bit words so that the two inner loops
// run on the packed DPX instruction VIADDMNMX.S16x2 (min(a + b, c) on both halves at once):
//   - all real values are <= 3 * 84^2 < 0x3FFF = D2P_INF, and D2P_INF + 87^2 < 2^15, so no sum overflows;
//   - column (j, k) owns 16 consecutive words: word w holds slices 2w (low half) and 2w + 1.  A thread reads its
//     32 slices with 4 x LDS.128; the 128-bit chunk q of column c sits at chunk q ^ ((k >> 1) & 3), which makes
//     the accesses of the 32 lanes (consecutive k, 64-byte stride) bank-conflict free without padding.
constexpr uint32_t D2P_INF = 0x3FFFu, D2P_INF2 = 0x3FFF3FFFu;
constexpr int SQ_OFF = 85, SQ_N = 172;   // sq2[d + SQ_OFF] = pack(d^2, (d + 1)^2), d in [-85, 86]

struct EdtSmem {
  uint32_t d2p[L * L * (L / 2)];    // 64 KB running squared distances, see above
  uint32_t g2c[EXT][L];             // per NON-EMPTY row n of the current plane (compact index): (g^2, g^2) packed,
                                    // g = distance along a2 to the nearest set bit (D2P_INF = none)
  uint32_t sqc[EXT][16];            // per non-empty row n and warp w: pack((4w - jrel)^2, (4w+1 - jrel)^2), pack((4w+2..)^2, (4w+3..)^2)
  uint32_t rowbits[EXT][ROWW];      // bit window of every row of the current plane
  uint32_t sq2[SQ_N];
  int32_t cellid[NC][NC][NC];
  int32_t slab_any[NC];
  int32_t rowlist[EXT];
  int32_t nrows;
  uint32_t red[8];
};
__device__ __forceinline__ int d2p_chunk(int k, int q) { return q ^ ((k >> 1) & 3); }

// 64 window bits starting at bit position b of a row (b + 64 <= 32 * ROWW)
__device__ __forceinline__ unsigned long long row_bits64(const uint32_t* row, int b) {
  const int q = b >> 5, sh = b & 31;
  const uint32_t w0 = row[q], w1 = row[q + 1], w2 = row[q + 2];
  const uint32_t lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
  return ((unsigned long long)hi << 32) | lo;
}

// One plane a0 = o0 + prel of the window: fold it into the block's squared distances.
// rlim: only rows / output slices within rlim of the block can still improve a distance.
__device__ __forceinline__ void edt_plane(EdtSmem& S, const EdtParams& p, int o0, int o1, int cb0, int cb1, int xoff,
                                          int prel, int rlim) {
  const int tid = threadIdx.x;
  const int a0 = o0 + prel;
  const int cz = (a0 >> 5) - cb0;
  if (!S.slab_any[cz]) return;                       // uniform: no cell in this slab of the window
  // ---- (1) fetch the bit windows of the rows within rlim of the block
  const int r_lo = RMAX - rlim, r_hi = RMAX + L - 1 + rlim;
  for (int idx = tid; idx < EXT * NC; idx += kThreads) {
    const int r = idx / NC, cx = idx - r * NC;
    uint32_t w = 0;
    if (r >= r_lo && r <= r_hi) {
      const int a1 = o1 + r - RMAX;
      const int cid = S.cellid[cz][(a1 >> 5) - cb1][cx];
      if (cid >= 0) w = __ldg(p.T.masks + (size_t)cid * 1024 + (a0 & 31) * 32 + (a1 & 31));
    }
    S.rowbits[r][2 + cx] = w;
  }
  __syncthreads();
  // ---- (2) ordered list of the non-empty rows (warp 0)
  if (tid < 32) {
    int base = 0;
    for (int it = 0; it < (EXT + 31) / 32; ++it) {
      const int r = it * 32 + tid;
      bool ne = false;
      if (r < EXT) {
        uint32_t o = 0;
#pragma unroll
        for (int c = 0; c < NC; ++c) o |= S.rowbits[r][2 + c];
        ne = o != 0;
      }
      const uint32_t b = __ballot_sync(0xffffffffu, ne);
      if (ne) S.rowlist[base + __popc(b & ((1u << tid) - 1u))] = r;
      base += __popc(b);
    }
    if (tid == 0) S.nrows = base;
  }
  __syncthreads();
  const int nrows = S.nrows;
  if (nrows == 0) return;                            // uniform
  // ---- (3) squared distance along a2 to the nearest set bit, for the 32 columns of the block, stored per
  //          compact row index; and the (j - row)^2 pairs every warp needs for that row
  for (int idx = tid; idx < nrows * L; idx += kThreads) {
    const int n = idx >> 5, k = idx & 31;
    const uint32_t* row = S.rowbits[S.rowlist[n]];
    const int c = 64 + xoff + RMAX + k;              // bit position of column k in the padded row
    const unsigned long long below = row_bits64(row, c - 63);   // bit 63 = position c
    const unsigned long long above = row_bits64(row, c);        // bit 0 = position c
    uint32_t g = 64;
    if (below) g = (uint32_t)__clzll((long long)below);
    if (above) g = min(g, (uint32_t)(__ffsll((long long)above) - 1));
    S.g2c[n][k] = (g >= 64 ? D2P_INF : g * g) * 0x10001u;
  }
  for (int idx = tid; idx < nrows * 16; idx += kThreads) {
    const int n = idx >> 4, e = idx & 15;
    S.sqc[n][e] = S.sq2[SQ_OFF + 2 * e - (S.rowlist[n] - RMAX)];      // rows j = 2e, 2e + 1
  }
  __syncthreads();
  // ---- (4) thread (k, rows j0..j0+3): h(j) = min over rows of g2 + (j - row)^2, two rows j per DPX instruction
  const int k = tid & 31, wid = tid >> 5, j0 = wid * 4;
  uint32_t h01 = D2P_INF2, h23 = D2P_INF2;
  {
    const uint32_t* gp = &S.g2c[0][k];
    const uint2* sp = reinterpret_cast<const uint2*>(&S.sqc[0][2 * wid]);
#pragma unroll 4
    for (int n = 0; n < nrows; ++n) {
      const uint32_t vv = gp[n * L];
      const uint2 sq = sp[n * 8];
      h01 = __viaddmin_s16x2(vv, sq.x, h01);
      h23 = __viaddmin_s16x2(vv, sq.y, h23);
    }
  }
  //      then d2(i) = min(d2(i), h + (i - prel)^2) for the slices within rlim of the plane, eight slices per LDS.128
  const int i_lo = max(0, prel - rlim), i_hi = min(L - 1, prel + rlim);
  if (i_lo > i_hi) return;
  const int q_lo = i_lo >> 3, q_hi = i_hi >> 3;
  const uint32_t* dd = S.sq2 + SQ_OFF - prel;        // dd[2w] = pack((2w - prel)^2, (2w + 1 - prel)^2)
#pragma unroll
  for (int t = 0; t < 4; ++t) {
    const uint32_t ht = ((t < 2 ? h01 : h23) >> (16 * (t & 1))) & 0xFFFFu;
    if (ht >= D2P_INF) continue;
    const uint32_t hh = ht * 0x10001u;
    uint4* col = reinterpret_cast<uint4*>(S.d2p + ((j0 + t) * L + k) * (L / 2));
    for (int q = q_lo; q <= q_hi; ++q) {
      uint4 c = col[d2p_chunk(k, q)];
      c.x = __viaddmin_s16x2(hh, dd[8 * q], c.x);
      c.y = __viaddmin_s16x2(hh, dd[8 * q + 2], c.y);
      c.z = __viaddmin_s16x2(hh, dd[8 * q + 4], c.z);
      c.w = __viaddmin_s16x2(hh, dd[8 * q + 6], c.w);
      col[d2p_chunk(k, q)] = c;
    }
  }
  // no trailing barrier: the next plane writes rowbits in its step (1), which nobody reads after the barrier that ended
  // step (3) above, and touches rowlist / g2c / sqc only after its own first barrier, which every thread reaches after
  // finishing this step; the d2p columns are private to their thread.
}

__device__ __forceinline__ int isqrt_floor(uint32_t v) {
  int r = (int)sqrtf((float)v);
  while ((uint32_t)(r * r) > v) --r;
  while ((uint32_t)((r + 1) * (r + 1)) <= v) ++r;
  return r;
}

__global__ void __launch_bounds__(kThreads, 2) k_edt_blocks(EdtParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  EdtSmem& S = *reinterpret_cast<EdtSmem*>(smem_raw);
  const int tid = threadIdx.x;
  const int n = blockIdx.x;
  const int o0 = p.origins[3 * n], o1 = p.origins[3 * n + 1], o2 = p.origins[3 * n + 2];
  const int cb0 = (o0 - RMAX) >> 5, cb1 = (o1 - RMAX) >> 5, cb2 = (o2 - RMAX) >> 5;
  const int xoff = (o2 - RMAX) - 32 * cb2;           // bit offset of the window start in data word 0
  // ---- setup: cells of the window, zero pad words, table of squares, distances = infinity
  if (tid < NC) S.slab_any[tid] = 0;
  __syncthreads();
  for (int i = tid; i < NC * NC * NC; i += kThreads) {
    const int cx = i % NC, cy = (i / NC) % NC, cz = i / (NC * NC);
    const int id = cell_lookup(p.T, cb0 + cz, cb1 + cy, cb2 + cx);
    S.cellid[cz][cy][cx] = id;
    if (id >= 0) S.slab_any[cz] = 1;
  }
  for (int r = tid; r < EXT; r += kThreads) {
    S.rowbits[r][0] = 0; S.rowbits[r][1] = 0; S.rowbits[r][ROWW - 2] = 0; S.rowbits[r][ROWW - 1] = 0;
  }
  for (int i = tid; i < SQ_N; i += kThreads) {
    const int d = i - SQ_OFF;
    S.sq2[i] = (uint32_t)(d * d) | ((uint32_t)((d + 1) * (d + 1)) << 16);
  }
  for (int i = tid; i < L * L * (L / 2); i += kThreads) S.d2p[i] = D2P_INF2;
  __syncthreads();
  const int R = min(max(p.max_radius, 0), RMAX);
  // ---- own planes
  for (int prel = 0; prel < L; ++prel) edt_plane(S, p, o0, o1, cb0, cb1, xoff, prel, R);
  __syncthreads();
  // ---- largest squared distance so far bounds the remaining search radius
  uint32_t m = 0;
  for (int i = tid; i < L * L * (L / 2); i += kThreads) {
    const uint32_t v = S.d2p[i];
    m = max(m, max(v & 0xFFFFu, v >> 16));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = max(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((tid & 31) == 0) S.red[tid >> 5] = m;
  __syncthreads();
  m = 0;
#pragma unroll
  for (int w = 0; w < kThreads / 32; ++w) m = max(m, S.red[w]);
  const int rlim = m >= D2P_INF ? R : min(R, isqrt_floor(m));
  // ---- outer planes, nearest first
  for (int dz = 1; dz <= rlim; ++dz) {
    edt_plane(S, p, o0, o1, cb0, cb1, xoff, -dz, rlim);
    edt_plane(S, p, o0, o1, cb0, cb1, xoff, L - 1 + dz, rlim);
  }
  __syncthreads();
  // ---- outputs, [i][j][k] order
  const size_t base = (size_t)n * (L * L * L);
  bool missing = false;
  for (int i = tid; i < L * L * L; i += kThreads) {
    const int sl = i >> 10, c = i & 1023;
    const int w = sl >> 1;
    const uint32_t v = (S.d2p[c * (L / 2) + 4 * d2p_chunk(c & 31, w >> 2) + (w & 3)] >> (16 * (sl & 1))) & 0xFFFFu;
    const bool none = v >= D2P_INF;
    missing |= none;
    const double d = none ? __longlong_as_double(0x7ff0000000000000ll) : sqrt((double)v);
    if (p.gt) p.gt[base + i] = v == 0 ? 1 : 0;
    if (p.dist64) p.dist64[base + i] = d;
    if (p.dist32) p.dist32[base + i] = (float)d;
    if (p.d2) p.d2[base + i] = none ? (uint16_t)D2_INF : (uint16_t)v;
  }
  if (missing) atomicOr(p.T.status, GRID_STATUS_NOT_FOUND);
}

}  // namespace grids
}  // namespace nvf
