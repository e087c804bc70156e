/*
 * nvf_metrics_b200.h - C ABI of the point-cloud distortion metrics: exact nearest
 * neighbours of integer lattice clouds and the D1 (point-to-point) / D2
 * (point-to-plane) mean squared errors of a reconstruction against its source.
 * Exported by the same shared library as include/nvf_b200.h (libnvf_b200.so) and
 * following the same conventions: plain C, device pointers, caller-owned memory
 * and workspace, asynchronous on `stream`, negative error codes decoded by
 * nvf_strerror(), nothing throws or exits across the boundary.
 *
 * Semantics, for a target cloud T and a query point q (integer voxel coordinates):
 *   d2(q)    = min over t in T of |q - t|^2, exact in int64 at any distance (no search radius);
 *   ties(q)  = number of target points at exactly d2(q); duplicate target points count separately;
 *   index(q) = the LOWEST target index among them (what np.argmin over exact distances returns).
 * Direction 0 is source -> reconstruction (each source point queries the reconstruction),
 * direction 1 is reconstruction -> source.  D1 per direction is the mean of d2(q); D2 per
 * direction is the mean over queries of the squared plane error averaged over ALL tied
 * neighbours t of the query:
 *   direction 0: ((s_i - r_t) . n_i)^2   (normal of the query source point)
 *   direction 1: ((r_i - s_t) . n_t)^2   (normal of the tied source point)
 * Averaging over ties makes D2 independent of the order of the points (up to the last bits of
 * float64 sums).  Sums run in a fixed order without float atomics: two calls with the same
 * inputs give bit-identical results.
 *
 * Coordinates must lie in [-2^20, 2^20) on every axis (the range of the 21-bit biased
 * fields of the grid builder's cell key); a point outside sets NVF_METRIC_STATUS_RANGE and
 * the results are then undefined (but every access stays in bounds).
 */
#ifndef NVF_METRICS_B200_H_
#define NVF_METRICS_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

enum {
  NVF_METRIC_STATUS_RANGE = 1,       /* a coordinate outside [-2^20, 2^20)                          */
  NVF_METRIC_STATUS_SUM_OVERFLOW = 2 /* an NvfDistortion.d1_sum does not fit int64 (disjoint clouds
                                        over 2^31 points tens of thousands of voxels apart)        */
};
#define NVF_METRIC_COORD_LIMIT (1 << 20)

/* Device-resident result of nvf_pc_distortion; [0] = source -> reconstruction, [1] = reconstruction -> source. */
typedef struct {
  int64_t n[2];      /* number of queries                                                  */
  int64_t d1_sum[2]; /* sum of the exact squared nearest-neighbour distances              */
  int64_t d1_max[2]; /* largest one (squared Hausdorff distance of the direction)         */
  double d2_sum[2];  /* sum of the tie-averaged squared plane errors (0 without normals)  */
} NvfDistortion;

/*
 * Nearest target point of every query point.
 *   target     [n_target,3] int32, 1 <= n_target <= INT32_MAX
 *   query      [n_query,3] int32, 0 <= n_query <= INT32_MAX
 *   index_out  [n_query] int32 lowest index of a nearest target point, or NULL
 *   d2_out     [n_query] int64 exact squared distance, or NULL
 *   ties_out   [n_query] int32 number of target points at that distance, or NULL
 *   status_out [1] int32 device word, OR of NVF_METRIC_STATUS_* (0 = exact result)
 *   workspace  nvf_nn_workspace_bytes(n_target) bytes
 */
int nvf_nn_workspace_bytes(int64_t n_target, size_t* bytes_out);
int nvf_nearest_points(const int32_t* target, int64_t n_target, const int32_t* query, int64_t n_query,
                       int32_t* index_out, int64_t* d2_out, int32_t* ties_out, int32_t* status_out, void* workspace,
                       size_t workspace_bytes, void* stream);

/*
 * D1 / D2 sums of both directions between a source cloud and its reconstruction.
 *   source          [n_source,3] int32, 1 <= n_source <= INT32_MAX
 *   source_normals  [n_source,3] float64 unit normals of the source, used as given, or NULL (d2_sum = 0)
 *   rec             [n_rec,3] int32, 1 <= n_rec <= INT32_MAX
 *   out             one device NvfDistortion
 *   status_out      [1] int32 device word, OR of NVF_METRIC_STATUS_*
 *   workspace       nvf_distortion_workspace_bytes(n_source, n_rec) bytes
 * PSNR = 10 log10(3 peak^2 / mse) with mse = max over the two directions of sum / n.
 */
int nvf_distortion_workspace_bytes(int64_t n_source, int64_t n_rec, size_t* bytes_out);
int nvf_pc_distortion(const int32_t* source, int64_t n_source, const double* source_normals, const int32_t* rec,
                      int64_t n_rec, NvfDistortion* out, int32_t* status_out, void* workspace,
                      size_t workspace_bytes, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NVF_METRICS_B200_H_ */
