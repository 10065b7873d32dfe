/*
 * cupoch_b200.h -- C ABI of the B200-native ICP / kNN / voxel-grid engine.
 *
 * This is the drop-in boundary for cupoch's hot path (SURVEY.md section 8b).
 * cupoch has no FFI/plugin registry: its boundary is the public C++ headers
 * (and the pybind11 module built on them).  Each entry point below names the
 * reference interface it replaces; include/cupoch/ holds the header-compatible
 * C++ facade that forwards to these symbols, cupoch_b200/ the Python mirror,
 * and INTEGRATION.md the binding a cupoch maintainer would add.
 *
 * Conventions
 *   - extern "C", plain pointers + sizes, no torch / thrust / Eigen types.
 *   - all data pointers are DEVICE pointers unless the name starts with h_;
 *     they are borrowed for the duration of the call and never retained
 *     (contexts keep private re-packed copies), outputs are caller-allocated.
 *   - points / normals / colors: packed float32 xyz, 12-byte stride (the
 *     layout of cupoch's device_vector<Eigen::Vector3f>, pointcloud.h:259-262).
 *   - covariances: 9 float32 per point; cov_col_major=1 for Eigen's default
 *     column-major Matrix3f (pointcloud.h:262), 0 for row-major (numpy).
 *   - 4x4 transforms: float32[16], ROW-major.  (Eigen::Matrix4f is column-major:
 *     the facade transposes 16 floats on the host.)
 *   - sizes are 64-bit; indices are int32 like the reference.
 *   - return value: 0 = CPHB_OK, <0 = error (message via cphb_last_error()).
 *     Nothing here calls exit() (the reference's cudaSafeCall does,
 *     platform.cu:60-67).
 *   - stream: a cudaStream_t passed as void* (NULL = default stream).  Calls
 *     are asynchronous on that stream unless they return host values, in which
 *     case they synchronise the stream before returning (documented per call).
 */
#ifndef CUPOCH_B200_H
#define CUPOCH_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CPHB_VERSION 100 /* 0.1.0 */

enum cphb_status {
    CPHB_OK = 0,
    CPHB_ERR_INVALID = -1,  /* bad argument (the reference logs and continues / returns -1) */
    CPHB_ERR_CUDA = -2,     /* CUDA runtime error */
    CPHB_ERR_NO_DEVICE = -3,
    CPHB_ERR_NCCL = -4,
    CPHB_ERR_UNSUPPORTED = -5
};

/* registration::TransformationEstimationType, transformation_estimation.h:40-47 */
enum cphb_estimation {
    CPHB_EST_UNSPECIFIED = 0,
    CPHB_EST_POINT_TO_POINT = 1,
    CPHB_EST_POINT_TO_PLANE = 2,
    CPHB_EST_SYMMETRIC = 3,
    CPHB_EST_COLORED_ICP = 4,
    CPHB_EST_GENERALIZED_ICP = 5
};

int cphb_version(void);
const char *cphb_last_error(void);
/* number of kernels launched by this library since load (bench.py's gpu_launches) */
uint64_t cphb_launch_count(void);
/* cudaGetDeviceCount / properties without torch */
int cphb_device_count(void);
int cphb_set_device(int device);

/* ------------------------------------------------------------------------ *
 * Spatial index  (replaces knn::KDTreeFlann + the vendored FLANN CUDA kd-tree,
 * kdtree_flann.h:43-124, kdtree_flann.inl:125-144, kdtree_cuda_builder.h)
 * ------------------------------------------------------------------------ */
typedef struct cphb_index cphb_index;

/* KDTreeFlann::SetRawData (kdtree_flann.inl:125-144).  Like the reference the
 * index owns a private re-packed copy of the points: xyz may be freed after
 * the call returns (the call is stream-ordered; no host sync). n may be 0. */
int cphb_index_create(const float *xyz, size_t n, void *stream, cphb_index **out);
void cphb_index_destroy(cphb_index *index);
size_t cphb_index_size(const cphb_index *index);

/* KDTreeFlann::SearchRadius(query, radius, max_nn, indices, distance2)
 * (kdtree_flann.h:66-72, .inl:97-122; result set result_set.h:372-474):
 * for each query the <= max_nn nearest points with d2 < radius*radius (strict,
 * radius squared in float), ascending by (d2, index).  idx / d2 are
 * [n_query * max_nn]; unfilled slots idx=-1, d2=+inf.  1 <= max_nn <= 100
 * (NUM_MAX_NN, kdtree_search_param.h:26) else CPHB_ERR_INVALID (reference: -1).
 * h_count (optional, host): number of filled slots = the reference's return
 * value; requesting it synchronises the stream. */
int cphb_search_radius(const cphb_index *index, const float *query, size_t n_query,
                       float radius, int max_nn, int32_t *idx, float *d2,
                       int64_t *h_count, void *stream);
/* KDTreeFlann::SearchKNN (kdtree_flann.h:60-65, .inl:70-95). */
int cphb_search_knn(const cphb_index *index, const float *query, size_t n_query,
                    int knn, int32_t *idx, float *d2, int64_t *h_count, void *stream);
/* north_star's name for the same operation (SURVEY.md section 0). */
int cphb_search_hybrid(const cphb_index *index, const float *query, size_t n_query,
                       float radius, int max_nn, int32_t *idx, float *d2,
                       int64_t *h_count, void *stream);

/* ------------------------------------------------------------------------ *
 * geometry::PointCloud operations (pointcloud.h)
 * ------------------------------------------------------------------------ */
typedef struct cphb_cloud {
    const float *points;         /* n x 3 */
    const float *normals;        /* n x 3 or NULL  (HasNormals, pointcloud.h:82-94) */
    const float *colors;         /* n x 3 or NULL */
    const float *covariances;    /* n x 9 or NULL */
    const float *color_gradient; /* n x 3 or NULL (PointCloudForColoredICP, colored_icp.cu:36-40) */
    size_t n;
    int cov_col_major;
} cphb_cloud;

/* PointCloud::Transform (pointcloud.cu:293-299): in place p<-Rp+t, n<-Rn,
 * C<-R C R^T; any of normals/covariances may be NULL. */
int cphb_transform(float *points, float *normals, float *covariances, int cov_col_major,
                   size_t n, const float h_T[16], void *stream);
/* PointCloud::GetMinBound / GetMaxBound (eigen.inl:197-221). Synchronises. */
int cphb_min_max_bound(const float *points, size_t n, float h_min[3], float h_max[3], void *stream);

/* PointCloud::VoxelDownSample (down_sample.cu:170-273).  normals / colors in
 * and out may be NULL (together).  out_* must hold n elements; *h_n_out gets
 * the voxel count (synchronises).  Output order: lexicographic by voxel
 * (x,y,z) like the reference's sort.  voxel<=0 or voxel*INT_MAX < extent
 * return CPHB_OK with *h_n_out = 0 (the reference warns and returns an empty
 * cloud). */
int cphb_voxel_down_sample(const float *points, const float *normals, const float *colors,
                           size_t n, float voxel_size, float *out_points, float *out_normals,
                           float *out_colors, size_t *h_n_out, void *stream);

/* The same with a caller-supplied grid origin (every component <= the cloud's minimum): several ranks can
 * down-sample disjoint parts of one cloud on one common grid (cupoch_b200.distributed.voxel_down_sample). */
int cphb_voxel_down_sample_origin(const float *points, const float *normals, const float *colors,
                                  size_t n, float voxel_size, const float h_origin[3], float *out_points,
                                  float *out_normals, float *out_colors, size_t *h_n_out, void *stream);
/* Batched VoxelGrid::GetVoxel (voxelgrid.cu:338-341): out_indices (device, n x 3 int32) =
 * floor((p - origin) / voxel_size), the key arithmetic of every voxel kernel in this library. */
int cphb_voxel_indices(const float *points, size_t n, float voxel_size, const float h_origin[3],
                       int32_t *out_indices, void *stream);

/* PointCloud::EstimateNormals (estimate_normals.cu:82-127).  knn>0: KNN search
 * (k includes the point itself, default 30); knn<=0: radius + max_nn. */
int cphb_estimate_normals(const float *points, size_t n, int knn, float radius, int max_nn,
                          float *out_normals, void *stream);
/* Multi-GPU building block: the normals of points [first, first + count) only (out_normals holds count rows),
 * neighbours searched in the whole cloud.  Ranks estimate disjoint blocks and all-gather them; the union equals
 * cphb_estimate_normals bit for bit (same search, same per-point arithmetic). */
int cphb_estimate_normals_range(const float *points, size_t n, int knn, float radius, int max_nn, size_t first,
                                size_t count, float *out_normals, void *stream);
/* InitializePointCloudForGeneralizedICP covariance step (generalized_icp.cu:53-60). */
int cphb_covariances_from_normals(const float *normals, size_t n, float epsilon,
                                  float *out_cov, int cov_col_major, void *stream);
/* InitializePointCloudForColoredICP (colored_icp.cu:120-148): radius search
 * (radius, max_nn) + per-point intensity-gradient fit. */
int cphb_color_gradient(const float *points, const float *normals, const float *colors, size_t n,
                        float radius, int max_nn, float *out_gradient, void *stream);

/* VoxelGrid::CreateFromPointCloudWithinBounds (voxelgrid_factory.cu:164-219): grid index
 * floor((p - min_bound) / voxel_size) per point (negative below the bound, as in the reference), one voxel per
 * distinct index in lexicographic (x, y, z) order, colour = mean colour of its points ((1,1,1) when colors is
 * NULL).  out_keys (device, n x 3 int32) / out_colors (device, n x 3 float) must hold n rows; *h_n_out = voxel
 * count (synchronises).  For VoxelGrid::CreateFromPointCloud pass the cloud's bounds widened by half a voxel
 * (:221-228).  voxel_size <= 0 or voxel_size * INT_MAX < extent give an empty grid. */
int cphb_voxel_grid_from_point_cloud(const float *points, const float *colors, size_t n, float voxel_size,
                                     const float h_min_bound[3], const float h_max_bound[3], int32_t *out_keys,
                                     float *out_colors, size_t *h_n_out, void *stream);

/* PointCloud::RemoveRadiusOutliers (down_sample.cu:317-354): search the cloud against itself with
 * (radius, nb_points + 1) and keep the points all of whose slots are filled (more than nb_points neighbours
 * inside the radius, the point itself included).  indices_out (device, n int32) receives the ascending indices
 * of the kept points, *h_n_out their number (synchronises).  As in the reference a negative radius acts as
 * |radius| and radius == 0 keeps nothing; nb_points + 1 > 100 (NUM_MAX_NN) is CPHB_ERR_INVALID. */
int cphb_remove_radius_outliers(const float *points, size_t n, int nb_points, float radius,
                                int32_t *indices_out, size_t *h_n_out, void *stream);
/* PointCloud::RemoveStatisticalOutliers (down_sample.cu:356-438): per point the mean of the squared distances
 * to its nb_neighbors nearest points (itself included), cloud mean and Bessel-corrected standard deviation of
 * those means, keep 0 < mean_i < cloud mean + std_ratio * std.  h_stats (optional) = {cloud mean, std,
 * threshold}.  Outputs as above. */
int cphb_remove_statistical_outliers(const float *points, size_t n, int nb_neighbors, float std_ratio,
                                     int32_t *indices_out, size_t *h_n_out, float h_stats[3], void *stream);
/* PointCloud::GaussianFilter (pointcloud.cu:56-106,387-433): radius search of the cloud against itself
 * (search_radius, num_max_search_points <= 100), every row replaced by the exp(-0.5 d2 / sigma2)-weighted mean of
 * its neighbours' rows.  normals / colors in and out may be NULL (together); outputs hold n rows; *h_n_out = n, or
 * 0 for illegal parameters (the reference returns an empty cloud).  Synchronises. */
int cphb_gaussian_filter(const float *points, const float *normals, const float *colors, size_t n,
                         float search_radius, float sigma2, int num_max_search_points, float *out_points,
                         float *out_normals, float *out_colors, size_t *h_n_out, void *stream);
/* PointCloud::SelectByIndex (down_sample.cu:40-127, invert = false): out row t = in row indices[t].
 * normals / colors in and out may be NULL (together). */
int cphb_select_by_index(const float *points, const float *normals, const float *colors, size_t n,
                         const int32_t *indices, size_t n_indices, float *out_points, float *out_normals,
                         float *out_colors, void *stream);

/* ------------------------------------------------------------------------ *
 * registration  (registration.h:35-91, transformation_estimation.h:36-143,
 * generalized_icp.h, colored_icp.h)
 * ------------------------------------------------------------------------ */
typedef struct cphb_icp_params {
    int estimation;               /* enum cphb_estimation */
    float max_correspondence_distance;
    float relative_fitness;       /* ICPConvergenceCriteria, registration.h:35-49 */
    float relative_rmse;
    int max_iteration;
    float det_thresh;             /* PointToPlane / Symmetric / Colored: 1e-6; ignored for GICP */
    float lambda_geometric;       /* Colored ICP, default 0.968 */
    int flags;                    /* CPHB_ICP_* */
    /* Multi-GPU: with shard_world > 1 every rank passes the FULL source; the library orders it along the
     * Hilbert curve and keeps the shard_rank-th contiguous block of that order (a spatially compact
     * shard at full density).  correspondence indices stay global.  0/0 or 1 = no library-side sharding
     * (a caller may still pass its own shard together with a communicator). */
    int shard_rank;
    int shard_world;
} cphb_icp_params;

#define CPHB_ICP_NO_RETILE 2 /* keep the source in its initial Hilbert order for the whole run (debug/ablation) */

typedef struct cphb_icp_result {
    float transformation[16];     /* row-major */
    float fitness;
    float inlier_rmse;
    int64_t n_correspondences;    /* global count (all ranks) */
    int64_t n_local_correspondences; /* pairs written to corr_out by this rank (== global on one GPU) */
    int iterations;               /* updates applied */
    int converged;
    float loop_ms;                /* device time of the launch loop (CUDA events on `stream`) */
    int loop_launches;            /* kernels launched inside that region */
} cphb_icp_result;

typedef struct cphb_icp cphb_icp;
typedef struct cphb_comm cphb_comm; /* multi-GPU communicator, see the end of this header */

/* Build the per-call state of RegistrationICP (registration.cu:146-147): the
 * spatial index over target.points and a Hilbert-ordered working copy of the
 * source.  Nothing of either cloud is retained: the target points live in the
 * index, the target attributes the estimator reads (normals, colour
 * intensity, colour gradient, covariances) are copied into index order, the
 * source into its working copy -- both clouds may be freed or overwritten
 * as soon as this call's work on `stream` has completed. */
int cphb_icp_create(const cphb_cloud *source, const cphb_cloud *target,
                    const cphb_icp_params *params, void *stream, cphb_icp **out);
void cphb_icp_destroy(cphb_icp *icp);

/* Run the loop of RegistrationICP (registration.cu:148-172) from init.  One
 * fused kernel per iteration, no host round trip inside the loop.
 * comm: NULL (single GPU) or a communicator whose ranks each hold a contiguous
 * shard of the source; the 32 partial sums are exchanged once per iteration
 * (NCCL all-reduce, or the peer-memory exchange fused into the reduce kernel).  corr_out (device, optional): 2*source.n int32 receiving the
 * final correspondence set (i, j) ascending in i (local shard indices).
 * Synchronises the stream before returning h_result. */
int cphb_icp_run(cphb_icp *icp, const float h_init[16], cphb_comm *comm,
                 cphb_icp_result *h_result, int32_t *corr_out, void *stream);

/* Debug / test hook: one GetRegistrationResultAndCorrespondences +
 * ComputeJTJandJTr step at pose h_T applied to the pristine source:
 * h_sums[32] doubles = 21 JTJ upper | 6 JTr | sum r^2 | sum d^2 | count | 0 0
 * (P2P: sum s(3) sum t(3) sum s t^T(9) ... | sum d^2 | count); corr_index
 * (device, optional, source.n int32): matched target index per source point
 * or -1.  Synchronises. */
int cphb_icp_step(cphb_icp *icp, const float h_T[16], double h_sums[32],
                  int32_t *corr_index, void *stream);

/* One-shot registration::RegistrationICP / RegistrationGeneralizedICP /
 * RegistrationColoredICP on device-resident clouds.  For GICP the clouds must
 * carry covariances, for Colored ICP the target must carry color_gradient
 * (use cphb_covariances_from_normals / cphb_color_gradient, as the reference's
 * Initialize* helpers do). */
int cphb_registration_icp(const cphb_cloud *source, const cphb_cloud *target,
                          const float h_init[16], const cphb_icp_params *params,
                          cphb_comm *comm, cphb_icp_result *h_result, int32_t *corr_out,
                          void *stream);

/* The same from HOST buffers (every pointer of the two clouds is a host pointer, pinned for full speed): the
 * uploads are issued on a separate stream in the order the loop first needs them (target points, source, target
 * attributes) and overlap the index build and the source ordering.  h_corr_out (optional, host, 2 * source.n
 * int32) receives the (i, j) pairs.  Complete on return. */
int cphb_registration_icp_host(const cphb_cloud *h_source, const cphb_cloud *h_target,
                               const float h_init[16], const cphb_icp_params *params, cphb_comm *comm,
                               cphb_icp_result *h_result, int32_t *h_corr_out, void *stream);

/* TransformationEstimation*::ComputeTransformation / ComputeRMSE on an explicit correspondence list
 * (transformation_estimation.h:49-77; corr = device (i, j) pairs).  Synchronise. */
int cphb_compute_transformation(int estimation, const cphb_cloud *source, const cphb_cloud *target,
                                const int32_t *corr, size_t n_corr, const cphb_icp_params *params,
                                float h_T[16], void *stream);
int cphb_compute_rmse(int estimation, const cphb_cloud *source, const cphb_cloud *target,
                      const int32_t *corr, size_t n_corr, const cphb_icp_params *params,
                      float *h_rmse, void *stream);
/* registration::Kabsch(model, target[, corres]) (kabsch.h:30-49); corr NULL pairs i<->i. */
int cphb_kabsch(const float *model, size_t n_model, const float *target, const int32_t *corr,
                size_t n_corr, float h_T[16], void *stream);

/* registration::KabschWeighted(model, target, weight) (kabsch.h:46-49, kabsch.cu:138-201; FilterReg's M-step,
 * filterreg.cu:80): weighted centres, H = sum w^2 (m - mc)(t - tc)^T / sum w^2, R = V diag(1,1,det(UV)) U^T. */
int cphb_kabsch_weighted(const float *model, const float *target, const float *weight, size_t n,
                         float h_T[16], void *stream);

/* The other users of the normal-equation reducer (SURVEY 8f rank 3), on EXPLICIT rows: J [n][num_j][6] and r [n][num_j]
 * float32, device.  utility::ComputeJTJandJTr<Matrix6f, Vector6f, NumJ> (eigen.inl:120-145; RGB-D odometry,
 * odometry.cu:618): h_sums[32] = 21 JTJ upper | 6 JTr | sum r^2 | 0... */
int cphb_compute_jtj_jtr(const float *J, const float *r, size_t n, int num_j, double h_sums[32], void *stream);
/* utility::ComputeWeightedJTJandJTr (eigen.inl:147-195) with the Student-t weights of the RGB-D odometry
 * (odometry.cu:633-648, :688): w_sum = sum_i r2_i (nu + 1) / (nu + r2_i / sigma2), w_i = (nu + 1) / (nu + r2_i / w_sum),
 * h_sums = sums of w_i * (JTJ_i, JTr_i, r2_i) laid out as above; *h_w_sum = w_sum (the caller's next sigma2). */
int cphb_compute_weighted_jtj_jtr(const float *J, const float *r, size_t n, int num_j, float sigma2, float nu,
                                  double h_sums[32], float *h_w_sum, void *stream);

/* registration::ComputeFPFHFeature(input, search_param) (feature.h, fpfh.cu:192-229): out_features [n][33] float32.
 * knn > 0: KDTreeSearchParamKNN(knn); else KDTreeSearchParamRadius(radius, max_nn).  Normals are required. */
int cphb_compute_fpfh_feature(const float *points, const float *normals, size_t n, int knn, float radius,
                              int max_nn, float *out_features, void *stream);

/* geometry::PointCloud::ClusterDBSCAN(eps, min_points, print_progress, max_edges) (pointcloud.h:195-199,
 * pointcloud_cluster.cu:84-179): labels_out (device, n int32), -1 = noise; *h_n_clusters (optional) = cluster ids
 * handed out.  max_edges in [1, 255] (reference default NUM_MAX_NN = 100). */
int cphb_cluster_dbscan(const float *points, size_t n, float eps, int min_points, int max_edges,
                        int32_t *labels_out, int *h_n_clusters, void *stream);

/* ------------------------------------------------------------------------ *
 * geometry::OccupancyGrid (occupancygrid.h:74-147, occupancygrid.cu): a dense
 * resolution^3 log-odds grid.  Cells are float prob_log (NaN = unknown); voxel
 * (x, y, z) of the grid covers origin + (x - resolution/2 .. +1) * voxel_size.
 * ------------------------------------------------------------------------ */
typedef struct cphb_occgrid cphb_occgrid;
typedef struct cphb_occgrid_params { /* occupancygrid.h:139-143 (defaults -2.0, 3.5, 0.85, -0.4, 0.0) */
    float clamping_thres_min, clamping_thres_max, prob_hit_log, prob_miss_log, occ_prob_thres_log;
} cphb_occgrid_params;
void cphb_occgrid_default_params(cphb_occgrid_params *p);
/* OccupancyGrid(voxel_size, resolution = 512, origin = 0) (occupancygrid.cu:289-297); the grid owns its device memory */
int cphb_occgrid_create(float voxel_size, int resolution, const float origin[3], void *stream, cphb_occgrid **out);
void cphb_occgrid_destroy(cphb_occgrid *grid);
int cphb_occgrid_clear(cphb_occgrid *grid, void *stream);                       /* Clear (:310-315) */
int cphb_occgrid_set_params(cphb_occgrid *grid, const cphb_occgrid_params *p);  /* the public members :139-143 */
int cphb_occgrid_set_geometry(cphb_occgrid *grid, float voxel_size, const float origin[3]); /* voxel_size_ / origin_ */
const float *cphb_occgrid_data(const cphb_occgrid *grid);                       /* device prob_log[resolution^3], borrowed */
int cphb_occgrid_resolution(const cphb_occgrid *grid);
/* OccupancyGrid::Insert(points, viewpoint, max_range = -1) (occupancygrid.cu:462-526): every voxel crossed by a ray
 * viewpoint -> point gets prob_miss_log once, every voxel holding a point within max_range gets prob_hit_log once
 * (occupied wins), both clamped.  points: device, packed xyz. */
int cphb_occgrid_insert(cphb_occgrid *grid, const float *points, size_t n, const float viewpoint[3], float max_range,
                        void *stream);
/* AddVoxels(voxels, occupied) (:579-600): device [n][3] int32 grid indices inside the grid; AddVoxel (:554-577): one
 * host index, range-checked (CPHB_ERR_INVALID outside, where the reference logs an error). */
int cphb_occgrid_add_voxels(cphb_occgrid *grid, const int32_t *voxels, size_t n, int occupied, void *stream);
int cphb_occgrid_add_voxel(cphb_occgrid *grid, const int32_t voxel[3], int occupied, void *stream);
/* SetFreeArea(min_bound, max_bound) (:415-460): adds prob_miss_log to every cell of the (clipped) box and REPLACES the
 * grid's bound box by it, as the reference does. */
int cphb_occgrid_set_free_area(cphb_occgrid *grid, const float min_bound[3], const float max_bound[3], void *stream);
/* min_bound_ / max_bound_ (grid indices; GetMinBound / GetMaxBound :317-333 convert them to coordinates) */
int cphb_occgrid_bounds(const cphb_occgrid *grid, int32_t h_min[3], int32_t h_max[3], void *stream);
/* ExtractKnownVoxels / ExtractFreeVoxels / ExtractOccupiedVoxels (:358-408): which = 0 / 1 / 2.  Voxels of the bound
 * box that satisfy the predicate, in box order; out_index (device [capacity][3], the voxel's stored grid_index_) and
 * out_prob (device [capacity]) may be null; *h_count = number of matching voxels (call with capacity 0 to size). */
int cphb_occgrid_extract(const cphb_occgrid *grid, int which, int32_t *out_index, float *out_prob, size_t capacity,
                         size_t *h_count, void *stream);
/* GetVoxel(point) (:351-356, densegrid.inl:137-146): *h_known = inside the grid and not NaN */
int cphb_occgrid_get_voxel(const cphb_occgrid *grid, const float point[3], int *h_known, float *h_prob_log,
                           int32_t h_grid_index[3], void *stream);

/* registration::EvaluateRegistration (registration.cu:106-119). */
int cphb_evaluate_registration(const cphb_cloud *source, const cphb_cloud *target,
                               float max_correspondence_distance, const float h_T[16],
                               cphb_icp_result *h_result, int32_t *corr_out, void *stream);

/* ------------------------------------------------------------------------ *
 * Global registration: registration::FastGlobalRegistration
 * (fast_global_registration.h:43-104, fast_global_registration.cu) and
 * knn::BruteForceNN (bruteforce_nn.h).  Features are device [n][dim] float32
 * rows, dim 33 (FPFH) or 352 (SHOT, supplied by the caller).
 * ------------------------------------------------------------------------ */
typedef struct cphb_fgr_option { /* FastGlobalRegistrationOption, fast_global_registration.h:55-68 */
    float division_factor;                 /* 1.4 */
    int use_absolute_scale;                /* 0 */
    int decrease_mu;                       /* 1 */
    float maximum_correspondence_distance; /* 0.025 */
    int iteration_number;                  /* 64 */
    float tuple_scale;                     /* 0.95 */
    int maximum_tuple_count;               /* 1000 (pairs, not triplets) */
} cphb_fgr_option;
void cphb_fgr_default_option(cphb_fgr_option *option);

/* knn::BruteForceNN<dim>(ref, query, indices, distances) (bruteforce_nn.inl:101-135): for every query row the
 * nearest ref row (smallest index among equal distances) and its squared distance, exact, without the reference's
 * n_ref x n_query distance matrix.  ref_idx_out / ref_d2_out (optional, device, n_ref): also the nearest query row of
 * every ref row -- the reverse direction, taken from the same distance evaluations (the matcher FastGlobalRegistration
 * runs).  CPHB_ERR_INVALID for dim other than 33 / 352, an empty set on one side of a requested direction, or a
 * non-finite feature (found by the kernel; the outputs are then undefined).  Synchronises. */
int cphb_feature_nn(const float *ref, size_t n_ref, const float *query, size_t n_query, int dim, int32_t *idx_out,
                    float *d2_out, int32_t *ref_idx_out, float *ref_d2_out, void *stream);

/* Test hook: NormalizePointCloud + AdvancedMatching (fast_global_registration.cu:103-265) on raw clouds and features.
 * pairs_out (device, 2 * maximum_tuple_count int32) receives the final (source, target) pair list; h_counts =
 * {pairs written, mutual matches, tuple trials, pairs of passing trials before truncation}.  Synchronises. */
int cphb_fgr_advanced_matching(const float *source_points, size_t n_source, const float *target_points, size_t n_target,
                               const float *source_features, size_t n_source_features, const float *target_features,
                               size_t n_target_features, int dim, const cphb_fgr_option *option, int32_t *pairs_out,
                               int64_t h_counts[4], void *stream);

/* registration::FastGlobalRegistration<dim> (fast_global_registration.cu:391-431): matching, the graduated
 * non-convexity pose loop in one device block, then EvaluateRegistration on the original clouds.  corr_out as in
 * cphb_evaluate_registration; trace_T (device, optional, iteration_number * 16 floats): the normalised pose after
 * every iteration; h_result->loop_ms is the device time of the pose loop (CUDA events), iterations the updates
 * applied (0 with fewer than 10 pairs).  A feature count other than the point count, dim other than 33 / 352 (both before any launch)
 * and non-finite features are CPHB_ERR_INVALID; empty clouds or features give the default result (identity,
 * fitness 0) and CPHB_OK, as the reference's LogError + RegistrationResult().  Synchronises. */
int cphb_fast_global_registration(const cphb_cloud *source, const cphb_cloud *target, const float *source_features,
                                  size_t n_source_features, const float *target_features, size_t n_target_features,
                                  int dim, const cphb_fgr_option *option, cphb_icp_result *h_result, int32_t *corr_out,
                                  float *trace_T, void *stream);

/* ------------------------------------------------------------------------ *
 * Host-buffer convenience used by bench.py's e2e leg and the Python mirror:
 * thin wrappers that cudaMalloc/cudaMemcpyAsync around the calls above.
 * ------------------------------------------------------------------------ */
/* utility::InitializeAllocator(PoolAllocation, initial_pool_size, ...) (device_vector.cu:28-69): pre-reserve
 * physical memory in the stream-ordered pool that every allocation of this library comes from, so that no call
 * on the hot path ever has to grow the pool (a growth step costs tens of milliseconds). */
int cphb_reserve_pool(size_t bytes);
void *cphb_malloc(size_t bytes);              /* pool allocation on the default stream, NULL on failure */
void cphb_free(void *p);
void *cphb_malloc_host(size_t bytes);         /* pinned */
void cphb_free_host(void *p);
int cphb_memcpy_h2d(void *dst, const void *src, size_t bytes, void *stream);
int cphb_memcpy_d2h(void *dst, const void *src, size_t bytes, void *stream);
int cphb_memset(void *dst, int value, size_t bytes, void *stream);
int cphb_stream_synchronize(void *stream);
int cphb_memcpy_d2d(void *dst, const void *src, size_t bytes, void *stream);
/* CUDA events on `stream` (bench.py times the hot path on the device, not by wall clock) */
void *cphb_event_create(void);
void cphb_event_destroy(void *event);
int cphb_event_record(void *event, void *stream);
int cphb_event_elapsed_ms(void *start, void *stop, float *h_ms); /* synchronises on stop */
/* ------------------------------------------------------------------------ *
 * Multi-GPU communicator (one process per GPU, one node).  Two kinds:
 *  NCCL: rank 0 calls cphb_nccl_unique_id, the 128 bytes reach every rank by any means
 *        (torch.distributed broadcast, MPI, a file), every rank calls cphb_comm_nccl_create.
 *  P2P : every rank calls cphb_comm_p2p_create (allocates a mailbox in its HBM and returns a 64-byte
 *        CUDA IPC handle), the handles are all-gathered in rank order by any means, every rank calls
 *        cphb_comm_p2p_connect.  The per-iteration exchange is then fused into the ICP reduce kernel:
 *        NVLink stores into the peers' mailboxes + flags, no collective library on the path.
 * ------------------------------------------------------------------------ */
int cphb_nccl_unique_id(char h_id[128]);
int cphb_comm_nccl_create(const char h_id[128], int world_size, int rank, cphb_comm **out);
int cphb_comm_p2p_create(int world_size, int rank, char h_handle[64], cphb_comm **out);
int cphb_comm_p2p_connect(cphb_comm *comm, const char *h_handles /* world_size * 64 bytes */);
int cphb_comm_destroy(cphb_comm *comm);
/* in-place sum over ranks of <= 32 doubles (device buffer); what the ICP loop uses, exposed for tests */
int cphb_comm_allreduce_f64(cphb_comm *comm, double *buf, int count, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* CUPOCH_B200_H */
