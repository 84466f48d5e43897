/*
 * apc.h - C ABI of the B200-native per-scan point-cloud preprocessing hot path.
 *
 * "apc" = autodriver point cloud.  This is the drop-in boundary: plain C types, device
 * pointers and sizes, no torch / Open3D types, no exceptions.  Each entry point replaces a
 * call the reference (privvyledge/autodriver_pointcloud_preprocessor, all Python) makes
 * into numpy / torch / Open3D / sensor_msgs_py; the replaced call site is cited on every
 * declaration as <file>:<line> relative to the reference root, with
 *   pp.py    = autodriver_pointcloud_preprocessor/pointcloud_preprocessor.py
 *   utils.py = autodriver_pointcloud_preprocessor/utils.py
 *   concat.py= autodriver_pointcloud_preprocessor/pointcloud_concatenator.py
 * The Python binding a maintainer adds on the reference side is ctypes; see INTEGRATION.md.
 *
 * Conventions
 *   - every pointer named *_dev / documented "device" is a CUDA device pointer owned by the
 *     caller (a torch tensor in the Python host code); the context owns only scratch.
 *   - point clouds are SoA: `xyzi` is float4[N] = (x, y, z, intensity) per point, 16-byte
 *     aligned; other attributes travel as separate arrays gathered with apc_gather /
 *     averaged with apc_voxel_mean_attr.
 *   - variable-size results never force a host sync: a stage takes its input size as
 *     `n_max` (host upper bound, sizes the grid) plus an optional device counter `n_dev`
 *     (when non-NULL the kernels read the true size from it) and writes its output size to
 *     a device counter.  Output buffers must hold `n_max` elements.
 *   - `stream` is a cudaStream_t passed as void* (0 = default stream).  Calls are
 *     asynchronous; a context is bound to one device (which must be the calling thread's
 *     current device: APC_ERR_BAD_ARG otherwise) and must be used from one thread / stream
 *     at a time (the reference runs one callback at a time, pp.py:1056).
 *   - return value: APC_OK or a negative apc_status; apc_last_error(ctx) gives the text.
 *     Data-dependent failures (key range, table capacity) are raised on the device and
 *     reported by apc_check(ctx) after the stream has been synchronised.
 */
#ifndef APC_H_
#define APC_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define APC_VERSION 120 /* 0.1.2: + mirrored outputs (multi-GPU exchange fused into the final stage) */

typedef enum apc_status {
  APC_OK = 0,
  APC_ERR_CUDA = -1,       /* a CUDA runtime call failed */
  APC_ERR_BAD_ARG = -2,    /* NULL pointer, size over the context limit, bad enum ... */
  APC_ERR_KEY_RANGE = -3,  /* voxel index outside +-2^20 or |coordinate| >= 2^16 m */
  APC_ERR_CAPACITY = -4,   /* hash table / scratch too small for this input */
  APC_ERR_TOO_FEW = -5     /* fewer points than ransac_n (segment_plane) */
} apc_status;

/* sensor_msgs/PointField datatype codes (utils.py:28-37 FIELD_DTYPE_MAP) */
enum { APC_INT8 = 1, APC_UINT8 = 2, APC_INT16 = 3, APC_UINT16 = 4, APC_INT32 = 5,
       APC_UINT32 = 6, APC_FLOAT32 = 7, APC_FLOAT64 = 8 };

#define APC_MAX_FIELDS 16     /* fields read_points may test for NaN */
#define APC_MAX_CLOUDS 8      /* sensors merged in one launch */
#define APC_MAX_TRANSFORMS 3  /* offset(lidar) -> TF -> offset(robot), pp.py:480-491 */
#define APC_MAX_NEIGHBORS 1024 /* statistical nb_neighbors and normals max_nn */

typedef struct apc_field {
  int32_t offset;   /* byte offset inside a point record */
  int32_t datatype; /* APC_INT8 .. APC_FLOAT64; 0 = field absent */
} apc_field;

/* One PointCloud2 byte buffer (= one sensor).  Mirrors the message attributes read by
 * read_points (utils.py:206-211) and convert_pointcloud_to_numpy (utils.py:102-131). */
typedef struct apc_cloud_desc {
  const void* data_dev;   /* device: width*height*point_step bytes */
  uint32_t n_points;      /* width*height */
  uint32_t point_step;
  apc_field x, y, z;      /* any numeric datatype; cast to float32 like .astype(np.float32) */
  apc_field intensity;    /* datatype 0 -> intensity 0.0f */
  uint32_t n_nan_fields;  /* read_points NaN test: every selected field; ints never NaN */
  apc_field nan_fields[APC_MAX_FIELDS];
  int32_t has_transform;  /* per-sensor extrinsic applied before the common transforms */
  float transform[16];    /* row-major float32 4x4 (concat.py:1-5 "transform to a target frame") */
} apc_cloud_desc;

/* crop back ends, utils.py:254,272,298 */
enum { APC_CROP_NUMPY = 0,  /* float64 compare; invert = any(p<=min | p>=max) */
       APC_CROP_TORCH = 1,  /* float32 compare; invert as numpy */
       APC_CROP_OPEN3D = 2  /* float32 inclusive; invert = logical NOT */ };

/* duplicate-removal back ends, utils.py:520,535,543 */
enum { APC_DEDUP_OFF = 0,
       APC_DEDUP_OPEN3D = 1, /* remove_duplicated_points: bit-pattern key, lowest index kept, order preserved */
       APC_DEDUP_NUMPY = 2,  /* np.unique(axis=0, return_index): sorted unique rows, -0 == +0, NaN rows kept */
       APC_DEDUP_TORCH_COMPAT = 3 /* utils.py:538-542 as written: points[inverse of torch.unique], N rows */ };

typedef struct apc_filter_cfg {
  int32_t skip_nans;      /* read_points: (skip_nans && !is_dense), utils.py:209 */
  int32_t dedup_mode;     /* APC_DEDUP_* , pp.py:450-463 */
  int32_t remove_nan;     /* pp.py:469-471 */
  int32_t remove_inf;
  uint32_t n_transforms;  /* applied back to back, each rounded to float32 (pp.py:480-491) */
  float transforms[APC_MAX_TRANSFORMS][16];
  int32_t crop_enable;    /* pp.py:494-506 */
  int32_t crop_mode;      /* APC_CROP_* */
  int32_t crop_invert;
  double roi_min[3];
  double roi_max[3];
} apc_filter_cfg;

/* bits of the optional per-input-point stage mask written by apc_frontend */
enum { APC_STAGE_NANSKIP = 1, APC_STAGE_DEDUP = 2, APC_STAGE_FINITE = 4, APC_STAGE_CROP = 8 };

typedef struct apc_ctx apc_ctx;

/* ---- lifecycle ------------------------------------------------------------------ */

/* Creates a context on `device` with scratch for clouds of up to `max_points` points
 * (sum over sensors).  Replaces the reference's per-node Open3D device/point-cloud setup
 * (pp.py:272-280, pp.py:309). */
int apc_ctx_create(int device, uint32_t max_points, apc_ctx** out);
int apc_ctx_destroy(apc_ctx* ctx);
/* text of the last error recorded on this context ("" if none); ctx may be NULL for
 * errors raised by apc_ctx_create */
const char* apc_last_error(const apc_ctx* ctx);
/* Synchronises `stream`, then reports (and clears) data-dependent device-side errors of
 * the calls issued since the previous check: APC_OK / APC_ERR_KEY_RANGE / APC_ERR_CAPACITY. */
int apc_check(apc_ctx* ctx, void* stream);
int apc_version(void);
/* Low-latency mode for a context that has ONE scan in flight at a time (the reference's callback model,
 * pp.py:1056): the kernels of the per-scan chain are launched as programmatic dependents, so every kernel
 * is set up while its predecessor still runs and starts the moment that one has completed.  Shortens a
 * scan's latency by the launch gaps between its ~13 kernels; leave it off when several contexts share the
 * GPU for throughput (the waiting CTAs take room).  Affects launches and graphs captured afterwards.
 * Measured: inside a captured graph the gaps are already small (-1.6 ... +5 us per scan over the round's
 * runs, i.e. no reliable gain); it is meant for eager call sequences. */
int apc_ctx_set_low_latency(apc_ctx* ctx, int on);
uint32_t apc_ctx_max_points(const apc_ctx* ctx);

/* Per-kernel timing, the device-side counterpart of the reference's processing_times dict
 * (pp.py:322, filled at pp.py:417-678).  While enabled, every kernel launched through this
 * context is bracketed by CUDA events on its launching stream (eager calls only - not while
 * capturing a graph).  apc_profile_report synchronises the device, writes one line
 * "<kernel> <total_ms> <launches>\n" per kernel name into buf (NUL-terminated, truncated to
 * buf_len), clears the collected samples and returns the number of bytes written. */
int apc_profile_enable(apc_ctx* ctx, int on);
int apc_profile_report(apc_ctx* ctx, char* buf, uint32_t buf_len);

/* ---- (1)+(2)+(6) unpack, transform, filter, compact, concat --------------------- */

/* Fused front end over 1..APC_MAX_CLOUDS PointCloud2 byte buffers, in one launch:
 *   read_points NaN skip (utils.py:206-211) -> [duplicate removal, utils.py:509-546] ->
 *   remove_non_finite_points (pp.py:469) -> per-sensor transform (concat.py:1-5) ->
 *   common transforms (pp.py:482,487,490) -> crop_pointcloud (utils.py:240-301) ->
 *   order-preserving select_by_mask (utils.py:271,297).
 * Outputs (device, capacity = sum of n_points): out_xyzi float4[], out_src_idx uint32[]
 * (index of each survivor in the concatenated input; NULL to skip), out_stage_mask
 * uint8[sum n_points] (APC_STAGE_* bits per input point; NULL to skip),
 * out_count_dev uint32[1]. */
int apc_frontend(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                 const apc_filter_cfg* cfg, float* out_xyzi, uint32_t* out_src_idx,
                 uint8_t* out_stage_mask, uint32_t* out_count_dev, void* stream);

/* PointCloud2 bytes -> SoA float4 without filtering (utils.py:51-133 positions+intensity). */
int apc_unpack(apc_ctx* ctx, const apc_cloud_desc* cloud, float* out_xyzi, void* stream);

/* t.PointCloud.transform on an SoA cloud, in place allowed (pp.py:482,487,490). */
int apc_transform(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                  const float* T16_host, float* out_xyzi, void* stream);

/* Masks computed stand-alone for the Open3D-like carrier methods:
 * crop (utils.py:267-299), remove_non_finite_points (pp.py:469),
 * remove_duplicated_points (utils.py:544).  out_mask uint8[n_max], 1 = keep. */
int apc_crop_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                  const double* roi_min, const double* roi_max, int mode, int invert,
                  uint8_t* out_mask, void* stream);
int apc_non_finite_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                        int remove_nan, int remove_inf, uint8_t* out_mask, void* stream);
int apc_duplicate_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                       uint8_t* out_mask, void* stream);

/* np.unique(points, axis=0, return_index=True, return_inverse=True) on the positions of an SoA
 * cloud (utils.py:532-533 numpy back end; torch.unique(dim=0, return_inverse=True),
 * utils.py:538-540): rows ordered lexicographically x, y, z with float comparison (-0 == +0, NaN
 * last), a row holding a NaN is never merged.  out_first_idx uint32[n_max]: lowest input index of
 * every unique row, in sorted row order; out_inverse uint32[n_max]: unique-row number of every
 * input point; either may be NULL.  out_count_dev uint32[1]: number of unique rows.  A stable
 * 96-bit-key radix sort (12 passes of 8 bits) on the device. */
int apc_unique_rows(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                    uint32_t* out_first_idx, uint32_t* out_inverse, uint32_t* out_count_dev,
                    void* stream);

/* select_by_mask (utils.py:271,297; pp.py:542 with invert): order-preserving compaction.
 * out_idx (uint32[n_max], may be NULL) receives the surviving indices. */
int apc_select_by_mask(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                       const uint8_t* mask, int invert, float* out_xyzi, uint32_t* out_idx,
                       uint32_t* out_count_dev, void* stream);

/* select_by_index for attribute arrays (pp.py:801 copy_fields after filtering):
 * out[i] = src[idx[i]] for elem_size in {1,2,4,8,12,16} bytes. */
int apc_gather(apc_ctx* ctx, const void* src, uint32_t elem_size, const uint32_t* idx,
               uint32_t n_max, const uint32_t* n_dev, void* out, void* stream);

/* Carrier layout glue: the Open3D-style carrier keeps positions as float32[N,3] plus an
 * optional float32[N] intensity (utils.py:102-104,121; pp.py:426); the kernels work on SoA
 * float4.  Both directions stay on the device.  intensity / out_intensity may be NULL. */
int apc_pack_xyzi(apc_ctx* ctx, const float* pos3, const float* intensity, uint32_t n,
                  float* out_xyzi, void* stream);
int apc_split_xyzi(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                   float* out_pos3, float* out_intensity, void* stream);

/* ---- (3) voxel grid ---------------------------------------------------------------- */

/* voxel_down_sample(voxel_size) (pp.py:509-512), mean reduction, float32 voxel index
 * floor(x / voxel_size), output in first-occurrence order, centroids by deterministic
 * fixed-point accumulation (see DESIGN.md).  out_p2v int32[n_max] (voxel row of every input
 * point) and out_voxel_counts uint32[n_max] may be NULL. */
int apc_voxel_downsample(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                         float voxel_size, float* out_xyzi, int32_t* out_p2v,
                         uint32_t* out_voxel_counts, uint32_t* out_count_dev, void* stream);

/* The same voxel grid by SORTING instead of hashing - the alternative BASELINE.json north_star (3) names
 * ("a hand-written onesweep radix sort, followed by a segmented centroid reduce"): biased 21-bit voxel
 * indices -> stable LSD radix sort of {ix, iy, iz, index} (9 byte passes, identity passes collapse) ->
 * segmented fixed-point reduce.  Same voxels, counts and bit-identical centroids as
 * apc_voxel_downsample, but in ASCENDING (ix, iy, iz) order instead of first-occurrence order.  Kept
 * for the hash-vs-sort comparison (profiles/voxel_ab.py, DESIGN.md); the pipeline uses the hash. */
int apc_voxel_downsample_sorted(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                float voxel_size, float* out_xyzi, uint32_t* out_voxel_counts,
                                uint32_t* out_count_dev, void* stream);

/* Per-attribute voxel mean (Open3D index_add per attribute then sum / count, SURVEY.md B7; the caller
 * casts the result back to the attribute's dtype, pp.py:511) for a float32 attribute array, using p2v /
 * counts from apc_voxel_downsample or apc_pipeline_run_maps.  Order-independent like the positions:
 * values are accumulated as rint(v * 2^frac_bits) in 64-bit integers, the mean is one float64 divide
 * rounded to float32.  frac_bits = 0 for integer-valued attributes (ring, return_type: exact), up to 30
 * for real-valued ones; |v * 2^frac_bits| must stay below 2^40 (APC_ERR_KEY_RANGE at apc_check). */
int apc_voxel_mean_attr(apc_ctx* ctx, const float* attr, const int32_t* p2v, uint32_t n_max,
                        const uint32_t* n_dev, const uint32_t* n_voxels_dev, int32_t frac_bits,
                        float* out_attr, void* stream);

/* ---- (5) outlier removal ----------------------------------------------------------- */

/* remove_radius_outliers(nb_points, search_radius) (TODO at pp.py:37; Open3D semantics):
 * keep iff #{j : d2(i,j) <= r^2, self included} >= nb_points.  out_mask uint8[n_max];
 * out_neighbor_counts uint32[n_max] may be NULL. */
int apc_radius_outliers(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                        int nb_points, double radius, uint8_t* out_mask,
                        uint32_t* out_neighbor_counts, void* stream);

/* remove_statistical_outliers(nb_neighbors, std_ratio) (pp.py:514-519), nb_neighbors in
 * 1..APC_MAX_NEIGHBORS (APC_ERR_BAD_ARG beyond).  out_avg
 * float32[n_max] (mean distance to the k nearest, self included) may be NULL;
 * out_stats_dev double[3] = (mu, sigma, threshold) may be NULL. */
int apc_statistical_outliers(apc_ctx* ctx, const float* xyzi, uint32_t n_max,
                             const uint32_t* n_dev, int nb_neighbors, double std_ratio,
                             uint8_t* out_mask, float* out_avg, double* out_stats_dev,
                             void* stream);

/* estimate_normals(radius, max_nn) (pp.py:521-530, on by default pp.py:176; Open3D hybrid search):
 * neighbourhood = the max_nn (1..APC_MAX_NEIGHBORS) nearest of the points with d2 <= float32(radius)^2, query
 * included, ties by lower index; normal = eigenvector of the smallest eigenvalue of the
 * neighbourhood covariance (analytic symmetric 3x3 solver), not oriented; fewer than 3 neighbours
 * -> (0, 0, 1).  out_normals float32[3*n_max]; out_neighbor_counts uint32[n_max] and
 * out_covariances double[9*n_max] (row-major, divided by the count) may be NULL. */
int apc_estimate_normals(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                         int max_nn, double radius, float* out_normals,
                         uint32_t* out_neighbor_counts, double* out_covariances, void* stream);

/* estimate_normals(max_nn) (Open3D KNN search): the same, with the neighbourhood = the min(max_nn, n) points
 * first in the order (d2, index), query included, no distance bound; max_nn in 1..APC_MAX_NEIGHBORS
 * (APC_ERR_BAD_ARG beyond).  Points the grid cannot key get the normal (0, 0, 0) and the count 0. */
int apc_estimate_normals_knn(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                             int max_nn, float* out_normals, uint32_t* out_neighbor_counts,
                             double* out_covariances, void* stream);

/* estimate_normals(radius) (Open3D radius search): the same, with the neighbourhood = every point with
 * d2 <= float32(radius)^2, query included, no cap on the count; radius finite and > 0 (APC_ERR_BAD_ARG
 * otherwise).  Moments are accumulated in 64-bit fixed point (2^-40 r): the covariances and normals are
 * bit-identical across runs and input orders, within 1e-11 r^2 of the float64 covariance. */
int apc_estimate_normals_radius(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                                double radius, float* out_normals, uint32_t* out_neighbor_counts,
                                double* out_covariances, void* stream);

/* cluster_dbscan(eps, min_points) (Open3D PointCloud::ClusterDBSCAN): N(i) = every point with
 * d2 <= float32(eps)^2, i included; i is core iff |N(i)| >= min_points; clusters are the connected components of
 * the core points linked by N, numbered 0, 1, ... in the order of each component's lowest core index.
 * out_labels int32[n_max]: a core point's cluster; a non-core point's smallest cluster among the core points in
 * N(i); else -1 (noise).  out_cluster_count_dev uint32[1] (device, may be NULL): the number of clusters.
 * out_neighbor_counts uint32[n_max] (may be NULL): |N(i)|.  eps finite and > 0 with float32(eps)^2 finite,
 * min_points >= 0 (APC_ERR_BAD_ARG otherwise); no cap on |N(i)|.  The labels do not depend on the thread
 * schedule.  Points the grid cannot key get -1 and are in no N(i).  No host synchronisation. */
int apc_cluster_dbscan(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                       double eps, int min_points, int32_t* out_labels,
                       uint32_t* out_cluster_count_dev, uint32_t* out_neighbor_counts, void* stream);

/* ---- (3b) ICP registration (Open3D t.pipelines.registration) -------------------------- */

enum { APC_ICP_POINT_TO_POINT = 0, APC_ICP_POINT_TO_PLANE = 1, APC_ICP_GENERALIZED = 2 };
enum { APC_ICP_OK = 0, APC_ICP_NO_CORRESPONDENCE = 1, APC_ICP_DEGENERATE = 2 };

/* evaluate_registration(source, target, max_correspondence_distance, transformation) (Open3D
 * t::pipelines::registration::EvaluateRegistration).  Contract (oracle/registration.py): s' = float32(T s) with
 * T = T16_host (float64, row-major, passed to the kernels by value); the correspondence of source point i is the
 * target point with the smallest (d2, index) among those with d2 = (dx*dx + dy*dy) + dz*dz (float32, unfused)
 * <= float32(r)^2, else -1.  out_correspondences int32[n_src] and out_d2 float32[n_src] (d2, 0 for none) may be
 * NULL; out_stats_dev double[2] (device) = {fitness = n_corr / n_src, inlier_rmse = sqrt(sum d2 / n_corr)}, both
 * 0 when n_corr = 0.  xyzi clouds (float4 per point); r finite and > 0 with float32(r)^2 finite (APC_ERR_BAD_ARG
 * otherwise).  Target points the grid cannot key raise APC_ERR_KEY_RANGE at apc_check; a transformed source
 * point the grid cannot key has no correspondence.  Every target point within r is found for coordinates below
 * 16384 r.  No host synchronisation. */
int apc_evaluate_registration(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev,
                              const float* tgt_xyzi, uint32_t n_tgt, const uint32_t* n_tgt_dev,
                              double max_correspondence_distance, const double* T16_host,
                              int32_t* out_correspondences, float* out_d2, double* out_stats_dev, void* stream);

/* icp(source, target, max_correspondence_distance, init, estimation, criteria) (Open3D
 * t::pipelines::registration::ICP, one scale; DoSingleScaleICPIterations).  Every iteration matches the ORIGINAL
 * source transformed by the T accumulated so far (as apc_evaluate_registration), computes fitness and rmse, and
 * estimates an update: APC_ICP_POINT_TO_POINT Kabsch (no scaling), APC_ICP_POINT_TO_PLANE one Gauss-Newton step
 * of sum ((s' - t) . n)^2 over the pose (alpha, beta, gamma, tx, ty, tz) -> Rz Ry Rx (PoseToTransformation), with
 * the 6x6 system solved by Cholesky; T = update T.  The loop stops after max_iteration iterations, when
 * |delta fitness| < relative_fitness and |delta rmse| < relative_rmse (never at the first iteration), at an
 * iteration without correspondences (APC_ICP_NO_CORRESPONDENCE; Open3D raises) or when the 6x6 system is not
 * positive definite (APC_ICP_DEGENERATE, no update).  Outputs (device): out_T16_dev double[16] (row-major),
 * out_stats_dev double[2] {fitness, inlier_rmse} and out_correspondences int32[n_src] (may be NULL) of the last
 * matching, out_info_dev int32[4] {iterations, converged, APC_ICP_* status, 0}.  max_iteration = 0 gives init,
 * 0, 0, all -1, 0 iterations.  tgt_normals float32[3 * n_tgt] (point-to-plane only).  init_T16_host is passed to
 * the kernels by value, and all max_iteration (match, solve) pairs are launched up front and return at once
 * after the loop has stopped: the call makes no host synchronisation and can be captured in a CUDA graph.
 * APC_ERR_BAD_ARG: NULL pointers, n_src or n_tgt above the context's max_points, r as in
 * apc_evaluate_registration, max_iteration < 0, an unknown method, point-to-plane without normals. */
int apc_icp(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev,
            const float* tgt_xyzi, const float* tgt_normals, uint32_t n_tgt, const uint32_t* n_tgt_dev,
            double max_correspondence_distance, const double* init_T16_host, int method, int max_iteration,
            double relative_fitness, double relative_rmse, double* out_T16_dev, double* out_stats_dev,
            int32_t* out_info_dev, int32_t* out_correspondences, void* stream);

/* icp(source, target, max_correspondence_distance, init, TransformationEstimationForGeneralizedICP(epsilon),
 * criteria) (Open3D t::pipelines::registration::ICP with TransformationEstimationForGeneralizedICP; the
 * covariances are those of t::geometry::PointCloud::EstimateCovariances).  Matching, metrics, the loop, its
 * statuses and outputs are those of apc_icp with APC_ICP_POINT_TO_PLANE; only the per-correspondence system
 * differs (Segal et al. 2009, plane-to-plane).  Every point's regularisation axis a is the eigenvector of the
 * smallest eigenvalue of its covariance (the solver of apc_estimate_normals; NaN when an entry is not finite), and
 * its regularised covariance I - (1 - epsilon) a a^T = U diag(1, 1, epsilon) U^T.  For s' matched to t:
 * W = (R C_s,reg R^T + C_t,reg)^-1 with R the rotation of the T accumulated so far, e = s' - t,
 * J = [-[s']x | I]; one Gauss-Newton step of sum e^T W e solves (sum J^T W J) x = -(sum J^T W e) by Cholesky
 * (APC_ICP_DEGENERATE when it is not positive definite or not finite).  An isotropic covariance has no defined
 * axis: the identity (neighbourhoods of fewer than 3 points) gives (0, 0, 1), a zero covariance the axis 0 and so
 * C_reg = I.  src_cov / tgt_cov float32[9 * n] (row-major 3x3 per point).  out_src_axes_dev / out_tgt_axes_dev
 * double[3 * n] (may be NULL) receive the axes used, 0 beyond the device count or when a cloud is empty.  The
 * axes are computed once per call (k_gicp_prep).  No host synchronisation; the call can be captured in a CUDA
 * graph.  APC_ERR_BAD_ARG: everything apc_icp rejects, NULL covariances, epsilon not finite or not > 0. */
int apc_icp_generalized(apc_ctx* ctx, const float* src_xyzi, const float* src_cov, uint32_t n_src, const uint32_t* n_src_dev,
                        const float* tgt_xyzi, const float* tgt_cov, uint32_t n_tgt, const uint32_t* n_tgt_dev,
                        double max_correspondence_distance, const double* init_T16_host, double epsilon, int max_iteration,
                        double relative_fitness, double relative_rmse, double* out_T16_dev, double* out_stats_dev,
                        int32_t* out_info_dev, int32_t* out_correspondences,
                        double* out_src_axes_dev, double* out_tgt_axes_dev, void* stream);

/* ---- (3c) FPFH features and feature matching (Open3D t.pipelines.registration) --------- */

/* compute_fpfh_feature(input, max_nn, radius) (Open3D t::pipelines::registration::ComputeFPFHFeature, hybrid
 * search).  Contract (oracle/features.py): the neighbourhood of estimate_normals' hybrid search (the max_nn nearest
 * of the points with d2 <= float32(radius)^2 by (d2, index), query included), m points; entry 0 is at d2 = 0 and is
 * skipped as Open3D skips it.  SPFH: the 3 x 11 bins of Open3D's pair features (float64) of the query with entries
 * 1..m-1, each count times 100 / (m - 1) (all zero for m <= 1); a pair whose feature is not finite adds to no bin.
 * FPFH: spfh[k] / d2_k summed over the entries with d2 > 0 in key order (float64), each group of 11 scaled by
 * 100 / its sum, plus spfh[i].  normals float32[3 * n_max]; out_features and out_spfh float32[33 * n_max] (out_spfh
 * may be NULL); out_neighbor_counts uint32[n_max] (m, may be NULL).  Points the grid cannot key get zeros and are
 * in no neighbourhood.  max_nn in 1..APC_MAX_NEIGHBORS and radius finite and > 0 (APC_ERR_BAD_ARG otherwise).
 * Two passes of the search; no host synchronisation, the call can be captured in a CUDA graph. */
int apc_compute_fpfh(apc_ctx* ctx, const float* xyzi, const float* normals, uint32_t n_max, const uint32_t* n_dev,
                     int max_nn, double radius, float* out_features, float* out_spfh,
                     uint32_t* out_neighbor_counts, void* stream);

/* compute_fpfh_feature(input, max_nn) (KNN search): the same, with the neighbourhood of apc_estimate_normals_knn
 * (the min(max_nn, n) points first in the order (d2, index), no distance bound). */
int apc_compute_fpfh_knn(apc_ctx* ctx, const float* xyzi, const float* normals, uint32_t n_max, const uint32_t* n_dev,
                         int max_nn, float* out_features, float* out_spfh, uint32_t* out_neighbor_counts,
                         void* stream);

/* correspondences_from_features(source_features, target_features, mutual_filter, mutual_consistency_ratio) (Open3D
 * t::pipelines::registration::CorrespondencesFromFeatures).  Rows of dim (1..64) float32 values, row-major.  The
 * match of source row i is the target row with the smallest (d2, index), d2 = sum_j (a_j - b_j)^2 in float32 in
 * increasing j, unfused; NaN and infinite d2 never win, and a row without a finite d2 has no match.
 * out_pairs int32[2 * n_src]: the first count rows hold (i, match) in ascending i, for every source row with a match
 * or, with mutual_filter, only those whose match's own match is i - unless that set has no more than
 * ratio * n_src pairs, when the unfiltered set is returned and fell_back is 1 (Open3D warns); the rows past the
 * unfiltered set's count are (-1, -1).  out_nearest
 * int32[n_src] (may be NULL): every row's match, -1 for none.  out_info_dev uint32[2] (device) = {count,
 * fell_back}.  Brute force, O(n_src * n_tgt * dim) per direction (the target-to-source search runs only with
 * mutual_filter).  APC_ERR_BAD_ARG: NULL pointers, dim outside 1..64, ratio not finite or < 0, more rows than
 * max_points.  No host synchronisation; the call can be captured in a CUDA graph. */
int apc_correspondences_from_features(apc_ctx* ctx, const float* src, uint32_t n_src, const uint32_t* n_src_dev,
                                      const float* tgt, uint32_t n_tgt, const uint32_t* n_tgt_dev, int dim,
                                      int mutual_filter, double ratio, int32_t* out_pairs, int32_t* out_nearest,
                                      uint32_t* out_info_dev, void* stream);

enum { APC_FGR_OK = 0, APC_FGR_TOO_FEW = 1, APC_FGR_DEGENERATE = 2 };

/* registration_fgr_based_on_feature_matching(source, target, source_feature, target_feature, option) (Open3D
 * pipelines::registration::FastGlobalRegistrationBasedOnFeatureMatching; Zhou, Park, Koltun 2016).  Contract
 * (oracle/fgr.py):
 *   pairs: the mutual set of apc_correspondences_from_features (every source row whose match's own match is itself,
 *     in ascending row), never the fallback;
 *   tuple test (tuple_test != 0): K pairs, trials t = 0 .. 100 K - 1; draw k of trial t is ((z >> 32) * K) >> 32
 *     with z = splitmix64(seed + (t << 32) + k); the tuple is accepted iff on each edge (0,1), (1,2), (2,0)
 *     li * tuple_scale < lj and lj < li / tuple_scale (l = sqrt((dx*dx + dy*dy) + dz*dz), float64, the source
 *     points' li, the target points' lj), and its three pairs are kept in draw order, in trial order, up to
 *     maximum_tuple_count tuples;
 *   normalisation: the means of all points of each cloud, D the largest centred norm; relative scale divides by D
 *     and starts with par = 1, use_absolute_scale keeps metres and starts with par = D;
 *   iteration_number Gauss-Newton steps of sum s |p - T q|^2, s = (par / (|r|^2 + par))^2, from T = I, with
 *     par /= division_factor before iterations 0, 4, 8, ... while par > maximum_correspondence_distance
 *     (decrease_mu); the 6x6 system is solved as point-to-plane ICP's (APC_FGR_DEGENERATE when it is not positive
 *     definite or not finite: the loop stops) and T = Rz Ry Rx update T;
 *   out_T16_dev double[16] (device, row-major): the source-to-target transform in metres, [R^T | mu_t - R^T mu_s -
 *     g R^T t] (g = D relative, 1 absolute); fewer than 10 pairs reaching the loop is APC_FGR_TOO_FEW and gives the
 *     identity, 0 iterations.
 * out_info_dev int32[6] (device) = {iterations, pairs in, pairs used, APC_FGR_* status, trials (the index of the
 * last trial examined + 1, 0 without the tuple test), pairs dropped}.  out_pairs_used int32[2 * cap] (may be NULL):
 * the pairs used, in order; cap = 3 * maximum_tuple_count with the tuple test, n_src without.  Features are rows of
 * dim float32 values as apc_correspondences_from_features takes them.  No host synchronisation; launch
 * configurations depend on the host sizes only, and the call can be captured in a CUDA graph.  APC_ERR_BAD_ARG:
 * NULL pointers, sizes above the context's max_points, dim outside 1..64, division_factor not finite or not > 1,
 * maximum_correspondence_distance not finite or not > 0, iteration_number < 0, tuple_scale outside (0, 1],
 * maximum_tuple_count outside 1..max_points. */
int apc_fgr_from_features(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev,
                          const float* tgt_xyzi, uint32_t n_tgt, const uint32_t* n_tgt_dev, const float* src_feat,
                          const float* tgt_feat, int dim, double division_factor, int use_absolute_scale,
                          int decrease_mu, double maximum_correspondence_distance, int iteration_number,
                          double tuple_scale, int maximum_tuple_count, int tuple_test, uint64_t seed,
                          double* out_T16_dev, int32_t* out_info_dev, int32_t* out_pairs_used, void* stream);

/* registration_fgr_based_on_correspondence(source, target, corres, option) (Open3D
 * FastGlobalRegistrationBasedOnCorrespondence): the normalisation, loop and outputs of apc_fgr_from_features on the
 * caller's pairs int32[2 * n_pairs] (source index, target index; the device count n_pairs_dev, may be NULL), with
 * no tuple test (trials = 0).  A pair with an index outside its cloud's count is never read: it is dropped and
 * counted.  out_pairs_used int32[2 * n_pairs] (may be NULL): the pairs kept, in order.  APC_ERR_BAD_ARG as
 * apc_fgr_from_features, and NULL pairs with n_pairs > 0. */
int apc_fgr(apc_ctx* ctx, const float* src_xyzi, uint32_t n_src, const uint32_t* n_src_dev, const float* tgt_xyzi,
            uint32_t n_tgt, const uint32_t* n_tgt_dev, const int32_t* pairs, uint32_t n_pairs,
            const uint32_t* n_pairs_dev, double division_factor, int use_absolute_scale, int decrease_mu,
            double maximum_correspondence_distance, int iteration_number, double* out_T16_dev, int32_t* out_info_dev,
            int32_t* out_pairs_used, void* stream);

/* ---- (4) RANSAC ground plane --------------------------------------------------------- */

/* segment_plane(distance_threshold, ransac_n, num_iterations, probability) (pp.py:533-543).
 * Hypotheses come from the counter-based generator seeded with `seed`, or from
 * `sample_table_dev` (int32[num_iterations*ransac_n], device) when non-NULL.
 * out_plane_dev double[8]: [0..3] least-squares refit on the final inliers (the returned
 * plane_model), [4..7] the winning hypothesis.  out_inlier_mask uint8[n_max] (1 = inlier).
 * out_info_dev uint32[4]: {best_iteration or 0xFFFFFFFF, n_inliers, 0, 0}. */
int apc_segment_plane(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
                      double distance_threshold, int ransac_n, int num_iterations,
                      double probability, uint64_t seed, const int32_t* sample_table_dev,
                      double* out_plane_dev, uint8_t* out_inlier_mask, uint32_t* out_info_dev,
                      void* stream);

/* Per-hypothesis tallies of the most recent apc_segment_plane / pipeline call on this context:
 * out_scores_dev uint64[2*num_iterations] = {inlier count, integer error sum} per iteration
 * (the quantities Open3D's fitness / inlier_rmse are derived from, pp.py:535-540).  Diagnostic
 * and test surface for the batched scoring kernel. */
int apc_segment_plane_scores(apc_ctx* ctx, uint64_t* out_scores_dev, uint32_t num_iterations,
                             void* stream);

/* ---- (1 inverse) repack to PointCloud2 bytes ------------------------------------------ */

typedef struct apc_out_field {
  int32_t offset;    /* byte offset in the packed output record (utils.py:152-163) */
  int32_t datatype;  /* APC_* */
  int32_t source;    /* 0 = zeros, 1 = x, 2 = y, 3 = z, 4 = intensity, 5 = extra attr array */
  int32_t attr_datatype; /* source 5: APC_* element type of attr_dev */
  const void* attr_dev;  /* source 5: device array [n_max] holding the attribute values */
} apc_out_field;

/* prepare_pointcloud + create_cloud (pp.py:576-625, pp.py:769): write the surviving points
 * into the packed output layout; fields without a source are zeros (pp.py:593). */
int apc_repack(apc_ctx* ctx, const float* xyzi, uint32_t n_max, const uint32_t* n_dev,
               const apc_out_field* fields, uint32_t n_fields, uint32_t point_step,
               uint8_t* out_bytes, void* stream);

/* ---- whole per-scan pipeline ----------------------------------------------------------- */

typedef struct apc_pipeline_cfg {
  apc_filter_cfg filter;
  float voxel_size;            /* <= 0 disables (pp.py:509) */
  int32_t stat_enable;         /* pp.py:514 */
  int32_t stat_nb_neighbors;   /* 1..APC_MAX_NEIGHBORS */
  double stat_std_ratio;
  int32_t radius_enable;       /* additive stage, TODO pp.py:37 */
  int32_t radius_nb_points;
  double radius_search_radius;
  int32_t ground_enable;       /* pp.py:533 */
  double ground_distance_threshold;
  int32_t ground_ransac_n;
  int32_t ground_num_iterations;
  double ground_probability;
  uint64_t ground_seed;
  int32_t normals_enable;      /* estimate_normals (pp.py:521-530, on by default pp.py:176): runs on the cloud that
                                  enters the ground stage; the normals travel through its selection (pp.py:542) */
  int32_t normals_max_nn;      /* 1..APC_MAX_NEIGHBORS */
  double normals_radius;
} apc_pipeline_cfg;

/* counters mirrored to the host after a pipeline run (index into out_counts_dev uint32[8]) */
enum { APC_CNT_INPUT = 0, APC_CNT_FILTERED = 1, APC_CNT_VOXELS = 2, APC_CNT_AFTER_STAT = 3,
       APC_CNT_AFTER_RADIUS = 4, APC_CNT_GROUND_INLIERS = 5, APC_CNT_OUTPUT = 6, APC_CNT_STATUS = 7 };

/* preprocess() (pp.py:447-544) end to end on the device: front end -> voxel -> statistical
 * -> radius -> RANSAC ground removal, no host synchronisation.  out_xyzi float4[sum
 * n_points]; out_counts_dev uint32[8] (APC_CNT_*); out_plane_dev double[8] (may be NULL). */
int apc_pipeline_run(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                     const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                     double* out_plane_dev, void* stream);

/* Index maps of one pipeline run, for carrying attributes the kernels do not touch (ring, time,
 * return_type, rgb, any extra field: pp.py:593-618 copy_fields) through the fused pipeline: gather
 * by src_idx, average per voxel with apc_voxel_mean_attr (p2v, voxel_counts), gather by out_row.
 * Every pointer is a device array of sum(n_points) elements and may be NULL.
 *   src_idx_dev       uint32: input index of every point that left the front end
 *   p2v_dev           int32:  voxel row of every such point (voxel stage enabled)
 *   voxel_counts_dev  uint32: points per voxel row
 *   out_row_dev       uint32: for every output point, its row in the cloud after the voxel stage
 *                             (after the front end when the voxel stage is off)
 *   normals_dev       float32[3*]: with cfg.normals_enable, the normal of every output point (required then) */
typedef struct apc_pipeline_maps {
  uint32_t* src_idx_dev;
  int32_t* p2v_dev;
  uint32_t* voxel_counts_dev;
  uint32_t* out_row_dev;
  float* normals_dev;           /* float32[3 * sum n_points]: normal of every OUTPUT point (cfg.normals_enable) */
} apc_pipeline_maps;
int apc_pipeline_run_maps(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                          const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                          double* out_plane_dev, const apc_pipeline_maps* maps, void* stream);

/* Multi-GPU exchange fused into the pipeline's final stage (batched replay configuration, SURVEY.md
 * section 8e: "NCCL all-gather of per-GPU outputs"): besides out_xyzi / out_counts_dev, the kernel
 * that writes the final cloud stores every surviving row - and k_pipeline_counts the 8 counters -
 * into up to APC_MAX_MIRRORS further buffers, typically the same slot of every peer GPU's slab,
 * mapped into this process (CUDA peer access / symmetric memory).  Only the real rows cross NVLink.
 * With xyzi_multicast != 0, xyzi_dev[0] is an NVLS multicast address covering all peers (one
 * multimem.st per row, replicated by the switch).  The final stage must be a selection
 * (statistical / radius outlier removal or ground removal): APC_ERR_BAD_ARG otherwise.  The rows are
 * complete on the peers when the launching stream has passed the launch (follow with a barrier
 * between the ranks before the peers read them). */
#define APC_MAX_MIRRORS 8
typedef struct apc_out_mirror {
  uint32_t n_xyzi;
  int32_t xyzi_multicast;
  float* xyzi_dev[APC_MAX_MIRRORS];        /* float4[sum n_points] each */
  uint32_t n_counts;
  uint32_t* counts_dev[APC_MAX_MIRRORS];   /* uint32[8] each (APC_CNT_*) */
} apc_out_mirror;
int apc_pipeline_run_mirrored(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                              const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                              double* out_plane_dev, const apc_out_mirror* mirror, void* stream);

/* Most general form: index maps / normals (maps may be NULL) and mirrored outputs (mirror may be NULL). */
int apc_pipeline_run_ex(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                        const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                        double* out_plane_dev, const apc_pipeline_maps* maps, const apc_out_mirror* mirror,
                        void* stream);

/* The same pipeline captured once into a CUDA graph (fixed buffers, sizes and config) and
 * replayed per scan: one launch per frame instead of ~25.  The per-frame input is whatever
 * the captured data_dev buffers hold when apc_graph_launch runs. */
typedef struct apc_graph apc_graph;
int apc_graph_capture_pipeline(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                               const apc_pipeline_cfg* cfg, float* out_xyzi,
                               uint32_t* out_counts_dev, double* out_plane_dev,
                               apc_graph** out_graph);
/* as apc_graph_capture_pipeline, with mirrored outputs (mirror may be NULL) */
int apc_graph_capture_pipeline_mirrored(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                        const apc_pipeline_cfg* cfg, float* out_xyzi,
                                        uint32_t* out_counts_dev, double* out_plane_dev,
                                        const apc_out_mirror* mirror, apc_graph** out_graph);
int apc_graph_capture_pipeline_ex(apc_ctx* ctx, const apc_cloud_desc* clouds, uint32_t n_clouds,
                                  const apc_pipeline_cfg* cfg, float* out_xyzi, uint32_t* out_counts_dev,
                                  double* out_plane_dev, const apc_pipeline_maps* maps,
                                  const apc_out_mirror* mirror, apc_graph** out_graph);
int apc_graph_launch(apc_ctx* ctx, apc_graph* graph, void* stream);
/* number of kernel nodes one replay of the graph launches (>= 0) or a negative apc_status */
int apc_graph_kernel_count(const apc_graph* graph);
int apc_graph_destroy(apc_graph* graph);

#ifdef __cplusplus
}
#endif
#endif /* APC_H_ */
