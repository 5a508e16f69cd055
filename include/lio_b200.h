/* lio_b200.h — C-ABI of liblio_b200.so: the B200-native (sm_100a) replacement of the compute hot
 * path of hyye/lio-mapping.  Plain pointers and sizes only; no C++/torch types.
 *
 * Each entry point names the reference interface (file:line under the reference tree) it stands
 * in for.  The reference has no FFI layer of its own: the seams are its C++ member functions and
 * the ceres::CostFunction contract (SURVEY.md §8b); INTEGRATION.md shows the shim a maintainer
 * adds at each seam.
 *
 * Conventions
 *   - point clouds are arrays of float4 {x, y, z, intensity}  (pcl::PointXYZI payload);
 *   - poses are double[7] {px,py,pz,qx,qy,qz,qw} (para_pose_ layout, Estimator.cc:2445-2452),
 *     float transforms are float[7] {qx,qy,qz,qw,px,py,pz} (Twist<float>);
 *   - every function returns LIO_OK (0) or a negative lio_status; lio_last_error() gives text;
 *   - "_host" variants take host buffers and copy in/out on the context's stream (synchronous
 *     on return); "_dev" variants take device pointers and are stream-ordered (asynchronous);
 *   - one thread drives a given handle at a time (same rule as the reference objects).
 */
#ifndef LIO_B200_H_
#define LIO_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef enum lio_status {
  LIO_OK = 0,
  LIO_ERR_CUDA = -1,        /* a CUDA runtime call failed (text in lio_last_error) */
  LIO_ERR_INVALID = -2,     /* bad argument */
  LIO_ERR_CAPACITY = -3,    /* input exceeds the capacity given at create time */
  LIO_ERR_NO_DEVICE = -4,   /* no CUDA device: there is NO CPU fallback in this library */
  LIO_ERR_NUMERIC = -5      /* solver breakdown (non-finite / not positive definite) */
} lio_status;

const char *lio_last_error(void);
int lio_version(void);
/* Number of usable CUDA devices (0 => every compute entry point returns LIO_ERR_NO_DEVICE). */
int lio_device_count(void);

/* ------------------------------------------------------------------------------------------
 * Stage A — lio::PointProcessor  (include/point_processor/PointProcessor.h:122-229,
 *           src/point_processor/PointProcessor.cc:185-783)
 * ---------------------------------------------------------------------------------------- */
typedef struct lio_pp_config {      /* PointProcessorConfig, PointProcessor.h:104-120 + ctor :76-80 */
  float lower_bound;                /* deg */
  float upper_bound;                /* deg */
  int num_rings;
  double scan_period;
  int num_scan_subregions;
  int num_curvature_regions;
  float surf_curv_th;
  int max_corner_sharp;
  int max_corner_less_sharp;
  int max_surf_flat;
  float less_flat_filter_size;
} lio_pp_config;

typedef struct lio_pp lio_pp;

/* Which output of the processor (names follow the reference members, PointProcessor.h:170-194). */
typedef enum lio_pp_cloud {
  LIO_PP_LASER_SCANS = 0,           /* laser_scans concatenated: intensity = ring + rel_time      */
  LIO_PP_CLOUD_IN_RINGS = 1,        /* cloud_in_rings_: intensity = int(I) + rel_time             */
  LIO_PP_CORNER_SHARP = 2,          /* corner_points_sharp_                                       */
  LIO_PP_CORNER_LESS_SHARP = 3,     /* corner_points_less_sharp_                                  */
  LIO_PP_SURF_FLAT = 4,             /* surface_points_flat_                                       */
  LIO_PP_SURF_LESS_FLAT = 5,        /* surface_points_less_flat_ (per-ring VoxelGrid(0.2) output) */
  LIO_PP_NUM_CLOUDS = 6
} lio_pp_cloud;

typedef enum lio_pp_index {         /* index sets into the ring-ordered cloud (parity / debug)   */
  LIO_PP_IDX_SHARP = 0,
  LIO_PP_IDX_LESS_SHARP = 1,
  LIO_PP_IDX_FLAT = 2,
  LIO_PP_IDX_ORIG = 3               /* input index of every ring-ordered point                   */
} lio_pp_index;

void lio_pp_default_config(lio_pp_config *cfg);                 /* PointProcessor.h:104-120 defaults */
/* PointProcessor::PointProcessor(lower, upper, rings) + SetupConfig  (PointProcessor.cc:74-95) */
int lio_pp_create(const lio_pp_config *cfg, int max_points, int device, void *cuda_stream, lio_pp **out);
int lio_pp_destroy(lio_pp *pp);
/* SetInputCloud + PointToRing + ExtractFeaturePoints (PointProcessor.cc:96-100,140-172,185-783);
 * xyzi: n x float4 on the HOST (pinned or pageable).  Synchronous. */
int lio_pp_process_host(lio_pp *pp, const float *xyzi, int n);
/* Same, input already on the device; asynchronous on the stream. */
int lio_pp_process_dev(lio_pp *pp, const float *xyzi_dev, int n);
/* The overload for sensors that deliver the ring index (lio::PointXYZIR, include/point_processor/point_types.h:37-52):
 * PointToRing(PointCloud<PointIR>) PointProcessor.cc:428-536 — ring id from `rings` (n x uint16), rel_time scaled by the
 * observed azimuth range end_ori_ - start_ori_ — followed by the shared ExtractFeaturePoints.  Synchronous.
 * Round-1 status: restated in the oracle and pinned by a CPU test; the device path was written after the round's GPU
 * budget was spent and is exercised by a non-strict xfail test until it has run on hardware. */
int lio_pp_process_host_ring(lio_pp *pp, const float *xyzi, const uint16_t *rings, int n);
/* Sizes of the six output clouds (synchronises the stream). */
int lio_pp_cloud_sizes(lio_pp *pp, int sizes[LIO_PP_NUM_CLOUDS]);
/* Copy one output cloud to the host (cap in points).  Returns the point count via *n. */
int lio_pp_download_cloud(lio_pp *pp, int which, float *out, int cap, int *n);
/* Device pointer of one output cloud (float4 array, valid until the next process call). */
int lio_pp_cloud_dev(lio_pp *pp, int which, const float **ptr);
int lio_pp_download_index(lio_pp *pp, int which, int32_t *out, int cap, int *n);
/* scan_ranges (PointProcessor.h:172): R pairs (start,end) exactly as the reference stores them. */
int lio_pp_download_scan_ranges(lio_pp *pp, int32_t *out_2R);
/* scan_ring_mask_ after the last subregion and PointLabel of every ring-ordered point. */
int lio_pp_download_mask_labels(lio_pp *pp, uint8_t *mask, int8_t *labels, int cap);
int lio_pp_start_ori(lio_pp *pp, float *start_ori);
/* Number of kernels launched by the last process call (bench bookkeeping). */
int lio_pp_last_launches(lio_pp *pp);

/* ------------------------------------------------------------------------------------------
 * Stage B primitives on explicit host arrays (parity entries; the estimator context below keeps
 * the same kernels device-resident).
 * ---------------------------------------------------------------------------------------- */
/* pcl::VoxelGrid<PointXYZI>::filter with setLeafSize(leaf,leaf,leaf)
 * (call sites Estimator.cc:679-687, :1518-1519; PointProcessor.cc:737-751).  out sized cap points. */
int lio_voxel_grid_host(const float *cloud, int n, float leaf, float *out, int cap, int *n_out, int device);
/* Estimator::CalculateFeatures (Estimator.cc:970-1097) with the kd-tree replaced by the voxel-hash
 * k-NN: map (K x float4) = local_surf_points_filtered_ptr_, surf (M x float4) = surf_stack_[idx],
 * tf7 = local_transform {qx,qy,qz,qw,px,py,pz}.  Outputs (sized M): pts4 = {point.xyz, score},
 * coef4 = coeffs, src = index of the originating surf point. */
int lio_calculate_features_host(const float *map, int K, const float *surf, int M, const float *tf7,
                                float min_match_sq_dis, float min_plane_dis, float *pts4, float *coef4, int32_t *src,
                                int *n_out, int device);
/* Point-to-line branch of Estimator::CalculateFeatures (Estimator.cc:1101-1227, compiled out in the reference build:
 * USE_CORNER is undefined, Estimator.h:55-56) == the live corner matching of PointMapping::OptimizeTransformTobeMapped
 * (PointMapping.cc:381-512): 5-NN in the corner map, centroid + 3x3 covariance eigen-decomposition, line accepted iff
 * lambda_3 > 3 lambda_2; a line is emitted as TWO consecutive half-weight plane-like features (normal_to_point and
 * normal_cross_point), which go through the same PivotPointPlaneFactor / fused stage-C kernel.
 * corner_map (K x float4) = local corner map, corner (M x float4) = corner stack of the frame; outputs sized 2*M. */
int lio_calculate_line_features_host(const float *corner_map, int K, const float *corner, int M, const float *tf7,
                                     float min_match_sq_dis, float *pts4, float *coef4, int32_t *src, int *n_out, int device);
/* TransformToEnd (Estimator.cc:62-103): in-place motion compensation of a sweep whose intensity carries
 * ring + relative time; tf7_es = transform_es {qx,qy,qz,qw,px,py,pz}; time_factor = 10 at the call site
 * (Estimator.cc:560).  float32, device sinf/acosf: parity tolerance 2e-6 relative to the range. */
int lio_transform_to_end_host(float *cloud, int n, const float *tf7_es, float time_factor, int device);
/* Estimator::CalculateLaserOdom (Estimator.cc:1099-1360): up to max_iter rounds of CalculateFeatures +
 * 6-DoF point-to-plane Gauss-Newton (float features, double normal equations, degeneracy projection at
 * the first round) refining tf7 in place.  Outputs are sized M * (keep_features ? max_iter : 1); *iters =
 * rounds executed before the delta_r / delta_t < 0.05 exit. */
int lio_laser_odom_host(const float *map, int K, const float *surf, int M, float *tf7, float min_match_sq_dis,
                        float min_plane_dis, int keep_features, int max_iter, float *pts4, float *coef4, int32_t *src,
                        int *n_out, int *iters, int device);

/* ---- lio::PointMapping with its rolling cube map resident in HBM (src/point_processor/PointMapping.cc) -------------------
 * The 21 x 21 x 11 cubes of 50 m (:77-82, :121-122) hold their corner / surf clouds as HBM segments; the cube directory
 * (pointer, count, capacity) is host state.  lio_pm_process_host is PointMapping::Process (:765-1052, imu_inited_ == false,
 * num_stack_frames_ == 1): associate the odometry increment (:753-756), bring the last features to the map frame and back
 * (:782-800, :1013-1016), re-centre the cube array (:809-931), select the cubes in the field of view (:944-1003), pull
 * laser_cloud_{corner,surf}_from_map_ (:1005-1011), VoxelGrid the stacks (:1016-1022), OptimizeTransformTobeMapped
 * (:325-753) and UpdateMapDatabase (:1112-1208: order-preserving insert + VoxelGrid of every valid cube).  The insert runs
 * on the device (stable sort by cube, scatter to the append positions); the host only grows segments from the per-cube add
 * counts.  The per-cube VoxelGrid workspace grows with the largest cube, so a cube above max_points is no error.
 * transform_sum7 = transform_sum_ from the odometry (qx qy qz qw px py pz); out: transform_tobe_mapped_ and
 * info3 = {iterations, corner_from_map size, surf_from_map size}.  Cube index = i + 21 j + 441 k (PointMapping.h:150-153). */
typedef struct lio_pm lio_pm;
int lio_pm_create(int max_points, float corner_filter_size, float surf_filter_size, float min_match_sq_dis, float min_plane_dis,
                  int max_iterations, int device, void *cuda_stream, lio_pm **out);
int lio_pm_destroy(lio_pm *pm);
int lio_pm_process_host(lio_pm *pm, const float *corner_last, int nc, const float *surf_last, int ns, const float transform_sum7[7],
                        float transform_tobe_mapped7[7], int info3[3]);
int lio_pm_map_centre(lio_pm *pm, int centre3[3]);                 /* laser_cloud_cen_length_ / width_ / height_ */
int lio_pm_cube_size(lio_pm *pm, int cube_index, int which, int *n);  /* which: 0 corner, 1 surf */
int lio_pm_cube_download(lio_pm *pm, int cube_index, int which, float *out_xyzi, int cap);

/* ---- lio::PointOdometry: scan-to-scan odometry of the pre-initialisation phase + the /compact_data pass-through ---------
 * (src/point_processor/PointOdometry.cc; include/point_processor/PointOdometry.h).  lio_po_create mirrors the constructor
 * PointOdometry(scan_period, io_ratio, num_max_iterations) (:66-86; defaults 0.1, 2, 25); the capacities bound the four feature
 * clouds and the full-resolution cloud of one sweep.  lio_po_process_host is Process() + PublishResults() (:294-766) for one
 * synchronised set of the five /laser_cloud_* topics (what HasNewData() :227-235 gates): the first sweep only becomes the
 * "last" clouds (:302-310); afterwards, while odometry is enabled, up to num_max_iterations rounds of corner (:338-441) and
 * surf (:443-549) matching against the last sweep + the damped 6 x 6 float Gauss-Newton (:551-664) refine transform_es_
 * (sweep end -> start), transform_sum_ accumulates its inverse (:667-669) and the less-sharp / less-flat clouds are de-skewed
 * to the sweep end (:673-674) before they replace the last clouds.  After lio_po_set_enable_odom(po, 0) - the /enable_odom
 * service the estimator calls once the IMU is initialised (:126-131) - the call is the pure pass-through: clouds swapped in,
 * transform_sum_ untouched.  Outputs (any may be NULL): transform_sum_ and transform_es_ as (qx qy qz qw px py pz),
 * info4 = {iterations executed, published (io_ratio gate :726), frame_count_, matches of the last round}.
 * lio_po_compact_data writes the /compact_data payload of the sweep just processed (:732-762, 3 + corner + surf + full points of
 * 4 floats; LIO_ERR_INVALID when the io_ratio gate did not publish it) - feed it to lio_xyzi_to_pcl32 for the PointCloud2 bytes or
 * to lio_compact_decode / lio_pm_process_host on the receiving side.  which: 0 last_corner_cloud_, 1 last_surf_cloud_,
 * 2 full_cloud_ (de-skewed when published while odometry is enabled, :728-730). */
typedef struct lio_po lio_po;
int lio_po_create(float scan_period, int io_ratio, int num_max_iterations, int max_feature_points, int max_full_points, int device,
                  void *cuda_stream, lio_po **out);
int lio_po_destroy(lio_po *po);
int lio_po_set_enable_odom(lio_po *po, int enable);
int lio_po_process_host(lio_po *po, const float *corner_points_sharp, int n_sharp, const float *corner_points_less_sharp, int n_less_sharp,
                        const float *surf_points_flat, int n_flat, const float *surf_points_less_flat, int n_less_flat,
                        const float *full_cloud, int n_full, float transform_sum7[7], float transform_es7[7], int info4[4]);
int lio_po_cloud_size(lio_po *po, int which, int *n);
int lio_po_cloud_download(lio_po *po, int which, float *out_xyzi, int cap);
int lio_po_compact_data(lio_po *po, float *out_xyzi, int cap_points, int *n_points);
int lio_po_last_launches(lio_po *po);
int lio_po_matches(lio_po *po, int kind, int32_t *out, int cap_queries);   /* test aid: indices of the last search, 2 (corner) / 3 (surf) per query */

/* ---- The pre-initialisation chain on the device: stage A -> PointOdometry -> PointMapping without host copies ------------
 * (the reference's processor -> odometry -> mapping node graph; Estimator::ProcessCompactData runs PointMapping::Process
 * before IMU initialisation, Estimator.cc:776-848).  Semantics and outputs equal the _host entries; errors follow them.
 * Streams: the entries enqueue on the context's own stream.  The caller orders them after the producer, by sharing one
 * stream or by recording an event, exactly as with lio_est_process_scan_dev.
 * Lifetime of inputs: the input clouds are only read during the call (each call ends with its read-back).  The odometry
 * context copies into its own buffers whatever must outlive the call - the less-sharp / less-flat clouds that become the
 * "last" clouds and the full cloud of the payload - so the producer (lio_pp) may process the next sweep right away. */
/* A cloud on the device whose point count lives in device memory (e.g. lio_pp_cloud_dev + lio_pp_cloud_count_dev).
 * The count is read on the device and clamped there to n_max; n_max above the context's capacity is LIO_ERR_CAPACITY
 * before anything is enqueued.  n_max == 0 stands for an empty cloud (xyzi / n_dev may then be NULL). */
typedef struct lio_dev_cloud { const float *xyzi; const int *n_dev; int n_max; } lio_dev_cloud;

/* PointOdometry::Process + PublishResults on device clouds, in the order sharp, less_sharp, flat, less_flat, full.
 * At most one host synchronisation: the final read-back of transform_es_, the iteration / match counts and the five counts. */
int lio_po_process_dev(lio_po *po, const lio_dev_cloud clouds[5], float transform_sum7[7], float transform_es7[7], int info4[4]);
/* last_corner_cloud_ / last_surf_cloud_ / full_cloud_ (which 0/1/2) with a device count; valid until the next lio_po_process_*. */
int lio_po_cloud_dev(lio_po *po, int which, const float **xyzi, const int **n_dev);
/* PointMapping::Process on device clouds (e.g. lio_po_cloud_dev 0 and 1); transform_sum7 on the host as lio_po_process_* returns it.
 * At most 4 host synchronisations in a call that grows no workspace (growing a cube segment is stream-ordered and costs none;
 * re-allocating the scan-to-map or re-filter workspace adds one). */
int lio_pm_process_dev(lio_pm *pm, const lio_dev_cloud *corner_last, const lio_dev_cloud *surf_last, const float transform_sum7[7],
                       float transform_tobe_mapped7[7], int info3[3]);
/* What the last process call cost the host: {kernel launches, host synchronisations (stream synchronisations and the device
 * synchronisation of a workspace re-allocation), bytes host->device, bytes device->host}. */
int lio_po_last_stats(lio_po *po, long long out[4]);
int lio_pm_last_stats(lio_pm *pm, long long out[4]);

/* PointMapping::OptimizeTransformTobeMapped (PointMapping.cc:325-753): scan-to-map 6-DoF float Gauss-Newton of
 * transform_tobe_mapped_ (tf7, in/out) against explicit corner / surf maps (laser_cloud_corner_from_map_ /
 * laser_cloud_surf_from_map_; the cube-map store that selects them is outside this operator).  Per round: corner matching
 * (:381-512, one feature per line), surf matching (:514-606, sign-normalised plane), skip when fewer than 50 matches
 * (:609-611), 6x6 normal equations + colPivHouseholderQr + first-round degeneracy projection + quaternion update (:613-715),
 * exit when delta_r < delta_r_abort (deg) and delta_t < delta_t_abort (cm).  Returns immediately (tf7 untouched) when
 * Kc <= 10 or Ks <= 100 (:327-329).  Optional outputs (sized Mc + Ms): the matches of the last executed round, corner
 * then surf; *iters = rounds executed.
 * variant 1 = MapBuilder::OptimizeMap (MapBuilder.cc:624-1014): the same loop with the rotation information matrix
 * J_r <- J_r R^-1 diag(5e-3, 5e-3, 1) (:905-911) and the left-multiplicative update rot = DeltaQ(x) * rot (:984-985). */
int lio_scan_to_map_host(const float *corner_map, int Kc, const float *surf_map, int Ks, const float *corner, int Mc,
                         const float *surf, int Ms, float *tf7, float min_match_sq_dis, float min_plane_dis, int max_iter,
                         double delta_r_abort, double delta_t_abort, int variant, float *pts4, float *coef4, int32_t *src,
                         int *n_out, int *iters, int device);

/* ------------------------------------------------------------------------------------------
 * fp64 factor operators — the ceres::CostFunction::Evaluate seam (SURVEY.md §8b).
 * Same contract as the reference: residuals always written, each jacobian pointer may be NULL,
 * blocks are row-major num_residuals x global_size (pose = 7 with a zero last column).
 * ---------------------------------------------------------------------------------------- */
/* PivotPointPlaneFactor::Evaluate (src/factor/PivotPointPlaneFactor.cc:43-137), one factor, host math. */
int lio_ppp_evaluate(const double point[3], const double coeff[4], const double pose_pivot[7], const double pose_i[7],
                     const double pose_ex[7], double *residual, double *J_pivot_1x7, double *J_i_1x7, double *J_ex_1x7);
/* The same operator for N factors sharing (pose_pivot, pose_i, pose_ex), evaluated on the GPU through
 * the rank-6 form used by the fused kernel: r_out[N], J_out[N][18] = [pivot(6) | i(6) | ex(6)] tangent columns. */
int lio_ppp_evaluate_batch_host(const float *pts4, const float *coef4, int n, const double pose_pivot[7],
                                const double pose_i[7], const double pose_ex[7], double *r_out, double *J_out, int device);

/* The fused stage-C reduction for ONE frame on explicit host arrays: with R9 = R_lpi (row-major), t3 = R_lpi^T P_lpi,
 * out32[0..27] = upper triangle (row-major) of S = sum_k rho'(r_k^2) [g_k;r_k][g_k;r_k]^T, out32[28] = sum_k rho(r_k^2)
 * (CauchyLoss(1.0), Estimator.cc:1664).  J^T J / J^T r of the frame's PivotPointPlaneFactors = M^T S M. */
int lio_asm_ppp_host(const float *pts4, const float *coef4, int n, const double R9[9], const double t3[3],
                     double out32[32], int device);

/* Streaming-rate measurement of the fused stage-C kernel on n synthetic features (32 B each) split over 8 frames;
 * CUDA events around each launch.  out = {avg ms / launch, min ms, algorithmic bytes / launch, launches}. */
int lio_asm_stream_bench(long long n_features, int iters, int device, double out[4]);
/* Test seam: number of TMA stages between folds of the per-thread product of (1 + r^2) into the cost accumulator of the
 * fused kernel (default 1024, i.e. one log per 2048 features and thread). */
int lio_asm_set_fold_chunks(int chunks);

/* Test seam of the device-resident solver: solves A x = b (A symmetric positive definite, n x n row-major, n <= 216) with
 * the tiled shared-memory Cholesky (fp64 tensor-core MMA trailing update) that the dogleg step of the device solver uses
 * in place of Ceres' dense factorisation (Estimator.cc:1911 DENSE_SCHUR).  *ok = 0 when a pivot is not positive.
 * prof (optional, 4 * ceil(n / 8) + 1 entries): SM cycles per 8-column panel {panel solve, own tile update, diagonal-tile
 * factorisation, trailing update incl. barrier} as seen by the warp that runs the serial chain, then the back substitution. */
int lio_dev_cholesky_solve_host(const double *A, const double *b, int n, double *x, int *ok, long long *prof, int device);

/* IntegrationBase (include/imu_processor/IntegrationBase.h:72-388) */
typedef struct lio_pim lio_pim;
int lio_pim_create(const double acc0[3], const double gyr0[3], const double ba[3], const double bg[3],
                   const double noise5[5] /* acc_n gyr_n acc_w gyr_w g_norm */, lio_pim **out);
int lio_pim_destroy(lio_pim *p);
int lio_pim_push_back(lio_pim *p, double dt, const double acc[3], const double gyr[3]);
/* state11 = delta_p(3) delta_q(xyzw) delta_v(3) sum_dt; jac225 / cov225 row-major 15x15 (may be NULL) */
int lio_pim_get(lio_pim *p, double *state11, double *jac225, double *cov225);
/* ImuFactor::Evaluate (include/factor/ImuFactor.h:53-167): J blocks 15x7, 15x9, 15x7, 15x9 row-major or NULL */
int lio_imu_factor_evaluate(lio_pim *p, const double pose_i[7], const double sb_i[9], const double pose_j[7],
                            const double sb_j[9], double *res15, double *J0, double *J1, double *J2, double *J3);

/* ------------------------------------------------------------------------------------------
 * Stages B+C+D — lio::Estimator in steady state (stage_flag_ == INITED)
 * (include/imu_processor/Estimator.h:110-170, src/imu_processor/Estimator.cc:338-427, 430-774,
 *  970-1646, 1648-2438, 2440-2666).
 * ---------------------------------------------------------------------------------------- */
typedef struct lio_est_config {   /* EstimatorConfig (Estimator.h:77-108), lidar/solver subset */
  int window_size;
  int opt_window_size;
  float min_match_sq_dis;
  float min_plane_dis;
  float surf_filter_size;
  int keep_features;
  int estimate_extrinsic;
  int opt_extrinsic;
  int imu_factor;
  int point_distance_factor;
  int prior_factor;
  int marginalization_factor;
  int enable_deskew;
  int cutoff_deskew;
  double acc_n, gyr_n, acc_w, gyr_w, g_norm;   /* IntegrationBaseConfig */
  int max_num_iterations;        /* ceres options.max_num_iterations, Estimator.cc:1916 */
  int odom_max_iterations;       /* PointMapping num_max_iterations_, PointMapping.h:171 */
  int max_frame_points;          /* capacity of one down-sampled frame cloud (surf_stack_ entry) */
  int max_scan_points;           /* capacity of the incoming laser_cloud_surf_last_ */
  int device_solver;             /* 1 (default): ImuFactor / marginalisation prior / PriorFactor evaluation, the dense normal
                                    equations, the tiled Cholesky and the dogleg controller all resident on the GPU (no host
                                    sync inside a solve; opt windows up to 13); 0: host controller around the fused kernel */
  int overlap_marginalization;   /* 1 (default): the Schur-complement / eigen algebra of scan k's marginalisation runs on a
                                    worker thread beside scan k+1's device front end (started at that call's entry, joined
                                    before its solve); 0: inline at the end of scan k, the reference's order.  Same result. */
  int solver_graph;              /* 1 (default): the device solver's launches of one solve are captured once as a CUDA graph
                                    and replayed per scan (single-GPU contexts); 0: plain stream launches.  Same result. */
} lio_est_config;

typedef struct lio_est lio_est;

void lio_est_default_config(lio_est_config *cfg);
int lio_est_create(const lio_est_config *cfg, int device, void *cuda_stream, lio_est **out);
int lio_est_destroy(lio_est *est);
/* transform_lb_ (Estimator.h:89): float {qx,qy,qz,qw,px,py,pz} */
int lio_est_set_extrinsic(lio_est *est, const float tf7[7]);
int lio_est_get_extrinsic(lio_est *est, float tf7[7]);
/* Warm start of window frame k in [0, W): state16 = P(3) Q(xyzw) V(3) Ba(3) Bg(3), the frame's own
 * down-sampled surf cloud (host), and the pre-integration ending at the frame (NULL for k = 0;
 * ownership of pim passes to the estimator). */
int lio_est_init_frame(lio_est *est, int k, const double state16[16], const float *surf_ds, int n, lio_pim *pim);
int lio_est_finish_init(lio_est *est, const double acc_last[3], const double gyr_last[3]);
/* Estimator::ProcessImu (Estimator.cc:338-427) */
int lio_est_process_imu(lio_est *est, double dt, const double acc[3], const double gyr[3], double stamp);
/* The same for n consecutive messages (dt[n], acc3[n][3], gyr3[n][3], stamp[n]) in one call: bag playback / batched drivers. */
int lio_est_process_imu_batch(lio_est *est, int n, const double *dt, const double *acc3, const double *gyr3, const double *stamp);
/* Estimator::ProcessLaserOdom, INITED branch (Estimator.cc:618-774): de-skew + VoxelGrid + SolveOptimization +
 * SlideWindow.  surf_last = laser_cloud_surf_last_ (surface_points_less_flat of the new sweep), HOST buffer.
 * Error behaviour: the window bookkeeping (pre-integration buffer, frame slots) advances before the device work, as in
 * the reference.  If a scan fails after that point (LIO_ERR_CAPACITY: down-sampled scan > max_frame_points, local map or
 * feature buffers full, voxel index overflow; LIO_ERR_NUMERIC; LIO_ERR_CUDA) the context is POISONED: every later
 * lio_est_process_scan_* call returns LIO_ERR_INVALID until the context is destroyed and re-created. */
int lio_est_process_scan_host(lio_est *est, const float *surf_last, int n);
/* ---- The same scan, phase by phase - for callers that keep the reference's control flow (Estimator::ProcessLaserOdom ->
 * SolveOptimization, Estimator.cc:618-774, 1648-2438) and only swap the heavy parts:
 *
 *   lio_est_open_scan_host / _dev   push the sweep (TransformToEnd :62-103, VoxelGrid :678-693), BuildLocalMap (:1361-1646:
 *                                   local map, k-NN + plane fit of every window frame, CalculateLaserOdom), VectorToDouble
 *                                   (:2440-2478).  The window stays "open" until lio_est_close_scan.
 *   lio_est_get_parameters          the ceres parameter blocks para_pose_ (O + 1 x 7: px py pz qx qy qz qw), para_speed_bias_
 *                                   (O + 1 x 9: v ba bg), para_ex_pose_ (7) of the open window (Estimator.h:282-284)
 *   lio_est_assemble                what ceres::Problem would evaluate at the given blocks (NULL = the estimator's own): the
 *                                   normal equations H = J^T J (n x n row-major), g = J^T r and the cost 1/2 sum rho, over
 *                                   every residual block added at :1747-1904 (ImuFactors, PivotPointPlaneFactors with
 *                                   CauchyLoss, MarginalizationFactor, PriorFactor).  n = 15 (O + 1) + 6, or 6 less while the
 *                                   extrinsic block is constant.  No gates, no step; nothing of the estimator changes.
 *   lio_est_solve                   ceres::Solve (:1989-1990) from the given blocks (in/out; NULL = the estimator's own) with
 *                                   at most max_iter iterations (<= 22 with the device solver); gates :1924-1985 included.
 *                                   summary[8] = iterations, successful steps, termination (0 no convergence / 1 convergence /
 *                                   2 failure), initial cost, final cost, evaluations, convergence_flag, extrinsic held constant.
 *   lio_est_close_scan              DoubleToVector (:2479-2568) from the given blocks (NULL = the estimator's own),
 *                                   marginalisation of the oldest frame (:2040-2275), SlideWindow (:2570-2666).
 *
 * lio_est_process_scan_* == open + solve(max_num_iterations) + close.  Errors poison the context as described above;
 * LIO_ERR_INVALID when the calls come out of order. */
int lio_est_open_scan_host(lio_est *est, const float *surf_last, int n);
int lio_est_open_scan_dev(lio_est *est, const float *surf_last_dev, const int *n_dev, int n_max);
int lio_est_get_parameters(lio_est *est, double *pose, double *speed_bias, double *ex);
int lio_est_assemble(lio_est *est, const double *pose, const double *speed_bias, const double *ex, double *H, double *g,
                     double *cost, int *n);
int lio_est_solve(lio_est *est, double *pose, double *speed_bias, double *ex, int max_iter, double summary[8]);
int lio_est_close_scan(lio_est *est, const double *pose, const double *speed_bias, const double *ex);
/* Optional: announce that the next sweep has arrived (call before stage A / lio_pp_process_*).  Starts the background
 * marginalisation algebra of the previous scan now instead of at the lio_est_process_scan_* entry, so it also overlaps
 * the feature extraction of the new sweep.  No effect with overlap_marginalization = 0. */
int lio_est_begin_scan(lio_est *est);
/* Same with the cloud already on the device (e.g. lio_pp_cloud_dev(LIO_PP_SURF_LESS_FLAT)); n is read
 * from *n_dev on the device and clamped there to n_max (n_max itself is clamped to max_scan_points). */
int lio_est_process_scan_dev(lio_est *est, const float *surf_last_dev, const int *n_dev, int n_max);
/* Device pointer to the point count of one stage-A output cloud, to chain stage A into the estimator. */
int lio_pp_cloud_count_dev(lio_pp *pp, int which, const int **n_dev);
/* window states: (W+1) x 16 doubles (layout of state16) */
int lio_est_get_states(lio_est *est, double *out);
/* summary[32]: see lio_mapping_b200/estimator.py SUMMARY_KEYS */
int lio_est_summary(lio_est *est, double *out32);
int lio_est_feature_count(lio_est *est, int frame, int *n);
int lio_est_get_features(lio_est *est, int frame, float *pts4, float *coef4, int32_t *src, int cap);
int lio_est_map_size(lio_est *est, int *n);
int lio_est_get_map(lio_est *est, float *out, int cap);
int lio_est_frame_size(lio_est *est, int frame, int *n);
int lio_est_get_frame(lio_est *est, int frame, float *out, int cap);
int lio_est_get_local_transform(lio_est *est, int frame, float tf7[7]);
/* Marginalisation prior kept for the next solve, as normal-equation terms over the kept blocks in
 * canonical order [pose_0,sb_0,...,pose_{O-1},sb_{O-1},ex] (tangent, 15*O+6): Hp = J^T J, bp = J^T r0. */
int lio_est_prior_dim(lio_est *est, int *n);
int lio_est_get_prior(lio_est *est, double *Hp, double *bp);
/* Normal equations at the INITIAL point of the last solve (after the convergence gates; tangent order
 * [pose_0,sb_0,...,pose_O,sb_O,ex], n = 15*(O+1)+6): H n x n row-major, g n, cost. */
int lio_est_last_normal_equations(lio_est *est, double *H, double *g, double *cost, int *n);
/* Kernels launched by the last process_scan call. */
int lio_est_last_launches(lio_est *est);
/* Text of the last failed scan-level call on THIS context (lio_last_error() is per calling thread; a process that drives
 * several estimators from one thread reads the per-handle copy). */
const char *lio_est_last_error(lio_est *est);
/* Diagnostic: the device-side timeline of the last solve, stamped by the kernels themselves.  out[24][16]:
 * rows 0..11 = evaluations: [0] / [11] %globaltimer (ns) at k_step entry / exit, [1..10] SM clock at its phase boundaries (entry,
 * verdict, lidar blocks, gradient, H tiles, Cauchy scale, tiles ready, Cholesky + solve, dogleg, exit), [12] / [13] %globaltimer when
 * the first k_factors CTA starts / the last one ends, [14] when the last k_hpart CTA ends;
 * row 12 = launch counters of asm_ppp, row 13 / 14 = %globaltimer when its first CTA starts / its tail ends, one column per
 * evaluation; row 16 = SM clock inside the lidar block expansion of evaluation 2 (entry, operands staged, S M, M^T (S M)).
 * Followed by 4 * 28 + 4 entries: the per-panel profile of evaluation 1's Cholesky in the layout of
 * lio_dev_cholesky_solve_host's prof (column 1 = %globaltimer at the start of the panel's diagonal tile), and after the back
 * substitution cycles four %globaltimer stamps (entry, loop start, loop end, exit).  cap >= 24 * 16 + 116.  Zeros when the host
 * controller is in use.  `LIO_BENCH_TRACE=1 python bench.py` prints it. */
int lio_est_solver_trace(lio_est *est, long long *out, int cap);
/* CUDA-event timing of the fused residual+Jacobian kernel accumulated since the last reset (events recorded
 * on the estimator's stream around every launch): out[0..3] = {sum ms, launches, features processed, bytes/feature};
 * out[4..7] = the same for the frame-batched k-NN + plane-fit launch of BuildLocalMap {sum ms, launches, queries,
 * algorithmic bytes/query = 128}. */
int lio_est_kernel_profile(lio_est *est, double out[8], int reset);
/* Multi-GPU (SURVEY.md §8e): frames i with (i-1) % world == rank are matched/assembled locally; the
 * callback must sum-allreduce `count` doubles in place on the DEVICE buffer `buf` across ranks
 * (e.g. ncclAllReduce / torch.distributed.all_reduce on the estimator's stream). */
typedef int (*lio_allreduce_fn)(void *user, double *buf_dev, int count);
int lio_est_set_shard(lio_est *est, int rank, int world, lio_allreduce_fn fn, void *user);
/* Fused exchange over peer memory (preferred on one NVLink / NVSwitch node; `fn` may then be NULL in set_shard).  Every
 * rank owns one small device exchange buffer; once each rank knows the device pointers of all of them (its own, and the
 * peers' opened through CUDA IPC with lio_ipc_export / lio_ipc_open, or raw pointers when the contexts share a process),
 * the last CTA of the fused stage-C kernel stores the S blocks of the frames it owns straight into EVERY rank's buffer
 * (P2P stores) and publishes an epoch with system-scope release; a one-warp kernel on each rank acquires the epochs of
 * all ranks before the 2.5 kB result goes to the host.  No collective call, no extra pass over the data. */
int lio_est_exchange_buffer(lio_est *est, void **dev_ptr, size_t *bytes);
int lio_est_set_peers(lio_est *est, int world, void *const *peer_ptrs /* [world], entry [rank] ignored */);
/* Per-scan feature exchange (preferred on one NVLink / NVSwitch node).  After lio_est_set_shard(rank, world, NULL, NULL) each rank
 * still matches only the frames it owns, but copies their features (xyz + score, coefficients, count) into the same place of every
 * peer's feature slab with P2P stores and publishes the scan's epoch; once all epochs have arrived every rank holds ALL frames'
 * features and runs the complete solve exactly like a single-GPU context (one rendezvous per scan instead of one per evaluation, the
 * solve graph stays in use).  lio_est_feature_slab returns this context's slab (all feature buffers of both scan parities, the
 * counts and the epoch flags are ONE allocation: export it with lio_ipc_export); lio_est_set_feature_peers takes every rank's slab
 * as mapped in this process (entry [rank] ignored).  Replaces a previous lio_est_set_peers; LIO_ERR_INVALID inside an open scan. */
int lio_est_feature_slab(lio_est *est, void **dev_ptr, size_t *bytes);
int lio_est_set_feature_peers(lio_est *est, int world, void *const *peer_slabs /* [world], entry [rank] ignored */);
int lio_ipc_export(const void *dev_ptr, unsigned char handle[64]);      /* cudaIpcGetMemHandle */
int lio_ipc_open(const unsigned char handle[64], void **dev_ptr);       /* cudaIpcOpenMemHandle, lazy peer access */
int lio_ipc_close(void *dev_ptr);
/* Owner rank of window frame pivot+frame_rel (frame_rel = 1..O) under `world` ranks: (frame_rel-1) % world. */
int lio_est_frame_owner(int frame_rel, int world);

/* ------------------------------------------------------------------------------------------
 * /compact_data wire format (host only; no device needed).  Encoder PointOdometry.cc:732-762, decoder
 * PointMapping::CompactDataHandler PointMapping.cc:171-238: point 0 = transform_sum_.pos, point 1 = quaternion
 * (x, y, z | intensity = w), point 2 = (corner_size, surf_size, full_size) as floats, then corner || surf || full.
 * Clouds are packed (x, y, z, intensity) float4; tf7 = {qx,qy,qz,qw,px,py,pz}.
 * ---------------------------------------------------------------------------------------- */
/* out_xyzi sized cap_points float4; *n_points = 3 + nc + ns + nf.  LIO_ERR_CAPACITY when a size is >= 2^24 (not exact as
 * a float) or the output is too small. */
int lio_compact_encode(const float tf7[7], const float *corner, int nc, const float *surf, int ns, const float *full, int nf,
                       float *out_xyzi, int cap_points, int *n_points);
/* Header check of the decoder (:180-195): LIO_ERR_INVALID when n_points < 4 or 3 + sizes != n_points. */
int lio_compact_sizes(const float *xyzi, int n_points, int sizes[3]);
/* corner / surf / full sized by lio_compact_sizes. */
int lio_compact_decode(const float *xyzi, int n_points, float tf7[7], float *corner, float *surf, float *full);
/* packed float4 <-> the 32-byte pcl::PointXYZI records a sensor_msgs/PointCloud2 of this type carries
 * (x, y, z at 0/4/8, data[3] = 1.0f, intensity at 16). */
int lio_xyzi_to_pcl32(const float *xyzi, int n, uint8_t *out32);
int lio_pcl32_to_xyzi(const uint8_t *in32, int n, float *xyzi);

/* ------------------------------------------------------------------------------------------
 * Dense fp64 kernels of the host shell (host only; test seams).
 * ---------------------------------------------------------------------------------------- */
/* Lower Cholesky A = L L^T (blocked, the factorisation behind every dogleg step: Ceres DENSE_SCHUR at n <= 261,
 * Estimator.cc:1909-1921) and the solve A x = b.  A n x n row-major symmetric (lower triangle read); L_out optional
 * (n x n, upper triangle zeroed).  LIO_ERR_NUMERIC when A is not positive definite. */
int lio_host_cholesky_solve(int n, const double *A, const double *b, double *L_out, double *x);
/* Symmetric eigen-decomposition (Eigen::SelfAdjointEigenSolver call sites MarginalizationFactor.cc:276, :293):
 * ascending eigenvalues, eigenvectors in the COLUMNS of evecs (n x n row-major).  threads > 1 applies the QL rotations
 * on disjoint row ranges in parallel (bit-identical result). */
int lio_host_sym_eigen(int n, const double *A, double *evals, double *evecs, int threads);
/* The trust-region / traditional-dogleg controller that stands in for ceres::Solve (options of Estimator.cc:1909-1921,
 * Ceres 1.14 defaults otherwise) on a toy nonlinear least-squares problem assembled on the host:
 * r_k = a_k . x + amp sin(b_k . x) - y_k  (A, B: m x n row-major), optional CauchyLoss(1.0) with the Ceres corrector.
 * x in/out; summary[8] = {iterations, successful steps, termination (0 no convergence, 1 convergence, 2 failure),
 * initial cost, final cost, evaluations}. */
int lio_host_dogleg_toy(int n, int m, const double *A, const double *B, const double *y, double amp, int use_cauchy, double *x,
                        int max_iter, double *summary);

#ifdef __cplusplus
}
#endif
#endif /* LIO_B200_H_ */
