/* b200reg.h — C-ABI of the B200-native scan-registration engine.
 *
 * Drop-in boundary: the pcl::Registration<PointXYZI,PointXYZI> surface that lidarslam_ros2's nodes hold
 * (scanmatcher/include/scanmatcher/scanmatcher_component.h:93, graph_based_slam/include/graph_based_slam/
 * graph_based_slam_component.h:106) and through which they drive pclomp::NormalDistributionsTransform and
 * pclomp::GeneralizedIterativeClosestPoint. Every entry point below names the reference interface it
 * replaces (paths relative to the reference root; "ndt.h" = Thirdparty/ndt_omp_ros2/include/pclomp/ndt_omp.h,
 * "gicp.h" = .../gicp_omp.h, "sm.cpp" = scanmatcher/src/scanmatcher_component.cpp,
 * "gbs.cpp" = graph_based_slam/src/graph_based_slam_component.cpp).
 *
 * Conventions
 *  - plain C, opaque handle, no exceptions; every call returns 0 (B200REG_OK) or a negative error code,
 *    b200reg_last_error() gives the text. PCL-style soft failure: an empty cloud is rejected and ignored.
 *  - 4x4 matrices are 16 floats COLUMN-MAJOR — exactly Eigen::Matrix4f::data().
 *  - clouds are (const float* base, size_t n, size_t stride_bytes) with x,y,z at byte offsets 0,4,8 of every
 *    point: pass pcl::PointCloud<PointXYZI>::points.data() with stride 32 (PointXYZ: 16).
 *  - the library copies what it needs to the GPU inside set_input_*; caller memory (host or device) may be freed or
 *    overwritten on return. A device buffer must be complete (its producer stream synchronised) at the call.
 *  - one handle = one CUDA stream + its device buffers; a handle is used from one host thread at a time,
 *    different handles may be used concurrently from different threads (lidarslam/src/lidarslam.cpp:12-17).
 *  - there is NO CPU fallback: without a CUDA device b200reg_create fails with B200REG_ERR_CUDA.
 */
#ifndef B200REG_H_
#define B200REG_H_

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct b200reg_engine* b200reg_t;

enum b200reg_kind { B200REG_NDT = 0, B200REG_GICP = 1 };

/* pclomp::NeighborSearchMethod (ndt.h:52-57), same numeric order */
enum b200reg_search { B200REG_KDTREE = 0, B200REG_DIRECT26 = 1, B200REG_DIRECT7 = 2, B200REG_DIRECT1 = 3 };

enum b200reg_status {
  B200REG_OK = 0,
  B200REG_ERR_ARG = -1,       /* bad argument / wrong engine kind                                    */
  B200REG_ERR_NO_TARGET = -2, /* align/fitness without setInputTarget (PCL: initCompute() fails)      */
  B200REG_ERR_NO_SOURCE = -3, /* align without setInputSource                                          */
  B200REG_ERR_CUDA = -4,      /* CUDA runtime error, or no device                                      */
  B200REG_ERR_TIMEOUT = -5,   /* device-side watchdog fired inside the persistent solver               */
  B200REG_ERR_GRID = -6       /* voxel grid would overflow int32 (voxel_grid_covariance_omp_impl.hpp:79) */
};

/* ---- lifetime --------------------------------------------------------------------------------------- */
/* replaces `new pclomp::NormalDistributionsTransform<...>()` / `new pclomp::GeneralizedIterativeClosestPoint
 * <...>()` (sm.cpp:105-106,116-117; gbs.cpp:64-65,74-75). Defaults are the reference constructors'
 * (ndt_omp_impl.hpp:47-76: resolution 1.0, step 0.1, outlier 0.55, eps 0.1, 35 iterations, DIRECT7;
 * gicp.h:108-128: k=20, gicp_eps 1e-3, rot_eps 2e-3, 20 inner, 200 outer, eps 5e-4, corr-dist 5). */
int b200reg_create(int kind, int device, b200reg_t* out);
int b200reg_destroy(b200reg_t h);
const char* b200reg_last_error(b200reg_t h);

/* ---- pcl::Registration setters (sm.cpp:109,118-119; gbs.cpp:66-69,76-81) ---------------------------- */
int b200reg_set_transformation_epsilon(b200reg_t h, double eps);      /* setTransformationEpsilon      */
int b200reg_set_maximum_iterations(b200reg_t h, int n);               /* setMaximumIterations          */
int b200reg_set_max_correspondence_distance(b200reg_t h, double d);   /* setMaxCorrespondenceDistance  */
int b200reg_set_euclidean_fitness_epsilon(b200reg_t h, double eps);   /* stored; unused by both engines */
int b200reg_set_ransac_iterations(b200reg_t h, int n);                /* stored; unused by both engines */

/* ---- pclomp::NormalDistributionsTransform setters / getters (ndt.h:110-233) ------------------------- */
int b200reg_ndt_set_resolution(b200reg_t h, float resolution);        /* ndt.h:127-137                 */
int b200reg_ndt_set_step_size(b200reg_t h, double step);              /* ndt.h:162-166                 */
int b200reg_ndt_set_outlier_ratio(b200reg_t h, double ratio);         /* ndt.h:180-184 (setOulierRatio) */
int b200reg_ndt_set_neighborhood_search_method(b200reg_t h, int m);   /* ndt.h:186-188                 */
int b200reg_ndt_set_num_threads(b200reg_t h, int n);                  /* ndt.h:110-112; accepted, no-op */
int b200reg_ndt_get_transformation_probability(b200reg_t h, double* out); /* ndt.h:193-197             */
int b200reg_ndt_get_final_num_iteration(b200reg_t h, int* out);       /* ndt.h:202-206                 */
/* ndt.h:233 calculateScore(cloud): cloud is an already-transformed source */
int b200reg_ndt_calculate_score(b200reg_t h, const float* base, size_t n, size_t stride_bytes, double* out);

/* ---- pclomp::GeneralizedIterativeClosestPoint setters (gicp.h:156-252) ------------------------------- */
int b200reg_gicp_set_rotation_epsilon(b200reg_t h, double eps);       /* setRotationEpsilon            */
int b200reg_gicp_set_correspondence_randomness(b200reg_t h, int k);   /* setCorrespondenceRandomness   */
int b200reg_gicp_set_maximum_optimizer_iterations(b200reg_t h, int n);/* setMaximumOptimizerIterations */
int b200reg_gicp_set_epsilon(b200reg_t h, double gicp_epsilon);       /* gicp_epsilon_ (gicp.h:110)    */

/* ---- clouds ----------------------------------------------------------------------------------------- */
/* setInputTarget (ndt.h:117-122 → init() ndt.h:271-278 → VoxelGridCovariance::filter; gicp.h:156-170):
 * uploads the cloud and, for NDT, builds the voxel map (mean / regularised inverse covariance) on the GPU. */
int b200reg_set_input_target(b200reg_t h, const float* base, size_t n, size_t stride_bytes);
/* setInputSource (pcl::Registration; gicp.h:133-149) */
int b200reg_set_input_source(b200reg_t h, const float* base, size_t n, size_t stride_bytes);
/* Same, from a DEVICE buffer of n float4 (x,y,z,ignored) already resident in HBM on the handle's device. */
int b200reg_set_input_target_device(b200reg_t h, const void* dev_float4, size_t n);
int b200reg_set_input_source_device(b200reg_t h, const void* dev_float4, size_t n);

/* ---- align ------------------------------------------------------------------------------------------ */
/* pcl::Registration::align(output, guess) (sm.cpp:353, gbs.cpp:230, apps/align.cpp:27,33) →
 * computeTransformation (ndt_omp_impl.hpp:80-171 / gicp_omp_impl.hpp:369-515). guess == NULL means identity.
 * Synchronous: on return final_out (may be NULL) holds getFinalTransformation(). */
int b200reg_align(b200reg_t h, const float* guess, float* final_out);
int b200reg_get_final_transformation(b200reg_t h, float* out16);      /* sm.cpp:356; gbs.cpp:244,253   */
int b200reg_has_converged(b200reg_t h, int* out);                     /* sm.cpp:375                    */
/* getFitnessScore(max_range) (gbs.cpp:231, sm.cpp:376): mean squared 1-NN distance of the aligned source
 * to the target, over points with d^2 <= max_range; DBL_MAX if none. */
int b200reg_get_fitness_score(b200reg_t h, double max_range, double* out);
/* the `output` cloud of align(): source transformed by the final transformation; out has n_source points */
int b200reg_get_aligned(b200reg_t h, float* out, size_t stride_bytes);

/* align() on `count` independent handles (each with its own target and source already set), one after the other — a
 * convenience loop: every solve is a persistent kernel that owns all SMs, so solves never overlap; what overlaps between
 * pairs is done by b200reg_ndt_sweep below (uploads, map builds, fitness passes). guesses may be NULL (identity);
 * finals = 16*count floats. Results are those of b200reg_align on each handle. */
int b200reg_align_batch(b200reg_t* handles, int count, const float* guesses, float* finals);

/* K independent NDT registrations against the handle's CURRENT target in ONE persistent launch — repeated
 * align() calls of apps/align.cpp:32-36 ("10times"), multi-hypothesis initial guesses, or the candidate scans of a
 * loop-closure sweep sharing one map. Up to three registrations are in flight inside the kernel: while one registration's
 * Newton step (fixed-order reduction, 6x6 solve, next pose) runs on its controller SM, the evaluator SMs compute the
 * other registrations' derivatives, so the sequential part of ndt_omp_impl.hpp:121-166 no longer idles the GPU.
 * Every result is BITWISE the result b200reg_align gives for the same (source, guess).
 * guesses: 16*count floats column-major, or NULL (identity). results[k].status is B200REG_OK or an error code.
 * After the call the handle's getters (final transformation, converged, ...) describe the LAST registration;
 * b200reg_get_stats reports evaluations / hits_total / solve_ms summed over the batch. */
typedef struct b200reg_batch_result {
  float final_T[16];         /* getFinalTransformation(), column-major                                     */
  double trans_probability;  /* getTransformationProbability()                                              */
  int converged, iterations, evaluations, status;
  long long hits_total;
} b200reg_batch_result;
/* sources in HOST memory: (base, n, stride) clouds as in b200reg_set_input_source, one bulk copy + unpack each, no
 * synchronisation in between */
int b200reg_ndt_align_batch(b200reg_t h, int count, const float* const* sources, const size_t* n_points,
                            size_t stride_bytes, const float* guesses, b200reg_batch_result* results);
/* sources already in HBM as float4 (x, y, z, ignored) on the handle's device; read in place (no copy) — they must
 * be complete when the call is made and stay untouched until it returns */
int b200reg_ndt_align_batch_device(b200reg_t h, int count, const void* const* dev_sources, const size_t* n_points,
                                   const float* guesses, b200reg_batch_result* results);
/* The loop-closure candidate sweep on one GPU (generalises gbs.cpp:187-233 from the arg-min candidate to all of them):
 * `count` independent (source, target) pairs, each through the node's own sequence setInputTarget (gbs.cpp:227) ->
 * setInputSource (:181) -> align (:230) -> getFitnessScore (:231) with the handle's parameters. Two internal engines
 * (stream + buffers each) driven by two host threads take the pairs in turn, so that the upload and voxel-map build of
 * one pair overlap the solve and fitness pass of the other. Results equal those of the sequential calls.
 * guesses: 16*count floats column-major or NULL (identity). Sharding pairs across GPUs is the caller's (one process per
 * GPU, include/b200comm.h for the all-gather of the result rows). */
typedef struct b200reg_sweep_result {
  float final_T[16];         /* column-major */
  double fitness;            /* getFitnessScore(fitness_max_range) */
  double trans_probability;
  int converged, iterations, status, pad;
} b200reg_sweep_result;
int b200reg_ndt_sweep(b200reg_t h, int count, const float* const* sources, const size_t* n_src,
                      const float* const* targets, const size_t* n_tgt, size_t stride_bytes, const float* guesses,
                      double fitness_max_range, b200reg_sweep_result* results);
/* Multi-GPU form of the batch calls (SURVEY.md section 8e: the shards are independent, the only exchange is the 4x4 poses):
 * attach a pose board (include/b200comm.h, b200comm_board_create) and every b200reg_ndt_align_batch[_device] call on this
 * handle also publishes its poses to all ranks FROM INSIDE the solver kernel — peer-memory stores over NVLink as each
 * registration converges — and returns when all ranks' poses of the call have arrived here. Such calls are collective:
 * all ranks of the board make the same sequence of them (counts may differ; 1 <= count <= the board's max_rows).
 * b200reg_ndt_gathered_poses then copies them out: poses[(r * max_rows + k) * 16 ..] = column-major pose of rank r's
 * registration k, counts[r] = how many rank r registered. board = NULL detaches. */
struct b200comm_board;
int b200reg_ndt_attach_pose_board(b200reg_t h, struct b200comm_board* board);
int b200reg_ndt_gathered_poses(b200reg_t h, float* poses, int* counts, int max_rows);
/* registrations in flight per batch launch (1..3; default 3; larger values act as 3). Developer / measurement switch.
 * Any handle kind: b200reg_gicp_align_batch[_device] honours it too. */
int b200reg_ndt_set_batch_slots(b200reg_t h, int slots);

/* K independent GICP registrations against the handle's CURRENT target in one call — the repeated align() of
 * apps/align.cpp:32-36 ("10times"), multi-hypothesis initial guesses, or candidate scans sharing one map. Each one runs
 * computeTransformation (gicp_omp_impl.hpp:369-515) with the handle's parameters; the outer loops advance in lock-step
 * rounds, and the inner BFGS solves of a round share one persistent launch with up to three of them in flight
 * (b200reg_ndt_set_batch_slots), so one registration's BFGS arithmetic overlaps the others' cost / gradient sums.
 * Every result is BITWISE the result b200reg_align gives for the same (source, guess).
 * guesses: 16*count floats column-major, or NULL (identity). results[k].status is B200REG_OK or an error code
 * (B200REG_ERR_TIMEOUT: the device watchdog fired during registration k). The target covariances are the handle's
 * cached ones; the handle's own source and its covariances are not touched (a later align() registers that source as
 * before). After the call the getters (final transformation, converged, iterations, correspondences) describe the LAST
 * registration; b200reg_get_stats reports evaluations, gicp_inner_ms, gicp_inner_launches and gicp_pair_evaluations
 * summed over the batch. count == 0 is a no-op. */
typedef struct b200reg_gicp_batch_result {
  float final_T[16];    /* getFinalTransformation(), column-major                          */
  int converged;        /* hasConverged()                                                   */
  int iterations;       /* outer iterations (nr_iterations_)                                */
  int evaluations;      /* cost / gradient evaluations over all inner loops                 */
  int correspondences;  /* m of the last outer iteration (b200reg_gicp_num_correspondences) */
  int status, pad;      /* B200REG_OK or an error code                                      */
} b200reg_gicp_batch_result;
/* sources in HOST memory: (base, n, stride) clouds as in b200reg_set_input_source, one bulk copy + unpack each, no
 * synchronisation in between */
int b200reg_gicp_align_batch(b200reg_t h, int count, const float* const* sources, const size_t* n_points,
                             size_t stride_bytes, const float* guesses, b200reg_gicp_batch_result* results);
/* sources already in HBM as float4 (x, y, z, ignored) on the handle's device; read in place (no copy) — they must be
 * complete when the call is made and stay untouched until it returns */
int b200reg_gicp_align_batch_device(b200reg_t h, int count, const void* const* dev_sources, const size_t* n_points,
                                    const float* guesses, b200reg_gicp_batch_result* results);

/* ---- pcl::VoxelGrid<PointXYZI>::filter (sm.cpp:266-269,311-314,325-328,444-447; gbs.cpp:225-226) ------ */
/* Centroid downsample of all fields (x,y,z,intensity). intensity_offset_bytes < 0: no intensity field.
 * out: same point layout as in (stride_bytes), capacity in points; *m = number of output points (ascending
 * leaf index). If the grid would overflow int32 the input is returned unchanged (PCL behaviour). */
int b200reg_voxelgrid(int device, const float* in, size_t n, size_t stride_bytes, long intensity_offset_bytes,
                      float leaf, float* out, size_t out_capacity, size_t* m);

/* ---- introspection (parity tests, roofline accounting) ---------------------------------------------- */
typedef struct b200reg_stats {
  int evaluations;        /* computeDerivatives passes of the last align (ndt_omp_impl.hpp:179)          */
  int iterations;         /* nr_iterations_                                                              */
  long long hits;         /* (point, voxel) pairs visited in the last evaluation                         */
  long long hits_total;   /* ... summed over all evaluations of the last align                           */
  float solve_ms;         /* device time of the last align's solver kernel (CUDA events, handle stream)  */
  float target_build_ms;  /* device time of the last setInputTarget                                      */
  int kernel_launches;    /* kernels launched by this handle since creation                              */
  int grid_ctas, block_threads, index_in_smem;
  long long n_voxels, n_cells, n_source, n_target;
  /* GICP: the persistent inner-loop kernel(s) of the last align or GICP batch (estimateRigidTransformationBFGS on the
   * device)                                                                                                          */
  float gicp_inner_ms;             /* their summed device time (CUDA events on the handle's stream)                  */
  int gicp_inner_launches;         /* = outer iterations                                                            */
  double gicp_pair_evaluations;    /* sum over cost / gradient evaluations of the number of correspondences          */
} b200reg_stats;
int b200reg_get_stats(b200reg_t h, b200reg_stats* out);

/* one fused derivative pass (ndt_omp_impl.hpp:179-284) at a given transform T (col-major) with the angle
 * tables taken at p6[3..5]; out: score, g[6], H[36] row-major. */
int b200reg_ndt_derivatives(b200reg_t h, const float* T, const double* p6, int compute_hessian, double* score,
                            double* g6, double* H36);
/* Hessian-only pass over the radius neighbourhood in f64 (ndt_omp_impl.hpp:538-629) */
int b200reg_ndt_hessian_radius(b200reg_t h, const float* T, const double* p6, double* H36);
/* voxel map read-back, voxels with >= 6 points in ascending leaf index (voxel_grid_covariance_omp_impl.hpp:
 * 282-367). Any pointer may be NULL. mean3/icov9 doubles, centroid3 floats. */
int b200reg_ndt_num_voxels(b200reg_t h, size_t* out);
int b200reg_ndt_get_voxels(b200reg_t h, int* leaf_idx, int* npts, double* mean3, double* icov9, float* centroid3);
/* GICP read-back for parity tests: per-point 3x3 covariances (row-major doubles, gicp_omp_impl.hpp:48-122) of the
 * source (which = 0) or target (which = 1) cloud after an align(); *n = number of points (out9 may be NULL). */
int b200reg_gicp_get_covariances(b200reg_t h, int which, double* out9, size_t* n);
int b200reg_gicp_num_correspondences(b200reg_t h, int* out);
/* exact 1-NN of n query points against the target cloud (building block of getFitnessScore / GICP) */
int b200reg_nn1(b200reg_t h, const float* base, size_t n, size_t stride_bytes, int* idx, float* d2);

/* ---- scan-matcher frontend session: device-resident map maintenance (SURVEY.md section 8f, rows 1 and 3) --------
 * The callers either side of align() in scanmatcher/src/scanmatcher_component.cpp, rebuilt so that a frame costs ONE
 * host-to-device copy: the submaps (voxel-filtered, sensor frame) and the targeted cloud stay in HBM.
 * Poses are position (x, y, z) + quaternion (x, y, z, w) in double, like geometry_msgs/Pose.                       */
typedef struct b200sm_session* b200sm_t;
int b200sm_create(int device, b200sm_t* out);
void b200sm_destroy(b200sm_t s);
const char* b200sm_last_error(b200sm_t s);
int b200reg_get_kind(b200reg_t h, int* kind);
/* node parameters: vg_size_for_input, vg_size_for_map, num_targeted_cloud, trans_for_mapupdate, use_min_max_filter,
 * scan_min_range, scan_max_range (sm.cpp:34-50; defaults 0.2, 0.1, 10, 1.5, false, 0.1, 100)                        */
int b200sm_set_params(b200sm_t s, float vg_size_for_input, float vg_size_for_map, int num_targeted_cloud,
                      double trans_for_mapupdate, int use_min_max_filter, double scan_min_range, double scan_max_range);
int b200sm_set_initial_pose(b200sm_t s, const double* position3, const double* quat_xyzw); /* sm.cpp:57-69, 127-141 */
/* cloud_callback range filter (sm.cpp:211-219) + receiveCloud's VoxelGrid(vg_size_for_input) and
 * registration->setInputSource (sm.cpp:323-328): uploads the frame once and keeps it on the device for a later
 * b200sm_update_map. *n_filtered = points of the filtered source.                                                    */
int b200sm_set_scan(b200sm_t s, b200reg_t reg, const float* points, size_t n, size_t stride_bytes,
                    long intensity_offset_bytes, size_t* n_filtered);
/* updateMap (sm.cpp:438-491; the first call is initializeMap, sm.cpp:257-297) on the frame given to the last
 * b200sm_set_scan / b200sm_receive_cloud: VoxelGrid(vg_size_for_map) -> new submap (kept untransformed with its
 * pose); targeted cloud = transformPointCloud(filtered, final_T [float]) followed by the previous
 * num_targeted_cloud-1 submaps, newest first, each through its pose matrix [double]. adopt_now != 0 also performs
 * receiveCloud's registration->setInputTarget(targeted) (sm.cpp:300-322; GICP: VoxelGrid(vg_size_for_input) first). */
int b200sm_update_map(b200sm_t s, b200reg_t reg, const float* final_T_colmajor16, const double* position3,
                      const double* quat_xyzw, int adopt_now);
/* One frame of the frontend: cloud_callback + initializeMap (first frame) + receiveCloud + publishMapAndPose
 * (sm.cpp:201-235, 299-434): adopt a pending target, filter, setInputSource, align(guess = current pose), pose
 * bookkeeping, and updateMap when the sensor moved >= trans_for_mapupdate (performed immediately; the new target is
 * adopted at the start of the next frame — the reference's mapping thread finishing before the next scan).
 * pose7_out = position + quaternion after the frame; *map_updated = 1 if updateMap ran.                             */
int b200sm_receive_cloud(b200sm_t s, b200reg_t reg, const float* points, size_t n, size_t stride_bytes,
                         long intensity_offset_bytes, double* pose7_out, float* final_T_colmajor16_out, int* map_updated);
/* read-back (parity tests; the node's map / map_array publishers). Clouds are x, y, z, intensity floats. */
int b200sm_num_submaps(b200sm_t s, size_t* out);
int b200sm_get_targeted(b200sm_t s, float* out_xyzi, size_t capacity, size_t* n);
int b200sm_get_submap(b200sm_t s, size_t index, float* out_xyzi, size_t capacity, size_t* n, double* pose_colmajor16,
                      double* distance);
int b200sm_get_filtered_scan(b200sm_t s, float* out_xyzi, size_t capacity, size_t* n);
/* GraphBasedSlamComponent::searchLoop (gbs.cpp:144-258) on the session's submaps, device-resident: the newest submap is the
 * source; among the older submaps with (travelled-distance gap > distance_loop_closure) and (position distance <
 * range_of_searching_loop_closure) the closest one, id_min, is the candidate; target = VoxelGrid(voxel_leaf_size) of the
 * submaps id_min +- search_submap_num, each moved by its pose cast to float; align() without guess, getFitnessScore();
 * accepted iff fitness < threshold_loop_closure_score, then relative_pose = from^-1 * (final * init) as in the LoopEdge.
 * `reg` is the backend's registration object (gbs.cpp:47-64 sets its parameters). 4x4 matrices are column-major.       */
typedef struct b200sm_loop_result {
  int is_candidate, id_min, accepted, pad;
  double min_dist, fitness;
  float final_T[16];
  double relative_pose[16];
  size_t n_source, n_target;
} b200sm_loop_result;
int b200sm_search_loop(b200sm_t s, b200reg_t reg, float voxel_leaf_size, double threshold_loop_closure_score,
                       double distance_loop_closure, double range_of_searching_loop_closure, int search_submap_num,
                       b200sm_loop_result* out);
/* ---- IMU de-skew (use_imu; sm.cpp:205-209, 222-235): LidarUndistortion of scanmatcher/include/scanmatcher/
 * lidar_undistortion.hpp. getImu (:52-106) is the per-message ring-buffer update (host state); adjustDistortion
 * (:110-226) runs as kernels on the uploaded scan: the half-turn switch is a first-index reduction, the carried IMU
 * ring pointer an exclusive prefix-max scan, interpolation + rigid correction per point.                          */
int b200sm_imu_set_scan_period(b200sm_t s, double scan_period);                        /* setScanPeriod :228  */
int b200sm_imu_push(b200sm_t s, const float* angular_velocity3, const float* linear_acceleration3,
                    const float* orientation_xyzw, double stamp_sec);                  /* getImu :52-106      */
/* arm the de-skew for the NEXT frame given to b200sm_set_scan / b200sm_receive_cloud: it then runs on the device right
 * after the upload, before the range filter — cloud_callback's order (sm.cpp:205-219)                              */
int b200sm_deskew_next_scan(b200sm_t s, double scan_time_sec);
/* adjustDistortion (:110-226) on a HOST cloud, in place (x, y, z rewritten; points in firing order)               */
int b200sm_imu_adjust_distortion(b200sm_t s, float* points, size_t n, size_t stride_bytes, long intensity_offset_bytes,
                                 double scan_time_sec);
/* read-back for the parity tests: imu_ptr_front_, imu_ptr_last_, imu_ptr_last_iter_; one ring entry                */
int b200sm_imu_get_state(b200sm_t s, int* ptr_front, int* ptr_last, int* ptr_last_iter);
int b200sm_imu_get_sample(b200sm_t s, int index, double* stamp, float* rpy3, float* shift3, float* velo3);

/* A backend in its OWN process gets the submaps as lidarslam_msgs/SubMap (voxel-filtered cloud in the sensor frame, pose,
 * travelled distance; gbs.cpp:91-101): append one to the session (uploaded once, then device-resident like the
 * frontend's own). pose: 4x4 column-major double (Eigen::Affine3d::matrix().data()).                                 */
int b200sm_import_submap(b200sm_t s, const float* points, size_t n, size_t stride_bytes, long intensity_offset_bytes,
                         const double* pose_colmajor16, double distance);

/* Every candidate instead of the closest one (SURVEY.md section 8f row 2): all older submaps that pass the two gates of
 * gbs.cpp:187-204 are registered against the newest submap, each exactly like b200sm_search_loop does its single one
 * (id_min = the candidate's submap id, min_dist = its distance), on the device-resident submaps — nothing is uploaded.
 * out[0..*n_out) in ascending submap id. shard_rank / shard_world (0 / 1 on one GPU) deal the candidates out across
 * processes (candidate k -> rank k mod shard_world; *n_candidates_total = all of them); the rows are then all-gathered
 * with include/b200comm.h.                                                                                          */
int b200sm_search_loop_all(b200sm_t s, b200reg_t reg, float voxel_leaf_size, double threshold_loop_closure_score,
                           double distance_loop_closure, double range_of_searching_loop_closure, int search_submap_num,
                           int shard_rank, int shard_world, b200sm_loop_result* out, size_t capacity, size_t* n_out,
                           size_t* n_candidates_total);

typedef struct b200sm_stats {
  size_t n_scan, n_filtered, n_targeted, n_submaps;
  int kernel_launches;
  double trans, latest_distance;
} b200sm_stats;
int b200sm_get_stats(b200sm_t s, b200sm_stats* out);

#ifdef __cplusplus
}
#endif
#endif /* B200REG_H_ */
