/* b200reg — B200-native scan-to-map registration engine, C ABI.
 *
 * Drop-in boundary for the hot path of matiable/pointcloud-slam (SURVEY.md §8b).
 * The reference has no C ABI of its own; each entry point below names the C++
 * interface it replaces (paths relative to the reference's src/).  Thin C++
 * adaptors that re-create those interfaces on top of this ABI live in
 * the pointcloud-slam_b200/host/ headers (see INTEGRATION.md).
 *
 * Conventions
 *   - every function returns int32 status: B200_OK, a positive "soft" status
 *     (no effective points / not converged) or a negative error; nothing throws;
 *   - handles are opaque; the caller owns every host buffer; device memory and
 *     one CUDA stream belong to the handle; a handle is not re-entrant, distinct
 *     handles may be used from different threads;
 *   - point clouds are passed as (const float* xyz, n, stride_bytes): x,y,z are the
 *     first three floats of each record (stride 48 = pcl::PointXYZINormal,
 *     32/16 = PointXYZI, 12 = packed);
 *   - there is no CPU fallback: without a CUDA device create() fails with
 *     B200_ERR_CUDA.
 */
#ifndef B200REG_H_
#define B200REG_H_
#include <stddef.h>
#include <stdint.h>
#ifdef __cplusplus
extern "C" {
#endif

#define B200_OK 0
#define B200_NO_EFFECTIVE_POINTS 1 /* dyn_share.valid == false on every pass (laser_mapping.cc:657-661) */
#define B200_NOT_CONVERGED 2       /* NDT: converged_ == false (NaN step, ndt_omp_impl.hpp:119-123) */
#define B200_ERR_ARG (-1)
#define B200_ERR_CUDA (-2)
#define B200_ERR_NOMEM (-3)
#define B200_ERR_RANGE (-4)    /* coordinate outside the +-2^20-cell key range, or NDT grid too large */
#define B200_ERR_CAPACITY (-5) /* voxel capacity too small to hold a single new voxel */
#define B200_ERR_NCCL (-6)

const char* b200_version(void);
const char* b200_last_error(void);

/* ------------------------------------------------------------------------- *
 * B1 — local map.  Replaces jueying_lio::IVox<3, DEFAULT, PointType>
 * (jueying_lio/include/ivox3d/ivox3d.h:53-88).
 * ------------------------------------------------------------------------- */
typedef struct b200_map b200_map;
typedef struct {
    float resolution;         /* IVox::Options::resolution_  (ivox3d.h:54) */
    int32_t nearby;           /* NearbyType: 0 CENTER, 6, 18, 26 (ivox3d.h:46-51); other -> 18 (laser_mapping.cc:138-149) */
    uint64_t capacity_voxels; /* IVox::Options::capacity_ (ivox3d.h:57) */
    float max_range;          /* GetClosestPoint max_range, 5.0 (ivox3d.h:79) */
    uint64_t max_points;      /* device point-pool size hint; 0 = 8M */
} b200_map_params;

/* IVox(Options) (ivox3d.h:64-67) */
int32_t b200_map_create(const b200_map_params* params, int32_t device, b200_map** out);
int32_t b200_map_destroy(b200_map* map);
/* IVox::AddPoints(const PointVector&) (ivox3d.h:73, 256-281).  Insertion ordinals continue across calls. */
int32_t b200_map_insert(b200_map* map, const float* xyz, int64_t n, int64_t stride_bytes);
/* IVox::GetClosestPoint(pt, closest_pt, 5, max_range) (ivox3d.h:79, 132-204) for n query points.
 * idx[n*5]: insertion ordinals ascending by (distance, stencil/in-voxel enumeration rank), -1 padded;
 * sqdist[n*5] float squared distances; count[n]. */
int32_t b200_map_knn5(b200_map* map, const float* xyz_world, int64_t n, int64_t stride_bytes, int32_t* idx, float* sqdist,
                      int32_t* count);
/* the same search, also returning the neighbours themselves: neighbours_xyz = n x 5 x 3 floats (rows past count[i] are zero).
 * This is what IVox::GetClosestPoint's closest_pt carries (ivox3d.h:79); a caller needs no host-side copy of the map, which
 * would go stale as soon as MapIncremental inserts on the device. */
int32_t b200_map_knn5_points(b200_map* map, const float* xyz_world, int64_t n, int64_t stride_bytes, int32_t* idx, float* sqdist,
                             int32_t* count, float* neighbours_xyz);
/* IVox::NumValidGrids() (ivox3d.h:88) / NumPoints() (ivox3d.h:85) */
int64_t b200_map_num_voxels(b200_map* map);
int64_t b200_map_num_points(b200_map* map);
/* Non-finite points and points outside the +-2^20-cell key range are NOT inserted (the reference's (int)round(NaN) is
 * undefined behaviour; ivox3d.h:284-286): the rest of the batch goes in, the call returns B200_OK, and this reports how
 * many points were dropped so far (return value) and by the last insert (*last_batch, may be NULL).  Dropped points
 * still consume insertion ordinals. */
int64_t b200_map_dropped(b200_map* map, int64_t* last_batch);

/* ------------------------------------------------------------------------- *
 * B2 — IEKF measurement update.  Replaces
 *   esekfom::esekf::update_iterated_dyn_share_modified (IKFoM_toolkit/esekfom/esekfom.hpp:1526-1834)
 *   driven with LaserMapping::ObsModel (jueying_lio/src/laser_mapping.cc:592-701),
 *   and LaserMapping::MapIncremental (laser_mapping.cc:525-583).
 * State vector x[26]: pos(3) rot(x,y,z,w) offset_R_L_I(x,y,z,w) offset_T_L_I(3) vel(3) bg(3) ba(3) grav(3)
 * (use-ikfom.hpp:14-15, Eigen quaternion coefficient order).  P[23*23] row-major.
 * ------------------------------------------------------------------------- */
typedef struct b200_iekf b200_iekf;
typedef struct {
    int32_t max_iter;         /* NUM_MAX_ITERATIONS (laser_mapping.cc:89) */
    float plane_thr;          /* ESTI_PLANE_THRESHOLD (laser_mapping.cc:90) */
    int32_t extrinsic_est_en; /* laser_mapping.cc:687 */
    double R;                 /* LASER_POINT_COV (options.h:12) */
    double limit[23];         /* epsi (laser_mapping.cc:19) */
    double filter_size_map;   /* filter_size_map_min_ (laser_mapping.cc:547) */
} b200_iekf_params;

#define B200_MAX_PASSES 8
typedef struct {
    int32_t status;
    int32_t passes;     /* ObsModel evaluations */
    int32_t knn_passes; /* of which searched the map (dyn_share.converge == true) */
    int32_t converged;  /* t > 1 at exit */
    int32_t n_eff[B200_MAX_PASSES];
    int32_t knn[B200_MAX_PASSES];
    float gpu_ms; /* device time of the whole update (CUDA events on the handle's stream) */
} b200_iekf_stats;

/* Page-locked host buffers (cudaHostAlloc).  A scan handed to b200_iekf_update in such a buffer (or in any memory the
 * caller registered with cudaHostRegister) crosses PCIe straight from the caller's memory and is unpacked on the device:
 * no host-side packing pass.  Pageable buffers (a PCL cloud) keep working and are packed through an internal pinned stage. */
int32_t b200_host_alloc(size_t bytes, void** out);
int32_t b200_host_free(void* p);

int32_t b200_iekf_create(const b200_iekf_params* params, b200_map* map, b200_iekf** out);
int32_t b200_iekf_destroy(b200_iekf* ekf);
/* kf_.update_iterated_dyn_share_modified(R, t) for one downsampled scan (laser_mapping.cc:335-351). */
int32_t b200_iekf_update(b200_iekf* ekf, const float* scan_body_xyz, int64_t n, int64_t stride_bytes, double* x26,
                         double* P23x23, b200_iekf_stats* stats);
/* Same update with the scan already resident on the device (float4 per point: x,y,z,unused).  The buffer must stay
 * valid and unchanged until the b200_iekf_map_incremental call that follows (it re-reads the scan). */
int32_t b200_iekf_update_device(b200_iekf* ekf, const void* d_scan_float4, int64_t n, double* x26, double* P23x23,
                                b200_iekf_stats* stats);
/* h_x^T h_x (12x12 row-major) and h_x^T h of pass `pass` of the last update (H/b parity, 1e-6 relative) */
int32_t b200_iekf_last_HtH(b200_iekf* ekf, int32_t pass, double* HtH144, double* Hth12, double* x_in26);
/* One ObsModel evaluation at state x with dyn_share.converge = converge (parity primitive). */
int32_t b200_iekf_obs_model(b200_iekf* ekf, const float* scan_body_xyz, int64_t n, int64_t stride_bytes, const double* x26,
                            int32_t converge, double* HtH144, double* Hth12, int32_t* n_eff);
/* Per-point arrays after the last ObsModel evaluation: plane_coef_, residuals_, point_selected_surf_,
 * nearest_points_ (as insertion ordinals) — any pointer may be NULL. */
int32_t b200_iekf_point_state(b200_iekf* ekf, int64_t n, float* plane4, float* residual, uint8_t* selected, int32_t* nn_idx5,
                              int32_t* nn_count);
/* esekf::predict (IKFoM_toolkit/esekfom/esekfom.hpp:269-374) with jueying_lio's process model (use-ikfom.hpp:36-77) over the K IMU
 * intervals of a scan, as ImuProcess::UndistortPcl drives it (imu_processing.hpp:190-241): steps8 = K x 8 doubles
 * {dt, offs_t, acc_avr[3], angvel_avr[3]}, Q12 = diagonal of Q_ (gyr, acc, bias gyr, bias acc).  x26 / P23x23 are propagated
 * in place on the device in one launch; poses22 (K x 22, may be NULL) receives the IMUpose_ entries b200_scan_undistort takes. */
int32_t b200_iekf_predict(b200_iekf* ekf, const double* steps8, int32_t K, const double* Q12, double* x26, double* P23x23,
                          double* poses22);
/* laserCloudWorld of LaserMapping::PublishFrameWorld (laser_mapping.cc:747-773): the last scan moved to the world frame by
 * PointBodyToWorld (:855-864, fp64) at state x, written as records of stride_bytes (x, y, z first, the rest zero; 48 = the
 * pcl::PointXYZINormal layout of the /cloud_registered message, see host/pcd_io.hpp pack_pointcloud2_xyzinormal). */
int32_t b200_iekf_world_scan(b200_iekf* ekf, const double* x26, float* out_xyz, int64_t stride_bytes, int64_t max_points, int64_t* n_out);
/* LaserMapping::MapIncremental() at state x using the neighbours cached by the last update. */
int32_t b200_iekf_map_incremental(b200_iekf* ekf, const double* x26, int32_t ekf_inited, int32_t* n_added,
                                  int32_t* n_no_downsample);

/* ------------------------------------------------------------------------- *
 * B3 — NDT registration.  Replaces pclomp::NormalDistributionsTransform
 * (pointcloud_match/ndt_omp/include/pclomp/ndt_omp.h:117-261, ndt_omp_impl.hpp) and
 * pclomp::VoxelGridCovariance (voxel_grid_covariance_omp_impl.hpp:49-442).
 * 4x4 matrices are float[16] column-major (Eigen::Matrix4f layout).
 * ------------------------------------------------------------------------- */
typedef struct b200_ndt b200_ndt;
typedef struct {
    float resolution;     /* setResolution (ndt_omp.h:142) */
    double step_size;     /* setStepSize */
    double outlier_ratio; /* setOutlierRatio */
    double trans_eps;     /* setTransformationEpsilon */
    int32_t max_iter;     /* setMaximumIterations */
    int32_t search;       /* 0 KDTREE (radiusSearch over the leaf centroids, ndt_omp_impl.hpp:217-219), 1 DIRECT1, 7 DIRECT7, 27 DIRECT26 (ndt_omp.h NeighborSearchMethod) */
    int32_t min_pts;      /* min_points_per_voxel_ = 6 (voxel_grid_covariance_omp.h:210) */
    double eig_ratio;     /* min_covar_eigvalue_mult_ = 0.01 (voxel_grid_covariance_omp.h:211) */
} b200_ndt_params;
typedef struct {
    int32_t converged;
    int32_t iters;      /* getFinalNumIteration */
    int32_t evals;      /* computeDerivatives calls */
    int32_t hess_evals; /* computeHessian calls */
    double trans_probability; /* getTransformationProbability */
    double hessian[36];
    double score;
    double p_final[6];
    float gpu_ms;
} b200_ndt_result;

int32_t b200_ndt_create(const b200_ndt_params* params, int32_t device, b200_ndt** out);
int32_t b200_ndt_destroy(b200_ndt* ndt);
/* setInputTarget -> init() -> VoxelGridCovariance::filter(true) (ndt_omp.h:125-130,299-306) */
int32_t b200_ndt_set_target(b200_ndt* ndt, const float* xyz, int64_t n, int64_t stride_bytes);
/* setInputSource */
int32_t b200_ndt_set_source(b200_ndt* ndt, const float* xyz, int64_t n, int64_t stride_bytes);
int64_t b200_ndt_num_voxels(b200_ndt* ndt); /* leaves with nr_points >= min_pts and a valid covariance */
/* valid leaves sorted by the reference's leaf id; any pointer may be NULL */
int64_t b200_ndt_leaves(b200_ndt* ndt, int64_t max, int64_t* ids, int32_t* npts, double* mean3, double* cov9, double* icov9);
/* align(output, guess) -> computeTransformation (ndt_omp_impl.hpp:70-156) */
int32_t b200_ndt_align(b200_ndt* ndt, const float* guess16, float* final16, b200_ndt_result* result);
/* computeDerivatives at pose vector p (x,y,z,roll,pitch,yaw) (ndt_omp_impl.hpp:169-267) */
int32_t b200_ndt_derivatives(b200_ndt* ndt, const double* p6, double* score, double* g6, double* H36);
/* computeHessian (double path, ndt_omp_impl.hpp:499-560) */
int32_t b200_ndt_hessian(b200_ndt* ndt, const double* p6, double* H36);
/* getMaxEigen() (ndt_omp.h:209-223): largest eigenvalue of the Hessian align() ended with (b200_ndt_result.hessian) / 100000 */
int32_t b200_ndt_max_eigen(const double* hessian36, double* max_eigen);
/* parity primitive: the Newton direction Eigen::JacobiSVD<Matrix<double,6,6>>(H, FullU | FullV).solve(rhs) of
 * computeTransformation (ndt_omp_impl.hpp:112-114) as the device computes it.  *path (may be NULL): 0 = pivoted-elimination
 * shortcut (H comfortably full rank), 1 = literal two-sided Jacobi SVD with Eigen's 6-eps rank threshold; force_svd = 1
 * always takes the latter. */
int32_t b200_ndt_newton_direction(b200_ndt* ndt, const double* H36, const double* rhs6, int32_t force_svd, double* x6, int32_t* path);
/* pcl::Registration::getFitnessScore(max_range) (PCL; loop-closure gate at jueying_slam/src/mapOptmization.cpp:693,719): mean
 * squared distance from the source, moved by T16 (column-major; NULL = final transformation of the last align), to its exact
 * nearest target points; points farther than max_range (squared distance) are skipped; DBL_MAX when none is in range */
int32_t b200_ndt_fitness_score(b200_ndt* ndt, const float* T16, double max_range, double* score, int64_t* n_in_range);
/* calculateScore for h <= 65535 candidate poses (ndt_omp_impl.hpp:836-880) — global relocalization primitive */
int32_t b200_ndt_score_batch(b200_ndt* ndt, const float* poses16, int64_t h, double* scores);
/* align() from h independent initial guesses in one batch (relocalization with refinement): finals16 h x 16, results[h] */
int32_t b200_ndt_align_batch(b200_ndt* ndt, const float* guesses16, int64_t h, float* finals16, b200_ndt_result* results);
/* min_b_ / div_b_ of the voxel grid (voxel_grid_covariance_omp_impl.hpp:86-96) */
int32_t b200_ndt_grid(b200_ndt* ndt, int32_t* min_b3, int32_t* div_b3);

/* Batched registration of independent (source, target, guess) pairs — the loop-closure call site
 * (jueying_slam/src/mapOptmization.cpp:683-693: a fresh NDT per candidate, the keyframe as source, the history submap as
 * target, align(guess), accepted when hasConverged() && getFitnessScore() <= historyKeyframeFitnessScore) for a whole batch
 * of candidates in one call, everything on the device from upload to results.  A separate handle: a b200_ndt's own target
 * and source are never touched.  A pair's result does not depend on the other pairs, on the chunking or on the ranks. */
typedef struct b200_comm b200_comm; /* NCCL communicator (sharded paths, below) */
typedef struct b200_ndt_pairs b200_ndt_pairs;
typedef struct {
    int32_t status;       /* B200_OK / B200_NOT_CONVERGED, or the error set_target / set_source / align would return for this pair alone */
    b200_ndt_result ndt;  /* as b200_ndt_align fills it; gpu_ms = device time of the whole call */
    double fitness;       /* getFitnessScore(max_range) at the final transformation; DBL_MAX when nothing is in range */
    int64_t n_in_range;
    float final16[16];    /* column-major */
} b200_ndt_pair_result;

int32_t b200_ndt_pairs_create(const b200_ndt_params* params, int32_t device, b200_ndt_pairs** out);
int32_t b200_ndt_pairs_destroy(b200_ndt_pairs* h);
/* Pair p: source = records src_off[p] .. src_off[p+1]-1 of src_xyz, target = records tgt_off[p] .. tgt_off[p+1]-1 of tgt_xyz
 * (stride_bytes as everywhere); guesses16 = P x 16 column-major, NULL = identity.  comm may be NULL.  With a communicator every
 * rank passes the same arguments, rank r registers the pairs p = r (mod N), uploads only their clouds, and every rank returns all P results.
 * Malformed arguments (null pointers, P < 1, decreasing offsets, stride < 12) fail the whole call with B200_ERR_ARG; a problem in
 * one pair's clouds (empty source, no finite target point, grid too large) is reported in that pair's status only. */
int32_t b200_ndt_pairs_align(b200_comm* comm, b200_ndt_pairs* h, const float* src_xyz, const int64_t* src_off, const float* tgt_xyz,
                             const int64_t* tgt_off, int64_t stride_bytes, int64_t P, const float* guesses16, double max_range,
                             b200_ndt_pair_result* results);
/* parity probe: the valid leaves of pair p's target from the last call on this rank (as b200_ndt_leaves, leaf ids local to
 * the pair), when pair p was built in the last chunk of that call; -1 otherwise */
int64_t b200_ndt_pairs_leaves(b200_ndt_pairs* h, int64_t p, int64_t max, int64_t* ids, int32_t* npts, double* mean3, double* cov9, double* icov9);

/* Loop closure from a device keyframe store: the front half of performLoopClosure (LIO-SAM mapOptmization.cpp, from which
 * jueying_slam derives) - detectLoopClosureDistance and loopFindNearKeyframes - on the device, feeding the pair registration
 * above.  A keyframe is ONE cloud in the lidar frame, x y z intensity: LIO-SAM keeps a corner and a surf cloud per keyframe
 * and loopFindNearKeyframes appends corner then surf, so pass them concatenated in that order (the order of the points sets
 * the order of VoxelGrid's fp32 sums).  Poses are PointTypePose {x, y, z, roll, pitch, yaw} (float), moved into the world
 * by pcl::getTransformation; times are seconds (double). */
typedef struct b200_keyframes b200_keyframes;
int32_t b200_keyframes_create(int32_t device, b200_keyframes** out);
int32_t b200_keyframes_destroy(b200_keyframes* h);
/* cornerCloudKeyFrames / surfCloudKeyFrames.push_back + cloudKeyPoses3D / cloudKeyPoses6D.push_back (saveKeyFramesAndFactor):
 * records x y z[ intensity] at stride_bytes (>= 16 carries the intensity, 12 stores 0); *key = the keyframe's index (may be NULL) */
int32_t b200_keyframes_add(b200_keyframes* h, const float* xyzi, int64_t n, int64_t stride_bytes, const float* pose6, double time, int64_t* key);
/* the same keyframe given as its two LOAM feature clouds: stores exactly what b200_keyframes_add stores for corner followed by
 * surf, and remembers n_corner so that the local map (b200_loam_set_map_from_keyframes) can split the cloud again */
int32_t b200_keyframes_add_features(b200_keyframes* h, const float* corner, int64_t n_corner, int64_t stride_corner, const float* surf, int64_t n_surf,
                                    int64_t stride_surf, const float* pose6, double time, int64_t* key);
/* correctPoses(): poses of keyframes first .. first+count-1 replaced by poses6 (count x 6 floats); clouds untouched */
int32_t b200_keyframes_set_poses(b200_keyframes* h, int64_t first, int64_t count, const float* poses6);
int64_t b200_keyframes_count(b200_keyframes* h); /* -1 for a NULL handle */

typedef struct {
    float search_radius;      /* historyKeyframeSearchRadius */
    double time_gap;          /* historyKeyframeSearchTimeDiff */
    int32_t search_num;       /* historyKeyframeSearchNum */
    float leaf;               /* downSizeFilterICP leaf size */
    int32_t min_source_points; /* 300: cureKeyframeCloud->size() below it is not registered */
    int32_t min_target_points; /* 1000: prevKeyframeCloud->size() below it is not registered */
    double max_range;         /* getFitnessScore argument */
} b200_loop_params;
typedef struct {
    int64_t cur, pre;         /* pre = -1: no candidate */
    float pre_sqdist;         /* squared distance of the detected candidate; 0 when pre was given or is -1 */
    int32_t n_source, n_target; /* sizes after the downsample; 0 when not assembled */
    b200_ndt_pair_result reg; /* B200_OK / B200_NOT_CONVERGED; B200_NO_EFFECTIVE_POINTS = no candidate or under a size gate (not
                                 registered); otherwise the status b200_ndt_pairs_align reports for these clouds */
} b200_loop_result;

/* detectLoopClosureDistance for Q queries (cur[q] = the keyframe that was the newest): the keyframe j < cur[q] nearest to it
 * (squared distance summed x, y, z in fp32, strictly below search_radius^2 = (float)((double)r * r)) with
 * |time_j - time_cur| > time_gap; ties to the lower index; pre[q] = -1 (sqdist 0) without one.  The loopIndexContainer check
 * stays with the caller: detect, filter, then b200_loop_close with explicit pre. */
int32_t b200_loop_detect(b200_keyframes* h, const int64_t* cur, int64_t Q, const b200_loop_params* prm, int64_t* pre, float* sqdist);
/* parity probe: loopFindNearKeyframes(key, search_num) = keyframes key-search_num .. key+search_num (clipped) moved by their
 * poses, appended in index order, VoxelGrid(leaf), min points 0: out_xyzi 4 floats per point in ascending leaf order (at most
 * max_out written, may be NULL), *n_out = points */
int32_t b200_loop_submap(b200_keyframes* h, int64_t key, int32_t search_num, float leaf, float* out_xyzi, int64_t max_out, int64_t* n_out);
/* performLoopClosure up to the fitness gate for Q queries: pre NULL = detect by distance (b200_loop_detect), otherwise pre[q]
 * is query q's partner (detectLoopClosureExternal; -1 = none).  Source = loopFindNearKeyframes(cur, 0), target =
 * loopFindNearKeyframes(pre, search_num), size gates, then align(identity) and getFitnessScore(max_range): reg is the record
 * b200_ndt_pairs_align gives the same two clouds.  comm may be NULL; with a communicator every rank holds the same store and
 * passes the same arguments, rank r assembles and registers the queries q = r (mod N) and every rank returns all Q results.
 * The store and the pairs handle must be on the same device. */
int32_t b200_loop_close(b200_comm* comm, b200_ndt_pairs* ndt, b200_keyframes* h, const int64_t* cur, const int64_t* pre, int64_t Q,
                        const b200_loop_params* prm, b200_loop_result* results);

/* extractSurroundingKeyFrames (LIO-SAM mapOptmization.cpp) from the store, for the scan at time_cur when keyframe cur is the
 * newest (only keyframes 0 .. cur exist; cur = -1: the last one):
 *   extractNearby: keyframes j <= cur strictly inside search_radius of keyframe cur (b200_loop_detect's squared distance and
 *     r^2), in ascending (d2, j) order -> VoxelGrid(density) of their positions -> each centroid's nearest keyframe among
 *     0 .. cur (ties to the lower index) -> then keyframes cur, cur-1, .. while time_cur - time_j < 10.0;
 *   extractCloud: entries whose point (centroid, or the keyframe's own position) lies farther than search_radius from
 *     keyframe cur (sqrtf of the squared distance) are skipped; each remaining keyframe's corner / surf cloud is moved into
 *     the world by its pose and appended (a keyframe listed twice is appended twice); VoxelGrid(corner_leaf) and
 *     VoxelGrid(surf_leaf), min points 0, give laserCloud{Corner,Surf}FromMapDS.
 * Every listed keyframe must have been added with b200_keyframes_add_features (otherwise B200_ERR_ARG).  An empty store is
 * B200_NO_EFFECTIVE_POINTS; a grid of more than 9e18 leaves is B200_ERR_RANGE. */
typedef struct {
    float search_radius; /* surroundingKeyframeSearchRadius (50) */
    float density;       /* surroundingKeyframeDensity (2.0) */
    float corner_leaf;   /* mappingCornerLeafSize (0.2) */
    float surf_leaf;     /* mappingSurfLeafSize (0.4) */
} b200_surround_params;
/* parity probe: the list after extractCloud's distance gate, in extraction order (at most max_keys written), *n_keys = its length */
int32_t b200_keyframes_surrounding(b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params* prm, int64_t* keys, int64_t max_keys,
                                   int64_t* n_keys);
/* parity probe: laserCloudCornerFromMapDS / laserCloudSurfFromMapDS, 4 floats per point in ascending leaf order (at most max_*
 * written), *n_* = their sizes */
int32_t b200_keyframes_surrounding_map(b200_keyframes* h, int64_t cur, double time_cur, const b200_surround_params* prm, float* corner_xyzi,
                                       int64_t max_corner, int64_t* n_corner, float* surf_xyzi, int64_t max_surf, int64_t* n_surf);

/* ------------------------------------------------------------------------- *
 * B3 (alternative) — Generalized ICP.  Replaces pclomp::GeneralizedIterativeClosestPoint<PointT, PointT>
 * (pointcloud_match/ndt_omp/include/pclomp/gicp_omp.h:60-135, gicp_omp_impl.hpp), the registration object
 * jueying_slam/src/localization.cpp:163,175-177 selects with ndt_neighbor_search_method == "GICP_OMP" and drives through
 * pcl::Registration (setInputTarget :277, setInputSource / align / hasConverged / getFitnessScore /
 * getFinalTransformation :323-328).  4x4 matrices are column-major floats like Eigen::Matrix4f::data().
 * ------------------------------------------------------------------------- */
typedef struct b200_gicp b200_gicp;
typedef struct {
    int32_t k_correspondences;     /* setCorrespondenceRandomness, 20 (gicp_omp.h:116) */
    double gicp_epsilon;           /* 0.001 (gicp_omp.h:117) */
    double rotation_epsilon;       /* setRotationEpsilon, 2e-3 (gicp_omp.h:118) */
    double transformation_epsilon; /* setTransformationEpsilon, 5e-4 (gicp_omp.h:125) */
    double corr_dist_threshold;    /* setMaxCorrespondenceDistance, 5.0 (gicp_omp.h:126) */
    int32_t max_iterations;        /* setMaximumIterations, 200 (gicp_omp.h:124) */
    int32_t max_inner_iterations;  /* setMaximumOptimizerIterations, 20 (gicp_omp.h:120) */
} b200_gicp_params;                /* a field <= 0 takes the reference's default */
typedef struct {
    int32_t converged;   /* hasConverged() */
    int32_t iterations;  /* nr_iterations_ */
    int32_t last_m;      /* correspondences of the last pass */
    int32_t last_inner;  /* BFGS steps of the last pass */
    int32_t last_status; /* BFGSSpace status the last pass ended with: 0 Success, 1 NoProgress, -1 Running */
    int32_t inner_total; /* BFGS steps over the whole align */
    int32_t n_f, n_df, n_fdf; /* cost-functor calls: operator(), df, fdf (gicp_omp_impl.hpp:245-368) */
    double delta;        /* the last pass's convergence measure (gicp_omp_impl.hpp:483-494) */
    float gpu_ms;
} b200_gicp_result;
int32_t b200_gicp_create(const b200_gicp_params* params, int32_t device, b200_gicp** out);
int32_t b200_gicp_destroy(b200_gicp* h);
/* setInputTarget (gicp_omp.h:173-178): builds the exact-search index (the kd-tree's role); target covariances are recomputed by the next align */
int32_t b200_gicp_set_target(b200_gicp* h, const float* xyz, int64_t n, int64_t stride_bytes);
/* setInputSource (gicp_omp.h:141-157) */
int32_t b200_gicp_set_source(b200_gicp* h, const float* xyz, int64_t n, int64_t stride_bytes);
/* align(output, guess) -> computeTransformation (gicp_omp_impl.hpp:371-516).  guess16 NULL = identity.  B200_OK, or
 * B200_NOT_CONVERGED when the loop broke on an optimiser exception (fewer than 4 correspondences). */
int32_t b200_gicp_align(b200_gicp* h, const float* guess16, float* final16, b200_gicp_result* result);
/* getFitnessScore(max_range) with the source moved by T16 (NULL = the last final transformation) */
int32_t b200_gicp_fitness_score(b200_gicp* h, const float* T16, double max_range, double* score, int64_t* n_in_range);
/* parity probes.  covariances: computeCovariances (gicp_omp_impl.hpp:49-123) of the source (which = 0) or the target (1), n x 9
 * doubles row-major, and optionally the k neighbour indices per point in ascending (distance, index) order.
 * correspondences: the matching half of one pass at (transformation_, guess): tgt_idx[i] = matched target point or -1, maha9[i] =
 * mahalanobis_[i].block<3,3>, d2[i] = squared distance to the nearest target point (exact whenever it is below the gate).
 * cost: the functor at x (x y z roll pitch yaw) on the correspondences of the last align / correspondences call. */
int32_t b200_gicp_covariances(b200_gicp* h, int32_t which, double* cov9, int32_t* knn_idx);
int32_t b200_gicp_correspondences(b200_gicp* h, const float* trans16, const float* guess16, int32_t* tgt_idx, float* maha9, float* d2, int64_t* m);
int32_t b200_gicp_cost(b200_gicp* h, const double* x6, double* f_op, double* f_fdf, double* g6, int64_t* m);
/* the search grid chosen for a cloud: cell size, dense cells, occupied cells */
int32_t b200_gicp_index_info(b200_gicp* h, int32_t which, float* leaf, int64_t* cells, int64_t* occupied);

/* ------------------------------------------------------------------------- *
 * Sharded paths (one process per GPU, NCCL over NVLink).  The reference is single-process and has no
 * counterpart (SURVEY.md F4): each hypothesis is scored with the reference's calculateScore arithmetic.
 * ------------------------------------------------------------------------- */
#define B200_NCCL_ID_BYTES 128
int32_t b200_comm_unique_id(uint8_t* id128);   /* on one rank; ship the 128 bytes to the others out of band */
int32_t b200_comm_init_rank(int32_t nranks, int32_t rank, const uint8_t* id128, int32_t device, b200_comm** out);
int32_t b200_comm_destroy(b200_comm* comm);
/* setInputTarget for a map replicated on every rank: `root` passes the cloud (xyz may be NULL elsewhere, n equal
 * everywhere), the packed points are ncclBroadcast once and every rank builds identical voxel Gaussians. */
int32_t b200_ndt_set_target_bcast(b200_comm* comm, b200_ndt* ndt, const float* xyz, int64_t n, int64_t stride_bytes, int32_t root);
/* Global relocalization.  Hypotheses h_begin..h_begin+h-1 of a global grid are scored on this rank with calculateScore;
 * the cost that is minimised is -score (the winner is the most likely pose).  Every rank receives the same global
 * winner through one collective: each rank's local winner travels as a 16-byte (order-preserving fp64 score key, index)
 * pair in an ncclAllGather and every rank reduces the gathered pairs (exact, ties to the lower index).
 * comm may be NULL (single GPU).  best = -1 and B200_NO_EFFECTIVE_POINTS when no rank had a hypothesis. */
int32_t b200_reloc_argmin(b200_comm* comm, b200_ndt* ndt, const float* poses16, int64_t h, int64_t h_begin, int64_t* best,
                          double* best_score, float* gpu_ms);
/* same with an interleaved slice: local hypothesis i = global hypothesis h_begin + i * h_stride (rank r of N: h_begin r, stride N) */
int32_t b200_reloc_argmin_strided(b200_comm* comm, b200_ndt* ndt, const float* poses16, int64_t h, int64_t h_begin, int64_t h_stride,
                                  int64_t* best, double* best_score, float* gpu_ms);
/* How b200_reloc_argmin[_strided] scores (per handle; default on): on = every hypothesis is first scored in fp32 with a
 * certified interval that contains its calculateScore value, and only those that can still be the winner are scored in
 * fp64; off = all of them in fp64.  The winner, its score bits and the return code are the same either way. */
int32_t b200_ndt_set_reloc_screen(b200_ndt* ndt, int32_t on);
/* The certified intervals behind the screen: lo[i] <= calculateScore(pose i) <= hi[i] for h <= 65535 poses, with
 * [-inf, +inf] where no finite bound holds (non-finite poses, a missing source ordering). */
int32_t b200_ndt_score_screen(b200_ndt* ndt, const float* poses16, int64_t h, double* lo, double* hi);
/* Global relocalization with NDT refinement: score -> global top-K -> align() of every candidate -> getFitnessScore -> winner.
 * Slices as for b200_reloc_argmin_strided (comm may be NULL).  The candidates are the top_k hypotheses of highest
 * calculateScore over all ranks (NaN scores and poses with a non-finite entry never qualify), ordered by score descending,
 * then global index ascending; *n_cands = how many there are (fewer than top_k when fewer hypotheses have a finite score).
 * Candidate j is aligned on rank j mod N from its hypothesis pose with computeTransformation against the handle's target and
 * source, then getFitnessScore(max_range) runs at its final transformation.  cands[0 .. top_k) receives the candidates in that
 * order (slots past *n_cands: hypothesis -1, everything else zero); refined.ndt.gpu_ms is 0 - the device time of the whole
 * call is *gpu_ms (may be NULL, as may n_cands).  A candidate's record depends only on its pose, the handle's target and
 * source and the parameters: it is bit-identical for any top_k, slicing and number of ranks.
 * *best = the hypothesis of the converged candidate (refined.status == B200_OK) with the highest trans_probability, ties to
 * the lower hypothesis, and the call returns B200_OK; with no converged candidate, the highest trans_probability among all of
 * them and B200_NOT_CONVERGED; with no candidate at all, -1 and B200_NO_EFFECTIVE_POINTS.
 * With a communicator every rank passes the same top_k and max_range (they set the sizes of the two ncclAllGathers), and every
 * rank returns the same code, *best and cands: a rank whose own part fails (a malformed slice, no target or source, a CUDA
 * error) still takes part in both collectives and its error is returned everywhere.  A NULL ndt or a top_k outside
 * 1 .. 65535 is B200_ERR_ARG at once, before any collective. */
typedef struct {
    int64_t hypothesis;           /* global index h_begin + i * h_stride on the rank that scored it; -1 = empty slot */
    double initial_score;         /* calculateScore at the hypothesis pose: the bits b200_ndt_score_batch returns */
    b200_ndt_pair_result refined; /* status (B200_OK / B200_NOT_CONVERGED), align result, fitness at the final pose, final16 */
} b200_reloc_candidate;
int32_t b200_reloc_refine(b200_comm* comm, b200_ndt* ndt, const float* poses16, int64_t h, int64_t h_begin, int64_t h_stride,
                          int64_t top_k, double max_range, int64_t* best, b200_reloc_candidate* cands, int64_t* n_cands, float* gpu_ms);

/* measurement aids (bench.py): device time of the scoring of the last score / relocalization call (the fp64 score kernel of
 * a score call; screen, selection, rescore and finish of a screened relocalization); the number of
 * (source point, occupied neighbourhood voxel) pairs over h poses (algorithmic bytes of the roofline); a device-side
 * rendezvous of the ranks on the handle's stream, so that a timed step starts on all ranks together */
float b200_ndt_last_score_kernel_ms(b200_ndt* ndt);
int32_t b200_ndt_score_pairs(b200_ndt* ndt, const float* poses16, int64_t h, int64_t* pairs);
int32_t b200_ndt_stream_barrier(b200_comm* comm, b200_ndt* ndt);

/* ------------------------------------------------------------------------- *
 * Voxel-grid reductions.
 *   b200_voxel_downsample replaces pcl::VoxelGrid<PointType>::filter as jueying_lio runs it on every scan
 *   (jueying_lio/src/laser_mapping.cc:323-328; arithmetic as vendored in jueying_slam/include/voxel_grid_large.cpp:25-258).
 *   b200_mapbuild_* replaces dynamic_map/construct_full_map <poses.txt> <frames_dir> <out.pcd> <leaf>
 *   (scripts/construct_full_map.sh:6; sources absent from the reference - keyframes moved by their poses, merged,
 *   VoxelGrid(leaf)); with a communicator the keyframes are split over GPUs and partial voxel sums are exchanged.
 * ------------------------------------------------------------------------- */
typedef struct b200_downsampler b200_downsampler;
int32_t b200_downsampler_create(int32_t device, b200_downsampler** out);
int32_t b200_downsampler_destroy(b200_downsampler* d);
/* records x, y, z[, intensity] at stride_bytes; out_xyzi 4 floats per voxel in ascending leaf-index order, out_count
 * points per voxel (either may be NULL; at most max_out are written), *n_out = number of voxels.  min_points < 0 is
 * B200_ERR_ARG; a grid of more than 9e18 leaves is B200_ERR_RANGE.  The cloud replaces a scan staged by
 * b200_scan_undistort: b200_voxel_downsample_staged then returns B200_ERR_ARG until the next undistort. */
int32_t b200_voxel_downsample(b200_downsampler* d, const float* xyzi, int64_t n, int64_t stride_bytes, float leaf, int32_t min_points,
                              float* out_xyzi, int32_t* out_count, int64_t max_out, int64_t* n_out);
/* ImuProcess::UndistortPcl, backward half (jueying_lio/include/imu_processing.hpp:175-177,247-284): time-sorts the raw
 * scan and moves every point to the end-of-scan frame.  Float records at stride_bytes (x y z first, time offset in ms at
 * float index time_index - pcl curvature, 9 in PointXYZINormal - intensity at intensity_index or < 0); poses22 = K x 22
 * doubles {offset_time, acc[3], gyr[3], vel[3], pos[3], rot[9]} (IMUpose_ of the forward propagation, which stays on the
 * host); x_end26 = state after the last predict.  The result is staged on the device; out_xyzi / out_order optional. */
int32_t b200_scan_undistort(b200_downsampler* d, const float* points, int64_t n, int64_t stride_bytes, int32_t time_index,
                            int32_t intensity_index, const double* poses22, int32_t K, const double* x_end26, float* out_xyzi,
                            int32_t* out_order);
/* pcl::VoxelGrid::filter on the staged (undistorted) scan - raw scan -> undistort -> downsample -> IEKF update without
 * a host round trip */
int32_t b200_voxel_downsample_staged(b200_downsampler* d, float leaf, int32_t min_points, int64_t* n_out);
/* the last result as it sits on the device (float4 per voxel): pass it to b200_iekf_update_device */
const void* b200_downsampler_device_points(b200_downsampler* d, int64_t* n);

typedef struct b200_mapbuild b200_mapbuild;
int32_t b200_mapbuild_create(float leaf, uint64_t capacity_voxels, int32_t device, b200_mapbuild** out);
int32_t b200_mapbuild_destroy(b200_mapbuild* h);
/* one keyframe (frames/<i>.pcd, x y z intensity) with its pose (a line of poses.txt: x y z qw qx qy qz); asynchronous */
int32_t b200_mapbuild_add_keyframe(b200_mapbuild* h, const float* xyzi, int64_t n, int64_t stride_bytes, const double* pose7);
int32_t b200_mapbuild_add_keyframe_device(b200_mapbuild* h, const void* d_xyzi_float4, int64_t n, const double* pose7);
/* `count` device-resident keyframes in one call (poses7 = count x 7 doubles): they are accumulated several per kernel
 * launch, which is what fills the GPU - one 100k-point keyframe alone is latency bound. */
int32_t b200_mapbuild_add_keyframes_device(b200_mapbuild* h, const void* const* d_xyzi_float4, const int64_t* n, const double* poses7,
                                           int64_t count);
int64_t b200_mapbuild_num_voxels(b200_mapbuild* h);
/* collective: afterwards every voxel lives on exactly one rank with the sums of all ranks.  With comm NULL or one rank
 * nothing is exchanged; the call still waits for the queued keyframes and returns the builder's error, like num_voxels */
int32_t b200_mapbuild_merge(b200_comm* comm, b200_mapbuild* h);
/* centroids held by this rank, ascending (z, y, x) voxel order; returns the voxel count */
int64_t b200_mapbuild_extract(b200_mapbuild* h, float* out_xyzi, int32_t* out_count, int64_t max_out);

/* ------------------------------------------------------------------------- *
 * LOAM-style scan-to-map optimisation (the estimator of jueying_slam).  Replaces cornerOptimization, surfOptimization,
 * combineOptimizationCoeffs, LMOptimization and the loop of scan2MapOptimization
 * (jueying_slam/src/mapOptmization.cpp:1255-1590).  transformTobeMapped = t6 (roll, pitch, yaw, x, y, z), float.
 * ------------------------------------------------------------------------- */
typedef struct b200_loam b200_loam;
typedef struct {
    int32_t iters;        /* passes of the scan2MapOptimization loop that ran */
    int32_t n_sel;        /* laserCloudSelNum of the last pass */
    int32_t converged;    /* LMOptimization returned true */
    int32_t degenerate;   /* isDegenerate */
    float gpu_ms;
    double AtA_first[36]; /* matAtA of the first pass (parity) */
} b200_loam_stats;
int32_t b200_loam_create(int64_t max_map_points, int32_t device, b200_loam** out);
int32_t b200_loam_destroy(b200_loam* h);
/* kdtreeCornerFromMap / kdtreeSurfFromMap ->setInputCloud(laserCloud{Corner,Surf}FromMapDS) (:1568-1569) */
int32_t b200_loam_set_map(b200_loam* h, const float* corner_xyz, int64_t n_corner, int64_t stride_corner, const float* surf_xyz, int64_t n_surf,
                          int64_t stride_surf);
/* the optimisation loop for one scan (laserCloud{Corner,Surf}LastDS, lidar frame); t6 updated in place */
int32_t b200_loam_optimize(b200_loam* h, const float* corner_xyz, int64_t n_corner, int64_t stride_corner, const float* surf_xyz, int64_t n_surf,
                           int64_t stride_surf, float* t6, int32_t iter_num, b200_loam_stats* stats);
/* one cornerOptimization + surfOptimization pass at t6 (parity probe) */
int32_t b200_loam_features(b200_loam* h, const float* corner_xyz, int64_t n_corner, int64_t stride_corner, const float* surf_xyz, int64_t n_surf,
                           int64_t stride_surf, const float* t6, uint8_t* flags, float* coeff4, int32_t* n_sel);
typedef struct {
    int64_t n_list;                 /* surroundingKeyPosesDS entries (centroids + recent keyframes) */
    int64_t n_kept;                 /* entries left by extractCloud's distance gate */
    int64_t n_corner_raw, n_surf_raw; /* laserCloud{Corner,Surf}FromMap sizes */
    int64_t n_corner, n_surf;       /* laserCloudCornerFromMapDSNum, laserCloudSurfFromMapDSNum */
    float gpu_ms;                   /* device time of the call, selection to the last insert */
    int32_t pad;
} b200_surround_info;
/* extractSurroundingKeyFrames (b200_keyframes_surrounding_map) followed by b200_loam_set_map with the two clouds, without the
 * points leaving the device: the maps afterwards are byte for byte those b200_loam_set_map builds from the probe's clouds.
 * The store and the handle must be on the same device.  B200_NO_EFFECTIVE_POINTS (empty store), B200_ERR_CAPACITY (a
 * downsampled map larger than max_map_points) and the argument / range errors leave the previous maps in place.  info may be
 * NULL. */
int32_t b200_loam_set_map_from_keyframes(b200_loam* h, b200_keyframes* store, int64_t cur, double time_cur, const b200_surround_params* prm,
                                         b200_surround_info* info);

/* the scan-to-map optimisation on clouds that already sit on the device (float4 x y z intensity records, b200_features_device_cloud):
 * b200_loam_optimize with a device copy in place of the pack and upload; the same t6 bits and stats.  Buffers on another device
 * than the handle are B200_ERR_ARG. */
int32_t b200_loam_optimize_device(b200_loam* h, const void* d_corner, int64_t n_corner, const void* d_surf, int64_t n_surf, float* t6, int32_t iter_num,
                                  b200_loam_stats* stats);
/* b200_keyframes_add_features from device clouds (float4 x y z intensity): stores the bytes b200_keyframes_add_features stores
 * for their host copies at a stride of 16 bytes.  Buffers on another device than the store are B200_ERR_ARG. */
int32_t b200_keyframes_add_features_device(b200_keyframes* h, const void* d_corner, int64_t n_corner, const void* d_surf, int64_t n_surf,
                                           const float* pose6, double time, int64_t* key);

/* ------------------------------------------------------------------------- *
 * LOAM front end (LIO-SAM imageProjection without deskew, featureExtraction, mapOptimization's downsampleCurrentScan), the
 * contract restated in oracle/feature_oracle.cpp.  One scan per call on one device.
 * ------------------------------------------------------------------------- */
typedef struct b200_features b200_features;
typedef struct {
    int32_t n_scan;          /* N_SCAN, 1 .. 1024 */
    int32_t horizon_scan;    /* Horizon_SCAN; n_scan * horizon_scan <= 2^26 */
    int32_t downsample_rate; /* >= 1 */
    int32_t sensor;          /* 0: velodyne / ouster (column from the azimuth), 1: livox (column = arrival order in the line) */
    float min_range, max_range;          /* lidarMinRange, lidarMaxRange */
    float edge_threshold, surf_threshold; /* edgeThreshold, surfThreshold */
    float odometry_surf_leaf;            /* odometrySurfLeafSize (per-ring surf VoxelGrid) */
    float mapping_corner_leaf, mapping_surf_leaf; /* downsampleCurrentScan */
    int32_t pad;
} b200_feature_params;
typedef struct {
    int64_t n_in;
    int64_t dropped_nonfinite, dropped_range, dropped_row, dropped_col, dropped_dup;
    int64_t n_extracted;                /* extracted cloud (cloud_info) */
    int64_t n_corner, n_surface;        /* cornerCloud, surfaceCloud */
    int64_t n_corner_ds, n_surf_ds;     /* laserCloud{Corner,Surf}LastDS */
    float gpu_ms;                       /* device time of the call, upload to the last downsample */
    int32_t pad;
} b200_feature_info;
#define B200_FEATURES_CORNER 0
#define B200_FEATURES_SURFACE 1
#define B200_FEATURES_CORNER_DS 2
#define B200_FEATURES_SURF_DS 3
/* parameters out of bounds are B200_ERR_ARG */
int32_t b200_features_create(const b200_feature_params* prm, int32_t device, b200_features** out);
int32_t b200_features_destroy(b200_features* h);
/* steps 1-6 for one scan: n records of stride bytes (a multiple of 4; x y z the first three floats), the intensity a float at
 * intensity_offset (< 0: none, 0 is used), the ring an unsigned integer of ring_bytes (1 or 2) at ring_offset.  One upload of
 * the scan; synchronises before it returns.  An empty extracted cloud is B200_NO_EFFECTIVE_POINTS with empty clouds; a
 * VoxelGrid of more than 9e18 leaves is B200_ERR_RANGE.  info may be NULL. */
int32_t b200_features_extract(b200_features* h, const void* points, int64_t n, int64_t stride, int64_t intensity_offset, int64_t ring_offset,
                              int32_t ring_bytes, b200_feature_info* info);
/* parity probes of the last extract (any output may be NULL; *n the full size, at most max written): the extracted cloud (x y z
 * intensity), pointColInd, pointRange, start / endRingIndex (n_scan each); curvature, label, picked flags */
int32_t b200_features_cloud_info(b200_features* h, float* cloud_xyzi, int32_t* col, float* range, int32_t* start_ring, int32_t* end_ring, int64_t max,
                                 int64_t* n);
int32_t b200_features_labels(b200_features* h, float* curvature, int8_t* label, uint8_t* picked, int64_t max, int64_t* n);
/* cornerCloud (pick order), surfaceCloud, or the two DS clouds (which = B200_FEATURES_*), x y z intensity */
int32_t b200_features_cloud(b200_features* h, int32_t which, float* out_xyzi, int64_t max, int64_t* n);
/* the same cloud as it sits on the device (float4 per point), valid until the next extract: pass it to
 * b200_loam_optimize_device / b200_keyframes_add_features_device */
const void* b200_features_device_cloud(b200_features* h, int32_t which, int64_t* n);
int32_t b200_features_device(b200_features* h);

#ifdef __cplusplus
}
#endif
#endif
