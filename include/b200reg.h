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

/* measurement aids (bench.py): device time of the score kernel of the last score / relocalization call; the number of
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

#ifdef __cplusplus
}
#endif
#endif
