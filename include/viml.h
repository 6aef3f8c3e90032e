/*
 * viml.h — C-ABI of the B200-native sliding-window linearisation hot path of TC-VIML.
 *
 * This is the drop-in boundary (SURVEY.md §8b).  Every entry point is `extern "C"`, takes plain
 * pointers and sizes, and replaces one reference interface on the hot path (paths are relative to
 * the reference tree, /root/reference):
 *
 *   viml_linearize_batch   <- ProjectionFactor::Evaluate        vins_estimator/src/factor/projection_factor.cpp:21-124
 *                             LineProjectionFactor::Evaluate    vins_estimator/src/factor/line_projection_factor.cpp:19-120
 *                             ResidualBlockInfo::Evaluate       vins_estimator/src/factor/marginalization_factor.cpp:3-69
 *                             ThreadsConstructA (J^T J, J^T r)  vins_estimator/src/factor/marginalization_factor.cpp:141-172
 *                             landmark part of MarginalizationInfo::marginalize  marginalization_factor.cpp:267-282
 *   viml_marginalize_batch <- MarginalizationInfo::marginalize  marginalization_factor.cpp:174-299 (dense prior part)
 *   viml_line_associate    <- Estimator::UpdateLinesInFoV       vins_estimator/src/estimator.cpp:385-447
 *                             Estimator::LineCorrespondenceInFrame  estimator.cpp:671-885
 *                             (+ CalAngleDist :601-613, CalEulerDist :615-669, Line2D fm.cpp:4-15,:46-71)
 *   viml_set_map           <- lines3d_map ingest                vins_estimator/src/parameters.cpp:50-59, estimator.cpp:54-58
 *   viml_load_line_map     <- the line_3d.txt reader            vins_estimator/src/parameters.cpp:50-59
 *   viml_reduced_system    <- the prior and IMU residual blocks of the window entering the normal equations:
 *                             MarginalizationFactor::Evaluate   marginalization_factor.cpp:335-384
 *                             IMUFactor::Evaluate               vins_estimator/src/factor/imu_factor.h:19-181
 *                             (evaluated by their owners; their r / J blocks are inputs here), ThreadsConstructA rule :141-172
 *   viml_gn_step           <- one solver iteration of ceres::Solve  estimator.cpp:1888-1905 (normal equations, Schur elimination of
 *                             the landmarks, dense solve, PoseLocalParameterization::Plus  pose_local_parameterization.cpp:3-19)
 *   viml_inertial_evaluate <- IMUFactor::Evaluate               vins_estimator/src/factor/imu_factor.h:19-181
 *                             IntegrationBase::evaluate         vins_estimator/src/factor/integration_base.h
 *                             MarginalizationFactor::Evaluate   marginalization_factor.cpp:335-384
 *                             (pre-integration itself stays with the host)
 *   viml_gn_step_vi        <- viml_gn_step over the window's whole problem: the IMU and prior factors evaluated on the device at
 *                             x (system) and at x+ (cost[1] = f(x+))
 *   viml_solve_vi          <- ceres::Solve of the window's whole problem  estimator.cpp:1888-1905 (TrustRegionMinimizer with
 *                             LevenbergMarquardtStrategy; every step is viml_gn_step_vi's; deviations at the declaration)
 *   viml_fov_update / viml_fov_slide / VIML_FOV_CACHED
 *                          <- the per-slot FoV lists the estimator keeps between frames: UpdateLinesInFoV at frame entry
 *                             (estimator.cpp:342) and their shifts in slideWindowWithLinesFoV (estimator.cpp:2148, :2160, :2218)
 *   viml_track_gate        <- FeatureManager::removeLineOutlier + lineDiff  vins_estimator/src/feature_manager.cpp:494-541
 *   viml_triangulate_batch <- FeatureManager::triangulate       feature_manager.cpp:440-492
 *   viml_config            <- the fields Estimator::setParameters reads for this path, estimator.cpp:54-124
 *
 * Conventions
 *   - parameter-block layout is the reference's (estimator.cpp:1492-1532): pose = [px,py,pz,qx,qy,qz,qw],
 *     feature = inverse depth, extrinsic pose like pose.  All arithmetic is IEEE binary64 unless noted.
 *   - every function returns VIML_OK (0) or a negative error code; viml_last_error() gives the text.
 *     No exception crosses the ABI.  Buffers are caller-owned.
 *   - a context belongs to one CUDA device and one calling host thread; all device work of a context is
 *     ordered on its own stream.  There is NO CPU fallback: without a usable CUDA device viml_create fails.
 *   - pointers in the in/out structs are HOST pointers (pinned preferred, see viml_host_alloc) unless
 *     VIML_PTRS_DEVICE is set, in which case they are device pointers on the context's device, the call only
 *     enqueues work on the context stream, and the caller synchronises with viml_sync().
 */
#ifndef VIML_H_
#define VIML_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VIML_ABI_VERSION 5

/* ---- error codes ---------------------------------------------------------------------------- */
#define VIML_OK 0
#define VIML_ERR_INVALID (-1)  /* bad argument / inconsistent sizes                               */
#define VIML_ERR_CUDA (-2)     /* CUDA runtime error (text in viml_last_error)                    */
#define VIML_ERR_NO_DEVICE (-3)/* no usable sm_100 device: there is deliberately no CPU fallback  */
#define VIML_ERR_NOMAP (-4)    /* viml_line_associate or a line table before viml_set_map         */
#define VIML_ERR_UNSUPPORTED (-5)

/* ---- flags ---------------------------------------------------------------------------------- */
#define VIML_OUT_RESIDUAL_JACOBIAN 0x01u /* mode A: per-factor r and J blocks (Ceres Evaluate layouts) */
#define VIML_OUT_HB 0x02u                /* mode B: per-window block-structured H = J^T J, b = +J^T r  */
#define VIML_OUT_SCHUR 0x04u             /* landmark-eliminated S, g per window                        */
#define VIML_LOSS_CAUCHY 0x10u           /* apply the ResidualBlockInfo::Evaluate loss correction      */
#define VIML_S_PACKED 0x20u              /* with VIML_OUT_SCHUR: S is written as its upper triangle, [W][D(D+1)/2], row r holds
                                            columns r..D-1 (entry (r,c) at r*D - r(r-1)/2 + c - r): half the bytes back to the host */
#define VIML_PTRS_DEVICE 0x100u          /* in/out pointers are device pointers; call is asynchronous  */

typedef struct viml_ctx viml_ctx;

/* Fields of Estimator::setParameters (estimator.cpp:54-124) that the hot path reads. */
typedef struct viml_config {
  double fx, fy, cx, cy;      /* pixel intrinsics K (estimator.cpp:66-71)                          */
  int32_t width, height;      /* image size (estimator.cpp:78-79)                                  */
  double Rbw[9];              /* map -> VIO-world rotation, row-major (estimator.cpp:91-100)       */
  double Tbw[3];              /* map -> VIO-world translation                                      */
  double overlap_th;          /* estimator.cpp:116                                                 */
  double dist_th;             /* estimator.cpp:117                                                 */
  double angle_th;            /* estimator.cpp:119                                                 */
  double sqrt_info;           /* ProjectionFactor::sqrt_info = s*I2, s = FOCAL_LENGTH/1.5 (:85)    */
  double cauchy_a;            /* ceres::CauchyLoss(a), a = 1.0 (estimator.cpp:1682)                */
} viml_config;

/* ---- lifetime -------------------------------------------------------------------------------- */
int viml_abi_version(void);
int viml_create(viml_ctx** out, const viml_config* cfg, int device);
void viml_destroy(viml_ctx* ctx);
const char* viml_last_error(const viml_ctx* ctx);
int viml_sync(viml_ctx* ctx);                 /* cudaStreamSynchronize on the context stream        */
void* viml_stream(viml_ctx* ctx);             /* the context's cudaStream_t (for event timing)      */
int viml_host_alloc(void** p, size_t bytes);  /* pinned host memory (cudaHostAlloc)                 */
int viml_host_free(void* p);
int viml_device_alloc(viml_ctx* ctx, void** p, size_t bytes);
int viml_device_free(viml_ctx* ctx, void* p);
int viml_memcpy_h2d(viml_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
int viml_memcpy_d2h(viml_ctx* ctx, void* dst, const void* src, size_t bytes); /* async on ctx stream */
int64_t viml_kernel_launches(const viml_ctx* ctx); /* kernels launched by this context so far       */

/* ---- measurement hooks (bench.py roofline; not needed for results) -----------------------------
 * Between viml_profile_begin and viml_profile_end every kernel launch of the context is bracketed by a
 * pair of CUDA events on the context stream.  viml_profile_end synchronises and returns, per kernel id
 * (see viml_kernel_name), the summed device time in ms and the number of launches.                  */
#define VIML_NUM_KERNELS 16
int viml_profile_begin(viml_ctx* ctx);
int viml_profile_end(viml_ctx* ctx, double* ms_per_kernel, int64_t* launches_per_kernel);
const char* viml_kernel_name(int kernel_id);
/* FP64 peaks of this device measured with register-resident micro-kernels on the context stream:
 * dfma_tflops counts 2 flop per DFMA; dmul_dadd_tops counts 1 op per un-fused DMUL or DADD (the
 * association translation unit is compiled without FMA contraction).                               */
int viml_microbench_fp64(viml_ctx* ctx, double* dfma_tflops, double* dmul_dadd_tops);
/* FP64 tensor-core peak: mma.sync m8n8k4.f64 (DMMA), 512 flop per warp instruction.                 */
int viml_microbench_dmma(viml_ctx* ctx, double* dmma_tflops);
/* Self-test of the association kernels' division with a hoisted reciprocal (the bit-exact contract of
 * viml_line_associate rests on it): computes a[k] / b[k] both ways on the device for n HOST pairs and returns the
 * number of quotients that differ in any bit (NaN == NaN). Must be 0. */
int viml_selftest_division(viml_ctx* ctx, const double* a, const double* b, int64_t n, int64_t* mismatches);

/* ---- prior line map -------------------------------------------------------------------------- */
/* lines_xyzxyz: N rows of [sx sy sz ex ey ez] exactly as line_3d.txt (parameters.cpp:50-59).
 * Always a HOST pointer.  The map is packed once into six SoA planes in HBM.                    */
int viml_set_map(viml_ctx* ctx, const double* lines_xyzxyz, int64_t n_lines);
/* Reads a line_3d.txt prior map like the loop of readParameters (parameters.cpp:50-59): every text line of the file is one map
 * row of six whitespace-separated doubles, sx sy sz ex ey ez, and is pushed whether or not it parsed (the reference leaves the
 * fields after a failed extraction uninitialised; here they are 0 — defined where the reference is not).  Installs the map with
 * viml_set_map; *n_lines (optional) receives the number of rows.  VIML_ERR_INVALID when the file cannot be opened.        */
int viml_load_line_map(viml_ctx* ctx, const char* path, int64_t* n_lines);

/* ---- linearisation ---------------------------------------------------------------------------
 * A batch of W independent sliding windows.  Factors are grouped by window (CSR offsets); inside a
 * window the order is free (it only fixes floating-point summation order).
 *
 * Point factor k (ProjectionFactor, projection_factor.h:10-21) couples pose i, pose j, the extrinsic
 * and feature `feat` of its window:   pf_idx[k] = i | (j << 8) | (feat << 16).
 * pf_obs[k] = {pts_i.x, pts_i.y, pts_j.x, pts_j.y}; pts_i.z = pf_pts_i_z[k] or 1.0 when that is NULL
 * (the tracker always publishes z = 1, feature_tracker_node.cpp:121-189; pts_j.z is never read).
 *
 * Observation table (optional, instead of pf_obs): the reference builds every factor of a feature from the feature's FIRST
 * observation and the observing frame's own one (pts_i = it_per_id.feature_per_frame[0].point, pts_j = it_per_frame.point;
 * estimator.cpp:1747-1766, :1961-1982), so pts_i repeats over the factors of a feature.  With pf_obs == NULL the batch carries
 * feat_obs[w][feat] = {pts_i.x, pts_i.y} once per feature and pf_obs_j[k] = {pts_j.x, pts_j.y} per factor (16 + 16/n_obs bytes per
 * factor instead of 32); the library expands them on the device, results are identical to the pf_obs form.
 * The tracker publishes these points as geometry_msgs::Point32 (feature_tracker_node.cpp:159-162) and the estimator widens them
 * (double x = img_msg->points[j].x, estimator_node.cpp:388-390): a caller that still holds the float32 values can pass the table as
 * feat_obs_f32 / pf_obs_j_f32 instead (same shapes, float; 8 + 8/n_obs bytes per factor).  The device widens them exactly like the
 * host would: identical results.
 *
 * Line factor k (LineProjectionFactor, line_projection_factor.h:13-34) couples pose lf_frame[k] only.
 * lf_geom is SoA, nine planes of n_line_factors doubles: P_start.xyz, P_end.xyz (already in VIO world,
 * estimator.cpp:1832-1833), then the detected line's A, B, C (raw-pixel, un-normalised, fm.cpp:11-13).
 * Its K is viml_config's; its b_c_R/b_c_T are the window's extrinsic, rotation normalised
 * (estimator.cpp:1777-1781).
 *
 * Line table (optional, instead of lf_geom): the estimator builds a line factor from the matched MAP line and the detected 2D
 * segment — ptr_start = Rbw * lineWorld.PtrStart + Tbw, ptr_end likewise (estimator.cpp:1832-1833), line_param = (A, B, C) of
 * Line2D(Vector4d) on the float32 channel endpoints (feature_manager.cpp:11-13, estimator_node.cpp:406-410).  With lf_geom == NULL
 * the batch carries lf_map_index[k] (index into the map installed by viml_set_map) and lf_seg2d_f32[k] = {sx, sy, ex, ey}: 20 bytes
 * per line factor instead of 72.  The device forms the nine lf_geom values with the reference's operation order (no fused
 * multiply-add): identical results.  Needs a map (VIML_ERR_NOMAP otherwise); an index outside the map is VIML_ERR_INVALID on the
 * host-pointer path and is clamped on the device-pointer path.
 *
 * Every entry point that takes a batch checks it the same way.  Both flavours check the sizes, the null arrays and the map of a line
 * table (VIML_ERR_NOMAP) before anything is launched.  With host pointers both window offsets must also be CSRs of their factor
 * arrays and every pose, feature, line frame and map index must be in range, else VIML_ERR_INVALID; no kernel ever reads a bad index.
 * The offsets are checked before anything is launched, and so are the indices, except in viml_linearize_batch on 512 windows or more:
 * it checks them chunk by chunk of windows, so the outputs of the chunks before a bad one may already be written.  With device
 * pointers the offsets and indices are the caller's to keep.                                                                        */
typedef struct viml_window_batch {
  int32_t n_windows;         /* W                                                               */
  int32_t poses_per_window;  /* P  (WINDOW_SIZE+1 = 11; up to 255)                              */
  int32_t feats_per_window;  /* F  stride of inv_depth (<= 65535)                               */
  int32_t reserved0;
  const double* poses;       /* [W][P][7]                                                       */
  const double* ex_pose;     /* [W][7]                                                          */
  const double* inv_depth;   /* [W][F]                                                          */
  int64_t n_point_factors;   /* NP                                                              */
  const int32_t* pf_window_offset; /* [W+1], pf_window_offset[W] == NP                          */
  const uint32_t* pf_idx;    /* [NP]                                                            */
  const double* pf_obs;      /* [NP][4]                                                         */
  const double* pf_pts_i_z;  /* [NP] or NULL                                                    */
  int64_t n_line_factors;    /* NL                                                              */
  const int32_t* lf_window_offset; /* [W+1]                                                     */
  const int32_t* lf_frame;   /* [NL]                                                            */
  const double* lf_geom;     /* [9][NL]                                                         */
  const double* feat_obs;    /* [W][F][2] or NULL; read only when pf_obs == NULL                */
  const double* pf_obs_j;    /* [NP][2]   or NULL; read only when pf_obs == NULL                */
  const float* feat_obs_f32; /* [W][F][2] or NULL; read only when pf_obs, feat_obs, pf_obs_j are NULL */
  const float* pf_obs_j_f32; /* [NP][2]   or NULL                                               */
  const int32_t* lf_map_index; /* [NL]    or NULL; read only when lf_geom == NULL               */
  const float* lf_seg2d_f32;   /* [NL][4] or NULL                                               */
} viml_window_batch;

/* Any pointer may be NULL (= not wanted).  D = 6*(P+1): pose blocks 0..P-1 then the extrinsic.
 * Jacobians are row-major 2x7 with column 6 zero, exactly what Evaluate writes
 * (projection_factor.cpp:77-119, line_projection_factor.cpp:102-114).
 * H blocks: H_pp [W][D][D] row-major, full symmetric; H_lp [W][F][D] (row l = landmark l against
 * all pose columns); H_ll [W][F]; b_p [W][D]; b_l [W][F];  b = +J^T r (marginalization_factor.cpp:168).
 * Schur: S = H_pp - sum_l H_lp[l]^T H_lp[l] / H_ll[l],  g = b_p - sum_l H_lp[l]^T b_l[l] / H_ll[l],
 * landmarks with H_ll <= 1e-8 (MarginalizationInfo::eps) are skipped like the reference's pseudo-inverse. */
typedef struct viml_linearize_out {
  double* pf_residual;   /* [NP][2]  */
  double* pf_jac_pose_i; /* [NP][14] */
  double* pf_jac_pose_j; /* [NP][14] */
  double* pf_jac_ex;     /* [NP][14] */
  double* pf_jac_feat;   /* [NP][2]  */
  double* lf_residual;   /* [NL][2]  */
  double* lf_jac_pose;   /* [NL][14] */
  double* H_pp;          /* [W][D][D] */
  double* H_lp;          /* [W][F][D] */
  double* H_ll;          /* [W][F]    */
  double* b_p;           /* [W][D]    */
  double* b_l;           /* [W][F]    */
  double* S;             /* [W][D][D] */
  double* g;             /* [W][D]    */
} viml_linearize_out;

int viml_linearize_batch(viml_ctx* ctx, const viml_window_batch* in, const viml_linearize_out* out,
                         uint32_t flags);

/* ---- dense-block factors and the reduced system of the whole window ----------------------------------
 * Cost functions that are NOT evaluated here — the previous prior (MarginalizationFactor) and the IMU factors — enter as
 * evaluated blocks: factor k has n_k residuals and c_k TANGENT columns (a size-7 pose block contributes its first 6 Jacobian
 * columns, marginalization_factor.cpp:150-151); col_index maps each local column to a column of the window's tangent vector
 *     [ pose 0 .. pose P-1 | extrinsic | X extra columns ]     (D = 6(P+1) pose/extrinsic columns, then e.g. 9 per speed-bias block)
 * Any loss correction has been applied by the owner (the reference passes loss = NULL for both, estimator.cpp:1927, :1939).
 * The three prefix arrays are CSR offsets over the factors; jacobian is row-major n_k x c_k per factor.
 *
 * viml_reduced_system:  Sx = embed(S) + sum_k J_k^T J_k,  gx = embed(g) + sum_k J_k^T r_k   ([W][Dx][Dx], [W][Dx], Dx = D + X),
 * with S, g the landmark-eliminated system of the window's ProjectionFactors / LineProjectionFactors (viml_linearize_batch,
 * VIML_OUT_SCHUR; VIML_LOSS_CAUCHY in `flags` applies to those).  dense == NULL gives the embedding alone.
 * The host-pointer flavour validates the arrays (VIML_ERR_INVALID: offsets that start at 0, window_offset a non-decreasing CSR of
 * the factors, jac_offset steps of n_k * c_k, col_index in [0, D+X) and without a column repeated inside a factor).  The device
 * flavour reads back only the three totals: the rest, col_index distinct inside a factor included, is the caller's to keep.  A
 * repeated column there gives a step that depends on which kernel solves it.                                              */
typedef struct viml_dense_factors {
  int32_t extra_dim;             /* X                                              */
  int32_t reserved0;
  int64_t n_factors;             /* ND                                             */
  const int32_t* window_offset;  /* [W+1] factors of window w                      */
  const int64_t* row_offset;     /* [ND+1] prefix of n_k   -> residual             */
  const int64_t* col_offset;     /* [ND+1] prefix of c_k   -> col_index            */
  const int64_t* jac_offset;     /* [ND+1] prefix of n_k*c_k -> jacobian           */
  const int32_t* col_index;      /* [sum c_k] in [0, D+X), distinct inside a factor */
  const double* residual;        /* [sum n_k]                                      */
  const double* jacobian;        /* [sum n_k*c_k]                                  */
} viml_dense_factors;

typedef struct viml_reduced_out {
  double* Sx; /* [W][Dx][Dx] */
  double* gx; /* [W][Dx]     */
} viml_reduced_out;

int viml_reduced_system(viml_ctx* ctx, const viml_window_batch* in, const viml_dense_factors* dense,
                        const viml_reduced_out* out, uint32_t flags);
/* The same accumulation onto S [W][D][D], g [W][D] the caller already holds (e.g. from viml_linearize_batch with
 * VIML_OUT_SCHUR): what MarginalizationInfo::marginalize does with its IMU and prior factors after the landmarks are gone. */
int viml_reduced_from_schur(viml_ctx* ctx, int32_t n_windows, int32_t D, const double* S, const double* g,
                            const viml_dense_factors* dense, const viml_reduced_out* out, uint32_t flags);

/* ---- one Gauss-Newton / Levenberg-Marquardt iteration for a batch of windows, device resident -------------------
 * What one iteration of ceres::Solve(SPARSE_SCHUR) does with the window's problem (estimator.cpp:1888-1905), on the normal
 * equations this library assembles (b = +J^T r, so the step solves  H dx = -b):
 *   1. linearise every ProjectionFactor / LineProjectionFactor at the given state, eliminate the landmarks, add the dense-block
 *      factors:  Sx, gx  (viml_reduced_system);
 *   2. dx = -(Sx + lambda diag(Sx))^-1 gx   by Cholesky (lambda = 0: Gauss-Newton);  solved[w] = 0 if a pivot is not positive
 *      (the window's state is then returned unchanged);
 *   3. landmarks:  d(inv_depth_l) = -(b_l + H_lp[l] . dx_pose) / H_ll[l]   (0 where H_ll <= 1e-8);
 *   4. update:  p += dp,  q = normalized(q * deltaQ(dtheta))  (PoseLocalParameterization::Plus, pose_local_parameterization.cpp:3-19;
 *      Utility::deltaQ, utility.h:16-28) for poses and extrinsic; inverse depths and the extra state add their increments;
 *   5. cost[w] = { f(x), f(x+), model decrease }  with  f = 1/2 sum rho(|r|^2) over the point and line factors (Cauchy when
 *      VIML_LOSS_CAUCHY, else |r|^2) + 1/2 sum |r_k + J_k dx|^2 over the dense-block factors (their linearisation: re-evaluating
 *      an IMU factor is its owner's job), model decrease = -gx.dx - 1/2 dx.Sx.dx of the damped-free quadratic model.
 * The caller decides acceptance (f(x+) < f(x)) and the next lambda.  All pointers follow VIML_PTRS_DEVICE.            */
typedef struct viml_gn_options {
  double lambda;   /* Levenberg-Marquardt damping on diag(Sx); 0 = Gauss-Newton */
  double reserved0;
} viml_gn_options;

typedef struct viml_gn_out {
  double* poses;      /* [W][P][7]  updated */
  double* ex_pose;    /* [W][7]              */
  double* inv_depth;  /* [W][F]              */
  double* extra;      /* [W][X] or NULL      */
  double* dx;         /* [W][Dx] or NULL: the reduced step */
  double* cost;       /* [W][3]              */
  int32_t* solved;    /* [W]                 */
} viml_gn_out;

int viml_gn_step(viml_ctx* ctx, const viml_window_batch* in, const viml_dense_factors* dense, const double* extra_state /* [W][X] or NULL */,
                 const viml_gn_options* opt, const viml_gn_out* out, uint32_t flags);

/* ---- the window's IMU factors and the prior, evaluated on the device --------------------------------------------------
 * IMUFactor::Evaluate + IntegrationBase::evaluate (vins_estimator/src/factor/imu_factor.h:19-181, integration_base.h) and
 * MarginalizationFactor::Evaluate (marginalization_factor.cpp:335-384) at the current state.  IMU pre-integration stays with the
 * host (IntegrationBase::push_back / midPointIntegration / repropagate): its outputs are inputs here, and so is sqrt_info
 * = LLT(covariance.inverse()).matrixL().transpose(), which the reference recomputes in every Evaluate but which depends on the
 * pre-integration's covariance alone (fixed during a solve).  The library does not invert the badly scaled 15 x 15 covariance.
 *
 * Parameter blocks of a window: pose p (7 values, tangent columns 6p .. 6p+5), the extrinsic (tangent 6P .. 6P+5) and an extra
 * state of X values per window (tangent D + k for value k, D = 6(P+1)), e.g. the speed-bias blocks [V, Ba, Bg] (9 values each).
 * IMU factor k couples pose imu_pose[k][0] (i), the 9 extra values at imu_sb[k][0], pose imu_pose[k][1] (j) and the 9 at
 * imu_sb[k][1]; its reduced block is 15 x 30 over the tangent columns [pose_i(6) | sb_i(9) | pose_j(6) | sb_j(9)].
 * The prior of window w (prior_n[w] = n_w > 0) has n_w rows; block b (prior_block[w][b] = {kind, index, size, first column}) maps its
 * local columns first .. first + local - 1 (local = 6 for a size-7 pose / extrinsic block, else size) to the block's tangent
 * columns; the blocks cover [0, n_w) exactly once.  Extra blocks are vectors (size != 7, size <= VIML_PRIOR_X0_STRIDE): index is their offset
 * in the extra state.
 * The host-pointer flavour validates them (VIML_ERR_INVALID: pose indices in [0, P), i != j, speed-bias offsets with sb + 9 <= X
 * and disjoint, n_w <= n_max, block kinds / sizes / columns as above, D + X <= 232).  The device flavour reads no input back: it
 * checks what the struct fields alone tell (D + X <= 232, X >= 9 when there are IMU factors, extra_state given when X > 0, no
 * null array), clamps pose and block indices, and leaves the rest to the caller.                                            */
#define VIML_BLOCK_POSE 0   /* pose `index` of the window: 7 values                          */
#define VIML_BLOCK_EX 1     /* the extrinsic: 7 values (index unused)                        */
#define VIML_BLOCK_EXTRA 2  /* `size` values at offset `index` of the window's extra state    */
#define VIML_PRIOR_X0_STRIDE 9   /* values per kept block in prior_x0: a speed-bias block (9) is the largest a prior keeps */

typedef struct viml_inertial_factors {
  int32_t extra_dim;                 /* X: extra state per window [W][X]                                                  */
  int32_t reserved0;
  double gravity[3];                 /* G (parameters.cpp: G.z() = g_norm)                                                */
  /* IMUFactor : SizedCostFunction<15, 7, 9, 7, 9> (imu_factor.h)                                                        */
  int64_t n_imu;                     /* NI                                                                                */
  const int32_t* imu_window_offset;  /* [W+1], imu_window_offset[W] == NI                                                 */
  const int32_t* imu_pose;           /* [NI][2]  pose i, pose j                                                           */
  const int32_t* imu_sb;             /* [NI][2]  offsets of speed-bias i / j = [V, Ba, Bg] in the extra state             */
  const double* imu_preint;          /* [NI][17] sum_dt, delta_p[3], delta_q[4] (x y z w), delta_v[3], linearized_ba[3], linearized_bg[3] */
  const double* imu_jacobian;        /* [NI][15][15] ROW-major pre_integration->jacobian (Eigen stores it column-major)    */
  const double* imu_sqrt_info;       /* [NI][15][15] row-major LLT(covariance.inverse()).matrixL().transpose()            */
  /* MarginalizationFactor (last_marginalization_info): at most one per window                                           */
  int32_t prior_n_max;               /* stride: n_w <= prior_n_max                                                        */
  int32_t prior_max_blocks;          /* stride of the block lists                                                         */
  const int32_t* prior_n;            /* [W] n_w, 0 = the window has no prior                                              */
  const double* prior_jacobian;      /* [W][n_max][n_max] linearized_jacobians (the leading n_w x n_w block is read)      */
  const double* prior_residual;      /* [W][n_max]        linearized_residuals                                            */
  const int32_t* prior_n_blocks;     /* [W]                                                                               */
  const int32_t* prior_block;        /* [W][max_blocks][4] kind, index, global size, first column (keep_block_idx - m)    */
  const double* prior_x0;            /* [W][max_blocks][VIML_PRIOR_X0_STRIDE] keep_block_data (first `size` values used)  */
} viml_inertial_factors;

/* Ceres Evaluate layouts, row-major; column 6 of a pose block is exactly 0.  Any pointer may be NULL (= not wanted). */
typedef struct viml_inertial_out {
  double* imu_residual;    /* [NI][15]    */
  double* imu_jac_pose_i;  /* [NI][15][7] */
  double* imu_jac_sb_i;    /* [NI][15][9] */
  double* imu_jac_pose_j;  /* [NI][15][7] */
  double* imu_jac_sb_j;    /* [NI][15][9] */
  double* prior_residual;  /* [W][n_max] (first n_w written; the prior's Jacobian is its input, marginalization_factor.cpp:371-380) */
} viml_inertial_out;

/* Mode A for these factors: r and J at the state (poses / ex_pose of `state`, extra_state [W][X]).  Only n_windows,
 * poses_per_window, poses and ex_pose of `state` are read.  Pointers follow VIML_PTRS_DEVICE.                             */
int viml_inertial_evaluate(viml_ctx* ctx, const viml_window_batch* state, const double* extra_state, const viml_inertial_factors* vi,
                           const viml_inertial_out* out, uint32_t flags);
/* viml_gn_step with the window's prior and IMU factors as its dense-block factors, evaluated on the device: at x for Sx, gx and
 * cost[0]; at x+ for cost[1], which is then f(x+) exactly:  1/2 sum rho(|r|^2) over the visual factors + 1/2 sum |r|^2 over the
 * IMU and prior factors (the reference gives both a NULL loss, estimator.cpp:1927, :1939).  Per window the dense factors are the
 * prior first, then the IMU factors in input order.  Everything else is viml_gn_step's contract (the model decrease, unsolved
 * windows returned unchanged); extra_state is required when X > 0.  With VIML_PTRS_DEVICE the call does not synchronise.     */
int viml_gn_step_vi(viml_ctx* ctx, const viml_window_batch* in, const viml_inertial_factors* vi, const double* extra_state,
                    const viml_gn_options* opt, const viml_gn_out* out, uint32_t flags);

/* ---- a whole Levenberg-Marquardt solve per window, on the device --------------------------------------------------------
 * Replaces the ceres::Solve call of Estimator::OptimizationWithLine (estimator.cpp:1888-1905) for the window's whole problem: the
 * trust-region loop of Ceres' TrustRegionMinimizer with its default LevenbergMarquardtStrategy, restated from Ceres' documented
 * behaviour (not pinned against its source).  Every window keeps its own radius and stops on its own.  Per window:
 *   f(x0) is computed first; if it is not finite the window stops with VIML_SOLVE_FAILURE after 0 iterations, state unchanged.
 *   state: x, radius = initial_radius, decrease_factor = 2, counters.  Each iteration of a running window:
 *   1. lambda = 1 / radius; the step viml_gn_step_vi takes at x with that lambda gives f(x), f(x+), the model decrease m, solved.
 *   2. invalid (solved == 0, f(x+) not finite, or !(m > 0)): consecutive_invalid += 1, radius /= decrease_factor,
 *      decrease_factor *= 2; FAILURE when consecutive_invalid > max_consecutive_invalid.
 *   3. otherwise consecutive_invalid = 0, then in order:
 *      |dx| <= parameter_tolerance (|x| + parameter_tolerance)  -> PARAMETER_TOL at x (dx: the reduced step and the landmark
 *         increments x+ - x; |x| over every state value: 7 per pose, 7 for the extrinsic, the inverse depths, the extra state);
 *      |f(x) - f(x+)| <= function_tolerance f(x)                 -> FUNCTION_TOL at x;
 *      rho = (f(x) - f(x+)) / m;  rho > min_relative_decrease: accept (x = x+), t = 2 rho - 1,
 *         radius = min(max_radius, radius / max(1/3, 1 - t^3)), decrease_factor = 2;
 *      else reject: radius /= decrease_factor, decrease_factor *= 2.
 *   4. iterations += 1; a window still running stops with MIN_RADIUS when radius < min_radius, else with NO_CONVERGENCE when
 *      iterations == max_iterations.
 * A stopped window's state, counters and outputs never change again.  The policy arithmetic is plain IEEE binary64 without fused
 * multiply-adds, so a scalar restatement reproduces it bit for bit.
 * Deviations from Ceres' Solve as the reference configures it:
 *   - the strategy is LEVENBERG_MARQUARDT; the reference asks for DOGLEG, which needs the full-space gradient and the Cauchy point;
 *   - the damping is viml_gn_step's lambda diag(Sx) on the landmark-reduced system (Ceres damps J^T J before the elimination and
 *     clamps the diagonal to [1e-6, 1e32]);
 *   - no gradient tolerance (the full-problem gradient is not formed) and no max_solver_time.
 * Input validation is viml_gn_step_vi's, plus the options below and the required outputs.  W == 0 returns VIML_OK.  With
 * VIML_PTRS_DEVICE the call neither synchronises nor reads anything back: all max_iterations rounds are enqueued on the context
 * stream, and rounds after every window has stopped do only the ungated work (linearisation, Schur step, IMU / prior evaluation).  */
typedef struct viml_solve_options {
  int32_t max_iterations;           /* > 0; every computed step counts, accepted or not   (ceres: max_num_iterations, 50)         */
  int32_t max_consecutive_invalid;  /* >= 0                                                (max_num_consecutive_invalid_steps, 5)  */
  double initial_radius;            /* 0 < min_radius <= initial_radius <= max_radius, all finite  (initial_trust_region_radius, 1e4) */
  double max_radius;                /*                                                     (max_trust_region_radius, 1e16)          */
  double min_radius;                /*                                                     (min_trust_region_radius, 1e-32)         */
  double min_relative_decrease;     /* >= 0                                                (min_relative_decrease, 1e-3)            */
  double function_tolerance;        /* >= 0                                                (function_tolerance, 1e-6)               */
  double parameter_tolerance;       /* >= 0                                                (parameter_tolerance, 1e-8)              */
} viml_solve_options;

#define VIML_SOLVE_NO_CONVERGENCE 0   /* max_iterations reached */
#define VIML_SOLVE_FUNCTION_TOL 1
#define VIML_SOLVE_PARAMETER_TOL 2
#define VIML_SOLVE_MIN_RADIUS 3
#define VIML_SOLVE_FAILURE 4          /* f(x0) not finite, or more than max_consecutive_invalid invalid steps in a row */

typedef struct viml_solve_out {
  double* poses;        /* [W][P][7]  the final state */
  double* ex_pose;      /* [W][7]                     */
  double* inv_depth;    /* [W][F]     (required when F > 0) */
  double* extra;        /* [W][X]     (required when X > 0) */
  int32_t* status;      /* [W] VIML_SOLVE_*          */
  int32_t* iterations;  /* [W] steps computed        */
  int32_t* accepted;    /* [W] steps accepted        */
  double* cost;         /* [W][2] f(x0), f(final state) */
  double* radius;       /* [W] final radius, or NULL */
  double* trace;        /* [W][max_iterations][4] or NULL: f(x), f(x+), model decrease, lambda of every step; NaN rows after
                           the window stopped */
} viml_solve_out;

int viml_solve_vi(viml_ctx* ctx, const viml_window_batch* in, const viml_inertial_factors* vi, const double* extra_state,
                  const viml_solve_options* opt, const viml_solve_out* out, uint32_t flags);

/* ---- dense marginalisation (marginalization_factor.cpp:264-293) --------------------------------
 * Per problem k: A [pos][pos] row-major, b [pos], marginalised block = leading m rows, kept n = pos-m.
 *   Amm <- (Amm+Amm^T)/2;  Amm^+ by symmetric eigen-decomposition, eigenvalues <= eps dropped;
 *   Ar = Arr - Arm Amm^+ Amr;  br = brr - Arm Amm^+ bmm;  second eigen-decomposition of Ar gives
 *   linearized_jacobians = sqrt(S) V^T  [n][n]  and  linearized_residuals = sqrt(S^+) V^T br  [n].
 * Outputs A_schur [n][n], b_schur [n] are always written when non-NULL.                           */
typedef struct viml_marg_batch {
  int32_t n_problems;
  int32_t pos;   /* m + n, <= 256 */
  int32_t m;
  int32_t reserved0;
  double eps;    /* 1e-8 */
  const double* A; /* [K][pos][pos] */
  const double* b; /* [K][pos]      */
} viml_marg_batch;

typedef struct viml_marg_out {
  double* A_schur;              /* [K][n][n] */
  double* b_schur;              /* [K][n]    */
  double* linearized_jacobians; /* [K][n][n] */
  double* linearized_residuals; /* [K][n]    */
} viml_marg_out;

int viml_marginalize_batch(viml_ctx* ctx, const viml_marg_batch* in, const viml_marg_out* out,
                           uint32_t flags);

/* ---- 2D-3D line association --------------------------------------------------------------------
 * For every pose p: (1) FoV cull of the whole map with cull_poses[p] (UpdateLinesInFoV; the reference
 * caches this list at frame entry, estimator.cpp:342), (2) for each of the L detected 2D lines the
 * arg-min candidate under match_poses[p] (LineCorrespondenceInFrame).  match_poses == NULL means the
 * cull pose is used for both.  lines2d are raw-pixel endpoints [sx sy ex ey] as doubles (they arrive as
 * float32 ROS channels, estimator_node.cpp:406-410).  n_lines2d[p] (optional) gives ragged counts <= L. */
typedef struct viml_assoc_query {
  int32_t n_poses;           /* Pq                                  */
  int32_t lines_per_pose;    /* L (stride)                          */
  const double* cull_poses;  /* [Pq][7]                             */
  const double* match_poses; /* [Pq][7] or NULL                     */
  const double* ex_pose;     /* [Pq][7]                             */
  const double* lines2d;     /* [Pq][L][4]                          */
  const int32_t* n_lines2d;  /* [Pq] or NULL (= L everywhere)       */
  const double* cull_ex_pose;/* [Pq][7] or NULL: extrinsic at frame entry (UpdateLinesInFoV's _Ric/_Tic
                                argument, estimator.cpp:385); NULL = ex_pose for both                    */
  const int32_t* fov_slot;   /* with VIML_FOV_CACHED: [Pq] window slot whose cached FoV list pose p is matched against
                                (NULL = slot p); always a HOST pointer                                       */
} viml_assoc_query;

/* match_index: MAP index of the chosen 3D line, -1 = none (est.cpp:869-878 / :703-713).
 * err: {errA, errD, overlap} as the reference's Vector3f (-1,-1,-1 when unmatched).
 * projected: the chosen candidate's projected 2D segment (xx,yy,xx_,yy_ / clipped endpoint); for an unmatched
 *            query the detected line itself (est.cpp:874 returns detectLine).  Queries past n_lines2d[p] are not
 *            processed: their match_index / err / projected entries keep the caller's content.
 * fov_count [Pq]; fov_index [Pq][fov_capacity] = map indices in map order (the WorldLinesInFOV list);
 * a list longer than fov_capacity is truncated in the output only (fov_count still exact, matching
 * still uses the full list).  fov_mask: [Pq][ceil(N/32)] bitset, bit j of word j/32.              */
typedef struct viml_assoc_out {
  int32_t* match_index; /* [Pq][L]    */
  float* err;           /* [Pq][L][3] */
  double* projected;    /* [Pq][L][4] */
  int32_t* fov_count;   /* [Pq]       */
  int32_t* fov_index;   /* [Pq][fov_capacity] */
  int32_t fov_capacity;
  int32_t reserved0;
  uint32_t* fov_mask;   /* [Pq][ceil(N/32)] */
} viml_assoc_out;

int viml_line_associate(viml_ctx* ctx, const viml_assoc_query* q, const viml_assoc_out* out,
                        uint32_t flags);

/* ---- FoV cache and sliding-window bookkeeping on the device ------------------------------------------
 * The reference computes WorldLinesInFOV[i] once, when frame i enters the window (estimator.cpp:342, :385-447), shifts the lists
 * with the window (estimator.cpp:2148, :2160 MARGIN_OLD; :2218 MARGIN_NEW) and re-matches every observation of every track
 * against the cached lists under the current poses (estimator.cpp:449-481).  Here the lists stay in HBM as one bit mask per
 * window slot (VIML_FOV_SLOTS = WINDOW_SIZE + 1):
 *   viml_fov_update(slot, pose, ex)   UpdateLinesInFoV(slot): cull the map for this frame, keep the result in the slot; *count
 *                                     (optional) receives the list length.  pose / ex are HOST pointers (7 doubles each).
 *   viml_fov_slide(marginalize_old)   != 0: slot i <- slot i+1 for i < WINDOW_SIZE, the newest slot keeps its list (:2148, :2160);
 *                                     == 0: slot WINDOW_SIZE-1 <- slot WINDOW_SIZE (:2218).
 *   viml_line_associate(..., VIML_FOV_CACHED)   match against the cached lists: cull_poses / cull_ex_pose are not read, no cull
 *                                     runs; fov_count / fov_index / fov_mask outputs report the cached lists.
 * A slot that was never updated holds an empty list (every query unmatched, as estimator.cpp:703-713).                  */
#define VIML_FOV_SLOTS 11
#define VIML_FOV_CACHED 0x200u
int viml_fov_update(viml_ctx* ctx, int32_t slot, const double* pose, const double* ex_pose, int32_t* count);
int viml_fov_slide(viml_ctx* ctx, int32_t marginalize_old);

/* FeatureManager::triangulate (feature_manager.cpp:440-492) for a batch of point features: feature l of window feat_window[l]
 * starts in frame start_frame[l] and has observations obs_offset[l] .. obs_offset[l+1]-1 in consecutive frames (points = the
 * normalised image points x y z of lineFeaturePerFrame / FeaturePerFrame::point).  depth[l] = svd_V[2] / svd_V[3] of the DLT
 * system in the start camera's frame, INIT_DEPTH when that is below 0.1 (:482-485).  The caller keeps the reference's gates
 * (used_num >= 2 && start_frame < WINDOW_SIZE - 2, estimated_depth > 0 skipped, :444-449).  Pointers follow VIML_PTRS_DEVICE. */
typedef struct viml_triangulate_in {
  int32_t n_windows;
  int32_t poses_per_window;     /* P                                  */
  const double* poses;          /* [W][P][7]                          */
  const double* ex_pose;        /* [W][7]                             */
  int64_t n_features;           /* NF                                 */
  const int32_t* feat_window;   /* [NF]                               */
  const int32_t* start_frame;   /* [NF]                               */
  const int64_t* obs_offset;    /* [NF+1]                             */
  const double* points;         /* [obs_offset[NF]][3]                */
} viml_triangulate_in;
int viml_triangulate_batch(viml_ctx* ctx, const viml_triangulate_in* in, double init_depth, double* depth, uint32_t flags);

/* FeatureManager::removeLineOutlier (feature_manager.cpp:494-541) for T line tracks on the device.  Track t owns observations
 * track_offset[t] .. track_offset[t+1]-1; line_index[k] is the map index of observation k's lineWorld (the matched line, or the
 * first line of the frame's FoV list for an unmatched observation, estimator.cpp:874; -1 = the zero-length fake line of :709).
 *   credible_line[k]     = !( (float)|LineVec(first observation) - LineVec(k)| > 0.1 ),  LineVec = PtrEnd - PtrStart of the map row
 *   credible_matching[t] = !( (count_incredible / n_observations) >= 0.5 )  with the reference's INTEGER division (:524);
 *                          a track without observations keeps credible_matching = 1.
 * Pointers follow VIML_PTRS_DEVICE.                                                                                  */
int viml_track_gate(viml_ctx* ctx, int32_t n_tracks, const int32_t* track_offset, const int32_t* line_index,
                    uint8_t* credible_line, uint8_t* credible_matching, uint32_t flags);
/* Work counters of the last viml_line_associate call (synchronises): gate_tests = CalAngleDist evaluations executed (the
 * angular bins a 2D line's window touches; the reference evaluates the whole FoV list per line), gated = pairs that passed the angle gate (what the reference runs CalEulerDist
 * on), overlap_scored = pairs that survived the distance lower bound and ran the overlap half of CalEulerDist,
 * distance_scored = pairs whose overlap passed and ran the distance half.  For roofline accounting. */
int viml_assoc_stats(viml_ctx* ctx, int64_t* gate_tests, int64_t* gated, int64_t* overlap_scored,
                     int64_t* distance_scored);

/* Sum partial [S | g] (or H/b) buffers of the single-huge-window case across ranks.  `comm` is an
 * ncclComm_t; buf is a device pointer of `count` doubles; in-place ncclAllReduce(sum) on the context
 * stream.  Returns VIML_ERR_UNSUPPORTED when libnccl cannot be loaded.                            */
int viml_allreduce_hb(viml_ctx* ctx, void* nccl_comm, double* buf, int64_t count);

#ifdef __cplusplus
}
#endif
#endif /* VIML_H_ */
