/* mcba.h -- C ABI of the B200 bundle-adjustment engine (libmcba.so).
 *
 * The reference (dattalab-6-cam/multicam-calibration) is pure Python and has no
 * FFI of its own; the drop-in boundary is the set of Python functions in
 * multicam_calibration/bundle_adjustment.py and geometry.py.  Each entry point
 * below names the reference function (file:line under /root/reference/
 * multicam_calibration/) whose arithmetic it replaces; INTEGRATION.md shows the
 * ctypes binding a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes only; every function returns 0 on
 * success or a negative MCBA_ERR_* code (mcba_last_error() gives the text); no
 * exceptions cross the boundary; buffers are caller-owned; a handle is bound to
 * one CUDA device and one stream and is not thread-safe.  Pointers named d_*
 * are DEVICE pointers, h_* are HOST pointers.  All floating point is float64.
 *
 * Parameter vector x (bundle_adjustment.py:128-157): per camera
 * [fx fy cx cy k1 k2 rx ry rz tx ty tz] (12), then per frame [rho(3) tau(3)].
 * Observations: (C, F, N, 2) row-major, NaN = missing (bundle_adjustment.py:82-84).
 */
#ifndef MCBA_H_
#define MCBA_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCBA_OK 0
#define MCBA_ERR_ARG (-1)
#define MCBA_ERR_CUDA (-2)
#define MCBA_ERR_SOLVER (-3)
#define MCBA_ERR_NONFINITE (-4) /* residuals not finite at x0 (scipy least_squares.py:946) */
#define MCBA_ERR_NCCL (-5)
#define MCBA_ERR_STATE (-6)

#define MCBA_LOSS_LINEAR 0
#define MCBA_LOSS_SOFT_L1 1
/* OR-ed into a loss code: Gauss-Newton weight rho' (IRLS majoriser) instead of scipy's
 * rho' + 2 rho'' z (common.py:720-731).  Gradient, cost and fixed point are unchanged. */
#define MCBA_LOSS_IRLS 0x100

#define MCBA_HESSIAN_AUTO 0   /* IRLS while the cost still drops by > 1 % per step, then Triggs */
#define MCBA_HESSIAN_TRIGGS 1 /* scipy's scaling throughout */
#define MCBA_HESSIAN_IRLS 2

typedef struct mcba_handle mcba_handle;

/* Options of the Levenberg-Marquardt loop; field names follow the keyword
 * arguments bundle_adjust forwards to scipy.optimize.least_squares
 * (bundle_adjustment.py:301-313).  Termination tests follow scipy
 * optimize/_lsq/common.py:705-717 and trf.py:466-468. */
typedef struct mcba_options {
  double ftol;      /* default 1e-4 (bundle_adjustment.py:302) */
  double xtol;      /* scipy default 1e-8 */
  double gtol;      /* scipy default 1e-8 */
  int32_t max_nfev; /* <= 0: 100 * n (scipy default for trf) */
  int32_t loss;     /* MCBA_LOSS_* ; reference default soft_l1 */
  double f_scale;   /* scipy default 1.0 */
  int32_t verbose;  /* 0 silent, 1 summary, 2 per-iteration table (reference default 2) */
  int32_t hessian;  /* MCBA_HESSIAN_*: Gauss-Newton weights of the robust loss (default AUTO) */
  double lambda0;   /* initial damping, relative to the Jacobian scaling; <= 0: 1e-3 */
  double lambda_min;
  double lambda_max;
  /* Called once per accepted/rejected iteration when non-NULL (the host side
   * prints scipy's verbose=2 table from it, trf.py:556-558). */
  void (*iter_callback)(void* user, int iteration, int nfev, double cost, double cost_reduction,
                        double step_norm, double optimality);
  void* callback_user;
} mcba_options;

typedef struct mcba_result {
  double cost;       /* 0.5 * sum rho(f^2) at the solution */
  double cost0;      /* at x0 */
  double optimality; /* ||g||_inf */
  double rms;        /* sqrt(mean f^2) over finite scalar residuals, px */
  double step_norm;  /* last accepted ||dx|| */
  double lambda;     /* final damping */
  double solve_ms;   /* device time of the loop (CUDA events) */
  int64_t n_residuals;
  int32_t nfev;
  int32_t njev;
  int32_t iterations;
  int32_t status; /* scipy codes: 0 max_nfev, 1 gtol, 2 ftol, 3 xtol, 4 ftol+xtol, -1 failure */
  int64_t kernel_launches;
} mcba_result;

const char* mcba_last_error(void);
int mcba_version(void);
void mcba_default_options(mcba_options* opt);

/* One handle per (device, problem shape). n_frames is THIS rank's frame count. */
int mcba_create(mcba_handle** out, int n_cameras, int64_t n_frames, int n_points, int device);
int mcba_destroy(mcba_handle* h);
/* Run on a caller-provided cudaStream_t (e.g. torch's current stream); NULL = handle-owned stream. */
int mcba_set_stream(mcba_handle* h, void* cuda_stream);
int mcba_synchronize(mcba_handle* h);

/* Observations (C,F,N,2) + board points (N,3); host or device pointers
 * (is_device != 0).  Builds the frame-tiled layout the kernels stream and the
 * row offsets of the NaN compaction of bundle_adjustment.py:97. */
int mcba_set_observations(mcba_handle* h, const double* uvs, const double* objpoints, int is_device);
int mcba_num_residuals(mcba_handle* h, int64_t* m, int64_t* n_observations);

/* bundle_adjustment.py:66-98  residuals(params, uvs, objpoints): d_r has m entries,
 * C order over (c,f,n,uv) with NaN observations removed element-wise. */
int mcba_residuals(mcba_handle* h, const double* d_x, double* d_r);
/* bundle_adjustment.py:33-63  predict_calib_uvs: d_uv is (C,F,N,2). */
int mcba_predict(mcba_handle* h, const double* d_x, double* d_uv);
/* Analytic replacement of the finite-difference Jacobian (scipy _numdiff.py:288 through
 * jac_sparsity, bundle_adjustment.py:101-125,310): per (c,f,n) blocks of the RESIDUAL
 * Jacobian, d_Jc (C,F,N,2,12) w.r.t. camera c, d_Jp (C,F,N,2,6) w.r.t. frame f.
 * Debug / parity path. */
int mcba_jacobian_blocks(mcba_handle* h, const double* d_x, double* d_Jc, double* d_Jp);
/* 0.5*sum rho, sum f^2, count at x (scipy least_squares.py:226-252 loss_function cost_only). */
int mcba_cost(mcba_handle* h, const double* d_x, int loss, double f_scale, double* h_cost,
              double* h_sumsq, int64_t* h_count);

/* Residual + analytic Jacobian + robust scaling + Schur elimination of the
 * pose blocks in one pass: reduced camera system S (12C x 12C, row major),
 * b (12C), the camera gradient and cost, with pose damping lambda * D_f^2 folded
 * in and NO camera damping (added by the solve).  Replaces scipy trf's
 * J / LSMR machinery (trf.py:415-587).  Outputs are HOST pointers (may be NULL). */
int mcba_build_reduced(mcba_handle* h, const double* d_x, double lambda, int loss, double f_scale,
                       double* h_S, double* h_b, double* h_gcam, double* h_cost);
/* Same, through HOST buffers end to end: uploads uvs (C,F,N,2) and x, runs the
 * pass, downloads S, b.  This is the call bench.py times as "e2e".  With page-locked
 * buffers and >= 16384 frames the observations cross PCIe in eight frame ranges, each
 * tiled, evaluated and reduced while the next is in flight (sums over frames are added
 * at the end); the handle is afterwards usable exactly as after
 * mcba_set_observations + mcba_build_reduced.  MCBA_NO_HOST_PIPELINE=1 forces the
 * single-upload path; pageable buffers always take it (staged by mcba_upload). */
int mcba_build_reduced_host(mcba_handle* h, const double* h_uvs, const double* h_objpoints,
                            const double* h_x, double lambda, int loss, double f_scale,
                            double* h_S, double* h_b, double* h_cost);
/* One damped step from the system built by the last mcba_build_reduced:
 * Cholesky of S + lambda*D_c^2, back-substitution of every pose. d_dx: 12C + 6F. */
int mcba_solve_step(mcba_handle* h, const double* d_x, double lambda, double* d_x_new);

/* Camera parameters held at their initial values.  h_fixed: 12C bytes (host), camera-major in the order of
 * serialize_params (fx fy cx cy k1 k2 rvec tvec), 1 = held, 0 = free; NULL or all zero = none (the solve then
 * takes exactly the unmasked path).  Board poses are always free.  Handle state read by mcba_lm_run,
 * mcba_solve_step and mcba_covariance until the next call.  A masked step is Levenberg-Marquardt on the free
 * sub-problem: held rows / columns of S + lambda D^2 become the identity and their right-hand side 0, held
 * entries of delta_cam are exactly 0 and d_x_new copies d_x there; mcba_lm_run leaves held entries out of the
 * gtol norm, of |x| in the xtol test and of the default budget 100 n.  The gradient it returns stays complete.
 * MCBA_ERR_ARG for an entry other than 0 / 1. */
int mcba_set_fixed(mcba_handle* h, const uint8_t* h_fixed);

/* The whole Levenberg-Marquardt loop on the device (replaces the
 * least_squares call of bundle_adjustment.py:307-313).  d_x: in x0, out solution.
 * d_grad (12C + 6F, may be NULL) receives the gradient at the solution. */
int mcba_lm_run(mcba_handle* h, double* d_x, const mcba_options* opt, mcba_result* res,
                double* d_grad);

/* Covariance of the calibration at d_x: the block inverse of the Gauss-Newton matrix H = J~^T J~, J~ the residual
 * Jacobian row-scaled as scipy's scale_for_robust_loss_function does (weights max(rho' + 2 rho'' z, EPS) for
 * soft_l1, whatever a solve's hessian option was; lambda = 0), times the residual variance s^2.  The 6 extrinsic
 * parameters of reference_camera are held fixed (the gauge).  One evaluation (K2p, K2c, SYRK, finalize), the
 * gauge-fixed inverse of the reduced camera system and one pass over the frames.
 * With a mask (mcba_set_fixed) the held set is the mask together with the gauge: when the mask holds all six
 * extrinsics of some camera no gauge is added and reference_camera must be -1 or such a camera; otherwise
 * reference_camera is the gauge and the mask may hold no extrinsic entry (a partial extrinsic mask would leave a
 * sub-gauge that the reference camera over-constrains).  The result is conditional on the held parameters.
 *   h_cam_cov   (12C x 12C, host, row major, caller's parameter basis): s^2 S^-1; exactly 0 on the rows / columns
 *               of held parameters (which wins over NaN) and of the gauge, NaN on the rows / columns of cameras
 *               without observations.
 *   d_pose_cov  (F, 6, 6, device, may be NULL): s^2 (V^-1 + V^-1 W^T S^-1 W V^-1) per frame, [rvec | tvec];
 *               NaN for frames without observations.
 *   sigma2      > 0: s^2 = sigma2; <= 0: s^2 = 2 cost / (m - p), m finite scalar residuals,
 *               p = free non-gauge parameters of the observed cameras + 6 (observed frames).
 *   h_stats     (host, may be NULL) [9]: s^2, m - p, m, cost, frames without observations, smallest relative
 *               Cholesky pivot of the observed frames' pose blocks, then device ms of {evaluation + frame check,
 *               camera inverse, pose pass}.
 * Errors: MCBA_ERR_ARG for a bad loss / reference_camera, a reference camera without observations or m <= p
 * (sigma2 <= 0); MCBA_ERR_NONFINITE for residuals that are not finite at d_x; MCBA_ERR_SOLVER when an observed
 * frame's pose block or the Jacobi-scaled gauge-fixed camera system has a relative Cholesky pivot <= 1e-12.
 * Single-rank handles only.  The running Marquardt scaling is left as it was; as after mcba_build_reduced, a
 * following mcba_solve_step / mcba_gradient refer to this call's (lambda = 0) evaluation. */
int mcba_covariance(mcba_handle* h, const double* d_x, int loss, double f_scale, int reference_camera, double sigma2,
                    double* h_cam_cov, double* d_pose_cov, double* h_stats);

/* Gradient of 0.5*sum rho at the last evaluated point, [g_cam (12C) | g_pose (6F)] (device). */
int mcba_gradient(mcba_handle* h, double* d_grad);

/* Multi-GPU: frames are sharded across ranks; only the packed reduced system is
 * all-reduced (NCCL).  id is the 128-byte ncclUniqueId made on rank 0. */
int mcba_comm_unique_id(void* id128);
int mcba_comm_init(mcba_handle* h, const void* id128, int rank, int nranks);
/* One-shot all-reduce over NVLink peer memory (one process per GPU of one node): every rank
 * exports the CUDA IPC handle (64 bytes) of its exchange buffer, the host side gathers the handles
 * of all ranks (rank order) and hands them back; from then on the reduced-system and step-scalar
 * sums run as ONE kernel that pushes into every peer's buffer and adds the slots in rank order
 * (bit-identical on all ranks) instead of a library all-reduce.  Without these two calls the
 * NCCL communicator of mcba_comm_init is used. */
int mcba_comm_ipc_export(mcba_handle* h, int rank, int nranks, void* handle64);
int mcba_comm_ipc_open(mcba_handle* h, const void* handles64 /* nranks x 64 bytes, rank order */);
/* Switch between the peer-memory kernel and the NCCL all-reduce (all ranks must agree: the host
 * side turns the peer path off everywhere when any rank failed to map a buffer). */
int mcba_comm_ipc_enable(mcba_handle* h, int enable);

/* Front end of bundle_adjust on the device (bundle_adjustment.py:265-285): frame eligibility
 * (> 1 camera with a complete detection, :266), per-point reprojection errors of the initial
 * guess on eligible frames (:269-276), worst per-camera mean error per frame (:279), outlier
 * threshold (outlier_threshold, or 5 * nanmedian(err) when it is NaN, :281-282) and exclusion
 * (:284-285).  d_uvs (C,F,N,2), d_obj (N,3), d_x = 12C camera parameters + 6F poses of ALL
 * frames (device).  d_use (F bytes, device) receives 1 for every kept frame; h_stats[4] (host) =
 * {threshold used, eligible frames, frames excluded as outliers, finite error values}.
 * The random sub-sampling of :293-296 stays with the caller (numpy's global RNG). */
int mcba_select_frames(int device, void* cuda_stream, const double* d_uvs, int n_cameras,
                       int64_t n_frames, int n_points, const double* d_obj, const double* d_x,
                       double outlier_threshold, uint8_t* d_use, double* h_stats);
/* The same front end in stages, for frame-sharded (multi-GPU) runs: every rank holds a contiguous
 * range of F frames (d_x = 12C camera parameters + the 6F poses of ITS frames) and only counters
 * and 256-bin histograms cross ranks (summed by the host side through torch.distributed).
 *   mcba_frame_errors    bundle_adjustment.py:266-279 on this rank's frames: d_elig (F bytes),
 *                        d_err (C,F,N) per-point errors (NaN = not counted), d_mean (C,F) nanmean
 *                        per camera and frame; h_counts[2] = {eligible frames, finite error values}.
 *   mcba_key_histogram   one pass of an exact radix selection (for the GLOBAL nanmedian of :281-282):
 *                        counts, by their next 8 bits, the finite values of d_vals whose leading
 *                        prefix_bits bits (a multiple of 8, <= 56) equal prefix; d_hist: 256 x uint64
 *                        (device, overwritten).  Values must be non-negative (error norms are).
 *   mcba_apply_threshold bundle_adjustment.py:279-285 with the (global) threshold: d_use (F bytes),
 *                        *h_excluded = eligible frames of this rank excluded as outliers. */
int mcba_frame_errors(int device, void* cuda_stream, const double* d_uvs, int n_cameras,
                      int64_t n_frames, int n_points, const double* d_obj, const double* d_x,
                      double* d_err, double* d_mean, uint8_t* d_elig, int64_t* h_counts);
int mcba_key_histogram(int device, void* cuda_stream, const double* d_vals, int64_t n,
                       uint64_t prefix, int prefix_bits, uint64_t* d_hist);
int mcba_apply_threshold(int device, void* cuda_stream, const double* d_mean, const uint8_t* d_elig,
                         int n_cameras, int64_t n_frames, double threshold, uint8_t* d_use,
                         int64_t* h_excluded);
/* all_calib_uvs[:, use_frames] (bundle_adjustment.py:299-312) on the device:
 * d_out (C, n_used, N, 2) = d_uvs (C, F, N, 2)[:, d_idx]. */
int mcba_gather_frames(int device, void* cuda_stream, const double* d_uvs, int n_cameras,
                       int64_t n_frames, int n_points, const int64_t* d_idx, int64_t n_used,
                       double* d_out);

/* ---- initialisation algebra (the step before bundle_adjust; calibration.py) ----
 * calibration.py:116-143 estimate_pairwise_camera_transform: d_poses1, d_poses2 (F,6) board poses
 * seen by two cameras (NaN rows = not detected); h_transform[6] = per-component median over the
 * common frames of vec(T2_f T1_f^-1) (geometry.py:178-197 vector form); *h_n_common = number of
 * common frames (may be NULL).  No common frame -> NaN, like np.median of an empty array. */
int mcba_pairwise_transform(int device, void* cuda_stream, const double* d_poses1,
                            const double* d_poses2, int64_t n_frames, double* h_transform,
                            int64_t* h_n_common);
/* calibration.py:245-277 consensus_calib_poses: d_all_poses (C,F,6), h_extrinsics (C,6) world ->
 * camera; d_poses (F,6) = nanmedian over cameras of vec(T_world->cam^-1 T_board->cam), NaN rows
 * where no camera detected the board. */
int mcba_consensus_poses(int device, void* cuda_stream, const double* d_all_poses,
                         const double* h_extrinsics, int n_cameras, int64_t n_frames,
                         double* d_poses);
/* geometry.py:38-65 rodrigues_inv (dim = 3: d_matrices (P,3,3) -> d_vectors (P,3)) and
 * geometry.py:178-197 get_transformation_vector (dim = 4: (P,4,4) -> (P,6)). */
int mcba_transformation_vectors(int device, void* cuda_stream, const double* d_matrices,
                                int64_t n, int dim, double* d_vectors);

/* geometry.py:277-325 project_points for P points and one camera:
 * d_points (P,3), ext (6), K (3x3 row major, skew honoured), dist (k1,k2) or NULL. */
int mcba_project_points(int device, void* cuda_stream, const double* d_points, int64_t n_points,
                        const double* h_ext, const double* h_K, const double* h_dist,
                        double* d_uv);
/* The same projection into all C cameras of a rig in one pass over the points (what
 * bundle_adjustment.py:56-62 predict_calib_uvs and a reprojection-error evaluation loop over):
 * h_ext (C,6), h_K (C,3,3), h_dist (C,2) or NULL; d_uv (C,P,2). */
int mcba_project_points_multi(int device, void* cuda_stream, const double* d_points,
                              int64_t n_points, int n_cameras, const double* h_ext,
                              const double* h_K, const double* h_dist, double* d_uv);
/* bundle_adjustment.py:10-30 embed_calib_objpoints: d_poses (F,6), d_obj (N,3) -> d_world (F,N,3). */
int mcba_embed_points(int device, void* cuda_stream, const double* d_poses, int64_t n_frames,
                      const double* d_obj, int n_points, double* d_world);
/* geometry.py:328-358 undistort_points (cv2.undistortPoints(uv, K, dist5, None, K): exactly
 * five fixed-point iterations; rows with a NaN stay NaN): d_uv_in/out (P,2), h_K (3x3), h_dist (5). */
int mcba_undistort_points(int device, void* cuda_stream, const double* d_uv_in, int64_t n_points,
                          const double* h_K, const double* h_dist, double* d_uv_out);
/* geometry.py:361-433 triangulate: d_uvs (C,P,2) NaN = missing, h_ext (C,6), h_K (C,3,3),
 * h_dist (C,5); d_points (P,3). */
int mcba_triangulate(int device, void* cuda_stream, const double* d_uvs, int n_cameras,
                     int64_t n_points, const double* h_ext, const double* h_K,
                     const double* h_dist, double* d_points);

/* Refinement of triangulated points (geometry.refine_points): per point, Levenberg-Marquardt on
 *   0.5 sum_views sum_{u,v} f_scale^2 rho((f / f_scale)^2),  f = observed - project_points(X, ext_c, K_c, k1_c, k2_c)
 * (fx, skew, cx, fy, cy of K; k1, k2 of dist), with scipy's robust losses and its ftol / xtol / gtol tests
 * (least_squares.py:183-219, common.py:705-731) applied per point.  A view is seen when its pixel undistorts
 * to a finite point with the 5-coefficient model, as mcba_triangulate decides it.  These loss codes are this
 * call's own; the bundle-adjustment entry points keep MCBA_LOSS_*. */
#define MCBA_REFINE_LOSS_LINEAR 0
#define MCBA_REFINE_LOSS_SOFT_L1 1
#define MCBA_REFINE_LOSS_HUBER 2
#define MCBA_REFINE_LOSS_CAUCHY 3
#define MCBA_REFINE_LOSS_ARCTAN 4
typedef struct mcba_refine_options {
  int32_t loss;     /* MCBA_REFINE_LOSS_* */
  double f_scale;   /* > 0 */
  double sigma;     /* > 0: pixel noise of the covariance, sigma^2 inv(J~^T J~) */
  double ftol, xtol, gtol;
  int32_t max_iter; /* 1 .. 32767 trial steps per point */
  int32_t flags;    /* reserved, 0 */
} mcba_refine_options;
/* d_uvs (C,P,2) NaN = missing, h_ext (C,6), h_K (C,3,3), h_dist (C,5); d_init (P,3) start, or NULL for the
 * mcba_triangulate result computed in the call.  Outputs (device): d_points (P,3) (may be d_init), d_cost (P)
 * 0.5 sum rho, d_rms (P) reprojection RMS over the point's scalars, d_status (P) {1 gtol, 2 ftol, 3 xtol,
 * 4 ftol + xtol, 0 max_iter, -1 fewer than two seen views (point NaN), -2 non-finite start or cost at the
 * start, or damping beyond its bound (start returned)}, d_iters (P) trial steps, d_cov (P,6) upper triangle
 * xx xy xz yy yz zz of sigma^2 inv(J~^T J~) at the result, J~ scaled as scipy's result.jac (may be NULL),
 * d_view_err (C,P) reprojection distance per view, NaN where unseen (may be NULL), d_n_views (P) seen views
 * (may be NULL).  1 <= C <= 32. */
int mcba_refine_points(int device, void* cuda_stream, const double* d_uvs, int n_cameras, int64_t n_points,
                       const double* h_ext, const double* h_K, const double* h_dist, const double* d_init,
                       const mcba_refine_options* opt, double* d_points, double* d_cost, double* d_rms,
                       int8_t* d_status, int16_t* d_iters, double* d_cov, double* d_view_err, int8_t* d_n_views);

/* Calibration uncertainty carried into refined points (covariance.point_covariance).  At each point X (d_points,
 * e.g. mcba_refine_points' result) and over its seen views V (the rule above), with J~ scaled as d_cov of
 * mcba_refine_points (same loss, f_scale):  H = J~_X^T J~_X,  S_c = -H^-1 J~_X^T J~_c (3 x 12, dX/dtheta_c, J~_c
 * w.r.t. camera c's [fx fy cx cy k1 k2 rvec tvec]; skew held),  d_cov_meas = sigma^2 H^-1 (bit-identical to
 * d_cov of mcba_refine_points at the same point),  d_cov_cal = sum_{c,d in V} S_c cov[c,d] S_d^T with h_cam_cov the
 * (12C, 12C) row-major camera covariance (mcba_covariance's gauge).  Outputs (P,6) upper triangle xx xy xz yy yz
 * zz; d_sens (P,3,12C) S with zero columns for unseen cameras (may be NULL); d_cov_meas may be NULL.  NaN where a
 * point has fewer than two seen views, a non-finite X or a non-positive-definite H; d_cov_cal also NaN where a
 * (c,d) block of h_cam_cov with c, d in V holds a non-finite entry.  loss MCBA_REFINE_LOSS_*, 1 <= C <= 32. */
int mcba_point_covariance(int device, void* cuda_stream, const double* d_uvs, int n_cameras, int64_t n_points,
                          const double* h_ext, const double* h_K, const double* h_dist, const double* d_points,
                          const double* h_cam_cov, int loss, double f_scale, double sigma, double* d_cov_meas,
                          double* d_cov_cal, double* d_sens);

/* ---- reprojection-error QC (the step after bundle_adjust; viz.py:155-177 plot_residuals) ----
 * Per camera and frame whose N corners were all detected: undistort the detections (geometry.py:328-358),
 * homography detections -> board plane as cv2.findHomography computes it (float32-rounded points,
 * normalised DLT, <= 10 iterations of OpenCV's LM refinement; viz.py:166), cv2.perspectiveTransform of
 * the distortion-free projections of the corners d_reproj (C,F,N,2) -- made with
 * mcba_project_points_multi(dist = NULL) from mcba_embed_points, viz.py:159-163 -- into the board's own
 * coordinates (:167-169), and the distance of every transferred corner to the true one (:171-174).
 * d_uvs (C,F,N,2) NaN = missing, d_obj (N,3), h_K (C,3,3), h_dist (C,5);
 * d_transformed (C,F,N,2) and d_err (C,F,N) are NaN for frames with a missing corner.  N <= 128. */
int mcba_homography_transfer(int device, void* cuda_stream, const double* d_uvs, const double* d_reproj,
                             const double* d_obj, int n_cameras, int64_t n_frames, int n_points,
                             const double* h_K, const double* h_dist, double* d_transformed,
                             double* d_err);

/* Per-kernel device timing of the evaluation pass (CUDA events on the handle's stream).
 * Synchronises, returns in ms_out[4] the summed durations of {K2p corner walk, K2c per-frame
 * Schur, SYRK, finalize + all-reduce} over the n evaluations since the last call, resets the
 * counters and switches recording on/off. */
int mcba_profile(mcba_handle* h, int enable, double* ms_out, int* n_out);

/* FP64 vector-pipe peak of the device, measured with a dependency-free DFMA loop (fused
 * multiply-adds per second): the compute ceiling bench.py quotes beside the HBM roofline. */
int mcba_measure_fp64_peak(int device, double* fma_per_s);

/* Caller-owned PAGEABLE host buffers <-> device at PCIe rate: the numpy arrays that cross the
 * reference's Python boundary (all_calib_uvs in, bundle_adjustment.py:195; the residual vector
 * out, :97-98).  Host threads stage 4 MB chunks through pinned bounce buffers on their own copy
 * streams, overlapping the host memcpy / first-touch page faults with the DMA; pinned buffers
 * take one async copy.  Ordered after the work already queued on cuda_stream; the data is in
 * place when the call returns. */
int mcba_upload(int device, void* cuda_stream, void* d_dst, const void* h_src, size_t bytes);
int mcba_download(int device, void* cuda_stream, void* h_dst, const void* d_src, size_t bytes);

/* Number of kernels this handle has launched (bench.py gpu_launches). */
int64_t mcba_kernel_launches(mcba_handle* h);

/* Kernel variants the handle's evaluation and solve take for its shape and observations (the launch
 * heuristics' choices, for tests that must show which branches they reached).  out[n] receives, at the
 * indices below: K2p warps per CTA and grid; K2c mode (1 staged ring, 2 streamed pair), warps of the
 * streamed pair (0 otherwise) and its per-CTA partial count; SYRK warps, CTA rows (gy) and the block
 * count of its compiled tile list (0: listed at run time); the reduced solve (0 cuSOLVER, 3 / 8 register
 * tiles per warp, 119 = 19 tiles per warp with the trailing ones in shared memory); frame
 * tiles; back-substitution grid; C; then the live (tile, camera) units of every camera (C entries).
 * n must be at least MCBA_PLAN_UNITS + C.  Synchronises the handle's stream. */
#define MCBA_PLAN_K2P_WARPS 0
#define MCBA_PLAN_K2P_GRID 1
#define MCBA_PLAN_K2C_MODE 2
#define MCBA_PLAN_K2C_WARPS 3
#define MCBA_PLAN_K2C_PARTS 4
#define MCBA_PLAN_SYRK_WARPS 5
#define MCBA_PLAN_SYRK_GY 6
#define MCBA_PLAN_SYRK_STATIC_NB 7
#define MCBA_PLAN_SOLVE 8
#define MCBA_PLAN_TILES 9
#define MCBA_PLAN_BACKSUB_GRID 10
#define MCBA_PLAN_CAMERAS 11
#define MCBA_PLAN_UNITS 12
int mcba_plan_info(mcba_handle* h, int64_t* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* MCBA_H_ */
