/*
 * svs_b200.h -- C ABI of libsvsb200.so: B200-native (sm_100a) implementation of
 * ScaViSLAM's double-window bundle-adjustment iteration and dense stereo
 * front-end kernels.  Plain pointers and sizes only; no C++ or torch types.
 *
 * Every entry point names the reference interface it replaces
 * (paths relative to the ScaViSLAM tree, commit b29d070).
 *
 * Conventions
 *   SE3      double[7] = qx qy qz qw tx ty tz   (Eigen coeffs order; T_me_from_world)
 *   tangent  (upsilon, omega): translation first, left-multiplicative update
 *            T <- exp(delta) * T          (anchored_points.cpp:53-58)
 *   points   psi = (x/z, y/z, 1/z) in the anchor frame (maths_utils.h:66-69)
 *   status   0 = ok, <0 = error (svs_last_error gives the text); never throws
 *   threads  a handle may be used by one host thread at a time; distinct
 *            handles are independent (own stream, own workspaces)
 */
#ifndef SVS_B200_H
#define SVS_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define SVS_OK 0
#define SVS_ERR_INVALID (-1)      /* bad argument / index out of range */
#define SVS_ERR_CUDA (-2)         /* CUDA runtime error (text in svs_last_error) */
#define SVS_ERR_UNSUPPORTED (-3)  /* structurally valid input this build cannot take */
#define SVS_ERR_STATE (-4)        /* call order (e.g. optimize before set_problem) */
#define SVS_ERR_NOGPU (-5)        /* no CUDA device: there is NO CPU fallback */
#define SVS_ERR_NUMERIC (-6)      /* NaN residual (the reference throws std::runtime_error("Res is NaN!")) */

/* ------------------------------------------------------------------ BA */

typedef struct svs_ba svs_ba;

/* G2oCameraParameters (g2o_types/anchored_points.h:40-58) */
typedef struct {
  double f, px, py, b;
} svs_cam;

typedef struct {
  int device;        /* CUDA device ordinal, -1 = current device */
  int flags;         /* SVS_BA_* */
  int reserved[6];
} svs_ba_opts;

#define SVS_BA_DEFAULT 0
/* Skip the spurious J1'WJ1 prior g2o adds to the anchor pose for an observation
 * made in the landmark's own anchor frame (SURVEY.md B5).  Off = reference behaviour. */
#define SVS_BA_SKIP_SELF_ANCHOR_HESSIAN 1
/* Keep the pose ordering of the caller instead of the fill-reducing one. */
#define SVS_BA_NATURAL_ORDER 2

#define SVS_BA_MAX_ITERS 64

/* Mirrors g2o's per-iteration verbose line (slam_graph.cpp:1066) and
 * SlamGraph::Statistics (slam_graph.hpp:366-386). */
typedef struct {
  int iterations;                       /* return value of g2o optimize() */
  int trials_total;                     /* Levenberg trials (factorisations) */
  double chi2_init;
  double chi2_final;
  double lambda_final;
  double chi2_iter[SVS_BA_MAX_ITERS];   /* robust chi2 after outer iteration i */
  double lambda_iter[SVS_BA_MAX_ITERS];
  int trials_iter[SVS_BA_MAX_ITERS];
  int num_frames, num_points;           /* Statistics::num_frames / num_points */
  int num_point_edges, num_frame_edges; /* Statistics::num_point_edges / num_frame_edges */
  int nnzb_S;                           /* lower blocks of the reduced system incl. diagonal */
  int nnzb_L;                           /* blocks of its Cholesky factor */
  int max_track;                        /* longest landmark track (slots incl. anchor) */
  float ms_total;                       /* device time of the whole optimize() */
  float ms_build;                       /* fused linearise + Schur kernel, summed over trials */
  float ms_solve;                       /* reduced-system factor + solve + pose update */
  float ms_update;                      /* back-substitution + point update + trial chi2 */
  float ms_control;                     /* sharded window: the two all-reduces + LM decision kernel per trial */
  int launches;                         /* kernels launched by this call */
} svs_ba_stats;

/* Replaces: constructing g2o::SparseOptimizer + BlockSolver_6_3 + LinearSolverCSparse +
 * OptimizationAlgorithmLevenberg in SlamGraph::setupG2o (slam_graph.cpp:1063-1080). */
int svs_ba_create(const svs_ba_opts *opts, svs_ba **out);
void svs_ba_destroy(svs_ba *h);
const char *svs_last_error(const svs_ba *h);

/* Replaces SlamGraph::copyDataToG2o (slam_graph.cpp:985-1032) and the vertex/edge builders
 * addPoseToG2o / addPointToG2o / addObsToG2o / addConstraintToG2o
 * (slam_graph.cpp:907-920, slam_graph-impl.cpp:29-126).
 *   T_qt[P][7], fixed[P] (may be NULL = none fixed), psi[L][3]
 *   e_point/e_pose/e_anchor[E]: vertex 0/1/2 of each G2oEdgeProjectPSI2UVU as indices into the
 *     arrays above; all edges of a point must share one anchor (Point::anchorframe_id);
 *   e_obs[E][3] = (u, v, u_right); e_info_diag[E][3] = diagonal of Lambda
 *   c_i/c_j[C]: vertex 0/1 of each G2oEdgeSE3; c_T_ji[C][7] = measurement T_2_from_1;
 *   c_Lambda[C][36] row-major information.
 * Host buffers; copied to the device before the call returns.  Also performs the symbolic
 * analysis g2o does in BlockSolver::buildStructure + CSparse's symbolic phase. */
int svs_ba_set_problem(svs_ba *h, int P, const double *T_qt, const unsigned char *fixed,
                       int L, const double *psi,
                       int E, const int *e_point, const int *e_pose, const int *e_anchor,
                       const double *e_obs, const double *e_info_diag,
                       int C, const int *c_i, const int *c_j, const double *c_T_ji,
                       const double *c_Lambda, const svs_cam *cam);

/* Replaces optimizer.initializeOptimization(); lm->setUserLambdaInit(lambda);
 * optimizer.optimize(num_iters) (slam_graph.cpp:336-346) with RobustKernelHuber(delta) on the
 * observation edges when `robust` (slam_graph-impl.cpp:86-90; the reference leaves delta = 1).
 * All iterations run on the device.  Returns g2o's value: iterations performed, -1 if the
 * problem is empty; <= -100 encodes an SVS_ERR_* as (-100 + err). */
int svs_ba_optimize(svs_ba *h, int num_iters, int robust, double huber_delta,
                    double lambda_init, int max_trials, svs_ba_stats *stats);

/* Replaces SlamGraph::restoreDataFromG2o (slam_graph.cpp:1037-1058); psi is returned in
 * inverse-depth form, xyz_anchor = invert_depth(psi). */
int svs_ba_get_poses(svs_ba *h, double *T_qt);
int svs_ba_get_points(svs_ba *h, double *psi);

/* Restore the state uploaded by set_problem (device-to-device; for repeated measurement). */
int svs_ba_reset_state(svs_ba *h);

/* SlamGraph::optimize(const OptParams&) in one call from host buffers
 * (north-star name; slam_graph.cpp:319-355): set_problem + optimize + get_*.
 * T_qt and psi are updated in place. */
int svs_optimiseInnerAndOuterWindow(svs_ba *h, int P, double *T_qt, const unsigned char *fixed,
                                    int L, double *psi,
                                    int E, const int *e_point, const int *e_pose, const int *e_anchor,
                                    const double *e_obs, const double *e_info_diag,
                                    int C, const int *c_i, const int *c_j, const double *c_T_ji,
                                    const double *c_Lambda, const svs_cam *cam,
                                    int num_iters, int robust, double huber_delta,
                                    svs_ba_stats *stats);

/* ---- one window split by landmarks across ranks (SURVEY.md 8e): every rank holds all poses, its
 * share of the landmarks and their edges; the reduced camera system is summed across ranks once per
 * Levenberg trial by the caller (ncclAllReduce / torch.distributed on the device buffers below), the
 * solve is replicated, back-substitution stays local.  Call order per trial:
 *   svs_ba_trial_build -> all-reduce(S, bp, bc) -> svs_ba_trial_solve -> all-reduce(totals) -> svs_ba_trial_decide */
/* Pose pairs that must be present in the block pattern of the reduced system although this rank
 * may hold no landmark coupling them (the whole window's pattern); call before svs_ba_set_problem.
 * A handle with a prescribed pattern adds no pose pairs of its own (its tracks with visibility drop-outs are
 * not completed with zero-weight edges), so that all handles of the window lay the system out identically;
 * npairs = 0 takes the prescription back. */
int svs_ba_set_structure(svs_ba *h, int npairs, const int *pose_i, const int *pose_j);
/* lm->setUserLambdaInit(lambda); ni = 2 (slam_graph.cpp:338-342) */
int svs_ba_lm_begin(svs_ba *h, double lambda_init, int max_trials);
int svs_ba_trial_build(svs_ba *h, int robust, double huber_delta);
/* Device pointers: S (nS doubles), bp and bc (nb doubles each), totals (3 doubles: chi2 at the
 * accepted state, chi2 at the trial state, sum dpsi (lambda dpsi + b_l) of this rank's landmarks). */
int svs_ba_system_buffers(svs_ba *h, double **S, long long *nS, double **bp, double **bc, long long *nb,
                          double **totals);
int svs_ba_trial_solve(svs_ba *h, int robust, double huber_delta);
int svs_ba_trial_decide(svs_ba *h, int *again, int *stop, int *iterations_done);
int svs_ba_lm_stats(svs_ba *h, svs_ba_stats *stats);

/* The same sharding driven INSIDE the library (one process per GPU): after svs_ba_comm_init the handle
 * owns an NCCL communicator, svs_ba_set_problem_sharded takes the WHOLE window on every rank and keeps
 * landmarks l with l % nranks == rank (poses replicated, pose-pose edges on rank 0, block pattern of the
 * whole window), and svs_ba_optimize runs every Levenberg trial as
 *   fused build -> ncclAllReduce(S | bp | bc, one packed buffer) -> replicated solve -> local
 *   back-substitution -> ncclAllReduce(3 scalars) -> identical decision on every rank
 * on the handle's stream without a host synchronisation in between (SlamGraph::optimize,
 * slam_graph.cpp:319-355, on a window too large for one GPU's latency budget).  Only a problem loaded by
 * svs_ba_set_problem_sharded is summed across ranks: a whole window loaded into the same handle by
 * svs_ba_set_problem, svs_optimiseInnerAndOuterWindow or svs_ba_set_problem_from_map is solved by this rank alone.
 *   svs_comm_unique_id: rank 0 creates the 128-byte rendezvous id; the caller broadcasts it (MPI,
 *   torch.distributed, a socket).  NCCL is bound at run time (libnccl.so.2); SVS_ERR_STATE without it. */
int svs_comm_unique_id(char id[128]);
int svs_ba_comm_init(svs_ba *h, int nranks, int rank, const char id[128]);
int svs_ba_set_problem_sharded(svs_ba *h, int P, const double *T_qt, const unsigned char *fixed,
                               int L, const double *psi,
                               int E, const int *e_point, const int *e_pose, const int *e_anchor,
                               const double *e_obs, const double *e_info_diag,
                               int C, const int *c_i, const int *c_j, const double *c_T_ji,
                               const double *c_Lambda, const svs_cam *cam);
/* restoreDataFromG2o (slam_graph.cpp:1037-1058) for a sharded window: psi[L][3] of the WHOLE window on
 * every rank (svs_ba_get_points fills only this rank's landmarks of the same full-size array). */
int svs_ba_get_points_all(svs_ba *h, double *psi);

/* Inspection hooks used by the parity tests (device results copied to host buffers). */
/* g2o SparseOptimizer::activeRobustChi2 at the current state. */
int svs_ba_chi2(svs_ba *h, int robust, double huber_delta, double *chi2);
/* Reduced camera system the fused kernel produces at the current state:
 * S dense (6P x 6P row-major, symmetric, lambda included), bs (6P).  BlockSolver::solve
 * Schur part (g2o) on the system of BlockSolver::buildSystem. */
int svs_ba_reduced_system(svs_ba *h, int robust, double huber_delta, double lambda,
                          double *S_dense, double *bs, double *chi2);
/* Solve the reduced system once: x (6P) = S^-1 bs with the device block Cholesky
 * (LinearSolverCSparse::solve, slam_graph.cpp:55-60).  Returns 1 if not positive definite. */
int svs_ba_solve_reduced(svs_ba *h, int robust, double huber_delta, double lambda, double *x);

/* ------------------------------------------------------------------ FAST grid detector */

typedef struct svs_fast svs_fast;

/* FastGridCell (keyframes.h:30-43): cv::Range urange [u0,u1), vrange [v0,v1), fast_thr */
typedef struct {
  int u0, u1, v0, v1, thr;
} svs_fast_cell;

/* Private members of FastGrid (fast_grid.h:52-63) */
typedef struct {
  int grid_w, grid_h, fast_min, fast_max;
  int min_inner, min_outer, max_inner, max_outer;
} svs_fast_grid_params;

int svs_fast_create(int device, int max_w, int max_h, int max_keypoints, svs_fast **out);
void svs_fast_destroy(svs_fast *h);
const char *svs_fast_last_error(const svs_fast *h);

/* FastGrid::FastGrid (fast_grid.cpp:23-58): fills the band limits and grid_w*grid_h cells. */
int svs_fast_grid_init(int img_w, int img_h, int num_features_per_cell, int boundary_per_cell, int fast_thr,
                       int grid_w, int grid_h, int fast_min, int fast_max, svs_fast_grid_params *grid,
                       svs_fast_cell *cells);

/* The uint8 pyramid level the detector runs on (cv::Mat img of FastGrid::detect*).  Host buffer
 * (copied H2D) or a device buffer already resident (copied D2D into the handle's pitched image). */
int svs_fast_set_image(svs_fast *h, const unsigned char *img, int pitch, int w, int height);
int svs_fast_set_image_device(svs_fast *h, const unsigned char *d_img, int pitch, int w, int height);

/* FastGrid::detect (fast_grid.cpp:60-83): cv::FastFeatureDetector(cell.thr, false) on every cell
 * ROI.  out_xy[n][2] = (x + u0, y + v0) grouped by cell in list order, raster order inside a cell,
 * so the reference's quadtree content (index within the cell) is i - cell_off[c].
 * cell_off[ncells + 1].  Returns the total number of keypoints (may exceed max_out; only
 * max_out are written) or a negative SVS_ERR_*. */
int svs_fast_detect(svs_fast *h, const svs_fast_cell *cells, int ncells, int *out_xy, int max_out, int *cell_off);

/* FastGrid::detectAdaptively (fast_grid.cpp:86-152): up to `trials` re-detections per cell with
 * the threshold walk of the reference (state shared along a grid row); cells[].thr is updated in
 * place like FastGrid::cell_grid2d_. */
int svs_fast_detect_adaptively(svs_fast *h, const svs_fast_grid_params *grid, svs_fast_cell *cells, int trials,
                               int *out_xy, int max_out, int *cell_off);

/* ------------------------------------------------------------------ dense photometric tracker */

typedef struct svs_dt svs_dt;

#define SVS_DT_MAX_LEVELS 8
/* Bilinear taps with exact float weights instead of the texture unit's 8-fractional-bit weights
 * (the reference binds the images as linearly filtered textures, gpu/dense_tracking.cu:285-287). */
#define SVS_DT_EXACT_BILINEAR 1

typedef struct {
  double chi2[SVS_DT_MAX_LEVELS];   /* final photometric chi2 per level */
  int passes[SVS_DT_MAX_LEVELS];    /* fused (chi2 + J^T J + J^T r) pixel passes per level */
  int launches;
  float ms_total;
} svs_dt_stats;

/* Replaces GpuTracker::GpuTracker (gpu/dense_tracking.cu:265-299) + the GpuMat members of
 * DenseTracker / FrameData: device images for `nlevels` pyramid levels of a w0 x h0 frame. */
int svs_dt_create(int device, int w0, int h0, int nlevels, int flags, svs_dt **out);
void svs_dt_destroy(svs_dt *h);
const char *svs_dt_last_error(const svs_dt *h);

/* GpuIntrinsics::set (gpu/dense_tracking.cuh:28-41) of level l (cam_vec[l], dense_tracking.cpp:82-84) */
int svs_dt_set_intrinsics(svs_dt *h, int level, float focal_length, float px, float py);
/* The float images GpuTracker::bindTexture / jacobianReduction take (dense_tracking.cpp:88-104):
 * previous-frame intensity, current intensity and its x/y derivatives; host buffers with
 * `stride_floats` floats per row; NULL keeps the resident plane. */
int svs_dt_set_images(svs_dt *h, int level, const float *prev, const float *cur, const float *dx,
                      const float *dy, int stride_floats);
/* frame_data_.gpu_disp_32f (level-0 disparity) for computePointCloud */
int svs_dt_set_disparity(svs_dt *h, const float *disp, int stride_floats, int w, int height);
/* DenseTracker::computeDensePointCloudGpu (dense_tracking.cpp:195-216): cams[nlevels] are the
 * per-level StereoCamera parameters (frame_grabber-impl.cpp:50-59). */
int svs_dt_compute_point_cloud(svs_dt *h, const double T_cur_from_actkey[7], const svs_cam *cams);
/* dev_ref_dense_points_[level] as packed float4 (w*h*4 floats) */
int svs_dt_set_point_cloud(svs_dt *h, int level, const float *cloud_xyzw);
int svs_dt_get_point_cloud(svs_dt *h, int level, float *cloud_xyzw);
/* GpuTracker::chi2 (gpu/dense_tracking.cu:455-491) */
int svs_dt_chi2(svs_dt *h, int level, const double T_cur_from_prev[7], double *chi2);
/* GpuTracker::jacobianReduction (gpu/dense_tracking.cu:318-356): Hessian in GpuSymMatrix6 packing
 * (21 values: for r: for c <= r), jacobian_times_res (6) */
int svs_dt_jacobian_reduction(svs_dt *h, int level, const double T_cur_from_prev[7], double H21[21],
                              double b6[6], double *chi2);
/* GpuTracker::residualImage (gpu/dense_tracking.cu:494-567; called once per level at the end of
 * denseTrackingGpu, dense_tracking.cpp:180-188): res_rgba = w*h packed float4 -- grey max(0, 1 - 50 r^2) where the
 * pixel contributes, (1,0,0,1) where it projects outside the frame, (0,1,0,1) where it has no depth */
int svs_dt_residual_image(svs_dt *h, int level, const double T_cur_from_prev[7], float *res_rgba);
/* DenseTracker::denseTrackingGpu (dense_tracking.cpp:62-193): coarse-to-fine LM, T updated in place */
int svs_dt_track(svs_dt *h, double T_cur_from_actkey[7], svs_dt_stats *stats);

/* ---- the tracker the reference builds WITHOUT SCAVISLAM_CUDA_SUPPORT (SURVEY.md 8 row a18):
 * DenseTracker::denseTrackingCpu / computeDensePointCloudCpu (dense_tracking.cpp:222-423): every 4th pixel,
 * previous intensity from the uint8 pyramid, residual clamped to +-0.1, exact software bilinear taps, FP64
 * point transform, border test isInFrame(uv, 2), disparity scaled by 2^-level, H not damped.  Level sizes
 * must be multiples of 4 (the reference asserts the same).  Pixel sums are FP64 (reference: sequential FP32). */
typedef struct svs_dtc svs_dtc;
int svs_dtc_create(int device, int w0, int h0, int nlevels, svs_dtc **out);
void svs_dtc_destroy(svs_dtc *h);
const char *svs_dtc_last_error(const svs_dtc *h);
/* frame_data_.prev_left().pyr_uint8[level]; on_device != 0: img is a device pointer (e.g. svs_prep_level) */
int svs_dtc_set_prev_u8(svs_dtc *h, int level, const unsigned char *img, int pitch, int on_device);
/* frame_data_.pyr_float32 / pyr_float32_dx / pyr_float32_dy [level]; NULL planes are left as they are */
int svs_dtc_set_cur(svs_dtc *h, int level, const float *cur, const float *dx, const float *dy, int stride_floats,
                    int on_device);
/* frame_data_.disp (level-0 float disparity, host) */
int svs_dtc_set_disparity(svs_dtc *h, const float *disp, int stride_floats);
/* computeDensePointCloudCpu(T_cur_from_actkey) with cam_vec[level] = cams[level] */
int svs_computeDensePointCloudCpu(svs_dtc *h, const double T_cur_from_actkey[7], const svs_cam *cams);
/* ref_dense_points_[level]: (h/4) x (w/4) float4, tightly packed */
int svs_dtc_get_point_cloud(svs_dtc *h, int level, float *cloud_xyzw);
int svs_dtc_set_point_cloud(svs_dtc *h, int level, const float *cloud_xyzw);
/* denseTrackingCpu(&T_cur_from_actkey): coarse-to-fine, T updated in place */
int svs_denseTrackingCpu(svs_dtc *h, const svs_cam *cams, double T_cur_from_actkey[7], svs_dt_stats *stats);

/* ------------------------------------------------------------------ guided patch matcher */

typedef struct svs_matcher svs_matcher;
#define SVS_MATCH_MAX_LEVELS 4

/* cam_vec[level] (LinearCamera part of StereoCamera): image size, focal length, principal point */
typedef struct {
  int w, h;
  double f, px, py;
} svs_match_level;

/* CandidatePoint<3> (data_structures.h): anchor keyframe (slot given to svs_matcher_set_keyframe,
 * -1 = not in vertex_map), xyz in the anchor frame, its (u, v) observation at anchor_level */
typedef struct {
  int keyframe;
  int anchor_level;
  double xyz_anchor[3];
  double anchor_obs_pyr[2];
} svs_match_point;

/* One entry per candidate point, in input order.  matched == 1 entries, in order, are what the
 * reference appends to TrackData::obs_list / point_list / ba2globalptr. */
typedef struct {
  int predicted;       /* computePrediction succeeded */
  int textured;        /* key patch passed the thr_std test */
  int matched;         /* a candidate beat thr_mean and the disparity is valid */
  int n_candidates;    /* FAST corners inside the search window */
  int index;           /* quadtree content of the best candidate, -1 = none */
  int min_dist;        /* its score (literal formula of matcher.cpp:73) */
  int uv_pyr[2];       /* its position at anchor_level */
  double obs[3];       /* (u, v, u_right) at level 0 */
  double xyz_actkey[3];
} svs_match_result;

int svs_matcher_create(int device, int nlevels, const svs_match_level *levels, int max_keyframes, int max_points,
                     int max_keypoints, svs_matcher **out);
void svs_matcher_destroy(svs_matcher *h);
const char *svs_matcher_last_error(const svs_matcher *h);
/* keyframe_map[id].pyr + vertex_map[id].T_me_from_w for one anchor keyframe (uint8 pyramid, host) */
int svs_matcher_set_keyframe(svs_matcher *h, int slot, const double T_me_from_w[7], const unsigned char *const *pyr,
                           const int *pitch);
/* cur_frame.pyr + cur_frame.disp (level-0 float disparity); either may be NULL to keep what is loaded */
int svs_matcher_set_current(svs_matcher *h, const unsigned char *const *pyr, const int *pitch, const float *disp,
                          int disp_pitch_floats);
/* feature_tree.at(level): the FAST corners (x, y) and their quadtree content (index within the cell) */
int svs_matcher_set_features(svs_matcher *h, int level, const int *xy, const int *content, int n);
/* The same from the FAST handle's last svs_fast_detect* result where it lies on the device (content = ordinal of the
 * corner inside its cell, fast_grid.cpp:75-80): the corners never travel through host memory. */
int svs_matcher_set_features_from_fast(svs_matcher *h, int level, svs_fast *fast);
/* GuidedMatcher<StereoCamera>::match (matcher.cpp:312-398).  T_actkey_from_w replaces
 * vertex_map[actkey_id].  Returns the number of matched points or a negative SVS_ERR_*. */
int svs_match(svs_matcher *h, const double T_cur_from_actkey[7], const double T_actkey_from_w[7],
              const svs_match_point *pts, int n, int search_radius, int thr_mean, int thr_std,
              svs_match_result *out);

/* ------------------------------------------------------------------ frame preprocessing ("next" row, SURVEY 8f) */

typedef struct svs_prep svs_prep;
/* FrameGrabber::preprocessing (frame_grabber.cpp:287-336): uint8 pyramid (cv::buildPyramid), float
 * image / 255, float pyramid (cv::gpu::pyrDown), x/y derivatives ([-1 0 1], replicated border,
 * frame_grabber.cpp:104-115) for `nlevels` levels; everything stays on the device. */
int svs_prep_create(int device, int w, int height, int nlevels, svs_prep **out);
void svs_prep_destroy(svs_prep *h);
const char *svs_prep_last_error(const svs_prep *h);
int svs_prep_process(svs_prep *h, const unsigned char *img, int pitch);
/* device pointers of one level (any output pointer may be NULL) */
int svs_prep_level(svs_prep *h, int level, int *w, int *height, const unsigned char **u8, int *pitch_u8,
                   const float **f32, const float **dx, const float **dy, int *stride_f32);
int svs_prep_get_u8(svs_prep *h, int level, unsigned char *out);          /* tightly packed w*h */
int svs_prep_get_f32(svs_prep *h, int level, int which, float *out);      /* which: 0 image, 1 dx, 2 dy */
/* device-to-device hand-over into the consumers */
int svs_dt_set_images_device(svs_dt *h, int level, const float *prev, const float *cur, const float *dx,
                             const float *dy, int stride_floats);
int svs_dt_swap_prev_cur(svs_dt *h);
int svs_matcher_set_pyramid_device(svs_matcher *h, int which, const double T_me_from_w[7],
                                   const unsigned char *const *d_pyr, const int *pitch);

/* ------------------------------------------------------------------ motion-only pose refinement
 * ("next" row, SURVEY.md 8f-1).  BA_SE3_XYZ_STEREO::calcFastMotionOnly (pose_optimizer.h:135-298) with
 * SE3XYZ_STEREO (transformations.h:414-460): 6-DoF Levenberg-Marquardt over fixed 3-D points with the
 * pseudo-Huber reweighting; callers stereo_frontend.cpp:1058, backend.cpp:754-779. */

typedef struct svs_pose svs_pose;

/* PoseOptimizerParams (pose_optimizer.h:38-58); SVS_POSE_PARAMS_DEFAULT mirrors its constructor */
typedef struct {
  int robust_kernel;
  double kernel_param;
  int num_iter;
  double initial_mu;   /* -1: tau * max diag(J^T J) */
  double tau;
} svs_pose_params;
#define SVS_POSE_PARAMS_DEFAULT {1, 1.0, 50, -1.0, 0.00001}

/* OptimizerStatistics (pose_optimizer.h:60-98) + counters */
typedef struct {
  double initial_chi2, chi2, max_err;
  int num_obs;
  int iterations;   /* accepted steps */
  int trials;       /* 6x6 solves */
  float ms;         /* device time of the LM kernel */
} svs_pose_stats;

int svs_pose_create(int device, int max_obs, svs_pose **out);
void svs_pose_destroy(svs_pose *h);
const char *svs_pose_last_error(const svs_pose *h);
/* obs_list as (point_id, obs = (u, v, u_right)) arrays, point_list as xyz[3 * npoints]; T_frame in/out.
 * Returns SVS_OK or a negative SVS_ERR_* (SVS_ERR_NUMERIC where the reference throws). */
int svs_calcFastMotionOnly(svs_pose *h, int n, const int *obs_point_id, const double *obs_uvu, int npoints,
                           const double *point_xyz, const svs_cam *cam, const svs_pose_params *params,
                           double T_frame[7], svs_pose_stats *stats);
/* Same, on the TrackData of the last svs_match(m, ...) where it lies on the device (matched entries'
 * obs / xyz_actkey): no host trip between matching and pose refinement. */
int svs_calcFastMotionOnly_matched(svs_pose *h, svs_matcher *m, const svs_cam *cam, const svs_pose_params *params,
                                   double T_frame[7], svs_pose_stats *stats);

/* ------------------------------------------------------------------ pose-pose constraint weights
 * ("next" row, SURVEY.md 8f-4).  SlamGraph::computeConstraint (slam_graph.cpp:785-846) for a batch of pose
 * pairs: T_1_from_2 = T_1 T_2^-1, n = number of points in both feature tables, median distance of those
 * points in frame 1, Lambda = n diag((350 |t_12| / median)^2 I3, 100^2 I3) (row-major 6x6).
 * Inputs: T_me_from_world[P][7]; the feature_table keys of every pose as CSR (feat_ptr[P+1], feat_point,
 * strictly ascending per pose); for every point the index of its anchor pose and xyz_anchor.  Anchor frames
 * outside the double window (computeAbsolutePose in the reference) are passed like any other pose.
 * A pair without shared points gets Lambda = 0 and visibility_strength = 0 (the reference calls median() of an empty
 * multiset there: undefined).  median(): VisionTools is not vendored with the reference, so its rule for an EVEN
 * number of shared points is an assumption written down here -- the mean of the two middle depths (odd n: the middle
 * one); constraint_oracle.c and csrc/constraint.cu both implement exactly this. */
typedef struct svs_constraints svs_constraints;
int svs_constraints_create(int device, svs_constraints **out);
void svs_constraints_destroy(svs_constraints *h);
const char *svs_constraints_last_error(const svs_constraints *h);
int svs_computeConstraint_batch(svs_constraints *h, int P, const double *T_me_from_world, const int *feat_ptr,
                                const int *feat_point, int L, const int *point_anchor, const double *xyz_anchor,
                                int npairs, const int *v1, const int *v2, double *T_1_from_2, double *Lambda,
                                int *visibility_strength);

/* ------------------------------------------------------------------ device-resident map and window assembly
 * ("next" row, SURVEY.md 8f-3).  The part of SlamGraph the optimiser reads (slam_graph.hpp:65-137) kept in device
 * memory -- vertices with T_me_from_world, points with anchorframe_id / xyz_anchor, observations as CSR per point
 * (vis_set order: vertex, feature centre (u, v, u_right) at level 0, pyramid level) -- and copyDataToG2o /
 * copyPosesToG2o / addPointToG2o / addObsToG2o (slam_graph.cpp:907-1032) as kernels: for the double window
 * `window_vertex` (BA pose i = vertex window_vertex[i]) and the active points (BA point l = map point
 * active_point[l]) every observation whose frame is in the window becomes an edge, in the reference's order;
 * psi = invert_depth(xyz_anchor), Lambda = diag(s, s, 0.333^2) with s = (2^-level)^2.  Observations and weights
 * never leave the device; only the index triples return to the host for the structure analysis.
 * Pose-pose constraints are passed as for svs_ba_set_problem (indices into the window). */
typedef struct svs_map svs_map;
int svs_map_create(int device, svs_map **out);
void svs_map_destroy(svs_map *h);
const char *svs_map_last_error(const svs_map *h);
int svs_map_set(svs_map *h, int V, const double *T_me_from_world, int Np, const int *point_anchor,
                const double *xyz_anchor, const int *vis_ptr, const int *vis_pose, const double *feat_center,
                const int *feat_level);
/* restoreDataFromG2o's counterpart for the map: overwrite the poses of n vertices */
int svs_map_update_poses(svs_map *h, int n, const int *vertex, const double *T_me_from_world);
/* ... and the anchored positions of n points (restoreDataFromG2o writes Point::xyz_anchor, slam_graph.cpp:1054) */
int svs_map_update_points(svs_map *h, int n, const int *point, const double *xyz_anchor);
/* read the map back (either output may be NULL): T_me_from_world[V][7], xyz_anchor[Np][3] */
int svs_map_get(svs_map *h, double *T_me_from_world, double *xyz_anchor);
/* SlamGraph::restoreDataFromG2o (slam_graph.cpp:1037-1058) device to device: after svs_ba_optimize on the window
 * svs_ba_set_problem_from_map assembled last, the vertex poses and xyz_anchor = invert_depth(psi) of its points go
 * back into the map without touching the host */
int svs_map_absorb(svs_map *h, svs_ba *ba);
/* = svs_ba_set_problem on the window assembled from the map; *num_edges receives E */
int svs_ba_set_problem_from_map(svs_ba *ba, svs_map *map, int P, const int *window_vertex, const unsigned char *fixed,
                                int L, const int *active_point, int C, const int *c_i, const int *c_j,
                                const double *c_T_ji, const double *c_Lambda, const svs_cam *cam, int *num_edges);
/* The pose graph of the map: for every vertex its neighbours in the order SlamGraph::computeInitialDoubleWin pushes them
 * (Vertex::neighbor_ids_ordered_by_strength from the strongest, slam_graph.cpp:584-590; an entry in either direction is a
 * direct edge of edge_table_), and per directed entry the marginalised constraint copyContraintsToG2o reads
 * (T_nbr_from_me as qx qy qz qw tx ty tz, Lambda 6x6 row-major; both NULL when the caller brings its own constraints).
 * To be called again after svs_map_set / svs_map_add_keyframe. */
int svs_map_set_graph(svs_map *h, const int *nbr_ptr, const int *nbr_id, const double *nbr_T, const double *nbr_Lambda);
/* SlamGraph::computeInitialDoubleWin + computeActivePointsAndExtendOuterWindow (slam_graph.cpp:556-663) and the pair
 * selection of copyContraintsToG2o (:938-981) on the device tables.  Returns the double window in ascending vertex order
 * (the order of the reference's std::map; inner[i] = 1 for INNER frames; frames added by the outer-window extension are
 * OUTER), the active points in ascending order, and -- when c_i is not NULL -- the constraints between window frames of
 * which at least one is OUTER, as (c_i, c_j, T_j_from_i, Lambda) with c_i / c_j positions in window_vertex, ordered by
 * (vertex i, vertex j).  The outputs feed svs_ba_set_problem_from_map unchanged.  SVS_ERR_INVALID if a capacity is too
 * small (*P, *L, *C then hold the required sizes). */
int svs_map_select_window(svs_map *h, int root, int inner_window_size, int double_window_size, int cap_P, int *P,
                          int *window_vertex, unsigned char *inner, int cap_L, int *L, int *active_point, int cap_C, int *C,
                          int *c_i, int *c_j, double *c_T_ji, double *c_Lambda);
/* SlamGraph::addKeyframe (slam_graph.cpp:144-186) with addNewPointsToMap / addNewObsToOldPoints (:359-421) on the device
 * tables: one new vertex with T_me_from_world = T_newkey_from_oldkey * T_oldkey_from_world (composed where the map lies,
 * so a pose absorbed from the optimiser never visits the host); n_new points, each anchored in an EXISTING frame and seen
 * by that frame (new_anchor_center at level 0, new_anchor_level) and by the new keyframe (new_center, new_level); n_track
 * existing points gain an observation by the new keyframe.  The observation lists are rebuilt by kernels (count, scan,
 * move); the strength bookkeeping of computeStrength / addNewEdges stays with the caller, who passes the new pose graph
 * with svs_map_set_graph.  *vertex_index = index of the new vertex, *first_new_point = index of the first new point. */
int svs_map_add_keyframe(svs_map *h, int oldkey, const double *T_newkey_from_oldkey, int n_new, const int *new_anchor,
                         const double *new_xyz_anchor, const double *new_anchor_center, const int *new_anchor_level,
                         const double *new_center, const int *new_level, int n_track, const int *track_point,
                         const double *track_center, const int *track_level, int *vertex_index, int *first_new_point);
/* the edge list of the last assembly (any output may be NULL); E must equal *num_edges */
int svs_map_last_edges(svs_map *h, int E, int *e_point, int *e_pose, int *e_anchor, double *e_obs, double *e_info);

/* Library/device info: writes "name;sm;SMs;..." into buf. */
int svs_device_info(char *buf, int buflen);

#ifdef __cplusplus
}
#endif
#endif /* SVS_B200_H */
