/*
 * ba_cuda.h -- C ABI of the B200-native bundle-adjustment hot path.
 *
 * This is the drop-in boundary that replaces the reference's use of the Ceres
 * public API on its one hot path (all citations relative to the reference tree):
 *
 *   ceres::Problem problem;                       Main_Calibration/bundle_adjustment_manager.cpp:19
 *   problem.AddResidualBlock(cost, NULL, ...)     bundle_adjustment_manager.cpp:37,50,67,81
 *                                                 Test1_BundleAdjustment/main.cpp:76-79
 *                                                 Test2_BundleAdjustment/main.cpp:75-78,90-94
 *   Solver::Options{DENSE_SCHUR, progress}        bundle_adjustment_manager.cpp:90-92
 *   ceres::Solve(options, &problem, &summary)     bundle_adjustment_manager.cpp:94
 *   summary.FullReport()                          bundle_adjustment_manager.cpp:95
 *   cv::projectPoints + error sum                 Main_Calibration/reprojection_check.cpp:69,81,100-101
 *
 * Conventions: every function returns 0 (BA_OK) or a negative ba_status; no
 * exceptions and no exit() cross this boundary.  All host pointers are borrowed
 * only for the duration of the call (the library copies / re-lays-out into HBM),
 * unlike Ceres which optimises caller memory in place: the host calls
 * ba_cuda_get_parameters() after ba_cuda_solve() to see the "in place" result.
 * Indices are int32, counts int64, arithmetic fp64.  One host thread drives one
 * ba_cuda_problem; one ba_cuda_problem is bound to one GPU.  There is NO CPU
 * fallback in this library: without a CUDA device ba_cuda_create() fails.
 *
 * Multi-GPU: one process (rank) per GPU.  Every rank holds ALL f-blocks
 * (cameras / markers) and a SHARD of the eliminated blocks (Model A: points with
 * all their observations; Model B: frames with all their marker observations).
 * ba_cuda_comm_init() joins the ranks through NCCL; ba_cuda_solve() is then a
 * collective call (partial reduced camera systems are summed with one
 * ncclAllReduce per linear solve, scalars with a second small one).
 */
#ifndef BA_CUDA_H_
#define BA_CUDA_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct ba_cuda_problem ba_cuda_problem; /* opaque */

typedef enum ba_status {
  BA_OK = 0,
  BA_ERR_INVALID_ARGUMENT = -1,
  BA_ERR_CUDA = -2,          /* CUDA runtime error, see ba_cuda_last_error() */
  BA_ERR_STATE = -3,         /* call order (e.g. solve before set_model_*) */
  BA_ERR_NCCL = -4,
  BA_ERR_OUT_OF_MEMORY = -5,
  BA_ERR_NO_DEVICE = -6,
  BA_ERR_UNSUPPORTED = -7,
  BA_ERR_RANK_DEFICIENT = -8  /* ba_cuda_covariance: the normal equations at x are singular */
} ba_status;

/* How the reduced camera system (RCS) is solved; replaces
 * options.linear_solver_type = DENSE_SCHUR (bundle_adjustment_manager.cpp:91). */
typedef enum ba_rcs_solver {
  BA_RCS_AUTO = 0,            /* dense Cholesky while the RCS is rig sized, PCG above */
  BA_RCS_DENSE_CHOLESKY = 1,  /* == Ceres DENSE_SCHUR */
  BA_RCS_PCG = 2              /* block-Jacobi PCG on the explicit block-sparse RCS
                                 (Ceres ITERATIVE_SCHUR / SCHUR_JACOBI stopping rule) */
} ba_rcs_solver;

/* Mirrors ceres::TerminationType as far as this path can produce it. */
typedef enum ba_termination {
  BA_CONVERGENCE = 0,
  BA_NO_CONVERGENCE = 1,
  BA_FAILURE = 2
} ba_termination;

typedef enum ba_termination_reason {
  BA_REASON_NONE = 0,
  BA_REASON_GRADIENT_TOLERANCE = 1,
  BA_REASON_PARAMETER_TOLERANCE = 2,
  BA_REASON_FUNCTION_TOLERANCE = 3,
  BA_REASON_MIN_TRUST_REGION_RADIUS = 4,
  BA_REASON_MAX_ITERATIONS = 5,
  BA_REASON_TOO_MANY_INVALID_STEPS = 6,
  BA_REASON_INITIAL_EVALUATION_FAILED = 7
} ba_termination_reason;

/* The Ceres 1.14 Solver::Options fields the trust-region LM path reads; the
 * defaults written by ba_cuda_options_init() are Ceres 1.14's (SURVEY.md 5.9). */
typedef struct ba_cuda_options {
  int32_t max_num_iterations;                /* 50 */
  int32_t max_num_consecutive_invalid_steps; /* 5 */
  int32_t jacobi_scaling;                    /* 1 */
  int32_t rcs_solver;                        /* ba_rcs_solver, BA_RCS_AUTO */
  int32_t pcg_max_iterations;                /* 500  (max_linear_solver_iterations) */
  int32_t pcg_min_iterations;                /* 0 */
  int32_t pcg_residual_reset_period;         /* 10 */
  int32_t minimizer_progress_to_stdout;      /* 0 */
  int32_t profile_kernels;                   /* 0; 1 = CUDA-event timing of every kernel family member
                                                (ba_cuda_get_kernel_stats), costs ~2 us of host time per launch */
  int32_t force_generic_path;                /* 0; 1 = Model A through the generic materialised-Jacobian pipeline
                                                (the one Model B uses) instead of the fused tile kernels: A/B testing */
  double initial_trust_region_radius;        /* 1e4 */
  double max_trust_region_radius;            /* 1e16 */
  double min_trust_region_radius;            /* 1e-32 */
  double min_relative_decrease;              /* 1e-3 */
  double min_lm_diagonal;                    /* 1e-6 */
  double max_lm_diagonal;                    /* 1e32 */
  double function_tolerance;                 /* 1e-6 */
  double gradient_tolerance;                 /* 1e-10 */
  double parameter_tolerance;                /* 1e-8 */
  double pcg_eta;                            /* 1e-1 (q_tolerance) */
  double pcg_r_tolerance;                    /* -1 (disabled, as LevenbergMarquardtStrategy does) */
  /* Robust loss on every residual block (an observation of Model A: 2 residuals; a marker observation of Model B: 8).
   * The reference passes NULL to AddResidualBlock (bundle_adjustment_manager.cpp:38,51,68,82; Test1 main.cpp:77): BA_LOSS_NONE,
   * the default, reproduces it bit for bit.  Huber / Cauchy restate ceres::HuberLoss(a) / ceres::CauchyLoss(a) and Ceres'
   * Corrector: residuals and Jacobian rows of a block are scaled by sqrt(rho'(s)), s = |r|^2, the cost is sum rho(s) / 2. */
  int32_t loss_function;                     /* ba_loss, BA_LOSS_NONE */
  int32_t reserved_;
  double loss_scale;                         /* a, 1.0 */
} ba_cuda_options;

typedef enum ba_loss {
  BA_LOSS_NONE = 0,
  BA_LOSS_HUBER = 1,
  BA_LOSS_CAUCHY = 2
} ba_loss;

/* One row of Ceres' minimizer_progress_to_stdout table (IterationSummary). */
typedef struct ba_cuda_iteration {
  int32_t iteration;
  int32_t step_is_valid;
  int32_t step_is_successful;
  int32_t linear_solver_iterations;
  double cost;
  double cost_change;
  double gradient_max_norm;
  double gradient_norm;
  double step_norm;
  double relative_decrease;   /* tr_ratio */
  double trust_region_radius;
  double iteration_time_s;
} ba_cuda_iteration;

typedef struct ba_cuda_summary {
  int32_t termination_type;    /* ba_termination */
  int32_t termination_reason;  /* ba_termination_reason */
  int32_t num_iterations;      /* rows recorded, including row 0 */
  int32_t num_successful_steps;
  int32_t num_unsuccessful_steps;
  int32_t rcs_solver_used;     /* ba_rcs_solver actually run */
  int32_t rcs_dim;             /* scalar dimension of the reduced camera system */
  int32_t num_jacobian_evaluations;
  int32_t num_cost_evaluations;
  int32_t num_linear_solves;
  int64_t num_residuals;
  int64_t num_free_parameters;
  double initial_cost;
  double final_cost;
  double total_time_s;         /* host wall clock of ba_cuda_solve */
  /* device time per kernel family, CUDA events on the solve stream, milliseconds */
  double ms_jacobian;          /* K1 residual + Jacobian */
  double ms_schur;             /* K2 elimination + RCS assembly */
  double ms_rcs_solve;         /* K3 */
  double ms_update;            /* K4 back-substitution / model cost / candidate */
  double ms_cost;              /* K5-style cost-only evaluation */
  double ms_collective;        /* NCCL */
  int32_t path_used;           /* ba_path: which pipeline ran the LM loop */
  int32_t reserved_;
} ba_cuda_summary;

/* Which pipeline a solve ran on.  Model B and ba_cuda_eval always use the generic (materialised-Jacobian) pipeline.
 * Model A uses the fused two-pass pipeline when every point has at most 64 observations: pass 1 on strips of tiles
 * (register-resident Schur accumulators) when the cameras of a strip fit 64 table slots and no point is seen twice
 * by one camera, else on single tiles; a problem that fits neither falls back to the generic pipeline (about 3x
 * slower at BAL scale) -- the reason is printed once on stderr. */
typedef enum ba_path {
  BA_PATH_GENERIC = 0,
  BA_PATH_FUSED_TILES = 1,
  BA_PATH_FUSED_STRIPS = 2,
  BA_PATH_RIG = 3            /* rig-size problems: the whole trust-region loop in one launch of one CTA (ba_rig.cuh) */
} ba_path;

void ba_cuda_options_init(ba_cuda_options* options);

/* ---- lifetime -------------------------------------------------------------- */
int ba_cuda_create(ba_cuda_problem** out, int device_id);
void ba_cuda_destroy(ba_cuda_problem* p);
const char* ba_cuda_last_error(void); /* thread-local message of the last failure */
int ba_cuda_device_count(void);

/* Device buffers are recycled through a caching allocator (cudaMalloc / cudaFree cost milliseconds and synchronise
 * the device; rebuilding a problem reuses the previous buffers).  The cache is emptied when the last problem is
 * destroyed; this call empties it at once, e.g. before handing the GPU to another library. */
void ba_cuda_release_cached_memory(void);

/* All work of a problem is enqueued on one CUDA stream: by default a private non-blocking stream; a caller
 * that wants to order / time the work with its own events passes its cudaStream_t here (NULL restores the
 * private stream).  Must not be called while a solve is in flight. */
int ba_cuda_set_stream(ba_cuda_problem* p, void* cuda_stream);

/* Per-kernel accounting since the last ba_cuda_reset_stats(): number of launches of this library's own
 * kernels (always counted) and, with options.profile_kernels = 1, CUDA-event device time per kernel together
 * with the ALGORITHMIC bytes one launch has to move (DESIGN.md, "kernels and rooflines"). */
typedef struct ba_cuda_kernel_stat {
  char name[32];
  int64_t launches;
  double total_ms;                     /* 0 unless profile_kernels was set */
  double algorithmic_bytes_per_launch; /* compulsory HBM traffic of one launch on the current problem */
} ba_cuda_kernel_stat;
int ba_cuda_get_kernel_stats(ba_cuda_problem* p, ba_cuda_kernel_stat* stats, int cap); /* returns the count */
int64_t ba_cuda_num_launches(const ba_cuda_problem* p);
void ba_cuda_reset_stats(ba_cuda_problem* p);

/* ---- multi-GPU plumbing (NCCL; rendezvous bytes travel by the caller's own
 *      channel, e.g. torch.distributed broadcast) ------------------------------ */
#define BA_CUDA_UNIQUE_ID_BYTES 128
int ba_cuda_comm_unique_id(uint8_t id[BA_CUDA_UNIQUE_ID_BYTES]);
int ba_cuda_comm_init(ba_cuda_problem* p, int rank, int world_size,
                      const uint8_t id[BA_CUDA_UNIQUE_ID_BYTES]);
/* Deterministic shard map used by every host (C++ and Python): splits eliminated
 * blocks [0,n_blocks) into world_size contiguous ranges balanced by `weight`
 * (observations per block).  range_begin has world_size+1 entries. */
int ba_cuda_shard_blocks(int64_t n_blocks, const int64_t* weight, int world_size,
                         int64_t* range_begin);

/* ---- Model A: (camera 6-DoF angle-axis pose, free 3-D point), 2 residuals.
 *      Replaces ReprojectionError / AutoDiffCostFunction<...,2,6,3> and the
 *      AddResidualBlock loop, Test1_BundleAdjustment/bundle_adjustmenter.cpp:106-148,
 *      Test1_BundleAdjustment/main.cpp:67-80.
 *      cam_idx/pt_idx/obs_xy are exactly BALProblem::camera_index_/point_index_/
 *      observations_ (bundle_adjustmenter.cpp:66-77).  intr = fx,fy,ppx,ppy per
 *      camera; intr_stride = 4 for per-camera intrinsics or 0 when one set is
 *      shared by every observation (Test1 uses serial_numbers[1] for all,
 *      main.cpp:73-74).  Parameter layout == BALProblem::parameters_:
 *      [n_cam x 6 | n_pt x 3] (bundle_adjustmenter.cpp:33-41).  Blocks that no
 *      observation references are not part of the problem (as in Ceres). -------- */
int ba_cuda_set_model_a(ba_cuda_problem* p, int32_t n_cam, int64_t n_pt, int64_t n_obs,
                        const int32_t* cam_idx, const int32_t* pt_idx,
                        const double* obs_xy, const double* intr, int32_t intr_stride);

/* ---- Model B: 8-residual marker factor over (camera, per-frame base-marker
 *      pose, marker-in-rig pose).  Replaces the four functors of
 *      Main_Calibration/bundle_adjustment.h:56-343 and the dispatch of
 *      bundle_adjustment_manager.cpp:21-88 (fix_marker0 = 1), or the two functors
 *      and dispatch of Test2_BundleAdjustment/main.cpp:64-97 (fix_marker0 = 0).
 *      Camera 0 is never a parameter block (fix_cam0 must be 1, as in every
 *      reference program).  obs8 = BALProblem::observations_ (8 per marker
 *      observation, corner order TL,TR,BR,BL).  intr4_per_cam = fx,fy,ppx,ppy x
 *      n_cam.  Parameter layout == BALProblem::parameters_:
 *      [n_cam x 6 | n_time x 6 | n_marker x 6] (bundle_adjustment.cpp:155). ----- */
int ba_cuda_set_model_b(ba_cuda_problem* p, int32_t n_cam, int32_t n_time, int32_t n_marker,
                        int64_t n_mobs, const int32_t* time_idx, const int32_t* cam_idx,
                        const int32_t* marker_idx, const double* obs8,
                        const double* intr4_per_cam, double marker_side,
                        int32_t fix_cam0, int32_t fix_marker0);

int ba_cuda_set_parameters(ba_cuda_problem* p, const double* params, int64_t n);
int ba_cuda_get_parameters(ba_cuda_problem* p, double* params, int64_t n);
int64_t ba_cuda_num_parameters(const ba_cuda_problem* p);
/* Device-side snapshot / rollback of the whole parameter vector (no host traffic): the in-HBM analogue of a
 * caller keeping a copy of BALProblem::parameters_ to re-run ceres::Solve from the same start. */
int ba_cuda_save_parameters(ba_cuda_problem* p);
int ba_cuda_restore_parameters(ba_cuda_problem* p);

/* ---- the hot path: replaces ceres::Solve (bundle_adjustment_manager.cpp:94) -- */
int ba_cuda_solve(ba_cuda_problem* p, const ba_cuda_options* options, ba_cuda_summary* summary);
/* The same solve in three calls, so that a caller (bench.py, an interactive tool) can run the LM loop a few
 * iterations at a time: begin = TrustRegionMinimizer's IterationZero; iterate = up to max_new_iterations more
 * rows of the progress table (*finished = 1 once a termination rule fired); end = the summary.
 * ba_cuda_solve(p,o,s) == begin(p,o); iterate(p, INT32_MAX, &f); end(p,s). */
int ba_cuda_solve_begin(ba_cuda_problem* p, const ba_cuda_options* options);
int ba_cuda_solve_iterate(ba_cuda_problem* p, int32_t max_new_iterations, int32_t* finished);
int ba_cuda_solve_end(ba_cuda_problem* p, ba_cuda_summary* summary);
/* rows of the progress table; returns the number of rows available (>= 0) */
int ba_cuda_get_iterations(ba_cuda_problem* p, ba_cuda_iteration* rows, int cap);

/* k independent solves of this problem's structure in one launch, one CTA each (Monte Carlo runs under fresh corner
 * noise, multi-start against the planar-marker pose ambiguity).  The model, intrinsics, marker side and fixed-block dispatch
 * are the problem's; one `options` applies to every instance (NULL = ba_cuda_options_init defaults; the loss is validated as
 * ba_cuda_solve_begin validates it).  Arguments:
 *   params        k x n_params, caller layout of ba_cuda_set_parameters: instance i starts from params + i n_params and
 *                 its solution is written there.  Blocks that are not parameters or that no observation references come
 *                 back as given.
 *   observations  NULL (every instance uses the model's own observations) or k x (2 n_obs | 8 n_mobs), each instance in the
 *                 caller's order of ba_cuda_set_model_a / ba_cuda_set_model_b.
 *   summaries     k, or NULL.
 *   rows          k x rows_cap, or NULL: instance i's first rows_cap rows of the progress table at rows + i rows_cap;
 *                 summaries[i].num_iterations is its full count.
 * Instance i gives what ba_cuda_set_model_* with its observations, ba_cuda_set_parameters(params + i n_params) and
 * ba_cuda_solve(options) give, bit for bit in the parameters, in every row field except iteration_time_s and in every
 * summary field except total_time_s (here the host wall clock of the whole call) and the ms_* timings (0 here).  Results do
 * not depend on k or on which CTA ran an instance.  A numerical failure of an instance (e.g. a non-finite start ->
 * BA_REASON_INITIAL_EVALUATION_FAILED) is reported in its summary and the call still returns BA_OK, as ba_cuda_solve does.
 * minimizer_progress_to_stdout is not honoured.
 * The problem is left as it was: its parameters, progress rows, summary and saved snapshot are untouched; the batch works
 * in per-instance buffers of its own (DESIGN.md 3.2c gives the bytes per instance).
 * BA_ERR_UNSUPPORTED wherever ba_cuda_solve would not run on BA_PATH_RIG for size or configuration: a reduced system above
 * 160, more than 8192 residual rows, PCG, force_generic_path, world size > 1.  BA_ERR_STATE without a model or inside an open
 * solve; BA_ERR_INVALID_ARGUMENT for k < 1, NULL params or rows with rows_cap < 1; BA_ERR_OUT_OF_MEMORY when the
 * per-instance buffers cannot be allocated (the problem stays usable).  The launches are counted in
 * ba_cuda_get_kernel_stats as "rig_lm_batch"; the work runs on the problem's stream and the call returns after a
 * synchronise. */
int ba_cuda_solve_batch(ba_cuda_problem* p, const ba_cuda_options* options, int32_t k, double* params,
                        const double* observations, ba_cuda_summary* summaries, ba_cuda_iteration* rows,
                        int32_t rows_cap);

/* One residual + Jacobian evaluation at the current parameters (test hook and
 * the "residual+Jacobian Mobs/s" measurement).  Outputs may be NULL.  Layouts,
 * in the caller's observation order:
 *   Model A: residuals 2/obs; jac 18/obs = [d r/d cam (2x6 row-major) | d r/d point (2x3)]
 *   Model B: residuals 8/mobs; jac 144/mobs = [d r/d cam (8x6) | d r/d frame (8x6) | d r/d marker (8x6)],
 *            blocks the functor does not take are zero. */
int ba_cuda_eval(ba_cuda_problem* p, double* cost, double* residuals, double* jac);

/* ceres::Covariance (apply_loss_function = true) over the free parameters at the CURRENT parameters, Model B only:
 * C = (J^T J)^-1, J = the Jacobian the solver sees (rows scaled by Ceres' Corrector when options->loss_function is set;
 * NULL options = ba_cuda_options_init defaults; only loss_function / loss_scale are read, and profile_kernels for the
 * per-kernel timing).  Not multiplied by a residual variance (Ceres does not either).  Outputs, any of them may be NULL:
 *   cov_kept   [6(n_cam+n_marker)]^2 row-major, blocks in parameter order [cameras | markers] (camera c at row 6c, marker m
 *              at 6(n_cam+m)); rows / columns of blocks that are not parameters (camera 0, marker 0 under fix_marker0,
 *              blocks no observation references) are 0.  Exactly symmetric.
 *   cov_frames n_time x 36: the 6x6 diagonal block of every frame pose (0 for unobserved frames)
 *   smallest_pivot_ratio: min_k d_k / max_k S_kk over the parameter rows of the Jacobi-scaled reduced system S = L D L^T
 *              (a diagnostic of its conditioning; 0 when the factorisation meets a pivot <= 0)
 * The rank test is a pivot test, not Ceres' eigenvalue criterion: BA_ERR_RANK_DEFICIENT (cov_kept and cov_frames untouched,
 * smallest_pivot_ratio written) when E^T E of a frame pose does not factor or smallest_pivot_ratio <= min_pivot_ratio
 * (<= 0: 1e-12), e.g. the 6-dimensional gauge freedom of frame poses against marker poses when no marker is fixed.
 * BA_ERR_STATE without a model and parameters or inside an open solve; BA_ERR_UNSUPPORTED for Model A (every camera is
 * free: J^T J always has a 7-dimensional gauge null space and this ABI has no constant blocks), for world size > 1 and
 * for a reduced system above 1536 (256 cameras + markers).  Uses the solve's workspace: call it between solves. */
int ba_cuda_covariance(ba_cuda_problem* p, const ba_cuda_options* options, double min_pivot_ratio,
                       double* cov_kept, double* cov_frames, double* smallest_pivot_ratio);

/* device time (ms, CUDA events) of the last ba_cuda_eval / ba_cuda_reprojection_error kernel */
/* ---- the numeric part of the correspondence stage that runs just before the path (SURVEY.md 8 f1).  ArUco detection and
 *      solvePnP (EPnP) stay with OpenCV; these are the pose algebra and corner construction around them, in the conventions of
 *      cv::Rodrigues.
 *      ba_cuda_marker_corners: Correspondencer::GetCornersInCameraWorld (Main_Calibration/correspondencer.cpp:5-39) for n marker
 *        poses (rvec | tvec): corners[n][4][3] in the order top left, top right, bottom right, bottom left.
 *      ba_cuda_compose_poses: out = a o b (marker-from-camera = base o marker-from-base, correspondencer.cpp:141-146) or, with
 *        invert_b, out = a o b^-1 (base-from-camera from another marker of the object, correspondencer.cpp:118-121).
 *      The before-BA reprojection error (correspondencer.cpp:284-339) is ba_cuda_project_points_error on those corners. ---- */
int ba_cuda_marker_corners(ba_cuda_problem* p, int64_t n, const double* rvec_tvec6, double marker_side, double* corners);
int ba_cuda_compose_poses(ba_cuda_problem* p, int64_t n, const double* a6, const double* b6, int32_t invert_b, double* out6);

double ba_cuda_last_kernel_ms(const ba_cuda_problem* p);

/* Reprojection check, the numeric part of ReprojectionCheck::Reproject
 * (reprojection_check.cpp:69,81,100-101): sum over corners of
 * ((x^ - x)^2 + (y^ - y)^2) / 2 and sqrt(err*2 / (n_points*2)). */
int ba_cuda_reprojection_error(ba_cuda_problem* p, double* sum_half_sq, double* rms_per_coord);
/* Stand-alone form working on explicit 3-D points as Reproject does: points are
 * projected with (rvec,tvec,intr4) of camera cam_of_point[i] and compared with
 * image_xy (float pixels widened to double, reprojection_check.cpp:78-81). */
int ba_cuda_project_points_error(ba_cuda_problem* p, int64_t n_points, const double* xyz,
                                 const int32_t* cam_of_point, int32_t n_cam,
                                 const double* rvec_tvec6, const double* intr4,
                                 const float* image_xy, double* sum_half_sq,
                                 double* rms_per_coord, double* reprojected_xy /* opt */);

/* Same, with the rotations given as 3x3 matrices (row-major) the way Main_Calibration's Camera_Transform.xml
 * stores them (bundle_adjustment_manager.cpp:130; read back at reprojection_check.cpp:65). */
int ba_cuda_project_points_error_rt(ba_cuda_problem* p, int64_t n_points, const double* xyz,
                                    const int32_t* cam_of_point, int32_t n_cam, const double* rot9,
                                    const double* tvec3, const double* intr4, const float* image_xy,
                                    double* sum_half_sq, double* rms_per_coord, double* reprojected_xy /* opt */);

/* Post-BA outputs of BAManager::Write (bundle_adjustment_manager.cpp:121,135-149)
 * and BALProblem::getPoint3dCoordinates (bundle_adjustment.cpp:89-130), Model B:
 *   rot9    n_cam x 9  Rodrigues(rvec) row-major
 *   inv12   n_cam x 12 rows of [R^T | -R^T t]
 *   corners n_mobs x 4 x 3 composed marker corners in the base-camera frame. */
int ba_cuda_model_b_outputs(ba_cuda_problem* p, double* rot9, double* inv12, double* corners);

#ifdef __cplusplus
}
#endif
#endif /* BA_CUDA_H_ */
