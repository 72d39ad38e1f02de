/* ba_b200.h -- C-ABI of the B200-native bundle-adjustment engine (libba_b200.so).
 *
 * The reference (ChanghyeonKim93/bundle_adjustment_solver) has no FFI / plugin
 * interface: its boundary is the C++ class
 *   visual_navigation::analytic_solver::FullBundleAdjustmentSolver
 *   (core/full_bundle_adjustment_solver.h:127-146) and
 *   PoseOnlyBundleAdjustmentSolver (core/pose_only_bundle_adjustment_solver.h:19-67).
 * The drop-in C++ classes with those exact names/signatures live in
 * include/ba_b200/ and are thin host shims over the entry points below; each
 * entry point cites the reference code it replaces.  Plain pointers and sizes
 * only; no C++ / torch types cross this boundary; no exceptions cross it
 * (every call returns 0 on success, <0 on error, see ba_last_error()).
 *
 * Units: the engine works in the reference's *internal* units -- everything
 * already multiplied by scaler_ = 0.01 and poses already inverted to T_jw
 * (core/full_bundle_adjustment_solver.cpp:38,72-117,176).  The host shim does
 * that conversion exactly where the reference does (Add*).
 */
#ifndef BA_B200_H_
#define BA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BA_OK 0
#define BA_ERR_INVALID (-1)
#define BA_ERR_CUDA (-2)
#define BA_ERR_STATE (-3)
#define BA_ERR_NCCL (-4)

typedef struct ba_solver ba_solver; /* opaque handle, one per host thread / GPU */

/* Mirrors Options (core/solver_option_and_summary.h:47-72); float fields stay
 * float and are promoted in comparisons exactly as the reference does. */
typedef struct ba_options {
  int solver_type;               /* ignored by the full-BA path, as in the reference (:630-658) */
  float threshold_step_size;     /* convergence_handle */
  float threshold_cost_change;
  float threshold_huber_loss;    /* outlier_handle */
  float threshold_outlier_rejection;
  int max_num_iterations;        /* iteration_handle */
  float initial_lambda;          /* trust_region_handle */
  float decrease_ratio_lambda;
  float increase_ratio_lambda;
  int b_accumulate;              /* 0 = reference-exact B_ji assignment (full...cpp:826, last
                                    observation of a (pose,point) pair wins); 1 = corrected `+=` */
  double inverse_scaler;         /* inverse_scaler_ in rho (full...cpp:39,930); 100 for the shim */
  int check_every;               /* host polls the device convergence flag every this many LM
                                    iterations (device decides; extra iterations are no-ops). 0 = default */
  int use_graph;                 /* 1 = replay one LM iteration as a CUDA graph (default), 0 = plain launches */
  int method;                    /* BA_METHOD_*: which loop of the reference ba_solve runs (0 = the default) */
} ba_options;

/* ba_options.method.  FullBundleAdjustmentSolver::Solve is always Levenberg-Marquardt (it ignores
 * Options::solver_type, full_bundle_adjustment_solver.cpp:630-1044); FullBundleAdjustmentSolverRefactor::Solve
 * switches on it (full_bundle_adjustment_solver_refactor.cpp:944-982) and adds SolveByGradientDescent (:1075-1367). */
#define BA_METHOD_LEVENBERG_MARQUARDT 0 /* trial step, rho test, lambda update */
#define BA_METHOD_GAUSS_NEWTON 1        /* refactor.cpp:976-982: same damped system (lambda stays initial_lambda),
                                           the step is always kept */
#define BA_METHOD_GRADIENT_DESCENT 2    /* refactor.cpp:1159-1330: step = the gradient blocks a_j, b_i clipped to a
                                           norm of 0.001, always kept; single GPU only */

/* Mirrors OptimizationInfo (core/solver_option_and_summary.h:37-46). */
typedef struct ba_iter_info {
  double cost;
  double cost_change;
  double average_reprojection_error;
  double abs_gradient;
  double abs_step;
  double damping_term;
  double iter_time;              /* ms; device time averaged over the polled batch */
  int iteration_status;          /* IterationStatus: 0 UPDATE, 1 UPDATE_TRUST_MORE, 2 SKIPPED */
  int _pad;
} ba_iter_info;

typedef struct ba_result {
  int n_iterations;              /* LM iterations executed (rows written to infos, up to cap) */
  int converged;                 /* Summary::convergence_status_ (full...cpp:971-979,1026) */
  double initial_cost;           /* EvaluateCurrentCost() before the loop (:707) */
  double final_cost;
  double total_time_ms;          /* wall time of ba_solve */
  double device_time_ms;         /* CUDA-event time of the LM loop */
  /* per-phase CUDA-event sums (ms), filled when ba_set_profile(s,1) */
  double t_linearize_ms;         /* K1+K2: projection/Jacobians/A,B,C,a,b + damping + C^-1 */
  double t_schur_ms;             /* K4: S = A - B C^-1 B^T, rhs */
  double t_solve_ms;             /* K5: Cholesky + triangular solves */
  double t_backsub_ms;           /* K6: y, model change (point part) */
  double t_update_cost_ms;       /* K7: se3Exp update, trial cost, accept/lambda/convergence */
  long long kernel_launches;     /* kernels launched inside ba_solve (graph nodes counted per replay) */
} ba_result;

/* ---- lifetime ---------------------------------------------------------- */
int ba_create(ba_solver **out, int device);           /* replaces FullBundleAdjustmentSolver() (full...cpp:6-42) */
void ba_destroy(ba_solver *s);                        /* ~FullBundleAdjustmentSolver (:241) */
int ba_reset(ba_solver *s);                           /* Reset() (:44-70) */
const char *ba_last_error(const ba_solver *s);
int ba_set_stream(ba_solver *s, void *cuda_stream);   /* run on the caller's stream (e.g. torch's current stream) */
int ba_set_profile(ba_solver *s, int enable);         /* per-phase CUDA events */
int ba_set_debug(ba_solver *s, int keep_blocks);      /* keep S/rhs before factorisation and every pair's B for ba_debug_dump */

/* ---- problem definition (host buffers; copied, never retained) --------- */
/* AddCamera (full...cpp:72-85): ids are the user's camera indices; intr = fx,fy,cx,cy per camera
 * (scaled); T_cam_body = 12 doubles per camera, R row-major then t (pose_this_to_cam0, t scaled). */
int ba_set_cameras(ba_solver *s, int n_cam, const int *ids, const double *intr, const double *T_cam_body);
/* AddPose + MakePoseFixed (:87-101,119-134): T_jw = 12 doubles per pose (R row-major | t), fixed[n]. */
int ba_set_poses(ba_solver *s, int n, const double *T_jw, const uint8_t *fixed);
/* AddPoint + MakePointFixed (:103-117,136-153). */
int ba_set_points(ba_solver *s, int m, const double *X, const uint8_t *fixed);
/* AddObservation (:155-180), insertion order preserved (it decides the last-writer B block).
 * pose / point are indices into the arrays above; uv scaled pixels (2 per observation).
 * Observations with an unknown camera id or out-of-range index are dropped, as the reference
 * drops them; the number kept is returned through n_kept (may be NULL). */
int ba_set_observations(ba_solver *s, long long n_obs, const int *cam_id, const int *pose, const int *point,
                        const double *uv, long long *n_kept);
/* The same with the pixels in the caller's units: every coordinate is multiplied by uv_scale (the reference's
 * scaler_ = 0.01, core/full_bundle_adjustment_solver.cpp:38, :176) while it is copied. */
int ba_set_observations_scaled(ba_solver *s, long long n_obs, const int *cam_id, const int *pose, const int *point,
                               const double *uv, double uv_scale, long long *n_kept);
/* FinalizeParameters + SetProblemSize + connectivity (:182-206,243-308,669-700): index assignment,
 * the two sort orders, last-writer flags, chunking, and the H2D pack into SoA device buffers.
 * Idempotent. */
int ba_finalize(ba_solver *s);
/* Re-upload parameter values only (same structure), e.g. to re-run a solve from a new initial guess. */
int ba_update_parameters(ba_solver *s, const double *T_jw, const double *X);

/* ---- the hot path ------------------------------------------------------ */
/* Solve (:630-1044) from :707 to :1008 on the device.  infos may be NULL. */
int ba_solve(ba_solver *s, const ba_options *opt, ba_iter_info *infos, int cap, ba_result *result);
/* One linearisation + Schur build (+ optional reduced solve/back-substitution) at the current
 * parameters without updating them: (:711-917).  Used for block parity and phase timing. */
int ba_build_only(ba_solver *s, const ba_options *opt, double lambda, int do_solve);
/* EvaluateCurrentCost (:381-433) at the current parameters. */
int ba_cost(ba_solver *s, double *cost);

/* Per-observation residuals and a status per row, for the solve / reject outliers / solve loop of a front-end. */
#define BA_OBS_INLIER 0
#define BA_OBS_OUTLIER 1        /* |r_u| + |r_v| > threshold */
#define BA_OBS_BEHIND_CAMERA 2  /* depth in the observing camera <= 0, or a non-finite residual; wins over OUTLIER */
#define BA_OBS_DROPPED 3        /* row rejected by ba_set_observations (unknown camera id, pose or point) */
/* Residual r = projection - pixel of every row of the last ba_set_observations(_scaled) call, in that call's row order,
 * at the accepted parameters, in internal units (pixels x scaler_ = 0.01 for the shims).  threshold is in the same
 * internal units and uses the same L1 norm of the residual as the full-BA Huber weight (full...cpp:763-766); a row
 * whose norm equals the threshold is an inlier; +inf classifies depth only; NaN or negative is BA_ERR_INVALID.
 * residuals [2*n_rows], status [n_rows] (BA_OBS_*), counts [4] (rows per BA_OBS_* value): each may be NULL.
 * Dropped rows get NaN residuals.  Finalizes first, as ba_cost does; does not change the parameters, the LM state or
 * the next ba_solve.  On a solver joined to a communicator: this rank's rows, no communication. */
int ba_observation_residuals(ba_solver *s, double threshold, double *residuals, uint8_t *status, long long *counts);

/* Structure-only bundle adjustment: refines landmarks while every pose stays where it is. */
#define BA_POINT_CONVERGED 0       /* the loop ended on the step / cost-change test */
#define BA_POINT_MAX_ITERATIONS 1  /* max_num_iterations reached without converging */
#define BA_POINT_SKIPPED 2         /* fixed, or not selected: untouched */
#define BA_POINT_UNOBSERVED 3      /* selected and free, but no observation: untouched */
#define BA_POINT_NONFINITE 4       /* cost at the start is not finite: untouched, no iteration */
/* Every selected free landmark i runs Solve's LM loop (:707-1008) on the problem made of landmark i alone, every pose
 * fixed, and all of i's observations (those from poses that are fixed in the registered problem included): its own
 * lambda (from initial_lambda), iteration count and convergence verdict, step = ||y||.  opt->method must be
 * BA_METHOD_LEVENBERG_MARQUARDT and max_num_iterations >= 1 (else BA_ERR_INVALID); check_every, use_graph and
 * b_accumulate are ignored.  select [M_total] (order of ba_set_points), or NULL for every free landmark.
 * costs [2*M_total]: the cost sum ||r||_2 of each landmark's observations at entry and at the returned point, for
 * every landmark (skipped ones included; 0 without observations), internal units as ba_iter_info.cost.
 * iterations [M_total], status [M_total] (BA_POINT_*), counts [5] (landmarks per BA_POINT_* value): each may be NULL.
 * Finalizes first, as ba_cost does.  Afterwards the poses are unchanged and the solver is in the state
 * ba_update_parameters(s, NULL, refined points) leaves: the next ba_solve, ba_cost or ba_observation_residuals
 * behaves as on a solver given these parameters.  BA_ERR_STATE on a solver joined to a communicator. */
int ba_refine_points(ba_solver *s, const ba_options *opt, const uint8_t *select, double *costs, int *iterations,
                     uint8_t *status, long long *counts);

/* Triangulation: places landmarks from the accepted poses and their observations, e.g. new landmarks before a solve. */
#define BA_TRI_TRIANGULATED 0
#define BA_TRI_SKIPPED 1              /* fixed, or not selected: untouched */
#define BA_TRI_TOO_FEW_OBSERVATIONS 2 /* fewer than two observations */
#define BA_TRI_LOW_PARALLAX 3         /* rays too close to parallel, or the solve is not finite */
#define BA_TRI_BEHIND_CAMERA 4        /* depth <= 0 in some observing camera */
#define BA_TRI_LARGE_RESIDUAL 5       /* some observation's |r_u| + |r_v| > max_residual */
/* Landmark i, over all of its observations k in point order (lowest pose index first, then insertion order; those
 * from fixed poses included): the observing camera is R_k = R_c R_jw, t_k = R_c t_jw + t_c, its centre
 * c_k = -R_k^T t_k and the unit ray d_k = R_k^T m_k / ||m_k||, m_k = ((u - cx) / fx, (v - cy) / fy, 1); f is the first
 * observation.  The status rules, first match wins:
 *   1. fixed or not selected: BA_TRI_SKIPPED;  2. fewer than two observations: BA_TRI_TOO_FEW_OBSERVATIONS;
 *   3. min_k d_f . d_k > cos(min_parallax): BA_TRI_LOW_PARALLAX;
 *   4. X = c_f + A^-1 g, A = sum_k (I - d_k d_k^T), g = sum_k (I - d_k d_k^T)(c_k - c_f) (the multi-view midpoint;
 *      A^-1 by the pivoted LDL^T of the landmark side); X not finite: BA_TRI_LOW_PARALLAX;
 *   5. some observation has depth <= 0 at X, or a non-finite residual: BA_TRI_BEHIND_CAMERA;
 *   6. some observation has |r_u| + |r_v| > max_residual at X: BA_TRI_LARGE_RESIDUAL;
 *   7. otherwise BA_TRI_TRIANGULATED.
 * Rules 5 and 6 are the BA_OBS_BEHIND_CAMERA and BA_OBS_OUTLIER tests of ba_observation_residuals, so after the call
 * every observation of a triangulated landmark is BA_OBS_INLIER at threshold max_residual.
 * select [M_total] (order of ba_set_points), or NULL for every free landmark.  min_parallax in radians, in (0, pi];
 * max_residual in internal units (pixels x scaler_), >= 0, +inf disables rule 6; anything else (NaN included) is
 * BA_ERR_INVALID.  status [M_total] (BA_TRI_*), counts [6] (landmarks per BA_TRI_* value): each may be NULL.
 * Only BA_TRI_TRIANGULATED landmarks are written; every other landmark keeps its accepted value bit for bit (NaN
 * included).  Finalizes first, as ba_cost does.  Afterwards the poses are unchanged and the solver is in the state
 * ba_update_parameters(s, NULL, X) leaves.  BA_ERR_STATE on a solver joined to a communicator. */
int ba_triangulate_points(ba_solver *s, const uint8_t *select, double min_parallax, double max_residual,
                          uint8_t *status, long long *counts);

/* ---- results ----------------------------------------------------------- */
int ba_get_poses(ba_solver *s, double *T_jw);  /* all poses, 12 doubles each, internal units */
int ba_get_points(ba_solver *s, double *X);    /* all points */
int ba_get_sizes(ba_solver *s, long long *out6); /* N_opt, M_opt, P(pairs), n_obs, N_total, M_total */

/* Debug dumps of the block storage after the last executed iteration, in the oracle's layout:
 * which: 0 A (N*36, damped, row-major 6x6)  1 a (N*6)  2 C (M*9, damped)  3 b (M*3)  4 Cinv (M*9)
 *        5 B (P*18, row-major 6x3, pairs sorted by (point,pose))  6 S (n*n, symmetric, n=6N)
 *        7 rhs (n)  8 x (n)  9 y (M*3)  10 scalars {cost_prev,cost_new,model,rho,lambda}
 * buf == NULL returns the element count.  Free blocks are indexed by free index in id order.  S, rhs and B are
 * kept only with ba_set_debug(s, 1): without it these return BA_ERR_STATE. */
long long ba_debug_dump(ba_solver *s, int which, double *buf);
int ba_debug_pairs(ba_solver *s, int *pair_pose_id, int *pair_point_id); /* original ids per pair */
/* In-situ timing of parts of the reduced solve (bit 0 diag, 1 trsm, 2 syrk, 3 backward); timing only. */
int ba_debug_time_solve(ba_solver *s, int parts, int reps, float *ms_per_rep);
/* Reduced-solve path selected by the plan and its flop / byte counts (measurement only, bench.py):
 * vals[8] = algorithmic flops (envelope Cholesky + solves), executed flops, dense equivalent, half-bandwidth,
 * CTAs, dependent panel steps, band-only clearing (0/1), algorithmic bytes. */
int ba_debug_solve_info(ba_solver *s, char *name, int cap, double *vals);
/* Host-only (no device): partition plan of the banded reduced solve (csrc/ba_nd_plan.h) for N free poses and track
 * span b.  nodes_out [cap][20]; meta [8]; returns the number of tree nodes.  Used by the CPU test that emulates the
 * fronts in numpy. */
int ba_debug_nd_plan(int N, int b, int max_ctas, int force_depth, int force_chunk, long long *meta,
                     long long *nodes_out, int cap);

/* ---- multi-GPU (one process per GPU; landmarks sharded, S all-reduced) -- */
/* 128-byte NCCL unique id; rank 0 creates it, the host distributes it (torch.distributed, MPI...). */
int ba_comm_get_unique_id(void *id128);
/* Joins the communicator.  After this, ba_solve all-reduces [S | rhs] and the LM scalars over NCCL
 * every iteration; each rank must hold ALL poses and only ITS landmarks + their observations.
 * global_num_opt_points = sum over ranks of free points (for the step-size average, :968-970).
 * May be called before or after ba_finalize: whichever comes second min-reduces the co-visibility envelope over the
 * ranks, so that every rank factors the summed reduced system with the same (global) plan. */
int ba_comm_init(ba_solver *s, const void *id128, int rank, int nranks, long long global_num_opt_points,
                 long long global_num_observations);
/* Attaches the solver to the communicator this process already created on the solver's device with ba_comm_init
 * (communicator creation costs ~0.4 s per rank; a process that solves problem after problem joins once). */
int ba_comm_attach(ba_solver *s, long long global_num_opt_points, long long global_num_observations);
/* Detaches the solver.  The communicator lives until ba_comm_shutdown(device) and its last attached solver is gone. */
int ba_comm_destroy(ba_solver *s);
int ba_comm_shutdown(int device);

/* ---- batched pose-only solvers (pose_only_bundle_adjustment_solver.cpp:8-900) ---------- */
typedef struct ba_poseonly_options {
  float threshold_step_size;
  float threshold_cost_change;
  float threshold_huber_loss;
  float threshold_outlier_rejection;
  int max_num_iterations;
} ba_poseonly_options;

typedef struct ba_poseonly_result {
  int n_iterations;  /* loop trips executed, including the converging one */
  int converged;     /* is_converged (:55,116-122) */
  int success;       /* 0 only if the pose went NaN (:159-167); the pose is then left untouched */
  int n_summary;     /* OptimizationInfo rows the reference would have pushed (:128-147) */
  float final_error;
  float final_step;
} ba_poseonly_result;

#define BA_POSEONLY_MONO_6DOF 0      /* Solve_Monocular_6Dof        (:8-170)   */
#define BA_POSEONLY_STEREO_6DOF 1    /* Solve_Stereo_6Dof           (:172-399) */
#define BA_POSEONLY_MONO_PLANAR3DOF 2   /* Solve_Monocular_Planar3Dof (:401-615) */
#define BA_POSEONLY_STEREO_PLANAR3DOF 3 /* Solve_Stereo_Planar3Dof    (:617-900) */

/* n_frames independent problems; frame f owns points [offsets[f], offsets[f+1]).
 * points: 3 floats each (reference/world positions); px_left/px_right: 2 floats each (px_right may
 * be NULL for mono; a right pixel with x<0 or y<0 is skipped, :298); intr_*: fx,fy,cx,cy;
 * poses are 12 floats (R row-major | t): left_to_right, base_to_camera (planar only),
 * world_to_last (planar only, one per frame), poses_io (one per frame: reference_to_current /
 * world_to_current, in/out).  masks: one byte per point (1 = inlier), may be NULL.
 * hist_cost / hist_step: [n_frames * max_num_iterations] floats or NULL; debug_poses:
 * [n_frames * max_num_iterations * 12] floats or NULL (GetDebugPoses, :902-905).
 * All pointers are HOST pointers; the call copies in, solves every frame on the device, copies out. */
int ba_poseonly_solve_batched(int device, int kind, int n_frames, const int *offsets, const float *points,
                              const float *px_left, const float *px_right, const float *intr_left,
                              const float *intr_right, const float *left_to_right,
                              const float *base_to_camera, const float *world_to_last, float *poses_io,
                              uint8_t *mask_left, uint8_t *mask_right, const ba_poseonly_options *opt,
                              ba_poseonly_result *results, float *hist_cost, float *hist_step,
                              float *debug_poses);

/* Device-resident variant for throughput measurement: the same problem is uploaded once
 * (ba_poseonly_upload) and solved repeatedly from the initial poses (ba_poseonly_run). */
typedef struct ba_poseonly_batch ba_poseonly_batch;
int ba_poseonly_upload(ba_poseonly_batch **out, int device, int kind, int n_frames, const int *offsets,
                       const float *points, const float *px_left, const float *px_right,
                       const float *intr_left, const float *intr_right, const float *left_to_right,
                       const float *base_to_camera, const float *world_to_last, const float *poses_init);
int ba_poseonly_run(ba_poseonly_batch *b, const ba_poseonly_options *opt, void *cuda_stream);
int ba_poseonly_download(ba_poseonly_batch *b, float *poses_out, uint8_t *mask_left, uint8_t *mask_right,
                         ba_poseonly_result *results);
void ba_poseonly_free(ba_poseonly_batch *b);

const char *ba_version(void);

/* ---- batched geometry helpers (utility/geometry_library.cpp:93-736 on the device) ---------------------------
 * One element per thread; host buffers in and out.  Rotation matrices row-major (9), rigid transforms as R (9) | t (3),
 * quaternions (w, x, y, z), twists [v; w].  in2 is only read by the two-operand ops. */
enum {
  BA_GEOM_SE3_EXP = 0,       /* se3Exp   :370   6 -> 12 */
  BA_GEOM_SE3_LOG = 1,       /* SE3Log   :488  12 -> 6  */
  BA_GEOM_SO3_EXP = 2,       /* so3Exp   :590   3 -> 9  */
  BA_GEOM_SO3_LOG = 3,       /* SO3Log   :659   9 -> 3  */
  BA_GEOM_Q2R = 4,           /* q2r      :93    4 -> 9  */
  BA_GEOM_R2Q = 5,           /* r2q      :206   9 -> 4  */
  BA_GEOM_ROTVEC2Q = 6,      /* rotvec2q :146   3 -> 4  */
  BA_GEOM_R2EULER = 7,       /* r2euler  :322   9 -> 3  */
  BA_GEOM_A2R = 8,           /* a2r      :181   3 (roll, pitch, yaw) -> 9 */
  BA_GEOM_INVERSE_SE3 = 9,   /* inverseSE3 :729 12 -> 12 */
  BA_GEOM_ADD_FRONT_SE3 = 10,/* addFrontse3 :712  xi (6), dxi (6) -> 6 */
  BA_GEOM_Q_MULT = 11        /* q1_mult_q2 :74   4, 4 -> 4 */
};
int ba_geometry_batched(int device, int op, long long n, const double *in, const double *in2, double *out);
int ba_geometry_batched_f(int device, int op, long long n, const float *in, const float *in2, float *out);

#ifdef __cplusplus
}
#endif
#endif /* BA_B200_H_ */
