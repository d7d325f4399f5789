/*
 * rootba_b200.h -- C ABI of the B200-native square-root bundle-adjustment inner loop.
 *
 * This is the drop-in boundary for the ONE hot path of NikolausDemmel/rootba that this
 * repository accelerates: the QR (square-root) Levenberg-Marquardt inner loop.  The
 * reference has no C ABI; its seam is the C++ strategy interface
 *     rootba::Linearizor<Scalar>          (src/rootba/solver/linearizor.hpp:47-83)
 * implemented for the QR solver by
 *     rootba::LinearizorQR<Scalar>        (src/rootba/solver/linearizor_qr.cpp:52-291)
 * on top of
 *     rootba::LinearizationQR<Scalar, 9>  (src/rootba/qr/linearization_qr.hpp:54-841).
 * Every entry point below names the reference member function it replaces.  A reference
 * maintainer binds them from a `LinearizorQR_B200 : LinearizorBase<Scalar>` shim -- see
 * INTEGRATION.md.
 *
 * Conventions
 *  - plain pointers and sizes only; all pointers are HOST pointers unless the name says _dev;
 *  - Scalar-typed arrays are `float` for handles created with rba_create_f32 and `double`
 *    for rba_create_f64 (the reference instantiates float and double, linearizor.cpp:67-73);
 *  - camera state = 10 scalars (qx,qy,qz,qw, tx,ty,tz, f,k1,k2)  (bal_problem.hpp:72,84-89),
 *    landmark = 3 scalars, observation = 2 scalars (already in the loaded convention);
 *  - every function returns RBA_OK (0), RBA_NUMERICAL_FAILURE (1: the reference returns an
 *    empty vector / NaN, linearization_qr.hpp:702-711, linearizor_qr.cpp:275-277) or a negative
 *    fatal code (the reference CHECK/LOG(FATAL)-aborts; we return instead);
 *  - there is NO CPU fallback: without a CUDA device rba_create_* fails with RBA_ERR_NO_DEVICE.
 */
#ifndef ROOTBA_B200_H_
#define ROOTBA_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RBA_OK 0
#define RBA_NUMERICAL_FAILURE 1
#define RBA_ERR_INVALID_ARGUMENT (-1)
#define RBA_ERR_NO_DEVICE (-2)
#define RBA_ERR_CUDA (-3)
#define RBA_ERR_UNSUPPORTED (-4)
#define RBA_ERR_NCCL (-5)
#define RBA_ERR_STATE (-6)

#define RBA_ABI_VERSION 1

typedef struct rba_handle rba_handle; /* opaque; one per (problem, rank) */

/* BalProblem topology + observations (bal/bal_problem.hpp:61-234) in CSR-by-landmark form.
 * Per landmark the observations are ordered by ascending camera index -- the std::map order
 * the reference iterates in (bal_problem.hpp:137, landmark_block_dynamic.hpp:49-54). */
typedef struct {
  int32_t num_cameras;
  int32_t num_landmarks;
  int64_t num_observations;
  const int64_t* lm_obs_offset; /* [num_landmarks + 1] */
  const int32_t* obs_cam_idx;   /* [num_observations] */
  const void* obs_xy;           /* [2 * num_observations] Scalar */
} rba_problem_view;

/* Subset of SolverOptions (bal/solver_options.hpp:46-284) read by the QR path, plus placement. */
typedef struct {
  int32_t use_householder_marginalization; /* :258 ; 1 = Householder (ipp:717-743), 0 = Givens (ipp:700-715); both run on the device */
  int32_t use_valid_projections_only;      /* SolverOptions::use_projection_validity_check() */
  int32_t robust_norm;                     /* 0 NONE, 1 HUBER  (bal_residual_options.hpp:52) */
  double huber_parameter;                  /* bal_residual_options.hpp:58 */
  double jacobi_scaling_epsilon;           /* :208 ; 0 -> Sophus epsilonSqrt (linearizor_base.cpp:72-79) */
  int32_t preconditioner_type;             /* 0 JACOBI, 1 SCHUR_JACOBI (:217) */
  int32_t min_linear_solver_iterations;    /* :180 */
  int32_t max_linear_solver_iterations;    /* :184 */
  double eta;                              /* :189 */
  int32_t residual_reset_period;           /* ConjugateGradientsSolver::Options (conjugate_gradient.hpp:87) = 10 */
  /* placement */
  int32_t device;                          /* CUDA device ordinal, -1 = current */
  int32_t rank;                            /* landmark shard owned by this handle */
  int32_t nranks;                          /* 1 = single GPU */
  int32_t pcg_check_period;                /* CG iterations the host enqueues ahead of the progress the device publishes (NCCL exchange: poll period) (0 -> 4) */
  int32_t use_cuda_graphs;                 /* reserved, ignored: the kernels of a PCG iteration are chained with programmatic
                                              dependent launch + a device-side convergence flag instead of graph capture */
  int32_t operator_form;                   /* PCG operator (Q2^T Jp)^T (Q2^T Jp) x: 0 = dense Q2 panels, as the reference
                                              (ipp:400-441; default, the contract kernel); 1 = implicit
                                              Jp^T Jp x - (Q1d^T Jp)^T (Q1d^T Jp) x from the per-observation records
                                              (same result up to rounding, ~n/2.7 x fewer bytes, but the subtraction gives
                                              up the float32 robustness of the square-root form: recommended with f64) */
  int32_t stage2_form;                     /* gradient b and SCHUR_JACOBI blocks of the reduced system: 0 = from the stored Q2 panels
                                              like the reference (ipp:443-466, :520-552: sums of squares, no cancellation;
                                              default), 1 = through the orthogonality identities Jp^T r - Q1d^T (Q1^T r)_d and
                                              Jp^T Jp - Q1d^T Q1d (O(n) per landmark, but they cancel: float64 only).  With
                                              operator_form = 1 no panels exist and form 1 is used. */
  int32_t solver_type;                     /* SolverOptions::solver_type (:63-76): 0 = SQUARE_ROOT (LinearizorQR, default), 1 = SCHUR_COMPLEMENT
                                              (LinearizorSC, solver/linearizor_sc.cpp: landmark eliminated through the normal equations,
                                              PCG on the reduced camera system), 2 = POWER_SCHUR_COMPLEMENT (LinearizorPowerSC,
                                              solver/linearizor_power_sc.cpp: power-series solve, sc/linearization_power_sc.hpp:130-160;
                                              one GPU).  Types 1 and 2 store no Q2 panels; same entry points, same protocol. */
  int32_t power_order;                     /* :270 ; maximum number of terms of the power series (0 -> 20) */
  int32_t reserved[2];
} rba_solver_opts;

/* ResidualInfo (bal/residual_info.hpp:59-89) */
typedef struct {
  int64_t all_num_obs;
  double all_error;
  double all_residual_sum;
  int64_t valid_num_obs;
  double valid_error;
  double valid_residual_sum;
  int32_t is_numerically_valid;
  int32_t pad_;
} rba_residual_info;

/* ConjugateGradientsSolver::Summary (cg/conjugate_gradient.hpp:97-107) */
typedef struct {
  int32_t termination_type; /* 0 NO_CONVERGENCE, 1 SUCCESS, 2 FAILURE */
  int32_t num_iterations;
  int32_t num_matvecs;
  int32_t reason;           /* detail code for the message (see DESIGN.md) */
} rba_cg_summary;

/* Device times (CUDA events on the solver stream) of the IterationSummary fields
 * (solver/solver_summary.hpp:165-205), in seconds, for the LAST call of each entry point. */
typedef struct {
  double stage1_time;               /* linearize */
  double stage2_time;               /* solve: damping + gradient + precond blocks */
  double compute_preconditioner_time; /* solve: block inversion */
  double solve_reduced_system_time; /* solve: PCG */
  double back_substitution_time;    /* apply */
  double update_cameras_time;       /* apply */
  double residual_evaluation_time;  /* compute_error */
  double matvec_time;               /* inside PCG: sum over all rcs_matvec launches */
  int64_t matvec_launches;
  int64_t kernel_launches;          /* cumulative number of kernels launched by this handle since create */
} rba_stage_timings;

/* Workload statistics (computed at create; per rank) */
typedef struct {
  int64_t num_landmarks_local;
  int64_t num_observations_local;
  int64_t sum_n2;                 /* M2 = sum n_l^2 over local landmarks */
  int32_t max_n;
  int32_t num_tiles;
  int64_t panel_scalars;          /* allocated (padded) Q2 panel size in scalars */
  int64_t panel_scalars_algorithmic; /* 18 * M2 */
  int64_t device_bytes;           /* total device allocation */
  int64_t matvec_algorithmic_bytes;  /* 18*M2*s + 18*Nobs*s + 4*Nobs (SURVEY 8d) */
  int32_t landmark_begin, landmark_end; /* shard [begin, end) in problem order */
  int32_t num_matvec_items;
  int32_t reserved_;
} rba_workload_stats;

/* ---- lifecycle -------------------------------------------------------------------------- */

int32_t rba_abi_version(void);
/* message of the last failure on this thread */
const char* rba_last_error(void);
void rba_default_solver_opts(rba_solver_opts* opts);

/* replaces LinearizorQR ctor (linearizor_qr.cpp:52-72) + LinearizationQR ctor (linearization_qr.hpp:80-111):
 * uploads topology, classifies landmark blocks by track length (the reference's static n=2..8 / dynamic
 * split, qr/landmark_block.cpp:51-80, becomes sub-warp group classes), allocates device storage. */
int32_t rba_create_f32(const rba_problem_view* problem, const rba_solver_opts* opts, rba_handle** out);
int32_t rba_create_f64(const rba_problem_view* problem, const rba_solver_opts* opts, rba_handle** out);
int32_t rba_destroy(rba_handle* h);
int32_t rba_get_workload_stats(const rba_handle* h, rba_workload_stats* out);
/* 4 = float32, 8 = float64 */
int32_t rba_scalar_size(const rba_handle* h);

/* contiguous landmark shards equalising sum n^2 (SURVEY 8e); bounds[nranks + 1]; pure host code */
int32_t rba_partition_landmarks(int32_t num_landmarks, const int64_t* lm_obs_offset, int32_t nranks,
                                int32_t* bounds);

/* Host-only self check of the data model built for (problem, rank, nranks): every observation is assigned to exactly one
 * slot with the right camera, tiles are homogeneous in track length, the matvec row chunks tile every panel exactly once,
 * the camera-major CSRs list every (y) slot exactly once under its camera, shards cover the landmarks.  Needs no GPU.
 * scalar_size selects the float (4) or double (8) class limits.  Returns RBA_OK or RBA_ERR_STATE (see rba_last_error). */
int32_t rba_layout_selftest(const rba_problem_view* problem, int32_t rank, int32_t nranks, int32_t scalar_size);

/* ---- BAL file loader (SURVEY 8f row 1; host only, no GPU) ----------------------------------- */

/* load_normalized_bal_problem (bal/bal_problem.cpp:773-852) = load_bal (:189-282: whitespace-separated
 * "Nc Nl Nobs", Nobs x (cam lm x y), 9 values per camera, 3 per landmark; y of the image and y/z of the camera frame
 * flipped; observations of a landmark in ascending camera order like the reference's std::map, bal_problem.hpp:137;
 * duplicate observation / short or malformed file -> RBA_ERR_INVALID_ARGUMENT where the reference LOG(FATAL)s)
 * + normalize(scale) (:428-469, median-centre + MAD-scale, in double) when `normalize` != 0.
 * A file whose name contains "bundle" is read as a Bundler "bundle.out" v0.3 file instead (load_bundler :284-404, chosen like
 * autodetect_input_type :124-135; cameras with focal length 0 are dropped).
 * The file is parsed by `num_threads` threads (<= 0: all hardware threads) straight into the flat arrays of
 * rba_problem_view; the result is bit-identical to a one-fscanf-per-line loader (from_chars and "%lf" both round
 * correctly).  All values are double, as in the reference (cast to float happens after normalisation, :813-832). */
typedef struct rba_bal_file rba_bal_file;
int32_t rba_bal_load(const char* path, int32_t normalize, double scale, int32_t num_threads, rba_bal_file** out);
/* BalProblem::filter_obs (bal_problem.cpp:471-505; BalDatasetOptions::init_depth_threshold): drop the observations whose
 * landmark is closer than `threshold` in front of the camera, then the landmarks left with fewer than 2 observations
 * (landmark indices are compacted).  Call after rba_bal_load, before rba_bal_dims / rba_bal_copy; threshold <= 0: no-op. */
int32_t rba_bal_filter_obs(rba_bal_file* f, double threshold);
/* BalProblem::perturb (bal_problem.cpp:507-554; BalDatasetOptions rotation_sigma / translation_sigma / point_sigma /
 * random_seed, default seed 38401): Gaussian perturbation of the camera centres (world frame), the camera rotations
 * (left-multiplied exp) and the landmarks, drawn from one std::default_random_engine exactly as the reference draws them
 * (same random stream when the reference is built against libstdc++).  Call after rba_bal_load (which normalises) and
 * before rba_bal_filter_obs -- the order of load_normalized_bal_problem (bal_problem.cpp:813-826).  seed < 0: random device. */
int32_t rba_bal_perturb(rba_bal_file* f, double rotation_sigma, double translation_sigma, double point_sigma, int32_t seed);
/* sizes, to allocate the arrays for rba_bal_copy */
int32_t rba_bal_dims(const rba_bal_file* f, int32_t* num_cameras, int32_t* num_landmarks, int64_t* num_observations);
/* cams [10*Nc] (qx,qy,qz,qw,t,f,k1,k2 = Camera::params(), bal_problem.hpp:84-89), lms [3*Nl], lm_obs_offset [Nl+1],
 * obs_cam_idx [Nobs], obs_xy [2*Nobs]; any pointer may be NULL */
int32_t rba_bal_copy(const rba_bal_file* f, double* cams, double* lms, int64_t* lm_obs_offset, int32_t* obs_cam_idx, double* obs_xy);
/* seconds spent reading / counting tokens / parsing / building the CSR / normalising in rba_bal_load */
int32_t rba_bal_load_timings(const rba_bal_file* f, double* out5);
int32_t rba_bal_free(rba_bal_file* f);

/* ---- optimisation state: BalProblem cameras()/landmarks() mirror ------------------------- */

/* host -> device; cams [10*Nc], lms [3*Nl] (full problem; a sharded handle reads its slice) */
int32_t rba_set_state(rba_handle* h, const void* cams, const void* lms);
/* device -> host; a sharded handle writes only its landmark slice of lms */
int32_t rba_get_state(rba_handle* h, void* cams, void* lms);
/* BalProblem::backup / restore (bal/bal_problem.cpp:590-608) on device */
int32_t rba_backup(rba_handle* h);
int32_t rba_restore(rba_handle* h);

/* ---- Linearizor interface (solver/linearizor.hpp:56-82) ---------------------------------- */

/* LinearizorBase::compute_error (linearizor_base.cpp:59-67) -> BalBundleAdjustmentHelper::compute_error
 * (bal_bundle_adjustment_helper.cpp:68-109) */
int32_t rba_compute_error(rba_handle* h, rba_residual_info* out);
/* LinearizorQR::linearize (linearizor_qr.cpp:78-138): stage 1 */
int32_t rba_linearize(rba_handle* h);
/* LinearizorQR::solve (linearizor_qr.cpp:140-265): stage 2 + preconditioner + PCG.
 * inc_out [9*Nc] (Jacobi-scaled space, already negated) may be NULL: the increment then stays on
 * the device for rba_apply(h, NULL, ...). */
int32_t rba_solve_f32(rba_handle* h, float lambda, float* inc_out, rba_cg_summary* cg);
int32_t rba_solve_f64(rba_handle* h, double lambda, double* inc_out, rba_cg_summary* cg);
/* LinearizorQR::apply (linearizor_qr.cpp:267-291): back-substitution, landmark and camera update.
 * inc == NULL uses the device-resident increment of the last rba_solve. l_diff is NaN on failure. */
int32_t rba_apply_f32(rba_handle* h, const float* inc, float* l_diff_out);
int32_t rba_apply_f64(rba_handle* h, const double* inc, double* l_diff_out);
/* One LM inner iteration of optimize_lm_ours (bal_bundle_adjustment.cpp:324-521) with a SINGLE host synchronisation
 * (SURVEY 8f row 2): [rba_linearize when linearize_first] + rba_solve(lambda) + rba_backup + rba_apply with the
 * device-resident increment + rba_compute_error, enqueued back to back.  Same kernels in the same order as the separate
 * calls: bit-identical results.  The caller keeps the reference's accept / reject and lambda logic and calls rba_restore
 * on a rejected step -- also when `solve_failed` is set (PCG FAILURE = the reference's non-finite increment, which it
 * does not apply; here the step is applied on the device first and undone by the restore).
 * Returns like rba_apply: RBA_NUMERICAL_FAILURE when l_diff is not finite (l_diff = NaN). */
typedef struct {
  rba_cg_summary cg;
  double l_diff;              /* model cost change (Scalar precision, widened) */
  rba_residual_info cost;     /* ResidualInfo after the step */
  int32_t solve_failed;
  int32_t pad_;
} rba_lm_step_result;
int32_t rba_lm_step_f32(rba_handle* h, int32_t linearize_first, float lambda, rba_lm_step_result* out);
int32_t rba_lm_step_f64(rba_handle* h, int32_t linearize_first, double lambda, rba_lm_step_result* out);
/* The LM loop itself, natively: optimize_lm_ours (solver/bal_bundle_adjustment.cpp:291-521) on top of rba_lm_step, so that
 * consecutive iterations are separated by one host synchronisation and a few scalar operations instead of an interpreter.
 * Starts a NEW solve at the handle's current state (lambda = 1 / initial_trust_region_radius, vee = initial_vee) and runs
 * until the reference's stopping rule fires -- after a successful step, |previous logged cost - cost| <= function_tolerance *
 * cost (:69-72, :174-201), where the previous logged cost is that of the iteration before (the initial cost, a rejected step's
 * cost, or 0 after a failed solve) and both are in the ERROR / ERROR_VALID sense; lambda > 1 / min_trust_region_radius
 * (:378-379); max_num_iterations (:291) -- or `max_steps` iterations have been done.
 * Same Scalar arithmetic for lambda / vee / step quality as the reference loop (and as the Python / C++ host mirrors, which
 * stay the tested restatements).  One rba_lm_iteration is written per iteration. */
typedef struct {
  double initial_trust_region_radius, min_trust_region_radius, max_trust_region_radius;  /* solver_options.hpp:119-133 */
  double min_relative_decrease, initial_vee, vee_factor, function_tolerance;              /* :146-148, :136-143, :113 */
  int32_t max_num_iterations;                                                              /* :106 */
  int32_t optimized_cost;                                                                  /* 0 ERROR, 1 ERROR_VALID, 2 ERROR_VALID_AVG (:80-96) */
} rba_lm_opts;
typedef struct {
  double lambda;             /* damping used for this iteration's solve */
  double cost;               /* optimized cost after the step (NaN when the solve failed) */
  double l_diff;             /* model cost change */
  double relative_decrease;  /* step quality */
  double device_seconds;     /* device time of this iteration's stages (CUDA events) */
  int32_t cg_iterations;
  int32_t cg_termination;
  int32_t accepted;          /* step_is_successful */
  int32_t terminated;        /* the stopping rule fired after this iteration */
} rba_lm_iteration;
void rba_default_lm_opts(rba_lm_opts* o);
/* phase_totals (may be NULL): sums of the stage timings over the iterations done (same fields as rba_get_timings) */
int32_t rba_lm_run_f32(rba_handle* h, const rba_lm_opts* o, int32_t max_steps, rba_lm_iteration* log, int32_t* steps_done,
                       int32_t* terminated, rba_stage_timings* phase_totals);
int32_t rba_lm_run_f64(rba_handle* h, const rba_lm_opts* o, int32_t max_steps, rba_lm_iteration* log, int32_t* steps_done,
                       int32_t* terminated, rba_stage_timings* phase_totals);
/* device timings of the last calls */
int32_t rba_get_timings(const rba_handle* h, rba_stage_timings* out);

/* ---- LinearizationQR-level access used by the parity tests -------------------------------- */

/* pose_jacobian_scaling_ (linearizor_qr.cpp:130-132) [9*Nc] and the squared column norms
 * LinearizationQR::get_stage1 returns (linearization_qr.hpp:634-712) */
int32_t rba_get_jacobian_scaling(rba_handle* h, void* scaling_out, void* diag2_out);
/* RHS b of the reduced camera system after the last rba_solve (get_stage2, linearization_qr.hpp:716-815) */
int32_t rba_get_rhs(rba_handle* h, void* b_out);
/* explicit inverse of the block-Jacobi preconditioner (cg/preconditioner.hpp:79-120) [81*Nc] and the
 * blocks it was built from (damping already added) [81*Nc] */
int32_t rba_get_preconditioner(rba_handle* h, void* inv_out, void* blocks_out);
/* LinearizationQR::right_multiply (linearization_qr.hpp:823-825): y = (Q2^T Jp)^T (Q2^T Jp) x + lambda x
 * with the damping of the last rba_solve */
int32_t rba_right_multiply(rba_handle* h, const void* x, void* y);
/* LinearizationQR::back_substitute (linearization_qr.hpp:165-179) without the camera update */
int32_t rba_back_substitute_f32(rba_handle* h, const float* pose_inc, float* l_diff_out);
int32_t rba_back_substitute_f64(rba_handle* h, const double* pose_inc, double* l_diff_out);
/* One landmark block in the reference's storage layout, rows x cols row-major with
 * cols = 9n + pad + 4 (landmark_block_dynamic.hpp:56-66): rows 0..2 = Q1^T[Jp|Jl|r] (damped if damping is
 * active), rows 3..2n-1 = Q2^T Jp (Jl and r columns of these rows are reported as 0 / not stored),
 * rows 2n..2n+2 = damping rows.  `lm` is the landmark index in problem order (must be in this shard).
 * RBA_ERR_UNSUPPORTED with operator_form = 1 (no Q2 panels exist in that mode). */
int32_t rba_debug_get_block(rba_handle* h, int32_t lm, void* out, int32_t rows, int32_t cols,
                            void* jl_col_scale3_out);

/* ---- timing hooks for bench.py -------------------------------------------------------------- */

/* Runs `reps` back-to-back rcs_matvec launches (operator only, x = current p buffer) and returns the mean
 * device time per launch in seconds (CUDA events on the solver stream). */
int32_t rba_time_matvec(rba_handle* h, int32_t reps, double* seconds_per_launch);
/* CUDA-event stopwatch on the solver stream: start records an event, stop records a second one,
 * synchronises and returns the device time between them in seconds */
int32_t rba_timer_start(rba_handle* h);
int32_t rba_timer_stop(rba_handle* h, double* seconds);
/* the CUDA stream all work of this handle is enqueued on (as void* = cudaStream_t) */
void* rba_stream(rba_handle* h);
int32_t rba_synchronize(rba_handle* h);

/* ---- multi-GPU (landmarks sharded by index; cameras replicated; SURVEY 8e) ------------------ */

/* 128-byte NCCL unique id (ncclGetUniqueId); call on rank 0, broadcast by the host, pass to every rank */
int32_t rba_nccl_unique_id(void* out128);
/* create the communicator for this handle (opts.rank / opts.nranks); collective across ranks */
int32_t rba_comm_init(rba_handle* h, const void* unique_id128);
/* Optional (same box, NVLink/NVSwitch peers): fuse the per-PCG-iteration all-reduce of the operator output into the PCG
 * vector kernel over peer memory.  Every rank exports 128 bytes (two CUDA IPC handles), the host all-gathers them in
 * rank order and passes the nranks * 128 bytes to every rank.  Without it (or if peer mapping fails) NCCL is used. */
int32_t rba_ipc_export(rba_handle* h, void* out128);
int32_t rba_ipc_import(rba_handle* h, const void* all_handles /* nranks * 128 bytes */);

#ifdef __cplusplus
}
#endif
#endif /* ROOTBA_B200_H_ */
