/* hyperb200.h -- C-ABI of the B200-native HyperSLAM hot path (libhyperb200.so).
 *
 * Drop-in boundary (SURVEY.md section 8b): one context owns the flattened sliding window that the
 * reference's optimizer holds as a pointer graph, and runs what ceres::Solve runs per iteration --
 * every residual block's Evaluate(), the normal equations and the linear solve -- as batched sm_100a
 * kernels.  All pointers are plain host pointers unless a name says "device"; buffers are copied in
 * or out, never aliased across calls.  Every function returns 0 on success, <0 for an invalid
 * argument, >0 for a CUDA / numerical failure; hb200_last_error_string() describes the last one.
 * (The reference aborts through glog CHECKs and Evaluate() always returns true,
 * reference internal/hyper/optimizers/ceres/costs/exteroceptive.cpp:159,162-178.)
 * A context is not thread-safe (the reference runs everything optimiser-side on one backend thread,
 * reference internal/hyper/system/components/backend.cpp:124-158).
 */
#ifndef HYPERB200_H_
#define HYPERB200_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef struct hb200_ctx hb200_ctx;

typedef struct hb200_options {
  int device;        /* CUDA device ordinal */
  void* stream;      /* cudaStream_t to run on; NULL => the context creates its own */
  int use_graph;     /* capture hb200_iterate() in a CUDA graph (1) or launch kernels directly (0) */
  int reserved;      /* bit 0: force the dense cooperative Cholesky instead of the banded-arrow solver */
  void* nccl_comm;   /* ncclComm_t spanning the ranks that share this window, or NULL (single GPU); not owned */
  int nranks, rank;  /* size of / position in that communicator (ignored when nccl_comm is NULL) */
} hb200_options;

/* Per-iteration record, the analogue of ceres::IterationSummary printed through
 * summary.BriefReport() (reference internal/hyper/optimizers/ceres/optimizer.cpp:279). */
typedef struct hb200_iteration {
  double cost;          /* 1/2 sum rho(|r|^2) at the linearisation point */
  double cost_new;      /* cost at the trial point */
  double model_change;  /* predicted decrease of the quadratic model */
  double rho;           /* (cost - cost_new) / model_change */
  double radius;        /* trust-region radius after the update */
  int accepted;         /* step accepted */
  int spd;              /* reduced system was positive definite */
} hb200_iteration;

enum { HB200_PIXEL = 0, HB200_INERTIAL = 1, HB200_BEARING = 2, HB200_MANIFOLD = 3 };
enum { HB200_EVAL_JACOBIANS = 1, HB200_EVAL_TRIAL = 2 };

int hb200_create(const hb200_options* options, hb200_ctx** out);
void hb200_destroy(hb200_ctx* ctx);
const char* hb200_last_error_string(void);
int hb200_synchronize(hb200_ctx* ctx);

/* ---- window state: replaces the parameter blocks Ceres aliases ------------------------------
 * knots  [K][8] = Stamped<SE3> blocks [qx qy qz qw px py pz | stamp] ordered by stamp
 *         (reference optimizer.cpp:287-305 AddParameterBlock per state element; storage order
 *         reference settings.yaml:34-36, stamped.hpp:35-36).  order = layout().outer.size.      */
/* Knots must be UNIFORMLY spaced (relative tolerance 1e-6; the reference only creates uniform knots,
 * abstract.cpp:89,128), likewise the bias knots.  RE-BIND RULE: the index maps of hb200_bind follow from the
 * stamps, so changing the order, the number of knots OR ANY STAMP (a window slid by one knot keeps K) unbinds the
 * factor lists -- call hb200_bind again; hb200_optimize rejects blocks whose stamps differ from the bound window. */
int hb200_set_spline(hb200_ctx* ctx, int order, int num_knots, const double* knots);
/* bias control points [Kb][4] = Stamped<R3> [bx by bz | stamp] (reference imu.cpp:64-80). */
int hb200_set_bias_splines(hb200_ctx* ctx, int order, int num_gyro, const double* gyro, int num_accel, const double* accel);
/* gravity parameter block, 3 doubles on the sphere (reference optimizer.cpp:104). */
int hb200_set_gravity(hb200_ctx* ctx, const double* gravity);
/* cameras [C][15] = T_bs(7) | intrinsics cx cy fx fy | radtan k1 k2 p1 p2
 * (Sensor::parameters order, reference pixel.cpp:43-45). */
int hb200_set_cameras(hb200_ctx* ctx, int num_cameras, const double* cameras);
/* IMU static blocks (37) = T_bs(7) | i_g(6) | i_a(6) | S_g(9) | X_a(9) (reference inertial.cpp:35-39,45-49). */
int hb200_set_imu(hb200_ctx* ctx, const double* imu);
/* landmark position blocks [L][3] (reference optimizer.cpp:347-358). */
int hb200_set_landmarks(hb200_ctx* ctx, int num_landmarks, const double* xyz);
/* constancy: SetParameterBlockConstant on state elements (reference optimizer.cpp:322-328),
 * setGravityConstant (reference abstract.cpp:57-61), bias manifolds (reference optimizer.cpp:62-63). */
int hb200_set_constant(hb200_ctx* ctx, const unsigned char* knot_constant, int gravity_constant, int bias_constant);
/* losses: HuberLoss(huber_pixel) (reference optimizer.cpp:226), ScaledLoss(NULL, imu_loss_scale)
 * (:267-268); radius = initial trust-region radius (Ceres default 1e4). */
int hb200_set_options(hb200_ctx* ctx, double huber_pixel, double imu_loss_scale, double radius);

/* HYPER_REFERENCE_QUIRKS (SURVEY.md section 8a): 0 (default) = the mathematically consistent inertial Jacobians;
 * bits switch on the in-tree formulas verbatim -- 1: gyroscope intrinsics in the accelerometer rows (reference
 * inertial.cpp:136,142,148,158), 2: no Jacobian of the S_g a_b_m term (:135,147), 4: extrinsics block without R_sb
 * (:157-158), 8: X_a ignored in the rate / acceleration coefficients (:142,148); 15 = the reference as written.
 * All variants coincide on the calibration every reference fixture uses (I_g = I_a = I, S_g = X_a = 0, R_bs = I). */
int hb200_set_reference_quirks(hb200_ctx* ctx, int quirks);

/* ---- factor lists: replace problem_.AddResidualBlock (reference optimizer.cpp:212-232,253-274) */
int hb200_set_pixel_factors(hb200_ctx* ctx, int n, const double* stamp, const int* camera, const int* landmark, const double* pixel);
int hb200_set_inertial_factors(hb200_ctx* ctx, int n, const double* stamp, const double* measurement /* [n][6] gyro|accel */);
/* VisualBearingObservation -> AngularMetric residual behind HuberLoss(1.6e-3) (reference
 * optimizer.cpp:189-210, evaluators/bearing.cpp:14-79); bearing = [n][3] direction in the sensor frame
 * (any positive length).  Same parameter blocks as a pixel factor. */
int hb200_set_bearing_factors(hb200_ctx* ctx, int n, const double* stamp, const int* camera, const int* landmark, const double* bearing);
int hb200_set_bearing_loss(hb200_ctx* ctx, double huber_bearing);
/* ManifoldObservation<SE3> -> ManifoldMetric residual, no loss (reference optimizer.cpp:234-251,
 * evaluators/manifold.cpp:12-61).  Pose sensors carry only T_bs [q(4) p(3)] (plain Sensor, reference
 * manifold.cpp:30); pose = [n][7] measured T_ws. */
int hb200_set_pose_sensors(hb200_ctx* ctx, int num_sensors, const double* T_bs /* [P][7] */);
int hb200_set_manifold_factors(hb200_ctx* ctx, int n, const double* stamp, const int* sensor, const double* pose /* [n][7] */);
/* ExteroceptiveCost::update() for every factor (reference exteroceptive.cpp:25-99): resolves the
 * knot base index of each stamp and the segment / landmark incidence lists.  num_invalid receives
 * the number of factors whose stamp or indices fall outside the window (they are an error). */
int hb200_bind(hb200_ctx* ctx, int* num_invalid);
int hb200_get_index_maps(hb200_ctx* ctx, int* pixel_base, int* inertial_base, int* gyro_bias_base, int* accel_bias_base);

/* ---- sliding-window bookkeeping on the device (SURVEY.md section 8f rank 3) ---------------------------------
 * What the reference does per message on its pointer graph, applied to the flattened window that already lives in
 * HBM -- no host re-sort, no re-upload of the factor lists (all four kinds: pixel, bearing, inertial, pose).  After any
 * of these calls the factor "user order" is the order of the device lists: pixel factor i is the i-th pixel factor of
 * the visual list, bearing factor i the i-th bearing factor of it (the visual list holds both, in arrival order), the
 * inertial and pose lists as they stand.  hb200_get_*_outputs, hb200_factor_evaluate and a full hb200_bind use it.
 *   hb200_append_knots:    `count` state elements appended by the reference's extrapolation -- the new elements AND
 *                          the current last one take the variable of the second to last, stamps continue at the knot
 *                          separation (reference internal/hyper/optimizers/abstract.cpp:126-136).
 *   hb200_append_*:        a frame's residual blocks / new landmarks (reference optimizer.cpp:189-274,347-358).
 *                          Stamps must not precede the end of the list they are appended to (arrival order); the new
 *                          factors are bound on the device (index maps of the tail only).  A rejected append (rc 2: a
 *                          stamp outside the spline, a camera / sensor / landmark index out of range; rc 3: arrival
 *                          order) leaves the window unchanged.
 *   hb200_append_bearing_factors:  add(VisualBearingObservation&) for one frame (reference optimizer.cpp:189-210; the
 *                          same HuberLoss as hb200_set_bearing_loss); bearing [n][3], any positive length.
 *   hb200_append_manifold_factors: add(ManifoldObservation&) (reference optimizer.cpp:234-251, reached through
 *                          process(ManifoldMeasurement), abstract.cpp:266-270); needs hb200_set_pose_sensors first.
 *   hb200_append_stereo_tracks: process(VisualTracks) in one call (reference abstract.cpp:243-260): per track the
 *                          undistorted unit bearings of both views; landmark_in[i] == -1 triangulates a new landmark
 *                          at the CURRENT state's pose at stamp[i] (as hb200_ingest_stereo; no validity threshold,
 *                          :253) and appends it -- new landmarks take slots L, L+1, ... in track order -- any other
 *                          value is an existing slot in [0, L).  Two bearing factors per track, camera0's then
 *                          camera1's (:258-259: add(observation_0); add(observation_1)).  landmark_out (may be NULL)
 *                          receives every track's slot, num_new (may be NULL) the number of new landmarks.  Call it
 *                          after hb200_append_knots, as the reference does (abstract.cpp:119-144).  One H2D copy,
 *                          one small read-back.
 *   hb200_slide:           new window lower bound -- landmarks whose observation range left the window are removed
 *                          with their residuals (optimizer.cpp:360-382), state elements at or before the bound become
 *                          constant (:322-328), the ones in front of the window that no residual touches are removed
 *                          (:331-341), gravity becomes constant (abstract.cpp:57-61).  Bearing residuals go only
 *                          with their landmark (:360-382).  The reference never removes inertial or pose-prior
 *                          residuals; HB200_SLIDE_DROP_INERTIAL / HB200_SLIDE_DROP_POSE additionally drop those whose
 *                          control points all lie at or before the lower bound (all constant), so that the window
 *                          stays bounded.  Kept ones pin the leading state elements they touch.
 *   hb200_slide_stats:     visual_factors* count pixel + bearing factors; pose priors are not in the struct (its
 *                          layout is fixed) -- hb200_factor_counts reports every kind. */
typedef struct hb200_slide_stats {
  int knots_dropped, knots_constant, landmarks_dropped, visual_factors_dropped, inertial_factors_dropped;
  int knots, landmarks, visual_factors, inertial_factors;   /* sizes after the call */
} hb200_slide_stats;
enum { HB200_SLIDE_DROP_INERTIAL = 1, HB200_SLIDE_DROP_POSE = 2 };
int hb200_append_knots(hb200_ctx* ctx, int count);
int hb200_append_landmarks(hb200_ctx* ctx, int n, const double* xyz);
int hb200_append_pixel_factors(hb200_ctx* ctx, int n, const double* stamp, const int* camera, const int* landmark, const double* pixel);
int hb200_append_inertial_factors(hb200_ctx* ctx, int n, const double* stamp, const double* measurement);
int hb200_append_bearing_factors(hb200_ctx* ctx, int n, const double* stamp, const int* camera, const int* landmark, const double* bearing /* [n][3] */);
int hb200_append_manifold_factors(hb200_ctx* ctx, int n, const double* stamp, const int* sensor, const double* pose /* [n][7] */);
int hb200_append_stereo_tracks(hb200_ctx* ctx, int n, const double* stamp, const int* camera0, const int* camera1, const double* pixel0 /* [n][2] */,
                               const double* pixel1 /* [n][2] */, const int* landmark_in, int* landmark_out, int* num_new);
int hb200_slide(hb200_ctx* ctx, double lower_bound, int flags, hb200_slide_stats* stats /* may be NULL */);
/* visual_factors = pixel + bearing factors */
int hb200_window_sizes(hb200_ctx* ctx, int* knots, int* landmarks, int* visual_factors, int* inertial_factors);
int hb200_factor_counts(hb200_ctx* ctx, int* pixel, int* bearing, int* inertial, int* manifold);

/* ---- the hot path --------------------------------------------------------------------------
 * hb200_evaluate: residual (+ Jacobian) of every factor at the current state (flags 0 / JACOBIANS)
 * or at the trial state (TRIAL).  Compact outputs (DESIGN.md "HBM layout"):
 *   pixel   : r[n][2], Jp[n][2][6k], Jl[n][2][3]
 *   inertial: r[n][6], Jp[n][6][6k], wg[n][kb], wa[n][kb], Jg[n][6][2]                       */
int hb200_evaluate(hb200_ctx* ctx, int flags);
int hb200_get_pixel_outputs(hb200_ctx* ctx, double* r, double* Jp, double* Jl);
int hb200_get_inertial_outputs(hb200_ctx* ctx, double* r, double* Jp, double* wg, double* wa, double* Jg);
/*   bearing : r[n], Jp[n][6k], Jl[n][3]            manifold: r[n][6], Jp[n][6][6k]             */
int hb200_get_bearing_outputs(hb200_ctx* ctx, double* r, double* Jp, double* Jl);
int hb200_get_manifold_outputs(hb200_ctx* ctx, double* r, double* Jp);
/* Ceres-shaped copy-out of one factor after hb200_evaluate(JACOBIANS): same signature, block order
 * and row-major ambient Jacobians as ExteroceptiveCost::Evaluate (reference exteroceptive.hpp:31,
 * exteroceptive.cpp:149-156).  parameters must be the blocks the window was uploaded from.  Every block is served,
 * the calibration blocks too (extrinsics, intrinsics, distortion; i_g, i_a, S_g, X_a -- reference pixel.cpp:91-135,141,
 * inertial.cpp:155-194): they are constant in the live configuration (optimizer.cpp:59-63), so their Jacobians are
 * computed by separate kernels the first time one is requested after an evaluation, not on the iteration path. */
int hb200_factor_evaluate(hb200_ctx* ctx, int kind, int index, const double* const* parameters, double* residuals, double** jacobians);

/* normal equations + landmark Schur complement at the current linearisation point;
 * requires hb200_evaluate(JACOBIANS).  System layout: [6K pose | 3Kbg | 3Kba | 2 gravity]. */
int hb200_reduced_size(hb200_ctx* ctx);
int hb200_build_system(hb200_ctx* ctx);
/* dense copy of what the solver factors: damped (mu * clamp(diag H)), constant dofs masked to identity. */
int hb200_get_system(hb200_ctx* ctx, double* S /* n x n */, double* b /* n */);
/* dense Cholesky of the reduced system, back-substitution, landmark back-substitution. */
int hb200_solve(hb200_ctx* ctx);
int hb200_get_delta(hb200_ctx* ctx, double* delta_pose /* n */, double* delta_landmark /* 3L */);
/* full LM iterations: evaluate -> build -> [allreduce] -> solve -> retract -> cost at trial ->
 * accept/reject, all on the device.  records may be NULL. */
int hb200_iterate(hb200_ctx* ctx, int iterations, hb200_iteration* records);
int hb200_cost(hb200_ctx* ctx, double* cost);
/* ceres::Solver::Options termination tests (the reference leaves them at Ceres' defaults, optimizer.cpp:38-54:
 * function_tolerance 1e-6, gradient_tolerance 1e-10, parameter_tolerance 1e-8, min_trust_region_radius 1e-32), evaluated
 * on the device in the step-acceptance kernel exactly where ceres::TrustRegionMinimizer evaluates them; a value <= 0
 * switches a test off, all four off (the default of this library) makes hb200_iterate / hb200_optimize run exactly the
 * requested number of iterations.  Once a test fires the remaining iterations of the call are no-ops and their records
 * are zero.  hb200_get_termination: 0 none (iteration limit), 1 function, 2 parameter, 3 gradient tolerance, 4 minimum
 * trust-region radius, 5 five consecutive invalid steps; plus the number of iterations performed by the last call
 * that fetched records and the last |x - Plus(x, -g)|_inf, |step|, |x| the tests saw.
 * hb200_optimize starts every call at the initial radius of hb200_set_options (as ceres::Solve does); hb200_iterate
 * continues the trust region of the previous call.  At N > 1 the gradient test needs the peer mailbox. */
int hb200_set_termination(hb200_ctx* ctx, double function_tolerance, double gradient_tolerance, double parameter_tolerance, double min_trust_region_radius);
int hb200_get_termination(hb200_ctx* ctx, int* type, int* iterations_performed, double* gradient_max_norm, double* step_norm, double* x_norm);
/* The drop-in for CeresOptimizer::optimize() (reference optimizer.cpp:276-280) with the parameter
 * blocks in HOST memory, as Ceres aliases them: uploads the five variable families, runs
 * `iterations` LM iterations on the device, downloads the updated blocks into the same buffers and
 * synchronises once.  Factor lists stay bound.  Buffers should be pinned for asynchronous copies. */
int hb200_optimize(hb200_ctx* ctx, int iterations, double* knots, double* gyro, double* accel, double* gravity, double* landmarks,
                   hb200_iteration* records);
/* device-side snapshot / restore of the variable blocks and the trust-region state (benchmarks,
 * step rejection experiments). */
int hb200_snapshot(hb200_ctx* ctx);
int hb200_restore(hb200_ctx* ctx);
/* Runs `reps` LM iterations with a CUDA event after every kernel and returns the average duration of
 * each launch in issue order (names are kernel names, 32 chars each).  Not for timing the step --
 * for attributing it (bench.py roofline / kernel shares).  A negative `reps` profiles |reps| plain
 * Evaluate sweeps (what hb200_evaluate(HB200_EVAL_JACOBIANS) launches) instead of full iterations. */
int hb200_profile_iteration(hb200_ctx* ctx, int reps, int max_entries, char* names /* [max_entries][32] */, double* ms, int* count);
/* Spline interpolation of the current state at `n` stamps (device kernel): pose [n][7] = [q|p], and
 * optionally (may be NULL) body velocity [n][6] = [omega | R^T pdot] and acceleration [n][6]. Stamps
 * outside the valid span give identity/zero rows and are counted in num_invalid.  Replaces
 * state->evaluate(StateQuery{stamp, derivative}) for trajectory dumps (reference apps/hyperslam/main.cpp:69-80). */
int hb200_interpolate(hb200_ctx* ctx, int n, const double* stamps, double* pose, double* velocity, double* acceleration, int* num_invalid);
int hb200_get_state(hb200_ctx* ctx, double* knots, double* gyro, double* accel, double* gravity, double* landmarks);
/* Ingest of stereo tracks in front of the factor lists (reference internal/hyper/optimizers/abstract.cpp:186-264):
 * per track i the unit bearings of both views (C.convertPixelsToBearings, :221-223) and the landmark
 * triangulated from them and moved to the world frame with the CURRENT state's pose at stamp[i]
 * (Camera::Triangulate(T_01, b0, b1) :252, T_w0.vectorPlus :253).  Outputs may not be NULL.  Tracks whose stamp
 * or camera index is invalid are zero-filled and counted. */
int hb200_ingest_stereo(hb200_ctx* ctx, int n, const double* stamp, const int* camera0, const int* camera1, const double* pixel0 /* [n][2] */,
                        const double* pixel1 /* [n][2] */, double* bearing0 /* [n][3] */, double* bearing1 /* [n][3] */,
                        double* landmark /* [n][3] */, int* num_invalid);

/* ---- multi-GPU (SURVEY.md section 8e) ---------------------------------------------------------
 * Factors shard over ranks, the window state is replicated.  Per iteration every rank builds its partial
 * reduced system, ONE ncclAllReduce sums it on the context's stream (enqueued from C, so the iteration stays
 * one CUDA graph), every rank solves redundantly and retracts its replica; the three step-acceptance scalars
 * (trial cost, landmark parts of the model decrease) are exchanged through peer memory inside accept_kernel
 * (hb200_peer_*), with a second 4-double ncclAllReduce as the fallback when no peer mapping exists.
 *
 * SHARDING CONTRACT (the caller's responsibility; violating it gives silently wrong steps):
 *   - every observation (pixel / bearing factor) of a landmark must live on ONE rank -- the landmark's owner.
 *     The landmark block is eliminated rank-locally (Schur complement of a sum is not the sum of Schur
 *     complements) and only the owner updates the landmark, so non-owned landmarks of a replica are stale;
 *     read each landmark back from its owner.
 *   - inertial and manifold factors may be split arbitrarily; every factor lives on exactly one rank.
 *   - knots, bias splines, gravity, calibration, constancy flags and options must be identical on all ranks,
 *     and every rank must make the same sequence of hb200_iterate / hb200_optimize / hb200_build_system calls.
 *
 * Reduced buffer (what is summed): the band-only packed system, hb200_system_device_ptr(), in doubles
 *   [ P K*h*6 | A m*6K | C m*m | b n | diagH n | g n | scal 8 ],  h = 6 + 6*beta, m = n - 6K
 * (block-banded pose part of half-bandwidth beta = longest landmark track in control points, arrowhead of
 * the bias / gravity dofs; scal[0] = cost at the linearisation point).  K = 50: 20 k doubles (0.16 MB). */
/* ncclGetUniqueId / ncclCommInitRank through the library (libnccl.so.2 is bound with dlopen at the first call):
 * rank 0 creates the 128-byte id, the host program ships it to the other ranks (MPI, torch.distributed, ...). */
int hb200_comm_unique_id(char* id /* [128] */);
int hb200_comm_init_rank(hb200_ctx* ctx, int nranks, int rank, const char* id /* [128] */);
/* or attach an existing ncclComm_t (not owned; NULL detaches).  Same as hb200_options.nccl_comm at creation. */
int hb200_set_nccl_comm(hb200_ctx* ctx, void* nccl_comm, int nranks, int rank);
/* peer-memory mailbox for the step-acceptance scalars: every rank exports a 64-byte cudaIpcMemHandle_t, the
 * host program all-gathers them, every rank maps its peers' mailboxes.  Ranks must be processes on one node
 * with NVLink / PCIe peer access.  Optional: without it the scalars take a second ncclAllReduce. */
int hb200_peer_handle(hb200_ctx* ctx, char* handle /* [64] */);
int hb200_peer_connect(hb200_ctx* ctx, int nranks, int rank, const char* handles /* [nranks][64] */);
/* all ranks or none: when the mapping failed on any rank, every rank drops it (collective protocol). */
int hb200_peer_disconnect(hb200_ctx* ctx);
int hb200_comm_info(hb200_ctx* ctx, int* nranks, int* rank, int* nccl, int* peer_mailbox, int* graph, long long* payload_doubles);
/* Block half-bandwidth beta of the packed layout.  It follows from the longest landmark track of the local factor
 * shard; with a communicator attached hb200_bind / hb200_set_nccl_comm agree on the maximum over the ranks
 * themselves (collective).  Hosts using the callback hook below must do that: read it after hb200_bind, take the
 * maximum over ranks, set it as the lower bound everywhere. */
int hb200_get_bandwidth(hb200_ctx* ctx, int* beta);
int hb200_set_min_bandwidth(hb200_ctx* ctx, int beta);
/* Escape hatch for hosts without NCCL: the caller sums `count_doubles` doubles at `device_buffer` across ranks
 * on `stream` (called twice per iteration: packed system, then 4 scalars).  Disables CUDA-graph capture. */
typedef int (*hb200_allreduce_fn)(void* user, void* device_buffer, long long count_doubles, void* stream);
int hb200_set_allreduce(hb200_ctx* ctx, hb200_allreduce_fn fn, void* user);
void* hb200_system_device_ptr(hb200_ctx* ctx, long long* count_doubles);
void* hb200_stream(hb200_ctx* ctx);

/* Measured FP64 FMA throughput of the device in TFLOP/s (DFMA chains, all SMs): the second roofline ceiling of the
 * FP64 factor kernels next to the HBM copy bandwidth (bench.py reports both). */
int hb200_measure_fp64_peak(hb200_ctx* ctx, double* tflops);

/* kernel-launch counter (number of this library's kernels launched since creation). */
long long hb200_launch_count(hb200_ctx* ctx);

#ifdef __cplusplus
}
#endif
#endif /* HYPERB200_H_ */
