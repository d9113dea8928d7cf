/*
 * mpc_b200.h -- C-ABI of the B200-native batched nonlinear-MPC solver.
 *
 * This is the drop-in boundary for the reference's one hot path,
 *     std::vector<double> MPC::solve(VectorXd &state, double target_velocity,
 *                                    vector<double>* x_trajectory, vector<double>* y_trajectory, double dir)
 *     /root/reference/src/control/MPC.h:42-43, /root/reference/src/control/MPC.cpp:183-325
 * (NLP assembly MPC.cpp:204-281, FG_eval MPC.cpp:50-154, CppAD::ipopt::solve call MPC.cpp:290-292,
 * output unpacking MPC.cpp:306-324) and its hidden inputs: the fitted polynomial held in
 * MPC::roadGeometry (MPC.h:26) and the Config:: statics (src/utils/Config.h:66-177).
 *
 * Plain pointers and sizes only; no exceptions cross the boundary; every entry point returns
 * 0 on success or a negative MPC_E* code.  There is NO CPU fallback: without a CUDA device every
 * compute entry point returns MPC_ENODEV.
 */
#ifndef MPC_B200_H
#define MPC_B200_H

#ifdef __cplusplus
extern "C" {
#endif

#define MPC_NCOEF 5        /* polynomial coefficients per problem, low -> high order, zero padded
                              (Config::maxFitOrder = 5 => order <= 4, RoadGeometry.cpp:27-34) */
#define MPC_NTAB 16        /* capacity of the steers / steer-speeds tables (9 in config-*.json) */
#define MPC_NWEIGHTS 12    /* Config::weights, indices Config.h:14-61 */
#define MPC_NMAX 64        /* maximum horizon N (the reference's examples/ grid goes to N = 50) */

/* error codes */
#define MPC_OK 0
#define MPC_EINVAL (-1)    /* bad argument (NULL pointer, N out of range, B < 0 ...) */
#define MPC_ENODEV (-2)    /* no CUDA device / device index out of range */
#define MPC_ECUDA (-3)     /* CUDA runtime error; mpc_last_error() has the text */
#define MPC_ENOMEM (-4)
#define MPC_EIO (-5)       /* config file unreadable */
#define MPC_EPARSE (-6)    /* config file is not the JSON Config::load expects */

/* Per-problem solver status: the integers of CppAD::ipopt::solve_result<>::status_type that
 * MPC.cpp:295-303 compares against / prints ("Ipopt failed with <int>"). */
#define MPC_STATUS_NOT_DEFINED 0
#define MPC_STATUS_SUCCESS 1
#define MPC_STATUS_MAXITER_EXCEEDED 2
#define MPC_STATUS_STOP_AT_TINY_STEP 3
#define MPC_STATUS_STOP_AT_ACCEPTABLE_POINT 4
#define MPC_STATUS_LOCAL_INFEASIBILITY 5
#define MPC_STATUS_RESTORATION_FAILURE 9        /* the restoration phase itself failed (it is entered like Ipopt's) */
#define MPC_STATUS_ERROR_IN_STEP_COMPUTATION 10
#define MPC_STATUS_INVALID_NUMBER_DETECTED 11
#define MPC_STATUS_INTERNAL_ERROR 13

/* The Config:: statics the hot path reads, AFTER Config::load's unit conversions
 * (Config.cpp:39-86): SI units, radians.  POD, caller-owned, copied by mpc_create. */
typedef struct mpc_config {
  int N;                         /* Config::N      -- horizon length (2..MPC_NMAX) */
  int n_steers;                  /* Config::steers.size() */
  int n_steer_speeds;            /* Config::steerSpeeds.size() */
  int max_iter;                  /* Ipopt max_iter; replaces the wall-clock cap max_cpu_time
                                    (MPC.cpp:178), default 3000 */
  double dt;                     /* Config::dt */
  double Lf;                     /* Config::Lf */
  double cte_panic;              /* Config::ctePanic */
  double epsi_panic;             /* Config::epsiPanic */
  double max_speed;              /* Config::maxSpeed          [m/s] */
  double max_steering;           /* Config::maxSteering       [rad] */
  double max_accel;              /* Config::maxAcceleration   [m/s^2] */
  double max_decel;              /* Config::maxDeceleration   [m/s^2], negative */
  double weights[MPC_NWEIGHTS];  /* Config::weights */
  double steers[MPC_NTAB];       /* Config::steers            [rad] */
  double steer_speeds[MPC_NTAB]; /* Config::steerSpeeds       [m/s] */
  double tol;                    /* Ipopt tol, default 1e-8 */
  int watchdog_trigger;          /* Ipopt watchdog_shortened_iter_trigger, default 10 (0 = no watchdog) */
  int filter_reset_trigger;      /* Ipopt filter_reset_trigger, default 5 */
  double tiny_step_tol;          /* Ipopt tiny_step_tol, default 10 * machine epsilon (0 = off) */
  /* ---- fields below are only used by MPC::run-level helpers (not by the NLP) ---- */
  int max_fit_order;             /* Config::maxFitOrder */
  int latency_ms;                /* Config::latency */
  double max_fit_error;          /* Config::maxFitError */
  double lookahead;              /* Config::lookahead [s] */
  double ipopt_timeout;          /* Config::ipoptTimeout (kept for fidelity; not used) */
  double steer_adjust_thresh;    /* Config::steerAdjustmentThresh */
  double steer_adjust_ratio;     /* Config::steerAdjustmentRatio */
  int n_yaw_changes;             /* Config::yawChanges.size() */
  int n_yaw_change_speeds;       /* Config::yawChangeSpeeds.size() */
  double yaw_changes[MPC_NTAB];
  double yaw_change_speeds[MPC_NTAB];
} mpc_config;

typedef struct mpc_handle mpc_handle;

/* Config.cpp:5-29 -- the compiled-in defaults of the Config statics (before any load). */
int mpc_config_defaults(mpc_config *cfg);
/* Config::load(fileName), Config.cpp:31-87 -- same JSON keys, same unit conversions. */
int mpc_config_load_json(const char *path, mpc_config *cfg);
/* same, from an in-memory JSON text */
int mpc_config_parse_json(const char *text, mpc_config *cfg);

/* The controller's command line (src/mpc_main.cpp:55-79: -config <file>, -speed <mph>, -latency <ms>, -fast,
 * -stable; argv WITHOUT the program name) and its effect on the configuration at connection time
 * (mpc_main.cpp:238-246): picks the config file (config_dir stands for the reference's "..", NULL = ".."),
 * loads it, then overrides latency and max speed -- without rescaling the speed tables and without touching
 * lookahead, exactly like the reference.  Unknown options and malformed numbers return MPC_EINVAL (the
 * reference prints and exits).  config_file_out (or NULL) receives the chosen path. */
int mpc_config_from_cli(int argc, const char *const *argv, const char *config_dir, mpc_config *cfg,
                        char *config_file_out, int config_file_cap);

/* Create a solver bound to CUDA device `device` (workspace, stream-ordered work queue counter).
 * Replaces `MPC::MPC()` (MPC.cpp:160-179): the Ipopt option string becomes max_iter / tol.
 * Concurrency: handles are independent (no global mutable state; any number of handles, threads and devices), but ONE
 * call may be in flight per handle -- the launches of a solve share the handle's work queue, record buffers and scratch.
 * mpc_solve_batch is asynchronous on the caller's stream: issue the next call on the same handle to the same stream
 * (ordered after it), or use a second handle. */
int mpc_create(const mpc_config *cfg, int device, mpc_handle **out);
void mpc_destroy(mpc_handle *h);
/* replace the configuration of an existing handle (Config::load on a live controller) */
int mpc_set_config(mpc_handle *h, const mpc_config *cfg);

/*
 * Solve B independent MPC problems.  ALL POINTERS ARE DEVICE POINTERS on the handle's device;
 * the launch is asynchronous on `cuda_stream` (a cudaStream_t, NULL = default stream).
 *
 * Inputs (struct-of-arrays, batch index fastest):
 *   state   [6][B]  x, y, psi, v, cte, epsi                      (MPC.cpp:213-218)
 *   coeffs  [5][B]  polynomial, low -> high, zero padded          (RoadGeometry::polynomial)
 *   yaw_lo, yaw_hi [B]  Config::yawLow / yawHigh                  (MPC.cpp:229-232, 345-352)
 *   weights [12][B] or NULL: per-problem Config::weights override (weight sweeps)
 *   N_per   [B] or NULL: per-problem horizon (<= cfg.N); dt_per [B] or NULL: per-problem dt
 * Outputs:
 *   result  [9][B]  x1,y1,psi1,v1,cte1,epsi1,delta0,a0,cost       (MPC.cpp:322-324)
 *   traj_x, traj_y [cfg.N][B] or NULL: predicted x_i, y_i, stage 0 included (MPC.cpp:306-311);
 *                   rows >= the problem's N are left untouched
 *   full    [8*cfg.N-2][B] or NULL: solution.x in the reference's layout (MPC.cpp:189-196),
 *                   only valid when N_per is NULL
 *   status  [B]     MPC_STATUS_* ; iters [B] interior-point iterations (either may be NULL)
 */
int mpc_solve_batch(mpc_handle *h, int B,
                    const double *state, const double *coeffs,
                    const double *yaw_lo, const double *yaw_hi,
                    const double *weights, const int *N_per, const double *dt_per,
                    double *result, double *traj_x, double *traj_y, double *full,
                    int *status, int *iters, void *cuda_stream);

/* Same contract with HOST pointers: copies inputs to the device, solves, copies the outputs
 * back and synchronises.  This is the call the reference-facing C++ `MPC` shim uses.
 * Inputs in pinned, device-mapped host memory are read in place; if every output array is pinned too, the copies
 * back start before the last launch of a large batch has finished (see MPC_TAIL_LATE_COPY).  Same results either way. */
int mpc_solve_batch_host(mpc_handle *h, int B,
                         const double *state, const double *coeffs,
                         const double *yaw_lo, const double *yaw_hi,
                         const double *weights, const int *N_per, const double *dt_per,
                         double *result, double *traj_x, double *traj_y, double *full,
                         int *status, int *iters);

/* ---- all the GPUs of one box from one host thread ----------------------------------------------------------------
 * The reference is a single-threaded C++ program (src/mpc_main.cpp:51); a C++ caller of this header gets several GPUs
 * without Python or MPI: one solver handle and stream per device, the batch cut into contiguous shards
 * [g*B/G, (g+1)*B/G) (problems are independent: no exchange step, no collective), every shard's host->device copies,
 * launches and device->host copies queued asynchronously on its device's stream, one wait per device at the end.
 * HOST pointers, same layout and meaning as mpc_solve_batch_host; every output array is gathered.  Page-locked
 * (cudaMallocHost / cudaHostRegister) caller arrays let the copies of different devices overlap.  devices may name
 * a device more than once (two handles on one GPU).  mpc_multi_handle(m, g) gives shard g's handle for the
 * mpc_set_* calls. */
typedef struct mpc_multi mpc_multi;
int mpc_create_multi(const mpc_config *cfg, const int *devices, int n_devices, mpc_multi **out);
void mpc_destroy_multi(mpc_multi *m);
int mpc_multi_device_count(const mpc_multi *m);
mpc_handle *mpc_multi_handle(mpc_multi *m, int g);
int mpc_solve_batch_multi(mpc_multi *m, int B,
                          const double *state, const double *coeffs,
                          const double *yaw_lo, const double *yaw_hi,
                          const double *weights, const int *N_per, const double *dt_per,
                          double *result, double *traj_x, double *traj_y, double *full,
                          int *status, int *iters);

/* Kernel selection.  MPC_KERNEL_AUTO (default): batches of at least MPC_LANE_MIN_BATCH problems (N <= 32) or more
 * than MPC_COOP_MAX_BATCH_LONG problems (N > 32) run the throughput kernel (one problem per lane, tail handled as
 * mpc_set_tail describes); smaller batches -- where the time is set by the longest-running problem, not by
 * throughput -- run the coop kernel (one problem per group of 16/32 lanes, rows in shared memory; a lane holds one
 * stage, or two for N > 32).  The crossover was measured on B200 (profiles/r01_kernel_crossover.txt).
 * lane_threads (CTA size 32..256, multiple of 32; 0 = automatic, balanced over the SMs) and
 * lane_ctas_per_sm (0 = one) tune the persistent grid of the lane kernel. */
#define MPC_KERNEL_AUTO 0
#define MPC_KERNEL_LANE 2   /* one problem per lane; problems that need a rare branch of the algorithm (restoration phase,
                               watchdog, tiny steps, more than 8 filter entries) finish in a last launch of the coop kernel */
#define MPC_KERNEL_COOP 3   /* one problem per group of 16/32 lanes, rows in shared memory: every branch of the algorithm
                               (values 1 and 4 were the first-version warp kernel and the solo kernel, removed in round 2) */
#define MPC_LANE_MIN_BATCH 9216
#define MPC_COOP_MAX_BATCH_LONG 8192   /* AUTO, N > 32: up to this many problems run the coop kernel */
int mpc_set_kernel(mpc_handle *h, int kind, int lane_threads, int lane_ctas_per_sm);
#define MPC_HANDOFF_MAX_BATCH 300000
/* Iteration rule (off by default, `iterations` = 0).  Batches of MPC_LANE_MIN_BATCH .. MPC_HANDOFF_MAX_BATCH
 * problems: the lane kernel parks the problems that are still running after `iterations`
 * interior-point iterations and the launches that finish the tail (see mpc_set_tail) take them over.  13 is
 * the best value for the config-stable workload on its own (~6 % of the problems); with tail packing on it adds
 * nothing there and costs time on workloads whose iteration counts spread wider (weight sweeps).  All kernels
 * run identical arithmetic, so results do not depend on this setting. */
int mpc_set_handoff(mpc_handle *h, int iterations);
/* Tail packing.  A warp of the lane kernel costs the same per trip whether 32 of its lanes hold a problem or one.
 * Once the work queue is empty, a warp with at most `park_lanes` problems left (default MPC_PARK_LANES_DEFAULT,
 * 0 = off) parks them; up to `resume_launches` further launches of the lane kernel (default
 * MPC_RESUME_PHASES_DEFAULT) pick the parked problems up 32 to a warp -- each decides on the device whether there are
 * more than `resume_min_records` of them (default MPC_RESUME_MIN_DEFAULT), and otherwise returns at once -- and a
 * final launch of the coop kernel finishes what is left.  All
 * launches are on the caller's stream, results are bit-identical for every setting.  Applies to batches of at
 * least MPC_TAIL_MIN_BATCH problems.
 * flags (default MPC_TAIL_SORT_RAGGED): MPC_TAIL_SORT_RAGGED -- batches with N_per hand the problems out longest
 * horizon first, so that the lanes of a warp hold horizons of similar length; MPC_TAIL_LATE_COPY -- mpc_solve_batch_host starts its
 * device->host copies only after the final launch (by default, when every output array is pinned, device-mapped
 * host memory, they run beside the final launch and the few thousand problems that launch finishes are then
 * rewritten in the host arrays by a small kernel: same bytes, ~0.25 ms less per 64K batch). */
#define MPC_TAIL_MIN_BATCH 1024
#define MPC_PARK_LANES_DEFAULT 16
#define MPC_RESUME_PHASES_DEFAULT 3
#define MPC_RESUME_MIN_DEFAULT 8192
#define MPC_TAIL_SORT_RAGGED 1
#define MPC_TAIL_LATE_COPY 4
int mpc_set_tail(mpc_handle *h, int park_lanes, int resume_launches, int resume_min_records, int flags);
/* accounting: parked[k] = problems parked by launch k (0 = main, 1.. = resume launches) of the last lane-kernel
 * chain of this handle; synchronises the device */
int mpc_tail_counts(mpc_handle *h, int *parked, int n);

/* Multiplier outputs for the following mpc_solve_batch calls on this handle (lane and coop kernels): DEVICE
 * buffers lambda [6*cfg.N][B] (solution.lambda, rows in the reference's constraint order MPC.cpp:116-153) and
 * zl, zu [8*cfg.N-2][B] (solution.zl / zu, variable order MPC.cpp:189-196; zero where a variable is unbounded;
 * the caller clears them), for the UNSCALED problem.  With them a result can be certified as a KKT point of the
 * reference's NLP independently of the solver.  All NULL switches the outputs off.  Only with N_per == NULL. */
int mpc_set_dual_outputs(mpc_handle *h, double *lambda, double *zl, double *zu);

/* Warm start (Ipopt's warm_start_init_point) for the following mpc_solve_batch / _host / _multi calls on this handle
 * (lane and coop kernels; mpc_run_batch and mpc_rollout start cold; mpc_solve_one: mpc_set_warm_start_one).  DEVICE buffers on the
 * handle's device, in the layouts of the outputs, for the UNSCALED problem (what `full` and mpc_set_dual_outputs
 * return, so that a solution can be fed straight back):
 *   x0      [8*cfg.N-2][B]  solution.x as `full` (MPC.cpp:189-196), SI units, radians
 *   lambda0 [6*cfg.N][B]    solution.lambda as mpc_set_dual_outputs, or NULL: least-squares estimate as a cold start
 *   zl0, zu0 [8*cfg.N-2][B] solution.zl / zu as mpc_set_dual_outputs, or NULL: 1 (bound_mult_init_val) as a cold start
 * The point is pushed into the bounds with warm_start_bound_push = warm_start_bound_frac = 1e-3, the bound multipliers
 * are raised to warm_start_mult_bound_push = 1e-3 (Ipopt's defaults).  mu_init replaces Ipopt's initial barrier
 * parameter 0.1 for these solves (0 = keep 0.1; < 0 is MPC_EINVAL): a start point near the solution only helps
 * with a small one.  x0 NULL switches the warm start off (the default); the multiplier pointers are then ignored.
 * The buffers are bound to the handle and read by every later solve, so they must hold B columns for the B of that
 * solve -- for mpc_solve_batch_multi, bind each shard's handle (mpc_multi_handle(m, g)) to buffers of that shard's
 * [g*B/G, (g+1)*B/G) problems on its device.  Only with N_per == NULL: a solve with N_per and a warm start set
 * returns MPC_EINVAL. */
int mpc_set_warm_start(mpc_handle *h, const double *x0, const double *lambda0, const double *zl0, const double *zu0,
                       double mu_init);
/* Receding-horizon shift, asynchronous on cuda_stream (DEVICE pointers, layouts as above): from a solution (x,
 * lambda, zl, zu) write the next control step's start point (x0, lambda0, zl0, zu0): stages 1..N-1 move to 0..N-2;
 * the new last stage of the states continues with the increment of the old last stage, actuations and multipliers
 * repeat their last stage.  lambda / zl / zu may each be NULL together with its output.  No output may alias
 * another array of the call. */
int mpc_warm_start_shift(mpc_handle *h, int B, const double *x, const double *lambda, const double *zl,
                         const double *zu, double *x0, double *lambda0, double *zl0, double *zu0, void *cuda_stream);

/* Parametric sensitivity (Ipopt's sIPOPT) of solutions of mpc_solve_batch with respect to the initial state, for the
 * UNSCALED problem at the given point.  DEVICE pointers on the handle's device, asynchronous on cuda_stream, one launch.
 * Inputs: the problem arrays of the solve (state [6][B], coeffs [5][B], yaw_lo, yaw_hi [B], weights [12][B] or NULL,
 *   dt_per [B] or NULL; per-problem horizons are not supported), the solution full [8*cfg.N-2][B] and the multipliers
 *   lambda [6*cfg.N][B], zl, zu [8*cfg.N-2][B] in the layouts of mpc_set_dual_outputs, and status [B] or NULL.
 * Outputs, slice k = derivative with respect to state component k (x, y, psi, v, cte, epsi):
 *   dresult [6][9][B]            in the layout of `result` (x1..epsi1, delta0, a0, cost)
 *   dfull   [6][8*cfg.N-2][B] or NULL, in the layout of `full`
 * A problem whose status is neither MPC_STATUS_SUCCESS nor MPC_STATUS_STOP_AT_ACCEPTABLE_POINT (status NULL: every
 * problem is computed), or whose reduced Hessian is not positive definite at the point, gets NaN in all its outputs.
 * The derivative is that of the KKT system at the point, with the barrier term Sigma = zl / (z - lo) + zu / (hi - z) on
 * the bounds relaxed as the solver relaxes them, and FG_eval's branches frozen at the problem's own state.  The cost
 * row is grad f(z)^T dz, so it equals -lambda of the initial-condition row up to the barrier term and the solve's
 * tolerance.  Independent of the handle's kernel choice, tail settings, warm start and dual outputs; changes none. */
int mpc_solution_sensitivity(mpc_handle *h, int B, const double *state, const double *coeffs, const double *yaw_lo,
                             const double *yaw_hi, const double *weights, const double *dt_per, const double *full,
                             const double *lambda, const double *zl, const double *zu, const int *status,
                             double *dresult, double *dfull, void *cuda_stream);

/* One problem, host pointers: state[6], coeffs[5] -> result[9], traj_x/traj_y[N] (or NULL).
 * What `MPC::solve` calls once per telemetry message. */
int mpc_solve_one(mpc_handle *h, const double *state, const double *coeffs,
                  double yaw_lo, double yaw_hi,
                  double *result, double *traj_x, double *traj_y, int *status, int *iters);
/* Warm start of mpc_solve_one (off by default): with on != 0 the handle keeps each mpc_solve_one solution (x and
 * multipliers) on its device and starts the next mpc_solve_one from it, moved one stage on as mpc_warm_start_shift
 * does, with initial barrier parameter mu_init (0 = 0.1).  The first call after switching on, a call after a solve
 * that did not succeed and a call after mpc_set_config start cold.  The point stays in the previous call's
 * coordinates: it suits problems that share a frame; MPC::run re-expresses every problem in the vehicle's frame, so
 * there the primal start point is off by the vehicle's own motion. */
int mpc_set_warm_start_one(mpc_handle *h, int on, double mu_init);
/* Latency of mpc_solve_one measured in native code: `reps` calls after `warmup`, problem k % n of the given set
 * ([n][6] states, [n][MPC_NCOEF] coefficients, row-major), host clock around each call; median and 99th percentile
 * in microseconds.  bench.py reports it beside the latency seen through the Python binding. */
int mpc_measure_solve_latency(mpc_handle *h, int n, const double *state, const double *coeffs,
                              const double *yaw_lo, const double *yaw_hi, int reps, int warmup,
                              double *p50_us, double *p99_us);

/* ---- one control step around the solve: MPC::run (MPC.cpp:327-382), host-side, pure functions ---- */
#define MPC_MAX_WAYPOINTS 16
typedef struct mpc_run_aux {
  double max_yaw_change;   /* MPC.cpp:339 */
  double max_speed;        /* Vehicle::computeYawChangeSpeedLimit, MPC.cpp:340 */
  double target_speed;     /* Vehicle::computeSpeedTarget(steering, max_speed), MPC.cpp:342 */
  double fit_error;        /* sum of squared residuals of the accepted fit, RoadGeometry.cpp:30-33 */
  int fit_order;           /* 2 .. max_fit_order-1 */
} mpc_run_aux;
/* pose = (x, y, psi, v) in the global frame, steering = Vehicle::getSteering().  ptsx/ptsy (3..16
 * global waypoints) are transformed to the vehicle frame IN PLACE, as MPC.cpp:329 does (mpc_main.cpp
 * sends them back to the simulator).  Outputs the NLP inputs of mpc_solve_one. */
int mpc_run_prepare(const mpc_config *cfg, const double *pose, double steering, double *ptsx, double *ptsy,
                    int npts, double *state, double *coeffs, double *yaw_lo, double *yaw_hi, mpc_run_aux *aux);
/* result9 of the solve -> MPC::run's return vector {x1, y1, psi1, v1, steer in [-1,1], accel, cte1, epsi1}
 * (sharp-turn steering adjustment, acceleration clamp, normalisation: MPC.cpp:361-381).  v = pose[3]. */
int mpc_run_finish(const mpc_config *cfg, const mpc_run_aux *aux, double v, const double *result9, double *out8);

/* Vehicle::computeThrottle (Vehicle.cpp:81-103) and Vehicle::move (Vehicle.cpp:145-168, pose4 = x, y, psi, v in/out) */
double mpc_compute_throttle(const mpc_config *cfg, double accel, double target);
void mpc_vehicle_move(double *pose4, double steering, double accel, double length, double dt);

/* ---- the simulator protocol without the socket (src/mpc_main.cpp:26-36, 81-222; fields: DATA.md) ----
 * uWebSockets and the Unity simulator are not part of this library; these two calls are the message handler's
 * logic, so that recorded SocketIO text can be replayed through the controller. */
#define MPC_MSG_IGNORED 0     /* not a "42" event, or an event other than "telemetry": nothing is sent */
#define MPC_MSG_MANUAL 1      /* "42" event without data: the reply is 42["manual",{}] */
#define MPC_MSG_TELEMETRY 2
typedef struct mpc_telemetry {
  int kind, npts;
  double x, y, psi, speed_mph, steering_angle;     /* as sent: psi unnormalised, speed in mph, simulator steering sign */
  double ptsx[MPC_MAX_WAYPOINTS], ptsy[MPC_MAX_WAYPOINTS];
} mpc_telemetry;
/* hasData() + json::parse + field extraction (mpc_main.cpp:26-36, 92-124). Pure; no device needed. */
int mpc_telemetry_parse(const char *msg, mpc_telemetry *out);
/* One message through the controller (mpc_main.cpp:99-214): unit/sign conversion, latency compensation with the
 * fixed solve-time estimate tau_solve (the reference averages its last five measured solve times), MPC::run,
 * throttle map; writes the text the reference would send into reply ("" when nothing is sent).  *throttle_prev is
 * the reference's static throttle_value: the previous reply's throttle, updated here.  with_trajectory = the
 * PLOT_TRAJECTORY build (mpc_x/mpc_y/next_x/next_y arrays); otherwise they are 0, as the reference's NULL
 * assignments serialise. */
int mpc_telemetry_step(mpc_handle *h, const char *msg, double *throttle_prev, double tau_solve,
                       int with_trajectory, char *reply, int reply_cap);

/* MPC::run for a batch, entirely on the device (DEVICE pointers, async on cuda_stream): one kernel does the
 * pre-processing of mpc_run_prepare for every vehicle, the solve follows, one kernel does mpc_run_finish.
 *   pose [4][B] x, y, psi, v;  steering [B] or NULL;  ptsx, ptsy [npts][B] global waypoints (3..16)
 *   out8 [8][B]  MPC::run's return vector;  traj_x/traj_y [N][B] or NULL;  coeffs_out [5][B] or NULL;
 *   ptsx_v, ptsy_v [npts][B] or NULL: the waypoints in the vehicle frame (what MPC.cpp:329 leaves behind) */
int mpc_run_batch(mpc_handle *h, int B, const double *pose, const double *steering, const double *ptsx,
                  const double *ptsy, int npts, double *out8, double *traj_x, double *traj_y, double *coeffs_out,
                  double *ptsx_v, double *ptsy_v, int *status, int *iters, void *cuda_stream);

/* Closed loop for V vehicles x T control steps on the device (BASELINE config 5): the message handler of
 * src/mpc_main.cpp:113-214 with the simulator replaced by the reference's own kinematic plant.  Per step and
 * vehicle: 6-waypoint window starting at the last waypoint behind the car; psi normalised; acceleration
 * estimate (throttle - v/50)*6; if cfg.latency_ms != 0 the pose is moved ahead by lookahead + tau_solve
 * (tau_solve replaces the reference's running mean of measured solve times, which is not reproducible);
 * MPC::run; throttle = computeThrottle; the command reaches the actuators one control interval later when
 * cfg.latency_ms != 0 (the reference sleeps `latency` ms before answering), immediately otherwise; the
 * plant advances dt_ctrl with Vehicle::move and acceleration (throttle - v/50)*6.
 *   track_x, track_y [n_track] closed centre line;  veh [6][V] in/out: x, y, psi, v, steering angle [rad],
 *   last throttle;  seg [V] in/out: first waypoint of the window;  pending [2][V] in/out: command in flight
 *   (delta, throttle), required when cfg.latency_ms != 0;  rec [T][8][V] or NULL: per step cte, epsi, v,
 *   steer in [-1,1], throttle, cost, status, iterations.   DEVICE pointers; async on cuda_stream.
 * Up to MPC_ROLLOUT_PERSISTENT_MAX vehicles run as ONE launch (a lane group owns a vehicle for all T steps and
 * vehicles never wait for one another); larger fleets as three launches per control step around the throughput
 * kernel.  Same arithmetic, same bits either way (mpc_set_rollout_mode forces one or the other). */
int mpc_rollout(mpc_handle *h, int V, int T, const double *track_x, const double *track_y, int n_track,
                double *veh, int *seg, double *pending, double dt_ctrl, double tau_solve, double *rec,
                void *cuda_stream);
#define MPC_ROLLOUT_AUTO 0
#define MPC_ROLLOUT_PER_STEP 1
#define MPC_ROLLOUT_PERSISTENT 2
#define MPC_ROLLOUT_PERSISTENT_MAX 4096
int mpc_set_rollout_mode(mpc_handle *h, int mode);

/* Measure the device's FP64 FMA peak with a dependent-chain-free DFMA micro-kernel (8 independent
 * chains per thread, every SM full): the roofline denominator bench.py reports against, since
 * MEASURED_PEAKS.json holds no FP64 figure.  *tflops = 2 * FMAs / seconds / 1e12. */
int mpc_measure_fp64_peak(int device, double *tflops);

/* kernels launched by this handle since creation (bench.py's gpu_launches) */
long long mpc_launch_count(const mpc_handle *h);
/* text of the last CUDA error seen by this thread's calls ("" if none) */
const char *mpc_last_error(void);
const char *mpc_version(void);

#ifdef __cplusplus
}
#endif
#endif
