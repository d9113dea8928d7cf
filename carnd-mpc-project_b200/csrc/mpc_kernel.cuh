// mpc_kernel.cuh -- what every sm_100a kernel of the solver shares: Ipopt's constants, the launch parameters,
// the lane-group collectives and the speed-target table lookup.
//
// The kernels (mpc_lane_kernel.cuh) replace, for a whole batch at once, what the reference does once per telemetry
// message in   MPC::solve -> CppAD::ipopt::solve -> Ipopt + MUMPS   (/root/reference/src/control/MPC.cpp:183-325).
// FP64 throughout (the parity contract is 1e-4 abs / 1e-6 rel against an FP64 Ipopt solve); no tensor cores: the
// work is a chain of structured 6x8 products per horizon stage, not a dense contraction.
// (The first version of the solver -- one problem per warp, one stage per lane, mpc_ipm_kernel -- lived here until
// round 2; the coop kernel superseded it everywhere and it was removed when the restoration phase went in.)
#pragma once
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

namespace mpcb200 {

// ---- Ipopt 3.12 defaults in force in the reference (only print_level, linear_solver and
// max_cpu_time are overridden at MPC.cpp:163-178)
#define K_KAPPA_EPS 10.0
#define K_KAPPA_MU 0.2
#define K_THETA_MU 1.5
#define K_TAU_MIN 0.99
#define K_KAPPA_1 0.01
#define K_KAPPA_2 0.01
#define K_BOUND_RELAX 1e-8
#define K_S_MAX 100.0
#define K_KAPPA_SIGMA 1e10
#define K_GAMMA_THETA 1e-5
#define K_GAMMA_PHI 1e-8
#define K_S_THETA 1.1
#define K_S_PHI 2.3
#define K_ETA_PHI 1e-8
#define K_KAPPA_SOC 0.99
#define K_MAX_SOC 4
#define K_ALPHA_MIN_FRAC 0.05
#define K_DW_FIRST 1e-4
#define K_DW_MIN 1e-20
#define K_DW_MAX 1e20
#define K_DW_INC_FIRST 100.0
#define K_DW_INC 8.0
#define K_DW_DEC (1.0 / 3.0)
#define K_DUAL_INF_TOL 1.0
#define K_CONSTR_VIOL_TOL 1e-4
#define K_COMPL_INF_TOL 1e-4
#define K_ACCEPT_TOL 1e-6
#define K_ACCEPT_ITER 15
#define K_ACCEPT_CONSTR_VIOL_TOL 1e-2
#define K_ACCEPT_COMPL_INF_TOL 1e-2
#define K_CONSTR_MULT_INIT_MAX 1e3
#define K_NLP_INF 1e19
#define K_EPS 2.220446049250313e-16
#define K_NFILT 8            // filter entries a one-problem-per-lane kernel holds (a 9th hands the problem to the coop kernel)
#define K_NFILT_FULL 128     // filter entries of the coop kernel (the oracle's FILTER_MAX)
#define K_OBJ_MAX_INC 5.0
#define K_MAX_FILTER_RESETS 5
#define K_WATCHDOG_TRIAL_MAX 3
#define K_TINY_STEP_Y_TOL 1e-2
#define K_RESTO_RHO 1000.0
#define K_RESTO_KAPPA 0.9
#define K_RESTO_THETA_MAX_FACT 1e8
#define K_BOUND_MULT_RESET 1e3

struct KParams {
  int B, Nmax, max_iter, n_steers, n_steer_speeds;
  double dt, Lf, cte_panic, epsi_panic, max_speed, max_steering, max_accel, max_decel, tol;
  double weights[12];
  double steers[16];
  double steer_speeds[16];
  const double *state, *coeffs, *yaw_lo, *yaw_hi, *weights_pp;
  const int *N_pp;
  const double *dt_pp;
  double *result, *traj_x, *traj_y, *full;
  int *status, *iters;
  int *counter;
  // migration of long-running problems from the lane kernel to the coop kernel (mpc_lane_kernel.cuh)
  double *ckpt;      // [ckpt_cap] records of lane_ckpt_doubles(NS) doubles, or NULL
  int *ckpt_count;   // records written (may run past ckpt_cap: the surplus problems simply stay where they are)
  int *ckpt_next;    // next record the coop kernel takes
  int ckpt_cap, handoff_iter;
  // tail packing (mpc_lane_kernel.cuh): once the queue is empty, a warp with at most park_lanes problems left parks
  // them too; a resume launch reads the records of the previous launch (ckpt_in, *ckpt_in_count of them) packed 32 to
  // a warp and parks into the other buffer
  int park_lanes;
  const double *ckpt_in;
  const int *ckpt_in_count;
  // a chain of launches (main, resume..., final): counters [2j] = records parked by launch j, [2j + 1] = cursor of
  // launch j over its input; the two record buffers; this launch's position, the final launch's, and the number of
  // records below which a resume launch leaves them to the next launch
  int *chain_counts;
  double *chain_buf0, *chain_buf1;
  int chain_pos, chain_last, resume_min;
  const int *perm;   // order in which the work queue hands out the problems (ragged batches: longest horizon first), or NULL
  // optional multiplier outputs (solution.lambda / zl / zu of CppAD::ipopt::solve_result), unscaled
  double *dual_lam, *dual_zl, *dual_zu;
  // Ipopt options with a counterpart here (mpc_config): watchdog_shortened_iter_trigger, filter_reset_trigger, tiny_step_tol
  int watchdog_trigger, filter_reset_trigger;
  double tiny_step_tol;
  // problems a one-problem-per-lane kernel hands to the coop kernel because they need the rare branches of the
  // algorithm (restoration phase, watchdog, a big filter, tiny steps) and no record slot was free: their indices; the
  // final launch of the chain solves them from the start (same arithmetic, same path, same bits)
  int *restart_list, *restart_count, *restart_cursor;
  // coop kernels: global scratch per lane group (watchdog backup, restoration-phase rows), scratch_stride doubles each
  double *scratch;
  long long scratch_stride;
  // warm start (mpc_set_warm_start): start point in the layouts of `full` and of the multiplier outputs, unscaled
  // problem; ws_x == NULL is a cold start.  ws_lam / ws_zl / ws_zu may be NULL (cold-start estimate of that part).
  // ws_mu: the initial barrier parameter of a warm start (Ipopt's mu_init).
  const double *ws_x, *ws_lam, *ws_zl, *ws_zu;
  double ws_mu;
};

// Ipopt's warm_start_init_point options at their defaults (IpWarmStartIterInitializer)
#define K_WS_BOUND_PUSH 1e-3        // warm_start_bound_push
#define K_WS_BOUND_FRAC 1e-3        // warm_start_bound_frac
#define K_WS_MULT_BOUND_PUSH 1e-3   // warm_start_mult_bound_push

// ------------------------------------------------------------------------------------------------
// group (G lanes) collectives: xor butterflies give every lane the bit-identical result, which
// keeps all control flow of a problem uniform across its lanes
// ------------------------------------------------------------------------------------------------
template <int G> __device__ __forceinline__ double gsum(double v, unsigned m) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(m, v, o, G);
  return v;
}
__device__ __forceinline__ double nanmax(double a, double b) { return (a > b || a != a) ? a : b; }
template <int G> __device__ __forceinline__ double gmax(double v, unsigned m) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = nanmax(v, __shfl_xor_sync(m, v, o, G));
  return v;
}
template <int G> __device__ __forceinline__ double gmin(double v, unsigned m) {
#pragma unroll
  for (int o = G / 2; o > 0; o >>= 1) v = fmin(v, __shfl_xor_sync(m, v, o, G));
  return v;
}

// Vehicle::computeSpeedTarget(AD<double>, double), Vehicle.cpp:50-64
__device__ inline double speed_target(const KParams &P, double angle, double mx) {
  double y = fabs(angle);
  double back = P.steer_speeds[P.n_steer_speeds - 1];
  for (int i = 0; i < P.n_steers; i++) {
    if (y <= P.steers[i]) {
      if (P.n_steer_speeds > i) return P.steer_speeds[i] < mx ? P.steer_speeds[i] : mx;
      return back < mx ? back : mx;
    }
  }
  return back < mx ? back : mx;
}
}  // namespace mpcb200
