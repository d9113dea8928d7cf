// mpc_lane_kernel.cuh -- the solver: one source, two mappings onto the machine.
//
// The NLP of FG_eval (/root/reference/src/control/MPC.cpp:50-154) with hand-derived derivatives, Ipopt's primal-dual
// filter line-search iteration (Ipopt 3.12 defaults, MPC.cpp:160-179) and a stage-wise Riccati factorisation of the
// block-banded KKT system instead of MUMPS (MPC.cpp:175), written once as `struct Lane` and instantiated as
//   mpc_lane_kernel         one problem per LANE, rows in thread-private memory: the throughput kernel (common path of the
//                           algorithm; a problem that needs a rare branch is handed to the coop kernel)
//   mpc_coop_kernel etc.    one problem per GROUP of 16/32 lanes, rows in shared memory: every branch of the algorithm
//                           (restoration phase, watchdog, ...); single solves, small batches, closed loops, the tail of a batch
// Same floating-point operations in the same order per problem either way, so a problem can move between them at any trip
// boundary without changing a bit of its result.
//
// A batch of 64K problems has far more problem-level parallelism than the chip has lanes, so in the lane kernel every lane
// owns one problem, runs the whole recursion on its own registers and keeps the per-stage iterate in thread-private
// (lane-interleaved, hence fully coalesced) memory.  (The first version -- one problem per warp, one stage per lane -- kept
// 17 of 32 lanes busy and spent most of its issue slots on shuffles: profiles/r01_v1_*.  Removed in round 2.)
//
// Lanes of a warp work on different problems with different iteration counts.  To keep them
// converged the solver is written as a state machine whose trip has a fixed shape
//        [evaluate a point] -> [accept / update / KKT errors / mu] -> [Riccati] -> [forward + costate]
// and every lane executes the slots its state needs.  A lane that finishes pulls the next problem
// from a global counter, so the spread of iteration counts (10 typical, 50 worst) costs nothing.
// The rare paths (inertia correction 0.3 % of iterations, second-order correction and backtracking
// ~0.002 %) simply take extra trips.
//
// Memory.  The per-stage state of a problem does not fit in registers, and the state of all resident
// lanes should fit in the 126 MB L2 or every sweep streams it through HBM (profiles/r01_v2_*: 16.5 GB
// of DRAM traffic per 64K batch; today 8.8 GB).  So only what cannot be recomputed cheaply is stored -- iterate
// (x, lambda, z), step, Riccati gains, and the trig/polynomial values and residuals at the iterate:
// 56 doubles per stage.  Slack reciprocals, trial-point values and the new multipliers are recomputed
// (the FP64 pipe has the headroom); the costate recursion that yields the new multipliers runs inside
// the sweep that accepts the step, the step-length ratios inside the forward sweep.
#pragma once
#include "mpc_kernel.cuh"

namespace mpcb200 {

enum {
  LM_IDLE = 0,    // no problem: fetch one
  LM_EV0,         // evaluate the start point
  LM_LSQ,         // least-squares multiplier estimate (Riccati with H = I)
  LM_LSQ_DONE,    // take the multipliers, compute the KKT error, go to NEWTON
  LM_LSQ_ZERO,    // the estimate was rejected (|lambda| > 1e3): multipliers = 0, KKT error, go to NEWTON
  LM_NEWTON,      // factor (with inertia correction) and solve for the search direction
  LM_TRIAL,       // evaluate x + alpha dx and test it against the filter
  LM_SOC,         // solve with the second-order-corrected right-hand side
  LM_SOC_TRIAL,   // evaluate the corrected trial point
  LM_RESOLVE,     // SOC failed: recompute the uncorrected direction, then backtrack
  LM_FINISH,      // write the outputs
  LM_DONE,        // queue empty
  LM_LSFAIL       // the step size fell below alpha_min: Ipopt's restoration phase (coop kernel only)
};

// constants of one problem (thread-private)
enum { LC_DT = 0, LC_DTLF, LC_SF, LC_CW, LC_WC2, LC_WE2, LC_WV2, LC_VREF, LC_WD2, LC_WC2_0, LC_WE2_0,
       LC_VREF_0, LC_NV2_0, LC_C0, LC_S0 = LC_C0 + 5, LC_LO = LC_S0 + 6, LC_HI = LC_LO + 4,
       LC_LO0 = LC_HI + 4, LC_HI0 = LC_LO0 + 4, LC_SIZE = LC_HI0 + 4 };

// 1/a for a normal, finite a (slacks, 1 + f'^2, pivots): hardware seed (20 bits) + two Newton steps.  Accurate to
// ~1 ulp (measured on B200: seed 1e-6, one step 1e-12, two steps exact to rounding); a third of the instructions of the correctly-rounded division, which dominated the sweeps.
__device__ __forceinline__ double rcp(double a) {
  double x;
  asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(x) : "d"(a));
  double e = fma(-a, x, 1.0);
  x = fma(x, e, x);
  e = fma(-a, x, 1.0);
  return fma(x, e, x);
}
// min / max without fmin/fmax's NaN handling: FP64 has no min/max instruction and the library versions
// expand to ~13 instructions each; the sweeps take ~50 of them per stage.  NaN in `b` is returned.
__device__ __forceinline__ double dmin(double a, double b) { return a < b ? a : b; }
__device__ __forceinline__ double dmax(double a, double b) { return a > b ? a : b; }

// per-stage row layout (doubles)
enum { ST_S = 0,      // iterate: x, y, psi, v, cte, epsi
       ST_U = 6,      //          delta, a
       ST_LAM = 8,    //          multipliers of the constraint defining s_i
       ST_ZL = 14,    //          bound multipliers of psi, v, delta, a
       ST_ZU = 18,
       ST_TG = 22,    // sin/cos psi, sin/cos epsi, f', f'', a61, g3 at the iterate
       ST_CN = 30,    // c_{i+1} at the iterate
       ST_DS = 36,    // primal search direction
       ST_DU = 42,
       ST_KG = 44,    // Riccati gains: K0[x,y,psi,v,dprev], K1[..], k0, k1
       ST_CS = 56,    // second-order-correction right-hand side (rare path only)
       ST_KEEP = 62,  // what is live at a trip boundary: the rows of the one-problem-per-lane kernels, and of a record
       ST_ROW = 62,   // thread-private rows (a multiple of 16 bytes that is not one of 64)
       ST_TT = 62,    // coop kernel only: TG / CN at the trial point, handed from the evaluation to the acceptance sweep
       ST_CT = 70,    //   (the one-problem-per-lane kernels recompute them there instead: 14 doubles less per stage to stream)
       ST_LH = 76,    // coop kernel only: StageLin (10) + StageHess (18) of the stage, built one stage per lane
       ST_ROW_SH = 106 };   // shared-memory rows: 104 used; 106 keeps neighbouring lanes' rows 2-way bank-conflict free
template <int NS, bool SH, bool PAR> struct LaneRows { typedef double type[NS][ST_ROW]; enum { ROW = ST_ROW }; };
template <int NS> struct LaneRows<NS, true, true> { typedef double (*type)[ST_ROW_SH]; enum { ROW = ST_ROW_SH }; };
template <int NS> struct LaneRows<NS, true, false> { typedef double (*type)[ST_ROW]; enum { ROW = ST_ROW }; };

struct StageLin { double a13, a14, a23, a24, a34, b3, a51, a54, a56, a61; };
struct StageHess { double qxx, qyy, qpp, qpv, qvv, qve, qcc, qee, svd, rdd, raa, gp, gv, gc, ge, gdp, gd, ga; };

template <int NS, bool SH, bool PAR = SH>
struct Lane {
  // Per-stage data: one row of ST_ROW doubles per horizon stage (offsets ST_*; 56 of them are touched on the common
  // path).  SH = false: thread-private memory (one problem per lane; rows 16-byte aligned, so neighbouring doubles pair
  // into 128-bit local accesses).  SH = true: a pointer into shared memory.  PAR = true (needs SH): one problem per lane
  // GROUP, the sweeps that are parallel over the horizon run one stage per lane (mpc_coop_kernel).
  enum { NS_GROUP = PAR ? (NS <= 16 ? 16 : 32) : 1, NPASS = (NS + NS_GROUP - 1) / NS_GROUP };   // stages per lane of a group
  // FULL: the kernel carries every branch of the algorithm.  The one-problem-per-lane kernel keeps to the branches
  // that occur on almost every problem (Newton step, inertia correction, second-order correction, backtracking); a
  // problem that needs another one -- restoration phase, watchdog, tiny step, a 9th filter entry -- sets `escalate`
  // at a point where nothing of the trip has been committed, and the coop kernel repeats that trip and goes on.
  static constexpr bool FULL = PAR;
  enum { NFILT = PAR ? K_NFILT_FULL : K_NFILT };
  typedef typename LaneRows<NS, SH, PAR>::type Rows;
  alignas(16) Rows ST;
  alignas(16) double PC[LC_SIZE];
  alignas(16) double FLT[2 * NFILT];
  double c0[6], c0t[6], cs0[6];
  // ---- lane group (coop kernel): this lane's index in its group, group size, member mask; (0, 1, -) for
  // the one-problem-per-lane kernel
  int g0, gstep;
  unsigned gm;
  __device__ __forceinline__ void gsync() const { if (PAR) __syncwarp(gm); }
  // ---- scalars ----
  int m1, m3;
  bool solve_ok, lh_stale, no_handoff;
  int b, N, mode, status, iter, accept_cnt, nfilt, ntrial, soc_cnt;
  // line-search state beyond one iteration (Ipopt's BacktrackingLineSearch / FilterLSAcceptor members)
  int wd_short;                    // watchdog_shortened_iter_: successive iterations that needed backtracking
  int trips;                       // trips spent on this problem in this kernel (progress guard)
  int n_filter_resets, succ_filter_rej;
  bool last_rej_filter, acceptable_now, escalate, tiny_screen;
  double tiny_tol;                 // KParams::tiny_step_tol
  // FULL only
  bool in_watchdog, wd_skip, force_accept, tiny_last, tiny_flag, was_tiny;
  int wd_trial;
  double alpha_max, wd_alpha_test, tiny_all, dy_max;
  double *scratch;                 // this group's global scratch (watchdog backup, restoration rows)
  double mu, tau, theta_min, theta_max, dw, dw_last, dw_used;
  double alpha, alpha_z, alpha_test, alpha_soc, alpha_min;
  double ls_theta, ls_phi, ls_gbd, pow_gbd, pow_theta;
  double fx, lsum, theta, ft, lt, tht, theta_soc_old;
  double dinf, cviol, amin, amax, lam1, z1, lsq_lmax, gbd_new;

  __device__ __forceinline__ double wc2(int i) const { return i == 0 ? PC[LC_WC2_0] : PC[LC_WC2]; }
  __device__ __forceinline__ double we2(int i) const { return i == 0 ? PC[LC_WE2_0] : PC[LC_WE2]; }
  __device__ __forceinline__ double vref(int i) const { return i == 0 ? PC[LC_VREF_0] : PC[LC_VREF]; }
  __device__ __forceinline__ double nv2(int i) const { return i == 0 ? PC[LC_NV2_0] : 0.0; }

  // ------------------------------------------------------------------------------------------
  // problem set-up: MPC.cpp:204-281 (start point, bounds), frozen branches of FG_eval at the
  // start point (MPC.cpp:72,79,87,89), Ipopt's objective scaling and bound relaxation / push
  // ------------------------------------------------------------------------------------------
  // WARM: the kernel is instantiated for warm-started launches (KParams::ws_x); the cold instantiations compile to
  // the code they had before the warm start existed (the persistent lane kernel is sensitive to its code size)
  template <bool WARM = false>
  __device__ void init(const KParams &P, int b_) {
    b = b_;
    const int B = P.B;
    N = P.N_pp ? P.N_pp[b] : P.Nmax;
    if (N > NS) N = NS;
    if (N > P.Nmax) N = P.Nmax;
    if (N < 2) N = 2;
    double w[12];
#pragma unroll
    for (int k = 0; k < 12; k++) w[k] = P.weights_pp ? P.weights_pp[(size_t)k * B + b] : P.weights[k];
#pragma unroll
    for (int k = 0; k < 6; k++) PC[LC_S0 + k] = P.state[(size_t)k * B + b];
#pragma unroll
    for (int k = 0; k < 5; k++) PC[LC_C0 + k] = P.coeffs[(size_t)k * B + b];
    const double ylo = P.yaw_lo[b], yhi = P.yaw_hi[b];
    const double dt = P.dt_pp ? P.dt_pp[b] : P.dt;
    const double cte0 = PC[LC_S0 + 4], epsi0 = PC[LC_S0 + 5], psi0 = PC[LC_S0 + 2], v0 = PC[LC_S0 + 3];
    const double wc0 = fabs(cte0) < P.cte_panic ? w[0] : w[11];
    const double wcN = 0.0 < P.cte_panic ? w[0] : w[11];
    const double we0 = fabs(epsi0) > P.epsi_panic ? w[10] : w[1];
    const double weN = 0.0 > P.epsi_panic ? w[10] : w[1];
    const double vr0 = speed_target(P, psi0, P.max_speed), vrN = speed_target(P, 0.0, P.max_speed);
    const double nvw0 = v0 < 0.0 ? w[9] : 0.0;
    double gmx = fmax(fabs(2.0 * wc0 * cte0), fabs(2.0 * we0 * epsi0));
    gmx = fmax(gmx, fabs(2.0 * w[2] * (v0 - vr0) + 2.0 * nvw0 * v0));
    gmx = fmax(gmx, fabs(2.0 * w[2] * vrN));
    const double sf = gmx > 100.0 ? fmax(100.0 / gmx, 1e-8) : 1.0;
    PC[LC_DT] = dt;
    PC[LC_DTLF] = dt / P.Lf;
    PC[LC_SF] = sf;
    PC[LC_CW] = 2.0 * sf * w[4];
    PC[LC_WC2] = 2.0 * sf * wcN; PC[LC_WE2] = 2.0 * sf * weN; PC[LC_WV2] = 2.0 * sf * w[2];
    PC[LC_VREF] = vrN; PC[LC_WD2] = 2.0 * sf * w[3];
    PC[LC_WC2_0] = 2.0 * sf * wc0; PC[LC_WE2_0] = 2.0 * sf * we0; PC[LC_VREF_0] = vr0;
    PC[LC_NV2_0] = 2.0 * sf * nvw0;
    const double lo0[4] = {ylo, -P.max_speed, -P.max_steering, P.max_decel};
    const double hi0[4] = {yhi, P.max_speed, P.max_steering, P.max_accel};
    double x0[4];   // pushed start values of psi, v, delta, a for stages >= 1 (start point 0)
    double x00[2];  // pushed psi, v of stage 0
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const double lo = lo0[k] - fmin(K_CONSTR_VIOL_TOL, K_BOUND_RELAX * fmax(1.0, fabs(lo0[k])));
      const double hi = hi0[k] + fmin(K_CONSTR_VIOL_TOL, K_BOUND_RELAX * fmax(1.0, fabs(hi0[k])));
      PC[LC_LO0 + k] = lo0[k]; PC[LC_HI0 + k] = hi0[k]; PC[LC_LO + k] = lo; PC[LC_HI + k] = hi;
      const double span = hi - lo;
      const double pl = fmin(K_KAPPA_1 * fmax(1.0, fabs(lo)), K_KAPPA_2 * span);
      const double pu = fmin(K_KAPPA_1 * fmax(1.0, fabs(hi)), K_KAPPA_2 * span);
      double v = 0.0;
      if (v < lo + pl) v = lo + pl;
      if (v > hi - pu) v = hi - pu;
      x0[k] = v;
      if (k < 2) {
        double v2 = k == 0 ? psi0 : v0;
        if (v2 < lo + pl) v2 = lo + pl;
        if (v2 > hi - pu) v2 = hi - pu;
        x00[k] = v2;
      }
    }
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
#pragma unroll
      for (int k = 0; k < 6; k++) { ST[i][ST_S + k] = (i == 0) ? PC[LC_S0 + k] : 0.0; ST[i][ST_LAM + k] = 0.0; ST[i][ST_DS + k] = 0.0; }
#pragma unroll
      for (int k = 0; k < 8; k++) ST[i][ST_TG + k] = 0.0;   // read (times alpha = 0) by the first advance sweep
      ST[i][ST_S + 2] = i == 0 ? x00[0] : x0[0];
      ST[i][ST_S + 3] = i == 0 ? x00[1] : x0[1];
      ST[i][ST_U + 0] = x0[2]; ST[i][ST_U + 1] = x0[3];
      ST[i][ST_DU + 0] = 0.0; ST[i][ST_DU + 1] = 0.0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        const bool valid = k < 2 || i < N - 1;
        ST[i][ST_ZL + k] = valid ? 1.0 : 0.0;
        ST[i][ST_ZU + k] = valid ? 1.0 : 0.0;
      }
    }
    mu = 0.1;
    tau = fmax(K_TAU_MIN, 1.0 - mu);
    dw = 0.0; dw_last = 0.0; dw_used = 0.0;
    nfilt = 0; iter = 0; accept_cnt = 0; status = 0; ntrial = 0; soc_cnt = 0;
    alpha = 0.0; alpha_z = 0.0;
    reset_line_search();
    n_filter_resets = 0; acceptable_now = false; escalate = false; tiny_screen = false; tiny_flag = false;
    force_accept = false; wd_skip = false; was_tiny = false; wd_trial = 0; trips = 0;
    tiny_tol = P.tiny_step_tol;
    mode = LM_EV0;
    gsync();
    if (WARM && P.ws_x) warm_init(P);
  }
  // Ipopt's warm_start_init_point: the caller's primal point pushed into the bounds with warm_start_bound_push /
  // warm_start_bound_frac (the formula of the cold start with 1e-3 for 1e-2), the caller's multipliers taken over to
  // the gradient-scaled problem -- times the objective factor sf, the factor write_outputs divides out; constraints
  // and variables are not scaled -- with the bound multipliers raised to at least warm_start_mult_bound_push.
  // lambda without a caller's value is the least-squares estimate (trip_accept), zl / zu without one stay at 1.
  // The scaling factor and the frozen branches of FG_eval stay those of the problem's own start point (above), so
  // a warm-started solve iterates on the same scaled problem as a cold one.
  __device__ void warm_init(const KParams &P) {
    const size_t B = (size_t)P.B;
    const int Nf = P.Nmax;
    const double sf = PC[LC_SF];
    double pl[4], pu[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const double lo = PC[LC_LO + k], hi = PC[LC_HI + k], span = hi - lo;
      pl[k] = fmin(K_WS_BOUND_PUSH * fmax(1.0, fabs(lo)), K_WS_BOUND_FRAC * span);
      pu[k] = fmin(K_WS_BOUND_PUSH * fmax(1.0, fabs(hi)), K_WS_BOUND_FRAC * span);
    }
    // rows of the reference's layout (MPC.cpp:189-196) holding psi, v, delta, a of stage i
    const int zrow[4] = {2 * Nf, 3 * Nf, 6 * Nf, 7 * Nf - 1};
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const bool hasu = i < N - 1;
      double v[8];
#pragma unroll
      for (int k = 0; k < 6; k++) v[k] = P.ws_x[(size_t)(k * Nf + i) * B + b];
      v[6] = hasu ? P.ws_x[(size_t)(6 * Nf + i) * B + b] : ST[i][ST_U + 0];
      v[7] = hasu ? P.ws_x[(size_t)(7 * Nf - 1 + i) * B + b] : ST[i][ST_U + 1];
#pragma unroll
      for (int k = 0; k < 4; k++) {
        double &x = v[k < 2 ? k + 2 : k + 4];
        if (k >= 2 && !hasu) continue;
        if (x < PC[LC_LO + k] + pl[k]) x = PC[LC_LO + k] + pl[k];
        if (x > PC[LC_HI + k] - pu[k]) x = PC[LC_HI + k] - pu[k];
      }
#pragma unroll
      for (int k = 0; k < 6; k++) ST[i][ST_S + k] = v[k];
      ST[i][ST_U + 0] = v[6]; ST[i][ST_U + 1] = v[7];
      if (P.ws_lam) {
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_LAM + k] = P.ws_lam[(size_t)(k * Nf + i) * B + b] * sf;
      }
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (k >= 2 && !hasu) continue;
        const size_t at = (size_t)(zrow[k] + i) * B + b;
        if (P.ws_zl) ST[i][ST_ZL + k] = fmax(P.ws_zl[at] * sf, K_WS_MULT_BOUND_PUSH);
        if (P.ws_zu) ST[i][ST_ZU + k] = fmax(P.ws_zu[at] * sf, K_WS_MULT_BOUND_PUSH);
      }
    }
    mu = P.ws_mu;
    tau = fmax(K_TAU_MIN, 1.0 - mu);
    gsync();
  }
  // BacktrackingLineSearch::Reset (at every change of the barrier parameter): empty filter, no watchdog
  __device__ __forceinline__ void reset_line_search() {
    nfilt = 0; succ_filter_rej = 0; last_rej_filter = false;
    wd_short = 0; in_watchdog = false; tiny_last = false;
  }


  // F(s, u): right-hand sides of MPC.cpp:144-152 with polyeval/polyder (utils.h:28-47), and the
  // transcendental/polynomial values the derivatives need (App. A.4 of SURVEY.md)
  __device__ __forceinline__ void point_eval(const double *s, double u0, double u1, double *tg, double *F) const {
    const double dt = PC[LC_DT], dtLf = PC[LC_DTLF];
    const double c0_ = PC[LC_C0], c1_ = PC[LC_C0 + 1], c2_ = PC[LC_C0 + 2], c3_ = PC[LC_C0 + 3], c4_ = PC[LC_C0 + 4];
    double sp, cp, se, ce;
    sincos(s[2], &sp, &cp);
    sincos(s[5], &se, &ce);
    const double x = s[0];
    const double f = fma(fma(fma(fma(c4_, x, c3_), x, c2_), x, c1_), x, c0_);
    const double f1 = fma(fma(fma(4.0 * c4_, x, 3.0 * c3_), x, 2.0 * c2_), x, c1_);
    const double f2 = fma(fma(12.0 * c4_, x, 6.0 * c3_), x, 2.0 * c2_);
    const double f3 = fma(24.0 * c4_, x, 6.0 * c3_);
    const double q = fma(f1, f1, 1.0), iq = rcp(q);
    tg[0] = sp; tg[1] = cp; tg[2] = se; tg[3] = ce; tg[4] = f1; tg[5] = f2;
    tg[6] = -f2 * iq;                                    // d/dx of -atan(f')
    tg[7] = fma(f3, q, -(2.0 * f1 * f2 * f2)) * iq * iq;      // and its derivative
    const double vdt = s[3] * dt;
    F[0] = fma(cp, vdt, s[0]);
    F[1] = fma(sp, vdt, s[1]);
    F[2] = fma(u0 * s[3], dtLf, s[2]);
    F[3] = fma(u1, dt, s[3]);
    F[4] = fma(se, vdt, f - s[1]);
    F[5] = F[2] - atan(f1);
  }
  __device__ __forceinline__ void lin_at(const double *tg, double v, double d0, StageLin &L) const {
    const double dt = PC[LC_DT], dtLf = PC[LC_DTLF], vdt = v * dt;
    L.a13 = -vdt * tg[0]; L.a14 = dt * tg[1]; L.a23 = vdt * tg[1]; L.a24 = dt * tg[0];
    L.a34 = d0 * dtLf; L.b3 = v * dtLf; L.a51 = tg[4]; L.a54 = dt * tg[2]; L.a56 = vdt * tg[3];
    L.a61 = tg[6];
  }
  // slack reciprocals of psi, v, delta, a at a point
  __device__ __forceinline__ void slack_rcp(double psi, double v, double u0, double u1, bool hasu, double *il, double *iu) const {
    il[0] = rcp(psi - PC[LC_LO]); iu[0] = rcp(PC[LC_HI] - psi);
    il[1] = rcp(v - PC[LC_LO + 1]); iu[1] = rcp(PC[LC_HI + 1] - v);
    if (hasu) {
      il[2] = rcp(u0 - PC[LC_LO + 2]); iu[2] = rcp(PC[LC_HI + 2] - u0);
      il[3] = rcp(u1 - PC[LC_LO + 3]); iu[3] = rcp(PC[LC_HI + 3] - u1);
    } else {
      il[2] = iu[2] = il[3] = iu[3] = 0.0;
    }
  }
  // Hessian of the Lagrangian + barrier Sigma + dw on the primal diagonal, gradient of the barrier
  // objective, all from register values.  ls: the least-squares multiplier system (Hessian = I,
  // gradient = grad f - zl + zu).  ln = multipliers of stage i+1, dprev = delta_{i-1}.
  __device__ __forceinline__ void hess_at(int i, bool ls, double dwv, const double *tg, double v, double c, double e,
                                          double d0, double dprev, const double *ln, const double *zl, const double *zu,
                                          const double *il, const double *iu, StageHess &H) const {
    const bool hasu = i < N - 1;
    const bool cpl = hasu && i >= 1;
    const double dt = PC[LC_DT], dtLf = PC[LC_DTLF], cw = PC[LC_CW], wd2 = PC[LC_WD2], wv2 = PC[LC_WV2];
    double sig[4], gb[4];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      sig[k] = fma(zl[k], il[k], zu[k] * iu[k]);
      gb[k] = ls ? (zu[k] - zl[k]) : mu * (iu[k] - il[k]);
    }
    H.gp = gb[0];
    H.gv = fma(nv2(i), v, wv2 * (v - vref(i))) + gb[1];
    H.gc = wc2(i) * c;
    H.ge = we2(i) * e;
    H.gdp = 0.0; H.gd = 0.0; H.ga = 0.0;
    if (hasu) {
      const double dd = cpl ? d0 - dprev : 0.0;
      H.gdp = -cw * dd;
      H.gd = fma(cw, dd, wd2 * d0) + gb[2];
      H.ga = gb[3];
    }
    if (ls) {
      H.qxx = 1.0; H.qyy = 1.0; H.qpp = 1.0; H.qpv = 0.0; H.qvv = 1.0; H.qve = 0.0; H.qcc = 1.0; H.qee = 1.0;
      H.svd = 0.0; H.rdd = 1.0; H.raa = 1.0;
      return;
    }
    H.qyy = dwv;
    H.qvv = wv2 + nv2(i) + sig[1] + dwv;
    H.qcc = wc2(i) + dwv;
    if (hasu) {
      const double vdt = v * dt;
      H.qxx = fma(ln[5], tg[7], -(ln[4] * tg[5])) + dwv;
      H.qpp = fma(fma(ln[0], tg[1], ln[1] * tg[0]), vdt, sig[0]) + dwv;
      H.qpv = fma(ln[0], tg[0], -(ln[1] * tg[1])) * dt;
      H.qve = -ln[4] * tg[3] * dt;
      H.qee = fma(ln[4] * tg[2], vdt, we2(i)) + dwv;
      H.svd = -(ln[2] + ln[5]) * dtLf;
      H.rdd = wd2 + (cpl ? cw : 0.0) + sig[2] + dwv;
      H.raa = sig[3] + dwv;
    } else {
      H.qxx = dwv; H.qpp = sig[0] + dwv; H.qpv = 0.0; H.qve = 0.0; H.qee = we2(i) + dwv;
      H.svd = 0.0; H.rdd = 0.0; H.raa = 0.0;
    }
  }

  // ------------------------------------------------------------------------------------------
  // slot 1 (forward sweep): ||c||_1, scaled objective and log-barrier sum at x + a*dx; the residuals and
  // trig/polynomial values of the trial point are kept (TT, CT) and become the iterate's on acceptance
  // ------------------------------------------------------------------------------------------
  __device__ void eval_sweep(double a) {
    if (PAR) { eval_par(a); return; }
    const double lo_p = PC[LC_LO], hi_p = PC[LC_HI], lo_v = PC[LC_LO + 1], hi_v = PC[LC_HI + 1];
    const double lo_d = PC[LC_LO + 2], hi_d = PC[LC_HI + 2], lo_a = PC[LC_LO + 3], hi_a = PC[LC_HI + 3];
    double F[6] = {0, 0, 0, 0, 0, 0};
    double th = 0.0, fl = 0.0, ll = 0.0, dprev = 0.0;
    // the rows are a long way off (L2 or DRAM): the iterate and step of stage i+1 are loaded at the top of iteration i
    // and only touched at the top of iteration i+1, so that their latency runs under the transcendental work of
    // stage i instead of being waited for
    double sl[6], dl[6], ul0, ul1, dul0, dul1;
#pragma unroll
    for (int k = 0; k < 6; k++) { sl[k] = ST[0][ST_S + k]; dl[k] = ST[0][ST_DS + k]; }
    ul0 = ST[0][ST_U + 0]; ul1 = ST[0][ST_U + 1]; dul0 = ST[0][ST_DU + 0]; dul1 = ST[0][ST_DU + 1];
#pragma unroll 1
    for (int i = 0; i < N; i++) {
      double s[6];
#pragma unroll
      for (int k = 0; k < 6; k++) s[k] = fma(a, dl[k], sl[k]);
      const double u0 = fma(a, dul0, ul0), u1 = fma(a, dul1, ul1);
      {
        const int j = i + 1 < N ? i + 1 : i;
#pragma unroll
        for (int k = 0; k < 6; k++) { sl[k] = ST[j][ST_S + k]; dl[k] = ST[j][ST_DS + k]; }
        ul0 = ST[j][ST_U + 0]; ul1 = ST[j][ST_U + 1]; dul0 = ST[j][ST_DU + 0]; dul1 = ST[j][ST_DU + 1];
      }
      if (i == 0) {
#pragma unroll
        for (int k = 0; k < 6; k++) { const double c = s[k] - PC[LC_S0 + k]; c0t[k] = c; th += fabs(c); }
      } else {
#pragma unroll
        for (int k = 0; k < 6; k++) th += fabs(s[k] - F[k]);
      }
      const double dv = s[3] - vref(i);
      fl = fma(0.5, fma(nv2(i) * s[3], s[3], fma(PC[LC_WV2] * dv, dv, fma(we2(i) * s[5], s[5], wc2(i) * s[4] * s[4]))), fl);
      double prod = (s[2] - lo_p) * (hi_p - s[2]) * (s[3] - lo_v) * (hi_v - s[3]);
      if (i < N - 1) {
        double tg[8];
        point_eval(s, u0, u1, tg, F);
        fl = fma(0.5 * PC[LC_WD2] * u0, u0, fl);
        if (i >= 1) { const double dd = u0 - dprev; fl = fma(0.5 * PC[LC_CW] * dd, dd, fl); }
        dprev = u0;
        prod *= (u0 - lo_d) * (hi_d - u0) * (u1 - lo_a) * (hi_a - u1);
      }
      ll += log(prod);
    }
    ft = fl; lt = ll; tht = th;
  }
  // the same evaluation with one stage per lane of the group: the residual of the constraint that defines
  // s_i needs F(s_{i-1}, u_{i-1}) from the lane below; the three sums are butterfly reductions
  __device__ void eval_par(double a) {
    if (NPASS > 1) { eval_parN(a); return; }
    const int G = PAR ? NS_GROUP : 1;
    const int i = g0;
    const bool act = i < N, hasu = i < N - 1;
    const int ii = act ? i : 0;
    double s[6], F[6] = {0, 0, 0, 0, 0, 0}, tg[8], u0 = 0.0, u1 = 0.0;
#pragma unroll
    for (int k = 0; k < 6; k++) s[k] = fma(a, ST[ii][ST_DS + k], ST[ii][ST_S + k]);
    double fl = 0.0, ll = 0.0, th = 0.0;
    if (hasu) {
      u0 = fma(a, ST[i][ST_DU + 0], ST[i][ST_U + 0]);
      u1 = fma(a, ST[i][ST_DU + 1], ST[i][ST_U + 1]);
      point_eval(s, u0, u1, tg, F);
#pragma unroll
      for (int k = 0; k < 8; k++) ST[i][ST_TT + k] = tg[k];
    }
    const double dprev = __shfl_up_sync(gm, u0, 1, G);
#pragma unroll
    for (int k = 0; k < 6; k++) {
      const double Fp = __shfl_up_sync(gm, F[k], 1, G);
      // every lane keeps the stage-0 residual (it is part of the uniform per-problem state)
      c0t[k] = fma(a, ST[0][ST_DS + k], ST[0][ST_S + k]) - PC[LC_S0 + k];
      if (act && i >= 1) { const double c = s[k] - Fp; ST[i - 1][ST_CT + k] = c; th += fabs(c); }
      if (i == 0) th += fabs(c0t[k]);
    }
    if (act) {
      const double dv = s[3] - vref(i);
      fl = 0.5 * fma(nv2(i) * s[3], s[3], fma(PC[LC_WV2] * dv, dv, fma(we2(i) * s[5], s[5], wc2(i) * s[4] * s[4])));
      double prod = (s[2] - PC[LC_LO]) * (PC[LC_HI] - s[2]) * (s[3] - PC[LC_LO + 1]) * (PC[LC_HI + 1] - s[3]);
      if (hasu) {
        fl = fma(0.5 * PC[LC_WD2] * u0, u0, fl);
        if (i >= 1) { const double dd = u0 - dprev; fl = fma(0.5 * PC[LC_CW] * dd, dd, fl); }
        prod *= (u0 - PC[LC_LO + 2]) * (PC[LC_HI + 2] - u0) * (u1 - PC[LC_LO + 3]) * (PC[LC_HI + 3] - u1);
      }
      ll = log(prod);
    }
    ft = gsum<NS_GROUP>(fl, gm); lt = gsum<NS_GROUP>(ll, gm); tht = gsum<NS_GROUP>(th, gm);
    gsync();
  }
  // More stages than lanes in the group (N > 32): lane g holds stages g, g + G, ...  F(s_i, u_i) travels to the owner
  // of stage i + 1 through the CT slot of row i (which that owner then overwrites with the residual), the neighbour's
  // trial delta is recomputed from its row.  Same operations per stage as eval_par / eval_sweep.
  __device__ void eval_parN(double a) {
    const int G = PAR ? NS_GROUP : 1;
    double s[NPASS][6], u0[NPASS];
    double fl = 0.0, ll = 0.0, th = 0.0;
#pragma unroll
    for (int p = 0; p < NPASS; p++) {
      const int i = g0 + p * G;
      const bool act = i < N, hasu = i < N - 1;
      const int ii = act ? i : 0;
      u0[p] = 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) s[p][k] = fma(a, ST[ii][ST_DS + k], ST[ii][ST_S + k]);
      if (hasu) {
        double tg[8], F[6];
        u0[p] = fma(a, ST[i][ST_DU + 0], ST[i][ST_U + 0]);
        const double u1 = fma(a, ST[i][ST_DU + 1], ST[i][ST_U + 1]);
        point_eval(s[p], u0[p], u1, tg, F);
#pragma unroll
        for (int k = 0; k < 8; k++) ST[i][ST_TT + k] = tg[k];
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_CT + k] = F[k];
        double prod = (s[p][2] - PC[LC_LO]) * (PC[LC_HI] - s[p][2]) * (s[p][3] - PC[LC_LO + 1]) * (PC[LC_HI + 1] - s[p][3]);
        prod *= (u0[p] - PC[LC_LO + 2]) * (PC[LC_HI + 2] - u0[p]) * (u1 - PC[LC_LO + 3]) * (PC[LC_HI + 3] - u1);
        ll += log(prod);
      } else if (act) {
        ll += log((s[p][2] - PC[LC_LO]) * (PC[LC_HI] - s[p][2]) * (s[p][3] - PC[LC_LO + 1]) * (PC[LC_HI + 1] - s[p][3]));
      }
    }
    gsync();
#pragma unroll
    for (int k = 0; k < 6; k++) {
      c0t[k] = fma(a, ST[0][ST_DS + k], ST[0][ST_S + k]) - PC[LC_S0 + k];
      if (g0 == 0) th += fabs(c0t[k]);
    }
#pragma unroll
    for (int p = 0; p < NPASS; p++) {
      const int i = g0 + p * G;
      const bool act = i < N, hasu = i < N - 1;
      if (act && i >= 1) {
#pragma unroll
        for (int k = 0; k < 6; k++) { const double c = s[p][k] - ST[i - 1][ST_CT + k]; ST[i - 1][ST_CT + k] = c; th += fabs(c); }
      }
      if (act) {
        const double dv = s[p][3] - vref(i);
        double f = 0.5 * fma(nv2(i) * s[p][3], s[p][3], fma(PC[LC_WV2] * dv, dv, fma(we2(i) * s[p][5], s[p][5], wc2(i) * s[p][4] * s[p][4])));
        if (hasu) {
          f = fma(0.5 * PC[LC_WD2] * u0[p], u0[p], f);
          if (i >= 1) {
            const double dd = u0[p] - fma(a, ST[i - 1][ST_DU + 0], ST[i - 1][ST_U + 0]);
            f = fma(0.5 * PC[LC_CW] * dd, dd, f);
          }
        }
        fl += f;
      }
    }
    ft = gsum<NS_GROUP>(fl, gm); lt = gsum<NS_GROUP>(ll, gm); tht = gsum<NS_GROUP>(th, gm);
    gsync();
  }
  // CS = a * (first ? CN : CS) + CT     (Ipopt's accumulated second-order-correction rhs)
  __device__ void soc_rhs(bool first, double a) {
#pragma unroll
    for (int k = 0; k < 6; k++) cs0[k] = a * (first ? c0[k] : cs0[k]) + c0t[k];
    if (PAR) {
#pragma unroll 1
      for (int i = g0; i < N - 1; i += gstep) {
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_CS + k] = a * (first ? ST[i][ST_CN + k] : ST[i][ST_CS + k]) + ST[i][ST_CT + k];
      }
    } else {
      // the residuals of the trial point just evaluated (step a along DS) are not kept: recompute them
      double F[6] = {0, 0, 0, 0, 0, 0};
#pragma unroll 1
      for (int i = 0; i < N; i++) {
        double t[6];
#pragma unroll
        for (int k = 0; k < 6; k++) t[k] = fma(a, ST[i][ST_DS + k], ST[i][ST_S + k]);
        if (i >= 1) {
#pragma unroll
          for (int k = 0; k < 6; k++) ST[i - 1][ST_CS + k] = a * (first ? ST[i - 1][ST_CN + k] : ST[i - 1][ST_CS + k]) + (t[k] - F[k]);
        }
        if (i < N - 1) {
          double tg[8];
          point_eval(t, fma(a, ST[i][ST_DU + 0], ST[i][ST_U + 0]), fma(a, ST[i][ST_DU + 1], ST[i][ST_U + 1]), tg, F);
        }
      }
    }
    gsync();
  }

  // ------------------------------------------------------------------------------------------
  // slot 2 (backward sweep), three jobs in one pass over the stages:
  //  (1) costate recursion at the OLD iterate: the new multipliers lambda+ of the step just tried
  //      (or, ls: the least-squares multiplier estimate);
  //  (2) do_update: accept the step -- x += alpha dx, lambda += alpha (lambda+ - lambda), z with Ipopt's
  //      kappa_sigma safeguard -- and re-evaluate trig/polynomial values and residuals there;
  //  (3) Ipopt's optimality error terms at the resulting iterate.
  // ------------------------------------------------------------------------------------------
  __device__ void advance(bool do_update, bool ls, bool zero_lam) {
    if (PAR) { advance_par(do_update, ls, zero_lam); return; }
    const double dt = PC[LC_DT], cw = PC[LC_CW], wd2 = PC[LC_WD2], wv2 = PC[LC_WV2];
    const double a = alpha, az = alpha_z;
    const double dwv = ls ? 0.0 : dw_used;
    const double zcap = K_KAPPA_SIGMA * mu, zfloor = mu / K_KAPPA_SIGMA;   // Ipopt's kappa_sigma safeguard
    const bool costate = do_update || ls;
    double lo_n[6] = {0, 0, 0, 0, 0, 0};   // OLD multipliers of stage i+1
    double lp_n[6] = {0, 0, 0, 0, 0, 0};   // lambda+ of stage i+1
    double ln_n[6] = {0, 0, 0, 0, 0, 0};   // NEW multipliers of stage i+1
    double dnext = 0.0;                    // NEW delta_{i+1}
    double sn[6] = {0, 0, 0, 0, 0, 0};     // NEW state of stage i+1
    double r = 0.0, cv = 0.0, l1 = 0.0, zz = 0.0, am = 1e300, aM = 0.0, lmax = 0.0;
#pragma unroll 1
    for (int i = N - 1; i >= 0; i--) {
      const bool hasu = i < N - 1;
      double s[6], lam[6], zl[4], zu[4], tg[8], u0 = 0.0, u1 = 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) { s[k] = ST[i][ST_S + k]; lam[k] = ST[i][ST_LAM + k]; }
#pragma unroll
      for (int k = 0; k < 4; k++) { zl[k] = ST[i][ST_ZL + k]; zu[k] = ST[i][ST_ZU + k]; }
      // every load of the stage is issued here, needed on this lane's path or not (rows hold all fields for all stages):
      // a load behind a branch is a second, third, ... latency to wait out
      double ds_l[6], cn_l[6];
#pragma unroll
      for (int k = 0; k < 6; k++) { ds_l[k] = ST[i][ST_DS + k]; cn_l[k] = ST[i][ST_CN + k]; }
      const double du0_l = ST[i][ST_DU + 0], du1_l = ST[i][ST_DU + 1];
      const int im = i >= 1 ? i - 1 : 0;
      const double up_l = ST[im][ST_U + 0], dup_l = ST[im][ST_DU + 0];
      if (hasu) {
        u0 = ST[i][ST_U + 0]; u1 = ST[i][ST_U + 1];
#pragma unroll
        for (int k = 0; k < 8; k++) tg[k] = ST[i][ST_TG + k];
      } else {
#pragma unroll
        for (int k = 0; k < 8; k++) tg[k] = 0.0;
      }
      const double dprev_old = (hasu && i >= 1) ? up_l : 0.0;
      double dprev = dprev_old;            // NEW delta_{i-1}
      double lp[6] = {0, 0, 0, 0, 0, 0};
      StageLin L;
      if (hasu) lin_at(tg, s[3], u0, L);
      if (costate) {
        double ds[6], du0 = 0.0, du1 = 0.0, il[4], iu[4];
#pragma unroll
        for (int k = 0; k < 6; k++) ds[k] = ds_l[k];
        if (hasu) { du0 = du0_l; du1 = du1_l; }
        slack_rcp(s[2], s[3], u0, u1, hasu, il, iu);
        StageHess H;
        hess_at(i, ls, dwv, tg, s[3], s[4], s[5], u0, dprev_old, lo_n, zl, zu, il, iu, H);
        double h[6];
        h[0] = H.qxx * ds[0];
        h[1] = H.qyy * ds[1];
        h[2] = fma(H.qpv, ds[3], H.qpp * ds[2]) + H.gp;
        h[3] = fma(H.svd, du0, fma(H.qve, ds[5], fma(H.qvv, ds[3], H.qpv * ds[2])) + H.gv);
        h[4] = fma(H.qcc, ds[4], H.gc);
        h[5] = fma(H.qee, ds[5], H.qve * ds[3]) + H.ge;
        if (hasu) {
          const double l25 = lp_n[2] + lp_n[5];
          lp[0] = fma(L.a61, lp_n[5], fma(L.a51, lp_n[4], lp_n[0])) - h[0];
          lp[1] = lp_n[1] - lp_n[4] - h[1];
          lp[2] = fma(L.a23, lp_n[1], L.a13 * lp_n[0]) + l25 - h[2];
          lp[3] = fma(L.a54, lp_n[4], fma(L.a34, l25, fma(L.a24, lp_n[1], L.a14 * lp_n[0])) + lp_n[3]) - h[3];
          lp[4] = -h[4];
          lp[5] = fma(L.a56, lp_n[4], -h[5]);
        } else {
#pragma unroll
          for (int k = 0; k < 6; k++) lp[k] = -h[k];
        }
#pragma unroll
        for (int k = 0; k < 6; k++) lmax = nanmax(lmax, fabs(lp[k]));
#pragma unroll
        for (int k = 0; k < 6; k++) lo_n[k] = lam[k];
        if (do_update) {
          const double dx[4] = {ds[2], ds[3], du0, du1};
#pragma unroll
          for (int k = 0; k < 6; k++) { s[k] = fma(a, ds[k], s[k]); lam[k] = fma(a, lp[k] - lam[k], lam[k]); ST[i][ST_S + k] = s[k]; }
          if (hasu) {
            u0 = fma(a, du0, u0); u1 = fma(a, du1, u1);
            ST[i][ST_U + 0] = u0; ST[i][ST_U + 1] = u1;
          }
          if (i >= 1 && hasu) dprev = fma(a, dup_l, dprev_old);
          double iln[4], iun[4];
          slack_rcp(s[2], s[3], u0, u1, hasu, iln, iun);
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (k < 2 || hasu) {
              const double dzl = fma(fma(-zl[k], dx[k], mu), il[k], -zl[k]);
              const double dzu = fma(fma(zu[k], dx[k], mu), iu[k], -zu[k]);
              zl[k] = dmax(dmin(fma(az, dzl, zl[k]), zcap * iln[k]), zfloor * iln[k]);
              zu[k] = dmax(dmin(fma(az, dzu, zu[k]), zcap * iun[k]), zfloor * iun[k]);
              ST[i][ST_ZL + k] = zl[k]; ST[i][ST_ZU + k] = zu[k];
            }
          }
        } else {
#pragma unroll
          for (int k = 0; k < 6; k++) lam[k] = lp[k];
        }
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_LAM + k] = lam[k];
      } else if (zero_lam) {
#pragma unroll
        for (int k = 0; k < 6; k++) { lam[k] = 0.0; ST[i][ST_LAM + k] = 0.0; }
      }
      // ---- residuals and trig/polynomial values at the (new) iterate
      double cn[6] = {0, 0, 0, 0, 0, 0};
      if (hasu) {
        if (do_update) {
          // the trial point the evaluation sweep accepted is the new iterate: same inputs, same bits
          double F[6];
          point_eval(s, u0, u1, tg, F);
#pragma unroll
          for (int k = 0; k < 6; k++) { cn[k] = sn[k] - F[k]; ST[i][ST_CN + k] = cn[k]; }
#pragma unroll
          for (int k = 0; k < 8; k++) ST[i][ST_TG + k] = tg[k];
          lin_at(tg, s[3], u0, L);
        } else {
#pragma unroll
          for (int k = 0; k < 6; k++) cn[k] = cn_l[k];
        }
      }
#pragma unroll
      for (int k = 0; k < 6; k++) sn[k] = s[k];
      if (i == 0 && do_update) {
#pragma unroll
        for (int k = 0; k < 6; k++) c0[k] = c0t[k];
      }
      // ---- optimality error terms
      double os[6] = {0, 0, 0, 0, 0, 0}, ou0 = 0.0, ou1 = 0.0;
      const double v = s[3];
      if (hasu) {
        const double l25 = ln_n[2] + ln_n[5];
        os[0] = fma(L.a61, ln_n[5], fma(L.a51, ln_n[4], ln_n[0]));
        os[1] = ln_n[1] - ln_n[4];
        os[2] = fma(L.a23, ln_n[1], L.a13 * ln_n[0]) + l25;
        os[3] = fma(L.a54, ln_n[4], fma(L.a34, l25, fma(L.a24, ln_n[1], L.a14 * ln_n[0])) + ln_n[3]);
        os[5] = L.a56 * ln_n[4];
        ou0 = L.b3 * l25;
        ou1 = dt * ln_n[3];
      }
      double gs[6];
      gs[0] = 0.0; gs[1] = 0.0;
      gs[2] = -zl[0] + zu[0];
      gs[3] = fma(nv2(i), v, wv2 * (v - vref(i))) - zl[1] + zu[1];
      gs[4] = wc2(i) * s[4];
      gs[5] = we2(i) * s[5];
#pragma unroll
      for (int k = 0; k < 6; k++) {
        r = nanmax(r, fabs(gs[k] + lam[k] - os[k]));
        l1 += fabs(lam[k]);
        cv = nanmax(cv, fabs(cn[k]));
      }
      zz += fabs(zl[0]) + fabs(zu[0]) + fabs(zl[1]) + fabs(zu[1]);
      {
        const double p0 = (s[2] - PC[LC_LO]) * zl[0], p1 = (PC[LC_HI] - s[2]) * zu[0];
        const double p2 = (s[3] - PC[LC_LO + 1]) * zl[1], p3 = (PC[LC_HI + 1] - s[3]) * zu[1];
        am = dmin(am, dmin(dmin(p0, p1), dmin(p2, p3)));
        aM = dmax(aM, dmax(dmax(p0, p1), dmax(p2, p3)));
      }
      if (hasu) {
        double gd = wd2 * u0;
        if (i >= 1) gd = fma(cw, u0 - dprev, gd);
        if (i <= N - 3) gd = fma(-cw, dnext - u0, gd);
        r = nanmax(r, fabs(gd - ou0 - zl[2] + zu[2]));
        r = nanmax(r, fabs(-ou1 - zl[3] + zu[3]));
        zz += fabs(zl[2]) + fabs(zu[2]) + fabs(zl[3]) + fabs(zu[3]);
        const double p0 = (u0 - PC[LC_LO + 2]) * zl[2], p1 = (PC[LC_HI + 2] - u0) * zu[2];
        const double p2 = (u1 - PC[LC_LO + 3]) * zl[3], p3 = (PC[LC_HI + 3] - u1) * zu[3];
        am = dmin(am, dmin(dmin(p0, p1), dmin(p2, p3)));
        aM = dmax(aM, dmax(dmax(p0, p1), dmax(p2, p3)));
        dnext = u0;
      }
#pragma unroll
      for (int k = 0; k < 6; k++) { ln_n[k] = lam[k]; lp_n[k] = lp[k]; }
    }
#pragma unroll
    for (int k = 0; k < 6; k++) cv = nanmax(cv, fabs(c0[k]));
    dinf = r; cviol = cv; lam1 = l1; z1 = zz; amin = am; amax = aM; lsq_lmax = lmax;
  }
  // the same sweep with one stage per lane of the group.  The costate recursion is the only sequential
  // part: N steps of a 6-vector handed down the lanes by shuffle; neighbours' new values (lambda_{i+1},
  // delta_{i+-1}) travel by shuffle too, the six error terms are butterfly reductions.
  __device__ void advance_par(bool do_update, bool ls, bool zero_lam) {
    if (NPASS > 1) { advance_parN(do_update, ls, zero_lam); return; }
    const int G = PAR ? NS_GROUP : 1;
    const double dt = PC[LC_DT], cw = PC[LC_CW], wd2 = PC[LC_WD2], wv2 = PC[LC_WV2];
    const double a = alpha, az = alpha_z;
    const double dwv = ls ? 0.0 : dw_used;
    const double zcap = K_KAPPA_SIGMA * mu, zfloor = mu / K_KAPPA_SIGMA;
    const bool costate = do_update || ls;
    const int i = g0;
    const bool act = i < N, hasu = i < N - 1;
    const int ii = act ? i : 0;
    double s[6], lam[6], zl[4], zu[4], tg[8], u0 = 0.0, u1 = 0.0;
#pragma unroll
    for (int k = 0; k < 6; k++) { s[k] = ST[ii][ST_S + k]; lam[k] = act ? ST[ii][ST_LAM + k] : 0.0; }
#pragma unroll
    for (int k = 0; k < 4; k++) { zl[k] = act ? ST[ii][ST_ZL + k] : 0.0; zu[k] = act ? ST[ii][ST_ZU + k] : 0.0; }
#pragma unroll
    for (int k = 0; k < 8; k++) tg[k] = hasu ? ST[ii][ST_TG + k] : 0.0;
    if (hasu) { u0 = ST[i][ST_U + 0]; u1 = ST[i][ST_U + 1]; }
    const double dprev_old = __shfl_up_sync(gm, u0, 1, G);
    double lo_n[6];
#pragma unroll
    for (int k = 0; k < 6; k++) { const double t = __shfl_down_sync(gm, lam[k], 1, G); lo_n[k] = hasu ? t : 0.0; }
    StageLin L;
    lin_at(tg, s[3], u0, L);
    double lp[6] = {0, 0, 0, 0, 0, 0}, lmax = 0.0, dym = 0.0;
    double ds[6] = {0, 0, 0, 0, 0, 0}, du0 = 0.0, du1 = 0.0, il[4], iu[4];
    if (costate) {
      double h[6] = {0, 0, 0, 0, 0, 0};
      if (act) {
#pragma unroll
        for (int k = 0; k < 6; k++) ds[k] = ST[i][ST_DS + k];
        if (hasu) { du0 = ST[i][ST_DU + 0]; du1 = ST[i][ST_DU + 1]; }
        slack_rcp(s[2], s[3], u0, u1, hasu, il, iu);
        StageHess H;
        hess_at(i, ls, dwv, tg, s[3], s[4], s[5], u0, (hasu && i >= 1) ? dprev_old : 0.0, lo_n, zl, zu, il, iu, H);
        h[0] = H.qxx * ds[0];
        h[1] = H.qyy * ds[1];
        h[2] = fma(H.qpv, ds[3], H.qpp * ds[2]) + H.gp;
        h[3] = fma(H.svd, du0, fma(H.qve, ds[5], fma(H.qvv, ds[3], H.qpv * ds[2])) + H.gv);
        h[4] = fma(H.qcc, ds[4], H.gc);
        h[5] = fma(H.qee, ds[5], H.qve * ds[3]) + H.ge;
      }
      // lambda+_i = A_i^T lambda+_{i+1} - h_i, from the last stage down
#pragma unroll 1
      for (int j = N - 1; j >= 0; j--) {
        double n[6];
#pragma unroll
        for (int k = 0; k < 6; k++) n[k] = __shfl_down_sync(gm, lp[k], 1, G);
        if (i == j) {
          if (hasu) {
            const double l25 = n[2] + n[5];
            lp[0] = fma(L.a61, n[5], fma(L.a51, n[4], n[0])) - h[0];
            lp[1] = n[1] - n[4] - h[1];
            lp[2] = fma(L.a23, n[1], L.a13 * n[0]) + l25 - h[2];
            lp[3] = fma(L.a54, n[4], fma(L.a34, l25, fma(L.a24, n[1], L.a14 * n[0])) + n[3]) - h[3];
            lp[4] = -h[4];
            lp[5] = fma(L.a56, n[4], -h[5]);
          } else {
#pragma unroll
            for (int k = 0; k < 6; k++) lp[k] = -h[k];
          }
        }
      }
      if (act) {
#pragma unroll
        for (int k = 0; k < 6; k++) { lmax = nanmax(lmax, fabs(lp[k])); dym = nanmax(dym, fabs(lp[k] - lam[k])); }
      }
      if (do_update) {
        if (act) {
          const double dx[4] = {ds[2], ds[3], du0, du1};
#pragma unroll
          for (int k = 0; k < 6; k++) { s[k] = fma(a, ds[k], s[k]); lam[k] = fma(a, lp[k] - lam[k], lam[k]); ST[i][ST_S + k] = s[k]; }
          if (hasu) {
            u0 = fma(a, du0, u0); u1 = fma(a, du1, u1);
            ST[i][ST_U + 0] = u0; ST[i][ST_U + 1] = u1;
          }
          double iln[4], iun[4];
          slack_rcp(s[2], s[3], u0, u1, hasu, iln, iun);
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (k < 2 || hasu) {
              const double dzl = fma(fma(-zl[k], dx[k], mu), il[k], -zl[k]);
              const double dzu = fma(fma(zu[k], dx[k], mu), iu[k], -zu[k]);
              zl[k] = dmax(dmin(fma(az, dzl, zl[k]), zcap * iln[k]), zfloor * iln[k]);
              zu[k] = dmax(dmin(fma(az, dzu, zu[k]), zcap * iun[k]), zfloor * iun[k]);
              ST[i][ST_ZL + k] = zl[k]; ST[i][ST_ZU + k] = zu[k];
            }
          }
        }
      } else if (act) {
#pragma unroll
        for (int k = 0; k < 6; k++) lam[k] = lp[k];
      }
      if (act) {
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_LAM + k] = lam[k];
      }
    } else if (zero_lam && act) {
#pragma unroll
      for (int k = 0; k < 6; k++) { lam[k] = 0.0; ST[i][ST_LAM + k] = 0.0; }
    }
    // ---- residuals and trig/polynomial values at the (new) iterate
    double cn[6] = {0, 0, 0, 0, 0, 0};
    if (hasu) {
      if (do_update) {
#pragma unroll
        for (int k = 0; k < 6; k++) { cn[k] = ST[i][ST_CT + k]; ST[i][ST_CN + k] = cn[k]; }
#pragma unroll
        for (int k = 0; k < 8; k++) { tg[k] = ST[i][ST_TT + k]; ST[i][ST_TG + k] = tg[k]; }
        lin_at(tg, s[3], u0, L);
      } else {
#pragma unroll
        for (int k = 0; k < 6; k++) cn[k] = ST[i][ST_CN + k];
      }
    }
    if (do_update) {
#pragma unroll
      for (int k = 0; k < 6; k++) c0[k] = c0t[k];
    }
    // ---- optimality error terms
    const double dprev = __shfl_up_sync(gm, u0, 1, G), dnext = __shfl_down_sync(gm, u0, 1, G);
    double ln_n[6];
#pragma unroll
    for (int k = 0; k < 6; k++) { const double t = __shfl_down_sync(gm, lam[k], 1, G); ln_n[k] = hasu ? t : 0.0; }
    double r = 0.0, cv = 0.0, l1 = 0.0, zz = 0.0, am = 1e300, aM = 0.0;
    if (act) {
      double os[6] = {0, 0, 0, 0, 0, 0}, ou0 = 0.0, ou1 = 0.0;
      const double v = s[3];
      if (hasu) {
        const double l25 = ln_n[2] + ln_n[5];
        os[0] = fma(L.a61, ln_n[5], fma(L.a51, ln_n[4], ln_n[0]));
        os[1] = ln_n[1] - ln_n[4];
        os[2] = fma(L.a23, ln_n[1], L.a13 * ln_n[0]) + l25;
        os[3] = fma(L.a54, ln_n[4], fma(L.a34, l25, fma(L.a24, ln_n[1], L.a14 * ln_n[0])) + ln_n[3]);
        os[5] = L.a56 * ln_n[4];
        ou0 = L.b3 * l25;
        ou1 = dt * ln_n[3];
      }
      double gs[6];
      gs[0] = 0.0; gs[1] = 0.0;
      gs[2] = -zl[0] + zu[0];
      gs[3] = fma(nv2(i), v, wv2 * (v - vref(i))) - zl[1] + zu[1];
      gs[4] = wc2(i) * s[4];
      gs[5] = we2(i) * s[5];
#pragma unroll
      for (int k = 0; k < 6; k++) {
        r = nanmax(r, fabs(gs[k] + lam[k] - os[k]));
        l1 += fabs(lam[k]);
        cv = nanmax(cv, fabs(cn[k]));
        if (i == 0) cv = nanmax(cv, fabs(c0[k]));
      }
      zz = fabs(zl[0]) + fabs(zu[0]) + fabs(zl[1]) + fabs(zu[1]);
      {
        const double p0 = (s[2] - PC[LC_LO]) * zl[0], p1 = (PC[LC_HI] - s[2]) * zu[0];
        const double p2 = (s[3] - PC[LC_LO + 1]) * zl[1], p3 = (PC[LC_HI + 1] - s[3]) * zu[1];
        am = dmin(dmin(p0, p1), dmin(p2, p3));
        aM = dmax(dmax(p0, p1), dmax(p2, p3));
      }
      if (hasu) {
        double gd = wd2 * u0;
        if (i >= 1) gd = fma(cw, u0 - dprev, gd);
        if (i <= N - 3) gd = fma(-cw, dnext - u0, gd);
        r = nanmax(r, fabs(gd - ou0 - zl[2] + zu[2]));
        r = nanmax(r, fabs(-ou1 - zl[3] + zu[3]));
        zz += fabs(zl[2]) + fabs(zu[2]) + fabs(zl[3]) + fabs(zu[3]);
        const double p0 = (u0 - PC[LC_LO + 2]) * zl[2], p1 = (PC[LC_HI + 2] - u0) * zu[2];
        const double p2 = (u1 - PC[LC_LO + 3]) * zl[3], p3 = (PC[LC_HI + 3] - u1) * zu[3];
        am = dmin(am, dmin(dmin(p0, p1), dmin(p2, p3)));
        aM = dmax(aM, dmax(dmax(p0, p1), dmax(p2, p3)));
      }
    }
    dinf = gmax<NS_GROUP>(r, gm); cviol = gmax<NS_GROUP>(cv, gm); lam1 = gsum<NS_GROUP>(l1, gm); z1 = gsum<NS_GROUP>(zz, gm);
    amin = gmin<NS_GROUP>(am, gm); amax = gmax<NS_GROUP>(aM, gm); lsq_lmax = gmax<NS_GROUP>(lmax, gm);
    dy_max = gmax<NS_GROUP>(dym, gm);
    gsync();
  }
  // More stages than lanes in the group: the neighbours' old values are read from their rows before anything is
  // written, the costate vector is handed from the owner of stage j + 1 to the owner of stage j by an indexed
  // shuffle, the neighbours' new values are read back after the update.  Same operations per stage as advance_par.
  __device__ void advance_parN(bool do_update, bool ls, bool zero_lam) {
    const int G = PAR ? NS_GROUP : 1;
    const double dt = PC[LC_DT], cw = PC[LC_CW], wd2 = PC[LC_WD2], wv2 = PC[LC_WV2];
    const double a = alpha, az = alpha_z;
    const double dwv = ls ? 0.0 : dw_used;
    const double zcap = K_KAPPA_SIGMA * mu, zfloor = mu / K_KAPPA_SIGMA;
    const bool costate = do_update || ls;
    double lp[NPASS][6], h[NPASS][6], lmax = 0.0, dym = 0.0;
    StageLin L[NPASS];
    // ---- phase 1: h_i = (W + Sigma) d_i + grad terms at the OLD iterate (reads only)
#pragma unroll
    for (int p = 0; p < NPASS; p++) {
      const int i = g0 + p * G;
      const bool act = i < N, hasu = i < N - 1;
      const int ii = act ? i : 0;
#pragma unroll
      for (int k = 0; k < 6; k++) { lp[p][k] = 0.0; h[p][k] = 0.0; }
      double tg[8];
#pragma unroll
      for (int k = 0; k < 8; k++) tg[k] = hasu ? ST[ii][ST_TG + k] : 0.0;
      const double v = ST[ii][ST_S + 3], u0 = hasu ? ST[ii][ST_U + 0] : 0.0, u1 = hasu ? ST[ii][ST_U + 1] : 0.0;
      lin_at(tg, v, u0, L[p]);
      if (costate && act) {
        double zl[4], zu[4], lo_n[6], il[4], iu[4], ds[6], du0 = 0.0;
#pragma unroll
        for (int k = 0; k < 4; k++) { zl[k] = ST[i][ST_ZL + k]; zu[k] = ST[i][ST_ZU + k]; }
#pragma unroll
        for (int k = 0; k < 6; k++) { lo_n[k] = hasu ? ST[i + 1][ST_LAM + k] : 0.0; ds[k] = ST[i][ST_DS + k]; }
        if (hasu) du0 = ST[i][ST_DU + 0];
        const double dprev_old = (hasu && i >= 1) ? ST[i - 1][ST_U + 0] : 0.0;
        slack_rcp(ST[i][ST_S + 2], v, u0, u1, hasu, il, iu);
        StageHess H;
        hess_at(i, ls, dwv, tg, v, ST[i][ST_S + 4], ST[i][ST_S + 5], u0, dprev_old, lo_n, zl, zu, il, iu, H);
        h[p][0] = H.qxx * ds[0];
        h[p][1] = H.qyy * ds[1];
        h[p][2] = fma(H.qpv, ds[3], H.qpp * ds[2]) + H.gp;
        h[p][3] = fma(H.svd, du0, fma(H.qve, ds[5], fma(H.qvv, ds[3], H.qpv * ds[2])) + H.gv);
        h[p][4] = fma(H.qcc, ds[4], H.gc);
        h[p][5] = fma(H.qee, ds[5], H.qve * ds[3]) + H.ge;
      }
    }
    // ---- phase 2: lambda+_j = A_j^T lambda+_{j+1} - h_j, from the last stage down
    if (costate) {
#pragma unroll 1
      for (int j = N - 1; j >= 0; j--) {
        const int src = (j + 1) % G, sp = (j + 1) / G;
        double n[6];
#pragma unroll
        for (int k = 0; k < 6; k++) {
          double v = lp[0][k];
#pragma unroll
          for (int p = 1; p < NPASS; p++) v = (sp == p) ? lp[p][k] : v;
          n[k] = __shfl_sync(gm, v, src, G);
        }
        if (j % G == g0) {
          const int pj = j / G;
#pragma unroll
          for (int p = 0; p < NPASS; p++) {
            if (p == pj) {
              if (j < N - 1) {
                const double l25 = n[2] + n[5];
                lp[p][0] = fma(L[p].a61, n[5], fma(L[p].a51, n[4], n[0])) - h[p][0];
                lp[p][1] = n[1] - n[4] - h[p][1];
                lp[p][2] = fma(L[p].a23, n[1], L[p].a13 * n[0]) + l25 - h[p][2];
                lp[p][3] = fma(L[p].a54, n[4], fma(L[p].a34, l25, fma(L[p].a24, n[1], L[p].a14 * n[0])) + n[3]) - h[p][3];
                lp[p][4] = -h[p][4];
                lp[p][5] = fma(L[p].a56, n[4], -h[p][5]);
              } else {
#pragma unroll
                for (int k = 0; k < 6; k++) lp[p][k] = -h[p][k];
              }
            }
          }
        }
      }
    }
    gsync();   // every lane has read its neighbours' old rows
    // ---- phase 3: accept the step
#pragma unroll
    for (int p = 0; p < NPASS; p++) {
      const int i = g0 + p * G;
      const bool act = i < N, hasu = i < N - 1;
      if (!act) continue;
      if (costate) {
#pragma unroll
        for (int k = 0; k < 6; k++) lmax = nanmax(lmax, fabs(lp[p][k]));
        double lam[6];
#pragma unroll
        for (int k = 0; k < 6; k++) { lam[k] = ST[i][ST_LAM + k]; dym = nanmax(dym, fabs(lp[p][k] - lam[k])); }
        if (do_update) {
          double sv[6], ds[6], zl[4], zu[4], il[4], iu[4], iln[4], iun[4];
          double u0 = hasu ? ST[i][ST_U + 0] : 0.0, u1 = hasu ? ST[i][ST_U + 1] : 0.0;
          const double du0 = hasu ? ST[i][ST_DU + 0] : 0.0, du1 = hasu ? ST[i][ST_DU + 1] : 0.0;
#pragma unroll
          for (int k = 0; k < 6; k++) { sv[k] = ST[i][ST_S + k]; ds[k] = ST[i][ST_DS + k]; }
#pragma unroll
          for (int k = 0; k < 4; k++) { zl[k] = ST[i][ST_ZL + k]; zu[k] = ST[i][ST_ZU + k]; }
          slack_rcp(sv[2], sv[3], u0, u1, hasu, il, iu);
          const double dx[4] = {ds[2], ds[3], du0, du1};
#pragma unroll
          for (int k = 0; k < 6; k++) { sv[k] = fma(a, ds[k], sv[k]); lam[k] = fma(a, lp[p][k] - lam[k], lam[k]); ST[i][ST_S + k] = sv[k]; }
          if (hasu) {
            u0 = fma(a, du0, u0); u1 = fma(a, du1, u1);
            ST[i][ST_U + 0] = u0; ST[i][ST_U + 1] = u1;
          }
          slack_rcp(sv[2], sv[3], u0, u1, hasu, iln, iun);
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (k < 2 || hasu) {
              const double dzl = fma(fma(-zl[k], dx[k], mu), il[k], -zl[k]);
              const double dzu = fma(fma(zu[k], dx[k], mu), iu[k], -zu[k]);
              zl[k] = dmax(dmin(fma(az, dzl, zl[k]), zcap * iln[k]), zfloor * iln[k]);
              zu[k] = dmax(dmin(fma(az, dzu, zu[k]), zcap * iun[k]), zfloor * iun[k]);
              ST[i][ST_ZL + k] = zl[k]; ST[i][ST_ZU + k] = zu[k];
            }
          }
          if (hasu) {
#pragma unroll
            for (int k = 0; k < 6; k++) ST[i][ST_CN + k] = ST[i][ST_CT + k];
#pragma unroll
            for (int k = 0; k < 8; k++) ST[i][ST_TG + k] = ST[i][ST_TT + k];
          }
        } else {
#pragma unroll
          for (int k = 0; k < 6; k++) lam[k] = lp[p][k];
        }
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_LAM + k] = lam[k];
      } else if (zero_lam) {
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_LAM + k] = 0.0;
      }
    }
    if (do_update) {
#pragma unroll
      for (int k = 0; k < 6; k++) c0[k] = c0t[k];
    }
    gsync();   // the new rows are visible
    // ---- phase 4: optimality error terms at the (new) iterate
    double r = 0.0, cv = 0.0, l1 = 0.0, zz = 0.0, am = 1e300, aM = 0.0;
#pragma unroll
    for (int p = 0; p < NPASS; p++) {
      const int i = g0 + p * G;
      const bool act = i < N, hasu = i < N - 1;
      if (!act) continue;
      double sv[6], lam[6], zl[4], zu[4], ln_n[6], cn[6], tg[8];
#pragma unroll
      for (int k = 0; k < 6; k++) { sv[k] = ST[i][ST_S + k]; lam[k] = ST[i][ST_LAM + k]; ln_n[k] = hasu ? ST[i + 1][ST_LAM + k] : 0.0; cn[k] = hasu ? ST[i][ST_CN + k] : 0.0; }
#pragma unroll
      for (int k = 0; k < 4; k++) { zl[k] = ST[i][ST_ZL + k]; zu[k] = ST[i][ST_ZU + k]; }
#pragma unroll
      for (int k = 0; k < 8; k++) tg[k] = hasu ? ST[i][ST_TG + k] : 0.0;
      const double u0 = hasu ? ST[i][ST_U + 0] : 0.0, u1 = hasu ? ST[i][ST_U + 1] : 0.0;
      const double v = sv[3];
      StageLin Ln;
      lin_at(tg, v, u0, Ln);
      double os[6] = {0, 0, 0, 0, 0, 0}, ou0 = 0.0, ou1 = 0.0;
      if (hasu) {
        const double l25 = ln_n[2] + ln_n[5];
        os[0] = fma(Ln.a61, ln_n[5], fma(Ln.a51, ln_n[4], ln_n[0]));
        os[1] = ln_n[1] - ln_n[4];
        os[2] = fma(Ln.a23, ln_n[1], Ln.a13 * ln_n[0]) + l25;
        os[3] = fma(Ln.a54, ln_n[4], fma(Ln.a34, l25, fma(Ln.a24, ln_n[1], Ln.a14 * ln_n[0])) + ln_n[3]);
        os[5] = Ln.a56 * ln_n[4];
        ou0 = Ln.b3 * l25;
        ou1 = dt * ln_n[3];
      }
      double gs[6];
      gs[0] = 0.0; gs[1] = 0.0;
      gs[2] = -zl[0] + zu[0];
      gs[3] = fma(nv2(i), v, wv2 * (v - vref(i))) - zl[1] + zu[1];
      gs[4] = wc2(i) * sv[4];
      gs[5] = we2(i) * sv[5];
#pragma unroll
      for (int k = 0; k < 6; k++) {
        r = nanmax(r, fabs(gs[k] + lam[k] - os[k]));
        l1 += fabs(lam[k]);
        cv = nanmax(cv, fabs(cn[k]));
        if (i == 0) cv = nanmax(cv, fabs(c0[k]));
      }
      zz += fabs(zl[0]) + fabs(zu[0]) + fabs(zl[1]) + fabs(zu[1]);
      {
        const double p0 = (sv[2] - PC[LC_LO]) * zl[0], p1 = (PC[LC_HI] - sv[2]) * zu[0];
        const double p2 = (sv[3] - PC[LC_LO + 1]) * zl[1], p3 = (PC[LC_HI + 1] - sv[3]) * zu[1];
        am = dmin(am, dmin(dmin(p0, p1), dmin(p2, p3)));
        aM = dmax(aM, dmax(dmax(p0, p1), dmax(p2, p3)));
      }
      if (hasu) {
        double gd = wd2 * u0;
        if (i >= 1) gd = fma(cw, u0 - ST[i - 1][ST_U + 0], gd);
        if (i <= N - 3) gd = fma(-cw, ST[i + 1][ST_U + 0] - u0, gd);
        r = nanmax(r, fabs(gd - ou0 - zl[2] + zu[2]));
        r = nanmax(r, fabs(-ou1 - zl[3] + zu[3]));
        zz += fabs(zl[2]) + fabs(zu[2]) + fabs(zl[3]) + fabs(zu[3]);
        const double p0 = (u0 - PC[LC_LO + 2]) * zl[2], p1 = (PC[LC_HI + 2] - u0) * zu[2];
        const double p2 = (u1 - PC[LC_LO + 3]) * zl[3], p3 = (PC[LC_HI + 3] - u1) * zu[3];
        am = dmin(am, dmin(dmin(p0, p1), dmin(p2, p3)));
        aM = dmax(aM, dmax(dmax(p0, p1), dmax(p2, p3)));
      }
    }
    dinf = gmax<NS_GROUP>(r, gm); cviol = gmax<NS_GROUP>(cv, gm); lam1 = gsum<NS_GROUP>(l1, gm); z1 = gsum<NS_GROUP>(zz, gm);
    amin = gmin<NS_GROUP>(am, gm); amax = gmax<NS_GROUP>(aM, gm); lsq_lmax = gmax<NS_GROUP>(lmax, gm);
    dy_max = gmax<NS_GROUP>(dym, gm);
    gsync();
  }
  // max_i |slack_i * z_i - m|  from the extreme complementarity products
  __device__ __forceinline__ double compl_err(double m) const { return nanmax(fabs(amax - m), fabs(amin - m)); }

  // coop kernel: derivative pieces of every stage at the iterate, one stage per lane, into the shared row
  // (dw is added by the Riccati sweep, so an inertia-correction retry does not rebuild them)
  __device__ void build_lh(bool ls) {
#pragma unroll 1
    for (int i = g0; i < N; i += NS_GROUP) {
      const bool hasu = i < N - 1;
      double tg[8], ln[6], zl[4], zu[4], il[4], iu[4];
#pragma unroll
      for (int k = 0; k < 8; k++) tg[k] = hasu ? ST[i][ST_TG + k] : 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) ln[k] = hasu ? ST[i + 1][ST_LAM + k] : 0.0;
#pragma unroll
      for (int k = 0; k < 4; k++) { zl[k] = (k < 2 || hasu) ? ST[i][ST_ZL + k] : 0.0; zu[k] = (k < 2 || hasu) ? ST[i][ST_ZU + k] : 0.0; }
      const double psi = ST[i][ST_S + 2], v = ST[i][ST_S + 3], c = ST[i][ST_S + 4], e = ST[i][ST_S + 5];
      const double u0 = hasu ? ST[i][ST_U + 0] : 0.0, u1 = hasu ? ST[i][ST_U + 1] : 0.0;
      const double dprev = (hasu && i >= 1) ? ST[i - 1][ST_U + 0] : 0.0;
      slack_rcp(psi, v, u0, u1, hasu, il, iu);
      StageLin L;
      StageHess H;
      lin_at(tg, v, u0, L);
      hess_at(i, ls, 0.0, tg, v, c, e, u0, dprev, ln, zl, zu, il, iu, H);
      double *q = &ST[i][ST_LH];
      q[0] = L.a13; q[1] = L.a14; q[2] = L.a23; q[3] = L.a24; q[4] = L.a34; q[5] = L.b3; q[6] = L.a51; q[7] = L.a54;
      q[8] = L.a56; q[9] = L.a61;
      q[10] = H.qxx; q[11] = H.qyy; q[12] = H.qpp; q[13] = H.qpv; q[14] = H.qvv; q[15] = H.qve; q[16] = H.qcc; q[17] = H.qee;
      q[18] = H.svd; q[19] = H.rdd; q[20] = H.raa; q[21] = H.gp; q[22] = H.gv; q[23] = H.gc; q[24] = H.ge; q[25] = H.gdp;
      q[26] = H.gd; q[27] = H.ga;
    }
    gsync();
  }
  __device__ __forceinline__ void load_lin(int i, StageLin &L) const {
    const double *q = &ST[i][PAR ? ST_LH : 0];
    L.a13 = q[0]; L.a14 = q[1]; L.a23 = q[2]; L.a24 = q[3]; L.a34 = q[4]; L.b3 = q[5]; L.a51 = q[6]; L.a54 = q[7];
    L.a56 = q[8]; L.a61 = q[9];
  }
  // ls: H = I has no dw (the least-squares system is not regularised)
  __device__ __forceinline__ void load_hess(int i, double dwv, StageHess &H) const {
    const double *q = &ST[i][PAR ? ST_LH : 0];
    H.qxx = q[10] + dwv; H.qyy = q[11] + dwv; H.qpp = q[12] + dwv; H.qpv = q[13]; H.qvv = q[14] + dwv; H.qve = q[15];
    H.qcc = q[16] + dwv; H.qee = q[17] + dwv; H.svd = q[18]; H.rdd = q[19] + dwv; H.raa = q[20] + dwv;
    H.gp = q[21]; H.gv = q[22]; H.gc = q[23]; H.ge = q[24]; H.gdp = q[25]; H.gd = q[26]; H.ga = q[27];
  }

  // ------------------------------------------------------------------------------------------
  // slot 3: backward Riccati sweep.  Cost-to-go over (x, y, psi, v, epsi, delta_prev) as a dense
  // symmetric 6x6 in registers; cte enters only its own stage cost and the next cte linearly, so
  // it is carried as a scalar (P44, p4).  Returns whether every 2x2 control pivot was positive
  // definite, i.e. the KKT matrix has inertia (n, m, 0)  -- what Ipopt asks of MUMPS.
  // ------------------------------------------------------------------------------------------
  __device__ bool riccati(bool ls, bool soc, double dwv) {
    const double dt = PC[LC_DT];
    const double cwv = ls ? 0.0 : PC[LC_CW];
    double Pm[6][6], pv[6], P44, p4;
    double zero8[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    {
      const int t = N - 1;
      StageHess H;
      if (PAR) {
        load_hess(t, dwv, H);
      } else {
        double zl[4] = {ST[t][ST_ZL + 0], ST[t][ST_ZL + 1], 0.0, 0.0}, zu[4] = {ST[t][ST_ZU + 0], ST[t][ST_ZU + 1], 0.0, 0.0}, il[4], iu[4];
        const double psi = ST[t][ST_S + 2], v = ST[t][ST_S + 3];
        slack_rcp(psi, v, 0.0, 0.0, false, il, iu);
        hess_at(t, ls, dwv, zero8, v, ST[t][ST_S + 4], ST[t][ST_S + 5], 0.0, 0.0, zero8, zl, zu, il, iu, H);
      }
#pragma unroll
      for (int r = 0; r < 6; r++) {
#pragma unroll
        for (int c = 0; c < 6; c++) Pm[r][c] = 0.0;
      }
      Pm[0][0] = H.qxx; Pm[1][1] = H.qyy; Pm[2][2] = H.qpp; Pm[3][3] = H.qvv; Pm[4][4] = H.qee;
      P44 = H.qcc;
      pv[0] = 0.0; pv[1] = 0.0; pv[2] = H.gp; pv[3] = H.gv; pv[4] = H.ge; pv[5] = 0.0;
      p4 = H.gc;
    }
    bool ok = true;
#pragma unroll 1
    for (int i = N - 2; i >= 0; i--) {
      StageLin L;
      StageHess H;
      double d[6], cn_l[6];
#pragma unroll
      for (int k = 0; k < 6; k++) cn_l[k] = ST[i][ST_CN + k];   // with the other loads of the stage, not behind them
      if (PAR) {
        load_lin(i, L);
        load_hess(i, ls ? 0.0 : dwv, H);
      } else {
        double tg[8], ln[6], zl[4], zu[4], il[4], iu[4];
#pragma unroll
        for (int k = 0; k < 8; k++) tg[k] = ST[i][ST_TG + k];
#pragma unroll
        for (int k = 0; k < 6; k++) ln[k] = ST[i + 1][ST_LAM + k];
#pragma unroll
        for (int k = 0; k < 4; k++) { zl[k] = ST[i][ST_ZL + k]; zu[k] = ST[i][ST_ZU + k]; }
        const double psi = ST[i][ST_S + 2], v = ST[i][ST_S + 3], c = ST[i][ST_S + 4], e = ST[i][ST_S + 5], u0 = ST[i][ST_U + 0], u1 = ST[i][ST_U + 1];
        const double dprev = i >= 1 ? ST[i - 1][ST_U + 0] : 0.0;
        slack_rcp(psi, v, u0, u1, true, il, iu);
        lin_at(tg, v, u0, L);
        hess_at(i, ls, dwv, tg, v, c, e, u0, dprev, ln, zl, zu, il, iu, H);
      }
      if (ls) {
#pragma unroll
        for (int k = 0; k < 6; k++) d[k] = 0.0;
      } else if (soc) {
#pragma unroll
        for (int k = 0; k < 6; k++) d[k] = -ST[i][ST_CS + k];
      } else {
#pragma unroll
        for (int k = 0; k < 6; k++) d[k] = -cn_l[k];
      }
      const bool cpl = i >= 1;
      const double cwe = cpl ? cwv : 0.0;
      // v = P+ d + p+   (rows X, Y, PSI, V, E, DP; d over x, y, psi, v, epsi; cte apart)
      double vv[6];
#pragma unroll
      for (int r = 0; r < 6; r++)
        vv[r] = fma(Pm[r][4], d[5], fma(Pm[r][3], d[3], fma(Pm[r][2], d[2], fma(Pm[r][1], d[1], fma(Pm[r][0], d[0], pv[r])))));
      const double v4 = fma(P44, d[4], p4);
      // T = P+ G, columns x, y, psi, v, delta, a
      double T[6][6];
#pragma unroll
      for (int r = 0; r < 6; r++) {
        const double pe = Pm[r][2] + Pm[r][4];
        T[r][0] = fma(L.a61, Pm[r][4], Pm[r][0]);
        T[r][1] = Pm[r][1];
        T[r][2] = fma(L.a23, Pm[r][1], L.a13 * Pm[r][0]) + pe;
        T[r][3] = fma(L.a34, pe, fma(L.a24, Pm[r][1], L.a14 * Pm[r][0])) + Pm[r][3];
        T[r][4] = fma(L.b3, pe, Pm[r][5]);
        T[r][5] = dt * Pm[r][3];
      }
      // M = G^T T (upper triangle over x, y, psi, v, delta, a), then + cte rank-1 + stage Hessian
      double M[6][6];
#pragma unroll
      for (int c = 0; c < 6; c++) {
        const double te = T[2][c] + T[4][c];
        M[0][c] = fma(L.a61, T[4][c], T[0][c]);
        if (c >= 1) M[1][c] = T[1][c];
        if (c >= 2) M[2][c] = fma(L.a23, T[1][c], L.a13 * T[0][c]) + te;
        if (c >= 3) M[3][c] = fma(L.a34, te, fma(L.a24, T[1][c], L.a14 * T[0][c])) + T[3][c];
        if (c >= 4) M[4][c] = fma(L.b3, te, T[5][c]);
        if (c >= 5) M[5][c] = dt * T[3][c];
      }
      // cte row of G: (a51 [x], -1 [y], a54 [v], a56 [epsi])
      const double g4x = P44 * L.a51, g4v = P44 * L.a54, g4e = P44 * L.a56;
      const double Mxx = fma(g4x, L.a51, M[0][0]) + H.qxx;
      const double Mxy = M[0][1] - g4x;
      const double Mxp = M[0][2];
      const double Mxv = fma(g4x, L.a54, M[0][3]);
      const double Mxe = g4x * L.a56;
      const double Mxd = M[0][4], Mxa = M[0][5];
      const double Myy = M[1][1] + P44 + H.qyy;
      const double Myp = M[1][2];
      const double Myv = M[1][3] - g4v;
      const double Mye = -g4e;
      const double Myd = M[1][4], Mya = M[1][5];
      const double Mpp = M[2][2] + H.qpp;
      const double Mpv = M[2][3] + H.qpv;
      const double Mpd = M[2][4], Mpa = M[2][5];
      const double Mvv = fma(g4v, L.a54, M[3][3]) + H.qvv;
      const double Mve = fma(g4v, L.a56, H.qve);
      const double Mvd = M[3][4] + H.svd, Mva = M[3][5];
      const double Mee = fma(g4e, L.a56, H.qee);
      const double Mdd = M[4][4] + H.rdd, Mda = M[4][5], Maa = M[5][5] + H.raa;
      // delta_prev row: only the rate coupling:  M[dp][dp] = cwe, M[dp][delta] = -cwe
      // m = G^T v + g
      const double ve = vv[2] + vv[4];
      const double mx = fma(L.a51, v4, fma(L.a61, vv[4], vv[0]));
      const double my = vv[1] - v4;
      const double mp = fma(L.a23, vv[1], L.a13 * vv[0]) + ve + H.gp;
      const double mv = fma(L.a54, v4, fma(L.a34, ve, fma(L.a24, vv[1], L.a14 * vv[0])) + vv[3]) + H.gv;
      const double me = fma(L.a56, v4, H.ge);
      const double mdp = H.gdp;
      const double md = fma(L.b3, ve, vv[5]) + H.gd;
      const double ma = fma(dt, vv[3], H.ga);
      // 2x2 control pivot
      const double det = fma(Mdd, Maa, -(Mda * Mda));
      ok = ok && (Mdd > 0.0) && (det > 0.0);
      const double idet = rcp(det);
      const double i11 = Maa * idet, i12 = -Mda * idet, i22 = Mdd * idet;
      // gains K0 (delta), K1 (a) over columns x, y, psi, v, delta_prev (epsi column is zero)
      const double cd[5] = {Mxd, Myd, Mpd, Mvd, -cwe};
      const double ca[5] = {Mxa, Mya, Mpa, Mva, 0.0};
      double K0[5], K1[5];
#pragma unroll
      for (int c = 0; c < 5; c++) {
        K0[c] = -fma(i11, cd[c], i12 * ca[c]);
        K1[c] = -fma(i12, cd[c], i22 * ca[c]);
        ST[i][ST_KG + c] = K0[c];
        ST[i][ST_KG + 5 + c] = K1[c];
      }
      const double k0 = -fma(i11, md, i12 * ma), k1 = -fma(i12, md, i22 * ma);
      ST[i][ST_KG + 10] = k0; ST[i][ST_KG + 11] = k1;
      // Schur complement -> new cost-to-go (index order X, Y, PSI, V, E, DP)
      Pm[0][0] = fma(Mxa, K1[0], fma(Mxd, K0[0], Mxx));
      Pm[0][1] = fma(Mxa, K1[1], fma(Mxd, K0[1], Mxy));
      Pm[0][2] = fma(Mxa, K1[2], fma(Mxd, K0[2], Mxp));
      Pm[0][3] = fma(Mxa, K1[3], fma(Mxd, K0[3], Mxv));
      Pm[0][4] = Mxe;
      Pm[0][5] = fma(Mxa, K1[4], Mxd * K0[4]);
      Pm[1][1] = fma(Mya, K1[1], fma(Myd, K0[1], Myy));
      Pm[1][2] = fma(Mya, K1[2], fma(Myd, K0[2], Myp));
      Pm[1][3] = fma(Mya, K1[3], fma(Myd, K0[3], Myv));
      Pm[1][4] = Mye;
      Pm[1][5] = fma(Mya, K1[4], Myd * K0[4]);
      Pm[2][2] = fma(Mpa, K1[2], fma(Mpd, K0[2], Mpp));
      Pm[2][3] = fma(Mpa, K1[3], fma(Mpd, K0[3], Mpv));
      Pm[2][4] = 0.0;
      Pm[2][5] = fma(Mpa, K1[4], Mpd * K0[4]);
      Pm[3][3] = fma(Mva, K1[3], fma(Mvd, K0[3], Mvv));
      Pm[3][4] = Mve;
      Pm[3][5] = fma(Mva, K1[4], Mvd * K0[4]);
      Pm[4][4] = Mee;
      Pm[4][5] = 0.0;
      Pm[5][5] = fma(-cwe, K0[4], cwe);
#pragma unroll
      for (int r = 1; r < 6; r++) {
#pragma unroll
        for (int c = 0; c < r; c++) Pm[r][c] = Pm[c][r];
      }
      pv[0] = fma(Mxa, k1, fma(Mxd, k0, mx));
      pv[1] = fma(Mya, k1, fma(Myd, k0, my));
      pv[2] = fma(Mpa, k1, fma(Mpd, k0, mp));
      pv[3] = fma(Mva, k1, fma(Mvd, k0, mv));
      pv[4] = me;
      pv[5] = fma(-cwe, k0, mdp);
      P44 = H.qcc;
      p4 = H.gc;
    }
    gsync();   // coop kernel: every lane of the group ran the same recursion and stored the same gains
    return ok;
  }

  // ------------------------------------------------------------------------------------------
  // slot 4 (forward sweep): primal step from the gains, fused with the step-length ratios (fraction
  // to the boundary for x and for z) and grad(phi_mu)^T dx of the line search
  // ------------------------------------------------------------------------------------------
  __device__ void forward_and_ratios(bool ls, bool soc) {
    if (PAR) { forward_par(ls, soc); return; }
    const double dt = PC[LC_DT], cw = PC[LC_CW], wd2 = PC[LC_WD2], wv2 = PC[LC_WV2];
    double t[6], dp = 0.0;
#pragma unroll
    for (int k = 0; k < 6; k++) t[k] = ls ? 0.0 : (soc ? -cs0[k] : -c0[k]);
    double rmax = 0.0;             // max over bounds of  -dx/(x-lo)  or  dx/(hi-x)
    double zn = 1.0, zd = 0.0;     // running minimum of z / (-dz) as a fraction zn / zd (zd > 0)
    double acc = 0.0, dprev = 0.0;
#pragma unroll 1
    for (int i = 0; i < N; i++) {
      const bool hasu = i < N - 1;
      double du0 = 0.0, du1 = 0.0, u0 = 0.0, u1 = 0.0;
      // every load of the stage in one batch at the top (see advance): rows hold all fields for all stages
      const double psi = ST[i][ST_S + 2], v = ST[i][ST_S + 3], s4_l = ST[i][ST_S + 4], s5_l = ST[i][ST_S + 5];
      double kg[12], tg[8], cn_l[6], zl_l[4], zu_l[4];
#pragma unroll
      for (int k = 0; k < 12; k++) kg[k] = ST[i][ST_KG + k];
#pragma unroll
      for (int k = 0; k < 8; k++) tg[k] = ST[i][ST_TG + k];
#pragma unroll
      for (int k = 0; k < 6; k++) cn_l[k] = ST[i][ST_CN + k];
#pragma unroll
      for (int k = 0; k < 4; k++) { zl_l[k] = ST[i][ST_ZL + k]; zu_l[k] = ST[i][ST_ZU + k]; }
      const double u0_l = ST[i][ST_U + 0], u1_l = ST[i][ST_U + 1];
      const double un_l = ST[i + 1 < N ? i + 1 : i][ST_U + 0];
#pragma unroll
      for (int k = 0; k < 6; k++) ST[i][ST_DS + k] = t[k];
      double tn[6] = {0, 0, 0, 0, 0, 0};
      if (hasu) {
        double d[6];
        u0 = u0_l; u1 = u1_l;
        du0 = fma(kg[4], dp, fma(kg[3], t[3], fma(kg[2], t[2], fma(kg[1], t[1], fma(kg[0], t[0], kg[10])))));
        du1 = fma(kg[9], dp, fma(kg[8], t[3], fma(kg[7], t[2], fma(kg[6], t[1], fma(kg[5], t[0], kg[11])))));
        ST[i][ST_DU + 0] = du0; ST[i][ST_DU + 1] = du1;
        // a "tiny step" (Ipopt's DetectTinyStep) needs every component of the step relatively tiny: screen on one
        if (i == 0) tiny_screen = fabs(du0) <= 2.0 * tiny_tol * (1.0 + fabs(u0));
        if (ls) {
#pragma unroll
          for (int k = 0; k < 6; k++) d[k] = 0.0;
        } else if (soc) {
#pragma unroll
          for (int k = 0; k < 6; k++) d[k] = -ST[i][ST_CS + k];
        } else {
#pragma unroll
          for (int k = 0; k < 6; k++) d[k] = -cn_l[k];
        }
        StageLin L;
        lin_at(tg, v, u0, L);
        tn[0] = fma(L.a14, t[3], fma(L.a13, t[2], t[0])) + d[0];
        tn[1] = fma(L.a24, t[3], fma(L.a23, t[2], t[1])) + d[1];
        tn[2] = fma(L.b3, du0, fma(L.a34, t[3], t[2])) + d[2];
        tn[3] = fma(dt, du1, t[3]) + d[3];
        tn[4] = fma(L.a56, t[5], fma(L.a54, t[3], fma(L.a51, t[0], -t[1]))) + d[4];
        tn[5] = fma(L.b3, du0, fma(L.a34, t[3], fma(L.a61, t[0], t[2]))) + d[5];
      }
      if (!ls) {
        acc += fma(we2(i) * s5_l, t[5], fma(wc2(i) * s4_l, t[4], fma(nv2(i), v, wv2 * (v - vref(i))) * t[3]));
        if (hasu) {
          double gd = wd2 * u0;
          if (i >= 1) gd = fma(cw, u0 - dprev, gd);
          if (i <= N - 3) gd = fma(-cw, un_l - u0, gd);
          acc = fma(gd, du0, acc);
          dprev = u0;
        }
        double il[4], iu[4];
        slack_rcp(psi, v, u0, u1, hasu, il, iu);
        const double dx[4] = {t[2], t[3], du0, du1};
#pragma unroll
        for (int k = 0; k < 4; k++) {
          if (k < 2 || hasu) {
            const double zl = zl_l[k], zu = zu_l[k];
            acc = fma(mu * (iu[k] - il[k]), dx[k], acc);
            rmax = dmax(rmax, dmax(-dx[k] * il[k], dx[k] * iu[k]));
            const double dzl = fma(fma(-zl, dx[k], mu), il[k], -zl);
            const double dzu = fma(fma(zu, dx[k], mu), iu[k], -zu);
            // z/(-dz) < zn/zd  <=>  z*zd < zn*(-dz)   (all denominators positive)
            if (dzl < 0.0 && (zd == 0.0 || zl * zd < zn * (-dzl))) { zn = zl; zd = -dzl; }
            if (dzu < 0.0 && (zd == 0.0 || zu * zd < zn * (-dzu))) { zn = zu; zd = -dzu; }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 6; k++) t[k] = tn[k];
      dp = du0;
    }
    gsync();
    gbd_new = acc;
    if (ls) return;
    // alpha_max = min(1, tau / rmax),  alpha_z = min(1, tau * zn / zd)
    alpha_soc = (rmax > tau) ? tau / rmax : 1.0;
    alpha_z = (zd > 0.0 && tau * zn < zd) ? tau * zn / zd : 1.0;
  }

  // coop kernel: the recursion runs identically in every lane of the group (on the derivative pieces of
  // build_lh); each lane keeps the step of its own stage and computes that stage's step-length ratios
  __device__ void forward_par(bool ls, bool soc) {
    const int G = PAR ? NS_GROUP : 1;
    const double dt = PC[LC_DT], cw = PC[LC_CW], wd2 = PC[LC_WD2], wv2 = PC[LC_WV2];
    double t[6], dp = 0.0;
#pragma unroll
    for (int k = 0; k < 6; k++) t[k] = ls ? 0.0 : (soc ? -cs0[k] : -c0[k]);
    double mts[NPASS][6], mdu0s[NPASS], mdu1s[NPASS];
#pragma unroll
    for (int p = 0; p < NPASS; p++) {
      mdu0s[p] = 0.0; mdu1s[p] = 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) mts[p][k] = 0.0;
    }
#pragma unroll 1
    for (int i = 0; i < N; i++) {
      const bool hasu = i < N - 1;
      double du0 = 0.0, du1 = 0.0, tn[6] = {0, 0, 0, 0, 0, 0};
      if (hasu) {
        double kg[12], d[6];
#pragma unroll
        for (int k = 0; k < 12; k++) kg[k] = ST[i][ST_KG + k];
        du0 = fma(kg[4], dp, fma(kg[3], t[3], fma(kg[2], t[2], fma(kg[1], t[1], fma(kg[0], t[0], kg[10])))));
        du1 = fma(kg[9], dp, fma(kg[8], t[3], fma(kg[7], t[2], fma(kg[6], t[1], fma(kg[5], t[0], kg[11])))));
        if (ls) {
#pragma unroll
          for (int k = 0; k < 6; k++) d[k] = 0.0;
        } else if (soc) {
#pragma unroll
          for (int k = 0; k < 6; k++) d[k] = -ST[i][ST_CS + k];
        } else {
#pragma unroll
          for (int k = 0; k < 6; k++) d[k] = -ST[i][ST_CN + k];
        }
        StageLin L;
        load_lin(i, L);
        tn[0] = fma(L.a14, t[3], fma(L.a13, t[2], t[0])) + d[0];
        tn[1] = fma(L.a24, t[3], fma(L.a23, t[2], t[1])) + d[1];
        tn[2] = fma(L.b3, du0, fma(L.a34, t[3], t[2])) + d[2];
        tn[3] = fma(dt, du1, t[3]) + d[3];
        tn[4] = fma(L.a56, t[5], fma(L.a54, t[3], fma(L.a51, t[0], -t[1]))) + d[4];
        tn[5] = fma(L.b3, du0, fma(L.a34, t[3], fma(L.a61, t[0], t[2]))) + d[5];
      }
      if (i % G == g0) {
#pragma unroll
        for (int p = 0; p < NPASS; p++) {
          if (p == i / G) {
#pragma unroll
            for (int k = 0; k < 6; k++) mts[p][k] = t[k];
            mdu0s[p] = du0; mdu1s[p] = du1;
          }
        }
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_DS + k] = t[k];
        if (hasu) { ST[i][ST_DU + 0] = du0; ST[i][ST_DU + 1] = du1; }
      }
#pragma unroll
      for (int k = 0; k < 6; k++) t[k] = tn[k];
      dp = du0;
    }
    double rmax = 0.0, zn = 1.0, zd = 0.0, gbd = 0.0, tall = 1.0;
#pragma unroll
    for (int p = 0; p < NPASS; p++) {
    const int i = g0 + p * G;
    const double *mt = mts[p];
    const double mdu0 = mdu0s[p], mdu1 = mdu1s[p];
    if (!ls && i < N) {
      const bool hasu = i < N - 1;
      const double psi = ST[i][ST_S + 2], v = ST[i][ST_S + 3];
      const double u0 = hasu ? ST[i][ST_U + 0] : 0.0, u1 = hasu ? ST[i][ST_U + 1] : 0.0;
      {   // DetectTinyStep: |dx| <= tiny_step_tol (1 + |x|) in every component
        bool t = fabs(mdu0) <= tiny_tol * (1.0 + fabs(u0)) && fabs(mdu1) <= tiny_tol * (1.0 + fabs(u1));
#pragma unroll
        for (int k = 0; k < 6; k++) t = t && fabs(mt[k]) <= tiny_tol * (1.0 + fabs(ST[i][ST_S + k]));
        if (!t) tall = 0.0;
      }
      double acc = fma(we2(i) * ST[i][ST_S + 5], mt[5], fma(wc2(i) * ST[i][ST_S + 4], mt[4], fma(nv2(i), v, wv2 * (v - vref(i))) * mt[3]));
      if (hasu) {
        double gd = wd2 * u0;
        if (i >= 1) gd = fma(cw, u0 - ST[i - 1][ST_U + 0], gd);
        if (i <= N - 3) gd = fma(-cw, ST[i + 1][ST_U + 0] - u0, gd);
        acc = fma(gd, mdu0, acc);
      }
      double il[4], iu[4];
      slack_rcp(psi, v, u0, u1, hasu, il, iu);
      const double dx[4] = {mt[2], mt[3], mdu0, mdu1};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (k < 2 || hasu) {
          const double zl = ST[i][ST_ZL + k], zu = ST[i][ST_ZU + k];
          acc = fma(mu * (iu[k] - il[k]), dx[k], acc);
          rmax = dmax(rmax, dmax(-dx[k] * il[k], dx[k] * iu[k]));
          const double dzl = fma(fma(-zl, dx[k], mu), il[k], -zl);
          const double dzu = fma(fma(zu, dx[k], mu), iu[k], -zu);
          if (dzl < 0.0 && (zd == 0.0 || zl * zd < zn * (-dzl))) { zn = zl; zd = -dzl; }
          if (dzu < 0.0 && (zd == 0.0 || zu * zd < zn * (-dzu))) { zn = zu; zd = -dzu; }
        }
      }
      gbd = (p == 0) ? acc : gbd + acc;
    }
    }
    gsync();
    // group minimum of zn / zd (zd == 0 stands for +infinity), maximum of rmax, sum of acc
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      const double on = __shfl_xor_sync(gm, zn, o, G), od = __shfl_xor_sync(gm, zd, o, G);
      const bool take = od > 0.0 && (zd == 0.0 || on * zd < zn * od || (on * zd == zn * od && on < zn));
      if (take) { zn = on; zd = od; }
    }
    rmax = gmax<NS_GROUP>(rmax, gm);
    gbd_new = gsum<NS_GROUP>(gbd, gm);
    tiny_all = gmin<NS_GROUP>(tall, gm);
    if (ls) return;
    alpha_soc = (rmax > tau) ? tau / rmax : 1.0;
    alpha_z = (zd > 0.0 && tau * zn < zd) ? tau * zn / zd : 1.0;
  }

  // ---- filter (Ipopt's FilterLSAcceptor) ---------------------------------------------------------
  __device__ __forceinline__ static bool cmp_le(double lhs, double rhs, double basis) {
    return lhs - rhs <= 10.0 * K_EPS * fabs(basis);
  }
  __device__ __forceinline__ bool is_ftype(double a) const { return ls_gbd < 0.0 && a * pow_gbd > pow_theta; }
  __device__ __forceinline__ bool armijo(double a, double phi_t) const {
    return cmp_le(phi_t - ls_phi, K_ETA_PHI * a * ls_gbd, ls_phi);
  }
  // FilterLSAcceptor::IsAcceptableToCurrentIterate (obj_max_inc test unless called from the restoration phase)
  __device__ bool acceptable_to_current(double theta_t, double phi_t, bool from_resto) const {
    if (!from_resto && phi_t > ls_phi) {
      double basval = 1.0;
      if (fabs(ls_phi) > 10.0) basval = log10(fabs(ls_phi));
      if (log10(phi_t - ls_phi) > K_OBJ_MAX_INC + basval) return false;
    }
    return cmp_le(theta_t, (1.0 - K_GAMMA_THETA) * ls_theta, ls_theta) ||
           cmp_le(phi_t - ls_phi, -K_GAMMA_PHI * ls_theta, ls_phi);
  }
  __device__ bool filter_ok(double theta_t, double phi_t) const {
    for (int k = 0; k < nfilt; k++) {
      const double f_t = FLT[2 * k], f_p = FLT[2 * k + 1];
      if (!(cmp_le(theta_t, f_t, f_t) || cmp_le(phi_t, f_p, f_p))) return false;
    }
    return true;
  }
  // FilterLSAcceptor::CheckAcceptabilityOfTrialPoint without its side effects: 2 = acceptable, 1 = rejected by the
  // filter, 0 = rejected by the tests against the current iterate, -1 = not a number / above theta_max
  __device__ int ls_accept(double a, double theta_t, double phi_t) const {
    if (!(theta_t == theta_t) || !(phi_t == phi_t) || isinf(phi_t)) return -1;
    if (theta_t > theta_max) return -1;
    bool ok;
    if (a > 0.0 && is_ftype(a) && ls_theta <= theta_min) ok = armijo(a, phi_t);
    else ok = acceptable_to_current(theta_t, phi_t, false);
    if (!ok) return 0;
    return filter_ok(theta_t, phi_t) ? 2 : 1;
  }
  // entries the filter would hold after filter_add(th, ph) if it had room
  __device__ int filter_count_after(double th, double ph) const {
    int k = 1;
    for (int j = 0; j < nfilt; j++) k += !(FLT[2 * j] >= th && FLT[2 * j + 1] >= ph);
    return k;
  }
  // drop the entries the new one dominates, then add it (a full filter keeps what it has, like the oracle's)
  __device__ void filter_add(double th, double ph) {
    int k = 0;
    for (int j = 0; j < nfilt; j++) {
      const double f_t = FLT[2 * j], f_p = FLT[2 * j + 1];
      if (!(f_t >= th && f_p >= ph)) { FLT[2 * k] = f_t; FLT[2 * k + 1] = f_p; k++; }
    }
    if (k < NFILT) { FLT[2 * k] = th; FLT[2 * k + 1] = ph; k++; }
    nfilt = k;
  }

  // Ipopt's convergence tests and monotone barrier update at the (new) iterate; sets mode
  __device__ void check_and_update_mu(const KParams &P) {
    const double sf = PC[LC_SF];
    const int nz = 4 * N + 4 * (N - 1), m = 6 * N;
    const double sd = fmax(K_S_MAX, (lam1 + z1) / (double)(m + nz)) / K_S_MAX;
    const double sc = fmax(K_S_MAX, z1 / (double)nz) / K_S_MAX;
    const double compl0 = compl_err(0.0);
    const double E0 = nanmax(dinf / sd, nanmax(cviol, compl0 / sc));
    const double dinf_u = dinf / sf, compl_u = compl0 / sf;
    if (E0 <= P.tol && dinf_u <= K_DUAL_INF_TOL && cviol <= K_CONSTR_VIOL_TOL && compl_u <= K_COMPL_INF_TOL) {
      status = 1; mode = LM_FINISH; return;
    }
    acceptable_now = false;
    if (E0 <= K_ACCEPT_TOL && cviol <= K_ACCEPT_CONSTR_VIOL_TOL && compl_u <= K_ACCEPT_COMPL_INF_TOL) {
      acceptable_now = true;
      if (++accept_cnt >= K_ACCEPT_ITER) { status = 4; mode = LM_FINISH; return; }
    } else {
      accept_cnt = 0;
    }
    if (!(E0 == E0)) { status = 11; mode = LM_FINISH; return; }
    if (iter >= P.max_iter) { status = 2; mode = LM_FINISH; return; }
    // monotone barrier update; a repeated tiny step (FULL kernels only) forces a decrease, and ends the run when
    // the barrier parameter is at its floor
    bool tf = FULL && tiny_flag;
    for (;;) {
      const double cm = compl_err(mu);
      const double Emu = nanmax(dinf / sd, nanmax(cviol, cm / sc));
      if (!(Emu <= K_KAPPA_EPS * mu) && !tf) break;
      const double mu_min = fmin(P.tol, K_COMPL_INF_TOL) / (K_KAPPA_EPS + 1.0);
      const double new_mu = fmax(mu_min, fmin(K_KAPPA_MU * mu, mu * sqrt(mu)));
      if (new_mu == mu) {
        if (tf) { status = 3; mode = LM_FINISH; return; }
        break;
      }
      mu = new_mu;
      tau = fmax(K_TAU_MIN, 1.0 - mu);
      tf = false;
      reset_line_search();
    }
    tiny_flag = false;
    dw = 0.0;
    mode = LM_NEWTON;
  }

  // honor_original_bounds, unscaled objective, outputs of MPC.cpp:306-324
  __device__ void write_outputs(const KParams &P) {
    const size_t B = (size_t)P.B;
    const double cw = PC[LC_CW], wd2 = PC[LC_WD2], wv2 = PC[LC_WV2];
    double fl = 0.0, dprev = 0.0;
    // a few lanes of a warp retire per trip and the whole warp waits for their rows: load them one stage ahead
    double sl[6], ul0 = ST[0][ST_U + 0], ul1 = ST[0][ST_U + 1];
#pragma unroll
    for (int k = 0; k < 6; k++) sl[k] = ST[0][ST_S + k];
#pragma unroll 1
    for (int i = 0; i < N; i++) {
      const bool hasu = i < N - 1;
      double s[6];
#pragma unroll
      for (int k = 0; k < 6; k++) s[k] = sl[k];
      const double ur0 = ul0, ur1 = ul1;
      {
        const int j = i + 1 < N ? i + 1 : i;
#pragma unroll
        for (int k = 0; k < 6; k++) sl[k] = ST[j][ST_S + k];
        ul0 = ST[j][ST_U + 0]; ul1 = ST[j][ST_U + 1];
      }
      s[2] = fmin(fmax(s[2], PC[LC_LO0]), PC[LC_HI0]);
      s[3] = fmin(fmax(s[3], PC[LC_LO0 + 1]), PC[LC_HI0 + 1]);
      const double dv = s[3] - vref(i);
      fl = fma(0.5, fma(nv2(i) * s[3], s[3], fma(wv2 * dv, dv, fma(we2(i) * s[5], s[5], wc2(i) * s[4] * s[4]))), fl);
      double u0 = 0.0, u1 = 0.0;
      if (hasu) {
        u0 = fmin(fmax(ur0, PC[LC_LO0 + 2]), PC[LC_HI0 + 2]);
        u1 = fmin(fmax(ur1, PC[LC_LO0 + 3]), PC[LC_HI0 + 3]);
        fl = fma(0.5 * wd2 * u0, u0, fl);
        if (i >= 1) { const double dd = u0 - dprev; fl = fma(0.5 * cw * dd, dd, fl); }
        dprev = u0;
      }
      if (i == 1) {
#pragma unroll
        for (int k = 0; k < 6; k++) P.result[(size_t)k * B + b] = s[k];
      }
      if (i == 0) { P.result[6 * B + b] = u0; P.result[7 * B + b] = u1; }
      if (P.dual_lam) {   // multipliers of the reference's NLP (objective unscaled): rows k*N+i, variables as MPC.cpp:189-196
        const int Nf = P.Nmax;
        const double isf = 1.0 / PC[LC_SF];
#pragma unroll
        for (int k = 0; k < 6; k++) P.dual_lam[(size_t)(k * Nf + i) * B + b] = ST[i][ST_LAM + k] * isf;
        P.dual_zl[(size_t)(2 * Nf + i) * B + b] = ST[i][ST_ZL + 0] * isf; P.dual_zu[(size_t)(2 * Nf + i) * B + b] = ST[i][ST_ZU + 0] * isf;
        P.dual_zl[(size_t)(3 * Nf + i) * B + b] = ST[i][ST_ZL + 1] * isf; P.dual_zu[(size_t)(3 * Nf + i) * B + b] = ST[i][ST_ZU + 1] * isf;
        if (hasu) {
          P.dual_zl[(size_t)(6 * Nf + i) * B + b] = ST[i][ST_ZL + 2] * isf; P.dual_zu[(size_t)(6 * Nf + i) * B + b] = ST[i][ST_ZU + 2] * isf;
          P.dual_zl[(size_t)(7 * Nf - 1 + i) * B + b] = ST[i][ST_ZL + 3] * isf; P.dual_zu[(size_t)(7 * Nf - 1 + i) * B + b] = ST[i][ST_ZU + 3] * isf;
        }
      }
      if (P.traj_x) P.traj_x[(size_t)i * B + b] = s[0];
      if (P.traj_y) P.traj_y[(size_t)i * B + b] = s[1];
      if (P.full) {
        const int Nf = P.Nmax;
#pragma unroll
        for (int k = 0; k < 6; k++) P.full[(size_t)(k * Nf + i) * B + b] = s[k];
        if (hasu) {
          P.full[(size_t)(6 * Nf + i) * B + b] = u0;
          P.full[(size_t)(7 * Nf - 1 + i) * B + b] = u1;
        }
      }
    }
    P.result[8 * B + b] = fl / PC[LC_SF];
    if (P.status) P.status[b] = status;
    if (P.iters) P.iters[b] = iter;
  }


  // ---- migration: the complete state of a problem at a trip boundary as a flat record of doubles.  The
  // lane kernel and the coop kernel run the same arithmetic on the same state, so a problem can be moved
  // from one to the other between any two trips without changing a single bit of its result.
  enum { CK_ROWS = NS * ST_KEEP, CK_PC = CK_ROWS, CK_FLT = CK_PC + LC_SIZE, CK_C = CK_FLT + 2 * K_NFILT, CK_D = CK_C + 18,
         CK_I = CK_D + 32, CK_SIZE = CK_I + 12 };
  __device__ void save(double *r) const {
#pragma unroll 1
    for (int i = g0; i < N; i += gstep)
      for (int k = 0; k < ST_KEEP; k++) r[i * ST_KEEP + k] = ST[i][k];
    if (g0 != 0) return;
    for (int k = 0; k < LC_SIZE; k++) r[CK_PC + k] = PC[k];
    for (int k = 0; k < 2 * K_NFILT; k++) r[CK_FLT + k] = FLT[k];
    for (int k = 0; k < 6; k++) { r[CK_C + k] = c0[k]; r[CK_C + 6 + k] = c0t[k]; r[CK_C + 12 + k] = cs0[k]; }
    const double d[32] = {mu, tau, theta_min, theta_max, dw, dw_last, dw_used, alpha, alpha_z, alpha_test, alpha_soc,
                          alpha_min, ls_theta, ls_phi, ls_gbd, pow_gbd, pow_theta, fx, lsum, theta, ft, lt, tht,
                          theta_soc_old, dinf, cviol, amin, amax, lam1, z1, lsq_lmax, gbd_new};
    for (int k = 0; k < 32; k++) r[CK_D + k] = d[k];
    const int n[12] = {b, N, mode, status, iter, accept_cnt, nfilt, ntrial, soc_cnt, wd_short,
                       n_filter_resets * 8 + succ_filter_rej, (last_rej_filter ? 1 : 0) | (acceptable_now ? 2 : 0)};
    for (int k = 0; k < 12; k++) r[CK_I + k] = (double)n[k];
  }
  __device__ void load(const double *r) {
    N = (int)r[CK_I + 1];
#pragma unroll 1
    for (int i = g0; i < N; i += gstep)
      for (int k = 0; k < ST_KEEP; k++) ST[i][k] = r[i * ST_KEEP + k];
    for (int k = 0; k < LC_SIZE; k++) PC[k] = r[CK_PC + k];
    for (int k = 0; k < 2 * K_NFILT; k++) FLT[k] = r[CK_FLT + k];
    for (int k = 0; k < 6; k++) { c0[k] = r[CK_C + k]; c0t[k] = r[CK_C + 6 + k]; cs0[k] = r[CK_C + 12 + k]; }
    const double *d = r + CK_D;
    mu = d[0]; tau = d[1]; theta_min = d[2]; theta_max = d[3]; dw = d[4]; dw_last = d[5]; dw_used = d[6]; alpha = d[7];
    alpha_z = d[8]; alpha_test = d[9]; alpha_soc = d[10]; alpha_min = d[11]; ls_theta = d[12]; ls_phi = d[13];
    ls_gbd = d[14]; pow_gbd = d[15]; pow_theta = d[16]; fx = d[17]; lsum = d[18]; theta = d[19]; ft = d[20]; lt = d[21];
    tht = d[22]; theta_soc_old = d[23]; dinf = d[24]; cviol = d[25]; amin = d[26]; amax = d[27]; lam1 = d[28];
    z1 = d[29]; lsq_lmax = d[30]; gbd_new = d[31];
    const double *n = r + CK_I;
    b = (int)n[0]; mode = (int)n[2]; status = (int)n[3]; iter = (int)n[4]; accept_cnt = (int)n[5]; nfilt = (int)n[6];
    ntrial = (int)n[7]; soc_cnt = (int)n[8];
    wd_short = (int)n[9]; n_filter_resets = (int)n[10] >> 3; succ_filter_rej = (int)n[10] & 7;
    last_rej_filter = ((int)n[11] & 1) != 0; acceptable_now = ((int)n[11] & 2) != 0;
    escalate = false; tiny_screen = false; tiny_flag = false; tiny_last = false; in_watchdog = false;
    force_accept = false; wd_skip = false; was_tiny = false; wd_trial = 0; trips = 0;
    lh_stale = true;
    gsync();
  }

  // ---- global scratch of a lane group (FULL kernels): watchdog backup, restoration-phase backup and rows
  enum { SC_WD_ROWS = 0, SC_WD_SC = NS * ST_KEEP, SC_BK_ROWS = SC_WD_SC + 32, SC_BK_SC = SC_BK_ROWS + NS * ST_KEEP,
         SC_RS = SC_BK_SC + 32, SC_SIZE = SC_RS + NS * 64 };
  // StartWatchDog: remember the iterate, the search direction and the line search's reference values
  __device__ void watchdog_start() {
    in_watchdog = true; wd_trial = 0; wd_alpha_test = alpha_max;
    double *r = scratch + SC_WD_ROWS;
#pragma unroll 1
    for (int i = g0; i < N; i += gstep)
      for (int k = 0; k < ST_KEEP; k++) r[i * ST_KEEP + k] = ST[i][k];
    if (g0 == 0) {
      double *q = scratch + SC_WD_SC;
      const double d[26] = {alpha_max, alpha_z, ls_theta, ls_phi, ls_gbd, pow_gbd, pow_theta, alpha_min, fx, lsum, theta,
                            dw_used, dinf, cviol, amin, amax, lam1, z1, c0[0], c0[1], c0[2], c0[3], c0[4], c0[5], 0.0, 0.0};
      for (int k = 0; k < 26; k++) q[k] = d[k];
    }
    gsync();
  }
  // StopWatchDog: back to that iterate and direction; the line search goes on from there by backtracking
  __device__ void watchdog_stop() {
    gsync();
    const double *r = scratch + SC_WD_ROWS;
#pragma unroll 1
    for (int i = g0; i < N; i += gstep)
      for (int k = 0; k < ST_KEEP; k++) ST[i][k] = r[i * ST_KEEP + k];
    const double *q = scratch + SC_WD_SC;
    alpha_max = q[0]; alpha_z = q[1]; ls_theta = q[2]; ls_phi = q[3]; ls_gbd = q[4]; pow_gbd = q[5]; pow_theta = q[6];
    alpha_min = q[7]; fx = q[8]; lsum = q[9]; theta = q[10]; dw_used = q[11]; dinf = q[12]; cviol = q[13]; amin = q[14];
    amax = q[15]; lam1 = q[16]; z1 = q[17];
    for (int k = 0; k < 6; k++) c0[k] = q[18 + k];
    in_watchdog = false; wd_short = 0; lh_stale = true;
    gsync();
  }
  // ==========================================================================================================
  // Ipopt's feasibility restoration phase (IpRestoMinC_1Nrm, restated in oracle/mpc_oracle.c: restoration()):
  //     min  rho sum(n + p) + eta/2 ||D_R (x - x_R)||^2     s.t.  c(x) + n - p = 0,  bounds on x,  n, p >= 0
  // with eta = sqrt(mu), D_R = diag(1 / max(1, |x_R|)), solved from x_R by the same interior-point iteration until
  // the point is acceptable to the ORIGINAL problem's filter and has reduced its infeasibility by K_RESTO_KAPPA.
  // The slacks n, p (one pair per constraint row) and their multipliers are eliminated from the Newton system; what
  // remains is the original stage structure with "soft" dynamics: row block i reads  ds_i = w_i + D_i y+_i  with
  // D_i = 1/Sigma_n + 1/Sigma_p > 0, where w_i is the successor the hard constraint would give.  In the Riccati
  // recursion that is one extra step per stage, P~ = (I + P D)^-1 P and p~ = (I + P D)^-1 p (computed as a 5x5
  // Cholesky of I + D^1/2 P D^1/2, whose pivots join the 2x2 control pivots in the inertia test), and the new
  // multipliers fall out of the forward sweep: y+_i = -(P~ w_i + p~).
  // FULL (coop) kernels only; runs to completion inside one trip.  Iterate x lives in the rows as usual, the
  // multipliers y of the restoration problem in ST_LAM, its bound multipliers in ST_ZL / ST_ZU; x_R and the original
  // multipliers are the backup rows in the group's global scratch, which also holds n, p, z_n, z_p, y+, P~, D.
  // ==========================================================================================================
  enum { RS_N = 0, RS_P = 6, RS_ZN = 12, RS_ZP = 18, RS_YP = 24, RS_PT = 30, RS_D = 52, RS_DH = 58, RS_ROW = 64 };
  __device__ __forceinline__ double *rs(int blk) const { return scratch + SC_RS + (size_t)blk * RS_ROW; }
  __device__ __forceinline__ const double *bk(int i) const { return scratch + SC_BK_ROWS + (size_t)i * ST_KEEP; }
  __device__ __forceinline__ static double dr2_of(double xr) { const double d = 1.0 / fmax(1.0, fabs(xr)); return d * d; }
  // restoration-phase scalars (uniform over the group)
  double mu_r, tau_r, dw_r, eta_r, alpha_max_r, alpha_z_r, gbd_r;
  double r_dinf, r_cviol, r_infpr, r_amin, r_amax, r_ysum, r_zsum, r_thR, r_fR, r_lR;

  // optimality error terms of the restoration problem at its current iterate (eta_r, mu-independent parts)
  __device__ void resto_errors() {
    const double dt = PC[LC_DT], eta = eta_r;
    double r = 0.0, cv = 0.0, ip = 0.0, ys = 0.0, zs = 0.0, am = 1e300, aM = 0.0;
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const bool hasu = i < N - 1;
      const double *b = bk(i);
      const double *q = rs(i);
      double s[6], y[6], yn[6], zl[4], zu[4], tg[8], u0 = 0.0, u1 = 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) { s[k] = ST[i][ST_S + k]; y[k] = ST[i][ST_LAM + k]; yn[k] = hasu ? ST[i + 1][ST_LAM + k] : 0.0; }
#pragma unroll
      for (int k = 0; k < 4; k++) { zl[k] = (k < 2 || hasu) ? ST[i][ST_ZL + k] : 0.0; zu[k] = (k < 2 || hasu) ? ST[i][ST_ZU + k] : 0.0; }
#pragma unroll
      for (int k = 0; k < 8; k++) tg[k] = hasu ? ST[i][ST_TG + k] : 0.0;
      if (hasu) { u0 = ST[i][ST_U + 0]; u1 = ST[i][ST_U + 1]; }
      StageLin L;
      lin_at(tg, s[3], u0, L);
      double os[6] = {0, 0, 0, 0, 0, 0}, ou0 = 0.0, ou1 = 0.0;
      if (hasu) {
        const double l25 = yn[2] + yn[5];
        os[0] = fma(L.a61, yn[5], fma(L.a51, yn[4], yn[0]));
        os[1] = yn[1] - yn[4];
        os[2] = fma(L.a23, yn[1], L.a13 * yn[0]) + l25;
        os[3] = fma(L.a54, yn[4], fma(L.a34, l25, fma(L.a24, yn[1], L.a14 * yn[0])) + yn[3]);
        os[5] = L.a56 * yn[4];
        ou0 = L.b3 * l25;
        ou1 = dt * yn[3];
      }
      double g[6];
#pragma unroll
      for (int k = 0; k < 6; k++) g[k] = eta * dr2_of(b[ST_S + k]) * (s[k] - b[ST_S + k]);
      g[2] += -zl[0] + zu[0];
      g[3] += -zl[1] + zu[1];
#pragma unroll
      for (int k = 0; k < 6; k++) {
        r = nanmax(r, fabs(g[k] + y[k] - os[k]));
        ys += fabs(y[k]);
        const double c = (i == 0) ? c0[k] : ST[i - 1][ST_CN + k];
        const double n = q[RS_N + k], p = q[RS_P + k], zn = q[RS_ZN + k], zp = q[RS_ZP + k];
        cv = nanmax(cv, fabs(c + n - p));
        ip = nanmax(ip, fabs(c));
        r = nanmax(r, nanmax(fabs(K_RESTO_RHO + y[k] - zn), fabs(K_RESTO_RHO - y[k] - zp)));
        const double v = n * zn, w = p * zp;
        am = dmin(am, dmin(v, w));
        aM = dmax(aM, dmax(v, w));
        zs += fabs(zn) + fabs(zp);
      }
      zs += fabs(zl[0]) + fabs(zu[0]) + fabs(zl[1]) + fabs(zu[1]);
      {
        const double p0 = (s[2] - PC[LC_LO]) * zl[0], p1 = (PC[LC_HI] - s[2]) * zu[0];
        const double p2 = (s[3] - PC[LC_LO + 1]) * zl[1], p3 = (PC[LC_HI + 1] - s[3]) * zu[1];
        am = dmin(am, dmin(dmin(p0, p1), dmin(p2, p3)));
        aM = dmax(aM, dmax(dmax(p0, p1), dmax(p2, p3)));
      }
      if (hasu) {
        const double gd = eta * dr2_of(b[ST_U + 0]) * (u0 - b[ST_U + 0]);
        const double ga = eta * dr2_of(b[ST_U + 1]) * (u1 - b[ST_U + 1]);
        r = nanmax(r, fabs(gd - ou0 - zl[2] + zu[2]));
        r = nanmax(r, fabs(ga - ou1 - zl[3] + zu[3]));
        zs += fabs(zl[2]) + fabs(zu[2]) + fabs(zl[3]) + fabs(zu[3]);
        const double p0 = (u0 - PC[LC_LO + 2]) * zl[2], p1 = (PC[LC_HI + 2] - u0) * zu[2];
        const double p2 = (u1 - PC[LC_LO + 3]) * zl[3], p3 = (PC[LC_HI + 3] - u1) * zu[3];
        am = dmin(am, dmin(dmin(p0, p1), dmin(p2, p3)));
        aM = dmax(aM, dmax(dmax(p0, p1), dmax(p2, p3)));
      }
    }
    r_dinf = gmax<NS_GROUP>(r, gm); r_cviol = gmax<NS_GROUP>(cv, gm); r_infpr = gmax<NS_GROUP>(ip, gm);
    r_ysum = gsum<NS_GROUP>(ys, gm); r_zsum = gsum<NS_GROUP>(zs, gm);
    r_amin = gmin<NS_GROUP>(am, gm); r_amax = gmax<NS_GROUP>(aM, gm);
  }

  // derivative pieces of every stage for the restoration problem's Newton system, into the shared rows (ST_LH):
  // W = sum_j y_j Hess c_j + eta D_R^2 (no objective term), gradient eta D_R^2 (x - x_R) + barrier terms
  __device__ void resto_build_lh() {
    const double dt = PC[LC_DT], dtLf = PC[LC_DTLF], eta = eta_r;
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const bool hasu = i < N - 1;
      const double *b = bk(i);
      double tg[8], ln[6], zl[4], zu[4], il[4], iu[4], s[6];
#pragma unroll
      for (int k = 0; k < 8; k++) tg[k] = hasu ? ST[i][ST_TG + k] : 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) { ln[k] = hasu ? ST[i + 1][ST_LAM + k] : 0.0; s[k] = ST[i][ST_S + k]; }
#pragma unroll
      for (int k = 0; k < 4; k++) { zl[k] = (k < 2 || hasu) ? ST[i][ST_ZL + k] : 0.0; zu[k] = (k < 2 || hasu) ? ST[i][ST_ZU + k] : 0.0; }
      const double u0 = hasu ? ST[i][ST_U + 0] : 0.0, u1 = hasu ? ST[i][ST_U + 1] : 0.0;
      slack_rcp(s[2], s[3], u0, u1, hasu, il, iu);
      StageLin L;
      lin_at(tg, s[3], u0, L);
      double sig[4], gb[4], e[8];
#pragma unroll
      for (int k = 0; k < 4; k++) { sig[k] = fma(zl[k], il[k], zu[k] * iu[k]); gb[k] = mu_r * (iu[k] - il[k]); }
#pragma unroll
      for (int k = 0; k < 6; k++) e[k] = eta * dr2_of(b[ST_S + k]);
      e[6] = hasu ? eta * dr2_of(b[ST_U + 0]) : 0.0;
      e[7] = hasu ? eta * dr2_of(b[ST_U + 1]) : 0.0;
      const double vdt = s[3] * dt;
      double *q = &ST[i][ST_LH];
      q[0] = L.a13; q[1] = L.a14; q[2] = L.a23; q[3] = L.a24; q[4] = L.a34; q[5] = L.b3; q[6] = L.a51; q[7] = L.a54;
      q[8] = L.a56; q[9] = L.a61;
      q[10] = (hasu ? fma(ln[5], tg[7], -(ln[4] * tg[5])) : 0.0) + e[0];                       // qxx
      q[11] = e[1];                                                                             // qyy
      q[12] = (hasu ? fma(ln[0], tg[1], ln[1] * tg[0]) * vdt : 0.0) + sig[0] + e[2];           // qpp
      q[13] = hasu ? fma(ln[0], tg[0], -(ln[1] * tg[1])) * dt : 0.0;                           // qpv
      q[14] = sig[1] + e[3];                                                                    // qvv
      q[15] = hasu ? -ln[4] * tg[3] * dt : 0.0;                                                // qve
      q[16] = e[4];                                                                             // qcc
      q[17] = (hasu ? ln[4] * tg[2] * vdt : 0.0) + e[5];                                       // qee
      q[18] = hasu ? -(ln[2] + ln[5]) * dtLf : 0.0;                                            // svd
      q[19] = hasu ? e[6] + sig[2] : 0.0;                                                      // rdd
      q[20] = hasu ? e[7] + sig[3] : 0.0;                                                      // raa
      q[21] = e[2] * (s[2] - b[ST_S + 2]) + gb[0];                                             // gp
      q[22] = e[3] * (s[3] - b[ST_S + 3]) + gb[1];                                             // gv
      q[23] = e[4] * (s[4] - b[ST_S + 4]);                                                     // gc
      q[24] = e[5] * (s[5] - b[ST_S + 5]);                                                     // ge
      q[25] = 0.0;                                                                              // gdp
      q[26] = hasu ? e[6] * (u0 - b[ST_U + 0]) + gb[2] : 0.0;                                  // gd
      q[27] = hasu ? e[7] * (u1 - b[ST_U + 1]) + gb[3] : 0.0;                                  // ga
      q[28] = e[0] * (s[0] - b[ST_S + 0]);                                                     // gx
      q[29] = e[1] * (s[1] - b[ST_S + 1]);                                                     // gy
    }
    gsync();
  }

  // (2,2) diagonal D and right-hand side of every constraint block after the elimination of n and p:
  //   D = 1/(Sigma_n + dw) + 1/(Sigma_p + dw),   dh = rc - (rho - mu/n)/(Sigma_n + dw) + (rho - mu/p)/(Sigma_p + dw)
  // rc = c + n - p, or the accumulated second-order-correction residual (ST_CS / cs0)
  __device__ void resto_rhs(bool soc, double dwv) {
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      double *q = rs(i);
#pragma unroll
      for (int k = 0; k < 6; k++) {
        const double n = q[RS_N + k], p = q[RS_P + k];
        const double sn = q[RS_ZN + k] / n + dwv, sp = q[RS_ZP + k] / p + dwv;
        double rc;
        if (soc) rc = (i == 0) ? cs0[k] : ST[i - 1][ST_CS + k];
        else rc = ((i == 0) ? c0[k] : ST[i - 1][ST_CN + k]) + n - p;
        q[RS_D + k] = 1.0 / sn + 1.0 / sp;
        q[RS_DH + k] = rc - (K_RESTO_RHO - mu_r / n) / sn + (K_RESTO_RHO - mu_r / p) / sp;
      }
    }
    gsync();
  }

  // P~ = (I + P D)^-1 P, p~ = (I + P D)^-1 p for the cost-to-go entering constraint block blk; stored for the forward
  // sweep.  Over (x, y, psi, v, epsi) as a 5x5 Cholesky of I + E P E, E = D^1/2; the cte term is a scalar.  Returns
  // whether every pivot was positive (part of the inertia test).
  __device__ __forceinline__ bool resto_soften(int blk, double (&Pm)[6][6], double (&pv)[6], double &P44, double &p4) {
    const double *q = rs(blk);
    const double Dk[5] = {q[RS_D + 0], q[RS_D + 1], q[RS_D + 2], q[RS_D + 3], q[RS_D + 5]};
    const double Dc = q[RS_D + 4];
    double e[5], S[5][5], X[5][5], qv[5];
    bool ok = true;
#pragma unroll
    for (int j = 0; j < 5; j++) e[j] = sqrt(Dk[j]);
#pragma unroll
    for (int r = 0; r < 5; r++) {
#pragma unroll
      for (int c = 0; c < 5; c++) { S[r][c] = e[r] * Pm[r][c] * e[c] + (r == c ? 1.0 : 0.0); X[r][c] = e[r] * Pm[r][c]; }
      qv[r] = e[r] * pv[r];
    }
    // Cholesky S = L L^T in place (lower), then X <- L^-1 X, qv <- L^-1 qv
#pragma unroll
    for (int j = 0; j < 5; j++) {
      double d = S[j][j];
#pragma unroll
      for (int k = 0; k < j; k++) d -= S[j][k] * S[j][k];
      ok = ok && (d > 0.0);
      const double l = sqrt(d), il = 1.0 / l;
      S[j][j] = l;
#pragma unroll
      for (int i = j + 1; i < 5; i++) {
        double v = S[i][j];
#pragma unroll
        for (int k = 0; k < j; k++) v -= S[i][k] * S[j][k];
        S[i][j] = v * il;
      }
    }
#pragma unroll
    for (int i = 0; i < 5; i++) {
      const double il = 1.0 / S[i][i];
#pragma unroll
      for (int c = 0; c < 5; c++) {
        double v = X[i][c];
#pragma unroll
        for (int k = 0; k < i; k++) v -= S[i][k] * X[k][c];
        X[i][c] = v * il;
      }
      double v = qv[i];
#pragma unroll
      for (int k = 0; k < i; k++) v -= S[i][k] * qv[k];
      qv[i] = v * il;
    }
    double Pt[5][5], pt[5];
#pragma unroll
    for (int r = 0; r < 5; r++) {
#pragma unroll
      for (int c = r; c < 5; c++) {
        double v = Pm[r][c];
#pragma unroll
        for (int k = 0; k < 5; k++) v -= X[k][r] * X[k][c];
        Pt[r][c] = v;
      }
      double v = pv[r];
#pragma unroll
      for (int k = 0; k < 5; k++) v -= X[k][r] * qv[k];
      pt[r] = v;
    }
    const double den = fma(Dc, P44, 1.0);
    ok = ok && (den > 0.0);
    const double P44t = P44 / den, p4t = p4 / den;
    if (g0 == 0) {
      double *w = rs(blk) + RS_PT;
      int t = 0;
#pragma unroll
      for (int r = 0; r < 5; r++) {
#pragma unroll
        for (int c = r; c < 5; c++) w[t++] = Pt[r][c];
      }
#pragma unroll
      for (int r = 0; r < 5; r++) w[15 + r] = pt[r];
      w[20] = P44t; w[21] = p4t;
    }
#pragma unroll
    for (int r = 0; r < 5; r++) {
#pragma unroll
      for (int c = r; c < 5; c++) { Pm[r][c] = Pt[r][c]; Pm[c][r] = Pt[r][c]; }
      pv[r] = pt[r];
      Pm[r][5] = 0.0; Pm[5][r] = 0.0;
    }
    Pm[5][5] = 0.0; pv[5] = 0.0;
    P44 = P44t; p4 = p4t;
    return ok;
  }

  // backward Riccati sweep of the restoration problem: riccati()'s stage algebra on the pieces of resto_build_lh, with
  // the cost-to-go softened at every constraint block (the initial-state block included) and no steering-rate coupling
  __device__ bool riccati_resto(double dwv) {
    const double dt = PC[LC_DT];
    double Pm[6][6], pv[6], P44, p4;
    {
      StageHess H;
      load_hess(N - 1, dwv, H);
      const double *q = &ST[N - 1][ST_LH];
#pragma unroll
      for (int r = 0; r < 6; r++) {
#pragma unroll
        for (int c = 0; c < 6; c++) Pm[r][c] = 0.0;
      }
      Pm[0][0] = H.qxx; Pm[1][1] = H.qyy; Pm[2][2] = H.qpp; Pm[3][3] = H.qvv; Pm[4][4] = H.qee;
      P44 = H.qcc;
      pv[0] = q[28]; pv[1] = q[29]; pv[2] = H.gp; pv[3] = H.gv; pv[4] = H.ge; pv[5] = 0.0;
      p4 = H.gc;
    }
    bool ok = true;
#pragma unroll 1
    for (int i = N - 2; i >= 0; i--) {
      ok = resto_soften(i + 1, Pm, pv, P44, p4) && ok;
      StageLin L;
      StageHess H;
      load_lin(i, L);
      load_hess(i, dwv, H);
      const double gx = ST[i][ST_LH + 28], gy = ST[i][ST_LH + 29];
      const double *dh = rs(i + 1) + RS_DH;
      double d[6];
#pragma unroll
      for (int k = 0; k < 6; k++) d[k] = -dh[k];
      // v = P+ d + p+   (rows X, Y, PSI, V, E, DP; d over x, y, psi, v, epsi; cte apart)
      double vv[6];
#pragma unroll
      for (int r = 0; r < 6; r++)
        vv[r] = fma(Pm[r][4], d[5], fma(Pm[r][3], d[3], fma(Pm[r][2], d[2], fma(Pm[r][1], d[1], fma(Pm[r][0], d[0], pv[r])))));
      const double v4 = fma(P44, d[4], p4);
      double T[6][6];
#pragma unroll
      for (int r = 0; r < 6; r++) {
        const double pe = Pm[r][2] + Pm[r][4];
        T[r][0] = fma(L.a61, Pm[r][4], Pm[r][0]);
        T[r][1] = Pm[r][1];
        T[r][2] = fma(L.a23, Pm[r][1], L.a13 * Pm[r][0]) + pe;
        T[r][3] = fma(L.a34, pe, fma(L.a24, Pm[r][1], L.a14 * Pm[r][0])) + Pm[r][3];
        T[r][4] = fma(L.b3, pe, Pm[r][5]);
        T[r][5] = dt * Pm[r][3];
      }
      double M[6][6];
#pragma unroll
      for (int c = 0; c < 6; c++) {
        const double te = T[2][c] + T[4][c];
        M[0][c] = fma(L.a61, T[4][c], T[0][c]);
        if (c >= 1) M[1][c] = T[1][c];
        if (c >= 2) M[2][c] = fma(L.a23, T[1][c], L.a13 * T[0][c]) + te;
        if (c >= 3) M[3][c] = fma(L.a34, te, fma(L.a24, T[1][c], L.a14 * T[0][c])) + T[3][c];
        if (c >= 4) M[4][c] = fma(L.b3, te, T[5][c]);
        if (c >= 5) M[5][c] = dt * T[3][c];
      }
      // the softened cost-to-go is dense over (x, y, psi, v, epsi): the epsi column of M = G^T P~ G, which is zero
      // with a hard constraint, is not (G's epsi column is only the cte row, handled below; P~'s epsi row is T[.][.])
      // epsi enters s_{i+1} only through cte (a56), so G^T P~ G has no epsi entries beyond the cte rank-1 term.
      const double g4x = P44 * L.a51, g4v = P44 * L.a54, g4e = P44 * L.a56;
      const double Mxx = fma(g4x, L.a51, M[0][0]) + H.qxx;
      const double Mxy = M[0][1] - g4x;
      const double Mxp = M[0][2];
      const double Mxv = fma(g4x, L.a54, M[0][3]);
      const double Mxe = g4x * L.a56;
      const double Mxd = M[0][4], Mxa = M[0][5];
      const double Myy = M[1][1] + P44 + H.qyy;
      const double Myp = M[1][2];
      const double Myv = M[1][3] - g4v;
      const double Mye = -g4e;
      const double Myd = M[1][4], Mya = M[1][5];
      const double Mpp = M[2][2] + H.qpp;
      const double Mpv = M[2][3] + H.qpv;
      const double Mpd = M[2][4], Mpa = M[2][5];
      const double Mvv = fma(g4v, L.a54, M[3][3]) + H.qvv;
      const double Mve = fma(g4v, L.a56, H.qve);
      const double Mvd = M[3][4] + H.svd, Mva = M[3][5];
      const double Mee = fma(g4e, L.a56, H.qee);
      const double Mdd = M[4][4] + H.rdd, Mda = M[4][5], Maa = M[5][5] + H.raa;
      const double ve = vv[2] + vv[4];
      const double mx = fma(L.a51, v4, fma(L.a61, vv[4], vv[0])) + gx;
      const double my = vv[1] - v4 + gy;
      const double mp = fma(L.a23, vv[1], L.a13 * vv[0]) + ve + H.gp;
      const double mv = fma(L.a54, v4, fma(L.a34, ve, fma(L.a24, vv[1], L.a14 * vv[0])) + vv[3]) + H.gv;
      const double me = fma(L.a56, v4, H.ge);
      const double md = fma(L.b3, ve, vv[5]) + H.gd;
      const double ma = fma(dt, vv[3], H.ga);
      const double det = fma(Mdd, Maa, -(Mda * Mda));
      ok = ok && (Mdd > 0.0) && (det > 0.0);
      const double idet = 1.0 / det;
      const double i11 = Maa * idet, i12 = -Mda * idet, i22 = Mdd * idet;
      const double cd[5] = {Mxd, Myd, Mpd, Mvd, 0.0};
      const double ca[5] = {Mxa, Mya, Mpa, Mva, 0.0};
      double K0[5], K1[5];
#pragma unroll
      for (int c = 0; c < 5; c++) {
        K0[c] = -fma(i11, cd[c], i12 * ca[c]);
        K1[c] = -fma(i12, cd[c], i22 * ca[c]);
        ST[i][ST_KG + c] = K0[c];
        ST[i][ST_KG + 5 + c] = K1[c];
      }
      const double k0 = -fma(i11, md, i12 * ma), k1 = -fma(i12, md, i22 * ma);
      ST[i][ST_KG + 10] = k0; ST[i][ST_KG + 11] = k1;
      Pm[0][0] = fma(Mxa, K1[0], fma(Mxd, K0[0], Mxx));
      Pm[0][1] = fma(Mxa, K1[1], fma(Mxd, K0[1], Mxy));
      Pm[0][2] = fma(Mxa, K1[2], fma(Mxd, K0[2], Mxp));
      Pm[0][3] = fma(Mxa, K1[3], fma(Mxd, K0[3], Mxv));
      Pm[0][4] = Mxe;
      Pm[0][5] = 0.0;
      Pm[1][1] = fma(Mya, K1[1], fma(Myd, K0[1], Myy));
      Pm[1][2] = fma(Mya, K1[2], fma(Myd, K0[2], Myp));
      Pm[1][3] = fma(Mya, K1[3], fma(Myd, K0[3], Myv));
      Pm[1][4] = Mye;
      Pm[1][5] = 0.0;
      Pm[2][2] = fma(Mpa, K1[2], fma(Mpd, K0[2], Mpp));
      Pm[2][3] = fma(Mpa, K1[3], fma(Mpd, K0[3], Mpv));
      Pm[2][4] = 0.0;
      Pm[2][5] = 0.0;
      Pm[3][3] = fma(Mva, K1[3], fma(Mvd, K0[3], Mvv));
      Pm[3][4] = Mve;
      Pm[3][5] = 0.0;
      Pm[4][4] = Mee;
      Pm[4][5] = 0.0;
      Pm[5][5] = 0.0;
#pragma unroll
      for (int r = 1; r < 6; r++) {
#pragma unroll
        for (int c = 0; c < r; c++) Pm[r][c] = Pm[c][r];
      }
      pv[0] = fma(Mxa, k1, fma(Mxd, k0, mx));
      pv[1] = fma(Mya, k1, fma(Myd, k0, my));
      pv[2] = fma(Mpa, k1, fma(Mpd, k0, mp));
      pv[3] = fma(Mva, k1, fma(Mvd, k0, mv));
      pv[4] = me;
      pv[5] = 0.0;
      P44 = H.qcc;
      p4 = H.gc;
    }
    ok = resto_soften(0, Pm, pv, P44, p4) && ok;
    gsync();
    return ok;
  }

  // forward sweep of the restoration problem: the soft successor of every constraint block gives the new multipliers
  // y+ (kept in the scratch rows) and the primal step; then, one stage per lane, the slack steps
  //   dn = (mu/n - rho - y+) / (Sigma_n + dw),   dp = (mu/p - rho + y+) / (Sigma_p + dw)
  // the fraction-to-the-boundary ratios over x, n, p and their multipliers, and grad(phi_R)^T d
  __device__ void forward_resto(double dwv) {
    const double dt = PC[LC_DT], eta = eta_r;
    double t[6], w[6];
    {
      const double *dh = rs(0) + RS_DH;
#pragma unroll
      for (int k = 0; k < 6; k++) w[k] = -dh[k];
    }
#pragma unroll 1
    for (int i = 0; i < N; i++) {
      const bool hasu = i < N - 1;
      // soft step of block i: y+ = -(P~ w + p~) over (x, y, psi, v, epsi | cte), then ds = w + D y+
      const double *q = rs(i);
      const double *pt = q + RS_PT;
      const double w5[5] = {w[0], w[1], w[2], w[3], w[5]};
      double y5[5];
      {
        double Pt[5][5];
        int c = 0;
#pragma unroll
        for (int r = 0; r < 5; r++) {
#pragma unroll
          for (int cc = r; cc < 5; cc++) { Pt[r][cc] = pt[c]; Pt[cc][r] = pt[c]; c++; }
        }
#pragma unroll
        for (int r = 0; r < 5; r++) {
          double v = pt[15 + r];
#pragma unroll
          for (int cc = 0; cc < 5; cc++) v = fma(Pt[r][cc], w5[cc], v);
          y5[r] = -v;
        }
      }
      const double yc = -fma(pt[20], w[4], pt[21]);
      const double yp[6] = {y5[0], y5[1], y5[2], y5[3], yc, y5[4]};
#pragma unroll
      for (int k = 0; k < 6; k++) t[k] = fma(q[RS_D + k], yp[k], w[k]);
      if (g0 == 0) {
        double *qq = rs(i);
#pragma unroll
        for (int k = 0; k < 6; k++) qq[RS_YP + k] = yp[k];
      }
      double du0 = 0.0, du1 = 0.0;
      if (hasu) {
        double kg[12];
#pragma unroll
        for (int k = 0; k < 12; k++) kg[k] = ST[i][ST_KG + k];
        du0 = fma(kg[3], t[3], fma(kg[2], t[2], fma(kg[1], t[1], fma(kg[0], t[0], kg[10]))));
        du1 = fma(kg[8], t[3], fma(kg[7], t[2], fma(kg[6], t[1], fma(kg[5], t[0], kg[11]))));
        StageLin L;
        load_lin(i, L);
        const double *dh = rs(i + 1) + RS_DH;
        w[0] = fma(L.a14, t[3], fma(L.a13, t[2], t[0])) - dh[0];
        w[1] = fma(L.a24, t[3], fma(L.a23, t[2], t[1])) - dh[1];
        w[2] = fma(L.b3, du0, fma(L.a34, t[3], t[2])) - dh[2];
        w[3] = fma(dt, du1, t[3]) - dh[3];
        w[4] = fma(L.a56, t[5], fma(L.a54, t[3], fma(L.a51, t[0], -t[1]))) - dh[4];
        w[5] = fma(L.b3, du0, fma(L.a34, t[3], fma(L.a61, t[0], t[2]))) - dh[5];
      }
      if (i % gstep == g0) {
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_DS + k] = t[k];
        ST[i][ST_DU + 0] = du0; ST[i][ST_DU + 1] = du1;
      }
    }
    gsync();
    // ---- step-length ratios and the directional derivative, one stage per lane
    double rmax = 0.0, zn = 1.0, zd = 0.0, gbd = 0.0;
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const bool hasu = i < N - 1;
      const double *b = bk(i);
      const double *q = rs(i);
      double s[6], ds[6];
#pragma unroll
      for (int k = 0; k < 6; k++) { s[k] = ST[i][ST_S + k]; ds[k] = ST[i][ST_DS + k]; }
      const double u0 = hasu ? ST[i][ST_U + 0] : 0.0, u1 = hasu ? ST[i][ST_U + 1] : 0.0;
      const double du0 = hasu ? ST[i][ST_DU + 0] : 0.0, du1 = hasu ? ST[i][ST_DU + 1] : 0.0;
      double acc = 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) acc = fma(eta * dr2_of(b[ST_S + k]) * (s[k] - b[ST_S + k]), ds[k], acc);
      if (hasu) {
        acc = fma(eta * dr2_of(b[ST_U + 0]) * (u0 - b[ST_U + 0]), du0, acc);
        acc = fma(eta * dr2_of(b[ST_U + 1]) * (u1 - b[ST_U + 1]), du1, acc);
      }
      double il[4], iu[4];
      slack_rcp(s[2], s[3], u0, u1, hasu, il, iu);
      const double dx[4] = {ds[2], ds[3], du0, du1};
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (k < 2 || hasu) {
          const double zl = ST[i][ST_ZL + k], zu = ST[i][ST_ZU + k];
          acc = fma(mu_r * (iu[k] - il[k]), dx[k], acc);
          rmax = dmax(rmax, dmax(-dx[k] * il[k], dx[k] * iu[k]));
          const double dzl = fma(fma(-zl, dx[k], mu_r), il[k], -zl);
          const double dzu = fma(fma(zu, dx[k], mu_r), iu[k], -zu);
          if (dzl < 0.0 && (zd == 0.0 || zl * zd < zn * (-dzl))) { zn = zl; zd = -dzl; }
          if (dzu < 0.0 && (zd == 0.0 || zu * zd < zn * (-dzu))) { zn = zu; zd = -dzu; }
        }
      }
#pragma unroll
      for (int k = 0; k < 6; k++) {
        const double n = q[RS_N + k], p = q[RS_P + k], z_n = q[RS_ZN + k], z_p = q[RS_ZP + k], yp = q[RS_YP + k];
        const double sn = z_n / n, sp = z_p / p;
        const double dn = (mu_r / n - K_RESTO_RHO - yp) / (sn + dwv), dp = (mu_r / p - K_RESTO_RHO + yp) / (sp + dwv);
        acc += (K_RESTO_RHO - mu_r / n) * dn + (K_RESTO_RHO - mu_r / p) * dp;
        rmax = dmax(rmax, dmax(-dn / n, -dp / p));
        const double dzn = mu_r / n - z_n - sn * dn, dzp = mu_r / p - z_p - sp * dp;
        if (dzn < 0.0 && (zd == 0.0 || z_n * zd < zn * (-dzn))) { zn = z_n; zd = -dzn; }
        if (dzp < 0.0 && (zd == 0.0 || z_p * zd < zn * (-dzp))) { zn = z_p; zd = -dzp; }
      }
      gbd += acc;
    }
    const int G = PAR ? NS_GROUP : 1;
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) {
      const double on = __shfl_xor_sync(gm, zn, o, G), od = __shfl_xor_sync(gm, zd, o, G);
      const bool take = od > 0.0 && (zd == 0.0 || on * zd < zn * od || (on * zd == zn * od && on < zn));
      if (take) { zn = on; zd = od; }
    }
    rmax = gmax<NS_GROUP>(rmax, gm);
    gbd_r = gsum<NS_GROUP>(gbd, gm);
    alpha_max_r = (rmax > tau_r) ? tau_r / rmax : 1.0;
    alpha_z_r = (zd > 0.0 && tau_r * zn < zd) ? tau_r * zn / zd : 1.0;
  }

  // restoration-problem terms of a trial point x + a dx, n + a dn, p + a dp -- after eval_sweep(a) has left the
  // original problem's values (ft, lt, tht) and the trial residuals (ST_CT, c0t; cur: the iterate's own, a = 0): theta_R = ||c + n - p||_1,
  // rho sum(n + p) + eta/2 ||D_R (x - x_R)||^2, sum of log n + log p
  __device__ void resto_eval_extra(double a, double dwv, bool cur) {
    const double eta = eta_r;
    double th = 0.0, f = 0.0, l = 0.0;
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const bool hasu = i < N - 1;
      const double *b = bk(i);
      const double *q = rs(i);
#pragma unroll
      for (int k = 0; k < 6; k++) {
        const double n = q[RS_N + k], p = q[RS_P + k], yp = q[RS_YP + k];
        const double dn = (mu_r / n - K_RESTO_RHO - yp) / (q[RS_ZN + k] / n + dwv), dp = (mu_r / p - K_RESTO_RHO + yp) / (q[RS_ZP + k] / p + dwv);
        const double nt = fma(a, dn, n), pt = fma(a, dp, p);
        const double ct = cur ? ((i == 0) ? c0[k] : ST[i - 1][ST_CN + k]) : ((i == 0) ? c0t[k] : ST[i - 1][ST_CT + k]);
        th += fabs(ct + nt - pt);
        f = fma(K_RESTO_RHO, nt + pt, f);
        l += log(nt) + log(pt);
        const double xt = fma(a, ST[i][ST_DS + k], ST[i][ST_S + k]) - b[ST_S + k];
        f = fma(0.5 * eta * dr2_of(b[ST_S + k]) * xt, xt, f);
      }
      if (hasu) {
#pragma unroll
        for (int k = 0; k < 2; k++) {
          const double xt = fma(a, ST[i][ST_DU + k], ST[i][ST_U + k]) - b[ST_U + k];
          f = fma(0.5 * eta * dr2_of(b[ST_U + k]) * xt, xt, f);
        }
      }
    }
    r_thR = gsum<NS_GROUP>(th, gm); r_fR = gsum<NS_GROUP>(f, gm); r_lR = gsum<NS_GROUP>(l, gm);
  }

  // second-order-correction residual of the restoration problem:  CS = a (first ? rc : CS) + rc_trial
  __device__ void resto_soc_rhs(bool first, double a, double dwv) {
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const double *q = rs(i);
#pragma unroll
      for (int k = 0; k < 6; k++) {
        const double n = q[RS_N + k], p = q[RS_P + k], yp = q[RS_YP + k];
        const double dn = (mu_r / n - K_RESTO_RHO - yp) / (q[RS_ZN + k] / n + dwv), dp = (mu_r / p - K_RESTO_RHO + yp) / (q[RS_ZP + k] / p + dwv);
        const double nt = fma(a, dn, n), pt = fma(a, dp, p);
        if (i == 0) {
          const double old = first ? (c0[k] + n - p) : cs0[k];
          cs0[k] = a * old + (c0t[k] + nt - pt);
        } else {
          const double old = first ? (ST[i - 1][ST_CN + k] + n - p) : ST[i - 1][ST_CS + k];
          ST[i - 1][ST_CS + k] = a * old + (ST[i - 1][ST_CT + k] + nt - pt);
        }
      }
    }
    // cs0 is uniform per-problem state: every lane needs block 0's value
    if (gstep > 1) {
#pragma unroll
      for (int k = 0; k < 6; k++) cs0[k] = __shfl_sync(gm, cs0[k], 0, PAR ? NS_GROUP : 1);
    }
    gsync();
  }

  // accept the trial point of the restoration problem: x, n, p with a; y with a; every bound multiplier with az and
  // Ipopt's kappa_sigma safeguard; the trial residuals and trig/polynomial values become the iterate's
  __device__ void resto_accept(double a, double az, double dwv) {
    const double zcap = K_KAPPA_SIGMA * mu_r, zfloor = mu_r / K_KAPPA_SIGMA;
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const bool hasu = i < N - 1;
      double *q = rs(i);
      double s[6], ds[6], zl[4], zu[4], il[4], iu[4], iln[4], iun[4];
      double u0 = hasu ? ST[i][ST_U + 0] : 0.0, u1 = hasu ? ST[i][ST_U + 1] : 0.0;
      const double du0 = hasu ? ST[i][ST_DU + 0] : 0.0, du1 = hasu ? ST[i][ST_DU + 1] : 0.0;
#pragma unroll
      for (int k = 0; k < 6; k++) { s[k] = ST[i][ST_S + k]; ds[k] = ST[i][ST_DS + k]; }
#pragma unroll
      for (int k = 0; k < 4; k++) { zl[k] = ST[i][ST_ZL + k]; zu[k] = ST[i][ST_ZU + k]; }
      slack_rcp(s[2], s[3], u0, u1, hasu, il, iu);
      const double dx[4] = {ds[2], ds[3], du0, du1};
#pragma unroll
      for (int k = 0; k < 6; k++) {
        s[k] = fma(a, ds[k], s[k]);
        ST[i][ST_S + k] = s[k];
        const double n = q[RS_N + k], p = q[RS_P + k], z_n = q[RS_ZN + k], z_p = q[RS_ZP + k], yp = q[RS_YP + k];
        const double sn = z_n / n, sp = z_p / p;
        const double dn = (mu_r / n - K_RESTO_RHO - yp) / (sn + dwv), dp = (mu_r / p - K_RESTO_RHO + yp) / (sp + dwv);
        const double dzn = mu_r / n - z_n - sn * dn, dzp = mu_r / p - z_p - sp * dp;
        const double nn = fma(a, dn, n), pn = fma(a, dp, p);
        q[RS_ZN + k] = dmax(dmin(fma(az, dzn, z_n), zcap / nn), zfloor / nn);
        q[RS_ZP + k] = dmax(dmin(fma(az, dzp, z_p), zcap / pn), zfloor / pn);
        q[RS_N + k] = nn; q[RS_P + k] = pn;
        const double y = ST[i][ST_LAM + k];
        ST[i][ST_LAM + k] = fma(a, yp - y, y);
      }
      if (hasu) {
        u0 = fma(a, du0, u0); u1 = fma(a, du1, u1);
        ST[i][ST_U + 0] = u0; ST[i][ST_U + 1] = u1;
      }
      slack_rcp(s[2], s[3], u0, u1, hasu, iln, iun);
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (k < 2 || hasu) {
          const double dzl = fma(fma(-zl[k], dx[k], mu_r), il[k], -zl[k]);
          const double dzu = fma(fma(zu[k], dx[k], mu_r), iu[k], -zu[k]);
          ST[i][ST_ZL + k] = dmax(dmin(fma(az, dzl, zl[k]), zcap * iln[k]), zfloor * iln[k]);
          ST[i][ST_ZU + k] = dmax(dmin(fma(az, dzu, zu[k]), zcap * iun[k]), zfloor * iun[k]);
        }
      }
      if (hasu) {
#pragma unroll
        for (int k = 0; k < 6; k++) ST[i][ST_CN + k] = ST[i][ST_CT + k];
#pragma unroll
        for (int k = 0; k < 8; k++) ST[i][ST_TG + k] = ST[i][ST_TT + k];
      }
    }
#pragma unroll
    for (int k = 0; k < 6; k++) c0[k] = c0t[k];
    gsync();
  }

  // the restoration phase's own line-search state (same tests as the main algorithm's, separate filter)
  struct RestoLS {
    double theta, phi, gbd, pow_gbd, pow_theta;
    int nf, n_resets, succ_rej;
    bool last_rej;
  };
  __device__ static bool r_is_ftype(const RestoLS &R, double a) { return R.gbd < 0.0 && a * R.pow_gbd > R.pow_theta; }
  __device__ static bool r_armijo(const RestoLS &R, double a, double phi_t) {
    return cmp_le(phi_t - R.phi, K_ETA_PHI * a * R.gbd, R.phi);
  }
  // CheckAcceptabilityOfTrialPoint for the restoration problem (theta_min = 1e-4, theta_max = 1e8: its theta_0 is 0)
  __device__ int resto_ls_accept(const RestoLS &R, const double *F, double a, double theta_t, double phi_t) const {
    if (!(theta_t == theta_t) || !(phi_t == phi_t) || isinf(phi_t)) return -1;
    if (theta_t > K_RESTO_THETA_MAX_FACT) return -1;
    bool ok;
    if (a > 0.0 && r_is_ftype(R, a) && R.theta <= 1e-4) {
      ok = r_armijo(R, a, phi_t);
    } else {
      ok = true;
      if (phi_t > R.phi) {
        double basval = 1.0;
        if (fabs(R.phi) > 10.0) basval = log10(fabs(R.phi));
        if (log10(phi_t - R.phi) > K_OBJ_MAX_INC + basval) ok = false;
      }
      ok = ok && (cmp_le(theta_t, (1.0 - K_GAMMA_THETA) * R.theta, R.theta) || cmp_le(phi_t - R.phi, -K_GAMMA_PHI * R.theta, R.phi));
    }
    if (!ok) return 0;
    for (int k = 0; k < R.nf; k++) {
      const double f_t = F[2 * k], f_p = F[2 * k + 1];
      if (!(cmp_le(theta_t, f_t, f_t) || cmp_le(phi_t, f_p, f_p))) return 1;
    }
    return 2;
  }

  __device__ void restoration(const KParams &P) {
    // ---- entry (BacktrackingLineSearch): the current point joins the filter; stop here if it is already acceptable
    // or almost feasible (nothing for a feasibility restoration to do)
    filter_add((1.0 - K_GAMMA_THETA) * ls_theta, ls_phi - K_GAMMA_PHI * ls_theta);
    if (acceptable_now) { status = 4; mode = LM_FINISH; return; }
    if (theta <= 1e-2 * P.tol) { status = 9; mode = LM_FINISH; return; }
    // ---- backup of the outer iterate: x_R, and the multipliers the outer algorithm goes on with
    {
      double *r = scratch + SC_BK_ROWS;
#pragma unroll 1
      for (int i = g0; i < N; i += gstep)
        for (int k = 0; k < ST_KEEP; k++) r[i * ST_KEEP + k] = ST[i][k];
    }
    double c0_R[6];
#pragma unroll
    for (int k = 0; k < 6; k++) c0_R[k] = c0[k];
    gsync();
    // ---- RestoIterateInitializer
    mu_r = fmax(mu, cviol);
    tau_r = fmax(K_TAU_MIN, 1.0 - mu_r);
    double tol_r = P.tol;
    const double theta_R = theta, infpr_R = cviol;
    const double orig_inf_pr_max = fmax(K_RESTO_KAPPA * infpr_R, fmin(P.tol, K_CONSTR_VIOL_TOL));
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      double *q = rs(i);
#pragma unroll
      for (int k = 0; k < 6; k++) {
        const double c = (i == 0) ? c0[k] : ST[i - 1][ST_CN + k];
        const double a = mu_r / (2.0 * K_RESTO_RHO) - 0.5 * c, b = c * mu_r / (2.0 * K_RESTO_RHO);
        const double n = a + sqrt(a * a + b), p = c + n;
        q[RS_N + k] = n; q[RS_P + k] = p; q[RS_ZN + k] = mu_r / n; q[RS_ZP + k] = mu_r / p;
      }
    }
    gsync();   // everybody has read the residuals before the multipliers change
#pragma unroll 1
    for (int i = g0; i < N; i += gstep) {
      const bool hasu = i < N - 1;
#pragma unroll
      for (int k = 0; k < 6; k++) ST[i][ST_LAM + k] = 0.0;
#pragma unroll
      for (int k = 0; k < 4; k++) {
        if (k < 2 || hasu) {
          ST[i][ST_ZL + k] = fmin(K_RESTO_RHO, ST[i][ST_ZL + k]);
          ST[i][ST_ZU + k] = fmin(K_RESTO_RHO, ST[i][ST_ZU + k]);
        }
      }
    }
    gsync();
    RestoLS R;
    R.nf = 0; R.n_resets = 0; R.succ_rej = 0; R.last_rej = false;
    double FR[2 * NFILT];
    double dw_last_r = 0.0;
    int accept_cnt_r = 0;
    bool first = true;
    int rstatus = -1;
    const int nz = 4 * N + 4 * (N - 1) + 12 * N, m = 6 * N;
    for (;;) {
      eta_r = sqrt(mu_r);
      resto_errors();
      const double sd = fmax(K_S_MAX, (r_ysum + r_zsum) / (double)(m + nz)) / K_S_MAX;
      const double sc = fmax(K_S_MAX, r_zsum / (double)nz) / K_S_MAX;
      const double cp0 = nanmax(fabs(r_amax), fabs(r_amin));
      const double E0 = nanmax(r_dinf / sd, nanmax(r_cviol, cp0 / sc));
      // ---- IpRestoConvCheck / IpRestoFilterConvCheck: is this point good enough for the original problem?
      if (!first) {
        const double theta_t = theta, infpr_t = r_infpr;
        bool conv = false;
        if (K_RESTO_KAPPA * theta_R < theta_t) conv = false;
        else if (infpr_t > orig_inf_pr_max) conv = false;
        else {
          const double phi_t = fma(-mu, lsum, fx);
          conv = filter_ok(theta_t, phi_t) && acceptable_to_current(theta_t, phi_t, true);
        }
        if (conv) { rstatus = 0; break; }
        bool solved = E0 <= tol_r && r_dinf <= K_DUAL_INF_TOL && r_cviol <= K_CONSTR_VIOL_TOL && cp0 <= K_COMPL_INF_TOL;
        if (!solved) {
          if (E0 <= K_ACCEPT_TOL && r_cviol <= K_ACCEPT_CONSTR_VIOL_TOL && cp0 <= K_ACCEPT_COMPL_INF_TOL) {
            if (++accept_cnt_r >= K_ACCEPT_ITER) solved = true;
          } else {
            accept_cnt_r = 0;
          }
        }
        if (solved) {
          if (infpr_t <= 1e2 * P.tol) {
            if (tol_r > 1e-1 * P.tol) { tol_r *= 1e-2; accept_cnt_r = 0; }
            else { rstatus = 9; break; }
          } else { rstatus = 5; break; }
        }
        if (!(E0 == E0)) { rstatus = 11; break; }
      }
      if (iter >= P.max_iter) { rstatus = 2; break; }
      // ---- monotone barrier update (not in the first restoration iteration)
      if (!first) {
        for (;;) {
          const double cpm = nanmax(fabs(r_amax - mu_r), fabs(r_amin - mu_r));
          const double Emu = nanmax(r_dinf / sd, nanmax(r_cviol, cpm / sc));
          if (!(Emu <= K_KAPPA_EPS * mu_r)) break;
          const double mu_min = fmin(tol_r, K_COMPL_INF_TOL) / (K_KAPPA_EPS + 1.0);
          const double new_mu = fmax(mu_min, fmin(K_KAPPA_MU * mu_r, mu_r * sqrt(mu_r)));
          if (new_mu == mu_r) break;
          mu_r = new_mu;
          tau_r = fmax(K_TAU_MIN, 1.0 - mu_r);
          R.nf = 0; R.succ_rej = 0; R.last_rej = false;
          eta_r = sqrt(mu_r);
          resto_errors();   // the dual infeasibility depends on eta
        }
      }
      first = false;
      // ---- search direction (inertia correction with its own delta_w history) and filter line search on
      // (theta_R, phi_R), written as one loop around a single copy of each sweep: `need` says which system to solve
      // next -- the Newton system (again with a larger delta_w if the inertia is wrong), the second-order-corrected
      // one, or the uncorrected one again after the corrections failed
      resto_build_lh();
      enum { SOLVE_NONE = 0, SOLVE_NEWTON, SOLVE_SOC, SOLVE_BACK };
      int need = SOLVE_NEWTON, nt = 0, cnt = 0;
      double dwv = 0.0, a = 0.0, a_soc = 0.0, a_test = 0.0, phi_acc = 0.0, th_old = 0.0, alpha_min_r = 0.0;
      bool first_try = true, accepted = false, on_soc = false;
      for (;;) {
        if (need != SOLVE_NONE) {
          resto_rhs(need == SOLVE_SOC, dwv);
          const bool okf = riccati_resto(dwv);
          if (need == SOLVE_NEWTON && !okf) {
            if (first_try) { dwv = (dw_last_r == 0.0) ? K_DW_FIRST : fmax(K_DW_MIN, dw_last_r * K_DW_DEC); first_try = false; }
            else dwv = (dw_last_r == 0.0) ? dwv * K_DW_INC_FIRST : dwv * K_DW_INC;
            if (dwv > K_DW_MAX) { rstatus = 10; break; }
            continue;
          }
          forward_resto(dwv);
          if (need == SOLVE_NEWTON) {
            if (dwv > 0.0) dw_last_r = dwv;
            resto_eval_extra(0.0, dwv, true);   // the current point's restoration terms (eval_sweep's part is fx, lsum, theta)
            R.theta = r_thR;
            R.phi = r_fR - mu_r * (lsum + r_lR);
            R.gbd = gbd_r;
            R.pow_gbd = R.gbd < 0.0 ? pow(-R.gbd, K_S_PHI) : 0.0;
            R.pow_theta = pow(R.theta, K_S_THETA);
            double amin_ = K_GAMMA_THETA;
            if (R.gbd < 0.0) {
              amin_ = fmin(K_GAMMA_THETA, K_GAMMA_PHI * R.theta / (-R.gbd));
              if (R.theta <= 1e-4) amin_ = fmin(amin_, R.pow_theta / R.pow_gbd);
            }
            alpha_min_r = amin_ * K_ALPHA_MIN_FRAC;
            a = alpha_max_r; nt = 0; on_soc = false;
          } else if (need == SOLVE_SOC) {
            a_soc = alpha_max_r; on_soc = true;
          } else {   // the uncorrected direction is back: go on backtracking
            on_soc = false;
            a *= 0.5; nt++;
            if (!(a > alpha_min_r)) break;   // (not `a < alpha_min`: theta_R = 0 gives alpha_min = 0, and a NaN must end the search too)
          }
          need = SOLVE_NONE;
        }
        const double a_eval = on_soc ? a_soc : a;
        eval_sweep(a_eval);
        resto_eval_extra(a_eval, dwv, false);
        const double th_t = r_thR, ph_t = r_fR - mu_r * (lt + r_lR);
        if (!on_soc) a_test = a;
        const int acc = resto_ls_accept(R, FR, a_test, th_t, ph_t);
        if (acc == 2) { accepted = true; phi_acc = ph_t; if (on_soc) a = a_soc; break; }
        if (acc >= 0) R.last_rej = acc == 1;
        if (!on_soc) {
          if (nt == 0 && th_t >= R.theta) {   // second-order correction
            cnt = 0; th_old = th_t;
            resto_soc_rhs(true, a, dwv);
            need = SOLVE_SOC;
          } else {
            a *= 0.5; nt++;
            if (!(a > alpha_min_r)) break;   // (not `a < alpha_min`: theta_R = 0 gives alpha_min = 0, and a NaN must end the search too)
          }
        } else {
          cnt++;
          if (cnt < K_MAX_SOC && th_t <= K_KAPPA_SOC * th_old) {
            th_old = th_t;
            resto_soc_rhs(false, a_soc, dwv);
            need = SOLVE_SOC;
          } else {
            need = SOLVE_BACK;
          }
        }
      }
      if (rstatus >= 0) break;
      if (!accepted) { rstatus = 9; break; }   // no restoration phase inside the restoration phase
      // filter reset heuristic, then the filter update (as in commit_accept)
      {
        const bool add = !r_is_ftype(R, a_test) || !r_armijo(R, a_test, phi_acc);
        if (R.n_resets < K_MAX_FILTER_RESETS) {
          if (R.last_rej) {
            if (R.succ_rej + 1 >= P.filter_reset_trigger) { R.n_resets++; R.nf = 0; R.succ_rej = 0; } else R.succ_rej++;
          } else {
            R.succ_rej = 0;
          }
          R.last_rej = false;
        }
        if (add) {
          const double th = (1.0 - K_GAMMA_THETA) * R.theta, ph = R.phi - K_GAMMA_PHI * R.theta;
          int k = 0;
          for (int j = 0; j < R.nf; j++) {
            const double f_t = FR[2 * j], f_p = FR[2 * j + 1];
            if (!(f_t >= th && f_p >= ph)) { FR[2 * k] = f_t; FR[2 * k + 1] = f_p; k++; }
          }
          if (k < NFILT) { FR[2 * k] = th; FR[2 * k + 1] = ph; k++; }
          R.nf = k;
        }
      }
      resto_accept(a, alpha_z_r, dwv);
      fx = ft; lsum = lt; theta = tht;
      iter++;
    }
    if (rstatus == 0) {
      // ---- back to the original problem (PerformRestoration): the bound multipliers take one primal-dual "step"
      // from x_R to the new point (reset to 1 if that leaves any above bound_mult_reset_threshold), the constraint
      // multipliers are reset to zero (constr_mult_reset_threshold = 0)
      double zn = 1.0, zd = 0.0, zmax = 0.0;
      double dzl[NPASS][4], dzu[NPASS][4];
#pragma unroll
      for (int p = 0; p < NPASS; p++) {
        const int i = g0 + p * gstep;
#pragma unroll
        for (int k = 0; k < 4; k++) { dzl[p][k] = 0.0; dzu[p][k] = 0.0; }
        if (i < N) {
          const bool hasu = i < N - 1;
          const double *b = bk(i);
          const double xn[4] = {ST[i][ST_S + 2], ST[i][ST_S + 3], hasu ? ST[i][ST_U + 0] : 0.0, hasu ? ST[i][ST_U + 1] : 0.0};
          const double xr[4] = {b[ST_S + 2], b[ST_S + 3], b[ST_U + 0], b[ST_U + 1]};
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (k < 2 || hasu) {
              const double zl = b[ST_ZL + k], zu = b[ST_ZU + k];
              const double sRl = xr[k] - PC[LC_LO + k], sNl = xn[k] - PC[LC_LO + k];
              const double sRu = PC[LC_HI + k] - xr[k], sNu = PC[LC_HI + k] - xn[k];
              dzl[p][k] = (zl * (sRl - sNl) + mu) / sRl - zl;
              dzu[p][k] = (zu * (sRu - sNu) + mu) / sRu - zu;
              if (dzl[p][k] < 0.0 && (zd == 0.0 || zl * zd < zn * (-dzl[p][k]))) { zn = zl; zd = -dzl[p][k]; }
              if (dzu[p][k] < 0.0 && (zd == 0.0 || zu * zd < zn * (-dzu[p][k]))) { zn = zu; zd = -dzu[p][k]; }
            }
          }
        }
      }
      const int G = PAR ? NS_GROUP : 1;
#pragma unroll
      for (int o = G / 2; o > 0; o >>= 1) {
        const double on = __shfl_xor_sync(gm, zn, o, G), od = __shfl_xor_sync(gm, zd, o, G);
        const bool take = od > 0.0 && (zd == 0.0 || on * zd < zn * od || (on * zd == zn * od && on < zn));
        if (take) { zn = on; zd = od; }
      }
      const double az = (zd > 0.0 && tau * zn < zd) ? tau * zn / zd : 1.0;
#pragma unroll
      for (int p = 0; p < NPASS; p++) {
        const int i = g0 + p * gstep;
        if (i < N) {
          const bool hasu = i < N - 1;
          const double *b = bk(i);
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (k < 2 || hasu) {
              const double zl = fma(az, dzl[p][k], b[ST_ZL + k]), zu = fma(az, dzu[p][k], b[ST_ZU + k]);
              ST[i][ST_ZL + k] = zl; ST[i][ST_ZU + k] = zu;
              zmax = dmax(zmax, dmax(fabs(zl), fabs(zu)));
            }
          }
        }
      }
      zmax = gmax<NS_GROUP>(zmax, gm);
      if (zmax > K_BOUND_MULT_RESET) {
#pragma unroll 1
        for (int i = g0; i < N; i += gstep) {
          const bool hasu = i < N - 1;
#pragma unroll
          for (int k = 0; k < 4; k++) {
            if (k < 2 || hasu) { ST[i][ST_ZL + k] = 1.0; ST[i][ST_ZU + k] = 1.0; }
          }
        }
      }
      gsync();
      iter++;   // the call itself is an iteration of the outer algorithm
      wd_short = 0; wd_skip = false; in_watchdog = false;
      lh_stale = true;
      // multipliers to zero, optimality errors at the new iterate, then Ipopt's tests and the barrier update
      advance(false, false, true);
      check_and_update_mu(P);
    } else {
      // the restoration failed: the outer algorithm stops with its own iterate
      gsync();
      const double *r = scratch + SC_BK_ROWS;
#pragma unroll 1
      for (int i = g0; i < N; i += gstep)
        for (int k = 0; k < ST_KEEP; k++) ST[i][k] = r[i * ST_KEEP + k];
#pragma unroll
      for (int k = 0; k < 6; k++) c0[k] = c0_R[k];
      gsync();
      status = rstatus; mode = LM_FINISH;
    }
  }

  // ---- one trip of the state machine, in four slots (shared by the lane kernel and the coop kernel) -------
  // slot 1: evaluate a point
  __device__ __forceinline__ void trip_eval() {
    m1 = mode;
    if (m1 == LM_EV0 || m1 == LM_TRIAL || m1 == LM_SOC_TRIAL) {
      const double a = m1 == LM_EV0 ? 0.0 : (m1 == LM_TRIAL ? alpha : alpha_soc);
      eval_sweep(a);
    }
  }
  // the trial point is the new iterate: filter reset heuristic, filter update (FilterLSAcceptor::
  // CheckAcceptabilityOfTrialPoint's tail and UpdateForNextIteration), watchdog counter.  Returns false if a
  // one-problem-per-lane kernel cannot hold the filter entry: nothing has been changed, the problem escalates.
  __device__ __forceinline__ bool commit_accept(const KParams &P, double phi_t) {
    const bool add = !is_ftype(alpha_test) || !armijo(alpha_test, phi_t);
    const bool heur = n_filter_resets < K_MAX_FILTER_RESETS;
    const bool reset = heur && last_rej_filter && succ_filter_rej + 1 >= P.filter_reset_trigger;
    const double th_add = (1.0 - K_GAMMA_THETA) * ls_theta, ph_add = ls_phi - K_GAMMA_PHI * ls_theta;
    if (!FULL && add && !reset && filter_count_after(th_add, ph_add) > NFILT) return false;
    if (heur) {
      if (last_rej_filter) {
        if (reset) { n_filter_resets++; nfilt = 0; succ_filter_rej = 0; } else succ_filter_rej++;
      } else {
        succ_filter_rej = 0;
      }
      last_rej_filter = false;
    }
    if (add) filter_add(th_add, ph_add);
    if (ntrial == 0) wd_short = 0; else wd_short++;
    return true;
  }
  // slot 2: acceptance logic, then the sweep that accepts the step and measures the KKT error
  template <bool WARM = false>
  __device__ __forceinline__ void trip_accept(const KParams &P) {
    bool upd = false, lsq = false, zero = false, err = false;
    if (m1 == LM_EV0) {
      alpha = 0.0; alpha_z = 0.0;
      theta_max = 1e4 * fmax(1.0, tht);
      theta_min = 1e-4 * fmax(1.0, tht);
      upd = true;
    } else if (m1 == LM_LSQ_DONE) {
      lsq = true; err = true;
    } else if (m1 == LM_LSQ_ZERO) {
      zero = true; err = true;
    } else if (m1 == LM_LSFAIL) {
      // A one-problem-per-lane kernel meets this mode only in a record it has just loaded (a resume launch reading a
      // problem that an earlier launch handed over): hand it on.  Without this the lane would idle on it, and a warp
      // holding more than park_lanes such records would never be sparse enough for rule 2 to park them.
      if (FULL) restoration(P); else escalate = true;
    } else if (m1 == LM_TRIAL || m1 == LM_SOC_TRIAL) {
      const double phi_t = fma(-mu, lt, ft);
      // the step size the switching condition and the Armijo test are made with: this trial's, or -- while the
      // watchdog runs -- the one of the step it started with
      if (m1 == LM_TRIAL) alpha_test = (FULL && in_watchdog) ? wd_alpha_test : alpha;
      bool take = false;
      if (FULL && force_accept) {
        // a tiny step (trip_solve): taken untested, the filter and the watchdog counter stay as they are
        force_accept = false;
        take = true;
      } else {
        const int acc = ls_accept(alpha_test, tht, phi_t);
        if (acc == 2) {
          // (no early return here: it would move the reconvergence point of this whole if-chain behind the sweep
          // below, and the lanes of a warp would run it in two or three passes)
          if (commit_accept(P, phi_t)) { if (FULL) in_watchdog = false; take = true; }
          else escalate = true;
        } else {
          if (acc >= 0) last_rej_filter = acc == 1;
          if (FULL && in_watchdog) {
            // BacktrackingLineSearch's watchdog: up to watchdog_trial_iter_max full steps without a test; if none of
            // the points they lead to is acceptable to the point where it started, go back there and backtrack
            if (++wd_trial > K_WATCHDOG_TRIAL_MAX) {
              watchdog_stop();
              alpha = 0.5 * alpha_max; ntrial = 0; wd_skip = true;
              mode = LM_TRIAL;
            } else {
              wd_short = 0;
              take = true;
            }
          } else if (m1 == LM_TRIAL) {
            if (ntrial == 0 && !(FULL && wd_skip) && tht >= ls_theta) {
              // second-order correction (Ipopt max_soc = 4): same matrix, corrected constraint rhs
              soc_cnt = 0;
              theta_soc_old = tht;
              soc_rhs(true, alpha);
              mode = LM_SOC;
            } else {
              alpha *= 0.5;
              ntrial++;
              if (!(alpha > alpha_min)) line_search_failed();
            }
          } else {   // rejected SOC trial
            soc_cnt++;
            if (soc_cnt < K_MAX_SOC && tht <= K_KAPPA_SOC * theta_soc_old) {
              theta_soc_old = tht;
              soc_rhs(false, alpha_soc);
              mode = LM_SOC;
            } else {
              mode = LM_RESOLVE;
            }
          }
        }
      }
      if (take) {
        if (m1 == LM_SOC_TRIAL) alpha = alpha_soc;
        upd = true; err = true;
      }
    }
    // one copy of the sweep for every path: keep the compiler from cloning it per state (a clone run
    // by two or three lanes costs the warp a full pass)
    int flags = (upd ? 1 : 0) | (lsq ? 2 : 0) | (zero ? 4 : 0) | (err ? 8 : 0);
    asm volatile("" : "+r"(flags));
    upd = flags & 1; lsq = flags & 2; zero = flags & 4; err = flags & 8;
    if (flags) {
      advance(upd, lsq, zero);
      if (upd) { fx = ft; lsum = lt; theta = tht; }
      if (m1 == LM_EV0 && !(WARM && P.ws_lam)) {
        mode = LM_LSQ;
      } else if (lsq && !(lsq_lmax <= K_CONSTR_MULT_INIT_MAX)) {
        mode = LM_LSQ_ZERO;
      } else {
        // (a warm start with the caller's lambda goes from the start point straight to the convergence test: the
        // sweep above has measured the errors there with those multipliers)
        if (upd && !(WARM && m1 == LM_EV0)) iter++;
        if (FULL && was_tiny) {
          // the second tiny step in a row with a small dual step asks for a smaller barrier parameter
          if (tiny_last && dy_max < K_TINY_STEP_Y_TOL) tiny_flag = true;
          tiny_last = true; was_tiny = false;
        }
        if (FULL) wd_skip = false;
        check_and_update_mu(P);
      }
    }
  }
  // the line search ran below alpha_min: Ipopt's restoration phase.  One-problem-per-lane kernels hand over.
  __device__ __forceinline__ void line_search_failed() {
    mode = LM_LSFAIL;
    if (!FULL) escalate = true;
  }
  // coop kernels: trips until the problem is finished.  Every iteration costs a handful of trips (one in the common
  // case, a few with inertia correction, second-order corrections or backtracking); a problem that has taken 64 trips
  // per allowed iteration is not making progress and ends as an internal error instead of holding the device.
  template <bool WARM = false>
  __device__ __forceinline__ void run_to_completion(const KParams &P) {
    long long budget = 64LL * (long long)(P.max_iter + 16);
    while (mode != LM_FINISH) {
      trip_eval();
      trip_accept<WARM>(P);
      if (mode == LM_FINISH) break;
      trip_factor();
      trip_solve(P);
      if (--budget < 0) { status = 13; mode = LM_FINISH; }
    }
  }
  // slot 3: factor
  __device__ __forceinline__ void trip_factor() {
    m3 = mode;
    const bool solve = m3 == LM_LSQ || m3 == LM_NEWTON || m3 == LM_SOC || m3 == LM_RESOLVE;
    solve_ok = true;
    if (solve && !escalate) {
      const bool ls = m3 == LM_LSQ;
      const double dwv = ls ? 0.0 : (m3 == LM_NEWTON ? dw : dw_used);
      if (PAR && (lh_stale || ls || (m3 == LM_NEWTON && dw == 0.0))) { build_lh(ls); lh_stale = false; }
      solve_ok = riccati(ls, m3 == LM_SOC, dwv);
    } else {
      m3 = LM_IDLE;
    }
  }
  // slot 4: solve, step lengths, line-search set-up
  __device__ __forceinline__ void trip_solve(const KParams &P) {
    if (m3 == LM_IDLE) return;
    if (m3 == LM_NEWTON && !solve_ok) {
      // Ipopt's inertia correction schedule (delta_w)
      double d = dw;
      if (d == 0.0) d = (dw_last == 0.0) ? K_DW_FIRST : fmax(K_DW_MIN, dw_last * K_DW_DEC);
      else d = (dw_last == 0.0) ? d * K_DW_INC_FIRST : d * K_DW_INC;
      dw = d;
      if (d > K_DW_MAX) { status = 10; mode = LM_FINISH; }
      return;
    }
    forward_and_ratios(m3 == LM_LSQ, m3 == LM_SOC);
    if (m3 == LM_LSQ) {
      dw_used = 0.0;
      mode = LM_LSQ_DONE;
    } else if (m3 == LM_NEWTON) {
      if (!FULL && ((tiny_tol > 0.0 && tiny_screen) || (P.watchdog_trigger > 0 && wd_short >= P.watchdog_trigger))) {
        // a step that may be "tiny", or the watchdog's trigger: nothing of this trip is committed (mode and dw are
        // as they were when it began), the coop kernel repeats it and takes the branch
        escalate = true;
        return;
      }
      if (dw > 0.0) dw_last = dw;
      dw_used = dw;
      alpha_max = alpha_soc;
      bool tiny = false;
      if (FULL) {
        // DetectTinyStep: every component of the step is relatively tiny and the point is (almost) feasible
        tiny = tiny_tol > 0.0 && tiny_all != 0.0 && theta <= 1e-4;
        if (in_watchdog && tiny) { watchdog_stop(); tiny = false; }
      }
      if (!(FULL && in_watchdog)) {   // InitThisLineSearch: reference values of the current iterate
        ls_gbd = gbd_new;
        ls_theta = theta;
        ls_phi = fma(-mu, lsum, fx);
        pow_gbd = ls_gbd < 0.0 ? pow(-ls_gbd, K_S_PHI) : 0.0;
        pow_theta = pow(ls_theta, K_S_THETA);
        double amin_ = K_GAMMA_THETA;
        if (ls_gbd < 0.0) {
          amin_ = fmin(K_GAMMA_THETA, K_GAMMA_PHI * ls_theta / (-ls_gbd));
          if (ls_theta <= theta_min) amin_ = fmin(amin_, pow_theta / pow_gbd);
        }
        alpha_min = amin_ * K_ALPHA_MIN_FRAC;
      }
      if (FULL && P.watchdog_trigger > 0 && !in_watchdog && !tiny && wd_short >= P.watchdog_trigger) watchdog_start();
      alpha = alpha_max;
      ntrial = 0;
      if (FULL && tiny) { force_accept = true; was_tiny = true; }
      else if (FULL) tiny_last = false;
      mode = LM_TRIAL;
    } else if (m3 == LM_SOC) {
      mode = LM_SOC_TRIAL;
    } else {   // LM_RESOLVE: the uncorrected direction is back; continue backtracking
      alpha *= 0.5;
      ntrial++;
      mode = LM_TRIAL;
      if (!(alpha > alpha_min)) line_search_failed();
    }
  }
};

// Which records does launch chain_pos of a chain work on, and where does it park?  A resume launch that would find
// no more than resume_min records does nothing -- the final launch copes with that many at a lower cost than another
// pass of the lane kernel -- so the records stay where they are; every launch replays those decisions from the
// counters of the launches before it (all final: same stream).  No host round trip anywhere in a chain.
struct ChainIO { const double *in; int n; double *out; int *out_count; int *cursor; bool run; };
__device__ __forceinline__ ChainIO chain_resolve(const KParams &P) {
  int slot = 0, buf = 0;
  ChainIO io;
  for (int j = 1;; j++) {
    int n = P.chain_counts[2 * slot];
    if (n > P.ckpt_cap) n = P.ckpt_cap;
    const bool run = j == P.chain_last || n > P.resume_min;
    if (j >= P.chain_pos) {
      io.in = buf ? P.chain_buf1 : P.chain_buf0; io.n = n;
      io.out = buf ? P.chain_buf0 : P.chain_buf1; io.out_count = P.chain_counts + 2 * j; io.cursor = P.chain_counts + 2 * j + 1;
      io.run = run;
      return io;
    }
    if (run) { slot = j; buf ^= 1; }
  }
}

// Persistent grid, one CTA per SM; every lane pulls problems from the global counter until the batch is
// exhausted.  The warps of a CTA start every trip together (the exit vote is a __syncthreads): the loop
// body is ~100 KB of code, and warps at unrelated places in it thrash the instruction cache
// (profiles/r01_v3_*: 3.3 issue slots lost per instruction to "no instruction" with independent one-warp
// CTAs).  Further barriers between the slots of a trip were measured to make no difference (+-2 %).
//
// A warp costs the same per trip whether 32 of its lanes hold a problem or one.  Two rules move problems out
// of warps that would run nearly empty (both at a trip boundary, as flat records, see Lane::save):
//   1. a problem still running after handoff_iter iterations is parked;
//   2. once the queue is empty (a lane of the warp found nothing to fetch), a warp with at most park_lanes
//      problems left parks them all.
// RESUME = true is the same kernel started from the records of the previous launch instead of fresh problems,
// 32 consecutive records to a warp, warps dealt round-robin to the CTAs -- so the survivors of many sparse
// warps run in a few full ones.  The last launch of a chain parks nothing (P.ckpt == NULL).
// The largest CTA the lane kernel is compiled for, one CTA per SM: a register budget of 65536 / 256 a thread
// (profiles/r01_lane_threads_sweep.txt).
enum { LANE_MAX_THREADS = 256 };
// WARM: launches with a warm start (Lane::init); a resume launch may hold a warm problem parked before its first trip
template <int NS, bool RESUME, bool WARM>
__global__ void __launch_bounds__(LANE_MAX_THREADS, 1) mpc_lane_kernel(const KParams P) {
  Lane<NS, false> Z;
  Z.mode = LM_IDLE;
  Z.b = 0;
  Z.g0 = 0; Z.gstep = 1; Z.gm = 0xffffffffu;
  Z.lh_stale = false; Z.no_handoff = false; Z.escalate = false;
  Z.tiny_tol = P.tiny_step_tol;
  Z.scratch = nullptr;
  int n_in = 0, next_in = 0;
  double *park_buf = P.ckpt;
  int *park_count = P.ckpt_count;
  const double *rec_in = nullptr;
  if (RESUME) {
    const ChainIO io = chain_resolve(P);
    if (!io.run) return;
    n_in = io.n; rec_in = io.in; park_buf = io.out; park_count = io.out_count;
    next_in = (int)(((threadIdx.x >> 5) * gridDim.x + blockIdx.x) * 32 + (threadIdx.x & 31));
  }
  for (;;) {
    // ---- slot 0: retire / migrate / fetch
    if (Z.mode == LM_FINISH) { Z.write_outputs(P); Z.mode = LM_IDLE; }
    // two passes over one copy of the park / fetch code: rule 1 and escalation then fetch, rule 2 after the fetch
#pragma unroll 1
    for (int pass = 0; pass < 2; pass++) {
      unsigned live = 0xffffffffu;
      if (pass == 1) live = __ballot_sync(0xffffffffu, Z.mode != LM_DONE);
      const bool esc = pass == 0 && Z.escalate;
      const bool can = park_buf && Z.mode != LM_IDLE && Z.mode != LM_DONE && (!Z.no_handoff || esc);
      // rule 2: a lane is only ever DONE when the queue had nothing left for it
      const bool park = can && (pass == 0 ? (Z.iter >= P.handoff_iter || esc)
                                          : (live != 0xffffffffu && __popc(live) <= P.park_lanes));
      bool parked = false;
      if (park) {
        const int slot = atomicAdd(park_count, 1);
        if (slot < P.ckpt_cap) { Z.save(park_buf + (size_t)slot * Lane<NS, false>::CK_SIZE); Z.mode = pass == 0 ? LM_IDLE : LM_DONE; parked = true; }
        else Z.no_handoff = true;
      }
      if (esc && !parked) {
        // no record slot: the final launch of the chain solves this problem from the start with every branch of the
        // algorithm on board -- same arithmetic, so it walks the same path up to here and then takes the branch
        P.restart_list[atomicAdd(P.restart_count, 1)] = Z.b;
        Z.mode = LM_IDLE;
      }
      if (pass == 0) Z.escalate = false;
      if (pass == 0 && Z.mode == LM_IDLE) {
        Z.no_handoff = false;
        if (RESUME) {
          if (next_in < n_in) { Z.load(rec_in + (size_t)next_in * Lane<NS, false>::CK_SIZE); next_in += (int)(gridDim.x * blockDim.x); }
          else Z.mode = LM_DONE;
        } else {
          const int nb = atomicAdd(P.counter, 1);
          if (nb < P.B) Z.template init<WARM>(P, P.perm ? P.perm[nb] : nb); else Z.mode = LM_DONE;
        }
      }
    }
    if (__syncthreads_and(Z.mode == LM_DONE)) break;
    Z.trip_eval();
    Z.template trip_accept<WARM>(P);
    Z.trip_factor();
    Z.trip_solve(P);
    // progress guard (see run_to_completion): a problem that stops making progress must not hold the whole grid
    if (Z.mode != LM_IDLE && Z.mode != LM_DONE && Z.mode != LM_FINISH && ++Z.trips > 64 * (P.max_iter + 16)) { Z.status = 13; Z.mode = LM_FINISH; }
  }
}

// The same solver with one problem per GROUP of 16 (N <= 16) or 32 lanes and the per-stage rows in shared
// memory: the two sweeps that are parallel over the horizon (point evaluation; step acceptance + KKT
// errors) run one stage per lane with shuffles for the neighbours and butterfly reductions, the two
// recursions (Riccati, forward) run identically in every lane of the group on broadcast shared-memory
// reads.  A trip takes a fraction of the time a lone lane needs, which is what matters when there are
// fewer problems than lanes: single solves (MPC::solve called once per telemetry message), closed-loop
// steps of a few thousand vehicles, and the last long-running problems of a big batch.
template <int NS, bool WARM>
__global__ void __launch_bounds__(128, 2) mpc_coop_kernel(const KParams P) {
  extern __shared__ double coop_smem[];
  const int G = Lane<NS, true>::NS_GROUP;
  const int lane = threadIdx.x & 31;
  Lane<NS, true> Z;
  Z.g0 = lane % G; Z.gstep = G;
  Z.gm = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane - Z.g0));
  Z.ST = reinterpret_cast<double (*)[ST_ROW_SH]>(coop_smem + (size_t)(threadIdx.x / G) * NS * ST_ROW_SH);
  Z.lh_stale = false; Z.no_handoff = false;
  Z.scratch = P.scratch + (size_t)((blockIdx.x * blockDim.x + threadIdx.x) / G) * P.scratch_stride;
  int pass = 0;
  for (;;) {
    int nb = 0;
    if (P.counter) {
      if (Z.g0 == 0) nb = atomicAdd(P.counter, 1);
      nb = __shfl_sync(Z.gm, nb, 0, G);
    } else {   // no work queue (single solves: saves the host a memset): one problem per group, one pass
      nb = pass++ ? P.B : (int)((blockIdx.x * blockDim.x + threadIdx.x) / G);
    }
    if (nb >= P.B) break;
    Z.template init<WARM>(P, nb);
    Z.template run_to_completion<WARM>(P);
    if (Z.g0 == 0) Z.write_outputs(P);
    Z.gsync();
  }
}

// The coop kernel on the problems the lane kernel parked or handed over: each group takes a record, restores the
// state and carries on from the trip where the lane stopped; then the problems that were handed over when no record
// slot was free (restart_list) are solved from the start.
template <int NS, bool WARM>
__global__ void __launch_bounds__(128, 2) mpc_coop_resume_kernel(const KParams P) {
  extern __shared__ double coop_smem[];
  const int G = Lane<NS, true>::NS_GROUP;
  const int lane = threadIdx.x & 31;
  Lane<NS, true> Z;
  Z.g0 = lane % G; Z.gstep = G;
  Z.gm = (G == 32) ? 0xffffffffu : (((1u << G) - 1u) << (lane - Z.g0));
  Z.ST = reinterpret_cast<double (*)[ST_ROW_SH]>(coop_smem + (size_t)(threadIdx.x / G) * NS * ST_ROW_SH);
  Z.no_handoff = true;
  Z.scratch = P.scratch + (size_t)((blockIdx.x * blockDim.x + threadIdx.x) / G) * P.scratch_stride;
  Z.tiny_tol = P.tiny_step_tol;
  int n = 0;
  const double *rec_in = nullptr;
  int *cursor = P.restart_cursor;
  if (P.chain_counts) {
    const ChainIO io = chain_resolve(P);
    n = io.n; rec_in = io.in; cursor = io.cursor;
  }
  int n_restart = *P.restart_count;
  if (n_restart > P.B) n_restart = P.B;
  for (int phase = 0; phase < 2; phase++) {
    if (phase == 0 && !rec_in) continue;
    const int cnt = phase == 0 ? n : n_restart;
    int *cur = phase == 0 ? cursor : P.restart_cursor;
    for (;;) {
      int k = 0;
      if (Z.g0 == 0) k = atomicAdd(cur, 1);
      k = __shfl_sync(Z.gm, k, 0, G);
      if (k >= cnt) break;
      if (phase == 0) Z.load(rec_in + (size_t)k * Lane<NS, true>::CK_SIZE);
      else Z.template init<WARM>(P, P.restart_list[k]);
      Z.template run_to_completion<WARM>(P);
      if (Z.g0 == 0) Z.write_outputs(P);
      Z.gsync();
    }
  }
}

}  // namespace mpcb200
