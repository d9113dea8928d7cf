// mpc_sensitivity.cuh -- parametric sensitivity (Ipopt's sIPOPT) of solutions of the batched solve with respect to
// the initial state, one problem per thread, after the solve.
//
// The state enters the NLP only through the initial-condition rows g_{kN}(z) = z_{kN}, gl = gu = state_k
// (MPC.cpp:261-281).  At a solution (z, lambda, zl, zu) the derivative of z with respect to state_k solves
//     [ W + Sigma   J^T ] [dz]   [ 0  ]
//     [ J           0   ] [dl] = [ e_k ]
// with W the Hessian of the Lagrangian of the unscaled NLP and Sigma = zl / (z - lo) + zu / (hi - z) on the bounds
// relaxed as the solver relaxes them (Lane::init, PC[LC_LO]).  That is the Newton system of the solver with a zero
// right-hand side except the initial-condition residual, so the gains of Lane::riccati at the solution (with lambda,
// zl, zu in the scaled problem: times sf; the gains do not change under that uniform scaling) give dz by the forward
// recursion alone, without feed-forward terms:
//     ds_0 = e_k,   du_i = K_i [ds_i; du_{i-1}],   ds_{i+1} = A_i ds_i + B_i du_i.
// The six parameter columns run through one forward pass together.  Lane is reused unchanged: init for the
// per-problem constants (objective factor, frozen branches of FG_eval, relaxed bounds), the loader below instead of
// a start point, riccati(ls = false, soc = false, dw = 0).  No existing kernel changes.
//
// The instantiation is Lane<NS, true, false> (rows behind a pointer, one problem per thread), which no solver kernel
// uses, with the pointer aimed at a thread-private array.  Lane<NS, false>, the lane kernel's own, would work the same,
// but a second kernel calling its riccati / init changes the compiler's inlining decisions inside mpc_lane_kernel
// (its SASS differed in 16 instantiations); separate instantiations leave every existing kernel as it was.
#pragma once
#include "../../include/mpc_b200.h"
#include "mpc_lane_kernel.cuh"

namespace mpcb200 {

template <int NS> using SensLane = Lane<NS, true, false>;

// the solution a sensitivity is taken at, and the outputs (mpc_solution_sensitivity)
struct SensArgs {
  const double *full, *lam, *zl, *zu;   // [8N-2][B], [6N][B], [8N-2][B] x2: layouts of `full` and of the dual outputs
  const int *status;                    // [B] or NULL
  double *dresult, *dfull;              // [6][9][B], [6][8N-2][B] or NULL
};

// The rows of the solution: iterate, multipliers of the scaled problem, trig/polynomial values.  The constraint
// residuals (ST_CN) only enter the feed-forward terms k0, k1 of the Riccati sweep, which the sensitivity does not use:
// they are set to zero.  Unlike warm_init, no bound push: the point is taken as it is, so Sigma is the solution's.
template <int NS>
__device__ void sens_load(SensLane<NS> &Z, const KParams &P, const SensArgs &A) {
  const size_t B = (size_t)P.B;
  const int Nf = P.Nmax, b = Z.b;
  const double sf = Z.PC[LC_SF];
  // rows of the reference's layout (MPC.cpp:189-196) holding psi, v, delta, a of stage i
  const int zrow[4] = {2 * Nf, 3 * Nf, 6 * Nf, 7 * Nf - 1};
#pragma unroll 1
  for (int i = 0; i < Z.N; i++) {
    const bool hasu = i < Z.N - 1;
    double s[6], tg[8], F[6];
#pragma unroll
    for (int k = 0; k < 6; k++) s[k] = A.full[(size_t)(k * Nf + i) * B + b];
    const double u0 = hasu ? A.full[(size_t)(6 * Nf + i) * B + b] : 0.0;
    const double u1 = hasu ? A.full[(size_t)(7 * Nf - 1 + i) * B + b] : 0.0;
    Z.point_eval(s, u0, u1, tg, F);
#pragma unroll
    for (int k = 0; k < 6; k++) {
      Z.ST[i][ST_S + k] = s[k];
      Z.ST[i][ST_LAM + k] = A.lam[(size_t)(k * Nf + i) * B + b] * sf;
      Z.ST[i][ST_CN + k] = 0.0;
    }
    Z.ST[i][ST_U + 0] = u0; Z.ST[i][ST_U + 1] = u1;
#pragma unroll
    for (int k = 0; k < 8; k++) Z.ST[i][ST_TG + k] = tg[k];
#pragma unroll
    for (int k = 0; k < 4; k++) {
      const bool valid = k < 2 || hasu;
      const size_t at = (size_t)(zrow[k] + i) * B + b;
      Z.ST[i][ST_ZL + k] = valid ? A.zl[at] * sf : 0.0;
      Z.ST[i][ST_ZU + k] = valid ? A.zu[at] * sf : 0.0;
    }
  }
}

// Forward recursion of the six parameter columns (forward_and_ratios' stage algebra with the feed-forward terms and
// residuals zero), writing dfull and the rows of dresult; the cost row is grad f(z)^T dz of the unscaled objective,
// accumulated here (not taken from lambda, so that the envelope identity d cost / d state_k = -lambda_k stays a check).
template <int NS>
__device__ void sens_forward(SensLane<NS> &Z, const KParams &P, const SensArgs &A) {
  const size_t B = (size_t)P.B;
  const int Nf = P.Nmax, nx = 8 * Nf - 2, b = Z.b, N = Z.N;
  const double dt = Z.PC[LC_DT], cw = Z.PC[LC_CW], wd2 = Z.PC[LC_WD2], wv2 = Z.PC[LC_WV2];
  double t[6][6], dp[6], acc[6];
#pragma unroll
  for (int c = 0; c < 6; c++) {
#pragma unroll
    for (int k = 0; k < 6; k++) t[c][k] = k == c ? 1.0 : 0.0;
    dp[c] = 0.0; acc[c] = 0.0;
  }
  double dprev = 0.0;
#pragma unroll 1
  for (int i = 0; i < N; i++) {
    const bool hasu = i < N - 1;
    const double v = Z.ST[i][ST_S + 3], s4 = Z.ST[i][ST_S + 4], s5 = Z.ST[i][ST_S + 5], u0 = Z.ST[i][ST_U + 0];
    const double un = Z.ST[i + 1 < N ? i + 1 : i][ST_U + 0];
    double kg[10], tg[8];
#pragma unroll
    for (int k = 0; k < 10; k++) kg[k] = Z.ST[i][ST_KG + k];
#pragma unroll
    for (int k = 0; k < 8; k++) tg[k] = Z.ST[i][ST_TG + k];
    StageLin L;
    Z.lin_at(tg, v, u0, L);
    const double gv = fma(Z.nv2(i), v, wv2 * (v - Z.vref(i))), gc = Z.wc2(i) * s4, ge = Z.we2(i) * s5;
    double gd = wd2 * u0;
    if (i >= 1) gd = fma(cw, u0 - dprev, gd);
    if (i <= N - 3) gd = fma(-cw, un - u0, gd);
#pragma unroll
    for (int c = 0; c < 6; c++) {
      double *dr = A.dresult + (size_t)c * 9 * B + b;
      double *df = A.dfull ? A.dfull + (size_t)c * nx * B + b : nullptr;
      if (df) {
#pragma unroll
        for (int k = 0; k < 6; k++) df[(size_t)(k * Nf + i) * B] = t[c][k];
      }
      if (i == 1) {
#pragma unroll
        for (int k = 0; k < 6; k++) dr[(size_t)k * B] = t[c][k];
      }
      acc[c] = fma(ge, t[c][5], fma(gc, t[c][4], fma(gv, t[c][3], acc[c])));
      if (hasu) {
        const double du0 = fma(kg[4], dp[c], fma(kg[3], t[c][3], fma(kg[2], t[c][2], fma(kg[1], t[c][1], kg[0] * t[c][0]))));
        const double du1 = fma(kg[9], dp[c], fma(kg[8], t[c][3], fma(kg[7], t[c][2], fma(kg[6], t[c][1], kg[5] * t[c][0]))));
        if (df) { df[(size_t)(6 * Nf + i) * B] = du0; df[(size_t)(7 * Nf - 1 + i) * B] = du1; }
        if (i == 0) { dr[6 * B] = du0; dr[7 * B] = du1; }
        acc[c] = fma(gd, du0, acc[c]);
        double tn[6];
        tn[0] = fma(L.a14, t[c][3], fma(L.a13, t[c][2], t[c][0]));
        tn[1] = fma(L.a24, t[c][3], fma(L.a23, t[c][2], t[c][1]));
        tn[2] = fma(L.b3, du0, fma(L.a34, t[c][3], t[c][2]));
        tn[3] = fma(dt, du1, t[c][3]);
        tn[4] = fma(L.a56, t[c][5], fma(L.a54, t[c][3], fma(L.a51, t[c][0], -t[c][1])));
        tn[5] = fma(L.b3, du0, fma(L.a34, t[c][3], fma(L.a61, t[c][0], t[c][2])));
#pragma unroll
        for (int k = 0; k < 6; k++) t[c][k] = tn[k];
        dp[c] = du0;
      }
    }
    dprev = u0;
  }
#pragma unroll
  for (int c = 0; c < 6; c++) A.dresult[(size_t)(c * 9 + 8) * B + b] = acc[c] / Z.PC[LC_SF];
}

// one problem per thread; a problem whose status is not a solution, or whose reduced Hessian is not positive definite
// at the point (a control pivot of the Riccati sweep is not), gets NaN in every output
template <int NS>
__global__ void __launch_bounds__(128) mpc_sensitivity_kernel(const KParams P, const SensArgs A) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= P.B) return;
  alignas(16) double rows[NS][ST_ROW];
  SensLane<NS> Z;
  Z.ST = rows;
  Z.g0 = 0; Z.gstep = 1; Z.gm = 0xffffffffu;
  Z.init(P, b);
  bool ok = !A.status || A.status[b] == MPC_STATUS_SUCCESS || A.status[b] == MPC_STATUS_STOP_AT_ACCEPTABLE_POINT;
  if (ok) {
    sens_load(Z, P, A);
    ok = Z.riccati(false, false, 0.0);
  }
  if (ok) { sens_forward(Z, P, A); return; }
  const size_t B = (size_t)P.B;
  const int nx = 8 * P.Nmax - 2;
  for (int r = 0; r < 6 * 9; r++) A.dresult[(size_t)r * B + b] = NAN;
  if (A.dfull)
    for (int r = 0; r < 6 * nx; r++) A.dfull[(size_t)r * B + b] = NAN;
}

}  // namespace mpcb200
