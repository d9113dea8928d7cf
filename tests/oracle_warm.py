"""The CPU oracle with Ipopt's warm start (``warm_start_init_point yes``), for the warm-start tests.

oracle/mpc_oracle.c is compiled a second time, into a temporary directory, with its start-point initialisation
replaced by the one of Ipopt's IpWarmStartIterInitializer::SetInitialIterates (Ipopt 3.12 option defaults):
  - the caller's primal point is pushed into the bounds by the formula of the cold start, with
    warm_start_bound_push = warm_start_bound_frac = 1e-3 in place of bound_push = bound_frac = 1e-2;
  - the caller's bound multipliers are taken over to the scaled problem (times the objective factor sf; variables are
    not scaled) and raised to at least warm_start_mult_bound_push = 1e-3; without them, bound_mult_init_val = 1;
  - the caller's lambda is taken over to the scaled problem (times sf / c_scale) instead of the least-squares
    estimate; without it, the least-squares estimate;
  - the initial barrier parameter is cfg.mu_init, as in a cold start.
The NLP scaling stays the one computed at the problem's own start point, so a warm-started solve iterates on the same
scaled problem as a cold one and multipliers convert with the factors the oracle's outputs divide out.  Everything
else -- iteration, line search, restoration phase -- is the oracle's own code: each edit below must match the source
exactly once, so a change of the oracle that touches these places stops the build instead of going unnoticed.
"""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")

EDITS = [
    ("#define BOUND_MULT_RESET_THRESHOLD 1e3\n", """#define BOUND_MULT_RESET_THRESHOLD 1e3
/* warm_start_init_point yes (IpWarmStartIterInitializer, Ipopt 3.12 option defaults) */
#define WS_BOUND_PUSH 1e-3      /* warm_start_bound_push: bound_push of the warm start */
#define WS_BOUND_FRAC 1e-3      /* warm_start_bound_frac: bound_frac of the warm start */
#define WS_MULT_BOUND_PUSH 1e-3 /* warm_start_mult_bound_push: the given bound multipliers are raised to this */
/* the start point and multipliers of the UNSCALED problem, layouts of orc_result's z / lambda / zl / zu;
 * x is required, lambda / zl / zu may be NULL (cold-start initialisation of that part) */
typedef struct orc_warm { const double *x, *lambda, *zl, *zu; } orc_warm;
int orc_ipm_solve_warm(const orc_nlp *nlp, const orc_config *cfg, const double *xi_in, const double *xl_in,
                       const double *xu_in, const double *gl_in, const double *gu_in, const orc_warm *warm,
                       double *x_out, double *lam_out, double *zl_out, double *zu_out, orc_ipm_stats *out);
int orc_solve_warm(const orc_config *cfg, const orc_problem *prob, const orc_warm *warm, orc_result *out);
"""),
    ("""                  double *lam_out, double *zl_out, double *zu_out, orc_ipm_stats *out) {
""", """                  double *lam_out, double *zl_out, double *zu_out, orc_ipm_stats *out) {
  return orc_ipm_solve_warm(nlp, cfg, xi_in, xl_in, xu_in, gl_in, gu_in, NULL, x_out, lam_out, zl_out, zu_out, out);
}

int orc_ipm_solve_warm(const orc_nlp *nlp, const orc_config *cfg, const double *xi_in, const double *xl_in,
                       const double *xu_in, const double *gl_in, const double *gu_in, const orc_warm *warm,
                       double *x_out, double *lam_out, double *zl_out, double *zu_out, orc_ipm_stats *out) {
"""),
    ("""  for (int i = 0; i < n; i++) {
    double v = xi[i];
""", """  const double push = warm ? WS_BOUND_PUSH : KAPPA_1, frac = warm ? WS_BOUND_FRAC : KAPPA_2;
  for (int i = 0; i < n; i++) {
    double v = warm ? warm->x[i] : xi[i];
"""),
    ("""      double pl = fmin(KAPPA_1 * fmax(1.0, fabs(s->xl[i])), KAPPA_2 * span);
      double pu = fmin(KAPPA_1 * fmax(1.0, fabs(s->xu[i])), KAPPA_2 * span);
""", """      double pl = fmin(push * fmax(1.0, fabs(s->xl[i])), frac * span);
      double pu = fmin(push * fmax(1.0, fabs(s->xu[i])), frac * span);
"""),
    ("      double pl = KAPPA_1 * fmax(1.0, fabs(s->xl[i]));\n", "      double pl = push * fmax(1.0, fabs(s->xl[i]));\n"),
    ("      double pu = KAPPA_1 * fmax(1.0, fabs(s->xu[i]));\n", "      double pu = push * fmax(1.0, fabs(s->xu[i]));\n"),
    ("""    s->zu[i] = s->has_u[i] ? 1.0 : 0.0;
  }
""", """    s->zu[i] = s->has_u[i] ? 1.0 : 0.0;
    if (warm && warm->zl && s->has_l[i]) s->zl[i] = fmax(warm->zl[i] * s->sf, WS_MULT_BOUND_PUSH);
    if (warm && warm->zu && s->has_u[i]) s->zu[i] = fmax(warm->zu[i] * s->sf, WS_MULT_BOUND_PUSH);
  }
"""),
    ("""  /* least-squares multiplier estimate: [[I, J^T],[J, 0]] [r; lam] = [-(grad - zl + zu); 0] */
  {
""", """  /* least-squares multiplier estimate: [[I, J^T],[J, 0]] [r; lam] = [-(grad - zl + zu); 0];
   * a warm start with the caller's lambda takes that over to the scaled problem instead */
  if (warm && warm->lambda) {
    for (int j = 0; j < m; j++) s->lam[j] = warm->lambda[j] * s->sf / s->cs[j];
  } else {
"""),
    ("""int orc_solve(const orc_config *cfg, const orc_problem *prob, orc_result *out) {
""", """int orc_solve(const orc_config *cfg, const orc_problem *prob, orc_result *out) {
  return orc_solve_warm(cfg, prob, NULL, out);
}

int orc_solve_warm(const orc_config *cfg, const orc_problem *prob, const orc_warm *warm, orc_result *out) {
"""),
    ("  int rc = orc_ipm_solve(&nlp, cfg, xi, xl, xu, gl, gu, out->z,",
     "  int rc = orc_ipm_solve_warm(&nlp, cfg, xi, xl, xu, gl, gu, warm, out->z,"),
    ("""  const orc_problem *p;
  orc_result *out;
""", """  const orc_problem *p;
  const orc_warm *warm;
  orc_result *out;
"""),
    ("    orc_solve(j->cfg, &j->p[b], r);\n", "    orc_solve_warm(j->cfg, &j->p[b], j->warm ? &j->warm[b] : NULL, r);\n"),
    ("int orc_solve_batch_compact(", """/* orc_solve_batch from per-problem warm starts warm[B] */
int orc_solve_batch_warm(const orc_config *cfg, const orc_problem *p, const orc_warm *warm, int B,
                         orc_result *out, int nt) {
  job_t j;
  memset(&j, 0, sizeof(j));
  j.cfg = cfg; j.p = p; j.warm = warm; j.out = out; j.B = B;
  return run_jobs(&j, B, nt);
}

int orc_solve_batch_compact("""),
]


class OrcWarm(C.Structure):
    _fields_ = [("x", C.POINTER(C.c_double)), ("lam", C.POINTER(C.c_double)),
                ("zl", C.POINTER(C.c_double)), ("zu", C.POINTER(C.c_double))]


def warm_source():
    """oracle/mpc_oracle.c with the warm-start edits applied."""
    with open(os.path.join(ORACLE, "mpc_oracle.c")) as f:
        src = f.read()
    for old, new in EDITS:
        n = src.count(old)
        if n != 1:
            raise RuntimeError("warm-start edit matches oracle/mpc_oracle.c %d times (expected once): %r" % (n, old[:60]))
        src = src.replace(old, new)
    return src


_lib = None


def lib():
    global _lib
    if _lib is None:
        d = tempfile.mkdtemp(prefix="mpc_oracle_warm_")
        atexit.register(shutil.rmtree, d, True)
        src, so = os.path.join(d, "mpc_oracle_warm.c"), os.path.join(d, "libmpc_oracle_warm.so")
        with open(src, "w") as f:
            f.write(warm_source())
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-std=c99", "-Wall", "-Wextra", "-fno-fast-math", "-I", ORACLE,
                               "-shared", "-o", so, src, "-lm", "-lpthread"])
        from oracle import pyoracle as po
        L = C.CDLL(so)
        L.orc_solve_batch_warm.argtypes = [C.POINTER(po.OrcConfig), C.POINTER(po.OrcProblem), C.POINTER(OrcWarm), C.c_int,
                                           C.POINTER(po.OrcResult), C.c_int]
        _lib = L
    return _lib


def solve_batch_warm(cfg, probs, x, lam=None, zl=None, zu=None, n_threads=1):
    """Warm-started oracle solves (initial barrier parameter cfg.mu_init): cfg / probs as for pyoracle.solve_batch;
    x [B][8N-2], lam [B][6N], zl / zu [B][8N-2] (each of lam / zl / zu may be None), unscaled, in the layouts of
    pyoracle.solve's z / lam / zl / zu.  -> list of B dicts with status, iters, obj, result, z, lam, zl, zu and the
    branch counters of pyoracle.solve (n_resto, n_watchdog, n_tiny, n_filter_reset, n_filter_max)."""
    from oracle import pyoracle as po
    B = len(probs)
    n, m = 8 * cfg.N - 2, 6 * cfg.N
    arrs = [None if a is None else np.ascontiguousarray(np.asarray(a, dtype=np.float64).reshape(B, -1))
            for a in (x, lam, zl, zu)]
    assert arrs[0].shape[1] == n and (arrs[1] is None or arrs[1].shape[1] == m)
    dp = lambda a: a.ctypes.data_as(C.POINTER(C.c_double))
    warm = (OrcWarm * B)()
    for b in range(B):
        warm[b].x, warm[b].lam, warm[b].zl, warm[b].zu = [None if a is None else dp(a[b]) for a in arrs]
    out = (po.OrcResult * B)()
    lib().orc_solve_batch_warm(C.byref(cfg), probs, warm, B, out, n_threads)
    return [{"status": r.status, "iters": r.iters, "obj": r.obj, "result": np.array(r.result[:9]),
             "z": np.array(r.z[:n]), "lam": np.array(r.lam[:m]), "zl": np.array(r.zl[:n]), "zu": np.array(r.zu[:n]),
             "n_resto": r.n_resto, "n_watchdog": r.n_watchdog, "n_tiny": r.n_tiny, "n_filter_reset": r.n_filter_reset,
             "n_filter_max": r.n_filter_max}
            for r in out]
