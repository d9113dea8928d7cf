"""CPU restatement of mpc_solution_sensitivity: the derivative of a solution of the reference NLP with respect to the
initial state, from one dense solve of the KKT system (Ipopt's sIPOPT).  It shares no code with the kernel: the Hessian
of the Lagrangian and the Jacobian are the oracle's (oracle/mpc_oracle.c, orc_eval_hess / orc_eval_jac), the barrier
term is built here from the bounds the oracle states, and the system is solved by LU, not by a Riccati recursion.

    [ W + Sigma   J^T ] [dz]   [ 0   ]
    [ J           0   ] [dl] = [ e_k ]      e_k: 1 in the initial-condition row of state component k (row k*N)

W: Hessian of f + lambda^T g of the UNSCALED problem (the sign convention grad f + J^T lambda - zl + zu = 0 of the
dual outputs), Sigma = zl / (z - lo) + zu / (hi - z) with the bounds relaxed as the solver relaxes them
(lo - min(1e-4, 1e-8 max(1, |lo|))): the outputs are clamped to the unrelaxed bounds, so at an active bound the slack
to the relaxed one is at least the relaxation."""
import numpy as np
import scipy.linalg

BIG = 1.0e19
RESULT_ROWS = 9


def relaxed_bounds(xl, xu):
    """Ipopt's bound_relax_factor 1e-8 capped at constr_viol_tol 1e-4; infinite where the NLP has no bound."""
    lo = np.where(xl > -BIG, xl - np.minimum(1e-4, 1e-8 * np.maximum(1.0, np.abs(xl))), -np.inf)
    hi = np.where(xu < BIG, xu + np.minimum(1e-4, 1e-8 * np.maximum(1.0, np.abs(xu))), np.inf)
    return lo, hi


def kkt_matrix(po, cfg, p, z, lam, zl, zu):
    """The dense KKT matrix [[W + Sigma, J^T], [J, 0]] at (z, lam, zl, zu), the size n of its primal block, and Sigma."""
    n, m = 8 * cfg.N - 2, 6 * cfg.N
    W = po.eval_hess(cfg, p, z, 1.0, lam)
    J = po.eval_jac(cfg, p, z)
    xl, xu = po.bounds(cfg, p)[:2]
    lo, hi = relaxed_bounds(xl, xu)
    with np.errstate(divide="ignore", invalid="ignore"):
        sig = np.where(np.isfinite(lo), zl / (z - lo), 0.0) + np.where(np.isfinite(hi), zu / (hi - z), 0.0)
    K = np.zeros((n + m, n + m))
    K[:n, :n] = W + np.diag(sig)
    K[:n, n:] = J.T
    K[n:, :n] = J
    return K, n, sig


def reduced_hessian_pd(K, n):
    """Whether W + Sigma is positive definite on the null space of J (the inertia Ipopt asks of the factorisation)."""
    Z = scipy.linalg.null_space(K[n:, :n])
    R = Z.T @ K[:n, :n] @ Z
    try:
        np.linalg.cholesky(0.5 * (R + R.T))
        return True
    except np.linalg.LinAlgError:
        return False


def sensitivity(po, cfg, p, z, lam, zl, zu):
    """-> dict: dfull [6][8N-2] (slice k = dz / d state_k, layout of `full`), dresult [6][9] (layout of `result`; the
    cost row is grad f^T dz), dlam [6][6N], pd (reduced Hessian positive definite), sigma_max (largest barrier term)."""
    N = cfg.N
    K, n, sig = kkt_matrix(po, cfg, p, z, lam, zl, zu)
    rhs = np.zeros((K.shape[0], 6))
    for k in range(6):
        rhs[n + k * N, k] = 1.0
    sol = np.linalg.solve(K, rhs).T
    dz, dl = sol[:, :n], sol[:, n:]
    grad = po.eval_grad(cfg, p, z)
    rows = [k * N + 1 for k in range(6)] + [6 * N, 7 * N - 1]
    dres = np.concatenate([dz[:, rows], (dz @ grad)[:, None]], axis=1)
    return {"dfull": dz, "dresult": dres, "dlam": dl, "pd": reduced_hessian_pd(K, n), "sigma_max": sig.max()}


def batch(po, cfg, probs, full, lam, zl, zu, idx=None):
    """sensitivity() for problems idx (default all) of a batch; arrays [B][...] -> dfull [B][6][8N-2], dresult [B][6][9],
    pd [B]."""
    idx = range(len(probs)) if idx is None else idx
    out = [sensitivity(po, cfg, probs[i], full[i], lam[i], zl[i], zu[i]) for i in idx]
    return (np.array([o["dfull"] for o in out]), np.array([o["dresult"] for o in out]),
            np.array([o["pd"] for o in out]))


def strictly_complementary(cfg, po, p, z, zl, zu, margin=1e-3):
    """Every bound has an unscaled slack >= margin or a multiplier >= margin: the active set does not change under a
    small perturbation, so finite differences of solves measure the same derivative."""
    xl, xu = po.bounds(cfg, p)[:2]
    fl, fu = xl > -BIG, xu < BIG
    okl = (z - xl >= margin) | (zl >= margin)
    oku = (xu - z >= margin) | (zu >= margin)
    return bool(np.all(okl[fl]) and np.all(oku[fu]))


def active_bound(cfg, po, p, z, tol=1e-6):
    xl, xu = po.bounds(cfg, p)[:2]
    return bool(np.any((xl > -BIG) & (z - xl < tol)) or np.any((xu < BIG) & (xu - z < tol)))


def branch_distance(cd, state):
    """Distance of each problem's state from the thresholds of FG_eval's frozen branches (MPC.cpp:72,79,87,89): the
    cte and epsi panic levels, the steer table of the speed target, v = 0."""
    d = np.abs(np.abs(state[:, 4]) - cd["cte_panic"])
    d = np.minimum(d, np.abs(np.abs(state[:, 5]) - cd["epsi_panic"]))
    for s in cd["steers"]:
        d = np.minimum(d, np.abs(np.abs(state[:, 2]) - s))
    return np.minimum(d, np.abs(state[:, 3]))


def finite_differences(po, cfg, probs_fn, state, h):
    """Central differences of oracle solves: probs_fn(state) -> problems; -> dfull [B][6][8N-2], dresult [B][6][9],
    and whether every perturbed solve succeeded [B]."""
    B = state.shape[0]
    N = cfg.N
    n = 8 * N - 2
    dfull, dres, ok = np.zeros((B, 6, n)), np.zeros((B, 6, RESULT_ROWS)), np.ones(B, dtype=bool)
    for k in range(6):
        sols = []
        for sgn in (1.0, -1.0):
            st = state.copy()
            st[:, k] += sgn * h
            probs = probs_fn(st)
            r = [po.solve(cfg, probs[i]) for i in range(B)]
            ok &= np.array([x["status"] == 1 for x in r])
            sols.append((np.array([x["z"] for x in r]), np.array([x["result"] for x in r])))
        dfull[:, k] = (sols[0][0] - sols[1][0]) / (2 * h)
        dres[:, k] = (sols[0][1] - sols[1][1]) / (2 * h)
    return dfull, dres, ok
