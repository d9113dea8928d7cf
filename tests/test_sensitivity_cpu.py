"""The CPU reference of the solution sensitivity (tests/sensitivity_numpy.py) pinned without a GPU: against central
finite differences of oracle solves, and against two identities of the reference NLP that hold exactly -- the state
enters only through the initial-condition rows, and cte / epsi of stage 0 reach no later stage but the next cte."""
import numpy as np
import pytest

import sensitivity_numpy as sn

H = 1e-5
TOL = 1e-10


def _solved(mpc, po, cd, B, seed):
    """B problems of the perturbed-state workload at horizon cd["N"], solved by the oracle at tol 1e-10."""
    b = mpc.workloads.batch_perturbed_states(B, seed, cd)
    cfg = po.make_config(cd, tol=TOL)
    mk = lambda st: po.problems_from_arrays(st, b["coeffs"], b["yaw_lo"], b["yaw_hi"])
    probs = mk(b["state"])
    r = [po.solve(cfg, probs[i]) for i in range(B)]
    sol = {k: np.array([x[k] for x in r]) for k in ("z", "lam", "zl", "zu", "status", "result")}
    return b, cfg, mk, probs, sol


@pytest.mark.parametrize("N", [10, 33])
def test_reference_matches_finite_differences(mpc, po, stable_cd, N):
    """Central differences (h = 1e-5) of tol-1e-10 oracle solves agree with the reference to 1e-4 max(1, |S|) on every
    row of `full` and of `result`, on the problems where the derivative exists and the solves measure it: strictly
    complementary with margin 1e-3, and at least 10 h from every frozen-branch threshold."""
    cd = dict(stable_cd, N=N)
    b, cfg, mk, probs, sol = _solved(mpc, po, cd, 24, 11)
    ok = sol["status"] == 1
    ok &= sn.branch_distance(cd, b["state"]) >= 10 * H
    ok &= np.array([sn.strictly_complementary(cfg, po, probs[i], sol["z"][i], sol["zl"][i], sol["zu"][i])
                    for i in range(len(probs))])
    idx = np.flatnonzero(ok)
    assert len(idx) >= 12, len(idx)
    dfull, dres, pd = sn.batch(po, cfg, probs, sol["z"], sol["lam"], sol["zl"], sol["zu"], idx)
    assert pd.all()
    fd_full, fd_res, fd_ok = sn.finite_differences(po, cfg, lambda st: _mk_sub(mk, b, idx, st), b["state"][idx], H)
    assert fd_ok.all()
    err_full = np.abs(fd_full - dfull) / np.maximum(1.0, np.abs(dfull))
    err_res = np.abs(fd_res - dres) / np.maximum(1.0, np.abs(dres))
    assert err_full.max() < 1e-4, err_full.max()
    assert err_res.max() < 1e-4, err_res.max()


def _mk_sub(mk, b, idx, st):
    """problems idx of the batch with their states replaced by st"""
    full_state = b["state"].copy()
    full_state[idx] = st
    probs = mk(full_state)
    return [probs[i] for i in idx]


@pytest.mark.parametrize("N", [10, 33])
def test_reference_cte_epsi_structure(mpc, po, stable_cd, N):
    """d full / d cte0 is e_{4N}; d full / d epsi0 is e_{5N} plus cos(epsi0) v0 dt in the cte_1 row; both to
    1e-12 max|S| (the dense solve's rounding)."""
    cd = dict(stable_cd, N=N)
    b, cfg, mk, probs, sol = _solved(mpc, po, cd, 12, 5)
    assert (sol["status"] == 1).all()
    dfull, dres, pd = sn.batch(po, cfg, probs, sol["z"], sol["lam"], sol["zl"], sol["zu"])
    assert pd.all()
    n = 8 * N - 2
    for i in range(len(probs)):
        want_c = np.zeros(n)
        want_c[4 * N] = 1.0
        want_e = np.zeros(n)
        want_e[5 * N] = 1.0
        want_e[4 * N + 1] = np.cos(b["state"][i, 5]) * b["state"][i, 3] * cd["dt"]
        for k, want in ((4, want_c), (5, want_e)):
            assert np.abs(dfull[i, k] - want).max() <= 1e-12 * np.abs(dfull[i, k]).max()


@pytest.mark.parametrize("N", [10, 33])
def test_reference_envelope_identity(mpc, po, stable_cd, N):
    """d cost / d state_k = -lambda_{kN} (grad f + J^T lambda - zl + zu = 0 and J dz = e_k), up to the barrier term
    (zl - zu)^T dz and the solve's dual tolerance: to 1e-6 max(1, |lambda|)."""
    cd = dict(stable_cd, N=N)
    b, cfg, mk, probs, sol = _solved(mpc, po, cd, 12, 6)
    assert (sol["status"] == 1).all()
    dfull, dres, pd = sn.batch(po, cfg, probs, sol["z"], sol["lam"], sol["zl"], sol["zu"])
    lam0 = sol["lam"][:, [k * N for k in range(6)]]
    err = np.abs(dres[:, :, 8] + lam0) / np.maximum(1.0, np.abs(lam0))
    assert err.max() < 1e-6, err.max()
