"""Warm start without a GPU: the oracle's restatement of Ipopt's warm_start_init_point, the CPU shift that the device
shift is checked against, and the argument checks of the C-ABI's warm-start calls."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import nlp_numpy as nn
import oracle_warm as ow
import warm_start_numpy as wsn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _batch(mpc, po, cd, B, seed):
    b = mpc.workloads.batch_perturbed_states(B, seed, cd)
    return b, po.problems_from_arrays(b["state"], b["coeffs"], b["yaw_lo"], b["yaw_hi"])


def _cold(po, cd, probs):
    cfg = po.make_config(cd)
    return [po.solve(cfg, probs[i]) for i in range(len(probs))]


def _kkt_scaled(cd, b, idx, z, lam, zl, zu):
    """Largest scaled stationarity error and constraint violation per problem, from the independent numpy NLP."""
    N = cd["N"]
    state, coeffs = b["state"][idx], b["coeffs"][idx]
    fz = nn.frozen(cd, state)
    g = nn.lagrangian_gradient(cd, fz, state, coeffs, z, lam, zl, zu)
    sd = np.maximum(100.0, (np.abs(lam).sum(axis=1) + zl.sum(axis=1) + zu.sum(axis=1)) / (6 * N + 4 * N + 4 * (N - 1))) / 100.0
    return np.abs(g).max(axis=1) / sd, np.abs(nn.constraints(cd, state, coeffs, z)).max(axis=1)


def test_restart_at_own_solution_stops_at_once(mpc, po, stable_cd):
    """Warm-started at its own converged solution with a small mu_init, the oracle is done within two iterations, at the
    same point, and that point is a KKT point of the NLP as stated independently in tests/nlp_numpy.py.  (The two points
    are both 1e-8 KKT points; they differ by the solution's own conditioning: ~5e-8 in the actuations, up to ~2e-6 in
    the late-stage positions, which the objective barely weighs.)"""
    cd = stable_cd
    b, probs = _batch(mpc, po, cd, 48, 3)
    cold = _cold(po, cd, probs)
    assert all(r["status"] == 1 for r in cold)
    X, L = np.array([r["z"] for r in cold]), np.array([r["lam"] for r in cold])
    ZL, ZU = np.array([r["zl"] for r in cold]), np.array([r["zu"] for r in cold])
    warm = ow.solve_batch_warm(po.make_config(cd, mu_init=1e-9), probs, X, L, ZL, ZU, 8)
    assert [r["status"] for r in warm] == [1] * 48
    assert max(r["iters"] for r in warm) <= 2
    R, R0 = np.array([r["result"] for r in warm]), np.array([r["result"] for r in cold])
    assert np.abs(R[:, :8] - R0[:, :8]).max() < 2e-7
    assert (np.abs(R[:, 8] - R0[:, 8]) / np.abs(R0[:, 8])).max() < 1e-8
    Z = np.array([r["z"] for r in warm])
    assert np.abs(Z - X).max() < 1e-5
    gn, cv = _kkt_scaled(cd, b, np.arange(48), Z, np.array([r["lam"] for r in warm]),
                         np.array([r["zl"] for r in warm]), np.array([r["zu"] for r in warm]))
    assert gn.max() < 1e-4 and np.median(gn) < 5e-6, (gn.max(), np.median(gn))
    assert cv.max() < 2e-7


@pytest.mark.parametrize("mu_init", [0.1, 1e-4])
def test_perturbed_start_converges_to_cold_solution(mpc, po, stable_cd, mu_init):
    """From a perturbed solution (primal point and multipliers), the warm-started oracle reaches the cold-start solution
    on problems whose cold solve converged well (success in at most 15 iterations)."""
    cd = stable_cd
    b, probs = _batch(mpc, po, cd, 64, 11)
    cold = _cold(po, cd, probs)
    good = np.array([r["status"] == 1 and r["iters"] <= 15 for r in cold])
    assert good.mean() > 0.9
    rng = np.random.default_rng(5)
    X = np.array([r["z"] for r in cold])
    X = X + rng.normal(0.0, 0.02, X.shape) * (1.0 + np.abs(X))
    L = np.array([r["lam"] for r in cold]) * rng.uniform(0.5, 1.5, (64, 6 * cd["N"]))
    ZL = np.array([r["zl"] for r in cold]) * rng.uniform(0.5, 1.5, X.shape)
    ZU = np.array([r["zu"] for r in cold]) * rng.uniform(0.5, 1.5, X.shape)
    warm = ow.solve_batch_warm(po.make_config(cd, mu_init=mu_init), probs, X, L, ZL, ZU, 8)
    for i in np.flatnonzero(good):
        assert warm[i]["status"] == 1, (i, warm[i]["status"])
        assert np.abs(warm[i]["result"][:8] - cold[i]["result"][:8]).max() < 1e-6, i
        assert warm[i]["result"][8] == pytest.approx(cold[i]["result"][8], rel=1e-8)
    # the primal point alone (multipliers from the cold-start initialisation) converges too
    primal = ow.solve_batch_warm(po.make_config(cd), probs, X, n_threads=8)
    for i in np.flatnonzero(good):
        assert primal[i]["status"] == 1 and np.abs(primal[i]["result"][:8] - cold[i]["result"][:8]).max() < 1e-6, i


def test_shift_helper_layout(mpc, po, stable_cd):
    """The CPU shift on the layouts of `full` / lambda / zl / zu: on a real solution, stage i of the next start point is
    stage i+1 of the solution in every block (nlp_numpy.split is the reference's layout), the last state stage continues
    the last increment, the last actuation / multiplier repeats, and multipliers of unbounded variables stay 0."""
    cd = stable_cd
    N = cd["N"]
    b, probs = _batch(mpc, po, cd, 4, 2)
    cold = _cold(po, cd, probs)
    # [rows][B], as the device buffers hold them
    x, lam = np.array([r["z"] for r in cold]).T.copy(), np.array([r["lam"] for r in cold]).T.copy()
    zl, zu = np.array([r["zl"] for r in cold]).T.copy(), np.array([r["zu"] for r in cold]).T.copy()
    x0, lam0, zl0, zu0 = wsn.shift(N, x, lam, zl, zu)
    assert x0.shape == x.shape and lam0.shape == lam.shape and zl0.shape == zl.shape
    for a, a0, states in ((x, x0, True), (zl, zl0, False), (zu, zu0, False)):
        blk, blk0 = nn.split(a.T, N), nn.split(a0.T, N)
        for k in range(8):
            assert np.array_equal(blk0[k][:, :-1], blk[k][:, 1:])
            want = 2 * blk[k][:, -1] - blk[k][:, -2] if (states and k < 6) else blk[k][:, -1]
            np.testing.assert_allclose(blk0[k][:, -1], want, rtol=0, atol=1e-12)
    for k in range(6):
        assert np.array_equal(lam0[k * N:k * N + N - 1], lam[k * N + 1:k * N + N])
        assert np.array_equal(lam0[k * N + N - 1], lam[k * N + N - 1])
    xl, xu = nn.var_bounds(cd, b["yaw_lo"], b["yaw_hi"])
    assert (zl0.T[xl < -1e18] == 0).all() and (zu0.T[xu > 1e18] == 0).all()
    assert wsn.shift(N, x)[1:] == (None, None, None)


def test_warm_start_argument_errors_without_device(mpc, stable_cfg):
    """The C-ABI's warm-start calls refuse a NULL handle (MPC_EINVAL); without a device there is no handle at all
    (mpc_create: MPC_ENODEV).  mu_init < 0 and N_per with a warm start are checked on the GPU (tests/test_gpu_warm_start.py)."""
    L = mpc.lib()
    buf = (C.c_double * 64)()
    assert L.mpc_set_warm_start(None, buf, None, None, None, 0.0) == -1
    assert L.mpc_set_warm_start(None, None, None, None, None, -1.0) == -1
    assert L.mpc_warm_start_shift(None, 1, buf, None, None, None, buf, None, None, None, None) == -1
    assert L.mpc_set_warm_start_one(None, 1, 0.0) == -1
    import torch
    if not torch.cuda.is_available():
        h = C.c_void_p()
        assert L.mpc_create(C.byref(stable_cfg), 0, C.byref(h)) == -2 and not h


def test_cpp_header_warm_start_compiles(tmp_path):
    """MPC::setWarmStart of include/mpc_b200.hpp compiles with the header alone (no CUDA headers), as the drop-in needs."""
    src = tmp_path / "w.cpp"
    src.write_text('#include "mpc_b200.hpp"\nvoid f(mpcb200::MPC &m) { m.setWarmStart(true, 1e-4); m.setWarmStart(false); }\n')
    subprocess.run(["g++", "-std=c++11", "-fsyntax-only", "-I", os.path.join(ROOT, "include"), str(src)], check=True)
