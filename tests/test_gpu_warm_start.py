"""Warm-started solves on the GPU: parity with the warm-started oracle, the shift kernel against its CPU restatement,
bit-identical results across kernels and entry points, restarts at the solution, argument errors, and switching the
warm start off."""
import json

import numpy as np
import pytest

import oracle_warm as ow
import warm_start_numpy as wsn

pytestmark = pytest.mark.gpu
ABS_TOL, REL_TOL = 1e-4, 1e-6
LANE, COOP = 2, 3


@pytest.fixture(scope="module")
def torch_dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch, torch.device("cuda:0")


def _up(torch, dev, a):
    return torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).to(dev)


def _solve(S, torch, dev, b, state=None):
    """One mpc_solve_batch on device copies of the batch; -> numpy outputs ([B, ...]) and the device solution arrays
    ([rows][B]) that a warm start / the shift take."""
    B, N = b["state"].shape[0], S.cfg.N
    st = _up(torch, dev, b["state"] if state is None else state)
    co, yl, yh = _up(torch, dev, b["coeffs"]), _up(torch, dev, b["yaw_lo"]), _up(torch, dev, b["yaw_hi"])
    f64 = lambda r: torch.zeros(r, B, dtype=torch.float64, device=dev)
    res, tx, ty, full = f64(9), f64(N), f64(N), f64(8 * N - 2)
    lam, zl, zu = f64(6 * N), f64(8 * N - 2), f64(8 * N - 2)
    status, iters = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
    S.set_dual_outputs(lam, zl, zu)
    S.solve_batch_device(B, st, co, yl, yh, res, tx, ty, full, status, iters)
    torch.cuda.synchronize()
    S.set_dual_outputs(None, None, None)
    T = lambda t: t.cpu().numpy().T.copy()
    return {"result": T(res), "traj_x": T(tx), "traj_y": T(ty), "full": T(full), "status": status.cpu().numpy(),
            "iters": iters.cpu().numpy(), "dev": (full, lam, zl, zu)}


def _next_step(b, sol, seed):
    """One control step later in the same frame: each problem's stage-1 state with a small seeded perturbation."""
    rng = np.random.default_rng(seed)
    s1 = sol["result"][:, :6].copy()
    B = s1.shape[0]
    s1[:, 4] += rng.normal(0.0, 0.02, B)
    s1[:, 5] += rng.normal(0.0, 0.005, B)
    s1[:, 3] += rng.normal(0.0, 0.1, B)
    return s1


def _shifted_start(S, torch, sol):
    full, lam, zl, zu = sol["dev"]
    B = full.shape[1]
    out = [torch.zeros_like(a) for a in (full, lam, zl, zu)]
    S.warm_start_shift(B, full, out[0], lam, out[1], zl, out[2], zu, out[3])
    torch.cuda.synchronize()
    return out


@pytest.mark.parametrize("seed,B,kind", [(0, 4096, LANE), (7, 1000, COOP), (9, 1, COOP)])
def test_shifted_warm_start_vs_oracle(mpc, po, stable_cfg, stable_cd, torch_dev, seed, B, kind):
    """Warm-started GPU solves against warm-started oracle solves from the same start point (the shifted previous
    solution, mu_init 1e-4): statuses, actuations and trajectory 1e-4, cost 1e-6 relative, iterations {0, +1}."""
    torch, dev = torch_dev
    b = mpc.workloads.batch_perturbed_states(B, seed, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    S.set_kernel(kind)
    sol = _solve(S, torch, dev, b)
    start = _shifted_start(S, torch, sol)
    s1 = _next_step(b, sol, seed)
    S.set_warm_start(*start, mu_init=1e-4)
    g = _solve(S, torch, dev, b, state=s1)
    S.close()
    x0, lam0, zl0, zu0 = [a.cpu().numpy().T.copy() for a in start]
    probs = po.problems_from_arrays(s1, b["coeffs"], b["yaw_lo"], b["yaw_hi"])
    c = ow.solve_batch_warm(po.make_config(stable_cd, mu_init=1e-4), probs, x0, lam0, zl0, zu0, 16)
    cst = np.array([r["status"] for r in c])
    ok = cst == 1
    assert ok.mean() > 0.99
    assert np.array_equal(g["status"][ok], cst[ok])
    cres = np.array([r["result"] for r in c])
    d = np.abs(g["result"] - cres)[ok]
    assert d[:, :8].max() < ABS_TOL and (d[:, 8] / np.abs(cres[ok, 8])).max() < REL_TOL
    N = stable_cd["N"]
    cz = np.array([r["z"] for r in c])
    assert np.abs(g["traj_x"] - cz[:, :N])[ok].max() < ABS_TOL and np.abs(g["traj_y"] - cz[:, N:2 * N])[ok].max() < ABS_TOL
    di = g["iters"].astype(int)[ok] - np.array([r["iters"] for r in c])[ok]
    assert di.min() >= 0 and di.max() <= 1, np.unique(di, return_counts=True)


def test_shift_kernel_equals_cpu_shift(mpc, stable_cfg, stable_cd, torch_dev):
    torch, dev = torch_dev
    b = mpc.workloads.batch_perturbed_states(3000, 4, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    sol = _solve(S, torch, dev, b)
    start = _shifted_start(S, torch, sol)
    want = wsn.shift(stable_cd["N"], *[a.cpu().numpy() for a in sol["dev"]])
    for got, w in zip(start, want):
        assert np.array_equal(got.cpu().numpy(), w)
    # primal only: the multiplier outputs are untouched
    x0 = torch.zeros_like(start[0])
    S.warm_start_shift(3000, sol["dev"][0], x0)
    torch.cuda.synchronize()
    assert np.array_equal(x0.cpu().numpy(), want[0])
    S.close()


def test_lane_chain_and_coop_kernel_bit_identical_warm(mpc, stable_cfg, stable_cd, torch_dev):
    """A warm-started batch large enough for the lane kernel's tail handling: lane chain and coop kernel agree bit for bit."""
    torch, dev = torch_dev
    B = 16384
    b = mpc.workloads.batch_perturbed_states(B, 5, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    sol = _solve(S, torch, dev, b)
    start = _shifted_start(S, torch, sol)
    s1 = _next_step(b, sol, 5)
    out = {}
    for kind in (LANE, COOP):
        S.set_kernel(kind)
        for mu in (0.1, 1e-6):
            S.set_warm_start(*start, mu_init=mu)
            out[kind, mu] = _solve(S, torch, dev, b, state=s1)
    S.close()
    for mu in (0.1, 1e-6):
        a, c = out[LANE, mu], out[COOP, mu]
        for k in ("result", "full", "traj_x", "traj_y", "status", "iters"):
            assert np.array_equal(a[k], c[k]), (mu, k)
        assert (a["status"] == 1).mean() > 0.99


def test_restart_at_solution(mpc, stable_cfg, stable_cd, torch_dev):
    """Warm-started at its own solution with a small mu_init, a solve returns the cold result with at most two
    iterations on >= 99 % of the problems (both are 1e-8 KKT points: they agree to the solution's conditioning)."""
    torch, dev = torch_dev
    B = 16384
    b = mpc.workloads.batch_perturbed_states(B, 0, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    cold = _solve(S, torch, dev, b)
    S.set_warm_start(*cold["dev"], mu_init=1e-9)
    w = _solve(S, torch, dev, b)
    S.close()
    ok = (cold["status"] == 1) & (w["status"] == 1)
    assert ok.mean() > 0.99
    assert (w["iters"] <= 2).mean() >= 0.99, np.bincount(w["iters"])
    assert np.abs(w["result"][ok, :8] - cold["result"][ok, :8]).max() < 1e-6
    assert np.median(np.abs(w["result"][ok, :8] - cold["result"][ok, :8]).max(axis=1)) < 1e-8
    assert (np.abs(w["result"][ok, 8] - cold["result"][ok, 8]) / np.abs(cold["result"][ok, 8])).max() < 1e-8


def test_warm_start_argument_errors(mpc, stable_cfg, stable_cd, torch_dev):
    torch, dev = torch_dev
    B, N = 64, stable_cfg.N
    b = mpc.workloads.batch_perturbed_states(B, 1, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    x0 = torch.zeros(8 * N - 2, B, dtype=torch.float64, device=dev)
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):
        S.set_warm_start(x0, mu_init=-1.0)
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):
        S.set_warm_start_one(True, mu_init=float("nan"))
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):      # an output without its input
        S.warm_start_shift(B, x0, torch.zeros_like(x0), zl0=torch.zeros_like(x0))
    S.set_warm_start(x0)
    Np = np.full(B, N, dtype=np.int32)
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):
        S.solve_batch_host(b["state"], b["coeffs"], b["yaw_lo"], b["yaw_hi"], N_per=Np)
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):
        st, co, yl, yh = (_up(torch, dev, b[k]) for k in ("state", "coeffs", "yaw_lo", "yaw_hi"))
        res = torch.zeros(9, B, dtype=torch.float64, device=dev)
        S.solve_batch_device(B, st, co, yl, yh, res, N_per=torch.from_numpy(Np).to(dev))
    S.set_warm_start(None)
    S.solve_batch_host(b["state"], b["coeffs"], b["yaw_lo"], b["yaw_hi"], N_per=Np)   # fine again
    S.close()
    M = mpc.MultiSolver(stable_cfg, [0, 0])
    M.set_warm_start(1, torch.zeros(8 * N - 2, B // 2, dtype=torch.float64, device=dev))
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):
        M.solve_batch_host(b["state"], b["coeffs"], b["yaw_lo"], b["yaw_hi"], N_per=Np)
    M.close()


def test_switching_off_restores_cold_bits(mpc, stable_cfg, stable_cd, torch_dev):
    torch, dev = torch_dev
    for kind, B in ((LANE, 12000), (COOP, 700)):
        b = mpc.workloads.batch_perturbed_states(B, 13, stable_cd)
        S = mpc.Solver(stable_cfg, 0)
        S.set_kernel(kind)
        cold = _solve(S, torch, dev, b)
        S.set_warm_start(*_shifted_start(S, torch, cold), mu_init=1e-4)
        warm = _solve(S, torch, dev, b)
        assert not np.array_equal(warm["iters"], cold["iters"])
        S.set_warm_start(None, *cold["dev"][1:], mu_init=1e-4)   # x0 NULL: off, whatever else is passed
        again = _solve(S, torch, dev, b)
        S.close()
        for k in ("result", "full", "traj_x", "traj_y", "status", "iters"):
            assert np.array_equal(again[k], cold[k]), (kind, k)


def test_host_and_multi_entry_points_same_bits(mpc, stable_cfg, stable_cd, torch_dev):
    """mpc_solve_batch_host and mpc_solve_batch_multi (two handles on one device, each bound to its shard's start point)
    give the bits of mpc_solve_batch with the same warm start."""
    torch, dev = torch_dev
    B = 12288
    b = mpc.workloads.batch_perturbed_states(B, 17, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    cold = _solve(S, torch, dev, b)
    start = _shifted_start(S, torch, cold)
    s1 = _next_step(b, cold, 17)
    S.set_warm_start(*start, mu_init=1e-2)
    d = _solve(S, torch, dev, b, state=s1)
    h = S.solve_batch_host(s1, b["coeffs"], b["yaw_lo"], b["yaw_hi"], want_full=True)
    S.close()
    M = mpc.MultiSolver(stable_cfg, [0, 0])
    cuts = [0, B // 2, B]
    for g in range(2):
        M.set_warm_start(g, *[a[:, cuts[g]:cuts[g + 1]].contiguous() for a in start], mu_init=1e-2)
    m = M.solve_batch_host(s1, b["coeffs"], b["yaw_lo"], b["yaw_hi"], want_full=True)
    M.close()
    for o in (h, m):
        for k in ("result", "full", "traj_x", "traj_y", "status", "iters"):
            assert np.array_equal(o[k], d[k]), k
    assert (d["status"] == 1).mean() > 0.99


def test_solve_one_warm_start_follows_cold_solutions(mpc, stable_cfg, stable_cd, torch_dev):
    """mpc_set_warm_start_one (MPC::setWarmStart of the C++ header): a sequence of single solves, each one control step
    after the previous in the same frame, gives the cold solutions with fewer iterations in total."""
    b = mpc.workloads.batch_perturbed_states(4, 21, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    W = mpc.Solver(stable_cfg, 0)
    W.set_warm_start_one(True, mu_init=1e-4)
    it_cold = it_warm = 0
    for i in range(4):
        state = b["state"][i]
        for step in range(12):
            c = S.solve_one(state, b["coeffs"][i], b["yaw_lo"][i], b["yaw_hi"][i])
            w = W.solve_one(state, b["coeffs"][i], b["yaw_lo"][i], b["yaw_hi"][i])
            assert c["status"] == w["status"] == 1
            assert np.abs(w["result"][:8] - c["result"][:8]).max() < ABS_TOL
            assert w["result"][8] == pytest.approx(c["result"][8], rel=REL_TOL)
            it_cold += c["iters"]; it_warm += w["iters"]
            state = c["result"][:6].copy()
        W.set_config(stable_cfg)   # another vehicle: the next solve starts cold
    S.close(); W.close()
    assert it_warm < it_cold, (it_warm, it_cold)
