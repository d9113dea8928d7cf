"""Solution sensitivities on the GPU (mpc_solution_sensitivity): parity with the dense CPU restatement
(tests/sensitivity_numpy.py) on identical inputs, finite differences of GPU solves, the exact cte / epsi structure and
the envelope identity, NaN for problems that are not solutions, bit identity and the argument checks."""
import json

import numpy as np
import pytest

import sensitivity_numpy as sn

pytestmark = pytest.mark.gpu
LANE, COOP = 2, 3
PARITY = 1e-6        # per problem, relative to max(1, max |S_cpu|), where every barrier term Sigma is <= SIGMA_WELL
SIGMA_WELL = 1e10
PARITY_STIFF = 1e-3  # the same where some Sigma exceeds 1e10 (see _assert_parity)
H = 1e-5


@pytest.fixture(scope="module")
def torch_dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch, torch.device("cuda:0")


def _up(torch, dev, a):
    return torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).to(dev)


def _cfgs(mpc, po, refdata, **over):
    """(product config, oracle config dict) of config-stable with JSON keys overridden."""
    js = dict(refdata["configs"]["stable"], **over)
    return mpc.config_from_json_text(json.dumps(js)), po.load_config_dict(js)


def _solve(S, torch, dev, b, weights=None, dt_per=None, state=None):
    """mpc_solve_batch with dual outputs; -> dict of the device arrays a sensitivity call takes, and numpy copies."""
    B, N = b["state"].shape[0], S.cfg.N
    d = {"state": _up(torch, dev, b["state"] if state is None else state), "coeffs": _up(torch, dev, b["coeffs"]),
         "yaw_lo": _up(torch, dev, b["yaw_lo"]), "yaw_hi": _up(torch, dev, b["yaw_hi"]),
         "weights": None if weights is None else _up(torch, dev, weights),
         "dt_per": None if dt_per is None else _up(torch, dev, dt_per)}
    f64 = lambda r: torch.zeros(r, B, dtype=torch.float64, device=dev)
    res, full, lam, zl, zu = f64(9), f64(8 * N - 2), f64(6 * N), f64(8 * N - 2), f64(8 * N - 2)
    status, iters = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
    S.set_dual_outputs(lam, zl, zu)
    S.solve_batch_device(B, d["state"], d["coeffs"], d["yaw_lo"], d["yaw_hi"], res, None, None, full, status, iters,
                         weights=d["weights"], dt_per=d["dt_per"])
    torch.cuda.synchronize()
    S.set_dual_outputs(None, None, None)
    d.update(full=full, lam=lam, zl=zl, zu=zu, status=status, result=res)
    T = lambda t: t.cpu().numpy().T.copy()
    d["np"] = {"full": T(full), "lam": T(lam), "zl": T(zl), "zu": T(zu), "status": status.cpu().numpy(),
               "result": T(res), "iters": iters.cpu().numpy()}
    return d


def _sens(S, torch, dev, d, with_full=True, with_status=True, B=None):
    """mpc_solution_sensitivity on the solve's arrays -> dresult [B][6][9], dfull [B][6][8N-2] (numpy, or None)."""
    B = d["state"].shape[1] if B is None else B
    nx = 8 * S.cfg.N - 2
    dres = torch.full((6, 9, B), -7.0, dtype=torch.float64, device=dev)
    dfull = torch.full((6, nx, B), -7.0, dtype=torch.float64, device=dev) if with_full else None
    S.solution_sensitivity(B, d["state"], d["coeffs"], d["yaw_lo"], d["yaw_hi"], d["full"], d["lam"], d["zl"], d["zu"],
                           dres, dfull, status=d["status"] if with_status else None, weights=d["weights"],
                           dt_per=d["dt_per"])
    torch.cuda.synchronize()
    return (dres.cpu().numpy().transpose(2, 0, 1).copy(),
            None if dfull is None else dfull.cpu().numpy().transpose(2, 0, 1).copy())


def _cpu(po, cd, b, sol, idx, weights=None, dt_per=None, state=None):
    """The CPU reference on the GPU's own solution, problem by problem (per-problem weights / dt as that problem's
    config) -> dresult [n][6][9], dfull [n][6][8N-2], pd [n], largest Sigma [n]."""
    st = b["state"] if state is None else state
    probs = po.problems_from_arrays(st, b["coeffs"], b["yaw_lo"], b["yaw_hi"])
    base = po.make_config(cd)
    out = []
    for i in idx:
        cfg = base
        if weights is not None or dt_per is not None:
            over = {}
            if dt_per is not None:
                over["dt"] = float(dt_per[i])
            cfg = po.make_config(dict(cd, weights=list(weights[i]) if weights is not None else cd["weights"], **over))
        out.append(sn.sensitivity(po, cfg, probs[i], sol["full"][i], sol["lam"][i], sol["zl"][i], sol["zu"][i]))
    return (np.array([o["dresult"] for o in out]), np.array([o["dfull"] for o in out]), np.array([o["pd"] for o in out]),
            np.array([o["sigma_max"] for o in out]))


def _assert_parity(S, torch, dev, po, cd, b, d, idx=None, **kw):
    """GPU against CPU on the GPU's own solution: 1e-6 max(1, max|S_cpu|) per problem on dresult and dfull, where every
    barrier term Sigma = z / slack is at most 1e10 (the conditioning expected from the solver's tolerances).  A bound held
    by a multiplier of ~1e7 at a slack of ~1e-8 (the relaxation of the bound) gives Sigma of 1e15 and a KKT matrix of
    condition ~1e23; there a Riccati recursion and a dense LU, both stable, were measured to agree to 2e-4 (N = 32), while
    the CPU reference agrees with itself under equilibration and refinement to 1e-8: the difference is the system's
    conditioning, not a defect, so those problems are held to 1e-3."""
    sol = d["np"]
    ok = (sol["status"] == 1) | (sol["status"] == 4)
    idx = np.flatnonzero(ok) if idx is None else idx
    assert len(idx) > 0.8 * len(ok)
    gres, gfull = _sens(S, torch, dev, d)
    cres, cfull, pd, sig = _cpu(po, cd, b, sol, idx, **kw)
    assert pd.all()
    scale = np.maximum(1.0, np.abs(cfull).max(axis=(1, 2)))
    err = np.maximum(np.abs(gres[idx] - cres).max(axis=(1, 2)), np.abs(gfull[idx] - cfull).max(axis=(1, 2))) / scale
    well = sig <= SIGMA_WELL
    print("parity: %d problems, %d with Sigma <= 1e10: worst %.3g; %d stiffer (max Sigma %.3g): worst %.3g" % (
        len(idx), well.sum(), err[well].max(initial=0.0), (~well).sum(), sig.max(), err[~well].max(initial=0.0)))
    assert well.any()
    assert err[well].max(initial=0.0) < PARITY, (err[well].max(), idx[well][np.argmax(err[well])])
    assert err[~well].max(initial=0.0) < PARITY_STIFF
    return err.max()


@pytest.mark.parametrize("B,kind", [(4096, LANE), (1000, COOP)], ids=["lane-4096", "coop-1000"])
def test_parity_stable_batch(mpc, po, stable_cfg, stable_cd, torch_dev, B, kind):
    torch, dev = torch_dev
    b = mpc.workloads.batch_perturbed_states(B, 0, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    S.set_kernel(kind)
    d = _solve(S, torch, dev, b)
    _assert_parity(S, torch, dev, po, stable_cd, b, d)
    S.close()


@pytest.mark.parametrize("N", [2, 3, 10, 11, 20, 21, 32, 33, 40, 64])
def test_parity_horizon_grid(mpc, po, refdata, torch_dev, N):
    """Every horizon instantiation NS = 10, 20, 32, 64, with N = NS and N < NS."""
    torch, dev = torch_dev
    cfg, cd = _cfgs(mpc, po, refdata, N=N)
    B = 64 if N >= 40 else 256
    b = mpc.workloads.batch_perturbed_states(B, 100 + N, cd)
    S = mpc.Solver(cfg, 0)
    d = _solve(S, torch, dev, b)
    _assert_parity(S, torch, dev, po, cd, b, d)
    S.close()


def test_parity_per_problem_weights_and_dt(mpc, po, stable_cfg, stable_cd, torch_dev):
    torch, dev = torch_dev
    B = 256
    b = mpc.workloads.batch_perturbed_states(B, 21, stable_cd)
    rng = np.random.default_rng(21)
    w = np.asarray(stable_cd["weights"])[None, :] * rng.uniform(0.3, 3.0, (B, 12))
    dt = rng.uniform(0.05, 0.15, B)
    S = mpc.Solver(stable_cfg, 0)
    d = _solve(S, torch, dev, b, weights=w, dt_per=dt)
    _assert_parity(S, torch, dev, po, stable_cd, b, d, weights=w, dt_per=dt)
    S.close()


def test_parity_warm_started_solution(mpc, po, stable_cfg, stable_cd, torch_dev):
    """A solution of a warm-started solve (one control step later, from the shifted previous solution)."""
    torch, dev = torch_dev
    B = 1024
    b = mpc.workloads.batch_perturbed_states(B, 31, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    d0 = _solve(S, torch, dev, b)
    start = [torch.zeros_like(d0[k]) for k in ("full", "lam", "zl", "zu")]
    S.warm_start_shift(B, d0["full"], start[0], d0["lam"], start[1], d0["zl"], start[2], d0["zu"], start[3])
    rng = np.random.default_rng(31)
    s1 = d0["np"]["result"][:, :6].copy()
    s1[:, 3] += rng.normal(0.0, 0.1, B)
    S.set_warm_start(*start, mu_init=1e-4)
    d = _solve(S, torch, dev, b, state=s1)
    S.set_warm_start(None)
    assert d["np"]["iters"].mean() < d0["np"]["iters"].mean()   # the warm start was taken
    _assert_parity(S, torch, dev, po, stable_cd, b, d, state=s1)
    S.close()


def test_parity_active_steering_bound(mpc, po, refdata, torch_dev):
    """max_steering tightened until at least 20 % of the problems hold the steering bound at stage 0: Sigma of ~1e8 and
    more on those rows."""
    torch, dev = torch_dev
    cfg, cd = _cfgs(mpc, po, refdata, **{"max steering": np.degrees(0.05)})
    B = 512
    b = mpc.workloads.batch_perturbed_states(B, 41, cd)
    S = mpc.Solver(cfg, 0)
    d = _solve(S, torch, dev, b)
    N = cd["N"]
    active = np.abs(np.abs(d["np"]["full"][:, 6 * N]) - cd["max_steering"]) < 1e-6
    assert active.mean() >= 0.2, active.mean()
    _assert_parity(S, torch, dev, po, cd, b, d)
    S.close()


def test_finite_differences_of_gpu_solves(mpc, po, refdata, torch_dev):
    """Central differences (h = 1e-5) of tol-1e-10 GPU solves against the sensitivity, to 1e-4 max(1, |S|), on the
    problems that are strictly complementary with margin 1e-3 and 10 h from every frozen-branch threshold."""
    torch, dev = torch_dev
    cfg, cd = _cfgs(mpc, po, refdata)
    cfg.tol = 1e-10
    B = 256
    b = mpc.workloads.batch_perturbed_states(B, 51, cd)
    S = mpc.Solver(cfg, 0)
    d = _solve(S, torch, dev, b)
    sol = d["np"]
    ocfg = po.make_config(cd)
    probs = po.problems_from_arrays(b["state"], b["coeffs"], b["yaw_lo"], b["yaw_hi"])
    qual = (sol["status"] == 1) & (sn.branch_distance(cd, b["state"]) >= 10 * H)
    qual &= np.array([sn.strictly_complementary(ocfg, po, probs[i], sol["full"][i], sol["zl"][i], sol["zu"][i])
                      for i in range(B)])
    assert qual.mean() >= 0.5, qual.mean()
    assert any(sn.active_bound(ocfg, po, probs[i], sol["full"][i]) for i in np.flatnonzero(qual))
    gres, gfull = _sens(S, torch, dev, d)
    fd_full, fd_res = np.zeros_like(gfull), np.zeros_like(gres)
    ok = np.ones(B, dtype=bool)
    for k in range(6):
        outs = []
        for sgn in (1.0, -1.0):
            st = b["state"].copy()
            st[:, k] += sgn * H
            dk = _solve(S, torch, dev, b, state=st)
            ok &= dk["np"]["status"] == 1
            outs.append(dk["np"])
        fd_full[:, k] = (outs[0]["full"] - outs[1]["full"]) / (2 * H)
        fd_res[:, k] = (outs[0]["result"] - outs[1]["result"]) / (2 * H)
    S.close()
    q = qual & ok
    assert q.mean() >= 0.5
    err = max((np.abs(fd_full - gfull) / np.maximum(1.0, np.abs(gfull)))[q].max(),
              (np.abs(fd_res - gres) / np.maximum(1.0, np.abs(gres)))[q].max())
    assert err < 1e-4, err


@pytest.mark.parametrize("kind", [LANE, COOP], ids=["lane", "coop"])
def test_cte_epsi_structure_and_envelope(mpc, po, refdata, torch_dev, kind):
    """On the GPU's own outputs (solve at tol 1e-10): d full / d cte0 = e_{4N} and d full / d epsi0 = e_{5N} +
    cos(epsi0) v0 dt e_{4N+1}, exactly up to the rounding of v0 dt cos(epsi0); and d cost / d state_k = -lambda_{kN} +
    (zl - zu)^T dz to 1e-6 max(1, |lambda|).  The barrier term is part of the check: at a bound held at the relaxation's
    slack (~1e-8 |bound|) it is slack times the stationarity row, and was measured at up to 1.6e-6 of |lambda|."""
    torch, dev = torch_dev
    cfg, cd = _cfgs(mpc, po, refdata)
    cfg.tol = 1e-10
    B = 2048
    b = mpc.workloads.batch_perturbed_states(B, 61, cd)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(kind)
    d = _solve(S, torch, dev, b)
    gres, gfull = _sens(S, torch, dev, d)
    S.close()
    sol = d["np"]
    ok = sol["status"] == 1
    assert ok.mean() > 0.99
    N = cd["N"]
    n = 8 * N - 2
    want_c = np.zeros(n)
    want_c[4 * N] = 1.0
    assert np.array_equal(gfull[ok, 4], np.broadcast_to(want_c, (ok.sum(), n)))
    e = gfull[ok, 5].copy()
    expect = np.cos(b["state"][ok, 5]) * b["state"][ok, 3] * cd["dt"]
    assert np.abs(e[:, 4 * N + 1] - expect).max() <= 1e-12 * np.abs(expect).max()
    e[:, 4 * N + 1] = 0.0
    want_e = np.zeros(n)
    want_e[5 * N] = 1.0
    assert np.array_equal(e, np.broadcast_to(want_e, e.shape))
    lam0 = sol["lam"][ok][:, [k * N for k in range(6)]]
    barrier = np.einsum("bj,bkj->bk", sol["zl"][ok] - sol["zu"][ok], gfull[ok])
    err = np.abs(gres[ok, :, 8] + lam0 - barrier) / np.maximum(1.0, np.abs(lam0))
    assert err.max() < 1e-6, err.max()


def test_invalid_problems_get_nan(mpc, po, refdata, stable_cd, torch_dev):
    """max_iter = 9, so that the batch has both MAXITER problems and solved ones (none of this workload converges in
    fewer than 7 iterations: at max_iter = 3 every problem is MAXITER)."""
    torch, dev = torch_dev
    cfg, cd = _cfgs(mpc, po, refdata)
    cfg.max_iter = 9
    B = 512
    b = mpc.workloads.batch_perturbed_states(B, 71, cd)
    S = mpc.Solver(cfg, 0)
    d = _solve(S, torch, dev, b)
    st = d["np"]["status"]
    solved = np.isin(st, [1, 4])
    assert (st == 2).any() and solved.any()
    gres, gfull = _sens(S, torch, dev, d)
    assert np.isnan(gres[~solved]).all() and np.isnan(gfull[~solved]).all()
    assert np.isfinite(gres[solved]).all() and np.isfinite(gfull[solved]).all()
    # status NULL: every problem is computed, the solved ones to the same bits
    nres, nfull = _sens(S, torch, dev, d, with_status=False)
    assert np.isfinite(nres[~solved]).any()
    assert np.array_equal(nres[solved], gres[solved]) and np.array_equal(nfull[solved], gfull[solved])
    # hand-made multipliers: a large negative zl on every steering bound makes the reduced Hessian indefinite
    N = cd["N"]
    zl = d["np"]["zl"].copy()
    zl[:, 6 * N:7 * N - 1] = -1e6
    d["zl"] = _up(torch, dev, zl)
    d["np"]["zl"] = zl
    ok = np.flatnonzero(solved)[:8]
    pd = _cpu(po, cd, b, d["np"], ok)[2]
    assert not pd.any()
    hres, hfull = _sens(S, torch, dev, d, with_status=False)
    assert np.isnan(hres[ok]).all() and np.isnan(hfull[ok]).all()
    S.close()


def test_bits_launches_and_arguments(mpc, stable_cfg, stable_cd, torch_dev):
    torch, dev = torch_dev
    B = 4096
    b = mpc.workloads.batch_perturbed_states(B, 81, stable_cd)
    S = mpc.Solver(stable_cfg, 0)
    d = _solve(S, torch, dev, b)
    n0 = S.launches
    r1, f1 = _sens(S, torch, dev, d)
    assert S.launches == n0 + 1
    r2, f2 = _sens(S, torch, dev, d)
    assert np.array_equal(r1, r2) and np.array_equal(f1, f2)
    r3, f3 = _sens(S, torch, dev, d, with_full=False)
    assert f3 is None and np.array_equal(r3, r1)
    # a 1000-problem slice alone: the same bits as inside the 4096 batch
    sl = {k: (None if v is None else v[..., 1000:2000].contiguous()) for k, v in d.items() if k != "np"}
    r4, f4 = _sens(S, torch, dev, sl)
    assert np.array_equal(r4, r1[1000:2000]) and np.array_equal(f4, f1[1000:2000])
    # the handle's solves are not changed by a sensitivity call
    d2 = _solve(S, torch, dev, b)
    _sens(S, torch, dev, d2)
    d3 = _solve(S, torch, dev, b)
    for k in ("full", "lam", "zl", "zu", "status", "result", "iters"):
        assert np.array_equal(d2["np"][k], d3["np"][k])
    # arguments
    L = mpc.lib()
    p = lambda t: None if t is None else t.data_ptr()
    dres = torch.zeros(6, 9, B, dtype=torch.float64, device=dev)
    args = [p(d[k]) for k in ("state", "coeffs", "yaw_lo", "yaw_hi")] + [None, None] + \
           [p(d[k]) for k in ("full", "lam", "zl", "zu", "status")] + [p(dres), None, None]
    assert L.mpc_solution_sensitivity(S._h, B, *args) == 0
    torch.cuda.synchronize()
    assert L.mpc_solution_sensitivity(None, B, *args) == -1
    assert L.mpc_solution_sensitivity(S._h, -1, *args) == -1
    for j in (0, 1, 2, 3, 6, 7, 8, 9, 11):
        bad = list(args)
        bad[j] = None
        assert L.mpc_solution_sensitivity(S._h, B, *bad) == -1, j
    n1 = S.launches
    assert L.mpc_solution_sensitivity(S._h, 0, *args) == 0 and S.launches == n1
    S.close()
