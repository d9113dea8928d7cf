"""Warm-started solves away from the N = 10 stable batch: every horizon kernel instantiation (NS = 10, 20, 32, 64;
lane groups of 16 and 32; two stages per lane at NS = 64), partial start points, warm problems that escalate from the
lane kernel to the coop kernel (records, resume launches, the restart list), the rare branches of the algorithm with a
warm start, per-problem weights and dt, the shift kernel, the single-solve warm start at long horizons, and the entry
points that ignore a bound warm start.

The reference is the warm-started CPU oracle (tests/oracle_warm.py) given the very start arrays the GPU was given:
the device start point is downloaded after the shift and passed unchanged.  Bars are the project's: status equal,
1e-4 absolute on actuations and trajectory, 1e-6 relative on cost.

Every GPU test asserts its own precondition (a branch fired in the oracle, records were parked, the intended kernel
ran), so that none can pass without running its path.  The tests at the end need no GPU: they check that the oracle-side
recipes still reach those branches, so that a change of the oracle or of the workload generator shows up there
instead of leaving the GPU tests without their subject."""
import ctypes
import json
import os

import numpy as np
import pytest

import oracle_warm as ow
import warm_start_numpy as wsn

ABS_TOL, REL_TOL = 1e-4, 1e-6
LANE, COOP = 2, 3
NT = os.cpu_count() or 4


@pytest.fixture(scope="module")
def torch_dev():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch, torch.device("cuda:0")


def _cell(mpc, po, refdata, N, dt, **knobs):
    """The stable config at horizon N, step dt -> (oracle config dict, device config with the solver knobs)."""
    js = dict(refdata["configs"]["stable"], N=N, dt=dt)
    cfg = mpc.config_from_json_text(json.dumps(js))
    for k, v in knobs.items():
        setattr(cfg, k, v)
    return po.load_config_dict(js), cfg


# ---- device side ---------------------------------------------------------------------------------------------------
def _up(torch, dev, a):
    return torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).to(dev)


def _solve(S, torch, dev, b, state=None, weights=None, dt_per=None):
    """One mpc_solve_batch on device copies of the batch, with the multiplier outputs on -> numpy outputs ([B, ...]),
    the device solution arrays ([rows][B]: full, lambda, zl, zu) and the number of kernel launches it took."""
    B, N = b["state"].shape[0], S.cfg.N
    st = _up(torch, dev, b["state"] if state is None else state)
    co, yl, yh = _up(torch, dev, b["coeffs"]), _up(torch, dev, b["yaw_lo"]), _up(torch, dev, b["yaw_hi"])
    w = None if weights is None else _up(torch, dev, weights)
    dtp = None if dt_per is None else _up(torch, dev, dt_per)
    f64 = lambda r: torch.zeros(r, B, dtype=torch.float64, device=dev)
    res, tx, ty, full = f64(9), f64(N), f64(N), f64(8 * N - 2)
    lam, zl, zu = f64(6 * N), f64(8 * N - 2), f64(8 * N - 2)
    status, iters = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
    S.set_dual_outputs(lam, zl, zu)
    n0 = S.launches
    S.solve_batch_device(B, st, co, yl, yh, res, tx, ty, full, status, iters, weights=w, dt_per=dtp)
    torch.cuda.synchronize()
    S.set_dual_outputs(None, None, None)
    T = lambda t: t.cpu().numpy().T.copy()
    return {"result": T(res), "traj_x": T(tx), "traj_y": T(ty), "full": T(full), "status": status.cpu().numpy(),
            "iters": iters.cpu().numpy(), "dev": (full, lam, zl, zu), "launches": S.launches - n0}


def _shifted(S, torch, sol):
    """mpc_warm_start_shift of a solution's device arrays -> the next step's start point (device, [rows][B])."""
    full, lam, zl, zu = sol["dev"]
    out = [torch.zeros_like(a) for a in (full, lam, zl, zu)]
    S.warm_start_shift(full.shape[1], full, out[0], lam, out[1], zl, out[2], zu, out[3])
    torch.cuda.synchronize()
    return out


def _next_step(b, sol, seed):
    """One control step later in the same frame: each problem's stage-1 state with a small seeded perturbation."""
    rng = np.random.default_rng(seed)
    s1 = sol["result"][:, :6].copy()
    B = s1.shape[0]
    s1[:, 4] += rng.normal(0.0, 0.02, B)
    s1[:, 5] += rng.normal(0.0, 0.005, B)
    s1[:, 3] += rng.normal(0.0, 0.1, B)
    return s1


# which parts of a start point a caller passes: x always, each multiplier or NULL
PARTS = {"full": (1, 1, 1, 1), "x": (1, 0, 0, 0), "x_lam": (1, 1, 0, 0), "x_zl_zu": (1, 0, 1, 1), "x_zl": (1, 0, 1, 0)}


def _pick(start, parts):
    return [a if p else None for a, p in zip(start, PARTS[parts])]


def _host(start):
    """Device start arrays ([rows][B]) -> the oracle's layout ([B][rows]); None stays None."""
    return [None if a is None else a.cpu().numpy().T.copy() for a in start]


# ---- oracle side ---------------------------------------------------------------------------------------------------
def _oracle_warm(po, cd, b, state, start, **knobs):
    """Warm-started oracle solves of the batch at `state` from host start arrays ([B][rows], None = not given)."""
    probs = po.problems_from_arrays(state, b["coeffs"], b["yaw_lo"], b["yaw_hi"])
    r = ow.solve_batch_warm(po.make_config(cd, **knobs), probs, *start, n_threads=NT)
    return {k: np.array([d[k] for d in r]) for k in r[0]}


def _oracle_cold(po, cd, b):
    """Cold oracle solutions of the batch -> (x, lambda, zl, zu) in the oracle's layout ([B][rows]) and the results."""
    B, n, m = b["state"].shape[0], 8 * cd["N"] - 2, 6 * cd["N"]
    probs = po.problems_from_arrays(b["state"], b["coeffs"], b["yaw_lo"], b["yaw_hi"])
    out = (po.OrcResult * B)()
    po.lib().orc_solve_batch(ctypes.byref(po.make_config(cd)), probs, B, out, NT)
    sol = [np.array([list(r.z[:n]) for r in out]), np.array([list(r.lam[:m]) for r in out]),
           np.array([list(r.zl[:n]) for r in out]), np.array([list(r.zu[:n]) for r in out])]
    return sol, np.array([list(r.result) for r in out])


def _natural_start_cpu(po, cd, b, seed):
    """The receding-horizon start on the CPU: the shifted cold oracle solution, the next state one step on."""
    sol, res = _oracle_cold(po, cd, b)
    start = [a.T.copy() for a in wsn.shift(cd["N"], *[s.T.copy() for s in sol])]
    return start, _next_step(b, {"result": res}, seed)


def _assert_matches(g, c, N, mask, long_horizon):
    """GPU outputs against the oracle on the problems of `mask`: status, actuations and first step, cost, trajectory;
    iterations {0, +1} (DESIGN.md section 3), or -- from N = LONG_N on -- equal on > 85 % (see LONG_N)."""
    assert mask.sum() > 0
    assert np.array_equal(g["status"][mask], c["status"][mask]), \
        (np.nonzero(mask & (g["status"] != c["status"]))[0][:10], g["status"][mask & (g["status"] != c["status"])][:10])
    d = np.abs(g["result"] - c["result"])[mask]
    assert d[:, :8].max() < ABS_TOL, d[:, :8].max()
    assert (d[:, 8] / np.maximum(1.0, np.abs(c["result"][mask, 8]))).max() < REL_TOL
    assert np.abs(g["traj_x"] - c["z"][:, :N])[mask].max() < ABS_TOL
    assert np.abs(g["traj_y"] - c["z"][:, N:2 * N])[mask].max() < ABS_TOL
    di = g["iters"].astype(int)[mask] - c["iters"].astype(int)[mask]
    if long_horizon:
        assert (di == 0).mean() > 0.85, np.unique(di, return_counts=True)
    else:
        assert di.min() >= 0 and di.max() <= 1, np.unique(di, return_counts=True)
    return d


# From N = 30 on, the iteration bar is the one of the cold long-horizon tests (tests/test_gpu_restoration.py): equal on
# more than 85 % of the problems -- over a long horizon the Riccati recursion and the oracle's dense LDL^T round
# differently enough to move a step-size decision now and then.
LONG_N = 30


def _warm_solve(S, torch, dev, b, start, parts, mu, state=None, **kw):
    S.set_warm_start(*_pick(start, parts), mu_init=mu)
    g = _solve(S, torch, dev, b, state=state, **kw)
    S.set_warm_start(None)
    return g


# ======================================================================================================================
# 1. every horizon kernel, natural receding-horizon start
# ======================================================================================================================
GRID = [2, 3, 10, 11, 20, 21, 32, 33, 40, 64]


@pytest.mark.gpu
@pytest.mark.parametrize("mu", [1e-4, 0.1])
@pytest.mark.parametrize("N", GRID)
def test_horizon_grid_natural_start(mpc, po, refdata, torch_dev, N, mu, kernel_kind):
    """N = 2 (the last stage has no controls), 3, 10 | 11 (NS = 10 with groups of 16 lanes | NS = 20 with groups of
    32), 20 | 21, 32 | 33 (NS = 32 | NS = 64, two stages per lane), 40, 64: the shifted solution of a cold solve as the
    start point of the next step, against the oracle from the same arrays."""
    torch, dev = torch_dev
    dt = 0.05 if N == 64 else 0.1
    B = 60 if N == 64 else 128
    cd, cfg = _cell(mpc, po, refdata, N, dt)
    b = mpc.workloads.batch_perturbed_states(B, 1, cd)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(kernel_kind)
    cold = _solve(S, torch, dev, b)
    start = _shifted(S, torch, cold)
    s1 = _next_step(b, cold, N)
    g = _warm_solve(S, torch, dev, b, start, "full", mu, state=s1)
    S.close()
    assert g["launches"] == (2 if kernel_kind == LANE else 1)     # lane kernel + its finisher, or the coop kernel
    c = _oracle_warm(po, cd, b, s1, _host(start), mu_init=mu)
    ok = c["status"] == 1
    assert ok.mean() > 0.99
    _assert_matches(g, c, N, ok, N >= LONG_N)
    assert not np.array_equal(g["iters"], cold["iters"])         # the start point did change the solves


# ======================================================================================================================
# 2. partial start points
# ======================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("parts", ["x", "x_lam", "x_zl_zu", "x_zl"])
@pytest.mark.parametrize("N", [10, 40])
def test_partial_start_points(mpc, po, refdata, torch_dev, N, parts, kernel_kind):
    """x alone (lambda from the least-squares trip, zl / zu = 1), x with lambda, x with zl and zu, x with zl alone:
    the oracle given the same NULLs.  At N = 40 the primal start leads some problems to more than 8 filter entries,
    which the lane kernel hands to the coop kernel."""
    torch, dev = torch_dev
    B = 128 if N == 10 else 120
    cd, cfg = _cell(mpc, po, refdata, N, 0.1)
    b = mpc.workloads.batch_perturbed_states(B, 1, cd)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(kernel_kind)
    cold = _solve(S, torch, dev, b)
    start = _shifted(S, torch, cold)
    s1 = _next_step(b, cold, N)
    g = _warm_solve(S, torch, dev, b, start, parts, 1e-4, state=s1)
    S.close()
    assert g["launches"] == (2 if kernel_kind == LANE else 1)
    c = _oracle_warm(po, cd, b, s1, _pick(_host(start), parts), mu_init=1e-4)
    if N == 40 and parts == "x":
        assert (c["n_filter_max"] > 8).sum() >= 1
    ok = c["status"] == 1
    assert ok.mean() > 0.99
    _assert_matches(g, c, N, ok, N >= LONG_N)


# ======================================================================================================================
# 3. warm problems that escalate: mismatched start points
# ======================================================================================================================
MISMATCHED = [(30, 0.1, 240), (64, 0.05, 60)]


def _mismatched(torch, sol):
    """Each problem started from its neighbour's solution (column b from column b - 1): far enough from the problem's
    own solution to reach every rare branch of the algorithm, the restoration phase included."""
    return [torch.roll(a, 1, dims=1).contiguous() for a in sol["dev"]]


@pytest.mark.gpu
@pytest.mark.parametrize("parts", ["full", "x"])
@pytest.mark.parametrize("N,dt,B", MISMATCHED)
def test_mismatched_start_matches_oracle_unmasked(mpc, po, refdata, torch_dev, N, dt, B, parts, kernel_kind):
    """Every problem of the batch, whatever its status; the ones that went through the restoration phase match the
    oracle's optimum to 1e-6, as in the cold restoration cells (tests/test_gpu_restoration.py)."""
    torch, dev = torch_dev
    cd, cfg = _cell(mpc, po, refdata, N, dt)
    b = mpc.workloads.batch_perturbed_states(B, 1, cd)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(kernel_kind)
    start = _mismatched(torch, _solve(S, torch, dev, b))
    g = _warm_solve(S, torch, dev, b, start, parts, 1e-4)
    S.close()
    c = _oracle_warm(po, cd, b, b["state"], _pick(_host(start), parts), mu_init=1e-4)
    r = c["n_resto"] > 0
    assert r.sum() >= 3                                       # the restoration phase does run
    assert (c["n_filter_max"] > 8).sum() >= 3                 # ... and filters beyond what a lane holds
    d = _assert_matches(g, c, N, np.ones(B, dtype=bool), True)
    assert d[r][:, :8].max() < 1e-6


def _hard_mismatched(mpc, torch, dev, N, dt, refdata, po, B_out):
    """The mismatched start on the (30, 0.1, 240) / (64, 0.05, 60) batch; the problems that take more than 40
    iterations in the coop kernel (the ones that escalate), tiled to B_out problems with their start columns."""
    B = {30: 240, 64: 60}[N]
    cd, cfg = _cell(mpc, po, refdata, N, dt)
    b = mpc.workloads.batch_perturbed_states(B, 1, cd)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(COOP)
    start = _mismatched(torch, _solve(S, torch, dev, b))
    g = _warm_solve(S, torch, dev, b, start, "full", 1e-4)
    S.close()
    hard = np.nonzero(g["iters"] > 40)[0]
    assert len(hard) >= 5, np.sort(g["iters"])[-10:]
    idx = np.tile(hard, B_out // len(hard) + 1)[:B_out]
    it = torch.from_numpy(idx).to(dev)
    bt = {k: b[k][idx] for k in ("state", "coeffs", "yaw_lo", "yaw_hi")}
    return cfg, bt, [a[:, it].contiguous() for a in start]


@pytest.mark.gpu
@pytest.mark.parametrize("N,dt", [(30, 0.1), (64, 0.05)])
def test_lane_chain_and_coop_kernel_same_bits_warm_escalations(mpc, po, refdata, torch_dev, N, dt):
    """Warm problems that all escalate, 1500 of them: the lane chain gives the bits of the coop kernel with tail packing
    off (0, 0), on (16, 3) and (8, 1).  The lane kernel parks a problem it hands over as a record where a slot is free
    -- a warm one possibly before its first trip -- and otherwise puts it on the restart list, from which the finisher
    solves it again from its start point (init with the warm start).  With tail packing off the records hold
    max(B / 8, 1024) = 1024 problems here, so more than 1024 hand-overs send the rest through the restart list."""
    torch, dev = torch_dev
    cfg, b, start = _hard_mismatched(mpc, torch, dev, N, dt, refdata, po, 1500)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(COOP)
    ref = _warm_solve(S, torch, dev, b, start, "full", 1e-4)
    assert ref["launches"] == 1 and ref["iters"].max() > 100
    S.set_kernel(LANE)
    for park, resume in ((0, 0), (16, 3), (8, 1)):
        S.set_tail(park, resume)
        got = _warm_solve(S, torch, dev, b, start, "full", 1e-4)
        parked = S.tail_counts(4)
        assert got["launches"] == 2 + resume, (park, resume, got["launches"])
        if park == 0:
            assert parked[0] > 1024, parked                   # hand-overs beyond the records: the restart list
        else:
            assert parked[0] > 0, parked
        for k in ("result", "traj_x", "traj_y", "full", "status", "iters"):
            assert np.array_equal(got[k], ref[k]), (park, resume, k)
    S.close()
    assert (ref["status"] == 1).mean() > 0.99


@pytest.mark.gpu
def test_warm_resume_launches_same_bits_as_coop_kernel(mpc, po, refdata, torch_dev):
    """16384 warm problems that all escalate: more than 8192 parked records, so the resume launches of the lane kernel
    run (with the default threshold of 8192 records) on warm records, hand them on, and the finisher completes them --
    bit-identical to the coop kernel (cf. test_resume_launches_hand_on_the_problems_they_cannot_finish, cold)."""
    torch, dev = torch_dev
    cfg, b, start = _hard_mismatched(mpc, torch, dev, 30, 0.1, refdata, po, 16384)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(COOP)
    ref = _warm_solve(S, torch, dev, b, start, "full", 1e-4)
    S.set_kernel(LANE)
    g = _warm_solve(S, torch, dev, b, start, "full", 1e-4)
    parked = S.tail_counts(4)
    S.close()
    assert parked[0] > 8192, parked                           # the main launch handed over enough for a resume launch
    assert parked[1] > 0, parked                              # ... and the first resume launch ran and handed on
    for k in ("result", "traj_x", "traj_y", "full", "status", "iters"):
        assert np.array_equal(g[k], ref[k]), k


# ======================================================================================================================
# 4. forced rare branches with a warm start
# ======================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("knobs,counter", [({"watchdog_trigger": 1}, "n_watchdog"), ({"tiny_step_tol": 1e-7}, "n_tiny")])
def test_watchdog_and_tiny_step_warm(mpc, po, refdata, torch_dev, knobs, counter, kernel_kind):
    """The watchdog after one shortened step and the tiny-step test at 1e-7, forced through Ipopt's options, on the
    mismatched start at N = 30.  As in test_watchdog_tiny_step_and_filter_reset_branches, problems whose oracle answer
    does not survive a 1e-13 relative change of v0 are chaotic and compared with nothing; the branch must have fired
    on problems that do survive."""
    torch, dev = torch_dev
    N, dt, B = MISMATCHED[0]
    cd, cfg = _cell(mpc, po, refdata, N, dt, **knobs)
    b = mpc.workloads.batch_perturbed_states(B, 1, cd)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(kernel_kind)
    start = _mismatched(torch, _solve(S, torch, dev, b))
    g = _warm_solve(S, torch, dev, b, start, "full", 1e-4)
    S.close()
    hs = _host(start)
    c = _oracle_warm(po, cd, b, b["state"], hs, mu_init=1e-4, **knobs)
    c2 = _oracle_warm(po, cd, b, b["state"] * np.array([1, 1, 1, 1 + 1e-13, 1, 1]), hs, mu_init=1e-4, **knobs)
    stable = (np.abs(c2["result"] - c["result"])[:, :8].max(axis=1) < 1e-6) & (c2["status"] == c["status"])
    assert stable.mean() > 0.9, stable.mean()
    f = stable & (c[counter] > 0)
    assert f.sum() >= 1, "the branch did not fire in the oracle"
    d = _assert_matches(g, c, N, stable, True)
    assert np.abs(g["result"] - c["result"])[f][:, :8].max() < 1e-6
    assert d.shape[0] == stable.sum()


# ======================================================================================================================
# 5. per-problem weights and dt with a warm start
# ======================================================================================================================
def _weight_groups(cd):
    """Weight vectors of a sweep: the config's own, and ones that move the objective factor sf (Ipopt's gradient-based
    objective scaling, 100 / max |grad f| at the start point) to ~1e-2 and below -- the factor by which the kernel
    takes the caller's multipliers over to the scaled problem."""
    w0 = np.array(cd["weights"], dtype=np.float64)
    out = [w0.copy()]
    for k, v in ((2, 100.0), (2, 1000.0), (0, 2e4)):
        w = w0.copy()
        w[k] = v
        out.append(w)
    return out


def _objective_factor(po, cd, b, w):
    """sf of every problem of the batch under weights w: from the oracle's gradient at the cold start point."""
    cfg = po.make_config(dict(cd, weights=list(w)))
    probs = po.problems_from_arrays(b["state"], b["coeffs"], b["yaw_lo"], b["yaw_hi"])
    sf = []
    for i in range(len(probs)):
        xi = po.bounds(cfg, probs[i])[4]
        gmx = np.abs(po.eval_grad(cfg, probs[i], xi)).max()
        sf.append(max(100.0 / gmx, 1e-8) if gmx > 100.0 else 1.0)
    return np.array(sf)


@pytest.mark.gpu
def test_per_problem_weights_warm(mpc, po, refdata, torch_dev, kernel_kind):
    """A weight sweep, warm-started: per-problem weights in one batch against the oracle run once per weight vector."""
    torch, dev = torch_dev
    cd, cfg = _cell(mpc, po, refdata, 10, 0.1)
    G, per = 4, 64
    b = mpc.workloads.batch_perturbed_states(G * per, 3, cd)
    groups = _weight_groups(cd)
    W = np.repeat(np.array(groups), per, axis=0)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(kernel_kind)
    cold = _solve(S, torch, dev, b, weights=W)
    start = _shifted(S, torch, cold)
    s1 = _next_step(b, cold, 3)
    g = _warm_solve(S, torch, dev, b, start, "full", 1e-4, state=s1, weights=W)
    S.close()
    hs = _host(start)
    sf_min = []
    for k, w in enumerate(groups):
        sl = slice(k * per, (k + 1) * per)
        bk = {key: b[key][sl] for key in ("state", "coeffs", "yaw_lo", "yaw_hi")}
        bk1 = dict(bk, state=s1[sl])
        sf_min.append(_objective_factor(po, cd, bk1, w).min())
        c = _oracle_warm(po, dict(cd, weights=list(w)), bk, s1[sl], [a[sl] for a in hs], mu_init=1e-4)
        ok = c["status"] == 1
        assert ok.mean() > 0.95, (k, ok.mean())
        gk = {key: g[key][sl] for key in ("result", "traj_x", "traj_y", "status", "iters")}
        _assert_matches(gk, c, 10, ok, False)
    assert min(sf_min) <= 1e-2, sf_min


@pytest.mark.gpu
def test_per_problem_dt_warm(mpc, po, refdata, torch_dev, kernel_kind):
    """dt_per in {0.05, 0.1} at N = 20, warm-started: against the oracle run once per dt."""
    torch, dev = torch_dev
    N = 20
    cd, cfg = _cell(mpc, po, refdata, N, 0.1)
    B = 192
    b = mpc.workloads.batch_perturbed_states(B, 4, cd)
    dtp = np.where(np.arange(B) % 2 == 0, 0.05, 0.1)
    S = mpc.Solver(cfg, 0)
    S.set_kernel(kernel_kind)
    cold = _solve(S, torch, dev, b, dt_per=dtp)
    start = _shifted(S, torch, cold)
    s1 = _next_step(b, cold, 4)
    g = _warm_solve(S, torch, dev, b, start, "full", 1e-4, state=s1, dt_per=dtp)
    S.close()
    hs = _host(start)
    for dt in (0.05, 0.1):
        sel = np.nonzero(dtp == dt)[0]
        bk = {key: b[key][sel] for key in ("state", "coeffs", "yaw_lo", "yaw_hi")}
        c = _oracle_warm(po, dict(cd, dt=dt), bk, s1[sel], [a[sel] for a in hs], mu_init=1e-4)
        ok = c["status"] == 1
        assert ok.mean() > 0.99, (dt, ok.mean())
        gk = {key: g[key][sel] for key in ("result", "traj_x", "traj_y", "status", "iters")}
        _assert_matches(gk, c, N, ok, False)


# ======================================================================================================================
# 6. the shift kernel at every horizon shape
# ======================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("N", [2, 3, 17, 33, 64])
def test_shift_kernel_equals_cpu_shift_all_shapes(mpc, refdata, torch_dev, N):
    """Random non-trivial columns (no structure the kernel could get right by accident) for B = 1, 255, 257 (one
    thread block and one more thread) and 3000: the device shift equals the CPU shift bit for bit -- the full start
    point, the primal point alone and each multiplier alone -- and writes nothing it was not given."""
    torch, dev = torch_dev
    S = mpc.Solver(mpc.config_from_json_text(json.dumps(refdata["configs"]["stable"])), 0)
    S.set_config(mpc.config_from_json_text(json.dumps(dict(refdata["configs"]["stable"], N=N))))
    rows = (8 * N - 2, 6 * N, 8 * N - 2, 8 * N - 2)
    rng = np.random.default_rng(N)
    for B in (1, 255, 257, 3000):
        h = [rng.normal(0.0, 1.0, (r, B)) * np.exp(rng.uniform(-5, 5, (r, B))) for r in rows]
        d = [torch.from_numpy(a).to(dev) for a in h]
        for use in ((1, 1, 1, 1), (1, 0, 0, 0), (1, 1, 0, 0), (1, 0, 1, 0), (1, 0, 0, 1)):
            out = [torch.full_like(a, float("nan")) for a in d]
            args = []
            for a, o, u in zip(d, out, use):
                args += [a, o] if u else [None, None]
            S.warm_start_shift(B, *args)
            torch.cuda.synchronize()
            want = wsn.shift(N, *[a if u else None for a, u in zip(h, use)])
            for o, w, u in zip(out, want, use):
                o = o.cpu().numpy()
                if u:
                    assert np.array_equal(o, w), (N, B, use)
                else:
                    assert np.isnan(o).all(), (N, B, use)
    S.close()


# ======================================================================================================================
# 7. mpc_set_warm_start_one at long horizons
# ======================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("N,dt", [(20, 0.1), (33, 0.1), (64, 0.05)])
def test_solve_one_warm_start_long_horizons(mpc, po, refdata, torch_dev, N, dt):
    """Eight single solves one control step apart in one frame with mpc_set_warm_start_one give the bits of the same
    sequence done by hand on a B = 1 coop-kernel handle (solve with dual outputs, mpc_warm_start_shift,
    mpc_set_warm_start, next solve); after mpc_set_config to another horizon the next single solve is a cold one."""
    torch, dev = torch_dev
    cd, cfg = _cell(mpc, po, refdata, N, dt)
    b = mpc.workloads.batch_perturbed_states(1, 5, cd)
    W = mpc.Solver(cfg, 0)
    W.set_warm_start_one(True, mu_init=1e-4)
    H = mpc.Solver(cfg, 0)
    H.set_kernel(COOP)
    C = mpc.Solver(cfg, 0)
    state = b["state"][0].copy()
    start, n_warm, it_w, it_c = None, 0, 0, 0
    for step in range(8):
        w = W.solve_one(state, b["coeffs"][0], b["yaw_lo"][0], b["yaw_hi"][0])
        bs = dict(b, state=state[None, :])
        h = _warm_solve(H, torch, dev, bs, start, "full", 1e-4) if start is not None else _solve(H, torch, dev, bs)
        for k in ("result", "traj_x", "traj_y"):
            assert np.array_equal(w[k], h[k][0]), (step, k)
        assert w["status"] == h["status"][0] and w["iters"] == h["iters"][0], step
        c = C.solve_one(state, b["coeffs"][0], b["yaw_lo"][0], b["yaw_hi"][0])
        if start is not None:
            n_warm += 1
            it_w += w["iters"]; it_c += c["iters"]
        start = _shifted(H, torch, h) if w["status"] == 1 else None   # a failed solve is no start point
        state = w["result"][:6].copy()
    assert n_warm >= 6 and it_w < it_c, (n_warm, it_w, it_c)     # the warm start was used and did help
    cd10, cfg10 = _cell(mpc, po, refdata, 10, 0.1)
    b10 = mpc.workloads.batch_perturbed_states(1, 6, cd10)
    one = (b10["state"][0], b10["coeffs"][0], b10["yaw_lo"][0], b10["yaw_hi"][0])
    W.set_config(cfg10)
    w = W.solve_one(*one)
    C.set_config(cfg10)
    c = C.solve_one(*one)
    for k in ("result", "traj_x", "traj_y", "status", "iters"):
        assert np.array_equal(np.asarray(w[k]), np.asarray(c[k])), k
    W.close(); H.close(); C.close()


# ======================================================================================================================
# 8. entry points that start cold whatever warm start is bound
# ======================================================================================================================
@pytest.mark.gpu
@pytest.mark.parametrize("rollout_mode", [1, 2])
def test_run_batch_and_rollout_ignore_bound_warm_start(mpc, po, refdata, torch_dev, rollout_mode):
    """A warm start bound to the handle (of another batch size: 2B columns, so that reading it can only go wrong in
    value, not out of bounds) changes nothing in mpc_run_batch and mpc_rollout, in either rollout mode."""
    torch, dev = torch_dev
    cd, cfg = _cell(mpc, po, refdata, 10, 0.1)
    B, T = 96, 4
    b = mpc.workloads.batch_perturbed_states(B, 8, cd)
    wx, wy = np.array(refdata["waypoints"]["x"]), np.array(refdata["waypoints"]["y"])
    win = (b["segment"][:, None] + np.arange(6)[None, :]) % len(wx)
    pose = _up(torch, dev, np.stack([b["px"], b["py"], b["psi"], b["v"]], axis=1))
    ptsx, ptsy = _up(torch, dev, wx[win]), _up(torch, dev, wy[win])
    veh0 = np.stack([b["px"], b["py"], b["psi"], np.clip(b["v"], 8, 30), np.zeros(B), np.zeros(B)], axis=1)

    def run(S):
        out8 = torch.zeros(8, B, dtype=torch.float64, device=dev)
        tx, ty = torch.zeros(10, B, dtype=torch.float64, device=dev), torch.zeros(10, B, dtype=torch.float64, device=dev)
        st, it = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
        S.run_batch_device(B, pose, ptsx, ptsy, 6, out8, traj_x=tx, traj_y=ty, status=st, iters=it)
        veh, seg = _up(torch, dev, veh0), _up(torch, dev, b["segment"].astype(np.int32))
        pending = torch.zeros(2, B, dtype=torch.float64, device=dev)
        rec = torch.zeros(T, 8, B, dtype=torch.float64, device=dev)
        S.rollout_device(B, T, _up(torch, dev, wx), _up(torch, dev, wy), veh, seg, pending, 0.1, 0.0, rec)
        torch.cuda.synchronize()
        return [a.cpu().numpy() for a in (out8, tx, ty, st, it, veh, seg, pending, rec)]

    S = mpc.Solver(cfg, 0)
    S.set_rollout_mode(rollout_mode)
    ref = run(S)
    b2 = mpc.workloads.batch_perturbed_states(2 * B, 9, cd)
    start = _shifted(S, torch, _solve(S, torch, dev, b2))
    S.set_warm_start(*start, mu_init=1e-4)
    got = run(S)
    # the same warm start does change a batch solve of 2B problems on this handle: it is bound and live
    warm = _solve(S, torch, dev, b2)
    S.set_warm_start(None)
    cold = _solve(S, torch, dev, b2)
    S.close()
    assert not np.array_equal(warm["iters"], cold["iters"])
    assert (ref[3] == 1).mean() > 0.9
    for k, (x, y) in enumerate(zip(got, ref)):
        assert np.array_equal(x, y), k


# ======================================================================================================================
# 9. without a GPU: the oracle-side recipes still reach the branches the GPU tests above are about
# ======================================================================================================================
@pytest.mark.parametrize("N,dt,B", MISMATCHED)
def test_mismatched_start_reaches_rare_branches_in_oracle(mpc, po, refdata, N, dt, B):
    """The mismatched start (each problem from its neighbour's solution) sends problems through the restoration phase
    and past 8 filter entries, for the full start point and the primal point alone, and -- at N = 30 -- the forced
    watchdog and tiny-step options fire."""
    cd = po.load_config_dict(dict(refdata["configs"]["stable"], N=N, dt=dt))
    b = mpc.workloads.batch_perturbed_states(B, 1, cd)
    sol, _ = _oracle_cold(po, cd, b)
    start = [np.roll(a, 1, axis=0) for a in sol]
    for parts in ("full", "x"):
        c = _oracle_warm(po, cd, b, b["state"], _pick(start, parts), mu_init=1e-4)
        assert (c["n_resto"] > 0).sum() >= 3, parts
        assert (c["n_filter_max"] > 8).sum() >= 3, parts
    if N == 30:
        for knobs, counter in (({"watchdog_trigger": 1}, "n_watchdog"), ({"tiny_step_tol": 1e-7}, "n_tiny")):
            c = _oracle_warm(po, cd, b, b["state"], start, mu_init=1e-4, **knobs)
            assert (c[counter] > 0).sum() >= 1, knobs


def test_primal_start_fills_filter_at_n40_in_oracle(mpc, po, refdata):
    """The natural primal-only start at N = 40 leads the oracle past 8 filter entries on some problems: the lane
    kernel's hand-over of a problem that has no caller multipliers."""
    cd = po.load_config_dict(dict(refdata["configs"]["stable"], N=40, dt=0.1))
    b = mpc.workloads.batch_perturbed_states(120, 1, cd)
    start, s1 = _natural_start_cpu(po, cd, b, 40)
    c = _oracle_warm(po, cd, b, s1, _pick(start, "x"), mu_init=1e-4)
    assert (c["n_filter_max"] > 8).sum() >= 1
    assert (c["status"] == 1).mean() > 0.99


def test_weight_groups_move_objective_factor(mpc, po, refdata):
    """The weight vectors of test_per_problem_weights_warm put sf at ~1e-2 and below on their problems, as computed
    from the oracle's gradient at the start point; and nlp_numpy's statement of the gradient agrees there."""
    import nlp_numpy as nn
    cd = po.load_config_dict(refdata["configs"]["stable"])
    b = mpc.workloads.batch_perturbed_states(64, 3, cd)
    sfs = [_objective_factor(po, cd, b, w) for w in _weight_groups(cd)]
    assert np.median(sfs[0]) > 0.5                            # the config's own weights: sf near 1
    assert np.median(sfs[1]) <= 2e-2 and np.median(sfs[2]) <= 2e-3 and sfs[3].min() <= 1e-2, [np.median(s) for s in sfs]
    # the same factor from the independent numpy NLP (objective gradient = Lagrangian gradient with no multipliers)
    w = _weight_groups(cd)[2]
    cdw = dict(cd, weights=list(w))
    N = cd["N"]
    z0 = nn.start_point(cdw, b["state"])
    zero = np.zeros((64, 8 * N - 2))
    g = nn.lagrangian_gradient(cdw, nn.frozen(cdw, b["state"], np.tile(w, (64, 1))), b["state"], b["coeffs"], z0,
                               np.zeros((64, 6 * N)), zero, zero)
    gmx = np.abs(g).max(axis=1)
    np.testing.assert_allclose(np.where(gmx > 100, np.maximum(100 / gmx, 1e-8), 1.0), sfs[2], rtol=1e-12)
