"""The oracle and the host-side run() logic against vectors produced by the REFERENCE'S OWN sources.

tests/golden/ref_golden.json was written by tests/golden/make_ref_golden.py from oracle/_ref/libmpc_ref.so =
/root/reference/src/{control/MPC,model/Vehicle,model/RoadGeometry,utils/utils,utils/Config}.cpp compiled
unmodified against the CppAD/Ipopt stand-ins of oracle/ref_shim.  The objective with its branches
frozen at the start point, the constraints, bounds, start point, outputs, Config::load conversions and
MPC::run's pre/post-processing in those vectors all come from the reference's text, not from a
restatement.  (What remains restated is Ipopt itself: DESIGN.md, "parity".)"""
import json
import os

import numpy as np
import pytest

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
ABS_TOL, REL_TOL = 1e-4, 1e-6          # the north star's tolerances
TIGHT = 1e-7                            # what same-algorithm implementations actually achieve


@pytest.fixture(scope="module")
def gold():
    return json.load(open(os.path.join(GOLD, "ref_golden.json")))


def _cmp(res, ref, tol=TIGHT):
    res, ref = np.asarray(res), np.asarray(ref)
    assert np.abs(res[:8] - ref[:8]).max() < tol
    assert res[8] == pytest.approx(ref[8], rel=1e-9)


def test_oracle_matches_reference_testcpp(gold, po, stable_cd):
    """src/test.cpp:64-111 -- run() then 25 x solve(), four fixtures."""
    cfg = po.make_config(stable_cd)
    for sc in gold["testcpp"]:
        run = sc["run"]
        for step in sc["steps"]:
            r = po.solve(cfg, po.make_problem(step["state"], run["coeffs"], run["yaw_lo"], run["yaw_hi"]))
            assert r["status"] == step["status"] == 1
            assert r["iters"] == step["iters"]
            _cmp(r["result"], step["result"])
            assert np.abs(r["z"][:cfg.N] - np.array(step["traj_x"])).max() < TIGHT


def test_oracle_matches_reference_weight_sweep(gold, po, stable_cd):
    """Config::weights varied, including WEIGHT_A / WEIGHT_DA / WEIGHT_DECEL_LOW_V, which the reference's
    recorded tape never contains (its `if (a > 0)` branches are decided at the all-zero start point)."""
    for c in gold["weights"]:
        cd = dict(stable_cd, weights=c["weights"])
        r = po.solve(po.make_config(cd), po.make_problem(c["state"], c["coeffs"], c["yaw_lo"], c["yaw_hi"]))
        assert r["status"] == c["status"]
        if c["status"] == 1:
            _cmp(r["result"], c["result"])
        # and the dead weights really are dead in the oracle's statement too
        w2 = list(c["weights"]); w2[6] = 0.0; w2[7] = 123.0; w2[8] = 0.5
        r2 = po.solve(po.make_config(dict(stable_cd, weights=w2)), po.make_problem(c["state"], c["coeffs"], c["yaw_lo"], c["yaw_hi"]))
        assert np.array_equal(r2["result"], r["result"])


def test_oracle_matches_reference_horizon_grid(gold, po, stable_cd):
    for c in gold["grid"]:
        cd = dict(stable_cd, N=c["N"], dt=c["dt"])
        r = po.solve(po.make_config(cd), po.make_problem(c["state"], c["coeffs"], c["yaw_lo"], c["yaw_hi"]))
        assert r["status"] == c["status"] == 1
        _cmp(r["result"], c["result"], tol=1e-6)
        assert np.abs(r["z"][c["N"]:2 * c["N"]] - np.array(c["traj_y"])).max() < 1e-6


def test_oracle_matches_reference_on_restoration_cases(gold, po, stable_cd):
    """The analytic restatement and the reference's own FG_eval (through the AD tape) walk the same path through the
    restoration phase: same status, same iteration count, same point."""
    assert len(gold["resto"]) >= 8
    for c in gold["resto"]:
        cd = dict(stable_cd, N=c["N"], dt=c["dt"])
        r = po.solve(po.make_config(cd), po.make_problem(c["state"], c["coeffs"], c["yaw_lo"], c["yaw_hi"]))
        assert r["n_resto"] == c["oracle_n_resto"] >= 1
        assert r["status"] == c["status"] == 1
        assert r["iters"] == c["iters"]
        _cmp(r["result"], c["result"], tol=1e-6)


def test_host_run_logic_matches_reference(gold, mpc, po, refdata):
    """mpc_run_prepare / mpc_run_finish (product, host C++) == MPC::run of the reference: vehicle-frame
    waypoints, adaptive-order fit, cte/epsi, yaw bounds; then steer adjustment, accel clamp, normalisation
    applied to the oracle's solve."""
    cfgs = {n: mpc.config_from_json_text(json.dumps(refdata["configs"][n])) for n in refdata["configs"]}
    ocfg = {n: po.make_config(po.load_config_dict(refdata["configs"][n])) for n in refdata["configs"]}
    orders = set()
    for c in gold["run"]:
        cfg = cfgs[c["config"]]
        p = mpc.run_prepare(cfg, c["pose"], c["ptsx"], c["ptsy"])
        assert np.allclose(p["ptsx"], c["ptsx_vehicle"], rtol=0, atol=1e-12)
        assert np.allclose(p["ptsy"], c["ptsy_vehicle"], rtol=0, atol=1e-12)
        assert p["aux"].fit_order + 1 == c["ncoef"]
        orders.add(c["ncoef"])
        assert np.allclose(p["coeffs"], c["coeffs"], rtol=1e-7, atol=1e-10)
        assert (p["yaw_lo"], p["yaw_hi"]) == pytest.approx((c["yaw_lo"], c["yaw_hi"]), rel=1e-8, abs=1e-10)
        # solve on the REFERENCE's coefficients (isolates the post-processing from fit rounding)
        r = po.solve(ocfg[c["config"]], po.make_problem(p["state"], c["coeffs"], c["yaw_lo"], c["yaw_hi"]))
        assert r["status"] == c["status"]
        if c["status"] != 1:
            continue
        out8 = mpc.run_finish(cfg, p["aux"], c["pose"][3], r["result"])
        assert np.abs(out8 - np.array(c["result"])).max() < 1e-6
    assert orders == {3, 4, 5}          # fit orders 2, 3 and 4 all occur


def test_host_run_logic_errors(mpc, stable_cfg):
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):
        mpc.run_prepare(stable_cfg, (0, 0, 0, 10), [0.0, 1.0], [0.0, 0.0])             # fewer than 3 waypoints
    with pytest.raises(mpc.MpcError, match="MPC_EINVAL"):
        mpc.run_prepare(stable_cfg, (0, 0, 0, 10), list(range(17)), [0.0] * 17)       # more than MPC_MAX_WAYPOINTS


def test_live_reference_build_agrees_with_oracle(po, refdata):
    """Where oracle/_ref exists (built by `make -C oracle/ref_shim REF=<checkout of the original project>`; the
    original project's sources are not part of this repository), run the reference's code live: Config::load and
    fresh random problems."""
    from oracle import pyref as pr
    if not pr.available():
        pytest.skip("oracle/_ref/libmpc_ref.so not built (needs the original project's sources: make -C oracle/ref_shim REF=...)")
    import mpc_b200 as mpc
    for name in ("stable", "fast", "no-latency"):
        js = refdata["configs"][name]
        pr.config_load(js)
        cd = po.load_config_dict(js)
        got = pr.config_get()
        for k, v in got.items():
            assert np.array_equal(np.array(v, dtype=float), np.array(cd[k], dtype=float)), (name, k)
        b = mpc.workloads.batch_perturbed_states(12, 900, cd)
        cfg = po.make_config(cd)
        for i in range(12):
            r = pr.solve(b["state"][i], b["coeffs"][i], b["yaw_lo"][i], b["yaw_hi"][i], cd["N"])
            o = po.solve(cfg, po.make_problem(b["state"][i], b["coeffs"][i], b["yaw_lo"][i], b["yaw_hi"][i]))
            assert r["status"] == o["status"]
            if o["status"] == 1:
                _cmp(o["result"], r["result"])
    # panic branches and negative speed: the branch outcomes come from the reference's own comparisons
    js = refdata["configs"]["stable"]
    pr.config_load(js)
    cd = po.load_config_dict(js)
    cfg = po.make_config(cd)
    for st in ([0, 0, 0.0, 20.0, 1.5, 0.02], [0, 0, 0.0, 20.0, 0.1, 0.3], [0, 0, 0.05, -2.0, 0.3, 0.0], [0, 0, 0.02, 15.0, -2.0, -0.25]):
        co = [st[4], -np.tan(st[5]), 0.002, 0.0, 0.0]
        r = pr.solve(st, co, -0.1, 0.4, cd["N"])
        o = po.solve(cfg, po.make_problem(st, co, -0.1, 0.4))
        assert r["status"] == o["status"] == 1
        _cmp(o["result"], r["result"])


def test_plant_and_throttle_map_match_reference(gold, mpc, refdata):
    """mpc_vehicle_move / mpc_compute_throttle (product, shared host/device code) == Vehicle::move /
    Vehicle::computeThrottle of the reference; so does the test-side restatement used for the rollout oracle."""
    import closed_loop_restated as clr
    for c in gold["plant"]["move"]:
        cfg = mpc.config_from_json_text(json.dumps(refdata["configs"][c["config"]]))
        p = c["pose"]
        got = mpc.vehicle_move(p[:4], p[4], p[5], cfg.Lf, c["dt"])
        assert np.allclose(got, c["moved"], rtol=0, atol=1e-12)
        assert np.allclose(clr.vehicle_move(p[0], p[1], p[2], p[3], p[4], p[5], cfg.Lf, c["dt"]), c["moved"], rtol=0, atol=1e-12)
    for c in gold["plant"]["throttle"]:
        cfg = mpc.config_from_json_text(json.dumps(refdata["configs"][c["config"]]))
        assert mpc.compute_throttle(cfg, c["accel"], c["target"]) == pytest.approx(c["throttle"], abs=1e-14)
        assert clr.compute_throttle(cfg.as_dict(), c["accel"], c["target"]) == pytest.approx(c["throttle"], abs=1e-14)
