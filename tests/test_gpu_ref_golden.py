"""GPU parity against the vectors of the reference's own sources (tests/golden/ref_golden.json, see
tests/test_ref_golden.py), through the C-ABI, the C++ host class and the drop-in MPC.cpp."""
import json
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
ABS_TOL, REL_TOL = 1e-4, 1e-6


@pytest.fixture(scope="module")
def gold():
    return json.load(open(os.path.join(GOLD, "ref_golden.json")))


def _cmp(res, ref):
    res, ref = np.asarray(res), np.asarray(ref)
    assert np.abs(res[:8] - ref[:8]).max() < ABS_TOL
    assert res[8] == pytest.approx(ref[8], rel=REL_TOL)


def test_testcpp_scenarios(gold, solver):
    for sc in gold["testcpp"]:
        run = sc["run"]
        for step in sc["steps"]:
            r = solver.solve_one(step["state"], run["coeffs"], run["yaw_lo"], run["yaw_hi"])
            assert r["status"] == step["status"] == 1
            _cmp(r["result"], step["result"])
            assert np.abs(r["traj_x"] - np.array(step["traj_x"])).max() < ABS_TOL
            assert np.abs(r["traj_y"] - np.array(step["traj_y"])).max() < ABS_TOL
            assert 0 <= r["iters"] - step["iters"] <= 1      # the reference build's count, or one more (DESIGN.md section 3)


def test_run_cases_all_configs(gold, mpc, refdata, kernel_kind):
    """pose + waypoints -> mpc_run_prepare -> CUDA solve -> mpc_run_finish == MPC::run of the reference."""
    for name in refdata["configs"]:
        cfg = mpc.config_from_json_text(json.dumps(refdata["configs"][name]))
        S = mpc.Solver(cfg, 0)
        S.set_kernel(kernel_kind)
        cases = [c for c in gold["run"] if c["config"] == name]
        prep = [mpc.run_prepare(cfg, c["pose"], c["ptsx"], c["ptsy"]) for c in cases]
        g = S.solve_batch_host(np.array([p["state"] for p in prep]), np.array([p["coeffs"] for p in prep]),
                               np.array([p["yaw_lo"] for p in prep]), np.array([p["yaw_hi"] for p in prep]))
        S.close()
        for i, (c, p) in enumerate(zip(cases, prep)):
            assert g["status"][i] == c["status"]
            if c["status"] != 1:
                continue
            out8 = mpc.run_finish(cfg, p["aux"], c["pose"][3], g["result"][i])
            assert np.abs(out8 - np.array(c["result"])).max() < ABS_TOL
            assert np.abs(g["traj_x"][i] - np.array(c["traj_x"])).max() < ABS_TOL
            assert np.abs(g["traj_y"][i] - np.array(c["traj_y"])).max() < ABS_TOL


def test_weight_sweep_cases(gold, solver):
    cs = gold["weights"]
    g = solver.solve_batch_host(np.array([c["state"] for c in cs]), np.array([c["coeffs"] for c in cs]),
                                np.array([c["yaw_lo"] for c in cs]), np.array([c["yaw_hi"] for c in cs]),
                                weights=np.array([c["weights"] for c in cs]))
    for i, c in enumerate(cs):
        assert g["status"][i] == c["status"] == 1
        _cmp(g["result"][i], c["result"])


def test_horizon_grid_cases(gold, mpc, refdata, kernel_kind):
    for c in gold["grid"]:
        cfg = mpc.config_from_json_text(json.dumps(dict(refdata["configs"]["stable"], N=c["N"], dt=c["dt"])))
        S = mpc.Solver(cfg, 0)
        S.set_kernel(kernel_kind)
        r = S.solve_batch_host(np.array([c["state"]]), np.array([c["coeffs"]]), np.array([c["yaw_lo"]]), np.array([c["yaw_hi"]]))
        S.close()
        assert r["status"][0] == c["status"] == 1
        _cmp(r["result"][0], c["result"])
        assert np.abs(r["traj_y"][0] - np.array(c["traj_y"])).max() < ABS_TOL


def test_restoration_cases_of_the_reference_sources(gold, mpc, refdata, kernel_kind):
    """Problems whose solve ENTERS Ipopt's restoration phase (N = 30, 40 at dt = 0.1), as solved by the reference's
    own MPC::solve / FG_eval compiled against the AD + interior-point stand-ins: same status, same optimum."""
    assert len(gold["resto"]) >= 8
    for c in gold["resto"]:
        assert c["oracle_n_resto"] >= 1 and c["status"] == 1
        cfg = mpc.config_from_json_text(json.dumps(dict(refdata["configs"]["stable"], N=c["N"], dt=c["dt"])))
        S = mpc.Solver(cfg, 0)
        S.set_kernel(kernel_kind)
        r = S.solve_batch_host(np.array([c["state"]]), np.array([c["coeffs"]]), np.array([c["yaw_lo"]]), np.array([c["yaw_hi"]]))
        S.close()
        assert r["status"][0] == c["status"]
        _cmp(r["result"][0], c["result"])
        assert np.abs(r["traj_x"][0] - np.array(c["traj_x"])).max() < ABS_TOL
        assert np.abs(r["traj_y"][0] - np.array(c["traj_y"])).max() < ABS_TOL


def _scenario_args(refdata, fx, tmp_path):
    path = tmp_path / "config-stable.json"
    path.write_text(json.dumps(refdata["configs"]["stable"]))
    args = [str(path), repr(fx["x"]), repr(fx["y"]), repr(fx["psi"]), repr(fx["v"])]
    for x, y in zip(fx["ptsx"], fx["ptsy"]):
        args += [repr(x), repr(y)]
    return args


def _check_scenario_output(text, sc):
    lines = [ln for ln in text.splitlines() if ln.startswith(("run", "solve"))]
    assert len(lines) == 26
    run = np.array([float(x) for x in lines[0].split("|")[0].split()[1:]])
    assert np.abs(run - np.array(sc["run"]["result"])).max() < ABS_TOL
    for ln, step in zip(lines[1:], sc["steps"]):
        vals = np.array([float(x) for x in ln.split("|")[0].split()[1:]])
        _cmp(vals, step["result"])


def test_cpp_host_class_runs_testcpp_scenario(gold, refdata, tmp_path):
    """include/mpc_b200.hpp (the C++ `MPC` with the reference's interface) compiled with g++ here and run:
    run() + 25 x solve() of src/test.cpp, all four fixtures."""
    exe = tmp_path / "test_host_mpc"
    pkg = os.path.join(ROOT, "carnd-mpc-project_b200")
    subprocess.run(["g++", "-O2", "-std=c++11", "-I", os.path.join(ROOT, "include"), "-o", str(exe),
                    os.path.join(ROOT, "tests", "cpp", "test_host_mpc.cpp"), "-L", pkg, "-lmpc_b200",
                    "-Wl,-rpath," + pkg, "-Wl,-rpath,/usr/local/cuda/lib64"], check=True)
    for fx, sc in zip(refdata["test_cpp_fixtures"], gold["testcpp"]):
        assert fx["name"] == sc["name"]
        out = subprocess.run([str(exe)] + _scenario_args(refdata, fx, tmp_path), capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stderr
        _check_scenario_output(out.stdout, sc)


def test_dropin_mpc_cpp_in_reference_tree(gold, refdata, tmp_path):
    """oracle/_ref/dropin_testcpp = the reference's Vehicle/RoadGeometry/utils/Config sources + OUR
    src/control/MPC.cpp (integration/reference_tree) + a driver making test.cpp's calls; built by
    `make -C oracle/ref_shim REF=<checkout of the original project>` (those sources are not part of this
    repository), run here on the GPU."""
    exe = os.path.join(ROOT, "oracle", "_ref", "dropin_testcpp")
    if not os.path.exists(exe):
        pytest.skip("oracle/_ref/dropin_testcpp not built (needs the original project's sources: make -C oracle/ref_shim REF=...)")
    for fx, sc in zip(refdata["test_cpp_fixtures"][:2], gold["testcpp"][:2]):
        out = subprocess.run([exe] + _scenario_args(refdata, fx, tmp_path), capture_output=True, text=True, timeout=300)
        assert out.returncode == 0, out.stderr
        _check_scenario_output(out.stdout, sc)
