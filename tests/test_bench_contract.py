"""bench.py's output contract, checked where no GPU is needed: the reference arm (`--impl reference`) runs the CPU
implementation of the path and must put exactly ONE JSON line on stdout -- everything else (library chatter such as
NCCL's version line in multi-GPU runs, warnings) goes to stderr -- with the keys a reader of the line relies on.
The last test (GPU) checks --dump-outputs and --steps against the product path itself."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + args, cwd=ROOT, env=e,
                          capture_output=True, text=True, timeout=600)


def test_reference_arm_prints_one_json_line():
    p = run_bench(["--impl", "reference", "--steps", "1", "--warmup", "0"])
    assert p.returncode == 0, p.stderr[-2000:]
    lines = [ln for ln in p.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, p.stdout[:2000]
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["unit"] == "solves/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["cpu_baseline"]["value"] == d["value"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "sample" in d["config"]["workload"]
    # the reference arm runs without the product: no CUDA library of this repository in the process
    assert all("mpc_b200" not in x for x in d["loaded_repo_libraries"]), d["loaded_repo_libraries"]
    assert any(x.startswith("oracle") for x in d["loaded_repo_libraries"])


def test_reference_arm_other_ranks_do_no_work():
    """Under torchrun (N > 1) rank 0 alone runs the reference arm; the other ranks exit 0 and print nothing."""
    p = run_bench(["--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "0"],
                  env={"RANK": "1", "LOCAL_RANK": "1", "WORLD_SIZE": "2"})
    assert p.returncode == 0, p.stderr[-2000:]
    assert p.stdout.strip() == ""


def test_our_arm_fails_loudly_without_a_gpu():
    """No CPU fallback: without a CUDA device the product arm must refuse, not fall back to the oracle."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = run_bench(["--steps", "1", "--warmup", "3"])
    assert p.returncode != 0
    assert p.stdout.strip() == ""
    assert "no CUDA device" in p.stderr


def test_steps_must_be_at_least_one():
    p = run_bench(["--steps", "0"])
    assert p.returncode != 0 and "--steps" in p.stderr
    assert p.stdout.strip() == ""


@pytest.mark.parametrize("cap,sampled", [(1 << 20, False), (20000, True)])
def test_dump_outputs_keep_a_fixed_sample_under_the_cap(tmp_path, monkeypatch, cap, sampled):
    """Every array is written in float64; past the size cap, all arrays keep the same seeded sample of problems (last
    axis) and its indices are written too, the same from run to run."""
    import bench
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", cap)
    n = 1000
    arrays = {"result": np.arange(9 * n, dtype=np.float64).reshape(9, n) / 7, "status": np.arange(n, dtype=np.int32)}
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), arrays)
    files = sorted(os.listdir(tmp_path / "a"))
    assert files == (["result.npy", "sample_index.npy", "status.npy"] if sampled else ["result.npy", "status.npy"])
    assert sum(os.path.getsize(tmp_path / "a" / f) for f in files) <= cap
    got = {f[:-4]: np.load(tmp_path / "a" / f) for f in files}
    for f in files:
        assert got[f[:-4]].dtype == np.float64 and np.array_equal(got[f[:-4]], np.load(tmp_path / "b" / f))
    idx = got["sample_index"].astype(np.int64) if sampled else np.arange(n)
    assert len(idx) > n // 10 and (np.diff(idx) > 0).all()
    assert np.array_equal(got["result"], arrays["result"][:, idx]) and np.array_equal(got["status"], idx)


@pytest.mark.gpu
def test_dump_outputs_hold_the_last_timed_step(mpc, stable_cfg, tmp_path):
    """--dump-outputs writes what the timed path computed in its last step: the same bits as one solve of the seed-0
    batch outside the bench.  The launch count of the timed region shows that --steps steps ran in it."""
    import torch
    B, K = 12288, 2                                   # >= LANE_MIN_BATCH: the lane-kernel chain
    p = run_bench(["--steps", str(K), "--warmup", "3", "--batch", str(B), "--only-timed", "--dump-outputs", str(tmp_path)])
    assert p.returncode == 0, p.stderr[-2000:]
    d = json.loads(p.stdout)
    b = mpc.workloads.batch_perturbed_states(B, 0, stable_cfg.as_dict())
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).cuda()
    N = stable_cfg.N
    res = torch.zeros(9, B, dtype=torch.float64, device="cuda")
    tx, ty = (torch.zeros(N, B, dtype=torch.float64, device="cuda") for _ in range(2))
    st, it = (torch.zeros(B, dtype=torch.int32, device="cuda") for _ in range(2))
    S = mpc.Solver(stable_cfg, 0)
    n0 = S.launches
    S.solve_batch_device(B, up(b["state"]), up(b["coeffs"]), up(b["yaw_lo"]), up(b["yaw_hi"]), res, tx, ty, None, st, it)
    torch.cuda.synchronize()
    per_solve = S.launches - n0
    S.close()
    assert d["steps"] == K and d["gpu_launches"] == K * per_solve
    want = {"result": res, "traj_x": tx, "traj_y": ty, "status": st, "iters": it}
    assert sorted(os.listdir(tmp_path)) == sorted(k + ".npy" for k in want)
    for k, v in want.items():
        got = np.load(tmp_path / (k + ".npy"))
        assert got.dtype == np.float64 and np.array_equal(got, v.cpu().numpy().astype(np.float64)), k
