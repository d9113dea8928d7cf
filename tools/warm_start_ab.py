"""Warm start against cold start on the BASELINE configs[1] batch (65,536 problems of config-stable, N = 10, dt = 0.1,
seed 0 -- the batch bench.py's headline line solves on rank 0), for several initial barrier parameters.

Three cases per mu_init:
  cold      every problem from the reference's start point (Ipopt's default initialisation)
  restart   the same problems again, warm-started from the cold solution (x, lambda, zl, zu)
  shifted   one control step later: each vehicle moved one dt along its predicted trajectory (the state of stage 1 of
            its cold solution) with a small seeded perturbation of cte, epsi and v, same road polynomial; solved cold
            and warm-started from mpc_warm_start_shift of the previous solution
Reported per case: iteration histogram, ms per batch (CUDA events around mpc_solve_batch, L2 flushed before every
timed solve with a 256 MiB write, as bench.py does), success fraction, and for the warm cases the largest difference
of the actuations from the cold solve of the same problems.

    python tools/warm_start_ab.py [--reps 10] [--mu 0.1,1e-2,1e-4,1e-6] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--mu", default="0.1,1e-2,1e-4,1e-6")
    ap.add_argument("--seed", type=int, default=0)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    import mpc_b200 as mpc
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    lines = []

    def say(s=""):
        print(s, flush=True)
        lines.append(s)

    dev = torch.device("cuda:0")
    try:
        smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:   # the measurement does not depend on it
        smi = "nvidia-smi unavailable (%s)" % e
    rd = mpc.workloads.reference_data()
    cfg = mpc.config_from_json_text(json.dumps(rd["configs"]["stable"]))
    N, B = cfg.N, args.batch
    nx, nl = 8 * N - 2, 6 * N
    b = mpc.workloads.batch_perturbed_states(B, args.seed, cfg.as_dict())
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).to(dev)
    coeffs, ylo, yhi = up(b["coeffs"]), up(b["yaw_lo"]), up(b["yaw_hi"])
    f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
    i32 = lambda *s: torch.zeros(*s, dtype=torch.int32, device=dev)
    result, full, status, iters = f64(9, B), f64(nx, B), i32(B), i32(B)
    lam, zl, zu = f64(nl, B), f64(nx, B), f64(nx, B)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    S = mpc.Solver(cfg, 0)
    S.set_dual_outputs(lam, zl, zu)
    say("warm start vs cold start, BASELINE configs[1]: %d problems, config-stable (N = %d, dt = %g), seed %d" % (B, N, cfg.dt, args.seed))
    say("device: %s | %s" % (torch.cuda.get_device_name(0), smi))
    say("timing: CUDA events around one mpc_solve_batch (AUTO kernel choice: lane-kernel chain), L2 flushed before each, "
        "median of %d after 2 warm-up solves" % args.reps)

    def solve(state):
        """timed solves of `state`; returns (median ms, outputs of the last solve)"""
        ts = []
        for k in range(2 + args.reps):
            flush.fill_(k & 0xFF)
            zl.zero_(); zu.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            S.solve_batch_device(B, state, coeffs, ylo, yhi, result, None, None, full, status, iters)
            e1.record()
            torch.cuda.synchronize()
            if k >= 2:
                ts.append(e0.elapsed_time(e1))
        out = {"result": result.cpu().numpy().T.copy(), "status": status.cpu().numpy().copy(),
               "iters": iters.cpu().numpy().copy(), "x": full.clone(), "lam": lam.clone(), "zl": zl.clone(), "zu": zu.clone()}
        return float(np.median(ts)), float(np.min(ts)), float(np.max(ts)), out

    def report(name, t, o, ref=None):
        it = o["iters"]
        ok = o["status"] == 1
        hist = np.bincount(it, minlength=1)
        hs = " ".join("%d:%d" % (k, c) for k, c in enumerate(hist) if c)
        extra = ""
        if ref is not None:
            both = ok & (ref["status"] == 1)
            d = np.abs(o["result"][both, :8] - ref["result"][both, :8]).max() if both.any() else float("nan")
            extra = " | max |actuations, stage-1 state - cold| %.2e" % d
        say("  %-34s %8.3f ms (min %.3f, max %.3f) | success %.5f | mean iters %6.3f | %s%s" % (
            name, t[0], t[1], t[2], ok.mean(), it.mean(), hs, extra))

    mus = [float(m) for m in args.mu.split(",")]
    state0 = up(b["state"])
    S.set_warm_start(None)
    *t, cold = solve(state0)
    say("")
    say("case 1, same problems")
    report("cold", t, cold)
    for mu in mus:
        S.set_warm_start(cold["x"], cold["lam"], cold["zl"], cold["zu"], mu_init=mu)
        *t, w = solve(state0)
        report("restart from the solution, mu_init %g" % mu, t, w, cold)
    # one control step later, in the same frame: stage 1 of each predicted trajectory, perturbed
    rng = np.random.default_rng(1000 + args.seed)
    s1 = cold["result"][:, :6].copy()
    s1[:, 4] += rng.normal(0.0, 0.02, B)      # cte [m]
    s1[:, 5] += rng.normal(0.0, 0.005, B)     # epsi [rad]
    s1[:, 3] += rng.normal(0.0, 0.1, B)       # v [m/s]
    state1 = up(s1)
    x0, lam0, zl0, zu0 = f64(nx, B), f64(nl, B), f64(nx, B), f64(nx, B)
    S.warm_start_shift(B, cold["x"], x0, cold["lam"], lam0, cold["zl"], zl0, cold["zu"], zu0)
    torch.cuda.synchronize()
    S.set_warm_start(None)
    *t, cold1 = solve(state1)
    say("")
    say("case 2, one control step later (stage-1 state + N(0, 0.02 m) cte, N(0, 0.005 rad) epsi, N(0, 0.1 m/s) v)")
    report("cold", t, cold1)
    for mu in mus:
        S.set_warm_start(x0, lam0, zl0, zu0, mu_init=mu)
        *t, w = solve(state1)
        report("shifted warm start, mu_init %g" % mu, t, w, cold1)
    for mu in mus[:1]:
        S.set_warm_start(x0, mu_init=mu)
        *t, w = solve(state1)
        report("shifted, primal only, mu_init %g" % mu, t, w, cold1)
    S.set_warm_start(None)
    S.close()
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
