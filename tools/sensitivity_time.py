"""Cost and use of mpc_solution_sensitivity on the BASELINE configs[1] batch (65,536 problems of config-stable, seed 0)
and the same generator at N = 32 and N = 64.

Per horizon: the solve with dual outputs, and the sensitivity with and without dfull, each timed with CUDA events
around one call, L2 flushed (256 MiB write) before every timed call, median of --reps after 2 warm-up calls; the bytes
each sensitivity call must move (inputs it reads, outputs it writes, at 8 bytes a double; the kernel's thread-private
rows come on top and are not counted), the bandwidth that implies against the 7.7 TB/s of HBM3e, and the ratio to
the solve.  Then the latency correction of the N = 10 batch: y, psi and v perturbed by N(0, 0.02 m), N(0, 0.005 rad)
and N(0, 0.1 m/s); delta0 and a0 of the re-solve against the first-order prediction u + S dx and the zeroth-order u.

    python tools/sensitivity_time.py [--reps 10] [--out FILE]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
HBM_TBS = 7.7


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batch", type=int, default=65536)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--horizons", default="10,32,64")
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
    B = args.batch
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    up = lambda a: torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).to(dev)
    f64 = lambda *s: torch.zeros(*s, dtype=torch.float64, device=dev)
    say("solution sensitivity (mpc_solution_sensitivity) vs solve, BASELINE configs[1] generator: %d problems, "
        "config-stable, seed %d" % (B, args.seed))
    say("device: %s | %s" % (torch.cuda.get_device_name(0), smi))
    say("timing: CUDA events around one call, L2 flushed before each, median of %d after 2 warm-up calls" % args.reps)

    def timed(fn):
        ts = []
        for k in range(2 + args.reps):
            flush.fill_(k & 0xFF)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            if k >= 2:
                ts.append(e0.elapsed_time(e1))
        return float(np.median(ts))

    keep = {}
    for N in [int(x) for x in args.horizons.split(",")]:
        js = dict(rd["configs"]["stable"], N=N)
        cfg = mpc.config_from_json_text(json.dumps(js))
        b = mpc.workloads.batch_perturbed_states(B, args.seed, cfg.as_dict())
        nx, nl = 8 * N - 2, 6 * N
        state, coeffs, ylo, yhi = up(b["state"]), up(b["coeffs"]), up(b["yaw_lo"]), up(b["yaw_hi"])
        result, full, lam, zl, zu = f64(9, B), f64(nx, B), f64(nl, B), f64(nx, B), f64(nx, B)
        status, iters = torch.zeros(B, dtype=torch.int32, device=dev), torch.zeros(B, dtype=torch.int32, device=dev)
        dres, dfull = f64(6, 9, B), f64(6, nx, B)
        S = mpc.Solver(cfg, 0)
        S.set_dual_outputs(lam, zl, zu)
        solve = lambda: S.solve_batch_device(B, state, coeffs, ylo, yhi, result, None, None, full, status, iters)
        t_solve = timed(solve)
        sens = lambda df: (lambda: S.solution_sensitivity(B, state, coeffs, ylo, yhi, full, lam, zl, zu, dres, df,
                                                          status=status))
        t_full = timed(sens(dfull))
        t_res = timed(sens(None))
        nan = torch.isnan(dres[0, 6]).sum().item()
        read = (6 + 5 + 2 + nx + nl + 2 * nx) * 8 * B + 4 * B
        wr_res, wr_full = 6 * 9 * 8 * B, 6 * nx * 8 * B
        say()
        say("N = %d: solve %.3f ms (mean iterations %.2f, success %.5f)" % (N, t_solve, iters.float().mean().item(),
                                                                           (status == 1).float().mean().item()))
        for name, t, by in (("sensitivity, dresult + dfull", t_full, read + wr_res + wr_full),
                            ("sensitivity, dresult only  ", t_res, read + wr_res)):
            say("  %s %.3f ms = %.1f %% of the solve | %.1f MB moved -> %.2f TB/s = %.1f %% of %.1f TB/s" % (
                name, t, 100.0 * t / t_solve, by / 1e6, by / t / 1e9, 100.0 * by / t / 1e9 / HBM_TBS, HBM_TBS))
        say("  problems with NaN sensitivity (status not a solution, or reduced Hessian not positive definite): %d" % nan)
        if N == 10:
            keep = dict(S=S, cfg=cfg, b=b, state=state, coeffs=coeffs, ylo=ylo, yhi=yhi, result=result.clone(),
                        dres=dres.clone(), status=status.clone())
        else:
            S.close()

    if keep:
        # latency correction: the state actually measured differs from the predicted one by dx
        S, b = keep["S"], keep["b"]
        rng = np.random.default_rng(1)
        dx = np.zeros((B, 6))
        dx[:, 1] = rng.normal(0.0, 0.02, B)
        dx[:, 2] = rng.normal(0.0, 0.005, B)
        dx[:, 3] = rng.normal(0.0, 0.1, B)
        st1 = up(b["state"] + dx)
        S.set_dual_outputs(None, None, None)
        r1 = f64(9, B)
        st_out = torch.zeros(B, dtype=torch.int32, device=dev)
        S.solve_batch_device(B, st1, keep["coeffs"], keep["ylo"], keep["yhi"], r1, None, None, None, st_out, None)
        torch.cuda.synchronize()
        u0 = keep["result"][6:8].cpu().numpy().T
        u1 = r1[6:8].cpu().numpy().T
        Sx = keep["dres"][:, 6:8, :].cpu().numpy().transpose(2, 1, 0)     # [B][2][6]
        pred = u0 + np.einsum("bjk,bk->bj", Sx, dx)
        ok = (keep["status"].cpu().numpy() == 1) & (st_out.cpu().numpy() == 1) & np.isfinite(pred).all(axis=1)
        say()
        say("latency correction, N = 10: y, psi, v perturbed by N(0, 0.02 m), N(0, 0.005 rad), N(0, 0.1 m/s); "
            "%d of %d problems solved both times" % (ok.sum(), B))
        for j, nm in ((0, "delta0 [rad]"), (1, "a0 [m/s^2]  ")):
            e1 = np.abs(pred[ok, j] - u1[ok, j])
            e0 = np.abs(u0[ok, j] - u1[ok, j])
            say("  %s first order u + S dx: median %.3g p99 %.3g | zeroth order u: median %.3g p99 %.3g" % (
                nm, np.median(e1), np.percentile(e1, 99), np.median(e0), np.percentile(e0, 99)))
        S.close()
    if args.out:
        with open(args.out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
