#!/usr/bin/env python
"""bench.py -- MPC solves/s on the BASELINE.json workloads.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--batch B] [--impl ours|reference]
                  [--workload batch64k|weights1M|grid256k|rollout8192x1000] [--dump-outputs DIR]

Default workload (the metric BASELINE.json is quoted on, configs[1]): a "step" is one pass of the hot path (one
`mpc_solve_batch` launch chain) over one batch of B = 65 536 synthetic problems per GPU -- perturbed poses along
lake_track_waypoints.csv, config-stable knobs (SURVEY.md 8d item 2).  With N GPUs (one process per GPU under
torchrun) every rank solves its own B problems (weak scaling; problems are independent, no collective in the solve,
one gather of result/status/iters per step, overlapped with the next step's solve); the same line also carries the
strong-scaling reading of the metric (64K problems in total, cut N ways).  Rank 0 prints ONE JSON line.

The other workloads are BASELINE.json configs[2..4] as written, sharded by batch index over the ranks:
  weights1M          1 048 576 problems with per-problem cost weights (config 4)
  grid256k           262 144 problems over the N x dt grid of examples/, one ragged launch per rank (config 3)
  rollout8192x1000   8192 vehicles x 1000 control steps, config-fast, 100 ms latency (config 5)

`--impl reference` times the reference's CPU path.  Ipopt/CppAD/MUMPS cannot be installed in this image
(DESIGN.md), so that arm runs oracle/_ref (the reference's own sources against AD / interior-point stand-ins) or the
plain-C oracle port on all host threads, on a bounded sample per step -- without importing the CUDA library.
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "MPC solves/sec (N=10 bicycle, batch 64K per GPU)"
UNIT = "solves/s"
FP64_NOMINAL_TFLOPS = 37.2     # 148 SMs x 64 DFMA/clk x 1.965 GHz x 2
PAIRS = [(10, .1), (20, .1), (30, .1), (40, .1), (10, .05), (20, .05), (30, .05), (40, .05), (50, .05), (10, .02), (20, .02),
         (30, .02), (40, .02), (50, .02)]     # submission-report.md:250-265


def f_iter(N):
    """Algorithmic FLOPs per interior-point iteration, SURVEY.md 8d / BASELINE.md section 4."""
    return (N - 1) * (1235 + 250) + 30 * (14 * N - 2)


BYTES_PER_SOLVE = lambda N: 104 + 8 * (9 + 2 * N) + 8   # in: 13 doubles; out: result+traj+status,iters


def load_workloads():
    """The synthetic-workload generator (pure numpy) WITHOUT importing the package's ctypes binding: the reference arm
    must not load the CUDA library."""
    spec = importlib.util.spec_from_file_location("_mpc_workloads", os.path.join(ROOT, "carnd-mpc-project_b200", "workloads.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


class NvmlSampler:
    """SM clock, power and throttle reasons polled through NVML every 2 ms DURING the timed region (a timed region of a few
    tens of milliseconds is over before an nvidia-smi process has printed its first line)."""

    def __init__(self, index):
        import pynvml
        self.nv = pynvml
        pynvml.nvmlInit()
        self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
        self.sm, self.pw, self.reasons, self.run = [], [], 0, False

    def start(self):
        self.run = True
        self.t = threading.Thread(target=self._poll, daemon=True)
        self.t.start()

    def _poll(self):
        nv = self.nv
        while self.run:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                self.pw.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1e3)
                self.reasons |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
            except Exception:
                break
            time.sleep(0.002)

    def stop(self):
        nv = self.nv
        self.run = False
        self.t.join(timeout=1)
        names = []
        for bit, nm in ((getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8), "hw_slowdown"),
                        (getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40), "hw_thermal_slowdown"),
                        (getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20), "sw_thermal_slowdown"),
                        (getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4), "sw_power_cap")):
            if self.reasons & int(bit):
                names.append(nm)
        try:
            mx = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
        except Exception:
            mx = None
        return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": mx, "power_w_max": max(self.pw) if self.pw else None,
                "samples": len(self.sm), "reasons": sorted(names), "source": "NVML, 2 ms poll"}


def make_sampler(index):
    try:
        return NvmlSampler(index)
    except Exception:
        return ClockSampler(index)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (fallback when NVML's Python binding is missing)."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "50"], stdout=subprocess.PIPE, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.06)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            p = [x.strip() for x in ln.split(",")]
            if len(p) < 7:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1])); pw.append(float(p[2]))
            except ValueError:
                continue
            for nm, v in zip(names, p[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def smi_index(local_rank):
    cvd = os.environ.get("CUDA_VISIBLE_DEVICES", "")
    if cvd:
        ids = [x.strip() for x in cvd.split(",") if x.strip()]
        if local_rank < len(ids) and ids[local_rank].isdigit():
            return int(ids[local_rank])
    return local_rank


def cpu_port(rd, batch, n_problems, threads):
    """The oracle (CPU restatement of the reference path) on the first n_problems of the batch."""
    from oracle import pyoracle as po
    ocfg = po.make_config(po.load_config_dict(rd["configs"]["stable"]))
    s = slice(0, n_problems)
    probs = po.problems_from_arrays(batch["state"][s], batch["coeffs"][s], batch["yaw_lo"][s], batch["yaw_hi"][s])
    t0 = time.perf_counter()
    out = po.solve_batch(ocfg, probs, threads)
    return time.perf_counter() - t0, out


def _ref_worker(job):
    """One worker process of the reference arm: the reference's own sources (oracle/_ref) keep global mutable
    Config statics, so parallelism is by process, one solve at a time per process."""
    js, state, coeffs, ylo, yhi, N = job
    from oracle import pyref as pr
    pr.config_load(js)
    t0 = time.perf_counter()
    ok, its = 0, 0
    for i in range(state.shape[0]):
        r = pr.solve(state[i], coeffs[i], ylo[i], yhi[i], N)
        ok += int(r["status"] == 1); its += r["iters"]
    return time.perf_counter() - t0, ok, its


def ref_build_run(rd, batch, n_problems, procs, pool):
    js = rd["configs"]["stable"]
    idx = np.array_split(np.arange(n_problems), procs)
    jobs = [(js, batch["state"][i], batch["coeffs"][i], batch["yaw_lo"][i], batch["yaw_hi"][i], js["N"]) for i in idx if len(i)]
    t0 = time.perf_counter()
    res = pool.map(_ref_worker, jobs)
    wall = time.perf_counter() - t0
    return wall, sum(r[1] for r in res), sum(r[2] for r in res)


def run_reference(args, rank):
    """The reference arm.  Where oracle/_ref exists (the reference's own MPC.cpp / Vehicle / RoadGeometry / Config
    compiled unmodified against the CppAD / Ipopt stand-ins of oracle/ref_shim -- built in the build container, it
    travels with the snapshot) that is what is timed: MPC::solve as the reference runs it, tape recording and AD
    sweeps per solve included, one process per host core.  Otherwise the plain-C oracle port.  Neither the package
    nor libmpc_b200.so is imported here."""
    if rank != 0:
        return
    from oracle import pyoracle as po
    wl = load_workloads()
    rd = wl.reference_data()
    cd = po.load_config_dict(rd["configs"]["stable"])
    batch = wl.batch_perturbed_states(args.batch, 0, cd)
    cores = os.cpu_count() or 1
    n_pilot = min(args.batch, 64 * cores)
    cpu_port(rd, batch, n_pilot, cores)
    t_pilot, _ = cpu_port(rd, batch, n_pilot, cores)
    per = t_pilot / n_pilot                                          # wall seconds per solve, all cores busy
    sample = int(max(cores, min(args.batch, 2.0 / max(per, 1e-9))))  # ~2 s of wall per step
    t_port, out_port = cpu_port(rd, batch, sample, cores)
    port_value = sample / t_port
    from oracle import pyref
    kind = "reference" if pyref.available() else "port"
    if kind == "reference":
        import multiprocessing as mp
        pool = mp.get_context("spawn").Pool(cores)
        w, _, _ = ref_build_run(rd, batch, 2 * cores, cores, pool)          # pilot (also pages the library in)
        w, _, _ = ref_build_run(rd, batch, 2 * cores, cores, pool)
        sample = int(max(cores, min(args.batch, 2.0 / max(w / (2 * cores), 1e-9))))
        for _ in range(args.warmup):
            ref_build_run(rd, batch, sample, cores, pool)
        times, ok, its = [], 0, 0
        for _ in range(args.steps):
            w, ok, its = ref_build_run(rd, batch, sample, cores, pool)
            times.append(w)
        pool.close()
        ok_frac, it_mean = ok / sample, its / sample
        sample_txt = ("first %d of the %d-problem batch per step, %d processes (one per host core); the reference's own "
                      "MPC::solve / FG_eval / Config sources (oracle/_ref, compiled unmodified against the CppAD/Ipopt "
                      "stand-ins of oracle/ref_shim: tape recorded per solve, AD Jacobian/Hessian, dense LDL^T; the "
                      "interior-point core is the oracle's restatement of Ipopt, which is not installable here)" % (sample, args.batch, cores))
    else:
        for _ in range(args.warmup):
            cpu_port(rd, batch, sample, cores)
        times = []
        for _ in range(args.steps):
            t, out = cpu_port(rd, batch, sample, cores)
            times.append(t)
        ok_frac, it_mean = float((out["status"] == 1).mean()), float(out["iters"].mean())
        sample_txt = ("first %d of the %d-problem batch per step, %d host threads, CPU restatement of "
                      "MPC::solve+Ipopt (oracle/mpc_oracle.c; Ipopt/CppAD not installable here)" % (sample, args.batch, cores))
    ms = 1e3 * float(np.mean(times))
    val = sample / (ms * 1e-3)
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[1]: batch 64K independent N=10 dt=0.1 solves, perturbed (cte, epsi, v), config-stable; "
                                   "each timed step solves a bounded sample of it: the first %d problems (about 2 s of wall on %d cores)" % (sample, cores),
                       "batch": args.batch, "batch_per_step": sample, "N": cd["N"], "dt": cd["dt"]},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample_txt},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "status_ok_frac": ok_frac, "iters_mean": it_mean, "host": {"cpu": cpu_model(), "logical_cpus": os.cpu_count()},
            "oracle_port_value": {"value": port_value, "unit": UNIT, "what": "the plain-C restatement (analytic derivatives, no tape) on the same cores, for comparison"},
            "loaded_repo_libraries": loaded_repo_libraries()}
    emit(line)


def loaded_repo_libraries():
    """Shared objects of this repository mapped into this process (the reference arm must show only oracle/ ones)."""
    libs = set()
    try:
        with open("/proc/self/maps") as f:
            for ln in f:
                p = ln.split()[-1] if ln.split() else ""
                if p.endswith(".so") and os.path.realpath(p).startswith(os.path.realpath(ROOT)):
                    libs.add(os.path.relpath(os.path.realpath(p), os.path.realpath(ROOT)))
    except OSError:
        pass
    return sorted(libs)


def cpu_model():
    """CPU model of the box (the host the cpu_baseline / reference arm runs on)."""
    try:
        with open("/proc/cpuinfo") as f:
            for ln in f:
                if ln.lower().startswith("model name"):
                    return ln.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


_REAL_STDOUT = None


def quiet_stdout():
    """The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version line at the first
    collective), so everything but that line goes to stderr: fd 1 is pointed at fd 2, the real stdout is kept aside."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


_T0 = time.time()


def log(msg):
    """progress on stderr (stdout carries the one JSON line)"""
    if os.environ.get("RANK", "0") == "0":
        sys.stderr.write("[bench %6.1fs] %s\n" % (time.time() - _T0, msg))
        sys.stderr.flush()


class Ctx:
    """torch / device / distributed plumbing of one rank."""

    def __init__(self):
        import torch
        import mpc_b200 as mpc
        self.torch, self.mpc = torch, mpc
        self.rank = int(os.environ.get("RANK", "0"))
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device -- the MPC solve has no CPU fallback")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        self.dist = None
        if self.world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)   # > 126 MB L2

    def up(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a)).to(self.dev)

    def sync_all(self):
        self.torch.cuda.synchronize()
        if self.dist:
            self.dist.barrier()
            self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.item()

    def sum_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return t.item()

    def close(self):
        if self.dist:
            self.dist.barrier()
            self.dist.destroy_process_group()


def timed_steps(ctx, step, steps, warmup, tail=None):
    """W untimed steps, then K steps each bracketed by CUDA events on the launching stream, L2 flushed between steps
    (outside the events); barrier + synchronize on both sides; returns (per-step ms on this rank, wall seconds)."""
    torch = ctx.torch
    for k in range(warmup):
        ctx.flush.fill_(1)
        step(k)
    if tail:
        tail()
    ctx.sync_all()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    t0 = time.perf_counter()
    for k in range(steps):
        ctx.flush.fill_(k & 0xFF)
        ev[k][0].record()
        step(k)
        ev[k][1].record()
    if tail:
        tail()
    ctx.sync_all()
    wall = time.perf_counter() - t0
    return [a.elapsed_time(b) for a, b in ev], wall


def status_hist(st):
    u, c = np.unique(np.asarray(st), return_counts=True)
    return {str(int(k)): int(v) for k, v in zip(u, c)}


DUMP_MAX_BYTES = 64 * 10 ** 6


def dump_outputs(out_dir, arrays):
    """--dump-outputs: write each array as out_dir/<name>.npy in float64 (status and iteration counts are exact there).
    The last axis of every array indexes the problem (or vehicle).  When all of them together would pass DUMP_MAX_BYTES,
    every array keeps the same fixed, seeded sample of problems, whose indices go to sample_index.npy."""
    arrays = {k: np.asarray(v.cpu().numpy() if hasattr(v, "cpu") else v, dtype=np.float64) for k, v in arrays.items()}
    n = next(iter(arrays.values())).shape[-1]
    assert all(a.shape[-1] == n for a in arrays.values()), {k: a.shape for k, a in arrays.items()}
    per_problem = 8 * sum(a.size // max(n, 1) for a in arrays.values())
    room = DUMP_MAX_BYTES - 128 * (len(arrays) + 1)          # an .npy header is 128 bytes
    if per_problem * n > room:
        keep = room // (per_problem + 8)
        idx = np.sort(np.random.default_rng(0).choice(n, keep, replace=False))
        arrays = {k: a[..., idx] for k, a in arrays.items()}
        arrays["sample_index"] = idx.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    for k, a in arrays.items():
        np.save(os.path.join(out_dir, k + ".npy"), np.ascontiguousarray(a))
    log("outputs of the last timed step written to %s: %s" % (out_dir, ", ".join(sorted(arrays))))


# ---------------------------------------------------------------------------------------------------------------
# BASELINE configs[2..4] as written, sharded over the ranks
# ---------------------------------------------------------------------------------------------------------------
def run_weights1M(ctx, args):
    """config 4: cost-weight sweep, 1 048 576 problems over all ranks, per-problem Config::weights."""
    mpc, torch = ctx.mpc, ctx.torch
    rd = mpc.workloads.reference_data()
    cfg = mpc.config_from_json_text(json.dumps(rd["configs"]["stable"]))
    cd = cfg.as_dict()
    Btot = args.batch if args.batch != 65536 else 1 << 20
    lo, hi = mpc.sharding.shard_bounds(Btot, ctx.rank, ctx.world)
    B = hi - lo
    base = mpc.workloads.batch_perturbed_states(4096, 0, cd)       # SURVEY 8d item 4: states from a 4096-element subset
    rng = np.random.default_rng(2)
    sel = rng.integers(0, 4096, Btot)[lo:hi]
    rngw = np.random.default_rng(1000 + ctx.rank)
    W = np.tile(np.array(cd["weights"]), (B, 1))
    W[:, 3] = np.exp(rngw.uniform(np.log(1), np.log(5000), B)); W[:, 4] = np.exp(rngw.uniform(np.log(1), np.log(5000), B))
    W[:, 1] = np.exp(rngw.uniform(np.log(1), np.log(1000), B)); W[:, 2] = rngw.choice([0.01, 0.1, 1, 10, 100], B)
    W[:, 6] = rngw.uniform(0, 1e4, B); W[:, 7] = rngw.uniform(0, 1e4, B)       # dead in the recorded tape
    ins = [ctx.up(base["state"][sel].T), ctx.up(base["coeffs"][sel].T), ctx.up(base["yaw_lo"][sel]), ctx.up(base["yaw_hi"][sel])]
    Wd = ctx.up(W.T)
    res = torch.zeros(9, B, dtype=torch.float64, device=ctx.dev)
    st = torch.zeros(B, dtype=torch.int32, device=ctx.dev); it = torch.zeros(B, dtype=torch.int32, device=ctx.dev)
    S = mpc.Solver(cfg, ctx.local_rank)
    step = lambda k: S.solve_batch_device(B, *ins, res, None, None, None, st, it, weights=Wd)
    ms, _ = timed_steps(ctx, step, args.steps, max(3, args.warmup))
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, {"result": res, "status": st, "iters": it})
    ms_step = ctx.max_over_ranks(sum(ms)) / args.steps
    iters_sum = ctx.sum_over_ranks(float(it.sum().item()))
    ok = ctx.sum_over_ranks(float((st == 1).sum().item())) / Btot
    fp64 = mpc.measure_fp64_peak(ctx.local_rank)
    tf = f_iter(cfg.N) * iters_sum / (ms_step * 1e-3) / 1e12
    line = {"metric": "MPC solves/sec (cost-weight sweep, 1M problems, N=10)", "value": Btot / (ms_step * 1e-3), "unit": UNIT,
            "n_gpus": ctx.world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[3]: cost-weight sweep (delta, delta-rate, epsi, velocity weights; acceleration weights varied too -- dead), "
                                   "%d problems in total, contiguous shards over %d rank(s), states from a 4096-element subset of the 64K batch" % (Btot, ctx.world),
                       "problems_total": Btot, "problems_per_gpu": B, "N": cfg.N, "l2": "flushed between timed steps"},
            "roofline": {"bound": "fp64_fma", "achieved": tf / ctx.world, "peak": fp64, "unit": "TFLOP/s per GPU", "frac": tf / ctx.world / fp64,
                         "frac_of_nominal": tf / ctx.world / FP64_NOMINAL_TFLOPS, "flops_model": "sum_b iters_b * F_iter(10)"},
            "status_ok_frac": ok, "status_hist_rank0": status_hist(st.cpu().numpy()), "iters_max_rank0": int(it.max().item()),
            "gpu_launches": int(S.launches)}
    S.close()
    return line


def run_grid256k(ctx, args):
    """config 3: N x dt grid of examples/ (submission-report.md:250-265), 262 144 problems, one ragged launch per rank."""
    mpc, torch = ctx.mpc, ctx.torch
    rd = mpc.workloads.reference_data()
    js = rd["configs"]["stable"]
    cd = mpc.config_from_json_text(json.dumps(js)).as_dict()
    Btot = args.batch if args.batch != 65536 else 262144
    lo, hi = mpc.sharding.shard_bounds(Btot, ctx.rank, ctx.world)
    B = hi - lo
    b = mpc.workloads.batch_perturbed_states(Btot, 1, cd)
    pick = np.random.default_rng(1).integers(0, len(PAIRS), Btot)
    Nall = np.array([PAIRS[k][0] for k in pick], dtype=np.int32); dtall = np.array([PAIRS[k][1] for k in pick])
    ins = [ctx.up(b["state"][lo:hi].T), ctx.up(b["coeffs"][lo:hi].T), ctx.up(b["yaw_lo"][lo:hi]), ctx.up(b["yaw_hi"][lo:hi])]
    Np, dtp = ctx.up(Nall[lo:hi]), ctx.up(dtall[lo:hi])
    cfg = mpc.config_from_json_text(json.dumps(dict(js, N=50)))
    S = mpc.Solver(cfg, ctx.local_rank)
    res = torch.zeros(9, B, dtype=torch.float64, device=ctx.dev)
    st = torch.zeros(B, dtype=torch.int32, device=ctx.dev); it = torch.zeros(B, dtype=torch.int32, device=ctx.dev)
    step = lambda k: S.solve_batch_device(B, *ins, res, None, None, None, st, it, N_per=Np, dt_per=dtp)
    ms, _ = timed_steps(ctx, step, args.steps, max(3, args.warmup))
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, {"result": res, "status": st, "iters": it})
    ms_step = ctx.max_over_ranks(sum(ms)) / args.steps
    stn, itn = st.cpu().numpy(), it.cpu().numpy()
    flops = float(sum(f_iter(n) * itn[Nall[lo:hi] == n].sum() for n in (10, 20, 30, 40, 50)))
    flops = ctx.sum_over_ranks(flops)
    ok = ctx.sum_over_ranks(float((stn == 1).sum())) / Btot
    fp64 = mpc.measure_fp64_peak(ctx.local_rank)
    tf = flops / (ms_step * 1e-3) / 1e12
    cells = {}
    for (n, d) in PAIRS:
        m = (Nall[lo:hi] == n) & (dtall[lo:hi] == d)
        cells["N=%d dt=%g" % (n, d)] = {"ok_frac": float((stn[m] == 1).mean()), "iters_p50": float(np.percentile(itn[m], 50)), "iters_max": int(itn[m].max())}
    line = {"metric": "MPC solves/sec (horizon/timestep grid, 256K problems, N in 10..50)", "value": Btot / (ms_step * 1e-3), "unit": UNIT,
            "n_gpus": ctx.world, "steps": args.steps, "warmup": max(3, args.warmup), "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[2]: horizon/timestep sweep N in {10..50} x dt in {0.02,0.05,0.1} (the 14 cells of examples/), %d problems in total, "
                                   "contiguous shards over %d rank(s), one ragged launch per rank (per-problem N and dt)" % (Btot, ctx.world),
                       "problems_total": Btot, "problems_per_gpu": B, "l2": "flushed between timed steps"},
            "roofline": {"bound": "fp64_fma", "achieved": tf / ctx.world, "peak": fp64, "unit": "TFLOP/s per GPU", "frac": tf / ctx.world / fp64,
                         "frac_of_nominal": tf / ctx.world / FP64_NOMINAL_TFLOPS, "flops_model": "sum_b iters_b * F_iter(N_b)"},
            "status_ok_frac": ok, "status_hist_rank0": status_hist(stn), "iters_max_rank0": int(itn.max()), "cells_rank0": cells,
            "gpu_launches": int(S.launches)}
    S.close()
    return line


def run_rollout(ctx, args):
    """config 5: 100 ms latency-compensated closed-loop rollouts, 8192 vehicles x 1000 control steps, config-fast."""
    mpc, torch = ctx.mpc, ctx.torch
    rd = mpc.workloads.reference_data()
    cfg = mpc.config_from_json_text(json.dumps(rd["configs"]["fast"]))
    cd = cfg.as_dict()
    Vtot = args.batch if args.batch != 65536 else 8192
    T = args.rollout_steps
    lo, hi = mpc.sharding.shard_bounds(Vtot, ctx.rank, ctx.world)
    V = hi - lo
    bv = mpc.workloads.batch_perturbed_states(Vtot, 3, cd)
    veh0 = np.stack([bv["px"], bv["py"], bv["psi"], np.clip(bv["v"], 8, 30), np.zeros(Vtot), np.zeros(Vtot)])[:, lo:hi]
    seg0 = bv["segment"].astype(np.int32)[lo:hi]
    wx, wy = ctx.up(np.array(rd["waypoints"]["x"])), ctx.up(np.array(rd["waypoints"]["y"]))
    rec = torch.zeros(T, 8, V, dtype=torch.float64, device=ctx.dev)
    S = mpc.Solver(cfg, ctx.local_rank)
    state = {}

    def step(k):
        state["veh"], state["seg"] = ctx.up(veh0), ctx.up(seg0)
        state["pend"] = torch.zeros(2, V, dtype=torch.float64, device=ctx.dev)
        S.rollout_device(V, T, wx, wy, state["veh"], state["seg"], state["pend"], 0.1, 0.02, rec)

    n0 = S.launches
    ms, _ = timed_steps(ctx, step, args.steps, 1)
    if args.dump_outputs and ctx.rank == 0:
        dump_outputs(args.dump_outputs, {"rec": rec, "veh": state["veh"], "seg": state["seg"], "pending": state["pend"]})
    launches = (S.launches - n0) // (args.steps + 1)
    ms_roll = ctx.max_over_ranks(sum(ms)) / args.steps
    r = rec.cpu().numpy()
    ok = ctx.sum_over_ranks(float((r[:, 6] == 1).sum())) / (Vtot * T)
    iters_sum = ctx.sum_over_ranks(float(r[:, 7].sum()))
    fp64 = mpc.measure_fp64_peak(ctx.local_rank)
    tf = f_iter(cfg.N) * iters_sum / (ms_roll * 1e-3) / 1e12
    line = {"metric": "closed-loop vehicle-steps/sec (8192 vehicles x 1000 steps, config-fast, 100 ms latency)", "value": Vtot * T / (ms_roll * 1e-3),
            "unit": "vehicle-steps/s", "n_gpus": ctx.world, "steps": args.steps, "warmup": 1, "ms_per_step": ms_roll, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "configs[4]: 100 ms latency-compensated closed-loop rollouts, %d vehicles x %d control steps of 0.1 s (config-fast, tau_solve 0.02 s), "
                                   "vehicles sharded over %d rank(s); a 'step' of this line is one whole rollout" % (Vtot, T, ctx.world),
                       "vehicles_total": Vtot, "vehicles_per_gpu": V, "control_steps": T, "kernel": "mpc_rollout_kernel (one launch per rollout)" if launches == 1 else "three launches per control step"},
            "ms_per_control_step": ms_roll / T, "launches_per_rollout": int(launches),
            "roofline": {"bound": "fp64_fma", "achieved": tf / ctx.world, "peak": fp64, "unit": "TFLOP/s per GPU", "frac": tf / ctx.world / fp64,
                         "frac_of_nominal": tf / ctx.world / FP64_NOMINAL_TFLOPS, "flops_model": "sum over solves iters * F_iter(10)"},
            "status_ok_frac": ok, "median_abs_cte_final_m_rank0": float(np.median(np.abs(r[-1, 0]))), "mean_speed_final_rank0": float(r[-1, 2].mean()),
            "gpu_launches": int(S.launches - n0)}
    S.close()
    return line


# ---------------------------------------------------------------------------------------------------------------
# the headline: configs[1]
# ---------------------------------------------------------------------------------------------------------------
def run_batch64k(ctx, args):
    mpc, torch = ctx.mpc, ctx.torch
    world, rank, dev = ctx.world, ctx.rank, ctx.dev
    B = args.batch
    rd = mpc.workloads.reference_data()
    cfg = mpc.config_from_json_text(json.dumps(rd["configs"]["stable"]))
    batch = mpc.workloads.batch_perturbed_states(B, rank, cfg.as_dict())     # rank r solves the seed-r batch (rank 0 = SURVEY's seed 0)
    N = cfg.N
    upT = lambda a: ctx.up(a.T if a.ndim == 2 else a)
    state, coeffs, ylo, yhi = upT(batch["state"]), upT(batch["coeffs"]), upT(batch["yaw_lo"]), upT(batch["yaw_hi"])
    # outputs double-buffered (--gather overlap: the gather of step k runs on NCCL's stream beside the solve of step k+1).
    # result[9][B] and status/iters[2][B] share one buffer of 10 x B x 8 bytes, so the exchange is ONE collective.
    nbuf = 2 if world > 1 else 1
    packed = [torch.zeros(10, B, dtype=torch.float64, device=dev) for _ in range(nbuf)]
    result = [p[:9] for p in packed]
    si = [p[9].view(torch.int32).view(2, B) for p in packed]       # status, iters
    tx = torch.zeros(N, B, dtype=torch.float64, device=dev)
    ty = torch.zeros(N, B, dtype=torch.float64, device=dev)
    g_out = [torch.zeros(world, 10, B, dtype=torch.float64, device=dev) for _ in range(nbuf)] if world > 1 else None
    pending = [None] * nbuf
    serial_gather = args.gather == "serial"
    S = mpc.Solver(cfg, ctx.local_rank)
    log('batch64k: inputs resident, B=%d world=%d' % (B, world))

    def step(k):
        j = k % nbuf
        if pending[j] is not None:             # the buffers of step k - 2 are about to be overwritten
            for w in pending[j]:
                w.wait()
            pending[j] = None
        S.solve_batch_device(B, state, coeffs, ylo, yhi, result[j], tx, ty, None, si[j][0], si[j][1])
        if world > 1 and not os.environ.get("MPC_BENCH_NO_GATHER"):   # the only exchange the path has: result / status / iters of every shard, after its solve
            # (MPC_BENCH_NO_GATHER: development switch -- how much of a step is the exchange?  The line then says so.)
            pending[j] = [ctx.dist.all_gather_into_tensor(g_out[j].view(-1), packed[j].view(-1), async_op=True)]
            if serial_gather:
                # the solve's persistent grid wants every SM: the next solve starts after the gather kernels have left
                for w in pending[j]:
                    w.wait()
                pending[j] = None

    def drain():
        for j in range(nbuf):
            if pending[j] is not None:
                for w in pending[j]:
                    w.wait()
                pending[j] = None

    sampler = make_sampler(smi_index(ctx.local_rank))
    for k in range(args.warmup):
        ctx.flush.fill_(1)
        step(k)
    drain()
    ctx.sync_all()
    sampler.start()
    launches0 = S.launches
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    ev_all = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
    t_wall0 = time.perf_counter()
    ev_all[0].record()
    for k in range(args.steps):
        ctx.flush.fill_(k & 0xFF)           # L2 flush between timed iterations
        ev[k][0].record()
        step(k)
        ev[k][1].record()
    drain()                                 # the last gathers are inside the timed region
    ev_all[1].record()
    ctx.sync_all()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    launches = S.launches - launches0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    flush_ms = 0.0
    if world > 1:
        # whole timed region on the device (solves + overlapped gathers + the last gather) minus the L2 flushes
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for k in range(8):
            ctx.flush.fill_(k)
        e1.record(); torch.cuda.synchronize()
        flush_ms = e0.elapsed_time(e1) / 8
        region_ms = ev_all[0].elapsed_time(ev_all[1]) - flush_ms * args.steps
        ms_per_step = ctx.max_over_ranks(region_ms) / args.steps
        per_rank = torch.zeros(world, dtype=torch.float64, device=dev)
        ctx.dist.all_gather_into_tensor(per_rank, torch.tensor([sum(step_ms) / args.steps], dtype=torch.float64, device=dev))
        per_rank_ms = [float(x) for x in per_rank.cpu().numpy()]
    else:
        ms_per_step = sum(step_ms) / args.steps
    value = B * world / (ms_per_step * 1e-3)
    jl = (args.steps - 1) % nbuf
    it = si[jl][1].cpu().numpy()
    st = si[jl][0].cpu().numpy()
    res_last = result[jl]
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"result": res_last, "traj_x": tx, "traj_y": ty, "status": st, "iters": it})
    flops_per_launch = float(f_iter(N)) * float(it.sum())
    kernel_ms = float(np.mean(step_ms))      # the launches of one solve on this rank

    log('timed region done: %.3f ms per step' % ms_per_step)
    # ---- strong scaling (the metric as written: 64K problems in total at 1/2/4/8 GPUs)
    strong = None
    if world > 1 and not args.only_timed:
        Bs_lo, Bs_hi = mpc.sharding.shard_bounds(B, rank, world)
        Bs = Bs_hi - Bs_lo
        b0 = mpc.workloads.batch_perturbed_states(B, 0, cfg.as_dict())
        s_in = [upT(b0["state"][Bs_lo:Bs_hi]), upT(b0["coeffs"][Bs_lo:Bs_hi]), upT(b0["yaw_lo"][Bs_lo:Bs_hi]), upT(b0["yaw_hi"][Bs_lo:Bs_hi])]
        s_res = torch.zeros(9, Bs, dtype=torch.float64, device=dev)
        s_si = torch.zeros(2, Bs, dtype=torch.int32, device=dev)
        s_g = torch.zeros(world, 9, Bs, dtype=torch.float64, device=dev) if B % world == 0 else None

        def sstep(k):
            S.solve_batch_device(Bs, *s_in, s_res, None, None, None, s_si[0], s_si[1])
            if s_g is not None:
                ctx.dist.all_gather_into_tensor(s_g.view(-1), s_res.view(-1))

        ms_s, _ = timed_steps(ctx, sstep, args.steps, 3)
        ms_strong = ctx.max_over_ranks(sum(ms_s)) / args.steps
        strong = {"value": B / (ms_strong * 1e-3), "unit": UNIT, "ms_per_step": ms_strong, "problems_total": B, "problems_per_gpu": Bs,
                  "what": "the same 64K batch (seed 0) cut into contiguous shards over the ranks, gather of result included; "
                          "below ~9K problems per GPU the coop kernel runs (latency-bound), so this does not scale like the weak reading"}

    log('e2e leg')
    # ---- e2e: the reference-facing call with HOST buffers (pinned), H2D + solve + D2H per step
    pin = lambda a: torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).pin_memory().numpy()
    h_state, h_coef, h_ylo, h_yhi = pin(batch["state"]), pin(batch["coeffs"]), pin(batch["yaw_lo"]), pin(batch["yaw_hi"])
    h_res = torch.zeros(9, B, dtype=torch.float64).pin_memory().numpy()
    h_tx = torch.zeros(N, B, dtype=torch.float64).pin_memory().numpy()
    h_ty = torch.zeros(N, B, dtype=torch.float64).pin_memory().numpy()
    h_st = torch.zeros(B, dtype=torch.int32).pin_memory().numpy()
    h_it = torch.zeros(B, dtype=torch.int32).pin_memory().numpy()
    L = mpc.lib()
    ptr = lambda a: a.ctypes.data

    def e2e_step():
        rc = L.mpc_solve_batch_host(S._h, B, ptr(h_state), ptr(h_coef), ptr(h_ylo), ptr(h_yhi), None, None, None,
                                    ptr(h_res), ptr(h_tx), ptr(h_ty), None, ptr(h_st), ptr(h_it))
        if rc != 0:
            raise SystemExit("mpc_solve_batch_host failed: %d %s" % (rc, L.mpc_last_error().decode()))

    for _ in range(0 if args.only_timed else 3):
        e2e_step()
    ctx.sync_all()
    e2e_t = []
    for k in range(0 if args.only_timed else args.steps):
        ctx.flush.fill_(k & 0xFF)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e2e_step()                      # returns after the D2H copies completed
        e2e_t.append(time.perf_counter() - t0)
    ctx.sync_all()
    e2e_tot = ctx.max_over_ranks(sum(e2e_t))
    e2e_value = B * world / (e2e_tot / args.steps) if e2e_t else None
    assert args.only_timed or np.allclose(h_res, res_last.cpu().numpy(), rtol=0, atol=0), "host-path result differs from device path"
    h2d = 13 * 8 * B
    d2h = (9 + 2 * N) * 8 * B + 8 * B

    if rank != 0:
        S.close()
        return None
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    fp64_peak = mpc.measure_fp64_peak(ctx.local_rank)
    traffic, traffic_src = None, None
    try:   # dram__bytes_read.sum + dram__bytes_write.sum of the dominant kernel at this batch, from the committed ncu capture
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            tj = json.load(f)
        if tj.get("batch") == B and tj.get("N") == N:
            traffic, traffic_src = tj["dram_bytes_per_launch"], "static: " + str(tj.get("source"))
    except Exception:
        pass
    achieved_tf = flops_per_launch / (kernel_ms * 1e-3) / 1e12
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    hbm_gbs = BYTES_PER_SOLVE(N) * B / (kernel_ms * 1e-3) / 1e9
    lane = B >= mpc.LANE_MIN_BATCH
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "configs[1]: batch 64K independent N=10 dt=0.1 solves from perturbed (cte, epsi, v), config-stable, seed=rank",
                   "batch_per_gpu": B, "N": N, "dt": cfg.dt, "l2": "flushed between timed steps (256 MiB write)",
                   "sharding": ("independent batch shard per rank, no collective in the solve; per step ONE all_gather of result[9][B] + "
                                "status/iters[2][B] (one packed buffer) after the solve, " + ("finished before the next step's solve starts (the solve's persistent grid wants every SM; "
                                "NCCL kernels resident beside it cost more than they hide: DESIGN.md section 7); " if serial_gather else "overlapped with the next step's solve (double-buffered); ") +
                                "ms_per_step = device time of the whole timed region (gathers included, L2 flushes subtracted) / steps, max over ranks") if world > 1 else "single GPU"},
        "roofline": {"bound": "fp64_fma", "achieved": achieved_tf, "peak": fp64_peak, "unit": "TFLOP/s",
                     "frac": achieved_tf / fp64_peak if fp64_peak else None, "frac_of_nominal": achieved_tf / FP64_NOMINAL_TFLOPS,
                     "peak_nominal": FP64_NOMINAL_TFLOPS, "traffic": traffic, "traffic_source": traffic_src,
                     "kernel": ("mpc_lane_kernel<10,1,false> (one problem per lane; dominant) + the launches that finish its tail: up to 3x mpc_lane_kernel<10,1,true> "
                                "(parked problems, 32 to a warp; each returns at once when at most 8192 are parked) + mpc_coop_resume_kernel<10> (every branch of the "
                                "algorithm: also the problems the lane kernel hands over); %d launches per step, kernel_ms is their sum" % (launches // args.steps))
                               if lane else "mpc_coop_kernel<10> (one problem per group of 16 lanes)",
                     "peak_source": "measured in this run by mpc_measure_fp64_peak (DFMA chains; MEASURED_PEAKS.json has no FP64 figure); peak_nominal = 148 SMs x 64 DFMA/clk x 1.965 GHz x 2",
                     "flops_per_launch": flops_per_launch, "flops_model": "sum_b iters_b * F_iter(N), F_iter(10)=17505 (SURVEY.md 8d)",
                     "kernel_ms": kernel_ms},
        "roofline_hbm": {"bound": "hbm", "achieved": hbm_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": hbm_gbs / hbm_peak,
                         "bytes_per_solve": BYTES_PER_SOLVE(N),
                         "peak_source": "MEASURED_PEAKS.json" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"},
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * e2e_tot / args.steps, "api": "mpc_solve_batch_host (pinned host buffers: inputs read in place over PCIe by the kernels; outputs copied back on a second stream beside the chain's final launch, whose problems a small kernel then rewrites in the host arrays)"},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "wall_ms_per_step_incl_flush": 1e3 * t_wall / args.steps,
        "iters": {"mean": float(it.mean()), "p50": float(np.percentile(it, 50)), "p99": float(np.percentile(it, 99)), "max": int(it.max()),
                  "hist": {str(k): int(c) for k, c in enumerate(np.bincount(np.asarray(it, dtype=np.int64).clip(0))) if c}},
        "host": {"cpu": cpu_model(), "logical_cpus": os.cpu_count()},
        "status_ok_frac": float((st == 1).mean()), "status_hist": status_hist(st),
    }
    if os.environ.get("MPC_BENCH_NO_GATHER"):
        line["config"]["sharding"] = "DEVELOPMENT RUN WITHOUT THE GATHER (MPC_BENCH_NO_GATHER): not a bench line"
    if world > 1:
        # rank r solves the seed-r batch: the ranks' own solve times differ with their longest-running problem; the job
        # runs at the pace of the slowest
        line["per_rank_solve_ms"] = per_rank_ms
    if strong:
        line["strong_scaling"] = strong
    if world == 1 and not args.no_latency:
        log('latency leg')
        one = mpc.Solver(cfg, ctx.local_rank)
        lat = []
        for k in range(1200):
            i = k % B
            t0 = time.perf_counter()
            one.solve_one(batch["state"][i], batch["coeffs"][i], batch["yaw_lo"][i], batch["yaw_hi"][i])
            lat.append(time.perf_counter() - t0)
        lat = np.array(lat[200:]) * 1e6
        n50, n99 = one.measure_solve_latency(batch["state"][:1000], batch["coeffs"][:1000], batch["yaw_lo"][:1000], batch["yaw_hi"][:1000], 1000, 200)
        line["latency"] = {"p50_us": float(np.percentile(lat, 50)), "p99_us": float(np.percentile(lat, 99)),
                           "native_p50_us": n50, "native_p99_us": n99,
                           "what": "mpc_solve_one host call -> result (B=1; inputs and result in mapped pinned host memory, one kernel launch + stream sync); p50/p99 through the Python binding, native_* from a C++ loop (mpc_measure_solve_latency) on the same 1000 problems", "batch_ms": ms_per_step}
        one.close()
        line["latency"].update(dropin_latency(rd))
    if world == 1 and not args.no_extras:
        log('extras')
        line["extras"] = extras(ctx, rd, fp64_peak)
    if world == 1 and not args.no_cpu_baseline:
        log('cpu_baseline leg')
        cores = os.cpu_count() or 1
        t_pilot, _ = cpu_port(rd, batch, min(B, 4 * cores), cores)
        per = t_pilot / min(B, 4 * cores)
        sample = int(max(cores, min(B, 10.0 / max(per, 1e-9))))          # ~10 s of wall on all cores
        t, out = cpu_port(rd, batch, sample, cores)
        gres = res_last.cpu().numpy().T[:sample]
        dmax = float(np.abs(gres - out["result"])[:, :8].max())
        line["cpu_baseline"] = {"value": sample / t, "unit": UNIT, "cores": cores, "kind": "port",
                                "sample": "first %d problems of the same batch, one solve per host thread (%d threads), %.1f s; CPU restatement "
                                          "oracle/mpc_oracle.c (dense LDL^T), not Ipopt+CppAD+MUMPS" % (sample, cores, t),
                                "max_abs_diff_vs_gpu": dmax, "status_equal": bool(np.array_equal(st[:sample], out["status"])),
                                "iters_equal_frac": float((it[:sample] == out["iters"]).mean()),
                                "iters_diff_hist_gpu_minus_cpu": {str(int(k)): int(c) for k, c in zip(*np.unique(it[:sample].astype(np.int64) - out["iters"].astype(np.int64), return_counts=True))}}
    S.close()
    return line


def dropin_latency(rd):
    """p50/p99 of MPC::solve measured INSIDE the drop-in (integration/reference_tree/src/control/MPC.cpp built against the
    reference's own headers: oracle/_ref/dropin_testcpp, present where the build container made it)."""
    exe = os.path.join(ROOT, "oracle", "_ref", "dropin_testcpp")
    if not os.path.exists(exe):
        return {"dropin_p50_us": None, "dropin_note": "oracle/_ref/dropin_testcpp not present"}
    import tempfile
    fx = rd["test_cpp_fixtures"][0]
    with tempfile.NamedTemporaryFile("w", suffix=".json", delete=False) as f:
        json.dump(rd["configs"]["stable"], f)
        path = f.name
    try:
        a = [exe, path, repr(fx["x"]), repr(fx["y"]), repr(fx["psi"]), repr(fx["v"])]
        for x, y in zip(fx["ptsx"], fx["ptsy"]):
            a += [repr(x), repr(y)]
        out = subprocess.run(a + ["latency", "2000"], capture_output=True, text=True, timeout=120)
        for ln in out.stdout.splitlines():
            if ln.startswith("latency_us"):
                p = ln.split()
                return {"dropin_p50_us": float(p[2]), "dropin_p99_us": float(p[4]),
                        "dropin_what": "MPC::solve of the reference's class (src/control/MPC.h) with integration/reference_tree/src/control/MPC.cpp swapped in, timed inside a C++ program built against the reference's headers; the solver handle is kept across calls"}
        return {"dropin_p50_us": None, "dropin_note": "no latency line (rc %d): %s" % (out.returncode, out.stderr[-200:])}
    except Exception as e:   # noqa: BLE001
        return {"dropin_p50_us": None, "dropin_note": str(e)[:200]}
    finally:
        os.unlink(path)


def extras(ctx, rd, fp64_peak=None):
    """On ONE GPU, informational (the headline stays configs[1]): a 1M batch (the steady-state rate without the tail) and
    one GPU's share of configs[2..4] (the --workload runs are those configs as written)."""
    mpc, torch, dev = ctx.mpc, ctx.torch, ctx.dev

    def timed(fn, reps=3):
        best = 1e9
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); fn(); e1.record(); torch.cuda.synchronize()
            best = min(best, e0.elapsed_time(e1))
        return best

    out = {}
    js = rd["configs"]["stable"]
    cfg = mpc.config_from_json_text(json.dumps(js))
    cd = cfg.as_dict()
    B = 1 << 20
    b = mpc.workloads.batch_perturbed_states(B, 0, cd)
    ins = [ctx.up(b["state"].T), ctx.up(b["coeffs"].T), ctx.up(b["yaw_lo"]), ctx.up(b["yaw_hi"])]
    res = torch.zeros(9, B, dtype=torch.float64, device=dev)
    st = torch.zeros(B, dtype=torch.int32, device=dev); it = torch.zeros(B, dtype=torch.int32, device=dev)
    S = mpc.Solver(cfg, ctx.local_rank)
    ms = timed(lambda: S.solve_batch_device(B, *ins, res, None, None, None, st, it))
    out["batch_1M"] = {"solves_per_s": B / ms * 1e3, "ms": ms, "status_ok_frac": float((st == 1).float().mean().item())}
    log('  extras: 1M batch %.2f ms' % ms)
    out["batch_1M"]["tflops"] = f_iter(cfg.N) * float(it.sum().item()) / (ms * 1e-3) / 1e12
    if fp64_peak:
        out["batch_1M"]["fp64_flops_frac_of_measured_peak"] = out["batch_1M"]["tflops"] / fp64_peak
        out["batch_1M"]["fp64_flops_frac_of_nominal"] = out["batch_1M"]["tflops"] / FP64_NOMINAL_TFLOPS
    # config 4 share: per-problem weights, 128K problems (1/8 of the 1M sweep)
    B4 = 131072
    rng = np.random.default_rng(2)
    sel = rng.integers(0, 4096, B4)
    W = np.tile(np.array(cd["weights"]), (B4, 1))
    W[:, 3] = np.exp(rng.uniform(np.log(1), np.log(5000), B4)); W[:, 4] = np.exp(rng.uniform(np.log(1), np.log(5000), B4))
    W[:, 1] = np.exp(rng.uniform(np.log(1), np.log(1000), B4)); W[:, 2] = rng.choice([0.01, 0.1, 1, 10, 100], B4)
    ins4 = [ctx.up(b["state"][sel].T), ctx.up(b["coeffs"][sel].T), ctx.up(b["yaw_lo"][sel]), ctx.up(b["yaw_hi"][sel])]
    Wd = ctx.up(W.T)
    r4 = res[:, :B4].contiguous()
    ms = timed(lambda: S.solve_batch_device(B4, *ins4, r4, None, None, None, st[:B4], it[:B4], weights=Wd), 2)
    log('  extras: weight sweep 128K %.2f ms' % ms)
    out["config4_weight_sweep_128K"] = {"solves_per_s": B4 / ms * 1e3, "ms": ms, "status_ok_frac": float((st[:B4] == 1).float().mean().item()),
                                        "iters_max": int(it[:B4].max().item())}
    S.close()
    # config 3: N x dt grid, one ragged launch of 256K problems
    B3 = 262144
    pick = np.random.default_rng(1).integers(0, len(PAIRS), B3)
    Np = ctx.up(np.array([PAIRS[k][0] for k in pick], dtype=np.int32)); dtp = ctx.up(np.array([PAIRS[k][1] for k in pick]))
    cfg3 = mpc.config_from_json_text(json.dumps(dict(js, N=50)))
    S3 = mpc.Solver(cfg3, ctx.local_rank)
    b3 = mpc.workloads.batch_perturbed_states(B3, 1, cd)
    ins3 = [ctx.up(b3["state"].T), ctx.up(b3["coeffs"].T), ctx.up(b3["yaw_lo"]), ctx.up(b3["yaw_hi"])]
    r3 = res[:, :B3].contiguous()
    ms = timed(lambda: S3.solve_batch_device(B3, *ins3, r3, None, None, None, st[:B3], it[:B3], N_per=Np, dt_per=dtp), 2)   # best of 2: the first call allocates the record buffers
    log('  extras: horizon grid 256K %.2f ms' % ms)
    out["config3_horizon_grid_256K"] = {"solves_per_s": B3 / ms * 1e3, "ms": ms, "status_ok_frac": float((st[:B3] == 1).float().mean().item()),
                                        "status_hist": status_hist(st[:B3].cpu().numpy()), "iters_max": int(it[:B3].max().item()),
                                        "note": "N in 10..50 x dt in {0.1,0.05,0.02}; the long-horizon cells need Ipopt's restoration phase on ~10 % of their problems"}
    S3.close()
    # config 5 share: closed loop, config-fast (100 ms latency), 1024 vehicles (one GPU's share of 8192) x 200 steps, one launch
    cfgf = mpc.config_from_json_text(json.dumps(rd["configs"]["fast"]))
    cdf = cfgf.as_dict()
    V, T = 1024, 200
    bv = mpc.workloads.batch_perturbed_states(V, 3, cdf)
    veh = ctx.up(np.stack([bv["px"], bv["py"], bv["psi"], np.clip(bv["v"], 8, 30), np.zeros(V), np.zeros(V)]))
    seg = ctx.up(bv["segment"].astype(np.int32))
    pend = torch.zeros(2, V, dtype=torch.float64, device=dev)
    rec = torch.zeros(T, 8, V, dtype=torch.float64, device=dev)
    wx, wy = ctx.up(np.array(rd["waypoints"]["x"])), ctx.up(np.array(rd["waypoints"]["y"]))
    S5 = mpc.Solver(cfgf, ctx.local_rank)
    torch.cuda.synchronize()
    n0 = S5.launches
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); S5.rollout_device(V, T, wx, wy, veh, seg, pend, 0.1, 0.02, rec); e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    log('  extras: rollout 1024x200 %.2f ms' % ms)
    out["config5_closed_loop_1024x200"] = {"vehicle_steps_per_s": V * T / ms * 1e3, "ms_per_control_step": ms / T, "launches": int(S5.launches - n0),
                                           "status_ok_frac": float((rec[:, 6] == 1).float().mean().item()),
                                           "median_abs_cte_final_m": float(rec[-1, 0].abs().median().item())}
    S5.close()
    return out


def main():
    quiet_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--batch", type=int, default=65536, help="problems per GPU per step (batch64k); total problems / vehicles for the other workloads")
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="batch64k", choices=["batch64k", "weights1M", "grid256k", "rollout8192x1000"])
    ap.add_argument("--rollout-steps", type=int, default=1000)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the one-GPU shares of the other BASELINE configs")
    ap.add_argument("--gather", default="serial", choices=["overlap", "serial"],
                    help="multi-GPU: the gather of step k finishes before the solve of step k+1 starts (default), or runs beside it (see DESIGN.md section 7)")
    ap.add_argument("--only-timed", action="store_true", help="development: the timed region only (no strong-scaling, host-API, latency, extras or CPU legs)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed (rank 0's arrays, [k][B] layout as the caller "
                         "receives them) as DIR/<name>.npy in float64, at most 64 MB in all: a fixed, seeded sample of the "
                         "problems beyond that.  The inputs depend only on the arguments, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of --impl ours (the reference arm times a sample sized by its own speed)")
    rank = int(os.environ.get("RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.only_timed:
        args.no_latency = args.no_extras = args.no_cpu_baseline = True
    if args.warmup < 3:
        args.warmup = 3
    ctx = Ctx()
    fn = {"batch64k": run_batch64k, "weights1M": run_weights1M, "grid256k": run_grid256k, "rollout8192x1000": run_rollout}[args.workload]
    line = fn(ctx, args)
    if ctx.rank == 0 and line is not None:
        emit(line)
    ctx.close()


if __name__ == "__main__":
    main()
