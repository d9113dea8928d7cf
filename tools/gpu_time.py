"""Timing only: lane kernel on the bench workload for a list of (threads, ctas/sm) settings given as argv."""
import json, sys, os
import numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import mpc_b200 as mpc
B = int(sys.argv[1])
sets = [tuple(int(x) for x in a.split(",")) for a in sys.argv[2:]] or [(32, 0)]
rd = mpc.workloads.reference_data()
cfg = mpc.config_from_json_text(json.dumps(rd['configs']['stable']))
S = mpc.Solver(cfg, 0)
b = mpc.workloads.batch_perturbed_states(B, 0, cfg.as_dict())
dev = torch.device('cuda:0')
up = lambda a: torch.from_numpy(np.ascontiguousarray(a.T if a.ndim == 2 else a)).to(dev)
state, coeffs, ylo, yhi = up(b['state']), up(b['coeffs']), up(b['yaw_lo']), up(b['yaw_hi'])
N = cfg.N
result = torch.zeros(9, B, dtype=torch.float64, device=dev)
tx = torch.zeros(N, B, dtype=torch.float64, device=dev); ty = torch.zeros(N, B, dtype=torch.float64, device=dev)
status = torch.zeros(B, dtype=torch.int32, device=dev); iters = torch.zeros(B, dtype=torch.int32, device=dev)
for thr, ctas in sets:
    S.set_kernel(mpc.KERNEL_LANE, thr, ctas)
    best = 1e9
    for _ in range(6):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); S.solve_batch_device(B, state, coeffs, ylo, yhi, result, tx, ty, None, status, iters); e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    print('lane threads=%d ctas/sm=%d  B=%d  %.3f ms  %.0f solves/s  ok=%.4f iters=%.2f csum=%.6f' % (thr, ctas, B, best, B / best * 1e3, (status == 1).float().mean().item(), iters.float().mean().item(), result[8].sum().item()))
