"""One of the large BASELINE configurations (radial200 / meshed1000) on cuda:0: set-up + timed solves.
usage: run_other.py kind B reps"""
import os, sys, time
R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (R, os.path.join(R, "tests"), os.path.join(R, "oracle")):
    sys.path.insert(0, p)
import numpy as np, torch
import bench
from harmonic_power_flow_b200 import BatchSolver, scenarios
kind = sys.argv[1]; B = int(sys.argv[2]); reps = int(sys.argv[3]) if len(sys.argv) > 3 else 1
net = bench.load_other(kind)
sol = BatchSolver(net)
t0 = time.perf_counter(); info = sol.struct_info(); torch.cuda.synchronize(); ts = time.perf_counter() - t0
P, Q, I_N = scenarios.make_batch(net, B, "tight")
dP, dQ, dI = sol.prepare(P, Q, I_N)
r = sol.solve(dP, dQ, dI); torch.cuda.synchronize()
sol.set_profiling(True)
best = None
for _ in range(reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); r = sol.solve(dP, dQ, dI, out=r); e1.record(); torch.cuda.synchronize()
    k = sol.last_kernel_ms(); ms = e0.elapsed_time(e1)
    if best is None or ms < best[0]: best = (ms, k)
it = r.n_iter_h.double()
print("%s B=%d setup %.2fs step %.1f ms (fund %.1f harm %.1f) %.1f solves/s mean it %.2f conv %d checksum %.13e" % (
    kind, B, ts, best[0], best[1][0], best[1][1],
    B / best[0] * 1e3, it.mean().item(), int((r.status == 0).sum().item()), float(r.V_m.sum())))
