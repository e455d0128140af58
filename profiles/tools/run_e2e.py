"""hpf_solve_host end to end (pinned host buffers) for config 3 - chunk-plan sweep via $HPF_HOST_PLAN."""
import os, sys, tempfile, time
R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (R, os.path.join(R, "tests"), os.path.join(R, "oracle")):
    sys.path.insert(0, p)
import numpy as np, torch, helpers
from harmonic_power_flow_b200 import BatchSolver, scenarios
net, _, _ = helpers.packed_from_files("net3", 25, True, tempfile.mkdtemp())
B = int(sys.argv[1]) if len(sys.argv) > 1 else 65536
sol = BatchSolver(net)
P, Q, I_N = scenarios.make_batch(net, B, "tight")
hP, hQ, hI = (torch.as_tensor(x).pin_memory().numpy() for x in (P, Q, I_N))
for _ in range(3):
    r = sol.solve_host(hP, hQ, hI)
best = 1e9
for _ in range(10):
    t0 = time.perf_counter(); r = sol.solve_host(hP, hQ, hI); best = min(best, time.perf_counter() - t0)
print("plan=%s B=%d solve_host best %.3f ms (%.1f M solves/s) conv %d" % (os.environ.get("HPF_HOST_PLAN", "default"), B, best * 1e3,
      B / best / 1e6, int((r["status"] == 0).sum())))
