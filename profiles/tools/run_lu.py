"""Kernel 4 standalone (hpf_lu_solve) on config-3 Jacobians - target of ncu captures / A-B timings.
usage: run_lu.py [B] [reps]   env: HPF_LU_CLASSIC=1 (rank-1 LU)"""
import os
import sys
import tempfile

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (R, os.path.join(R, "tests"), os.path.join(R, "oracle")):
    sys.path.insert(0, p)
import numpy as np
import torch
import helpers
from harmonic_power_flow_b200 import BatchSolver, scenarios

net, st, _ = helpers.packed_from_files("net3", 25, True, tempfile.mkdtemp())
B = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 3
sol = BatchSolver(net)
P, Q, I_N = scenarios.make_batch(net, B, "tight")
raw = sol.solve(P, Q, I_N, raw=True, max_iter_h=3, want_I_inj=False)
f, _ = sol.mismatch(raw.V_m, raw.V_a, P, Q, I_N)
J = sol.jacobian(raw.V_m, raw.V_a)
dx, info = sol.lu_solve(J, f)
torch.cuda.synchronize()
best = 1e9
for _ in range(reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); dx, info = sol.lu_solve(J, f); e1.record(); torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1))
N = sol.N
fl = (2.0 / 3.0 * N ** 3 + 2.0 * N * N) * B
print("B=%d N=%d lu_solve %.3f ms  %.3f TFLOP/s  info!=0: %d  checksum %.12e" % (
    B, N, best, fl / best / 1e9, int((info != 0).sum()), float(dx.sum())))
