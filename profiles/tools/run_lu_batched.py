"""Batched LU of hpf_lockstep.cuh standalone (hpf_lu_solve with $HPF_LOCKSTEP=1) on random systems of
order N = 1038 (net1, H <= 51) - target of ncu captures / A-B timings of the panel / interchange /
tensor-core update kernels.  usage: run_lu_batched.py [B] [reps]"""
import os
import sys
import tempfile

R = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (R, os.path.join(R, "tests"), os.path.join(R, "oracle")):
    sys.path.insert(0, p)
os.environ.setdefault("HPF_LOCKSTEP", "1")
import numpy as np
import torch
import helpers
from harmonic_power_flow_b200 import BatchSolver

net, st, _ = helpers.packed_from_files("net1", 51, True, tempfile.mkdtemp(), julia_schema=True)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 512
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 2
sol = BatchSolver(net)
N = sol.N
stride = sol.jacobian_stride()
g = torch.Generator(device="cuda").manual_seed(5)
J = torch.zeros((B, stride), dtype=torch.float64, device="cuda")
J[:, :N * N] = torch.randn((B, N * N), dtype=torch.float64, device="cuda", generator=g)
f = torch.randn((N, B), dtype=torch.float64, device="cuda", generator=g)
dx, info = sol.lu_solve(J, f)
torch.cuda.synchronize()
best = 1e9
for _ in range(reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); dx, info = sol.lu_solve(J, f); e1.record(); torch.cuda.synchronize()
    best = min(best, e0.elapsed_time(e1))
fl = (2.0 / 3.0 * N ** 3 + 2.0 * N * N) * B
Jv = J[:, :N * N].view(B, N, N)
res = torch.einsum("bij,jb->ib", Jv[:8], dx[:, :8]) - f[:, :8]
print("B=%d N=%d batched lu_solve %.2f ms  %.2f TFLOP/s  info!=0: %d  residual %.2e" % (
    B, N, best, fl / best / 1e9, int((info != 0).sum()), float(res.abs().max())))
