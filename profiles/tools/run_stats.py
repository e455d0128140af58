"""Batch statistics on the bench workload (net3, 13 orders, 65,536 scenarios of bench.py's generator), one
process on one GPU: the device-resident solve against hpf_batch_stats (K = 3) with CUDA events, then
hpf_solve_host against hpf_solve_host_stats end to end (pinned inputs, alternating calls, host clock around
calls that synchronise), with the bytes each copies in each direction.  Writes one JSON line.

    python profiles/tools/run_stats.py [--out profiles/r3_batch_stats_1gpu.json] [--reps 50] [--e2e-reps 20]
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                       capture_output=True, text=True)
    name, power = (q.stdout.strip().splitlines() or ["?, ?"])[0].split(",", 1)
    return {"name": name.strip(), "power_limit": power.strip()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_batch_stats_1gpu.json"))
    ap.add_argument("--reps", type=int, default=50)
    ap.add_argument("--e2e-reps", type=int, default=20)
    a = ap.parse_args()
    import numpy as np
    import torch
    import bench
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    assert torch.cuda.is_available(), "needs a CUDA device"
    B, quant = bench.B_PER_GPU, (0.05, 0.5, 0.95)
    net = bench.load_net()
    sol = BatchSolver(net, 0)
    P, Q, I_N = scenarios.make_batch(net, B, bench.SPREAD, seed0=0)
    dP, dQ, dI = sol.prepare(P, Q, I_N)
    hP, hQ, hI = (torch.as_tensor(x).pin_memory().numpy() for x in (P, Q, I_N))
    r = sol.solve(dP, dQ, dI)
    for _ in range(3):                                              # warm-up of every shape timed below
        r = sol.solve(dP, dQ, dI, out=r)
        s = sol.batch_stats(r.V_m, r.status, quantiles=quant)
        sol.solve_host(hP, hQ, hI)
        sol.solve_host_stats(hP, hQ, hI, quantiles=quant)
    torch.cuda.synchronize()

    # device-resident: each repetition = one solve then one statistics call, events around each
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(a.reps)]
    for e in ev:
        e[0].record()
        r = sol.solve(dP, dQ, dI, out=r)
        e[1].record()
        s = sol.batch_stats(r.V_m, r.status, quantiles=quant)
        e[2].record()
    torch.cuda.synchronize()
    solve_ms = np.array([e[0].elapsed_time(e[1]) for e in ev])
    stats_ms = np.array([e[1].elapsed_time(e[2]) for e in ev])
    conv = int((r.status == 0).sum().item())

    # end to end, alternating
    t_host, t_stats = [], []
    for _ in range(a.e2e_reps):
        t0 = time.perf_counter(); sol.solve_host(hP, hQ, hI); t_host.append(time.perf_counter() - t0)
        t0 = time.perf_counter(); hs = sol.solve_host_stats(hP, hQ, hI, quantiles=quant); t_stats.append(time.perf_counter() - t0)
    t_host, t_stats = np.array(t_host) * 1e3, np.array(t_stats) * 1e3
    n, H, q = net.n, net.H, net.q
    R = n * H + 2 * n
    h2d = (2 * n + 2 * q * H) * 8 * B
    d2h_host = (2 * n * H * 8 + 2 * q * H * 8 + 8 + 3 * 4) * B
    d2h_stats = (5 + len(quant)) * R * 8 + 4 * 4
    same = bool(np.array_equal(hs.planes.view(np.uint64), s.planes.cpu().numpy().view(np.uint64)))
    out = {
        "what": "hpf_batch_stats (K = 3) and hpf_solve_host_stats on the bench workload",
        "gpu": gpu_info(), "B": B, "rows": R, "quantiles": list(quant), "converged": conv,
        "device": {"reps": a.reps, "solve_ms_median": float(np.median(solve_ms)), "stats_ms_median": float(np.median(stats_ms)),
                   "stats_ms_min": float(stats_ms.min()), "stats_over_solve": float(np.median(stats_ms) / np.median(solve_ms)),
                   "note": "events around each call, a solve before each statistics call (its V_m is L2-resident)"},
        "e2e": {"reps": a.e2e_reps,
                "solve_host_ms_median": float(np.median(t_host)), "solve_host_ms_min": float(t_host.min()),
                "solve_host_stats_ms_median": float(np.median(t_stats)), "solve_host_stats_ms_min": float(t_stats.min()),
                "solve_host_solves_per_s": conv / (np.median(t_host) / 1e3),
                "solve_host_stats_solves_per_s": conv / (np.median(t_stats) / 1e3),
                "speedup": float(np.median(t_host) / np.median(t_stats)),
                "h2d_bytes": {"solve_host": h2d, "solve_host_stats": h2d},
                "d2h_bytes": {"solve_host": d2h_host, "solve_host_stats": d2h_stats},
                "note": "pinned inputs, pinned phasor buffers for solve_host; host clock around each call (both synchronise)"},
        "host_stats_equals_device_stats": same,
    }
    line = json.dumps(out)
    print(line)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
