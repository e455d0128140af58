#!/usr/bin/env python
"""Benchmark of the harmonic power-flow solve path (driver contract, see DESIGN.md "Measurement").

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path
    python bench.py --strong ...                                   # 65,536 scenarios IN TOTAL over the ranks
    python bench.py --impl reference [--steps K] [--warmup W]      # CPU arm (oracle port; + the reference
                                                                   #   itself when its checkout is present)
    torchrun ... bench.py --gpus N ...                             # N > 1, one rank per GPU
    python bench.py --dump-outputs DIR ...                         # + what the timed solve returned (.npy)

Workload (BASELINE.json configs[2], the configuration the metric and target are quoted on):
net3, coupled SMPS Norton equivalent, fundamental + odd harmonics to the 25th (N = 101),
65,536 seeded randomised load / spectrum scenarios PER GPU (weak scaling: scenarios are
independent, each rank solves its own block, no data-path collective); with --strong 65,536
scenarios in total, split over the ranks (the north-star target).  The default run also measures
the strong-scaling share (65,536 / N per rank) and reports it under `strong_scaling`.  One "step"
= one complete solve of the batch: fundamental NR + harmonic NR + post-processing.

Keys: `value` = converged solves/s with the default (structured Newton step) strategy, inputs
resident in HBM, CUDA-event timed on the launch stream, max over ranks; `dense_lu_path` = the
same workload forced through the dense shared-memory LU kernel (HPF_SOLVE_DENSE).  `e2e` = the
same through the host-buffer C-ABI entry point (hpf_solve_host / hpf_solve_host_keep): pinned host
inputs -> H2D -> solve -> D2H of every result on every rank, plus (N > 1) the final NCCL gather of
flags and results to rank 0.  `roofline` = the dominant kernel (fused Newton kernel) against the
FP64 pipe; `roofline_kernels` = the standalone mismatch / Jacobian kernels against measured HBM
bandwidth.  `cpu_baseline` = the oracle port on the host cores; `parity` = GPU (both strategies)
against that oracle run on the SAME scenarios, next to the oracle's own SuperLU-vs-LAPACK floor.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True       # the tree may be read-only: no bytecode caches next to the sources

NET, H_MAX, COUPLED, SPREAD = "net3", 25, True, "tight"
B_PER_GPU = 65536
B_TARGET = 65536                     # north-star target: this many scenarios in total (strong scaling)
PARITY_SCENARIOS = 16384
METRIC = "converged harmonic-PF solves/sec (FP64)"
UNIT = "solves/s"
NCU_CSV = os.path.join(ROOT, "profiles", "r2_ncu_kernels.csv")


def load_net():
    """net3 + smps Norton equivalent from the committed fixtures (tests/golden/, SI units),
    through the product's own per-unit conversion (netio)."""
    import numpy as np
    from harmonic_power_flow_b200 import netio
    import pandas as pd
    g = os.path.join(ROOT, "tests", "golden")
    tab = json.load(open(os.path.join(g, "networks.json")))[NET]
    st = netio.Settings(H_MAX=H_MAX)
    buses, lines = pd.DataFrame(tab["buses"]), pd.DataFrame(tab["lines"])
    for col in ("S", "P", "Q"):
        buses[col] = buses[col].astype(float) / st.BASE_POWER
    buses["X_sh"] = buses["X_sh"].astype(float) / st.base_impedance
    for col in ("R", "X"):
        lines[col] = lines[col].astype(float) / st.base_impedance
    for col in ("G", "B"):
        lines[col] = lines[col].astype(float) / st.base_admittance
    nl = buses.index[buses["type"] == "nonlinear"]
    m, n = int(min(nl)), len(buses)
    c = int((buses.type == "PV").sum()) + 1
    dev = np.load(os.path.join(g, "ne_devices.npz"))
    freqs = np.array(st.HARMONICS_FREQ)
    col = np.searchsorted(dev["smps__freqs"], freqs)
    row = np.searchsorted(dev["smps__Y_N_c_rowfreq"], freqs)
    net = netio.pack_network(buses, lines, m, n, c, st.HARMONICS)
    net.devices = ["smps"]
    net.dev_of_nl_bus = np.zeros(n - m, np.int32)
    net.coupled = True
    net.Y_N = np.ascontiguousarray((dev["smps__Y_N_c"][np.ix_(row, col)] / st.base_admittance)[None])
    net.I_N = np.ascontiguousarray(np.repeat((dev["smps__I_N_c"][col] / st.base_current)[None], n - m, 0))
    return net


def load_other(kind):
    """Networks of the other BASELINE configurations through the product's own CSV loaders:
    'net2ev' (configs[1]: net2 with an SMPS and an EV Norton-equivalent load, odd harmonics to the
    19th), 'radial200' (configs[3]) and 'meshed1000' (configs[4]) from the seeded generators."""
    import tempfile
    import numpy as np
    import pandas as pd
    from harmonic_power_flow_b200 import netio, synthetic
    g = os.path.join(ROOT, "tests", "golden")
    tmp = tempfile.mkdtemp(prefix="hpf_bench_")
    dev = np.load(os.path.join(g, "ne_devices.npz"))
    for d in ("smps", "ev"):
        netio.write_ne_csv(os.path.join(tmp, d + "_NE.csv"), dev[d + "__freqs"], dev[d + "__Y_N_c"],
                           dev[d + "__I_N_c"], dev[d + "__Y_N_uc"], dev[d + "__I_N_uc"])
    if kind in ("net2ev", "net1"):
        tab = json.load(open(os.path.join(g, "networks.json")))[kind]
        pb, pl = os.path.join(tmp, kind + "_buses.csv"), os.path.join(tmp, kind + "_lines.csv")
        pd.DataFrame(tab["buses"]).to_csv(pb, sep=";", index=False)
        pd.DataFrame(tab["lines"]).to_csv(pl, sep=";", index=False)
        h_max = 19 if kind == "net2ev" else 51
    elif kind == "radial200":
        pb, pl = synthetic.radial_feeder(tmp, tmp, n=200, load_scale=0.005)
        h_max = 25
    else:
        pb, pl = synthetic.meshed(tmp, tmp, n=1000, load_scale=0.002)
        h_max = 25
    st = netio.Settings(H_MAX=h_max, ne_dir=tmp)
    buses, lines, m, n, c = netio.init_network(pb, pl, st)
    NE = netio.import_Norton_Equivalents(buses, True, st)
    return netio.pack_network(buses, lines, m, n, c, st.HARMONICS, NE, True)


OTHER_CONFIGS = [
    ("configs[0]: net1 (20 buses, 7 SMPS loads) coupled, odd harmonics <= 51 (N=1038), ONE scenario (latency)",
     "net1", 1, 5),
    ("configs[1]: net2 + SMPS/EV Norton loads, odd harmonics <= 19 (N=78)", "net2ev", 1024, 3),
    ("configs[3]: synthetic 200-bus radial feeder, 40% nonlinear buses, odd harmonics <= 25 (N=5198)",
     "radial200", 8192, 2),
    ("configs[4]: synthetic 1000-bus meshed network, 40% nonlinear buses, full coupled Norton, odd "
     "harmonics <= 25 (N=25998)", "meshed1000", 1024, 1),
]


def lu_flops(k):
    return 2.0 / 3.0 * k ** 3 + 2.0 * k * k


def structured_flops(n, H, m, c, q, nnzY, it_f, it_h, B):
    """Algorithmic FP64 flops of B scenarios (it_f, it_h = iteration counts summed over the batch) solved with the structured Newton step (DESIGN.md
    "Roofline accounting"; complex MAC = 8 flops): per harmonic iteration the mismatch through the
    non-zeros of Y(h) + the Norton contraction, G (V_F + u_F), the polar conversion and the LU of the
    (2m-1-c) border system; per fundamental iteration the LU of the (2n-1-c) system; once w_N."""
    nZ, nx, Nf = n * H - m, 2 * m - 1 - c, 2 * n - 1 - c
    per_h = 8.0 * (nnzY + q * H * H) + 8.0 * nZ * m + 10.0 * n * H + lu_flops(nx) + 8.0 * m * m
    per_f = 24.0 * n * n + lu_flops(Nf)
    once = 8.0 * nZ * q * H
    return it_h * per_h + it_f * per_f + once * B, per_h


def run_other_configs(torch, dist, BatchSolver, scenarios, local, rank, world, fp64_peak):
    """Device-resident solves/s of the other BASELINE configurations (weak scaling like the
    headline: every rank solves its own block of scenarios of the same network), each with its
    roofline fraction against the measured DGEMM peak.  The operator set-up (once per network) is
    timed separately."""
    out = []
    for label, kind, B, steps in OTHER_CONFIGS:
        net = load_other(kind)
        sol = BatchSolver(net, local)
        t0 = time.perf_counter()
        info = sol.struct_info()
        torch.cuda.synchronize()
        t_setup = time.perf_counter() - t0
        P, Q, I_N = scenarios.make_batch(net, B, SPREAD, seed0=rank * B)
        dP, dQ, dI = sol.prepare(P, Q, I_N)
        r = sol.solve(dP, dQ, dI)                                   # warm-up
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            r = sol.solve(dP, dQ, dI, out=r)
        e1.record(); torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        vals = torch.tensor([ms, float((r.status == 0).sum().item()), r.n_iter_h.double().sum().item(),
                             r.n_iter_f.double().sum().item()], dtype=torch.float64, device=r.status.device)
        if world > 1:
            mx = vals.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
            sm = vals.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        else:
            mx, sm = vals, vals
        nnzY = int((sol.Y != 0).sum().item())
        fl, fl_iter = structured_flops(net.n, net.H, net.m, net.c, net.q, nnzY, vals[3].item(), vals[2].item(), B)
        ach = fl / (ms / 1e3) / 1e12                               # this rank's flops over this rank's time
        path = sol.last_solve_path
        sol.set_profiling(True)
        sol.solve(dP, dQ, dI, out=r)
        torch.cuda.synchronize()
        kms = sol.last_kernel_ms()
        sol.set_profiling(False)
        out.append({"config": label, "batch_per_gpu": B, "N": int(sol.N), "strategy_variant": int(info["available"]),
                    "harmonic_stage_path": BatchSolver.PATHS.get(path, str(path)),
                    "kernel_ms_per_step": {"fundamental_stage": kms[0], "harmonic_stage": kms[1]},
                    "value": sm[1].item() / (mx[0].item() / 1e3), "unit": UNIT, "ms_per_step": mx[0].item(),
                    "converged_fraction": sm[1].item() / (B * world),
                    "mean_harmonic_iterations": sm[2].item() / (B * world),
                    "operator_setup_s": t_setup,
                    "roofline": {"bound": "fp64", "achieved": ach, "peak": fp64_peak, "unit": "TFLOP/s",
                                 "frac": ach / fp64_peak if fp64_peak else None,
                                 "flops_per_harmonic_iteration": fl_iter,
                                 "border_system_order": 2 * net.m - 1 - net.c, "fundamental_system_order": 2 * net.n - 1 - net.c,
                                 "note": "algorithmic flops of the structured step (LU of the border system, G product, "
                                         "mismatch through nnz(Y), w_N once) over the whole-step time, rank 0"}})
        sol.close()
        del sol, r, dP, dQ, dI
        torch.cuda.empty_cache()
    return out


def source_hash():
    """sha1 over the CUDA sources: identifies the binary a profile was taken from (the GPU box has
    no .git, so the SHA of the commit cannot be read there)."""
    h = hashlib.sha1()
    d = os.path.join(ROOT, "harmonic_power_flow_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if f.endswith((".cu", ".cuh")):
            h.update(f.encode()); h.update(open(os.path.join(d, f), "rb").read())
    return h.hexdigest()[:12]


def ncu_traffic(kernel_substr):
    """DRAM bytes (read + write) of one launch of a kernel from the committed ncu --set full summary
    (profiles/r2_ncu_kernels.csv, written by profiles/tools/ncu_summary.py; its first line records the
    git SHA and the source hash of the binary it was captured from).  -> (bytes or None, provenance);
    `stale` is True when the sources have changed since the capture."""
    import csv
    prov = {"file": os.path.relpath(NCU_CSV, ROOT), "git_sha": None, "src_hash": None, "stale": None}
    if not os.path.exists(NCU_CSV):
        prov["file"] = None
        return None, prov
    lines = open(NCU_CSV).read().splitlines()
    if lines and lines[0].startswith("#"):
        for tok in lines[0][1:].split():
            if "=" in tok:
                k, v = tok.split("=", 1)
                if k in prov:
                    prov[k] = v
        lines = lines[1:]
    prov["stale"] = (prov["src_hash"] != source_hash())
    rows = list(csv.reader(lines))
    hdr, units = rows[0], rows[1]
    ir, iw = hdr.index("dram__bytes_read.sum"), hdr.index("dram__bytes_write.sum")
    scale = {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0, "Tbyte": 1e12}
    for r in rows[2:]:
        if kernel_substr in r[0]:
            return float(r[ir]) * scale[units[ir]] + float(r[iw]) * scale[units[iw]], prov
    return None, prov


def workload_text():
    return ("BASELINE configs[2]: net3 coupled (smps_NE), fundamental + odd harmonics <= 25 "
            "(N=101), randomised load/spectrum scenarios (P,Q x U(0.9,1.1), I_N x U(0.95,1.05) "
            "e^{jU(-0.02,0.02)}; scenario s = numpy default_rng(s)), thresh 1e-6/1e-4, caps 30/50")


def config_dict(n_gpus, per_gpu, strong):
    return {"workload": workload_text(),
            "batch_per_gpu": per_gpu, "global_batch": B_TARGET if strong else per_gpu * n_gpus,
            "parallelism": "scenario-sharded x%d, no data-path collective" % n_gpus,
            "cache": "L2 flushed (256 MiB write) between timed steps"}


# ------------------------------------------------------------------------------- CPU arm
def oracle_pool(procs=None):
    """Oracle port (numpy + SuperLU step, like the reference) fanned out over the host cores
    (oracle/oracle_pool.py: test / bench infrastructure, never on the product path)."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import hpf_oracle as O
    import oracle_pool as OP
    on = O.net_from_golden(os.path.join(ROOT, "tests", "golden"), NET, H_MAX, COUPLED)
    return OP.OraclePool(on, procs or os.cpu_count() or 1), OP, on


def reference_root():
    for cand in (os.environ.get("HPF_REFERENCE_ROOT"), "/root/reference"):
        if cand and os.path.isdir(os.path.join(cand, "Harmonic Power Flow")):
            return cand
    return None


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from harmonic_power_flow_b200 import scenarios
    cores = os.cpu_count() or 1
    per_step = 256 * cores           # ~6.5 ms per solve per core -> ~2 s per step
    pool, OP, on = oracle_pool(cores)
    for _ in range(a.warmup):
        P, Q, I_N = scenarios.make_batch(on, 16 * cores, SPREAD)
        pool.solve(P, Q, I_N, "superlu", keep_V=False)
    conv = iters = 0
    dt = 0.0
    for k in range(a.steps):
        P, Q, I_N = scenarios.make_batch(on, per_step, SPREAD, seed0=k * per_step)      # untimed
        r = pool.solve(P, Q, I_N, "superlu", keep_V=False)
        conv += int((r["status"] == 0).sum()); iters += int(r["n_iter_h"].sum()); dt += r["wall_s"]
    pool.close()
    v = conv / dt
    sample = "%d scenarios per step x %d steps of the same seeded workload (seeds 0..%d), %d worker processes" % (
        per_step, a.steps, per_step * a.steps - 1, cores)
    cfg = {"workload": workload_text(), "scenarios_per_step": per_step, "worker_processes": cores,
           "gpu_arm_batch_per_gpu": B_PER_GPU,
           "note": "bounded sample of the GPU arm's workload: the CPU cannot solve 65,536 scenarios per step "
                   "inside a bench run; solves/s is per-scenario throughput and extrapolates linearly"}
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus,
            "steps": a.steps, "warmup": a.warmup, "ms_per_step": dt / a.steps * 1e3,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": cfg,
            "ms_per_nr_iteration_per_core": dt * 1e3 * cores / max(iters, 1),
            "cpu_baseline": {"value": v, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                             "note": "oracle/hpf_oracle.py: numpy restatement of the reference solve path "
                                     "(SuperLU step like the reference), ~100-200x faster per core than the "
                                     "reference's own pandas code (below / BASELINE.md section 2)"},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    # the reference ITSELF (its own hpf(), HG:511-560) when its checkout is present: kind "exec"
    root = reference_root()
    if root and not a.no_exec:
        try:
            os.environ.setdefault("HPF_REFERENCE_ROOT", root)
            sys.path.insert(0, os.path.join(ROOT, "oracle"))
            import time_reference as TR
            ex = TR.run(n_scen=max(4 * cores, 32), procs=cores)
            line["reference_exec"] = {k: ex[k] for k in ("kind", "what", "config", "scenarios", "procs", "cpu_model",
                                                        "wall_s", "solves_per_s", "solves_per_s_per_core",
                                                        "s_per_solve_median", "ms_per_nr_iteration_loop_only")}
        except Exception as e:                                   # the port line stands on its own
            line["reference_exec"] = {"kind": "exec", "unavailable": "%s: %s" % (type(e).__name__, e)}
    else:
        line["reference_exec"] = {"kind": "exec", "unavailable": "no reference checkout on this box "
                                  "($HPF_REFERENCE_ROOT); builder-measured: profiles/r2_reference_exec_timing.json"}
    print(json.dumps(line))


# ------------------------------------------------------------------------------- clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.rows.append([x.strip() for x in ln.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [nm for k, nm in enumerate(names)
                   if any(len(r) > 3 + k and r[3 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------- GPU arm
def measure_fp64_peak(torch, dev):
    """FP64 denominator: cuBLAS DGEMM 8192^3 (uses the DMMA path) - MEASURED_PEAKS.json has no
    FP64 figure.  Burst (best of 5) in TFLOP/s."""
    n = 8192
    a = torch.randn(n, n, dtype=torch.float64, device=dev)
    b = torch.randn(n, n, dtype=torch.float64, device=dev)
    torch.matmul(a, b)
    best = 1e9
    for _ in range(5):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); torch.matmul(a, b); e1.record(); torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1))
    del a, b
    return 2 * n ** 3 / best / 1e9


RESULT_KEYS = ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status")
DUMP_BYTES = 60 * 10 ** 6            # --dump-outputs: the sample of scenarios is as large as this allows


def dump_outputs(res, dirname):
    """Write what the timed solve returned (the BatchResult fields, batch innermost) as DIR/<name>.npy,
    all float64: complex fields as <name>_re / <name>_im, integer fields converted.  Only a fixed,
    seeded sample of the batch's scenarios is kept (all 65,536 of net3 come to ~70 MB); scenario.npy
    holds their indices.  Same arguments, same inputs: two builds compare file for file."""
    import numpy as np
    import torch
    arrays = {}
    for k in RESULT_KEYS:
        v = getattr(res, k)
        if v is None:
            continue
        if v.is_complex():
            arrays[k + "_re"], arrays[k + "_im"] = v.real, v.imag
        else:
            arrays[k] = v
    per_scenario = 8 * (1 + sum(v[..., 0].numel() for v in arrays.values()))
    S = min(res.B, DUMP_BYTES // per_scenario)
    idx = np.sort(np.random.default_rng(0).choice(res.B, S, replace=False))
    sel = torch.as_tensor(idx, device=res.status.device)
    os.makedirs(dirname, exist_ok=True)
    np.save(os.path.join(dirname, "scenario.npy"), idx.astype(np.float64))
    for k, v in arrays.items():
        np.save(os.path.join(dirname, k + ".npy"), v.index_select(-1, sel).to(torch.float64).cpu().numpy())


class E2E:
    """The end-to-end step through the reference-facing entry point, N ranks.

    Every rank: hpf_solve_host_keep (C ABI, HOST buffers: H2D, fundamental + harmonic solve and D2H of
    all results pipelined in chunks inside the call; results also left on the device), then - N > 1 -
    the only inter-GPU traffic of the path: the NCCL gather of the convergence flags and of the
    results to rank 0.  The gather of step k runs on NCCL's stream while step k+1 is being solved
    (NVLink and PCIe are independent links; two result slabs alternate), the timed region ends when
    the last gather has completed."""

    def __init__(self, torch, dist, sol, net, B, world, rank):
        from harmonic_power_flow_b200 import solver as hsolver
        from harmonic_power_flow_b200 import dist as hdist
        self.torch, self.dist, self.hdist, self.sol, self.world, self.rank, self.B = torch, dist, hdist, sol, world, rank, B
        self.slabs, self.stacks, self.works = [], [], [[], []]
        self.flag_off = 0
        if world > 1:
            lay, total = hsolver.result_slab_layout(net.H, net.n, net.q, B)
            self.flag_off = lay["err_h"][0]
            for _ in range(2):
                self.slabs.append(sol.alloc_result_slab(B))
                self.stacks.append(torch.empty((world, total), dtype=torch.uint8, device=sol.device) if rank == 0 else None)
        self.k = 0

    def wait(self, slot):
        if self.works[slot]:
            for w in self.works[slot]:
                w.wait()
            # hpf_solve_host_keep writes the slab from the library's own streams: the host must know the
            # gather that read it has completed (it was issued a whole step ago - this does not stall)
            self.torch.cuda.current_stream().synchronize()
        self.works[slot] = []

    def step(self, P, Q, I_N):
        if self.world == 1:
            return self.sol.solve_host(P, Q, I_N)
        slot = self.k & 1
        self.k += 1
        self.wait(slot)                                   # the gather that last used this slab
        res, slab = self.slabs[slot]
        r = self.sol.solve_host(P, Q, I_N, keep=res)
        _, self.works[slot] = self.hdist.gather_slab_to_root(slab, self.flag_off, 0, out=self.stacks[slot], async_op=True)
        return r

    def finish(self):
        self.wait(0); self.wait(1)
        self.torch.cuda.synchronize()

    def timed(self, P, Q, I_N, steps, barrier):
        barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = self.step(P, Q, I_N)
        self.finish()
        barrier()
        return time.perf_counter() - t0, r

    def phases(self, P, Q, I_N, hP, hQ, hI, barrier, reps=5):
        """Per-phase breakdown, each phase alone with all ranks running it at the same time (ms, this rank)."""
        torch = self.torch
        out = {}
        barrier(); t0 = time.perf_counter()
        for _ in range(reps):
            self.sol.solve_host(P, Q, I_N) if self.world == 1 else self.sol.solve_host(P, Q, I_N, keep=self.slabs[0][0])
        out["solve_host_call_ms"] = (time.perf_counter() - t0) / reps * 1e3
        dev = self.sol.device
        dP, dQ, dI = (torch.empty_like(x, device=dev) for x in (hP, hQ, hI))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); e0.record()
        for _ in range(reps):
            dP.copy_(hP, non_blocking=True); dQ.copy_(hQ, non_blocking=True); dI.copy_(hI, non_blocking=True)
        e1.record(); torch.cuda.synchronize()
        out["h2d_alone_ms"] = e0.elapsed_time(e1) / reps
        nbytes = sum(x.nbytes for x in self.sol._host_out)
        dsrc = torch.empty(nbytes, dtype=torch.uint8, device=dev)
        hdst = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
        barrier(); e0.record()
        for _ in range(reps):
            hdst.copy_(dsrc, non_blocking=True)
        e1.record(); torch.cuda.synchronize()
        out["d2h_alone_ms"] = e0.elapsed_time(e1) / reps
        out["d2h_GBps"] = nbytes / (out["d2h_alone_ms"] / 1e3) / 1e9
        if self.world > 1:
            barrier(); t0 = time.perf_counter()
            for _ in range(reps):
                _, w = self.hdist.gather_slab_to_root(self.slabs[0][1], self.flag_off, 0, out=self.stacks[0], async_op=True)
                for x in w:
                    x.wait()
                torch.cuda.synchronize()
            out["nccl_gather_alone_ms"] = (time.perf_counter() - t0) / reps * 1e3
        return out


def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    from harmonic_power_flow_b200 import dist as hdist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    cpu_pool = None
    if world == 1 and not a.no_cpu:        # fork the CPU workers BEFORE the CUDA context exists
        cpu_pool, OP, _ = oracle_pool()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the product path has no CPU fallback "
                         "(use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    affinity = None
    if world > 1:
        # one process per GPU: run on the CPUs next to this GPU, so that the pinned host buffers (first
        # touch) and the copy threads live on the GPU's own NUMA node / PCIe root
        try:
            import pynvml
            pynvml.nvmlInit()
            hnd = pynvml.nvmlDeviceGetHandleByIndex(local)
            pynvml.nvmlDeviceSetCpuAffinity(hnd)
            affinity = sorted(os.sched_getaffinity(0))
            affinity = "%d CPUs: %d..%d" % (len(affinity), affinity[0], affinity[-1])
        except Exception as e:                                   # not fatal: the numbers just stand as they are
            affinity = "not set (%s)" % type(e).__name__
        dist.init_process_group("nccl", device_id=dev)
    if a.gpus != world:
        a.gpus = world

    net = load_net()
    sol = BatchSolver(net, local)
    # weak scaling (default): a.batch scenarios per rank, rank r owns seeds r B .. (r+1) B - 1;
    # strong scaling: B_TARGET scenarios in total, rank r owns its contiguous shard
    s_lo, s_hi = hdist.shard_bounds(B_TARGET, world, rank)
    if a.strong:
        B, seed0 = s_hi - s_lo, s_lo
    else:
        B, seed0 = a.batch, rank * a.batch
    P, Q, I_N = scenarios.make_batch(net, B, SPREAD, seed0=seed0)
    hP = torch.as_tensor(P).pin_memory(); hQ = torch.as_tensor(Q).pin_memory()
    hI = torch.as_tensor(I_N).pin_memory()
    dP, dQ, dI = sol.prepare(hP, hQ, hI)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    N = sol.N
    n, H, q, m, c = net.n, net.H, net.q, net.m, net.c
    Nf = 2 * n - 1 - c

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def allreduce(vals):
        v = torch.tensor(vals, dtype=torch.float64, device=dev)
        if world == 1:
            return v.tolist(), v.tolist()
        mx = v.clone(); dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        sm = v.clone(); dist.all_reduce(sm, op=dist.ReduceOp.SUM)
        return mx.tolist(), sm.tolist()

    def device_timed(dP_, dQ_, dI_, steps, out_=None, **kw):
        """K steps, device-resident, CUDA events on the launch stream, L2 flushed before each step
        (the flush is outside the event pair).  -> (sum of step ms, result, per-kernel ms list)."""
        ev, kms = [], []
        for _ in range(steps):
            flush.fill_(1)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); out_ = sol.solve(dP_, dQ_, dI_, out=out_, **kw); e1.record()
            ev.append((e0, e1))
            kms.append(sol.last_kernel_ms())          # waits for this step's kernels
        torch.cuda.synchronize()
        return sum(x.elapsed_time(y) for x, y in ev), out_, kms

    # ---- device-resident timing (value) ----
    out = None
    for _ in range(a.warmup):
        out = sol.solve(dP, dQ, dI, out=out)
    sol.set_profiling(True)
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    l0 = sol.launch_count
    t_wall0 = time.perf_counter()
    ms, out, kms = device_timed(dP, dQ, dI, a.steps, out)
    barrier()
    t_wall = time.perf_counter() - t_wall0
    launches = sol.launch_count - l0
    if a.dump_outputs and rank == 0:
        dump_outputs(out, a.dump_outputs)
    ms_fund = sum(k[0] for k in kms) / a.steps
    ms_harm = sum(k[1] for k in kms) / a.steps
    conv = int((out.status == 0).sum().item())
    it_h = out.n_iter_h.double().sum().item()
    it_f = out.n_iter_f.double().sum().item()
    strategy = "structured" if sol.struct_info()["available"] else "dense"
    gpu_struct = None
    S_par = min(PARITY_SCENARIOS, B) if cpu_pool is not None else 0
    if S_par:
        gpu_struct = {k: getattr(out, k)[..., :S_par].cpu().numpy() for k in RESULT_KEYS}

    # ---- the same workload forced through the dense-LU kernel ----
    dense_info = gpu_dense = None
    if rank == 0 and not a.no_dense:
        od = sol.solve(dP, dQ, dI, dense=True)
        torch.cuda.synchronize()
        nd = 2
        tot, od, kd = device_timed(dP, dQ, dI, nd, od, dense=True)
        dense_info = dict(ms=tot / nd, kernel_ms=sum(k[1] for k in kd) / nd, conv=int((od.status == 0).sum().item()),
                          it_h=od.n_iter_h.double().sum().item(), it_f=od.n_iter_f.double().sum().item(),
                          iter_mismatch_vs_structured=int((od.n_iter_h != out.n_iter_h).sum().item()))
        if S_par:
            gpu_dense = {k: getattr(od, k)[..., :S_par].cpu().numpy() for k in RESULT_KEYS}
        del od

    # ---- small-batch / strong-scaling share, device-resident: B_TARGET / world scenarios on this rank ----
    strong = None
    if not a.strong:
        Bs = (s_hi - s_lo) if world > 1 else min(8192, B)        # N = 1: the 8-GPU share, as a probe of small batches
        if world > 1:
            Ps, Qs, Is = scenarios.make_batch(net, Bs, SPREAD, seed0=s_lo)
            hPs, hQs, hIs = (torch.as_tensor(x).pin_memory() for x in (Ps, Qs, Is))
            sP, sQ, sI = sol.prepare(hPs, hQs, hIs)
        else:
            sP, sQ, sI = dP[:, :Bs].contiguous(), dQ[:, :Bs].contiguous(), dI[:, :, :Bs].contiguous()
            hPs, hQs, hIs = (torch.as_tensor(np.ascontiguousarray(x[..., :Bs])).pin_memory() for x in (P, Q, I_N))
        so = sol.solve(sP, sQ, sI)
        barrier()
        ms_s, so, _ = device_timed(sP, sQ, sI, a.steps, so)
        barrier()
        strong = dict(Bs=Bs, ms=ms_s / a.steps, conv=int((so.status == 0).sum().item()),
                      host=(hPs.numpy(), hQs.numpy(), hIs.numpy()))
    sol.set_profiling(False)

    # ---- end to end through the host-buffer C-ABI entry point (e2e) ----
    npP, npQ, npI = hP.numpy(), hQ.numpy(), hI.numpy()
    e2e = E2E(torch, dist, sol, net, B, world, rank)
    for _ in range(max(1, a.warmup - 1)):
        r = e2e.step(npP, npQ, npI)
    e2e.finish()
    t_e2e, r = e2e.timed(npP, npQ, npI, a.steps, barrier)
    clk = clocks.stop()       # sampled over the device-timed AND the end-to-end region
    conv_e2e = int((r["status"] == 0).sum())
    h2d = npP.nbytes + npQ.nbytes + npI.nbytes
    d2h = sum(r[k].nbytes for k in RESULT_KEYS)
    phases = e2e.phases(npP, npQ, npI, hP, hQ, hI, barrier)
    # pageable host buffers (what a numpy caller of the reference holds): same call, N = 1 only
    t_pageable = None
    if world == 1:
        pgP, pgQ, pgI = P.copy(), Q.copy(), I_N.copy()
        sol.solve_host(pgP, pgQ, pgI)
        t0 = time.perf_counter()
        for _ in range(3):
            sol.solve_host(pgP, pgQ, pgI)
        t_pageable = (time.perf_counter() - t0) / 3
    # the reference's own return set (HG:560: V, err_h, n_iter_h - no Norton injection currents): same call with I_inj = NULL
    t_noinj = d2h_noinj = None
    if world == 1:
        rn = sol.solve_host(npP, npQ, npI, want_I_inj=False)
        t0 = time.perf_counter()
        for _ in range(a.steps):
            rn = sol.solve_host(npP, npQ, npI, want_I_inj=False)
        t_noinj = (time.perf_counter() - t0) / a.steps
        d2h_noinj = sum(rn[k].nbytes for k in RESULT_KEYS if rn[k] is not None)
    # strong-scaling share end to end
    if strong is not None:
        e2s = E2E(torch, dist, sol, net, strong["Bs"], world, rank)
        for _ in range(2):
            e2s.step(*strong["host"])
        e2s.finish()
        strong["t_e2e"], rs = e2s.timed(*strong["host"], a.steps, barrier)
        strong["conv_e2e"] = int((rs["status"] == 0).sum())
        del e2s

    # ---- standalone kernels against the HBM roofline (rank 0) ----
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    hbm_peak, hbm_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks \
        else (6650.0, "fallback (B200_PROFILING.md)")
    kernels = []
    fp64_peak = measure_fp64_peak(torch, dev)
    if rank == 0 and not a.no_kernels:
        def timed(fns, reps=12):
            """Average device time of one launch: `reps` launches captured in ONE CUDA graph and
            replayed between two events (no host launch overhead between the kernels: the Python
            wrapper costs ~30 us per call, as much as the mismatch kernel itself), rotating over
            input/output sets whose total footprint exceeds the 126 MB L2; best of 5 replays."""
            side = torch.cuda.Stream()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.stream(side):
                for fn in fns:
                    fn()
                torch.cuda.synchronize()
                with torch.cuda.graph(g, stream=side):
                    for r_ in range(reps):
                        fns[r_ % len(fns)]()
            torch.cuda.synchronize()
            best = float("inf")
            for _ in range(5):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                flush.fill_(1)
                e0.record(); g.replay(); e1.record(); torch.cuda.synchronize()
                best = min(best, e0.elapsed_time(e1) / reps)
            del g
            return best
        raw = sol.solve(dP, dQ, dI, raw=True, max_iter_h=3, want_I_inj=False)   # a mid-iteration state
        Vm, Va = raw.V_m, raw.V_a
        nset = 3                                             # 3 x 124 MB of traffic per rotation
        sets = [(Vm.clone(), Va.clone(), dP.clone(), dQ.clone(), dI.clone(),
                 (torch.empty((N, B), dtype=torch.float64, device=dev), torch.empty(B, dtype=torch.float64, device=dev)))
                for _ in range(nset)]
        t_mis = timed([(lambda s_=s_: sol.mismatch(s_[0], s_[1], s_[2], s_[3], s_[4], out=s_[5])) for s_ in sets])
        del sets
        by_mis = 16 * n * H + 8 * N + 16 * q * H + 16 * (m - 1) + 8
        tr, prov = ncu_traffic("mismatch_lane_kernel")
        kernels.append({"kernel": "mismatch_lane_kernel (one thread per scenario)", "bound": "hbm",
                        "ms": t_mis,
                        "achieved": by_mis * B / t_mis / 1e6, "peak": hbm_peak, "unit": "GB/s",
                        "frac": by_mis * B / t_mis / 1e6 / hbm_peak, "bytes_per_scenario": by_mis,
                        "frac_is_of": "ALGORITHMIC bytes (inputs read once + f written once), not DRAM bytes: under "
                                      "ncu part of the f output is still in L2 when the kernel ends",
                        "traffic": tr, "traffic_provenance": prov,
                        "timing": "CUDA graph of 12 launches over 3 rotating buffer sets (372 MB > L2), best of 5 replays"})
        Bj = min(B, 16384)
        Vmj, Vaj = Vm[:, :, :Bj].contiguous(), Va[:, :, :Bj].contiguous()
        Js = [sol.jacobian(Vmj, Vaj) for _ in range(2)]      # 2 x 1.35 GB outputs
        t_jac = timed([(lambda J_=J_: sol.jacobian(Vmj, Vaj, out=J_)) for J_ in Js], reps=6)
        J = Js[0]
        del Js
        by_jac = 8 * N * N + 16 * n * H
        tr, prov = ncu_traffic("jacobian_kernel")
        kernels.append({"kernel": "jacobian_kernel", "bound": "hbm", "ms": t_jac, "batch": Bj,
                        "achieved": by_jac * Bj / t_jac / 1e6, "peak": hbm_peak, "unit": "GB/s",
                        "frac": by_jac * Bj / t_jac / 1e6 / hbm_peak, "bytes_per_scenario": by_jac,
                        "traffic": tr, "traffic_provenance": prov})
        f, _ = sol.mismatch(Vmj, Vaj, dP[:, :Bj].contiguous(), dQ[:, :Bj].contiguous(), dI[:, :, :Bj].contiguous())
        t_lu = timed([lambda: sol.lu_solve(J, f)], reps=3)
        fl_lu = lu_flops(N)
        del J
        kernels.append({"kernel": "lu_solve_kernel", "bound": "fp64", "ms": t_lu, "batch": Bj,
                        "achieved": fl_lu * Bj / t_lu / 1e9, "peak": fp64_peak, "unit": "TFLOP/s",
                        "frac": fl_lu * Bj / t_lu / 1e9 / fp64_peak, "flops_per_scenario": fl_lu})

    # ---- the other BASELINE configurations (all ranks, weak scaling) ----
    other = None
    if not a.no_other:
        other = run_other_configs(torch, dist, BatchSolver, scenarios, local, rank, world, fp64_peak)

    # ---- reduce over ranks ----
    vals = [ms, t_e2e, float(conv), float(conv_e2e), it_h, it_f, t_wall, ms_harm, ms_fund] + \
           [phases.get(k, 0.0) for k in ("solve_host_call_ms", "h2d_alone_ms", "d2h_alone_ms", "nccl_gather_alone_ms")] + \
           [float(B)]
    if strong is not None:
        vals += [strong["ms"], strong["t_e2e"], float(strong["conv"]), float(strong["conv_e2e"])]
    mx, sm = allreduce(vals)
    ms_max, e2e_max = mx[0], mx[1]
    conv_tot, conv_e2e_tot, it_h_tot, it_f_tot, B_tot = sm[2], sm[3], sm[4], sm[5], sm[13]

    if rank == 0:
        value = conv_tot * a.steps / (ms_max / 1e3)
        e2e_v = conv_e2e_tot * a.steps / e2e_max
        # algorithmic FP64 work per Newton iteration of one scenario (DESIGN.md "Roofline accounting")
        nZ = n * H - m
        fl_mis = 8 * (H * n * n + q * H * H + (m - 1) * n)
        # structured step: u_Z = -V_Z - G (V_F + u_F) - w_N, polar conversion, small border system
        fl_struct = fl_mis + 8 * nZ * m + 10 * n * H + 8 * (2 * m) ** 2
        fl_dense = fl_mis + 16 * (H * n * n + q * H * H) + lu_flops(N)
        fl_f = 24 * n * n + lu_flops(Nf)
        # one FP64 sin + cos pair per phasor per iteration (Cody-Waite + two minimax polynomials): ~44 flops
        fl_sincos = 44 * n * H
        if strategy == "structured":
            kname = "harm_hw_kernel (harmonic Newton, structured step, one warp per harmonic, lane = scenario)"
            # n_iter+1 mismatches, n_iter steps
            flops = (it_h + B) * fl_mis + it_h * (fl_struct - fl_mis)
            flops_sc = flops + (it_h + B) * fl_sincos
            fl_iter = fl_struct
        else:
            kname = "solve_kernel<0> (fused fundamental + harmonic Newton, dense LU)"
            flops = it_h * fl_dense + it_f * fl_f
            flops_sc = flops + (it_h + B) * fl_sincos
            fl_iter = fl_dense
        t_kernel = ms_harm / 1e3
        ach = flops / t_kernel / 1e12
        ach_sc = flops_sc / t_kernel / 1e12
        by_solve = 16 * n + 16 * q * H + 16 * n * H + 16 * q * H + 24 + 2 * 16 * n   # in + out + fundamental hand-over
        sms = torch.cuda.get_device_properties(dev).multi_processor_count
        lanes = 2 * sms * 32                                      # 2 CTAs per SM x 32 scenario lanes
        traffic, prov = ncu_traffic("harm_hw_kernel") if strategy == "structured" else (None, None)
        step_ms = ms_max / a.steps
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": step_ms, "higher_is_better": True,
                "scaling": "strong" if a.strong else "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": config_dict(world, B, a.strong), "strategy": strategy,
                "converged_fraction": conv_tot / B_tot,
                "mean_nr_iterations": {"fundamental": it_f_tot / B_tot, "harmonic": it_h_tot / B_tot},
                "ns_per_scenario_nr_iteration": step_ms * 1e6 / max(it_h, 1.0),
                "newton_round_latency_us": {"value": mx[7] * 1e3 * lanes / max(it_h + B, 1.0),
                                            "what": "average duration of ONE Newton round (one iteration of all %d resident "
                                                    "scenario lanes of the GPU) = harmonic-kernel time x lanes / "
                                                    "(iterations + 1 per scenario); the latency a single scenario sees per "
                                                    "NR iteration inside the batch" % lanes},
                "gpu_launches": int(launches),
                "kernel_ms_per_step": {"fundamental_stage": mx[8], "harmonic_stage": mx[7]},
                "wall_s_timed_region": t_wall,
                "clocks": clk,
                "e2e": {"value": e2e_v, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                        "ms_per_step": e2e_max / a.steps * 1e3,
                        "host_buffers": "pinned (torch pin_memory); pageable numpy buffers through the same call: see pageable",
                        "cpu_affinity_rank0": affinity,
                        "path": ("BatchSolver.solve_host -> hpf_solve_host (C ABI, host buffers)" if world == 1 else
                                 "per rank: BatchSolver.solve_host(keep=slab) -> hpf_solve_host_keep (C ABI, host buffers: "
                                 "chunk-pipelined H2D / solve / D2H of the rank's own results to its own host buffers, "
                                 "results also left in one contiguous device slab) -> NCCL gather TO RANK 0 of the flags "
                                 "(20 B per scenario) and of the results, issued asynchronously: it overlaps the next "
                                 "step's solve; the timed region ends after the last gather"),
                        "phases_alone_ms_max_over_ranks": {
                            "solve_host_call": mx[9], "h2d_copy": mx[10], "d2h_copy": mx[11],
                            "nccl_gather_to_rank0": mx[12] if world > 1 else None,
                            "device_solve": step_ms,
                            "note": "each phase timed alone with all ranks running it concurrently; the step is "
                                    "bounded below by the D2H copy of the results over PCIe"},
                        "limiter": max([("solve_host_call (H2D + solve + D2H pipeline; PCIe D2H is its floor)", mx[9]),
                                        ("nccl_gather_to_rank0", mx[12] if world > 1 else 0.0)], key=lambda t: t[1])[0],
                        "host_path": {
                            "d2h_gbs_slowest_rank_all_ranks_copying": d2h / mx[11] / 1e6 if mx[11] else None,
                            "d2h_gbs_one_rank_alone": 56.0,
                            "what": "rate of the slowest rank's D2H copy of its result slab while all ranks copy at "
                                    "once (measured in this run) against one GPU copying alone on this pool "
                                    "(profiles/r2_host_path_8gpu.txt: with 8 ranks 12.0 / 18.8 GB/s per GPU, 123.5 GB/s "
                                    "in total): the multi-GPU end-to-end step is bounded "
                                    "by the host side of the box that all GPUs share, not by the solver"}},
                "roofline": {"kernel": kname, "bound": "fp64", "achieved": ach, "peak": fp64_peak,
                             "unit": "TFLOP/s", "frac": (ach / fp64_peak) if fp64_peak else None,
                             "achieved_incl_sincos": ach_sc,
                             "frac_incl_sincos": (ach_sc / fp64_peak) if fp64_peak else None,
                             "traffic": traffic, "traffic_provenance": prov,
                             "traffic_source": "dram__bytes_read.sum + dram__bytes_write.sum of one launch, ncu --set full",
                             "peak_source": "cuBLAS DGEMM 8192^3 burst measured in this run (no FP64 figure "
                                            "in MEASURED_PEAKS.json)",
                             "flops_per_nr_iteration": fl_iter,
                             "sincos_per_nr_iteration": n * H, "flops_per_sincos_pair": 44,
                             "note": "latency/issue-bound kernel; `achieved` counts the complex MACs of the mismatch and "
                                     "of the structured step only, `achieved_incl_sincos` adds the FP64 sin/cos pair per "
                                     "phasor per iteration (~44 flops each, evaluated in FP64 FMA arithmetic)",
                             "hbm_bytes_per_scenario": by_solve,
                             "hbm_gbs_of_whole_solve": by_solve * B / step_ms / 1e6},
                "roofline_kernels": kernels, "hbm_peak_source": hbm_src}
        if t_noinj is not None:
            line["e2e"]["without_I_inj"] = {"value": conv_e2e / t_noinj, "unit": UNIT, "ms_per_step": t_noinj * 1e3,
                                            "d2h_bytes_per_step": d2h_noinj,
                                            "what": "the same hpf_solve_host call returning what the reference's hpf() returns "
                                                    "(V_m, V_a, err_h, iteration counts, status); the headline e2e above also "
                                                    "copies back the Norton injection currents I_inj"}
        if t_pageable is not None:
            line["e2e"]["pageable"] = {"value": conv_e2e / t_pageable, "unit": UNIT, "ms_per_step": t_pageable * 1e3,
                                       "what": "the same hpf_solve_host call with ordinary (pageable) numpy arrays"}
        if strong is not None:
            # mx[14], mx[15]: device ms / e2e seconds of the share; sm[16], sm[17]: converged counts
            sv = sm[16] / (mx[14] / 1e3)
            se = sm[17] * a.steps / mx[15]
            line["strong_scaling"] = {
                "what": ("north-star target: %d scenarios IN TOTAL over %d GPU(s), %d per GPU" % (B_TARGET, world, strong["Bs"]))
                if world > 1 else
                ("N = 1 probe of the 8-GPU share of the north-star target: a batch of %d scenarios on one GPU" % strong["Bs"]),
                "batch_per_gpu": strong["Bs"], "value": sv, "unit": UNIT, "ms_per_step": mx[14],
                "e2e": {"value": se, "unit": UNIT, "ms_per_step": mx[15] / a.steps * 1e3},
                "per_scenario_efficiency_vs_full_batch": sv / value,
                "ms_ratio_vs_ideal": mx[14] / (step_ms * strong["Bs"] / B),
                "note": "ms_ratio_vs_ideal = ms per step of the share / (ms per full 65,536 step x share / 65,536); "
                        "1.0 = a small batch is as efficient per scenario as the full one"}
        if other is not None:
            line["other_configs"] = other
        if dense_info is not None:
            fld = dense_info["it_h"] * fl_dense + dense_info["it_f"] * fl_f
            achd = fld / (dense_info["kernel_ms"] / 1e3) / 1e12
            line["dense_lu_path"] = {
                "value": dense_info["conv"] / (dense_info["ms"] / 1e3), "unit": UNIT,
                "ms_per_step": dense_info["ms"],
                "iteration_count_mismatches_vs_structured": dense_info["iter_mismatch_vs_structured"],
                "roofline": {"kernel": "solve_kernel<0> (fused Newton, dense smem LU, warp-shuffle pivoting)",
                             "bound": "fp64", "achieved": achd, "peak": fp64_peak, "unit": "TFLOP/s",
                             "frac": achd / fp64_peak if fp64_peak else None,
                             "flops_per_nr_iteration": fl_dense}}
        if cpu_pool is not None:
            # the oracle on the SAME first S scenarios (one generator: scenario s is default_rng(s)
            # everywhere): timed as the CPU baseline, and its answers are the parity reference
            cores = cpu_pool.procs
            S = S_par
            ref = cpu_pool.solve(P[:, :S], Q[:, :S], I_N[:, :, :S], "superlu")
            lap = cpu_pool.solve(P[:, :S], Q[:, :S], I_N[:, :, :S], "lapack")
            cpu_pool.close()
            c_ = int((ref["status"] == 0).sum())
            line["cpu_baseline"] = {
                "value": c_ / ref["wall_s"], "unit": UNIT, "cores": cores, "kind": "port",
                "sample": "scenarios 0..%d of the same seeded workload, %d worker processes, %.1f s" % (
                    S - 1, cores, ref["wall_s"]),
                "ms_per_nr_iteration_per_core": ref["wall_s"] * 1e3 * cores / max(int(ref["n_iter_h"].sum()), 1)}
            par = {"scenarios": S,
                   "what": "iteration-count mismatches and scenarios whose phasors differ by > 1e-9 relative, against "
                           "the oracle port with the reference's SuperLU step on the SAME scenarios; `oracle_floor` = "
                           "the oracle with a LAPACK step against the oracle with the SuperLU step (the reference's "
                           "own sensitivity to round-off, SURVEY 7.3)",
                   "oracle_floor": OP.parity_rates(lap, ref)["vs_oracle"],
                   "gpu_structured": OP.parity_rates(gpu_struct, ref)["vs_oracle"]}
            if gpu_dense is not None:
                par["gpu_dense"] = OP.parity_rates(gpu_dense, ref)["vs_oracle"]
            fl_ = par["oracle_floor"]

            def within(g):
                lim = lambda k: k + 3.0 * (k + 1.0) ** 0.5          # floor + 3 sigma of its sampling error
                return bool(g["iteration_mismatches"] <= lim(fl_["iteration_mismatches"]) and
                            g["phasor_diff_gt_1e9"] <= lim(fl_["phasor_diff_gt_1e9"]))
            par["gpu_within_floor"] = {k: within(par[k]) for k in ("gpu_structured", "gpu_dense") if k in par}
            line["parity"] = par
        print(json.dumps(line))
    sol.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=B_PER_GPU, help="scenarios per GPU per step (weak scaling)")
    ap.add_argument("--strong", action="store_true", help="65,536 scenarios IN TOTAL, split over the ranks")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline / parity leg")
    ap.add_argument("--no-dense", action="store_true", help="skip the dense-LU comparison leg")
    ap.add_argument("--no-other", action="store_true", help="skip the other BASELINE configurations")
    ap.add_argument("--no-kernels", action="store_true", help="skip the standalone-kernel rooflines")
    ap.add_argument("--no-exec", action="store_true", help="reference arm: skip timing the reference's own code")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one returned (rank 0) as DIR/<name>.npy")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3) if a.impl == "ours" else a.warmup
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)


if __name__ == "__main__":
    main()
