"""Launch list of one build of the library over a fixed list of cases, for an A/B of two builds that must
issue the same kernels.  Loads the build given by $HPF_LIB (default: the in-tree library), runs every case
under torch.profiler with CUDA activities, and writes per case: the ordered list of kernel launches
(name, grid, block, shared memory, stream in order of first use; ordered by the launch's correlation id,
i.e. the order in which the host issued them), the hpf_launch_count delta of the case's handle, and a
sha1 of the case's outputs.  Two records are compared with --diff.

    HPF_LIB=/path/to/parent/libhpf_b200.so python profiles/tools/launch_list_ab.py --out parent.json
    python profiles/tools/launch_list_ab.py --out new.json
    python profiles/tools/launch_list_ab.py --diff parent.json new.json
"""
import argparse
import hashlib
import json
import os
import re
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "oracle")):
    sys.path.insert(0, p)
sys.dont_write_bytecode = True

# switches read at hpf_create / per call; every case starts from none of them set
SWITCHES = ["HPF_MAX_CTAS", "HPF_HARM_KERNEL", "HPF_NO_SPECIALISE", "HPF_STRUCT_VARIANT", "HPF_LOCKSTEP",
            "HPF_LOCKSTEP_GB", "HPF_GJ_SINGLE_MAX", "HPF_GJ_UNBLOCKED", "HPF_SETUP", "HPF_WN_KERNEL",
            "HPF_MISMATCH_TILE", "HPF_LU_CLASSIC", "HPF_HOST_PLAN", "HPF_HOST_STREAMS"]


def digest(outs):
    import numpy as np
    import torch
    h = hashlib.sha1()
    for o in outs:
        if o is None:
            h.update(b"none")
            continue
        a = o.detach().cpu().numpy() if isinstance(o, torch.Tensor) else np.asarray(o)
        h.update(str(a.dtype).encode() + str(a.shape).encode())
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


def result_outs(r):
    return [r.V_m, r.V_a, r.I_inj, r.n_iter_f, r.n_iter_h, r.err_h, r.status, r.err_hist_f, r.err_hist_h]


def cases(tmp):
    import numpy as np
    import bench
    import helpers
    from harmonic_power_flow_b200 import BatchSolver, scenarios

    nets = {}

    def net(key):
        if key not in nets:
            d = os.path.join(tmp, key)
            os.makedirs(d, exist_ok=True)
            if key == "meshed70":
                nets[key] = helpers.synthetic_packed("meshed", d, h_max=25, n=70, load_scale=0.02)[0]
            elif key in ("radial200", "meshed1000"):
                nets[key] = bench.load_other(key)
            else:
                name, cp, h = key.split("_")
                nets[key] = helpers.packed_from_files(name, int(h[1:]), cp == "c", d, julia_schema=name == "net1")[0]
        return nets[key]

    def batch(nt, B, seed=0):
        return scenarios.make_batch(nt, B, "tight", seed0=seed)

    def solves(key, B, dense=False, history=True, extra=()):
        """hpf_solve (and the standalone calls in `extra`) on one handle -> (launch delta, outputs)"""
        def run():
            nt = net(key)
            sol = BatchSolver(nt)
            P, Q, I_N = batch(nt, B)
            r = sol.solve(P, Q, I_N, history=history, dense=dense)
            outs = result_outs(r)
            for x in extra:
                outs += x(sol, nt, P, Q, I_N, r)
            n = sol.launch_count
            sol.close()
            return n, outs
        return run

    def standalone(sol, nt, P, Q, I_N, r):
        f, err = sol.mismatch(r.V_m, r.V_a, P, Q, I_N)
        return [f, err]

    def jac_lu(sol, nt, P, Q, I_N, r):
        J = sol.jacobian(r.V_m, r.V_a)
        f, _ = sol.mismatch(r.V_m, r.V_a, P, Q, I_N)
        dx, info = sol.lu_solve(J, f)
        return [J, dx, info]

    def step(sol, nt, P, Q, I_N, r):
        return [sol.newton_step(r.V_m, r.V_a, P, Q, I_N)]

    def wn(sol, nt, P, Q, I_N, r):
        return [sol.norton_wn(I_N)]

    def post(sol, nt, P, Q, I_N, r):
        st = sol.batch_stats(r.V_m, r.status, quantiles=(0.05, 0.5, 0.95))
        return [sol.thd(r.V_m), sol.bus_currents(r.V_m, r.V_a), st.status_counts, st.planes]

    def fund(sol, nt, P, Q, I_N, r):
        return list(sol.fund_solve(P, Q, history=True))

    def host(key, B):
        def run():
            nt = net(key)
            sol = BatchSolver(nt)
            P, Q, I_N = batch(nt, B)
            a = sol.solve_host(P, Q, I_N)
            outs = [a[k].copy() for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status")]
            k = sol.solve_host(P, Q, I_N, keep=True)
            outs += [k["V_m"].copy()] + result_outs(k["device"])[:7]
            s = sol.solve_host_stats(P, Q, I_N, quantiles=(0.5, 0.95), want_flags=True)
            outs += [s.status_counts, s.planes] + [s.flags[x] for x in ("n_iter_f", "n_iter_h", "err_h", "status")]
            n = sol.launch_count
            sol.close()
            return n, outs
        return run

    def ne():
        from harmonic_power_flow_b200 import ne_from_sim
        d = np.load(os.path.join(ROOT, "tests", "golden", "ne_extract_smps.npz"))
        o = ne_from_sim.get_NE_from_sim(ne_from_sim.Simulation(d["freq"], d["Vf"], d["Vh"], d["I_f"], d["I_h"]))
        return None, [o[k] for k in sorted(o) if isinstance(o[k], np.ndarray)]

    all_ = (standalone, jac_lu, step, wn, post, fund)
    v3 = {"HPF_STRUCT_VARIANT": "3"}
    return [
        ("net3_c_h25", {}, solves("net3_c_h25", 256, extra=all_)),
        ("net3_c_h25 tile", {"HPF_HARM_KERNEL": "tile"}, solves("net3_c_h25", 256)),
        ("net3_c_h25 no-specialise", {"HPF_NO_SPECIALISE": "1"}, solves("net3_c_h25", 256, extra=(standalone, step, wn))),
        ("net3_c_h25 max-ctas 2", {"HPF_MAX_CTAS": "2"}, solves("net3_c_h25", 256)),
        ("net3_c_h25 mismatch-tile", {"HPF_MISMATCH_TILE": "1"}, solves("net3_c_h25", 64, extra=(standalone,))),
        ("net3_c_h25 dense", {}, solves("net3_c_h25", 256, dense=True)),
        ("net3_c_h25 lu-classic", {"HPF_LU_CLASSIC": "1"}, solves("net3_c_h25", 64, dense=True, extra=(jac_lu,))),
        ("net3_uc_h25", {}, solves("net3_uc_h25", 256, extra=(standalone, step, wn))),
        ("net2ev_c_h19", {}, solves("net2ev_c_h19", 256, extra=all_)),
        ("net2ev_uc_h19", {}, solves("net2ev_uc_h19", 256, extra=(standalone, step, wn))),
        ("net2ev_c_h19 tile", {"HPF_HARM_KERNEL": "tile"}, solves("net2ev_c_h19", 256)),
        ("net2ev_c_h19 mismatch-tile", {"HPF_MISMATCH_TILE": "1"}, solves("net2ev_c_h19", 64, extra=(standalone,))),
        ("net2_c_h51", {}, solves("net2_c_h51", 128, extra=(standalone, jac_lu, step, wn))),
        ("net2_c_h51 dense", {}, solves("net2_c_h51", 64, dense=True)),
        ("net1_c_h25", {}, solves("net1_c_h25", 64, extra=all_)),
        ("net1_c_h25 lockstep 0", {"HPF_LOCKSTEP": "0"}, solves("net1_c_h25", 64, dense=True, extra=(jac_lu,))),
        ("net1_c_h51", {}, solves("net1_c_h51", 64, extra=(standalone, step))),
        ("net1_c_h51 dense", {"HPF_LOCKSTEP": "0"}, solves("net1_c_h51", 16, dense=True, extra=(jac_lu,))),
        ("net1_c_h51 batched lu", {"HPF_LOCKSTEP": "1"}, solves("net1_c_h51", 16, dense=True, extra=(jac_lu,))),
        ("net1_c_h25 wn fma", {"HPF_WN_KERNEL": "fma"}, solves("net1_c_h25", 64, extra=(wn,))),
        ("net1_c_h25 wn dmma", {"HPF_WN_KERNEL": "dmma"}, solves("net1_c_h25", 64, extra=(wn,))),
        ("meshed70 v3 lockstep 0", dict(v3, HPF_LOCKSTEP="0"), solves("meshed70", 96, extra=(standalone, step, wn))),
        ("meshed70 v3 lockstep 1", dict(v3, HPF_LOCKSTEP="1"), solves("meshed70", 96)),
        ("meshed70 v3 lockstep 1 waves", dict(v3, HPF_LOCKSTEP="1", HPF_LOCKSTEP_GB="0.002"), solves("meshed70", 96)),
        ("meshed70 v3 max-ctas 2", dict(v3, HPF_LOCKSTEP="0", HPF_MAX_CTAS="2"), solves("meshed70", 32)),
        ("meshed70 v3 gj blocked", dict(v3, HPF_LOCKSTEP="0", HPF_GJ_SINGLE_MAX="0"), solves("meshed70", 32)),
        ("meshed70 v3 gj unblocked", dict(v3, HPF_LOCKSTEP="0", HPF_GJ_SINGLE_MAX="0", HPF_GJ_UNBLOCKED="1"),
         solves("meshed70", 32)),
        ("meshed70 v3 setup gj", dict(v3, HPF_LOCKSTEP="0", HPF_SETUP="gj", HPF_GJ_SINGLE_MAX="0"), solves("meshed70", 32)),
        ("meshed70 v3 wn fma", dict(v3, HPF_LOCKSTEP="0", HPF_WN_KERNEL="fma"), solves("meshed70", 32, extra=(wn,))),
        ("meshed70 dense", {}, solves("meshed70", 16, dense=True)),
        ("net3_c_h25 host plan", {"HPF_HOST_PLAN": "64,128"}, host("net3_c_h25", 1024)),
        ("meshed70 v3 host plan", dict(v3, HPF_LOCKSTEP="1", HPF_HOST_PLAN="64"), host("meshed70", 160)),
        ("ne_extract", {}, ne),
        ("radial200", {"HPF_LOCKSTEP": "1"}, solves("radial200", 128)),
        ("radial200 lockstep 0", {"HPF_LOCKSTEP": "0"}, solves("radial200", 16, extra=(standalone, step))),
        ("meshed1000", {"HPF_LOCKSTEP": "1"}, solves("meshed1000", 32)),
        ("meshed1000 lockstep 0", {"HPF_LOCKSTEP": "0"}, solves("meshed1000", 4)),
    ]


def record(out, only=None):
    import torch
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.set_device(0)
    res = {"lib": os.environ.get("HPF_LIB", "in-tree"), "cases": {}}
    with tempfile.TemporaryDirectory(prefix="hpf_ab_") as tmp:
        for name, env, fn in cases(tmp):
            if only and only not in name:
                continue
            for k in SWITCHES:
                os.environ.pop(k, None)
            os.environ.update(env)
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                try:
                    n, outs = fn()
                except Exception as e:            # recorded: both builds must fail the same way
                    n, outs = repr(e), []
                torch.cuda.synchronize()
            path = os.path.join(tmp, "trace.json")
            prof.export_chrome_trace(path)
            ev = [e for e in json.load(open(path))["traceEvents"] if e.get("cat") == "kernel"]
            os.remove(path)
            ev.sort(key=lambda e: e["args"]["correlation"])
            streams = {}
            lst = [[e["name"], e["args"].get("grid"), e["args"].get("block"), e["args"].get("shared memory"),
                    streams.setdefault(e["args"].get("stream"), len(streams))] for e in ev]
            res["cases"][name] = {"launch_count": n, "kernels": lst, "outputs": digest(outs)}
            print("%-36s %6d kernels, launch count %s, outputs %s" % (name, len(lst), n, res["cases"][name]["outputs"][:12]),
                  flush=True)
    for k in SWITCHES:
        os.environ.pop(k, None)
    json.dump(res, open(out, "w"))


def diff(a_path, b_path, sass_names=None):
    a, b = json.load(open(a_path))["cases"], json.load(open(b_path))["cases"]
    bad = 0
    for name in sorted(set(a) | set(b)):
        if name not in a or name not in b:
            print("%s: only in %s" % (name, a_path if name in a else b_path)); bad += 1
            continue
        x, y = a[name], b[name]
        same = [x[k] == y[k] for k in ("kernels", "launch_count", "outputs")]
        print("%-36s kernels %6d %s  launch count %s %s  outputs %s" % (
            name, len(x["kernels"]), "same" if same[0] else "DIFFER (%d)" % len(y["kernels"]),
            x["launch_count"], "same" if same[1] else "DIFFER (%s)" % y["launch_count"], "same" if same[2] else "DIFFER"))
        if not same[0]:
            for i, (p, q) in enumerate(zip(x["kernels"], y["kernels"])):
                if p != q:
                    print("   first difference at launch %d: %s | %s" % (i, p, q)); break
        bad += not all(same)
    # a kernel is named by its function and template arguments (the profiler and c++filt print types apart)
    key = lambda s: re.sub(r"\s+", "", s.split("(")[0]).replace("void", "", 1) if s.startswith("void") else \
        re.sub(r"\s+", "", s.split("(")[0])
    seen = {key(k[0]) for c in b.values() for k in c["kernels"]}
    print("kernel names seen: %d" % len(seen))
    if sass_names:
        names = [l.strip() for l in open(sass_names) if l.strip()]
        miss = [n for n in names if key(n) not in seen]
        print("functions of the SASS: %d, not seen: %d %s" % (len(names), len(miss), miss))
    print("RESULT: %s" % ("identical" if bad == 0 else "%d case(s) differ" % bad))
    return bad


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out")
    ap.add_argument("--only", help="run the cases whose name contains this")
    ap.add_argument("--diff", nargs=2)
    ap.add_argument("--sass-names", help="file of demangled function names (cuobjdump -sass | c++filt) to cover")
    a = ap.parse_args()
    if a.diff:
        sys.exit(1 if diff(*a.diff, a.sass_names) else 0)
    record(a.out, a.only)


if __name__ == "__main__":
    main()
