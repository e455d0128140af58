"""GPU parity tests: the CUDA path (through the C ABI) against the committed fixtures that
the reference itself produced (tests/golden/) and against the CPU oracle on seeded inputs.

Tolerances (FP64): Y(h), mismatch and Jacobian are elementwise formulas -> 1e-13 relative.
One Newton step is limited by cond(J) ~ 1e5..2e7 -> 1e-8.  Converged results are compared as
phasors to 1e-9 relative where the reference agrees with ITSELF to that level (its SuperLU
step vs a LAPACK step, stored in the fixtures), see SURVEY 7.3."""
import numpy as np
import pytest
import torch

import helpers
import hpf_oracle as O
from conftest import GOLDEN

pytestmark = pytest.mark.gpu

SMALL_CASES = ["net2_uc_h51", "net2_c_h51", "net2_c_h19", "net3_c_h25", "net3_uc_h25",
               "net2ev_c_h19", "net2ev_uc_h19", "net3_c_h5"]
ALL_CASES = SMALL_CASES + ["net1_c_h25", "net1_uc_h51", "net1_c_h51"]


@pytest.fixture(scope="module")
def solvers(tmp_path_factory):
    from harmonic_power_flow_b200 import BatchSolver
    cache = {}

    def get(case):
        if case not in cache:
            d = helpers.load_case(case)
            net, st, _ = helpers.packed_from_files(str(d["net"]), int(d["h_max"]), bool(d["coupled"]),
                                                   tmp_path_factory.mktemp(case),
                                                   julia_schema=str(d["net"]) == "net1")
            cache[case] = (BatchSolver(net), net, d)
        return cache[case]
    yield get
    for s, _, _ in cache.values():
        s.close()


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max()


# ---------------------------------------------------------------- kernel 1
@pytest.mark.parametrize("case", ALL_CASES)
def test_ybus_matches_reference(solvers, case):
    sol, net, d = solvers(case)
    Y = sol.Y.cpu().numpy()
    assert Y.shape == d["Y_all"].shape
    assert _rel(Y, d["Y_all"]) <= 1e-15
    assert np.array_equal(Y == 0, d["Y_all"] == 0)          # same sparsity pattern


def test_ybus_quirks_parallel_lines_and_pi_shunt(tmp_path):
    """HG:150-155 (parallel lines overwrite) and HG:163-168 (pi-shunt lands on bus ID+1)."""
    from harmonic_power_flow_b200 import BatchSolver
    net, _, _ = helpers.packed_from_files("net3", 7, True, tmp_path)
    net.from_id = np.append(net.from_id, [1, 2]).astype(np.int32)
    net.to_id = np.append(net.to_id, [2, 3]).astype(np.int32)
    net.R = np.append(net.R, [0.01, 0.02]); net.X = np.append(net.X, [0.03, 0.01])
    net.G = np.append(net.G * 0 + 0.001, [0.002, 0.0]); net.B = np.append(net.B * 0 + 0.004, [0.0, 0.003])
    sol = BatchSolver(net)
    on = O.Net(n=net.n, m=net.m, c=net.c, harmonics=net.harmonics, line_from=net.from_id, line_to=net.to_id,
               R=net.R, X=net.X, G=net.G, B=net.B, X_sh=net.X_sh, P=net.P, Q=net.Q)
    Yo = O.build_admittance_matrices(on)
    assert _rel(sol.Y.cpu().numpy(), Yo) <= 1e-15
    sol.close()


# ---------------------------------------------------------------- fundamental stage
@pytest.mark.parametrize("case", ALL_CASES)
def test_fundamental_newton_matches_reference(solvers, case):
    sol, net, d = solvers(case)
    V_m, V_a, nf, err, hist = sol.fund_solve(net.P[:, None], net.Q[:, None], history=True)
    assert int(nf.item()) == int(d["n_iter_f"])
    V = helpers.phasor(V_m[:, :, 0].cpu().numpy(), V_a[:, :, 0].cpu().numpy())
    assert np.abs(V - helpers.phasor(d["V_fund_m"], d["V_fund_a"])).max() < 1e-12
    h = hist[:, 0].cpu().numpy()
    k = len(d["err_f_hist"])
    assert np.allclose(h[:k], d["err_f_hist"], rtol=1e-6, atol=1e-12)   # last entry is round-off
    assert np.isnan(h[k:]).all()


# ---------------------------------------------------------------- kernel 2
@pytest.mark.parametrize("case", ALL_CASES)
def test_mismatch_matches_reference(solvers, case):
    sol, net, d = solvers(case)
    Vm, Va = d["V_fund_m"][:, :, None], d["V_fund_a"][:, :, None]
    f, err, inj = sol.mismatch(Vm, Va, net.P[:, None], net.Q[:, None], net.I_N[:, :, None], want_I_inj=True)
    f = f[:, 0].cpu().numpy()
    assert f.shape == d["f0"].shape
    assert _rel(f, d["f0"]) <= 1e-13
    assert float(err.item()) == pytest.approx(np.abs(d["f0"]).max(), rel=1e-13)
    on = O.net_from_golden(GOLDEN, str(d["net"]), int(d["h_max"]), bool(d["coupled"]))
    inj_o = O.current_injections(on, helpers.phasor(d["V_fund_m"], d["V_fund_a"]), on.I_N)
    assert _rel(inj[:, :, 0].cpu().numpy(), inj_o) <= 1e-13


def test_mismatch_ragged_batch_and_nan(solvers):
    """B not a multiple of the 32-scenario tile; NaN in one scenario must not leak."""
    sol, net, d = solvers("net3_c_h25")
    B = 77
    rng = np.random.default_rng(5)
    Vm = np.repeat(d["V_fund_m"][:, :, None], B, 2) * rng.uniform(0.9, 1.1, (net.H, net.n, B))
    Va = np.repeat(d["V_fund_a"][:, :, None], B, 2) + rng.uniform(-0.1, 0.1, (net.H, net.n, B))
    P = np.repeat(net.P[:, None], B, 1); Q = np.repeat(net.Q[:, None], B, 1)
    I_N = np.repeat(net.I_N[:, :, None], B, 2)
    Vm[2, 1, 40] = np.nan
    f, err = sol.mismatch(Vm, Va, P, Q, I_N)
    f, err = f.cpu().numpy(), err.cpu().numpy()
    on = O.net_from_golden(GOLDEN, "net3", 25, True)
    Y = O.build_admittance_matrices(on)
    for b in (0, 31, 32, 63, 76):
        fo, eo = O.harmonic_mismatch(on, on.P, on.Q, Vm[:, :, b], Va[:, :, b], Y, on.I_N)
        assert _rel(f[:, b], fo) <= 1e-13 and err[b] == pytest.approx(eo, rel=1e-13)
    assert np.isnan(err[40]) and np.isfinite(np.delete(err, 40)).all()


# ---------------------------------------------------------------- kernel 3
@pytest.mark.parametrize("case", SMALL_CASES + ["net1_c_h25"])
def test_jacobian_matches_reference(solvers, case):
    sol, net, d = solvers(case)
    Vm, Va = d["V_fund_m"][:, :, None], d["V_fund_a"][:, :, None]
    J = sol.jacobian_view(sol.jacobian(Vm, Va))[0].cpu().numpy()
    if "J0" in d:
        Jg = d["J0"]
    else:
        Jg = np.zeros((net.N, net.N)); Jg[d["J0_rows"], d["J0_cols"]] = d["J0_vals"]
    assert J.shape == Jg.shape
    assert _rel(J, Jg) <= 1e-13
    assert np.array_equal(J != 0, Jg != 0)                   # nnz pattern of SURVEY 4.3


def test_jacobian_batch_with_negative_magnitudes(solvers):
    """Signed-V_m normalisation (HG:405,455): iterates with V_m < 0 must match the oracle."""
    sol, net, d = solvers("net2ev_c_h19")
    B = 5
    rng = np.random.default_rng(11)
    Vm = rng.uniform(-0.3, 0.3, (net.H, net.n, B)); Vm[0] = rng.uniform(0.9, 1.1, (net.n, B))
    Va = rng.uniform(-4, 4, (net.H, net.n, B))
    J = sol.jacobian_view(sol.jacobian(Vm, Va)).cpu().numpy()
    on = O.net_from_golden(GOLDEN, "net2ev", 19, True)
    Y = O.build_admittance_matrices(on)
    for b in range(B):
        assert _rel(J[b], O.build_harmonic_jacobian(on, Vm[:, :, b], Va[:, :, b], Y)) <= 1e-13


# ---------------------------------------------------------------- kernel 4
@pytest.mark.parametrize("case", SMALL_CASES)
def test_lu_solve_newton_step(solvers, case):
    sol, net, d = solvers(case)
    Vm, Va = d["V_fund_m"][:, :, None], d["V_fund_a"][:, :, None]
    J = sol.jacobian(Vm, Va)
    f = torch.as_tensor(d["f0"][:, None])
    dx, info = sol.lu_solve(J, f)
    assert int(info.item()) == 0
    dx = dx[:, 0].cpu().numpy()
    Jd = d["J0"]
    # backward error of the GPU LU (partial pivoting): ~ eps
    resid = np.abs(Jd @ dx - d["f0"]).max() / (np.abs(Jd).max() * np.abs(dx).max())
    assert resid < 1e-13
    x0 = helpers.state_vectors(d["V_fund_m"], d["V_fund_a"], net.c)
    assert np.abs((x0 - dx) - d["x1"]).max() <= 1e-8 * np.abs(d["x1"]).max()


@pytest.mark.parametrize("case,B", [("net3_c_h5", 67), ("net2_c_h51", 9), ("net1_c_h25", 7), ("net1_c_h51", 7)])
def test_lu_solve_random_batch_and_singular(solvers, case, B):
    """Shared-memory LU (N <= 192) and the blocked global-memory LU with the tensor-core
    trailing update (N = 206, 518, 1038: several panels, ragged last panel / slices)."""
    sol, net, d = solvers(case)
    N = sol.N
    rng = np.random.default_rng(3)
    A = rng.standard_normal((B, N, N))
    A[5, :, 3] = 0.0                                         # exactly singular -> zero pivot
    f = rng.standard_normal((N, B))
    stride = sol.jacobian_stride()
    J = torch.zeros((B, stride), dtype=torch.float64, device=sol.device)
    J[:, :N * N] = torch.as_tensor(A.reshape(B, -1)).to(sol.device)
    dx, info = sol.lu_solve(J, f)
    dx, info = dx.cpu().numpy(), info.cpu().numpy()
    assert info[5] != 0 and (np.delete(info, 5) == 0).all()
    for b in range(B):
        if b == 5:
            continue
        ref = np.linalg.solve(A[b], f[:, b])
        assert np.abs(dx[:, b] - ref).max() <= 1e-9 * max(1.0, np.abs(ref).max())


@pytest.mark.parametrize("case,B", [("net3_c_h25", 70), ("net3_c_h5", 33), ("net2_c_h51", 9), ("net2ev_c_h19", 40)])
def test_panel_lu_is_bit_identical_to_rank1_lu(solvers, case, B, monkeypatch):
    """Kernel 4: the panel-blocked shared-memory LU (hpf_lu_panel.cuh, default) applies to every
    matrix element exactly the FMAs of the rank-1 elimination (lu_solve_smem, $HPF_LU_CLASSIC=1) in
    the same order, with the same pivots: dx, info and the whole fused dense solve (iteration
    counts, error history, phasors) are BIT-identical.  Includes N not a multiple of the panel
    width (N = 101, 21, 206 -> blocked LU instead, 78) and a singular matrix."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    sol, net, d = solvers(case)
    P, Q, I_N = scenarios.make_batch(net, B, "wide")
    raw = sol.solve(P, Q, I_N, raw=True, max_iter_h=2)
    f, _ = sol.mismatch(raw.V_m, raw.V_a, P, Q, I_N)
    J = sol.jacobian(raw.V_m, raw.V_a)
    Jv = sol.jacobian_view(J)
    Jv[B // 2, 3, :] = Jv[B // 2, 5, :]                      # one exactly singular matrix
    dx, info = sol.lu_solve(J, f)
    full = sol.solve(P, Q, I_N, dense=True, history=True).to_host()
    monkeypatch.setenv("HPF_LU_CLASSIC", "1")
    classic = BatchSolver(net)
    dx0, info0 = classic.lu_solve(J, f)
    full0 = classic.solve(P, Q, I_N, dense=True, history=True).to_host()
    classic.close()
    ok = torch.ones(B, dtype=torch.bool, device=dx.device)
    ok[B // 2] = False
    assert torch.equal(info, info0) and int(info[B // 2]) != 0 and int((info[ok] != 0).sum()) == 0
    assert torch.equal(dx[:, ok], dx0[:, ok])
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status", "err_hist_f", "err_hist_h"):
        assert np.array_equal(full[k], full0[k], equal_nan=True), k
    # and it solves the system: residual against the row-major Jacobian
    res = torch.einsum("bij,jb->ib", Jv[ok], dx[:, ok]) - f[:, ok]
    assert float(res.abs().max()) <= 1e-9 * float(f.abs().max())


# ---------------------------------------------------------------- fused solve
@pytest.mark.parametrize("strategy", ["structured", "dense"])
@pytest.mark.parametrize("case", SMALL_CASES)
def test_fused_solve_nominal_cases(solvers, case, strategy):
    """Every nominal fixture on BOTH Newton-step strategies - "structured" is the default kernel
    the headline number runs on (harm_hw_kernel / harm_tile_kernel), with the per-iteration error
    history: exact iteration counts, V within 1e-9, the reference's error path, THD."""
    sol, net, d = solvers(case)
    if strategy == "structured":
        assert sol.struct_info()["available"] == 1
    r = sol.solve(net.P[:, None], net.Q[:, None], net.I_N[:, :, None], history=True, dense=(strategy == "dense"))
    assert int(r.n_iter_f.item()) == int(d["n_iter_f"])
    assert int(r.n_iter_h.item()) == int(d["n_iter_h"])           # identical iteration counts
    assert int(r.status.item()) == 0
    V = helpers.phasor(r.V_m[:, :, 0].cpu().numpy(), r.V_a[:, :, 0].cpu().numpy())
    Vg = helpers.phasor(d["V_m"], d["V_a"])
    tol = 1e-9 if float(d["err_h"]) < 1e-6 else 1e-7             # poorly converged last step: noise floor
    assert (np.abs(V - Vg) / np.abs(Vg)).max() < tol
    Va = r.V_a[:, :, 0].cpu().numpy()
    assert (Va >= 0).all() and (Va <= 2 * np.pi).all() and (r.V_m.cpu().numpy() >= 0).all()
    hist = r.err_hist_h[:, 0].cpu().numpy()
    k = len(d["err_h_hist"])
    assert np.isnan(hist[k:]).all() and np.isfinite(hist[:k]).all()
    hf = r.err_hist_f[:, 0].cpu().numpy()
    kf = len(d["err_f_hist"])
    assert np.isnan(hf[kf:]).all() and np.allclose(hf[:kf], d["err_f_hist"], rtol=1e-6, atol=1e-11)
    # the error PATH, not only the end: tight at the start, then round-off is amplified by the
    # non-contractive early iterations (cond(J) up to 2e7, SURVEY 7.3)
    assert np.allclose(hist[:4], d["err_h_hist"][:4], rtol=1e-9)
    assert np.allclose(hist[:k - 1], d["err_h_hist"][:k - 1], rtol=0.05)
    assert hist[k - 1] == pytest.approx(float(r.err_h.item()))
    thd = sol.thd(r.V_m)[:, :, 0].cpu().numpy().T
    assert np.abs(thd - d["THD"]).max() < 1e-7


@pytest.mark.parametrize("strategy", ["structured", "dense"])
@pytest.mark.parametrize("name", ["net3_c_h25_tight", "net3_c_h25_wide", "net2ev_c_h19_tight",
                                  "net3_uc_h25_tight"])
def test_fused_solve_scenario_sets_vs_reference(solvers, name, strategy):
    d = helpers.load_set(name)
    case = name.rsplit("_", 1)[0]
    sol, net, _ = solvers(case)
    S = len(d["seed"])
    P, Q, I_N = d["P"].T.copy(), d["Q"].T.copy(), np.moveaxis(d["I_N"], 0, 2).copy()
    if strategy == "structured":
        assert sol.struct_info()["available"]
    r = sol.solve(P, Q, I_N, dense=(strategy == "dense")).to_host()
    assert (r["n_iter_f"] == d["n_iter_f"]).all()
    assert (r["status"] == 0).all()
    V = np.moveaxis(helpers.phasor(r["V_m"], r["V_a"]), 2, 0)
    Vg = helpers.phasor(d["V_m"], d["V_a"])
    Vl = helpers.phasor(d["V_m_lapack"], d["V_a_lapack"])
    rel = (np.abs(V - Vg) / np.abs(Vg)).reshape(S, -1).max(1)
    floor = (np.abs(Vl - Vg) / np.abs(Vg)).reshape(S, -1).max(1)
    mism = int((r["n_iter_h"] != d["n_iter_h"]).sum())
    floor_mism = int((d["n_iter_h"] != d["n_iter_h_lapack"]).sum())
    print("\n%s [%s]: GPU-vs-reference iteration mismatches %d/%d (reference SuperLU-vs-LAPACK: %d); "
          "phasor rel diff > 1e-9: %d (reference floor: %d); max %.2e (floor %.2e); median %.2e"
          % (name, strategy, mism, S, floor_mism, (rel > 1e-9).sum(), (floor > 1e-9).sum(), rel.max(),
             floor.max(), np.median(rel)))
    assert mism <= floor_mism + 1
    assert (rel > 1e-9).sum() <= (floor > 1e-9).sum() + max(2, S // 20)
    assert np.median(rel) < 1e-11
    same = r["n_iter_h"] == d["n_iter_h"]
    assert rel[same].max() < 1e-5


@pytest.mark.parametrize("case", SMALL_CASES)
def test_structured_newton_step_equals_dense_step(solvers, case):
    """hpf_newton_step (block elimination through A_ZZ^-1) against J^-1 f: the reference's
    first update x1, and random iterates against numpy on the oracle's Jacobian."""
    sol, net, d = solvers(case)
    info = sol.struct_info()
    assert info["available"] == 1 and info["nZ"] == net.n * net.H - net.m
    Vm, Va = d["V_fund_m"][:, :, None], d["V_fund_a"][:, :, None]
    dx = sol.newton_step(Vm, Va, net.P[:, None], net.Q[:, None], net.I_N[:, :, None])[:, 0].cpu().numpy()
    x0 = helpers.state_vectors(d["V_fund_m"], d["V_fund_a"], net.c)
    assert np.abs((x0 - dx) - d["x1"]).max() <= 1e-8 * np.abs(d["x1"]).max()
    # residual of the step against the reference's own Jacobian and mismatch
    Jd = d["J0"]
    assert np.abs(Jd @ dx - d["f0"]).max() <= 1e-10 * np.abs(d["f0"]).max()
    on = O.net_from_golden(GOLDEN, str(d["net"]), int(d["h_max"]), bool(d["coupled"]))
    Y = O.build_admittance_matrices(on)
    B = 40
    rng = np.random.default_rng(17)
    Vmb = rng.uniform(0.05, 0.3, (net.H, net.n, B)) * rng.choice([-1.0, 1.0], (net.H, net.n, B))
    Vmb[0] = rng.uniform(0.9, 1.1, (net.n, B))
    Vab = rng.uniform(-3, 3, (net.H, net.n, B)); Vab[0, 0] = 0.0; Vmb[0, 0] = 1.0
    P = np.repeat(net.P[:, None], B, 1) * rng.uniform(0.8, 1.2, (net.n, B))
    Q = np.repeat(net.Q[:, None], B, 1) * rng.uniform(0.8, 1.2, (net.n, B))
    I_N = np.repeat(net.I_N[:, :, None], B, 2) * rng.uniform(0.9, 1.1, (net.q, net.H, B))
    dxb = sol.newton_step(Vmb, Vab, P, Q, I_N).cpu().numpy()
    for b in range(0, B, 3):
        J = O.build_harmonic_jacobian(on, Vmb[:, :, b], Vab[:, :, b], Y)
        f, _ = O.harmonic_mismatch(on, P[:, b], Q[:, b], Vmb[:, :, b], Vab[:, :, b], Y, I_N[:, :, b])
        ref = np.linalg.solve(J, f)
        assert np.abs(dxb[:, b] - ref).max() <= 1e-7 * np.abs(ref).max()
        assert np.abs(J @ dxb[:, b] - f).max() <= 1e-9 * np.abs(f).max()


def test_host_buffer_entry_point_is_bit_identical(solvers):
    sol, net, _ = solvers("net3_c_h25")
    d = helpers.load_set("net3_c_h25_tight")
    P, Q, I_N = d["P"].T.copy(), d["Q"].T.copy(), np.moveaxis(d["I_N"], 0, 2).copy()
    a = sol.solve(P, Q, I_N).to_host()
    b = sol.solve_host(P, Q, I_N)
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(a[k], b[k]), k
    # the reference's return set (no Norton injection currents): I_inj = NULL in the C call
    c = sol.solve_host(P, Q, I_N, want_I_inj=False)
    assert c["I_inj"] is None
    for k in ("V_m", "V_a", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(a[k], c[k]), k


def test_host_entry_point_keeps_device_copy(solvers):
    """hpf_solve_host_keep: the device-resident copy of the results (what a multi-GPU run feeds to
    its final NCCL gather) equals the host results bit for bit, on a chunked batch."""
    from harmonic_power_flow_b200 import scenarios
    sol, net, _ = solvers("net3_c_h25")
    B = 20000
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    r = sol.solve_host(P, Q, I_N, keep=True)
    dev = r["device"].to_host()
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(dev[k], r[k]), k
    assert (r["status"] == 0).all()


def test_host_entry_point_chunked_pipeline(solvers, tmp_path):
    """B large enough for the 4-chunk copy/solve/copy pipeline with a ragged last chunk: same
    bits as the device-resident call (results do not depend on the position in the batch)."""
    from harmonic_power_flow_b200 import scenarios
    sol, net, _ = solvers("net3_c_h25")
    B = 40001
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    a = sol.solve(P, Q, I_N).to_host()
    b = sol.solve_host(P, Q, I_N)
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(a[k], b[k]), k
    assert (b["status"] == 0).all()


@pytest.mark.parametrize("plan,streams,B", [("96,160,1000,64", 3, 4099), ("32", 4, 2001), ("4096,8192,12288,16384", 2, 70001),
                                             ("100000", 2, 777)])
def test_host_entry_point_chunk_plans(solvers, monkeypatch, plan, streams, B):
    """$HPF_HOST_PLAN / $HPF_HOST_STREAMS (growing chunks of hpf_solve_host over 1..4 compute streams,
    more sizes than chunk slots, a last chunk of odd length, a plan larger than the batch): host results
    and the device copy of hpf_solve_host_keep carry the bits of the device-resident call, and the
    per-chunk w_N scratch of the call leaves hpf_norton_wn unchanged."""
    from harmonic_power_flow_b200 import scenarios
    sol, net, _ = solvers("net3_c_h25")
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    a = sol.solve(P, Q, I_N).to_host()
    wn = sol.norton_wn(I_N).cpu().numpy()
    monkeypatch.setenv("HPF_HOST_PLAN", plan)
    monkeypatch.setenv("HPF_HOST_STREAMS", str(streams))
    b = sol.solve_host(P, Q, I_N, keep=True)
    dev = b["device"].to_host()
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(a[k], b[k]), k
        assert np.array_equal(a[k], dev[k]), k
    assert (b["status"] == 0).all()
    assert np.array_equal(sol.norton_wn(I_N).cpu().numpy(), wn)


def test_fused_solve_equals_stepwise_kernels(solvers, tmp_path, monkeypatch):
    """The fused kernel and a host loop over kernels 2-4 share their arithmetic: identical
    iteration counts and (bitwise) identical iterates.  (The standalone mismatch is forced onto
    the 32-scenario tile kernel, the variant that shares hpf_device.cuh with the fused kernel;
    the default one-thread-per-scenario variant is compared with it in the next test.)"""
    from harmonic_power_flow_b200 import BatchSolver
    monkeypatch.setenv("HPF_MISMATCH_TILE", "1")
    net, _, _ = helpers.packed_from_files("net3", 25, True, tmp_path)
    sol = BatchSolver(net)
    d = helpers.load_set("net3_c_h25_tight")
    S = 8
    P, Q, I_N = d["P"][:S].T.copy(), d["Q"][:S].T.copy(), np.moveaxis(d["I_N"][:S], 0, 2).copy()
    fused = sol.solve(P, Q, I_N, raw=True, dense=True).to_host()
    V_m, V_a, nf, _, _ = sol.fund_solve(P, Q)
    nH, c = net.n * net.H, net.c
    for b in range(S):
        vm, va = V_m[:, :, b:b + 1].clone(), V_a[:, :, b:b + 1].clone()
        it = 0
        f, err = sol.mismatch(vm, va, P[:, b:b + 1], Q[:, b:b + 1], I_N[:, :, b:b + 1])
        while float(err.item()) > 1e-4 and it < 50:
            dx, info = sol.lu_solve(sol.jacobian(vm, va), f)
            va.view(-1)[1:] -= dx[:nH - 1, 0]
            vm.view(-1)[c:] -= dx[nH - 1:, 0]
            f, err = sol.mismatch(vm, va, P[:, b:b + 1], Q[:, b:b + 1], I_N[:, :, b:b + 1])
            it += 1
        assert it == fused["n_iter_h"][b]
        assert np.array_equal(vm[:, :, 0].cpu().numpy(), fused["V_m"][:, :, b])
        assert np.array_equal(va[:, :, 0].cpu().numpy(), fused["V_a"][:, :, b])


@pytest.mark.parametrize("case", ["net3_c_h25", "net3_uc_h25", "net2ev_c_h19", "net2ev_uc_h19"])
def test_mismatch_lane_kernel_equals_tile_kernel(case, tmp_path, monkeypatch):
    """The shape-specialised one-thread-per-scenario mismatch kernel (default for the BASELINE
    4-bus shapes) against the generic tile kernel on a ragged random batch: wild angles (both
    sides of the large-argument bound of its sin/cos), negative magnitudes, NaN and Inf lanes.
    Its sin/cos differs from the library routine by <= 1 ulp, hence 1e-14 instead of bitwise."""
    from harmonic_power_flow_b200 import BatchSolver
    d = helpers.load_case(case)
    net, _, _ = helpers.packed_from_files(str(d["net"]), int(d["h_max"]), bool(d["coupled"]), tmp_path)
    B = 333
    rng = np.random.default_rng(11)
    Vm = rng.uniform(-1.2, 1.2, (net.H, net.n, B))
    Va = rng.uniform(-50.0, 50.0, (net.H, net.n, B))
    Va[:, :, 100:140] *= 1e4                      # up to 5e5 rad: beyond the fast-path bound 105615
    Va[3, 1, 7] = 105615.0
    Va[4, 2, 8] = -105614.99
    P = rng.uniform(-2, 2, (net.n, B)); Q = rng.uniform(-2, 2, (net.n, B))
    I_N = rng.normal(size=(net.q, net.H, B)) + 1j * rng.normal(size=(net.q, net.H, B))
    Vm[1, 1, 5] = np.nan
    Va[2, 0, 6] = np.inf
    Vm[0, 2, 9] = np.inf
    lane = BatchSolver(net)
    f1, e1, i1 = lane.mismatch(Vm, Va, P, Q, I_N, want_I_inj=True)
    monkeypatch.setenv("HPF_MISMATCH_TILE", "1")
    tile = BatchSolver(net)
    f2, e2, i2 = tile.mismatch(Vm, Va, P, Q, I_N, want_I_inj=True)
    f1, e1, i1, f2, e2, i2 = [t.cpu().numpy() for t in (f1, e1, i1, f2, e2, i2)]
    bad = np.zeros(B, bool); bad[[5, 6, 9]] = True
    assert np.isnan(e1[[5, 6]]).all() and np.isnan(e2[[5, 6]]).all()
    assert not np.isfinite(e1[9]) and not np.isfinite(e2[9])
    assert np.isfinite(e1[~bad]).all()
    scale = np.abs(f2[:, ~bad]).max(0)
    assert (np.abs(f1[:, ~bad] - f2[:, ~bad]).max(0) / scale).max() <= 1e-14
    assert np.abs(e1[~bad] - e2[~bad]).max() <= 1e-14 * np.abs(e2[~bad]).max()
    assert np.abs(i1[:, :, ~bad] - i2[:, :, ~bad]).max() <= 1e-14 * np.abs(i2[:, :, ~bad]).max()
    lane.close(); tile.close()


@pytest.mark.parametrize("dense", [False, True])
def test_status_words_and_edge_batches(solvers, dense):
    sol, net, d = solvers("net3_c_h25")
    P, Q, I_N = net.P[:, None], net.Q[:, None], net.I_N[:, :, None]
    _solve = sol.solve
    sol = type("S", (), {"solve": staticmethod(lambda *a_, **k: _solve(*a_, dense=dense, **k))})()
    r = sol.solve(P, Q, I_N, max_iter_h=3)
    assert int(r.n_iter_h.item()) == 3 and int(r.status.item()) == 1      # HG:558: max-iter
    r = sol.solve(P, Q, I_N, max_iter_h=int(d["n_iter_h"]))              # converges ON the cap
    assert int(r.status.item()) == 1 and float(r.err_h.item()) < 1e-4     # reference reports max-iter too
    r = sol.solve(P, Q, I_N, thresh_h=1e9)                                # zero iterations
    assert int(r.n_iter_h.item()) == 0 and int(r.status.item()) == 0
    Pn = P.copy(); Pn[2, 0] = np.nan
    r = sol.solve(Pn, Q, I_N)
    assert int(r.status.item()) == 3
    # empty batch: no launch, no error
    r = sol.solve(np.zeros((net.n, 0)), np.zeros((net.n, 0)), np.zeros((net.q, net.H, 0), complex))
    assert r.B == 0
    # a batch of identical scenarios gives identical results in every slot (scenario independence)
    B = 300
    r = sol.solve(np.repeat(P, B, 1), np.repeat(Q, B, 1), np.repeat(I_N, B, 2)).to_host()
    assert (r["n_iter_h"] == int(d["n_iter_h"])).all()
    assert (r["V_m"] == r["V_m"][:, :, :1]).all() and (r["V_a"] == r["V_a"][:, :, :1]).all()


@pytest.mark.parametrize("kernel", ["warp", "tile", "dense"])
@pytest.mark.parametrize("case", ["net3_c_h25", "net2ev_uc_h19"])
def test_queue_refill_few_ctas_ragged_batch(solvers, case, kernel, tmp_path, monkeypatch):
    """The persistent kernels pull scenarios from a global queue and refill lanes / CTAs as
    scenarios finish.  With the grid capped at 2 CTAs ($HPF_MAX_CTAS) a ragged batch of 333
    scenarios exercises every refill path; per-scenario arithmetic does not depend on the lane,
    tile or CTA a scenario lands in, so the results must be BIT-identical to the uncapped run.
    kernel: "warp" = one warp per harmonic (default for the BASELINE shapes), "tile" = 32-scenario
    tile kernel ($HPF_HARM_KERNEL=tile), "dense" = fused dense-LU kernel."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    sol, net, _ = solvers(case)
    B = 333
    P, Q, I_N = scenarios.make_batch(net, B, "wide")
    if kernel == "tile":
        monkeypatch.setenv("HPF_HARM_KERNEL", "tile")
        sol = BatchSolver(net)
    want = sol.solve(P, Q, I_N, dense=(kernel == "dense"), history=True).to_host()
    monkeypatch.setenv("HPF_MAX_CTAS", "2")
    capped = BatchSolver(net)
    got = capped.solve(P, Q, I_N, dense=(kernel == "dense"), history=True).to_host()
    capped.close()
    if kernel == "tile":
        sol.close()
    assert (want["status"] == 0).all()
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status", "err_hist_h", "err_hist_f"):
        assert np.array_equal(got[k], want[k], equal_nan=True), k
    assert len(np.unique(want["n_iter_h"])) > 3              # lanes really finish at different times


def test_warp_kernel_agrees_with_tile_kernel(solvers, monkeypatch):
    """The two structured kernels assemble the border system differently (reduced complex form vs
    entry by entry) - same Newton step, different round-off: counts agree except for a few
    round-off-decided scenarios, phasors agree to 1e-9 wherever the counts do."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    sol, net, _ = solvers("net3_c_h25")
    B = 4096
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    a = sol.solve(P, Q, I_N).to_host()
    monkeypatch.setenv("HPF_HARM_KERNEL", "tile")
    tile = BatchSolver(net)
    b = tile.solve(P, Q, I_N).to_host()
    tile.close()
    same = a["n_iter_h"] == b["n_iter_h"]
    Va, Vb = helpers.phasor(a["V_m"], a["V_a"]), helpers.phasor(b["V_m"], b["V_a"])
    rel = (np.abs(Va - Vb) / np.abs(Vb)).reshape(-1, B).max(0)
    print("\nwarp vs tile kernel: %d/%d iteration-count differences, median phasor diff %.2e" % (
        (~same).sum(), B, np.median(rel)))
    assert (~same).mean() < 0.03 and np.median(rel) < 1e-11


@pytest.mark.parametrize("case", ["net1_c_h25", "net1_uc_h51", "net1_c_h51", "net2_c_h51", "net2_uc_h51"])
def test_large_networks_structured_cta_path(solvers, case):
    """net1 (20 buses, N = 518 / 1038) and net2 with 26 harmonics through the structured step
    (per-CTA variant for net1): identical iteration counts except on net1/H<=51, same solution."""
    sol, net, d = solvers(case)
    info = sol.struct_info()
    assert info["available"] in (1, 2)
    r = sol.solve(net.P[:, None], net.Q[:, None], net.I_N[:, :, None], history=True)
    hist = r.err_hist_h[:, 0].cpu().numpy()
    ref_hist = np.asarray(d["err_h_hist"])
    k = min(len(ref_hist), int(r.n_iter_h.item()) + 1)
    dev = np.abs(hist[:k] - ref_hist[:k]) / ref_hist[:k]
    split = int(np.argmax(dev > 1e-6)) if (dev > 1e-6).any() else k
    print("\n%s: structured variant %d, n_iter_h GPU %d, reference %d; error path equal to 1e-6 for the first %d steps" % (
        case, info["available"], int(r.n_iter_h.item()), int(d["n_iter_h"]), split))
    assert int(r.n_iter_f.item()) == int(d["n_iter_f"])
    if case == "net1_c_h51":
        # cond(J) reaches 4e9 and ||f|| wanders around 1e3 for ~20 steps: the count is decided by
        # round-off - the reference itself needs 23 steps with its SuperLU step and 36 with a LAPACK
        # step (DESIGN.md sec. 4); B200 builds of this kernel have given 23 and 28.  Pinned instead:
        # the first steps of the reference's error path, convergence, and the (unique) solution.
        assert np.allclose(hist[:6], ref_hist[:6], rtol=1e-4)
        assert 15 <= int(r.n_iter_h.item()) < 50
    else:
        assert int(r.n_iter_h.item()) == int(d["n_iter_h"])
    assert int(r.status.item()) == 0
    V = helpers.phasor(r.V_m[:, :, 0].cpu().numpy(), r.V_a[:, :, 0].cpu().numpy())
    Vg = helpers.phasor(d["V_m"], d["V_a"])
    assert (np.abs(V - Vg) / np.abs(Vg)).max() < (1e-6 if case == "net1_c_h51" else 1e-7)
    thd = sol.thd(r.V_m)[:, :, 0].cpu().numpy().T
    assert np.abs(thd - d["THD"]).max() < 1e-6
    # one structured step equals J^-1 f of the reference's first iteration
    Vm, Va = d["V_fund_m"][:, :, None], d["V_fund_a"][:, :, None]
    dx = sol.newton_step(Vm, Va, net.P[:, None], net.Q[:, None], net.I_N[:, :, None])[:, 0].cpu().numpy()
    x0 = helpers.state_vectors(d["V_fund_m"], d["V_fund_a"], net.c)
    assert np.abs((x0 - dx) - d["x1"]).max() <= 1e-8 * np.abs(d["x1"]).max()


@pytest.mark.parametrize("case", ["net1_c_h25", "net1_c_h51"])
def test_large_system_dense_global_memory_path(solvers, case):
    """The dense-LU strategy for N = 518 / 1038 (matrix in a global-memory workspace)."""
    sol, net, d = solvers(case)
    r = sol.solve(net.P[:, None], net.Q[:, None], net.I_N[:, :, None], dense=True, history=True)
    assert int(r.n_iter_f.item()) == int(d["n_iter_f"])
    print("\n%s dense: n_iter_h GPU %d, reference %d" % (case, int(r.n_iter_h.item()), int(d["n_iter_h"])))
    if case == "net1_c_h51":
        # cond(J) reaches 4e9 here and the iteration wanders at ||f|| ~ 1e3 for ~20 steps: a dense LU
        # of J reproduces the reference's path only for the first steps (DESIGN.md section 4)
        hist = r.err_hist_h[:, 0].cpu().numpy()
        assert np.allclose(hist[:6], d["err_h_hist"][:6], rtol=1e-4)
        assert 15 <= int(r.n_iter_h.item()) < 50
    else:
        assert int(r.n_iter_h.item()) == int(d["n_iter_h"])
    assert int(r.status.item()) == 0
    V = helpers.phasor(r.V_m[:, :, 0].cpu().numpy(), r.V_a[:, :, 0].cpu().numpy())
    Vg = helpers.phasor(d["V_m"], d["V_a"])
    assert (np.abs(V - Vg) / np.abs(Vg)).max() < 1e-7


def test_invalid_arguments_are_refused_loudly(solvers):
    from harmonic_power_flow_b200 import _lib
    sol, net, d = solvers("net3_c_h25")
    with pytest.raises(ValueError):
        sol.solve(net.P[:, None], net.Q[:, None], net.I_N[:, :1, None])       # wrong I_N shape
    lib, h = sol.lib, sol._h

    def refused(rc, msg):
        with pytest.raises(_lib.HpfError) as e:
            _lib.check(h, rc)
        assert e.value.code == _lib.HPF_E_INVALID and msg in str(e.value), str(e.value)

    # every solve entry point, with each of its paths, checks its request before it runs
    for flags in (0, _lib.SOLVE_DENSE):
        refused(lib.hpf_solve(h, 1, None, None, None, 1e-6, 30, 1e-4, 50, flags, *[None] * 10),
                "hpf_solve: NULL buffer")
    refused(lib.hpf_solve(h, -1, None, None, None, 1e-6, 30, 1e-4, 50, 0, *[None] * 10), "hpf_solve: B < 0")
    refused(lib.hpf_fund_solve(h, 1, None, None, 1e-6, 30, *[None] * 6), "hpf_fund_solve: NULL buffer")
    refused(lib.hpf_solve_host(h, 1, None, None, None, 1e-6, 30, 1e-4, 50, *[None] * 7),
            "hpf_solve_host: NULL buffer")
    refused(lib.hpf_solve_host(h, -1, None, None, None, 1e-6, 30, 1e-4, 50, *[None] * 7), "hpf_solve_host: B < 0")


# ---------------------------------------------------------------- drop-in API
def test_reference_shaped_api(tmp_path):
    from harmonic_power_flow_b200 import hcne_generalized as hg
    d = helpers.load_case("net3_c_h25")
    pb, pl = helpers.write_net_csvs("net3", str(tmp_path))
    helpers.write_ne_csvs(str(tmp_path))
    hg.configure(H_MAX=25, ne_dir=str(tmp_path))
    buses, lines, m, n, c = hg.init_network(pb, pl)
    assert (m, n, c) == (3, 4, 2) and hg.HARMONICS == list(d["harmonics"])
    Y = hg.build_admittance_matrices(buses, lines, hg.HARMONICS)
    assert _rel(Y.to_numpy().reshape(d["Y_all"].shape), d["Y_all"]) <= 1e-15
    assert _rel(np.array(Y.loc[5]), d["Y_all"][2]) <= 1e-15
    V_f, err_t, n_iter_f = hg.pf(Y, buses)
    assert n_iter_f == int(d["n_iter_f"]) and len(err_t) == n_iter_f
    assert np.abs(helpers.phasor(V_f["V_m"], V_f["V_a"]) -
                  helpers.phasor(d["V_fund_m"], d["V_fund_a"]).ravel()).max() < 1e-12
    V, err_h, n_iter_h, J = hg.hpf(buses, lines, coupled=True)
    assert n_iter_h == int(d["n_iter_h"]) and err_h < 1e-4
    assert list(V.columns) == ["V_m", "V_a"] and V.index.names == ["harmonic", "bus"]
    assert V.loc[(5, 3), "V_m"] == pytest.approx(2.823989096210703e-01, rel=1e-9)
    assert V.loc[(5, 3), "V_a"] == pytest.approx(1.899824023109353, rel=1e-9)
    assert isinstance(J, hg.LastJacobian) and J._J is None       # assembled on first use only
    assert J.shape == (101, 101) and J.nnz == 1221
    assert _rel(J.toarray(), d["J_last"]) < 1e-6
    # a second call on the same network reuses the cached GPU handle and gives the same answer
    n_handles = len(hg._SOLVERS)
    V2, err_h2, n_iter_h2, _ = hg.hpf(buses, lines, coupled=True)
    assert len(hg._SOLVERS) == n_handles and n_iter_h2 == n_iter_h and V2.equals(V)
    THD = hg.get_THD(V)
    assert np.abs(THD.to_numpy() - d["THD"]).max() < 1e-8
    hg.release_solvers()
    assert not hg._SOLVERS
    hg.configure(H_MAX=51)


# ---------------------------------------------------------------- full-size properties
def test_full_size_batch_properties(solvers):
    """BASELINE config 3 at full size (65,536 scenarios): size-independent properties.
    (a) every scenario converges; (b) the returned iterate really has ||f||_inf <= 1e-4 when the
    mismatch is re-evaluated by the standalone kernel on the raw iterate, and it equals the
    reported err_h; (c) splitting the batch differently (as another GPU count would) gives
    bit-identical results; (d) I_inj equals I_N - Y_N V recomputed on the host for a sample."""
    from harmonic_power_flow_b200 import scenarios
    sol, net, _ = solvers("net3_c_h25")
    B = 65536
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    dP, dQ, dI = sol.prepare(P, Q, I_N)
    raw = sol.solve(dP, dQ, dI, raw=True)
    assert int((raw.status == 0).sum()) == B
    assert int(raw.n_iter_f.min()) == 2 and int(raw.n_iter_f.max()) == 2
    f, err = sol.mismatch(raw.V_m, raw.V_a, dP, dQ, dI)
    # the standalone kernel's sin/cos differs from the solver's by <= 1 ulp; through |Y| ~ 1e4
    # that moves an entry of f by ~1e-12, i.e. 1e-8 relative at the 1e-4 threshold
    assert float(err.max()) <= 1e-4 * (1 + 1e-6)
    assert torch.allclose(err, raw.err_h, rtol=1e-6, atol=1e-11)
    # (c) three unequal shards vs one batch
    cuts = [0, 21845, 43691, B]
    for lo, hi in zip(cuts, cuts[1:]):
        part = sol.solve(dP[:, lo:hi].contiguous(), dQ[:, lo:hi].contiguous(), dI[:, :, lo:hi].contiguous(),
                         raw=True)
        assert torch.equal(part.V_m, raw.V_m[:, :, lo:hi]) and torch.equal(part.V_a, raw.V_a[:, :, lo:hi])
        assert torch.equal(part.n_iter_h, raw.n_iter_h[lo:hi]) and torch.equal(part.I_inj, raw.I_inj[:, :, lo:hi])
    # (d) Norton injection identity on a sample
    V = (raw.V_m * torch.exp(1j * raw.V_a))[:, net.m:, ::4099].cpu().numpy()          # [H, q, S]
    inj = raw.I_inj[:, :, ::4099].cpu().numpy()
    want = I_N[:, :, ::4099] - np.einsum("qhp,pqs->qhs", net.Y_N[net.dev_of_nl_bus], V)
    assert np.abs(inj - want).max() <= 1e-12 * np.abs(want).max()
    # post-processed output is the same phasor, magnitudes >= 0, angles in [0, 2 pi]
    pp = sol.solve(dP, dQ, dI)
    Vr = raw.V_m * torch.exp(1j * raw.V_a)
    Vp = pp.V_m * torch.exp(1j * pp.V_a)
    # (the raw angles are un-reduced: reducing an angle a by the DOUBLE 2 pi - what numpy's % does too,
    # HG:548 - moves the phasor by |a| * 3.9e-17 relative; torch.exp on |a| adds ~|a| ulp)
    tol = raw.V_m.abs() * (raw.V_a.abs() * 1e-15 + 1e-14) + 1e-14
    assert bool(((Vr - Vp).abs() <= tol).all()), float(((Vr - Vp).abs() / tol).max())
    assert float(pp.V_m.min()) >= 0 and float(pp.V_a.min()) >= 0 and float(pp.V_a.max()) <= 2 * np.pi


def test_parity_rates_at_scale_vs_oracle(solvers):
    """BASELINE config 3, 2,048 seeded scenarios (the SAME generator the bench and the golden sets
    use) solved by both GPU strategies and by the oracle with the reference's SuperLU step and
    with a LAPACK step.  The reference's iteration is chaotic before it converges, so its own
    iteration count depends on round-off (SURVEY 7.3): "identical counts" can only mean that the
    GPU disagrees with the reference no more often than the reference disagrees with itself.
    Asserted: both GPU disagreement counts <= the SuperLU-vs-LAPACK floor + 3 sigma of its
    sampling error; the median phasor difference is < 1e-11 and its tail stays within 10x the reference's own."""
    import oracle_pool
    from harmonic_power_flow_b200 import scenarios
    sol, net, _ = solvers("net3_c_h25")
    S = 2048
    P, Q, I_N = scenarios.make_batch(net, S, "tight")
    pool = oracle_pool.OraclePool(O.net_from_golden(GOLDEN, "net3", 25, True))
    try:
        ref = pool.solve(P, Q, I_N, "superlu")
        lap = pool.solve(P, Q, I_N, "lapack")
    finally:
        pool.close()
    floor = oracle_pool.parity_rates(lap, ref)["vs_oracle"]
    for strategy in ("structured", "dense"):
        r = sol.solve(P, Q, I_N, dense=(strategy == "dense")).to_host()
        assert (r["status"] == 0).all() and (ref["status"] == 0).all()
        st = oracle_pool.parity_rates(r, ref)["vs_oracle"]
        print("\nnet3 tight x%d [%s]: iteration mismatches %d (floor %d), phasor diff > 1e-9: %d (floor %d), "
              "median %.2e, max where counts agree %.2e" % (S, strategy, st["iteration_mismatches"],
              floor["iteration_mismatches"], st["phasor_diff_gt_1e9"], floor["phasor_diff_gt_1e9"],
              st["phasor_diff_median"], st["phasor_diff_max_same_count"]))
        assert st["n_iter_f_mismatches"] == 0
        margin = lambda k: k + 3.0 * np.sqrt(k + 1.0)
        assert st["iteration_mismatches"] <= margin(floor["iteration_mismatches"])
        assert st["phasor_diff_gt_1e9"] <= margin(floor["phasor_diff_gt_1e9"])
        assert st["phasor_diff_median"] < 1e-11
        # (a last accepted step of ||f|| ~ 1e-4 leaves the iterate ~1e-5 from the converged one: the
        # reference against itself reaches 2.6e-5 on the first 1,024 scenarios)
        assert st["phasor_diff_max_same_count"] <= max(1e-6, 10 * floor["phasor_diff_max_same_count"])


def test_config2_batch_1024_against_oracle(solvers):
    """BASELINE config 2: net2 with two Norton loads (SMPS + EV), odd harmonics to the 19th,
    1,024 scenarios; a sample is checked against the CPU oracle, the whole batch for convergence."""
    from harmonic_power_flow_b200 import scenarios
    sol, net, _ = solvers("net2ev_c_h19")
    B = 1024
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    r = sol.solve(P, Q, I_N).to_host()
    assert (r["status"] == 0).all()
    on = O.net_from_golden(GOLDEN, "net2ev", 19, True)
    Y = O.build_admittance_matrices(on)
    mism = 0
    for b in range(0, B, 37):
        o = O.hpf(on, P=P[:, b], Q=Q[:, b], I_N=I_N[:, :, b], Y=Y)
        mism += int(o["n_iter_h"] != r["n_iter_h"][b])
        if o["n_iter_h"] == r["n_iter_h"][b]:
            V = helpers.phasor(r["V_m"][:, :, b], r["V_a"][:, :, b])
            Vo = helpers.phasor(o["V_m"], o["V_a"])
            assert (np.abs(V - Vo) / np.abs(Vo)).max() < 1e-6
    assert mism <= 2            # 28 samples; the reference disagrees with itself at this rate


# ---------------------------------------------------------------- large synthetic networks (configs 4, 5)
def _check_against_oracle(net, res, P, Q, I_N, scen, tol):
    on = helpers.oracle_net(net)
    Y = O.build_admittance_matrices(on)
    for b in scen:
        o = O.hpf(on, P=P[:, b], Q=Q[:, b], I_N=I_N[:, :, b], Y=Y)
        tag = "scenario %d: oracle it %d/%d err %.2e, gpu it %d/%d err %.2e" % (
            b, o["n_iter_f"], o["n_iter_h"], o["err_h"], res["n_iter_f"][b], res["n_iter_h"][b], res["err_h"][b])
        assert o["status"] == 0 and res["status"][b] == 0, tag
        assert res["n_iter_f"][b] == o["n_iter_f"], tag
        assert res["n_iter_h"][b] == o["n_iter_h"], tag
        Vo, Vg = helpers.phasor(o["V_m"], o["V_a"]), helpers.phasor(res["V_m"][:, :, b], res["V_a"][:, :, b])
        tag += " dV %.2e" % (np.abs(Vo - Vg).max() / np.abs(Vo).max())
        # both stop at the same iteration with ||f||_inf <= 1e-4 (HG:536); the iterate is only
        # defined to the mismatch it was accepted with: round-off histories that end at err 1e-9
        # agree to 1e-9, one that ends at err 4e-5 is 1e-6 away from the fully converged one
        t = max(tol, 0.1 * max(o["err_h"], res["err_h"][b]))
        assert np.abs(Vo - Vg).max() <= t * np.abs(Vo).max(), tag
        assert np.abs(o["I_inj"] - res["I_inj"][:, :, b]).max() <= 10 * t * np.abs(o["I_inj"]).max(), tag


@pytest.mark.parametrize("kind,n,scale,variant", [("radial", 40, 0.02, 0), ("radial", 40, 0.02, 3),
                                                  ("meshed", 30, 0.02, 3)])
def test_synthetic_networks_small_against_oracle(kind, n, scale, variant, tmp_path, monkeypatch):
    """Seeded synthetic feeder / meshed network (generators of BASELINE configs 4-5) at a size the
    oracle solves in a fraction of a second; variant 3 = the large-network code path (scenario
    state in global memory, multi-CTA operator inversion when nZ > 768, blocked tensor-core LU
    for the border system) forced onto the small network."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    if variant:
        monkeypatch.setenv("HPF_STRUCT_VARIANT", str(variant))
    net, _ = helpers.synthetic_packed(kind, tmp_path, h_max=25, n=n, load_scale=scale)
    sol = BatchSolver(net)
    assert sol.struct_info()["available"] == (variant or 2)
    B = 40
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    res = sol.solve(P, Q, I_N).to_host()
    assert (res["status"] == 0).all()
    _check_against_oracle(net, res, P, Q, I_N, range(0, B, 5), 1e-9)
    # the host-buffer entry point goes through the same variant and gives the same bits
    rh = sol.solve_host(P, Q, I_N)
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(rh[k], res[k]), k
    sol.close()


def test_config4_radial_200_bus_against_oracle(tmp_path):
    """BASELINE config 4 network (200-bus radial feeder, 40 % nonlinear buses, odd harmonics to
    the 25th: N = 5198 unknowns) - two scenarios checked against the oracle (about 10 s each),
    plus batch-split invariance of a 300-scenario batch."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    net, _ = helpers.synthetic_packed("radial", tmp_path, h_max=25, n=200, load_scale=0.005)
    sol = BatchSolver(net)
    info = sol.struct_info()
    assert info["available"] == 3 and info["nZ"] == 2480
    B = 300
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    r = sol.solve(P, Q, I_N)
    res = r.to_host()
    assert (res["status"] == 0).all() and (res["n_iter_f"] == 3).all()
    # 16 scenarios against the oracle (about 10 s of CPU each, fanned out over the host cores), with the
    # reference's SuperLU step and with a LAPACK step: a scenario whose mismatch norm lands within
    # round-off of the 1e-4 threshold stops one or two iterations earlier or later (seen: oracle
    # 8.06e-5 after 24 steps, GPU 26 steps), so the GPU count must equal the SuperLU oracle's except
    # for at most one scenario more than the oracle disagrees with itself
    import oracle_pool
    pool = oracle_pool.OraclePool(helpers.oracle_net(net))
    try:
        o = pool.solve(P[:, :16], Q[:, :16], I_N[:, :, :16], "superlu", chunk=1)
        ol = pool.solve(P[:, :16], Q[:, :16], I_N[:, :, :16], "lapack", keep_V=False, chunk=1)
    finally:
        pool.close()
    floor = int((o["n_iter_h"] != ol["n_iter_h"]).sum())
    mism = 0
    for b in range(16):
        tag = "scenario %d: oracle it %d/%d err %.2e (lapack step: %d), gpu it %d/%d err %.2e" % (
            b, o["n_iter_f"][b], o["n_iter_h"][b], o["err_h"][b], ol["n_iter_h"][b], res["n_iter_f"][b],
            res["n_iter_h"][b], res["err_h"][b])
        assert o["status"][b] == 0, tag
        assert res["n_iter_f"][b] == o["n_iter_f"][b], tag
        if res["n_iter_h"][b] != o["n_iter_h"][b]:
            mism += 1
            print("\n" + tag)
        Vo = helpers.phasor(o["V_m"][:, :, b], o["V_a"][:, :, b])
        Vg = helpers.phasor(res["V_m"][:, :, b], res["V_a"][:, :, b])
        # (an iterate accepted at mismatch norm e is ~ ||J^-1|| e away from the solution; ||J^-1|| < 1 here)
        t = max(1e-9, max(o["err_h"][b], res["err_h"][b]))
        assert np.abs(Vo - Vg).max() <= t * np.abs(Vo).max(), tag
        # (the current rows of f ARE the residual of I_inj in p.u.: two iterates accepted at mismatch
        # norms e1, e2 differ by up to e1 + e2 in the injected currents)
        assert np.abs(o["I_inj"][:, :, b] - res["I_inj"][:, :, b]).max() <= max(
            10 * t * np.abs(o["I_inj"][:, :, b]).max(), 2 * (o["err_h"][b] + res["err_h"][b])), tag
    print("\nconfig 4: %d/16 iteration-count differences against the SuperLU oracle (oracle vs itself: %d)" % (mism, floor))
    assert mism <= floor + 1
    # (both parts are >= the lock-step threshold of 128 scenarios: the same strategy solves them)
    part = sol.solve(P[:, 100:250].copy(), Q[:, 100:250].copy(), I_N[:, :, 100:250].copy()).to_host()
    assert np.array_equal(part["V_m"], res["V_m"][:, :, 100:250]) and np.array_equal(part["n_iter_h"], res["n_iter_h"][100:250])
    sol.close()


# ---------------------------------------------------------------- Norton-equivalent extraction (next-1)
@pytest.mark.parametrize("name", ["smps", "circuit_sim"])
def test_ne_extract_matches_reference_script(name):
    """hpf_ne_extract against the reference's own NE_from_sim.py outputs (golden fixtures)."""
    from harmonic_power_flow_b200 import ne_from_sim
    import os
    d = np.load(os.path.join(GOLDEN, "ne_extract_%s.npz" % name))
    sim = ne_from_sim.Simulation(d["freq"], d["Vf"], d["Vh"], d["I_f"], d["I_h"])
    ne = ne_from_sim.get_NE_from_sim(sim)
    for k in ("Y_N_c", "I_N_c", "Y_N_uc", "I_N_uc"):
        assert np.abs(ne[k] - d[k]).max() <= 1e-12 * np.abs(d[k]).max(), k


def test_ne_extract_batch_round_trip_and_csv(tmp_path):
    """64 perturbed SMPS devices with 26 frequencies: measurements synthesised from a known coupled
    Norton equivalent (forward model HG:313-323), extracted on the GPU in one launch; the
    extraction must return the equivalents it started from, agree with the oracle, flag a
    singular measurement set, and survive the CSV round trip into the solve path's loader."""
    import ne_oracle as NO
    from harmonic_power_flow_b200 import ne_from_sim, netio
    import os
    dev = np.load(os.path.join(GOLDEN, "ne_devices.npz"))
    N, D = 26, 64
    rng = np.random.default_rng(7)
    freq = dev["smps__freqs"][:N]
    sims, truth = [], []
    for s in range(D):
        Y = dev["smps__Y_N_c"][:N, :N] * (1 + 0.1 * rng.standard_normal((N, N))) * np.exp(0.1j * rng.standard_normal((N, N)))
        I = dev["smps__I_N_c"][:N] * (1 + 0.1 * rng.standard_normal(N))
        Vf = 230.0 * np.sqrt(2) * np.array([1.0, np.exp(1j * 0.05)])
        Vh = np.array([np.full(N - 1, 2.3), np.full(N - 1, 4.6)]) * np.exp(1j * rng.uniform(-0.2, 0.2))
        if s == 9:
            Vh[0][0] = 0.0                      # no harmonic excitation at freq[1]: a zero column -> singular
        I_f, I_h = NO.synth_measurements(Y, I, Vf, Vh)
        sims.append(ne_from_sim.Simulation(freq, Vf, Vh, I_f, I_h)); truth.append((Y, I))
    from harmonic_power_flow_b200.solver import ne_extract
    out = {k: v.cpu().numpy() for k, v in ne_extract(np.stack([s.Vf for s in sims]), np.stack([s.Vh for s in sims]),
                                                      np.stack([s.I_f for s in sims]), np.stack([s.I_h for s in sims])).items()}
    assert out["info"][9] != 0 and (np.delete(out["info"], 9) == 0).all()
    with pytest.raises(np.linalg.LinAlgError):
        ne_from_sim.get_NE_from_sim(sims)
    for s in range(D):
        if s == 9:
            continue
        Y, I = truth[s]
        assert np.abs(out["Y_N_c"][s] - Y).max() <= 1e-9 * np.abs(Y).max()
        assert np.abs(out["I_N_c"][s] - I).max() <= 1e-9 * np.abs(I).max()
        Yo, Io = NO.coupled(sims[s].Vf, sims[s].Vh, sims[s].I_f, sims[s].I_h)
        Yuo, Iuo = NO.uncoupled(sims[s].Vf, sims[s].Vh, sims[s].I_f, sims[s].I_h)
        assert np.abs(out["Y_N_c"][s] - Yo).max() <= 1e-10 * np.abs(Yo).max()
        assert np.abs(out["Y_N_uc"][s] - Yuo).max() <= 1e-12 * np.abs(Yuo).max()
        assert np.abs(out["I_N_uc"][s] - Iuo).max() <= 1e-12 * np.abs(Iuo).max()
    ne0 = {k: out[k][0] for k in ("Y_N_c", "I_N_c", "Y_N_uc", "I_N_uc")}
    path = os.path.join(str(tmp_path), "dev0_NE.csv")
    ne_from_sim.export_NE(path, freq, ne0)
    tab = netio.read_ne_csv(path)
    assert np.array_equal(tab.loc["I_N_c"].to_numpy().ravel(), ne0["I_N_c"])
    assert np.array_equal(tab.loc[("Y_N_c", list(freq)), list(freq)].to_numpy(), ne0["Y_N_c"])


# ---------------------------------------------------------------- transformer branches in Y(h) (next-3)
@pytest.mark.parametrize("tag", ["a", "b"])
def test_trafo_ybus_matches_reference_function(tag):
    """ybus_kernel with hpf_set_transformers against the reference's own
    FPF/pi_trafo_pf_test.py:build_admittance_matrices outputs; clearing the transformer data
    restores the plain HG:132-171 result."""
    import os
    from harmonic_power_flow_b200 import BatchSolver
    from harmonic_power_flow_b200.netio import PackedNet
    d = np.load(os.path.join(GOLDEN, "ybus_trafo.npz"))
    n = len(d[tag + "_X_sh"])
    net = PackedNet(n=n, m=n, c=1, harmonics=np.ascontiguousarray(d[tag + "_harmonics"], np.int32),
                    from_id=np.ascontiguousarray(d[tag + "_frm"], np.int32),
                    to_id=np.ascontiguousarray(d[tag + "_to"], np.int32),
                    R=np.ascontiguousarray(d[tag + "_R"]), X=np.ascontiguousarray(d[tag + "_X"]),
                    G=np.ascontiguousarray(d[tag + "_G"]), B=np.ascontiguousarray(d[tag + "_B"]),
                    X_sh=np.ascontiguousarray(d[tag + "_X_sh"]), P=np.zeros(n), Q=np.zeros(n))
    sol = BatchSolver(net)
    Y_plain = sol.Y.cpu().numpy().copy()
    Y = sol.set_transformers(d[tag + "_tau"], d[tag + "_ph"]).cpu().numpy()
    want = d[tag + "_Y"]
    assert np.abs(Y - want).max() <= 4e-15 * np.abs(want).max()
    assert ((Y == 0) == (want == 0)).all()
    assert np.array_equal(sol.set_transformers(None).cpu().numpy(), Y_plain)
    with pytest.raises(Exception):
        sol.set_transformers(np.zeros(len(net.R)), np.zeros(len(net.R)))      # tau = 0
    sol.close()


def test_config5_meshed_1000_bus_nominal_against_oracle_run(tmp_path):
    """BASELINE config 5 network (1000-bus meshed, 400 nonlinear buses, odd harmonics to the 25th:
    N = 25,998 unknowns).  The oracle needs 98 minutes for ONE scenario of this size, so it was run
    once in the build container (scratch/probe_synth.py meshed 1000 0.002) and its summary is the
    fixture: n_iter_f = 2, n_iter_h = 26, err_h = 4.085e-06, max |V| at the fundamental and at the
    3rd harmonic.  The GPU path (multi-CTA operator inversion of order 12,400, global-state CTA
    kernel, blocked tensor-core LU of order 1198 / 1999) must reproduce them."""
    from harmonic_power_flow_b200 import BatchSolver
    net, _ = helpers.synthetic_packed("meshed", tmp_path, h_max=25, n=1000, load_scale=0.002)
    assert (net.n, net.m, net.H, net.N) == (1000, 600, 13, 25998)
    sol = BatchSolver(net)
    info = sol.struct_info()
    assert info["available"] == 3 and info["nZ"] == 12400
    r = sol.solve(net.P[:, None].copy(), net.Q[:, None].copy(), net.I_N[:, :, None].copy()).to_host()
    assert r["status"][0] == 0 and r["n_iter_f"][0] == 2 and r["n_iter_h"][0] == 26
    assert r["err_h"][0] == pytest.approx(4.085e-06, rel=0.05)
    assert r["V_m"][0, :, 0].min() == 1.0
    assert r["V_m"][0, :, 0].max() == pytest.approx(1.1649555668183993, rel=1e-11)
    assert r["V_m"][1, :, 0].max() == pytest.approx(0.5791799507662769, rel=1e-11)
    sol.close()


def test_ybus_corrected_options_match_textbook_admittance_matrix():
    """hpf_set_y_options(FIX_SHUNT_INDEX | SUM_PARALLEL) against the textbook nodal admittance
    matrix (incidence form) on a seeded 6-bus network with parallel branches and pi-shunts; the
    default flags keep the reference's behaviour (covered by test_ybus_matches_reference)."""
    from harmonic_power_flow_b200 import BatchSolver
    from harmonic_power_flow_b200.netio import PackedNet
    rng = np.random.default_rng(4)
    n, L = 6, 9
    frm = np.array([1, 2, 3, 4, 5, 1, 2, 2, 6], np.int32); to = np.array([2, 3, 4, 5, 6, 3, 5, 3, 1], np.int32)
    R, X = rng.uniform(1e-3, 6e-3, L), rng.uniform(3e-3, 3e-2, L)
    G, B = rng.uniform(0, 1e-2, L), rng.uniform(0, 1e-3, L)
    X_sh = np.array([3e-5, 0, 0, 2e-4, 0, 0])
    harmonics = np.arange(1, 26, 2).astype(np.int32)
    net = PackedNet(n=n, m=n, c=1, harmonics=harmonics, from_id=frm, to_id=to, R=R, X=X, G=G, B=B, X_sh=X_sh,
                    P=np.zeros(n), Q=np.zeros(n))
    sol = BatchSolver(net)
    Y_ref_behaviour = sol.Y.cpu().numpy().copy()
    Y = sol.set_y_options(fix_shunt_index=True, sum_parallel=True).cpu().numpy()
    want = np.zeros((len(harmonics), n, n), dtype=complex)
    for hi, h in enumerate(harmonics):
        for l in range(L):
            f, t = frm[l] - 1, to[l] - 1
            y = 1 / (R[l] + 1j * X[l] * h)
            sh = (G[l] + 1j * h * B[l]) / 2
            want[hi, f, f] += y + sh; want[hi, t, t] += y + sh
            want[hi, f, t] -= y; want[hi, t, f] -= y
        for k in range(n):
            if X_sh[k] != 0 and h != 1:
                want[hi, k, k] += 1 / (1j * X_sh[k] * h)
    assert np.abs(Y - want).max() <= 1e-13 * np.abs(want).max()
    assert np.abs(Y - Y_ref_behaviour).max() > 1e-3 * np.abs(want).max()      # the quirks do matter here
    assert np.array_equal(sol.set_y_options().cpu().numpy(), Y_ref_behaviour)
    sol.close()


@pytest.mark.parametrize("variant", [0, 2, 3, 34])
def test_degenerate_shapes_linear_only_and_fundamental_only(tmp_path, monkeypatch, variant):
    """Edge shapes of the data contract: a network WITHOUT nonlinear buses (q = 0: the harmonic
    stage has nothing to inject, harmonic voltages go to zero) and a fundamental-only run
    (H = 1: the harmonic Newton loop works on the fundamental alone), through the tile kernel,
    both per-CTA variants and the lock-step batched path, against the oracle."""
    from harmonic_power_flow_b200 import BatchSolver, netio
    if variant == 34:                                        # variant 3 through the lock-step batched path
        monkeypatch.setenv("HPF_LOCKSTEP", "1")
        variant = 3
    if variant:
        monkeypatch.setenv("HPF_STRUCT_VARIANT", str(variant))
    # (a) q = 0: net2 with its SMPS bus turned into a linear PQ load
    pb, pl = helpers.write_net_csvs("net2", str(tmp_path))
    txt = open(pb).read().replace("nonlinear", "PQ")
    open(pb, "w").write(txt)
    st = netio.Settings(H_MAX=9, ne_dir=str(tmp_path))
    buses, lines, m, n, c = netio.init_network(pb, pl, st)
    assert m == n
    net = netio.pack_network(buses, lines, m, n, c, st.HARMONICS)
    sol = BatchSolver(net)
    B = 5
    rng = np.random.default_rng(1)
    P = net.P[:, None] * rng.uniform(0.9, 1.1, (n, B)); Q = net.Q[:, None] * rng.uniform(0.9, 1.1, (n, B))
    res = sol.solve(P, Q, np.zeros((0, net.H, B), complex)).to_host()
    on = helpers.oracle_net(net)
    on.I_N = np.zeros((0, net.H), complex); on.Y_N = np.zeros((0, net.H, net.H), complex)
    for b in range(B):
        o = O.hpf(on, P=P[:, b], Q=Q[:, b], I_N=on.I_N)
        assert res["status"][b] == o["status"] == 0
        assert res["n_iter_f"][b] == o["n_iter_f"] and res["n_iter_h"][b] == o["n_iter_h"]
        assert np.abs(res["V_m"][0, :, b] - o["V_m"][0]).max() <= 1e-12
        assert np.abs(res["V_m"][1:, :, b]).max() <= 1e-12 and np.abs(o["V_m"][1:]).max() <= 1e-12
    sol.close()
    # (b) H = 1: net3 with the SMPS equivalent restricted to the fundamental
    net1, _, _ = helpers.packed_from_files("net3", 1, True, tmp_path)
    assert net1.H == 1 and net1.q == 1
    sol = BatchSolver(net1)
    res = sol.solve(net1.P[:, None], net1.Q[:, None], net1.I_N[:, :, None]).to_host()
    o = O.hpf(helpers.oracle_net(net1))
    assert res["status"][0] == o["status"]
    assert res["n_iter_f"][0] == o["n_iter_f"] and res["n_iter_h"][0] == o["n_iter_h"]
    if o["status"] == 0:
        Vo, Vg = helpers.phasor(o["V_m"], o["V_a"]), helpers.phasor(res["V_m"][:, :, 0], res["V_a"][:, :, 0])
        assert np.abs(Vo - Vg).max() <= 1e-9 * np.abs(Vo).max()
    sol.close()


@pytest.mark.parametrize("case", ["net3_c_h25", "net1_c_h25"])
def test_bus_current_spectra(solvers, case):
    """hpf_bus_currents (next-2): I = Y(h) V per harmonic and bus against numpy on the reference's
    converged voltages; at the nonlinear buses the current balance makes it equal -I_inj."""
    sol, net, d = solvers(case)
    r = sol.solve(net.P[:, None], net.Q[:, None], net.I_N[:, :, None])
    I = sol.bus_currents(r.V_m, r.V_a).cpu().numpy()[:, :, 0]
    V = helpers.phasor(r.V_m.cpu().numpy()[:, :, 0], r.V_a.cpu().numpy()[:, :, 0])
    Y = sol.Y.cpu().numpy()
    want = np.einsum("hij,hj->hi", Y, V)
    assert np.abs(I - want).max() <= 1e-12 * np.abs(want).max()
    inj = r.I_inj.cpu().numpy()[:, :, 0]                       # [q, H]
    resid = np.abs(I[:, net.m:].T + inj).max()
    assert resid <= 2e-4                                        # the accepted current mismatch (thresh_h = 1e-4)


# ---------------------------------------------------------------- memory / race checks of our own
def _guarded_result(sol, B, max_f, max_h, guard=4096):
    """BatchResult whose fields are views into ONE device buffer with `guard` canary bytes before,
    between and after the fields: an out-of-bounds write of any kernel lands in a canary band."""
    from harmonic_power_flow_b200.solver import BatchResult
    n, H, q = sol.net.n, sol.net.H, sol.net.q
    fields = [("V_m", (H, n, B), torch.float64), ("V_a", (H, n, B), torch.float64),
              ("I_inj", (q, H, B), torch.complex128), ("n_iter_f", (B,), torch.int32),
              ("n_iter_h", (B,), torch.int32), ("err_h", (B,), torch.float64), ("status", (B,), torch.int32),
              ("err_hist_f", (max_f + 1, B), torch.float64), ("err_hist_h", (max_h + 1, B), torch.float64)]
    off, lay = guard, []
    for name, shape, dt in fields:
        nb = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
        lay.append((name, off, nb, shape, dt))
        off = (off + nb + guard + 255) // 256 * 256
    buf = torch.full((off + guard,), 0xA5, dtype=torch.uint8, device=sol.device)
    views = {name: buf[o:o + nb].view(dt).view(shape) for name, o, nb, shape, dt in lay}
    mask = torch.ones(buf.numel(), dtype=torch.bool, device=sol.device)
    for _, o, nb, _, _ in lay:
        mask[o:o + nb] = False
    return BatchResult(**views), buf, mask


@pytest.mark.parametrize("kernel,case,B", [("warp", "net3_c_h25", 333), ("warp", "net2ev_uc_h19", 77),
                                           ("tile", "net3_c_h25", 333), ("dyn", "net3_c_h25", 45),
                                           ("dense", "net3_c_h25", 37), ("cta", "net1_c_h25", 5),
                                           ("blocked", "net1_c_h25", 3), ("warp", "net3_c_h25", 1)])
def test_guard_bands_and_repeatability(solvers, kernel, case, B, monkeypatch):
    """compute-sanitizer is closed on this GPU pool (profiles/sanitizer_unavailable.txt), so the
    persistent / warp-specialised kernels are checked with instruments of our own: (a) every output
    array sits between canary bands that must come back untouched (out-of-bounds writes), with the
    grid capped at 2 CTAs and a ragged batch so that every refill path runs; (b) three runs give
    bit-identical outputs and error histories (a data race between the warp roles, the
    double-buffered reductions or the work queue shows up as run-to-run differences); (c) the
    result equals the uncapped run's bit for bit (scheduling independence)."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    sol0, net, _ = solvers(case)
    if kernel == "tile":
        monkeypatch.setenv("HPF_HARM_KERNEL", "tile")
    if kernel == "dyn":
        monkeypatch.setenv("HPF_NO_SPECIALISE", "1")
    monkeypatch.setenv("HPF_MAX_CTAS", "2")
    sol = BatchSolver(net)
    dense = kernel in ("dense", "blocked")
    P, Q, I_N = scenarios.make_batch(net, B, "wide")
    dP, dQ, dI = sol.prepare(P, Q, I_N)
    runs = []
    for _ in range(3):
        res, buf, mask = _guarded_result(sol, B, 30, 50)
        sol.solve(dP, dQ, dI, dense=dense, out=res)
        torch.cuda.synchronize()
        assert bool((buf[mask] == 0xA5).all()), "a kernel wrote outside its output arrays"
        runs.append(buf.clone())
    assert torch.equal(runs[0], runs[1]) and torch.equal(runs[0], runs[2])
    got = res.to_host()
    sol.close()
    monkeypatch.delenv("HPF_MAX_CTAS")
    ref = BatchSolver(net) if kernel in ("tile", "dyn") else sol0
    want = ref.solve(dP, dQ, dI, dense=dense, history=True).to_host()
    if ref is not sol0:
        ref.close()
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status", "err_hist_f", "err_hist_h"):
        assert np.array_equal(got[k], want[k], equal_nan=True), k
    assert ((got["status"] == 0) | (got["status"] == 1)).all()       # ("wide" scenarios of net1 may hit the cap)
    assert (got["status"] == 0).any()


def test_guard_bands_large_network_variant(tmp_path, monkeypatch):
    """Same canary / repeatability check for the global-memory-state variant (variant 3: scenario
    state slabs, blocked tensor-core LU, multi-CTA operator set-up) on a small synthetic network."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    monkeypatch.setenv("HPF_STRUCT_VARIANT", "3")
    monkeypatch.setenv("HPF_MAX_CTAS", "2")
    net, _ = helpers.synthetic_packed("meshed", tmp_path, h_max=25, n=70, load_scale=0.02)
    sol = BatchSolver(net)
    assert sol.struct_info()["available"] == 3
    B = 7
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    runs = []
    for _ in range(2):
        res, buf, mask = _guarded_result(sol, B, 30, 50)
        sol.solve(P, Q, I_N, out=res)
        torch.cuda.synchronize()
        assert bool((buf[mask] == 0xA5).all()), "a kernel wrote outside its output arrays"
        runs.append(buf.clone())
    assert torch.equal(runs[0], runs[1])
    assert (res.to_host()["status"] == 0).all()
    sol.close()


@pytest.mark.parametrize("kind,n,variant,B", [("meshed", 70, 3, 200), ("radial", 40, 3, 67), ("net1", 0, 2, 130)])
def test_norton_contraction_dmma_matches_fma_and_definition(kind, n, variant, B, tmp_path, monkeypatch):
    """hpf_norton_wn: w_N = W_NL I_N of a whole batch on the FP64 tensor cores (zgemm_dmma_kernel,
    $HPF_WN_KERNEL=dmma) against the CUDA-core kernel ($HPF_WN_KERNEL=fma) and against the definition
    A_ZZ w_N = I_N,Z with A = blockdiag Y(h) - scatter(Y_N) built on the host (HG:313-357); ragged
    sizes (nZ, qH and B are not multiples of the 64 x 64 x 8 tiles)."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    if kind == "net1":
        net, _, _ = helpers.packed_from_files("net1", 25, True, tmp_path, julia_schema=True)
    else:
        monkeypatch.setenv("HPF_STRUCT_VARIANT", str(variant))
        net, _ = helpers.synthetic_packed(kind, tmp_path, h_max=25, n=n, load_scale=0.02)
    _, _, I_N = scenarios.make_batch(net, B, "wide")
    out = {}
    for kern in ("fma", "dmma"):
        monkeypatch.setenv("HPF_WN_KERNEL", kern)
        sol = BatchSolver(net)
        assert sol.struct_info()["available"] == variant
        out[kern] = sol.norton_wn(I_N).cpu().numpy()
        Y = sol.Y.cpu().numpy()
        sol.close()
    scale = np.abs(out["fma"]).max()
    assert np.abs(out["dmma"] - out["fma"]).max() <= 1e-13 * scale
    # definition: A_ZZ w = I_N,Z
    nn, m, H, q = net.n, net.m, net.H, net.q
    A = np.zeros((nn * H, nn * H), dtype=complex)
    for h in range(H):
        A[h * nn:(h + 1) * nn, h * nn:(h + 1) * nn] = Y[h]
    YN = net.Y_N[net.dev_of_nl_bus]                              # [q, H, H]
    for k in range(q):
        idx = np.arange(H) * nn + m + k
        A[np.ix_(idx, idx)] -= YN[k]
    Azz = A[m:, m:]
    rhs = np.zeros((nn * H - m, B), dtype=complex)
    for k in range(q):
        rhs[np.arange(H) * nn + k, :] = I_N[k]                    # row z = s - m = h n + k
    res = Azz @ out["dmma"] - rhs
    assert np.abs(res).max() <= 1e-9 * np.abs(rhs).max()


@pytest.mark.parametrize("gj", ["default", "blocked", "unblocked"])
@pytest.mark.parametrize("kind,n,coupled", [("meshed", 70, True), ("radial", 40, True), ("meshed", 30, False)])
def test_woodbury_setup_matches_gauss_jordan_setup(kind, n, coupled, gj, tmp_path, monkeypatch):
    """Large-network set-up (variant 3): the operators W_NL = A_ZZ^-1 E and G = A_ZZ^-1 A_ZF built
    through the block structure of A_ZZ (Woodbury identity: H block inversions, one inversion of
    order qH, complex GEMMs on the tensor cores) against the round-1 path (Gauss-Jordan inversion
    of the whole A_ZZ, $HPF_SETUP=gj): same w_N, same Newton step, same solve."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    monkeypatch.setenv("HPF_STRUCT_VARIANT", "3")
    net, _ = helpers.synthetic_packed(kind, tmp_path, h_max=25, coupled=coupled, n=n, load_scale=0.02)
    B = 24
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    out = {}
    # gj: which inversion kernels the Woodbury path uses - "default" (one-CTA kernel for these small
    # blocks), "blocked" (multi-CTA, panels of 64 pivots + tensor-core GEMM update: what the 1000-bus
    # configuration runs; partial panels and panels narrower than 64 included), "unblocked" (multi-CTA,
    # one rank-1 update per pivot)
    for setup in ("gj", "woodbury"):
        monkeypatch.setenv("HPF_SETUP", setup)
        if setup == "woodbury" and gj != "default":
            monkeypatch.setenv("HPF_GJ_SINGLE_MAX", "0")
            monkeypatch.setenv("HPF_GJ_UNBLOCKED", "1" if gj == "unblocked" else "0")
        sol = BatchSolver(net)
        info = sol.struct_info()
        assert info["available"] == 3 and info["pivot_min"] > 0
        if setup == "gj":                                      # ONE iterate for both (early iterations amplify round-off)
            raw = sol.solve(P, Q, I_N, raw=True, max_iter_h=2)
            Vm0, Va0 = raw.V_m.cpu().numpy(), raw.V_a.cpu().numpy()
        out[setup] = dict(wn=sol.norton_wn(I_N).cpu().numpy(),
                          dx=sol.newton_step(Vm0, Va0, P, Q, I_N).cpu().numpy(),
                          res=sol.solve(P, Q, I_N).to_host())
        sol.close()
    a, b = out["gj"], out["woodbury"]
    assert np.abs(a["wn"] - b["wn"]).max() <= 1e-11 * np.abs(a["wn"]).max()
    assert np.abs(a["dx"] - b["dx"]).max() <= 1e-9 * np.abs(a["dx"]).max()
    assert (b["res"]["status"] == 0).all()
    same = a["res"]["n_iter_h"] == b["res"]["n_iter_h"]
    assert same.mean() >= 0.75                                 # (round-off-decided counts, DESIGN.md section 4)
    Va, Vb = helpers.phasor(a["res"]["V_m"], a["res"]["V_a"]), helpers.phasor(b["res"]["V_m"], b["res"]["V_a"])
    # (an iterate accepted at mismatch norm e is ~e away from the solution)
    tol = np.maximum(a["res"]["err_h"], b["res"]["err_h"])[same]
    assert (np.abs(Va - Vb)[..., same].reshape(-1, same.sum()).max(0) <= np.maximum(1e-9, tol)).all()


def test_prepare_then_async_solves_two_streams_and_graph_capture(solvers):
    """hpf_prepare (ADVICE round 1): after it a solve of <= B_max scenarios neither allocates nor
    synchronises, so (a) two solves issued back to back on two different streams are ordered on the
    device by the handle (one kernel sequence in flight per handle) and both come out bit-identical
    to a solve alone, and (b) the solve can be captured into a CUDA graph and replayed."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    _, net, _ = solvers("net3_c_h25")
    sol = BatchSolver(net)
    B = 700
    sol.prepare_batch(B)
    Pa, Qa, Ia = sol.prepare(*scenarios.make_batch(net, B, "tight"))
    Pb, Qb, Ib = sol.prepare(*scenarios.make_batch(net, B, "wide"))
    torch.cuda.synchronize()
    want_a = sol.solve(Pa, Qa, Ia).to_host()
    want_b = sol.solve(Pb, Qb, Ib).to_host()
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(3):
        with torch.cuda.stream(s1):
            ra = sol.solve(Pa, Qa, Ia)
        with torch.cuda.stream(s2):
            rb = sol.solve(Pb, Qb, Ib)
        torch.cuda.synchronize()
        ga, gb = ra.to_host(), rb.to_host()
        for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
            assert np.array_equal(ga[k], want_a[k], equal_nan=True), k
            assert np.array_equal(gb[k], want_b[k], equal_nan=True), k
    # CUDA-graph capture of one solve, replayed on new inputs written into the captured buffers
    res, _slab = sol.alloc_result_slab(B)
    g = torch.cuda.CUDAGraph()
    sc = torch.cuda.Stream()
    sc.wait_stream(torch.cuda.current_stream())
    with torch.cuda.graph(g, stream=sc):
        rg = sol.solve(Pa, Qa, Ia, out=res)
    for want, src in ((want_a, None), (want_b, (Pb, Qb, Ib)), (want_a, (Pa.clone(), Qa.clone(), Ia.clone()))):
        if src is not None:
            Pa.copy_(src[0]); Qa.copy_(src[1]); Ia.copy_(src[2])
        g.replay()
        torch.cuda.synchronize()
        got = rg.to_host()
        for k in ("V_m", "V_a", "n_iter_h", "err_h", "status"):
            assert np.array_equal(got[k], want[k], equal_nan=True), k
    sol.close()


# ---------------------------------------------------------------- lock-step batched path (large networks)
@pytest.mark.parametrize("case,B", [("net2_c_h51", 9), ("net1_c_h25", 7), ("net1_c_h51", 7)])
def test_batched_lu_random_batch_and_singular(case, B, tmp_path, monkeypatch):
    """Kernel 4 through the BATCHED LU of hpf_lockstep.cuh ($HPF_LOCKSTEP=1): all matrices panel by
    panel - register panel (rows <= 512), register sub-panels of 8 columns with 2 / 4 rows per thread
    (N = 518 / 1038), panel staged in shared memory or in place, ragged last panel, tensor-core update
    tiles with ragged edges - against numpy and against the per-CTA blocked LU; one singular matrix."""
    from harmonic_power_flow_b200 import BatchSolver
    d = helpers.load_case(case)
    net, st, _ = helpers.packed_from_files(str(d["net"]), int(d["h_max"]), bool(d["coupled"]), tmp_path,
                                           julia_schema=str(d["net"]) == "net1")
    monkeypatch.setenv("HPF_LOCKSTEP", "0")
    ref_sol = BatchSolver(net)
    monkeypatch.setenv("HPF_LOCKSTEP", "1")
    sol = BatchSolver(net)
    N = sol.N
    rng = np.random.default_rng(3)
    A = rng.standard_normal((B, N, N))
    A[5, :, 3] = 0.0                                         # exactly singular -> zero pivot
    A[2, 40:60, :] *= 1e-3                                   # rows that lose every pivot search of their panel
    f = rng.standard_normal((N, B))
    stride = sol.jacobian_stride()
    J = torch.zeros((B, stride), dtype=torch.float64, device=sol.device)
    J[:, :N * N] = torch.as_tensor(A.reshape(B, -1)).to(sol.device)
    n0 = sol.launch_count
    dx, info = sol.lu_solve(J, f)
    assert sol.launch_count - n0 > 3 * (N // 32), "the batched LU did not run"
    dx0, info0 = ref_sol.lu_solve(J, f)
    dx, info, dx0 = dx.cpu().numpy(), info.cpu().numpy(), dx0.cpu().numpy()
    assert info[5] != 0 and (np.delete(info, 5) == 0).all()
    assert np.array_equal(info, info0.cpu().numpy())
    for b in range(B):
        if b == 5:
            continue
        ref = np.linalg.solve(A[b], f[:, b])
        assert np.abs(dx[:, b] - ref).max() <= 1e-9 * max(1.0, np.abs(ref).max()), b
        assert np.abs(dx[:, b] - dx0[:, b]).max() <= 1e-9 * max(1.0, np.abs(ref).max()), b
    sol.close()
    ref_sol.close()


@pytest.mark.parametrize("kind,n,B", [("meshed", 70, 150), ("radial", 40, 67), ("meshed", 30, 3)])
def test_lockstep_path_against_oracle_and_cta_path(kind, n, B, tmp_path, monkeypatch):
    """The lock-step batched harmonic stage (all scenarios take their Newton iteration together: batched
    tensor-core LU of the border systems, G products as complex GEMMs) forced onto small synthetic
    networks: against the oracle, against the per-CTA kernel, history / status outputs, bit-identical
    repeat, host-buffer entry point."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    monkeypatch.setenv("HPF_STRUCT_VARIANT", "3")
    net, _ = helpers.synthetic_packed(kind, tmp_path, h_max=25, n=n, load_scale=0.02)
    monkeypatch.setenv("HPF_LOCKSTEP", "0")
    cta = BatchSolver(net)
    monkeypatch.setenv("HPF_LOCKSTEP", "1")
    sol = BatchSolver(net)
    assert sol.struct_info()["available"] == 3
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    n0 = sol.launch_count
    r = sol.solve(P, Q, I_N, history=True)
    assert sol.launch_count - n0 > 50 and sol.last_solve_path == 4, "the lock-step path did not run"
    res = r.to_host()
    ref = cta.solve(P, Q, I_N, history=True).to_host()
    assert cta.last_solve_path == 3
    assert (res["status"] == 0).all()
    # The iteration count of these networks is decided by round-off in ~10 % of the scenarios (the oracle
    # with a LAPACK step against the oracle with the reference's SuperLU step: 19 of 150 on the 70-bus
    # network, lock-step 17, per-CTA kernel 21 - profiles/r2_lockstep_iteration_rates.txt), so the bar is
    # the oracle's own disagreement on the same sample; scenarios with equal counts must agree in V.
    import oracle_pool
    sample = np.arange(0, B, max(1, B // 24))
    pool = oracle_pool.OraclePool(helpers.oracle_net(net))
    try:
        o = pool.solve(P[:, sample], Q[:, sample], I_N[:, :, sample], "superlu", chunk=1)
        ol = pool.solve(P[:, sample], Q[:, sample], I_N[:, :, sample], "lapack", keep_V=False, chunk=1)
    finally:
        pool.close()
    floor = int((o["n_iter_h"] != ol["n_iter_h"]).sum())
    mism = int((res["n_iter_h"][sample] != o["n_iter_h"]).sum())
    print("\nlock-step %s-%d: %d/%d iteration-count differences against the SuperLU oracle (oracle vs itself: %d)" % (
        kind, n, mism, len(sample), floor))
    assert mism <= floor + max(1, len(sample) // 10)
    assert np.array_equal(res["n_iter_f"][sample], o["n_iter_f"]) and (o["status"] == 0).all()
    Vg, Vo = helpers.phasor(res["V_m"], res["V_a"]), helpers.phasor(o["V_m"], o["V_a"])
    for k, b in enumerate(sample):
        if res["n_iter_h"][b] == o["n_iter_h"][k]:
            t = max(1e-9, 0.1 * max(o["err_h"][k], res["err_h"][b]))
            assert np.abs(Vo[:, :, k] - Vg[:, :, b]).max() <= t * np.abs(Vo[:, :, k]).max(), b
    assert np.array_equal(res["n_iter_f"], ref["n_iter_f"])
    same = res["n_iter_h"] == ref["n_iter_h"]
    assert (~same).sum() <= max(1, B // 10), "iteration counts differ from the per-CTA kernel in %d of %d" % ((~same).sum(), B)
    V = helpers.phasor(res["V_m"], res["V_a"])
    V0 = helpers.phasor(ref["V_m"], ref["V_a"])
    for b in np.nonzero(same)[0]:
        t = max(1e-9, 0.1 * max(res["err_h"][b], ref["err_h"][b]))
        assert np.abs(V[:, :, b] - V0[:, :, b]).max() <= t * np.abs(V0[:, :, b]).max(), b
        k = int(res["n_iter_h"][b]) + 1
        # (the first steps agree to round-off; later the iteration amplifies it, see above)
        assert np.allclose(res["err_hist_h"][:3, b], ref["err_hist_h"][:3, b], rtol=1e-6), b
        assert res["err_hist_h"][k - 1, b] == res["err_h"][b] and np.isfinite(res["err_hist_h"][:k, b]).all()
        assert np.isnan(res["err_hist_h"][k:, b]).all()
    # bit-identical when repeated and for a split of the batch (positions in the batch do not enter the arithmetic)
    again = sol.solve(P, Q, I_N).to_host()
    for k in ("V_m", "V_a", "I_inj", "n_iter_h", "err_h", "status"):
        assert np.array_equal(again[k], res[k]), k
    if B - B // 3 >= 64:                                      # (w_N of batches under 64 scenarios comes from the CUDA-core kernel)
        lo = B // 3
        part = sol.solve(P[:, lo:].copy(), Q[:, lo:].copy(), I_N[:, :, lo:].copy()).to_host()
        assert np.array_equal(part["V_m"], res["V_m"][:, :, lo:]) and np.array_equal(part["n_iter_h"], res["n_iter_h"][lo:])
    rh = sol.solve_host(P, Q, I_N)
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(rh[k], res[k]), k
    # iteration cap: status 1 (max-iter) and the count at the cap
    capped = sol.solve(P, Q, I_N, max_iter_h=3).to_host()
    assert (capped["n_iter_h"] == 3).all() and (capped["status"] == 1).all()
    sol.close()
    cta.close()


def test_lockstep_waves_when_memory_budget_is_small(tmp_path, monkeypatch):
    """A memory budget that holds only part of the batch: the lock-step path runs in waves of slots and
    gives the same bits as one wave."""
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    monkeypatch.setenv("HPF_STRUCT_VARIANT", "3")
    monkeypatch.setenv("HPF_LOCKSTEP", "1")
    net, _ = helpers.synthetic_packed("radial", tmp_path, h_max=25, n=40, load_scale=0.02)
    sol = BatchSolver(net)
    B = 45
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    n0 = sol.launch_count
    one = sol.solve(P, Q, I_N).to_host()
    n_one = sol.launch_count - n0
    sol.close()
    monkeypatch.setenv("HPF_LOCKSTEP_GB", "0.001")           # ~1 MB: about a dozen slots
    sol = BatchSolver(net)
    n0 = sol.launch_count
    waves = sol.solve(P, Q, I_N).to_host()
    assert sol.launch_count - n0 > 2 * n_one, "the batch was not split into waves"
    for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
        assert np.array_equal(waves[k], one[k]), k
    sol.close()


def test_config5_lockstep_nominal_against_oracle_run(tmp_path, monkeypatch):
    """BASELINE config 5 network through the lock-step path (border systems of order 1198: register
    sub-panels with 4 and 2 rows per thread, panels in place and staged): the oracle's summary for the
    nominal scenario (see test_config5_meshed_1000_bus_nominal_against_oracle_run), three copies."""
    from harmonic_power_flow_b200 import BatchSolver
    monkeypatch.setenv("HPF_LOCKSTEP", "1")
    net, _ = helpers.synthetic_packed("meshed", tmp_path, h_max=25, n=1000, load_scale=0.002)
    sol = BatchSolver(net)
    B = 3
    r = sol.solve(np.repeat(net.P[:, None], B, 1), np.repeat(net.Q[:, None], B, 1),
                  np.repeat(net.I_N[:, :, None], B, 2)).to_host()
    for b in range(B):
        assert r["status"][b] == 0 and r["n_iter_f"][b] == 2 and r["n_iter_h"][b] == 26
        assert r["err_h"][b] == pytest.approx(4.085e-06, rel=0.05)
        assert r["V_m"][0, :, b].max() == pytest.approx(1.1649555668183993, rel=1e-11)
        assert r["V_m"][1, :, b].max() == pytest.approx(0.5791799507662769, rel=1e-11)
    assert np.array_equal(r["V_m"][:, :, 0], r["V_m"][:, :, 2])
    sol.close()
