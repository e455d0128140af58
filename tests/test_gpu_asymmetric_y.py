"""Every solve path on admittance tables other than the reference builder's symmetric Y(h).

A phase-shifting transformer makes Y(h) asymmetric (Y[f,t] != Y[t,f]), the corrected Y options
change the diagonal and sum parallel lines, and hpf_set_Y takes any table.  The kernels read Y(h)
by rows, through host mirrors in kernel parameter banks, through the ELL pattern and through the
structured operators A_ZZ / A_ZF, G and W_NL: a transposed read, or an operator not rebuilt after
Y(h) changed, passes every test on a symmetric table and fails here.  References: the CPU oracle
given the same table (hpf_oracle.hpf / pf take any Y), and fresh handles bit for bit."""
import contextlib
import os

import numpy as np
import pytest
import torch

import helpers
import hpf_oracle as O

pytestmark = pytest.mark.gpu


def trafo(L, k, seed, tmax, pmax):
    """Seeded transformer draw: k of the L lines get tap tau ~ U(1 - tmax, 1 + tmax) and phase
    shift phi ~ U(-pmax, pmax) degrees, the others stay plain lines.  -> (tau, phi)."""
    rng = np.random.default_rng(seed)
    tau, phi = np.ones(L), np.zeros(L)
    idx = rng.choice(L, k, replace=False)
    tau[idx] = rng.uniform(1 - tmax, 1 + tmax, k)
    phi[idx] = rng.uniform(-pmax, pmax, k)
    return tau, phi


# network: how it is built, the transformer draw (lines, seed, tau range, phi range), batch size,
# scenarios checked against the oracle (the oracle needs seconds per scenario on the larger two).
# capped: some "tight" scenarios of net1 stop at the 50-iteration cap, with and without transformers
# and in the oracle too (6 or 7 of these 40 with this draw); the sampled ones converge.
NETS = {
    "net3_c_h25": dict(files=("net3", 25, True), draw=(None, 1, 0.05, 5.0), B=333, sample=16),
    "net3_uc_h25": dict(files=("net3", 25, False), draw=(None, 1, 0.05, 5.0), B=333, sample=16),
    "net2ev_c_h19": dict(files=("net2ev", 19, True), draw=(None, 1, 0.05, 5.0), B=333, sample=16),
    "net1_c_h25": dict(files=("net1", 25, True), draw=(3, 2, 0.02, 3.0), B=40, sample=3,
                       capped=True),
    "meshed70": dict(synthetic=("meshed", 70, 0.02), draw=(8, 5, 0.02, 3.0), B=40, sample=3),
}

# configuration: (network, environment of the handle, struct_info()["available"], last_solve_path, dense)
CONFIGS = {
    "net3_c_h25": ("net3_c_h25", {}, 1, 1, False),              # shape 1: harm_hw / lane kernels
    "net3_uc_h25": ("net3_uc_h25", {}, 1, 1, False),            # uncoupled harm_hw_kernel
    "net2ev_c_h19": ("net2ev_c_h19", {}, 1, 1, False),          # shape 2
    "net3_c_h25-tile": ("net3_c_h25", {"HPF_HARM_KERNEL": "tile"}, 1, 1, False),
    "net3_c_h25-dyn": ("net3_c_h25", {"HPF_NO_SPECIALISE": "1"}, 1, 1, False),
    "net1_c_h25": ("net1_c_h25", {}, 2, 2, False),              # per-CTA kernel, ELL pattern
    "meshed70-v3": ("meshed70", {"HPF_STRUCT_VARIANT": "3", "HPF_LOCKSTEP": "0"}, 3, 3, False),
    "meshed70-lockstep": ("meshed70", {"HPF_STRUCT_VARIANT": "3", "HPF_LOCKSTEP": "1"}, 3, 4, False),
    "net3_c_h25-dense": ("net3_c_h25", {}, 1, 5, True),         # shared-memory LU
    "net1_c_h25-dense": ("net1_c_h25", {}, 2, 5, True),         # global-memory LU
}
STRUCTURED = [k for k, v in CONFIGS.items() if not v[4]]
FIELDS = ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status")


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / np.abs(np.asarray(b)).max()


@contextlib.contextmanager
def _env(env):
    """The handle reads its switches when it is created."""
    old = {k: os.environ.get(k) for k in env}
    os.environ.update(env)
    try:
        yield
    finally:
        for k, v in old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _make(net, env):
    from harmonic_power_flow_b200 import BatchSolver
    with _env(env):
        return BatchSolver(net)


def _with_parallel_line_and_shunts(net, seed):
    """Copy of `net` with a second line in parallel to the first line at bus 1 and a pi-shunt on
    every line, so that both corrected Y options change Y(h) and FIX_SHUNT_INDEX puts a shunt on
    the slack bus."""
    import copy
    net = copy.deepcopy(net)
    rng = np.random.default_rng(seed)
    l0 = int(np.nonzero((net.from_id == 1) | (net.to_id == 1))[0][0])
    net.from_id = np.append(net.from_id, net.from_id[l0]).astype(np.int32)
    net.to_id = np.append(net.to_id, net.to_id[l0]).astype(np.int32)
    net.R = np.append(net.R, 1.5 * net.R[l0]); net.X = np.append(net.X, 1.2 * net.X[l0])
    y = np.abs(1 / (net.R + 1j * net.X))                       # shunts of 0.1 .. 1 % of the series admittance
    net.G = y * rng.uniform(1e-3, 1e-2, len(net.R)); net.B = y * rng.uniform(1e-3, 1e-2, len(net.R))
    return net


@pytest.fixture(scope="module")
def nets(tmp_path_factory):
    """key -> dict(net=PackedNet, on=oracle Net, tau, phi, Yt=oracle table with transformers,
    P, Q, I_N: nominal scenario first, then seeded "tight" scenarios)."""
    from harmonic_power_flow_b200 import scenarios
    cache = {}

    def get(key):
        if key not in cache:
            spec = NETS[key]
            tmp = tmp_path_factory.mktemp(key)
            if "files" in spec:
                name, h_max, coupled = spec["files"]
                net, _, _ = helpers.packed_from_files(name, h_max, coupled, tmp, julia_schema=name == "net1")
            else:
                kind, n, scale = spec["synthetic"]
                net, _ = helpers.synthetic_packed(kind, tmp, h_max=25, n=n, load_scale=scale)
            on = helpers.oracle_net(net)
            L = len(net.R)
            k, seed, tmax, pmax = spec["draw"]
            tau, phi = trafo(L, L if k is None else k, seed, tmax, pmax)
            B = spec["B"]
            P, Q, I_N = scenarios.make_batch(net, B - 1, "tight")
            P = np.concatenate([net.P[:, None], P], 1)
            Q = np.concatenate([net.Q[:, None], Q], 1)
            I_N = np.concatenate([net.I_N[:, :, None], I_N], 2)
            sample = np.unique(np.linspace(0, B - 1, spec["sample"]).astype(int))
            cache[key] = dict(net=net, on=on, tau=tau, phi=phi, Yt=O.build_admittance_matrices_trafo(on, tau, phi),
                              P=P, Q=Q, I_N=I_N, sample=sample, capped=spec.get("capped", False), oracle={})
        return cache[key]
    return get


@pytest.fixture(scope="module")
def handles(nets):
    """config -> (handle with the network's transformers set, network record)."""
    cache = {}

    def get(config):
        if config not in cache:
            key, env, avail, _, _ = CONFIGS[config]
            d = nets(key)
            sol = _make(d["net"], env)
            sol.set_transformers(d["tau"], d["phi"])
            assert sol.struct_info()["available"] == avail
            cache[config] = (sol, d)
        return cache[config]
    yield get
    for sol, _ in cache.values():
        sol.close()


def _oracle(d, tag, Y, b, solver):
    """O.hpf of scenario b on table Y, cached per network record (configurations share it)."""
    key = (tag, int(b), solver)
    if key not in d["oracle"]:
        d["oracle"][key] = O.hpf(d["on"], P=d["P"][:, b], Q=d["Q"][:, b], I_N=d["I_N"][:, :, b], Y=Y, solver=solver)
    return d["oracle"][key]


def _check_fund(sol, on, Y):
    """Fundamental stage against O.pf on the same table."""
    V_m, V_a, nf, err, hist = sol.fund_solve(on.P[:, None], on.Q[:, None], history=True)
    Vo_m, Vo_a, errs, n_iter_f = O.pf(on, Y)
    assert int(nf.item()) == n_iter_f
    V = helpers.phasor(V_m[:, :, 0].cpu().numpy(), V_a[:, :, 0].cpu().numpy())
    assert np.abs(V - helpers.phasor(Vo_m, Vo_a)).max() < 1e-12
    h = hist[:, 0].cpu().numpy()
    k = len(errs)
    assert np.allclose(h[:k], errs, rtol=1e-6, atol=1e-12)             # last entry is round-off
    assert np.isnan(h[k:]).all()


def _check_solve(sol, d, tag, Y, dense, path):
    """Whole solve of the record's batch against O.hpf on table Y (SuperLU and LAPACK steps)."""
    on, P, Q, I_N = d["on"], d["P"], d["Q"], d["I_N"]
    res = sol.solve(P, Q, I_N, dense=dense, history=True).to_host()
    assert sol.last_solve_path == path
    assert np.isin(res["status"], (0, 1) if d["capped"] else (0,)).all()
    mism = floor = 0
    for b in d["sample"]:
        o, ol = _oracle(d, tag, Y, b, "superlu"), _oracle(d, tag, Y, b, "lapack")
        tag_b = "scenario %d: oracle it %d/%d err %.2e (lapack step: %d), gpu it %d/%d err %.2e" % (
            b, o["n_iter_f"], o["n_iter_h"], o["err_h"], ol["n_iter_h"], res["n_iter_f"][b], res["n_iter_h"][b],
            res["err_h"][b])
        assert o["status"] == 0 and res["status"][b] == 0, tag_b
        assert res["n_iter_f"][b] == o["n_iter_f"], tag_b
        floor += int(o["n_iter_h"] != ol["n_iter_h"])
        # the error path: tight at the start, before the iteration amplifies round-off (1e-9, or 10x
        # what the oracle's two steps differ by there: 3.8e-9 on one net3 scenario)
        self4 = (np.abs(o["err_h_hist"][:4] - ol["err_h_hist"][:4]) / ol["err_h_hist"][:4]).max()
        assert np.allclose(res["err_hist_h"][:4, b], o["err_h_hist"][:4], rtol=max(1e-9, 10 * self4)), tag_b
        V = helpers.phasor(res["V_m"][:, :, b], res["V_a"][:, :, b])
        if res["n_iter_h"][b] != o["n_iter_h"]:
            mism += 1
        else:
            # an iterate accepted at mismatch norm e is ~||J^-1|| e away from the converged one: two
            # iterates accepted at 1.8e-8 and 3e-9 after 19 steps differ by 1.1e-8 (corrected options, net3)
            t = max(1e-9, max(o["err_h"], res["err_h"][b]))
            Vo = helpers.phasor(o["V_m"], o["V_a"])
            assert (np.abs(V - Vo) / np.abs(Vo)).max() <= t, tag_b
        want = O.current_injections(on, V, I_N[:, :, b])
        assert np.abs(res["I_inj"][:, :, b] - want).max() <= 1e-12 * np.abs(want).max(), tag_b
    print("\n%s: %d/%d iteration-count differences against the SuperLU oracle (oracle vs itself: %d)" % (
        tag, mism, len(d["sample"]), floor))
    assert mism <= floor + 1


def _iterates(net, B, seed, near=None):
    """Random iterates as the Newton step tests draw them; `near` = (V_m, V_a) [H, n]: magnitudes
    within 10 % and angles within 0.1 rad of it instead (as the mismatch tests draw them)."""
    rng = np.random.default_rng(seed)
    H, n = net.H, net.n
    if near is None:
        Vm = rng.uniform(0.05, 0.3, (H, n, B)) * rng.choice([-1.0, 1.0], (H, n, B))
        Vm[0] = rng.uniform(0.9, 1.1, (n, B))
        Va = rng.uniform(-3, 3, (H, n, B)); Va[0, 0] = 0.0; Vm[0, 0] = 1.0
    else:
        Vm = near[0][:, :, None] * rng.uniform(0.9, 1.1, (H, n, B))
        Va = near[1][:, :, None] + rng.uniform(-0.1, 0.1, (H, n, B))
    P = net.P[:, None] * rng.uniform(0.8, 1.2, (n, B))
    Q = net.Q[:, None] * rng.uniform(0.8, 1.2, (n, B))
    I_N = net.I_N[:, :, None] * rng.uniform(0.9, 1.1, (net.q, H, B))
    return Vm, Va, P, Q, I_N


def _A_ZZ(net, Y):
    """A_ZZ of the structured step: rows / columns z = s - m of blockdiag Y(h) - scatter(Y_N)."""
    nn, m, H = net.n, net.m, net.H
    A = np.zeros((nn * H, nn * H), dtype=complex)
    for h in range(H):
        A[h * nn:(h + 1) * nn, h * nn:(h + 1) * nn] = Y[h]
    YN = net.Y_N[net.dev_of_nl_bus]
    for k in range(net.q):
        idx = np.arange(H) * nn + m + k
        A[np.ix_(idx, idx)] -= YN[k] if net.coupled else np.diag(YN[k])
    return A[m:, m:]


# ---------------------------------------------------------------- 1. Y(h) with transformers
@pytest.mark.parametrize("key", ["net3_c_h25", "net2ev_c_h19", "net1_c_h25", "meshed70"])
def test_trafo_ybus_with_nonlinear_buses_is_asymmetric(nets, key):
    from harmonic_power_flow_b200 import BatchSolver
    d = nets(key)
    sol = BatchSolver(d["net"])
    Y = sol.set_transformers(d["tau"], d["phi"]).cpu().numpy()
    sol.close()
    want = d["Yt"]
    assert np.abs(Y - want).max() <= 4e-15 * np.abs(want).max()
    assert ((Y == 0) == (want == 0)).all()
    assert np.abs(Y - np.swapaxes(Y, 1, 2)).max() > 1e-4 * np.abs(Y).max()


# ---------------------------------------------------------------- 2. elementwise kernels and one step
@pytest.mark.parametrize("config", STRUCTURED)
def test_kernels_at_asymmetric_y_against_oracle(handles, config):
    """Mismatch and I_inj (default kernel and the tile kernel), Jacobian, bus currents, w_N and one
    structured Newton step on a ragged random batch, against the oracle on the transformer table."""
    sol, d = handles(config)
    net, on, Y = d["net"], d["on"], d["Yt"]
    B = 77
    fm, fa, _, _ = O.pf(on, Y)
    Vm, Va, P, Q, I_N = _iterates(net, B, 5, near=(fm, fa))
    sample = (0, 31, 32, 63, 76)
    tile = _make(net, dict(CONFIGS[config][1], HPF_MISMATCH_TILE="1"))
    tile.set_transformers(d["tau"], d["phi"])
    got = [[t.cpu().numpy() for t in s.mismatch(Vm, Va, P, Q, I_N, want_I_inj=True)] for s in (sol, tile)]
    tile.close()
    J = sol.jacobian_view(sol.jacobian(Vm[:, :, sample], Va[:, :, sample])).cpu().numpy()
    I = sol.bus_currents(Vm, Va).cpu().numpy()
    for k, b in enumerate(sample):
        fo, eo = O.harmonic_mismatch(on, P[:, b], Q[:, b], Vm[:, :, b], Va[:, :, b], Y, I_N[:, :, b])
        V = helpers.phasor(Vm[:, :, b], Va[:, :, b])
        inj_o = O.current_injections(on, V, I_N[:, :, b])
        for f, err, inj in got:
            assert _rel(f[:, b], fo) <= 1e-13 and err[b] == pytest.approx(eo, rel=1e-13), b
            assert _rel(inj[:, :, b], inj_o) <= 1e-13, b
        assert _rel(J[k], O.build_harmonic_jacobian(on, Vm[:, :, b], Va[:, :, b], Y)) <= 1e-13, b
        want = np.einsum("hij,hj->hi", Y, V)
        assert np.abs(I[:, :, b] - want).max() <= 1e-12 * np.abs(want).max(), b
    # w_N: A_ZZ w = I_N,Z with A built from the asymmetric table
    wn = sol.norton_wn(I_N).cpu().numpy()
    rhs = np.zeros((net.n * net.H - net.m, B), dtype=complex)
    for k in range(net.q):
        rhs[np.arange(net.H) * net.n + k, :] = I_N[k]
    assert np.abs(_A_ZZ(net, Y) @ wn - rhs).max() <= 1e-9 * np.abs(rhs).max()
    # one structured Newton step against J^-1 f on the oracle's J and f
    Vm, Va, P, Q, I_N = _iterates(net, B, 17)
    dx = sol.newton_step(Vm, Va, P, Q, I_N).cpu().numpy()
    for b in sample:
        Jo = O.build_harmonic_jacobian(on, Vm[:, :, b], Va[:, :, b], Y)
        fo, _ = O.harmonic_mismatch(on, P[:, b], Q[:, b], Vm[:, :, b], Va[:, :, b], Y, I_N[:, :, b])
        ref = np.linalg.solve(Jo, fo)
        assert np.abs(dx[:, b] - ref).max() <= 1e-7 * np.abs(ref).max(), b
        assert np.abs(Jo @ dx[:, b] - fo).max() <= 1e-9 * np.abs(fo).max(), b


# ---------------------------------------------------------------- 3. fundamental stage
@pytest.mark.parametrize("config", STRUCTURED)
def test_fundamental_stage_at_asymmetric_y(handles, config):
    sol, d = handles(config)
    _check_fund(sol, d["on"], d["Yt"])


# ---------------------------------------------------------------- 4. whole solve
@pytest.mark.parametrize("config", list(CONFIGS))
def test_solve_at_asymmetric_y_against_oracle(handles, config):
    """Nominal scenario plus seeded "tight" scenarios (333 on the 4-bus networks: the work queue
    refills lanes) on the transformer table, a sample against the oracle."""
    sol, d = handles(config)
    _, _, _, path, dense = CONFIGS[config]
    _check_solve(sol, d, "trafo", d["Yt"], dense, path)


# ---------------------------------------------------------------- 5. corrected Y options
@pytest.mark.parametrize("key", ["net3_c_h25", "net1_c_h25"])
def test_corrected_y_options_through_a_solve(nets, key):
    """FIX_SHUNT_INDEX | SUM_PARALLEL on a network with a parallel line at bus 1 and pi-shunts:
    Y(h) is the textbook matrix, and the fundamental stage and the whole solve on it match the
    oracle given the same table."""
    from harmonic_power_flow_b200 import BatchSolver
    base = nets(key)
    net = _with_parallel_line_and_shunts(base["net"], 3)
    d = dict(base, net=net, on=helpers.oracle_net(net), oracle={})
    sol = BatchSolver(net)
    Y_ref_behaviour = sol.Y.cpu().numpy().copy()
    Y = sol.set_y_options(fix_shunt_index=True, sum_parallel=True).cpu().numpy()
    want = helpers.textbook_admittance(net)
    assert np.abs(Y - want).max() <= 1e-13 * np.abs(want).max()
    assert np.abs(Y - Y_ref_behaviour).max() > 1e-3 * np.abs(want).max()
    # the pi-shunts at the slack bus (FIX_SHUNT_INDEX only) are far above the tolerance of that check
    sh0 = sum((net.G[l] + 1j * net.B[l]) / 2 for l in range(len(net.R)) if 1 in (net.from_id[l], net.to_id[l]))
    assert abs(sh0) > 1e-6 * np.abs(want).max()
    _check_fund(sol, d["on"], Y)
    _check_solve(sol, d, "options", Y, False, CONFIGS[key][3])
    sol.close()


# ---------------------------------------------------------------- 6. Y(h) changed on a live handle
def _calls(sol, inp, B_dense):
    """Every entry point that reads Y(h) or something derived from it; numpy copies."""
    Vm, Va, P, Q, I_N = inp
    out = {}
    r = sol.solve(P, Q, I_N, history=True).to_host()
    out.update({"s_" + k: v for k, v in r.items()})
    r = sol.solve(P[:, :B_dense], Q[:, :B_dense], I_N[:, :, :B_dense], dense=True, history=True).to_host()
    out.update({"d_" + k: v for k, v in r.items()})
    f, err, inj = sol.mismatch(Vm, Va, P, Q, I_N, want_I_inj=True)
    out.update(f=f.cpu().numpy(), err=err.cpu().numpy(), inj=inj.cpu().numpy())
    out["dx"] = sol.newton_step(Vm, Va, P, Q, I_N).cpu().numpy()
    out["wn"] = sol.norton_wn(I_N).cpu().numpy()
    r = sol.solve_host(P, Q, I_N)
    out.update({"h_" + k: np.array(v, copy=True) for k, v in r.items()})
    return out


def _same(a, b):
    for k in a:
        assert np.array_equal(a[k], b[k], equal_nan=True), k


@pytest.mark.parametrize("prepared", [False, True])
@pytest.mark.parametrize("config", ["net3_c_h25", "net1_c_h25", "meshed70-v3", "meshed70-lockstep"])
def test_y_changes_on_a_live_handle(nets, config, prepared):
    """set_transformers, set_y_options and set_Y on a handle that has already solved: every entry
    point then gives the bits of a fresh handle that had the same table before its first solve, and
    undoing the change gives the first bits again (no stale constant bank, host mirror, ELL pattern,
    structured operator or lock-step state)."""
    key, env, _, _, _ = CONFIGS[config]
    base = nets(key)
    net = _with_parallel_line_and_shunts(base["net"], 4)
    on = helpers.oracle_net(net)
    tau, phi = trafo(len(net.R), len(net.R) if NETS[key]["draw"][0] is None else NETS[key]["draw"][0], 7, 0.02, 3.0)
    Yx = O.build_admittance_matrices_trafo(on, tau, phi)
    B = 64 if net.n <= 4 else 8
    Vm, Va, P, Q, I_N = _iterates(net, B, 9)
    inp = (Vm, Va, P, Q, I_N)
    Bd = min(B, 8)
    sol = _make(net, env)
    if prepared:
        sol.prepare_batch(B)
    plain = _calls(sol, inp, Bd)
    Y0 = sol.Y.cpu().numpy().copy()
    changes = [("transformers", lambda s: s.set_transformers(tau, phi), lambda s: s.set_transformers(None)),
               ("options", lambda s: s.set_y_options(True, True), lambda s: s.set_y_options()),
               ("table", lambda s: s.set_Y(Yx), lambda s: s.set_Y(Y0))]
    for what, change, undo in changes:
        change(sol)
        got = _calls(sol, inp, Bd)
        fresh = _make(net, env)
        change(fresh)
        want = _calls(fresh, inp, Bd)
        fresh.close()
        assert not np.array_equal(got["s_V_m"], plain["s_V_m"]), what     # the change matters
        _same(got, want)
        undo(sol)
        _same(_calls(sol, inp, Bd), plain)
    sol.close()


# ---------------------------------------------------------------- 7. drop-in pf(Y, buses)
def test_reference_shaped_pf_twice_on_its_cached_handle(tmp_path):
    """pf(Y, buses) keeps one GPU handle per bus table: a plain table and then a transformer table
    through the same handle, each against the oracle's pf on that table."""
    from harmonic_power_flow_b200 import hcne_generalized as hg
    pb, pl = helpers.write_net_csvs("net3", str(tmp_path))
    helpers.write_ne_csvs(str(tmp_path))
    hg.configure(H_MAX=25, ne_dir=str(tmp_path))
    try:
        buses, lines, m, n, c = hg.init_network(pb, pl)
        Y = hg.build_admittance_matrices(buses, lines, hg.HARMONICS)
        on = O.net_from_golden(helpers.GOLDEN, "net3", 25, True)
        tau, phi = trafo(len(on.R), len(on.R), 1, 0.05, 5.0)
        Yt = O.build_admittance_matrices_trafo(on, tau, phi)
        Ydf = Y.copy()
        Ydf.loc[:, :] = Yt.reshape(Y.shape)
        n_handles = None
        for table, Yo in ((Y, Y.to_numpy().reshape(Yt.shape)), (Ydf, Yt)):
            V_f, err_t, n_iter_f = hg.pf(table, buses)
            if n_handles is None:
                n_handles = len(hg._SOLVERS)
            assert len(hg._SOLVERS) == n_handles
            Vo_m, Vo_a, _, nfo = O.pf(on, Yo)
            assert n_iter_f == nfo and len(err_t) == n_iter_f
            assert np.abs(helpers.phasor(V_f["V_m"], V_f["V_a"]) - helpers.phasor(Vo_m, Vo_a).ravel()).max() < 1e-12
    finally:
        hg.release_solvers()
        hg.configure(H_MAX=51)


# ---------------------------------------------------------------- 8. hpf_set_Y after in-flight work
def test_set_Y_waits_for_a_solve_in_flight(nets):
    """A solve enqueued on a side stream behind a long sleep, then set_Y from the host at once: the
    solve must finish on the table it was issued with."""
    d = nets("net3_c_h25")
    net = d["net"]
    sol = _make(net, {})
    Y1 = d["Yt"]
    Y2 = sol.Y.cpu().numpy().copy()
    B = 333
    sol.prepare_batch(B)
    sol.set_Y(Y1)
    P, Q, I_N = sol.prepare(d["P"], d["Q"], d["I_N"])
    # warm-up: the first solve after a Y(h) change synchronises the device (host mirrors, set-up)
    want = sol.solve(P, Q, I_N).to_host()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        torch.cuda._sleep(500_000_000)
        r = sol.solve(P, Q, I_N)
    sol.set_Y(Y2)
    torch.cuda.synchronize()
    got = r.to_host()
    for k in FIELDS:
        assert np.array_equal(got[k], want[k], equal_nan=True), k
    sol.close()
