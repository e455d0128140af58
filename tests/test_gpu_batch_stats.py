"""Batch statistics on the device (hpf_batch_stats) and the host solve that returns only them
(hpf_solve_host_stats), against the numpy reference (oracle/stats_oracle.py) on the same device arrays.
THD is taken from hpf_thd: the reference takes it as an input (an FMA-free numpy restatement differs in
the last bit)."""
import contextlib
import ctypes as C
import os

import numpy as np
import pytest
import torch

import helpers
import stats_oracle as S

pytestmark = pytest.mark.gpu

B_BIG = 65536
Q3 = (0.05, 0.5, 0.95)
Q16 = (0.0, 0.001, 0.01, 0.05, 0.1, 0.25, 1 / 3, 0.5, 0.5, 2 / 3, 0.75, 0.9, 0.95, 0.99, 0.999, 1.0)


@contextlib.contextmanager
def _env(env):
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


def _bits(a):
    return np.ascontiguousarray(np.asarray(a, np.float64)).view(np.uint64)


def _np(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def _check(bs, V_m, thd, status, q, lim_rows):
    """GPU statistics against the reference: counts, min, max, exceed and quantiles bit for bit, mean and
    std to 1e-12 of the row's largest magnitude."""
    counts, want = S.batch_stats(_np(V_m), _np(thd), None if status is None else _np(status), q, lim_rows)
    got = _np(bs.planes)
    assert np.array_equal(_np(bs.status_counts), counts)
    assert got.shape == want.shape
    exact = [2, 3, 4] + list(range(5, 5 + len(q)))
    assert np.array_equal(_bits(got[exact]), _bits(want[exact])), np.nonzero(_bits(got[exact]) != _bits(want[exact]))
    X = np.concatenate([_np(V_m).reshape(-1, _np(V_m).shape[2]), _np(thd).reshape(-1, _np(thd).shape[2])])
    inc = np.ones(X.shape[1], bool) if status is None else _np(status) == 0
    if inc.any():
        scale = np.abs(X[:, inc]).max(axis=1)
        for p in (0, 1):
            assert (np.abs(got[p] - want[p]) <= 1e-12 * scale).all(), (p, np.abs(got[p] - want[p]).max())
    else:
        assert np.isnan(got[[0, 1]]).all()


@pytest.fixture(scope="module")
def net3(tmp_path_factory):
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    net, _, _ = helpers.packed_from_files("net3", 25, True, tmp_path_factory.mktemp("net3"))
    sol = BatchSolver(net)
    P, Q, I_N = scenarios.make_batch(net, B_BIG, "tight")
    return dict(net=net, sol=sol, P=P, Q=Q, I_N=I_N)


@pytest.fixture(scope="module")
def solved(net3):
    sol = net3["sol"]
    r = sol.solve(net3["P"], net3["Q"], net3["I_N"])
    thd = sol.thd(r.V_m)
    torch.cuda.synchronize()
    return r, thd


def _limits(net, V_m):
    """Limits that some rows' scenarios exceed and others' do not: the median of the first 1,000
    scenarios for V_m, none for THD_R, one value for THD_F."""
    return {"V_m": np.median(_np(V_m)[:, :, :1000], axis=2), "THD_F": 0.02}


@pytest.mark.parametrize("q", [(), Q3, Q16], ids=["K0", "K3", "K16"])
def test_solved_batch_matches_reference(net3, solved, q):
    from harmonic_power_flow_b200.solver import stats_limit_rows
    sol, net = net3["sol"], net3["net"]
    r, thd = solved
    lim = _limits(net, r.V_m)
    bs = sol.batch_stats(r.V_m, r.status, quantiles=q, limits=lim)
    rows = stats_limit_rows(lim, net.n, net.H)
    _check(bs, r.V_m, thd, r.status, q, rows)
    ex = _np(bs.planes[4])
    assert (ex > 0).any() and (ex == 0).any()
    # the accessors pick the layout apart
    nH = net.n * net.H
    assert np.array_equal(_np(bs.V_m("max")), _np(bs.planes[3, :nH]).reshape(net.H, net.n))
    assert np.array_equal(_np(bs.THD_R("min")), _np(bs.planes[2, nH + net.n:]))
    for k, p in enumerate(q):
        assert np.array_equal(_np(bs.THD_F(p)), _np(bs.planes[5 + k, nH:nH + net.n]))


def test_masking_by_status(net3, solved):
    """A cap at the median harmonic iteration count leaves many scenarios HPF_ST_MAXITER; a cap of 3
    leaves none converged."""
    sol = net3["sol"]
    cap = int(np.median(_np(solved[0].n_iter_h)))
    r = sol.solve(net3["P"], net3["Q"], net3["I_N"], max_iter_h=cap)
    thd = sol.thd(r.V_m)
    st = _np(r.status)
    assert (st == 1).sum() > 1000 and (st == 0).sum() > 1000
    bs = sol.batch_stats(r.V_m, r.status, quantiles=Q3)
    assert np.array_equal(_np(bs.status_counts), np.bincount(st, minlength=4)[:4])
    _check(bs, r.V_m, thd, r.status, Q3, None)
    # excluded values have no effect: overwrite them with extremes, the bits stay
    Vx = r.V_m.clone()
    bad = torch.as_tensor(st != 0, device=Vx.device)
    Vx[:, :, bad] = torch.tensor(float("nan"), dtype=torch.float64, device=Vx.device)
    Vx[0, :, bad] = -1e300
    bx = sol.batch_stats(Vx, r.status, quantiles=Q3)
    assert np.array_equal(_bits(_np(bx.planes)), _bits(_np(bs.planes)))
    # no converged scenario
    r3 = sol.solve(net3["P"], net3["Q"], net3["I_N"], max_iter_h=3)
    bn = sol.batch_stats(r3.V_m, r3.status, quantiles=Q3, limits={"V_m": 0.0})
    p = _np(bn.planes)
    assert np.array_equal(_np(bn.status_counts), np.bincount(_np(r3.status), minlength=4)[:4])
    assert _np(bn.status_counts)[0] == 0
    assert np.isnan(p[[0, 1, 2, 3, 5, 6, 7]]).all() and (p[4] == 0).all()


def _synthetic(net, B, seed):
    """[H, n, B] with negatives, ties, +-0, a constant row and huge and tiny magnitudes."""
    rng = np.random.default_rng(seed)
    V = rng.normal(0.0, 1.0, (net.H, net.n, B))
    V[1] = np.round(V[1] * 4) / 4                              # heavy ties
    V[2, 0] = 0.0
    V[2, 0, rng.random(B) < 0.5] = -0.0                        # only signed zeros
    V[2, 1, rng.random(B) < 0.3] = 0.0
    V[2, 1, rng.random(B) < 0.3] = -0.0
    V[3, 2] = 0.25                                             # constant
    V[4] *= 1e-200
    V[5] = np.abs(V[5]) * 1e100
    V[6] = -np.abs(V[6])                                       # negative only
    return V


@pytest.mark.parametrize("B", [1, 33, 100003])
@pytest.mark.parametrize("masked", [False, True])
def test_synthetic_values(net3, B, masked):
    from harmonic_power_flow_b200.solver import stats_limit_rows
    sol, net = net3["sol"], net3["net"]
    V = _synthetic(net, B, 7 + B)
    Vd = torch.as_tensor(V, device=sol.device)
    thd = sol.thd(Vd)
    status = None
    if masked:
        rng = np.random.default_rng(B)
        status = torch.as_tensor(rng.choice(4, B, p=[0.7, 0.1, 0.1, 0.1]).astype(np.int32), device=sol.device)
    lim = {"V_m": np.where(np.arange(net.H)[:, None] % 2 == 0, 0.5, np.inf) * np.ones((net.H, net.n)),
           "THD_R": 0.9}
    for q in ((0.0, 0.5, 1.0), Q16):
        bs = sol.batch_stats(Vd, status, quantiles=q, limits=lim)
        _check(bs, Vd, thd, status, q, stats_limit_rows(lim, net.n, net.H))


def test_empty_batch(net3):
    sol, net = net3["sol"], net3["net"]
    bs = sol.batch_stats(torch.empty((net.H, net.n, 0), dtype=torch.float64, device=sol.device), quantiles=Q3)
    p = _np(bs.planes)
    assert np.array_equal(_np(bs.status_counts), [0, 0, 0, 0])
    assert np.isnan(p[[0, 1, 2, 3, 5, 6, 7]]).all() and (p[4] == 0).all()


@pytest.mark.parametrize("env", [{}, {"HPF_HOST_PLAN": "4096"}, {"HPF_HOST_PLAN": "65536"},
                                 {"HPF_HOST_STREAMS": "1"}, {"HPF_HOST_STREAMS": "2"}],
                         ids=["default", "plan4096", "plan65536", "streams1", "streams2"])
def test_host_stats_solve_is_bit_identical(net3, solved, env):
    sol, net = net3["sol"], net3["net"]
    r, _ = solved
    lim = _limits(net, r.V_m)
    ref = sol.batch_stats(r.V_m, r.status, quantiles=Q3, limits=lim)
    with _env(env):
        hs = sol.solve_host_stats(net3["P"], net3["Q"], net3["I_N"], quantiles=Q3, limits=lim, want_flags=True)
    assert np.array_equal(hs.status_counts, _np(ref.status_counts))
    assert np.array_equal(_bits(hs.planes), _bits(_np(ref.planes)))
    for k in ("n_iter_f", "n_iter_h", "status"):
        assert np.array_equal(hs.flags[k], _np(getattr(r, k))), k
    assert np.array_equal(_bits(hs.flags["err_h"]), _bits(_np(r.err_h)))
    # without flags and without limits
    h2 = sol.solve_host_stats(net3["P"], net3["Q"], net3["I_N"], quantiles=Q3)
    ref2 = sol.batch_stats(r.V_m, r.status, quantiles=Q3)
    assert h2.flags is None and np.array_equal(_bits(h2.planes), _bits(_np(ref2.planes)))


@pytest.mark.parametrize("case", ["net1_c_h25", "meshed70-lockstep"])
def test_host_stats_solve_on_other_paths(case, tmp_path):
    from harmonic_power_flow_b200 import BatchSolver, scenarios
    if case == "net1_c_h25":
        net, _, _ = helpers.packed_from_files("net1", 25, True, tmp_path, julia_schema=True)
        env, path, B = {}, 2, 96
    else:
        net, _ = helpers.synthetic_packed("meshed", tmp_path, h_max=25, n=70, load_scale=0.02)
        env, path, B = {"HPF_STRUCT_VARIANT": "3", "HPF_LOCKSTEP": "1"}, 4, 160
    with _env(env):
        sol = BatchSolver(net)
    P, Q, I_N = scenarios.make_batch(net, B, "tight")
    # On these paths a chunk's solve can differ in the last bits from the whole batch's (the kernel of
    # the Norton contraction depends on the batch size), so the reference is the phasor host solve with
    # the same chunk plan, its device copies (hpf_solve_host_keep) reduced by hpf_batch_stats.
    with _env({"HPF_HOST_PLAN": "64"}):                       # several chunks
        r = sol.solve_host(P, Q, I_N, keep=True)["device"]
        assert sol.last_solve_path == path
        hs = sol.solve_host_stats(P, Q, I_N, quantiles=Q3, want_flags=True)
    assert sol.last_solve_path == path
    ref = sol.batch_stats(r.V_m, r.status, quantiles=Q3)
    assert np.array_equal(hs.status_counts, _np(ref.status_counts))
    assert np.array_equal(_bits(hs.planes), _bits(_np(ref.planes)))
    assert np.array_equal(hs.flags["status"], _np(r.status))
    _check(ref, r.V_m, sol.thd(r.V_m), r.status, Q3, None)
    sol.close()


def test_repeatable_ordered_and_capturable(net3, solved):
    sol = net3["sol"]
    r, _ = solved
    a = sol.batch_stats(r.V_m, r.status, quantiles=Q3)
    b = sol.batch_stats(r.V_m, r.status, quantiles=Q3)
    ref = _bits(_np(a.planes))
    assert np.array_equal(_bits(_np(b.planes)), ref)
    # a call on another stream right after a solve on this one is ordered after the solve
    r2 = sol.solve(net3["P"], net3["Q"], net3["I_N"])
    s2 = torch.cuda.Stream()
    with torch.cuda.stream(s2):
        c = sol.batch_stats(r2.V_m, r2.status, quantiles=Q3)
    s2.synchronize()
    assert np.array_equal(_bits(_np(c.planes)), ref)
    # captured into a CUDA graph after one warm-up call, then replayed
    s3 = torch.cuda.Stream()
    with torch.cuda.stream(s3):
        sol.batch_stats(r.V_m, r.status, quantiles=Q3)
    s3.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s3):
        d = sol.batch_stats(r.V_m, r.status, quantiles=Q3)
    d.planes.fill_(0.0)
    g.replay()
    torch.cuda.synchronize()
    assert np.array_equal(_bits(_np(d.planes)), ref)


def test_invalid_arguments(net3, solved):
    from harmonic_power_flow_b200 import _lib
    sol = net3["sol"]
    lib, h = sol.lib, sol._h
    r, _ = solved
    vm, st = C.c_void_p(r.V_m.data_ptr()), C.c_void_p(r.status.data_ptr())
    counts = torch.empty(4, dtype=torch.int32, device=sol.device)
    out = torch.empty((5 + 16) * 60, dtype=torch.float64, device=sol.device)
    pc, po = C.c_void_p(counts.data_ptr()), C.c_void_p(out.data_ptr())
    qs = lambda *v: (C.c_double * max(1, len(v)))(*v)
    E = _lib.HPF_E_INVALID

    def call(B=B_BIG, V=vm, K=1, q=qs(0.5), c=pc, o=po, handle=h):
        return lib.hpf_batch_stats(handle, B, V, st, K, q, None, c, o, None)

    assert call() == _lib.HPF_OK
    torch.cuda.synchronize()
    assert call(B=-1) == E
    assert call(K=-1) == E and call(K=17, q=qs(*([0.5] * 17))) == E
    assert call(q=qs(float("nan"))) == E and call(q=qs(1.5)) == E and call(q=qs(-0.1)) == E
    assert b"quantile" in lib.hpf_last_error(h)
    assert call(c=None) == E and call(o=None) == E and call(K=2, q=None) == E
    assert call(V=None) == E and call(B=0, V=None) == _lib.HPF_OK
    bare = C.c_void_p()
    _lib.check(None, lib.hpf_create(C.byref(bare), sol.device_index))
    try:
        assert call(handle=bare) == E and b"network" in lib.hpf_last_error(bare)
    finally:
        lib.hpf_destroy(bare)
    # the host solve takes the same checks
    P = np.ascontiguousarray(net3["P"][:, :64]); Q = np.ascontiguousarray(net3["Q"][:, :64])
    I = np.ascontiguousarray(net3["I_N"][:, :, :64])
    hc, ho = np.zeros(4, np.int32), np.zeros((6, 60))
    vp = lambda a: C.c_void_p(None if a is None else a.ctypes.data)

    def host(B=64, K=1, q=qs(0.5), c=hc, o=ho):
        return lib.hpf_solve_host_stats(h, B, vp(P), vp(Q), vp(I), 1e-6, 30, 1e-4, 50, K, q, None, vp(c), vp(o),
                                        None, None, None, None)

    assert host() == _lib.HPF_OK
    assert host(B=-1) == E and host(K=17) == E and host(q=qs(2.0)) == E and host(c=None) == E and host(o=None) == E
