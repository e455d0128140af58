"""Batched solver: Python host over the C ABI.  PyTorch tensors are only the buffer
container (device memory + the current CUDA stream); every computation is a kernel of
libhpf_b200.so.  There is no CPU fallback."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass

import numpy as np
import torch

from . import _lib
from .netio import PackedNet


def _ptr(t):
    return C.c_void_p(0 if t is None else t.data_ptr())


def _np_i(a):
    return a.ctypes.data_as(C.POINTER(C.c_int))


def _np_d(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


@dataclass
class BatchResult:
    """Results of a batch, batch-innermost device tensors exactly as the kernels wrote them."""
    V_m: torch.Tensor          # [H, n, B] f64
    V_a: torch.Tensor          # [H, n, B] f64
    I_inj: torch.Tensor        # [q, H, B] c128 (or None)
    n_iter_f: torch.Tensor     # [B] i32
    n_iter_h: torch.Tensor     # [B] i32
    err_h: torch.Tensor        # [B] f64
    status: torch.Tensor       # [B] i32  (0 converged, 1 max-iter, 2 singular, 3 non-finite)
    err_hist_f: torch.Tensor = None
    err_hist_h: torch.Tensor = None

    @property
    def B(self):
        return self.status.shape[0]

    def converged(self):
        return self.status == _lib.ST_CONVERGED

    def to_pinned(self, cache: dict):
        """Device -> pinned host buffers (kept in ``cache``), one synchronisation."""
        out = {}
        for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status"):
            v = getattr(self, k)
            if v is None:
                out[k] = None
                continue
            buf = cache.get(k)
            if buf is None or buf.shape != v.shape or buf.dtype != v.dtype:
                buf = cache[k] = torch.empty(v.shape, dtype=v.dtype).pin_memory()
            buf.copy_(v, non_blocking=True)
            out[k] = buf
        torch.cuda.current_stream(self.status.device).synchronize()
        return {k: (None if b is None else b.numpy()) for k, b in out.items()}

    def to_host(self):
        out = {}
        for k in ("V_m", "V_a", "I_inj", "n_iter_f", "n_iter_h", "err_h", "status",
                  "err_hist_f", "err_hist_h"):
            v = getattr(self, k)
            out[k] = None if v is None else v.cpu().numpy()
        return out


@dataclass
class BatchStats:
    """Statistics of a batch (hpf_batch_stats / hpf_solve_host_stats) over R = n*H + 2n rows: V_m of
    order harmonics[h] at bus i (row h*n + i), THD_F (row n*H + i), THD_R (row n*H + n + i).
    ``planes`` [5 + K, R]: mean, std (population), min, max, exceed (count above the limit), then one
    nearest-rank quantile per level of ``quantiles``.  Device tensors from ``batch_stats``, numpy
    arrays from ``solve_host_stats`` (which also puts the optional flag arrays in ``flags``)."""
    status_counts: object      # [4] int32: scenarios per HPF_ST_* value
    quantiles: tuple
    planes: object             # [5 + K, R] f64
    n: int
    H: int
    flags: dict = None

    STATS = ("mean", "std", "min", "max", "exceed")

    def plane(self, stat):
        """[R] row of a statistic: one of STATS or a quantile level given to the call."""
        if isinstance(stat, str):
            return self.planes[self.STATS.index(stat)]
        return self.planes[5 + [float(p) for p in self.quantiles].index(float(stat))]

    def V_m(self, stat):
        """[H, n] for V_m."""
        return self.plane(stat)[:self.n * self.H].reshape(self.H, self.n)

    def THD_F(self, stat):
        """[n] for THD_F."""
        return self.plane(stat)[self.n * self.H:self.n * self.H + self.n]

    def THD_R(self, stat):
        """[n] for THD_R."""
        return self.plane(stat)[self.n * self.H + self.n:]


def stats_limit_rows(limits, n, H):
    """{"V_m": [H, n] or broadcastable, "THD_F" / "THD_R": [n] or scalar} -> [R] float64 rows (a missing
    key = +inf: never exceeded), or None for no limits."""
    if limits is None:
        return None
    unknown = set(limits) - {"V_m", "THD_F", "THD_R"}
    if unknown:
        raise ValueError("unknown limit keys %s" % sorted(unknown))
    inf = np.inf
    vm = np.broadcast_to(np.asarray(limits.get("V_m", inf), np.float64), (H, n))
    tf = np.broadcast_to(np.asarray(limits.get("THD_F", inf), np.float64), (n,))
    tr = np.broadcast_to(np.asarray(limits.get("THD_R", inf), np.float64), (n,))
    return np.ascontiguousarray(np.concatenate([vm.ravel(), tf, tr]))


def result_slab_layout(H, n, q, B):
    """Byte offsets of the result fields in ONE contiguous slab (multi-GPU runs gather and copy
    the slab with one collective / one D2H instead of seven): -> (dict name -> (offset, shape,
    dtype), total bytes).  Every field starts on a 256-byte boundary."""
    fields = [("V_m", (H, n, B), torch.float64), ("V_a", (H, n, B), torch.float64),
              ("I_inj", (q, H, B), torch.complex128), ("err_h", (B,), torch.float64),
              ("n_iter_f", (B,), torch.int32), ("n_iter_h", (B,), torch.int32), ("status", (B,), torch.int32)]
    lay, off = {}, 0
    for name, shape, dt in fields:
        nbytes = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
        lay[name] = (off, shape, dt)
        off = (off + nbytes + 255) // 256 * 256
    return lay, off


def result_from_slab(slab, H, n, q, B):
    """BatchResult (or dict of numpy views for a CPU slab) whose fields are VIEWS into `slab`
    (1-D uint8 tensor of result_slab_layout(...)[1] bytes)."""
    lay, total = result_slab_layout(H, n, q, B)
    assert slab.dtype == torch.uint8 and slab.numel() >= total
    views = {}
    for name, (off, shape, dt) in lay.items():
        nbytes = int(np.prod(shape)) * torch.empty((), dtype=dt).element_size()
        views[name] = slab[off:off + nbytes].view(dt).view(shape) if nbytes else None
    return BatchResult(**views)


class BatchSolver:
    """One handle = one GPU.  ``net`` is a PackedNet (netio.pack_network)."""

    def __init__(self, net: PackedNet, device: int | None = None):
        self.lib = _lib.load()
        if not torch.cuda.is_available():
            raise RuntimeError("harmonic_power_flow_b200 needs a CUDA device (B200); no CPU fallback")
        self.device_index = torch.cuda.current_device() if device is None else int(device)
        self.device = torch.device("cuda", self.device_index)
        self.net = net
        self._h = C.c_void_p()
        _lib.check(None, self.lib.hpf_create(C.byref(self._h), self.device_index))
        n = net
        _lib.check(self._h, self.lib.hpf_set_network(
            self._h, n.n, n.m, n.c, n.H, _np_i(n.harmonics), len(n.R), _np_i(n.from_id), _np_i(n.to_id),
            _np_d(n.R), _np_d(n.X), _np_d(n.G), _np_d(n.B), _np_d(n.X_sh)))
        if n.q > 0:
            if n.Y_N is None:
                raise ValueError("network has nonlinear buses but no Norton equivalents attached")
            yn = np.ascontiguousarray(n.Y_N).view(np.float64)
            _lib.check(self._h, self.lib.hpf_set_devices(self._h, len(n.devices), int(n.coupled),
                                                         _np_d(yn), _np_i(n.dev_of_nl_bus)))
        else:
            _lib.check(self._h, self.lib.hpf_set_devices(self._h, 0, int(n.coupled), None, None))
        self.Y = self.build_Y()

    # -- plumbing ----------------------------------------------------------------------
    def _stream(self):
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.lib.hpf_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _f64(self, *shape):
        return torch.empty(shape, dtype=torch.float64, device=self.device)

    def _i32(self, *shape):
        return torch.empty(shape, dtype=torch.int32, device=self.device)

    def _c128(self, *shape):
        return torch.empty(shape, dtype=torch.complex128, device=self.device)

    def _dev(self, a, dtype):
        if isinstance(a, torch.Tensor):
            t = a.to(device=self.device, dtype=dtype)
        else:
            t = torch.as_tensor(np.array(a, copy=True, order="C"), dtype=dtype).to(self.device)
        return t.contiguous()

    @property
    def N(self):
        return self.lib.hpf_dim_N(self._h)

    @property
    def launch_count(self):
        return int(self.lib.hpf_launch_count(self._h))

    PATHS = {0: "none", 1: "lane-per-scenario / one-warp-per-harmonic kernels", 2: "one CTA per scenario (shared memory)",
             3: "one CTA per scenario (global-memory state)", 4: "lock-step batched rounds", 5: "dense Jacobian + LU"}

    @property
    def last_solve_path(self):
        """Which kernels the last solve ran for the harmonic stage (hpf_last_solve_path)."""
        return int(self.lib.hpf_last_solve_path(self._h))

    # -- kernel 1 ----------------------------------------------------------------------
    def build_Y(self):
        """Y(h) [H, n, n] complex128 on the device (HG:132-171)."""
        n = self.net
        Y = self._c128(n.H, n.n, n.n)
        _lib.check(self._h, self.lib.hpf_build_Y(self._h, _ptr(Y), self._stream()))
        return Y

    def bus_currents(self, V_m, V_a):
        """Per-bus current spectra I = Y(h) V, complex [H, n, B] (hpf_bus_currents)."""
        V_m, V_a = self._dev(V_m, torch.float64), self._dev(V_a, torch.float64)
        B = V_m.shape[2]
        out = self._c128(self.net.H, self.net.n, B)
        _lib.check(self._h, self.lib.hpf_bus_currents(self._h, B, _ptr(V_m), _ptr(V_a), _ptr(out), self._stream()))
        return out

    def set_transformers(self, tau=None, phase_shift_deg=None):
        """Transformer taps / phase shifts per line (FPF/pi_trafo_pf_test.py:117-145) and rebuild
        Y(h); ``None`` restores plain lines."""
        if tau is None:
            _lib.check(self._h, self.lib.hpf_set_transformers(self._h, None, None))
        else:
            t = np.ascontiguousarray(tau, dtype=np.float64)
            p = np.ascontiguousarray(phase_shift_deg, dtype=np.float64)
            if t.shape != (len(self.net.R),) or p.shape != t.shape:
                raise ValueError("tau and phase_shift_deg must have one entry per line")
            _lib.check(self._h, self.lib.hpf_set_transformers(self._h, _np_d(t), _np_d(p)))
        self.Y = self.build_Y()
        return self.Y

    def set_y_options(self, fix_shunt_index=False, sum_parallel=False):
        """Opt-in corrections of the reference's Y(h) quirks (hpf_set_y_options); rebuilds Y(h)."""
        flags = (1 if fix_shunt_index else 0) | (2 if sum_parallel else 0)
        _lib.check(self._h, self.lib.hpf_set_y_options(self._h, flags))
        self.Y = self.build_Y()
        return self.Y

    def set_Y(self, Y):
        """Replace Y(h) by a caller-supplied [H, n, n] complex table (pf(Y, buses), HG:244)."""
        Y = np.ascontiguousarray(Y, dtype=np.complex128)
        n = self.net
        if Y.shape != (n.H, n.n, n.n):
            raise ValueError("Y must be [H, n, n]")
        _lib.check(self._h, self.lib.hpf_set_Y(self._h, _np_d(Y.view(np.float64))))
        self.Y = torch.as_tensor(Y).to(self.device)

    def thd(self, V_m):
        """THD_F, THD_R [2, n, B] from magnitudes [H, n, B] (HG:563-572)."""
        V_m = self._dev(V_m, torch.float64)
        B = V_m.shape[2]
        out = self._f64(2, self.net.n, B)
        _lib.check(self._h, self.lib.hpf_thd(self._h, B, _ptr(V_m), _ptr(out), self._stream()))
        return out

    def _quantile_levels(self, quantiles):
        q = np.ascontiguousarray(np.asarray(quantiles, dtype=np.float64).ravel())
        if q.size > _lib.HPF_STATS_MAX_Q:
            raise ValueError("at most %d quantile levels" % _lib.HPF_STATS_MAX_Q)
        return q

    def batch_stats(self, V_m, status=None, quantiles=(0.5, 0.95), limits=None) -> BatchStats:
        """Statistics of V_m [H, n, B] and its THD over the converged scenarios (all of them when
        ``status`` is None), on the device (hpf_batch_stats).  ``limits``: see stats_limit_rows."""
        n = self.net
        V_m = self._dev(V_m, torch.float64)
        if tuple(V_m.shape[:2]) != (n.H, n.n) or V_m.dim() != 3:
            raise ValueError("V_m must be [H, n, B]")
        B = V_m.shape[2]
        if status is not None:
            status = self._dev(status, torch.int32)
            if tuple(status.shape) != (B,):
                raise ValueError("status must be [B]")
        q = self._quantile_levels(quantiles)
        lim = stats_limit_rows(limits, n.n, n.H)
        lim = None if lim is None else self._dev(lim, torch.float64)
        R = n.n * n.H + 2 * n.n
        counts, planes = self._i32(4), self._f64(5 + q.size, R)
        _lib.check(self._h, self.lib.hpf_batch_stats(self._h, B, _ptr(V_m), _ptr(status), int(q.size), _np_d(q),
                                                     _ptr(lim), _ptr(counts), _ptr(planes), self._stream()))
        return BatchStats(counts, tuple(float(p) for p in q), planes, n.n, n.H)

    def solve_host_stats(self, P, Q, I_N, thresh_f=1e-6, max_iter_f=30, thresh_h=1e-4, max_iter_h=50,
                         quantiles=(0.5, 0.95), limits=None, want_flags=False) -> BatchStats:
        """hpf_solve_host_stats: numpy in, statistics out (numpy); only the inputs and a few KB of
        statistics cross the host link.  ``want_flags=True`` also returns the per-scenario n_iter_f,
        n_iter_h, err_h and status in ``flags``."""
        n = self.net
        P = np.ascontiguousarray(P, dtype=np.float64)
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        B = P.shape[1]
        I_N = np.ascontiguousarray(I_N, dtype=np.complex128) if n.q > 0 else np.zeros(0, np.complex128)
        q = self._quantile_levels(quantiles)
        lim = stats_limit_rows(limits, n.n, n.H)
        R = n.n * n.H + 2 * n.n
        counts, planes = np.empty(4, np.int32), np.empty((5 + q.size, R), np.float64)
        flags = dict(n_iter_f=np.empty(B, np.int32), n_iter_h=np.empty(B, np.int32), err_h=np.empty(B, np.float64),
                     status=np.empty(B, np.int32)) if want_flags else None
        vp = lambda a: C.c_void_p(None if a is None else a.ctypes.data)
        f = flags or {}
        _lib.check(self._h, self.lib.hpf_solve_host_stats(
            self._h, B, vp(P), vp(Q), vp(I_N), thresh_f, max_iter_f, thresh_h, max_iter_h,
            int(q.size), _np_d(q), vp(lim), vp(counts), vp(planes),
            vp(f.get("n_iter_f")), vp(f.get("n_iter_h")), vp(f.get("err_h")), vp(f.get("status"))))
        return BatchStats(counts, tuple(float(p) for p in q), planes, n.n, n.H, flags)

    # -- inputs ------------------------------------------------------------------------
    def prepare(self, P, Q, I_N=None):
        """Move scenario inputs to the device in batch-innermost layout.
        P, Q: [n, B]; I_N: [q, H, B] complex."""
        P = self._dev(P, torch.float64)
        Q = self._dev(Q, torch.float64)
        n = self.net
        if P.shape[0] != n.n or P.shape != Q.shape:
            raise ValueError("P, Q must be [n, B]")
        B = P.shape[1]
        if n.q > 0:
            I_N = self._dev(I_N, torch.complex128)
            if tuple(I_N.shape) != (n.q, n.H, B):
                raise ValueError("I_N must be [q, H, B]")
        else:
            I_N = None
        return P, Q, I_N

    # -- fused solve -------------------------------------------------------------------
    def solve(self, P, Q, I_N=None, thresh_f=1e-6, max_iter_f=30, thresh_h=1e-4, max_iter_h=50,
              raw=False, want_I_inj=True, history=False, dense=False,
              out: BatchResult | None = None) -> BatchResult:
        """Fundamental + harmonic Newton-Raphson for the whole batch (hpf_solve).
        dense=True forces the dense-LU Newton step; the default picks the structured step when
        the network admits it (``struct_info()``).  history=True also returns the mismatch norm
        before every step and after the last one (err_hist_f / err_hist_h, unused tail NaN)."""
        P, Q, I_N = self.prepare(P, Q, I_N)
        n = self.net
        B = P.shape[1]
        if out is None:
            out = BatchResult(
                V_m=self._f64(n.H, n.n, B), V_a=self._f64(n.H, n.n, B),
                I_inj=self._c128(n.q, n.H, B) if (want_I_inj and n.q > 0) else None,
                n_iter_f=self._i32(B), n_iter_h=self._i32(B), err_h=self._f64(B), status=self._i32(B),
                err_hist_f=self._f64(max_iter_f + 1, B) if history else None,
                err_hist_h=self._f64(max_iter_h + 1, B) if history else None)
        _lib.check(self._h, self.lib.hpf_solve(
            self._h, B, _ptr(P), _ptr(Q), _ptr(I_N), thresh_f, max_iter_f, thresh_h, max_iter_h,
            (_lib.SOLVE_RAW if raw else 0) | (_lib.SOLVE_DENSE if dense else 0), _ptr(out.V_m), _ptr(out.V_a), _ptr(out.I_inj),
            _ptr(out.n_iter_f), _ptr(out.n_iter_h), _ptr(out.err_h), _ptr(out.status),
            _ptr(out.err_hist_f), _ptr(out.err_hist_h), self._stream()))
        return out

    def alloc_result_slab(self, B):
        """-> (BatchResult whose fields are views into one contiguous device slab, the slab)."""
        n = self.net
        _, total = result_slab_layout(n.H, n.n, n.q, B)
        slab = torch.empty(total, dtype=torch.uint8, device=self.device)
        return result_from_slab(slab, n.H, n.n, n.q, B), slab

    def solve_host(self, P, Q, I_N, thresh_f=1e-6, max_iter_f=30, thresh_h=1e-4, max_iter_h=50, keep=None,
                   want_I_inj=True):
        """hpf_solve_host: numpy in, numpy out, all copies inside the C call.  ``keep``: a
        BatchResult of device tensors that additionally receives the results (hpf_solve_host_keep),
        e.g. for the NCCL gather of a multi-GPU run; ``keep=True`` allocates one (returned under
        the key "device").  ``want_I_inj=False``: the Norton injection currents (which the reference's
        hpf() does not return either, HG:560) are not copied back (I_inj = NULL in the C call)."""
        n = self.net
        P = np.ascontiguousarray(P, dtype=np.float64)
        Q = np.ascontiguousarray(Q, dtype=np.float64)
        B = P.shape[1]
        I_N = np.ascontiguousarray(I_N, dtype=np.complex128) if n.q > 0 else np.zeros(0, np.complex128)
        key = (B,)
        if getattr(self, "_host_out_key", None) != key:      # pinned result buffers, reused
            pin = lambda shape, dt: torch.empty(shape, dtype=dt).pin_memory().numpy()
            self._host_out = (pin((n.H, n.n, B), torch.float64), pin((n.H, n.n, B), torch.float64),
                              pin((n.q, n.H, B), torch.complex128), pin((B,), torch.int32),
                              pin((B,), torch.int32), pin((B,), torch.int32), pin((B,), torch.float64))
            self._host_out_key = key
        V_m, V_a, I_inj, nf, nh, st, err = self._host_out
        vp = lambda a: C.c_void_p(a.ctypes.data)
        if keep is None:
            _lib.check(self._h, self.lib.hpf_solve_host(
                self._h, B, vp(P), vp(Q), vp(I_N), thresh_f, max_iter_f, thresh_h, max_iter_h,
                vp(V_m), vp(V_a), vp(I_inj) if want_I_inj else None, vp(nf), vp(nh), vp(err), vp(st)))
            return dict(V_m=V_m, V_a=V_a, I_inj=I_inj if want_I_inj else None, n_iter_f=nf, n_iter_h=nh, err_h=err, status=st)
        if keep is True:
            keep = BatchResult(self._f64(n.H, n.n, B), self._f64(n.H, n.n, B), self._c128(n.q, n.H, B),
                               self._i32(B), self._i32(B), self._f64(B), self._i32(B))
        _lib.check(self._h, self.lib.hpf_solve_host_keep(
            self._h, B, vp(P), vp(Q), vp(I_N), thresh_f, max_iter_f, thresh_h, max_iter_h,
            vp(V_m), vp(V_a), vp(I_inj), vp(nf), vp(nh), vp(err), vp(st),
            _ptr(keep.V_m), _ptr(keep.V_a), _ptr(keep.I_inj), _ptr(keep.n_iter_f), _ptr(keep.n_iter_h),
            _ptr(keep.err_h), _ptr(keep.status)))
        return dict(V_m=V_m, V_a=V_a, I_inj=I_inj, n_iter_f=nf, n_iter_h=nh, err_h=err, status=st, device=keep)

    def fund_solve(self, P, Q, thresh_f=1e-6, max_iter_f=30, history=False):
        P, Q, _ = self.prepare(P, Q, None) if self.net.q == 0 else (self._dev(P, torch.float64),
                                                                    self._dev(Q, torch.float64), None)
        n = self.net
        B = P.shape[1]
        V_m, V_a = self._f64(n.H, n.n, B), self._f64(n.H, n.n, B)
        nf, err = self._i32(B), self._f64(B)
        hist = self._f64(max_iter_f + 1, B) if history else None
        _lib.check(self._h, self.lib.hpf_fund_solve(self._h, B, _ptr(P), _ptr(Q), thresh_f, max_iter_f,
                                                    _ptr(V_m), _ptr(V_a), _ptr(nf), _ptr(err), _ptr(hist),
                                                    self._stream()))
        return V_m, V_a, nf, err, hist

    def set_profiling(self, enabled=True):
        _lib.check(self._h, self.lib.hpf_set_profiling(self._h, int(enabled)))

    def last_kernel_ms(self):
        """(fundamental-stage kernel ms, harmonic / fused kernel ms) of the last solve."""
        ms = (C.c_double * 2)()
        _lib.check(self._h, self.lib.hpf_last_kernel_ms(self._h, ms))
        return float(ms[0]), float(ms[1])

    def struct_info(self):
        """-> dict(available: 0 no / 1 tile kernels / 2 per-CTA kernel, nZ, pivot_min, pivot_max)."""
        av, nz = C.c_int(), C.c_int()
        pmin, pmax = C.c_double(), C.c_double()
        _lib.check(self._h, self.lib.hpf_struct_info(self._h, C.byref(av), C.byref(nz), C.byref(pmin),
                                                     C.byref(pmax)))
        return dict(available=int(av.value), nZ=nz.value, pivot_min=pmin.value, pivot_max=pmax.value)

    def newton_step(self, V_m, V_a, P, Q, I_N=None):
        """One structured Newton step: dx [N, B] with x_new = x - dx (hpf_newton_step)."""
        V_m, V_a = self._dev(V_m, torch.float64), self._dev(V_a, torch.float64)
        P, Q, I_N = self.prepare(P, Q, I_N)
        B = P.shape[1]
        dx = self._f64(self.N, B)
        _lib.check(self._h, self.lib.hpf_newton_step(self._h, B, _ptr(V_m), _ptr(V_a), _ptr(P), _ptr(Q),
                                                     _ptr(I_N), _ptr(dx), self._stream()))
        return dx

    def prepare_batch(self, B_max):
        """hpf_prepare: all lazy set-up and scratch allocation for batches of up to B_max scenarios now."""
        _lib.check(self._h, self.lib.hpf_prepare(self._h, int(B_max), self._stream()))

    def norton_wn(self, I_N):
        """w_N = A_ZZ^-1 I_N,Z = W_NL I_N for the batch, complex [nZ, B] (hpf_norton_wn): the Norton
        contraction of the structured step as one complex GEMM."""
        I_N = self._dev(I_N, torch.complex128)
        B = I_N.shape[2]
        out = self._c128(self.struct_info()["nZ"], B)
        _lib.check(self._h, self.lib.hpf_norton_wn(self._h, B, _ptr(I_N), _ptr(out), self._stream()))
        return out

    # -- standalone kernels --------------------------------------------------------------
    def mismatch(self, V_m, V_a, P, Q, I_N=None, want_I_inj=False, out=None):
        n = self.net
        V_m, V_a = self._dev(V_m, torch.float64), self._dev(V_a, torch.float64)
        P, Q, I_N = self.prepare(P, Q, I_N)
        B = P.shape[1]
        f, err = out if out is not None else (self._f64(self.N, B), self._f64(B))
        I_inj = self._c128(n.q, n.H, B) if want_I_inj else None
        _lib.check(self._h, self.lib.hpf_mismatch(self._h, B, _ptr(V_m), _ptr(V_a), _ptr(P), _ptr(Q),
                                                  _ptr(I_N), _ptr(f), _ptr(err), _ptr(I_inj), self._stream()))
        return (f, err, I_inj) if want_I_inj else (f, err)

    def jacobian_stride(self):
        return int(self.lib.hpf_jacobian_stride(self._h))

    def jacobian(self, V_m, V_a, out=None):
        """-> J [B, stride]; use ``jacobian_view`` for the [B, N, N] row-major matrices."""
        V_m, V_a = self._dev(V_m, torch.float64), self._dev(V_a, torch.float64)
        B = V_m.shape[2]
        J = self._f64(B, self.jacobian_stride()) if out is None else out
        _lib.check(self._h, self.lib.hpf_jacobian(self._h, B, _ptr(V_m), _ptr(V_a), _ptr(J), self._stream()))
        return J

    def jacobian_view(self, J):
        N = self.N
        return J[:, :N * N].view(J.shape[0], N, N)

    def lu_solve(self, J, f):
        f = self._dev(f, torch.float64)
        B = f.shape[1]
        dx, info = self._f64(self.N, B), self._i32(B)
        _lib.check(self._h, self.lib.hpf_lu_solve(self._h, B, _ptr(J), _ptr(f), _ptr(dx), _ptr(info),
                                                  self._stream()))
        return dx, info


def ne_extract(Vf, Vh, I_f, I_h, device=0):
    """Norton-equivalent extraction for a batch of devices (hpf_ne_extract): Vf [D,2], Vh [D,2,K],
    I_f [D,2,N], I_h [D,2,K,N] complex -> dict of device tensors Y_N_c [D,N,N], I_N_c, Y_N_uc,
    I_N_uc [D,N] (complex128) and info [D] (int32)."""
    lib = _lib.load()
    if not torch.cuda.is_available():
        raise RuntimeError("harmonic_power_flow_b200 needs a CUDA device (B200); no CPU fallback")
    dev = torch.device("cuda", int(device))
    c = lambda a: torch.as_tensor(np.ascontiguousarray(a, dtype=np.complex128)).to(dev).contiguous() \
        if not isinstance(a, torch.Tensor) else a.to(dev, torch.complex128).contiguous()
    Vf, Vh, I_f, I_h = c(Vf), c(Vh), c(I_f), c(I_h)
    D, K = Vh.shape[0], Vh.shape[2]
    N = K + 1
    if Vf.shape != (D, 2) or Vh.shape != (D, 2, K) or I_f.shape != (D, 2, N) or I_h.shape != (D, 2, K, N):
        raise ValueError("ne_extract: inconsistent shapes")
    out = {"Y_N_c": torch.empty((D, N, N), dtype=torch.complex128, device=dev),
           "I_N_c": torch.empty((D, N), dtype=torch.complex128, device=dev),
           "Y_N_uc": torch.empty((D, N), dtype=torch.complex128, device=dev),
           "I_N_uc": torch.empty((D, N), dtype=torch.complex128, device=dev),
           "info": torch.empty(D, dtype=torch.int32, device=dev)}
    h = C.c_void_p()
    _lib.check(None, lib.hpf_create(C.byref(h), dev.index))
    try:
        _lib.check(h, lib.hpf_ne_extract(h, D, N, _ptr(Vf), _ptr(Vh), _ptr(I_f), _ptr(I_h), _ptr(out["Y_N_c"]),
                                         _ptr(out["I_N_c"]), _ptr(out["Y_N_uc"]), _ptr(out["I_N_uc"]),
                                         _ptr(out["info"]),
                                         C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)))
        torch.cuda.current_stream(dev).synchronize()
    finally:
        lib.hpf_destroy(h)
    return out
