"""ctypes binding of the C ABI (include/hpf_b200.h).  No compute happens in Python.

The library must exist: there is NO fallback implementation.  A missing or
unloadable ``libhpf_b200.so`` raises immediately.
"""
from __future__ import annotations

import ctypes as C
import os

PKG = os.path.dirname(os.path.abspath(__file__))
# $HPF_LIB: load another build of the same ABI (A/B measurements); default = the in-tree library
LIB_PATH = os.environ.get("HPF_LIB") or os.path.join(PKG, "libhpf_b200.so")

HPF_OK, HPF_E_INVALID, HPF_E_CUDA, HPF_E_UNSUPPORTED, HPF_E_NOMEM = 0, -1, -2, -3, -4
ST_CONVERGED, ST_MAXITER, ST_SINGULAR, ST_NONFINITE = 0, 1, 2, 3
SOLVE_RAW = 1
SOLVE_DENSE = 2
ABI_VERSION = 12
HPF_STATS_MAX_Q = 16

_vp, _i, _d, _ll = C.c_void_p, C.c_int, C.c_double, C.c_longlong
_ip, _dp = C.POINTER(C.c_int), C.POINTER(C.c_double)

# name -> (restype, argtypes).  Must list EVERY symbol include/hpf_b200.h declares
# (tests/test_host_cpu.py parses the header and compares).
SIGNATURES = {
    "hpf_abi_version": (_i, []),
    "hpf_create": (_i, [C.POINTER(_vp), _i]),
    "hpf_destroy": (_i, [_vp]),
    "hpf_last_error": (C.c_char_p, [_vp]),
    "hpf_set_network": (_i, [_vp, _i, _i, _i, _i, _ip, _i, _ip, _ip, _dp, _dp, _dp, _dp, _dp]),
    "hpf_set_devices": (_i, [_vp, _i, _i, _dp, _ip]),
    "hpf_set_transformers": (_i, [_vp, _dp, _dp]),
    "hpf_set_y_options": (_i, [_vp, _i]),
    "hpf_build_Y": (_i, [_vp, _vp, _vp]),
    "hpf_set_Y": (_i, [_vp, _dp]),
    "hpf_struct_info": (_i, [_vp, _ip, _ip, _dp, _dp]),
    "hpf_newton_step": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hpf_norton_wn": (_i, [_vp, _i, _vp, _vp, _vp]),
    "hpf_prepare": (_i, [_vp, _i, _vp]),
    "hpf_set_profiling": (_i, [_vp, _i]),
    "hpf_last_kernel_ms": (_i, [_vp, _dp]),
    "hpf_thd": (_i, [_vp, _i, _vp, _vp, _vp]),
    "hpf_bus_currents": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "hpf_batch_stats": (_i, [_vp, _i, _vp, _vp, _i, _dp, _vp, _vp, _vp, _vp]),
    "hpf_solve": (_i, [_vp, _i, _vp, _vp, _vp, _d, _i, _d, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp,
                       _vp, _vp, _vp]),
    "hpf_solve_host": (_i, [_vp, _i, _vp, _vp, _vp, _d, _i, _d, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hpf_solve_host_keep": (_i, [_vp, _i, _vp, _vp, _vp, _d, _i, _d, _i] + [_vp] * 14),
    "hpf_solve_host_stats": (_i, [_vp, _i, _vp, _vp, _vp, _d, _i, _d, _i, _i, _dp, _vp] + [_vp] * 6),
    "hpf_fund_solve": (_i, [_vp, _i, _vp, _vp, _d, _i, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hpf_mismatch": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hpf_jacobian": (_i, [_vp, _i, _vp, _vp, _vp, _vp]),
    "hpf_jacobian_stride": (_ll, [_vp]),
    "hpf_lu_solve": (_i, [_vp, _i, _vp, _vp, _vp, _vp, _vp]),
    "hpf_ne_extract": (_i, [_vp, _i, _i, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp, _vp]),
    "hpf_dim_N": (_i, [_vp]),
    "hpf_dim_Nf": (_i, [_vp]),
    "hpf_launch_count": (_ll, [_vp]),
    "hpf_last_solve_path": (_i, [_vp]),
}

_lib = None


class HpfError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__("hpf_b200 error %d: %s" % (code, msg))
        self.code = code


def load():
    """Load libhpf_b200.so and bind every symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "harmonic_power_flow_b200: CUDA library %s not built. Run "
            "`python -c 'import __graft_entry__ as g; g.build()'` (needs nvcc). "
            "There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)          # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    v = lib.hpf_abi_version()
    if v != ABI_VERSION:
        raise ImportError("libhpf_b200.so has ABI version %d, the Python layer expects %d - rebuild"
                          % (v, ABI_VERSION))
    _lib = lib
    return lib


def check(handle, rc):
    if rc != HPF_OK:
        msg = load().hpf_last_error(handle)
        raise HpfError(rc, (msg or b"").decode("utf-8", "replace"))
