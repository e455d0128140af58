"""harmonic_power_flow_b200 - B200-native batched harmonic power flow (solve path only).

Host side = thin Python over the C ABI of ``libhpf_b200.so`` (include/hpf_b200.h);
all arithmetic runs in hand-written sm_100a CUDA kernels.  No CPU fallback.

    from harmonic_power_flow_b200 import hcne_generalized as hg   # reference-shaped API
    from harmonic_power_flow_b200 import BatchSolver, netio       # batched API
    from harmonic_power_flow_b200 import ne_from_sim              # Norton-equivalent extraction
"""
from . import netio  # noqa: F401
from .netio import Settings, PackedNet, pack_network  # noqa: F401

__all__ = ["netio", "Settings", "PackedNet", "pack_network", "BatchSolver", "BatchResult", "BatchStats",
           "hcne_generalized", "ne_from_sim", "scenarios", "synthetic", "dist"]


def __getattr__(name):
    # torch-dependent modules are imported lazily so that the data-contract layer
    # (netio) stays importable in tools that only read/write the CSV formats
    import importlib
    if name in ("BatchSolver", "BatchResult", "BatchStats"):
        return getattr(importlib.import_module(".solver", __name__), name)
    if name in ("hcne_generalized", "ne_from_sim", "scenarios", "synthetic", "dist", "solver", "_lib", "build"):
        return importlib.import_module("." + name, __name__)
    raise AttributeError(name)
