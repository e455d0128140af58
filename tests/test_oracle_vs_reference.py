"""The oracle port (oracle/hpf_oracle.py) against what the REFERENCE ITSELF computed: its own hpf()
(HG:511-560, run through oracle/ref_exec.py) on net3 / coupled / H <= 25, stored by
oracle/make_golden.py in tests/golden/case_net3_c_h25.npz (nominal solve with the trace of the first
iteration) and tests/golden/scen_net3_c_h25_tight.npz (seeded scenarios, SuperLU and LAPACK step).

The comparisons are those of a live run of the reference, at its tolerances: identical iteration
counts, the first iteration's intermediates and the phasors to 1e-12 (nominal) or 1e-10 (scenarios).
CPU only.  oracle/make_golden.py regenerates the stored outputs where a reference checkout exists."""
import os

import numpy as np
import pytest

import hpf_oracle as O
import make_golden as MG
from conftest import GOLDEN


def _phasor(Vm, Va):
    return Vm * np.exp(1j * Va)


def test_port_matches_reference_nominal():
    """hpf() of the reference vs the port on net3 / coupled / H <= 25: identical iteration counts,
    every intermediate of the first iteration and the result to 1e-12."""
    ref = np.load(os.path.join(GOLDEN, "case_net3_c_h25.npz"))
    net = O.net_from_golden(GOLDEN, "net3", 25, True)
    assert np.abs(O.build_admittance_matrices(net) - ref["Y_all"]).max() == 0.0
    o = O.hpf(net, trace=True)
    assert (o["n_iter_f"], o["n_iter_h"]) == (int(ref["n_iter_f"]), int(ref["n_iter_h"])) == (2, 11)
    close = lambda a, b, tol: np.abs(np.asarray(a) - np.asarray(b)).max() <= tol * np.abs(np.asarray(b)).max()
    assert close(o["trace"]["f"][0], ref["f0"], 1e-12)           # (entries cancel to ~1e-10 next to ones of ~300)
    assert close(o["trace"]["J"][0], ref["J0"], 1e-12)
    assert np.allclose(o["err_h_hist"], ref["err_h_hist"], rtol=1e-6)
    V, Vr = _phasor(o["V_m"], o["V_a"]), _phasor(ref["V_m"], ref["V_a"])
    assert (np.abs(V - Vr) / np.abs(Vr)).max() < 1e-12
    assert np.abs(o["THD"] - ref["THD"]).max() < 1e-12
    assert close(o["J_last"], ref["J_last"], 1e-9)               # HG:536-549: the returned J


@pytest.mark.parametrize("dense", [False, True])
def test_port_matches_reference_on_seeded_scenarios(dense):
    """Eight seeded scenarios of BASELINE config 3 (scenarios.draw_scenario = the generator of the
    golden sets and the bench), SuperLU step and LAPACK step: the port follows the reference's own
    round-off path - identical counts, phasors to 1e-10."""
    from harmonic_power_flow_b200 import scenarios
    ref = np.load(os.path.join(GOLDEN, "scen_net3_c_h25_tight.npz"))
    sfx = "_lapack" if dense else ""
    net = O.net_from_golden(GOLDEN, "net3", 25, True)
    Y = O.build_admittance_matrices(net)
    for seed in range(8):
        assert int(ref["seed"][seed]) == seed
        P, Q, I_N = scenarios.draw_scenario(seed, net.P, net.Q, net.I_N, "tight")
        Pm, Qm, _ = MG.draw_scenario(seed, net.P, net.Q, net.n - net.m, net.H, MG.SPREADS["tight"])
        assert np.array_equal(P, Pm) and np.array_equal(Q, Qm)
        assert np.array_equal(P, ref["P"][seed]) and np.array_equal(Q, ref["Q"][seed])
        assert np.abs(ref["I_N"][seed] - I_N).max() < 1e-15
        o = O.hpf(net, P=P, Q=Q, I_N=I_N, Y=Y, solver="lapack" if dense else "superlu")
        # the reference's fundamental iteration count is stored from its SuperLU run only
        assert (o["n_iter_f"], o["n_iter_h"]) == (int(ref["n_iter_f"][seed]), int(ref["n_iter_h" + sfx][seed])), seed
        V, Vr = _phasor(o["V_m"], o["V_a"]), _phasor(ref["V_m" + sfx][seed], ref["V_a" + sfx][seed])
        assert (np.abs(V - Vr) / np.abs(Vr)).max() < 1e-10, seed
