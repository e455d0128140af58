"""Exec-oracle: run the UNMODIFIED reference solver in this container.

TEST INFRASTRUCTURE ONLY.  Nothing in the product path imports this file.  It
only works where the reference checkout is mounted (``/root/reference``); it is
used by ``oracle/make_golden.py`` to generate the committed fixtures under
``tests/golden/``; the tests compare against those fixtures.

Nothing is copied: the reference text of
``Harmonic Power Flow/hcne_generalized.py`` (``HG``) is read at run time,
patched IN MEMORY for the library versions of this image and ``exec``-ed:

* ``X.loc[:, "col"] = ...`` -> ``X["col"] = ...`` (HG:57-60,70-73,89-92,105-109;
  pandas 3 refuses to write floats into an int64 column through ``.loc``),
* ``np.Inf`` (HG:389) aliased to ``np.inf`` (removed in numpy 2),
* a stub ``matplotlib.pyplot`` module (HG:30; matplotlib is not installed),
* ``$HOME`` redirected to a scratch directory that holds
  ``Git/harmonic-power-flow/Circuit Simulation/<component>_NE.csv`` (HG:289-291
  hard-codes that path; net2/net3 say ``SMPS`` while the file is ``smps_NE.csv``),
* the module-level configuration (HG:581 ``H_MAX``, HG:596-597 network files,
  HG:602 ``coupled``) replaced textually.

After the module-level run (HG:575-623) the globals dict exposes every function
of the reference, and scenarios are solved by calling the reference's own
``hpf()`` (HG:511-560) with ``buses.P/Q`` and the Norton-equivalent dict swapped.
"""
from __future__ import annotations

import contextlib
import io
import os
import re
import shutil
import sys
import tempfile
import types
import warnings

import numpy as np

REF_ROOT = os.environ.get("HPF_REFERENCE_ROOT", "/root/reference")
HG_PATH = os.path.join(REF_ROOT, "Harmonic Power Flow", "hcne_generalized.py")
NE_DIR = os.path.join(REF_ROOT, "Circuit Simulation")
NET_DIR = os.path.join(REF_ROOT, "Harmonic Power Flow")


def available() -> bool:
    return os.path.isfile(HG_PATH)


def _install_matplotlib_stub():
    if "matplotlib.pyplot" in sys.modules:
        return
    try:
        import matplotlib.pyplot  # noqa: F401
        return
    except Exception:
        pass
    mpl = types.ModuleType("matplotlib")
    plt = types.ModuleType("matplotlib.pyplot")
    plt.plot = lambda *a, **k: None
    plt.bar = lambda *a, **k: None
    plt.show = lambda *a, **k: None
    mpl.pyplot = plt
    sys.modules["matplotlib"] = mpl
    sys.modules["matplotlib.pyplot"] = plt


class RefSession:
    """One exec-ed instance of the reference module for (network, H_MAX, coupled).

    ``buses_csv`` / ``lines_csv`` are paths to files in the HG schema
    (``ID;type;component;S;P;Q;X_sh[;V_nom]`` and ``ID;fromID;toID;R;X;G;B``).
    ``ne_files`` maps component name (as written in the bus file) to an NE CSV.
    """

    def __init__(self, buses_csv, lines_csv, h_max, coupled, ne_files):
        if not available():
            raise RuntimeError("reference checkout not found at " + REF_ROOT)
        _install_matplotlib_stub()
        if not hasattr(np, "Inf"):
            np.Inf = np.inf  # HG:389
        self.coupled = bool(coupled)
        self.scratch = tempfile.mkdtemp(prefix="hpf_ref_")
        home = os.path.join(self.scratch, "home")
        ne_home = os.path.join(home, "Git", "harmonic-power-flow", "Circuit Simulation")
        os.makedirs(ne_home)
        for comp, path in ne_files.items():
            os.symlink(os.path.abspath(path), os.path.join(ne_home, comp + "_NE.csv"))
        cwd = os.path.join(self.scratch, "cwd")
        os.makedirs(cwd)
        shutil.copy(buses_csv, os.path.join(cwd, "case_buses.csv"))
        shutil.copy(lines_csv, os.path.join(cwd, "case_lines.csv"))

        src = open(HG_PATH).read()
        src, nsub = re.subn(r'(\w+)\.loc\[:, "(\w+)"\] = ', r'\1["\2"] = ', src)
        assert nsub >= 17, nsub  # 17 live lines + the commented HG:93
        src, k = re.subn(r"^H_MAX = 51$", "H_MAX = %d" % h_max, src, flags=re.M)
        assert k == 1
        src, k = re.subn(r'init_network\("net2_buses.csv",\s*"net2_lines.csv"\)',
                         'init_network("case_buses.csv", "case_lines.csv")', src)
        assert k == 1
        src, k = re.subn(r"hpf\(buses, lines, coupled=False,",
                         "hpf(buses, lines, coupled=%s," % self.coupled, src)
        assert k == 1

        self._old_home = os.environ.get("HOME")
        self._old_cwd = os.getcwd()
        os.environ["HOME"] = home
        os.chdir(cwd)
        self.g = {"__name__": "hcne_generalized_ref"}
        try:
            with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
                warnings.simplefilter("ignore")
                exec(compile(src, HG_PATH, "exec"), self.g)
        finally:
            os.chdir(self._old_cwd)
        g = self.g
        self.n, self.m, self.c = int(g["n"]), int(g["m"]), int(g["c"])
        self.harmonics = list(g["HARMONICS"])
        self.base_buses = g["buses"].copy()
        self.lines = g["lines"]
        with contextlib.redirect_stdout(io.StringIO()):
            self.base_NE = g["import_Norton_Equivalents"](self.base_buses, self.coupled)
        self._orig_spsolve = g["spsolve"]
        # result of the module-level run itself (the "nominal" solve)
        self.nominal = dict(V=g["V_h"][["V_m", "V_a"]].to_numpy().copy(),
                            err_h=float(g["err_h_final"]), n_iter_h=int(g["n_iter_h"]))

    def close(self):
        if self._old_home is not None:
            os.environ["HOME"] = self._old_home
        shutil.rmtree(self.scratch, ignore_errors=True)

    # -- pieces -------------------------------------------------------------
    def Y_all(self):
        """(H, n, n) complex128 from the reference's build_admittance_matrices (HG:132-171)."""
        g = self.g
        Y = g["build_admittance_matrices"](self.base_buses, self.lines, self.harmonics)
        return Y.to_numpy().reshape(len(self.harmonics), self.n, self.n).copy()

    def ne_arrays(self, NE=None):
        """Per nonlinear bus: I_N (q,H) and Y_N (q,H,H) or (q,H) in p.u."""
        NE = self.base_NE if NE is None else NE
        I, Y = [], []
        for i in range(self.m, self.n):
            I_N, Y_N = NE[self.base_buses.loc[i, "component"]]
            I.append(np.asarray(I_N, dtype=complex).reshape(-1))
            Yn = np.asarray(Y_N, dtype=complex)
            Y.append(Yn if self.coupled else Yn.reshape(-1))
        return np.array(I), np.array(Y)

    def solve(self, P=None, Q=None, I_N_scale=None, dense=False, trace=False,
              thresh_h=1e-4, max_iter_h=50):
        """Run the reference's hpf() (HG:511-560) for one scenario.

        P, Q: p.u. arrays (n) replacing buses.P/Q.  I_N_scale: dict
        component -> complex (H) factor applied to that device's I_N.
        dense=True swaps spsolve for LAPACK (noise-floor variant, SURVEY 7.3).
        """
        g = self.g
        buses = self.base_buses.copy()
        if P is not None:
            buses["P"] = np.asarray(P, dtype=float)
        if Q is not None:
            buses["Q"] = np.asarray(Q, dtype=float)
        NE = {}
        for comp, (I_N, Y_N) in self.base_NE.items():
            I2 = I_N.copy()
            if I_N_scale is not None and comp in I_N_scale:
                I2 = I2 * np.asarray(I_N_scale[comp])
            NE[comp] = [I2, Y_N]
        g["buses"] = buses
        g["import_Norton_Equivalents"] = lambda b, cpl: NE
        if dense:
            def _dense(J, f):
                A = J.toarray()
                b = f.toarray().ravel() if hasattr(f, "toarray") else np.asarray(f).ravel()
                return np.linalg.solve(A, b)
            g["spsolve"] = _dense
        else:
            g["spsolve"] = self._orig_spsolve

        log = dict(err_f=[], err_h=[], f_h=[], J_h=[], x_h=[], V_fund=None)
        orig = {k: g[k] for k in ("fund_mismatch", "harmonic_mismatch",
                                  "build_harmonic_jacobian", "pf",
                                  "update_harmonic_state_vec")}

        def fm(b, V, Y1):
            f, err = orig["fund_mismatch"](b, V, Y1)
            log["err_f"].append(float(err))
            return f, err

        def hm(V, Y, b, ne):
            f, err = orig["harmonic_mismatch"](V, Y, b, ne)
            log["err_h"].append(float(err))
            if trace:
                log["f_h"].append(np.array(f))
            return f, err

        def bj(V, Y, ne, cpl):
            J = orig["build_harmonic_jacobian"](V, Y, ne, cpl)
            if trace:
                log["J_h"].append(J.toarray())
            return J

        def pf(Y, b, *a, **k):
            V, err_t, nf = orig["pf"](Y, b, *a, **k)
            log["V_fund"] = V[["V_m", "V_a"]].to_numpy().copy()
            log["n_iter_f"] = int(nf)
            return V, err_t, nf

        def us(J, x, f):
            xn = orig["update_harmonic_state_vec"](J, x, f)
            if trace:
                log["x_h"].append(np.array(xn))
            return xn

        g["fund_mismatch"], g["harmonic_mismatch"] = fm, hm
        g["build_harmonic_jacobian"], g["pf"] = bj, pf
        g["update_harmonic_state_vec"] = us
        try:
            with warnings.catch_warnings(), contextlib.redirect_stdout(io.StringIO()):
                warnings.simplefilter("ignore")
                V, err_h, n_iter_h, J = g["hpf"](buses, self.lines, self.coupled,
                                                 thresh_h=thresh_h, max_iter_h=max_iter_h)
                thd = g["get_THD"](V).to_numpy().copy()
        finally:
            for k, v in orig.items():
                g[k] = v
            g["spsolve"] = self._orig_spsolve
        H = len(self.harmonics)
        Vn = V[["V_m", "V_a"]].to_numpy().reshape(H, self.n, 2)
        I_N_arr, _ = self.ne_arrays(NE)
        out = dict(V_m=Vn[:, :, 0].copy(), V_a=Vn[:, :, 1].copy(),
                   err_h=float(err_h), n_iter_h=int(n_iter_h),
                   n_iter_f=log["n_iter_f"], err_f_hist=np.array(log["err_f"]),
                   err_h_hist=np.array(log["err_h"]), THD=thd,
                   V_fund=log["V_fund"].reshape(H, self.n, 2), I_N=I_N_arr,
                   J_last=J.toarray())
        if trace:
            out.update(f_h=log["f_h"], J_h=log["J_h"], x_h=log["x_h"])
        return out
