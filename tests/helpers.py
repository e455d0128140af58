"""Shared helpers: build PackedNet / CSV files from the committed golden fixtures."""
import json
import os

import numpy as np
import pandas as pd

from conftest import GOLDEN
from harmonic_power_flow_b200 import netio


def load_case(name):
    return np.load(os.path.join(GOLDEN, "case_%s.npz" % name))


def load_set(name):
    return np.load(os.path.join(GOLDEN, "scen_%s.npz" % name))


def write_net_csvs(net_name, outdir, julia_schema=False):
    """Materialise <net>_buses.csv / <net>_lines.csv in the reference's formats."""
    tab = json.load(open(os.path.join(GOLDEN, "networks.json")))[net_name]
    b, l = pd.DataFrame(tab["buses"]), pd.DataFrame(tab["lines"])
    if julia_schema:          # HPF/net1_*.csv: X_shunt, no G/B
        b = b.rename(columns={"X_sh": "X_shunt"})[["ID", "type", "component", "S", "X_shunt", "P", "Q"]]
        l = l[["ID", "fromID", "toID", "R", "X"]]
    pb = os.path.join(outdir, net_name + "_buses.csv")
    pl = os.path.join(outdir, net_name + "_lines.csv")
    b.to_csv(pb, sep=";", index=False)
    l.to_csv(pl, sep=";", index=False)
    return pb, pl


def write_ne_csvs(outdir):
    """smps_NE.csv / ev_NE.csv in the reference's text format from ne_devices.npz (SI units)."""
    dev = np.load(os.path.join(GOLDEN, "ne_devices.npz"))
    for d in ("smps", "ev"):
        netio.write_ne_csv(os.path.join(outdir, d + "_NE.csv"), dev[d + "__freqs"], dev[d + "__Y_N_c"],
                           dev[d + "__I_N_c"], dev[d + "__Y_N_uc"], dev[d + "__I_N_uc"])
    return outdir


def packed_from_files(net_name, h_max, coupled, tmpdir, julia_schema=False):
    """CSV files -> Settings -> PackedNet through the PRODUCT's own loaders."""
    tmpdir = str(tmpdir)
    pb, pl = write_net_csvs(net_name, tmpdir, julia_schema)
    write_ne_csvs(tmpdir)
    st = netio.Settings(H_MAX=h_max, ne_dir=tmpdir)
    buses, lines, m, n, c = netio.init_network(pb, pl, st)
    NE = netio.import_Norton_Equivalents(buses, coupled, st) if m < n else None
    return netio.pack_network(buses, lines, m, n, c, st.HARMONICS, NE, coupled), st, (buses, lines)


def phasor(Vm, Va):
    return np.asarray(Vm) * np.exp(1j * np.asarray(Va))


def state_vectors(V_m, V_a, c):
    """x = [theta[1:], V_m[c:]] (HG:393-398) from (H, n) arrays."""
    return np.append(V_a.ravel()[1:], V_m.ravel()[c:])


def oracle_net(net):
    """PackedNet (product loaders) -> oracle Net: same per-unit numbers, Y_N expanded per bus."""
    import hpf_oracle as O
    Y_N = None if net.Y_N is None else net.Y_N[net.dev_of_nl_bus]
    return O.Net(n=net.n, m=net.m, c=net.c, harmonics=np.asarray(net.harmonics), line_from=net.from_id,
                 line_to=net.to_id, R=net.R, X=net.X, G=net.G, B=net.B, X_sh=net.X_sh, P=net.P, Q=net.Q,
                 I_N=net.I_N, Y_N=Y_N, coupled=bool(net.coupled))


def textbook_admittance(net):
    """Textbook nodal admittance matrices Y(h) [H, n, n] in incidence form: every branch adds its
    series admittance and both halves of its pi-shunt at the buses it connects, parallel branches
    add up, and the bus shunt 1/(j X_sh h) applies above the fundamental.  This is what
    hpf_set_y_options(FIX_SHUNT_INDEX | SUM_PARALLEL) builds."""
    harmonics, n = np.asarray(net.harmonics), net.n
    want = np.zeros((len(harmonics), n, n), dtype=complex)
    for hi, h in enumerate(harmonics):
        for l in range(len(net.R)):
            f, t = net.from_id[l] - 1, net.to_id[l] - 1
            y = 1 / (net.R[l] + 1j * net.X[l] * h)
            sh = (net.G[l] + 1j * h * net.B[l]) / 2
            want[hi, f, f] += y + sh; want[hi, t, t] += y + sh
            want[hi, f, t] -= y; want[hi, t, f] -= y
        for k in range(n):
            if net.X_sh[k] != 0 and h != 1:
                want[hi, k, k] += 1 / (1j * net.X_sh[k] * h)
    return want


def synthetic_packed(kind, tmpdir, h_max=25, coupled=True, **kw):
    """Synthetic network (config 4 / 5 generators) through the product's own CSV loaders."""
    from harmonic_power_flow_b200 import synthetic
    tmpdir = str(tmpdir)
    write_ne_csvs(tmpdir)
    gen = synthetic.radial_feeder if kind == "radial" else synthetic.meshed
    pb, pl = gen(tmpdir, tmpdir, **kw)
    st = netio.Settings(H_MAX=h_max, ne_dir=tmpdir)
    buses, lines, m, n, c = netio.init_network(pb, pl, st)
    NE = netio.import_Norton_Equivalents(buses, coupled, st)
    return netio.pack_network(buses, lines, m, n, c, st.HARMONICS, NE, coupled), st
