"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  Not imported by the product package.

NumPy/SciPy restatement of the AC power flow that the reference reaches through
``pp.runpp(net, enforce_q_lims=True)`` (reference ``opfgym/opf_env.py:696-709``).
The arithmetic lives in the third-party dependency **pandapower >=2.13.1,<3.0**
(``/root/reference/pyproject.toml:32``; no lock file, so the exact version is
unpinned), which is absent from ``/root/reference`` and not installable here.
This file restates its published PYPOWER-derived algorithm (SURVEY.md App. B.4,
B.5): ``makeYbus``, ``makeSbus``, ``makeBdc``/``dcpf`` (angle initialisation),
``newtonpf`` with ``dSbus_dV``, the q-limit outer loop, ``pfsoln`` and the
result-table formulas.

PARITY STATUS: **unpinned at the pandapower boundary** -- the reference's own
tests hold no power-flow number (SURVEY.md §8c).  What *is* pinned
(tests/test_oracle_pf.py, tests/test_ieee14.py): the WSCC 9-bus textbook solution
(App. C.4), the published IEEE 14-bus solution (off-nominal taps, bus shunt, five
PV buses; voltages, angles, generator P/Q and losses to the printed precision), the
2-bus closed form (App. C.5), and the invariants of App. C.6.

Only ``tests/``, ``__graft_entry__.smoke()`` and ``bench.py``'s CPU-baseline /
``--impl reference`` legs may import this module.
"""
from __future__ import annotations

import numpy as np
import scipy.sparse as sp
from scipy.sparse.linalg import spsolve

from oracle.ppc_ref import (BASE_KV, BR_B, BR_G, BR_R, BR_STATUS, BR_X, BS, BUS_TYPE,
                            F_BUS, GEN_BUS, GEN_STATUS, GS, PD, PG, PQ, PV, QD, QG,
                            QMAX, QMIN, REF, SHIFT, T_BUS, TAP, VA, VG, VM, RefBuilder)

Ppc = object     # any namespace with base_mva / bus / gen / branch / rate_f / rate_t and the lookups


# ------------------------------------------------------------------ admittances
def branch_admittances(branch):
    """pypower ``makeYbus.py`` branch part: returns (Yff, Yft, Ytf, Ytt)."""
    stat = branch[:, BR_STATUS]
    ys = stat / (branch[:, BR_R] + 1j * branch[:, BR_X])
    ysh = stat * (branch[:, BR_G] + 1j * branch[:, BR_B])
    ratio = np.where(branch[:, TAP] == 0, 1.0, branch[:, TAP])
    tap = ratio * np.exp(1j * np.pi / 180.0 * branch[:, SHIFT])
    ytt = ys + ysh / 2.0
    yff = ytt / (tap * np.conj(tap))
    yft = -ys / np.conj(tap)
    ytf = -ys / tap
    return yff, yft, ytf, ytt


def make_ybus(base_mva, bus, branch):
    nb, nl = bus.shape[0], branch.shape[0]
    yff, yft, ytf, ytt = branch_admittances(branch)
    f = branch[:, F_BUS].astype(int)
    t = branch[:, T_BUS].astype(int)
    ysh = (bus[:, GS] + 1j * bus[:, BS]) / base_mva
    il = np.arange(nl)
    yf = sp.csr_matrix((np.r_[yff, yft], (np.r_[il, il], np.r_[f, t])), (nl, nb))
    yt = sp.csr_matrix((np.r_[ytf, ytt], (np.r_[il, il], np.r_[f, t])), (nl, nb))
    cf = sp.csr_matrix((np.ones(nl), (il, f)), (nl, nb))
    ct = sp.csr_matrix((np.ones(nl), (il, t)), (nl, nb))
    ybus = cf.T @ yf + ct.T @ yt + sp.diags(ysh)
    return ybus.tocsr(), yf, yt


def make_sbus(base_mva, bus, gen):
    nb = bus.shape[0]
    on = gen[:, GEN_STATUS] > 0
    gbus = gen[on, GEN_BUS].astype(int)
    sg = np.zeros(nb, dtype=complex)
    np.add.at(sg, gbus, (gen[on, PG] + 1j * gen[on, QG]))
    return (sg - (bus[:, PD] + 1j * bus[:, QD])) / base_mva


def bus_types(bus, gen):
    ref = np.nonzero(bus[:, BUS_TYPE] == REF)[0]
    pv = np.nonzero(bus[:, BUS_TYPE] == PV)[0]
    pq = np.nonzero(bus[:, BUS_TYPE] == PQ)[0]
    return ref, pv, pq


# ------------------------------------------------------------------------ DC init
def make_bdc(bus, branch):
    nb, nl = bus.shape[0], branch.shape[0]
    stat = branch[:, BR_STATUS]
    b = stat / branch[:, BR_X]
    ratio = np.where(branch[:, TAP] == 0, 1.0, branch[:, TAP])
    b = b / ratio
    f = branch[:, F_BUS].astype(int)
    t = branch[:, T_BUS].astype(int)
    il = np.arange(nl)
    cft = sp.csr_matrix((np.r_[np.ones(nl), -np.ones(nl)], (np.r_[il, il], np.r_[f, t])), (nl, nb))
    bf = sp.csr_matrix((np.r_[b, -b], (np.r_[il, il], np.r_[f, t])), (nl, nb))
    bbus = cft.T @ bf
    pfinj = b * (-branch[:, SHIFT] * np.pi / 180.0)
    pbusinj = cft.T @ pfinj
    return bbus.tocsr(), pbusinj


def dc_angles(base_mva, bus, gen, branch):
    """pandapower ``_run_dc_pf`` + pypower ``dcpf``: angles [rad] for init='dc'."""
    ref, pv, pq = bus_types(bus, gen)
    bbus, pbusinj = make_bdc(bus, branch)
    pbus = make_sbus(base_mva, bus, gen).real - pbusinj - bus[:, GS] / base_mva
    va = bus[:, VA] * np.pi / 180.0
    pvpq = np.r_[pv, pq]
    if len(pvpq):
        rhs = pbus[pvpq] - bbus[pvpq][:, ref] @ va[ref]
        va = va.copy()
        va[pvpq] = spsolve(bbus[pvpq][:, pvpq].tocsc(), rhs)
    return va


# --------------------------------------------------------------------- Newton-Raphson
def ds_dv(ybus, v):
    """pypower ``dSbus_dV.py`` (sparse, polar)."""
    ibus = ybus @ v
    n = len(v)
    dv = sp.diags(v)
    di = sp.diags(ibus)
    dvn = sp.diags(v / np.abs(v))
    ds_dvm = dv @ np.conj(ybus @ dvn) + np.conj(di) @ dvn
    ds_dva = 1j * dv @ np.conj(di - ybus @ dv)
    return ds_dvm.tocsr(), ds_dva.tocsr()


def newtonpf(ybus, sbus, v0, ref, pv, pq, tol=1e-8, max_it=10):
    """pandapower ``pypower/newtonpf.py``: returns (V, converged, iterations)."""
    v = v0.astype(complex).copy()
    va, vm = np.angle(v), np.abs(v)
    pvpq = np.r_[pv, pq]
    npv, npq = len(pv), len(pq)

    def mismatch(v):
        mis = v * np.conj(ybus @ v) - sbus
        return np.r_[mis[pvpq].real, mis[pq].imag]

    f = mismatch(v)
    converged = bool(len(f) == 0 or np.max(np.abs(f)) < tol)
    i = 0
    while not converged and i < max_it:
        i += 1
        ds_dvm, ds_dva = ds_dv(ybus, v)
        j11 = ds_dva[pvpq][:, pvpq].real
        j12 = ds_dvm[pvpq][:, pq].real
        j21 = ds_dva[pq][:, pvpq].imag
        j22 = ds_dvm[pq][:, pq].imag
        jac = sp.bmat([[j11, j12], [j21, j22]], format="csc")
        with np.errstate(all="ignore"):
            dx = -spsolve(jac, f)
        if not np.all(np.isfinite(dx)):
            break
        va[pvpq] += dx[: npv + npq]
        vm[pq] += dx[npv + npq:]
        v = vm * np.exp(1j * va)
        vm, va = np.abs(v), np.angle(v)
        f = mismatch(v)
        converged = bool(np.max(np.abs(f)) < tol)
    return v, converged, i


def initial_voltage(ppc: Ppc, init="dc"):
    """pandapower ``_get_pf_variables_from_ppci``: V0 from bus VM/VA, generator
    buses rescaled to their set-point."""
    bus, gen = ppc.bus, ppc.gen
    va = dc_angles(ppc.base_mva, bus, gen, ppc.branch) if init == "dc" else bus[:, VA] * np.pi / 180.0
    v0 = bus[:, VM] * np.exp(1j * va)
    on = gen[:, GEN_STATUS] > 0
    gbus = gen[on, GEN_BUS].astype(int)
    v0[gbus] = gen[on, VG] / np.abs(v0[gbus]) * v0[gbus]
    return v0


def run_pf(ppc: Ppc, tolerance_mva=1e-8, max_iteration=10, enforce_q_lims=True,
           init="dc"):
    """One AC power flow on ppc tables.  Returns a dict with V, converged,
    iterations, branch flows [MVA] and generator P/Q [MW/MVAr]."""
    bus = ppc.bus.copy()
    gen = ppc.gen.copy()
    branch = ppc.branch
    base = ppc.base_mva
    tol = tolerance_mva / base
    ybus, yf, yt = make_ybus(base, bus, branch)
    v0 = initial_voltage(ppc, init)
    total_it = 0
    while True:
        ref, pv, pq = bus_types(bus, gen)
        sbus = make_sbus(base, bus, gen)
        v, ok, it = newtonpf(ybus, sbus, v0, ref, pv, pq, tol, max_iteration)
        total_it = it          # pandapower keeps the iteration count of the last inner run
        # pfsoln: generator reactive power and slack active power
        sinj = v * np.conj(ybus @ v) * base + (bus[:, PD] + 1j * bus[:, QD])
        on = gen[:, GEN_STATUS] > 0
        gbus = gen[:, GEN_BUS].astype(int)
        ngb = np.bincount(gbus[on], minlength=bus.shape[0])
        is_pvref = np.isin(bus[gbus, BUS_TYPE], (PV, REF)) & on
        # Q: bus total minus fixed-Q (PQ-typed) generators, shared equally
        fixed_q = np.zeros(bus.shape[0])
        np.add.at(fixed_q, gbus[on & ~is_pvref], gen[on & ~is_pvref, QG])
        nfree = np.bincount(gbus[is_pvref], minlength=bus.shape[0])
        gen[is_pvref, QG] = (sinj.imag[gbus[is_pvref]] - fixed_q[gbus[is_pvref]]) / nfree[gbus[is_pvref]]
        for r in ref:
            at = np.nonzero(on & (gbus == r))[0]
            gen[at[0], PG] = sinj.real[r] - gen[at[1:], PG].sum()
        if not (ok and enforce_q_lims):
            break
        # pandapower _run_ac_pf_with_qlims_enforced: a generator with QMAX == 0 or QMIN == 0 is skipped
        lim = (gen[:, QMAX] != 0.0) & (gen[:, QMIN] != 0.0) & on & (bus[gbus, BUS_TYPE] == PV)
        mx = np.nonzero(lim & (gen[:, QG] > gen[:, QMAX]))[0]
        mn = np.nonzero(lim & (gen[:, QG] < gen[:, QMIN]))[0]
        if len(mx) == 0 and len(mn) == 0:
            break
        gen[mx, QG] = gen[mx, QMAX]
        gen[mn, QG] = gen[mn, QMIN]
        for g in np.r_[mx, mn]:
            bus[gbus[g], BUS_TYPE] = PQ
        v0 = v
    f = branch[:, F_BUS].astype(int)
    t = branch[:, 1].astype(int)
    sf = v[f] * np.conj(yf @ v) * base
    st = v[t] * np.conj(yt @ v) * base
    return dict(V=v, converged=ok, iterations=total_it, Sf=sf, St=st, gen=gen, bus=bus,
                Ybus=ybus, ppc=ppc)


def branch_loading(ppc: Ppc, res):
    """``results_branch.py``: loading percent of every branch row (lines: i_ka
    vs max_i_ka; trafos: trafo_loading='current')."""
    v = np.abs(res["V"])
    f = ppc.branch[:, F_BUS].astype(int)
    t = ppc.branch[:, T_BUS].astype(int)
    return 100.0 * np.maximum(np.abs(res["Sf"]) * ppc.rate_f / v[f],
                              np.abs(res["St"]) * ppc.rate_t / v[t])


# ------------------------------------------------------------ net-level convenience
def runpp(net, builder=None, enforce_q_lims=True, tolerance_mva=1e-8,
          max_iteration=10, init="dc", **kwargs):
    """Drop-in for ``pp.runpp``: fills ``net.res_*`` or raises
    ``LoadflowNotConverged`` (reference call site ``opfgym/opf_env.py:703``)."""
    import pandas as pd

    from opfgym_b200.net import LoadflowNotConverged      # the stand-in for pandapower's exception type

    # the oracle's OWN net -> ppc conversion (oracle/ppc_ref.py), not the product's
    builder = builder or RefBuilder()
    ppc = builder.build(net)
    res = run_pf(ppc, tolerance_mva, max_iteration, enforce_q_lims, init)
    if not res["converged"]:
        net.converged = False
        raise LoadflowNotConverged("Power Flow nr did not converge after "
                                   f"{max_iteration} iterations!")
    net.converged = True
    v = res["V"]
    lk = ppc.bus_lookup
    ok = lk >= 0
    vm = np.full(len(lk), np.nan)
    va = np.full(len(lk), np.nan)
    vm[ok] = np.abs(v)[lk[ok]]
    va[ok] = np.degrees(np.angle(v))[lk[ok]]
    net.res_bus = pd.DataFrame({"vm_pu": vm, "va_degree": va}, index=net.bus.index)
    loading = branch_loading(ppc, res)

    pos_of = {int(b): i for i, b in enumerate(net.bus.index)}

    def per_branch(mapping, arr, table, ends):
        # a branch that is not in the ppc (out of service): pandapower never writes its rows of ppc['branch'], so
        # its flows are 0 and its current 0 / |V| -- 0 between energised buses, NaN next to a dropped bus
        # (results_branch.py `_get_branch_flows` [ext-mem])
        live = np.array([all(ok[pos_of[int(net[table][c].iloc[i])]] for c in ends) for i in range(len(mapping))], bool) \
            if len(mapping) else np.zeros(0, bool)
        out = np.where(live, 0.0, np.nan).astype(arr.dtype)
        out[mapping >= 0] = arr[mapping[mapping >= 0]]
        return out

    for table, mapping, (a, b) in (("line", ppc.line_branch, ("from", "to")),
                                   ("trafo", ppc.trafo_branch, ("hv", "lv"))):
        ends = (f"{a}_bus", f"{b}_bus")
        sf = per_branch(mapping, res["Sf"], table, ends)
        st = per_branch(mapping, res["St"], table, ends)
        df = pd.DataFrame({
            f"p_{a}_mw": sf.real, f"q_{a}_mvar": sf.imag,
            f"p_{b}_mw": st.real, f"q_{b}_mvar": st.imag,
            "pl_mw": (sf + st).real, "ql_mvar": (sf + st).imag,
            "loading_percent": per_branch(mapping, loading, table, ends)}, index=net[table].index)
        net["res_" + table] = df
    gen = res["gen"]
    eg = ppc.ext_grid_gen
    net.res_ext_grid = pd.DataFrame(
        {"p_mw": np.where(eg >= 0, gen[np.maximum(eg, 0), PG], np.nan),
         "q_mvar": np.where(eg >= 0, gen[np.maximum(eg, 0), QG], np.nan)},
        index=net.ext_grid.index)
    if len(net.gen):
        gg = ppc.gen_gen
        gb = gen[np.maximum(gg, 0), GEN_BUS].astype(int)
        net.res_gen = pd.DataFrame(
            {"p_mw": np.where(gg >= 0, gen[np.maximum(gg, 0), PG], np.nan),
             "q_mvar": np.where(gg >= 0, gen[np.maximum(gg, 0), QG], np.nan),
             "va_degree": np.degrees(np.angle(v))[gb], "vm_pu": np.abs(v)[gb]},
            index=net.gen.index)
    for table in ("load", "sgen", "storage"):
        df = net[table]
        w = df.scaling.to_numpy(float) * df.in_service.to_numpy(bool) if len(df) else 1.0
        net["res_" + table] = pd.DataFrame(
            {"p_mw": df.p_mw.to_numpy(float) * w, "q_mvar": df.q_mvar.to_numpy(float) * w},
            index=df.index)
    return res
