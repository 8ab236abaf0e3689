"""Parity against the REAL pandapower (``pp.runpp(net, enforce_q_lims=True)``, the call the reference makes
at opfgym/opf_env.py:703) -- runs wherever pandapower is importable, skips (with the reason printed)
where it is not, which includes the build image and the GPU boxes of this project.

What it pins when it runs, with BASELINE.json's tolerances: converged flag exact; |V| and angle 1e-6
pu / rad; line and transformer loading 1e-4 %; slack P/Q 1e-6 relative.  Three arms:
  1. the oracle (oracle/pf.py on oracle/ppc_ref.py) against pandapower -- pins the oracle itself;
  2. the engine fed by ``from_pandapower(net)`` (pandapower's own ppc) against pandapower;
  3. the engine fed by the product's own net -> ppc conversion against pandapower.
Arms 2 and 3 need the CUDA library and a GPU (marked gpu); arm 1 runs on any CPU box."""
import numpy as np
import pytest

pp = pytest.importorskip("pandapower", reason="pandapower is not installed: parity against the real "
                         "pp.runpp cannot run here (SURVEY.md 8c); the oracle stays 'parity unpinned'")
import pandapower.networks as pn      # noqa: E402

TOL = dict(vm=1e-6, va=1e-6, loading=1e-4, slack_rel=1e-6)


def _nets():
    yield "case14", pn.case14()
    yield "case30", pn.case30()
    yield "mv_oberrhein", pn.mv_oberrhein()
    # ward + (symmetric) impedance elements: pins the [ext-mem] conversions of opfgym_b200/ppc.py and oracle/ppc_ref.py
    # (tests/test_ward_impedance.py can only hold the two restatements against each other)
    extra = pn.case14()
    pp.create_ward(extra, 4, ps_mw=3.0, qs_mvar=1.0, pz_mw=2.0, qz_mvar=-1.5)
    pp.create_ward(extra, 9, ps_mw=-1.0, qs_mvar=0.5, pz_mw=0.0, qz_mvar=2.0, in_service=False)
    same_level = [b for b in extra.bus.index if extra.bus.vn_kv[b] == extra.bus.vn_kv[10] and b != 10]
    pp.create_impedance(extra, 10, same_level[-1], rft_pu=0.02, xft_pu=0.07, sn_mva=50.0)
    yield "case14+ward+impedance", extra
    # one-sided generator Q limits (pandapower skips a generator with QMIN == 0 or QMAX == 0) next to tight two-sided
    # ones that bind: pins the skip rule of oracle/pf.py and of the engine's q-limit tables
    one_sided = pn.case14()
    one_sided.gen["min_q_mvar"] = [0.0, -5.0, -3.0, -3.0][:len(one_sided.gen)]
    one_sided.gen["max_q_mvar"] = [5.0, 0.0, 3.0, 3.0][:len(one_sided.gen)]
    yield "case14+one-sided-q-limits", one_sided
    try:
        import simbench as sb
        yield "1-MV-semiurb--1-sw", sb.get_simbench_net("1-MV-semiurb--1-sw")
        yield "1-HV-urban--0-sw", sb.get_simbench_net("1-HV-urban--0-sw")
    except ImportError:
        pass


def _to_container(net):
    """pandapower net -> the in-repo Net container (same tables; used by the oracle and by arm 3)."""
    from opfgym_b200 import net as N
    out = N.Net(sn_mva=float(net.sn_mva), f_hz=float(net.f_hz))
    for table in ("bus", "line", "trafo", "impedance", "switch", "load", "sgen", "storage", "ward", "gen", "ext_grid",
                  "shunt"):
        if table in net and len(net[table]):
            out[table] = net[table].copy()
    return out


def _compare(ref, got, label):
    assert bool(ref.converged) == bool(got.converged), label
    if not ref.converged:
        return
    np.testing.assert_allclose(got.res_bus.vm_pu, ref.res_bus.vm_pu, atol=TOL["vm"], err_msg=label)
    np.testing.assert_allclose(np.radians(got.res_bus.va_degree), np.radians(ref.res_bus.va_degree),
                               atol=TOL["va"], err_msg=label)
    for table in ("res_line", "res_trafo"):
        if len(ref[table]):
            np.testing.assert_allclose(got[table].loading_percent, ref[table].loading_percent,
                                       atol=TOL["loading"], err_msg=label + " " + table)
    np.testing.assert_allclose(got.res_ext_grid[["p_mw", "q_mvar"]].to_numpy(float),
                               ref.res_ext_grid[["p_mw", "q_mvar"]].to_numpy(float),
                               rtol=TOL["slack_rel"], atol=1e-7, err_msg=label)


def _cases(net, n=6, seed=0):
    rng = np.random.default_rng(seed)
    base_p, base_q = net.load.p_mw.to_numpy().copy(), net.load.q_mvar.to_numpy().copy()
    for k in range(n):
        f = rng.uniform(0.4, 1.6, len(base_p)) * (1.0 if k < n - 1 else 40.0)     # the last one diverges
        net.load["p_mw"], net.load["q_mvar"] = base_p * f, base_q * f
        yield k


@pytest.mark.parametrize("name,net", list(_nets()), ids=lambda x: x if isinstance(x, str) else "")
def test_oracle_vs_pandapower(name, net):
    from oracle import pf
    from opfgym_b200.net import LoadflowNotConverged
    for k in _cases(net):
        try:
            pp.runpp(net, enforce_q_lims=True)
        except pp.powerflow.LoadflowNotConverged:
            net.converged = False
        mine = _to_container(net)
        try:
            pf.runpp(mine, enforce_q_lims=True)
        except LoadflowNotConverged:
            mine.converged = False
        _compare(net, mine, f"{name} case {k}")


@pytest.mark.gpu
@pytest.mark.parametrize("source", ["from_pandapower", "own_conversion"])
@pytest.mark.parametrize("name,net", list(_nets()), ids=lambda x: x if isinstance(x, str) else "")
def test_engine_vs_pandapower(name, net, source):
    from opfgym_b200 import adapter
    from opfgym_b200.net import LoadflowNotConverged
    from opfgym_b200.pandapower_adapter import from_pandapower
    target = net if source == "from_pandapower" else _to_container(net)
    solver = adapter.PowerFlowSolver(target, builder=from_pandapower(net) if source == "from_pandapower" else None)
    for k in _cases(net):
        try:
            pp.runpp(net, enforce_q_lims=True)
        except pp.powerflow.LoadflowNotConverged:
            net.converged = False
        import copy
        ref = copy.deepcopy(net)                  # pandapower's results, before the engine overwrites res_*
        if source != "from_pandapower":
            target.load["p_mw"], target.load["q_mvar"] = net.load.p_mw.to_numpy(), net.load.q_mvar.to_numpy()
        try:
            solver(target)
        except LoadflowNotConverged:
            target.converged = False
        _compare(ref, target, f"{name} {source} case {k}")


def test_oracle_topology_semantics_vs_pandapower():
    """The restated topology rules (oracle/ppc_ref.py, all [ext-mem]) against pandapower itself: an
    out-of-service line, a line opened at one end by its switch (auxiliary bus), an outage that islands part of
    a feeder (`_check_connectivity`: dropped buses report NaN).  The engine is pinned to the oracle on exactly
    these cases by tests/test_islands.py and tests/test_switch_cells.py."""
    from oracle import pf
    net = pn.mv_oberrhein()
    line_switches = net.switch.index[(net.switch.et == "l") & net.switch.closed]
    cases = {"line out of service": lambda n: n.line.__setitem__("in_service", n.line.in_service.where(n.line.index != n.line.index[7], False)),
             "line open at one end": lambda n: n.switch.__setitem__("closed", n.switch.closed.where(n.switch.index != line_switches[3], False)),
             "islanding outage": lambda n: n.line.__setitem__("in_service", n.line.in_service.where(n.line.index != n.line.index[40], False))}
    import copy
    for label, change in cases.items():
        ref = copy.deepcopy(net)
        change(ref)
        pp.runpp(ref, enforce_q_lims=True)
        mine = _to_container(ref)
        pf.runpp(mine, enforce_q_lims=True)
        for table, column, tol in (("res_bus", "vm_pu", TOL["vm"]), ("res_line", "loading_percent", TOL["loading"]),
                                   ("res_trafo", "loading_percent", TOL["loading"])):
            a, b = ref[table][column].to_numpy(float), mine[table][column].to_numpy(float)
            assert (np.isnan(a) == np.isnan(b)).all(), f"{label}: NaN pattern of {table}.{column}"
            np.testing.assert_allclose(b[~np.isnan(a)], a[~np.isnan(a)], atol=tol, err_msg=f"{label} {table}.{column}")
