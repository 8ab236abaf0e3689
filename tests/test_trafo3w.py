"""``net.trafo3w``: the star-point conversion of the in-repo builder against the oracle's net-level expansion
(``oracle/trafo3w.py``), closed forms, and the engine per environment against the oracle -- ``tap_pos`` as an action,
``res_trafo3w.loading_percent`` as an observation and as the auto-discovered ``Trafo3wOverloadConstraint``; the
single-net plug-in and ``from_pandapower`` fill ``res_trafo3w``."""
import math

import numpy as np
import pytest

from opfgym_b200 import adapter, constraints as CN, grids, net as N, ppc as P, reward as RW
from opfgym_b200.compiler import Compiler
from opfgym_b200.engine import Engine
from opfgym_b200.pandapower_adapter import from_pandapower
from oracle import ppc_ref as R, scoring, trafo3w as O3
from tests.hostsim.harness import TorchHostSimEngine

T3 = dict(vn_hv_kv=110.0, vn_mv_kv=20.0, vn_lv_kv=10.0, sn_hv_mva=40.0, sn_mv_mva=30.0, sn_lv_mva=15.0,
          vk_hv_percent=12.0, vk_mv_percent=8.0, vk_lv_percent=14.0, vkr_hv_percent=0.3, vkr_mv_percent=0.2,
          vkr_lv_percent=0.25, pfe_kw=20.0, i0_percent=0.05, tap_neutral=0.0, tap_step_percent=1.5, tap_pos=0.0,
          tap_min=-4.0, tap_max=4.0)


def _grid(name, **kw):
    """A stand-in with one trafo3w feeding two new buses (20 kV and 10 kV) that carry a load and a sgen each."""
    net, _ = grids.build_simbench_net(name, n_profile_steps=96)
    hv = 0 if net.bus.vn_kv.loc[0] == 110.0 else int(net.bus.index[net.bus.vn_kv == 110.0][5])
    mv, lv = N.create_bus(net, 20.0), N.create_bus(net, 10.0)
    if "min_vm_pu" in net.bus:
        net.bus.loc[[mv, lv], ["min_vm_pu", "max_vm_pu"]] = [0.9, 1.1]
    params = {**T3, **kw}
    t = N.create_transformer3w_from_parameters(net, hv, mv, lv, **params)
    loads = N.create_loads(net, [mv, lv], [9.0, 4.0], [2.0, 1.0])
    sgens = N.create_sgens(net, [mv, lv], [2.0, 1.0])
    for table, idx in (("load", loads), ("sgen", sgens)):
        for c in ("p_mw", "q_mvar"):
            if f"min_min_{c}" in net[table]:
                net[table].loc[idx, f"min_min_{c}"] = 0.3 * net[table].loc[idx, c]
                net[table].loc[idx, f"max_max_{c}"] = 1.5 * net[table].loc[idx, c]
    return net, t, hv, mv, lv


def _perm(a, b):
    """Product ppc bus -> oracle ppc bus, through the pandapower buses and the branch ends."""
    ok = a.bus_lookup >= 0
    perm = np.full(a.bus.shape[0], -1)
    perm[a.bus_lookup[ok]] = b.bus_lookup[ok]
    for ma, mb in ((a.line_branch, b.line_branch), (a.trafo3w_branch.reshape(-1), b.trafo3w_branch.reshape(-1))):
        for ra, rb in zip(ma, mb):
            if ra >= 0:
                for col in (P.F_BUS, P.T_BUS):
                    perm[int(a.branch[ra, col])] = int(b.branch[rb, col])
    return perm


def _rows_agree(a, b):
    assert np.array_equal(a.trafo3w_branch >= 0, b.trafo3w_branch >= 0)
    perm = _perm(a, b)
    for k, (ra3, rb3) in enumerate(zip(a.trafo3w_branch, b.trafo3w_branch)):
        for w, (ra, rb) in enumerate(zip(ra3, rb3)):
            if ra < 0:
                continue
            assert perm[int(a.branch[ra, P.F_BUS])] == int(b.branch[rb, P.F_BUS])
            assert perm[int(a.branch[ra, P.T_BUS])] == int(b.branch[rb, P.T_BUS])
            for col in (P.BR_R, P.BR_X, P.BR_B, P.BR_G, P.TAP, P.SHIFT):
                assert a.branch[ra, col] == pytest.approx(b.branch[rb, col], rel=1e-12, abs=1e-16), (k, w, col)
            outer = a.rate_f[ra] if w == 0 else a.rate_t[ra]
            star = a.rate_t[ra] if w == 0 else a.rate_f[ra]
            assert star == 0.0 and outer == pytest.approx(b.trafo3w_rate[k, w], rel=1e-13)
    assert a.bus.shape == b.bus.shape and a.branch.shape == b.branch.shape
    for col in (P.BASE_KV, P.BUS_TYPE):
        np.testing.assert_array_equal(a.bus[:, col], b.bus[perm, col])


CASES = {
    "tap_hv": dict(tap_side="hv", tap_pos=3.0),
    "tap_mv": dict(tap_side="mv", tap_pos=-2.0, shift_mv_degree=150.0, shift_lv_degree=30.0),
    "tap_lv": dict(tap_side="lv", tap_pos=4.0, shift_lv_degree=-30.0),
    "star_hv": dict(tap_side="hv", tap_pos=-3.0, tap_at_star_point=True),
    "star_lv": dict(tap_side="lv", tap_pos=2.0, tap_at_star_point=True),
    "negative_x": dict(vk_hv_percent=5.0, vk_mv_percent=20.0, vk_lv_percent=16.0, tap_side="mv", tap_pos=1.0),
}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("name", ["1-MV-semiurb--1-sw", "1-HV-urban--0-sw"])
def test_builders_agree(name, case):
    net, *_ = _grid(name, **CASES[case])
    a, b = P.PpcBuilder(net).build(net), O3.build(net)
    _rows_agree(a, b)
    if case == "negative_x":
        assert (a.branch[a.trafo3w_branch[0], P.BR_X] < 0).any()


def test_builders_agree_on_an_out_of_service_trafo3w_and_its_island():
    net, t, hv, mv, lv = _grid("1-MV-semiurb--1-sw")
    net.trafo3w.loc[t, "in_service"] = False
    a, b = P.PpcBuilder(net).build(net), O3.build(net)
    assert (a.trafo3w_branch == -1).all() and (b.trafo3w_branch == -1).all()
    pos = {int(x): i for i, x in enumerate(net.bus.index)}
    assert a.bus_lookup[pos[hv]] >= 0 and a.bus_lookup[pos[mv]] < 0 and a.bus_lookup[pos[lv]] < 0
    np.testing.assert_array_equal(a.bus_lookup >= 0, b.bus_lookup >= 0)
    assert a.bus.shape == b.bus.shape and a.branch.shape == b.branch.shape
    # loading: 0 next to the live hv bus, NaN next to the dropped mv / lv buses -> NaN
    O3.runpp(net)
    assert np.isnan(net.res_trafo3w.loading_percent.iloc[0])
    assert net.res_trafo3w.p_hv_mw.iloc[0] == 0.0 and np.isnan(net.res_trafo3w.p_mv_mw.iloc[0])


def test_symmetric_unit_star_impedances_are_half_vk():
    """Equal ratings and equal pairwise vk: every star branch has vk/2 (and vkr/2), on its own rating."""
    t = dict(sn_hv_mva=25.0, sn_mv_mva=25.0, sn_lv_mva=25.0, vk_hv_percent=10.0, vk_mv_percent=10.0,
             vk_lv_percent=10.0, vkr_hv_percent=0.4, vkr_mv_percent=0.4, vkr_lv_percent=0.4)
    import pandas as pd
    vk, vkr, sn = P.trafo3w_star_parameters(pd.DataFrame({k: [v] for k, v in t.items()}))
    np.testing.assert_allclose(vk[:, 0], 5.0, rtol=1e-14)
    np.testing.assert_allclose(vkr[:, 0], 0.2, rtol=1e-14)
    ovk, ovkr = O3.star_impedances(t)
    np.testing.assert_allclose(ovk, 5.0, rtol=1e-14)
    np.testing.assert_allclose(ovkr, 0.2, rtol=1e-14)


def test_loading_of_a_two_winding_path_by_hand():
    """hv slack, a load on the mv bus, nothing on the lv bus: loading = 100 * |S_hv| / (vm_hv * sn_hv) (the hv
    terminal carries the most current, vn_hv_kv = bus vn_kv), ld_lv = 0."""
    net = N.create_empty_network(sn_mva=1.0)
    hv, mv, lv = N.create_buses(net, 3, [110.0, 20.0, 10.0])
    N.create_ext_grid(net, hv, vm_pu=1.02)
    N.create_transformer3w_from_parameters(net, hv, mv, lv, **{**T3, "sn_hv_mva": 30.0})
    N.create_load(net, mv, 12.0, 3.0)
    O3.runpp(net)
    r = net.res_trafo3w.iloc[0]
    s_hv = math.hypot(r.p_hv_mw, r.q_hv_mvar)
    assert r.loading_percent == pytest.approx(100.0 * s_hv / (1.02 * 30.0), rel=1e-12)
    assert r.p_lv_mw == pytest.approx(0.0, abs=1e-9) and r.p_mv_mw == pytest.approx(-12.0, rel=1e-9)
    assert r.pl_mw > 0 and r.pl_mw == pytest.approx(r.p_hv_mw + r.p_mv_mw + r.p_lv_mw)
    ld_mv = math.hypot(r.p_mv_mw, r.q_mv_mvar) / net.res_bus.vm_pu.loc[mv] / 30.0 * 100.0
    assert r.loading_percent > ld_mv
    # the product's rows carry the same factors
    p = P.PpcBuilder(net).build(net)
    rows = p.trafo3w_branch[0]
    assert p.rate_f[rows[0]] == pytest.approx(1.0 / 30.0) and p.rate_t[rows[1]] == pytest.approx(1.0 / 30.0)
    assert p.rate_t[rows[2]] == pytest.approx(1.0 / 15.0)


# --------------------------------------------------------------------------- engine per environment
def _program(name, max_loading):
    net, t, *_ = _grid(name, tap_side="mv", shift_mv_degree=150.0, shift_lv_degree=150.0)
    net.trafo3w["max_loading_percent"] = max_loading
    net.trafo3w["min_tap_pos"], net.trafo3w["max_tap_pos"] = -4.0, 4.0
    cons = CN.create_default_constraints(net, {})
    assert any(isinstance(c, CN.Trafo3wOverloadConstraint) for c in cons)
    state = [(tb, c, net[tb].index) for tb, c in (("load", "p_mw"), ("load", "q_mvar"), ("sgen", "p_mw"))]
    obs = [("res_trafo3w", "loading_percent", net.trafo3w.index), ("res_bus", "vm_pu", net.bus.index[-3:])]
    act = [("trafo3w", "tap_pos", net.trafo3w.index)]
    program = Compiler(net, P.PpcBuilder(net)).compile(act, obs, state, cons, RW.Summation())
    return net, program, cons, state, act, obs


def _np(x):
    return x if isinstance(x, np.ndarray) else x.detach().cpu().numpy()


def _engine_vs_oracle(engine_cls, name, kernel, n=24, sync=lambda: None):
    net, program, cons, state, act, obs = _program(name, max_loading=32.0)
    eng = engine_cls(program, n, obs_dtype="float64")
    assert eng.info["pf_kernel_used"] == kernel
    rng = np.random.default_rng(11)
    cols = {}
    for tb, c, idx in state:
        base = net[tb][c].to_numpy(float)
        cols[tb, c] = base * rng.uniform(0.3, 1.6, (n, len(base)))
        view = eng.column(tb, c)
        view[:] = cols[tb, c] if isinstance(view, np.ndarray) else eng._from_numpy(cols[tb, c])
    a = rng.uniform(0.0, 1.0, (n, 1))
    eng.actions[:] = a if isinstance(eng.actions, np.ndarray) else eng._from_numpy(a)
    eng.step()
    sync()
    taps = np.round(a[:, 0] * 8.0 - 4.0)
    assert len(np.unique(taps)) >= 5
    got_ld = _np(eng.column("res_trafo3w", "loading_percent"))[:, 0]
    lk = program.ppc.bus_lookup
    live = lk >= 0
    n_violated = 0
    for b in range(n):
        one = net.deepcopy()
        for (tb, c), v in cols.items():
            one[tb][c] = v[b]
        one.trafo3w["tap_pos"] = taps[b]
        O3.runpp(one)
        assert bool(_np(eng.converged)[b])
        np.testing.assert_allclose(_np(eng.vm[b])[lk[live]], one.res_bus.vm_pu.to_numpy()[live], atol=1e-9)
        np.testing.assert_allclose(np.degrees(_np(eng.va[b])[lk[live]]), one.res_bus.va_degree.to_numpy()[live],
                                   atol=1e-7)
        want = one.res_trafo3w.loading_percent.iloc[0]
        assert got_ld[b] == pytest.approx(want, rel=1e-9)
        assert _np(eng.obs[b])[0] == pytest.approx(want, rel=1e-9)         # the observation key
        out = scoring.step_reward(one, cons, RW.Summation())
        assert (_np(eng.valids[b])[:len(cons)].astype(bool) == out["valids"]).all()
        np.testing.assert_allclose(_np(eng.violations[b])[:len(cons)], out["violations"], rtol=1e-9, atol=1e-12)
        np.testing.assert_allclose(_np(eng.penalties[b])[:len(cons)], out["unscaled_penalties"], rtol=1e-9,
                                   atol=1e-12)
        assert float(_np(eng.reward)[b]) == pytest.approx(out["reward"], rel=1e-9, abs=1e-12)
        assert float(_np(eng.penalty)[b]) == pytest.approx(out["penalty"], rel=1e-9, abs=1e-12)
        n_violated += int(want > 32.0)
    assert 0 < n_violated < n                     # the bound splits the batch


def test_engine_vs_oracle_radial_hostsim():
    _engine_vs_oracle(TorchHostSimEngine, "1-MV-semiurb--1-sw", kernel=3)


def test_engine_vs_oracle_meshed_hostsim():
    _engine_vs_oracle(TorchHostSimEngine, "1-HV-urban--0-sw", kernel=1, n=8)


@pytest.mark.gpu
@pytest.mark.parametrize("name,kernel,n", [("1-MV-semiurb--1-sw", 3, 300), ("1-HV-urban--0-sw", 1, 64)])
def test_engine_vs_oracle_cuda(cuda_lib, name, kernel, n):
    import torch
    _engine_vs_oracle(Engine, name, kernel, n=n, sync=torch.cuda.synchronize)


# --------------------------------------------------------------------------------------- rejections
def test_in_service_cell_is_rejected():
    net, *_ = _grid("1-MV-semiurb--1-sw", tap_side="hv")
    net.trafo3w["min_in_service"], net.trafo3w["max_in_service"] = 0.0, 1.0
    with pytest.raises(NotImplementedError, match="trafo3w.in_service"):
        Compiler(net).compile([("trafo3w", "in_service", net.trafo3w.index)], [], [], [], RW.Summation())


def test_phase_shifting_tap_is_rejected():
    net, *_ = _grid("1-MV-semiurb--1-sw", tap_side="hv", tap_step_degree=1.0)
    with pytest.raises(NotImplementedError, match="tap_step_degree"):
        P.PpcBuilder(net)


def test_table_without_parameter_columns_names_them():
    import pandas as pd
    net, _ = grids.build_simbench_net("1-MV-semiurb--1-sw", n_profile_steps=96)
    net.trafo3w = pd.DataFrame({"hv_bus": [0], "mv_bus": [1], "lv_bus": [2]})
    with pytest.raises(NotImplementedError, match=r"net\.trafo3w.*sn_hv_mva"):
        P.PpcBuilder(net)


# ------------------------------------------------------------------------------------------ plug-ins
def _check_plug_in(engine_cls):
    net, t, *_ = _grid("1-MV-semiurb--1-sw", tap_side="lv", tap_pos=2.0, shift_mv_degree=150.0)
    one = net.deepcopy()
    adapter.PowerFlowSolver(net, engine_cls=engine_cls)(net)
    O3.runpp(one)
    for c in one.res_trafo3w.columns:
        np.testing.assert_allclose(net.res_trafo3w[c].to_numpy(float), one.res_trafo3w[c].to_numpy(float),
                                   rtol=1e-9, atol=1e-9, err_msg=c)
    np.testing.assert_allclose(net.res_bus.vm_pu, one.res_bus.vm_pu, atol=1e-9)


def test_single_net_plug_in_fills_res_trafo3w_hostsim():
    _check_plug_in(TorchHostSimEngine)


@pytest.mark.gpu
def test_single_net_plug_in_fills_res_trafo3w_cuda(cuda_lib):
    _check_plug_in(Engine)


def _fabricate(net):
    """``net._ppc`` / ``_pd2ppc_lookups`` in pandapower's layout (see pandapower_adapter's notes): rows of lines,
    trafos, then 3 rows per trafo3w in hv, mv, lv blocks, from the oracle's conversion."""
    r = O3.build(net)
    ex, _ = O3.expand(net)
    rex = R.build(ex)
    nb = r.bus.shape[0]
    dead = nb
    bus = np.vstack([r.bus, np.zeros((1, r.bus.shape[1]))])
    bus[dead, R.BUS_I], bus[dead, R.BUS_TYPE], bus[dead, R.VM], bus[dead, R.BASE_KV] = dead, 4, 1.0, 1.0
    lookup = np.full(int(net.bus.index.max()) + 1, -1, dtype=np.int64)
    for idx, k in zip(net.bus.index, r.bus_lookup):
        lookup[int(idx)] = k if k >= 0 else dead
    rows, ranges = [], {}
    for table, mapping in (("line", r.line_branch), ("trafo", r.trafo_branch),
                           ("trafo3w", r.trafo3w_branch.T.reshape(-1))):
        first = len(rows)
        for k in mapping:
            if k >= 0:
                rows.append(rex.branch[k].copy())
            else:                                          # out of service: a row stays, status 0
                row = np.zeros(rex.branch.shape[1])
                row[R.F_BUS] = row[R.T_BUS] = dead
                row[R.TAP] = 1.0
                rows.append(row)
        ranges[table] = (first, len(rows))
    net._ppc = {"baseMVA": r.base_mva, "bus": bus, "gen": r.gen.copy(), "branch": np.array(rows)}
    net._pd2ppc_lookups = {"bus": lookup, "branch": ranges}


@pytest.fixture
def _pandapower_column_index(monkeypatch):
    import sys
    import types
    pp, pyp, idx = types.ModuleType("pandapower"), types.ModuleType("pandapower.pypower"), \
        types.ModuleType("pandapower.pypower.idx_brch")
    idx.BR_G = R.BR_G
    pp.pypower, pyp.idx_brch = pyp, idx
    for name, mod in (("pandapower", pp), ("pandapower.pypower", pyp), ("pandapower.pypower.idx_brch", idx)):
        monkeypatch.setitem(sys.modules, name, mod)


def test_from_pandapower_reads_trafo3w_rows(_pandapower_column_index):
    net, *_ = _grid("1-MV-semiurb--1-sw", tap_side="mv", tap_pos=-1.0, shift_mv_degree=150.0)
    _fabricate(net)
    got = from_pandapower(net).build(net)
    own = P.PpcBuilder(net).build(net)
    assert (got.trafo3w_branch >= 0).all()
    for w in range(3):
        ra, rb = own.trafo3w_branch[0, w], got.trafo3w_branch[0, w]
        for col in (P.BR_R, P.BR_X, P.TAP, P.SHIFT):
            assert own.branch[ra, col] == pytest.approx(got.branch[rb, col], rel=1e-12, abs=1e-16)
        assert own.rate_f[ra] == pytest.approx(got.rate_f[rb], rel=1e-12)
        assert own.rate_t[ra] == pytest.approx(got.rate_t[rb], rel=1e-12)
    a, b = net.deepcopy(), net.deepcopy()
    b._ppc, b._pd2ppc_lookups = net._ppc, net._pd2ppc_lookups
    adapter.PowerFlowSolver(a, engine_cls=TorchHostSimEngine)(a)
    adapter.PowerFlowSolver(b, engine_cls=TorchHostSimEngine, builder=from_pandapower(b))(b)
    np.testing.assert_allclose(a.res_trafo3w.loading_percent, b.res_trafo3w.loading_percent, rtol=1e-9)
    assert np.isfinite(b.res_trafo3w.loading_percent.to_numpy()).all()
