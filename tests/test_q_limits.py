"""enforce_q_lims (SURVEY.md §8f rank 1): PV -> PQ switching outer loop of
pandapower's `_run_ac_pf_with_qlims_enforced`, per environment, on the device."""
import numpy as np
import pytest

from opfgym_b200 import adapter, capi, grids
from opfgym_b200 import net as pn
from opfgym_b200.ppc import PpcBuilder
from oracle import pf
from tests.hostsim.harness import TorchHostSimEngine

HOST = dict(engine_cls=TorchHostSimEngine)
# one-sided limits (a zero limit: pandapower skips the generator) next to two-sided ones that bind
MIXED = [(0.0, 8.0), (-8.0, 8.0), (-8.0, 0.0), (-15.0, 25.0), (-30.0, 5.0)]


def _net(qlim):
    net, _ = grids.build_simbench_net("1-HV-urban--0-sw", n_profile_steps=96)
    net.gen["min_q_mvar"] = -qlim
    net.gen["max_q_mvar"] = qlim
    net.gen["vm_pu"] = np.linspace(0.99, 1.03, len(net.gen))
    return net


def _set_limits(net, lims):
    net.gen["min_q_mvar"] = [lo for lo, _ in lims]
    net.gen["max_q_mvar"] = [hi for _, hi in lims]


def _twin_net(lims):
    """The 372-bus grid with a sixth generator on the bus of the third one (same set-point)."""
    net = _net(1e4)
    g = net.gen.index[2]
    pn.create_gen(net, int(net.gen.bus[g]), p_mw=10.0, vm_pu=float(net.gen.vm_pu[g]))
    _set_limits(net, lims)
    return net, g, net.gen.index[-1]


def _solve_both(net, engine_kwargs):
    """Oracle and engine on the same net: |V| within 1e-9, angle within 1e-7 deg, gen Q within 1e-6 MVAr."""
    ref = net.deepcopy()
    pf.runpp(ref, enforce_q_lims=True)
    solver = adapter.PowerFlowSolver(net, **engine_kwargs)
    solver(net)
    np.testing.assert_allclose(net.res_bus.vm_pu, ref.res_bus.vm_pu, atol=1e-9)
    np.testing.assert_allclose(net.res_bus.va_degree, ref.res_bus.va_degree, atol=1e-7)
    np.testing.assert_allclose(net.res_gen.q_mvar, ref.res_gen.q_mvar, atol=1e-6)
    np.testing.assert_allclose(net.res_ext_grid.to_numpy(), ref.res_ext_grid.to_numpy(), atol=1e-6)
    return solver, ref


def _check(engine_kwargs):
    for qlim, expect_binding in ((1e4, False), (8.0, True)):
        net = _net(qlim)
        ref = net.deepcopy()
        res = pf.runpp(ref, enforce_q_lims=True)
        solver = adapter.PowerFlowSolver(net, **engine_kwargs)
        assert (solver.engine.info["nb"], solver.program.ppc.gen.shape[0]) == (372, 6)
        solver(net)
        q = ref.res_gen.q_mvar.to_numpy()
        binding = np.isclose(np.abs(q), qlim, atol=1e-6)
        assert binding.any() == expect_binding
        np.testing.assert_allclose(net.res_bus.vm_pu, ref.res_bus.vm_pu, atol=1e-9)
        np.testing.assert_allclose(net.res_bus.va_degree, ref.res_bus.va_degree, atol=1e-7)
        np.testing.assert_allclose(net.res_gen.q_mvar, q, atol=1e-6)
        np.testing.assert_allclose(net.res_ext_grid.to_numpy(), ref.res_ext_grid.to_numpy(), atol=1e-6)
        if expect_binding:   # the limited buses float: their |V| left the set-point
            free = ref.res_gen.vm_pu.to_numpy()[binding]
            assert (np.abs(free - net.gen.vm_pu.to_numpy()[binding]) > 1e-5).all()
            without = net.deepcopy()
            pf.runpp(without, enforce_q_lims=False)
            assert np.abs(without.res_bus.vm_pu - ref.res_bus.vm_pu).max() > 1e-5


def _check_one_sided(engine_kwargs):
    """A generator with exactly one zero limit is skipped (pandapower: (QMAX != 0) & (QMIN != 0)): its Q stays
    free even where it leaves [QMIN, QMAX], while the two-sided limits on the same grid bind."""
    for lims in (MIXED, [(lo, hi) if lo and hi else (-hi, -lo) for lo, hi in MIXED]):
        net = _net(1e4)
        _set_limits(net, lims)
        _, ref = _solve_both(net, engine_kwargs)
        q = ref.res_gen.q_mvar.to_numpy()
        lo, hi = np.array(lims).T
        one_sided = (lo == 0.0) | (hi == 0.0)
        outside = (q < lo - 1e-3) | (q > hi + 1e-3)
        at_limit = np.isclose(q, lo, atol=1e-6) | np.isclose(q, hi, atol=1e-6)
        assert outside[one_sided].all(), (lims, q)      # the rule decides the result: a limit would have bound
        assert at_limit[~one_sided].sum() >= 2, (lims, q)
        vm = ref.res_gen.vm_pu.to_numpy()
        np.testing.assert_array_equal(np.abs(vm - net.gen.vm_pu.to_numpy())[one_sided] < 1e-12, True)


def _check_twin_generators(engine_kwargs):
    """Two generators with the same limit pair on one PV bus: the pooled limit is the per-generator rule."""
    big = (-1e4, 1e4)
    net, g, twin = _twin_net([big, big, (-20.0, 20.0), big, big, (-20.0, 20.0)])
    solver, ref = _solve_both(net, engine_kwargs)
    assert solver.program.ppc.gen.shape[0] == 7
    q = ref.res_gen.q_mvar
    assert abs(q[g]) == abs(q[twin]) == pytest.approx(20.0, abs=1e-6), q
    assert q[g] == pytest.approx(q[twin], abs=1e-9)


def test_q_limits_hostsim():
    _check(HOST)


def test_one_sided_limits_are_skipped_like_pandapower_hostsim():
    _check_one_sided(HOST)


def test_twin_generators_with_equal_limits_hostsim():
    _check_twin_generators(HOST)


@pytest.mark.parametrize("engine_kwargs", [pytest.param(HOST, id="hostsim"),
                                           pytest.param({}, id="cuda", marks=pytest.mark.gpu)])
def test_different_limits_on_one_bus_are_rejected(request, engine_kwargs):
    """The limits of a PV bus are pooled into one sum: a second generator with another pair is refused when the
    grid is created (Python and C callers alike), with the bus in the message."""
    if not engine_kwargs:
        request.getfixturevalue("cuda_lib")
    big = (-1e4, 1e4)
    net, g, _ = _twin_net([big, big, (-60.0, 60.0), big, big, (-5.0, 5.0)])
    ppc_bus = int(PpcBuilder(net).build(net).bus_lookup[net.bus.index.get_loc(net.gen.bus[g])])
    with pytest.raises(capi.OpfgError, match=rf"PV bus {ppc_bus} .*\(-60, 60\) and \(-5, 5\)"):
        adapter.PowerFlowSolver(net, **engine_kwargs)
    # the same pair on both generators is accepted; enforce_q_lims=False needs no per-bus limit at all
    _set_limits(net, [big, big, (-5.0, 5.0), big, big, (-5.0, 5.0)])
    adapter.PowerFlowSolver(net, **engine_kwargs)
    _set_limits(net, [big, big, (-60.0, 60.0), big, big, (-5.0, 5.0)])
    adapter.PowerFlowSolver(net, enforce_q_lims=False, **engine_kwargs)


def test_both_zero_limits_are_skipped_like_pandapower():
    net = _net(0.0)      # EcoDispatch sets both limits to 0 (envs/eco_dispatch.py:86-88)
    ref = net.deepcopy()
    pf.runpp(ref, enforce_q_lims=True)
    solver = adapter.PowerFlowSolver(net, engine_cls=TorchHostSimEngine)
    solver(net)
    np.testing.assert_allclose(net.res_gen.vm_pu if "vm_pu" in net.res_gen else net.gen.vm_pu,
                               net.gen.vm_pu, atol=1e-12)
    np.testing.assert_allclose(net.res_bus.vm_pu, ref.res_bus.vm_pu, atol=1e-9)
    assert np.abs(ref.res_gen.q_mvar).max() > 1.0     # PV buses still regulate


@pytest.mark.gpu
def test_q_limits_cuda(cuda_lib):
    _check({})


@pytest.mark.gpu
def test_one_sided_limits_are_skipped_like_pandapower_cuda(cuda_lib):
    _check_one_sided({})


@pytest.mark.gpu
def test_twin_generators_with_equal_limits_cuda(cuda_lib):
    _check_twin_generators({})
