"""Host logic of the native library (symbolic phase, schedule, Newton-Raphson walk)
exercised through the host-sim build, against the oracle's known answers."""
import ctypes as C

import numpy as np
import pytest

from opfgym_b200 import capi
from opfgym_b200 import ppc as P
from oracle import pf
from tests import common
from tests.hostsim import harness
from tests.test_oracle_pf import VA9, VM9, wscc9


def solve_ppc(ppc, sbus, init_dc=0, tol=1e-8, ordering=0, threads=0, max_iter=10):
    lib = harness.load()
    gd = capi.GridDesc(nb=ppc.bus.shape[0], ng=ppc.gen.shape[0], nbr=ppc.branch.shape[0],
                       base_mva=ppc.base_mva,
                       bus=ppc.bus.ctypes.data_as(C.POINTER(C.c_double)), bus_cols=ppc.bus.shape[1],
                       gen=ppc.gen.ctypes.data_as(C.POINTER(C.c_double)), gen_cols=ppc.gen.shape[1],
                       branch=ppc.branch.ctypes.data_as(C.POINTER(C.c_double)),
                       branch_cols=ppc.branch.shape[1], tol_pu=tol, max_iter=max_iter,
                       init_dc=init_dc, enforce_q_lims=0, threads_per_env=threads, ordering=ordering)
    h = C.c_void_p()
    capi.check(lib, lib.opfg_grid_create(C.byref(gd), C.byref(h)))
    B, nb = sbus.shape[0], ppc.bus.shape[0]
    vm, va = np.zeros((B, nb)), np.zeros((B, nb))
    conv, it = np.zeros(B, np.uint8), np.zeros(B, np.int32)
    sb = np.ascontiguousarray(np.stack([sbus.real, sbus.imag], axis=-1))
    batch = capi.Batch(n_env=B, sbus=sb.ctypes.data, vm=vm.ctypes.data, va=va.ctypes.data,
                       converged=conv.ctypes.data, iterations=it.ctypes.data)
    capi.check(lib, lib.opfg_pf_solve(h, C.byref(batch), None))
    info = capi.GridInfo()
    lib.opfg_grid_info(h, C.byref(info))
    perm = np.zeros(info.n_nonref, np.int32)
    lvl = np.zeros(info.n_levels + 1, np.int32)
    lib.opfg_grid_symbolic(h, perm.ctypes.data_as(C.POINTER(C.c_int32)),
                           lvl.ctypes.data_as(C.POINTER(C.c_int32)))
    lib.opfg_grid_destroy(h)
    return vm, va, conv, it, info, perm, lvl


@pytest.mark.parametrize("ordering", [0, 1, 2])
def test_wscc9_through_the_c_abi(ordering):
    ppc = wscc9()
    sbus = pf.make_sbus(ppc.base_mva, ppc.bus, ppc.gen)[None, :]
    vm, va, conv, it, info, perm, lvl = solve_ppc(ppc, sbus, tol=1e-8, ordering=ordering)
    assert conv[0] == 1 and it[0] == 4
    np.testing.assert_allclose(vm[0], VM9, atol=5e-10)
    np.testing.assert_allclose(np.degrees(va[0]), VA9, atol=5e-9)
    assert sorted(perm.tolist()) == list(range(1, 9))
    assert lvl[0] == 0 and lvl[-1] == 8 and (np.diff(lvl) > 0).all()


def test_dc_start_matches_oracle_iteration_count():
    case = common.make_case("1-MV-comm--2-sw", n_profile_steps=96)
    ppc = case.program.ppc
    res = pf.run_pf(ppc, init="dc")
    sbus = pf.make_sbus(ppc.base_mva, ppc.bus, ppc.gen)[None, :]
    vm, va, conv, it, info, _, _ = solve_ppc(ppc, sbus, init_dc=1)
    assert conv[0] == 1 and it[0] == res["iterations"]
    np.testing.assert_allclose(vm[0], np.abs(res["V"]), atol=1e-10)
    np.testing.assert_allclose(va[0], np.angle(res["V"]), atol=1e-10)
    # the 150-degree transformer shift must be in the angles (flat start would diverge)
    assert np.abs(np.degrees(va[0])).max() > 140


def test_orderings_agree_and_independent_sets_are_shallower():
    case = common.make_case("1-MV-semiurb--1-sw", n_profile_steps=96)
    ppc = case.program.ppc
    sbus = pf.make_sbus(ppc.base_mva, ppc.bus, ppc.gen)[None, :]
    out = {o: solve_ppc(ppc, sbus, init_dc=1, ordering=o) for o in (1, 2)}
    np.testing.assert_allclose(out[1][0], out[2][0], atol=1e-11)
    np.testing.assert_allclose(out[1][1], out[2][1], atol=1e-11)
    assert out[1][4].n_fill_blocks == 0               # minimum degree: no fill on a radial grid
    assert out[2][4].n_levels < out[1][4].n_levels    # tree contraction: shorter critical path


def test_meshed_grid_and_nonconvergence_flag():
    case = common.make_case("1-HV-urban--0-sw", n_profile_steps=96)
    ppc = case.program.ppc
    s0 = pf.make_sbus(ppc.base_mva, ppc.bus, ppc.gen)
    sbus = np.stack([s0, s0 * 40.0])        # second env: far beyond collapse
    vm, va, conv, it, info, _, _ = solve_ppc(ppc, sbus, init_dc=1)
    res = pf.run_pf(ppc, init="dc")
    assert conv.tolist() == [1, 0] and it[0] == res["iterations"] and it[1] == 10
    np.testing.assert_allclose(vm[0], np.abs(res["V"]), atol=1e-10)
    assert info.n_fill_blocks > 0 and info.smem_bytes_pf < 227 * 1024


def test_bad_tables_are_rejected():
    lib = harness.load()
    ppc = wscc9()
    bus = ppc.bus.copy()
    bus[0, P.BUS_TYPE] = P.PQ       # no reference bus
    gd = capi.GridDesc(nb=9, ng=3, nbr=9, base_mva=100.0,
                       bus=bus.ctypes.data_as(C.POINTER(C.c_double)), bus_cols=bus.shape[1],
                       gen=ppc.gen.ctypes.data_as(C.POINTER(C.c_double)), gen_cols=ppc.gen.shape[1],
                       branch=ppc.branch.ctypes.data_as(C.POINTER(C.c_double)),
                       branch_cols=ppc.branch.shape[1], tol_pu=1e-8, max_iter=10)
    h = C.c_void_p()
    assert lib.opfg_grid_create(C.byref(gd), C.byref(h)) != 0
    assert b"reference bus" in lib.opfg_last_error()


@pytest.mark.parametrize("name", ["1-MV-semiurb--1-sw", "1-HV-urban--0-sw"])
def test_dense_dc_prepass_equals_sparse_dc_start(name, monkeypatch):
    """The schedule with and without the eager gather of far Schur updates seeds and runs the same Newton
    iteration, bit for bit (the partial sums keep the order of additions of the single gather).  The DC start
    comes from the dense pre-pass in both runs; the CTA kernel is the one that runs the schedule."""
    from tests import common
    from tests.hostsim.harness import HostSimEngine
    case = common.make_case(name)
    results = {}
    for eager in ("0", "1"):
        monkeypatch.setenv("OPFG_EAGER_GATHER", eager)
        eng = HostSimEngine(case.program, 6, pf_kernel="cta")
        assert eng.info["pf_kernel_used"] == 1, eng.info
        common.randomize(case, eng, seed=5)
        eng.assemble()
        eng.pf_solve()
        results[eager] = (eng.converged.copy(), eng.iterations.copy(), eng.vm.copy(), eng.va.copy())
    assert results["0"][0].all()
    for a, b in zip(results["0"], results["1"]):
        assert np.array_equal(a, b)
