"""Every power-flow and scoring build the library ships, not only the one the dispatcher picks by default.

Which build runs depends on the grid, on what fits shared memory and on ``OPFG_*`` knobs; each case below sets
the knobs, asserts from ``Engine.info`` that the intended build is the one that runs (a knob that stops applying
fails the case instead of passing it vacuously) and compares it with a second implementation on the same inputs:

* ``k_pf_multi`` (every stage level, threads per environment and launch bound) and ``k_pf`` (one CTA per
  environment) against ``k_pf_lanes``, the row-wise implementation of the same factorisation: bit for bit.
  Both engines use ordering 1 and the same threads per environment, hence the same schedule.
* ``k_pf_tree`` (8 / 16 / 32 lanes, both 16-lane register builds) against the same: flag and iteration count
  exact, |V| and angle within 1e-11 (the radial kernel forms sum(L W) before subtracting it from J_kk).
* ``k_score<T>`` and ``k_score_warps`` against the default scoring build of the grid.

Two input regimes: converged, and across the collapse boundary (injections scaled by U(5, 12) on MV grids,
U(5, 14) on HV grids).  Batches of 1, 3, 149 and 2051 environments leave environment groups, CTA shares and radial
half-warps idle; environments outside the batch must stay untouched.  The lane kernel itself is checked against
the CPU oracle on a sample of the converged regime.
"""
import concurrent.futures
import functools
import os
import subprocess
import sys

import numpy as np
import pytest

from opfgym_b200 import capi
from opfgym_b200 import grids
from opfgym_b200 import constraints as CN
from opfgym_b200 import reward as RW
from opfgym_b200.compiler import Compiler
from opfgym_b200.ppc import PpcBuilder
from tests import common

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BATCHES = (1, 3, 149, 2051)
N = max(BATCHES)
MV, HV = "1-MV-semiurb--1-sw", "1-HV-urban--0-sw"
LAM = {MV: (5.0, 12.0), HV: (5.0, 14.0), "taps": (5.0, 12.0), "1-MV-rural--0-sw": (2.0, 6.0)}
PF_TOL = dict(vm=1e-6, va=1e-6, loading=1e-4, reward_rel=1e-6)        # tests/test_gpu_parity.py


def _taps_case():
    """The 111-bus grid with transformer tap actions: the Ybus values are per environment (MODE 4-6 of k_pf_multi,
    the DYN builds of k_pf, k_pf_tree and k_pf_lanes).  With tap cells only the grid stays radial and no outage can
    island a bus, so the lane kernel runs there as the reference.  (Switchable ties would make every line's
    in_service a cell and turn the island walk on, and the lane kernel has no island handling.)"""
    net, _ = grids.build_simbench_net("1-MV-comm--2-sw", n_profile_steps=96, load_scaling=1.5, gen_scaling=1.3)
    net.trafo["min_tap_pos"] = -3.0
    net.trafo["max_tap_pos"] = 3.0
    act_keys = [("trafo", "tap_pos", net.trafo.index)]
    obs_keys = [(t, c, net[t].index) for t, c in common.SAMPLED if len(net[t])] + \
        [("res_bus", "vm_pu", net.bus.index[:5])]
    cons = CN.create_default_constraints(net, {})
    rf = RW.Summation()
    builder = PpcBuilder(net)
    program = Compiler(net, builder).compile(act_keys, obs_keys, obs_keys, cons, rf)
    return common.Case(net, builder, program, act_keys, obs_keys, cons, rf)


@functools.lru_cache(maxsize=None)
def _case(key):
    if key == "taps":
        return _taps_case()
    return common.make_case(key, n_profile_steps=96)


def _engine(key, monkeypatch, knobs=(), **kw):
    from opfgym_b200.engine import Engine
    names = ("OPFG_STAGE", "OPFG_ENVS_PER_CTA", "OPFG_TREE_LANES", "OPFG_TREE_ENVS", "OPFG_SCORE_THREADS")
    for k in names:
        monkeypatch.delenv(k, raising=False)
    for k, v in dict(knobs).items():
        monkeypatch.setenv(k, str(v))          # all read when the grid is created
    try:
        return Engine(_case(key).program, N, obs_dtype="float64", **kw)
    finally:
        for k in dict(knobs):
            monkeypatch.delenv(k)


def _sync():
    import torch
    torch.cuda.synchronize()


@functools.lru_cache(maxsize=None)
def _inputs(key):
    """Seeded injections (and per-environment Ybus values) of N environments, both regimes, kernel 1 on the
    device; the lane kernel's result at ordering 1 / default threads is checked against the oracle here."""
    import pytest as _p
    mp = _p.MonkeyPatch()
    try:
        eng = _engine(key, mp, pf_kernel="lanes", ordering=1)
    finally:
        mp.undo()
    case = _case(key)
    common.randomize(case, eng, seed=61)
    eng.assemble()
    _sync()
    sbus = eng.sbus.clone()
    f = np.random.default_rng(62).uniform(*LAM[key], N)
    out = {"converged": dict(sbus=sbus), "collapse": dict(sbus=sbus * eng._from_numpy(f)[:, None, None])}
    if eng.yval is not None:
        for r in out.values():
            r["yval"] = eng.yval.clone()
    if key != "taps":      # (tests/test_dynamic_branches.py replays tap actions on the oracle)
        eng.pf_solve()
        eng.score()
        _sync()
        assert bool(eng.converged.all())
        worst = common.compare_with_oracle(case, eng, envs=range(5, N, 256))
        assert worst["flag_mismatch"] == worst["iter_mismatch"] == worst["valid_mismatch"] == 0, worst
        for k, tol in PF_TOL.items():
            assert worst[k] <= tol, (k, worst)
    eng.close()
    return out


def _solve(eng, inp, n):
    """opfg_pf_solve on the first n environments; the others must keep their sentinel values."""
    eng.sbus.copy_(inp["sbus"])
    if eng.yval is not None:
        eng.yval.copy_(inp["yval"])
    for name, fill in (("vm", -3.0), ("va", -3.0), ("converged", 7), ("iterations", -5)):
        getattr(eng, name).fill_(fill)
    batch = capi.Batch.from_buffer_copy(eng.batch)
    batch.n_env = n
    eng.pf_solve(batch)
    _sync()
    out = {}
    for name, fill in (("vm", -3.0), ("va", -3.0), ("converged", 7), ("iterations", -5)):
        a = getattr(eng, name).cpu().numpy()
        assert (a[n:] == fill).all(), (name, n)
        out[name] = a[:n]
    return out


@functools.lru_cache(maxsize=None)
def _reference(key, threads):
    """The lane kernel on all N environments of both regimes."""
    import pytest as _p
    mp = _p.MonkeyPatch()
    try:
        eng = _engine(key, mp, pf_kernel="lanes", ordering=1, threads_per_env=threads)
    finally:
        mp.undo()
    assert eng.info["pf_kernel_used"] == 2, eng.info
    ref = {regime: _solve(eng, inp, N) for regime, inp in _inputs(key).items()}
    eng.close()
    assert ref["converged"]["converged"].all()
    assert 0.1 < ref["collapse"]["converged"].mean() < 0.9
    return ref


def _compare(key, eng, threads, exact):
    worst = 0.0
    for regime, inp in _inputs(key).items():
        ref = _reference(key, threads)[regime]
        for n in BATCHES:
            got = _solve(eng, inp, n)
            want = {k: v[:n] for k, v in ref.items()}
            for k in ("converged", "iterations"):
                assert np.array_equal(got[k], want[k]), (regime, n, k)
            ok = want["converged"].astype(bool)
            if exact:
                for k in ("vm", "va"):
                    assert np.array_equal(got[k][ok].view(np.int64), want[k][ok].view(np.int64)), (regime, n, k)
                # diverging environments: the iterates agree bit for bit as well (NaN patterns included)
                assert np.array_equal(got["vm"].view(np.int64), want["vm"].view(np.int64)), (regime, n)
            else:
                for k in ("vm", "va"):
                    if ok.any():
                        d = np.abs(got[k][ok] - want[k][ok]).max()
                        worst = max(worst, d)
                        assert d <= 1e-11, (regime, n, k, d)
    return worst


def _bound(threads, envs):
    return 256 if threads * envs <= 256 else (384 if threads * envs <= 384 else 768)


# ------------------------------------------------------------------------------------- CTA kernel builds
# (grid, threads per environment or 0 = the grid's default, knobs, expected threads, E, stage); E = 1 is k_pf<T>
CTA_CASES = [
    (MV, 64, {"OPFG_STAGE": 0}, 64, 12, 0),
    (MV, 64, {"OPFG_STAGE": 1}, 64, 12, 1),
    (MV, 64, {"OPFG_STAGE": 2}, 64, 12, 2),
    (MV, 64, {"OPFG_ENVS_PER_CTA": 6}, 64, 6, 2),
    (MV, 64, {"OPFG_ENVS_PER_CTA": 6, "OPFG_STAGE": 1}, 64, 6, 1),
    (MV, 64, {"OPFG_ENVS_PER_CTA": 4, "OPFG_STAGE": 1}, 64, 4, 1),
    (MV, 64, {"OPFG_ENVS_PER_CTA": 1}, 64, 1, None),
    (MV, 32, {}, 32, 13, 2),
    (MV, 32, {"OPFG_ENVS_PER_CTA": 12, "OPFG_STAGE": 0}, 32, 12, 0),
    (MV, 32, {"OPFG_ENVS_PER_CTA": 8, "OPFG_STAGE": 1}, 32, 8, 1),
    (MV, 128, {"OPFG_STAGE": 1}, 128, 6, 1),
    (MV, 128, {"OPFG_ENVS_PER_CTA": 3}, 128, 3, 2),
    (MV, 128, {"OPFG_ENVS_PER_CTA": 2, "OPFG_STAGE": 0}, 128, 2, 0),
    (MV, 128, {"OPFG_ENVS_PER_CTA": 1}, 128, 1, None),
    (MV, 256, {}, 256, 3, 2),
    (MV, 256, {"OPFG_ENVS_PER_CTA": 1}, 256, 1, None),
    (HV, 0, {}, 128, 3, 0),
    (HV, 0, {"OPFG_STAGE": 1}, 128, 2, 1),
    (HV, 0, {"OPFG_STAGE": 2}, 128, 2, 2),
    (HV, 0, {"OPFG_ENVS_PER_CTA": 1}, 128, 1, None),
    (HV, 32, {}, 32, 3, 0),
    (HV, 64, {"OPFG_STAGE": 1}, 64, 2, 1),
    (HV, 256, {}, 256, 3, 0),
    (HV, 256, {"OPFG_STAGE": 2}, 256, 2, 2),
    ("taps", 0, {"OPFG_STAGE": 0}, 64, 12, 0),
    ("taps", 0, {"OPFG_STAGE": 1}, 64, 12, 1),
    ("taps", 0, {"OPFG_STAGE": 2}, 64, 12, 2),
    ("taps", 0, {"OPFG_STAGE": 1, "OPFG_ENVS_PER_CTA": 4}, 64, 4, 1),
    ("taps", 0, {"OPFG_ENVS_PER_CTA": 1}, 64, 1, None),
    ("taps", 128, {"OPFG_ENVS_PER_CTA": 1}, 128, 1, None),
]


def _cta_id(c):
    key, threads, knobs, _, E, stage = c
    name = {MV: "mv122", HV: "hv372", "taps": "taps111"}[key]
    return f"{name}-T{threads or 'auto'}-E{E}-S{stage}"


@pytest.mark.gpu
@pytest.mark.parametrize("case", CTA_CASES, ids=[_cta_id(c) for c in CTA_CASES])
def test_cta_kernel_builds_match_lane_kernel(cuda_lib, monkeypatch, case):
    key, threads, knobs, want_T, want_E, want_stage = case
    eng = _engine(key, monkeypatch, knobs, pf_kernel="cta", ordering=1, threads_per_env=threads)
    info = eng.info
    assert info["pf_kernel_used"] == 1, info
    assert info["threads_per_env"] == want_T and info["cta_envs_per_cta"] == want_E, info
    if want_E > 1:
        assert info["cta_tables_staged"] == want_stage, info
        assert _bound(want_T, want_E) in (256, 384, 768)
    _compare(key, eng, threads, exact=True)
    eng.close()


def test_cta_cases_cover_every_stage_and_launch_bound():
    """The table above reaches every (stage, launch bound) instantiation of k_pf_multi, every stage with
    per-environment Ybus, and k_pf for T = 64 and 128 with and without per-environment Ybus."""
    seen = {(key == "taps", "k_pf" if E == 1 else stage, T if E == 1 else _bound(T, E))
            for key, _, _, T, E, stage in CTA_CASES}
    want = {(False, s, b) for s in (0, 1, 2) for b in (256, 384, 768)} | {(True, s, 768) for s in (0, 1, 2)} | \
        {(d, "k_pf", T) for d in (False, True) for T in (64, 128)}
    assert want <= seen, want - seen


def test_cta_case_table_hostsim(monkeypatch):
    """grid_create picks environments per CTA and the stage level the same way in the host build: the expectations
    of the table hold before any GPU runs them."""
    from tests.hostsim.harness import HostSimEngine
    for key, threads, knobs, want_T, want_E, want_stage in CTA_CASES:
        for k in ("OPFG_STAGE", "OPFG_ENVS_PER_CTA"):
            monkeypatch.delenv(k, raising=False)
        for k, v in knobs.items():
            monkeypatch.setenv(k, str(v))
        info = HostSimEngine(_case(key).program, 2, pf_kernel="cta", ordering=1, threads_per_env=threads).info
        assert (info["threads_per_env"], info["cta_envs_per_cta"]) == (want_T, want_E), (key, knobs, info)
        if want_E > 1:
            assert info["cta_tables_staged"] == want_stage, (key, knobs, info)


# ---------------------------------------------------------------------------------------- radial builds
# (grid, knobs, lanes, register build): 384 = the 16-lane build capped at 24 environments, 512 = the plain one
TREE_CASES = [
    (MV, {"OPFG_TREE_LANES": 8}, 8, None),
    (MV, {"OPFG_TREE_LANES": 16, "OPFG_TREE_ENVS": 24}, 16, 384),
    (MV, {"OPFG_TREE_LANES": 32}, 32, None),
    ("1-MV-rural--0-sw", {}, 16, 512),
    ("1-MV-rural--0-sw", {"OPFG_TREE_LANES": 8}, 8, None),
    ("taps", {"OPFG_TREE_LANES": 8}, 8, None),
    ("taps", {"OPFG_TREE_LANES": 16, "OPFG_TREE_ENVS": 24}, 16, 384),
    ("taps", {"OPFG_TREE_LANES": 32}, 32, None),
]
TREE_WORST = {}


@pytest.mark.gpu
@pytest.mark.parametrize("case", TREE_CASES, ids=[f"{c[0][:8]}-L{c[2]}-{c[3]}" for c in TREE_CASES])
def test_radial_kernel_builds_match_lane_kernel(cuda_lib, monkeypatch, case):
    key, knobs, lanes, build = case
    eng = _engine(key, monkeypatch, knobs, ordering=1)
    info = eng.info
    assert info["pf_kernel_used"] == 3 and info["radial_lanes_per_env"] == lanes, info
    E = info["radial_envs_per_cta"]
    assert E % (32 // lanes) == 0 and E <= (24 if lanes == 32 else 32), info
    if build == 384:
        assert E <= 24, info
    elif build == 512:
        assert E > 24, info
    if key == "taps":
        assert eng.yval is not None
    TREE_WORST[(key, lanes, build)] = _compare(key, eng, 0, exact=False)
    eng.close()


# ---------------------------------------------------------------------------------------- scoring builds
SCORE_CASES = [(MV, None, 32), (MV, 64, 64), (MV, 128, 128), (MV, 256, 256), (HV, None, 128), (HV, 32, 32)]
SCORE_BATCHES = (1, 3, 2051)
EXACT_STATS = [0, 1, 2, 7] + list(range(8, capi.N_STATS))     # counts: N, converged, valid, iterations, violated


@functools.lru_cache(maxsize=None)
def _scored_inputs(key):
    """State, injections and power-flow results of both regimes (default power-flow build)."""
    import pytest as _p
    mp = _p.MonkeyPatch()
    try:
        eng = _engine(key, mp)
    finally:
        mp.undo()
    case = _case(key)
    common.randomize(case, eng, seed=61)            # the state of the injections of _inputs
    eng.assemble()
    _sync()
    state0 = eng.state.clone()
    out = {}
    for regime, inp in _inputs(key).items():
        eng.state.copy_(state0)
        eng.sbus.copy_(inp["sbus"])
        eng.pf_solve()
        _sync()
        out[regime] = {k: getattr(eng, k).clone() for k in ("state", "sbus", "vm", "va", "converged", "iterations")}
    eng.close()
    return out


def _score(eng, inp, n):
    for k, v in inp.items():
        getattr(eng, k).copy_(v)
    for k in ("reward", "objective", "penalty", "cost", "violations", "penalties", "obs"):
        getattr(eng, k).fill_(-11.0)
    eng.valids.fill_(9)
    eng.stats.zero_()
    batch = capi.Batch.from_buffer_copy(eng.batch)
    batch.n_env = n
    eng.score(batch)
    _sync()
    out = {k: getattr(eng, k).cpu().numpy()[:n].copy() for k in
           ("reward", "objective", "penalty", "cost", "valids", "violations", "penalties", "obs", "state")}
    assert (eng.reward.cpu().numpy()[n:] == -11.0).all()
    out["stats"] = eng.stats.cpu().numpy().sum(axis=0)
    return out


@functools.lru_cache(maxsize=None)
def _score_reference(key):
    import pytest as _p
    mp = _p.MonkeyPatch()
    try:
        eng = _engine(key, mp)
    finally:
        mp.undo()
    out = {(regime, n): _score(eng, inp, n) for regime, inp in _scored_inputs(key).items() for n in SCORE_BATCHES}
    info = eng.info
    eng.close()
    return info, out


@pytest.mark.gpu
@pytest.mark.parametrize("case", SCORE_CASES, ids=[f"{'mv122' if c[0] == MV else 'hv372'}-{c[1] or 'default'}"
                                                   for c in SCORE_CASES])
def test_scoring_builds_agree(cuda_lib, monkeypatch, case):
    key, threads, want = case
    ref_info, ref = _score_reference(key)
    default = SCORE_CASES[0][2] if key == MV else SCORE_CASES[4][2]
    assert ref_info["score_threads_per_env"] == default, ref_info
    eng = _engine(key, monkeypatch, {"OPFG_SCORE_THREADS": threads} if threads else {})
    assert eng.info["score_threads_per_env"] == want, eng.info
    n_in = _case(key).program.layout.n_inputs
    for regime, inp in _scored_inputs(key).items():
        for n in SCORE_BATCHES:
            got, exp = _score(eng, inp, n), ref[(regime, n)]
            assert np.array_equal(got["valids"], exp["valids"]), (regime, n)
            assert np.array_equal(got["stats"][EXACT_STATS], exp["stats"][EXACT_STATS]), (regime, n)
            cells, cells_ref = got["state"][:, n_in:], exp["state"][:, n_in:]
            assert np.array_equal(np.isnan(cells), np.isnan(cells_ref)), (regime, n)
            assert np.array_equal(cells[~np.isnan(cells)], cells_ref[~np.isnan(cells_ref)]), (regime, n)
            assert np.array_equal(got["state"][:, :n_in], exp["state"][:, :n_in])
            for k in ("reward", "objective", "penalty", "cost", "violations", "penalties", "obs", "stats"):
                a, b = got[k], exp[k]
                assert np.array_equal(np.isnan(a), np.isnan(b)), (regime, n, k)
                ok = ~np.isnan(b)
                scale = np.abs(b[ok]).max(initial=0.0)
                assert np.abs(a[ok] - b[ok]).max(initial=0.0) <= 1e-12 * scale, (regime, n, k)
    eng.close()


# ------------------------------------------------------------------------------- knobs read once per process
# `static` in the library: each setting runs in a process of its own (tests/_build_variant_run.py).  Register
# caps and launch shapes change no arithmetic: every output bit must agree with the default build.
VARIANTS = [
    {"OPFG_AUX_WARPS": 1, "OPFG_ASSEMBLE_CAP": 3, "OPFG_SCORE_CAP": 3},
    {"OPFG_ASSEMBLE_CAP": 1, "OPFG_SCORE_CAP": 1},
    {"OPFG_ASSEMBLE_CAP": 2, "OPFG_SCORE_CAP": 4},
    {"OPFG_SCORE_CAP": 0, "OPFG_TREE_WIDE_REGS": 0, "OPFG_MULTI_ROOMY": 0},
    {"OPFG_PREFER_ENVS": 0},
]
VARIANT_BASE = {"OPFG_TREE_ENVS": 24}        # the 122-bus grid then runs the 16-lane build TREE_WIDE_REGS selects


@pytest.mark.gpu
def test_process_wide_knobs_change_no_bit(cuda_lib, monkeypatch, tmp_path):
    from tests import _build_variant_run as helper
    for k, v in VARIANT_BASE.items():
        monkeypatch.setenv(k, str(v))
    base = helper.run_all()
    info = {k: base.pop(k) for k in list(base) if k.endswith("/info")}

    def child(i):
        env = dict(os.environ)
        env.update({k: str(v) for k, v in {**VARIANT_BASE, **VARIANTS[i]}.items()})
        out = tmp_path / f"variant{i}.npz"
        flags = ["-s"] if sys.flags.no_user_site else []
        res = subprocess.run([sys.executable, *flags, os.path.join(ROOT, "tests", "_build_variant_run.py"), str(out)],
                             env=env, cwd=ROOT, capture_output=True, text=True, timeout=600)
        assert res.returncode == 0, (VARIANTS[i], res.stderr[-3000:])
        return dict(np.load(out))

    with concurrent.futures.ThreadPoolExecutor(len(VARIANTS)) as pool:
        results = list(pool.map(child, range(len(VARIANTS))))
    for knobs, got in zip(VARIANTS, results):
        got_info = {k: got.pop(k) for k in list(got) if k.endswith("/info")}
        assert set(got) == set(base)
        for k in base:
            assert np.array_equal(got[k].view(np.uint8), base[k].view(np.uint8)), (knobs, k)
        if "OPFG_PREFER_ENVS" in knobs:     # the knob applies: the 372-bus grid stages every table for 2 environments
            assert tuple(info[f"{HV}/info"][:3]) == (1, 3, 0), info
            assert tuple(got_info[f"{HV}/info"][:3]) == (1, 2, 2), got_info
        else:
            for k in info:
                assert np.array_equal(info[k], got_info[k]), (knobs, k)
