"""The radial power-flow kernel's schedule: on a radial grid the default analysis roots every tree of the
non-slack bus graph at its centre, so the elimination runs radius + 1 dependent levels per tree -- the
fewest a fill-free order has -- with at most 16 pivots per level and no fill.  The radial kernel on that
order solves the same power flows as the CTA kernel on the minimum-degree order."""
import ctypes as C
from collections import deque

import numpy as np
import pytest

from opfgym_b200 import ppc as P
from tests import common
from tests.test_lane_kernel import _same2

MV = ("1-MV-semiurb--1-sw", "1-MV-rural--0-sw", "1-MV-comm--2-sw")
LEVEL_CAP = 16          # lanes per environment of the radial kernel


def _radius_levels(ppc):
    """max over the trees of the non-slack bus graph (in-service branches) of radius + 1, by brute force:
    the radius is the smallest eccentricity of a node of the tree."""
    nodes = [b for b in range(ppc.bus.shape[0]) if ppc.bus[b, P.BUS_TYPE] != P.REF]
    adj = {b: set() for b in nodes}
    for f, t, on in ppc.branch[:, [P.F_BUS, P.T_BUS, P.BR_STATUS]]:
        f, t = int(f), int(t)
        if on != 0 and f != t and f in adj and t in adj:
            adj[f].add(t)
            adj[t].add(f)

    def dist(src):
        d, q = {src: 0}, deque([src])
        while q:
            v = q.popleft()
            for a in adj[v]:
                if a not in d:
                    d[a] = d[v] + 1
                    q.append(a)
        return d

    edges = sum(len(a) for a in adj.values()) // 2
    seen, levels, components = set(), 0, 0
    for v in nodes:
        if v in seen:
            continue
        comp = list(dist(v))
        seen.update(comp)
        components += 1
        levels = max(levels, min(max(dist(u).values()) for u in comp) + 1)
    assert edges == len(nodes) - components, "not a radial grid"
    return levels


@pytest.mark.parametrize("name", MV)
def test_levels_are_the_tree_radius_hostsim(name):
    from tests.hostsim.harness import HostSimEngine
    case = common.make_case(name, n_profile_steps=96)
    eng = HostSimEngine(case.program, 2)
    info = eng.info
    assert info["pf_kernel_used"] == 3, info
    lvl = np.zeros(info["n_levels"] + 1, np.int32)
    eng.lib.opfg_grid_symbolic(eng.handle, None, lvl.ctypes.data_as(C.POINTER(C.c_int32)))
    assert info["n_levels"] == _radius_levels(case.program.ppc)
    assert lvl[0] == 0 and lvl[-1] == info["n_nonref"]
    assert 0 < np.diff(lvl).min() and np.diff(lvl).max() <= LEVEL_CAP
    assert info["n_fill_blocks"] == 0


def _solve(engine_cls, case, n_env, seed, lam, sync, **kw):
    eng = engine_cls(case.program, n_env, obs_dtype="float64", **kw)
    common.randomize(case, eng, seed=seed)
    eng.assemble()
    sync()
    if lam is not None:
        f = np.random.default_rng(seed).uniform(lam[0], lam[1], n_env)
        sb = common._np(eng.sbus) * f[:, None, None]
        eng.sbus[:] = sb if isinstance(eng.sbus, np.ndarray) else eng._from_numpy(sb)
    eng.pf_solve()
    eng.score()
    sync()
    out = {k: common._np(getattr(eng, k)).copy() for k in ("vm", "va", "converged", "iterations", "reward", "obs")}
    return eng.info, out


def _radial_matches_cta(engine_cls, name, n_env, seed, lam=None, sync=lambda: None):
    """Radial kernel on the default (centre-rooted) order against the CTA kernel on the minimum-degree order:
    the same flags and iteration counts, values within the radial kernel's tolerances (its sums run in
    another order)."""
    case = common.make_case(name)
    info_c, cta = _solve(engine_cls, case, n_env, seed, lam, sync, pf_kernel="cta", ordering=1)
    info_r, radial = _solve(engine_cls, case, n_env, seed, lam, sync)
    assert info_c["pf_kernel_used"] == 1 and info_r["pf_kernel_used"] == 3
    assert info_r["n_levels"] == _radius_levels(case.program.ppc) < info_c["n_levels"]
    _same2(cta, radial, mixed=lam is not None, exact=False)


@pytest.mark.parametrize("name,n_env,lam", [("1-MV-semiurb--1-sw", 24, None),
                                            ("1-MV-semiurb--1-sw", 96, (5.0, 12.0)),
                                            ("1-MV-rural--0-sw", 24, None)])
def test_radial_on_centre_order_matches_cta_hostsim(name, n_env, lam):
    from tests.hostsim.harness import HostSimEngine
    _radial_matches_cta(HostSimEngine, name, n_env, seed=34, lam=lam)


@pytest.mark.gpu
@pytest.mark.parametrize("name,n_env,lam", [("1-MV-semiurb--1-sw", 4133, None),
                                            ("1-MV-semiurb--1-sw", 4096, (5.0, 12.0)),
                                            ("1-MV-rural--0-sw", 2000, None)])
def test_radial_on_centre_order_matches_cta_cuda(cuda_lib, name, n_env, lam):
    import torch
    from opfgym_b200.engine import Engine
    _radial_matches_cta(Engine, name, n_env, seed=33, lam=lam, sync=torch.cuda.synchronize)
