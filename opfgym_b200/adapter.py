"""Single-environment plug-in: the CUDA engine as ``power_flow_solver=`` of an
(unmodified) ``OpfEnv``.

The reference calls ``self._run_power_flow(self.net, **kwargs)`` and expects the
solver to fill ``net.res_*`` in place or raise ``LoadflowNotConverged``
(``opfgym/opf_env.py:53,70,646-662``).  ``power_flow_solver(net)`` does exactly
that with a batch of ONE environment: kernel 1 scatters the net's injections,
kernels 2-4 solve, kernel 5 produces the result cells, which are copied back
into ``res_bus / res_line / res_trafo / res_trafo3w / res_ext_grid / res_gen /
res_load / res_sgen / res_storage``.  The compiled grid is cached per net object; the
topology (switches, in_service) is read at first use.

A batch of one cannot be fast (one CTA on a 148-SM part) -- this adapter exists
for drop-in parity checks inside the reference's own code, not for throughput.
"""
from __future__ import annotations

import weakref

import numpy as np
import pandas as pd

from . import reward as reward_mod
from .compiler import Compiler
from .engine import Engine
from .net import LoadflowNotConverged
from .ppc import PpcBuilder

_INPUTS = (("load", "p_mw"), ("load", "q_mvar"), ("sgen", "p_mw"), ("sgen", "q_mvar"),
           ("storage", "p_mw"), ("storage", "q_mvar"), ("gen", "p_mw"))
_RESULTS = (("res_bus", "vm_pu"), ("res_bus", "va_degree"), ("res_line", "loading_percent"),
            ("res_trafo", "loading_percent"), ("res_line", "_flows4"), ("res_trafo", "_flows4"),
            ("res_ext_grid", "p_mw"), ("res_ext_grid", "q_mvar"), ("res_gen", "q_mvar"),
            ("res_trafo3w", "loading_percent"), ("res_trafo3w", "_flows12"))


class PowerFlowSolver:
    def __init__(self, net, device=None, engine_cls=Engine, tolerance_mva=1e-8, max_iteration=10,
                 builder=None, **engine_kwargs):
        # a real pandapower net brings its own ppc (net._ppc): read it instead of restating the conversion
        if builder is None and type(net).__module__.startswith("pandapower"):
            from .pandapower_adapter import from_pandapower
            builder = from_pandapower(net)
        self.builder = builder or PpcBuilder(net)
        comp = Compiler(net, self.builder)
        inputs = [(t, c, net[t].index) for t, c in _INPUTS if len(net[t])]
        results = [(t, c) for t, c in _RESULTS if t == "res_bus" or (t[4:] in net and len(net[t[4:]]))]
        self.program = comp.compile(act_keys=[], obs_keys=[], state_keys=inputs, constraints=[],
                                    reward_function=reward_mod.Summation(), extra_results=results)
        from .engine import check_engine_class
        check_engine_class(engine_cls)
        self.engine = engine_cls(self.program, 1, device=device, tolerance_mva=tolerance_mva,
                                 max_iteration=max_iteration, obs_dtype="float64", **engine_kwargs)
        self.inputs = inputs

    def __call__(self, net, **kwargs):
        e = self.engine
        for t, c, _ in self.inputs:
            v = np.asarray(net[t][c].to_numpy(), dtype=float)[None, :]
            e.column(t, c).copy_(e._from_numpy(v))
        e.assemble(apply_actions=False)
        e.pf_solve()
        e.score()
        state = e.state[0].cpu().numpy() if hasattr(e.state, "cpu") else np.asarray(e.state[0])
        converged = bool(np.asarray(e.converged.cpu() if hasattr(e.converged, "cpu") else e.converged)[0])
        net.converged = converged
        if not converged:
            raise LoadflowNotConverged(f"Power Flow nr did not converge after "
                                       f"{int(np.asarray(e.iterations.cpu() if hasattr(e.iterations, 'cpu') else e.iterations)[0])} iterations!")
        lay = self.program.layout

        def cells(table, column):
            return state[lay.slice(table, column)]
        net.res_bus = pd.DataFrame({"vm_pu": cells("res_bus", "vm_pu"),
                                    "va_degree": cells("res_bus", "va_degree")}, index=net.bus.index)
        for table, (a, b) in (("line", ("from", "to")), ("trafo", ("hv", "lv"))):
            if not len(net[table]):
                continue
            f4 = cells("res_" + table, "_flows4").reshape(-1, 4)
            net["res_" + table] = pd.DataFrame({
                f"p_{a}_mw": f4[:, 0], f"q_{a}_mvar": f4[:, 1], f"p_{b}_mw": f4[:, 2],
                f"q_{b}_mvar": f4[:, 3], "pl_mw": f4[:, 0] + f4[:, 2], "ql_mvar": f4[:, 1] + f4[:, 3],
                "loading_percent": cells("res_" + table, "loading_percent")}, index=net[table].index)
        if "trafo3w" in net and len(net.trafo3w):
            # per winding branch p/q at its from and to end; the outer ends: hv from, mv / lv to
            f12 = cells("res_trafo3w", "_flows12").reshape(-1, 3, 4)
            f6 = np.stack([f12[:, 0, 0], f12[:, 0, 1], f12[:, 1, 2], f12[:, 1, 3], f12[:, 2, 2], f12[:, 2, 3]], axis=1)
            net.res_trafo3w = pd.DataFrame({
                "p_hv_mw": f6[:, 0], "q_hv_mvar": f6[:, 1], "p_mv_mw": f6[:, 2], "q_mv_mvar": f6[:, 3],
                "p_lv_mw": f6[:, 4], "q_lv_mvar": f6[:, 5], "pl_mw": f6[:, 0] + f6[:, 2] + f6[:, 4],
                "ql_mvar": f6[:, 1] + f6[:, 3] + f6[:, 5],
                "loading_percent": cells("res_trafo3w", "loading_percent")}, index=net.trafo3w.index)
        net.res_ext_grid = pd.DataFrame({"p_mw": cells("res_ext_grid", "p_mw"),
                                         "q_mvar": cells("res_ext_grid", "q_mvar")},
                                        index=net.ext_grid.index)
        if len(net.gen):
            net.res_gen = pd.DataFrame({"p_mw": net.gen.p_mw.to_numpy(float) * net.gen.scaling.to_numpy(float),
                                        "q_mvar": cells("res_gen", "q_mvar")}, index=net.gen.index)
        for table in ("load", "sgen", "storage"):
            df = net[table]
            w = df.scaling.to_numpy(float) * df.in_service.to_numpy(bool) if len(df) else 1.0
            net["res_" + table] = pd.DataFrame({"p_mw": df.p_mw.to_numpy(float) * w,
                                                "q_mvar": df.q_mvar.to_numpy(float) * w}, index=df.index)


_CACHE: "weakref.WeakKeyDictionary" = weakref.WeakKeyDictionary()


def power_flow_solver(net, **kwargs):
    """Drop-in for ``OpfEnv(power_flow_solver=...)``: fills ``net.res_*`` or raises
    ``LoadflowNotConverged``.  ``enforce_q_lims`` / ``lightsim2grid`` keywords of the
    reference's default solver are accepted and ignored (see DESIGN.md §8)."""
    solver = _CACHE.get(net)
    if solver is None:
        solver = _CACHE[net] = PowerFlowSolver(net)
    solver(net)
