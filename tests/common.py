"""Shared fixtures of the test tiers: a compiled VoltageControl-like case on a
synthetic stand-in grid, seeded inputs, and the per-environment oracle replay."""
from __future__ import annotations

from dataclasses import dataclass

import numpy as np

from opfgym_b200 import constraints as CN
from opfgym_b200 import grids
from opfgym_b200 import net as pn
from opfgym_b200 import ppc as P
from opfgym_b200 import reward as RW
from opfgym_b200.compiler import Compiler

SAMPLED = (("load", "p_mw"), ("load", "q_mvar"), ("sgen", "p_mw"), ("storage", "p_mw"))


@dataclass
class Case:
    net: object
    builder: object
    program: object
    act_keys: list
    obs_keys: list
    constraints: list
    reward: object


def make_case(name="1-MV-semiurb--1-sw", n_profile_steps=672, reward=None, constraint_kwargs=None,
              load_scaling=1.5, gen_scaling=1.3, tight=False, prepare=None, extra_obs=()) -> Case:
    net, _ = grids.build_simbench_net(name, n_profile_steps=n_profile_steps,
                                      load_scaling=load_scaling, gen_scaling=gen_scaling)
    if prepare is not None:      # net tweaks before the tables are compiled (e.g. generator Q limits)
        prepare(net)
    thr = np.sort(net.sgen.max_max_p_mw.to_numpy())[-10]
    net.sgen["controllable"] = net.sgen.max_max_p_mw >= thr
    qlim = 0.5 * net.sgen.max_max_p_mw.to_numpy()
    net.sgen["min_q_mvar"] = -qlim
    net.sgen["max_q_mvar"] = qlim
    net.ext_grid["max_q_mvar"] = 0.5 if not tight else 0.05
    net.ext_grid["min_q_mvar"] = -0.5 if not tight else -0.05
    if tight:   # provoke voltage and loading violations
        net.bus["max_vm_pu"] = 1.01
        net.bus["min_vm_pu"] = 0.99
        net.line["max_loading_percent"] = 15.0
        net.trafo["max_loading_percent"] = 10.0
    ctrl = net.sgen.index[net.sgen.controllable]
    for idx in ctrl:
        pn.create_poly_cost(net, idx, "sgen", cp1_eur_per_mw=0.03, cq2_eur_per_mvar2=0.01)
    for idx in net.ext_grid.index:
        pn.create_poly_cost(net, idx, "ext_grid", cp1_eur_per_mw=0.03, cq1_eur_per_mvar=0.002)
        pn.create_pwl_cost(net, idx, "ext_grid", points=[[-1000, 0, 0.01], [0, 1000, 0.05]])
    obs_keys = [("sgen", "p_mw", net.sgen.index), ("storage", "p_mw", net.storage.index),
                ("load", "p_mw", net.load.index), ("load", "q_mvar", net.load.index),
                ("res_bus", "vm_pu", net.bus.index[:5]),
                ("res_line", "loading_percent", net.line.index[:4]),
                ("res_ext_grid", "p_mw", net.ext_grid.index)] + \
        [(t, c, net[t[len("res_"):]].index) for t, c in extra_obs]      # result columns of every element
    act_keys = [("sgen", "q_mvar", ctrl)]
    cons = CN.create_default_constraints(net, constraint_kwargs or {})
    rf = reward or RW.Summation()
    builder = P.PpcBuilder(net)
    program = Compiler(net, builder).compile(act_keys, obs_keys, obs_keys, cons, rf)
    return Case(net, builder, program, act_keys, obs_keys, cons, rf)


def random_inputs(case: Case, n_env: int, seed: int):
    rng = np.random.default_rng(seed)
    cols = {}
    for t, c in SAMPLED:
        df = case.net[t]
        if not len(df):
            continue
        lo, hi = df["min_min_" + c].to_numpy(), df["max_max_" + c].to_numpy()
        cols[(t, c)] = rng.uniform(lo, hi, (n_env, len(df))) / df.scaling.to_numpy()
    actions = rng.uniform(-0.05, 1.05, (n_env, case.program.n_act))
    return cols, actions


def randomize(case: Case, eng, seed: int):
    """Write seeded inputs into an engine (torch or numpy buffers alike)."""
    cols, actions = random_inputs(case, eng.num_envs, seed)
    for (t, c), v in cols.items():
        view = eng.column(t, c)
        view[:] = v if isinstance(view, np.ndarray) else eng._from_numpy(v)
    if isinstance(eng.actions, np.ndarray):
        eng.actions[:] = actions
    else:
        eng.actions.copy_(eng._from_numpy(actions))
    return cols, actions


def _np(x):
    return x if isinstance(x, np.ndarray) else x.detach().cpu().numpy()


def oracle_env(case: Case, eng, b: int):
    """Replay environment b on the CPU oracle from the engine's own input cells."""
    from oracle import pf, scoring
    net = case.net.deepcopy()
    for t, c in SAMPLED:
        if len(net[t]):
            net[t][c] = _np(eng.column(t, c)[b])
    a = np.clip(_np(eng.actions[b]), 0.0, 1.0)
    k = 0
    for t, c, idxs in case.act_keys:     # opfgym/opf_env.py:432-483
        df = net[t]
        lo, hi = df[f"min_{c}"].loc[idxs].to_numpy(), df[f"max_{c}"].loc[idxs].to_numpy()
        sp = a[k:k + len(idxs)] * (hi - lo) + lo
        net[t].loc[idxs, c] = sp / df.scaling.loc[idxs].to_numpy()
        k += len(idxs)
    out = {"net": net}
    try:
        res = pf.runpp(net)            # the oracle's own net -> ppc conversion (oracle/ppc_ref.py)
        out.update(converged=True, iterations=res["iterations"], pf=res,
                   vm=net.res_bus.vm_pu.to_numpy(float), va=np.radians(net.res_bus.va_degree.to_numpy(float)))
        out.update(scoring.step_reward(net, case.constraints, case.reward))
        obs = [net[t].loc[idxs, c].to_numpy(float) for t, c, idxs in case.obs_keys]
        out["obs"] = np.concatenate(obs)
    except pn.LoadflowNotConverged:
        out.update(converged=False)
    return out


def compare_with_oracle(case: Case, eng, envs):
    worst = dict(vm=0.0, va=0.0, reward_rel=0.0, violation=0.0, obs=0.0, loading=0.0,
                 flag_mismatch=0, iter_mismatch=0, valid_mismatch=0)
    conv = _np(eng.converged)
    for b in envs:
        o = oracle_env(case, eng, b)
        if bool(conv[b]) != o["converged"]:
            worst["flag_mismatch"] += 1
            continue
        if not o["converged"]:
            continue
        worst["iter_mismatch"] += int(_np(eng.iterations)[b] != o["iterations"])
        lk = case.program.ppc.bus_lookup      # pandapower bus order on both sides (the numberings differ)
        has = lk >= 0
        worst["vm"] = max(worst["vm"], np.abs(_np(eng.vm[b])[lk[has]] - o["vm"][has]).max())
        worst["va"] = max(worst["va"], np.abs(_np(eng.va[b])[lk[has]] - o["va"][has]).max())
        r = float(_np(eng.reward)[b])
        worst["reward_rel"] = max(worst["reward_rel"], abs(r - o["reward"]) / max(1e-12, abs(o["reward"])))
        worst["violation"] = max(worst["violation"], np.abs(_np(eng.violations[b]) - o["violations"]).max())
        worst["valid_mismatch"] += int((_np(eng.valids[b]).astype(bool) != o["valids"]).any())
        worst["obs"] = max(worst["obs"], np.abs(_np(eng.obs[b]).astype(float) - o["obs"]).max())
        lay = case.program.layout
        if lay.has("res_line", "loading_percent"):
            got = _np(eng.column("res_line", "loading_percent")[b])
            exp = o["net"].res_line.loading_percent.to_numpy()
            ok = ~np.isnan(exp)
            worst["loading"] = max(worst["loading"], np.abs(got[ok] - exp[ok]).max())
    return worst
