#!/usr/bin/env python
"""Generate tests/golden/scoring_cases.npz.xz: outputs of the reference's OWN
``opfgym/objective.py``, ``opfgym/constraints.py`` and ``opfgym/reward.py``
(imported unmodified from /root/reference, pandapower stubbed for the type hint
only) on random result tables.  Run from the repo root in the build container."""
import io
import lzma
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)

N_CASES = 48


def random_net(rng, pn):
    import pandas as pd
    net = pn.create_empty_network()
    nb = int(rng.integers(4, 9))
    pn.create_buses(net, nb, 20.0)
    nl, nt = int(rng.integers(2, 6)), int(rng.integers(1, 3))
    pn.create_lines_from_parameters(net, rng.integers(0, nb, nl), rng.integers(0, nb, nl), 1.0,
                                    0.1, 0.1, 10.0, 0.4)
    for _ in range(nt):
        pn.create_transformer_from_parameters(net, 0, 1, 40.0, 110.0, 20.0, 0.3, 16.0, 18.0, 0.05)
    pn.create_ext_grid(net, 0)
    for table, n in (("load", 3), ("sgen", 3), ("storage", 2), ("gen", 2)):
        for _ in range(n):
            if table == "gen":
                pn.create_gen(net, int(rng.integers(0, nb)), 1.0)
            else:
                getattr(pn, f"create_{table}")(net, int(rng.integers(0, nb)), 1.0, 0.5)
    for table in ("load", "sgen", "storage", "gen"):
        net[table]["scaling"] = rng.uniform(0.5, 2.0, len(net[table]))
    net.bus["min_vm_pu"] = rng.uniform(0.9, 1.0, nb)
    net.bus["max_vm_pu"] = rng.uniform(1.0, 1.1, nb)
    if rng.random() < 0.3:
        net.bus.loc[rng.integers(0, nb), "max_vm_pu"] = np.nan
    net.line["max_loading_percent"] = rng.uniform(40, 120, nl)
    net.trafo["max_loading_percent"] = rng.uniform(40, 120, nt)
    net.ext_grid["min_p_mw"] = rng.uniform(-2, 0, 1)
    net.ext_grid["max_p_mw"] = rng.uniform(0, 2, 1)
    net.ext_grid["min_q_mvar"] = rng.uniform(-1, 0, 1)
    net.ext_grid["max_q_mvar"] = rng.uniform(0, 1, 1)
    net.ext_grid["mean_p_mw"] = rng.uniform(0.5, 3.0, 1)
    net.ext_grid["mean_q_mvar"] = rng.uniform(0.5, 3.0, 1)
    net.res_bus = pd.DataFrame({"vm_pu": rng.uniform(0.88, 1.12, nb)}, index=net.bus.index)
    net.res_line = pd.DataFrame({"loading_percent": rng.uniform(0, 140, nl)}, index=net.line.index)
    net.res_trafo = pd.DataFrame({"loading_percent": rng.uniform(0, 140, nt)}, index=net.trafo.index)
    net.res_ext_grid = pd.DataFrame({"p_mw": rng.uniform(-3, 3, 1), "q_mvar": rng.uniform(-2, 2, 1)},
                                    index=net.ext_grid.index)
    for table in ("load", "sgen", "storage", "gen"):
        n = len(net[table])
        net["res_" + table] = pd.DataFrame({"p_mw": rng.uniform(-2.5, 2.5, n),
                                            "q_mvar": rng.uniform(-2.5, 2.5, n)}, index=net[table].index)
    for _ in range(int(rng.integers(0, 5))):
        et = str(rng.choice(["load", "sgen", "storage", "gen", "ext_grid"]))
        coef = rng.uniform(-2, 2, 6) * (rng.random(6) < 0.6)
        pn.create_poly_cost(net, int(rng.integers(0, len(net[et]))), et, cp0_eur=coef[0],
                            cp1_eur_per_mw=coef[1], cp2_eur_per_mw2=coef[2], cq0_eur=coef[3],
                            cq1_eur_per_mvar=coef[4], cq2_eur_per_mvar2=coef[5])
    n_seg = int(rng.integers(1, 4))
    for _ in range(int(rng.integers(0, 4))):
        et = str(rng.choice(["load", "sgen", "storage", "gen", "ext_grid"]))
        lo = float(rng.choice([-2.0, -1.0, 0.0]))
        edges = lo + np.cumsum(np.r_[0.0, rng.uniform(0.3, 1.5, n_seg)])
        if rng.random() < 0.3:
            edges = -edges[::-1]
        pts = [[edges[i], edges[i + 1], float(rng.uniform(-5, 50))] for i in range(n_seg)]
        pn.create_pwl_cost(net, int(rng.integers(0, len(net[et]))), et, pts,
                           power_type=str(rng.choice(["p", "q"])))
    return net


def main():
    import _ref_stubs
    _ref_stubs.install(profile_steps=96)
    import opfgym.constraints as rc
    import opfgym.objective as ro
    import opfgym.reward as rr
    from opfgym_b200 import net as pn
    from tests.golden_scoring_util import dump_net, CONSTRAINT_KW, REWARD_SPECS

    rng = np.random.default_rng(2024)
    arrays = {"n_cases": np.array(N_CASES)}
    for k in range(N_CASES):
        net = random_net(rng, pn)
        ckw = CONSTRAINT_KW[k % len(CONSTRAINT_KW)]
        rname, rkw = REWARD_SPECS[k % len(REWARD_SPECS)]
        cons = rc.create_default_constraints(net, dict(ckw))
        costs = ro.get_pandapower_costs(net)
        objective = float(np.sum(-costs))
        res = [c.get_violation_metrics(net) for c in cons]
        valids = np.array([bool(r["valid"]) for r in res])
        viol = np.array([float(r["violation"]) for r in res])
        pens = np.array([float(r["penalty"]) for r in res])
        rf = getattr(rr, rname)(**rkw)
        penalty, valid = float(pens.sum()), bool(valids.all())
        arrays.update(dump_net(net, f"case{k}"))
        arrays[f"case{k}/costs"] = np.asarray(costs, float)
        arrays[f"case{k}/valids"] = valids
        arrays[f"case{k}/violations"] = viol
        arrays[f"case{k}/penalties"] = pens
        arrays[f"case{k}/reward"] = np.array(float(rf(objective, penalty, valid)))
        arrays[f"case{k}/cost"] = np.array(float(rf.calculate_cost(penalty, valid)))
        arrays[f"case{k}/constraint_names"] = np.array([type(c).__name__ for c in cons])
    # an uncompressed npz under one xz stream: the ~5 000 small members share one dictionary, and their zip
    # headers and names compress away
    path = os.path.join(HERE, "scoring_cases.npz.xz")
    buf = io.BytesIO()
    np.savez(buf, **arrays)
    with lzma.open(path, "wb", preset=9 | lzma.PRESET_EXTREME) as f:
        f.write(buf.getvalue())
    print("wrote", path, os.path.getsize(path) // 1024, "KiB")


if __name__ == "__main__":
    main()
