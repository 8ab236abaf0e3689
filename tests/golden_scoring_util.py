"""(De)serialisation of the small random nets of tests/golden/scoring_cases.npz.xz and
the parameter sets cycled through by its generator."""
import numpy as np
import pandas as pd

from opfgym_b200 import net as pn

TABLES = ("bus", "line", "trafo", "ext_grid", "load", "sgen", "storage", "gen", "poly_cost",
          "res_bus", "res_line", "res_trafo", "res_ext_grid", "res_load", "res_sgen",
          "res_storage", "res_gen")
ET = ["load", "sgen", "storage", "gen", "ext_grid"]

CONSTRAINT_KW = [
    {},
    {"only_worst_case_violations": True},
    {"penalty_factor": 2.0, "penalty_power": 2.0},
    {"violation_count_penalty": 0.25, "penalty_power": 0.5},
    {"autoscale_violation": False},
    {"autoscale_violation": 0.5, "only_worst_case_violations": True},
]
REWARD_SPECS = [
    ("Summation", {}),
    ("Summation", {"penalty_weight": None, "clip_range": (-2.0, 2.0)}),
    ("Replacement", {"valid_reward": 0.5, "penalty_weight": None}),
    ("Parameterized", {"valid_reward": 0.7, "invalid_penalty": 0.3, "invalid_objective_share": 0.5,
                       "penalty_weight": 0.25}),
    ("OnlyObjective", {}),
    ("Summation", {"reward_scaling": "minmax11",
                   "scaling_params": {"min_objective": -10.0, "max_objective": 5.0,
                                      "min_penalty": -20.0, "max_penalty": 0.0}}),
    ("Replacement", {"valid_reward": 1.0, "reward_scaling": "normalization",
                     "scaling_params": {"std_objective": 2.0, "mean_objective": -1.0,
                                        "std_penalty": 3.0, "mean_penalty": -2.0}}),
]


def dump_net(net, prefix):
    out = {}
    for t in TABLES:
        df = net[t]
        for c in df.columns:
            if df[c].dtype.kind in "fiub":
                out[f"{prefix}/{t}/{c}"] = df[c].to_numpy(float).copy()
            elif c == "et":
                out[f"{prefix}/{t}/{c}"] = np.array([ET.index(e) for e in df[c]], dtype=float)
    pw = net.pwl_cost
    out[f"{prefix}/pwl_cost/element"] = pw.element.to_numpy(float) if len(pw) else np.zeros(0)
    out[f"{prefix}/pwl_cost/et"] = np.array([ET.index(e) for e in pw.et], dtype=float)
    out[f"{prefix}/pwl_cost/is_p"] = np.array([pt == "p" for pt in pw.power_type], dtype=float)
    pts = np.array([p for p in pw.points], dtype=float) if len(pw) else np.zeros((0, 0, 3))
    out[f"{prefix}/pwl_cost/points"] = pts
    return out


def load_net(z, prefix):
    net = pn.create_empty_network()
    cols = {}
    for key in z.files:
        if key.startswith(prefix + "/"):
            parts = key.split("/")
            if len(parts) == 3:
                cols.setdefault(parts[1], {})[parts[2]] = z[key]
    for t in TABLES:
        if t in cols and t != "poly_cost":
            df = pd.DataFrame(cols[t])
            for c in ("bus", "from_bus", "to_bus", "hv_bus", "lv_bus"):
                if c in df:
                    df[c] = df[c].astype(int)
            for c in ("in_service",):
                if c in df:
                    df[c] = df[c].astype(bool)
            net[t] = df
    pc = cols.get("poly_cost", {})
    if pc and len(pc.get("element", [])):
        df = pd.DataFrame({k: v for k, v in pc.items()})
        df["et"] = [ET[int(e)] for e in pc["et"]]
        df["element"] = df["element"].astype(int)
        net.poly_cost = df
    pw = cols["pwl_cost"]
    for i in range(len(pw["element"])):
        pn.create_pwl_cost(net, int(pw["element"][i]), ET[int(pw["et"][i])],
                           pw["points"][i].tolist(), power_type="p" if pw["is_p"][i] else "q")
    return net
