"""Known-answer cases of the reference's own scoring tests (SURVEY.md App. C.1-C.3:
tests/test_constraints.py, tests/test_objective.py, tests/test_reward.py), replayed on
(a) the CPU oracle (oracle/scoring.py) and (b) the product's scalar host mirror; plus
the randomised fixture produced by the reference's own modules."""
import io
import lzma

import numpy as np
import pandas as pd
import pytest

from opfgym_b200 import constraints as C
from opfgym_b200 import net as pn
from opfgym_b200 import reward as R
from oracle import scoring
from tests import golden_scoring_util as gs


@pytest.fixture
def net():
    """Shape of pandapower's ``example_simple`` as far as scoring needs it."""
    net = pn.create_empty_network()
    pn.create_buses(net, 7, 20.0)
    pn.create_lines_from_parameters(net, [0, 1, 2, 3], [1, 2, 3, 4], 1.0, 0.1, 0.1, 10.0, 0.4)
    pn.create_transformer_from_parameters(net, 5, 6, 25.0, 110.0, 20.0, 0.41, 12.0, 14.0, 0.07)
    pn.create_ext_grid(net, 0)
    pn.create_load(net, 3, 2.0, 4.0)
    pn.create_sgen(net, 4, 2.0, -0.5)
    pn.create_gen(net, 2, 6.0, 1.03)
    net.res_bus = pd.DataFrame({"vm_pu": np.ones(7)})
    net.res_line = pd.DataFrame({"loading_percent": np.full(4, 30.0)})
    net.res_trafo = pd.DataFrame({"loading_percent": [40.0]})
    net.res_ext_grid = pd.DataFrame({"p_mw": [1.0], "q_mvar": [0.5]})
    for t in ("load", "sgen", "gen"):
        net["res_" + t] = pd.DataFrame({"p_mw": [1.0], "q_mvar": [0.5]})
    return net


# ---------------------------------------------------------------- C.1 constraints
def test_voltage_constraint(net):       # reference tests/test_constraints.py:17-30
    con = C.VoltageConstraint(autoscale_violation=False, only_worst_case_violations=True)
    net.bus["min_vm_pu"], net.bus["max_vm_pu"] = 0.95, 1.05
    net.res_bus["vm_pu"] = 1.0
    net.res_bus.at[0, "vm_pu"] = 0.9
    net.res_bus.at[1, "vm_pu"] = 0.94
    r = scoring.violation_metrics(con, net)
    assert not r["valid"] and np.isclose(r["violation"], 0.05) and np.isclose(r["penalty"], -0.05)


def test_line_and_trafo_overload(net):  # :32-56
    net.line["max_loading_percent"] = 100
    net.res_line["loading_percent"] = 50.0
    net.res_line.at[0, "loading_percent"] = 110.0
    r = scoring.violation_metrics(C.LineOverloadConstraint(autoscale_violation=False, penalty_factor=2.0), net)
    assert not r["valid"] and r["violation"] == 10 and r["penalty"] == -20
    net.trafo["max_loading_percent"] = 100
    net.res_trafo.at[0, "loading_percent"] = 110.0
    r = scoring.violation_metrics(C.TrafoOverloadConstraint(autoscale_violation=False, penalty_power=2.0), net)
    assert not r["valid"] and r["violation"] == 10 and r["penalty"] == -100


def test_ext_grid_constraints(net):     # :58-78
    net.ext_grid["min_p_mw"] = 0
    net.res_ext_grid.at[0, "p_mw"] = -0.5
    r = scoring.violation_metrics(C.ExtGridActivePowerConstraint(autoscale_violation=0.5), net)
    assert not r["valid"] and r["violation"] == 0.25 and r["penalty"] == -0.25
    net.ext_grid["min_q_mvar"] = 0
    net.res_ext_grid.at[0, "q_mvar"] = -0.5
    r = scoring.violation_metrics(C.ExtGridReactivePowerConstraint(autoscale_violation=0.5), net)
    assert not r["valid"] and r["violation"] == 0.25 and r["penalty"] == -0.25


def test_create_default_constraints(net):   # :80-128
    assert len(C.create_default_constraints(net, {})) == 0
    net.bus["min_vm_pu"], net.bus["max_vm_pu"] = 0.95, 1.05
    assert [type(c) for c in C.create_default_constraints(net, {})] == [C.VoltageConstraint]
    net.line["max_loading_percent"] = 100
    assert len(C.create_default_constraints(net, {})) == 2
    net.trafo["max_loading_percent"] = 100
    assert len(C.create_default_constraints(net, {})) == 3
    net.ext_grid["min_p_mw"] = 0
    assert len(C.create_default_constraints(net, {})) == 4
    net.ext_grid["min_q_mvar"] = 0
    found = C.create_default_constraints(net, {})
    assert len(found) == 5 and isinstance(found[-1], C.ExtGridReactivePowerConstraint)
    net.ext_grid["min_q_mvar"], net.ext_grid["max_q_mvar"] = -np.inf, np.inf
    net.ext_grid["min_p_mw"], net.ext_grid["max_p_mw"] = np.nan, np.nan
    net.bus["min_vm_pu"], net.bus["max_vm_pu"] = None, None
    kinds = [type(c) for c in C.create_default_constraints(net, {})]
    assert kinds == [C.LineOverloadConstraint, C.TrafoOverloadConstraint]


def test_custom_constraint(net):            # :131-147, callable replaced by value_scale
    con = C.Constraint("sgen", "p_mw", value_scale=0.5)
    net.sgen["scaling"] = 1.0
    net.sgen["min_p_mw"] = 0.0
    net.sgen["max_p_mw"] = 1.0
    net.res_sgen["p_mw"] = 1.5
    assert scoring.violation_metrics(con, net)["valid"]
    net.res_sgen["p_mw"] = 3.0
    r = scoring.violation_metrics(con, net)
    assert not r["valid"] and r["violation"] == 0.5
    with pytest.raises(ValueError):             # a callable constraint needs both callables
        C.Constraint("sgen", "p_mw", get_values=lambda env: None)


def test_custom_constraint_def_batched():   # reference tests/test_constraints.py:131-147 with BATCHED callables
    import torch
    from types import SimpleNamespace
    env = SimpleNamespace(xp=torch, device=torch.device("cpu"), num_envs=2,
                          res_sgen_p=torch.tensor([[1.5], [3.0]], dtype=torch.float64),
                          max_p=torch.tensor([1.0], dtype=torch.float64))
    con = C.Constraint("sgen", "p_mw", get_values=lambda env: env.res_sgen_p / 2,
                       get_boundaries=lambda env: {"min": 0, "max": env.max_p})
    assert con.is_batched_callable
    valid, violation, penalty = con.batched_metrics(env)
    assert valid.tolist() == [True, False]              # 1.5 / 2 = 0.75 inside [0, 1]; 3 / 2 - 1 = 0.5 outside
    assert violation.tolist() == [0.0, 0.5] and penalty.tolist() == [-0.0, -0.5]
    worst = C.Constraint("sgen", "p_mw", only_worst_case_violations=True, autoscale_violation=3.0, penalty_power=2.0,
                         penalty_factor=0.5, violation_count_penalty=0.25,
                         get_values=lambda env: torch.tensor([[0.0, 2.0, 4.0, -3.0]] * 2, dtype=torch.float64),
                         get_boundaries=lambda env: {"min": torch.tensor([-1.0] * 4), "max": 1.0})
    valid, violation, penalty = worst.batched_metrics(env)
    # worst upper violation 3 + worst lower violation 2, autoscale 3 -> 15; three violations
    assert not valid.any() and violation.tolist() == [15.0, 15.0]
    assert penalty.tolist() == [-(15.0 ** 2 * 0.5 + 3 * 0.25)] * 2


# ------------------------------------------------------------------ C.2 objective
def test_piecewise_linear_costs(net):       # reference tests/test_objective.py:30-51
    pts = [[0, 1, 30], [1, 2, 50]]
    pn.create_pwl_cost(net, 0, "load", pts, power_type="p")
    net.res_load.loc[0, "p_mw"] = 1.5
    assert scoring.pwl_costs(net).sum() == 55
    pn.create_pwl_cost(net, 0, "load", pts, power_type="q")
    net.res_load.loc[0, "q_mvar"] = 2.0
    assert scoring.pwl_costs(net).sum() == 55 + 80
    pn.create_pwl_cost(net, 0, "gen", pts, power_type="p")
    net.res_gen.loc[0, "p_mw"] = 0.5
    assert scoring.pwl_costs(net).sum() == 55 + 80 + 15


def test_pwl_negative_segment_and_undefined_sign(net):   # :45-51 (own net: zip truncation)
    pn.create_pwl_cost(net, 0, "gen", [[-1, 0, 40], [0, 1, 30], [1, 2, 50]], power_type="q")
    net.res_gen.loc[0, "q_mvar"] = -0.5
    assert scoring.pwl_costs(net).sum() == -20
    net2 = net.deepcopy()
    net2.pwl_cost = net2.pwl_cost.iloc[0:0]
    pn.create_pwl_cost(net2, 0, "sgen", [[0, 1, 30], [1, 2, 50]], power_type="p")
    net2.res_sgen.loc[0, "p_mw"] = -0.5
    assert scoring.pwl_costs(net2).sum() == 0


def test_polynomial_costs(net):             # :65-88
    pn.create_poly_cost(net, 0, "load", cp1_eur_per_mw=2)
    net.res_load.loc[0, ["p_mw", "q_mvar"]] = [1.5, 2.0]
    assert scoring.poly_costs(net).sum() == 3
    pn.create_poly_cost(net, 0, "sgen", cp1_eur_per_mw=2, cq1_eur_per_mvar=2)
    net.res_sgen.loc[0, ["p_mw", "q_mvar"]] = [1.2, 2.0]
    np.testing.assert_array_equal(scoring.poly_costs(net), [3.0, 2.4, 0, 4.0])
    net.poly_cost.loc[0, "cp0_eur"] = 1
    net.poly_cost.loc[1, "cq2_eur_per_mvar2"] = 2
    np.testing.assert_array_equal(scoring.poly_costs(net), [4.0, 2.4, 0, 12.0])
    pn.create_pwl_cost(net, 0, "load", [[0, 1, 30], [1, 2, 50]], power_type="p")
    np.testing.assert_array_equal(scoring.pandapower_costs(net), [4.0, 2.4, 0, 12.0, 55.0])
    empty = pn.create_empty_network()
    assert scoring.pandapower_costs(empty).shape == (0,)


# --------------------------------------------------------------------- C.3 reward
@pytest.mark.parametrize("call", ["mirror", "oracle"])
def test_reward_known_answers(call):        # reference tests/test_reward.py:8-78
    def ev(rf, penalty, objective, valid):
        return rf(objective, penalty, valid) if call == "mirror" else scoring.reward(rf, objective, penalty, valid)
    rf = R.Summation(clip_range=(0.0, 1.0))
    assert rf.clip_reward(1.5) == 1.0 and rf.clip_reward(-1.5) == 0.0
    rf = R.Summation(penalty_weight=0.8)
    assert rf.compute_total_reward(penalty=1.0, objective=0.0) == 0.8
    assert np.isclose(rf.compute_total_reward(penalty=0.5, objective=1.0), 0.6)
    rf = R.Summation(penalty_weight=None)
    assert rf.compute_total_reward(penalty=1.0, objective=0.2) == 1.2
    sp = {"min_objective": 2.0, "max_objective": 10.0, "min_penalty": 0.0, "max_penalty": 5.0}
    rf = R.Summation(reward_scaling="minmax11", scaling_params=dict(sp))
    assert [rf.scale_objective(v) for v in (6.0, 2.0, 10.0)] == [0.0, -1.0, 1.0]
    assert [rf.scale_penalty(v) for v in (2.5, 0.0, 5.0)] == [0.0, -1.0, 1.0]
    rf = R.Summation(reward_scaling="minmax01", scaling_params=dict(sp))
    assert [rf.scale_objective(v) for v in (6.0, 2.0, 10.0)] == [0.5, 0.0, 1.0]
    assert [rf.scale_penalty(v) for v in (2.5, 0.0, 5.0)] == [0.5, 0.0, 1.0]
    rf = R.Summation(reward_scaling="normalization", scaling_params={
        "std_objective": 2.0, "mean_objective": 6.0, "std_penalty": 1.0, "mean_penalty": 2.5})
    assert [rf.scale_objective(v) for v in (6.0, 2.0, 8.0)] == [0.0, -2.0, 1.0]
    assert [rf.scale_penalty(v) for v in (2.5, 1.5, 4.5)] == [0.0, -1.0, 2.0]
    rf = R.Summation(penalty_weight=None)
    assert ev(rf, -1.0, 0.0, True) == -1.0 and ev(rf, -0.5, 1.0, False) == 0.5 and ev(rf, 0.0, 0.8, True) == 0.8
    rf = R.Replacement(valid_reward=0.5, penalty_weight=None)
    assert ev(rf, 0.0, 0.2, True) == 0.7 and ev(rf, -0.3, 0.2, False) == -0.3 and ev(rf, 0.0, 0.2, False) == 0.0
    rf = R.Parameterized(valid_reward=0.7, invalid_penalty=0.3, invalid_objective_share=0.5, penalty_weight=None)
    assert np.isclose(ev(rf, 0.0, 0.2, True), 0.9) and np.isclose(ev(rf, -0.3, 0.2, False), -0.5)
    assert R.load_reward_class("summation") is R.Summation
    assert R.load_reward_class("Replacement") is R.Replacement
    with pytest.raises(AttributeError):
        R.load_reward_class("nope")


# -------------------------------------------- randomised cases from the reference modules
def _cases():
    with lzma.open(gs.__file__.replace("golden_scoring_util.py", "golden/scoring_cases.npz.xz")) as f:
        z = np.load(io.BytesIO(f.read()))
    return z, int(z["n_cases"])


def test_oracle_matches_reference_modules_on_random_tables():
    z, n = _cases()
    for k in range(n):
        net = gs.load_net(z, f"case{k}")
        ckw = gs.CONSTRAINT_KW[k % len(gs.CONSTRAINT_KW)]
        rname, rkw = gs.REWARD_SPECS[k % len(gs.REWARD_SPECS)]
        cons = C.create_default_constraints(net, dict(ckw))
        assert [type(c).__name__ for c in cons] == list(z[f"case{k}/constraint_names"]), k
        np.testing.assert_allclose(scoring.pandapower_costs(net), z[f"case{k}/costs"], rtol=1e-12, atol=1e-12)
        rf = getattr(R, rname)(**{kk: (dict(v) if isinstance(v, dict) else v) for kk, v in rkw.items()})
        out = scoring.step_reward(net, cons, rf)
        np.testing.assert_array_equal(out["valids"], z[f"case{k}/valids"])
        np.testing.assert_allclose(out["violations"], z[f"case{k}/violations"], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(out["unscaled_penalties"], z[f"case{k}/penalties"], rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(out["reward"], float(z[f"case{k}/reward"]), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(out["cost"], float(z[f"case{k}/cost"]), rtol=1e-12, atol=1e-12)
        # scalar host mirror of the kernel epilogue agrees as well
        mirror = rf(out["objective"], out["penalty"], out["valid"])
        np.testing.assert_allclose(mirror, float(z[f"case{k}/reward"]), rtol=1e-12, atol=1e-12)
        np.testing.assert_allclose(rf.calculate_cost(out["penalty"], out["valid"]),
                                   float(z[f"case{k}/cost"]), rtol=1e-12, atol=1e-12)
