"""The drop-in boundary: the reference env's step loop with this repo's power flow handed in as its constructor
argument `power_flow_solver=` (opfgym/opf_env.py:53,70,657) must reproduce what the reference computed with its
default power flow.

What the reference computed is stored in tests/golden/env_{VoltageControl,EcoDispatch}.npz (made by
tests/golden/make_golden.py from the unmodified reference): the state after each reset, the action, and the
outputs of `step`.  Here the net of the oracle env port (oracle/env_port.py, the reference's `_apply_actions`,
observation and scoring restated) takes that state and action, `adapter.PowerFlowSolver` solves it, and the
power-flow results, observation, reward and constraint info must match the stored ones."""
import numpy as np
import pytest

from opfgym_b200 import adapter
from opfgym_b200.net import LoadflowNotConverged
from oracle import env_port, scoring
from tests import golden_util as gu


def _run(name, **solver_kwargs):
    z, kwargs = gu.load(name)
    assert kwargs == {}, kwargs                       # the env port builds the default configuration
    env = env_port.OracleEnv(name, seed=7, n_profile_steps=gu.PROFILE_STEPS)
    net = env.net
    solver = adapter.PowerFlowSolver(net, **solver_kwargs)
    n = z["out/action"].shape[0]
    for i in range(n):
        for key in z.files:                           # the reference's net after reset
            if key.startswith("col/") and not key.endswith("/points") and z[key].shape[1]:
                _, table, column = key.split("/")
                v = z[key][i]
                net[table][column] = v.astype(net[table][column].dtype) if column in net[table] else v
        if name == "EcoDispatch":                     # eco_dispatch.py:121-123: points follow the sampled price
            for idx in net.pwl_cost.index:
                net.pwl_cost.at[idx, "points"] = [[0, 10000, net.pwl_cost.at[idx, "cp1_eur_per_mw"]]]
        env._apply_actions(z["out/action"][i])
        solver(net)
        assert net.converged, (name, i)
        label = f"{name} sample {i}"
        np.testing.assert_allclose(net.res_bus.vm_pu, z["out/vm_pu"][i], rtol=0, atol=1e-6, err_msg=label)
        np.testing.assert_allclose(net.res_bus.va_degree, z["out/va_degree"][i], rtol=0, atol=1e-5, err_msg=label)
        np.testing.assert_allclose(net.res_line.loading_percent, z["out/line_loading"][i], rtol=0, atol=1e-4,
                                   err_msg=label)
        np.testing.assert_allclose(net.res_trafo.loading_percent, z["out/trafo_loading"][i], rtol=0, atol=1e-4,
                                   err_msg=label)
        np.testing.assert_allclose(net.res_ext_grid.p_mw, z["out/ext_p"][i], rtol=0, atol=1e-6, err_msg=label)
        np.testing.assert_allclose(net.res_ext_grid.q_mvar, z["out/ext_q"][i], rtol=0, atol=1e-6, err_msg=label)
        out = scoring.step_reward(net, env.constraints, env.reward_function)
        np.testing.assert_allclose(env._obs(), z["out/obs"][i], rtol=0, atol=1e-6, err_msg=label)
        np.testing.assert_allclose(out["reward"], z["out/reward"][i], rtol=0, atol=1e-8, err_msg=label)
        np.testing.assert_allclose(out["cost"], z["out/cost"][i], rtol=0, atol=1e-8, err_msg=label)
        np.testing.assert_array_equal(out["valids"], z["out/valids"][i], err_msg=label)
        np.testing.assert_allclose(out["violations"], z["out/violations"][i], atol=1e-7, err_msg=label)
        np.testing.assert_allclose(out["unscaled_penalties"], z["out/penalties"][i], atol=1e-7, err_msg=label)
    # the reference's flag mapping: a diverging state raises LoadflowNotConverged, which makes its
    # run_power_flow() return False (opf_env.py:656-662)
    net.load["p_mw"] *= 500.0
    with pytest.raises(LoadflowNotConverged):
        solver(net)
    assert not net.converged
    return n


def test_reference_env_with_plugged_power_flow_hostsim():
    from tests.hostsim.harness import TorchHostSimEngine
    for name in ("VoltageControl", "EcoDispatch"):
        assert _run(name, engine_cls=TorchHostSimEngine) >= 3


@pytest.mark.gpu
def test_reference_env_with_plugged_power_flow_cuda(cuda_lib):
    for name in ("VoltageControl", "EcoDispatch"):
        assert _run(name) >= 3
