"""BatchedOpfEnv host logic on the host-sim build (CPU tier): vector-env API,
sampling, auto-reset, determinism, sharding invariance, reference-style identities."""
import numpy as np
import pytest
import torch

from opfgym_b200 import envs
from opfgym_b200 import reward as R
from opfgym_b200.data_split import define_test_train_split
from opfgym_b200.engine import Engine
from tests.hostsim.harness import TorchHostSimEngine

KW = dict(engine_cls=TorchHostSimEngine, n_profile_steps=672, obs_dtype="float64")


def make(cls=envs.VoltageControl, n=6, **kw):
    args = dict(KW, train_data="full_uniform", test_data="full_uniform", seed=3)
    args.update(kw)
    return cls(num_envs=n, **args)


def test_vector_env_api_shapes_and_types():
    env = make()
    assert env.num_envs == 6
    assert env.single_observation_space.shape == (442,) and env.single_action_space.shape == (14,)
    assert env.observation_space.shape == (6, 442) and env.action_space.shape == (6, 14)
    obs, info = env.reset(seed=1)
    assert obs.shape == (6, 442) and isinstance(info, dict) and not torch.isnan(obs).any()
    act = torch.rand(6, 14, dtype=torch.float64)
    obs2, reward, term, trunc, info = env.step(act)
    assert obs2.shape == (6, 442) and reward.shape == (6,)
    assert term.all() and not trunc.any()                       # steps_per_episode == 1
    for key in ("valids", "violations", "unscaled_penalties", "cost", "converged", "final_obs"):
        assert key in info
    assert info["valids"].shape == (6, len(env.constraints))
    assert not torch.equal(obs2, info["final_obs"])             # same-step auto-reset happened
    assert not torch.isnan(reward).any()
    env.step(act.numpy().astype(np.float32))                    # numpy / float32 actions accepted
    # a NaN action is data, not a crash: that env alone comes back non-converged with NaN reward
    bad = torch.rand(6, 14, dtype=torch.float64)
    bad[2, 3] = float("nan")
    _, reward, term, _, info = env.step(bad)
    assert info["converged"].tolist() == [True, True, False, True, True, True]
    assert torch.isnan(reward[2]) and not torch.isnan(reward[[0, 1, 3, 4, 5]]).any()
    assert (info["violations"][2] == 1).all() and not info["valids"][2].any()   # opf_env.py:395-398
    strict = make(validate_actions=True)
    strict.reset(seed=1)
    with pytest.raises(AssertionError):                           # opf_env.py:382
        strict.step(torch.full((6, 14), float("nan"), dtype=torch.float64))


def test_sampled_state_within_bounds_and_hook_columns():
    env = make(envs.QMarket, n=32)
    env.reset(seed=5)
    for table, column in (("load", "p_mw"), ("load", "q_mvar"), ("sgen", "p_mw")):
        df = env.net[table]
        v = env.col(table, column) * env.static(table, "scaling")
        assert (v >= env.static(table, "min_min_" + column) - 1e-12).all()
        assert (v <= env.static(table, "max_max_" + column) + 1e-12).all()
    price = env.col("poly_cost", "cq2_eur_per_mvar2")
    assert (price >= 0).all() and (price <= 0.03).all() and price.std() > 0
    # the reactive range is only computed for the rows an action reads it from (row-level pruning;
    # keep_all_columns=True materialises every row the reference's hook writes)
    ctrl = env.positions("sgen", env.act_keys[0][2])
    q_max = env.col("sgen", "max_q_mvar")[:, ctrl]
    assert torch.isfinite(q_max).all() and (q_max > 0).all()
    assert torch.allclose(env.col("sgen", "min_q_mvar")[:, ctrl], -q_max)
    assert (env.col("sgen", "q_mvar") == 0).all()               # centre action of a symmetric range


def test_seed_determinism_and_sharding_invariance():
    a, b = make(n=8), make(n=8)
    oa, _ = a.reset(seed=11)
    ob, _ = b.reset(seed=11)
    assert torch.equal(oa, ob)
    act = torch.rand(8, 14, dtype=torch.float64)
    ra, rb = a.step(act), b.step(act)
    assert torch.equal(ra[0], rb[0]) and torch.equal(ra[1], rb[1])
    oc, _ = make(n=8).reset(seed=12)
    assert not torch.equal(oa, oc)
    # rank 1 of 2 with 4 envs == envs 4..7 of one rank with 8 (RNG keyed by global env id)
    shard = make(n=4, rank=1, world_size=2)
    os_, _ = shard.reset(seed=11)
    assert torch.equal(os_, oa[4:])
    rs = shard.step(act[4:])
    assert torch.equal(rs[1], ra[1][4:]) and torch.equal(rs[0], ra[0][4:])


def test_action_round_trip_identity():
    """reference tests/test_opf_env.py:63-72: allclose(random_action, get_current_actions())."""
    env = make(envs.MaxRenewable, n=16)
    env.reset(seed=2)
    act = torch.rand(16, env.single_action_space.shape[0], dtype=torch.float64)
    env._apply_actions(act)
    assert torch.allclose(env.get_current_actions(), act, atol=1e-9)


def test_power_flow_availability_and_getters():
    from opfgym_b200.opf_env import PowerFlowNotAvailable
    env = make(n=4)
    env.reset(seed=1)
    with pytest.raises(PowerFlowNotAvailable):
        env.get_objective()
    conv = env.run_power_flow()
    assert conv.all()
    assert env.get_objective().shape == (4,) and env.is_state_valid().shape == (4,)
    assert env.get_state().shape == (4, env.state_space.shape[0])
    valids, viol, pens = env.calculate_violations()
    assert valids.shape == viol.shape == pens.shape == (4, len(env.constraints))


def test_res_observations_run_a_power_flow_in_reset():
    env = make(envs.VoltageControl, n=4, add_res_obs=True)
    assert env.pf_for_obs
    obs, _ = env.reset(seed=4)
    n_base = 442
    assert obs.shape[1] > n_base
    vm = obs[:, n_base:n_base + 5]
    assert ((vm > 0.8) & (vm < 1.2)).all()
    # like pandapower, out-of-service lines between energised buses (the open ring ties) report ZERO loading: their
    # rows of ppc['branch'] are never written, so the current is 0 / |V| (NaN only next to a dropped bus) -- and the
    # observation stays free of NaN
    k = n_base + sum(len(i) for t, c, i in env.obs_keys[4:] if (t, c) != ("res_line", "loading_percent")
                     and env.obs_keys.index((t, c, i)) < [kk[:2] for kk in env.obs_keys].index(("res_line", "loading_percent")))
    n_line = len(env.net.line)
    loading = obs[0, k:k + n_line].numpy()
    off = ~env.net.line.in_service.to_numpy(bool)
    assert off.any() and (loading[off] == 0.0).all() and (loading[~off] > 0.0).all()
    assert not torch.isnan(obs).any()


def test_simbench_sampling_modes():
    env = make(envs.VoltageControl, n=8, train_data="simbench", test_data="simbench",
               n_profile_steps=4 * 672)     # week 0 = test, week 1 = validation, 2-3 = train
    env.reset(seed=9)
    steps = env.current_simbench_step
    assert steps.shape == (8,) and set(steps.tolist()) <= set(env.train_steps.tolist())
    prof = torch.as_tensor(env.profiles[("load", "p_mw")].to_numpy().copy())
    assert torch.allclose(env.col("load", "p_mw"), prof[steps])
    env.reset(seed=9, options={"test": True})
    assert set(env.current_simbench_step.tolist()) <= set(env.validation_steps.tolist())
    env.reset(options={"step": 17})
    assert (env.current_simbench_step == 17).all()
    noisy = make(envs.VoltageControl, n=8, train_data="noisy_simbench", test_data="simbench",
                 n_profile_steps=4 * 672)
    noisy.reset(seed=9)
    prof = torch.as_tensor(noisy.profiles[("load", "p_mw")].to_numpy().copy())
    ratio = noisy.col("load", "p_mw") / prof[noisy.current_simbench_step]
    assert (ratio >= 0.9 - 1e-9).all() and (ratio <= 1.1 + 1e-9).all() and ratio.std() > 0


def test_reward_function_selection_and_scaling_estimate():
    env = make(n=8, reward_function="replacement",
               reward_function_params=dict(valid_reward=0.5, penalty_weight=None))
    assert isinstance(env.reward_function, R.Replacement)
    env.reset(seed=1)
    _, reward, _, _, info = env.step(torch.rand(8, 14, dtype=torch.float64))
    valid = info["valids"].all(dim=1)
    pen = info["unscaled_penalties"].sum(dim=1)
    assert torch.allclose(reward[~valid], pen[~valid])           # invalid: objective replaced by 0
    # reward_scaling without parameters samples the engine (reference reward.py:33-38)
    env2 = make(n=16, reward_function="summation",
                reward_function_params=dict(reward_scaling="normalization",
                                            scaling_params=dict(num_samples=48)))
    sp = env2.reward_function.scaling_params
    assert np.isfinite(sp["objective_factor"]) and sp["std_objective"] > 0


def test_unknown_kwargs_and_unsupported_modes_raise():
    with pytest.raises(TypeError):
        make(penalty_weight=0.3)        # reference silently swallows this (A.6 quirk 12)
    with pytest.raises(NotImplementedError):
        make(add_time_obs=True)
    with pytest.raises(TypeError):
        make(power_flow_solver="runpp")     # must be a callable on the batched env (see test_batched_plugin_callables)


def test_episode_statistics_accumulate():
    env = make(n=8)
    env.reset(seed=1)
    env.reset_statistics()
    for _ in range(3):
        env.step(torch.rand(8, 14, dtype=torch.float64))
    s = env.episode_statistics()
    assert s["steps"] == 24 and s["converged"] == 24 and 3.0 <= s["mean_iterations"] <= 6.0
    assert len(s["violated_share"]) == len(env.constraints)


def test_data_split_matches_reference_anchors():
    test, val, train = define_test_train_split()
    assert test[0] == 0 and val[0] == 672          # reference tests/test_simbench.py:83-85
    assert len(set(test) & set(val)) == 0 and len(set(train) & set(test)) == 0
    assert len(test) + len(val) + len(train) == 24 * 4 * 366
    t2, v2, tr2 = define_test_train_split(test_share=1.0, validation_share=0.0)
    assert len(t2) == 35136 and len(v2) == 0 and len(tr2) == 0


@pytest.mark.parametrize("cls,n_obs,n_act", [(envs.VoltageControl, 442, 14), (envs.EcoDispatch, 201, 42),
                                             (envs.QMarket, 305, 10), (envs.LoadShedding, 386, 16),
                                             (envs.MaxRenewable, 172, 18)])
def test_benchmark_sizes_and_three_steps(cls, n_obs, n_act):
    """reference tests/test_benchmarks_integration.py + docs/source/benchmarks.rst:19-27."""
    env = make(cls, n=3)
    assert env.single_observation_space.shape == (n_obs,) and env.single_action_space.shape == (n_act,)
    obs, _ = env.reset(seed=0)
    for _ in range(3):
        obs, reward, term, trunc, info = env.step(torch.rand(3, n_act, dtype=torch.float64))
        assert obs.shape == (3, n_obs) and term.all() and info["converged"].all()
    assert envs.make(f"{cls.__name__}-v0", num_envs=2, **dict(KW, train_data="full_uniform",
                                                             test_data="full_uniform")).num_envs == 2


def test_normal_and_mixed_sampling():
    """opf_env.py:240-251, 286-315 (SURVEY.md §8f rank 3)."""
    env = make(n=2048, train_data="normal_around_mean", n_profile_steps=4 * 672,
               sampling_params={"relative_std": 0.3})
    env.reset(seed=3)
    df = env.net.load
    p = env.col("load", "p_mw")
    lo = torch.as_tensor((df.min_min_p_mw / df.scaling).to_numpy().copy())
    hi = torch.as_tensor((df.max_max_p_mw / df.scaling).to_numpy().copy())
    assert (p >= lo - 1e-12).all() and (p <= hi + 1e-12).all()
    inside = (p > lo + 1e-9) & (p < hi - 1e-9)
    col = 5
    want_sigma = 0.3 * float(hi[col] - lo[col]) ** 2              # quirk 9: range applied twice
    sample = p[:, col][inside[:, col]]
    assert abs(float(sample.std()) - want_sigma) < 0.35 * want_sigma or inside[:, col].float().mean() < 0.9
    mixed = make(n=4096, train_data="mixed", n_profile_steps=4 * 672)
    mixed.reset(seed=4)
    share = torch.bincount(mixed.sample_source, minlength=3).double() / 4096
    assert torch.allclose(share, torch.tensor([0.5, 0.25, 0.25], dtype=torch.float64), atol=0.03)
    prof = torch.as_tensor(mixed.profiles[("load", "p_mw")].to_numpy().copy())
    sb = mixed.sample_source == 0
    noise = mixed.col("load", "p_mw")[sb] / prof[mixed.current_simbench_step[sb]]
    assert (noise >= 0.9 - 1e-9).all() and (noise <= 1.1 + 1e-9).all()   # default noise_factor 0.1
    # a storage sampled exactly at its rated power makes the reference's VoltageControl hook take
    # sqrt(max_s^2 - (p + 1e-9)^2) of a negative number (envs/voltage_control.py:128-131): NaN Q
    # bounds there, and here -- such envs come back non-converged, all others solve
    nan_bounds = torch.isnan(mixed.col("storage", "max_q_mvar")).any(dim=1)
    obs, reward, term, _, info = mixed.step(torch.rand(4096, 14, dtype=torch.float64))
    assert info["converged"][~nan_bounds].all() and info["converged"].float().mean() > 0.7


def test_diff_objective_and_incremental_actions():
    """opf_env.py:150-153, 216, 497-498 (diff_objective) and :451-470 (diff_action_step_size)."""
    plain = make(n=6, add_res_obs=("voltage_magnitude",))
    diff = make(n=6, add_res_obs=("voltage_magnitude",), diff_objective=True)
    plain.reset(seed=5)
    diff.reset(seed=5)
    initial = plain.get_objective()                       # objective of the reset state (centre action)
    assert torch.allclose(diff.engine.objective_offset, initial)
    act = torch.rand(6, 14, dtype=torch.float64)
    _, r_plain, _, _, _ = plain.step(act)
    _, r_diff, _, _, _ = diff.step(act)
    w = plain.reward_function.penalty_weight
    assert torch.allclose(r_plain - r_diff, initial * (1 - w), atol=1e-12)
    # incremental set-points: a = 0.5 keeps the set-point, a = 1 moves it by step*(max-min), clamped
    inc = make(n=4, diff_action_step_size=0.25)
    inc.reset(seed=5)
    pos = inc.positions("sgen", inc.act_keys[0][2])
    q0 = inc.col("sgen", "q_mvar")[:, pos].clone()
    lo, hi = inc.col("sgen", "min_q_mvar")[:, pos].clone(), inc.col("sgen", "max_q_mvar")[:, pos].clone()
    scal = inc.static("sgen", "scaling")[pos]
    assert torch.allclose(q0 * scal, (lo + hi) / 2, atol=1e-12)   # reset: absolute centre action (:207)
    a = torch.full((4, 14), 0.5, dtype=torch.float64)
    inc._apply_actions(a)
    assert torch.allclose(inc.col("sgen", "q_mvar")[:, pos], q0)
    a[:] = 1.0
    inc._apply_actions(a)
    want = torch.minimum(0.25 * (hi - lo) + q0 * scal, hi) / scal
    assert torch.allclose(inc.col("sgen", "q_mvar")[:, pos], want, atol=1e-12)
    for _ in range(5):
        inc._apply_actions(a)
    assert torch.allclose(inc.col("sgen", "q_mvar")[:, pos] * scal, hi, atol=1e-12)   # clamped at max


def test_bus_wise_obs():
    """opf_env.py:535-536, 780-784, 806-810: loads at one bus are observed as their sum."""
    class Shared(envs.VoltageControl):
        def _define_opf(self, *a, **kw):
            net, profiles = super()._define_opf(*a, **kw)
            net.load.loc[net.load.index[:30], "bus"] = np.repeat(net.load.bus.to_numpy()[:10], 3)
            return net, profiles

    plain = make(Shared, n=5)
    agg = make(Shared, n=5, bus_wise_obs=True)
    o_plain, _ = plain.reset(seed=9)
    o_agg, _ = agg.reset(seed=9)
    net = plain.net
    buses = net.load.bus.to_numpy()
    groups = sorted(set(buses.tolist()))
    assert len(groups) < len(buses), "stand-in grid needs buses with several loads for this test"
    k_plain = k_agg = 0
    for (table, column, idxs) in plain.obs_keys:
        n = len(idxs)
        if table == "load":
            at = buses[np.asarray(idxs, int)]
            part = o_plain[:, k_plain:k_plain + n]
            want = torch.stack([part[:, torch.as_tensor(at == b)].sum(dim=1) for b in groups], dim=1)
            got = o_agg[:, k_agg:k_agg + len(groups)]
            assert torch.allclose(got.double(), want.double(), rtol=1e-6, atol=1e-7)
            k_agg += len(groups)
        else:
            assert torch.equal(o_agg[:, k_agg:k_agg + n], o_plain[:, k_plain:k_plain + n])
            k_agg += n
        k_plain += n
    assert o_agg.shape[1] == k_agg == agg.single_observation_space.shape[0]
    lo, hi = agg.single_observation_space.low, agg.single_observation_space.high
    assert (lo <= hi).all()
    # the means appended by add_mean_obs follow the grouped layout
    both = make(Shared, n=3, bus_wise_obs=True, add_mean_obs=True)
    o, _ = both.reset(seed=9)
    assert o.shape[1] == both.single_observation_space.shape[0]


def test_step_host_matches_step():
    """numpy-in / numpy-out step (pinned buffers, overlapped copies on the GPU) returns exactly what
    the tensor API returns."""
    a_env, b_env = make(n=5), make(n=5)
    a_env.reset(seed=21)
    b_env.reset(seed=21)
    for k in range(3):
        act = np.random.default_rng(k).random((5, 14))
        obs, reward, term, trunc, info = a_env.step(torch.as_tensor(act))
        h_obs, h_reward, h_term, h_trunc, h_info = b_env.step_host(act)
        assert isinstance(h_obs, np.ndarray) and h_obs.shape == (5, 442)
        np.testing.assert_array_equal(h_obs, obs.numpy())
        np.testing.assert_array_equal(h_reward, reward.numpy())
        np.testing.assert_array_equal(h_info["cost"], info["cost"].numpy())
        np.testing.assert_array_equal(h_info["converged"], info["converged"].numpy())
        assert h_term.all() and not h_trunc.any()
    # in-place use of the pinned action buffer
    b_env.host_actions[:] = 0.25
    a_env.step(torch.full((5, 14), 0.25, dtype=torch.float64))
    _, r_dev, _, _, _ = a_env.step(torch.full((5, 14), 0.5, dtype=torch.float64))
    b_env.step_host()
    b_env.host_actions[:] = 0.5
    _, r_host, _, _, _ = b_env.step_host()
    np.testing.assert_array_equal(r_host, r_dev.numpy())


FUSED_RESET_ENVS = [("VoltageControl", {}), ("LoadShedding", {}), ("EcoDispatch", {"initial_action": "random"}),
                    ("MaxRenewable", {}), ("QMarket", {}), ("LoadSheddingReconfiguration", {})]
FUSED_RESET_CASES = \
    [pytest.param(name, kw, 4, "host", id=f"{name}-kw{k}") for k, (name, kw) in enumerate(FUSED_RESET_ENVS)] + \
    [pytest.param(name, kw, n, "host", id=f"{name}-n{n}") for name, kw in FUSED_RESET_ENVS[:3] for n in (1, 129)] + \
    [pytest.param(name, kw, n, "cuda", id=f"{name}-n{n}-cuda", marks=pytest.mark.gpu)
     for name, kw in FUSED_RESET_ENVS for n in (1, 4, 129)]


@pytest.mark.parametrize("cls_name,kw,n,engine", FUSED_RESET_CASES)
def test_fused_reset_equals_kernel_sequence(request, cls_name, kw, n, engine):
    """opfg_reset_episode (one launch) vs the recorded sequence sampler / hook programs / initial
    action / set-points / observe: bit-identical state rows and observations, episode after episode.
    On CUDA the fused reset runs one 128-thread CTA per environment with the row in shared memory,
    where a wrong stage grouping is a race; the sequence is the separate CUDA kernels."""
    cls = getattr(envs, cls_name)
    if engine == "cuda":
        request.getfixturevalue("cuda_lib")
        kw = dict(kw, engine_cls=Engine, prefetch_reset=False)
    fused = make(cls, n=n, **kw)                     # automatic for the built-in envs at small batch sizes
    plain = make(cls, n=n, fused_reset=False, **kw)
    assert fused.fused_reset and not plain.fused_reset
    of, _ = fused.reset(seed=31)          # recorded
    op, _ = plain.reset(seed=31)
    assert torch.equal(of, op)
    n_act = fused.single_action_space.shape[0]
    for k in range(3):
        act = torch.rand(n, n_act, dtype=torch.float64, generator=torch.Generator().manual_seed(k)).to(fused.device)
        rf, rp = fused.step(act), plain.step(act)      # auto-reset: replayed by the fused kernel
        assert fused._reset_plans and not plain._reset_plans
        assert torch.equal(rf[0], rp[0]) and torch.equal(rf[1], rp[1])
        n_in = fused.program.layout.n_inputs
        same = lambda t: t.nan_to_num(nan=-7.0)      # cells that no kernel reads stay NaN (pruned hook rows)
        assert torch.equal(same(fused.engine.state[:, :n_in]), same(plain.engine.state[:, :n_in]))
        assert torch.equal(fused.engine.actions_reset, plain.engine.actions_reset)
    of, _ = fused.reset(seed=77)
    op, _ = plain.reset(seed=77)
    assert torch.equal(of, op)


def test_truncated_normal_noise_and_interpolation_samplers():
    """opf_env.py:304-308 (truncnorm), :349-353 (interpolate_steps), :360-363 (normal noise)."""
    env = make(n=2048, train_data="normal_around_mean", n_profile_steps=4 * 672,
               sampling_params={"relative_std": 0.3, "truncated": True})
    env.reset(seed=3)
    df = env.net.load
    lo = torch.as_tensor((df.min_min_p_mw / df.scaling).to_numpy().copy())
    hi = torch.as_tensor((df.max_max_p_mw / df.scaling).to_numpy().copy())
    mean = torch.as_tensor(df.mean_p_mw.to_numpy().copy())
    sigma = 0.3 * (hi - lo) ** 2
    z = (env.col("load", "p_mw") - mean) / sigma
    # scipy's truncnorm(a, b, loc, scale): the STANDARD normal is truncated to [a, b] = [min, max]
    assert (z >= lo - 1e-9).all() and (z <= hi + 1e-9).all()
    wide = (hi - lo) > 0.05
    assert z[:, wide].std() > 0

    noisy = make(n=4096, train_data="noisy_simbench", n_profile_steps=4 * 672,
                 sampling_params={"noise_factor": 0.05, "noise_distribution": "normal"})
    noisy.reset(seed=4, options={"step": 100})
    prof = noisy.profiles[("load", "p_mw")]
    data = torch.as_tensor(prof.to_numpy()[100].copy())
    pmin, pmax = torch.as_tensor(prof.to_numpy().min(axis=0)), torch.as_tensor(prof.to_numpy().max(axis=0))
    p = noisy.col("load", "p_mw")
    assert (p >= pmin - 1e-12).all() and (p <= pmax + 1e-12).all()
    col = int(torch.argmax(torch.minimum(data - pmin, pmax - data) / data.abs().clamp_min(1e-9)))   # least clipped
    rel = (p[:, col] - data[col]) / data[col].abs()
    assert abs(float(rel.mean())) < 0.01 and abs(float(rel.std()) - 0.05) < 0.01

    inter = make(n=64, train_data="noisy_simbench", n_profile_steps=4 * 672,
                 sampling_params={"noise_factor": 0.0, "interpolate_steps": True})
    inter.reset(seed=5, options={"step": 200})
    a, b = (torch.as_tensor(prof.to_numpy()[k].copy()) for k in (200, 201))
    p = inter.col("load", "p_mw")
    lo2, hi2 = torch.minimum(a, b), torch.maximum(a, b)
    assert (p >= lo2 - 1e-12).all() and (p <= hi2 + 1e-12).all()
    moved = (a - b).abs() > 1e-9
    r = ((p - b) / (a - b))[:, moved]                  # data*r + next*(1-r): one r per environment
    assert torch.allclose(r, r[:, :1].expand_as(r), atol=1e-9) and r[:, 0].std() > 0.1


def test_reset_power_flow_leaves_step_results_and_statistics_alone():
    """Round-1 advisor finding: with a power flow in reset (add_res_obs) the auto-reset used to
    overwrite the buffers `step` had just returned as aliases (copy_outputs=False) and to count the
    reset-state scores in the episode statistics."""
    outs = {}
    for copy_outputs in (True, False):
        env = make(add_res_obs=True, copy_outputs=copy_outputs, n=6)
        env.reset(seed=5)
        env.reset_statistics()
        act = torch.rand(6, 14, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
        for _ in range(3):
            obs, reward, term, trunc, info = env.step(act)
        outs[copy_outputs] = (reward.clone(), info["violations"].clone(), info["cost"].clone(),
                              info["iterations"].clone(), obs.clone())
        stats = env.episode_statistics()
        assert stats["steps"] == 6 * 3
        # the getters describe the LAST power flow, which is the reset one (opf_env.py:209-216)
        assert env.power_flow_available
        assert not torch.equal(env.get_objective(), env.engine.objective)
    for a, b in zip(outs[True], outs[False]):
        assert torch.equal(a.nan_to_num(nan=-7.0), b.nan_to_num(nan=-7.0))


def test_clipped_action_penalty_is_measured_against_the_clipped_action():
    """opf_env.py:429, 488-491: an out-of-range action is clipped first, so it costs nothing extra."""
    env = make(clipped_action_penalty=2.0, n=4)
    base = make(n=4)
    act = torch.full((4, 14), 1.5, dtype=torch.float64)
    for e in (env, base):
        e.reset(seed=9)
    r1 = env.step(act)[1]
    r0 = base.step(act)[1]
    assert torch.allclose(r1, r0, atol=1e-12)


def test_step_host_is_refused_where_it_would_skip_episode_logic():
    from opfgym_b200.multi_stage import MultiStageBatchedOpfEnv
    from opfgym_b200.security_constrained import SecurityConstrainedBatchedOpfEnv
    assert "step_host" in MultiStageBatchedOpfEnv.__dict__ and "step_host" in SecurityConstrainedBatchedOpfEnv.__dict__
    with pytest.raises(NotImplementedError):
        MultiStageBatchedOpfEnv.step_host(object())
    with pytest.raises(NotImplementedError):
        SecurityConstrainedBatchedOpfEnv.step_host(object())


def test_step_host_with_half_precision_host_observations():
    """Opt-in: the observation matrix crosses to the host as float16 (the transfer that bounds
    step_host on a multi-GPU box); values equal the float32 ones to half precision."""
    a = make(n=5, obs_dtype="float32")
    b = make(n=5, obs_dtype="float32", host_obs_dtype="float16")
    act = np.random.default_rng(0).uniform(0, 1, (5, 14)).astype(np.float32)
    for e in (a, b):
        e.reset(seed=4)
    oa, ra = a.step_host(act)[:2]
    ob, rb = b.step_host(act)[:2]
    assert ob.dtype == np.float16 and oa.dtype == np.float32
    np.testing.assert_allclose(ob.astype(np.float32), oa, rtol=1e-3, atol=1e-3)
    np.testing.assert_array_equal(ra, rb)


@pytest.mark.parametrize("mode", [dict(noise_factor=0.0), dict(noise_factor=0.1), dict(noise_factor=0.2, noise_distribution="normal"),
                                  dict(noise_factor=0.1, interpolate_steps=True)])
def test_profile_sampler_kernel_equals_the_tensor_formula(mode):
    """opfg_sample_profiles (one launch per profile table) against opf_env.py:317-372 written with
    tensor ops on the same Philox rows."""
    env = make(n=7, train_data="noisy_simbench", test_data="simbench", sampling_params=mode, n_profile_steps=4 * 672)
    env.reset(seed=9)
    env._episode, env._stream_in_episode = 40, 0
    env._set_simbench_state(**mode)
    got = {k: env.col(*k).clone() for k in env._prof_dev if env.program.layout.has(*k)}
    steps = env.current_simbench_step
    # the same draws, by hand
    env._stream_in_episode = 1                      # stream 1 chose the time steps
    B = env.num_envs
    r = None
    if mode.get("interpolate_steps"):
        r = torch.empty(B, 1, dtype=torch.float64)
        env.engine.philox_uniform(r, env.seed, env.first_env, env._next_stream())
    for key, (table, pmin, pmax, slots) in env._prof_dev.items():
        if slots is None:
            continue
        v = table[steps]
        if r is not None:
            v = v * r + table[(steps + 1).clamp(max=table.shape[0] - 1)] * (1.0 - r)
        nf, n = mode["noise_factor"], v.shape[1]
        if nf and mode.get("noise_distribution", "uniform") == "uniform":
            u = torch.empty(B, n, dtype=torch.float64)
            env.engine.philox_uniform(u, env.seed, env.first_env, env._next_stream())
            v = v * (u * 2 * nf + (1 - nf))
        elif nf:
            u = torch.empty(B, 2 * n, dtype=torch.float64)
            env.engine.philox_uniform(u, env.seed, env.first_env, env._next_stream())
            v = v + v.abs() * nf * torch.sqrt(-2.0 * torch.log1p(-u[:, :n])) * torch.cos(2.0 * np.pi * u[:, n:])
        want = torch.minimum(torch.maximum(v, pmin), pmax)
        torch.testing.assert_close(got[key], want, rtol=1e-13, atol=1e-15)


def test_batched_plugin_callables():
    """`power_flow_solver=` / `objective_function=` of the reference (opf_env.py:52-53, 70-84) in batched
    form: the callables receive the env (device tensors for all environments)."""
    calls = {"pf": 0, "obj": 0}

    def solver(env):                       # delegate to the built-in kernels, count the calls
        calls["pf"] += 1
        env.engine.pf_solve()

    def objective(env):                    # the built-in objective of VoltageControl: loss costs 0.03 eur/MW
        calls["obj"] += 1
        ext = env.col("res_ext_grid", "p_mw").sum(dim=1)
        ctrl_s = env.positions("sgen", env.net.poly_cost.element[env.net.poly_cost.et == "sgen"].to_numpy())
        ctrl_t = env.positions("storage", env.net.poly_cost.element[env.net.poly_cost.et == "storage"].to_numpy())
        sg = (env.col("sgen", "p_mw") * env.static("sgen", "scaling"))[:, ctrl_s].sum(dim=1)
        st = (env.col("storage", "p_mw") * env.static("storage", "scaling"))[:, ctrl_t].sum(dim=1)
        return 0.03 * (ext + sg - st)

    a = make(n=6)
    b = make(n=6, power_flow_solver=solver, objective_function=objective)
    act = torch.rand(6, 14, dtype=torch.float64, generator=torch.Generator().manual_seed(2))
    for e in (a, b):
        e.reset(seed=8)
    ra, rb = a.step(act), b.step(act)
    assert calls == {"pf": 1, "obj": 1}
    torch.testing.assert_close(rb[1], ra[1], rtol=1e-9, atol=1e-12)          # reward
    torch.testing.assert_close(rb[4]["cost"], ra[4]["cost"], rtol=1e-9, atol=1e-12)
    torch.testing.assert_close(rb[4]["final_obs"], ra[4]["final_obs"])
    with pytest.raises(TypeError):
        make(n=2, objective_function="costs")
    with pytest.raises(NotImplementedError):
        b.step_host(act.numpy())


@pytest.mark.parametrize("cls", [envs.VoltageControl, envs.EcoDispatch, envs.LoadShedding])
def test_tensor_objective_module_equals_kernel_objective(cls):
    """opfgym_b200.objective.get_pandapower_costs (tensor ops, the plug-in building block) against the
    objective kernel 5 computes -- poly and pwl costs, sampled prices, reference ordering."""
    from opfgym_b200 import objective as O
    env = make(cls, n=5)
    env.reset(seed=6)
    n_act = env.single_action_space.shape[0]
    e = env.engine
    e.actions.copy_(torch.rand(5, n_act, dtype=torch.float64, generator=torch.Generator().manual_seed(1)))
    e.step()
    costs = O.get_pandapower_costs(env)
    assert costs.shape == (5, 2 * len(env.net.poly_cost) + len(env.net.pwl_cost))
    assert len(O.cost_vector_layout(env.net)) == costs.shape[1]
    torch.testing.assert_close(-costs.sum(dim=1), e.objective, rtol=1e-12, atol=1e-12)
    plug = make(cls, n=5, objective_function=O.get_pandapower_costs)
    plug.reset(seed=6)
    act = torch.rand(5, n_act, dtype=torch.float64, generator=torch.Generator().manual_seed(1))
    base = make(cls, n=5)
    base.reset(seed=6)
    torch.testing.assert_close(plug.step(act)[1], base.step(act)[1], rtol=1e-10, atol=1e-12)


def test_engine_cls_is_a_gated_test_seam():
    """A CPU engine cannot be injected into the product path unnoticed (round-1 review): `engine_cls=` only
    accepts the CUDA engine or classes that mark themselves as test infrastructure."""
    from opfgym_b200.engine import Engine, check_engine_class

    class Sneaky(Engine):
        pass

    with pytest.raises(TypeError):
        check_engine_class(Sneaky)
    check_engine_class(Engine)
    check_engine_class(TorchHostSimEngine)


def test_failed_reset_states_are_resampled():
    """opf_env.py:209-214: a reset state whose power flow fails is sampled again (the reference recurses into
    reset()).  Batched: only the failed environments take the new draw; the others keep their state."""
    kw = dict(num_envs=48, add_res_obs=True, train_data="full_uniform", test_data="full_uniform", load_scaling=6.5,
              engine_cls=TorchHostSimEngine, seed=3, n_profile_steps=96)
    env = envs.VoltageControl(max_reset_resamples=0, **kw)
    env.reset(seed=1)
    first = env._results.converged.numpy().astype(bool).copy()
    first_loads = env.col("load", "p_mw").numpy().copy()
    assert 0.1 < first.mean() < 0.9                      # the operating point sits at the collapse boundary
    env = envs.VoltageControl(**kw)
    obs, _ = env.reset(seed=1)
    assert env._results.converged.numpy().all()
    loads = env.col("load", "p_mw").numpy()
    np.testing.assert_array_equal(loads[first], first_loads[first])          # good states untouched
    assert (loads[~first] != first_loads[~first]).any(axis=1).all()          # failed ones drawn again
    vm = env.col("res_bus", "vm_pu").numpy()
    assert np.isfinite(vm).all()


@pytest.mark.parametrize("env_name", ["VoltageControl", "QMarket", "EcoDispatch", "LoadShedding", "MaxRenewable"])
def test_reset_observation_written_by_the_sampler(env_name):
    _check_reset_observation_by_sampler(env_name, dict(engine_cls=TorchHostSimEngine), lambda t: t.numpy())


@pytest.mark.gpu
@pytest.mark.parametrize("env_name", ["VoltageControl", "EcoDispatch", "LoadShedding"])
def test_reset_observation_written_by_the_sampler_cuda(cuda_lib, env_name):
    _check_reset_observation_by_sampler(env_name, dict(prefetch_reset=False), lambda t: t.cpu().numpy())


def _check_reset_observation_by_sampler(env_name, kw, to_np):
    """From the second reset on, the uniform sampler writes the observation itself where that is provably the
    same thing (every observed cell is a sampled cell that nothing writes afterwards) and `opfg_observe` is
    skipped: the result must be what the gather produces, bit for bit."""
    cls = getattr(envs, env_name)
    env = cls(num_envs=7, train_data="full_uniform", test_data="full_uniform", seed=11, n_profile_steps=96,
              fused_reset=False, **kw)
    plain = cls(num_envs=7, train_data="full_uniform", test_data="full_uniform", seed=11, n_profile_steps=96,
                fused_reset=False, fuse_reset_obs=False, **kw)
    took_shortcut = []
    calls = []
    real_observe = env.engine.observe
    env.engine.observe = lambda: (calls.append(1), real_observe())[1]
    for episode in range(4):
        del calls[:]
        obs, _ = env.reset(seed=20 + episode)
        used = len(calls)
        ref, _ = plain.reset(seed=20 + episode)
        np.testing.assert_array_equal(to_np(obs), to_np(ref))
        gathered = env.engine.obs.clone()
        real_observe()                                    # the gather, on the same state
        np.testing.assert_array_equal(to_np(gathered), to_np(env.engine.obs))
        took_shortcut.append(used)
    assert not plain._obs_by_sampler
    assert took_shortcut[0] == 1                          # the first reset gathers (and decides)
    assert took_shortcut[1:] == [0 if env._obs_by_sampler else 1] * 3
    # which envs qualify is a property of their observation keys; VoltageControl (loads and sgens only) must
    if env_name == "VoltageControl":
        assert env._obs_by_sampler
