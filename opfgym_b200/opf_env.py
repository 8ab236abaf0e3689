"""``BatchedOpfEnv``: thousands of instances of one OPF environment stepping in
lock-step on one GPU, behind the constructor and method surface of the
reference ``OpfEnv`` (``opfgym/opf_env.py:26-175``) and a gymnasium-style
vector-env interface (``num_envs``, ``single_*_space``, batched ``reset`` /
``step``, same-step auto-reset).

What happens where (reference ``step`` call stack, SURVEY.md §3.1):

===========================  ====================================================
reference (per env, pandas)  here (all envs, device)
===========================  ====================================================
``_sampling``                ``opfg_sample_uniform`` / profile gather + the
                             subclass hook written as tensor ops on column views
``_apply_actions``           kernel 1 (``opfg_assemble``)
``pp.runpp``                 kernels 2-4 (``opfg_pf_solve``)
``calculate_reward``         kernel 5 (``opfg_score``)
``_get_obs``                 kernel 5 epilogue / ``opfg_observe``
===========================  ====================================================

Differences from the reference, on purpose: unknown keyword arguments raise
instead of being swallowed (SURVEY.md §5); features that the reference itself
ships broken (``add_time_obs``, A.6 quirk 1) raise ``NotImplementedError``.
"""
from __future__ import annotations

import os

import copy

import numpy as np

from . import constraints as constraints_mod
from . import reward as reward_mod
from .compiler import Compiler
from .data_split import define_test_train_split
from .engine import Engine
from .ppc import PpcBuilder
from .spaces import Box, batch_space, get_obs_and_state_space

_SPLIT_KWARGS = {"test_share", "random_test_steps", "validation_share", "random_validation_steps"}


_BUILD_KWARGS = ("voltage_band", "max_loading", "storage_scaling", "n_profile_steps")


def split_build_kwargs(kwargs: dict) -> dict:
    """Pop the keyword arguments that the reference forwards through ``*args, **kwargs``
    to ``build_simbench_net`` (opfgym/simbench/build_simbench_net.py:5-7)."""
    return {k: kwargs.pop(k) for k in _BUILD_KWARGS if k in kwargs and kwargs[k] is not None}


class PowerFlowNotAvailable(Exception):
    pass


class BatchedOpfEnv:
    metadata = {"autoreset_mode": "same_step"}

    def __init__(self, net, action_keys, observation_keys, state_keys=None, profiles=None,
                 num_envs: int = 1,
                 evaluate_on: str = "validation", steps_per_episode: int = 1,
                 bus_wise_obs: bool = False,
                 reward_function="summation", reward_function_params: dict | None = None,
                 diff_objective: bool = False, add_res_obs=False, add_time_obs: bool = False,
                 add_act_obs: bool = False, add_mean_obs: bool = False,
                 train_data: str = "simbench", test_data: str = "simbench",
                 sampling_params: dict | None = None, constraint_params: dict | None = None,
                 custom_constraints: list | None = None, autoscale_actions: bool = True,
                 diff_action_step_size: float | None = None,
                 clipped_action_penalty: float = 0.0, initial_action: str = "center",
                 objective_function=None, power_flow_solver=None,
                 optimal_power_flow_solver=None, seed: int | None = None,
                 # --- engine-side arguments (not in the reference) ---
                 device=None, rank: int = 0, world_size: int = 1, obs_dtype: str = "float32",
                 dynamic_columns=(), pwl_price_columns=None, tolerance_mva: float = 1e-8,
                 max_iteration: int = 10, engine_cls=Engine, engine_kwargs: dict | None = None,
                 copy_outputs: bool = True, validate_actions: bool = False, host_obs_dtype: str | None = None,
                 prefetch_reset: bool = True, keep_all_columns: bool = False,
                 fused_reset: bool | None = None, max_reset_resamples: int = 8,
                 fuse_reset_obs: bool | None = None, **kwargs):
        unknown = set(kwargs) - _SPLIT_KWARGS
        if unknown:
            raise TypeError(f"unknown keyword arguments: {sorted(unknown)}")
        if add_time_obs:
            raise NotImplementedError("add_time_obs raises TypeError in the reference itself "
                                      "(opf_env.py:545-546 vs time_observation.py:4)")
        # The reference's plug-in points (opf_env.py:52-53, 70-84) in BATCHED form: the callables get the
        # env (all environments at once, device tensors) instead of one pandapower net.
        #   power_flow_solver(env)   -- replaces kernels 2-4: read env.engine.sbus [B, nb, 2] (and .yval),
        #                               fill env.engine.vm / .va [B, nb], .converged [B] u8, .iterations [B] i32
        #   objective_function(env)  -- replaces the poly / pwl costs of kernel 5: return the COSTS as a
        #                               tensor [B] or [B, k] (the objective is minus their sum, opf_env.py:493-500);
        #                               result columns are read with env.col("res_bus", "vm_pu") etc.
        for name, fn in (("objective_function", objective_function), ("power_flow_solver", power_flow_solver)):
            if fn is not None and not callable(fn):
                raise TypeError(f"{name} must be callable: {name}(env) on batched device tensors")
        self._custom_solver = power_flow_solver
        self._custom_objective = objective_function
        if steps_per_episode != 1 and not getattr(self, "_multi_step_ok", False):
            raise NotImplementedError("multi-step episodes: use opfgym_b200.multi_stage.MultiStageBatchedOpfEnv")

        self.net = net
        self.copy_outputs = copy_outputs   # False: returned tensors alias engine buffers
        # step_host only: dtype of the observation matrix on the HOST (None = the engine's obs dtype, float32
        # like the reference's Box).  The observation transfer is what bounds step_host on a multi-GPU box
        # (profiles/r02_d2h_probe_8gpu.txt); "float16" halves it for agents that consume half precision anyway.
        self.host_obs_dtype = host_obs_dtype
        # The reference asserts `not isnan(action)` (opf_env.py:382).  Checking on the host costs a
        # device sync per step; by default a NaN action simply propagates: that env comes back
        # non-converged with NaN reward/obs (its neighbours in the batch are unaffected).
        self.validate_actions = validate_actions
        self.max_reset_resamples = int(max_reset_resamples)
        self.num_envs = int(num_envs)
        self.profiles = profiles
        self.obs_keys = list(observation_keys)
        self.state_keys = list(state_keys) if state_keys is not None else copy.copy(self.obs_keys)
        self.act_keys = list(action_keys)
        if not profiles:
            assert "simbench" not in test_data and "simbench" not in train_data
        self.evaluate_on = evaluate_on
        self.train_data, self.test_data = train_data, test_data
        self.sampling_params = sampling_params or {}
        self.add_act_obs = add_act_obs
        if add_act_obs:
            self.obs_keys.extend(self.act_keys)
        if add_res_obs is True:
            add_res_obs = ("voltage_magnitude", "voltage_angle", "line_loading",
                           "trafo_loading", "ext_grid_power")
        if add_res_obs:   # opf_env.py:99-118
            buses = set(net.load.bus) | set(net.sgen.bus) | set(net.gen.bus) | set(net.storage.bus)
            buses = np.sort(list(buses))
            extra = {"voltage_magnitude": [("res_bus", "vm_pu", buses)],
                     "voltage_angle": [("res_bus", "va_degree", buses)],
                     "line_loading": [("res_line", "loading_percent", net.line.index)],
                     "trafo_loading": [("res_trafo", "loading_percent", net.trafo.index)],
                     "ext_grid_power": [("res_ext_grid", "p_mw", net.ext_grid.index),
                                        ("res_ext_grid", "q_mvar", net.ext_grid.index)]}
            for name in ("voltage_magnitude", "voltage_angle", "line_loading", "trafo_loading",
                         "ext_grid_power"):
                if name in add_res_obs:
                    self.obs_keys.extend(extra[name])
        self.add_mean_obs = add_mean_obs
        self.bus_wise_obs = bool(bus_wise_obs)
        self.observation_space_single = get_obs_and_state_space(
            net, self.obs_keys, False, add_mean_obs, seed=seed, bus_wise_obs=bus_wise_obs)
        self.state_space = get_obs_and_state_space(net, self.state_keys, seed=seed)
        n_actions = sum(len(idxs) for _, _, idxs in self.act_keys)
        self.single_action_space = Box(0, 1, shape=(n_actions,), seed=seed)
        self.single_observation_space = self.observation_space_single
        self.action_space = batch_space(self.single_action_space, self.num_envs)
        self.observation_space = batch_space(self.single_observation_space, self.num_envs)

        self.autoscale_actions = autoscale_actions
        self.clipped_action_penalty = clipped_action_penalty
        self.initial_action = initial_action
        self.steps_per_episode = steps_per_episode
        self.pf_for_obs = any("res_" in unit_type for unit_type, _, _ in self.obs_keys)
        self.diff_objective = bool(diff_objective)
        self.diff_action_step_size = diff_action_step_size
        if self.diff_objective:
            self.pf_for_obs = True      # opf_env.py:150-153: the initial objective needs a power flow
        self.test_steps, self.validation_steps, self.train_steps = define_test_train_split(**kwargs)

        if custom_constraints is None:
            self.constraints = constraints_mod.create_default_constraints(net, constraint_params or {})
        else:
            self.constraints = custom_constraints
        # constraints with batched callables (reference constraints.py:27-64 ``get_values`` / ``get_boundaries``,
        # examples/custom_constraint.py) are evaluated behind kernel 5; ``self.constraints`` keeps the ones the
        # kernel scores.  Their columns of valids / violations / unscaled_penalties FOLLOW the kernel's columns.
        self.batched_constraints = [c for c in self.constraints if getattr(c, "is_batched_callable", False)]
        self.constraints = [c for c in self.constraints if not getattr(c, "is_batched_callable", False)]
        if self.batched_constraints and type(self).step is not BatchedOpfEnv.step:
            raise NotImplementedError("callable constraints on an env with its own step() (multi-stage, N-1)")

        # ---- compile + device buffers ------------------------------------------------
        self.rank, self.world_size = int(rank), int(world_size)
        dyn_service = {t for t, c, _ in self.act_keys if c == "in_service" and t in ("line", "trafo")}
        dyn_service |= {t for t, c in dynamic_columns if c == "in_service" and t in ("line", "trafo")}
        # `switch.closed` as action / contingency cell (examples/network_reconfiguration.py:34): line-bus and
        # trafo-bus switches only -- a bus-bus switch would change the bus count
        sw_keys = [(t, c, i) for t, c, i in self.act_keys if (t, c) == ("switch", "closed")]
        if sw_keys or ("switch", "closed") in [tuple(tc) for tc in dynamic_columns]:
            dyn_service.add("switch")
            for _, _, idxs in sw_keys:
                if (net.switch.et.loc[list(idxs)] == "b").any():
                    raise NotImplementedError("bus-bus switches as actions change the bus count; only line-bus "
                                              "and trafo-bus switches can be switched per environment")
        self._builder = PpcBuilder(net, dynamic_service=tuple(sorted(dyn_service)))
        compiler = Compiler(net, self._builder)
        placeholder = reward_mod.Summation()
        dynamic = list(dynamic_columns) + list(self._dynamic_columns())
        self._compile_args = dict(act_keys=self.act_keys, obs_keys=self.obs_keys,
                                  state_keys=self.state_keys, constraints=self.constraints,
                                  extra_dynamic=dynamic, autoscale_actions=autoscale_actions,
                                  pwl_price_columns=pwl_price_columns,
                                  # hook-written columns that no kernel reads (they only feed the
                                  # reference's pandapower-OPF baseline) are not materialised
                                  prune_unused=not keep_all_columns,
                                  diff_action_step_size=diff_action_step_size,
                                  bus_wise_obs=bus_wise_obs)
        self._engine_args = dict(device=device, tolerance_mva=tolerance_mva,
                                 max_iteration=max_iteration, obs_dtype=obs_dtype,
                                 **(engine_kwargs or {}))
        from .engine import check_engine_class
        check_engine_class(engine_cls)
        self._engine_cls = engine_cls
        self.program = compiler.compile(reward_function=placeholder, **self._compile_args)
        self.pruned_columns = {tuple(tc) for tc in dynamic if not self.program.layout.has(*tc)}
        self.engine = engine_cls(self.program, self.num_envs, **self._engine_args)
        self.xp = self.engine.torch
        self.device = self.engine.device
        self.seed = 0 if seed is None else int(seed)
        self._episode = 0
        self._stream_in_episode = 0
        self._sample_cache = {}
        self._static_cache = {}
        self._row_programs = {}
        # reset observation written by the sampler itself (see `_plan_reset_observation`)
        self._program_writes = {}
        self._reset_log = []
        self._obs_by_sampler = False
        self._obs_sampler_plans = {}        # data distribution -> log of the reset the decision was taken on, or None
        self._sample_obs_pos = {}
        self._obs_cell_pos = None
        self._flags = None
        # Every step ends every episode, and the next episode's state depends only on the RNG: sample
        # it (sampler, hook programs, centre action, reset observation) on a side stream into a second
        # state buffer while the main stream solves the current episode.
        # Fused reset (one launch instead of sampler + hook programs + set-points + observe): the
        # first eligible reset is recorded, later ones replay the recording.  Only calls that go
        # through `_sample_keys` / `run_row_program` can be recorded, so hooks of user subclasses
        # (which may touch the state with arbitrary tensor code) have to opt in explicitly.
        # Measured on B200 (VoltageControl): one launch beats six up to ~1.5k environments (+40 % at
        # 64-512), the separate full-occupancy kernels win beyond that -- hence the automatic rule.
        self.fused_reset = (type(self).__module__.startswith("opfgym_b200.") and self.num_envs <= 1024) \
            if fused_reset is None else bool(fused_reset)
        self._fuse_reset_obs = type(self).__module__.startswith("opfgym_b200.") if fuse_reset_obs is None \
            else bool(fuse_reset_obs)
        self._reset_plans = {}
        self._prefetch = bool(prefetch_reset) and getattr(self.device, "type", "cpu") == "cuda" \
            and not self.pf_for_obs
        if self._prefetch:
            self.engine.enable_double_buffer()
            self._side = self.xp.cuda.Stream(device=self.device)
            self._copy_stream = self.xp.cuda.Stream(device=self.device)      # step_host: observation transfers
            self._pf_done = self.xp.cuda.Event()
            self._sampled_events = [self.xp.cuda.Event() for _ in range(3)]
            self._main_done = self.xp.cuda.Event()
            self._side_done = self.xp.cuda.Event()
            self._side_kernels = self.xp.cuda.Event()
            self._ready_events = (self.xp.cuda.Event(enable_timing=bool(os.environ.get("OPFG_TIMING_EVENTS"))), self.xp.cuda.Event(enable_timing=bool(os.environ.get("OPFG_TIMING_EVENTS"))))
            self._results_copied = self.xp.cuda.Event()
        self._pipe = None     # step_host's look-ahead: episode k+1 already sampled, its observation on the host
        self.test = False
        self.power_flow_available = False
        self._results = self.engine

        # ---- reward function (may sample the engine for its scaling parameters) --------
        reward_function_params = reward_function_params or {}
        if isinstance(reward_function, str):
            reward_cls = reward_mod.load_reward_class(reward_function)
            self.reward_function = reward_cls(env=self, **reward_function_params)
        elif isinstance(reward_function, reward_mod.RewardFunction):
            self.reward_function = reward_function
        else:
            raise TypeError("reward_function must be a name or an opfgym_b200.reward.RewardFunction")
        if repr(self.reward_function.device_params()) != repr(placeholder.device_params()):
            self._rebuild_engine()

    # subclasses list the per-environment columns their `_sampling` hook writes
    def _dynamic_columns(self):
        return ()

    def _rebuild_engine(self):
        state = self.engine.state
        compiler = Compiler(self.net, self._builder)
        self.program = compiler.compile(reward_function=self.reward_function, **self._compile_args)
        self.engine.close()
        self.engine = self._engine_cls(self.program, self.num_envs, **self._engine_args)
        self.engine.state.copy_(state)
        if getattr(self, "_prefetch", False):
            self.engine.enable_double_buffer()
        self._sample_cache.clear()
        self._row_programs.clear()
        self._reset_plans.clear()
        self._program_writes.clear()
        self._obs_sampler_plans.clear()
        self._sample_obs_pos.clear()
        self._obs_by_sampler = False

    # ------------------------------------------------------------------ column access
    def col(self, table: str, column: str):
        """[num_envs, n_rows] view of a per-environment column."""
        return self.engine.column(table, column)

    def static(self, table: str, column: str):
        key = (table, column)
        if key not in self._static_cache:
            v = np.asarray(self.net[table][column].to_numpy(), dtype=float)
            self._static_cache[key] = self.engine._from_numpy(v)
        return self._static_cache[key]

    def positions(self, table: str, idxs):
        return self.net[table].index.get_indexer(np.asarray(idxs))

    # ---------------------------------------------------------------- hook programs
    def run_row_program(self, name: str, table: str, build):
        """Run the row program ``name`` (compiled on first use from ``build(r)``, which
        writes the hook's formulas on a ``RowProgram``) for all environments: ONE launch."""
        from .rowprog import CompiledRowProgram, RowProgram
        key = (name, table)
        if key not in self._row_programs:
            if not len(self.net[table]):
                self._row_programs[key] = None
            else:
                rp = RowProgram(self, table)
                build(rp)
                # column-level pruning happened in `store`; row-level pruning here: only the cells some
                # kernel table reads are computed (VoltageControl: 14 of 198 sgen rows carry an action
                # and hence need their reactive range; the rest only need `q_mvar = 0`)
                live = self.program.read_cells if self._compile_args["prune_unused"] else None
                self._row_programs[key] = [CompiledRowProgram(self.engine, rp.n_rows, ops, statics, rows)
                                           for rows, ops, statics in rp.compile_groups(live)]
                self._program_writes[key] = [(start, rp.n_rows) for start, _ in rp.stores]
        self._reset_log.append(("program", key))
        for prog in self._row_programs[key] or ():
            prog.run()

    # ------------------------------------------------------------------------ sampling
    def _next_stream(self) -> int:
        self._stream_in_episode += 1
        return self._episode * 64 + self._stream_in_episode

    @property
    def first_env(self) -> int:
        return self.rank * self.num_envs

    def _sample_from_range(self, unit_type, column, idxs):
        """``OpfEnv._sample_from_range`` (opf_env.py:266-284) for all environments."""
        self._sample_keys([(unit_type, column, idxs)])

    def _sample_keys(self, keys):
        cache_key = tuple((t, c, tuple(np.asarray(i).tolist())) for t, c, i in keys)
        if cache_key not in self._sample_cache:
            slots, lo, hi, div = [], [], [], []
            for unit_type, column, idxs in keys:
                if "res_" in unit_type or len(idxs) == 0:
                    continue
                df = self.net[unit_type]
                pos = self.positions(unit_type, idxs)
                lo_c = f"min_min_{column}" if f"min_min_{column}" in df.columns else f"min_{column}"
                hi_c = f"max_max_{column}" if f"max_max_{column}" in df.columns else f"max_{column}"
                start = self.program.layout.columns[(unit_type, column)][0]
                slots.append(start + pos)
                lo.append(df[lo_c].to_numpy(float)[pos])
                hi.append(df[hi_c].to_numpy(float)[pos])
                div.append(df.scaling.to_numpy(float)[pos] if "scaling" in df.columns
                           else np.ones(len(pos)))
            if not slots:
                self._sample_cache[cache_key] = None
            else:
                f = self.engine._from_numpy
                self._sample_cache[cache_key] = (
                    f(np.concatenate(slots).astype(np.int32)), f(np.concatenate(lo)),
                    f(np.concatenate(hi)), f(np.concatenate(div)))
        plan = self._sample_cache[cache_key]
        if plan is not None:
            self._reset_log.append(("sample", cache_key))
            obs_pos = None
            if self._obs_by_sampler:         # the observation is made of sampled cells only: written on the way
                if cache_key not in self._sample_obs_pos:
                    pos = self._obs_cell_pos[plan[0].cpu().numpy()]
                    self._sample_obs_pos[cache_key] = self.engine._from_numpy(pos.astype(np.int32)) if (pos >= 0).any() else False
                obs_pos = self._sample_obs_pos[cache_key]
                obs_pos = None if obs_pos is False else obs_pos
            self.engine.sample_uniform(*plan[:4], seed=self.seed, first_env=self.first_env,
                                       stream_id=self._next_stream(), obs_pos=obs_pos)

    def _sample_uniform(self, sample_keys=None, sample_new=True):
        """opf_env.py:253-264."""
        assert sample_new, "Currently only implemented for sample_new=True"
        self._sample_keys(list(sample_keys or self.state_keys))

    def _sample_normal(self, relative_std=None, truncated=False, sample_new=True, **_):
        """opf_env.py:286-315: N(mean, std*diff) around the profile mean, clipped to the data range.
        (As in the reference, `relative_std` ends up multiplied by the range twice, A.6 quirk 9.)"""
        assert sample_new, "Currently only implemented for sample_new=True"
        xp = self.xp
        if "_normal" not in self._sample_cache:
            plan = []
            for unit_type, column, idxs in self.state_keys:
                if "res_" in unit_type or "poly_cost" in unit_type or len(idxs) == 0:
                    continue
                df = self.net[unit_type]
                pos = self.positions(unit_type, idxs)
                scal = df.scaling.to_numpy(float)[pos]
                hi = df[f"max_max_{column}"].to_numpy(float)[pos] / scal
                lo = df[f"min_min_{column}"].to_numpy(float)[pos] / scal
                std = relative_std * (hi - lo) if relative_std else df[f"std_dev_{column}"].to_numpy(float)[pos]
                start = self.program.layout.columns[(unit_type, column)][0]
                f = self.engine._from_numpy
                plan.append((xp.as_tensor(start + pos, device=self.device), f(df[f"mean_{column}"].to_numpy(float)[pos]),
                             f(std * (hi - lo)), f(lo), f(hi)))
            self._sample_cache["_normal"] = plan
        for cols, mean, sigma, lo, hi in self._sample_cache["_normal"]:
            n = cols.shape[0]
            u = xp.empty((self.num_envs, 2 * n), dtype=xp.float64, device=self.device)
            self.engine.philox_uniform(u, self.seed, self.first_env, self._next_stream())
            if truncated:
                # scipy.stats.truncnorm.rvs(a, b, loc, scale) as the reference calls it (:307-308): a
                # standard normal truncated to [a, b] = [min, max] -- bounds in STANDARD units, A.6
                # quirk -- then shifted and scaled; inverse-CDF sampling from one uniform per value
                std_normal = xp.distributions.Normal(0.0, 1.0)
                ca, cb = std_normal.cdf(lo), std_normal.cdf(hi)
                p = (ca + u[:, :n] * (cb - ca)).clamp(1e-300, 1.0 - 1e-16)
                self.engine.state[:, cols] = mean + sigma * xp.special.ndtri(p)
            else:
                z = xp.sqrt(-2.0 * xp.log1p(-u[:, :n])) * xp.cos(2.0 * np.pi * u[:, n:])    # Box-Muller
                self.engine.state[:, cols] = xp.minimum(xp.maximum(mean + sigma * z, lo), hi)

    def _set_simbench_state(self, step=None, test=False, noise_factor=0.1,
                            noise_distribution="uniform", interpolate_steps=False, **_):
        """opf_env.py:317-372: gather one profile row per environment, multiply by
        uniform noise, clip to the profile range, store unscaled."""
        if noise_distribution not in ("uniform", "normal"):
            raise NotImplementedError(f"noise distribution {noise_distribution!r}")
        xp, B = self.xp, self.num_envs
        if not hasattr(self, "_prof_dev"):
            self._prof_dev = {}
            for key, df in self.profiles.items():
                if df.shape[1] == 0:
                    continue
                unit_type, column = key
                cols = df[self.net[unit_type].index].to_numpy(float)
                slots = None
                if self.program.layout.has(unit_type, column):
                    start = self.program.layout.columns[(unit_type, column)][0]
                    slots = self.engine._from_numpy(np.arange(start, start + cols.shape[1], dtype=np.int32))
                self._prof_dev[key] = (self.engine._from_numpy(cols),
                                       self.engine._from_numpy(cols.min(axis=0)),
                                       self.engine._from_numpy(cols.max(axis=0)), slots)
            n_prof = len(next(iter(self.profiles.values())))
            self._steps_dev = {name: self.engine._from_numpy(
                np.asarray(v, dtype=np.int64)[np.asarray(v, dtype=np.int64) < n_prof])
                               for name, v in (("test", self.test_steps),
                                               ("validation", self.validation_steps),
                                               ("train", self.train_steps))}
        if step is None:
            pool = self._steps_dev[self.evaluate_on if test else "train"]
            u = xp.empty((B, 1), dtype=xp.float64, device=self.device)
            self.engine.philox_uniform(u, self.seed, self.first_env, self._next_stream())
            step_idx = pool[(u[:, 0] * pool.shape[0]).long().clamp_(max=pool.shape[0] - 1)]
        else:
            step_idx = xp.as_tensor(step, device=self.device).long()
            step_idx = step_idx.expand(B) if step_idx.dim() == 0 else step_idx
        self.current_simbench_step = step_idx
        step_idx = step_idx.contiguous()
        r = None
        if interpolate_steps:                          # :349-353 random point between two profile steps
            r = xp.empty((B, 1), dtype=xp.float64, device=self.device)
            self.engine.philox_uniform(r, self.seed, self.first_env, self._next_stream())
        kind = 0 if not noise_factor else (1 if noise_distribution == "uniform" else 2)
        for key, (table, pmin, pmax, slots) in self._prof_dev.items():
            if slots is None:
                continue
            # one launch per profile table: gather + interpolation + noise (:355-363) + clip (:365-370)
            self.engine.sample_profiles(slots, table, step_idx, r, pmin, pmax, float(noise_factor or 0.0), kind,
                                        self.seed, self.first_env, self._next_stream() if kind else 0)

    def _sampling(self, step=None, test=False, sample_new=True, **kwargs):
        """opf_env.py:222-251 (dispatch on the data distribution)."""
        self.power_flow_available = False
        distr = self.test_data if test else self.train_data
        kwargs.update(self.sampling_params)
        if distr == "noisy_simbench" or "noise_factor" in kwargs:
            if sample_new:
                self._set_simbench_state(step, test, **kwargs)
        elif distr == "simbench":
            if sample_new:
                self._set_simbench_state(step, test, noise_factor=0.0, **kwargs)
        elif distr == "full_uniform":
            self._sample_uniform(sample_new=sample_new)
        elif distr == "normal_around_mean":
            self._sample_normal(sample_new=sample_new, **kwargs)
        elif distr == "mixed":
            # opf_env.py:242-251 draws ONE data source per episode; here every environment draws its
            # own: all three samplers run and each env keeps the columns of the source it drew
            probs = kwargs.pop("data_probabilities", (0.5, 0.75, 1.0))
            xp = self.xp
            r = xp.empty((self.num_envs, 1), dtype=xp.float64, device=self.device)
            self.engine.philox_uniform(r, self.seed, self.first_env, self._next_stream())
            n_in = self.program.layout.n_inputs
            state = self.engine.state
            self._set_simbench_state(step, test, **{k: v for k, v in kwargs.items()
                                                    if k in ("noise_factor", "noise_distribution")})
            from_simbench = state[:, :n_in].clone()
            self._sample_uniform(sample_new=sample_new)
            from_uniform = state[:, :n_in].clone()
            self._sample_normal(sample_new=sample_new, **{k: v for k, v in kwargs.items()
                                                          if k in ("relative_std", "truncated")})
            pick = xp.where(r < probs[0], from_simbench, xp.where(r < probs[1], from_uniform, state[:, :n_in]))
            state[:, :n_in] = pick
            self.sample_source = (r[:, 0] >= probs[0]).long() + (r[:, 0] >= probs[1]).long()
        else:
            raise NotImplementedError(f"unknown data distribution {distr!r}")

    # --------------------------------------------------------------------- gym interface
    def reset(self, seed: int | None = None, options: dict | None = None):
        if seed is not None:
            self.seed = int(seed)
            self._episode = 0
        options = options or {}
        if self._pipe is not None:
            # step_host's look-ahead may still be sampling / copying on the side stream, and it shares
            # the device observation buffer with the reset below
            self.xp.cuda.current_stream(self.device).wait_stream(self._side)
            self.xp.cuda.current_stream(self.device).wait_stream(self._copy_stream)
        self._pipe = None
        self.test = options.get("test", False)
        self._begin_episode(options.get("step", None))
        return self._obs_out(), {}

    def _begin_episode(self, step=None):
        self._episode += 1
        self._stream_in_episode = 0
        self.current_simbench_step = None
        self._reset_log = []
        distr = self.test_data if self.test else self.train_data
        fusable = self.fused_reset and distr == "full_uniform" and not self.pf_for_obs \
            and not self.sampling_params and step is None
        random_action = self.initial_action == "random"
        if fusable and distr in self._reset_plans:
            plan, n_streams = self._reset_plans[distr]
            self.power_flow_available = False
            self.engine.reset_episode(plan, self.seed, self.first_env, self._episode * 64, random_action,
                                      n_streams + 1)
            self._stream_in_episode = n_streams + int(random_action)
            return
        if fusable:
            self.engine.trace = []
        try:
            self._sampling(step, self.test, True)
        finally:
            trace, self.engine.trace = self.engine.trace, None
        if fusable:
            self._reset_plans[distr] = (self.engine.make_reset_plan(trace, self._episode * 64),
                                        self._stream_in_episode)
        self._apply_initial_action(random_action)
        if not self.pf_for_obs:
            if not (self._obs_by_sampler and self._reset_log == self._obs_sampler_plans.get(distr)):
                self.engine.observe()
                if step is None and not self.sampling_params:
                    self._plan_reset_observation(distr)
            return
        self._reset_power_flow()
        # The reference re-samples a state whose reset power flow fails (opf_env.py:209-214: `return self.reset()`).
        # Batched: every environment draws again (the next RNG streams), the new state is kept only where the
        # previous one failed; bounded (the reference recurses without limit), one host sync per reset in this
        # mode.  What still fails after `max_reset_resamples` rounds starts with a NaN observation, converged = 0.
        e, xp = self.engine, self.xp
        for _ in range(self.max_reset_resamples):
            failed = self._results.converged == 0
            if not bool(failed.any()):
                break
            good_state, good_actions = e.state.clone(), e.actions_reset.clone()
            self._sampling(step, self.test, True)
            self._apply_initial_action(random_action, assemble=False)
            e.state.copy_(xp.where(failed[:, None], e.state, good_state))
            e.actions_reset.copy_(xp.where(failed[:, None], e.actions_reset, good_actions))
            self._apply_initial_action(random_action, draw=False)
            self._reset_power_flow()

    def _plan_reset_observation(self, distr):
        """Can the reset observation be written by the sampler itself?  Yes if every observed cell is a cell the
        uniform sampler wrote during this reset and nothing else writes it afterwards (hook programs, the
        initial action's set-points).  Then later resets of the same shape pass the observation positions to
        `opfg_sample_uniform_obs` and skip `opfg_observe` (which re-reads 3.5 KB of state per environment from
        DRAM: 117 MB per reset of 32 768 VoltageControl environments).  Built-in envs only: a user hook may
        touch the state with arbitrary tensor code."""
        if distr in self._obs_sampler_plans or distr != "full_uniform":
            return
        self._obs_sampler_plans[distr] = None
        if not self._fuse_reset_obs:
            return
        sc = self.program.scoring
        if sc.get("obs_ptr") is not None or not len(sc["obs_ref"]) or (np.asarray(sc["obs_ref"]) < 0).any():
            return
        obs_cells = np.asarray(sc["obs_ref"], np.int64)
        if len(np.unique(obs_cells)) != len(obs_cells):
            return
        sampled, later = set(), set()
        for kind, key in self._reset_log:
            if kind == "sample":
                sampled.update(self._sample_cache[key][0].cpu().numpy().tolist())
            else:
                for start, n in self._program_writes.get(key, ()):
                    later.update(range(start, start + n))
        later.update(np.asarray(self.program.assembly["act_slot"]).tolist())
        cells = set(obs_cells.tolist())
        if not cells <= sampled or cells & later:
            return
        pos = -np.ones(self.program.layout.n, np.int64)
        pos[obs_cells] = np.arange(len(obs_cells))
        self._obs_cell_pos = pos
        self._obs_sampler_plans[distr] = list(self._reset_log)
        self._obs_by_sampler = True

    def _apply_initial_action(self, random_action, draw=True, assemble=True):
        """opf_env.py:199-207: the initial (centre / random) action and its set-points."""
        if draw:
            if random_action:
                self.engine.philox_uniform(self.engine.actions_reset, self.seed, self.first_env,
                                           self._next_stream())
            else:
                self.engine.actions_reset.fill_(0.5)
        if not assemble:
            return
        if self.pf_for_obs:
            self.engine.actions.copy_(self.engine.actions_reset)
        self.engine.assemble(scatter_sbus=self.pf_for_obs, absolute=True)   # opf_env.py:207

    def _reset_power_flow(self):
        """Power flow + scoring of the freshly reset state (opf_env.py:209-216).  It goes to the
        engine's auxiliary result buffers without statistics: what ``step`` just returned (possibly
        as aliases, ``copy_outputs=False``) stays intact and ``episode_statistics`` counts agent
        steps only."""
        e = self.engine
        aux = e.enable_aux_results()
        if self.diff_objective:
            e.enable_objective_offset().zero_()
        e.pf_solve(e.batch_aux)
        e.score(e.batch_aux)
        if self.diff_objective:      # opf_env.py:216: initial_obj = objective of the reset state
            e.objective_offset.copy_(aux.objective)
        self.power_flow_available = True
        self._results = aux

    def _apply_plugins(self):
        """``objective_function=`` plug-in and callable constraints: costs from the callable, callable constraints
        evaluated with tensor ops; reward / cost recombined with the constraint results of kernel 5
        (reward.py:61-98, constraints.py:70-88)."""
        e, xp = self.engine, self.xp
        ok = e.converged.bool()
        if self._custom_objective is not None:
            costs = xp.as_tensor(self._custom_objective(self), device=self.device).to(xp.float64)
            objective = -(costs.reshape(self.num_envs, -1).sum(dim=1))
            if e.objective_offset is not None:
                objective = objective - e.objective_offset
        else:
            objective = e.objective.clone()
        nc = max(len(self.constraints), 1)
        valid = e.valids[:, :nc].bool().all(dim=1)
        penalty = e.penalties[:, :nc].sum(dim=1)
        self._batched_metrics = []
        for c in self.batched_constraints:
            v, viol, pen = c.batched_metrics(self)
            # a failed power flow reports every constraint violated (opf_env.py:390-399), as kernel 5 does for its own
            one = xp.ones_like(viol)
            self._batched_metrics.append((v & ok, xp.where(ok, viol, one), xp.where(ok, pen, one)))
            valid = valid & v
            penalty = penalty + pen
        nan = xp.full_like(objective, float("nan"))
        e.objective.copy_(xp.where(ok, objective, nan))
        e.reward.copy_(xp.where(ok, self.reward_function.batched(objective, penalty, valid), nan))
        e.cost.copy_(xp.where(ok, self.reward_function.batched_cost(penalty, valid), nan))

    def _obs_out(self, final: bool = False, obs=None):
        if obs is None:
            obs = self.engine.obs_final if final else self.engine.obs
        if self.add_mean_obs:
            parts, k = [], 0
            for n in self.program.obs_segments:
                if n > 1:
                    parts.append(obs[:, k:k + n].mean(dim=1, keepdim=True))
                k += n
            return self.xp.cat([obs] + parts, dim=1)
        return obs.clone() if self.copy_outputs else obs

    def step(self, actions):
        """Apply ``actions[num_envs, n_act]`` (torch or numpy, any float dtype), run the
        batched power flow, score, auto-reset.  Returns torch tensors on the device:
        ``(obs, reward, terminated, truncated, info)``; ``info['final_obs']`` holds the
        observation of the finished episode."""
        act = self._step_begin(actions)
        e = self.engine
        if self._custom_solver is None:
            e.step(final_obs=True)
        else:                                         # plug-in power flow between kernel 1 and kernel 5
            e.assemble()
            self._custom_solver(self)
            e.score(e.batch_final)
        return self._step_end(act)

    # step() in three parts, so that a mixed batch (opfgym_b200.mixed) can run the kernels of several
    # envs as shared launches between the parts
    def _step_begin(self, actions):
        xp = self.xp
        act = xp.as_tensor(actions, device=self.device)
        if self.validate_actions and xp.isnan(act).any():   # host sync; off by default
            raise AssertionError("NaN in actions")     # opf_env.py:382
        e = self.engine
        if self._pipe is not None:
            raise RuntimeError("step() after step_host(): the host pipeline holds pre-sampled episodes; "
                               "call reset() before switching back to the tensor API")
        if self._prefetch:
            # The next episode is needed at the end of THIS step: its kernels go first (measured: issued behind
            # the power flow instead, sharing the GPU with kernel 5, the step is 1.290 instead of 1.266 ms).
            main = xp.cuda.current_stream(self.device)
            self._main_done.record(main)
            cur, nxt = e.cur, (e.cur + 1) % len(e._states)
            e.select(nxt)                             # launches below target the NEXT episode's buffer
            with xp.cuda.stream(self._side):
                self._side.wait_event(self._main_done)
                self._begin_episode()
                self._side_done.record(self._side)
            e.select(cur)
            self._next_buffer = nxt
        self.engine.actions.copy_(act.reshape(self.engine.actions.shape))
        return act

    def _step_end(self, act):
        xp, e = self.xp, self.engine
        self.power_flow_available = True
        self._results = e
        keep = (lambda t: t.clone()) if self.copy_outputs else (lambda t: t)
        if self._custom_objective is not None or self.batched_constraints:
            self._apply_plugins()
        reward = keep(e.reward)
        if self.clipped_action_penalty:
            # opf_env.py:429, 488-491: the correction is measured against the CLIPPED action
            reward = reward - self._mean_correction(act.clamp(0.0, 1.0)) * self.clipped_action_penalty
        nc = max(len(self.constraints), 1)
        info = {"valids": e.valids[:, :nc].bool(), "violations": keep(e.violations[:, :nc]),
                "unscaled_penalties": keep(e.penalties[:, :nc]), "cost": keep(e.cost),
                "converged": e.converged.bool(), "iterations": keep(e.iterations),
                "final_obs": self._obs_out(final=True)}
        if self.batched_constraints:          # their columns follow the kernel's (none of the kernel's if it has none)
            k = len(self.constraints)
            for key, i in (("valids", 0), ("violations", 1), ("unscaled_penalties", 2)):
                extra = xp.stack([m[i] for m in self._batched_metrics], dim=1)
                info[key] = xp.cat([info[key][:, :k], extra], dim=1)
        if self._flags is None:
            self._flags = (xp.ones(self.num_envs, dtype=xp.bool, device=self.device),
                           xp.zeros(self.num_envs, dtype=xp.bool, device=self.device))
        terminated, truncated = (keep(self._flags[0]), keep(self._flags[1]))
        if self._prefetch:
            xp.cuda.current_stream(self.device).wait_event(self._side_done)
            e.select(self._next_buffer)               # the prefetched episode becomes the current one
        else:
            self._begin_episode()
        return self._obs_out(), reward, terminated, truncated, info

    # ------------------------------------------------------------- host-buffer (numpy) step
    def enable_host_io(self):
        """Pinned host buffers for :meth:`step_host` (the reference's numpy-in / numpy-out
        ``step``, opf_env.py:371-419).  ``host_actions`` may be filled in place by the caller."""
        if getattr(self, "_host", None) is None:
            xp, B = self.xp, self.num_envs
            cuda = self.device.type == "cuda"
            pin = lambda *shape, dtype: (xp.empty(shape, dtype=dtype).pin_memory() if cuda
                                         else xp.empty(shape, dtype=dtype))
            n_obs = self.single_observation_space.shape[0]
            host_dt = getattr(xp, self.host_obs_dtype) if self.host_obs_dtype else self.engine.obs.dtype
            self._obs_cast = None if host_dt == self.engine.obs.dtype else \
                xp.empty((B, n_obs), dtype=host_dt, device=self.device)
            self._host = dict(
                actions=pin(B, max(self.program.n_act, 1), dtype=xp.float64),
                obs=pin(B, n_obs, dtype=host_dt),
                obs_alt=pin(B, n_obs, dtype=host_dt), reward=pin(B, dtype=xp.float64),
                cost=pin(B, dtype=xp.float64), converged=pin(B, dtype=self.engine.converged.dtype),
                terminated=xp.ones(B, dtype=xp.bool).numpy(), truncated=xp.zeros(B, dtype=xp.bool).numpy())
            self.host_actions = self._host["actions"].numpy()
            self._host_np = {k: (v.numpy() if hasattr(v, "numpy") else v) for k, v in self._host.items()}
        return self._host

    def step_host(self, actions=None):
        """``step`` for callers that live on the host: ``actions`` is a numpy array / CPU tensor
        (``None``: use ``self.host_actions`` as filled by the caller); returns numpy views of pinned
        buffers ``(obs, reward, terminated, truncated, info)`` that stay valid until the next call.

        The copies are part of the pipeline instead of a tail: the next episode's observation is
        produced by the side stream while the power flow of this step still runs, so its
        device->host transfer (the bulk of the bytes) overlaps kernel 3/4; only the small per-env
        results (reward, cost, converged) are copied after kernel 5."""
        xp, e = self.xp, self.engine
        if self._custom_solver is not None or self._custom_objective is not None or self.batched_constraints:
            raise NotImplementedError("step_host pipelines the built-in kernels; with a plug-in power flow or "
                                      "objective use step()")
        h = self.enable_host_io()
        src = h["actions"]
        if actions is not None:
            a = xp.as_tensor(actions)
            if a.is_floating_point() and a.is_contiguous() and (a.is_pinned() or self.device.type != "cuda"):
                src = a.reshape(src.shape)             # already DMA-able (any float dtype; gym's Box
                                                       # default is float32): no staging copy
            elif a.data_ptr() != src.data_ptr():
                src.copy_(a.reshape(src.shape))
        if self.validate_actions and xp.isnan(src).any():
            raise AssertionError("NaN in actions")     # opf_env.py:382
        def obs_to_host(dst, dev_obs=None):
            keep, self.copy_outputs = self.copy_outputs, False     # no device-side clone on the way out
            obs = self._obs_out(obs=dev_obs)
            if self._obs_cast is not None:                         # narrower host dtype: cast on the device
                self._obs_cast.copy_(obs)
                obs = self._obs_cast
            dst.copy_(obs, non_blocking=True)
            self.copy_outputs = keep

        main = xp.cuda.current_stream(self.device) if self.device.type == "cuda" else None
        obs_now = h["obs"]
        if self._prefetch:
            # Two episodes ahead.  The persistent power-flow kernel fills every SM (registers and
            # shared memory): kernels of another stream cannot run beside it, but a copy can.  So the
            # observation this call returns (episode k+1) was sampled and sent to the host during the
            # PREVIOUS call; this call's side-stream work prepares episode k+2 behind the step's own
            # kernels, and its 58 MB transfer runs on the copy engine under the next power flow (and
            # under whatever the caller does between two calls).
            e.enable_double_buffer(3)
            pipe = self._pipe

            def sample_ahead(buf, dst, after=None, start_after=None):
                """Side stream: kernels of the next episode into state buffer `buf`; then (once the
                event `after` has passed -- the copy engine serves requests in order, and the
                small per-step results must not queue behind 58 MB) its observation to `dst`."""
                cur = e.cur
                e.select(buf)
                sampled = self._sampled_events[buf]
                with xp.cuda.stream(self._side):
                    self._side.wait_event(start_after or self._main_done)
                    self._begin_episode()
                    sampled.record(self._side)
                dev_obs = e.obs                        # every episode buffer has its own device observation ...
                e.select(cur)

                def copy():
                    # ... so the transfer runs on a stream of its own: the side stream's kernels of the NEXT
                    # call do not queue behind 58 MB on the copy engine (they used to, and then had to find a
                    # gap next to the persistent power-flow kernel: 1.43 instead of 1.35 ms per step)
                    with xp.cuda.stream(self._copy_stream):
                        self._copy_stream.wait_event(sampled)
                        if after is not None:
                            self._copy_stream.wait_event(after)
                        obs_to_host(dst, dev_obs)
                        ready = self._ready_events[dst is h["obs"]]
                        ready.record(self._copy_stream)
                    return ready
                return copy

            self._main_done.record(main)               # buffers of finished episodes are free from here on
            if pipe is None:                           # first call after reset: episode k+1 is not there yet
                nxt = (e.cur + 1) % 3
                pipe = dict(buf=nxt, obs="obs", ready=sample_ahead(nxt, h["obs"])())
            e.actions.copy_(src, non_blocking=True)    # this step's own work goes to the GPU first
            # The look-ahead episode is not needed before the NEXT call: its kernels are issued behind the
            # power flow (the persistent kernel fills every SM, nothing runs beside it), where they share
            # the GPU with kernel 5 and fill the gap between two calls -- 1.33 instead of 1.46 ms per call
            # against issuing them at the start of the step, where they contend with kernel 1 / the DC GEMM
            e.assemble()
            e.pf_solve()
            self._pf_done.record(main)
            e.score(e.batch_final)
            free = 3 - e.cur - pipe["buf"]             # the buffer of the episode before this one
            other = "obs_alt" if pipe["obs"] == "obs" else "obs"
            copy_ahead = sample_ahead(free, h[other], after=self._results_copied, start_after=self._pf_done)
        else:
            e.actions.copy_(src, non_blocking=True)
            e.step(final_obs=True)
        self.power_flow_available = True
        self._results = e
        reward = e.reward
        if self.clipped_action_penalty:
            reward = reward - self._mean_correction(e.actions.clamp(0.0, 1.0)) * self.clipped_action_penalty
        h["reward"].copy_(reward, non_blocking=True)
        h["cost"].copy_(e.cost, non_blocking=True)
        h["converged"].copy_(e.converged, non_blocking=True)
        if self._prefetch:
            self._results_copied.record(main)
            ahead = dict(buf=free, obs=other, ready=copy_ahead())
            main.synchronize()                         # the caller needs the results to act
            pipe["ready"].synchronize()                # (sent during the previous call)
            obs_now = h[pipe["obs"]]
            e.select(pipe["buf"])                      # episode k+1 becomes the current one
            self._pipe = ahead
        else:
            self._begin_episode()
            obs_to_host(h["obs"])
            if main is not None:
                main.synchronize()
        n = self._host_np
        info = {"cost": n["cost"], "converged": n["converged"].astype(bool, copy=False)}
        return obs_now.numpy(), n["reward"], n["terminated"], n["truncated"], info

    def _mean_correction(self, act):
        """opf_env.py:488-491: mean |applied action - requested action|."""
        return (self.get_current_actions(from_results_table=False) - act).abs().mean(dim=1)

    def close(self):
        self.engine.close()

    # ----------------------------------------------------------------- OpfEnv-style API
    def run_power_flow(self, **kwargs):
        """opf_env.py:646-662; returns the per-environment converged mask."""
        e = self.engine
        e.assemble(apply_actions=False)   # re-scatter Sbus from the current cells
        batch = e.nostats_batch()         # not an agent step: no contribution to the statistics
        e.pf_solve(batch)
        e.score(batch)
        if (self._custom_objective is not None or self.batched_constraints) and self._custom_solver is None:
            self._apply_plugins()         # plug-in objective / callable constraints see this power flow
        self.power_flow_available = True
        self._results = e
        return e.converged.bool()

    def ensure_power_flow_available(self):
        if not self.power_flow_available:
            raise PowerFlowNotAvailable("Please call `run_power_flow` first!")

    def _apply_actions(self, actions):
        self.engine.actions.copy_(self.xp.as_tensor(actions, device=self.device))
        self.engine.assemble()
        self.power_flow_available = False

    def get_state(self):
        return self._gather(self.state_keys)

    def _gather(self, keys):
        parts = []
        for unit_type, column, idxs in keys:
            pos = self.xp.as_tensor(self.positions(unit_type.replace("res_", "", 1)
                                                   if unit_type.startswith("res_") else unit_type,
                                                   idxs), device=self.device)
            if self.program.layout.has(unit_type, column):
                parts.append(self.col(unit_type, column)[:, pos])
            else:
                parts.append(self.static(unit_type, column)[pos].expand(self.num_envs, -1))
        return self.xp.cat(parts, dim=1)

    def get_current_actions(self, from_results_table=True):
        """opf_env.py:566-588: the [0, 1] actions that the current set-points represent."""
        out = []
        for unit_type, column, idxs in self.act_keys:
            pos = self.xp.as_tensor(self.positions(unit_type, idxs), device=self.device)
            sp = self.col(unit_type, column)[:, pos]
            if "scaling" in self.net[unit_type].columns:
                sp = sp * self.static(unit_type, "scaling")[pos]
            lo_c, hi_c = (f"min_{column}", f"max_{column}") if self.autoscale_actions else \
                         (f"min_min_{column}", f"max_max_{column}")
            lo = self._value(unit_type, lo_c, pos)
            hi = self._value(unit_type, hi_c, pos)
            out.append((sp - lo) / (hi - lo))
        return self.xp.cat(out, dim=1)

    get_actions = get_current_actions

    def _value(self, table, column, pos):
        if self.program.layout.has(table, column):
            return self.col(table, column)[:, pos]
        return self.static(table, column)[pos]

    # the getters read the results of the LAST power flow: the agent's step, or the reset power flow
    def is_state_valid(self):
        self.ensure_power_flow_available()
        nc = max(len(self.constraints), 1)
        valid = self._results.valids[:, :nc].bool().all(dim=1)
        if self.batched_constraints and self._results is self.engine and getattr(self, "_batched_metrics", None):
            for m in self._batched_metrics:            # callable constraints of the last step
                valid = valid & m[0]
        return valid

    def get_objective(self):
        self.ensure_power_flow_available()
        return self._results.objective.clone()

    def calculate_violations(self):
        self.ensure_power_flow_available()
        nc = max(len(self.constraints), 1)
        r = self._results
        out = (r.valids[:, :nc].bool(), r.violations[:, :nc], r.penalties[:, :nc])
        if self.batched_constraints and r is self.engine and getattr(self, "_batched_metrics", None):
            k = len(self.constraints)                  # the callable constraints' columns follow the kernel's
            out = tuple(self.xp.cat([o[:, :k], self.xp.stack([m[i] for m in self._batched_metrics], dim=1)], dim=1)
                        for i, o in enumerate(out))
        return out

    def sample_objective_penalty(self, num_samples: int):
        """Feeds ``reward.estimate_reward_distribution`` (reference reward.py:181-216:
        reset, random action, power flow -- ``num_samples`` times) from batched launches."""
        objs, pens = [], []
        done = 0
        while done < num_samples:
            self._episode += 1
            self._stream_in_episode = 0
            self._sampling(None, False, True)
            self.engine.philox_uniform(self.engine.actions, self.seed, self.first_env,
                                       self._next_stream())
            self.engine.step()
            ok = self.engine.converged.bool()
            objs.append(self.xp.where(ok, self.engine.objective, float("nan")))
            pens.append(self.xp.where(ok, self.engine.penalty, float("nan")))
            done += self.num_envs
        objs = self.xp.cat(objs)[:num_samples].cpu().numpy()
        pens = self.xp.cat(pens)[:num_samples].cpu().numpy()
        return objs, pens

    # ------------------------------------------------------------- episode statistics
    def episode_statistics(self, reduce: bool = True) -> dict:
        """Running sums accumulated by kernel 5's epilogue; with ``torch.distributed``
        initialised they are all-reduced over ranks (the path's only collective)."""
        stats = self.engine.stats.sum(dim=0)
        if reduce and self.world_size > 1:
            import torch.distributed as dist
            if dist.is_available() and dist.is_initialized():
                dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        s = stats.cpu().numpy()
        n = max(s[0], 1.0)
        nconv = max(s[1], 1.0)
        return {"steps": s[0], "converged": s[1], "valid": s[2],
                "mean_reward": s[3] / nconv,
                "std_reward": float(np.sqrt(max(s[4] / nconv - (s[3] / nconv) ** 2, 0.0))),
                "mean_objective": s[5] / nconv, "mean_penalty": s[6] / nconv,
                "mean_iterations": s[7] / nconv, "converged_share": s[1] / n,
                "valid_share": s[2] / n,
                "violated_share": (s[8:8 + len(self.constraints)] / n).tolist()}

    def reset_statistics(self):
        self.engine.stats.zero_()
