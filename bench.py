#!/usr/bin/env python
"""Headline benchmark: AC power-flow env steps/s of the batched environments.

  python bench.py --gpus N --steps K --warmup W          # this repo's CUDA path
  python bench.py --impl reference ...                    # CPU arm: oracle port on host cores
  torchrun --nproc-per-node N bench.py --gpus N ...       # one rank per GPU, weak scaling
  python bench.py --config {vc32k,ed64k,mixed,ls_dyn}     # which BASELINE.json workload

--config (default vc32k = BASELINE.json configs[1], the one the metric is quoted on):
  vc32k   VoltageControl, 32 768 envs of the 122-bus MV grid per GPU            (configs[1])
  ed64k   EcoDispatch, 372-bus HV grid, 8 192 envs per GPU = 64k on 8 GPUs      (configs[2])
  mixed   MaxRenewable (HV) + QMarket (MV) stepped as one batch                 (configs[3])
  ls_dyn  LoadShedding + tap / tie-switch actions, per-env Ybus values          (configs[4])
configs[0] (one env, reset + step, CPU) is reported inside every N=1 line as `single_env`.

One "step" = `env.step(actions)` for the whole batch: apply actions, batched
Newton-Raphson power flow, fused scoring/observation, same-step auto-reset
(sample a new grid state for every env).  Prints ONE JSON line (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

# stdout carries exactly one JSON line: NCCL's own banner ("NCCL version ...") goes to stderr
os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "ac_power_flow_env_steps_per_sec"
UNIT = "env_steps/s"
CONFIGS = {
    "vc32k": dict(members=[("VoltageControl", 32768)],
                  workload="VoltageControl batched 32k envs (BASELINE configs[1]): synthetic stand-in of SimBench "
                           "1-MV-semiurb--1-sw (122 buses, 442 obs, 14 reactive-power actions), shared Ybus, "
                           "full_uniform sampling, U[0,1] actions"),
    "ed64k": dict(members=[("EcoDispatch", 8192)],
                  workload="EcoDispatch, 64k envs sharded over 8 GPUs = 8 192 per GPU (BASELINE configs[2]): "
                           "synthetic stand-in of SimBench 1-HV-urban--0-sw (372 buses, 201 obs, 42 actions)"),
    "mixed": dict(members=[("MaxRenewable", 8192), ("QMarket", 24576)],
                  workload="MaxRenewable (355-bus HV) + QMarket (97-bus MV) mixed batch (BASELINE configs[3]), "
                           "8 192 + 24 576 envs per GPU"),
    "ls_dyn": dict(members=[("LoadSheddingReconfiguration", 32768)],
                   workload="LoadShedding with tap / tie-switch actions, per-env Ybus values (BASELINE configs[4]): "
                            "111-bus MV grid + 4 tie lines, 32 768 envs per GPU"),
}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="vc32k", choices=sorted(CONFIGS))
    ap.add_argument("--envs-per-gpu", type=int, default=0, help="override (single-member configs)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="budget of the cpu_baseline sample")
    ap.add_argument("--host-obs-dtype", default=None, choices=[None, "float32", "float16"],
                    help="e2e leg: dtype of the observations on the host (default: float32, the reference's Box dtype)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed env.step returned (rank 0) as DIR/<name>.npy "
                         "in float32 / float64, at most 64 MB in all: above that, every array keeps the rows "
                         "sorted(np.random.default_rng(0).permutation(n)[:k]) of its n environments, k = n x budget "
                         "share; bool and integer outputs are stored as float32 / float64")
    return ap.parse_args()


# ------------------------------------------------------------------------- CPU arm
def cpu_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def run_cpu_pool(n_per_worker: int, rounds: int, warm_rounds: int = 1, kinds=("VoltageControl",)):
    """Oracle env port under multiprocessing.Pool(all cores); returns (steps/s, total steps,
    converged, seconds, cores, per-round seconds)."""
    import multiprocessing as mp
    from oracle import env_port
    cores = cpu_cores()
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        # mixed configs: the workers are split over the member environments
        kind_of = [kinds[s % len(kinds)] for s in range(cores)]
        for _ in range(warm_rounds):
            pool.map(env_port._worker_steps, [(s, 2, kind_of[s]) for s in range(cores)])
        times, done, ok = [], 0, 0
        for _ in range(rounds):
            t0 = time.perf_counter()
            out = pool.map(env_port._worker_steps, [(s, n_per_worker, kind_of[s]) for s in range(cores)])
            times.append(time.perf_counter() - t0)
            done += sum(o[0] for o in out)
            ok += sum(o[1] for o in out)
    total = sum(times)
    return done / total, done, ok, total, cores, times


def reference_arm(args):
    """--impl reference: the reference's CPU path for the same metric.  pandapower is not
    installable on this image, so the arm is the oracle port (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = cpu_cores()
    per_worker = 4
    kinds = tuple(k for k, _ in CONFIGS[args.config]["members"])
    # bounded: the arm must end within a few minutes whatever --steps says (one round = cores x 4 env
    # steps at ~0.1 s each on the oracle port)
    rounds = max(1, min(args.steps, 40))
    rate, done, ok, secs, cores, times = run_cpu_pool(per_worker, rounds=rounds,
                                                      warm_rounds=max(1, min(args.warmup, 2)), kinds=kinds)
    sample = (f"{rounds} rounds x {cores} workers x {per_worker} (reset+step) of the "
              f"oracle env port ({'+'.join(kinds)}) = {done} env steps in {secs:.1f} s")
    line = {"impl": "reference", "metric": METRIC, "value": rate, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * secs / rounds,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64",
            "data": "synthetic", "config": {"workload": CONFIGS[args.config]["workload"], "name": args.config,
                                            "envs_per_step": cores * per_worker, "timed_rounds": rounds},
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0, "converged_share": ok / max(done, 1)}
    print(json.dumps(line))


# ------------------------------------------------------------------------ clocks
class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                 "-lms", "100", "-i", str(self.gpu)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2]))
            except (ValueError, IndexError):
                continue
            for name, col in (("hw_slowdown", 5), ("hw_thermal_slowdown", 6),
                              ("sw_thermal_slowdown", 7), ("sw_power_cap", 8)):
                if len(r) > col and r[col].lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# -------------------------------------------------------------------------- GPU arm
def gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device: there is no CPU fallback")
    torch.cuda.set_device(local_rank)
    affinity = "default"
    if world > 1 and not os.environ.get("OPFG_NO_NUMA_BIND"):
        # One process per GPU: keep it (and the pinned buffers it is about to allocate, first touch)
        # on the CPU socket the GPU hangs off, so the 58 MB/step of observations of eight ranks do not
        # cross the socket interconnect.
        try:
            import pynvml
            pynvml.nvmlInit()
            pr = torch.cuda.get_device_properties(local_rank)
            bus_id = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByPciBusId(bus_id.encode()))
            affinity = f"nvml numa-local ({len(os.sched_getaffinity(0))} cpus)"
        except Exception as exc:              # affinity is an optimisation, never a requirement
            affinity = f"default ({type(exc).__name__})"
    if world > 1:
        # NCCL prints its version banner to stdout while the communicator is created (it honours
        # NCCL_DEBUG_FILE only above the VERSION level): stdout points at stderr for that moment
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    dev = torch.device("cuda", local_rank)

    import __graft_entry__
    if not os.path.exists(__graft_entry__.LIB):
        if rank == 0:
            __graft_entry__.build()
        if world > 1:
            dist.barrier()
    from opfgym_b200 import envs
    from opfgym_b200.mixed import MixedBatchEnv

    cfg = CONFIGS[args.config]
    members = [(k, (args.envs_per_gpu or n) if len(cfg["members"]) == 1 else n) for k, n in cfg["members"]]
    B = sum(n for _, n in members)
    first = 0
    parts = []
    for kind, n in members:
        parts.append(getattr(envs, kind)(num_envs=n, train_data="full_uniform", test_data="full_uniform",
                                         n_profile_steps=672, rank=rank, world_size=world, device=dev,
                                         seed=1234, copy_outputs=False,
                                         host_obs_dtype=None if args.host_obs_dtype in (None, "float32") else args.host_obs_dtype))
    env = parts[0] if len(parts) == 1 else MixedBatchEnv(parts)
    engines = [p.engine for p in parts]
    eng = engines[0]                      # the member whose power-flow kernel the roofline describes
    n_act = max(p.single_action_space.shape[0] for p in parts)
    n_obs = max(p.single_observation_space.shape[0] for p in parts)
    # action pool, resident in HBM before the timed region (Philox, stream = global env id)
    pool = [torch.empty(B, n_act, dtype=torch.float64, device=dev) for _ in range(8)]
    for i, a in enumerate(pool):
        eng.philox_uniform(a, 4321, rank * B, 1000 + i)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(i)
        e1.record()
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    env.reset(seed=1234)

    # ---- device-resident throughput ("value") ------------------------------------------
    last = [None]

    def dev_step(i):
        last[0] = env.step(pool[i % len(pool)])

    for i in range(args.warmup):
        dev_step(i)
    for p in parts:
        p.reset_statistics()
    eng.pf_events = []
    launches0 = eng.launch_count()
    clocks = ClockSampler(local_rank)
    if rank == 0:
        clocks.start()
    ms_total = timed(dev_step, args.steps)
    clock_info = clocks.stop() if rank == 0 else None
    launches = eng.launch_count() - launches0       # one library: the counter covers every member
    pf_ms = sum(a.elapsed_time(b) for a, b in eng.pf_events) / max(len(eng.pf_events), 1)
    eng.pf_events = None
    stats = env.episode_statistics(reduce=True)
    member_stats = stats.get("members", [stats])
    value = world * B * args.steps / (ms_total * 1e-3)
    if args.dump_outputs and rank == 0:
        # copy_outputs=False: the returned tensors alias engine buffers that the e2e leg below overwrites
        dump_outputs(args.dump_outputs, last[0])

    # ---- end to end through the public API with HOST buffers ("e2e") ---------------------
    # env.step_host: actions from a pinned host buffer, results (next observation, reward, cost,
    # converged) back in pinned host memory, stream-synchronised before it returns -- every step
    # float32 actions: the dtype of the reference's action space (gym.spaces.Box default, opf_env.py:130)
    h_act = [torch.rand(B, n_act, dtype=torch.float32).pin_memory() for _ in range(4)]
    e2e_sink = []

    def e2e_step(i):
        obs, reward, term, trunc, info = env.step_host(h_act[i % len(h_act)])
        e2e_sink[:] = [obs, reward, info["converged"]]   # numpy views of the pinned result buffers

    for i in range(min(args.warmup, 3)):
        e2e_step(i)
    e2e_steps = max(5, args.steps // 2)
    ms_e2e = timed(e2e_step, e2e_steps)
    e2e_value = world * B * e2e_steps / (ms_e2e * 1e-3)
    obs_bytes = 2 if args.host_obs_dtype == "float16" else 4
    if len(parts) > 1:
        # mixed batch: ONE padded action matrix in, ONE padded observation matrix out (MixedBatchEnv.step_host)
        h2d = B * n_act * 4
        d2h = B * (env.n_obs * 4 + 8 + 8 + 1 + 1 + 1)        # obs (float32), reward, cost, converged, terminated, truncated
    else:
        h2d = sum(p.num_envs * p.single_action_space.shape[0] * 4 for p in parts)
        d2h = sum(p.num_envs * (p.single_observation_space.shape[0] * obs_bytes + 8 + 8 + 1) for p in parts)   # obs, reward, cost, flag

    # ---- FP64 peak probe (roofline denominator not in MEASURED_PEAKS.json) -----------------
    fp64_tflops = None
    if rank == 0:
        blocks, iters = 148 * 16, 20000
        eng.fp64_probe(blocks, 200)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        eng.fp64_probe(blocks, iters)
        e1.record()
        torch.cuda.synchronize()
        fp64_tflops = 2.0 * 8 * iters * blocks * 256 / (e0.elapsed_time(e1) * 1e-3) / 1e12

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    info = eng.info
    B0 = parts[0].num_envs
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        hbm_peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    else:
        hbm_peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    bytes_per_step = info["bytes_per_step"]
    achieved_gbs = bytes_per_step * B0 / (pf_ms * 1e-3) / 1e9
    iters = member_stats[0]["mean_iterations"]
    kernel_name = {1: "k_pf_multi (one CTA group per environment: mismatch + Jacobian + level-scheduled block LU in shared memory)",
                   2: "k_pf_lanes (one lane per environment)",
                   3: "k_pf_tree (fused radial kernel: mismatch + on-the-fly Jacobian + leaf-first block LU, "
                      f"{info['radial_lanes_per_env']} lanes x {info['radial_envs_per_cta']} environments per SM)"}[info["pf_kernel_used"]]
    # DRAM traffic of the dominant kernel: taken from an ncu capture of THIS source (tools/ncu_traffic.py
    # writes profiles/pf_traffic.json with a hash of csrc/); any other source -> null, never a stale constant
    traffic, traffic_src = None, "no ncu capture of this source (tools/ncu_traffic.py)"
    try:
        rec = json.load(open(os.path.join(ROOT, "profiles", "pf_traffic.json"))).get(args.config)
        if rec and rec["csrc_sha256"] == csrc_hash():
            traffic = rec["dram_bytes_per_launch"] * B0 / rec["n_env"]
            traffic_src = rec["source"]
        elif rec:
            traffic_src = "profiles/pf_traffic.json is from another source revision"
    except (OSError, ValueError, KeyError):
        pass
    # FP64 work of one env step: `iters` full iterations + the final mismatch-only pass + scoring
    flops_mismatch = 8.0 * info["nnz_y"] + 8.0 * info["nb"]
    flops_pf = info["flops_per_iter"] * iters + flops_mismatch
    flops_per_step = flops_pf + info["flops_score"]
    roofline = {"bound": "hbm", "kernel": "opfg_pf_solve = k_dc_start (DC-start GEMM) + " + kernel_name,
                "achieved": achieved_gbs, "peak": hbm_peak, "unit": "GB/s", "frac": achieved_gbs / hbm_peak,
                "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
                "kernel_ms": pf_ms, "kernel_share_of_step": pf_ms / (ms_total / args.steps),
                "algorithmic_bytes_per_env_step": bytes_per_step, "envs_per_launch": B0,
                "note": "latency-bound FP64 sparse path: HBM fraction is small by construction "
                        "(SURVEY.md 8d); see fp64 for the pipe-side figure"}
    fp64 = {"flops_per_env_step": flops_per_step, "mean_nr_iterations": iters,
            "achieved_tflops_kernel": flops_pf * B0 / (pf_ms * 1e-3) / 1e12,
            "peak_tflops_measured": fp64_tflops,
            "frac_kernel": (flops_pf * B0 / (pf_ms * 1e-3) / 1e12) / fp64_tflops,
            "note": "flops = iterations x flops_per_iter + one mismatch-only pass (the last convergence check)"}

    cpu_baseline = single_env = None
    if world == 1 and not args.no_cpu_baseline:
        kinds = tuple(k for k, _ in members)
        per_worker = 4
        rate1, _, _, secs1, cores, _ = run_cpu_pool(per_worker, rounds=1, kinds=kinds)
        rounds = max(1, int(args.cpu_seconds / max(secs1, 1e-3)))
        rate, done, ok, secs, cores, _ = run_cpu_pool(per_worker, rounds=rounds, warm_rounds=0, kinds=kinds)
        cpu_baseline = {"value": rate, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{done} env steps (reset+step of the oracle env port, same grid and "
                                  f"sampler) on {cores} host cores in {secs:.1f} s",
                        "converged_share": ok / max(done, 1)}
        single_env = single_env_row(kinds[0], dev)

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": cfg["workload"], "name": args.config, "envs_per_gpu": B, "global_batch": world * B,
                       "members": [{"env": k, "envs_per_gpu": n} for k, n in members],
                       "parallelism": f"env-sharded x{world}, no data-path collective", "cpu_affinity": affinity,
                       "l2": f"inputs larger than L2: per-GPU state matrix "
                             f"{B0 * info['n_state'] * 8 / 1e6:.0f} MB is re-sampled every step",
                       "n_state": info["n_state"], "n_levels": info["n_levels"],
                       "n_blocks": info["n_blocks"], "pf_kernel": info["pf_kernel_used"]},
            "clocks": clock_info,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / e2e_steps,
                    "host_obs_dtype": args.host_obs_dtype or "float32",
                    "host_ingest_gbs_per_rank": d2h / (ms_e2e / e2e_steps * 1e-3) / 1e9},
            "gpu_launches": launches,
            "roofline": roofline, "fp64": fp64, "cpu_baseline": cpu_baseline, "single_env": single_env,
            "converged_share": sum(m["converged"] for m in member_stats) / max(sum(m["steps"] for m in member_stats), 1.0),
            "valid_share": sum(m["valid"] for m in member_stats) / max(sum(m["steps"] for m in member_stats), 1.0),
            "mean_reward": member_stats[0]["mean_reward"]}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def csrc_hash():
    import hashlib
    h = hashlib.sha256()
    for name in ("opfg_core.h", "opfg_api.cu", "symbolic.cpp", "symbolic.hpp"):
        h.update(open(os.path.join(ROOT, "opfgym_b200", "csrc", name), "rb").read())
    return h.hexdigest()


DUMP_BUDGET = 60 << 20          # bytes of array data: with the .npy headers, under 64 MB


def dump_outputs(out_dir, result):
    """Write the tensors of one ``env.step`` result ``(obs, reward, terminated, truncated, info)`` -- nested
    info entries (a mixed batch's ``member`` list) included -- as ``out_dir/<name>.npy``."""
    import numpy as np
    import torch

    arrays = {}

    def walk(name, x):
        if isinstance(x, torch.Tensor):
            arrays[name] = x
        elif isinstance(x, dict):
            for k, v in x.items():
                walk(f"{name}_{k}", v)
        elif isinstance(x, (list, tuple)):
            for k, v in enumerate(x):
                walk(f"{name}_{k}", v)

    for name, x in zip(("obs", "reward", "terminated", "truncated", "info"), result):
        walk(name, x)

    def as_float(t):
        if t.dtype in (torch.float32, torch.float64):
            return t
        if t.is_floating_point() or t.dtype == torch.bool or t.element_size() <= 2:
            return t.to(torch.float32)
        return t.to(torch.float64)

    arrays = {k: as_float(v.detach()) for k, v in arrays.items()}
    total = sum(v.numel() * v.element_size() for v in arrays.values())
    share = min(1.0, DUMP_BUDGET / max(total, 1))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        if share < 1.0 and t.dim() > 0:
            n = t.shape[0]
            rows = np.sort(np.random.default_rng(0).permutation(n)[:max(1, int(n * share))])
            t = t.index_select(0, torch.as_tensor(rows, device=t.device))
        np.save(os.path.join(out_dir, f"{name}.npy"), t.cpu().numpy())


def single_env_row(kind, dev, n=200):
    """BASELINE.json configs[0]: ONE environment, `reset(); step(action_space.sample())` n times, wall
    clock per (reset + step): the CPU path (oracle env port; pandapower is not installable) next to
    this engine with num_envs = 1 (fused one-launch reset; launch-latency bound)."""
    import numpy as np
    import torch
    from opfgym_b200 import envs
    from oracle import env_port
    cpu = env_port.OracleEnv(kind, seed=0)
    rng = np.random.default_rng(0)
    for _ in range(3):
        cpu.reset(); cpu.step(rng.uniform(0, 1, cpu.n_act))
    n_cpu = min(n, 100)
    t0 = time.perf_counter()
    for _ in range(n_cpu):
        cpu.reset()
        cpu.step(rng.uniform(0, 1, cpu.n_act))
    cpu_ms = 1e3 * (time.perf_counter() - t0) / n_cpu
    env = getattr(envs, kind)(num_envs=1, train_data="full_uniform", test_data="full_uniform",
                              n_profile_steps=672, device=dev, seed=0)
    act = np.random.default_rng(0).uniform(0, 1, (n, 1, env.single_action_space.shape[0])).astype(np.float32)
    env.reset(seed=0)
    for i in range(5):
        env.step_host(act[i])
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(n):
        env.step_host(act[i])             # same-step auto-reset: one call = step + reset, results on the host
    torch.cuda.synchronize()
    gpu_ms = 1e3 * (time.perf_counter() - t0) / n
    env.close()
    return {"env": kind, "cpu_ms_per_reset_step": cpu_ms, "cpu_steps": n_cpu, "cpu_kind": "port (oracle env, 1 core)",
            "b200_ms_per_reset_step": gpu_ms, "b200_steps": n,
            "note": "BASELINE configs[0]; wall clock, host buffers in and out"}


def main():
    args = parse()
    if args.impl == "reference":
        reference_arm(args)
    else:
        gpu_arm(args)


if __name__ == "__main__":
    main()
