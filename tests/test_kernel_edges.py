"""Kernels whose output the end-to-end tests cannot see, checked directly against plain references at the
edges of their tiles and launch grids.

* The DC start (pandapower init='dc'): Newton-Raphson overwrites it and converges from a wrong start as well,
  so it is read back with ``max_iteration=0`` -- ``va`` then holds the start angles untouched.  Reference:
  the oracle's own B' and P, one sparse solve per environment.  ``k_dc_start`` tiles 128 environments x 64
  angles per CTA with K in 16-bus slices; the grids and batch sizes below leave partial tiles in all three
  dimensions (97 buses: a last K slice of one bus; 372 buses: six angle tiles, the last 51 wide; 4133
  environments: 37 live rows in the last tile).
* The Philox generator and the two samplers built on it, against ``oracle/philox.py`` and the host build,
  at the edges of the elementwise launch grid: more than 128 column pairs (several blocks in x), more than
  8192 environment groups (the env-stride loop), environment ids across 2^32, seeds and streams >= 2^32.
"""
import ctypes as C
import functools

import numpy as np
import pytest
from scipy.sparse.linalg import splu

from oracle import pf, philox
from oracle.ppc_ref import GS, VA
from tests import common
from tests.hostsim import harness

DC_GRIDS = ("1-MV-rural--0-sw", "1-MV-comm--2-sw", "1-MV-semiurb--1-sw", "1-HV-urban--0-sw")   # 97 / 111 / 122 / 372 buses
DC_BATCHES = (1, 2, 127, 128, 129, 1000, 4133)
DC_BATCHES_HOST = (1, 2, 129)
N_INPUT = max(DC_BATCHES)
# name -> (pf_kernel, pf_kernel_used); every path launches the GEMM pre-pass, then the power-flow kernel
#   prepass      the GEMM pre-pass in front of whatever kernel auto picks (radial kernel on radial grids)
#   prepass_cta  the GEMM pre-pass in front of the CTA kernel
DC_PATHS = {"prepass": ("auto", None), "prepass_cta": ("cta", 1)}


@functools.lru_cache(maxsize=None)
def _case(name):
    return common.make_case(name, n_profile_steps=96)


@functools.lru_cache(maxsize=None)
def _dc_inputs(name):
    """Seeded Sbus of N_INPUT environments (kernel 1 on the host build) and the scipy DC angles of each."""
    case = _case(name)
    eng = harness.HostSimEngine(case.program, N_INPUT, max_iteration=0)
    common.randomize(case, eng, seed=5)
    eng.assemble()
    sbus = eng.sbus.copy()
    # spread the injections further apart than the sampled ranges do: angles of +-1 rad and more
    sbus *= np.random.default_rng(6).uniform(0.2, 3.0, N_INPUT)[:, None, None]
    ppc = case.program.ppc
    ref, pv, pq = pf.bus_types(ppc.bus, ppc.gen)
    pvpq = np.r_[pv, pq]
    bbus, pinj = pf.make_bdc(ppc.bus, ppc.branch)
    va_ref = np.radians(ppc.bus[:, VA])
    P = sbus[:, :, 0] - pinj[None, :] - ppc.bus[:, GS][None, :] / ppc.base_mva
    rhs = P[:, pvpq] - (bbus[pvpq][:, ref] @ va_ref[ref])[None, :]
    theta = splu(bbus[pvpq][:, pvpq].tocsc()).solve(np.ascontiguousarray(rhs.T)).T
    want = np.tile(va_ref, (N_INPUT, 1))
    want[:, pvpq] = theta
    return sbus, want, ref


def _radial(name):
    return name.startswith("1-MV")


def _paths(name):
    return [p for p in DC_PATHS if _radial(name) or p == "prepass"]


def _dc_engine(engine_cls, name, path, n=N_INPUT):
    pf_kernel, used = DC_PATHS[path]
    eng = engine_cls(_case(name).program, n, max_iteration=0, pf_kernel=pf_kernel)
    expect = used if used is not None else (3 if _radial(name) else 1)
    assert eng.info["pf_kernel_used"] == expect, (name, path, eng.info)
    return eng


def _dc_run(eng, sbus, n, sync=lambda: None):
    """Start angles of the first n environments; rows >= n of va must stay untouched."""
    put = (lambda dst, a: dst.__setitem__(slice(None), a)) if isinstance(eng.va, np.ndarray) else \
        (lambda dst, a: dst.copy_(eng._from_numpy(a)))
    put(eng.sbus, sbus[:eng.num_envs])
    put(eng.va, np.full(eng.va.shape, 7.0))
    batch = type(eng.batch).from_buffer_copy(eng.batch)
    batch.n_env = n
    before = eng.launch_count()
    eng.pf_solve(batch)
    sync()
    va = common._np(eng.va).copy()
    assert (va[n:] == 7.0).all(), "environments outside the batch were written"
    return va[:n], eng.launch_count() - before


def _check_dc(eng, name, path, batches, sync=lambda: None):
    sbus, want, ref = _dc_inputs(name)
    out = {}
    for n in batches:
        va, launches = _dc_run(eng, sbus, n, sync)
        if not isinstance(eng.va, np.ndarray):
            assert launches == 2, (path, launches)                     # the pre-pass ran
        assert np.isfinite(va).all()
        err = np.abs(va - want[:n]).max()
        assert err <= 1e-11, (name, path, n, err)
        assert np.array_equal(va[:, ref], want[:n, ref])               # slack angles are the bus table's
        out[n] = va
    return out


@pytest.mark.parametrize("name", DC_GRIDS)
def test_dc_prepass_matches_scipy_hostsim(name):
    for path in _paths(name):
        eng = _dc_engine(harness.HostSimEngine, name, path, n=max(DC_BATCHES_HOST))
        _check_dc(eng, name, path, DC_BATCHES_HOST)


@pytest.mark.gpu
@pytest.mark.parametrize("name", DC_GRIDS)
def test_dc_prepass_matches_scipy_and_host_loop_cuda(cuda_lib, name):
    """Every DC path within 1e-11 rad of scipy; the GEMM pre-pass equal, value for value, to the host build's
    plain loop (both accumulate fma(P, Binv, acc) in bus order; a padded term is fma(0, 0, acc))."""
    import torch
    from opfgym_b200.engine import Engine
    sbus = _dc_inputs(name)[0]
    for path in _paths(name):
        eng = _dc_engine(Engine, name, path)
        got = _check_dc(eng, name, path, DC_BATCHES, sync=torch.cuda.synchronize)
        # the same configuration on the host: B'^-1 is built with the factor of the grid's own ordering
        want_host, _ = _dc_run(_dc_engine(harness.HostSimEngine, name, path), sbus, N_INPUT)
        for n, va in got.items():
            assert (va == want_host[:n]).all(), (name, path, n)
        eng.close()


def _nan_row(engine_cls, sync=lambda: None):
    """One environment of a 128-environment tile gets NaN injections: only its row turns NaN, every other row
    is bit-identical to the run without it."""
    name = "1-MV-semiurb--1-sw"
    sbus = _dc_inputs(name)[0][:256].copy()
    ref = _dc_inputs(name)[2]
    eng = engine_cls(_case(name).program, 256, max_iteration=0, pf_kernel="cta")
    clean, _ = _dc_run(eng, sbus, 256, sync)
    sbus[77] = np.nan
    dirty, _ = _dc_run(eng, sbus, 256, sync)
    nonref = np.setdiff1d(np.arange(sbus.shape[1]), ref)
    assert np.isnan(dirty[77, nonref]).all()
    assert np.array_equal(dirty[77, ref], clean[77, ref])
    keep = np.arange(256) != 77
    assert np.array_equal(dirty[keep].view(np.int64), clean[keep].view(np.int64))


def test_dc_start_rows_do_not_leak_hostsim():
    _nan_row(harness.HostSimEngine)


@pytest.mark.gpu
def test_dc_start_rows_do_not_leak_cuda(cuda_lib):
    import torch
    from opfgym_b200.engine import Engine
    _nan_row(Engine, torch.cuda.synchronize)


# ---------------------------------------------------------------------------------------------------- RNG
PHILOX_COLS = (1, 2, 3, 7, 64, 65, 511, 513)
PHILOX_ENVS = (1, 3, 255, 257, 10000)
PHILOX_KEYS = [(first, seed, stream) for first in (0, 2**32 - 3) for seed in (0, 2**40 + 7) for stream in (0, 2**33 + 1)]


@functools.lru_cache(maxsize=None)
def _oracle_uniform(first, seed, stream):
    # column j of row b depends on (j // 2, first + b) only: one table serves every (n_env, n_cols) prefix
    return philox.uniform(seed, first, stream, max(PHILOX_ENVS), max(PHILOX_COLS))


class _HostBuffers:
    """numpy buffers + the host build (stream argument ignored)."""
    sync = staticmethod(lambda: None)

    def __init__(self):
        self.lib = harness.load()

    def empty(self, shape, dtype, fill):
        return np.full(shape, fill, dtype=dtype)

    def put(self, a):
        return np.ascontiguousarray(a).copy()

    def ptr(self, a):
        return a.ctypes.data

    def get(self, a):
        return a

    stream = None


class _CudaBuffers:
    """torch device buffers + the CUDA library on the current stream."""

    def __init__(self, lib):
        import torch
        self.torch, self.lib = torch, lib
        self.stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
        self.sync = torch.cuda.synchronize

    def empty(self, shape, dtype, fill):
        return self.torch.full(shape, fill, dtype=getattr(self.torch, np.dtype(dtype).name), device="cuda")

    def put(self, a):
        return self.torch.from_numpy(np.ascontiguousarray(a).copy()).cuda()

    def ptr(self, a):
        return a.data_ptr()

    def get(self, a):
        return a.cpu().numpy()


def _philox_cases(bufs):
    for first, seed, stream in PHILOX_KEYS:
        table = _oracle_uniform(first, seed, stream)
        for n_env in PHILOX_ENVS:
            out = bufs.empty((n_env, max(PHILOX_COLS)), np.float64, -1.0)
            for n_cols in PHILOX_COLS:
                assert bufs.lib.opfg_philox_uniform(seed, first, stream, n_env, n_cols, bufs.ptr(out), bufs.stream) == 0
                bufs.sync()
                flat = bufs.get(out).reshape(-1)          # out is [n_env, n_cols] row-major
                assert np.array_equal(flat[:n_env * n_cols].reshape(n_env, n_cols), table[:n_env, :n_cols]), \
                    (first, seed, stream, n_env, n_cols)
                assert (flat[n_env * n_cols:] == -1.0).all()


def test_philox_matches_oracle_at_grid_edges_hostsim():
    _philox_cases(_HostBuffers())


@pytest.mark.gpu
def test_philox_matches_oracle_at_grid_edges_cuda(cuda_lib):
    _philox_cases(_CudaBuffers(cuda_lib))


SAMPLE_COLS = (1, 2, 7, 65, 257, 513)
SAMPLE_ENVS = (1, 257, 10000)
SAMPLE_KEY = (2**32 - 3, 2**40 + 7, 2**33 + 1)      # first_env, seed, stream


def _ulps(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return np.abs(a - b) / np.spacing(np.maximum(np.abs(a), np.abs(b)))


def _sample_obs_cases(bufs, obs_dtype):
    """state[b, slots[j]] = (lo + (hi - lo) u) / dv and the observation cells obs_pos[j] on the way.
    lo >= 0, hi >= lo and dv a power of two: no cancellation and an exact division, so the FMA that nvcc forms
    of lo + w u moves the result by at most one ulp."""
    first, seed, stream = SAMPLE_KEY
    rng = np.random.default_rng(9)
    for n_cols in SAMPLE_COLS:
        n_state, n_obs = n_cols + 5, n_cols + 3
        slots = rng.permutation(n_state)[:n_cols].astype(np.int32)
        lo = rng.uniform(0.0, 5.0, n_cols)
        hi = lo + rng.uniform(0.0, 7.0, n_cols)
        dv = 2.0 ** rng.integers(-2, 3, n_cols)
        obs_pos = np.where(rng.random(n_cols) < 0.6, rng.permutation(n_obs)[:n_cols], -1).astype(np.int32)
        d_slots, d_lo, d_hi, d_dv, d_pos = (bufs.put(a) for a in (slots, lo, hi, dv, obs_pos))
        for n_env in SAMPLE_ENVS:
            state = bufs.empty((n_env, n_state), np.float64, -7.0)
            obs = bufs.empty((n_env, n_obs), obs_dtype, -9.0)
            o32, o64 = (bufs.ptr(obs), None) if obs_dtype == np.float32 else (None, bufs.ptr(obs))
            assert bufs.lib.opfg_sample_uniform_obs(seed, first, stream, n_env, n_cols, bufs.ptr(d_slots),
                                                    bufs.ptr(d_lo), bufs.ptr(d_hi), bufs.ptr(d_dv), bufs.ptr(state),
                                                    n_state, bufs.ptr(d_pos), o32, o64, n_obs, bufs.stream) == 0
            bufs.sync()
            S, O = bufs.get(state), bufs.get(obs)
            u = _oracle_uniform(first, seed, stream)[:n_env, :n_cols]
            want = (lo + (hi - lo) * u) / dv
            assert _ulps(S[:, slots], want).max() <= 1.0, (n_cols, n_env)
            untouched = np.setdiff1d(np.arange(n_state), slots)
            assert (S[:, untouched] == -7.0).all()
            seen = obs_pos >= 0
            assert np.array_equal(O[:, obs_pos[seen]], S[:, slots[seen]].astype(obs_dtype)), (n_cols, n_env)
            assert (np.delete(O, obs_pos[seen], axis=1) == -9.0).all()
            # the raw uniforms: the same generator with lo = 0, hi = 1, dv = 1 returns u itself
            if n_env == SAMPLE_ENVS[-1]:
                raw = bufs.empty((n_env, n_state), np.float64, -7.0)
                zero, one = bufs.put(np.zeros(n_cols)), bufs.put(np.ones(n_cols))
                assert bufs.lib.opfg_sample_uniform(seed, first, stream, n_env, n_cols, bufs.ptr(d_slots),
                                                    bufs.ptr(zero), bufs.ptr(one), bufs.ptr(one), bufs.ptr(raw),
                                                    n_state, bufs.stream) == 0
                bufs.sync()
                assert np.array_equal(bufs.get(raw)[:, slots], u)


@pytest.mark.parametrize("obs_dtype", [np.float32, np.float64])
def test_sample_uniform_obs_hostsim(obs_dtype):
    _sample_obs_cases(_HostBuffers(), obs_dtype)


@pytest.mark.gpu
@pytest.mark.parametrize("obs_dtype", [np.float32, np.float64])
def test_sample_uniform_obs_cuda(cuda_lib, obs_dtype):
    _sample_obs_cases(_CudaBuffers(cuda_lib), obs_dtype)


PROFILE_COLS = (1, 3, 64, 65, 257, 513)
PROFILE_ENVS = (1, 255, 10000)
# largest difference CUDA vs host build, in ulps of the larger result (B200: 1 / 3 / 3 measured).  none: the
# interpolation v r + t (1 - r) is one FMA on the device, one ulp; uniform: the factor u 2f + (1 - f) is an FMA as
# well, and a one-ulp change of the factor moves the product by up to two ulps, plus the interpolation's; normal:
# CUDA's log1p / cos / sqrt against glibc's on the noise term, which is at most noise_factor |z| < 0.9 of the value
PROFILE_ULPS = {0: 1.0, 1: 3.0, 2: 4.0}


def _profile_inputs(n_cols, n_env):
    rng = np.random.default_rng(11 + n_cols)
    n_steps = 40
    table = rng.uniform(0.1, 2.0, (n_steps, n_cols))
    table[:, ::5] *= -1.0                     # negative profile values (generation in load convention)
    slots = rng.permutation(n_cols + 3)[:n_cols].astype(np.int32)
    step = rng.integers(0, n_steps, n_env).astype(np.int64)
    step[-1] = n_steps - 1                    # interpolation towards the clamped last row
    return dict(slots=slots, table=table, step=step, r=rng.uniform(0.0, 1.0, n_env),
                pmin=np.full(n_cols, -1.7), pmax=np.full(n_cols, 1.8))      # some values are clipped


PROFILE_NOISE = 0.1


def _profile_run(bufs, inp, kind, interp):
    first, seed, stream = SAMPLE_KEY
    (n_steps, n_cols), n_env = inp["table"].shape, inp["step"].shape[0]
    n_state = n_cols + 3
    d = {k: bufs.put(v) for k, v in inp.items()}
    state = bufs.empty((n_env, n_state), np.float64, -7.0)
    assert bufs.lib.opfg_sample_profiles(seed, first, stream, n_env, n_cols, bufs.ptr(d["slots"]), bufs.ptr(d["table"]),
                                         n_steps, bufs.ptr(d["step"]), bufs.ptr(d["r"]) if interp else None,
                                         bufs.ptr(d["pmin"]), bufs.ptr(d["pmax"]), PROFILE_NOISE, kind, bufs.ptr(state),
                                         n_state, bufs.stream) == 0
    bufs.sync()
    out = bufs.get(state)
    assert (np.delete(out, inp["slots"], axis=1) == -7.0).all()
    return out[:, inp["slots"]]


def test_sample_profiles_host_semantics():
    """The host build against a numpy restatement: row gather, interpolation, noise, clip."""
    bufs = _HostBuffers()
    first, seed, stream = SAMPLE_KEY
    n_cols, n_env = 65, 257
    inp = _profile_inputs(n_cols, n_env)
    table, step, r, f = inp["table"], inp["step"], inp["r"][:, None], PROFILE_NOISE
    for kind in (0, 1, 2):
        for interp in (False, True):
            got = _profile_run(bufs, inp, kind, interp)
            v = table[step]
            if interp:
                v = v * r + table[np.minimum(step + 1, len(table) - 1)] * (1.0 - r)
            if kind == 1:
                u = philox.uniform(seed, first, stream, n_env, n_cols)
                v = v * (u * (2.0 * f) + (1.0 - f))
            elif kind == 2:
                u = philox.uniform(seed, first, stream, n_env, 2 * n_cols)
                z = np.sqrt(-2.0 * np.log1p(-u[:, :n_cols])) * np.cos(2.0 * np.pi * u[:, n_cols:])
                v = v + np.abs(v) * f * z
            want = np.clip(v, inp["pmin"], inp["pmax"])
            if kind < 2:
                assert np.array_equal(got, want), (kind, interp)
            else:                              # numpy's log1p / cos need not be glibc's
                assert _ulps(got, want).max() <= PROFILE_ULPS[2], (kind, interp)


@pytest.mark.gpu
@pytest.mark.parametrize("kind", [0, 1, 2])
def test_sample_profiles_cuda_vs_host(cuda_lib, kind):
    cuda, host = _CudaBuffers(cuda_lib), _HostBuffers()
    worst = 0.0
    for n_cols in PROFILE_COLS:
        for n_env in PROFILE_ENVS:
            inp = _profile_inputs(n_cols, n_env)
            for interp in (False, True):
                a = _profile_run(cuda, inp, kind, interp)
                b = _profile_run(host, inp, kind, interp)
                assert np.isfinite(a).all()
                worst = max(worst, _ulps(a, b).max())
    assert worst <= PROFILE_ULPS[kind], (kind, worst)
