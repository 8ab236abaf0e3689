"""The kernels that prepare every next episode, checked directly against plain references.

* ``k_row_program`` (the env hooks) against a numpy restatement of ``row_program_exec``, vectorised over
  (environment, item): every op, NaN / +-inf / -0.0 / negative square roots / division by zero, all 16 registers
  live at once, the 96-op maximum, LOAD_STATIC, a permuted ``select_rows`` subset; 1 to 600 items (several blocks
  in x once the item width is capped at 256) and up to 10 000 environments (past the 8192-group cap of the
  env-stride loop).  One op per statement on both sides, no FMA: equal to the bit (NaN payloads aside).
* The hook compiler (``rowprog.py``) against the value semantics of the hook as written: random expression DAGs
  over real columns, evaluated with torch float64 in statement order, handles read before and after a store to
  their own column.
* ``k_reset<128>`` (the fused reset) against the same trace replayed as separate launches on the same engine, from
  a sentinel-filled state: stage grouping and hazards, item spreading, the row placement rules (copy-in, no
  copy-in, global row), random / centre initial action, f32 / f64 observations.  Bit for bit.
* ``k_observe`` against a numpy gather, with and without ``bus_wise_obs`` sums, with constant references.
"""
import ctypes as C
import functools

import numpy as np
import pytest
import torch

from opfgym_b200 import capi, envs
from opfgym_b200 import ppc as P
from opfgym_b200.compiler import Compiler
from opfgym_b200.rowprog import (ABS, ADD, CONST, DIV, LOAD_STATE, LOAD_STATIC, MAX, MIN, MUL, N_REG, NEG, SQRT,
                                 STORE_STATE, SUB, CompiledRowProgram)
from tests import common
from tests.hostsim import harness
from tests.test_kernel_edges import _CudaBuffers, _HostBuffers


def _same(a, b):
    """Equal to the bit, except that any NaN equals any NaN (x86 and CUDA produce different NaN payloads)."""
    a, b = np.asarray(a), np.asarray(b)
    if a.shape != b.shape or a.dtype != b.dtype:
        return False
    na, nb = np.isnan(a), np.isnan(b)
    if not np.array_equal(na, nb):
        return False
    ia = a[~na].view(np.int64 if a.dtype == np.float64 else np.int32)
    ib = b[~nb].view(np.int64 if b.dtype == np.float64 else np.int32)
    return np.array_equal(ia, ib)


# ------------------------------------------------------------------------------- A. k_row_program vs numpy
ROW_ITEMS = (1, 255, 256, 257, 600)
SENTINEL = -7.25


def _col(k, n_items):
    """Start of program column k: columns n_items apart (items never share a cell), cell 0 left as padding."""
    return 1 + k * n_items


def _prog_every_op(n):
    """Every op once, in the register pattern of the hooks (a result overwriting one of its operands)."""
    c = functools.partial(_col, n_items=n)
    ops = [(LOAD_STATE, 0, c(0), 0, 0.0), (LOAD_STATE, 1, c(1), 0, 0.0), (LOAD_STATIC, 2, 0, 0, 0.0),
           (CONST, 3, 0, 0, 2.5),
           (ADD, 4, 0, 1, 0.0), (SUB, 5, 0, 2, 0.0), (MUL, 6, 1, 3, 0.0), (DIV, 7, 0, 1, 0.0),
           (SQRT, 8, 0, 0, 0.0), (NEG, 9, 1, 0, 0.0), (MIN, 10, 0, 2, 0.0), (MAX, 11, 1, 3, 0.0),
           (ABS, 12, 0, 0, 0.0), (ADD, 4, 4, 7, 0.0), (DIV, 3, 3, 1, 0.0)]
    ops += [(STORE_STATE, 0, c(2 + k), r, 0.0) for k, r in enumerate((4, 5, 6, 8, 9, 10, 11, 12, 3))]
    ops.append((STORE_STATE, 0, c(1), 7, 0.0))           # in place over an input column
    return ops, 1, 11


def _prog_all_registers(n):
    """All 16 registers loaded before the first one is combined: 8 state columns (stored back in place), 4 statics,
    4 constants."""
    c = functools.partial(_col, n_items=n)
    ops = [(LOAD_STATE, k, c(k), 0, 0.0) for k in range(8)]
    ops += [(LOAD_STATIC, 8 + k, k * n, 0, 0.0) for k in range(4)]
    ops += [(CONST, 12 + k, 0, 0, v) for k, v in enumerate((0.75, -3.0, 1e300, -1e-300))]
    ops += [(MUL, 0, 0, 8, 0.0), (ADD, 1, 1, 9, 0.0), (SUB, 2, 2, 10, 0.0), (DIV, 3, 3, 11, 0.0),
            (MIN, 4, 4, 12, 0.0), (MAX, 5, 5, 13, 0.0), (MUL, 6, 6, 14, 0.0), (DIV, 7, 7, 15, 0.0)]
    ops += [(STORE_STATE, 0, c(k), k, 0.0) for k in range(8)]
    return ops, 4, 8


def _prog_max_ops(n):
    """Exactly 96 ops.  MIN / MAX always meet the constant 1.25 (fmin of +0 and -0 may return either zero)."""
    c = functools.partial(_col, n_items=n)
    ops = [(LOAD_STATE, 0, c(0), 0, 0.0), (LOAD_STATE, 1, c(1), 0, 0.0), (CONST, 2, 0, 0, 1.25),
           (LOAD_STATIC, 3, 0, 0, 0.0)]
    cycle = [(ADD, 0, 0, 1), (MUL, 1, 1, 2), (SUB, 3, 3, 0), (DIV, 0, 0, 3), (ABS, 1, 1, 0), (SQRT, 3, 1, 0),
             (NEG, 0, 0, 0), (MIN, 1, 1, 2), (MAX, 3, 2, 3), (ADD, 1, 3, 0), (DIV, 3, 2, 1)]
    k = 0
    while len(ops) < 94:
        ops.append((*cycle[k % len(cycle)], 0.0))
        k += 1
    ops += [(STORE_STATE, 0, c(2), 0, 0.0), (STORE_STATE, 0, c(3), 3, 0.0)]
    assert len(ops) == 96
    return ops, 1, 4


ROW_PROGRAMS = {"every_op": _prog_every_op, "all_registers": _prog_all_registers, "max_ops": _prog_max_ops}
N_INPUT_COLS = {"every_op": 2, "all_registers": 8, "max_ops": 2}


def _special_values(rng, shape, zeros=True):
    """Uniform values with NaN, +-inf, -0.0 (and +0.0 if `zeros`) and negatives mixed in."""
    v = rng.uniform(-4.0, 4.0, shape)
    pick = rng.random(shape)
    specials = [np.nan, np.inf, -np.inf, -0.0] + ([0.0] if zeros else [])
    for k, s in enumerate(specials):
        v[(pick >= 0.02 * k) & (pick < 0.02 * (k + 1))] = s
    return v


def _row_inputs(name, n, n_env, n_state, seed):
    rng = np.random.default_rng(seed)
    S = np.full((n_env, n_state), SENTINEL)
    for k in range(N_INPUT_COLS[name]):
        # column 0 meets the statics and constants in MIN / MAX: -0.0 only, never +0.0
        S[:, _col(k, n):_col(k, n) + n] = _special_values(rng, (n_env, n), zeros=k != 0)
    n_static = ROW_PROGRAMS[name](n)[1]
    statics = _special_values(rng, n_static * n, zeros=False)
    statics[statics == 0.0] = 0.5
    return S, statics


def _row_reference(ops, statics, rows, S):
    """row_program_exec, one op at a time over every (environment, item); S is updated in place."""
    items = np.asarray(rows)
    R = {}
    with np.errstate(all="ignore"):
        for op, dst, a, b, imm in ops:
            if op == LOAD_STATE:
                R[dst] = S[:, a + items].copy()
            elif op == LOAD_STATIC:
                R[dst] = np.broadcast_to(statics[a + items], (S.shape[0], len(items))).copy()
            elif op == CONST:
                R[dst] = np.full((S.shape[0], len(items)), imm)
            elif op == STORE_STATE:
                S[:, a + items] = R[b]
            else:
                x = R[a]
                y = R[b] if op in (ADD, SUB, MUL, DIV, MIN, MAX) else None
                R[dst] = {ADD: lambda: x + y, SUB: lambda: x - y, MUL: lambda: x * y, DIV: lambda: x / y,
                          SQRT: lambda: np.sqrt(x), NEG: lambda: -x, MIN: lambda: np.fmin(x, y),
                          MAX: lambda: np.fmax(x, y), ABS: lambda: np.abs(x)}[op]()
    return S


def _row_program(lib, n_rows, ops, statics, rows=None):
    arr = (capi.RowOp * len(ops))(*[capi.RowOp(*o) for o in ops])
    st = np.ascontiguousarray(statics if len(statics) else np.zeros(1), np.float64)
    h = C.c_void_p()
    capi.check(lib, lib.opfg_row_program_create(n_rows, len(ops), arr, len(statics),
                                                st.ctypes.data_as(C.POINTER(C.c_double)), C.byref(h)))
    if rows is not None:
        r = np.ascontiguousarray(rows, np.int32)
        capi.check(lib, lib.opfg_row_program_select_rows(h, len(r), r.ctypes.data_as(C.POINTER(C.c_int32))))
    return h


def _row_program_cases(bufs, env_counts):
    lib = bufs.lib
    for name, make in ROW_PROGRAMS.items():
        for n in ROW_ITEMS:
            ops, _, n_cols = make(n)
            n_state = _col(n_cols, n) + 2                       # two padding cells behind the last column
            selections = [None]
            if name == "every_op":
                selections.append(np.random.default_rng(n).permutation(n)[:max(1, 2 * n // 3)])
            for rows in selections:
                for n_env in env_counts:
                    S0, statics = _row_inputs(name, n, n_env, n_state, seed=n_env + n)
                    h = _row_program(lib, n, ops, statics, rows)
                    try:
                        d = bufs.put(S0)
                        capi.check(lib, lib.opfg_row_program_run(h, n_env, bufs.ptr(d), n_state, bufs.stream))
                        bufs.sync()
                        got = bufs.get(d)
                    finally:
                        lib.opfg_row_program_destroy(h)
                    items = np.arange(n) if rows is None else rows
                    want = S0.copy()
                    for e0 in range(0, n_env, 2000):               # bounded memory at 10 000 x 600 items
                        want[e0:e0 + 2000] = _row_reference(ops, statics, items, S0[e0:e0 + 2000].copy())
                    key = (name, n, rows is not None, n_env)
                    assert _same(got, want), key
                    stored = np.zeros(n_state, bool)
                    for o in ops:
                        if o[0] == STORE_STATE:
                            stored[o[2] + items] = True
                    assert _same(got[:, ~stored], S0[:, ~stored]), key      # sentinels and inputs untouched


def test_row_program_matches_numpy_hostsim():
    _row_program_cases(_HostBuffers(), (1, 3, 257))


@pytest.mark.gpu
def test_row_program_matches_numpy_cuda(cuda_lib):
    _row_program_cases(_CudaBuffers(cuda_lib), (1, 3, 10000))


def test_row_program_rejects_more_than_96_ops():
    lib = harness.load()
    ops = _prog_max_ops(4)[0]
    ops = ops[:-1] + [(NEG, 0, 0, 0, 0.0)] + ops[-1:]
    with pytest.raises(capi.OpfgError, match="96"):
        _row_program(lib, 4, ops, np.ones(4))


# ------------------------------------------------------------------------------- E. cells past the state row
def test_row_program_rejects_cells_past_the_state_row():
    """opfg_row_program_run refuses a program whose largest cell (column start + largest item row) does not fit the
    row.  The buffer is padded past the last row, so a write that slipped through lands in memory the test owns."""
    lib = harness.load()
    n_state, n_env = 10, 3
    buf = np.full(n_env * n_state + 16, SENTINEL)

    def run(a, n_rows, rows=None, op=STORE_STATE):
        o = (LOAD_STATE, 0, a, 0, 0.0) if op == LOAD_STATE else (CONST, 0, 0, 0, 1.5)
        ops = [o, (STORE_STATE, 0, 0 if op == LOAD_STATE else a, 0, 0.0)]
        h = _row_program(lib, n_rows, ops, np.zeros(0), rows)
        try:
            return lib.opfg_row_program_run(h, n_env, buf.ctypes.data, n_state, None)
        finally:
            lib.opfg_row_program_destroy(h)

    assert run(7, 4) != 0                           # cells 7..10 of a 10-cell row
    assert b"cell 10 of a 10-cell" in lib.opfg_last_error()
    assert run(7, 4, op=LOAD_STATE) != 0            # reading past the row is refused as well
    assert (buf == SENTINEL).all()
    assert run(9, 8, rows=[0]) == 0                 # the selected rows decide: cell 9 only
    assert run(8, 8, rows=[3, 1]) != 0              # cell 11
    assert (buf.reshape(-1)[n_env * n_state:] == SENTINEL).all()
    assert run(6, 4) == 0                           # cells 6..9: the last cell of the row is fine
    assert (buf[:n_env * n_state].reshape(n_env, n_state)[:, 6:] == 1.5).all()
    assert (buf[n_env * n_state:] == SENTINEL).all()
    with pytest.raises(capi.OpfgError, match="negative state cell"):
        _row_program(lib, 2, [(LOAD_STATE, 0, -1, 0, 0.0), (STORE_STATE, 0, 4, 0, 0.0)], np.zeros(0))


# ------------------------------------------------------------------------------- B. the hook compiler
def _vc_env(engine):
    kw = dict(num_envs=3, train_data="full_uniform", test_data="full_uniform", seed=3, n_profile_steps=96)
    if engine == "host":
        return envs.VoltageControl(engine_cls=harness.TorchHostSimEngine, **kw)
    return envs.VoltageControl(prefetch_reset=False, **kw)


class _Shadow:
    """A handle paired with the value the hook means by it (torch float64, [n_env, n_rows])."""

    def __init__(self, expr, value):
        self.expr, self.value = expr, value


def _value_equal(a, b):
    """Exact equality of values; NaN equals NaN and -0.0 equals +0.0 (fmin / fmax of two opposite zeros may return
    either of them)."""
    return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


def _sqrt(t):
    """IEEE square root (torch's vectorised CPU sqrt is not always correctly rounded; numpy's is)."""
    return torch.as_tensor(np.sqrt(t.cpu().numpy()), device=t.device)


def _random_hook(rng, env, table, n_stores):
    """A random hook on ``table``; after it ran, ``build.want`` holds the reference's column values.  Handles are taken before and after stores to their own column, subexpressions are shared."""
    lay = env.program.layout
    state_cols = [c for (t, c) in lay.columns if t == table]
    static_cols = [c for c in ("scaling", "max_max_p_mw", "mean_p_mw") if c in env.net[table] and not lay.has(table, c)]
    targets = state_cols + [c for (t, c) in env.pruned_columns if t == table]

    def build(r):
        cur = {c: env.col(table, c).clone().double() for c in state_cols}
        pool = []

        def handle(c):
            if c in state_cols:
                return _Shadow(r.col(c), cur[c].clone())
            return _Shadow(r.col(c), env.static(table, c).double().expand_as(next(iter(cur.values()))))

        def combine(depth):
            if depth == 0 or rng.random() < 0.25:
                if pool and rng.random() < 0.5:
                    return pool[rng.integers(len(pool))]              # shared subexpression / older handle
                cols = state_cols + static_cols
                h = handle(cols[rng.integers(len(cols))])
                pool.append(h)
                return h
            kind = rng.integers(12)
            x = combine(depth - 1)
            k = float(rng.choice([0.5, 1.5, -2.0, 3.0]))
            if kind < 4:
                y = combine(depth - 1)
                f = [(lambda p, q: p + q), (lambda p, q: p - q), (lambda p, q: p * q), (lambda p, q: p / q)][kind]
                out = _Shadow(f(x.expr, y.expr), f(x.value, y.value))
            elif kind == 4:
                out = _Shadow(k - x.expr, k - x.value)                 # reflected ops with constants
            elif kind == 5:
                out = _Shadow(k / x.expr, torch.full_like(x.value, k) / x.value)   # not k * x.reciprocal()
            elif kind == 6:
                out = _Shadow(x.expr ** 2, x.value * x.value)
            elif kind == 7:
                out = _Shadow(abs(x.expr) ** 0.5, _sqrt(torch.abs(x.value)))
            elif kind == 8:
                y = combine(depth - 1)
                out = _Shadow(x.expr.minimum(y.expr), torch.fmin(x.value, y.value))
            elif kind == 9:
                out = _Shadow(x.expr.maximum(k), torch.fmax(x.value, torch.full_like(x.value, k)))
            elif kind == 10:
                out = _Shadow(-x.expr, -x.value)
            else:
                out = _Shadow(k * x.expr + k, x.value * k + k)
            if rng.random() < 0.4:
                pool.append(out)
            return out

        for _ in range(n_stores):
            v = combine(3)
            col = targets[rng.integers(len(targets))]
            r.store(col, v.expr)
            if col in cur:
                cur[col] = v.value.clone()
            if rng.random() < 0.5:
                pool.append(handle(col) if col in cur else v)        # a handle taken after the store
        build.want, build.stores = cur, r.stores

    return build


def _check_hook(env, name, table, build):
    before = {c: env.col(table, c).clone() for (t, c) in env.program.layout.columns if t == table}
    env.run_row_program(name, table, build)
    live = env.program.read_cells
    lay = env.program.layout
    loaded, stack = set(), [e for _, e in build.stores]
    while stack:
        e = stack.pop()
        loaded.add(e.start) if e.op == LOAD_STATE else None
        stack += e.args
    for col, old in before.items():
        got, want = env.col(table, col).double().cpu(), build.want[col].cpu()
        start = lay.columns[(table, col)][0]
        rows = np.arange(old.shape[1])
        # a store is computed where some kernel reads the cell, or everywhere if the hook reads the column itself
        on = torch.as_tensor([(start + r) in live or start in loaded for r in rows])
        assert _value_equal(got[:, on], want[:, on]), (name, col)
        assert _same(got[:, ~on].numpy(), old.double().cpu()[:, ~on].numpy()), (name, col)     # pruned rows


def _hook_cases(engine):
    env = _vc_env(engine)
    env.reset(seed=3)
    for k in range(12):
        build = _random_hook(np.random.default_rng(100 + k), env, "sgen", n_stores=4 + k % 3)
        _check_hook(env, f"random{k}", "sgen", build)


def test_hook_compiler_matches_statement_order_hostsim():
    _hook_cases("host")


@pytest.mark.gpu
def test_hook_compiler_matches_statement_order_cuda(cuda_lib):
    _hook_cases("cuda")


def test_handle_read_before_a_store_to_its_column_keeps_the_old_value():
    """``a = r.col("p_mw"); r.store("p_mw", 0); r.store("max_q_mvar", 2 a)``: the second store sees the p_mw the
    handle was taken on, as the same statements on pandas columns would; a handle taken afterwards sees 0."""
    env = _vc_env("host")
    env.reset(seed=3)
    p_old = env.col("sgen", "p_mw").clone()

    def build(r):
        a = r.col("p_mw")
        r.store("p_mw", 0.0)
        r.store("max_q_mvar", a * 2.0)
        r.store("min_q_mvar", r.col("p_mw") - 1.0)
    env.run_row_program("probe", "sgen", build)
    assert (env.col("sgen", "p_mw") == 0.0).all()
    live = np.asarray([env.program.layout.columns[("sgen", "max_q_mvar")][0] + r in env.program.read_cells
                       for r in range(p_old.shape[1])])
    assert live.sum() >= 10
    assert torch.equal(env.col("sgen", "max_q_mvar")[:, live], p_old[:, live] * 2.0)
    assert (env.col("sgen", "min_q_mvar")[:, live] == -1.0).all()


def test_hook_register_pressure():
    """A right-nested sum ``1 + (2 + (... + p_mw))`` holds one register per term: 16 terms compile and give the
    right value, 17 are refused."""
    env = _vc_env("host")
    env.reset(seed=3)

    def nested(n):
        def build(r):
            e = r.col("p_mw")
            for k in range(n - 1, 0, -1):
                e = float(k) + e
            r.store("max_q_mvar", e)
        return build
    p = env.col("sgen", "p_mw").clone()
    env.run_row_program("p16", "sgen", nested(16))
    want = p.clone()
    for k in range(15, 0, -1):
        want = float(k) + want
    live = np.asarray([env.program.layout.columns[("sgen", "max_q_mvar")][0] + r in env.program.read_cells
                       for r in range(p.shape[1])])
    assert torch.equal(env.col("sgen", "max_q_mvar")[:, live], want[:, live])
    with pytest.raises(RuntimeError, match="more than 16 registers"):
        env.run_row_program("p17", "sgen", nested(17))
    assert N_REG == 16


# ------------------------------------------------------------------------------- C. the fused reset
@functools.lru_cache(maxsize=None)
def _reset_case():
    return common.make_case("1-MV-semiurb--1-sw", n_profile_steps=96)


def _compile(obs_keys, bus_wise_obs=False, prepare=None):
    """The stand-in case's layout (state keys, actions, constraints) with other observation keys."""
    case = _reset_case() if prepare is None else common.make_case("1-MV-semiurb--1-sw", n_profile_steps=96,
                                                                     prepare=prepare)
    net = case.net
    obs = [(t, c, idx(net) if callable(idx) else idx) for t, c, idx in obs_keys]
    return Compiler(net, P.PpcBuilder(net)).compile(case.act_keys, obs, case.obs_keys, case.constraints,
                                                     case.reward, bus_wise_obs=bus_wise_obs)


@functools.lru_cache(maxsize=None)
def _input_obs_program():
    """Observation of input cells only (so the fused reset may keep the row in shared memory); its first run of
    consecutive cells is longer than 3 x 128, which takes both loops of gather_obs at 128 threads."""
    return _compile([("sgen", "p_mw", lambda n: n.sgen.index), ("storage", "p_mw", lambda n: n.storage.index),
                     ("load", "p_mw", lambda n: n.load.index), ("load", "q_mvar", lambda n: n.load.index),
                     ("sgen", "q_mvar", lambda n: n.sgen.index[::20])])


def _runs(obs_ref):
    runs, i = [], 0
    while i < len(obs_ref):
        j = i + 1
        while j < len(obs_ref) and obs_ref[j] == obs_ref[j - 1] + 1:
            j += 1
        runs.append(j - i)
        i = j
    return runs


def _put(dst, a):
    if isinstance(dst, np.ndarray):
        dst[...] = a
    elif np.isscalar(a):
        dst.fill_(a)
    else:
        dst.copy_(torch.as_tensor(np.ascontiguousarray(a)).to(dst.device, dst.dtype))


def _sampler(eng, rng, cells, stream_id):
    n = len(cells)
    lo = rng.uniform(-2.0, 3.0, n)
    hi = lo + rng.uniform(0.0, 4.0, n)
    dv = 2.0 ** rng.integers(-2, 3, n)
    return ("sample", eng._from_numpy(np.asarray(cells, np.int32)), eng._from_numpy(lo), eng._from_numpy(hi),
            eng._from_numpy(dv), stream_id)


def _program(eng, rng, n_rows, src, dst, rows=None):
    """dst[row] = src[row] * static[row] + 0.5 (src == dst: a read-modify-write)."""
    ops = [(LOAD_STATE, 0, src, 0, 0.0), (LOAD_STATIC, 1, 0, 0, 0.0), (MUL, 0, 0, 1, 0.0), (CONST, 2, 0, 0, 0.5),
           (ADD, 0, 0, 2, 0.0), (STORE_STATE, 0, dst, 0, 0.0)]
    return ("program", CompiledRowProgram(eng, n_rows, ops, rng.uniform(0.5, 1.5, n_rows), rows))


def _plans(eng, n_in, base):
    """Traces that steer each branch of opfg_reset_plan_create / opfg_reset_episode.  Input cells are 0..n_in-1."""
    rng = np.random.default_rng(17)
    S = lambda cells, k: _sampler(eng, rng, cells, base + k)
    everything_but = lambda lo, hi: [c for c in rng.permutation(n_in) if not lo <= c < hi]
    yield "one_group_wrapping", [           # disjoint: one group, 51 + 39 + 150 items spread over 128 threads
        S(range(0, 101), 1), S(range(101, 178), 2),
        _program(eng, rng, 150, 200, 400)]
    yield "hazards", [                      # RAW, WAR, WAW between neighbours: four groups
        S(range(0, 64), 1),
        _program(eng, rng, 64, 0, 100, rows=rng.permutation(64)[:45]),
        S(range(50, 61), 2),
        S(range(55, 71), 3),
        _program(eng, rng, 200, 300, 100)]
    yield "big_stage_untouched_cells", [    # a 300-item program stage; most cells keep the state's values
        _program(eng, rng, 300, 10, 320), S(range(0, 7), 1)]
    yield "all_written_first", [            # every input cell written before it is read: no copy-in
        S(rng.permutation(n_in), 1), _program(eng, rng, 200, 0, 300)]
    yield "read_before_write", [            # reads cells 0..149 before the sampler writes them
        _program(eng, rng, 150, 0, 200), S(everything_but(200, 350), 1)]
    yield "read_modify_write", [            # the first writer of cells 0..149 reads them itself
        _program(eng, rng, 150, 0, 0), S(everything_but(0, 150), 1)]
    yield "global_row", [                   # a store at or above n_inputs: the row stays in global memory
        S(range(0, 99), 1), _program(eng, rng, 99, 0, n_in + 5)]


def _replay(eng, trace, seed, first_env, base, random_action, act_off):
    for item in trace:
        if item[0] == "sample":
            _, slots, lo, hi, dv, sid = item
            eng.sample_uniform(slots, lo, hi, dv, seed, first_env, sid)
        else:
            item[1].run()
    if random_action:
        eng.philox_uniform(eng.actions_reset, seed, first_env, base + act_off)
    else:
        _put(eng.actions_reset, 0.5)
    eng.assemble(scatter_sbus=False)
    eng.observe()


def _fused_reset_cases(engine_cls, env_counts, sync=lambda: None):
    program = _input_obs_program()
    n_in, n_state = program.layout.n_inputs, program.layout.n
    obs_ref = np.asarray(program.scoring["obs_ref"])
    runs = _runs(obs_ref)
    assert (obs_ref < n_in).all() and program.scoring["obs_ptr"] is None
    assert max(runs) > 3 * 128 and max(runs) % 128 and len(runs) <= 64 and 8 * len(runs) <= len(obs_ref)
    seed, first_env, base = 2**40 + 3, 2**32 - 2, 64 * 5
    for obs_dtype in ("float32", "float64"):
        for n_env in env_counts:
            eng = engine_cls(program, n_env, obs_dtype=obs_dtype)
            sentinel = -1000.0 - np.arange(n_state) - 1e4 * np.arange(n_env)[:, None]
            for name, trace in _plans(eng, n_in, base):
                plan = eng.make_reset_plan(trace, base)
                act_off = len(trace) + 1
                for random_action in (0, 1):
                    out = []
                    for fused in (True, False):
                        _put(eng.state, sentinel)
                        _put(eng.actions_reset, -3.0)
                        _put(eng.obs, -9.0)
                        if fused:
                            eng.reset_episode(plan, seed, first_env, base, random_action, act_off)
                        else:
                            _replay(eng, trace, seed, first_env, base, random_action, act_off)
                        sync()
                        out.append([common._np(t).copy() for t in (eng.state, eng.actions_reset, eng.obs)])
                    key = (name, obs_dtype, n_env, random_action)
                    for what, f, s in zip(("state", "actions_reset", "obs"), *out):
                        assert _same(f, s), (what, key)
                    assert not (out[0][0][:, :n_in] == sentinel[:, :n_in]).all(), key
            eng.close()


def test_fused_reset_plans_equal_separate_launches_hostsim():
    _fused_reset_cases(harness.HostSimEngine, (1, 3))


@pytest.mark.gpu
def test_fused_reset_plans_equal_separate_launches_cuda(cuda_lib):
    from opfgym_b200.engine import Engine
    _fused_reset_cases(Engine, (1, 3, 129, 1000), torch.cuda.synchronize)


# ------------------------------------------------------------------------------- D. k_observe vs numpy
def _shared_load_buses(net):
    """Loads 0..29 move to ten buses, three each: groups of several loads for bus_wise_obs."""
    net.load.loc[net.load.index[:30], "bus"] = np.repeat(net.load.bus.to_numpy()[:10], 3)


@functools.lru_cache(maxsize=None)
def _observe_program(bus_wise):
    return _compile([("load", "p_mw", lambda n: n.load.index), ("load", "q_mvar", lambda n: n.load.index),
                     ("sgen", "p_mw", lambda n: n.sgen.index),
                     ("sgen", "mean_p_mw", lambda n: n.sgen.index[:7]),           # static column: constant refs
                     ("res_bus", "vm_pu", lambda n: n.bus.index[:5])],
                    bus_wise_obs=bus_wise, prepare=_shared_load_buses)


def _observe_reference(program, S, obs_dtype):
    ref = np.asarray(program.scoring["obs_ref"])
    consts = np.asarray(program.consts, float)
    vals = np.where(ref >= 0, S[:, np.maximum(ref, 0)], consts[np.maximum(-ref - 1, 0)][None, :])
    if program.scoring["obs_ptr"] is None:                  # one reference per observation
        return vals.astype(obs_dtype)
    ptr = np.asarray(program.scoring["obs_ptr"])
    out = np.zeros((S.shape[0], len(ptr) - 1))
    for k in range(np.diff(ptr).max()):                     # v = 0.0; v += each member, in order
        j = np.nonzero(ptr[:-1] + k < ptr[1:])[0]
        out[:, j] = out[:, j] + vals[:, ptr[j] + k]
    return out.astype(obs_dtype)


def _observe_cases(engine_cls, env_counts, sync=lambda: None):
    for bus_wise in (False, True):
        program = _observe_program(bus_wise)
        ref = np.asarray(program.scoring["obs_ref"])
        assert (ref < 0).sum() >= 7 and program.n_obs > 256
        assert (program.scoring["obs_ptr"] is not None) == bus_wise
        if bus_wise:
            assert np.diff(program.scoring["obs_ptr"]).max() == 3
        for obs_dtype in ("float32", "float64"):
            for n_env in env_counts:
                eng = engine_cls(program, n_env, obs_dtype=obs_dtype)
                rng = np.random.default_rng(n_env)
                S = rng.uniform(-50.0, 50.0, (n_env, program.layout.n))
                S[rng.random(S.shape) < 0.002] = np.nan
                _put(eng.state, S)
                _put(eng.obs, -9.0)
                eng.observe()
                sync()
                got = common._np(eng.obs)
                assert _same(got, _observe_reference(program, S, obs_dtype)), (bus_wise, obs_dtype, n_env)
                eng.close()


def test_observe_matches_numpy_hostsim():
    _observe_cases(harness.HostSimEngine, (1, 257))


@pytest.mark.gpu
def test_observe_matches_numpy_cuda(cuda_lib):
    from opfgym_b200.engine import Engine
    _observe_cases(Engine, (1, 10000), torch.cuda.synchronize)
