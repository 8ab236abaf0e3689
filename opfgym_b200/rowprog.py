"""Row programs: the per-sample hooks of the reference envs as ONE kernel launch.

The reference's ``_sampling`` overrides (``opfgym/envs/voltage_control.py:121-133``,
``load_shedding.py:131-149``, ``max_renewable.py:101-105``) are row-wise formulas
on the columns of one net table.  Here a hook writes the same formulas with
ordinary Python operators on column handles; the expression DAG is compiled once
into a short register program (``OpfgRowOp`` list, see ``include/opfg_b200.h``)
that the library runs for all environments and rows in a single launch.

    with env.row_program("sgen") as r:
        p = r.col("p_mw") * r.col("scaling")
        r.store("max_p_mw", p + 1e-9)
        q = ((r.col("max_s_mva") ** 2 - (p + 1e-9) ** 2)).sqrt()
        r.store("min_q_mvar", -q); r.store("max_q_mvar", q); r.store("q_mvar", 0.0)
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import capi

LOAD_STATE, LOAD_STATIC, CONST, ADD, SUB, MUL, DIV, SQRT, NEG, MIN, MAX, ABS, STORE_STATE = range(13)
N_REG = 16


class Expr:
    __slots__ = ("op", "args", "imm", "start", "seq")

    def __init__(self, op, args=(), imm=0.0, start=0, seq=0):
        # seq (LOAD_STATE): stores made before the handle -- it reads the column as it was then
        self.op, self.args, self.imm, self.start, self.seq = op, tuple(args), float(imm), int(start), int(seq)

    @staticmethod
    def wrap(v):
        return v if isinstance(v, Expr) else Expr(CONST, imm=float(v))

    def __add__(self, o): return Expr(ADD, (self, Expr.wrap(o)))
    def __radd__(self, o): return Expr(ADD, (Expr.wrap(o), self))
    def __sub__(self, o): return Expr(SUB, (self, Expr.wrap(o)))
    def __rsub__(self, o): return Expr(SUB, (Expr.wrap(o), self))
    def __mul__(self, o): return Expr(MUL, (self, Expr.wrap(o)))
    def __rmul__(self, o): return Expr(MUL, (Expr.wrap(o), self))
    def __truediv__(self, o): return Expr(DIV, (self, Expr.wrap(o)))
    def __rtruediv__(self, o): return Expr(DIV, (Expr.wrap(o), self))
    def __neg__(self): return Expr(NEG, (self,))
    def __abs__(self): return Expr(ABS, (self,))

    def __pow__(self, e):
        if e == 2:
            return Expr(MUL, (self, self))
        if e == 0.5:
            return Expr(SQRT, (self,))
        raise NotImplementedError("only **2 and **0.5")

    def sqrt(self): return Expr(SQRT, (self,))
    def minimum(self, o): return Expr(MIN, (self, Expr.wrap(o)))
    def maximum(self, o): return Expr(MAX, (self, Expr.wrap(o)))


class RowProgram:
    """Context manager collecting stores; compiled and cached by the env on exit."""

    def __init__(self, env, table: str):
        self.env, self.table = env, table
        self.n_rows = len(env.net[table])
        self.statics: list[np.ndarray] = []
        self._static_index: dict[str, int] = {}
        self.stores: list[tuple[int, Expr]] = []
        self._cols: dict[str, Expr] = {}

    def col(self, column: str) -> Expr:
        if column not in self._cols:
            lay = self.env.program.layout
            if lay.has(self.table, column):
                self._cols[column] = Expr(LOAD_STATE, start=lay.columns[(self.table, column)][0],
                                          seq=len(self.stores))
            else:
                if column not in self._static_index:
                    self._static_index[column] = len(self.statics) * self.n_rows
                    self.statics.append(np.asarray(self.env.net[self.table][column].to_numpy(), float))
                self._cols[column] = Expr(LOAD_STATIC, start=self._static_index[column])
        return self._cols[column]

    def store(self, column: str, value):
        lay = self.env.program.layout
        if not lay.has(self.table, column):
            if (self.table, column) in self.env.pruned_columns:
                return                     # nothing reads this column: not materialised
            raise KeyError(f"{self.table}.{column} is not a per-environment column")
        self._cols.pop(column, None)   # later reads see the stored value
        self.stores.append((lay.columns[(self.table, column)][0], Expr.wrap(value)))

    # ------------------------------------------------------------------ compile
    def compile_groups(self, live_cells):
        """Row-level pruning: a store whose cell no kernel table reads need not happen.  Rows are grouped
        by the set of their live stores; every group gets its own (shorter) program over its rows.
        Returns a list of ``(rows, ops, statics)``; ``live_cells=None`` keeps everything (one group)."""
        if live_cells is None:
            ops, statics = self.compile()
            return [(None, ops, statics)] if ops else []
        # a column that the program itself reads back later counts as live for every row
        loaded = set()

        def walk(e):
            if e.op == LOAD_STATE:
                loaded.add(e.start)
            for a in e.args:
                walk(a)
        for _, e in self.stores:
            walk(e)
        groups: dict[tuple, list] = {}
        for r in range(self.n_rows):
            sig = tuple(i for i, (start, _) in enumerate(self.stores)
                        if (start + r) in live_cells or start in loaded)
            if sig:
                groups.setdefault(sig, []).append(r)
        out = []
        for sig, rows in groups.items():
            ops, statics = self.compile(sig)
            out.append((None if len(rows) == self.n_rows else np.asarray(rows, np.int32), ops, statics))
        return out

    def compile(self, keep=None):
        """Register program of the stores ``keep`` (indices into ``self.stores``; default all of them)."""
        stores = [(i, *self.stores[i]) for i in (range(len(self.stores)) if keep is None else keep)]
        uses: dict[int, int] = {}

        def count(e):
            uses[id(e)] = uses.get(id(e), 0) + 1
            if uses[id(e)] == 1:
                for a in e.args:
                    count(a)
        for _, _, e in stores:
            count(e)
        # LOAD_STATE handles per column, with the last store that reads each of them
        loads_of: dict[int, dict[int, tuple]] = {}

        def find_loads(e, i, seen):
            if id(e) in seen:
                return
            seen.add(id(e))
            if e.op == LOAD_STATE:
                loads_of.setdefault(e.start, {})[id(e)] = (e, i)
            for a in e.args:
                find_loads(a, i, seen)
        for i, _, e in stores:
            find_loads(e, i, set())
        ops, reg_of, free = [], {}, list(range(N_REG - 1, -1, -1))

        def release(e):
            uses[id(e)] -= 1
            if uses[id(e)] == 0:
                free.append(reg_of.pop(id(e)))

        def emit(e) -> int:
            if id(e) in reg_of:
                return reg_of[id(e)]
            regs = [emit(a) for a in e.args]
            for a in e.args:
                release(a)
            if not free:
                raise RuntimeError("row program needs more than 16 registers")
            dst = free.pop()
            reg_of[id(e)] = dst
            if e.op in (LOAD_STATE, LOAD_STATIC):
                ops.append((e.op, dst, e.start, 0, 0.0))
            elif e.op == CONST:
                ops.append((CONST, dst, 0, 0, e.imm))
            else:
                ops.append((e.op, dst, regs[0], regs[1] if len(regs) > 1 else 0, 0.0))
            return dst
        for i, start, e in stores:
            # a handle taken before this store still reads the old value: load it now if a later store uses it
            for h, last in loads_of.get(start, {}).values():
                if h.seq <= i < last and id(h) not in reg_of and uses[id(h)] > 0:
                    emit(h)
            r = emit(e)
            ops.append((STORE_STATE, 0, start, r, 0.0))
            release(e)
        statics = np.concatenate(self.statics) if self.statics else np.zeros(0)
        return ops, statics

    def __enter__(self):
        return self

    def __exit__(self, exc_type, exc, tb):
        return False


class CompiledRowProgram:
    def __init__(self, engine, n_rows, ops, statics, rows=None):
        self.engine, self.lib = engine, engine.lib
        arr = (capi.RowOp * len(ops))(*[capi.RowOp(*o) for o in ops])
        statics = np.ascontiguousarray(statics, dtype=np.float64)
        h = C.c_void_p()
        capi.check(self.lib, self.lib.opfg_row_program_create(
            n_rows, len(ops), arr, len(statics), statics.ctypes.data_as(C.POINTER(C.c_double)),
            C.byref(h)))
        self.handle, self.n_ops = h, len(ops)
        self.n_items = n_rows
        if rows is not None:
            rows = np.ascontiguousarray(rows, dtype=np.int32)
            capi.check(self.lib, self.lib.opfg_row_program_select_rows(
                h, len(rows), rows.ctypes.data_as(C.POINTER(C.c_int32))))
            self.n_items = len(rows)

    def run(self):
        e = self.engine
        if e.trace is not None:
            e.trace.append(("program", self))
        capi.check(self.lib, self.lib.opfg_row_program_run(
            self.handle, e.num_envs, e._ptr(e.state), e.program.layout.n, e._stream()))

    def __del__(self):
        try:
            self.lib.opfg_row_program_destroy(self.handle)
        except Exception:
            pass
