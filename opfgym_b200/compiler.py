"""Compile a net + RL problem definition into the flat tables of the C ABI.

The reference keeps one mutable pandas ``net`` per environment and walks it in
Python every step (``opfgym/opf_env.py:421-491, 493-549``).  Here the net is
compiled ONCE into

* a **state layout**: which ``(table, column)`` cells differ between
  environments (sampled values, set-points, per-sample bounds, prices) and which
  result columns are materialised -- all of them columns of one row-major
  matrix ``S[B, n_state]``;
* a **constant table** for every value shared by all environments;
* the **assembly / scoring programs** (``OpfgAssemblyDesc`` / ``OpfgScoringDesc``
  of ``include/opfg_b200.h``) whose operands are references into ``S`` or the
  constant table.
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field

import numpy as np

from . import capi as capi_flags
from . import ppc as P
from .constraints import Constraint
from .reward import RewardFunction

RES_PREFIX = "res_"
_I32 = np.int32


class ConstTable:
    def __init__(self):
        self.values: list[float] = []
        self._index: dict = {}

    def ref(self, value) -> int:
        value = float(value)
        key = "nan" if math.isnan(value) else value
        if key not in self._index:
            self._index[key] = len(self.values)
            self.values.append(value)
        return -self._index[key] - 1


class StateLayout:
    """Columns of S: every registered (table, column) occupies one contiguous
    slice covering ALL rows of the table, in table order."""

    def __init__(self):
        self.columns: dict[tuple[str, str], tuple[int, int]] = {}
        self.n = 0
        self.n_inputs = 0

    def add(self, table: str, column: str, n_rows: int) -> int:
        key = (table, column)
        if key not in self.columns:
            self.columns[key] = (self.n, n_rows)
            self.n += n_rows
        return self.columns[key][0]

    def has(self, table, column) -> bool:
        return (table, column) in self.columns

    def slice(self, table, column) -> slice:
        start, n = self.columns[(table, column)]
        return slice(start, start + n)


@dataclass
class EnvProgram:
    ppc: P.Ppc
    layout: StateLayout
    consts: np.ndarray
    initial_state: np.ndarray        # one row of S, static values of the dynamic columns
    assembly: dict
    scoring: dict
    n_act: int
    n_obs: int
    constraints: list
    act_low_refs: np.ndarray
    act_high_refs: np.ndarray
    sample_plan: dict = field(default_factory=dict)
    index_pos: dict = field(default_factory=dict)
    dyn_branches: dict | None = None     # OpfgDynBranchDesc arrays, if any branch cell is per-environment
    obs_segments: list | None = None     # observation entries per obs key (after bus-wise grouping)
    read_cells: frozenset = frozenset()  # state cells that some kernel table reads (or an action overwrites)


def _positions(net, table: str, idxs) -> np.ndarray:
    index = net[table].index
    pos = index.get_indexer(np.asarray(idxs))
    if (pos < 0).any():
        raise KeyError(f"unknown index in {table}: {np.asarray(idxs)[pos < 0]}")
    return pos.astype(np.int64)


def _is_res(table: str) -> bool:
    return table.startswith(RES_PREFIX)


class Compiler:
    def __init__(self, net, builder: P.PpcBuilder | None = None):
        self.net = net
        self.builder = builder or P.PpcBuilder(net)
        self.ppc = self.builder.build(net)
        self.layout = StateLayout()
        self.consts = ConstTable()
        self.referenced: set[tuple[str, str]] = set()   # columns some compiled table actually reads
        self.read_cells: set[int] = set()               # ... and the state cells (row-level pruning of hooks)

    # ---------------------------------------------------------------- references
    def declare_dynamic(self, table: str, column: str):
        if _is_res(table):
            raise ValueError("result columns are materialised automatically")
        if column not in self.net[table].columns:
            self.net[table][column] = np.nan
        self.layout.add(table, column, len(self.net[table]))

    def value_ref(self, table: str, column: str, pos: int) -> int:
        self.referenced.add((table, column))
        if self.layout.has(table, column):
            cell = self.layout.columns[(table, column)][0] + int(pos)
            self.read_cells.add(cell)
            return cell
        if _is_res(table):
            raise KeyError(f"result column {table}.{column} was not materialised")
        v = self.net[table][column].iloc[int(pos)]
        return self.consts.ref(np.nan if v is None else v)

    def _absent_branch_value(self, table, pos, ends=None) -> float:
        """pandapower's result of a branch that is out of service: its rows of ppc['branch'] are never written, so
        flows are 0 and the current 0 / |V| -- 0 between energised buses, NaN if an end bus was dropped
        (results_branch.py `_get_branch_flows` [ext-mem])."""
        net, lk = self.net, self.ppc.bus_lookup
        ends = ends or (("from_bus", "to_bus") if table == "line" else ("hv_bus", "lv_bus"))
        pos_of = {int(b): i for i, b in enumerate(net.bus.index)}
        live = all(lk[pos_of[int(net[table][c].iloc[pos])]] >= 0 for c in ends)
        return 0.0 if live else float("nan")

    def _nominally_on(self, table, pos) -> bool:
        """In service, with every switch at its ends closed, in the net as given (ties are not)."""
        net = self.net
        if not bool(net[table].in_service.iloc[pos]):
            return False
        sw = net.switch
        if len(sw):
            idx = net[table].index[pos]
            mine = (sw.et == ("l" if table == "line" else "t")) & (sw.element == idx)
            if (~sw.closed[mine].astype(bool)).any():
                return False
        return True

    def optional_ref(self, table, column, pos, default) -> int:
        if self.layout.has(table, column) or column in self.net[table].columns:
            return self.value_ref(table, column, pos)
        return self.consts.ref(default)

    # -------------------------------------------------------------------- compile
    def compile(self, act_keys, obs_keys, state_keys, constraints: list[Constraint],
                reward_function: RewardFunction, extra_dynamic=(),
                autoscale_actions: bool = True, pwl_price_columns=None,
                extra_results=(), prune_unused: bool = False,
                diff_action_step_size: float | None = None, bus_wise_obs: bool = False) -> EnvProgram:
        if prune_unused and extra_dynamic:
            # dry run: find out which hook-written columns any kernel table actually reads
            # (e.g. max_p_mw / min_p_mw exist in the reference only for the pandapower OPF)
            probe = Compiler(self.net, self.builder)
            probe.compile(act_keys, obs_keys, state_keys, constraints, reward_function, extra_dynamic,
                          autoscale_actions, pwl_price_columns, extra_results, prune_unused=False,
                          diff_action_step_size=diff_action_step_size, bus_wise_obs=bus_wise_obs)
            extra_dynamic = [tc for tc in extra_dynamic if tuple(tc) in probe.referenced]
        net, lay, ppc = self.net, self.layout, self.ppc
        for table, column, _ in list(state_keys) + list(act_keys):
            if not _is_res(table):
                self.declare_dynamic(table, column)
        for table, column in extra_dynamic:
            self.declare_dynamic(table, column)
        lay.n_inputs = lay.n

        # ---- result cells ---------------------------------------------------
        wanted = set()
        for table, column, _ in list(obs_keys) + list(state_keys):
            if _is_res(table):
                wanted.add((table, column))
        for c in constraints:
            wanted.add((RES_PREFIX + c.unit_type, c.values_column))
        for table, column in extra_results:
            wanted.add((table, column))
        cost_sources = []
        for cost_table in ("poly_cost", "pwl_cost"):
            for et in net[cost_table].et if len(net[cost_table]) else []:
                cost_sources.append(et)
        if any(et == "ext_grid" for et in cost_sources):
            wanted |= {("res_ext_grid", "p_mw"), ("res_ext_grid", "q_mvar")}
        if any(et == "gen" for et in cost_sources):
            wanted |= {("res_gen", "q_mvar")}

        nbr = ppc.branch.shape[0]
        ng = ppc.gen.shape[0]
        res_vm = res_va = -1
        loading_slot = -np.ones(nbr, dtype=_I32)
        flow_slot = -np.ones(nbr, dtype=_I32)
        absent_cells = {}      # result cells of branches that are not in the ppc: 0 between live buses, else NaN
        gen_p_slot = -np.ones(ng, dtype=_I32)
        gen_q_slot = -np.ones(ng, dtype=_I32)
        n_t3 = len(ppc.trafo3w_branch)
        t3_loading_slot = -np.ones(n_t3, dtype=_I32)
        t3_row_slot = -np.ones(n_t3, dtype=_I32)
        for table, column in sorted(wanted):
            base = table[len(RES_PREFIX):]
            n_rows = len(net[base])
            if table == "res_bus" and column == "vm_pu":
                res_vm = lay.add(table, column, n_rows)
            elif table == "res_bus" and column == "va_degree":
                if res_vm < 0:
                    res_vm = lay.add("res_bus", "vm_pu", n_rows)
                res_va = lay.add(table, column, n_rows)
            elif table in ("res_line", "res_trafo") and column == "loading_percent":
                start = lay.add(table, column, n_rows)
                mapping = ppc.line_branch if base == "line" else ppc.trafo_branch
                for pos, br in enumerate(mapping):
                    if br >= 0:
                        loading_slot[br] = start + pos
                    else:
                        absent_cells[start + pos] = self._absent_branch_value(base, pos)
            elif table == "res_ext_grid" and column in ("p_mw", "q_mvar"):
                start = lay.add(table, column, n_rows)
                tgt = gen_p_slot if column == "p_mw" else gen_q_slot
                for pos, g in enumerate(ppc.ext_grid_gen):
                    if g >= 0:
                        tgt[g] = start + pos
            elif table == "res_gen" and column == "q_mvar":
                start = lay.add(table, column, n_rows)
                for pos, g in enumerate(ppc.gen_gen):
                    if g >= 0:
                        gen_q_slot[g] = start + pos
            elif table in ("res_line", "res_trafo") and column == "_flows4":
                # 4 cells per element: p_from/hv, q_from/hv, p_to/lv, q_to/lv  (adapter only)
                start = lay.add(table, column, 4 * n_rows)
                mapping = ppc.line_branch if base == "line" else ppc.trafo_branch
                for pos, br in enumerate(mapping):
                    if br >= 0:
                        flow_slot[br] = start + 4 * pos
                    else:
                        for k in range(4):
                            absent_cells[start + 4 * pos + k] = self._absent_branch_value(base, pos)
            elif table == "res_trafo3w" and column == "loading_percent":
                # kernel 5: the branch loop writes the outer-end loading of each of the three star branches into
                # three hidden cells (the star ends have factor 0), then one lane per element takes their max.  A
                # winding whose branch is absent is 0 next to a live bus and NaN next to a dropped one
                # (PANDAPOWER_ASSUMPTIONS 16): a constant cell
                start = lay.add(table, column, n_rows)
                rows3 = lay.add(table, "_rows3", 3 * n_rows)
                for pos in range(n_rows):
                    t3_loading_slot[pos] = start + pos
                    t3_row_slot[pos] = rows3 + 3 * pos
                    for w, (side, br) in enumerate(zip(("hv", "mv", "lv"), ppc.trafo3w_branch[pos])):
                        if br >= 0:
                            loading_slot[br] = rows3 + 3 * pos + w
                        else:
                            absent_cells[rows3 + 3 * pos + w] = self._absent_branch_value("trafo3w", pos, (f"{side}_bus",))
            elif table == "res_trafo3w" and column == "_flows12":
                # 4 cells per winding branch, as for res_trafo _flows4 (adapter only): the outer end is the hv
                # branch's from end and the mv / lv branches' to end
                start = lay.add(table, column, 12 * n_rows)
                for pos in range(n_rows):
                    for w, (side, br) in enumerate(zip(("hv", "mv", "lv"), ppc.trafo3w_branch[pos])):
                        if br >= 0:
                            flow_slot[br] = start + 12 * pos + 4 * w
                        else:
                            for k in range(4):
                                absent_cells[start + 12 * pos + 4 * w + k] = \
                                    self._absent_branch_value("trafo3w", pos, (f"{side}_bus",))
            elif table in ("res_load", "res_sgen", "res_storage", "res_gen") and column in ("p_mw", "q_mvar"):
                pass   # = set-point * scaling, referenced with a multiplier (no cell needed)
            else:
                raise NotImplementedError(f"result column {table}.{column} is not produced by the engine")

        # ---- initial state row (even width: rows are moved as 16-byte words) --------
        lay.n += lay.n & 1
        init = np.full(lay.n, np.nan)
        for (table, column), (start, n_rows) in lay.columns.items():
            if _is_res(table):
                continue
            col = net[table][column]
            init[start:start + n_rows] = np.asarray(
                [np.nan if v is None else float(v) for v in col.to_numpy()], dtype=float)
        for cell, value in absent_cells.items():
            init[cell] = value

        # ---- actions (opf_env.py:421-491) -----------------------------------
        a_slot, a_lo, a_hi, a_div, a_kind, a_clo, a_chi = [], [], [], [], [], [], []
        for table, column, idxs in act_keys:
            pos = _positions(net, table, idxs)
            lo_c, hi_c = (f"min_{column}", f"max_{column}") if autoscale_actions else \
                         (f"min_min_{column}", f"max_max_{column}")
            for p in pos:
                a_slot.append(self.value_ref(table, column, p))
                a_lo.append(self.value_ref(table, lo_c, p))
                a_hi.append(self.value_ref(table, hi_c, p))
                a_div.append(self.optional_ref(table, "scaling", p, 1.0))
                a_kind.append(1 if column in ("closed", "in_service") else
                              2 if column in ("tap_pos", "step") else 0)
                if not autoscale_actions:
                    a_clo.append(self.optional_ref(table, f"min_{column}", p, -np.inf))
                    a_chi.append(self.optional_ref(table, f"max_{column}", p, np.inf))
        n_act = len(a_slot)

        # ---- injections (pandapower build_bus PD/QD + makeSbus [ext-mem]) ----
        inj_bus, inj_p, inj_q, inj_c = [], [], [], []
        zero = self.consts.ref(0.0)
        for table, sign in (("load", -1.0), ("sgen", 1.0), ("storage", -1.0)):
            df = net[table]
            if not len(df):
                continue
            buses = self.builder.element_bus(net, table)
            for pos in range(len(df)):
                if buses[pos] < 0:
                    continue
                if self.layout.has(table, "in_service") or self.layout.has(table, "scaling"):
                    raise NotImplementedError("per-environment scaling/in_service of injections")
                coef = sign * float(df.scaling.iloc[pos]) * float(bool(df.in_service.iloc[pos]))
                inj_bus.append(buses[pos])
                inj_p.append(self.value_ref(table, "p_mw", pos))
                inj_q.append(self.value_ref(table, "q_mvar", pos))
                inj_c.append(self.consts.ref(coef))
        if len(net.ward):
            # constant-power part of a ward: a load without a scaling column (its pz / qz sit in the bus shunt)
            buses = self.builder.element_bus(net, "ward")
            if self.layout.has("ward", "in_service") or self.layout.has("ward", "pz_mw") \
                    or self.layout.has("ward", "qz_mvar"):
                raise NotImplementedError("per-environment ward.in_service / pz_mw / qz_mvar")
            for pos in range(len(net.ward)):
                if buses[pos] < 0:
                    continue
                inj_bus.append(buses[pos])
                inj_p.append(self.value_ref("ward", "ps_mw", pos))
                inj_q.append(self.value_ref("ward", "qs_mvar", pos))
                inj_c.append(self.consts.ref(-float(bool(net.ward.in_service.iloc[pos]))))
        for pos, g in enumerate(ppc.gen_gen):
            if g < 0:
                continue
            inj_bus.append(int(ppc.gen[g, P.GEN_BUS]))
            inj_p.append(self.value_ref("gen", "p_mw", pos))
            inj_q.append(zero)
            inj_c.append(self.consts.ref(float(net.gen.scaling.iloc[pos])))
        # static ppc bus demand not represented by an element table (none today) is ignored

        # ---- per-environment voltage set-points: gen.vm_pu / ext_grid.vm_pu as state cells ----
        # (pandapower `_get_pf_variables_from_ppci`: V0[gen bus] = VG for generators on PV / slack buses)
        bus_vm_ref = None
        NO_REF = -2**31
        for table, lookup in (("ext_grid", ppc.ext_grid_gen), ("gen", ppc.gen_gen)):
            if not lay.has(table, "vm_pu"):
                continue
            if bus_vm_ref is None:
                bus_vm_ref = np.full(ppc.bus.shape[0], NO_REF, dtype=np.int64)
            for pos, g in enumerate(lookup):
                if g >= 0 and ppc.bus[int(ppc.gen[g, P.GEN_BUS]), P.BUS_TYPE] != P.PQ:
                    bus_vm_ref[int(ppc.gen[g, P.GEN_BUS])] = self.value_ref(table, "vm_pu", pos)

        assembly = dict(
            n_state=lay.n, act_slot=np.asarray(a_slot, _I32), act_lo=np.asarray(a_lo, _I32),
            act_hi=np.asarray(a_hi, _I32), act_div=np.asarray(a_div, _I32),
            act_kind=np.asarray(a_kind, _I32),
            act_clamp_lo=np.asarray(a_clo, _I32) if a_clo else None,
            act_clamp_hi=np.asarray(a_chi, _I32) if a_chi else None,
            act_diff_step=float(diff_action_step_size or 0.0),
            inj_bus=np.asarray(inj_bus, _I32), inj_p=np.asarray(inj_p, _I32),
            inj_q=np.asarray(inj_q, _I32), inj_coef=np.asarray(inj_c, _I32),
            bus_vm_ref=None if bus_vm_ref is None else bus_vm_ref.astype(_I32))

        # ---- constraints (constraints.py:70-128) ------------------------------
        con_ptr = [0]
        c_val, c_vs, c_min, c_max, c_mul = [], [], [], [], []
        c_auto, c_worst, c_pf, c_pp, c_pc = [], [], [], [], []
        nan_ref = self.consts.ref(np.nan)
        for c in constraints:
            table = net[c.unit_type]
            res_table = RES_PREFIX + c.unit_type
            mult = c.boundary_multiplier(net)
            mult = np.broadcast_to(np.asarray(mult, float), (len(table),))
            has_min = f"min_{c.values_column}" in table.columns
            has_max = f"max_{c.values_column}" in table.columns
            for pos in range(len(table)):
                vref, vmul = self._result_ref(res_table, c.values_column, pos)
                c_val.append(vref)
                c_vs.append(vmul * c.value_scale)
                c_min.append(self.value_ref(c.unit_type, f"min_{c.values_column}", pos) if has_min else nan_ref)
                c_max.append(self.value_ref(c.unit_type, f"max_{c.values_column}", pos) if has_max else nan_ref)
                c_mul.append(float(mult[pos]))
            con_ptr.append(len(c_val))
            c_auto.append(c.autoscale_factor(net))
            c_worst.append(int(c.only_worst_case_violations))
            c_pf.append(c.penalty_factor)
            c_pp.append(c.penalty_power)
            c_pc.append(c.violation_count_penalty)

        # ---- costs (objective.py) -------------------------------------------
        pc = net.poly_cost
        poly_p, poly_pm, poly_q, poly_qm, poly_cf = [], [], [], [], []
        coef_cols = ("cp0_eur", "cp1_eur_per_mw", "cp2_eur_per_mw2",
                     "cq0_eur", "cq1_eur_per_mvar", "cq2_eur_per_mvar2")
        for pos in range(len(pc)):
            et, el = pc.et.iloc[pos], int(pc.element.iloc[pos])
            epos = int(_positions(net, et, [el])[0])
            r, m = self._result_ref(RES_PREFIX + et, "p_mw", epos)
            poly_p.append(r); poly_pm.append(m)
            r, m = self._result_ref(RES_PREFIX + et, "q_mvar", epos)
            poly_q.append(r); poly_qm.append(m)
            poly_cf.extend(self.value_ref("poly_cost", col, pos) for col in coef_cols)
        pw = net.pwl_cost
        pwl_v, pwl_vm, pwl_seg = [], [], []
        n_seg = min((len(pts) for pts in pw.points), default=0) if len(pw) else 0
        for pos in range(len(pw)):
            et, el = pw.et.iloc[pos], int(pw.element.iloc[pos])
            epos = int(_positions(net, et, [el])[0])
            col = "p_mw" if pw.power_type.iloc[pos] == "p" else "q_mvar"
            r, m = self._result_ref(RES_PREFIX + et, col, epos)
            pwl_v.append(r); pwl_vm.append(m)
            pts = pw.points.iloc[pos]
            for s in range(n_seg):
                lo, hi, price = pts[s]
                pwl_seg.append(self.consts.ref(lo))
                pwl_seg.append(self.consts.ref(hi))
                if pwl_price_columns and s < len(pwl_price_columns) and pwl_price_columns[s]:
                    pwl_seg.append(self.value_ref("pwl_cost", pwl_price_columns[s], pos))
                else:
                    pwl_seg.append(self.consts.ref(price))

        # ---- observation gather (opf_env.py:532-549) --------------------------
        obs_ref, obs_ptr, obs_segments = [], [0], []
        for table, column, idxs in obs_keys:
            base = table[len(RES_PREFIX):] if _is_res(table) else table
            if bus_wise_obs and table == "load":
                # loads at the same bus are observed as one sum, groups sorted by bus
                # (get_bus_aggregated_obs, opf_env.py:806-810 -- note its .iloc[idxs])
                buses = net.load.bus.to_numpy()[np.asarray(idxs, int)]
                for bus in sorted(set(buses.tolist())):
                    for p in np.asarray(idxs, int)[buses == bus]:
                        obs_ref.append(self.value_ref(table, column, int(p)))
                    obs_ptr.append(len(obs_ref))
                obs_segments.append(len(set(buses.tolist())))
                continue
            obs_segments.append(len(idxs))
            for p in _positions(net, base, idxs):
                obs_ptr.append(len(obs_ref) + 1)
                if _is_res(table):
                    r, m = self._result_ref(table, column, p)
                    if m != 1.0:
                        raise NotImplementedError(f"observation of scaled column {table}.{column}")
                    obs_ref.append(r)
                else:
                    obs_ref.append(self.value_ref(table, column, p))

        # ---- per-environment branch parameters (tap_pos / in_service cells) ------------
        dyn = None
        dyn_rows = []
        one, nan = self.consts.ref(1.0), self.consts.ref(np.nan)
        # `switch.closed` cells of line-bus / trafo-bus switches (examples/network_reconfiguration.py:34,
        # security_constrained.py:31): one reference per branch end; bus-bus switches would change the bus count
        sw_ends = {}
        if lay.has("switch", "closed"):
            sw = net.switch
            bus_pos = {int(b): i for i, b in enumerate(net.bus.index)}
            for spos, (et, el, bus) in enumerate(zip(sw.et.to_numpy(object), sw.element.to_numpy(), sw.bus.to_numpy())):
                if et == "b":
                    continue           # static (fused by the builder); as an ACTION it is rejected in opf_env
                table = "line" if et == "l" else "trafo"
                epos = int(np.nonzero(net[table].index.to_numpy() == int(el))[0][0])
                first = net[table]["from_bus" if et == "l" else "hv_bus"].iloc[epos]
                end = 0 if int(bus) == int(first) else 1
                if (table, epos, end) in sw_ends:
                    raise NotImplementedError(f"two switches at one end of {table} {el}")
                sw_ends[table, epos, end] = self.value_ref("switch", "closed", spos)
        for pos, br in enumerate(ppc.line_branch):
            has_sw = ("line", pos, 0) in sw_ends or ("line", pos, 1) in sw_ends
            if br >= 0 and (lay.has("line", "in_service") or has_sw):
                svc = self.value_ref("line", "in_service", pos) if lay.has("line", "in_service") else one
                dyn_rows.append((int(br), nan, 0.0, 0.0, 1.0, svc, sw_ends.get(("line", pos, 0), one),
                                 sw_ends.get(("line", pos, 1), one),
                                 0 if self._nominally_on("line", pos) else capi_flags.DYN_NORMALLY_OPEN))
        tr = net.trafo
        for pos, br in enumerate(ppc.trafo_branch):
            has_sw = ("trafo", pos, 0) in sw_ends or ("trafo", pos, 1) in sw_ends
            if br < 0 or not (lay.has("trafo", "tap_pos") or lay.has("trafo", "in_service") or has_sw):
                continue
            k = int(np.nonzero(self.builder.trafo_pos == pos)[0][0])
            tap, flags = nan, capi_flags.DYN_TRAFO
            if not self._nominally_on("trafo", pos):
                flags |= capi_flags.DYN_NORMALLY_OPEN
            if lay.has("trafo", "tap_pos"):
                tap = self.value_ref("trafo", "tap_pos", pos)
                if self.builder.trafo_tap_on_lv[k]:
                    flags |= capi_flags.DYN_TAP_LV
                elif not self.builder.trafo_tap_on_hv[k]:
                    tap = nan          # no tap changer: the cell has no effect (pandapower ignores tap_pos then)
            svc = self.value_ref("trafo", "in_service", pos) if lay.has("trafo", "in_service") else one
            dyn_rows.append((int(br), tap, float(tr.tap_neutral.iloc[pos]),
                             float(tr.tap_step_percent.iloc[pos]),
                             float(self.builder.trafo_ratio_neutral[k]), svc,
                             sw_ends.get(("trafo", pos, 0), one), sw_ends.get(("trafo", pos, 1), one), flags))
        if lay.has("trafo3w", "in_service"):
            raise NotImplementedError("trafo3w.in_service as a per-environment cell is not modelled")
        if lay.has("trafo3w", "tap_pos"):
            # the tapped winding's equivalent branch is a 2-winding transformer: kernel 1's trafo tap math
            # applies, on its HV or LV end (PANDAPOWER_ASSUMPTIONS 14)
            t3 = net.trafo3w
            if not hasattr(self.builder, "trafo3w_tap_w"):
                raise NotImplementedError("per-environment trafo3w.tap_pos needs the in-repo net conversion (PpcBuilder)")
            for pos, rows in enumerate(ppc.trafo3w_branch):
                w = int(self.builder.trafo3w_tap_w[pos])
                if w < 0 or rows[w] < 0:
                    continue           # no tap changer (pandapower ignores tap_pos then), or the branch is absent
                br = int(rows[w])
                k = br - self.builder.trafo3w_first          # position in the builder's trafo3w rows
                flags = capi_flags.DYN_TRAFO | (capi_flags.DYN_TAP_LV if self.builder.trafo3w_tap_at_lv[pos] else 0)
                dyn_rows.append((br, self.value_ref("trafo3w", "tap_pos", pos), float(t3.tap_neutral.iloc[pos]),
                                 float(t3.tap_step_percent.iloc[pos]), float(self.builder.trafo3w_ratio_neutral[k]),
                                 one, one, one, flags))
        if dyn_rows:
            cols = list(zip(*dyn_rows))
            dyn = dict(branch=np.asarray(cols[0], _I32), tap_pos=np.asarray(cols[1], _I32),
                       tap_neutral=np.asarray(cols[2], float), tap_step_percent=np.asarray(cols[3], float),
                       ratio_neutral=np.asarray(cols[4], float), in_service=np.asarray(cols[5], _I32),
                       closed_from=np.asarray(cols[6], _I32), closed_to=np.asarray(cols[7], _I32),
                       flags=np.asarray(cols[8], _I32))

        rp = reward_function.device_params()
        scoring = dict(
            n_inputs=lay.n_inputs, n_pp_bus=len(net.bus), pp_bus_lookup=ppc.bus_lookup.astype(_I32),
            res_bus_vm_slot=res_vm, res_bus_va_slot=res_va,
            branch_loading_slot=loading_slot, branch_flow_slot=flow_slot,
            rate_f=ppc.rate_f.astype(float), rate_t=ppc.rate_t.astype(float),
            gen_p_slot=gen_p_slot, gen_q_slot=gen_q_slot,
            n_constraints=len(constraints), con_ptr=np.asarray(con_ptr, _I32),
            con_value=np.asarray(c_val, _I32), con_value_scale=np.asarray(c_vs, float),
            con_min=np.asarray(c_min, _I32), con_max=np.asarray(c_max, _I32),
            con_bound_mul=np.asarray(c_mul, float), con_autoscale=np.asarray(c_auto, float),
            con_worst_case=np.asarray(c_worst, _I32), con_penalty_factor=np.asarray(c_pf, float),
            con_penalty_power=np.asarray(c_pp, float), con_count_penalty=np.asarray(c_pc, float),
            n_poly=len(pc), poly_p=np.asarray(poly_p, _I32), poly_p_mul=np.asarray(poly_pm, float),
            poly_q=np.asarray(poly_q, _I32), poly_q_mul=np.asarray(poly_qm, float),
            poly_coef=np.asarray(poly_cf, _I32),
            n_pwl=len(pw), n_pwl_seg=n_seg, pwl_v=np.asarray(pwl_v, _I32),
            pwl_v_mul=np.asarray(pwl_vm, float), pwl_seg=np.asarray(pwl_seg, _I32),
            reward=rp, n_obs=len(obs_ptr) - 1, obs_ref=np.asarray(obs_ref, _I32),
            obs_ptr=np.asarray(obs_ptr, _I32) if len(obs_ref) != len(obs_ptr) - 1 else None,
            n_trafo3w=n_t3 if (t3_loading_slot >= 0).any() else 0,
            trafo3w_row_slot=t3_row_slot, trafo3w_loading_slot=t3_loading_slot)

        return EnvProgram(ppc=ppc, layout=lay, consts=np.asarray(self.consts.values, float),
                          initial_state=init, assembly=assembly, scoring=scoring,
                          n_act=n_act, n_obs=len(obs_ptr) - 1, constraints=list(constraints),
                          obs_segments=obs_segments,
                          act_low_refs=np.asarray(a_lo, _I32), act_high_refs=np.asarray(a_hi, _I32),
                          dyn_branches=dyn, read_cells=frozenset(self.read_cells) | frozenset(int(x) for x in a_slot))

    def _result_ref(self, res_table: str, column: str, pos: int) -> tuple[int, float]:
        """Reference (and multiplier) that yields ``net[res_table][column]`` of row ``pos``."""
        base = res_table[len(RES_PREFIX):]
        if self.layout.has(res_table, column):
            return self.layout.columns[(res_table, column)][0] + int(pos), 1.0
        if base in ("load", "sgen", "storage") or (base == "gen" and column == "p_mw"):
            # res_<unit>.p_mw = p_mw * scaling * in_service  (pandapower results_gen/_bus [ext-mem])
            df = self.net[base]
            mul = float(df.scaling.iloc[pos])
            if "in_service" in df.columns:
                mul *= float(bool(df.in_service.iloc[pos]))
            return self.value_ref(base, column, pos), mul
        raise KeyError(f"result column {res_table}.{column} was not materialised")


# ----------------------------------------------------------- ctypes marshalling
def fill_descs(capi, program: EnvProgram, tol_pu, max_iter, init_dc, enforce_q_lims,
               threads_per_env=0, ordering=0, pf_kernel=0):
    """Build the three ctypes descriptor structs.  Returns (grid, assembly,
    scoring, keepalive) -- ``keepalive`` holds the numpy arrays the structs point to."""
    import ctypes as C
    keep = []

    def dptr(a):
        a = np.ascontiguousarray(a, dtype=np.float64)
        keep.append(a)
        return a.ctypes.data_as(C.POINTER(C.c_double))

    def iptr(a):
        if a is None:
            return None
        a = np.ascontiguousarray(a, dtype=np.int32)
        keep.append(a)
        return a.ctypes.data_as(C.POINTER(C.c_int32))

    ppc = program.ppc
    gd = capi.GridDesc(nb=ppc.bus.shape[0], ng=ppc.gen.shape[0], nbr=ppc.branch.shape[0],
                       base_mva=ppc.base_mva, bus=dptr(ppc.bus), bus_cols=ppc.bus.shape[1],
                       gen=dptr(ppc.gen), gen_cols=ppc.gen.shape[1], branch=dptr(ppc.branch),
                       branch_cols=ppc.branch.shape[1], tol_pu=tol_pu, max_iter=max_iter,
                       init_dc=int(init_dc), enforce_q_lims=int(enforce_q_lims),
                       threads_per_env=threads_per_env, ordering=ordering,
                       pf_kernel=pf_kernel)
    a = program.assembly
    ad = capi.AssemblyDesc(n_state=a["n_state"], n_const=len(program.consts),
                           consts=dptr(program.consts), n_act=len(a["act_slot"]),
                           act_slot=iptr(a["act_slot"]), act_lo=iptr(a["act_lo"]),
                           act_hi=iptr(a["act_hi"]), act_div=iptr(a["act_div"]),
                           act_kind=iptr(a["act_kind"]), act_clamp_lo=iptr(a["act_clamp_lo"]),
                           act_clamp_hi=iptr(a["act_clamp_hi"]), act_diff_step=a["act_diff_step"],
                           n_inj=len(a["inj_bus"]),
                           inj_bus=iptr(a["inj_bus"]), inj_p=iptr(a["inj_p"]),
                           inj_q=iptr(a["inj_q"]), inj_coef=iptr(a["inj_coef"]),
                           bus_vm_ref=iptr(a.get("bus_vm_ref")))
    s = program.scoring
    r = s["reward"]
    sd = capi.ScoringDesc(
        n_inputs=s["n_inputs"], n_pp_bus=s["n_pp_bus"], pp_bus_lookup=iptr(s["pp_bus_lookup"]),
        res_bus_vm_slot=s["res_bus_vm_slot"], res_bus_va_slot=s["res_bus_va_slot"],
        branch_loading_slot=iptr(s["branch_loading_slot"]), branch_flow_slot=iptr(s["branch_flow_slot"]),
        rate_f=dptr(s["rate_f"]), rate_t=dptr(s["rate_t"]),
        gen_p_slot=iptr(s["gen_p_slot"]), gen_q_slot=iptr(s["gen_q_slot"]),
        n_constraints=s["n_constraints"], con_ptr=iptr(s["con_ptr"]), con_value=iptr(s["con_value"]),
        con_value_scale=dptr(s["con_value_scale"]), con_min=iptr(s["con_min"]), con_max=iptr(s["con_max"]),
        con_bound_mul=dptr(s["con_bound_mul"]), con_autoscale=dptr(s["con_autoscale"]),
        con_worst_case=iptr(s["con_worst_case"]), con_penalty_factor=dptr(s["con_penalty_factor"]),
        con_penalty_power=dptr(s["con_penalty_power"]), con_count_penalty=dptr(s["con_count_penalty"]),
        n_poly=s["n_poly"], poly_p=iptr(s["poly_p"]), poly_p_mul=dptr(s["poly_p_mul"]),
        poly_q=iptr(s["poly_q"]), poly_q_mul=dptr(s["poly_q_mul"]), poly_coef=iptr(s["poly_coef"]),
        n_pwl=s["n_pwl"], n_pwl_seg=s["n_pwl_seg"], pwl_v=iptr(s["pwl_v"]),
        pwl_v_mul=dptr(s["pwl_v_mul"]), pwl_seg=iptr(s["pwl_seg"]),
        reward_kind=r["kind"], penalty_weight=r["penalty_weight"], clip_lo=r["clip_lo"],
        clip_hi=r["clip_hi"], objective_factor=r["objective_factor"],
        objective_bias=r["objective_bias"], penalty_factor=r["penalty_factor"],
        penalty_bias=r["penalty_bias"], valid_reward=r["valid_reward"],
        invalid_penalty=r["invalid_penalty"], invalid_objective_share=r["invalid_objective_share"],
        n_obs=s["n_obs"], obs_ref=iptr(s["obs_ref"]), obs_ptr=iptr(s["obs_ptr"]),
        n_trafo3w=s["n_trafo3w"])
    if s["n_trafo3w"]:
        sd.trafo3w_row_slot, sd.trafo3w_loading_slot = iptr(s["trafo3w_row_slot"]), iptr(s["trafo3w_loading_slot"])
    dd = None
    if program.dyn_branches is not None:
        d = program.dyn_branches
        dd = capi.DynBranchDesc(n_dyn=len(d["branch"]), branch=iptr(d["branch"]), tap_pos=iptr(d["tap_pos"]),
                                tap_neutral=dptr(d["tap_neutral"]), tap_step_percent=dptr(d["tap_step_percent"]),
                                ratio_neutral=dptr(d["ratio_neutral"]), in_service=iptr(d["in_service"]),
                                closed_from=iptr(d["closed_from"]), closed_to=iptr(d["closed_to"]),
                                flags=iptr(d["flags"]))
    return gd, ad, sd, dd, keep
