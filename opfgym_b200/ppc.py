"""Net tables -> PYPOWER-style ``ppc`` matrices (the input side of the hot path).

This restates, from memory of pandapower 2.x, the conversion that
``pp.runpp`` performs before its Newton-Raphson (``pd2ppc.py``,
``build_bus.py``, ``build_branch.py``, ``build_gen.py``) -- SURVEY.md App.
B.2/B.3, rows a4(i) of §8.  pandapower itself is absent from the build
image, so everything here is marked [ext-mem]; see
``PANDAPOWER_ASSUMPTIONS`` for the full list of behaviours assumed.

The product path (``opfgym_b200.engine``) hands the matrices produced here to
the C-ABI library (``opfg_grid_create``); the CPU oracle consumes the same
matrices.  Matrix column order is PYPOWER's (``idx_bus/idx_gen/idx_brch``)
plus one extension column ``BR_G`` for line conductance.
"""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

PANDAPOWER_ASSUMPTIONS = """
[ext-mem] behaviours of pandapower 2.x `runpp` assumed by this module and by
oracle/pf.py (none could be checked here: pandapower is not installed):
 1. loads (+), sgens (-), storages (+) are summed into bus PD/QD as
    value*scaling*in_service; const_z/const_i percent are 0.
 2. closed bus-bus switches fuse buses; a line with one open line-switch keeps
    its other end connected and gets an auxiliary bus at the open end; with
    both ends open (or in_service=False) it is dropped.
 3. buses not connected to an in-service ext_grid are dropped (results NaN).
 4. line pu parameters on baseR = vn_kv(from bus)^2/sn_mva; trafo on the LV
    bus voltage, T-model converted to pi by a wye-delta transform, tap on
    `tap_side`, ratio relative to the bus nominal voltages, `shift_degree`
    applied because calculate_voltage_angles is True for grids with a
    110-kV level.
 5. init='auto' -> DC-power-flow angles, |V| start = mean of ext_grid/gen
    vm_pu set-points, gen/ext-grid buses at their set-point.
 6. max_iteration='auto' -> 10, tolerance_mva=1e-8 compared against the
    per-unit mismatch (identical for sn_mva=1, the SimBench value).
 7. enforce_q_lims skips generators with QMIN == 0 or QMAX == 0 (pandapower's
    `non_refs = (QMAX != 0) & (QMIN != 0)`).  The in-service generators of one PV
    bus must share one (QMIN, QMAX) pair; other pairs are rejected by the engine.
 8. trafo_loading='current'.
 9. trafo3w (build_branch._trafo_df_from_trafo3w): one auxiliary star-point bus and three 2-winding
    equivalent branches hv->star, star->mv, star->lv, stacked behind the trafos in three blocks (all hv
    rows, all mv rows, all lv rows) and before the impedances.
10. trafo3w vk_hv/mv/lv_percent and vkr_* are the pairwise hv-mv, mv-lv and hv-lv values; each pair is
    referred to sn_hv_mva through min(sn) of its two windings (z_br_to_bus_vector), then converted
    delta->star separately for the real part and the reactance: z_i = 0.5*sn_i/sn_hv*(z_ij+z_ik-z_jk)
    (wye_delta_vector); vk_i = sign(x_i)*sqrt(x_i^2+r_i^2), so a star impedance may be negative.
11. equivalent branch i has sn = sn_<i>_mva, vn_hv_kv = vn_hv_kv, vn_lv_kv = vn_<i>_kv, parallel = df = 1,
    and is then converted like a trafo (item 4).
12. trafo3w_losses='hv': pfe_kw and i0_percent sit on the hv branch only.
13. shift_mv_degree on the mv branch, shift_lv_degree on the lv branch, none on the hv branch.
14. the trafo3w tap changer sits on the branch of the winding named by tap_side, at its outer end
    (hv branch: hv side; mv / lv branch: lv side); with tap_at_star_point at the star end of that
    branch instead.  tap_step_degree != 0 (phase shifter) is not modelled.
15. the star bus has the hv bus's nominal voltage as base kV.
16. res_trafo3w.loading_percent (trafo_loading='current', _get_trafo3w_results) = max(ld_hv, ld_mv, ld_lv),
    ld_i = current at the outer bus of branch i * vn_<i>_kv / sn_<i>_mva * sqrt3 * 100 (star ends are not
    counted), numpy's NaN-propagating max; an absent branch contributes 0 next to a live bus, NaN next to a
    dropped one.
"""

# PYPOWER column indices
BUS_I, BUS_TYPE, PD, QD, GS, BS, BUS_AREA, VM, VA, BASE_KV, ZONE, VMAX, VMIN = range(13)
GEN_BUS, PG, QG, QMAX, QMIN, VG, MBASE, GEN_STATUS, PMAX, PMIN = range(10)
(F_BUS, T_BUS, BR_R, BR_X, BR_B, RATE_A, RATE_B, RATE_C, TAP, SHIFT,
 BR_STATUS, ANGMIN, ANGMAX, BR_G) = range(14)
BUS_COLS, GEN_COLS, BRANCH_COLS = 13, 10, 14
PQ, PV, REF, NONE = 1, 2, 3, 4


@dataclass
class Ppc:
    base_mva: float
    bus: np.ndarray           # [nb, 13]
    gen: np.ndarray           # [ng, 10]  ext_grids first, then gens
    branch: np.ndarray        # [nbr, 14] lines first, then trafos
    bus_lookup: np.ndarray    # pandapower bus position -> ppc bus (-1: dropped)
    line_branch: np.ndarray   # net.line position -> branch row (-1: out)
    trafo_branch: np.ndarray  # net.trafo position -> branch row (-1: out)
    ext_grid_gen: np.ndarray  # net.ext_grid position -> gen row (-1: out)
    gen_gen: np.ndarray       # net.gen position -> gen row (-1: out)
    rate_f: np.ndarray        # loading% = 100*max(|Sf|*rate_f/vm_f, |St|*rate_t/vm_t), S in MVA
    rate_t: np.ndarray
    init_vm_pu: float = 1.0
    meta: dict = field(default_factory=dict)
    impedance_branch: np.ndarray = field(default_factory=lambda: np.zeros(0, np.int64))  # net.impedance position -> branch row
    # net.trafo3w position -> branch rows of its hv->star, star->mv, star->lv equivalents (-1: out).  Their loading
    # factors sit at the outer end (rate_f of the hv row, rate_t of the mv / lv rows); the star ends have 0.
    trafo3w_branch: np.ndarray = field(default_factory=lambda: np.zeros((0, 3), np.int64))

    @property
    def nb(self):
        return self.bus.shape[0]


class _DSU:
    def __init__(self, n):
        self.p = np.arange(n)

    def find(self, a):
        p = self.p
        while p[a] != a:
            p[a] = p[p[a]]
            a = p[a]
        return a

    def union(self, a, b):
        ra, rb = self.find(a), self.find(b)
        if ra != rb:
            if ra < rb:
                self.p[rb] = ra
            else:
                self.p[ra] = rb


UNSUPPORTED_TABLES = ("xward", "dcline", "motor", "asymmetric_load",
                      "asymmetric_sgen", "svc", "tcsc", "ssc", "vsc")


TRAFO3W_COLUMNS = ("hv_bus", "mv_bus", "lv_bus", "sn_hv_mva", "sn_mv_mva", "sn_lv_mva", "vn_hv_kv", "vn_mv_kv",
                   "vn_lv_kv", "vk_hv_percent", "vk_mv_percent", "vk_lv_percent", "vkr_hv_percent", "vkr_mv_percent",
                   "vkr_lv_percent", "pfe_kw", "i0_percent", "shift_mv_degree", "shift_lv_degree", "tap_side",
                   "tap_neutral", "tap_step_percent", "tap_pos", "in_service")


def trafo_branch_values(vn_hv, vn_lv, vn_hv_bus, vn_lv_bus, sn_t, vk, vkr, pfe_kw, i0, steps, on_hv, on_lv, par,
                        sn, trafo_model):
    """2-winding transformer -> pi branch (pandapower build_branch ``_calc_branch_values_from_trafo_df``
    [ext-mem]), on arrays.  Returns r, x, g, b, ratio and the ratio at the neutral tap."""
    vnh = np.where(on_hv, vn_hv * (1.0 + steps), vn_hv)
    vnl = np.where(on_lv, vn_lv * (1.0 + steps), vn_lv)
    ratio = (vnh / vnl) / (vn_hv_bus / vn_lv_bus)
    ratio_neutral = (vn_hv / vn_lv) / (vn_hv_bus / vn_lv_bus)
    # short-circuit impedance, referred to the LV bus voltage
    tap_lv = (vnl / vn_lv_bus) ** 2 * sn
    z_sc = vk / 100.0 / sn_t * tap_lv
    r_sc = vkr / 100.0 / sn_t * tap_lv
    x_sc = np.sign(z_sc) * np.sqrt(z_sc ** 2 - r_sc ** 2)
    r = r_sc / par
    x = x_sc / par
    # magnetising branch
    base_r = vn_lv_bus ** 2 / sn
    vnl_sq = vn_lv ** 2
    pfe = pfe_kw * 1e-3
    g_m = pfe / vnl_sq * base_r
    b_sq = (i0 / 100.0 * sn_t) ** 2 - pfe ** 2
    b_sq[b_sq < 0] = 0.0
    b_m = np.sqrt(b_sq) * base_r / vnl_sq * np.sign(i0)
    y_sh = (g_m - 1j * b_m) / (vnl / vn_lv) ** 2 * par
    if trafo_model == "t":
        nz = y_sh != 0
        za = (r[nz] + 1j * x[nz]) / 2.0
        zc = 1.0 / y_sh[nz]
        zsum = za * za + 2.0 * za * zc
        zab = zsum / zc
        zbc = zsum / za
        r = r.copy()
        x = x.copy()
        r[nz], x[nz] = zab.real, zab.imag
        y_sh = y_sh.copy()
        y_sh[nz] = 2.0 / zbc
    return r, x, y_sh.real, y_sh.imag, ratio, ratio_neutral


def trafo3w_star_parameters(t3):
    """Star-equivalent (vk, vkr) [%] of every trafo3w, each row [hv, mv, lv] on its own sn_<side>_mva
    (pandapower ``_calculate_sc_voltages_of_equivalent_transformers`` [ext-mem])."""
    sn = np.stack([t3.sn_hv_mva.to_numpy(float), t3.sn_mv_mva.to_numpy(float), t3.sn_lv_mva.to_numpy(float)])

    def to_hv_base(z):          # pairs hv-mv, mv-lv, hv-lv, each referred to sn_hv through min(sn) of the pair
        return sn[0] * np.array([z[0] / np.minimum(sn[0], sn[1]), z[1] / np.minimum(sn[1], sn[2]),
                                 z[2] / np.minimum(sn[0], sn[2])])

    def delta_to_star(z):
        return 0.5 * sn / sn[0] * np.array([z[0] + z[2] - z[1], z[1] + z[0] - z[2], z[2] + z[1] - z[0]])

    vk = to_hv_base(np.stack([t3[f"vk_{s}_percent"].to_numpy(float) for s in ("hv", "mv", "lv")]))
    vkr = to_hv_base(np.stack([t3[f"vkr_{s}_percent"].to_numpy(float) for s in ("hv", "mv", "lv")]))
    vki = np.sqrt(vk ** 2 - vkr ** 2)
    vkr_s, vki_s = delta_to_star(vkr), delta_to_star(vki)
    return np.sign(vki_s) * np.sqrt(vki_s ** 2 + vkr_s ** 2), vkr_s, sn


class PpcBuilder:
    """Topology is analysed once; ``build(net)`` refreshes the numeric columns.

    ``build`` may be called with any net that has the same tables/indices
    (e.g. after a sampler wrote new ``p_mw`` values).
    """

    def __init__(self, net, calculate_voltage_angles: bool = True,
                 trafo_model: str = "t", dynamic_service=()):
        """``dynamic_service``: tables ('line', 'trafo') whose ``in_service`` flag is a
        per-environment cell: their elements stay in the topology (status is applied per
        environment by kernel 1), so that e.g. normally-open ties can be switched on.
        'switch': ``switch.closed`` of line-bus / trafo-bus switches is a per-environment cell;
        such switches count as closed here (no auxiliary buses), kernel 1 applies them."""
        self.calculate_voltage_angles = calculate_voltage_angles
        self.trafo_model = trafo_model
        self.dynamic_service = tuple(dynamic_service)
        # element tables of pandapower that this builder does not model: fail loudly instead of
        # solving a different network (SURVEY.md 8f: adapter coverage)
        for table in UNSUPPORTED_TABLES:
            df = getattr(net, table, None) if not isinstance(net, dict) else net.get(table)
            if df is not None and len(df):
                raise NotImplementedError(
                    f"net.{table} has {len(df)} rows: {table} elements are not modelled by PpcBuilder "
                    "(supported: bus, line, trafo, trafo3w, impedance, switch, load, sgen, storage, ward, gen, ext_grid, shunt)")
        t3 = getattr(net, "trafo3w", None) if not isinstance(net, dict) else net.get("trafo3w")
        if t3 is not None and len(t3):
            missing = [c for c in TRAFO3W_COLUMNS if c not in t3.columns]
            if missing:
                raise NotImplementedError(f"net.trafo3w lacks the parameter columns {missing} of the star-point model")
            step_deg = np.nan_to_num(t3.tap_step_degree.to_numpy(float))
            if (step_deg != 0).any():
                raise NotImplementedError("net.trafo3w with tap_step_degree != 0: phase-shifting tap changers of "
                                          "three-winding transformers are not modelled")
            if len(net.switch) and (net.switch.et == "t3").any():
                raise NotImplementedError("switches at net.trafo3w (et='t3') are not modelled")
        self._analyse(net)

    # ------------------------------------------------------------------ topology
    def _analyse(self, net):
        bus_index = net.bus.index.to_numpy()
        n_pp = len(bus_index)
        pos_of = {int(b): i for i, b in enumerate(bus_index)}
        self._pos_of = pos_of
        bus_in = net.bus.in_service.to_numpy(bool)

        # bus-bus switch fusion
        dsu = _DSU(n_pp)
        sw = net.switch
        if len(sw):
            bb = sw[(sw.et == "b") & sw.closed.astype(bool)]
            for a, b in zip(bb.bus.to_numpy(), bb.element.to_numpy()):
                ia, ib = pos_of[int(a)], pos_of[int(b)]
                if bus_in[ia] and bus_in[ib]:
                    dsu.union(ia, ib)
        root = np.array([dsu.find(i) for i in range(n_pp)])

        # line terminals, with open line switches
        line_index = net.line.index.to_numpy()
        nl = len(line_index)
        lf = np.array([pos_of[int(b)] for b in net.line.from_bus.to_numpy()], dtype=np.int64)
        lt = np.array([pos_of[int(b)] for b in net.line.to_bus.to_numpy()], dtype=np.int64)
        l_in = net.line.in_service.to_numpy(bool).copy() if nl else np.zeros(0, bool)
        if "line" in self.dynamic_service:
            l_in[:] = True
        open_f = np.zeros(nl, bool)
        open_t = np.zeros(nl, bool)
        if len(sw) and "switch" not in self.dynamic_service:
            ls = sw[(sw.et == "l") & ~sw.closed.astype(bool)]
            lpos = {int(l): i for i, l in enumerate(line_index)}
            for b, e in zip(ls.bus.to_numpy(), ls.element.to_numpy()):
                i = lpos[int(e)]
                if pos_of[int(b)] == lf[i]:
                    open_f[i] = True
                else:
                    open_t[i] = True
        l_in &= ~(open_f & open_t)
        l_in &= bus_in[lf] & bus_in[lt] if nl else l_in

        trafo_index = net.trafo.index.to_numpy()
        nt = len(trafo_index)
        th = np.array([pos_of[int(b)] for b in net.trafo.hv_bus.to_numpy()], dtype=np.int64)
        tl = np.array([pos_of[int(b)] for b in net.trafo.lv_bus.to_numpy()], dtype=np.int64)
        t_in = net.trafo.in_service.to_numpy(bool).copy() if nt else np.zeros(0, bool)
        if "trafo" in self.dynamic_service:
            t_in[:] = True
        if len(sw) and "switch" not in self.dynamic_service:
            ts = sw[(sw.et == "t") & ~sw.closed.astype(bool)]
            tpos = {int(t): i for i, t in enumerate(trafo_index)}
            for e in ts.element.to_numpy():
                t_in[tpos[int(e)]] = False
        if nt:
            t_in &= bus_in[th] & bus_in[tl]

        # node set: fused roots + auxiliary buses for half-open lines
        n_aux = int((l_in & (open_f ^ open_t)).sum())
        node_f = root[lf].copy() if nl else lf
        node_t = root[lt].copy() if nl else lt
        aux_vn = []
        k = n_pp
        vn = net.bus.vn_kv.to_numpy(float)
        for i in np.nonzero(l_in & (open_f ^ open_t))[0]:
            if open_f[i]:
                node_f[i] = k
                aux_vn.append(vn[lf[i]])
            else:
                node_t[i] = k
                aux_vn.append(vn[lt[i]])
            k += 1
        # three-winding transformers: one star-point node per element, auxiliary like the buses above (a star
        # that nothing in service reaches is dropped by the connectivity walk)
        t3 = getattr(net, "trafo3w", None)
        n3 = len(t3) if t3 is not None else 0
        if n3:
            t3_end = np.array([[pos_of[int(b)] for b in t3[c].to_numpy()] for c in ("hv_bus", "mv_bus", "lv_bus")],
                              dtype=np.int64).T                             # [n3, 3]
            t3_row_in = t3.in_service.to_numpy(bool)[:, None] & bus_in[t3_end]
            t3_star = n_pp + n_aux + np.arange(n3)
            aux_vn.extend(vn[t3_end[:, 0]])
        else:
            t3_end = np.zeros((0, 3), np.int64)
            t3_row_in = np.zeros((0, 3), bool)
            t3_star = np.zeros(0, np.int64)
        n_nodes = n_pp + n_aux + n3

        # impedance elements (pandapower build_branch._calc_impedance_parameter): plain series branches
        imp = getattr(net, "impedance", None)
        ni = len(imp) if imp is not None else 0
        if ni:
            imf = np.array([pos_of[int(b)] for b in imp.from_bus.to_numpy()], dtype=np.int64)
            imt = np.array([pos_of[int(b)] for b in imp.to_bus.to_numpy()], dtype=np.int64)
            i_in = imp.in_service.to_numpy(bool) & bus_in[imf] & bus_in[imt]
        else:
            imf = imt = np.zeros(0, np.int64)
            i_in = np.zeros(0, bool)

        # connectivity from in-service ext_grid buses
        adj = [[] for _ in range(n_nodes)]
        for i in np.nonzero(i_in)[0]:
            a, b = root[imf[i]], root[imt[i]]
            adj[a].append(b)
            adj[b].append(a)
        for i in np.nonzero(l_in)[0]:
            adj[node_f[i]].append(node_t[i])
            adj[node_t[i]].append(node_f[i])
        for i in np.nonzero(t_in)[0]:
            a, b = root[th[i]], root[tl[i]]
            adj[a].append(b)
            adj[b].append(a)
        for k, w in zip(*np.nonzero(t3_row_in)):
            a, b = t3_star[k], root[t3_end[k, w]]
            adj[a].append(b)
            adj[b].append(a)
        eg_in = net.ext_grid.in_service.to_numpy(bool) if len(net.ext_grid) else np.zeros(0, bool)
        eg_pos = np.array([pos_of[int(b)] for b in net.ext_grid.bus.to_numpy()], dtype=np.int64)
        seen = np.zeros(n_nodes, bool)
        stack = [int(root[p]) for p, s in zip(eg_pos, eg_in) if s and bus_in[p]]
        if len(net.gen) and "slack" in net.gen:
            for b, s, ins in zip(net.gen.bus.to_numpy(), net.gen.slack.to_numpy(),
                                 net.gen.in_service.to_numpy()):
                if s and ins:
                    stack.append(int(root[pos_of[int(b)]]))
        for s in stack:
            seen[s] = True
        while stack:
            a = stack.pop()
            for b in adj[a]:
                if not seen[b]:
                    seen[b] = True
                    stack.append(b)

        keep_nodes = [i for i in range(n_nodes)
                      if seen[i] and (i >= n_pp or (root[i] == i and bus_in[i]))]
        node_id = -np.ones(n_nodes, dtype=np.int64)
        node_id[keep_nodes] = np.arange(len(keep_nodes))
        self.nb = len(keep_nodes)
        self.bus_lookup = np.where(bus_in & seen[root], node_id[root], -1)
        base_kv_nodes = np.concatenate([vn, np.array(aux_vn, float)])
        self.base_kv = base_kv_nodes[keep_nodes]
        self._rep_bus_pos = np.array([i if i < n_pp else -1 for i in keep_nodes])

        l_in &= (node_id[node_f] >= 0) & (node_id[node_t] >= 0) if nl else l_in
        if nt:
            t_in &= (node_id[root[th]] >= 0) & (node_id[root[tl]] >= 0)
        self.line_pos = np.nonzero(l_in)[0]
        self.trafo_pos = np.nonzero(t_in)[0]
        self.line_f = node_id[node_f[self.line_pos]] if nl else np.zeros(0, np.int64)
        self.line_t = node_id[node_t[self.line_pos]] if nl else np.zeros(0, np.int64)
        self.trafo_h = node_id[root[th[self.trafo_pos]]] if nt else np.zeros(0, np.int64)
        self.trafo_l = node_id[root[tl[self.trafo_pos]]] if nt else np.zeros(0, np.int64)
        self.line_branch = -np.ones(nl, dtype=np.int64)
        self.line_branch[self.line_pos] = np.arange(len(self.line_pos))
        self.trafo_branch = -np.ones(nt, dtype=np.int64)
        self.trafo_branch[self.trafo_pos] = len(self.line_pos) + np.arange(len(self.trafo_pos))
        # trafo3w rows in pandapower's stacking: every hv row, then every mv row, then every lv row
        if n3:
            t3_row_in &= (node_id[t3_star][:, None] >= 0) & (node_id[root[t3_end]] >= 0)
        self.trafo3w_rows = [(int(k), w) for w in range(3) for k in np.nonzero(t3_row_in[:, w])[0]]
        star = [int(node_id[t3_star[k]]) for k, _ in self.trafo3w_rows]
        outer = [int(node_id[root[t3_end[k, w]]]) for k, w in self.trafo3w_rows]
        self.trafo3w_f = np.array([o if w == 0 else st for (_, w), st, o in zip(self.trafo3w_rows, star, outer)],
                                  dtype=np.int64)
        self.trafo3w_t = np.array([st if w == 0 else o for (_, w), st, o in zip(self.trafo3w_rows, star, outer)],
                                  dtype=np.int64)
        first3 = self.trafo3w_first = len(self.line_pos) + len(self.trafo_pos)
        self.trafo3w_branch = -np.ones((n3, 3), dtype=np.int64)
        for r, (k, w) in enumerate(self.trafo3w_rows):
            self.trafo3w_branch[k, w] = first3 + r
        if ni:
            i_in &= (node_id[root[imf]] >= 0) & (node_id[root[imt]] >= 0)
        self.imp_pos = np.nonzero(i_in)[0]
        self.imp_f = node_id[root[imf[self.imp_pos]]] if ni else np.zeros(0, np.int64)
        self.imp_t = node_id[root[imt[self.imp_pos]]] if ni else np.zeros(0, np.int64)
        self.impedance_branch = -np.ones(ni, dtype=np.int64)
        self.impedance_branch[self.imp_pos] = first3 + len(self.trafo3w_rows) + np.arange(len(self.imp_pos))
        self.n_pp_bus = n_pp

    def element_bus(self, net, table) -> np.ndarray:
        """ppc bus of every row of ``net[table]`` (-1 if the bus was dropped)."""
        pos = np.array([self._pos_of[int(b)] for b in net[table].bus.to_numpy()], dtype=np.int64)
        return self.bus_lookup[pos] if len(pos) else pos

    # ------------------------------------------------------------------- numbers
    def branch_table(self, net) -> tuple[np.ndarray, np.ndarray, np.ndarray]:
        sn = net.sn_mva
        nl, nt, ni = len(self.line_pos), len(self.trafo_pos), len(self.imp_pos)
        n3r = len(self.trafo3w_rows)
        br = np.zeros((nl + nt + n3r + ni, BRANCH_COLS))
        br[:, TAP] = 1.0
        br[:, BR_STATUS] = 1.0
        br[:, ANGMIN], br[:, ANGMAX] = -360.0, 360.0
        rate_f = np.zeros(nl + nt + n3r + ni)
        rate_t = np.zeros(nl + nt + n3r + ni)
        if nl:
            ln = net.line.iloc[self.line_pos]
            vn_f = self.base_kv[self.line_f]
            base_r = vn_f ** 2 / sn
            length = ln.length_km.to_numpy(float)
            par = ln.parallel.to_numpy(float)
            br[:nl, F_BUS] = self.line_f
            br[:nl, T_BUS] = self.line_t
            br[:nl, BR_R] = ln.r_ohm_per_km.to_numpy(float) * length / base_r / par
            br[:nl, BR_X] = ln.x_ohm_per_km.to_numpy(float) * length / base_r / par
            br[:nl, BR_B] = (2 * np.pi * net.f_hz * ln.c_nf_per_km.to_numpy(float)
                             * 1e-9 * base_r * length * par)
            br[:nl, BR_G] = ln.g_us_per_km.to_numpy(float) * 1e-6 * base_r * length * par
            imax = ln.max_i_ka.to_numpy(float) * ln.df.to_numpy(float) * par
            br[:nl, RATE_A] = imax * vn_f * np.sqrt(3.0)
            rate_f[:nl] = 1.0 / (np.sqrt(3.0) * vn_f * imax)
            rate_t[:nl] = 1.0 / (np.sqrt(3.0) * self.base_kv[self.line_t] * imax)
        if nt:
            tr = net.trafo.iloc[self.trafo_pos]
            vn_hv_bus = self.base_kv[self.trafo_h]
            vn_lv_bus = self.base_kv[self.trafo_l]
            # tap changer (ratio only; tap_step_degree == 0)
            tap_pos = tr.tap_pos.to_numpy(float)
            tap_neutral = tr.tap_neutral.to_numpy(float)
            tap_step = tr.tap_step_percent.to_numpy(float)
            steps = np.nan_to_num(tap_step * (tap_pos - tap_neutral) / 100.0)
            side = tr.tap_side.to_numpy(object)
            on_hv = np.array([s == "hv" for s in side])
            on_lv = np.array([s == "lv" for s in side])
            r, x, g, b, ratio, self.trafo_ratio_neutral = trafo_branch_values(
                tr.vn_hv_kv.to_numpy(float), tr.vn_lv_kv.to_numpy(float), vn_hv_bus, vn_lv_bus,
                tr.sn_mva.to_numpy(float), tr.vk_percent.to_numpy(float), tr.vkr_percent.to_numpy(float),
                tr.pfe_kw.to_numpy(float), tr.i0_percent.to_numpy(float), steps, on_hv, on_lv,
                tr.parallel.to_numpy(float), sn, self.trafo_model)
            self.trafo_tap_on_hv = on_hv
            self.trafo_tap_on_lv = on_lv
            shift = tr.shift_degree.to_numpy(float) if self.calculate_voltage_angles else np.zeros(nt)
            par = tr.parallel.to_numpy(float)
            sn_t = tr.sn_mva.to_numpy(float)
            sl = slice(nl, nl + nt)
            br[sl, F_BUS] = self.trafo_h
            br[sl, T_BUS] = self.trafo_l
            br[sl, BR_R], br[sl, BR_X] = r, x
            br[sl, BR_G], br[sl, BR_B] = g, b
            br[sl, TAP] = ratio
            br[sl, SHIFT] = shift
            df = tr.df.to_numpy(float)
            br[sl, RATE_A] = sn_t * par * df
            # trafo_loading='current': 100*max(i_hv*vn_hv, i_lv*vn_lv)*sqrt3/sn
            rate_f[sl] = tr.vn_hv_kv.to_numpy(float) / (vn_hv_bus * sn_t * par * df)
            rate_t[sl] = tr.vn_lv_kv.to_numpy(float) / (vn_lv_bus * sn_t * par * df)
        if n3r:
            self._trafo3w_table(net, br, rate_f, rate_t, nl + nt)
        if ni:
            # pandapower build_branch._calc_impedance_parameter [ext-mem]: per unit on the element's own
            # sn_mva, rescaled to the net's; no shunt part, ratio 1, no rating (res_impedance has no loading)
            im = net.impedance.iloc[self.imp_pos]
            k = sn / im.sn_mva.to_numpy(float)
            rft, xft = im.rft_pu.to_numpy(float) * k, im.xft_pu.to_numpy(float) * k
            rtf, xtf = im.rtf_pu.to_numpy(float) * k, im.xtf_pu.to_numpy(float) * k
            if not (np.array_equal(rft, rtf) and np.array_equal(xft, xtf)):
                raise NotImplementedError("net.impedance with rtf_pu != rft_pu or xtf_pu != xft_pu: the branch "
                                          "model of the kernels is symmetric (pandapower's BR_R_ASYM / BR_X_ASYM)")
            sl = slice(nl + nt + n3r, nl + nt + n3r + ni)
            br[sl, F_BUS], br[sl, T_BUS] = self.imp_f, self.imp_t
            br[sl, BR_R], br[sl, BR_X] = rft, xft
        return br, rate_f, rate_t

    def _trafo3w_table(self, net, br, rate_f, rate_t, first):
        """Rows of the three 2-winding equivalents of every trafo3w (PANDAPOWER_ASSUMPTIONS 9-16)."""
        t3 = net.trafo3w
        n3 = len(t3)
        vk_s, vkr_s, sn_s = trafo3w_star_parameters(t3)
        vn_s = np.stack([t3[f"vn_{s}_kv"].to_numpy(float) for s in ("hv", "mv", "lv")])
        zero = np.zeros(n3)
        shift_s = np.stack([zero, t3.shift_mv_degree.to_numpy(float), t3.shift_lv_degree.to_numpy(float)])
        side = t3.tap_side.to_numpy(object)
        star = t3.tap_at_star_point.to_numpy(bool) if "tap_at_star_point" in t3 else np.zeros(n3, bool)
        steps = np.nan_to_num(t3.tap_step_percent.to_numpy(float) * (t3.tap_pos.to_numpy(float) -
                                                                    t3.tap_neutral.to_numpy(float)) / 100.0)
        # winding w's branch carries the tap changer: at its outer end (hv row: hv side, mv / lv rows: lv side), at
        # the star end with tap_at_star_point
        self.trafo3w_tap_w = np.array([("hv", "mv", "lv").index(x) if x in ("hv", "mv", "lv") else -1 for x in side])
        self.trafo3w_tap_at_lv = np.where(self.trafo3w_tap_w == 0, star, ~star)
        ks = np.array([k for k, _ in self.trafo3w_rows], dtype=np.int64)
        ws = np.array([w for _, w in self.trafo3w_rows], dtype=np.int64)
        tapped = self.trafo3w_tap_w[ks] == ws
        on_lv = tapped & self.trafo3w_tap_at_lv[ks]
        on_hv = tapped & ~self.trafo3w_tap_at_lv[ks]
        n = len(ks)
        one = np.ones(n)
        vn_f, vn_t = self.base_kv[self.trafo3w_f], self.base_kv[self.trafo3w_t]
        hv_row = ws == 0
        pfe = np.where(hv_row, t3.pfe_kw.to_numpy(float)[ks], 0.0)
        i0 = np.where(hv_row, t3.i0_percent.to_numpy(float)[ks], 0.0)
        r, x, g, b, ratio, self.trafo3w_ratio_neutral = trafo_branch_values(
            vn_s[0, ks], vn_s[ws, ks], vn_f, vn_t, sn_s[ws, ks], vk_s[ws, ks], vkr_s[ws, ks], pfe, i0,
            steps[ks], on_hv, on_lv, one, net.sn_mva, self.trafo_model)
        sl = slice(first, first + n)
        br[sl, F_BUS], br[sl, T_BUS] = self.trafo3w_f, self.trafo3w_t
        br[sl, BR_R], br[sl, BR_X] = r, x
        br[sl, BR_G], br[sl, BR_B] = g, b
        br[sl, TAP] = ratio
        br[sl, SHIFT] = shift_s[ws, ks] if self.calculate_voltage_angles else 0.0
        br[sl, RATE_A] = sn_s[ws, ks]
        # loading factors at the outer end only: vn_<side>_kv / (bus vn_kv * sn_<side>_mva)
        rate = vn_s[ws, ks] / (np.where(hv_row, vn_f, vn_t) * sn_s[ws, ks])
        rate_f[sl] = np.where(hv_row, rate, 0.0)
        rate_t[sl] = np.where(hv_row, 0.0, rate)

    def build(self, net) -> Ppc:
        sn = net.sn_mva
        nb = self.nb
        bus = np.zeros((nb, BUS_COLS))
        bus[:, BUS_I] = np.arange(nb)
        bus[:, BUS_TYPE] = PQ
        bus[:, BUS_AREA] = 1
        bus[:, ZONE] = 1
        bus[:, BASE_KV] = self.base_kv
        bus[:, VMAX], bus[:, VMIN] = 2.0, 0.0

        for table, sign in (("load", 1.0), ("sgen", -1.0), ("storage", 1.0)):
            df = net[table]
            if not len(df):
                continue
            b = self.element_bus(net, table)
            w = df.scaling.to_numpy(float) * df.in_service.to_numpy(bool) * sign
            ok = b >= 0
            bus[:, PD] += np.bincount(b[ok], (df.p_mw.to_numpy(float) * w)[ok], nb)
            bus[:, QD] += np.bincount(b[ok], (df.q_mvar.to_numpy(float) * w)[ok], nb)
        if len(net.shunt):
            df = net.shunt
            b = self.element_bus(net, "shunt")
            ok = (b >= 0) & df.in_service.to_numpy(bool)
            ratio = (self.base_kv[np.maximum(b, 0)] / df.vn_kv.to_numpy(float)) ** 2
            step = df.step.to_numpy(float)
            bus[:, GS] += np.bincount(b[ok], (df.p_mw.to_numpy(float) * step * ratio)[ok], nb)
            bus[:, BS] -= np.bincount(b[ok], (df.q_mvar.to_numpy(float) * step * ratio)[ok], nb)

        if len(net.ward):
            # pandapower build_bus: ps/qs join the loads (_calc_pq_elements_and_add_on_ppc), pz/qz the shunts
            # at the bus's own rated voltage (_calc_shunts_and_add_on_ppc) [ext-mem]
            df = net.ward
            b = self.element_bus(net, "ward")
            ok = (b >= 0) & df.in_service.to_numpy(bool)
            bus[:, PD] += np.bincount(b[ok], df.ps_mw.to_numpy(float)[ok], nb)
            bus[:, QD] += np.bincount(b[ok], df.qs_mvar.to_numpy(float)[ok], nb)
            bus[:, GS] += np.bincount(b[ok], df.pz_mw.to_numpy(float)[ok], nb)
            bus[:, BS] -= np.bincount(b[ok], df.qz_mvar.to_numpy(float)[ok], nb)

        # generators: ext_grids (REF) first, then gens (PV)
        eg, gn = net.ext_grid, net.gen
        eg_bus = self.element_bus(net, "ext_grid") if len(eg) else np.zeros(0, np.int64)
        gn_bus = self.element_bus(net, "gen") if len(gn) else np.zeros(0, np.int64)
        eg_ok = (eg_bus >= 0) & (eg.in_service.to_numpy(bool) if len(eg) else True)
        gn_ok = (gn_bus >= 0) & (gn.in_service.to_numpy(bool) if len(gn) else True)
        n_eg, n_gn = int(np.sum(eg_ok)), int(np.sum(gn_ok))
        gen = np.zeros((n_eg + n_gn, GEN_COLS))
        gen[:, MBASE] = sn
        gen[:, GEN_STATUS] = 1
        ext_grid_gen = -np.ones(len(eg), dtype=np.int64)
        gen_gen = -np.ones(len(gn), dtype=np.int64)
        if n_eg:
            ext_grid_gen[eg_ok] = np.arange(n_eg)
            gen[:n_eg, GEN_BUS] = eg_bus[eg_ok]
            gen[:n_eg, VG] = eg.vm_pu.to_numpy(float)[eg_ok]
            bus[eg_bus[eg_ok], BUS_TYPE] = REF
            bus[eg_bus[eg_ok], VA] = eg.va_degree.to_numpy(float)[eg_ok]
        if n_gn:
            gen_gen[gn_ok] = n_eg + np.arange(n_gn)
            sl = slice(n_eg, n_eg + n_gn)
            gen[sl, GEN_BUS] = gn_bus[gn_ok]
            gen[sl, PG] = (gn.p_mw.to_numpy(float) * gn.scaling.to_numpy(float))[gn_ok]
            gen[sl, VG] = gn.vm_pu.to_numpy(float)[gn_ok]
            qmax = gn.max_q_mvar.to_numpy(float)[gn_ok] if "max_q_mvar" in gn else np.full(n_gn, np.nan)
            qmin = gn.min_q_mvar.to_numpy(float)[gn_ok] if "min_q_mvar" in gn else np.full(n_gn, np.nan)
            gen[sl, QMAX] = np.where(np.isnan(qmax), 1e9, qmax)
            gen[sl, QMIN] = np.where(np.isnan(qmin), -1e9, qmin)
            pv_bus = gn_bus[gn_ok]
            is_slack = gn.slack.to_numpy(bool)[gn_ok] if "slack" in gn else np.zeros(n_gn, bool)
            bus[pv_bus, BUS_TYPE] = np.where(
                is_slack, REF, np.maximum(bus[pv_bus, BUS_TYPE], PV))
            bus[pv_bus[bus[pv_bus, BUS_TYPE] == PQ], BUS_TYPE] = PV

        vm_set = np.concatenate([eg.vm_pu.to_numpy(float) if len(eg) else np.zeros(0),
                                 gn.vm_pu.to_numpy(float) if len(gn) else np.zeros(0)])
        init_vm = float(vm_set.sum() / len(vm_set)) if len(vm_set) else 1.0
        bus[:, VM] = init_vm
        bus[gen[:, GEN_BUS].astype(int), VM] = gen[:, VG]

        branch, rate_f, rate_t = self.branch_table(net)
        return Ppc(base_mva=sn, bus=bus, gen=gen, branch=branch,
                   bus_lookup=self.bus_lookup.copy(),
                   line_branch=self.line_branch.copy(),
                   trafo_branch=self.trafo_branch.copy(),
                   ext_grid_gen=ext_grid_gen, gen_gen=gen_gen,
                   rate_f=rate_f, rate_t=rate_t, init_vm_pu=init_vm,
                   impedance_branch=self.impedance_branch.copy(),
                   trafo3w_branch=self.trafo3w_branch.copy())


def build_ppc(net, **kwargs) -> Ppc:
    return PpcBuilder(net, **kwargs).build(net)
