"""CPU ORACLE -- TEST INFRASTRUCTURE ONLY.  Not imported by the product package.

Three-winding transformers for the oracle, restated the way pandapower 2.x itself handles them
(``build_branch._trafo_df_from_trafo3w`` and ``results_branch._get_trafo3w_results`` [ext-mem]): every
``net.trafo3w`` row is expanded, on a copy of the net, into one star-point BUS and three 2-winding ``net.trafo``
rows (hv->star, star->mv, star->lv).  The expanded net then goes through the unchanged ``oracle/ppc_ref.py``
conversion and ``oracle/pf.py`` solver; ``res_trafo3w`` is assembled afterwards from the three equivalents.

This is a different structure from the product's ``opfgym_b200/ppc.py`` on purpose: a net-level expansion
with scalar element loops, against the product's matrix-level rows on arrays.  Both follow the items of
``opfgym_b200.ppc.PANDAPOWER_ASSUMPTIONS`` numbered 9-16.

PARITY STATUS: unpinned at the pandapower boundary, like ``oracle/pf.py``.
"""
from __future__ import annotations

import math

import numpy as np
import pandas as pd

from oracle import pf, ppc_ref

SIDES = ("hv", "mv", "lv")


def _num(v, default=0.0):
    try:
        v = float(v)
    except (TypeError, ValueError):
        return default
    return default if math.isnan(v) else v


def star_impedances(t):
    """(vk, vkr) in % of the three star branches of one trafo3w row, each on its own winding rating."""
    sn = [float(t[f"sn_{s}_mva"]) for s in SIDES]
    pairs = ((0, 1), (1, 2), (0, 2))                          # vk_hv: hv-mv, vk_mv: mv-lv, vk_lv: hv-lv
    out_r, out_x = [], []
    delta_r, delta_x = [], []
    for (i, j), s in zip(pairs, SIDES):
        k = sn[0] / min(sn[i], sn[j])                         # referred to sn_hv
        vk, vkr = float(t[f"vk_{s}_percent"]) * k, float(t[f"vkr_{s}_percent"]) * k
        delta_r.append(vkr)
        delta_x.append(math.sqrt(vk * vk - vkr * vkr))
    hm, ml, hl = 0, 1, 2
    for w, (a, b, c) in enumerate(((hm, hl, ml), (ml, hm, hl), (hl, ml, hm))):
        f = 0.5 * sn[w] / sn[0]
        out_r.append(f * (delta_r[a] + delta_r[b] - delta_r[c]))
        out_x.append(f * (delta_x[a] + delta_x[b] - delta_x[c]))
    vk = [math.copysign(math.hypot(x, r), x) for r, x in zip(out_r, out_x)]
    return vk, out_r


def expand(net):
    """Copy of ``net`` with every trafo3w replaced by a star bus and three trafo rows.  Returns
    (copy, rows) where ``rows[(idx, w)]`` is the trafo index of winding w of trafo3w ``idx``."""
    ex = net.deepcopy()
    t3 = net.trafo3w
    rows = {}
    if not len(t3):
        return ex, rows
    star = {}
    next_bus = int(ex.bus.index.max()) + 1
    for idx, t in zip(t3.index, t3.to_dict("records")):
        star[int(idx)] = next_bus
        ex.bus.loc[next_bus, ["vn_kv", "in_service"]] = [float(net.bus.vn_kv.loc[int(t["hv_bus"])]), True]
        next_bus += 1
    ex.bus["in_service"] = ex.bus.in_service.astype(bool)
    next_tr = int(ex.trafo.index.max()) + 1 if len(ex.trafo) else 0
    new = []
    for w, side in enumerate(SIDES):                          # pandapower's stacking: hv rows, mv rows, lv rows
        for idx, t in zip(t3.index, t3.to_dict("records")):
            vk, vkr = star_impedances(t)
            at_star = bool(t.get("tap_at_star_point", False))
            tapped = t.get("tap_side") == side
            # the tap changer at the winding's terminal, or at the star end of its branch
            tap_side = None
            if tapped:
                outer_is_hv = w == 0
                tap_side = ("lv" if at_star else "hv") if outer_is_hv else ("hv" if at_star else "lv")
            row = dict(
                hv_bus=int(t["hv_bus"]) if w == 0 else star[int(idx)],
                lv_bus=star[int(idx)] if w == 0 else int(t[f"{side}_bus"]),
                sn_mva=float(t[f"sn_{side}_mva"]), vn_hv_kv=float(t["vn_hv_kv"]), vn_lv_kv=float(t[f"vn_{side}_kv"]),
                vk_percent=vk[w], vkr_percent=vkr[w],
                pfe_kw=float(t["pfe_kw"]) if w == 0 else 0.0, i0_percent=float(t["i0_percent"]) if w == 0 else 0.0,
                shift_degree=0.0 if w == 0 else _num(t[f"shift_{side}_degree"]),
                tap_side=tap_side, tap_neutral=_num(t["tap_neutral"]) if tapped else np.nan,
                tap_pos=_num(t["tap_pos"]) if tapped else np.nan,
                tap_step_percent=_num(t["tap_step_percent"]) if tapped else np.nan,
                tap_step_degree=0.0, parallel=1.0, df=1.0, in_service=bool(t["in_service"]))
            rows[(int(idx), w)] = next_tr
            new.append(pd.DataFrame({k: [v] for k, v in row.items()}, index=[next_tr]))
            next_tr += 1
    ex.trafo = pd.concat([ex.trafo] + new) if len(ex.trafo) else pd.concat(new)
    ex.trafo["tap_side"] = ex.trafo.tap_side.astype(object)
    ex.trafo3w = ex.trafo3w.iloc[:0]
    return ex, rows


def build(net, **kwargs):
    """``oracle.ppc_ref.build`` of the expanded net, with the lookups of the original one and
    ``trafo3w_branch`` [n, 3] (branch rows of the hv, mv, lv equivalents, -1 out) and ``trafo3w_rate``
    [n, 3] (loading factor at the outer end of each)."""
    ex, rows = expand(net)
    r = ppc_ref.build(ex, **kwargs)
    n_tr = len(net.trafo)
    pos_tr = {int(i): k for k, i in enumerate(ex.trafo.index)}
    r.bus_lookup = r.bus_lookup[:len(net.bus)]
    r.trafo3w_branch = -np.ones((len(net.trafo3w), 3), dtype=np.int64)
    r.trafo3w_rate = np.zeros((len(net.trafo3w), 3))
    for k, idx in enumerate(net.trafo3w.index):
        t = net.trafo3w.loc[idx]
        for w, side in enumerate(SIDES):
            row = int(r.trafo_branch[pos_tr[rows[(int(idx), w)]]])
            r.trafo3w_branch[k, w] = row
            if row >= 0:
                outer = int(r.branch[row, ppc_ref.F_BUS if w == 0 else ppc_ref.T_BUS])
                r.trafo3w_rate[k, w] = float(t[f"vn_{side}_kv"]) / (r.bus[outer, ppc_ref.BASE_KV] *
                                                                    float(t[f"sn_{side}_mva"]))
    r.trafo_branch = r.trafo_branch[:n_tr]
    return r


def runpp(net, **kwargs):
    """``oracle.pf.runpp`` on the expanded net; fills every ``res_*`` table of ``net`` itself, including
    ``res_trafo3w`` (flows at the outer ends, their sums, loading_percent)."""
    ex, rows = expand(net)
    res = pf.runpp(ex, **kwargs)
    for table in ("res_line", "res_ext_grid", "res_gen", "res_load", "res_sgen", "res_storage"):
        if table in vars(ex):
            net[table] = ex[table]
    net.res_bus = ex.res_bus.loc[net.bus.index]
    if "res_trafo" in vars(ex) and len(net.trafo):
        net.res_trafo = ex.res_trafo.loc[net.trafo.index]
    net.converged = ex.converged
    cols = {c: [] for c in ("p_hv_mw", "q_hv_mvar", "p_mv_mw", "q_mv_mvar", "p_lv_mw", "q_lv_mvar",
                            "loading_percent")}
    vm = ex.res_bus.vm_pu
    for idx in net.trafo3w.index:
        t = net.trafo3w.loc[idx]
        loading = 0.0
        for w, side in enumerate(SIDES):
            tr = ex.res_trafo.loc[rows[(int(idx), w)]]
            end = "hv" if w == 0 else "lv"                    # the outer end of the equivalent
            outer = int(t[f"{side}_bus"])
            p, q = float(tr[f"p_{end}_mw"]), float(tr[f"q_{end}_mvar"])
            if np.isnan(vm.loc[outer]):
                p = q = np.nan
            elif np.isnan(p):                                 # absent equivalent next to a live bus: no flow
                p = q = 0.0
            cols[f"p_{side}_mw"].append(p)
            cols[f"q_{side}_mvar"].append(q)
            i_ka = math.hypot(p, q) / (math.sqrt(3.0) * vm.loc[outer] * float(net.bus.vn_kv.loc[outer]))
            ld = i_ka * float(t[f"vn_{side}_kv"]) / float(t[f"sn_{side}_mva"]) * math.sqrt(3.0) * 100.0
            loading = np.nan if (np.isnan(ld) or np.isnan(loading)) else max(loading, ld)
        cols["loading_percent"].append(loading)
    df = pd.DataFrame(cols, index=net.trafo3w.index, dtype=float)
    df["pl_mw"] = df.p_hv_mw + df.p_mv_mw + df.p_lv_mw
    df["ql_mvar"] = df.q_hv_mvar + df.q_mv_mvar + df.q_lv_mvar
    net.res_trafo3w = df
    return res


class RefBuilder(ppc_ref.RefBuilder):
    """``build(net)`` that understands trafo3w (for ``oracle.pf.runpp(net, builder=...)`` style use)."""

    def build(self, net):
        return build(net, **self.kwargs)

