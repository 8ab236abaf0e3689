"""Minimal pandapower-shaped network container.

pandapower is not installable in the build image (SURVEY.md §8c), yet the
reference's whole host API is written against ``pandapowerNet``: a bag of
pandas tables reached as ``net.bus`` / ``net['bus']`` (reference
``opfgym/opf_env.py:267,436,534``; ``opfgym/constraints.py:90-98``;
``opfgym/objective.py:48-54``).  This module provides just that shape --
tables, column names and ``create_*`` helpers -- so that env definitions,
tests and the oracle read like the reference's own code.  It is an input
*data format*, not a solver: nothing here computes a power flow.

Column names and defaults follow pandapower 2.x ``create.py`` [ext-mem]
(SURVEY.md App. B.2-B.3).
"""
from __future__ import annotations

import copy

import numpy as np
import pandas as pd

_TABLES = {
    "bus": ["name", "vn_kv", "type", "in_service"],
    "line": ["name", "from_bus", "to_bus", "length_km", "r_ohm_per_km",
             "x_ohm_per_km", "c_nf_per_km", "g_us_per_km", "max_i_ka", "df",
             "parallel", "in_service"],
    "trafo": ["name", "hv_bus", "lv_bus", "sn_mva", "vn_hv_kv", "vn_lv_kv",
              "vk_percent", "vkr_percent", "pfe_kw", "i0_percent",
              "shift_degree", "tap_side", "tap_neutral", "tap_min", "tap_max",
              "tap_step_percent", "tap_step_degree", "tap_pos", "parallel",
              "df", "in_service"],
    "trafo3w": ["name", "hv_bus", "mv_bus", "lv_bus", "sn_hv_mva", "sn_mv_mva", "sn_lv_mva",
                "vn_hv_kv", "vn_mv_kv", "vn_lv_kv", "vk_hv_percent", "vk_mv_percent",
                "vk_lv_percent", "vkr_hv_percent", "vkr_mv_percent", "vkr_lv_percent",
                "pfe_kw", "i0_percent", "shift_mv_degree", "shift_lv_degree", "tap_side",
                "tap_neutral", "tap_min", "tap_max", "tap_step_percent", "tap_step_degree",
                "tap_pos", "tap_at_star_point", "in_service"],
    "load": ["name", "bus", "p_mw", "q_mvar", "const_z_percent",
             "const_i_percent", "scaling", "in_service"],
    "sgen": ["name", "bus", "p_mw", "q_mvar", "scaling", "in_service"],
    "storage": ["name", "bus", "p_mw", "q_mvar", "scaling", "in_service"],
    "gen": ["name", "bus", "p_mw", "vm_pu", "min_q_mvar", "max_q_mvar",
            "scaling", "slack", "in_service"],
    "ext_grid": ["name", "bus", "vm_pu", "va_degree", "in_service"],
    "shunt": ["name", "bus", "p_mw", "q_mvar", "vn_kv", "step", "in_service"],
    "ward": ["name", "bus", "ps_mw", "qs_mvar", "pz_mw", "qz_mvar", "in_service"],
    "impedance": ["name", "from_bus", "to_bus", "rft_pu", "xft_pu", "rtf_pu", "xtf_pu", "sn_mva", "in_service"],
    "switch": ["bus", "element", "et", "closed"],
    "poly_cost": ["element", "et", "cp0_eur", "cp1_eur_per_mw",
                  "cp2_eur_per_mw2", "cq0_eur", "cq1_eur_per_mvar",
                  "cq2_eur_per_mvar2"],
    "pwl_cost": ["power_type", "element", "et", "points"],
}

_RES_TABLES = {
    "res_bus": ["vm_pu", "va_degree", "p_mw", "q_mvar"],
    "res_line": ["p_from_mw", "q_from_mvar", "p_to_mw", "q_to_mvar", "pl_mw",
                 "ql_mvar", "i_from_ka", "i_to_ka", "i_ka", "vm_from_pu",
                 "vm_to_pu", "loading_percent"],
    "res_trafo": ["p_hv_mw", "q_hv_mvar", "p_lv_mw", "q_lv_mvar", "pl_mw",
                  "ql_mvar", "i_hv_ka", "i_lv_ka", "vm_hv_pu", "vm_lv_pu",
                  "loading_percent"],
    "res_trafo3w": ["p_hv_mw", "q_hv_mvar", "p_mv_mw", "q_mv_mvar", "p_lv_mw", "q_lv_mvar",
                    "pl_mw", "ql_mvar", "loading_percent"],
    "res_ext_grid": ["p_mw", "q_mvar"],
    "res_load": ["p_mw", "q_mvar"],
    "res_sgen": ["p_mw", "q_mvar"],
    "res_storage": ["p_mw", "q_mvar"],
    "res_gen": ["p_mw", "q_mvar", "va_degree", "vm_pu"],
}


class LoadflowNotConverged(Exception):
    """Same role as ``pandapower.powerflow.LoadflowNotConverged`` (reference
    ``opfgym/opf_env.py:660,704``): raised by a single-env solver adapter."""


class Net:
    """Attribute/item-addressable bag of pandas tables (``pandapowerNet`` shape)."""

    def __init__(self, name: str = "", f_hz: float = 50.0, sn_mva: float = 1.0):
        self.name = name
        self.f_hz = float(f_hz)
        self.sn_mva = float(sn_mva)
        self.converged = False
        for table, cols in {**_TABLES, **_RES_TABLES}.items():
            setattr(self, table, pd.DataFrame(columns=cols))
        for table in _TABLES:
            df = getattr(self, table)
            for c in df.columns:
                if c in ("name", "type", "tap_side", "et", "power_type", "points"):
                    df[c] = df[c].astype(object)
                elif c in ("in_service", "closed", "slack", "tap_at_star_point"):
                    df[c] = df[c].astype(bool)
                elif c in ("bus", "from_bus", "to_bus", "hv_bus", "lv_bus",
                           "mv_bus", "element"):
                    df[c] = df[c].astype(np.int64)
                else:
                    df[c] = df[c].astype(np.float64)

    def __getitem__(self, key):
        return getattr(self, key)

    def __setitem__(self, key, value):
        setattr(self, key, value)

    def __contains__(self, key):
        return hasattr(self, key)

    def deepcopy(self) -> "Net":
        return copy.deepcopy(self)

    def __repr__(self):
        sizes = {t: len(getattr(self, t)) for t in _TABLES if len(getattr(self, t))}
        return f"Net({self.name!r}, sn_mva={self.sn_mva}, {sizes})"


def _append(net: Net, table: str, row: dict, index=None) -> int:
    df = net[table]
    if index is None:
        index = 0 if len(df) == 0 else int(df.index.max()) + 1
    for k in row:
        if k not in df.columns:
            df[k] = np.nan if not isinstance(row[k], (str, list, bool)) else None
    df.loc[index, list(row.keys())] = pd.Series(row, dtype=object)
    return index


def _bulk(net: Net, table: str, data: dict) -> np.ndarray:
    """Append many rows at once (much faster than row-wise ``.loc``)."""
    df = net[table]
    n = len(next(iter(data.values())))
    start = 0 if len(df) == 0 else int(df.index.max()) + 1
    new = pd.DataFrame(data, index=np.arange(start, start + n))
    for c in df.columns:
        if c not in new.columns:
            new[c] = _DEFAULTS.get((table, c), _DEFAULTS.get(c, np.nan))
    new = new[list(df.columns) + [c for c in new.columns if c not in df.columns]]
    out = new if len(df) == 0 else pd.concat([df, new])
    for c in df.columns:
        if len(df) == 0 and c in new.columns:
            try:
                out[c] = out[c].astype(df[c].dtype)
            except (TypeError, ValueError):
                pass
    net[table] = out
    return new.index.to_numpy()


_DEFAULTS = {
    "name": None, "in_service": True, "scaling": 1.0, "parallel": 1.0,
    "df": 1.0, "g_us_per_km": 0.0, "const_z_percent": 0.0,
    "const_i_percent": 0.0, "q_mvar": 0.0, "type": "b", "va_degree": 0.0,
    "slack": False, "tap_step_degree": 0.0, "tap_at_star_point": False, "step": 1.0, "closed": True,
    "min_q_mvar": np.nan, "max_q_mvar": np.nan,
    "cp0_eur": 0.0, "cp1_eur_per_mw": 0.0, "cp2_eur_per_mw2": 0.0,
    "cq0_eur": 0.0, "cq1_eur_per_mvar": 0.0, "cq2_eur_per_mvar2": 0.0,
}


def create_empty_network(name="", f_hz=50.0, sn_mva=1.0) -> Net:
    return Net(name, f_hz, sn_mva)


def create_buses(net, n, vn_kv, **cols) -> np.ndarray:
    data = {"vn_kv": np.broadcast_to(np.asarray(vn_kv, float), (n,)).copy()}
    data.update({k: np.broadcast_to(np.asarray(v), (n,)).copy() for k, v in cols.items()})
    return _bulk(net, "bus", data)


def create_bus(net, vn_kv, **cols) -> int:
    return int(create_buses(net, 1, vn_kv, **cols)[0])


def create_lines_from_parameters(net, from_buses, to_buses, length_km,
                                 r_ohm_per_km, x_ohm_per_km, c_nf_per_km,
                                 max_i_ka, **cols) -> np.ndarray:
    n = len(from_buses)
    data = {"from_bus": np.asarray(from_buses, np.int64),
            "to_bus": np.asarray(to_buses, np.int64)}
    for k, v in dict(length_km=length_km, r_ohm_per_km=r_ohm_per_km,
                     x_ohm_per_km=x_ohm_per_km, c_nf_per_km=c_nf_per_km,
                     max_i_ka=max_i_ka, **cols).items():
        data[k] = np.broadcast_to(np.asarray(v), (n,)).copy()
    return _bulk(net, "line", data)


def create_line_from_parameters(net, from_bus, to_bus, length_km, r_ohm_per_km,
                                x_ohm_per_km, c_nf_per_km, max_i_ka, **cols) -> int:
    return int(create_lines_from_parameters(
        net, [from_bus], [to_bus], length_km, r_ohm_per_km, x_ohm_per_km,
        c_nf_per_km, max_i_ka, **cols)[0])


def create_transformer_from_parameters(net, hv_bus, lv_bus, sn_mva, vn_hv_kv,
                                       vn_lv_kv, vkr_percent, vk_percent,
                                       pfe_kw, i0_percent, shift_degree=0.0,
                                       tap_side=None, tap_neutral=np.nan,
                                       tap_min=np.nan, tap_max=np.nan,
                                       tap_step_percent=np.nan, tap_pos=np.nan,
                                       **cols) -> int:
    if np.isnan(tap_pos) and not np.isnan(tap_neutral):
        tap_pos = tap_neutral
    data = dict(hv_bus=[int(hv_bus)], lv_bus=[int(lv_bus)], sn_mva=[sn_mva],
                vn_hv_kv=[vn_hv_kv], vn_lv_kv=[vn_lv_kv],
                vkr_percent=[vkr_percent], vk_percent=[vk_percent],
                pfe_kw=[pfe_kw], i0_percent=[i0_percent],
                shift_degree=[shift_degree], tap_side=[tap_side],
                tap_neutral=[tap_neutral], tap_min=[tap_min], tap_max=[tap_max],
                tap_step_percent=[tap_step_percent], tap_pos=[tap_pos])
    data.update({k: [v] for k, v in cols.items()})
    return int(_bulk(net, "trafo", data)[0])


def create_transformer3w_from_parameters(net, hv_bus, mv_bus, lv_bus, vn_hv_kv, vn_mv_kv, vn_lv_kv,
                                         sn_hv_mva, sn_mv_mva, sn_lv_mva, vk_hv_percent, vk_mv_percent,
                                         vk_lv_percent, vkr_hv_percent, vkr_mv_percent, vkr_lv_percent,
                                         pfe_kw, i0_percent, shift_mv_degree=0.0, shift_lv_degree=0.0,
                                         tap_side=None, tap_step_percent=np.nan, tap_step_degree=np.nan,
                                         tap_pos=np.nan, tap_neutral=np.nan, tap_max=np.nan, tap_min=np.nan,
                                         name=None, in_service=True, index=None, max_loading_percent=np.nan,
                                         tap_at_star_point=False, **cols) -> int:
    """Same call shape as ``pp.create_transformer3w_from_parameters``.  The short-circuit voltages are
    pairwise: ``vk_hv_percent`` hv-mv, ``vk_mv_percent`` mv-lv, ``vk_lv_percent`` hv-lv."""
    if np.isnan(tap_pos) and not np.isnan(tap_neutral):
        tap_pos = tap_neutral
    data = dict(hv_bus=[int(hv_bus)], mv_bus=[int(mv_bus)], lv_bus=[int(lv_bus)],
                sn_hv_mva=[sn_hv_mva], sn_mv_mva=[sn_mv_mva], sn_lv_mva=[sn_lv_mva],
                vn_hv_kv=[vn_hv_kv], vn_mv_kv=[vn_mv_kv], vn_lv_kv=[vn_lv_kv],
                vk_hv_percent=[vk_hv_percent], vk_mv_percent=[vk_mv_percent], vk_lv_percent=[vk_lv_percent],
                vkr_hv_percent=[vkr_hv_percent], vkr_mv_percent=[vkr_mv_percent],
                vkr_lv_percent=[vkr_lv_percent], pfe_kw=[pfe_kw], i0_percent=[i0_percent],
                shift_mv_degree=[shift_mv_degree], shift_lv_degree=[shift_lv_degree], tap_side=[tap_side],
                tap_neutral=[tap_neutral], tap_min=[tap_min], tap_max=[tap_max],
                tap_step_percent=[tap_step_percent], tap_step_degree=[tap_step_degree], tap_pos=[tap_pos],
                tap_at_star_point=[bool(tap_at_star_point)], in_service=[bool(in_service)], name=[name])
    if not np.isnan(max_loading_percent):
        data["max_loading_percent"] = [float(max_loading_percent)]
    data.update({k: [v] for k, v in cols.items()})
    out = int(_bulk(net, "trafo3w", data)[0])
    if index is not None:
        net.trafo3w = net.trafo3w.rename(index={out: int(index)})
        out = int(index)
    return out


def _create_pq(net, table, buses, p_mw, q_mvar, **cols) -> np.ndarray:
    n = len(buses)
    data = {"bus": np.asarray(buses, np.int64),
            "p_mw": np.broadcast_to(np.asarray(p_mw, float), (n,)).copy(),
            "q_mvar": np.broadcast_to(np.asarray(q_mvar, float), (n,)).copy()}
    data.update({k: np.broadcast_to(np.asarray(v), (n,)).copy() for k, v in cols.items()})
    return _bulk(net, table, data)


def create_loads(net, buses, p_mw, q_mvar=0.0, **cols):
    return _create_pq(net, "load", buses, p_mw, q_mvar, **cols)


def create_sgens(net, buses, p_mw, q_mvar=0.0, **cols):
    return _create_pq(net, "sgen", buses, p_mw, q_mvar, **cols)


def create_storages(net, buses, p_mw, q_mvar=0.0, **cols):
    return _create_pq(net, "storage", buses, p_mw, q_mvar, **cols)


def create_load(net, bus, p_mw, q_mvar=0.0, **cols) -> int:
    return int(create_loads(net, [bus], p_mw, q_mvar, **cols)[0])


def create_sgen(net, bus, p_mw, q_mvar=0.0, **cols) -> int:
    return int(create_sgens(net, [bus], p_mw, q_mvar, **cols)[0])


def create_storage(net, bus, p_mw, q_mvar=0.0, **cols) -> int:
    return int(create_storages(net, [bus], p_mw, q_mvar, **cols)[0])


def create_gen(net, bus, p_mw, vm_pu=1.0, **cols) -> int:
    data = {"bus": [int(bus)], "p_mw": [float(p_mw)], "vm_pu": [float(vm_pu)]}
    data.update({k: [v] for k, v in cols.items()})
    return int(_bulk(net, "gen", data)[0])


def create_ext_grid(net, bus, vm_pu=1.0, va_degree=0.0, **cols) -> int:
    data = {"bus": [int(bus)], "vm_pu": [float(vm_pu)], "va_degree": [float(va_degree)]}
    data.update({k: [v] for k, v in cols.items()})
    return int(_bulk(net, "ext_grid", data)[0])


def create_shunt(net, bus, q_mvar, p_mw=0.0, **cols) -> int:
    vn = float(net.bus.vn_kv.loc[bus])
    data = {"bus": [int(bus)], "p_mw": [float(p_mw)], "q_mvar": [float(q_mvar)],
            "vn_kv": [vn]}
    data.update({k: [v] for k, v in cols.items()})
    return int(_bulk(net, "shunt", data)[0])


def create_ward(net, bus, ps_mw, qs_mvar, pz_mw, qz_mvar, **cols) -> int:
    data = {"bus": [int(bus)], "ps_mw": [float(ps_mw)], "qs_mvar": [float(qs_mvar)], "pz_mw": [float(pz_mw)],
            "qz_mvar": [float(qz_mvar)]}
    data.update({k: [v] for k, v in cols.items()})
    return int(_bulk(net, "ward", data)[0])


def create_impedance(net, from_bus, to_bus, rft_pu, xft_pu, sn_mva, rtf_pu=None, xtf_pu=None, **cols) -> int:
    data = {"from_bus": [int(from_bus)], "to_bus": [int(to_bus)], "rft_pu": [float(rft_pu)], "xft_pu": [float(xft_pu)],
            "rtf_pu": [float(rft_pu if rtf_pu is None else rtf_pu)], "xtf_pu": [float(xft_pu if xtf_pu is None else xtf_pu)],
            "sn_mva": [float(sn_mva)]}
    data.update({k: [v] for k, v in cols.items()})
    return int(_bulk(net, "impedance", data)[0])


def create_switch(net, bus, element, et, closed=True) -> int:
    data = {"bus": [int(bus)], "element": [int(element)], "et": [et],
            "closed": [bool(closed)]}
    return int(_bulk(net, "switch", data)[0])


def create_poly_cost(net, element, et, cp1_eur_per_mw=0.0, cp0_eur=0.0,
                     cq1_eur_per_mvar=0.0, cq0_eur=0.0, cp2_eur_per_mw2=0.0,
                     cq2_eur_per_mvar2=0.0) -> int:
    """Same call shape as ``pp.create_poly_cost`` (used at reference
    ``opfgym/envs/voltage_control.py:88-100``)."""
    data = dict(element=[int(element)], et=[et], cp0_eur=[cp0_eur],
                cp1_eur_per_mw=[cp1_eur_per_mw], cp2_eur_per_mw2=[cp2_eur_per_mw2],
                cq0_eur=[cq0_eur], cq1_eur_per_mvar=[cq1_eur_per_mvar],
                cq2_eur_per_mvar2=[cq2_eur_per_mvar2])
    return int(_bulk(net, "poly_cost", data)[0])


def create_pwl_cost(net, element, et, points, power_type="p") -> int:
    """Same call shape as ``pp.create_pwl_cost`` (reference
    ``opfgym/envs/eco_dispatch.py:95``, ``envs/load_shedding.py:104``)."""
    df = net.pwl_cost
    idx = 0 if len(df) == 0 else int(df.index.max()) + 1
    row = pd.DataFrame({"power_type": [power_type], "element": [int(element)],
                        "et": [et], "points": [None]}, index=[idx])
    for c in df.columns:
        if c not in row.columns:
            row[c] = np.nan
    out = row if len(df) == 0 else pd.concat([df, row])
    out["points"] = out["points"].astype(object)
    out.at[idx, "points"] = [list(map(float, p)) for p in points]
    net.pwl_cost = out
    return idx


def clear_results(net: Net) -> None:
    for table, cols in _RES_TABLES.items():
        net[table] = pd.DataFrame(columns=cols, dtype=float)
    net.converged = False
