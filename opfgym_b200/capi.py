"""ctypes declarations of the C ABI in ``include/opfg_b200.h``.

``load()`` opens the CUDA library built in-tree by ``__graft_entry__.build()``
(``opfgym_b200/lib/libopfg_b200.so``).  There is no CPU implementation behind
this module: if the library is missing, loading fails loudly.
"""
from __future__ import annotations

import ctypes as C
import os

LIB_NAME = "libopfg_b200.so"
LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "lib", LIB_NAME)
N_STATS = 24
DYN_TAP_LV, DYN_TRAFO, DYN_NORMALLY_OPEN = 1, 2, 4      # OpfgDynBranchDesc.flags bits (include/opfg_b200.h)

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


class GridDesc(C.Structure):
    _fields_ = [("nb", C.c_int32), ("ng", C.c_int32), ("nbr", C.c_int32),
                ("base_mva", C.c_double),
                ("bus", _dp), ("bus_cols", C.c_int32),
                ("gen", _dp), ("gen_cols", C.c_int32),
                ("branch", _dp), ("branch_cols", C.c_int32),
                ("tol_pu", C.c_double), ("max_iter", C.c_int32), ("init_dc", C.c_int32),
                ("enforce_q_lims", C.c_int32), ("threads_per_env", C.c_int32),
                ("ordering", C.c_int32), ("pf_kernel", C.c_int32)]


class GridInfo(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("nb", "n_nonref", "nnz_y", "n_blocks", "n_fill_blocks", "n_levels",
                 "threads_per_env", "smem_bytes_pf", "smem_bytes_score", "n_state",
                 "n_const", "n_act", "n_obs", "n_constraints")] + \
               [(n, C.c_double) for n in
                ("flops_per_iter", "flops_score", "lu_flops", "bytes_per_step")] + \
               [(n, C.c_int32) for n in ("pf_kernel_used", "lane_max_row", "lane_warps_per_cta",
                                         "lane_tables_staged")] + [("lane_scratch_bytes", C.c_double)] + \
               [(n, C.c_int32) for n in ("radial_lanes_per_env", "radial_envs_per_cta",
                                         "radial_smem_bytes_per_env", "n_island_critical",
                                         "cta_envs_per_cta", "cta_tables_staged", "score_threads_per_env")]


class AssemblyDesc(C.Structure):
    _fields_ = [("n_state", C.c_int32), ("n_const", C.c_int32), ("consts", _dp),
                ("n_act", C.c_int32), ("act_slot", _ip), ("act_lo", _ip), ("act_hi", _ip),
                ("act_div", _ip), ("act_kind", _ip), ("act_clamp_lo", _ip),
                ("act_clamp_hi", _ip), ("act_diff_step", C.c_double),
                ("n_inj", C.c_int32), ("inj_bus", _ip), ("inj_p", _ip), ("inj_q", _ip),
                ("inj_coef", _ip), ("bus_vm_ref", _ip)]


class ScoringDesc(C.Structure):
    _fields_ = [("n_inputs", C.c_int32), ("n_pp_bus", C.c_int32), ("pp_bus_lookup", _ip),
                ("res_bus_vm_slot", C.c_int32), ("res_bus_va_slot", C.c_int32),
                ("branch_loading_slot", _ip), ("branch_flow_slot", _ip),
                ("rate_f", _dp), ("rate_t", _dp), ("gen_p_slot", _ip), ("gen_q_slot", _ip),
                ("n_constraints", C.c_int32), ("con_ptr", _ip), ("con_value", _ip),
                ("con_value_scale", _dp), ("con_min", _ip), ("con_max", _ip),
                ("con_bound_mul", _dp), ("con_autoscale", _dp), ("con_worst_case", _ip),
                ("con_penalty_factor", _dp), ("con_penalty_power", _dp),
                ("con_count_penalty", _dp),
                ("n_poly", C.c_int32), ("poly_p", _ip), ("poly_p_mul", _dp), ("poly_q", _ip),
                ("poly_q_mul", _dp), ("poly_coef", _ip),
                ("n_pwl", C.c_int32), ("n_pwl_seg", C.c_int32), ("pwl_v", _ip),
                ("pwl_v_mul", _dp), ("pwl_seg", _ip),
                ("reward_kind", C.c_int32), ("penalty_weight", C.c_double),
                ("clip_lo", C.c_double), ("clip_hi", C.c_double),
                ("objective_factor", C.c_double), ("objective_bias", C.c_double),
                ("penalty_factor", C.c_double), ("penalty_bias", C.c_double),
                ("valid_reward", C.c_double), ("invalid_penalty", C.c_double),
                ("invalid_objective_share", C.c_double),
                ("n_obs", C.c_int32), ("obs_ref", _ip), ("obs_ptr", _ip)]


class DynBranchDesc(C.Structure):
    _fields_ = [("n_dyn", C.c_int32), ("branch", _ip), ("tap_pos", _ip), ("tap_neutral", _dp),
                ("tap_step_percent", _dp), ("ratio_neutral", _dp), ("in_service", _ip),
                ("closed_from", _ip), ("closed_to", _ip), ("flags", _ip)]


class RowOp(C.Structure):
    _fields_ = [("op", C.c_int32), ("dst", C.c_int32), ("a", C.c_int32), ("b", C.c_int32),
                ("imm", C.c_double)]


class ResetStage(C.Structure):
    _fields_ = [("kind", C.c_int32), ("n_cols", C.c_int32), ("slots", C.c_void_p), ("lo", C.c_void_p),
                ("hi", C.c_void_p), ("div", C.c_void_p), ("stream_offset", C.c_uint32),
                ("program", C.c_void_p)]


class Batch(C.Structure):
    _fields_ = [("n_env", C.c_int64)] + [(n, C.c_void_p) for n in
                ("actions", "state", "sbus", "vm", "va", "converged", "iterations",
                 "reward", "objective", "penalty", "cost", "valids", "violations",
                 "penalties", "obs_f32", "obs_f64", "stats", "yval", "bry", "objective_offset")] + [
                ("absolute_actions", C.c_int32), ("stats_slots", C.c_int32)]


# every symbol include/opfg_b200.h declares: name -> (restype, argtypes)
PROTOTYPES = {
    "opfg_version": (C.c_int, []),
    "opfg_last_error": (C.c_char_p, []),
    "opfg_grid_create": (C.c_int, [C.POINTER(GridDesc), C.POINTER(C.c_void_p)]),
    "opfg_grid_destroy": (None, [C.c_void_p]),
    "opfg_set_assembly": (C.c_int, [C.c_void_p, C.POINTER(AssemblyDesc)]),
    "opfg_set_scoring": (C.c_int, [C.c_void_p, C.POINTER(ScoringDesc)]),
    "opfg_set_dynamic_branches": (C.c_int, [C.c_void_p, C.POINTER(DynBranchDesc)]),
    "opfg_grid_info": (C.c_int, [C.c_void_p, C.POINTER(GridInfo)]),
    "opfg_grid_symbolic": (C.c_int, [C.c_void_p, _ip, _ip]),
    "opfg_philox_uniform": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int64,
                                      C.c_int32, C.c_void_p, C.c_void_p]),
    "opfg_sample_uniform": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int64,
                                      C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                      C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "opfg_sample_uniform_obs": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int64,
                                          C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p,
                                          C.c_int32, C.c_void_p]),
    "opfg_sample_profiles": (C.c_int, [C.c_uint64, C.c_uint64, C.c_uint64, C.c_int64, C.c_int32, C.c_void_p,
                                       C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                       C.c_double, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "opfg_assemble": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "opfg_pf_solve": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "opfg_score": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "opfg_observe": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "opfg_mixed_create": (C.c_int, [C.c_int32, C.POINTER(C.c_void_p), C.POINTER(Batch), C.POINTER(C.c_void_p)]),
    "opfg_mixed_destroy": (None, [C.c_void_p]),
    "opfg_assemble_mixed": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "opfg_score_mixed": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "opfg_step": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p]),
    "opfg_row_program_create": (C.c_int, [C.c_int32, C.c_int32, C.POINTER(RowOp), C.c_int32,
                                          _dp, C.POINTER(C.c_void_p)]),
    "opfg_row_program_destroy": (None, [C.c_void_p]),
    "opfg_row_program_select_rows": (C.c_int, [C.c_void_p, C.c_int32, _ip]),
    "opfg_row_program_run": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p]),
    "opfg_reset_plan_create": (C.c_int, [C.POINTER(ResetStage), C.c_int32, C.POINTER(C.c_void_p)]),
    "opfg_reset_plan_destroy": (None, [C.c_void_p]),
    "opfg_reset_episode": (C.c_int, [C.c_void_p, C.POINTER(Batch), C.c_void_p, C.c_uint64, C.c_uint64,
                                     C.c_uint64, C.c_int32, C.c_uint32, C.c_void_p]),
    "opfg_fp64_probe": (C.c_int, [C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]),
    "opfg_launch_count": (C.c_int64, []),
}


def declare(lib):
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


_lib = None


def load(path: str | None = None):
    """Open the CUDA library.  Raises ``OSError`` with a build hint if absent."""
    global _lib
    if path is None and _lib is not None:
        return _lib
    p = path or LIB_PATH
    if not os.path.exists(p):
        raise OSError(f"{p} not found: build it with `python -c 'import __graft_entry__ as g; "
                      "g.build()'` (nvcc, sm_100a). opfgym_b200 has no CPU fallback.")
    lib = declare(C.CDLL(p))
    if path is None:
        _lib = lib
    return lib


class OpfgError(RuntimeError):
    pass


def check(lib, rc: int):
    if rc != 0:
        raise OpfgError(lib.opfg_last_error().decode())
