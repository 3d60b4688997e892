"""ctypes binding of libdto.so (include/dto.h). The product path goes through this C ABI and
nothing else: if the library or a CUDA device is missing, calls fail loudly."""
from __future__ import annotations

import ctypes as C
import os
import re

from .build import LIB, build_runtime

_HEADER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", "include", "dto.h")


class DtoError(RuntimeError):
    def __init__(self, status: int, message: str):
        super().__init__(f"dto status {status}: {message}")
        self.status = status


class ShapeDesc(C.Structure):
    _fields_ = [
        ("T", C.c_int32),
        ("dynamics_kind", C.POINTER(C.c_int32)),
        ("cost_kind", C.POINTER(C.c_int32)),
        ("stage_kind", C.POINTER(C.c_int32)),
        ("use_general", C.c_int32),
        ("parameter_dim", C.POINTER(C.c_int32)),
        ("parameter_offset", C.POINTER(C.c_int32)),
        ("num_parameter", C.c_int32),
    ]


class SqpOptions(C.Structure):
    """dto_sqp_options (include/dto.h): SQPOptions of sqp.py for the native solver"""
    _fields_ = [("max_iter", C.c_int32), ("max_refactor", C.c_int32), ("max_backtrack", C.c_int32), ("soc", C.c_int32)] + [
        (n, C.c_double) for n in ("tol_constraint", "tol_dual", "dual_reg", "reg_first", "reg_min", "reg_max", "reg_inc_first", "reg_inc",
                                  "reg_dec", "armijo", "merit_margin", "merit_rho", "merit_min", "lm_first", "lm_min", "lm_grow", "lm_shrink",
                                  "lm_grow_below", "lm_zero", "lam_max", "exact_below", "mu_init", "barrier_kappa_eps", "barrier_kappa_mu",
                                  "barrier_theta_mu", "tau_min", "bound_push", "bound_frac", "kappa_sigma", "tiny_step", "bound_relax")] + [
        ("hessian_approximation", C.c_int32)]


_lib = None


def declared_symbols() -> list:
    """Every function include/dto.h declares (used by the CPU-side export test)."""
    with open(_HEADER) as f:
        src = f.read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(dto_[a-z0-9_]+)\s*\(", src)))


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    build_runtime()
    if not os.path.exists(LIB):
        raise RuntimeError(f"{LIB} is missing: the native runtime was not built (no fallback exists)")
    L = C.CDLL(LIB)
    vp, i64, i32, dp = C.c_void_p, C.c_int64, C.c_int32, C.POINTER(C.c_double)
    i64p, i32p, ip = C.POINTER(C.c_int64), C.POINTER(C.c_int32), C.POINTER(C.c_int)
    sig = {
        "dto_abi_version": (C.c_int, []),
        "dto_last_error": (C.c_char_p, []),
        "dto_status_string": (C.c_char_p, [C.c_int]),
        "dto_device_count": (C.c_int, []),
        "dto_model_load": (C.c_int, [C.c_char_p, C.POINTER(vp)]),
        "dto_model_destroy": (None, [vp]),
        "dto_model_name": (C.c_char_p, [vp]),
        "dto_model_hash": (C.c_char_p, [vp]),
        "dto_model_num_kinds": (C.c_int, [vp, C.c_int]),
        "dto_model_kind_dims": (C.c_int, [vp, C.c_int, C.c_int, i32p]),
        "dto_model_has_general": (C.c_int, [vp]),
        "dto_shape_create": (C.c_int, [vp, C.POINTER(ShapeDesc), C.POINTER(vp)]),
        "dto_shape_destroy": (None, [vp]),
        "dto_num_variables": (i64, [vp]),
        "dto_num_constraint": (i64, [vp]),
        "dto_num_jacobian": (i64, [vp]),
        "dto_num_hessian": (i64, [vp]),
        "dto_num_hessian_nonunique": (i64, [vp]),
        "dto_num_parameter": (i64, [vp]),
        "dto_hessian_available": (C.c_int, [vp]),
        "dto_jacobian_structure": (C.c_int, [vp, i64p, i64p]),
        "dto_hessian_lagrangian_structure": (C.c_int, [vp, i64p, i64p]),
        "dto_constraint_bounds": (C.c_int, [vp, dp, dp]),
        "dto_knot_layout": (C.c_int, [vp, i64p, i32p, i64p, i32p]),
        "dto_batch_create": (C.c_int, [vp, i64, ip, C.c_int, C.POINTER(vp)]),
        "dto_batch_destroy": (None, [vp]),
        "dto_batch_size": (i64, [vp]),
        "dto_batch_num_shards": (C.c_int, [vp]),
        "dto_set_parameters": (C.c_int, [vp, vp]),
        "dto_set_x": (C.c_int, [vp, vp]),
        "dto_set_duals": (C.c_int, [vp, vp, vp]),
        "dto_eval_objective": (C.c_int, [vp, vp]),
        "dto_eval_objective_gradient": (C.c_int, [vp, vp]),
        "dto_eval_constraint": (C.c_int, [vp, vp]),
        "dto_eval_constraint_jacobian": (C.c_int, [vp, vp]),
        "dto_eval_hessian_lagrangian": (C.c_int, [vp, vp]),
        "dto_eval_jacobian_hessian": (C.c_int, [vp, vp, vp]),
        "dto_eval_jacobian_hessian_host": (C.c_int, [vp, vp, vp, vp, vp, vp, C.c_int]),
        "dto_get_problem": (C.c_int, [vp, C.c_int, i64, vp]),
        "dto_get_last_x": (C.c_int, [vp, i64, vp]),
        "dto_device_pointer": (vp, [vp, C.c_int, C.c_int]),
        "dto_shard_begin": (i64, [vp, C.c_int]),
        "dto_shard_size": (i64, [vp, C.c_int]),
        "dto_shard_device": (C.c_int, [vp, C.c_int]),
        "dto_get_stream": (vp, [vp, C.c_int]),
        "dto_set_stream": (C.c_int, [vp, C.c_int, vp]),
        "dto_launch": (C.c_int, [vp, C.c_int]),
        "dto_sync": (C.c_int, [vp]),
        "dto_launch_count": (i64, [vp]),
        "dto_algorithmic_bytes_per_problem": (i64, [vp]),
        "dto_kernel_smem_bytes": (i64, [vp, C.c_int]),
        "dto_shape_compiled_gather": (C.c_int, [vp]),
        "dto_kkt_analyze": (C.c_int, [vp, i64p, i64p]),
        "dto_kkt_analyze_ex": (C.c_int, [vp, C.c_int, i64p, i64p]),
        "dto_hessian_block_count": (i64, [vp]),
        "dto_hessian_block_structure": (C.c_int, [vp, i64p, i64p]),
        "dto_kkt_create": (C.c_int, [vp, C.c_double, C.c_double, C.POINTER(vp)]),
        "dto_kkt_create_ex": (C.c_int, [vp, C.c_double, C.c_double, C.c_int, C.POINTER(vp)]),
        "dto_kkt_set_hessian_blocks": (C.c_int, [vp, vp]),
        "dto_kkt_get_hessian_blocks": (C.c_int, [vp, vp]),
        "dto_kkt_destroy": (None, [vp]),
        "dto_kkt_dim": (i64, [vp]),
        "dto_kkt_bandwidth": (i64, [vp]),
        "dto_kkt_row_width": (i64, [vp]),
        "dto_kkt_factor_bytes_per_problem": (i64, [vp]),
        "dto_kkt_permutation": (C.c_int, [vp, i64p]),
        "dto_kkt_solve": (C.c_int, [vp, vp]),
        "dto_kkt_solve_host": (C.c_int, [vp, vp, vp, vp, vp, C.c_int]),
        "dto_kkt_launch": (C.c_int, [vp, C.c_int]),
        "dto_kkt_get": (C.c_int, [vp, C.c_int, vp]),
        "dto_kkt_matrix": (C.c_int, [vp, i64, vp]),
        "dto_kkt_factor": (C.c_int, [vp, i64, vp, vp]),
        "dto_kkt_device_pointer": (vp, [vp, C.c_int, C.c_int]),
        "dto_kkt_set_primal_reg": (C.c_int, [vp, vp]),
        "dto_kkt_inertia": (C.c_int, [vp, vp]),
        "dto_kkt_launch_subset": (C.c_int, [vp, vp, i64]),
        "dto_kkt_set_fixed": (C.c_int, [vp, vp]),
        "dto_kkt_resolve": (C.c_int, [vp, vp, i64]),
        "dto_sqp_default_options": (None, [C.POINTER(SqpOptions)]),
        "dto_sqp_solve": (C.c_int, [vp, C.POINTER(SqpOptions)] + [vp] * 12),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def check(status: int) -> None:
    if status != 0:
        raise DtoError(status, lib().dto_last_error().decode(errors="replace"))
