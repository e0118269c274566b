"""ctypes binding of libmpcmmd.so (include/mpcmmd.h).  There is deliberately NO fallback: if the
CUDA library is missing or cannot create a handle the import / call raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmpcmmd.so")

FP = C.POINTER(C.c_float)
IP = C.POINTER(C.c_int32)
UP = C.POINTER(C.c_uint32)

COST_KINDS = {"mmd_opt": 0, "mmd_random": 1, "cvar": 2, "saa": 3}
NOISE_KINDS = {"gaussian": 0, "beta": 1}
MMD_KERNELS = {"laplace": 0, "gaussian": 1}      # MPCMMD_KERNEL_*


class MpcmmdConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in ("num_batch", "num_prime", "num_reduced", "num_obs", "maxiter_cem", "ellite_num",
                                         "ellite_num_cost", "noise_kind", "num_samples_cem", "maxiter_beta_cem",
                                         "num_ellite_beta", "max_episodes")] + \
               [(n, C.c_float) for n in ("sigma_acc", "sigma_steer", "ksig_steer", "acc_const_noise", "steer_const_noise",
                                         "beta_a", "beta_b", "v_min", "v_max", "a_max", "y_lb", "y_ub", "a_obs_sq", "b_obs_sq",
                                         "wheel_base", "dt", "steer_max", "steer_rate_pen", "alpha_quant", "ker_wt", "lamda_inv",
                                         "alpha_mean", "alpha_cov", "one_minus_alpha_mean", "one_minus_alpha_cov",
                                         "sigma_clip", "sigma_random")] + \
               [(n, FP) for n in ("P", "Pdot", "Pddot", "Gx", "Gy", "Kx", "Ky", "Wfit")]


class MpcmmdOut(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("cx", "cy", "cost_lane", "cost_obs", "beta", "sigma", "res_beta")]


class MpcmmdRiskOut(C.Structure):
    """mpcmmd_risk_out (include/mpcmmd.h): the Monte-Carlo risk statistics of the validation entry points"""
    _fields_ = [("alpha", C.c_double), ("ker_wt", C.c_double)] + \
               [(n, C.c_void_p) for n in ("sigma", "p_coll", "p_lane", "mean_obs", "var_obs", "cvar_obs", "mmd_obs", "c_obs", "c_lane")]


EXPORTS = ("mpcmmd_last_error", "mpcmmd_version", "mpcmmd_create", "mpcmmd_create_with_kernel", "mpcmmd_destroy", "mpcmmd_solve", "mpcmmd_solve_host",
           "mpcmmd_last_launch_count", "mpcmmd_inner_cem_path", "mpcmmd_profile_solve", "mpcmmd_fp32_peak", "mpcmmd_xu_peaks", "mpcmmd_selfcheck_ieee", "mpcmmd_math_vec", "mpcmmd_rng_normal", "mpcmmd_rng_beta", "mpcmmd_get_tables",
           "mpcmmd_stage_project", "mpcmmd_stage_risk", "mpcmmd_stage_risk_injected", "mpcmmd_stage_init", "mpcmmd_stage_select", "mpcmmd_stage_noise", "mpcmmd_validate_host",
           "mpcmmd_validate_seeded_host", "mpcmmd_validate_threefry_host", "mpcmmd_validate_risk_host", "mpcmmd_validate_threefry_risk_host",
           "mpcmmd_risk_stats_host")

_lib = None


class MpcmmdError(RuntimeError):
    pass


def load():
    """Load libmpcmmd.so (built in-tree by __graft_entry__.build()).  Raises if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise MpcmmdError(f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU fallback)")
    lib = C.CDLL(LIB_PATH)
    lib.mpcmmd_last_error.restype = C.c_char_p
    V = C.c_void_p
    lib.mpcmmd_create.argtypes = [C.POINTER(MpcmmdConfig), C.c_int, C.POINTER(V)]
    lib.mpcmmd_create_with_kernel.argtypes = [C.POINTER(MpcmmdConfig), C.c_int, C.c_int, C.POINTER(V)]
    lib.mpcmmd_destroy.argtypes = [V]
    lib.mpcmmd_solve.argtypes = [V, C.c_int, C.c_int] + [V] * 7 + [C.POINTER(MpcmmdOut), V]
    lib.mpcmmd_solve_host.argtypes = [V, C.c_int, C.c_int] + [V] * 7 + [C.POINTER(MpcmmdOut)]
    lib.mpcmmd_last_launch_count.argtypes = [V]
    lib.mpcmmd_inner_cem_path.argtypes = [V]
    lib.mpcmmd_inner_cem_path.restype = C.c_char_p
    lib.mpcmmd_profile_solve.argtypes = [V, C.c_int, C.c_int, V, V]
    lib.mpcmmd_fp32_peak.argtypes = [C.c_int, V, V]
    lib.mpcmmd_xu_peaks.argtypes = [C.c_int, V]
    lib.mpcmmd_selfcheck_ieee.argtypes = [C.c_int, V]
    lib.mpcmmd_math_vec.argtypes = [C.c_int, V, V, V, C.c_int, C.c_int]
    lib.mpcmmd_rng_normal.argtypes = [C.c_uint32, C.c_uint32, C.c_int, V, C.c_int]
    lib.mpcmmd_rng_beta.argtypes = [C.c_uint32, C.c_uint32, V, V, C.c_int, V, C.c_int]
    lib.mpcmmd_get_tables.argtypes = [V, V, V, V]
    lib.mpcmmd_stage_project.argtypes = [V, C.c_int, V, V, V, C.c_float] + [V] * 9
    lib.mpcmmd_stage_risk.argtypes = [V, C.c_int, C.c_int] + [V] * 14
    lib.mpcmmd_stage_risk_injected.argtypes = [V, C.c_int, C.c_int] + [V] * 13
    lib.mpcmmd_stage_init.argtypes = [V, V, V, V]
    lib.mpcmmd_stage_select.argtypes = [V, C.c_int] + [V] * 8
    lib.mpcmmd_stage_noise.argtypes = [V, C.c_int32, C.c_int32] + [V] * 5
    lib.mpcmmd_validate_host.argtypes = [C.c_int] * 6 + [C.c_double] * 6 + [V] * 9
    lib.mpcmmd_validate_seeded_host.argtypes = [C.c_int] * 7 + [C.c_double] * 12 + [V] * 11
    lib.mpcmmd_validate_threefry_host.argtypes = [C.c_int] * 7 + [C.c_double] * 12 + [V] * 10
    RP = C.POINTER(MpcmmdRiskOut)
    lib.mpcmmd_validate_risk_host.argtypes = [C.c_int] * 6 + [C.c_double] * 6 + [V] * 7 + [RP]
    lib.mpcmmd_validate_threefry_risk_host.argtypes = [C.c_int] * 7 + [C.c_double] * 12 + [V] * 8 + [RP]
    lib.mpcmmd_risk_stats_host.argtypes = [C.c_int] * 3 + [V] * 2 + [RP]
    _lib = lib
    return lib


def check(rc: int):
    if rc != 0:
        raise MpcmmdError(load().mpcmmd_last_error().decode())
