"""ctypes binding of libbrov.so (include/brov.h).  No torch types cross this boundary: pointers and sizes only.

The library is loaded from the package directory (built in-tree by `python -m bluerov2_dynamics_b200.build`).
There is no CPU fallback: if the library is missing the import of this module raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BROV_LIB") or os.path.join(_HERE, "libbrov.so")  # BROV_LIB: a tuning variant

ABI_VERSION = 8
THRUSTER8_LAG3, WRENCH_EULER12, WRENCH_QUAT13 = 0, 1, 2
DI_EULER12_U8, DI_EULER12_U6, DI_QUAT13_U6 = 3, 4, 5
F64, F32 = 0, 1
RK4, EULER = 0, 1
LAG_THRUSTER, LAG_PROJECTED = 0, 1
NPHYS, NKP, MAX_H = 37, 36, 4
PH_M, PH_W, PH_B, PH_XB, PH_I, PH_ADDED, PH_LIN, PH_QUAD, PH_MINV, PH_CURRENT, PH_TLAG1 = 0, 1, 2, 3, 6, 9, 15, 21, 27, 33, 36


class BrovError(RuntimeError):
    pass


class InputGen(C.Structure):
    """brov_input_gen: the in-kernel command-signal generator (see include/brov.h)."""
    _fields_ = [("enable", C.c_int32), ("reserved", C.c_int32), ("seed", C.c_uint64), ("vehicle0", C.c_longlong),
                ("rho", C.c_double), ("sigma", C.c_double), ("clip", C.c_double), ("scale", C.c_double * 8),
                ("state_in_dev", C.c_void_p), ("state_out_dev", C.c_void_p)]


class RolloutDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("dt", C.c_double), ("x0_dev", C.c_void_p), ("xT_dev", C.c_void_p), ("u_dev", C.c_void_p),
                ("u_stride_t", C.c_longlong), ("u_stride_n", C.c_longlong), ("lag_in_dev", C.c_void_p),
                ("lag_out_dev", C.c_void_p), ("traj_dev", C.c_void_p), ("stride", C.c_longlong),
                ("step0", C.c_longlong), ("snap_base", C.c_longlong), ("lag_in_repr", C.c_int32),
                ("lag_out_repr", C.c_int32), ("time_slices", C.c_int32), ("min_abs_cos_accumulate", C.c_int32),
                ("health_dev", C.c_void_p), ("min_abs_cos_dev", C.c_void_p), ("singular_eps", C.c_double),
                ("gen", InputGen)]


class GenInputsDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("dtype", C.c_int32), ("nu", C.c_int32), ("device", C.c_int32),
                ("first", C.c_longlong), ("vstride", C.c_longlong), ("n_sel", C.c_longlong),
                ("step0", C.c_longlong), ("steps", C.c_longlong), ("gen", InputGen), ("out_dev", C.c_void_p)]


class SeDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("rows", C.c_longlong),
                ("n_windows", C.c_longlong), ("dt", C.c_double), ("X_dev", C.c_void_p), ("U_dev", C.c_void_p),
                ("lag0_dev", C.c_void_p), ("n_horizons", C.c_int32), ("horizons", C.c_int32 * MAX_H),
                ("se_out_dev", C.c_void_p), ("count_out", C.POINTER(C.c_longlong)), ("workspace_dev", C.c_void_p),
                ("workspace_bytes", C.c_size_t), ("lag_carry", C.c_int32), ("time_slices", C.c_int32),
                ("window0", C.c_longlong), ("row0", C.c_longlong), ("health_dev", C.c_void_p),
                ("singular_eps", C.c_double)]


class SeSweepDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("rows", C.c_longlong),
                ("n_windows", C.c_longlong), ("dt", C.c_double), ("X_dev", C.c_void_p), ("U_dev", C.c_void_p),
                ("lag0_dev", C.c_void_p), ("n_horizons", C.c_int32), ("horizons", C.c_int32 * MAX_H),
                ("lag_carry", C.c_int32), ("window0", C.c_longlong), ("row0", C.c_longlong),
                ("n_candidates", C.c_longlong), ("kp_soa_dev", C.c_void_p), ("any_current", C.c_int32),
                ("reserved", C.c_int32), ("se_out_dev", C.c_void_p), ("count_out", C.POINTER(C.c_longlong)),
                ("health_dev", C.c_void_p), ("singular_eps", C.c_double), ("workspace_dev", C.c_void_p),
                ("workspace_bytes", C.c_size_t)]


class SeGradDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("rows", C.c_longlong),
                ("n_windows", C.c_longlong), ("dt", C.c_double), ("X_dev", C.c_void_p), ("U_dev", C.c_void_p),
                ("lag0_dev", C.c_void_p), ("n_horizons", C.c_int32), ("horizons", C.c_int32 * MAX_H),
                ("lag_carry", C.c_int32), ("window0", C.c_longlong), ("row0", C.c_longlong),
                ("kp_dev", C.c_void_p), ("any_current", C.c_int32), ("n_dirs", C.c_int32), ("dirs_dev", C.c_void_p),
                ("se_out_dev", C.c_void_p), ("grad_out_dev", C.c_void_p), ("gn_out_dev", C.c_void_p),
                ("count_out", C.POINTER(C.c_longlong)), ("health_dev", C.c_void_p), ("singular_eps", C.c_double),
                ("workspace_dev", C.c_void_p), ("workspace_bytes", C.c_size_t)]


class LinearizeDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("dt", C.c_double), ("z0_dev", C.c_void_p), ("u_dev", C.c_void_p), ("u_stride_t", C.c_longlong),
                ("u_stride_n", C.c_longlong), ("z_out_dev", C.c_void_p), ("z_traj_dev", C.c_void_p),
                ("jac_dev", C.c_void_p), ("health_dev", C.c_void_p), ("singular_eps", C.c_double)]


class ClosedLoopDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("dt", C.c_double), ("z0_dev", C.c_void_p), ("z_out_dev", C.c_void_p), ("K_dev", C.c_void_p),
                ("K_stride_t", C.c_longlong), ("K_stride_n", C.c_longlong), ("z_ref_dev", C.c_void_p),
                ("z_ref_stride_t", C.c_longlong), ("z_ref_stride_n", C.c_longlong), ("u_ref_dev", C.c_void_p),
                ("u_ref_stride_t", C.c_longlong), ("u_ref_stride_n", C.c_longlong), ("u_min", C.c_double * 8),
                ("u_max", C.c_double * 8), ("q", C.c_double * 30), ("r", C.c_double * 8), ("traj_dev", C.c_void_p),
                ("u_traj_dev", C.c_void_p), ("stride", C.c_longlong), ("cost_dev", C.c_void_p),
                ("cost_accumulate", C.c_int32), ("reserved", C.c_int32), ("health_dev", C.c_void_p),
                ("singular_eps", C.c_double)]


class EkfDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("dt", C.c_double), ("z0_dev", C.c_void_p), ("P0_dev", C.c_void_p), ("u_dev", C.c_void_p),
                ("u_stride_t", C.c_longlong), ("u_stride_n", C.c_longlong), ("y_dev", C.c_void_p),
                ("y_stride_t", C.c_longlong), ("y_stride_n", C.c_longlong), ("q_dev", C.c_void_p),
                ("q_stride_n", C.c_longlong), ("r_dev", C.c_void_p), ("r_stride_n", C.c_longlong),
                ("z_out_dev", C.c_void_p), ("P_out_dev", C.c_void_p), ("x_traj_dev", C.c_void_p),
                ("P_traj_dev", C.c_void_p), ("stride", C.c_longlong), ("loglik_dev", C.c_void_p),
                ("nis_dev", C.c_void_p), ("count_dev", C.c_void_p), ("stats_accumulate", C.c_int32),
                ("reserved", C.c_int32), ("health_dev", C.c_void_p), ("singular_eps", C.c_double)]


class RolloutVjpDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("dt", C.c_double), ("z0_dev", C.c_void_p), ("u_dev", C.c_void_p), ("u_stride_t", C.c_longlong),
                ("u_stride_n", C.c_longlong), ("gtraj_dev", C.c_void_p), ("stride", C.c_longlong),
                ("gzT_dev", C.c_void_p), ("gz0_dev", C.c_void_p), ("gu_dev", C.c_void_p), ("z_out_dev", C.c_void_p),
                ("workspace_dev", C.c_void_p), ("workspace_bytes", C.c_size_t), ("health_dev", C.c_void_p),
                ("singular_eps", C.c_double)]


class RolloutVjpCoefDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("reserved", C.c_int32), ("vjp", RolloutVjpDesc), ("gkp_dev", C.c_void_p)]


class ClosedLoopVjpDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("dt", C.c_double), ("z0_dev", C.c_void_p), ("K_dev", C.c_void_p), ("K_stride_t", C.c_longlong),
                ("K_stride_n", C.c_longlong), ("z_ref_dev", C.c_void_p), ("z_ref_stride_t", C.c_longlong),
                ("z_ref_stride_n", C.c_longlong), ("u_ref_dev", C.c_void_p), ("u_ref_stride_t", C.c_longlong),
                ("u_ref_stride_n", C.c_longlong), ("u_min", C.c_double * 8), ("u_max", C.c_double * 8),
                ("q", C.c_double * 30), ("r", C.c_double * 8), ("gtraj_dev", C.c_void_p), ("stride", C.c_longlong),
                ("gzT_dev", C.c_void_p), ("gcost_dev", C.c_void_p), ("gz0_dev", C.c_void_p), ("gK_dev", C.c_void_p),
                ("gz_ref_dev", C.c_void_p), ("gu_ref_dev", C.c_void_p), ("z_out_dev", C.c_void_p),
                ("workspace_dev", C.c_void_p), ("workspace_bytes", C.c_size_t), ("health_dev", C.c_void_p),
                ("singular_eps", C.c_double)]


class RolloutHostDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("integrator", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("dt", C.c_double), ("x0_host", C.c_void_p), ("xT_host", C.c_void_p), ("u_host", C.c_void_p),
                ("u_shared", C.c_int32), ("reserved", C.c_int32), ("lag_in_host", C.c_void_p),
                ("lag_out_host", C.c_void_p), ("traj_host", C.c_void_p), ("stride", C.c_longlong),
                ("chunk_steps", C.c_longlong), ("lag_in_repr", C.c_int32), ("lag_out_repr", C.c_int32),
                ("gen", InputGen), ("health_host", C.POINTER(C.c_ulonglong)), ("singular_eps", C.c_double)]


class PincWeights(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_hidden_layers", C.c_int32), ("hidden", C.c_int32),
                ("reserved", C.c_int32), ("W", C.c_void_p * 5), ("b", C.c_void_p * 5), ("beta", C.c_float * 4),
                ("ln_w", C.c_void_p * 4), ("ln_b", C.c_void_p * 4)]


class PincRolloutDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("reserved", C.c_int32), ("n", C.c_longlong), ("steps", C.c_longlong),
                ("x0_dev", C.c_void_p), ("u_dev", C.c_void_p), ("u_stride_t", C.c_longlong),
                ("u_stride_n", C.c_longlong), ("lag_in_dev", C.c_void_p), ("lag_out_dev", C.c_void_p),
                ("traj_dev", C.c_void_p), ("stride", C.c_longlong), ("x9T_dev", C.c_void_p)]


class PincSeDesc(C.Structure):
    _fields_ = [("struct_size", C.c_uint32), ("n_horizons", C.c_int32), ("horizons", C.c_int32 * MAX_H),
                ("rows", C.c_longlong), ("n_windows", C.c_longlong), ("X_dev", C.c_void_p), ("U_dev", C.c_void_p),
                ("se_out_dev", C.c_void_p), ("carry_steps", C.c_int32), ("reserved", C.c_int32),
                ("window0", C.c_longlong), ("row0", C.c_longlong), ("carry_lag0_dev", C.c_void_p)]


_DP = C.POINTER(C.c_double)
_PROTOS = {
    "brov_abi_version": (C.c_int, []),
    "brov_last_error": (C.c_char_p, []),
    "brov_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.POINTER(C.c_void_p)]),
    "brov_destroy": (None, [C.c_void_p]),
    "brov_default_physical": (C.c_int, [C.c_double, _DP]),
    "brov_derive_params": (C.c_int, [_DP, _DP]),
    "brov_default_allocation": (C.c_int, [_DP, _DP, _DP]),
    "brov_set_params": (C.c_int, [C.c_void_p, _DP]),
    "brov_get_params": (C.c_int, [C.c_void_p, _DP]),
    "brov_set_allocation": (C.c_int, [C.c_void_p, _DP]),
    "brov_set_di_gains": (C.c_int, [C.c_void_p, _DP, _DP]),
    "brov_set_vehicle_params": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_int]),
    "brov_set_wrench_lag1": (C.c_int, [C.c_void_p, C.c_int]),
    "brov_lag_discretize": (C.c_int, [C.c_double, _DP, _DP]),
    "brov_set_lag_discrete": (C.c_int, [C.c_void_p, C.c_double, _DP, _DP]),
    "brov_rhs": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    "brov_thruster_wrench": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p]),
    "brov_thruster_wrench_series": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "brov_rhs_host": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]),
    "brov_thruster_wrench_host": (C.c_int, [C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p]),
    "brov_rollout": (C.c_int, [C.c_void_p, C.POINTER(RolloutDesc), C.c_void_p]),
    "brov_generate_inputs": (C.c_int, [C.POINTER(GenInputsDesc), C.c_void_p]),
    "brov_step": (C.c_int, [C.c_void_p, C.c_int, C.c_longlong, C.c_void_p, C.c_void_p, C.c_double, C.c_void_p, C.c_void_p, C.c_void_p]),
    "brov_se_workspace_bytes": (C.c_size_t, [C.c_longlong]),
    "brov_multistep_se": (C.c_int, [C.c_void_p, C.POINTER(SeDesc), C.c_void_p]),
    "brov_se_carry_steps": (C.c_int, [C.c_void_p, C.c_double, C.c_int, C.POINTER(C.c_longlong)]),
    "brov_se_sweep_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_longlong, C.c_int]),
    "brov_multistep_se_sweep": (C.c_int, [C.c_void_p, C.POINTER(SeSweepDesc), C.c_void_p]),
    "brov_se_grad_workspace_bytes": (C.c_size_t, [C.c_longlong, C.c_int, C.c_int]),
    "brov_multistep_se_grad": (C.c_int, [C.c_void_p, C.POINTER(SeGradDesc), C.c_void_p]),
    "brov_linearize": (C.c_int, [C.c_void_p, C.POINTER(LinearizeDesc), C.c_void_p]),
    "brov_closed_loop": (C.c_int, [C.c_void_p, C.POINTER(ClosedLoopDesc), C.c_void_p]),
    "brov_ekf": (C.c_int, [C.c_void_p, C.POINTER(EkfDesc), C.c_void_p]),
    "brov_rollout_vjp": (C.c_int, [C.c_void_p, C.POINTER(RolloutVjpDesc), C.c_void_p]),
    "brov_rollout_vjp_workspace_bytes": (C.c_size_t, [C.c_int, C.c_longlong, C.c_longlong]),
    "brov_rollout_vjp_coef": (C.c_int, [C.c_void_p, C.POINTER(RolloutVjpCoefDesc), C.c_void_p]),
    "brov_closed_loop_vjp": (C.c_int, [C.c_void_p, C.POINTER(ClosedLoopVjpDesc), C.c_void_p]),
    "brov_closed_loop_vjp_workspace_bytes": (C.c_size_t, [C.c_int, C.c_longlong, C.c_longlong]),
    "brov_reduced9_rhs": (C.c_int, [C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "brov_koopman_create": (C.c_int, [C.c_int, C.c_int, C.c_int, C.c_int, C.c_double, _DP, _DP, _DP, C.POINTER(C.c_void_p)]),
    "brov_koopman_destroy": (None, [C.c_void_p]),
    "brov_koopman_lift": (C.c_int, [C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p, C.c_void_p]),
    "brov_koopman_multistep_se": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]),
    "brov_koopman_multistep_se_multi": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_int,
                                                 C.POINTER(C.c_int), C.c_void_p, C.c_void_p]),
    "brov_koopman_simulate": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_longlong, C.c_int, C.c_void_p, C.c_void_p]),
    "brov_pinc_create": (C.c_int, [C.c_int, C.POINTER(PincWeights), C.POINTER(C.c_void_p)]),
    "brov_pinc_destroy": (None, [C.c_void_p]),
    "brov_pinc_set_thruster_map": (C.c_int, [C.c_void_p, C.c_double, _DP, _DP, _DP]),
    "brov_pinc_forward": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_longlong, C.c_void_p]),
    "brov_pinc_rollout": (C.c_int, [C.c_void_p, C.POINTER(PincRolloutDesc), C.c_void_p]),
    "brov_pinc_multistep_se": (C.c_int, [C.c_void_p, C.POINTER(PincSeDesc), C.c_void_p]),
    "brov_rollout_host": (C.c_int, [C.c_void_p, C.POINTER(RolloutHostDesc)]),
    "brov_host_alloc": (C.c_int, [C.c_size_t, C.POINTER(C.c_void_p)]),
    "brov_host_free": (C.c_int, [C.c_void_p]),
    "brov_fma_peak": (C.c_int, [C.c_int, C.c_int, C.c_int, _DP, _DP]),
}


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build it with `python -m bluerov2_dynamics_b200.build` (needs nvcc). "
            "bluerov2_dynamics_b200 has no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in _PROTOS.items():
        fn = getattr(lib, name)  # AttributeError if the .so is stale
        fn.restype = res
        fn.argtypes = args
    if lib.brov_abi_version() != ABI_VERSION:
        raise ImportError(f"libbrov.so ABI {lib.brov_abi_version()} != binding ABI {ABI_VERSION}: rebuild")
    return lib


lib = _load()


def check(rc: int) -> None:
    if rc != 0:
        raise BrovError(f"libbrov error {rc}: {lib.brov_last_error().decode(errors='replace')}")


def dptr(a):
    """double* view of a C-contiguous float64 numpy array."""
    return a.ctypes.data_as(_DP)
