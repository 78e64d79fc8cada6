"""ctypes binding of libmpcb200.so (include/mpc_b200.h).  Thin by design: structs, prototypes,
error translation.  There is no fallback: a missing library or device raises."""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libmpcb200.so")

ABI_VERSION = 2
MAX_OBSTACLES = 16
N_REF = 85

STATUS_CONVERGED = 0
STATUS_MAX_ITER = 1
STATUS_LINESEARCH_FAIL = 2
STATUS_NAN = 4
STATUS_INFEASIBLE_START = 8
STATUS_STALLED = 16
STATUS_KINK = 32
MAX_STARTS = 8

ERR_BAD_ARG, ERR_NO_DEVICE, ERR_CUDA, ERR_TOO_LARGE = -1, -2, -3, -4

_f = C.POINTER(C.c_float)
_i = C.POINTER(C.c_int32)
_b = C.POINTER(C.c_uint8)


class MpcConfig(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("horizon", C.c_int32), ("vehicles_count", C.c_int32), ("dt", C.c_float),
                ("weight_speed", C.c_float), ("weight_control", C.c_float), ("weight_input_diff", C.c_float),
                ("weight_distance", C.c_float), ("weight_collision", C.c_float), ("collision_check", C.c_int32),
                ("literal_no_collision", C.c_int32), ("max_iter", C.c_int32), ("tol_step", C.c_float),
                ("reg_min", C.c_float), ("threads_per_block", C.c_int32), ("blocks_per_sm", C.c_int32),
                ("n_starts", C.c_int32)]


class MpcProblemBatch(C.Structure):
    _fields_ = [("s0", C.c_void_p), ("ego_index", C.c_void_p), ("w_speed", C.c_void_p), ("w_control", C.c_void_p),
                ("w_diff", C.c_void_p), ("vr_a", C.c_void_p), ("vr_slope", C.c_void_p), ("vr_b", C.c_void_p),
                ("vr_n", C.c_void_p), ("is_collide", C.c_void_p), ("n_obs", C.c_void_p), ("obstacles", C.c_void_p)]


class MpcSolveOut(C.Structure):
    _fields_ = [("actions", C.c_void_p), ("status", C.c_void_p), ("iters", C.c_void_p), ("cost", C.c_void_p),
                ("U", C.c_void_p)]


class MpcLatchState(C.Structure):
    _fields_ = [("collision_memory", C.c_void_p), ("memo_conflict", C.c_void_p), ("is_collide", C.c_void_p)]


class MpcCollisionOut(C.Structure):
    _fields_ = [("agent_collide", C.c_void_p), ("conflict_index", C.c_void_p), ("is_collide", C.c_void_p),
                ("ego_index", C.c_void_p), ("stop_index", C.c_void_p), ("degenerate", C.c_void_p),
                ("conflict_point", C.c_void_p)]


class MpcEnvStep(C.Structure):
    _fields_ = [("ego", C.c_void_p), ("others", C.c_void_p), ("t", C.c_void_p), ("crashed_state", C.c_void_p),
                ("counter", C.c_void_p), ("action", C.c_void_p), ("obs", C.c_void_p), ("terminal_obs", C.c_void_p),
                ("reward", C.c_void_p), ("done", C.c_void_p), ("crashed", C.c_void_p), ("arrived", C.c_void_p),
                ("truncated", C.c_void_p), ("speed", C.c_void_p), ("B", C.c_int32), ("n_others", C.c_int32),
                ("substeps", C.c_int32), ("duration_steps", C.c_int32), ("raw_action", C.c_int32), ("dt_sim", C.c_float),
                ("arrive_x", C.c_float), ("arrive_y", C.c_float)]


EXPORTS = ["mpc_create", "mpc_destroy", "mpc_last_error", "mpc_workspace_batch", "mpc_rollout_cost", "mpc_solve",
           "mpc_prepare", "mpc_predict", "mpc_predict_host", "mpc_launch_count", "mpc_fp32_peak", "mpc_timing_begin",
           "mpc_timing_end", "mpc_device_info", "mpc_set_warm_start", "mpc_set_adaptive_starts", "mpc_solve_config",
           "mpc_env_step"]


class MpcError(RuntimeError):
    def __init__(self, code: int, text: str):
        super().__init__(f"libmpcb200 error {code}: {text}")
        self.code = code


_lib = None


def load() -> C.CDLL:
    """Loads the in-tree library.  Raises if it has not been built (python mpc-rl_for_avs_b200/build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: build it with `python mpc-rl_for_avs_b200/build.py` "
                          f"(nvcc, sm_100a).  There is no CPU implementation of the MPC path.")
    lib = C.CDLL(LIB_PATH)
    vp = C.c_void_p
    lib.mpc_create.argtypes = [C.POINTER(MpcConfig), C.c_int, C.c_int, C.POINTER(vp)]
    lib.mpc_create.restype = C.c_int
    lib.mpc_destroy.argtypes = [vp]
    lib.mpc_destroy.restype = C.c_int
    lib.mpc_last_error.argtypes = [vp]
    lib.mpc_last_error.restype = C.c_char_p
    lib.mpc_workspace_batch.argtypes = [vp, C.POINTER(MpcProblemBatch)]
    lib.mpc_workspace_batch.restype = C.c_int
    lib.mpc_rollout_cost.argtypes = [vp, C.POINTER(MpcProblemBatch), C.c_int, vp, vp, vp, vp, vp]
    lib.mpc_rollout_cost.restype = C.c_int
    lib.mpc_solve.argtypes = [vp, C.POINTER(MpcProblemBatch), C.c_int, C.POINTER(MpcSolveOut), vp]
    lib.mpc_solve.restype = C.c_int
    lib.mpc_prepare.argtypes = [vp, vp, vp, vp, vp, C.POINTER(MpcLatchState), C.c_int, C.POINTER(MpcCollisionOut), vp]
    lib.mpc_prepare.restype = C.c_int
    lib.mpc_predict.argtypes = [vp, vp, vp, vp, vp, C.POINTER(MpcLatchState), C.c_int, C.POINTER(MpcSolveOut),
                                C.POINTER(MpcCollisionOut), vp]
    lib.mpc_predict.restype = C.c_int
    lib.mpc_predict_host.argtypes = [vp, vp, vp, vp, vp, C.c_int, vp, vp, vp, C.POINTER(MpcCollisionOut), C.POINTER(C.c_int64),
                                     C.POINTER(C.c_int64)]
    lib.mpc_predict_host.restype = C.c_int
    lib.mpc_set_warm_start.argtypes = [vp, vp]
    lib.mpc_set_warm_start.restype = C.c_int
    lib.mpc_set_adaptive_starts.argtypes = [vp, C.c_int, C.c_float, vp, vp]
    lib.mpc_set_adaptive_starts.restype = C.c_int
    lib.mpc_launch_count.argtypes = [vp]
    lib.mpc_launch_count.restype = C.c_int64
    lib.mpc_fp32_peak.argtypes = [vp, C.c_int, C.POINTER(C.c_float)]
    lib.mpc_fp32_peak.restype = C.c_int
    lib.mpc_timing_begin.argtypes = [vp]
    lib.mpc_timing_begin.restype = C.c_int
    lib.mpc_timing_end.argtypes = [vp, C.POINTER(C.c_float), C.POINTER(C.c_float), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.mpc_timing_end.restype = C.c_int
    lib.mpc_solve_config.argtypes = [vp, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.mpc_solve_config.restype = C.c_int
    lib.mpc_env_step.argtypes = [C.POINTER(MpcEnvStep), vp]
    lib.mpc_env_step.restype = C.c_int
    lib.mpc_device_info.argtypes = [vp, C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int), C.POINTER(C.c_int)]
    lib.mpc_device_info.restype = C.c_int
    _lib = lib
    return lib


def check(lib, handle, rc: int) -> None:
    if rc != 0:
        text = lib.mpc_last_error(handle)
        raise MpcError(rc, text.decode() if text else "")
