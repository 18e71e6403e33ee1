"""ctypes binding of libearl_b200.so (the C ABI declared in include/earl_b200.h).

There is no CPU fallback: if the CUDA library is missing this module raises at import of the first
symbol, and every compute entry point fails without a CUDA device.
"""
import ctypes as C
import os

_PKG = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_PKG, "libearl_b200.so")

# mirror of include/earl_b200.h ------------------------------------------------------------------
EARL_ABI_VERSION = 1
ENV_TABLETOP, ENV_SAWYER_DOOR, ENV_SAWYER_PEG, ENV_KITCHEN = 0, 1, 2, 3
FLAG_DENSE_REWARD = 0x01
FLAG_WIDE_INIT = 0x02
FLAG_STATE_F64 = 0x04
FLAG_LIFELONG = 0x08
FLAG_AUTO_RESET = 0x10
FLAG_RESET_AT_GOAL = 0x20
FLAG_EVAL_STATS = 0x40
TABLETOP_MAGIC = 0x54544142


class EarlConfig(C.Structure):
    _fields_ = [("env_kind", C.c_int32), ("num_envs", C.c_int32), ("device", C.c_int32), ("flags", C.c_uint32),
                ("episode_horizon", C.c_int64), ("goal_change_frequency", C.c_int64),
                ("goal_stream_rows", C.c_int32), ("reserved", C.c_int32)]


class TabletopModel(C.Structure):
    _fields_ = [("magic", C.c_uint32), ("num_goals", C.c_int32), ("threshold", C.c_double),
                ("move_distance", C.c_double), ("clip", C.c_double), ("success_radius", C.c_double),
                ("initial_state", C.c_double * 6), ("goal_table", (C.c_double * 6) * 256)]


class Tt3Config(C.Structure):
    """earl_tt3_config (include/earl_tt3_b200.h)"""
    _fields_ = [("num_envs", C.c_int32), ("device", C.c_int32), ("flags", C.c_uint32), ("num_goals", C.c_int32),
                ("episode_horizon", C.c_int64), ("threshold", C.c_double), ("move_distance", C.c_double),
                ("clip", C.c_double), ("success_radius", C.c_double), ("initial_state", C.c_double * 10),
                ("goal_table", (C.c_double * 10) * 16)]


class MjConfig(C.Structure):
    """earl_mj_config (include/earl_mj_b200.h)"""
    _fields_ = [("env_kind", C.c_int32), ("num_envs", C.c_int32), ("device", C.c_int32), ("flags", C.c_uint32),
                ("episode_horizon", C.c_int64), ("goal_change_frequency", C.c_int64)]


class MjTask(C.Structure):
    """earl_mj_task (include/earl_mj_b200.h)"""
    _fields_ = [("frame_skip", C.c_int32), ("hand_site", C.c_int32), ("ree_site", C.c_int32), ("lee_site", C.c_int32),
                ("obj_geom", C.c_int32), ("obj_site", C.c_int32), ("max_newton", C.c_int32), ("obj_qpos_count", C.c_int32),
                ("mocap_low", C.c_float * 3), ("mocap_high", C.c_float * 3), ("action_scale", C.c_float),
                ("success_radius", C.c_float), ("obj_init_pos", C.c_float * 3), ("hand_init_pos", C.c_float * 3),
                ("grasp_site", C.c_int32), ("lpad_site", C.c_int32), ("rpad_site", C.c_int32), ("corner_site", C.c_int32 * 4)]


# (name, restype, argtypes) for EVERY symbol the header declares; tests/test_abi.py checks the list
# against the header text and the built library.
_VP, _I32, _I64, _U32, _SZ = C.c_void_p, C.c_int32, C.c_int64, C.c_uint32, C.c_size_t
SIGNATURES = [
    ("earl_abi_version", C.c_int, []),
    ("earl_last_error", C.c_char_p, []),
    ("earl_tabletop_thresholds", None, [C.c_double, C.c_double, C.POINTER(C.c_double), C.POINTER(C.c_float)]),
    ("earl_create", C.c_int, [C.POINTER(EarlConfig), _VP, _SZ, C.POINTER(_VP)]),
    ("earl_destroy", C.c_int, [_VP]),
    ("earl_num_envs", C.c_int, [_VP]),
    ("earl_obs_dim", C.c_int, [_VP]),
    ("earl_action_dim", C.c_int, [_VP]),
    ("earl_set_goal_stream", C.c_int, [_VP, _VP, _I32]),
    ("earl_reset", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_set_goal", C.c_int, [_VP, _VP, _VP, _VP]),
    ("earl_set_goal_table", C.c_int, [_VP, _VP, _I32, _I32]),
    ("earl_step", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_rollout", C.c_int, [_VP, _VP, _I32, _I32, _VP, _VP, _VP, _VP, _I32, _VP]),
    ("earl_step_host", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_set_host_zerocopy", C.c_int, [_VP, _I32]),
    ("earl_get_obs", C.c_int, [_VP, _VP, _VP]),
    ("earl_compute_reward", C.c_int, [_VP, _VP, _I64, _VP, _VP, _VP]),
    ("earl_counters", C.c_int, [_VP, C.POINTER(_I64), _VP, _VP, _VP, _VP]),
    ("earl_eval_stats", C.c_int, [_VP, _VP, _VP]),
    ("earl_state_nbytes", _SZ, [_VP]),
    ("earl_get_state", C.c_int, [_VP, _VP, _SZ]),
    ("earl_set_state", C.c_int, [_VP, _VP, _SZ]),
    ("earl_launch_count", _I64, [_VP]),
    ("earl_rng_create", _VP, [_I32, _VP, _I32]),
    ("earl_rng_destroy", None, [_VP]),
    ("earl_rng_next_u32", _U32, [_VP]),
    ("earl_rng_py_randbelow", None, [_VP, _U32, _I64, _VP]),
    ("earl_rng_tabletop_goal_rows", None, [_VP, _VP, _U32, _I64, _VP]),
    ("earl_rng_np_randint", None, [_VP, _U32, _I64, _VP]),
    ("earl_rng_np_uniform", None, [_VP, C.c_double, C.c_double, _I64, _VP]),
    ("earl_rng_peg_reset_draws", None, [_VP, _I32, _I32, _I64, _VP, _VP]),
    # include/earl_tt3_b200.h: three-object tabletop
    ("earl_tt3_create", C.c_int, [C.POINTER(Tt3Config), _SZ, C.POINTER(_VP)]),
    ("earl_tt3_destroy", C.c_int, [_VP]),
    ("earl_tt3_reset", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_tt3_set_goal", C.c_int, [_VP, _VP, _VP, _VP]),
    ("earl_tt3_step", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_tt3_rollout", C.c_int, [_VP, _VP, _I32, _I32, _VP, _VP, _VP, _VP, _I32, _VP]),
    ("earl_tt3_step_host", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_tt3_get_obs", C.c_int, [_VP, _VP, _VP]),
    ("earl_tt3_compute_reward", C.c_int, [_VP, _VP, _I64, _VP, _VP, _VP]),
    ("earl_tt3_counters", C.c_int, [_VP, C.POINTER(_I64), _VP, _VP, _VP]),
    ("earl_tt3_get_state", C.c_int, [_VP, _VP, _VP, _VP]),
    ("earl_tt3_set_state", C.c_int, [_VP, _VP, _VP, _VP]),
    ("earl_tt3_launch_count", _I64, [_VP]),
    # include/earl_mj_b200.h
    ("earl_mj_create", C.c_int, [C.POINTER(MjConfig), C.c_char_p, _SZ, C.POINTER(MjTask), C.POINTER(_VP)]),
    ("earl_mj_destroy", C.c_int, [_VP]),
    ("earl_mj_obs_dim", C.c_int, [_VP]),
    ("earl_mj_action_dim", C.c_int, [_VP]),
    ("earl_mj_nq", C.c_int, [_VP]),
    ("earl_mj_nv", C.c_int, [_VP]),
    ("earl_mj_set_goal_table", C.c_int, [_VP, _VP, _I32]),
    ("earl_mj_build_reset_template", C.c_int, [_VP, _VP, _VP, _I32]),
    ("earl_mj_set_reset_stream", C.c_int, [_VP, _VP, _VP, _I32, _VP]),
    ("earl_mj_reset", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_mj_step", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_mj_step_host", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_mj_get_obs", C.c_int, [_VP, _VP, _VP]),
    ("earl_mj_get_state", C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    ("earl_mj_set_state", C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    ("earl_mj_counters", C.c_int, [_VP, C.POINTER(_I64), _VP, _VP, _VP, _VP]),
    ("earl_mj_eval_stats", C.c_int, [_VP, _VP, _VP]),
    ("earl_mj_work_counters", C.c_int, [_VP, _VP]),
    ("earl_mj_launch_count", _I64, [_VP]),
    ("earl_mj_redo_count", _I64, [_VP]),
    # include/earl_mj_kitchen_b200.h: engine-level entry points of the kitchen capacity set
    ("earl_mjk_engine_create", C.c_int, [_VP, _SZ, C.c_int32, C.POINTER(_VP)]),
    ("earl_mjk_engine_destroy", C.c_int, [_VP]),
    ("earl_mjk_engine_nv", C.c_int, [_VP]),
    ("earl_mjk_engine_substeps", C.c_int, [_VP, C.c_int32, C.c_int32, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_mjk_create", C.c_int, [_VP, _VP, _SZ, C.POINTER(_VP)]),
    ("earl_mjk_destroy", C.c_int, [_VP]),
    ("earl_mjk_seed", C.c_int, [_VP, _VP]),
    ("earl_mjk_set_reset_stream", C.c_int, [_VP, _VP, _I32, _VP, _I32]),
    ("earl_mjk_reset", C.c_int, [_VP, _VP, C.c_int32, _VP, _VP, _VP]),
    ("earl_mjk_step", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_mjk_get_state", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_mjk_set_state", C.c_int, [_VP, _VP, _VP, _VP, _VP, _VP]),
    ("earl_mjk_counters", C.c_int, [_VP, C.POINTER(_I64), _VP, _VP, _VP, _VP]),
    ("earl_mjk_work_counters", C.c_int, [_VP, _VP]),
    ("earl_mjk_redo_count", _I64, [_VP]),
]

_lib = None


class EarlError(RuntimeError):
    def __init__(self, code, msg):
        super().__init__(f"libearl_b200 error {code}: {msg}")
        self.code = code


def lib():
    """Load the CUDA library.  Fails loudly when it has not been built (no fallback path exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: build it with `python -m earl_benchmark_b200.build` "
                "(nvcc, sm_100a). earl_benchmark_b200 has no CPU or PyTorch fallback.")
        L = C.CDLL(LIB_PATH)
        for name, res, args in SIGNATURES:
            fn = getattr(L, name)
            fn.restype, fn.argtypes = res, args
        if L.earl_abi_version() != EARL_ABI_VERSION:
            raise ImportError(f"{LIB_PATH}: ABI version {L.earl_abi_version()} != {EARL_ABI_VERSION}; rebuild")
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise EarlError(rc, lib().earl_last_error().decode("utf-8", "replace"))
