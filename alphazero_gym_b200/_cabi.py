"""ctypes binding of libazg.so (include/azg.h).  No torch types cross this boundary: pointers, sizes, ints.

The library is built in-tree by `alphazero_gym_b200/build.py` (nvcc, sm_100a).  There is no CPU fallback:
if the shared library is missing, import of the engine fails with a clear error.
"""
from __future__ import annotations

import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("AZG_LIB_PATH") or os.path.join(HERE, "lib", "libazg.so")  # override: kernel experiments only

AZG_OK, AZG_EINVAL, AZG_ECUDA, AZG_ETERMINAL, AZG_ENAN, AZG_ECAPACITY = 0, -1, -2, -3, -4, -5
AZG_EWRAP = -6  # Acrobot-v1: an angle reached the wrap loop's cap (include/azg.h)
DISCRETE, CONTINUOUS = 0, 1
ACT_RELU, ACT_ELU, ACT_LEAKYRELU, ACT_RELU6, ACT_SILU, ACT_HARDSWISH = 0, 1, 2, 3, 4, 5
# nonlinearity strings of config/policy/*.yaml (alphazero/network/utils.py:5-14) and torch module names -> AZG_ACT_*
ACT_BY_NAME = {"relu": 0, "elu": 1, "leakyrelu": 2, "relu6": 3, "swish": 4, "silu": 4, "hardswish": 5}
VT = {"off_policy": 0, "on_policy": 1, "greedy": 2}
FLAG_NO_GRAPH = 1
FLAG_EVAL_Q8 = 2
FLAG_FUSED = 4
FLAG_RNG_MT19937 = 8
FLAG_ENV_MOUNTAIN_CAR_CONTINUOUS = 16
FLAG_ENV_MOUNTAIN_CAR = 32
FLAG_ENV_ACROBOT = 64

EXPORTS = [
    "azg_create", "azg_destroy", "azg_last_error", "azg_version", "azg_num_weights", "azg_set_weights",
    "azg_search_discrete", "azg_search_continuous", "azg_cmax", "azg_root_results", "azg_search_host", "azg_status",
    "azg_rows", "azg_set_tapes", "azg_dump_tree_discrete", "azg_dump_tree_continuous", "azg_get_counters",
    "azg_head_dim", "azg_mlp_forward", "azg_env_step", "azg_profile_search", "azg_set_seed", "azg_selfplay_seed",
    "azg_selfplay_step", "azg_fused_stats", "azg_search_host_begin", "azg_search_host_end", "azg_set_reward_model",
]


class AzgConfig(C.Structure):
    _fields_ = [
        ("variant", C.c_int32), ("max_rollouts", C.c_int32), ("max_trees", C.c_int32), ("num_actions", C.c_int32),
        ("num_components", C.c_int32), ("state_dim", C.c_int32), ("hidden", C.c_int32), ("n_hidden", C.c_int32),
        ("activation", C.c_int32), ("v_target", C.c_int32), ("puct_f32", C.c_int32), ("device", C.c_int32),
        ("c_uct", C.c_double), ("gamma", C.c_double), ("epsilon", C.c_double), ("c_pw", C.c_double), ("kappa", C.c_double),
        ("action_bound", C.c_float), ("log_std_min", C.c_float), ("log_std_max", C.c_float),
        ("flags", C.c_uint32), ("seed", C.c_uint64),
    ]


class DumpDiscrete(C.Structure):
    FIELDS = ("n_nodes", "parent", "paction", "node_n", "terminal", "V", "r", "state", "prior", "eW", "en", "echild")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


class DumpContinuous(C.Structure):
    FIELDS = ("n_rows", "parent", "action", "eW", "en", "expanded", "node_n", "terminal", "V", "r", "state", "head")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


class SelfPlayIO(C.Structure):
    FIELDS = ("d_env_state", "d_ep_step", "d_episode", "d_root_n", "d_obs", "d_actions", "d_counts", "d_Q", "d_V_target",
              "d_n_children", "d_action_taken", "d_reward", "d_done")
    _fields_ = [(n, C.c_void_p) for n in FIELDS]


class AzgError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"azg error {code}: {msg}")
        self.code = code


_lib = None


def load():
    """dlopen libazg.so and declare every prototype of include/azg.h."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} is missing: build the CUDA engine with `python -m alphazero_gym_b200.build` "
            "(needs nvcc).  alphazero_gym_b200 has no CPU fallback.")
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.azg_create.restype, L.azg_create.argtypes = C.c_int, [C.POINTER(AzgConfig), C.POINTER(vp)]
    L.azg_destroy.restype, L.azg_destroy.argtypes = None, [vp]
    L.azg_last_error.restype, L.azg_last_error.argtypes = C.c_char_p, []
    L.azg_version.restype, L.azg_version.argtypes = C.c_char_p, []
    L.azg_num_weights.restype, L.azg_num_weights.argtypes = i64, [vp]
    L.azg_set_weights.restype, L.azg_set_weights.argtypes = C.c_int, [vp, vp, i64, vp]
    L.azg_search_discrete.restype, L.azg_search_discrete.argtypes = C.c_int, [vp, i32, vp, vp, i32, i64, vp]
    L.azg_search_continuous.restype, L.azg_search_continuous.argtypes = C.c_int, [vp, i32, vp, i32, i64, vp]
    L.azg_cmax.restype, L.azg_cmax.argtypes = i32, [vp]
    L.azg_root_results.restype, L.azg_root_results.argtypes = C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp]
    L.azg_search_host.restype = C.c_int
    L.azg_search_host.argtypes = [vp, i32, vp, vp, i32, i64, vp, vp, vp, vp, vp]
    L.azg_search_host_begin.restype = C.c_int
    L.azg_search_host_begin.argtypes = [vp, i32, i32, vp, vp, i32, i64, vp, vp, vp, vp, vp]
    L.azg_search_host_end.restype, L.azg_search_host_end.argtypes = C.c_int, [vp, i32]
    L.azg_status.restype, L.azg_status.argtypes = C.c_int, [vp, vp]
    L.azg_rows.restype, L.azg_rows.argtypes = i32, [vp]
    L.azg_set_tapes.restype, L.azg_set_tapes.argtypes = C.c_int, [vp, vp, vp, vp]
    L.azg_dump_tree_discrete.restype, L.azg_dump_tree_discrete.argtypes = C.c_int, [vp, i32, C.POINTER(DumpDiscrete)]
    L.azg_dump_tree_continuous.restype, L.azg_dump_tree_continuous.argtypes = C.c_int, [vp, i32, C.POINTER(DumpContinuous)]
    L.azg_get_counters.restype, L.azg_get_counters.argtypes = C.c_int, [vp, i32, C.POINTER(i64 * 8)]
    L.azg_fused_stats.restype, L.azg_fused_stats.argtypes = C.c_int, [vp, C.POINTER(i64 * 8)]
    L.azg_profile_search.restype = C.c_int
    L.azg_profile_search.argtypes = [vp, i32, vp, vp, i32, i64, vp, C.POINTER(C.c_float * 3), C.POINTER(i32 * 3)]
    L.azg_head_dim.restype, L.azg_head_dim.argtypes = i32, [vp]
    L.azg_mlp_forward.restype, L.azg_mlp_forward.argtypes = C.c_int, [vp, i32, vp, vp, vp, vp]
    L.azg_env_step.restype, L.azg_env_step.argtypes = C.c_int, [vp, i32, vp, vp, vp, vp, vp, vp, vp]
    L.azg_set_seed.restype, L.azg_set_seed.argtypes = C.c_int, [vp, C.c_uint64, vp]
    L.azg_set_reward_model.restype, L.azg_set_reward_model.argtypes = C.c_int, [vp, C.c_double, C.c_double]
    L.azg_selfplay_seed.restype, L.azg_selfplay_seed.argtypes = C.c_uint64, [C.c_uint64, i64]
    L.azg_selfplay_step.restype = C.c_int
    L.azg_selfplay_step.argtypes = [vp, i32, C.POINTER(SelfPlayIO), i32, i64, i64, C.c_uint64, i32, i32, i32, C.c_double, vp]
    _lib = L
    return L


def check(rc: int) -> None:
    if rc != AZG_OK:
        msg = load().azg_last_error().decode()
        if rc == AZG_ETERMINAL:
            raise ValueError("Can't do tree search from a terminal node")
        raise AzgError(rc, msg)
