"""ctypes binding of libwalker_b200.so (include/walker_b200.h).  No CPU fallback: a missing library or a
missing CUDA device raises."""
from __future__ import annotations

import ctypes as C
import os
import re

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("WB_LIB_PATH") or os.path.join(_HERE, "lib", "libwalker_b200.so")  # WB_LIB_PATH: A/B builds of the same library
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "walker_b200.h")

WB_OK = 0
STATE_FLOATS = 92
STATE_INTS = 2
OBS = 12
ACT = 4
PAIR_SLOTS = 9
FLAG_TERMINAL = 1 << 5
FLAG_FLOOR_FIRST = 1 << 6


class WalkerB200Error(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"libwalker_b200 status {code}: {message}")
        self.code = code


class Hyperparams(C.Structure):
    """wb_hyperparams (Hyperparameters.cs:83-121)."""
    _fields_ = [("iterations", C.c_int32), ("max_timesteps", C.c_int32), ("batch_size", C.c_int32), ("use_gae", C.c_int32),
                ("normalize_advantages", C.c_int32), ("alpha", C.c_float), ("beta1", C.c_float), ("beta2", C.c_float),
                ("adam_epsilon", C.c_float), ("gamma", C.c_float), ("lambda_", C.c_float), ("epsilon", C.c_float),
                ("log_std", C.c_float)]


class BodyDesc(C.Structure):
    """wb_body_desc: one IObject of a general scene."""
    _fields_ = [("n_vertices", C.c_int32), ("is_static", C.c_int32), ("is_floor", C.c_int32), ("material", C.c_int32),
                ("associated_mask", C.c_uint32), ("accel_x", C.c_float), ("accel_y", C.c_float), ("inverse_inertia", C.c_float)]


class JointDesc(C.Structure):
    """wb_joint_desc: new Joint(bodyA, bodyB, indexA, indexB)."""
    _fields_ = [("body_a", C.c_int32), ("vertex_a", C.c_int32), ("body_b", C.c_int32), ("vertex_b", C.c_int32)]


def declared_symbols() -> list[str]:
    """Every function include/walker_b200.h declares."""
    text = open(HEADER_PATH).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(wb_[a-z0-9_]+)\s*\(", text)))


_lib = None


def lib() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise WalkerB200Error(-1, f"{LIB_PATH} is not built (run `python __graft_entry__.py`); there is no CPU fallback")
    L = C.CDLL(LIB_PATH)
    fp, ip, u8p, vp, i64p = C.POINTER(C.c_float), C.POINTER(C.c_int32), C.POINTER(C.c_uint8), C.c_void_p, C.POINTER(C.c_int64)
    hpp = C.POINTER(Hyperparams)
    sig = {
        "wb_version": (C.c_char_p, []),
        "wb_last_error": (C.c_int32, [C.c_char_p, C.c_size_t]),
        "wb_init": (C.c_int32, [C.c_int32]),
        "wb_hyperparams_default": (C.c_int32, [hpp]),
        "wb_material_register": (C.c_int32, [C.c_float, C.c_float, C.c_float, ip]),
        "wb_material_get": (C.c_int32, [C.c_int32, fp, fp, fp]),
        "wb_env_create": (C.c_int32, [C.c_int32, vp, vp, hpp, C.POINTER(vp)]),
        "wb_env_destroy": (C.c_int32, [vp]),
        "wb_env_count": (C.c_int32, [vp, ip]),
        "wb_env_set_stream": (C.c_int32, [vp, vp]),
        "wb_env_sync": (C.c_int32, [vp]),
        "wb_env_reset": (C.c_int32, [vp, vp, C.c_int32]),
        "wb_env_set_state": (C.c_int32, [vp, vp, vp]),
        "wb_env_get_state": (C.c_int32, [vp, vp, vp]),
        "wb_env_take_actions": (C.c_int32, [vp, vp]),
        "wb_env_step_objects": (C.c_int32, [vp, C.c_float]),
        "wb_env_debug_contacts": (C.c_int32, [vp, C.c_float, vp, vp]),
        "wb_env_observe": (C.c_int32, [vp, vp, vp, vp]),
        "wb_env_get_obs": (C.c_int32, [vp, vp]),
        "wb_env_step": (C.c_int32, [vp, vp, C.c_float, C.c_int32, vp, vp, vp]),
        "wb_env_step_dev": (C.c_int32, [vp, vp, C.c_float, C.c_int32, vp, vp, vp]),
        "wb_env_launch_count": (C.c_int32, [vp, i64p]),
        "wb_host_pin": (C.c_int32, [vp, C.c_size_t]),
        "wb_host_unpin": (C.c_int32, [vp]),
        "wb_env_set_variant": (C.c_int32, [vp, C.c_int32]),
        "wb_env_get_variant": (C.c_int32, [vp, ip]),
        "wb_debug_rotz": (C.c_int32, [C.c_int32, vp, C.c_int32, vp, vp]),
        "wb_scene_create": (C.c_int32, [C.c_int32, C.POINTER(BodyDesc), C.c_int32, vp, C.POINTER(JointDesc), C.c_int32, C.c_int32, C.POINTER(vp)]),
        "wb_scene_destroy": (C.c_int32, [vp]),
        "wb_scene_set_stream": (C.c_int32, [vp, vp]),
        "wb_scene_state_floats": (C.c_int32, [vp, ip]),
        "wb_scene_set_state": (C.c_int32, [vp, vp, vp]),
        "wb_scene_get_state": (C.c_int32, [vp, vp, vp]),
        "wb_scene_set_torques": (C.c_int32, [vp, vp]),
        "wb_scene_step_objects": (C.c_int32, [vp, C.c_float]),
        "wb_terrain_env_create": (C.c_int32, [C.c_int32, C.POINTER(BodyDesc), C.c_int32, vp, C.c_int32, hpp, C.POINTER(vp)]),
        "wb_terrain_env_destroy": (C.c_int32, [vp]),
        "wb_terrain_env_set_stream": (C.c_int32, [vp, vp]),
        "wb_terrain_env_state_floats": (C.c_int32, [vp, ip]),
        "wb_terrain_env_set_terrain": (C.c_int32, [vp, vp]),
        "wb_terrain_env_reset": (C.c_int32, [vp, vp, C.c_int32]),
        "wb_terrain_env_get_state": (C.c_int32, [vp, vp, vp]),
        "wb_terrain_env_set_state": (C.c_int32, [vp, vp, vp]),
        "wb_terrain_env_get_obs": (C.c_int32, [vp, vp]),
        "wb_terrain_env_step": (C.c_int32, [vp, vp, C.c_float, C.c_int32, vp, vp, vp]),
        "wb_terrain_env_step_dev": (C.c_int32, [vp, vp, C.c_float, C.c_int32, vp, vp, vp]),
        "wb_terrain_env_launch_count": (C.c_int32, [vp, i64p]),
        "wb_debug_rcp_sqrt_check": (C.c_int32, [C.c_uint32, C.c_uint64, C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)]),
        "wb_policy_create": (C.c_int32, [C.c_int32, C.c_int32, vp, vp, C.c_int32, vp, vp, C.c_int32, hpp, C.POINTER(vp)]),
        "wb_policy_destroy": (C.c_int32, [vp]),
        "wb_policy_set_stream": (C.c_int32, [vp, vp]),
        "wb_policy_sync": (C.c_int32, [vp]),
        "wb_policy_set_variant": (C.c_int32, [vp, C.c_int32]),
        "wb_policy_set_hyperparams": (C.c_int32, [vp, hpp]),
        "wb_policy_num_params": (C.c_int32, [vp, C.c_int32, ip]),
        "wb_policy_set_weights": (C.c_int32, [vp, C.c_int32, vp]),
        "wb_policy_get_weights": (C.c_int32, [vp, C.c_int32, vp]),
        "wb_policy_get_grads": (C.c_int32, [vp, C.c_int32, vp]),
        "wb_policy_get_adam": (C.c_int32, [vp, C.c_int32, vp, vp, vp]),
        "wb_policy_set_adam": (C.c_int32, [vp, C.c_int32, vp, vp, vp]),
        "wb_policy_forward": (C.c_int32, [vp, C.c_int32, vp, vp, vp]),
        "wb_policy_forward_dev": (C.c_int32, [vp, C.c_int32, vp, vp, vp]),
        "wb_policy_sample": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp]),
        "wb_policy_sample_dev": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp]),
        "wb_policy_sample_philox_dev": (C.c_int32, [vp, C.c_int32, vp, C.c_uint64, C.c_uint64, vp, vp, vp]),
        "wb_policy_act_dev": (C.c_int32, [vp, C.c_int32, vp, C.c_uint64, C.c_uint64, vp, vp, vp, vp]),
        "wb_comm_local_handle": (C.c_int32, [vp, vp]),
        "wb_comm_connect": (C.c_int32, [vp, C.c_int32, C.c_int32, vp]),
        "wb_comm_status": (C.c_int32, [vp, ip, ip]),
        "wb_ppo_grad_allreduce_dev": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp]),
        "wb_ppo_train_dev": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp]),
        "wb_ppo_train_indexed_dev": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp, vp]),
        "wb_ppo_train": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp]),
        "wb_ppo_train_trajectories": (C.c_int32, [vp, C.c_int32, vp, C.c_int32] + [vp] * 10),
        "wb_ppo_train_trajectories_dev": (C.c_int32, [vp, C.c_int32, vp, C.c_int32] + [vp] * 10),
        "wb_segment_returns_dev": (C.c_int32, [vp, C.c_int32, C.c_int32, vp, vp, vp, vp, vp, vp]),
        "wb_normalize_advantages_dev": (C.c_int32, [vp, C.c_int32, C.c_int64, C.c_int64, vp]),
        "wb_normalize_stats_buffer": (C.c_int32, [vp, C.POINTER(vp), ip]),
        "wb_gather_minibatch_dev": (C.c_int32, [vp, C.c_int32] + [vp] * 11),
        "wb_ppo_grad": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp, vp, vp]),
        "wb_ppo_grad_dev": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp]),
        "wb_adam_step": (C.c_int32, [vp]),
        "wb_policy_grad_buffer": (C.c_int32, [vp, C.POINTER(vp), ip]),
        "wb_policy_launch_count": (C.c_int32, [vp, i64p]),
        "wb_returns_advantages": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp]),
        "wb_debug_tc_gemm": (C.c_int32, [C.c_int32] * 6 + [vp, vp, vp]),
        "wb_population_create": (C.c_int32, [C.c_int32, hpp, C.POINTER(vp)]),
        "wb_population_create_net": (C.c_int32, [C.c_int32, C.c_int32, C.c_int32, vp, vp, C.c_int32, vp, vp, C.c_int32, hpp, C.POINTER(vp)]),
        "wb_population_num_params": (C.c_int32, [vp, C.c_int32, ip]),
        "wb_population_destroy": (C.c_int32, [vp]),
        "wb_population_set_stream": (C.c_int32, [vp, vp]),
        "wb_population_sync": (C.c_int32, [vp]),
        "wb_population_launch_count": (C.c_int32, [vp, i64p]),
        "wb_population_set_weights": (C.c_int32, [vp, C.c_int32, vp]),
        "wb_population_get_weights": (C.c_int32, [vp, C.c_int32, vp]),
        "wb_population_get_grads": (C.c_int32, [vp, C.c_int32, vp]),
        "wb_population_get_adam": (C.c_int32, [vp, C.c_int32, vp, vp, vp]),
        "wb_population_sample": (C.c_int32, [vp, C.c_int32, vp, vp, vp, vp, vp]),
        "wb_population_act_dev": (C.c_int32, [vp, C.c_int32, vp, C.c_uint64, C.c_uint64, vp, vp, vp, vp]),
        "wb_population_train_trajectories": (C.c_int32, [vp, C.c_int32, vp, vp, C.c_int32] + [vp] * 10),
        "wb_population_train_dev": (C.c_int32, [vp, C.c_int32, vp, C.c_int32, C.c_int32, C.c_int32, C.c_uint64] + [vp] * 10),
    }
    for name, (res, args) in sig.items():
        fn = getattr(L, name)  # AttributeError here = the library does not export what the header declares
        fn.restype = res
        fn.argtypes = args
    _lib = L
    return L


def last_error() -> str:
    buf = C.create_string_buffer(512)
    lib().wb_last_error(buf, 512)
    return buf.value.decode(errors="replace")


def check(code: int) -> None:
    if code != WB_OK:
        raise WalkerB200Error(code, last_error())


def ptr(a) -> C.c_void_p:
    """numpy array (C-contiguous) / int device pointer / None -> void*."""
    if a is None:
        return C.c_void_p(0)
    if isinstance(a, int):
        return C.c_void_p(a)
    if hasattr(a, "ctypes"):
        assert a.flags["C_CONTIGUOUS"], "array must be C-contiguous"
        return C.c_void_p(a.ctypes.data)
    if hasattr(a, "data_ptr"):  # torch tensor (host pinned or device)
        assert a.is_contiguous()
        return C.c_void_p(a.data_ptr())
    raise TypeError(type(a))
