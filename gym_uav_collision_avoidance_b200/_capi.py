"""ctypes binding of the C-ABI (include/uavca.h).  The library is the product: if it is missing or cannot be
loaded this module raises — there is no CPU or PyTorch fallback."""
from __future__ import annotations

import ctypes as C
import os

from .build import LIB_PATH

KIND_MULTI, KIND_SINGLE = 0, 1
ACTION_CARTESIAN, ACTION_POLAR, ACTION_SCALED = 0, 1, 2
RESET_ON_DONE0, RESET_ON_ALL_DONE, RESET_ON_ANY_DONE = 1, 2, 4
SOURCE_PHILOX, SOURCE_POOL = 0, 1
FLAG_PARKED, FLAG_COLLIDED = 1, 2
OBS_DIM = {KIND_MULTI: 10, KIND_SINGLE: 4}
MAX_AGENTS = 1024


class Config(C.Structure):
    """`uavca_config` (include/uavca.h) — constructor kwargs of the reference worlds
    (multi_uav_world_2d.py:13-28, uav_world_2d.py:14-26) plus episode control."""

    _fields_ = [
        ("kind", C.c_int32),
        ("num_envs", C.c_int32),
        ("num_agents", C.c_int32),
        ("reset_mode", C.c_int32),
        ("max_episode_steps", C.c_int32),
        ("reset_source", C.c_int32),
        ("circular", C.c_int32),
        ("single_f32_first_step", C.c_int32),
        ("env_index_base", C.c_int64),
        ("seed", C.c_uint64),
        ("x_size", C.c_double),
        ("y_size", C.c_double),
        ("max_speed", C.c_double),
        ("max_acceleration", C.c_double),
        ("tau", C.c_double),
        ("collider_radius", C.c_double),
        ("hard_collision_radius", C.c_double),
        ("d_sense", C.c_double),
        ("reach_distance", C.c_double),
        ("reach_speed", C.c_double),
        ("polar_scale", C.c_double),
        ("track_scores", C.c_int32),
        ("reserved0", C.c_int32),
    ]


class Layout(C.Structure):
    """`uavca_layout`: byte offsets of the SoA fields inside a state blob."""

    _fields_ = [(n, C.c_size_t) for n in
                ("total_bytes", "stats", "pos", "vel", "tgt", "init", "prev", "flags", "steps", "reach", "coll", "episode", "score", "pos64", "tgt64", "init64", "prev64")]


# every symbol include/uavca.h declares: name -> (restype, argtypes)
_VP = C.c_void_p
SYMBOLS = {
    "uavca_last_error": (C.c_char_p, []),
    "uavca_version": (C.c_int, []),
    "uavca_default_config": (C.c_int, [C.c_int, C.POINTER(Config)]),
    "uavca_create": (C.c_int, [C.POINTER(Config), C.c_int, C.POINTER(_VP)]),
    "uavca_destroy": (C.c_int, [_VP]),
    "uavca_get_config": (C.c_int, [_VP, C.POINTER(Config)]),
    "uavca_state_layout": (C.c_int, [_VP, C.POINTER(Layout)]),
    "uavca_set_reset_pool": (C.c_int, [_VP, _VP, C.c_int32]),
    "uavca_pool_layout": (C.c_int, [_VP, C.c_int32, C.POINTER(Layout)]),
    "uavca_reset": (C.c_int, [_VP, _VP, _VP, _VP, _VP]),
    "uavca_observe": (C.c_int, [_VP, _VP, _VP, _VP]),
    "uavca_step_multi": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP]),
    "uavca_step_single": (C.c_int, [_VP, _VP, _VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "uavca_step_f64": (C.c_int, [_VP, _VP, _VP, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "uavca_step_sync": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_int, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "uavca_map_action": (C.c_int, [_VP, _VP, C.c_int, _VP, _VP]),
    "uavca_stats": (C.c_int, [_VP, _VP, _VP, _VP]),
    "uavca_step_host": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_int, _VP, _VP, _VP, _VP]),
    "uavca_rollout": (C.c_int, [_VP, _VP, C.c_int32, _VP, C.c_int, C.c_int, C.c_uint64, C.c_uint64, _VP, _VP, _VP, _VP, _VP,
                                _VP, _VP, _VP]),
    "uavca_sample_actions": (C.c_int, [_VP, C.c_uint64, C.c_uint64, _VP, _VP]),
    "uavca_step_multi_replay": (C.c_int, [_VP, _VP, _VP, C.c_int, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP,
                                           _VP, C.c_int64, _VP, _VP]),
    "uavca_replay_sample": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int64, C.c_int32, C.c_int32, _VP, C.c_int64, C.c_uint64,
                                      C.c_uint64, C.c_int, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "uavca_replay_sample_nstep": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int64, C.c_int32, C.c_int32, _VP, C.c_int64,
                                            C.c_uint64, C.c_uint64, C.c_int, C.c_int64, C.c_int32, C.c_double, _VP, _VP, _VP,
                                            _VP, _VP, _VP, _VP]),
    "uavca_replay_push_dev": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int64, C.c_int32, C.c_int32, _VP, _VP, _VP, _VP, _VP,
                                        C.c_int64, _VP, _VP]),
    "uavca_replay_push": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int64, C.c_int32, C.c_int32, _VP, _VP, _VP, _VP, _VP,
                                    C.c_int64, C.c_int64, _VP]),
    "uavca_per_sync": (C.c_int, [_VP, C.c_int64, _VP, _VP, C.c_int64, _VP]),
    "uavca_per_update": (C.c_int, [_VP, C.c_int64, C.c_int64, _VP, _VP, _VP, C.c_int64, _VP]),
    "uavca_per_sample": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int64, C.c_int32, C.c_int32, _VP, _VP, C.c_int64, C.c_int64,
                                   C.c_double, C.c_uint64, C.c_uint64, _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "uavca_per_sample_nstep": (C.c_int, [_VP, _VP, _VP, _VP, _VP, C.c_int64, C.c_int32, C.c_int32, _VP, _VP, C.c_int64,
                                         C.c_int64, C.c_double, C.c_int64, C.c_int32, C.c_double, C.c_uint64, C.c_uint64,
                                         _VP, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "uavca_policy_act": (C.c_int, [_VP, C.c_int64, _VP, _VP, _VP, _VP, _VP, _VP, C.c_uint64, C.c_uint64, _VP, _VP, _VP, _VP]),
    "uavca_launch_count": (C.c_int64, [_VP]),
}


class UavcaError(RuntimeError):
    pass


_lib = None


def load() -> C.CDLL:
    """Load gym_uav_collision_avoidance_b200/libuavca.so (built by build.py / __graft_entry__.build())."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("UAVCA_LIB") or LIB_PATH  # override: kernel-variant experiments only
    if path == LIB_PATH and not os.path.exists(path):
        # a fresh checkout (built artefacts are git-ignored): compile the product once, loudly, or fail below
        try:
            from . import build as _build

            _build.build()
        except Exception as exc:  # nvcc missing / compile error: no fallback of any kind
            raise UavcaError(f"{path} is missing and could not be built ({exc}).  This package has no CPU fallback.") from exc
    if not os.path.exists(path):
        raise UavcaError(
            f"{path} is missing: build the CUDA extension first (python -m gym_uav_collision_avoidance_b200.build "
            "or __graft_entry__.build()).  This package has no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def last_error() -> str:
    return (load().uavca_last_error() or b"").decode()


def check(rc: int, what: str) -> None:
    if rc != 0:
        raise UavcaError(f"{what} failed (code {rc}): {last_error()}")


def default_config(kind: int) -> Config:
    cfg = Config()
    check(load().uavca_default_config(kind, C.byref(cfg)), "uavca_default_config")
    return cfg
