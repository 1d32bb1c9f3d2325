"""gym_uav_collision_avoidance_b200 — B200-native batched environment step of
dazchi/gym-uav-collision-avoidance (UAVWorld2D / MultiUAVWorld2D), hand-written sm_100a CUDA behind a C-ABI."""
from ._capi import (ACTION_CARTESIAN, ACTION_POLAR, ACTION_SCALED, FLAG_COLLIDED, FLAG_PARKED, KIND_MULTI, KIND_SINGLE,
                    RESET_ON_ALL_DONE, RESET_ON_ANY_DONE, RESET_ON_DONE0, SOURCE_PHILOX, SOURCE_POOL, UavcaError)
from .batched import BatchedMultiUAVWorld2D, BatchedUAVWorld2D, Box, StateBlob
from .replay import DeviceReplay, PrioritizedDeviceReplay
from .rollout import BatchedRollout, FusedGaussianPolicy, GaussianPolicy

__all__ = [
    "BatchedMultiUAVWorld2D", "BatchedUAVWorld2D", "Box", "StateBlob", "UavcaError", "DeviceReplay", "PrioritizedDeviceReplay",
    "BatchedRollout", "GaussianPolicy", "FusedGaussianPolicy",
    "ACTION_CARTESIAN", "ACTION_POLAR", "ACTION_SCALED", "FLAG_PARKED", "FLAG_COLLIDED", "KIND_MULTI", "KIND_SINGLE",
    "RESET_ON_DONE0", "RESET_ON_ALL_DONE", "RESET_ON_ANY_DONE", "SOURCE_PHILOX", "SOURCE_POOL",
]
