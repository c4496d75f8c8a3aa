"""active_gym_b200 — B200-native batched implementation of Active-Gym's active-perception
observation path (frame-skip max-pool, grayscale + resize, frame-stack ring, foveal crop,
peripheral view, merge) behind the reference's gymnasium-style API.

Public names mirror ``active_gym/__init__.py:3-9,10-16,58-64`` of the reference; every factory
takes an extra ``num_envs`` (batched, uint8 CUDA observations) and defaults to the single-env
drop-in that returns the reference's types.
"""
from .engine import LUMA_DMC, LUMA_RGB, ObservationPath  # noqa: F401
from .pipeline import PipelinedPath  # noqa: F401
from .vector import FovealVectorEnv, ShardedVecEnv  # noqa: F401
from .atari_env import (  # noqa: F401
    AtariBaseEnv, AtariEnvArgs, AtariFixedFovealEnv, AtariFixedFovealPeripheralEnv, AtariFlexibleFovealEnv,
    AtariFlexibleFovealPeripheralEnv, AtariVecEnv,
)
from .dmc_env import (  # noqa: F401
    DMCBaseEnv, DMCEnvArgs, DMCFixedFovealEnv, DMCFixedFovealPeripheralEnv, DMCFlexibleFovealEnv,
    DMCFlexibleFovealPeripheralEnv, DMCVecEnv,
)
from .fov_env import (  # noqa: F401
    FixedFovealEnv, FixedFovealPeripheralEnv, FlexibleFovealEnv, FlexibleFovealEnvActionType,
    FlexibleFovealPeripheralEnv, RecordWrapper, SingleEnvAdapter,
)

__all__ = [
    "AtariBaseEnv", "AtariFixedFovealEnv", "AtariFlexibleFovealEnv", "AtariFixedFovealPeripheralEnv", "AtariEnvArgs",
    "DMCBaseEnv", "DMCFixedFovealEnv", "DMCFlexibleFovealEnv", "DMCFixedFovealPeripheralEnv", "DMCEnvArgs",
    "RecordWrapper", "FixedFovealEnv", "FlexibleFovealEnv", "FlexibleFovealEnvActionType", "FixedFovealPeripheralEnv",
    "AtariVecEnv", "DMCVecEnv", "SingleEnvAdapter", "ObservationPath", "PipelinedPath", "FovealVectorEnv", "ShardedVecEnv",
    "LUMA_RGB", "LUMA_DMC",
    # supersets of the reference
    "AtariFlexibleFovealPeripheralEnv", "DMCFlexibleFovealPeripheralEnv", "FlexibleFovealPeripheralEnv",
]
