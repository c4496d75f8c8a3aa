"""DeepMind-Control base env: ``DMCEnvArgs``, the batched ``DMCVecEnv`` and the factories.

Mirrors the pixel branch of ``active_gym/dmc_env.py`` (citations refer to it).  MuJoCo
physics and rendering stay on the host (``sources.DMCPool``); luma (``grey=True``) or the
channel split (``grey=False``) + frame stack + the foveal wrappers run on the GPU.
``from_pixels=False`` is outside the hot path and raises.

``grey=False`` observations have the layout the reference declares, ``(K, 3, H, W)`` (dmc_env.py:122;
its stacking at :230 is of HWC frames, inconsistent with that declaration): oldest frame first, each frame
the render's channels in render order (RGB), unconverted.  The foveal wrappers act on the last two axes of
every one of the 3K planes with one fov_loc / fov_res per env, as fov_env.py's slicing and Resize do on any
array with leading axes.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np

from .atari_env import _VecBase
from .engine import LUMA_DMC
from .spaces import Box


class DMCEnvArgs:
    """Source-compatible with dmc_env.py:56-76 (+ ``resize_to_full``, ``resize_to_fov`` and ``fov_memory`` defaults, see AtariEnvArgs)."""

    def __init__(self, domain_name: str, task_name: str, seed: int, obs_size: Tuple[int, int], **kwargs):
        self.env_backend = "dmc"
        self.seed = seed
        self.domain_name = domain_name
        self.task_name = task_name
        self.obs_size = obs_size
        self.task_kwargs = {}
        self.visualize_reward = False
        self.from_pixels = True
        self.grey = True
        self.camera_id = 0
        self.action_repeat = 4
        self.frame_stack = 3
        self.mask_out = False
        self.environment_kwargs = {}
        self.clip_reward = False
        self.record = False
        self.resize_to_full = False
        self.resize_to_fov = False
        self.fov_memory = 0
        for k, v in kwargs.items():
            self.__setattr__(k, v)


class DMCVecEnv(_VecBase):
    """N DMC environments; observation = (N, K, S_h, S_w) uint8 CUDA tensor, or (N, K, 3, S_h, S_w) with
    ``grey=False`` (dmc_env.py:78-253)."""

    def __init__(self, args, num_envs: int = 1, source=None, device=None):
        if not args.from_pixels:
            raise NotImplementedError("only the from_pixels=True branch is on the observation hot path")
        if source is None:
            from .sources import DMCPool
            source = DMCPool(args, int(num_envs), workers=getattr(args, "sim_workers", 1))
        # dmc_env.py:182 applies COLOR_BGR2GRAY to an RGB render: channel 0 gets the blue weight
        self._init_engine(args, num_envs, source, LUMA_DMC, device, channels=1 if args.grey else 3)
        self._true_low, self._true_high = source.true_low, source.true_high
        self.action_space = Box(low=-1.0, high=1.0, shape=self._true_low.shape, dtype=np.float32)  # dmc_env.py:110-115

    @property
    def reward_range(self):
        return 0, self.action_repeat

    def _info(self, raw_reward):  # dmc_env.py:188-191
        info = self.source.extra_info() if hasattr(self.source, "extra_info") else {}
        info["raw_reward"] = raw_reward
        return info

    def reset(self, seed=None, options=None, mask=None, return_state=True):
        """dmc_env.py:197-209."""
        frames, flags = self.source.reset(mask)
        self.path.ingest_dmc(frames, flags)
        self._frames_enqueued()
        state = self.path.stack() if return_state else None
        return state, self._info(np.zeros(self.num_envs))

    def step_async(self, action, after_ingest=None, before_ingest=None):
        """dmc_env.py:211-226: steps the simulators (host), `before_ingest(reward, done)`, enqueues copy + ingest, then
        `after_ingest(reward, done)` (see AtariVecEnv.step_async)."""
        action = np.asarray(action, np.float32).reshape(self.num_envs, -1)
        assert (action >= -1.0).all() and (action <= 1.0).all()  # dmc_env.py:212

        def job():
            frames, flags, reward, done = self.source.step(action)
            if before_ingest is not None:
                before_ingest(reward, done)
            self.path.ingest_dmc(frames, flags)
            self._frames_enqueued()
            if after_ingest is not None:
                after_ingest(reward, done)
            return reward, done
        self._submit(job)

    def step_wait(self, return_state=True):
        """dmc_env.py:227-234."""
        reward, done = self._collect()
        state = self.path.stack() if return_state else None
        return_reward = np.sign(reward) if self.clip_reward else reward
        return state, return_reward, done, np.zeros(self.num_envs, bool), self._info(reward)

    def train(self):
        pass

    def eval(self):
        pass


def DMCBaseEnv(args, num_envs: Optional[int] = None, source=None, device=None):  # dmc_env.py:255-258
    from .fov_env import RecordWrapper, SingleEnvAdapter
    env = RecordWrapper(DMCVecEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def DMCFixedFovealEnv(args, num_envs: Optional[int] = None, source=None, device=None):  # :260-263
    from .fov_env import FixedFovealEnv, SingleEnvAdapter
    env = FixedFovealEnv(DMCBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def DMCFlexibleFovealEnv(args, num_envs: Optional[int] = None, source=None, device=None):  # :265-268
    from .fov_env import FlexibleFovealEnv, SingleEnvAdapter
    env = FlexibleFovealEnv(DMCBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def DMCFixedFovealPeripheralEnv(args, num_envs: Optional[int] = None, source=None, device=None):  # :270-273
    from .fov_env import FixedFovealPeripheralEnv, SingleEnvAdapter
    env = FixedFovealPeripheralEnv(DMCBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def DMCFlexibleFovealPeripheralEnv(args, num_envs: Optional[int] = None, source=None, device=None):
    """Superset: the flexible fovea over the peripheral background (fov_env.FlexibleFovealPeripheralEnv)."""
    from .fov_env import FlexibleFovealPeripheralEnv, SingleEnvAdapter
    env = FlexibleFovealPeripheralEnv(DMCBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env
