"""Atari base env: ``AtariEnvArgs``, the batched ``AtariVecEnv`` and the factory functions.

Mirrors ``active_gym/atari_env.py`` of the reference (file:line citations refer to it).  The
simulator part (ALE stepping, no-op / fire reset, episodic life) lives in a host-side frame
source (``sources.ALEPool``); everything from the raw screen to the stacked observation runs
on the GPU through ``ObservationPath``.
"""
from __future__ import annotations

from typing import Optional, Tuple

import numpy as np
import torch

from . import _lib
from .engine import LUMA_RGB
from .pipeline import PipelinedPath
from .spaces import Box, Discrete, Env


class AtariEnvArgs:
    """Source-compatible with atari_env.py:25-39; adds defaults for the attributes the reference's
    wrappers require but do not default (README quick-start raises AttributeError without them)."""

    def __init__(self, game, seed, obs_size: Tuple[int, int], **kwargs):
        self.env_backend = "atari_py"
        self.device = None
        self.seed = seed
        self.max_episode_length = 108e3
        self.game = game
        self.frame_stack = 4
        self.action_repeat = 4
        self.obs_size = obs_size
        self.mask_out = False
        self.record = False
        self.clip_reward = False
        self.resize_to_full = False  # superset: no default in the reference (fov_env.py:120)
        # superset: FlexibleFovealEnv returns the glimpse, the window resampled to fov_size (N, K, f_h, f_w)
        self.resize_to_fov = False
        # superset: FixedFovealEnv with mask_out merges the last fov_memory (0..16; 0 = off) observations by pixelwise max
        self.fov_memory = 0
        # superset: how the memory merges its windows — "max" (pixelwise max of the mask_out observations) or "paste"
        # (the windows laid oldest to newest over the background: zeros, or the periphery of FixedFovealPeripheralEnv)
        self.fov_memory_merge = "max"
        for k, v in kwargs.items():
            self.__setattr__(k, v)


def _path_from_args(args, num_envs, obs_size, raw_shape, luma, device, host_source: bool, channels: int = 1) -> PipelinedPath:
    """The per-GPU engine of an env batch.  ``args.shards`` (default: 2 for host frame sources, whose copies should
    overlap the kernels and the copies back; 1 for device-resident sources) cuts the batch into env-index shards with
    their own streams (pipeline.PipelinedPath).  Few, large copies win: a process has 8 hardware work queues by
    default (CUDA_DEVICE_MAX_CONNECTIONS), and streams beyond that alias onto the same queue and serialise each
    other's copies (B200, 16,384 envs, two env groups: 1-2 shards 18.8-19.2 ms per step against a pure-copy floor of
    17.1 ms; 8 shards 22.3 ms)."""
    fov = getattr(args, "fov_size", None)
    shards = getattr(args, "shards", None)
    if shards is None:
        shards = 2 if host_source and num_envs >= 64 else 1
    return PipelinedPath(
        num_envs, args.frame_stack, obs_size, raw_shape, shards=shards, luma=luma,
        fov_size=tuple(fov) if fov is not None else None,
        fov_init_loc=getattr(args, "fov_init_loc", (0, 0)),
        sensory_action_mode=getattr(args, "sensory_action_mode", "absolute"),
        sensory_action_space=getattr(args, "sensory_action_space", (0.0, 0.0)),
        peripheral_res=getattr(args, "peripheral_res", None), device=device,
        cache_peripheral=getattr(args, "cache_peripheral", True), side_streams=host_source,
        antialias=bool(getattr(args, "antialias", True)), **({"channels": channels} if channels != 1 else {}),
        **({"fov_memory": int(args.fov_memory)} if getattr(args, "fov_memory", 0) else {}))


class _VecBase(Env):
    """What AtariVecEnv and DMCVecEnv share: the frame source below, the pipelined engine, and the asynchronous
    protocol ``step_async`` / ``step_wait`` (``step`` = both), which lets a caller run two env groups
    alternately — the simulators of one group step on the host while the other group's frames are copied and
    transformed on the GPU (SURVEY.md §8f row 1)."""

    def _init_engine(self, args, num_envs, source, luma, device, channels: int = 1):
        self.args = args
        self.num_envs = int(num_envs)
        self.frame_stack = args.frame_stack
        self.action_repeat = args.action_repeat
        self.obs_size = tuple(args.obs_size)
        if getattr(args, "cv2_dsize_quirk", False):
            # atari_env.py:74 hands obs_size = (h, w) to cv2.resize as dsize = (width, height): a non-square obs_size
            # comes out transposed, (w, h), in the reference.  Off by default (obs_size means (h, w) here).
            self.obs_size = self.obs_size[::-1]
        self.clip_reward = args.clip_reward
        self.source = source
        host_source = not hasattr(source, "device")
        self.path = _path_from_args(args, self.num_envs, self.obs_size, tuple(source.raw_shape), luma,
                                    device or getattr(args, "device", None), host_source, channels)
        self.device = self.path.device
        self.host_obs = bool(getattr(args, "host_obs", False))
        if host_source and hasattr(source, "set_used_rows") and self.path.run is not None:
            source.set_used_rows(self.path.used_rows)   # only the sampled raw rows cross PCIe, as one block per shard
        # RGB: (K, 3, H, W) as dmc_env.py:122 declares
        frame_axes = (self.frame_stack,) if channels == 1 else (self.frame_stack, channels)
        self.observation_space = Box(low=-1., high=1., shape=frame_axes + self.obs_size, dtype=np.float32)
        self._pending = None
        # args.async_sim: step_async hands the simulator stepping (host CPU) + the enqueueing of copies and kernels to a
        # worker thread and returns at once; step_wait joins it.  The caller's thread is free while the simulators run
        # (SURVEY.md section 8f row 1: sim step t+1 overlaps whatever the caller does with the result of step t).
        self.async_sim = bool(getattr(args, "async_sim", False))
        self._future = None
        self._pool = None
        if self.async_sim:
            from concurrent.futures import ThreadPoolExecutor
            self._pool = ThreadPoolExecutor(max_workers=1, thread_name_prefix="agym-step")

    def _submit(self, job):
        """Runs `job` (simulators + enqueue) now, or on the step thread when async_sim is set."""
        if self._pool is None:
            self._pending = job()
            return

        def run():
            if self.device.type == "cuda":
                with torch.cuda.device(self.device):   # the current device is per thread
                    return job()
            return job()
        self._future = self._pool.submit(run)

    def _collect(self):
        if self._future is not None:
            self._pending, self._future = self._future.result(), None
        r, self._pending = self._pending, None
        return r

    def _frames_enqueued(self):
        """Tells the source that the copies reading its current staging set are in the streams."""
        if hasattr(self.source, "frames_consumed"):
            self.source.frames_consumed(self.path.record_events())

    def step(self, action, return_state=True):
        self.step_async(action)
        return self.step_wait(return_state=return_state)

    def close(self):
        if self._future is not None:
            self._future.result()
        if self._pool is not None:
            self._pool.shutdown(wait=True)
            self._pool = None
        if hasattr(self.source, "close"):
            self.source.close()

    def render(self, mode="rgb_array", obs_size=None):
        raise NotImplementedError("recording/rendering is outside the observation hot path (SURVEY.md §2 row 2)")


class AtariVecEnv(_VecBase):
    """N Atari environments; observation = (N, K, S_h, S_w) uint8 CUDA tensor.

    Replaces AtariEnv (atari_env.py:41-172) for a batch.  ``source`` supplies the simulators
    (default ``ALEPool`` when atari_py is importable).  The reference returns normalised
    float64 = float32(u8)/255; values are identical after that conversion.
    """

    def __init__(self, args, num_envs: int = 1, source=None, device=None):
        self.training = True
        if source is None:
            from .sources import ALEPool
            source = ALEPool(args, int(num_envs), workers=getattr(args, "sim_workers", 1))
        self._init_engine(args, num_envs, source, getattr(args, "luma", LUMA_RGB), device)
        self.action_space = Discrete(source.n_actions)
        self.reward_range = (-float("inf"), float("inf"))

    def _info(self, raw_reward):
        return {"raw_reward": raw_reward}  # atari_env.py:77-78

    def _ingest(self, fa, fb, flags):
        self.path.ingest_atari(fa, fb, flags, packed=bool(getattr(self.source, "packed_rows", False)))
        self._frames_enqueued()

    def reset(self, seed=None, options=None, mask=None, return_state=True):
        """atari_env.py:84-117.  ``mask`` (N,) bool selects the envs to reset (default: all)."""
        fa, fb, flags = self.source.reset(mask)
        self._ingest(fa, fb, flags)
        state = self.path.stack() if return_state else None
        return state, self._info(np.zeros(self.num_envs))

    def step_async(self, action, after_ingest=None, before_ingest=None):
        """atari_env.py:119-133: steps the simulators (host), calls `before_ingest(reward, done)` (the wrappers upload
        their small host arrays ahead of the frames), enqueues copy + ingest, then `after_ingest(reward, done)` (the
        wrappers' observe / record launches: they must follow the ingest in stream order)."""
        def job():
            fa, fb, flags, reward, done = self.source.step(action)
            if before_ingest is not None:
                before_ingest(reward, done)
            self._ingest(fa, fb, flags)
            if after_ingest is not None:
                after_ingest(reward, done)
            return reward, done
        self._submit(job)

    def step_wait(self, return_state=True):
        """atari_env.py:134-148."""
        reward, done = self._collect()
        state = self.path.stack() if return_state else None
        return_reward = np.sign(reward) if self.clip_reward else reward
        truncated = np.zeros(self.num_envs, bool)
        return state, return_reward, done, truncated, self._info(reward)

    def train(self):  # atari_env.py:158-159
        self.training = True
        if hasattr(self.source, "training"):
            self.source.training = True

    def eval(self):  # atari_env.py:162-163
        self.training = False
        if hasattr(self.source, "training"):
            self.source.training = False


# ---- factories: atari_env.py:174-192, batched.  num_envs=1 + as_reference=True gives the single-env
# drop-in whose reset()/step() return reference-typed values (see fov_env.SingleEnvAdapter).
def AtariBaseEnv(args, num_envs: Optional[int] = None, source=None, device=None):
    from .fov_env import RecordWrapper, SingleEnvAdapter
    env = RecordWrapper(AtariVecEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def AtariFixedFovealEnv(args, num_envs: Optional[int] = None, source=None, device=None):
    from .fov_env import FixedFovealEnv, SingleEnvAdapter
    env = FixedFovealEnv(AtariBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def AtariFlexibleFovealEnv(args, num_envs: Optional[int] = None, source=None, device=None):
    from .fov_env import FlexibleFovealEnv, SingleEnvAdapter
    env = FlexibleFovealEnv(AtariBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def AtariFixedFovealPeripheralEnv(args, num_envs: Optional[int] = None, source=None, device=None):
    from .fov_env import FixedFovealPeripheralEnv, SingleEnvAdapter
    env = FixedFovealPeripheralEnv(AtariBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env


def AtariFlexibleFovealPeripheralEnv(args, num_envs: Optional[int] = None, source=None, device=None):
    """Superset: the flexible fovea over the peripheral background (fov_env.FlexibleFovealPeripheralEnv)."""
    from .fov_env import FlexibleFovealPeripheralEnv, SingleEnvAdapter
    env = FlexibleFovealPeripheralEnv(AtariBaseEnv(args, num_envs or 1, source, device), args)
    return SingleEnvAdapter(env) if num_envs is None else env
