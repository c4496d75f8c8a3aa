"""Active-vision wrappers over a batched base env: ``RecordWrapper``, ``FixedFovealEnv``,
``FlexibleFovealEnv``, ``FixedFovealPeripheralEnv`` — same names, constructor signature
``(env, args)``, ``reset`` / ``step`` protocol, Dict action space and ``info`` keys as
``active_gym/fov_env.py`` (citations refer to it), with a leading N axis on every array.

The pixel work of ``_fov_step`` / ``_get_fov_state`` runs on the GPU (``ObservationPath``);
these classes keep only the host-side bookkeeping of the reference.
"""
from __future__ import annotations

from enum import IntEnum
from typing import Optional

import numpy as np
import torch

from . import _lib
from .spaces import Box, Dict, Discrete, Wrapper


class RecordWrapper(Wrapper):
    """fov_env.py:15-105 for N envs, on the device: ``ep_len`` / ``cumulative_reward`` are (N,) CUDA tensors
    updated by ``agym_record_step`` (one launch per step, issued after the fovea update so that the same launch
    appends ``fov_loc`` / ``fov_res`` to the trace); ``info["reward"]`` is the cumulative raw reward and
    ``info["ep_len"]`` the step count of every env.

    ``record=True`` keeps, like the reference's ``record_buffer``, the per-step ``fov_loc`` (``fov_res``) of every
    env that is not done — in a device trace ring of ``args.record_capacity`` calls (default 4096) — and the actions /
    rewards / done flags of the same calls on the host; ``save_record_to_file`` writes one env's last completed
    episode as the reference's ``.pt`` dictionary (fov_env.py:90-102).  The mp4 of rendered frames is not written
    (no renderer on this path): ``"rgb"`` is ``None``."""

    def __init__(self, env, args):
        super().__init__(env)
        self.args = args
        self.record = bool(args.record)
        base = env.unwrapped
        self._path = base.path
        self.num_envs = base.num_envs
        self.host_obs = bool(getattr(base, "host_obs", False))
        self.record_capacity = int(getattr(args, "record_capacity", 4096))
        self.trace = None
        self._calls = 0        # record calls so far (reset or step); call c lives in trace row c % capacity
        self._host_log = None
        if self.record:
            import collections
            self.trace = torch.zeros((self.record_capacity, self.num_envs, 6), dtype=torch.int32, device=self._path.device)
            self._host_log = collections.deque(maxlen=self.record_capacity)
        self._deferred = None
        self._with_res = False
        self._counters_host = None

    # ---- state the reference exposes as attributes
    @property
    def ep_len(self) -> torch.Tensor:
        return self._path.ep_len

    @property
    def cumulative_reward(self) -> torch.Tensor:
        return self._path.cum_reward

    def _commit(self, with_res: bool = False):
        """Issues the deferred counter / trace update (after the wrapper above has moved the fovea, if there is one)."""
        kw, log = self._deferred
        self._deferred = None
        row = None
        if self.record:
            row = self.trace[self._calls % self.record_capacity]
            self._host_log.append(log)
            self._calls += 1
        self._counters_host = self._path.record_step(trace_row=row, with_res=with_res, host_out=self.host_obs, **kw)

    def _add_info(self, info):
        if self.host_obs:   # pinned host copies, valid once the step has been waited for
            info["ep_len"], info["reward"] = self._counters_host[0].numpy(), self._counters_host[1].numpy()
        else:
            info["reward"] = self._path.cum_reward.clone()
            info["ep_len"] = self._path.ep_len.clone()
        return info

    def reset(self, seed=None, options=None, mask=None, return_state=True, defer_record=False):
        state, info = self.env.reset(seed, options, mask=mask, return_state=return_state)
        self._deferred = (dict(reset_mask=mask, is_reset=True), dict(reset=True, mask=None if mask is None else np.array(mask, bool)))
        if not defer_record:
            self._commit()
            info = self._add_info(info)
        return state, info

    def step_async(self, action, after_ingest=None, before_ingest=None, full_action=None):
        """Everything of the step is enqueued here, in stream order: [reward / done upload] -> frames -> ingest ->
        `after_ingest` (the wrapper above moves the fovea and observes) -> counters + trace (fov_env.py:27-46).  Nothing
        is left for ``step_wait`` to enqueue: a second env group's frame copies queued in between would delay it."""
        self._action = action if full_action is None else full_action
        base = self.env.unwrapped

        def before(reward, done):
            self._path.prestage(raw_reward=reward, done=done)
            if before_ingest is not None:
                before_ingest(reward, done)

        def after(reward, done):
            if after_ingest is not None:
                after_ingest(reward, done)
            log = None
            if self.record:
                ret = np.sign(reward) if getattr(base, "clip_reward", False) else reward
                log = dict(action=self._action, return_reward=np.array(ret), raw_reward=np.array(reward), done=np.array(done, bool))
            self._deferred = (dict(raw_reward=reward, done=done, is_reset=False), log)
            self._commit(with_res=self._with_res)

        self.env.step_async(action, after_ingest=after, before_ingest=before)

    def step_wait(self, return_state=True):
        state, return_reward, done, truncated, info = self.env.step_wait(return_state=return_state)
        if self.host_obs:
            self._path.sync()   # the pinned counters are valid once the shard streams are idle
        return state, return_reward, done, truncated, self._add_info(info)

    def step(self, action, return_state=True):
        self.step_async(action)
        return self.step_wait(return_state=return_state)

    def episode_record(self, env_index: int = 0) -> dict:
        """The last COMPLETED episode of one env (what the reference keeps in ``prev_record_buffer`` after the reset
        that follows it), in the reference's record layout."""
        if not self.record:
            raise RuntimeError("record=False: nothing was recorded")
        n_calls = min(self._calls, self.record_capacity)
        first = self._calls - n_calls
        order = [(c % self.record_capacity) for c in range(first, self._calls)]
        self._path.sync()
        tr = self.trace[order, env_index].cpu().numpy()        # (calls, 6) in call order
        logs = list(self._host_log)
        resets = [i for i, lg in enumerate(logs) if lg.get("reset") and (lg["mask"] is None or lg["mask"][env_index])]
        if len(resets) < 2:
            raise RuntimeError("no completed episode in the trace yet (the reference keeps it only after the next reset)")
        i0, i1 = resets[-2], resets[-1]
        rec = {"rgb": None, "state": [], "action": [], "reward": [], "done": [], "truncated": [], "info": [],
               "return_reward": [], "fov_loc": [], "fov_size": tuple(getattr(self.args, "fov_size", ()) or ())}
        if self._with_res:
            rec["fov_res"] = []
        cum, n_states = 0.0, 0
        for i in range(i0, i1):
            lg, t = logs[i], tr[i]
            if t[5]:   # reset entry, or a step that was not done (fov_env.py:72-75, 216-219)
                n_states += 1
                rec["fov_loc"].append(t[0:2].copy())
                if self._with_res:
                    rec["fov_res"].append(t[2:4].copy())
            if lg.get("reset"):
                continue
            a = lg["action"]
            rec["action"].append({k: np.asarray(v.cpu() if isinstance(v, torch.Tensor) else v)[env_index] for k, v in a.items()}
                                 if isinstance(a, dict) else np.asarray(a)[env_index])
            cum += float(np.asarray(lg["raw_reward"])[env_index])
            rec["reward"].append(cum)          # the reference logs the cumulative raw reward (fov_env.py:62-66)
            rec["return_reward"].append(float(np.asarray(lg["return_reward"])[env_index]))
            if n_states > 1:   # fov_env.py:80-85: done / info are kept only once a second state exists
                rec["done"].append(bool(lg["done"][env_index]))
                rec["info"].append({"ep_len": int(t[4]), "fov_loc": t[0:2].copy()})
            rec["truncated"].append(False)
        rec["state"] = [0] * len(rec["reward"])   # fov_env.py:99
        return rec

    def save_record_to_file(self, file_path: str, env_index: int = 0):
        """fov_env.py:90-102 without the video: ``torch.save`` of the episode dictionary."""
        if self.record:
            torch.save(self.episode_record(env_index), file_path)


class FixedFovealEnv(Wrapper):
    """fov_env.py:107-234 for N envs.  Observation: uint8 CUDA tensor (N, K, f_h, f_w), or
    (N, K, S_h, S_w) with ``mask_out`` / ``resize_to_full``; RGB base envs (DMC ``grey=False``) add a channel axis
    after K, (N, K, 3, h, w).

    ``args.fov_memory = M`` (superset, 0..16, default 0 = off; ``mask_out=True`` only): the observation keeps mask_out's
    shape and is the pixelwise max of the mask_out observations of the env's last min(j, M) fovea updates since its last
    reset, missing ones counting as zero frames.  A step and a reset push this step's window; envs a masked ``reset``
    leaves alone push nothing and keep their observation.  The memory follows the fovea's resets only: a life loss inside
    the base env does not clear it.  ``fov_memory_loc`` / ``fov_memory_count`` expose the state.

    ``args.fov_memory_merge`` (superset, ``"max"`` by default) selects how the held windows merge.  ``"paste"`` lays them
    over a zero background from the oldest to the newest, so at each pixel the newest window covering it wins (a bright
    sprite that moved away does not linger over the fresh view of its old place).  The memory, its state and the rules
    above are the same under both; other values raise ``ValueError``."""

    _kind = "fixed"

    def __init__(self, env, args):
        super().__init__(env)
        self.fov_size = tuple(args.fov_size)
        self.fov_init_loc = tuple(args.fov_init_loc)
        assert (np.array(self.fov_size) < np.array(self.obs_size)).all()  # fov_env.py:112
        self.sensory_action_mode = args.sensory_action_mode
        if self.sensory_action_mode == "relative":
            self.sensory_action_space = np.array(args.sensory_action_space)
        elif self.sensory_action_mode == "absolute":
            self.sensory_action_space = np.array(self.obs_size) - np.array(self.fov_size)
        else:
            raise ValueError(self.sensory_action_mode)
        self.resize = bool(getattr(args, "resize_to_full", False))
        self.mask_out = bool(args.mask_out)
        base = self.env.unwrapped
        self.path = base.path
        self.num_envs = base.num_envs
        self.host_obs = bool(getattr(base, "host_obs", False))
        if self.path.fov_size != self.fov_size:
            raise ValueError("the base env was built from different args (fov_size mismatch)")
        self.fov_memory = int(getattr(args, "fov_memory", 0) or 0)
        if not 0 <= self.fov_memory <= 16:
            raise ValueError(f"fov_memory must be within 0..16, got {self.fov_memory}")
        self.fov_memory_merge = getattr(args, "fov_memory_merge", "max")
        if self.fov_memory_merge not in ("max", "paste"):
            raise ValueError(f"fov_memory_merge must be 'max' or 'paste', got {self.fov_memory_merge!r}")
        if self.fov_memory and self._kind == "peripheral":
            if self.fov_memory_merge != "paste":
                raise ValueError("fov_memory on FixedFovealPeripheralEnv needs fov_memory_merge=\"paste\": a max over the "
                                 "blurred backgrounds of past frames is not a useful observation")
            if self.path.pcache is None:
                raise ValueError("fov_memory on FixedFovealPeripheralEnv pastes over the squeeze cache: build the base env "
                                 "with cache_peripheral=True")
        elif self.fov_memory and self._kind != "fixed":
            raise ValueError("fov_memory is defined for FixedFovealEnv and FixedFovealPeripheralEnv only (windows of the "
                             "flexible fovea vary in size)")
        elif self.fov_memory and not self.mask_out:
            raise ValueError("fov_memory merges mask_out observations: it needs mask_out=True")
        if self.fov_memory != getattr(self.path, "fov_memory", 0):
            raise ValueError("the base env was built from different args (fov_memory mismatch)")
        # fov_env.py:125-129 declares Box(low=sas[0], high=sas[1], dtype=int): shape (1,) and, in
        # absolute mode, degenerate.  Kept for compatibility; step() accepts any real (N,2) array.
        self.action_space = Dict({
            "motor_action": self.env.action_space,
            "sensory_action": Box(low=self.sensory_action_space[0], high=self.sensory_action_space[1], dtype=int),
        })
        shape = self.obs_size if (self.mask_out or self.resize) else self.fov_size
        self.observation_space = Box(low=-1., high=1., shape=self._frame_axes() + tuple(shape), dtype=np.float32)
        self._rec = self.env if isinstance(self.env, RecordWrapper) else None
        self._obs = None
        self._host = None
        # args.obs_dtype = torch.float16 / bfloat16 / float32: observations come back NORMALISED, float32(u8) / 255
        # (what the reference returns, atari_env.py:75), written by the observe kernel as a second output next to the
        # u8 tensor (kept in `last_obs_u8`).  Device observations only.
        self.obs_dtype = getattr(args, "obs_dtype", None)
        if self.obs_dtype is not None and self.host_obs:
            raise ValueError("obs_dtype (normalised device observations) and host_obs (pinned u8 host observations) exclude each other")
        self.last_obs_u8 = None
        self._out = None          # set_output(): where the observe kernels store the u8 observations

    def _frame_axes(self):
        """(K,) or, for RGB, (K, 3): the axes in front of the two pixel axes."""
        c = getattr(self.path, "channels", 1)
        return (self.env.frame_stack,) if c == 1 else (self.env.frame_stack, c)

    @property
    def obs_shape(self):
        """Shape of the batched u8 observation tensor, (N, K, h, w) or (N, K, 3, h, w)."""
        return tuple(self.path.out_shape(self._kind, self.variant))

    def set_output(self, out: Optional[torch.Tensor]) -> None:
        """The observe kernels write the u8 observations into ``out`` (``obs_shape``, contiguous) instead of a fresh
        tensor.  ``out`` may live on ANOTHER GPU whose memory this env's device can access as a peer (NVLink): the
        kernels' stores then cross the link themselves, there is no gather copy (``vector.ShardedVecEnv(learner_device=)``)."""
        if out is not None:
            if tuple(out.shape) != self.obs_shape or out.dtype != torch.uint8 or not out.is_contiguous() or not out.is_cuda:
                raise ValueError(f"output must be a contiguous uint8 CUDA tensor of shape {self.obs_shape}")
            if self.host_obs:
                raise ValueError("set_output and host_obs exclude each other")
        self._out = out

    # ---- state the reference exposes as attributes
    @property
    def fov_loc(self) -> torch.Tensor:
        return self.path.loc

    @property
    def variant(self) -> str:
        return "mask" if self.mask_out else ("resize_full" if self.resize else "crop")

    @property
    def fov_memory_loc(self) -> Optional[torch.Tensor]:
        """(N, M, 2) int32: the fov_loc of each memory slot (``fov_memory_count`` of them are held); None without memory."""
        return self.path.mem_loc if self.fov_memory else None

    @property
    def fov_memory_count(self) -> Optional[torch.Tensor]:
        """(N,) int32: entries the memory of each env holds; None without memory."""
        return self.path.mem_state[:, 1] if self.fov_memory else None

    def _norm_buffer(self):
        if self.obs_dtype is None:
            return None
        kind = "peripheral" if self._kind == "peripheral" else self._kind
        return torch.empty(self.path.out_shape(kind, self.variant), dtype=self.obs_dtype, device=self.path.device)

    def _observe_memory(self, action, ctrl, norm_out):
        if self.fov_memory_merge == "paste":
            bg = "periphery" if self._kind == "peripheral" else "zero"
            return self.path.observe_memory_paste(action, ctrl=ctrl, background=bg, out=self._out, host_out=self.host_obs,
                                                  norm_out=norm_out)
        return self.path.observe_fixed_memory(action, ctrl=ctrl, out=self._out, host_out=self.host_obs, norm_out=norm_out)

    def _observe(self, action, ctrl, action_type=None, norm_out=None):
        if self.fov_memory:
            return self._observe_memory(action, ctrl, norm_out)
        return self.path.observe_fixed(action, variant=self.variant, ctrl=ctrl, out=self._out, host_out=self.host_obs, norm_out=norm_out)

    def _run_observe(self, action, ctrl, action_type=None):
        norm = self._norm_buffer()
        r = self._observe(action, ctrl, action_type, norm_out=norm) if norm is not None else self._observe(action, ctrl, action_type)
        if self.host_obs:
            self._obs, self._host = r
        elif norm is not None:
            self.last_obs_u8, self._obs, self._host = r, norm, None
        else:
            self._obs, self._host = r, None

    def _result_obs(self):
        """Device tensor, or (host_obs) the pinned host tensor once the shard streams have finished."""
        if self.host_obs:
            self.path.sync()
            return self._host[0]
        return self._obs

    def _fov_info(self, info):
        info["fov_loc"] = self._host[1].numpy() if self.host_obs else self.path.loc.clone()
        return info

    @staticmethod
    def _ctrl_for_reset(mask, n):
        if mask is None:
            return "reset"
        return np.where(np.asarray(mask, bool), _lib.FOV_RESET, _lib.FOV_KEEP).astype(np.uint8)

    _with_res = False

    def reset(self, mask=None):
        """fov_env.py:156-164 (takes no seed/options, like the reference)."""
        rec = self._rec
        _, info = self.env.reset(mask=mask, return_state=False, **({"defer_record": True} if rec is not None else {}))
        self._run_observe(None, self._ctrl_for_reset(mask, self.num_envs))
        if rec is not None:
            rec._with_res = self._with_res
            rec._commit(with_res=self._with_res)
        obs = self._result_obs()
        if rec is not None:
            info = rec._add_info(info)
        return obs, self._fov_info(info)

    def step_async(self, action):
        """Steps the simulators, then enqueues the action upload, copy + ingest, fovea update + observation and the
        record update; returns at once."""
        self._action = action
        sa, sat = action["sensory_action"], action.get("sensory_action_type")
        rec = self._rec
        kw = {}
        if rec is not None:
            rec._with_res = self._with_res
            kw["full_action"] = action
        self.env.step_async(action["motor_action"],
                            before_ingest=lambda reward, done: self.path.prestage(action=sa, action_type=sat),
                            after_ingest=lambda reward, done: self._run_observe(sa, None, sat), **kw)

    def step_wait(self):
        """fov_env.py:209-221: collects (obs, reward, done, truncated, info) of the step submitted last."""
        _, reward, done, truncated, info = self.env.step_wait(return_state=False)
        obs = self._result_obs()
        self._raise_device_errors()
        return obs, reward, done, truncated, self._fov_info(info)

    def step(self, action):
        """fov_env.py:209-221.  action = {"motor_action": (N,), "sensory_action": (N,2)}."""
        self.step_async(action)
        return self.step_wait()

    def _raise_device_errors(self):
        pass


class FlexibleFovealEnvActionType(IntEnum):  # fov_env.py:236-238
    FOV_LOC = 0
    FOV_RES = 1


class FlexibleFovealEnv(FixedFovealEnv):
    """fov_env.py:240-355 for N envs.  Without mask_out / resize_to_full the reference returns a
    variable-shape (K, rh, rw) crop; the batched form writes it into the top-left corner of a
    zeroed (N, K, S_h, S_w) tensor and reports the shape in ``info["fov_res"]``.

    ``args.resize_to_fov`` (superset, default False): the observation is the glimpse, a fixed-shape (N, K, f_h, f_w)
    tensor — each plane's unblurred window after this step's fovea update, resampled to fov_size by torchvision's
    ``Resize(fov_size)`` (fov_env.py:248,284-285) under the same ``antialias`` switch.  It excludes ``mask_out`` and
    ``resize_to_full``."""

    _kind = "flexible"

    def __init__(self, env, args):
        self.resize_to_fov = bool(getattr(args, "resize_to_fov", False))
        if self.resize_to_fov and (bool(getattr(args, "mask_out", False)) or bool(getattr(args, "resize_to_full", False))):
            raise ValueError("resize_to_fov excludes mask_out and resize_to_full: each selects a different observation")
        super().__init__(env, args)
        self.action_space["sensory_action_type"] = Discrete(len(FlexibleFovealEnvActionType))
        self.fov_init_res = tuple(args.fov_size)
        self.validate_actions = bool(getattr(args, "validate_actions", True))

    @property
    def fov_res(self) -> torch.Tensor:
        return self.path.res

    @property
    def variant(self) -> str:
        return "resize_fov" if self.resize_to_fov else super().variant

    def _check_res(self, action, action_type):
        """The reference raises for a window larger than the frame; do it before the launch
        when the action lives on the host (a device tensor would need a sync)."""
        if not self.validate_actions or action is None or isinstance(action, torch.Tensor):
            return
        a = np.asarray(action, np.float64).reshape(self.num_envs, 2)
        t = np.zeros(self.num_envs, np.int64) if action_type is None else \
            np.asarray(action_type.cpu() if isinstance(action_type, torch.Tensor) else action_type).reshape(-1)
        sel = t == int(FlexibleFovealEnvActionType.FOV_RES)
        if sel.any():
            r = a[sel]
            if (r < 1).any() or (r > np.array(self.obs_size)).any() or (r != np.floor(r)).any():
                raise ValueError("FOV_RES actions must be integer window sizes within [1, obs_size]")

    def _observe(self, action, ctrl, action_type=None, norm_out=None):
        self._check_res(action, action_type)
        self._device_actions = isinstance(action, torch.Tensor) and action.device.type == "cuda"
        return self.path.observe_flexible(action, action_type, variant=self.variant, ctrl=ctrl, out=self._out,
                                          host_out=self.host_obs, norm_out=norm_out)

    def _raise_device_errors(self):
        """FOV_RES actions given as device tensors cannot be validated before the launch; the kernels report what they
        had to clamp / truncate in a device error word.  It is polled without stalling the device pipeline (an
        asynchronous 4-byte copy per step, looked at one step later), so the error surfaces at the latest on the
        step after the offending one."""
        if self.validate_actions and getattr(self, "_device_actions", False):
            bits = self.path.read_errors() if self.host_obs else self.path.poll_errors()
            if bits:
                what = [m for b, m in ((_lib.ERR_RES_RANGE, "outside [1, obs_size]"), (_lib.ERR_RES_FRACTION, "not integral")) if bits & b]
                raise ValueError("FOV_RES actions must be integer window sizes within [1, obs_size] (fov_env.py:322-324 would fail): "
                                 + ", ".join(what) + "; the affected windows were clamped")

    _with_res = True

    def _fov_info(self, info):
        if self.host_obs:
            info["fov_loc"], info["fov_res"] = self._host[1].numpy(), self._host[2].numpy()
        else:
            info["fov_loc"] = self.path.loc.clone()
            info["fov_res"] = self.path.res.clone()
        return info


class FixedFovealPeripheralEnv(FixedFovealEnv):
    """fov_env.py:358-388 for N envs: blurred periphery (squeeze to ``peripheral_res``, expand
    back) with the full-resolution fovea pasted at ``fov_loc``; (N, K, S_h, S_w) uint8.

    ``args.fov_memory = M`` (superset, 1..16) needs ``fov_memory_merge="paste"`` and the squeeze cache
    (``cache_peripheral=True``); either missing raises ``ValueError``.  The observation is then the periphery of the current
    frames with the env's last min(j, M) windows since its last fovea reset pasted over it from the oldest to the newest,
    the newest being this step's fovea; ``args.mask_out`` is ignored, as the reference's constructor forces it off.  Pushes,
    resets, ``fov_memory_loc`` and ``fov_memory_count`` are FixedFovealEnv's."""

    _kind = "peripheral"

    def __init__(self, env, args):
        super().__init__(env, args)
        self.mask_out = False
        self.resize_to_full = True
        self.peripheral_res = tuple(args.peripheral_res)
        self.observation_space = Box(low=-1., high=1., shape=self._frame_axes() + tuple(self.obs_size), dtype=np.float32)
        if self.path.peripheral_res != self.peripheral_res:
            raise ValueError("the base env was built from different args (peripheral_res mismatch)")

    def _observe(self, action, ctrl, action_type=None, norm_out=None):
        if self.fov_memory:
            return self._observe_memory(action, ctrl, norm_out)
        return self.path.observe_peripheral(action, ctrl=ctrl, out=self._out, host_out=self.host_obs, norm_out=norm_out)


class FlexibleFovealPeripheralEnv(FlexibleFovealEnv):
    """Superset (the reference has no such wrapper): ``FlexibleFovealEnv`` whose background is
    ``FixedFovealPeripheralEnv``'s periphery instead of ``mask_out``'s zeros.  Per env, after this step's fovea update
    (fov_env.py:300-330, unchanged, FOV_RES checks included), each plane of the stack is
    ``Resize(obs_size)(Resize(peripheral_res)(full))`` (fov_env.py:366-368, 376) with the window
    ``full[r:r+rh, c:c+rw]`` pasted at its place (fov_env.py:385-386), blurred by ``Resize(fov_res)(Resize(fov_size)(.))``
    iff ``rh > f_h`` (fov_env.py:276-280, 286-287).  Observation: uint8 (N, K, S_h, S_w), or (N, K, 3, S_h, S_w) for RGB;
    ``info`` carries ``fov_loc`` and ``fov_res``; the action space is the flexible one.

    Like the reference's peripheral constructor (fov_env.py:361) it forces ``mask_out = False``.  ``resize_to_fov``
    selects a different observation and raises ``ValueError``, as do a ``peripheral_res`` other than the base env's and
    a base env built with ``cache_peripheral=False`` (the kernels expand the squeeze cache the ingest keeps)."""

    _kind = "flexible_peripheral"

    def __init__(self, env, args):
        if bool(getattr(args, "resize_to_fov", False)):
            raise ValueError("resize_to_fov selects the glimpse; FlexibleFovealPeripheralEnv returns full frames")
        super().__init__(env, args)
        self.mask_out = False
        self.peripheral_res = tuple(args.peripheral_res)
        self.observation_space = Box(low=-1., high=1., shape=self._frame_axes() + tuple(self.obs_size), dtype=np.float32)
        if self.path.peripheral_res != self.peripheral_res:
            raise ValueError("the base env was built from different args (peripheral_res mismatch)")
        if self.path.pcache is None:
            raise ValueError("FlexibleFovealPeripheralEnv needs the squeeze cache: build the base env with cache_peripheral=True")

    @property
    def variant(self) -> str:
        return "mask"   # full frames: the output shape of mask_out

    def _observe(self, action, ctrl, action_type=None, norm_out=None):
        self._check_res(action, action_type)
        self._device_actions = isinstance(action, torch.Tensor) and action.device.type == "cuda"
        return self.path.observe_flexible_peripheral(action, action_type, ctrl=ctrl, out=self._out, host_out=self.host_obs,
                                                     norm_out=norm_out)


class SingleEnvAdapter:
    """The N=1 drop-in: presents a batched env with the reference's single-env types — float64
    NumPy observations normalised to [0,1] (= float32(u8)/255), scalar reward / done, NumPy
    ``fov_loc`` — so code written against the reference runs unchanged."""

    def __init__(self, env):
        assert env.num_envs == 1
        self.env = env
        self.action_space = env.action_space
        self.observation_space = env.observation_space

    def __getattr__(self, name):
        if name.startswith("_") or name == "env":
            raise AttributeError(name)
        return getattr(self.env, name)

    @property
    def fov_loc(self):
        return self.env.path.loc[0].cpu().numpy()

    @property
    def fov_res(self):
        return self.env.path.res[0].cpu().numpy()

    @property
    def unwrapped(self):
        return self.env.unwrapped

    def _obs(self, obs):
        o = obs[0].cpu().numpy()
        if getattr(self.env, "_kind", "") == "flexible" and self.env.variant == "crop":
            rh, rw = self.fov_res
            o = o[..., :rh, :rw]
        return (o.astype(np.float32) / np.float32(255.0)).astype(np.float64)

    @staticmethod
    def _unbatch(info):
        out = {}
        for k, v in info.items():
            if isinstance(v, torch.Tensor):
                v = v.cpu().numpy()
            v = np.asarray(v)
            v = v[0] if v.ndim >= 1 and v.shape[0] == 1 else v
            out[k] = v.item() if isinstance(v, np.ndarray) and v.ndim == 0 else v
        return out

    def reset(self, seed=None, options=None):
        wrapped_fov = isinstance(self.env, FixedFovealEnv)
        obs, info = self.env.reset() if wrapped_fov else self.env.reset(seed, options)
        return self._obs(obs), self._unbatch(info)

    def step(self, action):
        if isinstance(action, dict):
            action = dict(action)
            sa = action["sensory_action"]
            sa = sa.detach().cpu().numpy() if isinstance(sa, torch.Tensor) else np.asarray(sa)
            action["sensory_action"] = sa.reshape(1, 2)
            action["motor_action"] = np.asarray(action["motor_action"]).reshape(1, *np.shape(action["motor_action"]))
            if "sensory_action_type" in action:
                t = action["sensory_action_type"]
                t = t.detach().cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
                action["sensory_action_type"] = t.reshape(-1)[:1].astype(np.int64)
        else:
            action = np.asarray(action).reshape(1, *np.shape(action))
        obs, reward, done, truncated, info = self.env.step(action)
        return (self._obs(obs), np.asarray(reward).reshape(-1)[0].item(), bool(np.asarray(done).reshape(-1)[0]),
                False, self._unbatch(info))

    def train(self):
        self.env.train()

    def eval(self):
        self.env.eval()

    def close(self):
        self.env.close()
