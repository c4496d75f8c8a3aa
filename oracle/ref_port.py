"""TEST / BASELINE INFRASTRUCTURE — the reference's per-environment CPU path, restated.

``bench.py`` times this module as the CPU baseline (``cpu_baseline.kind = "port"`` and the
``--impl reference`` arm) wherever there is no checkout of the reference (see oracle/ref_harness.py),
whose own files are then not importable.  This port performs, per environment and
per step, the same library calls in the same order and dtypes as the reference does —
``cv2.resize(INTER_LINEAR)``, ``astype(float32)/255``, a float64 two-frame max, a
``deque`` + ``np.stack`` frame stack, ``np.rint(np.clip())`` for the fovea location, NumPy
slicing for the crop and ``torchvision.transforms.Resize`` for every resample — so that its
cost per step is the reference's cost per step (simulator time excluded: frames are inputs).

It is pinned like the C oracle: tests/test_ref_port_golden.py replays tests/golden/*.npz
(outputs of the unmodified reference) through it and requires identical values.

Reference lines: atari_env.py:73-75,80-82,111-114,121-133,143; dmc_env.py:175-183,193-195,
228-230; fov_env.py:149-150,166-203,270-330,375-388.
"""
from __future__ import annotations

from collections import deque

import numpy as np


class RefPortEnv:
    """One environment's observation pipeline (base env buffer + one foveal wrapper)."""

    def __init__(self, kind="atari", wrapper="fixed", frame_stack=4, obs_size=(84, 84), fov_size=(30, 30),
                 fov_init_loc=(0, 0), mode="absolute", lo=-10.0, hi=10.0, variant="crop", peripheral_res=None):
        import cv2
        import torch
        from torchvision.transforms import Resize
        self.cv2, self.torch, self.Resize = cv2, torch, Resize
        self.kind, self.wrapper, self.variant, self.mode = kind, wrapper, variant, mode
        self.K, self.obs_size, self.fov_size = frame_stack, tuple(obs_size), tuple(fov_size)
        self.init_loc, self.sas = fov_init_loc, (lo, hi)
        self.buf = deque([], maxlen=frame_stack)
        self.to_full = Resize(self.obs_size) if variant == "resize_full" else None
        self.to_fov = Resize(self.fov_size)
        if peripheral_res:
            self.squeeze_expand = torch.nn.Sequential(Resize(tuple(peripheral_res)), Resize(self.obs_size))
        self.loc = np.zeros(2, np.int32)
        self.res = np.array(self.fov_size, np.int32)

    # ---- base env ---------------------------------------------------------------
    def _gray_state(self, screen):
        s = self.cv2.resize(screen, self.obs_size, interpolation=self.cv2.INTER_LINEAR)
        return s.astype(np.float32) / 255.

    def _dmc_state(self, rgb):
        return self.cv2.cvtColor(rgb, self.cv2.COLOR_BGR2GRAY).astype(np.float32) / 255.

    def push_reset(self, frame, hard):
        if hard:
            for _ in range(self.K):
                self.buf.append(np.zeros(self.obs_size))
        self.buf.append(self._dmc_state(frame) if self.kind == "dmc" else self._gray_state(frame))
        return np.stack(self.buf, axis=0)

    def push_step(self, fa, fb, flags=3):
        if self.kind == "dmc":
            self.buf.append(self._dmc_state(fa))
        else:
            two = np.zeros((2, *self.obs_size))
            if flags & 1:
                two[0] = self._gray_state(fa)
            if flags & 2:
                two[1] = self._gray_state(fb)
            self.buf.append(two.max(0))
        return np.stack(self.buf, axis=0)

    # ---- foveal wrappers ------------------------------------------------------------
    def reset_fov(self):
        self.loc = np.rint(np.array(self.init_loc, copy=True)).astype(np.int32)
        self.res = np.rint(np.array(self.fov_size, copy=True)).astype(np.int32)

    def _clip_loc(self, loc):
        win = self.res if self.wrapper == "flexible" else np.array(self.fov_size)
        return np.rint(np.clip(loc, 0, np.array(self.obs_size) - win)).astype(int)

    def move(self, action, atype=0):
        action = np.asarray(action)
        if self.wrapper == "flexible" and atype == 1:
            self.res = action.copy()
            self.loc = self._clip_loc(self.loc)
        elif self.mode == "absolute":
            self.loc = self._clip_loc(action)
        else:
            d = np.rint(np.clip(action, *self.sas)).astype(int)
            self.loc = self._clip_loc(self.loc + d)

    def view(self, full):
        t = self.torch
        r, c = int(self.loc[0]), int(self.loc[1])
        if self.wrapper == "peripheral":
            fh, fw = self.fov_size
            fov = full[..., r:r + fh, c:c + fw]
            out = self.squeeze_expand(t.from_numpy(full)).numpy()
            out[..., r:r + fh, c:c + fw] = fov
            return out
        if self.wrapper == "flexible":
            rh, rw = int(self.res[0]), int(self.res[1])
            fov = full[..., r:r + rh, c:c + rw]
            if rh > self.fov_size[0]:
                fov = self.Resize((rh, rw))(self.to_fov(t.from_numpy(fov))).numpy()
        else:
            rh, rw = self.fov_size
            fov = full[..., r:r + rh, c:c + rw]
        if self.variant == "mask":
            m = np.zeros_like(full)
            m[..., r:r + rh, c:c + rw] = fov
            return m
        if self.variant == "resize_full":
            return self.to_full(t.from_numpy(fov)).numpy()
        return fov

    def step(self, fa, fb, action, atype=0, flags=3):
        full = self.push_step(fa, fb, flags)
        self.move(action, atype)
        return self.view(full)

    def reset(self, frame, hard=True):
        full = self.push_reset(frame, hard)
        self.reset_fov()
        return self.view(full)
