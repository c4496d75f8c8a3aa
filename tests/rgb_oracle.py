"""TEST INFRASTRUCTURE — the RGB (DMC ``grey=False``) observation path restated by composition of the pinned grey
oracles, with no new arithmetic.

Why composition is exact: cv2's BGR2GRAY weights sum to 2^15 (3735 + 19235 + 9798), so the luma of a pixel (v, v, v)
is v.  Channel c of an RGB frame therefore goes through the grey DMC ingest unchanged when fed as the frame whose
three channels all equal channel c.  Every wrapper operation acts on the last two axes with one fov_loc / fov_res per
env, so the observation of the plane stack is the observation of each plane.

* ``ingest_dmc_rgb``: the grey C oracle once per channel on channel-replicated frames, interleaved into the
  ``[N][K*C]`` plane ring with the plane-head rule of ``include/agym_b200.h`` (head = C*slot + C-1);
* ``RefPortRGBEnv``: ``oracle/ref_port.RefPortEnv`` with the reference's declared RGB observation (dmc_env.py:122):
  the render transposed to CHW, ``float32 / 255``, stacked to (K, 3, H, W); ``view`` runs unchanged.
"""
from __future__ import annotations

import numpy as np

from oracle import agym_oracle as orc
from oracle.ref_port import RefPortEnv

C = 3


def new_state(n, K, obs_size):
    """Fresh plane ring (n, K*C, h, w) and head = K*C - 1: the first push lands in planes 0 .. C-1."""
    return np.zeros((n, K * C) + tuple(obs_size), np.uint8), np.full((n,), K * C - 1, np.int32)


def replicate(frames, c):
    """The frames whose three channels all equal channel c of ``frames`` (..., H, W, 3)."""
    return np.ascontiguousarray(np.repeat(frames[..., c:c + 1], 3, axis=-1))


def ingest_dmc_rgb(f, flags, ring, head):
    n, P, sh, sw = ring.shape
    K = P // C
    planes = ring.reshape(n, K, C, sh, sw)   # a view: written through below
    new_head = None
    for c in range(C):
        grey = np.ascontiguousarray(planes[:, :, c])
        h = (head // C).astype(np.int32)
        orc.ingest_dmc(replicate(f, c), flags, grey, h)
        planes[:, :, c] = grey
        new_head = h
    head[:] = C * new_head + C - 1


def stack(ring, head):
    n, P, sh, sw = ring.shape
    return orc.stack(ring, head).reshape(n, P // C, C, sh, sw)


def _frames(out, n, K):
    return out.reshape((n, K, C) + out.shape[2:])


# use_f32: resample in float32, as torchvision does on the reference's float32 stacks (DMC frames once the float64 zero
# frames of a hard reset are evicted, dmc_env.py:183,195)
def observe_fixed(ring, head, loc, fov_size, variant="crop", use_f32=False):
    return _frames(orc.observe_fixed(ring, head, loc, fov_size, variant=variant, use_f32=use_f32), ring.shape[0],
                   ring.shape[1] // C)


def observe_peripheral(ring, head, loc, fov_size, peripheral_res, use_f32=False):
    return _frames(orc.observe_peripheral(ring, head, loc, fov_size, peripheral_res, use_f32=use_f32), ring.shape[0],
                   ring.shape[1] // C)


def observe_flexible(ring, head, loc, res, fov_size, variant="mask", pad=None, use_f32=False):
    return _frames(orc.observe_flexible(ring, head, loc, res, fov_size, variant=variant, pad=pad, use_f32=use_f32),
                   ring.shape[0], ring.shape[1] // C)


class RefPortRGBEnv(RefPortEnv):
    """``kind="dmc_rgb"``: one DMC environment with ``grey=False``."""

    def __init__(self, **kw):
        super().__init__(kind="dmc", **kw)
        self.kind = "dmc_rgb"

    def _dmc_state(self, rgb):
        return rgb.transpose(2, 0, 1).astype(np.float32) / 255.

    def push_reset(self, frame, hard):
        if hard:
            for _ in range(self.K):
                self.buf.append(np.zeros((C,) + self.obs_size))
        self.buf.append(self._dmc_state(frame))
        return np.stack(self.buf, axis=0)

    def push_step(self, fa, fb, flags=3):
        self.buf.append(self._dmc_state(fa))
        return np.stack(self.buf, axis=0)
