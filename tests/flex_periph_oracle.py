"""TEST INFRASTRUCTURE — the flexible fovea over the peripheral background, restated by composition with no new
arithmetic.

Per env and plane, after this step's fovea update (fov_env.py:300-330):
  1. ``bg = Resize(obs_size)(Resize(peripheral_res)(plane))`` (fov_env.py:366-368, 376): ``orc.aa_resize`` twice;
  2. the window ``plane[r:r+rh, c:c+rw]``, blurred by ``Resize(fov_res)(Resize(fov_size)(win))`` iff ``rh > f_h``
     (fov_env.py:276-280, 286-287): the window of ``orc.observe_flexible(..., variant="mask")``;
  3. ``bg[r:r+rh, c:c+rw] = win`` (fov_env.py:385-386 at the flexible window).
Planes are indexed oldest -> newest from ``head + 1`` (``tests/glimpse_oracle.py``); RGB rings hold K * 3 planes and
every plane is treated alike.

``RefPortFlexPeriphEnv`` restates steps 1-3 on the reference port (``oracle/ref_port.py``) with its torchvision calls.
"""
from __future__ import annotations

import numpy as np

from oracle import agym_oracle as orc
from oracle.ref_port import RefPortEnv


def observe_flexible_peripheral(ring, head, loc, res, fov_size, peripheral_res, use_f32=False):
    """``ring`` u8 (n, P, S_h, S_w), ``head`` (n,), ``loc`` / ``res`` int (n, 2) -> float64 (n, P, S_h, S_w) in u8 units."""
    n, P, S_h, S_w = ring.shape
    win = orc.observe_flexible(ring, head, np.ascontiguousarray(loc, np.int32), np.ascontiguousarray(res, np.int32),
                               fov_size, "mask", use_f32=use_f32)
    out = np.empty((n, P, S_h, S_w), np.float64)
    for e in range(n):
        r, c = int(loc[e][0]), int(loc[e][1])
        rh, rw = int(res[e][0]), int(res[e][1])
        for k in range(P):
            plane = ring[e, (int(head[e]) + 1 + k) % P].astype(np.float64)
            bg = orc.aa_resize(orc.aa_resize(plane, tuple(peripheral_res), use_f32=use_f32), (S_h, S_w), use_f32=use_f32)
            bg[r:r + rh, c:c + rw] = win[e, k, r:r + rh, c:c + rw]
            out[e, k] = bg
    return out


class RefPortFlexPeriphEnv(RefPortEnv):
    """The port's flexible wrapper with the peripheral wrapper's background (steps 1-3 above).  ``antialias`` selects
    the torchvision ``Resize`` mode of every resample."""

    def __init__(self, peripheral_res, antialias=True, **kw):
        super().__init__(wrapper="flexible", variant="mask", peripheral_res=peripheral_res, **kw)
        self.antialias = bool(antialias)
        self.to_fov = self.Resize(self.fov_size, antialias=self.antialias)
        self.squeeze_expand = self.torch.nn.Sequential(self.Resize(tuple(peripheral_res), antialias=self.antialias),
                                                       self.Resize(self.obs_size, antialias=self.antialias))

    def view(self, full):
        t = self.torch
        r, c = int(self.loc[0]), int(self.loc[1])
        rh, rw = int(self.res[0]), int(self.res[1])
        fov = full[..., r:r + rh, c:c + rw]
        if rh > self.fov_size[0]:   # fov_env.py:286: rows only
            fov = self.Resize((rh, rw), antialias=self.antialias)(self.to_fov(t.from_numpy(fov))).numpy()
        out = self.squeeze_expand(t.from_numpy(full)).numpy()
        out[..., r:r + rh, c:c + rw] = fov
        return out
