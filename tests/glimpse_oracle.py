"""TEST INFRASTRUCTURE — the flexible fovea's glimpse (``resize_to_fov``) restated by composition of the pinned C
oracle, with no new arithmetic.

The glimpse of an env is, per plane, torchvision's ``Resize(fov_size)`` of the unblurred window
``full_state[..., r:r+rh, c:c+rw]`` (fov_env.py:248,284-285): the first of the two resamples the reference's blur
performs (fov_env.py:276-278).  ``observe_glimpse`` reads each plane's window with the ring indexing of
``or_observe_flexible`` (oldest -> newest from ``head + 1``) and resamples it with ``agym_oracle.aa_resize``, the
oracle's ``or_aa_resize_plane`` that every other resample of the oracle uses (under the same ``set_antialias`` switch).
"""
from __future__ import annotations

import numpy as np

from oracle import agym_oracle as orc


def observe_glimpse(ring, head, loc, res, fov_size, use_f32=False):
    """``ring`` u8 (n, P, S_h, S_w), ``head`` (n,), ``loc`` / ``res`` int (n, 2) -> float64 (n, P, f_h, f_w) in u8 units."""
    n, P = ring.shape[:2]
    fov = tuple(int(v) for v in fov_size)
    out = np.empty((n, P) + fov, np.float64)
    for e in range(n):
        r, c = int(loc[e][0]), int(loc[e][1])
        rh, rw = int(res[e][0]), int(res[e][1])
        for k in range(P):
            plane = ring[e, (int(head[e]) + 1 + k) % P]
            out[e, k] = orc.aa_resize(plane[r:r + rh, c:c + rw].astype(np.float64), fov, use_f32=use_f32)
    return out
