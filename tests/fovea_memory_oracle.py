"""TEST INFRASTRUCTURE — the fixed fovea's memory (``fov_memory``) restated by composition of the pinned C oracle, with
no new arithmetic.

Per env, each observe call runs the fixed fovea update; then its control decides: RESET empties the memory and pushes,
APPLY pushes, KEEP pushes nothing.  A push keeps the call's mask_out observation (``orc.observe_fixed(..., "mask")``, or
``tests/rgb_oracle.observe_fixed`` for RGB) in a deque of length M; the observation is ``np.maximum.reduce`` over the
deque, all zeros when it is empty.
"""
from __future__ import annotations

from collections import deque

import numpy as np

from oracle import agym_oracle as orc

APPLY, RESET, KEEP = 0, 1, 2


class MemoryOracle:
    def __init__(self, n_envs: int, depth: int):
        self.depth = int(depth)
        self.entries = [deque(maxlen=self.depth) for _ in range(int(n_envs))]

    def observe(self, ring, head, loc, fov_size, ctrl=None, rgb=False):
        """``ring`` / ``head`` / ``loc`` after this call's ingest and fovea update; ``ctrl`` (n,) u8 or None (all APPLY).
        Returns u8 (n, P, S_h, S_w), or (n, K, 3, S_h, S_w) with ``rgb``."""
        if rgb:
            from tests import rgb_oracle
            masks = rgb_oracle.observe_fixed(ring, head, loc, fov_size, variant="mask")
        else:
            masks = orc.observe_fixed(ring, head, loc, fov_size, variant="mask")
        out = np.zeros_like(masks)
        for e, q in enumerate(self.entries):
            c = APPLY if ctrl is None else int(ctrl[e])
            if c == RESET:
                q.clear()
            if c != KEEP:
                q.append(masks[e].copy())
            if q:
                out[e] = np.maximum.reduce(list(q))
        return out

    def count(self):
        return np.array([len(q) for q in self.entries], np.int32)
