"""TEST INFRASTRUCTURE — the fixed fovea's memory merged by pasting (``fov_memory_merge="paste"``) restated by
composition of the pinned C oracle, with no new arithmetic.

Per env, each observe call runs the fixed fovea update; then its control decides: RESET empties the memory and pushes,
APPLY pushes, KEEP pushes nothing.  A push keeps ``(orc.observe_fixed(..., "crop")[e], loc[e])`` in a deque of length M.
The observation starts as the background — zeros, or the periphery of the current ring,
``orc.observe_peripheral`` in float64 — and the held crops are written over it from the oldest to the newest.
``orc.observe_peripheral`` carries the current fovea at ``loc``; where the newest held window is not at ``loc`` (an
empty memory), the background is the bare ``Resize(S)(Resize(p)(plane))`` of ``orc.aa_resize``, which that call
composes.

RGB rings hold K * 3 planes and every plane is treated alike, so the oracle works on the plane ring; callers reshape to
(n, K, 3, S_h, S_w).
"""
from __future__ import annotations

from collections import deque

import numpy as np

from oracle import agym_oracle as orc

APPLY, RESET, KEEP = 0, 1, 2


class PasteOracle:
    def __init__(self, n_envs: int, depth: int):
        self.depth = int(depth)
        self.entries = [deque(maxlen=self.depth) for _ in range(int(n_envs))]

    def observe(self, ring, head, loc, fov_size, ctrl=None, peripheral_res=None):
        """``ring`` / ``head`` / ``loc`` after this call's ingest and fovea update; ``ctrl`` (n,) u8 or None (all APPLY);
        ``peripheral_res`` None for the zero background.  Returns float64 (n, P, S_h, S_w) in u8 units (integers for the
        zero background and wherever a window was pasted)."""
        n, P, S_h, S_w = ring.shape
        fh, fw = fov_size
        loc = np.ascontiguousarray(loc, np.int32)
        crops = orc.observe_fixed(ring, head, loc, fov_size, variant="crop")
        if peripheral_res is None:
            out = np.zeros(ring.shape, np.float64)
        else:
            out = orc.observe_peripheral(ring, head, loc, fov_size, peripheral_res)
        for e, q in enumerate(self.entries):
            c = APPLY if ctrl is None else int(ctrl[e])
            if c == RESET:
                q.clear()
            if c != KEEP:
                q.append((crops[e].copy(), (int(loc[e, 0]), int(loc[e, 1]))))
            if peripheral_res is not None and (not q or q[-1][1] != (int(loc[e, 0]), int(loc[e, 1]))):
                for k in range(P):
                    plane = ring[e, (int(head[e]) + 1 + k) % P].astype(np.float64)
                    out[e, k] = orc.aa_resize(orc.aa_resize(plane, tuple(peripheral_res)), (S_h, S_w))
            for crop, (r, cc) in q:
                out[e, :, r:r + fh, cc:cc + fw] = crop
        return out

    def pasted(self, shape_hw, fov_size):
        """bool (n, S_h, S_w): the pixels some held window covers."""
        fh, fw = fov_size
        m = np.zeros((len(self.entries),) + tuple(shape_hw), bool)
        for e, q in enumerate(self.entries):
            for _, (r, c) in q:
                m[e, r:r + fh, c:c + fw] = True
        return m

    def count(self):
        return np.array([len(q) for q in self.entries], np.int32)
