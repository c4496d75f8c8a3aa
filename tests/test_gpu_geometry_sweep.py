"""GPU: every kernel family against the C oracle at plan shapes other than 84x84 x 4 frames.

The launchers pick kernels and template specialisations from the plan's geometry (obs (S_h, S_w), ring depth, fovea,
periphery); most of those choices are reached only away from the standard 84x84 shape.  Each case of ``CASES`` runs end
to end — ingest with ragged flags, every fixed and flexible observation, the fixed fovea's memory — on guarded buffers,
against the oracle, and asserts which kernel served each call (``EXPECTED``): a geometry that silently lands on another
kernel would test nothing.  Non-square frames catch an H/W swap and a per-axis clamp taken against the wrong axis;
frames smaller than 84x84 catch a kernel that assumes a 7,056-byte plane (it writes into the guard bands).
"""
import collections
import json
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from tests import rgb_oracle
from tests.flex_periph_oracle import observe_flexible_peripheral
from tests.fovea_memory_oracle import MemoryOracle
from tests.glimpse_oracle import observe_glimpse
from tests.test_gpu_flexible_glimpse import _kernels
from tests.test_gpu_guard_bands import Guarded, _flags

pytestmark = pytest.mark.gpu

TOL = 0.5 + 1e-2
DEV = "cuda:0"
N = 301      # above 2 x 148 (several envs per persistent CTA) and not a multiple of any CTA's env count
STEPS = 3
DEPTH = 3    # fixed fovea memory
UNSUPPORTED = "geometry not supported by the sm_100a kernels"

# base "atari": 210x160 raw frames (`channels` of them, 3 = RGB through the luma) into a grey ring;
# base "dmc": renders at obs size, `channels` ring planes per frame (3 = RGB observations, K * 3 planes)
Case = collections.namedtuple("Case", "base channels obs frame_stack fov periph")
CASES = {
    "tall-std-width": Case("atari", 1, (100, 84), 4, (30, 30), (25, 20)),
    "wrap0": Case("atari", 1, (70, 88), 4, (24, 36), (14, 20)),
    "wide-p5": Case("atari", 1, (84, 112), 6, (30, 30), (20, 28)),
    "plane7056": Case("atari", 1, (126, 56), 4, (40, 20), (28, 16)),
    "rgb-narrow": Case("atari", 3, (84, 64), 4, (30, 30), (20, 16)),
    "rgb-wide": Case("atari", 3, (96, 128), 2, (30, 40), (24, 32)),
    "tiny": Case("atari", 1, (48, 32), 4, (16, 12), (12, 8)),
    "k1": Case("atari", 1, (84, 84), 1, (30, 30), (20, 20)),
    "k8": Case("atari", 1, (84, 84), 8, (30, 30), (42, 42)),
    "big": Case("atari", 1, (128, 128), 4, (16, 16), (64, 64)),
    "huge": Case("atari", 1, (176, 176), 2, (40, 40), (44, 44)),
    "dmc64": Case("dmc", 1, (64, 64), 3, (24, 24), (16, 16)),
    "dmc64-rgb": Case("dmc", 3, (64, 64), 3, (24, 24), (16, 16)),
    "dmc-rgb-k1": Case("dmc", 3, (84, 84), 1, (30, 30), (20, 20)),
    "dmc-rgb-k4": Case("dmc", 3, (84, 84), 4, (30, 30), (20, 20)),
    "dmc-wide": Case("dmc", 1, (48, 96), 3, (20, 40), (12, 24)),
}

FIXED_CALLS = ("ingest", "crop", "mask", "resize_full", "peripheral", "peripheral_uncached")
FLEX_CALLS = ("flex_mask", "flex_crop", "flex_resize_full", "flex_resize_fov", "flex_peripheral")
CALLS = FIXED_CALLS + ("memory",) + FLEX_CALLS

# the kernel each (case, call) must run: base name, plus the template arguments where the geometry selects them.
# Calls not listed in a case run the same kernel in every case (_ALWAYS).  The flexible mask / crop / glimpse /
# peripheral calls take the persistent kernel (_V3) unless its shared-memory budget or its blur tables (a band of at
# most 16 taps) rule it out; then k_observe_flexible_fast (mask, crop: up to 200 KB) or the table-driven kernel.
# None = the call must fail with AGYM_ERR_UNSUPPORTED: the table-driven flexible kernel keeps two f32 planes in shared
# memory, which past ~172 x 172 do not fit the 227 KB a block may have, and the faster kernels do not fit either.
_ALWAYS = {"mask": "k_observe_fixed<1>", "resize_full": "k_observe_fixed<2>", "peripheral_uncached": "k_observe_peripheral<false>",
           "memory": "k_observe_fixed_memory", "flex_resize_full": "k_observe_flexible<2>"}
_V3 = {"flex_mask": "k_observe_flexible_v3<1>", "flex_crop": "k_observe_flexible_v3<0>",
       "flex_resize_fov": "k_observe_flexible_v3<3>", "flex_peripheral": "k_observe_flexible_v3<4>"}
_FAST = {"flex_mask": "k_observe_flexible_fast<1>", "flex_crop": "k_observe_flexible_fast<0>",
         "flex_resize_fov": "k_observe_flexible_v3<3>", "flex_peripheral": "k_observe_flexible<4>"}
_GENERIC = {"flex_mask": "k_observe_flexible<1>", "flex_crop": "k_observe_flexible<0>",
            "flex_resize_fov": "k_observe_flexible<3>", "flex_peripheral": "k_observe_flexible<4>"}


def _expect(ingest, crop, peripheral, flex, **other):
    return {**_ALWAYS, **flex, "ingest": ingest, "crop": crop, "peripheral": peripheral, **other}


EXPECTED = {
    # the standard width bakes 160 / 84 into the TMA ingest whatever S_h; 100 rows are not the period-5 pattern
    "tall-std-width": _expect("k_ingest_atari_tma<160, 84, 1, false, 2>", "k_observe_fixed_crop_v3<30, 8>",
                              "k_observe_peripheral_v2<4, 0>", _FAST),
    "wrap0": _expect("k_ingest_atari_tma<0, 0, 1, false, 2>", "k_observe_fixed_crop_v3<0, 8>",
                     "k_observe_peripheral_v2<4, 0>", _V3),
    # period-5 rows at a width of 112: the tensor copies with the generic template; K = 6 stages too much for crop v3
    "wide-p5": _expect("k_ingest_atari_tma<0, 0, 1, true, 2>", "k_observe_fixed_crop_v2", "k_observe_peripheral_v2<3, 0>", _FAST),
    # 126 x 56 = 7,056 pixels: the 1,764-word tiles of the 84 x 84 plane, at S_w = 56
    "plane7056": _expect("k_ingest_atari_tma<0, 0, 1, false, 2>", "k_observe_fixed_crop_v3<0, 8>",
                         "k_observe_peripheral_v2<4, 1764>", _V3),
    # 64 columns from 160: a column pair's RGB source pixels do not lie within four, so no TMA ingest
    "rgb-narrow": _expect("k_ingest_atari_fast<3>", "k_observe_fixed_crop_v3<30, 8>", "k_observe_peripheral_v2<4, 0>", _V3),
    "rgb-wide": _expect("k_ingest_atari_tma<0, 0, 3, false, 2>", "k_observe_fixed_crop_v3<0, 8>",
                        "k_observe_peripheral_v2<2, 0>", _FAST),
    # 32 columns from 160: no fast ingest at all
    "tiny": _expect("k_ingest_atari<1>", "k_observe_fixed_crop_v3<0, 8>", "k_observe_peripheral_v2<4, 0>", _V3),
    "k1": _expect("k_ingest_gray_std<160, true, 2>", "k_observe_fixed_crop_v3<30, 8>", "k_observe_peripheral_v2<1, 0>", _V3),
    # K = 8 x 30 x 30 fits neither crop v3 nor crop v2; the v2 peripheral kernel would need 243,752 B
    "k8": _expect("k_ingest_atari_tma<160, 84, 1, true, 2>", "k_observe_fixed_crop_warp", "k_observe_peripheral<true>",
                  {**_GENERIC, "flex_resize_fov": "k_observe_flexible_v3<3>"}),
    # 128 -> 16: the composed blur band is wider than 16 taps (no persistent kernel); the v2 peripheral kernel would
    # need 271,816 B
    "big": _expect("k_ingest_atari_tma<0, 0, 1, false, 2>", "k_observe_fixed_crop_v3<0, 8>", "k_observe_peripheral<true>",
                   _GENERIC),
    "huge": _expect("k_ingest_atari_tma<0, 0, 1, false, 2>", "k_observe_fixed_crop_v3<0, 8>",
                    "k_observe_peripheral_v2<2, 0>", {c: None for c in _V3}, flex_resize_full=None),
    "dmc64": _expect("k_ingest_dmc", "k_observe_fixed_crop_v3<0, 8>", "k_observe_peripheral_v2<3, 0>", _V3),
    "dmc64-rgb": _expect("k_ingest_dmc_rgb", "k_observe_fixed_crop_v3<0, 4>", "k_observe_peripheral_v2<3, 0>", _V3),
    "dmc-rgb-k1": _expect("k_ingest_dmc_rgb", "k_observe_fixed_crop_v3<30, 8>", "k_observe_peripheral_std<3, 0, true>", _V3),
    "dmc-rgb-k4": _expect("k_ingest_dmc_rgb", "k_observe_fixed_crop_warp", "k_observe_peripheral_v2<3, 1764>",
                          {**_V3, "flex_peripheral": "k_observe_flexible<4>"}),
    "dmc-wide": _expect("k_ingest_dmc", "k_observe_fixed_crop_v3<0, 8>", "k_observe_peripheral_v2<3, 0>", _V3),
}

_KNAME = re.compile(r"\b(k_\w+)(<[^()]*>)?")


def _canon(spec):
    """'k_x<4, true>' -> ('k_x', '<4,1>'): profiler names print bool template arguments as 1 / 0 or true / false."""
    m = _KNAME.search(spec)
    args = m.group(2) or ""
    args = re.sub(r"\(bool\)|\s", "", args).replace("true", "1").replace("false", "0")
    return m.group(1), args


def assert_ran(names, spec):
    """One of the profiled kernel `names` has the base name of `spec` and, if `spec` names them, its template arguments."""
    base, args = _canon(spec)
    ran = [_canon(n) for n in names if _KNAME.search(n)]
    assert any(b == base and (not args or a == args) for b, a in ran), (spec, names)


def _planes(c):
    return c.frame_stack * (c.channels if c.base == "dmc" else 1)


def _path(c, n, memory=False):
    """An ObservationPath whose every state buffer sits between guard bands, and those bands."""
    from active_gym_b200 import LUMA_DMC, LUMA_RGB, ObservationPath
    P = _planes(c)
    g = dict(ring=Guarded((n, P) + c.obs, torch.uint8, DEV), head=Guarded((n,), torch.int32, DEV, P - 1),
             loc=Guarded((n, 2), torch.int32, DEV), res=Guarded((n, 2), torch.int32, DEV),
             pcache=Guarded((n, P) + c.periph, torch.float32, DEV))
    g["res"].t[:, 0], g["res"].t[:, 1] = c.fov
    if memory:
        E = (P * c.fov[0] * c.fov[1] + 15) // 16 * 16
        g.update(mem=Guarded((n, DEPTH, E), torch.uint8, DEV), mem_loc=Guarded((n, DEPTH, 2), torch.int32, DEV),
                 mem_state=Guarded((n, 2), torch.int32, DEV))
    dmc = c.base == "dmc"
    raw = c.obs + (3,) if dmc else (210, 160, c.channels)
    p = ObservationPath(n, c.frame_stack, c.obs, raw, luma=LUMA_DMC if dmc else LUMA_RGB, fov_size=c.fov,
                        peripheral_res=c.periph, sensory_action_mode="absolute", device=DEV,
                        channels=c.channels if dmc else 1, fov_memory=DEPTH if memory else 0,
                        buffers={k: v.t for k, v in g.items()})
    return p, g


class State:
    """The oracle's copy of one path's state."""

    def __init__(self, c, n):
        self.c = c
        self.ring, self.head = orc.new_state(n, _planes(c), c.obs)
        self.loc = np.zeros((n, 2), np.int32)
        self.res = np.tile(np.array([c.fov], np.int32), (n, 1))

    def update(self, a, ctrl=None, atype=None):
        """The fovea update of one observe call: APPLY = the reference's step, RESET = init (0, 0) / fov, KEEP = none."""
        loc, res = self.loc.copy(), self.res.copy()
        orc.update_loc(a, loc, obs_size=self.c.obs, fov_size=self.c.fov, atype=atype, res=res if atype is not None else None)
        k = np.zeros(len(a), np.uint8) if ctrl is None else ctrl
        self.loc[k == 0], self.loc[k == 1] = loc[k == 0], 0
        if atype is not None:
            self.res[k == 0], self.res[k == 1] = res[k == 0], self.c.fov


def _ingest(c, p, st, rng, step):
    n = p.n_envs
    fl = _flags(n, step, rng)
    if c.base == "dmc":
        fl = np.where(fl == 8, 8, np.where(fl & 4, 5, 1)).astype(np.uint8)
        f = rng.integers(0, 256, (n,) + c.obs + (3,), dtype=np.uint8)
        p.ingest_dmc(f, fl)
        (rgb_oracle.ingest_dmc_rgb if c.channels == 3 else orc.ingest_dmc)(f, fl, st.ring, st.head)
    else:
        fa, fb = rng.integers(0, 256, (2, n, 210, 160) + ((3,) if c.channels == 3 else ()), dtype=np.uint8)
        p.ingest_atari(fa, fb, fl)
        orc.ingest_atari(fa, fb, fl, st.ring, st.head)


def _fixed_actions(c, n, rng):
    """Targets over and past the valid range, with each axis's extremes and far overshoots first."""
    (S_h, S_w), (f_h, f_w) = c.obs, c.fov
    a = np.stack([rng.integers(-3, S_h - f_h + 4, n), rng.integers(-3, S_w - f_w + 4, n)], 1).astype(np.float64)
    edge = [(0, 0), (S_h - f_h, 0), (0, S_w - f_w), (S_h - f_h, S_w - f_w), (-1e6, 1e6), (1e6, -1e6), (S_h, S_w)]
    a[:len(edge)] = edge
    return a


def _flex_actions(c, n, rng, out_of_range):
    """FOV_LOC / FOV_RES actions: window corners, full-frame and one-pixel-wide windows along each axis.  With
    `out_of_range`, envs 11 and 12 ask for a window one row / one column larger than the frame: the kernels clamp that
    axis alone and report ERR_RES_RANGE.  Returns (actions, types, the actions the oracle applies)."""
    (S_h, S_w), (f_h, f_w) = c.obs, c.fov
    at = rng.integers(0, 2, n).astype(np.int32)
    res = np.stack([rng.integers(1, S_h + 1, n), rng.integers(1, S_w + 1, n)], 1)
    loc = np.stack([rng.integers(-3, S_h + 3, n), rng.integers(-3, S_w + 3, n)], 1)
    a = np.where(at[:, None] == 1, res, loc).astype(np.float64)
    ext = [((0, 0), 0), ((S_h - f_h, 0), 0), ((0, S_w - f_w), 0), ((-1e6, 1e6), 0), ((1e6, -1e6), 0),
           ((S_h, 1), 1), ((1, S_w), 1), ((S_h, S_w), 1), (c.fov, 1), ((f_h + 1, f_w - 1), 1), ((S_h - 1, 2), 1)]
    for i, (v, t) in enumerate(ext):
        a[i], at[i] = v, t
    want = a.copy()
    if out_of_range:
        a[11], a[12], at[11:13] = (S_h + 1, 1), (1, S_w + 1), 1
        want[11], want[12] = (S_h, 1), (1, S_w)
    return a, at, want


def _ctrl(n, rng, step):
    k = rng.choice(np.array([0, 0, 0, 1, 2], np.uint8), n)
    k[:16] = 0
    return k if step else None


def _u8(t, st):
    """A device output as (n, planes, ...) u8, the oracle's layout (RGB observations regroup the planes as (K, 3))."""
    a = t.cpu().numpy()
    return a.reshape(st.ring.shape[:2] + a.shape[-2:])


def _intact(*bufs):
    return all(b.intact() for b in bufs)


def _probe(name, n=N):
    """The kernel names of every call of case `name`, each call made once more in a profiler session of its own on idle
    envs / KEEP controls (the selection depends on the geometry, the buffers' alignment and the call, not on the
    flags or actions).  '<unsupported>' = the call was refused as a geometry no kernel serves."""
    c = CASES[name]
    p, g = _path(c, n, memory=True)
    st = State(c, n)
    rng = np.random.default_rng(0)
    for step in range(2):
        _ingest(c, p, st, rng, step)
    frames = torch.zeros(p.raw_frame_shape(), dtype=torch.uint8, device=DEV)
    idle, keep = np.full(n, 8, np.uint8), np.full(n, 2, np.uint8)

    def out(kind, v):
        return Guarded(p.out_shape(kind, v), torch.uint8, DEV).t

    calls = {"ingest": (lambda: p.ingest_dmc(frames, idle)) if c.base == "dmc" else (lambda: p.ingest_atari(frames, frames, idle)),
             "peripheral": lambda: p.observe_peripheral(None, ctrl=keep, out=out("peripheral", "mask")),
             "peripheral_uncached": lambda: p.observe_peripheral(None, ctrl=keep, use_cache=False, out=out("peripheral", "mask")),
             "memory": lambda: p.observe_fixed_memory(None, ctrl=keep, out=out("fixed_memory", "mask")),
             "flex_peripheral": lambda: p.observe_flexible_peripheral(None, ctrl=keep, out=out("flexible_peripheral", "mask"))}
    for v in ("crop", "mask", "resize_full"):
        calls[v] = lambda v=v: p.observe_fixed(None, variant=v, ctrl=keep, out=out("fixed", v))
    for v in ("mask", "crop", "resize_full", "resize_fov"):
        calls["flex_" + v] = lambda v=v: p.observe_flexible(None, variant=v, ctrl=keep, out=out("flexible", v))
    names = {}
    for call in CALLS:
        try:
            names[call] = _kernels(calls[call])
        except RuntimeError as ex:
            names[call] = ["<unsupported>" if UNSUPPORTED in str(ex) else f"<failed: {ex}>"]
    return names


@pytest.fixture(scope="module")
def kernel_names():
    """`_probe` of every case, in a process of its own: profiler sessions in a process that has already run many (the
    rest of the suite) can come back without any device activity at all, which would say nothing about the kernels."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, "-m", "tests.test_gpu_geometry_sweep"], cwd=root, capture_output=True, text=True,
                       timeout=600)
    assert r.returncode == 0, r.stderr[-4000:]
    return json.loads(r.stdout.strip().splitlines()[-1])


@pytest.mark.parametrize("name", list(CASES))
def test_ingest_and_fixed_fovea_match_the_oracle(name, kernel_names):
    c, exp = CASES[name], EXPECTED[name]
    rng = np.random.default_rng(sum(map(ord, name)))
    n, P = N, _planes(CASES[name])
    p, g = _path(c, n)
    st = State(c, n)
    keep = np.full(n, 2, np.uint8)
    outs = {v: Guarded((n, P) + (c.fov if v == "crop" else c.obs), torch.uint8, DEV)
            for v in ("crop", "mask", "resize_full", "peripheral", "peripheral_uncached")}
    p.observe_fixed(None, ctrl="reset", out=outs["crop"].t.view(p.out_shape("fixed", "crop")))
    for step in range(STEPS):
        _ingest(c, p, st, rng, step)
        torch.cuda.synchronize()
        assert np.array_equal(g["head"].t.cpu().numpy(), st.head), step
        assert np.array_equal(g["ring"].t.cpu().numpy(), st.ring), step
        for v in ("crop", "mask", "resize_full"):
            a = _fixed_actions(c, n, rng)
            out = outs[v].t.view(p.out_shape("fixed", v))
            p.observe_fixed(a, variant=v, out=out)
            st.update(a)
            torch.cuda.synchronize()
            assert np.array_equal(g["loc"].t.cpu().numpy(), st.loc), (v, step)
            want = orc.observe_fixed(st.ring, st.head, st.loc, c.fov, variant=v)
            got = _u8(outs[v].t, st)
            if v == "resize_full":
                assert np.abs(got - want).max() <= TOL, step
            else:
                assert np.array_equal(got, want), (v, step)
        a = _fixed_actions(c, n, rng)
        ctrl = _ctrl(n, rng, step)
        p.observe_peripheral(a, ctrl=ctrl, out=outs["peripheral"].t.view(p.out_shape("peripheral", "mask")))
        st.update(a, ctrl)
        p.observe_peripheral(None, ctrl=keep, use_cache=False,
                             out=outs["peripheral_uncached"].t.view(p.out_shape("peripheral", "mask")))
        torch.cuda.synchronize()
        assert np.array_equal(g["loc"].t.cpu().numpy(), st.loc), step
        got = _u8(outs["peripheral"].t, st)
        assert np.abs(got - orc.observe_peripheral(st.ring, st.head, st.loc, c.fov, c.periph)).max() <= TOL, step
        full = orc.stack(st.ring, st.head)
        f_h, f_w = c.fov
        for e in range(n):   # the pasted fovea is bit exact
            r, q = st.loc[e]
            assert np.array_equal(got[e, :, r:r + f_h, q:q + f_w], full[e, :, r:r + f_h, q:q + f_w]), (e, step)
        # the squeeze cache the ingest kernel wrote == the squeeze recomputed from the ring
        assert (outs["peripheral_uncached"].t.int() - outs["peripheral"].t.int()).abs().max().item() <= 1, step
    assert _intact(*g.values(), *outs.values())
    for call in FIXED_CALLS:
        assert_ran(kernel_names[name][call], exp[call])


@pytest.mark.parametrize("name", list(CASES))
def test_fixed_memory_matches_the_oracle(name, kernel_names):
    c = CASES[name]
    rng = np.random.default_rng(sum(map(ord, name)) + 1)
    n = N
    p, g = _path(c, n, memory=True)
    st = State(c, n)
    mo = MemoryOracle(n, DEPTH)
    out = Guarded((n, _planes(c)) + c.obs, torch.uint8, DEV)
    view = out.t.view(p.out_shape("fixed_memory", "mask"))
    for step in range(STEPS + 1):
        _ingest(c, p, st, rng, step)
        a = _fixed_actions(c, n, rng)
        ctrl = _ctrl(n, rng, step)
        p.observe_fixed_memory(a, ctrl=ctrl, out=view)
        st.update(a, ctrl)
        torch.cuda.synchronize()
        assert np.array_equal(g["loc"].t.cpu().numpy(), st.loc), step
        assert np.array_equal(_u8(out.t, st), mo.observe(st.ring, st.head, st.loc, c.fov, ctrl)), step
    assert _intact(*g.values(), out)
    assert_ran(kernel_names[name]["memory"], EXPECTED[name]["memory"])


def _flex_oracle(variant, st, c):
    if variant == "flex_resize_fov":
        return observe_glimpse(st.ring, st.head, st.loc, st.res, c.fov)
    if variant == "flex_peripheral":
        return observe_flexible_peripheral(st.ring, st.head, st.loc, st.res, c.fov, c.periph)
    return orc.observe_flexible(st.ring, st.head, st.loc, st.res, c.fov, variant=variant[5:])


@pytest.mark.parametrize("variant", FLEX_CALLS)
@pytest.mark.parametrize("name", list(CASES))
def test_flexible_fovea_matches_the_oracle(name, variant, kernel_names):
    from active_gym_b200 import _lib
    c, spec = CASES[name], EXPECTED[name][variant]
    rng = np.random.default_rng(sum(map(ord, name + variant)))
    n = N
    p, g = _path(c, n)
    st = State(c, n)
    kind, v = ("flexible_peripheral", "mask") if variant == "flex_peripheral" else ("flexible", variant[5:])
    out = Guarded(p.out_shape(kind, v), torch.uint8, DEV)

    def observe(a, at, ctrl=None):
        if variant == "flex_peripheral":
            return p.observe_flexible_peripheral(a, at, ctrl=ctrl, out=out.t)
        return p.observe_flexible(a, at, variant=v, ctrl=ctrl, out=out.t)

    _ingest(c, p, st, rng, 0)
    if spec is None:   # the geometry no kernel serves: a clean error, nothing sticky on the context
        with pytest.raises(RuntimeError, match=UNSUPPORTED):
            observe(None, None, ctrl="reset")
        torch.cuda.synchronize()
        p.observe_fixed(None, ctrl="reset")   # the next call does not inherit an error either
        torch.cuda.synchronize()
        assert _intact(*g.values(), out)
        return
    for step in range(STEPS):
        if step:
            _ingest(c, p, st, rng, step)
        a, at, want_a = _flex_actions(c, n, rng, out_of_range=step == 1)
        ctrl = _ctrl(n, rng, step)
        observe(a, at, ctrl)
        st.update(want_a, ctrl, at)
        assert p.read_errors() == (_lib.ERR_RES_RANGE if step == 1 else 0), step
        assert np.array_equal(g["loc"].t.cpu().numpy(), st.loc) and np.array_equal(g["res"].t.cpu().numpy(), st.res), step
        got = _u8(out.t, st).astype(np.float64)
        want = _flex_oracle(variant, st, c)
        assert got.shape == want.shape
        assert np.abs(got - want).max() <= TOL, step
        # an unblurred window is bit exact (fov_env.py:286 looks at rows only)
        for e in np.flatnonzero(st.res[:, 0] <= c.fov[0]) if variant in ("flex_mask", "flex_crop", "flex_peripheral") else ():
            (r, q), (rh, rw) = (st.loc[e], st.res[e]) if variant != "flex_crop" else ((0, 0), st.res[e])
            assert np.array_equal(got[e, :, r:r + rh, q:q + rw], want[e, :, r:r + rh, q:q + rw]), (e, step)
    assert _intact(*g.values(), out)
    assert_ran(kernel_names[name][variant], spec)


# (obs, fovea, the rows' cyclic run (P, o, L) in 210 raw rows): wrap == max(o + L - P, 0) == 0 is one strided copy,
# wrap > 0 a head, a strided body and a tail
PIPELINED = {"wrap0": ((70, 88), (24, 36), (3, 1, 2)), "wrap0-42": ((42, 88), (24, 36), (5, 2, 2)),
             "tall-std-width": ((100, 84), (30, 30), (21, 11, 20))}


@pytest.mark.parametrize("name", list(PIPELINED))
def test_pipelined_host_frames_at_other_heights(name):
    from active_gym_b200.pipeline import PipelinedPath
    obs, fov, run = PIPELINED[name]
    rng = np.random.default_rng(obs[0])
    n, K = 203, 4
    pp = PipelinedPath(n, K, obs, (210, 160, 1), shards=3, fov_size=fov, sensory_action_mode="absolute")
    assert pp.run == run
    rows = pp.used_rows
    ring, head = orc.new_state(n, K, obs)
    for step in range(4):
        fa, fb = rng.integers(0, 256, (2, n, 210, 160), dtype=np.uint8)
        fl = _flags(n, step, rng)
        if step % 2:   # frames that hold only the sampled rows
            pp.ingest_atari(torch.from_numpy(np.ascontiguousarray(fa[:, rows])).pin_memory(),
                            torch.from_numpy(np.ascontiguousarray(fb[:, rows])).pin_memory(), fl, packed=True)
        else:          # full pinned frames: the strided copy of the sampled rows
            pp.ingest_atari(torch.from_numpy(fa).pin_memory(), torch.from_numpy(fb).pin_memory(), fl)
        orc.ingest_atari(fa, fb, fl, ring, head)
        pp.sync()
        assert np.array_equal(pp.head.cpu().numpy(), head), step
        assert np.array_equal(pp.ring.cpu().numpy(), ring), step


def test_plans_whose_plane_is_not_a_multiple_of_16_pixels_are_refused():
    """obs (70, 84) and (42, 84) give the single-copy row runs too, but their planes (5,880 / 3,528 pixels) are not a
    multiple of 16: the plan refuses them rather than running kernels that move planes in 16-byte vectors."""
    from active_gym_b200 import ObservationPath
    for obs in [(70, 84), (42, 84)]:
        with pytest.raises(RuntimeError, match=UNSUPPORTED):
            ObservationPath(4, 4, obs, (210, 160, 1), fov_size=(24, 36), device=DEV)


if __name__ == "__main__":   # the kernel_names fixture's process
    print(json.dumps({name: _probe(name) for name in CASES}))
