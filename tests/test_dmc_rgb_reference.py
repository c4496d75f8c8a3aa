"""CPU: the semantics of DMC ``grey=False`` observations, pinned to the reference itself.

An RGB observation is (K, 3, h, w): the render's channels, unconverted, through the same wrapper operations as a grey
plane, with one fov_loc / fov_res per env.  Since cv2's BGR2GRAY maps a pixel (v, v, v) to v, channel c of that
observation must equal the ``grey=True`` observation of the reference fed renders whose three channels all equal
channel c, under the same sensory actions.  That is checked here on fresh seeded renders against two stand-ins for the
reference (as in tests/test_oracle_vs_reference.py): the unmodified reference run live where a checkout exists, and
the restated port everywhere.  Then the composed oracle (tests/rgb_oracle.py), which the GPU tests compare the kernels
with, is checked against the RGB port.  Last, the C ABI's handling of ``obs_c``."""
import ctypes as C
import random

import numpy as np
import pytest

from active_gym_b200 import _lib
from oracle import agym_oracle as orc
from oracle import ref_harness as rh
from oracle.ref_port import RefPortEnv
from tests import rgb_oracle as rgb
from tests.test_oracle_vs_reference import REFS, _Reference, _u8_exact

S, FA, FH = (84, 84), 1, 4
K = 3

# (wrapper, sensory_action_mode, variant, fovea, periphery)
CASES = [
    ("fixed", "absolute", "crop", (30, 30), None),
    ("fixed", "relative", "crop", (30, 30), None),
    ("fixed", "absolute", "mask", (21, 37), None),
    ("fixed", "relative", "resize_full", (30, 30), None),
    ("peripheral", "relative", "mask", (30, 30), (20, 20)),
    ("flexible", "absolute", "mask", (30, 30), None),
    ("flexible", "absolute", "resize_full", (30, 30), None),
    ("flexible", "absolute", "crop", (30, 30), None),
]
IDS = [f"{w}-{m}-{v}" for w, m, v, _, _ in CASES]
CLS = {"fixed": "DMCFixedFovealEnv", "peripheral": "DMCFixedFovealPeripheralEnv", "flexible": "DMCFlexibleFovealEnv"}


def _actions(rng, wrapper, mode, steps):
    out = []
    for i in range(steps):
        atype = int(rng.integers(0, 2)) if wrapper == "flexible" else 0
        if atype == 1:
            a = rng.integers(20, 51, 2)   # FOV_RES: integer window sizes
        elif mode == "relative":
            a = rng.uniform(-14, 14, 2) if i % 3 else rng.integers(-10, 11, 2) + 0.5
        else:
            a = rng.uniform(-5, 70, 2) if i % 3 else rng.integers(0, 55, 2) + 0.5
        out.append((np.asarray(a), atype))
    return out


def _port_kw(wrapper, mode, variant, fov, periph, init):
    return dict(wrapper=wrapper, frame_stack=K, obs_size=S, fov_size=fov, fov_init_loc=init, mode=mode, lo=-10.0,
                hi=10.0, variant=variant, peripheral_res=periph)


def _grey_run(ref, screens, case, init, actions):
    """The grey=True observations of one env fed ``screens``: [(obs, fov_loc, fov_res, index of the screen it shows)]."""
    wrapper, mode, variant, fov, periph = case
    out = []
    if ref == "reference":
        _, _, dmc = rh.load_reference()
        script = rh.ScreenScript(screens)
        rh.ScreenScript.current = script
        kw = dict(fov_size=fov, fov_init_loc=init, sensory_action_mode=mode, frame_stack=K, action_repeat=2,
                  mask_out=variant == "mask", resize_to_full=variant == "resize_full")
        if mode == "relative":
            kw["sensory_action_space"] = (-10.0, 10.0)
        if periph:
            kw["peripheral_res"] = periph
        env = _Reference(getattr(dmc, CLS[wrapper])(dmc.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0,
                                                                   obs_size=S, **kw)), script)
        random.seed(0)
        obs, info, idx = env.reset()
        out.append((obs, info["fov_loc"], info.get("fov_res"), idx[-1]))
        for a, atype in actions:
            act = {"motor_action": np.zeros(2, np.float32), "sensory_action": a}
            if wrapper == "flexible":
                act["sensory_action_type"] = atype
            obs, info, idx = env.step(act)
            out.append((obs, info["fov_loc"], info.get("fov_res"), idx[-1]))
        return out
    env = RefPortEnv(kind="dmc", **_port_kw(*case, init))
    out.append((env.reset(screens[0]), env.loc.copy(), env.res.copy(), 0))
    for t, (a, atype) in enumerate(actions, start=1):
        out.append((env.step(screens[t], None, a, atype), env.loc.copy(), env.res.copy(), t))
    return out


def _rgb_port_run(screens, case, init, actions, shown):
    """The RGB port fed the screens the grey runs showed."""
    env = rgb.RefPortRGBEnv(**_port_kw(*case, init))
    out = [(env.reset(screens[shown[0]]), env.loc.copy(), env.res.copy())]
    for t, (a, atype) in enumerate(actions, start=1):
        out.append((env.step(screens[shown[t]], None, a, atype), env.loc.copy(), env.res.copy()))
    return out


def _setup(seed, case):
    rng = np.random.default_rng(seed)
    screens = rng.integers(0, 256, (60, 84, 84, 3), dtype=np.uint8)
    init = (int(rng.integers(0, 50)), int(rng.integers(0, 50)))
    return screens, init, _actions(rng, case[0], case[1], 10)


@pytest.mark.parametrize("ref", REFS)
@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_rgb_channel_equals_grey_run_of_replicated_renders(ref, case):
    screens, init, actions = _setup(7 + CASES.index(case), case)
    greys = [_grey_run(ref, rgb.replicate(screens, c), case, init, actions) for c in range(3)]
    shown = [g[3] for g in greys[0]]
    for g in greys[1:]:
        assert [x[3] for x in g] == shown
    port = _rgb_port_run(screens, case, init, actions, shown)
    for t, (obs, loc, res) in enumerate(port):
        obs = np.asarray(obs)
        assert obs.ndim == 4 and obs.shape[:2] == (K, 3), obs.shape
        for c in range(3):
            g_obs, g_loc, g_res, _ = greys[c][t]
            assert np.array_equal(np.asarray(g_loc), loc)
            if case[0] == "flexible":
                assert np.array_equal(np.asarray(g_res), res)
            assert np.array_equal(obs[:, c], np.asarray(g_obs, obs.dtype)), (t, c)


@pytest.mark.parametrize("case", CASES, ids=IDS)
def test_composed_oracle_equals_rgb_port(case):
    wrapper, mode, variant, fov, periph = case
    screens, init, actions = _setup(107 + CASES.index(case), case)
    port = _rgb_port_run(screens, case, init, actions, list(range(len(actions) + 1)))
    ring, head = rgb.new_state(1, K, S)
    loc = np.array([init], np.int32)
    res = np.array([fov], np.int32)

    def check(obs):
        f32 = np.asarray(obs).dtype == np.float32
        if wrapper == "flexible":
            got = rgb.observe_flexible(ring, head, loc, res, fov, variant=variant, use_f32=f32)[0]
            if variant == "crop":
                got = got[..., :res[0, 0], :res[0, 1]]
        elif wrapper == "peripheral":
            got = rgb.observe_peripheral(ring, head, loc, fov, periph, use_f32=f32)[0]
        else:
            got = rgb.observe_fixed(ring, head, loc, fov, variant=variant, use_f32=f32)[0]
        assert got.shape == np.shape(obs)
        if got.dtype == np.uint8:
            assert np.array_equal(orc.to_reference_float(got), np.asarray(obs, np.float64))
            assert np.array_equal(got, _u8_exact(obs))
        else:   # resampled planes: the oracle keeps the f64 value the reference rounds through float32
            assert np.abs(got - np.asarray(obs, np.float64) * 255.0).max() <= 1e-4

    rgb.ingest_dmc_rgb(screens[0][None], np.array([FA | FH], np.uint8), ring, head)
    assert head[0] == 2
    check(port[0][0])
    for t, (a, atype) in enumerate(actions, start=1):
        rgb.ingest_dmc_rgb(screens[t][None], np.array([FA], np.uint8), ring, head)
        assert head[0] == 3 * (t % K) + 2
        orc.update_loc(np.asarray(a, np.float64), loc, obs_size=S, fov_size=fov, relative=mode == "relative", lo=-10.0,
                       hi=10.0, atype=np.array([atype]) if wrapper == "flexible" else None,
                       res=res if wrapper == "flexible" else None)
        assert np.array_equal(loc[0], port[t][1])
        if wrapper == "flexible":
            assert np.array_equal(res[0], port[t][2])
        check(port[t][0])


def test_composed_ingest_writes_the_channel_planes_and_keeps_idle_envs():
    rng = np.random.default_rng(3)
    n = 5
    ring, head = rgb.new_state(n, K, S)
    for step in range(5):
        f = rng.integers(0, 256, (n,) + S + (3,), dtype=np.uint8)
        flags = np.array([FA | FH if step == 0 else FA, FA, 8, FA | FH, FA], np.uint8)   # env 2 idle
        before, h0 = ring.copy(), head.copy()
        rgb.ingest_dmc_rgb(f, flags, ring, head)
        for e in range(n):
            if flags[e] & 8:
                assert head[e] == h0[e] and np.array_equal(ring[e], before[e])
                continue
            s = (h0[e] // 3 + 1) % K
            assert head[e] == 3 * s + 2
            assert np.array_equal(ring[e, 3 * s:3 * s + 3], f[e].transpose(2, 0, 1))
            if flags[e] & FH:
                others = [p for p in range(3 * K) if p // 3 != s]
                assert not ring[e, others].any()
    st = rgb.stack(ring, head)
    assert st.shape == (n, K, 3) + S
    assert np.array_equal(st[0, -1], f[0].transpose(2, 0, 1))


# ---------------------------------------------------------------------------------------------- C ABI
def _cfg(**kw):
    cfg = _lib.Config()
    cfg.n_envs, cfg.frame_stack, cfg.obs_h, cfg.obs_w = 4, 3, 84, 84
    cfg.raw_h, cfg.raw_w, cfg.raw_c = 84, 84, 3
    cfg.luma_w[:] = list(orc.LUMA_DMC)
    cfg.fov_h = cfg.fov_w = 30
    for k, v in kw.items():
        setattr(cfg, k, v)
    return cfg


def test_abi_version_4_and_obs_c_is_the_last_field():
    L = C.CDLL(_lib.LIB_PATH)
    assert _lib.ABI_VERSION == 4 and L.agym_abi_version() == 4
    assert [f[0] for f in _lib.Config._fields_][-1] == "obs_c"
    assert _lib.Config.obs_c.offset == _lib.Config.no_antialias.offset + 4
    assert hasattr(L, "agym_ingest_dmc")


@pytest.mark.parametrize("bad", [
    dict(obs_c=2), dict(obs_c=-1), dict(obs_c=4),
    dict(obs_c=3, raw_h=210, raw_w=160),        # an Atari raw shape: RGB is DMC-only
    dict(obs_c=3, raw_c=1),                      # grey frames have no channels to keep
    dict(obs_c=3, raw_h=96),                     # not rendered at obs_size
])
def test_plan_create_rejects_bad_obs_c_without_touching_the_gpu(bad):
    plan = C.c_void_p()
    assert _lib.lib().agym_plan_create(C.byref(_cfg(**bad)), C.byref(plan)) == -1
    assert not plan.value


@pytest.mark.parametrize("obs_c", [0, 1, 3])
def test_plan_create_accepts_grey_and_rgb(obs_c):
    """Past validation, plan creation only fails for want of a device (status -3) in a CPU-only container."""
    plan = C.c_void_p()
    L = _lib.lib()
    st = L.agym_plan_create(C.byref(_cfg(obs_c=obs_c)), C.byref(plan))
    assert st in (0, -3)
    if st == 0:
        planes = 3 * (3 if obs_c == 3 else 1)
        assert L.agym_plan_ring_bytes(plan) == 4 * planes * 84 * 84
        L.agym_plan_destroy(plan)
