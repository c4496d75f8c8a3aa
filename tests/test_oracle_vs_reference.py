"""CPU: the restated oracle against the reference's env step on fresh random screens and actions that are NOT in
tests/golden, through two stand-ins for the reference:
  * ``reference``: the UNMODIFIED reference executed live (oracle/ref_harness.py imports
    active_gym/{fov_env,atari_env,dmc_env}.py from $AGYM_REFERENCE_ROOT, default oracle/_ref, under simulator stubs);
    skipped where no checkout of it exists, since the repository does not contain one;
  * ``port``: oracle/ref_port.py, the reference's per-env library calls restated and pinned to the reference's recorded
    outputs by tests/test_ref_port_golden.py; fed the screens in order (one on reset, the max-pooled pair per Atari step,
    one per DMC step).  Runs everywhere."""
import random

import numpy as np
import pytest

from oracle import agym_oracle as orc
from oracle import ref_harness as rh
from oracle.ref_port import RefPortEnv

REFS = [pytest.param("reference", marks=pytest.mark.skipif(not rh.reference_available(),
                                                           reason="no checkout of the reference in oracle/_ref or at AGYM_REFERENCE_ROOT")),
        "port"]

S, FA, FB, FH = (84, 84), 1, 2, 4


def _u8_exact(ref):
    u = np.rint(np.asarray(ref, np.float64) * 255.0).astype(np.uint8)
    assert np.array_equal((u.astype(np.float32) / np.float32(255)).astype(np.float64), np.asarray(ref, np.float64))
    return u


class _Reference:
    """The reference env; which screens it read comes from the fake simulator's log."""

    def __init__(self, env, script):
        self.env, self.script = env, script

    def reset(self):
        n0 = len(self.script.log)
        obs, info = self.env.reset()
        return obs, info, self.script.log[n0:]

    def step(self, act):
        n0 = len(self.script.log)
        obs, _, done, _, info = self.env.step(act)
        assert not done
        return obs, info, self.script.log[n0:]


class _Port:
    def __init__(self, screens, **kw):
        self.env, self.screens, self.t = RefPortEnv(**kw), screens, 0

    def _info(self):
        return {"fov_loc": self.env.loc.copy(), "fov_res": self.env.res.copy()}

    def _take(self, k):
        self.t += k
        return list(range(self.t - k, self.t))

    def reset(self):
        idx = self._take(1)
        return self.env.reset(self.screens[idx[0]]), self._info(), idx

    def step(self, act):
        idx = self._take(1 if self.env.kind == "dmc" else 2)
        fb = self.screens[idx[-1]]
        obs = self.env.step(self.screens[idx[0]], fb, np.asarray(act["sensory_action"]), act.get("sensory_action_type", 0))
        return obs, self._info(), idx


def _drive_atari(ref, cls_name, seed, *, mode, variant="crop", periph=None, flexible=False, K=4, fov=(30, 30), steps=14):
    import torch
    rng = np.random.default_rng(seed)
    screens = rng.integers(0, 256, (4 * steps + 40, 210, 160, 1), dtype=np.uint8)
    kw = dict(fov_size=fov, fov_init_loc=(int(rng.integers(0, 50)), int(rng.integers(0, 50))), sensory_action_mode=mode,
              frame_stack=K, mask_out=(variant == "mask"), resize_to_full=(variant == "resize_full"))
    if mode == "relative":
        kw["sensory_action_space"] = (-10.0, 10.0)
    if periph:
        kw["peripheral_res"] = periph
    if ref == "reference":
        _, atari, _ = rh.load_reference()
        script = rh.ScreenScript(screens)
        rh.ScreenScript.current = script
        env = _Reference(getattr(atari, cls_name)(atari.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)), script)
        random.seed(seed)
    else:
        env = _Port(screens[..., 0], kind="atari", wrapper="flexible" if flexible else ("peripheral" if periph else "fixed"),
                    frame_stack=K, obs_size=S, fov_size=fov, fov_init_loc=kw["fov_init_loc"], mode=mode, lo=-10.0, hi=10.0,
                    variant=variant, peripheral_res=periph)

    ring, head = orc.new_state(1, K, S)
    loc = np.rint(np.array([kw["fov_init_loc"]], np.float64)).astype(np.int32)
    res = np.array([fov], np.int32)

    def check(obs, info):
        assert np.array_equal(info["fov_loc"], loc[0])
        if flexible:
            assert np.array_equal(info["fov_res"], res[0])
            got = orc.observe_flexible(ring, head, loc, res, fov, variant=variant)[0]
            if variant == "crop":
                got = got[:, :res[0, 0], :res[0, 1]]
        elif periph:
            got = orc.observe_peripheral(ring, head, loc, fov, periph)[0]
        else:
            got = orc.observe_fixed(ring, head, loc, fov, variant=variant)[0]
        want = np.asarray(obs, np.float64) * 255.0
        assert got.shape == want.shape
        if got.dtype == np.uint8:
            assert np.array_equal(got, _u8_exact(obs))
        else:
            assert np.abs(got - want).max() <= 1e-4  # f32(u)/255 carries 3e-8 relative error into the f64 resample

    obs, info, idx = env.reset()
    orc.ingest_atari(screens[idx[0], :, :, 0][None], screens[idx[0], :, :, 0][None], np.array([FA | FH], np.uint8), ring, head)
    check(obs, info)
    for i in range(steps):
        atype = int(rng.integers(0, 2)) if flexible else 0
        if atype == 1:
            a = rng.integers(20, 51, 2)  # integer dtype: the reference slices with fov_res unvalidated (fov_env.py:284,323)
        elif mode == "relative":
            a = rng.uniform(-14, 14, 2) if i % 3 else rng.integers(-10, 11, 2) + 0.5
        else:
            a = rng.uniform(-5, 70, 2) if i % 3 else rng.integers(0, 55, 2) + 0.5
        act = {"motor_action": 0, "sensory_action": torch.tensor(a) if (i % 2 and atype == 0) else a}
        if flexible:
            act["sensory_action_type"] = atype
        obs, info, idx = env.step(act)
        assert len(idx) == 2
        orc.ingest_atari(screens[idx[0], :, :, 0][None], screens[idx[1], :, :, 0][None], np.array([FA | FB], np.uint8), ring, head)
        orc.update_loc(np.asarray(a, np.float64), loc, obs_size=S, fov_size=fov, relative=(mode == "relative"), lo=-10.0, hi=10.0,
                       atype=np.array([atype]) if flexible else None, res=res if flexible else None)
        check(obs, info)


@pytest.mark.parametrize("ref", REFS)
@pytest.mark.parametrize("seed", [11, 12])
@pytest.mark.parametrize("mode", ["absolute", "relative"])
def test_fixed_crop_and_mask_live(ref, seed, mode):
    _drive_atari(ref, "AtariFixedFovealEnv", seed, mode=mode, variant="crop")
    _drive_atari(ref, "AtariFixedFovealEnv", seed + 100, mode=mode, variant="mask", K=3, fov=(21, 37))


@pytest.mark.parametrize("ref", REFS)
@pytest.mark.parametrize("seed", [21, 22])
def test_peripheral_live(ref, seed):
    _drive_atari(ref, "AtariFixedFovealPeripheralEnv", seed, mode="relative", periph=(20, 20), steps=8)


@pytest.mark.parametrize("ref", REFS)
@pytest.mark.parametrize("variant", ["mask", "resize_full", "crop"])
def test_flexible_live(ref, variant):
    _drive_atari(ref, "AtariFlexibleFovealEnv", 31, mode="absolute", variant=variant, flexible=True, steps=10)


@pytest.mark.parametrize("ref", REFS)
def test_resize_to_full_live(ref):
    _drive_atari(ref, "AtariFixedFovealEnv", 41, mode="absolute", variant="resize_full", steps=6)


@pytest.mark.parametrize("ref", REFS)
def test_dmc_live(ref):
    rng = np.random.default_rng(51)
    screens = rng.integers(0, 256, (40, 84, 84, 3), dtype=np.uint8)
    K, fov = 3, (30, 30)
    if ref == "reference":
        _, _, dmc = rh.load_reference()
        script = rh.ScreenScript(screens)
        rh.ScreenScript.current = script
        args = dmc.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, fov_size=fov, fov_init_loc=(3, 4),
                              sensory_action_mode="absolute", frame_stack=K, action_repeat=2, mask_out=False, resize_to_full=False)
        env = _Reference(dmc.DMCFixedFovealEnv(args), script)
    else:
        env = _Port(screens, kind="dmc", wrapper="fixed", frame_stack=K, obs_size=S, fov_size=fov, fov_init_loc=(3, 4),
                    mode="absolute")
    ring, head = orc.new_state(1, K, S)
    loc = np.array([[3, 4]], np.int32)
    obs, info, idx = env.reset()
    orc.ingest_dmc(screens[idx[-1]][None], np.array([FA | FH], np.uint8), ring, head)
    assert np.array_equal(orc.observe_fixed(ring, head, loc, fov)[0], _u8_exact(obs))
    for i in range(8):
        a = rng.uniform(-3, 60, 2)
        obs, info, idx = env.step({"motor_action": np.zeros(2, np.float32), "sensory_action": a})
        orc.ingest_dmc(screens[idx[-1]][None], np.array([FA], np.uint8), ring, head)
        orc.update_loc(np.asarray(a, np.float64), loc, obs_size=S, fov_size=fov)
        assert np.array_equal(info["fov_loc"], loc[0])
        assert np.array_equal(orc.observe_fixed(ring, head, loc, fov)[0], _u8_exact(obs))
