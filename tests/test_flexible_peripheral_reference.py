"""CPU: the flexible fovea over the peripheral background — the composed oracle against the reference port, and the env's
host logic.

``tests/flex_periph_oracle.py`` composes the pinned C oracle (no new arithmetic); ``RefPortFlexPeriphEnv`` restates the
same three steps with the port's torchvision calls.  Both run the same seeded episodes (FOV_LOC and FOV_RES actions,
windows of 20..50 and at the frame's edges, unblurred ``rh <= f_h < rw`` and blurred ``rh > f_h``) on stacks in the
reference's dtype: float64 for Atari (atari_env.py:75 and the float64 max of :111-114), float32 for DMC and RGB.  The
env tests run the wrappers on an ``OraclePath`` subclass, with the oracle standing in for the kernels."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from tests.fake_path import OraclePath
from tests.flex_periph_oracle import RefPortFlexPeriphEnv, observe_flexible_peripheral

S = (84, 84)

# (name, frame_stack, channels, dtype, fov, periphery)
CASES = [("atari_k4", 4, 1, np.float64, (30, 30), (20, 20)),
         ("dmc_k3", 3, 1, np.float32, (30, 30), (20, 20)),
         ("dmc_rgb", 3, 3, np.float32, (30, 30), (20, 20)),
         ("odd_fovea", 3, 1, np.float64, (21, 33), (16, 24))]


def _actions(rng, fov, steps):
    """(action, atype) per step: FOV_RES sizes in 20..50 (forced cases first), FOV_LOC targets incl. the frame's edges."""
    forced = [(fov[0], 50), (fov[0] - 1, fov[1] + 9), (min(50, fov[0] + 7), 20), (50, 50), (20, 20)]
    out = []
    for i in range(steps):
        if i % 2 == 0:
            res = forced[(i // 2) % len(forced)] if i < 2 * len(forced) else tuple(int(v) for v in rng.integers(20, 51, 2))
            out.append((np.array(res, np.float64), 1))
        else:
            edge = [(0, 0), (84, 84), (0, 84), (84, 0)]
            loc = edge[(i // 2) % 4] if i % 4 == 1 else tuple(int(v) for v in rng.integers(0, 70, 2))
            out.append((np.array(loc, np.float64), 0))
    return out


@pytest.mark.parametrize("antialias", [True, False])
@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_composed_oracle_matches_the_port_over_episodes(case, antialias):
    _, K, Cc, dtype, fov, per = case
    rng = np.random.default_rng(K * 10 + Cc + 7 * antialias + fov[1])
    port = RefPortFlexPeriphEnv(per, antialias=antialias, frame_stack=K, fov_size=fov, fov_init_loc=(3, 5))
    port.reset_fov()
    P = K * Cc
    loc = port.loc.astype(np.int32).reshape(1, 2).copy()
    res = port.res.astype(np.int32).reshape(1, 2).copy()
    f32 = dtype == np.float32
    bound = 1e-6 if not f32 else (2e-4 if antialias else 1.5e-3)
    worst, blurred = 0.0, 0
    for action, at in _actions(rng, fov, 14):
        stack = rng.integers(0, 256, (P,) + S, dtype=np.uint8)
        port.move(action.copy(), at)
        orc.update_loc(action.reshape(1, 2), loc, obs_size=S, fov_size=fov, atype=np.array([at], np.int32), res=res)
        assert np.array_equal(loc[0], port.loc) and np.array_equal(res[0], port.res)
        full = stack.astype(dtype) if Cc == 1 else stack.reshape(K, Cc, *S).astype(dtype)
        want = port.view(full).reshape(P, *S).astype(np.float64)
        orc.set_antialias(antialias)
        try:
            got = observe_flexible_peripheral(stack[None], np.array([P - 1], np.int32), loc, res, fov, per, use_f32=f32)[0]
        finally:
            orc.set_antialias(True)
        (r, c), (rh, rw) = loc[0], res[0]
        if rh <= fov[0]:   # the unblurred window is pasted as is
            assert np.array_equal(got[:, r:r + rh, c:c + rw], stack[:, r:r + rh, c:c + rw].astype(np.float64))
        blurred += rh > fov[0]
        worst = max(worst, float(np.abs(got - want).max()))
    assert blurred >= 2
    assert worst <= bound, worst


@pytest.mark.parametrize("fov,per", [((30, 30), (20, 20)), ((21, 33), (16, 24))])
def test_oracle_at_fov_res_is_the_fixed_peripheral_view(fov, per):
    rng = np.random.default_rng(11)
    n, K = 12, 4
    ring = rng.integers(0, 256, (n, K) + S, dtype=np.uint8)
    head = rng.integers(0, K, n).astype(np.int32)
    loc = np.stack([rng.integers(0, S[0] - fov[0] + 1, n), rng.integers(0, S[1] - fov[1] + 1, n)], 1).astype(np.int32)
    loc[0], loc[1] = (0, 0), (S[0] - fov[0], S[1] - fov[1])
    res = np.tile(np.array([fov], np.int32), (n, 1))
    for aa in (True, False):
        orc.set_antialias(aa)
        try:
            got = observe_flexible_peripheral(ring, head, loc, res, fov, per)
            want = orc.observe_peripheral(ring, head, loc, fov, per)
        finally:
            orc.set_antialias(True)
        assert np.array_equal(got, want)


# ------------------------------------------------------------------------------------------------ C ABI without a GPU
def test_entry_point_is_exported_and_checks_its_arguments():
    from active_gym_b200 import _lib
    L = _lib.lib()
    assert "agym_observe_flexible_peripheral" in _lib.EXPORTS and _lib.ABI_VERSION == 4
    assert hasattr(C.CDLL(_lib.LIB_PATH), "agym_observe_flexible_peripheral")
    dummy = C.c_void_p(16)
    # NULL plan, then NULL buffers: rejected before any device work
    assert L.agym_observe_flexible_peripheral(None, dummy, dummy, dummy, dummy, None, None, dummy, dummy, dummy, None,
                                              None, 0, None) == -1
    assert L.agym_observe_flexible_peripheral(None, None, None, None, None, None, None, None, None, None, None,
                                              None, 0, None) == -1


# ------------------------------------------------------------------------------------------------ env host logic
class FlexPeriphOraclePath(OraclePath):
    """OraclePath with the peripheral flexible observation: its output shape, the squeeze cache's presence and the
    composed oracle standing in for the kernels."""

    def __init__(self, *a, cache_peripheral=True, **kw):
        super().__init__(*a, cache_peripheral=cache_peripheral, **kw)
        self.pcache = object() if (self.peripheral_res and cache_peripheral) else None

    def out_shape(self, kind, variant, pad=None):
        if kind == "flexible_peripheral":
            return (self.n_envs, self.frame_stack) + self.obs_size
        return super().out_shape(kind, variant, pad)

    def observe_flexible_peripheral(self, action, action_type=None, ctrl=None, out=None, host_out=False, norm_out=None):
        self._update(action, action_type, ctrl, True)
        o = self._oracle(observe_flexible_peripheral, self._ring, self._head, self.loc.numpy(), self.res.numpy(),
                         self.fov_size, self.peripheral_res)
        return self._finish(o, host_out, flexible=True, norm_out=norm_out)


def _env(monkeypatch, n, record=False, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    monkeypatch.setattr("active_gym_b200.atari_env.PipelinedPath", FlexPeriphOraclePath)
    kw = dict(fov_size=(30, 30), fov_init_loc=(3, 4), sensory_action_mode="absolute", peripheral_res=(20, 20), record=record)
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return ag.AtariFlexibleFovealPeripheralEnv(args, num_envs=n, source=SyntheticAtariSource(n, device="cpu")), args


def test_factories_are_exported():
    import active_gym_b200 as ag
    for name in ("AtariFlexibleFovealPeripheralEnv", "DMCFlexibleFovealPeripheralEnv", "FlexibleFovealPeripheralEnv"):
        assert name in ag.__all__ and hasattr(ag, name)
    assert issubclass(ag.FlexibleFovealPeripheralEnv, ag.FlexibleFovealEnv)


def test_env_spaces_info_and_values(monkeypatch):
    n = 5
    env, _ = _env(monkeypatch, n, mask_out=True)
    assert env.mask_out is False and env.variant == "mask" and env._kind == "flexible_peripheral"
    assert env.observation_space.shape == (4,) + S and env.obs_shape == (n, 4) + S
    assert all(k in env.action_space for k in ("motor_action", "sensory_action", "sensory_action_type"))
    obs, info = env.reset()
    assert tuple(obs.shape) == (n, 4) + S and obs.dtype == torch.uint8
    assert {"fov_loc", "fov_res"} <= set(info)
    rng = np.random.default_rng(5)
    for step in range(4):
        at = np.array([1, 0, 1, 0, 1]) if step % 2 == 0 else np.array([0, 1, 0, 1, 0])
        a = np.where(at[:, None] == 1, rng.integers(20, 51, (n, 2)), rng.integers(0, 85, (n, 2))).astype(np.float64)
        obs, _, _, _, info = env.step({"motor_action": np.zeros(n, np.int64), "sensory_action": a, "sensory_action_type": at})
        res = np.asarray(info["fov_res"])
        assert np.array_equal(res[at == 1], a[at == 1].astype(np.int32))
        p = env.path
        want = observe_flexible_peripheral(p._ring, p._head, p.loc.numpy(), p.res.numpy(), (30, 30), (20, 20))
        assert np.array_equal(obs.numpy(), np.clip(np.rint(want), 0, 255).astype(np.uint8))


def test_constructor_rejections(monkeypatch):
    with pytest.raises(ValueError, match="resize_to_fov"):
        _env(monkeypatch, 2, resize_to_fov=True)
    with pytest.raises(ValueError, match="cache"):
        _env(monkeypatch, 2, cache_peripheral=False)
    import active_gym_b200 as ag
    from active_gym_b200.fov_env import FlexibleFovealPeripheralEnv
    env, args = _env(monkeypatch, 2)
    args.peripheral_res = (16, 16)
    with pytest.raises(ValueError, match="peripheral_res"):
        FlexibleFovealPeripheralEnv(env.env, args)
    with pytest.raises(ValueError, match="FOV_RES"):
        env.reset()
        env.step({"motor_action": np.zeros(2, np.int64), "sensory_action": np.array([[90.0, 30.0], [30.0, 30.0]]),
                  "sensory_action_type": np.array([1, 1])})
    assert ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S).mask_out is False


def test_record_wrapper_traces_fov_res(monkeypatch):
    n = 2
    env, _ = _env(monkeypatch, n, record=True)
    env.reset()
    sizes = [(40, 22), (25, 50)]
    for a in sizes:
        env.step({"motor_action": np.zeros(n, np.int64), "sensory_action": np.tile(np.array(a, np.float64), (n, 1)),
                  "sensory_action_type": np.ones(n, np.int64)})
    rec = env.env
    assert rec._with_res
    env.reset()
    ep = rec.episode_record(0)
    assert [tuple(int(v) for v in r) for r in ep["fov_res"]] == [(30, 30)] + sizes


def test_single_env_adapter_returns_full_frames(monkeypatch):
    from active_gym_b200 import SingleEnvAdapter
    env, _ = _env(monkeypatch, 1)
    env = SingleEnvAdapter(env)
    obs, _ = env.reset()
    assert obs.dtype == np.float64 and obs.shape == (4,) + S
    obs, _, _, _, info = env.step({"motor_action": 0, "sensory_action": np.array([47.0, 12.0]), "sensory_action_type": 1})
    assert obs.shape == (4,) + S and np.array_equal(info["fov_res"], [47, 12])
