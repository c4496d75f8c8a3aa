"""CPU: the fixed fovea's memory (``fov_memory``) — the composed oracle against a direct restatement over the reference
port (and the reference itself where a checkout exists), and the env's host logic.

The memory's observation is the pixelwise max of the env's last min(j, M) mask_out observations since its last fovea
reset.  Restated over ``oracle/ref_port.RefPortEnv(variant="mask")``: a deque of the port's float observations, maxed.
``tests/fovea_memory_oracle.py`` must give the same values through ``to_reference_float``, bit for bit, with ragged
resets (hard, zero-filling the stack) and envs that sit a call out (KEEP).  The env tests run the wrappers on
``tests/fake_path.OraclePath``, with the oracle standing in for the kernels."""
import random
from collections import deque

import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from oracle import ref_harness as rh
from oracle.ref_port import RefPortEnv
from tests.fake_path import OraclePath
from tests.fovea_memory_oracle import APPLY, KEEP, RESET, MemoryOracle
from tests.test_oracle_vs_reference import REFS, _Reference

S, FA, FH, IDLE = (84, 84), 1, 4, 8
K = 3


def _schedule(rng, n, T):
    """Per call and env: 'reset' (hard), 'step' or 'idle'; every env starts with a reset, later resets are ragged."""
    ev = [["reset"] * n]
    for _ in range(T):
        ev.append([str(rng.choice(["step"] * 6 + ["reset", "idle"])) for _ in range(n)])
    return ev


def _actions(rng, mode, n, T):
    lo, hi = (-14, 15) if mode == "relative" else (-6, 64)
    return rng.integers(lo, hi, (T + 1, n, 2)).astype(np.float64)


def _run_env(ref, e, screens, events, actions, mode, fov, init):
    """One env's observations per call (None when it sat the call out) and the index of the screen each call used."""
    kw = dict(fov_size=fov, fov_init_loc=init)
    out, t = [], 0
    if ref == "reference":
        _, _, dmc = rh.load_reference()
        script = rh.ScreenScript(screens)
        rh.ScreenScript.current = script
        akw = dict(sensory_action_mode=mode, frame_stack=K, action_repeat=2, mask_out=True, **kw)
        if mode == "relative":
            akw["sensory_action_space"] = (-10.0, 10.0)
        env = _Reference(dmc.DMCFixedFovealEnv(dmc.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S,
                                                              **akw)), script)
        random.seed(e)
        for c, ev in enumerate(events):
            if ev[e] == "idle":
                out.append((None, None))
                continue
            if ev[e] == "reset":
                obs, info, idx = env.reset()
            else:
                obs, info, idx = env.step({"motor_action": np.zeros(2, np.float32), "sensory_action": actions[c, e]})
            out.append((np.asarray(obs, np.float64), idx[-1]))
        return out
    env = RefPortEnv(kind="dmc", wrapper="fixed", frame_stack=K, obs_size=S, mode=mode, lo=-10.0, hi=10.0, variant="mask", **kw)
    for c, ev in enumerate(events):
        if ev[e] == "idle":
            out.append((None, None))
            continue
        obs = env.reset(screens[t], hard=True) if ev[e] == "reset" else env.step(screens[t], None, actions[c, e])
        out.append((np.asarray(obs, np.float64), t))
        t += 1
    return out


@pytest.mark.parametrize("ref", REFS)
@pytest.mark.parametrize("mode", ["relative", "absolute"])
@pytest.mark.parametrize("depth", [1, 3, 8])
def test_composed_oracle_equals_restatement_over_the_port(ref, mode, depth):
    rng = np.random.default_rng(depth * 7 + (mode == "relative"))
    n, T, fov, init = 4, 24, (30, 30), (11, 23)
    screens = rng.integers(0, 256, (80, 84, 84, 3), dtype=np.uint8)
    events = _schedule(rng, n, T)
    actions = _actions(rng, mode, n, T)
    runs = [_run_env(ref, e, screens, events, actions, mode, fov, init) for e in range(n)]
    # the restatement: a deque of the port's observations per env, maxed
    dq = [deque(maxlen=depth) for _ in range(n)]
    # the composed oracle over the batched C oracle
    ring, head = orc.new_state(n, K, S)
    loc = np.zeros((n, 2), np.int32)
    mem = MemoryOracle(n, depth)
    prev = None
    for c, ev in enumerate(events):
        flags = np.array([FA | FH if x == "reset" else (IDLE if x == "idle" else FA) for x in ev], np.uint8)
        frames = np.zeros((n,) + S + (3,), np.uint8)
        for e in range(n):
            if runs[e][c][1] is not None:
                frames[e] = screens[runs[e][c][1]]
        orc.ingest_dmc(frames, flags, ring, head)
        ctrl = np.array([RESET if x == "reset" else (KEEP if x == "idle" else APPLY) for x in ev], np.uint8)
        new = loc.copy()
        orc.update_loc(actions[c], new, obs_size=S, fov_size=fov, relative=mode == "relative", lo=-10.0, hi=10.0)
        loc[ctrl == APPLY] = new[ctrl == APPLY]
        loc[ctrl == RESET] = init
        got = mem.observe(ring, head, loc, fov, ctrl)
        for e in range(n):
            obs = runs[e][c][0]
            if obs is None:
                assert np.array_equal(got[e], prev[e]), (c, e)   # KEEP: the observation is unchanged
                continue
            if ev[e] == "reset":
                dq[e].clear()
            dq[e].append(obs)
            want = np.maximum.reduce(list(dq[e]))
            assert np.array_equal(orc.to_reference_float(got[e]), want), (c, e)
        assert np.array_equal(mem.count(), [len(q) for q in dq])
        prev = got


def test_depth_one_is_mask_out():
    rng = np.random.default_rng(5)
    n, fov = 6, (21, 33)
    ring = rng.integers(0, 256, (n, 4) + S, dtype=np.uint8)
    head = rng.integers(0, 4, n).astype(np.int32)
    mem = MemoryOracle(n, 1)
    for _ in range(3):
        loc = np.stack([rng.integers(0, 84 - fov[0] + 1, n), rng.integers(0, 84 - fov[1] + 1, n)], 1).astype(np.int32)
        assert np.array_equal(mem.observe(ring, head, loc, fov), orc.observe_fixed(ring, head, loc, fov, variant="mask"))


# ------------------------------------------------------------------------------------------------ env host logic
class MemoryOraclePath(OraclePath):
    """OraclePath with the fovea memory: the composed oracle standing in for ``observe_fixed_memory``."""

    def __init__(self, *a, fov_memory=0, **kw):
        super().__init__(*a, **kw)
        self.fov_memory = int(fov_memory)
        self._mem = MemoryOracle(self.n_envs, max(self.fov_memory, 1))
        self.mem_loc = torch.zeros((self.n_envs, max(self.fov_memory, 1), 2), dtype=torch.int32)
        self.mem_state = torch.zeros((self.n_envs, 2), dtype=torch.int32)

    def observe_fixed_memory(self, action, ctrl=None, out=None, host_out=False, norm_out=None):
        self._update(action, None, ctrl, False)
        c = np.full(self.n_envs, RESET, np.uint8) if isinstance(ctrl, str) else \
            (np.full(self.n_envs, APPLY, np.uint8) if ctrl is None else np.asarray(ctrl, np.uint8))
        o = self._mem.observe(self._ring, self._head, self.loc.numpy(), self.fov_size, c)
        self.mem_state[:, 1] = torch.from_numpy(self._mem.count())
        return self._finish(o, host_out, norm_out=norm_out)


def _env(monkeypatch, n, wrapper="AtariFixedFovealEnv", **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    monkeypatch.setattr("active_gym_b200.atari_env.PipelinedPath", MemoryOraclePath)
    kw = dict(fov_size=(30, 30), fov_init_loc=(3, 4), sensory_action_mode="absolute", mask_out=True, fov_memory=3)
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return getattr(ag, wrapper)(args, num_envs=n, source=SyntheticAtariSource(n, device="cpu"))


def test_args_default_to_no_memory():
    import active_gym_b200 as ag
    assert ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S).fov_memory == 0
    assert ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S).fov_memory == 0


def _step(env, n, a):
    return env.step({"motor_action": np.zeros(n, np.int64), "sensory_action": a})


def test_env_shapes_spaces_and_values(monkeypatch):
    n = 5
    env = _env(monkeypatch, n)
    assert env.variant == "mask" and env.fov_memory == 3
    assert env.observation_space.shape == (4, 84, 84) and env.obs_shape == (n, 4, 84, 84)
    obs, info = env.reset()
    assert tuple(obs.shape) == (n, 4, 84, 84) and obs.dtype == torch.uint8
    assert np.array_equal(env.fov_memory_count.numpy(), np.ones(n))
    assert tuple(env.fov_memory_loc.shape) == (n, 3, 2)
    rng = np.random.default_rng(5)
    masks = deque(maxlen=3)
    p = env.path
    masks.append(orc.observe_fixed(p._ring, p._head, p.loc.numpy(), (30, 30), variant="mask"))
    for step in range(5):
        obs, _, _, _, info = _step(env, n, rng.integers(0, 55, (n, 2)).astype(np.float64))
        masks.append(orc.observe_fixed(p._ring, p._head, p.loc.numpy(), (30, 30), variant="mask"))
        assert np.array_equal(obs.numpy(), np.maximum.reduce(list(masks)))
        assert np.array_equal(env.fov_memory_count.numpy(), np.full(n, min(step + 2, 3)))
        assert "fov_loc" in info and set(info) == {"fov_loc", "raw_reward", "reward", "ep_len"}


@pytest.mark.parametrize("extra", [{"fov_memory": 17}, {"fov_memory": -1}, {"mask_out": False}, {"mask_out": False, "resize_to_full": True}])
def test_invalid_memory_raises(monkeypatch, extra):
    with pytest.raises(ValueError, match="fov_memory"):
        _env(monkeypatch, 2, **extra)


@pytest.mark.parametrize("wrapper,extra", [("AtariFlexibleFovealEnv", {}),
                                           ("AtariFixedFovealPeripheralEnv", {"peripheral_res": (20, 20)}),
                                           ("AtariFlexibleFovealPeripheralEnv", {"peripheral_res": (20, 20)})])
def test_other_wrappers_reject_memory(monkeypatch, wrapper, extra):
    with pytest.raises(ValueError, match="fov_memory"):
        _env(monkeypatch, 2, wrapper=wrapper, **extra)


def test_masked_reset_clears_only_the_selected_envs(monkeypatch):
    n = 6
    env = _env(monkeypatch, n, fov_memory=4)
    env.reset()
    rng = np.random.default_rng(9)
    for _ in range(4):
        obs, *_ = _step(env, n, rng.integers(0, 55, (n, 2)).astype(np.float64))
    assert np.array_equal(env.fov_memory_count.numpy(), np.full(n, 4))
    mask = np.array([True, False, True, False, False, True])
    obs2, _ = env.reset(mask=mask)
    assert np.array_equal(env.fov_memory_count.numpy(), np.where(mask, 1, 4))
    assert np.array_equal(obs2[~torch.from_numpy(mask)].numpy(), obs[~torch.from_numpy(mask)].numpy())
    p = env.path
    want = orc.observe_fixed(p._ring, p._head, p.loc.numpy(), (30, 30), variant="mask")
    assert np.array_equal(obs2[torch.from_numpy(mask)].numpy(), want[mask])


def test_single_env_adapter(monkeypatch):
    from active_gym_b200 import SingleEnvAdapter
    env = SingleEnvAdapter(_env(monkeypatch, 1))
    assert env.observation_space.shape == (4, 84, 84)
    obs, _ = env.reset()
    assert obs.dtype == np.float64 and obs.shape == (4, 84, 84)
    seen = obs
    for a in ([40.0, 5.0], [2.0, 50.0], [50.0, 50.0]):
        obs, _, _, _, info = env.step({"motor_action": 0, "sensory_action": np.array(a)})
        assert obs.dtype == np.float64 and obs.shape == (4, 84, 84)
        assert (obs >= 0).all() and obs.max() <= 1.0
        assert info["fov_loc"].tolist() == [int(v) for v in a]
    assert (seen >= 0).all()
