"""CPU: the fixed fovea's memory merged by pasting (``fov_memory_merge="paste"``) — the composed oracle against a direct
restatement over the reference port (and the reference itself where a checkout exists), and the env's host logic.

Paste lays the env's held windows over a background from the oldest to the newest, so at each pixel the newest window
that covers it wins.  Restated over ``oracle/ref_port.RefPortEnv``: the wrapper's observation (the peripheral view, or
mask_out for the zero background) plus a deque of the windows it showed, pasted over it.
``tests/memory_paste_oracle.py`` must give the same values: pasted pixels bit for bit through ``to_reference_float``,
the periphery within the tolerance the peripheral live test uses, with ragged hard resets, envs that sit a call out
(KEEP) and masked resets.  The env tests run the wrappers on ``tests/fake_path.OraclePath``, with the oracle standing in
for the kernels."""
import random
from collections import deque

import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from oracle import ref_harness as rh
from oracle.ref_port import RefPortEnv
from tests.fake_path import OraclePath
from tests.fovea_memory_oracle import MemoryOracle
from tests.memory_paste_oracle import APPLY, KEEP, RESET, PasteOracle
from tests.test_oracle_vs_reference import REFS, _Reference

S, FA, FH, IDLE = (84, 84), 1, 4, 8
K, PER = 3, (20, 20)


def _schedule(rng, n, T):
    """Per call and env: 'reset' (hard), 'step', 'idle' (KEEP, no frame) or 'soft' (a masked reset: the fovea resets,
    the frame stack does not); every env starts with a hard reset, later events are ragged."""
    ev = [["reset"] * n]
    for _ in range(T):
        ev.append([str(rng.choice(["step"] * 6 + ["reset", "idle", "soft"])) for _ in range(n)])
    return ev


def _run_env(ref, e, screens, events, actions, mode, fov, init, background):
    """One env's (observation, window loc, screen index) per call; (None, None, None) when it sat the call out."""
    kw = dict(fov_size=fov, fov_init_loc=init)
    periph = background == "periphery"
    out, t = [], 0
    if ref == "reference":
        _, _, dmc = rh.load_reference()
        script = rh.ScreenScript(screens)
        rh.ScreenScript.current = script
        akw = dict(sensory_action_mode=mode, frame_stack=K, action_repeat=2, mask_out=not periph, **kw)
        if periph:
            akw["peripheral_res"] = PER
        if mode == "relative":
            akw["sensory_action_space"] = (-10.0, 10.0)
        cls = dmc.DMCFixedFovealPeripheralEnv if periph else dmc.DMCFixedFovealEnv
        env = _Reference(cls(dmc.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, **akw)), script)
        random.seed(e)
        for c, ev in enumerate(events):
            if ev[e] == "idle":
                out.append((None, None, None))
                continue
            if ev[e] in ("reset", "soft"):
                obs, info, idx = env.reset()
            else:
                obs, info, idx = env.step({"motor_action": np.zeros(2, np.float32), "sensory_action": actions[c, e]})
            out.append((np.asarray(obs, np.float64), tuple(int(v) for v in info["fov_loc"]), idx[-1]))
        return out
    env = RefPortEnv(kind="dmc", wrapper="peripheral" if periph else "fixed", frame_stack=K, obs_size=S, mode=mode, lo=-10.0,
                     hi=10.0, variant="mask", peripheral_res=PER if periph else None, **kw)
    for c, ev in enumerate(events):
        if ev[e] == "idle":
            out.append((None, None, None))
            continue
        if ev[e] in ("reset", "soft"):
            obs = env.reset(screens[t], hard=ev[e] == "reset")
        else:
            obs = env.step(screens[t], None, actions[c, e])
        out.append((np.asarray(obs, np.float64), (int(env.loc[0]), int(env.loc[1])), t))
        t += 1
    return out


@pytest.mark.parametrize("ref", REFS)
@pytest.mark.parametrize("mode", ["relative", "absolute"])
@pytest.mark.parametrize("depth", [1, 3, 8])
@pytest.mark.parametrize("background", ["zero", "periphery"])
def test_composed_oracle_equals_restatement_over_the_port(ref, mode, depth, background):
    rng = np.random.default_rng(depth * 7 + (mode == "relative") + 100 * (background == "zero"))
    n, T, fov, init = 4, 24, (30, 30), (11, 23)
    fh, fw = fov
    screens = rng.integers(0, 256, (80, 84, 84, 3), dtype=np.uint8)
    events = _schedule(rng, n, T)
    if ref == "reference":   # the reference has no masked reset: every reset is a hard one
        events = [["reset" if x == "soft" else x for x in ev] for ev in events]
    actions = rng.integers(-14, 15, (T + 1, n, 2)).astype(np.float64) if mode == "relative" else \
        rng.integers(-6, 64, (T + 1, n, 2)).astype(np.float64)
    runs = [_run_env(ref, e, screens, events, actions, mode, fov, init, background) for e in range(n)]
    per = PER if background == "periphery" else None
    dq = [deque(maxlen=depth) for _ in range(n)]   # the restatement: the windows each env showed
    ring, head = orc.new_state(n, K, S)
    loc = np.zeros((n, 2), np.int32)
    mem = PasteOracle(n, depth)
    prev = None
    for c, ev in enumerate(events):
        flags = np.array([FA | FH if x == "reset" else (IDLE if x == "idle" else FA) for x in ev], np.uint8)
        frames = np.zeros((n,) + S + (3,), np.uint8)
        for e in range(n):
            if runs[e][c][2] is not None:
                frames[e] = screens[runs[e][c][2]]
        orc.ingest_dmc(frames, flags, ring, head)
        ctrl = np.array([RESET if x in ("reset", "soft") else (KEEP if x == "idle" else APPLY) for x in ev], np.uint8)
        new = loc.copy()
        orc.update_loc(actions[c], new, obs_size=S, fov_size=fov, relative=mode == "relative", lo=-10.0, hi=10.0)
        loc[ctrl == APPLY] = new[ctrl == APPLY]
        loc[ctrl == RESET] = init
        got = mem.observe(ring, head, loc, fov, ctrl, peripheral_res=per)
        pasted = mem.pasted(S, fov)
        for e in range(n):
            obs, wloc, _ = runs[e][c]
            if obs is None:
                assert np.array_equal(got[e], prev[e]), (c, e)   # KEEP on an idle env: the observation is unchanged
                continue
            assert wloc == tuple(loc[e]), (c, e)
            r, cc = wloc
            if ev[e] in ("reset", "soft"):
                dq[e].clear()
            dq[e].append((obs[:, r:r + fh, cc:cc + fw].copy(), wloc))
            want = obs.copy()
            for w, (wr, wc) in dq[e]:
                want[:, wr:wr + fh, wc:wc + fw] = w
            m = np.broadcast_to(pasted[e], got[e].shape)
            assert np.array_equal(orc.to_reference_float(got[e][m].astype(np.uint8)), want[m]), (c, e)
            if per is None:
                assert np.array_equal(orc.to_reference_float(got[e].astype(np.uint8)), want), (c, e)
            else:
                assert np.abs(got[e] - want * 255.0).max() <= 1e-4, (c, e)
        assert np.array_equal(mem.count(), [len(q) for q in dq])
        prev = got


def _random_state(rng, n, P=4):
    ring = rng.integers(0, 256, (n, P) + S, dtype=np.uint8)
    head = rng.integers(0, P, n).astype(np.int32)
    return ring, head


def _random_loc(rng, n, fov):
    return np.stack([rng.integers(0, 84 - fov[0] + 1, n), rng.integers(0, 84 - fov[1] + 1, n)], 1).astype(np.int32)


@pytest.mark.parametrize("fov", [(30, 30), (21, 33)])
def test_depth_one_is_mask_out_and_the_peripheral_view(fov):
    rng = np.random.default_rng(5)
    n = 6
    ring, head = _random_state(rng, n)
    zero, periph = PasteOracle(n, 1), PasteOracle(n, 1)
    for _ in range(3):
        loc = _random_loc(rng, n, fov)
        assert np.array_equal(zero.observe(ring, head, loc, fov), orc.observe_fixed(ring, head, loc, fov, variant="mask"))
        assert np.array_equal(periph.observe(ring, head, loc, fov, peripheral_res=PER),
                              orc.observe_peripheral(ring, head, loc, fov, PER))


def test_zero_background_with_disjoint_windows_is_the_max_memory():
    """Four windows in the four quadrants never overlap: paste and max agree (values of the same pushes)."""
    rng = np.random.default_rng(7)
    n, fov = 5, (30, 30)
    ring, head = _random_state(rng, n)
    paste, mx = PasteOracle(n, 4), MemoryOracle(n, 4)
    corners = [(0, 0), (0, 54), (54, 0), (54, 54), (2, 3)]
    for i, (r, c) in enumerate(corners[:4]):
        ring, _ = _random_state(rng, n)
        loc = np.tile(np.array([[r, c]], np.int32), (n, 1))
        ctrl = np.full(n, RESET if i == 0 else APPLY, np.uint8)
        assert np.array_equal(paste.observe(ring, head, loc, fov, ctrl), mx.observe(ring, head, loc, fov, ctrl)), i


def test_newest_window_wins_where_windows_overlap():
    n, fov = 1, (30, 30)
    ring = np.zeros((n, 4) + S, np.uint8)
    head = np.zeros(n, np.int32)
    mem = PasteOracle(n, 3)
    ring[:] = 200
    mem.observe(ring, head, np.array([[10, 10]], np.int32), fov, np.array([RESET], np.uint8))
    ring[:] = 7
    out = mem.observe(ring, head, np.array([[20, 20]], np.int32), fov, np.array([APPLY], np.uint8))
    assert (out[0, :, 20:50, 20:50] == 7).all()           # the newest window over the older one
    assert (out[0, :, 10:20, 10:40] == 200).all()         # the older window where only it reaches
    assert (out[0, :, 60:, :] == 0).all()


# ------------------------------------------------------------------------------------------------ env host logic
class PasteOraclePath(OraclePath):
    """OraclePath with the fovea memory and both merges: the composed oracles standing in for ``observe_fixed_memory``
    and ``observe_memory_paste``."""

    def __init__(self, *a, fov_memory=0, cache_peripheral=True, **kw):
        super().__init__(*a, cache_peripheral=cache_peripheral, **kw)
        self.fov_memory = int(fov_memory)
        self.pcache = object() if (self.peripheral_res and cache_peripheral) else None
        self._max = MemoryOracle(self.n_envs, max(self.fov_memory, 1))
        self._paste = PasteOracle(self.n_envs, max(self.fov_memory, 1))
        self.mem_loc = torch.zeros((self.n_envs, max(self.fov_memory, 1), 2), dtype=torch.int32)
        self.mem_state = torch.zeros((self.n_envs, 2), dtype=torch.int32)
        self.backgrounds = []

    def _ctrl_np(self, ctrl):
        return np.full(self.n_envs, RESET, np.uint8) if isinstance(ctrl, str) else \
            (np.full(self.n_envs, APPLY, np.uint8) if ctrl is None else np.asarray(ctrl, np.uint8))

    def observe_fixed_memory(self, action, ctrl=None, out=None, host_out=False, norm_out=None):
        self._update(action, None, ctrl, False)
        o = self._max.observe(self._ring, self._head, self.loc.numpy(), self.fov_size, self._ctrl_np(ctrl))
        self.mem_state[:, 1] = torch.from_numpy(self._max.count())
        return self._finish(o, host_out, norm_out=norm_out)

    def observe_memory_paste(self, action, ctrl=None, background="zero", out=None, host_out=False, norm_out=None):
        self.backgrounds.append(background)
        self._update(action, None, ctrl, False)
        per = self.peripheral_res if background == "periphery" else None
        o = self._oracle(self._paste.observe, self._ring, self._head, self.loc.numpy(), self.fov_size, self._ctrl_np(ctrl),
                         peripheral_res=per)
        self.mem_state[:, 1] = torch.from_numpy(self._paste.count())
        return self._finish(o, host_out, norm_out=norm_out)


def _env(monkeypatch, n, wrapper="AtariFixedFovealPeripheralEnv", **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    monkeypatch.setattr("active_gym_b200.atari_env.PipelinedPath", PasteOraclePath)
    kw = dict(fov_size=(30, 30), fov_init_loc=(3, 4), sensory_action_mode="absolute", fov_memory=3,
              fov_memory_merge="paste", peripheral_res=PER)
    if wrapper == "AtariFixedFovealEnv":
        kw["mask_out"] = True
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return getattr(ag, wrapper)(args, num_envs=n, source=SyntheticAtariSource(n, device="cpu"))


def _step(env, n, a):
    return env.step({"motor_action": np.zeros(n, np.int64), "sensory_action": a})


def test_args_default_to_the_max_merge():
    import active_gym_b200 as ag
    assert ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S).fov_memory_merge == "max"
    assert ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S).fov_memory_merge == "max"


@pytest.mark.parametrize("wrapper,mask_out", [("AtariFixedFovealEnv", True), ("AtariFixedFovealPeripheralEnv", True),
                                              ("AtariFixedFovealPeripheralEnv", False)])
def test_env_pastes_the_memory(monkeypatch, wrapper, mask_out):
    """Values of both wrappers against the composed oracle; the peripheral env ignores ``mask_out``."""
    n = 5
    periph = wrapper == "AtariFixedFovealPeripheralEnv"
    env = _env(monkeypatch, n, wrapper=wrapper, mask_out=mask_out)
    assert env.fov_memory == 3 and env.fov_memory_merge == "paste"
    assert env.observation_space.shape == (4, 84, 84) and env.obs_shape == (n, 4, 84, 84)
    p = env.path
    want = PasteOracle(n, 3)
    per = PER if periph else None
    obs, info = env.reset()
    assert tuple(obs.shape) == (n, 4, 84, 84) and obs.dtype == torch.uint8
    w = want.observe(p._ring, p._head, p.loc.numpy(), (30, 30), np.full(n, RESET, np.uint8), peripheral_res=per)
    assert np.array_equal(obs.numpy(), np.clip(np.rint(w), 0, 255).astype(np.uint8))
    rng = np.random.default_rng(5)
    for step in range(5):
        obs, _, _, _, info = _step(env, n, rng.integers(0, 55, (n, 2)).astype(np.float64))
        w = want.observe(p._ring, p._head, p.loc.numpy(), (30, 30), None, peripheral_res=per)
        assert np.array_equal(obs.numpy(), np.clip(np.rint(w), 0, 255).astype(np.uint8)), step
        assert np.array_equal(env.fov_memory_count.numpy(), np.full(n, min(step + 2, 3)))
        assert tuple(env.fov_memory_loc.shape) == (n, 3, 2)
        assert "fov_loc" in info
    assert set(p.backgrounds) == {"periphery" if periph else "zero"}


@pytest.mark.parametrize("value", ["min", "MAX", None, 1])
@pytest.mark.parametrize("wrapper", ["AtariFixedFovealEnv", "AtariFixedFovealPeripheralEnv"])
def test_bad_merge_values_raise(monkeypatch, wrapper, value):
    with pytest.raises(ValueError, match="fov_memory_merge"):
        _env(monkeypatch, 2, wrapper=wrapper, fov_memory_merge=value)


def test_max_on_the_peripheral_env_names_paste(monkeypatch):
    with pytest.raises(ValueError, match='fov_memory.*fov_memory_merge="paste"'):
        _env(monkeypatch, 2, fov_memory_merge="max")


def test_peripheral_paste_needs_the_squeeze_cache(monkeypatch):
    with pytest.raises(ValueError, match="cache_peripheral"):
        _env(monkeypatch, 2, cache_peripheral=False)


@pytest.mark.parametrize("extra", [{"mask_out": False}, {"mask_out": False, "resize_to_full": True}, {"fov_memory": 17}])
def test_fixed_paste_keeps_the_memory_rules(monkeypatch, extra):
    with pytest.raises(ValueError, match="fov_memory"):
        _env(monkeypatch, 2, wrapper="AtariFixedFovealEnv", **extra)


@pytest.mark.parametrize("wrapper", ["AtariFlexibleFovealEnv", "AtariFlexibleFovealPeripheralEnv"])
def test_flexible_wrappers_still_reject_memory(monkeypatch, wrapper):
    with pytest.raises(ValueError, match="fov_memory"):
        _env(monkeypatch, 2, wrapper=wrapper)


def test_merge_has_no_effect_without_memory(monkeypatch):
    env = _env(monkeypatch, 2, fov_memory=0)
    env.reset()
    assert env.fov_memory_count is None and env.path.backgrounds == []


@pytest.mark.parametrize("wrapper", ["AtariFixedFovealEnv", "AtariFixedFovealPeripheralEnv"])
def test_masked_reset_clears_only_the_selected_envs(monkeypatch, wrapper):
    n = 6
    env = _env(monkeypatch, n, wrapper=wrapper, fov_memory=4)
    env.reset()
    rng = np.random.default_rng(9)
    for _ in range(4):
        obs, *_ = _step(env, n, rng.integers(0, 55, (n, 2)).astype(np.float64))
    assert np.array_equal(env.fov_memory_count.numpy(), np.full(n, 4))
    mask = np.array([True, False, True, False, False, True])
    obs2, _ = env.reset(mask=mask)
    assert np.array_equal(env.fov_memory_count.numpy(), np.where(mask, 1, 4))
    keep = ~torch.from_numpy(mask)
    assert np.array_equal(obs2[keep].numpy(), obs[keep].numpy())
    p = env.path
    if wrapper == "AtariFixedFovealEnv":
        want = orc.observe_fixed(p._ring, p._head, p.loc.numpy(), (30, 30), variant="mask")
    else:
        want = np.clip(np.rint(orc.observe_peripheral(p._ring, p._head, p.loc.numpy(), (30, 30), PER)), 0, 255).astype(np.uint8)
    assert np.array_equal(obs2[torch.from_numpy(mask)].numpy(), want[mask])


def test_single_env_adapter(monkeypatch):
    from active_gym_b200 import SingleEnvAdapter
    env = SingleEnvAdapter(_env(monkeypatch, 1))
    assert env.observation_space.shape == (4, 84, 84)
    obs, _ = env.reset()
    assert obs.dtype == np.float64 and obs.shape == (4, 84, 84)
    for a in ([40.0, 5.0], [2.0, 50.0], [50.0, 50.0]):
        obs, _, _, _, info = env.step({"motor_action": 0, "sensory_action": np.array(a)})
        assert obs.dtype == np.float64 and obs.shape == (4, 84, 84)
        assert (obs >= 0).all() and obs.max() <= 1.0
        assert info["fov_loc"].tolist() == [int(v) for v in a]
