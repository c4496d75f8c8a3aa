"""CPU: the flexible fovea's glimpse (``resize_to_fov``) — the composed oracle against torchvision, and the env's host logic.

The glimpse is, per plane, torchvision's ``Resize(fov_size)`` of the unblurred window ``full_state[..., r:r+rh, c:c+rw]``
(fov_env.py:248,284-285).  ``tests/glimpse_oracle.py`` must equal it in the reference's dtype: float64 for
Atari (atari_env.py:75 hands the wrappers float64 stacks) and float32 for DMC's steady state (dmc_env.py:183).  The env
tests run the wrappers on ``tests/fake_path.OraclePath``, with the oracle standing in for the kernels."""
import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from tests.fake_path import OraclePath
from tests.glimpse_oracle import observe_glimpse

S = (84, 84)
FOVS = [(30, 30), (21, 33), (50, 28)]


def _windows(fov, rng, m=24):
    """Window sizes over [1, S]^2 with the corners and res == fov always included."""
    fixed = [(1, 1), (1, 84), (84, 1), (84, 84), tuple(fov), (fov[0] + 1, fov[1] - 1)]
    return fixed + [tuple(int(v) for v in rng.integers(1, 85, 2)) for _ in range(m)]


def _torchvision_resize(window, fov, antialias, dtype):
    from torchvision.transforms import Resize
    t = torch.from_numpy(window.astype(dtype))[None]
    return Resize(fov, antialias=antialias)(t)[0].numpy().astype(np.float64)


def _oracle(ring, loc, res, fov, antialias, use_f32):
    orc.set_antialias(antialias)
    try:
        return observe_glimpse(ring, np.full(len(loc), ring.shape[1] - 1, np.int32), loc, res, fov, use_f32=use_f32)
    finally:
        orc.set_antialias(True)


# bounds in LSB: float64 agrees to rounding; float32 within SURVEY A3's 8.9e-5 LSB fp32-vs-fp64 spread, with margin.
# Plain bilinear (antialias=False) in float32 gets 1.5e-3: ATen's fp32 upsample kernel itself differs from its fp64
# evaluation by up to 1.0e-3 LSB on these windows (e.g. 20 x 77 -> 30 x 30), so no fp32 restatement is closer than that.
@pytest.mark.parametrize("fov", FOVS)
@pytest.mark.parametrize("antialias", [True, False])
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
def test_oracle_glimpse_is_torchvision_resize_of_the_window(fov, antialias, dtype):
    bound = 1e-6 if dtype == np.float64 else (2e-4 if antialias else 1.5e-3)
    rng = np.random.default_rng(sum(fov) + 2 * antialias + (dtype == np.float32))
    wins = _windows(fov, rng)
    n, K = len(wins), 2
    ring = rng.integers(0, 256, (n, K) + S, dtype=np.uint8)
    res = np.array(wins, np.int32)
    loc = np.stack([rng.integers(0, S[0] - res[:, 0] + 1), rng.integers(0, S[1] - res[:, 1] + 1)], 1).astype(np.int32)
    got = _oracle(ring, loc, res, fov, antialias, use_f32=dtype == np.float32)
    assert got.shape == (n, K) + fov
    worst = 0.0
    for e in range(n):
        (r, c), (rh, rw) = loc[e], res[e]
        for k in range(K):   # head = K-1: plane k is slot k
            want = _torchvision_resize(ring[e, k, r:r + rh, c:c + rw], fov, antialias, dtype)
            worst = max(worst, float(np.abs(got[e, k] - want).max()))
    assert worst <= bound, worst


def test_oracle_glimpse_at_fov_res_is_the_crop():
    rng = np.random.default_rng(3)
    n, K, fov = 20, 3, (21, 33)
    ring = rng.integers(0, 256, (n, K) + S, dtype=np.uint8)
    loc = np.stack([rng.integers(0, S[0] - fov[0] + 1, n), rng.integers(0, S[1] - fov[1] + 1, n)], 1).astype(np.int32)
    res = np.tile(np.array([fov], np.int32), (n, 1))
    head = np.full(n, K - 1, np.int32)
    for aa in (True, False):
        orc.set_antialias(aa)
        try:
            g = observe_glimpse(ring, head, loc, res, fov)
        finally:
            orc.set_antialias(True)
        assert np.array_equal(g, orc.observe_fixed(ring, head, loc, fov, variant="crop").astype(np.float64))


def test_abi_constant_mirrors_the_header():
    import os
    from active_gym_b200 import _lib
    from active_gym_b200.engine import VARIANTS
    hdr = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "include", "agym_b200.h")).read()
    assert "#define AGYM_OUT_RESIZE_FOV 3" in hdr and "#define AGYM_ABI_VERSION 4" in hdr
    assert _lib.OUT_RESIZE_FOV == 3 and VARIANTS["resize_fov"] == 3 and _lib.ABI_VERSION == 4


# ------------------------------------------------------------------------------------------------ env host logic
class GlimpseOraclePath(OraclePath):
    """OraclePath with the glimpse: its output shape (the product's ObservationPath.out_shape) and the composed oracle
    standing in for the kernels."""

    def out_shape(self, kind, variant, pad=None):
        if kind == "flexible" and variant == "resize_fov":
            return (self.n_envs, self.frame_stack) + self.fov_size
        return super().out_shape(kind, variant, pad)

    def observe_flexible(self, action, action_type=None, variant="mask", ctrl=None, pad=None, out=None, host_out=False, norm_out=None):
        if variant != "resize_fov":
            return super().observe_flexible(action, action_type, variant, ctrl, pad, out, host_out, norm_out)
        self._update(action, action_type, ctrl, True)
        o = self._oracle(observe_glimpse, self._ring, self._head, self.loc.numpy(), self.res.numpy(), self.fov_size)
        return self._finish(o, host_out, flexible=True, norm_out=norm_out)


def _env(monkeypatch, n, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    monkeypatch.setattr("active_gym_b200.atari_env.PipelinedPath", GlimpseOraclePath)
    kw = dict(fov_size=(30, 30), fov_init_loc=(3, 4), sensory_action_mode="absolute", resize_to_fov=True)
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return ag.AtariFlexibleFovealEnv(args, num_envs=n, source=SyntheticAtariSource(n, device="cpu"))


def test_args_default_to_no_glimpse():
    import active_gym_b200 as ag
    assert ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S).resize_to_fov is False
    assert ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S).resize_to_fov is False


@pytest.mark.parametrize("conflict", [{"mask_out": True}, {"resize_to_full": True}])
def test_glimpse_excludes_mask_out_and_resize_to_full(monkeypatch, conflict):
    with pytest.raises(ValueError, match="resize_to_fov"):
        _env(monkeypatch, 2, **conflict)


def test_env_shapes_spaces_and_values(monkeypatch):
    n = 5
    env = _env(monkeypatch, n)
    assert env.variant == "resize_fov"
    assert env.observation_space.shape == (4, 30, 30) and env.obs_shape == (n, 4, 30, 30)
    obs, info = env.reset()
    assert tuple(obs.shape) == (n, 4, 30, 30) and obs.dtype == torch.uint8
    assert np.array_equal(np.asarray(info["fov_res"]), np.tile([30, 30], (n, 1)))
    rng = np.random.default_rng(5)
    for step in range(3):
        at = np.array([1, 0, 1, 0, 1])
        a = np.where(at[:, None] == 1, rng.integers(1, 85, (n, 2)), rng.integers(0, 60, (n, 2))).astype(np.float64)
        obs, _, _, _, info = env.step({"motor_action": np.zeros(n, np.int64), "sensory_action": a, "sensory_action_type": at})
        assert tuple(obs.shape) == (n, 4, 30, 30)
        res = np.asarray(info["fov_res"])
        assert np.array_equal(res[at == 1], a[at == 1].astype(np.int32))
        p = env.path
        want = observe_glimpse(p._ring, p._head, p.loc.numpy(), p.res.numpy(), (30, 30))
        assert np.array_equal(obs.numpy(), np.clip(np.rint(want), 0, 255).astype(np.uint8))


def test_single_env_adapter_keeps_the_fixed_shape(monkeypatch):
    from active_gym_b200 import SingleEnvAdapter
    env = SingleEnvAdapter(_env(monkeypatch, 1))
    assert env.observation_space.shape == (4, 30, 30)
    obs, _ = env.reset()
    assert obs.dtype == np.float64 and obs.shape == (4, 30, 30)
    obs, _, _, _, info = env.step({"motor_action": 0, "sensory_action": np.array([47.0, 12.0]), "sensory_action_type": 1})
    assert obs.dtype == np.float64 and obs.shape == (4, 30, 30)   # no slicing to fov_res
    assert np.array_equal(info["fov_res"], [47, 12])
