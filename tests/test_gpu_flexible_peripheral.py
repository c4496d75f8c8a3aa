"""GPU: the flexible fovea over the peripheral background (agym_observe_flexible_peripheral) against the composed C
oracle (``tests/flex_periph_oracle.py``), the two identities that make most checks tolerance-free, and the env level.

(I1) inside the window the output is agym_observe_flexible(AGYM_OUT_MASK)'s on the same state, bit for bit;
(I2) outside it, agym_observe_peripheral's from the same cache, bit for bit where that call runs its standard-geometry
     kernel (grey, 84x84, 20x20 periphery).
Grey Atari (K=4), grey DMC (K=3) and RGB DMC (K*C=9); the oracle reads the ring the kernels ingested."""
import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from tests.flex_periph_oracle import observe_flexible_peripheral
from tests.test_gpu_flexible_glimpse import (CFG, INIT, _actions, _ingest, _kernels, _motor, _normalized, _one_path,
                                             _oracle_update)

pytestmark = pytest.mark.gpu

TOL = 0.5 + 2e-2
S = (84, 84)


def _path(cfg, n, fov=(30, 30), per=(20, 20), antialias=True, buffers=None):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    K, C, raw = CFG[cfg]
    kw = {} if cfg == "atari" else {"luma": LUMA_DMC}
    return ObservationPath(n, K, S, raw, fov_size=fov, fov_init_loc=INIT, sensory_action_mode="absolute", device="cuda:0",
                           antialias=antialias, channels=C, peripheral_res=per, buffers=buffers, **kw)


def _twins(cfg, n, m=2, **kw):
    return [_path(cfg, n, **kw) for _ in range(m)]


def _ingest_all(paths, cfg, seed, step):
    for p in paths:
        _ingest(p, cfg, np.random.default_rng(seed), step)


def _oracle(p, loc, res, fov, per, antialias=True, envs=None):
    """The composed oracle on an ObservationPath's ring (optionally a subset of envs), in the output's layout."""
    ring, head = p.ring.cpu().numpy(), p.head.cpu().numpy()
    sel = slice(None) if envs is None else envs
    orc.set_antialias(antialias)
    try:
        o = observe_flexible_peripheral(ring[sel], head[sel], loc[sel], res[sel], fov, per)
    finally:
        orc.set_antialias(True)
    return o.reshape((o.shape[0], p.frame_stack) + ((p.channels,) if p.channels > 1 else ()) + S)


def _window_mask(loc, res, shape):
    """True inside each env's window, broadcast to the output's shape."""
    n = len(loc)
    yy, xx = np.arange(S[0])[None, :, None], np.arange(S[1])[None, None, :]
    m = ((yy >= loc[:, 0, None, None]) & (yy < (loc[:, 0] + res[:, 0])[:, None, None]) &
         (xx >= loc[:, 1, None, None]) & (xx < (loc[:, 1] + res[:, 1])[:, None, None]))
    return np.broadcast_to(m.reshape((n,) + (1,) * (len(shape) - 3) + S), shape)


def _check(got, want, loc, res, fov):
    """Unblurred windows bit exact; everything within TOL of the oracle's float64 value."""
    assert np.abs(got.astype(np.float64) - want).max() <= TOL
    sharp = _window_mask(loc, res, got.shape) & (res[:, 0] <= fov[0]).reshape((-1,) + (1,) * (got.ndim - 1))
    assert np.array_equal(got[sharp], want[sharp].astype(np.uint8))


CASES = [("atari", (30, 30), (20, 20)), ("atari", (20, 20), (20, 20)), ("dmc", (30, 30), (20, 20)),
         ("rgb", (30, 30), (20, 20)), ("dmc", (21, 33), (16, 24))]


@pytest.mark.parametrize("case", CASES, ids=[f"{c}-{f[0]}x{f[1]}-p{p[0]}x{p[1]}" for c, f, p in CASES])
@pytest.mark.parametrize("antialias", [True, False])
def test_kernels_match_the_composed_oracle(case, antialias):
    cfg, fov, per = case
    rng = np.random.default_rng(hash((cfg, fov, antialias)) % 2**32)
    n = 336
    p = _path(cfg, n, fov, per, antialias)
    loc = np.tile(np.array([INIT], np.int32), (n, 1))
    res = np.tile(np.array([fov], np.int32), (n, 1))
    p.observe_flexible_peripheral(None, ctrl="reset")
    for step in range(4):
        _ingest(p, cfg, rng, step)
        a, at, ctrl = _actions(n, fov, rng, step)
        nrm = torch.empty(p.out_shape("flexible_peripheral", "mask"), dtype=torch.float32, device="cuda:0")
        out = p.observe_flexible_peripheral(a, at, ctrl=ctrl, norm_out=nrm)
        _oracle_update(a, at, ctrl, loc, res, fov)
        torch.cuda.synchronize()
        assert np.array_equal(p.loc.cpu().numpy(), loc) and np.array_equal(p.res.cpu().numpy(), res), step
        got = out.cpu().numpy()
        assert got.shape == p.out_shape("flexible_peripheral", "mask")
        _check(got, _oracle(p, loc, res, fov, per, antialias), loc, res, fov)
        assert torch.equal(nrm.cpu(), _normalized(out, torch.float32))


@pytest.mark.parametrize("cfg", ["atari", "dmc", "rgb"])
def test_identities_window_is_mask_out_and_background_is_the_peripheral_view(cfg):
    """(I1) bit for bit everywhere; (I2) bit for bit at the standard grey geometry, within TOL for RGB (whose peripheral
    call runs k_observe_peripheral_v2, which adds the two W taps in the other order)."""
    rng = np.random.default_rng(5)
    n, fov = 1000, (30, 30)
    fp, mk, pe = _twins(cfg, n, 3)
    for step in range(4):
        _ingest_all((fp, mk, pe), cfg, int(rng.integers(1 << 30)), step)
        a, at, ctrl = _actions(n, fov, rng, step)
        out = fp.observe_flexible_peripheral(a, at, ctrl=ctrl)
        m = mk.observe_flexible(a, at, variant="mask", ctrl=ctrl)
        pv = pe.observe_peripheral(np.zeros((n, 2)))   # its own fovea at (0, 0): compared outside it below
        torch.cuda.synchronize()
        assert torch.equal(fp.loc, mk.loc) and torch.equal(fp.res, mk.res)
        loc, res = fp.loc.cpu().numpy(), fp.res.cpu().numpy()
        got, mask_out, periph = out.cpu().numpy(), m.cpu().numpy(), pv.cpu().numpy()
        inside = _window_mask(loc, res, got.shape)
        assert np.array_equal(got[inside], mask_out[inside]), step
        outside = ~inside & ~_window_mask(np.zeros_like(loc), np.tile(np.array([fov], np.int32), (n, 1)), got.shape)
        if cfg == "rgb":
            assert np.abs(got[outside].astype(int) - periph[outside].astype(int)).max() <= 1
        else:
            assert np.array_equal(got[outside], periph[outside]), step


@pytest.mark.parametrize("cfg", ["atari", "dmc"])
def test_at_fov_res_it_is_the_fixed_peripheral_env(cfg):
    rng = np.random.default_rng(9)
    n, fov = 777, (30, 30)
    fp, pe = _twins(cfg, n)
    fp.observe_flexible_peripheral(None, ctrl="reset")
    pe.observe_peripheral(None, ctrl="reset")
    for step in range(4):
        _ingest_all((fp, pe), cfg, int(rng.integers(1 << 30)), step)
        a = rng.integers(-5, 90, (n, 2)).astype(np.float64)
        out = fp.observe_flexible_peripheral(a, np.zeros(n, np.int32))
        pv = pe.observe_peripheral(a)
        torch.cuda.synchronize()
        assert torch.equal(fp.loc, pe.loc) and torch.equal(out, pv), step


@pytest.mark.parametrize("cfg,fov,per", [("atari", (30, 30), (20, 20)), ("rgb", (30, 30), (20, 20)),
                                         ("dmc", (21, 33), (16, 24))])
def test_fast_and_table_driven_kernels_agree_bit_for_bit(cfg, fov, per):
    """An output view at an odd address forces the table-driven kernel; profiler names pin which kernel ran."""
    rng = np.random.default_rng(13)
    n = 600
    fast, slow = _twins(cfg, n, fov=fov, per=per)
    shape = fast.out_shape("flexible_peripheral", "mask")
    numel = int(np.prod(shape))
    raw = torch.empty(numel + 16, dtype=torch.uint8, device="cuda:0")
    odd = raw[1:1 + numel].view(shape)
    for step in range(4):
        _ingest_all((fast, slow), cfg, int(rng.integers(1 << 30)), step)
        a, at, ctrl = _actions(n, fov, rng, step)
        names_fast = _kernels(lambda: fast.observe_flexible_peripheral(a, at, ctrl=ctrl))
        out = fast.observe_flexible_peripheral(None, ctrl=np.full(n, 2, np.uint8))   # KEEP: the same windows again
        names_slow = _kernels(lambda: slow.observe_flexible_peripheral(a, at, ctrl=ctrl, out=odd))
        torch.cuda.synchronize()
        assert torch.equal(fast.loc, slow.loc) and torch.equal(fast.res, slow.res)
        assert torch.equal(out, odd), step
        if fov == (30, 30):   # configs[2] geometry and RGB: the persistent kernel
            assert any("k_observe_flexible_v3<4>" in k for k in names_fast), names_fast
        assert any("k_observe_flexible<4>" in k for k in names_slow), names_slow
        assert not any("k_observe_flexible_v3" in k for k in names_slow), names_slow


class _Guarded:
    """A tensor inside a canary-filled allocation: writes past either end are detected."""

    def __init__(self, shape, dtype=torch.uint8, guard=4096):
        numel = int(np.prod(shape))
        self.g = guard
        self.buf = torch.full((numel + 2 * guard,), 0xA5, dtype=torch.uint8, device="cuda:0") if dtype == torch.uint8 else \
            torch.full((numel + 2 * guard,), -7.0, dtype=dtype, device="cuda:0")
        self.t = self.buf[guard:guard + numel].view(shape)
        self.c = self.buf[:guard].clone(), self.buf[guard + numel:].clone()

    def intact(self):
        return torch.equal(self.buf[:self.g], self.c[0]) and torch.equal(self.buf[self.buf.numel() - self.g:], self.c[1])


@pytest.mark.parametrize("n", [1, 37, 333, 1001])
@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_guard_bands(cfg, n):
    rng = np.random.default_rng(n)
    fov, per = (30, 30), (20, 20)
    p = _path(cfg, n)
    out = _Guarded(p.out_shape("flexible_peripheral", "mask"))
    norm = _Guarded(p.out_shape("flexible_peripheral", "mask"), torch.bfloat16)
    loc = np.tile(np.array([INIT], np.int32), (n, 1))
    res = np.tile(np.array([fov], np.int32), (n, 1))
    p.observe_flexible_peripheral(None, ctrl="reset")
    for step in range(3):
        _ingest(p, cfg, rng, step)
        a, at, ctrl = _actions(n, fov, rng, step)
        p.observe_flexible_peripheral(a, at, ctrl=ctrl, out=out.t, norm_out=norm.t)
        _oracle_update(a, at, ctrl, loc, res, fov)
    torch.cuda.synchronize()
    assert out.intact() and norm.intact()
    _check(out.t.cpu().numpy(), _oracle(p, loc, res, fov, per), loc, res, fov)
    assert torch.equal(norm.t.cpu(), _normalized(out.t, torch.bfloat16))


@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_a_step_is_deterministic(cfg):
    rng = np.random.default_rng(17)
    n = 2500
    p = _path(cfg, n)
    for step in range(CFG[cfg][0] + 1):
        _ingest(p, cfg, rng, step)
    a, at, ctrl = _actions(n, (30, 30), rng, 1)
    state0 = [p.loc.clone(), p.res.clone()]
    ref = None
    for rep in range(6):
        p.loc.copy_(state0[0]); p.res.copy_(state0[1])
        out = p.observe_flexible_peripheral(a, at, ctrl=ctrl)
        torch.cuda.synchronize()
        snap = [out.clone(), p.loc.clone(), p.res.clone()]
        if ref is None:
            ref = snap
        else:
            assert all(torch.equal(x, y) for x, y in zip(ref, snap)), rep


@pytest.mark.parametrize("n", [4096, 16384])
def test_full_size_parity_on_boundary_envs(n):
    rng = np.random.default_rng(n)
    fov, per = (30, 30), (20, 20)
    p = _path("atari", n)
    loc = np.tile(np.array([INIT], np.int32), (n, 1))
    res = np.tile(np.array([fov], np.int32), (n, 1))
    p.observe_flexible_peripheral(None, ctrl="reset")
    for step in range(3):
        _ingest(p, "atari", rng, step)
        a, at, ctrl = _actions(n, fov, rng, step)
        out = p.observe_flexible_peripheral(a, at, ctrl=ctrl)
        _oracle_update(a, at, ctrl, loc, res, fov)
    torch.cuda.synchronize()
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    envs = np.unique(np.clip([0, 1, sms - 1, sms, 2 * sms - 1, 2 * sms, 4 * sms, n // 2, n - 2, n - 1], 0, n - 1))
    assert np.array_equal(p.loc.cpu().numpy(), loc) and np.array_equal(p.res.cpu().numpy(), res)
    _check(out.cpu().numpy()[envs], _oracle(p, loc, res, fov, per, envs=envs), loc[envs], res[envs], fov)


def test_device_error_word_for_fov_res_given_as_cuda_tensors():
    from active_gym_b200 import _lib
    n = 64
    p = _path("atari", n)
    _ingest(p, "atari", np.random.default_rng(0), 0)
    a = torch.full((n, 2), 30.0, dtype=torch.float64, device="cuda:0")
    a[3] = torch.tensor([90.0, 30.0])
    a[5] = torch.tensor([30.5, 30.0])
    p.observe_flexible_peripheral(a, torch.ones(n, dtype=torch.int32, device="cuda:0"))
    assert p.read_errors() == _lib.ERR_RES_RANGE | _lib.ERR_RES_FRACTION
    assert p.read_errors() == 0


def test_entry_point_rejects_plans_without_a_periphery_and_a_null_cache():
    from active_gym_b200 import _lib
    from active_gym_b200.engine import _ptr
    L = _lib.lib()
    from active_gym_b200 import ObservationPath
    for p in (_path("atari", 8), ObservationPath(8, 4, S, (210, 160, 1), fov_size=(30, 30), device="cuda:0")):
        out = torch.empty(p.out_shape("flexible_peripheral", "mask"), dtype=torch.uint8, device="cuda:0")
        act = torch.zeros((8, 2), dtype=torch.float64, device="cuda:0")
        # NULL cache, or a plan without a periphery (whose path has no cache either)
        st = L.agym_observe_flexible_peripheral(p._plan, _ptr(p.ring), _ptr(p.head), None, _ptr(act), None, None,
                                                _ptr(p.loc), _ptr(p.res), _ptr(out), None, None, 0, p._stream())
        assert st == -1
    with pytest.raises(ValueError, match="cache"):
        p.observe_flexible_peripheral(act)


# ------------------------------------------------------------------------------------------------ env level
def _atari_env(n, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", peripheral_res=(20, 20))
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return ag.AtariFlexibleFovealPeripheralEnv(args, num_envs=n, source=SyntheticAtariSource(n, device="cuda"))


def _dmc_env(n, grey, device=None, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import DMCPool
    from tests.test_gpu_dmc_rgb import _FakeDMC
    rng = np.random.default_rng(3)
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", frame_stack=3, action_repeat=2,
              grey=grey, peripheral_res=(20, 20))
    kw.update(extra)
    args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, **kw)
    return ag.DMCFlexibleFovealPeripheralEnv(args, num_envs=n, source=DMCPool(
        args, n if n else 1, env_factory=lambda i: _FakeDMC(rng.integers(0, 256, (7,) + S + (3,), dtype=np.uint8))), device=device)


def _env(kind, n, **extra):
    return _atari_env(n, **extra) if kind == "atari" else _dmc_env(n, kind == "dmc", **extra)


@pytest.mark.parametrize("kind", ["atari", "dmc", "rgb"])
@pytest.mark.parametrize("extra", [{}, {"obs_dtype": torch.float32}, {"obs_dtype": torch.float16},
                                   {"obs_dtype": torch.bfloat16}, {"host_obs": True}])
def test_env_returns_the_peripheral_flexible_view(kind, extra):
    rng = np.random.default_rng(23)
    n = 20
    env = _env(kind, n, **extra)
    K = 4 if kind == "atari" else 3
    frame = (K,) if kind != "rgb" else (K, 3)
    assert env.observation_space.shape == frame + S and env.obs_shape == (n,) + frame + S
    obs, info = env.reset()
    assert {"fov_loc", "fov_res"} <= set(info)
    for step in range(4):
        at = rng.integers(0, 2, n).astype(np.int64)
        a = np.where(at[:, None] == 1, rng.integers(20, 51, (n, 2)), rng.integers(0, 55, (n, 2))).astype(np.float64)
        obs, _, _, _, info = env.step({"motor_action": _motor(kind, n), "sensory_action": a, "sensory_action_type": at})
        path = _one_path(env)
        loc = np.asarray(info["fov_loc"].cpu() if isinstance(info["fov_loc"], torch.Tensor) else info["fov_loc"])
        res = np.asarray(info["fov_res"].cpu() if isinstance(info["fov_res"], torch.Tensor) else info["fov_res"])
        torch.cuda.synchronize()
        assert tuple(obs.shape) == (n,) + frame + S
        assert np.array_equal(res[at == 1], a[at == 1].astype(np.int32))
        u8 = env.last_obs_u8 if extra.get("obs_dtype") is not None else obs
        got = (u8.cpu() if isinstance(u8, torch.Tensor) else torch.as_tensor(u8)).numpy()
        if path is not None:
            _check(got, _oracle(path, loc.astype(np.int32), res.astype(np.int32), (30, 30), (20, 20)), loc, res, (30, 30))
        if extra.get("obs_dtype") is not None:
            assert obs.dtype == extra["obs_dtype"]
            assert torch.equal(obs.cpu(), _normalized(torch.from_numpy(got), extra["obs_dtype"]))
            ref = env.path.normalize(u8, extra["obs_dtype"])   # agym_normalize
            assert torch.equal(obs, ref)
        if extra.get("host_obs"):
            assert not obs.is_cuda
    env.close()


@pytest.mark.parametrize("kind", ["atari", "rgb"])
def test_single_env_adapter(kind):
    from active_gym_b200 import SingleEnvAdapter
    env = SingleEnvAdapter(_env(kind, 1))
    frame = (4,) if kind == "atari" else (3, 3)
    obs, _ = env.reset()
    assert obs.dtype == np.float64 and obs.shape == frame + S
    for step in range(4):
        at = step % 2
        a = np.array([20 + 9 * step, 45 - 7 * step] if at else [10 * step, 50 - 9 * step], np.float64)
        obs, _, _, _, info = env.step({"motor_action": _motor(kind, 1)[0], "sensory_action": a, "sensory_action_type": at})
        torch.cuda.synchronize()
        assert obs.dtype == np.float64 and obs.shape == frame + S
        p = _one_path(env.env)
        want = _oracle(p, p.loc.cpu().numpy(), p.res.cpu().numpy(), (30, 30), (20, 20))[0]
        assert np.abs(obs * 255.0 - want).max() <= TOL + 1e-4
    env.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more GPUs")
def test_sharded_learner_device_receives_the_view():
    from active_gym_b200.vector import ShardedVecEnv
    n = 40
    venv = ShardedVecEnv(lambda m, dev, lo, hi: _dmc_env(m, True, device=dev), n, devices=["cuda:0", "cuda:1"],
                         learner_device="cuda:0")
    obs, _ = venv.reset()
    assert tuple(obs.shape) == (n, 3) + S and obs.device == torch.device("cuda:0")
    rng = np.random.default_rng(1)
    at = rng.integers(0, 2, n).astype(np.int64)
    a = {"motor_action": np.zeros((n, 2), np.float32), "sensory_action_type": at,
         "sensory_action": np.where(at[:, None] == 1, rng.integers(20, 51, (n, 2)), rng.integers(0, 55, (n, 2))).astype(np.float64)}
    obs, *_ = venv.step(a)
    torch.cuda.synchronize("cuda:0")
    torch.cuda.synchronize("cuda:1")
    lo = 0
    for e in venv.envs:
        p = _one_path(e)
        if p is not None:
            loc, res = p.loc.cpu().numpy(), p.res.cpu().numpy()
            _check(obs[lo:lo + e.num_envs].cpu().numpy(), _oracle(p, loc, res, (30, 30), (20, 20)), loc, res, (30, 30))
        lo += e.num_envs
    venv.close()
