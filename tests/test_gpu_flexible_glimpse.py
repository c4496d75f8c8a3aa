"""GPU: the flexible fovea's glimpse (``resize_to_fov``, AGYM_OUT_RESIZE_FOV) against the composed C oracle
(``tests/glimpse_oracle.py``).

The glimpse of an env is, per plane, torchvision's ``Resize(fov_size)`` of the unblurred window after this step's
fovea update (fov_env.py:248,284-285).  Grey Atari (K=4), grey DMC (K=3) and RGB DMC (K*C=9); the oracle reads the
ring the kernels ingested (ingest is pinned elsewhere), so these tests isolate the observe step.  Resampled pixels
within TOL of the oracle's float64 value, fov_loc / fov_res exact."""
import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from tests.glimpse_oracle import observe_glimpse

pytestmark = pytest.mark.gpu

TOL = 0.5 + 1e-2
S = (84, 84)
GUARD, CANARY = 4096, 0xA5
INIT = (3, 4)
# name: (frame_stack, channels, raw frame)
CFG = {"atari": (4, 1, (210, 160, 1)), "dmc": (3, 1, S + (3,)), "rgb": (3, 3, S + (3,))}


def _path(cfg, n, fov, antialias=True, buffers=None):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    K, C, raw = CFG[cfg]
    kw = {} if cfg == "atari" else {"luma": LUMA_DMC}
    return ObservationPath(n, K, S, raw, fov_size=fov, fov_init_loc=INIT, sensory_action_mode="absolute", device="cuda:0",
                           antialias=antialias, channels=C, buffers=buffers, **kw)


def _ingest(p, cfg, rng, step):
    n = p.n_envs
    fl = np.full(n, 5 if step == 0 else 1, np.uint8)
    if step:
        fl[rng.random(n) < 0.15] = 8
    if cfg == "atari":
        fa = rng.integers(0, 256, (n, 210, 160), dtype=np.uint8)
        p.ingest_atari(fa, rng.integers(0, 256, (n, 210, 160), dtype=np.uint8), fl | 3 if step else fl)
    else:
        p.ingest_dmc(rng.integers(0, 256, (n,) + S + (3,), dtype=np.uint8), fl)


def _actions(n, fov, rng, step):
    """Mixed FOV_LOC / FOV_RES actions with extreme windows, and ragged APPLY / RESET / KEEP control."""
    at = rng.integers(0, 2, n).astype(np.int32)
    a = np.where(at[:, None] == 1, rng.integers(1, 85, (n, 2)), rng.integers(-5, 90, (n, 2))).astype(np.float64)
    ext = [[1, 1], [1, 84], [84, 1], [84, 84], list(fov), [fov[0] + 1, fov[1] - 1]]
    k = min(n, len(ext))
    a[:k], at[:k] = ext[:k], 1
    ctrl = rng.choice(np.array([0, 0, 0, 1, 2], np.uint8), n) if step else None
    if ctrl is not None and n > 8:
        ctrl[:k] = 0
    return a, at, ctrl


def _oracle_update(a, at, ctrl, loc, res, fov):
    """fov update as the kernels do it: APPLY = the reference's _fov_step, RESET = init, KEEP = unchanged."""
    nl, nr = loc.copy(), res.copy()
    orc.update_loc(a, nl, obs_size=S, fov_size=fov, atype=at, res=nr)
    c = np.zeros(len(a), np.uint8) if ctrl is None else ctrl
    loc[c == 0], res[c == 0] = nl[c == 0], nr[c == 0]
    loc[c == 1], res[c == 1] = INIT, fov


def _oracle_glimpse(p, loc, res, fov, antialias=True):
    """The oracle's glimpse of an ObservationPath's ring, planes regrouped as (K, C) for RGB."""
    ring, head = p.ring.cpu().numpy(), p.head.cpu().numpy()
    orc.set_antialias(antialias)
    try:
        o = observe_glimpse(ring, head, loc, res, fov)
    finally:
        orc.set_antialias(True)
    return o.reshape((len(loc), p.frame_stack) + ((p.channels,) if p.channels > 1 else ()) + tuple(fov))


def _one_path(env):
    """The single ObservationPath behind an env, or None when the env is split into several shards."""
    paths = getattr(env.path, "paths", [env.path])
    return paths[0] if len(paths) == 1 else None


def _normalized(u8, dtype):
    """float32(u) / 255 as an IEEE division (torch's CUDA division by a scalar multiplies by the reciprocal), then dtype."""
    return torch.from_numpy(u8.cpu().numpy().astype(np.float32) / np.float32(255)).to(dtype)


def _kernels(fn):
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    return [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]


@pytest.mark.parametrize("cfg", ["atari", "dmc", "rgb"])
@pytest.mark.parametrize("fov", [(30, 30), (21, 33), (50, 28)])
@pytest.mark.parametrize("antialias", [True, False])
def test_glimpse_matches_the_oracle(cfg, fov, antialias):
    rng = np.random.default_rng(hash((cfg, fov, antialias)) % 2**32)
    n = 336   # every geometry's output is then a multiple of 16 pixels: the normalised copy is checked everywhere
    p = _path(cfg, n, fov, antialias)
    K, C, _ = CFG[cfg]
    loc = np.tile(np.array([INIT], np.int32), (n, 1))
    res = np.tile(np.array([fov], np.int32), (n, 1))
    p.observe_flexible(None, ctrl="reset", variant="resize_fov")
    for step in range(4):
        _ingest(p, cfg, rng, step)
        a, at, ctrl = _actions(n, fov, rng, step)
        nrm = torch.empty(p.out_shape("flexible", "resize_fov"), dtype=torch.float32, device="cuda:0")
        out = p.observe_flexible(a, at, variant="resize_fov", ctrl=ctrl, norm_out=nrm)
        _oracle_update(a, at, ctrl, loc, res, fov)
        torch.cuda.synchronize()
        assert np.array_equal(p.loc.cpu().numpy(), loc) and np.array_equal(p.res.cpu().numpy(), res), step
        got = out.cpu().numpy()
        assert got.shape == (n, K) + ((C,) if C > 1 else ()) + fov
        want = _oracle_glimpse(p, loc, res, fov, antialias)
        assert np.abs(got.astype(np.float64) - want).max() <= TOL, step
        assert torch.equal(nrm.cpu(), _normalized(out, torch.float32))


@pytest.mark.parametrize("cfg", ["atari", "dmc", "rgb"])
def test_fov_state_equals_the_mask_variant(cfg):
    rng = np.random.default_rng(7)
    n, fov = 500, (30, 30)
    g, m = _path(cfg, n, fov), _path(cfg, n, fov)
    for step in range(4):
        seed = int(rng.integers(1 << 30))
        _ingest(g, cfg, np.random.default_rng(seed), step)
        _ingest(m, cfg, np.random.default_rng(seed), step)
        a, at, ctrl = _actions(n, fov, rng, step)
        g.observe_flexible(a, at, variant="resize_fov", ctrl=ctrl)
        m.observe_flexible(a, at, variant="mask", ctrl=ctrl)
        torch.cuda.synchronize()
        assert torch.equal(g.loc, m.loc) and torch.equal(g.res, m.res), step


@pytest.mark.parametrize("cfg", ["atari", "dmc", "rgb"])
@pytest.mark.parametrize("fov", [(30, 30), (21, 33)])
def test_glimpse_at_fov_res_is_the_fixed_crop_bit_exact(cfg, fov):
    rng = np.random.default_rng(11)
    n = 401
    g, f = _path(cfg, n, fov), _path(cfg, n, fov)
    for step in range(3):
        seed = int(rng.integers(1 << 30))
        _ingest(g, cfg, np.random.default_rng(seed), step)
        _ingest(f, cfg, np.random.default_rng(seed), step)
    g.observe_flexible(None, ctrl="reset", variant="resize_fov")
    f.observe_fixed(None, ctrl="reset")
    for _ in range(3):   # FOV_LOC only: res stays fov_size
        a = rng.integers(-5, 90, (n, 2)).astype(np.float64)
        got = g.observe_flexible(a, np.zeros(n, np.int32), variant="resize_fov")
        want = f.observe_fixed(a, variant="crop")
        torch.cuda.synchronize()
        assert torch.equal(g.loc, f.loc)
        assert torch.equal(got, want)


# (cfg, fov, byte offset of the output view, kernel expected): the persistent kernel serves any tile that is a multiple
# of 4 bytes at a 4-byte-aligned address (bulk store at 16, word stores otherwise); the table-driven kernel the rest
PATHS = [("atari", (30, 30), 0, "k_observe_flexible_v3<3>"),     # 3,600 B tiles: one bulk store
         ("dmc", (30, 30), 0, "k_observe_flexible_v3<3>"),       # 2,700 B tiles: word stores
         ("rgb", (30, 30), 0, "k_observe_flexible_v3<3>"),       # 8,100 B tiles: word stores
         ("atari", (30, 30), 4, "k_observe_flexible_v3<3>"),     # 4-byte-aligned view
         ("atari", (21, 33), 0, "k_observe_flexible_v3<3>"),     # 2,772 B
         ("dmc", (21, 33), 0, "k_observe_flexible<3>"),          # 2,079 B: by geometry
         ("atari", (30, 30), 1, "k_observe_flexible<3>"),        # odd address
         ("rgb", (21, 33), 3, "k_observe_flexible<3>")]


@pytest.mark.parametrize("cfg,fov,offset,kernel", PATHS)
def test_kernel_selection_and_both_paths_match_the_oracle(cfg, fov, offset, kernel):
    rng = np.random.default_rng(offset + 13)
    n = 257
    p = _path(cfg, n, fov)
    K, C, _ = CFG[cfg]
    shape = p.out_shape("flexible", "resize_fov")
    nb = int(np.prod(shape))
    raw = torch.full((GUARD + nb + GUARD,), CANARY, dtype=torch.uint8, device="cuda:0")
    out = raw[GUARD + offset:GUARD + offset + nb].view(shape)
    loc = np.tile(np.array([INIT], np.int32), (n, 1))
    res = np.tile(np.array([fov], np.int32), (n, 1))
    p.observe_flexible(None, ctrl="reset", variant="resize_fov")
    for step in range(2):
        _ingest(p, cfg, rng, step)
    a, at, _ = _actions(n, fov, rng, 0)
    names = _kernels(lambda: p.observe_flexible(a, at, variant="resize_fov", out=out))
    _oracle_update(a, at, None, loc, res, fov)
    assert any(kernel in k for k in names), names
    assert np.array_equal(p.loc.cpu().numpy(), loc) and np.array_equal(p.res.cpu().numpy(), res)
    assert np.abs(out.cpu().numpy().astype(np.float64) - _oracle_glimpse(p, loc, res, fov)).max() <= TOL
    assert bool((raw[:GUARD + offset] == CANARY).all()) and bool((raw[GUARD + offset + nb:] == CANARY).all())


def test_fast_and_generic_kernels_agree_bit_for_bit():
    """Same tables, same evaluation order: the persistent kernel's glimpse equals the table-driven kernel's."""
    rng = np.random.default_rng(19)
    n, fov = 600, (30, 30)
    p = _path("atari", n, fov)
    for step in range(2):
        _ingest(p, "atari", rng, step)
    a, at, _ = _actions(n, fov, rng, 0)
    loc0, res0 = p.loc.clone(), p.res.clone()
    fast = p.observe_flexible(a, at, variant="resize_fov").clone()
    p.loc.copy_(loc0); p.res.copy_(res0)
    raw = torch.empty(fast.numel() + 1, dtype=torch.uint8, device="cuda:0")
    slow = raw[1:].view(fast.shape)
    p.observe_flexible(a, at, variant="resize_fov", out=slow)
    torch.cuda.synchronize()
    assert torch.equal(fast, slow)


class Guarded:
    def __init__(self, shape, dtype, fill=0):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        self.raw = torch.full((GUARD + n + (-n) % 256 + GUARD,), CANARY, dtype=torch.uint8, device="cuda:0")
        self.t = self.raw[GUARD:GUARD + n].view(dtype).view(shape)
        self.t.fill_(fill)
        self.n = n

    def intact(self):
        return bool((self.raw[:GUARD] == CANARY).all()) and bool((self.raw[GUARD + self.n:] == CANARY).all())


@pytest.mark.parametrize("cfg", ["atari", "rgb"])
@pytest.mark.parametrize("n", [1, 37, 333, 1001])
def test_glimpse_stays_inside_its_buffers(cfg, n):
    rng = np.random.default_rng(n)
    fov = (30, 30)
    K, C, _ = CFG[cfg]
    P = K * C
    g = dict(ring=Guarded((n, P) + S, torch.uint8), head=Guarded((n,), torch.int32, P - 1),
             loc=Guarded((n, 2), torch.int32), res=Guarded((n, 2), torch.int32))
    g["res"].t[:, 0], g["res"].t[:, 1] = fov
    p = _path(cfg, n, fov, buffers={k: v.t for k, v in g.items()})
    shape = p.out_shape("flexible", "resize_fov")
    out = Guarded(shape, torch.uint8)
    norm = Guarded(shape, torch.bfloat16) if int(np.prod(shape)) % 16 == 0 else None
    loc = np.zeros((n, 2), np.int32)
    res = np.tile(np.array([fov], np.int32), (n, 1))
    for step in range(4):
        _ingest(p, cfg, rng, step)
        a, at, ctrl = _actions(n, fov, rng, step)
        p.observe_flexible(a, at, variant="resize_fov", ctrl=ctrl, out=out.t, norm_out=None if norm is None else norm.t)
        _oracle_update(a, at, ctrl, loc, res, fov)
    torch.cuda.synchronize()
    assert all(v.intact() for v in list(g.values()) + [out] + ([norm] if norm is not None else []))
    assert np.array_equal(g["loc"].t.cpu().numpy(), loc) and np.array_equal(g["res"].t.cpu().numpy(), res)
    assert np.abs(out.t.cpu().numpy().astype(np.float64) - _oracle_glimpse(p, loc, res, fov)).max() <= TOL
    if norm is not None:
        assert torch.equal(norm.t.cpu(), _normalized(out.t, torch.bfloat16))


@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_a_glimpse_step_is_deterministic(cfg):
    rng = np.random.default_rng(17)
    n, fov = 2500, (30, 30)
    p = _path(cfg, n, fov)
    for step in range(CFG[cfg][0] + 1):
        _ingest(p, cfg, rng, step)
    torch.cuda.synchronize()
    a, at, ctrl = _actions(n, fov, rng, 1)
    state0 = [p.loc.clone(), p.res.clone()]
    ref = None
    for rep in range(6):
        p.loc.copy_(state0[0]); p.res.copy_(state0[1])
        out = p.observe_flexible(a, at, variant="resize_fov", ctrl=ctrl)
        torch.cuda.synchronize()
        snap = [out.clone(), p.loc.clone(), p.res.clone()]
        if ref is None:
            ref = snap
        else:
            assert all(torch.equal(x, y) for x, y in zip(ref, snap)), rep


# ------------------------------------------------------------------------------------------------ env level
def _atari_env(n, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", resize_to_fov=True)
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return ag.AtariFlexibleFovealEnv(args, num_envs=n, source=SyntheticAtariSource(n, device="cuda"))


def _dmc_env(n, grey, device=None, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import DMCPool
    from tests.test_gpu_dmc_rgb import _FakeDMC
    rng = np.random.default_rng(3)
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", frame_stack=3, action_repeat=2,
              grey=grey, resize_to_fov=True)
    kw.update(extra)
    args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, **kw)
    return ag.DMCFlexibleFovealEnv(args, num_envs=n, source=DMCPool(
        args, n if n else 1, env_factory=lambda i: _FakeDMC(rng.integers(0, 256, (7,) + S + (3,), dtype=np.uint8))), device=device)


def _motor(kind, n):
    return np.zeros(n, np.int64) if kind == "atari" else np.zeros((n, 2), np.float32)


def _env(kind, n, **extra):
    return _atari_env(n, **extra) if kind == "atari" else _dmc_env(n, kind == "dmc", **extra)


@pytest.mark.parametrize("kind", ["atari", "dmc", "rgb"])
@pytest.mark.parametrize("extra", [{}, {"obs_dtype": torch.float32}, {"obs_dtype": torch.float16},
                                   {"obs_dtype": torch.bfloat16}, {"host_obs": True}])
def test_env_returns_the_glimpse(kind, extra):
    rng = np.random.default_rng(23)
    n = 20
    env = _env(kind, n, **extra)
    K = 4 if kind == "atari" else 3
    frame = (K,) if kind != "rgb" else (K, 3)
    assert env.variant == "resize_fov" and env.observation_space.shape == frame + (30, 30)
    assert env.obs_shape == (n,) + frame + (30, 30)
    obs, info = env.reset()
    for step in range(4):
        at = rng.integers(0, 2, n).astype(np.int64)
        a = np.where(at[:, None] == 1, rng.integers(20, 51, (n, 2)), rng.integers(0, 55, (n, 2))).astype(np.float64)
        obs, _, _, _, info = env.step({"motor_action": _motor(kind, n), "sensory_action": a, "sensory_action_type": at})
        path = _one_path(env)
        loc = np.asarray(info["fov_loc"].cpu() if isinstance(info["fov_loc"], torch.Tensor) else info["fov_loc"])
        res = np.asarray(info["fov_res"].cpu() if isinstance(info["fov_res"], torch.Tensor) else info["fov_res"])
        torch.cuda.synchronize()
        assert tuple(obs.shape) == (n,) + frame + (30, 30)
        want = None if path is None else _oracle_glimpse(path, loc, res, (30, 30))
        u8 = env.last_obs_u8 if extra.get("obs_dtype") is not None else obs
        got = (u8.cpu() if isinstance(u8, torch.Tensor) else torch.as_tensor(u8)).numpy()
        if want is not None:
            assert np.abs(got.astype(np.float64) - want).max() <= TOL, step
        if extra.get("obs_dtype") is not None:
            assert obs.dtype == extra["obs_dtype"]
            assert torch.equal(obs.cpu(), _normalized(torch.from_numpy(got), extra["obs_dtype"]))
        if extra.get("host_obs"):
            assert not obs.is_cuda
    env.close()


@pytest.mark.parametrize("kind", ["atari", "rgb"])
def test_single_env_adapter_returns_float64_glimpses(kind):
    from active_gym_b200 import SingleEnvAdapter
    env = SingleEnvAdapter(_env(kind, 1))
    frame = (4,) if kind == "atari" else (3, 3)
    obs, _ = env.reset()
    assert obs.dtype == np.float64 and obs.shape == frame + (30, 30)
    res = np.array([30, 30])
    for step in range(4):
        at = step % 2
        a = np.array([20 + 9 * step, 45 - 7 * step] if at else [10 * step, 50 - 9 * step], np.float64)
        obs, _, _, _, info = env.step({"motor_action": _motor(kind, 1)[0], "sensory_action": a, "sensory_action_type": at})
        torch.cuda.synchronize()
        if at:
            res = a.astype(np.int64)
        assert obs.dtype == np.float64 and obs.shape == frame + (30, 30)   # fixed shape: no slicing to fov_res
        assert np.array_equal(np.asarray(info["fov_res"]), res)
        p = _one_path(env.env)
        want = _oracle_glimpse(p, p.loc.cpu().numpy(), p.res.cpu().numpy(), (30, 30))[0]
        assert np.abs(obs * 255.0 - want).max() <= TOL + 1e-4
    env.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more GPUs")
def test_sharded_learner_device_receives_the_glimpse():
    from active_gym_b200.vector import ShardedVecEnv
    n = 40
    venv = ShardedVecEnv(lambda m, dev, lo, hi: _dmc_env(m, True, device=dev), n, devices=["cuda:0", "cuda:1"],
                         learner_device="cuda:0")
    obs, _ = venv.reset()
    assert tuple(obs.shape) == (n, 3, 30, 30) and obs.device == torch.device("cuda:0")
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
            want = _oracle_glimpse(p, p.loc.cpu().numpy(), p.res.cpu().numpy(), (30, 30))
            assert np.abs(obs[lo:lo + e.num_envs].cpu().numpy().astype(np.float64) - want).max() <= TOL
        lo += e.num_envs
    venv.close()
