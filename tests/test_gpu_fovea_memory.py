"""GPU: the fixed fovea's memory (``fov_memory``, ``agym_observe_fixed_memory``) against the composed C oracle
(``tests/fovea_memory_oracle.py``), bit for bit.

Grey Atari (K=4), grey DMC (K=3) and RGB DMC (K*C=9); the oracle reads the ring the kernels ingested (ingest is pinned
elsewhere), so these tests isolate the observe step and the memory it keeps."""
import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from tests.fovea_memory_oracle import APPLY, KEEP, RESET, MemoryOracle

pytestmark = pytest.mark.gpu

S = (84, 84)
GUARD, CANARY = 4096, 0xA5
INIT = (3, 4)
# name: (frame_stack, channels, raw frame)
CFG = {"atari": (4, 1, (210, 160, 1)), "dmc": (3, 1, S + (3,)), "rgb": (3, 3, S + (3,))}


def _path(cfg, n, fov, depth, mode="absolute", buffers=None):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    K, C, raw = CFG[cfg]
    kw = {} if cfg == "atari" else {"luma": LUMA_DMC}
    return ObservationPath(n, K, S, raw, fov_size=fov, fov_init_loc=INIT, sensory_action_mode=mode,
                           sensory_action_space=(-10.0, 10.0), device="cuda:0", channels=C, buffers=buffers,
                           fov_memory=depth, **kw)


def _ingest(p, cfg, rng, step):
    """Ragged ingest: a hard reset first, later random hard resets and idle envs."""
    n = p.n_envs
    fl = np.full(n, 5 if step == 0 else 1, np.uint8)
    if step:
        fl[rng.random(n) < 0.1] = 5
        fl[rng.random(n) < 0.15] = 8
    if cfg == "atari":
        fa = rng.integers(0, 256, (n, 210, 160), dtype=np.uint8)
        p.ingest_atari(fa, rng.integers(0, 256, (n, 210, 160), dtype=np.uint8), np.where(fl == 8, fl, fl | 3) if step else fl)
    else:
        p.ingest_dmc(rng.integers(0, 256, (n,) + S + (3,), dtype=np.uint8), fl)


def _actions(n, fov, rng, step, mode="absolute"):
    """Actions that reach every border, and ragged APPLY / RESET / KEEP control."""
    if mode == "absolute":
        a = rng.integers(-5, 90, (n, 2)).astype(np.float64)
        ext = [[0, 0], [0, 84], [84, 0], [84, 84], [-3, 40], [40, 99]]
    else:
        a = rng.integers(-14, 15, (n, 2)).astype(np.float64)
        ext = [[-14, -14], [14, 14], [-14, 14], [14, -14]]
    k = min(n, len(ext))
    a[:k] = ext[:k]
    ctrl = rng.choice(np.array([APPLY, APPLY, APPLY, RESET, KEEP], np.uint8), n) if step else None
    return a, ctrl


def _update(a, ctrl, loc, fov, mode):
    new = loc.copy()
    orc.update_loc(a, new, obs_size=S, fov_size=fov, relative=mode == "relative", lo=-10.0, hi=10.0)
    c = np.zeros(len(a), np.uint8) if ctrl is None else ctrl
    loc[c == APPLY] = new[c == APPLY]
    loc[c == RESET] = INIT


def _want(p, mem, loc, fov, ctrl):
    ring, head = p.ring.cpu().numpy(), p.head.cpu().numpy()
    return mem.observe(ring, head, loc, fov, ctrl, rgb=p.channels == 3)


def _normalized(u8, dtype):
    """float32(u) / 255 as an IEEE division, then dtype."""
    return torch.from_numpy(u8.cpu().numpy().astype(np.float32) / np.float32(255)).to(dtype)


@pytest.mark.parametrize("cfg", ["atari", "dmc", "rgb"])
@pytest.mark.parametrize("fov", [(30, 30), (21, 33), (50, 28)])
@pytest.mark.parametrize("depth", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("mode", ["absolute", "relative"])
def test_memory_matches_the_oracle(cfg, fov, depth, mode):
    rng = np.random.default_rng(hash((cfg, fov, depth, mode)) % 2**32)
    n = 131
    p = _path(cfg, n, fov, depth, mode)
    mem = MemoryOracle(n, depth)
    loc = np.zeros((n, 2), np.int32)
    for step in range(20 if depth < 16 else 24):
        _ingest(p, cfg, rng, step)
        a, ctrl = _actions(n, fov, rng, step, mode)
        out = p.observe_fixed_memory(a, ctrl=ctrl if step else "reset")
        _update(a, ctrl if step else np.full(n, RESET, np.uint8), loc, fov, mode)
        want = _want(p, mem, loc, fov, ctrl if step else np.full(n, RESET, np.uint8))
        torch.cuda.synchronize()
        assert np.array_equal(p.loc.cpu().numpy(), loc), step
        assert np.array_equal(out.cpu().numpy(), want), step
        assert np.array_equal(p.mem_state[:, 1].cpu().numpy(), mem.count()), step


@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_identities(cfg):
    """M = 1 is mask_out; the newest entry is the crop and its loc; KEEP repeats the output; the output bounds mask_out."""
    rng = np.random.default_rng(3)
    n, fov = 300, (21, 33)
    one, m8, ref = _path(cfg, n, fov, 1), _path(cfg, n, fov, 8), _path(cfg, n, fov, 0)
    K, C, _ = CFG[cfg]
    E = m8.mem.shape[2]
    for step in range(10):
        seed = int(rng.integers(1 << 30))
        for p in (one, m8, ref):
            _ingest(p, cfg, np.random.default_rng(seed), step)
        a, ctrl = _actions(n, fov, rng, step)
        c = ctrl if step else "reset"
        o1, o8 = one.observe_fixed_memory(a, ctrl=c), m8.observe_fixed_memory(a, ctrl=c)
        mask = ref.observe_fixed(a, variant="mask", ctrl=c)
        crop = ref.observe_fixed(None, variant="crop", ctrl=np.full(n, KEEP, np.uint8))
        torch.cuda.synchronize()
        pushed = np.ones(n, bool) if ctrl is None else ctrl != KEEP
        assert torch.equal(one.loc, ref.loc) and torch.equal(m8.loc, ref.loc)
        assert np.array_equal(o1.cpu().numpy()[pushed], mask.cpu().numpy()[pushed]), step
        assert bool((o8[torch.from_numpy(pushed).cuda()] >= mask[torch.from_numpy(pushed).cuda()]).all())
        st = m8.mem_state.cpu().numpy()
        mem = m8.mem.cpu().numpy()
        idx = np.flatnonzero(pushed)
        newest = mem[idx, st[idx, 0]]
        nb = K * C * fov[0] * fov[1]
        crop = crop.cpu().numpy()[idx]
        assert np.array_equal(newest[:, :nb].reshape(crop.shape), crop), step
        assert not newest[:, nb:E].any()
        assert np.array_equal(m8.mem_loc.cpu().numpy()[idx, st[idx, 0]], ref.loc.cpu().numpy()[idx])
        again = m8.observe_fixed_memory(None, ctrl=np.full(n, KEEP, np.uint8))
        torch.cuda.synchronize()
        assert torch.equal(again, o8), step
        assert np.array_equal(m8.mem_state.cpu().numpy(), st)


@pytest.mark.parametrize("offset", [1, 3, 4])
def test_unaligned_output_equals_the_aligned_output(offset):
    rng = np.random.default_rng(offset)
    n, fov = 77, (30, 30)
    a_p, u_p = _path("atari", n, fov, 3), _path("atari", n, fov, 3)
    shape = a_p.out_shape("fixed_memory", "mask")
    nb = int(np.prod(shape))
    raw = torch.full((GUARD + nb + GUARD,), CANARY, dtype=torch.uint8, device="cuda:0")
    view = raw[GUARD + offset:GUARD + offset + nb].view(shape)
    for step in range(6):
        seed = int(rng.integers(1 << 30))
        _ingest(a_p, "atari", np.random.default_rng(seed), step)
        _ingest(u_p, "atari", np.random.default_rng(seed), step)
        a, ctrl = _actions(n, fov, rng, step)
        want = a_p.observe_fixed_memory(a, ctrl=ctrl if step else "reset")
        u_p.observe_fixed_memory(a, ctrl=ctrl if step else "reset", out=view)
        torch.cuda.synchronize()
        assert torch.equal(view, want), step
    assert bool((raw[:GUARD + offset] == CANARY).all()) and bool((raw[GUARD + offset + nb:] == CANARY).all())


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
def test_memory_stays_inside_its_buffers(cfg, n):
    rng = np.random.default_rng(n)
    fov, depth = (50, 28), 3
    K, C, _ = CFG[cfg]
    P = K * C
    E = (P * fov[0] * fov[1] + 15) // 16 * 16
    g = dict(ring=Guarded((n, P) + S, torch.uint8), head=Guarded((n,), torch.int32, P - 1),
             loc=Guarded((n, 2), torch.int32), res=Guarded((n, 2), torch.int32),
             mem=Guarded((n, depth, E), torch.uint8), mem_loc=Guarded((n, depth, 2), torch.int32),
             mem_state=Guarded((n, 2), torch.int32))
    p = _path(cfg, n, fov, depth, buffers={k: v.t for k, v in g.items()})
    shape = p.out_shape("fixed_memory", "mask")
    out, norm = Guarded(shape, torch.uint8), Guarded(shape, torch.bfloat16)
    mem = MemoryOracle(n, depth)
    loc = np.zeros((n, 2), np.int32)
    for step in range(7):
        _ingest(p, cfg, rng, step)
        a, ctrl = _actions(n, fov, rng, step)
        c = ctrl if step else np.full(n, RESET, np.uint8)
        p.observe_fixed_memory(a, ctrl=c, out=out.t, norm_out=norm.t)
        _update(a, c, loc, fov, "absolute")
        want = _want(p, mem, loc, fov, c)
    torch.cuda.synchronize()
    assert all(v.intact() for v in list(g.values()) + [out, norm])
    assert np.array_equal(g["loc"].t.cpu().numpy(), loc)
    assert np.array_equal(out.t.cpu().numpy(), want)
    assert torch.equal(norm.t.cpu(), _normalized(out.t, torch.bfloat16))


@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_a_memory_step_is_deterministic(cfg):
    rng = np.random.default_rng(17)
    n, fov = 2500, (30, 30)
    p = _path(cfg, n, fov, 8)
    for step in range(6):
        _ingest(p, cfg, rng, step)
        a, ctrl = _actions(n, fov, rng, step)
        p.observe_fixed_memory(a, ctrl=ctrl if step else "reset")
    torch.cuda.synchronize()
    a, ctrl = _actions(n, fov, rng, 1)
    state0 = [t.clone() for t in (p.loc, p.mem, p.mem_loc, p.mem_state)]
    ref = None
    for rep in range(6):
        for t, s in zip((p.loc, p.mem, p.mem_loc, p.mem_state), state0):
            t.copy_(s)
        out = p.observe_fixed_memory(a, ctrl=ctrl)
        torch.cuda.synchronize()
        snap = [out.clone()] + [t.clone() for t in (p.loc, p.mem, p.mem_loc, p.mem_state)]
        if ref is None:
            ref = snap
        else:
            assert all(torch.equal(x, y) for x, y in zip(ref, snap)), rep


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
def test_normalised_output_equals_agym_normalize(dtype):
    rng = np.random.default_rng(29)
    n, fov = 200, (21, 33)
    p = _path("rgb", n, fov, 4)
    for step in range(5):
        _ingest(p, "rgb", rng, step)
        a, ctrl = _actions(n, fov, rng, step)
        nrm = torch.empty(p.out_shape("fixed_memory", "mask"), dtype=dtype, device="cuda:0")
        out = p.observe_fixed_memory(a, ctrl=ctrl if step else "reset", norm_out=nrm)
        want = p.normalize(out, dtype)
        torch.cuda.synchronize()
        assert torch.equal(nrm, want), step


def test_abi_rejects_invalid_arguments():
    from active_gym_b200 import _lib
    p = _path("atari", 8, (30, 30), 2)
    L, P = _lib.lib(), p._plan
    assert L.agym_plan_memory_bytes(P, 2) == 8 * 2 * 3600 and L.agym_plan_memory_bytes(P, 0) == 0
    assert L.agym_plan_memory_bytes(P, 17) == 0
    out = torch.empty(p.out_shape("fixed_memory", "mask"), dtype=torch.uint8, device="cuda:0")
    ptr = lambda t: t.data_ptr()
    ctrl = torch.full((8,), RESET, dtype=torch.uint8, device="cuda:0")

    def call(depth=2, mem=None, mem_loc=None, mem_state=None):
        return L.agym_observe_fixed_memory(P, ptr(p.ring), ptr(p.head), None, ptr(ctrl), ptr(p.loc), depth,
                                           ptr(p.mem) if mem is None else mem, ptr(p.mem_loc) if mem_loc is None else mem_loc,
                                           ptr(p.mem_state) if mem_state is None else mem_state, ptr(out), None, 0,
                                           torch.cuda.current_stream().cuda_stream)
    # depth outside 1..16, a NULL memory buffer (0 is passed as NULL), a d_mem that is not 16-byte aligned
    for bad in (dict(depth=0), dict(depth=17), dict(mem=0), dict(mem_loc=0), dict(mem_state=0), dict(mem=ptr(p.mem) + 4)):
        assert call(**bad) == -1, bad
    assert call() == 0
    torch.cuda.synchronize()


# ------------------------------------------------------------------------------------------------ env level
def _atari_env(n, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", mask_out=True, fov_memory=3)
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return ag.AtariFixedFovealEnv(args, num_envs=n, source=SyntheticAtariSource(n, device="cuda"))


def _dmc_env(n, grey, device=None, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import DMCPool
    from tests.test_gpu_dmc_rgb import _FakeDMC
    rng = np.random.default_rng(3)
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", frame_stack=3, action_repeat=2,
              grey=grey, mask_out=True, fov_memory=3)
    kw.update(extra)
    args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, **kw)
    return ag.DMCFixedFovealEnv(args, num_envs=n, source=DMCPool(
        args, n if n else 1, env_factory=lambda i: _FakeDMC(rng.integers(0, 256, (7,) + S + (3,), dtype=np.uint8))), device=device)


def _motor(kind, n):
    return np.zeros(n, np.int64) if kind == "atari" else np.zeros((n, 2), np.float32)


def _env(kind, n, **extra):
    return _atari_env(n, **extra) if kind == "atari" else _dmc_env(n, kind == "dmc", **extra)


def _host(v):
    return np.asarray(v.cpu() if isinstance(v, torch.Tensor) else v)


@pytest.mark.parametrize("kind", ["atari", "dmc", "rgb"])
@pytest.mark.parametrize("extra", [{}, {"obs_dtype": torch.float32}, {"obs_dtype": torch.bfloat16}, {"host_obs": True}])
def test_env_returns_the_memory(kind, extra):
    rng = np.random.default_rng(23)
    n = 20
    env = _env(kind, n, **extra)
    K = 4 if kind == "atari" else 3
    frame = (K,) if kind != "rgb" else (K, 3)
    assert env.observation_space.shape == frame + S and env.obs_shape == (n,) + frame + S
    mem = MemoryOracle(n, 3)
    obs, info = env.reset()
    path = env.path
    for step in range(5):
        if step:
            a = rng.integers(0, 55, (n, 2)).astype(np.float64)
            obs, _, _, _, info = env.step({"motor_action": _motor(kind, n), "sensory_action": a})
        torch.cuda.synchronize()
        ctrl = np.full(n, APPLY if step else RESET, np.uint8)
        want = mem.observe(path.ring.cpu().numpy(), path.head.cpu().numpy(), _host(info["fov_loc"]).astype(np.int32),
                           (30, 30), ctrl, rgb=kind == "rgb").reshape((n,) + frame + S)
        u8 = env.last_obs_u8 if extra.get("obs_dtype") is not None else obs
        got = _host(u8)
        assert np.array_equal(got, want), step
        assert np.array_equal(_host(env.fov_memory_count), mem.count())
        if extra.get("obs_dtype") is not None:
            assert obs.dtype == extra["obs_dtype"]
            assert torch.equal(obs.cpu(), _normalized(torch.from_numpy(got), extra["obs_dtype"]))
        if extra.get("host_obs"):
            assert not obs.is_cuda
    env.close()


def test_single_env_adapter_returns_float64_memories():
    from active_gym_b200 import SingleEnvAdapter
    env = SingleEnvAdapter(_env("atari", 1))
    obs, _ = env.reset()
    assert obs.dtype == np.float64 and obs.shape == (4,) + S
    for step in range(4):
        obs, _, _, _, info = env.step({"motor_action": 0, "sensory_action": np.array([10.0 * step, 50.0 - 9 * step])})
        assert obs.dtype == np.float64 and obs.shape == (4,) + S
        assert np.array_equal(np.rint(obs * 255.0).astype(np.uint8), env.env._obs[0].cpu().numpy())
    env.close()


def test_vector_env_autoreset_clears_exactly_the_finished_envs():
    import active_gym_b200 as ag
    from active_gym_b200.sources import PinnedFrameSource
    n = 8
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, fov_size=(30, 30), fov_init_loc=INIT,
                           sensory_action_mode="absolute", mask_out=True, fov_memory=4)
    vec = ag.FovealVectorEnv(ag.AtariFixedFovealEnv(args, num_envs=n, source=PinnedFrameSource(n, pool=3, done_every=3)))
    vec.reset()
    env = vec.env
    count = np.ones(n, np.int32)
    rng = np.random.default_rng(2)
    seen_done = False
    for step in range(9):
        a = {"motor_action": np.zeros(n, np.int64), "sensory_action": rng.integers(0, 55, (n, 2)).astype(np.float64)}
        _, _, term, trunc, _ = vec.step(a)
        fin = np.asarray(term, bool) | np.asarray(trunc, bool)
        seen_done |= bool(fin.any())
        count = np.where(fin, 1, np.minimum(count + 1, 4))
        torch.cuda.synchronize()
        assert np.array_equal(_host(env.fov_memory_count), count), step
    assert seen_done
    vec.close()


def _sampled(n):
    rng = np.random.default_rng(n)
    edges = [0, 1, n - 1, n - 2] + [k for b in range(1024, n, 1024) for k in (b - 1, b)]
    return np.unique(np.concatenate([edges, rng.choice(n, 1024, replace=False)]))


@pytest.mark.parametrize("kind,n", [("atari", 16384), ("rgb", 8192)])
def test_full_size_parity_on_sampled_envs(kind, n):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource, SyntheticDMCSource
    rng = np.random.default_rng(41)
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", mask_out=True, fov_memory=8)
    if kind == "atari":
        env = ag.AtariFixedFovealEnv(ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw), num_envs=n,
                                     source=SyntheticAtariSource(n, device="cuda"))
    else:
        args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, frame_stack=3, action_repeat=2,
                             grey=False, **kw)
        env = ag.DMCFixedFovealEnv(args, num_envs=n, source=SyntheticDMCSource(n, device="cuda"))
    K = 4 if kind == "atari" else 3
    frame = (K,) if kind != "rgb" else (K, 3)
    idx = _sampled(n)
    mem = MemoryOracle(len(idx), 8)
    obs, info = env.reset()
    path = env.path
    for step in range(10):
        if step:
            a = rng.integers(0, 55, (n, 2)).astype(np.float64)
            obs, _, _, _, info = env.step({"motor_action": _motor(kind, n), "sensory_action": a})
        torch.cuda.synchronize()
        ring, head = path.ring[torch.from_numpy(idx).cuda()].cpu().numpy(), path.head.cpu().numpy()[idx]
        want = mem.observe(ring, head, _host(info["fov_loc"])[idx].astype(np.int32), (30, 30),
                           np.full(len(idx), APPLY if step else RESET, np.uint8), rgb=kind == "rgb")
        assert np.array_equal(_host(obs)[idx], want.reshape((len(idx),) + frame + S)), step
    env.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more GPUs")
def test_sharded_learner_device_receives_the_memory():
    from active_gym_b200.vector import ShardedVecEnv
    n = 40
    venv = ShardedVecEnv(lambda m, dev, lo, hi: _dmc_env(m, True, device=dev), n, devices=["cuda:0", "cuda:1"],
                         learner_device="cuda:0")
    obs, _ = venv.reset()
    assert tuple(obs.shape) == (n, 3) + S and obs.device == torch.device("cuda:0")
    mems = [MemoryOracle(e.num_envs, 3) for e in venv.envs]
    rng = np.random.default_rng(1)
    for step in range(3):
        if step:
            a = {"motor_action": np.zeros((n, 2), np.float32), "sensory_action": rng.integers(0, 55, (n, 2)).astype(np.float64)}
            obs, *_ = venv.step(a)
        torch.cuda.synchronize("cuda:0")
        torch.cuda.synchronize("cuda:1")
        lo = 0
        for e, m in zip(venv.envs, mems):
            p = e.path
            want = m.observe(p.ring.cpu().numpy(), p.head.cpu().numpy(), p.loc.cpu().numpy(), (30, 30),
                             np.full(e.num_envs, APPLY if step else RESET, np.uint8))
            assert np.array_equal(obs[lo:lo + e.num_envs].cpu().numpy(), want), step
            lo += e.num_envs
    venv.close()
