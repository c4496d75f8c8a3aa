"""GPU: the fixed fovea's memory merged by pasting (``fov_memory_merge="paste"``, ``agym_observe_fixed_memory_paste``)
against the composed C oracle (``tests/memory_paste_oracle.py``): pasted pixels bit for bit, the periphery within
0.5 LSB + 0.01 of the oracle's float value, ``loc`` and the memory's state equal to the oracle's.

Grey Atari (K=4), grey DMC (K=3) and RGB DMC (K*C=9); the oracle reads the ring the kernels ingested (ingest is pinned
elsewhere), so these tests isolate the observe step and the memory it keeps."""
import numpy as np
import pytest
import torch

from tests.memory_paste_oracle import APPLY, KEEP, RESET, PasteOracle
from tests.test_gpu_fovea_memory import (CFG, INIT, Guarded, _actions, _host, _ingest, _motor, _normalized, _sampled,
                                         _update)

pytestmark = pytest.mark.gpu

S = (84, 84)
TOL = 0.5 + 1e-2
GUARD, CANARY = 4096, 0xA5


def _path(cfg, n, fov, depth, mode="absolute", per=(20, 20), antialias=True, buffers=None):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    K, C, raw = CFG[cfg]
    kw = {} if cfg == "atari" else {"luma": LUMA_DMC}
    return ObservationPath(n, K, S, raw, fov_size=fov, fov_init_loc=INIT, sensory_action_mode=mode,
                           sensory_action_space=(-10.0, 10.0), device="cuda:0", channels=C, buffers=buffers,
                           peripheral_res=per, antialias=antialias, fov_memory=depth, **kw)


def _planes(t):
    """(n, K[, 3], S_h, S_w) -> numpy (n, P, S_h, S_w)."""
    a = t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
    return a.reshape((a.shape[0], -1) + a.shape[-2:])


def _want(p, mem, loc, fov, ctrl, per, envs=None):
    ring, head = p.ring.cpu().numpy(), p.head.cpu().numpy()
    if envs is not None:
        ring, head = ring[envs], head[envs]
    return mem.observe(ring, head, loc, fov, ctrl, peripheral_res=per)


def _check(got, want, mem, fov, what):
    """Pasted pixels exact; the zero background exact; the periphery within TOL."""
    got = _planes(got).astype(np.float64)
    m = np.broadcast_to(mem.pasted(S, fov)[:, None], got.shape)
    assert np.array_equal(got[m], want[m]), what
    assert np.abs(got - want).max() <= TOL, what


def _ctrl(ctrl, step, n):
    return ctrl if step else np.full(n, RESET, np.uint8)


def _run_parity(cfg, fov, depth, mode, background, per=(20, 20), antialias=True, n=131, steps=12):
    from oracle import agym_oracle as orc
    rng = np.random.default_rng(hash((cfg, fov, depth, mode, background, per, antialias)) % 2**32)
    p = _path(cfg, n, fov, depth, mode, per=per, antialias=antialias)
    mem = PasteOracle(n, depth)
    loc = np.zeros((n, 2), np.int32)
    op = per if background == "periphery" else None
    orc.set_antialias(antialias)
    try:
        for step in range(steps):
            _ingest(p, cfg, rng, step)
            a, ctrl = _actions(n, fov, rng, step, mode)
            out = p.observe_memory_paste(a, ctrl=ctrl if step else "reset", background=background)
            c = _ctrl(ctrl, step, n)
            _update(a, c, loc, fov, mode)
            want = _want(p, mem, loc, fov, c, op)
            torch.cuda.synchronize()
            assert np.array_equal(p.loc.cpu().numpy(), loc), step
            _check(out, want, mem, fov, step)
            assert np.array_equal(p.mem_state[:, 1].cpu().numpy(), mem.count()), step
    finally:
        orc.set_antialias(True)


@pytest.mark.parametrize("cfg", ["atari", "dmc", "rgb"])
@pytest.mark.parametrize("fov", [(30, 30), (21, 33), (50, 28)])
@pytest.mark.parametrize("depth", [1, 2, 3, 8, 16])
@pytest.mark.parametrize("mode", ["absolute", "relative"])
@pytest.mark.parametrize("background", ["zero", "periphery"])
def test_paste_matches_the_oracle(cfg, fov, depth, mode, background):
    _run_parity(cfg, fov, depth, mode, background, steps=12 if depth < 16 else 20)


EXTRA = [("atari", (24, 40), (16, 24), True),    # the geometry of the golden atari_peripheral_abs_p16x24
         ("dmc", (30, 30), (15, 21), True),      # a squeeze of 315 floats: loaded without a bulk copy
         ("atari", (30, 30), (84, 42), True),    # expand tables that are not two-tap lerps: the generic passes
         ("atari", (30, 30), (20, 20), False),   # plain bilinear
         ("rgb", (21, 33), (16, 24), False)]


@pytest.mark.parametrize("case", EXTRA, ids=[f"{c}-{f[0]}x{f[1]}-p{p[0]}x{p[1]}-aa{int(a)}" for c, f, p, a in EXTRA])
@pytest.mark.parametrize("background", ["zero", "periphery"])
def test_paste_matches_the_oracle_at_other_geometries(case, background):
    cfg, fov, per, aa = case
    _run_parity(cfg, fov, 3, "absolute", background, per=per, antialias=aa, n=97, steps=8)


@pytest.mark.parametrize("cfg", ["atari", "dmc", "rgb"])
def test_depth_one_is_mask_out_and_the_peripheral_view(cfg):
    """M = 1, every env pushing: zero background = observe_fixed("mask") and periphery = observe_peripheral, bit for bit
    (RGB's peripheral call runs k_observe_peripheral_v2, which adds the W taps in another order: within 1)."""
    rng = np.random.default_rng(3)
    n, fov = 300, (21, 33)
    z, pp, ref = _path(cfg, n, fov, 1), _path(cfg, n, fov, 1), _path(cfg, n, fov, 0)
    for step in range(8):
        seed = int(rng.integers(1 << 30))
        for p in (z, pp, ref):
            _ingest(p, cfg, np.random.default_rng(seed), step)
        a, ctrl = _actions(n, fov, rng, step)
        ctrl = None if ctrl is None else np.where(ctrl == KEEP, APPLY, ctrl).astype(np.uint8)
        c = ctrl if step else "reset"
        oz = z.observe_memory_paste(a, ctrl=c, background="zero")
        op = pp.observe_memory_paste(a, ctrl=c, background="periphery")
        mask = ref.observe_fixed(a, variant="mask", ctrl=c)
        torch.cuda.synchronize()
        ref.loc.copy_(z.loc)
        pv = ref.observe_peripheral(None, ctrl=np.full(n, KEEP, np.uint8))
        torch.cuda.synchronize()
        assert torch.equal(z.loc, pp.loc)
        assert torch.equal(oz, mask), step
        if cfg == "rgb":
            assert (op.int() - pv.int()).abs().max().item() <= 1, step
        else:
            assert torch.equal(op, pv), step


@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_zero_background_with_disjoint_windows_is_the_max_memory(cfg):
    """Windows cycling through the four corners never overlap while M = 4 of them are held."""
    rng = np.random.default_rng(11)
    n, fov = 257, (30, 30)
    pa, mx = _path(cfg, n, fov, 4), _path(cfg, n, fov, 4)
    corners = np.array([[0, 0], [0, 54], [54, 0], [54, 54]], np.float64)
    for step in range(9):
        seed = int(rng.integers(1 << 30))
        for p in (pa, mx):
            _ingest(p, cfg, np.random.default_rng(seed), step)
        a = np.tile(corners[step % 4], (n, 1))
        c = None if step else "reset"
        o1 = pa.observe_memory_paste(a, ctrl=c, background="zero")
        o2 = mx.observe_fixed_memory(a, ctrl=c)
        torch.cuda.synchronize()
        assert torch.equal(o1, o2), step


@pytest.mark.parametrize("background", ["zero", "periphery"])
@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_memory_buffers_equal_the_max_memory(cfg, background):
    """After the same sequence of calls, mem, mem_loc and mem_state hold the same bytes under either merge; KEEP repeats
    the output."""
    rng = np.random.default_rng(13)
    n, fov = 300, (50, 28)
    pa, mx = _path(cfg, n, fov, 8), _path(cfg, n, fov, 8)
    for step in range(12):
        seed = int(rng.integers(1 << 30))
        for p in (pa, mx):
            _ingest(p, cfg, np.random.default_rng(seed), step)
        a, ctrl = _actions(n, fov, rng, step)
        c = ctrl if step else "reset"
        o = pa.observe_memory_paste(a, ctrl=c, background=background)
        mx.observe_fixed_memory(a, ctrl=c)
        torch.cuda.synchronize()
        for x, y in ((pa.loc, mx.loc), (pa.mem, mx.mem), (pa.mem_loc, mx.mem_loc), (pa.mem_state, mx.mem_state)):
            assert torch.equal(x, y), step
        again = pa.observe_memory_paste(None, ctrl=np.full(n, KEEP, np.uint8), background=background)
        torch.cuda.synchronize()
        assert torch.equal(again, o), step


@pytest.mark.parametrize("background", ["zero", "periphery"])
@pytest.mark.parametrize("offset", [1, 3, 4])
def test_unaligned_output_equals_the_aligned_output(offset, background):
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
        want = a_p.observe_memory_paste(a, ctrl=ctrl if step else "reset", background=background)
        u_p.observe_memory_paste(a, ctrl=ctrl if step else "reset", background=background, out=view)
        torch.cuda.synchronize()
        assert torch.equal(view, want), step
    assert bool((raw[:GUARD + offset] == CANARY).all()) and bool((raw[GUARD + offset + nb:] == CANARY).all())


@pytest.mark.parametrize("cfg", ["atari", "rgb"])
@pytest.mark.parametrize("n", [1, 37, 333, 1001])
def test_paste_stays_inside_its_buffers(cfg, n):
    rng = np.random.default_rng(n)
    fov, depth, per = (50, 28), 3, (20, 20)
    K, C, _ = CFG[cfg]
    P = K * C
    E = (P * fov[0] * fov[1] + 15) // 16 * 16
    g = dict(ring=Guarded((n, P) + S, torch.uint8), head=Guarded((n,), torch.int32, P - 1),
             loc=Guarded((n, 2), torch.int32), res=Guarded((n, 2), torch.int32), pcache=Guarded((n, P) + per, torch.float32),
             mem=Guarded((n, depth, E), torch.uint8), mem_loc=Guarded((n, depth, 2), torch.int32),
             mem_state=Guarded((n, 2), torch.int32))
    p = _path(cfg, n, fov, depth, per=per, buffers={k: v.t for k, v in g.items()})
    shape = p.out_shape("fixed_memory", "mask")
    out, norm = Guarded(shape, torch.uint8), Guarded(shape, torch.bfloat16)
    mem = PasteOracle(n, depth)
    loc = np.zeros((n, 2), np.int32)
    for step in range(7):
        _ingest(p, cfg, rng, step)
        a, ctrl = _actions(n, fov, rng, step)
        c = _ctrl(ctrl, step, n)
        p.observe_memory_paste(a, ctrl=c, background="periphery", out=out.t, norm_out=norm.t)
        _update(a, c, loc, fov, "absolute")
        want = _want(p, mem, loc, fov, c, per)
    torch.cuda.synchronize()
    assert all(v.intact() for v in list(g.values()) + [out, norm])
    assert np.array_equal(g["loc"].t.cpu().numpy(), loc)
    _check(out.t, want, mem, fov, "final")
    assert torch.equal(norm.t.cpu(), _normalized(out.t, torch.bfloat16))


@pytest.mark.parametrize("background", ["zero", "periphery"])
@pytest.mark.parametrize("cfg", ["atari", "rgb"])
def test_a_paste_step_is_deterministic(cfg, background):
    rng = np.random.default_rng(17)
    n, fov = 2500, (30, 30)
    p = _path(cfg, n, fov, 8)
    for step in range(6):
        _ingest(p, cfg, rng, step)
        a, ctrl = _actions(n, fov, rng, step)
        p.observe_memory_paste(a, ctrl=ctrl if step else "reset", background=background)
    torch.cuda.synchronize()
    a, ctrl = _actions(n, fov, rng, 1)
    state0 = [t.clone() for t in (p.loc, p.mem, p.mem_loc, p.mem_state)]
    ref = None
    for rep in range(6):
        for t, s in zip((p.loc, p.mem, p.mem_loc, p.mem_state), state0):
            t.copy_(s)
        out = p.observe_memory_paste(a, ctrl=ctrl, background=background)
        torch.cuda.synchronize()
        snap = [out.clone()] + [t.clone() for t in (p.loc, p.mem, p.mem_loc, p.mem_state)]
        if ref is None:
            ref = snap
        else:
            assert all(torch.equal(x, y) for x, y in zip(ref, snap)), rep


@pytest.mark.parametrize("dtype", [torch.float32, torch.float16, torch.bfloat16])
@pytest.mark.parametrize("background", ["zero", "periphery"])
def test_normalised_output_equals_agym_normalize(dtype, background):
    rng = np.random.default_rng(29)
    n, fov = 200, (21, 33)
    p = _path("rgb", n, fov, 4)
    for step in range(5):
        _ingest(p, "rgb", rng, step)
        a, ctrl = _actions(n, fov, rng, step)
        nrm = torch.empty(p.out_shape("fixed_memory", "mask"), dtype=dtype, device="cuda:0")
        out = p.observe_memory_paste(a, ctrl=ctrl if step else "reset", background=background, norm_out=nrm)
        want = p.normalize(out, dtype)
        torch.cuda.synchronize()
        assert torch.equal(nrm, want), step


def test_abi_rejects_invalid_arguments():
    from active_gym_b200 import _lib
    p = _path("atari", 8, (30, 30), 2)
    nop = _path("atari", 8, (30, 30), 2, per=None)
    L = _lib.lib()
    out = torch.empty(p.out_shape("fixed_memory", "mask"), dtype=torch.uint8, device="cuda:0")
    ptr = lambda t: t.data_ptr()
    ctrl = torch.full((8,), RESET, dtype=torch.uint8, device="cuda:0")

    def call(path=p, depth=2, bg=_lib.BG_PERIPHERY, pcache=None, mem=None, mem_loc=None, mem_state=None):
        pc = (ptr(path.pcache) if path.pcache is not None else None) if pcache is None else pcache
        return L.agym_observe_fixed_memory_paste(
            path._plan, ptr(path.ring), ptr(path.head), pc, None, ptr(ctrl), ptr(path.loc), depth, bg,
            ptr(path.mem) if mem is None else mem, ptr(path.mem_loc) if mem_loc is None else mem_loc,
            ptr(path.mem_state) if mem_state is None else mem_state, ptr(out), None, 0, torch.cuda.current_stream().cuda_stream)
    # depth outside 1..16, a NULL memory buffer (0 is passed as NULL), a d_mem that is not 16-byte aligned, an unknown
    # background, the periphery with a NULL squeeze cache or on a plan without a periphery
    for bad in (dict(depth=0), dict(depth=17), dict(mem=0), dict(mem_loc=0), dict(mem_state=0), dict(mem=ptr(p.mem) + 4),
                dict(bg=2), dict(bg=-1), dict(pcache=0), dict(path=nop)):
        assert call(**bad) == -1, bad
    # a plan without a fovea
    from active_gym_b200 import ObservationPath
    nf = ObservationPath(8, 4, S, (210, 160, 1), device="cuda:0")
    assert L.agym_observe_fixed_memory_paste(nf._plan, ptr(nf.ring), ptr(nf.head), None, None, ptr(ctrl), ptr(nf.loc), 2,
                                             _lib.BG_ZERO, ptr(p.mem), ptr(p.mem_loc), ptr(p.mem_state), ptr(out), None, 0,
                                             torch.cuda.current_stream().cuda_stream) == -1
    assert call() == 0 and call(bg=_lib.BG_ZERO, pcache=0) == 0 and call(path=nop, bg=_lib.BG_ZERO) == 0
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="background"):
        p.observe_memory_paste(None, ctrl="reset", background="max")
    with pytest.raises(ValueError, match="cache"):
        nop.observe_memory_paste(None, ctrl="reset", background="periphery")


# ------------------------------------------------------------------------------------------------ env level
def _atari_env(n, wrapper="AtariFixedFovealPeripheralEnv", **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", fov_memory=3, fov_memory_merge="paste",
              peripheral_res=(20, 20), mask_out=wrapper == "AtariFixedFovealEnv")
    kw.update(extra)
    args = ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw)
    return getattr(ag, wrapper)(args, num_envs=n, source=SyntheticAtariSource(n, device="cuda"))


def _dmc_env(n, grey, device=None, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import DMCPool
    from tests.test_gpu_dmc_rgb import _FakeDMC
    rng = np.random.default_rng(3)
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="absolute", frame_stack=3, action_repeat=2,
              grey=grey, fov_memory=3, fov_memory_merge="paste", peripheral_res=(20, 20))
    kw.update(extra)
    args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, **kw)
    return ag.DMCFixedFovealPeripheralEnv(args, num_envs=n, source=DMCPool(
        args, n if n else 1, env_factory=lambda i: _FakeDMC(rng.integers(0, 256, (7,) + S + (3,), dtype=np.uint8))), device=device)


def _env(kind, n, **extra):
    return _atari_env(n, **extra) if kind == "atari" else _dmc_env(n, kind == "dmc", **extra)


@pytest.mark.parametrize("kind", ["atari", "dmc", "rgb", "atari_fixed"])
@pytest.mark.parametrize("extra", [{}, {"obs_dtype": torch.float32}, {"obs_dtype": torch.bfloat16}, {"host_obs": True}])
def test_env_returns_the_memory(kind, extra):
    rng = np.random.default_rng(23)
    n = 20
    fixed = kind == "atari_fixed"
    env = _atari_env(n, wrapper="AtariFixedFovealEnv", **extra) if fixed else _env(kind, n, **extra)
    K = 3 if kind in ("dmc", "rgb") else 4
    frame = (K,) if kind != "rgb" else (K, 3)
    assert env.observation_space.shape == frame + S and env.obs_shape == (n,) + frame + S
    mem = PasteOracle(n, 3)
    per = None if fixed else (20, 20)
    obs, info = env.reset()
    path = env.path
    for step in range(5):
        if step:
            a = rng.integers(0, 55, (n, 2)).astype(np.float64)
            obs, _, _, _, info = env.step({"motor_action": _motor("dmc" if kind in ("dmc", "rgb") else "atari", n),
                                           "sensory_action": a})
        torch.cuda.synchronize()
        ctrl = np.full(n, APPLY if step else RESET, np.uint8)
        want = mem.observe(path.ring.cpu().numpy(), path.head.cpu().numpy(), _host(info["fov_loc"]).astype(np.int32),
                           (30, 30), ctrl, peripheral_res=per)
        u8 = env.last_obs_u8 if extra.get("obs_dtype") is not None else obs
        got = _host(u8)
        assert got.shape == (n,) + frame + S
        _check(got, want, mem, (30, 30), step)
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
                           sensory_action_mode="absolute", peripheral_res=(20, 20), fov_memory=4, fov_memory_merge="paste")
    vec = ag.FovealVectorEnv(ag.AtariFixedFovealPeripheralEnv(args, num_envs=n, source=PinnedFrameSource(n, pool=3, done_every=3)))
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


@pytest.mark.parametrize("kind,n", [("atari", 16384), ("rgb", 8192)])
def test_full_size_parity_on_sampled_envs(kind, n):
    import active_gym_b200 as ag
    from active_gym_b200.sources import SyntheticAtariSource, SyntheticDMCSource
    rng = np.random.default_rng(41)
    kw = dict(fov_size=(30, 30), fov_init_loc=INIT, sensory_action_mode="relative", sensory_action_space=(-10.0, 10.0),
              peripheral_res=(20, 20), fov_memory=8, fov_memory_merge="paste")
    if kind == "atari":
        env = ag.AtariFixedFovealPeripheralEnv(ag.AtariEnvArgs(game="boxing", seed=0, obs_size=S, **kw), num_envs=n,
                                               source=SyntheticAtariSource(n, device="cuda"))
    else:
        args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, frame_stack=3, action_repeat=2,
                             grey=False, **kw)
        env = ag.DMCFixedFovealPeripheralEnv(args, num_envs=n, source=SyntheticDMCSource(n, device="cuda"))
    idx = _sampled(n)
    mem = PasteOracle(len(idx), 8)
    obs, info = env.reset()
    path = env.path
    for step in range(10):
        if step:
            a = rng.integers(-14, 15, (n, 2)).astype(np.float64)
            obs, _, _, _, info = env.step({"motor_action": _motor(kind, n), "sensory_action": a})
        torch.cuda.synchronize()
        ring, head = path.ring[torch.from_numpy(idx).cuda()].cpu().numpy(), path.head.cpu().numpy()[idx]
        want = mem.observe(ring, head, _host(info["fov_loc"])[idx].astype(np.int32), (30, 30),
                           np.full(len(idx), APPLY if step else RESET, np.uint8), peripheral_res=(20, 20))
        _check(_host(obs)[idx], want, mem, (30, 30), step)
    env.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more GPUs")
def test_sharded_learner_device_receives_the_memory():
    from active_gym_b200.vector import ShardedVecEnv
    n = 40
    venv = ShardedVecEnv(lambda m, dev, lo, hi: _dmc_env(m, True, device=dev), n, devices=["cuda:0", "cuda:1"],
                         learner_device="cuda:0")
    obs, _ = venv.reset()
    assert tuple(obs.shape) == (n, 3) + S and obs.device == torch.device("cuda:0")
    mems = [PasteOracle(e.num_envs, 3) for e in venv.envs]
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
                             np.full(e.num_envs, APPLY if step else RESET, np.uint8), peripheral_res=(20, 20))
            _check(obs[lo:lo + e.num_envs], want, m, (30, 30), step)
            lo += e.num_envs
    venv.close()
