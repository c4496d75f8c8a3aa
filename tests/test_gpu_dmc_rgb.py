"""GPU: DMC ``grey=False`` — the RGB ingest kernel and every observe path on a ring of frame_stack * 3 planes, against
the composed oracle (tests/rgb_oracle.py, pinned to the reference by tests/test_dmc_rgb_reference.py).

Tolerances are those of the grey path: bit exact for ingest, stack, crop and mask; within TOL for resampled pixels;
fov_loc / fov_res exact."""
import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc
from oracle import ref_harness as rh
from tests import rgb_oracle as rgb

pytestmark = pytest.mark.gpu

TOL = 0.5 + 1e-2
S, K, FOV, PERIPH = (84, 84), 3, (30, 30), (20, 20)
GUARD, CANARY = 4096, 0xA5


def _path(n, fov=FOV, periph=None, mode="absolute", channels=3, cache=True, buffers=None):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    return ObservationPath(n, K, S, S + (3,), luma=LUMA_DMC, fov_size=fov, peripheral_res=periph, sensory_action_mode=mode,
                           sensory_action_space=(-10.0, 10.0), device="cuda:0", cache_peripheral=cache, channels=channels,
                           buffers=buffers)


def _flags(n, step, rng):
    """Ragged DMC flags: hard reset first, then pushes with idle envs and hard resets mixed in."""
    fl = np.full(n, 5 if step == 0 else 1, np.uint8)
    if step:
        fl[rng.random(n) < 0.15] = 8
        fl[rng.random(n) < 0.1] = 5
    return fl


def _frames(n, rng):
    return rng.integers(0, 256, (n,) + S + (3,), dtype=np.uint8)


def _edge_actions(n, rng, hi):
    a = rng.integers(0, hi + 1, (n, 2)).astype(np.float64)
    a[0::9] = (0, 0); a[1::9] = (hi, hi); a[2::9] = (hi, 0); a[3::9] = (-1e6, 1e6)
    return a


def _np(t):
    return t.cpu().numpy()


@pytest.mark.parametrize("n", [1, 37, 1001])
def test_ingest_and_stack_are_bit_exact_with_head_and_cache(n):
    rng = np.random.default_rng(n)
    p = _path(n, periph=PERIPH)
    ref = _path(n, periph=PERIPH, cache=False)   # cache refresh checked through the cached vs uncached peripheral below
    assert tuple(p.ring.shape) == (n, 3 * K) + S and tuple(p.pcache.shape) == (n, 3 * K) + PERIPH
    assert _np(p.head).tolist() == [3 * K - 1] * n
    ring, head = rgb.new_state(n, K, S)
    for step in range(2 * K + 1):
        f, fl = _frames(n, rng), _flags(n, step, rng)
        p.ingest_dmc(f, fl)
        ref.ingest_dmc(f, fl)
        rgb.ingest_dmc_rgb(f, fl, ring, head)
        torch.cuda.synchronize()
        assert np.array_equal(_np(p.ring), ring) and np.array_equal(_np(p.head), head), step
        st = p.stack()
        assert tuple(st.shape) == (n, K, 3) + S
        assert np.array_equal(_np(st), rgb.stack(ring, head))
    loc = np.zeros((n, 2), np.int32)
    p.observe_peripheral(None, ctrl="reset")
    ref.observe_peripheral(None, ctrl="reset", use_cache=False)
    a = _edge_actions(n, rng, 54)
    got, want = p.observe_peripheral(a), ref.observe_peripheral(a, use_cache=False)
    orc.update_loc(a, loc, obs_size=S, fov_size=FOV)
    o = rgb.observe_peripheral(ring, head, loc, FOV, PERIPH)
    assert np.abs(_np(got).astype(np.float64) - o).max() <= TOL
    assert np.abs(_np(want).astype(np.float64) - o).max() <= TOL


def _drive(n, kind, variant, mode, rng, steps=4, cache=True, norm=None):
    """n envs of one workload through the kernels and the oracle; returns the last outputs of both."""
    p = _path(n, periph=PERIPH if kind == "peripheral" else None, mode=mode, cache=cache)
    ring, head = rgb.new_state(n, K, S)
    loc = np.zeros((n, 2), np.int32)
    res = np.tile(np.array([FOV], np.int32), (n, 1))
    for step in range(steps):
        f, fl = _frames(n, rng), _flags(n, step, rng)
        p.ingest_dmc(f, fl)
        rgb.ingest_dmc_rgb(f, fl, ring, head)
        at = None
        if kind == "flexible":
            at = rng.integers(0, 2, n).astype(np.int32)
            a = np.where(at[:, None] == 1, rng.integers(1, 85, (n, 2)), _edge_actions(n, rng, 83)).astype(np.float64)
        elif mode == "relative":
            a = rng.uniform(-14, 14, (n, 2))
        else:
            a = _edge_actions(n, rng, 54)
        nrm = None if norm is None else torch.empty(p.out_shape(kind, variant), dtype=norm, device="cuda:0")
        if kind == "peripheral":
            out = p.observe_peripheral(a, use_cache=cache, norm_out=nrm)
        elif kind == "flexible":
            out = p.observe_flexible(a, at, variant=variant, norm_out=nrm)
        else:
            out = p.observe_fixed(a, variant=variant, norm_out=nrm)
        orc.update_loc(a, loc, obs_size=S, fov_size=FOV, relative=mode == "relative", lo=-10.0, hi=10.0,
                       atype=at, res=res if kind == "flexible" else None)
    torch.cuda.synchronize()
    assert np.array_equal(_np(p.loc), loc)
    if kind == "flexible":
        assert np.array_equal(_np(p.res), res)
        want = rgb.observe_flexible(ring, head, loc, res, FOV, variant=variant)
    elif kind == "peripheral":
        want = rgb.observe_peripheral(ring, head, loc, FOV, PERIPH)
    else:
        want = rgb.observe_fixed(ring, head, loc, FOV, variant=variant)
    return p, out, want, nrm


@pytest.mark.parametrize("kind,variant,mode,cache", [
    ("fixed", "crop", "absolute", True), ("fixed", "crop", "relative", True), ("fixed", "mask", "absolute", True),
    ("fixed", "resize_full", "relative", True), ("peripheral", "mask", "relative", True),
    ("peripheral", "mask", "absolute", False), ("flexible", "mask", "absolute", True),
    ("flexible", "crop", "absolute", True), ("flexible", "resize_full", "absolute", True)])
def test_every_observe_variant_matches_the_oracle(kind, variant, mode, cache):
    rng = np.random.default_rng(sum(map(ord, kind + variant + mode)) + int(cache))
    n = 333
    p, out, want, nrm = _drive(n, kind, variant, mode, rng, cache=cache, norm=torch.float32)
    got = _np(out)
    assert got.shape == want.shape and got.shape[1:3] == (K, 3)
    if want.dtype == np.uint8:
        assert np.array_equal(got, want)
    else:
        assert np.abs(got.astype(np.float64) - want).max() <= TOL
    assert np.array_equal(_np(nrm), (got.astype(np.float32) / np.float32(255)))


@pytest.mark.parametrize("kind,variant", [("fixed", "crop"), ("fixed", "mask"), ("fixed", "resize_full"),
                                          ("peripheral", "mask"), ("flexible", "mask"), ("flexible", "crop")])
def test_channel_replicated_frames_give_the_grey_outputs_three_times(kind, variant):
    rng = np.random.default_rng(5)
    n = 257
    periph = PERIPH if kind == "peripheral" else None
    p3, p1 = _path(n, periph=periph, mode="relative"), _path(n, periph=periph, mode="relative", channels=1)
    for step in range(K + 2):
        g = rng.integers(0, 256, (n,) + S, dtype=np.uint8)
        f = np.repeat(g[..., None], 3, axis=-1)
        fl = _flags(n, step, rng)
        at = rng.integers(0, 2, n).astype(np.int32)
        a = (np.where(at[:, None] == 1, rng.integers(20, 51, (n, 2)), rng.integers(0, 55, (n, 2))) if kind == "flexible"
             else rng.uniform(-14, 14, (n, 2))).astype(np.float64)
        outs = []
        for p in (p3, p1):
            p.ingest_dmc(f, fl)
            if kind == "peripheral":
                outs.append(p.observe_peripheral(a))
            elif kind == "flexible":
                outs.append(p.observe_flexible(a, at, variant=variant))
            else:
                outs.append(p.observe_fixed(a, variant=variant))
        torch.cuda.synchronize()
        o3, o1 = _np(outs[0]), _np(outs[1])
        assert o3.shape == o1.shape[:2] + (3,) + o1.shape[2:]
        assert np.array_equal(o3, np.repeat(o1[:, :, None], 3, axis=2)), step
        assert np.array_equal(_np(p3.loc), _np(p1.loc)) and np.array_equal(_np(p3.res), _np(p1.res))


class Guarded:
    def __init__(self, shape, dtype, fill=0):
        n = int(np.prod(shape)) * torch.empty((), dtype=dtype).element_size()
        self.raw = torch.full((GUARD + n + (-n) % 256 + GUARD,), CANARY, dtype=torch.uint8, device="cuda:0")
        self.t = self.raw[GUARD:GUARD + n].view(dtype).view(shape)
        self.t.fill_(fill)
        self.n = n

    def intact(self):
        return bool((self.raw[:GUARD] == CANARY).all()) and bool((self.raw[GUARD + self.n:] == CANARY).all())


@pytest.mark.parametrize("n", [1, 37, 333, 1001])
def test_every_kernel_stays_inside_its_buffers(n):
    rng = np.random.default_rng(n)
    P = 3 * K
    g = dict(ring=Guarded((n, P) + S, torch.uint8), head=Guarded((n,), torch.int32, P - 1),
             loc=Guarded((n, 2), torch.int32), res=Guarded((n, 2), torch.int32), pcache=Guarded((n, P) + PERIPH, torch.float32))
    g["res"].t[:, 0], g["res"].t[:, 1] = FOV
    p = _path(n, periph=PERIPH, buffers={k: v.t for k, v in g.items()})
    outs = {"crop": Guarded((n, K, 3) + FOV, torch.uint8), "mask": Guarded((n, K, 3) + S, torch.uint8),
            "periph": Guarded((n, K, 3) + S, torch.uint8), "flex": Guarded((n, K, 3) + S, torch.uint8),
            "stack": Guarded((n, K, 3) + S, torch.uint8)}
    norms = {"crop": Guarded((n, K, 3) + FOV, torch.float16), "periph": Guarded((n, K, 3) + S, torch.float32),
             "flex": Guarded((n, K, 3) + S, torch.bfloat16)}
    ring, head = rgb.new_state(n, K, S)
    loc = np.zeros((n, 2), np.int32)
    res = np.tile(np.array([FOV], np.int32), (n, 1))
    for step in range(4):
        f, fl = _frames(n, rng), _flags(n, step, rng)
        p.ingest_dmc(f, fl)
        rgb.ingest_dmc_rgb(f, fl, ring, head)
        a = _edge_actions(n, rng, 54)
        p.observe_fixed(a, out=outs["crop"].t, norm_out=norms["crop"].t)
        orc.update_loc(a, loc, obs_size=S, fov_size=FOV)
        loc_fixed = loc.copy()   # what the mask and the peripheral view below see; the flexible step moves loc again
        keep = np.full(n, 2, np.uint8)
        p.observe_fixed(None, variant="mask", ctrl=keep, out=outs["mask"].t)
        p.observe_peripheral(None, ctrl=keep, out=outs["periph"].t, norm_out=norms["periph"].t)
        at = rng.integers(0, 2, n).astype(np.int32)
        fa = np.where(at[:, None] == 1, rng.integers(1, 85, (n, 2)), _edge_actions(n, rng, 83)).astype(np.float64)
        if step == 2 and n >= 6:
            fa[:6] = [[1, 1], [84, 84], [84, 1], [1, 84], [31, 2], [2, 31]]
            at[:6] = 1
        p.observe_flexible(fa, at, variant="mask", out=outs["flex"].t, norm_out=norms["flex"].t)
        orc.update_loc(fa, loc, obs_size=S, fov_size=FOV, atype=at, res=res)
        p.stack(out=outs["stack"].t)
    torch.cuda.synchronize()
    assert all(v.intact() for v in list(g.values()) + list(outs.values()) + list(norms.values()))
    assert np.array_equal(_np(g["ring"].t), ring) and np.array_equal(_np(g["head"].t), head)
    assert np.array_equal(_np(g["loc"].t), loc) and np.array_equal(_np(g["res"].t), res)
    assert np.array_equal(_np(outs["stack"].t), rgb.stack(ring, head))
    assert np.array_equal(_np(outs["mask"].t), rgb.observe_fixed(ring, head, loc_fixed, FOV, variant="mask"))
    assert np.abs(_np(outs["periph"].t).astype(np.float64) - rgb.observe_peripheral(ring, head, loc_fixed, FOV, PERIPH)).max() <= TOL
    assert np.abs(_np(outs["flex"].t).astype(np.float64) - rgb.observe_flexible(ring, head, loc, res, FOV)).max() <= TOL


@pytest.mark.parametrize("kind", ["ingest", "fixed", "peripheral", "flexible"])
def test_a_step_is_deterministic(kind):
    rng = np.random.default_rng(17)
    n = 2500
    p = _path(n, periph=PERIPH if kind == "peripheral" else None, mode="relative" if kind != "flexible" else "absolute")
    p.ingest_dmc(_frames(n, rng), np.full(n, 5, np.uint8))
    for _ in range(K):
        p.ingest_dmc(_frames(n, rng), np.full(n, 1, np.uint8))
    torch.cuda.synchronize()
    state = [t for t in (p.ring, p.head, p.loc, p.res, p.pcache) if t is not None]
    state0 = [t.clone() for t in state]
    f, fl = _frames(n, rng), _flags(n, 1, rng)
    at = rng.integers(0, 2, n).astype(np.int32)
    a = (np.where(at[:, None] == 1, rng.integers(20, 51, (n, 2)), rng.integers(0, 55, (n, 2))) if kind == "flexible"
         else rng.integers(-10, 11, (n, 2))).astype(np.float64)
    ref = None
    for rep in range(2):
        for t, t0 in zip(state, state0):
            t.copy_(t0)
        p.ingest_dmc(f, fl)
        out = {"ingest": lambda: p.stack(), "fixed": lambda: p.observe_fixed(a),
               "peripheral": lambda: p.observe_peripheral(a), "flexible": lambda: p.observe_flexible(a, at)}[kind]()
        torch.cuda.synchronize()
        snap = [out.clone()] + [t.clone() for t in state]
        if ref is None:
            ref = snap
        else:
            assert all(torch.equal(x, y) for x, y in zip(ref, snap))


# ------------------------------------------------------------------------------------------------ env level
class _FakeDMC:
    """A dm_control task that renders a scripted sequence of its own frames."""

    def __init__(self, screens):
        self.screens, self.t, self.physics = screens, 0, self

    def action_spec(self):
        return rh._BoundedArray((2,), np.float64, -np.ones(2), np.ones(2))

    def reset(self):
        self.t += 1
        return rh._TimeStep(None, False)

    def step(self, action):
        self.t += 1
        return rh._TimeStep(1.0, False)

    def render(self, height, width, camera_id=0):
        return self.screens[self.t % len(self.screens)].copy()

    def get_state(self):
        return np.zeros(4)

    def shown(self):
        return self.screens[self.t % len(self.screens)]


def _env(factory, n, rng, sims, **extra):
    import active_gym_b200 as ag
    from active_gym_b200.sources import DMCPool
    kw = dict(fov_size=FOV, fov_init_loc=(3, 4), sensory_action_mode="absolute", frame_stack=K, action_repeat=2,
              grey=False, mask_out=False, resize_to_full=False)
    kw.update(extra)
    args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, **kw)

    def make(i):
        sims.append(_FakeDMC(rng.integers(0, 256, (7,) + S + (3,), dtype=np.uint8)))
        return sims[-1]
    return getattr(ag, factory)(args, num_envs=n, source=DMCPool(args, n if n else 1, env_factory=make))


@pytest.mark.parametrize("factory,extra", [
    ("DMCFixedFovealEnv", {}), ("DMCFixedFovealEnv", {"obs_dtype": torch.float32}),
    ("DMCFixedFovealEnv", {"host_obs": True, "mask_out": True}),
    ("DMCFlexibleFovealEnv", {"mask_out": True}), ("DMCFlexibleFovealEnv", {}),
    ("DMCFixedFovealPeripheralEnv", {"peripheral_res": PERIPH, "sensory_action_mode": "relative",
                                     "sensory_action_space": (-10.0, 10.0)})])
def test_batched_envs_equal_independent_oracle_envs(factory, extra):
    rng = np.random.default_rng(23)
    n, sims = 19, []
    env = _env(factory, n, rng, sims, **extra)
    kind = {"DMCFixedFovealEnv": "fixed", "DMCFlexibleFovealEnv": "flexible", "DMCFixedFovealPeripheralEnv": "peripheral"}[factory]
    variant = "mask" if extra.get("mask_out") else ("mask" if kind == "peripheral" else "crop")
    shape = (K, 3) + (FOV if variant == "crop" and kind == "fixed" else S)   # the flexible crop arrives padded to S
    declared = (K, 3) + (FOV if variant == "crop" else S)                    # as the grey path declares it
    assert env.observation_space.shape == declared and env.unwrapped.observation_space.shape == (K, 3) + S
    ring, head = rgb.new_state(n, K, S)
    loc = np.tile(np.array([[3, 4]], np.int32), (n, 1))
    res = np.tile(np.array([FOV], np.int32), (n, 1))
    relative = extra.get("sensory_action_mode") == "relative"

    def check(obs, info):
        if kind == "flexible":
            want = rgb.observe_flexible(ring, head, loc, res, FOV, variant=variant)
        elif kind == "peripheral":
            want = rgb.observe_peripheral(ring, head, loc, FOV, PERIPH)
        else:
            want = rgb.observe_fixed(ring, head, loc, FOV, variant=variant)
        got = obs.numpy() if not obs.is_cuda else obs.cpu().numpy()
        assert got.shape == (n,) + shape
        if extra.get("obs_dtype") is not None:
            assert got.dtype == np.float32
            assert np.array_equal(got, orc.to_reference_float(want).astype(np.float32))
        elif want.dtype == np.uint8:
            assert np.array_equal(got, want)
        else:
            assert np.abs(got.astype(np.float64) - want).max() <= TOL
        fl = info["fov_loc"]
        assert np.array_equal(fl if isinstance(fl, np.ndarray) else fl.cpu().numpy(), loc)

    obs, info = env.reset()
    rgb.ingest_dmc_rgb(np.stack([s.shown() for s in sims]), np.full(n, 5, np.uint8), ring, head)
    check(obs, info)
    for step in range(5):
        at = rng.integers(0, 2, n).astype(np.int64)
        if kind == "flexible":
            a = np.where(at[:, None] == 1, rng.integers(20, 51, (n, 2)), rng.integers(0, 55, (n, 2))).astype(np.float64)
        elif relative:
            a = rng.integers(-10, 11, (n, 2)).astype(np.float64)
        else:
            a = rng.integers(0, 55, (n, 2)).astype(np.float64)
        act = {"motor_action": np.zeros((n, 2), np.float32), "sensory_action": a}
        if kind == "flexible":
            act["sensory_action_type"] = at
        obs, _, _, _, info = env.step(act)
        rgb.ingest_dmc_rgb(np.stack([s.shown() for s in sims]), np.full(n, 1, np.uint8), ring, head)
        orc.update_loc(a, loc, obs_size=S, fov_size=FOV, relative=relative, lo=-10.0, hi=10.0,
                       atype=at if kind == "flexible" else None, res=res if kind == "flexible" else None)
        check(obs, info)
    env.close()


def test_single_env_adapter_returns_reference_floats():
    rng = np.random.default_rng(29)
    sims = []
    env = _env("DMCFlexibleFovealEnv", None, rng, sims)
    assert env.observation_space.shape == (K, 3) + FOV
    ring, head = rgb.new_state(1, K, S)
    loc, res = np.array([[3, 4]], np.int32), np.array([FOV], np.int32)
    obs, _ = env.reset()
    rgb.ingest_dmc_rgb(sims[0].shown()[None], np.array([5], np.uint8), ring, head)
    for step in range(4):
        at = step % 2
        a = np.array([20 + 7 * step, 45 - 5 * step] if at else [10 * step, 50 - 9 * step], np.float64)
        obs, _, _, _, info = env.step({"motor_action": np.zeros(2, np.float32), "sensory_action": a, "sensory_action_type": at})
        rgb.ingest_dmc_rgb(sims[0].shown()[None], np.array([1], np.uint8), ring, head)
        orc.update_loc(a[None], loc, obs_size=S, fov_size=FOV, atype=np.array([at]), res=res)
        want = rgb.observe_flexible(ring, head, loc, res, FOV, variant="crop")[0][..., :res[0, 0], :res[0, 1]]
        assert obs.dtype == np.float64 and obs.shape == (K, 3, res[0, 0], res[0, 1])
        assert np.abs(obs * 255.0 - want).max() <= TOL + 1e-4
        assert np.array_equal(info["fov_res"], res[0])
    env.close()


def test_fixed_crop_env_returns_k_3_f_f_uint8():
    rng = np.random.default_rng(31)
    env = _env("DMCFixedFovealEnv", 64, rng, [])
    obs, _ = env.reset()
    assert obs.is_cuda and obs.dtype == torch.uint8 and tuple(obs.shape) == (64, 3, 3, 30, 30)
    assert env.observation_space.shape == (3, 3, 30, 30)
    env.close()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two or more GPUs")
def test_sharded_learner_device_output_carries_the_channel_axis():
    from active_gym_b200.vector import ShardedVecEnv
    rng = np.random.default_rng(37)
    n, sims = 40, {}

    def make(m, dev, lo, hi):
        sims[lo] = []
        return _env_dev("DMCFixedFovealEnv", m, rng, sims[lo], dev)
    venv = ShardedVecEnv(make, n, devices=["cuda:0", "cuda:1"], learner_device="cuda:0")
    obs, _ = venv.reset()
    assert tuple(obs.shape) == (n, K, 3) + FOV and obs.device == torch.device("cuda:0")
    a = {"motor_action": np.zeros((n, 2), np.float32), "sensory_action": rng.integers(0, 55, (n, 2)).astype(np.float64)}
    obs, *_ = venv.step(a)
    torch.cuda.synchronize("cuda:0")
    torch.cuda.synchronize("cuda:1")
    for lo, e in zip(sorted(sims), venv.envs):
        path = e.path
        want = rgb.observe_fixed(path.ring.cpu().numpy(), path.head.cpu().numpy(), path.loc.cpu().numpy(), FOV)
        assert np.array_equal(obs[lo:lo + e.num_envs].cpu().numpy(), want)
    venv.close()


def _env_dev(factory, n, rng, sims, dev):
    import active_gym_b200 as ag
    from active_gym_b200.sources import DMCPool
    args = ag.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, fov_size=FOV, fov_init_loc=(3, 4),
                         sensory_action_mode="absolute", frame_stack=K, action_repeat=2, grey=False, mask_out=False,
                         resize_to_full=False)

    def make(i):
        sims.append(_FakeDMC(rng.integers(0, 256, (7,) + S + (3,), dtype=np.uint8)))
        return sims[-1]
    return getattr(ag, factory)(args, num_envs=n, source=DMCPool(args, n, env_factory=make), device=dev)
