"""GPU: the standard-geometry peripheral kernel (`k_observe_peripheral_std`) runs one pipeline per frame plane — a
3-warp group per plane with its own buffers, barrier and TMA stores, and the fov_loc batches handed between the groups
through mbarriers.  These cases hold it to the oracle where that structure is stressed: env counts that give some CTAs
one env fewer than others (K = 3 and K = 4), and a 16,384-env batch compared over EVERY env, six steps deep, so each
CTA walks ~55 envs through the input ring, the store ring and two fov_loc batches, with and without the fused f16 copy.
"""
import numpy as np
import pytest
import torch

from oracle import agym_oracle as orc

pytestmark = pytest.mark.gpu

TOL = 0.5 + 1e-2
S, FOV, PER = (84, 84), (30, 30), (20, 20)


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _flags(rng, n):
    choices = np.array([3, 3, 3, 3, 1, 0, 5, 1 | 4, 8, 3 | 4], np.uint8)
    return choices[rng.integers(0, len(choices), n)]


def _run(n, K, steps, seed, norm_dtype=None):
    """`steps` synthetic steps; after each, the device output over all envs against the oracle's merge of the device's
    own ring (the ingest is checked elsewhere; the merge is what is under test here)."""
    from active_gym_b200 import ObservationPath
    rng = np.random.default_rng(seed)
    p = ObservationPath(n, K, S, (210, 160, 1), fov_size=FOV, peripheral_res=PER, sensory_action_mode="relative",
                        sensory_action_space=(-10.0, 10.0), fov_init_loc=(7, 40))
    fa = torch.empty(p.raw_frame_shape(), dtype=torch.uint8, device="cuda")
    fb = torch.empty_like(fa)
    loc = np.zeros((n, 2), np.int32)
    nrm = torch.empty((n, K) + S, dtype=norm_dtype, device="cuda") if norm_dtype is not None else None
    for step in range(steps):
        p.synth_frames(fa, 300 + 2 * step); p.synth_frames(fb, 301 + 2 * step)
        p.ingest_atari(fa, fb, _dev(np.full(n, 5, np.uint8) if step == 0 else _flags(rng, n)))
        ctrl = np.full(n, 1, np.uint8) if step == 0 else rng.choice(np.array([0, 0, 0, 0, 1, 2], np.uint8), size=n)
        a = rng.uniform(-14, 14, (n, 2))
        a[0::7] = (-1e6, 1e6)   # windows at the frame's edges
        a[1::7] = (1e6, -1e6)
        got = p.observe_peripheral(_dev(a), ctrl=_dev(ctrl), norm_out=nrm)
        new = loc.copy()
        orc.update_loc(a, new, obs_size=S, fov_size=FOV, relative=True, lo=-10.0, hi=10.0)
        loc[ctrl == 0] = new[ctrl == 0]
        loc[ctrl == 1] = (7, 40)
        torch.cuda.synchronize()
        assert np.array_equal(p.loc.cpu().numpy(), loc), step
        ring, head = p.ring.cpu().numpy(), p.head.cpu().numpy()
        g = got.cpu().numpy()
        for lo in range(0, n, 1024):   # the oracle's float64 output in slices (3.7 GB at 16,384 envs)
            sl = slice(lo, min(lo + 1024, n))
            want = orc.observe_peripheral(ring[sl], head[sl], loc[sl], FOV, PER)
            assert np.abs(g[sl].astype(np.float64) - want).max() <= TOL, (step, lo)
        for e in range(0, n, max(1, n // 97)):   # the fovea itself is a bit-exact paste
            r, c = loc[e]
            st = orc.stack(ring[e:e + 1], head[e:e + 1])[0]
            assert np.array_equal(g[e][:, r:r + FOV[0], c:c + FOV[1]], st[:, r:r + FOV[0], c:c + FOV[1]]), (step, e)
        if nrm is not None:
            ref = torch.from_numpy(g.astype(np.float32) / np.float32(255)).to(norm_dtype)
            assert torch.equal(nrm.cpu(), ref), step


@pytest.mark.parametrize("K", [3, 4])
@pytest.mark.parametrize("n", [1, 5, 297, 593])
def test_ragged_env_counts_match_the_oracle(K, n):
    # 148 SMs x 2 CTAs: 297 and 593 envs leave every CTA but the first one iteration short of it
    _run(n, K, steps=3, seed=n + K)


def test_16384_envs_every_env_matches_the_oracle():
    _run(16384, 4, steps=6, seed=11)


def test_16384_envs_with_the_f16_copy():
    _run(16384, 4, steps=2, seed=12, norm_dtype=torch.float16)
