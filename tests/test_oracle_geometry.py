"""CPU: the oracle's primitives are the reference libraries' at the plan shapes of ``tests/test_gpu_geometry_sweep.py``.

That sweep checks the kernels against the oracle at non-square frames, small and large frames and other stack depths;
this file pins the oracle itself there, so a failure of the sweep points at a kernel:
* ``orc.cv2_resize_linear`` is ``cv2.resize(src, (w, h), INTER_LINEAR)`` (atari_env.py:74) from 210x160 and 84x84 frames;
* ``orc.aa_resize`` is torchvision's ``Resize((h, w))`` in both antialias modes, in float64, for every squeeze,
  expand, glimpse and resize_full pair of the sweep;
* ``periodic_run`` finds the cyclic row runs the pipelined host copies rely on.
"""
import numpy as np
import pytest
import torch

from active_gym_b200 import _lib
from active_gym_b200.pipeline import periodic_run
from oracle import agym_oracle as orc
from tests.test_gpu_geometry_sweep import CASES

OBS = sorted({c.obs for c in CASES.values()} | {(70, 84), (42, 84), (42, 88)})


@pytest.mark.parametrize("src", [(210, 160), (84, 84)])
@pytest.mark.parametrize("obs", OBS)
def test_cv2_resize_matches_cv2(src, obs):
    cv2 = pytest.importorskip("cv2")
    rng = np.random.default_rng(obs[0] * 1000 + obs[1])
    x = rng.integers(0, 256, src, dtype=np.uint8)
    assert np.array_equal(orc.cv2_resize_linear(x, obs), cv2.resize(x, (obs[1], obs[0]), interpolation=cv2.INTER_LINEAR))


def _pairs():
    """(name, from, to) of every resample the sweep's observations perform: squeeze obs -> periphery, expand back,
    glimpse window -> fovea (a few window sizes, the frame and one-pixel-wide ones included), fovea -> obs."""
    out = []
    for name, c in CASES.items():
        (S_h, S_w), f = c.obs, c.fov
        out += [(name, c.obs, c.periph), (name, c.periph, c.obs), (name, f, c.obs)]
        for win in [c.obs, (S_h, 1), (1, S_w), (f[0] + 1, f[1] - 1), (S_h // 2 + 3, S_w - 5)]:
            out.append((name, win, f))
    return out


@pytest.mark.parametrize("antialias", [True, False])
@pytest.mark.parametrize("name,ish,osh", _pairs())
def test_aa_resize_matches_torchvision(name, ish, osh, antialias):
    from torchvision.transforms import Resize
    rng = np.random.default_rng(ish[0] * 7 + ish[1] * 13 + osh[0] * 17 + osh[1])
    x = rng.integers(0, 256, ish).astype(np.float64)
    want = Resize(osh, antialias=antialias)(torch.from_numpy(x)[None])[0].numpy()
    orc.set_antialias(antialias)
    try:
        got = orc.aa_resize(x, osh)
    finally:
        orc.set_antialias(True)
    assert np.abs(got - want).max() <= 1e-9


def _used_rows(raw_h, obs_h):
    """Raw rows the plan's cv2 table samples (the rows ObservationPath.used_rows lists)."""
    s0, s1, cf = (np.zeros(obs_h, np.int32) for _ in range(3))
    assert _lib.lib().agym_table_cv2(raw_h, obs_h, 0, s0.ctypes.data, s1.ctypes.data, cf.ctypes.data) == 0
    return np.union1d(s0, s1)


@pytest.mark.parametrize("obs_h,run", [(84, (5, 3, 4)), (70, (3, 1, 2)), (42, (5, 2, 2)), (100, (21, 11, 20)),
                                       (126, None), (112, None), (96, None), (64, None), (48, None), (128, None),
                                       (176, None)])
def test_periodic_run_of_the_sampled_rows(obs_h, run):
    used = _used_rows(210, obs_h)
    assert periodic_run(used, 210) == run
    # the rows the oracle's resize reads: a row outside `used` never changes the output
    rng = np.random.default_rng(obs_h)
    x = rng.integers(0, 256, (210, 160), dtype=np.uint8)
    y = x.copy()
    y[np.setdiff1d(np.arange(210), used)] ^= 0xFF
    assert np.array_equal(orc.cv2_resize_linear(x, (obs_h, 84)), orc.cv2_resize_linear(y, (obs_h, 84)))
    if run is not None:
        P, o, L = run
        assert np.array_equal(used, np.flatnonzero((np.arange(210) - o) % P < L))
