"""TEST INFRASTRUCTURE — runs the UNMODIFIED reference under simulator stubs.

Only usable where a checkout of the reference package (elicassion/active-gym, the
directory that holds ``active_gym/fov_env.py``) is named by ``AGYM_REFERENCE_ROOT`` or sits
in the git-ignored ``oracle/_ref/``; the repository does not contain it.  It is used by ``oracle/make_golden.py`` to generate the
committed fixtures in ``tests/golden/`` and by ``tests/test_oracle_vs_reference.py``
(skipped when the reference is absent) to pin the restated oracle against the reference itself.

What is stubbed (absent third-party modules, SURVEY.md §8c): ``gymnasium``
(``Env``/``Wrapper``/``spaces``), ``atari_py`` (``ALEInterface`` replaced by a fake
that replays a scripted screen sequence), ``dm_control.suite`` and ``dm_env.specs``
(fake physics that replays scripted renders).  Every pixel operation still runs in the
real numpy / OpenCV / torchvision code that the reference calls.
"""
from __future__ import annotations

import importlib
import os
import sys
import types

import numpy as np

REFERENCE_ROOT = os.environ.get("AGYM_REFERENCE_ROOT") or os.path.join(os.path.dirname(os.path.abspath(__file__)), "_ref")


def reference_available() -> bool:
    return os.path.isfile(os.path.join(REFERENCE_ROOT, "active_gym", "fov_env.py"))


# --------------------------------------------------------------------------- gymnasium
class _Space:
    def __init__(self, shape=None, dtype=None):
        self.shape = shape
        self.dtype = dtype
        self._rng = np.random.default_rng(0)

    def seed(self, seed=None):
        self._rng = np.random.default_rng(seed)
        return [seed]


class _Box(_Space):
    def __init__(self, low, high, shape=None, dtype=np.float32):
        if shape is None:
            shape = np.shape(low) if np.ndim(low) > 0 else (1,)
        super().__init__(tuple(shape), dtype)
        self.low = np.broadcast_to(np.asarray(low, dtype=dtype), self.shape).copy()
        self.high = np.broadcast_to(np.asarray(high, dtype=dtype), self.shape).copy()

    def contains(self, x):
        x = np.asarray(x)
        return x.shape == self.shape and bool(np.all(x >= self.low) and np.all(x <= self.high))

    def sample(self):
        lo = np.where(np.isfinite(self.low), self.low, -1.0)
        hi = np.where(np.isfinite(self.high), self.high, 1.0)
        return (lo + (hi - lo) * self._rng.random(self.shape)).astype(self.dtype)


class _Discrete(_Space):
    def __init__(self, n):
        super().__init__((), np.int64)
        self.n = int(n)

    def contains(self, x):
        return 0 <= int(x) < self.n

    def sample(self):
        return int(self._rng.integers(self.n))


class _Dict(dict):
    def __init__(self, spaces=None, **kw):
        super().__init__(spaces or {}, **kw)

    def sample(self):
        return {k: v.sample() for k, v in self.items()}

    def seed(self, seed=None):
        for v in self.values():
            v.seed(seed)


class _Env:
    metadata = {}

    def reset(self, seed=None, options=None):
        raise NotImplementedError

    def step(self, action):
        raise NotImplementedError

    @property
    def unwrapped(self):
        return self


class _Wrapper(_Env):
    def __init__(self, env):
        self.env = env

    def __getattr__(self, name):
        if name.startswith("_") or name == "env":
            raise AttributeError(name)
        return getattr(self.env, name)

    def reset(self, *a, **k):
        return self.env.reset(*a, **k)

    def step(self, action):
        return self.env.step(action)


# --------------------------------------------------------------------------- simulators
class ScreenScript:
    """The scripted frame source shared by the fake ALE / fake physics.

    ``screens[i]`` is what the simulator shows after ``i`` simulator steps since
    construction; ``game_over_at`` / ``lives_at`` map a step count to the value the
    fake reports from that count on.  ``log`` records which screen index every
    screen read returned, in call order.
    """

    current: "ScreenScript | None" = None

    def __init__(self, screens, game_over_at=None, lives_at=None, n_actions=18):
        self.screens = screens
        self.game_over_at = set(game_over_at or ())
        self.lives_at = dict(lives_at or {})
        self.n_actions = n_actions
        self.acts = 0
        self.lives = 3
        self.log = []

    def advance(self):
        self.acts += 1
        if self.acts in self.lives_at:
            self.lives = self.lives_at[self.acts]

    def screen(self):
        idx = self.acts % len(self.screens)
        self.log.append(idx)
        return self.screens[idx]


class _FakeALE:
    def __init__(self):
        self.script = ScreenScript.current

    def setInt(self, *a):
        pass

    setFloat = setBool = setInt

    def loadROM(self, *a):
        pass

    def getMinimalActionSet(self):
        return list(range(self.script.n_actions))

    def act(self, a):
        self.script.advance()
        return 1.0

    def game_over(self):
        return self.script.acts in self.script.game_over_at

    def lives(self):
        return self.script.lives

    def reset_game(self):
        pass

    def getScreenGrayscale(self):
        return self.script.screen().copy()

    def getScreenRGB(self):
        g = self.script.screens[self.script.acts % len(self.script.screens)]
        return np.repeat(g.reshape(g.shape[0], g.shape[1], 1), 3, axis=2)


class _BoundedArray:
    def __init__(self, shape, dtype, minimum, maximum):
        self.shape, self.dtype = shape, dtype
        self.minimum, self.maximum = minimum, maximum


class _Array:
    def __init__(self, shape, dtype):
        self.shape, self.dtype = shape, dtype


class _TimeStep:
    def __init__(self, reward, last):
        self.reward, self.discount, self._last = reward, 1.0, last
        self.observation = {"position": np.zeros(2), "velocity": np.zeros(2)}

    def last(self):
        return self._last


class _FakePhysics:
    def __init__(self, script):
        self.script = script

    def render(self, height, width, camera_id=0):
        s = self.script.screen()
        assert s.shape[:2] == (height, width)
        return s.copy()

    def get_state(self):
        return np.zeros(4)


class _FakeDMC:
    def __init__(self):
        self.script = ScreenScript.current
        self.physics = _FakePhysics(self.script)

    def action_spec(self):
        return _BoundedArray((2,), np.float64, -np.ones(2), np.ones(2))

    def observation_spec(self):
        return {"position": _Array((2,), np.float64), "velocity": _Array((2,), np.float64)}

    def reset(self):
        self.script.advance()
        return _TimeStep(None, False)

    def step(self, action):
        self.script.advance()
        return _TimeStep(1.0, self.script.acts in self.script.game_over_at)


def install_stubs():
    """Put the stand-in modules into ``sys.modules`` (idempotent)."""
    if "gymnasium" not in sys.modules:
        gym = types.ModuleType("gymnasium")
        spaces = types.ModuleType("gymnasium.spaces")
        vector = types.ModuleType("gymnasium.vector")
        gym.Env, gym.Wrapper, gym.Space = _Env, _Wrapper, _Space
        spaces.Box, spaces.Discrete, spaces.Dict, spaces.Space = _Box, _Discrete, _Dict, _Space
        gym.spaces, gym.vector = spaces, vector
        sys.modules.update({"gymnasium": gym, "gymnasium.spaces": spaces, "gymnasium.vector": vector})
    if "atari_py" not in sys.modules:
        ap = types.ModuleType("atari_py")
        ap.ALEInterface = _FakeALE
        ap.get_game_path = lambda game: game
        sys.modules["atari_py"] = ap
    if "dm_control" not in sys.modules:
        dmc = types.ModuleType("dm_control")
        suite = types.ModuleType("dm_control.suite")
        suite.load = lambda **kw: _FakeDMC()
        dmc.suite = suite
        dm_env = types.ModuleType("dm_env")
        specs = types.ModuleType("dm_env.specs")
        specs.Array, specs.BoundedArray = _Array, _BoundedArray
        dm_env.specs = specs
        sys.modules.update({"dm_control": dmc, "dm_control.suite": suite, "dm_env": dm_env, "dm_env.specs": specs})


def load_reference():
    """Import the reference's three hot-path modules, unmodified, from REFERENCE_ROOT.

    The package ``__init__`` is bypassed (it imports robosuite/rlbench back-ends) by
    registering an empty package object whose ``__path__`` points at the reference.
    Returns ``(fov_env, atari_env, dmc_env)`` modules.
    """
    if not reference_available():
        raise RuntimeError(f"reference not found under {REFERENCE_ROOT}")
    install_stubs()
    pkg_name = "active_gym"
    if pkg_name not in sys.modules:
        pkg = types.ModuleType(pkg_name)
        pkg.__path__ = [os.path.join(REFERENCE_ROOT, "active_gym")]
        sys.modules[pkg_name] = pkg
    fov = importlib.import_module("active_gym.fov_env")
    atari = importlib.import_module("active_gym.atari_env")
    dmc = importlib.import_module("active_gym.dmc_env")
    return fov, atari, dmc
