"""TEST INFRASTRUCTURE — generates tests/golden/*.npz from the UNMODIFIED reference.

Needs a checkout of the reference package (see oracle/ref_harness.py):

    AGYM_REFERENCE_ROOT=<reference checkout> python oracle/make_golden.py

The reference's fov_env.py / atari_env.py / dmc_env.py are imported as they are, under
the simulator stubs of oracle/ref_harness.py, and driven through their public
``reset()`` / ``step()`` API on scripted screens.  For every call the fixture records
which scripted screens the reference read (and therefore the ingest flags), the
sensory action, the reference's observation, ``fov_loc`` and ``fov_res``.

Stored observation encodings
  * ``obs_u8``  — exact paths (crop / stack / max-pool / mask / cv2 resize / luma): the
    generator asserts ``ref == float64(float32(u)/255)`` and stores ``u``.
  * ``obs_f32`` — resampled paths (torchvision Resize): ``float32(255 * ref)``.
Library versions used are recorded in ``tests/golden/MANIFEST.json``.
"""
from __future__ import annotations

import json
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref_harness as rh  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
FLAG_A, FLAG_B, FLAG_HARD, FLAG_IDLE = 1, 2, 4, 8


def make_atari_screens(n=40, seed=1234):
    """(n,210,160) u8: a mix of iid noise, ramps and moving sprites."""
    rng = np.random.default_rng(seed)
    s = np.empty((n, 210, 160), np.uint8)
    yy, xx = np.mgrid[0:210, 0:160]
    for i in range(n):
        kind = i % 4
        if kind == 0:
            s[i] = rng.integers(0, 256, (210, 160), dtype=np.uint8)
        elif kind == 1:
            s[i] = ((yy * 3 + xx * 5 + i * 17) % 256).astype(np.uint8)
        elif kind == 2:
            f = np.full((210, 160), (i * 29) % 256, np.uint8)
            for _ in range(12):
                r, c = rng.integers(0, 202), rng.integers(0, 152)
                f[r:r + 8, c:c + 8] = rng.integers(0, 256)
            s[i] = f
        else:
            base = ((xx * 255) // 159).astype(np.uint8)
            noise = rng.integers(0, 256, (210, 160), dtype=np.uint8)
            s[i] = np.where(rng.random((210, 160)) < 0.3, noise, base)
    return s


def make_dmc_screens(n=24, seed=4321):
    rng = np.random.default_rng(seed)
    s = rng.integers(0, 256, (n, 84, 84, 3), dtype=np.uint8)
    yy, xx = np.mgrid[0:84, 0:84]
    for i in range(0, n, 3):  # every third: structured colour ramps
        s[i, ..., 0] = (xx * 3 + i) % 256
        s[i, ..., 1] = (yy * 3 + 2 * i) % 256
        s[i, ..., 2] = ((xx + yy) * 2) % 256
    return s


def exact_u8(ref):
    u = np.rint(np.asarray(ref, np.float64) * 255.0).astype(np.uint8)
    back = (u.astype(np.float32) / np.float32(255.0)).astype(np.float64)
    assert np.array_equal(back, np.asarray(ref, np.float64)), "reference value is not u8-equivalent"
    return u


class Recorder:
    def __init__(self, meta):
        self.meta = meta
        self.rows = {k: [] for k in ("ia", "ib", "flags", "action", "atype", "loc", "res", "done")}
        self.obs = []

    def add(self, idx, flags, action, atype, obs, info, done):
        ia = idx[0] if len(idx) > 0 else -1
        ib = idx[1] if len(idx) > 1 else -1
        self.rows["ia"].append(ia); self.rows["ib"].append(ib); self.rows["flags"].append(flags)
        self.rows["action"].append(np.asarray(action, np.float64)); self.rows["atype"].append(atype)
        self.rows["loc"].append(np.asarray(info["fov_loc"], np.int32) if "fov_loc" in info else np.zeros(2, np.int32))
        self.rows["res"].append(np.asarray(info.get("fov_res", (0, 0)), np.int32))
        self.rows["done"].append(bool(done))
        self.obs.append(np.asarray(obs))

    def save(self, name):
        out = {k: np.asarray(v) for k, v in self.rows.items()}
        exact = self.meta["exact"]
        if self.meta.get("ragged"):
            # variable-shape crops: pad into (T,K,S,S), top-left aligned
            K, S = self.meta["frame_stack"], self.meta["obs_size"]
            pad = np.zeros((len(self.obs), K, S[0], S[1]), np.float64)
            for i, o in enumerate(self.obs):
                pad[i, :, :o.shape[1], :o.shape[2]] = o
            obs = pad
        else:
            obs = np.stack(self.obs, 0)
        # blurred / resampled calls are float, untouched crops are exact: store both forms
        if exact:
            out["obs_u8"] = exact_u8(obs)
        else:
            out["obs_f32"] = (obs.astype(np.float64) * 255.0).astype(np.float32)
        out["meta"] = np.array(json.dumps(self.meta))
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
        print(f"  {name}: {len(self.obs)} calls, obs {obs.shape} {'u8' if exact else 'f32'}")


# ------------------------------------------------------------------------------- Atari
ACTIONS_ABS = [(10.5, 53.5), (2.5, 3.5), (-3.0, 99.7), (54.0, 0.49), (17, 23), (53.5, 54.5), (30.2, 11.8), (0.5, 1.5)]
ACTIONS_REL = [(3.5, -2.5), (10.49, 10.51), (-15.0, 4.4), (9.5, 9.5), (-0.5, 0.5), (7, -7), (-10, -10), (2.5, -3.5)]


def run_atari(name, atari, screens, cls, *, mode, variant="crop", K=4, fov=(30, 30), init=(0, 0),
              action_repeat=4, periph=None, flexible_plan=None, game_over_at=(), lives_at=None,
              n_steps=6, training=True, tensor_actions=False):
    import torch
    script = rh.ScreenScript(screens[..., None], game_over_at=game_over_at, lives_at=lives_at)
    rh.ScreenScript.current = script
    kw = dict(fov_size=fov, fov_init_loc=init, sensory_action_mode=mode, frame_stack=K,
              action_repeat=action_repeat, mask_out=(variant == "mask"), resize_to_full=(variant == "resize_full"))
    if mode == "relative":
        kw["sensory_action_space"] = (-10.0, 10.0)
    if periph:
        kw["peripheral_res"] = periph
    args = atari.AtariEnvArgs(game="boxing", seed=0, obs_size=(84, 84), **kw)
    env = cls(args)
    if not training:
        env.eval()
    flexible = flexible_plan is not None
    exact = (variant in ("crop", "mask")) and not periph and not flexible
    meta = dict(kind="atari", env=cls.__name__, mode=mode, variant=variant, frame_stack=K, obs_size=(84, 84),
                fov_size=fov, fov_init_loc=init, action_repeat=action_repeat, peripheral_res=periph,
                lo=-10.0, hi=10.0, exact=exact, flexible=flexible, ragged=(flexible and variant == "crop"),
                script=dict(game_over_at=list(game_over_at), lives_at={str(k): v for k, v in (lives_at or {}).items()}),
                random_seed=7, training=training, tensor_actions=tensor_actions)
    rec = Recorder(meta)
    random.seed(7)

    def do_reset():
        soft = bool(env.life_termination)
        n0 = len(script.log)
        obs, info = env.reset()
        idx = script.log[n0:]
        assert len(idx) == 1
        rec.add(idx, FLAG_A | (0 if soft else FLAG_HARD), (0, 0), -1, obs, info, False)

    do_reset()
    acts = ACTIONS_ABS if mode == "absolute" else ACTIONS_REL
    for i in range(n_steps):
        a = acts[i % len(acts)]
        atype = 0
        if flexible:
            atype, a = flexible_plan[i % len(flexible_plan)]
        n0 = len(script.log)
        act = {"motor_action": 0,
               "sensory_action": (torch.tensor(a) if tensor_actions and i % 2 else np.array(a))}
        if flexible:
            act["sensory_action_type"] = np.array([atype]) if i % 2 else atype
        obs, r, done, trunc, info = env.step(act)
        idx = script.log[n0:]
        flags = (FLAG_A if len(idx) > 0 else 0) | (FLAG_B if len(idx) > 1 else 0)
        rec.add(idx, flags, a, atype, obs, info, done)
        if done:
            do_reset()
    rec.save(name)


def run_dmc(name, dmc, screens, cls, *, mode, variant="crop", K=3, fov=(30, 30), init=(0, 0), action_repeat=2,
            periph=None, n_steps=5):
    script = rh.ScreenScript(screens)
    rh.ScreenScript.current = script
    kw = dict(fov_size=fov, fov_init_loc=init, sensory_action_mode=mode, frame_stack=K, action_repeat=action_repeat,
              mask_out=(variant == "mask"), resize_to_full=(variant == "resize_full"))
    if mode == "relative":
        kw["sensory_action_space"] = (-10.0, 10.0)
    if periph:
        kw["peripheral_res"] = periph
    args = dmc.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=(84, 84), **kw)
    env = cls(args)
    exact = (variant in ("crop", "mask")) and not periph
    meta = dict(kind="dmc", env=cls.__name__, mode=mode, variant=variant, frame_stack=K, obs_size=(84, 84), fov_size=fov,
                fov_init_loc=init, action_repeat=action_repeat, peripheral_res=periph, lo=-10.0, hi=10.0,
                exact=exact, flexible=False, ragged=False)
    rec = Recorder(meta)
    n0 = len(script.log)
    obs, info = env.reset()
    rec.add(script.log[n0:], FLAG_A | FLAG_HARD, (0, 0), -1, obs, info, False)
    acts = ACTIONS_ABS if mode == "absolute" else ACTIONS_REL
    dtypes = [str(obs.dtype)]
    for i in range(n_steps):
        n0 = len(script.log)
        obs, r, done, trunc, info = env.step({"motor_action": np.zeros(2, np.float32), "sensory_action": np.array(acts[i])})
        dtypes.append(str(obs.dtype))
        rec.add(script.log[n0:], FLAG_A, acts[i], 0, obs, info, done)
    meta["obs_dtypes"] = dtypes
    rec.save(name)


def primitives(screens_a, screens_d):
    """Known-answer vectors for the library calls themselves."""
    import cv2
    import torch
    from torchvision.transforms import Resize
    rng = np.random.default_rng(99)
    out = {}
    # cv2.resize INTER_LINEAR (atari_env.py:74): note dsize is (w,h)
    srcs = [screens_a[0], screens_a[1], screens_a[3], np.full((210, 160), 255, np.uint8),
            rng.integers(0, 256, (210, 160), dtype=np.uint8)]
    out["resize_src"] = np.stack(srcs)
    out["resize_84"] = np.stack([cv2.resize(s[..., None], (84, 84), interpolation=cv2.INTER_LINEAR) for s in srcs])
    out["resize_64x96"] = np.stack([cv2.resize(s[..., None], (96, 64), interpolation=cv2.INTER_LINEAR) for s in srcs[:2]])
    # cvtColor BGR2GRAY (dmc_env.py:182)
    rgb = rng.integers(0, 256, (4096, 16, 3), dtype=np.uint8)
    out["luma_src"] = rgb
    out["luma_bgr2gray"] = cv2.cvtColor(rgb, cv2.COLOR_BGR2GRAY)
    out["luma_rgb2gray"] = cv2.cvtColor(rgb, cv2.COLOR_RGB2GRAY)
    # torchvision Resize (fov_env.py:120,248,278,366-368), float64 and float32 inputs
    cases = [((84, 84), (20, 20)), ((20, 20), (84, 84)), ((30, 30), (84, 84)), ((44, 50), (30, 30)),
             ((30, 30), (44, 50)), ((31, 20), (30, 30)), ((30, 30), (31, 20)), ((84, 84), (30, 30)), ((50, 21), (84, 84))]
    for i, (ish, osh) in enumerate(cases):
        x = rng.integers(0, 256, ish).astype(np.float64)
        y64 = Resize(osh)(torch.from_numpy(x)[None])[0].numpy()
        y32 = Resize(osh)(torch.from_numpy(x.astype(np.float32))[None])[0].numpy()
        out[f"aa{i}_in"] = x.astype(np.uint8)
        out[f"aa{i}_out64"] = y64
        out[f"aa{i}_out32"] = y32
    out["aa_cases"] = np.array(json.dumps(cases))
    np.savez_compressed(os.path.join(GOLD, "primitives.npz"), **out)
    print("  primitives: cv2.resize x%d, luma %d px, Resize x%d" % (len(srcs), rgb.shape[0] * rgb.shape[1], len(cases)))


def main():
    import cv2
    import torch
    import torchvision
    os.makedirs(GOLD, exist_ok=True)
    fov, atari, dmc = rh.load_reference()
    sa, sd = make_atari_screens(), make_dmc_screens()
    np.savez_compressed(os.path.join(GOLD, "screens_atari.npz"), screens=sa)
    np.savez_compressed(os.path.join(GOLD, "screens_dmc.npz"), screens=sd)
    print("generating golden fixtures from", rh.REFERENCE_ROOT)
    primitives(sa, sd)
    A = atari
    # BASELINE config 1: Boxing single env, absolute, K=4, fov 30 (crop)
    run_atari("atari_fixed_abs_crop", A, sa, A.AtariFixedFovealEnv, mode="absolute", n_steps=8, tensor_actions=True)
    # BASELINE config 2 semantics: relative, skip-4 max-pool; with an early game-over and a life loss
    run_atari("atari_fixed_rel_crop_events", A, sa, A.AtariFixedFovealEnv, mode="relative", init=(27, 27), n_steps=12,
              game_over_at=(22, 37), lives_at={70: 2})
    run_atari("atari_fixed_rel_mask", A, sa, A.AtariFixedFovealEnv, mode="relative", variant="mask", init=(10, 40), n_steps=5)
    run_atari("atari_fixed_abs_resize_full", A, sa, A.AtariFixedFovealEnv, mode="absolute", variant="resize_full", n_steps=4)
    run_atari("atari_fixed_abs_crop_k3_rep1", A, sa, A.AtariFixedFovealEnv, mode="absolute", K=3, action_repeat=1, fov=(50, 50), n_steps=4)
    run_atari("atari_fixed_abs_crop_rep3", A, sa, A.AtariFixedFovealEnv, mode="absolute", action_repeat=3, fov=(20, 36), n_steps=4)
    # BASELINE config 4: foveal 30 + peripheral 20
    run_atari("atari_peripheral_rel", A, sa, A.AtariFixedFovealPeripheralEnv, mode="relative", init=(5, 9), periph=(20, 20), n_steps=4)
    run_atari("atari_peripheral_abs_p16x24", A, sa, A.AtariFixedFovealPeripheralEnv, mode="absolute", fov=(24, 40), periph=(16, 24), n_steps=3)
    # BASELINE config 3: flexible fovea, res 20..50
    L, R = 0, 1
    plan = [(R, (44, 50)), (L, (50.5, 3.5)), (R, (31, 20)), (L, (10, 70)), (R, (30, 50)), (R, (50, 20)), (L, (0.5, 1.5)), (R, (20, 33))]
    plan_rel = [(R, (44, 50)), (L, (9.5, -3.5)), (R, (31, 20)), (L, (-10.5, 7)), (R, (30, 50)), (R, (50, 20)), (L, (2.5, 1.5)), (R, (20, 33))]
    run_atari("atari_flexible_abs_mask", A, sa, A.AtariFlexibleFovealEnv, mode="absolute", variant="mask", flexible_plan=plan, n_steps=6)
    run_atari("atari_flexible_rel_resize_full", A, sa, A.AtariFlexibleFovealEnv, mode="relative", variant="resize_full", init=(20, 20), flexible_plan=plan_rel, n_steps=4)
    run_atari("atari_flexible_abs_crop", A, sa, A.AtariFlexibleFovealEnv, mode="absolute", variant="crop", flexible_plan=plan, n_steps=8)
    # BASELINE config 5: DMC, K=3, action repeat 2
    D = dmc
    run_dmc("dmc_fixed_abs_crop", D, sd, D.DMCFixedFovealEnv, mode="absolute", n_steps=6)
    run_dmc("dmc_fixed_rel_mask", D, sd, D.DMCFixedFovealEnv, mode="relative", variant="mask", init=(30, 30), n_steps=4)
    run_dmc("dmc_peripheral_abs", D, sd, D.DMCFixedFovealPeripheralEnv, mode="absolute", periph=(20, 20), n_steps=4)
    manifest = {"generator": "oracle/make_golden.py", "reference": "elicassion/active-gym (fov_env.py, atari_env.py, dmc_env.py, unmodified)",
                "numpy": np.__version__, "opencv": cv2.__version__, "torch": torch.__version__, "torchvision": torchvision.__version__}
    with open(os.path.join(GOLD, "MANIFEST.json"), "w") as f:
        json.dump(manifest, f, indent=1)
    print("done")


if __name__ == "__main__":
    main()
