#!/usr/bin/env python
"""Benchmark of the active-perception observation path (see DESIGN.md §Measurement).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--workload NAME] [--dump-outputs DIR]

One "step" = one full environment step of the hot path over a batch of synthetic frames that
is already resident in HBM: ingest (gray/RGB -> resize -> 2-frame max -> ring push) followed by
the observe kernel of the workload.  Prints ONE JSON line (rank 0).

Workloads (BASELINE.json configs[1..4]; per-GPU env counts, weak scaling):
  atari_peripheral  configs[3]  N=16384  gray 210x160, fovea 30 + periphery 20, relative   (default:
                    the configuration the north-star target "foveal+peripheral 84x84x4 obs/s" is quoted on)
  atari_fixed       configs[1]  N=4096   RGB 210x160x3, fovea 30 crop, relative
  atari_fixed_gray  configs[1]  N=4096   the same with gray 210x160 input (SURVEY 8d's gray-input variant: the reference's
                    boundary is ALE's gray screen, which is what the CPU arm is fed)
  atari_flexible    configs[2]  N=4096   gray, per-env res 20..50, mask_out output
  dmc_fixed         configs[4]  N=8192   RGB 84x84x3, fovea 30 crop, K=3
The line's `value` / `roofline` / `e2e` / `cpu_baseline` are those of --workload; the other configs are timed
briefly in the same run and reported under `workloads`, and configs[3] as literally stated in BASELINE.json (a GLOBAL
batch of 16,384 envs sharded by env index over the GPUs, step captured in a CUDA graph) under `strong_scaling`.

`e2e` goes through the public env API — `Atari*Env(args, num_envs=...).step_async / step_wait` with a host frame
source (pinned memory) and `host_obs=True` — and is checked against the CPU oracle in an untimed pass first.
"""
from __future__ import annotations

import argparse
import hashlib
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# The e2e leg drives several copy streams per GPU (2 env groups x shards, both directions).  With the default of 8
# hardware work queues, streams created later alias onto the same queue and falsely serialise each other's copies
# (measured: the same pipeline 18.8 ms / step on fresh streams, 22-25 ms once more than 8 streams had been created).
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

_STDOUT_FD = None


def quiet_stdout():
    """Rank 0 prints ONE JSON line on stdout.  Libraries write there too (NCCL's version banner under NCCL_DEBUG=VERSION,
    which this image sets): from here on file descriptor 1 is stderr, and `emit` writes the line to the real stdout."""
    global _STDOUT_FD
    if _STDOUT_FD is None:
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)


def emit(line: dict):
    data = (json.dumps(line) + "\n").encode()
    if _STDOUT_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_STDOUT_FD, data)

import numpy as np  # noqa: E402

METRIC, UNIT = "foveal_obs_per_sec", "obs/s"

WORKLOADS = {
    "atari_peripheral": dict(config="configs[3] AtariFixedFovealPeripheralEnv", kind="atari", wrapper="peripheral", n=16384,
                             K=4, raw=(210, 160, 1), fov=(30, 30), periph=(20, 20), mode="relative", variant="crop"),
    "atari_fixed": dict(config="configs[1] AtariFixedFovealEnv", kind="atari", wrapper="fixed", n=4096, K=4,
                        raw=(210, 160, 3), fov=(30, 30), periph=None, mode="relative", variant="crop"),
    # SURVEY 8d's gray-input variant of configs[1] (81,456 B/obs): the reference's real boundary is ALE's GRAY screen, which is
    # also what the CPU arm is fed; the RGB form above pays the luma and 3x the PCIe bytes on the GPU side only
    "atari_fixed_gray": dict(config="configs[1] AtariFixedFovealEnv, gray-input variant", kind="atari", wrapper="fixed", n=4096, K=4,
                             raw=(210, 160, 1), fov=(30, 30), periph=None, mode="relative", variant="crop"),
    "atari_flexible": dict(config="configs[2] AtariFlexibleFovealEnv", kind="atari", wrapper="flexible", n=4096, K=4,
                           raw=(210, 160, 1), fov=(30, 30), periph=None, mode="absolute", variant="mask"),
    "dmc_fixed": dict(config="configs[4] DMCFixedFovealEnv", kind="dmc", wrapper="fixed", n=8192, K=3,
                      raw=(84, 84, 3), fov=(30, 30), periph=None, mode="absolute", variant="crop"),
}
S = (84, 84)
KERNEL_NAMES = {  # the kernels the two legs of a step launch for the benchmark geometries (GPUTEST / ncu launch lists)
    ("atari_peripheral", "ingest"): "k_ingest_gray_std<160,true,2>", ("atari_peripheral", "observe"): "k_observe_peripheral_std<4,0,true>",
    ("atari_fixed", "ingest"): "k_ingest_atari_tma<480,84,3,true,2>", ("atari_fixed", "observe"): "k_observe_fixed_crop_v3<30>",
    ("atari_fixed_gray", "ingest"): "k_ingest_gray_std<160,false,2>", ("atari_fixed_gray", "observe"): "k_observe_fixed_crop_v3<30>",
    ("atari_flexible", "ingest"): "k_ingest_gray_std<160,false,2>", ("atari_flexible", "observe"): "k_observe_flexible_v3<MASK>",
    ("dmc_fixed", "ingest"): "k_ingest_dmc", ("dmc_fixed", "observe"): "k_observe_fixed_crop_v3<30>",
}


def algorithmic_bytes(w):
    """SURVEY.md §8(d): compulsory reads once + writes once, u8 everywhere, per observation."""
    K, plane = w["K"], S[0] * S[1]
    f2 = w["fov"][0] * w["fov"][1]
    rh, rw, rc = w["raw"]
    n_frames = 2 if w["kind"] == "atari" else 1
    ingest = n_frames * rh * rw * rc + plane
    if w["wrapper"] == "peripheral":
        observe = K * plane + K * plane                 # 56,448: the north-star contract figure
    elif w["wrapper"] == "flexible":
        observe = K * 1225 + K * plane                  # E[rh*rw] = 35^2 for res ~ U[20,50]; mask_out output
    else:
        observe = K * f2 + K * f2
    return dict(ingest=ingest, observe=observe, step=ingest + observe)


def working_set_mb(w, n, pool=3):
    """Bytes one GPU cycles through per `pool` steps: the rotating raw-frame batches + ring + output (MB)."""
    rh, rw, rc = w["raw"]
    frames = pool * (2 if w["kind"] == "atari" else 1) * rh * rw * rc
    out = w["K"] * (S[0] * S[1] if w["wrapper"] != "fixed" else w["fov"][0] * w["fov"][1])
    return n * (frames + w["K"] * S[0] * S[1] + out) / 1e6


def config_for(wname, envs_per_gpu, world):
    """The `config` object of the JSON line — the same keys and values for the b200 arm and the reference arm."""
    w = WORKLOADS[wname]
    return {"workload": wname,
            "l2": f"inputs larger than L2: {working_set_mb(w, envs_per_gpu):.0f} MB of raw-frame batches (3 rotated) / ring / output "
                  "per GPU vs 126 MB L2; no flush needed", "reference_config": w["config"], "envs_per_gpu": envs_per_gpu,
            "global_envs": envs_per_gpu * world, "frame_stack": w["K"], "raw_frame": list(w["raw"]), "obs_size": list(S),
            "fov_size": list(w["fov"]), "peripheral_res": list(w["periph"]) if w["periph"] else None,
            "sensory_action_mode": w["mode"], "step": "ingest + observe (full env step)",
            "parallelism": f"env-index shards over {world} GPU(s), no collective"}


def _code_only(text):
    """Source text without // comments, /* */ blocks, indentation and blank lines (what the hash below covers)."""
    import re
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    out = []
    for line in text.splitlines():
        i = line.find("//")
        while i >= 0 and line.count('"', 0, i) % 2:   # a // inside a string literal is not a comment
            i = line.find("//", i + 2)
        line = (line if i < 0 else line[:i]).strip()
        if line:
            out.append(line)
    return "\n".join(out)


# the translation units a workload's two kernels are compiled from (the shared headers, the launcher / plan code and
# the coefficient tables count for every workload)
_KERNEL_TUS = {"atari_peripheral": ("agym_ingest_std.cu", "agym_observe.cu"), "atari_fixed": ("agym_ingest.cu", "agym_observe.cu"),
               "atari_fixed_gray": ("agym_ingest_std.cu", "agym_observe.cu"),
               "atari_flexible": ("agym_ingest_std.cu", "agym_flexible.cu"), "dmc_fixed": ("agym_ingest.cu", "agym_observe.cu")}


def sources_hash(workload=None):
    """Hash of the kernel sources' CODE (comments and blank lines do not count): ties profiles/traffic.json (ncu DRAM
    bytes) to the code it was captured on.  With `workload`, only the files that workload's kernels are built from."""
    h = hashlib.sha256()
    d = os.path.join(ROOT, "active_gym_b200", "csrc")
    for f in sorted(os.listdir(d)):
        if workload is not None and f.endswith(".cu") and f != "agym_abi.cu" and f not in _KERNEL_TUS[workload]:
            continue
        if f.endswith((".cu", ".cuh", ".cpp", ".h")):
            with open(os.path.join(d, f), "r", encoding="utf-8", errors="replace") as fh:
                h.update(f.encode() + b"\0" + _code_only(fh.read()).encode())
    return h.hexdigest()[:16]


# ----------------------------------------------------------------------------- CPU baseline
_W = {}


def reference_root():
    """Where the UNMODIFIED reference package can be imported from ($AGYM_REFERENCE_ROOT, else oracle/_ref; see oracle/ref_harness.py).
    None = not available: the port is timed instead."""
    from oracle import ref_harness as rh
    return rh.REFERENCE_ROOT if rh.reference_available() else None


class RealReferenceEnv:
    """One env of the unmodified reference (fov_env.py / atari_env.py / dmc_env.py imported from `root`) under the
    simulator stubs of oracle/ref_harness.py: the fake ALE / physics cycles pre-generated screens, every pixel
    operation is the reference's own numpy / cv2 / torchvision call."""

    def __init__(self, root, w, screens):
        from oracle import ref_harness as rh
        rh.REFERENCE_ROOT = root
        fov, atari, dmc = rh.load_reference()
        rh.ScreenScript.current = rh.ScreenScript(screens)
        kw = dict(fov_size=w["fov"], fov_init_loc=(0, 0), sensory_action_mode=w["mode"], frame_stack=w["K"],
                  mask_out=w["variant"] == "mask", resize_to_full=False)
        if w["mode"] == "relative":
            kw["sensory_action_space"] = (-10.0, 10.0)
        if w["periph"]:
            kw["peripheral_res"] = w["periph"]
        self.w = w
        if w["kind"] == "atari":
            args = atari.AtariEnvArgs(game="boxing", seed=0, obs_size=S, action_repeat=4, **kw)
            cls = {"peripheral": atari.AtariFixedFovealPeripheralEnv, "flexible": atari.AtariFlexibleFovealEnv,
                   "fixed": atari.AtariFixedFovealEnv}[w["wrapper"]]
            self.motor = 0
        else:
            args = dmc.DMCEnvArgs(domain_name="reacher", task_name="easy", seed=0, obs_size=S, action_repeat=2, **kw)
            cls = dmc.DMCFixedFovealEnv
            self.motor = np.zeros(2, np.float32)
        self.env = cls(args)
        self.flexible = w["wrapper"] == "flexible"

    def reset(self, frame=None):
        return self.env.reset()[0]

    def step(self, fa, fb, action, atype=0):
        act = {"motor_action": self.motor, "sensory_action": np.asarray(action)}
        if self.flexible:
            act["sensory_action_type"] = atype
        return self.env.step(act)[0]


def _cpu_worker_init(wname, seed_base):
    """Per process: import the libraries once and build one reference env (the real one when importable)."""
    import cv2
    import torch
    cv2.setNumThreads(1)
    torch.set_num_threads(1)
    w = WORKLOADS[wname]
    rng = np.random.default_rng(seed_base + os.getpid())
    rh, rw, rc = w["raw"]
    # the reference's Atari boundary is ALE's gray screen; RGB workloads pay the luma on the GPU side only
    shape = (32, rh, rw, 1) if w["kind"] == "atari" else (32, rh, rw, 3)
    frames = rng.integers(0, 256, shape, dtype=np.uint8)
    root = reference_root()
    if root is not None:
        env = RealReferenceEnv(root, w, frames)
    else:
        from oracle.ref_port import RefPortEnv
        env = RefPortEnv(kind=w["kind"], wrapper=w["wrapper"], frame_stack=w["K"], obs_size=S, fov_size=w["fov"],
                         fov_init_loc=(0, 0), mode=w["mode"], lo=-10.0, hi=10.0, variant=w["variant"],
                         peripheral_res=w["periph"])
    acts = rng.integers(-10, 11, (64, 2)) if w["mode"] == "relative" else rng.integers(0, 55, (64, 2))
    res = rng.integers(20, 51, (64, 2))
    env.reset(frames[0])
    for i in range(3):
        env.step(frames[i], frames[i + 1], acts[i])
    _W.update(env=env, frames=frames, acts=acts, res=res, w=w)


def _cpu_worker(n_steps):
    """`n_steps` env steps of this process's env; returns its busy time."""
    env, frames, acts, res, w = _W["env"], _W["frames"], _W["acts"], _W["res"], _W["w"]
    t0 = time.perf_counter()
    for i in range(n_steps):
        if w["wrapper"] == "flexible" and i % 2:
            env.step(frames[i % 32], frames[(i + 1) % 32], res[i % 64], atype=1)
        else:
            env.step(frames[i % 32], frames[(i + 1) % 32], acts[i % 64])
    return time.perf_counter() - t0


def _cpu_proc_main(conn, wname, seed_base):
    _cpu_worker_init(wname, seed_base)
    conn.send("ready")
    while True:
        n = conn.recv()
        if n is None:
            return
        conn.send(_cpu_worker(n))


class CpuReference:
    """`procs` single-env processes (one per host core), the way the reference scales on a CPU."""

    def __init__(self, wname, procs):
        import multiprocessing as mp
        ctx = mp.get_context("fork")
        self.procs, self.conns, self.ps = procs, [], []
        self.kind = "reference" if reference_root() is not None else "port"
        for i in range(procs):
            parent, child = ctx.Pipe()
            pr = ctx.Process(target=_cpu_proc_main, args=(child, wname, 100 + i), daemon=True)
            pr.start()
            self.conns.append(parent); self.ps.append(pr)
        for c in self.conns:
            assert c.recv() == "ready"

    def run(self, n_steps):
        """One bounded sample: every process does n_steps env steps at the same time; returns
        (obs/s over the wall time of the slowest process, seconds)."""
        t0 = time.perf_counter()
        for c in self.conns:
            c.send(n_steps)
        [c.recv() for c in self.conns]
        wall = time.perf_counter() - t0
        return self.procs * n_steps / wall, wall

    def calibrate(self, target_s, probe=64):
        """Env-steps per process that take about `target_s` seconds of wall time."""
        self.run(probe)
        rate, wall = self.run(probe)
        return max(probe, int(probe * target_s / max(wall, 1e-6)))

    def describe(self):
        if self.kind == "reference":
            return "the unmodified reference ($AGYM_REFERENCE_ROOT: fov_env.py + atari_env.py / dmc_env.py) under oracle/ref_harness.py's fake simulators"
        return "oracle/ref_port.py (the reference's per-env cv2 / numpy / torchvision call sequence)"

    def close(self):
        for c in self.conns:
            c.send(None)
        for pr in self.ps:
            pr.join(timeout=5)


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def cpu_baseline_for(wname, seconds, steps_per_proc=0):
    procs = host_cores()
    ref = CpuReference(wname, procs)
    n_cpu = steps_per_proc or ref.calibrate(seconds)
    rate, wall = ref.run(n_cpu)
    kind, what = ref.kind, ref.describe()
    ref.close()
    return {"value": rate, "unit": UNIT, "cores": procs, "kind": kind,
            "sample": f"{procs} single-env processes x {n_cpu} env-steps of {what}, {wall:.1f}s wall = {wall * procs:.0f} core-seconds"}


def run_reference_arm(a):
    """--impl reference: the reference's CPU path (one env per core) on this host."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    w = WORKLOADS[a.workload]
    procs = host_cores()
    ref = CpuReference(a.workload, procs)
    # each bench step = a bounded sample of about --cpu-seconds / steps seconds on every host core
    per_step = a.cpu_steps_per_proc or ref.calibrate(max(a.cpu_seconds / max(a.steps, 1), 0.5))
    for _ in range(max(a.warmup, 1)):
        ref.run(max(per_step // 4, 8))
    t_steps = [ref.run(per_step)[1] for _ in range(a.steps)]
    kind, what = ref.kind, ref.describe()
    ref.close()
    total = procs * per_step * a.steps / sum(t_steps)
    line = {
        "impl": "reference", "metric": METRIC, "value": total, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * sum(t_steps) / a.steps, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": config_for(a.workload, a.envs or w["n"], max(a.gpus, 1)),
        "cpu_baseline": {"value": total, "unit": UNIT, "cores": procs, "kind": kind,
                         "sample": f"{procs} procs x {per_step} env-steps per bench step of {what}"},
        "e2e": {"value": total, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ------------------------------------------------------------------------------ clocks
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-i", str(self.index), "-lms", "100"], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip().split(", "))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for nme, v in zip(names, r[3:7]):
                    if v.strip().lower() == "active":
                        reasons.add(nme)
            except (ValueError, IndexError):
                pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------------- GPU arm
class Workload:
    """Device-resident benchmark state of one workload on one GPU: `pool` independent frame
    batches (cycled so that no step re-reads what the previous one left in L2) and one env batch."""

    def __init__(self, name, device, n=None, pool=3):
        import torch
        from active_gym_b200 import LUMA_DMC, LUMA_RGB, ObservationPath
        self.torch, self.name = torch, name
        w = self.w = WORKLOADS[name]
        self.n = n or w["n"]
        self.device = device
        self.path = ObservationPath(self.n, w["K"], S, w["raw"], luma=LUMA_RGB if w["kind"] == "atari" else LUMA_DMC,
                                    fov_size=w["fov"], fov_init_loc=(0, 0), sensory_action_mode=w["mode"],
                                    sensory_action_space=(-10.0, 10.0), peripheral_res=w["periph"], device=device)
        shape = self.path.raw_frame_shape()
        self.frames = [torch.empty(shape, dtype=torch.uint8, device=device) for _ in range(pool * (2 if w["kind"] == "atari" else 1))]
        for i, f in enumerate(self.frames):
            self.path.synth_frames(f, 1234 + 17 * i)
        g = torch.Generator(device=device).manual_seed(4321)
        if w["mode"] == "relative":
            self.actions = [torch.randint(-10, 11, (self.n, 2), device=device, generator=g).double() for _ in range(4)]
        else:
            self.actions = [torch.randint(0, 55, (self.n, 2), device=device, generator=g).double() for _ in range(4)]
        self.atypes = [torch.randint(0, 2, (self.n,), device=device, generator=g, dtype=torch.int32) for _ in range(4)]
        if w["wrapper"] == "flexible":  # FOV_RES actions carry a window size in 20..50
            for a, t in zip(self.actions, self.atypes):
                r = torch.randint(20, 51, (self.n, 2), device=device, generator=g).double()
                a.copy_(torch.where(t[:, None] == 1, r, a))
        self.flags_reset = torch.full((self.n,), 5, dtype=torch.uint8, device=device)
        self.flags_step = torch.full((self.n,), 3 if w["kind"] == "atari" else 1, dtype=torch.uint8, device=device)
        self.out = torch.empty(self.path.out_shape(w["wrapper"], w["variant"]), dtype=torch.uint8, device=device)
        self.t = 0
        self.ingest(reset=True)
        self.observe(reset=True)

    def ingest(self, reset=False):
        fl = self.flags_reset if reset else self.flags_step
        if self.w["kind"] == "atari":
            k = (2 * self.t) % len(self.frames)
            self.path.ingest_atari(self.frames[k], self.frames[k + 1], fl)
        else:
            self.path.ingest_dmc(self.frames[self.t % len(self.frames)], fl)

    def observe(self, reset=False):
        a = None if reset else self.actions[self.t % 4]
        ctrl = "reset" if reset else None
        wr = self.w["wrapper"]
        if wr == "peripheral":
            self.path.observe_peripheral(a, ctrl=ctrl, out=self.out)
        elif wr == "flexible":
            self.path.observe_flexible(a, None if reset else self.atypes[self.t % 4], variant=self.w["variant"], ctrl=ctrl, out=self.out)
        else:
            self.path.observe_fixed(a, variant=self.w["variant"], ctrl=ctrl, out=self.out)

    def step(self):
        self.ingest()
        self.observe()
        self.t += 1

    def outputs(self, sample=256, seed=0):
        """What a caller of the step received from the last one, for a fixed seeded sample of envs (the full observation
        batch is up to 462 MB): observation, fovea location and, for the flexible fovea, its window size; as float arrays."""
        idx = np.sort(np.random.default_rng(seed).choice(self.n, min(sample, self.n), replace=False))
        sel = self.torch.from_numpy(idx).to(self.device)
        d = {"env_index": idx.astype(np.float64), "obs": self.out.index_select(0, sel).float().cpu().numpy(),
             "fov_loc": self.path.loc.index_select(0, sel).double().cpu().numpy()}
        if self.w["wrapper"] == "flexible":
            d["fov_res"] = self.path.res.index_select(0, sel).double().cpu().numpy()
        return d

    def free(self):
        self.frames = self.actions = self.atypes = self.out = self.path = None
        self.torch.cuda.empty_cache()

    # the flexible launcher also enqueues a 16-byte memset of its work counter (not a kernel)
    launches_per_step = 2


def time_steps(torch, fn, steps, warmup, dist=None):
    """CUDA-event timing of `steps` calls on the current stream, bracketed by barrier + synchronize."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    return e0.elapsed_time(e1) / 1e3  # seconds


def time_steps_graph(torch, wl, steps, warmup, dist=None):
    """The same `steps` steps captured ONCE in a CUDA graph (2 * steps kernel nodes over the rotated frame batches and
    action sets) and replayed: what a learner loop with static buffers does, and the launch path whose timing does not
    depend on how fast this host's Python can issue launches (the DMC / crop steps are shorter than two eager launches
    through ctypes on a loaded host).  One replay = exactly `steps` steps; returns seconds."""
    device = wl.device
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(side):
        for _ in range(max(warmup, 2)):   # warm-up on the capture stream (function attributes, plan state)
            wl.step()
    torch.cuda.current_stream(device).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for _ in range(steps):
            wl.step()
    graph.replay()   # untimed: `steps` more warm-up steps through the graph
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    return e0.elapsed_time(e1) / 1e3


def time_kernel(torch, fn, reps, warmup=3):
    """Average device time of one launch, events around each launch on the launching stream."""
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
    for a, b in evs:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    ts = [a.elapsed_time(b) / 1e3 for a, b in evs]
    # the same launches back to back inside ONE event pair: an event between two launches makes the second wait for the
    # first to drain completely (5-10 us for a 35 us kernel), which the launches of a real step do not pay
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return sum(ts) / len(ts), min(ts), e0.elapsed_time(e1) / 1e3 / reps


def max_over_ranks(torch, dist, device, v):
    if dist is None:
        return v
    t = torch.tensor([v], device=device, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


# ---- end to end through the env API
def make_env(wname, n, device, shards, source=None, host_obs=True):
    """The public drop-in env of a workload over `n` envs, fed by a pinned host frame source."""
    import active_gym_b200 as ag
    from active_gym_b200.sources import PinnedFrameSource
    w = WORKLOADS[wname]
    kw = dict(fov_size=w["fov"], fov_init_loc=(0, 0), sensory_action_mode=w["mode"], sensory_action_space=(-10.0, 10.0),
              frame_stack=w["K"], mask_out=w["variant"] == "mask", host_obs=host_obs, shards=shards)
    if w["periph"]:
        kw["peripheral_res"] = w["periph"]
    if w["kind"] == "atari":
        args = ag.AtariEnvArgs(game="synthetic", seed=0, obs_size=S, **kw)
        src = source or PinnedFrameSource(n, kind="atari", channels=w["raw"][2], pool=2, seed=7)
        cls = {"peripheral": ag.AtariFixedFovealPeripheralEnv, "flexible": ag.AtariFlexibleFovealEnv,
               "fixed": ag.AtariFixedFovealEnv}[w["wrapper"]]
    else:
        args = ag.DMCEnvArgs(domain_name="synthetic", task_name="synthetic", seed=0, obs_size=S, **kw)
        src = source or PinnedFrameSource(n, kind="dmc", obs_size=S, pool=2, seed=7)
        cls = ag.DMCFixedFovealEnv
    return cls(args, num_envs=n, source=src, device=device), src


def e2e_actions(w, m, rng):
    if w["mode"] == "relative":
        a = rng.integers(-10, 11, (m, 2)).astype(np.float64)
    else:
        a = rng.integers(0, 55, (m, 2)).astype(np.float64)
    act = {"motor_action": np.zeros(m, np.int64) if w["kind"] == "atari" else np.zeros((m, 2), np.float32), "sensory_action": a}
    if w["wrapper"] == "flexible":
        t = rng.integers(0, 2, m).astype(np.int32)
        act["sensory_action"] = np.where(t[:, None] == 1, rng.integers(20, 51, (m, 2)), a).astype(np.float64)
        act["sensory_action_type"] = t
    return act


def verify_env_against_oracle(wname, device, shards, n=256, steps=3, sample=(0, 1, 97, 255)):
    """Untimed: the same env class + host source + host_obs path the e2e leg times, at a small batch, against the CPU
    oracle for a few sampled envs (every step).  Raises on a mismatch."""
    from oracle import agym_oracle as orc
    w = WORKLOADS[wname]
    env, src = make_env(wname, n, device, shards)
    rows = env.unwrapped.path.used_rows if w["kind"] == "atari" else None
    K, fov = w["K"], w["fov"]
    idx = np.array([i for i in sample if i < n])
    ring, head = orc.new_state(len(idx), K, S)
    loc = np.zeros((len(idx), 2), np.int32)
    res = np.tile(np.array([fov], np.int32), (len(idx), 1))
    rng = np.random.default_rng(3)
    luma = orc.LUMA_RGB if w["kind"] == "atari" else orc.LUMA_DMC

    def full(t):   # sampled envs' frames of a source batch, unpacked to full screens for the oracle
        f = t.numpy()[idx]
        if rows is None or not getattr(src, "packed_rows", False):
            return f
        out = np.zeros((len(idx), 210) + f.shape[2:], np.uint8)
        out[:, rows] = f
        return out

    def check(obs, info, what):
        if w["wrapper"] == "peripheral":
            want = orc.observe_peripheral(ring, head, loc, fov, w["periph"])
        elif w["wrapper"] == "flexible":
            want = orc.observe_flexible(ring, head, loc, res, fov, variant=w["variant"])
        else:
            want = orc.observe_fixed(ring, head, loc, fov, variant=w["variant"]).astype(np.float64)
        got = np.asarray(obs)[idx].astype(np.float64)
        err = np.abs(got - want).max()
        tol = 0.0 if w["wrapper"] == "fixed" else 0.5 + 1e-2
        if err > tol or not np.array_equal(np.asarray(info["fov_loc"])[idx], loc):
            raise AssertionError(f"e2e env path differs from the oracle at {what}: max err {err} LSB")

    t0 = src.t
    obs, info = env.reset()
    b = src.batches[t0 % len(src.batches)]
    if w["kind"] == "atari":
        orc.ingest_atari(full(b), full(b), np.full(len(idx), 5, np.uint8), ring, head, luma)
    else:
        orc.ingest_dmc(full(b), np.full(len(idx), 5, np.uint8), ring, head, luma)
    check(obs, info, "reset")
    for k in range(steps):
        act = e2e_actions(w, n, rng)
        t0 = src.t
        obs, r, d, tr, info = env.step(act)
        if w["kind"] == "atari":
            fa, fb = src.batches[t0 % len(src.batches)], src.batches[(t0 + 1) % len(src.batches)]
            orc.ingest_atari(full(fa), full(fb), np.full(len(idx), 3, np.uint8), ring, head, luma)
        else:
            orc.ingest_dmc(full(src.batches[t0 % len(src.batches)]), np.full(len(idx), 1, np.uint8), ring, head, luma)
        at = act.get("sensory_action_type")
        orc.update_loc(act["sensory_action"][idx], loc, obs_size=S, fov_size=fov, relative=w["mode"] == "relative", lo=-10.0,
                       hi=10.0, atype=None if at is None else at[idx], res=res if w["wrapper"] == "flexible" else None)
        check(obs, info, f"step {k}")
    env.close()
    return len(idx) * (steps + 1)


def measure_e2e(torch, wname, n, device, steps, warmup, shards):
    """The env step through the public API with HOST buffers: two env groups of n/2 envs (`Atari*Env(args, num_envs)`
    over a pinned host frame source, `host_obs=True`) are stepped alternately the way double-buffered samplers drive
    host simulators — wait A(t), [agent], submit A(t+1), wait B(t), submit B(t+1) ... — so a group's actions still
    depend on its own previous observations while the PCIe link stays busy across step boundaries.  Every step copies
    the group's raw rows + actions host -> device and observations + fov_loc + counters device -> host inside the
    timed region.  Returns (seconds, h2d bytes per full step, d2h bytes per full step)."""
    w = WORKLOADS[wname]
    halves = [n // 2, n - n // 2]
    groups = [make_env(wname, m, device, shards) for m in halves]
    envs = [g[0] for g in groups]
    rng = np.random.default_rng(7)
    acts = [e2e_actions(w, m, rng) for m in halves]
    for env in envs:
        env.reset()
    checks = [0]

    def submit(g):
        envs[g].step_async(acts[g])

    def wait(g):
        obs, reward, done, trunc, info = envs[g].step_wait()   # observations are in host memory now
        checks[0] += int(obs[0, 0, 0, 0]) + int(info["fov_loc"][0, 0]) + int(info["ep_len"][0])

    for g in (0, 1):
        submit(g)
    for _ in range(warmup):
        for g in (0, 1):
            wait(g); submit(g)
    for g in (0, 1):
        wait(g)
    torch.cuda.synchronize()
    paths = [e.unwrapped.path for e in envs]
    for p in paths:
        p.reset_counters()
    # timed: `steps` full steps of both groups, first submits to last wait
    t0 = time.perf_counter()
    for g in (0, 1):
        submit(g)
    for _ in range(steps - 1):
        for g in (0, 1):
            wait(g); submit(g)
    for g in (0, 1):
        wait(g)
    dt = time.perf_counter() - t0
    h2d = sum(p.h2d_bytes for p in paths) // steps
    d2h = sum(p.d2h_bytes for p in paths) // steps
    for env in envs:
        env.close()
    return dt, h2d, d2h


# ---- configs[3] as literally stated: a global batch sharded over the GPUs, step in a CUDA graph
def strong_scaling(torch, dist, device, world, global_envs=16384, instances=8, reps=10):
    """BASELINE configs[3] as written: N = 16,384 envs IN TOTAL, sharded by env index over the GPUs of the box
    (2,048 per GPU at 8).  A per-GPU batch that small would largely sit in the 126 MB L2 from one step to the next, so
    `instances` independent env batches (own frames, ring, cache, output) are stepped in rotation, and the rotation of
    `instances` steps is captured once in a CUDA graph and replayed (launch overhead out of the picture, SURVEY §8e)."""
    from active_gym_b200.sharding import env_shard
    rank = dist.get_rank() if dist is not None else 0
    lo, hi = env_shard(global_envs, rank, world)
    n = hi - lo
    wls = [Workload("atari_peripheral", device, n=n, pool=1) for _ in range(instances)]
    side = torch.cuda.Stream(device=device)
    side.wait_stream(torch.cuda.current_stream(device))
    with torch.cuda.stream(side):
        for wl in wls:   # warm-up on the capture stream (function attributes, plan state)
            wl.step(); wl.step()
    torch.cuda.current_stream(device).wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for wl in wls:
            wl.ingest(); wl.observe()
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        graph.replay()
    e1.record()
    torch.cuda.synchronize()
    dt = max_over_ranks(torch, dist, device, e0.elapsed_time(e1) / 1e3)
    steps = reps * instances
    ws = working_set_mb(wls[0].w, n, pool=1) * instances
    for wl in wls:
        wl.free()
    return {"config": "configs[3] as stated: global batch sharded by env index over the GPUs", "global_envs": global_envs,
            "envs_per_gpu": n, "n_gpus": world, "instances_rotated": instances, "cuda_graph": True, "steps": steps,
            "ms_per_step": dt / steps * 1e3, "value": global_envs * steps / dt, "unit": UNIT, "scaling": "strong",
            "l2": f"{ws:.0f} MB of frames / ring / output per GPU over {instances} rotated env batches vs 126 MB L2"}


def measure_device(torch, dist, device, world, wname, n, steps, warmup, peak, peak_src, traffic_db, no_graph=False, dump=False):
    """Device-timed step (inputs resident in HBM), per-kernel times and the roofline of one workload.  With `dump`, the
    result carries `Workload.outputs()` of the last timed step under "outputs"."""
    wl = Workload(wname, device, n=n)
    w = wl.w
    bytes_ = algorithmic_bytes(w)
    dt_eager = max_over_ranks(torch, dist, device, time_steps(torch, wl.step, steps, warmup, dist))
    dt, launch = dt_eager, "eager: one ctypes call per kernel launch"
    if not no_graph:
        try:
            dt = max_over_ranks(torch, dist, device, time_steps_graph(torch, wl, steps, warmup, dist))
            launch = f"cuda graph: the {steps} timed steps ({steps * wl.launches_per_step} kernel nodes) captured once, one replay timed"
        except Exception as ex:   # keep the eager number rather than lose the line
            launch = "eager (graph capture failed: " + repr(ex)[:120] + ")"
    total_envs = wl.n * world
    out = {"config": config_for(wname, wl.n, world), "value": total_envs * steps / dt, "unit": UNIT, "steps": steps,
           "ms_per_step": dt / steps * 1e3, "ms_per_step_eager": dt_eager / steps * 1e3, "launch": launch,
           "gpu_launches": steps * wl.launches_per_step}
    if dump:   # now: the per-kernel timing below steps the state further
        out["outputs"] = wl.outputs()
    kern = {}
    reps = max(steps, 10)
    for kname, fn, nb in (("ingest", wl.ingest, bytes_["ingest"]), ("observe", wl.observe, bytes_["observe"])):
        def call(fn=fn):
            fn(); wl.t += 1
        avg, best, b2b = time_kernel(torch, call, reps)
        kern[kname] = {"kernel": KERNEL_NAMES.get((wname, kname)), "ms": avg * 1e3, "ms_best": best * 1e3, "ms_back_to_back": b2b * 1e3,
                       "alg_bytes_per_obs": nb,
                       "achieved_gbs": nb * wl.n / avg / 1e9, "obs_per_s": wl.n / avg}
    dom = max(kern, key=lambda k: kern[k]["ms"])
    captured_on = traffic_db.get("sources_sha16", {})
    captured_on = captured_on.get(wname) if isinstance(captured_on, dict) else None
    tr = traffic_db.get("workloads", {}).get(wname, {}).get(dom) if captured_on == sources_hash(wname) else None
    out["kernels"] = kern
    out["alg_bytes_per_obs"] = bytes_
    out["roofline"] = {
        "bound": "hbm", "kernel": f"{dom}: {kern[dom]['kernel']}", "achieved": kern[dom]["achieved_gbs"], "peak": peak,
        "unit": "GB/s", "frac": kern[dom]["achieved_gbs"] / peak, "traffic": tr,
        "traffic_source": ("profiles/traffic.json: ncu dram__bytes_read.sum + dram__bytes_write.sum per launch, captured on sources "
                           + str(captured_on)) if tr is not None else
                          "null: profiles/traffic.json was captured on other kernel sources than the ones running (or has no entry)",
        "peak_source": peak_src, "peak_nominal": 8000.0, "frac_nominal": kern[dom]["achieved_gbs"] / 8000.0,
        "alg_bytes_per_launch": kern[dom]["alg_bytes_per_obs"] * wl.n,
        "note": "achieved = SURVEY 8d algorithmic bytes / kernel time; the kernels move fewer real bytes than that (the Atari "
                "resize never samples a fifth of the raw rows, which are left in HBM; the peripheral kernel reads the cached "
                "squeeze instead of the ring), so frac can exceed traffic / time and even 1: compare with traffic"}
    out["observe_only_obs_per_s"] = kern["observe"]["obs_per_s"]
    return out, wl


def measure_e2e_leg(torch, dist, device, world, rank, a, wname, n, e_steps):
    """The `e2e` object of one workload: oracle check (untimed, rank 0), then the timed host-buffer loop on every rank."""
    w = WORKLOADS[wname]
    n = n or w["n"]
    err, checked = None, 0
    try:
        checked = verify_env_against_oracle(wname, device, a.shards) if rank == 0 else 0
        if dist is not None:
            dist.barrier()
        edt, h2d, d2h = measure_e2e(torch, wname, n, device, e_steps, 2, a.shards)
    except Exception as ex:  # never lose the line over the e2e leg
        edt, h2d, d2h, err = float("inf"), 0, 0, repr(ex)[:300]
    edt = max_over_ranks(torch, dist, device, edt if edt != float("inf") else 1e30)
    if err is not None or edt >= 1e29:
        return {"value": None, "unit": UNIT, "error": err or "a rank failed"}
    return {"value": n * world * e_steps / edt, "unit": UNIT, "h2d_bytes_per_step": h2d * world,
            "d2h_bytes_per_step": d2h * world, "n_gpus": world, "steps": e_steps, "ms_per_step": edt / e_steps * 1e3,
            "api": "Atari*/DMC*FovealEnv(args, num_envs=N/2, source=PinnedFrameSource).step_async / step_wait, host_obs=True, "
                   f"shards={a.shards}; two env groups double buffered",
            "oracle_checked": f"{checked} observations of the same env path (256 envs, sampled envs, every step) against oracle/ before timing",
            "note": "pinned host frames (sampled rows only) + actions -> H2D -> ingest + observe + counters -> D2H "
                    "observations / fov_loc / ep_len / reward; host wall clock, max over ranks"}


def run_b200_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    others = [] if a.only else [k for k in WORKLOADS if k != a.workload]
    cpu = {}
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        # before CUDA is initialised in this process (workers are forked)
        cpu[a.workload] = cpu_baseline_for(a.workload, a.cpu_seconds, a.cpu_steps_per_proc)
        for k in others:
            cpu[k] = cpu_baseline_for(k, min(a.cpu_seconds, 0.8))
    import torch
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py --impl b200 needs a CUDA device (B200); there is no CPU fallback")
    dist = None
    if world > 1:
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        dist_mod.init_process_group("nccl", device_id=torch.device(f"cuda:{local}"))
        dist = dist_mod
    device = torch.device(f"cuda:{local}")
    torch.cuda.set_device(device)
    from active_gym_b200 import _lib
    _lib.lib()
    peaks, traffic_db = {}, {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            traffic_db = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6650 GB/s"

    clocks = ClockSampler(local)
    clocks.start()
    main, wl = measure_device(torch, dist, device, world, a.workload, a.envs, a.steps, a.warmup, peak, peak_src, traffic_db, a.no_graph,
                              dump=a.dump_outputs is not None)
    if a.dump_outputs is not None and rank == 0:
        os.makedirs(a.dump_outputs, exist_ok=True)
        for name, arr in main.pop("outputs").items():
            np.save(os.path.join(a.dump_outputs, name + ".npy"), arr)
    # the timed region is only tens of milliseconds: keep the same step loop running (untimed) until the
    # sampler has had about half a second under identical load, so that the clock record means something
    t_load = time.perf_counter()
    extra = 0
    while time.perf_counter() - t_load < 0.5:
        for _ in range(20):
            wl.step()
        torch.cuda.synchronize()
        extra += 20
    clk = clocks.stop()
    clk["window"] = f"timed region + {extra} further untimed steps of the same loop (0.5 s)"
    wl.free()
    if not a.no_e2e:
        main["e2e"] = measure_e2e_leg(torch, dist, device, world, rank, a, a.workload, a.envs, max(a.steps // 2, 3))
    extra_w = {}
    for k in others:
        r, wl = measure_device(torch, dist, device, world, k, None, a.other_steps, 3, peak, peak_src, traffic_db, a.no_graph)
        wl.free()
        if not a.no_e2e:
            r["e2e"] = measure_e2e_leg(torch, dist, device, world, rank, a, k, None, max(a.other_steps // 2, 3))
        r["cpu_baseline"] = cpu.get(k)
        extra_w[k] = r
    strong = None
    if a.workload == "atari_peripheral" and not a.only:
        try:
            strong = strong_scaling(torch, dist, device, world)
        except Exception as ex:
            strong = {"error": repr(ex)[:300]}
    if rank == 0:
        line = {
            "metric": METRIC, "value": main["value"], "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
            "ms_per_step": main["ms_per_step"], "ms_per_step_eager": main["ms_per_step_eager"], "launch": main["launch"],
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": main["config"],
            "clocks": clk, "e2e": main.get("e2e"), "gpu_launches": main["gpu_launches"],
            "roofline": main["roofline"], "cpu_baseline": cpu.get(a.workload),
            "kernels": main["kernels"], "alg_bytes_per_obs": main["alg_bytes_per_obs"],
            "observe_only_obs_per_s": main["observe_only_obs_per_s"],
            "workloads": extra_w, "strong_scaling": strong,
            "collectives": "none on the data path; NCCL is initialised only for this benchmark's barrier and the max-over-ranks of the time",
            "sources_sha16": sources_hash(),
        }
        emit(line)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="atari_peripheral", choices=sorted(WORKLOADS))
    ap.add_argument("--envs", type=int, default=None, help="envs per GPU (default: the BASELINE config's N)")
    ap.add_argument("--only", action="store_true", help="time only --workload (no `workloads` / `strong_scaling` extras)")
    ap.add_argument("--other-steps", type=int, default=20, help="timed steps of each extra workload")
    ap.add_argument("--shards", type=int, default=2, help="env-index shards (streams) per env group of the e2e leg")
    ap.add_argument("--cpu-steps-per-proc", type=int, default=0, help="env-steps per CPU process and sample (0 = calibrate from --cpu-seconds)")
    ap.add_argument("--cpu-seconds", type=float, default=1.5, help="wall seconds of the bounded CPU sample (x host cores = CPU work)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="time the eager launch loop only (default: the timed steps are captured in a CUDA graph; the eager time is reported next to it)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step of --workload returned (observation, fov_loc, fov_res for the flexible "
                         "fovea; 256 sampled envs, indices in env_index) as DIR/<name>.npy in float32 / float64")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3) if a.impl == "b200" else a.warmup
    quiet_stdout()
    if a.impl == "reference":
        run_reference_arm(a)
    else:
        run_b200_arm(a)


if __name__ == "__main__":
    main()
