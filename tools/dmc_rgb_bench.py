"""Throughput of the DMC ``grey=False`` (RGB) workloads on one GPU; prints one JSON line.

    python tools/dmc_rgb_bench.py [--envs 8192] [--steps 200] [--warmup 20]

Geometry of BASELINE configs[4] with colour: 84x84 renders, frame_stack K = 3, C = 3 planes per frame (a ring of 9
planes per env).  One step = the RGB ingest of a rendered batch + one observe launch.  Inputs rotate over 8 frame
batches (8 x 173 MB, well past the 126 MB L2) and 8 action sets, all device resident.  For every workload:

* env-steps/s from CUDA events over a timed window after warm-up, with the steps captured in a CUDA graph and replayed,
  and with eager launches;
* the kernels that ran and their mean device time, from ``torch.profiler`` in a separate, shorter run;
* the algorithmic bytes per env-step (what the step must read and write at least) and the share of the measured
  6,546 GB/s HBM copy bandwidth of a B200 that the graph replay reaches;
* an oracle check of a fixed sample of envs after the last timed step (tests/rgb_oracle.py).

The card's name and power limit are read in the same run.  There is no CPU fallback: without a GPU this exits non-zero.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

COPY_BW = 6546e9   # measured HBM copy bandwidth of one B200 (BASELINE.md), bytes/s
S, K, C, FOV, PERIPH = (84, 84), 3, 3, (30, 30), (20, 20)
PLANE = S[0] * S[1]
FRAME_IO = 2 * C * PLANE   # the render read (HWC) + its three planes written: 21,168 + 21,168 B
# algorithmic bytes per env-step: ingest + what the observe must read and write
WORKLOADS = {
    # relative 30x30 fovea, crop: the K*C fovea windows read + written
    "dmc_rgb_fixed": FRAME_IO + 2 * K * C * FOV[0] * FOV[1],
    # 30x30 fovea + 20x20 periphery: ring and output planes (the cached squeeze is not counted)
    "dmc_rgb_peripheral": FRAME_IO + 2 * K * C * PLANE,
    # res 20..50, mask_out: the largest window's planes read (35 x 35 on average) + the full output
    "dmc_rgb_flexible": FRAME_IO + K * C * 35 * 35 + K * C * PLANE,
}
N_BATCHES = 8
SAMPLE = 16


def card(torch):
    name = torch.cuda.get_device_name(0)
    try:
        pl = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                            capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(pl.splitlines()[0]) if pl else None
    except (OSError, ValueError, subprocess.TimeoutExpired):
        power = None
    return name, power


class Workload:
    def __init__(self, torch, name, n):
        from active_gym_b200 import LUMA_DMC, ObservationPath
        self.torch, self.name, self.n = torch, name, n
        kind = name.split("_")[-1]
        self.kind = kind
        mode = "absolute" if kind == "flexible" else "relative"
        self.p = ObservationPath(n, K, S, S + (3,), luma=LUMA_DMC, fov_size=FOV, sensory_action_mode=mode,
                                 sensory_action_space=(-10.0, 10.0), peripheral_res=PERIPH if kind == "peripheral" else None,
                                 device="cuda:0", channels=C)
        dev = self.p.device
        self.frames = [self.p.synth_frames(torch.empty((n,) + S + (3,), dtype=torch.uint8, device=dev), 1000 + i)
                       for i in range(N_BATCHES)]
        self.flags = torch.full((n,), 1, dtype=torch.uint8, device=dev)
        g = torch.Generator(device="cpu").manual_seed(7)
        if kind == "flexible":
            self.atypes = [torch.randint(0, 2, (n,), generator=g, dtype=torch.int32).to(dev) for _ in range(N_BATCHES)]
            self.actions = [torch.where(t.cpu()[:, None] == 1, torch.randint(20, 51, (n, 2), generator=g),
                                        torch.randint(0, 55, (n, 2), generator=g)).to(dev, torch.float64) for t in self.atypes]
        else:
            self.atypes = [None] * N_BATCHES
            self.actions = [torch.randint(-10, 11, (n, 2), generator=g).to(dev, torch.float64) for _ in range(N_BATCHES)]
        variant = "crop" if kind == "fixed" else "mask"
        self.variant = variant
        self.out = torch.empty(self.p.out_shape(kind, variant), dtype=torch.uint8, device=dev)
        self.i = 0
        # every env starts from a hard reset and a full ring
        self.p.ingest_dmc(self.frames[0], torch.full((n,), 5, dtype=torch.uint8, device=dev))
        for k in range(1, K):
            self.p.ingest_dmc(self.frames[k], self.flags)
        self.observe(None, "reset")

    def observe(self, a, ctrl=None, at=None):
        if self.kind == "fixed":
            return self.p.observe_fixed(a, variant="crop", ctrl=ctrl, out=self.out)
        if self.kind == "peripheral":
            return self.p.observe_peripheral(a, ctrl=ctrl, out=self.out)
        return self.p.observe_flexible(a, at, variant="mask", ctrl=ctrl, out=self.out)

    def step(self):
        j = self.i % N_BATCHES
        self.last = j
        self.p.ingest_dmc(self.frames[j], self.flags)
        self.observe(self.actions[j], at=self.atypes[j])
        self.i += 1

    def oracle_check(self):
        """A fixed sample of envs after the last step: the newest planes hold the last batch's channels, and the
        observation equals the composed oracle's on the sampled state."""
        from tests import rgb_oracle as rgb
        torch = self.torch
        torch.cuda.synchronize()
        idx = np.linspace(0, self.n - 1, SAMPLE).astype(np.int64)
        ti = torch.as_tensor(idx, device=self.p.device)
        ring, head = self.p.ring[ti].cpu().numpy(), self.p.head[ti].cpu().numpy()
        loc, res = self.p.loc[ti].cpu().numpy(), self.p.res[ti].cpu().numpy()
        frames = self.frames[self.last][ti].cpu().numpy()
        ok = all(np.array_equal(ring[e, head[e] - 2:head[e] + 1], frames[e].transpose(2, 0, 1)) for e in range(SAMPLE))
        got = self.out[ti].cpu().numpy()
        if self.kind == "fixed":
            want = rgb.observe_fixed(ring, head, loc, FOV)
            err = float(np.abs(got.astype(np.float64) - want).max())
            ok = ok and np.array_equal(got, want)
        elif self.kind == "peripheral":
            want = rgb.observe_peripheral(ring, head, loc, FOV, PERIPH)
            err = float(np.abs(got.astype(np.float64) - want).max())
            ok = ok and err <= 0.5 + 1e-2
        else:
            want = rgb.observe_flexible(ring, head, loc, res, FOV)
            err = float(np.abs(got.astype(np.float64) - want).max())
            ok = ok and err <= 0.5 + 1e-2
        return {"envs": SAMPLE, "max_abs_err_lsb": err, "ok": bool(ok)}


def time_eager(torch, wl, steps, warmup):
    for _ in range(warmup):
        wl.step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        wl.step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3


def time_graph(torch, wl, steps, warmup):
    side = torch.cuda.Stream(device=wl.p.device)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        for _ in range(max(warmup, 2)):
            wl.step()
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    steps = max(N_BATCHES, steps - steps % N_BATCHES)   # whole rotations, so every replay starts at batch 0
    wl.i = 0
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        for _ in range(steps):
            wl.step()
    graph.replay()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    graph.replay()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / 1e3, steps


def kernels(torch, wl, steps):
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(steps):
            wl.step()
        torch.cuda.synchronize()
    out = []
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None)
        if t is None:
            t = ev.cuda_time_total
        if t <= 0 or ev.count == 0:
            continue
        out.append({"name": ev.key[:160], "calls": ev.count, "mean_us": round(t / ev.count, 2)})
    return sorted(out, key=lambda k: -k["mean_us"] * k["calls"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=8192)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--profile-steps", type=int, default=16)
    ap.add_argument("--workloads", default=",".join(WORKLOADS))
    args = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        sys.exit("tools/dmc_rgb_bench.py needs a CUDA device (B200); there is no CPU fallback")
    torch.cuda.set_device(0)
    name, power = card(torch)
    result = {"tool": "dmc_rgb_bench", "gpu": name, "power_limit_w": power, "envs": args.envs, "frame_stack": K,
              "channels": C, "obs_size": list(S), "frame_batches": N_BATCHES, "steps": args.steps, "workloads": {}}
    for wname in args.workloads.split(","):
        wl = Workload(torch, wname, args.envs)
        eager_s = time_eager(torch, wl, args.steps, args.warmup)
        graph_s, gsteps = time_graph(torch, wl, args.steps, args.warmup)
        check = wl.oracle_check()
        kern = kernels(torch, wl, args.profile_steps)
        b = WORKLOADS[wname]
        rate_g = args.envs * gsteps / graph_s
        result["workloads"][wname] = {
            "env_steps_per_s_graph": round(rate_g), "env_steps_per_s_eager": round(args.envs * args.steps / eager_s),
            "step_ms_graph": round(1e3 * graph_s / gsteps, 4), "step_ms_eager": round(1e3 * eager_s / args.steps, 4),
            "algorithmic_bytes_per_env_step": b, "roofline_env_steps_per_s": round(COPY_BW / b),
            "share_of_copy_bw_graph": round(rate_g * b / COPY_BW, 3), "kernels": kern, "oracle_check": check,
        }
        del wl
        torch.cuda.empty_cache()
    print(json.dumps(result))
    if not all(w["oracle_check"]["ok"] for w in result["workloads"].values()):
        sys.exit("oracle check failed")


if __name__ == "__main__":
    main()
