"""Timing of the flexible fovea over the peripheral background (agym_observe_flexible_peripheral) on one GPU; prints one
JSON line.

Workloads: BASELINE configs[2] (Atari grey, K=4, fov 30x30, periphery 20x20, res uniform 20..50, action type
Bernoulli(0.5)) at 4,096 and 16,384 envs, and DMC RGB (K=3, C=3, same fovea and periphery) at 8,192 envs.  Each workload
rotates 8 independent env batches whose rings and squeeze caches were filled by the ingest kernels from random frames,
so the rings and caches read per rotation (1.1 to 4.6 GB) exceed the 126 MB L2.  Per workload:
  * the observe step of one batch (mean over the rotation), CUDA graph and eager, for the fused kernel, for mask_out
    (k_observe_flexible_v3<MASK>) and for the peripheral kernel the plan selects (agym_observe_peripheral) on the same
    batches, and for the table-driven fused kernel (reached by an output view at an odd address);
  * the full step, ingest (refreshing the squeeze cache) + fused observe, graph and eager;
  * per-kernel time from torch.profiler in a separate run;
  * algorithmic bytes per observation, K * E[rh * rw] window bytes + the fp32 cache read K * p_h * p_w * 4 + the
    K * S_h * S_w bytes written (39,524 B at configs[2]), from the res each env holds;
  * an oracle check of 64 sampled envs of batch 0 after the timed steps.
The card's name and power limit are read in the same call.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

S, FOV, PER, ROT = (84, 84), (30, 30), (20, 20), 8


def _card():
    name, power = torch.cuda.get_device_name(0), None
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader,nounits", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        name, power = [v.strip() for v in q.stdout.strip().split(",")][:2]
        power = float(power)
    except Exception:
        pass
    return name, power


def _frames(n, C, g):
    """One set of random frames per workload, shared by its batches: Atari (a, b) screens or DMC renders."""
    if C == 1:
        return [torch.randint(0, 256, (n, 210, 160), dtype=torch.uint8, device="cuda", generator=g) for _ in range(2)]
    return [torch.randint(0, 256, (n,) + S + (3,), dtype=torch.uint8, device="cuda", generator=g)]


def _ingest(p, frames, flags):
    if p.channels == 1 and p.raw_shape[0] != S[0]:
        p.ingest_atari(frames[0], frames[1], flags)
    else:
        p.ingest_dmc(frames[0], flags)


def _batches(n, K, C, seed):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    raw = (210, 160, 1) if C == 1 else S + (3,)
    g = torch.Generator(device="cuda").manual_seed(seed)
    frames = _frames(n, C, g)
    out = []
    for b in range(ROT):
        p = ObservationPath(n, K, S, raw, fov_size=FOV, peripheral_res=PER, sensory_action_mode="absolute",
                            device="cuda:0", channels=C, **({} if C == 1 else {"luma": LUMA_DMC}))
        flags = torch.full((n,), 1, dtype=torch.uint8, device="cuda")
        for k in range(K):   # fill the ring and the squeeze cache with distinct frames
            fr = [torch.randint(0, 256, f.shape, dtype=torch.uint8, device="cuda", generator=g) for f in frames]
            _ingest(p, fr, torch.full((n,), 5 if k == 0 else 1, dtype=torch.uint8, device="cuda"))
        at = (torch.rand(n, device="cuda", generator=g) < 0.5).to(torch.int32)
        res = torch.randint(20, 51, (n, 2), device="cuda", generator=g).to(torch.float64)
        loc = torch.randint(0, 85, (n, 2), device="cuda", generator=g).to(torch.float64)
        a = torch.where(at[:, None] == 1, res, loc).contiguous()
        # start from windows of 20..50 as well, so FOV_LOC envs also carry a drawn res
        p.observe_flexible_peripheral(res, torch.ones(n, dtype=torch.int32, device="cuda"))
        out.append((p, a, at, flags))
    torch.cuda.synchronize()
    return out, frames


def _call(kind, p, a, at, o):
    if kind == "fused":
        p.observe_flexible_peripheral(a, at, out=o)
    elif kind == "mask_out":
        p.observe_flexible(a, at, variant="mask", out=o)
    else:
        p.observe_peripheral(a, out=o)


def _time(fn, steps, warmup, graph):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    run = fn
    if graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            fn()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            fn()
        gr.replay()
        run = gr.replay
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        run()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (steps * ROT)   # ms per step of one batch


def _kernel_times(fn, reps=5):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            fn()
        torch.cuda.synchronize()
    agg = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and ("observe" in e.key or "ingest" in e.key):
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
            agg[e.key.replace("void agym::(anonymous namespace)::", "").split("(")[0]] = round(t / 1e3 / (reps * ROT), 5)
    return agg   # ms per launch


def _oracle_check(p, out, m=64):
    from tests.flex_periph_oracle import observe_flexible_peripheral
    idx = np.random.default_rng(0).choice(p.n_envs, min(m, p.n_envs), replace=False)
    ring, head = p.ring[idx].cpu().numpy(), p.head[idx].cpu().numpy()
    want = observe_flexible_peripheral(ring, head, p.loc[idx].cpu().numpy(), p.res[idx].cpu().numpy(), FOV, PER)
    got = out[idx].cpu().numpy().reshape(want.shape).astype(np.float64)
    return float(np.abs(got - want).max())


def workload(name, n, K, C, steps, warmup):
    b, frames = _batches(n, K, C, seed=n + C)
    shp = b[0][0].out_shape("flexible_peripheral", "mask")
    outs = [torch.empty(shp, dtype=torch.uint8, device="cuda") for _ in b]
    nb = int(np.prod(shp))
    raw = torch.empty(nb + 16, dtype=torch.uint8, device="cuda")
    odd = raw[1:1 + nb].view(shp)   # the table-driven kernel: an output that is not 16-byte aligned
    r = {"workload": name, "envs": n, "frame_stack": K, "channels": C, "rotation": ROT,
         "ring_and_cache_bytes_per_rotation": int(sum(p.ring.numel() + 4 * p.pcache.numel() for p, *_ in b))}

    def rotation(kind, o=None):
        return lambda: [_call(kind, p, a, at, outs[i] if o is None else o) for i, (p, a, at, _) in enumerate(b)]

    def full_step():
        for i, (p, a, at, fl) in enumerate(b):
            _ingest(p, frames, fl)
            p.observe_flexible_peripheral(a, at, out=outs[i])

    cases = (("fused", rotation("fused")), ("mask_out", rotation("mask_out")), ("peripheral", rotation("peripheral")),
             ("fused_generic", rotation("fused", odd)), ("full_step", full_step))
    for label, fn in cases:
        r[f"{label}_ms_graph"] = round(_time(fn, steps, warmup, True), 5)
        r[f"{label}_ms_eager"] = round(_time(fn, steps, warmup, False), 5)
    for label, fn in cases:   # the profiler in runs of its own
        r[f"{label}_kernels_ms"] = _kernel_times(fn)
    r["bar_fused_lt_mask_plus_peripheral_graph"] = r["fused_ms_graph"] < r["mask_out_ms_graph"] + r["peripheral_ms_graph"]
    r["fast_over_generic"] = round(r["fused_generic_ms_graph"] / r["fused_ms_graph"], 3)
    # one more fused step on batch 0, then the algorithmic bytes from its res and the oracle on sampled envs
    p, a, at, _ = b[0]
    p.observe_flexible_peripheral(a, at, out=outs[0])
    torch.cuda.synchronize()
    res = p.res.to(torch.float64)
    win = float((res[:, 0] * res[:, 1]).mean())
    alg = K * C * (win + PER[0] * PER[1] * 4 + S[0] * S[1])
    r["alg_bytes_per_obs"] = round(alg, 1)
    r["alg_GBps_fused_graph"] = round(alg * n / (r["fused_ms_graph"] * 1e-3) / 1e9, 1)
    r["env_steps_per_sec_fused_graph"] = round(n / (r["fused_ms_graph"] * 1e-3), 0)
    r["oracle_max_abs_lsb"] = _oracle_check(p, outs[0])
    del b, outs, raw, frames
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=30, help="timed rotations (8 steps each)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="one tiny workload (a smoke run of this tool)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("flexible_peripheral_bench needs a CUDA device")
    name, power = _card()
    line = {"what": "flexible fovea over the peripheral background: the fused kernel vs mask_out and the peripheral kernel "
                    "on the same batches, the table-driven fused kernel, and the full step (ingest + observe); "
                    "8 independent env batches rotated (working set > 126 MB L2)",
            "gpu": name, "power_limit_w": power, "steps": args.steps, "workloads": []}
    todo = [("smoke", 64, 4, 1)] if args.small else [("configs2_atari_grey", 4096, 4, 1), ("configs2_atari_grey", 16384, 4, 1),
                                                     ("dmc_rgb", 8192, 3, 3)]
    for w in todo:
        line["workloads"].append(workload(*w, steps=args.steps, warmup=args.warmup))
    print(json.dumps(line))


if __name__ == "__main__":
    main()
