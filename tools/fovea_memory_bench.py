"""Timing of the fixed fovea's memory (agym_observe_fixed_memory) against the composed PyTorch form on one GPU; prints one
JSON line.

Workloads: Atari grey (K=4, fov 30x30, relative mode) at 4,096 and 16,384 envs and DMC RGB (K*C=9, fov 30x30) at 8,192
envs, each at depth M = 3 and M = 8.  Each workload rotates 8 independent env batches whose rings were filled by the
ingest kernels from random frames and whose memories hold M entries, so the state read per rotation exceeds the 126 MB
L2.  Per workload:
  * the fused step (one agym_observe_fixed_memory launch per batch), CUDA graph and eager;
  * the composed step on the same batches: the mask_out kernel writing into one slot of a rolling (M, N, P, S_h, S_w)
    buffer (slot-major, so that a slot is the contiguous output the kernel needs), then torch.amax over the slots;
  * per-kernel time from torch.profiler in a separate run;
  * algorithmic bytes per env-step from shapes: fused P S_h S_w + (M + 1) P f_h f_w, composed
    P f_h f_w + (M + 2) P S_h S_w, and their rate at the measured time as a share of 6,546 GB/s;
  * an oracle check of 64 sampled envs of batch 0 (tests/fovea_memory_oracle.py over M + 1 fresh steps).
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

S, FOV, ROT, HBM_GBPS = (84, 84), (30, 30), 8, 6546.0


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


def _ingest(p, g):
    n = p.n_envs
    fl = torch.full((n,), 1, dtype=torch.uint8, device="cuda")
    if p.channels == 1:
        p.ingest_atari(*[torch.randint(0, 256, (n, 210, 160), dtype=torch.uint8, device="cuda", generator=g) for _ in range(2)], fl)
    else:
        p.ingest_dmc(torch.randint(0, 256, (n,) + S + (3,), dtype=torch.uint8, device="cuda", generator=g), fl)


def _batches(n, K, C, M, seed):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    raw = (210, 160, 1) if C == 1 else S + (3,)
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = []
    for b in range(ROT):
        p = ObservationPath(n, K, S, raw, fov_size=FOV, fov_init_loc=(27, 27), sensory_action_mode="relative",
                            sensory_action_space=(-10.0, 10.0), device="cuda:0", channels=C, fov_memory=M,
                            **({} if C == 1 else {"luma": LUMA_DMC}))
        p.observe_fixed_memory(None, ctrl="reset")
        for k in range(max(K, M)):   # distinct frames in the ring, a full memory
            _ingest(p, g)
            p.observe_fixed_memory(torch.randint(-10, 11, (n, 2), device="cuda", generator=g).to(torch.float64))
        a = torch.randint(-10, 11, (n, 2), device="cuda", generator=g).to(torch.float64)
        out.append((p, a))
    torch.cuda.synchronize()
    return out


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
        if e.device_type == torch.autograd.DeviceType.CUDA:
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
            key = e.key.replace("void ", "").replace("agym::(anonymous namespace)::", "").split("(")[0][:60]
            agg[key] = round(agg.get(key, 0.0) + t / 1e3 / (reps * ROT), 5)
    return agg   # ms per launch


def _oracle_check(p, M, m=64):
    """M + 1 fresh steps of batch 0 from an empty memory, the composed oracle on 64 sampled envs."""
    from tests.fovea_memory_oracle import APPLY, RESET, MemoryOracle
    idx = np.random.default_rng(0).choice(p.n_envs, min(m, p.n_envs), replace=False)
    mem = MemoryOracle(len(idx), M)
    g = torch.Generator(device="cuda").manual_seed(5)
    out = None
    for step in range(M + 1):
        _ingest(p, g)
        a = torch.randint(-10, 11, (p.n_envs, 2), device="cuda", generator=g).to(torch.float64)
        out = p.observe_fixed_memory(a, ctrl=None if step else "reset")
        torch.cuda.synchronize()
        want = mem.observe(p.ring[idx].cpu().numpy(), p.head[idx].cpu().numpy(), p.loc[idx].cpu().numpy(), FOV,
                           np.full(len(idx), APPLY if step else RESET, np.uint8), rgb=p.channels == 3)
    return bool(np.array_equal(out[idx].cpu().numpy().reshape(want.shape), want))


def workload(name, n, K, C, M, steps, warmup):
    b = _batches(n, K, C, M, seed=n + C + M)
    P, plane, A = K * C, S[0] * S[1], FOV[0] * FOV[1]
    shp = b[0][0].out_shape("fixed_memory", "mask")
    outs = [torch.empty(shp, dtype=torch.uint8, device="cuda") for _ in b]
    # the composed form: a rolling buffer of M mask_out observations per batch, slot-major
    rolls = [torch.zeros((M,) + tuple(shp), dtype=torch.uint8, device="cuda") for _ in b]
    r = {"workload": name, "envs": n, "frame_stack": K, "channels": C, "depth": M, "rotation": ROT,
         "state_bytes_per_rotation_fused": int(sum(p.ring.numel() + p.mem.numel() for p, _ in b)),
         "state_bytes_per_rotation_composed": int(sum(p.ring.numel() for p, _ in b) + sum(x.numel() for x in rolls))}

    def fused():
        for i, (p, a) in enumerate(b):
            p.observe_fixed_memory(a, out=outs[i])

    def composed():
        for i, (p, a) in enumerate(b):
            p.observe_fixed(a, variant="mask", out=rolls[i][i % M])
            torch.amax(rolls[i], dim=0, out=outs[i])

    cases = (("fused", fused), ("composed", composed))
    for label, fn in cases:
        r[f"{label}_ms_graph"] = round(_time(fn, steps, warmup, True), 5)
        r[f"{label}_ms_eager"] = round(_time(fn, steps, warmup, False), 5)
    for label, fn in cases:   # the profiler in runs of its own
        r[f"{label}_kernels_ms"] = _kernel_times(fn)
    alg_f = P * plane + (M + 1) * P * A
    alg_c = P * A + (M + 2) * P * plane
    r["alg_bytes_per_env_step_fused"], r["alg_bytes_per_env_step_composed"] = alg_f, alg_c
    for label, alg in (("fused", alg_f), ("composed", alg_c)):
        gbps = alg * n / (r[f"{label}_ms_graph"] * 1e-3) / 1e9
        r[f"alg_GBps_{label}_graph"] = round(gbps, 1)
        r[f"alg_share_of_6546GBps_{label}_graph"] = round(gbps / HBM_GBPS, 3)
    r["speedup_graph"] = round(r["composed_ms_graph"] / r["fused_ms_graph"], 3)
    r["bar_fused_faster_graph"] = r["fused_ms_graph"] < r["composed_ms_graph"]
    r["oracle_64_envs_bit_exact"] = _oracle_check(b[0][0], M)
    del b, outs, rolls
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=30, help="timed rotations (8 steps each)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="one tiny workload (a smoke run of this tool)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("fovea_memory_bench needs a CUDA device")
    name, power = _card()
    line = {"what": "fixed fovea memory: the fused kernel vs mask_out into a rolling buffer + torch.amax on the same "
                    "batches; 8 independent env batches rotated (working set > 126 MB L2)",
            "gpu": name, "power_limit_w": power, "steps": args.steps, "workloads": []}
    todo = [("smoke", 64, 4, 1, 3)] if args.small else [
        (w, n, K, C, M) for M in (3, 8) for (w, n, K, C) in (("atari_grey_relative", 4096, 4, 1), ("atari_grey_relative", 16384, 4, 1),
                                                            ("dmc_rgb", 8192, 3, 3))]
    for w in todo:
        line["workloads"].append(workload(*w, steps=args.steps, warmup=args.warmup))
    print(json.dumps(line))


if __name__ == "__main__":
    main()
