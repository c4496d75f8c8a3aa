"""Timing of the flexible fovea's glimpse (``resize_to_fov``, AGYM_OUT_RESIZE_FOV) on one GPU; prints one JSON line.

Workloads: BASELINE configs[2] (Atari grey, K=4, fov 30x30, res uniform 20..50, action type Bernoulli(0.5)) at 4,096 and
16,384 envs, and DMC RGB (K=3, C=3) at 8,192 envs.  Each workload rotates 8 independent env batches (rings filled with
random pixels), so the rings read per rotation (0.9 to 4.2 GB) exceed the 126 MB L2.  Per workload:
  * the observe step of one batch (mean over the rotation), CUDA graph and eager, for the glimpse and for mask_out on
    the same batches, and for the table-driven glimpse kernel (reached by an output view at an odd address);
  * per-kernel time from torch.profiler in a separate run;
  * algorithmic bytes of the glimpse step from the step's actual res, K * (sum rh * rw + N * f_h * f_w), and their share
    of 6,546 GB/s (measured copy bandwidth of the card, DESIGN section 3);
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

S, FOV, ROT, PEAK_GBS = (84, 84), (30, 30), 8, 6546.0


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


def _batches(n, K, C, seed):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    raw = (210, 160, 1) if C == 1 else S + (3,)
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = []
    for b in range(ROT):
        p = ObservationPath(n, K, S, raw, fov_size=FOV, sensory_action_mode="absolute", device="cuda:0", channels=C,
                            **({} if C == 1 else {"luma": LUMA_DMC}))
        p.ring.copy_(torch.randint(0, 256, p.ring.shape, dtype=torch.uint8, device="cuda", generator=g))
        at = (torch.rand(n, device="cuda", generator=g) < 0.5).to(torch.int32)
        res = torch.randint(20, 51, (n, 2), device="cuda", generator=g).to(torch.float64)
        loc = torch.randint(0, 85, (n, 2), device="cuda", generator=g).to(torch.float64)
        a = torch.where(at[:, None] == 1, res, loc).contiguous()
        # start from windows of 20..50 as well, so FOV_LOC envs also carry a drawn res
        p.observe_flexible(res, torch.ones(n, dtype=torch.int32, device="cuda"), variant="mask")
        out.append((p, a, at))
    torch.cuda.synchronize()
    return out


def _time(batches, variant, outs, steps, warmup, graph):
    def rotation():
        for (p, a, at), o in zip(batches, outs):
            p.observe_flexible(a, at, variant=variant, out=o)
    for _ in range(warmup):
        rotation()
    torch.cuda.synchronize()
    fn = rotation
    if graph:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            rotation()
        torch.cuda.current_stream().wait_stream(s)
        torch.cuda.synchronize()
        gr = torch.cuda.CUDAGraph()
        with torch.cuda.graph(gr):
            rotation()
        gr.replay()
        fn = gr.replay
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (steps * len(batches))   # ms per observe step of one batch


def _kernel_times(batches, variant, outs, reps=5):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(reps):
            for (p, a, at), o in zip(batches, outs):
                p.observe_flexible(a, at, variant=variant, out=o)
        torch.cuda.synchronize()
    agg = {}
    for e in prof.key_averages():
        if e.device_type == torch.autograd.DeviceType.CUDA and "observe_flexible" in e.key:
            t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
            agg[e.key.replace("void agym::(anonymous namespace)::", "").split("(")[0]] = round(t / 1e3 / (reps * len(batches)), 5)
    return agg   # ms per launch


def _oracle_check(p, out, m=64):
    from tests.glimpse_oracle import observe_glimpse
    idx = np.random.default_rng(0).choice(p.n_envs, min(m, p.n_envs), replace=False)
    ring, head = p.ring[idx].cpu().numpy(), p.head[idx].cpu().numpy()
    want = observe_glimpse(ring, head, p.loc[idx].cpu().numpy(), p.res[idx].cpu().numpy(), FOV)
    got = out[idx].cpu().numpy().reshape(want.shape).astype(np.float64)
    return float(np.abs(got - want).max())


def workload(name, n, K, C, steps, warmup):
    b = _batches(n, K, C, seed=n + C)
    shp = b[0][0].out_shape("flexible", "resize_fov")
    glimpse = [torch.empty(shp, dtype=torch.uint8, device="cuda") for _ in b]
    mask = torch.empty(b[0][0].out_shape("flexible", "mask"), dtype=torch.uint8, device="cuda")
    nb = int(np.prod(shp))
    raw = torch.empty(nb + 16, dtype=torch.uint8, device="cuda")
    odd = raw[1:1 + nb].view(shp)   # the table-driven kernel: an output that is not 4-byte aligned
    r = {"workload": name, "envs": n, "frame_stack": K, "channels": C, "rotation": ROT,
         "ring_bytes_per_rotation": int(sum(p.ring.numel() for p, _, _ in b))}
    for label, variant, outs in (("glimpse", "resize_fov", glimpse), ("mask_out", "mask", [mask] * ROT),
                                 ("glimpse_generic", "resize_fov", [odd] * ROT)):
        r[f"{label}_ms_graph"] = round(_time(b, variant, outs, steps, warmup, True), 5)
        r[f"{label}_ms_eager"] = round(_time(b, variant, outs, steps, warmup, False), 5)
        r[f"{label}_kernels_ms"] = _kernel_times(b, variant, outs)
    # algorithmic bytes of one glimpse step, from the res each env holds after the timed steps
    res = torch.stack([p.res.to(torch.float64) for p, _, _ in b])
    alg = K * C * (float((res[..., 0] * res[..., 1]).sum()) / ROT + n * FOV[0] * FOV[1])
    r["glimpse_alg_bytes_per_step"] = int(alg)
    r["glimpse_alg_GBps_graph"] = round(alg / (r["glimpse_ms_graph"] * 1e-3) / 1e9, 1)
    r["glimpse_share_of_6546_GBps"] = round(r["glimpse_alg_GBps_graph"] / PEAK_GBS, 4)
    r["glimpse_env_steps_per_sec_graph"] = round(n / (r["glimpse_ms_graph"] * 1e-3), 0)
    r["fast_over_generic"] = round(r["glimpse_generic_ms_graph"] / r["glimpse_ms_graph"], 3)
    # one more glimpse step on batch 0, then the oracle on sampled envs
    p, a, at = b[0]
    p.observe_flexible(a, at, variant="resize_fov", out=glimpse[0])
    torch.cuda.synchronize()
    r["oracle_max_abs_lsb"] = _oracle_check(p, glimpse[0])
    del b, glimpse, mask, raw
    torch.cuda.empty_cache()
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=40, help="timed rotations (8 observe steps each)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="one tiny workload (a smoke run of this tool)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("flexible_glimpse_bench needs a CUDA device")
    name, power = _card()
    line = {"what": "flexible glimpse (resize_to_fov) vs mask_out vs the table-driven glimpse kernel; observe step only, "
                    "8 independent env batches rotated (working set > 126 MB L2)",
            "gpu": name, "power_limit_w": power, "steps": args.steps, "workloads": []}
    todo = [("smoke", 64, 4, 1)] if args.small else [("configs2_atari_grey", 4096, 4, 1), ("configs2_atari_grey", 16384, 4, 1),
                                                     ("dmc_rgb", 8192, 3, 3)]
    for w in todo:
        line["workloads"].append(workload(*w, steps=args.steps, warmup=args.warmup))
    print(json.dumps(line))


if __name__ == "__main__":
    main()
