"""Timing of the pasted foveal memory (agym_observe_fixed_memory_paste) against the composed PyTorch form a user runs
without it, on one GPU; prints one JSON line.

Workloads: Atari grey (K=4, fov 30x30, periphery 20x20, relative mode) at 4,096 and 16,384 envs and DMC RGB (K*C=9) at
8,192 envs, each at depth M = 3 and M = 8 and over both backgrounds (zero = mask_out's, periphery =
FixedFovealPeripheralEnv's).  Each workload rotates 8 independent env batches whose rings and squeeze caches were filled
by the ingest kernels from random frames and whose memories hold M entries, so the state read per rotation exceeds the
126 MB L2.  Per workload:
  * the fused step (one agym_observe_fixed_memory_paste launch per batch), CUDA graph and eager;
  * the composed step on the same batches: observe_peripheral (or observe_fixed("mask")), observe_fixed("crop") with
    every env on KEEP into one slot of a rolling (M, N, P, f_h, f_w) crop buffer and the loc into an (M, N, 2) one
    (slot-major, so that a slot is the contiguous output the kernel needs), then the M - 1 older crops pasted over the
    output oldest to newest and the current crop last, by torch advanced indexing;
  * per-kernel time from torch.profiler in a separate run;
  * algorithmic bytes per env-step from shapes: periphery 4 P p_h p_w + (M + 1) P f_h f_w + P S_h S_w (squeeze, window,
    M - 1 older entries, new entry, output: 38,224 + 3,600 M at configs[3]), zero (M + 1) P f_h f_w + P S_h S_w, and
    their rate at the measured time as a share of 6,546 GB/s (the measured copy bandwidth of the card);
  * an oracle check of 64 sampled envs of batch 0 (tests/memory_paste_oracle.py over M + 1 fresh steps: pasted pixels
    exact, the periphery within 0.5 LSB + 0.01).
The card's name and power limit are read in the same call.  Needs a CUDA device.
"""
from __future__ import annotations

import argparse
import json
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tools.fovea_memory_bench import HBM_GBPS, ROT, S, _card, _ingest, _kernel_times, _time  # noqa: E402

FOV, PER = (30, 30), (20, 20)


def _batches(n, K, C, M, seed):
    from active_gym_b200 import LUMA_DMC, ObservationPath
    raw = (210, 160, 1) if C == 1 else S + (3,)
    g = torch.Generator(device="cuda").manual_seed(seed)
    out = []
    for b in range(ROT):
        p = ObservationPath(n, K, S, raw, fov_size=FOV, fov_init_loc=(27, 27), sensory_action_mode="relative",
                            sensory_action_space=(-10.0, 10.0), device="cuda:0", channels=C, fov_memory=M,
                            peripheral_res=PER, **({} if C == 1 else {"luma": LUMA_DMC}))
        p.observe_memory_paste(None, ctrl="reset")
        for k in range(max(K, M)):   # distinct frames in the ring, a full memory
            _ingest(p, g)
            p.observe_memory_paste(torch.randint(-10, 11, (n, 2), device="cuda", generator=g).to(torch.float64))
        a = torch.randint(-10, 11, (n, 2), device="cuda", generator=g).to(torch.float64)
        out.append((p, a))
    torch.cuda.synchronize()
    return out


def _oracle_check(p, M, background, m=64):
    """M + 1 fresh steps of batch 0 from an empty memory, the composed oracle on 64 sampled envs."""
    from oracle import agym_oracle  # noqa: F401  (builds the oracle library on first use)
    from tests.memory_paste_oracle import APPLY, RESET, PasteOracle
    idx = np.random.default_rng(0).choice(p.n_envs, min(m, p.n_envs), replace=False)
    mem = PasteOracle(len(idx), M)
    g = torch.Generator(device="cuda").manual_seed(5)
    per = PER if background == "periphery" else None
    ok = True
    for step in range(M + 1):
        _ingest(p, g)
        a = torch.randint(-10, 11, (p.n_envs, 2), device="cuda", generator=g).to(torch.float64)
        out = p.observe_memory_paste(a, ctrl=None if step else "reset", background=background)
        torch.cuda.synchronize()
        want = mem.observe(p.ring[idx].cpu().numpy(), p.head[idx].cpu().numpy(), p.loc[idx].cpu().numpy(), FOV,
                           np.full(len(idx), APPLY if step else RESET, np.uint8), peripheral_res=per)
        got = out[idx].cpu().numpy().reshape(want.shape).astype(np.float64)
        pasted = np.broadcast_to(mem.pasted(S, FOV)[:, None], got.shape)
        ok = ok and bool(np.array_equal(got[pasted], want[pasted])) and float(np.abs(got - want).max()) <= 0.5 + 1e-2
    return ok


def workload(b, name, n, K, C, M, background, steps, warmup):
    P, plane, A = K * C, S[0] * S[1], FOV[0] * FOV[1]
    shp = b[0][0].out_shape("fixed_memory", "mask")
    outs = [torch.empty(shp, dtype=torch.uint8, device="cuda") for _ in b]
    # the composed form: rolling crop and loc buffers of M slots per batch, slot-major
    crops = [torch.zeros((M, n, P) + FOV, dtype=torch.uint8, device="cuda") for _ in b]
    locs = [torch.zeros((M, n, 2), dtype=torch.int32, device="cuda") for _ in b]
    keep = torch.full((n,), 2, dtype=torch.uint8, device="cuda")
    nn = torch.arange(n, device="cuda")[:, None, None]
    dy, dx = torch.arange(FOV[0], device="cuda")[None, :, None], torch.arange(FOV[1], device="cuda")[None, None, :]
    r = {"workload": name, "background": background, "envs": n, "frame_stack": K, "channels": C, "depth": M,
         "rotation": ROT, "state_bytes_per_rotation_fused": int(sum(p.ring.numel() + p.mem.numel() + p.pcache.numel() * 4
                                                                    for p, _ in b))}

    def fused():
        for i, (p, a) in enumerate(b):
            p.observe_memory_paste(a, background=background, out=outs[i])

    def composed():
        for i, (p, a) in enumerate(b):
            s = i % M   # this step's slot (a graph replays one slot: the work per step is the same)
            if background == "periphery":
                p.observe_peripheral(a, out=outs[i])
            else:
                p.observe_fixed(a, variant="mask", out=outs[i])
            p.observe_fixed(None, variant="crop", ctrl=keep, out=crops[i][s])
            locs[i][s].copy_(p.loc)
            o = outs[i].view(n, P, S[0], S[1])
            for j in range(1, M + 1):   # oldest to newest, the current crop last
                t = (s + j) % M
                rr = locs[i][t][:, 0, None, None] + dy
                cc = locs[i][t][:, 1, None, None] + dx
                o[nn, :, rr, cc] = crops[i][t].permute(0, 2, 3, 1)

    cases = (("fused", fused), ("composed", composed))
    for label, fn in cases:
        try:
            r[f"{label}_ms_graph"] = round(_time(fn, steps, warmup, True), 5)
        except RuntimeError as e:   # a capture the composed form cannot take: report its eager time alone
            r[f"{label}_ms_graph"], r[f"{label}_graph_error"] = None, str(e).splitlines()[0][:200]
        r[f"{label}_ms_eager"] = round(_time(fn, steps, warmup, False), 5)
    for label, fn in cases:   # the profiler in runs of its own
        r[f"{label}_kernels_ms"] = _kernel_times(fn)
    alg = (M + 1) * P * A + P * plane + (4 * P * PER[0] * PER[1] if background == "periphery" else 0)
    r["alg_bytes_per_env_step_fused"] = alg
    gbps = alg * n / (r["fused_ms_graph"] * 1e-3) / 1e9
    r["alg_GBps_fused_graph"] = round(gbps, 1)
    r["alg_share_of_6546GBps_fused_graph"] = round(gbps / HBM_GBPS, 3)
    r["copy_floor_ms"] = round(alg * n / (HBM_GBPS * 1e9) * 1e3, 5)
    if r["composed_ms_graph"] is not None:
        r["speedup_graph"] = round(r["composed_ms_graph"] / r["fused_ms_graph"], 3)
    r["speedup_eager"] = round(r["composed_ms_eager"] / r["fused_ms_eager"], 3)
    del outs, crops, locs
    return r


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--steps", type=int, default=30, help="timed rotations (8 steps each)")
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--small", action="store_true", help="one tiny workload (a smoke run of this tool)")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("memory_paste_bench needs a CUDA device")
    name, power = _card()
    line = {"what": "pasted foveal memory: the fused kernel vs the composed observe + rolling crop buffer + torch indexing "
                    "paste on the same batches; 8 independent env batches rotated (working set > 126 MB L2)",
            "gpu": name, "power_limit_w": power, "steps": args.steps, "workloads": []}
    todo = [("smoke", 64, 4, 1, 3)] if args.small else [
        (w, n, K, C, M) for M in (3, 8) for (w, n, K, C) in (("atari_grey_relative", 4096, 4, 1), ("atari_grey_relative", 16384, 4, 1),
                                                            ("dmc_rgb", 8192, 3, 3))]
    for w, n, K, C, M in todo:
        b = _batches(n, K, C, M, seed=n + C + M)
        for bg in ("periphery", "zero"):
            r = workload(b, w, n, K, C, M, bg, steps=args.steps, warmup=args.warmup)
            r["oracle_64_envs"] = _oracle_check(b[0][0], M, bg)
            line["workloads"].append(r)
        del b
        torch.cuda.empty_cache()
    print(json.dumps(line))


if __name__ == "__main__":
    main()
