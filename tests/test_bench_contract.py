"""CPU: the bench.py contract that can be checked without a GPU — the reference arm prints ONE JSON line with
the agreed keys, and the b200 arm refuses to run (loudly) when there is no CUDA device."""
import json
import os
import subprocess
import sys

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(*args, env=None):
    e = dict(os.environ)
    e.update(env or {})
    return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                          cwd=ROOT, env=e, timeout=600)


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    r = _run("--impl", "reference", "--steps", "2", "--warmup", "1", "--cpu-seconds", "0.6")
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "foveal_obs_per_sec" and d["unit"] == "obs/s"
    assert d["higher_is_better"] is True and d["steps"] == 2 and d["warmup"] == 1 and d["value"] > 0
    assert d["config"]["workload"] == "atari_peripheral"
    cb = d["cpu_baseline"]
    # "reference" = the unmodified reference from $AGYM_REFERENCE_ROOT or oracle/_ref under the simulator stubs; "port" otherwise
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and "sample" in cb
    sys.path.insert(0, ROOT)
    from oracle import ref_harness
    assert cb["kind"] == ("reference" if ref_harness.reference_available() else "port")
    import bench
    assert d["config"] == bench.config_for("atari_peripheral", 16384, 1)   # the b200 arm prints the same object
    assert d["e2e"] == {"value": d["value"], "unit": "obs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_reference_arm_other_ranks_exit_quietly():
    r = _run("--impl", "reference", "--gpus", "2", "--steps", "1", "--warmup", "1", env={"RANK": "1", "WORLD_SIZE": "2", "LOCAL_RANK": "1"})
    assert r.returncode == 0 and r.stdout.strip() == ""


@pytest.mark.skipif(torch.cuda.is_available(), reason="needs a machine without a GPU")
def test_b200_arm_fails_loudly_without_a_gpu():
    r = _run("--steps", "1", "--warmup", "1", "--no-cpu-baseline", "--no-e2e")
    assert r.returncode != 0
    assert "CUDA" in (r.stderr + r.stdout) or "cuda" in (r.stderr + r.stdout)


@pytest.mark.gpu
def test_dump_outputs_writes_the_last_timed_step_as_float_arrays(tmp_path):
    import numpy as np
    r = _run("--workload", "atari_flexible", "--envs", "300", "--steps", "3", "--warmup", "1", "--only", "--no-e2e",
             "--no-cpu-baseline", "--dump-outputs", str(tmp_path))
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == 3
    d = {f[:-4]: np.load(tmp_path / f) for f in os.listdir(tmp_path)}
    assert set(d) == {"env_index", "obs", "fov_loc", "fov_res"}
    assert all(a.dtype in (np.float32, np.float64) for a in d.values())
    assert sum(a.nbytes for a in d.values()) <= 64 << 20
    idx = d["env_index"]
    assert len(idx) == 256 and np.all(np.diff(idx) > 0) and 0 <= idx[0] and idx[-1] < 300
    assert d["obs"].shape == (256, 4, 84, 84) and d["obs"].min() >= 0 and d["obs"].max() <= 255
    assert d["fov_loc"].shape == d["fov_res"].shape == (256, 2) and d["fov_res"].min() >= 20 and d["fov_res"].max() <= 50
    # the content: the sampled envs replayed through the CPU oracle, on the same seeded inputs, for every step the bench
    # ran before the dump (reset; eager warm-up + eager timed steps + graph warm-up; the captured steps replayed twice)
    sys.path.insert(0, ROOT)
    import bench
    from oracle import agym_oracle as orc
    idx = idx.astype(np.int64)
    wl = bench.Workload("atari_flexible", "cuda:0", n=300)
    frames = [f.cpu().numpy()[idx] for f in wl.frames]
    acts, atypes = [a.cpu().numpy()[idx] for a in wl.actions], [t.cpu().numpy()[idx] for t in wl.atypes]
    wl.free()
    m, fov, W, S = len(idx), (30, 30), 3, 3   # --warmup 1 runs as 3
    ring, head = orc.new_state(m, 4, bench.S)
    loc, res = np.zeros((m, 2), np.int32), np.tile(np.array([fov], np.int32), (m, 1))
    orc.ingest_atari(frames[0], frames[1], np.full(m, 5, np.uint8), ring, head)
    t0 = W + S + W
    for t in list(range(t0)) + 2 * list(range(t0, t0 + S)):
        k = (2 * t) % len(frames)
        orc.ingest_atari(frames[k], frames[k + 1], np.full(m, 3, np.uint8), ring, head)
        orc.update_loc(acts[t % 4], loc, obs_size=bench.S, fov_size=fov, relative=False, lo=-10.0, hi=10.0, atype=atypes[t % 4],
                       res=res)
    assert np.array_equal(d["fov_loc"], loc) and np.array_equal(d["fov_res"], res)
    assert np.abs(d["obs"] - orc.observe_flexible(ring, head, loc, res, fov, variant="mask")).max() <= 0.5 + 1e-2


def test_traffic_capture_is_tied_to_the_code_it_was_measured_on():
    """roofline.traffic comes from profiles/traffic.json only while the code of the workload's kernels is what the ncu
    capture ran: the hash ignores comments and blank lines, covers the workload's own translation units plus the shared
    headers / launcher, and the committed captures match the committed sources."""
    sys.path.insert(0, ROOT)
    import bench
    a = "int x = 1; // note\n\n  /* block\n comment */ const char *s = \"a//b\";  // tail\n"
    assert bench._code_only(a) == 'int x = 1;\nconst char *s = "a//b";'
    assert bench._code_only(a) == bench._code_only("int x = 1;\n  const char *s = \"a//b\";")
    assert bench._code_only("int x = 2;") != bench._code_only("int x = 1;")
    # a workload's hash covers only the translation units its kernels come from
    assert bench.sources_hash("atari_fixed") == bench.sources_hash("dmc_fixed")           # same two TUs
    assert bench.sources_hash("atari_flexible") != bench.sources_hash("atari_peripheral")
    assert set(bench._KERNEL_TUS) == set(bench.WORKLOADS)
    with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
        tj = json.load(f)
    import warnings
    for w, sha in tj["sources_sha16"].items():
        assert w in bench.WORKLOADS and tj["workloads"][w], w
        if sha != bench.sources_hash(w):   # legitimate (bench.py then prints traffic = null), but worth a line in the test log
            warnings.warn(f"profiles/traffic.json: the capture of {w} is stale (re-run tools/ncu_summary.py on a fresh ncu report)")
