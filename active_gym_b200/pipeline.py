"""``PipelinedPath``: the observation path of one GPU cut into env-index shards, each with its own CUDA
stream, so that the host->device copy of shard i+1 overlaps the kernels and the device->host copy of shard i
(the two copy engines run in both directions at once).  Shards are independent — the same property that lets
the batch shard over GPUs with no collective (SURVEY.md §8e).

It presents the surface of ``ObservationPath`` (``ingest_*``, ``observe_*``, ``stack``, ``ring`` / ``head`` /
``loc`` / ``res`` / ``pcache`` as ONE tensor each), so the env classes drive either.  Inputs may live on the
device (no copy: the shard kernels read slices of the caller's tensors) or on the host (pinned memory is copied
asynchronously on the shard's stream; for Atari frames only the raw rows the resize samples cross PCIe).

Ordering: every call first makes the shard streams wait for the caller's current stream, and ``join()`` makes
the current stream wait for the shards — device-side event waits, no host synchronisation.  ``sync()`` blocks
the host until the shards are idle (needed before reading pinned outputs).
"""
from __future__ import annotations

import collections
from typing import List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib
from .engine import LUMA_RGB, ObservationPath
from .sharding import all_shards

_cudart = None


def _rt():
    """libcudart through ctypes, for the strided (row-skipping) pinned copies torch has no call for."""
    global _cudart
    if _cudart is None:
        import ctypes as C
        last = None
        for name in ("libcudart.so.12", "libcudart.so"):
            try:
                _cudart = C.CDLL(name)
                break
            except OSError as ex:
                last = ex
        if _cudart is None:
            raise RuntimeError(f"libcudart not found: {last}")
        vp, sz = C.c_void_p, C.c_size_t
        _cudart.cudaMemcpy2DAsync.argtypes = [vp, sz, vp, sz, sz, sz, C.c_int, vp]
        _cudart.cudaMemcpyAsync.argtypes = [vp, vp, sz, C.c_int, vp]
        _cudart.cudaDeviceEnablePeerAccess.argtypes = [C.c_int, C.c_uint]
    return _cudart


def periodic_run(used: np.ndarray, n_rows: int):
    """If the sampled rows repeat with a period P that divides n_rows and form ONE cyclic run of L rows
    starting at offset o inside a period, returns (P, o, L); else None.  (210 -> 84: every row except
    g % 5 == 2, i.e. P = 5, o = 3, L = 4.)"""
    mask = np.zeros(n_rows, bool)
    mask[used] = True
    for P in range(1, n_rows + 1):
        if n_rows % P or not np.array_equal(mask, np.tile(mask[:P], n_rows // P)):
            continue
        m = mask[:P]
        if m.all():
            return None  # nothing to skip
        starts = [i for i in range(P) if m[i] and not m[i - 1]]
        if len(starts) != 1:
            return None
        return P, starts[0], int(m.sum())
    return None


def _as_u8(v):
    """bool / integer per-env flags as uint8 (host arrays stay on the host, device tensors on the device)."""
    if isinstance(v, torch.Tensor):
        return v if v.dtype == torch.uint8 else v.to(torch.uint8)
    return np.asarray(v).astype(np.uint8, copy=False)


def _pin(shape, dtype) -> torch.Tensor:
    return torch.empty(shape, dtype=dtype).pin_memory()


class PipelinedPath:
    """``n_envs`` environments on one device as ``shards`` independent ``ObservationPath`` slices."""

    def __init__(self, n_envs: int, frame_stack: int, obs_size, raw_shape, shards: int = 1, device=None,
                 luma: Sequence[int] = LUMA_RGB, fov_size=None, fov_init_loc=(0, 0), sensory_action_mode: str = "absolute",
                 sensory_action_space=(0.0, 0.0), peripheral_res=None, cache_peripheral: bool = True,
                 packed_h2d: bool = True, side_streams: bool = False, antialias: bool = True, channels: int = 1,
                 fov_memory: int = 0):
        if not torch.cuda.is_available():
            raise RuntimeError("active_gym_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.n_envs, self.frame_stack = int(n_envs), int(frame_stack)
        self.obs_size = (int(obs_size[0]), int(obs_size[1]))
        self.raw_shape = tuple(int(v) for v in raw_shape)
        self.fov_size = None if fov_size is None else (int(fov_size[0]), int(fov_size[1]))
        self.peripheral_res = None if peripheral_res is None else (int(peripheral_res[0]), int(peripheral_res[1]))
        self.relative = sensory_action_mode == "relative"
        self.channels = int(channels)
        # K: ring planes per env (frame_stack * channels, see ObservationPath)
        N, K, (S_h, S_w), dev = self.n_envs, self.frame_stack * self.channels, self.obs_size, self.device
        shards = max(1, min(int(shards), N))
        self.ranges: List[Tuple[int, int]] = [r for r in all_shards(N, shards) if r[1] > r[0]]
        with torch.cuda.device(dev):
            self.ring = torch.zeros((N, K, S_h, S_w), dtype=torch.uint8, device=dev)
            self.head = torch.full((N,), K - 1, dtype=torch.int32, device=dev)
            self.loc = torch.zeros((N, 2), dtype=torch.int32, device=dev)
            self.res = torch.zeros((N, 2), dtype=torch.int32, device=dev)
            if self.fov_size:
                self.res[:, 0], self.res[:, 1] = self.fov_size
            self.pcache = None
            if self.peripheral_res and cache_peripheral:
                self.pcache = torch.zeros((N, K) + self.peripheral_res, dtype=torch.float32, device=dev)
            self.err = torch.zeros((1,), dtype=torch.int32, device=dev)
            # the fixed fovea's memory (ObservationPath.observe_fixed_memory): one allocation, sliced per shard
            if not 0 <= int(fov_memory) <= 16:
                raise ValueError(f"fov_memory must be within 0..16, got {fov_memory!r}")
            self.fov_memory = int(fov_memory)
            self.mem = self.mem_loc = self.mem_state = None
            if self.fov_memory:
                if self.fov_size is None:
                    raise ValueError("fov_memory needs a fovea (fov_size)")
                M, E = self.fov_memory, (K * self.fov_size[0] * self.fov_size[1] + 15) // 16 * 16
                self.mem = torch.zeros((N, M, E), dtype=torch.uint8, device=dev)
                self.mem_loc = torch.zeros((N, M, 2), dtype=torch.int32, device=dev)
                self.mem_state = torch.zeros((N, 2), dtype=torch.int32, device=dev)
            mem = (lambda lo, hi: dict(mem=self.mem[lo:hi], mem_loc=self.mem_loc[lo:hi], mem_state=self.mem_state[lo:hi])) \
                if self.fov_memory else (lambda lo, hi: {})
            # RecordWrapper's episode counters (fov_env.py:20-21) live with the rest of the per-env state
            self.ep_len = torch.zeros((N,), dtype=torch.int64, device=dev)
            self.cum_reward = torch.zeros((N,), dtype=torch.float64, device=dev)
            self.paths = [
                ObservationPath(hi - lo, self.frame_stack, self.obs_size, self.raw_shape, luma=luma, fov_size=fov_size,
                                fov_init_loc=fov_init_loc, sensory_action_mode=sensory_action_mode,
                                sensory_action_space=sensory_action_space, peripheral_res=peripheral_res, device=dev,
                                cache_peripheral=cache_peripheral, antialias=antialias, channels=self.channels,
                                fov_memory=self.fov_memory,
                                buffers=dict(ring=self.ring[lo:hi], head=self.head[lo:hi], loc=self.loc[lo:hi],
                                             res=self.res[lo:hi], pcache=None if self.pcache is None else self.pcache[lo:hi],
                                             err=self.err, **mem(lo, hi)))
                for lo, hi in self.ranges]
            # one shard: work is issued on the caller's stream (unless `side_streams`: a host-driven env group keeps its
            # own stream so that two groups overlap each other's copies); several: one side stream each
            self.streams = [torch.cuda.Stream(device=dev) for _ in self.ranges] if (len(self.ranges) > 1 or side_streams) else None
            self._fork_ev = torch.cuda.Event()
            self._join_evs = [torch.cuda.Event() for _ in self.ranges]
        rh, rw, rc = self.raw_shape
        self.row_bytes = rw * rc
        self.run = periodic_run(self.used_rows, rh) if (packed_h2d and rh != S_h) else None
        # staging, allocated on first use: device copies of host inputs, pinned copies of small host arrays
        self._d_frames = {}
        self._d_small = {}
        self._h_out = {}
        self._stage = {}        # key -> [use counter, [pinned buffer A, B], [events of the copies that last read A, B]]
        self._keep = collections.deque(maxlen=16)   # device-side conversion temporaries the shard streams may still read
        self._d_out = {}
        self._h_err, self._err_ev = None, None
        self._pre = {}          # key -> (the caller's object, per-shard device slices): small arrays uploaded ahead of the frames
        self.h2d_bytes = 0  # bytes copied host -> device / device -> host since the last reset_counters()
        self.d2h_bytes = 0
        torch.cuda.synchronize(dev)  # the fills above ran on the current stream; shard streams start after them

    # ------------------------------------------------------------------ plumbing
    @property
    def used_rows(self) -> np.ndarray:
        return self.paths[0].used_rows

    def raw_frame_shape(self) -> Tuple[int, ...]:
        h, w, c = self.raw_shape
        return (self.n_envs, h, w) if c == 1 else (self.n_envs, h, w, 3)

    def out_shape(self, kind: str, variant: str, pad=None) -> Tuple[int, ...]:
        return (self.n_envs,) + tuple(self.paths[0].out_shape(kind, variant, pad)[1:])

    @property
    def stack_shape(self) -> Tuple[int, ...]:
        return (self.n_envs,) + tuple(self.paths[0].stack_shape[1:])

    def reset_counters(self) -> None:
        self.h2d_bytes = self.d2h_bytes = 0

    def _fork(self) -> None:
        """Shard streams wait for what the caller has enqueued so far (device tensors it produced)."""
        if self.streams is None:
            return
        cur = torch.cuda.current_stream(self.device)
        self._fork_ev.record(cur)
        for s in self.streams:
            s.wait_event(self._fork_ev)

    def join(self) -> None:
        """The caller's stream waits for every shard (device-side; the host does not block)."""
        if self.streams is None:
            return
        cur = torch.cuda.current_stream(self.device)
        for s, ev in zip(self.streams, self._join_evs):
            ev.record(s)
            cur.wait_event(ev)

    def record_events(self) -> list:
        """One event per shard stream, recorded now: they complete when everything enqueued so far has run."""
        cur = torch.cuda.current_stream(self.device)
        evs = []
        for i in range(len(self.ranges)):
            e = torch.cuda.Event()
            e.record(cur if self.streams is None else self.streams[i])
            evs.append(e)
            if self.streams is None:
                break
        return evs

    def sync(self) -> None:
        """Blocks the host until every shard stream is idle."""
        if self.streams is None:
            torch.cuda.current_stream(self.device).synchronize()
        else:
            for s in self.streams:
                s.synchronize()

    def _shards(self):
        for i, (lo, hi) in enumerate(self.ranges):
            if self.streams is None:
                yield i, lo, hi
            else:
                with torch.cuda.stream(self.streams[i]):
                    yield i, lo, hi

    def _small_to_device(self, key: str, value, dtype: torch.dtype, width: Optional[int]) -> Optional[List[torch.Tensor]]:
        """(N,) / (N, width) per-env array -> one contiguous device slice per shard.  Device tensors are sliced in
        place; host arrays go through pinned staging + an async copy on the shard's stream.  The pinned staging of
        every key is double buffered with its own events: a buffer is rewritten only after the copies that read it
        two uses ago have completed — in a running pipeline they always have, so the host never blocks here."""
        if value is None:
            return None
        shape = (self.n_envs,) if width is None else (self.n_envs, width)
        if isinstance(value, torch.Tensor) and value.device.type == "cuda":
            t = value.detach().reshape(shape)
            if t.dtype != dtype or not t.is_contiguous():
                t = t.to(dtype).contiguous()
            self._keep.append(t)  # possibly a temporary made on the caller's stream, read on the shard streams
            return [t[lo:hi] for lo, hi in self.ranges]
        st = self._stage.get(key)
        if st is None:
            st = self._stage[key] = [0, [_pin(shape, dtype), _pin(shape, dtype)], [None, None]]
            self._d_small[key] = torch.empty(shape, dtype=dtype, device=self.device)
        st[0] ^= 1
        which = st[0]
        h, evs = st[1][which], st[2][which]
        if evs is not None:
            for e in evs:
                e.synchronize()
        else:
            evs = st[2][which] = [torch.cuda.Event() for _ in self.ranges]
        src = value.detach().cpu().numpy() if isinstance(value, torch.Tensor) else np.asarray(value)
        h.numpy()[...] = src.reshape(shape)
        d = self._d_small[key]
        out = []
        for i, lo, hi in self._shards():
            d[lo:hi].copy_(h[lo:hi], non_blocking=True)
            evs[i].record(torch.cuda.current_stream(self.device))
            out.append(d[lo:hi])
        self.h2d_bytes += h.numel() * h.element_size()
        return out

    _PRE = {"act": (torch.float64, 2), "atype": (torch.int32, None), "raw_reward": (torch.float64, None), "done": (torch.uint8, None)}

    def prestage(self, action=None, action_type=None, raw_reward=None, done=None) -> None:
        """Uploads the step's small per-env HOST arrays now — before the frames are enqueued.  Copies of one direction
        are served in issue order, so an action array enqueued after 55 MB of frames per shard would hold back the
        observe launch (and the copies back) of EVERY shard until the last frame byte has crossed the link.  The later
        ``observe_*`` / ``record_step`` call finds the device copy by the identity of the object passed here."""
        vals = {"act": action, "atype": action_type, "raw_reward": raw_reward, "done": done}
        vals = {k: v for k, v in vals.items() if v is not None and not (isinstance(v, torch.Tensor) and v.device.type == "cuda")}
        if not vals:
            return
        self._fork()
        for k, v in vals.items():
            dt, width = self._PRE[k]
            src = _as_u8(v) if k == "done" else v
            self._pre[k] = (v, self._small_to_device(k, src, dt, width))

    def _small(self, key: str, value, dtype: torch.dtype, width: Optional[int]):
        """`_small_to_device`, unless `value` is the object `prestage` already uploaded for this step."""
        pre = self._pre.pop(key, None)
        if pre is not None and pre[0] is value:
            return pre[1]
        if key == "done" and value is not None:
            value = _as_u8(value)
        return self._small_to_device(key, value, dtype, width)

    def _h2d_rows(self, dst: torch.Tensor, src: torch.Tensor, lo: int, hi: int) -> None:
        """Rows g of envs [lo, hi) of full host frames with (g % P) inside the cyclic run [o, o + L) -> dst, in row order."""
        P, o, L = self.run
        rb, rt = self.row_bytes, _rt()
        stream = torch.cuda.current_stream(self.device).cuda_stream
        raw_h = self.raw_shape[0]
        periods = (hi - lo) * (raw_h // P)
        s0 = src.data_ptr() + lo * raw_h * rb
        d0 = dst.data_ptr()
        wrap = max(o + L - P, 0)
        H2D = 1
        if wrap == 0:
            err = rt.cudaMemcpy2DAsync(d0, L * rb, s0 + o * rb, P * rb, L * rb, periods, H2D, stream)
        else:
            err = rt.cudaMemcpyAsync(d0, s0, wrap * rb, H2D, stream)                       # rows 0 .. wrap-1 of the first period
            if not err and periods > 1:
                err = rt.cudaMemcpy2DAsync(d0 + wrap * rb, L * rb, s0 + o * rb, P * rb, L * rb, periods - 1, H2D, stream)
            if not err:                                                                     # rows o .. P-1 of the last period
                tail = (P - o) * rb
                err = rt.cudaMemcpyAsync(d0 + wrap * rb + (periods - 1) * L * rb, s0 + ((periods - 1) * P + o) * rb, tail, H2D, stream)
        if err:
            raise RuntimeError(f"packed H2D copy failed: cudaError {err}")

    def _frames_plan(self, key: str, frames, packed: bool):
        """Validates raw frames and returns a per-shard copier: ``stage(i, lo, hi) -> (device tensor, is_packed)``, to be
        called on shard i's stream.  Device frames are sliced; host frames are copied into a per-key staging tensor
        (only the sampled rows when the source already packs them or the rows are periodic)."""
        h, w, c = self.raw_shape
        t = torch.as_tensor(frames)
        if c == 1 and t.dim() == 4 and t.shape[-1] == 1:
            t = t[..., 0]  # ALE's getScreenGrayscale() is (210,160,1)
        nu = len(self.used_rows)
        rows = nu if packed else h
        want = (self.n_envs, rows, w) if c == 1 else (self.n_envs, rows, w, c)
        if tuple(t.shape) != want:
            raise ValueError(f"expected frames of shape {want}, got {tuple(t.shape)}")
        if t.dtype != torch.uint8:
            raise TypeError(f"expected uint8 frames, got {t.dtype}")
        t = t.contiguous()
        if t.device.type == "cuda":
            return lambda i, lo, hi: (t[lo:hi], packed)
        strided = (not packed) and self.run is not None and t.is_pinned()
        dev_packed = packed or strided
        dshape = (self.n_envs, nu if dev_packed else h) + want[2:]
        dk = (key, dev_packed)
        if dk not in self._d_frames:
            self._d_frames[dk] = torch.empty(dshape, dtype=torch.uint8, device=self.device)
        d = self._d_frames[dk]
        self.h2d_bytes += d.numel()

        def stage(i, lo, hi):
            if strided:
                self._h2d_rows(d[lo:hi], t, lo, hi)
            else:
                d[lo:hi].copy_(t[lo:hi], non_blocking=True)
            return d[lo:hi], dev_packed
        return stage

    # ------------------------------------------------------------------ ingest
    def ingest_atari(self, frames_a, frames_b, flags, packed: bool = False) -> None:
        """AtariEnv._get_state + frame logic of _step/_reset (atari_env.py:73-75, 121-133) on every shard.
        ``packed``: the frames hold only ``used_rows`` (N, 168, 160[, 3])."""
        self._fork()
        fa = self._frames_plan("fa", frames_a, packed)
        fb = None if frames_b is frames_a else self._frames_plan("fb", frames_b, packed)
        fl = self._small_to_device("flags", flags, torch.uint8, None)
        # shard by shard: both frames of shard i cross the link before any byte of shard i + 1, so shard i's kernels
        # and its copies back start while the later shards are still uploading
        for i, lo, hi in self._shards():
            a, pk = fa(i, lo, hi)
            b = a if fb is None else fb(i, lo, hi)[0]
            (self.paths[i].ingest_atari_packed if pk else self.paths[i].ingest_atari)(a, b, fl[i])

    def ingest_atari_packed(self, rows_a, rows_b, flags) -> None:
        self.ingest_atari(rows_a, rows_b, flags, packed=True)

    def ingest_dmc(self, frames, flags) -> None:
        """DMCEnv._get_obs (pixel, grey) + stack logic (dmc_env.py:175-183, 228-230) on every shard."""
        self._fork()
        f = self._frames_plan("f", frames, False)
        fl = self._small_to_device("flags", flags, torch.uint8, None)
        for i, lo, hi in self._shards():
            self.paths[i].ingest_dmc(f(i, lo, hi)[0], fl[i])

    # ------------------------------------------------------------------ outputs
    def stack(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        if out is None:
            out = torch.empty_like(self.ring)
        self._fork()
        for i, lo, hi in self._shards():
            self.paths[i].stack(out=out[lo:hi])
        self.join()
        return out.view(self.stack_shape)

    def _observe(self, kind: str, action, action_type, variant: str, ctrl, pad, out, host_out: bool, norm_out=None,
                 background=None):
        shape = self.out_shape(kind, variant, pad)
        if norm_out is not None and tuple(norm_out.shape) != tuple(shape):
            raise ValueError(f"norm_out must have the observation's shape {tuple(shape)}")
        if out is None and host_out:   # shard streams keep writing it after this call returns: never hand it to the allocator
            ok = (kind, variant, tuple(shape))
            if ok not in self._d_out:
                self._d_out[ok] = torch.empty(shape, dtype=torch.uint8, device=self.device)
            out = self._d_out[ok]
        elif out is None:
            out = torch.empty(shape, dtype=torch.uint8, device=self.device)
        self._fork()
        act = self._small("act", action, torch.float64, 2)
        at = self._small("atype", action_type, torch.int32, None)
        if isinstance(ctrl, str):
            assert ctrl == "reset"
            ct = ["reset"] * len(self.ranges)
        else:
            ct = self._small_to_device("ctrl", ctrl, torch.uint8, None)
        h_obs = h_loc = None
        flex = kind in ("flexible", "flexible_peripheral")   # fov_res travels with the observation
        if host_out:
            hk = (kind, variant, tuple(shape))
            if hk not in self._h_out:
                self._h_out[hk] = (_pin(shape, torch.uint8), _pin((self.n_envs, 2), torch.int32), _pin((self.n_envs, 2), torch.int32))
            h_obs, h_loc, h_res = self._h_out[hk]
        for i, lo, hi in self._shards():
            p, a = self.paths[i], None if act is None else act[i]
            c = None if ct is None else ct[i]
            nrm = None if norm_out is None else norm_out[lo:hi]
            if kind == "peripheral":
                p.observe_peripheral(a, ctrl=c, out=out[lo:hi], norm_out=nrm)
            elif kind == "flexible":
                p.observe_flexible(a, None if at is None else at[i], variant=variant, ctrl=c, pad=pad, out=out[lo:hi], norm_out=nrm)
            elif kind == "flexible_peripheral":
                p.observe_flexible_peripheral(a, None if at is None else at[i], ctrl=c, out=out[lo:hi], norm_out=nrm)
            elif kind == "fixed_memory":
                p.observe_fixed_memory(a, ctrl=c, out=out[lo:hi], norm_out=nrm)
            elif kind == "memory_paste":
                p.observe_memory_paste(a, ctrl=c, background=background, out=out[lo:hi], norm_out=nrm)
            else:
                p.observe_fixed(a, variant=variant, ctrl=c, out=out[lo:hi], norm_out=nrm)
            if host_out:
                h_obs[lo:hi].copy_(out[lo:hi], non_blocking=True)
                h_loc[lo:hi].copy_(self.loc[lo:hi], non_blocking=True)
                if flex:
                    h_res[lo:hi].copy_(self.res[lo:hi], non_blocking=True)
        if host_out:
            self.d2h_bytes += h_obs.numel() + h_loc.numel() * 4 * (2 if flex else 1)
            return out, (h_obs, h_loc, h_res if flex else None)
        self.join()
        return out

    def observe_fixed(self, action, variant: str = "crop", ctrl=None, out=None, host_out: bool = False, norm_out=None):
        """FixedFovealEnv._fov_step + _get_fov_state (fov_env.py:166-203).  ``host_out``: also copy the
        observations and fov_loc to pinned host memory on the shard streams; returns (out, (h_obs, h_loc, None)),
        valid after ``sync()``."""
        return self._observe("fixed", action, None, variant, ctrl, None, out, host_out, norm_out)

    def observe_fixed_memory(self, action, ctrl=None, out=None, host_out: bool = False, norm_out=None):
        """The fixed fovea's memory (ObservationPath.observe_fixed_memory) on every shard; ``host_out`` as for
        ``observe_fixed``."""
        if not self.fov_memory:
            raise ValueError("observe_fixed_memory needs a path built with fov_memory > 0")
        return self._observe("fixed_memory", action, None, "mask", ctrl, None, out, host_out, norm_out)

    def observe_memory_paste(self, action, ctrl=None, background: str = "zero", out=None, host_out: bool = False,
                             norm_out=None):
        """The fixed fovea's memory merged by pasting (ObservationPath.observe_memory_paste) on every shard;
        ``host_out`` as for ``observe_fixed``."""
        if not self.fov_memory:
            raise ValueError("observe_memory_paste needs a path built with fov_memory > 0")
        if background == "periphery" and self.pcache is None:
            raise ValueError("the periphery background needs the squeeze cache: build with cache_peripheral=True")
        return self._observe("memory_paste", action, None, "mask", ctrl, None, out, host_out, norm_out, background=background)

    def observe_peripheral(self, action, ctrl=None, out=None, use_cache: bool = True, host_out: bool = False, norm_out=None):
        """FixedFovealPeripheralEnv._get_fov_state (fov_env.py:375-388), loc update fused."""
        if not use_cache:
            raise ValueError("the sharded path always uses the cached squeeze (build with cache_peripheral=False to drop it)")
        return self._observe("peripheral", action, None, "mask", ctrl, None, out, host_out, norm_out)

    def observe_flexible(self, action, action_type=None, variant: str = "mask", ctrl=None, pad=None, out=None,
                         host_out: bool = False, norm_out=None):
        """FlexibleFovealEnv._fov_step + _get_fov_state (fov_env.py:270-330)."""
        pad = tuple(pad) if pad is not None else self.obs_size
        return self._observe("flexible", action, action_type, variant, ctrl, pad, out, host_out, norm_out)

    def observe_flexible_peripheral(self, action, action_type=None, ctrl=None, out=None, host_out: bool = False,
                                    norm_out=None):
        """The flexible fovea over the peripheral background (ObservationPath.observe_flexible_peripheral)."""
        if self.pcache is None:
            raise ValueError("observe_flexible_peripheral needs the squeeze cache: build with cache_peripheral=True")
        return self._observe("flexible_peripheral", action, action_type, "mask", ctrl, None, out, host_out, norm_out)

    def record_step(self, raw_reward=None, done=None, reset_mask=None, is_reset: bool = False,
                    trace_row: Optional[torch.Tensor] = None, with_res: bool = False, host_out: bool = False):
        """RecordWrapper's counters + fov trace (fov_env.py:15-67, 152-154, 205-207) on every shard's stream, after
        the observe call that produced ``loc`` / ``res``.  ``raw_reward`` (N,) float, ``done`` / ``reset_mask`` (N,) bool,
        host or device.  ``host_out``: returns pinned (ep_len, cum_reward), valid after ``sync()``."""
        self._fork()
        rr = self._small("raw_reward", raw_reward, torch.float64, None)
        dn = self._small("done", done, torch.uint8, None)
        rm = self._small_to_device("reset_mask", None if reset_mask is None else _as_u8(reset_mask), torch.uint8, None)
        h = None
        if host_out:
            if "counters" not in self._h_out:
                self._h_out["counters"] = (_pin((self.n_envs,), torch.int64), _pin((self.n_envs,), torch.float64))
            h = self._h_out["counters"]
        for i, lo, hi in self._shards():
            self.paths[i].record_step(self.ep_len[lo:hi], self.cum_reward[lo:hi], None if rr is None else rr[i],
                                      None if dn is None else dn[i], None if rm is None else rm[i], is_reset,
                                      None if trace_row is None else trace_row[lo:hi], with_res)
            if host_out:
                h[0][lo:hi].copy_(self.ep_len[lo:hi], non_blocking=True)
                h[1][lo:hi].copy_(self.cum_reward[lo:hi], non_blocking=True)
        if host_out:
            self.d2h_bytes += 16 * self.n_envs
            return h
        self.join()
        return None

    def normalize(self, obs: torch.Tensor, dtype: torch.dtype = torch.float32, out=None) -> torch.Tensor:
        return self.paths[0].normalize(obs, dtype, out)

    def synth_frames(self, out: torch.Tensor, seed: int) -> torch.Tensor:
        return self.paths[0].synth_frames(out, seed)

    def read_errors(self) -> int:
        """Device error word (``_lib.ERR_RES_*`` bits), read now: blocks until the device has caught up.  Cleared
        when non-zero."""
        self.join()
        v = int(self.err.item())
        if v:
            self.err.zero_()
        return v

    def poll_errors(self) -> int:
        """Non-blocking variant: returns the value an asynchronous copy enqueued by an EARLIER call has delivered
        (0 while none has completed) and enqueues the next copy behind the work issued so far."""
        v = 0
        if self._err_ev is not None and self._err_ev.query():
            v = int(self._h_err[0])
            self._err_ev = None
            if v:
                self.err.zero_()   # bits set between that copy and this clear are dropped: the caller raises anyway
        if self._err_ev is None:
            if self._h_err is None:
                self._h_err = _pin((1,), torch.int32)
            self.join()
            self._h_err.copy_(self.err, non_blocking=True)
            self._err_ev = torch.cuda.Event()
            self._err_ev.record(torch.cuda.current_stream(self.device))
        return v
