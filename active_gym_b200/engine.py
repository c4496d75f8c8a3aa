"""Host side of the observation path for one GPU: owns the HBM-resident state of a batch of
environments (frame-stack ring, fovea location / resolution, peripheral cache) as torch
tensors and issues the sm_100a kernels through the C ABI (``include/agym_b200.h``).

PyTorch is used here for device memory and streams only; all arithmetic is in
``csrc/agym_{ingest,observe,flexible,misc}.cu``.  There is no CPU fallback.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib

# cv2's 15-bit luma weights by channel position.  LUMA_RGB is the declared stand-in for ALE's
# palette grayscale when frames arrive as RGB; LUMA_DMC reproduces dmc_env.py:182, which applies
# COLOR_BGR2GRAY to an RGB render (channel 0 gets the blue weight).
LUMA_RGB = (9798, 19235, 3735)
LUMA_DMC = (3735, 19235, 9798)

VARIANTS = {"crop": _lib.OUT_CROP, "mask": _lib.OUT_MASK, "resize_full": _lib.OUT_RESIZE_FULL,
            "resize_fov": _lib.OUT_RESIZE_FOV}


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


class ObservationPath:
    """Ring + fovea state of ``n_envs`` environments on one device and the kernels over it.

    Parameters mirror the attributes the reference wrappers read from ``AtariEnvArgs`` /
    ``DMCEnvArgs`` (atari_env.py:25-39, dmc_env.py:56-76, fov_env.py:110-122, 244, 365).
    """

    def __init__(self, n_envs: int, frame_stack: int, obs_size: Tuple[int, int], raw_shape: Tuple[int, int, int],
                 luma: Sequence[int] = LUMA_RGB, fov_size: Optional[Tuple[int, int]] = None,
                 fov_init_loc: Sequence[float] = (0, 0), sensory_action_mode: str = "absolute",
                 sensory_action_space: Sequence[float] = (0.0, 0.0), peripheral_res: Optional[Tuple[int, int]] = None,
                 device: Optional[torch.device] = None, cache_peripheral: bool = True, buffers: Optional[dict] = None,
                 antialias: bool = True, channels: int = 1, fov_memory: int = 0):
        """``channels``: planes per frame — 1 (grey, the luma of the frames) or 3 (RGB: the channels of DMC renders,
        which must have ``raw_shape == obs_size + (3,)``).  The ring then holds ``frame_stack * channels`` planes
        (``include/agym_b200.h``) and every observation gains a channel axis, ``(N, K, C, h, w)``.

        ``antialias``: how the wrappers' ``torchvision.transforms.Resize`` calls (fov_env.py:120, 248, 366-368) are
        restated — antialiased bilinear (the installed torchvision's default, what the fixtures were recorded with) or
        plain bilinear (the default of older torchvision releases on tensors; SURVEY.md section 8c).

        ``fov_memory``: depth M (1..16) of the fixed fovea's memory (``observe_fixed_memory``), 0 = none.  The path then
        holds ``mem`` u8 (N, M, E), ``mem_loc`` i32 (N, M, 2) and ``mem_state`` i32 (N, 2), zero = empty
        (``agym_observe_fixed_memory``), or takes them from ``buffers``."""
        if not torch.cuda.is_available():
            raise RuntimeError("active_gym_b200 needs a CUDA device (B200, sm_100a); there is no CPU fallback")
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.n_envs, self.frame_stack = int(n_envs), int(frame_stack)
        self.obs_size = (int(obs_size[0]), int(obs_size[1]))
        self.raw_shape = tuple(int(v) for v in raw_shape)
        self.fov_size = None if fov_size is None else (int(fov_size[0]), int(fov_size[1]))
        self.peripheral_res = None if peripheral_res is None else (int(peripheral_res[0]), int(peripheral_res[1]))
        if sensory_action_mode not in ("absolute", "relative"):
            raise ValueError(f"sensory_action_mode must be 'absolute' or 'relative', got {sensory_action_mode!r}")
        self.relative = sensory_action_mode == "relative"
        if channels not in (1, 3):
            raise ValueError(f"channels must be 1 (grey) or 3 (RGB), got {channels!r}")
        self.channels = int(channels)
        if not 0 <= int(fov_memory) <= 16:
            raise ValueError(f"fov_memory must be within 0..16, got {fov_memory!r}")
        if fov_memory and self.fov_size is None:
            raise ValueError("fov_memory needs a fovea (fov_size)")
        self.fov_memory = int(fov_memory)
        cfg = _lib.Config()
        cfg.n_envs, cfg.frame_stack = self.n_envs, self.frame_stack
        cfg.obs_h, cfg.obs_w = self.obs_size
        cfg.raw_h, cfg.raw_w, cfg.raw_c = self.raw_shape
        cfg.luma_w[:] = [int(v) for v in luma]
        if self.fov_size:
            cfg.fov_h, cfg.fov_w = self.fov_size
        if self.peripheral_res:
            cfg.periph_h, cfg.periph_w = self.peripheral_res
        cfg.relative = int(self.relative)
        lo, hi = (float(sensory_action_space[0]), float(sensory_action_space[1])) if self.relative else (0.0, 0.0)
        cfg.act_lo, cfg.act_hi = lo, hi
        cfg.fov_init_loc[:] = [float(fov_init_loc[0]), float(fov_init_loc[1])]
        cfg.no_antialias = 0 if antialias else 1
        cfg.obs_c = self.channels
        self.antialias = bool(antialias)
        self._cfg = cfg
        self._L = _lib.lib()
        self._plan = C.c_void_p()
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_plan_create(C.byref(cfg), C.byref(self._plan)), "agym_plan_create")
        N, K, (S_h, S_w) = self.n_envs, self.frame_stack * self.channels, self.obs_size   # K: ring planes
        dev = self.device
        if buffers is not None:
            # slices of a larger batch owned by the caller (PipelinedPath): contiguous, already initialised
            self.ring, self.head, self.loc, self.res = buffers["ring"], buffers["head"], buffers["loc"], buffers["res"]
            self.pcache, self.err = buffers.get("pcache"), buffers.get("err")
            for t, shape in ((self.ring, (N, K, S_h, S_w)), (self.head, (N,)), (self.loc, (N, 2)), (self.res, (N, 2))):
                if tuple(t.shape) != shape or not t.is_contiguous() or t.device != dev:
                    raise ValueError("buffers must be contiguous device tensors of this path's shapes")
            if self.err is None:
                self.err = torch.zeros((1,), dtype=torch.int32, device=dev)
        else:
            self.ring = torch.zeros((N, K, S_h, S_w), dtype=torch.uint8, device=dev)
            self.head = torch.full((N,), K - 1, dtype=torch.int32, device=dev)
            self.loc = torch.zeros((N, 2), dtype=torch.int32, device=dev)
            self.res = torch.zeros((N, 2), dtype=torch.int32, device=dev)
            if self.fov_size:
                self.res[:, 0], self.res[:, 1] = self.fov_size
            self.pcache = None
            if self.peripheral_res and cache_peripheral:
                self.pcache = torch.zeros((N, K) + self.peripheral_res, dtype=torch.float32, device=dev)
            # device error word of the flexible fovea (AGYM_ERR_RES_*): see read_errors()
            self.err = torch.zeros((1,), dtype=torch.int32, device=dev)
        self.mem = self.mem_loc = self.mem_state = None
        if self.fov_memory:
            M = self.fov_memory
            E = self._L.agym_plan_memory_bytes(self._plan, M) // (N * M)
            if buffers is not None:
                self.mem, self.mem_loc, self.mem_state = buffers["mem"], buffers["mem_loc"], buffers["mem_state"]
                for t, shape in ((self.mem, (N, M, E)), (self.mem_loc, (N, M, 2)), (self.mem_state, (N, 2))):
                    if tuple(t.shape) != shape or not t.is_contiguous() or t.device != dev:
                        raise ValueError("buffers must be contiguous device tensors of this path's shapes")
            else:
                self.mem = torch.zeros((N, M, E), dtype=torch.uint8, device=dev)
                self.mem_loc = torch.zeros((N, M, 2), dtype=torch.int32, device=dev)
                self.mem_state = torch.zeros((N, 2), dtype=torch.int32, device=dev)
        self._ctrl_reset = torch.full((N,), _lib.FOV_RESET, dtype=torch.uint8, device=dev)

    def __del__(self):
        plan, self._plan = getattr(self, "_plan", None), None
        if plan:
            try:
                self._L.agym_plan_destroy(plan)
            except Exception:  # interpreter shutdown
                pass

    # ------------------------------------------------------------------ helpers
    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _dev_u8(self, t, shape) -> torch.Tensor:
        t = torch.as_tensor(t)
        if t.dtype != torch.uint8:
            raise TypeError(f"expected uint8, got {t.dtype}")
        if tuple(t.shape) != tuple(shape):
            raise ValueError(f"expected shape {tuple(shape)}, got {tuple(t.shape)}")
        if t.device != self.device:
            t = t.to(self.device, non_blocking=True)
        return t.contiguous()

    def _dev_action(self, action) -> torch.Tensor:
        """Any real (N,2) array / tensor -> float64 device tensor (exact for ints and float32)."""
        if isinstance(action, torch.Tensor):
            t = action.detach()
        else:
            t = torch.as_tensor(np.asarray(action))
        t = t.reshape(self.n_envs, 2)
        return t.to(device=self.device, dtype=torch.float64, non_blocking=True).contiguous()

    def _dev_atype(self, action_type) -> Optional[torch.Tensor]:
        """(N,) FOV_LOC / FOV_RES action types -> int32 device tensor (None: every env FOV_LOC)."""
        if action_type is None:
            return None
        at = torch.as_tensor(np.asarray(action_type) if not isinstance(action_type, torch.Tensor) else action_type)
        return at.reshape(self.n_envs).to(device=self.device, dtype=torch.int32, non_blocking=True).contiguous()

    def raw_frame_shape(self) -> Tuple[int, ...]:
        h, w, c = self.raw_shape
        return (self.n_envs, h, w) if c == 1 else (self.n_envs, h, w, 3)

    # ------------------------------------------------------------------ ingest
    def ingest_atari(self, frames_a, frames_b, flags) -> None:
        """AtariEnv._get_state + frame logic of _step/_reset (atari_env.py:73-75, 121-133)."""
        h, w, c = self.raw_shape
        fa = self._as_frames(frames_a, (h, w, c))
        fb = self._as_frames(frames_b, (h, w, c))
        fl = self._dev_u8(flags, (self.n_envs,))
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_ingest_atari(self._plan, _ptr(fa), _ptr(fb), _ptr(fl), _ptr(self.ring), _ptr(self.head),
                                                 _ptr(self.pcache), self._stream()), "agym_ingest_atari")

    @property
    def used_rows(self) -> np.ndarray:
        """Raw rows the resize samples, ascending (atari_env.py:74 reads two rows per output row)."""
        if getattr(self, "_used_rows", None) is None:
            n = self._L.agym_plan_used_rows(self._plan, None, 0)
            buf = (C.c_int32 * n)()
            self._L.agym_plan_used_rows(self._plan, buf, n)
            self._used_rows = np.frombuffer(buf, dtype=np.int32).copy()
        return self._used_rows

    def ingest_atari_packed(self, rows_a, rows_b, flags) -> None:
        """``ingest_atari`` on frames that carry only ``used_rows`` (shape (N, len(used_rows), raw_w[, 3])):
        a transport optimisation for host frame sources; bit-identical results."""
        h, w, c = self.raw_shape
        nu = len(self.used_rows)
        fa = self._as_frames(rows_a, (nu, w, c))
        fb = self._as_frames(rows_b, (nu, w, c))
        fl = self._dev_u8(flags, (self.n_envs,))
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_ingest_atari_packed(self._plan, _ptr(fa), _ptr(fb), _ptr(fl), _ptr(self.ring),
                                                        _ptr(self.head), _ptr(self.pcache), self._stream()),
                       "agym_ingest_atari_packed")

    def ingest_dmc(self, frames, flags) -> None:
        """DMCEnv._get_obs (pixel, grey) + stack logic (dmc_env.py:175-183, 228-230)."""
        h, w, c = self.raw_shape
        f = self._as_frames(frames, (h, w, c))
        fl = self._dev_u8(flags, (self.n_envs,))
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_ingest_dmc(self._plan, _ptr(f), _ptr(fl), _ptr(self.ring), _ptr(self.head),
                                               _ptr(self.pcache), self._stream()), "agym_ingest_dmc")

    def _as_frames(self, t, hwc) -> torch.Tensor:
        t = torch.as_tensor(t)
        h, w, c = hwc
        if c == 1 and t.dim() == 4 and t.shape[-1] == 1:
            t = t[..., 0]  # ALE's getScreenGrayscale() is (210,160,1)
        return self._dev_u8(t, (self.n_envs, h, w) if c == 1 else (self.n_envs, h, w, c))

    # ------------------------------------------------------------------ outputs
    def stack(self, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """np.stack(state_buffer), oldest -> newest (atari_env.py:143, dmc_env.py:230): (N, K, S_h, S_w), or
        (N, K, C, S_h, S_w) for RGB (a view of the plane stack the kernel writes)."""
        if out is None:
            out = torch.empty_like(self.ring)
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_stack(self._plan, _ptr(self.ring), _ptr(self.head), _ptr(out), self._stream()), "agym_stack")
        return out.view(self.stack_shape)

    @property
    def stack_shape(self) -> Tuple[int, ...]:
        return (self.n_envs,) + self._frame_axes() + self.obs_size

    def _frame_axes(self) -> Tuple[int, ...]:
        """(K,) for grey, (K, C) for RGB: the planes of the ring in observation order."""
        return (self.frame_stack,) if self.channels == 1 else (self.frame_stack, self.channels)

    def out_shape(self, kind: str, variant: str, pad: Optional[Tuple[int, int]] = None) -> Tuple[int, ...]:
        NK, S = (self.n_envs,) + self._frame_axes(), self.obs_size
        if kind in ("peripheral", "flexible_peripheral") or variant in ("mask", "resize_full"):
            return NK + S
        if kind == "flexible" and variant == "resize_fov":   # the glimpse: every window resampled to fov_size
            return NK + self.fov_size
        if kind == "flexible":
            return NK + tuple(pad if pad is not None else S)
        return NK + self.fov_size

    def _ctrl(self, ctrl) -> Optional[torch.Tensor]:
        if ctrl is None:
            return None
        if isinstance(ctrl, str):
            assert ctrl == "reset"
            return self._ctrl_reset
        return self._dev_u8(ctrl, (self.n_envs,))

    def _norm(self, out: torch.Tensor, norm_out: Optional[torch.Tensor]):
        """(pointer, AGYM_DTYPE_*) of the optional normalised second output: a contiguous f32 / f16 / bf16 tensor of
        ``out``'s shape that receives float32(u) / 255 (atari_env.py:75) in the same launch."""
        if norm_out is None:
            return None, 0
        if norm_out.shape != out.shape or norm_out.device != self.device or not norm_out.is_contiguous() \
                or norm_out.dtype not in self._NORM_DTYPES:
            raise TypeError("norm_out must be a contiguous float32 / float16 / bfloat16 tensor of the observation's shape on the path's device")
        return norm_out.data_ptr(), self._NORM_DTYPES[norm_out.dtype]

    def observe_fixed(self, action, variant: str = "crop", ctrl=None, out: Optional[torch.Tensor] = None,
                      norm_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """FixedFovealEnv._fov_step + _get_fov_state (fov_env.py:166-203).  ``norm_out``: see ``_norm``."""
        ctrl_t = self._ctrl(ctrl)
        act = None if action is None else self._dev_action(action)
        if out is None:
            out = torch.empty(self.out_shape("fixed", variant), dtype=torch.uint8, device=self.device)
        np_, nd = self._norm(out, norm_out)
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_observe_fixed(self._plan, _ptr(self.ring), _ptr(self.head), _ptr(act), _ptr(ctrl_t),
                                                  _ptr(self.loc), VARIANTS[variant], _ptr(out), np_, nd, self._stream()),
                       "agym_observe_fixed")
        return out

    def observe_fixed_memory(self, action, ctrl=None, out: Optional[torch.Tensor] = None,
                             norm_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The fixed fovea's memory (``agym_observe_fixed_memory``): the fovea update of ``observe_fixed``, a push of the
        new window unless the env's control is KEEP (RESET empties the memory first), and the pixelwise max of the
        mask_out frames of the entries held, (N, K, S_h, S_w) or (N, K, 3, S_h, S_w)."""
        if not self.fov_memory:
            raise ValueError("observe_fixed_memory needs a path built with fov_memory > 0")
        ctrl_t = self._ctrl(ctrl)
        act = None if action is None else self._dev_action(action)
        if out is None:
            out = torch.empty(self.out_shape("fixed_memory", "mask"), dtype=torch.uint8, device=self.device)
        np_, nd = self._norm(out, norm_out)
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_observe_fixed_memory(self._plan, _ptr(self.ring), _ptr(self.head), _ptr(act), _ptr(ctrl_t),
                                                         _ptr(self.loc), self.fov_memory, _ptr(self.mem), _ptr(self.mem_loc),
                                                         _ptr(self.mem_state), _ptr(out), np_, nd, self._stream()),
                       "agym_observe_fixed_memory")
        return out

    def observe_peripheral(self, action, ctrl=None, out: Optional[torch.Tensor] = None, use_cache: bool = True,
                           norm_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """FixedFovealPeripheralEnv._get_fov_state (fov_env.py:375-388), loc update fused."""
        ctrl_t = self._ctrl(ctrl)
        act = None if action is None else self._dev_action(action)
        if out is None:
            out = torch.empty(self.out_shape("peripheral", "mask"), dtype=torch.uint8, device=self.device)
        pc = self.pcache if use_cache else None
        np_, nd = self._norm(out, norm_out)
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_observe_peripheral(self._plan, _ptr(self.ring), _ptr(self.head), _ptr(pc), _ptr(act),
                                                       _ptr(ctrl_t), _ptr(self.loc), _ptr(out), np_, nd, self._stream()),
                       "agym_observe_peripheral")
        return out

    def observe_flexible(self, action, action_type=None, variant: str = "mask", ctrl=None,
                         pad: Optional[Tuple[int, int]] = None, out: Optional[torch.Tensor] = None,
                         norm_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """FlexibleFovealEnv._fov_step + _get_fov_state (fov_env.py:270-330)."""
        ctrl_t = self._ctrl(ctrl)
        act = None if action is None else self._dev_action(action)
        at = self._dev_atype(action_type)
        pad = tuple(pad) if pad is not None else self.obs_size
        if out is None:
            out = torch.empty(self.out_shape("flexible", variant, pad), dtype=torch.uint8, device=self.device)
        np_, nd = self._norm(out, norm_out)
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_observe_flexible(self._plan, _ptr(self.ring), _ptr(self.head), _ptr(act), _ptr(at),
                                                     _ptr(ctrl_t), _ptr(self.loc), _ptr(self.res), VARIANTS[variant],
                                                     int(pad[0]), int(pad[1]), _ptr(out), _ptr(self.err), np_, nd, self._stream()),
                       "agym_observe_flexible")
        return out

    def observe_flexible_peripheral(self, action, action_type=None, ctrl=None, out: Optional[torch.Tensor] = None,
                                    norm_out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """The flexible fovea over the peripheral background: FlexibleFovealEnv._fov_step (fov_env.py:300-330), then
        FixedFovealPeripheralEnv's observation (fov_env.py:366-368, 376, 385-386) with the window, blurred iff
        rh > f_h, pasted at its flexible place.  Needs the squeeze cache (``cache_peripheral=True``)."""
        if self.pcache is None:
            raise ValueError("observe_flexible_peripheral needs the squeeze cache: build the path with cache_peripheral=True")
        ctrl_t = self._ctrl(ctrl)
        act = None if action is None else self._dev_action(action)
        at = self._dev_atype(action_type)
        if out is None:
            out = torch.empty(self.out_shape("flexible_peripheral", "mask"), dtype=torch.uint8, device=self.device)
        np_, nd = self._norm(out, norm_out)
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_observe_flexible_peripheral(
                self._plan, _ptr(self.ring), _ptr(self.head), _ptr(self.pcache), _ptr(act), _ptr(at), _ptr(ctrl_t),
                _ptr(self.loc), _ptr(self.res), _ptr(out), _ptr(self.err), np_, nd, self._stream()),
                "agym_observe_flexible_peripheral")
        return out

    def read_errors(self) -> int:
        """Device error word (``_lib.ERR_RES_*`` bits: FOV_RES actions the reference would have failed on were
        clamped / truncated by a kernel).  Reading it synchronises with the device; it is cleared when non-zero."""
        v = int(self.err.item())
        if v:
            self.err.zero_()
        return v

    def record_step(self, ep_len: torch.Tensor, cum_reward: torch.Tensor, raw_reward=None, done=None, reset_mask=None,
                    is_reset: bool = False, trace_row: Optional[torch.Tensor] = None, with_res: bool = False) -> None:
        """RecordWrapper's counters and fov trace (fov_env.py:15-67, 152-154, 205-207) on the device: see
        ``agym_record_step``.  ``ep_len`` int64 (N,), ``cum_reward`` float64 (N,), updated in place."""
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_record_step(self.n_envs, int(is_reset), _ptr(raw_reward), _ptr(done), _ptr(reset_mask),
                                                _ptr(ep_len), _ptr(cum_reward), _ptr(self.loc),
                                                _ptr(self.res) if with_res else None, _ptr(trace_row), self._stream()),
                       "agym_record_step")

    _NORM_DTYPES = {torch.float32: 0, torch.float16: 1, torch.bfloat16: 2}

    def normalize(self, obs: torch.Tensor, dtype: torch.dtype = torch.float32, out: Optional[torch.Tensor] = None) -> torch.Tensor:
        """u8 observations -> the reference's normalised float32(u)/255 (atari_env.py:75, dmc_env.py:183) on the
        device; float32 is bit-identical to the reference's value, float16 / bfloat16 round it once more."""
        if obs.dtype != torch.uint8 or obs.device != self.device or not obs.is_contiguous():
            raise TypeError("normalize expects a contiguous uint8 tensor on the path's device")
        if obs.numel() % 16 != 0:
            raise ValueError("the number of pixels must be a multiple of 16")
        if out is None:
            out = torch.empty(obs.shape, dtype=dtype, device=self.device)
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_normalize(_ptr(obs), obs.numel(), self._NORM_DTYPES[dtype], _ptr(out), self._stream()),
                       "agym_normalize")
        return out

    def synth_frames(self, out: torch.Tensor, seed: int) -> torch.Tensor:
        """Fills a device u8 tensor with hashed pseudo-random bytes (benchmark input)."""
        assert out.dtype == torch.uint8 and out.is_contiguous() and out.device == self.device
        with torch.cuda.device(self.device):
            _lib.check(self._L.agym_synth_frames(_ptr(out), out.numel(), int(seed) & (2**64 - 1), self._stream()),
                       "agym_synth_frames")
        return out
