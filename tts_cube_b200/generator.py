"""``CubeGenerator`` - drop-in for the reference's ``hifigan.models.Generator``.

Same constructor argument (the AttrDict/dict of ``hifigan/config_v*.json``), same
``load_state_dict`` keys (weight-norm ``weight_g``/``weight_v`` or folded ``weight``), same
``remove_weight_norm()`` / ``eval()`` / ``to(device)`` calls and the same forward contract
``wav[B,1,T] = generator(cond[B,80,F])`` (reference hifigan/models.py:72-125; callers
cube/networks/cubegan.py:83, cube/io_utils/runtime.py:51-54,78).  Inference only.
"""
from __future__ import annotations

import ctypes as C
from typing import Dict, List, Mapping, Optional, Sequence, Tuple

import torch

from . import _lib
from ._lib import VocConfig, check, lib
from .streaming import HifiganStream, step_streams


def _cfg_get(h, key, default=None):
    if isinstance(h, Mapping):
        return h.get(key, default)
    return getattr(h, key, default)


def _stream_ptr(device: torch.device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


class _Handle:
    """Owns one cube_voc_t*."""

    def __init__(self, cfg: VocConfig, device: torch.device):
        self.ptr = C.c_void_p()
        self.device = device
        self.num_mels = int(cfg.num_mels)
        check(lib().cube_voc_create(C.byref(self.ptr), C.byref(cfg), device.index or 0))

    def load(self, sd: Mapping[str, torch.Tensor]) -> None:
        for name, t in sd.items():
            a = t.detach().to("cpu", torch.float32).contiguous()
            shape = (C.c_int64 * max(a.dim(), 1))(*a.shape)
            check(lib().cube_voc_load_weight(self.ptr, name.encode(), C.c_void_p(a.data_ptr()), shape, a.dim()))

    def finalize(self) -> None:
        check(lib().cube_voc_finalize(self.ptr))

    def out_len(self, n_frames: int) -> int:
        n = lib().cube_voc_out_len(self.ptr, int(n_frames))
        if n < 0:
            check(1)
        return int(n)

    def forward(self, mel: torch.Tensor, n_frames: Optional[Sequence[int]], noise: Optional[torch.Tensor],
                want_int16: bool = False):
        if mel.device.type != "cuda":
            raise _lib.CubeVocError("mel must live on a CUDA device (no CPU path)")
        if mel.dtype != torch.float32 or mel.dim() != 3:
            raise _lib.CubeVocError(f"mel must be float32 [B, C, F], got {mel.dtype} {tuple(mel.shape)}")
        self._check_shapes(mel, n_frames)
        if mel.device != self.device:
            raise _lib.CubeVocError(f"mel lives on {mel.device} but this vocoder's weights live on {self.device}")
        mel = mel.contiguous()
        B, _, F = mel.shape
        T = self.out_len(F)
        wav = torch.empty(B, 1, T, device=mel.device, dtype=torch.float32)
        w16 = torch.empty(B, T, device=mel.device, dtype=torch.int16) if want_int16 else None
        nf = None
        if n_frames is not None:
            nf = (C.c_int32 * B)(*[int(v) for v in n_frames])
        if noise is not None:
            noise = noise.to(mel.device, torch.float32).contiguous()
            if noise.numel() != B * T:
                raise _lib.CubeVocError(f"noise must have B*T={B * T} elements, got {noise.numel()}")
        with torch.cuda.device(mel.device):
            check(lib().cube_voc_forward(
                self.ptr, C.c_void_p(mel.data_ptr()), nf, C.c_void_p(noise.data_ptr()) if noise is not None else None,
                C.c_void_p(wav.data_ptr()), C.c_void_p(w16.data_ptr()) if w16 is not None else None,
                B, F, C.c_void_p(_stream_ptr(mel.device))))
        return (wav, w16) if want_int16 else wav

    def forward_range(self, mel: torch.Tensor, n_frames: Optional[Sequence[int]], begin: Sequence[int],
                      end: Sequence[int], want_int16: bool = False, out: Optional[torch.Tensor] = None):
        """cube_voc_forward_range: only samples [begin[b], end[b]) of item b are written (into `out`, [B, 1, T] float32
        or [B, T] int16, when given).  Returns (out, list of the B requested slices)."""
        if mel.device.type != "cuda" or mel.dtype != torch.float32 or mel.dim() != 3:
            raise _lib.CubeVocError(f"mel must be float32 [B, C, F] on a CUDA device, got {mel.dtype} {tuple(mel.shape)} on {mel.device}")
        self._check_shapes(mel, n_frames)
        if mel.device != self.device:
            raise _lib.CubeVocError(f"mel lives on {mel.device} but this vocoder's weights live on {self.device}")
        mel = mel.contiguous()
        B, _, F = mel.shape
        if len(begin) != B or len(end) != B:
            raise _lib.CubeVocError(f"begin / end need {B} entries, got {len(begin)} / {len(end)}")
        T = self.out_len(F)
        shape, dt = ((B, T), torch.int16) if want_int16 else ((B, 1, T), torch.float32)
        if out is None:
            out = torch.empty(*shape, device=mel.device, dtype=dt)
        elif tuple(out.shape) != shape or out.dtype != dt or out.device != mel.device or not out.is_contiguous():
            raise _lib.CubeVocError(f"`out` must be a contiguous {dt} {shape} tensor on {mel.device}")
        nf = (C.c_int32 * B)(*[int(v) for v in n_frames]) if n_frames is not None else None
        b0 = (C.c_int64 * B)(*[int(v) for v in begin])
        b1 = (C.c_int64 * B)(*[int(v) for v in end])
        wav = None
        if want_int16:   # the float32 samples go to a scratch tensor the caller never sees
            wav = torch.empty(B, 1, T, device=mel.device, dtype=torch.float32)
        with torch.cuda.device(mel.device):
            check(lib().cube_voc_forward_range(
                self.ptr, C.c_void_p(mel.data_ptr()), nf, b0, b1,
                C.c_void_p((wav if want_int16 else out).data_ptr()), C.c_void_p(out.data_ptr()) if want_int16 else None,
                B, F, C.c_void_p(_stream_ptr(mel.device))))
        flat = out.view(B, T)
        return out, [flat[b, int(begin[b]):int(end[b])] for b in range(B)]

    def _check_shapes(self, mel: torch.Tensor, n_frames) -> None:
        """The engine trusts num_mels and B: a narrower tensor or a short n_frames list would be read out of bounds."""
        if mel.shape[1] != self.num_mels:
            raise _lib.CubeVocError(f"mel has {mel.shape[1]} channels, this vocoder was built for num_mels={self.num_mels}")
        if mel.shape[0] < 1 or mel.shape[2] < 1:
            raise _lib.CubeVocError(f"empty batch {tuple(mel.shape)}")
        if n_frames is not None and len(n_frames) != mel.shape[0]:
            raise _lib.CubeVocError(f"n_frames has {len(n_frames)} entries for a batch of {mel.shape[0]}")

    def forward_host(self, mel: torch.Tensor, n_frames, noise: Optional[torch.Tensor], out: torch.Tensor):
        """Host buffers in, host buffer out (H2D + forward + D2H inside the library)."""
        if mel.dim() != 3:
            raise _lib.CubeVocError(f"mel must be [B, C, F], got {tuple(mel.shape)}")
        for name, t in (("mel", mel), ("noise", noise), ("out", out)):
            if t is None:
                continue
            if t.device.type != "cpu" or not t.is_contiguous():
                raise _lib.CubeVocError(f"forward_host takes contiguous HOST tensors; `{name}` is {t.device}, contiguous={t.is_contiguous()}")
        if mel.dtype != torch.float32 or (noise is not None and noise.dtype != torch.float32):
            raise _lib.CubeVocError("forward_host takes float32 mel / noise")
        if out.dtype not in (torch.float32, torch.int16):
            raise _lib.CubeVocError(f"`out` must be float32 or int16, got {out.dtype}")
        self._check_shapes(mel, n_frames)
        B, _, F = mel.shape
        T = self.out_len(F)
        if out.numel() != B * T:
            raise _lib.CubeVocError(f"`out` must hold B*T = {B}*{T} samples, got {tuple(out.shape)}")
        if noise is not None and noise.numel() != B * T:
            raise _lib.CubeVocError(f"noise must have B*T = {B * T} elements, got {noise.numel()}")
        nf = (C.c_int32 * B)(*[int(v) for v in n_frames]) if n_frames is not None else None
        wav_p = C.c_void_p(out.data_ptr()) if out.dtype == torch.float32 else None
        i16_p = C.c_void_p(out.data_ptr()) if out.dtype == torch.int16 else None
        check(lib().cube_voc_forward_host(self.ptr, C.c_void_p(mel.data_ptr()), nf,
                                          C.c_void_p(noise.data_ptr()) if noise is not None else None,
                                          wav_p, i16_p, B, F))
        return out

    def launches(self) -> int:
        return int(lib().cube_voc_last_launches(self.ptr))

    def workspace_bytes(self) -> int:
        return int(lib().cube_voc_workspace_bytes(self.ptr))

    def set_profile(self, on: bool) -> None:
        check(lib().cube_voc_set_profile(self.ptr, int(on)))

    def get_profile(self) -> Dict[str, float]:
        cap = 64
        names = C.create_string_buffer(cap * 64)
        ms = (C.c_float * cap)()
        n = lib().cube_voc_get_profile(self.ptr, names, ms, cap)
        if n < 0:
            check(1)
        return {names.raw[i * 64:(i + 1) * 64].split(b"\0")[0].decode(): float(ms[i]) for i in range(n)}

    def close(self):
        if self.ptr:
            lib().cube_voc_destroy(self.ptr)
            self.ptr = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def hifigan_tc_supported(h) -> bool:
    """The tcgen05 path covers ResBlock1 generators whose stage widths are all in {32,...,512}."""
    c0 = int(_cfg_get(h, "upsample_initial_channel"))
    n = len(list(_cfg_get(h, "upsample_rates")))
    widths = [c0 >> i for i in range(n + 1)]
    return (str(_cfg_get(h, "resblock")) == "1" and all(w in (32, 64, 128, 256, 512) for w in widths)
            and int(_cfg_get(h, "num_mels", 80) or 80) % 8 == 0)


def hifigan_config(h, math=None) -> VocConfig:
    if math is None:  # auto: tensor cores where the architecture fits, else the fp32 kernels
        math = _lib.MATH_TC_SPLIT16 if hifigan_tc_supported(h) else _lib.MATH_FP32_SIMT
    cfg = VocConfig()
    cfg.arch = _lib.ARCH_HIFIGAN
    cfg.math = math
    cfg.num_mels = int(_cfg_get(h, "num_mels", 80) or 80)
    cfg.upsample_initial_channel = int(_cfg_get(h, "upsample_initial_channel"))
    rates = list(_cfg_get(h, "upsample_rates"))
    ks = list(_cfg_get(h, "upsample_kernel_sizes"))
    if len(rates) != len(ks) or len(rates) > _lib.MAX_UPS:
        raise _lib.CubeVocError("bad upsample_rates / upsample_kernel_sizes")
    cfg.n_ups = len(rates)
    for i, (u, k) in enumerate(zip(rates, ks)):
        cfg.upsample_rates[i], cfg.upsample_kernel_sizes[i] = int(u), int(k)
    cfg.resblock_type = 1 if str(_cfg_get(h, "resblock")) == "1" else 2
    rk = list(_cfg_get(h, "resblock_kernel_sizes"))
    rd = list(_cfg_get(h, "resblock_dilation_sizes"))
    cfg.n_resblock_kernels = len(rk)
    for j, (k, d) in enumerate(zip(rk, rd)):
        cfg.resblock_kernel_sizes[j] = int(k)
        cfg.n_dilations[j] = len(d)
        for m, dd in enumerate(d):
            cfg.resblock_dilations[j][m] = int(dd)
    return cfg


class CubeGenerator(torch.nn.Module):
    """B200 replacement for ``hifigan.models.Generator`` (inference)."""

    def __init__(self, h, math=None):
        """math: None = auto (tcgen05 split-fp16 when the architecture fits, else fp32 FFMA),
        _lib.MATH_FP32_SIMT or _lib.MATH_TC_SPLIT16 to force one."""
        super().__init__()
        self.h = h
        self._cfg = hifigan_config(h, math)
        self._sd: Dict[str, torch.Tensor] = {}
        self._handle: Optional[_Handle] = None
        # parameter-free module: a buffer tracks the device the way the reference's parameters do
        self.register_buffer("_device_tracker", torch.zeros(1), persistent=False)
        lib()  # fail at construction time when the CUDA library is absent

    # ---- reference-compatible surface -------------------------------------------------------
    def load_state_dict(self, state_dict, strict: bool = True, assign: bool = False):  # noqa: D102
        sd = {k: v for k, v in state_dict.items()}
        self._sd = {k: v.detach().to("cpu", torch.float32).clone() for k, v in sd.items()}
        self._drop_handle()
        return torch.nn.modules.module._IncompatibleKeys([], [])

    def state_dict(self, *a, **k):  # noqa: D102
        return dict(self._sd)

    def remove_weight_norm(self):
        """hifigan/models.py:118-125.  Folding happens once inside cube_voc_finalize()."""
        return self

    def _drop_handle(self):
        if self._handle is not None:
            self._handle.close()
            self._handle = None

    def _apply(self, fn, *a, **k):
        before = self._device_tracker.device
        r = super()._apply(fn, *a, **k)
        if self._device_tracker.device != before:
            self._drop_handle()
        return r

    @property
    def device(self) -> torch.device:
        return self._device_tracker.device

    def _ensure(self) -> _Handle:
        if self._handle is None:
            dev = self.device
            if dev.type != "cuda":
                raise _lib.CubeVocError("CubeGenerator must be moved to a CUDA device (.to('cuda:0')); there is no CPU path")
            if not self._sd:
                raise _lib.CubeVocError("load_state_dict() must be called before forward()")
            dev = torch.device("cuda", dev.index if dev.index is not None else torch.cuda.current_device())
            hd = _Handle(self._cfg, dev)
            hd.load(self._sd)
            hd.finalize()
            self._handle = hd
        return self._handle

    def out_len(self, n_frames: int) -> int:
        return self._ensure().out_len(n_frames)

    def forward(self, x: torch.Tensor, n_frames: Optional[Sequence[int]] = None) -> torch.Tensor:
        """x [B, 80, F] float32 cuda -> [B, 1, T] float32 cuda (hifigan/models.py:100-116)."""
        if torch.is_grad_enabled() and x.requires_grad:
            raise _lib.CubeVocError("CubeGenerator is inference-only: call it under torch.no_grad() "
                                    "(training goes through the reference Generator)")
        return self._ensure().forward(x, n_frames, None)

    def forward_int16(self, x: torch.Tensor, n_frames: Optional[Sequence[int]] = None):
        """Fused cube/api.py:64-65 epilogue: returns (wav float32 [B,1,T], int16 [B,T])."""
        return self._ensure().forward(x, n_frames, None, want_int16=True)

    # ---- streaming (tts_cube_b200/streaming.py) ------------------------------------------------
    @property
    def hop(self) -> int:
        """Output samples per mel frame: prod(upsample_rates)."""
        n = 1
        for i in range(self._cfg.n_ups):
            n *= int(self._cfg.upsample_rates[i])
        return n

    def sample_support(self, s0: int, s1: int) -> Tuple[int, int]:
        """Mel frames [f0, f1) that output samples [s0, s1) depend on (f0 clipped at 0, f1 not clipped).  No GPU needed."""
        f0, f1 = C.c_int64(), C.c_int64()
        check(lib().cube_voc_hifigan_support(C.byref(self._cfg), int(s0), int(s1), C.byref(f0), C.byref(f1)))
        return int(f0.value), int(f1.value)

    def forward_range(self, mel: torch.Tensor, n_frames: Optional[Sequence[int]], begin: Sequence[int],
                      end: Sequence[int], int16: bool = False, out: Optional[torch.Tensor] = None) -> List[torch.Tensor]:
        """Samples [begin[b], end[b]) of generator(mel[b, :, :n_frames[b]]), bit-identical to forward(); one tensor of
        end[b] - begin[b] samples per item (views into `out` when given: [B, 1, T] float32 or [B, T] int16, whose other
        elements are left untouched)."""
        return self._ensure().forward_range(mel, n_frames, begin, end, want_int16=int16, out=out)[1]

    def open_stream(self, int16: bool = False) -> HifiganStream:
        """A session fed mel chunks [num_mels, f]; see HifiganStream."""
        return HifiganStream(self.sample_support, self.out_len, self.hop, int(self._cfg.num_mels), int16=int16, owner=self)

    def step_streams(self, streams: Sequence[HifiganStream]) -> List[torch.Tensor]:
        """One batched forward_range over the sessions (one per output type) -> each session's newly final samples."""
        out: List[Optional[torch.Tensor]] = [None] * len(streams)
        for i16 in (False, True):
            idx = [i for i, s in enumerate(streams) if s.int16 == i16]
            if not idx:
                continue
            vr = lambda m, nf, b, e, i16=i16: self.forward_range(m, nf, b, e, int16=i16)  # noqa: E731
            for i, piece in zip(idx, step_streams([streams[i] for i in idx], vr, device=self.device)):
                out[i] = piece
        return out  # type: ignore

    def forward_host(self, mel: torch.Tensor, n_frames=None, out: Optional[torch.Tensor] = None,
                     int16: bool = False) -> torch.Tensor:
        """End-to-end call with HOST tensors: pinned/pageable mel in, audio out (float32 or int16)."""
        hd = self._ensure()
        B, _, F = mel.shape
        T = hd.out_len(F)
        if out is None:
            out = torch.empty(B, T, dtype=torch.int16 if int16 else torch.float32).pin_memory()
        return hd.forward_host(mel.contiguous(), n_frames, None, out)


def install_into_cubegan(model, math=None):
    """Replace ``model._generator`` (reference cube/networks/cubegan.py:43) by a CubeGenerator that
    carries the same weights, on the same device.  ``model.inference`` then runs unchanged."""
    ref = model._generator
    g = CubeGenerator(ref.h, math=math)
    g.load_state_dict(ref.state_dict())
    dev = next(ref.parameters()).device
    g.to(dev)
    model._generator = g
    return model
