"""Incremental HiFi-GAN synthesis: stream sessions over ``CubeGenerator.forward_range``.

HiFi-GAN is non-causal and zero-pads every conv edge, so cutting a mel into chunks and vocoding each chunk gives
different samples near every cut.  A session instead keeps the mel frames it has been fed and, at every step, emits the
samples that no future frame can change: samples ``[E, S)`` where ``E`` is what it has emitted so far and ``S`` is the
largest end whose support (``cube_voc_hifigan_support``) lies inside the frames fed.  It vocodes the window of frames
that support names and keeps only the requested samples, which are bit-identical to the whole-utterance call.
Concatenating every piece a session returns gives ``generator(mel)[0, 0, :out_len(F)]`` for any chunking.

The layer geometry lives in the library; this module only asks it.  ``step_streams`` takes the range vocoder as a
callable (``vocode_range(mel [B, C, F], n_frames, begin, end) -> list of B tensors``), so the schedule can be driven
through any reference implementation.
"""
from __future__ import annotations

from typing import Callable, List, Optional, Sequence, Tuple

import torch

from .api import pad_mels

Support = Callable[[int, int], Tuple[int, int]]


class HifiganStream:
    """One utterance being vocoded while its mel is still arriving.

    ``feed(mel_chunk [num_mels, f])`` appends frames (``f`` may be 0), ``close_input()`` marks the end of the mel.
    ``push`` / ``finish`` are those two followed by a step of this session alone; batch many sessions with
    ``CubeGenerator.step_streams``.
    """

    def __init__(self, support: Support, out_len: Callable[[int], int], hop: int, num_mels: int = 80,
                 int16: bool = False, owner=None):
        self._support = support
        self._out_len = out_len
        self.hop = int(hop)
        self.num_mels = int(num_mels)
        self.int16 = bool(int16)
        self._owner = owner
        self._frames: Optional[torch.Tensor] = None   # kept frames [num_mels, n], the first one is frame `_base`
        self._base = 0
        self.n_fed = 0          # N: frames fed
        self.emitted = 0        # E: samples [0, E) have been returned
        self.closed = False

    # ---- input -------------------------------------------------------------------------------------------------
    def feed(self, mel_chunk: torch.Tensor) -> None:
        if self.closed:
            raise ValueError("feed() after close_input()")
        if mel_chunk.dim() != 2 or mel_chunk.shape[0] != self.num_mels:
            raise ValueError(f"mel chunk must be [{self.num_mels}, f], got {tuple(mel_chunk.shape)}")
        chunk = mel_chunk.to(torch.float32)
        if self._frames is None:
            self._frames = chunk.clone()
        elif chunk.shape[1]:
            self._frames = torch.cat([self._frames, chunk.to(self._frames.device)], dim=1)
        self.n_fed += int(chunk.shape[1])

    def close_input(self) -> None:
        self.closed = True

    @property
    def done(self) -> bool:
        return self.closed and self.emitted == self.total_len()

    def total_len(self) -> int:
        return self._out_len(self.n_fed) if self.n_fed else 0

    def kept_frames(self) -> int:
        return 0 if self._frames is None else int(self._frames.shape[1])

    # ---- schedule ----------------------------------------------------------------------------------------------
    def _next_end(self) -> int:
        """S: the end of the samples that are final now."""
        E, N = self.emitted, self.n_fed
        if N == 0:
            return E
        if self.closed:
            return self.total_len()
        ready = lambda s: self._support(E, s)[1] <= N   # noqa: E731  (monotone in s)
        if not ready(E + 1):
            return E
        lo, hi = E + 1, E + 2
        while ready(hi):
            lo, hi = hi, E + 2 * (hi - E)
        while hi - lo > 1:
            mid = (lo + hi) // 2
            if ready(mid):
                lo = mid
            else:
                hi = mid
        return lo

    def plan(self):
        """(window mel [num_mels, f1 - f0], begin, end) in window samples for the next step, or None."""
        E, S = self.emitted, self._next_end()
        if S <= E:
            return None
        f0, f1 = self._support(E, S)
        f1 = min(f1, self.n_fed)
        off = f0 * self.hop
        win = self._frames[:, f0 - self._base: f1 - self._base]
        return win, E - off, S - off

    def _advance(self, end: int) -> None:
        self.emitted = end
        if self.emitted >= self.total_len() and self.closed:
            self._frames = self._frames[:, :0] if self._frames is not None else None
            return
        keep = self._support(self.emitted, self.emitted + 1)[0]   # later windows start at or after this frame
        if keep > self._base and self._frames is not None:
            self._frames = self._frames[:, keep - self._base:]
            self._base = keep

    # ---- one-session conveniences ------------------------------------------------------------------------------
    def push(self, mel_chunk: torch.Tensor) -> torch.Tensor:
        self.feed(mel_chunk)
        return self._owner.step_streams([self])[0]

    def finish(self) -> torch.Tensor:
        self.close_input()
        return self._owner.step_streams([self])[0]


def step_streams(streams: Sequence[HifiganStream], vocode_range: Callable, device=None) -> List[torch.Tensor]:
    """One batched range call over every session with samples ready; returns each session's newly final samples
    (an empty tensor where there are none)."""
    plans = [s.plan() for s in streams]
    live = [i for i, p in enumerate(plans) if p is not None]
    out: List[Optional[torch.Tensor]] = [None] * len(streams)
    if live:
        mb = pad_mels([plans[i][0] for i in live])
        if device is not None:
            mb = mb.to(device)
        pieces = vocode_range(mb, [int(plans[i][0].shape[1]) for i in live], [plans[i][1] for i in live],
                              [plans[i][2] for i in live])
        for k, i in enumerate(live):
            s = streams[i]
            s._advance(s.emitted + (plans[i][2] - plans[i][1]))
            out[i] = pieces[k]
    for i, s in enumerate(streams):
        if out[i] is None:
            dev = device if device is not None else (s._frames.device if s._frames is not None else "cpu")
            out[i] = torch.empty(0, dtype=torch.int16 if s.int16 else torch.float32, device=dev)
    return out  # type: ignore
