"""Sample-rate conversion on the B200: scipy's ``resample_poly`` (Kaiser-windowed sinc, ``padtype='constant'``) as one CUDA
kernel (``csrc/resample.cu`` behind ``include/smoltts_b200_resample.h``) for whole clips and for streams fed a chunk at a time.

For rates ``r_in -> r_out``: ``up / down = r_out / r_in`` in lowest terms, ``m = max(up, down)`` (at most 320), ``hl = 10 m``
and the filter ``h = up * firwin(2 hl + 1, 1 / m, window=('kaiser', 5.0))`` (``design_filter``, numpy only).  A clip of ``L``
samples gives ``ceil(L up / down)``; a stream emits an output as soon as its filter support has arrived (``output_count``) and
the rest at ``finish``.  A stream's samples are the same bits however its input was chunked and whatever shared the calls, and
its chunks concatenate to the whole-clip result.
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import List, Sequence, Tuple, Union

import numpy as np
import torch

from . import _capi
from .mimi import _aligned

def ratio(rate_in: int, rate_out: int) -> Tuple[int, int]:
    """(up, down): ``rate_out / rate_in`` in lowest terms."""
    g = math.gcd(int(rate_in), int(rate_out))
    return int(rate_out) // g, int(rate_in) // g


def design_filter(rate_in: int, rate_out: int) -> np.ndarray:
    """float64 taps ``up * firwin(2 hl + 1, 1 / m, window=('kaiser', 5.0))``: a Kaiser-windowed sinc with cutoff at the lower
    Nyquist frequency, normalised to unit DC gain, times ``up`` -- what ``scipy.signal.resample_poly`` builds."""
    up, down = ratio(rate_in, rate_out)
    m = max(up, down)
    hl = 10 * m
    cutoff = 1.0 / m
    n = np.arange(0, 2 * hl + 1, dtype=np.float64) - hl
    h = cutoff * np.sinc(cutoff * n)
    h *= np.kaiser(2 * hl + 1, 5.0)
    h /= np.sum(h)
    return h * up


def output_count(n_in: int, up: int, down: int, finish: bool) -> int:
    """Outputs a stream has emitted in all after ``n_in`` input samples: those whose filter support is complete, or with
    ``finish`` (the input ends there) all ``ceil(n_in up / down)``."""
    a = int(n_in) * up
    if finish:
        return -(-a // down)
    hl = 10 * max(up, down)
    return 0 if a <= hl else (a - 1 - hl) // down + 1


@dataclass
class ResamplerState:
    """One stream of a ``Resampler``: its slot and the samples consumed / emitted so far."""
    slot: int
    consumed: int = 0
    emitted: int = 0


class Resampler:
    """``rate_in -> rate_out`` for up to ``max_streams`` streams at once on one CUDA device.  Every call is asynchronous on the
    current CUDA stream and returns fp32 device tensors."""

    def __init__(self, rate_in: int, rate_out: int, max_streams: int = 1, device: Union[str, torch.device, None] = None):
        if not torch.cuda.is_available():
            raise RuntimeError("smoltts_b200.Resampler needs a CUDA device (there is no CPU path)")
        self.rate_in, self.rate_out = int(rate_in), int(rate_out)
        self.up, self.down = ratio(rate_in, rate_out)
        self.max_streams = int(max_streams)
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self._lib = _capi.load()
        cfg = _capi.SmolResampleConfig(rate_in=self.rate_in, rate_out=self.rate_out, max_streams=self.max_streams)
        h = C.c_void_p()
        _capi.check(self._lib.smol_resampler_create(C.byref(cfg), C.byref(h)))
        self._h = h
        taps = torch.from_numpy(design_filter(rate_in, rate_out).astype(np.float32)).to(self.device)
        assert taps.numel() == self._lib.smol_resampler_taps(h)
        n = int(self._lib.smol_resampler_workspace_bytes(h))
        self._ws = torch.empty(n + 256, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _capi.check(self._lib.smol_resampler_bind(h, C.c_void_p(taps.data_ptr()), C.c_void_p(_aligned(self._ws)), C.c_size_t(n),
                                                      C.c_void_p(self._stream())))
            torch.cuda.current_stream().synchronize()   # `taps` may go now: the kernel packed them into the workspace
        self._free = list(range(self.max_streams - 1, -1, -1))   # every free slot is at the start of a stream

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.smol_resampler_destroy(self._h)
                self._h = None
        except Exception:
            pass

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    @property
    def free_slots(self) -> int:
        return len(self._free)

    def _call(self, chunks: Sequence[torch.Tensor], states: Sequence[ResamplerState], finish: bool) -> List[torch.Tensor]:
        """One launch per SMOL_RESAMPLE_MAX_CALL streams: streams are independent, so the split changes no bits."""
        if len({s.slot for s in states}) != len(states):
            raise ValueError("Resampler: two chunks of a call name the same stream")
        g = _capi.SMOL_RESAMPLE_MAX_CALL
        return [y for i in range(0, len(states), g) for y in self._launch(chunks[i:i + g], states[i:i + g], finish)]

    def _launch(self, chunks: Sequence[torch.Tensor], states: Sequence[ResamplerState], finish: bool) -> List[torch.Tensor]:
        lens = [int(c.numel()) for c in chunks]
        counts = [output_count(s.consumed + n, self.up, self.down, finish) - s.emitted for s, n in zip(states, lens)]
        xs = [c.reshape(-1).to(device=self.device, dtype=torch.float32) for c in chunks if c.numel()]
        x = (xs[0].contiguous() if len(xs) == 1 else torch.cat(xs)) if xs else None
        out = torch.empty(sum(counts), dtype=torch.float32, device=self.device)
        n = len(states)
        got = (C.c_int64 * n)()
        _capi.check(self._lib.smol_resample(self._h, C.c_void_p(x.data_ptr() if x is not None else 0), (C.c_int64 * n)(*lens),
                                            (C.c_int32 * n)(*[s.slot for s in states]), n, int(finish),
                                            C.c_void_p(out.data_ptr() if out.numel() else 0), got, C.c_void_p(self._stream())))
        assert list(got) == counts, (list(got), counts)
        for s, k, c in zip(states, lens, counts):
            s.consumed, s.emitted = (0, 0) if finish else (s.consumed + k, s.emitted + c)
        return [out] if n == 1 else list(torch.split(out, counts))

    # ---- whole clips ----
    def resample(self, clips: Sequence[torch.Tensor]) -> List[torch.Tensor]:
        """Ragged 1-D clips -> their resampled clips (``ceil(L up / down)`` samples each), in one launch per 256 clips."""
        clips = list(clips)
        if not clips:
            return []
        if len(clips) > len(self._free):
            raise RuntimeError(f"Resampler.resample: {len(clips)} clips, {len(self._free)} free stream slots")
        states = [ResamplerState(s) for s in self._free[-len(clips):]]
        return self._call(clips, states, finish=True)   # a finished slot is back at the start: it stays free

    # ---- streams ----
    def make_state(self) -> ResamplerState:
        """A fresh stream in a free slot (zero history)."""
        if not self._free:
            raise RuntimeError(f"Resampler: all {self.max_streams} stream slots are in use (release_state() one)")
        return ResamplerState(self._free.pop())

    def step(self, chunks: Sequence[torch.Tensor], states: Sequence[ResamplerState]) -> List[torch.Tensor]:
        """The next chunk of every listed stream (ragged, any may be empty) -> the outputs each one completes, in one launch per 256
        streams."""
        if len(chunks) != len(states):
            raise ValueError(f"Resampler.step: {len(chunks)} chunks for {len(states)} streams")
        return self._call(chunks, states, finish=False) if states else []

    def finish(self, states: Sequence[ResamplerState]) -> List[torch.Tensor]:
        """The end of every listed stream: the outputs still owed (the input past the end is zero).  Each stream is then back at
        its start, in the same slot."""
        return self._call([torch.zeros(0)] * len(states), states, finish=True) if states else []

    def release_state(self, state: ResamplerState) -> None:
        if state.consumed:   # given back mid-stream: zero its history so that the free slot starts clean
            _capi.check(self._lib.smol_resampler_reset(self._h, (C.c_int32 * 1)(state.slot), 1, C.c_void_p(self._stream())))
            state.consumed = state.emitted = 0
        self._free.append(state.slot)
