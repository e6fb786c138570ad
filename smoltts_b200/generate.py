"""Generate API of the reference (mlx_inference/src/smoltts_mlx/lm/generate.py) over the B200 engine.

``GenerationSettings`` (:12-16), ``VQToken`` (:19-22), ``SingleBatchGenerator`` (:25-171) and
``generate_blocking`` (:174-216) keep the reference's names, arguments and loop semantics
(prefill on the first ``next``, one Mimi frame per ``next``, ``<|im_end|>`` stop rule under
``audio_only``, at most ``max_new_tokens + 1`` frames).  Differences, all deliberate:
  * sampling runs on the device with a counter-based RNG; ``top_k`` / ``top_p`` / ``seed`` are
    added, and ``min_p`` follows the *intended* rule (the reference's is a no-op, SURVEY §8(g)-8)
    only when ``min_p_intended=True``;
  * ``generate_batch`` is new (the reference is bs=1 only): B utterances advance together inside
    one persistent kernel launch per chunk of frames, with the stop rule evaluated on the device;
    each utterance may carry its own ``GenerationSettings`` (a device table of per-row sampling
    parameters, ``row_sampling_table``).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass
from typing import Any, List, Optional, Sequence, Union

import torch

from . import _capi
from .model import DecodeBatch, RQTransformer, SlowCache


@dataclass
class GenerationSettings:
    default_temp: float = 0.7
    default_fast_temp: Optional[float] = 0.7
    min_p: Optional[float] = None
    max_new_tokens: int = 1024
    # additions (north star): nucleus / top-k on the slow token, RNG seed
    top_k: int = 0
    top_p: float = 1.0
    seed: int = 0
    min_p_intended: bool = False


@dataclass
class VQToken:
    semantic_code: int
    audio_codes: Optional[Any]
    vq_tensor: Any


def _min_p(s: GenerationSettings) -> float:
    return float(s.min_p) if (s.min_p is not None and s.min_p_intended) else 0.0


def _sampling(model: RQTransformer, s: GenerationSettings, audio_only: bool, ignore_stop: bool = False):
    return model.sampling(temp=s.default_temp, fast_temp=s.default_fast_temp or 0.0, top_k=s.top_k, top_p=s.top_p,
                          min_p=_min_p(s), seed=s.seed, audio_only=audio_only, ignore_stop=ignore_stop)


def _check_settings(s: GenerationSettings, where: str) -> None:
    for name, t in (("default_temp", s.default_temp), ("default_fast_temp", s.default_fast_temp or 0.0)):
        if not (math.isfinite(t) and t >= 0.0):
            raise ValueError(f"{where}: {name} = {t} must be a finite number >= 0")
    if s.top_k < 0:
        raise ValueError(f"{where}: top_k = {s.top_k} must be >= 0")
    if not (0.0 < s.top_p <= 1.0):
        raise ValueError(f"{where}: top_p = {s.top_p} must lie in (0, 1]")
    if s.min_p is not None and not (0.0 <= s.min_p < 1.0):
        raise ValueError(f"{where}: min_p = {s.min_p} must lie in [0, 1)")


def row_sampling_table(settings: Sequence[GenerationSettings]) -> torch.Tensor:
    """Host tensor [B, 32] uint8: one ``SmolRowSampling`` record per settings object (include/smoltts_b200.h), the values
    ``_sampling`` would put in a call's ``SmolSampling``.  Raises ``ValueError`` for parameters the sampler does not define."""
    settings = list(settings)
    if not settings:
        raise ValueError("row_sampling_table: no settings")
    recs = (_capi.SmolRowSampling * len(settings))()
    for i, s in enumerate(settings):
        _check_settings(s, f"settings[{i}]")
        recs[i] = _capi.SmolRowSampling(temp=float(s.default_temp), fast_temp=float(s.default_fast_temp or 0.0), top_k=int(s.top_k),
                                        top_p=float(s.top_p), min_p=_min_p(s), seed=int(s.seed))
    return torch.frombuffer(bytearray(recs), dtype=torch.uint8).view(len(settings), C.sizeof(_capi.SmolRowSampling))


class SingleBatchGenerator:
    """One utterance, one frame per ``next()`` (reference :25-171)."""

    def __init__(self, model: RQTransformer, prompt: torch.Tensor, generation_settings: GenerationSettings,
                 audio_only: bool = True, seq_id: int = 0):
        self.model = model
        self.input_pos = 0
        self.max_new_tokens = (generation_settings.max_new_tokens
                               if generation_settings.max_new_tokens is not None else model.config.max_seq_len)
        self.generation_settings = generation_settings
        self.audio_only = audio_only
        p = prompt if prompt.ndim == 3 else prompt[None]
        self.prompt: Optional[torch.Tensor] = p.to(device=model.device, dtype=torch.int32).contiguous()
        need = p.shape[2] + self.max_new_tokens + 1
        self.slow_cache = SlowCache(model, max_positions=min(need, model.max_seq_len), seq_id=seq_id)
        self._sampling = _sampling(model, generation_settings, audio_only)
        self._prefilled = False

    def __iter__(self):
        return self

    def __next__(self) -> VQToken:
        if self.input_pos > self.max_new_tokens:
            raise StopIteration
        if self.prompt is None:  # previous iteration told us to stop
            raise StopIteration
        model, batch = self.model, self.slow_cache.batch
        if not self._prefilled:
            S = self.prompt.shape[2]
            model.prefill(batch, self.prompt, torch.tensor([S], dtype=torch.int32, device=model.device))
            self._prefilled = True
        model.decode_frames(batch, self._sampling, 1)
        vq = batch.tokens[0].clone()  # [R]: row 0 vocab id, rows 1.. depth codes (reference :143-145)
        host = vq.tolist()
        slow = host[0]
        tc, cfg = model.token_config, model.config
        codes_tensor = vq.view(1, -1, 1)
        audio = None
        if tc.semantic_end_id is not None and tc.semantic_start_id <= slow <= tc.semantic_end_id:
            # (built from the device copy of the column: no host -> device copy per frame on the streaming path)
            audio = (vq[1:] if cfg.duplicate_code_0 else torch.cat([vq[0:1] - tc.semantic_start_id, vq[1:]])).view(1, -1, 1)
        self.input_pos += 1
        if self.audio_only and slow == tc.im_end_id:
            self.prompt = None
        return VQToken(semantic_code=slow, audio_codes=audio, vq_tensor=codes_tensor)


def generate_blocking(model: RQTransformer, prompt: torch.Tensor, generation_settings: GenerationSettings,
                      audio_only: bool = True) -> torch.Tensor:
    """reference :174-216.  Returns codes [1, N, T] (audio_only) or [1, 1+N, T]."""
    gen = SingleBatchGenerator(model, prompt, generation_settings, audio_only)
    first = next(gen)
    kept: List[torch.Tensor] = []
    item = first.audio_codes if audio_only else first.vq_tensor
    if item is not None:  # the reference crashes in mx.concat here when the first id is not audio (§8(g)-9)
        kept.append(item)
    for tok in gen:
        if audio_only:
            if tok.audio_codes is not None:
                kept.append(tok.audio_codes)
        else:
            kept.append(tok.vq_tensor)
    if not kept:
        n = model.config.num_codebooks if audio_only else model.config.n_rows
        return torch.zeros(1, n, 0, dtype=torch.int32, device=model.device)
    return torch.cat(kept, dim=-1)


def pack_prompts(model: RQTransformer, prompts: Sequence[torch.Tensor]):
    """list of [R, S_i] -> (padded [B, R, s_max] int32 device, lengths [B] int32 device)."""
    R = model.config.n_rows
    s_max = max(int(p.shape[-1]) for p in prompts)
    pin = model.device.type == "cuda"      # page-locked staging: the copy below is one asynchronous DMA
    out = torch.zeros(len(prompts), R, s_max, dtype=torch.int32, pin_memory=pin)
    lens = []
    for b, p in enumerate(prompts):
        p2 = p if p.ndim == 2 else p[0]
        if p2.shape[0] != R:
            raise ValueError(f"prompt {b} has {p2.shape[0]} rows, model expects {R}")
        out[b, :, : p2.shape[1]] = p2.to(torch.int32).cpu()
        lens.append(int(p2.shape[1]))
    lens_h = torch.tensor(lens, dtype=torch.int32, pin_memory=pin)
    return out.to(model.device, non_blocking=pin), lens_h.to(model.device, non_blocking=pin)


def generate_batch(model: RQTransformer, prompts: Sequence[torch.Tensor],
                   generation_settings: Union[GenerationSettings, Sequence[GenerationSettings]],
                   audio_only: bool = True, fixed_frames: Optional[int] = None, chunk: int = 64,
                   seq_ids: Optional[Sequence[int]] = None, return_batch: bool = False):
    """B utterances decoded together; per-sequence semantics identical to the bs=1 loop.

    Returns a list of int32 tensors: audio_only -> codes [N, T_b] of the audio frames;
    otherwise [1+N, T_b] of every emitted column.  ``fixed_frames`` disables the stop rule
    (benchmarks: random weights never emit <|im_end|> reliably, SURVEY §8(d)).

    ``generation_settings`` is one ``GenerationSettings`` for every utterance, or one per prompt: each then samples with
    its own temperatures, top-k / top-p / min-p and seed, and keeps at most its own ``max_new_tokens + 1`` frames (the call
    runs the largest budget; a row's frames do not depend on the others' settings or budgets)."""
    B = len(prompts)
    per_row = not isinstance(generation_settings, GenerationSettings)
    rows = list(generation_settings) if per_row else [generation_settings] * B
    if len(rows) != B:
        raise ValueError(f"{len(rows)} settings for {B} prompts")
    budgets = [fixed_frames if fixed_frames is not None else r.max_new_tokens + 1 for r in rows]
    table = model.row_sampling(rows) if per_row else None
    padded, lens = pack_prompts(model, prompts)
    n_frames = max(budgets)
    need = int(padded.shape[2]) + n_frames
    if need > model.max_seq_len:
        raise ValueError(f"prompt + frames = {need} positions exceed max_seq_len {model.max_seq_len}")
    batch = model.new_batch(B, max_positions=need, max_frames=n_frames, seq_ids=seq_ids)
    batch.set_row_sampling(table)
    sampling = _sampling(model, rows[0], audio_only, ignore_stop=fixed_frames is not None)
    model.prefill(batch, padded, lens)
    done = 0
    while done < n_frames:
        n = min(chunk, n_frames - done)
        model.decode_frames(batch, sampling, n)
        done += n
        if fixed_frames is None and done < n_frames and bool(batch.finished.all().item()):
            break
    steps = [min(st, bud) for st, bud in zip(batch.step.tolist(), budgets)]
    codes = batch.out_codes.cpu()
    tc, cfg = model.token_config, model.config
    outs: List[torch.Tensor] = []
    for b in range(B):
        cols = codes[b, : steps[b]].t().contiguous()  # [R, T]
        if audio_only:
            lo, hi = tc.semantic_start_id, tc.semantic_end_id if tc.semantic_end_id is not None else -1
            keep = (cols[0] >= lo) & (cols[0] <= hi)
            if cfg.duplicate_code_0:
                cols = cols[1:, keep]
            else:
                cols = torch.cat([(cols[0:1, keep] - lo), cols[1:, keep]], dim=0)
        outs.append(cols)
    if return_batch:
        return outs, batch
    batch.release()
    return outs
