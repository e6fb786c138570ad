"""Text -> PCM: the reference's ``SmolTTS`` front object (mlx_inference/src/smoltts_mlx/__init__.py:25-151) over the two
B200 engines -- the DualAR decode step (``RQTransformer``) and the Mimi streaming decoder (``MimiModel``).

Same call surface: ``SmolTTS(...)(text, voice)`` returns the flattened PCM of one utterance (:64-83), ``stream(text,
voice)`` yields one 80 ms chunk per generated frame (:85-95: a fresh Mimi cache per utterance, ``decode_step`` on the
frame's codes).  ``synthesize_batch`` is new: B utterances decode together (``generate_batch``), then their frames go
through the codec as one batch of B streams per step.

Parity note: the reference's ``__call__`` decodes the whole code sequence with ``codec.decode`` (the upsampler sees the
sequence) while its ``stream`` upsamples every frame alone (codec/mimi.py:73-104): the two give different audio in the
reference, and so do they here -- ``__call__`` uses a codec stream with the upsampler's carry, ``stream`` one without.
"""
from __future__ import annotations

from typing import Iterator, List, Optional, Sequence

import numpy as np
import torch

from .generate import GenerationSettings, SingleBatchGenerator, generate_batch, generate_blocking
from .mimi import MimiModel
from .model import RQTransformer
from .serving import PromptEncoder

VOICES = ["heart", "bella", "nova", "sky", "sarah", "michael", "fenrir", "liam", "emma", "isabella", "fable"]   # :127-143


class SmolTTS:
    def __init__(self, lm: RQTransformer, prompt_encoder: PromptEncoder, codec_stream: MimiModel, codec_full: Optional[MimiModel] = None,
                 settings: Optional[GenerationSettings] = None):
        """codec_stream: a MimiModel with the reference's decode_step rule (upsample_carry=False); codec_full: one with
        upsample_carry=True for ``__call__`` / ``synthesize_batch`` (defaults to codec_stream if it already carries)."""
        self.lm = lm
        self.prompt_encoder = prompt_encoder
        self.codec = codec_stream
        self.codec_full = codec_full if codec_full is not None else codec_stream
        self.settings = settings or GenerationSettings()
        self.sampling_rate = 24_000

    # ---- prompt assembly (:123-151) ----
    def _get_prompt(self, input: str, voice: str, sysprompt: Optional[torch.Tensor] = None) -> torch.Tensor:
        voice_id = VOICES.index(voice) if voice in VOICES else 0
        return self.prompt_encoder.tts_prompt(input, speaker=voice_id, sysprompt=sysprompt)[None]

    def create_speaker(self, samples: Sequence[dict], system_prompt: Optional[str] = None) -> torch.Tensor:
        """Voice-clone prefix (__init__.py:97-118) from ``{"text", "audio"}`` samples -- 1-D float PCM at 24 kHz, mono -- or
        ``{"text", "codes"}`` samples with ready-made Mimi codes.  The audio of all samples is encoded in one
        ``MimiModel.encode`` call (the codec must have been built with ``encode_max_samples > 0``)."""
        samples = list(samples)
        with_audio = [i for i, s in enumerate(samples) if "audio" in s and "codes" not in s]
        if with_audio:
            codec = next((c for c in (self.codec, self.codec_full) if c._enc is not None), None)
            if codec is None:
                raise ValueError("create_speaker: samples carry 'audio' but the codec has no encoder "
                                 "(build the MimiModel with encode_max_samples > 0, or pass 'codes')")
            clips = [torch.as_tensor(samples[i]["audio"], dtype=torch.float32).reshape(-1) for i in with_audio]
            codes = codec.encode(clips)
            samples = [dict(s) for s in samples]
            for i, c in zip(with_audio, codes):
                samples[i].pop("audio")
                samples[i]["codes"] = c.cpu()
        return self.prompt_encoder.create_speaker(samples, system_prompt)

    # ---- one utterance (:64-83) ----
    def __call__(self, input: str, voice: Optional[str] = "heart", speaker: Optional[torch.Tensor] = None) -> np.ndarray:
        prompt = self._get_prompt(input, voice if voice is not None else "heart", sysprompt=speaker)
        codes = generate_blocking(self.lm, prompt, self.settings)          # [1, N, T]
        if codes.shape[-1] == 0:
            return np.zeros(0, dtype=np.float32)
        pcm = self.codec_full.decode(codes.to(torch.int64))
        return pcm.flatten().cpu().numpy()

    # ---- streaming (:85-95) ----
    def stream(self, input: str, voice: Optional[str] = "heart", overlap: bool = True, lm_ctas: int = 96,
               stats: Optional[dict] = None) -> Iterator[np.ndarray]:
        """One 80 ms PCM chunk per generated audio frame.  ``overlap=False`` is the reference's loop as written: one frame per
        ``SingleBatchGenerator.__next__`` (launch, host read-back), then the codec step, then the chunk.  ``overlap`` (default)
        keeps both engines busy: the decode step of frame t + 1 is launched BEFORE the host looks at frame t, and frame t's ids,
        its codec step and its PCM go through a side stream -- the data-flow kernel is told to take ``lm_ctas`` of the GPU's SMs (a
        bs=1 frame takes the same 600-612 us on 96 .. 148 CTAs, DESIGN.md section 4), the codec's kernels run on the others.
        Throughput is then bound by the slower engine instead of the sum plus the host's time per frame.  Same chunks, bit for bit."""
        prompt = self._get_prompt(input, voice if voice is not None else "0")
        codec = self.codec
        cache = codec.make_cache()
        n_frames = n_audio = 0
        old_ctas = None
        batch = None
        try:
            if not overlap:
                for frame in SingleBatchGenerator(self.lm, prompt, self.settings):
                    n_frames += 1
                    if frame.audio_codes is None:      # the <|im_end|> frame (the reference would hand None to the codec here)
                        continue
                    if cache.frames >= codec.max_frames:
                        break
                    n_audio += 1
                    yield codec.decode_step(frame.audio_codes, cache).flatten().cpu().numpy()
                return
            from .generate import _sampling

            lm, s = self.lm, self.settings
            tc, cfg = lm.token_config, lm.config
            if lm_ctas > 0:
                old_ctas = lm.get_option("n_ctas_override")
                lm.set_option("n_ctas", lm_ctas)
            budget = s.max_new_tokens + 1                                   # frames of the reference loop (lm/generate.py:60,161)
            p = prompt.to(device=lm.device, dtype=torch.int32).contiguous()
            S = int(p.shape[2])
            batch = lm.new_batch(1, max_positions=min(S + budget + 1, lm.max_seq_len), max_frames=budget)
            sampling = _sampling(lm, s, audio_only=True)
            lm.prefill(batch, p, torch.tensor([S], dtype=torch.int32, device=lm.device))
            main, side = torch.cuda.current_stream(lm.device), torch.cuda.Stream(device=lm.device)
            done_ev = {}

            def launch(t: int) -> None:
                lm.decode_frames(batch, sampling, 1)
                ev = torch.cuda.Event()
                ev.record(main)
                done_ev[t] = ev

            launch(0)
            lo, hi = tc.semantic_start_id, tc.semantic_end_id if tc.semantic_end_id is not None else -1
            for t in range(budget):
                if t + 1 < budget:
                    launch(t + 1)                                            # runs while the host and the codec deal with frame t
                with torch.cuda.stream(side):
                    side.wait_event(done_ev.pop(t))
                    col = batch.out_codes[0, t]
                    slow = int(col[0].item())                                # (a read on the side stream: it does not wait for frame t + 1)
                    n_frames += 1
                    out = None
                    if lo <= slow <= hi and cache.frames < codec.max_frames:
                        codes = col[1:] if cfg.duplicate_code_0 else torch.cat([col[0:1] - lo, col[1:]])
                        out = codec.decode_step(codes.view(1, -1, 1), cache).flatten().cpu().numpy()
                        n_audio += 1
                if out is not None:
                    yield out
                if slow == tc.im_end_id or (lo <= slow <= hi and out is None):
                    break
        finally:
            torch.cuda.synchronize(codec.device)
            codec.release_cache(cache)
            if batch is not None:
                batch.release()
            if old_ctas is not None:
                self.lm.set_option("n_ctas", old_ctas)
            if stats is not None:
                stats["frames"], stats["audio_frames"] = n_frames, n_audio

    # ---- many utterances at once (new) ----
    def synthesize_batch(self, inputs: Sequence[str], voices: Optional[Sequence[str]] = None, fixed_frames: Optional[int] = None) -> List[np.ndarray]:
        voices = list(voices) if voices is not None else ["heart"] * len(inputs)
        prompts = [self._get_prompt(t, v)[0] for t, v in zip(inputs, voices)]
        codes = generate_batch(self.lm, prompts, self.settings, fixed_frames=fixed_frames)   # list of [N, T_b]
        return self.decode_codes(codes)

    def serve(self, inputs: Sequence[str], voices: Optional[Sequence[str]] = None, slots: int = 8, chunk: int = 16,
              max_prompt: int = 512) -> Iterator[tuple]:
        """Continuous batching with audio out (replaces the one-blocking-call-per-request loop of server/tts_core.py:28-47):
        the utterances share ``slots`` rows of one resident decode batch (``ContinuousBatcher``); whatever retires at a chunk
        boundary goes through the codec together, as one batch of streams.  Yields ``(index, pcm)`` in retirement order."""
        from .serving import ContinuousBatcher

        voices = list(voices) if voices is not None else ["heart"] * len(inputs)
        cb = ContinuousBatcher(self.lm, self.settings, slots=slots, max_prompt=max_prompt, chunk=chunk)
        try:
            uid_to_index = {cb.submit(self._get_prompt(t, v)[0]): i for i, (t, v) in enumerate(zip(inputs, voices))}
            while cb.pending or cb.running:
                done = cb.step_chunk()
                for g0 in range(0, len(done), self.codec_full.max_streams):
                    group = done[g0:g0 + self.codec_full.max_streams]
                    for (uid, _), pcm in zip(group, self.decode_codes([c for _, c in group])):
                        yield uid_to_index[uid], pcm
        finally:
            cb.close()

    def serve_stream(self, inputs: Sequence[str], voices: Optional[Sequence[str]] = None, slots: int = 8, chunk: int = 16,
                     max_prompt: int = 512) -> Iterator[tuple]:
        """``serve`` with audio as it is generated: every utterance in a decode slot owns a codec stream, and after each chunk
        of ``chunk`` frames the new frames of all running utterances go through the codec together.  Yields ``(index, pcm of
        the chunk, done)``; the chunks of an utterance concatenate to what ``serve`` / ``synthesize_batch`` return for it."""
        from .serving import ContinuousBatcher

        codec = self.codec_full
        if slots > codec.max_streams:
            raise ValueError(f"serve_stream: {slots} slots, the codec was built for {codec.max_streams} streams")
        voices = list(voices) if voices is not None else ["heart"] * len(inputs)
        cb = ContinuousBatcher(self.lm, self.settings, slots=slots, max_prompt=max_prompt, chunk=chunk)
        caches: dict = {}
        try:
            uid_to_index = {cb.submit(self._get_prompt(t, v)[0]): i for i, (t, v) in enumerate(zip(inputs, voices))}
            while cb.pending or cb.running:
                items = cb.step_chunk_stream()
                live = [(uid, codes) for uid, codes, _ in items if codes.shape[-1] > 0]
                for uid, _ in live:
                    if uid not in caches:
                        caches[uid] = codec.make_cache()
                pcms = dict(zip((u for u, _ in live), self.decode_codes([c for _, c in live], [caches[u] for u, _ in live]))) if live else {}
                for uid, codes, done in items:
                    if done and uid in caches:
                        codec.release_cache(caches.pop(uid))
                    yield uid_to_index[uid], pcms.get(uid, np.zeros(0, dtype=np.float32)), done
        finally:
            for c in caches.values():
                codec.release_cache(c)
            cb.close()

    def decode_codes(self, codes: Sequence[torch.Tensor], caches: Optional[Sequence] = None) -> List[np.ndarray]:
        """Ragged code sequences [N, T_b] -> PCM, all streams stepping together while they last (fresh codec streams, or the
        given ones continued)."""
        codec = self.codec_full
        B = len(codes)
        if B > codec.max_streams:
            raise ValueError(f"decode_codes: {B} utterances, the codec was built for {codec.max_streams} streams")
        lens = [int(c.shape[-1]) for c in codes]
        own = caches is None
        caches = [codec.make_cache() for _ in range(B)] if own else list(caches)
        spf = codec.samples_per_frame
        t_max = max(lens) if lens else 0
        order = sorted(range(B), key=lambda b: -lens[b])          # live streams are always a prefix of this order
        n_q = codec.num_codebooks
        grid = torch.zeros(B, n_q, max(t_max, 1), dtype=torch.int32, device=codec.device)   # one padded tensor: one slice per step
        for i, b in enumerate(order):
            if lens[b]:
                grid[i, :, : lens[b]] = codes[b].to(device=codec.device, dtype=torch.int32)
        pcm_all = torch.empty(B, max(t_max, 1) * spf, dtype=torch.float32, device=codec.device)
        sorted_caches = [caches[b] for b in order]
        n_live = B
        for t in range(t_max):
            while n_live > 0 and lens[order[n_live - 1]] <= t:
                n_live -= 1
            pcm = codec.decode_step(grid[:n_live, :, t], sorted_caches[:n_live])
            pcm_all[:n_live, t * spf:(t + 1) * spf] = pcm[:, 0]
        outs = [None] * B
        for i, b in enumerate(order):
            outs[b] = pcm_all[i, : lens[b] * spf]
        if own:
            for c in caches:
                codec.release_cache(c)
        return [o.cpu().numpy() for o in outs]
