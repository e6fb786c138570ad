"""Text -> PCM: the reference's ``SmolTTS`` front object (mlx_inference/src/smoltts_mlx/__init__.py:25-151) over the two
B200 engines -- the DualAR decode step (``RQTransformer``) and the Mimi streaming decoder (``MimiModel``).

Same call surface: ``SmolTTS(...)(text, voice)`` returns the flattened PCM of one utterance (:64-83), ``stream(text,
voice)`` yields one 80 ms chunk per generated frame (:85-95: a fresh Mimi cache per utterance, ``decode_step`` on the
frame's codes).  ``synthesize_batch`` is new: B utterances decode together (``generate_batch``), then their frames go
through the codec as one batch of B streams per step.

Parity note: the reference's ``__call__`` decodes the whole code sequence with ``codec.decode`` (the upsampler sees the
sequence) while its ``stream`` upsamples every frame alone (codec/mimi.py:73-104): the two give different audio in the
reference, and so do they here -- ``__call__`` uses a codec stream with the upsampler's carry, ``stream`` one without.

Rates (new): the codec works at 24 kHz mono.  ``SmolTTS(..., output_rate=r)`` converts every entry point's PCM to ``r`` on the
GPU (``resample.Resampler``), and ``create_speaker`` takes reference audio at any supported rate, mono or multi-channel.
"""
from __future__ import annotations

import dataclasses
from typing import Dict, Iterator, List, Optional, Sequence

import numpy as np
import torch

from .generate import GenerationSettings, SingleBatchGenerator, generate_batch, generate_blocking
from .mimi import MimiModel
from .model import RQTransformer
from .resample import Resampler
from .serving import PromptEncoder

CODEC_RATE = 24_000   # Mimi's sampling rate
VOICES = ["heart", "bella", "nova", "sky", "sarah", "michael", "fenrir", "liam", "emma", "isabella", "fable"]   # :127-143


class SmolTTS:
    def __init__(self, lm: RQTransformer, prompt_encoder: PromptEncoder, codec_stream: MimiModel, codec_full: Optional[MimiModel] = None,
                 settings: Optional[GenerationSettings] = None, output_rate: Optional[int] = None):
        """codec_stream: a MimiModel with the reference's decode_step rule (upsample_carry=False); codec_full: one with
        upsample_carry=True for ``__call__`` / ``synthesize_batch`` (defaults to codec_stream if it already carries).

        output_rate: the sampling rate of the PCM every entry point returns.  None or 24 000 is the codec's own rate: nothing
        is resampled and no resampler is built.  Any other rate (``max(up, down) <= 320`` against 24 kHz: 8, 11.025, 16,
        22.05, 32, 44.1, 48, 88.2, 96, 176.4, 192 kHz ...) converts on the GPU: whole utterances in one launch per codec call (per 256 streams),
        streams a frame at a time; ``stream``'s first chunk is shorter by the filter's look-ahead, and its last chunk is the
        filter's tail."""
        self.lm = lm
        self.prompt_encoder = prompt_encoder
        self.codec = codec_stream
        self.codec_full = codec_full if codec_full is not None else codec_stream
        self.settings = settings or GenerationSettings()
        self.sampling_rate = CODEC_RATE
        self.resampler: Optional[Resampler] = None
        if output_rate is not None and int(output_rate) != CODEC_RATE:
            # a resampler stream runs beside each codec stream; whole utterances take free slots for the length of one call
            streams = self.codec.max_streams + (self.codec_full.max_streams if self.codec_full is not self.codec else 0)
            self.resampler = Resampler(CODEC_RATE, int(output_rate), max_streams=streams, device=self.codec.device)
            self.sampling_rate = int(output_rate)
        self._input_resamplers: Dict[int, Resampler] = {}

    # ---- prompt assembly (:123-151) ----
    def _get_prompt(self, input: str, voice: str, sysprompt: Optional[torch.Tensor] = None) -> torch.Tensor:
        voice_id = VOICES.index(voice) if voice in VOICES else 0
        return self.prompt_encoder.tts_prompt(input, speaker=voice_id, sysprompt=sysprompt)[None]

    def create_speaker(self, samples: Sequence[dict], system_prompt: Optional[str] = None) -> torch.Tensor:
        """Voice-clone prefix (__init__.py:97-118) from ``{"text", "audio"}`` samples -- 1-D float PCM at 24 kHz, mono -- or
        ``{"text", "codes"}`` samples with ready-made Mimi codes.  The audio of all samples is encoded in one
        ``MimiModel.encode`` call (the codec must have been built with ``encode_max_samples > 0``).

        A sample with ``"sampling_rate"`` may carry audio at that rate, 1-D ``[L]`` or ``[C, L]``: the channels are averaged on
        the device and the clips of each rate resampled to 24 kHz together (one launch per 256 clips) before the encode."""
        samples = list(samples)
        with_audio = [i for i, s in enumerate(samples) if "audio" in s and "codes" not in s]
        if with_audio:
            codec = next((c for c in (self.codec, self.codec_full) if c._enc is not None), None)
            if codec is None:
                raise ValueError("create_speaker: samples carry 'audio' but the codec has no encoder "
                                 "(build the MimiModel with encode_max_samples > 0, or pass 'codes')")
            clips, by_rate = [], {}
            for k, i in enumerate(with_audio):
                s = samples[i]
                if "sampling_rate" not in s:
                    clips.append(torch.as_tensor(s["audio"], dtype=torch.float32).reshape(-1))
                    continue
                a = torch.as_tensor(s["audio"]).to(device=codec.device, dtype=torch.float32)
                if a.dim() not in (1, 2) or (a.dim() == 2 and a.shape[0] > a.shape[1]):
                    raise ValueError(f"create_speaker: audio of shape {tuple(a.shape)}; expected [L] or [channels, L] "
                                     "(channels first: transpose [L, channels] audio)")
                clips.append(a.mean(dim=0) if a.dim() == 2 else a)
                if int(s["sampling_rate"]) != CODEC_RATE:
                    by_rate.setdefault(int(s["sampling_rate"]), []).append(k)
            for rate, ks in by_rate.items():
                if rate not in self._input_resamplers:
                    self._input_resamplers[rate] = Resampler(rate, CODEC_RATE, max_streams=codec.encode_max_clips, device=codec.device)
                for k, y in zip(ks, self._input_resamplers[rate].resample([clips[k] for k in ks])):
                    clips[k] = y
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
        pcm = self.codec_full.decode(codes.to(torch.int64)).flatten()
        if self.resampler is not None:
            pcm = self.resampler.resample([pcm])[0]
        return pcm.cpu().numpy()

    # ---- streaming (:85-95) ----
    def stream(self, input: str, voice: Optional[str] = "heart", overlap: bool = True, lm_ctas: int = 96,
               stats: Optional[dict] = None) -> Iterator[np.ndarray]:
        """One 80 ms PCM chunk per generated audio frame.  ``overlap=False`` is the reference's loop as written: one frame per
        ``SingleBatchGenerator.__next__`` (launch, host read-back), then the codec step, then the chunk.  ``overlap`` (default)
        keeps both engines busy: the decode step of frame t + 1 is launched BEFORE the host looks at frame t, and frame t's ids,
        its codec step and its PCM go through a side stream -- the data-flow kernel is told to take ``lm_ctas`` of the GPU's SMs (a
        bs=1 frame takes the same 600-612 us on 96 .. 148 CTAs, DESIGN.md section 4), the codec's kernels run on the others.
        Throughput is then bound by the slower engine instead of the sum plus the host's time per frame.  Same chunks, bit for bit.

        With an ``output_rate``, each frame's PCM goes through a resampler stream right after its codec step (on the side stream
        in overlap mode) and the filter's tail follows the last frame as one more chunk."""
        prompt = self._get_prompt(input, voice if voice is not None else "0")
        codec = self.codec
        cache = codec.make_cache()
        rs = self.resampler
        rstate = None

        def pcm_out(pcm: torch.Tensor) -> np.ndarray:
            return (pcm if rstate is None else rs.step([pcm], [rstate])[0]).cpu().numpy()
        n_frames = n_audio = 0
        old_ctas = None
        batch = None
        try:
            if rs is not None:
                rstate = rs.make_state()
            if not overlap:
                for frame in SingleBatchGenerator(self.lm, prompt, self.settings):
                    n_frames += 1
                    if frame.audio_codes is None:      # the <|im_end|> frame (the reference would hand None to the codec here)
                        continue
                    if cache.frames >= codec.max_frames:
                        break
                    n_audio += 1
                    yield pcm_out(codec.decode_step(frame.audio_codes, cache).flatten())
                if rstate is not None and n_audio:
                    yield rs.finish([rstate])[0].cpu().numpy()
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
                        out = pcm_out(codec.decode_step(codes.view(1, -1, 1), cache).flatten())
                        n_audio += 1
                if out is not None:
                    yield out
                if slow == tc.im_end_id or (lo <= slow <= hi and out is None):
                    break
            if rstate is not None and n_audio:
                with torch.cuda.stream(side):
                    tail = rs.finish([rstate])[0].cpu().numpy()
                yield tail
        finally:
            torch.cuda.synchronize(codec.device)
            codec.release_cache(cache)
            if rstate is not None:
                rs.release_state(rstate)
            if batch is not None:
                batch.release()
            if old_ctas is not None:
                self.lm.set_option("n_ctas", old_ctas)
            if stats is not None:
                stats["frames"], stats["audio_frames"] = n_frames, n_audio

    # ---- many utterances at once (new) ----
    def _batcher(self, n_inputs: int, settings: Optional[Sequence[GenerationSettings]], slots: int, chunk: int, max_prompt: int):
        """A ContinuousBatcher for ``serve`` / ``serve_stream`` and each input's settings (None: this object's).  With a
        settings list the batcher's frame budget is the largest of the list, so that no input's own budget is cut."""
        from .serving import ContinuousBatcher

        if settings is None:
            return ContinuousBatcher(self.lm, self.settings, slots=slots, max_prompt=max_prompt, chunk=chunk), [None] * n_inputs
        settings = list(settings)
        if len(settings) != n_inputs:
            raise ValueError(f"{len(settings)} settings for {n_inputs} inputs")
        base = dataclasses.replace(self.settings, max_new_tokens=max(s.max_new_tokens for s in settings))
        return ContinuousBatcher(self.lm, base, slots=slots, max_prompt=max_prompt, chunk=chunk), settings

    def synthesize_batch(self, inputs: Sequence[str], voices: Optional[Sequence[str]] = None, fixed_frames: Optional[int] = None,
                         settings: Optional[Sequence[GenerationSettings]] = None) -> List[np.ndarray]:
        """``settings``: one ``GenerationSettings`` per input (sampling parameters, seed and frame budget), or None for this
        object's settings."""
        voices = list(voices) if voices is not None else ["heart"] * len(inputs)
        prompts = [self._get_prompt(t, v)[0] for t, v in zip(inputs, voices)]
        codes = generate_batch(self.lm, prompts, self.settings if settings is None else list(settings),
                               fixed_frames=fixed_frames)   # list of [N, T_b]
        return self.decode_codes(codes)

    def serve(self, inputs: Sequence[str], voices: Optional[Sequence[str]] = None, slots: int = 8, chunk: int = 16,
              max_prompt: int = 512, settings: Optional[Sequence[GenerationSettings]] = None) -> Iterator[tuple]:
        """Continuous batching with audio out (replaces the one-blocking-call-per-request loop of server/tts_core.py:28-47):
        the utterances share ``slots`` rows of one resident decode batch (``ContinuousBatcher``); whatever retires at a chunk
        boundary goes through the codec together, as one batch of streams.  Yields ``(index, pcm)`` in retirement order.
        ``settings``: one ``GenerationSettings`` per input, as in ``synthesize_batch``."""
        voices = list(voices) if voices is not None else ["heart"] * len(inputs)
        cb, per_input = self._batcher(len(inputs), settings, slots, chunk, max_prompt)
        try:
            uid_to_index = {cb.submit(self._get_prompt(t, v)[0], settings=per_input[i]): i
                            for i, (t, v) in enumerate(zip(inputs, voices))}
            while cb.pending or cb.running:
                done = cb.step_chunk()
                for g0 in range(0, len(done), self.codec_full.max_streams):
                    group = done[g0:g0 + self.codec_full.max_streams]
                    for (uid, _), pcm in zip(group, self.decode_codes([c for _, c in group])):
                        yield uid_to_index[uid], pcm
        finally:
            cb.close()

    def serve_stream(self, inputs: Sequence[str], voices: Optional[Sequence[str]] = None, slots: int = 8, chunk: int = 16,
                     max_prompt: int = 512, settings: Optional[Sequence[GenerationSettings]] = None) -> Iterator[tuple]:
        """``serve`` with audio as it is generated: every utterance in a decode slot owns a codec stream, and after each chunk
        of ``chunk`` frames the new frames of all running utterances go through the codec together.  Yields ``(index, pcm of
        the chunk, done)``; the chunks of an utterance concatenate to what ``serve`` / ``synthesize_batch`` return for it."""
        codec, rs = self.codec_full, self.resampler
        if slots > codec.max_streams:
            raise ValueError(f"serve_stream: {slots} slots, the codec was built for {codec.max_streams} streams")
        voices = list(voices) if voices is not None else ["heart"] * len(inputs)
        cb, per_input = self._batcher(len(inputs), settings, slots, chunk, max_prompt)
        caches: dict = {}
        rstates: dict = {}   # with an output_rate: one resampler stream per live utterance, next to its codec stream
        try:
            uid_to_index = {cb.submit(self._get_prompt(t, v)[0], settings=per_input[i]): i
                            for i, (t, v) in enumerate(zip(inputs, voices))}
            while cb.pending or cb.running:
                items = cb.step_chunk_stream()
                live = [(uid, codes) for uid, codes, _ in items if codes.shape[-1] > 0]
                for uid, _ in live:
                    if uid not in caches:
                        caches[uid] = codec.make_cache()
                        if rs is not None:
                            rstates[uid] = rs.make_state()
                uids = [u for u, _ in live]
                pcms = dict(zip(uids, self._decode_pcm([c for _, c in live], [caches[u] for u in uids]))) if live else {}
                if rs is not None:
                    pcms = dict(zip(uids, rs.step([pcms[u] for u in uids], [rstates[u] for u in uids])))
                    ended = [uid for uid, _, done in items if done and uid in rstates]
                    for uid, tail in zip(ended, rs.finish([rstates[u] for u in ended])):
                        pcms[uid] = torch.cat([pcms[uid], tail]) if uid in pcms else tail
                for uid, codes, done in items:
                    if done and uid in caches:
                        codec.release_cache(caches.pop(uid))
                        if rs is not None:
                            rs.release_state(rstates.pop(uid))
                    yield uid_to_index[uid], pcms[uid].cpu().numpy() if uid in pcms else np.zeros(0, dtype=np.float32), done
        finally:
            for c in caches.values():
                codec.release_cache(c)
            for st in rstates.values():
                rs.release_state(st)
            cb.close()

    def decode_codes(self, codes: Sequence[torch.Tensor], caches: Optional[Sequence] = None) -> List[np.ndarray]:
        """Ragged code sequences [N, T_b] -> PCM, all streams stepping together while they last (fresh codec streams, or the
        given ones continued).  With an ``output_rate`` the utterances (fresh streams only) are resampled together, in one
        launch."""
        if self.resampler is not None and caches is not None:
            raise ValueError("decode_codes: continued codec streams come out at 24 kHz; serve_stream resamples them as streams")
        outs = self._decode_pcm(codes, caches)
        if self.resampler is not None and outs:
            outs = self.resampler.resample(outs)
        return [o.cpu().numpy() for o in outs]

    def _decode_pcm(self, codes: Sequence[torch.Tensor], caches: Optional[Sequence] = None) -> List[torch.Tensor]:
        """``decode_codes`` at the codec's rate, as device tensors."""
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
        return outs
