"""Front end of the decode path (SURVEY §8(f)-3): prompt encoding and continuous batching.

``PromptEncoder`` mirrors the reference's encoder (mlx_inference/src/smoltts_mlx/lm/utils/prompt.py:10-63) and the
prompt assembly of ``SmolTTS`` (mlx_inference/src/smoltts_mlx/__init__.py:97-151) on torch int64 grids ``[1+N', S]``;
``byte_level_tokenizer`` rebuilds the byte tokenizer of the reference recipe
(data_pipeline/scripts/create_bytelevel_init.py:15-57) in memory, because a checkpoint's ``tokenizer.json`` is the only
thing the reference fetches from the network for this step.

``ContinuousBatcher`` replaces the reference's serving loop -- one blocking ``generate_blocking`` per request, bs=1
(mlx_inference/src/smoltts_mlx/server/tts_core.py:28-47) -- with a slot scheduler over ONE resident decode batch:
utterances are admitted into free slots and retired at frame-chunk boundaries, the stop rule and the frame counters live
on the device (``SmolBatch.finished`` / ``step``), and KV pages are handed out per utterance and recycled on retirement.
The decode arithmetic does not depend on which sequences share a launch (tested bit for bit), and sampling is keyed by
(utterance id, frame), so an utterance decodes to the same codes whatever the scheduler did around it.  Every request may
carry its own ``GenerationSettings``: its sampling parameters go into a resident per-slot table (``SmolBatch.row_sampling``).
"""
from __future__ import annotations

import collections
import ctypes as C
from dataclasses import dataclass
from typing import Deque, Dict, Iterator, List, Optional, Sequence, Tuple

import torch

from . import _capi
from .generate import GenerationSettings, _sampling, row_sampling_table
from .model import RQTransformer


# --------------------------------------------------------------------------------------------------------------------
# prompt encoding
# --------------------------------------------------------------------------------------------------------------------
_CONTROL_TOKENS = ("system", "user", "assistant", "<|british|>", "<|american|>", "<|male|>", "<|female|>", "<|unknown|>",
                   "<|endoftext|>", "<|voice|>", "<|semantic|>", "<|pad|>", "<|epad|>", "<|im_start|>", "<|im_end|>")


def byte_level_tokenizer(codebook_size: int = 2048):
    """The byte-level tokenizer of the reference recipe, built in memory: ids 0..255 are the latin-1 code points, then the 15
    control tokens, 49 speaker tokens (64 specials in all) and ``codebook_size`` semantic tokens -- 2368 ids for the shipped
    configs, ``<|im_end|>`` = 270, ``<|semantic:0|>`` = 320."""
    from tokenizers import Tokenizer, decoders, models
    from tokenizers.trainers import BpeTrainer

    tok = Tokenizer(models.BPE())
    tok.train_from_iterator([chr(i) for i in range(256)], trainer=BpeTrainer(vocab_size=256, special_tokens=[]))
    tok.pre_tokenizer = None
    tok.normalizer = None
    tok.decoder = decoders.ByteLevel()
    specials = list(_CONTROL_TOKENS)
    specials += [f"<|speaker:{i}|>" for i in range(64 - len(_CONTROL_TOKENS))]
    specials += [f"<|semantic:{i}|>" for i in range(codebook_size)]
    tok.add_special_tokens(specials)
    return tok


class PromptEncoder:
    """Token grids of the DualAR prompt format: row 0 carries text ids (or ``semantic_offset + code`` on audio columns), rows
    1.. the Mimi codebook ids (zeros on text columns).  Reference: lm/utils/prompt.py:10-63."""

    def __init__(self, tokenizer, semantic_offset: int, num_codebooks: int = 8, duplicate_code_0: bool = True):
        self.tokenizer = tokenizer
        self.depth = num_codebooks if duplicate_code_0 else num_codebooks - 1
        self.semantic_offset = semantic_offset

    @classmethod
    def from_model(cls, tokenizer, model: RQTransformer) -> "PromptEncoder":
        dc0 = model.config.duplicate_code_0
        return cls(tokenizer, semantic_offset=model.token_config.semantic_start_id, num_codebooks=model.config.num_codebooks,
                   duplicate_code_0=True if dc0 is None else bool(dc0))

    def tokenize_text(self, text: str) -> torch.Tensor:
        ids = self.tokenizer.encode(text, add_special_tokens=True).ids
        grid = torch.zeros(1 + self.depth, len(ids), dtype=torch.int64)
        grid[0] = torch.tensor(ids, dtype=torch.int64)
        return grid

    def encode_text_turn(self, role: str, content: Optional[str] = None) -> torch.Tensor:
        """``<|im_start|>role\\ncontent<|im_end|>``; without content the open turn the model continues."""
        suffix = f"{content}<|im_end|>" if content is not None else ""
        return self.tokenize_text(f"<|im_start|>{role}\n{suffix}")

    def encode_vq(self, codes: torch.Tensor) -> torch.Tensor:
        """Mimi codes ``[N, T]`` of a spoken turn -> audio columns followed by ``<|im_end|>\\n``."""
        if codes.ndim != 2:
            raise ValueError("Must be single batch")
        codes = codes.to(torch.int64)
        semantic = codes[0:1] + self.semantic_offset
        lower = codes[codes.shape[0] - self.depth:]
        return torch.cat([torch.cat([semantic, lower], dim=0), self.tokenize_text("<|im_end|>\n")], dim=1)

    # ---- prompt assembly of SmolTTS (smoltts_mlx/__init__.py:97-151) ----
    def create_speaker(self, samples: Sequence[dict], system_prompt: Optional[str] = None) -> torch.Tensor:
        """Voice-clone prefix from ``{"text": str, "codes": [N, T] Mimi codes}`` samples (the reference encodes ``"audio"``
        with the Mimi codec here; the codec is outside this path, so the codes come in ready-made)."""
        turns: List[torch.Tensor] = []
        for s in samples:
            if "codes" not in s or "text" not in s:
                raise ValueError(f"Sample must contain both 'text' and 'codes' but got {s.keys()}")
            turns.append(self.encode_text_turn("user", s["text"]))
            turns.append(self.encode_vq(torch.as_tensor(s["codes"])[:8]))
        if system_prompt is not None:
            turns.insert(0, self.encode_text_turn("system", system_prompt))
        return torch.cat(turns, dim=1)

    def tts_prompt(self, text: str, speaker: int = 0, sysprompt: Optional[torch.Tensor] = None) -> torch.Tensor:
        """system turn (``<|speaker:k|>`` or a ``create_speaker`` prefix) + user turn + open assistant turn."""
        if sysprompt is None:
            sysprompt = self.encode_text_turn("system", f"<|speaker:{speaker}|>")
        return torch.cat([sysprompt, self.encode_text_turn("user", text), self.encode_text_turn("assistant")], dim=1)


# --------------------------------------------------------------------------------------------------------------------
# continuous batching
# --------------------------------------------------------------------------------------------------------------------
@dataclass
class _Request:
    uid: int
    prompt: torch.Tensor     # [R, S] int32 (host)
    budget: int              # frames this utterance may emit (max_new_tokens + 1, as the reference loop)
    sampling: torch.Tensor   # [1, 32] uint8 (host): its SmolRowSampling record


@dataclass
class _Slot:
    uid: int
    budget: int
    pages: List[int]
    emitted: int = 0         # frames already handed out by step_chunk_stream


class ContinuousBatcher:
    """``slots`` sequences decode together; a finished one makes room for the next request at the next chunk boundary.

    * the batch is ONE ``SmolBatch`` of ``slots`` rows that stays resident; free rows carry ``finished = 1`` (the kernels
      skip their KV appends and freeze their counters);
    * admission: pages for ``prompt + budget + chunk`` positions come from the model's page pool, the row's counters are
      reset, and the new rows are prefilled through a VIEW of the batch (contiguous runs of new slots) so that running
      sequences are not touched and a single new utterance still gets the whole prompt in one pass over the weights;
    * every ``chunk`` frames the host reads ``finished`` and ``step`` (5 bytes per slot), retires rows whose stop rule fired or
      whose frame budget is spent, copies their codes and returns their pages to the pool.

    ``submit`` returns the utterance id that also seeds the sampler (``seq_id``), so results do not depend on arrival order;
    its ``settings`` (default: the batcher's) choose the utterance's temperatures, top-k / top-p / min-p, seed and frame budget.
    The batcher's settings also fix the largest budget; ``audio_only`` / ``ignore_stop`` hold for every utterance.
    """

    def __init__(self, model: RQTransformer, settings: GenerationSettings, slots: int, max_prompt: int = 512,
                 chunk: int = 16, audio_only: bool = True, ignore_stop: bool = False):
        if slots < 1 or slots > model.max_batch:
            raise ValueError(f"slots must be in [1, max_batch = {model.max_batch}]")
        self.model, self.settings, self.slots, self.chunk = model, settings, slots, chunk
        self.audio_only = audio_only
        self.max_frames = settings.max_new_tokens + 1
        self.max_positions = max_prompt + self.max_frames + chunk
        if self.max_positions > model.max_seq_len:
            raise ValueError(f"max_prompt + frames + chunk = {self.max_positions} positions exceed max_seq_len {model.max_seq_len}")
        dev, R, ps = model.device, model.config.n_rows, model.page_size
        self.max_pages = (self.max_positions + ps - 1) // ps
        self._scratch = model.allocate_pages(1)          # where the block table of an idle row points
        self.tokens = torch.zeros(slots, R, dtype=torch.int32, device=dev)
        self.seq_len = torch.zeros(slots, dtype=torch.int32, device=dev)
        self.block_table = torch.full((slots, self.max_pages), self._scratch[0], dtype=torch.int32, device=dev)
        self.finished = torch.ones(slots, dtype=torch.uint8, device=dev)
        self.seq_id = torch.zeros(slots, dtype=torch.int32, device=dev)
        self.step = torch.zeros(slots, dtype=torch.int32, device=dev)
        self._out_rows = self.max_frames + chunk
        self.out_codes = torch.zeros(slots, self._out_rows, R, dtype=torch.int32, device=dev)
        self.row_sampling = model.row_sampling([settings] * slots)   # [slots, 32]: rewritten for a slot at its admission
        self._default_sampling = row_sampling_table([settings])
        self.c = self._view(0)
        self.sampling = _sampling(model, settings, audio_only, ignore_stop=ignore_stop)
        self._queue: Deque[_Request] = collections.deque()
        self._active: List[Optional[_Slot]] = [None] * slots
        self._next_uid = 0
        self.stats = {"frames_decoded": 0, "slot_frames": 0, "chunks": 0, "admitted": 0, "retired": 0}

    # ---- plumbing ----
    def _view(self, b0: int) -> _capi.SmolBatch:
        """SmolBatch whose row 0 is slot ``b0`` (every field is a per-row array: offset the pointers)."""
        R = self.model.config.n_rows
        return _capi.SmolBatch(
            tokens=self.tokens.data_ptr() + 4 * b0 * R, seq_len=self.seq_len.data_ptr() + 4 * b0,
            block_table=self.block_table.data_ptr() + 4 * b0 * self.max_pages, max_pages=self.max_pages,
            finished=self.finished.data_ptr() + b0, seq_id=self.seq_id.data_ptr() + 4 * b0, step=self.step.data_ptr() + 4 * b0,
            out_codes=self.out_codes.data_ptr() + 4 * b0 * self._out_rows * R, max_frames=self._out_rows,
            row_sampling=self.row_sampling.data_ptr() + self.row_sampling.shape[1] * b0)

    def close(self) -> None:
        for s in self._active:
            if s is not None:
                self.model.free_pages(s.pages)
        self._active = [None] * self.slots
        if self._scratch:
            self.model.free_pages(self._scratch)
            self._scratch = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---- public surface ----
    def submit(self, prompt: torch.Tensor, max_new_tokens: Optional[int] = None, uid: Optional[int] = None,
               settings: Optional[GenerationSettings] = None) -> int:
        """Queue one utterance (token grid ``[1+N', S]`` or ``[1, 1+N', S]``); returns its id.  ``settings`` (None: the
        batcher's) sample this utterance; its frame budget is ``max_new_tokens``, else ``settings.max_new_tokens``, plus one,
        capped by the batcher's."""
        p = prompt if prompt.ndim == 2 else prompt[0]
        R = self.model.config.n_rows
        if p.shape[0] != R:
            raise ValueError(f"prompt has {p.shape[0]} rows, model expects {R}")
        sampling = self._default_sampling if settings is None else row_sampling_table([settings])
        if max_new_tokens is None and settings is not None:
            max_new_tokens = settings.max_new_tokens
        budget = self.max_frames if max_new_tokens is None else min(max_new_tokens + 1, self.max_frames)
        if p.shape[1] < 2 or p.shape[1] + budget + self.chunk > self.max_positions:
            raise ValueError(f"prompt of {p.shape[1]} columns does not fit the batcher (max_prompt / max_new_tokens)")
        if uid is None:
            uid = self._next_uid
        self._next_uid = max(self._next_uid, uid) + 1
        self._queue.append(_Request(uid, p.to(torch.int32).cpu().contiguous(), budget, sampling))
        return uid

    @property
    def pending(self) -> int:
        return len(self._queue)

    @property
    def running(self) -> int:
        return sum(s is not None for s in self._active)

    def _admit(self) -> None:
        new: List[Tuple[int, _Request]] = []
        ps = self.model.page_size
        for b in range(self.slots):
            if not self._queue:
                break
            if self._active[b] is not None:
                continue
            req = self._queue[0]
            need = (req.prompt.shape[1] + req.budget + self.chunk + ps - 1) // ps
            try:
                pages = self.model.allocate_pages(need)
            except _capi.SmolError:
                break                                   # pool exhausted: wait for a retirement
            self._queue.popleft()
            self._active[b] = _Slot(req.uid, req.budget, pages)
            new.append((b, req))
        if not new:
            return
        dev = self.model.device
        idx = torch.tensor([b for b, _ in new], device=dev)
        rows = torch.full((len(new), self.max_pages), self._scratch[0], dtype=torch.int32)
        for i, (b, _) in enumerate(new):
            pg = self._active[b].pages
            rows[i, : len(pg)] = torch.tensor(pg, dtype=torch.int32)
        self.block_table[idx] = rows.to(dev)
        self.seq_len[idx] = 0
        self.step[idx] = 0
        self.finished[idx] = 0
        self.seq_id[idx] = torch.tensor([r.uid for _, r in new], dtype=torch.int32, device=dev)
        self.row_sampling[idx] = torch.cat([r.sampling for _, r in new]).to(dev)
        # prefill the new rows, one call per contiguous run of slots (rows = the run only: every other sequence is untouched)
        i = 0
        R = self.model.config.n_rows
        while i < len(new):
            j = i
            while j + 1 < len(new) and new[j + 1][0] == new[j][0] + 1:
                j += 1
            run = new[i:j + 1]
            s_max = max(r.prompt.shape[1] for _, r in run)
            grid = torch.zeros(len(run), R, s_max, dtype=torch.int32, pin_memory=True)
            for k, (_, r) in enumerate(run):
                grid[k, :, : r.prompt.shape[1]] = r.prompt
            lens = torch.tensor([r.prompt.shape[1] for _, r in run], dtype=torch.int32, pin_memory=True)
            d_grid, d_lens = grid.to(dev, non_blocking=True), lens.to(dev, non_blocking=True)
            view = self._view(run[0][0])
            _capi.check(self.model.lib.smol_prefill(self.model._h, C.byref(view), len(run), C.c_void_p(d_grid.data_ptr()),
                                                    C.c_void_p(d_lens.data_ptr()), s_max, self.model._stream()))
            i = j + 1
        self.stats["admitted"] += len(new)

    def _retire(self) -> List[Tuple[int, torch.Tensor]]:
        fin = self.finished.cpu().tolist()
        steps = self.step.cpu().tolist()
        done: List[Tuple[int, torch.Tensor]] = []
        gone: List[int] = []
        for b, slot in enumerate(self._active):
            if slot is None or not (fin[b] or steps[b] >= slot.budget):
                continue
            n = min(steps[b], slot.budget)
            done.append((slot.uid, self._postprocess(self.out_codes[b, :n].cpu())))
            self.model.free_pages(slot.pages)
            self._active[b] = None
            gone.append(b)
        if gone:
            idx = torch.tensor(gone, device=self.model.device)
            self.finished[idx] = 1
            self.block_table[idx] = self._scratch[0]
            self.stats["retired"] += len(gone)
        return done

    def _postprocess(self, frames: torch.Tensor) -> torch.Tensor:
        """[T, R] emitted columns -> what ``generate_batch`` returns for the utterance."""
        cols = frames.t().contiguous()
        if not self.audio_only:
            return cols
        tc, cfg = self.model.token_config, self.model.config
        lo, hi = tc.semantic_start_id, tc.semantic_end_id if tc.semantic_end_id is not None else -1
        keep = (cols[0] >= lo) & (cols[0] <= hi)
        if cfg.duplicate_code_0:
            return cols[1:, keep]
        return torch.cat([(cols[0:1, keep] - lo), cols[1:, keep]], dim=0)

    def step_chunk(self) -> List[Tuple[int, torch.Tensor]]:
        """Admit what fits, decode one chunk of frames for every running sequence, retire what finished."""
        self._admit()
        n_run = self.running
        if n_run == 0:
            return []
        _capi.check(self.model.lib.smol_decode_frames(self.model._h, C.byref(self.c), self.slots, C.byref(self.sampling),
                                                      self.chunk, self.model._stream()))
        self.stats["chunks"] += 1
        self.stats["slot_frames"] += self.slots * self.chunk
        done = self._retire()
        self.stats["frames_decoded"] += n_run * self.chunk
        return done

    def step_chunk_stream(self) -> List[Tuple[int, torch.Tensor, bool]]:
        """``step_chunk`` for streaming consumers: ``(uid, codes of the frames this utterance emitted in the chunk, done)`` for
        every sequence that ran -- the same columns ``step_chunk`` / ``run`` hand out at retirement, a chunk at a time."""
        self._admit()
        n_run = self.running
        if n_run == 0:
            return []
        _capi.check(self.model.lib.smol_decode_frames(self.model._h, C.byref(self.c), self.slots, C.byref(self.sampling),
                                                      self.chunk, self.model._stream()))
        self.stats["chunks"] += 1
        self.stats["slot_frames"] += self.slots * self.chunk
        self.stats["frames_decoded"] += n_run * self.chunk
        fin = self.finished.cpu().tolist()
        steps = self.step.cpu().tolist()
        out: List[Tuple[int, torch.Tensor, bool]] = []
        gone: List[int] = []
        for b, slot in enumerate(self._active):
            if slot is None:
                continue
            n = min(steps[b], slot.budget)
            done = bool(fin[b]) or steps[b] >= slot.budget
            out.append((slot.uid, self._postprocess(self.out_codes[b, slot.emitted:n].cpu()), done))
            slot.emitted = n
            if done:
                self.model.free_pages(slot.pages)
                self._active[b] = None
                gone.append(b)
        if gone:
            idx = torch.tensor(gone, device=self.model.device)
            self.finished[idx] = 1
            self.block_table[idx] = self._scratch[0]
            self.stats["retired"] += len(gone)
        return out

    def run(self) -> Iterator[Tuple[int, torch.Tensor]]:
        """Decode until the queue and the slots are empty; yields ``(uid, codes)`` as utterances retire."""
        while self._queue or self.running:
            for item in self.step_chunk():
                yield item

    def generate(self, prompts: Sequence[torch.Tensor], max_new_tokens: Optional[Sequence[Optional[int]]] = None) -> List[torch.Tensor]:
        """Convenience: submit every prompt, run to completion, return the codes in the callers' order."""
        uids = [self.submit(p, None if max_new_tokens is None else max_new_tokens[i]) for i, p in enumerate(prompts)]
        got: Dict[int, torch.Tensor] = dict(self.run())
        return [got[u] for u in uids]
