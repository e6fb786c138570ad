"""Host side of the DualAR decode engine: checkpoint loading and the model-level calls.

Mirrors the reference's surfaces for this path (SURVEY §8(b)):
  * ``RQTransformer.from_pretrained(path, load_weights, weight_override, max_length, rope_base)``
    -- reference modeling/model/rq_transformer.py:273-319 (state-dict keys, config, tokenizer ids);
  * ``forward_generate(inputs, cache) -> (token_logits, hidden)`` and
    ``forward_generate_fast(x, input_pos, cache) -> logits`` -- reference
    mlx_inference/src/smoltts_mlx/lm/rq_transformer.py:173-220;
  * ``make_prompt_cache(model, is_fast)`` -- reference mlx_inference/src/smoltts_mlx/lm/cache.py:25-33;
  * checkpoint layout of train/convert_safetensors.py:6-16 (flattened ``fast_output.weight``), also
    accepting the trainer's 3-D form and ``_orig_mod.`` prefixes.
torch is used for device memory and streams only; all arithmetic runs in the CUDA library
behind the C-ABI (``_capi``).  There is no CPU fallback: constructing a model without a CUDA
device raises.
"""
from __future__ import annotations

import ctypes as C
import json
import os
from dataclasses import dataclass
from pathlib import Path
from typing import Dict, List, Optional, Sequence, Tuple

import torch

from . import _capi
from .config import RQTransformerModelArgs
from .synth import TOK_IM_END, TOK_PAD, TOK_SEMANTIC0


@dataclass
class TokenConfig:
    """reference mlx lm/rq_transformer.py:51-89."""
    im_end_id: int
    pad_id: int
    semantic_start_id: int
    semantic_end_id: Optional[int]

    @classmethod
    def from_tokenizer_file(cls, path: str, config: RQTransformerModelArgs) -> "TokenConfig":
        from tokenizers import Tokenizer

        tok = Tokenizer.from_file(path)
        im_end = tok.token_to_id("<|im_end|>")
        if im_end is None:
            raise ValueError("Tokenizer does not have <|im_end|>")
        start = tok.token_to_id("<|semantic:0|>")
        end = tok.token_to_id(f"<|semantic:{config.codebook_size - 1}|>")
        if start is None or end is None or end - start != config.codebook_size - 1:
            # reference modeling/model/rq_transformer.py:140-144
            raise ValueError("Semantic tokens are not contiguous in the tokenizer")
        return cls(im_end_id=im_end, pad_id=tok.token_to_id("<|semantic|>") or 5,
                   semantic_start_id=start, semantic_end_id=end)

    @classmethod
    def byte_level_default(cls, config: RQTransformerModelArgs) -> "TokenConfig":
        """ids of the byte-level tokenizer recipe (data_pipeline/scripts/create_bytelevel_init.py:15-57)."""
        return cls(im_end_id=TOK_IM_END, pad_id=TOK_PAD, semantic_start_id=TOK_SEMANTIC0,
                   semantic_end_id=TOK_SEMANTIC0 + config.codebook_size - 1)


LL_REPLICAS = 8      # replicas of every word region (dev_model.h: kLLRep)
LL_PSUM_SLICES = 7   # K-slices of the fused MLP's partial sums (dev_model.h: kLL2Warps)


def ll_bf16(payload: torch.Tensor) -> torch.Tensor:
    """Payloads of bf16 words (int32 [n]) -> their 2n bf16 values, the low half of each word first (pack_bf16; both the
    device and the host are little-endian)."""
    return payload.contiguous().view(torch.bfloat16)


def precompute_freqs_cis(seq_len: int, n_elem: int, base: float) -> torch.Tensor:
    """[seq_len, n_elem/2, 2] (cos, sin) rounded to bf16 -- same op sequence as the reference
    (modeling/model/rq_transformer.py:616-624) so the table is bit-identical."""
    freqs = 1.0 / (base ** (torch.arange(0, n_elem, 2)[: (n_elem // 2)].float() / n_elem))
    t = torch.arange(seq_len)
    freqs = torch.outer(t, freqs)
    cis = torch.polar(torch.ones_like(freqs), freqs)
    return torch.stack([cis.real, cis.imag], dim=-1).to(torch.bfloat16)


def normalise_state_dict(sd: Dict[str, torch.Tensor], cfg: RQTransformerModelArgs) -> Dict[str, torch.Tensor]:
    """Checkpoint -> the exported layout: strips ``_orig_mod.`` (train/convert_safetensors.py:9),
    merges legacy wq/wk/wv (reference :528-533) and flattens a 3-D ``fast_output.weight`` to
    [(i*C + k), D] (convert_safetensors.py:12-15, without its hard-coded 768)."""
    out: Dict[str, torch.Tensor] = {}
    for k, v in sd.items():
        out[k.replace("_orig_mod.", "")] = v
    for k in [k for k in out if k.endswith("attention.wq.weight")]:
        pre = k[: -len("wq.weight")]
        out[pre + "wqkv.weight"] = torch.cat([out.pop(pre + "wq.weight"), out.pop(pre + "wk.weight"),
                                              out.pop(pre + "wv.weight")], dim=0)
    fo = out.get("fast_output.weight")
    if fo is not None and fo.ndim == 3:
        nf, d, c = fo.shape
        out["fast_output.weight"] = fo.permute(0, 2, 1).reshape(nf * c, d).contiguous()
    return out


def expected_shapes(cfg: RQTransformerModelArgs) -> Dict[str, Tuple[int, ...]]:
    from .synth import state_dict_shapes

    return state_dict_shapes(cfg, flat_fast_output=True)


class DecodeBatch:
    """Device-side state of B utterances in flight (what the reference keeps in Python:
    SingleBatchGenerator fields, mlx lm/generate.py:25-57, and KVCache.offset, lm/cache.py:10)."""

    def __init__(self, model: "RQTransformer", batch: int, max_positions: int, max_frames: int,
                 seq_ids: Optional[Sequence[int]] = None):
        dev = model.device
        self.model = model
        self.batch = batch
        self.max_frames = max_frames
        ps = model.page_size
        self.max_pages = (max_positions + ps - 1) // ps
        self.pages = model.allocate_pages(batch * self.max_pages)
        R = model.config.n_rows
        self.tokens = torch.zeros(batch, R, dtype=torch.int32, device=dev)
        self.seq_len = torch.zeros(batch, dtype=torch.int32, device=dev)
        self.block_table = torch.tensor(self.pages, dtype=torch.int32).view(batch, self.max_pages).to(dev)
        self.finished = torch.zeros(batch, dtype=torch.uint8, device=dev)
        ids = list(seq_ids) if seq_ids is not None else list(range(batch))
        self.seq_id = torch.tensor(ids, dtype=torch.int32, device=dev)
        self.step = torch.zeros(batch, dtype=torch.int32, device=dev)
        self.out_codes = torch.zeros(batch, max(max_frames, 1), R, dtype=torch.int32, device=dev)
        # positions this batch may cache: its pages, and never past the RoPE table (max_seq_len rows)
        self.capacity = min(self.max_pages * ps, model.max_seq_len)
        self.host_len = [0] * batch  # upper bound of seq_len known on the host (capacity checks)
        self.row_sampling: Optional[torch.Tensor] = None
        self.c = _capi.SmolBatch(
            tokens=self.tokens.data_ptr(), seq_len=self.seq_len.data_ptr(), block_table=self.block_table.data_ptr(),
            max_pages=self.max_pages, finished=self.finished.data_ptr(), seq_id=self.seq_id.data_ptr(),
            step=self.step.data_ptr(), out_codes=self.out_codes.data_ptr(), max_frames=max(max_frames, 1))

    def set_row_sampling(self, table: Optional[torch.Tensor]) -> None:
        """Per-sequence sampling parameters: ``table`` from ``RQTransformer.row_sampling`` (one record per sequence), read by
        every later decode call; None returns every sequence to the call's ``SmolSampling``.  The batch keeps the tensor
        alive; its contents may be rewritten in place between calls."""
        if table is not None:
            rec = C.sizeof(_capi.SmolRowSampling)
            if (table.dtype != torch.uint8 or tuple(table.shape) != (self.batch, rec) or table.device != self.model.device
                    or not table.is_contiguous()):
                raise ValueError(f"row sampling table must be a contiguous uint8 [{self.batch}, {rec}] tensor on {self.model.device}")
        self.row_sampling = table
        self.c.row_sampling = table.data_ptr() if table is not None else None

    def release(self) -> None:
        if self.pages:
            self.model.free_pages(self.pages)
            self.pages = []

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class RQTransformer:
    """B200 decode engine behind the reference's model surface."""

    def __init__(self, config: RQTransformerModelArgs, token_config: Optional[TokenConfig] = None,
                 device: Optional[torch.device] = None, max_batch: int = 8, max_seq_len: Optional[int] = None,
                 page_size: int = 32, kv_pages: Optional[int] = None, mlx_embed_mask: bool = False,
                 tokenizer=None):
        if not torch.cuda.is_available():
            raise RuntimeError("smoltts_b200 needs a CUDA device: there is no CPU fallback")
        self.lib = _capi.load()
        self.config = config
        self.tokenizer = tokenizer
        self.token_config = token_config or TokenConfig.byte_level_default(config)
        self.device = torch.device(device) if device is not None else torch.device("cuda", torch.cuda.current_device())
        self.max_batch = max_batch
        self.max_seq_len = max_seq_len or config.max_seq_len
        self.page_size = page_size
        self.max_fast_seqlen = config.max_fast_seqlen  # reference :344-346
        self.weights: Dict[str, torch.Tensor] = {}
        cfg = config
        tc = self.token_config
        self._ccfg = _capi.SmolConfig(
            dim=cfg.dim, n_layer=cfg.n_layer, n_head=cfg.n_head, n_local_heads=cfg.n_local_heads,
            head_dim=cfg.head_dim, intermediate_size=cfg.intermediate_size, vocab_size=cfg.vocab_size,
            fast_dim=cfg.fast_dim, n_fast_layer=cfg.n_fast_layer, fast_n_head=cfg.fast_n_head,
            fast_n_local_heads=cfg.fast_n_local_heads, fast_head_dim=cfg.fast_head_dim,
            fast_intermediate_size=cfg.fast_intermediate_size, codebook_size=cfg.codebook_size,
            num_codebooks=cfg.num_codebooks, duplicate_code_0=int(bool(cfg.duplicate_code_0)),
            depthwise_wte=int(bool(cfg.depthwise_wte)), depthwise_output=int(bool(cfg.depthwise_output)),
            tie_word_embeddings=int(bool(cfg.tie_word_embeddings)), max_seq_len=self.max_seq_len,
            max_batch=max_batch, page_size=page_size, semantic_start_id=tc.semantic_start_id,
            semantic_end_id=tc.semantic_end_id if tc.semantic_end_id is not None else -1,
            im_end_id=tc.im_end_id, mlx_embed_mask=int(mlx_embed_mask), norm_eps=cfg.norm_eps)
        handle = C.c_void_p()
        _capi.check(self.lib.smol_create(C.byref(self._ccfg), C.byref(handle)))
        self._h = handle
        with torch.cuda.device(self.device):
            ws_bytes = self.lib.smol_workspace_bytes(self._h)
            self._workspace = torch.zeros(ws_bytes + 256, dtype=torch.uint8, device=self.device)
            base = self._workspace.data_ptr()
            self._ws_ptr = (base + 255) // 256 * 256
            _capi.check(self.lib.smol_bind_workspace(self._h, C.c_void_p(self._ws_ptr), ws_bytes))
            pages_per_seq = (self.max_seq_len + page_size - 1) // page_size
            self.n_pages = kv_pages if kv_pages is not None else max_batch * pages_per_seq
            self.page_bytes = self.lib.smol_kv_page_bytes(self._h)
            self._kv_pool = torch.zeros(self.n_pages * self.page_bytes, dtype=torch.uint8, device=self.device)
            _capi.check(self.lib.smol_kv_bind(self._h, C.c_void_p(self._kv_pool.data_ptr()), self.n_pages))
        self._free_pages: List[int] = list(range(self.n_pages - 1, -1, -1))
        self._force: Optional[torch.Tensor] = None
        self._weights_struct = None

    # ------------------------------------------------------------------ construction
    @staticmethod
    def from_pretrained(path: str, load_weights: bool = True, weight_override: Optional[Dict[str, torch.Tensor]] = None,
                        max_length: Optional[int] = None, rope_base: Optional[int] = None,
                        **engine_kwargs) -> "RQTransformer":
        """reference modeling/model/rq_transformer.py:273-319.  ``load_weights=False`` leaves the model
        unbound until ``load_state_dict`` (the reference would random-init; this engine has no
        initialiser of its own -- use ``smoltts_b200.synth.make_state_dict``)."""
        config = RQTransformerModelArgs.from_pretrained(str(path))
        if max_length is not None:
            config.max_seq_len = max_length
        if rope_base is not None:
            config.rope_base = rope_base
        p = Path(path)
        tok_file = p / "tokenizer.json"
        token_config = TokenConfig.from_tokenizer_file(str(tok_file), config) if tok_file.exists() else None
        model = RQTransformer(config, token_config=token_config, **engine_kwargs)
        weights = weight_override
        if weights is None and load_weights:
            if (p / "model.safetensors").exists():
                from safetensors.torch import load_file

                weights = load_file(str(p / "model.safetensors"))
            elif (p / "model.pth").exists():
                weights = torch.load(p / "model.pth", map_location="cpu", mmap=True, weights_only=True)
            else:
                raise FileNotFoundError(f"no model.safetensors / model.pth under {path}")
        if weights is not None:
            model.load_state_dict(weights)
        return model

    def load_state_dict(self, state_dict: Dict[str, torch.Tensor], strict: bool = True) -> None:
        """Binds a checkpoint (any accepted layout) as bf16 device tensors."""
        cfg = self.config
        sd = normalise_state_dict(state_dict, cfg)
        want = expected_shapes(cfg)
        missing = [k for k in want if k not in sd]
        if missing:
            raise KeyError(f"checkpoint is missing {missing[:4]}{'...' if len(missing) > 4 else ''}")
        unexpected = [k for k in sd if k not in want]
        if unexpected and strict:
            raise KeyError(f"unexpected checkpoint keys {unexpected[:4]}")
        for k, shape in want.items():
            if tuple(sd[k].shape) != tuple(shape):
                raise ValueError(f"shape mismatch for {k}: {tuple(sd[k].shape)} vs {tuple(shape)}")
        dev = self.device
        self.weights = {k: sd[k].to(device=dev, dtype=torch.bfloat16).contiguous() for k in want}
        hd = cfg.dim // cfg.n_head
        self.weights["__rope"] = precompute_freqs_cis(self.max_seq_len, hd, cfg.rope_base).to(dev).contiguous()
        self.weights["__fast_rope"] = precompute_freqs_cis(cfg.max_fast_seqlen, cfg.fast_dim // cfg.fast_n_head,
                                                           cfg.rope_base).to(dev).contiguous()
        w = _capi.SmolWeights()
        g = lambda name: self.weights[name].data_ptr()  # noqa: E731
        w.embeddings = g("embeddings.weight")
        w.codebook_embeddings = g("codebook_embeddings.weight")
        w.norm = g("norm.weight")
        w.output = g("output.weight") if not cfg.tie_word_embeddings else None
        w.fast_embeddings = g("fast_embeddings.weight")
        w.fast_norm = g("fast_norm.weight")
        w.fast_output = g("fast_output.weight")
        w.rope = g("__rope")
        w.fast_rope = g("__fast_rope")
        for pre, arr, n in (("layers", w.layers, cfg.n_layer), ("fast_layers", w.fast_layers, cfg.n_fast_layer)):
            for l in range(n):
                p = f"{pre}.{l}."
                arr[l].wqkv = g(p + "attention.wqkv.weight")
                arr[l].wo = g(p + "attention.wo.weight")
                arr[l].w1 = g(p + "feed_forward.w1.weight")
                arr[l].w3 = g(p + "feed_forward.w3.weight")
                arr[l].w2 = g(p + "feed_forward.w2.weight")
                arr[l].attention_norm = g(p + "attention_norm.weight")
                arr[l].ffn_norm = g(p + "ffn_norm.weight")
        self._weights_struct = w
        _capi.check(self.lib.smol_bind_weights(self._h, C.byref(w)))

    def state_dict(self) -> Dict[str, torch.Tensor]:
        return {k: v for k, v in self.weights.items() if not k.startswith("__")}

    def save_pretrained(self, pathname: str) -> None:
        """config.json + model.safetensors in the exported layout (SURVEY §8(b))."""
        from safetensors.torch import save_file

        os.makedirs(pathname, exist_ok=True)
        self.config.save(os.path.join(pathname, "config.json"))
        save_file({k: v.cpu() for k, v in self.state_dict().items()}, os.path.join(pathname, "model.safetensors"))

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self.lib.smol_destroy(self._h)
                self._h = None
        except Exception:
            pass

    # ------------------------------------------------------------------ KV pages
    def allocate_pages(self, n: int) -> List[int]:
        if n > len(self._free_pages):
            raise _capi.SmolError(_capi.SMOL_ERR_CAPACITY, f"KV pool exhausted: need {n} pages, {len(self._free_pages)} free")
        return [self._free_pages.pop() for _ in range(n)]

    def free_pages(self, pages: Sequence[int]) -> None:
        self._free_pages.extend(reversed(list(pages)))

    def new_batch(self, batch: int, max_positions: Optional[int] = None, max_frames: int = 0,
                  seq_ids: Optional[Sequence[int]] = None) -> DecodeBatch:
        if batch > self.max_batch:
            raise _capi.SmolError(_capi.SMOL_ERR_CAPACITY, f"batch {batch} > max_batch {self.max_batch}")
        if max_positions is not None and max_positions > self.max_seq_len:
            raise _capi.SmolError(_capi.SMOL_ERR_CAPACITY,
                                  f"max_positions {max_positions} > max_seq_len {self.max_seq_len} (rows of the RoPE table)")
        return DecodeBatch(self, batch, max_positions or self.max_seq_len, max_frames, seq_ids)

    # ------------------------------------------------------------------ engine calls
    def _stream(self) -> C.c_void_p:
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def sampling(self, temp: float = 0.0, fast_temp: Optional[float] = 0.0, top_k: int = 0, top_p: float = 1.0,
                 min_p: float = 0.0, seed: int = 0, audio_only: bool = True, ignore_stop: bool = False) -> _capi.SmolSampling:
        return _capi.SmolSampling(temp=float(temp), fast_temp=float(fast_temp or 0.0), top_k=int(top_k), top_p=float(top_p),
                                  min_p=float(min_p or 0.0), seed=int(seed), audio_only=int(audio_only),
                                  ignore_stop=int(ignore_stop))

    def row_sampling(self, settings: Sequence["GenerationSettings"]) -> torch.Tensor:
        """Device table [B, 32] uint8 of ``SmolRowSampling`` records, one per ``GenerationSettings`` (same min-p rule as a
        call's ``SmolSampling``), for ``DecodeBatch.set_row_sampling`` / ``SmolBatch.row_sampling``.  Validated on the host:
        ``ValueError`` for a negative or non-finite temperature, top_k < 0, top_p outside (0, 1], min_p outside [0, 1)."""
        from .generate import row_sampling_table

        return row_sampling_table(settings).to(self.device)

    def set_option(self, name: str, value: int) -> None:
        _capi.check(self.lib.smol_set_option(self._h, name.encode(), int(value)))

    def get_option(self, name: str) -> int:
        return int(self.lib.smol_get_option(self._h, name.encode()))

    def set_force(self, force: Optional[torch.Tensor]) -> None:
        """force [B, R] int32 device tensor or None (teacher forcing / resync)."""
        self._force = force
        _capi.check(self.lib.smol_set_force(self._h, C.c_void_p(force.data_ptr()) if force is not None else None))

    def set_profile(self, enable: bool = True) -> Optional[torch.Tensor]:
        """Per-phase ns accumulators [phase_count, 2] (CTA 0: work, barrier wait); None switches off."""
        if not enable:
            _capi.check(self.lib.smol_set_profile(self._h, None))
            self._prof = None
            return None
        # [0 : 2*512] per-phase (work, wait) pairs, then 16 x 4 sub-phase segments of the weight phases
        self._prof = torch.zeros(2 * 512 + 64 + 2 * 512 * 8 + 256 * 512 * 2, dtype=torch.int64, device=self.device)  # + cycle trace, + per-CTA skew trace (data-flow kernel)
        _capi.check(self.lib.smol_set_profile(self._h, C.c_void_p(self._prof.data_ptr())))
        return self._prof

    def set_frame_clock(self, capacity: int = 0) -> Optional[torch.Tensor]:
        """Device-side per-frame clock: returns an int64 tensor [capacity]; entry f receives %globaltimer (ns) when
        frame f of sequence 0 has been assembled.  capacity 0 switches it off."""
        if capacity <= 0:
            _capi.check(self.lib.smol_set_frame_clock(self._h, None, 0))
            self._frame_ns = None
            return None
        self._frame_ns = torch.zeros(capacity, dtype=torch.int64, device=self.device)
        _capi.check(self.lib.smol_set_frame_clock(self._h, C.c_void_p(self._frame_ns.data_ptr()), capacity))
        return self._frame_ns

    def prefill(self, batch: DecodeBatch, prompts: torch.Tensor, lengths: torch.Tensor) -> None:
        """prompts [B, R, s_max] int32 (device), lengths [B] int32 (device).  Leaves every
        sequence with its first len-1 columns cached and the last column pending."""
        B, R, s_max = prompts.shape
        host_len = lengths.tolist()
        # a prompt of n columns caches n - 1 positions on top of what the sequence already holds
        if any(batch.host_len[b] + host_len[b] - 1 > batch.capacity for b in range(B)):
            raise _capi.SmolError(_capi.SMOL_ERR_CAPACITY, "prompt (plus the positions already cached) exceeds the sequence's KV capacity")
        _capi.check(self.lib.smol_prefill(self._h, C.byref(batch.c), B, C.c_void_p(prompts.data_ptr()),
                                          C.c_void_p(lengths.data_ptr()), s_max, self._stream()))
        for b in range(B):
            batch.host_len[b] += host_len[b] - 1

    def decode_frames(self, batch: DecodeBatch, sampling: _capi.SmolSampling, n_frames: int) -> None:
        if max(batch.host_len) + n_frames > batch.capacity:
            raise _capi.SmolError(_capi.SMOL_ERR_CAPACITY,
                                  f"{n_frames} more frames exceed the KV capacity {batch.capacity} of the batch")
        _capi.check(self.lib.smol_decode_frames(self._h, C.byref(batch.c), batch.batch, C.byref(sampling), n_frames,
                                                self._stream()))
        for b in range(batch.batch):
            batch.host_len[b] += n_frames

    def slow_step(self, batch: DecodeBatch, advance: bool = True) -> None:
        if advance and max(batch.host_len) + 1 > batch.capacity:
            raise _capi.SmolError(_capi.SMOL_ERR_CAPACITY, f"one more position exceeds the KV capacity {batch.capacity} of the batch")
        _capi.check(self.lib.smol_slow_step(self._h, C.byref(batch.c), batch.batch, int(advance), self._stream()))
        if advance:
            for b in range(batch.batch):
                batch.host_len[b] += 1

    def fast_step(self, batch: DecodeBatch, depth_pos: int, from_xf: bool = False) -> None:
        _capi.check(self.lib.smol_fast_step(self._h, C.byref(batch.c), batch.batch, depth_pos, int(from_xf), self._stream()))

    def fast_embed(self, batch: DecodeBatch, codes: torch.Tensor, depth_pos: int) -> None:
        _capi.check(self.lib.smol_fast_embed(self._h, batch.batch, C.c_void_p(codes.data_ptr()), depth_pos, self._stream()))

    def run_phases(self, batch: DecodeBatch, sampling: _capi.SmolSampling, begin: int, end: int) -> None:
        _capi.check(self.lib.smol_run_phases(self._h, C.byref(batch.c), batch.batch, C.byref(sampling), begin, end,
                                             self._stream()))

    def sample(self, logits: torch.Tensor, sampling: _capi.SmolSampling, stream_id: int,
               batch: Optional[DecodeBatch] = None) -> torch.Tensor:
        """logits [B, n] fp32 device -> ids [B] int32 (the fused sampling kernel on its own)."""
        B, n = logits.shape
        out = torch.empty(B, dtype=torch.int32, device=logits.device)
        _capi.check(self.lib.smol_sample(self._h, C.byref(batch.c) if batch is not None else None, B,
                                         C.c_void_p(logits.data_ptr()), n, C.byref(sampling), stream_id,
                                         C.c_void_p(out.data_ptr()), self._stream()))
        return out

    @property
    def phase_count(self) -> int:
        return int(self.lib.smol_phase_count(self._h))

    @property
    def launch_count(self) -> int:
        return int(self.lib.smol_launch_count(self._h))

    def debug_buffer(self, name: str, batch: Optional[int] = None) -> torch.Tensor:
        """View of a workspace buffer (see include/smoltts_b200.h: smol_debug_buffer)."""
        cfg = self.config
        B = batch or self.max_batch
        spec = {
            "x": (torch.bfloat16, (self.max_batch, cfg.dim)),
            "h": (torch.bfloat16, (self.max_batch, max(cfg.dim, cfg.fast_dim))),
            "xf": (torch.bfloat16, (self.max_batch, cfg.fast_dim)),
            "q": (torch.bfloat16, (self.max_batch, max(cfg.n_head, cfg.fast_n_head) * 64)),
            "attn": (torch.bfloat16, (self.max_batch, max(cfg.dim, cfg.fast_dim))),
            "act": (torch.bfloat16, (self.max_batch, max(cfg.intermediate_size, cfg.fast_intermediate_size))),
            "fkv": (torch.bfloat16, (self.max_batch, cfg.n_fast_layer, 2, cfg.max_fast_seqlen, cfg.fast_n_local_heads * 64)),
            "token_logits": (torch.float32, (self.max_batch, cfg.vocab_size)),
            "depth_logits": (torch.float32, (self.max_batch, cfg.max_fast_seqlen, cfg.codebook_size)),
            "frame_tokens": (torch.int32, (self.max_batch, cfg.n_rows)),
        }[name]
        ptr = self.lib.smol_debug_buffer(self._h, name.encode())
        if not ptr:
            raise KeyError(name)
        dtype, shape = spec
        off = ptr - self._ws_ptr
        n = 1
        for s in shape:
            n *= s
        nbytes = n * torch.empty((), dtype=dtype).element_size()
        start = self._ws_ptr - self._workspace.data_ptr() + off
        return self._workspace[start:start + nbytes].view(dtype).view(*shape)[:B]

    # ---- word regions of the data-flow kernel (include/smoltts_b200.h: smol_debug_buffer "ll", "ll2_score", ..)
    def _words(self, name: str, word_offset: int, n_words: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(payload, epoch) int32 views [n_words] of 8-byte words of the named buffer, starting at word `word_offset`."""
        ptr = self.lib.smol_debug_buffer(self._h, name.encode())
        if not ptr:
            raise KeyError(name)
        start = ptr - self._workspace.data_ptr() + 8 * word_offset
        w = self._workspace[start:start + 8 * n_words].view(torch.int32).view(n_words, 2)
        return w[:, 0], w[:, 1]

    def ll_region(self, phase: int) -> Tuple[int, int]:
        """(word offset, words per sequence and replica) of phase `phase`'s region."""
        off, n = C.c_uint32(), C.c_uint32()
        _capi.check(self.lib.smol_ll_region(self._h, int(phase), C.byref(off), C.byref(n)))
        return int(off.value), int(n.value)

    def ll_words(self, phase: int, team: int = 0, rep: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        """(payload, epoch) int32 views [len] of phase `phase`'s words: sequence (team) `team`, replica `rep`."""
        off, n = self.ll_region(phase)
        return self._words("ll", off + (team * LL_REPLICAS + rep) * n, n)

    def ll_epoch(self) -> int:
        """Phases run by every data-flow launch so far: phase p of a launch's last frame carried ll_epoch() - phase_count + p + 1."""
        return int(self._words("ll_epoch", 0, 1)[0].item())

    def ll_scores(self, team: int, layer: int) -> Tuple[torch.Tensor, torch.Tensor]:
        """(fp32 q.k / 8 scores, epoch) [n_head, score_len] of slow layer `layer` (its parity's buffer: the last two layers
        of a frame are kept)."""
        H = self.config.n_head
        n = (self.max_seq_len + 511) // 512 * 512   # capi.cu: ll2_score_len
        pay, ep = self._words("ll2_score", (team * 2 + layer % 2) * H * n, H * n)
        return pay.view(torch.float32).view(H, n), ep.view(H, n)

    def ll_psums(self, phase: int, rep: int = 0) -> Tuple[torch.Tensor, torch.Tensor]:
        """(fp32 partial sums, epoch) [7 K-slices, dim] of the fused MLP's W2 phase `phase` (batch 1), replica `rep`."""
        cfg = self.config
        n_slow, per = 5 * cfg.n_layer, 4 * cfg.n_fast_layer + 2
        depth_pos, r = divmod(phase - n_slow - 2, per)   # fast phases: depth position, phase inside the depth step
        if 0 <= phase < n_slow and phase % 5 == 4:
            w2 = phase // 5
        elif phase >= n_slow + 2 and r < 4 * cfg.n_fast_layer and r % 4 == 3:
            w2 = cfg.n_layer + depth_pos * cfg.n_fast_layer + r // 4
        else:
            raise ValueError(f"phase {phase} is not a W2 phase")
        n = LL_PSUM_SLICES * cfg.dim
        pay, ep = self._words("ll2_psum", (w2 * LL_REPLICAS + rep) * n, n)
        return pay.view(torch.float32).view(LL_PSUM_SLICES, cfg.dim), ep.view(LL_PSUM_SLICES, cfg.dim)

    def kv_view(self) -> torch.Tensor:
        """[n_pages, n_layer, 2, n_kv, page_size, 64] bf16 view of the paged pool."""
        cfg = self.config
        return self._kv_pool.view(torch.bfloat16).view(self.n_pages, cfg.n_layer, 2, cfg.n_local_heads, self.page_size, 64)

    # ------------------------------------------------------------------ MLX-style model calls
    def forward_generate(self, inputs: torch.Tensor, cache: "SlowCache") -> Tuple[torch.Tensor, torch.Tensor]:
        """reference mlx lm/rq_transformer.py:173-192: inputs [1, R, S] (or [R, S]) ids; pushes S
        positions through the slow transformer against ``cache`` and returns
        (token_logits [1, V] fp32, hidden [1, D] bf16 -- the PRE-norm stream, quirk §8(g)-2)."""
        x = inputs if inputs.ndim == 3 else inputs[None]
        if x.shape[0] != 1:
            raise ValueError("forward_generate is the reference's bs=1 call; use generate_batch for batches")
        x = x.to(device=self.device, dtype=torch.int32).contiguous()
        S = x.shape[2]
        batch = cache.batch
        if S > 1:
            self.prefill(batch, x, torch.tensor([S], dtype=torch.int32, device=self.device))
        else:
            batch.tokens.copy_(x[:, :, 0])
        self.slow_step(batch, advance=True)
        logits = self.debug_buffer("token_logits", 1).clone()
        hidden = self.debug_buffer("x", 1).clone()
        return logits, hidden

    def forward_generate_fast(self, x: torch.Tensor, input_pos: int, cache: "FastCache") -> torch.Tensor:
        """reference mlx lm/rq_transformer.py:194-220: x [1, 1, Df] (hidden state or code embedding),
        depth position ``input_pos`` -> codebook logits [1, C] fp32."""
        xf = self.debug_buffer("xf", 1)
        xf.copy_(x.reshape(1, -1).to(device=self.device, dtype=torch.bfloat16))
        self.fast_step(cache.batch, int(input_pos), from_xf=True)
        return self.debug_buffer("depth_logits", 1)[:, int(input_pos)].clone()

    def fast_embeddings(self, ids: torch.Tensor) -> torch.Tensor:
        """reference fast_embeddings lookup (mlx lm/generate.py:140) -- a gather, done by torch indexing."""
        return self.weights["fast_embeddings.weight"][ids.to(self.device).long()]


class SlowCache:
    """Stand-in for the list of per-layer KVCache objects (mlx lm/cache.py:6-33): one sequence's
    pages in the paged pool plus its device-side length."""

    def __init__(self, model: RQTransformer, max_positions: Optional[int] = None, seq_id: int = 0):
        self.batch = model.new_batch(1, max_positions=max_positions, max_frames=0, seq_ids=[seq_id])

    @property
    def offset(self) -> int:
        return int(self.batch.seq_len.item())


class FastCache:
    """The depth transformer's <= depth positions live in the engine's workspace ("fkv"); this
    handle only names the sequence they belong to (the reference re-creates 4 KVCache objects per
    frame, mlx lm/generate.py:112)."""

    def __init__(self, slow: SlowCache):
        self.batch = slow.batch


def make_prompt_cache(model: RQTransformer, is_fast: bool = False, slow: Optional[SlowCache] = None,
                      max_positions: Optional[int] = None):
    """reference mlx lm/cache.py:25-33."""
    if is_fast:
        if slow is None:
            raise ValueError("the fast cache is tied to a sequence: pass slow=<SlowCache>")
        return FastCache(slow)
    return SlowCache(model, max_positions=max_positions)
