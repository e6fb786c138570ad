"""Mimi streaming decoder (codes -> 24 kHz PCM) on the B200 -- host-side mirror of the reference's codec API.

Reference (paths under mlx_inference/src/smoltts_mlx/): ``codec/mimi.py`` -- ``MimiConfig`` (:20-23), ``MimiModel.decode``
(:88-100), ``MimiModel.decode_step`` (:102-104), ``load_mimi`` (:107-156); its caller ``SmolTTS.stream``
(``__init__.py:85-92``) makes one transformer cache per utterance and calls ``decode_step`` once per generated frame.

Same names and argument meaning here; what differs is what an engine for many concurrent utterances needs:
* the state of a stream (transformer KV, convolution history rows of the SEANet, position) lives in a numbered *slot* of
  the engine's workspace instead of Python objects hung on the modules; ``make_cache()`` hands out a slot,
  ``decode_step(codes, cache)`` accepts one handle or a list of handles (one per row of ``codes``);
* all compute is CUDA (``csrc/mimi_kernels.cu`` behind ``include/smoltts_b200_mimi.h``); there is no CPU path -- the
  constructor raises without a CUDA device.

Checkpoint layout: kyutai/mimi's ``model.safetensors`` keys and torch layouts (what ``load_mimi`` reads).  The decode half
(``quantizer.*``, ``upsample``, ``decoder_transformer``, ``decoder``) is always bound; the encode half (``encoder``,
``encoder_transformer``, ``downsample``, the quantizers' ``input_proj``) only with ``encode_max_samples > 0``, for
``encode`` (audio -> codes, ``csrc/mimi_encoder.cu``, pinned to transformers' ``MimiModel.encode``).
"""
from __future__ import annotations

import ctypes as C
import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional, Sequence, Union

import torch

from . import _capi


@dataclass
class SeanetConfig:   # codec/conv.py:8-22
    dimension: int = 512
    channels: int = 1
    n_filters: int = 64
    n_residual_layers: int = 1
    compress: int = 2
    dilation_base: int = 2
    kernel_size: int = 7
    residual_kernel_size: int = 3
    last_kernel_size: int = 3
    ratios: List[int] = field(default_factory=lambda: [8, 6, 5, 4])
    trim_right_ratio: float = 1.0
    sampling_rate: float = 24_000.0
    upsample_groups: int = 512


@dataclass
class MimiTransformerConfig:   # codec/transformer.py:10-33
    d_model: int = 512
    num_heads: int = 8
    head_dim: int = 64
    num_layers: int = 8
    layer_scale: Optional[float] = 0.01
    context: int = 250
    dim_feedforward: int = 2048
    rope_theta: float = 10_000.0
    norm_eps: float = 1e-5


@dataclass
class RVQConfig:   # codec/rvq.py:7-13
    codebook_size: int = 2048
    codebook_dim: int = 256
    num_quantizers: int = 32
    num_semantic_quantizers: int = 1
    frame_rate: float = 12.5
    hidden_dim: int = 512


@dataclass
class MimiConfig:   # codec/mimi.py:20-23
    seanet: SeanetConfig = field(default_factory=SeanetConfig)
    transformer: MimiTransformerConfig = field(default_factory=MimiTransformerConfig)
    rvq: RVQConfig = field(default_factory=RVQConfig)


@dataclass
class MimiCache:
    """Handle of one stream's state (replaces ``make_prompt_cache(codec.decoder_transformer)`` + the per-module
    ``_stream_prev_*`` attributes of the reference)."""
    slot: int
    frames: int = 0


def mimi_rope_table(head_dim: int, theta: float, n_pos: int) -> torch.Tensor:
    """[n_pos][head_dim]: cos | sin of pos * theta^(-2i / head_dim) (nn.RoPE(traditional=False), transformer.py:60-64)."""
    inv = 1.0 / (theta ** (torch.arange(0, head_dim, 2, dtype=torch.float32) / head_dim))
    ang = torch.arange(n_pos, dtype=torch.float32)[:, None] * inv[None, :]
    return torch.cat([ang.cos(), ang.sin()], dim=1).contiguous()


def _aligned(ws: torch.Tensor) -> int:
    """The 256-byte-aligned start of a workspace allocated 256 bytes larger than the engine asked for."""
    return (ws.data_ptr() + 255) // 256 * 256


class _Binder:
    """What the decoder's and the encoder's bind share: state-dict tensors checked and made fp32 on the device (kept
    alive until the engine has repacked them), the codebooks, the transformer layers, the RoPE table and the workspace."""

    def __init__(self, sd: Dict[str, torch.Tensor], device: torch.device):
        self.sd, self.device = sd, device
        self.keep: List[torch.Tensor] = []

    def _hold(self, v: torch.Tensor) -> int:
        self.keep.append(v)
        return v.data_ptr()

    def __call__(self, key: str, shape: Sequence[int]) -> int:
        if key not in self.sd:
            raise KeyError(f"MimiModel.load_state_dict: missing key {key}")
        v = self.sd[key]
        if tuple(v.shape) != tuple(shape):
            raise ValueError(f"MimiModel.load_state_dict: {key} has shape {tuple(v.shape)}, expected {tuple(shape)}")
        return self._hold(v.detach().to(device=self.device, dtype=torch.float32).contiguous())

    def codebooks(self, w, n_q: int, c: RVQConfig) -> None:
        for i in range(n_q):
            p = ("quantizer.semantic_residual_vector_quantizer.layers.0" if i == 0
                 else f"quantizer.acoustic_residual_vector_quantizer.layers.{i - 1}")
            w.embed_sum[i] = self(p + ".codebook.embed_sum", (c.codebook_size, c.codebook_dim))
            w.cluster_usage[i] = self(p + ".codebook.cluster_usage", (c.codebook_size,))

    def layers(self, w, prefix: str, c: MimiTransformerConfig) -> None:
        D, F = c.d_model, c.dim_feedforward
        for l in range(c.num_layers):
            p = f"{prefix}.layers.{l}."
            L = w.layers[l]
            L.q_proj, L.k_proj = self(p + "self_attn.q_proj.weight", (D, D)), self(p + "self_attn.k_proj.weight", (D, D))
            L.v_proj, L.o_proj = self(p + "self_attn.v_proj.weight", (D, D)), self(p + "self_attn.o_proj.weight", (D, D))
            L.fc1, L.fc2 = self(p + "mlp.fc1.weight", (F, D)), self(p + "mlp.fc2.weight", (D, F))
            L.ln1_w, L.ln1_b = self(p + "input_layernorm.weight", (D,)), self(p + "input_layernorm.bias", (D,))
            L.ln2_w, L.ln2_b = self(p + "post_attention_layernorm.weight", (D,)), self(p + "post_attention_layernorm.bias", (D,))
            L.scale_attn, L.scale_mlp = self(p + "self_attn_layer_scale.scale", (D,)), self(p + "mlp_layer_scale.scale", (D,))

    def rope(self, c: MimiTransformerConfig, n_pos: int) -> int:
        return self._hold(mimi_rope_table(c.head_dim, c.rope_theta, n_pos).to(self.device))

    def bind(self, workspace_bytes, bind, handle, w) -> torch.Tensor:
        """Allocates the engine's workspace, binds `w` into it and waits for the repacking; returns the workspace."""
        n = int(workspace_bytes(handle))
        ws = torch.empty(n + 256, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            stream = torch.cuda.current_stream().cuda_stream
            _capi.check(bind(handle, C.byref(w), C.c_void_p(_aligned(ws)), C.c_size_t(n), C.c_void_p(stream)))
            torch.cuda.current_stream().synchronize()   # the source tensors in `keep` may go now: everything was repacked
        return ws


class MimiModel:
    """The decode half of the reference's ``MimiModel`` on one CUDA device."""

    def __init__(self, config: Optional[MimiConfig] = None, num_codebooks: int = 8, max_streams: int = 1, max_frames: int = 2048,
                 window: int = 0, upsample_carry: bool = False, mode: str = "graph", device: Union[str, torch.device, None] = None,
                 encode_max_samples: int = 0, encode_max_clips: int = 1):
        """mode: "graph" -- a step's 57 launches are captured once per (batch, buffers) and replayed as one CUDA graph (the
        default); "eager" -- plain launches with programmatic dependent launch (also what a caller's own graph capture
        records).  Both compute the same bits.

        encode_max_samples > 0 builds the encoder too (``encode``) for up to ``encode_max_clips`` clips and
        ``encode_max_samples`` samples in all per call; its workspace grows with ``encode_max_samples`` (about 660 bytes per
        sample).  At 0 nothing of the encoder is allocated or bound."""
        if not torch.cuda.is_available():
            raise RuntimeError("smoltts_b200.MimiModel needs a CUDA device (there is no CPU path)")
        self.config = config or MimiConfig()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.num_codebooks = num_codebooks
        self.max_streams = max_streams
        self.max_frames = max_frames
        self._lib = _capi.load()
        c = self.config
        if c.seanet.n_residual_layers != 1 or c.seanet.compress != 2 or c.seanet.trim_right_ratio != 1.0:
            raise ValueError("MimiModel: only kyutai/mimi's SEANet shape is built (1 residual layer, compress 2, right trim 1.0)")
        if c.rvq.num_semantic_quantizers != 1:
            raise ValueError("MimiModel: one semantic quantizer expected")
        cfg = _capi.SmolMimiConfig()
        cfg.n_q = num_codebooks
        cfg.codebook_size, cfg.codebook_dim = c.rvq.codebook_size, c.rvq.codebook_dim
        cfg.dim, cfg.n_layers, cfg.n_heads = c.transformer.d_model, c.transformer.num_layers, c.transformer.num_heads
        cfg.head_dim, cfg.ffn = c.transformer.head_dim, c.transformer.dim_feedforward
        cfg.n_filters, cfg.n_ratios = c.seanet.n_filters, len(c.seanet.ratios)
        for i, r in enumerate(c.seanet.ratios):
            cfg.ratios[i] = r
        cfg.kernel, cfg.res_kernel, cfg.last_kernel = c.seanet.kernel_size, c.seanet.residual_kernel_size, c.seanet.last_kernel_size
        cfg.max_streams, cfg.max_positions = max_streams, 2 * max_frames
        if mode not in ("graph", "eager"):
            raise ValueError(f"MimiModel: unknown mode {mode!r}")
        self.mode = mode
        cfg.window, cfg.upsample_carry, cfg.use_graph = window, int(upsample_carry), {"eager": 0, "graph": 1}[mode]
        cfg.norm_eps, cfg.codebook_eps = c.transformer.norm_eps, 1e-5
        self._cfg = cfg
        h = C.c_void_p()
        _capi.check(self._lib.smol_mimi_create(C.byref(cfg), C.byref(h)))
        self._h = h
        self.samples_per_frame = int(self._lib.smol_mimi_samples_per_frame(h))
        assert self.samples_per_frame == 2 * math.prod(c.seanet.ratios)
        self._ws: Optional[torch.Tensor] = None
        self._free = list(range(max_streams - 1, -1, -1))
        self._frames = [0] * max_streams
        self._io: Dict[int, tuple] = {}   # batch -> (codes, slots, pcm) device buffers with stable addresses (graph replay)
        self._io_slots: Dict[int, tuple] = {}
        self.encode_max_samples, self.encode_max_clips = int(encode_max_samples), int(encode_max_clips)
        self._enc = None
        self._enc_ws: Optional[torch.Tensor] = None
        if self.encode_max_samples > 0:
            ec = _capi.SmolMimiEncoderConfig()
            for name in ("n_q", "codebook_size", "codebook_dim", "dim", "n_layers", "n_heads", "head_dim", "ffn", "n_filters", "n_ratios",
                         "kernel", "res_kernel", "last_kernel", "norm_eps", "codebook_eps"):
                setattr(ec, name, getattr(cfg, name))
            for i, r in enumerate(c.seanet.ratios):
                ec.ratios[i] = r
            ec.max_clips, ec.max_samples, ec.window = self.encode_max_clips, self.encode_max_samples, c.transformer.context
            he = C.c_void_p()
            _capi.check(self._lib.smol_mimi_encoder_create(C.byref(ec), C.byref(he)))
            self._enc = he

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._lib.smol_mimi_destroy(self._h)
                self._h = None
            if getattr(self, "_enc", None):
                self._lib.smol_mimi_encoder_destroy(self._enc)
                self._enc = None
        except Exception:
            pass

    # ---- weights ------------------------------------------------------------------------------------------------------
    def load_state_dict(self, sd: Dict[str, torch.Tensor]) -> None:
        """kyutai/mimi keys (`initialized` buffers and unused codebooks are ignored, and so are the encoder half and
        `input_proj` unless the encoder was built)."""
        c = self.config
        t = _Binder(sd, self.device)
        w = _capi.SmolMimiWeights()
        D, cd = c.transformer.d_model, c.rvq.codebook_dim
        t.codebooks(w, self.num_codebooks, c.rvq)
        w.semantic_output_proj = t("quantizer.semantic_residual_vector_quantizer.output_proj.weight", (D, cd, 1))
        w.acoustic_output_proj = t("quantizer.acoustic_residual_vector_quantizer.output_proj.weight", (D, cd, 1))
        w.upsample = t("upsample.conv.weight", (D, 1, 4))
        t.layers(w, "decoder_transformer", c.transformer)
        s = c.seanet
        ch = s.n_filters * 2 ** len(s.ratios)
        w.conv_in.weight, w.conv_in.bias = t("decoder.layers.0.conv.weight", (ch, D, s.kernel_size)), t("decoder.layers.0.conv.bias", (ch,))
        idx = 1
        for i, r in enumerate(s.ratios):
            w.convtr[i].weight = t(f"decoder.layers.{idx + 1}.conv.weight", (ch, ch // 2, 2 * r))
            w.convtr[i].bias = t(f"decoder.layers.{idx + 1}.conv.bias", (ch // 2,))
            ch //= 2
            w.res_conv1[i].weight = t(f"decoder.layers.{idx + 2}.block.1.conv.weight", (ch // 2, ch, s.residual_kernel_size))
            w.res_conv1[i].bias = t(f"decoder.layers.{idx + 2}.block.1.conv.bias", (ch // 2,))
            w.res_conv2[i].weight = t(f"decoder.layers.{idx + 2}.block.3.conv.weight", (ch, ch // 2, 1))
            w.res_conv2[i].bias = t(f"decoder.layers.{idx + 2}.block.3.conv.bias", (ch,))
            idx += 3
        w.conv_out.weight = t(f"decoder.layers.{idx + 1}.conv.weight", (1, ch, s.last_kernel_size))
        w.conv_out.bias = t(f"decoder.layers.{idx + 1}.conv.bias", (1,))
        w.rope = t.rope(c.transformer, 2 * self.max_frames)
        self._ws = t.bind(self._lib.smol_mimi_workspace_bytes, self._lib.smol_mimi_bind, self._h, w)
        self._free = list(range(self.max_streams - 1, -1, -1))
        self._frames = [0] * self.max_streams
        if self._enc is not None:
            self._bind_encoder(sd)

    def _bind_encoder(self, sd: Dict[str, torch.Tensor]) -> None:
        c = self.config
        t = _Binder(sd, self.device)
        w = _capi.SmolMimiEncoderWeights()
        D, cd = c.transformer.d_model, c.rvq.codebook_dim
        t.codebooks(w, self.num_codebooks, c.rvq)
        w.semantic_input_proj = t("quantizer.semantic_residual_vector_quantizer.input_proj.weight", (cd, D, 1))
        w.acoustic_input_proj = t("quantizer.acoustic_residual_vector_quantizer.input_proj.weight", (cd, D, 1))
        w.downsample = t("downsample.conv.weight", (D, D, 4))
        t.layers(w, "encoder_transformer", c.transformer)
        s = c.seanet
        ch = s.n_filters
        w.conv_in.weight, w.conv_in.bias = t("encoder.layers.0.conv.weight", (ch, 1, s.kernel_size)), t("encoder.layers.0.conv.bias", (ch,))
        idx = 1
        for i, r in enumerate(reversed(s.ratios)):
            w.res_conv1[i].weight = t(f"encoder.layers.{idx}.block.1.conv.weight", (ch // 2, ch, s.residual_kernel_size))
            w.res_conv1[i].bias = t(f"encoder.layers.{idx}.block.1.conv.bias", (ch // 2,))
            w.res_conv2[i].weight = t(f"encoder.layers.{idx}.block.3.conv.weight", (ch, ch // 2, 1))
            w.res_conv2[i].bias = t(f"encoder.layers.{idx}.block.3.conv.bias", (ch,))
            w.conv_down[i].weight = t(f"encoder.layers.{idx + 2}.conv.weight", (2 * ch, ch, 2 * r))
            w.conv_down[i].bias = t(f"encoder.layers.{idx + 2}.conv.bias", (2 * ch,))
            ch, idx = 2 * ch, idx + 3
        w.conv_out.weight = t(f"encoder.layers.{idx + 1}.conv.weight", (D, ch, s.last_kernel_size))
        w.conv_out.bias = t(f"encoder.layers.{idx + 1}.conv.bias", (D,))
        w.rope = t.rope(c.transformer, -(-self.encode_max_samples // math.prod(s.ratios)))
        self._enc_ws = t.bind(self._lib.smol_mimi_encoder_workspace_bytes, self._lib.smol_mimi_encoder_bind, self._enc, w)

    # ---- encode (audio -> codes) --------------------------------------------------------------------------------------
    def encode(self, x: Union[torch.Tensor, Sequence[torch.Tensor]]) -> Union[torch.Tensor, List[torch.Tensor]]:
        """24 kHz mono fp32 PCM -> Mimi codes, as transformers' ``MimiModel.encode``: ``[B, 1, L]`` -> int64
        ``[B, n_q, ceil(L / 1920)]``, or a list of 1-D clips of any lengths -> a list of int64 ``[n_q, T_b]``.  Every clip is
        encoded exactly as it would be alone, in one call for all of them.  Asynchronous on the current CUDA stream."""
        if self._enc is None:
            raise RuntimeError("MimiModel.encode: this codec was built without an encoder (pass encode_max_samples > 0)")
        if self._enc_ws is None:
            raise RuntimeError("MimiModel: load_state_dict() first")
        batched = isinstance(x, torch.Tensor)
        if batched:
            if x.dim() != 3 or x.shape[1] != 1:
                raise ValueError(f"MimiModel.encode: expected [B, 1, L] mono audio, got {tuple(x.shape)}")
            clips = [x[b, 0] for b in range(x.shape[0])]
        else:
            clips = [torch.as_tensor(c) for c in x]
            if any(c.dim() != 1 for c in clips):
                raise ValueError("MimiModel.encode: every clip of a list must be 1-D mono audio")
        if not clips:
            return torch.zeros(0, self.num_codebooks, 0, dtype=torch.int64, device=self.device) if batched else []
        lens = [int(c.shape[0]) for c in clips]
        pcm = torch.cat([c.to(device=self.device, dtype=torch.float32) for c in clips]).contiguous()
        spf = self.samples_per_frame
        frames = [-(-n // spf) for n in lens]
        codes = torch.empty(sum(frames), self.num_codebooks, dtype=torch.int32, device=self.device)
        h_lens = (C.c_int64 * len(lens))(*lens)
        _capi.check(self._lib.smol_mimi_encode(self._enc, C.c_void_p(pcm.data_ptr()), h_lens, len(lens), C.c_void_p(codes.data_ptr()),
                                               C.c_void_p(self._stream())))
        self._enc_frames = sum(frames)
        per_clip = [c.t().to(torch.int64) for c in torch.split(codes, frames)]
        return torch.stack(per_clip) if batched else per_clip

    def encoder_latent(self) -> torch.Tensor:
        """Test hook: the pre-quantizer latent z of the last ``encode`` call, ``[sum_b T_b, dim]`` (clips back to back)."""
        p = self._lib.smol_mimi_encoder_debug_buffer(self._enc, b"latent")
        base = _aligned(self._enc_ws)
        n = int(self._lib.smol_mimi_encoder_workspace_bytes(self._enc))
        flat = self._enc_ws[base - self._enc_ws.data_ptr(): base - self._enc_ws.data_ptr() + n].view(torch.float32)
        off = (p - base) // 4
        D = self.config.transformer.d_model
        return flat[off: off + self._enc_frames * D].view(self._enc_frames, D).clone()

    @classmethod
    def from_safetensors(cls, path: str, **kw) -> "MimiModel":
        """load_mimi() (codec/mimi.py:107-156) from a local copy of kyutai/mimi's model.safetensors."""
        from safetensors.torch import load_file

        m = cls(**kw)
        m.load_state_dict(load_file(path))
        return m

    # ---- streams ------------------------------------------------------------------------------------------------------
    def make_cache(self) -> MimiCache:
        """A fresh stream (make_prompt_cache(codec.decoder_transformer), __init__.py:86, plus MimiDecoder.reset)."""
        if not self._free:
            raise RuntimeError(f"MimiModel: all {self.max_streams} stream slots are in use (release_cache() one)")
        slot = self._free.pop()
        self._reset([slot])
        return MimiCache(slot)

    def release_cache(self, cache: MimiCache) -> None:
        self._free.append(cache.slot)

    def _stream(self) -> int:
        return torch.cuda.current_stream(self.device).cuda_stream

    def _reset(self, slots: Sequence[int]) -> None:
        if self._ws is None:
            raise RuntimeError("MimiModel: load_state_dict() first")
        ids = torch.tensor(list(slots), dtype=torch.int32).to(self.device)
        _capi.check(self._lib.smol_mimi_reset(self._h, C.c_void_p(ids.data_ptr()), len(slots), C.c_void_p(self._stream())))
        for s in slots:
            self._frames[s] = 0

    def _buffers(self, batch: int):
        if batch not in self._io:
            self._io[batch] = (torch.zeros(batch, self.num_codebooks, dtype=torch.int32, device=self.device),
                               torch.zeros(batch, dtype=torch.int32, device=self.device),
                               torch.zeros(batch, self.samples_per_frame, dtype=torch.float32, device=self.device))
        return self._io[batch]

    def decode_step(self, codes: torch.Tensor, cache: Union[MimiCache, Sequence[MimiCache]]) -> torch.Tensor:
        """codes [B, n_q, 1] (or [B, n_q]) -> PCM [B, 1, samples_per_frame]; row b continues the stream of cache[b]
        (codec/mimi.py:102-104).  Asynchronous on the current CUDA stream; the result is a view of an internal buffer that the
        next call with the same batch size overwrites."""
        caches = [cache] if isinstance(cache, MimiCache) else list(cache)
        if codes.dim() == 3:
            if codes.shape[-1] != 1:
                raise ValueError("decode_step takes one frame: codes [B, n_q, 1]")
            codes = codes[..., 0]
        B = codes.shape[0]
        if B != len(caches) or codes.shape[1] != self.num_codebooks:
            raise ValueError(f"decode_step: codes {tuple(codes.shape)} vs {len(caches)} caches x {self.num_codebooks} codebooks")
        if len({c.slot for c in caches}) != B:
            raise ValueError("decode_step: two rows of the batch name the same stream")
        for c in caches:
            if self._frames[c.slot] >= self.max_frames:
                raise RuntimeError(f"MimiModel: stream in slot {c.slot} is at max_frames = {self.max_frames}")
        d_codes, d_slots, d_pcm = self._buffers(B)
        d_codes.copy_(codes.to(torch.int32), non_blocking=True)
        slots = tuple(c.slot for c in caches)
        if self._io_slots.get(B) != slots:      # the slot table of this batch size changes only when streams come and go
            d_slots.copy_(torch.tensor(slots, dtype=torch.int32), non_blocking=True)
            self._io_slots[B] = slots
        _capi.check(self._lib.smol_mimi_decode_step(self._h, C.c_void_p(d_codes.data_ptr()), C.c_void_p(d_slots.data_ptr()), B,
                                                    C.c_void_p(d_pcm.data_ptr()), C.c_void_p(self._stream())))
        for c in caches:
            self._frames[c.slot] += 1
            c.frames = self._frames[c.slot]
        return d_pcm.view(B, 1, self.samples_per_frame)

    def decode(self, audio_codes: torch.Tensor, cache: Optional[Sequence[MimiCache]] = None) -> torch.Tensor:
        """codes [B, n_q, T] -> PCM [B, 1, T * samples_per_frame] as a run of streaming steps over fresh (or the given) streams.
        With ``upsample_carry=True`` this equals the reference's whole-sequence ``decode`` (codec/mimi.py:88-100); with the
        default it is what a run of the reference's ``decode_step`` calls produces."""
        B, _, T = audio_codes.shape
        own = cache is None
        caches = [self.make_cache() for _ in range(B)] if own else list(cache)
        out = torch.empty(B, 1, T * self.samples_per_frame, dtype=torch.float32, device=self.device)
        codes = audio_codes.to(self.device)
        for t in range(T):
            out[:, :, t * self.samples_per_frame:(t + 1) * self.samples_per_frame] = self.decode_step(codes[:, :, t], caches)
        if own:
            for c in caches:
                self.release_cache(c)
        return out

    def flops_per_frame(self) -> int:
        """Multiply-adds x 2 of one decode_step of one stream, attention excluded (it grows with the history)."""
        c, s = self.config, self.config.seanet
        D, F = c.transformer.d_model, c.transformer.dim_feedforward
        macs = 2 * c.rvq.codebook_dim * D                                         # output projections
        macs += 2 * c.transformer.num_layers * (4 * D * D + 2 * D * F)            # two positions per frame
        ch, T = s.n_filters * 2 ** len(s.ratios), 2
        macs += T * s.kernel_size * D * ch
        for r in s.ratios:
            macs += T * 2 * ch * (r * ch // 2)                                    # transposed convolution: 2 taps per output
            T, ch = T * r, ch // 2
            macs += T * (s.residual_kernel_size * ch * (ch // 2) + (ch // 2) * ch)
        macs += T * s.last_kernel_size * ch
        return 2 * macs

    # ---- test / profiling hooks -----------------------------------------------------------------------------------------
    def _base(self) -> int:
        return _aligned(self._ws)

    def _flat(self, dtype) -> torch.Tensor:
        d = self._base() - self._ws.data_ptr()
        n = int(self._lib.smol_mimi_workspace_bytes(self._h))
        return self._ws[d: d + n].view(dtype)

    @property
    def launches_per_step(self) -> int:
        return int(self._lib.smol_mimi_launches_per_step(self._h))

    def debug_rows(self, name: str, slot: int, rows: int, cols: int) -> torch.Tensor:
        stride = C.c_int64()
        p = self._lib.smol_mimi_debug_buffer(self._h, name.encode(), C.byref(stride))
        if not p:
            raise KeyError(name)
        off = (p - self._base()) // 4 + slot * stride.value
        return self._flat(torch.float32)[off: off + rows * cols].view(rows, cols).clone()

    def overflowed(self) -> bool:
        p = self._lib.smol_mimi_error_word(self._h)
        return bool(self._flat(torch.int32)[(p - self._base()) // 4].item())


def load_mimi(path: str, format: str = "fp32", encode_max_samples: int = 0, encode_max_clips: int = 1, **kw) -> MimiModel:
    """codec/mimi.py:107 -- from a local model.safetensors (there is no hub access here).  Only fp32 is built: it is the
    reference's default and what its callers use (`load_mimi()` in __init__.py:54).  ``encode_max_samples > 0`` also
    builds the encoder (``MimiModel.encode``) for that many samples per call."""
    if format != "fp32":
        raise ValueError("load_mimi: only format='fp32' is built")
    return MimiModel.from_safetensors(path, encode_max_samples=encode_max_samples, encode_max_clips=encode_max_clips, **kw)
