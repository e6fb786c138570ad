"""Synthetic weights, prompts and token grids (SURVEY §8(d) "Synthetic inputs").

There is no network for checkpoints or datasets, so benchmarks and parity tests
use seeded random-init weights of the reference architecture and synthetic
byte-token prompts.  Everything here is deterministic in (name, seed) and does
not depend on generation order, so the GPU box regenerates bit-identical inputs.
"""
from __future__ import annotations

import hashlib
from typing import Dict, List, Optional

import torch

from .config import RQTransformerModelArgs

# Token ids of the byte-level tokenizer built by the reference recipe
# (reference: data_pipeline/scripts/create_bytelevel_init.py:15-57): 256 bytes,
# 15 control tokens, 49 speaker tokens, then codebook_size semantic tokens.
CONTROL_TOKENS = [
    "system", "user", "assistant", "<|british|>", "<|american|>", "<|male|>", "<|female|>",
    "<|unknown|>", "<|endoftext|>", "<|voice|>", "<|semantic|>", "<|pad|>", "<|epad|>",
    "<|im_start|>", "<|im_end|>",
]
TOK_SYSTEM, TOK_USER, TOK_ASSISTANT = 256, 257, 258
TOK_SEMANTIC, TOK_PAD = 266, 267
TOK_IM_START, TOK_IM_END = 269, 270
TOK_SPEAKER0 = 271
TOK_SEMANTIC0 = 320


def _key_seed(name: str, seed: int) -> int:
    h = hashlib.sha256(f"{seed}:{name}".encode()).digest()
    return int.from_bytes(h[:7], "little")


def _normal(name: str, shape, std: float, seed: int) -> torch.Tensor:
    g = torch.Generator(device="cpu")
    g.manual_seed(_key_seed(name, seed))
    return (torch.randn(*shape, generator=g, dtype=torch.float32) * std).to(torch.bfloat16)


def state_dict_shapes(cfg: RQTransformerModelArgs, flat_fast_output: bool = True) -> Dict[str, tuple]:
    """Key -> shape of the exported checkpoint (SURVEY §8(b) "Checkpoint layout";
    reference state_dict of modeling/model/rq_transformer.py + train/convert_safetensors.py:6-16)."""
    D, F, V = cfg.dim, cfg.intermediate_size, cfg.vocab_size
    Df, Ff = cfg.fast_dim, cfg.fast_intermediate_size
    C, N = cfg.codebook_size, cfg.num_codebooks
    shapes: Dict[str, tuple] = {
        "embeddings.weight": (V, D),
        "codebook_embeddings.weight": (N * C, D),
        "norm.weight": (D,),
        "fast_embeddings.weight": (cfg.fast_embedding_rows, Df),
        "fast_norm.weight": (Df,),
    }
    if not cfg.tie_word_embeddings:
        shapes["output.weight"] = (V, D)
    if cfg.fast_dim != cfg.dim:
        shapes["fast_project_in.weight"] = (Df, D)
        shapes["fast_project_in.bias"] = (Df,)
    for pre, n, d, f, rows in (("layers", cfg.n_layer, D, F, cfg.qkv_rows),
                               ("fast_layers", cfg.n_fast_layer, Df, Ff, cfg.fast_qkv_rows)):
        for l in range(n):
            p = f"{pre}.{l}."
            shapes[p + "attention.wqkv.weight"] = (rows, d)
            shapes[p + "attention.wo.weight"] = (d, d)
            shapes[p + "feed_forward.w1.weight"] = (f, d)
            shapes[p + "feed_forward.w3.weight"] = (f, d)
            shapes[p + "feed_forward.w2.weight"] = (d, f)
            shapes[p + "attention_norm.weight"] = (d,)
            shapes[p + "ffn_norm.weight"] = (d,)
    nf = cfg.max_fast_seqlen
    if cfg.depthwise_output:
        shapes["fast_output.weight"] = (nf * C, Df) if flat_fast_output else (nf, Df, C)
    else:
        shapes["fast_output.weight"] = (C, Df)
    return shapes


def make_state_dict(cfg: RQTransformerModelArgs, seed: int = 0, flat_fast_output: bool = True,
                    norm_jitter: float = 0.0) -> Dict[str, torch.Tensor]:
    """Seeded bf16 weights: every Linear/Embedding ~ N(0, initializer_range) as the
    reference's ``_init_weights`` does (rq_transformer.py:262-271); norm weights 1
    (optionally jittered so tests exercise the multiply); ``fast_output.weight``
    re-drawn N(0, initializer_range) because the reference leaves it at
    kaiming-uniform over a 3-D tensor, which makes codebook logits degenerate
    (SURVEY §7.1-0).  ``fast_output`` is always *generated* in the flat exported
    layout [(i*C + k), D] and reshaped for the 3-D trainer form on request."""
    std = cfg.initializer_range
    out: Dict[str, torch.Tensor] = {}
    for name, shape in state_dict_shapes(cfg, flat_fast_output=True).items():
        if name.endswith("norm.weight"):
            w = torch.ones(shape, dtype=torch.bfloat16)
            if norm_jitter:
                w = (1.0 + _normal(name, shape, norm_jitter, seed).float()).to(torch.bfloat16)
            out[name] = w
        elif name.endswith(".bias"):
            out[name] = _normal(name, shape, std, seed)
        else:
            out[name] = _normal(name, shape, std, seed)
    if cfg.depthwise_output and not flat_fast_output:
        out["fast_output.weight"] = flat_to_depthwise(out["fast_output.weight"], cfg)
    return out


def flat_to_depthwise(w_flat: torch.Tensor, cfg: RQTransformerModelArgs) -> torch.Tensor:
    """[(i*C + k), D] -> [i, D, k] (inverse of train/convert_safetensors.py:12-15)."""
    nf, C = cfg.max_fast_seqlen, cfg.codebook_size
    return w_flat.view(nf, C, -1).permute(0, 2, 1).contiguous()


def depthwise_to_flat(w3: torch.Tensor) -> torch.Tensor:
    """[i, D, k] -> [(i*C + k), D]; same result as the reference converter without
    its hard-coded 768 (train/convert_safetensors.py:14)."""
    nf, D, C = w3.shape
    return w3.permute(0, 2, 1).reshape(nf * C, D).contiguous()


def byte_prompt(n_bytes: int = 200, seed: int = 1, speaker: int = 0) -> List[int]:
    """Row-0 ids of a ChatML-framed synthetic byte prompt (MLX prompt format,
    reference: mlx_inference/src/smoltts_mlx/lm/utils/prompt.py:48-51 and
    mlx_inference/src/smoltts_mlx/__init__.py:142-150):
    <|im_start|>system\\n<|speaker:k|><|im_end|><|im_start|>user\\n<bytes><|im_end|><|im_start|>assistant\\n
    -> 12 + n_bytes tokens (212 for the 200-byte benchmark prompt)."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    body = torch.randint(0, 256, (n_bytes,), generator=g).tolist()
    return ([TOK_IM_START, TOK_SYSTEM, 10, TOK_SPEAKER0 + speaker, TOK_IM_END,
             TOK_IM_START, TOK_USER, 10] + body + [TOK_IM_END, TOK_IM_START, TOK_ASSISTANT, 10])


def prompt_grid(row0: List[int], cfg: RQTransformerModelArgs) -> torch.Tensor:
    """[1+N', S] int64 token grid: text ids in row 0, zeros below."""
    g = torch.zeros(cfg.n_rows, len(row0), dtype=torch.int64)
    g[0] = torch.tensor(row0, dtype=torch.int64)
    return g


def teacher_grid(cfg: RQTransformerModelArgs, n_text: int, n_audio: int, batch: int = 1,
                 seed: int = 7, zero_code_at: Optional[int] = None) -> torch.Tensor:
    """Random teacher-forcing grid [B, 1+N', n_text+n_audio]: text columns then audio
    columns with row0 = 320 + first depth code (dup0) as real data has
    (SURVEY §8(c) protocol 1).  ``zero_code_at`` forces row-1 code 0 at one audio
    column to exercise the PyTorch embed-mask quirk (§8(g)-1)."""
    g = torch.Generator(device="cpu")
    g.manual_seed(seed)
    R, C = cfg.n_rows, cfg.codebook_size
    S = n_text + n_audio
    grid = torch.zeros(batch, R, S, dtype=torch.int64)
    grid[:, 0, :n_text] = torch.randint(0, 256, (batch, n_text), generator=g)
    if n_audio:
        codes = torch.randint(0, C, (batch, R - 1, n_audio), generator=g)
        if zero_code_at is not None:
            codes[:, 0, zero_code_at] = 0
        grid[:, 1:, n_text:] = codes
        if cfg.duplicate_code_0:
            grid[:, 0, n_text:] = TOK_SEMANTIC0 + codes[:, 0]
        else:
            grid[:, 0, n_text:] = TOK_SEMANTIC0 + torch.randint(0, C, (batch, n_audio), generator=g)
    return grid


# ---- Mimi decoder (SURVEY §8(f)-2): seeded weights under kyutai/mimi's state-dict keys ----------------------------------
def mimi_state_dict_shapes(n_q: int = 8, codebook_size: int = 2048, codebook_dim: int = 256, dim: int = 512, n_layers: int = 8,
                           ffn: int = 2048, n_filters: int = 64, ratios=(8, 6, 5, 4), kernel: int = 7, res_kernel: int = 3,
                           last_kernel: int = 3, encoder: bool = False) -> Dict[str, tuple]:
    """Key -> shape of the decode half of kyutai/mimi's model.safetensors (the keys the reference's load_mimi() maps onto
    its module tree, mlx_inference/src/smoltts_mlx/codec/mimi.py:107-156; torch layouts: Conv1d [out, in, k],
    ConvTranspose1d [in, out, k]).  ``encoder=True`` appends the encode half (``encoder.*``, ``encoder_transformer.*``,
    ``downsample`` and the quantizers' ``input_proj``) after those keys."""
    s: Dict[str, tuple] = {}
    for half, n in (("semantic", 1), ("acoustic", n_q - 1)):
        p = f"quantizer.{half}_residual_vector_quantizer"
        for i in range(n):
            s[f"{p}.layers.{i}.codebook.embed_sum"] = (codebook_size, codebook_dim)
            s[f"{p}.layers.{i}.codebook.cluster_usage"] = (codebook_size,)
        s[f"{p}.output_proj.weight"] = (dim, codebook_dim, 1)
    s["upsample.conv.weight"] = (dim, 1, 4)
    for l in range(n_layers):
        p = f"decoder_transformer.layers.{l}"
        for w in ("q_proj", "k_proj", "v_proj", "o_proj"):
            s[f"{p}.self_attn.{w}.weight"] = (dim, dim)
        s[f"{p}.mlp.fc1.weight"] = (ffn, dim)
        s[f"{p}.mlp.fc2.weight"] = (dim, ffn)
        for nm in ("input_layernorm", "post_attention_layernorm"):
            s[f"{p}.{nm}.weight"] = (dim,)
            s[f"{p}.{nm}.bias"] = (dim,)
        s[f"{p}.self_attn_layer_scale.scale"] = (dim,)
        s[f"{p}.mlp_layer_scale.scale"] = (dim,)
    ch = n_filters * 2 ** len(ratios)
    s["decoder.layers.0.conv.weight"] = (ch, dim, kernel)
    s["decoder.layers.0.conv.bias"] = (ch,)
    idx = 1
    for r in ratios:
        s[f"decoder.layers.{idx + 1}.conv.weight"] = (ch, ch // 2, 2 * r)
        s[f"decoder.layers.{idx + 1}.conv.bias"] = (ch // 2,)
        ch //= 2
        s[f"decoder.layers.{idx + 2}.block.1.conv.weight"] = (ch // 2, ch, res_kernel)
        s[f"decoder.layers.{idx + 2}.block.1.conv.bias"] = (ch // 2,)
        s[f"decoder.layers.{idx + 2}.block.3.conv.weight"] = (ch, ch // 2, 1)
        s[f"decoder.layers.{idx + 2}.block.3.conv.bias"] = (ch,)
        idx += 3
    s[f"decoder.layers.{idx + 1}.conv.weight"] = (1, ch, last_kernel)
    s[f"decoder.layers.{idx + 1}.conv.bias"] = (1,)
    if encoder:
        # SEANet encoder: conv k7, then per ratio (reversed) [residual block, ELU, conv k = 2 r, stride r], ELU, conv k3
        s["encoder.layers.0.conv.weight"] = (n_filters, 1, kernel)
        s["encoder.layers.0.conv.bias"] = (n_filters,)
        ch, idx = n_filters, 1
        for r in reversed(ratios):
            s[f"encoder.layers.{idx}.block.1.conv.weight"] = (ch // 2, ch, res_kernel)
            s[f"encoder.layers.{idx}.block.1.conv.bias"] = (ch // 2,)
            s[f"encoder.layers.{idx}.block.3.conv.weight"] = (ch, ch // 2, 1)
            s[f"encoder.layers.{idx}.block.3.conv.bias"] = (ch,)
            s[f"encoder.layers.{idx + 2}.conv.weight"] = (2 * ch, ch, 2 * r)
            s[f"encoder.layers.{idx + 2}.conv.bias"] = (2 * ch,)
            ch, idx = 2 * ch, idx + 3
        s[f"encoder.layers.{idx + 1}.conv.weight"] = (dim, ch, last_kernel)
        s[f"encoder.layers.{idx + 1}.conv.bias"] = (dim,)
        for l in range(n_layers):
            p = f"encoder_transformer.layers.{l}"
            for w in ("q_proj", "k_proj", "v_proj", "o_proj"):
                s[f"{p}.self_attn.{w}.weight"] = (dim, dim)
            s[f"{p}.mlp.fc1.weight"] = (ffn, dim)
            s[f"{p}.mlp.fc2.weight"] = (dim, ffn)
            for nm in ("input_layernorm", "post_attention_layernorm"):
                s[f"{p}.{nm}.weight"] = (dim,)
                s[f"{p}.{nm}.bias"] = (dim,)
            s[f"{p}.self_attn_layer_scale.scale"] = (dim,)
            s[f"{p}.mlp_layer_scale.scale"] = (dim,)
        s["downsample.conv.weight"] = (dim, dim, 4)
        for half in ("semantic", "acoustic"):
            s[f"quantizer.{half}_residual_vector_quantizer.input_proj.weight"] = (codebook_dim, dim, 1)
    return s


def make_test_audio(seed: int, n_samples: int, sampling_rate: int = 24_000) -> torch.Tensor:
    """Seeded 1-D fp32 test clip: three sines (seeded frequencies 80 .. 2000 Hz, amplitudes 0.1 .. 0.3) plus seeded Gaussian
    noise of std 0.05.  Computed in float64 with numpy's PCG64 and rounded once to fp32, so every machine regenerates the
    same samples."""
    import numpy as np

    rng = np.random.default_rng(seed)
    freq = rng.uniform(80.0, 2000.0, 3)
    amp = rng.uniform(0.1, 0.3, 3)
    phase = rng.uniform(0.0, 2 * np.pi, 3)
    t = np.arange(n_samples, dtype=np.float64) / sampling_rate
    x = (amp[:, None] * np.sin(2 * np.pi * freq[:, None] * t[None, :] + phase[:, None])).sum(0)
    x = x + 0.05 * rng.standard_normal(n_samples)
    return torch.from_numpy(x.astype(np.float32))


def make_mimi_state_dict(seed: int = 0, **dims) -> Dict[str, torch.Tensor]:
    """Seeded fp32 weights of the Mimi decoder (and with ``encoder=True`` of the encoder too).  Scales keep every stage O(1)
    (fan-in scaled weights, layer scales of 0.1 .. 0.3 instead of the trained 0.01 .. so that all eight transformer layers
    matter in a parity check).  Every key is seeded by its name: the encoder keys leave the decoder's values unchanged."""
    out: Dict[str, torch.Tensor] = {}
    for name, shape in mimi_state_dict_shapes(**dims).items():
        g = torch.Generator(device="cpu")
        g.manual_seed(_key_seed("mimi." + name, seed))
        if name.endswith("cluster_usage"):
            t = 0.5 + 1.5 * torch.rand(*shape, generator=g)
        elif name.endswith("layer_scale.scale"):
            t = 0.1 + 0.2 * torch.rand(*shape, generator=g)
        elif name.endswith("layernorm.weight"):
            t = 1.0 + 0.1 * torch.randn(*shape, generator=g)
        elif name.endswith(".bias"):
            t = 0.05 * torch.randn(*shape, generator=g)
        elif name.endswith("embed_sum"):
            t = torch.randn(*shape, generator=g)
        elif name == "upsample.conv.weight":
            t = 0.7 * torch.randn(*shape, generator=g)
        else:
            if name.startswith("decoder.") and len(shape) == 3:
                # Conv1d [out, in, k]: fan-in = in * k; ConvTranspose1d [in, out, k = 2 stride]: two taps per output
                is_tr = shape[2] >= 8 and not name.startswith("decoder.layers.0.")
                fan = shape[0] * 2 if is_tr else shape[1] * shape[2]
            else:
                fan = shape[1] * (shape[2] if len(shape) == 3 else 1)
            t = torch.randn(*shape, generator=g) * (1.4 / fan ** 0.5)
        out[name] = t.to(torch.float32).contiguous()
    return out
