"""CPU oracle of the Mimi encoder (PCM -> codes) -- TEST INFRASTRUCTURE, never imported by the product.

Restates, with torch CPU fp32 ops, transformers 5.5.0 `MimiModel(MimiConfig(num_quantizers=8)).encode` (the model the
reference's MLX codec mirrors); `tests/test_mimi_encode_oracle_golden.py` pins it against goldens produced from transformers
(`tools/make_mimi_encode_goldens.py`):

* SEANet encoder   `encoder.layers.*`: conv k7, then per ratio (reversed) [residual block, ELU, conv k = 2 r stride r], ELU,
                   conv k3; every causal convolution pads k - stride zeros on the left of its input, and a strided one pads
                   zeros on the right up to a multiple of its stride (T_out = ceil(T_in / r))
* transformer      `encoder_transformer.layers.*`: the decoder's layer (`MimiOracle.transformer`, reused on the same keys
                   under the encoder's prefix) with a causal sliding window of 250 positions, positions from 0 per clip
* downsample       conv k4 stride 2, no bias, replicate padding
* split RVQ        the semantic codebook on its own projection of the latent z; the acoustic residual starts from the
                   acoustic projection of the same z and runs through n_q - 1 codebooks (first-index argmin of the
                   Euclidean distance, torch.cdist as transformers computes it)
"""
from __future__ import annotations

from typing import Dict, Optional

import torch
import torch.nn.functional as F

from oracle.mimi_oracle import MimiDims, MimiOracle


class MimiEncodeOracle:
    def __init__(self, sd: Dict[str, torch.Tensor], dims: Optional[MimiDims] = None, window: int = 250):
        self.d = dims or MimiDims()
        self.sd = {k: v.detach().to(torch.float32) for k, v in sd.items()}
        self.window = window
        # the encoder transformer is the decoder's layer under other keys: the decoder oracle on those keys
        pre = "encoder_transformer."
        self._xf = MimiOracle({"decoder_transformer." + k[len(pre):]: v for k, v in self.sd.items() if k.startswith(pre)},
                              self.d, window=window)

    def _conv(self, key: str, x: torch.Tensor, k: int, stride: int = 1, replicate: bool = False, bias: bool = True):
        """Causal Conv1d of transformers' MimiConv1d: k - stride rows on the left, and on the right whatever makes the
        length a multiple of the stride; zeros, or copies of the edge rows."""
        T = x.shape[-1]
        extra = -(-T // stride) * stride - T
        x = F.pad(x, (k - stride, extra), mode="replicate" if replicate else "constant")
        return F.conv1d(x, self.sd[key + ".conv.weight"], self.sd[key + ".conv.bias"] if bias else None, stride=stride)

    def seanet(self, pcm: torch.Tensor) -> torch.Tensor:
        """[B, 1, L] -> [B, dim, ceil(L / prod(ratios))]"""
        d = self.d
        x = self._conv("encoder.layers.0", pcm, d.kernel)
        idx = 1
        for r in reversed(d.ratios):
            h = self._conv(f"encoder.layers.{idx}.block.1", F.elu(x), d.res_kernel)
            x = x + self._conv(f"encoder.layers.{idx}.block.3", F.elu(h), 1)
            x = self._conv(f"encoder.layers.{idx + 2}", F.elu(x), 2 * r, stride=r)
            idx += 3
        return self._conv(f"encoder.layers.{idx + 1}", F.elu(x), d.last_kernel)

    def latent(self, pcm: torch.Tensor) -> torch.Tensor:
        """The pre-quantizer latent z [B, dim, ceil(L / 1920)]: SEANet encoder, encoder transformer, downsample."""
        x = self.seanet(pcm)
        x = self._xf.transformer(x.transpose(1, 2)).transpose(1, 2)
        return self._conv("downsample", x, 2 * self.d.up_stride, stride=self.d.up_stride, replicate=True, bias=False)

    def quantize(self, z: torch.Tensor) -> torch.Tensor:
        """Split RVQ: z [B, dim, T] -> codes [B, n_q, T]."""
        d, sd = self.d, self.sd
        codes = []
        for prefix, n in (("quantizer.semantic_residual_vector_quantizer", 1),
                          ("quantizer.acoustic_residual_vector_quantizer", d.n_q - 1)):
            r = F.conv1d(z, sd[f"{prefix}.input_proj.weight"]).transpose(1, 2)         # [B, T, codebook_dim]
            for i in range(n):
                es = sd[f"{prefix}.layers.{i}.codebook.embed_sum"]
                emb = es / torch.clamp(sd[f"{prefix}.layers.{i}.codebook.cluster_usage"], min=d.cb_eps)[:, None]
                idx = torch.cdist(r, emb[None].expand(r.shape[0], -1, -1), p=2).argmin(dim=-1)   # first index on a tie
                r = r - F.embedding(idx, emb)
                codes.append(idx)
        return torch.stack(codes, dim=1)

    def encode(self, pcm: torch.Tensor, return_latent: bool = False):
        """PCM [B, 1, L] (or one 1-D clip) -> codes [B, n_q, ceil(L / 1920)] (and the latent z [B, dim, T])."""
        if pcm.dim() == 1:
            pcm = pcm[None, None]
        z = self.latent(pcm.to(torch.float32))
        codes = self.quantize(z)
        return (codes, z) if return_latent else codes
