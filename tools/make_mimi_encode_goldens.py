"""Golden vectors of the Mimi encoder (tests/golden/mimi_encode.npz), produced from Hugging Face transformers' MimiModel
(transformers 5.5.0), the model the repository pins its codec to.

Weights: smoltts_b200.synth.make_mimi_state_dict(0, encoder=True) loaded into MimiModel(MimiConfig(num_quantizers=8)).
Audio: smoltts_b200.synth.make_test_audio(seed, n) for three clips, each encoded ALONE (transformers cannot batch clips of
different lengths):
  a  12.0 s      (seed 1)  300 transformer positions, past the 250-position sliding window
  b  7.3 s + 1   (seed 2)  not a multiple of 1920 samples
  c  0.05 s      (seed 3)  less than one frame: one code column
Stored per clip: the codes [n_q, T], the pre-quantizer latent z [dim, T] (the downsample's output), the fp64 relative gap
between the nearest and the second-nearest codebook row of every (codebook, frame) [n_q, T] -- where a code may flip under
a different summation order -- and the sha256 of the clip's fp32 samples.

    python tools/make_mimi_encode_goldens.py
"""
import hashlib
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from smoltts_b200.synth import make_mimi_state_dict, make_test_audio  # noqa: E402

CLIPS = {"a": (1, 288_000), "b": (2, 175_201), "c": (3, 1_200)}


def audio_sha256(x: torch.Tensor) -> str:
    return hashlib.sha256(x.numpy().astype("<f4").tobytes()).hexdigest()


def top2_gaps(hf, z: torch.Tensor, codes: torch.Tensor) -> np.ndarray:
    """[n_q, T]: (d_2 - d_1) / d_1 of the two nearest codebook rows, in fp64, along transformers' own residual path."""
    gaps = []
    q = hf.quantizer
    for rvq, sl in ((q.semantic_residual_vector_quantizer, slice(0, 1)), (q.acoustic_residual_vector_quantizer, slice(1, None))):
        r = rvq.input_proj(z)[0].t()                                   # [T, codebook_dim], fp32
        for layer, c in zip(rvq.layers, codes[0, sl]):
            emb = layer.codebook.embed
            d = torch.cdist(r.double(), emb.double()).sort(dim=-1).values
            gaps.append(((d[:, 1] - d[:, 0]) / d[:, 0].clamp(min=1e-300)).numpy())
            r = r - emb[c]
    return np.stack(gaps)


def main():
    from transformers import MimiConfig, MimiModel

    sd = make_mimi_state_dict(0, encoder=True)
    hf = MimiModel(MimiConfig(num_quantizers=8)).eval()
    res = hf.load_state_dict(sd, strict=False)
    assert not res.unexpected_keys, res.unexpected_keys
    assert not [k for k in res.missing_keys if not k.endswith("initialized")], res.missing_keys
    out = {}
    with torch.no_grad():
        for name, (seed, n) in CLIPS.items():
            x = make_test_audio(seed, n)
            codes = hf.encode(x[None, None], num_quantizers=8).audio_codes           # [1, 8, T]
            emb = hf.encoder(x[None, None])
            emb = hf.encoder_transformer(emb.transpose(1, 2))[0].transpose(1, 2)
            z = hf.downsample(emb)                                                  # [1, 512, T]
            assert torch.equal(hf.quantizer.encode(z, 8).transpose(0, 1), codes)
            gaps = top2_gaps(hf, z, codes)
            out[f"{name}_codes"] = codes[0].numpy().astype(np.int32)
            out[f"{name}_latent"] = z[0].numpy().astype(np.float32)
            out[f"{name}_gap"] = gaps.astype(np.float32)
            out[f"{name}_sha256"] = np.array(audio_sha256(x))
            out[f"{name}_n"] = np.array(n, dtype=np.int64)
            out[f"{name}_seed"] = np.array(seed, dtype=np.int64)
            print(name, n, "samples ->", tuple(codes.shape), "|z| max %.3g" % float(z.abs().max()),
                  "min gap %.3g" % float(gaps.min()), "gaps < 1e-3: %d" % int((gaps < 1e-3).sum()))
    path = os.path.join(ROOT, "tests", "golden", "mimi_encode.npz")
    np.savez_compressed(path, **out)
    print(path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
