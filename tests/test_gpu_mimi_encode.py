"""The Mimi encoder on the GPU (csrc/mimi_encoder.cu through include/smoltts_b200_mimi.h) against the goldens made from
transformers' MimiModel.encode and against the CPU oracle (oracle/mimi_encode_oracle.py), batch invariance, errors, the untouched
decoder, and SmolTTS.create_speaker from audio.

Bars: the latent z within 1e-4 x max |reference| (fp32 on both sides, different summation orders); codes under the margin
rule of mimi_encode_util.check_codes (a code may flip only where the reference's two nearest codebook rows are within a
relative 1e-3 of each other, and the rest of that frame is then not compared)."""
import ctypes

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from mimi_encode_util import check_codes, check_latent, oracle_gaps

pytestmark = pytest.mark.gpu

REL = 1e-4
_CACHE = {}


def _sd():
    from smoltts_b200.synth import make_mimi_state_dict

    if "sd" not in _CACHE:
        _CACHE["sd"] = make_mimi_state_dict(0, encoder=True)
    return _CACHE["sd"]


def _model(**kw):
    from smoltts_b200.mimi import MimiModel

    key = tuple(sorted(kw.items()))
    if key not in _CACHE:
        m = MimiModel(**kw)
        m.load_state_dict(_sd())
        _CACHE[key] = m
    return _CACHE[key]


def _encode(m, clips):
    """codes (list of [n_q, T_b] on the CPU) and latents (list of [dim, T_b]) of one encode call."""
    codes = m.encode([c.cuda() for c in clips])
    torch.cuda.synchronize()
    z = m.encoder_latent().cpu()
    out_z, r = [], 0
    for c in codes:
        out_z.append(z[r: r + c.shape[1]].t().contiguous())
        r += c.shape[1]
    return [c.cpu() for c in codes], out_z


def test_encode_matches_transformers_goldens():
    from smoltts_b200.synth import make_test_audio

    g = np.load(f"{GOLDEN_DIR}/mimi_encode.npz")
    clips = [make_test_audio(int(g[f"{c}_seed"]), int(g[f"{c}_n"])) for c in "abc"]
    m = _model(encode_max_samples=sum(len(c) for c in clips), encode_max_clips=3)
    codes, zs = _encode(m, clips)
    shares = []
    for name, c, z in zip("abc", codes, zs):
        T = -(-int(g[f"{name}_n"]) // 1920)
        assert c.shape == (8, T) and c.dtype == torch.int64
        check_latent(f"gpu {name} vs transformers", z.numpy(), g[f"{name}_latent"], REL)
        shares.append(check_codes(f"gpu {name} vs transformers", c.numpy(), g[f"{name}_codes"], g[f"{name}_gap"]))
    print("identical-frame shares vs transformers:", ", ".join(f"{s:.3f}" for s in shares))
    # the batched [B, 1, L] form of transformers' API
    x = torch.stack([clips[0][:96_000], clips[1][:96_000]])[:, None]
    both = m.encode(x.cuda())
    assert both.shape == (2, 8, 50) and both.dtype == torch.int64
    assert torch.equal(both[0].cpu(), m.encode([clips[0][:96_000].cuda()])[0].cpu())


@pytest.mark.parametrize("n", [1, 1919, 1920, 1921, 96_001, 1_440_000])
def test_encode_matches_the_oracle(n):
    from oracle.mimi_encode_oracle import MimiEncodeOracle
    from smoltts_b200.synth import make_test_audio

    x = make_test_audio(100 + n % 97, n)
    m = _model(encode_max_samples=1_440_000, encode_max_clips=1)
    codes, zs = _encode(m, [x])
    orc = MimiEncodeOracle(_sd())
    with torch.no_grad():
        want, z = orc.encode(x, return_latent=True)
    check_latent(f"gpu vs oracle n={n}", zs[0].numpy(), z[0].numpy(), REL)
    check_codes(f"gpu vs oracle n={n}", codes[0].numpy(), want[0].numpy(), oracle_gaps(orc, z, want))


def test_each_clip_is_encoded_as_if_alone_bit_for_bit():
    from smoltts_b200.synth import make_test_audio

    lens = [1921, 96_001, 1, 47_000, 240_000]
    clips = [make_test_audio(200 + i, n) for i, n in enumerate(lens)]
    m5 = _model(encode_max_samples=sum(lens), encode_max_clips=5)
    m8 = _model(encode_max_samples=2 * sum(lens), encode_max_clips=8)
    alone = [_encode(m5, [c]) for c in clips]
    batch_c, batch_z = _encode(m5, clips)
    rev_c, rev_z = _encode(m5, clips[::-1])
    other_c, other_z = _encode(m8, clips)
    for i in range(len(clips)):
        ac, az = alone[i][0][0], alone[i][1][0]
        assert ac.shape == (8, -(-lens[i] // 1920))
        for name, c, z in (("batch of 5", batch_c[i], batch_z[i]), ("reversed", rev_c[-1 - i], rev_z[-1 - i]),
                           ("max_clips 8", other_c[i], other_z[i])):
            assert torch.equal(c, ac), f"clip {i}: codes differ, {name} vs alone"
            assert torch.equal(z, az), f"clip {i}: latent bits differ, {name} vs alone"


def test_errors_write_nothing():
    from smoltts_b200 import _capi
    from smoltts_b200.synth import make_test_audio

    m = _model(encode_max_samples=10_000, encode_max_clips=2)
    lib = m._lib
    x = make_test_audio(9, 6_000).cuda()
    codes = torch.full((16, 8), -7, dtype=torch.int32, device="cuda")
    m.encode([x[:3_000]])
    torch.cuda.synchronize()
    z0 = m.encoder_latent()

    def call(lengths):
        h = (ctypes.c_int64 * len(lengths))(*lengths)
        rc = lib.smol_mimi_encode(m._enc, ctypes.c_void_p(x.data_ptr()), h, len(lengths), ctypes.c_void_p(codes.data_ptr()), None)
        return rc, lib.smol_last_error().decode()

    for lengths, want in (([6_000, 6_000], _capi.SMOL_ERR_CAPACITY), ([100, 100, 100], _capi.SMOL_ERR_CAPACITY),
                          ([100, 0], _capi.SMOL_ERR_INVALID), ([], _capi.SMOL_ERR_CAPACITY)):
        rc, msg = call(lengths) if lengths else (lib.smol_mimi_encode(m._enc, ctypes.c_void_p(x.data_ptr()), (ctypes.c_int64 * 1)(1), 0,
                                                                      ctypes.c_void_p(codes.data_ptr()), None), lib.smol_last_error().decode())
        assert rc == want, (lengths, rc, msg)
        assert msg
    torch.cuda.synchronize()
    assert (codes == -7).all(), "a refused call wrote codes"
    assert torch.equal(m.encoder_latent(), z0), "a refused call touched the workspace"
    with pytest.raises(_capi.SmolError):
        m.encode([x[:0]])
    with pytest.raises(RuntimeError, match="without an encoder"):
        _model(max_streams=2, max_frames=8).encode([x])


def test_decoder_is_untouched_by_the_encoder():
    from smoltts_b200.mimi import MimiModel

    g = np.load(f"{GOLDEN_DIR}/mimi.npz")
    codes = torch.from_numpy(g["codes"]).long()
    plain = MimiModel(max_streams=2, max_frames=16, upsample_carry=True)
    plain.load_state_dict(_sd())
    both = MimiModel(max_streams=2, max_frames=16, upsample_carry=True, encode_max_samples=48_000, encode_max_clips=2)
    both.load_state_dict(_sd())
    assert both._enc is not None and plain._enc is None
    a, b = plain.decode(codes).cpu(), both.decode(codes).cpu()
    assert torch.equal(a, b), "the decoder's PCM changed when the encoder is built"
    assert np.abs(a.numpy() - g["full"]).max() <= 1e-4 * np.abs(g["full"]).max()


def test_create_speaker_from_audio_end_to_end():
    from gpu_util import model_and_oracle
    from smoltts_b200 import GenerationSettings, MimiModel, PromptEncoder, SmolTTS, byte_level_tokenizer
    from smoltts_b200.synth import make_test_audio

    cfg, _, lm, _ = model_and_oracle("smoltts_byte_tiny", max_batch=8, max_seq_len=1024)
    enc = PromptEncoder.from_model(byte_level_tokenizer(cfg.codebook_size), lm)
    codec = MimiModel(max_streams=2, max_frames=32, upsample_carry=True, encode_max_samples=240_000, encode_max_clips=2)
    codec.load_state_dict(_sd())
    tts = SmolTTS(lm, enc, codec, settings=GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=9))
    audio = make_test_audio(11, 240_000)
    text = ("This reference clip is ten seconds of seeded sines and noise, and its transcript is long on purpose so that the "
            "voice-clone prompt built from it reaches the length of the reference notebook's example, which is a little over "
            "five hundred tokens; every byte of this sentence is one token of the byte-level tokenizer, and the audio adds one "
            "column per Mimi frame. It is read slowly and clearly.")
    prefix = tts.create_speaker([{"text": text, "audio": audio}])
    codes = codec.encode([audio.cuda()])[0].cpu()
    assert codes.shape == (8, 125)
    want = enc.create_speaker([{"text": text, "codes": codes}])
    assert torch.equal(prefix, want)
    assert prefix.shape[1] >= 500, prefix.shape
    mixed = tts.create_speaker([{"text": "a", "codes": codes}, {"text": text, "audio": audio}], system_prompt="clone")
    assert torch.equal(mixed, enc.create_speaker([{"text": "a", "codes": codes}, {"text": text, "codes": codes}], system_prompt="clone"))
    pcm = tts("Hello from a cloned voice.", speaker=prefix)
    assert pcm.dtype == np.float32 and np.isfinite(pcm).all()
    no_enc = SmolTTS(lm, enc, MimiModel(max_streams=1, max_frames=8))
    no_enc.codec.load_state_dict(_sd())
    with pytest.raises(ValueError, match="no encoder"):
        no_enc.create_speaker([{"text": "x", "audio": audio}])
