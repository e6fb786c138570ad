"""The Mimi encoder's oracle (oracle/mimi_encode_oracle.py) against the goldens made from transformers' MimiModel.encode
(tools/make_mimi_encode_goldens.py), the seeded test audio, the seeded encoder weights, and the encoder's C ABI checks that
need no GPU."""
import ctypes
import hashlib

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR
from mimi_encode_util import check_codes, check_latent
from oracle.mimi_encode_oracle import MimiEncodeOracle
from smoltts_b200.synth import make_mimi_state_dict, make_test_audio, mimi_state_dict_shapes

CLIPS = ("a", "b", "c")


@pytest.fixture(scope="module")
def golden():
    return np.load(f"{GOLDEN_DIR}/mimi_encode.npz")


@pytest.fixture(scope="module")
def oracle():
    return MimiEncodeOracle(make_mimi_state_dict(0, encoder=True))


def test_test_audio_reproduces_the_stored_checksums(golden):
    for c in CLIPS:
        x = make_test_audio(int(golden[f"{c}_seed"]), int(golden[f"{c}_n"]))
        assert x.dtype == torch.float32 and x.shape == (int(golden[f"{c}_n"]),)
        assert hashlib.sha256(x.numpy().astype("<f4").tobytes()).hexdigest() == str(golden[f"{c}_sha256"])


@pytest.mark.parametrize("clip", CLIPS)
def test_oracle_encode_matches_transformers(golden, oracle, clip):
    n = int(golden[f"{clip}_n"])
    x = make_test_audio(int(golden[f"{clip}_seed"]), n)
    with torch.no_grad():
        codes, z = oracle.encode(x, return_latent=True)
    T = -(-n // 1920)
    assert codes.shape == (1, 8, T) and z.shape == (1, 512, T)
    check_latent(f"oracle {clip}", z[0].numpy(), golden[f"{clip}_latent"], 2e-5)
    check_codes(f"oracle {clip}", codes[0].numpy(), golden[f"{clip}_codes"], golden[f"{clip}_gap"])


def test_padding_is_per_layer_not_of_the_audio(oracle):
    """Zero-padding the clip to a multiple of 1920 samples is not the same computation (a conv of zeros plus its bias is
    not zero), so the encoder must pad at every strided layer."""
    x = make_test_audio(5, 1921)
    with torch.no_grad():
        _, z = oracle.encode(x, return_latent=True)
        _, zp = oracle.encode(torch.cat([x, torch.zeros(2 * 1920 - 1921)]), return_latent=True)
    assert z.shape == zp.shape == (1, 512, 2)
    assert (z - zp).abs().max() > 1e-3


def test_encoder_keys_only_add_to_the_decoder_state_dict():
    base = make_mimi_state_dict(0)
    both = make_mimi_state_dict(0, encoder=True)
    assert list(both)[: len(base)] == list(base)
    for k, v in base.items():
        assert torch.equal(both[k], v), k
    extra = set(both) - set(base)
    assert len(extra) == 2 + 4 * 6 + 2 + 8 * 12 + 1 + 2
    assert set(mimi_state_dict_shapes()) == set(base)
    assert {k.split(".")[0] for k in extra} == {"encoder", "encoder_transformer", "downsample", "quantizer"}


def _enc_config(**over):
    from smoltts_b200 import _capi

    c = _capi.SmolMimiEncoderConfig(n_q=8, codebook_size=2048, codebook_dim=256, dim=512, n_layers=8, n_heads=8, head_dim=64,
                                    ffn=2048, n_filters=64, n_ratios=4, kernel=7, res_kernel=3, last_kernel=3, max_clips=4,
                                    max_samples=240_000, window=250, norm_eps=1e-5, codebook_eps=1e-5)
    for i, r in enumerate((8, 6, 5, 4)):
        c.ratios[i] = r
    for k, v in over.items():
        setattr(c, k, v)
    return c


def test_encoder_create_validates_shapes_and_capacities_without_a_gpu():
    from smoltts_b200 import _capi

    lib = _capi.load()
    h = ctypes.c_void_p()
    assert lib.smol_mimi_encoder_create(ctypes.byref(_enc_config()), ctypes.byref(h)) == 0
    assert lib.smol_mimi_encoder_samples_per_frame(h) == 1920
    small = lib.smol_mimi_encoder_workspace_bytes(h)
    # the packed weights of the encode half alone are 40+ M parameters
    assert small > 40e6 * 4
    n = (ctypes.c_int64 * 1)(1920)
    assert lib.smol_mimi_encode(h, ctypes.c_void_p(8), n, 1, ctypes.c_void_p(8), None) == _capi.SMOL_ERR_UNBOUND
    assert b"bound" in lib.smol_last_error()
    lib.smol_mimi_encoder_destroy(h)
    h2 = ctypes.c_void_p()
    assert lib.smol_mimi_encoder_create(ctypes.byref(_enc_config(max_samples=2_400_000)), ctypes.byref(h2)) == 0
    big = lib.smol_mimi_encoder_workspace_bytes(h2)
    assert big > small + 9 * 240_000 * 160 * 4 * 0.9, (small, big)
    lib.smol_mimi_encoder_destroy(h2)
    for bad, code in ((dict(head_dim=48), _capi.SMOL_ERR_INVALID), (dict(max_clips=0), _capi.SMOL_ERR_INVALID),
                      (dict(max_samples=0), _capi.SMOL_ERR_INVALID), (dict(window=0), _capi.SMOL_ERR_UNSUPPORTED),
                      (dict(max_clips=100_000), _capi.SMOL_ERR_CAPACITY), (dict(n_filters=6), _capi.SMOL_ERR_UNSUPPORTED),
                      (dict(codebook_size=102), _capi.SMOL_ERR_UNSUPPORTED)):
        assert lib.smol_mimi_encoder_create(ctypes.byref(_enc_config(**bad)), ctypes.byref(h2)) == code, bad
        assert lib.smol_last_error()
