"""The C-ABI library builds for sm_100a, loads without a GPU and exports every symbol that
include/smoltts_b200.h declares (no compute calls here)."""
import ctypes
import os
import re

import pytest

from conftest import ROOT


def _declared():
    text = "".join(open(os.path.join(ROOT, "include", h)).read() for h in sorted(os.listdir(os.path.join(ROOT, "include"))) if h.endswith(".h"))
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(smol_[a-z_0-9]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    from smoltts_b200 import _capi, build

    path = build.build()
    assert os.path.exists(path)
    lib = ctypes.CDLL(path)
    names = _declared()
    assert len(names) >= 25
    for n in names:
        assert hasattr(lib, n), f"{n} declared in the header but not exported by {path}"
    assert set(names) == set(_capi.PROTOTYPES), (set(names) ^ set(_capi.PROTOTYPES))
    assert _capi.load().smol_abi_version() == _capi.SMOL_ABI_VERSION


def test_create_validates_shapes_without_a_gpu():
    """smol_create is pure host code: shape checks and error strings work on the CPU box."""
    from smoltts_b200 import _capi
    from smoltts_b200.config import named_config

    lib = _capi.load()
    cfg = named_config("smoltts_byte_150m")

    def make(**over):
        kw = dict(dim=cfg.dim, n_layer=cfg.n_layer, n_head=cfg.n_head, n_local_heads=cfg.n_local_heads, head_dim=64,
                  intermediate_size=cfg.intermediate_size, vocab_size=cfg.vocab_size, fast_dim=cfg.fast_dim,
                  n_fast_layer=cfg.n_fast_layer, fast_n_head=cfg.fast_n_head, fast_n_local_heads=cfg.fast_n_local_heads,
                  fast_head_dim=64, fast_intermediate_size=cfg.fast_intermediate_size, codebook_size=2048, num_codebooks=8,
                  duplicate_code_0=1, depthwise_wte=1, depthwise_output=1, tie_word_embeddings=1, max_seq_len=2048,
                  max_batch=4, page_size=32, semantic_start_id=320, semantic_end_id=2367, im_end_id=270, mlx_embed_mask=0,
                  norm_eps=1e-5)
        kw.update(over)
        return _capi.SmolConfig(**kw)

    h = ctypes.c_void_p()
    assert lib.smol_create(ctypes.byref(make()), ctypes.byref(h)) == 0
    assert lib.smol_phase_count(h) == 5 * 10 + 2 + 8 * (4 * 4 + 2) == 196
    assert lib.smol_kv_page_bytes(h) == 10 * 2 * 4 * 32 * 64 * 2
    assert lib.smol_workspace_bytes(h) > 0
    # compute calls before binding fail loudly instead of touching a device
    b = _capi.SmolBatch()
    assert lib.smol_slow_step(h, ctypes.byref(b), 1, 1, None) == _capi.SMOL_ERR_UNBOUND
    assert b"bound" in lib.smol_last_error()
    # "mode" takes 0 and 2; 1 (one launch per phase) was removed and is refused without changing the mode
    assert lib.smol_set_option(h, b"mode", 1) == _capi.SMOL_ERR_INVALID
    assert b"mode 1" in lib.smol_last_error() and b"removed" in lib.smol_last_error()
    assert lib.smol_get_option(h, b"mode") == 2
    for mode in (0, 2):
        assert lib.smol_set_option(h, b"mode", mode) == 0
        assert lib.smol_get_option(h, b"mode") == mode
    lib.smol_destroy(h)
    h2 = ctypes.c_void_p()
    assert lib.smol_create(ctypes.byref(make(fast_dim=512, fast_n_head=8)), ctypes.byref(h2)) == _capi.SMOL_ERR_UNSUPPORTED
    assert b"fast_project_in" in lib.smol_last_error()
    assert lib.smol_create(ctypes.byref(make(head_dim=128)), ctypes.byref(h2)) == _capi.SMOL_ERR_UNSUPPORTED


@pytest.mark.parametrize("size,overrides", [("smoltts_byte_tiny", {}), ("smoltts_byte_70m", {}), ("smoltts_byte_150m", {}),
                                            ("smoltts_byte_tiny", {"duplicate_code_0": False})])
def test_ll_regions_follow_the_frame_program(size, overrides):
    """smol_ll_region (host code: smol_create alone) against a restatement of ll_phase_words / decode_phase: one region per
    phase, laid end to end for 8 sequences x 8 replicas, inside the workspace."""
    from ll2_checks import decode_phase, phase_count, phase_words
    from smoltts_b200 import _capi
    from smoltts_b200.config import named_config

    lib = _capi.load()
    cfg = named_config(size, **overrides)
    c = _capi.SmolConfig(
        dim=cfg.dim, n_layer=cfg.n_layer, n_head=cfg.n_head, n_local_heads=cfg.n_local_heads, head_dim=64,
        intermediate_size=cfg.intermediate_size, vocab_size=cfg.vocab_size, fast_dim=cfg.fast_dim, n_fast_layer=cfg.n_fast_layer,
        fast_n_head=cfg.fast_n_head, fast_n_local_heads=cfg.fast_n_local_heads, fast_head_dim=64,
        fast_intermediate_size=cfg.fast_intermediate_size, codebook_size=cfg.codebook_size, num_codebooks=cfg.num_codebooks,
        duplicate_code_0=int(cfg.duplicate_code_0), depthwise_wte=int(cfg.depthwise_wte), depthwise_output=int(cfg.depthwise_output),
        tie_word_embeddings=int(cfg.tie_word_embeddings), max_seq_len=512, max_batch=8, page_size=32, semantic_start_id=320,
        semantic_end_id=320 + cfg.codebook_size - 1, im_end_id=270, mlx_embed_mask=0, norm_eps=cfg.norm_eps)
    h = ctypes.c_void_p()
    assert lib.smol_create(ctypes.byref(c), ctypes.byref(h)) == 0
    try:
        n = lib.smol_phase_count(h)
        assert n == phase_count(cfg)
        off, words = ctypes.c_uint32(), ctypes.c_uint32()
        end = 0
        for p in range(n):
            assert lib.smol_ll_region(h, p, ctypes.byref(off), ctypes.byref(words)) == 0
            kind = decode_phase(p, cfg.n_layer, cfg.n_fast_layer)[0]
            assert words.value == phase_words(cfg, p), f"phase {p} (kind {kind}): {words.value} words"
            assert off.value == end, f"phase {p}: region at word {off.value}, the previous one ends at {end}"
            end += words.value * 8 * 8
        assert end * 8 < lib.smol_workspace_bytes(h)
        for bad in (-1, n):
            assert lib.smol_ll_region(h, bad, ctypes.byref(off), ctypes.byref(words)) == _capi.SMOL_ERR_INVALID
    finally:
        lib.smol_destroy(h)


def test_mimi_create_validates_shapes_without_a_gpu():
    """smol_mimi_create is pure host code too."""
    from smoltts_b200 import _capi

    lib = _capi.load()

    def make(**over):
        c = _capi.SmolMimiConfig(n_q=8, codebook_size=2048, codebook_dim=256, dim=512, n_layers=8, n_heads=8, head_dim=64, ffn=2048,
                                 n_filters=64, n_ratios=4, kernel=7, res_kernel=3, last_kernel=3, max_streams=2, max_positions=512,
                                 window=0, upsample_carry=0, use_graph=1, norm_eps=1e-5, codebook_eps=1e-5)
        for i, r in enumerate((8, 6, 5, 4)):
            c.ratios[i] = r
        for k, v in over.items():
            setattr(c, k, v)
        return c

    h = ctypes.c_void_p()
    assert lib.smol_mimi_create(ctypes.byref(make()), ctypes.byref(h)) == 0
    assert lib.smol_mimi_samples_per_frame(h) == 1920
    ws = lib.smol_mimi_workspace_bytes(h)
    # packed weights of the decode half (44.4 M parameters) + two streams' KV caches and arenas
    assert 44.3e6 * 4 < ws < 44.3e6 * 4 + 2 * (8 * 2 * 512 * 512 * 4 + 3.0e6) + 4e6
    assert lib.smol_mimi_decode_step(h, ctypes.c_void_p(8), None, 1, ctypes.c_void_p(8), None) == _capi.SMOL_ERR_UNBOUND
    lib.smol_mimi_destroy(h)
    h2 = ctypes.c_void_p()
    assert lib.smol_mimi_create(ctypes.byref(make(head_dim=48)), ctypes.byref(h2)) == _capi.SMOL_ERR_INVALID
    assert lib.smol_mimi_create(ctypes.byref(make(max_positions=7)), ctypes.byref(h2)) == _capi.SMOL_ERR_INVALID
    assert lib.smol_mimi_create(ctypes.byref(make(max_positions=4000000)), ctypes.byref(h2)) == _capi.SMOL_ERR_CAPACITY
