"""ctypes binding of ``include/smoltts_b200.h`` (the C-ABI of the CUDA decode engine).

Loading never falls back to another implementation: if the shared library is missing
it is built with nvcc (``smoltts_b200.build``); if that is impossible the import
raises.  Struct layouts mirror the header field by field.
"""
from __future__ import annotations

import ctypes as C
import os

from . import build as _build

SMOL_ABI_VERSION = 2
SMOL_MAX_LAYERS = 64
SMOL_MAX_FAST_LAYERS = 16

SMOL_OK = 0
SMOL_ERR_INVALID = -1
SMOL_ERR_UNBOUND = -2
SMOL_ERR_CUDA = -3
SMOL_ERR_UNSUPPORTED = -4
SMOL_ERR_CAPACITY = -5


class SmolConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "dim", "n_layer", "n_head", "n_local_heads", "head_dim", "intermediate_size", "vocab_size",
        "fast_dim", "n_fast_layer", "fast_n_head", "fast_n_local_heads", "fast_head_dim", "fast_intermediate_size",
        "codebook_size", "num_codebooks",
        "duplicate_code_0", "depthwise_wte", "depthwise_output", "tie_word_embeddings",
        "max_seq_len", "max_batch", "page_size",
        "semantic_start_id", "semantic_end_id", "im_end_id", "mlx_embed_mask")] + [("norm_eps", C.c_float)]


class SmolLayerWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("wqkv", "wo", "w1", "w3", "w2", "attention_norm", "ffn_norm")]


class SmolWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "embeddings", "codebook_embeddings", "norm", "output", "fast_embeddings", "fast_norm", "fast_output",
        "rope", "fast_rope")] + [
        ("layers", SmolLayerWeights * SMOL_MAX_LAYERS),
        ("fast_layers", SmolLayerWeights * SMOL_MAX_FAST_LAYERS)]


class SmolRowSampling(C.Structure):
    _fields_ = [
        ("temp", C.c_float), ("fast_temp", C.c_float), ("top_k", C.c_int32), ("top_p", C.c_float), ("min_p", C.c_float),
        ("pad", C.c_uint32), ("seed", C.c_uint64)]


class SmolBatch(C.Structure):
    _fields_ = [
        ("tokens", C.c_void_p), ("seq_len", C.c_void_p), ("block_table", C.c_void_p), ("max_pages", C.c_int32),
        ("finished", C.c_void_p), ("seq_id", C.c_void_p), ("step", C.c_void_p), ("out_codes", C.c_void_p),
        ("max_frames", C.c_int32), ("row_sampling", C.c_void_p)]


class SmolSampling(C.Structure):
    _fields_ = [
        ("temp", C.c_float), ("fast_temp", C.c_float), ("top_k", C.c_int32), ("top_p", C.c_float),
        ("min_p", C.c_float), ("seed", C.c_uint64), ("audio_only", C.c_int32), ("ignore_stop", C.c_int32)]


# ---- include/smoltts_b200_mimi.h ----
SMOL_MIMI_MAX_LAYERS = 16
SMOL_MIMI_MAX_RATIOS = 8
SMOL_MIMI_MAX_Q = 32


class SmolMimiConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_q", "codebook_size", "codebook_dim", "dim", "n_layers", "n_heads", "head_dim", "ffn", "n_filters", "n_ratios")] + [
        ("ratios", C.c_int32 * SMOL_MIMI_MAX_RATIOS)] + [(n, C.c_int32) for n in (
            "kernel", "res_kernel", "last_kernel", "max_streams", "max_positions", "window", "upsample_carry", "use_graph")] + [
        ("norm_eps", C.c_float), ("codebook_eps", C.c_float)]


class SmolMimiLayerWeights(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("q_proj", "k_proj", "v_proj", "o_proj", "fc1", "fc2", "ln1_w", "ln1_b", "ln2_w", "ln2_b",
                                          "scale_attn", "scale_mlp")]


class SmolMimiConv(C.Structure):
    _fields_ = [("weight", C.c_void_p), ("bias", C.c_void_p)]


class SmolMimiWeights(C.Structure):
    _fields_ = [
        ("embed_sum", C.c_void_p * SMOL_MIMI_MAX_Q), ("cluster_usage", C.c_void_p * SMOL_MIMI_MAX_Q),
        ("semantic_output_proj", C.c_void_p), ("acoustic_output_proj", C.c_void_p), ("upsample", C.c_void_p),
        ("layers", SmolMimiLayerWeights * SMOL_MIMI_MAX_LAYERS),
        ("conv_in", SmolMimiConv), ("convtr", SmolMimiConv * SMOL_MIMI_MAX_RATIOS),
        ("res_conv1", SmolMimiConv * SMOL_MIMI_MAX_RATIOS), ("res_conv2", SmolMimiConv * SMOL_MIMI_MAX_RATIOS),
        ("conv_out", SmolMimiConv), ("rope", C.c_void_p)]


class SmolMimiEncoderConfig(C.Structure):
    _fields_ = [(n, C.c_int32) for n in (
        "n_q", "codebook_size", "codebook_dim", "dim", "n_layers", "n_heads", "head_dim", "ffn", "n_filters", "n_ratios")] + [
        ("ratios", C.c_int32 * SMOL_MIMI_MAX_RATIOS)] + [(n, C.c_int32) for n in (
            "kernel", "res_kernel", "last_kernel", "max_clips", "max_samples", "window")] + [
        ("norm_eps", C.c_float), ("codebook_eps", C.c_float)]


class SmolMimiEncoderWeights(C.Structure):
    _fields_ = [
        ("embed_sum", C.c_void_p * SMOL_MIMI_MAX_Q), ("cluster_usage", C.c_void_p * SMOL_MIMI_MAX_Q),
        ("semantic_input_proj", C.c_void_p), ("acoustic_input_proj", C.c_void_p), ("downsample", C.c_void_p),
        ("layers", SmolMimiLayerWeights * SMOL_MIMI_MAX_LAYERS),
        ("conv_in", SmolMimiConv), ("res_conv1", SmolMimiConv * SMOL_MIMI_MAX_RATIOS),
        ("res_conv2", SmolMimiConv * SMOL_MIMI_MAX_RATIOS), ("conv_down", SmolMimiConv * SMOL_MIMI_MAX_RATIOS),
        ("conv_out", SmolMimiConv), ("rope", C.c_void_p)]


# name -> (restype, argtypes); every symbol the headers declare
PROTOTYPES = {
    "smol_abi_version": (C.c_int, []),
    "smol_last_error": (C.c_char_p, []),
    "smol_create": (C.c_int, [C.POINTER(SmolConfig), C.POINTER(C.c_void_p)]),
    "smol_destroy": (None, [C.c_void_p]),
    "smol_bind_weights": (C.c_int, [C.c_void_p, C.POINTER(SmolWeights)]),
    "smol_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "smol_bind_workspace": (C.c_int, [C.c_void_p, C.c_void_p, C.c_size_t]),
    "smol_kv_page_bytes": (C.c_size_t, [C.c_void_p]),
    "smol_kv_bind": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "smol_prefill": (C.c_int, [C.c_void_p, C.POINTER(SmolBatch), C.c_int32, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "smol_slow_step": (C.c_int, [C.c_void_p, C.POINTER(SmolBatch), C.c_int32, C.c_int32, C.c_void_p]),
    "smol_fast_step": (C.c_int, [C.c_void_p, C.POINTER(SmolBatch), C.c_int32, C.c_int32, C.c_int32, C.c_void_p]),
    "smol_fast_embed": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "smol_sample": (C.c_int, [C.c_void_p, C.POINTER(SmolBatch), C.c_int32, C.c_void_p, C.c_int32,
                              C.POINTER(SmolSampling), C.c_int32, C.c_void_p, C.c_void_p]),
    "smol_decode_frame": (C.c_int, [C.c_void_p, C.POINTER(SmolBatch), C.c_int32, C.POINTER(SmolSampling), C.c_void_p]),
    "smol_decode_frames": (C.c_int, [C.c_void_p, C.POINTER(SmolBatch), C.c_int32, C.POINTER(SmolSampling), C.c_int32,
                                     C.c_void_p]),
    "smol_set_force": (C.c_int, [C.c_void_p, C.c_void_p]),
    "smol_set_profile": (C.c_int, [C.c_void_p, C.c_void_p]),
    "smol_set_frame_clock": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "smol_run_phases": (C.c_int, [C.c_void_p, C.POINTER(SmolBatch), C.c_int32, C.POINTER(SmolSampling), C.c_int32,
                                  C.c_int32, C.c_void_p]),
    "smol_phase_count": (C.c_int32, [C.c_void_p]),
    "smol_set_option": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int64]),
    "smol_get_option": (C.c_int64, [C.c_void_p, C.c_char_p]),
    "smol_debug_buffer": (C.c_void_p, [C.c_void_p, C.c_char_p]),
    "smol_launches_per_frame": (C.c_int32, [C.c_void_p]),
    "smol_launch_count": (C.c_int64, [C.c_void_p]),
    # include/smoltts_b200_mimi.h
    "smol_mimi_create": (C.c_int, [C.POINTER(SmolMimiConfig), C.POINTER(C.c_void_p)]),
    "smol_mimi_destroy": (None, [C.c_void_p]),
    "smol_mimi_samples_per_frame": (C.c_int32, [C.c_void_p]),
    "smol_mimi_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "smol_mimi_bind": (C.c_int, [C.c_void_p, C.POINTER(SmolMimiWeights), C.c_void_p, C.c_size_t, C.c_void_p]),
    "smol_mimi_reset": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p]),
    "smol_mimi_decode_step": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "smol_mimi_debug_buffer": (C.c_void_p, [C.c_void_p, C.c_char_p, C.POINTER(C.c_int64)]),
    "smol_mimi_launches_per_step": (C.c_int32, [C.c_void_p]),
    "smol_mimi_error_word": (C.c_void_p, [C.c_void_p]),
    "smol_mimi_encoder_create": (C.c_int, [C.POINTER(SmolMimiEncoderConfig), C.POINTER(C.c_void_p)]),
    "smol_mimi_encoder_destroy": (None, [C.c_void_p]),
    "smol_mimi_encoder_samples_per_frame": (C.c_int32, [C.c_void_p]),
    "smol_mimi_encoder_workspace_bytes": (C.c_size_t, [C.c_void_p]),
    "smol_mimi_encoder_bind": (C.c_int, [C.c_void_p, C.POINTER(SmolMimiEncoderWeights), C.c_void_p, C.c_size_t, C.c_void_p]),
    "smol_mimi_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.POINTER(C.c_int64), C.c_int32, C.c_void_p, C.c_void_p]),
    "smol_mimi_encoder_debug_buffer": (C.c_void_p, [C.c_void_p, C.c_char_p]),
    "smol_mimi_encoder_launches": (C.c_int32, [C.c_void_p]),
}

_lib = None


class SmolError(RuntimeError):
    def __init__(self, code: int, message: str):
        super().__init__(f"smoltts_b200 error {code}: {message}")
        self.code = code


def library_path() -> str:
    return _build.LIB_PATH


def load() -> C.CDLL:
    """Loads (building first if necessary) the C-ABI library.  Raises if it cannot."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("SMOLTTS_B200_LIB")  # override: A/B runs of two builds on one GPU box
    if not path:
        # no-op when the digest of sources + headers + flags matches the stamp next to the .so: an edited kernel can
        # never be tested against a stale binary
        path = _build.build()
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.smol_abi_version() != SMOL_ABI_VERSION:
        raise RuntimeError(f"{path}: ABI version {lib.smol_abi_version()} != {SMOL_ABI_VERSION}")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc != SMOL_OK:
        msg = load().smol_last_error()
        raise SmolError(rc, msg.decode() if msg else "")
