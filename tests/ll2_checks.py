"""Op-level checks of the data-flow kernel (ll2_kernel.cu) on plain tensors.

Every phase of a frame publishes its output as words (include/smoltts_b200.h: smol_debug_buffer "ll").  Each check here
applies the reference's own op, in bf16 at the reference's rounding points (oracle/dualar_oracle.py: rmsnorm, F.linear,
apply_rope, SDPA, silu * up), to the inputs the kernel itself consumed, and compares with what the kernel published: no
chained drift, so the bars are those of tests/test_gpu_ops.py (gpu_util.close_report).  The fp32 side buffers (attention
scores, fused-MLP partial sums) are held to rigorous float64 error bounds instead.

Inputs are CPU tensors: bf16 vectors / matrices, fp32 scores and partial sums.  Each check raises AssertionError naming the
element that misses its bar, and returns (bit-exact share, max ulps) where that applies.
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.nn.functional as F

from gpu_util import close_report
from oracle.dualar_oracle import apply_rope, rmsnorm

# phase kinds in program order (dev_model.h: PhaseKind)
QKV, ATTN, WO, W13, W2, HEAD, SAMPLE = range(7)
KIND_NAMES = ("qkv", "attn", "wo", "w13", "w2", "head", "sample")
PSUM_SLICES = 7   # K-slices of the fused MLP (dev_model.h: kLL2Warps)

# (max ulps, min bit-exact share) per published tensor: tests/test_gpu_ops.py's bars for the same ops
BARS = {"qkv": (2.0, 0.98), "attn": (3.0, 0.65), "wo": (2.0, 0.98), "w13": (4.0, 0.98), "w2": (2.0, 0.98),
        "fast_wo": (3.0, 0.90), "head": (2.0, 0.98)}


# ---- the frame program, restated from dev_model.h (decode_phase, ll_phase_words) ------------------------------------
def depth_of(cfg) -> int:
    return cfg.num_codebooks - (0 if cfg.duplicate_code_0 else 1)


def phase_count(cfg) -> int:
    return 5 * cfg.n_layer + 2 + depth_of(cfg) * (4 * cfg.n_fast_layer + 2)


def decode_phase(p: int, n_layer: int, n_flayer: int) -> Tuple[int, int, int, int]:
    """Program index -> (kind, fast, layer, depth position)."""
    n_slow = 5 * n_layer
    if p < n_slow:
        return p % 5, 0, p // 5, 0
    if p == n_slow:
        return HEAD, 0, 0, 0
    if p == n_slow + 1:
        return SAMPLE, 0, 0, 0
    q = p - n_slow - 2
    per = 4 * n_flayer + 2
    i, r = divmod(q, per)
    if r < 4 * n_flayer:
        return (QKV, WO, W13, W2)[r % 4], 1, r // 4, i
    return (HEAD if r == 4 * n_flayer else SAMPLE), 1, 0, i


def phase_elems(cfg, kind: int, fast: int) -> int:
    """bf16 values a sequence publishes in a phase (SAMPLE: none)."""
    D = cfg.fast_dim if fast else cfg.dim
    if kind == QKV:
        H, Hkv = (cfg.fast_n_head, cfg.fast_n_local_heads) if fast else (cfg.n_head, cfg.n_local_heads)
        return (H + 2 * Hkv) * 64
    if kind in (ATTN, WO, W2):
        return D
    if kind == W13:
        return cfg.fast_intermediate_size if fast else cfg.intermediate_size
    if kind == HEAD:
        return cfg.codebook_size if fast else cfg.vocab_size
    return 0


def phase_words(cfg, p: int) -> int:
    """Words per sequence and replica of phase p's region: two values a word, rounded up to 16 words (128 bytes)."""
    kind, fast, _, _ = decode_phase(p, cfg.n_layer, cfg.n_fast_layer)
    n = phase_elems(cfg, kind, fast) // 2
    return (n + 15) // 16 * 16


# ---- reference ops: bf16 at the reference's rounding points (oracle/dualar_oracle.py) ----------------------------------
def _row(v: torch.Tensor) -> torch.Tensor:
    return v.reshape(1, 1, -1)


def ref_qkv(x, norm_w, wqkv, freqs_row, n_head, n_kv, eps):
    """RMSNorm + wqkv + interleaved-pair RoPE with the bf16 table row of the position -> flat q, k, v."""
    qkv = F.linear(rmsnorm(_row(x), norm_w, eps), wqkv)
    q, k, v = qkv.split([n_head * 64, n_kv * 64, n_kv * 64], dim=-1)
    fr = freqs_row.reshape(1, 32, 2)
    q = apply_rope(q.view(1, 1, n_head, 64), fr)
    k = apply_rope(k.view(1, 1, n_kv, 64), fr)
    return q.reshape(-1), k.reshape(-1), v.reshape(-1)


def ref_attention(q, K, V):
    """q [H * 64], K / V [n_kv, L, 64] -> [H * 64]: the reference's SDPA over positions 0 .. L - 1."""
    n_kv, L, _ = K.shape
    H = q.numel() // 64
    G = H // n_kv
    y = F.scaled_dot_product_attention(q.view(1, H, 1, 64), K.repeat_interleave(G, 0)[None], V.repeat_interleave(G, 0)[None],
                                       dropout_p=0.0)
    return y.reshape(-1)


def ref_linear_residual(inp, w, res):
    """res + w inp (wo and w2 with their residual)."""
    return (_row(res) + F.linear(_row(inp), w)).reshape(-1)


def ref_w13(h, norm_w, w1, w3, eps):
    hn = rmsnorm(_row(h), norm_w, eps)
    return (F.silu(F.linear(hn, w1)) * F.linear(hn, w3)).reshape(-1)


def ref_head(x, norm_w, head_w, eps):
    return F.linear(rmsnorm(_row(x), norm_w, eps), head_w).reshape(-1)


# ---- checks ---------------------------------------------------------------------------------------------------------
def _bar(name, got, want, bar):
    max_ulp, min_exact = BARS[bar]
    return close_report(name, got, want, max_ulp=max_ulp, min_exact=min_exact)


def check_qkv(name, x, norm_w, wqkv, freqs_row, n_head, n_kv, eps, q, k, v):
    """Returns the (bit-exact share, max ulps) of q, k and v."""
    rq, rk, rv = ref_qkv(x, norm_w, wqkv, freqs_row, n_head, n_kv, eps)
    return [_bar(f"{name}.{t}", got, want, "qkv") for t, got, want in (("q", q, rq), ("k", k, rk), ("v", v, rv))]


def check_attn(name, q, K, V, got):
    return _bar(name, got, ref_attention(q, K, V), "attn")


def check_wo(name, attn, res, wo, got):
    return _bar(name, got, ref_linear_residual(attn, wo, res), "wo")


def check_fast_wo(name, q, K, V, res, wo, got):
    """Depth attention over the frame's positions 0 .. i followed by wo + residual."""
    return _bar(name, got, ref_linear_residual(ref_attention(q, K, V), wo, res), "fast_wo")


def check_w13(name, h, norm_w, w1, w3, eps, got):
    return _bar(name, got, ref_w13(h, norm_w, w1, w3, eps), "w13")


def check_w2(name, act, res, w2, got):
    return _bar(name, got, ref_linear_residual(act, w2, res), "w2")


def check_head(name, x, norm_w, head_w, eps, got):
    return _bar(name, got, ref_head(x, norm_w, head_w, eps), "head")


def check_scores(name, scores, q, K):
    """scores fp32 [H, L] against (q . k) / 8 in float64, q [H * 64] bf16, K [n_kv, L, 64] bf16:
    |s - q.k / 8| <= 64 * 2^-24 * sum |q_i k_i| / 8 + 2^-126 at every position (a rounding-error bound, not a calibration)."""
    n_kv, L, _ = K.shape
    H = q.numel() // 64
    assert scores.shape == (H, L), f"{name}: shape {tuple(scores.shape)} vs {(H, L)}"
    t = q.double().view(H, 1, 64) * K.double().repeat_interleave(H // n_kv, 0)   # [H, L, 64]
    want = t.sum(-1) / 8
    bound = 64 * 2.0 ** -24 * t.abs().sum(-1) / 8 + 2.0 ** -126
    err = (scores.double() - want).abs()
    bad = ~(err <= bound)
    if bad.any():
        h, j = bad.nonzero()[0].tolist()
        raise AssertionError(f"{name}: {int(bad.sum())} scores outside the rounding bound; head {h} position {j}: "
                             f"got {scores[h, j].item():.8g} want {want[h, j].item():.8g} (bound {bound[h, j].item():.3g})")


def psum_range(F_: int, c: int) -> Tuple[int, int]:
    """Elements [lo, hi) of K-slice c of a w2 row: k-blocks [kb c / 7, kb (c + 1) / 7) of kb = K / 32."""
    kb = F_ // 32
    return 32 * (kb * c // PSUM_SLICES), 32 * (kb * (c + 1) // PSUM_SLICES)


def check_psums(name, psums, w2, act):
    """psums fp32 [7, D]: partial c within gamma_K * sum |w2 act| of the float64 dot product of w2 and act over K-slice c
    (gamma_K = K * 2^-24, K = the slice's length)."""
    D, F_ = w2.shape
    assert psums.shape == (PSUM_SLICES, D), f"{name}: shape {tuple(psums.shape)}"
    for c in range(PSUM_SLICES):
        lo, hi = psum_range(F_, c)
        t = w2[:, lo:hi].double() * act[lo:hi].double()
        want = t.sum(1)
        bound = (hi - lo) * 2.0 ** -24 * t.abs().sum(1)
        err = (psums[c].double() - want).abs()
        bad = ~(err <= bound)
        if bad.any():
            r = int(bad.nonzero()[0])
            raise AssertionError(f"{name}: slice {c} (elements {lo}..{hi}): {int(bad.sum())} rows outside the bound; row {r}: "
                                 f"got {psums[c, r].item():.8g} want {want[r].item():.8g} (bound {bound[r].item():.3g})")


def fused_output(psums, res):
    """What the fused MLP's consumers stage: bf16(res + bf16(sum of the 7 fp32 partials, in slice order))."""
    a = torch.zeros_like(psums[0])
    for c in range(PSUM_SLICES):
        a = a + psums[c]
    return (res.float() + a.to(torch.bfloat16).float()).to(torch.bfloat16)
