"""The op-level checks of tests/test_gpu_ll2_ops.py have teeth: on the CPU oracle's own outputs every check passes, and on the
output of a deliberately mutated op the check aimed at that op fails.  The mutations are computed here, as data; nothing
runs on a device."""
import pytest
import torch
import torch.nn.functional as F

import ll2_checks as lc
from oracle.dualar_oracle import DualAROracle, rmsnorm
from smoltts_b200.config import named_config
from smoltts_b200.synth import make_state_dict, teacher_grid

T = 35   # cached positions before the traced step: the step's own position


@pytest.fixture(scope="module")
def traced():
    """Tiny model: the oracle's trace of one cached slow step at position T and of depth steps 0 and 1 (all bf16)."""
    cfg = named_config("smoltts_byte_tiny")
    sd = make_state_dict(cfg, seed=0, norm_jitter=0.05)
    orc = DualAROracle(cfg, sd, max_seq_len=512)
    grid = teacher_grid(cfg, n_text=T - 5, n_audio=7, batch=1, seed=3)
    tr = {}
    with torch.no_grad():
        cache = orc.new_cache()
        orc.slow_forward(grid[:, :, :T], cache, all_positions=True)
        logits, hidden = orc.slow_forward(grid[:, :, T:T + 1], cache, trace=tr)
        fcache = orc.new_fast_cache()
        orc.fast_step(hidden, 0, fcache, trace=tr)
        x1 = orc.fast_embed(grid[:, 1, T + 1], 0)
        fl1 = orc.fast_step(x1, 1, fcache, trace=tr)
    tr = {k: v[0] for k, v in tr.items()}
    return dict(cfg=cfg, orc=orc, w=orc.w, tr=tr, cache=cache, fcache=fcache, logits=logits[0], hidden=hidden[0], x1=x1[0],
                fl1=fl1[0])


def _scores(q, K):
    """Exact q.k / 8 rounded once to fp32: what a correct score unit publishes up to its rounding."""
    H, n_kv = q.numel() // 64, K.shape[0]
    return ((q.double().view(H, 1, 64) * K.double().repeat_interleave(H // n_kv, 0)).sum(-1) / 8).float()


def _psums(w2, act, shift=0):
    """Exact partial sums of the 7 K-slices rounded to fp32; `shift` (0 or 32) moves every slice's range by that many
    elements (past the end of K: zeros)."""
    D, F_ = w2.shape
    w = torch.cat([w2.double(), torch.zeros(D, 32, dtype=torch.float64)], 1)
    a = torch.cat([act.double(), torch.zeros(32, dtype=torch.float64)])
    out = []
    for c in range(lc.PSUM_SLICES):
        lo, hi = lc.psum_range(F_, c)
        out.append((w[:, lo + shift:hi + shift] * a[lo + shift:hi + shift]).sum(1))
    return torch.stack(out).float()


def _slow(t, l):
    cfg, w, tr = t["cfg"], t["w"], t["tr"]
    p = f"layers.{l}."
    x_in = tr["embed"] if l == 0 else tr[f"l{l - 1}.out"]
    return cfg, w, tr, p, x_in


def test_checks_pass_on_the_oracles_outputs(traced):
    t = traced
    cfg, orc = t["cfg"], t["orc"]
    eps, H, Hkv = cfg.norm_eps, cfg.n_head, cfg.n_local_heads
    for l in range(cfg.n_layer):
        cfg, w, tr, p, x_in = _slow(t, l)
        g = f"l{l}."
        lc.check_qkv(g + "qkv", x_in, w[p + "attention_norm.weight"], w[p + "attention.wqkv.weight"], orc.freqs[T], H, Hkv, eps,
                     tr[g + "q"], tr[g + "k"], tr[g + "v"])
        K, V = t["cache"][l].k[0], t["cache"][l].v[0]
        assert K.shape[1] == T + 1
        lc.check_attn(g + "attn", tr[g + "q"], K, V, tr[g + "attn"])
        lc.check_scores(g + "scores", _scores(tr[g + "q"], K), tr[g + "q"], K)
        lc.check_wo(g + "wo", tr[g + "attn"], x_in, w[p + "attention.wo.weight"], tr[g + "h"])
        lc.check_w13(g + "w13", tr[g + "h"], w[p + "ffn_norm.weight"], w[p + "feed_forward.w1.weight"], w[p + "feed_forward.w3.weight"],
                     eps, tr[g + "act"])
        lc.check_psums(g + "psums", _psums(w[p + "feed_forward.w2.weight"], tr[g + "act"]), w[p + "feed_forward.w2.weight"], tr[g + "act"])
        lc.check_w2(g + "w2", tr[g + "act"], tr[g + "h"], w[p + "feed_forward.w2.weight"], tr[g + "out"])
        x = tr[g + "out"]
        fo = lc.fused_output(_psums(w[p + "feed_forward.w2.weight"], tr[g + "act"]), tr[g + "h"])
        lc.check_w2(g + "w2 (fused)", tr[g + "act"], tr[g + "h"], w[p + "feed_forward.w2.weight"], fo)
    assert torch.equal(x, t["hidden"])
    lc.check_head("head", x, w["norm.weight"], w["embeddings.weight"], eps, t["logits"])
    # depth step 1: attention over the two depth positions + wo, and the depthwise head of position 1
    fp, C = "fast_layers.0.", cfg.codebook_size
    lc.check_fast_wo("f1.wo", tr["f1.l0.q"], t["fcache"][0].k[0], t["fcache"][0].v[0], t["x1"], w[fp + "attention.wo.weight"], tr["f1.l0.h"])
    lc.check_head("f1.head", tr[f"f1.l{cfg.n_fast_layer - 1}.out"], w["fast_norm.weight"], w["fast_output.weight"][C:2 * C], eps, t["fl1"])


MUTATIONS = ["rope_row_off_by_one", "newest_position_left_out", "k_from_neighbouring_slot", "silu_of_unrounded_operand",
             "psum_range_shifted_one_k_block", "wrong_depthwise_head"]


@pytest.mark.parametrize("mutation", MUTATIONS)
def test_each_mutated_op_is_rejected(traced, mutation):
    t = traced
    cfg, orc = t["cfg"], t["orc"]
    eps, H, Hkv = cfg.norm_eps, cfg.n_head, cfg.n_local_heads
    l = 1
    cfg, w, tr, p, x_in = _slow(t, l)
    g = f"l{l}."
    q, K, V = tr[g + "q"], t["cache"][l].k[0], t["cache"][l].v[0]
    with pytest.raises(AssertionError) as e:
        if mutation == "rope_row_off_by_one":
            mq, mk, mv = lc.ref_qkv(x_in, w[p + "attention_norm.weight"], w[p + "attention.wqkv.weight"], orc.freqs[T + 1], H, Hkv, eps)
            lc.check_qkv("qkv", x_in, w[p + "attention_norm.weight"], w[p + "attention.wqkv.weight"], orc.freqs[T], H, Hkv, eps, mq, mk, mv)
        elif mutation == "newest_position_left_out":
            lc.check_attn("attn", q, K, V, lc.ref_attention(q, K[:, :-1], V[:, :-1]))
        elif mutation == "k_from_neighbouring_slot":
            Km = K.clone()
            Km[:, T - 3] = K[:, T - 2]
            lc.check_scores("scores", _scores(q, Km), q, K)
        elif mutation == "silu_of_unrounded_operand":
            hn = rmsnorm(tr[g + "h"][None, None], w[p + "ffn_norm.weight"], eps)
            a32 = F.linear(hn.float(), w[p + "feed_forward.w1.weight"].float())
            act = F.silu(a32).to(torch.bfloat16) * F.linear(hn, w[p + "feed_forward.w3.weight"])
            lc.check_w13("w13", tr[g + "h"], w[p + "ffn_norm.weight"], w[p + "feed_forward.w1.weight"], w[p + "feed_forward.w3.weight"],
                         eps, act.reshape(-1))
        elif mutation == "psum_range_shifted_one_k_block":
            w2 = w[p + "feed_forward.w2.weight"]
            lc.check_psums("psums", _psums(w2, tr[g + "act"], shift=32), w2, tr[g + "act"])
        elif mutation == "wrong_depthwise_head":
            C = cfg.codebook_size
            x = tr[f"f1.l{cfg.n_fast_layer - 1}.out"]
            wrong = lc.ref_head(x, w["fast_norm.weight"], w["fast_output.weight"][2 * C:3 * C], eps)
            lc.check_head("f1.head", x, w["fast_norm.weight"], w["fast_output.weight"][C:2 * C], eps, wrong)
    aimed = {"rope_row_off_by_one": "qkv.q", "newest_position_left_out": "attn", "k_from_neighbouring_slot": "scores",
             "silu_of_unrounded_operand": "w13", "psum_range_shifted_one_k_block": "psums", "wrong_depthwise_head": "f1.head"}
    assert str(e.value).startswith(aimed[mutation] + ":"), f"{mutation}: rejected for another reason: {e.value}"
