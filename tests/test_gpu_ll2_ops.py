"""Op-level parity of the data-flow kernel (ll2_kernel.cu, batches 1..8): every phase of one frame against the reference op.

After a one-frame launch the kernel's word regions still hold what every phase of that frame published (q | k | v, the
attention output, h, act, the layer output, the logits; the fp32 attention scores of the last two slow layers; the fused
MLP's fp32 partial sums).  Each phase is checked against the reference's op applied to the inputs the kernel itself
consumed (tests/ll2_checks.py), at the bars tests/test_gpu_ops.py holds the other kernels to -- no chained drift, so a
one-ulp bias, a dropped attention position, a wrong RoPE row or a mis-bounded K range cannot hide in an end-to-end bar.
On top: the hand-off protocol (every word of a phase carries that phase's epoch, every replica equals replica 0), the K/V
appended to the paged pool, the logits dumps and the ids the frame chose (forced, greedy, sampled).
"""
import numpy as np
import pytest
import torch

import ll2_checks as lc
from gpu_util import model_and_oracle
from oracle.sampler_oracle import sample_row
from smoltts_b200.generate import GenerationSettings
from smoltts_b200.model import LL_REPLICAS, ll_bf16
from smoltts_b200.synth import teacher_grid

pytestmark = pytest.mark.gpu


# ---- one frame, everything it published copied to the host ---------------------------------------------------------
def _grid(cfg, lens, seed):
    """Teacher grid with column lens[b] (the forced ids) after each sequence's prompt; the pending column is an audio one."""
    S = max(lens) + 1
    return teacher_grid(cfg, n_text=S - 6, n_audio=6, batch=len(lens), seed=seed)


def _run_frame(model, cfg, grid, lens, fused=False, force=True, sampling=None, table=None, seq_ids=None):
    B = grid.shape[0]
    dev = model.device
    model.set_option("ll_fused_mlp", 1 if fused else 0)
    batch = model.new_batch(B, max_positions=max(lens) + 8, max_frames=2, seq_ids=seq_ids)
    try:
        model.kv_view()[torch.tensor(batch.pages, device=dev)] = 0
        g32 = grid[:, :, :max(lens)].to(device=dev, dtype=torch.int32).contiguous()
        model.prefill(batch, g32, torch.tensor(lens, dtype=torch.int32, device=dev))
        if table is not None:
            batch.set_row_sampling(table)
        torch.cuda.synchronize()
        pos = batch.seq_len.tolist()
        assert pos == [n - 1 for n in lens], f"prefill left seq_len {pos}"
        rec = dict(pos=pos, pending=batch.tokens.cpu().clone(), step=batch.step.cpu().clone(), seq_id=batch.seq_id.cpu().clone(),
                   table=batch.block_table.cpu().clone())
        if force:
            rec["force"] = torch.stack([grid[b, :, lens[b]] for b in range(B)]).to(torch.int32)
            model.set_force(rec["force"].to(dev).contiguous())
        e0 = model.ll_epoch()
        model.decode_frames(batch, sampling or model.sampling(ignore_stop=True), 1)
        torch.cuda.synchronize()
        assert model.get_option("ll_ready") == 1, "the data-flow kernel did not run"
        rec["fused"] = model.get_option("ll_last_fused") == 1
        pc = model.phase_count
        rec["e_end"], rec["pc"] = model.ll_epoch(), pc
        assert rec["e_end"] - e0 == pc, "one frame must run every phase of the program once"
        rec["words"] = {}
        for p in range(pc):
            kind, fast, _, _ = lc.decode_phase(p, cfg.n_layer, cfg.n_fast_layer)
            if lc.phase_elems(cfg, kind, fast):
                rec["words"][p] = [torch.stack([torch.stack(model.ll_words(p, b, r)) for r in range(LL_REPLICAS)]).cpu()
                                   for b in range(B)]   # [replica, (payload, epoch), words]
        rec["scores"] = {(b, l): tuple(t.cpu().clone() for t in model.ll_scores(b, l))
                         for b in range(B) for l in range(max(0, cfg.n_layer - 2), cfg.n_layer)}
        if rec["fused"]:
            rec["psums"] = {p: tuple(torch.stack(t).cpu() for t in zip(*(model.ll_psums(p, r) for r in range(LL_REPLICAS))))
                            for p in rec["words"] if lc.decode_phase(p, cfg.n_layer, cfg.n_fast_layer)[0] == lc.W2}
        rec["kv"] = model.kv_view().cpu().clone()
        rec["chosen"] = batch.tokens.cpu().clone()
        rec["frame_tokens"] = model.debug_buffer("frame_tokens", B).cpu().clone()
        rec["token_logits"] = model.debug_buffer("token_logits", B).cpu().clone()
        rec["depth_logits"] = model.debug_buffer("depth_logits", B).cpu().clone()
        return rec
    finally:
        model.set_force(None)
        model.set_option("ll_fused_mlp", 1)
        batch.release()


# ---- the checks of one frame ----------------------------------------------------------------------------------------
def _epoch(rec, p):
    """Phase p of the frame carried epoch e_end - phase_count + p + 1 (ll2_kernel.cu: epoch of a phase; ll_epoch at exit)."""
    return rec["e_end"] - rec["pc"] + p + 1


def _check_protocol(cfg, rec, b, tag):
    for p, w in rec["words"].items():
        kind, fast, layer, dp = lc.decode_phase(p, cfg.n_layer, cfg.n_fast_layer)
        n = lc.phase_elems(cfg, kind, fast) // 2
        e = _epoch(rec, p)
        pay, ep = w[b][:, 0, :n], w[b][:, 1, :n]
        where = f"{tag}: phase {p} ({lc.KIND_NAMES[kind]}, {'fast' if fast else 'slow'} layer {layer}, depth {dp})"
        if rec["fused"] and kind in (lc.W13, lc.W2):
            assert (ep[0] != e).all(), f"{where}: the fused program must not publish this region"
            continue
        bad = (ep[0] != e).nonzero()
        assert bad.numel() == 0, f"{where}: word {int(bad[0])} has epoch {int(ep[0, bad[0]])}, not {e}"
        for r in range(1, 1 if kind == lc.HEAD else LL_REPLICAS):
            assert torch.equal(pay[r], pay[0]) and torch.equal(ep[r], ep[0]), f"{where}: replica {r} differs from replica 0"
    if rec["fused"]:
        for p, (ps, pe) in rec["psums"].items():
            e = _epoch(rec, p)
            assert (pe == e).all(), f"{tag}: partial sums of phase {p}: {int((pe != e).sum())} words without the W2 epoch {e}"
            for r in range(1, LL_REPLICAS):
                assert torch.equal(ps[r].view(torch.int32), ps[0].view(torch.int32)), f"{tag}: partial sums of phase {p}: replica {r}"


def _check_ops(cfg, orc, rec, b, tag, stats, unfused=None):
    """Every phase of team b against the reference op on the kernel's own inputs.  A fused frame's W13 / W2 are checked
    through its partial sums, against the act of `unfused` (the same frame run unfused from identical state)."""
    w, eps, fused = orc.w, cfg.norm_eps, rec["fused"]
    pos = rec["pos"][b]
    ps = rec["kv"].shape[4]
    assert not fused or unfused is not None

    def vec(p, r=rec):
        kind, fast, _, _ = lc.decode_phase(p, cfg.n_layer, cfg.n_fast_layer)
        return ll_bf16(r["words"][p][b][0, 0])[: lc.phase_elems(cfg, kind, fast)]

    def note(kind, res):
        for ex, mu in (res if isinstance(res, list) else [res]):
            s = stats.setdefault((tag, kind), [1.0, 0.0])
            s[0], s[1] = min(s[0], ex), max(s[1], mu)

    def pool(l, which):   # [n_kv, pos + 1, 64] of slow layer l through the block table
        pages = [int(rec["table"][b, i]) for i in range(pos // ps + 1)]
        return torch.cat([rec["kv"][pg, l, which] for pg in pages], dim=1)[:, :pos + 1]

    def mlp(p_w13, pre, h, name):   # W13 + W2 of the layer whose W13 phase is p_w13 -> the layer output
        w1, w3, w2 = (w[pre + f"feed_forward.{m}.weight"] for m in ("w1", "w3", "w2"))
        if fused:
            act = vec(p_w13, unfused)
            psum = rec["psums"][p_w13 + 1][0][0]
            lc.check_psums(name + ".psums", psum, w2, act)
            out = lc.fused_output(psum, h)
        else:
            act = vec(p_w13)
            note("w13", lc.check_w13(name + ".w13", h, w[pre + "ffn_norm.weight"], w1, w3, eps, act))
            out = vec(p_w13 + 1)
        note("w2", lc.check_w2(name + ".w2", act, h, w2, out))
        return out

    H, Hkv = cfg.n_head, cfg.n_local_heads
    x = orc.embed(rec["pending"][b].long().view(1, -1, 1))[0, 0]
    for l in range(cfg.n_layer):
        p, pre, name = 5 * l, f"layers.{l}.", f"{tag} team {b} l{l}"
        q, k, v = vec(p).split([H * 64, Hkv * 64, Hkv * 64])
        note("qkv", lc.check_qkv(name + ".qkv", x, w[pre + "attention_norm.weight"], w[pre + "attention.wqkv.weight"], orc.freqs[pos],
                                 H, Hkv, eps, q, k, v))
        K, V = pool(l, 0), pool(l, 1)
        assert torch.equal(K[:, pos].reshape(-1).view(torch.int16), k.view(torch.int16)), f"{name}: K appended at {pos} != k words"
        assert torch.equal(V[:, pos].reshape(-1).view(torch.int16), v.view(torch.int16)), f"{name}: V appended at {pos} != v words"
        attn = vec(p + 1)
        note("attn", lc.check_attn(name + ".attn", q, K, V, attn))
        if (b, l) in rec["scores"]:
            sc, se = rec["scores"][(b, l)]
            assert (se[:, :pos + 1] == _epoch(rec, p + 1)).all(), f"{name}: score words without the ATTN epoch"
            lc.check_scores(name + ".scores", sc[:, :pos + 1], q, K)
        h = vec(p + 2)
        note("wo", lc.check_wo(name + ".wo", attn, x, w[pre + "attention.wo.weight"], h))
        x = mlp(p + 3, pre, h, name)
    n_slow = 5 * cfg.n_layer
    logits = vec(n_slow)
    head = w["embeddings.weight"] if cfg.tie_word_embeddings else w["output.weight"]
    note("head", lc.check_head(f"{tag} team {b} head", x, w["norm.weight"], head, eps, logits))
    assert torch.equal(logits.float(), rec["token_logits"][b]), f"{tag}: logits words != token_logits"

    Hf, Hkvf, nf, C = cfg.fast_n_head, cfg.fast_n_local_heads, cfg.n_fast_layer, cfg.codebook_size
    per, hidden = 4 * nf + 2, x
    fk, fv = [[] for _ in range(nf)], [[] for _ in range(nf)]
    for i in range(lc.depth_of(cfg)):
        x = hidden if i == 0 else orc.fast_embed(rec["chosen"][b, i].long().view(1), i - 1)[0]
        for l in range(nf):
            p, pre, name = n_slow + 2 + i * per + 4 * l, f"fast_layers.{l}.", f"{tag} team {b} f{i}.l{l}"
            q, k, v = vec(p).split([Hf * 64, Hkvf * 64, Hkvf * 64])
            note("qkv", lc.check_qkv(name + ".qkv", x, w[pre + "attention_norm.weight"], w[pre + "attention.wqkv.weight"],
                                     orc.fast_freqs[i], Hf, Hkvf, eps, q, k, v))
            fk[l].append(k.view(Hkvf, 64))
            fv[l].append(v.view(Hkvf, 64))
            h = vec(p + 1)
            note("fast_wo", lc.check_fast_wo(name + ".wo", q, torch.stack(fk[l], 1), torch.stack(fv[l], 1), x,
                                             w[pre + "attention.wo.weight"], h))
            x = mlp(p + 2, pre, h, name)
        p = n_slow + 2 + i * per + 4 * nf
        fo = w["fast_output.weight"][i * C:(i + 1) * C] if cfg.depthwise_output else w["fast_output.weight"]
        logits = vec(p)
        note("head", lc.check_head(f"{tag} team {b} f{i}.head", x, w["fast_norm.weight"], fo, eps, logits))
        assert torch.equal(logits.float(), rec["depth_logits"][b, i]), f"{tag}: depth {i} logits words != depth_logits"


def _check_frame(cfg, orc, rec, tag, stats, unfused=None):
    for b in range(len(rec["pos"])):
        _check_protocol(cfg, rec, b, tag)
        _check_ops(cfg, orc, rec, b, tag, stats, unfused)
    assert torch.equal(rec["frame_tokens"], rec["chosen"]), f"{tag}: frame_tokens != the assembled column"
    if "force" in rec:
        assert torch.equal(rec["chosen"], rec["force"]), f"{tag}: the frame did not adopt the forced ids"


def _report(stats):
    for (tag, kind), (ex, mu) in sorted(stats.items()):
        print(f"{tag:42s} {kind:8s} bit-exact >= {ex:.3f}  max {mu:.1f} ulps")


def _both_programs(model, cfg, orc, grid, lens, tag, **kw):
    """The frame unfused, then fused from identical state (batch 1: the default program), both checked phase by phase."""
    stats = {}
    unf = _run_frame(model, cfg, grid, lens, fused=False, **kw)
    assert not unf["fused"]
    _check_frame(cfg, orc, unf, tag + " unfused", stats)
    fus = _run_frame(model, cfg, grid, lens, fused=True, **kw)
    fits = model.get_option("ll_mlp_cluster") > 0 and (model.get_option("n_ctas_override") <= 0)
    if fits:
        assert fus["fused"], f"{tag}: the fused program did not run"
    _check_frame(cfg, orc, fus, tag + (" fused" if fus["fused"] else " unfused (no cluster)"), stats, unfused=unf)
    assert torch.equal(fus["token_logits"], unf["token_logits"]) and torch.equal(fus["depth_logits"], unf["depth_logits"])
    _report(stats)


# ---- cases ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("size,pos", [("smoltts_byte_tiny", 40), ("smoltts_byte_70m", 90), ("smoltts_byte_150m", 130)])
def test_ll2_solo_frame_every_phase(size, pos):
    cfg, sd, model, orc = model_and_oracle(size, max_batch=1)
    lib, h = model.lib, model._h
    total = sum(lc.phase_words(cfg, p) for p in range(model.phase_count)) * LL_REPLICAS * 8
    assert lib.smol_debug_buffer(h, b"ll_epoch") - lib.smol_debug_buffer(h, b"ll") >= total * 8, "word regions overflow the buffer"
    _both_programs(model, cfg, orc, _grid(cfg, [pos + 1], seed=pos), [pos + 1], f"{size} bs=1 pos={pos}")


@pytest.mark.parametrize("size,B", [("smoltts_byte_70m", 3), ("smoltts_byte_tiny", 8)])
def test_ll2_team_frames_every_phase(size, B):
    """One team of CTAs per sequence, each with its own regions and score words (and its own position)."""
    cfg, sd, model, orc = model_and_oracle(size, max_batch=8)
    lens = [31 + 7 * b for b in range(B)]
    stats = {}
    rec = _run_frame(model, cfg, _grid(cfg, lens, seed=B), lens)
    assert not rec["fused"], "teams run the unfused program"
    _check_frame(cfg, orc, rec, f"{size} bs={B}", stats)
    _report(stats)


@pytest.mark.parametrize("pos,n_ctas", [(511, 0), (512, 0), (513, 0), (2100, 0), (2100, 40)])
def test_ll2_attention_block_edges(pos, n_ctas):
    """The new position at the last / first / second position of a 512-position softmax block, and deep into the fifth;
    n_ctas = 40 gives a CTA several attention units."""
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=1, max_seq_len=2304)
    if n_ctas:
        model.set_option("n_ctas", n_ctas)
    try:
        _both_programs(model, cfg, orc, _grid(cfg, [pos + 1], seed=pos), [pos + 1], f"tiny pos={pos} n_ctas={n_ctas or 'solo'}")
        if n_ctas:
            assert model.get_option("n_ctas") == n_ctas
    finally:
        model.set_option("n_ctas", 0)


def test_ll2_depth7_every_phase():
    """duplicate_code_0 = False: 7 depth positions, embeddings and heads shifted by one codebook."""
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=1, duplicate_code_0=False)
    assert lc.depth_of(cfg) == 7
    _both_programs(model, cfg, orc, _grid(cfg, [48], seed=7), [48], "tiny depth 7")


def test_ll2_greedy_and_sampled_ids():
    """An unforced greedy frame: every id is the first arg-max of its logits words.  A sampled frame with a per-row table
    (temperature, top-k / top-p, greedy and sampled depth codes): every id is the sampler specification's pick from the HEAD
    words with the row's own counters."""
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=8)
    lens, ids = [37, 45], [11, 12]
    grid = _grid(cfg, lens, seed=5)
    stats = {}
    n_slow, per = 5 * cfg.n_layer, 4 * cfg.n_fast_layer + 2
    heads = [n_slow] + [n_slow + 2 + i * per + 4 * cfg.n_fast_layer for i in range(lc.depth_of(cfg))]

    def head_logits(rec, b, r):
        return ll_bf16(rec["words"][heads[r]][b][0, 0]).float().numpy()

    rec = _run_frame(model, cfg, grid, lens, force=False, seq_ids=ids)
    _check_frame(cfg, orc, rec, "tiny bs=2 greedy", stats)
    for b in range(2):
        want = [int(np.argmax(head_logits(rec, b, r))) for r in range(cfg.n_rows)]
        assert rec["chosen"][b].tolist() == want, f"greedy team {b}: {rec['chosen'][b].tolist()} != {want}"

    gs = [GenerationSettings(default_temp=0.8, default_fast_temp=0.6, top_k=40, top_p=0.9, seed=77),
          GenerationSettings(default_temp=1.1, default_fast_temp=0.0, top_p=0.8, seed=5)]
    table = model.row_sampling(gs)
    rec = _run_frame(model, cfg, grid, lens, force=False, table=table, seq_ids=ids)
    _check_frame(cfg, orc, rec, "tiny bs=2 sampled", stats)
    for b, s in enumerate(gs):
        step, sid = int(rec["step"][b]), int(rec["seq_id"][b])
        want = [sample_row(head_logits(rec, b, 0), s.default_temp, s.top_k, s.top_p, 0.0, s.seed, step, sid, 0)]
        want += [sample_row(head_logits(rec, b, r), s.default_fast_temp, 0, 1.0, 0.0, s.seed, step, sid, r) for r in range(1, cfg.n_rows)]
        assert rec["chosen"][b].tolist() == want, f"sampled team {b}: {rec['chosen'][b].tolist()} != {want}"
    _report(stats)
