"""The tcgen05 variant of the decode kernel (batches / prefill tiles of 9+ rows, csrc/tc_phases.cuh + umma.cuh).

Its dot products are summed by the tensor core, so it is not bit-identical to the CUDA-core variants; it is held to
  * the oracle's greedy ids up to near-tie decisions (greedy-with-resync, same rule and TAU as tests/test_gpu_decode.py);
  * the CUDA-core variant's logits and cached K/V on the same inputs, within the spread the reference's own bf16
    executions show (rms 0.035 / 0.056 on token / codebook logits, DESIGN.md section 6);
  * bit-identity with itself across batch compositions and prefill tile sizes.
"""
import numpy as np
import pytest
import torch

from gpu_util import model_and_oracle
from oracle.dualar_oracle import OracleSettings
from smoltts_b200 import GenerationSettings, generate_batch
from smoltts_b200.generate import pack_prompts
from smoltts_b200.synth import byte_prompt, prompt_grid

pytestmark = pytest.mark.gpu

TAU = 0.15


@pytest.mark.parametrize("size", ["smoltts_byte_tiny", "smoltts_byte_70m", "smoltts_byte_150m"])
def test_tc_greedy_with_resync_vs_oracle(size):
    """16 utterances decoded together on the tensor-core variant, each checked against its own CPU-oracle decode."""
    cfg, sd, model, orc = model_and_oracle(size, max_batch=32)
    B = 16
    n_frames = 6 if size == "smoltts_byte_150m" else 10
    prompts = [prompt_grid(byte_prompt(24 + 2 * b, seed=40 + b), cfg) for b in range(B)]
    want, margins = [], []
    with torch.no_grad():
        for p in prompts:
            frames = orc.generate(p, OracleSettings(default_temp=0.0, default_fast_temp=0.0), fixed_frames=n_frames)
            want.append([f.vq for f in frames])
            margins.append([f.margins for f in frames])
    want = torch.tensor(want, dtype=torch.int32)          # [B, n, R]
    margins = np.array(margins)
    dev = model.device
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(B, max_positions=128, max_frames=n_frames)
    flips, exact = [], 0
    try:
        model.prefill(batch, padded, lens)
        s = model.sampling(ignore_stop=True)
        for f in range(n_frames):
            model.set_force(want[:, f].to(dev).contiguous())
            model.decode_frames(batch, s, 1)
            torch.cuda.synchronize()
            tl = model.debug_buffer("token_logits", B).cpu()
            dl = model.debug_buffer("depth_logits", B).cpu()
            assert torch.isfinite(tl).all() and torch.isfinite(dl).all()
            for b in range(B):
                mine = [int(tl[b].argmax())] + [int(dl[b, i].argmax()) for i in range(cfg.max_fast_seqlen)]
                for r, (a, w) in enumerate(zip(mine, want[b, f].tolist())):
                    if a == w:
                        exact += 1
                    else:
                        flips.append((b, f, r, float(margins[b, f, r])))
        assert model.get_option("tc_ready") == 1, "the tensor-core variant did not run"
    finally:
        model.set_force(None)
        batch.release()
    total = B * n_frames * cfg.n_rows
    print(f"{size}: {exact}/{total} greedy decisions identical; flips (seq,frame,row,oracle margin): {flips}")
    assert all(m <= TAU for *_, m in flips), f"argmax flipped at a confident decision: {flips}"
    assert exact >= 0.915 * total, f"{exact}/{total} identical decisions: below the measured rate (150m: 804/864 = 0.93)"


def _prefill_and_frames(model, prompts, n_frames, tc_min_batch, prefill_tile=0):
    model.set_option("tc_min_batch", tc_min_batch)
    model.set_option("prefill_tile", prefill_tile)
    B = len(prompts)
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(B, max_positions=max(256, int(max(lens)) + n_frames + 2), max_frames=n_frames)
    try:
        pages = torch.tensor(batch.pages, device=model.device)
        model.kv_view()[pages] = 0
        model.prefill(batch, padded, lens)
        torch.cuda.synchronize()
        kv0 = model.kv_view()[pages].clone()
        model.decode_frames(batch, model.sampling(ignore_stop=True), n_frames)
        torch.cuda.synchronize()
        return dict(kv_prefill=kv0, kv=model.kv_view()[pages].clone(), codes=batch.out_codes.clone(),
                    tl=model.debug_buffer("token_logits", B).clone(), dl=model.debug_buffer("depth_logits", B).clone(),
                    seq_len=batch.seq_len.clone())
    finally:
        model.set_option("tc_min_batch", 9)
        model.set_option("prefill_tile", 0)
        batch.release()


@pytest.mark.parametrize("size", ["smoltts_byte_tiny", "smoltts_byte_150m"])
def test_tc_close_to_cuda_core_variant(size):
    cfg, sd, model, orc = model_and_oracle(size, max_batch=32)
    B = 20
    prompts = [prompt_grid(byte_prompt(30 + b, seed=70 + b), cfg) for b in range(B)]
    tc = _prefill_and_frames(model, prompts, 1, 9)
    cc = _prefill_and_frames(model, prompts, 1, 0)          # CUDA-core tiles of 8 rows, 8 prompt positions per iteration
    assert torch.equal(tc["seq_len"], cc["seq_len"])
    # prefill K/V (every layer: the error compounds with depth) and the first frame's logits
    a, b = tc["kv_prefill"].float(), cc["kv_prefill"].float()
    rel = ((a - b).pow(2).mean().sqrt() / b.pow(2).mean().sqrt()).item()
    exact = (a == b).float().mean().item()
    print(f"{size}: prefill K/V rel rms diff {rel:.5f}, bit-exact {exact:.3f}")
    assert torch.isfinite(a).all() and rel < 0.03 and exact > 0.5
    # (depth logits: position 0 only -- later positions embed the codes each variant picked itself)
    for name in ("tl", "dl"):
        d = (tc[name] - cc[name]).float() if name == "tl" else (tc[name][:, 0] - cc[name][:, 0]).float()
        rms, mx = d.pow(2).mean().sqrt().item(), d.abs().max().item()
        print(f"{size}: {name} rms diff {rms:.4f} max {mx:.4f}")
        assert rms < (0.04 if name == "tl" else 0.06) and mx < 0.3   # the reference's own bf16-vs-fp32 rms: 0.035 / 0.056
    assert (tc["codes"] == cc["codes"]).float().mean().item() > 0.5   # a near-tie flip changes the rest of its frame


def test_tc_prefill_tile_sizes_and_batch_composition_bit_identical():
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_70m", max_batch=32)
    prompts = [prompt_grid(byte_prompt(20 + 5 * b, seed=90 + b), cfg) for b in range(24)]   # ragged lengths
    gs = GenerationSettings(default_temp=0.0, default_fast_temp=0.0)
    whole = generate_batch(model, prompts, gs, audio_only=False, fixed_frames=5, seq_ids=list(range(24)))
    sub = generate_batch(model, prompts[4:20], gs, audio_only=False, fixed_frames=5, seq_ids=list(range(4, 20)))
    for i in range(16):
        assert torch.equal(sub[i], whole[4 + i]), f"sequence {4 + i}: batch of 24 vs batch of 16"
    # one utterance, prefilled in tiles of 128 / 40 / 16 prompt positions (all tensor-core), then decoded at bs=1
    a = _prefill_and_frames(model, prompts[20:21], 3, 9)
    for tile in (40, 16):
        b = _prefill_and_frames(model, prompts[20:21], 3, 9, prefill_tile=tile)
        assert torch.equal(a["kv"].view(torch.int16), b["kv"].view(torch.int16)), f"prefill tile {tile}"
        assert torch.equal(a["codes"], b["codes"])
    # a long prompt: one iteration of 4 row tiles (420 positions; up to 1024 fit) against 128- and 100-position iterations
    long_prompt = [prompt_grid(byte_prompt(420, seed=77), cfg)]
    a = _prefill_and_frames(model, long_prompt, 2, 9)
    for tile in (128, 100):
        b = _prefill_and_frames(model, long_prompt, 2, 9, prefill_tile=tile)
        assert torch.equal(a["kv"].view(torch.int16), b["kv"].view(torch.int16)), f"long prompt, prefill tile {tile}"
        assert torch.equal(a["codes"], b["codes"])


def test_tc_ragged_tiles_three_row_tiles():
    """130 and 300 utterances (a second tile with 2 live rows; three tiles) against the same utterances in batches of 16:
    bit-identical ids -- rows past the batch inside a tile are inert, tiles do not see each other."""
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=300, max_seq_len=96)
    prompts = [prompt_grid(byte_prompt(8 + (b % 11), seed=500 + b), cfg) for b in range(300)]
    gs = GenerationSettings(default_temp=0.0, default_fast_temp=0.0)
    whole = generate_batch(model, prompts, gs, audio_only=False, fixed_frames=4, seq_ids=list(range(300)))
    part = generate_batch(model, prompts[:130], gs, audio_only=False, fixed_frames=4, seq_ids=list(range(130)))
    for b in range(130):
        assert torch.equal(part[b], whole[b]), f"sequence {b}: batch of 130 vs batch of 300"
    for lo in (0, 120, 284):
        sub = generate_batch(model, prompts[lo:lo + 16], gs, audio_only=False, fixed_frames=4, seq_ids=list(range(lo, lo + 16)))
        for i in range(16):
            assert torch.equal(sub[i], whole[lo + i]), f"sequence {lo + i}: batch of 16 vs batch of 300"
    for n in (9, 12):   # the smallest batches the tensor-core variant takes (tc_min_batch = 9)
        sub = generate_batch(model, prompts[40:40 + n], gs, audio_only=False, fixed_frames=4, seq_ids=list(range(40, 40 + n)))
        for i in range(n):
            assert torch.equal(sub[i], whole[40 + i]), f"sequence {40 + i}: batch of {n} vs batch of 300"


def test_tc_stop_rule_and_sampling_inside_a_batch():
    """<|im_end|> forced on some sequences of a 20-utterance batch in frame 2: they freeze (tokens, seq_len, step, codes)
    while the others keep decoding inside the same multi-frame launch; sampled ids follow the CPU sampler spec on the
    dumped logits with the counters (seed, step, seq_id, row) of each sequence."""
    from oracle.sampler_oracle import sample_row

    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=32)
    B, R = 20, cfg.n_rows
    seq_ids = list(range(700, 700 + B))
    prompts = [prompt_grid(byte_prompt(12 + b, seed=800 + b), cfg) for b in range(B)]
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(B, max_positions=96, max_frames=8, seq_ids=seq_ids)
    stopped = [3, 17]
    try:
        model.prefill(batch, padded, lens)
        s = model.sampling(temp=0.8, fast_temp=0.7, top_k=40, top_p=0.9, seed=99, audio_only=True)
        model.decode_frames(batch, s, 1)
        torch.cuda.synchronize()
        tl = model.debug_buffer("token_logits", B).cpu().numpy()
        dl = model.debug_buffer("depth_logits", B).cpu().numpy()
        got = batch.tokens.cpu().tolist()
        for b in (0, 7, 19):
            want = [sample_row(tl[b], 0.8, 40, 0.9, 0.0, 99, 0, seq_ids[b], 0)]
            want += [sample_row(dl[b, i], 0.7, 0, 1.0, 0.0, 99, 0, seq_ids[b], 1 + i) for i in range(cfg.max_fast_seqlen)]
            assert got[b] == want, f"seq {b}: {got[b]} != {want}"
        force = torch.zeros(B, R, dtype=torch.int32, device=model.device)
        force[:, 0] = 400
        for b in stopped:
            force[b, 0] = model.token_config.im_end_id
        model.set_force(force)
        model.decode_frames(batch, s, 1)
        model.set_force(None)
        frozen = (batch.tokens[stopped].clone(), batch.seq_len[stopped].clone())
        model.decode_frames(batch, s, 4)
        torch.cuda.synchronize()
        assert batch.finished.tolist() == [1 if b in stopped else 0 for b in range(B)]
        assert batch.step.tolist() == [2 if b in stopped else 6 for b in range(B)]
        assert torch.equal(batch.tokens[stopped], frozen[0]) and torch.equal(batch.seq_len[stopped], frozen[1])
        assert model.get_option("tc_ready") == 1
    finally:
        model.set_force(None)
        batch.release()


def test_tc_depth7_without_duplicate_code_0():
    """duplicate_code_0 = False (7 depth steps, shifted embedding offsets, SURVEY 8(g)-6) on the tensor-core variant:
    16 utterances greedy-with-resync against the oracle."""
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=16, duplicate_code_0=False)
    assert cfg.max_fast_seqlen == 7
    B, n_frames = 16, 6
    prompts = [prompt_grid(byte_prompt(20 + b, seed=900 + b), cfg) for b in range(B)]
    want, margins = [], []
    with torch.no_grad():
        for p in prompts:
            frames = orc.generate(p, OracleSettings(default_temp=0.0, default_fast_temp=0.0), fixed_frames=n_frames)
            want.append([f.vq for f in frames])
            margins.append([f.margins for f in frames])
    want = torch.tensor(want, dtype=torch.int32)
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(B, max_positions=96, max_frames=n_frames)
    flips, exact = [], 0
    try:
        model.prefill(batch, padded, lens)
        s = model.sampling(ignore_stop=True)
        for f in range(n_frames):
            model.set_force(want[:, f].to(model.device).contiguous())
            model.decode_frames(batch, s, 1)
            torch.cuda.synchronize()
            tl = model.debug_buffer("token_logits", B).cpu()
            dl = model.debug_buffer("depth_logits", B).cpu()
            for b in range(B):
                mine = [int(tl[b].argmax())] + [int(dl[b, i].argmax()) for i in range(cfg.max_fast_seqlen)]
                for r, (a, w) in enumerate(zip(mine, want[b, f].tolist())):
                    if a == w:
                        exact += 1
                    else:
                        flips.append((b, f, r, float(margins[b][f][r])))
    finally:
        model.set_force(None)
        batch.release()
    assert all(m <= TAU for *_, m in flips), f"argmax flipped at a confident decision: {flips}"
    assert exact >= 0.915 * B * n_frames * cfg.n_rows
