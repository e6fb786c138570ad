"""Frame-level parity on the GPU, through the C-ABI.

Tolerances are calibrated, not guessed (SURVEY §8(c), DESIGN.md "Parity"): on these seeded
random-init weights the reference's own eager bf16 forward differs from its fp32 forward by
rms 0.035 / 0.056 (token / codebook logits, 150m) and two bf16 executions that only differ in GEMM
shape differ by up to 0.19.  The north star's example (max-abs 2e-2) is tighter than the reference is
with itself, so the bars here are:
  * error of the CUDA path against the reference's fp32 logits <= 1.3x (rms) and 1.6x (max) the
    error of the reference's bf16 logits against the same fp32 logits;
  * argmax agreement with the fp32 reference wherever its top-2 margin exceeds TAU;
  * greedy ids bit-exact against the oracle up to decisions whose oracle margin is <= TAU
    (greedy-with-resync: the oracle's id is adopted and decoding continues).
"""
import numpy as np
import pytest
import torch

from conftest import bf16_bits_to_f32, load_golden
from gpu_util import model_and_oracle, np_rms
from oracle.dualar_oracle import OracleSettings
from oracle.sampler_oracle import OracleSampler, sample_row
from smoltts_b200.synth import byte_prompt, prompt_grid

pytestmark = pytest.mark.gpu

SIZES = ["smoltts_byte_tiny", "smoltts_byte_70m", "smoltts_byte_150m"]
TAU = 0.15  # logit margin below which bf16 noise may legitimately flip an argmax (largest flip margin ever observed: 0.14)
# share of greedy decisions that must be identical to the oracle's BEFORE any resync.  Decisions at a margin of one or two
# bf16 ulps of the logit (0.0156 .. 0.0625) are coin flips between two bf16 executions, so the count moves by a few
# decisions from build to build (measured: tiny 213/216, 70m 202..208/216, 150m 101/108); the hard bar is TAU
MIN_EXACT = {"smoltts_byte_tiny": 0.95, "smoltts_byte_70m": 0.90, "smoltts_byte_150m": 0.88}


def _teacher_forced(model, grid, t0):
    """Feeds grid [B, R, S] column by column; returns token logits for positions t0..S-2 and the
    depth logits of those frames (teacher-forced with the next column)."""
    B, R, S = grid.shape
    dev = model.device
    batch = model.new_batch(B, max_positions=S + 8, max_frames=S)
    tok, cb = [], []
    try:
        g32 = grid.to(device=dev, dtype=torch.int32).contiguous()
        lens = torch.full((B,), t0 + 1, dtype=torch.int32, device=dev)
        model.prefill(batch, g32[:, :, : t0 + 1].contiguous(), lens)
        s = model.sampling(ignore_stop=True)
        for t in range(t0, S - 1):
            force = g32[:, :, t + 1].contiguous()
            model.set_force(force)
            model.decode_frames(batch, s, 1)
            torch.cuda.synchronize()
            tok.append(model.debug_buffer("token_logits", B).cpu().clone())
            cb.append(model.debug_buffer("depth_logits", B).cpu().clone())
        model.set_force(None)
        assert batch.seq_len.tolist() == [S - 1] * B
        assert torch.equal(batch.tokens.cpu(), grid[:, :, S - 1].to(torch.int32))
    finally:
        model.set_force(None)
        batch.release()
    return torch.stack(tok, 1).numpy(), torch.stack(cb, 1).numpy()


@pytest.mark.parametrize("size", SIZES)
def test_teacher_forced_logits_vs_reference(size):
    g = load_golden(size)
    cfg, sd, model, orc = model_and_oracle(size)
    grid = torch.from_numpy(g["grid"].astype(np.int64))
    t0, sub = int(g["cb_t0"]), int(g["sub"])
    tok, cb = _teacher_forced(model, grid, t0)            # [B, n, V], [B, n, Nf, C]
    n = tok.shape[1]
    ref_bf = bf16_bits_to_f32(g["tok_bf16"])[:, t0:t0 + n]
    ref_f32 = g["tok_f32_sub"][:, t0:t0 + n]
    refc_bf = bf16_bits_to_f32(g["cb_bf16"])[:, :n]
    refc_f32 = g["cb_f32_sub"][:, :n]
    for name, ours, rbf, rf in (("token", tok, ref_bf, ref_f32), ("codebook", cb, refc_bf, refc_f32)):
        ours_s, rbf_s = ours[..., ::sub], rbf[..., ::sub]
        e_ours, e_ref = np_rms(ours_s, rf), np_rms(rbf_s, rf)
        m_ours, m_ref = np.abs(ours_s - rf).max(), np.abs(rbf_s - rf).max()
        print(f"{size} {name}: rms vs fp32 ours {e_ours:.4f} ref-bf16 {e_ref:.4f}; max ours {m_ours:.4f} ref {m_ref:.4f}; "
              f"ours vs ref-bf16 max {np.abs(ours - rbf).max():.4f} exact {(ours == rbf).mean():.3f}")
        assert e_ours <= 1.3 * e_ref + 1e-3, f"{name}: rms error {e_ours} vs reference-bf16's own {e_ref}"
        assert m_ours <= 1.6 * m_ref + 1e-2, f"{name}: max error {m_ours} vs reference-bf16's own {m_ref}"
    # argmax agreement with the fp32 reference wherever its decision is not a near-tie
    am, mg = g["tok_f32_argmax"][:, t0:t0 + n], g["tok_f32_margin"][:, t0:t0 + n]
    ok = (tok.argmax(-1) == am) | (mg <= TAU)
    assert ok.all(), f"token argmax differs from fp32 reference at margins {mg[~ok]}"
    amc, mgc = g["cb_f32_argmax"][:, :n], g["cb_f32_margin"][:, :n]
    okc = (cb.argmax(-1) == amc) | (mgc <= TAU)
    assert okc.all(), f"codebook argmax differs from fp32 reference at margins {mgc[~okc]}"


@pytest.mark.parametrize("size", SIZES)
def test_greedy_with_resync_vs_oracle(size):
    """Free-running greedy decode vs the CPU oracle on a synthetic byte prompt.  Every id must be
    identical unless the oracle's own top-2 margin at that decision is <= TAU; on such a flip the
    oracle's id is adopted (smol_set_force) and decoding continues."""
    cfg, sd, model, orc = model_and_oracle(size)
    n_frames = 24 if size != "smoltts_byte_150m" else 12
    prompt = prompt_grid(byte_prompt(40, seed=3), cfg)
    with torch.no_grad():
        frames = orc.generate(prompt, OracleSettings(default_temp=0.0, default_fast_temp=0.0), fixed_frames=n_frames)
    want = torch.tensor([f.vq for f in frames], dtype=torch.int32)          # [n, R]
    margins = np.array([f.margins for f in frames])
    dev = model.device
    batch = model.new_batch(1, max_positions=128, max_frames=n_frames)
    flips, exact = [], 0
    try:
        p32 = prompt[None].to(device=dev, dtype=torch.int32).contiguous()
        model.prefill(batch, p32, torch.tensor([prompt.shape[1]], dtype=torch.int32, device=dev))
        s = model.sampling(ignore_stop=True)
        for f in range(n_frames):
            model.set_force(want[f:f + 1].to(dev).contiguous())
            model.decode_frames(batch, s, 1)
            torch.cuda.synchronize()
            tl = model.debug_buffer("token_logits", 1)[0].cpu()
            dl = model.debug_buffer("depth_logits", 1)[0].cpu()
            mine = [int(tl.argmax())] + [int(dl[i].argmax()) for i in range(cfg.max_fast_seqlen)]
            for r, (a, b) in enumerate(zip(mine, want[f].tolist())):
                if a == b:
                    exact += 1
                else:
                    flips.append((f, r, float(margins[f, r])))
    finally:
        model.set_force(None)
        batch.release()
    total = n_frames * cfg.n_rows
    first = (f"first divergence at frame {flips[0][0]} row {flips[0][1]} (decision {flips[0][0] * cfg.n_rows + flips[0][1]} of {total}), "
             f"oracle margin {flips[0][2]:.4f}") if flips else "no divergence"
    print(f"{size}: {exact}/{total} greedy decisions identical; {first}; flips (frame,row,oracle margin): {flips}")
    assert all(m <= TAU for _, _, m in flips), f"argmax flipped at a confident decision: {flips}"
    assert exact >= MIN_EXACT[size] * total, f"{exact}/{total} identical decisions, below the measured rate"


@pytest.mark.parametrize("size", ["smoltts_byte_tiny", "smoltts_byte_70m"])
def test_greedy_vs_literal_reference_goldens(size):
    """Free-running greedy ids against the ids the UNMODIFIED reference emits when driven through
    RQTransformer.forward (tests/golden).  Compared up to the first reference decision whose margin is
    <= TAU (after a flip the histories differ)."""
    from smoltts_b200 import GenerationSettings, generate_batch

    g = load_golden(size)
    cfg, sd, model, orc = model_and_oracle(size)
    ids, margins = g["greedy_ids_bf16"], g["greedy_margin_bf16"]
    prompt = torch.from_numpy(g["greedy_prompt"].astype(np.int64))
    outs = generate_batch(model, [prompt], GenerationSettings(default_temp=0.0, default_fast_temp=0.0),
                          audio_only=False, fixed_frames=ids.shape[0])
    got = outs[0].t().numpy()  # [n, R]
    checked = 0
    for f in range(ids.shape[0]):
        for r in range(cfg.n_rows):
            if got[f, r] != ids[f, r]:
                assert margins[f, r] <= TAU, f"frame {f} row {r}: {got[f, r]} != {ids[f, r]} at margin {margins[f, r]}"
                print(f"{size}: matched {checked} ids, then a near-tie flip at margin {margins[f, r]:.4f}")
                return
            checked += 1
    print(f"{size}: all {checked} greedy ids equal the literal reference's")


def test_modes_and_batch_composition_are_bit_identical():
    """mode 0 == mode 2 whatever the number of frames per launch (chunks of 7, 20 and 9), and a sequence decodes to the
    same ids alone, inside a batch of 3, and inside a batch of 11 (two batch tiles) -- on the GEMV variants of the barrier
    kernel (the tcgen05 variant, which would take the batch of 11 and every prefill, is switched off here: it is
    bit-identical with itself, tests/test_gpu_tc.py, not with the GEMV kernels)."""
    from smoltts_b200 import GenerationSettings, generate_batch

    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=16)
    prompts = [prompt_grid(byte_prompt(10 + 3 * b, seed=20 + b), cfg) for b in range(11)]
    gs = GenerationSettings(default_temp=0.8, default_fast_temp=0.6, top_k=40, top_p=0.9, seed=77)
    try:
        model.set_option("tc_min_batch", 0)
        model.set_option("ll_max_batch", 0)   # the data-flow kernel (batches of 1..8 by default) has its own test: test_gpu_ll2.py
        _modes_and_composition(model, prompts, gs)
    finally:
        model.set_option("tc_min_batch", 9)
        model.set_option("ll_max_batch", 8)
        model.set_option("mode", 2)


def _modes_and_composition(model, prompts, gs):
    from smoltts_b200 import generate_batch

    model.set_option("mode", 0)
    try:
        ref = generate_batch(model, prompts, gs, audio_only=False, fixed_frames=20, chunk=7)
        alt = generate_batch(model, prompts, gs, audio_only=False, fixed_frames=20, chunk=20)
    finally:
        model.set_option("mode", 2)  # default: data-flow kernel up to 8 sequences, barrier kernel above
    for a, b in zip(ref, alt):
        assert torch.equal(a, b)
    dflt = generate_batch(model, prompts, gs, audio_only=False, fixed_frames=20, chunk=9)
    for a, b in zip(ref, dflt):
        assert torch.equal(a, b)
    # alone / in a batch of 3: still on the barrier kernel (the data-flow kernel sums its dot products on the tensor cores, in
    # another order; its own invariances are tests/test_gpu_ll2.py, its parity the oracle tests of this file)
    solo = generate_batch(model, prompts[4:5], gs, audio_only=False, fixed_frames=20, seq_ids=[4])
    assert torch.equal(solo[0], ref[4])
    trio = generate_batch(model, prompts[3:6], gs, audio_only=False, fixed_frames=20, seq_ids=[3, 4, 5])
    assert torch.equal(trio[1], ref[4])


@pytest.mark.parametrize("size,lens", [("smoltts_byte_tiny", [45]), ("smoltts_byte_70m", [70]), ("smoltts_byte_tiny", [33, 9, 58])])
def test_prefill_tiles_write_identical_kv(size, lens):
    """Prefill on the CUDA-core barrier kernel (fewer than 9 rows) -- 8 / 3 / 1 prompt positions per iteration -- then two
    frames: bit-identical K/V, seq_len, pending tokens and codes, also for ragged prompt lengths (rows of a tile past the end
    of a prompt are inert)."""
    from smoltts_b200.generate import pack_prompts

    cfg, sd, model, orc = model_and_oracle(size)
    B = len(lens)
    prompts = [prompt_grid(byte_prompt(n, seed=110 + b), cfg) for b, n in enumerate(lens)]
    tiles = [8 // B, 1] + ([3] if B == 1 else [])
    got = []
    model.set_option("ll_max_batch", 0)       # the two frames on the barrier kernel too
    try:
        for tile in tiles:
            model.set_option("prefill_tile", tile)
            padded, lens_t = pack_prompts(model, prompts)
            batch = model.new_batch(B, max_positions=128, max_frames=4)
            try:
                pages = torch.tensor(batch.pages, device=model.device)
                model.kv_view()[pages] = 0
                model.prefill(batch, padded, lens_t)
                model.decode_frames(batch, model.sampling(ignore_stop=True), 2)
                torch.cuda.synchronize()
                got.append((model.kv_view()[pages].clone(), batch.seq_len.clone(), batch.tokens.clone(), batch.out_codes.clone()))
            finally:
                batch.release()
    finally:
        model.set_option("prefill_tile", 0)
        model.set_option("ll_max_batch", 8)
    assert got[0][1].tolist() == [n + 12 - 1 + 2 for n in lens]
    for tile, g in zip(tiles[1:], got[1:]):
        assert torch.equal(g[0].view(torch.int16), got[0][0].view(torch.int16)), f"KV differs (tile {tile})"
        for a, b in zip(g[1:], got[0][1:]):
            assert torch.equal(a, b), f"state differs (tile {tile})"


@pytest.mark.parametrize("cfgset", [
    dict(temp=0.0, fast_temp=0.0),
    dict(temp=0.7, fast_temp=0.7),
    dict(temp=0.7, fast_temp=0.5, top_k=50, top_p=0.9),
    dict(temp=1.3, fast_temp=1.0, top_k=5),
    dict(temp=0.4, fast_temp=0.4, top_p=0.5, min_p=0.05),
    dict(temp=1.0, fast_temp=1.0, top_k=1),
])
def test_sampler_kernel_bit_exact_vs_oracle(cfgset):
    """Identical logits + identical Philox counters -> identical ids (integer-weight sampler)."""
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny")
    g = torch.Generator().manual_seed(123)
    for n, stream in ((2368, 0), (2048, 3), (100, 0), (4096, 1)):
        B = 37
        logits = (torch.randn(B, n, generator=g) * 3.0).to(torch.bfloat16).float()
        logits[0, : n // 2] = logits[0, 0]  # ties
        logits[1] = 0.0                     # all equal
        s = model.sampling(seed=0xABCDEF0123, **cfgset)
        got = model.sample(logits.to(model.device), s, stream).cpu().tolist()
        temp = cfgset["temp"] if stream == 0 else cfgset["fast_temp"]
        tk, tp = (cfgset.get("top_k", 0), cfgset.get("top_p", 1.0)) if stream == 0 else (0, 1.0)
        want = [sample_row(logits[b].numpy(), temp, tk, tp, cfgset.get("min_p", 0.0), 0xABCDEF0123, 0, b, stream)
                for b in range(B)]
        assert got == want, f"n={n} stream={stream}: {sum(a != b for a, b in zip(got, want))} of {B} ids differ"


def test_sampler_distribution_chi_square():
    """Empirical frequencies of the kernel's draws follow the exact filtered distribution of the spec."""
    from oracle.sampler_oracle import kept_distribution

    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny")
    g = torch.Generator().manual_seed(9)
    n, N = 64, 20000
    row = (torch.randn(n, generator=g) * 1.5).to(torch.bfloat16).float()
    logits = row[None].repeat(N, 1).contiguous()
    s = model.sampling(temp=0.9, fast_temp=0.9, top_k=20, top_p=0.95, seed=5)
    ids = model.sample(logits.to(model.device), s, 0).cpu().numpy()
    p = kept_distribution(row.numpy(), 0.9, 20, 0.95, 0.0)
    counts = np.bincount(ids, minlength=n).astype(np.float64)
    assert counts[p == 0].sum() == 0
    live = p > 0
    chi2 = (((counts[live] - N * p[live]) ** 2) / (N * p[live])).sum()
    dof = live.sum() - 1
    assert chi2 < dof + 6 * np.sqrt(2 * dof), f"chi2 {chi2:.1f} for {dof} dof"


def test_sampled_decode_counters_and_filters_inside_the_frame_kernel():
    """Whole-frame sampled decoding (temperature + top-k + top-p on the slow id, temperature on the
    depth codes): every id the frame kernel emitted must equal what the CPU sampler specification
    picks from the SAME logits (dumped by the kernel) with the counters (seed, step, seq_id, stream) the
    kernel is supposed to use.  Independent of bf16 noise: bit-exact."""
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny")
    n_frames, B = 12, 3
    seq_ids = [5, 9, 2]
    prompts = [prompt_grid(byte_prompt(24 + b, seed=8 + b), cfg) for b in range(B)]
    from smoltts_b200.generate import pack_prompts

    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(B, max_positions=128, max_frames=n_frames, seq_ids=seq_ids)
    try:
        model.prefill(batch, padded, lens)
        kw = dict(temp=0.7, fast_temp=0.6, top_k=50, top_p=0.9, seed=1234)
        s = model.sampling(ignore_stop=True, **kw)
        for f in range(n_frames):
            model.decode_frames(batch, s, 1)
            torch.cuda.synchronize()
            tl = model.debug_buffer("token_logits", B).cpu().numpy()
            dl = model.debug_buffer("depth_logits", B).cpu().numpy()
            got = batch.tokens.cpu().tolist()
            for b in range(B):
                want = [sample_row(tl[b], 0.7, 50, 0.9, 0.0, 1234, f, seq_ids[b], 0)]
                want += [sample_row(dl[b, i], 0.6, 0, 1.0, 0.0, 1234, f, seq_ids[b], 1 + i) for i in range(cfg.max_fast_seqlen)]
                assert got[b] == want, f"frame {f} seq {b}: {got[b]} != {want}"
        assert batch.step.tolist() == [n_frames] * B
    finally:
        batch.release()


def test_generate_api_and_stop_rule():
    from smoltts_b200 import GenerationSettings, SingleBatchGenerator, generate_batch, generate_blocking

    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny")
    prompt = prompt_grid(byte_prompt(16, seed=2), cfg)
    gs = GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=9)
    gen = SingleBatchGenerator(model, prompt, gs, audio_only=False)
    toks = list(gen)
    assert len(toks) == 10  # max_new_tokens + 1 frames (reference lm/generate.py:60,161)
    cols = torch.cat([t.vq_tensor for t in toks], dim=-1)[0].cpu()  # [R, 10]
    outs = generate_batch(model, [prompt], gs, audio_only=False)
    assert torch.equal(outs[0], cols)
    blk = generate_blocking(model, prompt, gs, audio_only=False)
    assert torch.equal(blk[0].cpu(), cols)
    # stop rule: force <|im_end|> as the slow id of frame 3
    R = cfg.n_rows
    force = torch.zeros(1, R, dtype=torch.int32, device=model.device)
    force[0, 0] = model.token_config.im_end_id
    gen = SingleBatchGenerator(model, prompt, gs, audio_only=True)
    seen = []
    for i, t in enumerate(gen):
        seen.append(t)
        model.set_force(force if i == 1 else None)  # applies to the NEXT frame
    model.set_force(None)
    assert len(seen) == 3 and seen[-1].semantic_code == model.token_config.im_end_id and seen[-1].audio_codes is None


def test_capacity_and_error_reporting():
    from smoltts_b200 import _capi

    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny")
    batch = model.new_batch(1, max_positions=32)
    try:
        with pytest.raises(_capi.SmolError) as ei:
            model.decode_frames(batch, model.sampling(), 64)
        assert ei.value.code == _capi.SMOL_ERR_CAPACITY
        with pytest.raises(_capi.SmolError):
            model.run_phases(batch, model.sampling(), 5, 3)
    finally:
        batch.release()
