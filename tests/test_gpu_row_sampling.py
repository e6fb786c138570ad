"""Per-sequence sampling settings (SmolBatch.row_sampling) on every kernel class: the data-flow kernel alone (bs=1) and in
teams (bs=4, 8), the barrier kernel (bs=3) and its tcgen05 variant (bs=16, 24).

  * a table whose rows all carry the settings s decodes exactly as the call's SmolSampling s without a table (ids, codes,
    dumped logits, KV), whatever the call's own sampling fields say;
  * in a mixed table every row decodes exactly as that row in a batch of the same size where every row carries its setting
    through SmolSampling (compared within a kernel class: the classes sum in different orders), and every sampled id is the
    CPU sampler specification's pick on the dumped logits with the row's parameters and counters;
  * forced ids still win over a table; the stand-alone sampler reads the table too;
  * serving: the continuous batcher with per-request settings == generate_batch with those settings, and SmolTTS.serve with
    per-input settings == synthesize_batch with the same list.
"""
from dataclasses import replace

import numpy as np
import pytest
import torch

from gpu_util import model_and_oracle
from oracle.sampler_oracle import sample_row
from smoltts_b200 import ContinuousBatcher, GenerationSettings, generate_batch
from smoltts_b200.generate import _min_p, pack_prompts
from smoltts_b200.synth import byte_prompt, prompt_grid

pytestmark = pytest.mark.gpu

# (kernel class, batch): ll_max_batch 0 sends a batch of 8 or fewer rows to the barrier kernel; 9+ rows run tcgen05
CLASSES = [("solo", 1), ("teams", 4), ("teams", 8), ("barrier", 3), ("tc", 16), ("tc", 24)]
CHUNKS = [1, 1, 4]   # frames per launch: logits are dumped after each launch, the last launch carries several frames

MIXED = [
    GenerationSettings(default_temp=0.0, default_fast_temp=0.0),
    GenerationSettings(default_temp=0.7, default_fast_temp=0.7, top_k=50, top_p=0.9),
    GenerationSettings(default_temp=1.0, default_fast_temp=1.0, min_p=0.1, min_p_intended=True),
    GenerationSettings(default_temp=0.0, default_fast_temp=0.8),      # greedy slow id, sampled depth codes
    GenerationSettings(default_temp=0.9, default_fast_temp=0.0),      # sampled slow id, greedy depth codes
    GenerationSettings(default_temp=0.6, default_fast_temp=0.5, top_k=10, min_p=0.05, min_p_intended=True),
]


def _mixed(B):
    """Row b carries MIXED[b % 6] with a seed of its own."""
    return [replace(MIXED[b % len(MIXED)], seed=1000 + 17 * b) for b in range(B)]


def _model():
    return model_and_oracle("smoltts_byte_tiny", max_batch=32, max_seq_len=256)


def _decode(model, kernel, prompts, seq_ids, call, table=None):
    """Prefill + CHUNKS frames; call: the SmolSampling of every launch, table: row settings or None."""
    B = len(prompts)
    n = sum(CHUNKS)
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(B, max_positions=int(padded.shape[2]) + n + 1, max_frames=n, seq_ids=seq_ids)
    model.set_option("ll_max_batch", 0 if kernel == "barrier" else 8)
    try:
        pages = torch.tensor(batch.pages, device=model.device)
        model.kv_view()[pages] = 0
        model.prefill(batch, padded, lens)
        batch.set_row_sampling(model.row_sampling(table) if table is not None else None)
        logits = []
        for c in CHUNKS:
            model.decode_frames(batch, call, c)
            torch.cuda.synchronize()
            logits.append((model.debug_buffer("token_logits", B).cpu().clone(), model.debug_buffer("depth_logits", B).cpu().clone()))
        if kernel == "tc":
            assert model.get_option("tc_ready") == 1, "the tcgen05 variant did not run"
        return dict(codes=batch.out_codes.cpu().clone(), tokens=batch.tokens.cpu().clone(), seq_len=batch.seq_len.cpu().clone(),
                    step=batch.step.cpu().clone(), kv=model.kv_view()[pages].cpu().clone().view(torch.int16).view(B, -1), logits=logits)
    finally:
        model.set_option("ll_max_batch", 8)
        batch.release()


def _same_rows(got, want, rows, what):
    for k in ("codes", "tokens", "seq_len", "step", "kv"):
        assert torch.equal(got[k][rows], want[k][rows]), f"{what}: {k} of rows {rows} differ"
    for (gt, gd), (wt, wd) in zip(got["logits"], want["logits"]):
        assert torch.equal(gt[rows], wt[rows]) and torch.equal(gd[rows], wd[rows]), f"{what}: logits of rows {rows} differ"


def _prompts(cfg, B, seed):
    return [prompt_grid(byte_prompt(14 + (5 * b) % 11, seed=seed + b), cfg) for b in range(B)]


@pytest.mark.parametrize("kernel,B", CLASSES)
def test_uniform_table_equals_call_settings(kernel, B):
    cfg, _, model, _ = _model()
    prompts, seq_ids = _prompts(cfg, B, 300), [50 + 3 * b for b in range(B)]
    gs = GenerationSettings(default_temp=0.8, default_fast_temp=0.7, top_k=40, top_p=0.9, min_p=0.02, min_p_intended=True, seed=7)
    want = _decode(model, kernel, prompts, seq_ids, model.sampling(temp=0.8, fast_temp=0.7, top_k=40, top_p=0.9, min_p=0.02, seed=7,
                                                                   ignore_stop=True))
    # the call's own temperature / top-k / top-p / min-p / seed say greedy: with a table they are ignored
    got = _decode(model, kernel, prompts, seq_ids, model.sampling(ignore_stop=True), table=[gs] * B)
    _same_rows(got, want, list(range(B)), f"{kernel} bs={B}: uniform table vs SmolSampling")
    greedy = _decode(model, kernel, prompts, seq_ids, model.sampling(ignore_stop=True))
    assert not torch.equal(greedy["codes"], want["codes"]), "sampled and greedy decoding agree: the test would prove nothing"


@pytest.mark.parametrize("kernel,B", [c for c in CLASSES if c[1] > 1])
def test_mixed_table_rows_equal_uniform_batches(kernel, B):
    cfg, _, model, _ = _model()
    prompts, seq_ids = _prompts(cfg, B, 500), [900 + b for b in range(B)]
    rows = _mixed(B)
    got = _decode(model, kernel, prompts, seq_ids, model.sampling(ignore_stop=True), table=rows)
    for b in range(min(B, 2 * len(MIXED))):   # one uniform batch per row: every setting twice, with two seeds
        s = rows[b]
        call = model.sampling(temp=s.default_temp, fast_temp=s.default_fast_temp, top_k=s.top_k, top_p=s.top_p, min_p=_min_p(s),
                              seed=s.seed, ignore_stop=True)
        want = _decode(model, kernel, prompts, seq_ids, call)
        _same_rows(got, want, [b], f"{kernel} bs={B}: row {b} in a mixed table vs a uniform batch")
    # sampled ids = the CPU sampler specification on the dumped logits, with the row's parameters and counters
    ends = np.cumsum(CHUNKS) - 1
    for (tl, dl), f in zip(got["logits"], ends):
        for b in range(B):
            s = rows[b]
            want = [sample_row(tl[b].numpy(), s.default_temp, s.top_k, s.top_p, _min_p(s), s.seed, int(f), seq_ids[b], 0)]
            want += [sample_row(dl[b, i].numpy(), s.default_fast_temp, 0, 1.0, _min_p(s), s.seed, int(f), seq_ids[b], 1 + i)
                     for i in range(cfg.max_fast_seqlen)]
            assert got["codes"][b, f].tolist() == want, f"{kernel} bs={B}: frame {f} row {b}: {got['codes'][b, f].tolist()} != {want}"


@pytest.mark.parametrize("kernel,B", [("teams", 4), ("barrier", 3), ("tc", 16)])
def test_forced_ids_win_over_the_table(kernel, B):
    cfg, _, model, _ = _model()
    prompts = _prompts(cfg, B, 650)
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(B, max_positions=int(padded.shape[2]) + 4, max_frames=3)
    model.set_option("ll_max_batch", 0 if kernel == "barrier" else 8)
    force = torch.randint(0, cfg.codebook_size, (3, B, cfg.n_rows), generator=torch.Generator().manual_seed(5), dtype=torch.int32)
    force[:, :, 0] += model.token_config.semantic_start_id
    try:
        model.prefill(batch, padded, lens)
        batch.set_row_sampling(model.row_sampling(_mixed(B)))
        for f in range(3):
            dforce = force[f].to(model.device).contiguous()
            model.set_force(dforce)
            model.decode_frames(batch, model.sampling(ignore_stop=True), 1)
            torch.cuda.synchronize()
        model.set_force(None)
        assert torch.equal(batch.out_codes.cpu(), force.permute(1, 0, 2)), f"{kernel}: forced ids must replace sampled and greedy ones"
    finally:
        model.set_force(None)
        model.set_option("ll_max_batch", 8)
        batch.release()


def test_standalone_sampler_reads_the_table():
    cfg, _, model, _ = _model()
    B, n = 6, cfg.vocab_size
    rows = _mixed(B)
    batch = model.new_batch(B, max_positions=32, max_frames=1, seq_ids=[40 + b for b in range(B)])
    try:
        batch.set_row_sampling(model.row_sampling(rows))
        logits = torch.randn(B, n, generator=torch.Generator().manual_seed(9)).mul(3.0).to(torch.bfloat16).float()
        for stream in (0, 2):
            got = model.sample(logits.to(model.device), model.sampling(), stream, batch).tolist()
            for b, s in enumerate(rows):
                temp = s.default_temp if stream == 0 else s.default_fast_temp
                top_k, top_p = (s.top_k, s.top_p) if stream == 0 else (0, 1.0)
                want = sample_row(logits[b].numpy(), temp, top_k, top_p, _min_p(s), s.seed, 0, 40 + b, stream)
                assert got[b] == want, f"stream {stream} row {b}: {got[b]} != {want}"
    finally:
        batch.release()


@pytest.mark.parametrize("slots", [16, 4])
def test_continuous_batcher_with_per_request_settings(slots):
    """Ragged budgets, late admissions, a setting and a seed per request; the stop rule stays on.  4 slots (data-flow teams)
    against generate_batch([prompt], settings_i) -- one utterance, the same kernel's solo grid --; 16 slots (tcgen05) against
    generate_batch over groups of 16 rows with per-row settings (the same kernel class)."""
    cfg, _, model, _ = _model()
    n = 2 * slots + 3
    prompts = [prompt_grid(byte_prompt(2 + (7 * i) % 23, seed=700 + i), cfg) for i in range(n)]
    budgets = [5 + (11 * i) % 19 for i in range(n)]
    uids = [200 + i for i in range(n)]
    per = [replace(MIXED[i % len(MIXED)], seed=31 * i, max_new_tokens=budgets[i] - 1) for i in range(n)]
    base = GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=23)
    cb = ContinuousBatcher(model, base, slots=slots, max_prompt=64, chunk=4, audio_only=False)
    for i in range(n):
        cb.submit(prompts[i], uid=uids[i], settings=per[i])
    got = dict(cb.run())
    cb.close()
    assert sorted(got) == sorted(uids) and cb.stats["admitted"] == n
    if slots <= 8:
        for i in range(n):
            want = generate_batch(model, [prompts[i]], [per[i]], audio_only=False, seq_ids=[uids[i]])[0]
            assert torch.equal(got[uids[i]], want), f"utterance {i}: batcher {tuple(got[uids[i]].shape)} vs generate_batch {tuple(want.shape)}"
    else:
        for g in range(0, n, slots):
            sel = list(range(g, min(g + slots, n)))
            sel += [sel[-1]] * (slots - len(sel))       # same batch size, same kernel class
            outs = generate_batch(model, [prompts[j] for j in sel], [per[j] for j in sel], audio_only=False, seq_ids=[uids[j] for j in sel])
            for j, o in zip(sel, outs):
                assert torch.equal(got[uids[j]], o), f"utterance {j}: batcher vs generate_batch with per-row settings"


def test_serve_with_per_input_settings_equals_synthesize_batch():
    from smoltts_b200 import MimiModel, PromptEncoder, SmolTTS, byte_level_tokenizer
    from smoltts_b200.synth import make_mimi_state_dict

    cfg, _, lm, _ = model_and_oracle("smoltts_byte_tiny", max_batch=8, max_seq_len=256)
    enc = PromptEncoder.from_model(byte_level_tokenizer(cfg.codebook_size), lm)
    codec = MimiModel(max_streams=8, max_frames=32, upsample_carry=True)
    codec.load_state_dict(make_mimi_state_dict(0))
    tts = SmolTTS(lm, enc, codec, settings=GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=9))
    texts = [f"Request {i} with its own voice settings{'?' * i}" for i in range(7)]
    per = [replace(MIXED[i % len(MIXED)], seed=5 + i, max_new_tokens=6 + 2 * i) for i in range(7)]
    got = dict(tts.serve(texts, slots=3, chunk=4, max_prompt=128, settings=per))
    want = tts.synthesize_batch(texts, settings=per)
    assert sorted(got) == list(range(7))
    for i in range(7):
        assert got[i].shape == want[i].shape, (i, got[i].shape, want[i].shape)
        assert np.array_equal(got[i], want[i]), f"input {i}: served audio differs from batch synthesis with the same settings"
    plain = tts.synthesize_batch(texts)
    assert any(p.shape != w.shape or not np.array_equal(p, w) for p, w in zip(plain, want)), "per-input settings changed nothing"
