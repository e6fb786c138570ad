"""Split staging of the fused MLP's partial sums (ll2_kernel.cu: gather_psum_split, option ll_psum_split): each CTA of a
cluster polls 1/S of the 7 x dim partial-sum words and forwards its quads to the whole cluster through DSMEM, instead of
every CTA polling all of them (ll_psum_split = 0).  The split staging, the per-CTA staging and the unfused program
(ll_fused_mlp = 0) must compute the same bits: codes, tokens, seq_len, step, finished, every cached K/V value and the
fp32 logits -- over one launch and several, long contexts, sampled ids, forced ids and the stop rule, and n_ctas grids with
and without the fused program.
"""
import pytest
import torch

from gpu_util import model_and_oracle
from smoltts_b200.generate import pack_prompts
from smoltts_b200.synth import byte_prompt, prompt_grid

pytestmark = pytest.mark.gpu

# (ll_fused_mlp, ll_psum_split) of each program
PROGRAMS = {"split": (1, 1), "per-CTA": (1, 0), "unfused": (0, 1)}


def _run(model, prompt, n_frames, chunks, program, force_at=None, expect_fused=None, **skw):
    fused, split = PROGRAMS[program]
    model.set_option("ll_fused_mlp", fused)
    model.set_option("ll_psum_split", split)
    padded, lens = pack_prompts(model, [prompt])
    batch = model.new_batch(1, max_positions=int(padded.shape[2]) + n_frames + 1, max_frames=n_frames, seq_ids=[3])
    try:
        pages = torch.tensor(batch.pages, device=model.device)
        model.kv_view()[pages] = 0
        model.prefill(batch, padded, lens)
        s = model.sampling(**skw)
        done = 0
        for n in chunks:
            if force_at is not None and done <= force_at < done + n:
                force = torch.zeros(1, model.config.n_rows, dtype=torch.int32, device=model.device)
                force[0, 0] = model.token_config.im_end_id
                model.set_force(force)
            model.decode_frames(batch, s, n)
            model.set_force(None)
            done += n
        torch.cuda.synchronize()
        assert model.get_option("ll_ready") == 1, "the data-flow kernel did not run"
        want_fused = fused if expect_fused is None else expect_fused
        assert model.get_option("ll_last_fused") == want_fused, f"{program}: the launch ran the other MLP program"
        assert model.get_option("ll_last_split") == (split if want_fused else 0), f"{program}: the launch staged the partial sums the other way"
        return dict(codes=batch.out_codes.clone(), tokens=batch.tokens.clone(), seq_len=batch.seq_len.clone(),
                    step=batch.step.clone(), finished=batch.finished.clone(), kv=model.kv_view()[pages].clone(),
                    logits=(model.debug_buffer("token_logits", 1).clone(), model.debug_buffer("depth_logits", 1).clone()))
    finally:
        model.set_force(None)
        model.set_option("ll_fused_mlp", 1)
        model.set_option("ll_psum_split", 1)
        batch.release()


def _same(a, b, what):
    for k in ("codes", "tokens", "seq_len", "step", "finished"):
        assert torch.equal(a[k], b[k]), f"{what}: {k} differ"
    assert torch.equal(a["kv"].view(torch.int16), b["kv"].view(torch.int16)), f"{what}: KV differs"
    assert torch.equal(a["logits"][0], b["logits"][0]) and torch.equal(a["logits"][1], b["logits"][1]), f"{what}: logits differ"


def _fused_fits(model):
    if model.get_option("ll_mlp_cluster") <= 0:
        pytest.skip("no thread-block cluster size of the fused MLP fits this GPU")


def _all_same(model, prompt, n_frames, chunk_sets, what, **kw):
    """Every program and every way of cutting the frames into launches against the unfused program in one launch."""
    ref = _run(model, prompt, n_frames, [n_frames], "unfused", **kw)
    _fused_fits(model)
    for chunks in chunk_sets:
        for program in ("split", "per-CTA"):
            _same(ref, _run(model, prompt, n_frames, chunks, program, **kw), f"{what}: {program}, launches {chunks}")


@pytest.mark.parametrize("size,n_prompt", [("smoltts_byte_tiny", 20), ("smoltts_byte_70m", 100), ("smoltts_byte_150m", 180)])
def test_psum_split_is_bit_identical(size, n_prompt):
    cfg, sd, model, orc = model_and_oracle(size, max_batch=1)
    prompt = prompt_grid(byte_prompt(n_prompt, seed=41), cfg)
    _all_same(model, prompt, 12, [[12], [5, 4, 3]], size, ignore_stop=True)


def test_psum_split_long_context():
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_70m", max_batch=1, max_seq_len=2304)
    prompt = prompt_grid(byte_prompt(1300, seed=71), cfg)
    _all_same(model, prompt, 14, [[14], [1] * 14], "70m, 1300-token prompt", ignore_stop=True)


@pytest.mark.parametrize("fast_temp", [0.6, 0.0])
def test_psum_split_sampled(fast_temp):
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=1)
    prompt = prompt_grid(byte_prompt(24, seed=9), cfg)
    kw = dict(temp=0.7, fast_temp=fast_temp, top_k=50, top_p=0.9, seed=1234, ignore_stop=True)
    _all_same(model, prompt, 12, [[12], [7, 5]], f"sampled, fast_temp {fast_temp}", **kw)


def test_psum_split_forced_ids_and_stop_rule():
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=1)
    prompt = prompt_grid(byte_prompt(14, seed=82), cfg)
    ref = _run(model, prompt, 8, [1, 3, 4], "unfused", force_at=1, audio_only=True)
    assert ref["finished"].tolist() == [1]
    _fused_fits(model)
    for program in ("split", "per-CTA"):
        _same(ref, _run(model, prompt, 8, [1, 3, 4], program, force_at=1, audio_only=True), f"forced <|im_end|>: {program}")


@pytest.mark.parametrize("size", ["smoltts_byte_tiny", "smoltts_byte_150m"])
def test_psum_split_under_an_n_ctas_override(size):
    """7 clusters of S CTAs (no idle cluster) keep the fused program with split staging; 7 S + 1 CTAs run unfused."""
    cfg, sd, model, orc = model_and_oracle(size, max_batch=1)
    prompt = prompt_grid(byte_prompt(30, seed=43), cfg)
    ref = _run(model, prompt, 6, [6], "unfused", ignore_stop=True)
    _fused_fits(model)
    S = model.get_option("ll_mlp_cluster")
    try:
        model.set_option("n_ctas", 7 * S)
        for program in ("split", "per-CTA"):
            _same(ref, _run(model, prompt, 6, [6], program, ignore_stop=True), f"{size}: n_ctas = 7 clusters of {S}, {program}")
        assert model.get_option("n_ctas") == 7 * S
        model.set_option("n_ctas", 7 * S + 1)
        _same(ref, _run(model, prompt, 6, [6], "split", expect_fused=0, ignore_stop=True), f"{size}: n_ctas = {7 * S + 1}")
    finally:
        model.set_option("n_ctas", 0)
