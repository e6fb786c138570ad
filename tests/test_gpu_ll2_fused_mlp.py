"""The fused gated MLP of the data-flow kernel (ll2_kernel.cu, batch 1: w13 + w2 of a layer in one phase, act handed on
inside thread-block clusters, w2 partial sums added by the next phase) against the unfused program (option
ll_fused_mlp = 0).  Both must compute the same bits: codes, tokens, seq_len, step, every cached K/V value and the fp32
logits -- over one launch and several, across 512-position softmax blocks, with sampled ids, forced ids and the stop rule.
"""
import pytest
import torch

from gpu_util import model_and_oracle
from smoltts_b200.generate import pack_prompts
from smoltts_b200.synth import byte_prompt, prompt_grid

pytestmark = pytest.mark.gpu


def _run(model, prompt, n_frames, chunks, fused, force_at=None, expect_fused=None, **skw):
    model.set_option("ll_fused_mlp", 1 if fused else 0)
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
        want = fused if expect_fused is None else expect_fused
        assert model.get_option("ll_last_fused") == (1 if want else 0), "fused MLP: the launch ran the other program"
        return dict(codes=batch.out_codes.clone(), tokens=batch.tokens.clone(), seq_len=batch.seq_len.clone(),
                    step=batch.step.clone(), finished=batch.finished.clone(), kv=model.kv_view()[pages].clone(),
                    logits=(model.debug_buffer("token_logits", 1).clone(), model.debug_buffer("depth_logits", 1).clone()))
    finally:
        model.set_force(None)
        model.set_option("ll_fused_mlp", 1)
        batch.release()


def _same(a, b, what):
    for k in ("codes", "tokens", "seq_len", "step", "finished"):
        assert torch.equal(a[k], b[k]), f"{what}: {k} differ"
    assert torch.equal(a["kv"].view(torch.int16), b["kv"].view(torch.int16)), f"{what}: KV differs"
    assert torch.equal(a["logits"][0], b["logits"][0]) and torch.equal(a["logits"][1], b["logits"][1]), f"{what}: logits differ"


def _fused_fits(model):
    if model.get_option("ll_mlp_cluster") <= 0:
        pytest.skip("no thread-block cluster size of the fused MLP fits this GPU")


@pytest.mark.parametrize("size,n_prompt", [("smoltts_byte_tiny", 20), ("smoltts_byte_70m", 100), ("smoltts_byte_150m", 180)])
def test_fused_mlp_is_bit_identical_to_unfused(size, n_prompt):
    cfg, sd, model, orc = model_and_oracle(size, max_batch=1)
    prompt = prompt_grid(byte_prompt(n_prompt, seed=41), cfg)
    ref = _run(model, prompt, 12, [12], fused=False, ignore_stop=True)
    _fused_fits(model)
    _same(ref, _run(model, prompt, 12, [12], fused=True, ignore_stop=True), f"{size}: one launch")
    _same(ref, _run(model, prompt, 12, [5, 4, 3], fused=True, ignore_stop=True), f"{size}: three launches")


@pytest.mark.parametrize("size,n_prompt", [("smoltts_byte_tiny", 505), ("smoltts_byte_70m", 1300)])
def test_fused_mlp_long_context(size, n_prompt):
    cfg, sd, model, orc = model_and_oracle(size, max_batch=1, max_seq_len=2304)
    prompt = prompt_grid(byte_prompt(n_prompt, seed=71), cfg)
    ref = _run(model, prompt, 14, [14], fused=False, ignore_stop=True)
    _fused_fits(model)
    _same(ref, _run(model, prompt, 14, [14], fused=True, ignore_stop=True), f"{size} {n_prompt}: one launch")
    _same(ref, _run(model, prompt, 14, [1] * 14, fused=True, ignore_stop=True), f"{size} {n_prompt}: frame by frame")


@pytest.mark.parametrize("fast_temp", [0.6, 0.0])
def test_fused_mlp_sampled(fast_temp):
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=1)
    prompt = prompt_grid(byte_prompt(24, seed=9), cfg)
    kw = dict(temp=0.7, fast_temp=fast_temp, top_k=50, top_p=0.9, seed=1234, ignore_stop=True)
    ref = _run(model, prompt, 12, [12], fused=False, **kw)
    _fused_fits(model)
    _same(ref, _run(model, prompt, 12, [12], fused=True, **kw), f"sampled, fast_temp {fast_temp}")


def test_fused_mlp_forced_ids_and_stop_rule():
    cfg, sd, model, orc = model_and_oracle("smoltts_byte_tiny", max_batch=1)
    prompt = prompt_grid(byte_prompt(14, seed=82), cfg)
    ref = _run(model, prompt, 8, [1, 3, 4], fused=False, force_at=1, audio_only=True)
    assert ref["finished"].tolist() == [1]
    _fused_fits(model)
    _same(ref, _run(model, prompt, 8, [1, 3, 4], fused=True, force_at=1, audio_only=True), "forced <|im_end|>")


@pytest.mark.parametrize("size", ["smoltts_byte_tiny", "smoltts_byte_150m"])
def test_fused_mlp_under_an_n_ctas_override(size):
    """An n_ctas override that is a grid of 7 clusters keeps the fused program; one that is not runs the unfused one."""
    cfg, sd, model, orc = model_and_oracle(size, max_batch=1)
    prompt = prompt_grid(byte_prompt(30, seed=43), cfg)
    ref = _run(model, prompt, 6, [6], fused=False, ignore_stop=True)
    _fused_fits(model)
    S = model.get_option("ll_mlp_cluster")
    try:
        model.set_option("n_ctas", 7 * S)
        _same(ref, _run(model, prompt, 6, [6], fused=True, ignore_stop=True), f"{size}: n_ctas = 7 clusters of {S}")
        assert model.get_option("n_ctas") == 7 * S
        model.set_option("n_ctas", 7 * S + 1)
        _same(ref, _run(model, prompt, 6, [6], fused=True, expect_fused=False, ignore_stop=True), f"{size}: n_ctas = {7 * S + 1}")
    finally:
        model.set_option("n_ctas", 0)
