"""Pins oracle/dualar_oracle.py against outputs of the UNMODIFIED reference.

tests/golden/*.npz were produced by tools/make_goldens.py, which imports
/root/reference/modeling (RQTransformer.forward, fp32 + bf16, and a literal greedy
loop through the same forward).  The reference's own tests hold no vectors for this
path (SURVEY §4), so these files are what pins the restatement.
"""
import hashlib

import numpy as np
import pytest
import torch

from conftest import bf16_bits_to_f32, load_golden
from oracle.dualar_oracle import DualAROracle, OracleSettings
from smoltts_b200.config import named_config
from smoltts_b200.synth import make_state_dict

SIZES = ["smoltts_byte_tiny", "smoltts_byte_70m", "smoltts_byte_150m"]

# The bf16 goldens are the reference's forward as torch's oneDNN bf16 kernels computed it with 8 intra-op threads.  The thread
# count decides how those GEMMs split their work, hence the fp32 summation order inside them and which bf16 roundings flip:
# on the same CPU, 7 to 9 threads reproduce the goldens bit for bit, other counts move 150m logits by up to 0.086 and the
# bf16 cases fail.  The oracle therefore runs with 8 threads whatever the host's core count.
GOLDEN_CPU_THREADS = 8


@pytest.fixture(scope="module", autouse=True)
def _golden_cpu_threads():
    prev = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_CPU_THREADS)
    yield
    torch.set_num_threads(prev)


def _digest(sd) -> str:
    h = hashlib.sha256()
    for k in sorted(sd):
        h.update(k.encode())
        h.update(sd[k].contiguous().view(torch.int16).numpy().tobytes())
    return h.hexdigest()


def _setup(size, dtype):
    g = load_golden(size)
    cfg = named_config(size)
    sd = make_state_dict(cfg, seed=int(g["seed"]), norm_jitter=0.05)
    return g, cfg, sd, DualAROracle(cfg, sd, dtype=dtype)


@pytest.mark.parametrize("size", SIZES)
def test_weights_regenerate_bit_identical(size):
    g = load_golden(size)
    cfg = named_config(size)
    sd = make_state_dict(cfg, seed=int(g["seed"]), norm_jitter=0.05)
    assert _digest(sd) == bytes(g["weights_sha256"]).decode()


@pytest.mark.parametrize("size", SIZES)
def test_fp32_teacher_forced_matches_reference(size):
    """fp32 oracle, full-sequence pass == reference forward (tolerance 2e-4: only
    summation order inside the fp32 GEMMs differs)."""
    g, cfg, sd, orc = _setup(size, torch.float32)
    grid = torch.from_numpy(g["grid"].astype(np.int64))
    t0, sub = int(g["cb_t0"]), int(g["sub"])
    n_audio = g["cb_f32_sub"].shape[1]
    with torch.no_grad():
        tok, cb = orc.teacher_forced(grid, fast_positions=list(range(t0, t0 + n_audio)))
    np.testing.assert_allclose(tok[..., ::sub].numpy(), g["tok_f32_sub"], atol=2e-4, rtol=0)
    cbs = torch.stack([cb[t] for t in range(t0, t0 + n_audio)], dim=1)
    np.testing.assert_allclose(cbs[..., ::sub].numpy(), g["cb_f32_sub"], atol=2e-4, rtol=0)
    assert (tok.argmax(-1).numpy() == g["tok_f32_argmax"]).all()


@pytest.mark.parametrize("size", SIZES)
def test_fp32_stepwise_cache_matches_full_forward(size):
    """KV-cached single-position steps (the MLX decode structure) reproduce the
    reference's full-sequence forward in fp32."""
    g, cfg, sd, orc = _setup(size, torch.float32)
    grid = torch.from_numpy(g["grid"].astype(np.int64))
    sub = int(g["sub"])
    with torch.no_grad():
        tok, _ = orc.teacher_forced(grid, stepwise_from=grid.shape[2] // 2)
    np.testing.assert_allclose(tok[..., ::sub].numpy(), g["tok_f32_sub"], atol=3e-4, rtol=0)


@pytest.mark.parametrize("size", SIZES)
def test_bf16_teacher_forced_matches_reference(size):
    """bf16 oracle, full-sequence pass.  The slow half issues the same ops on the same
    shapes as the reference's eager forward (bit-identical here); the depth half runs
    per position instead of as one [(b s), n, d] batch, so its GEMM blocking differs and a
    few percent of logits move by 1-2 bf16 ulps (measured: >= 93% bit-exact, max 0.039)."""
    g, cfg, sd, orc = _setup(size, torch.bfloat16)
    grid = torch.from_numpy(g["grid"].astype(np.int64))
    t0 = int(g["cb_t0"])
    n_audio = g["cb_bf16"].shape[1]
    with torch.no_grad():
        tok, cb = orc.teacher_forced(grid, fast_positions=list(range(t0, t0 + n_audio)))
    ref = bf16_bits_to_f32(g["tok_bf16"])
    got = tok.float().numpy()
    assert np.abs(got - ref).max() <= 2.0 ** -5
    assert (got == ref).mean() >= 0.99
    assert (got.argmax(-1) == ref.argmax(-1)).mean() >= 0.99
    cbs = torch.stack([cb[t] for t in range(t0, t0 + n_audio)], dim=1).float().numpy()
    refc = bf16_bits_to_f32(g["cb_bf16"])
    assert np.abs(cbs - refc).max() <= 2.0 ** -4
    assert (cbs == refc).mean() >= 0.9


@pytest.mark.parametrize("size", SIZES)
@pytest.mark.parametrize("tag,dtype", [("f32", torch.float32), ("bf16", torch.bfloat16)])
def test_greedy_loop_matches_literal_reference_greedy(size, tag, dtype):
    """The cached generate loop emits the ids the reference emits when driven
    greedily through RQTransformer.forward.  Decisions whose reference top-2 margin is
    below tau may flip (bf16 ties); after a flip the comparison stops (different
    history)."""
    g, cfg, sd, orc = _setup(size, dtype)
    prompt = torch.from_numpy(g["greedy_prompt"].astype(np.int64))
    ids, margins = g[f"greedy_ids_{tag}"], g[f"greedy_margin_{tag}"]
    # bf16: the literal loop runs full-sequence GEMMs, the cached loop single-position ones; two such executions of the
    # reference itself differ by up to 0.19 in a logit (tests/test_gpu_decode.py), so a decision at a margin of a few bf16
    # ulps may flip (observed: 150m frame 8 row 3 at margin 2^-5, after 75 identical decisions)
    tau = 1e-4 if tag == "f32" else 2.0 ** -4
    with torch.no_grad():
        frames = orc.generate(prompt, OracleSettings(default_temp=0.0, default_fast_temp=0.0),
                              fixed_frames=ids.shape[0])
    checked = 0
    for f, fr in enumerate(frames):
        for r in range(cfg.n_rows):
            if fr.vq[r] != ids[f, r]:
                assert margins[f, r] <= tau, f"frame {f} row {r}: {fr.vq[r]} != {ids[f, r]} at margin {margins[f, r]}"
                return
            checked += 1
    assert checked == ids.size
