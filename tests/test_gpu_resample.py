"""The sample-rate converter on the GPU (csrc/resample.cu through include/smoltts_b200_resample.h): against the float64
oracle on every golden pair and length, streaming and batch / slot invariance bit for bit, and SmolTTS with reference
audio at 48 kHz stereo and with an output_rate.

Bar against the oracle: 1e-5 x max |reference| (fp32 FMA chains of 21 .. 61 terms against float64)."""
import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR

pytestmark = pytest.mark.gpu

REL = 1e-5


def _pairs(g):
    return [tuple(int(v) for v in p) for p in g["pairs"]]


def test_every_golden_pair_matches_the_oracle():
    from oracle.resample_oracle import make_test_input, resample
    from smoltts_b200.resample import Resampler, design_filter

    g = np.load(f"{GOLDEN_DIR}/resample.npz")
    lengths = [int(v) for v in g["lengths"]]
    worst = 0.0
    for r_in, r_out in _pairs(g):
        rs = Resampler(r_in, r_out, max_streams=len(lengths))
        h = design_filter(r_in, r_out)
        xs = [make_test_input(int(g[f"{r_in}_{r_out}_{n}_seed"]), n, r_in) for n in lengths]
        got = [y.cpu().numpy() for y in rs.resample([torch.from_numpy(x) for x in xs])]
        for n, x, y in zip(lengths, xs, got):
            want = resample(x, rs.up, rs.down, h)
            assert y.shape == want.shape == (-(-n * rs.up // rs.down),)
            err = np.abs(y - want).max() / np.abs(want).max()
            worst = max(worst, err)
            assert err <= REL, (r_in, r_out, n, err)
    print(f"largest |gpu - oracle| / max |oracle| over the golden pairs and lengths: {worst:.3g}")


@pytest.mark.parametrize("r_in,r_out", [(24_000, 48_000), (24_000, 44_100), (24_000, 8_000), (48_000, 24_000), (11_025, 24_000),
                                        (24_000, 11_025)])
def test_streams_equal_whole_clips_bit_for_bit(r_in, r_out):
    """Five streams in five of eight slots, fed random ragged chunks (empty ones too) in interleaved calls, equal the whole-clip
    results; and whole clips are the same bits alone, in a batch, reversed, in other slots and on another handle."""
    from oracle.resample_oracle import make_test_input
    from smoltts_b200.resample import Resampler, output_count

    rng = np.random.default_rng(r_in + r_out)
    lens = [1, 1921, 30_011, 7, 48_000]
    xs = [torch.from_numpy(make_test_input(300 + i, n, r_in)).cuda() for i, n in enumerate(lens)]
    rs = Resampler(r_in, r_out, max_streams=8)
    whole = [y.clone() for y in rs.resample(xs)]
    alone = [rs.resample([x])[0].clone() for x in xs]
    rev = [y.clone() for y in rs.resample(xs[::-1])][::-1]
    other = Resampler(r_in, r_out, max_streams=16)
    _ = [other.make_state() for _ in range(9)]                     # the clips land in other slots
    moved = other.resample(xs)
    for i in range(len(xs)):
        for name, y in (("alone", alone[i]), ("reversed", rev[i]), ("other slots", moved[i])):
            assert torch.equal(y, whole[i]), f"clip {i}: {name} differs from the batch"
    _ = [rs.make_state() for _ in range(2)]                        # streams in slots 2 .. 6, not 0 .. 4
    states = [rs.make_state() for _ in xs]
    pos = [0] * len(xs)
    got = [[] for _ in xs]
    while any(p < len(x) for p, x in zip(pos, xs)):
        pick = [i for i in range(len(xs)) if rng.random() < 0.7] or [0]
        chunks = []
        for i in pick:
            n = min(int(rng.integers(0, 4000)), len(xs[i]) - pos[i])
            chunks.append(xs[i][pos[i]: pos[i] + n])
            pos[i] += n
        for i, c, y in zip(pick, chunks, rs.step(chunks, [states[i] for i in pick])):
            assert y.numel() == output_count(states[i].consumed, rs.up, rs.down, False) - sum(t.numel() for t in got[i])
            got[i].append(y.clone())
    for i, y in enumerate(rs.finish(states)):
        got[i].append(y.clone())
    for i, st in enumerate(states):
        assert st.consumed == st.emitted == 0
        assert torch.equal(torch.cat(got[i]), whole[i]), f"stream {i}: chunked output differs from the whole clip"
        rs.release_state(st)


def test_release_mid_stream_leaves_a_clean_slot():
    from oracle.resample_oracle import make_test_input
    from smoltts_b200.resample import Resampler

    rs = Resampler(24_000, 16_000, max_streams=1)
    x = torch.from_numpy(make_test_input(5, 5000, 24_000)).cuda()
    want = rs.resample([x])[0].clone()
    st = rs.make_state()
    rs.step([x[:3000]], [st])
    rs.release_state(st)
    assert rs.free_slots == 1
    assert torch.equal(rs.resample([x])[0], want)


def _sd():
    from smoltts_b200.synth import make_mimi_state_dict

    return make_mimi_state_dict(0, encoder=True)


def _tts(output_rate, lm_and_cfg=None, codecs=None):
    from gpu_util import model_and_oracle
    from smoltts_b200 import GenerationSettings, MimiModel, PromptEncoder, SmolTTS, byte_level_tokenizer

    cfg, sd, lm, _ = lm_and_cfg or model_and_oracle("smoltts_byte_tiny", max_batch=8, max_seq_len=256)
    enc = PromptEncoder.from_model(byte_level_tokenizer(cfg.codebook_size), lm)
    if codecs is None:
        msd = _sd()
        stream = MimiModel(max_streams=4, max_frames=32)
        stream.load_state_dict(msd)
        full = MimiModel(max_streams=4, max_frames=32, upsample_carry=True)
        full.load_state_dict(msd)
        codecs = (stream, full)
    gs = GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=9)
    return SmolTTS(lm, enc, codecs[0], codecs[1], gs, output_rate=output_rate), (cfg, sd, lm, None), codecs


def test_create_speaker_from_48k_stereo():
    from gpu_util import model_and_oracle
    from smoltts_b200 import MimiModel, PromptEncoder, SmolTTS, byte_level_tokenizer
    from smoltts_b200.resample import Resampler
    from smoltts_b200.synth import make_test_audio

    cfg, _, lm, _ = model_and_oracle("smoltts_byte_tiny", max_batch=8, max_seq_len=1024)
    enc = PromptEncoder.from_model(byte_level_tokenizer(cfg.codebook_size), lm)
    codec = MimiModel(max_streams=2, max_frames=32, upsample_carry=True, encode_max_samples=200_000, encode_max_clips=3)
    codec.load_state_dict(_sd())
    tts = SmolTTS(lm, enc, codec)
    stereo = torch.stack([make_test_audio(21, 96_007, 48_000), make_test_audio(22, 96_007, 48_000)])
    mono24 = make_test_audio(23, 30_000)
    prefix = tts.create_speaker([{"text": "stereo at 48 kHz", "audio": stereo, "sampling_rate": 48_000},
                                 {"text": "mono at 24 kHz", "audio": mono24},
                                 {"text": "mono at 48 kHz", "audio": stereo[0], "sampling_rate": 48_000}])
    ref = Resampler(48_000, 24_000, max_streams=2)
    a, b = ref.resample([stereo.cuda().mean(dim=0), stereo[0].cuda()])
    assert a.shape == (48_004,)
    codes = codec.encode([a, mono24.cuda(), b])
    want = enc.create_speaker([{"text": "stereo at 48 kHz", "codes": codes[0].cpu()}, {"text": "mono at 24 kHz", "codes": codes[1].cpu()},
                               {"text": "mono at 48 kHz", "codes": codes[2].cpu()}])
    assert torch.equal(prefix, want)
    assert torch.equal(tts.create_speaker([{"text": "x", "audio": mono24, "sampling_rate": 24_000}]),
                       tts.create_speaker([{"text": "x", "audio": mono24}])), "24 kHz with a sampling_rate must not be resampled"


def test_output_rate_none_builds_no_resampler():
    tts, _, _ = _tts(None)
    assert tts.resampler is None and tts.sampling_rate == 24_000
    tts2, _, _ = _tts(24_000)
    assert tts2.resampler is None and tts2.sampling_rate == 24_000


@pytest.mark.parametrize("rate", [48_000, 16_000])
def test_output_rate_on_every_entry_point(rate):
    from smoltts_b200.resample import Resampler, output_count

    base, lmc, codecs = _tts(None)
    tts, _, _ = _tts(rate, lmc, codecs)
    assert tts.sampling_rate == rate and tts.resampler is not None
    ref = Resampler(24_000, rate, max_streams=8)

    def resampled(pcm24):
        return ref.resample([torch.from_numpy(np.ascontiguousarray(pcm24)).cuda()])[0].cpu().numpy()

    text, voice = "Hello there, B200.", "nova"
    pcm24 = base(text, voice)
    assert pcm24.size > 0
    pcm = tts(text, voice)
    assert np.array_equal(pcm, resampled(pcm24)), "__call__ differs from the whole-clip resample of the 24 kHz utterance"

    chunks24 = list(base.stream(text, voice))
    want = resampled(np.concatenate(chunks24))
    for overlap in (True, False):
        chunks = list(tts.stream(text, voice, overlap=overlap))
        assert len(chunks) == len(chunks24) + 1, "one chunk per frame plus the filter's tail"
        S = E = 0
        for t, c in enumerate(chunks):
            finish = t == len(chunks24)
            S += 0 if finish else chunks24[t].size
            assert c.size == output_count(S, ref.up, ref.down, finish) - E, (overlap, t)
            E += c.size
        assert np.array_equal(np.concatenate(chunks), want), f"stream(overlap={overlap}) differs from the whole-clip resample"

    texts = ["One.", "A second, longer utterance.", "Three!"]
    voices = ["heart", "sky", "liam"]
    outs = tts.synthesize_batch(texts, voices, fixed_frames=6)
    for o, o24 in zip(outs, base.synthesize_batch(texts, voices, fixed_frames=6)):
        assert np.array_equal(o, resampled(o24))

    texts = [f"Streamed utterance {i} {'!' * i}" for i in range(5)]
    voices = ["heart", "nova", "sky", "liam", "emma"]
    served = dict(tts.serve(texts, voices, slots=3, chunk=4, max_prompt=128))
    parts = {i: [] for i in range(5)}
    for i, c, done in tts.serve_stream(texts, voices, slots=3, chunk=4, max_prompt=128):
        parts[i].append(c)
    for i in range(5):
        assert served[i].size > 0
        assert np.array_equal(np.concatenate(parts[i]), served[i]), f"utterance {i}: serve_stream chunks differ from serve"
    for c in codecs:
        assert len(c._free) == c.max_streams, "codec slots must all be given back"
    assert tts.resampler.free_slots == tts.resampler.max_streams, "resampler slots must all be given back"
    cache = codecs[1].make_cache()
    with pytest.raises(ValueError, match="24 kHz"):
        tts.decode_codes([torch.zeros(8, 1, dtype=torch.int64)], [cache])
    codecs[1].release_cache(cache)


def test_handles_of_other_ratios_do_not_break_each_other():
    """The kernel's shared-memory limit is one per function: binding a handle whose launches need little must not refuse the
    launches of a handle bound earlier that needs more (11.025 -> 24 kHz stages 27 KB, 24 -> 48 kHz under 1 KB)."""
    from oracle.resample_oracle import make_test_input
    from smoltts_b200.resample import Resampler

    x11 = torch.from_numpy(make_test_input(41, 20_000, 11_025)).cuda()
    x24 = torch.from_numpy(make_test_input(42, 20_000, 24_000)).cuda()
    big = Resampler(11_025, 24_000)
    want_big = big.resample([x11])[0].clone()
    small = Resampler(24_000, 48_000)
    want_small = small.resample([x24])[0].clone()
    assert torch.equal(big.resample([x11])[0], want_big), "the larger handle after a smaller one was bound"
    mid = Resampler(44_100, 24_000)
    mid.resample([x24])
    assert torch.equal(small.resample([x24])[0], want_small) and torch.equal(big.resample([x11])[0], want_big)


def test_more_streams_than_one_launch_takes():
    from smoltts_b200 import _capi
    from smoltts_b200.synth import make_test_audio
    from smoltts_b200.resample import Resampler

    n = _capi.SMOL_RESAMPLE_MAX_CALL + 44
    rs = Resampler(24_000, 16_000, max_streams=n)
    xs = [make_test_audio(500 + i, 100 + 7 * i).cuda() for i in range(n)]
    whole = [y.clone() for y in rs.resample(xs)]
    assert all(torch.equal(whole[i], rs.resample([xs[i]])[0]) for i in (0, 255, 256, n - 1))
    states = [rs.make_state() for _ in range(n)]
    parts = [[y.clone()] for y in rs.step([x[:50] for x in xs], states)]
    for p, y in zip(parts, rs.step([x[50:] for x in xs], states)):
        p.append(y.clone())
    for p, y in zip(parts, rs.finish(states)):
        p.append(y.clone())
    for i in range(n):
        assert torch.equal(torch.cat(parts[i]), whole[i]), f"stream {i}"
        rs.release_state(states[i])
    assert rs.free_slots == n


def test_output_rate_survives_create_speaker_at_another_rate():
    """SmolTTS at 44.1 kHz out, then a voice-clone reference at 48 kHz (a second resampler, 48 -> 24 kHz, bound after the
    first): synthesis still runs and gives the same audio as before."""
    from gpu_util import model_and_oracle
    from smoltts_b200 import GenerationSettings, MimiModel, PromptEncoder, SmolTTS, byte_level_tokenizer
    from smoltts_b200.synth import make_test_audio

    cfg, _, lm, _ = model_and_oracle("smoltts_byte_tiny", max_batch=8, max_seq_len=1024)
    enc = PromptEncoder.from_model(byte_level_tokenizer(cfg.codebook_size), lm)
    codec = MimiModel(max_streams=2, max_frames=32, upsample_carry=True, encode_max_samples=100_000, encode_max_clips=2)
    codec.load_state_dict(_sd())
    tts = SmolTTS(lm, enc, codec, settings=GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=9),
                  output_rate=44_100)
    before = tts("Hello there, B200.", "nova")
    assert before.size > 0
    stereo = torch.stack([make_test_audio(31, 96_000, 48_000), make_test_audio(32, 96_000, 48_000)])
    tts.create_speaker([{"text": "stereo at 48 kHz", "audio": stereo, "sampling_rate": 48_000}])
    assert np.array_equal(tts("Hello there, B200.", "nova"), before)
    assert sum(c.size for c in tts.stream("Hello there, B200.", "nova")) > 0
    with pytest.raises(ValueError, match="channels first"):
        tts.create_speaker([{"text": "soundfile layout", "audio": stereo.t(), "sampling_rate": 48_000}])
