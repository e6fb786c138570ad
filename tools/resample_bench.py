"""Timing of the sample-rate converter (smoltts_b200/resample.py, csrc/resample.cu) on seeded audio.

Writes resample_bench.txt to --out: the card name and power limit (read in the same run), then
  * one streaming step (one 80 ms frame of 1920 samples per stream at 24 kHz) at 1, 8 and 64 streams, 24 kHz -> 48 kHz and
    -> 44.1 kHz: the kernel's device time (torch.profiler, mean over the timed steps) and the host time of a
    ``Resampler.step`` call (wall clock over the steps, ending in a device synchronise);
  * one whole-clip call on 64 clips x 10 s of 48 kHz audio -> 24 kHz: CUDA events around the call (median of windows) and the
    kernel's device time;
  * ``SmolTTS.stream`` (smoltts_byte_150m with seeded weights, greedy, Mimi decoder) in us per frame with output_rate
    48 000 against 24 000, the two alternated in the same process.

    python tools/resample_bench.py --out DIR
"""
import argparse
import os
import statistics
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:   # (reported, not fatal: the numbers below still stand with the torch device name)
        return f"nvidia-smi unavailable: {e}"


def kernel_us(fn, n: int) -> float:
    """Mean device time of resample_kernel over n calls of fn, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(n):
            fn()
        torch.cuda.synchronize()
    ev = [e for e in prof.key_averages() if "resample_kernel" in e.key]
    assert ev and ev[0].count == n, [(e.key, e.count) for e in prof.key_averages()]
    total = getattr(ev[0], "device_time_total", None)
    if total is None:
        total = ev[0].cuda_time_total
    return total / n


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--stream-reps", type=int, default=4)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("resample_bench: needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    from smoltts_b200.resample import Resampler
    from smoltts_b200.synth import make_test_audio

    lines = [f"# GPU: {gpu_info()} (torch: {torch.cuda.get_device_name(0)})"]

    def say(s):
        print(s, flush=True)
        lines.append(s)

    say("# one streaming step: 1920 samples (80 ms at 24 kHz) per stream")
    say(f"{'rates':<22}{'streams':>8}{'kernel us':>12}{'host us per step()':>20}")
    for rate in (48_000, 44_100):
        for n in (1, 8, 64):
            rs = Resampler(24_000, rate, max_streams=n)
            states = [rs.make_state() for _ in range(n)]
            frames = [make_test_audio(i, 1920).cuda() for i in range(n)]
            for _ in range(50):
                rs.step(frames, states)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                rs.step(frames, states)
            torch.cuda.synchronize()
            host = (time.perf_counter() - t0) / args.steps * 1e6
            dev = kernel_us(lambda: rs.step(frames, states), 200)
            say(f"{'24000 -> ' + str(rate):<22}{n:>8}{dev:>12.2f}{host:>20.1f}")

    say("# whole clips: 64 x 10 s of 48 kHz audio -> 24 kHz, one call")
    rs = Resampler(48_000, 24_000, max_streams=64)
    clips = [make_test_audio(100 + i, 480_000, 48_000).cuda() for i in range(64)]
    for _ in range(5):
        rs.resample(clips)
    windows = []
    for _ in range(5):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(20):
            rs.resample(clips)
        b.record()
        torch.cuda.synchronize()
        windows.append(a.elapsed_time(b) / 20)
    dev = kernel_us(lambda: rs.resample(clips), 20)
    audio_s = 64 * 10.0
    say(f"call (events, median of 5 windows of 20 calls): {statistics.median(windows):.3f} ms (spread {min(windows):.3f} .. "
        f"{max(windows):.3f}); kernel {dev / 1e3:.3f} ms; {audio_s / (statistics.median(windows) * 1e-3):.0f} audio-s/s; "
        f"{64 * 480_000 * 4 * 1.5 / (dev * 1e-6) / 1e9:.0f} GB/s of input + output")

    from smoltts_b200 import GenerationSettings, MimiModel, PromptEncoder, RQTransformer, SmolTTS, byte_level_tokenizer, named_config
    from smoltts_b200.synth import make_mimi_state_dict, make_state_dict

    frames = 128
    cfg = named_config("smoltts_byte_150m")
    lm = RQTransformer(cfg, max_batch=1, max_seq_len=512 + frames)
    lm.load_state_dict(make_state_dict(cfg, seed=0))
    codec = MimiModel(max_streams=1, max_frames=frames + 8)
    codec.load_state_dict(make_mimi_state_dict(0))
    enc = PromptEncoder.from_model(byte_level_tokenizer(cfg.codebook_size), lm)
    gs = GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=frames - 1)
    ttss = {24_000: SmolTTS(lm, enc, codec, settings=gs), 48_000: SmolTTS(lm, enc, codec, settings=gs, output_rate=48_000)}
    text = "The quick brown fox jumps over the lazy dog. " * 4
    say(f"# SmolTTS.stream, smoltts_byte_150m greedy + Mimi decoder, one utterance of up to {frames} frames, overlap mode; "
        f"output_rate 24 000 and 48 000 alternated, {args.stream_reps} runs each")
    per = {r: [] for r in ttss}
    for rep in range(args.stream_reps + 2):
        for rate, tts in ttss.items():
            st = {}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = sum(c.size for c in tts.stream(text, "nova", stats=st))
            torch.cuda.synchronize()
            us = (time.perf_counter() - t0) * 1e6 / st["frames"]
            if rep >= 2:   # the first two rounds are warm-up
                per[rate].append(us)
            print(rate, st, n, f"{us:.1f}", flush=True)
    for rate, v in per.items():
        say(f"output_rate {rate:>6}: {statistics.median(v):8.1f} us per frame (median; runs {', '.join(f'{x:.1f}' for x in v)})")
    with open(os.path.join(args.out, "resample_bench.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
