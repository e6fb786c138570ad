"""Throughput of the Mimi encoder (MimiModel.encode, csrc/mimi_encoder.cu) on seeded weights and seeded audio.

Writes to --out:
  mimi_encode_bench.txt     card name and power limit (read in the same run), then per case (clips x seconds): ms per call
                            and audio-seconds per second from CUDA events over windows of >= 1 s after warm-up (median of
                            three windows, and their spread), achieved FLOP/s from the shape count below, and the CPU
                            oracle's time for one 10 s clip
  mimi_encode_profile.txt   a separate torch.profiler run: per-kernel CUDA time of one call per case

    python tools/mimi_encode_bench.py --out DIR
"""
import argparse
import math
import os
import subprocess
import sys
import time

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

CASES = [(1, 10.0), (16, 10.0), (64, 10.0), (1, 60.0)]
SR = 24_000


def encode_macs(n_samples: int, window: int = 250) -> int:
    """Multiply-adds of encoding one clip (kyutai/mimi shapes), counted from the layer shapes."""
    T, C, macs = n_samples, 64, n_samples * 64 * 7
    for r in (4, 5, 6, 8):
        macs += T * (3 * C * (C // 2) + (C // 2) * C)          # residual block
        T = -(-T // r)
        macs += T * (2 * r * C) * (2 * C)                       # strided conv
        C *= 2
    macs += T * 3 * C * 512                                     # last conv (1024 -> 512)
    D, Fd = 512, 2048
    macs += T * 8 * (4 * D * D + 2 * D * Fd)                    # transformer Linears
    macs += 8 * 2 * D * sum(min(i + 1, window) for i in range(T))   # scores and P V
    Fr = -(-T // 2)
    macs += Fr * (4 * D * D + 2 * D * 256 + 8 * 2048 * 256)     # downsample, projections, RVQ distances
    return macs


def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:   # (reported, not fatal: the numbers below still stand with the torch device name)
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--window-s", type=float, default=1.0)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("mimi_encode_bench: needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    from oracle.mimi_encode_oracle import MimiEncodeOracle
    from smoltts_b200.mimi import MimiModel
    from smoltts_b200.synth import make_mimi_state_dict, make_test_audio

    sd = make_mimi_state_dict(0, encoder=True)
    max_clips = max(b for b, _ in CASES)
    max_samples = max(int(b * s * SR) for b, s in CASES)
    m = MimiModel(max_streams=1, max_frames=8, encode_max_samples=max_samples, encode_max_clips=max_clips)
    m.load_state_dict(sd)
    lines = [f"card: {gpu_info()} | torch device: {torch.cuda.get_device_name()}",
             f"encoder workspace: {m._lib.smol_mimi_encoder_workspace_bytes(m._enc) / 2**30:.2f} GiB "
             f"(max_samples {max_samples}, max_clips {max_clips}); inputs are read once per call, no cache flushing",
             "case            ms/call   audio-s/s (median of 3 windows, min..max)   GFLOP/call   TFLOP/s   launches"]
    inputs = {}
    for b, s in CASES:
        n = int(s * SR)
        clips = [make_test_audio(1000 + i, n).cuda() for i in range(b)]
        inputs[(b, s)] = clips
        for _ in range(3):
            m.encode(clips)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        m.encode(clips)
        torch.cuda.synchronize()
        per = max(time.perf_counter() - t0, 1e-4)
        iters = max(2, int(math.ceil(args.window_s / per)))
        rates, mss = [], []
        for _ in range(3):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(iters):
                m.encode(clips)
            e1.record()
            e1.synchronize()
            ms = e0.elapsed_time(e1) / iters
            mss.append(ms)
            rates.append(b * s / (ms / 1e3))
        rates.sort()
        ms = sorted(mss)[1]
        gflop = 2 * b * encode_macs(n) / 1e9
        lines.append(f"{b:3d} x {s:4.0f} s    {ms:8.2f}   {rates[1]:10.0f} ({rates[0]:.0f} .. {rates[2]:.0f})"
                     f"{'':17s}{gflop:9.1f}   {gflop / ms:7.2f}   {m._lib.smol_mimi_encoder_launches(m._enc)}")
        print(lines[-1], flush=True)
    orc = MimiEncodeOracle(sd)
    x = make_test_audio(1000, 10 * SR)
    with torch.no_grad():
        orc.encode(x[:SR])
        t0 = time.perf_counter()
        orc.encode(x)
        cpu = time.perf_counter() - t0
    lines.append(f"CPU oracle (torch fp32, {torch.get_num_threads()} threads), 1 x 10 s: {cpu * 1e3:.0f} ms = {10 / cpu:.1f} audio-s/s")
    print(lines[-1])
    with open(os.path.join(args.out, "mimi_encode_bench.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")
    # ---- per-kernel split (a separate, profiled run) ----
    from torch.profiler import ProfilerActivity, profile

    prof_lines = []
    for key, clips in inputs.items():
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as p:
            m.encode(clips)
            torch.cuda.synchronize()
        prof_lines.append(f"==== {key[0]} x {key[1]:.0f} s ====")
        prof_lines.append(p.key_averages().table(sort_by="self_device_time_total", row_limit=15, max_name_column_width=60))
    with open(os.path.join(args.out, "mimi_encode_profile.txt"), "w") as f:
        f.write("\n".join(prof_lines) + "\n")


if __name__ == "__main__":
    main()
