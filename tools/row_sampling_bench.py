#!/usr/bin/env python
"""Cost of per-sequence sampling settings (SmolBatch.row_sampling) on the decode kernels: the same decode steps with no
table (every row samples with the call's SmolSampling), a uniform table (every row carries the call's settings: the same
work, read from the table) and a mixed table (rows alternate between greedy and three sampled settings, each with its own
seed: different sampling work per row).  Arms alternate inside every round, so drift of the card hits all three alike.

Workloads (smoltts_byte_150m, seeded weights, 200-byte prompts as bench.py):
  bs1   1 utterance, greedy, 1024 frames per step   (bench.py config 2: the data-flow kernel, fused MLP)
  bs8   8 utterances, greedy, 256 frames per step   (data-flow kernel, 8 teams of CTAs)
  bs64  64 utterances, sampled temp 0.7 / top-k 50 / top-p 0.9, 256 frames per step   (bench.py config 3: tcgen05 variant)
At bs=1 a "mixed" table is one row; it is left out.

Every window is timed with CUDA events around whole decode steps (state reset between steps, as bench.py's device-resident
arm) and lasts >= --window-s seconds after warm-up.  Writes --out/row_sampling_bench.txt: the card name and power limit read
in the same run, then per workload and arm the median and the range of us per frame step over --rounds windows.

    python tools/row_sampling_bench.py --out DIR
"""
from __future__ import annotations

import argparse
import math
import os
import subprocess
import sys
from dataclasses import replace

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

WORKLOADS = [("bs1", 1, 1024, False), ("bs8", 8, 256, False), ("bs64", 64, 256, True)]
PROMPT_BYTES = 200


def gpu_info() -> str:
    try:
        return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                              capture_output=True, text=True, timeout=60).stdout.strip()
    except Exception as e:   # (reported, not fatal: the numbers below still stand with the torch device name)
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--model", default="smoltts_byte_150m")
    ap.add_argument("--window-s", type=float, default=1.0)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("row_sampling_bench: needs a CUDA device")
    os.makedirs(args.out, exist_ok=True)
    from smoltts_b200 import GenerationSettings, RQTransformer, named_config
    from smoltts_b200.generate import _sampling, pack_prompts
    from smoltts_b200.synth import byte_prompt, make_state_dict, prompt_grid

    cfg = named_config(args.model)
    n_prompt = PROMPT_BYTES + 12
    max_frames = max(f for _, _, f, _ in WORKLOADS)
    max_batch = max(b for _, b, _, _ in WORKLOADS)
    need = n_prompt + max_frames + 8
    model = RQTransformer(cfg, max_batch=max_batch, max_seq_len=need, kv_pages=2 * max_batch * ((need + 31) // 32))
    model.load_state_dict(make_state_dict(cfg, seed=0))
    greedy = GenerationSettings(default_temp=0.0, default_fast_temp=0.0)
    sampled = GenerationSettings(default_temp=0.7, default_fast_temp=0.7, top_k=50, top_p=0.9, seed=1234)
    mix = [greedy, sampled, replace(sampled, top_k=0, top_p=1.0, default_temp=1.0, min_p=0.1, min_p_intended=True),
           replace(sampled, default_temp=0.0)]

    lines = [f"card: {gpu_info()} | torch device: {torch.cuda.get_device_name()}",
             f"{args.model}, {PROMPT_BYTES}-byte prompts ({n_prompt} tokens); CUDA events over whole decode steps, windows >= "
             f"{args.window_s:.1f} s after warm-up, arms alternating in each of {args.rounds} rounds",
             "workload  arm       us per frame step: median (min .. max)   spread of the median vs no table"]
    print(lines[0], flush=True)
    for key, B, frames, is_sampled in WORKLOADS:
        gs = sampled if is_sampled else greedy
        prompts = [prompt_grid(byte_prompt(PROMPT_BYTES, seed=1 + b), cfg) for b in range(B)]
        padded, lens = pack_prompts(model, prompts)
        batch = model.new_batch(B, max_positions=n_prompt + frames + 1, max_frames=frames, seq_ids=list(range(B)))
        call = _sampling(model, gs, audio_only=True, ignore_stop=True)
        model.prefill(batch, padded, lens)
        torch.cuda.synchronize()
        tokens0, len0, host0 = batch.tokens.clone(), batch.seq_len.clone(), list(batch.host_len)
        arms = {"none": None, "uniform": model.row_sampling([gs] * B)}
        if B > 1:
            arms["mixed"] = model.row_sampling([replace(mix[b % len(mix)], seed=1234 + b) for b in range(B)])

        def step(table):
            batch.tokens.copy_(tokens0)
            batch.seq_len.copy_(len0)
            batch.step.zero_()
            batch.finished.zero_()
            batch.host_len = list(host0)
            batch.set_row_sampling(table)
            model.decode_frames(batch, call, frames)

        iters = 1
        for table in arms.values():   # warm-up of every arm; the slowest sets the window length
            for _ in range(2):
                step(table)
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            step(table)
            e1.record()
            e1.synchronize()
            iters = max(iters, int(math.ceil(args.window_s * 1e3 / e0.elapsed_time(e1))))
        us = {name: [] for name in arms}
        for _ in range(args.rounds):
            for name, table in arms.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(iters):
                    step(table)
                e1.record()
                e1.synchronize()
                us[name].append(e0.elapsed_time(e1) * 1e3 / (iters * frames))
        batch.release()
        base = sorted(us["none"])[len(us["none"]) // 2]
        for name, v in us.items():
            v = sorted(v)
            med = v[len(v) // 2]
            lines.append(f"{key:8s}  {name:8s}  {med:9.1f} ({v[0]:.1f} .. {v[-1]:.1f})   {100.0 * (med / base - 1.0):+6.2f} %   "
                         f"[{iters} steps of {frames} frames per window]")
            print(lines[-1], flush=True)
    with open(os.path.join(args.out, "row_sampling_bench.txt"), "w") as f:
        f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
