#!/usr/bin/env python
"""Bring-up / tuning probe of the second-generation data-flow kernel (ll2_kernel.cu), bs=1.

  1. correctness: greedy ids of the tiny / 70m / 150m models against the barrier kernel (mode 0) and the CPU oracle
     (flips listed with the oracle's margin);
  2. time per frame (CUDA events) for a sweep of the hold-off, first- vs second-generation kernel;
  3. cycle trace of one frame (profiling build): per phase kind, cycles from phase start to: input staged | staging
     barrier | B fragments | MMAs | reduction barrier | end.

usage: python tools/ll2_probe.py [--skip-check] [--frames 256] [--holdoffs 0,200,400,600,800]
"""
from __future__ import annotations

import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import numpy as np  # noqa: E402
import torch  # noqa: E402

from smoltts_b200 import GenerationSettings, RQTransformer, generate_batch, named_config  # noqa: E402
from smoltts_b200.generate import _sampling, pack_prompts  # noqa: E402
from smoltts_b200.synth import byte_prompt, make_state_dict, prompt_grid  # noqa: E402

KINDS = ["QKV", "ATTN", "WO", "W13", "W2", "HEAD", "SAMPLE"]


def phase_kind(p, n_layer, n_flayer):
    n_slow = 5 * n_layer
    if p < n_slow:
        return "slow." + KINDS[p % 5]
    if p == n_slow:
        return "slow.HEAD"
    if p == n_slow + 1:
        return "slow.SAMPLE"
    r = (p - n_slow - 2) % (4 * n_flayer + 2)
    if r < 4 * n_flayer:
        return "fast." + ["QKV", "WO", "W13", "W2"][r % 4]
    return "fast.HEAD" if r == 4 * n_flayer else "fast.SAMPLE"


def check(size, n_frames, n_prompt):
    from oracle.dualar_oracle import DualAROracle, OracleSettings

    cfg = named_config(size)
    sd = make_state_dict(cfg, seed=0, norm_jitter=0.05)
    model = RQTransformer(cfg, max_batch=2, max_seq_len=max(256, n_prompt + n_frames + 32))
    model.load_state_dict(sd)
    prompt = prompt_grid(byte_prompt(n_prompt, seed=3), cfg)
    gs = GenerationSettings(default_temp=0.0, default_fast_temp=0.0)
    model.set_option("mode", 0)
    ref = generate_batch(model, [prompt], gs, audio_only=False, fixed_frames=n_frames)[0]
    model.set_option("mode", 2)
    got = generate_batch(model, [prompt], gs, audio_only=False, fixed_frames=n_frames)[0]
    torch.cuda.synchronize()
    print(f"[{size}] ll_ready={model.get_option('ll_ready')} "
          f"slots={model.get_option('ll_slots')} smem={model.get_option('ll_smem_bytes')}")
    orc = DualAROracle(cfg, sd, dtype=torch.bfloat16, max_seq_len=max(256, n_prompt + n_frames + 32))
    with torch.no_grad():
        frames = orc.generate(prompt, OracleSettings(default_temp=0.0, default_fast_temp=0.0), fixed_frames=n_frames)
    want = torch.tensor([f.vq for f in frames], dtype=torch.int32).t()
    same_ref = int((got == ref).sum()), got.numel()
    print(f"[{size}] ids equal to the barrier kernel: {same_ref[0]}/{same_ref[1]}")
    for name, ids in (("ll2", got), ("barrier", ref)):
        first = None
        for f in range(n_frames):
            for r in range(cfg.n_rows):
                if int(ids[r, f]) != int(want[r, f]):
                    first = (f, r, frames[f].margins[r])
                    break
            if first:
                break
        print(f"[{size}] {name} vs oracle: " + ("all ids identical" if first is None else
              f"first divergence at frame {first[0]} row {first[1]}, oracle margin {first[2]:.4f}"))
    del model
    torch.cuda.empty_cache()


def timing(args):
    cfg = named_config(args.model)
    need = args.prompt_bytes + 12 + args.frames + 8
    model = RQTransformer(cfg, max_batch=1, max_seq_len=max(need, 256))
    model.load_state_dict(make_state_dict(cfg, seed=0))
    prompts = [prompt_grid(byte_prompt(args.prompt_bytes, seed=1), cfg)]
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(1, max_positions=need, max_frames=args.frames)
    s = _sampling(model, GenerationSettings(default_temp=0.0, default_fast_temp=0.0), True, ignore_stop=True)
    model.prefill(batch, padded, lens)
    torch.cuda.synchronize()
    tokens0, len0 = batch.tokens.clone(), batch.seq_len.clone()
    host0 = list(batch.host_len)

    def run(n):
        batch.tokens.copy_(tokens0); batch.seq_len.copy_(len0); batch.step.zero_(); batch.finished.zero_()
        batch.host_len = list(host0)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        model.decode_frames(batch, s, n)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) * 1e3 / n

    for h in [int(h) for h in args.holdoffs.split(",")]:
        model.set_option("ll_holdoff", h)
        run(8)
        us = [run(args.frames) for _ in range(3)]
        codes = int(batch.out_codes.sum().item())
        print(f"holdoff={h:5d} cycles: {min(us):8.1f} us/frame (runs {', '.join(f'{u:.1f}' for u in us)}) check={codes}")
    model.set_option("ll_holdoff", args.trace_holdoff)
    for n in [int(x) for x in args.n_ctas.split(",") if x]:
        model.set_option("n_ctas", n)
        run(8)
        us = [run(args.frames) for _ in range(2)]
        print(f"n_ctas={n:4d}: {min(us):8.1f} us/frame")
    model.set_option("n_ctas", 0)
    # the fused gated MLP (clusters, DSMEM) against the unfused program
    for fused in (1, 0, 1):
        model.set_option("ll_fused_mlp", fused)
        run(8)
        us = [run(args.frames) for _ in range(2)]
        print(f"ll_fused_mlp={fused} (ran fused: {model.get_option('ll_last_fused')}, "
              f"cluster {model.get_option('ll_mlp_cluster')} x {model.get_option('ll_mlp_clusters')}, "
              f"grid {model.get_option('ll_mlp_cluster') * model.get_option('ll_mlp_clusters')}): {min(us):8.1f} us/frame")
    model.set_option("ll_fused_mlp", args.trace_fused)
    # cycle trace at the default hold-off
    model.set_option("ll_holdoff", args.trace_holdoff)
    run(8)
    prof = model.set_profile(True)
    us = run(args.frames)
    model.set_profile(False)
    fused = model.get_option("ll_last_fused") == 1

    def kind_of(p):   # fused MLP: the W13 phase runs w13 and w2; the W2 phase is not visited
        k = phase_kind(p, cfg.n_layer, cfg.n_fast_layer)
        return k + ("+W2 (fused)" if k.endswith("W13") else " (skipped)" if k.endswith("W2") else "") if fused else k
    trace = prof.cpu().numpy()[2 * 512 + 64: 2 * 512 + 64 + 2 * 512 * 8].reshape(2, 512, 8)
    print(f"profiling build, hold-off {args.trace_holdoff}: {us:.1f} us/frame")
    names = ["staged", "bar1", "bfrag", "weights", "mma", "bar2", "epilogue", "total"]
    print("cycle trace of the last frame, mean cycles per phase kind: " + " | ".join(names))
    for slot, label in ((0, "CTA 0"), (1, "CTA n/2")):
        acc, skipped = {}, {}
        for p in range(model.phase_count):
            t = trace[slot, p].astype(float)
            if t[0] == 0:   # a phase the consumer warps did not visit
                k = kind_of(p)
                skipped[k] = skipped.get(k, 0) + 1
                continue
            k = kind_of(p)
            if t[2] == 0:
                d = [0, 0, 0, 0, 0, 0, 0, t[6] - t[0]]
            else:
                t3 = t[3] if t[3] else t[2]
                t7 = t[7] if t[7] else t3
                t4 = t[4] if t[4] else t7
                t5 = t[5] if t[5] else t4
                d = [t[1] - t[0], t[2] - t[1], t3 - t[2], t7 - t3, t4 - t7, t5 - t4, t[6] - t5, t[6] - t[0]]
            a0, n0 = acc.get(k, ([0.0] * 8, 0))
            acc[k] = ([x + y for x, y in zip(a0, d)], n0 + 1)
        tot = 0.0
        for k, (v, n) in acc.items():
            print(f"  {label:8s} {k:24s} x{n:3d} " + " ".join(f"{x / n:8.0f}" for x in v))
            tot += v[7]
        for k, n in skipped.items():
            print(f"  {label:8s} {k:24s} x{n:3d} skipped")
        print(f"  {label}: {tot:.0f} cycles per frame in phases")
    # skew trace: %globaltimer of every CTA when its input is staged (0) and at the end of the phase (1)
    skew = prof.cpu().numpy()[2 * 512 + 64 + 2 * 512 * 8:].reshape(256, 512, 2).astype(float)
    n_ctas = int((skew[:, 0, 1] > 0).sum())
    if n_ctas > 1:
        P = model.phase_count
        acc, skipped = {}, {}
        prev = 0   # the last phase the CTAs ran: a skipped phase is no one's predecessor
        for p in range(1, P):
            end_prev, arr, end = skew[:n_ctas, prev, 1], skew[:n_ctas, p, 0], skew[:n_ctas, p, 1]
            k = kind_of(p)
            if (end <= 0).all():
                skipped[k] = skipped.get(k, 0) + 1
                continue
            prev = p
            if (end_prev <= 0).any() or (end <= 0).any():
                continue
            have = arr > 0
            a0 = acc.setdefault(k, [[], [], [], []])
            a0[0].append(end.max() - end_prev.max())                        # phase period: last end -> last end
            a0[1].append(end.max() - np.median(end))                        # spread of the ends
            if have.any():
                a0[2].append(np.median(arr[have]) - end_prev.max())         # last producer done -> median consumer staged
                a0[3].append(end.max() - np.median(arr[have]))              # median staged -> last end (the chain of the slowest CTA)
        print(f"skew trace of the last frame over {n_ctas} CTAs (ns): period (last end -> last end) | end spread (max - median) | "
              f"last end of the previous phase -> median input staged | median staged -> last end")
        for k, (per, sp, gap, chain) in acc.items():
            print(f"  {k:20s} x{len(per):3d} period {np.mean(per):7.0f} | spread {np.mean(sp):6.0f} | hand-off "
                  f"{(np.mean(gap) if gap else float('nan')):6.0f} | chain {(np.mean(chain) if chain else float('nan')):6.0f}")
        for k, n in skipped.items():
            print(f"  {k:20s} x{n:3d} skipped")


def teams(args):
    """Batches of 2..8 on the data-flow kernel: one team of CTAs per sequence.  Every sequence must decode exactly as it does
    alone (rows over CTAs, K over warps: the arithmetic does not depend on the team size)."""
    cfg = named_config(args.model)
    need = args.prompt_bytes + 12 + 64 + 8
    model = RQTransformer(cfg, max_batch=8, max_seq_len=max(need, 256))
    model.load_state_dict(make_state_dict(cfg, seed=0))
    model.set_option("ll_max_batch", 8)
    gs = GenerationSettings(default_temp=0.0, default_fast_temp=0.0)
    prompts = [prompt_grid(byte_prompt(args.prompt_bytes - 7 * b, seed=1 + b), cfg) for b in range(8)]
    solo = [generate_batch(model, [p], gs, audio_only=False, fixed_frames=12, seq_ids=[b])[0] for b, p in enumerate(prompts[:4])]
    for B in (2, 3, 4):
        outs = generate_batch(model, prompts[:B], gs, audio_only=False, fixed_frames=12, seq_ids=list(range(B)))
        same = [bool(torch.equal(outs[b], solo[b])) for b in range(B)]
        print(f"teams: batch of {B}: rows identical to their solo decode: {same}")
    grids = [int(x) for x in args.n_ctas.split(",") if x] or [0]
    for B, n_ctas in [(B, n) for n in grids for B in (1, 2, 3, 4, 6, 8)]:
        model.set_option("n_ctas", n_ctas)
        padded, lens = pack_prompts(model, prompts[:B])
        batch = model.new_batch(B, max_positions=need, max_frames=64)
        s = _sampling(model, gs, True, ignore_stop=True)
        model.prefill(batch, padded, lens)
        model.decode_frames(batch, s, 8)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        model.decode_frames(batch, s, 48)
        e1.record()
        torch.cuda.synchronize()
        us = e0.elapsed_time(e1) * 1e3 / 48
        print(f"teams: bs={B} grid {model.get_option('n_ctas')}: {us:8.1f} us per frame step -> {B / us * 1e6:9.0f} frames/s")
        batch.release()
    model.set_option("n_ctas", 0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="smoltts_byte_150m")
    ap.add_argument("--frames", type=int, default=256)
    ap.add_argument("--prompt-bytes", type=int, default=200)
    ap.add_argument("--holdoffs", default="0,200,400,600,800")
    ap.add_argument("--trace-holdoff", type=int, default=400)
    ap.add_argument("--trace-fused", type=int, default=1, help="ll_fused_mlp of the cycle / skew trace")
    ap.add_argument("--n-ctas", default="", help="comma list of grid sizes to time")
    ap.add_argument("--skip-check", action="store_true")
    ap.add_argument("--skip-timing", action="store_true")
    ap.add_argument("--teams", action="store_true")
    a = ap.parse_args()
    if not a.skip_check:
        check("smoltts_byte_tiny", 8, 20)
        check("smoltts_byte_70m", 6, 40)
        check("smoltts_byte_150m", 6, 40)
        check("smoltts_byte_150m", 4, 700)
    if not a.skip_timing:
        timing(a)
    if a.teams:
        teams(a)


if __name__ == "__main__":
    main()
