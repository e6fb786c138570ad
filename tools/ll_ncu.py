#!/usr/bin/env python
"""Small fixed workload for ncu captures of the decode kernel: prefill, a warm-up launch, then ONE
launch of --frames frames (the one to capture: ncu -k regex:smol_ll2_kernel --launch-skip 1 --launch-count 1)."""
from __future__ import annotations

import argparse
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from smoltts_b200 import RQTransformer, named_config  # noqa: E402
from smoltts_b200.generate import GenerationSettings, _sampling, pack_prompts  # noqa: E402
from smoltts_b200.synth import byte_prompt, make_state_dict, prompt_grid  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="smoltts_byte_150m")
    ap.add_argument("--frames", type=int, default=16)
    ap.add_argument("--prompt-bytes", type=int, default=200)
    ap.add_argument("--mode", type=int, default=2, choices=(0, 2), help="2: data-flow kernel (default), 0: barrier kernel")
    ap.add_argument("--n-ctas", type=int, default=0)
    a = ap.parse_args()
    cfg = named_config(a.model)
    need = a.prompt_bytes + 12 + 2 * a.frames + 16
    model = RQTransformer(cfg, max_batch=1, max_seq_len=max(need, 256))
    model.load_state_dict(make_state_dict(cfg, seed=0))
    model.set_option("mode", a.mode)
    if a.n_ctas:
        model.set_option("n_ctas", a.n_ctas)
    prompts = [prompt_grid(byte_prompt(a.prompt_bytes, seed=1), cfg)]
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(1, max_positions=need, max_frames=2 * a.frames + 8)
    s = _sampling(model, GenerationSettings(default_temp=0.0, default_fast_temp=0.0), True, ignore_stop=True)
    model.prefill(batch, padded, lens)          # launch 0
    tokens0, len0 = batch.tokens.clone(), batch.seq_len.clone()
    host_len0 = list(batch.host_len)
    batch.tokens.copy_(tokens0); batch.seq_len.copy_(len0); batch.step.zero_(); batch.host_len = list(host_len0)
    model.decode_frames(batch, s, a.frames)     # launch 1 (warm)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    model.decode_frames(batch, s, a.frames)     # launch 2 (captured)
    e1.record()
    torch.cuda.synchronize()
    print(f"{a.model} mode={a.mode}: {e0.elapsed_time(e1) * 1e3 / a.frames:.1f} us/frame over {a.frames} frames; "
          f"codes checksum {int(batch.out_codes.sum().item())}")


if __name__ == "__main__":
    main()
