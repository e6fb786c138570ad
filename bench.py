#!/usr/bin/env python
"""Benchmark of the DualAR decode step: Mimi frames/s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path
    python bench.py --impl reference [...]                          # the reference's CPU arithmetic (oracle port)
    torchrun --nproc-per-node N ... bench.py --gpus N ...           # one rank per GPU, utterance-sharded
    python bench.py --dump-outputs DIR [...]                        # + the outputs of every entry's last timed step as .npy

Outputs written by ``--dump-outputs`` (float32; ``_rank<r>`` appended to each name under N > 1 ranks): ``headline_codes``
and ``<key>_codes`` of the decode entries, the ids the last timed step left in the batch, [utterances, rows, frames];
``mimi_bs*_pcm``, every frame of the last timed end-to-end step, [streams, frames, samples]; ``tts_stream_bs1_pcm``, the
chunks of the last timed stream, concatenated.  The inputs are seeded, so two builds run with the same arguments can be
compared file by file.

A *step* is one pass of the hot path over one batch of synthetic input: ``frames`` Mimi frames decoded for
``batch`` utterances per GPU, starting from a prefilled synthetic prompt.  The headline (top-level keys) is
BASELINE.json configs[1]: smoltts_byte_150m greedy bs=1, 1024 frames -- ``value`` is whole-job frames/s with
everything resident in HBM (CUDA events around the step launches, max over ranks), ``e2e`` the same metric through
the public ``generate_batch`` API from pinned host prompts (H2D of the prompt grid, prefill, decode, D2H of the
codes, and for N > 1 the host-side gather of every rank's codes on rank 0), for the same number of steps.

The same line carries ``"configs"``: the other BASELINE.json configurations measured the same way in the same run
(configs[2] bs=64 sampled, configs[3] bs=256 per GPU at two prompt lengths, configs[4] long-form bs=32 at the
workload's mean context), each with its own ``roofline`` and ``e2e``, and two entries for the step AFTER the path
(SURVEY 8(f)-2, the Mimi streaming decoder: ``mimi_bs1``, ``mimi_bs64`` -- codes to PCM, frames/s) and one for the
reference's streaming loop through both engines (``tts_stream_bs1``: text to PCM chunks, one frame per host iteration).  Under ``--gpus N > 1`` every entry is the
per-GPU batch sharded over the N ranks (weak scaling), so the bs=256/GPU 1 -> 8 curve is in the driver's records.

Roofline: algorithmic bytes (SURVEY 8(d): unique weight bytes + KV bytes of the mean context) or flops per launch over
the CUDA-event duration of the launch, against MEASURED_PEAKS.json; the binding roof (HBM / bf16 tensor) is named.
``cpu_baseline``: the oracle port of the reference arithmetic timed on the host cores on a bounded sample taken AT THE
WORKLOAD'S MEAN CONTEXT (so that ``--impl reference`` measures the same configuration as the GPU arm).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time
from dataclasses import dataclass

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent
CPU_SAMPLE_FRAMES = 128    # frames of one CPU-arm step (a bounded sample of the workload, centred on its mean context)
DUMP_BYTES = 64 << 20      # --dump-outputs: all files together


@dataclass
class Work:
    """One workload: `frames` frames for `batch` utterances per GPU after a prompt of 12 + prompt_bytes tokens followed by
    `history` synthetic audio columns (long-form configurations are sampled at their mean context: the history stands for
    the frames already decoded)."""
    key: str
    model: str
    batch: int
    frames: int
    prompt_bytes: int
    sampled: bool = False
    history: int = 0
    note: str = ""

    @property
    def prompt_tokens(self) -> int:
        return self.prompt_bytes + 12 + self.history

    @property
    def mean_context(self) -> float:
        return self.prompt_tokens + (self.frames - 1) / 2.0

    def name(self) -> str:
        samp = "top-k50/top-p0.9/temp0.7 sampled" if self.sampled else "greedy"
        hist = f" + {self.history} cached audio frames" if self.history else ""
        return (f"{self.model} {samp} decode bs={self.batch}/GPU, {self.frames} frames/step, "
                f"{self.prompt_bytes}-byte synthetic prompt ({self.prompt_bytes + 12} tokens){hist}")


def headline_work(args) -> Work:
    return Work("config2" if (args.batch, args.frames, args.sampled) == (1, 1024, False) else "custom", args.model, args.batch,
                args.frames, args.prompt_bytes, args.sampled, args.history)


def extra_works(model: str):
    """BASELINE.json configs[2..4] (SURVEY 8(d)), each short enough for the default run."""
    return [
        Work("config3", model, 64, 256, 200, sampled=True, note="configs[2]: bs=64 sampled, 256 frames"),
        Work("config4i", model, 256, 128, 64, note="configs[3] (i): bs=256 per GPU, 64-byte prompts, 128 frames (tensor-bound regime)"),
        Work("config4ii", model, 256, 128, 200, note="configs[3] (ii): bs=256 per GPU, 200-byte prompts, 128 frames (KV-bound)"),
        Work("config5", model, 32, 256, 200, history=1920,
             note="configs[4]: long-form bs=32 per GPU, 4096-frame decode sampled at its mean context "
                  "(256 frames after 1920 cached frames: contexts 2132..2387, mean 2259.5 = 212 + 4095/2)"),
    ]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="smoltts_byte_150m")
    ap.add_argument("--batch", type=int, default=1, help="utterances per GPU (headline)")
    ap.add_argument("--frames", type=int, default=1024, help="Mimi frames per step (headline)")
    ap.add_argument("--prompt-bytes", type=int, default=200)
    ap.add_argument("--history", type=int, default=0, help="synthetic audio columns cached behind the prompt")
    ap.add_argument("--sampled", action="store_true", help="temp 0.7 / top-k 50 / top-p 0.9, fast temp 0.7")
    ap.add_argument("--mode", type=int, default=2, help="2 data-flow persistent kernel (default), 0 grid-barrier persistent "
                    "kernel, 1 per-phase launches in a CUDA graph")
    ap.add_argument("--configs", default="auto", help="'auto': configs[2..4] next to the headline when the headline is configs[1]; "
                    "'none'; or a comma list of config3,config4i,config4ii,config5")
    ap.add_argument("--config-steps", type=int, default=5, help="timed steps of each entry of \"configs\" (3 warm-up steps)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--stream-lm-ctas", type=int, default=96, help="tts_stream_bs1: CTAs of the decode kernel while the codec runs beside it")
    ap.add_argument("--no-stream-overlap", action="store_true", help="tts_stream_bs1: codec step after the decode step instead of beside the next one")
    ap.add_argument("--cpu-frames", type=int, default=0, help="frames of the CPU sample (0 = %d)" % CPU_SAMPLE_FRAMES)
    ap.add_argument("--opt", action="append", default=[], help="engine option name=value (smol_set_option), repeatable")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what each entry's last timed step computed as DIR/<name>.npy (float32, "
                         "%d MB at most in all), to compare two builds output for output" % (DUMP_BYTES >> 20))
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the CUDA path (--impl ours)")
    return args


def dump_outputs(out_dir: str, arrays: dict, budget: int) -> None:
    """Writes each array as out_dir/<name>.npy in float32 (the codes are small integers: exact).  When the arrays exceed
    `budget` bytes together, each keeps the same share of its elements: a fixed sample (flat indices drawn with seed 0, in
    increasing order) stored 1-D, so that two runs with the same arguments write the same elements."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    total = sum(a.size * 4 for a in arrays.values())
    keep = min(1.0, (budget - 1024 * len(arrays)) / total) if total else 1.0   # 1 KB per file for the .npy header
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if keep < 1.0:
            idx = np.random.default_rng(0).choice(a.size, int(a.size * keep), replace=False)
            a = a.reshape(-1)[np.sort(idx)]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def load_tensor_peak():
    """Dense bf16 TFLOP/s: the sustained cuBLAS figure of MEASURED_PEAKS.json (the kernel is timed inside a long step)."""
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            d = json.load(f)
        if "bf16_tflops_sustained" in d:
            return float(d["bf16_tflops_sustained"]), "measured sustained (MEASURED_PEAKS.json)"
    return 2250.0, "nominal dense bf16 (B200_PROFILING.md fallback)"


def load_traffic():
    """Measured DRAM bytes per frame (ncu dram__bytes_read.sum + dram__bytes_write.sum of the decode kernel, captured on
    the bench's own workloads; profiles/traffic.json names the capture each figure comes from)."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(path):
        try:
            with open(path) as f:
                return json.load(f)
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(self.gpu)],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, power = [], [], set(), []
        try:
            with open(self.path) as f:
                for line in f:
                    p = [x.strip() for x in line.split(",")]
                    if len(p) < 9:
                        continue
                    try:
                        sm.append(float(p[1])); mx.append(float(p[2])); power.append(float(p[3]))
                    except ValueError:
                        continue
                    for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[5:9]):
                        if v.lower().startswith("active"):
                            reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def synth_prompts(cfg, work: Work, first_seq: int):
    """Utterance b: byte prompt of seed 1 + global id, then `history` synthetic audio columns (row 0 = 320 + first code)."""
    import torch

    from smoltts_b200.synth import TOK_SEMANTIC0, byte_prompt, prompt_grid

    out = []
    for b in range(work.batch):
        g = prompt_grid(byte_prompt(work.prompt_bytes, seed=1 + first_seq + b), cfg)
        if work.history:
            gen = torch.Generator().manual_seed(10_000 + first_seq + b)
            codes = torch.randint(0, cfg.codebook_size, (cfg.n_rows - 1, work.history), generator=gen)
            cols = torch.zeros(cfg.n_rows, work.history, dtype=torch.int64)
            cols[1:] = codes
            cols[0] = TOK_SEMANTIC0 + codes[0]
            g = torch.cat([g, cols], dim=1)
        out.append(g)
    return out


def settings_for(work: Work):
    from smoltts_b200 import GenerationSettings

    if work.sampled:
        return GenerationSettings(default_temp=0.7, default_fast_temp=0.7, top_k=50, top_p=0.9, seed=1234)
    return GenerationSettings(default_temp=0.0, default_fast_temp=0.0)


def public_config(work: Work, world: int) -> dict:
    """What both arms (ours / --impl reference) report as the configuration they measure."""
    return {"workload": work.name(), "model": work.model, "batch_per_gpu": work.batch, "frames_per_step": work.frames,
            "prompt_tokens": work.prompt_tokens, "mean_context": work.mean_context,
            "l2": "no flush: each frame streams 271 MB of weights (> 126 MB L2) plus the KV cache",
            "sharding": f"utterance-parallel x{world}, no collective on the decode path"}


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle (a port of the reference's arithmetic with a KV cache) on the host cores
# ------------------------------------------------------------------------------------------------
class CpuArm:
    """`n_frames` frames decoded on the CPU for `work.batch` sequences with the KV cache pre-filled (untimed) so that the
    sample's contexts are centred on the workload's mean context: the same configuration, a bounded sample of its frames."""

    def __init__(self, work: Work, n_frames: int):
        import torch

        from oracle.dualar_oracle import DualAROracle, OracleSettings
        from oracle.sampler_oracle import OracleSampler
        from smoltts_b200.config import named_config
        from smoltts_b200.synth import make_state_dict

        torch.set_num_threads(os.cpu_count() or 1)
        self.torch = torch
        self.work = work
        self.n_frames = min(n_frames, work.frames)
        cfg = named_config(work.model)
        # columns cached before the sample starts: the prompt plus the frames the workload has decoded by then
        self.skip = (work.frames - self.n_frames) // 2
        w2 = Work(work.key, work.model, work.batch, work.frames, work.prompt_bytes, work.sampled, work.history + self.skip)
        self.orc = DualAROracle(cfg, make_state_dict(cfg, seed=0), dtype=torch.bfloat16,
                                max_seq_len=max(cfg.max_seq_len, w2.prompt_tokens + self.n_frames + 8))
        self.cols = torch.stack(synth_prompts(cfg, w2, 0), 0)
        self.st = (OracleSettings(default_temp=0.7, default_fast_temp=0.7, top_k=50, top_p=0.9, seed=1234) if work.sampled
                   else OracleSettings(default_temp=0.0, default_fast_temp=0.0))
        self.sampler = OracleSampler(seq_ids=list(range(work.batch))) if work.sampled else None
        self.first_context = w2.prompt_tokens
        self.threads = torch.get_num_threads()

    def step(self):
        torch = self.torch
        with torch.no_grad():
            cache = self.orc.new_cache()
            t0 = time.perf_counter()
            nxt, *_ = self.orc.decode_frame(self.cols, cache, self.st, 0, self.sampler)  # prefill + first frame: untimed (G:187-193)
            t1 = time.perf_counter()
            for f in range(1, self.n_frames + 1):
                nxt, *_ = self.orc.decode_frame(nxt[:, :, None], cache, self.st, f, self.sampler)
            t2 = time.perf_counter()
        return {"decode_s": t2 - t1, "prefill_s": t1 - t0, "frames": self.n_frames * self.work.batch}

    def sample_text(self) -> str:
        w = self.work
        return (f"{self.n_frames} of the step's {w.frames} frames, taken at the workload's mean context (contexts "
                f"{self.first_context + 1}..{self.first_context + self.n_frames}, KV cache pre-filled untimed), bs={w.batch}, bf16 eager "
                f"on CPU: oracle port of the reference's modeling/ arithmetic with a KV cache (prefill excluded as in lm/generate.py:187-214)")


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    work = headline_work(args)
    arm = CpuArm(work, args.cpu_frames or CPU_SAMPLE_FRAMES)
    per_step = []
    for i in range(args.warmup + args.steps):
        r = arm.step()
        if i >= args.warmup:
            per_step.append(r)
    total_frames = sum(r["frames"] for r in per_step)
    total_s = sum(r["decode_s"] for r in per_step)
    value = total_frames / total_s
    line = {
        "impl": "reference", "metric": "Mimi frames/sec", "value": value, "unit": "frames/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total_s / len(per_step),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
        "config": public_config(work, max(1, args.gpus)),
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": arm.threads, "kind": "port", "sample": arm.sample_text()},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def roofline_of(cfg, work: Work, kernel_ms: float, tensor_variant: bool, kernel_name: str, traffic_per_frame):
    hbm_gbs, peak_src = load_peaks()
    tf_peak, tf_src = load_tensor_peak()
    l_mean = work.mean_context
    bytes_per_frame = cfg.unique_weight_bytes() + work.batch * cfg.kv_bytes_per_position() * (l_mean + 1)
    flops_per_frame = work.batch * cfg.flops_per_frame(l_mean)
    t_bytes_us = bytes_per_frame / (hbm_gbs * 1e9) * 1e6
    t_flops_us = flops_per_frame / (tf_peak * 1e12) * 1e6
    common = {"kernel": kernel_name, "launch_ms": kernel_ms, "units_per_launch": work.frames,
              "roof_us_per_frame_step": {"flops": t_flops_us, "bytes": t_bytes_us},
              "traffic": (traffic_per_frame * work.frames) if traffic_per_frame else None}
    if tensor_variant and t_flops_us >= t_bytes_us:
        ach = flops_per_frame * work.frames / (kernel_ms * 1e-3) / 1e12
        return {"bound": "tensor", "achieved": ach, "peak": tf_peak, "unit": "TFLOP/s", "frac": ach / tf_peak, "peak_source": tf_src,
                "algorithmic_flops_per_launch": flops_per_frame * work.frames, **common}
    ach = bytes_per_frame * work.frames / (kernel_ms * 1e-3) / 1e9
    return {"bound": "hbm", "achieved": ach, "peak": hbm_gbs, "unit": "GB/s", "frac": ach / hbm_gbs, "peak_source": peak_src,
            "algorithmic_bytes_per_launch": bytes_per_frame * work.frames, **common}


def measure(work: Work, args, steps: int, warmup: int, ctx) -> dict:
    """Device-resident value, e2e through generate_batch (+ gather on rank 0) and the roofline of one workload."""
    import torch

    from smoltts_b200 import RQTransformer, generate_batch, named_config
    from smoltts_b200.generate import _sampling, pack_prompts
    from smoltts_b200.shard import gather_utterances
    from smoltts_b200.synth import make_state_dict

    dist, gloo, rank, world, local = ctx["dist"], ctx["gloo"], ctx["rank"], ctx["world"], ctx["local"]
    cfg = named_config(work.model)
    n_prompt = work.prompt_tokens
    need = max(n_prompt + work.frames + 8, 256)
    model = RQTransformer(cfg, max_batch=work.batch, max_seq_len=need, kv_pages=2 * work.batch * ((need + 31) // 32))
    model.load_state_dict(ctx["weights"](work.model))
    model.set_option("mode", args.mode)
    for kv in args.opt:
        k, v = kv.split("=")
        model.set_option(k, int(v))
    gs = settings_for(work)
    first = rank * work.batch
    prompts = synth_prompts(cfg, work, first)
    seq_ids = [first + b for b in range(work.batch)]
    dev = model.device

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- device-resident arm: prefill once, then every step decodes `frames` frames from the same state
    padded, lens = pack_prompts(model, prompts)
    batch = model.new_batch(work.batch, max_positions=n_prompt + work.frames + 1, max_frames=work.frames, seq_ids=seq_ids)
    sampling = _sampling(model, gs, audio_only=True, ignore_stop=True)
    model.prefill(batch, padded, lens)
    torch.cuda.synchronize()
    tokens0, len0 = batch.tokens.clone(), batch.seq_len.clone()
    host_len0 = list(batch.host_len)

    def reset():
        batch.tokens.copy_(tokens0)
        batch.seq_len.copy_(len0)
        batch.step.zero_()
        batch.finished.zero_()
        batch.host_len = list(host_len0)

    frame_clock = model.set_frame_clock(work.frames) if work.batch == 1 else None  # device-side per-frame stamps (sequence 0)
    for _ in range(warmup):
        reset()
        model.decode_frames(batch, sampling, work.frames)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    launches0 = model.launch_count
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for i in range(steps):
        reset()
        ev[i][0].record()
        model.decode_frames(batch, sampling, work.frames)
        ev[i][1].record()
    stop.record()
    barrier()
    launches = model.launch_count - launches0
    clocks = sampler.stop()
    total_ms = start.elapsed_time(stop)
    kernel_ms = statistics.mean(a.elapsed_time(b) for a, b in ev)
    codes_check = int(batch.out_codes.sum().item())  # the result is really produced
    # what the last timed step handed back: [batch, rows, frames] ids, as generate_batch(audio_only=False) returns per utterance
    outputs = {"codes": batch.out_codes.permute(0, 2, 1).cpu().numpy()} if args.dump_outputs else {}
    frame_lat = None
    if frame_clock is not None:  # stamps of the last timed step: p50 / p99 of the per-frame latency (BASELINE.json's second metric)
        ns = frame_clock.cpu().numpy().astype("float64")
        d = (ns[1:] - ns[:-1]) * 1e-3
        d = d[d > 0]
        if d.size:
            d.sort()
            frame_lat = {"p50_us": float(d[int(0.50 * (d.size - 1))]), "p99_us": float(d[int(0.99 * (d.size - 1))]),
                         "max_us": float(d[-1]), "frames": int(d.size) + 1, "clock": "%globaltimer at frame assembly, on the device"}
        model.set_frame_clock(0)
    batch.release()

    # ---- end-to-end arm: public API from pinned host prompts; H2D + prefill + decode + D2H (+ gather on rank 0) every step
    host_prompts = [p.pin_memory() for p in prompts]

    def e2e_step():
        outs = generate_batch(model, host_prompts, gs, audio_only=False, fixed_frames=work.frames, chunk=work.frames, seq_ids=seq_ids)
        return gather_utterances(outs, dist, group=gloo) if world > 1 else outs

    for _ in range(max(1, min(warmup, 2))):
        e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        got = e2e_step()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    if rank == 0:
        assert got is not None and len(got) == work.batch * world and tuple(got[-1].shape) == (cfg.n_rows, work.frames)
    h2d = int(padded.numel() * 4 + lens.numel() * 4)
    d2h = int(work.batch * work.frames * cfg.n_rows * 4 + work.batch * 4)

    # ---- max over ranks
    t = torch.tensor([total_ms, e2e_s * 1e3, kernel_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms, kernel_ms = (float(v) for v in t.tolist())

    dataflow = args.mode == 2 and work.batch <= model.get_option("ll_max_batch")
    tensor = not dataflow and work.batch >= model.get_option("tc_min_batch") > 0
    kernel_name = ("smol_ll2_kernel (tensor-core GEMV, LL flag words)" if dataflow
                   else "smol_decode_kernel<0> (tcgen05 tiles, TMA operand ring)" if tensor else "smol_decode_kernel")
    traffic = load_traffic() or {}
    tr = (traffic.get(work.key) or {}).get("dram_bytes_per_frame") if work.model == "smoltts_byte_150m" else None
    res = {
        "workload": work.name(), "note": work.note, "value": steps * work.frames * work.batch * world / (total_ms * 1e-3),
        "unit": "frames/s", "ms_per_step": total_ms / steps, "steps": steps, "warmup": warmup,
        "us_per_frame_step": 1e3 * kernel_ms / work.frames,
        "roofline": roofline_of(cfg, work, kernel_ms, tensor, kernel_name, tr),
        "e2e": {"value": steps * work.frames * work.batch * world / (e2e_ms * 1e-3), "unit": "frames/s",
                "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps,
                "includes": "H2D prompt grid + prefill + decode + D2H codes via generate_batch()"
                            + (", + host-side gather of all ranks' codes on rank 0 (gloo)" if world > 1 else "")},
        "clocks": clocks, "gpu_launches": launches, "check": codes_check, "frame_latency_bs1": frame_lat,
        "launch_mode": ("data-flow persistent kernel (LL flag words, TMA producer warp, one team of CTAs per sequence), one launch per step" if dataflow
                        else "persistent cooperative kernel with grid barriers, one launch per step" if args.mode != 1
                        else "per-phase launches in a CUDA graph"),
        "config": public_config(work, world), "outputs": outputs,
    }
    del model
    torch.cuda.empty_cache()
    return res


def measure_mimi(key: str, batch: int, frames: int, args, steps: int, warmup: int, ctx) -> dict:
    """The step after the path (SURVEY 8(f)-2): Mimi streaming decoder, `batch` streams x `frames` decode_step calls per
    bench step.  value: codes resident in HBM; e2e: codes from pinned host memory, PCM back to pinned host memory, through
    MimiModel.decode_step.  Roofline: every packed fp32 weight once per decode_step + the KV the step touches."""
    import torch

    from smoltts_b200.mimi import MimiModel
    from smoltts_b200.synth import make_mimi_state_dict

    dist, rank, world, local = ctx["dist"], ctx["rank"], ctx["world"], ctx["local"]
    sd = ctx["mimi_weights"]()
    m = MimiModel(max_streams=batch, max_frames=frames + 8)
    m.load_state_dict(sd)
    dev = m.device
    g = torch.Generator().manual_seed(100 + rank)
    codes_h = torch.randint(0, 2048, (frames, batch, 8), generator=g, dtype=torch.int32).pin_memory()
    codes_d = codes_h.to(dev)
    pcm_h = torch.empty(frames, batch, m.samples_per_frame, dtype=torch.float32).pin_memory()
    caches = [m.make_cache() for _ in range(batch)]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def run(resident: bool):
        m._reset([c.slot for c in caches])
        for t in range(frames):
            pcm = m.decode_step(codes_d[t] if resident else codes_h[t].to(dev, non_blocking=True), caches)
            if not resident:
                pcm_h[t].copy_(pcm[:, 0], non_blocking=True)
        return pcm

    for _ in range(warmup):
        run(True)
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    start, stop = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(steps):
        last = run(True)
    stop.record()
    barrier()
    clocks = sampler.stop()
    total_ms = start.elapsed_time(stop)
    check = float(last.abs().sum().item())
    for _ in range(max(1, min(warmup, 2))):
        run(False)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        run(False)
    torch.cuda.synchronize()
    e2e_ms = (time.perf_counter() - t0) * 1e3
    # the resident arm keeps only the last frame's PCM; the e2e arm's last step leaves every frame of the same codes in pcm_h
    outputs = {"pcm": pcm_h.permute(1, 0, 2).numpy().copy()} if args.dump_outputs else {}     # [streams, frames, samples]
    t = torch.tensor([total_ms, e2e_ms], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, e2e_ms = (float(v) for v in t.tolist())
    wbytes = sum(v.numel() * 4 for k, v in sd.items() if "codebook" not in k) + 8 * 256 * 4
    mean_pos = frames + 1            # 2 positions per frame, mean over the run
    kv = batch * 8 * 2 * 512 * 4 * (mean_pos + 2)
    us_step = 1e3 * total_ms / (steps * frames)
    hbm, src = load_peaks()
    ach = (wbytes + kv) / (us_step * 1e-6) / 1e9
    res = {
        "key": key, "workload": f"Mimi streaming decoder (kyutai/mimi shape, seeded fp32 weights): {batch} stream(s) x {frames} decode_step calls per step",
        "note": "SURVEY 8(f)-2: codes [B, 8] -> 1920 fp32 samples per frame; 57 launches per decode_step replayed as one CUDA graph",
        "value": steps * frames * batch * world / (total_ms * 1e-3), "unit": "frames/s", "ms_per_step": total_ms / steps, "steps": steps,
        "warmup": warmup, "us_per_frame_step": us_step,
        "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm, "unit": "GB/s", "frac": ach / hbm, "peak_source": src,
                     "traffic": ((load_traffic() or {}).get(key) or {}).get("dram_bytes_per_frame"),   # per decode_step, like algorithmic_bytes_per_launch
                     "kernel": "smol::mimi::rows_kernel (weight-streaming row products, fp32 FMA)",
                     "algorithmic_bytes_per_launch": wbytes + kv,
                     "bytes_model": "packed fp32 weights of the decode half once per decode_step + KV cache read/written",
                     "fp32_tflops_achieved": batch * m.flops_per_frame() / (us_step * 1e-6) / 1e12,
                     "fp32_note": "fp32 FMA on CUDA cores (the reference's precision); at 64 streams this, not HBM, is the nearer roof "
                                  "(B200 nominal ~75 TFLOP/s fp32 non-tensor)"},
        "e2e": {"value": steps * frames * batch * world / (e2e_ms * 1e-3), "unit": "frames/s", "h2d_bytes_per_step": frames * batch * 8 * 4,
                "d2h_bytes_per_step": frames * batch * m.samples_per_frame * 4, "steps": steps},
        "clocks": clocks, "gpu_launches": steps * frames * m.launches_per_step, "launch_mode": "57 launches per decode_step, CUDA-graph replay",
        "realtime_factor": steps * frames * batch * world / (total_ms * 1e-3) / 12.5, "check": check, "outputs": outputs,
    }
    if rank == 0 and world == 1 and batch == 1 and not args.no_cpu_baseline:
        from oracle.mimi_oracle import MimiOracle, StreamState   # CPU leg only (the checker, never the product)

        orc, st = MimiOracle(sd), StreamState()
        n = 24
        with torch.no_grad():
            orc.decode_step(codes_h[0][0:1].long()[:, :, None], st)      # warm-up call (allocator, thread pool)
            t1 = time.perf_counter()
            for t in range(1, 1 + n):
                orc.decode_step(codes_h[t % frames][0:1].long()[:, :, None], st)
            cpu_s = time.perf_counter() - t1
        res["cpu_baseline"] = {"value": n / cpu_s, "unit": "frames/s", "cores": torch.get_num_threads(), "kind": "port",
                               "sample": f"{n} decode_step calls of one stream (oracle/mimi_oracle.py, torch CPU fp32)"}
    del m
    torch.cuda.empty_cache()
    return res


def measure_tts_stream(args, steps: int, warmup: int, ctx, frames: int = 128) -> dict:
    """The reference's streaming loop end to end (smoltts_mlx/__init__.py:85-95) at one utterance: prompt -> one frame per
    SingleBatchGenerator.__next__ (one launch of the data-flow kernel, ids read back by the host) -> MimiModel.decode_step ->
    the 80 ms PCM chunk on the host.  There is no device-resident form of this loop: value == e2e."""
    import numpy as np
    import torch

    from smoltts_b200 import GenerationSettings, MimiModel, PromptEncoder, RQTransformer, SmolTTS, byte_level_tokenizer, named_config

    dist, rank, world, local = ctx["dist"], ctx["rank"], ctx["world"], ctx["local"]
    cfg = named_config(args.model)
    lm = RQTransformer(cfg, max_batch=1, max_seq_len=512 + frames)
    lm.load_state_dict(ctx["weights"](args.model))
    codec = MimiModel(max_streams=1, max_frames=frames + 8)
    codec.load_state_dict(ctx["mimi_weights"]())
    enc = PromptEncoder.from_model(byte_level_tokenizer(cfg.codebook_size), lm)
    tts = SmolTTS(lm, enc, codec, settings=GenerationSettings(default_temp=0.0, default_fast_temp=0.0, max_new_tokens=frames - 1))
    text = "The quick brown fox jumps over the lazy dog. " * 4          # 180 bytes
    chunks = []

    def run():
        # random-init weights emit non-audio ids now and then (they skip the codec, as in the reference) and may hit
        # <|im_end|> early: SmolTTS.stream reports what it generated
        st = {}
        chunks.clear()
        for chunk in tts.stream(text, "nova", overlap=not args.no_stream_overlap, lm_ctas=args.stream_lm_ctas, stats=st):
            chunks.append(chunk)
        return st["frames"], st["audio_frames"]

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(1, min(warmup, 2))):
        n_gen, n_pcm = run()
    barrier()
    sampler = ClockSampler(local)
    sampler.start()
    t0 = time.perf_counter()
    for _ in range(steps):
        n_gen, n_pcm = run()
    torch.cuda.synchronize()
    frames = n_gen
    ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()
    t = torch.tensor([ms], dtype=torch.float64, device=lm.device)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    value = steps * frames * world / (ms * 1e-3)
    res = {
        "key": "tts_stream_bs1", "workload": f"SmolTTS.stream: {args.model} greedy + Mimi decoder, one utterance, {frames} frames per step, one frame per host iteration",
        "note": "the reference's streaming loop (generator.__next__ -> codec.decode_step -> numpy chunk), prefill included; "
                f"{n_pcm} of {frames} frames were audio frames and went through the codec",
        "value": value, "unit": "frames/s", "ms_per_step": ms / steps, "steps": steps, "warmup": warmup, "us_per_frame_step": 1e3 * ms / (steps * frames),
        "roofline": None,
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": frames * (cfg.n_rows * 4) + n_pcm * 1920 * 4, "steps": steps},
        "clocks": clocks, "gpu_launches": steps * (frames * lm.get_option("ll_ready") + n_pcm * codec.launches_per_step),
        "launch_mode": "one data-flow kernel launch per frame + 57 codec launches per audio frame (CUDA-graph replay)"
                       + ("" if args.no_stream_overlap else "; pipelined: the decode step of frame t + 1 is launched before the host reads frame t, whose ids, "
                                                              "codec step and PCM go through a side stream (decode kernel on %d of the SMs)" % args.stream_lm_ctas),
        "realtime_factor": value / 12.5,
        "outputs": {"pcm": np.concatenate(chunks)} if args.dump_outputs and chunks else {},   # the chunks of the last timed run
    }
    del tts, lm, codec
    torch.cuda.empty_cache()
    return res


def run_ours(args):
    import torch

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (impl=ours) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dist = gloo = None
    if world > 1:
        import torch.distributed as dist_mod

        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        gloo = dist.new_group(backend="gloo")  # host-side gather of the emitted codes (SURVEY 8(e)); NCCL only times

    from smoltts_b200.config import named_config
    from smoltts_b200.synth import make_state_dict

    wcache = {}

    def weights(name):
        if name not in wcache:
            wcache[name] = make_state_dict(named_config(name), seed=0)
        return wcache[name]

    def mimi_weights():
        if "mimi" not in wcache:
            from smoltts_b200.synth import make_mimi_state_dict

            wcache["mimi"] = make_mimi_state_dict(0)
        return wcache["mimi"]

    ctx = {"dist": dist, "gloo": gloo, "rank": rank, "world": world, "local": local, "weights": weights, "mimi_weights": mimi_weights}
    head = headline_work(args)
    main = measure(head, args, args.steps, args.warmup, ctx)
    entries = []
    if args.configs != "none" and (args.configs != "auto" or head.key == "config2"):
        wanted = None if args.configs == "auto" else set(args.configs.split(","))
        for w in extra_works(args.model):
            if wanted is None or w.key in wanted:
                r = measure(w, args, max(1, min(args.steps, args.config_steps)), 3, ctx)
                r["key"] = w.key
                entries.append(r)
        for key, b, f in (("mimi_bs1", 1, 256), ("mimi_bs64", 64, 32)):     # the step after the path: codes -> PCM
            if wanted is None or key in wanted:
                entries.append(measure_mimi(key, b, f, args, max(1, min(args.steps, args.config_steps)), 3, ctx))
        if (wanted is None or "tts_stream_bs1" in wanted) and args.model == "smoltts_byte_150m":
            entries.append(measure_tts_stream(args, max(1, min(args.steps, 3)), 2, ctx))
    if args.dump_outputs:
        suffix = f"_rank{rank}" if world > 1 else ""
        dump_outputs(args.dump_outputs, {f"{key}_{name}{suffix}": a for key, outs in [("headline", main["outputs"])]
                                         + [(e["key"], e["outputs"]) for e in entries] for name, a in outs.items()},
                     DUMP_BYTES // world)

    if rank == 0:
        cfg_pub = dict(main["config"])  # identical in both arms (ours / --impl reference): the configuration measured
        line = {
            "metric": "Mimi frames/sec", "value": main["value"], "unit": "frames/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": cfg_pub, "roofline": main["roofline"],
            "e2e": {k: v for k, v in main["e2e"].items() if k != "includes"}, "clocks": main["clocks"],
            "gpu_launches": main["gpu_launches"] + sum(e["gpu_launches"] for e in entries), "check": main["check"],
            "latency": {"us_per_frame": main["us_per_frame_step"], "frame_latency_bs1": main["frame_latency_bs1"]},
            "detail": {"launch_mode": main["launch_mode"], "e2e_includes": main["e2e"]["includes"]},
            "configs": [{k: e[k] for k in ("key", "workload", "note", "value", "unit", "ms_per_step", "steps", "warmup",
                                           "us_per_frame_step", "roofline", "e2e", "clocks", "gpu_launches", "launch_mode",
                                           "realtime_factor", "cpu_baseline") if k in e}
                        for e in entries],
        }
        if world == 1 and not args.no_cpu_baseline:
            arm = CpuArm(head, args.cpu_frames or CPU_SAMPLE_FRAMES)
            rs = [arm.step() for _ in range(4)]  # ~10-15 s of CPU work; the first pass warms the allocator up
            rs = rs[1:]
            line["cpu_baseline"] = {"value": sum(r["frames"] for r in rs) / sum(r["decode_s"] for r in rs), "unit": "frames/s",
                                    "cores": arm.threads, "kind": "port", "sample": "3 x " + arm.sample_text()}
        print(json.dumps(line), flush=True)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
