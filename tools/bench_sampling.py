"""AR decode-step time of the three ways to pick the next id, on the bench.py model and workload (d=1024/16h/12L, bf16,
S=47 phonemes, 225-frame prompt, random weights):

  greedy   top_k=1: argmax in the sampler kernel, 8-step CUDA-graph replays
  torch    top_k=-100, T=1, no seeds: eager decode step + torch.multinomial on the CUDA logits + vb_ar_push_tokens
  seeded   top_k=-100, T=1, seeds: the draw in the sampler kernel, 8-step CUDA-graph replays

The modes alternate in one process, `--reps` times, at every batch size.  Per mode and size it reports the AR time per
decode step (EngineStats.ar_ms / ar_steps), the mean number of rows still running per step (a sampled decode can reach
EOS early on random weights), and the device kernels per decode step (torch.profiler, difference of two runs of
different length), plus the card name and power limit read in the same process.  Prints one JSON line.

    python tools/bench_sampling.py [--batches 64 1] [--frames 256] [--reps 3]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import bench  # noqa: E402

MODES = ("greedy", "torch", "seeded")


def run(eng, texts, prompts, mode, frames, seed):
    kw = dict(max_new_tokens=frames, return_device=True)
    if mode == "greedy":
        out = eng.generate(texts, prompts, top_k=1, **kw)
    elif mode == "torch":
        torch.manual_seed(seed)
        out = eng.generate(texts, prompts, top_k=-100, temperature=1.0, **kw)
    else:
        seeds = [(seed << 20) + b for b in range(len(texts))]
        out = eng.generate(texts, prompts, top_k=-100, temperature=1.0, seeds=seeds, **kw)
    torch.cuda.synchronize()
    steps = eng.stats.ar_steps
    running = sum(min(int(o.shape[0]), steps) for o in out) / max(1, steps)
    return eng.stats.ar_ms / max(1, steps), running, steps


def kernels_per_step(eng, texts, prompts, mode, frames):
    """device kernels per decode step: profiled runs of frames // 4 and frames steps, difference over the step counts"""
    from torch.profiler import ProfilerActivity, profile
    counts = []
    for f in (max(8, frames // 4), frames):
        run(eng, texts, prompts, mode, f, 1)      # capture graphs of this shape outside the profile
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            _, _, steps = run(eng, texts, prompts, mode, f, 1)
        n = sum(1 for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA)
        counts.append((n, steps))
    (n0, s0), (n1, s1) = counts
    return (n1 - n0) / (s1 - s0) if s1 != s0 else None


def card():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        r = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        info["power_limit"], info["sm_max_clock"] = [v.strip() for v in r.stdout.strip().split(",")]
    except Exception as e:  # noqa: BLE001
        info["power_limit"] = f"unavailable ({e})"
    return info


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", type=int, nargs="+", default=[64, 1])
    ap.add_argument("--frames", type=int, default=256, help="cap of generated frames per utterance")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--no-profile", action="store_true", help="skip the kernels-per-step count")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_sampling.py needs a CUDA device")
    dev = torch.device("cuda:0")
    model = bench.build_model(dev)
    eng = model.engine(torch.bfloat16)
    eng.quiet = True
    res = {"card": card(), "model": f"d={bench.D_MODEL}/{bench.N_HEAD}h/{bench.N_LAYER}L bf16",
           "workload": f"S={bench.S_TEXT}, prompt {bench.T_PROMPT} frames, cap {a.frames} frames", "reps": a.reps,
           "decode_fold": eng.use_decode_fold, "by_batch": {}}
    for B in a.batches:
        texts, prompts = bench.make_batch(B, 7, dev)
        for mode in MODES:
            run(eng, texts, prompts, mode, a.frames, 0)   # warm-up: graph capture, allocator
        samples = {m: [] for m in MODES}
        for rep in range(a.reps):
            for mode in MODES:
                samples[mode].append(run(eng, texts, prompts, mode, a.frames, rep + 1))
        out = {}
        for mode in MODES:
            ms = [s[0] for s in samples[mode]]
            out[mode] = {"ar_ms_per_step": statistics.median(ms), "ar_ms_per_step_all": ms,
                         "mean_running_rows": statistics.mean(s[1] for s in samples[mode]),
                         "ar_steps": [s[2] for s in samples[mode]]}
            if not a.no_profile:
                out[mode]["kernels_per_step"] = kernels_per_step(eng, texts, prompts, mode, a.frames)
        g = out["greedy"]["ar_ms_per_step"]
        out["seeded_vs_greedy"] = out["seeded"]["ar_ms_per_step"] / g - 1.0
        out["seeded_vs_torch"] = out["seeded"]["ar_ms_per_step"] / out["torch"]["ar_ms_per_step"] - 1.0
        res["by_batch"][str(B)] = out
    print(json.dumps(res))


if __name__ == "__main__":
    main()
