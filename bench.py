#!/usr/bin/env python
"""bench.py -- audio tokens/sec of the VALL-E AR+NAR decode hot path on B200.

The JSON line also carries, as sub-objects measured in the same run (N=1 unless noted): `parity` (the timed bf16
batch holds the inputs of the reference fixture big_full as utterance 0: token-match rate / first divergence vs the
reference's codes, and the fp32 engine's bit-exactness on the same inputs), `parity_mode` (fp32 tokens/s and its
roofline), `config2` (NAR B=32 x L=1500), `config3` (256 prompts, strong scaling, every N), `config4` (EnCodec
encode + decode), `roofline_b1` / `p50_utt_latency_ms` (configs[1]), `cpu_baseline`.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

A "step" = one pass of the hot path over one batch of synthetic utterances per GPU:
B utterances x (S=47 phonemes, 225-frame prompt) -> greedy AR decode to the reference's cap
(16*S+1 = 753 frames, valle.py:1047) + 7 NAR passes -> B x 753 x 8 audio tokens.
Weak scaling: every rank decodes its own B utterances (no data-path collective), then ONE
all-gather of the code matrices.  Prints ONE JSON line (rank 0).  See DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

D_MODEL, N_HEAD, N_LAYER = 1024, 16, 12
S_TEXT, T_PROMPT, N_Q = 47, 225, 8
FRAMES = 16 * S_TEXT + 1  # 753: cap-terminated generation with random weights


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=64, help="utterances per GPU per step")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "fp32"])
    ap.add_argument("--frames", type=int, default=0, help="cap generated frames (0 = reference cap 16*S+1)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-latency", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=20.0)
    ap.add_argument("--total-prompts", type=int, default=256,
                    help="BASELINE configs[3]: prompts of the strong-scaling job sharded over the ranks (0 = skip)")
    ap.add_argument("--no-extra", action="store_true",
                    help="skip the sub-objects (parity, parity_mode, config2/3/4, batch-1 latency, cpu_baseline)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the codes the timed path returned in its last step to DIR/codes.npy")
    return ap.parse_args()


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return dict(hbm_gbs=j["hbm_gbs"], tflops=j.get("bf16_tflops_sustained", j["bf16_tflops"]),
                    tflops_burst=j["bf16_tflops"], source="MEASURED_PEAKS.json (measured)")
    return dict(hbm_gbs=6650.0, tflops=1400.0, tflops_burst=1590.0, source="B200_PROFILING.md fallback")


# ----------------------------------------------------------------------------- synthetic workload
def make_batch(B, seed, device=None, pinned=False):
    g = torch.Generator().manual_seed(seed)
    texts = [torch.randint(3, 100, (S_TEXT,), generator=g) for _ in range(B)]
    prompts = [torch.randint(0, 1024, (T_PROMPT, N_Q), generator=g) for _ in range(B)]
    if device is not None:
        texts = [t.to(device) for t in texts]
        prompts = [p.to(device) for p in prompts]
    elif pinned:
        texts = [t.pin_memory() for t in texts]
        prompts = [p.pin_memory() for p in prompts]
    return texts, prompts


def build_model(device):
    from valle_b200.models import VALLE
    torch.manual_seed(0)
    m = VALLE(D_MODEL, N_HEAD, N_LAYER, norm_first=True, add_prenet=False, prefix_mode=1,
              share_embedding=True, nar_scale_factor=1.0, prepend_bos=False, num_quantizers=N_Q).eval()
    return m.to(device)


# ----------------------------------------------------------------------------- clocks sampler
class Clocks:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.samples, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------- algorithmic work
def ar_step_bytes(B, mean_len, esize):
    """SURVEY.md 8d: W + B * (KV_read(L) + KV_write); W = weights streamed once per step."""
    per_layer = 12 * D_MODEL * D_MODEL
    w = (N_LAYER * per_layer + 1025 * D_MODEL) * esize                # matrices + AR head
    w += N_LAYER * 13 * D_MODEL * 4 + 2 * D_MODEL * 4                 # biases / LN affine (fp32)
    kv = 2 * N_LAYER * D_MODEL * esize                                 # bytes per cached token (K+V)
    return w + B * (kv * mean_len + kv)


def nar_pass_flops(B, L, tgen):
    M = B * L
    return 2 * M * N_LAYER * 12 * D_MODEL * D_MODEL + N_LAYER * B * 4 * L * L * D_MODEL + 2 * B * tgen * D_MODEL * 1024


# ----------------------------------------------------------------------------- CPU baseline
def _host_threads():
    try:
        avail = len(os.sched_getaffinity(0))
    except Exception:
        avail = os.cpu_count() or 1
    try:  # cgroup v2 CPU quota, if any
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            avail = max(1, min(avail, int(int(q) / int(per))))
    except Exception:
        pass
    return avail


def cpu_reference_sample(seconds, threads=None, one_thread=True):
    """The reference's own algorithm (oracle port: full recompute per token, batch 1, fp32, no KV cache) timed on the
    host cores over a bounded sample: full-recompute AR iterations at three context lengths + one NAR pass,
    integrated over the 753-frame utterance (ESTIMATED: the whole utterance takes minutes).  Reported for the
    fastest thread count found and, scaled by one mid-context iteration, for 1 thread (valle/bin/infer.py:272 sets
    torch.set_num_threads(1), the as-shipped setting)."""
    from oracle import valle_oracle as O
    from valle_b200.models import VALLE
    threads = threads or _host_threads()
    torch.set_num_threads(threads)
    torch.manual_seed(0)
    m = VALLE(D_MODEL, N_HEAD, N_LAYER, norm_first=True, add_prenet=False, prefix_mode=1, share_embedding=True,
              nar_scale_factor=1.0, prepend_bos=False, num_quantizers=N_Q).eval()
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    cfg = O.OracleConfig(D_MODEL, N_HEAD, N_LAYER, 1, N_Q)
    g = torch.Generator().manual_seed(9)
    x = torch.randint(3, 100, (1, S_TEXT), generator=g)
    xe = O.pos_embed(sd["ar_text_embedding.word_embeddings.weight"][x], sd["ar_text_position.alpha"])

    def ar_iter(t):  # one iteration of valle.py:1012-1057 with t audio tokens in context
        yy = torch.randint(0, 1024, (1, t), generator=g)
        ye = O.pos_embed(sd["ar_audio_embedding.word_embeddings.weight"][yy], sd["ar_audio_position.alpha"])
        xy = torch.concat([xe, ye], dim=1)
        t0 = time.perf_counter()
        with torch.no_grad():
            dec = O.encoder(sd, "ar_decoder", xy, cfg, blocked=O.ar_inference_mask(S_TEXT, t))
            torch.nn.functional.linear(dec[:, -1], sd["ar_predict_layer.weight"])
        return time.perf_counter() - t0

    def nar_pass():
        L = S_TEXT + T_PROMPT + FRAMES
        xy = torch.randn(1, L, D_MODEL, generator=g)
        t0 = time.perf_counter()
        with torch.no_grad():
            dec = O.encoder(sd, "nar_decoder", xy, cfg,
                            stage_emb=sd["nar_stage_embeddings.0.word_embeddings.weight"])
            torch.nn.functional.linear(dec[:, S_TEXT + T_PROMPT:], sd["nar_predict_layers.0.weight"])
        return time.perf_counter() - t0

    ctx = [T_PROMPT, T_PROMPT + FRAMES // 2, T_PROMPT + FRAMES - 1]
    ar_iter(ctx[0])  # warm-up
    # "all the host threads it can use": pick the thread count that is actually fastest on this
    # box (a 128-thread pool on a small GEMM can be far slower than 16-32 threads)
    best_t, best_time = threads, None
    for cand in sorted({threads, 64, 32, 16, 8}, reverse=True):
        if cand > threads:
            continue
        torch.set_num_threads(cand)
        ar_iter(ctx[0])
        tt = ar_iter(ctx[0])
        if best_time is None or tt < best_time:
            best_t, best_time = cand, tt
    threads = best_t
    torch.set_num_threads(threads)
    t_budget = time.perf_counter()
    times = {c: [] for c in ctx}
    reps = 0
    while reps < 1 or (time.perf_counter() - t_budget < seconds * 0.7 and reps < 5):
        for c in ctx:
            times[c].append(ar_iter(c))
        reps += 1
    tm = [min(times[c]) for c in ctx]
    # piecewise-linear integral of the per-iteration time over the 753 iterations
    half = FRAMES / 2.0
    ar_total = half * (tm[0] + tm[1]) / 2 + half * (tm[1] + tm[2]) / 2
    t_nar = nar_pass()
    total = ar_total + 7 * t_nar
    r = dict(value=FRAMES * N_Q / total, seconds_per_utt=total, ar_seconds=ar_total, nar_pass_seconds=t_nar,
             cores=threads, host_threads_available=_host_threads(),
             sample=f"ESTIMATED from {reps}x3 full-recompute AR iterations at {ctx} audio tokens of context + 1 NAR pass "
                    f"(L={S_TEXT + T_PROMPT + FRAMES}), B=1 fp32, integrated over {FRAMES} frames + 7 passes")
    if one_thread:
        torch.set_num_threads(1)
        t1 = ar_iter(ctx[0])                       # one iteration at the shortest context, single thread
        torch.set_num_threads(threads)
        scale = t1 / tm[0]
        r["value_1thread"] = r["value"] / scale
        r["seconds_per_utt_1thread"] = total * scale
        r["sample_1thread"] = (f"ESTIMATED: the all-thread sample scaled by the 1-thread / {threads}-thread time of one AR "
                               f"iteration at {ctx[0]} audio tokens ({t1:.2f} s vs {tm[0]:.2f} s)")
    return r


# ----------------------------------------------------------------------------- sub-benchmarks (N = 1)
def _golden(name):
    p = os.path.join(ROOT, "tests", "golden", name)
    return torch.load(p, weights_only=False) if os.path.exists(p) else None


def dump_codes(out_dir, codes, max_bytes=64 << 20):
    """codes[b]: int64 [T_b, Q] ids of utterance b -> DIR/codes.npy, float32 [B, max T_b, Q], -1 past each T_b.
    Above max_bytes only a fixed, seeded sample of the utterances is written (in batch order).  The inputs are seeded
    and the default decode chain adds its partial sums in fixed order, so two runs with the same arguments write the
    same file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    codes = list(codes)
    row_bytes = max(int(c.shape[0]) for c in codes) * N_Q * 4
    if len(codes) * row_bytes > max_bytes:
        keep = torch.randperm(len(codes), generator=torch.Generator().manual_seed(0))[: max_bytes // row_bytes]
        codes = [codes[i] for i in sorted(keep.tolist())]
    padded = torch.nn.utils.rnn.pad_sequence(codes, batch_first=True, padding_value=-1)
    np.save(os.path.join(out_dir, "codes.npy"), padded.cpu().numpy().astype(np.float32))


def first_divergence(a, b):
    n = min(a.shape[0], b.shape[0])
    bad = (a[:n] != b[:n]).any(dim=1).nonzero()
    return int(bad[0]) if bad.numel() else n


def parity_block(model, dev, bf16_codes_utt0):
    """utterance 0 of the timed bf16 batch carries the inputs of the reference fixture big_full (BASELINE configs[1]:
    S=47, 225-frame prompt; weights = the same default init at seed 0): compare with the reference's codes."""
    g = _golden("big_full.pt")
    if g is None:
        return None
    ref = g["codes"][0].long()
    out = {"fixture": "tests/golden/big_full.pt (generated by the unmodified reference, oracle/gen_golden.py)",
           "frames": int(ref.shape[0]), "reference_min_top2_margin": float(g["min_margin"])}
    eng32 = model.engine(torch.float32)
    eng32.quiet = True
    c32 = eng32.generate([g["x"][0]], [g["y"][0]], top_k=1)[0].cpu()
    out["fp32_exact"] = bool(c32.shape == ref.shape and torch.equal(c32, ref))
    out["fp32_mismatching_ids"] = int((c32 != ref).sum()) if c32.shape == ref.shape else None
    if bf16_codes_utt0 is not None and bf16_codes_utt0.shape == ref.shape:
        b = bf16_codes_utt0.cpu()
        fd = first_divergence(b[:, :1], ref[:, :1])
        out.update(bf16_match_rate=float((b == ref).float().mean()), bf16_match_rate_ar=float((b[:, 0] == ref[:, 0]).float().mean()),
                   first_divergence=fd, first_divergence_any_codebook=first_divergence(b, ref),
                   note="bf16 decodes free-running inside the B=64 batch; after the first near-tie flips an argmax the "
                        "continuation differs by construction (teacher-forced per-step logit errors: "
                        "tests/test_parity_bf16_gpu.py)")
    return out


def parity_mode_block(model, dev, frames, pk):
    """the bit-exact mode (fp32 weights / KV cache / exact-order CUDA-core kernels) timed: 8 utterances per step"""
    B = 8
    eng = model.engine(torch.float32)
    eng.quiet = True
    mnt = None if frames >= FRAMES else frames
    batches = [make_batch(B, 500 + i, dev) for i in range(2)]
    eng.generate(*batches[0], top_k=1, max_new_tokens=mnt, return_device=True)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    eng.generate(*batches[1], top_k=1, max_new_tokens=mnt, return_device=True)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    mean_len = S_TEXT + T_PROMPT + frames / 2.0
    by = ar_step_bytes(B, mean_len, 4)
    step_s = eng.stats.ar_ms / 1000.0 / max(1, eng.stats.ar_steps)
    return {"dtype": "fp32", "batch": B, "value": B * frames * N_Q / (ms / 1000.0), "unit": "tokens/s",
            "ms_per_step": ms, "phase_ms": {"prefill": eng.stats.prefill_ms, "ar": eng.stats.ar_ms, "nar": eng.stats.nar_ms},
            "roofline": {"kernel": "AR decode step, fp32 exact-order kernels", "bound": "hbm", "achieved": by / step_s / 1e9,
                         "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": by / step_s / 1e9 / pk["hbm_gbs"],
                         "algorithmic_bytes_per_launch": by, "launch_seconds": step_s}}


def config2_block(eng, dev, pk, reps=3):
    """BASELINE configs[2]: NAR 7-codebook decode, B=32 x L=1500 (150 phonemes + 225 prompt + 1125 target frames), bf16"""
    B, S, T = 32, 150, 1350
    g = torch.Generator().manual_seed(42)
    texts = [torch.randint(3, 100, (S,), generator=g).to(dev) for _ in range(B)]
    ys = [torch.randint(0, 1024, (T, N_Q), generator=g).to(dev) for _ in range(B)]
    eng.continual(texts, ys)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        out = eng.continual(texts, ys)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    tg = out[0].shape[0]
    fl = 7 * nar_pass_flops(B, S + T, tg)
    return {"workload": f"NAR 7 passes, B={B} x L={S + T} ({S} phonemes + {T - tg} prompt + {tg} target frames), bf16, "
                        "through VALLE.continual's engine path", "ms": ms, "value": B * tg * 7 / (ms / 1000.0),
            "unit": "NAR tokens/s", "roofline": {"bound": "tensor", "achieved": fl / (ms / 1000.0) / 1e12, "peak": pk["tflops"],
                                                 "unit": "TFLOP/s", "frac": fl / (ms / 1000.0) / 1e12 / pk["tflops"],
                                                 "algorithmic_flops": fl}}


def config3_prompts(total, seed=2024):
    g = torch.Generator().manual_seed(seed)
    S = torch.randint(30, 61, (total,), generator=g).tolist()
    texts = [torch.randint(3, 100, (s,), generator=g) for s in S]
    prompts = [torch.randint(0, 1024, (T_PROMPT, N_Q), generator=g) for _ in range(total)]
    return texts, prompts


def config4_block(dev, n_utt=64, chunk=32):
    """BASELINE configs[4] (one GPU's share, bounded sample): EnCodec 24 kHz encode + decode of 10 s waveforms"""
    from valle_b200.data.tokenizer import AudioTokenizer, random_encodec_weights
    tok = AudioTokenizer(device=dev, weights=random_encodec_weights(0))
    g = torch.Generator().manual_seed(5)
    wav = (torch.randn(n_utt, 1, 240000, generator=g) * 0.1).clamp(-1, 1).pin_memory()
    (c, _), = tok.encode(wav[:chunk].to(dev))
    tok.decode([(c, None)])
    torch.cuda.synchronize()
    e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    enc_ms = dec_ms = 0.0
    t0 = time.perf_counter()
    for i in range(0, n_utt, chunk):
        w = wav[i:i + chunk].to(dev, non_blocking=True)
        e[0].record()
        (c, _), = tok.encode(w)
        e[1].record()
        out = tok.decode([(c, None)])
        e[2].record()
        codes_h = c.cpu()
        torch.cuda.synchronize()
        enc_ms += e[0].elapsed_time(e[1])
        dec_ms += e[1].elapsed_time(e[2])
    wall = time.perf_counter() - t0
    return {"workload": f"EnCodec 24 kHz, {n_utt} x 10 s waveforms (bounded sample of this GPU's share of 1000), "
                        f"encode -> [B,8,750] codes -> decode, fp32, random weights, chunks of {chunk}",
            "encode_ms_per_utt": enc_ms / n_utt, "decode_ms_per_utt": dec_ms / n_utt,
            "value": n_utt * 10.0 / wall, "unit": "seconds of audio / s (encode+decode, host waveforms in, codes out)",
            "est_seconds_for_1000_utts_on_this_gpu": 1000 * wall / n_utt, "codes_shape": list(codes_h.shape),
            "wav_out_shape": list(out.shape)}


# ----------------------------------------------------------------------------- main
def main():
    a = parse()
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    import torch.distributed as dist
    frames = a.frames or FRAMES

    if a.impl == "reference":
        # reference arm: the reference's CPU algorithm on the host cores (rank 0 only)
        if world > 1:
            dist.init_process_group("gloo")
            if rank != 0:
                dist.barrier()
                dist.destroy_process_group()
                return
        vals = []
        for i in range(a.warmup + a.steps):
            r = cpu_reference_sample(max(4.0, min(a.cpu_seconds, 30.0)) if i >= a.warmup else 2.0,
                                     one_thread=(i == a.warmup + a.steps - 1))
            if i >= a.warmup:
                vals.append(r)
        best = max(vals, key=lambda r: r["value"])
        v = statistics.median([r["value"] for r in vals])
        line = {"impl": "reference", "metric": "audio tokens/sec (AR+NAR d=1024/12L)", "value": v,
                "unit": "tokens/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": 1000.0 * statistics.median([r["seconds_per_utt"] for r in vals]),
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"AR+NAR infer, S={S_TEXT}, prompt {T_PROMPT} frames -> {FRAMES} frames x 8 "
                                       "codebooks; reference algorithm (no KV cache, batch 1) on host cores; "
                                       "ESTIMATED from a bounded sample of iterations"},
                "cpu_baseline": {"value": v, "unit": "tokens/s", "cores": best["cores"], "kind": "port",
                                 "sample": best["sample"], "estimated": True,
                                 "value_1thread": vals[-1].get("value_1thread"),
                                 "host_threads_available": best["host_threads_available"]},
                "e2e": {"value": v, "unit": "tokens/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    assert torch.cuda.is_available(), "bench.py needs a GPU (there is no CPU fallback for the product path)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from valle_b200 import dist as vdist
    dtype = torch.bfloat16 if a.dtype == "bf16" else torch.float32
    esize = 2 if a.dtype == "bf16" else 4
    model = build_model(dev)
    eng = model.engine(dtype)
    eng.quiet = True
    B = a.batch
    mnt = None if frames >= FRAMES else frames
    extra = (not a.no_extra)
    gold = _golden("big_full.pt") if (extra and rank == 0 and a.dtype == "bf16" and frames == FRAMES) else None

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_step(texts, prompts, e2e):
        if e2e:   # public API, pinned host inputs -> device, one device-side gather, codes -> host
            codes = model.inference_batch(texts, prompts, top_k=1, dtype=dtype, max_new_tokens=mnt,
                                          return_device=world > 1)
            if world > 1:
                codes, base = vdist.gather_codes(codes, N_Q, dev, b_max=B, g_max=B * frames, packed=eng.last_packed,
                                                 return_base=True)
                base_h = base.cpu()                      # one D2H of every rank's codes
                assert base_h.shape[0] == world
            return codes
        codes = eng.generate(texts, prompts, top_k=1, max_new_tokens=mnt, return_device=True)
        if world > 1:
            codes = vdist.gather_codes(codes, N_Q, dev, b_max=B, g_max=B * frames, packed=eng.last_packed)
        return codes

    def timed(e2e, steps, warmup):
        batches = [make_batch(B, 1000 * rank + i, None if e2e else dev, pinned=e2e) for i in range(2)]
        if gold is not None and not e2e:   # utterance 0 of batch 0 = the reference fixture's inputs (same shapes)
            batches[0][0][0] = gold["x"][0].to(dev)
            batches[0][1][0] = gold["y"][0].to(dev)
        for i in range(warmup):
            one_step(*batches[i % 2], e2e)
        barrier()
        n0 = eng.kernel_launches()
        ar_ms = nar_ms = pre_ms = 0.0
        t_wall = time.perf_counter()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        utt0 = codes = None
        ev0.record()
        for i in range(steps):
            codes = one_step(*batches[i % 2], e2e)
            assert len(codes) == B * world
            if i % 2 == 0:
                utt0 = codes[rank * B] if world > 1 else codes[0]
            ar_ms += eng.stats.ar_ms; nar_ms += eng.stats.nar_ms; pre_ms += eng.stats.prefill_ms
        ev1.record()
        barrier()
        ms = ev0.elapsed_time(ev1)
        wall = (time.perf_counter() - t_wall) * 1000.0
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return dict(ms=float(t.item()), wall_ms=wall, launches=eng.kernel_launches() - n0,
                    ar_ms=ar_ms, nar_ms=nar_ms, prefill_ms=pre_ms, steps=eng.stats.ar_steps, utt0=utt0, codes=codes)

    clocks = Clocks(local)
    if rank == 0:
        clocks.start()
    r = timed(False, a.steps, a.warmup)
    clk = clocks.stop() if rank == 0 else None
    if a.dump_outputs and rank == 0:
        dump_codes(a.dump_outputs, r["codes"])
    re = timed(True, a.steps, max(1, min(a.warmup, 1)))

    tokens_step = B * frames * N_Q                     # per GPU per step
    value = world * tokens_step * a.steps / (r["ms"] / 1000.0)
    e2e_value = world * tokens_step * a.steps / (re["ms"] / 1000.0)
    h2d = B * (S_TEXT + T_PROMPT * N_Q) * 8 + 4 * B * (4 + 2 * (S_TEXT + T_PROMPT) + 1)
    d2h = (world if world > 1 else 1) * B * frames * N_Q * 8 + 8 * B

    pk = peaks()
    mean_len = S_TEXT + T_PROMPT + frames / 2.0
    ar_bytes = ar_step_bytes(B, mean_len, esize)
    ar_step_s = (r["ar_ms"] / a.steps) / 1000.0 / max(1, r["steps"])
    ach = ar_bytes / ar_step_s / 1e9
    # DRAM bytes of one decode step from the committed ncu capture (tools/ar_step_traffic.py), if there is one
    traffic, traffic_src = None, None
    for tp in ("round2b_ar_step_traffic_fold.json", "round2_ar_step_traffic.json", "round1_ar_step_traffic.json"):
        tp = os.path.join(ROOT, "profiles", tp)
        if B == 64 and esize == 2 and os.path.exists(tp):
            with open(tp) as f:
                tj = json.load(f)
            traffic = tj["traffic_bytes"]
            traffic_src = (f"profiles/{os.path.basename(tp)}: ncu dram__bytes_read+write over the "
                           f"{tj['kernels_in_step']} kernels of one step at context {tj['context_len']} "
                           f"(algorithmic {tj['algorithmic_bytes']:.4g} B)")
            break
    nar_fl = 7 * nar_pass_flops(B, S_TEXT + T_PROMPT + frames, frames)
    nar_s = (r["nar_ms"] / a.steps) / 1000.0
    line = {
        "metric": "audio tokens/sec (AR+NAR d=1024/12L)", "value": value, "unit": "tokens/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": r["ms"] / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": a.dtype, "data": "synthetic",
        "config": {"workload": f"e2e AR+NAR infer: {B} utterances/GPU x (S={S_TEXT}, {T_PROMPT}-frame prompt) -> "
                               f"{frames} frames x {N_Q} codebooks, greedy, d={D_MODEL}/{N_HEAD}h/{N_LAYER}L",
                   "batch_per_gpu": B, "parallelism": f"dp{world} (independent utterances, one final all-gather)",
                   "l2": "working set (weights + KV cache > 1 GB) exceeds the 126 MB L2; inputs alternate between 2 batches"},
        "gpu_launches": r["launches"],
        "phase_ms_per_step": {"prefill": r["prefill_ms"] / a.steps, "ar": r["ar_ms"] / a.steps,
                              "nar": r["nar_ms"] / a.steps, "ar_decode_steps": r["steps"]},
        "e2e": {"value": e2e_value, "unit": "tokens/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": re["ms"] / a.steps},
        "roofline": {"kernel": "AR decode step (CUDA graph of the PDL-chained projection / KV-cache attention kernels)",
                     "chain": ("LayerNorms folded into the projections, 6 launches per layer"
                               if getattr(eng, "ar_head_fold", None) is not None else "8 launches per layer"),
                     "bound": "hbm", "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s",
                     "frac": ach / pk["hbm_gbs"], "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": pk["source"],
                     "algorithmic_bytes_per_launch": ar_bytes, "launch_seconds": ar_step_s},
        "roofline_nar": {"kernel": "7 NAR passes (QKV/out/FFN GEMMs + attention + heads)", "bound": "tensor",
                         "achieved": nar_fl / nar_s / 1e12 if nar_s > 0 else None, "peak": pk["tflops"],
                         "unit": "TFLOP/s", "frac": (nar_fl / nar_s / 1e12 / pk["tflops"]) if nar_s > 0 else None},
        "clocks": clk,
    }
    # ---- BASELINE configs[3]: a fixed list of prompts sharded over the ranks (strong scaling), every N ----
    if extra and a.total_prompts > 0:
        texts3, prompts3 = config3_prompts(a.total_prompts)
        lo, hi = vdist.shard_range(a.total_prompts, rank, world)

        # within a rank the prompts are decoded longest-first, so that the utterances of one batch stop together
        order = sorted(range(lo, hi), key=lambda u: -texts3[u].numel())

        def job():
            outs = [None] * (hi - lo)
            for b0 in range(0, len(order), B):
                ids = order[b0:b0 + B]
                c = eng.generate([texts3[u].to(dev) for u in ids], [prompts3[u].to(dev) for u in ids], top_k=1,
                                 max_new_tokens=mnt, return_device=True)
                for u, cu in zip(ids, c):
                    outs[u - lo] = cu
            if world > 1:
                outs = vdist.gather_codes(outs, N_Q, dev)
            return outs

        job()                                   # warm-up: graphs of these shapes are captured here
        barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        outs = job()
        ev1.record()
        barrier()
        t = torch.tensor([ev0.elapsed_time(ev1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        assert len(outs) == a.total_prompts
        toks = sum(int(o.shape[0]) for o in outs) * N_Q
        line["config3"] = {"workload": f"{a.total_prompts} prompts (S~U[30,60], {T_PROMPT}-frame prompt, cap-terminated), "
                                       f"contiguous shards of {hi - lo} per GPU decoded in batches of <= {B}, one all-gather",
                           "scaling": "strong", "value": toks / (float(t.item()) / 1000.0), "unit": "tokens/s",
                           "ms": float(t.item()), "tokens": toks, "prompts_per_gpu": hi - lo}
    if rank == 0 and a.gpus == 1 and extra:
        if gold is not None:
            line["parity"] = parity_block(model, dev, r["utt0"])
        # BASELINE.json configs[1]: batch-1 greedy AR decode latency (p50 over 3 utterances)
        if not a.no_latency:
            lat, ar1 = [], []
            t1, p1 = make_batch(1, 77, dev)
            eng.generate(t1, p1, top_k=1, max_new_tokens=mnt, return_device=True)
            for i in range(3):
                t1, p1 = make_batch(1, 78 + i, dev)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                eng.generate(t1, p1, top_k=1, max_new_tokens=mnt, return_device=True)
                torch.cuda.synchronize()
                lat.append((time.perf_counter() - t0) * 1000.0)
                ar1.append(eng.stats.ar_ms / max(1, eng.stats.ar_steps))
            b1 = ar_step_bytes(1, mean_len, esize)
            s1 = statistics.median(ar1) / 1000.0
            line["p50_utt_latency_ms"] = statistics.median(lat)
            line["roofline_b1"] = {"kernel": "AR decode step, batch 1", "bound": "hbm", "achieved": b1 / s1 / 1e9,
                                   "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": b1 / s1 / 1e9 / pk["hbm_gbs"],
                                   "ar_tokens_per_s": 1.0 / s1}
        if a.dtype == "bf16":
            line["config2"] = config2_block(eng, dev, pk)
            line["parity_mode"] = parity_mode_block(model, dev, frames, pk)
        try:
            line["config4"] = config4_block(dev)
        except Exception as ex:  # the codec is a separate row of the scope table: never lose the headline line over it
            line["config4"] = {"error": repr(ex)[:300]}
    if rank == 0 and a.gpus == 1 and not a.no_cpu_baseline and extra:
        cb = cpu_reference_sample(a.cpu_seconds)
        line["cpu_baseline"] = {"value": cb["value"], "unit": "tokens/s", "cores": cb["cores"], "kind": "port",
                                "estimated": True, "sample": cb["sample"], "value_1thread": cb.get("value_1thread"),
                                "sample_1thread": cb.get("sample_1thread"),
                                "host_threads_available": cb["host_threads_available"]}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
