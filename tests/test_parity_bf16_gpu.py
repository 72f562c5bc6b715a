"""GPU parity tests of the BENCHMARKED mode (bf16 weights / KV cache, tcgen05 projections, CUDA-graph decode step)
against the fp32 reference, plus sampling, stop-rule and boundary checks.

bf16 cannot be bit-exact with an fp32 reference over hundreds of dependent argmaxes (random-init logits have top-2
margins down to 6e-5, bf16 logits carry ~1e-2 of rounding noise), so the bars are:
  * teacher-forced (every appended id = the reference's id): max |logit error| per AR step and per NAR stage below a
    stated tolerance, and the bf16 argmax differs from the reference's id ONLY where the reference's own top-2 margin
    is below twice that error -- i.e. every disagreement is a near-tie, never a wrong distribution;
  * free-running: token-match rate and first-divergence step are measured and reported (gpurun_out/parity_bf16.json,
    bench.py "parity"), with a floor that catches a broken path.
fp32 mode stays bit-exact (tests/test_parity_gpu.py)."""
import json
import os

import pytest
import torch

from conftest import ROOT, assert_checksums, build_model, load_golden
from oracle import valle_oracle as O

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
AR_TOL = 0.03      # max abs logit error of a bf16 AR step vs the fp32 reference (AR logits: std 0.58, |max| 2.4;
                   # measured 0.0099 over the 754 steps of configs[1], profiles/round2_parity_bf16.json)
NAR_TOL_REL = 0.03  # NAR stages: max abs error relative to the standard deviation of that stage's reference logits
                    # (stages 0..5 project onto the N(0,1)-initialised tied embedding tables: std ~25, |max| ~95;
                    # the untied last stage: std 0.5)


def _model(g, dtype):
    m = build_model(g["config"], g["weight_seed"])
    assert_checksums(m, g["checksums"])
    m = m.to(DEV)
    m.engine_dtype = dtype
    m.engine().quiet = True
    return m


def _report(name, rec):
    out = os.path.join(ROOT, "gpurun_out")
    os.makedirs(out, exist_ok=True)
    p = os.path.join(out, "parity_bf16.json")
    cur = {}
    if os.path.exists(p):
        try:
            cur = json.load(open(p))
        except Exception:
            cur = {}
    cur[name] = rec
    with open(p, "w") as f:
        json.dump(cur, f, indent=1, sort_keys=True)


def _first_div(a, b):
    """first frame at which two [T, Q] code matrices differ (T if none)"""
    n = min(a.shape[0], b.shape[0])
    bad = (a[:n] != b[:n]).any(dim=1).nonzero()
    return int(bad[0]) if bad.numel() else n


def _teacher_forced(g, dtype):
    m = _model(g, dtype)
    eng = m.engine()
    ref = g["codes"][0].long()
    tr = {"steps": "all", "nar": True}
    out = eng.generate([g["x"][0]], [g["y"][0]], top_k=1, trace=tr, forced=[ref])[0].cpu()
    n = ref.shape[0]
    ar = torch.stack([tr["ar_logits"][i][0].cpu() for i in range(n + 1)])          # [n+1, 1025] (last = stop step)
    nar = [t.cpu() for t in tr["nar_logits"]]                                      # 7 x [n, 1024]
    nar_arg = [t.cpu() for t in tr["nar_argmax"]]
    return out, ar, nar, nar_arg


def test_bf16_teacher_forced_logits_vs_fp32_oracle_big_short():
    """d=1024/16h/12L, 97 frames: every AR step and every NAR stage of the bf16 tensor-core path against the CPU
    oracle (the reference's algorithm, fp32), teacher-forced with the reference's own ids."""
    g = load_golden("big_short.pt")
    m32 = build_model(g["config"], g["weight_seed"])
    sd = {k: v.detach() for k, v in m32.state_dict().items()}
    c = g["config"]
    cfg = O.OracleConfig(c["d_model"], c["nhead"], c["num_layers"], c["prefix_mode"], c["num_quantizers"])
    x, y = g["x"], g["y"]
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    tr = O.InferenceTrace([], [], [], [])
    with torch.no_grad():
        ref_codes = O.inference(sd, cfg, x, xl, y, None, top_k=1, trace=tr)
    assert torch.equal(ref_codes, g["codes"].long())          # the oracle reproduces the reference fixture
    ref_ar = torch.stack(tr.ar_logits)                          # [n+1, 1025]
    out, ar, nar, nar_arg = _teacher_forced(g, torch.bfloat16)
    ref = g["codes"][0].long()
    assert torch.equal(out, ref)                                # forced ids come back unchanged
    n = ref.shape[0]
    err = (ar - ref_ar).abs().amax(dim=1)                       # per AR step
    assert float(err.max()) < AR_TOL, float(err.max())
    margin = torch.tensor(tr.ar_margin)
    flips = ar[:n].argmax(dim=1) != ref[:, 0]
    assert not bool((flips & (margin[:n] > 2 * err[:n])).any()), "bf16 argmax differs where the reference is not a near-tie"
    nerr = []
    for i in range(7):
        e = (nar[i] - tr.nar_logits[i]).abs().amax(dim=1)       # per frame
        scale = float(tr.nar_logits[i].std())
        nerr.append(float(e.max()) / scale)
        assert float(e.max()) < NAR_TOL_REL * scale, (i, float(e.max()), scale)
        f = nar_arg[i] != ref[:, i + 1]
        assert not bool((f & (tr.nar_margin[i] > 2 * e)).any()), f"NAR stage {i}: flip outside a near-tie"
    _report("big_short_teacher_forced", dict(ar_max_abs_err=float(err.max()), ar_mean_abs_err=float(err.mean()),
                                              ar_argmax_flips=int(flips.sum()), ar_steps=n, nar_max_err_over_std=nerr,
                                              nar_argmax_flips=[int((nar_arg[i] != ref[:, i + 1]).sum()) for i in range(7)]))


def test_bf16_teacher_forced_vs_fp32_engine_config1():
    """BASELINE configs[1] (S=47, 225-frame prompt -> 753 frames): the reference needs 665 s for this utterance on the
    host, so the per-step fp32 logits come from the fp32 engine, itself bit-exact in ids with the reference fixture
    and within 2e-4 of the oracle's logits (tests/test_parity_gpu.py); the three logit rows the fixture stores pin it."""
    g = load_golden("big_full.pt")
    ref = g["codes"][0].long()
    out32, ar32, nar32, _ = _teacher_forced(g, torch.float32)
    assert torch.equal(out32, ref)
    for i, s in enumerate(g["ar_logit_steps"].tolist()):       # fp32 engine vs the reference's stored rows
        assert torch.allclose(ar32[s], g["ar_logits"][i], atol=3e-4, rtol=0), (s, (ar32[s] - g["ar_logits"][i]).abs().max())
    assert bool((ar32[: ref.shape[0]].argmax(dim=1) == ref[:, 0]).all())   # teacher-forced fp32 argmax == reference ids
    torch.cuda.empty_cache()
    out, ar, nar, nar_arg = _teacher_forced(g, torch.bfloat16)
    n = ref.shape[0]
    err = (ar - ar32).abs().amax(dim=1)
    assert float(err.max()) < AR_TOL, float(err.max())
    margin = g["ar_margin"]
    flips = ar[:n].argmax(dim=1) != ref[:, 0]
    assert not bool((flips & (margin[:n] > 2 * err[:n] + 6e-4)).any())
    nerr = []
    for i in range(7):
        e = (nar[i] - nar32[i]).abs().amax(dim=1)
        scale = float(nar32[i].std())
        nerr.append(float(e.max()) / scale)
        assert float(e.max()) < NAR_TOL_REL * scale, (i, float(e.max()), scale)
        f = nar_arg[i] != ref[:, i + 1]
        assert not bool((f & (g["nar_margin"][i] > 2 * e + 6e-4)).any()), f"NAR stage {i}: flip outside a near-tie"
    _report("config1_teacher_forced", dict(ar_max_abs_err=float(err.max()), ar_mean_abs_err=float(err.mean()),
                                            ar_argmax_flips=int(flips.sum()), ar_steps=n, nar_max_err_over_std=nerr,
                                            nar_argmax_flips=[int((nar_arg[i] != ref[:, i + 1]).sum()) for i in range(7)]))


@pytest.mark.parametrize("name", ["big_short.pt", "config0.pt", "big_full.pt"])
def test_bf16_free_running_match_rate(name):
    """The benchmarked configuration end to end (CUDA-graph decode step, greedy, bf16) against the reference codes:
    token-match rate and first divergence are measured; a correct bf16 path follows the reference until the first
    near-tie flips an argmax (random-init margins are ~1e-4, bf16 logit noise ~1e-2) and produces valid codes of the
    reference's length throughout."""
    g = load_golden(name)
    m = _model(g, torch.bfloat16)
    ref = g["codes"][0].long()
    x, y = g["x"].to(DEV), g["y"].to(DEV)
    out = m.inference(x, torch.tensor([x.shape[1]], dtype=torch.int32), y, None, top_k=1)[0].cpu()
    assert out.shape == ref.shape and int(out.min()) >= 0 and int(out.max()) < 1024
    fd_ar = _first_div(out[:, :1], ref[:, :1])
    rec = dict(frames=int(ref.shape[0]), first_divergence_ar=fd_ar, first_divergence_any=_first_div(out, ref),
               match_rate_ar=float((out[:, 0] == ref[:, 0]).float().mean()),
               match_rate_all=float((out == ref).float().mean()),
               match_rate_before_divergence=float((out[:fd_ar] == ref[:fd_ar]).float().mean()) if fd_ar else None,
               reference_min_margin=float(g["min_margin"]))
    _report("free_running_" + name[:-3], rec)
    assert fd_ar >= 1, rec                              # the very first id (margin-checked in the fixtures) agrees
    if fd_ar > 0:   # NAR codes of the frames decoded from an identical AR prefix mostly agree too
        assert rec["match_rate_before_divergence"] > 0.5, rec


def test_topk_sampling_matches_reference_at_fixed_seed():
    """valle.py:1040-1043,1287-1302: top-k / temperature sampling.  With the draw done on the host exactly as the
    reference does it (torch's CPU generator, one multinomial per token) the fp32 engine reproduces the reference's
    ids at the same torch seed, for top_k > 1, for the unfiltered default (top_k=-100) and with temperature."""
    g = load_golden("tiny_topk.pt")
    m = _model(g, torch.float32)
    eng = m.engine()
    eng.sample_on_host = True
    x, y = g["x"].to(DEV), g["y"].to(DEV)
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    for c in g["cases"]:
        torch.manual_seed(int(c["torch_seed"]))
        out = m.inference(x, xl, y, None, top_k=int(c["top_k"]), temperature=float(c["temperature"])).cpu()
        ref = c["codes"].long()
        assert out.shape == ref.shape, (c["top_k"], out.shape, ref.shape)
        assert torch.equal(out, ref), (c["top_k"], int((out != ref).sum()))


def test_topk_filter_and_device_draw_follow_the_reference_semantics():
    """Device-side sampling (the default): (1) the filtered distribution equals oracle.top_k_top_p_filtering of the
    same logits (same -inf set, ties with the k-th value kept, valle.py:1259); (2) under a fixed CUDA seed the ids the
    engine draws are exactly torch.multinomial(softmax(filtered)) of its own per-step logits -- one draw per token, in
    order, from the device generator, which is what the reference's topk_sampling does on a CUDA tensor."""
    from valle_b200.models.valle import top_k_top_p_filtering, topk_sampling
    g = load_golden("tiny_pm1.pt")
    m = _model(g, torch.float32)
    eng = m.engine()
    torch.manual_seed(3)
    lg = torch.randn(4, 1025)
    lg[1, 7] = lg[1].topk(5)[0][-1]                       # a tie with the k-th value must survive
    for k in (1, 5, 1025, -100):
        a = top_k_top_p_filtering(lg.clone().to(DEV), top_k=k).cpu()
        b = O.top_k_top_p_filtering(lg.clone(), top_k=k)
        assert torch.equal(a, b), k
    # replay: record the logits of every step of a sampled decode, then redraw from them under the same seed
    x, y = g["x"][0], g["y"][0]
    torch.cuda.manual_seed(11)
    tr = {"steps": "all"}
    out = eng.generate([x], [y], top_k=5, temperature=0.8, max_new_tokens=20, trace=tr)[0]
    torch.cuda.manual_seed(11)
    n = out.shape[0]
    redraw = [int(topk_sampling(tr["ar_logits"][i].clone(), top_k=5, temperature=0.8)) for i in range(n)]
    assert redraw == out[:, 0].tolist()
    assert 1 <= n <= 20 and int(out.min()) >= 0 and int(out.max()) < 1024


def test_finished_rows_leave_their_kv_cache_untouched():
    """Ragged batch: utterances that hit their cap early keep riding through the batched decode step.  Their KV cache
    rows must not change after they stopped (the scatter and attention kernels skip finished rows) and the codes of
    every utterance must equal its batch-1 decode."""
    g = load_golden("tiny_batch.pt")
    for dtype in (torch.float32, torch.bfloat16):
        m = _model(g, dtype)
        eng = m.engine()
        texts = [u["x"][0] for u in g["utts"]]
        prompts = [u["y"][0] for u in g["utts"]]
        S = [t.numel() for t in texts]
        outs = eng.generate(texts, prompts, top_k=1)
        buf = next(iter(eng._bufs.values()))
        short = min(range(len(S)), key=lambda b: S[b])
        long_ = max(range(len(S)), key=lambda b: S[b])
        assert outs[short].shape[0] < outs[long_].shape[0]
        k_after = buf.kcache[:, short].clone()
        # decode the short utterance alone: its cache must be identical over the rows it really wrote
        eng._bufs.clear()
        solo = eng.generate([texts[short]], [prompts[short]], top_k=1)[0]
        assert torch.equal(solo, outs[short])
        buf1 = next(iter(eng._bufs.values()))
        n_rows = S[short] + prompts[short].shape[0] + outs[short].shape[0]
        a = k_after[:, :, :n_rows].float()
        b = buf1.kcache[:, 0, :, :n_rows].float()
        # the batched and the batch-1 decode use different reduction orders (fp32: 4-row vs 1-row GEMV; bf16: tensor
        # cores vs the persistent small-batch kernel); a finished row overwritten by later steps would be off by O(1)
        tol = 1e-5 if dtype == torch.float32 else 0.05
        assert float((a - b).abs().max()) <= tol
        assert bool(torch.isfinite(buf.x_cur).all())
        if dtype == torch.float32:
            for u, o in zip(g["utts"], outs):
                assert torch.equal(o.cpu(), u["codes"][0].long())


def test_out_of_range_ids_raise_index_error():
    """nn.Embedding's contract (embedding.py:46): ids outside the table raise IndexError, on host and device inputs."""
    g = load_golden("tiny_pm1.pt")
    m = _model(g, torch.float32)
    x, y = g["x"].clone(), g["y"].clone()
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    bad = x.clone()
    bad[0, 2] = 512
    with pytest.raises(IndexError):
        m.inference(bad, xl, y, None, top_k=1, max_new_tokens=4)
    with pytest.raises(IndexError):
        m.inference(bad.to(DEV), xl, y.to(DEV), None, top_k=1, max_new_tokens=4)
    bady = y.clone()
    bady[0, 3, 5] = 1024           # EOS is not a valid prompt code for nar_audio_embeddings[1..7]
    with pytest.raises(IndexError):
        m.inference(x.to(DEV), xl, bady.to(DEV), None, top_k=1, max_new_tokens=4)
    out = m.inference(x.to(DEV), xl, y.to(DEV), None, top_k=1, max_new_tokens=4)   # the engine is still usable
    assert out.shape == (1, 4, 8)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_model_on_second_gpu_while_first_is_current():
    """kernels, streams and per-device function attributes follow the model's device, not the current device"""
    g = load_golden("tiny_pm1.pt")
    m = build_model(g["config"], g["weight_seed"]).to("cuda:1")
    m.engine().quiet = True
    torch.cuda.set_device(0)
    x, y = g["x"].to("cuda:1"), g["y"].to("cuda:1")
    out = m.inference(x, torch.tensor([x.shape[1]], dtype=torch.int32), y, None, top_k=1).cpu()
    assert torch.equal(out, g["codes"].long())
    m.engine_dtype = torch.bfloat16
    m.engine().quiet = True
    out = m.inference(x, torch.tensor([x.shape[1]], dtype=torch.int32), y, None, top_k=1, max_new_tokens=12).cpu()
    assert out.shape == (1, 12, 8)


def test_bf16_batches_above_64_are_decoded_in_tensor_core_groups():
    """B = 70 > 64 (one UMMA N tile): the engine decodes groups of <= 64 rows on the tensor-core chain instead of
    dropping onto the CUDA-core GEMV path; every utterance equals its decode inside a batch of <= 64."""
    g = load_golden("tiny_batch.pt")
    m = _model(g, torch.bfloat16)
    eng = m.engine()
    texts = ([u["x"][0] for u in g["utts"]] * 18)[:70]
    prompts = ([u["y"][0] for u in g["utts"]] * 18)[:70]
    n0 = eng.kernel_launches()
    out = eng.generate(texts, prompts, top_k=1, max_new_tokens=12, return_device=True)
    assert len(out) == 70 and eng.last_packed.shape == (70 * 12, 8)
    ref = eng.generate(texts[:4], prompts[:4], top_k=1, max_new_tokens=12)
    for i in range(70):
        assert torch.equal(out[i].cpu(), ref[i % 4]), i


# ---------------------------------------------------------------- LayerNorm-folded decode chain (vb_ln_fold)
def test_ln_fold_build_matches_its_definition():
    """vb_ln_fold_build: wf = bf16(W * gamma), c = row sums of wf, dvec = bias + W @ beta (include/valle_b200.h)"""
    import ctypes as C
    from valle_b200 import _lib as L
    lib = L.load()
    g = torch.Generator().manual_seed(11)
    N, K = 300, 256
    W = (torch.randn(N, K, generator=g) / 16).bfloat16()
    gamma, beta, bias = 1 + 0.1 * torch.randn(K, generator=g), 0.1 * torch.randn(K, generator=g), torch.randn(N, generator=g)
    Wd, gd, bd, biasd = W.to(DEV), gamma.to(DEV), beta.to(DEV), bias.to(DEV)
    wf = torch.empty_like(Wd)
    c = torch.empty(N, device=DEV)
    dv = torch.empty(N, device=DEV)
    L.check(lib.vb_ln_fold_build(Wd.data_ptr(), N, K, gd.data_ptr(), bd.data_ptr(), biasd.data_ptr(), wf.data_ptr(),
                                 c.data_ptr(), dv.data_ptr(), L.stream_ptr()))
    torch.cuda.synchronize()
    wf_ref = (W.float() * gamma).bfloat16()
    assert torch.equal(wf.cpu(), wf_ref)
    assert torch.allclose(c.cpu(), wf_ref.float().sum(1), atol=1e-4, rtol=1e-5)
    assert torch.allclose(dv.cpu(), bias + W.float() @ beta, atol=1e-4, rtol=1e-5)


@pytest.mark.parametrize("name", ["tiny_batch.pt", "big_short.pt"])
def test_folded_decode_chain_matches_the_unfolded_chain(name, monkeypatch):
    """The bf16 decode step with the LayerNorms folded into the projections (6 launches per layer: fp32-fed
    projections carrying the rows' moments, residual stream assembled by bulk reductions) against the chain with the
    separate residual + LayerNorm launches on the same weights: per-step logits within 2e-2 (both round to bf16 at
    different points) and the same early greedy ids.  The folded chain runs on request (VB_DECODE_FOLD=1)."""
    from valle_b200 import _lib as L
    lib = L.load()
    g = load_golden(name)
    monkeypatch.setenv("VB_DECODE_FOLD", "1")
    m = _model(g, torch.bfloat16)
    eng = m.engine()
    assert eng.ar_head_fold is not None, "VB_DECODE_FOLD=1 must turn the LayerNorm-folded chain on in bf16"
    if "utts" in g:
        texts = [u["x"][0] for u in g["utts"]] * 3
        prompts = [u["y"][0] for u in g["utts"]] * 3
    else:
        texts, prompts = [g["x"][0]] * 3, [g["y"][0]] * 3
    steps = {0, 1, 2, 7, 15}
    tr_f = {"steps": steps}
    out_f = eng.generate(texts, prompts, top_k=1, trace=tr_f, max_new_tokens=16)
    L.check(lib.vb_tune_set(b"VB_DECODE_FOLD", 0))
    try:
        eng._bufs.clear()
        tr_u = {"steps": steps}
        out_u = eng.generate(texts, prompts, top_k=1, trace=tr_u, max_new_tokens=16)
    finally:
        L.check(lib.vb_tune_set(b"VB_DECODE_FOLD", 1))
        eng._bufs.clear()
    for s in sorted(steps):
        err = (tr_f["ar_logits"][s] - tr_u["ar_logits"][s]).abs().max().item()
        assert err < 2e-2, (s, err)
    agree = sum(int((a[:6, 0] == b[:6, 0]).all()) for a, b in zip(out_f, out_u))
    assert agree >= len(out_f) - 1, agree
