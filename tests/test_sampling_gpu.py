"""GPU tests of seeded top-k / temperature sampling inside the graph-replayed AR decode step (generate(seeds=...)):
the sampler kernel draws what the restatement in tests/sampling_oracle.py draws from the same logits, an utterance's
codes depend only on its own seed, and the decode runs as CUDA-graph replays without a host-side draw."""
import numpy as np
import pytest
import torch

import sampling_oracle as SO
from conftest import load_golden
from oracle import valle_oracle as O
from test_parity_gpu import DEV, _model

pytestmark = pytest.mark.gpu

EOS = O.NUM_AUDIO_TOKENS
SEEDS3 = [11, 2 ** 64 - 5, 123456789]


def _oracle_cfg(g):
    c = g["config"]
    return O.OracleConfig(c["d_model"], c["nhead"], c["num_layers"], c["prefix_mode"], c["num_quantizers"])


def _cpu_sd(m):
    return {k: v.detach().cpu().clone() for k, v in m.state_dict().items()}


def _batch(n):
    g = load_golden("tiny_batch.pt")
    utts = g["utts"]
    return g, [utts[i % len(utts)]["x"][0] for i in range(n)], [utts[i % len(utts)]["y"][0] for i in range(n)]


def _engine(g, dtype, fold=False):
    m = _model(g, dtype)
    eng = m.engine()
    eng.quiet = True
    if fold:
        eng.use_decode_fold, eng._sig = True, None
        eng._refresh()
        assert eng.ar_head_fold is not None
    return eng


def _check_draws(codes, trace, seeds, ks, ts, S, max_new):
    """walk every utterance through the traced logits: each appended id is the restatement's draw at that step, and the
    utterance stops where the restated stop rule says.  Returns the excused disagreements (top-two keys within 1e-5)."""
    excused = []
    for b in range(len(codes)):
        n = 0
        cap = min(16 * S[b], max_new - 1)
        for t in sorted(trace):
            row = trace[t][b].cpu()
            want = SO.seeded_draw(row, seeds[b], n, ks[b], ts[b])
            stop = int(torch.argmax(row)) == EOS or want == EOS or n > cap
            got_stop = n == codes[b].shape[0]
            got = None if got_stop else int(codes[b][n, 0])
            if stop != got_stop or (not stop and got != want):
                gap = SO.key_gap(row, seeds[b], n, ks[b], ts[b])
                assert gap < 1e-5, (b, t, n, want, got, stop, got_stop, gap)
                excused.append((b, n, gap))
                if got_stop:
                    break
            elif stop:
                break
            n += 1
        assert n == codes[b].shape[0] or excused, (b, n, codes[b].shape[0])
    return excused


@pytest.mark.parametrize("chain", ["fp32", "bf16", "bf16_fold"])
@pytest.mark.parametrize("params", [([5, -100, 5], [1.0, 1.0, 0.8]), ([-100, 5, -100], [0.8, 0.8, 1.0])])
def test_kernel_draws_equal_the_restatement(chain, params):
    dtype = torch.float32 if chain == "fp32" else torch.bfloat16
    g, texts, prompts = _batch(3)
    eng = _engine(g, dtype, fold=chain == "bf16_fold")
    ks, ts = params
    tr = {"steps": "all"}
    max_new = 40
    out = eng.generate(texts, prompts, top_k=ks, temperature=ts, seeds=SEEDS3, max_new_tokens=max_new, trace=tr)
    excused = _check_draws(out, tr["ar_logits"], SEEDS3, ks, ts, [t.numel() for t in texts], max_new)
    print(f"{chain}: {sum(o.shape[0] for o in out)} draws, {len(excused)} near-tie disagreements {excused}")
    assert all(0 <= int(o.min()) and int(o.max()) < 1024 for o in out if o.numel())


@pytest.mark.parametrize("name", ["tiny_pm1.pt", "tiny_bos.pt"])
def test_fp32_seeded_inference_equals_the_oracle(name):
    g = load_golden(name)
    m = _model(g)
    m.engine().quiet = True
    sd = _cpu_sd(m)
    x, y = g["x"], g["y"]
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    bos = bool(g["config"].get("prepend_bos", False))
    n_ok = 0
    for seed in (3, 2 ** 63 + 17, 99):
        try:
            want = SO.inference(sd, _oracle_cfg(g), x, xl, y, None, top_k=5, temperature=0.8, seed=seed,
                                max_new_tokens=48, prepend_bos=bos)
        except SyntaxError:
            with pytest.raises(SyntaxError):
                m.inference(x.to(DEV), xl, y.to(DEV), None, top_k=5, temperature=0.8, max_new_tokens=48, seed=seed)
            continue
        got = m.inference(x.to(DEV), xl, y.to(DEV), None, top_k=5, temperature=0.8, max_new_tokens=48, seed=seed).cpu()
        assert torch.equal(got, want), (seed, got.shape, want.shape)
        n_ok += 1
    assert n_ok >= 1


def test_seeded_top_k_one_is_greedy():
    g, texts, prompts = _batch(4)
    for dtype in (torch.float32, torch.bfloat16):
        eng = _engine(g, dtype)
        greedy = eng.generate(texts, prompts, top_k=1, max_new_tokens=40)
        seeded = eng.generate(texts, prompts, top_k=1, temperature=0.7, seeds=[1, 2, 3, 4], max_new_tokens=40)
        assert all(torch.equal(a, b) for a, b in zip(greedy, seeded)), dtype


def test_batch_invariance():
    g, texts, prompts = _batch(4)
    eng = _engine(g, torch.float32)
    seeds = [5, 6, 77, 8]
    alone = eng.generate([texts[2]], [prompts[2]], top_k=-100, temperature=1.0, seeds=[77], max_new_tokens=40)[0]
    batch = eng.generate(texts, prompts, top_k=-100, temperature=1.0, seeds=seeds, max_new_tokens=40)
    assert torch.equal(alone, batch[2])
    # bf16: identical utterances with the same seed decode identically, in one batch and on a repeated call
    eng = _engine(g, torch.bfloat16)
    t2, p2 = [texts[1], texts[0], texts[1]], [prompts[1], prompts[0], prompts[1]]
    a = eng.generate(t2, p2, top_k=-100, temperature=1.0, seeds=[42, 7, 42], max_new_tokens=40)
    b = eng.generate(t2, p2, top_k=-100, temperature=1.0, seeds=[42, 7, 42], max_new_tokens=40)
    assert torch.equal(a[0], a[2])
    assert all(torch.equal(u, v) for u, v in zip(a, b))
    c = eng.generate(t2, p2, top_k=-100, temperature=1.0, seeds=[43, 7, 44], max_new_tokens=40)
    assert not torch.equal(c[0], a[0]) and not torch.equal(c[2], a[2])


def test_bf16_groups_above_64_keep_each_utterance_s_seed():
    g, texts, prompts = _batch(70)
    eng = _engine(g, torch.bfloat16)
    seeds = [1000 + 3 * i for i in range(70)]
    ks = [5 if i % 2 else -100 for i in range(70)]
    ts = [0.8 if i % 3 else 1.0 for i in range(70)]
    full = eng.generate(texts, prompts, top_k=ks, temperature=ts, seeds=seeds, max_new_tokens=24)
    lo = eng.generate(texts[:64], prompts[:64], top_k=ks[:64], temperature=ts[:64], seeds=seeds[:64], max_new_tokens=24)
    hi = eng.generate(texts[64:], prompts[64:], top_k=ks[64:], temperature=ts[64:], seeds=seeds[64:], max_new_tokens=24)
    assert all(torch.equal(a, b) for a, b in zip(full, lo + hi))


def test_seeded_decode_runs_in_the_graph(monkeypatch):
    from valle_b200 import _lib as L
    lib = L.load()
    g, texts, prompts = _batch(2)
    eng = _engine(g, torch.float32)
    kw = dict(top_k=5, temperature=0.8, seeds=[21, 22])

    def no_push(*a):
        raise AssertionError("vb_ar_push_tokens called on the seeded path")
    monkeypatch.setattr(lib, "vb_ar_push_tokens", no_push)

    eng.use_cuda_graph = False
    eager = eng.generate(texts, prompts, max_new_tokens=40, **kw)
    eng.use_cuda_graph = True
    graph = eng.generate(texts, prompts, max_new_tokens=40, **kw)
    assert all(torch.equal(a, b) for a, b in zip(eager, graph))

    # direct launches of a warm call (graphs captured) do not grow with the number of decode steps
    counts = {}
    for mnt in (16, 48):
        eng.generate(texts, prompts, max_new_tokens=mnt, **kw)       # capture at this shape
        n0, r0 = lib.vb_launch_count(), eng.replayed_launches
        eng.generate(texts, prompts, max_new_tokens=mnt, **kw)
        counts[mnt] = (lib.vb_launch_count() - n0, eng.stats.ar_steps, eng.replayed_launches - r0)
    (d16, s16, r16), (d48, s48, r48) = counts[16], counts[48]
    assert s48 > s16, counts           # more steps ...
    assert r48 > r16 > 0, counts       # ... all of them graph replays ...
    assert d48 == d16, counts          # ... and no extra direct launches


def test_sampled_eos_at_step_zero_raises():
    g = load_golden("tiny_pm1.pt")
    m = _model(g)
    eng = m.engine()
    eng.quiet = True
    x, y = g["x"][0], g["y"][0]
    tr = {"steps": {0}}
    eng.generate([x], [y], top_k=1, max_new_tokens=4, trace=tr)
    row = tr["ar_logits"][0][0].cpu()
    assert int(torch.argmax(row)) != EOS
    seeds = np.arange(20_000, dtype=np.uint64)
    draws = SO.seeded_draw(row, seeds, np.zeros_like(seeds), -100, 20.0)
    cand = [int(s) for s in seeds[draws == EOS]]
    cand = [s for s in cand if SO.key_gap(row, s, 0, -100, 20.0) > 1e-3]
    assert cand, "no seed draws EOS at step 0"
    with pytest.raises(SyntaxError, match="well trained model shouldn't reach here."):
        eng.generate([x], [y], top_k=-100, temperature=20.0, seeds=[cand[0]], max_new_tokens=4)
    # a seed whose step-0 draw is not EOS decodes
    ok = next(int(s) for s in seeds[draws != EOS][:1])
    assert eng.generate([x], [y], top_k=-100, temperature=20.0, seeds=[ok], max_new_tokens=4)[0].shape[0] >= 1


def test_invalid_seeded_arguments_raise_value_error():
    g, texts, prompts = _batch(2)
    eng = _engine(g, torch.float32)
    with pytest.raises(ValueError):
        eng.generate(texts, prompts, top_k=5, seeds=[1])                              # len(seeds) != B
    with pytest.raises(ValueError):
        eng.generate(texts, prompts, top_k=5, seeds=[1, -1])                          # seed outside [0, 2**64)
    for bad_t in (0.0, -1.0, float("inf"), float("nan")):
        with pytest.raises(ValueError):
            eng.generate(texts, prompts, top_k=5, temperature=bad_t, seeds=[1, 2])
    with pytest.raises(ValueError):
        eng.generate(texts, prompts, top_k=[5, 5], temperature=1.0)                   # per-utterance without seeds
    with pytest.raises(ValueError):
        eng.generate(texts, prompts, top_k=5, temperature=[1.0, 0.9])
    with pytest.raises(ValueError):
        eng.generate(texts, prompts, top_k=[5, 5, 5], seeds=[1, 2])                   # wrong length
    eng.sample_on_host = True
    try:
        with pytest.raises(ValueError):
            eng.generate(texts, prompts, top_k=5, seeds=[1, 2])
    finally:
        eng.sample_on_host = False
    forced = [torch.zeros((4, 8), dtype=torch.int64)] * 2
    with pytest.raises(ValueError):
        eng.generate(texts, prompts, top_k=5, seeds=[1, 2], forced=forced)
