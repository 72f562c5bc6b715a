"""CPU tests of the oracle against outputs of the reference itself, stored under tests/golden/ by
oracle/gen_golden.py."""
import random

import pytest
import torch

from conftest import assert_checksums, build_model, load_golden
from oracle import valle_oracle as O


def _sd(m):
    return {k: v.detach() for k, v in m.state_dict().items()}


@pytest.mark.parametrize("name", ["tiny_pm0.pt", "tiny_pm1.pt", "tiny_pm2.pt"])
def test_oracle_reproduces_golden_codes(name):
    g = load_golden(name)
    m = build_model(g["config"], g["weight_seed"])
    assert_checksums(m, g["checksums"])      # our init == the reference's init, bit for bit
    cfg = O.OracleConfig(**g["config"])
    x, y = g["x"], g["y"]
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    enroll = torch.tensor([g["enroll"]], dtype=torch.int32) if "enroll" in g else None
    tr = O.InferenceTrace([], [], [], [])
    with torch.no_grad():
        codes = O.inference(_sd(m), cfg, x, xl, y, enroll, top_k=1, trace=tr)
        cont = O.continual(_sd(m), cfg, x, xl, y)
    assert torch.equal(codes, g["codes"].long())
    assert torch.equal(cont, g["continual"].long())
    steps = g["ar_logit_steps"].tolist()
    got = torch.stack([tr.ar_logits[i] for i in steps])
    assert torch.allclose(got, g["ar_logits"], atol=1e-5, rtol=0)


def test_kv_cache_equals_full_recompute():
    """The engine's algorithm (prefill + cached single-row steps) is exact under the reference's
    mask (valle.py:1019-1030): same greedy tokens, logits within 1e-5."""
    g = load_golden("tiny_pm1.pt")
    m = build_model(g["config"], g["weight_seed"])
    cfg = O.OracleConfig(**g["config"])
    x, y = g["x"], g["y"]
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    with torch.no_grad():
        toks, logits = O.ar_decode_kv(_sd(m), cfg, x, xl, y, collect_logits=True)
    assert torch.equal(toks, g["codes"][..., 0].long())
    steps = g["ar_logit_steps"].tolist()
    got = torch.stack([logits[i] for i in steps])
    assert torch.allclose(got, g["ar_logits"], atol=2e-5, rtol=0)


def test_oracle_forward_matches_golden_loss():
    g = load_golden("config0.pt")
    m = build_model(g["config"], g["weight_seed"])
    cfg = O.OracleConfig(**g["config"])
    fw = g["forward"]
    for stage in (0, 1, 2):
        with torch.no_grad():
            loss, _ = O.forward_train(_sd(m), cfg, fw["x"], fw["x_lens"], fw["y"].long(), fw["y_lens"],
                                      fw["nar_stage"], fw["prefix_len"], train_stage=stage)
        ref = float(fw[f"loss_stage{stage}"])
        assert abs(float(loss) - ref) <= 1e-4 * abs(ref), (stage, float(loss), ref)


def test_sampling_restatement_greedy_is_argmax():
    torch.manual_seed(0)
    logits = torch.randn(4, 1025)
    tok = O.topk_sampling(logits.clone(), top_k=1)
    assert torch.equal(tok[:, 0], logits.argmax(-1))
    # top_k <= 0 leaves the distribution unfiltered (valle.py:1254)
    assert torch.equal(O.top_k_top_p_filtering(logits.clone(), top_k=-100), logits)


@pytest.mark.parametrize("pm", [0, 1])
def test_oracle_vs_reference_inference_and_forward(pm):
    """greedy and continual codes, top-k sampled codes at a fixed torch seed (the oracle consumes torch's RNG as the
    reference does) and a training loss, against the reference's own outputs on the same weights and inputs"""
    g = load_golden("ref_oracle.pt")[f"pm{pm}"]
    m = build_model(g["config"], g["weight_seed"])
    assert_checksums(m, g["checksums"])
    sd = _sd(m)
    cfg = O.OracleConfig(**g["config"])
    x, y = g["x"], g["y"]
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    with torch.no_grad():
        assert torch.equal(O.inference(sd, cfg, x, xl, y, None, top_k=1), g["codes"].long())
        assert torch.equal(O.continual(sd, cfg, x, xl, y), g["continual"].long())
        torch.manual_seed(3)
        assert torch.equal(O.inference(sd, cfg, x, xl, y, None, top_k=5, temperature=0.9), g["sampled"].long())
    fw = g["forward"]
    xx, xls, yy, yls = fw["x"], fw["x_lens"], fw["y"].long(), fw["y_lens"]
    # the NAR stage and the prompt prefix the reference drew with m.rng = random.Random(0) and torch.manual_seed(5)
    ns = random.Random(0).choices(list(range(1, 8)), weights=[1 / 7] * 7, k=1)[0]
    torch.manual_seed(5)
    int_low = (0.25 * yls.min()).type(torch.int64).item()
    pl = min(torch.randint(int_low, int_low * 2, size=()).item(), 225) if pm == 1 else 0
    with torch.no_grad():
        l2, _ = O.forward_train(sd, cfg, xx, xls, yy, yls, ns, pl)
    loss = float(fw["loss"])
    assert abs(loss - float(l2)) <= 1e-5 * abs(loss)


@pytest.mark.parametrize("prenet", [False, True])
def test_model_mirror_matches_reference_checkpoint_layout(prenet):
    """valle_b200.models.VALLE: same state_dict keys, shapes, dtypes, init values and strict loading -- also with the
    pre-nets of add_prenet=True (Conv1d / BatchNorm1d / Linear containers at the reference's Sequential indices)."""
    ref = load_golden("ref_layout.pt")[f"prenet{int(prenet)}"]
    cfg = dict(d_model=256, nhead=4, num_layers=2, prefix_mode=1, num_quantizers=8, add_prenet=prenet)
    b = build_model(cfg, 0)
    assert {k: (tuple(v.shape), v.dtype) for k, v in b.state_dict().items()} == ref["tensors"]
    assert_checksums(b, ref["checksums"])   # same keys in the same order, same init values
    b.load_state_dict({k: torch.zeros(s, dtype=dt) for k, (s, dt) in ref["tensors"].items()}, strict=True)
    assert [n for n, _ in b.named_parameters()] == ref["parameters"]
    assert [n for n, _ in b.named_buffers()] == ref["buffers"]
    assert (len(list(b.named_buffers())) == 0) == (not prenet)
