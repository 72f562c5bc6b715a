"""Generate the golden fixtures under tests/golden/ by running the UNMODIFIED reference
(/root/reference, through oracle/ref_loader.py) on CPU in fp32.  Runs only in the build
container; the fixtures travel to the GPU box, the reference does not.

    python -m oracle.gen_golden [tiny] [batch] [config0] [big_short] [big_full] [topk] [ref_oracle] [ref_layout]

Every fixture stores: the model config, the weight seed (weights = the reference's default init
under torch.manual_seed(seed); valle_b200.models.VALLE reproduces them bit-for-bit, checked by
per-parameter checksums stored here), the inputs, the reference outputs (codes), the top1-top2
logit margin of every argmax the reference took (so a parity test can tell a near-tie from a
bug), and a few raw logit rows for tolerance checks.
"""
from __future__ import annotations

import os
import sys
import time

import torch

from . import valle_oracle as O
from .ref_loader import load_reference

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def build_reference(ref, d, h, l, pm, seed):
    torch.manual_seed(seed)
    m = ref.VALLE(d, h, l, norm_first=True, add_prenet=False, prefix_mode=pm, share_embedding=True,
                  nar_scale_factor=1.0, prepend_bos=False, num_quantizers=8).eval()
    return m


def checksums(sd):
    return O.weight_checksums(sd)


def make_inputs(gen, S, Tp):
    x = torch.randint(3, 100, (1, S), generator=gen)            # ids >= 3 avoid pad/bos/eos
    y = torch.randint(0, 1024, (1, Tp, 8), generator=gen)
    return x, y


def run_inference(ref, m, cfg, x, y, enroll=None):
    """reference codes + oracle trace (margins/logits) on the same inputs; asserts they agree."""
    sd = {k: v.detach() for k, v in m.state_dict().items()}
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    t0 = time.time()
    with torch.no_grad():
        codes = m.inference(x, xl, y, enroll, top_k=1)
    t_ref = time.time() - t0
    tr = O.InferenceTrace([], [], [], [])
    with torch.no_grad():
        codes_o = O.inference(sd, cfg, x, xl, y, enroll, top_k=1, trace=tr)
    assert torch.equal(codes, codes_o), "oracle restatement disagrees with the reference"
    n = len(tr.ar_logits)
    keep = sorted({0, n // 2, n - 1})
    rec = {
        "x": x, "y": y, "codes": codes.to(torch.int16),
        "ar_margin": torch.tensor(tr.ar_margin),
        "nar_margin": torch.stack(tr.nar_margin) if tr.nar_margin else torch.zeros(0),
        "ar_logit_steps": torch.tensor(keep), "ar_logits": torch.stack([tr.ar_logits[i] for i in keep]),
        "nar_logits_row0": torch.stack([l[0] for l in tr.nar_logits]) if tr.nar_logits else torch.zeros(0),
        "ref_seconds": t_ref,
    }
    return rec


def pick_input_seed(ref, m, cfg, S, Tp, min_margin, seeds=range(1, 40)):
    best = None
    for s in seeds:
        g = torch.Generator().manual_seed(s)
        x, y = make_inputs(g, S, Tp)
        rec = run_inference(ref, m, cfg, x, y)
        mm = min(float(rec["ar_margin"][:-1].min()), float(rec["nar_margin"].min()))
        if best is None or mm > best[0]:
            best = (mm, s, rec)
        if mm >= min_margin:
            break
    mm, s, rec = best
    rec["input_seed"] = s
    rec["min_margin"] = mm
    return rec


def save(name, obj):
    os.makedirs(OUT, exist_ok=True)
    p = os.path.join(OUT, name)
    torch.save(obj, p)
    print(f"wrote {p} ({os.path.getsize(p) / 1024:.1f} KiB)")


def gen_tiny(ref):
    for pm in (0, 1, 2):
        d, h, l, seed = 256, 4, 2, 0
        m = build_reference(ref, d, h, l, pm, seed)
        cfg = O.OracleConfig(d, h, l, pm, 8)
        if pm == 2:
            g = torch.Generator().manual_seed(7)
            x, y = make_inputs(g, 12, 24)
            rec = run_inference(ref, m, cfg, x, y, enroll=torch.tensor([5], dtype=torch.int32))
            rec["enroll"] = 5
            rec["min_margin"] = min(float(rec["ar_margin"][:-1].min()), float(rec["nar_margin"].min()))
        else:
            rec = pick_input_seed(ref, m, cfg, 8, 20, 3e-4)
        xl = torch.tensor([rec["x"].shape[1]], dtype=torch.int32)
        with torch.no_grad():
            rec["continual"] = m.continual(rec["x"], xl, rec["y"]).to(torch.int16)
        rec.update(config=dict(d_model=d, nhead=h, num_layers=l, prefix_mode=pm, num_quantizers=8),
                   weight_seed=seed, checksums=checksums(m.state_dict()))
        print(f"tiny pm={pm}: frames={rec['codes'].shape[1]} min_margin={rec['min_margin']:.2e}")
        save(f"tiny_pm{pm}.pt", rec)


def gen_batch(ref):
    """ragged batch: the engine decodes all utterances together; each must equal the reference's
    batch-1 result (valle.py:989 asserts batch 1)."""
    d, h, l, pm, seed = 256, 4, 2, 1, 0
    m = build_reference(ref, d, h, l, pm, seed)
    cfg = O.OracleConfig(d, h, l, pm, 8)
    utts = []
    g = torch.Generator().manual_seed(11)
    for S, Tp in ((8, 20), (12, 31), (5, 9), (9, 17)):
        x, y = make_inputs(g, S, Tp)
        rec = run_inference(ref, m, cfg, x, y)
        rec["min_margin"] = min(float(rec["ar_margin"][:-1].min()), float(rec["nar_margin"].min()))
        print(f"batch utt S={S} Tp={Tp}: frames={rec['codes'].shape[1]} min_margin={rec['min_margin']:.2e}")
        utts.append(rec)
    save("tiny_batch.pt", dict(config=dict(d_model=d, nhead=h, num_layers=l, prefix_mode=pm, num_quantizers=8),
                               weight_seed=seed, checksums=checksums(m.state_dict()), utts=utts))


def gen_config0(ref):
    """BASELINE.json configs[0]: tiny VALLE d=256/4h/2L, 32 phonemes + 8x128 codec tokens:
    training forward (loss) and inference."""
    import random
    d, h, l, pm, seed = 256, 4, 2, 1, 0
    m = build_reference(ref, d, h, l, pm, seed)
    cfg = O.OracleConfig(d, h, l, pm, 8)
    g = torch.Generator().manual_seed(3)
    x, y = make_inputs(g, 32, 128)
    rec = run_inference(ref, m, cfg, x, y[:, :40])   # 40-frame prompt -> 513 generated frames
    rec["min_margin"] = min(float(rec["ar_margin"][:-1].min()), float(rec["nar_margin"].min()))
    # training forward on a padded batch of 3
    N = 3
    xx = torch.randint(3, 100, (N, 32), generator=g)
    xls = torch.tensor([32, 27, 19], dtype=torch.int32)
    yy = torch.randint(0, 1024, (N, 128, 8), generator=g)
    yls = torch.tensor([128, 101, 77], dtype=torch.int32)
    fw = {}
    for stage in (0, 1, 2):
        m.rng = random.Random(0)
        torch.manual_seed(5)
        with torch.no_grad():
            (_, _), loss, _ = m(xx, xls, yy, yls, train_stage=stage)
        fw[f"loss_stage{stage}"] = torch.as_tensor(float(loss))
    r = random.Random(0)
    fw["nar_stage"] = r.choices(list(range(1, 8)), weights=[1 / 7] * 7, k=1)[0]
    torch.manual_seed(5)
    int_low = (0.25 * yls.min()).type(torch.int64).item()
    fw["prefix_len"] = min(torch.randint(int_low, int_low * 2, size=()).item(), 225)
    fw.update(x=xx, x_lens=xls, y=yy.to(torch.int16), y_lens=yls, torch_seed=5)
    rec.update(config=dict(d_model=d, nhead=h, num_layers=l, prefix_mode=pm, num_quantizers=8),
               weight_seed=seed, checksums=checksums(m.state_dict()), forward=fw)
    print(f"config0: frames={rec['codes'].shape[1]} min_margin={rec['min_margin']:.2e} losses="
          f"{[float(fw[f'loss_stage{s}']) for s in (0, 1, 2)]}")
    save("config0.pt", rec)


def gen_big(ref, S, Tp, name):
    d, h, l, pm, seed = 1024, 16, 12, 1, 0
    m = build_reference(ref, d, h, l, pm, seed)
    cfg = O.OracleConfig(d, h, l, pm, 8)
    g = torch.Generator().manual_seed(2)
    x, y = make_inputs(g, S, Tp)
    rec = run_inference(ref, m, cfg, x, y)
    rec["min_margin"] = min(float(rec["ar_margin"][:-1].min()), float(rec["nar_margin"].min()))
    ck = checksums(m.state_dict())
    rec.update(config=dict(d_model=d, nhead=h, num_layers=l, prefix_mode=pm, num_quantizers=8),
               weight_seed=seed, checksums=ck)
    print(f"{name}: frames={rec['codes'].shape[1]} min_margin={rec['min_margin']:.2e} ref_s={rec['ref_seconds']:.1f}")
    save(f"{name}.pt", rec)


def gen_topk(ref):
    """top-k / temperature sampling at a fixed torch seed (valle.py:1040-1043,1287-1302): the reference draws with
    torch.multinomial from torch's CPU generator, once per generated token.  The engine reproduces the ids when it
    samples on the host (engine.sample_on_host) from logits that agree to ~1e-5."""
    d, h, l, pm, seed = 256, 4, 2, 1, 0
    m = build_reference(ref, d, h, l, pm, seed)
    g = torch.Generator().manual_seed(21)
    x, y = make_inputs(g, 7, 18)
    xl = torch.tensor([x.shape[1]], dtype=torch.int32)
    cases = []
    for top_k, temp, tseed in ((5, 0.9, 1234), (-100, 1.0, 7), (20, 1.3, 99)):
        torch.manual_seed(tseed)
        with torch.no_grad():
            codes = m.inference(x, xl, y, None, top_k=top_k, temperature=temp)
        sd = {k: v.detach() for k, v in m.state_dict().items()}
        torch.manual_seed(tseed)
        with torch.no_grad():
            codes_o = O.inference(sd, O.OracleConfig(d, h, l, pm, 8), x, xl, y, None, top_k=top_k, temperature=temp)
        assert torch.equal(codes, codes_o), "oracle restatement disagrees with the reference under sampling"
        print(f"topk case top_k={top_k} T={temp} seed={tseed}: {codes.shape[1]} frames")
        cases.append(dict(top_k=top_k, temperature=temp, torch_seed=tseed, codes=codes.to(torch.int16)))
    save("tiny_topk.pt", dict(config=dict(d_model=d, nhead=h, num_layers=l, prefix_mode=pm, num_quantizers=8),
                              weight_seed=seed, checksums=checksums(m.state_dict()), x=x, y=y, cases=cases))


def gen_switches(ref, only=()):
    """the constructor switches beyond the north-star configuration that the engine builds: prepend_bos (valle.py:
    1006-1007,1059-1065,329-332), nar_scale_factor != 1 (valle.py:83,231-247) and add_prenet (valle.py:96-131,
    181-214, with randomised BatchNorm running statistics stored in the fixture): greedy inference codes and the
    training losses of a small padded batch, from the unmodified reference"""
    import random
    for name, d, h, l, bos, f, pre in (("tiny_bos", 256, 4, 2, True, 1.0, False), ("tiny_scale", 512, 8, 2, False, 0.5, False),
                                       ("tiny_prenet", 256, 4, 2, False, 1.0, True)):
        if only and name not in only:
            continue
        torch.manual_seed(0)
        m = ref.VALLE(d, h, l, norm_first=True, add_prenet=pre, prefix_mode=1, share_embedding=True,
                      nar_scale_factor=f, prepend_bos=bos, num_quantizers=8).eval()
        g = torch.Generator().manual_seed(31)
        buffers = {}
        if pre:   # non-trivial BatchNorm running statistics (a fresh module has mean 0 / var 1)
            for k, v in m.named_buffers():
                if k.endswith("running_mean"):
                    v.copy_(torch.randn(v.shape, generator=g) * 0.05)
                elif k.endswith("running_var"):
                    v.copy_(torch.rand(v.shape, generator=g) + 0.5)
                if k.endswith(("running_mean", "running_var")):
                    buffers[k] = v.clone()
        x, y = make_inputs(g, 6, 14)
        xl = torch.tensor([x.shape[1]], dtype=torch.int32)
        with torch.no_grad():
            codes = m.inference(x, xl, y, None, top_k=1)
        N = 3
        xx = torch.randint(3, 100, (N, 12), generator=g)
        xls = torch.tensor([12, 9, 7], dtype=torch.int32)
        yy = torch.randint(0, 1024, (N, 40, 8), generator=g)
        yls = torch.tensor([40, 31, 22], dtype=torch.int32)
        fw = {}
        for stage in (0, 1, 2):
            m.rng = random.Random(0)
            torch.manual_seed(5)
            with torch.no_grad():
                (_, _), loss, _ = m(xx, xls, yy, yls, train_stage=stage)
            fw[f"loss_stage{stage}"] = torch.as_tensor(float(loss))
        fw.update(x=xx, x_lens=xls, y=yy.to(torch.int16), y_lens=yls, torch_seed=5)
        print(f"{name}: frames={codes.shape[1]} losses={[float(fw[f'loss_stage{s}']) for s in (0, 1, 2)]}")
        save(f"{name}.pt", dict(config=dict(d_model=d, nhead=h, num_layers=l, prefix_mode=1, num_quantizers=8,
                                            prepend_bos=bos, nar_scale_factor=f, add_prenet=pre),
                                weight_seed=0, checksums=checksums(m.state_dict()), buffers=buffers, x=x, y=y,
                                codes=codes.to(torch.int16), forward=fw))


def gen_ref_oracle(ref):
    """greedy, continual and top-k sampled codes and a training loss of the reference at prefix_mode 0 and 1, on the
    inputs tests/test_oracle.py feeds the oracle"""
    import random
    d, h, l, seed = 256, 4, 2, 0
    out = {}
    for pm in (0, 1):
        m = build_reference(ref, d, h, l, pm, seed)
        g = torch.Generator().manual_seed(21)
        x = torch.randint(3, 100, (1, 7), generator=g)
        y = torch.randint(0, 1024, (1, 15, 8), generator=g)
        xl = torch.tensor([7], dtype=torch.int32)
        with torch.no_grad():
            codes = m.inference(x, xl, y, None, top_k=1)
            cont = m.continual(x, xl, y)
            torch.manual_seed(3)
            sampled = m.inference(x, xl, y, None, top_k=5, temperature=0.9)
        xx = torch.randint(3, 100, (3, 9), generator=g)
        xls = torch.tensor([9, 7, 5], dtype=torch.int32)
        yy = torch.randint(0, 1024, (3, 40, 8), generator=g)
        yls = torch.tensor([40, 33, 28], dtype=torch.int32)
        m.rng = random.Random(0)
        torch.manual_seed(5)
        with torch.no_grad():
            (_, _), loss, _ = m(xx, xls, yy, yls)
        out[f"pm{pm}"] = dict(config=dict(d_model=d, nhead=h, num_layers=l, prefix_mode=pm, num_quantizers=8),
                              weight_seed=seed, checksums=checksums(m.state_dict()), x=x, y=y,
                              codes=codes.to(torch.int16), continual=cont.to(torch.int16),
                              sampled=sampled.to(torch.int16),
                              forward=dict(x=xx, x_lens=xls, y=yy.to(torch.int16), y_lens=yls,
                                           loss=torch.as_tensor(float(loss))))
        print(f"ref_oracle pm={pm}: frames={codes.shape[1]} sampled={sampled.shape[1]} loss={float(loss):.6f}")
    save("ref_oracle.pt", out)


def gen_ref_layout(ref):
    """the reference's state_dict layout (name -> shape, dtype in order), per-tensor fingerprints and parameter /
    buffer names: without and with the pre-nets at weight seed 0, and at seed 123 (tests/test_oracle.py,
    tests/test_boundary.py)"""
    out = {}
    for name, prenet, seed in (("prenet0", False, 0), ("prenet1", True, 0), ("seed123", False, 123)):
        torch.manual_seed(seed)
        m = ref.VALLE(256, 4, 2, norm_first=True, add_prenet=prenet, prefix_mode=1, share_embedding=True,
                      nar_scale_factor=1.0, prepend_bos=False, num_quantizers=8)
        sd = m.state_dict()
        out[name] = dict(tensors={k: (tuple(v.shape), v.dtype) for k, v in sd.items()}, checksums=checksums(sd),
                         parameters=[n for n, _ in m.named_parameters()], buffers=[n for n, _ in m.named_buffers()])
        print(f"ref_layout {name}: {len(sd)} tensors")
    save("ref_layout.pt", out)


def main(argv):
    ref = load_reference()
    what = argv or ["tiny", "batch", "config0", "big_short"]
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    if "tiny" in what:
        gen_tiny(ref)
    if "batch" in what:
        gen_batch(ref)
    if "config0" in what:
        gen_config0(ref)
    if "big_short" in what:
        gen_big(ref, 6, 30, "big_short")
    if "switches" in what:
        gen_switches(ref)
    if "prenet" in what:
        gen_switches(ref, only=("tiny_prenet",))
    if "topk" in what:
        gen_topk(ref)
    if "big_full" in what:
        gen_big(ref, 47, 225, "big_full")  # BASELINE.json configs[1]: 3 s prompt -> 753 frames
    if "ref_oracle" in what:
        gen_ref_oracle(ref)
    if "ref_layout" in what:
        gen_ref_layout(ref)


if __name__ == "__main__":
    main(sys.argv[1:])
