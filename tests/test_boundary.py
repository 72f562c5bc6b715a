"""Drop-in boundary (SURVEY.md 8b): the `valle` package name, get_model(AttributeDict(checkpoint)) and
load_state_dict(strict=True) of a checkpoint SAVED BY THE REFERENCE CLASS, the way valle/bin/infer.py:126-144 does it."""
import io
import os

import pytest
import torch

from conftest import ROOT

PARAMS = dict(model_name="VALL-E", decoder_dim=256, nhead=4, num_decoder_layers=2, scale_factor=1.0, norm_first=True,
              add_prenet=False, prefix_mode=1, share_embedding=True, prepend_bos=False, num_quantizers=8)


def test_valle_package_exports_the_reference_names():
    import valle
    from valle.data import AudioTokenizer, tokenize_audio  # noqa: F401
    from valle.models import VALLE, add_model_arguments, get_model  # noqa: F401
    from valle.models.valle import top_k_top_p_filtering, topk_sampling  # noqa: F401
    from valle.modules.activation import MultiheadAttention  # noqa: F401
    from valle.modules.embedding import SinePositionalEmbedding, TokenEmbedding  # noqa: F401
    from valle.modules.transformer import (AdaptiveLayerNorm, LayerNorm, TransformerEncoder,  # noqa: F401
                                           TransformerEncoderLayer)
    from valle.utils import AttributeDict, make_pad_mask
    import valle_b200
    assert valle.models.VALLE is valle_b200.models.VALLE
    assert os.path.dirname(os.path.abspath(valle.__file__)).startswith(ROOT)
    m = make_pad_mask(torch.tensor([3, 1]))
    assert m.tolist() == [[False, False, False], [False, True, True]]
    a = AttributeDict(x=1)
    assert a.x == 1


def _reference_checkpoint(seed):
    """the trainer's checkpoint, {"model": state_dict, ...flattened params} (valle/bin/trainer.py, icefall
    save_checkpoint), of the reference class initialised under torch.manual_seed(seed).  tests/golden/ref_layout.pt
    holds the reference's state_dict layout and per-tensor fingerprints; the tensors are rebuilt by this package's
    init, which must reproduce those fingerprints."""
    from conftest import assert_checksums, build_model, load_golden
    ref = load_golden("ref_layout.pt")[f"seed{seed}"]
    src = build_model(dict(d_model=PARAMS["decoder_dim"], nhead=PARAMS["nhead"], num_layers=PARAMS["num_decoder_layers"],
                           prefix_mode=1, num_quantizers=8), seed)
    assert_checksums(src, ref["checksums"])
    ckpt = dict(PARAMS)
    ckpt["model"] = src.state_dict()
    buf = io.BytesIO()
    torch.save(ckpt, buf)
    buf.seek(0)
    return ref, torch.load(buf, map_location="cpu", weights_only=False)


def test_infer_py_checkpoint_loading_from_a_reference_saved_checkpoint():
    """valle/bin/infer.py:126-144: checkpoint = torch.load(...); model = get_model(AttributeDict(checkpoint));
    missing, unexpected = model.load_state_dict(checkpoint["model"], strict=True); assert not missing"""
    from conftest import assert_checksums
    from valle.models import get_model
    from valle.utils import AttributeDict
    ref, ckpt = _reference_checkpoint(seed=123)
    torch.manual_seed(999)            # a different init, fully overwritten by the load
    model = get_model(AttributeDict(ckpt))
    missing, unexpected = model.load_state_dict(ckpt["model"], strict=True)
    assert not missing and not unexpected
    # the reference's keys in its order, shapes, dtypes and values
    assert {k: (tuple(v.shape), v.dtype) for k, v in model.state_dict().items()} == ref["tensors"]
    assert_checksums(model, ref["checksums"])
    # tied weights survive the load (valle.py:261-271)
    for j in range(6):
        assert model.nar_predict_layers[j].weight is model.nar_audio_embeddings[j + 2].weight
    # and the other way round: a checkpoint saved by this class loads into the reference class, whose strict load
    # needs exactly the key set and shapes checked above
    assert [n for n, _ in model.named_parameters()] == ref["parameters"]
    assert [n for n, _ in model.named_buffers()] == ref["buffers"]


@pytest.mark.gpu
def test_reference_saved_checkpoint_decodes_bit_exact_on_gpu():
    """GPU box (no /root/reference): the fixture's per-parameter fingerprints were taken from the REFERENCE's
    state_dict; a model built by get_model(AttributeDict(params)) + load_state_dict(strict=True) of the same weights
    must carry them and decode the reference's codes."""
    from conftest import assert_checksums, build_model, load_golden
    from valle.models import get_model
    from valle.utils import AttributeDict
    g = load_golden("tiny_pm1.pt")
    src = build_model(g["config"], g["weight_seed"])
    buf = io.BytesIO()
    ck = dict(PARAMS)
    ck["model"] = src.state_dict()
    torch.save(ck, buf)
    buf.seek(0)
    ckpt = torch.load(buf, map_location="cpu", weights_only=False)
    torch.manual_seed(999)            # a different init, fully overwritten by the load
    model = get_model(AttributeDict(ckpt))
    missing, unexpected = model.load_state_dict(ckpt["model"], strict=True)
    assert not missing and not unexpected
    assert_checksums(model, g["checksums"])
    model = model.to("cuda:0").eval()
    model.engine().quiet = True
    x, y = g["x"].to("cuda:0"), g["y"].to("cuda:0")
    out = model.inference(x, torch.tensor([x.shape[1]], dtype=torch.int32), y, None, top_k=1).cpu()
    assert torch.equal(out, g["codes"].long())
