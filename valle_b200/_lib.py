"""ctypes binding of libvalle_b200.so (include/valle_b200.h).

There is NO fallback: if the shared object is missing or a call fails, an exception is raised.
PyTorch is used by the callers only for device memory, streams and torch.distributed.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "lib", "libvalle_b200.so")

ABI_VERSION = 5
VB_F32, VB_BF16 = 0, 1
VB_EPI_NONE, VB_EPI_RELU, VB_EPI_RESIDUAL = 0, 1, 2
VB_MASK_FULL, VB_MASK_VALLE_AR, VB_MASK_PADDED_AR, VB_MASK_PADDED, VB_MASK_DENSE = 0, 1, 2, 3, 4

c_i32p = C.POINTER(C.c_int32)
c_i64p = C.POINTER(C.c_int64)
c_f32p = C.POINTER(C.c_float)
vp = C.c_void_p


class LayerParams(C.Structure):
    """vb_layer_params (include/valle_b200.h): device pointers of one TransformerEncoderLayer"""
    _fields_ = [(n, vp) for n in (
        "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "lin1_w", "lin1_b", "lin2_w", "lin2_b",
        "norm1_w", "norm1_b", "norm2_w", "norm2_b")]


class DecoderDesc(C.Structure):
    """vb_decoder_desc"""
    _fields_ = [("d_model", C.c_int32), ("n_head", C.c_int32), ("n_layer", C.c_int32),
                ("d_ff", C.c_int32), ("wdtype", C.c_int32), ("layers", C.POINTER(LayerParams)),
                ("final_norm_w", vp), ("final_norm_b", vp)]


class ArState(C.Structure):
    """vb_ar_state: device-resident state of the AR sampling loop (valle.py:1012-1057)"""
    _fields_ = [("B", C.c_int32), ("tok_stride", C.c_int32),
                ("text_len", vp), ("prompt_len", vp), ("max_new", vp),
                ("n_gen", vp), ("finished", vp), ("tokens", vp), ("x_cur", vp), ("logits", vp),
                ("kcache", vp), ("vcache", vp),
                ("cache_layer_stride", C.c_int64), ("cache_seq_stride", C.c_int64),
                ("cache_cap", C.c_int32), ("_unused", C.c_int32),
                ("seed", vp), ("top_k", vp), ("temperature", vp)]


class LnFold(C.Structure):
    """vb_ln_fold: a LayerNorm folded into the projection that consumes it (bf16 decode chain)"""
    _fields_ = [("wf", vp), ("c", vp), ("dvec", vp)]


class ArHead(C.Structure):
    """vb_ar_head: ar_predict_layer + the embedding / position tables the sampler needs for the next row"""
    _fields_ = [("predict_w", vp), ("n_vocab", C.c_int32), ("eos_id", C.c_int32),
                ("audio_emb", vp), ("alpha", vp), ("pe", vp),
                ("pe_rows", C.c_int32), ("greedy", C.c_int32), ("fold", LnFold)]


class LayerGrads(C.Structure):
    """vb_layer_grads: fp32 gradient buffers of one layer (accumulated)"""
    _fields_ = [(n, vp) for n in (
        "in_proj_w", "in_proj_b", "out_proj_w", "out_proj_b", "lin1_w", "lin1_b", "lin2_w", "lin2_b",
        "norm1_w", "norm1_b", "norm2_w", "norm2_b")]


class LayerWt(C.Structure):
    """vb_layer_wt: transposed matrices of one layer (storage dtype)"""
    _fields_ = [(n, vp) for n in ("in_proj_wt", "out_proj_wt", "lin1_wt", "lin2_wt")]


class VbError(RuntimeError):
    """a C-ABI call returned a non-zero status, or libvalle_b200.so is missing (there is no fallback path)"""


_lib: Optional[C.CDLL] = None

# name -> (restype, argtypes).  Every symbol declared in include/valle_b200.h is listed here;
# tests/test_abi.py checks the header and this table against the built library.
PROTOTYPES = {
    "vb_abi_version": (C.c_int, []),
    "vb_last_error": (C.c_char_p, []),
    "vb_launch_count": (C.c_int64, []),
    "vb_trace_bind": (C.c_int, [vp, vp, C.c_uint]),
    "vb_tune_set": (C.c_int, [C.c_char_p, C.c_int]),
    "vb_embed_sum": (C.c_int, [vp, C.c_int64, C.c_int64, C.POINTER(vp), c_i32p, C.c_int, C.c_int64, C.c_int, vp,
                               C.c_int64, vp, C.c_int, vp, vp]),
    "vb_add_pe": (C.c_int, [vp, C.c_int64, vp, C.c_int64, vp, vp, C.c_int64, C.c_int, vp, C.c_int64, vp, vp]),
    "vb_layernorm": (C.c_int, [vp, C.c_int64, vp, C.c_int64, C.c_int, vp, vp, vp, C.c_float, vp, C.c_int, vp]),
    "vb_adaln_project": (C.c_int, [vp, vp, vp, C.c_int, vp, vp]),
    "vb_linear": (C.c_int, [vp, C.c_int, C.c_int64, vp, C.c_int, vp, vp, C.c_int, C.c_int64, C.c_int64,
                            C.c_int, C.c_int, C.c_int, vp, C.c_size_t, vp]),
    "vb_attention": (C.c_int, [vp, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int,
                               vp, vp, vp, C.c_int64, C.c_int, vp, C.c_int64, vp]),
    "vb_decoder_create": (C.c_int, [C.POINTER(DecoderDesc), C.POINTER(vp)]),
    "vb_decoder_destroy": (None, [vp]),
    "vb_decoder_forward_workspace": (C.c_size_t, [C.POINTER(DecoderDesc), C.c_int64]),
    "vb_decoder_forward": (C.c_int, [vp, vp, C.c_int64, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp,
                                     C.c_int64, C.c_int64, C.c_int, vp, C.c_size_t, vp]),
    "vb_decoder_train_save_bytes": (C.c_size_t, [C.POINTER(DecoderDesc), C.c_int64]),
    "vb_decoder_forward_train": (C.c_int, [vp, vp, C.c_int64, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp,
                                           C.c_size_t, C.c_float, C.c_uint64, vp]),
    "vb_dropout": (C.c_int, [vp, vp, C.c_int, C.c_int64, C.c_float, C.c_uint64, C.c_uint32, vp]),
    "vb_decoder_backward_workspace": (C.c_size_t, [C.POINTER(DecoderDesc), C.c_int64]),
    "vb_decoder_backward": (C.c_int, [vp, vp, C.c_int64, C.c_int, vp, vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp,
                                      C.POINTER(LayerWt), C.POINTER(LayerGrads), vp, C.c_size_t, C.c_float, C.c_uint64,
                                      vp]),
    "vb_layernorm_backward": (C.c_int, [vp, C.c_int64, vp, C.c_int64, C.c_int, vp, vp, vp, C.c_float, vp, C.c_int64, vp,
                                        C.c_int64, vp, C.c_int, vp, vp, vp, vp]),
    "vb_cross_entropy_backward": (C.c_int, [vp, C.c_int64, vp, C.c_int64, C.c_int, C.c_int64, vp, C.c_float, vp, C.c_int,
                                            C.c_int64, C.c_int, vp]),
    "vb_embed_backward": (C.c_int, [vp, C.c_int64, C.c_int64, C.POINTER(vp), c_i32p, C.c_int, C.c_int64, C.c_int, vp,
                                    C.c_int64, vp, vp]),
    "vb_rowdot_accumulate": (C.c_int, [vp, C.c_int64, vp, C.c_int64, vp, C.c_int64, C.c_int, vp, vp]),
    "vb_adaln_project_backward": (C.c_int, [vp, vp, vp, C.c_int, vp, vp, vp, vp]),
    "vb_linear_backward_workspace": (C.c_size_t, [C.c_int, C.c_int64, C.c_int, C.c_int]),
    "vb_linear_backward": (C.c_int, [vp, C.c_int, C.c_int64, vp, vp, C.c_int64, vp, C.c_int, C.c_int64, C.c_int, vp, vp,
                                     C.c_int64, C.c_int, C.c_int, vp, C.c_size_t, vp]),
    "vb_attention_backward_workspace": (C.c_size_t, [C.c_int64, C.c_int]),
    "vb_attention_backward": (C.c_int, [vp, vp, vp, C.c_int, C.c_int64, C.c_int, C.c_int, C.c_int, vp, vp, vp, C.c_int,
                                        C.c_int, C.c_int, vp, vp, C.c_size_t, vp]),
    "vb_ln_fold_build": (C.c_int, [vp, C.c_int, C.c_int, vp, vp, vp, vp, vp, vp, vp]),
    "vb_decoder_set_decode_fold": (C.c_int, [vp, C.POINTER(LnFold), C.POINTER(LnFold)]),
    "vb_ar_step_workspace": (C.c_size_t, [C.POINTER(DecoderDesc), C.c_int, C.c_int]),
    "vb_ar_head_step": (C.c_int, [vp, C.POINTER(ArHead), vp, C.POINTER(ArState), vp, C.c_size_t, vp]),
    "vb_ar_decode_step": (C.c_int, [vp, C.POINTER(ArHead), C.POINTER(ArState), vp, C.c_size_t, vp]),
    "vb_ar_push_tokens": (C.c_int, [C.POINTER(ArHead), C.POINTER(ArState), vp, C.c_int, vp]),
    "vb_nar_argmax_accumulate": (C.c_int, [vp, C.c_int64, C.c_int, C.c_int64, vp, C.c_int64, vp, vp,
                                           C.c_int64, vp, C.c_int, vp]),
    "vb_cross_entropy": (C.c_int, [vp, C.c_int64, vp, C.c_int64, C.c_int, C.c_int64, vp, vp]),
    "vb_conv1d": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                            C.c_int, C.c_int, vp, vp, C.c_int, C.c_int, vp]),
    "vb_lstm_layer": (C.c_int, [vp, vp, C.c_int, C.c_int, C.c_int, vp, vp, vp]),
    "vb_rvq_encode": (C.c_int, [vp, C.c_int64, C.c_int, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int64, C.c_int64,
                                C.c_int64, C.c_int64, vp]),
    "vb_permute3": (C.c_int, [vp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, vp, vp]),
    "vb_gather_rows": (C.c_int, [vp, C.c_int64, vp, C.c_int64, C.c_int, vp, C.c_int64, vp]),
}


def load() -> C.CDLL:
    """Load libvalle_b200.so.  Raises if it has not been built (python -m valle_b200.build)."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("VB_LIB_PATH", LIB_PATH)  # profiling builds: valle_b200/lib/libvalle_b200_trace.so
    if not os.path.exists(path):
        raise VbError(
            f"{path} is missing: the CUDA engine has not been built. Run "
            "`python -m valle_b200.build` (or __graft_entry__.build()). There is no CPU/PyTorch fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the symbol is not exported
        fn.restype = res
        fn.argtypes = args
    if lib.vb_abi_version() != ABI_VERSION:
        raise VbError(f"ABI version mismatch: library {lib.vb_abi_version()} != binding {ABI_VERSION}")
    _lib = lib
    return lib


def check(status: int, what: str = "") -> None:
    if status != 0:
        msg = load().vb_last_error().decode("utf-8", "replace")
        raise VbError(f"{what or 'libvalle_b200'} failed (status {status}): {msg}")


def ptr(t) -> int:
    """device pointer of a torch tensor (None -> NULL)."""
    return 0 if t is None else t.data_ptr()


def stream_ptr() -> int:
    import torch
    return torch.cuda.current_stream().cuda_stream
