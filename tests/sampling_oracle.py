"""TEST INFRASTRUCTURE ONLY -- numpy / torch-CPU restatement of the seeded sampler of the AR decode step
(ar_sample_kernel in valle_b200/csrc/sample.cu, semantics in include/valle_b200.h under vb_ar_head):

    z = logits / T                      (fp32, as valle.py:1297-1298)
    keep z_i >= k-th largest z          (top_k > 0; ties with the k-th value kept, valle.py:1254-1260)
    key_i = z_i - log(-log(u_i)),       u_i = ((mix64(seed, step, i) >> 40) + 0.5) * 2**-24
    sample = argmax key                 (lowest id on an exact tie)

plus a free-running seeded VALLE.inference built from the operators of oracle/valle_oracle.py.  The kept set is
restated here on its own (sorting), so that tests can compare it with oracle.top_k_top_p_filtering.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from oracle import valle_oracle as O

_C_STREAM = np.uint64(0x9E3779B97F4A7C15)
_C_IDX = np.uint64(0xD1342543DE82EF95)


def mix64(seed, stream, idx) -> np.ndarray:
    """the splitmix64 finaliser of csrc/kernels.cuh (dropout masks, seeded sampling); numpy uint64, broadcasting"""
    with np.errstate(over="ignore"):
        z = (np.asarray(seed, dtype=np.uint64) + np.asarray(stream, dtype=np.uint64) * _C_STREAM
             + np.asarray(idx, dtype=np.uint64) * _C_IDX)
        z ^= z >> np.uint64(30)
        z *= np.uint64(0xBF58476D1CE4E5B9)
        z ^= z >> np.uint64(27)
        z *= np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
    return z


def gumbel_log_e(seed, step, idx) -> np.ndarray:
    """log(e), e = -log(u) in fp32 from the exact value of u (h < 2**23) or of 1 - u (h >= 2**23); key = z - log(e)"""
    h = (mix64(seed, step, idx) >> np.uint64(40)).astype(np.int64)
    lo = h < (1 << 23)
    scale = np.float32(2.0 ** -24)
    u = (np.where(lo, h, 0).astype(np.float32) + np.float32(0.5)) * scale
    v = (np.where(lo, 0, (1 << 24) - 1 - h).astype(np.float32) + np.float32(0.5)) * scale
    e = np.where(lo, -np.log(u), -np.log1p(-v)).astype(np.float32)
    return np.log(e).astype(np.float32)


def scaled(logits, temperature: float) -> np.ndarray:
    """z = logits / T in fp32 (IEEE division)"""
    if isinstance(logits, torch.Tensor):
        logits = logits.detach().to(torch.float32).cpu().numpy()
    return (np.asarray(logits, dtype=np.float32) / np.float32(temperature)).astype(np.float32)


def kept(logits, top_k: int, temperature: float = 1.0) -> np.ndarray:
    """bool [..., V]: ids that survive the top-k filter of the scaled logits"""
    z = scaled(logits, temperature)
    V = z.shape[-1]
    if top_k <= 0:
        return np.ones(z.shape, dtype=bool)
    k = min(max(top_k, 1), V)
    kth = np.sort(z, axis=-1)[..., V - k, None]
    return z >= kth


def seeded_keys(logits, seed, step, top_k: int, temperature: float) -> np.ndarray:
    """fp32 Gumbel keys [V] of the kept ids of one logits row [V], -inf elsewhere; with seed / step arrays [N] (one row
    drawn from N times) the keys are [N, V]"""
    z = scaled(logits, temperature)
    assert z.ndim == 1
    keep = kept(z, top_k)
    ids = np.nonzero(keep)[0].astype(np.uint64)
    seed = np.asarray(seed, dtype=np.uint64)[..., None]
    step = np.asarray(step, dtype=np.uint64)[..., None]
    key = np.full(np.broadcast_shapes(seed.shape, z.shape), -np.inf, dtype=np.float32)
    key[..., keep] = z[keep] - gumbel_log_e(seed, step, ids)
    return key


def seeded_draw(logits, seed, step, top_k: int, temperature: float):
    """the id the device sampler draws from one logits row [V] (an int; an array [N] for seed / step arrays [N])"""
    d = np.argmax(seeded_keys(logits, seed, step, top_k, temperature), axis=-1)
    return int(d) if np.ndim(d) == 0 else d


def key_gap(logits, seed, step, top_k: int, temperature: float) -> float:
    """top-1 minus top-2 key: a device / restatement disagreement is only excusable when this is tiny"""
    k = np.sort(seeded_keys(logits, seed, step, top_k, temperature))
    return float(k[-1] - k[-2]) if np.isfinite(k[-2]) else float("inf")


def inference(sd, cfg: O.OracleConfig, x, x_lens, y, enroll_x_lens=None, top_k: int = -100,
              temperature: float = 1.0, seed: int = 0, max_new_tokens: Optional[int] = None,
              prepend_bos: bool = False) -> torch.Tensor:
    """oracle.inference (valle.py:961-1137, full recompute per token) with the seeded draw at step t = number of ids
    generated so far; prepend_bos: <BOS> (id 1025) ahead of the AR audio stream (valle.py:1006-1007)"""
    S = int(x_lens.max())
    xe = O.pos_embed(sd["ar_text_embedding.word_embeddings.weight"][x], sd["ar_text_position.alpha"])
    Tp = y.shape[1]
    yy = y[..., 0]
    if prepend_bos:
        yy = torch.nn.functional.pad(yy, (1, 0), value=O.NUM_AUDIO_TOKENS + 1)
    n0 = yy.shape[1]
    while True:
        y_pos = O.pos_embed(sd["ar_audio_embedding.word_embeddings.weight"][yy], sd["ar_audio_position.alpha"])
        dec = O.encoder(sd, "ar_decoder", torch.concat([xe, y_pos], dim=1), cfg, blocked=O.ar_inference_mask(S, yy.shape[1]))
        logits = torch.nn.functional.linear(dec[:, -1], sd["ar_predict_layer.weight"])
        n_gen = yy.shape[1] - n0
        samp = seeded_draw(logits[0], seed, n_gen, top_k, temperature)
        n_new = yy.shape[1] - Tp
        if (int(torch.argmax(logits, dim=-1)[0]) == O.NUM_AUDIO_TOKENS or samp == O.NUM_AUDIO_TOKENS
                or n_new > S * 16 or (max_new_tokens is not None and n_gen >= max_new_tokens)):
            if n_gen == 0:
                raise SyntaxError("well trained model shouldn't reach here.")
            break
        yy = torch.concat([yy, torch.tensor([[samp]], dtype=yy.dtype)], dim=1)
    if prepend_bos:
        yy = yy[:, 1:]
    codes = [yy[:, Tp:]]
    if cfg.num_quantizers > 1:
        codes += O.nar_decode(sd, cfg, x, S, yy, y, Tp, enroll_x_lens)
    return torch.stack(codes, dim=-1)
