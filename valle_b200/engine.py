"""Batched VALL-E decoding engine: the host side of the hot path.

Implements the loops of `VALLE.inference` (valle/models/valle.py:961-1137) for B independent
utterances at once on one GPU:

  * AR: ragged prefill of text + acoustic prompt (fills the KV cache), then single-row decode
    steps against the growing KV cache (the reference recomputes the whole sequence per token,
    valle.py:1004 TODO).  The KV cache is exact under the reference's mask: text rows attend to
    text only, audio rows to text + causal audio (valle.py:1019-1030), so cached K/V never change.
    All loop state (lengths, tokens, stop flags) lives on the device; a decode step is one CUDA
    graph replay; the host only polls the stop flags every `poll` steps (the reference does a
    D2H sync + an H2D mask copy per token).
  * NAR: 7 full-attention passes over packed [text | prompt | generated] rows with AdaLN stage
    conditioning, argmax and the embedding accumulation fused on the device (valle.py:1115-1134).

torch is used for allocation, streams and index bookkeeping; all arithmetic runs in
libvalle_b200.so.  There is no CPU fallback.
"""
from __future__ import annotations

import math
import os

import ctypes as C
from dataclasses import dataclass
from typing import Dict, List, Optional, Sequence, Tuple

import numpy as np
import torch

from . import _lib as L
from . import ops

NUM_AUDIO_TOKENS = 1024  # valle/models/macros.py:5
NUM_TEXT_TOKENS = 512    # valle/models/macros.py:2


def _on_device(fn):
    """Run a method with the engine's GPU as the current CUDA device: every kernel launch, stream and event of the
    call then belongs to `self.device` even when the caller's current device is another GPU of the box."""
    import functools

    @functools.wraps(fn)
    def wrapper(self, *args, **kwargs):
        with torch.cuda.device(self.device):
            return fn(self, *args, **kwargs)
    return wrapper


def _check_ids(tensors, hi: int, what: str):
    """nn.Embedding raises IndexError for ids outside the table (valle/modules/embedding.py:46).  Host tensors are
    checked here before the copy; device tensors are checked by the kernels (clamped read + flag, ops.check_oob)."""
    for t in tensors:
        if not t.is_cuda and t.numel() > 0:
            lo_v, hi_v = int(t.min()), int(t.max())
            if lo_v < 0 or hi_v >= hi:
                raise IndexError(f"index out of range in self: {what} id {lo_v if lo_v < 0 else hi_v} not in [0, {hi})")


def _per_utterance(v) -> bool:
    """a list / tuple / 1-d array of per-utterance values rather than one scalar"""
    return isinstance(v, (list, tuple)) or (isinstance(v, (torch.Tensor, np.ndarray)) and v.ndim > 0)


def _sampling_params(B: int, seeds, top_k, temperature):
    """validated per-utterance (seeds, top_k, temperature) lists of a seeded generate(); None without seeds"""
    if seeds is None:
        if _per_utterance(top_k) or _per_utterance(temperature):
            raise ValueError("per-utterance top_k / temperature need per-utterance seeds")
        return None
    seeds = [int(s) for s in seeds]
    if len(seeds) != B:
        raise ValueError(f"{len(seeds)} seeds for {B} utterances")
    if any(s < 0 or s >= 1 << 64 for s in seeds):
        raise ValueError("a seed is not in [0, 2**64)")
    ks = [int(k) for k in top_k] if _per_utterance(top_k) else [int(top_k)] * B
    ts = [float(t) for t in temperature] if _per_utterance(temperature) else [float(temperature)] * B
    if len(ks) != B or len(ts) != B:
        raise ValueError(f"per-utterance top_k / temperature must have {B} entries")
    if any(not math.isfinite(t) or t <= 0.0 for t in ts):
        raise ValueError("temperature must be finite and > 0")
    return seeds, ks, ts


@dataclass
class EngineStats:
    """CUDA-event timings (ms) of the phases of the last generate() call and the number of decode steps"""
    ar_steps: int = 0
    ar_ms: float = 0.0
    prefill_ms: float = 0.0
    nar_ms: float = 0.0


class _ArBuffers:
    """Persistent device state for the AR loop at one (B, cache_cap, tok_stride) shape, plus the
    captured CUDA graph of one decode step."""

    def __init__(self, eng: "ValleEngine", B: int, cap: int, tok_stride: int):
        dev, d = eng.device, eng.d
        nd = eng.ar
        self.B, self.cap, self.tok_stride = B, cap, tok_stride
        i32 = dict(dtype=torch.int32, device=dev)
        self.text_len = torch.zeros(B, **i32)
        self.prompt_len = torch.zeros(B, **i32)
        self.max_new = torch.zeros(B, **i32)
        self.n_gen = torch.zeros(B, **i32)
        self.finished = torch.zeros(B, **i32)
        self.tokens = torch.zeros((B, tok_stride), **i32)
        self.x_cur = torch.zeros((B, d), dtype=torch.float32, device=dev)
        self.ldl = (eng.n_vocab + 3) // 4 * 4
        self.logits = torch.zeros((B, self.ldl), dtype=torch.float32, device=dev)
        # seeded sampling on the device (generate(seeds=...)): the uint64 seeds as int64 bit patterns, top_k, temperature
        self.seed = torch.zeros(B, dtype=torch.int64, device=dev)
        self.top_k = torch.zeros(B, **i32)
        self.temperature = torch.ones(B, dtype=torch.float32, device=dev)
        self.kcache = torch.zeros((nd.n_layer, B, nd.H, cap, 64), dtype=eng.dtype, device=dev)
        self.vcache = torch.zeros_like(self.kcache)
        st = L.ArState()
        st.B, st.tok_stride = B, tok_stride
        st.text_len, st.prompt_len, st.max_new = self.text_len.data_ptr(), self.prompt_len.data_ptr(), self.max_new.data_ptr()
        st.n_gen, st.finished, st.tokens = self.n_gen.data_ptr(), self.finished.data_ptr(), self.tokens.data_ptr()
        st.x_cur, st.logits = self.x_cur.data_ptr(), self.logits.data_ptr()
        st.kcache, st.vcache = self.kcache.data_ptr(), self.vcache.data_ptr()
        st.cache_layer_stride, st.cache_seq_stride, st.cache_cap = self.kcache.stride(0), self.kcache.stride(1), cap
        st.seed, st.top_k, st.temperature = self.seed.data_ptr(), self.top_k.data_ptr(), self.temperature.data_ptr()
        self.st = st
        nbytes = eng.lib.vb_ar_step_workspace(C.byref(nd.desc), B, cap)
        self.ws = torch.zeros(nbytes, dtype=torch.uint8, device=dev)
        self.graph: Optional[torch.cuda.CUDAGraph] = None
        self.eng = eng


def _seg_ranges(starts, lens):
    """Concatenated aranges: rows = [starts[b] + i for b for i in range(lens[b])], pos = the i's (int64 numpy)."""
    starts = np.asarray(starts, dtype=np.int64)
    lens = np.asarray(lens, dtype=np.int64)
    total = int(lens.sum())
    if total == 0:
        return np.zeros(0, np.int64), np.zeros(0, np.int64)
    seg_first = np.repeat(np.cumsum(lens) - lens, lens)
    pos = np.arange(total, dtype=np.int64) - seg_first
    return np.repeat(starts, lens) + pos, pos


class ValleEngine:
    """Batched VALLE.inference / VALLE.continual (valle.py:961-1238) for B independent utterances: prefill of the
    AR decoder with a KV cache, the AR sampling loop as one CUDA-graph replay per token with the stop rule on the
    device (valle.py:1012-1057), then the 7 NAR passes (valle.py:1059-1137) over packed ragged rows.  Per utterance the
    result is exactly what the reference's batch-1 call returns; everything below this class is the C ABI."""
    def __init__(self, model, dtype: torch.dtype = torch.float32, use_cuda_graph: bool = True):
        self.lib = L.load()
        self.model = model
        self.dtype = dtype
        self.use_cuda_graph = use_cuda_graph
        p = model.ar_predict_layer.weight
        if not p.is_cuda:
            raise L.VbError("valle_b200: move the model to a CUDA device first (no CPU fallback)")
        self.device = p.device
        self.d = p.shape[1]
        #: width of the NAR stack (valle.py:83: nar_d_model = d_model * nar_scale_factor)
        self.d_nar = model.nar_audio_embeddings[0].weight.shape[1] if model.num_quantizers > 1 else self.d
        #: AR sequences start with <BOS> (id 1025) ahead of the acoustic prompt (valle.py:1006-1007)
        self.prepend_bos = bool(getattr(model, "ar_audio_prepend_bos", False))
        self.n_vocab = p.shape[0]
        self.Q = model.num_quantizers
        self.prefix_mode = model.prefix_mode
        self.stats = EngineStats()
        self.quiet = False
        #: top_k != 1 only: draw on the host exactly as the reference does (logits -> CPU, torch's CPU generator,
        #: one utterance after the other), so that a fixed torch.manual_seed reproduces the reference's ids; the
        #: default draws on the device (torch.multinomial on CUDA logits, Philox stream) without a per-token sync
        self.sample_on_host = False
        self.last_packed: Optional[torch.Tensor] = None
        #: rows of one tensor-core decode group (gemm_decode.cu: one UMMA N tile); larger bf16 batches are split
        self.max_tc_batch = 64
        #: bf16 decode steps run the LayerNorm-folded chain (6 launches per layer instead of 8) only on request
        #: (VB_DECODE_FOLD=1): it adds the split-K partials of the residual updates in arrival order, so a greedy decode
        #: can differ between two runs after a near-tie; the default chain adds them in fixed order and is reproducible
        self.use_decode_fold = os.environ.get("VB_DECODE_FOLD", "0") != "0"
        #: decode steps captured per CUDA graph, greedy or seeded sampling (one replay per group; the stop flags are
        #: polled every `poll` steps)
        self.steps_per_graph = 8
        self.replayed_launches = 0   # kernels executed through CUDA-graph replays
        self.captured_launches = 0   # kernels recorded at capture time (counted by the library, not run)
        self._bufs: Dict[Tuple[int, int, int], _ArBuffers] = {}
        self._ada_cache = None
        self._sig = None
        self._refresh()

    # ---- weights -----------------------------------------------------------------------
    def _signature(self):
        return tuple((q.data_ptr(), q._version) for q in list(self.model.parameters()) + list(self.model.buffers()))

    def _refresh(self):
        sig = self._signature()
        if sig == self._sig:
            return
        m = self.model
        self._sig = sig
        self.ar = m.ar_decoder.native(self.dtype)
        self.nar = m.nar_decoder.native(self.dtype) if self.Q > 1 else None
        cast = (lambda t: t.detach().to(self.dtype).contiguous()) if self.dtype != torch.float32 \
            else (lambda t: t.detach())
        self.ar_predict_w = cast(m.ar_predict_layer.weight)
        # bf16 decode chain: LayerNorms folded into the projections that consume them (vb_ln_fold), incl. the final norm
        # into ar_predict_layer (valle.py:1039)
        self.ar_head_fold = None
        fn = m.ar_decoder.norm
        if self.dtype == torch.bfloat16 and self.use_decode_fold and fn is not None and self.ar.enable_decode_fold():
            self.ar_head_fold = self.ar.fold_layernorm(self.ar_predict_w, fn.weight.detach(), fn.bias.detach(), None)
        self.nar_predict_w = [cast(l.weight) for l in m.nar_predict_layers] if self.Q > 1 else []
        self._ada_cache = None
        self._bufs.clear()  # graphs hold stale weight pointers
        self._prep_prenets()

    # ---- pre-nets (add_prenet=True, valle.py:96-131,181-214; eval mode: Dropout = identity, BatchNorm1d on its
    #      running statistics) ------------------------------------------------------------------
    def _prep_prenets(self):
        """fp32 weights of the four pre-nets in the layout the kernels take: every Conv1d(k=5, 'same') + BatchNorm1d
        pair becomes ONE [Cout, 5 Cin] matrix (the batch-norm scale / shift folded into weight and bias, columns in
        shift-major order to match `_im2col`), and the AR audio pre-net -- a function of the single embedded token
        (valle.py:1013-1014) -- becomes a pre-computed table over the 1025 (+BOS) ids."""
        m = self.model
        self.pre = None
        self.ar_audio_table = m.ar_audio_embedding.weight.detach()
        if not getattr(m, "add_prenet", False):
            return

        def text(seq):
            convs = []
            for i in (1, 5, 9):
                conv, bn = seq[i], seq[i + 1]
                scale = (bn.weight / torch.sqrt(bn.running_var + bn.eps)).detach().float()
                w = conv.weight.detach().float() * scale[:, None, None]                   # [Cout, Cin, 5]
                b = (conv.bias.detach().float() - bn.running_mean.float()) * scale + bn.bias.detach().float()
                convs.append((w.permute(0, 2, 1).reshape(w.shape[0], -1).contiguous(), b.contiguous()))
            return convs, (seq[14].weight.detach().float().contiguous(), seq[14].bias.detach().float().contiguous())

        def audio(seq):
            return [(seq[i].weight.detach().float().contiguous(), seq[i].bias.detach().float().contiguous())
                    for i in (0, 3, 6)]

        self.pre = {"ar_text": text(m.ar_text_prenet), "ar_audio": audio(m.ar_audio_prenet)}
        if self.Q > 1:
            self.pre["nar_text"] = text(m.nar_text_prenet)
            self.pre["nar_audio"] = audio(m.nar_audio_prenet)
        self.ar_audio_table = self._audio_prenet(m.ar_audio_embedding.weight.detach().float().contiguous(), "ar_audio")

    def _audio_prenet(self, x: torch.Tensor, which: str) -> torch.Tensor:
        (w1, b1), (w2, b2), (w3, b3) = self.pre[which]
        h = ops.linear(x, w1, b1, L.VB_EPI_RELU)
        h = ops.linear(h, w2, b2, L.VB_EPI_RELU)
        return ops.linear(h, w3, b3, L.VB_EPI_NONE)

    def _text_prenet(self, x: torch.Tensor, S: Sequence[int], which: str) -> torch.Tensor:
        """x: packed [sum(S), d] embedded phonemes, utterance after utterance -> the pre-net output, same layout; every
        utterance is convolved on its own with zero padding, as the reference's batch-1 call does (valle.py:995-996)"""
        convs, (wl, bl) = self.pre[which]
        R, d = x.shape
        starts = np.cumsum([0] + list(S[:-1]), dtype=np.int64)
        base, pos = _seg_ranges(starts, S)                   # row index, position inside its utterance
        lens = np.repeat(np.asarray(S, dtype=np.int64), S)
        idx = np.stack([np.where((pos + k - 2 >= 0) & (pos + k - 2 < lens), base + k - 2, -1) for k in range(5)])
        idx_d = torch.from_numpy(idx.astype(np.int32)).to(self.device)
        for (w, b) in convs:
            xc = torch.empty((R, 5 * d), dtype=torch.float32, device=self.device)
            for k in range(5):
                ops.gather_rows(x, idx_d[k], out=xc[:, k * d:(k + 1) * d])
            x = ops.linear(xc, w, b, L.VB_EPI_RELU)
        return ops.linear(x, wl, bl, L.VB_EPI_NONE)

    def _pe(self, module, n: int) -> torch.Tensor:
        return module.table(n, self.device)

    def _ada_tables(self) -> List[torch.Tensor]:
        if self._ada_cache is None:
            self._ada_cache = [self.nar.ada_table(e.weight) for e in self.model.nar_stage_embeddings]
        return self._ada_cache

    def _head(self, pe: torch.Tensor, mode: int) -> L.ArHead:
        m = self.model
        h = L.ArHead()
        h.predict_w = self.ar_predict_w.data_ptr()
        h.n_vocab, h.eos_id = self.n_vocab, NUM_AUDIO_TOKENS
        h.audio_emb = self.ar_audio_table.data_ptr()      # the embedding table, or pre-net(embedding) (add_prenet)
        h.alpha = m.ar_audio_position.alpha.detach().data_ptr()
        h.pe, h.pe_rows = pe.data_ptr(), pe.shape[0]
        h.greedy = mode          # 0 logits only, 1 argmax, 2 seeded sampling (vb_ar_head.greedy)
        if self.ar_head_fold is not None:
            h.fold = self.ar_head_fold
        return h

    def _buffers(self, B: int, cap: int, tok_stride: int) -> _ArBuffers:
        key = (B, cap, tok_stride)
        b = self._bufs.get(key)
        if b is None:
            if len(self._bufs) > 4:
                self._bufs.clear()
            b = _ArBuffers(self, B, cap, tok_stride)
            self._bufs[key] = b
        return b

    # ---- public API ----------------------------------------------------------------------
    @torch.no_grad()
    @_on_device
    def generate(self, texts: Sequence[torch.Tensor], prompts: Sequence[torch.Tensor],
                 enroll_lens: Optional[Sequence[int]] = None, top_k=1, temperature=1.0,
                 max_new_tokens: Optional[int] = None, poll: int = 32,
                 return_device: bool = False, trace: Optional[dict] = None,
                 forced: Optional[Sequence[torch.Tensor]] = None,
                 seeds: Optional[Sequence[int]] = None) -> List[torch.Tensor]:
        """texts[b]: int64 [S_b] phoneme ids; prompts[b]: int64 [Tp_b, Q] codec ids (host or device).
        Returns codes[b]: int64 [Tgen_b, Q] -- per utterance exactly what VALLE.inference returns.

        Sampling (valle.py:1040-1043): top_k == 1 decodes greedily.  Otherwise, without `seeds`, the ids are drawn with
        torch's generator as the reference draws them (one multinomial over the batch per step, or per utterance on the
        host with `sample_on_host`), so a draw depends on the batch it is part of.  With `seeds` (one int in [0, 2**64)
        per utterance) the draw runs in the sampler kernel inside the graph-replayed decode step and depends only on the
        utterance's logits, seed, step, top_k and temperature (include/valle_b200.h): the same utterance and seed give
        the same codes alone, in any batch slot or group, on any rank.  top_k and temperature may then be one value per
        utterance.

        Test hooks: `trace` collects AR logits (trace["steps"] = set of iterations or "all") and, with
        trace["nar"] = True, the NAR logits / argmax of every stage; `forced[b]` = int64 [T_b, Q] codes the decode is
        teacher-forced with (every sampled id is replaced by the given one before it is appended, AR and NAR), so
        that per-step logits can be compared with a reference that took exactly those ids."""
        self._refresh()
        m, dev, d, Q = self.model, self.device, self.d, self.Q
        B = len(texts)
        assert B == len(prompts) and B >= 1
        sampling = _sampling_params(B, seeds, top_k, temperature)
        if sampling is not None and self.sample_on_host:
            raise ValueError("seeds draw on the device: they cannot be combined with sample_on_host=True")
        if sampling is not None and forced is not None:
            raise ValueError("seeds cannot be combined with forced ids")
        if B > self.max_tc_batch and self.dtype == torch.bfloat16 and trace is None and forced is None:
            # the tensor-core decode projections take up to 64 rows (one UMMA N tile): a larger batch is decoded as
            # consecutive groups of <= 64 utterances instead of falling onto the CUDA-core GEMV path
            outs: List[torch.Tensor] = []
            stats = EngineStats()
            packed = []
            for b0 in range(0, B, self.max_tc_batch):
                b1 = min(B, b0 + self.max_tc_batch)
                if sampling is None:
                    k_g, t_g, s_g = top_k, temperature, None
                else:  # every utterance keeps its own seed and parameters
                    s_g, k_g, t_g = (v[b0:b1] for v in sampling)
                outs += self.generate(texts[b0:b1], prompts[b0:b1], None if enroll_lens is None else enroll_lens[b0:b1],
                                      k_g, t_g, max_new_tokens, poll, return_device, None, None, seeds=s_g)
                stats.ar_steps += self.stats.ar_steps
                stats.ar_ms += self.stats.ar_ms
                stats.prefill_ms += self.stats.prefill_ms
                stats.nar_ms += self.stats.nar_ms
                packed.append(self.last_packed)
            self.stats = stats
            self.last_packed = torch.cat(packed) if return_device else None
            return outs
        S = [int(t.numel()) for t in texts]
        Tp = [int(p.shape[0]) for p in prompts]
        assert all(s > 0 for s in S) and all(p.shape[1] == Q for p in prompts)
        _check_ids(texts, NUM_TEXT_TOKENS, "phoneme")
        _check_ids([p[:, :1] for p in prompts], NUM_AUDIO_TOKENS + 1, "prompt code (first codebook)")  # 1025-row tables
        _check_ids([p[:, 1:] for p in prompts], NUM_AUDIO_TOKENS, "prompt code")
        cap_new = [16 * s for s in S]  # valle.py:1047: stop when n_new > 16 * S
        if self.prepend_bos:
            # y carries the <BOS> the prompt does not: (y.shape[1] - prompts.shape[1]) = n_new + 1 (valle.py:1045-1047)
            cap_new = [c - 1 for c in cap_new]
        if max_new_tokens is not None:
            cap_new = [min(c, max_new_tokens - 1) for c in cap_new]
        tok_stride = (max(cap_new) + 2 + 7) // 8 * 8
        cap = (max(S[b] + Tp[b] + cap_new[b] + 2 for b in range(B)) + 63) // 64 * 64
        greedy = sampling is None and top_k == 1 and forced is None
        seeded = sampling is not None
        on_device = greedy or seeded  # the sampler kernel picks the id: decode steps replay as CUDA graphs
        forced_steps = None
        if forced is not None:  # [steps, B] first-codebook ids, EOS once an utterance's forced ids run out
            n_f = max(int(f.shape[0]) for f in forced) + 1
            forced_steps = torch.full((n_f + 1, B), NUM_AUDIO_TOKENS, dtype=torch.int64)
            for b, f in enumerate(forced):
                forced_steps[: f.shape[0], b] = f[:, 0].to(torch.int64).cpu()
            forced_steps = forced_steps.to(dev)
            cap_new = [min(c, int(f.shape[0])) for c, f in zip(cap_new, forced)]

        # ---- host -> device (once per batch) ----
        text_all = torch.cat([t.reshape(-1).to(torch.int64) for t in texts]).to(dev, non_blocking=True)
        prm_all = torch.cat([p.to(torch.int64) for p in prompts]).contiguous().to(dev, non_blocking=True)
        Tp_nar = Tp
        if self.prepend_bos:   # the AR stack sees [<BOS> | first-codebook prompt]; the NAR stages see the prompt only
            bos = torch.full((1,), NUM_AUDIO_TOKENS + 1, dtype=torch.int64)
            ar_tok = torch.cat([torch.cat([bos, p[:, 0].to(torch.int64).cpu()]) for p in prompts]).to(dev, non_blocking=True)
            Tp = [t + 1 for t in Tp]
        seq_len = [S[b] + Tp[b] for b in range(B)]
        cu = [0]
        for n in seq_len:
            cu.append(cu[-1] + n)
        M = cu[-1]
        cu_np = np.asarray(cu, dtype=np.int64)
        text_rows, text_pos = _seg_ranges(cu_np[:-1], S)
        aud_rows, aud_pos = _seg_ranges(cu_np[:-1] + np.asarray(S, dtype=np.int64), Tp)
        meta = torch.from_numpy(np.concatenate([cu_np, S, Tp, cap_new, text_rows, text_pos, aud_rows, aud_pos,
                                                cu_np[1:] - 1]).astype(np.int32)).to(dev, non_blocking=True)
        o = 0
        def take(n):
            nonlocal o
            v = meta[o:o + n]
            o += n
            return v
        cu_d, S_d, Tp_d, capn_d = take(B + 1), take(B), take(B), take(B)
        trow_d, tpos_d = take(sum(S)), take(sum(S))
        arow_d, apos_d = take(sum(Tp)), take(sum(Tp))
        last_d = take(B)

        ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
        ev[0].record()
        # ---- AR prefill (valle.py:995-997,1013-1016) ----
        buf = self._buffers(B, cap, tok_stride)
        buf.text_len.copy_(S_d)
        buf.prompt_len.copy_(Tp_d)
        buf.max_new.copy_(capn_d)
        buf.n_gen.zero_()
        buf.finished.zero_()
        if seeded:
            s_l, k_l, t_l = sampling
            buf.seed.copy_(torch.tensor([s - (1 << 64) if s >= 1 << 63 else s for s in s_l], dtype=torch.int64))
            buf.top_k.copy_(torch.tensor(k_l, dtype=torch.int32))
            buf.temperature.copy_(torch.tensor(t_l, dtype=torch.float32))
        pe_t = self._pe(m.ar_text_position, max(S))
        pe_a = self._pe(m.ar_audio_position, max(Tp) + max(cap_new) + 2)
        x = torch.empty((M, d), dtype=torch.float32, device=dev)
        self._embed_pe(text_all, 1, m.ar_text_embedding.weight, pe_t, m.ar_text_position.alpha, sum(S), x, trow_d, tpos_d,
                       prenet=("ar_text", S) if self.pre else None)
        if self.prepend_bos:
            self._embed_pe(ar_tok, 1, self.ar_audio_table, pe_a, m.ar_audio_position.alpha, sum(Tp), x, arow_d, apos_d)
        else:
            self._embed_pe(prm_all, Q, self.ar_audio_table, pe_a, m.ar_audio_position.alpha, sum(Tp), x, arow_d, apos_d)
        self.ar.forward(x, cu_d, B, max(seq_len), L.VB_MASK_VALLE_AR, S_d, None, buf.kcache, buf.vcache, cap)
        h_last = ops.gather_rows(x, last_d)
        head = self._head(pe_a, 2 if seeded else int(greedy))
        self._head_ref = head
        L.check(self.lib.vb_ar_head_step(self.ar.handle, C.byref(head), h_last.data_ptr(), C.byref(buf.st),
                                         buf.ws.data_ptr(), buf.ws.numel(), L.stream_ptr()), "vb_ar_head_step")
        def want(step):
            st_ = trace.get("steps", ())
            return st_ == "all" or step in st_
        if trace is not None:  # test hook: AR logits of selected iterations (iteration 0 = prefill)
            trace.setdefault("ar_logits", {})
            if want(0):
                trace["ar_logits"][0] = buf.logits[:, : self.n_vocab].clone()
            poll = 1
        if forced_steps is not None:
            poll = 1
        if not on_device:
            self._sample_push(buf, head, top_k, temperature, None if forced_steps is None else forced_steps[0])
        if any(t.is_cuda for t in list(texts) + list(prompts)):
            ops.check_oob(dev)  # ids that were already on the device are range-checked by the embedding kernels
        ev[1].record()

        # ---- AR decode loop (valle.py:1012-1057) ----
        max_steps = max(cap_new) + 1
        steps = 0
        while steps < max_steps:
            n = min(poll, max_steps - steps)
            if on_device and self.use_cuda_graph:
                # whole groups of `steps_per_graph` decode steps as one graph replay (no launch gap between the
                # steps of a group), the remainder one step at a time
                done = 0
                while done < n:
                    k = self.steps_per_graph if n - done >= self.steps_per_graph else 1
                    self._replay_steps(buf, head, k)
                    done += k
            else:
                for _ in range(n):
                    fs = None
                    if forced_steps is not None:
                        fs = forced_steps[min(steps + 1, forced_steps.shape[0] - 1)]
                    self._decode_step(buf, head, on_device, top_k, temperature, fs)
            steps += n
            if trace is not None and want(steps):  # poll == 1 here: the logits row of iteration `steps`
                trace["ar_logits"][steps] = buf.logits[:, : self.n_vocab].clone()
            if bool((buf.finished != 0).all()):  # one D2H sync per `poll` steps
                break
        self.stats.ar_steps = steps
        ev[2].record()
        n_gen = buf.n_gen.cpu().tolist()
        fin = buf.finished.cpu().tolist()
        if any(f == 2 for f in fin):
            raise SyntaxError("well trained model shouldn't reach here.")  # valle.py:1049-1052
        if not self.quiet:
            for b in range(B):
                print(f"VALL-E EOS [{Tp_nar[b]} -> {Tp[b] + n_gen[b]}]")  # valle.py:1054

        # ---- NAR (valle.py:1059-1137) ----
        Tg = n_gen
        cu_g = [0]
        for n in Tg:
            cu_g.append(cu_g[-1] + n)
        G = cu_g[-1]
        codes = torch.empty((G, Q), dtype=torch.int64, device=dev)
        src = torch.from_numpy(_seg_ranges(np.arange(B, dtype=np.int64) * tok_stride, Tg)[0]).to(dev)
        codes[:, 0] = buf.tokens.view(-1).index_select(0, src).to(torch.int64)
        if Q > 1:
            fc = None
            if forced is not None:
                fc = torch.cat([forced[b][: Tg[b]].to(torch.int64) for b in range(B)]).to(dev)
            self._nar(texts, text_all, prm_all, S, Tp_nar, Tg, cu_g, codes, enroll_lens, forced_codes=fc,
                      trace=trace if (trace is not None and trace.get("nar")) else None)
        ev[3].record()
        ev[3].synchronize()
        if any(t.is_cuda for t in list(texts) + list(prompts)):
            ops.check_oob(dev)
        self.stats.prefill_ms = ev[0].elapsed_time(ev[1])
        self.stats.ar_ms = ev[1].elapsed_time(ev[2])
        self.stats.nar_ms = ev[2].elapsed_time(ev[3])
        #: the packed [sum(Tgen), Q] device tensor behind the returned per-utterance views (dist.gather_codes ships it
        #: as is instead of re-packing the views)
        self.last_packed = codes
        if return_device:
            return [codes[cu_g[b]:cu_g[b + 1]] for b in range(B)]
        host = codes.cpu()
        return [host[cu_g[b]:cu_g[b + 1]] for b in range(B)]

    @torch.no_grad()
    @_on_device
    def continual(self, texts: Sequence[torch.Tensor], ys: Sequence[torch.Tensor]) -> List[torch.Tensor]:
        """VALLE.continual (valle.py:1139-1238): first-codebook codes are given, the 7 NAR stages
        predict the rest; prefix = min(T // 2, 225) frames."""
        self._refresh()
        dev, Q = self.device, self.Q
        B = len(texts)
        S = [int(t.numel()) for t in texts]
        T = [int(y.shape[0]) for y in ys]
        Tp = [min(int(t * 0.5), 3 * 75) for t in T]
        Tg = [T[b] - Tp[b] for b in range(B)]
        _check_ids(texts, NUM_TEXT_TOKENS, "phoneme")
        _check_ids([y_[:, :1] for y_ in ys], NUM_AUDIO_TOKENS + 1, "code (first codebook)")
        _check_ids([y_[:, 1:] for y_ in ys], NUM_AUDIO_TOKENS, "code")
        text_all = torch.cat([t.reshape(-1).to(torch.int64) for t in texts]).to(dev)
        prm_all = torch.cat([ys[b][:Tp[b]].to(torch.int64) for b in range(B)]).contiguous().to(dev)
        cu_g = [0]
        for n in Tg:
            cu_g.append(cu_g[-1] + n)
        codes = torch.empty((cu_g[-1], Q), dtype=torch.int64, device=dev)
        codes[:, 0] = torch.cat([ys[b][Tp[b]:, 0].to(torch.int64) for b in range(B)]).to(dev)
        self._nar(texts, text_all, prm_all, S, Tp, Tg, cu_g, codes, None, trim_text=False)
        if any(t.is_cuda for t in list(texts) + list(ys)):
            ops.check_oob(dev)
        return [codes[cu_g[b]:cu_g[b + 1]] for b in range(B)]

    def kernel_launches(self) -> int:
        """kernels of libvalle_b200.so executed so far by this process (direct + graph replays)."""
        return int(self.lib.vb_launch_count()) - self.captured_launches + self.replayed_launches

    # ---- helpers ---------------------------------------------------------------------------
    def _embed_pe(self, tokens, tok_stride, table, pe, alpha, n, x, rows, pos, prenet=None):
        """x[rows[r]] = prenet(table[tokens[r*tok_stride]]) + alpha * pe[pos[r]]  (embedding, pre-net, position:
        valle.py:994-997 / 1013-1015); prenet = (name, lengths) of a text pre-net or None (identity)."""
        tmp = torch.empty((n, table.shape[1]), dtype=torch.float32, device=self.device)
        ops.embed_sum(tokens, tok_stride, 0, [table.detach()], n, tmp)
        if prenet is not None:
            tmp = self._text_prenet(tmp, prenet[1], prenet[0])
        ops.add_pe(tmp, pe, alpha.detach(), x, n, positions=pos, out_rows=rows)

    def _decode_step(self, buf: _ArBuffers, head: L.ArHead, on_device: bool, top_k: int, temperature: float,
                     forced_step: Optional[torch.Tensor] = None):
        """one decode step; on_device: the sampler kernel picks the id (greedy or seeded), else _sample_push draws it"""
        if on_device and self.use_cuda_graph:
            key = (head.pe, head.predict_w, head.audio_emb, head.greedy)
            if buf.graph is not None and buf.graph_key != key:
                buf.graph = None
            if buf.graph is None:
                # warm-up launch (also sets function attributes), then capture the same call
                self._launch_step(buf, head)
                g = torch.cuda.CUDAGraph()
                n0 = self.lib.vb_launch_count()
                with torch.cuda.graph(g):
                    self._launch_step(buf, head)
                buf.graph_kernels = self.lib.vb_launch_count() - n0  # kernels inside one replay
                self.captured_launches += buf.graph_kernels      # recorded, not executed
                buf.graph = g
                buf.graph_head = head  # keep the struct alive
                buf.graph_key = key
                return  # the warm-up launch was this step
            buf.graph.replay()
            self.replayed_launches += buf.graph_kernels
            return
        self._launch_step(buf, head)
        if not on_device:
            self._sample_push(buf, head, top_k, temperature, forced_step)

    def _replay_steps(self, buf: _ArBuffers, head: L.ArHead, k: int):
        """k decode steps (greedy or seeded sampling) as ONE CUDA graph (captured on first use per (buffer, head tables,
        head mode, k)); the seeds and sampling parameters are read from the buffer's device arrays at every replay"""
        key = (head.pe, head.predict_w, head.audio_emb, head.greedy, k)
        graphs = buf.__dict__.setdefault("graphs", {})
        ent = graphs.get(key)
        if ent is None:
            if any(kk[:3] != key[:3] for kk in graphs):
                graphs.clear()                      # tables moved: the old captures hold stale pointers
            for _ in range(k):
                self._launch_step(buf, head)        # warm-up launches (function attributes) == these k steps
            g = torch.cuda.CUDAGraph()
            n0 = self.lib.vb_launch_count()
            with torch.cuda.graph(g):
                for _ in range(k):
                    self._launch_step(buf, head)
            kernels = self.lib.vb_launch_count() - n0
            self.captured_launches += kernels
            graphs[key] = (g, kernels, head)        # keep the head struct alive
            return                                  # the warm-up launches were these steps
        ent[0].replay()
        self.replayed_launches += ent[1]

    def _launch_step(self, buf, head: L.ArHead):
        L.check(self.lib.vb_ar_decode_step(self.ar.handle, C.byref(head), C.byref(buf.st), buf.ws.data_ptr(),
                                           buf.ws.numel(), L.stream_ptr()), "vb_ar_decode_step")

    def _sample_push(self, buf: _ArBuffers, head: L.ArHead, top_k: int, temperature: float,
                     forced_step: Optional[torch.Tensor] = None):
        """valle.py:1287-1302 topk_sampling with torch's own RNG stream (so a fixed torch seed gives
        the reference's draws), then the stop rule + append on the device."""
        if forced_step is not None:  # teacher forcing (test hook): the given ids instead of a draw
            samp = forced_step.contiguous()
            L.check(self.lib.vb_ar_push_tokens(C.byref(head), C.byref(buf.st), samp.data_ptr(), self.d,
                                               L.stream_ptr()), "vb_ar_push_tokens")
            return
        from .models.valle import topk_sampling
        logits = buf.logits[:, : self.n_vocab].clone()
        if self.sample_on_host:
            host = logits.cpu()
            samp = torch.cat([topk_sampling(host[b:b + 1], top_k=top_k, top_p=1.0, temperature=temperature).view(-1)
                              for b in range(host.shape[0])]).to(self.device)
        else:
            samp = topk_sampling(logits, top_k=top_k, top_p=1.0, temperature=temperature).view(-1).contiguous()
        L.check(self.lib.vb_ar_push_tokens(C.byref(head), C.byref(buf.st), samp.data_ptr(), self.d,
                                           L.stream_ptr()), "vb_ar_push_tokens")

    def _nar(self, texts, text_all, prm_all, S, Tp, Tg, cu_g, codes, enroll_lens, trim_text: bool = True,
             forced_codes: Optional[torch.Tensor] = None, trace: Optional[dict] = None):
        m, dev, d, Q = self.model, self.device, self.d_nar, self.Q
        B = len(S)
        pm = self.prefix_mode
        # text seen by the NAR decoder (valle.py:1068-1079)
        if pm in (2, 4) and trim_text:
            assert enroll_lens is not None
            keep = []
            off = 0
            S2 = []
            for b in range(B):
                e = int(enroll_lens[b])
                idx = [off] + list(range(off + e - 1, off + S[b]))
                keep += idx
                S2.append(len(idx))
                off += S[b]
            text_nar = text_all.index_select(0, torch.tensor(keep, dtype=torch.int64, device=dev))
        else:
            text_nar, S2 = text_all, list(S)
        T = [Tp[b] + Tg[b] for b in range(B)]
        Ltot = [S2[b] + T[b] for b in range(B)]
        cu = [0]
        for n in Ltot:
            cu.append(cu[-1] + n)
        M = cu[-1]
        cu_t = [0]
        for n in T:
            cu_t.append(cu_t[-1] + n)
        NT = cu_t[-1]
        cu_p = [0]
        for n in Tp:
            cu_p.append(cu_p[-1] + n)
        # index maps (host-built with numpy, one H2D)
        cu_np, cut_np = np.asarray(cu, dtype=np.int64), np.asarray(cu_t, dtype=np.int64)
        S2_np, Tp_np = np.asarray(S2, dtype=np.int64), np.asarray(Tp, dtype=np.int64)
        trow, tpos = _seg_ranges(cu_np[:-1], S2)
        yrow, ypos = _seg_ranges(cu_np[:-1] + S2_np, T)
        y_prompt_rows = _seg_ranges(cut_np[:-1], Tp)[0]
        y_gen_rows = _seg_ranges(cut_np[:-1] + Tp_np, Tg)[0]
        tgt_rows = _seg_ranges(cu_np[:-1] + S2_np + Tp_np, Tg)[0]
        meta = torch.from_numpy(np.concatenate([cu_np, trow, tpos, yrow, ypos, y_prompt_rows, y_gen_rows,
                                                tgt_rows]).astype(np.int32)).to(dev)
        o = 0
        def take(n):
            nonlocal o
            v = meta[o:o + n]
            o += n
            return v
        cu_d = take(B + 1)
        trow_d, tpos_d = take(sum(S2)), take(sum(S2))
        yrow_d, ypos_d = take(NT), take(NT)
        yp_d, yg_d, tgt_d = take(sum(Tp)), take(sum(Tg)), take(sum(Tg))
        G = sum(Tg)

        emb = [e.weight.detach() for e in m.nar_audio_embeddings]
        # y_emb = nar_audio_embeddings[0](y)  (valle.py:1064); rows packed [prompt_b | generated_b]
        y_emb = torch.empty((NT, d), dtype=torch.float32, device=dev)
        ops.embed_sum(prm_all, Q, 0, [emb[0]], sum(Tp), y_emb, out_rows=yp_d)
        ops.embed_sum(codes, Q, 0, [emb[0]], G, y_emb, out_rows=yg_d)
        if pm != 0:  # valle.py:1110-1113: prompt rows get all 8 codebooks up front, in order j=1..7
            ops.embed_sum(prm_all[:, 1:], Q, 1, emb[1:Q], sum(Tp), y_emb, out_rows=yp_d, accumulate=True)
        pe_t = self._pe(m.nar_text_position, max(S2))
        pe_a = self._pe(m.nar_audio_position, max(T))
        ada = self._ada_tables()
        x = torch.empty((M, d), dtype=torch.float32, device=dev)
        logits = torch.empty((G, NUM_AUDIO_TOKENS), dtype=torch.float32, device=dev)
        x_text = None
        if self.pre:   # valle.py:1081-1083: the text side (embedding, pre-net) is computed once for all stages
            x_text = torch.empty((sum(S2), d), dtype=torch.float32, device=dev)
            ops.embed_sum(text_nar, 1, 0, [m.nar_text_embedding.weight.detach()], sum(S2), x_text)
            x_text = self._text_prenet(x_text, S2, "nar_text")
        for i in range(Q - 1):
            # xy_pos = concat([nar_text_position(nar_text_embedding(text)), nar_audio_position(y_emb)])
            if x_text is not None:
                ops.add_pe(x_text, pe_t, m.nar_text_position.alpha.detach(), x, sum(S2), positions=tpos_d, out_rows=trow_d)
            else:
                self._embed_pe(text_nar, 1, m.nar_text_embedding.weight, pe_t, m.nar_text_position.alpha, sum(S2), x, trow_d, tpos_d)
            # valle.py:1092,1121: y_pos = nar_audio_position(nar_audio_prenet(y_emb))
            y_in = self._audio_prenet(y_emb, "nar_audio") if self.pre else y_emb
            ops.add_pe(y_in, pe_a, m.nar_audio_position.alpha.detach(), x, NT, positions=ypos_d, out_rows=yrow_d)
            self.nar.forward(x, cu_d, B, max(Ltot), L.VB_MASK_FULL, None, ada[i])
            hn = self.nar.final_norm(x, ada[i], rows=tgt_d, out_dtype=self.dtype)
            ops.linear(hn, self.nar_predict_w[i], None, L.VB_EPI_NONE, out=logits)
            nxt = emb[i + 1] if i < Q - 2 else None
            if trace is not None:
                trace.setdefault("nar_logits", []).append(logits.clone())
            if forced_codes is not None:  # teacher forcing (test hook): record the argmax, continue with the given ids
                ops.nar_argmax_accumulate(logits, codes[:, i + 1], codes.stride(0), None, None, yg_d)
                if trace is not None:
                    trace.setdefault("nar_argmax", []).append(codes[:, i + 1].clone())
                codes[:, i + 1] = forced_codes[:, i + 1]
                if nxt is not None:
                    ops.embed_sum(codes[:, i + 1:], Q, 0, [nxt], G, y_emb, out_rows=yg_d, accumulate=True)
            else:
                # samples -> codes[:, i+1]; y_emb[generated rows] += emb[i+1][samples]  (valle.py:1130-1134)
                ops.nar_argmax_accumulate(logits, codes[:, i + 1], codes.stride(0), nxt,
                                          y_emb if nxt is not None else None, yg_d)
            if pm == 0 and i < Q - 2:  # valle.py:1104-1107
                ops.embed_sum(prm_all[:, i + 1:], Q, 0, [emb[i + 1]], sum(Tp), y_emb, out_rows=yp_d, accumulate=True)
