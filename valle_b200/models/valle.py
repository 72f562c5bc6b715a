"""VALLE with the reference's constructor, parameter names / shapes (checkpoint layout), init order
and `forward()` / `inference()` / `continual()` signatures (valle/models/valle.py:722-1238), so
`bin/infer.py` and `bin/trainer.py` call it unchanged -- the loops underneath run on the sm_100a
engine (`valle_b200.engine.ValleEngine`, libvalle_b200.so).  No CPU fallback.
"""
from __future__ import annotations

import random
from typing import Dict, Iterator, List, Optional, Sequence, Tuple, Union

import torch
import torch.nn as nn
import torch.nn.functional as F

from ..modules.embedding import SinePositionalEmbedding, TokenEmbedding
from ..modules.transformer import AdaptiveLayerNorm, LayerNorm, TransformerEncoder, TransformerEncoderLayer
from .macros import NUM_AUDIO_TOKENS, NUM_TEXT_TOKENS


def top_k_top_p_filtering(logits: torch.Tensor, top_k: int = 0, top_p: float = 1.0,
                          filter_value: float = -float("Inf"), min_tokens_to_keep: int = 1) -> torch.Tensor:
    """valle/models/valle.py:1242-1284: keep the k largest logits (`logits < kth -> filter_value`, so ties with the
    k-th value survive, :1259) and / or the smallest nucleus whose probability mass reaches top_p; (batch, vocab)
    logits on any device, modified in place like the reference."""
    if top_k > 0:
        k = min(max(top_k, min_tokens_to_keep), logits.size(-1))
        kth = torch.topk(logits, k)[0][..., -1, None]
        logits[logits < kth] = filter_value
    if top_p < 1.0:
        srt, order = torch.sort(logits, descending=True)
        drop = torch.cumsum(F.softmax(srt, dim=-1), dim=-1) > top_p
        if min_tokens_to_keep > 1:
            drop[..., :min_tokens_to_keep] = 0
        drop[..., 1:] = drop[..., :-1].clone()   # the first token above the threshold stays
        drop[..., 0] = 0
        logits[drop.scatter(1, order, drop)] = filter_value
    return logits


def topk_sampling(logits: torch.Tensor, top_k: int = 10, top_p: float = 1.0, temperature: float = 1.0) -> torch.Tensor:
    """valle/models/valle.py:1287-1302: temperature, top-k / top-p filter, softmax, one torch.multinomial draw from
    the default generator of the logits' device -- the same RNG consumption as the reference's call."""
    if temperature != 1.0:
        logits = logits / temperature
    logits = top_k_top_p_filtering(logits, top_k=top_k, top_p=top_p)
    return torch.multinomial(F.softmax(logits, dim=-1), num_samples=1)


class PromptedFeatures:
    """valle/data/input_strategies.py:16-36 pair container accepted by forward() (prefix_mode 4)."""

    def __init__(self, prompts, features):
        self.prompts = prompts
        self.features = features

    def to(self, device):
        return PromptedFeatures(self.prompts.to(device), self.features.to(device))

    def sum(self):
        return self.features.sum()

    @property
    def ndim(self):
        return self.features.ndim

    @property
    def data(self):
        return (self.prompts, self.features)


class Transpose(nn.Identity):
    """(N, T, D) -> (N, D, T) (valle/utils/__init__.py); parameter-free, position 0 / 13 of the text pre-net"""

    def forward(self, input: torch.Tensor) -> torch.Tensor:
        return input.transpose(1, 2)


def _text_prenet(d: int) -> nn.Sequential:
    """valle.py:97-113 / 182-204: 3 x (Conv1d k=5 'same' -> BatchNorm1d -> ReLU -> Dropout(0.5)) between two
    transposes, then Linear.  Parameter container with the reference's state_dict keys (ar_text_prenet.1.weight ...);
    the arithmetic runs in the engine (ValleEngine._text_prenet)."""
    layers: List[nn.Module] = [Transpose()]
    for _ in range(3):
        layers += [nn.Conv1d(d, d, kernel_size=5, padding="same"), nn.BatchNorm1d(d), nn.ReLU(), nn.Dropout(0.5)]
    layers += [Transpose(), nn.Linear(d, d)]
    return nn.Sequential(*layers)


def _audio_prenet(d: int) -> nn.Sequential:
    """valle.py:115-123 / 205-213: Linear(d,256) ReLU Dropout(0.25) Linear(256,256) ReLU Dropout(0.25) Linear(256,d)"""
    return nn.Sequential(nn.Linear(d, 256), nn.ReLU(), nn.Dropout(0.25), nn.Linear(256, 256), nn.ReLU(),
                         nn.Dropout(0.25), nn.Linear(256, d))


class VALLE(nn.Module):
    """Decoder-only VALL-E (https://arxiv.org/abs/2301.02111): AR stack + NAR stack."""

    def __init__(self, d_model: int, nhead: int, num_layers: int, norm_first: bool = True,
                 add_prenet: bool = False, prefix_mode: int = 0, share_embedding: bool = True,
                 nar_scale_factor: float = 1.0, **kwargs):
        super().__init__()
        prepend_bos = bool(kwargs.pop("prepend_bos", False))
        num_quantizers = int(kwargs.pop("num_quantizers", 8))
        if not norm_first:
            raise NotImplementedError(
                "valle_b200.VALLE: post-LN (norm_first=False) is not built; add_prenet, prepend_bos and "
                "nar_scale_factor are (DESIGN.md section 7)")
        self.add_prenet = bool(add_prenet)
        nar_d_model = int(d_model * nar_scale_factor)
        if nar_d_model % 256 != 0 or nar_d_model // max(1, int(nhead * nar_scale_factor)) != 64:
            raise NotImplementedError("valle_b200.VALLE: nar_scale_factor must keep d_model a multiple of 256 and 64-wide heads")
        # creation order == valle.py:85-259 so that a fixed torch seed yields the reference's weights
        self.ar_text_embedding = TokenEmbedding(d_model, NUM_TEXT_TOKENS)
        self.nar_text_embedding = TokenEmbedding(nar_d_model, NUM_TEXT_TOKENS)
        self.ar_audio_prepend_bos = prepend_bos
        self.ar_audio_embedding = TokenEmbedding(d_model, NUM_AUDIO_TOKENS + 1 + int(prepend_bos))
        self.ar_text_prenet = _text_prenet(d_model) if add_prenet else nn.Identity()
        self.ar_audio_prenet = _audio_prenet(d_model) if add_prenet else nn.Identity()
        self.ar_text_position = SinePositionalEmbedding(d_model, dropout=0.1, scale=False, alpha=True)
        self.ar_audio_position = SinePositionalEmbedding(d_model, dropout=0.1, scale=False, alpha=True)
        self.ar_decoder = TransformerEncoder(
            TransformerEncoderLayer(d_model, nhead, dim_feedforward=d_model * 4, dropout=0.1,
                                    batch_first=True, norm_first=norm_first),
            num_layers=num_layers, norm=LayerNorm(d_model) if norm_first else None)
        self.ar_predict_layer = nn.Linear(d_model, NUM_AUDIO_TOKENS + 1, bias=False)
        self.rng = random.Random(0)
        self.num_heads = nhead
        self.prefix_mode = prefix_mode
        self.num_quantizers = num_quantizers
        assert num_quantizers >= 1
        if num_quantizers > 1:
            self.nar_audio_embeddings = nn.ModuleList(
                [TokenEmbedding(nar_d_model, NUM_AUDIO_TOKENS + 1)]
                + [TokenEmbedding(nar_d_model, NUM_AUDIO_TOKENS) for _ in range(num_quantizers - 1)])
            self.nar_text_prenet = _text_prenet(nar_d_model) if add_prenet else nn.Identity()
            self.nar_audio_prenet = _audio_prenet(nar_d_model) if add_prenet else nn.Identity()
            self.nar_text_position = SinePositionalEmbedding(nar_d_model, dropout=0.0, scale=False, alpha=False)
            self.nar_audio_position = SinePositionalEmbedding(nar_d_model, dropout=0.1, scale=False, alpha=False)
            self.nar_decoder = TransformerEncoder(
                TransformerEncoderLayer(nar_d_model, int(nhead * nar_scale_factor),
                                        dim_feedforward=nar_d_model * 4, dropout=0.1, batch_first=True,
                                        norm_first=norm_first, adaptive_layer_norm=True),
                num_layers=int(num_layers * nar_scale_factor),
                norm=AdaptiveLayerNorm(nar_d_model, norm=nn.LayerNorm(nar_d_model)) if norm_first else None)
            self.nar_predict_layers = nn.ModuleList(
                [nn.Linear(nar_d_model, NUM_AUDIO_TOKENS, bias=False) for _ in range(num_quantizers - 1)])
            self.nar_stage_embeddings = nn.ModuleList(
                [TokenEmbedding(nar_d_model, 1) for _ in range(num_quantizers - 1)])
            if share_embedding:  # valle.py:261-271
                for j in range(0, num_quantizers - 2):
                    self.nar_predict_layers[j].weight = self.nar_audio_embeddings[j + 2].weight
        self._engines: Dict[torch.dtype, object] = {}
        #: storage/compute type of the engine used by inference(): torch.float32 (bit-exact greedy
        #: parity with the reference) or torch.bfloat16 (tensor-core path)
        self.engine_dtype = torch.float32

    # ---- reference helper API (valle.py:294-333) --------------------------------------------
    def stage_parameters(self, stage: int = 1) -> Iterator[nn.Parameter]:
        """parameters of training stage 1 (ar_*) or 2 (nar_*), valle.py:294-306"""
        assert stage > 0
        prefix = "ar_" if stage == 1 else "nar_"
        label = " AR" if stage == 1 else "NAR"
        if stage in (1, 2):
            for name, param in self.named_parameters():
                if name.startswith(prefix):
                    print(f"{label} parameter: {name}")
                    yield param

    def stage_named_parameters(self, stage: int = 1) -> Iterator[Tuple[str, nn.Parameter]]:
        """valle.py:308-320"""
        assert stage > 0
        prefix = "ar_" if stage == 1 else "nar_"
        if stage in (1, 2):
            for pair in self.named_parameters():
                if pair[0].startswith(prefix):
                    yield pair

    def pad_y_eos(self, y, y_mask_int, eos_id):
        """append EOS after the last valid frame and split into (input, target), valle.py:322-333; with prepend_bos the
        inputs are [BOS, y...] and the targets keep every position (:329-332)"""
        targets = F.pad(y, (0, 1), value=0) + eos_id * F.pad(y_mask_int, (0, 1), value=1)
        if self.ar_audio_prepend_bos:
            return F.pad(targets[:, :-1], (1, 0), value=NUM_AUDIO_TOKENS + 1), targets
        return targets[:, :-1], targets[:, 1:]

    # ---- engine -------------------------------------------------------------------------------
    def engine(self, dtype: Optional[torch.dtype] = None):
        """the batched decode engine bound to this model's parameters (one per storage dtype; `engine_dtype` default)"""
        from ..engine import ValleEngine
        dtype = dtype or self.engine_dtype
        e = self._engines.get(dtype)
        if e is None or e.device != self.ar_predict_layer.weight.device:
            e = ValleEngine(self, dtype)
            self._engines[dtype] = e
        return e

    def __getstate__(self):
        st = self.__dict__.copy()
        st["_engines"] = {}
        return st

    def __deepcopy__(self, memo):
        import copy
        new = self.__class__.__new__(self.__class__)
        memo[id(self)] = new
        for k, v in self.__dict__.items():
            new.__dict__[k] = {} if k == "_engines" else copy.deepcopy(v, memo)
        return new

    # ---- inference (valle.py:961-1137) ------------------------------------------------------
    @torch.no_grad()
    def inference(self, x: torch.Tensor, x_lens: torch.Tensor, y: torch.Tensor,
                  enroll_x_lens: Optional[torch.Tensor] = None, top_k: int = -100,
                  temperature: float = 1.0, max_new_tokens: Optional[int] = None,
                  seed: Optional[int] = None) -> torch.Tensor:
        """x: (1, S) phoneme ids, x_lens: (1,), y: (1, T, 8) acoustic prompt.
        Returns the predicted audio code matrix (1, T', 8) -- same contract as the reference.
        seed (engine feature, int in [0, 2**64)): draw on the device keyed by this seed instead of torch's generator, so
        the same call reproduces the same codes, alone or inside any inference_batch (ValleEngine.generate)."""
        assert x.ndim == 2, x.shape
        assert x_lens.ndim == 1, x_lens.shape
        assert y.ndim == 3, y.shape
        assert y.shape[0] == 1, y.shape
        assert torch.all(x_lens > 0)
        S = int(x_lens.max())
        enroll = [int(enroll_x_lens.max())] if (self.prefix_mode in (2, 4) and enroll_x_lens is not None) else None
        out = self.engine().generate([x[0, :S]], [y[0]], enroll_lens=enroll, top_k=top_k,
                                     temperature=temperature, max_new_tokens=max_new_tokens,
                                     return_device=True, seeds=None if seed is None else [seed])
        return out[0].unsqueeze(0).to(y.device)

    @torch.no_grad()
    def inference_batch(self, texts: Sequence[torch.Tensor], prompts: Sequence[torch.Tensor],
                        enroll_lens: Optional[Sequence[int]] = None, top_k: int = 1,
                        temperature: float = 1.0, max_new_tokens: Optional[int] = None,
                        dtype: Optional[torch.dtype] = None, return_device: bool = False,
                        seeds: Optional[Sequence[int]] = None) -> List[torch.Tensor]:
        """Engine feature (the reference asserts batch 1, valle.py:989): B independent utterances
        decoded together; result[b] equals `inference()` on utterance b alone.  Codes come back on the host, or
        (return_device=True) stay on the GPU, e.g. for the data-parallel gather of valle_b200.dist.
        seeds: one int per utterance for seeded sampling on the device; top_k / temperature may then be per utterance
        (ValleEngine.generate)."""
        return self.engine(dtype).generate(texts, prompts, enroll_lens=enroll_lens, top_k=top_k,
                                           temperature=temperature, max_new_tokens=max_new_tokens,
                                           return_device=return_device, seeds=seeds)

    @torch.no_grad()
    def continual(self, x: torch.Tensor, x_lens: torch.Tensor, y: torch.Tensor) -> torch.Tensor:
        """valle.py:1139-1238: NAR-only continuation of given first-codebook codes."""
        assert x.ndim == 2, x.shape
        assert x_lens.ndim == 1, x_lens.shape
        assert y.ndim == 3, y.shape
        assert y.shape[0] == 1, y.shape
        assert torch.all(x_lens > 0)
        assert self.num_quantizers == 8
        S = int(x_lens.max())
        out = self.engine().continual([x[0, :S]], [y[0]])
        return out[0].unsqueeze(0).to(y.device)

    # ---- training forward (valle.py:762-959) ------------------------------------------------
    def forward(self, x: torch.Tensor, x_lens: torch.Tensor, y: Union[torch.Tensor, PromptedFeatures],
                y_lens: Union[torch.Tensor, PromptedFeatures], reduction: str = "sum", train_stage: int = 0,
                **kwargs):
        """VALLE.forward (valle.py:762-959), forward only: ((x, codes), loss, metrics) with the reference's loss value in
        eval mode; raises in training mode (no backward pass is built) -> train_forward.valle_forward"""
        from ..train_forward import valle_forward
        return valle_forward(self, x, x_lens, y, y_lens, reduction=reduction, train_stage=train_stage, **kwargs)
