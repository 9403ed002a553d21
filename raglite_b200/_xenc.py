"""BERT cross-encoder engine on the GPU -- the arithmetic behind ``rerank_chunks``.

The reference calls ``reranker.rank(query=, docs=)`` (``_search.py:395``) on a ``rerankers``
FlashRankRanker: tokenise (query, passage) pairs, run ms-marco-MiniLM-L-12-v2 (BERT, 12 layers, H=384,
12 heads, FFN=1536) or ms-marco-MultiBERT-L-12 (BERT-base: H=768, 12 heads of 64, FFN=3072, two labels)
with onnxruntime, sigmoid the logit, sort.  Here the forward runs in
``rl_xenc_score`` (hand-written CUDA: tcgen05 linear layers with fused bias/GELU, attention,
LayerNorm, pooler+classifier) on packed variable-length batches -- no padding tokens are computed.
"""

from __future__ import annotations

import ctypes as C
import threading
from collections.abc import Sequence
from pathlib import Path
from typing import Any

import numpy as np
import torch

from . import _lib
from ._lib import XencLayer, XencWeights, check


def _stream() -> int:
    return int(torch.cuda.current_stream().cuda_stream)


def random_minilm_state_dict(seed: int = 0, *, n_layers: int = 12, hidden: int = 384, ffn: int = 1536,
                             vocab: int = 30522, max_pos: int = 512, n_labels: int = 1) -> dict[str, torch.Tensor]:
    """Seeded random weights with the HF ``BertForSequenceClassification`` names/shapes of
    ms-marco-MiniLM-L-12-v2 (real weights cannot be downloaded offline); for benchmarks and smoke tests.
    ``hidden=768, ffn=3072, vocab=105879, n_labels=2`` gives the shapes of ms-marco-MultiBERT-L-12."""
    g = torch.Generator().manual_seed(seed)

    def w(*shape: int) -> torch.Tensor:
        return torch.randn(shape, generator=g) * 0.02

    sd = {
        "bert.embeddings.word_embeddings.weight": w(vocab, hidden),
        "bert.embeddings.position_embeddings.weight": w(max_pos, hidden),
        "bert.embeddings.token_type_embeddings.weight": w(2, hidden),
        "bert.embeddings.LayerNorm.weight": torch.ones(hidden), "bert.embeddings.LayerNorm.bias": torch.zeros(hidden),
        "bert.pooler.dense.weight": w(hidden, hidden), "bert.pooler.dense.bias": torch.zeros(hidden),
        "classifier.weight": w(n_labels, hidden) * 8.0, "classifier.bias": torch.zeros(n_labels),
    }
    for l in range(n_layers):
        p = f"bert.encoder.layer.{l}."
        for n in ("query", "key", "value"):
            sd[p + f"attention.self.{n}.weight"], sd[p + f"attention.self.{n}.bias"] = w(hidden, hidden), torch.zeros(hidden)
        sd[p + "attention.output.dense.weight"], sd[p + "attention.output.dense.bias"] = w(hidden, hidden), torch.zeros(hidden)
        sd[p + "attention.output.LayerNorm.weight"], sd[p + "attention.output.LayerNorm.bias"] = torch.ones(hidden), torch.zeros(hidden)
        sd[p + "intermediate.dense.weight"], sd[p + "intermediate.dense.bias"] = w(ffn, hidden), torch.zeros(ffn)
        sd[p + "output.dense.weight"], sd[p + "output.dense.bias"] = w(hidden, ffn), torch.zeros(hidden)
        sd[p + "output.LayerNorm.weight"], sd[p + "output.LayerNorm.bias"] = torch.ones(hidden), torch.zeros(hidden)
    return sd


def classifier_row(weight: torch.Tensor, bias: torch.Tensor) -> tuple[torch.Tensor, torch.Tensor]:
    """The classifier row and bias whose sigmoid is FlashRank's score: column 0 of a one-label model, column 1
    of a model with more labels (FlashRank scores ``sigmoid(logits[:, 1])`` then).  Returns ``([H], [1])``."""
    weight = weight.detach()
    weight = weight.reshape(1, -1) if weight.dim() == 1 else weight
    bias = bias.detach().reshape(-1)
    if weight.shape[0] != bias.numel() or weight.shape[0] < 1:
        raise ValueError(f"classifier weight {tuple(weight.shape)} and bias {tuple(bias.shape)} do not match")
    col = 1 if weight.shape[0] > 1 else 0
    return weight[col].contiguous(), bias[col:col + 1].contiguous()


class CrossEncoderEngine:
    """Device-resident packed weights + tokenizer + batching.

    Geometries: head_dim 32 or 64 and hidden a multiple of 32 up to 768 (MiniLM-L12-H384 and BERT-base).  The
    classifier may have any number of labels; the engine keeps the one FlashRank scores (``classifier_row``), so
    the returned ``logit`` is that column (``logits[:, 1]`` of a two-label model) and ``score`` its sigmoid."""

    def __init__(self, state_dict: dict[str, torch.Tensor], *, n_layers: int, hidden: int, n_heads: int, ffn: int,
                 max_pos: int, ln_eps: float = 1e-12, tokenizer: Any | None = None, max_length: int = 512,
                 device: Any | None = None, max_tokens_per_call: int = 1 << 18) -> None:
        if not torch.cuda.is_available():
            raise RuntimeError("raglite_b200 needs a CUDA device (there is no CPU fallback)")
        self.lib = _lib.load()
        self.device = torch.device(device if device is not None else f"cuda:{torch.cuda.current_device()}")
        self.tokenizer = tokenizer
        self.max_length = min(max_length, max_pos)
        self.max_tokens_per_call = max_tokens_per_call
        self.hidden, self.n_layers = hidden, n_layers
        self._keep: list[torch.Tensor] = []
        sd = {k.removeprefix("bert."): v for k, v in state_dict.items()}

        def f32(name: str) -> torch.Tensor:
            t = sd[name].detach().to(device=self.device, dtype=torch.float32).contiguous()
            self._keep.append(t)
            return t

        def f16(name: str) -> torch.Tensor:
            t = sd[name].detach().to(device=self.device, dtype=torch.float16).contiguous()
            self._keep.append(t)
            return t

        def packed(weight: torch.Tensor) -> torch.Tensor:
            W = weight.detach().to(device=self.device, dtype=torch.float32).contiguous()
            N, K = W.shape
            img = torch.empty(int(self.lib.rl_xenc_linear_image_bytes(N, K)), dtype=torch.uint8, device=self.device)
            with torch.cuda.device(self.device):
                check(self.lib.rl_xenc_pack_linear(W.data_ptr(), N, K, img.data_ptr(), _stream()), "rl_xenc_pack_linear")
                torch.cuda.current_stream().synchronize()
            self._keep.append(img)
            return img

        self._layers = (XencLayer * n_layers)()
        for l in range(n_layers):
            pre = f"encoder.layer.{l}."
            qkv_w = torch.cat([sd[pre + f"attention.self.{n}.weight"] for n in ("query", "key", "value")], dim=0)
            qkv_b = torch.cat([sd[pre + f"attention.self.{n}.bias"] for n in ("query", "key", "value")], dim=0)
            qkv_b = qkv_b.detach().to(device=self.device, dtype=torch.float32).contiguous()
            self._keep.append(qkv_b)
            L = self._layers[l]
            L.qkv_img, L.qkv_bias = packed(qkv_w).data_ptr(), qkv_b.data_ptr()
            L.o_img, L.o_bias = packed(sd[pre + "attention.output.dense.weight"]).data_ptr(), f32(pre + "attention.output.dense.bias").data_ptr()
            L.ln1_g, L.ln1_b = f32(pre + "attention.output.LayerNorm.weight").data_ptr(), f32(pre + "attention.output.LayerNorm.bias").data_ptr()
            L.up_img, L.up_bias = packed(sd[pre + "intermediate.dense.weight"]).data_ptr(), f32(pre + "intermediate.dense.bias").data_ptr()
            L.down_img, L.down_bias = packed(sd[pre + "output.dense.weight"]).data_ptr(), f32(pre + "output.dense.bias").data_ptr()
            L.ln2_g, L.ln2_b = f32(pre + "output.LayerNorm.weight").data_ptr(), f32(pre + "output.LayerNorm.bias").data_ptr()
        w = XencWeights()
        w.n_layers, w.hidden, w.n_heads, w.ffn = n_layers, hidden, n_heads, ffn
        w.vocab, w.max_pos = int(sd["embeddings.word_embeddings.weight"].shape[0]), max_pos
        w.type_vocab, w.ln_eps = int(sd["embeddings.token_type_embeddings.weight"].shape[0]), ln_eps
        w.word_emb = f16("embeddings.word_embeddings.weight").data_ptr()
        w.pos_emb = f16("embeddings.position_embeddings.weight").data_ptr()
        w.type_emb = f16("embeddings.token_type_embeddings.weight").data_ptr()
        w.emb_ln_g, w.emb_ln_b = f32("embeddings.LayerNorm.weight").data_ptr(), f32("embeddings.LayerNorm.bias").data_ptr()
        w.layers = C.cast(self._layers, C.POINTER(XencLayer))
        w.pooler_w, w.pooler_b = f32("pooler.dense.weight").data_ptr(), f32("pooler.dense.bias").data_ptr()
        cls_w, cls_b = classifier_row(state_dict["classifier.weight"], state_dict["classifier.bias"])
        if cls_w.numel() != hidden:
            raise ValueError(f"classifier rows have {cls_w.numel()} columns, the model's hidden size is {hidden}")
        cls_w = cls_w.to(device=self.device, dtype=torch.float32).contiguous()
        cls_b = cls_b.to(device=self.device, dtype=torch.float32).contiguous()
        self._keep += [cls_w, cls_b]
        w.cls_w, w.cls_b = cls_w.data_ptr(), cls_b.data_ptr()
        self.weights = w
        self._ws: torch.Tensor | None = None
        self._host_bufs: dict[str, torch.Tensor] = {}   # pinned staging (double-buffered inputs / outputs)
        self._dev_bufs: dict[int, torch.Tensor] = {}
        self._lock = threading.RLock()   # reference callers rerank from thread pools (_rag.py:317)

    # ---- constructors ------------------------------------------------------------------------------
    @classmethod
    def from_hf(cls, model: Any, tokenizer: Any | None = None, **kw: Any) -> "CrossEncoderEngine":
        """From a ``transformers.BertForSequenceClassification`` (any ``num_labels``, see ``classifier_row``)."""
        c = model.config
        return cls(model.state_dict(), n_layers=c.num_hidden_layers, hidden=c.hidden_size, n_heads=c.num_attention_heads,
                   ffn=c.intermediate_size, max_pos=c.max_position_embeddings, ln_eps=c.layer_norm_eps,
                   tokenizer=tokenizer, **kw)

    @classmethod
    def from_pretrained(cls, path: Path | str, **kw: Any) -> "CrossEncoderEngine":
        """Load HF weights + ``tokenizer.json`` from a local directory (no network access is attempted)."""
        path = Path(path)
        if not (path / "config.json").exists():
            raise FileNotFoundError(f"No cross-encoder weights at {path} (expected an HF model directory)")
        from tokenizers import Tokenizer
        from transformers import BertForSequenceClassification

        model = BertForSequenceClassification.from_pretrained(path, local_files_only=True)
        tok = Tokenizer.from_file(str(path / "tokenizer.json")) if (path / "tokenizer.json").exists() else None
        return cls.from_hf(model, tok, **kw)

    # ---- scoring ---------------------------------------------------------------------------------------
    def score_tokens(self, ids: Sequence[np.ndarray], type_ids: Sequence[np.ndarray]) -> tuple[np.ndarray, np.ndarray]:
        """Logits and sigmoid scores for already-tokenised pairs (variable lengths, no padding).

        The pairs are cut into calls of at most ``max_tokens_per_call`` tokens.  Calls are pipelined: while
        the GPU runs call *i*, the host packs call *i+1* into the other half of a pinned double buffer and
        enqueues its upload and kernels; results come back through pinned memory and are only waited for
        once the next call is in the queue -- the host packing disappears behind the forward."""
        P = len(ids)
        logits = np.empty(P, np.float32)
        scores = np.empty(P, np.float32)
        lens = np.fromiter((len(x) for x in ids), dtype=np.int64, count=P)
        if P and lens.max() > self.max_length:
            raise ValueError("sequence longer than max_length")
        cuts = [0]
        tok = 0
        for i in range(P):
            if i > cuts[-1] and tok + lens[i] > self.max_tokens_per_call:
                cuts.append(i)
                tok = 0
            tok += int(lens[i])
        cuts.append(P)
        with self._lock, torch.cuda.device(self.device):
            pending: tuple[int, int, torch.Tensor, torch.cuda.Event] | None = None
            for c in range(len(cuts) - 1):
                lo, hi = cuts[c], cuts[c + 1]
                if hi == lo:
                    continue
                item = self._launch_packed(ids[lo:hi], type_ids[lo:hi], lens[lo:hi], slot=c & 1)
                if pending is not None:
                    self._collect(pending, logits, scores)
                pending = (lo, hi, *item)
            if pending is not None:
                self._collect(pending, logits, scores)
        return logits, scores

    def _collect(self, pending: tuple[int, int, torch.Tensor, torch.cuda.Event], logits: np.ndarray, scores: np.ndarray) -> None:
        lo, hi, host, ev = pending
        ev.synchronize()
        res = host.numpy()[: 2 * (hi - lo)].reshape(2, hi - lo)
        logits[lo:hi], scores[lo:hi] = res[0], res[1]

    def _pinned(self, name: str, n: int, dtype: torch.dtype) -> torch.Tensor:
        buf = self._host_bufs.get(name)
        if buf is None or buf.numel() < n:
            buf = torch.empty(max(n, 1024), dtype=dtype, pin_memory=True)
            self._host_bufs[name] = buf
        return buf

    def _launch_packed(self, ids: Sequence[np.ndarray], type_ids: Sequence[np.ndarray], lens: np.ndarray, *, slot: int
                       ) -> tuple[torch.Tensor, torch.cuda.Event]:
        """Pack one call into pinned buffer ``slot``, enqueue upload + forward + download; returns the pinned
        result buffer and the event that marks it complete.  Caller holds the lock."""
        P, T = len(ids), int(lens.sum())
        n_in = 3 * T + P + 1
        host_in = self._pinned(f"in{slot}", n_in, torch.int32)
        h = host_in.numpy()
        np.concatenate(ids, out=h[:T], casting="unsafe")
        np.concatenate(type_ids, out=h[T:2 * T], casting="unsafe")
        cu = h[3 * T:3 * T + P + 1]
        cu[0] = 0
        np.cumsum(lens, out=cu[1:])
        h[2 * T:3 * T] = np.arange(T, dtype=np.int32) - np.repeat(cu[:-1], lens)      # position ids 0..len-1 per pair
        # A tokenizer that does not match the weights would index past the embedding tables.
        w = self.weights
        if T and (int(h[:T].min()) < 0 or int(h[:T].max()) >= w.vocab):
            raise ValueError(f"token id outside the model's vocabulary [0, {w.vocab}) -- tokenizer / weights mismatch?")
        if T and (int(h[T:2 * T].min()) < 0 or int(h[T:2 * T].max()) >= w.type_vocab):
            raise ValueError(f"token type id outside [0, {w.type_vocab})")
        if P and int(lens.max()) > w.max_pos:
            raise ValueError(f"sequence longer than the model's {w.max_pos} positions")
        dev = self._dev_bufs.get(slot)
        if dev is None or dev.numel() < n_in:
            dev = torch.empty(max(n_in, 1024), dtype=torch.int32, device=self.device)
            self._dev_bufs[slot] = dev
        dev[:n_in].copy_(host_in[:n_in], non_blocking=True)
        d_ids, d_types, d_pos, d_cu = dev[:T], dev[T:2 * T], dev[2 * T:3 * T], dev[3 * T:n_in]
        out = torch.empty((2, P), dtype=torch.float32, device=self.device)
        need = int(self.lib.rl_xenc_workspace_bytes(C.byref(self.weights), T))
        if self._ws is None or self._ws.numel() < need:
            self._ws = torch.empty(need, dtype=torch.uint8, device=self.device)
        check(self.lib.rl_xenc_score(C.byref(self.weights), d_ids.data_ptr(), d_types.data_ptr(), d_pos.data_ptr(),
                                     d_cu.data_ptr(), P, T, int(lens.max()), out[0].data_ptr(), out[1].data_ptr(),
                                     self._ws.data_ptr(), self._ws.numel(), _stream()), "rl_xenc_score")
        host_out = self._pinned(f"out{slot}", 2 * P, torch.float32)
        host_out[: 2 * P].copy_(out.reshape(-1), non_blocking=True)
        ev = torch.cuda.Event()
        ev.record()
        return host_out, ev

    def _score_packed(self, ids: Sequence[np.ndarray], type_ids: Sequence[np.ndarray], lens: np.ndarray
                      ) -> tuple[np.ndarray, np.ndarray]:
        """One synchronous call (kept for callers that time a single forward)."""
        with self._lock, torch.cuda.device(self.device):
            host, ev = self._launch_packed(ids, type_ids, np.asarray(lens, dtype=np.int64), slot=0)
            ev.synchronize()
            res = host.numpy()[: 2 * len(ids)].reshape(2, len(ids)).copy()
        return res[0], res[1]

    def encode_pairs(self, queries: Sequence[str], docs: Sequence[str]) -> tuple[list[np.ndarray], list[np.ndarray]]:
        """[CLS] query [SEP] passage [SEP] with truncation to ``max_length`` (FlashRank's tokenizer setup)."""
        if self.tokenizer is None:
            raise ValueError("this engine was built without a tokenizer; use score_tokens")
        self.tokenizer.enable_truncation(max_length=self.max_length)
        self.tokenizer.no_padding()
        enc = self.tokenizer.encode_batch(list(zip(queries, docs, strict=True)))
        return [np.asarray(e.ids, np.int32) for e in enc], [np.asarray(e.type_ids, np.int32) for e in enc]

    def score_pairs(self, queries: Sequence[str], docs: Sequence[str]) -> list[float]:
        ids, types = self.encode_pairs(queries, docs)
        return [float(s) for s in self.score_tokens(ids, types)[1]]
