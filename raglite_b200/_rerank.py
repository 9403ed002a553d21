"""Cross-encoder rankers with the ``rerankers.BaseRanker`` calling convention used by
``rerank_chunks`` (reference ``_search.py:395-396``): ``rank(query=, docs=)`` returns an object whose
``.results`` are ordered best-first and carry ``.doc_id`` (index into ``docs``) and ``.score``."""

from __future__ import annotations

from collections.abc import Callable, Sequence
from dataclasses import dataclass
from pathlib import Path
from typing import Any


@dataclass
class Document:
    text: str
    doc_id: int


@dataclass
class Result:
    document: Document
    score: float
    rank: int

    @property
    def doc_id(self) -> int:
        return self.document.doc_id

    @property
    def text(self) -> str:
        return self.document.text


@dataclass
class RankedResults:
    results: list[Result]
    query: str
    has_scores: bool = True

    def top_k(self, k: int) -> list[Result]:
        return self.results[:k]


class ScoreFnRanker:
    """Rank with any ``score(query, docs) -> sequence of floats`` callable."""

    def __init__(self, score_fn: Callable[[str, Sequence[str]], Sequence[float]]):
        self.score_fn = score_fn

    def rank(self, query: str, docs: Sequence[str], doc_ids: Sequence[int] | None = None) -> RankedResults:
        scores = [float(s) for s in self.score_fn(query, docs)]
        ids = list(doc_ids) if doc_ids is not None else list(range(len(docs)))
        order = sorted(range(len(docs)), key=lambda i: -scores[i])
        results = [Result(Document(docs[i], ids[i]), scores[i], r + 1) for r, i in enumerate(order)]
        return RankedResults(results, query)


# Where the Hugging Face weights of the default rerankers (RAGLiteConfig) come from.  FlashRank's
# ms-marco-MultiBERT-L-12 is an ONNX export with no known Hugging Face twin, so none is named for it.
HF_SOURCES = {"ms-marco-MiniLM-L-12-v2": "cross-encoder/ms-marco-MiniLM-L-12-v2"}


class B200CrossEncoderRanker(ScoreFnRanker):
    """BERT cross-encoder scored on the GPU: any ``BertForSequenceClassification`` with head_dim 32 or 64 and
    hidden size up to 768, which covers both default rerankers (ms-marco-MiniLM-L-12-v2, H=384, and the BERT-base
    ms-marco-MultiBERT-L-12, H=768).  Weights are loaded lazily from ``cache_dir/<model_name>`` (HF
    ``config.json`` + ``safetensors`` + ``tokenizer.json``)."""

    def __init__(self, model_name: str, *, cache_dir: Path | str | None = None, max_length: int = 512,
                 device: Any | None = None):
        self.model_name = model_name
        self.cache_dir = Path(cache_dir) if cache_dir is not None else None
        self.max_length = max_length
        self.device = device
        self._engine: Any | None = None
        super().__init__(self._score)

    def _score(self, query: str, docs: Sequence[str]) -> Sequence[float]:
        if self._engine is None:
            from ._xenc import CrossEncoderEngine

            path = (self.cache_dir / self.model_name) if self.cache_dir else Path(self.model_name)
            if not (path / "config.json").exists():
                source = HF_SOURCES.get(self.model_name)
                where = (f"e.g. `huggingface-cli download {source} --local-dir {path}`" if source else
                         "a BERT-base-style BertForSequenceClassification directory converted from the model")
                raise FileNotFoundError(
                    f"B200CrossEncoderRanker: no Hugging Face model directory at {path}.  The reference's FlashRank "
                    "reranker downloads an ONNX file on first use; this ranker needs the same model as HF weights "
                    f"(config.json + model.safetensors + tokenizer.json; {where}), or pass any object with a "
                    ".rank(query=, docs=) method as RAGLiteConfig.reranker (None disables reranking).  See INTEGRATION.md.")
            self._engine = CrossEncoderEngine.from_pretrained(path, max_length=self.max_length, device=self.device)
        return self._engine.score_pairs([query] * len(docs), list(docs))
