"""CPU oracle pieces for BERT-base cross-encoders (TEST INFRASTRUCTURE), next to ``oracle.rerank``.

ms-marco-MultiBERT-L-12, the reference's default "other" reranker, is recalled (unpinned) as FlashRank's int8 ONNX
export of a fine-tuned bert-base-multilingual-uncased with a two-label classifier.  FlashRank scores a model with
more than one output column as ``sigmoid(logits[:, 1])`` and a one-column model as ``sigmoid(logits[:, 0])``.
"""

from __future__ import annotations

import numpy as np
import torch

from oracle import rerank as orr

MULTIBERT_VOCAB = 105879


def multibert_config(**over):  # noqa: ANN003, ANN201
    """ms-marco-MultiBERT-L-12's architecture: 12 layers, hidden 768, 12 heads of 64, FFN 3072, two labels."""
    cfg = dict(vocab_size=MULTIBERT_VOCAB, hidden_size=768, num_hidden_layers=12, num_attention_heads=12,
               intermediate_size=3072, max_position_embeddings=512, num_labels=2)
    cfg.update(over)
    return orr.minilm_config(**cfg)


def seeded_bert_base(seed: int = 0, **over):  # noqa: ANN003, ANN201
    """Deterministic random weights of that geometry, scaled like ``oracle.rerank.seeded_model`` so logits spread."""
    from transformers import BertForSequenceClassification

    torch.manual_seed(seed)
    model = BertForSequenceClassification(multibert_config(**over)).eval()
    with torch.no_grad():
        model.classifier.weight.mul_(8.0)
    return model


def flashrank_logit_column(logits: np.ndarray) -> np.ndarray:
    """The logit FlashRank applies the sigmoid to, from ``[P, num_labels]`` logits (a 1-D array is one column)."""
    logits = np.asarray(logits)
    if logits.ndim == 1:
        return logits
    return logits[:, 1] if logits.shape[1] > 1 else logits[:, 0]


def hf_flashrank_logits(model, ids, type_ids) -> np.ndarray:  # noqa: ANN001
    """``oracle.rerank.hf_logits`` (which flattens the logits) regrouped per pair, then FlashRank's column."""
    return flashrank_logit_column(orr.hf_logits(model, ids, type_ids, batch=16).reshape(len(ids), -1))
