"""BERT-base cross-encoders (hidden 768, 12 heads of 64, FFN 3072, two labels): the geometry of the default
"other" reranker, ms-marco-MultiBERT-L-12.  GPU parity against the float32 transformers oracle with seeded weights,
the default language routing end to end, and the host-side checks that run without a device."""

from __future__ import annotations

import ctypes
import json
import sys
import types

import numpy as np
import pytest
import torch

from bert_base_oracle import MULTIBERT_VOCAB, flashrank_logit_column, hf_flashrank_logits, multibert_config, seeded_bert_base
from oracle import rerank as orr

# Every length the attention kernel treats differently: 16 / 32 / 64-key tail blocks, one and several 64-query passes.
EDGE_LENGTHS = [1, 2, 3, 16, 31, 32, 33, 63, 64, 65, 200, 512]


def _pairs(lengths, vocab, rng):  # noqa: ANN001, ANN202
    ids, tys = [], []
    for L in lengths:
        a = rng.integers(1000, vocab, size=L).astype(np.int32)
        t = np.zeros(L, np.int32)
        if L >= 3:
            q = int(rng.integers(1, L - 1))
            a[0], a[q], a[-1] = 101, 102, 102
            t[q + 1:] = 1
        ids.append(a)
        tys.append(t)
    return ids, tys


def _check(got_logit, got_score, want):  # noqa: ANN001, ANN202
    from scipy.stats import kendalltau

    err = np.abs(got_logit - want).max()
    assert err < 4e-2, err
    assert np.abs(got_score - orr.flashrank_scores(want)).max() < 1e-2
    assert kendalltau(got_logit, want)[0] > 0.97


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_linear_layer_matches_torch_at_bert_base_shapes():
    from raglite_b200 import _lib

    lib = _lib.load()
    g = torch.Generator().manual_seed(0)
    # QKV, out-proj, FFN-up (GELU), FFN-down: all K = 768 / 3072, the streaming kernel
    for (T, N, K, act) in [(777, 2304, 768, 0), (1000, 768, 768, 0), (777, 3072, 768, 1), (1000, 768, 3072, 0)]:
        X = (torch.randn((T, K), generator=g) * 0.5).half().cuda()
        W = (torch.randn((N, K), generator=g) / K**0.5).float().cuda()
        b = torch.randn(N, generator=g).float().cuda()
        img = torch.empty(lib.rl_xenc_linear_image_bytes(N, K), dtype=torch.uint8, device="cuda")
        s = torch.cuda.current_stream().cuda_stream
        assert lib.rl_xenc_pack_linear(W.data_ptr(), N, K, img.data_ptr(), s) == 0
        Y = torch.empty((T, N), dtype=torch.float16, device="cuda")
        assert lib.rl_xenc_linear(X.data_ptr(), img.data_ptr(), b.data_ptr(), Y.data_ptr(), T, N, K, act, s) == 0, lib.rl_last_error()
        ref = X.float() @ W.half().float().T + b
        if act:
            ref = torch.nn.functional.gelu(ref)
        err = (Y.float() - ref).abs().max().item()
        assert err < 2e-2, (T, N, K, act, err)


@pytest.mark.gpu
@pytest.mark.parametrize("layers", [2, 12])
def test_bert_base_two_label_logits_match_transformers_fp32(layers):
    from raglite_b200._xenc import CrossEncoderEngine

    vocab = MULTIBERT_VOCAB if layers == 2 else 8000      # the full 105 879-row table once
    model = seeded_bert_base(seed=layers, num_hidden_layers=layers, vocab_size=vocab)
    eng = CrossEncoderEngine.from_hf(model, max_tokens_per_call=1500)     # forces several packed calls
    rng = np.random.default_rng(layers)
    lengths = EDGE_LENGTHS + [int(x) for x in rng.integers(4, 300, size=20)]
    ids, tys = _pairs(lengths, vocab, rng)
    ids[-1][1] = vocab - 1                                                # the last row of the embedding table
    ids[-2][1:3] = [vocab - 1, vocab - 2]
    got_logit, got_score = eng.score_tokens(ids, tys)
    _check(got_logit, got_score, hf_flashrank_logits(model, ids, tys))


@pytest.mark.gpu
def test_bert_base_one_label_logits_match_transformers_fp32():
    """head_dim 64 on its own, without the two-label column rule."""
    from raglite_b200._xenc import CrossEncoderEngine

    model = seeded_bert_base(seed=7, num_labels=1, num_hidden_layers=3, vocab_size=6000)
    eng = CrossEncoderEngine.from_hf(model, max_tokens_per_call=2000)
    rng = np.random.default_rng(7)
    ids, tys = _pairs(EDGE_LENGTHS + [int(x) for x in rng.integers(4, 300, size=12)], 6000, rng)
    got_logit, got_score = eng.score_tokens(ids, tys)
    want = orr.hf_logits(model, ids, tys, batch=16)
    _check(got_logit, got_score, want)


def _save_model(model, tok, path):  # noqa: ANN001, ANN202
    path.mkdir(parents=True)
    model.save_pretrained(path, safe_serialization=True)
    tok.save(str(path / "tokenizer.json"))


@pytest.mark.gpu
def test_default_routing_reranks_with_both_models(tmp_path, monkeypatch):
    """RAGLiteConfig's default {"en": MiniLM, "other": MultiBERT} shape: one call detected as English everywhere
    goes to "en", a mixed-language call to "other"; each returns the oracle's order."""
    from tokenizers import Tokenizer, models, pre_tokenizers, processors

    import raglite_b200 as rl
    from raglite_b200._rerank import B200CrossEncoderRanker

    words = ["[PAD]", "[UNK]", "[CLS]", "[SEP]"] + [f"w{i}" for i in range(200)]
    tok = Tokenizer(models.WordPiece({w: i for i, w in enumerate(words)}, unk_token="[UNK]"))
    tok.pre_tokenizer = pre_tokenizers.Whitespace()
    tok.post_processor = processors.TemplateProcessing(single="[CLS] $A [SEP]", pair="[CLS] $A [SEP] $B:1 [SEP]:1",
                                                       special_tokens=[("[CLS]", 2), ("[SEP]", 3)])
    minilm = orr.seeded_model(seed=5, num_hidden_layers=2, vocab_size=len(words))
    multibert = seeded_bert_base(seed=6, num_hidden_layers=2, vocab_size=len(words))
    _save_model(minilm, tok, tmp_path / "ms-marco-MiniLM-L-12-v2")
    _save_model(multibert, tok, tmp_path / "ms-marco-MultiBERT-L-12")
    assert json.loads((tmp_path / "ms-marco-MultiBERT-L-12" / "config.json").read_text())["hidden_size"] == 768
    rankers = {"en": B200CrossEncoderRanker("ms-marco-MiniLM-L-12-v2", cache_dir=tmp_path, max_length=128),
               "other": B200CrossEncoderRanker("ms-marco-MultiBERT-L-12", cache_dir=tmp_path, max_length=128)}
    cfg = rl.RAGLiteConfig(reranker=rankers)
    rng = np.random.default_rng(0)
    chunks = [rl.Chunk(id=f"c{i}", body=" ".join(f"w{j}" for j in rng.integers(0, 200, size=int(rng.integers(5, 140)))))
              for i in range(24)]
    query = "w1 w2 w3 w4"

    detected: list[str] = []
    fake = types.ModuleType("langdetect")
    fake.LangDetectException = type("LangDetectException", (Exception,), {})
    fake.detect = lambda text: detected.pop(0)
    monkeypatch.setitem(sys.modules, "langdetect", fake)

    def check_order(ranked, ranker, model):  # noqa: ANN001, ANN202
        ids, tys = ranker._engine.encode_pairs([query] * len(chunks), [str(c) for c in chunks])
        assert max(len(x) for x in ids) == 128                             # truncation applied
        ref_scores = orr.flashrank_scores(hf_flashrank_logits(model, ids, tys))
        want = orr.rank_order(ref_scores)
        got = [int(c.id[1:]) for c in ranked]
        assert sorted(got) == list(range(len(chunks)))
        for a, b in zip(got, want.tolist(), strict=True):
            assert a == b or abs(ref_scores[a] - ref_scores[b]) < 2e-2

    detected[:] = ["en"] * (len(chunks) + 1)
    ranked = rl.rerank_chunks(query, chunks, config=cfg)
    assert not detected                                                   # every chunk and the query were detected
    assert rankers["en"]._engine is not None and rankers["other"]._engine is None
    assert rankers["en"]._engine.hidden == 384
    check_order(ranked, rankers["en"], minilm)

    detected[:] = (["en", "de"] * len(chunks))[: len(chunks)] + ["en"]
    ranked = rl.rerank_chunks(query, chunks, config=cfg)
    assert not detected
    assert rankers["other"]._engine is not None and rankers["other"]._engine.hidden == 768
    check_order(ranked, rankers["other"], multibert)


# ---- no device needed -------------------------------------------------------------------------------------------
@pytest.mark.parametrize(("hidden", "heads"), [(768, 16), (1024, 16), (1024, 32), (600, 10)])
def test_score_rejects_unsupported_geometry_before_any_cuda_call(hidden, heads):
    """head_dim 48, H = 1024 (head_dim 64 or 32) and H % 32 != 0: RL_EUNSUPPORTED with the supported set, returned
    from the argument check (the pointers are never dereferenced and no device is needed)."""
    from raglite_b200 import _lib

    lib = _lib.load()
    layers = (_lib.XencLayer * 1)()
    w = _lib.XencWeights()
    w.n_layers, w.hidden, w.n_heads, w.ffn, w.vocab, w.max_pos, w.type_vocab = 1, hidden, heads, 4 * hidden, 100, 512, 2
    w.layers = ctypes.cast(layers, ctypes.POINTER(_lib.XencLayer))
    fake = 256   # never dereferenced
    rc = lib.rl_xenc_score(ctypes.byref(w), fake, fake, fake, fake, 4, 64, 16, fake, fake, fake, 1 << 30, None)
    assert rc == -4                                                  # RL_EUNSUPPORTED
    msg = lib.rl_last_error()
    assert b"head_dim 32 or 64" in msg and b"up to 768" in msg, msg


def test_classifier_row_follows_flashrank_column_rule():
    from raglite_b200._xenc import classifier_row, random_minilm_state_dict

    sd = random_minilm_state_dict(3, n_layers=1, hidden=768, ffn=3072, vocab=50, n_labels=2)
    W, b = sd["classifier.weight"], sd["classifier.bias"] + torch.tensor([0.25, -0.5])
    assert W.shape == (2, 768)
    row, bias = classifier_row(W, b)
    assert torch.equal(row, W[1]) and torch.equal(bias, b[1:2])
    one = random_minilm_state_dict(3, n_layers=1, vocab=50)
    row, bias = classifier_row(one["classifier.weight"], one["classifier.bias"])
    assert torch.equal(row, one["classifier.weight"][0]) and bias.shape == (1,)
    # the engine's row gives the logit FlashRank applies the sigmoid to
    h = torch.randn(5, 768, generator=torch.Generator().manual_seed(0))
    logits = (h @ W.T + b).numpy()
    row, bias = classifier_row(W, b)
    np.testing.assert_allclose((h @ row + bias).numpy(), flashrank_logit_column(logits), rtol=1e-6)
    with pytest.raises(ValueError, match="do not match"):
        classifier_row(W, torch.zeros(3))


def test_random_state_dict_defaults_are_unchanged():
    from raglite_b200._xenc import random_minilm_state_dict

    sd = random_minilm_state_dict(0, n_layers=1, vocab=100)
    assert sd["classifier.weight"].shape == (1, 384) and sd["classifier.bias"].shape == (1,)
    assert sd["bert.encoder.layer.0.intermediate.dense.weight"].shape == (1536, 384)


def test_multibert_config_and_missing_weights_message(tmp_path):
    from raglite_b200._rerank import B200CrossEncoderRanker

    cfg = multibert_config()
    assert (cfg.hidden_size, cfg.num_attention_heads, cfg.intermediate_size, cfg.num_labels) == (768, 12, 3072, 2)
    assert cfg.vocab_size == MULTIBERT_VOCAB and cfg.hidden_size // cfg.num_attention_heads == 64
    with pytest.raises(FileNotFoundError) as e:
        B200CrossEncoderRanker("ms-marco-MultiBERT-L-12", cache_dir=tmp_path).rank("q", ["d"])
    assert "BertForSequenceClassification" in str(e.value) and "cross-encoder/ms-marco-MultiBERT" not in str(e.value)
    with pytest.raises(FileNotFoundError) as e:
        B200CrossEncoderRanker("ms-marco-MiniLM-L-12-v2", cache_dir=tmp_path).rank("q", ["d"])
    assert "cross-encoder/ms-marco-MiniLM-L-12-v2" in str(e.value)
