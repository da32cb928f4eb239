"""GPU text encoders behind the reference's own encoder interfaces (SURVEY §8 f2 / f3).

* ``GpuSentenceEncoder`` stands in for ``SentenceTransformer("all-MiniLM-L6-v2")`` where the reference calls
  ``self.model.encode(texts)`` / ``get_sentence_embedding_dimension()`` / ``max_seq_length``
  (rag_search_engine/utils/semantic_search.py:45-46, :200, :221, :372): pass it as ``SemanticSearch(encoder=...)``.
* ``GpuCrossEncoder`` stands in for ``CrossEncoder("cross-encoder/ms-marco-TinyBERT-L2-v2").predict(pairs)``
  (rag_search_engine/utils/hybrid_search.py:296-297): pass it as ``HybridSearch(cross_encoder=...)``.

Both run csrc/encoder.cuh through the C-ABI (``rse_encoder_*``, ``rse_encode``): HuggingFace BERT weights handed
over under their state_dict names, fp32 throughout.  Tokenisation stays on the host and is pluggable: a
HuggingFace tokenizer when one is available (``from_sentence_transformer`` / ``from_cross_encoder`` take it from
the loaded reference model), or any callable returning token-id lists.  No weights are bundled and nothing is
downloaded: without ``sentence-transformers`` (and its checkpoints) on the machine the caller supplies a
``state_dict`` — the tests use a randomly initialised ``transformers.BertModel`` of the same architecture.
"""
from __future__ import annotations

from typing import Callable, Dict, List, Optional, Sequence

import itertools

import numpy as np

MINILM_L6_CONFIG = dict(vocab_size=30522, hidden=384, layers=6, heads=12, intermediate=1536, max_positions=512,
                        type_vocab=2, ln_eps=1e-12)          # sentence-transformers/all-MiniLM-L6-v2 config.json
TINYBERT_L2_CONFIG = dict(vocab_size=30522, hidden=128, layers=2, heads=2, intermediate=512, max_positions=512,
                          type_vocab=2, ln_eps=1e-12)        # cross-encoder/ms-marco-TinyBERT-L2-v2 config.json


def config_from_hf(cfg) -> dict:
    """transformers BertConfig -> the keyword arguments of ``Index.encoder_create``."""
    if getattr(cfg, "hidden_act", "gelu") != "gelu":
        raise ValueError("only the erf GELU of BERT is implemented")
    if getattr(cfg, "position_embedding_type", "absolute") != "absolute":
        raise ValueError("only absolute position embeddings are implemented")
    return dict(vocab_size=cfg.vocab_size, hidden=cfg.hidden_size, layers=cfg.num_hidden_layers,
                heads=cfg.num_attention_heads, intermediate=cfg.intermediate_size,
                max_positions=cfg.max_position_embeddings, type_vocab=cfg.type_vocab_size,
                ln_eps=cfg.layer_norm_eps)


def _load(index, slot: int, config: dict, head: int, state_dict) -> None:
    index.encoder_create(slot, head=head, **config)
    for name, t in state_dict.items():
        a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
        if a.dtype.kind != "f" or name.endswith("position_ids"):
            continue                                            # integer buffers (position_ids) are not weights
        if not any(k in name for k in ("embeddings.", "encoder.layer.", "pooler.", "classifier.")):
            continue
        index.encoder_set_tensor(slot, name, a.astype(np.float32))
    index.encoder_finalize(slot)


def random_state_dict(config: dict, seed: int = 0, head: int = 0) -> Dict[str, np.ndarray]:
    """A seeded random BERT of the given architecture under HuggingFace names — for benches and smoke tests on
    machines without the reference's checkpoints (the arithmetic does not depend on what the weights are)."""
    rng = np.random.default_rng(seed)
    H, I = config["hidden"], config["intermediate"]
    f = lambda *shape, scale=1.0: (scale * rng.standard_normal(shape)).astype(np.float32)      # noqa: E731
    sd = {"embeddings.word_embeddings.weight": f(config["vocab_size"], H, scale=0.5),
          "embeddings.position_embeddings.weight": f(config["max_positions"], H, scale=0.5),
          "embeddings.token_type_embeddings.weight": f(config["type_vocab"], H, scale=0.5),
          "embeddings.LayerNorm.weight": 1.0 + f(H, scale=0.1), "embeddings.LayerNorm.bias": f(H, scale=0.05)}
    for i in range(config["layers"]):
        p = f"encoder.layer.{i}."
        for nm, (o, k) in {"attention.self.query": (H, H), "attention.self.key": (H, H), "attention.self.value": (H, H),
                           "attention.output.dense": (H, H), "intermediate.dense": (I, H), "output.dense": (H, I)}.items():
            sd[p + nm + ".weight"] = f(o, k, scale=k ** -0.5)
            sd[p + nm + ".bias"] = f(o, scale=0.05)
        for nm in ("attention.output.LayerNorm", "output.LayerNorm"):
            sd[p + nm + ".weight"] = 1.0 + f(H, scale=0.1)
            sd[p + nm + ".bias"] = f(H, scale=0.05)
    if head == 1:
        sd.update({"pooler.dense.weight": f(H, H, scale=H ** -0.5), "pooler.dense.bias": f(H, scale=0.05),
                   "classifier.weight": f(1, H, scale=H ** -0.5), "classifier.bias": f(1, scale=0.05)})
    return sd


def pack(id_lists: Sequence[Sequence[int]], type_lists: Optional[Sequence[Sequence[int]]] = None):
    """Token-id lists -> (ids int32[T], type_ids int32[T] | None, cu_seqlens int32[n + 1])."""
    lens = np.fromiter(map(len, id_lists), np.int64, count=len(id_lists))
    cu = np.zeros(len(id_lists) + 1, np.int32)
    np.cumsum(lens, out=cu[1:])
    total = int(cu[-1])

    def flat(lists):
        # itertools.chain keeps the walk over the tokens in C (a generator expression costs ~50 ns per token: 10 ms for
        # the 200 k tokens of a 64-query rerank batch)
        if total and all(isinstance(x, np.ndarray) for x in lists):
            return np.concatenate(lists).astype(np.int32, copy=False)
        return np.fromiter(itertools.chain.from_iterable(lists), np.int32, count=total)
    ids = flat(id_lists)
    tt = flat(type_lists) if type_lists is not None else None
    return ids, tt, cu


def hf_text_tokenizer(hf_tok) -> Callable[[List[str]], List[List[int]]]:
    """A HuggingFace tokenizer as the single-text tokenizer of the batched rerank: ids without special tokens.  With a
    fast tokenizer these are exactly the segments its pair encoding (truncation=True) is built from."""
    return lambda texts: hf_tok(list(texts), add_special_tokens=False)["input_ids"]


class GpuSentenceEncoder:
    """``encode(texts) -> float32[n, hidden]`` like SentenceTransformer.encode (normalised mean-pooled BERT)."""

    def __init__(self, index, state_dict, config: dict = MINILM_L6_CONFIG,
                 tokenizer: Optional[Callable[[List[str]], List[List[int]]]] = None, *, slot: int = 0,
                 max_seq_length: int = 256):
        self.index, self.slot, self.config = index, slot, dict(config)
        self.tokenizer = tokenizer
        self.max_seq_length = min(int(max_seq_length), int(config["max_positions"]))       # semantic_search.py:372
        _load(index, slot, self.config, 0, state_dict)

    @classmethod
    def from_sentence_transformer(cls, index, st_model, *, slot: int = 0) -> "GpuSentenceEncoder":
        """From a loaded ``SentenceTransformer`` (the object semantic_search.py:45 builds): its BertModel weights,
        its tokenizer and its max_seq_length."""
        bert = st_model[0].auto_model
        hf_tok = st_model.tokenizer
        msl = int(getattr(st_model, "max_seq_length", 256) or 256)
        tok = lambda texts: hf_tok(list(texts), truncation=True, max_length=msl)["input_ids"]   # noqa: E731
        return cls(index, bert.state_dict(), config_from_hf(bert.config), tok, slot=slot, max_seq_length=msl)

    def get_sentence_embedding_dimension(self) -> int:
        return int(self.config["hidden"])

    def encode_ids(self, id_lists: Sequence[Sequence[int]], max_tokens_per_call: int = 1 << 16) -> np.ndarray:
        """Any number of sequences: the bulk embedding of an index build (semantic_search.py:199-206 encodes every
        chunk text in one ``model.encode`` call) goes through in slices of at most ``max_tokens_per_call`` tokens
        (scratch is ~10 KB per token)."""
        id_lists = [list(x)[: self.max_seq_length] for x in id_lists]
        out = np.empty((len(id_lists), int(self.config["hidden"])), np.float32)
        lo = 0
        while lo < len(id_lists):
            hi, tok = lo, 0
            while hi < len(id_lists) and (hi == lo or tok + len(id_lists[hi]) <= max_tokens_per_call):
                tok += len(id_lists[hi]); hi += 1
            ids, _, cu = pack(id_lists[lo:hi])
            out[lo:hi] = self.index.encode(self.slot, ids, cu)
            lo = hi
        return out

    def encode_ids_dev(self, id_lists: Sequence[Sequence[int]], out_ptr: int) -> int:
        """Result stays on the device at ``out_ptr`` ([n, hidden] fp32); returns n."""
        id_lists = [list(x)[: self.max_seq_length] for x in id_lists]
        ids, _, cu = pack(id_lists)
        self.index.encode_dev(self.slot, ids, cu, out_ptr)
        return len(id_lists)

    def encode(self, texts, show_progress_bar: bool = False, **_kw) -> np.ndarray:
        if self.tokenizer is None:
            raise RuntimeError("GpuSentenceEncoder has no tokenizer: pass tokenizer=<texts -> token-id lists> "
                               "(e.g. the reference model's HuggingFace tokenizer) or call encode_ids")
        single = isinstance(texts, str)
        out = self.encode_ids(self.tokenizer([texts] if single else list(texts)))
        return out[0] if single else out


class GpuCrossEncoder:
    """``predict(pairs) -> float32[n]`` like sentence_transformers.CrossEncoder.predict for a 1-label model.
    Returns the classifier LOGITS (``activation="sigmoid"`` applies the logistic function, which some
    sentence-transformers versions do by default for num_labels = 1; the reference only sorts by the score,
    hybrid_search.py:304-309, and the order is the same either way).

    The batched rerank of ``HybridSearch.rrf_search_batch(..., rerank_method="cross_encoder")`` builds the pairs on
    the device from single-text token ids: ``tokenizer`` (texts -> token-id lists WITHOUT special tokens) and the
    ``cls_id`` / ``sep_id`` it wraps them in."""

    def __init__(self, index, state_dict, config: dict = TINYBERT_L2_CONFIG,
                 pair_tokenizer: Optional[Callable[[List[Sequence[str]]], tuple]] = None, *, slot: int = 1,
                 max_length: int = 512, activation: Optional[str] = None,
                 tokenizer: Optional[Callable[[List[str]], List[List[int]]]] = None, cls_id: int = 101,
                 sep_id: int = 102):
        self.index, self.slot, self.config = index, slot, dict(config)
        self.pair_tokenizer = pair_tokenizer
        self.tokenizer = tokenizer
        self.cls_id, self.sep_id = int(cls_id), int(sep_id)
        self.max_length = min(int(max_length), int(config["max_positions"]))
        self.activation = activation
        _load(index, slot, self.config, 1, state_dict)

    @classmethod
    def from_cross_encoder(cls, index, ce_model, *, slot: int = 1) -> "GpuCrossEncoder":
        """From a loaded ``sentence_transformers.CrossEncoder`` (hybrid_search.py:296)."""
        model, hf_tok = ce_model.model, ce_model.tokenizer
        ml = int(getattr(ce_model, "max_length", None) or 512)

        def tok(pairs):
            enc = hf_tok([p[0] for p in pairs], [p[1] for p in pairs], truncation=True, max_length=ml)
            return enc["input_ids"], enc["token_type_ids"]
        sd = {k: v for k, v in model.state_dict().items()}
        return cls(index, sd, config_from_hf(model.config), tok, slot=slot, max_length=ml,
                   tokenizer=hf_text_tokenizer(hf_tok), cls_id=hf_tok.cls_token_id, sep_id=hf_tok.sep_token_id)

    def tokenize(self, texts) -> List[List[int]]:
        """Single texts -> token ids without special tokens (the pieces the device assembles into pairs)."""
        if self.tokenizer is None:
            raise RuntimeError("GpuCrossEncoder has no single-text tokenizer: pass tokenizer=<texts -> token-id lists "
                               "without special tokens> (e.g. hf_text_tokenizer(hf_tokenizer))")
        return self.tokenizer(list(texts))

    def predict_ids(self, id_lists, type_lists) -> np.ndarray:
        ml = self.max_length                                   # (copy only what has to be cut)
        id_lists = [x if len(x) <= ml else x[:ml] for x in id_lists]
        type_lists = [x if len(x) <= ml else x[:ml] for x in type_lists]
        ids, tt, cu = pack(id_lists, type_lists)
        out = self.index.encode(self.slot, ids, cu, type_ids=tt)
        if self.activation == "sigmoid":
            out = (1.0 / (1.0 + np.exp(-out.astype(np.float64)))).astype(np.float32)
        return out

    def predict(self, pairs, **_kw) -> np.ndarray:
        if self.pair_tokenizer is None:
            raise RuntimeError("GpuCrossEncoder has no tokenizer: pass pair_tokenizer=<pairs -> (ids, type_ids)> "
                               "or call predict_ids")
        if len(pairs) == 0:
            return np.zeros(0, np.float32)
        ids, tts = self.pair_tokenizer(list(pairs))
        return self.predict_ids(ids, tts)
