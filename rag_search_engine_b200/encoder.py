"""GPU text encoders behind the reference's own encoder interfaces (SURVEY §8 f2 / f3).

* ``GpuSentenceEncoder`` stands in for ``SentenceTransformer("all-MiniLM-L6-v2")`` where the reference calls
  ``self.model.encode(texts)`` / ``get_sentence_embedding_dimension()`` / ``max_seq_length``
  (rag_search_engine/utils/semantic_search.py:45-46, :200, :221, :372): pass it as ``SemanticSearch(encoder=...)``.
* ``GpuCrossEncoder`` stands in for ``CrossEncoder("cross-encoder/ms-marco-TinyBERT-L2-v2").predict(pairs)``
  (rag_search_engine/utils/hybrid_search.py:296-297): pass it as ``HybridSearch(cross_encoder=...)``.

Both run csrc/encoder.cuh through the C-ABI (``rse_encoder_*``, ``rse_encode``): HuggingFace BERT weights handed
over under their state_dict names, fp32 throughout.  The tokenizer is pluggable: ``DeviceWordPiece`` runs a BERT
WordPiece tokenizer on the device (csrc/wordpiece.cuh, ids identical to the HF fast tokenizer), and any callable
returning token-id lists runs on the host.  ``from_sentence_transformer`` / ``from_cross_encoder`` take the loaded
reference model's tokenizer and put it on the device when its pipeline is BERT WordPiece
(``wordpiece.build_tables`` decides from the tokenizer object).  No weights are bundled and nothing is
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


def _utf8(texts):
    """Texts -> (UTF-8 bytes back to back, int64 byte offsets [n + 1])."""
    raw = [t.encode("utf-8") for t in texts]
    offs = np.zeros(len(raw) + 1, np.int64)
    np.cumsum([len(r) for r in raw], out=offs[1:])
    return b"".join(raw), offs


from .wordpiece import host_ids, plain_backend  # noqa: E402


class DeviceTokenizer:
    """What the device tokenizers (``DeviceWordPiece``, ``clip.DeviceBPE``) share: ``maybe`` and the
    ``hf_tok(texts, ...)["input_ids"]``-shaped call over the subclass's ``tokenize``."""

    @classmethod
    def maybe(cls, index, hf_tok, **kw):
        """An instance, or None when ``hf_tok`` is not the pipeline the device implements."""
        from .wordpiece import UnsupportedTokenizer
        try:
            return cls(index, hf_tok, **kw)
        except UnsupportedTokenizer:
            return None

    def __call__(self, texts, add_special: Optional[bool] = None, max_length: Optional[int] = -1) -> List[List[int]]:
        ids, cu = self.tokenize(texts, add_special, max_length)
        ids = ids.tolist()
        return [ids[a:b] for a, b in zip(cu[:-1].tolist(), cu[1:].tolist())]


class DeviceWordPiece(DeviceTokenizer):
    """A BERT WordPiece tokenizer on the device (csrc/wordpiece.cuh) in a tokenizer slot of ``index``.

    Called on texts it returns what ``hf_tok(texts, add_special_tokens=..., truncation=..., max_length=...)
    ["input_ids"]`` returns, so it drops into every ``tokenizer=`` argument; ``add_special_tokens`` / ``max_length``
    fix which call it stands for (``max_length=None``: no cut).  The encoders use its device paths instead, where
    the ids never become Python lists.  A text NFD could reorder (two code points whose combining marks survive the
    accent stripping, see include/rse.h) goes to ``hf_tok``'s own Rust tokenizer on the host and is counted in
    ``host_texts``.  ``UnsupportedTokenizer`` when ``hf_tok`` is not BERT WordPiece; ``maybe`` returns None then."""

    def __init__(self, index, hf_tok, *, slot: int = 0, add_special_tokens: bool = True,
                 max_length: Optional[int] = None):
        from .wordpiece import build_tables
        self.tables = build_tables(hf_tok)
        self.backend = plain_backend(hf_tok)
        self.index, self.slot = index, int(slot)
        self.add_special_tokens = bool(add_special_tokens)
        self.max_length = None if max_length is None else int(max_length)
        self.cls_id, self.sep_id = self.tables.cls_id, self.tables.sep_id
        self.host_texts = 0
        index.tokenizer_load(self.slot, self.tables)

    def host_ids(self, texts, add_special: bool, max_length: Optional[int]) -> List[List[int]]:
        """The host tokenizer's ids under the same rule (the route of the texts the device refuses)."""
        self.host_texts += len(texts)
        return host_ids(self.backend, texts, add_special, max_length, self.cls_id, self.sep_id)

    def host_routed(self, texts) -> List[int]:
        return [i for i, t in enumerate(texts) if self.tables.needs_host(t)]

    def tokenize(self, texts, add_special: Optional[bool] = None, max_length: Optional[int] = -1):
        """-> (ids int32[total], cu_seqlens int32[n + 1]) on the host; defaults are this object's call rule."""
        sp = self.add_special_tokens if add_special is None else bool(add_special)
        ml = self.max_length if max_length == -1 else max_length
        texts = list(texts)
        routed = self.host_routed(texts)
        if routed:
            got = {i: ids for i, ids in zip(routed, self.host_ids([texts[i] for i in routed], sp, ml))}
            keep = [i for i in range(len(texts)) if i not in got]
            dev = self.__call__([texts[i] for i in keep], sp, ml) if keep else []
            got.update(zip(keep, dev))
            return pack([got[i] for i in range(len(texts))])[::2]
        if not texts:
            return np.zeros(0, np.int32), np.zeros(1, np.int32)
        data, offs = _utf8(texts)
        return self.index.tokenize(self.slot, data, offs, sp, ml or 0)


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
        tok = DeviceWordPiece.maybe(index, hf_tok, slot=slot, max_length=msl)
        if tok is None:
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

    def encode_texts_dev(self, texts: Sequence[str], out_ptr: int) -> int:
        """Texts -> [n, hidden] fp32 at ``out_ptr`` on the device; with a ``DeviceWordPiece`` the ids never leave
        the device, otherwise the host tokenizer's ids go through ``encode_ids_dev``.  Returns n."""
        texts = list(texts)
        tok = self.tokenizer
        if not isinstance(tok, DeviceWordPiece) or tok.host_routed(texts):
            return self.encode_ids_dev(self._host_tokenize(texts), out_ptr)
        data, offs = _utf8(texts)
        self.index.encode_texts_dev(tok.slot, self.slot, data, offs, self.max_seq_length, out_ptr)
        return len(texts)

    def _host_tokenize(self, texts):
        tok = self.tokenizer
        if isinstance(tok, DeviceWordPiece):
            return tok(texts, True, self.max_seq_length)
        return tok(texts)

    def encode(self, texts, show_progress_bar: bool = False, max_tokens_per_call: int = 1 << 16, **_kw) -> np.ndarray:
        if self.tokenizer is None:
            raise RuntimeError("GpuSentenceEncoder has no tokenizer: pass tokenizer=<texts -> token-id lists> "
                               "(e.g. the reference model's HuggingFace tokenizer) or call encode_ids")
        single = isinstance(texts, str)
        texts = [texts] if single else list(texts)
        tok = self.tokenizer
        if not texts or not isinstance(tok, DeviceWordPiece) or tok.host_routed(texts):
            out = self.encode_ids(self._host_tokenize(texts), max_tokens_per_call)
            return out[0] if single else out
        data, offs = _utf8(texts)
        msl = self.max_seq_length
        if int(np.minimum(np.diff(offs) + 2, msl).sum()) <= max_tokens_per_call:
            # a text has at most one id per UTF-8 byte plus [CLS] / [SEP]: the batch fits one call, and its ids
            # stay on the device
            out = self.index.encode_texts(tok.slot, self.slot, data, offs, msl)
        else:
            # a bulk embedding: ids tokenized on the device come back as arrays and are cut into slices of at most
            # max_tokens_per_call by their real lengths (the byte bound is ~6x the token count of English text)
            ids, cu = self.index.tokenize(tok.slot, data, offs, True, msl)
            out = np.empty((len(texts), int(self.config["hidden"])), np.float32)
            lo = 0
            while lo < len(texts):
                hi = max(lo + 1, int(np.searchsorted(cu, int(cu[lo]) + max_tokens_per_call, side="right")) - 1)
                out[lo:hi] = self.index.encode(self.slot, ids[cu[lo]:cu[hi]], cu[lo:hi + 1] - cu[lo])
                lo = hi
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
        single = DeviceWordPiece.maybe(index, hf_tok, slot=slot, add_special_tokens=False)
        return cls(index, sd, config_from_hf(model.config), tok, slot=slot, max_length=ml,
                   tokenizer=single if single is not None else hf_text_tokenizer(hf_tok), cls_id=hf_tok.cls_token_id,
                   sep_id=hf_tok.sep_token_id)

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
