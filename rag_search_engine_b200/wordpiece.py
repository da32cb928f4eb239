"""The tables of a BERT WordPiece tokenizer for csrc/wordpiece.cuh, read from the HuggingFace object itself.

``build_tables(tok)`` takes a ``transformers`` fast tokenizer or a ``tokenizers.Tokenizer`` and accepts exactly the
pipeline of the BERT tokenizers (all-MiniLM-L6-v2, ms-marco-TinyBERT-L2-v2): a ``WordPiece`` model, a
``BertNormalizer`` (any flags), the ``BertPreTokenizer``, a ``[CLS] $A [SEP]`` post-processor and special tokens as
the only added tokens, matched literally (``single_word`` / ``lstrip`` / ``rstrip`` / ``normalized`` all false).
Anything else raises ``UnsupportedTokenizer``; the caller then keeps its host tokenizer.

Every table is probed through the tokenizer's own components, so the device applies the Unicode version of the
``tokenizers`` build it was built from:

* ``cp_map`` uint32[0x110000]: what ``normalizer.normalize_str(chr(c))`` yields for code point c, as 0-3 code points.
  Bits 0-20 hold the code point (one output) or a row of ``extra`` (two or three outputs), bits 21-22 the count, and
  bit 23 is set when the output keeps a combining mark (canonical class != 0, per ``_non_starters``) and the
  normalizer runs NFD.  Joining
  the per-code-point outputs is ``normalize_str`` of the whole text, except for NFD's canonical reordering: only
  marks that survive the accent stripping can be reordered, and only when two code points of one text carry them.
  The device reports such texts instead of tokenizing them (``needs_host``).
* ``cp_class`` uint8[0x110000]: 0 other, 1 whitespace, 2 punctuation, as the pre-tokenizer splits on them.
* two tries over code points for the greedy longest match: node 0 is the root of the word-initial pieces, node 1 the
  root of the continuation pieces (the vocab entries that start with ``continuing_subword_prefix``, prefix removed).
  ``node_first`` [n_nodes + 1] delimits each node's edges, sorted by ``edge_cp``; ``node_id`` is the vocab id of the
  piece that ends at a node (-1: none).
"""
from __future__ import annotations

import functools
import json
import unicodedata
from dataclasses import dataclass

import numpy as np

N_CODE_POINTS = 0x110000
MAX_WORD_CHARS = 256          # csrc/wordpiece.cuh kWpMaxWordChars: the longest max_input_chars_per_word on the device
MAX_ADDED = 32                # kWpMaxAdded
REORDER_BIT = 1 << 23
CLASS_OTHER, CLASS_SPACE, CLASS_PUNCT = 0, 1, 2


class UnsupportedTokenizer(ValueError):
    """The tokenizer is not the BERT WordPiece pipeline the device implements."""


@dataclass
class WordPieceTables:
    cp_map: np.ndarray        # uint32[0x110000]
    extra: np.ndarray         # uint32[n_extra, 3]
    cp_class: np.ndarray      # uint8[0x110000]
    node_first: np.ndarray    # int32[n_nodes + 1]
    node_id: np.ndarray       # int32[n_nodes]
    edge_cp: np.ndarray       # int32[n_edges]
    edge_child: np.ndarray    # int32[n_edges]
    added: list               # [(content, id)] matched literally in the raw text, longest first at a position
    unk_id: int
    cls_id: int
    sep_id: int
    max_input_chars_per_word: int
    reorder_chars: str        # the code points whose bit 23 is set

    def needs_host(self, text: str) -> bool:
        """True when two code points of ``text`` carry bit 23 (NFD could reorder their marks): the device refuses
        such a text."""
        if text.isascii() or self._marks.isdisjoint(text):          # (a set walk: a regex class is ~15x slower)
            return False
        return sum(c in self._marks for c in text) >= 2

    def __post_init__(self):
        self._marks = frozenset(self.reorder_chars)


def _backend(tok):
    if hasattr(tok, "backend_tokenizer"):
        return tok.backend_tokenizer
    if hasattr(tok, "to_str") and hasattr(tok, "normalizer"):
        return tok
    raise UnsupportedTokenizer(f"not a HuggingFace fast tokenizer: {type(tok).__name__}")


def _post_processor_ids(pp, vocab):
    if pp is None:
        raise UnsupportedTokenizer("no post-processor: the device adds [CLS] / [SEP] like BertProcessing")
    if pp.get("type") == "BertProcessing":
        return int(pp["cls"][1]), int(pp["sep"][1])
    if pp.get("type") == "TemplateProcessing":
        single = pp.get("single") or []
        kinds = [next(iter(p)) for p in single]
        if kinds != ["SpecialToken", "Sequence", "SpecialToken"] or single[1]["Sequence"]["id"] != "A" \
                or any(next(iter(p.values()))["type_id"] != 0 for p in single):
            raise UnsupportedTokenizer("the post-processor's single template is not [CLS] $A [SEP]")
        ids = []
        for p in (single[0], single[2]):
            ids_ = pp["special_tokens"][p["SpecialToken"]["id"]]["ids"]
            if len(ids_) != 1:
                raise UnsupportedTokenizer("a special token of the template is not one id")
            ids.append(int(ids_[0]))
        return ids[0], ids[1]
    raise UnsupportedTokenizer(f"post-processor {pp.get('type')!r} is not BERT's")


@functools.lru_cache(maxsize=1)
def _non_starters() -> frozenset:
    """Code points the canonical reordering treats as marks: Python's ``unicodedata`` (canonical class != 0) united
    with a probe of the ``tokenizers`` build's own NFD, which moves U+0334 (class 1) in front of every mark of class
    >= 2 — a mark one of the two Unicode versions knows and the other does not still counts."""
    from tokenizers import normalizers
    nfd = normalizers.NFD().normalize_str
    out = set()
    for c in range(N_CODE_POINTS):
        if 0xD800 <= c < 0xE000:
            continue
        ch = chr(c)
        if unicodedata.combining(ch) or nfd(ch + "\u0334") == "\u0334" + ch:
            out.add(ch)
    return frozenset(out)


@functools.lru_cache(maxsize=8)
def _normalizer_tables(normalizer_json: str):
    from tokenizers import normalizers
    cfg = json.loads(normalizer_json)
    norm = normalizers.BertNormalizer(clean_text=cfg["clean_text"], handle_chinese_chars=cfg["handle_chinese_chars"],
                                      strip_accents=cfg["strip_accents"], lowercase=cfg["lowercase"])
    nfd = cfg["strip_accents"] if cfg["strip_accents"] is not None else cfg["lowercase"]
    cp_map = np.zeros(N_CODE_POINTS, np.uint32)
    extra, reorder = [], []
    ns = norm.normalize_str
    marks = _non_starters() if nfd else frozenset()
    for c in range(N_CODE_POINTS):
        if 0xD800 <= c < 0xE000:
            continue                                   # surrogates are not scalar values: malformed UTF-8 on the device
        ch = chr(c)
        s = ns(ch)
        if s == ch:
            cp_map[c] = c | (1 << 21)
            if ch in marks:
                cp_map[c] |= REORDER_BIT
                reorder.append(ch)
            continue
        if len(s) > 3:
            raise UnsupportedTokenizer(f"the normalizer maps U+{c:04X} to {len(s)} code points (the device takes 3)")
        if len(s) == 1:
            cp_map[c] = ord(s) | (1 << 21)
        elif len(s) > 1:
            cp_map[c] = (len(extra) | (len(s) << 21))
            extra.append([ord(x) for x in s] + [0] * (3 - len(s)))
        if any(x in marks for x in s):
            cp_map[c] |= REORDER_BIT
            reorder.append(ch)
    extra = np.asarray(extra if extra else [[0, 0, 0]], np.uint32).reshape(-1, 3)
    return cp_map, extra, "".join(reorder)


@functools.lru_cache(maxsize=1)
def _class_table():
    """BertPreTokenizer's view of every code point: each probed between two 'a' so that a punctuation mark comes
    out as a piece of its own, whitespace as no piece and anything else merged with its neighbours."""
    from tokenizers import pre_tokenizers
    pre = pre_tokenizers.BertPreTokenizer()
    cls = np.zeros(N_CODE_POINTS, np.uint8)
    step = 1 << 16
    for lo in range(0, N_CODE_POINTS, step):
        cps = [c for c in range(lo, min(lo + step, N_CODE_POINTS)) if not 0xD800 <= c < 0xE000]
        if not cps:
            continue
        s = "a" + "a".join(map(chr, cps)) + "a"
        covered = np.zeros(len(s), bool)
        single = np.zeros(len(s), bool)
        for _, (b, e) in pre.pre_tokenize_str(s):
            covered[b:e] = True
            if e - b == 1:
                single[b] = True
        pos = 1 + 2 * np.arange(len(cps))
        c = np.where(~covered[pos], CLASS_SPACE, np.where(single[pos], CLASS_PUNCT, CLASS_OTHER))
        cls[np.asarray(cps)] = c
    return cls


def _tries(vocab: dict, prefix: str):
    children = [{}, {}]
    node_id = [-1, -1]

    def insert(root, s, tid):
        n = root
        for ch in s:
            nxt = children[n].get(ord(ch))
            if nxt is None:
                nxt = len(children)
                children[n][ord(ch)] = nxt
                children.append({})
                node_id.append(-1)
            n = nxt
        node_id[n] = tid
    for tok, tid in vocab.items():
        if tok:
            insert(0, tok, int(tid))
        if prefix and tok.startswith(prefix) and len(tok) > len(prefix):
            insert(1, tok[len(prefix):], int(tid))
    first = np.zeros(len(children) + 1, np.int32)
    first[1:] = np.cumsum([len(c) for c in children])
    edge_cp = np.empty(int(first[-1]), np.int32)
    edge_child = np.empty(int(first[-1]), np.int32)
    for n, ch in enumerate(children):
        items = sorted(ch.items())
        edge_cp[first[n]:first[n + 1]] = [k for k, _ in items]
        edge_child[first[n]:first[n + 1]] = [v for _, v in items]
    return first, np.asarray(node_id, np.int32), edge_cp, edge_child


def plain_backend(tok):
    """A private copy of ``tok``'s ``tokenizers.Tokenizer`` with padding and truncation off: a tokenizer.json may
    leave them enabled on the backend, and ``hf_tok(texts, ...)`` resets them on every call."""
    from tokenizers import Tokenizer
    t = Tokenizer.from_str(_backend(tok).to_str())
    t.no_padding()
    t.no_truncation()
    return t


def host_ids(backend, texts, add_special: bool, max_length, cls_id: int, sep_id: int):
    """The ids ``hf_tok(texts, add_special_tokens=add_special, truncation=max_length is not None,
    max_length=max_length)["input_ids"]`` gives, from a ``plain_backend``: the pieces, cut, then [CLS] / [SEP]."""
    out = []
    for e in backend.encode_batch(list(texts), add_special_tokens=False):
        ids = e.ids
        if max_length is not None:
            ids = ids[:max_length - 2 * add_special]
        out.append([cls_id] + ids + [sep_id] if add_special else list(ids))
    return out


def build_tables(tok) -> WordPieceTables:
    """The device description of ``tok``; ``UnsupportedTokenizer`` for anything but the BERT WordPiece pipeline."""
    backend = _backend(tok)
    spec = json.loads(backend.to_str())
    model = spec.get("model") or {}
    if model.get("type") != "WordPiece":
        raise UnsupportedTokenizer(f"model {model.get('type')!r} is not WordPiece")
    norm = spec.get("normalizer") or {}
    if norm.get("type") != "BertNormalizer":
        raise UnsupportedTokenizer(f"normalizer {norm.get('type')!r} is not BertNormalizer")
    pre = spec.get("pre_tokenizer") or {}
    if pre.get("type") != "BertPreTokenizer":
        raise UnsupportedTokenizer(f"pre-tokenizer {pre.get('type')!r} is not BertPreTokenizer")
    vocab = model["vocab"]
    unk = model.get("unk_token")
    if unk not in vocab:
        raise UnsupportedTokenizer("the unk token is not in the vocab")
    max_chars = int(model.get("max_input_chars_per_word", 100))
    if not 1 <= max_chars <= MAX_WORD_CHARS:
        raise UnsupportedTokenizer(f"max_input_chars_per_word {max_chars} outside [1, {MAX_WORD_CHARS}]")
    cls_id, sep_id = _post_processor_ids(spec.get("post_processor"), vocab)
    added = []
    for a in spec.get("added_tokens") or []:
        flags = {k: a.get(k) for k in ("single_word", "lstrip", "rstrip", "normalized")}
        if not a.get("special") or any(flags.values()):
            raise UnsupportedTokenizer(f"added token {a.get('content')!r} is not a literal special token ({flags}, "
                                       f"special={a.get('special')})")
        if not a.get("content"):
            raise UnsupportedTokenizer("an added token is empty")
        added.append((a["content"], int(a["id"])))
    if len(added) > MAX_ADDED:
        raise UnsupportedTokenizer(f"{len(added)} added tokens (the device takes {MAX_ADDED})")
    nj = json.dumps({k: norm.get(k) for k in ("clean_text", "handle_chinese_chars", "strip_accents", "lowercase")},
                    sort_keys=True)
    cp_map, extra, reorder = _normalizer_tables(nj)
    node_first, node_id, edge_cp, edge_child = _tries(vocab, model.get("continuing_subword_prefix") or "")
    return WordPieceTables(cp_map=cp_map, extra=extra, cp_class=_class_table(), node_first=node_first,
                           node_id=node_id, edge_cp=edge_cp, edge_child=edge_child, added=added,
                           unk_id=int(vocab[unk]), cls_id=cls_id, sep_id=sep_id, max_input_chars_per_word=max_chars,
                           reorder_chars=reorder)
