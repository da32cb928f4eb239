"""The tables of a CLIP byte-level BPE tokenizer for csrc/bpe.cuh, read from the HuggingFace object itself.

``build_bpe_tables(tok)`` takes a ``transformers`` CLIP tokenizer or a ``tokenizers.Tokenizer`` and accepts exactly
the pipeline of the CLIP tokenizers (clip-ViT-B-32 and its family):

* normalizer ``Sequence[NFC, Replace(Regex \\s+ -> " "), Lowercase]``;
* pre-tokenizer ``Sequence[Split(CLIP_PATTERN, Removed, invert), ByteLevel(add_prefix_space=False)]``;
* a ``BPE`` model with ``end_of_word_suffix="</w>"``, no continuing-subword prefix, an ``unk_token``, no dropout,
  no byte fallback, ``fuse_unk`` and ``ignore_merges`` off;
* a ``<|startoftext|> $A <|endoftext|>`` post-processor (``RobertaProcessing`` or the same template);
* the special tokens as the only added tokens, matched literally in the raw text (``normalized`` / ``lstrip`` /
  ``rstrip`` / ``single_word`` false).

Anything else raises ``UnsupportedTokenizer`` (a WordPiece or GPT-2 tokenizer, the slow ftfy tokenizer); the caller
then keeps its host tokenizer.

Every table is probed through the tokenizer's own components, so the device applies the Unicode version of the
``tokenizers`` build it was built from:

* ``cp_map`` uint32[0x110000]: the 0-3 code points ``normalizer.normalize_str(chr(c))`` yields (bits 0-20: the code
  point, or a row of ``extra`` for two or three; bits 21-22 the count) and bit 23, ``ROUTE_BIT``, on the code points
  whose text must be tokenized on the host (see ``route_chars``).
* ``cp_class`` uint8[0x110000]: how the Split pattern sees a (normalized) code point: other, whitespace, ``\\p{L}`` or
  ``\\p{N}``, from ``pre_tokenize_str`` probes.
* ``byte_ids`` int32[512]: the initial symbol of byte b inside a piece (``[b]``) and as its last byte (``[256 + b]``,
  with ``</w>``), ``unk`` where the vocab lacks the symbol, as ``BPE::merge_word`` does.
* ``merges`` int32[slots, 4]: ``(left id, right id) -> (rank, merged id)`` in an open-addressing table (linear
  probing, ``hash_pair``); ``left == -1`` marks an empty slot, and at least half the slots are empty.

NFC is the one step that depends on context.  Joining the per-code-point outputs equals normalizing the whole text
when no code point of the text is in ``route_chars``: the code points whose full canonical decomposition starts with
a non-starter (canonical combining class != 0) or with a starter that can be the second member of a canonical
composition (NFC_QC=Maybe starters: Hangul V/T jamo, the Indic and Sinhala length marks).  Then every code point's
decomposition starts with a starter that composes with nothing before it, so canonical reordering never moves a
mark across two code points and composition never joins them: NFC(text) is the concatenation of NFC(c).  Replace and
Lowercase map code point by code point (``char::to_lowercase`` has no context; a run of whitespace becoming one space
or several changes no piece, as pieces never hold whitespace).  A text with a route code point goes to the host
tokenizer; the device refuses it.
"""
from __future__ import annotations

import functools
import json
import re
import unicodedata
from dataclasses import dataclass

import numpy as np

from .wordpiece import UnsupportedTokenizer, _backend, host_ids, plain_backend  # noqa: F401  (re-exported)

N_CODE_POINTS = 0x110000
MAX_WORD_BYTES = 256          # csrc/bpe.cuh kBpeMaxWord: the longest piece (in bytes) the device merges
MAX_ADDED = 32                # kWpMaxAdded (the added-token matcher is shared with WordPiece)
ROUTE_BIT = 1 << 23
CLASS_OTHER, CLASS_SPACE, CLASS_LETTER, CLASS_NUMBER = 0, 1, 2, 3
CLIP_PATTERN = r"""<\|startoftext\|>|<\|endoftext\|>|'s|'t|'re|'ve|'m|'ll|'d|[\p{L}]+|[\p{N}]|[^\s\p{L}\p{N}]+"""
SUFFIX = "</w>"
# the Split pattern's two literal alternatives (they match the lowercased text, e.g. "<|ENDOFTEXT|>"); ByteLevel's
# own GPT-2 pattern then cuts such a piece into three: "<|", the word, "|>"
LITERALS = ("<|startoftext|>", "<|endoftext|>")
HASH_MUL = 0x9E3779B97F4A7C15


def hash_pair(left, right, mask: int):
    """The slot a (left, right) pair starts probing at: the high 32 bits of (left << 32 | right) * HASH_MUL mod 2^64,
    masked (csrc/bpe.cuh bpe_merge)."""
    key = (np.asarray(left, np.uint64) << np.uint64(32)) | np.asarray(right, np.uint64)
    with np.errstate(over="ignore"):
        return ((key * np.uint64(HASH_MUL)) >> np.uint64(32)).astype(np.int64) & mask


@functools.lru_cache(maxsize=1)
def bytes_to_unicode() -> dict:
    """GPT-2's byte -> character map, the alphabet of ``pre_tokenizers.ByteLevel``."""
    bs = list(range(ord("!"), ord("~") + 1)) + list(range(ord("¡"), ord("¬") + 1)) + list(range(ord("®"), ord("ÿ") + 1))
    cs = bs[:]
    n = 0
    for b in range(256):
        if b not in bs:
            bs.append(b)
            cs.append(256 + n)
            n += 1
    return dict(zip(bs, map(chr, cs)))


@dataclass
class BpeTables:
    cp_map: np.ndarray        # uint32[0x110000]
    extra: np.ndarray         # uint32[n_extra, 3]
    cp_class: np.ndarray      # uint8[0x110000]
    byte_ids: np.ndarray      # int32[512]
    merges: np.ndarray        # int32[slots, 4]
    added: list               # [(content, id)] matched literally in the raw text, longest first at a position
    unk_id: int
    bos_id: int
    eos_id: int
    route_chars: str          # the code points whose bit 23 is set
    max_char_bytes: int       # the most UTF-8 bytes the normalizer makes of one code point
    space_chars: str          # the code points the normalizer turns into whitespace only

    def __post_init__(self):
        self._route = frozenset(self.route_chars)
        spaces = "".join(re.escape(c) for c in self.space_chars)
        # a run of this many code points without whitespace can hold a piece longer than the device's word buffer
        run = MAX_WORD_BYTES // max(1, self.max_char_bytes) + 1
        self._long = re.compile(f"[^{spaces}]{{{run},}}")
        self._long_ascii = re.compile(f"[^{spaces}]{{{MAX_WORD_BYTES + 1},}}")

    def needs_host(self, text: str) -> bool:
        """True when ``text`` holds a route code point (NFC could join or reorder across code points there): the
        device refuses such a text."""
        if text.isascii() or self._route.isdisjoint(text):       # (a set walk: a regex class is ~15x slower)
            return False
        return True

    def may_overflow(self, text: str) -> bool:
        """True when ``text`` could hold a piece longer than the device's word buffer (a run of non-whitespace code
        points that long): a superset of the texts the device refuses for that reason."""
        if text.isascii():                                          # ASCII normalizes byte for byte
            return len(text) > MAX_WORD_BYTES and self._long_ascii.search(text) is not None
        return self._long.search(text) is not None


def _post_processor_ids(pp, vocab, bos: str, eos: str):
    if pp is None:
        raise UnsupportedTokenizer("no post-processor: the device adds <|startoftext|> / <|endoftext|>")
    if pp.get("type") == "RobertaProcessing":
        cls_, sep = pp["cls"], pp["sep"]
        return int(cls_[1]), int(sep[1])
    if pp.get("type") == "TemplateProcessing":
        single = pp.get("single") or []
        kinds = [next(iter(p)) for p in single]
        if kinds != ["SpecialToken", "Sequence", "SpecialToken"] or single[1]["Sequence"]["id"] != "A":
            raise UnsupportedTokenizer("the post-processor's single template is not bos $A eos")
        ids = []
        for p in (single[0], single[2]):
            ids_ = pp["special_tokens"][p["SpecialToken"]["id"]]["ids"]
            if len(ids_) != 1:
                raise UnsupportedTokenizer("a special token of the template is not one id")
            ids.append(int(ids_[0]))
        return ids[0], ids[1]
    raise UnsupportedTokenizer(f"post-processor {pp.get('type')!r} is not CLIP's")


def _check_pipeline(spec):
    norm = spec.get("normalizer") or {}
    want_norm = [{"type": "NFC"}, {"type": "Replace", "pattern": {"Regex": r"\s+"}, "content": " "},
                 {"type": "Lowercase"}]
    if norm.get("type") != "Sequence" or norm.get("normalizers") != want_norm:
        raise UnsupportedTokenizer(f"normalizer {json.dumps(norm)[:200]} is not CLIP's NFC / Replace / Lowercase")
    pre = spec.get("pre_tokenizer") or {}
    parts = pre.get("pretokenizers") if pre.get("type") == "Sequence" else None
    if not parts or len(parts) != 2:
        raise UnsupportedTokenizer("the pre-tokenizer is not CLIP's Split + ByteLevel sequence")
    split, bl = parts
    if (split.get("type") != "Split" or split.get("pattern") != {"Regex": CLIP_PATTERN}
            or split.get("behavior") != "Removed" or split.get("invert") is not True):
        raise UnsupportedTokenizer("the Split pre-tokenizer is not CLIP's pattern (Removed, invert)")
    if bl.get("type") != "ByteLevel" or bl.get("add_prefix_space") is not False or bl.get("use_regex") is False:
        raise UnsupportedTokenizer("the ByteLevel pre-tokenizer is not add_prefix_space=False with its pattern")
    model = spec.get("model") or {}
    if model.get("type") != "BPE":
        raise UnsupportedTokenizer(f"model {model.get('type')!r} is not BPE")
    flags = {k: model.get(k) for k in ("dropout", "end_of_word_suffix", "continuing_subword_prefix", "fuse_unk",
                                       "byte_fallback", "ignore_merges")}
    if (flags["dropout"] is not None or flags["end_of_word_suffix"] != SUFFIX
            or flags["continuing_subword_prefix"] not in (None, "") or flags["fuse_unk"]
            or flags["byte_fallback"] or flags["ignore_merges"]):
        raise UnsupportedTokenizer(f"BPE flags {flags} are not CLIP's")
    if model.get("unk_token") not in model.get("vocab", {}):
        raise UnsupportedTokenizer("the BPE model has no unk token in its vocab")
    return model


@functools.lru_cache(maxsize=1)
def _route_set() -> frozenset:
    """The code points whose canonical decomposition starts with a non-starter or with a starter that can be the
    second member of a canonical composition.  Derived from Python's ``unicodedata`` and united with a probe of the
    ``tokenizers`` build's own NFD / NFC, so a code point either Unicode version treats so is routed."""
    from tokenizers import normalizers
    nfd = normalizers.NFD().normalize_str
    nfc = normalizers.NFC().normalize_str

    def canon(c):
        d = unicodedata.decomposition(c)
        if not d or d.startswith("<"):
            return c
        return "".join(canon(chr(int(x, 16))) for x in d.split())
    seconds = {chr(c) for c in range(0x1161, 0x1176)} | {chr(c) for c in range(0x11A8, 0x11C3)}   # Hangul V, T
    decomp = {}
    for c in range(N_CODE_POINTS):
        if 0xD800 <= c < 0xE000:
            continue
        ch = chr(c)
        d = unicodedata.decomposition(ch)
        if d and not d.startswith("<"):
            parts = [chr(int(x, 16)) for x in d.split()]
            if len(parts) == 2:
                seconds.add(parts[1])
            decomp[ch] = canon(ch)
        # the build's view: the decomposition of a composite that NFC rebuilds names its later members
        t = nfd(ch)
        if t != ch:
            decomp.setdefault(ch, t)
            if len(t) >= 2 and nfc(t) == ch:
                seconds.update(t[1:])
    out = set()
    for c in range(N_CODE_POINTS):
        if 0xD800 <= c < 0xE000:
            continue
        ch = chr(c)
        first = decomp.get(ch, ch)[0]
        if unicodedata.combining(ch) or unicodedata.combining(first) or first in seconds or ch in seconds:
            out.add(ch)
    # marks the build knows and Python's tables do not: NFD moves U+0334 (class 1) in front of them
    for c in range(N_CODE_POINTS):
        if 0xD800 <= c < 0xE000:
            continue
        ch = chr(c)
        if ch not in out and nfd(ch + "̴") == "̴" + ch:
            out.add(ch)
    return frozenset(out)


@functools.lru_cache(maxsize=1)
def _normalizer_tables():
    from tokenizers import Regex, normalizers
    norm = normalizers.Sequence([normalizers.NFC(), normalizers.Replace(Regex(r"\s+"), " "), normalizers.Lowercase()])
    ns = norm.normalize_str
    route = _route_set()
    cp_map = np.zeros(N_CODE_POINTS, np.uint32)
    extra, routed, spaces = [], [], []
    max_bytes = 1
    for c in range(N_CODE_POINTS):
        if 0xD800 <= c < 0xE000:
            continue                                   # surrogates are not scalar values: malformed UTF-8 on the device
        ch = chr(c)
        s = ns(ch)
        if ch in route or len(s) > 3:
            cp_map[c] = ROUTE_BIT
            routed.append(ch)
            continue
        if s == " " and ch != " ":
            spaces.append(ch)
        max_bytes = max(max_bytes, len(s.encode("utf-8")))
        if len(s) == 1:
            cp_map[c] = ord(s) | (1 << 21)
        elif len(s) > 1:
            cp_map[c] = len(extra) | (len(s) << 21)
            extra.append([ord(x) for x in s] + [0] * (3 - len(s)))
    extra = np.asarray(extra if extra else [[0, 0, 0]], np.uint32).reshape(-1, 3)
    return cp_map, extra, "".join(routed), max_bytes, " " + "".join(spaces)


@functools.lru_cache(maxsize=1)
def _class_table():
    """The Split pattern's view of every code point, each probed between two 'a' (a letter joins them) and between
    two '!' (an 'other' joins them); whitespace is in no piece, and a number is a piece of its own in both."""
    from tokenizers import Regex, pre_tokenizers
    pre = pre_tokenizers.Split(Regex(CLIP_PATTERN), behavior="removed", invert=True)
    cls = np.zeros(N_CODE_POINTS, np.uint8)
    step = 1 << 16
    for lo in range(0, N_CODE_POINTS, step):
        cps = [c for c in range(lo, min(lo + step, N_CODE_POINTS)) if not 0xD800 <= c < 0xE000]
        if not cps:
            continue
        pos = 1 + 2 * np.arange(len(cps))
        joined = {}
        for sep in ("a", "!"):
            s = sep + sep.join(map(chr, cps)) + sep
            covered = np.zeros(len(s), bool)
            merged = np.zeros(len(s), bool)
            for _, (b, e) in pre.pre_tokenize_str(s):
                covered[b:e] = True
                if e - b > 1:
                    merged[b:e] = True
            joined[sep] = merged[pos]
        c = np.where(~covered[pos], CLASS_SPACE,
                     np.where(joined["a"], CLASS_LETTER, np.where(joined["!"], CLASS_OTHER, CLASS_NUMBER)))
        cls[np.asarray(cps)] = c
    return cls


def _merge_table(vocab: dict, merges) -> np.ndarray:
    left, right, rank, new = [], [], [], []
    for r, m in enumerate(merges):
        a, b = (m.split(" ") if isinstance(m, str) else m)
        ia, ib, im = vocab.get(a), vocab.get(b), vocab.get(a + b)
        if ia is None or ib is None or im is None:
            raise UnsupportedTokenizer(f"merge {a!r} {b!r} names a symbol outside the vocab")
        left.append(ia); right.append(ib); rank.append(r); new.append(im)
    slots = 1 << max(4, int(2 * max(1, len(left)) - 1).bit_length())
    mask = slots - 1
    table = np.full((slots, 4), -1, np.int32)
    h = hash_pair(left, right, mask) if left else []
    for i in range(len(left)):
        s = int(h[i])
        while table[s, 0] >= 0:
            if table[s, 0] == left[i] and table[s, 1] == right[i]:
                break                                  # a repeated merge: the last one stands, as in HF's map
            s = (s + 1) & mask
        table[s] = (left[i], right[i], rank[i], new[i])
    return table


def build_bpe_tables(tok) -> BpeTables:
    """The device description of ``tok``; ``UnsupportedTokenizer`` for anything but the CLIP BPE pipeline."""
    backend = _backend(tok)
    spec = json.loads(backend.to_str())
    model = _check_pipeline(spec)
    vocab = model["vocab"]
    unk_id = int(vocab[model["unk_token"]])
    added = []
    for a in spec.get("added_tokens") or []:
        flags = {k: a.get(k) for k in ("single_word", "lstrip", "rstrip", "normalized")}
        if not a.get("special") or any(flags.values()) or a.get("content") not in LITERALS:
            raise UnsupportedTokenizer(f"added token {a.get('content')!r} is not a literal CLIP special token "
                                       f"({flags}, special={a.get('special')})")
        added.append((a["content"], int(a["id"])))
    bos_id, eos_id = _post_processor_ids(spec.get("post_processor"), vocab, *LITERALS)
    b2u = bytes_to_unicode()
    byte_ids = np.empty(512, np.int32)
    for b in range(256):
        byte_ids[b] = vocab.get(b2u[b], unk_id)
        byte_ids[256 + b] = vocab.get(b2u[b] + SUFFIX, unk_id)
    cp_map, extra, routed, max_bytes, spaces = _normalizer_tables()
    return BpeTables(cp_map=cp_map, extra=extra, cp_class=_class_table(), byte_ids=byte_ids,
                     merges=_merge_table(vocab, model.get("merges") or []), added=added, unk_id=unk_id,
                     bos_id=bos_id, eos_id=eos_id, route_chars=routed, max_char_bytes=max_bytes, space_chars=spaces)
