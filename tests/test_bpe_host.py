"""CPU: the tables of rag_search_engine_b200.bpe and a host restatement of csrc/bpe.cuh (tests/helpers/bpe_ref.py)
against the HuggingFace fast tokenizer, on a BpeTrainer-trained CLIP vocab and a tiny hand-made one; which texts go
to the host; which tokenizers are refused; the facts the device's piece cutting and per-code-point NFC rest on."""
import json
import random

import pytest

pytest.importorskip("transformers")
pytest.importorskip("tokenizers")

from helpers import bpe_corpus as corpus  # noqa: E402
from helpers import bpe_ref  # noqa: E402

N_TEXTS = 4000
CASES = ((False, None), (True, None), (True, 77), (True, 8), (False, 77))


@pytest.fixture(scope="module", params=["trained", "tiny"])
def tok_tables(request):
    from rag_search_engine_b200.bpe import build_bpe_tables
    tok = corpus.tokenizer(request.param)
    return tok, build_bpe_tables(tok)


def test_restatement_equals_hf(tok_tables):
    tok, t = tok_tables
    texts = corpus.texts(N_TEXTS, seed=5) + ["eeee", "eeeee", "theeee the", "hello hell", "cat's", "'S 'LL 'Re"]
    for special, ml in CASES:
        want = tok(texts, add_special_tokens=special, truncation=ml is not None, max_length=ml)["input_ids"]
        refused = 0
        for x, w in zip(texts, want):
            got = bpe_ref.tokenize(t, x, special, ml)
            if got is None:
                refused += 1
                assert t.needs_host(x) or t.may_overflow(x), repr(x)
                continue
            assert got == w, (special, ml, repr(x))
        assert refused < len(texts) // 4


def test_unk_symbols_are_exercised():
    from rag_search_engine_b200.bpe import build_bpe_tables
    tok = corpus.tokenizer("tiny")
    t = build_bpe_tables(tok)
    assert (t.byte_ids == t.unk_id).sum() > 200            # most "x</w>" are missing
    ids = bpe_ref.tokenize(t, "xyz the", False, None)
    assert ids == tok("xyz the", add_special_tokens=False)["input_ids"]
    assert t.unk_id in ids


def test_literals_and_cut():
    from rag_search_engine_b200.bpe import build_bpe_tables
    tok = corpus.tokenizer("trained")
    t = build_bpe_tables(tok)
    sot, eot = t.bos_id, t.eos_id
    # a literal special token is its id; its uppercase form lowercases into the pattern's literal, then three pieces
    assert bpe_ref.tokenize(t, "<|endoftext|>", False, None) == [eot]
    up = bpe_ref.tokenize(t, "<|ENDOFTEXT|>", False, None)
    assert eot not in up and up == tok("<|ENDOFTEXT|>", add_special_tokens=False)["input_ids"]
    assert bpe_ref.tokenize(t, "a<|startoftext|>b", True, None)[2] == sot
    long = " ".join(["movie"] * 200)
    assert len(bpe_ref.tokenize(t, long, True, 77)) == 77
    # a word longer than the device's buffer is refused before the cut and ignored after it
    word = "ab" * 200
    assert bpe_ref.tokenize(t, word, True, 77) is None
    assert bpe_ref.tokenize(t, "movie " * 80 + word, True, 77) == tok("movie " * 80 + word, truncation=True,
                                                                      max_length=77)["input_ids"]


def test_host_route_texts():
    from rag_search_engine_b200.bpe import build_bpe_tables
    t = build_bpe_tables(corpus.tokenizer("tiny"))
    for x in ("é", "́", "가", "ཱི", "xା", "ab\U0001d165"):
        assert t.needs_host(x), repr(x)
    for x in ("é", "가", "İstanbul", "　 \xa0\t\n", "plain", "😀 中文", ""):
        assert not t.needs_host(x), repr(x)
    texts = corpus.texts(2000, seed=8)
    routed = [x for x in texts if t.needs_host(x)]
    assert 0 < len(routed) < len(texts) // 4
    assert t.may_overflow("a" * 300) and not t.may_overflow("a " * 300)
    assert not t.may_overflow("x" * 256) and t.may_overflow("x" * 257)


def test_per_code_point_nfc_is_exact_outside_the_route_set():
    """NFC(starter + c) == NFC(starter) + NFC(c) for every code point c outside the route set, after starters that
    compose with marks, with Hangul V/T and with Indic length marks; and the route set covers every code point the
    tokenizers build's NFC joins with such a starter."""
    from tokenizers import normalizers
    from rag_search_engine_b200.bpe import _route_set
    nfc = normalizers.NFC().normalize_str
    route = _route_set()
    starters = ["a", "e", "A", "ᄀ", "가", "େ", "ෙ", "ె", "ೆ", "ে", "ᬅ", "െ"]
    for c in range(0x110000):
        if 0xD800 <= c < 0xE000:
            continue
        ch = chr(c)
        for s in starters:
            if nfc(s + ch) != nfc(s) + nfc(ch):
                assert ch in route, (hex(c), s)


def test_bytelevel_keeps_split_pieces_whole():
    """ByteLevel's own GPT-2 pattern cuts no piece of the CLIP split further, but the pattern's two literals, which it
    cuts into "<|", the word and "|>"."""
    from tokenizers import Regex, pre_tokenizers
    from rag_search_engine_b200.bpe import CLIP_PATTERN
    split = pre_tokenizers.Split(Regex(CLIP_PATTERN), behavior="removed", invert=True)
    bl = pre_tokenizers.ByteLevel(add_prefix_space=False, use_regex=True)
    b2u = __import__("rag_search_engine_b200.bpe", fromlist=["bytes_to_unicode"]).bytes_to_unicode()
    seen = 0
    tok = corpus.tokenizer("tiny")
    for text in corpus.texts(1500, seed=3) + ["<|endoftext|>", "<|startoftext|>!", "!<|endoftext|>"]:
        for piece, _ in split.pre_tokenize_str(tok.backend_tokenizer.normalizer.normalize_str(text)):
            parts = [p for p, _ in bl.pre_tokenize_str(piece)]
            mapped = "".join(b2u[b] for b in piece.encode())
            if piece in ("<|startoftext|>", "<|endoftext|>"):
                assert parts == ["<|", piece[2:-2], "|>"]
                seen += 1
            else:
                assert parts == [mapped], (piece, parts)
    assert seen >= 2


def _spec(tok):
    return json.loads(tok.backend_tokenizer.to_str())


def _from_spec(spec):
    from tokenizers import Tokenizer
    return Tokenizer.from_str(json.dumps(spec))


@pytest.mark.parametrize("change", [
    "bert", "gpt2", "suffix", "fuse_unk", "dropout", "ignore_merges", "byte_fallback", "no_lowercase",
    "pattern", "prefix_space", "no_regex", "added_normalized", "added_lstrip", "extra_added", "no_post", "no_unk"])
def test_unsupported_tokenizers(change):
    from rag_search_engine_b200.bpe import UnsupportedTokenizer, build_bpe_tables
    if change == "bert":
        from helpers import wp_corpus
        with pytest.raises(UnsupportedTokenizer):
            build_bpe_tables(wp_corpus.tokenizer("uncased", "tiny"))
        return
    if change == "gpt2":
        from tokenizers import Tokenizer, decoders, pre_tokenizers
        from tokenizers.models import BPE
        t = Tokenizer(BPE({"a": 0, "b": 1, "ab": 2}, [("a", "b")]))
        t.pre_tokenizer = pre_tokenizers.ByteLevel(add_prefix_space=False)
        t.decoder = decoders.ByteLevel()
        with pytest.raises(UnsupportedTokenizer):
            build_bpe_tables(t)
        return
    spec = _spec(corpus.tokenizer("tiny"))
    m = spec["model"]
    pre = spec["pre_tokenizer"]["pretokenizers"]
    if change == "suffix":
        m["end_of_word_suffix"] = None
    elif change in ("fuse_unk", "ignore_merges", "byte_fallback"):
        m[change] = True
    elif change == "dropout":
        m["dropout"] = 0.1
    elif change == "no_lowercase":
        spec["normalizer"]["normalizers"] = spec["normalizer"]["normalizers"][:2]
    elif change == "pattern":
        pre[0]["pattern"] = {"Regex": r"[\p{L}]+|[\p{N}]+|[^\s\p{L}\p{N}]+"}
    elif change == "prefix_space":
        pre[1]["add_prefix_space"] = True
    elif change == "no_regex":
        pre[1]["use_regex"] = False
    elif change == "added_normalized":
        spec["added_tokens"][0]["normalized"] = True
    elif change == "added_lstrip":
        spec["added_tokens"][1]["lstrip"] = True
    elif change == "extra_added":
        spec["added_tokens"].append(dict(spec["added_tokens"][1], id=len(m["vocab"]), content="<|pad|>"))
        m["vocab"]["<|pad|>"] = len(m["vocab"])
    elif change == "no_post":
        spec["post_processor"] = None
    elif change == "no_unk":
        m["unk_token"] = None
    with pytest.raises(UnsupportedTokenizer):
        build_bpe_tables(_from_spec(spec))


def test_tokenizers_object_and_merge_table():
    """A plain tokenizers.Tokenizer is accepted like the transformers object; every merge is found at its rank."""
    from rag_search_engine_b200.bpe import build_bpe_tables
    tok = corpus.tokenizer("trained")
    a = build_bpe_tables(tok)
    b = build_bpe_tables(_from_spec(_spec(tok)))
    assert (a.merges == b.merges).all() and a.bos_id == b.bos_id and a.eos_id == b.eos_id
    spec = _spec(tok)
    vocab = spec["model"]["vocab"]
    rng = random.Random(1)
    merges = spec["model"]["merges"]
    for r in rng.sample(range(len(merges)), 300):
        x, y = merges[r]
        assert bpe_ref.merge_lookup(a, vocab[x], vocab[y]) == (r, vocab[x + y])
    assert (a.merges[:, 0] < 0).sum() * 2 >= a.merges.shape[0]
