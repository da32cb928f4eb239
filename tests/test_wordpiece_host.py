"""CPU: the tables of rag_search_engine_b200.wordpiece against the HuggingFace tokenizers they are read from.  The
code-point map joined over a text is normalize_str of the text; the host restatement of the device algorithm
(helpers/wordpiece_ref.py) gives the HF ids; the builder refuses every pipeline the device does not implement."""
import unicodedata

import numpy as np
import pytest

pytest.importorskip("tokenizers")
pytest.importorskip("transformers")

from helpers import wordpiece_ref as ref  # noqa: E402
from helpers import wp_corpus as corpus  # noqa: E402


def _tables(config, vocab="trained"):
    from rag_search_engine_b200.wordpiece import build_tables
    return build_tables(corpus.tokenizer(config, vocab))


def _joined(t, text):
    out = []
    for ch in text:
        m = int(t.cp_map[ord(ch)])
        n = (m >> 21) & 3
        out += [chr(m & 0x1FFFFF)] if n == 1 else [chr(int(x)) for x in t.extra[m & 0x1FFFFF][:n]]
    return "".join(out)


@pytest.mark.parametrize("config", list(corpus.CONFIGS))
def test_code_point_map_reproduces_normalize_str(config):
    t = _tables(config)
    norm = corpus.tokenizer(config).backend_tokenizer.normalizer
    rng = np.random.default_rng(7)
    texts = corpus.texts(3000, seed=11)
    # strings drawn from every scalar value
    cps = rng.integers(0, 0x110000, 200000)
    cps = cps[(cps < 0xD800) | (cps >= 0xE000)]
    texts += ["".join(map(chr, cps[i:i + 40])) for i in range(0, len(cps), 40)]
    checked = 0
    for x in texts:
        if t.needs_host(x):
            continue
        assert _joined(t, x) == norm.normalize_str(x), repr(x)
        checked += 1
    assert checked > 0.9 * len(texts)


@pytest.mark.parametrize("config", list(corpus.CONFIGS))
@pytest.mark.parametrize("vocab", ["trained", "tiny"])
def test_host_restatement_equals_hf_ids(config, vocab):
    tok = corpus.tokenizer(config, vocab)
    t = _tables(config, vocab)
    texts = corpus.texts(2000, seed=3)
    for special, ml in ((False, None), (True, 8), (True, 128), (False, 8)):
        want = tok(texts, add_special_tokens=special, truncation=ml is not None, max_length=ml)["input_ids"]
        n = 0
        for x, w in zip(texts, want):
            got = ref.tokenize(t, x, special, ml)
            if got is None:
                assert t.needs_host(x)
                continue
            assert got == w, (repr(x), special, ml)
            n += 1
        assert n > 0.9 * len(texts)


def test_literal_special_tokens_and_unk_words():
    tok = corpus.tokenizer("uncased", "tiny")
    t = _tables("uncased", "tiny")
    for x in ["x[SEP]y", "x [sep] y", "[[SEP]]", "[mask][MASK]", "abcabcabc", "a" * 101, "the thé", "ΣΣ σς"]:
        assert ref.tokenize(t, x, True, None) == tok(x)["input_ids"], x


def test_reorder_rule():
    """With accent stripping, marks of two code points that survive it can be reordered by NFD: such texts go to the
    host; one code point's own marks cannot, and without NFD nothing is flagged."""
    t = _tables("uncased")
    assert t.reorder_chars and all(unicodedata.combining(c) or any(unicodedata.combining(x) for x in
                                                                   unicodedata.normalize("NFD", c))
                                   for c in t.reorder_chars)
    a, b = "\U0001d16d", "\U0001d165"                       # canonical classes 226 and 216: NFD swaps them
    norm = corpus.tokenizer("uncased").backend_tokenizer.normalizer
    assert _joined(t, "x" + a + b) != norm.normalize_str("x" + a + b)
    assert t.needs_host("x" + a + b) and not t.needs_host("x" + a) and not t.needs_host("plain")
    assert not _tables("cased").reorder_chars


def _fast(tokenizer_obj):
    import transformers
    return transformers.PreTrainedTokenizerFast(tokenizer_object=tokenizer_obj)


def test_builder_refuses_other_pipelines():
    from tokenizers import AddedToken, Tokenizer, normalizers, pre_tokenizers
    from tokenizers.models import BPE, WordPiece
    from rag_search_engine_b200.wordpiece import UnsupportedTokenizer, build_tables
    vocab = {"[UNK]": 0, "[CLS]": 1, "[SEP]": 2, "a": 3, "##b": 4}

    def bert(**over):
        t = Tokenizer(WordPiece(vocab, unk_token="[UNK]"))
        t.normalizer = normalizers.BertNormalizer()
        t.pre_tokenizer = pre_tokenizers.BertPreTokenizer()
        from tokenizers.processors import BertProcessing
        t.post_processor = BertProcessing(("[SEP]", 2), ("[CLS]", 1))
        t.add_special_tokens(["[UNK]", "[CLS]", "[SEP]"])
        for k, v in over.items():
            setattr(t, k, v)
        return t
    build_tables(bert())                                    # the BERT pipeline itself is accepted
    build_tables(_fast(bert()))
    bpe = Tokenizer(BPE({"a": 0, "b": 1}, [], unk_token="a"))
    for bad in (bpe, bert(normalizer=normalizers.NFKC()), bert(pre_tokenizer=pre_tokenizers.Whitespace()),
                bert(post_processor=None), object()):
        with pytest.raises(UnsupportedTokenizer):
            build_tables(bad)
    for flags in (dict(lstrip=True), dict(rstrip=True), dict(single_word=True), dict(normalized=True)):
        t = bert()
        t.add_special_tokens([AddedToken("[MASK]", **flags)])
        with pytest.raises(UnsupportedTokenizer):
            build_tables(t)
    t = bert()
    t.add_tokens(["plain"])                                 # a non-special added token
    with pytest.raises(UnsupportedTokenizer):
        build_tables(t)


def test_host_route_ignores_padding_and_truncation_left_on_the_backend(tmp_path):
    """A tokenizer.json may keep padding / truncation enabled on the backend; the texts the device refuses are
    tokenized with both off, as hf_tok(texts, ...) does on every call."""
    import transformers
    from rag_search_engine_b200.wordpiece import build_tables, host_ids, plain_backend
    base = corpus.tokenizer("uncased").backend_tokenizer
    from tokenizers import Tokenizer
    t = Tokenizer.from_str(base.to_str())
    t.enable_truncation(8)
    t.enable_padding(length=16, pad_id=0, pad_token="[PAD]")
    t.save(str(tmp_path / "tokenizer.json"))
    tok = transformers.BertTokenizerFast(tokenizer_file=str(tmp_path / "tokenizer.json"))
    assert tok.backend_tokenizer.truncation is not None and tok.backend_tokenizer.padding is not None
    tables = build_tables(tok)
    texts = ["x\U0001d16d\U0001d165 " + " ".join(["the movie of a war"] * 4), "\U0001d165\U0001d16d"]
    assert all(tables.needs_host(x) for x in texts)
    for special, ml in ((True, None), (True, 128), (False, None), (True, 8)):
        want = tok(texts, add_special_tokens=special, truncation=ml is not None, max_length=ml)["input_ids"]
        assert host_ids(plain_backend(tok), texts, special, ml, tables.cls_id, tables.sep_id) == want
        assert host_ids(plain_backend(t), texts, special, ml, tables.cls_id, tables.sep_id) == want
    assert len(want[0]) == 8 and len(tok(texts[0])["input_ids"]) > 16
