"""CPU tests of the batched cross-encoder rerank's host side: the pair truncation rule the device applies
(rse_pair_truncate) against HuggingFace's fast BERT tokenizer, the equivalence of tokenising a document text alone
with the second segment of its pair, and the validation that runs before anything reaches a device."""
import random

import numpy as np
import pytest

transformers = pytest.importorskip("transformers")

WORDS = ["the", "movie", "about", "a", "dog", "and", "cat", "space", "war", "love", "hero", "un", "##s", "##ing",
         "##believ", "##able", "##ly", "time", "night", "city"]
PUNCT = ["-", ".", ",", "!", "'", ":"]


@pytest.fixture(scope="module")
def hf_tok():
    vocab = {"[PAD]": 0, "[UNK]": 1, "[CLS]": 2, "[SEP]": 3, "[MASK]": 4}
    for w in WORDS + PUNCT:
        vocab.setdefault(w, len(vocab))
    # a vocabulary dict: in this transformers version ``vocab_file=`` silently yields the 5 special tokens only
    tok = transformers.BertTokenizerFast(vocab=vocab)
    assert len(tok) == len(vocab)
    return tok


def _text(rng, n_words):
    out = []
    for _ in range(n_words):
        r = rng.random()
        if r < 0.15:
            out.append(rng.choice(PUNCT))
        elif r < 0.3:
            out.append(rng.choice(["dogs", "unbelievably", "loving", "cats", "wars", "heros"]))   # word pieces
        else:
            out.append(rng.choice([w for w in WORDS if not w.startswith("#")]))
    return " ".join(out)


def _kept(n1, n2, M):
    from rag_search_engine_b200._lib import pair_truncate
    return pair_truncate(n1, n2, M + 3)


def test_pair_truncate_matches_the_fast_tokenizer(hf_tok):
    """tok(q, d, truncation=True, max_length=ml) == [CLS] q[:a] [SEP] d[:b] [SEP], types 0 * (a + 2) + 1 * (b + 1),
    with (a, b) from rse_pair_truncate — over every case of the longest_first rule."""
    rng = random.Random(7)
    seen = set()
    for i in range(1500):
        ml = rng.randint(5, 70)
        q, d = _text(rng, rng.randint(1, 30)), _text(rng, rng.randint(1, 60))
        if i % 10 == 0:
            d = q                                                      # equal lengths
        qi = hf_tok(q, add_special_tokens=False)["input_ids"]
        di = hf_tok(d, add_special_tokens=False)["input_ids"]
        a, b = _kept(len(qi), len(di), ml - 3)
        enc = hf_tok(q, d, truncation=True, max_length=ml)
        want = [hf_tok.cls_token_id] + qi[:a] + [hf_tok.sep_token_id] + di[:b] + [hf_tok.sep_token_id]
        assert enc["input_ids"] == want, (q, d, ml, a, b)
        assert enc["token_type_ids"] == [0] * (a + 2) + [1] * (b + 1)
        M, n1, n2 = ml - 3, len(qi), len(di)
        case = ("none" if n1 + n2 <= M else "one" if min(n1, n2) in (a, b) and (a, b) != (n1, n2) else "both")
        seen.add(case)
        seen.add(("n1>M" if n1 > M else "n1<=M", M % 2, n1 == n2))
    assert {"none", "one", "both"} <= seen
    assert ("n1>M", 0, False) in seen and ("n1>M", 1, False) in seen
    assert any(s[2] for s in seen if isinstance(s, tuple))


def test_pair_truncate_rule_table():
    """A few cases spelled out (M = max_length - 3)."""
    assert _kept(3, 4, 10) == (3, 4)          # no cut
    assert _kept(3, 100, 50) == (3, 47)       # only the longer side is cut
    assert _kept(100, 3, 50) == (47, 3)
    assert _kept(30, 40, 50) == (25, 25)      # both cut, even M
    assert _kept(30, 40, 51) == (25, 26)      # both cut, odd M: the longer side keeps the extra token
    assert _kept(40, 30, 51) == (26, 25)
    assert _kept(60, 60, 51) == (25, 26)      # equal lengths: the query counts as the shorter side
    assert _kept(60, 2, 51) == (49, 2)        # n1 > M
    assert _kept(0, 80, 51) == (0, 51)


def test_pair_truncate_rejects_bad_arguments():
    from rag_search_engine_b200._lib import RseError, pair_truncate
    for args in ((-1, 3, 10), (3, -1, 10), (3, 3, 3)):
        with pytest.raises(RseError):
            pair_truncate(*args)


def test_document_text_alone_is_the_second_segment(hf_tok):
    """The store tokenises f"{title} - {description}" once per document; that equals the pair's second segment."""
    rng = random.Random(11)
    for _ in range(300):
        title, desc = _text(rng, rng.randint(1, 5)), _text(rng, rng.randint(0, 40))
        doc = f"{title} - {desc}"
        q = _text(rng, rng.randint(1, 8))
        enc = hf_tok(q, doc)
        tt = enc["token_type_ids"]
        second = enc["input_ids"][tt.index(1):-1]
        assert second == hf_tok(doc, add_special_tokens=False)["input_ids"]
    assert hf_tok("<missing> - ", add_special_tokens=False)["input_ids"]                # the id-without-row text


def test_hf_text_tokenizer_strips_special_tokens(hf_tok):
    from rag_search_engine_b200.encoder import hf_text_tokenizer
    tok = hf_text_tokenizer(hf_tok)
    assert tok(["the dog", "cats"]) == [hf_tok("the dog", add_special_tokens=False)["input_ids"],
                                        hf_tok("cats", add_special_tokens=False)["input_ids"]]


def test_null_handle_is_refused():
    from rag_search_engine_b200 import _lib
    L = _lib.load_library()
    assert L.rse_rerank_docs_load(None, None, 0, None, None) == -1
    assert L.rse_hybrid_rerank_run(None, 1, 60.0, 0, 10, 10, 1.5, 0.75, None, None, 101, 102, 512, 0) == -1
    assert L.rse_hybrid_rerank_fetch(None, 10, None, None, None, None, None, None, None) == -1
    assert L.rse_set_rerank_token_budget(None, 1024) == -1


# ----------------------------------------------------------------------------- Python-side checks (no device)
class _FakeIndex:
    def __init__(self):
        self.loaded = None

    def rerank_docs_load(self, ids, indptr, tokens):
        self.loaded = (np.asarray(ids), np.asarray(indptr), np.asarray(tokens))


class _FakeCE:
    def __init__(self, index, activation=None):
        self.index, self.activation, self.slot, self.cls_id, self.sep_id, self.max_length = index, activation, 1, 2, 3, 64


def _hybrid(index, ce=None):
    from types import SimpleNamespace
    from rag_search_engine_b200 import HybridSearch
    hs = HybridSearch.__new__(HybridSearch)
    hs._index, hs.cross_encoder = index, ce
    hs.keyword = SimpleNamespace(_arr=SimpleNamespace(doc_ids=np.array([5, 9], np.int64)))
    hs.semantic = SimpleNamespace(_arr=SimpleNamespace(movie_ids=np.array([1, 9], np.int64)))
    return hs


def test_load_rerank_documents_builds_a_sorted_csr():
    idx = _FakeIndex()
    hs = _hybrid(idx)
    assert hs.load_rerank_documents([9, 1, 5], [[7, 8], [], [4]]) == 3
    ids, indptr, tokens = idx.loaded
    assert ids.tolist() == [1, 5, 9] and indptr.tolist() == [0, 0, 1, 3] and tokens.tolist() == [4, 7, 8]
    assert ids.dtype == np.int64 and indptr.dtype == np.int64 and tokens.dtype == np.int32
    with pytest.raises(ValueError, match="differ in length"):
        hs.load_rerank_documents([1, 2], [[1]])


def test_rerank_encoder_requirements():
    idx = _FakeIndex()
    with pytest.raises(RuntimeError, match="GpuCrossEncoder"):
        _hybrid(idx)._rerank_encoder("cross_encoder")
    with pytest.raises(ValueError, match="another handle"):
        _hybrid(idx, _FakeCE(_FakeIndex()))._rerank_encoder("cross_encoder")
    with pytest.raises(ValueError, match="rerank_method"):
        _hybrid(idx, _FakeCE(idx))._rerank_encoder("batch")
    with pytest.raises(ValueError, match="activation"):
        _hybrid(idx, _FakeCE(idx, "softmax"))._rerank_encoder("cross_encoder")
    ce = _FakeCE(idx, "sigmoid")
    assert _hybrid(idx, ce)._rerank_encoder("cross_encoder") is ce
    with pytest.raises(ValueError, match="rerank_query_ids"):
        _hybrid(idx, ce)._rerank_staged(ce, 2, [[1]], 60, 10, 10, 1.5, 0.75, False)
