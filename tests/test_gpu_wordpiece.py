"""GPU: BERT WordPiece on the device (csrc/wordpiece.cuh) against the HuggingFace fast tokenizer, bit for bit, and
the text entry points built on it (GpuSentenceEncoder.encode, the rerank store from texts, rrf_search_texts from
query strings) against the same calls fed with HF ids; the ABI's error paths."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
pytest.importorskip("transformers")

from helpers import wp_corpus as corpus  # noqa: E402

N_TEXTS = 20000


def _utf8(texts):
    from rag_search_engine_b200.encoder import _utf8
    return _utf8(texts)


def _device_ids(idx, slot, texts, special, ml):
    ids, cu = idx.tokenize(slot, *_utf8(texts), special, ml or 0)
    ids = ids.tolist()
    return [ids[a:b] for a, b in zip(cu[:-1].tolist(), cu[1:].tolist())]


@pytest.mark.parametrize("config", list(corpus.CONFIGS))
@pytest.mark.parametrize("vocab", ["trained", "tiny"])
def test_device_ids_equal_hf(gpu_index, config, vocab):
    from rag_search_engine_b200.wordpiece import build_tables
    tok = corpus.tokenizer(config, vocab)
    t = build_tables(tok)
    gpu_index.tokenizer_load(0, t)
    texts = [x for x in corpus.texts(N_TEXTS + 2000, seed=17) if not t.needs_host(x)][:N_TEXTS]
    assert len(texts) == N_TEXTS
    for special, ml in ((False, None), (True, None), (True, 8), (True, 128), (False, 256), (True, 256)):
        want = tok(texts, add_special_tokens=special, truncation=ml is not None, max_length=ml)["input_ids"]
        got = _device_ids(gpu_index, 0, texts, special, ml)
        bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
        assert not bad, (special, ml, len(bad), repr(texts[bad[0]]), got[bad[0]], want[bad[0]])


def test_batch_sizes_and_the_callable(gpu_index):
    from rag_search_engine_b200.encoder import DeviceWordPiece
    tok = corpus.tokenizer("uncased")
    dw = DeviceWordPiece(gpu_index, tok, slot=1, max_length=128)
    big = corpus.texts(100000, seed=23)
    for n in (1, 256, 100000):
        texts = big[:n]
        assert dw(texts) == tok(texts, truncation=True, max_length=128)["input_ids"], n
    # texts NFD could reorder are routed to the host tokenizer and counted; the result is the same
    mixed = ["x\U0001d16d\U0001d165 y", "plain text", "\U0001d165 and \U0001d16d"]
    before = dw.host_texts
    assert dw(mixed) == tok(mixed, truncation=True, max_length=128)["input_ids"]
    assert dw.host_texts - before == 2
    assert dw([]) == []
    assert dw(["", " 　 "], False, None) == [[], []]


def test_sentence_encoder_encode_texts(gpu_index):
    from rag_search_engine_b200.encoder import DeviceWordPiece, GpuSentenceEncoder, random_state_dict
    tok = corpus.tokenizer("uncased")
    cfg = dict(vocab_size=4000, hidden=384, layers=2, heads=12, intermediate=1536, max_positions=128, type_vocab=2,
               ln_eps=1e-12)
    dw = DeviceWordPiece(gpu_index, tok, slot=0, max_length=128)
    enc = GpuSentenceEncoder(gpu_index, random_state_dict(cfg, seed=5), cfg, dw, max_seq_length=128)
    texts = corpus.texts(3000, seed=29)
    texts = [x for x in texts if not dw.tables.needs_host(x)]
    want = enc.encode_ids(tok(texts, truncation=True, max_length=128)["input_ids"])
    got = enc.encode(texts)
    assert got.view(np.uint32).tobytes() == want.view(np.uint32).tobytes()
    got_small = enc.encode(texts, max_tokens_per_call=2048)        # tokenized on the device, encoded in slices
    assert got_small.view(np.uint32).tobytes() == want.view(np.uint32).tobytes()
    buf = torch.empty((len(texts), 384), dtype=torch.float32, device="cuda:0")
    assert enc.encode_texts_dev(texts, buf.data_ptr()) == len(texts)
    torch.cuda.synchronize()
    assert buf.cpu().numpy().view(np.uint32).tobytes() == want.view(np.uint32).tobytes()
    one = enc.encode("a single query")
    assert one.view(np.uint32).tobytes() == enc.encode_ids([tok("a single query")["input_ids"]])[0].view(np.uint32).tobytes()


@pytest.fixture(scope="module")
def text_setup(gpu_index):
    from rag_search_engine_b200 import HybridSearch, _lib, synth
    from rag_search_engine_b200.encoder import (TINYBERT_L2_CONFIG, DeviceWordPiece, GpuCrossEncoder,
                                                GpuSentenceEncoder, random_state_dict)
    tok = corpus.tokenizer("uncased")
    se = synth.synth_embeddings(3000, seed=41, device="cpu")
    bm = synth.synth_bm25(3000, 2000, seed=41, mean_len=30, sd_len=10)
    idx = _lib.Index(0)
    idx.load_embeddings(se.emb.numpy(), movie_idx=se.movie_of_chunk.numpy())
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    cfg = dict(vocab_size=4000, hidden=se.emb.shape[1], layers=2, heads=12, intermediate=4 * se.emb.shape[1],
               max_positions=256, type_vocab=2, ln_eps=1e-12)
    enc = GpuSentenceEncoder(idx, random_state_dict(cfg, seed=6), cfg, DeviceWordPiece(idx, tok, slot=0, max_length=256),
                             max_seq_length=256)
    ce = GpuCrossEncoder(idx, random_state_dict(TINYBERT_L2_CONFIG, seed=7, head=1), TINYBERT_L2_CONFIG, slot=1,
                         tokenizer=DeviceWordPiece(idx, tok, slot=1, add_special_tokens=False),
                         cls_id=tok.cls_token_id, sep_id=tok.sep_token_id)
    T = len(bm.df)
    names = [f"t{i}" for i in range(T)]
    hs = HybridSearch.from_loaded(idx, dict(zip(names, range(T))), se.movie_ids, se.movie_ids,
                                  registry_key="wordpiece-test", cross_encoder=ce)
    doc_ids = np.asarray(se.movie_ids, np.int64)
    doc_texts = [" ".join(corpus.texts(6, seed=1000 + i)) for i in range(len(doc_ids))]
    doc_texts = [x for x in doc_texts]
    yield dict(idx=idx, hs=hs, enc=enc, ce=ce, tok=tok, se=se, bm=bm, names=names, doc_ids=doc_ids,
               doc_texts=doc_texts, synth=synth)
    hs.close()
    idx.close()


def _queries(s, nq, seed):
    synth, names = s["synth"], s["names"]
    tok_indptr, terms = synth.synth_token_queries(s["bm"], nq, seed=seed)
    toks = [[names[t] if t >= 0 else "<oov>" for t in terms[tok_indptr[i]:tok_indptr[i + 1]]] for i in range(nq)]
    texts = [x or "q" for x in corpus.texts(nq, seed=seed)]
    texts = [x if not s["ce"].tokenizer.tables.needs_host(x) else "q" for x in texts]
    return toks, texts


def _same(a, b):
    return all(x.dtype == y.dtype and x.shape == y.shape and (x.view(np.uint8) == y.view(np.uint8)).all()
               for x, y in zip(a, b))


def test_rerank_store_from_texts_and_text_queries(text_setup):
    s = text_setup
    hs, idx, ce, enc, tok = s["hs"], s["idx"], s["ce"], s["enc"], s["tok"]
    docs = [x for x in s["doc_texts"]]
    routed = [i for i, x in enumerate(docs) if ce.tokenizer.tables.needs_host(x)]
    for i in routed:
        docs[i] = "replaced"
    hf_docs = tok(docs, add_special_tokens=False)["input_ids"]
    toks, texts = _queries(s, 200, seed=51)
    enc_ids = tok(texts, truncation=True, max_length=256)["input_ids"]
    q_ids = tok(texts, add_special_tokens=False)["input_ids"]
    kw = dict(k=60, limit=10, rerank_method="cross_encoder")
    for ml in (512, 48):                                   # whole documents, and cut pairs
        ce.max_length = ml
        hs.load_rerank_documents(s["doc_ids"], hf_docs)
        want = hs.rrf_search_texts(toks, enc_ids, enc, rerank_query_ids=q_ids, as_arrays=True, **kw)
        idx.rerank_docs_load_texts(ce.tokenizer.slot, s["doc_ids"], *_utf8(docs))
        got = hs.rrf_search_texts(toks, texts, enc, as_arrays=True, **kw)          # ids made on the device
        assert _same(want, got), ml
        assert int(got[6].sum()) > 0
        got_b = hs.rrf_search_batch(toks, enc.encode(texts), rerank_query_ids=texts, as_arrays=True, **kw)
        assert _same(want, got_b), ml
    ce.max_length = 512
    plain_want = hs.rrf_search_texts(toks, enc_ids, enc, k=60, limit=10, as_arrays=True)
    plain_got = hs.rrf_search_texts(toks, texts, enc, k=60, limit=10, as_arrays=True)
    assert _same(plain_want, plain_got)


def test_status_codes(fresh_index, text_setup):
    from rag_search_engine_b200._lib import RseError
    from rag_search_engine_b200.wordpiece import build_tables
    idx = fresh_index
    with pytest.raises(RseError) as e:                      # nothing loaded in the slot
        idx.tokenize(0, b"abc", [0, 3], True)
    assert e.value.code == -3 and "no tokenizer" in str(e.value)
    idx.tokenizer_load(0, build_tables(corpus.tokenizer("uncased")))
    for data, offs, code, what in ((b"ab\xffcd", [0, 2, 5], -1, "text 1 is not well-formed UTF-8"),
                                   (b"\xed\xa0\x80", [0, 3], -1, "text 0 is not well-formed UTF-8"),  # a surrogate
                                   (b"\xc3", [0, 1], -1, "not well-formed"),                           # cut short
                                   (b"abc", [0, 2, 1], -1, "offsets must not decrease"),
                                   (b"abc", [1, 3], -1, "offsets must start at 0"),
                                   ("x\U0001d16d\U0001d165".encode(), [0, 9], -4, "canonical reordering")):
        with pytest.raises(RseError) as e:
            idx.tokenize(0, data, offs, True)
        assert e.value.code == code and what in str(e.value), str(e.value)
    with pytest.raises(RseError) as e:
        idx.tokenize(2, b"abc", [0, 3], True)
    assert e.value.code == -1
    with pytest.raises(RseError) as e:
        idx.tokenize(0, b"abc", [0, 3], True, 1)
    assert e.value.code == -4
    ids, cu = idx.tokenize(0, b"abc", [0, 3], True)        # the handle still works after the errors
    assert cu.tolist() == [0, len(ids)] and ids[0] == 2
    s = text_setup
    with pytest.raises(RseError) as e:                      # encoder max_positions 256
        s["idx"].encode_texts(0, 0, b"abc", [0, 3], 257)
    assert e.value.code == -4
    with pytest.raises(RseError) as e:
        s["idx"].rerank_docs_load_texts(1, [5, 3], b"ab", [0, 1, 2])
    assert e.value.code == -1 and "ascending" in str(e.value)


def test_store_from_texts_through_load_rerank_documents(tmp_path, monkeypatch):
    """HybridSearch.load_rerank_documents() over a SQLite database takes the device branch when the cross-encoder
    has a DeviceWordPiece; its ids are the HF ids byte for byte (the store is written by the same count / write
    kernels as rse_tokenize without special tokens or cut), and the rerank over it equals the rerank over a store
    loaded from HF ids."""
    from rag_search_engine_b200 import HybridSearch, runtime, store
    from rag_search_engine_b200.encoder import (TINYBERT_L2_CONFIG, DeviceWordPiece, GpuCrossEncoder,
                                                GpuSentenceEncoder, random_state_dict)
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    from rag_search_engine_b200.wordpiece import build_tables
    tok = corpus.tokenizer("uncased")
    tables = build_tables(tok)
    texts = [x for x in corpus.texts(500, seed=61) if not tables.needs_host(x)]
    docs = [{"id": 5 + 2 * i, "title": texts[i][:30] or "t", "description": texts[i]} for i in range(200)]
    db = tmp_path / "wp.db"
    idx = runtime.acquire(db, 0)
    try:
        cfg = dict(vocab_size=4000, hidden=384, layers=2, heads=12, intermediate=1536, max_positions=256, type_vocab=2,
                   ln_eps=1e-12)
        enc = GpuSentenceEncoder(idx, random_state_dict(cfg, seed=8), cfg,
                                 DeviceWordPiece(idx, tok, slot=0, max_length=256), max_seq_length=256)
        store.write_reference_db(db, docs, whitespace_tokenizer, embed=enc.encode)
        dw = DeviceWordPiece(idx, tok, slot=1, add_special_tokens=False)
        ce = GpuCrossEncoder(idx, random_state_dict(TINYBERT_L2_CONFIG, seed=9, head=1), TINYBERT_L2_CONFIG, slot=1,
                             tokenizer=dw, cls_id=tok.cls_token_id, sep_id=tok.sep_token_id)
        hs = HybridSearch(docs_path=None, db_path=db, tokenizer=whitespace_tokenizer, encoder=enc, cross_encoder=ce)
        try:
            doc_texts = [f"{d['title']} - {d['description']}" for d in docs]
            assert not any(dw.tables.needs_host(x) for x in doc_texts)
            calls = []
            real = idx.rerank_docs_load_texts
            monkeypatch.setattr(idx, "rerank_docs_load_texts", lambda *a: (calls.append(a), real(*a))[1])
            assert hs.load_rerank_documents() == len(docs)
            assert len(calls) == 1                                  # the device branch
            hf = tok(doc_texts, add_special_tokens=False)["input_ids"]
            ids, cu = idx.tokenize(1, *_utf8(doc_texts), False, 0)
            want = np.fromiter((t for x in hf for t in x), np.int32)
            assert ids.tobytes() == want.tobytes()
            assert cu.tolist() == np.concatenate([[0], np.cumsum([len(x) for x in hf])]).tolist()
            qs = [x or "q" for x in texts[200:240]]
            toks = whitespace_tokenizer(qs)
            vecs = enc.encode(qs)
            got = hs.rrf_search_batch(toks, vecs, k=60, limit=10, rerank_method="cross_encoder",
                                      rerank_query_ids=qs, as_arrays=True)
            hs.load_rerank_documents([d["id"] for d in docs], hf)
            want_r = hs.rrf_search_batch(toks, vecs, k=60, limit=10, rerank_method="cross_encoder",
                                         rerank_query_ids=tok(qs, add_special_tokens=False)["input_ids"],
                                         as_arrays=True)
            assert _same(want_r, got) and int(got[6].sum()) > 0
        finally:
            hs.close()
    finally:
        runtime.release(db, 0)
