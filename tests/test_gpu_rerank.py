"""GPU: the batched cross-encoder rerank (rse_hybrid_rerank_run, csrc/rerank.cuh) against the single-query mirror
``HybridSearch.rrf_search(q, rerank_method="cross_encoder")`` (hybrid_search.py:279-312) and against the host
composition of today's device calls; ties, slicing, the text entry point and the ABI's error paths.

The cross-encoder is a seeded random TinyBERT-L2 (the checkpoint cannot be downloaded here); the arithmetic does not
depend on the weights.  Scores are compared bitwise: every encoder stage works per sequence (GEMM rows, attention per
(sequence, head), LayerNorm), so a pair's logit does not depend on which batch or slice carried it."""
import random

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
transformers = pytest.importorskip("transformers")

WORDS = [f"w{i}" for i in range(80)]
ACTIVATIONS = (None, "sigmoid")


@pytest.fixture(scope="module")
def hf_tok():
    vocab = {"[PAD]": 0, "[UNK]": 1, "[CLS]": 2, "[SEP]": 3, "[MASK]": 4}
    for w in WORDS + ["-", ".", ",", "<", ">", "missing", "##s", "##x"]:
        vocab.setdefault(w, len(vocab))
    return transformers.BertTokenizerFast(vocab=vocab)


def _cross_encoder(idx, hf_tok, seed=2, bias=None):
    from rag_search_engine_b200.encoder import TINYBERT_L2_CONFIG as C, GpuCrossEncoder, hf_text_tokenizer, random_state_dict
    sd = random_state_dict(C, seed=seed, head=1)
    if bias is not None:
        sd["classifier.bias"] = np.full(1, bias, np.float32)
    ce = None

    def pair_tok(pairs):                                 # the HF pair encoding, at the encoder's current max_length
        enc = hf_tok([p[0] for p in pairs], [p[1] for p in pairs], truncation=True, max_length=ce.max_length)
        return enc["input_ids"], enc["token_type_ids"]
    ce = GpuCrossEncoder(idx, sd, C, pair_tok, slot=1, tokenizer=hf_text_tokenizer(hf_tok), cls_id=hf_tok.cls_token_id,
                         sep_id=hf_tok.sep_token_id)
    return ce


# (every test takes the session's gpu_index fixture: it skips without a CUDA device)
def _same(a, b):
    return all(x.dtype == y.dtype and x.shape == y.shape and (x.view(np.uint8) == y.view(np.uint8)).all()
               for x, y in zip(a, b))


# ----------------------------------------------------------------------------- a / b: against the single-query mirror
def test_batch_rerank_equals_the_single_query_mirror(gpu_index, hf_tok, tmp_path):
    from rag_search_engine_b200 import HybridSearch, runtime, store
    from rag_search_engine_b200.encoder import MINILM_L6_CONFIG, GpuSentenceEncoder, random_state_dict
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    rng = random.Random(5)
    docs = [{"id": 7 + 3 * i, "title": " ".join(rng.choices(WORDS, k=2)),
             "description": " ".join(rng.choices(WORDS, k=rng.randint(8, 40))) + "."} for i in range(160)]
    # two movies with the same text: equal logits, so their order falls back to the RRF score and position
    docs.append({"id": 1000, "title": "w1 w2", "description": "w3 w4 w5 w6."})
    docs.append({"id": 1003, "title": "w1 w2", "description": "w3 w4 w5 w6."})
    db = tmp_path / "rerank.db"
    idx = runtime.acquire(db, 0)
    try:
        enc = GpuSentenceEncoder(idx, random_state_dict(MINILM_L6_CONFIG, seed=1), MINILM_L6_CONFIG,
                                 tokenizer=lambda texts: hf_tok(list(texts), truncation=True, max_length=256)["input_ids"])
        store.write_reference_db(db, docs, whitespace_tokenizer, embed=enc.encode)
        ce = _cross_encoder(idx, hf_tok)
        hs = HybridSearch(docs_path=None, db_path=db, tokenizer=whitespace_tokenizer, encoder=enc, cross_encoder=ce)
        try:
            n_docs = hs.load_rerank_documents()
            assert n_docs == len(docs)
            qs = ["w1 w2 w3"] + [" ".join(rng.choices(WORDS, k=rng.randint(1, 5))) for _ in range(39)]
            vecs = np.stack([hs.semantic.generate_embedding(q)[0] for q in qs])
            toks, qids = whitespace_tokenizer(qs), ce.tokenize(qs)
            tie_seen = False
            for ml in (512, 24, 16):                        # 24 / 16 cut documents, queries and both
                ce.max_length = ml
                for act in ACTIVATIONS:
                    ce.activation = act
                    for limit in (1, 5, 10, 64):
                        got = hs.rrf_search_batch(toks, vecs, k=60, limit=limit, rerank_method="cross_encoder",
                                                  rerank_query_ids=qids)
                        for q, g in zip(qs, got):
                            want = hs.rrf_search(q, k=60, limit=limit, rerank_method="cross_encoder")
                            assert [d["id"] for d in g] == [d["id"] for d in want], (ml, act, limit, q)
                            for x, y in zip(g, want):
                                for key in ("rrf_rank", "bm25_rank", "sem_rank", "score", "cross_encoder_score"):
                                    assert x[key] == y[key], (key, ml, act, limit, q)
                            ids = [d["id"] for d in g]
                            if 1000 in ids and 1003 in ids:
                                a, b = g[ids.index(1000)], g[ids.index(1003)]
                                assert a["cross_encoder_score"] == b["cross_encoder_score"]
                                first, second = (a, b) if ids.index(1000) < ids.index(1003) else (b, a)
                                assert (first["score"], -first["rrf_rank"]) > (second["score"], -second["rrf_rank"])
                                tie_seen = True
            assert tie_seen
            # a saturated sigmoid (classifier bias +40) scores every pair 1.0f: the result is the RRF order
            ce = hs.cross_encoder = _cross_encoder(idx, hf_tok, bias=40.0)
            ce.activation = "sigmoid"
            for limit in (5, 10):
                got = hs.rrf_search_batch(toks, vecs, k=60, limit=limit, rerank_method="cross_encoder",
                                          rerank_query_ids=qids, as_arrays=True)
                base = hs.rrf_search_batch(toks, vecs, k=60, limit=limit, as_arrays=True)
                assert (got[5] == np.float32(1.0))[got[0] >= 0].all()
                assert np.array_equal(got[0], base[0]) and np.array_equal(got[1], base[1])
                assert np.array_equal(got[6], base[4])
                assert all((got[4][q, :got[6][q]] == np.arange(1, got[6][q] + 1)).all() for q in range(len(qs)))
        finally:
            hs.close()
    finally:
        runtime.release(db, 0)


# ----------------------------------------------------------------------------- c / d / e / f: a synthetic corpus
@pytest.fixture(scope="module")
def synth_setup(gpu_index, hf_tok):
    from rag_search_engine_b200 import HybridSearch, _lib, synth
    from rag_search_engine_b200.encoder import MINILM_L6_CONFIG, GpuSentenceEncoder, random_state_dict
    se = synth.synth_embeddings(3000, seed=31, device="cpu")
    bm = synth.synth_bm25(3000, 2000, seed=31, mean_len=30, sd_len=10)
    idx = _lib.Index(0)
    idx.load_embeddings(se.emb.numpy(), movie_idx=se.movie_of_chunk.numpy())
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    enc = GpuSentenceEncoder(idx, random_state_dict(MINILM_L6_CONFIG, seed=3), MINILM_L6_CONFIG)
    ce = _cross_encoder(idx, hf_tok, seed=4)
    T = len(bm.df)
    names = [f"t{i}" for i in range(T)]
    hs = HybridSearch.from_loaded(idx, dict(zip(names, range(T))), se.movie_ids, se.movie_ids,
                                  registry_key="rerank-synth-test", cross_encoder=ce)
    rng = np.random.default_rng(32)
    doc_ids = np.asarray(se.movie_ids, np.int64)
    doc_toks = [rng.integers(1000, 30522, int(rng.integers(100, 201))).tolist() for _ in range(len(doc_ids))]
    yield dict(idx=idx, hs=hs, se=se, bm=bm, names=names, enc=enc, ce=ce, doc_ids=doc_ids, doc_toks=doc_toks,
               synth=synth)
    hs.close()
    idx.close()


def _queries(s, nq, seed):
    synth, names = s["synth"], s["names"]
    tok_indptr, terms = synth.synth_token_queries(s["bm"], nq, seed=seed)
    toks = [[names[t] if t >= 0 else "<oov>" for t in terms[tok_indptr[i]:tok_indptr[i + 1]]] for i in range(nq)]
    vecs = synth.synth_query_vectors(s["se"].emb, nq, seed=seed).numpy()
    qids = np.random.default_rng(seed).integers(1000, 30522, (nq, 8)).tolist()
    return toks, vecs, qids


def _oracle(s, toks, vecs, qids, limit, act):
    """The single-query mirror's composition, for the batch: BM25 + KNN -> RRF over the whole union -> pairs by the
    truncation rule -> GpuCrossEncoder.predict_ids -> Python's stable sort on (score, rrf score), reverse=True."""
    from rag_search_engine_b200._lib import pair_truncate
    idx, hs, ce = s["idx"], s["hs"], s["ce"]
    tok_indptr, rows = hs.keyword._term_rows(toks)
    score, doc, bc = idx.bm25(tok_indptr, rows, limit)
    _dist, _rowid, movie, sc = idx.knn_movies(vecs, limit, limit * 10)
    L2 = 2 * limit
    pad = lambda a, fill: np.concatenate([a, np.full((a.shape[0], L2 - limit), fill, a.dtype)], 1)  # noqa: E731
    bid = pad(np.where(doc >= 0, s["doc_ids"][np.clip(doc, 0, None)], -1), -1)
    sid = pad(np.where(movie >= 0, s["doc_ids"][np.clip(movie, 0, None)], -1), -1)
    oid, osc, orb, ors, oc = idx.fuse_rrf(L2, 60.0, bid, pad(score, 0.0), bc, sid, pad(_dist.astype(np.float64), 0.0), sc)
    row_of = {int(d): i for i, d in enumerate(s["doc_ids"])}
    ids, tts, where = [], [], []
    for q in range(len(toks)):
        for j in range(int(oc[q])):
            d = s["doc_toks"][row_of[int(oid[q, j])]]
            a, b = pair_truncate(len(qids[q]), len(d), ce.max_length)
            ids.append([ce.cls_id] + qids[q][:a] + [ce.sep_id] + d[:b] + [ce.sep_id])
            tts.append([0] * (a + 2) + [1] * (b + 1))
            where.append((q, j))
    ce.activation = act
    scores = ce.predict_ids(ids, tts)
    per_q = [[] for _ in toks]
    for (q, j), c in zip(where, scores.tolist()):
        per_q[q].append({"id": int(oid[q, j]), "score": float(osc[q, j]), "bm25_rank": int(orb[q, j]),
                         "sem_rank": int(ors[q, j]), "rrf_rank": j + 1, "cross_encoder_score": c})
    out = []
    for hits in per_q:
        hits.sort(key=lambda d: (d["cross_encoder_score"], d["score"]), reverse=True)
        out.append(hits[:limit])
    return out


@pytest.mark.parametrize("act", ACTIVATIONS)
def test_synthetic_batches_against_the_host_composition(synth_setup, act):
    s = synth_setup
    hs, idx, ce = s["hs"], s["idx"], s["ce"]
    hs.load_rerank_documents(s["doc_ids"], s["doc_toks"])
    ce.activation = act
    for nq, limit, ml in ((1, 10, 512), (40, 10, 512), (300, 10, 512), (40, 64, 128), (40, 5, 60)):
        ce.max_length = ml
        toks, vecs, qids = _queries(s, nq, seed=40 + nq)
        got = hs.rrf_search_batch(toks, vecs, k=60, limit=limit, rerank_method="cross_encoder", rerank_query_ids=qids)
        want = _oracle(s, toks, vecs, qids, limit, act)
        for g, w in zip(got, want):
            assert [d["id"] for d in g] == [d["id"] for d in w]
            for x, y in zip(g, w):
                assert x["bm25_rank"] == (y["bm25_rank"] if y["bm25_rank"] >= 0 else None)
                assert x["sem_rank"] == (y["sem_rank"] if y["sem_rank"] >= 0 else None)
                for key in ("rrf_rank", "score", "cross_encoder_score"):
                    assert x[key] == y[key], (key, nq, limit)
        assert sum(len(g) for g in got) > 0
    ce.max_length = 512


@pytest.mark.parametrize("act", ACTIVATIONS)
def test_slicing_and_text_entry_point_are_bitwise_equal(synth_setup, act):
    s = synth_setup
    hs, idx, ce, enc = s["hs"], s["idx"], s["ce"], s["enc"]
    hs.load_rerank_documents(s["doc_ids"], s["doc_toks"])
    ce.activation = act
    toks, _, qids = _queries(s, 96, seed=7)
    enc_ids = np.random.default_rng(8).integers(1000, 30522, (96, 12)).tolist()
    vecs = enc.encode_ids(enc_ids)
    kw = dict(k=60, limit=10, rerank_method="cross_encoder", rerank_query_ids=qids, as_arrays=True)
    whole = hs.rrf_search_batch(toks, vecs, **kw)
    idx.set_rerank_token_budget(300)                   # about one pair per encoder slice
    try:
        sliced = hs.rrf_search_batch(toks, vecs, **kw)
    finally:
        idx.set_rerank_token_budget(1 << 17)
    assert _same(whole, sliced)
    texts = hs.rrf_search_texts(toks, enc_ids, enc, **kw)
    assert _same(whole, texts)
    assert int(whole[6].sum()) > 0


def test_rerank_status_codes(synth_setup, hf_tok):
    from rag_search_engine_b200._lib import RseError
    s = synth_setup
    hs, idx, ce = s["hs"], s["idx"], s["ce"]
    hs._ensure_id_tables()
    toks, vecs, qids = _queries(s, 8, seed=9)
    tok_indptr, rows = hs.keyword._term_rows(toks)
    q_ptr = np.arange(0, 8 * 9, 8, dtype=np.int32)
    q_ids = np.asarray(qids, np.int32).ravel()

    def run(slot=1, limit=10, q_ids=q_ids, max_length=512, activation=0):
        idx.hybrid_rerank_run(slot, 60.0, limit, q_ptr, q_ids, cls_id=ce.cls_id, sep_id=ce.sep_id,
                              max_length=max_length, activation=activation)

    def code(fn, *a, **k):
        with pytest.raises(RseError) as e:
            fn(*a, **k)
        return e.value.code, str(e.value)

    fresh = s["idx"].__class__(0)                       # a handle without a store
    try:
        fresh.load_embeddings(s["se"].emb.numpy(), movie_idx=s["se"].movie_of_chunk.numpy())
        bm = s["bm"]
        fresh.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
        fresh.set_id_tables(s["doc_ids"], s["doc_ids"])
        fresh.hybrid_stage(vecs, tok_indptr, rows)
        assert code(fresh.hybrid_rerank_run, 1, 60.0, 10, q_ptr, q_ids, cls_id=2, sep_id=3, max_length=512)[0] == -3
    finally:
        fresh.close()
    # a store without one of the fused ids: STATE, naming it
    hs.load_rerank_documents(s["doc_ids"][1:], s["doc_toks"][1:])
    idx.hybrid_stage(np.tile(_chunk_vector(s, 0), (8, 1)), tok_indptr, rows)
    c, msg = code(run)
    assert c == -3 and str(int(s["doc_ids"][0])) in msg
    hs.load_rerank_documents(s["doc_ids"], s["doc_toks"])
    idx.hybrid_stage(vecs, tok_indptr, rows)
    run()                                               # the valid call works
    assert idx.hybrid_rerank_fetch(10)[6].sum() > 0
    assert code(run, limit=0)[0] == -4 and code(run, limit=129)[0] == -4
    assert code(run, max_length=3)[0] == -4 and code(run, max_length=513)[0] == -4
    assert code(run, activation=2)[0] == -1
    assert code(run, slot=0)[0] == -1                   # head 0: the sentence encoder
    bad = q_ids.copy(); bad[3] = 30522
    assert code(run, q_ids=bad)[0] == -1
    big = [list(t) for t in s["doc_toks"]]; big[5] = big[5] + [40000]
    hs.load_rerank_documents(s["doc_ids"], big)
    assert code(run)[0] == -1
    hs.load_rerank_documents(s["doc_ids"], s["doc_toks"])
    # submit tickets in flight
    t = idx.hybrid_submit(0, 60.0, 10, vecs, tok_indptr, rows)
    idx.hybrid_stage(vecs, tok_indptr, rows)
    assert code(run)[0] == -3
    idx.hybrid_collect(t)
    # nothing staged (the staged batch parked in a stash slot)
    idx.hybrid_stage(vecs, tok_indptr, rows)
    idx.hybrid_stash(0)
    assert code(run)[0] == -3
    idx.hybrid_stash(0)
    run()
    # a slot that is not a finalized head-1 BERT: not finalized, then a CLIP text tower
    idx.encoder_create(1, vocab_size=30522, hidden=128, layers=2, heads=2, intermediate=512, max_positions=512,
                       type_vocab=2, ln_eps=1e-12, head=1)
    assert code(run)[0] == -1
    idx.clip_create(1, tower=1, hidden=128, layers=1, heads=2, intermediate=256, projection_dim=64, ln_eps=1e-5,
                    vocab_size=1000, max_positions=77, eos_token_id=2)
    assert code(run)[0] == -1
    hs.cross_encoder = s["ce"] = _cross_encoder(idx, hf_tok, seed=4)
    run()


def _chunk_vector(s, movie_row):
    """A query vector equal to a chunk of movie ``movie_row``: its KNN hits include that movie."""
    se = s["se"]
    r = int(np.nonzero(se.movie_of_chunk.numpy() == movie_row)[0][0])
    return se.emb[r].numpy()
