"""GPU: the semantic index build on the device (device_build.py, csrc/chunk.cuh) against the host build: the chunk
texts against store.plan_chunks byte for byte, the matrix against encoder.encode bit for bit, the database against
the fallback_build=True build, and the searches on the device-built handle against a fresh open."""
import json
import sqlite3

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
pytest.importorskip("transformers")

from helpers import chunk_ref  # noqa: E402
from helpers import wp_corpus as corpus  # noqa: E402

CFG = dict(vocab_size=4000, hidden=384, layers=2, heads=12, intermediate=1536, max_positions=128, type_vocab=2,
           ln_eps=1e-12)
MARKS = "\U0001d16d\U0001d165"          # two code points whose marks NFD could reorder: the host tokenizer's route


@pytest.mark.parametrize("size,overlap", chunk_ref.SIZES)
def test_device_chunks_equal_plan_chunks(gpu_index, size, overlap):
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.device_build import chunk_movies
    movies = chunk_ref.adversarial_movies(seed=100 + size * 10 + overlap, n=20000)
    got = chunk_movies(gpu_index, movies, size, overlap)
    rows, want = store.plan_chunks(movies, size, overlap)
    texts = [got.text[a:b].decode("utf-8") for a, b in zip(got.offsets[:-1].tolist(), got.offsets[1:].tolist())]
    assert len(texts) == len(want)
    bad = [i for i, (g, w) in enumerate(zip(texts, want)) if g != w]
    assert not bad, (len(bad), repr(texts[bad[0]]), repr(want[bad[0]]))
    assert [(movies[m][0], i) for m, i in zip(got.movie.tolist(), got.chunk_index.tolist())] == \
        [(r[1], r[2]) for r in rows]


def test_device_chunking_refuses_bad_input(gpu_index):
    from rag_search_engine_b200._lib import RseError
    from rag_search_engine_b200.device_build import chunk_movies
    with pytest.raises(ValueError):
        chunk_movies(gpu_index, [(1, "T", "A. B.")], 0, 0)
    text = torch.zeros(8, dtype=torch.uint8, device="cuda:0")
    offs = torch.tensor([0, 4, 2], dtype=torch.int64, device="cuda:0")        # decreasing
    cu = torch.empty(2, dtype=torch.int64, device="cuda:0")
    with pytest.raises(RseError, match="offsets"):
        gpu_index.chunk_count(text.data_ptr(), 8, offs.data_ptr(), 1, 3, 1, cu.data_ptr(), cu.data_ptr())
    offs = torch.tensor([0, 4, 9], dtype=torch.int64, device="cuda:0")        # past the text
    with pytest.raises(RseError, match="offsets"):
        gpu_index.chunk_count(text.data_ptr(), 8, offs.data_ptr(), 1, 3, 1, cu.data_ptr(), cu.data_ptr())


def _movies(n, seed, routed_every=0):
    """Movie-shaped rows: wp_corpus text cut into 3-25 sentences; every routed_every-th description carries MARKS."""
    import random
    rnd = random.Random(seed)
    pool = corpus.texts(4 * n + 100, seed=seed)
    out = []
    for i in range(n):
        sents = [(" ".join(rnd.choice(pool).split()[:12]) or "x") + rnd.choice([".", "!", "?"])
                 for _ in range(rnd.randint(3, 25))]
        desc = " ".join(sents)
        if routed_every and i % routed_every == 3:
            desc = desc[:20] + MARKS + desc[20:]
        out.append((2 * i + 5, " ".join(rnd.choice(pool).split()[:5]) or "t", desc))
    return out


def _encoder(idx, slot=0):
    from rag_search_engine_b200.encoder import DeviceWordPiece, GpuSentenceEncoder, random_state_dict
    tok = corpus.tokenizer("uncased")
    dw = DeviceWordPiece(idx, tok, slot=slot, max_length=128)
    return GpuSentenceEncoder(idx, random_state_dict(CFG, seed=11), CFG, dw, slot=slot, max_seq_length=128)


def test_device_matrix_equals_encode(gpu_index):
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.device_build import build_embeddings
    enc = _encoder(gpu_index)
    movies = _movies(3000, seed=3, routed_every=97)
    _, texts = store.plan_chunks(movies, 3, 1)
    want = enc.encode(texts)
    nh = enc.tokenizer.tables.needs_host
    routed = [m for m, (_, t, d) in enumerate(movies) if nh(t) or nh(d)]
    assert set(range(3, 3000, 97)) <= set(routed) and len(routed) < len(movies)
    for kw in ({}, dict(part_bytes=1, max_tokens_per_call=300), dict(part_bytes=50000)):
        before = enc.tokenizer.host_texts
        b = build_embeddings(enc, movies, 3, 1, **kw)
        assert b.host_movies == len(routed)
        assert enc.tokenizer.host_texts - before == sum(int(b.chunks_per_movie[m]) for m in routed)
        got = b.emb.cpu().numpy()
        assert got.shape == want.shape and got.view(np.uint32).tobytes() == want.view(np.uint32).tobytes(), kw


def _docs(tmp_path, movies):
    p = tmp_path / "movies.json"
    p.write_text(json.dumps({"movies": [{"id": i, "title": t, "description": d} for i, t, d in movies]}))
    return p


def _tables(db):
    conn = sqlite3.connect(db)
    try:
        out = {t: conn.execute(q).fetchall() for t, q in (
            ("movies", "SELECT * FROM movies ORDER BY id"), ("chunks", "SELECT * FROM chunks ORDER BY id"),
            ("vec", "SELECT c.chunk_id, c.size, c.validity, c.rowids, v.vectors FROM chunk_embeddings_chunks c "
                    "JOIN chunk_embeddings_vector_chunks00 v ON v.rowid = c.chunk_id ORDER BY c.chunk_id"),
            ("rowids", "SELECT * FROM chunk_embeddings_rowids ORDER BY rowid"))}
    finally:
        conn.close()
    return out


@pytest.fixture(scope="module")
def built(tmp_path_factory, gpu_index):
    """The same docs built twice with the same encoder: fallback_build=True (host plan_chunks + encode) and
    device_build=True; the device-built handle stays open."""
    from rag_search_engine_b200 import runtime
    from rag_search_engine_b200.semantic_search import SemanticSearch
    tmp = tmp_path_factory.mktemp("devbuild")
    movies = _movies(2500, seed=7, routed_every=211)
    docs = _docs(tmp, movies)
    db_dev, db_host = tmp / "dev.db", tmp / "host.db"
    idx = runtime.acquire(db_dev, 0)
    enc = _encoder(idx)
    ss_host = SemanticSearch(docs_path=docs, db_path=db_host, encoder=enc, fallback_build=True)
    ss_host.close()
    ss_dev = SemanticSearch(docs_path=docs, db_path=db_dev, encoder=enc, device_build=True, fallback_build=True)
    yield dict(movies=movies, docs=docs, db_dev=db_dev, db_host=db_host, idx=idx, enc=enc, ss_dev=ss_dev)
    ss_dev.close()
    runtime.release(db_dev, 0)


def test_database_equals_fallback_build(built):
    assert _tables(built["db_dev"]) == _tables(built["db_host"])


def test_device_built_handle_serves_like_a_fresh_open(built, monkeypatch):
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.semantic_search import SemanticSearch
    ss_dev = built["ss_dev"]
    assert ss_dev._index.n_rows == len(store.plan_chunks(built["movies"], 3, 1)[0])
    rng = np.random.default_rng(5)
    Q = rng.standard_normal((64, 384)).astype(np.float32)
    fresh = SemanticSearch(db_path=built["db_host"], encoder=built["enc"])
    try:
        for q in (Q[:1], Q[:8], Q):
            assert ss_dev.query_top_k_vec(q, k=5) == fresh.query_top_k_vec(q, k=5)
        for h in (ss_dev._index, fresh._index):
            h.set_tc_mode(2)                                  # the tensor-core filter over the fp16 shadow (K4)
        try:
            assert ss_dev.query_top_k_vec(Q, k=10) == fresh.query_top_k_vec(Q, k=10)
        finally:
            for h in (ss_dev._index, fresh._index):
                h.set_tc_mode(0)
    finally:
        fresh.close()
    # a fresh open of the device-built database reads its sidecar: no export
    from rag_search_engine_b200 import runtime

    def no_export(*a, **k):
        raise AssertionError("the device-built database was exported again")
    monkeypatch.setattr(store, "export_embeddings", no_export)
    key = (str(built["db_dev"].resolve()), 0)              # set the live handle aside: a new one opens the file
    saved = runtime._handles.pop(key)
    try:
        again = SemanticSearch(db_path=built["db_dev"], encoder=built["enc"])
        try:
            assert again.query_top_k_vec(Q[:8], k=5) == ss_dev.query_top_k_vec(Q[:8], k=5)
        finally:
            again.close()
    finally:
        runtime._handles[key] = saved


def test_force_in_sync_and_errors(built, monkeypatch, tmp_path):
    from rag_search_engine_b200 import _lib, device_build, runtime
    from rag_search_engine_b200.semantic_search import SemanticSearch
    calls = []
    real = device_build.build_embeddings
    monkeypatch.setattr(device_build, "build_embeddings", lambda *a, **k: calls.append(1) or real(*a, **k))
    kw = dict(docs_path=built["docs"], db_path=built["db_dev"], encoder=built["enc"], device_build=True,
              fallback_build=True)
    SemanticSearch(**kw).close()                              # in sync: skipped
    assert calls == []
    s = SemanticSearch(force=True, **kw)                      # forced: rebuilt, same tables
    assert calls == [1]
    s.close()
    assert _tables(built["db_dev"]) == _tables(built["db_host"])
    other = _lib.Index(0)                                     # an encoder on another handle
    try:
        with pytest.raises(ValueError, match="handle"):
            SemanticSearch(docs_path=built["docs"], db_path=tmp_path / "x.db", encoder=_encoder(other),
                           device_build=True, fallback_build=True)
    finally:
        other.close()
    from rag_search_engine_b200.encoder import GpuSentenceEncoder, random_state_dict
    idx = runtime.acquire(tmp_path / "y.db", 0)
    try:
        tok = corpus.tokenizer("uncased")
        host_tok = GpuSentenceEncoder(idx, random_state_dict(CFG, seed=11), CFG,
                                      lambda t: tok(list(t))["input_ids"], max_seq_length=128)
        with pytest.raises(TypeError, match="DeviceWordPiece"):
            SemanticSearch(docs_path=built["docs"], db_path=tmp_path / "y.db", encoder=host_tok, device_build=True,
                           fallback_build=True)
        with pytest.raises(ValueError, match="max_chunk_size"):
            SemanticSearch(docs_path=built["docs"], db_path=tmp_path / "y.db", encoder=host_tok, device_build=True,
                           fallback_build=True, max_chunk_size=0)
    finally:
        runtime.release(tmp_path / "y.db", 0)


def test_sqlite_vec_opens_the_device_built_file(gpu_index, tmp_path):
    sqlite_vec = pytest.importorskip("sqlite_vec")
    from rag_search_engine_b200 import runtime, store
    from rag_search_engine_b200.semantic_search import SemanticSearch
    movies = _movies(300, seed=9)
    db = tmp_path / "v.db"
    idx = runtime.acquire(db, 0)
    try:
        SemanticSearch(docs_path=_docs(tmp_path, movies), db_path=db, encoder=_encoder(idx), device_build=True).close()
    finally:
        runtime.release(db, 0)
    conn = sqlite3.connect(db)
    conn.enable_load_extension(True)
    sqlite_vec.load(conn)
    n = len(store.plan_chunks(movies, 3, 1)[0])
    assert conn.execute("SELECT COUNT(*) FROM chunk_embeddings").fetchone()[0] == n
    assert sorted(r[0] for r in conn.execute("SELECT rowid FROM chunk_embeddings")) == list(range(n))
    conn.close()


def test_chunk_write_at_a_movie_offset(gpu_index):
    """A part of the movies (m0 > 0) is addressed through its slice of the offsets and reports rows m0 + m."""
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.device_build import _upload, _write, pack_movies
    movies = chunk_ref.adversarial_movies(seed=8, n=500)
    data, offs = pack_movies(movies)
    text, offs_dev = _upload(torch, data, offs, torch.device("cuda", 0))
    m0, m1 = 137, 402
    out, o_offs, o_movie, o_index, nb = _write(gpu_index, text, len(data), offs_dev, m0, m1, 3, 1, torch,
                                               torch.device("cuda", 0))
    o = o_offs.cpu().numpy()
    got = out[:nb].cpu().numpy().tobytes()
    rows, want = store.plan_chunks(movies[m0:m1], 3, 1)
    assert [got[a:b].decode("utf-8") for a, b in zip(o[:-1].tolist(), o[1:].tolist())] == want
    assert o_movie.cpu().numpy().tolist() == [m0 + [m[0] for m in movies[m0:m1]].index(r[1]) for r in rows]
    assert o_index.cpu().numpy().tolist() == [r[2] for r in rows]


def test_empty_docs_give_an_empty_index(gpu_index, tmp_path):
    from rag_search_engine_b200 import runtime
    from rag_search_engine_b200.semantic_search import SemanticSearch
    db = tmp_path / "e.db"
    idx = runtime.acquire(db, 0)
    try:
        ss = SemanticSearch(docs_path=_docs(tmp_path, []), db_path=db, encoder=_encoder(idx), device_build=True,
                            fallback_build=True)
        try:
            assert ss.query_top_k_vec(np.ones((2, 384), np.float32), k=5) == [[], []]
            assert ss.conn.execute("SELECT COUNT(*) FROM chunks").fetchone()[0] == 0
        finally:
            ss.close()
    finally:
        runtime.release(db, 0)


def test_reference_sync_is_used_and_its_rows_are_read_back(gpu_index, tmp_path, monkeypatch):
    """With the reference importable, its BaseSearchDB syncs the movies table (here a stand-in that stores fixed
    texts) and the build chunks the rows it finds in the table, not the JSON."""
    import sys
    import types
    from rag_search_engine_b200 import runtime, store
    from rag_search_engine_b200.semantic_search import SemanticSearch
    movies = _movies(40, seed=12)
    fixed = [(i, t.upper(), d.upper()) for i, t, d in movies]
    calls = []

    class BaseSearchDB:
        def __init__(self, docs_path=None, db_path=None):
            calls.append((docs_path, db_path))
            self.conn = sqlite3.connect(db_path)
            self.conn.execute("DELETE FROM movies")
            self.conn.executemany("INSERT INTO movies(id, title, description) VALUES (?, ?, ?)", fixed)
            self.conn.commit()

        def close(self):
            self.conn.close()
    pkg = types.ModuleType("rag_search_engine")
    utils = types.ModuleType("rag_search_engine.utils")
    mod = types.ModuleType("rag_search_engine.utils.basesearch_db")
    mod.BaseSearchDB = BaseSearchDB
    for name, m in (("rag_search_engine", pkg), ("rag_search_engine.utils", utils),
                    ("rag_search_engine.utils.basesearch_db", mod)):
        monkeypatch.setitem(sys.modules, name, m)
    db = tmp_path / "r.db"
    docs = _docs(tmp_path, movies)
    idx = runtime.acquire(db, 0)
    try:
        enc = _encoder(idx)
        ss = SemanticSearch(docs_path=docs, db_path=db, encoder=enc, device_build=True, fallback_build=True)
        try:
            assert calls == [(docs, db)]
            rows, texts = store.plan_chunks(fixed, 3, 1)
            assert ss.conn.execute("SELECT id, movie_id, chunk_index, max_chunk_size, overlap FROM chunks "
                                   "ORDER BY id").fetchall() == rows
            got = ss._arr.emb
            assert np.asarray(got).view(np.uint32).tobytes() == enc.encode(texts).view(np.uint32).tobytes()
        finally:
            ss.close()
    finally:
        runtime.release(db, 0)


def test_hybrid_search_device_build_equals_a_fresh_open_of_the_fallback_build(gpu_index, tmp_path):
    """HybridSearch passes device_build through; rrf_search_batch on the device-built handle equals a fresh open of
    the database HybridSearch(..., fallback_build=True) built with the same encoder."""
    from rag_search_engine_b200 import HybridSearch, runtime
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    movies = _movies(1500, seed=21, routed_every=301)
    docs = _docs(tmp_path, movies)
    db_dev, db_host = tmp_path / "hd.db", tmp_path / "hh.db"
    idx = runtime.acquire(db_dev, 0)
    try:
        enc = _encoder(idx)
        HybridSearch(docs_path=docs, db_path=db_host, tokenizer=whitespace_tokenizer, encoder=enc,
                     fallback_build=True).close()
        hd = HybridSearch(docs_path=docs, db_path=db_dev, tokenizer=whitespace_tokenizer, encoder=enc,
                          device_build=True, fallback_build=True)
        hh = HybridSearch(docs_path=None, db_path=db_host, tokenizer=whitespace_tokenizer, encoder=enc)
        try:
            assert hd.semantic._index is idx and "emb_dev" in runtime.parts(db_dev, 0)
            assert _tables(db_dev) == _tables(db_host)
            rng = np.random.default_rng(3)
            words = " ".join(d for _, _, d in movies[:50]).lower().split()
            toks = [[str(w) for w in rng.choice(words, rng.integers(1, 6))] for _ in range(64)]
            Q = enc.encode([" ".join(t) for t in toks])
            for nq, limit in ((1, 10), (8, 5), (64, 10)):
                assert hd.rrf_search_batch(toks[:nq], Q[:nq], limit=limit) == \
                    hh.rrf_search_batch(toks[:nq], Q[:nq], limit=limit)
        finally:
            hh.close()
            hd.close()
    finally:
        runtime.release(db_dev, 0)
