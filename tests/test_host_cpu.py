"""CPU tests of the host side: C-ABI library loads and exports every symbol include/rse.h declares
(no compute), the SQLite exporter/writer round trip, the text helpers against the reference's own
functions, the CPython-set emulation against the real set, and the oracle-stays-out-of-the-product rule."""
import ctypes
import json
import random
import re
import sqlite3
import subprocess
from pathlib import Path

import numpy as np
import pytest

from oracle import ref_import
from helpers.corpus import build_postings, to_csr

ROOT = Path(__file__).resolve().parents[1]
GOLDEN = ROOT / "tests" / "golden"


# ----------------------------------------------------------------------------- C-ABI surface
def test_library_exports_every_declared_symbol():
    from rag_search_engine_b200 import _lib
    header = (ROOT / "include" / "rse.h").read_text()
    declared = set(re.findall(r"^\s*(?:int|void|const char \*)\s*\*?(rse_[a-z0-9_]+)\(", header, re.M))
    assert len(declared) >= 25
    L = _lib.load_library()                                   # dlopen works without a GPU
    for name in declared:
        assert hasattr(L, name), f"{name} declared in rse.h but not exported by librse.so"
    assert declared == set(_lib.EXPORTED_SYMBOLS), declared ^ set(_lib.EXPORTED_SYMBOLS)
    assert L.rse_abi_version() == 2


def test_no_cpu_fallback_without_gpu():
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from rag_search_engine_b200 import _lib
    with pytest.raises(_lib.RseError) as e:
        _lib.Index(0)
    assert "no CPU fallback" in str(e.value) or "CUDA" in str(e.value)


def test_product_never_touches_the_oracle():
    """Only tests/, __graft_entry__.smoke() and bench.py's baseline legs may import oracle/."""
    for p in (ROOT / "rag_search_engine_b200").rglob("*"):
        if p.suffix in (".py", ".cu", ".cuh", ".h"):
            txt = p.read_text()
            assert not re.search(r"^\s*(from|import)\s+oracle\b", txt, re.M), p
            assert "liboracle" not in txt and "oracle/" not in txt.replace("oracle/make_golden", ""), p


# ----------------------------------------------------------------------------- CPython set emulation
@pytest.fixture(scope="module")
def pyset_shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("shim") / "pyset_shim.so"
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", str(so), str(ROOT / "tests" / "helpers" / "pyset_shim.cpp")],
                   check=True)
    return ctypes.CDLL(str(so))


def test_pyset_emulation_matches_cpython(pyset_shim):
    P = ctypes.POINTER(ctypes.c_int64)

    def emu(a, b):
        A, B = np.array(a, np.int64), np.array(b, np.int64)
        out = np.zeros(len(a) + len(b) + 1, np.int64)
        n = pyset_shim.pyset_shim_union(A.ctypes.data_as(P), len(a), B.ctypes.data_as(P), len(b), out.ctypes.data_as(P))
        return out[:n].tolist()

    def real(a, b):
        da, db = {x: None for x in a}, {x: None for x in b}
        return list(set(da.keys()) | set(db.keys()))          # hybrid_search.py:148, :248

    assert emu([9], [2]) == [9, 2] and emu([16, 3], [8, 1]) == [16, 8, 3, 1]     # SURVEY App. A.5
    rnd = random.Random(1)
    for _ in range(20000):
        na, nb = rnd.randint(0, rnd.choice([3, 10, 40, 128])), rnd.randint(0, rnd.choice([3, 10, 40, 128]))
        space = rnd.choice([16, 64, 1000, 10**6, 10**9, 2**40, 2**62])
        lo = -space if rnd.random() < 0.1 else 0
        a = list(dict.fromkeys(rnd.randrange(lo, space) for _ in range(na)))
        b = list(dict.fromkeys((rnd.choice(a) if a and rnd.random() < 0.3 else rnd.randrange(lo, space))
                               for _ in range(nb)))
        assert emu(a, b) == real(a, b), (a, b)


# ----------------------------------------------------------------------------- text helpers
def test_window_chunks_known_shapes():
    from rag_search_engine_b200.textutil import chunk_text, sentence_chunks, window_chunks
    # rag_search_engine/tests/test_utils.py:100-109
    ch = sentence_chunks("Sentence one. Sentence two! Sentence three?", 2, 1)
    assert ch == [["Sentence one.", "Sentence two!"], ["Sentence two!", "Sentence three?"]]
    # SURVEY App. B: S sentences → 1 if S<=3 else 1+ceil((S-3)/2) chunks at (3, 1)
    for S in range(1, 12):
        text = " ".join(f"s{i}." for i in range(S))
        assert len(sentence_chunks(text, 3, 1)) == (1 if S <= 3 else 1 + -(-(S - 3) // 2))
    assert window_chunks(list("abcdefg"), 3, 0) == [list("abc"), list("def"), ["g"]]
    assert chunk_text("T", "A. B. C. D.", 0, 3, 1) == "T"
    assert chunk_text("T", "A. B. C. D.", 2, 3, 1) == "C.D."          # joined without separator (:182)
    assert chunk_text("T", "A. B.", 5, 3, 1) == "A. B."                # out of range → description


@pytest.mark.skipif(not ref_import.available(), reason="reference checkout not present (GPU box)")
def test_text_helpers_match_reference():
    _, _, ref_utils = ref_import.load()
    from oracle.make_golden import chunk_inputs
    from rag_search_engine_b200.textutil import sentence_chunks, window_chunks
    want = json.loads((GOLDEN / "live_ref.json").read_text())["chunks"]
    for (items, cs, ov, text), pinned in zip(chunk_inputs(), want):
        ref = [ref_utils.chunk(list(items), cs, ov), ref_utils.semantic_chunk(text, cs, ov)]
        assert window_chunks(items, cs, ov) == ref[0]
        assert sentence_chunks(text, cs, ov) == ref[1]
        assert ref == pinned                                  # the pinned answers are the reference's


def test_text_helpers_match_pinned_answers():
    """test_text_helpers_match_reference against its pinned answers (tests/golden/live_ref.json)."""
    from oracle.make_golden import chunk_inputs
    from rag_search_engine_b200.textutil import sentence_chunks, window_chunks
    want = json.loads((GOLDEN / "live_ref.json").read_text())["chunks"]
    cases = chunk_inputs()
    assert len(cases) == len(want) == 400
    for (items, cs, ov, text), pinned in zip(cases, want):
        assert [window_chunks(items, cs, ov), sentence_chunks(text, cs, ov)] == pinned, (items, cs, ov, text)


# ----------------------------------------------------------------------------- SQLite exporter / writer
def _docs(seed=3, n=60):
    from oracle.make_golden import sentence_corpus
    return sentence_corpus(seed, n)


def test_export_bm25_round_trip_matches_reference_layout(tmp_path, monkeypatch):
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    docs, _, _ = _docs()
    db = store.write_reference_db(tmp_path / "m.db", docs, whitespace_tokenizer)
    conn = sqlite3.connect(db)
    arr = store.export_bm25(conn)
    postings, doclen = build_postings(docs)
    csr = to_csr(postings, doclen)
    assert arr.n_movies == len(docs) and arr.avgdl == csr["avgdl"]
    assert (arr.doc_ids == csr["doc_ids"]).all() and (arr.dl == csr["dl"]).all()
    for term, row in csr["row"].items():
        r = arr.term_row[term]
        a = slice(arr.indptr[r], arr.indptr[r + 1]); b = slice(csr["indptr"][row], csr["indptr"][row + 1])
        assert (arr.doc_idx[a] == csr["doc"][b]).all() and (arr.tf[a] == csr["tf"][b]).all()
        assert arr.df[r] == csr["df"][row]
    # the table is read in slices cut on cumulative per-term counts: tiny slices (many cuts, single-term slices,
    # a term larger than a slice) give the same arrays
    monkeypatch.setattr(store, "EXPORT_SLICE_POSTINGS", 7)
    arr_s = store.export_bm25(conn)
    for f in ("indptr", "doc_idx", "tf", "df", "dl", "doc_ids"):
        assert (getattr(arr_s, f) == getattr(arr, f)).all(), f
    monkeypatch.undo()
    # a posting whose doc has no doclen row is counted in df (:222) but dropped from the CSR (:235-236)
    tid = conn.execute("SELECT id FROM terms LIMIT 1").fetchone()[0]
    conn.execute("INSERT INTO postings(term_id, doc_id, positions) VALUES (?, ?, ?)", (tid, 10**9, "[0, 1]"))
    conn.commit()
    arr2 = store.export_bm25(conn)
    r = [v for k, v in arr2.term_row.items()][0]
    assert arr2.df.sum() == arr.df.sum() + 1 and len(arr2.doc_idx) == len(arr.doc_idx)
    conn.close()


@pytest.mark.skipif(not ref_import.available(), reason="reference checkout not present (GPU box)")
def test_writer_produces_the_tables_the_reference_build_produces(tmp_path):
    from oracle.make_golden import encode_tables, reference_tables
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    ref_kw, _, _ = ref_import.load()
    docs, _, _ = _docs(5, 40)
    a = reference_tables(ref_kw, docs, tmp_path)
    store.write_reference_db(tmp_path / "ours.db", docs, whitespace_tokenizer)
    b = store.export_bm25(sqlite3.connect(tmp_path / "ours.db"))
    assert a.n_movies == b.n_movies and a.avgdl == b.avgdl and (a.dl == b.dl).all() and (a.doc_ids == b.doc_ids).all()
    assert set(a.term_row) == set(b.term_row)
    for t in a.term_row:
        ra, rb = a.term_row[t], b.term_row[t]
        sa, sb = slice(a.indptr[ra], a.indptr[ra + 1]), slice(b.indptr[rb], b.indptr[rb + 1])
        assert (a.doc_idx[sa] == b.doc_idx[sb]).all() and (a.tf[sa] == b.tf[sb]).all()
    assert encode_tables(a) == json.loads((GOLDEN / "live_ref.json").read_text())["tables"]   # pinned = reference


def test_writer_tables_match_pinned_answers(tmp_path):
    """test_writer_produces_the_tables_the_reference_build_produces against its pinned answers
    (tests/golden/live_ref.json): documents, lengths, and every term's postings and term frequencies."""
    from oracle.make_golden import encode_tables
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    docs, _, _ = _docs(5, 40)
    store.write_reference_db(tmp_path / "ours.db", docs, whitespace_tokenizer)
    got = encode_tables(store.export_bm25(sqlite3.connect(tmp_path / "ours.db")))
    want = json.loads((GOLDEN / "live_ref.json").read_text())["tables"]
    assert got["n_movies"] == want["n_movies"] == 40 and got["avgdl"] == want["avgdl"]
    assert got["dl"] == want["dl"] and got["doc_ids"] == want["doc_ids"]
    assert got["postings"] == want["postings"]


def test_export_embeddings_physical_layout(tmp_path):
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    docs, _, _ = _docs(7, 300)                                # > 1024 chunks → 2+ vec0 blocks
    rng = np.random.default_rng(0)

    def embed(texts):
        return rng.standard_normal((len(texts), 16)).astype(np.float32)

    db = store.write_reference_db(tmp_path / "v.db", docs, whitespace_tokenizer, embed=embed)
    conn = sqlite3.connect(db)
    arr = store.export_embeddings(conn)
    n_chunks = conn.execute("SELECT COUNT(*) FROM chunks").fetchone()[0]
    assert arr.emb.shape == (n_chunks, 16) and arr.valid is None and n_chunks > 1024
    assert (arr.rowid == np.arange(n_chunks)).all()           # fresh build: rowid i at position i (:164-206)
    movie_of = dict(conn.execute("SELECT id, movie_id FROM chunks").fetchall())
    assert [int(arr.movie_ids[m]) for m in arr.movie_idx] == [movie_of[i] for i in range(n_chunks)]
    # punch holes (what a DELETE leaves behind) and orphan a chunk: export must flag them
    blob = conn.execute("SELECT validity FROM chunk_embeddings_chunks WHERE chunk_id = 1").fetchone()[0]
    bits = np.unpackbits(np.frombuffer(blob, np.uint8), bitorder="little"); bits[[5, 77]] = 0
    conn.execute("UPDATE chunk_embeddings_chunks SET validity = ? WHERE chunk_id = 1",
                 (np.packbits(bits, bitorder="little").tobytes(),))
    conn.execute("DELETE FROM chunks WHERE id = 9")
    conn.commit()
    arr2 = store.export_embeddings(conn)
    assert arr2.valid is not None and arr2.valid[5] == 0 and arr2.valid[77] == 0 and arr2.valid.sum() == n_chunks - 2
    assert arr2.movie_idx[9] == -1 and arr2.movie_idx[5] == -1
    # a chunk whose MOVIE is gone is dropped by the second JOIN (semantic_search.py:275-276); the other rows keep
    # their dense movie index into the shrunken movies table
    gone = movie_of[20]
    conn.execute("DELETE FROM movies WHERE id = ?", (gone,))
    conn.commit()
    arr3 = store.export_embeddings(conn)
    for i in range(n_chunks):
        want = -1 if (i in (5, 77, 9) or movie_of[i] == gone) else movie_of[i]
        got = -1 if arr3.movie_idx[i] < 0 else int(arr3.movie_ids[arr3.movie_idx[i]])
        assert got == want, i
    # a block with no live row at all is skipped: the rows of the later blocks move up by 1024 physical slots
    dead = np.zeros(1024, np.uint8)
    conn.execute("UPDATE chunk_embeddings_chunks SET validity = ? WHERE chunk_id = 1",
                 (np.packbits(dead, bitorder="little").tobytes(),))
    conn.commit()
    arr4 = store.export_embeddings(conn)
    assert arr4.emb.shape[0] == n_chunks - 1024 and (arr4.rowid == np.arange(1024, n_chunks)).all()
    assert (arr4.emb == arr.emb[1024:]).all() and (arr4.movie_idx == arr3.movie_idx[1024:]).all()
    conn.close()


def test_shard_bounds_and_query_slices():
    from rag_search_engine_b200.sharded import query_slices, shard_bounds
    for n in (1, 1023, 1024, 1025, 4_799_462, 100_000_000):
        for w in (1, 2, 3, 4, 8):
            b = shard_bounds(n, w)
            assert b[0] == 0 and b[-1] == n and len(b) == w + 1
            assert all(x % 1024 == 0 for x in b[:-1]) and all(b[i] <= b[i + 1] for i in range(w))
    assert query_slices(10, 4) == [0, 3, 6, 8, 10] and query_slices(2, 4) == [0, 1, 2, 2, 2]


def test_sidecar_cache_round_trip_and_invalidation(tmp_path):
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    docs, _, _ = _docs(9, 80)
    rng = np.random.default_rng(1)
    db = store.write_reference_db(tmp_path / "s.db", docs, whitespace_tokenizer,
                                  embed=lambda texts: rng.standard_normal((len(texts), 8)).astype(np.float32))
    conn = sqlite3.connect(db)
    a = store.load_or_export(conn, db, "bm25")
    e = store.load_or_export(conn, db, "emb")
    assert store.sidecar_path(db, "bm25").exists() and store.sidecar_path(db, "emb").exists()
    a2 = store.load_or_export(conn, db, "bm25")          # served from the sidecar
    e2 = store.load_or_export(conn, db, "emb")
    for f in ("indptr", "doc_idx", "tf", "df", "dl", "doc_ids"):
        assert (getattr(a, f) == getattr(a2, f)).all()
    assert a.term_row == a2.term_row and a.avgdl == a2.avgdl and a.n_movies == a2.n_movies
    assert (e.emb == e2.emb).all() and (e.rowid == e2.rowid).all() and (e.movie_idx == e2.movie_idx).all() and e2.valid is None
    # the matrix comes back memory-mapped from its own .npy, contiguous float32 (what the ctypes stub passes on as is)
    assert isinstance(e2.emb, np.memmap) and e2.emb.dtype == np.float32 and e2.emb.flags["C_CONTIGUOUS"]
    assert store.emb_matrix_path(db).exists()
    # a matrix file that does not belong to the sidecar (wrong shape) is not trusted: re-export
    np.save(store.emb_matrix_path(db), np.zeros((3, 8), np.float32))
    e4 = store.load_or_export(conn, db, "emb")
    assert (np.asarray(e4.emb) == np.asarray(e.emb)).all()
    # a change in the database invalidates the sidecar
    conn.execute("INSERT INTO movies(id, title, description) VALUES (999999, 'x', 'y')")
    conn.commit()
    a3 = store.load_or_export(conn, db, "bm25")
    assert a3.n_movies == a.n_movies + 1
    # ADVICE r01: an in-place rewrite that keeps every row count (a forced re-embed through ANOTHER connection
    # in WAL mode: file size and mtime of the main file unchanged) must invalidate the sidecar as well
    e5 = store.load_or_export(conn, db, "emb")
    conn.execute("PRAGMA journal_mode=WAL")
    other = sqlite3.connect(db)
    other.execute("PRAGMA journal_mode=WAL")
    (rid, blob) = other.execute("SELECT rowid, vectors FROM chunk_embeddings_vector_chunks00 ORDER BY rowid LIMIT 1").fetchone()
    vec = np.frombuffer(blob, np.float32).copy()
    vec[:8] += 1.0
    other.execute("UPDATE chunk_embeddings_vector_chunks00 SET vectors = ? WHERE rowid = ?", (vec.tobytes(), rid))
    other.commit()
    e6 = store.load_or_export(conn, db, "emb")
    assert not (np.asarray(e6.emb)[0, :8] == np.asarray(e5.emb)[0, :8]).any(), "stale sidecar served after an in-place rewrite"
    other.close()
    # no temporary files are left behind by the atomic writes
    assert not [p for p in Path(db).parent.iterdir() if ".tmp" in p.name]
    conn.close()


def test_query_only_open_without_vec0_tables_is_empty_not_an_error(tmp_path):
    """ADVICE r01: a keyword-only / fresh database has no vec0 shadow tables; the reference creates an empty
    chunk_embeddings table at open time and query_top_k returns [] — the exporter returns an empty matrix."""
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    docs = [{"id": 1, "title": "a b", "description": "c d."}, {"id": 2, "title": "e", "description": "f."}]
    db = store.write_reference_db(tmp_path / "k.db", docs, whitespace_tokenizer)       # keyword tables only
    conn = sqlite3.connect(db)
    e = store.export_embeddings(conn)
    assert e.emb.shape[0] == 0 and e.dim == 0 and e.movie_ids.tolist() == [1, 2]
    fresh = sqlite3.connect(tmp_path / "fresh.db")
    e = store.export_embeddings(fresh)
    assert e.emb.shape[0] == 0 and len(e.movie_ids) == 0
    conn.close(); fresh.close()


def test_synthetic_corpus_is_deterministic_and_keeps_its_tie_cases():
    """Every rank of a multi-GPU bench builds the corpus from the same seeds and the results are compared bit for
    bit across ranks, so the generator must not depend on scatter order: the duplicate / near-duplicate rows are
    written through de-duplicated destination indices (an indexed assignment with repeated destinations picks a
    different winner from run to run on CUDA)."""
    import torch
    from rag_search_engine_b200 import synth
    a = synth.synth_embeddings(4000, seed=7, device="cpu")
    b = synth.synth_embeddings(4000, seed=7, device="cpu")
    assert torch.equal(a.emb.view(torch.int32), b.emb.view(torch.int32))
    assert torch.equal(a.movie_of_chunk, b.movie_of_chunk)
    c = synth.synth_embeddings(4000, seed=8, device="cpu")
    assert not torch.equal(a.emb.view(torch.int32), c.emb.view(torch.int32))
    # exact duplicate rows (duplicate "titles", SURVEY §8d) are still there: ~2 % of the rows
    rows = a.emb.view(torch.int32).numpy()
    uniq = np.unique(rows, axis=0).shape[0]
    assert 0.005 * rows.shape[0] < rows.shape[0] - uniq < 0.04 * rows.shape[0]
    # rows stay unit length (a near-duplicate differs from its source by one ulp in one component)
    norms = np.linalg.norm(a.emb.numpy().astype(np.float64), axis=1)
    assert np.abs(norms - 1.0).max() < 1e-5


def test_rrf_search_stream_keeps_two_batches_in_flight_and_the_order(tmp_path):
    """Host logic of HybridSearch.rrf_search_stream against a fake handle: every batch is submitted before the
    previous one is collected (never more than two tickets outstanding), tickets are collected in submission
    order, an empty batch drains the pipeline and yields [], results come back in the order of the batches."""
    from pathlib import Path
    from rag_search_engine_b200 import hybrid_search as hsm, runtime
    from rag_search_engine_b200.keyword_search import KeywordSearch
    from rag_search_engine_b200.semantic_search import SemanticSearch

    class FakeIndex:
        def __init__(self):
            self.next, self.outstanding, self.log, self.max_outstanding = 0, [], [], 0
        def set_id_tables(self, a, b):
            self.log.append("ids")
        def hybrid_submit(self, mode, param, limit, Q, tok_indptr, rows, **kw):
            assert mode == 0 and param == 60.0 and len(tok_indptr) == len(Q) + 1
            assert len(self.outstanding) < 2, "a third batch in flight"
            t = self.next; self.next += 1
            self.outstanding.append((t, len(Q), limit))
            self.max_outstanding = max(self.max_outstanding, len(self.outstanding))
            self.log.append(("submit", t))
            return t
        def hybrid_collect(self, ticket):
            t, nq, limit = self.outstanding.pop(0)
            assert t == ticket, "collected out of order"
            self.log.append(("collect", t))
            oid = np.full((nq, limit), 100 * t, np.int64) + np.arange(limit)
            osc = np.tile(1.0 / (1 + np.arange(limit)), (nq, 1))
            oa = np.tile(np.arange(limit, dtype=np.float64), (nq, 1)); oa[:, -1] = -1.0
            ob = -np.ones((nq, limit))
            return oid, osc, oa, ob, np.full(nq, limit - 1, np.int32)
        def hybrid_drain(self):
            n = len(self.outstanding)
            self.outstanding.clear()
            self.log.append(("drain", n))
            return n

    class Arr:
        term_row = {"a": 0, "b": 1}
        doc_ids = np.arange(3, dtype=np.int64)
        movie_ids = np.arange(3, dtype=np.int64)

    db = tmp_path / "x.db"
    db.touch()
    hs = hsm.HybridSearch.__new__(hsm.HybridSearch)
    kw = KeywordSearch.__new__(KeywordSearch); kw._arr = Arr()
    sem = SemanticSearch.__new__(SemanticSearch); sem._arr = Arr()
    fake = FakeIndex()
    hs.keyword, hs.semantic, hs._index, hs.db_path, hs.device, hs.tie_mode = kw, sem, fake, Path(db), 0, 0
    key = (str(Path(db).resolve()), 0)
    runtime._handles[key] = [fake, 1, {}]
    try:
        sizes = [3, 1, 0, 2, 4]
        batches = [([["a", "zz"]] * n, np.zeros((n, 8), np.float32)) for n in sizes]
        out = list(hs.rrf_search_stream(iter(batches), k=60, limit=4))
        log_full = list(fake.log)
        # ADVICE r01: a consumer that stops early, or a failing submit, must not leave a ticket in flight on the
        # shared handle — the generator drains on exit and a second stream works
        gen = hs.rrf_search_stream(iter(batches), k=60, limit=4)
        first = next(gen)
        assert len(first) == 3 and len(fake.outstanding) == 1            # batch 1 is in flight behind batch 0
        gen.close()
        assert not fake.outstanding and fake.log[-1] == ("drain", 1)
        def boom():
            yield batches[0]
            yield batches[1]
            raise RuntimeError("tokenizer failed")
        with pytest.raises(RuntimeError, match="tokenizer failed"):
            list(hs.rrf_search_stream(boom(), k=60, limit=4))
        assert not fake.outstanding
        again = list(hs.rrf_search_stream(iter(batches[:2]), k=60, limit=4))
        assert [len(o) for o in again] == sizes[:2] and not fake.outstanding
    finally:
        del runtime._handles[key]
    assert [len(o) for o in out] == sizes
    assert fake.max_outstanding == 2 and not fake.outstanding
    assert log_full == ["ids", ("submit", 0), ("submit", 1), ("collect", 0), ("collect", 1),      # empty batch drains
                        ("submit", 2), ("submit", 3), ("collect", 2), ("collect", 3), ("drain", 0)]
    # batch i carries ticket i's ids, three hits per query (count = limit - 1), last rank None-able fields mapped
    assert out[0][0][0] == {"id": 0, "score": 1.0, "bm25_rank": 0, "sem_rank": None}
    assert [h["id"] for h in out[3][1]] == [200, 201, 202] and [h["id"] for h in out[4][0]] == [300, 301, 302]


def test_batch_entry_points_accept_both_token_forms(tmp_path):
    """rrf_search_batch / weighted_search_batch over a fake handle: token lists and the pre-flattened
    (tok_indptr, tokens) pair reach the handle as the same CSR and unpack to one result list PER QUERY (the flat
    form is a 2-tuple: its length is not the number of queries)."""
    from pathlib import Path
    from rag_search_engine_b200 import hybrid_search as hsm, runtime
    from rag_search_engine_b200.keyword_search import KeywordSearch
    from rag_search_engine_b200.semantic_search import SemanticSearch

    class FakeIndex:
        calls = []
        def set_id_tables(self, a, b):
            pass
        def hybrid(self, mode, param, limit, Q, tok_indptr, rows, **kw):
            nq = len(tok_indptr) - 1
            self.calls.append((mode, param, tok_indptr.tolist(), rows.tolist()))
            oid = np.arange(nq * limit, dtype=np.int64).reshape(nq, limit)
            osc = np.tile(1.0 / (1 + np.arange(limit)), (nq, 1))
            a = np.tile(np.arange(limit, dtype=np.float64), (nq, 1))
            b = -np.ones((nq, limit)) if mode == 0 else a / 2
            return oid, osc, a, b, np.arange(nq, dtype=np.int32) % (limit + 1)

    class Arr:
        term_row = {"a": 0, "b": 1, "c": 2}
        doc_ids = np.arange(3, dtype=np.int64)
        movie_ids = np.arange(3, dtype=np.int64)
        emb = np.zeros((4, 8), np.float32)

    db = tmp_path / "y.db"
    db.touch()
    hs = hsm.HybridSearch.__new__(hsm.HybridSearch)
    kw = KeywordSearch.__new__(KeywordSearch); kw._arr = Arr()
    sem = SemanticSearch.__new__(SemanticSearch); sem._arr = Arr()
    fake = FakeIndex()
    hs.keyword, hs.semantic, hs._index, hs.db_path, hs.device, hs.tie_mode = kw, sem, fake, Path(db), 0, 0
    key = (str(Path(db).resolve()), 0)
    runtime._handles[key] = [fake, 1, {}]
    try:
        lists = [["a", "zz"], ["c"], [], ["b", "b", "a"], ["a"]]
        flat = (np.cumsum([0] + [len(l) for l in lists]).astype(np.int32),
                np.array([t for l in lists for t in l], dtype=np.str_))
        Q = np.zeros((len(lists), 8), np.float32)
        r1 = hs.rrf_search_batch(lists, Q, k=60, limit=4)
        r2 = hs.rrf_search_batch(flat, Q, k=60, limit=4)
        w1 = hs.weighted_search_batch(lists, Q, alpha=0.5, limit=4)
        w2 = hs.weighted_search_batch(flat, Q, alpha=0.5, limit=4)
    finally:
        del runtime._handles[key]
    assert fake.calls[0] == fake.calls[1] == (0, 60.0, [0, 2, 3, 3, 6, 7], [0, -1, 2, 1, 1, 0, 0])
    assert fake.calls[2] == fake.calls[3] == (1, 0.5, [0, 2, 3, 3, 6, 7], [0, -1, 2, 1, 1, 0, 0])
    assert r1 == r2 and w1 == w2
    assert [len(x) for x in r1] == [0, 1, 2, 3, 4] == [len(x) for x in w1]
    assert r1[1][0] == {"id": 4, "score": 1.0, "bm25_rank": 0, "sem_rank": None}
    assert w1[4][3] == {"id": 19, "bm25": 3.0, "semantic": 1.5, "score": 0.25}


def test_rebuild_in_place_under_a_live_handle_is_reloaded(tmp_path, monkeypatch):
    """The (database, device) handle registry must not serve a stale index: a database rebuilt in place while an
    object of this process still holds the handle is re-exported and re-uploaded at the next open, every live
    object then reads the NEW arrays, and an unchanged database is not uploaded twice (the other part's build —
    vectors after keyword tables — is not a change of the keyword part)."""
    from rag_search_engine_b200 import _lib, runtime, store
    from rag_search_engine_b200.keyword_search import KeywordSearch
    from rag_search_engine_b200.semantic_search import SemanticSearch
    from rag_search_engine_b200.textutil import whitespace_tokenizer

    class FakeIndex:
        def __init__(self, device=0):
            self.bm25_loads, self.emb_loads, self.closed = [], [], False
        def load_bm25(self, indptr, doc_idx, tf, df, dl, n_movies, avgdl):
            self.bm25_loads.append((int(n_movies), int(len(doc_idx))))
        def load_embeddings(self, emb, valid=None, rowid=None, movie_idx=None):
            self.emb_loads.append(tuple(emb.shape)); self.dim, self.n_rows = emb.shape[1], emb.shape[0]
        def close(self):
            self.closed = True

    class Enc:
        def get_sentence_embedding_dimension(self):
            return 8

    monkeypatch.setattr(_lib, "Index", FakeIndex)
    # a registry of its own: handles adopted by earlier tests in this process (HybridSearch.from_loaded) stay registered
    monkeypatch.setattr(runtime, "_handles", {})
    docs, _, _ = _docs(5, 40)
    rng = np.random.default_rng(0)
    embed = lambda texts: rng.standard_normal((len(texts), 8)).astype(np.float32)      # noqa: E731
    db = store.write_reference_db(tmp_path / "r.db", docs, whitespace_tokenizer, embed=embed)
    kw1 = KeywordSearch(None, db, tokenizer=whitespace_tokenizer)
    sem1 = SemanticSearch(None, db, encoder=Enc())
    fake = kw1._index
    assert sem1._index is fake and len(fake.bm25_loads) == 1 and len(fake.emb_loads) == 1
    kw2 = KeywordSearch(None, db, tokenizer=whitespace_tokenizer)                       # unchanged: no second upload
    assert len(fake.bm25_loads) == 1 and kw2._arr is kw1._arr
    # rebuild in place with more documents while kw1 / kw2 / sem1 are alive
    docs2, _, _ = _docs(6, 55)
    store.write_reference_db(db, docs2, whitespace_tokenizer, embed=embed)
    kw3 = KeywordSearch(None, db, tokenizer=whitespace_tokenizer)
    assert kw3._index is fake and len(fake.bm25_loads) == 2 and fake.bm25_loads[-1][0] == 55
    assert kw1._arr is kw3._arr and kw1._arr.n_movies == 55                            # live objects follow
    ptr, rows = kw1._term_rows((np.array([0, 1], np.int32), np.array([next(iter(kw3._arr.term_row))], np.str_)))
    assert rows.tolist() == [kw3._arr.term_row[next(iter(kw3._arr.term_row))]]          # sorted vocabulary rebuilt
    assert len(fake.emb_loads) == 1                                                     # not reopened yet
    sem2 = SemanticSearch(None, db, encoder=Enc())
    assert len(fake.emb_loads) == 2 and sem1._arr is sem2._arr
    assert sem1._arr.emb.shape[0] == sqlite3.connect(db).execute("SELECT COUNT(*) FROM chunks").fetchone()[0]
    for o in (kw1, kw2, kw3, sem1, sem2):
        assert not fake.closed
        o.close()
    assert fake.closed and not runtime._handles


def test_query_top_k_vec_builds_reference_shaped_hits_from_batched_lookups(tmp_path, monkeypatch):
    """SemanticSearch.query_top_k_vec over a fake handle: the chunk / movie metadata of a whole batch comes from one
    lookup per table, and every hit is the reference's dict (keys, key order, reconstructed chunk text:
    semantic_search.py:321-340)."""
    from rag_search_engine_b200 import _lib, store
    from rag_search_engine_b200.semantic_search import SemanticSearch
    from rag_search_engine_b200.textutil import chunk_text, whitespace_tokenizer

    picks = {0: [7, 0, 33], 1: [], 2: [33, 12]}                  # query -> chunk rows returned by the "device"

    class FakeIndex:
        def __init__(self, device=0):
            pass
        def load_embeddings(self, emb, valid=None, rowid=None, movie_idx=None):
            self.rowid, self.movie_idx, self.dim, self.n_rows = rowid, movie_idx, emb.shape[1], emb.shape[0]
        def knn_movies(self, Q, k, kprime):
            nq = Q.shape[0]
            dist = np.zeros((nq, k), np.float32); row = np.full((nq, k), -1, np.int64)
            mov = np.full((nq, k), -1, np.int32); cnt = np.zeros(nq, np.int32)
            for q, rows in picks.items():
                for j, r in enumerate(rows):
                    dist[q, j], row[q, j], mov[q, j] = 0.125 * (j + 1), self.rowid[r], self.movie_idx[r]
                cnt[q] = len(rows)
            return dist, row, mov, cnt
        def close(self):
            pass

    class Enc:
        def get_sentence_embedding_dimension(self):
            return 8

    monkeypatch.setattr(_lib, "Index", FakeIndex)
    docs, _, _ = _docs(9, 30)
    rng = np.random.default_rng(1)
    db = store.write_reference_db(tmp_path / "q.db", docs, whitespace_tokenizer,
                                  embed=lambda t: rng.standard_normal((len(t), 8)).astype(np.float32))
    ss = SemanticSearch(None, db, encoder=Enc())
    try:
        out = ss.query_top_k_vec(np.zeros((3, 8), np.float32), k=4)
        conn = sqlite3.connect(db)
        assert [len(h) for h in out] == [3, 0, 2]
        for q, rows in picks.items():
            for j, r in enumerate(rows):
                mid, ci, mcs, ov = conn.execute("SELECT movie_id, chunk_index, max_chunk_size, overlap FROM chunks "
                                                "WHERE id = ?", (r,)).fetchone()
                title, desc = conn.execute("SELECT title, description FROM movies WHERE id = ?", (mid,)).fetchone()
                hit = out[q][j]
                assert list(hit) == ["chunk_id", "distance", "chunk", "movie_id", "title", "description"]
                assert hit == {"chunk_id": r, "distance": 0.125 * (j + 1), "chunk": chunk_text(title, desc, ci, mcs, ov),
                               "movie_id": mid, "title": title, "description": desc}
        conn.close()
    finally:
        ss.close()


def test_term_rows_list_form_and_flat_array_form_agree():
    """KeywordSearch._term_rows: dict lookups over token lists and one searchsorted over a flat numpy array of
    tokens give the same CSR rows (query order, duplicates kept, -1 = unknown term: keyword_search.py:205-210)."""
    from types import SimpleNamespace
    from rag_search_engine_b200.keyword_search import KeywordSearch
    rng = random.Random(5)
    vocab = [f"w{i}" for i in range(5000)]
    rng.shuffle(vocab)
    kw = KeywordSearch.__new__(KeywordSearch)
    kw._arr = SimpleNamespace(term_row={t: i for i, t in enumerate(vocab)})
    lists = [[rng.choice(vocab + ["<oov>", "zzz"]) for _ in range(rng.randint(0, 7))] for _ in range(300)]
    lists[5] = lists[5] + lists[5][:1] * 2                      # duplicates stay
    ptr, rows = kw._term_rows(lists)
    want = [kw._arr.term_row.get(t, -1) for l in lists for t in l]
    assert ptr.tolist() == np.cumsum([0] + [len(l) for l in lists]).tolist() and rows.tolist() == want
    flat = np.array([t for l in lists for t in l], dtype=np.str_)
    ptr2, rows2 = kw._term_rows((ptr, flat))
    assert ptr2.tolist() == ptr.tolist() and rows2.tolist() == want
    ptr3, rows3 = kw._term_rows([[], []])
    assert ptr3.tolist() == [0, 0, 0] and len(rows3) == 1


def test_gpu_fuzz_generators_run_without_a_gpu():
    """scripts/gpu_fuzz.py draws its cases on the host; a stub handle stops each case where the GPU would take over,
    so the generators (and the script's imports) are exercised by the CPU suite as well."""
    import importlib.util
    from pathlib import Path
    import oracle
    spec = importlib.util.spec_from_file_location("gpu_fuzz", Path(__file__).resolve().parents[1] / "scripts" / "gpu_fuzz.py")
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)

    class Reached(Exception):
        pass

    class StubLib:
        class Index:
            def __init__(self, device):
                raise Reached()

    reached = 0
    for seed in range(4):
        for kind in ("knn", "bm25", "hybrid"):
            try:
                mod.KINDS[kind](seed, StubLib, oracle)
            except Reached:
                reached += 1
    assert reached == 12


def test_probe_rank_is_the_binomial_tail_quantile():
    """DESIGN §5: the K4 probe takes the j-th best value of a 1-in-`stride` row sample as its bound, j = the smallest
    rank whose binomial tail P(Bin(K', 1/stride) >= j) is at most 1e-7 (the bound is verified on the device anyway;
    the tail is only how often a second filter pass is paid)."""
    from scipy.stats import binom
    from rag_search_engine_b200 import _lib
    L = _lib.load_library()
    for stride in (4, 8, 16, 32, 64, 128):
        for kprime in (1, 2, 5, 10, 50, 100, 256):
            j = L.rse_tc_probe_rank(kprime, stride)
            assert 1 <= j <= kprime
            if j < kprime:
                assert binom.sf(j - 1, kprime, 1.0 / stride) <= 1e-7 * (1 + 1e-6)
                assert j == 1 or binom.sf(j - 2, kprime, 1.0 / stride) > 1e-7 * (1 - 1e-6)
            else:
                assert kprime == 1 or binom.sf(kprime - 2, kprime, 1.0 / stride) > 1e-7 * (1 - 1e-6)
    assert L.rse_tc_probe_rank(100, 64) == 12 and L.rse_tc_probe_rank(100, 32) == 16
