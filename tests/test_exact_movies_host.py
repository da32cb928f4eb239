"""CPU tests of exact movie-level search (SemanticSearch(..., exact_movies=True), rse_knn_movies_exact): the Python
argument checks and the empty corpus over a fake handle, and the numpy restatement of the contract
(helpers/exact_movies_ref.py) held to the reference's aggregation wherever the shortlist covers k movies — the
prefix property of DESIGN §11."""
import sqlite3

import numpy as np
import pytest

import oracle
from helpers.exact_movies_ref import exact_movies, keys


def _docs(seed=3, n=60):
    from oracle.make_golden import sentence_corpus
    return sentence_corpus(seed, n)


def _fake_search(tmp_path, monkeypatch, with_embeddings=True):
    from rag_search_engine_b200 import _lib, store
    from rag_search_engine_b200.semantic_search import SemanticSearch
    from rag_search_engine_b200.textutil import whitespace_tokenizer

    calls = []

    class FakeIndex:
        def __init__(self, device=0):
            pass

        def load_embeddings(self, emb, valid=None, rowid=None, movie_idx=None):
            self.rowid, self.movie_idx, self.dim, self.n_rows = rowid, movie_idx, emb.shape[1], emb.shape[0]

        def knn_movies(self, Q, k, kprime):
            calls.append(("knn_movies", Q.shape[0], k, kprime))
            nq = Q.shape[0]
            return (np.zeros((nq, k), np.float32), np.full((nq, k), -1, np.int64), np.full((nq, k), -1, np.int32),
                    np.zeros(nq, np.int32))

        def knn_movies_exact(self, Q, k):
            calls.append(("knn_movies_exact", Q.shape[0], k))
            nq = Q.shape[0]
            dist = np.zeros((nq, k), np.float32); row = np.full((nq, k), -1, np.int64)
            mov = np.full((nq, k), -1, np.int32); cnt = np.zeros(nq, np.int32)
            rows = [0, 7]
            for j, r in enumerate(rows):
                dist[0, j], row[0, j], mov[0, j] = 0.25 * (j + 1), self.rowid[r], self.movie_idx[r]
            cnt[0] = len(rows)
            return dist, row, mov, cnt, nq

        def close(self):
            pass

    class Enc:
        def get_sentence_embedding_dimension(self):
            return 8

        def encode(self, texts):
            return np.ones((len(texts), 8), np.float32)

    monkeypatch.setattr(_lib, "Index", FakeIndex)
    docs, _, _ = _docs(9, 30)
    rng = np.random.default_rng(1)
    embed = (lambda t: rng.standard_normal((len(t), 8)).astype(np.float32)) if with_embeddings else None
    db = store.write_reference_db(tmp_path / "q.db", docs, whitespace_tokenizer, embed=embed)
    return SemanticSearch(None, db, encoder=Enc()), calls, db


def test_exact_movies_argument_checks_and_dispatch(tmp_path, monkeypatch):
    ss, calls, db = _fake_search(tmp_path, monkeypatch)
    try:
        for bad in (0, -1, 4097):
            with pytest.raises(ValueError):
                ss.query_top_k_vec(np.zeros((1, 8), np.float32), k=bad, exact_movies=True)
            with pytest.raises(ValueError):
                ss.query_top_k("anything", k=bad, exact_movies=True)
        assert calls == []
        out = ss.query_top_k_vec(np.zeros((2, 8), np.float32), k=4096, knn_multiplier=77, exact_movies=True)
        assert calls == [("knn_movies_exact", 2, 4096)]                 # knn_multiplier plays no part
        assert [len(h) for h in out] == [2, 0]
        conn = sqlite3.connect(db)
        for j, r in enumerate([0, 7]):
            mid = conn.execute("SELECT movie_id FROM chunks WHERE id = ?", (r,)).fetchone()[0]
            hit = out[0][j]
            assert list(hit) == ["chunk_id", "distance", "chunk", "movie_id", "title", "description"]
            assert hit["chunk_id"] == r and hit["movie_id"] == mid and hit["distance"] == 0.25 * (j + 1)
        conn.close()
        one = ss.query_top_k("anything", k=3, exact_movies=True)
        assert calls[-1] == ("knn_movies_exact", 1, 3) and len(one) == 2
        # the default path is untouched: K' = k * knn_multiplier
        ss.query_top_k_vec(np.zeros((1, 8), np.float32), k=3, knn_multiplier=4)
        assert calls[-1] == ("knn_movies", 1, 3, 12)
    finally:
        ss.close()


def test_exact_movies_on_an_empty_corpus_is_an_empty_list_per_query(tmp_path, monkeypatch):
    ss, calls, _ = _fake_search(tmp_path, monkeypatch, with_embeddings=False)
    try:
        assert ss.query_top_k_vec(np.zeros((3, 8), np.float32), k=5, exact_movies=True) == [[], [], []]
        assert ss.query_top_k_vec(np.zeros((2, 8), np.float32), k=4096, exact_movies=True) == [[], []]
        assert calls == []
    finally:
        ss.close()


def test_key_order_is_the_vec0_emit_order():
    d = np.array([0.5, 0.25, 0.25, 0.25, -0.0, 0.0, -1e-30], np.float32)
    pos = np.array([0, 5, 1024, 7, 3, 2, 9])
    order = np.argsort(keys(d, pos)).tolist()
    # distance ascending (-1e-30 < -0.0 < +0.0); among the 0.25 ties block ascending, then slot descending
    assert order == [6, 4, 5, 3, 1, 2, 0]


def _corpus(rng, n_movies, lo, hi, dim=64, spread=0.3):
    per = rng.integers(lo, hi, n_movies)
    movie_of = np.repeat(np.arange(n_movies, dtype=np.int32), per)
    centers = rng.standard_normal((n_movies, dim)).astype(np.float32)
    emb = centers[movie_of] + spread * rng.standard_normal((len(movie_of), dim)).astype(np.float32)
    emb /= np.linalg.norm(emb, axis=1, keepdims=True)
    return emb.astype(np.float32), movie_of, centers


@pytest.mark.parametrize("use_fma", [False, True])
def test_exact_oracle_agrees_with_the_reference_aggregation_where_the_shortlist_covers_k(use_fma):
    rng = np.random.default_rng(17 + use_fma)
    emb, movie_of, centers = _corpus(rng, 300, 2, 12)
    emb[100] = emb[3]                                   # exact ties across movies
    Q = np.concatenate([centers[:6], rng.standard_normal((6, emb.shape[1]))]).astype(np.float32)
    full = covered = 0
    for q in Q:
        d = oracle.all_distances(emb, q, use_fma)
        for k, kp in [(1, 1), (5, 10), (10, 20), (10, 100), (40, 400)]:
            ed, erow, emov = exact_movies(emb, q, movie_of, k, use_fma=use_fma, dist=d)
            assert len(erow) == k and len(set(emov.tolist())) == k
            od, orow = oracle.vec0_knn(emb, q, kp, use_fma=use_fma, literal=False)
            sel = oracle.aggregate_movies(od, movie_of[orow], k)
            ref_rows = orow[sel]
            if len(sel) == k:                           # the shortlist covers k movies: identical
                covered += 1
                assert erow.tolist() == ref_rows.tolist()
                assert ed.view(np.uint32).tolist() == od[sel].view(np.uint32).tolist()
            else:                                       # fewer: the reference's list is a prefix
                full += 1
                assert erow[:len(sel)].tolist() == ref_rows.tolist()
    assert covered > 0 and full > 0


def test_exact_oracle_skips_holes_and_orphans_and_caps_at_the_movie_count():
    rng = np.random.default_rng(5)
    emb, movie_of, centers = _corpus(rng, 40, 1, 6, dim=16)
    valid = rng.random(len(movie_of)) > 0.2
    movie_of = movie_of.copy()
    movie_of[rng.random(len(movie_of)) < 0.1] = -1
    q = centers[0]
    d = oracle.all_distances(emb, q)
    _, rows, mov = exact_movies(emb, q, movie_of, 1000, valid=valid, dist=d)
    live = valid & (movie_of >= 0)
    assert sorted(mov.tolist()) == sorted(set(movie_of[live].tolist()))
    assert valid[rows].all() and (movie_of[rows] >= 0).all()
    for r, m in zip(rows, mov):                         # each is its movie's smallest key among live rows
        cand = np.nonzero(live & (movie_of == m))[0]
        assert r == cand[np.argmin(keys(d[cand], cand))]
