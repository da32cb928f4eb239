"""CPU: the oracle restatements against the golden vectors generated from the reference's own
code (oracle/make_golden.py) and against the reference imported live when it is present."""
import json
from pathlib import Path

import numpy as np
import pytest

import oracle
from oracle import pyref, ref_import

GOLDEN = Path(__file__).parent / "golden"
from helpers.corpus import build_postings, to_csr


def load_bm25_cases():
    return json.loads((GOLDEN / "bm25_ref.json").read_text())["cases"]


def test_pyref_bm25_matches_reference_golden():
    for case in load_bm25_cases():
        postings, doclen = build_postings(case["docs"])
        assert len(postings) == case["n_terms"]
        assert sum(len(v) for v in postings.values()) == case["n_postings"]
        assert (sum(doclen.values()) / len(doclen)).hex() == case["avgdl"]
        for r in case["results"]:
            toks = r["query"].lower().split()
            got = pyref.bm25_search(postings, doclen, len(doclen), toks, k=r["k"], k1=r["k1"], b=r["b"])
            assert [[d, float(s).hex()] for d, s in got] == r["hits"], r["query"]


def test_c_oracle_bm25_matches_reference_golden():
    for case in load_bm25_cases():
        postings, doclen = build_postings(case["docs"])
        csr = to_csr(postings, doclen)
        by = {}
        for r in case["results"]:
            by.setdefault((r["k"], r["k1"], r["b"]), []).append(r)
        for (k, k1, b), rs in by.items():
            tok_indptr, terms = [0], []
            for r in rs:
                terms += [csr["row"].get(t, -1) for t in r["query"].lower().split()]
                tok_indptr.append(len(terms))
            sc, dc, cnt = oracle.bm25_batch(csr["indptr"], csr["doc"], csr["tf"], csr["df"], csr["dl"], len(csr["dl"]),
                                            csr["avgdl"], np.array(tok_indptr, np.int32),
                                            np.array(terms or [0], np.int32), k, k1, b)
            for i, r in enumerate(rs):
                got = [[int(csr["doc_ids"][dc[i, j]]), float(sc[i, j]).hex()] for j in range(cnt[i])]
                assert got == r["hits"], r["query"]


def test_pyref_fusion_matches_reference_golden():
    cases = json.loads((GOLDEN / "fusion_ref.json").read_text())["cases"]
    assert len(cases) > 100
    for c in cases:
        bm = [(i, float.fromhex(s)) for i, s in c["bm25"]]
        sem = [(i, float.fromhex(d)) for i, d in c["sem"]]
        w = pyref.weighted_fuse(bm, sem, float.fromhex(c["alpha"]), c["limit"])
        assert [[x["id"], x["bm25"].hex(), x["semantic"].hex(), x["score"].hex()] for x in w] == c["weighted"]
        r = pyref.rrf_fuse(bm, sem, c["k"], c["limit"])
        assert [[x["id"], float(x["score"]).hex(), x["bm25_rank"], x["sem_rank"]] for x in r] == c["rrf"]


def test_survey_known_answers():
    # SURVEY App. B fusion KAT (reference code + dummy retrievers)
    bm = [(912345, 9.5), (17, 7.25), (400001, 7.0), (8, 3.5), (33, 1.125)]
    sem = [(5, 0.20440000295639038), (700000, 0.23229999840259552), (17, 0.2764), (31, 0.5), (8, 0.75)]
    r = pyref.rrf_fuse(bm, sem, 60, 5)
    assert [x["id"] for x in r] == [17, 8, 5, 912345, 700000]
    assert r[0]["score"] == 0.03252247488101534 and r[2]["score"] == r[3]["score"] == 0.016676660770145613
    w = pyref.weighted_fuse(bm, sem, 0.5, 5)
    assert [x["id"] for x in w] == [17, 5, 912345, 700000, 400001]
    assert w[0]["score"] == 0.7996892394507322
    assert pyref.set_union_order([9], [2]) == [9, 2]
    assert pyref.set_union_order([16, 3], [8, 1]) == [16, 8, 3, 1]
    # BM25 tie KAT: first-seen order, not id order
    postings = {"a": [(50, 1), (70, 1)], "b": [(10, 1), (70, 1)]}
    doclen = {10: 3, 50: 3, 70: 3}
    got = pyref.bm25_search(postings, doclen, 3, ["a", "b"], k=3)
    assert [d for d, _ in got][0] == 70 and [d for d, _ in got][1:] == [50, 10]


def test_reference_utils_unit_tests_hold_for_pyref():
    # rag_search_engine/tests/test_utils.py:112-136
    out = pyref.min_max_norm([10.0, 20.0, 30.0])
    assert out[0] == 0.0 and out[-1] == 1.0 and all(0.0 <= x <= 1.0 for x in out)
    assert pyref.min_max_norm([5.0, 5.0, 5.0]) == [1.0, 1.0, 1.0]
    assert pyref.rrf_score(0) > pyref.rrf_score(1) > pyref.rrf_score(10)
    # tests/test_hybrid_search.py:94-124 degenerate orderings
    bm = [(1, 3.0), (3, 2.0), (2, 1.0)]
    assert [x["id"] for x in pyref.weighted_fuse(bm, [], 0.8, 10)] == [1, 3, 2]
    assert [x["id"] for x in pyref.rrf_fuse(bm, [], 60, 3)] == [1, 3, 2]
    assert [x["id"] for x in pyref.rrf_fuse([], [(2, 0.2), (4, 0.4)], 60, 3)][:2] == [2, 4]


def live_fixture():
    return json.loads((GOLDEN / "live_ref.json").read_text())


@pytest.mark.skipif(not ref_import.available(), reason="reference checkout not present (GPU box)")
def test_pyref_matches_live_reference_bm25(tmp_path):
    ref_kw, _, _ = ref_import.load()
    from oracle.make_golden import encode_hits, live_bm25_inputs, reference_bm25
    docs, queries = live_bm25_inputs()
    refs = reference_bm25(ref_kw, docs, queries, 7, tmp_path)
    postings, doclen = build_postings(docs)
    for q, ref in zip(queries, refs):
        got = pyref.bm25_search(postings, doclen, len(doclen), q.lower().split(), k=7)
        assert got == ref
    assert [encode_hits(h) for h in refs] == live_fixture()["bm25"]["hits"]      # the pinned answers are the reference's


def test_pyref_bm25_matches_pinned_live_answers():
    """test_pyref_matches_live_reference_bm25 against its pinned answers (tests/golden/live_ref.json)."""
    from oracle.make_golden import encode_hits, live_bm25_inputs
    docs, queries = live_bm25_inputs()
    fx = live_fixture()["bm25"]
    postings, doclen = build_postings(docs)
    got = [encode_hits(pyref.bm25_search(postings, doclen, len(doclen), q.lower().split(), k=fx["k"])) for q in queries]
    assert got == fx["hits"]


@pytest.mark.skipif(not ref_import.available(), reason="reference checkout not present (GPU box)")
def test_pyref_matches_live_reference_fusion(tmp_path):
    """1500 more random fusion cases than the committed fixture holds, straight against the reference's own
    HybridSearch through its dummy-retriever seam (tests/test_hybrid_search.py:73-76): empty sides, overlapping
    hit lists, huge and negative ids (CPython set order), exact score / distance ties, int and float k."""
    _, ref_hs, _ = ref_import.load()
    from oracle.make_golden import encode_fusion, live_fusion_inputs, reference_fusion
    cases = live_fusion_inputs()
    refs = reference_fusion(ref_hs, cases, tmp_path)
    for case, ((bm, sem, alpha, k, limit), (w, r)) in enumerate(zip(cases, refs)):
        pw = pyref.weighted_fuse(bm, sem, alpha, limit)
        pr = pyref.rrf_fuse(bm, sem, k, limit)
        assert [(x["id"], x["bm25"], x["semantic"], x["score"]) for x in w] == \
               [(x["id"], x["bm25"], x["semantic"], x["score"]) for x in pw], case
        assert [(x["id"], x["score"], x["bm25_rank"], x["sem_rank"]) for x in r] == \
               [(x["id"], x["score"], x["bm25_rank"], x["sem_rank"]) for x in pr], case
    fx = live_fixture()["fusion"]
    assert [list(encode_fusion(w, r)) for w, r in refs[::fx["stride"]]] == fx["cases"]


def test_pyref_fusion_matches_pinned_live_answers():
    """test_pyref_matches_live_reference_fusion against its pinned answers: every stride-th of its cases."""
    from oracle.make_golden import encode_fusion, live_fusion_inputs
    fx = live_fixture()["fusion"]
    cases = live_fusion_inputs()[::fx["stride"]]
    assert len(cases) == len(fx["cases"]) == 300
    for i, ((bm, sem, alpha, k, limit), want) in enumerate(zip(cases, fx["cases"])):
        got = encode_fusion(pyref.weighted_fuse(bm, sem, alpha, limit), pyref.rrf_fuse(bm, sem, k, limit))
        assert list(got) == want, i


def test_vec0_literal_scan_equals_key_order():
    rng = np.random.default_rng(5)
    emb = rng.standard_normal((3500, 48)).astype(np.float32)
    emb /= np.linalg.norm(emb, axis=1, keepdims=True)
    for dst, src in [(100, 7), (3000, 7), (1023, 7), (1024, 7), (2047, 7), (2048, 9), (5, 9)]:
        emb[dst] = emb[src]
    for qi, k in [(7, 10), (9, 3), (7, 1), (11, 1100), (12, 4000)]:
        q = emb[qi] + 0.05 * rng.standard_normal(48).astype(np.float32)
        d1, r1 = oracle.vec0_knn(emb, q, k, literal=True)
        d2, r2 = oracle.vec0_knn(emb, q, k, literal=False)
        assert (r1 == r2).all() and (d1 == d2).all()
        assert len(r1) == min(k, len(emb))
    # exact duplicates of the query row: highest slot of the earliest block first
    d, r = oracle.vec0_knn(emb, emb[7], 5)
    assert r.tolist() == [1023, 100, 7, 2047, 1024]   # block 0 slots desc, then block 1 slots desc


def test_vec0_knn_known_answers_fixture():
    """tests/golden/knn_kat.json (SURVEY §8c (3)): answers of the pure-Python second restatement
    (oracle/pyref.py::vec0_knn) — duplicates on both sides of block boundaries, mass ties on a coarse grid,
    deleted slots, k above the block size — against oracle.c, rows / emit order / distance bits, through both of
    its forms (literal block scan and closed-form key order)."""
    from oracle.make_golden import knn_kat_inputs
    fx = json.loads((GOLDEN / "knn_kat.json").read_text())
    n_checked = 0
    for case in fx["cases"]:
        emb, valid, Q = knn_kat_inputs(case)
        pos = np.nonzero(valid)[0].astype(np.int64)
        live = np.ascontiguousarray(emb[valid])
        for a in case["answers"]:
            want_d = np.array([float.fromhex(h) for h in a["dist"]], np.float32)
            for literal in (True, False):
                d, r = oracle.vec0_knn(live, Q[a["q"]], a["k"], pos=pos, literal=literal)
                assert pos[r].tolist() == a["rows"], (case["seed"], a["k"], a["q"], literal)
                assert d.view(np.uint32).tolist() == want_d.view(np.uint32).tolist()
            n_checked += 1
        # the fixture really holds the hard cases: a duplicate pair split by a block boundary, emitted block-first
        first = next(a for a in case["answers"] if a["q"] == 0 and a["k"] >= 3)
        assert len(set(first["dist"][:2])) == 1 and first["rows"][0] // 1024 <= first["rows"][1] // 1024
    assert n_checked == 27


def test_pyref_vec0_knn_still_generates_the_fixture():
    """The committed answers are what oracle/pyref.py::vec0_knn computes today (one small slice re-derived here:
    the fixture cannot drift from the script that made it)."""
    from oracle.make_golden import knn_kat_inputs
    fx = json.loads((GOLDEN / "knn_kat.json").read_text())
    case = fx["cases"][1]
    emb, valid, Q = knn_kat_inputs(case)
    for a in [x for x in case["answers"] if x["k"] <= 64][:4]:
        res = pyref.vec0_knn(emb, Q[a["q"]], a["k"], valid=valid)
        assert [r for r, _ in res] == a["rows"] and [float(d).hex() for _, d in res] == a["dist"]


def test_vec0_distance_is_sequential_fp32():
    rng = np.random.default_rng(6)
    a = rng.standard_normal(384).astype(np.float32)
    b = rng.standard_normal(384).astype(np.float32)
    dot = np.float32(0); am = np.float32(0); bm = np.float32(0)
    for i in range(384):
        dot = np.float32(dot + np.float32(a[i] * b[i]))
        am = np.float32(am + np.float32(a[i] * a[i]))
        bm = np.float32(bm + np.float32(b[i] * b[i]))
    want = np.float32(1.0 - float(dot) / (np.sqrt(float(am)) * np.sqrt(float(bm))))
    assert oracle.cosine_distance(a, b) == float(want)


def test_aggregate_matches_pyref():
    rng = np.random.default_rng(8)
    for _ in range(50):
        n = int(rng.integers(0, 60))
        dist = np.sort(rng.choice(np.arange(1, 20, dtype=np.float32) / 16, size=n))
        movie = rng.integers(0, 12, size=n)
        k = int(rng.integers(1, 12))
        sel = oracle.aggregate_movies(dist, movie, k)
        want = pyref.aggregate_movies([(i, float(dist[i]), int(movie[i])) for i in range(n)], k)
        assert [int(s) for s in sel] == [w[0] for w in want]
