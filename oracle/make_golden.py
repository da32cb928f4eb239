"""Generate tests/golden/*.json from the UNMODIFIED reference code.

Run from the repository root with a checkout of the reference under oracle/_ref (or
RSE_REFERENCE_ROOT pointing at one; see oracle/ref_import.py):
    python -m oracle.make_golden
Without the reference, ``--knn-only`` writes knn_kat.json and live_ref.json (the latter then from this
project's restatements).

What it pins (SURVEY §8c):
  * bm25_ref.json    — reference ``KeywordSearch.search`` (keyword_search.py:180-267) on a
                       synthetic corpus indexed by the reference's own ``_rebuild_index``
                       (:102-177), ``preprocess`` frozen to a whitespace tokenizer.
  * fusion_ref.json  — reference ``HybridSearch.weighted_search`` / ``rrf_search``
                       (hybrid_search.py:91-180,183-272,379) driven through the reference's own
                       plugin seam (dummy retrievers monkeypatched on the module, exactly as
                       tests/test_hybrid_search.py:73-76 does), including structural ties.
  * knn_kat.json     — vec0 KNN known answers (duplicates across block boundaries, mass ties, holes)
                       from the pure-Python second restatement ``pyref.vec0_knn`` (sqlite-vec is not
                       installable here: this fixture pins oracle.c against pyref, not against sqlite-vec).
  * live_ref.json    — what the four live comparisons with the reference compare against (see
                       live_golden; its ``source`` field says whether the reference or this
                       project's restatements produced it).
Floats are stored with float.hex() so the fixtures are bit-exact.
"""
from __future__ import annotations

import json
import random
import tempfile
from pathlib import Path

from oracle import ref_import

GOLDEN = Path(__file__).resolve().parents[1] / "tests" / "golden"


# ----------------------------------------------------------------------------- corpora
def make_corpus(seed: int, n_docs: int, vocab: int, dup_frac: float = 0.08):
    rnd = random.Random(seed)
    words = [f"w{i}" for i in range(vocab)]
    weights = [1.0 / (i + 1) ** 1.07 for i in range(vocab)]
    ids = sorted(rnd.sample(range(1, n_docs * 9), n_docs))
    docs = []
    for i, did in enumerate(ids):
        tl = rnd.randint(1, 4)
        bl = max(0, int(rnd.gauss(30, 14)))
        title = " ".join(rnd.choices(words, weights, k=tl))
        body = " ".join(rnd.choices(words, weights, k=bl))
        docs.append({"id": did, "title": title, "description": body})
    # exact duplicates (same title+description under another id) → exact BM25 score ties
    for _ in range(int(n_docs * dup_frac)):
        a, b = rnd.sample(range(n_docs), 2)
        docs[b]["title"] = docs[a]["title"]
        docs[b]["description"] = docs[a]["description"]
    return docs, words, weights


def make_queries(seed: int, words, weights, n: int):
    rnd = random.Random(seed)
    qs = []
    for i in range(n):
        nt = rnd.randint(1, 6)
        toks = rnd.choices(words, weights, k=nt)
        r = rnd.random()
        if r < 0.15:
            toks.insert(rnd.randrange(len(toks) + 1), "zzz_oov")       # unknown term
        elif r < 0.30:
            toks.append(toks[0])                                       # duplicate token
        elif r < 0.35:
            toks = [words[-1 - rnd.randrange(20)]]                     # rare single term
        qs.append(" ".join(toks))
    qs += ["", "   ", "zzz_oov qqq_oov", "[TITLE_END]", words[0], f"{words[0]} {words[0]} {words[0]}"]
    return qs


def bm25_golden():
    ref_kw, _, _ = ref_import.load()
    out = {"cases": []}
    for seed, n_docs, vocab, nq, k in [(11, 240, 150, 40, 10), (12, 60, 12, 25, 5), (13, 400, 600, 30, 25)]:
        docs, words, weights = make_corpus(seed, n_docs, vocab)
        queries = make_queries(seed + 100, words, weights, nq)
        with tempfile.TemporaryDirectory() as td:
            p = Path(td) / "movies.json"
            p.write_text(json.dumps({"movies": docs}), encoding="utf-8")
            ks = ref_kw.KeywordSearch.build_from_docs(docs_path=p, db_path=Path(td) / "kw.db", force=True)
            try:
                results = []
                for q in queries:
                    for (kk, k1, b) in [(k, 1.5, 0.75), (3, 1.2, 0.5)]:
                        res = ks.search(q, k=kk, k1=k1, b=b)
                        results.append({"query": q, "k": kk, "k1": k1, "b": b,
                                        "hits": [[r["id"], float(r["score"]).hex()] for r in res]})
                cur = ks.conn.cursor()
                cur.execute("SELECT COUNT(*) FROM terms"); (nterms,) = cur.fetchone()
                cur.execute("SELECT COUNT(*) FROM postings"); (npost,) = cur.fetchone()
                cur.execute("SELECT AVG(length) FROM doclen"); (avgdl,) = cur.fetchone()
            finally:
                ks.close()
        out["cases"].append({"seed": seed, "docs": docs, "results": results,
                             "n_terms": nterms, "n_postings": npost, "avgdl": float(avgdl).hex()})
    (GOLDEN / "bm25_ref.json").write_text(json.dumps(out, separators=(",", ":")))
    print("bm25_ref.json:", sum(len(c["results"]) for c in out["cases"]), "searches")


# ----------------------------------------------------------------------------- fusion
def fusion_golden():
    _, ref_hs, _ = ref_import.load()
    rnd = random.Random(7)

    class KW:
        hits = []
        def __init__(self, *a, **k): pass
        def search(self, query, k=10, k1=1.5, b=0.75): return [dict(h) for h in KW.hits[:k]]
        def close(self): pass

    class SEM:
        hits = []
        def __init__(self, *a, **k): pass
        def query_top_k(self, query_text, k=10, knn_multiplier=10): return [dict(h) for h in SEM.hits[:k]]
        def close(self): pass

    ref_hs.KeywordSearch = KW
    ref_hs.SemanticSearch = SEM
    cases = []

    def run(bm, sem, limit, alpha, k):
        KW.hits = [{"id": i, "title": f"t{i}", "description": f"d{i}", "score": s} for i, s in bm]
        SEM.hits = [{"chunk_id": 0, "distance": d, "chunk": "", "movie_id": i, "title": f"t{i}",
                     "description": f"d{i}"} for i, d in sem]
        with tempfile.TemporaryDirectory() as td:
            hs = ref_hs.HybridSearch(docs_path=None, db_path=Path(td) / "h.db")
            w = hs.weighted_search("q", alpha=alpha, limit=limit)
            r = hs.rrf_search("q", k=k, limit=limit)
        cases.append({
            "bm25": [[i, float(s).hex()] for i, s in bm[:limit]],
            "sem": [[i, float(d).hex()] for i, d in sem[:limit]],
            "limit": limit, "alpha": float(alpha).hex(), "k": k,
            "weighted": [[x["id"], float(x["bm25"]).hex(), float(x["semantic"]).hex(),
                          float(x["score"]).hex()] for x in w],
            "rrf": [[x["id"], float(x["score"]).hex(), x["bm25_rank"], x["sem_rank"]] for x in r],
        })

    import numpy as np
    # SURVEY App. B known-answer case
    run([(912345, 9.5), (17, 7.25), (400001, 7.0), (8, 3.5), (33, 1.125)],
        [(5, 0.20440000295639038), (700000, 0.23229999840259552), (17, 0.2764), (31, 0.5), (8, 0.75)],
        5, 0.5, 60)
    # reference unit-test shapes (tests/test_hybrid_search.py)
    run([(1, 3.0), (3, 2.0), (2, 1.0)], [(2, 0.2), (4, 0.4)], 10, 0.7, 60)
    run([(1, 3.0), (3, 2.0), (2, 1.0)], [], 10, 0.8, 60)
    run([], [(2, 0.2), (4, 0.4)], 3, 0.5, 60)
    run([], [], 5, 0.5, 60)
    run([(7, 2.5)], [(7, 0.3)], 5, 0.5, 60)            # single element → min_max all-equal → 1.0
    run([(7, 2.5), (9, 2.5)], [(11, 0.3), (12, 0.3)], 5, 0.25, 60)   # all-equal lists
    for case in range(160):
        limit = rnd.choice([1, 2, 3, 5, 10, 10, 10, 20, 40, 64])
        id_space = rnd.choice([max(30, 4 * limit), 200, 10**6, 10**9, 2**40])
        nb = rnd.randint(0, limit)
        ns = rnd.randint(0, limit)
        overlap = rnd.random()
        bids = rnd.sample(range(1, id_space), nb)
        sids = []
        pool = list(bids)
        while len(sids) < ns:
            if pool and rnd.random() < overlap:
                sids.append(pool.pop(rnd.randrange(len(pool))))
            else:
                c = rnd.randrange(1, id_space)
                if c not in sids and c not in bids:
                    sids.append(c)
        bs = sorted((rnd.choice([rnd.uniform(0.5, 20.0), float(rnd.randint(1, 4))]) for _ in range(nb)),
                    reverse=True)
        ds = sorted(float(np.float32(rnd.choice([rnd.uniform(0.05, 1.2), rnd.randint(1, 4) / 8.0])))
                    for _ in range(ns))
        alpha = rnd.choice([0.0, 0.2, 0.5, 0.5, 0.7, 1.0, rnd.random()])
        k = rnd.choice([60, 60, 60.0, 1, 10, 0.5])
        run(list(zip(bids, bs)), list(zip(sids, ds)), limit, alpha, k)
    (GOLDEN / "fusion_ref.json").write_text(json.dumps({"cases": cases}, separators=(",", ":")))
    print("fusion_ref.json:", len(cases), "cases")


# ----------------------------------------------------------------------------- vec0 KNN known answers
def knn_kat_inputs(case: dict):
    """(emb f32[n, dim], valid bool[n], queries f32[nq, dim]) of a fixture case, rebuilt from its seed — the fixture
    stores the seed and the ANSWERS, not the matrix."""
    import numpy as np
    rng = np.random.default_rng(case["seed"])
    n, dim = case["n"], case["dim"]
    emb = rng.standard_normal((n, dim)).astype(np.float32)
    emb *= rng.uniform(0.5, 2.0, (n, 1)).astype(np.float32)           # norms are recomputed per pair
    emb = (np.round(emb * 4) / 4).astype(np.float32) if case["coarse"] else emb   # coarse grid: exact distance ties
    for a, b in case["dups"]:
        emb[b] = emb[a]
    valid = np.ones(n, bool)
    valid[case["holes"]] = False
    Q = rng.standard_normal((case["nq"], dim)).astype(np.float32)
    for j, r in enumerate(case["query_rows"]):
        Q[j] = emb[r] * np.float32(1.5)
    return emb, valid, Q


def knn_golden():
    """tests/golden/knn_kat.json — SURVEY §8c (3): vec0 KNN known answers with duplicate rows on both sides of
    1024-row block boundaries, mass ties (coarse grid), deleted slots and k above a block's size, computed by the
    pure-Python restatement (pyref.vec0_knn); tests/test_oracle_golden.py checks oracle.c — the checker of every GPU
    parity test — against them."""
    from oracle import pyref
    cases = []
    specs = [dict(seed=21, n=2100, dim=8, coarse=False, nq=5, query_rows=[1023, 5], holes=[3, 1024, 2099],
                  dups=[[1023, 1024], [1023, 2047], [5, 900], [5, 2050], [2047, 2048]], ks=[1, 10, 100]),
             dict(seed=22, n=1500, dim=4, coarse=True, nq=4, query_rows=[7], holes=[0, 7, 1499],
                  dups=[[7, 8], [7, 1030], [100, 1023]], ks=[3, 64, 1100])]
    for sp in specs:
        emb, valid, Q = knn_kat_inputs(sp)
        answers = []
        for k in sp["ks"]:
            for qi in range(len(Q)):
                res = pyref.vec0_knn(emb, Q[qi], k, valid=valid)
                answers.append({"k": k, "q": qi, "rows": [r for r, _ in res],
                                "dist": [float(d).hex() for _, d in res]})
        cases.append({**{kk: v for kk, v in sp.items() if kk != "ks"}, "answers": answers})
    (GOLDEN / "knn_kat.json").write_text(json.dumps({"cases": cases}, separators=(",", ":")))
    print("knn_kat.json:", sum(len(c["answers"]) for c in cases), "answers")


# ----------------------------------------------------------------------------- the live comparisons, pinned
LIVE_FUSION_STRIDE = 5          # every 5th of the 1500 live fusion cases is stored: the fixture stays small


def live_bm25_inputs():
    """Corpus and queries of tests/test_oracle_golden.py::test_pyref_matches_live_reference_bm25 (top-7)."""
    docs, words, weights = make_corpus(77, 120, 40)
    return docs, make_queries(78, words, weights, 25)


def live_fusion_inputs():
    """The 1500 (bm25 hits, semantic hits, alpha, k, limit) cases of test_pyref_matches_live_reference_fusion: empty
    sides, overlapping hit lists, huge and negative ids (CPython set order), exact score / distance ties, int and
    float k."""
    import numpy as np
    rnd = random.Random(2026)
    cases = []
    for _ in range(1500):
        limit = rnd.choice([1, 2, 3, 5, 10, 10, 20])
        space = rnd.choice([3 * limit + 2, 70, 10**6, 2**40, 2**62])
        nb, ns = rnd.randint(0, limit), rnd.randint(0, limit)
        bids = rnd.sample(range(-3 if space > 70 else 0, space), nb) if nb else []
        pool = [i for i in bids]
        sids = []
        while len(sids) < ns:
            c = pool.pop(rnd.randrange(len(pool))) if pool and rnd.random() < 0.5 else rnd.randrange(space)
            if c not in sids:
                sids.append(c)
        bs = [rnd.choice([rnd.uniform(0.1, 30.0), float(rnd.randint(1, 3))]) for _ in bids]
        ds = [float(np.float32(rnd.choice([rnd.uniform(0.0, 1.4), rnd.randint(0, 4) / 8.0]))) for _ in sids]
        bs.sort(reverse=True); ds.sort()
        alpha = rnd.choice([0.0, 0.3, 0.5, 1.0, rnd.random()])
        k = rnd.choice([60, 60.0, 1, 0.5, 1000])
        cases.append((list(zip(bids, bs)), list(zip(sids, ds)), alpha, k, limit))
    return cases


def chunk_inputs():
    """(items, chunk size, overlap, text) cases of tests/test_host_cpu.py::test_text_helpers_match_reference."""
    rnd = random.Random(4)
    cases = []
    for _ in range(400):
        n = rnd.randint(0, 14)
        cs, ov = rnd.randint(1, 5), rnd.randint(0, 6)
        text = " ".join(rnd.choice(["Alpha beta.", "What now?", "Go!", "no stop", "x. "]) for _ in range(n))
        cases.append(([f"w{i}" for i in range(n)], cs, ov, text))
    return cases


def sentence_corpus(seed: int, n: int):
    """make_corpus with descriptions cut into short sentences (for the chunker)."""
    docs, words, weights = make_corpus(seed, n, 30)
    for d in docs:
        d["description"] = ". ".join(d["description"].split()[i] for i in range(min(7, len(d["description"].split())))) + "."
    return docs, words, weights


def reference_bm25(ref_kw, docs, queries, k, workdir: Path):
    """[(id, score)] per query from the reference's KeywordSearch built over ``docs``."""
    p = workdir / "m.json"
    p.write_text(json.dumps({"movies": docs}))
    ks = ref_kw.KeywordSearch.build_from_docs(docs_path=p, db_path=workdir / "k.db", force=True)
    try:
        return [[(r["id"], r["score"]) for r in ks.search(q, k=k)] for q in queries]
    finally:
        ks.close()


def reference_fusion(ref_hs, cases, workdir: Path):
    """(weighted_search, rrf_search) result lists per case, through the reference's own HybridSearch with dummy
    retrievers monkeypatched on its module (the seam of the reference's tests/test_hybrid_search.py:73-76)."""
    class KW:
        hits = []
        def __init__(self, *a, **k): pass
        def search(self, query, k=10, k1=1.5, b=0.75): return [dict(h) for h in KW.hits]
        def close(self): pass

    class SEM:
        hits = []
        def __init__(self, *a, **k): pass
        def query_top_k(self, query_text, k=10, knn_multiplier=10): return [dict(h) for h in SEM.hits]
        def close(self): pass

    old = ref_hs.KeywordSearch, ref_hs.SemanticSearch
    ref_hs.KeywordSearch, ref_hs.SemanticSearch = KW, SEM
    out = []
    try:
        hs = ref_hs.HybridSearch(docs_path=None, db_path=workdir / "h.db")
        for bm, sem, alpha, k, limit in cases:
            KW.hits = [{"id": i, "title": "t", "description": "d", "score": s} for i, s in bm]
            SEM.hits = [{"chunk_id": 0, "distance": d, "chunk": "", "movie_id": i, "title": "t", "description": "d"}
                        for i, d in sem]
            out.append((hs.weighted_search("q", alpha=alpha, limit=limit), hs.rrf_search("q", k=k, limit=limit)))
        hs.close()
    finally:
        ref_hs.KeywordSearch, ref_hs.SemanticSearch = old
    return out


def reference_tables(ref_kw, docs, workdir: Path):
    """The BM25 tables of the reference's own index build over ``docs``, read back by store.export_bm25."""
    import sqlite3
    from rag_search_engine_b200 import store
    p = workdir / "movies.json"
    p.write_text(json.dumps({"movies": docs}))
    ref_kw.KeywordSearch.build_from_docs(docs_path=p, db_path=workdir / "ref.db", force=True).close()
    return store.export_bm25(sqlite3.connect(workdir / "ref.db"))


def encode_hits(hits):
    return [[i, float(s).hex()] for i, s in hits]


def encode_fusion(w, r):
    return ([[x["id"], float(x["bm25"]).hex(), float(x["semantic"]).hex(), float(x["score"]).hex()] for x in w],
            [[x["id"], float(x["score"]).hex(), x["bm25_rank"], x["sem_rank"]] for x in r])


def encode_tables(a):
    post = {}
    for t, r in a.term_row.items():
        s = slice(int(a.indptr[r]), int(a.indptr[r + 1]))
        post[t] = [a.doc_idx[s].tolist(), a.tf[s].tolist()]
    return {"n_movies": int(a.n_movies), "avgdl": float(a.avgdl).hex(), "dl": a.dl.tolist(),
            "doc_ids": a.doc_ids.tolist(), "postings": post}


def live_golden():
    """tests/golden/live_ref.json — what the four live comparisons with the reference compare against (BM25 top-7,
    the fusion cases, the chunkers, the BM25 tables of an index build), so that a checkout without the reference
    still checks them.  Recorded from the reference when ref_import finds it; otherwise from this project's
    restatements (oracle/pyref.py, textutil, store), which those live tests held equal to the reference when they
    were written, and ``source`` says so.  With the reference present the live tests also compare it against this
    fixture."""
    import sqlite3
    from oracle import pyref
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import sentence_chunks, whitespace_tokenizer, window_chunks
    docs, queries = live_bm25_inputs()
    fusion = live_fusion_inputs()[::LIVE_FUSION_STRIDE]
    chunks = chunk_inputs()
    table_docs, _, _ = sentence_corpus(5, 40)
    with tempfile.TemporaryDirectory() as td:
        td = Path(td)
        if ref_import.available():
            ref_kw, ref_hs, ref_utils = ref_import.load()
            source = "reference"
            bm25 = reference_bm25(ref_kw, docs, queries, 7, td)
            fused = reference_fusion(ref_hs, fusion, td)
            chunk, semantic_chunk = ref_utils.chunk, ref_utils.semantic_chunk
            tables = reference_tables(ref_kw, table_docs, td)
        else:
            import importlib.util
            spec = importlib.util.spec_from_file_location("corpus", GOLDEN.parent / "helpers" / "corpus.py")
            corpus = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(corpus)
            source = "restatement"
            postings, doclen = corpus.build_postings(docs)
            bm25 = [pyref.bm25_search(postings, doclen, len(doclen), q.lower().split(), k=7) for q in queries]
            fused = [(pyref.weighted_fuse(bm, sem, alpha, limit), pyref.rrf_fuse(bm, sem, k, limit))
                     for bm, sem, alpha, k, limit in fusion]
            chunk, semantic_chunk = window_chunks, sentence_chunks
            tables = store.export_bm25(sqlite3.connect(store.write_reference_db(td / "ours.db", table_docs,
                                                                                whitespace_tokenizer)))
        out = {"source": source,
               "bm25": {"k": 7, "hits": [encode_hits(h) for h in bm25]},
               "fusion": {"stride": LIVE_FUSION_STRIDE, "cases": [encode_fusion(w, r) for w, r in fused]},
               "chunks": [[chunk(list(items), cs, ov), semantic_chunk(text, cs, ov)] for items, cs, ov, text in chunks],
               "tables": encode_tables(tables)}
    (GOLDEN / "live_ref.json").write_text(json.dumps(out, separators=(",", ":")))
    print("live_ref.json:", source, len(bm25), "BM25 queries,", len(fused), "fusion cases,", len(chunks), "chunker cases")


if __name__ == "__main__":
    import sys
    GOLDEN.mkdir(parents=True, exist_ok=True)
    if "--knn-only" not in sys.argv:
        bm25_golden()
        fusion_golden()
    knn_golden()
    live_golden()
