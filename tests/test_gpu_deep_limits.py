"""GPU: deep result lists — BM25 top-k up to 512, the fusion entry points up to limit 1024 and every hybrid entry
point up to limit 512 (409 at the reference's knn_multiplier 10) — against the oracle, and the Python mirrors over a
reference-format SQLite database at limit 300.  Fixtures live in this file."""
import hashlib
import random
import sqlite3
import threading

import numpy as np
import pytest

import oracle
from oracle import pyref
from helpers.corpus import build_postings

pytestmark = pytest.mark.gpu
DIM = 384
RANGE = 7168                         # documents per BM25 range (csrc/bm25.cuh kBmRange)


def _gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


@pytest.fixture()
def idx():
    if not _gpu():
        pytest.skip("no CUDA device")
    from rag_search_engine_b200 import _lib
    h = _lib.Index(0)
    yield h
    h.close()


def same(a, b):
    return all(x.shape == y.shape and (x.view(np.uint8) == y.view(np.uint8)).all() for x, y in zip(a, b))


# ----------------------------------------------------------------------------- fusion up to limit 1024
def _hits(rng, n, space, kind, scores):
    if kind == "big":
        ids = (2**62 - 1 - rng.integers(0, space, n)).tolist()
    elif kind == "neg":
        ids = (rng.integers(0, space, n) - space // 2).tolist()
    else:
        ids = rng.integers(0, space, n).tolist()
    ids = list(dict.fromkeys(ids)) if rng.random() < 0.9 else ids       # a plugged-in retriever may repeat an id
    vals = np.round(rng.uniform(0.0, 3.0, len(ids)), int(rng.choice([1, 2, 6])))   # mass score ties
    vals = sorted(vals.tolist(), reverse=scores)
    return list(zip(ids, vals))


def _by_id(rows, limit):
    """The fused order in RSE_TIE_BY_ID mode: ascending id, then the stable descending sort by score."""
    return sorted(rows, key=lambda r: (-r["score"], r["id"]))[:limit]


@pytest.mark.parametrize("limit", [129, 256, 409, 512, 1024])
def test_fusion_deep_limits_match_reference(idx, limit):
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(limit)
    nq = 24
    cases = []
    for q in range(nq):
        kind = ["small", "small", "big", "neg"][q % 4]
        space = int(rng.choice([limit // 2 + 1, 2 * limit, 10**6])) if kind == "small" else int(rng.choice([3 * limit, 10**9]))
        nb = int(rng.choice([0, limit, rng.integers(1, limit + 1)]))
        ns = int(rng.choice([limit, limit, rng.integers(0, limit + 1)]))
        cases.append((_hits(rng, nb, space, kind, True), _hits(rng, ns, space, kind, False)))
    bid = np.full((nq, limit), -1, np.int64); bsc = np.zeros((nq, limit)); bc = np.zeros(nq, np.int32)
    sid = np.full((nq, limit), -1, np.int64); sds = np.zeros((nq, limit)); sc = np.zeros(nq, np.int32)
    for q, (bm, sem) in enumerate(cases):
        bc[q], sc[q] = len(bm), len(sem)
        for j, (i, s) in enumerate(bm):
            bid[q, j], bsc[q, j] = i, s
        for j, (i, d) in enumerate(sem):
            sid[q, j], sds[q, j] = i, d
    for tie in (_lib.TIE_REFERENCE, _lib.TIE_BY_ID):
        oid, osc, orb, ors, oc = idx.fuse_rrf(limit, 60.0, bid, bsc, bc, sid, sds, sc, tie_mode=tie)
        wid, wb, wsem, wsc, wc = idx.fuse_weighted(limit, 0.3, bid, bsc, bc, sid, sds, sc, tie_mode=tie)
        for q, (bm, sem) in enumerate(cases):
            want = pyref.rrf_fuse(bm, sem, 60, limit)
            if tie == _lib.TIE_BY_ID:
                want = _by_id(pyref.rrf_fuse(bm, sem, 60, 10**9), limit)
            got = [(int(oid[q, j]), float(osc[q, j]).hex(), None if orb[q, j] < 0 else int(orb[q, j]),
                    None if ors[q, j] < 0 else int(ors[q, j])) for j in range(oc[q])]
            assert got == [(w["id"], float(w["score"]).hex(), w["bm25_rank"], w["sem_rank"]) for w in want], (tie, q)
            want = pyref.weighted_fuse(bm, sem, 0.3, limit)
            if tie == _lib.TIE_BY_ID:
                want = _by_id(pyref.weighted_fuse(bm, sem, 0.3, 10**9), limit)
            got = [(int(wid[q, j]), float(wb[q, j]).hex(), float(wsem[q, j]).hex(), float(wsc[q, j]).hex())
                   for j in range(wc[q])]
            assert got == [(w["id"], float(w["bm25"]).hex(), float(w["semantic"]).hex(), float(w["score"]).hex())
                           for w in want], (tie, q)


def test_fusion_limit_above_1024_is_refused(idx):
    from rag_search_engine_b200 import _lib
    z = np.zeros((1, 1025))
    with pytest.raises(_lib.RseError) as e:
        idx.fuse_rrf(1025, 60.0, z.astype(np.int64), z, np.zeros(1, np.int32), z.astype(np.int64), z, np.zeros(1, np.int32))
    assert e.value.code == -4


# ----------------------------------------------------------------------------- BM25 top-k up to 512
class Csr:
    pass


def _tie_corpus(seed=5, n_docs=5 * RANGE + 911, vocab=60):
    """5 ranges and a partial sixth.  Two document lengths and tf mostly 1: a common term gives a handful of distinct
    scores over thousands of documents (mass ties, ordered by first query token, then document).  Terms 50.. are
    rare (df < 400), so queries made of them touch fewer than k documents."""
    rng = np.random.default_rng(seed)
    dl = rng.choice([8, 12], n_docs).astype(np.uint32)
    rows_doc, rows_tf, df = [], [], []
    for t in range(vocab):
        p = 0.5 / (t + 1) if t < 50 else rng.uniform(20, 380) / n_docs
        d = np.nonzero(rng.random(n_docs) < p)[0].astype(np.uint32)
        rows_doc.append(d)
        rows_tf.append(np.where(rng.random(len(d)) < 0.9, 1, 2).astype(np.uint32))
        df.append(len(d))
    c = Csr()
    c.indptr = np.zeros(vocab + 1, np.int64)
    c.indptr[1:] = np.cumsum(df)
    c.doc, c.tf = np.concatenate(rows_doc), np.concatenate(rows_tf)
    c.df, c.dl, c.n, c.avgdl = np.array(df, np.int64), dl, n_docs, float(dl.sum()) / n_docs
    return c


def _queries(rng, nq, vocab=60):
    fixed = [[0], [0, 1], [1, 0], [55], [56, 57], [0, 55], [2, 3, 4], [], [-1], [58, 58], [0, 0, 1], [3, -1, 0]]
    qs = fixed + [rng.integers(-1, vocab, int(rng.integers(1, 6))).tolist() for _ in range(max(0, nq - len(fixed)))]
    qs = qs[:nq]
    tp = np.zeros(len(qs) + 1, np.int32)
    tp[1:] = np.cumsum([len(x) for x in qs])
    return tp, np.array([t for x in qs for t in x], np.int32)


def _load(h, c):
    h.load_bm25(c.indptr, c.doc, c.tf, c.df, c.dl, c.n, c.avgdl)


@pytest.mark.parametrize("mode", [0, 1, 2])
def test_bm25_deep_k_matches_oracle_in_every_mode(idx, mode):
    c = _tie_corpus()
    tp, tr = _queries(np.random.default_rng(1), 60)
    idx.set_bm25_mode(mode)
    _load(idx, c)
    for k in (257, 409, 512):
        osc, odc, ocnt = oracle.bm25_batch(c.indptr, c.doc, c.tf, c.df, c.dl, c.n, c.avgdl, tp, tr, k)
        score, doc, cnt = idx.bm25(tp, tr, k)
        assert (cnt == ocnt).all(), k
        assert (doc == odc).all(), k
        assert (score.view(np.uint64) == osc.view(np.uint64)).all(), k
        assert (ocnt < k).any() and (ocnt == k).any()        # both sides of "fewer than k touched documents"


def test_bm25_10k_queries_at_k512_within_the_candidate_budget(idx):
    import torch
    c = _tie_corpus(seed=9)
    _load(idx, c)
    tp, tr = _queries(np.random.default_rng(2), 10_000)
    idx.bm25(tp[:2], tr[:tp[1]], 10)                       # module, norms and small buffers in place
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    score, doc, cnt = idx.bm25(tp, tr, 512)
    free1, _ = torch.cuda.mem_get_info()
    nq, k = len(tp) - 1, 512
    # 256 MB of candidate lists (rse.cu bm25_run) + the [nq, k] results + the staged tokens, each allocated with a
    # quarter of headroom, plus allocator granularity
    bound = 1.25 * ((256 << 20) + nq * k * 12 + len(tr) * 12 + nq * 4 * 4) + (32 << 20)
    assert free0 - free1 <= bound, (free0 - free1, bound)
    osc, odc, ocnt = oracle.bm25_batch(c.indptr, c.doc, c.tf, c.df, c.dl, c.n, c.avgdl, tp, tr, k)
    assert (cnt == ocnt).all() and (doc == odc).all() and (score.view(np.uint64) == osc.view(np.uint64)).all()


def test_bm25_k_above_512_is_refused(idx):
    from rag_search_engine_b200 import _lib
    c = _tie_corpus()
    _load(idx, c)
    tp, tr = _queries(np.random.default_rng(1), 4)
    with pytest.raises(_lib.RseError) as e:
        idx.bm25(tp, tr, 513)
    assert e.value.code == -4


# ----------------------------------------------------------------------------- hybrid up to limit 512
@pytest.fixture(scope="module")
def world():
    if not _gpu():
        pytest.skip("no CUDA device")
    from rag_search_engine_b200 import synth
    se = synth.synth_embeddings(3000, seed=31, device="cpu", distribution="clustered")
    emb, movie_of, ids = se.emb.numpy(), se.movie_of_chunk.numpy(), se.movie_ids
    bm = synth.synth_bm25(3000, 400, seed=31, mean_len=25.0, sd_len=8.0)
    tp, tr = synth.synth_token_queries(bm, 300, seed=32, min_tok=1, max_tok=5)
    Q = synth.synth_query_vectors(se.emb, 300, seed=33).numpy()
    return {"emb": emb, "movie_of": movie_of, "ids": ids, "bm": bm, "tp": tp, "tr": tr, "Q": Q}


def _hybrid_index(w, rows=None, pos_base=0):
    from rag_search_engine_b200 import _lib
    h = _lib.Index(0)
    lo, hi = rows or (0, len(w["emb"]))
    h.load_embeddings(w["emb"][lo:hi], movie_idx=w["movie_of"][lo:hi], rowid=np.arange(lo, hi, dtype=np.int64) + 1,
                      pos_base=pos_base)
    bm = w["bm"]
    h.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    h.set_id_tables(w["ids"], w["ids"])
    return h


def _batch(w, nq):
    tp = w["tp"][:nq + 1].copy()
    return w["Q"][:nq], tp, w["tr"][:tp[-1]]


def _oracle_hybrid(w, Q, tp, tr, mode, param, limit, mult):
    """BM25 + KNN per movie + the reference's fusion, composed as scripts/gpu_fuzz.py composes it."""
    bm, ids, movie_of = w["bm"], w["ids"], w["movie_of"]
    osc, odc, ocnt = oracle.bm25_batch(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl, tp, tr, limit)
    kd, krow, kc = oracle.knn_movies_batch(w["emb"], Q, movie_of, limit, max(limit * mult, limit))
    out = []
    for qi in range(len(Q)):
        bmh = [(int(ids[odc[qi, j]]), float(osc[qi, j])) for j in range(ocnt[qi])]
        semh = [(int(ids[movie_of[krow[qi, j]]]), float(kd[qi, j])) for j in range(kc[qi])]
        if mode == 0:
            out.append([(x["id"], float(x["score"]).hex(), x["bm25_rank"], x["sem_rank"])
                        for x in pyref.rrf_fuse(bmh, semh, param, limit)])
        else:
            out.append([(x["id"], float(x["bm25"]).hex(), float(x["semantic"]).hex(), float(x["score"]).hex())
                        for x in pyref.weighted_fuse(bmh, semh, param, limit)])
    return out


def _rows(res, mode):
    oid, sc, a, b, cnt = res
    if mode == 0:
        return [[(int(oid[q, j]), float(sc[q, j]).hex(), None if a[q, j] < 0 else int(a[q, j]),
                  None if b[q, j] < 0 else int(b[q, j])) for j in range(cnt[q])] for q in range(len(cnt))]
    return [[(int(oid[q, j]), float(a[q, j]).hex(), float(b[q, j]).hex(), float(sc[q, j]).hex()) for j in range(cnt[q])]
            for q in range(len(cnt))]


DEEP = [(129, 10), (256, 10), (409, 10), (512, 8)]


@pytest.mark.parametrize("limit,mult", DEEP)
def test_hybrid_deep_limits_match_oracle_pipeline(world, limit, mult):
    h = _hybrid_index(world)
    try:
        for nq in (1, 37, 300):
            Q, tp, tr = _batch(world, nq)
            for mode, param in ((0, 60.0), (1, 0.5)):
                res = h.hybrid(mode, param, limit, Q, tp, tr, knn_multiplier=mult)
                assert _rows(res, mode) == _oracle_hybrid(world, Q, tp, tr, mode, param, limit, mult), (nq, mode)
                assert res[4].max() > 128
                # the serving loop and a parked batch give the blocking call's bytes
                t = h.hybrid_submit(mode, param, limit, Q, tp, tr, knn_multiplier=mult)
                assert same(h.hybrid_collect(t), res)
                h.hybrid_stage(Q, tp, tr)
                h.hybrid_stash(3)
                h.hybrid_stash(3)
                h.hybrid_run(mode, param, limit, knn_multiplier=mult)
                assert same(h.hybrid_fetch(limit), res)
    finally:
        h.close()


def test_hybrid_limit_410_at_multiplier_10_is_refused(world):
    from rag_search_engine_b200 import _lib
    h = _hybrid_index(world)
    try:
        Q, tp, tr = _batch(world, 2)
        for limit, mult in ((410, 10), (513, 1)):
            with pytest.raises(_lib.RseError) as e:
                h.hybrid(0, 60.0, limit, Q, tp, tr, knn_multiplier=mult)
            assert e.value.code == -4
    finally:
        h.close()


@pytest.mark.parametrize("limit,mult", [(409, 10), (512, 8)])
def test_merged_shards_equal_one_handle(world, limit, mult):
    import torch
    n = len(world["emb"])
    cut = (n // 2 // 1024) * 1024
    full = _hybrid_index(world)
    shards = [_hybrid_index(world, (0, cut)), _hybrid_index(world, (cut, n), pos_base=cut)]
    try:
        Q, tp, tr = _batch(world, 37)
        nq, kprime = len(Q), max(limit * mult, limit)
        qd = torch.as_tensor(Q, device="cuda")
        cands = []
        for s in shards:
            c = torch.empty((nq, kprime, 3), dtype=torch.int64, device="cuda")
            s.knn_local_dev(qd.data_ptr(), nq, kprime, c.data_ptr())
            s.synchronize()
            cands.append(c)
        gathered = torch.stack(cands).contiguous()
        for mode, param in ((0, 60.0), (1, 0.5)):
            want = full.hybrid(mode, param, limit, Q, tp, tr, knn_multiplier=mult)
            full.hybrid_stage(Q, tp, tr)
            out = (torch.empty((nq, limit), dtype=torch.int64, device="cuda"),
                   *[torch.empty((nq, limit), dtype=torch.float64, device="cuda") for _ in range(3)],
                   torch.empty((nq,), dtype=torch.int32, device="cuda"))
            full.hybrid_run_merged_dev(mode, param, limit, gathered.data_ptr(), 2, *[t.data_ptr() for t in out],
                                       knn_multiplier=mult)
            full.synchronize()
            assert same(tuple(t.cpu().numpy() for t in out), want), mode
    finally:
        for h in [full, *shards]:
            h.close()


def _sharded_run(h, mode, param, limit, mult, Q_all, nq_all, lo, hi, result):
    import torch
    dev = torch.device("cuda", h.device)
    with torch.cuda.device(dev):
        qd = torch.as_tensor(Q_all, device=dev)
        ns = hi - lo
        out = (torch.empty((max(ns, 1), limit), dtype=torch.int64, device=dev),
               *[torch.empty((max(ns, 1), limit), dtype=torch.float64, device=dev) for _ in range(3)],
               torch.empty((max(ns, 1),), dtype=torch.int32, device=dev))
        h.hybrid_sharded_run_dev(mode, param, limit, qd.data_ptr(), nq_all, *[t.data_ptr() for t in out],
                                 knn_multiplier=mult)
        h.synchronize()
        result[lo] = tuple(t.cpu().numpy()[:ns] for t in out)


def test_nccl_sharded_deep_limit_single_rank(world):
    """rse_hybrid_sharded_run_dev on a one-rank communicator (all-to-all with itself) at limit 409."""
    h = _hybrid_index(world)
    try:
        h.comm_init(h.comm_unique_id(), 1, 0)
        Q, tp, tr = _batch(world, 37)
        want = h.hybrid(0, 60.0, 409, Q, tp, tr)
        h.hybrid_stage(Q, tp, tr)
        res = {}
        _sharded_run(h, 0, 60.0, 409, 10, Q, len(Q), 0, len(Q), res)
        assert same(res[0], want)
        h.comm_destroy()
    finally:
        h.close()


def test_nccl_sharded_deep_limit_two_ranks(world):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("the two-rank NCCL step needs two GPUs; this machine has one")
    from rag_search_engine_b200 import _lib
    n = len(world["emb"])
    cut = (n // 2 // 1024) * 1024
    Q, tp, tr = _batch(world, 37)
    ref = _hybrid_index(world)
    try:
        want = ref.hybrid(1, 0.5, 409, Q, tp, tr)
    finally:
        ref.close()
    uid = _lib.Index.comm_unique_id()
    ranks = []
    for r, (lo, hi, base) in enumerate(((0, cut, 0), (cut, n, cut))):
        h = _lib.Index(r)
        h.load_embeddings(world["emb"][lo:hi], movie_idx=world["movie_of"][lo:hi],
                          rowid=np.arange(lo, hi, dtype=np.int64) + 1, pos_base=base)
        bm = world["bm"]
        h.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
        h.set_id_tables(world["ids"], world["ids"])
        ranks.append(h)
    try:
        inits = [threading.Thread(target=h.comm_init, args=(uid, 2, r)) for r, h in enumerate(ranks)]
        [t.start() for t in inits]
        [t.join() for t in inits]
        half = len(Q) - len(Q) // 2                         # query slices as rse.cu query_slice cuts them
        res, runs = {}, []
        for r, (lo, hi) in enumerate(((0, half), (half, len(Q)))):
            ranks[r].hybrid_stage(Q[lo:hi], (tp[lo:hi + 1] - tp[lo]).astype(np.int32), tr[tp[lo]:tp[hi]])
            runs.append(threading.Thread(target=_sharded_run, args=(ranks[r], 1, 0.5, 409, 10, Q, len(Q), lo, hi, res)))
        [t.start() for t in runs]
        [t.join() for t in runs]
        got = tuple(np.concatenate([res[0][i], res[half][i]]) for i in range(5))
        assert same(got, want)
    finally:
        for h in ranks:
            h.comm_destroy()
            h.close()


# ----------------------------------------------------------------------------- Python mirrors over SQLite
class HashEncoder:
    """Deterministic stand-in for the sentence encoder: a unit vector per text."""

    def get_sentence_embedding_dimension(self):
        return DIM

    def encode(self, texts, show_progress_bar=False):
        out = np.empty((len(texts), DIM), np.float32)
        for i, t in enumerate(texts):
            seed = int.from_bytes(hashlib.sha256(t.encode()).digest()[:8], "little")
            v = np.random.default_rng(seed).standard_normal(DIM).astype(np.float32)
            out[i] = v / np.linalg.norm(v)
        return out


class HashCrossEncoder:
    """Deterministic stand-in for the cross-encoder: a score per (query, text) pair, with ties."""

    def predict(self, pairs):
        return np.array([int.from_bytes(hashlib.sha256((q + "|" + t).encode()).digest()[:2], "little") % 97 / 7.0
                         for q, t in pairs], np.float32)


@pytest.fixture(scope="module")
def sqlite_world(tmp_path_factory):
    if not _gpu():
        pytest.skip("no CUDA device")
    from rag_search_engine_b200 import store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    rnd = random.Random(8)
    words = [f"w{i}" for i in range(60)]
    weights = [1.0 / (i + 1) for i in range(60)]
    docs = []
    for did in sorted(rnd.sample(range(5, 9000), 1200)):
        title = " ".join(rnd.choices(words, weights, k=rnd.randint(1, 3))).title()
        desc = " ".join(" ".join(rnd.choices(words, weights, k=rnd.randint(3, 9))) + "." for _ in range(rnd.randint(1, 4)))
        docs.append({"id": did, "title": title, "description": desc})
    enc = HashEncoder()
    db = store.write_reference_db(tmp_path_factory.mktemp("deepdb") / "movies.db", docs, whitespace_tokenizer,
                                  embed=enc.encode)
    return {"db": db, "docs": docs, "enc": enc}


def _oracle_semantic(w, text, k, mult=10):
    from rag_search_engine_b200.textutil import chunk_text
    conn = sqlite3.connect(w["db"])
    chunks = conn.execute("SELECT id, movie_id, chunk_index, max_chunk_size, overlap FROM chunks ORDER BY id").fetchall()
    movies = {r[0]: (r[1], r[2]) for r in conn.execute("SELECT id, title, description FROM movies")}
    conn.close()
    texts = [chunk_text(*movies[c[1]], c[2], c[3], c[4]) for c in chunks]
    emb = w["enc"].encode(texts)
    d, rows = oracle.vec0_knn(emb, w["enc"].encode([text])[0], max(k * mult, k))
    return [(m, dd) for _r, dd, m in pyref.aggregate_movies([(int(r), float(dd), chunks[r][1]) for dd, r in zip(d, rows)], k)]


def test_python_mirrors_at_limit_300(sqlite_world):
    from rag_search_engine_b200 import HybridSearch, _lib
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    w = sqlite_world
    postings, doclen = build_postings(w["docs"])
    meta = {d["id"]: d for d in w["docs"]}
    ce = HashCrossEncoder()
    hs = HybridSearch(docs_path=None, db_path=w["db"], tokenizer=whitespace_tokenizer, encoder=w["enc"], cross_encoder=ce)
    try:
        for q in ("w0 w1", "w2 w7 w30", "w0"):
            bm = pyref.bm25_search(postings, doclen, len(doclen), q.lower().split(), k=300)
            sem = _oracle_semantic(w, q, 300)
            assert len(bm) > 128 and len(sem) == 300
            want = pyref.rrf_fuse(bm, sem, 60, 300)
            got = hs.rrf_search(q, k=60, limit=300)
            assert [(g["id"], g["score"], g["bm25_rank"], g["sem_rank"]) for g in got] == \
                   [(x["id"], x["score"], x["bm25_rank"], x["sem_rank"]) for x in want]
            ww = pyref.weighted_fuse(bm, sem, 0.5, 300)
            gw = hs.weighted_search(q, 0.5, limit=300)
            assert [(g["id"], g["bm25"], g["semantic"], g["score"]) for g in gw] == \
                   [(x["id"], x["bm25"], x["semantic"], x["score"]) for x in ww]
            # hybrid_search.py:279-312: the cross-encoder scores the WHOLE fused union, then [:limit]
            union = pyref.rrf_fuse(bm, sem, 60, 10**9)
            scores = ce.predict([[q, f"{meta[x['id']]['title']} - {meta[x['id']]['description']}"] for x in union])
            ranked = sorted(zip(union, scores.tolist()), key=lambda p: (p[1], p[0]["score"]), reverse=True)[:300]
            gr = hs.rrf_search(q, k=60, limit=300, rerank_method="cross_encoder")
            assert [(g["id"], g["cross_encoder_score"]) for g in gr] == [(x["id"], float(s)) for x, s in ranked]
            # the batch path at the same depth
            qv = w["enc"].encode([q])
            gb = hs.rrf_search_batch([q.lower().split()], qv, k=60, limit=300)[0]
            assert [(g["id"], g["score"], g["bm25_rank"], g["sem_rank"]) for g in gb] == \
                   [(x["id"], x["score"], x["bm25_rank"], x["sem_rank"]) for x in want]
        got = hs.keyword.search("w0 w1", k=512)
        assert [(r["id"], r["score"]) for r in got] == pyref.bm25_search(postings, doclen, len(doclen), ["w0", "w1"], k=512)
        with pytest.raises((_lib.RseError, ValueError)):
            hs.rrf_search("w0", limit=410)
        with pytest.raises(_lib.RseError):
            hs.keyword.search("w0", k=513)
    finally:
        hs.close()
