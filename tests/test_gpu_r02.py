"""GPU tests of the round-2 additions, all through the C-ABI (ctypes -> librse.so): resident-batch rotation
(rse_hybrid_stash), rse_hybrid_drain, the lowered tensor-core threshold, deferred overflow flags for the
row-sharded path, the BM25 / byte counters of rse_stats, clustered corpora, a keyword-only database, and the
Python stream's array form."""
import numpy as np
import pytest

import oracle
from oracle import pyref

pytestmark = pytest.mark.gpu


def unit_rows(rng, n, d=384):
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


@pytest.fixture(scope="module")
def small_world():
    """4000 movies / ~32 k chunks + BM25 index + 3 x 24 queries, loaded once."""
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    from rag_search_engine_b200 import _lib, synth
    se = synth.synth_embeddings(4000, seed=12, device="cpu")
    bm = synth.synth_bm25(4000, 3000, seed=12, mean_len=30, sd_len=10)
    nq = 24
    tok_indptr, terms = synth.synth_token_queries(bm, 3 * nq, seed=13)
    Q = synth.synth_query_vectors(se.emb, 3 * nq, seed=13).numpy()
    idx = _lib.Index(0)
    idx.load_embeddings(se.emb.numpy(), movie_idx=se.movie_of_chunk.numpy())
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    idx.set_id_tables(se.movie_ids, se.movie_ids)
    batches = []
    for b in range(3):
        lo, hi = b * nq, (b + 1) * nq
        tp = (tok_indptr[lo:hi + 1] - tok_indptr[lo]).astype(np.int32)
        batches.append((Q[lo:hi], tp, terms[tok_indptr[lo]:tok_indptr[hi]]))
    yield idx, se, bm, batches
    idx.close()


def same(a, b):
    return all((x.view(np.uint8) == y.view(np.uint8)).all() for x, y in zip(a, b))


def test_stash_rotates_resident_batches(small_world):
    idx, se, bm, batches = small_world
    want = [idx.hybrid(0, 60.0, 10, *b) for b in batches]
    for b, (Q, tp, tr) in enumerate(batches):
        idx.hybrid_stage(Q, tp, tr)
        idx.hybrid_stash(b)
    for rounds in range(2):
        for b in (2, 0, 1):
            idx.hybrid_stash(b)
            idx.hybrid_run(0, 60.0, 10)
            got = idx.hybrid_fetch(10)
            idx.hybrid_stash(b)
            assert same(got, want[b]), f"stashed batch {b} differs from the host-buffer call"
    from rag_search_engine_b200._lib import RseError
    with pytest.raises(RseError):                       # nothing staged after the exchange
        idx.hybrid_run(0, 60.0, 10)
    with pytest.raises(RseError):
        idx.hybrid_stash(16)


def test_drain_discards_tickets_and_unwedges_the_handle(small_world):
    idx, se, bm, batches = small_world
    from rag_search_engine_b200._lib import RseError
    want = idx.hybrid(0, 60.0, 10, *batches[0])
    t0 = idx.hybrid_submit(0, 60.0, 10, *batches[0])
    t1 = idx.hybrid_submit(0, 60.0, 10, *batches[1])
    with pytest.raises(RseError):
        idx.hybrid_submit(0, 60.0, 10, *batches[2])          # two in flight
    assert idx.hybrid_drain() == 2
    with pytest.raises(KeyError):
        idx.hybrid_collect(t0)
    t2 = idx.hybrid_submit(0, 60.0, 10, *batches[0])
    assert same(idx.hybrid_collect(t2), want)
    assert idx.hybrid_drain() == 0
    # ADVICE r01: after a submit nothing is staged in the handle's own buffers
    with pytest.raises(RseError):
        idx.hybrid_run(0, 60.0, 10)
    with pytest.raises(RseError):
        idx.hybrid_fetch(10)


def test_stats_counters(small_world):
    idx, se, bm, batches = small_world
    idx.stats_reset()
    idx.hybrid(0, 60.0, 10, *batches[0])
    st = idx.stats()
    nq = len(batches[0][1]) - 1
    assert st.bm25_queries == nq and st.bm25_fallback_queries == 0
    assert st.bm25_finalists >= st.bm25_queries                  # at least one finalist per query that has postings
    assert st.bm25_candidates >= st.bm25_finalists
    assert st.h2d_bytes >= batches[0][0].nbytes and st.d2h_bytes == nq * 10 * 32 + nq * 4
    # a query with more than 16 tokens cannot take the fixed-point path: the device-side flag sends it to the
    # general kernel and the counter shows it (results stay exact either way, so only the counter can tell)
    known = np.nonzero(bm.df > 0)[0][:20].astype(np.int32)
    tp = np.array([0, 20, 22], np.int32)
    tr = np.concatenate([known, known[:2]]).astype(np.int32)
    idx.stats_reset()
    sc, dc, cnt = idx.bm25(tp, tr, 10)
    st = idx.stats()
    assert st.bm25_queries == 2 and st.bm25_fallback_queries == 1
    osc, odc, ocnt = oracle.bm25_batch(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl, tp, tr, 10)
    assert (odc == dc).all() and (osc.view(np.uint64) == sc.view(np.uint64)).all() and (ocnt == cnt).all()


def test_small_batches_take_the_tensor_core_path_and_match_the_exact_scan():
    """rse.h RSE_TC_MIN_BATCH = 2: on a corpus of >= 256 k rows a 2-query batch goes through K4 (r01: 48), a single
    query takes the streaming scan until a batch has built the shadow; results are identical to the exact scan either way."""
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(41)
    n = 262_144 + 1000
    emb = unit_rows(rng, n)
    emb[100_000] = emb[5]; emb[200_001] = emb[5]
    Q = unit_rows(rng, 8); Q[0] = emb[5]
    idx = _lib.Index(0)
    try:
        idx.load_embeddings(emb)
        idx.stats_reset()
        a3 = idx.knn(Q[:1], 100)
        assert idx.stats().tc_queries == 0
        a4 = idx.knn(Q[:2], 100)
        a8 = idx.knn(Q, 100)
        st = idx.stats()
        assert st.tc_queries == 10 and st.tc_fallback_queries == 0
        surv = idx.tc_last_survivors(8)
        assert (surv >= 100).all() and (surv <= 8192).all()
        a3b = idx.knn(Q[:1], 100)                     # the shadow exists now: a single query takes K4 as well
        assert idx.stats().tc_queries == 11 and same(a3, a3b)
        idx.set_tc_mode(1)
        e8 = idx.knn(Q, 100)
        assert same(a8, e8) and same([x[:1] for x in a8], a3) and same([x[:2] for x in a8], a4)
        od, orow = oracle.vec0_knn(emb, Q[0], 100, literal=False)
        assert a8[1][0].tolist() == orow.tolist() and a8[0][0].view(np.uint32).tolist() == od.view(np.uint32).tolist()
    finally:
        idx.close()


def test_deferred_flags_count_unfinished_queries_on_the_device():
    """Row-sharded path without a host round trip: rse_set_defer_flags + rse_knn_flags_dev.  12 000 copies of one
    vector make the K'-th distance a mass tie: the tensor-core path cannot finish that query."""
    import torch
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(77)
    n = 30_000
    emb = unit_rows(rng, n)
    emb[5000:17000] = emb[5000]
    Q = unit_rows(rng, 64)
    Q[3] = emb[5000] + 0.01 * unit_rows(rng, 1)[0]
    idx = _lib.Index(0)
    try:
        idx.set_tc_mode(2)
        idx.load_embeddings(emb)
        qd = torch.as_tensor(Q, device="cuda")
        cand = torch.empty((64, 100, 3), dtype=torch.int64, device="cuda")
        flag = torch.zeros((1,), dtype=torch.int32, device="cuda")
        idx.set_defer_flags(True)
        idx.knn_local_dev(qd.data_ptr(), 64, 100, cand.data_ptr())
        idx.knn_flags_dev(flag.data_ptr())
        idx.synchronize()
        assert int(flag.item()) >= 1
        assert int((cand[3, :, 0] == -1).sum()) == 100          # the unfinished query carries no candidates
        exact = torch.empty_like(cand)
        idx.set_defer_flags(False)
        idx.knn_local_dev(qd.data_ptr(), 64, 100, exact.data_ptr())
        idx.synchronize()
        assert int((exact[:, :, 0] == -1).sum()) == 0
        ok = [q for q in range(64) if int(cand[q, 0, 0]) != -1]
        assert len(ok) >= 48 and torch.equal(cand[ok], exact[ok])
        idx.set_tc_mode(1)
        scan = torch.empty_like(cand)
        idx.knn_local_dev(qd.data_ptr(), 64, 100, scan.data_ptr())
        idx.synchronize()
        assert torch.equal(scan, exact)
    finally:
        idx.close()


@pytest.mark.parametrize("spread,n_centres,nq", [(0.15, 60, 96), (0.06, 60, 96), (0.02, 40, 96), (0.06, 60, 700)])
def test_clustered_corpus_tensor_core_path_equals_exact_scan(spread, n_centres, nq):
    """VERDICT r01 weak #3: sentence-embedding corpora are clustered — the neighbourhood of a query is dense.
    The filter path must stay exact (and mostly stay ON the tensor cores) when hundreds of rows sit within
    +-2 eps of the K'-th neighbour."""
    from rag_search_engine_b200 import _lib, synth
    se = synth.synth_embeddings(18_000, seed=5, device="cpu", distribution="clustered", n_centres=n_centres, spread=spread)
    emb = se.emb.numpy()
    Q = synth.synth_query_vectors(se.emb, nq, seed=6).numpy()     # 700 queries: three query blocks in ONE launch per stage,
    c = Q[:16] @ emb.T                                            # second-chance gates per block
    kth = np.sort(c, axis=1)[:, -100]
    band = ((c >= (kth - 0.005)[:, None]) & (c <= (kth + 0.005)[:, None])).sum(1)
    out = {}
    for mode in (1, 2):
        idx = _lib.Index(0)
        try:
            idx.set_tc_mode(mode)
            idx.load_embeddings(emb, movie_idx=se.movie_of_chunk.numpy())
            out[mode] = idx.knn(Q, 100) + idx.knn_movies(Q, 10, 100)
            st = idx.stats()
            if mode == 2:
                assert st.tc_queries == 2 * nq
                rate = st.tc_fallback_queries / st.tc_queries
                print(f"spread {spread}: rows within +-2eps of the 100th neighbour median {int(np.median(band))} "
                      f"max {int(band.max())}; fallback rate {rate:.3f}")
                if spread >= 0.15:
                    assert rate <= 0.02, f"clustered neighbourhoods fell back to the exact scan: {rate:.3f}"
        finally:
            idx.close()
    assert same(out[1], out[2])


def test_python_stream_arrays_equal_dicts_and_oracle(small_world):
    """HybridSearch.from_loaded + rrf_search_stream: the list-of-dicts form, the packed-array form with flat
    numpy tokens, and the oracle pipeline agree."""
    idx, se, bm, batches = small_world
    from rag_search_engine_b200 import HybridSearch
    T = len(bm.df)
    names = np.array([f"t{i}" for i in range(T)], dtype=np.str_)
    hs = HybridSearch.from_loaded(idx, dict(zip(names.tolist(), range(T))), se.movie_ids, se.movie_ids,
                                  registry_key="r02-stream-test")
    lists, flat = [], []
    for Q, tp, tr in batches:
        toks = np.where(tr >= 0, names[np.clip(tr, 0, None)], "<oov>")
        tl = toks.tolist()
        lists.append(([tl[tp[i]:tp[i + 1]] for i in range(len(tp) - 1)], Q))
        flat.append(((tp, toks), Q))
    d = list(hs.rrf_search_stream(iter(lists), k=60, limit=10))
    a = list(hs.rrf_search_stream(iter(flat), k=60, limit=10, as_arrays=True))
    emb, movie_of, ids = se.emb.numpy(), se.movie_of_chunk.numpy(), se.movie_ids
    for b, (Q, tp, tr) in enumerate(batches):
        oid, osc, oa, ob, oc = a[b]
        osc_b, odc, ocnt = oracle.bm25_batch(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl, tp, tr, 10)
        kd, krow, kc = oracle.knn_movies_batch(emb, Q, movie_of, 10, 100)
        for q in range(len(tp) - 1):
            bmh = [(int(ids[odc[q, j]]), float(osc_b[q, j])) for j in range(ocnt[q])]
            semh = [(int(ids[movie_of[krow[q, j]]]), float(kd[q, j])) for j in range(kc[q])]
            want = pyref.rrf_fuse(bmh, semh, 60.0, 10)
            assert d[b][q] == [{"id": w["id"], "score": w["score"], "bm25_rank": w["bm25_rank"], "sem_rank": w["sem_rank"]}
                               for w in want]
            assert oid[q, :oc[q]].tolist() == [w["id"] for w in want]
            assert osc[q, :oc[q]].tolist() == [w["score"] for w in want]


def test_keyword_only_database_opens_and_degrades_like_the_reference(tmp_path):
    """ADVICE r01: a database without vec0 tables must open; query_top_k_vec returns [] (the reference creates an
    empty chunk_embeddings table and returns []), and the batch path degrades to BM25-only fusion
    (rag_search_engine/tests/test_hybrid_search.py:94-112)."""
    from rag_search_engine_b200 import HybridSearch, SemanticSearch, store
    from rag_search_engine_b200.textutil import whitespace_tokenizer
    docs = [{"id": 3 * i + 1, "title": f"w{i % 7} w{i % 3}", "description": f"w{i % 5} w{(i * 7) % 11} w1."} for i in range(60)]
    db = store.write_reference_db(tmp_path / "kw.db", docs, whitespace_tokenizer)
    ss = SemanticSearch(docs_path=None, db_path=db)
    assert ss.query_top_k_vec(np.ones((2, 384), np.float32), k=5) == [[], []]
    ss.close()
    hs = HybridSearch(docs_path=None, db_path=db, tokenizer=whitespace_tokenizer)
    try:
        res = hs.rrf_search_batch([["w1"], ["w2", "w4"], ["nope"]], np.ones((3, 384), np.float32), k=60, limit=5)
        kw = hs.keyword.search_tokens([["w1"], ["w2", "w4"], ["nope"]], k=5)
        assert res[2] == []
        for q in range(2):
            assert [h["id"] for h in res[q]] == [int(x) for x in kw[q][0]]
            assert all(h["sem_rank"] is None and h["bm25_rank"] == j for j, h in enumerate(res[q]))
    finally:
        hs.close()


def test_library_owned_nccl_comm_single_rank(small_world):
    """include/rse.h "multi-GPU": the handle owns the NCCL communicator.  With one rank the sharded entry points
    (local top-K' -> all-to-all (self) -> merge -> aggregation / fusion) must equal the single-handle calls; the
    N-rank form is checked against one handle by bench.py --gpus N (sharded_matches_single_gpu)."""
    import torch
    idx, se, bm, batches = small_world
    Q, tp, tr = batches[1]
    nq = Q.shape[0]
    idx.comm_init(idx.comm_unique_id(), 1, 0)
    try:
        n_ranks, rank, ver = idx.comm_info()
        assert (n_ranks, rank) == (1, 0) and ver >= 20000
        qd = torch.as_tensor(Q, device="cuda")
        od = torch.empty((nq, 10), dtype=torch.float32, device="cuda")
        orow = torch.empty((nq, 10), dtype=torch.int64, device="cuda")
        om = torch.empty((nq, 10), dtype=torch.int32, device="cuda")
        oc = torch.empty((nq,), dtype=torch.int32, device="cuda")
        flag = torch.zeros((1,), dtype=torch.int32, device="cuda")
        for fl in (flag.data_ptr(), 0):
            idx.knn_sharded_dev(qd.data_ptr(), nq, 10, 100, od.data_ptr(), orow.data_ptr(), om.data_ptr(), oc.data_ptr(), fl)
            idx.synchronize()
            wd, wrow, wm, wc = idx.knn_movies(Q, 10, 100)
            assert (oc.cpu().numpy() == wc).all() and (orow.cpu().numpy() == wrow).all()
            assert (od.cpu().numpy().view(np.uint32) == wd.view(np.uint32)).all() and (om.cpu().numpy() == wm).all()
        assert int(flag.item()) == 0
        want = idx.hybrid(0, 60.0, 10, Q, tp, tr)
        idx.hybrid_stage(Q, tp, tr)
        oid = torch.empty((nq, 10), dtype=torch.int64, device="cuda")
        osc = torch.empty((nq, 10), dtype=torch.float64, device="cuda")
        oa = torch.empty((nq, 10), dtype=torch.float64, device="cuda")
        ob = torch.empty((nq, 10), dtype=torch.float64, device="cuda")
        ocn = torch.empty((nq,), dtype=torch.int32, device="cuda")
        idx.hybrid_sharded_run_dev(0, 60.0, 10, qd.data_ptr(), nq, oid.data_ptr(), osc.data_ptr(), oa.data_ptr(),
                                   ob.data_ptr(), ocn.data_ptr(), flag.data_ptr())
        idx.synchronize()
        got = (oid.cpu().numpy(), osc.cpu().numpy(), oa.cpu().numpy(), ob.cpu().numpy(), ocn.cpu().numpy())
        assert same(got, want)
    finally:
        idx.comm_destroy()


def test_multimodal_search_ranks_like_the_reference_expression():
    """§8 f4: image -> text search (rag_search_engine/llm/multimodal.py:86-95) with the ranking on the GPU.
    Floating point: similarity within 4e-6 of the reference's numpy expression (fp32 dot products of 512 terms in a
    different summation order: BLAS blocks, the scan sums sequentially); same ids wherever neighbouring similarities
    are further apart than that."""
    import zlib
    from rag_search_engine_b200.multimodal import MultimodalSearch

    class FakeClip:                                   # the CLIP model is out of scope: any object with .encode
        def __init__(self, dim=512):
            self.dim = dim
        def encode(self, items, convert_to_numpy=True, show_progress_bar=False):
            out = np.empty((len(items), self.dim), np.float32)
            for i, t in enumerate(items):
                seed = zlib.crc32(t.encode()) if isinstance(t, str) else 7          # (str hashes differ per process)
                out[i] = np.random.default_rng(seed).standard_normal(self.dim).astype(np.float32) * 3.0
            return out

    docs = [{"id": 100 + i, "title": f"Movie {i}", "description": f"plot {i * 7 % 13} words {i}"} for i in range(6000)]
    docs[17] = {"id": 117, "title": "no description", "document": "fallback text"}
    ms = MultimodalSearch(documents=docs, model=FakeClip())
    try:
        rng = np.random.default_rng(3)
        for trial in range(4):
            img = (ms.text_embeddings[rng.integers(0, 6000)] + 2.0 * rng.standard_normal(512)).astype(np.float32)
            # the reference, verbatim (llm/multimodal.py:86-95)
            image_vec = img / (np.linalg.norm(img) + 1e-12)
            text_vecs = ms.text_embeddings
            text_normed = text_vecs / (np.linalg.norm(text_vecs, axis=1, keepdims=True) + 1e-12)
            similarities = (text_normed @ image_vec).astype(float)
            top = np.argsort(similarities)[::-1][:25]
            got = ms.search_with_vector(img, top_k=25)
            assert len(got) == 25 and list(got[0].keys()) == ["id", "title", "description", "similarity"]
            for j, (g, want) in enumerate(zip(got, top)):
                assert abs(g["similarity"] - similarities[want]) < 4e-6
                gap = min(abs(similarities[top[j]] - similarities[top[j - 1]]) if j else 1.0,
                          abs(similarities[top[j]] - similarities[top[j + 1]]) if j + 1 < len(top) else 1.0)
                if gap > 8e-6:
                    assert g["id"] == docs[want].get("id", want)
        assert ms.search_with_vector(img, top_k=10 ** 6 if False else 3)[0]["id"] == got[0]["id"]
        with pytest.raises(ValueError, match="initialized without documents"):
            MultimodalSearch(documents=None, model=FakeClip()).search_with_image("x.png")
    finally:
        ms.close()


def test_sharded_entry_points_need_a_communicator(small_world):
    import torch
    from rag_search_engine_b200._lib import RseError
    idx, se, bm, batches = small_world
    Q, tp, tr = batches[0]
    qd = torch.as_tensor(Q, device="cuda")
    out = torch.empty((Q.shape[0], 10), dtype=torch.float64, device="cuda")
    with pytest.raises(RseError, match="communicator"):
        idx.knn_sharded_dev(qd.data_ptr(), Q.shape[0], 10, 100, out.data_ptr(), out.data_ptr(), out.data_ptr(), out.data_ptr())
    n_ranks, rank, ver = idx.comm_info()
    assert n_ranks == 0


def test_torch_distributed_sharded_driver_single_rank(small_world):
    """sharded.ShardedHybrid + LibrseShardBackend (the torch.distributed form of the row-sharded step; the gloo test
    drives it with an oracle backend) on one rank must equal the single-handle call."""
    import torch
    from rag_search_engine_b200 import sharded
    idx, se, bm, batches = small_world
    Q, tp, tr = batches[2]
    dev = torch.device("cuda", 0)
    be = sharded.LibrseShardBackend(idx, Q, tp, tr, dev)
    sh = sharded.ShardedHybrid(be, Q.shape[0])
    r = sh.step(torch.as_tensor(Q, device=dev), 0, 60.0, 10)
    idx.synchronize()
    idx.use_own_stream()
    want = idx.hybrid(0, 60.0, 10, Q, tp, tr)
    assert int(r.flagged.item()) == 0
    assert (r.ids.cpu().numpy() == want[0]).all() and (r.score.cpu().numpy() == want[1]).all()
    assert (r.count.cpu().numpy() == want[4]).all()


# ----------------------------------------------------------------------------- the probe's row sample (verified bound)
class _env:
    """librse reads its RSE_* knobs when a handle is created."""
    def __init__(self, **kw):
        self.kw = {k: str(v) for k, v in kw.items()}

    def __enter__(self):
        import os
        self.old = {k: os.environ.get(k) for k in self.kw}
        os.environ.update(self.kw)

    def __exit__(self, *a):
        import os
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.mark.parametrize("distribution,knobs,expect_second", [
    ("isotropic", dict(RSE_TC_SAMPLE_MIN_TILES=1, RSE_TC_SAMPLE_STRIDE=8), False),     # the sample path as shipped
    ("clustered", dict(RSE_TC_SAMPLE_MIN_TILES=1, RSE_TC_SAMPLE_STRIDE=8), False),
    ("isotropic", dict(RSE_TC_SAMPLE_MIN_TILES=1, RSE_TC_SAMPLE_STRIDE=8, RSE_TC_PROBE_RANK=1), True),   # bound always far too tight
    ("isotropic", dict(RSE_TC_SAMPLE_MIN_TILES=1, RSE_TC_SAMPLE_STRIDE=8, RSE_TC_PROBE_RANK=12), True),  # too tight half the time
    ("clustered", dict(RSE_TC_SAMPLE_MIN_TILES=1, RSE_TC_SAMPLE_STRIDE=8, RSE_TC_PROBE_RANK=12), True),
    ("clustered", dict(RSE_TC_SAMPLE_MIN_TILES=1, RSE_TC_SAMPLE_STRIDE=16, RSE_TC_PROBE_RANK=2), True),
])
def test_sampled_probe_bound_is_verified_and_results_stay_exact(distribution, knobs, expect_second):
    """The probe's threshold on the sample path is the j-th best value of a stratified row sample, j << K': tight, and
    valid only with high probability — the refine kernel verifies it (s_K >= T) and re-arms the second filter pass with
    the exact bound when it fails (fewer than K' survivors: the exact scan).  Forcing a small j makes the bound fail for
    many queries: the answers must not change."""
    from rag_search_engine_b200 import _lib, synth
    se = synth.synth_embeddings(9_000, seed=21, device="cpu", distribution=distribution)     # ~72 k rows
    emb = se.emb.numpy()
    nq = 300                                                                                  # two query blocks
    Q = synth.synth_query_vectors(se.emb, nq, seed=22).numpy()
    out = {}
    for mode in (1, 2):
        with _env(**(knobs if mode == 2 else {})):
            idx = _lib.Index(0)
        try:
            idx.set_tc_mode(mode)
            idx.load_embeddings(emb, movie_idx=se.movie_of_chunk.numpy())
            out[mode] = idx.knn(Q, 100) + idx.knn_movies(Q, 10, 100) + idx.knn(Q[:40], 10)
            st = idx.stats()
            if mode == 2:
                assert st.tc_queries == 2 * nq + 40
                print(f"{distribution} {knobs}: second chance {st.tc_second_chance_queries}, fallback {st.tc_fallback_queries} "
                      f"of {st.tc_queries}; survivors p50 {int(np.median(idx.tc_last_survivors(40)))}")
                if expect_second:
                    assert st.tc_second_chance_queries + st.tc_fallback_queries > nq // 4
                else:
                    assert st.tc_second_chance_queries + st.tc_fallback_queries <= 3
        finally:
            idx.close()
    assert same(out[1], out[2])


def test_bench_resident_loop_returns_the_last_timed_batch(small_world, tmp_path):
    """bench.py --dump-outputs: measure_hybrid's last timed step is left staged, fetched after the timer and parked
    again — its results are those of rse_hybrid on batch (steps - 1) % nb, in both fusion modes, and every batch
    is back in its own stash slot afterwards."""
    import torch
    import bench
    idx, se, bm, batches = small_world
    stream = torch.cuda.current_stream()
    tm = bench.Timer(stream, 1, torch.device("cuda", 0))
    for mode, param, steps in ((0, 60.0, 5), (1, 0.5, 3), (0, 60.0, 1)):
        m = bench.measure_hybrid(idx, tm, batches, mode, param, 10, steps, 3, e2e=False)
        assert same(m["last"], idx.hybrid(mode, param, 10, *batches[(steps - 1) % len(batches)])), (mode, steps)
        for b in (2, 0, 1):
            idx.hybrid_stash(b)
            idx.hybrid_run(mode, param, 10)
            got = idx.hybrid_fetch(10)
            idx.hybrid_stash(b)
            assert same(got, idx.hybrid(mode, param, 10, *batches[b])), f"batch {b} not back in its slot"
    oid, osc, oa, ob, oc = m["last"]
    bench.dump_outputs(tmp_path, {"id": oid, "score": osc, "bm25": oa, "semantic": ob, "count": oc})
    assert (np.load(tmp_path / "id.npy") == oid).all() and (np.load(tmp_path / "count.npy") == oc).all()
    assert np.load(tmp_path / "score.npy").tobytes() == osc.tobytes()
