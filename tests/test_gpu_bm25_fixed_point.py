"""Fixed-point BM25 (bm25_fx_kernel + bm25_fx_finish_kernel, mode 0) at the edges of its exactness argument.

Every case runs modes 0, 1 and 2 and oracle.bm25_batch and compares counts, documents and score bits, and asserts
through stats() which path mode 0 took: where the fixed-point path must finish the queries, bm25_finalists > 0 and
no fallback; where a cap must trip, the exact number of queries handed to the general kernel.  A case that fell
back silently would test nothing.  The inputs are built with the CPU model in helpers/bm25_fx.py, and
test_bm25_fx_model.py checks on the CPU that each one reaches the edge it aims at."""
import math

import numpy as np
import pytest

import oracle
from oracle import pyref
from helpers import bm25_fx as fx
from helpers import bm25_fx_cases as cases
from helpers.bm25_fx_cases import pack

pytestmark = pytest.mark.gpu


def run_modes(idx, c, queries, k, k1=1.5, b=0.75, fallback=0, finalists=True):
    """Modes 0 / 1 / 2 against the oracle, bit for bit; mode 0's path through the stats counters."""
    tp, tr = pack(queries)
    osc, odc, ocnt = oracle.bm25_batch(*c.args(), tp, tr, k, k1, b)
    try:
        for mode in (0, 1, 2):
            idx.set_bm25_mode(mode)
            idx.stats_reset()
            sc, dc, cnt = idx.bm25(tp, tr, k, k1, b)
            st = idx.stats()
            bad = np.nonzero(cnt != ocnt)[0]
            assert not len(bad), f"mode {mode}: hit counts {cnt[bad[:8]].tolist()} vs oracle {ocnt[bad[:8]].tolist()} at queries {bad[:8].tolist()}"
            bad = np.nonzero((dc != odc).any(axis=1))[0]
            assert not len(bad), f"mode {mode}: documents differ at queries {bad[:8].tolist()}"
            bad = np.nonzero((sc.view(np.uint64) != osc.view(np.uint64)).any(axis=1))[0]
            assert not len(bad), f"mode {mode}: score bits differ at queries {bad[:8].tolist()}"
            if mode == 0:
                assert st.bm25_queries == len(queries)
                assert st.bm25_fallback_queries == fallback, f"mode 0 handed {st.bm25_fallback_queries} queries on, expected {fallback}"
                if finalists:
                    assert st.bm25_finalists > 0, "the fixed-point path finished no query"
                else:
                    assert st.bm25_finalists == 0, "the fixed-point path ran where it must not"
    finally:
        idx.set_bm25_mode(0)
    return ocnt


def unit_rows(rng, n, d=384):
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


# ----------------------------------------------------------------------------- zero contributions
def test_zero_contributions_term_in_every_document(fresh_index):
    """20 000 documents, k1 = 1000: U adds round(idfx * 512) = 0 to every document.  Each such document must
    still be a hit; with U in every document they are a mass tie, which the general kernel finishes."""
    case = cases.zero_small()
    c, U, R = case.corpus, case.terms["U"], case.terms["R"]
    fresh_index.load_bm25(*c.args())
    ocnt = run_modes(fresh_index, c, [[U], [U, R], [R, U]], 10, 1000.0, 0.75, fallback=3, finalists=False)
    assert ocnt.tolist() == [10, 10, 10]
    ocnt = run_modes(fresh_index, c, [[R]], 10, 1000.0, 0.75)
    assert ocnt.tolist() == [3]


def test_zero_contributions_long_document(fresh_index):
    """1000 documents, k1 = 4000, one document 666 times the average length: its posting of R rounds to wq = 0."""
    case = cases.zero_long_doc()
    c, U, R = case.corpus, case.terms["U"], case.terms["R"]
    fresh_index.load_bm25(*c.args())
    ocnt = run_modes(fresh_index, c, [[R], [R, R]], 10, 4000.0, 0.75)
    assert ocnt.tolist() == [5, 5]
    run_modes(fresh_index, c, [[U], [U, R], [R, U]], 10, 4000.0, 0.75, fallback=3, finalists=False)


def test_zero_contributions_hybrid_under_the_filter(fresh_index):
    """The 20 000-document case through the hybrid step with the tensor-core filter forced on, so BM25 runs in its
    896-thread shape on the second stream; compared with oracle BM25 + oracle KNN + the reference's RRF."""
    case = cases.zero_small()
    c, U, R = case.corpus, case.terms["U"], case.terms["R"]
    rng = np.random.default_rng(8)
    n = c.n_docs
    emb = unit_rows(rng, n)
    movie_of = np.arange(n, dtype=np.int32)
    ids = np.arange(n, dtype=np.int64) * 3 + 7
    queries = [[U], [U, R], [R, U], [R]] * 16
    tp, tr = pack(queries)
    Q = unit_rows(rng, len(queries))
    Q[3] = emb[case.info["r_docs"][0]]
    idx = fresh_index
    idx.set_tc_mode(2)
    idx.load_embeddings(emb, movie_idx=movie_of)
    idx.load_bm25(*c.args())
    idx.set_id_tables(ids, ids)
    idx.stats_reset()
    limit = 10
    oid, sc, _, _, cnt = idx.hybrid(0, 60.0, limit, Q, tp, tr, k1=1000.0, b=0.75)
    st = idx.stats()
    assert st.tc_queries >= len(queries), "the tensor-core filter did not run"
    assert st.bm25_fallback_queries == 48 and st.bm25_finalists > 0
    osc, odc, ocnt = oracle.bm25_batch(*c.args(), tp, tr, limit, 1000.0, 0.75)
    kd, krow, kc = oracle.knn_movies_batch(emb, Q, movie_of, limit, limit * 10, literal=False)
    for qi in range(len(queries)):
        bmh = [(int(ids[odc[qi, j]]), float(osc[qi, j])) for j in range(ocnt[qi])]
        semh = [(int(ids[movie_of[krow[qi, j]]]), float(kd[qi, j])) for j in range(kc[qi])]
        want = [(x["id"], x["score"]) for x in pyref.rrf_fuse(bmh, semh, 60.0, limit)]
        got = [(int(oid[qi, j]), float(sc[qi, j])) for j in range(cnt[qi])]
        assert got == want, f"hybrid query {qi} ({queries[qi]})"


def test_zero_contributions_largest_corpus(fresh_index):
    """14 680 064 documents (2048 ranges; the group count is capped at 32, 64 ranges each) at the default k1 and b:
    U adds 0 to every document and R's posting in the 1.3 M-token document has wq = 0.  One more document is
    refused."""
    case = cases.zero_largest()
    c, U, R, S = case.corpus, case.terms["U"], case.terms["R"], case.terms["S"]
    fresh_index.load_bm25(*c.args())
    threads = oracle.lib().oracle_num_threads()
    oracle.set_threads(min(threads, 8))           # the oracle keeps 16 B per document per thread
    try:
        ocnt = run_modes(fresh_index, c, [[R], [S], [S, R], [R, R, S]], 10)
        assert ocnt.tolist() == [3, 10, 10, 10]
        run_modes(fresh_index, c, [[U], [U, R], [R, U]], 10, fallback=3, finalists=False)
    finally:
        oracle.set_threads(threads)
    from rag_search_engine_b200._lib import RseError
    one = np.ones(1, np.uint32)
    with pytest.raises(RseError, match="14,680,064"):
        fresh_index.load_bm25(np.array([0, 1], np.int64), np.zeros(1, np.uint32), one, np.ones(1, np.int64),
                              np.full(fx.MAX_DOCS + 1, 2, np.uint32), fx.MAX_DOCS + 1, 2.0)


# ----------------------------------------------------------------------------- margin
@pytest.mark.parametrize("ntok", [2, 16])
@pytest.mark.parametrize("k", [1, 10, 32])
def test_margin_inverted_order_at_place_k(fresh_index, k, ntok):
    """k documents rank above k others exactly but sit more than kFxMargin below them in fixed point: a margin
    that does not grow with the query's tokens returns the wrong k."""
    check_margin_case(fresh_index, cases.margin_case(k, ntok), k)


@pytest.mark.parametrize("ntok", [2, 16])
@pytest.mark.parametrize("k", [1, 10, 32])
def test_margin_inverted_order_inside_one_group(fresh_index, k, ntok):
    """The document at place k and one document above it by more than kFxMargin in fixed point but below it exactly,
    in the same range group: bm25_fx_kernel's threshold and compaction must use the per-query margin, or the document
    never reaches the finish kernel."""
    check_margin_case(fresh_index, cases.margin_case(k, ntok, same_group=True), k)


def check_margin_case(idx, case, k):
    c = case.corpus
    idx.load_bm25(*c.args())
    tp, tr = pack([case.info["query"]])
    run_modes(idx, c, [case.info["query"]], k)
    sc, dc, cnt = idx.bm25(tp, tr, k)
    assert sorted(dc[0, :cnt[0]].tolist()) == case.info["answer"].tolist()


# ----------------------------------------------------------------------------- capacities
@pytest.mark.parametrize("n,splits,fallback", [(48, (48, 0, 0), 0), (49, (49, 0, 0), 1),
                                               (96, (32, 32, 32), 0), (97, (33, 32, 32), 1)])
def test_finalist_caps(fresh_index, n, splits, fallback):
    """kFxFinalCap = 48 finalists of one range group, kFxRescoreCap = 96 across groups: a group of that size whose
    fixed-point sums span just less than the margin is finished on the fixed-point path, one more document hands the
    query on."""
    case = cases.tie_group(n, splits)
    c = case.corpus
    fresh_index.load_bm25(*c.args())
    R, Z = case.terms["R"], case.terms["Z"]
    run_modes(fresh_index, c, [[R]], 10, fallback=fallback, finalists=not fallback)
    run_modes(fresh_index, c, [[R]] * 3, 32, fallback=3 * fallback, finalists=not fallback)


@pytest.mark.parametrize("n_cand,fallback", [(256, 0), (257, 1)])
def test_candidate_cap_and_compaction(fresh_index, n_cand, fallback):
    """kBsCandCap = 256 candidates in one range: 256 are compacted (>= kBsCompactAt) to the top k and finished,
    257 hand the query on."""
    case = cases.candidate_range(n_cand)
    c = case.corpus
    fresh_index.load_bm25(*c.args())
    run_modes(fresh_index, c, [[case.terms["R"]]], 10, fallback=fallback, finalists=not fallback)


@pytest.mark.parametrize("n_first,fallback", [(128, 0), (127, 1)])
def test_compaction_at_128(fresh_index, n_first, fallback):
    """kBsCompactAt = 128 candidates after the first range of a two-range group: compaction raises the threshold
    above range 1's low documents and the query is finished; at 127 it does not run and range 1 overflows the list."""
    case = cases.compaction_boundary(n_first)
    c = case.corpus
    fresh_index.load_bm25(*c.args())
    run_modes(fresh_index, c, [[case.terms["R"]]], 10, fallback=fallback, finalists=not fallback)


# ----------------------------------------------------------------------------- format edges
def test_sum_next_to_2p31(fresh_index):
    """16 tokens of the largest-idf term against the weight nearest k1 + 1 at the largest k1 the path accepts:
    the fixed-point sum is within 2^-4 of 2^31.  17 tokens leave the path."""
    case = cases.near_2p31()
    c, X = case.corpus, case.terms["X"]
    k1, b = case.info["k1"], case.info["b"]
    fresh_index.load_bm25(*c.args())
    run_modes(fresh_index, c, [[X] * 16, [X] * 8], 10, k1, b)
    run_modes(fresh_index, c, [[X] * 17], 10, k1, b, fallback=1, finalists=False)


@pytest.fixture(scope="module")
def rare_world():
    """A random corpus and 300 queries of 1..6 terms with df <= 8: at most 48 documents per query, so no cap can
    trip and every query must be finished on the fixed-point path."""
    c = cases.random_corpus(30_000, 20_000, seed=12)
    rng = np.random.default_rng(13)
    df = c.df
    rare = np.nonzero((df >= 1) & (df <= 8))[0]
    queries = [rng.choice(rare, int(rng.integers(1, 7))).tolist() for _ in range(300)]
    return c, rare, queries


@pytest.mark.parametrize("k,k1,b,path", [(32, 1.5, 0.75, "fx"), (33, 1.5, 0.75, "general"),
                                         (10, 0.0, 0.75, "fx"), (10, 1.5, 0.0, "fx"), (10, 1.5, 1.0, "fx"),
                                         (10, 1.5, math.nextafter(1.0, 2.0), "exact-order")])
def test_parameter_edges(fresh_index, rare_world, k, k1, b, path):
    """k = 32 is the last k of the streaming path; k1 = 0 clamps every weight at 2^19 - 1; b = 0 and b = 1 are the
    ends of the accepted b, the next double above 1 leaves the fixed-point path."""
    c, _, queries = rare_world
    fresh_index.load_bm25(*c.args())
    assert fx.eligible(k, 6, k1, b, c.n_movies) == (path == "fx")
    run_modes(fresh_index, c, queries, k, k1, b, finalists=(path == "fx"))


@pytest.mark.parametrize("n_docs", [2 * fx.BM_RANGE, 2 * fx.BM_RANGE + 1])
def test_range_edges(fresh_index, n_docs):
    """Documents at range offsets 0 and 7167, n_docs a multiple of 7168 and one more."""
    case = cases.range_edges(n_docs)
    c, E, F = case.corpus, case.terms["E"], case.terms["F"]
    fresh_index.load_bm25(*c.args())
    for k in (1, 10, 32):
        ocnt = run_modes(fresh_index, c, [[E], [E, F], [F, E], [F]], k)
        assert ocnt[0] == min(k, len(case.info["e_docs"]))


# ----------------------------------------------------------------------------- chunks
def test_chunks_of_4096_queries(fresh_index, rare_world):
    """10 000 queries: three chunks of at most 4096 queries, each with its own launches.  Queries the fixed-point path
    must hand on (17 tokens, a mass tie) sit at the chunk edges 4095, 4096, 8191, 8192 and at 9999; every query is
    compared with the oracle in every mode (mode 1 once wrote the lists of chunks after the first out of bounds)."""
    c0, rare, _ = rare_world
    c, M = cases.with_mass_tie(c0, np.arange(0, 3000))
    rng = np.random.default_rng(14)
    queries = [rng.choice(rare, int(rng.integers(1, 7))).tolist() for _ in range(10_000)]
    for pos in (4095, 8192, 9999):
        queries[pos] = rng.choice(rare, 17).tolist()
    for pos in (4096, 8191):
        queries[pos] = [M]
    fresh_index.load_bm25(*c.args())
    run_modes(fresh_index, c, queries, 10, fallback=5)
