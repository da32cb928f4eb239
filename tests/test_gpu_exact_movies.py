"""rse_knn_movies_exact (SemanticSearch(..., exact_movies=True)) against the numpy restatement of its contract
(helpers/exact_movies_ref.py over oracle.all_distances), bit for bit: rows, movies, distance bits, order, counts."""
import numpy as np
import pytest

from helpers.exact_movies_ref import exact_movies

pytestmark = pytest.mark.gpu
RSE_ERR_INVALID, RSE_ERR_STATE = -1, -3                          # include/rse.h


def unit_rows(rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def crowded(rng, n_movies, dim, lo=2, hi=12):
    """Movies whose chunks sit close together, so one movie fills many slots of a top-K' shortlist."""
    per = rng.integers(lo, hi, n_movies)
    movie_of = np.repeat(np.arange(n_movies, dtype=np.int32), per)
    centers = unit_rows(rng, n_movies, dim)
    emb = centers[movie_of] + 0.3 * unit_rows(rng, len(movie_of), dim)
    emb /= np.linalg.norm(emb, axis=1, keepdims=True)
    return emb.astype(np.float32), movie_of, centers


def check(got, emb, Q, movie_of, k, valid=None, use_fma=False):
    dist, rowid, movie, cnt = got[:4]
    for qi in range(len(Q)):
        od, orow, omov = exact_movies(emb, Q[qi], movie_of, k, valid=valid, use_fma=use_fma)
        c = int(cnt[qi])
        assert c == len(orow), (qi, c, len(orow))
        assert rowid[qi, :c].tolist() == orow.tolist(), qi
        assert movie[qi, :c].tolist() == omov.tolist(), qi
        assert dist[qi, :c].view(np.uint32).tolist() == od.view(np.uint32).tolist(), qi
        assert (rowid[qi, c:] == -1).all() and (movie[qi, c:] == -1).all()


def new_index(monkeypatch=None, budget=None):
    from rag_search_engine_b200 import _lib
    if budget is not None:
        monkeypatch.setenv("RSE_MOVIES_EXACT_BUDGET", str(budget))
    idx = _lib.Index(0)
    if budget is not None:
        monkeypatch.delenv("RSE_MOVIES_EXACT_BUDGET")
    return idx


def test_crowded_movies_get_k_results(fresh_index):
    """The corpus where knn_movies comes up short (test_gpu_parity's crowded movies): exact mode returns k."""
    rng = np.random.default_rng(21)
    emb, movie_of, centers = crowded(rng, 900, 384)
    src, dst = rng.integers(0, len(emb), 100), rng.integers(0, len(emb), 100)
    emb[dst] = emb[src]                                              # duplicate rows across movies
    fresh_index.load_embeddings(emb, movie_idx=movie_of)
    Q = centers[:4].astype(np.float32)
    _, _, _, short = fresh_index.knn_movies(Q, 10, 12)
    assert (short < 10).all()
    got = fresh_index.knn_movies_exact(Q, 10)
    assert got[3].tolist() == [10] * 4 and got[4] == 4
    check(got, emb, Q, movie_of, 10)
    Q2 = (centers[rng.integers(0, 900, 12)] + 0.2 * unit_rows(rng, 12, 384)).astype(np.float32)
    for k in (1, 10, 409, 4096):                                     # 4096 > 900 movies: every movie, once
        check(fresh_index.knn_movies_exact(Q2, k), emb, Q2, movie_of, k)


def test_ties_across_movies_follow_block_then_slot(fresh_index):
    rng = np.random.default_rng(3)
    n = 5000
    emb = unit_rows(rng, n, 384)
    movie_of = (np.arange(n) // 4).astype(np.int32)
    twins = [5, 1023, 1024, 2047, 2048, 3000, 4999]                  # one row in each of these movies is the same
    for r in twins:
        emb[r] = emb[100]
    fresh_index.load_embeddings(emb, movie_idx=movie_of)
    Q = np.stack([emb[100], emb[100] + 1e-3 * unit_rows(rng, 1, 384)[0]]).astype(np.float32)
    got = fresh_index.knn_movies_exact(Q, 20)
    check(got, emb, Q, movie_of, 20)
    rows = got[1][0, :len(twins) + 1].tolist()
    assert sorted(rows) == sorted(twins + [100])
    # equal distances: block ascending, then slot descending
    assert rows == sorted(rows, key=lambda r: (r // 1024, -(r % 1024)))


@pytest.mark.parametrize("use_fma", [False, True])
@pytest.mark.parametrize("dim", [384, 512, 100])
def test_widths_and_arithmetic(monkeypatch, dim, use_fma):
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(dim + use_fma)
    emb, movie_of, centers = crowded(rng, 700, dim)
    idx = _lib.Index(0)
    try:
        idx.set_fma(use_fma)
        idx.load_embeddings(emb, movie_idx=movie_of)
        Q = np.concatenate([centers[:3], unit_rows(rng, 3, dim)]).astype(np.float32)
        for k in (1, 10, 409):
            check(idx.knn_movies_exact(Q, k), emb, Q, movie_of, k, use_fma=use_fma)
    finally:
        idx.close()


def test_holes_orphans_and_shuffled_layout(fresh_index):
    """valid = 0 holes and movie_idx = -1 orphans never compete; a shuffled movie_idx takes the per-row atomic path;
    reloading the handle re-checks the layout."""
    rng = np.random.default_rng(8)
    emb, movie_of, centers = crowded(rng, 600, 384)
    n = len(emb)
    valid = (rng.random(n) > 0.15).astype(np.uint8)
    orphans = movie_of.copy()
    orphans[rng.random(n) < 0.1] = -1
    Q = np.concatenate([centers[:4], unit_rows(rng, 4, 384)]).astype(np.float32)
    # the hole rows keep their (finite) vectors: only `valid` takes them out
    fresh_index.load_embeddings(emb, valid=valid, movie_idx=orphans)
    for k in (1, 10, 700):
        check(fresh_index.knn_movies_exact(Q, k), emb, Q, orphans, k, valid=valid)
    shuffled = rng.permutation(600).astype(np.int32)[movie_of]      # runs stay contiguous but unsorted
    fresh_index.load_embeddings(emb, movie_idx=shuffled)
    for k in (1, 10, 700):
        check(fresh_index.knn_movies_exact(Q, k), emb, Q, shuffled, k)
    scattered = rng.permutation(movie_of).astype(np.int32)           # every movie spread over the corpus
    scattered[rng.random(n) < 0.05] = -1
    fresh_index.load_embeddings(emb, valid=valid, movie_idx=scattered)
    for k in (1, 10, 700):
        check(fresh_index.knn_movies_exact(Q, k), emb, Q, scattered, k, valid=valid)
    fresh_index.load_embeddings(emb, movie_idx=movie_of)             # sorted again
    check(fresh_index.knn_movies_exact(Q, 10), emb, Q, movie_of, 10)


def test_batch_sizes_and_query_chunks(monkeypatch):
    rng = np.random.default_rng(11)
    emb, movie_of, centers = crowded(rng, 400, 384)
    n_slots = 400
    idx = new_index(monkeypatch, budget=32 * 8 * n_slots)            # 32 queries per segmented-scan chunk
    try:
        idx.load_embeddings(emb, movie_idx=movie_of)
        Qall = (centers[rng.integers(0, 400, 256)] + 0.1 * unit_rows(rng, 256, 384)).astype(np.float32)
        for nq in (1, 2, 33, 256):
            Q = Qall[:nq]
            got = idx.knn_movies_exact(Q, 10)
            assert got[4] == nq
            check(got, emb, Q, movie_of, 10)
        assert idx.knn_movies_exact(Qall[:0], 10)[3].shape == (0,)
    finally:
        idx.close()


def test_staging_serves_full_queries_from_the_shortlist():
    """tc_mode 2 makes the tensor-core filter serve K' = 10 k: queries it gives k movies are final, the rest are
    gathered, take the segmented scan and are scattered back to their rows; both kinds match the contract."""
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(12)
    n_movies, dim, fat = 3000, 384, 5
    per = rng.integers(1, 30, n_movies)
    per[fat] = 400                                                   # one movie with 400 near-identical chunks
    movie_of = np.repeat(np.arange(n_movies, dtype=np.int32), per)
    centers = unit_rows(rng, n_movies, dim)
    spread = np.where(movie_of == fat, 0.02, 0.3).astype(np.float32)[:, None]
    emb = centers[movie_of] + spread * unit_rows(rng, len(movie_of), dim)
    emb = (emb / np.linalg.norm(emb, axis=1, keepdims=True)).astype(np.float32)
    Q = np.concatenate([centers[:8], unit_rows(rng, 24, dim)]).astype(np.float32)
    Q[:8] = emb[np.searchsorted(movie_of, np.arange(8))]            # on a movie's chunk: its neighbours crowd in
    short_at = [3, 17]
    Q[short_at] = centers[fat]            # its top 100 chunks are all the fat movie's: one movie, short of k = 10
    idx = _lib.Index(0)
    try:
        idx.set_tc_mode(2)
        idx.load_embeddings(emb, movie_idx=movie_of)
        _, _, _, first = idx.knn_movies(Q, 10, 100)
        assert first[short_at].tolist() == [1, 1]
        got = idx.knn_movies_exact(Q, 10)
        assert 2 <= got[4] < len(Q)                                  # the short queries took the scan, not all
        assert got[3].tolist() == [10] * len(Q)
        check(got, emb, Q, movie_of, 10)
        check(idx.knn_movies_exact(Q, 100), emb, Q, movie_of, 100)
        got = idx.knn_movies_exact(Q, 300)                            # 10 k > 2048: straight to the scan
        assert got[4] == len(Q)
        check(got, emb, Q, movie_of, 300)
    finally:
        idx.close()


def test_closing_a_handle_frees_its_exact_search_buffers():
    """Each call below fills a 512 MB [queries, movies] key buffer; closing the handle must give it back."""
    import torch
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(30)
    n = 2048
    emb = unit_rows(rng, n, 64)
    movie_of = np.arange(n, dtype=np.int32) * 64                     # 131 009 movie slots: 1 MB of keys per query
    Q = unit_rows(rng, 512, 64)

    def cycle():
        idx = _lib.Index(0)
        try:
            idx.load_embeddings(emb, movie_idx=movie_of)
            assert (idx.knn_movies_exact(Q, 5)[3] == 5).all()
        finally:
            idx.close()

    cycle()
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    for _ in range(8):
        cycle()
    free1 = torch.cuda.mem_get_info(0)[0]
    assert free0 - free1 < (3 << 29), f"{(free0 - free1) / 2**20:.0f} MB not returned after 8 handles"


def test_prefix_property_on_a_synthetic_corpus(gpu_index):
    """On a 120 k-movie synth corpus every query's exact list equals knn_movies' where that returned k movies and
    extends it where it returned fewer."""
    from rag_search_engine_b200 import synth
    s = synth.synth_embeddings(120_000, seed=7, distribution="clustered", n_centres=2000)
    emb = s.emb.numpy()
    movie_of = s.movie_of_chunk.numpy().astype(np.int32)
    Q = synth.synth_query_vectors(s.emb, 64, seed=5).numpy()
    gpu_index.load_embeddings(emb, movie_idx=movie_of)
    shorter = 0
    for k, kp in ((10, 20), (10, 100), (50, 100)):
        d0, r0, m0, c0 = gpu_index.knn_movies(Q, k, kp)
        d1, r1, m1, c1, _ = gpu_index.knn_movies_exact(Q, k)
        assert (c1 == k).all()
        for qi in range(len(Q)):
            c = int(c0[qi])
            shorter += c < k
            assert r1[qi, :c].tolist() == r0[qi, :c].tolist()
            assert m1[qi, :c].tolist() == m0[qi, :c].tolist()
            assert d1[qi, :c].view(np.uint32).tolist() == d0[qi, :c].view(np.uint32).tolist()
    assert shorter > 0
    check(gpu_index.knn_movies_exact(Q[:4], 50), emb, Q[:4], movie_of, 50)


def test_errors(fresh_index):
    from rag_search_engine_b200 import _lib
    q = np.zeros((1, 8), np.float32)
    with pytest.raises(_lib.RseError) as e:
        fresh_index.knn_movies_exact(q, 5)
    assert e.value.code == RSE_ERR_STATE
    rng = np.random.default_rng(1)
    emb = unit_rows(rng, 64, 8)
    fresh_index.load_embeddings(emb)                                 # no movie_idx
    with pytest.raises(_lib.RseError) as e:
        fresh_index.knn_movies_exact(q, 5)
    assert e.value.code == RSE_ERR_STATE and "movie_idx" in str(e.value)
    fresh_index.load_embeddings(emb, movie_idx=np.arange(64, dtype=np.int32))
    with pytest.raises(_lib.RseError) as e:
        fresh_index.knn_movies_exact(q, 0)
    assert e.value.code == RSE_ERR_INVALID
    with pytest.raises(_lib.RseError) as e:
        fresh_index.knn_movies_exact(q, 4097)
    assert e.value.code == _lib.RSE_ERR_UNSUPPORTED
    got = fresh_index.knn_movies_exact(q + 1, 4096)
    assert got[3].tolist() == [64]
