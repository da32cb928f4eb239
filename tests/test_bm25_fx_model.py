"""The CPU model of fixed-point BM25 (helpers/bm25_fx.py) against hand-worked values and the eligibility rules of
bm25_run, and every construction of test_gpu_bm25_fixed_point.py against the edge it claims to reach."""
import math

import numpy as np
import pytest

from helpers import bm25_fx as fx
from helpers import bm25_fx_cases as cases


# ----------------------------------------------------------------------------- the model itself
def test_scales_by_hand():
    # default k1: k1 + 1 = 2.5 = 0.625 * 2^2 → wq4 = 2^17; max sum 2.5 * ln(600 002) * 16 + 1 = 533.2 < 2^10 → 2^21
    assert fx.scales(1.5, 0.75, 600_000) == (2.0**17, 2.0**21)
    # k1 + 1 a power of two: (k1 + 1) * wq4 = 2^19 exactly
    assert fx.scales(1.0, 0.75, 1000)[0] == 2.0**18
    assert fx.scales(0.0, 0.75, 1000)[0] == 2.0**19
    assert fx.scales(3.0, 0.75, 1000)[0] == 2.0**17
    # k1 = 1000, 20 000 documents: 1001 * ln(20 002) * 16 + 1 = 158 606 < 2^18 → 2^13; 1001 < 2^10 → wq4 = 2^9
    assert fx.scales(1000.0, 0.75, 20_000) == (512.0, 8192.0)


def test_eligibility_boundaries():
    n = 20_000
    assert fx.scales(1.5, 0.0, n)[1] > 0 and fx.scales(1.5, 1.0, n)[1] > 0
    assert fx.scales(1.5, math.nextafter(1.0, 2.0), n) == (0.0, 0.0)
    assert fx.scales(1.5, -0.0, n)[1] > 0 and fx.scales(1.5, -1e-300, n) == (0.0, 0.0)
    assert fx.scales(-1e-300, 0.75, n) == (0.0, 0.0) and fx.scales(0.0, 0.75, n)[1] > 0
    # the 4-byte stream needs k1 + 1 < 2^20
    assert fx.scales(2.0**20 - 1.5, 0.75, n)[0] > 0 and fx.scales(2.0**20 - 1.0, 0.75, n)[0] == 0.0
    # the path needs fx_scale >= 2^12
    k1 = fx.largest_k1(n)
    assert fx.scales(k1, 0.75, n)[1] == 4096.0
    assert fx.scales(k1 + 1e-6, 0.75, n)[1] == 0.0
    assert fx.eligible(32, 16, 1.5, 0.75, n) and not fx.eligible(33, 16, 1.5, 0.75, n)
    assert not fx.eligible(10, 17, 1.5, 0.75, n) and not fx.eligible(10, 1, k1 + 1e-6, 0.75, n)


def test_weight_word_and_contribution_by_hand():
    assert float(fx.idf(1, 3)) == math.log(2.5 / 1.5 + 1.0)
    assert fx.wq(1.0, 2.0**17).item() == 131072
    assert fx.wq(2.5, 2.0**18).item() == fx.WQ_MAX                       # clamped at the top
    assert fx.wq(1e-9, 2.0**17).item() == 1 and fx.wq(1e-9, 2.0**17, zero_floor=False).item() == 0
    assert fx.wq(0.0, 2.0**17).item() == 0                                # tf = 0 stays "adds nothing"
    assert fx.wq(2.5 / 2**17, 2.0**17).item() == 2                       # half to even
    assert fx.contribution(0.3, 1).item() == 1 and fx.contribution(0.3, 1, zero_floor=False).item() == 0
    assert fx.contribution(1e-9, 1).item() == 1 and fx.contribution(3.0, 1).item() == 3   # rounded up
    assert fx.contribution(2.5, 1, zero_floor=False).item() == 2 and fx.contribution(3.5, 1, zero_floor=False).item() == 4
    assert fx.contribution(1e6, 0).item() == 0


def test_margin_by_hand():
    s = 16.0                                                              # fx_scale / wq4_scale at 600 k, default k1
    assert fx.margin([], 2.0**21, 2.0**17) == fx.FX_MARGIN
    assert fx.margin([100 / s], 2.0**21, 2.0**17) == 2 * 101 + 8
    assert fx.margin([100 / s, 0.1 / s, 0.1 / s], 2.0**21, 2.0**17) == 2 * 102 + 8   # 100.5 + 0.6 + 0.6 -> 102
    assert fx.margin([0.0] * 16, 2.0**21, 2.0**17) == fx.FX_MARGIN       # 2 * 8 + 8


def test_fixed_sums_are_within_the_bound_on_a_random_corpus():
    """A sum lies within [-sum_t idfx_t, sum_t (idfx_t + 1)) of its exact value (+ a little for the double sum), so two
    sums disagree with the exact order by less than the margin; every touched document has a non-zero sum."""
    c = cases.random_corpus(5000, 800, seed=1)
    rng = np.random.default_rng(2)
    for k1, b in [(1.5, 0.75), (0.0, 0.75), (1000.0, 0.75), (3000.0, 1.0), (1.2, 0.0)]:
        wq4, fxs = fx.scales(k1, b, c.n_movies)
        for _ in range(20):
            q = rng.integers(0, 800, int(rng.integers(1, 17))).tolist()
            fs, ex, touched = fx.fixed_sums(c, q, k1, b)
            sx = sum(v * fxs / wq4 for v in fx.query_idf(c, q))
            err = fs[touched] - ex[touched] * fxs
            slop = 1e-6 * fxs
            assert (err >= -sx - slop).all() and (err < sx + len(q) + slop).all()
            assert 2 * sx + len(q) <= fx.margin(fx.query_idf(c, q), fxs, wq4)
            assert (fs[touched] >= 1).all() and (fs[~touched] == 0).all()
            assert fs.max(initial=0) < 2**31


# ----------------------------------------------------------------------------- the constructions
def test_zero_small_reaches_zero_contributions():
    case = cases.zero_small()
    c, U, R = case.corpus, case.terms["U"], case.terms["R"]
    fs, ex, touched = fx.fixed_sums(c, [U], 1000.0, 0.75, zero_floor=False)
    assert touched.all() and (ex > 0).all() and (fs == 0).all()              # before: every sum 0
    wq4, _ = fx.scales(1000.0, 0.75, c.n_movies)
    assert (fx.wq(fx.weights(1, fx.normk(c.dl, 1000.0, 0.75, c.avgdl), 1000.0), wq4) > 0).all()
    fs, _, _ = fx.fixed_sums(c, [U], 1000.0, 0.75)
    assert (fs == 1).all()                                                   # now: a mass tie at 1
    fs, _, _ = fx.fixed_sums(c, [U, R], 1000.0, 0.75, zero_floor=False)
    assert np.count_nonzero(fs) == 3                                         # fewer than k = 10 candidates


def test_zero_long_doc_reaches_a_zero_weight_word():
    case = cases.zero_long_doc()
    c, R, d = case.corpus, case.terms["R"], case.info["long_doc"]
    assert abs(float(fx.idf(5, c.n_movies)) - 5.2) < 0.01 and c.dl[d] == 666 * c.dl[0]
    wq4, _ = fx.scales(4000.0, 0.75, c.n_movies)
    w = fx.weights(1, fx.normk(c.dl[d], 4000.0, 0.75, c.avgdl), 4000.0)
    assert fx.wq(w, wq4, zero_floor=False) == 0 and fx.wq(w, wq4) == 1
    fs, _, touched = fx.fixed_sums(c, [R], 4000.0, 0.75, zero_floor=False)
    assert touched.sum() == 5 and np.count_nonzero(fs) == 4
    fs, _, _ = fx.fixed_sums(c, [R], 4000.0, 0.75)
    assert np.count_nonzero(fs) == 5


def test_zero_largest_reaches_zero_contributions_at_the_default_parameters():
    case = cases.zero_largest()
    c, U, R = case.corpus, case.terms["U"], case.terms["R"]
    assert c.n_docs == fx.MAX_DOCS == 14_680_064
    fs, _, touched = fx.fixed_sums(c, [U], zero_floor=False)
    assert touched.all() and not fs.any()
    wq4, fxs = fx.scales(1.5, 0.75, c.n_movies)
    most = fx.wq(fx.weights(1, fx.normk(2, 1.5, 0.75, c.avgdl), 1.5), wq4)
    assert most == 133_622
    fs, _, touched = fx.fixed_sums(c, [R], zero_floor=False)
    assert touched.sum() == 3 and np.count_nonzero(fs) == 2 and fs[case.info["long_doc"]] == 0
    assert abs(float(fx.idf(3, c.n_movies)) - 15.2) < 0.1
    # the group count is capped: 2048 ranges in 32 groups of 64
    assert (c.n_docs + fx.BM_RANGE - 1) // fx.BM_RANGE == 2048 > 64 * fx.MAX_GROUPS - 1


def warp_of(offsets):
    """Warp of bm25_fx_kernel<512> whose threads read these range offsets (vector v = offset / 4 -> thread v % 512)."""
    return (np.asarray(offsets) // 4 % 512) // 32


@pytest.mark.parametrize("same_group", [False, True])
@pytest.mark.parametrize("ntok", [2, 16])
@pytest.mark.parametrize("k", [1, 10, 32])
def test_margin_case_inverts_the_order_at_place_k(k, ntok, same_group):
    case = cases.margin_case(k, ntok, same_group)
    c, q = case.corpus, case.info["query"]
    t, i, cd = case.info["t_docs"], case.info["i_docs"], case.info["c_docs"]
    fs, ex, touched = fx.fixed_sums(c, q)
    assert ex[t].min() > ex[i].max()                                        # T above I exactly...
    inversion = int(fs[i].min() - fs[t].max())
    assert inversion > fx.FX_MARGIN                                          # ...and more than 40 units below in fixed point
    assert set(fx.exact_order(ex, touched)[:k].tolist()) == set(case.info["answer"].tolist())
    wq4, fxs = fx.scales(1.5, 0.75, c.n_movies)
    margin = fx.margin(fx.query_idf(c, q), fxs, wq4)
    assert inversion < margin                                                # the per-query margin covers it
    if ntok == 16:                                                           # only the sum over all 16 tokens does
        assert inversion > fx.margin(fx.query_idf(c, q[:1] + q[8:9]), fxs, wq4)
    nr = (c.n_docs + fx.BM_RANGE - 1) // fx.BM_RANGE
    assert nr == 3                                                           # one range per group (ng = nr)
    if not same_group:
        # T and I in two groups: only the finish kernel compares them
        assert set((t // fx.BM_RANGE).tolist()) == {0} and set((i // fx.BM_RANGE).tolist()) == {1}
        assert 2 * k <= fx.FX_RESCORE_CAP
        return
    # one group: T (place k) is beaten by k documents by more than 40 units, by only the k - 1 documents C by more
    # than the per-query margin, so bm25_fx_body's compaction and threshold decide whether it stays
    group = np.nonzero(touched & (np.arange(c.n_docs) < fx.BM_RANGE))[0]
    assert set(group.tolist()) == set(cd.tolist()) | set(t.tolist()) | set(i.tolist())
    assert len(group) == k + 1 <= fx.FX_FINAL_CAP
    d = t[0]
    assert np.count_nonzero(fs[group] > fs[d] + fx.FX_MARGIN) == k
    assert np.count_nonzero(fs[group] > fs[d] + margin) == k - 1
    # the k-th largest warp maximum of the first range is I's sum: C and I take k warp slots, distinct threads
    slots = np.concatenate([cd, i])
    thread = slots // 4 % 512
    assert len(np.unique(thread)) == k and (d // 4 % 512) == thread[0]
    per_warp = np.bincount(warp_of(slots), minlength=16)
    assert per_warp.max() <= (1 if k <= 16 else 2)
    assert (fs[cd] > fs[i].max()).all() if k > 1 else True


@pytest.mark.parametrize("n,splits", [(48, (48, 0, 0)), (49, (49, 0, 0)), (96, (32, 32, 32)), (97, (33, 32, 32))])
def test_tie_groups_span_just_less_than_the_margin(n, splits):
    case = cases.tie_group(n, splits)
    c, R, docs = case.corpus, case.terms["R"], case.info["docs"]
    fs, ex, touched = fx.fixed_sums(c, [R])
    assert touched.sum() == n and set(np.nonzero(touched)[0].tolist()) == set(docs.tolist())
    wq4, fxs = fx.scales(1.5, 0.75, c.n_movies)
    margin = fx.margin(fx.query_idf(c, [R]), fxs, wq4)
    spread = int(fs[docs].max() - fs[docs].min())
    step = fx.idfx(fx.query_idf(c, [R])[0], fxs, wq4)                     # the sum moves by idfx per unit of wq
    assert spread == case.info["spread"] and margin - step <= spread < margin   # all are finalists, the last one barely
    assert len(np.unique(ex[docs])) == n // 2 + 1                            # exact ties and near-ties
    assert len(np.unique(ex[docs[0::2]])) == 1
    per_range = np.bincount(docs // fx.BM_RANGE, minlength=3)
    assert tuple(per_range.tolist()) == splits and per_range.max() <= fx.FX_FINAL_CAP + 1


@pytest.mark.parametrize("n_cand", [256, 257])
def test_candidate_range_compacts_to_the_top(n_cand):
    case = cases.candidate_range(n_cand)
    c, R, top, low = case.corpus, case.terms["R"], case.info["top"], case.info["low"]
    fs, ex, touched = fx.fixed_sums(c, [R])
    assert touched.sum() == n_cand and (np.nonzero(touched)[0] < fx.BM_RANGE).all()
    wq4, fxs = fx.scales(1.5, 0.75, c.n_movies)
    m = fx.margin(fx.query_idf(c, [R]), fxs, wq4)
    assert fs[top].max() - fs[top].min() <= m and fs[top].min() > fs[low].max() + m   # compaction keeps exactly the top
    assert len(np.unique(fs[low])) == 1 and len(np.unique(ex[top])) == 2
    assert (warp_of(top) == 0).all()
    lw = warp_of(low)
    assert lw.min() >= 1 and len(np.unique(lw)) >= case.info["k"]          # the k-th warp maximum is a low document


@pytest.mark.parametrize("n_first", [127, 128])
def test_compaction_boundary_after_one_range(n_first):
    case = cases.compaction_boundary(n_first)
    c, R, top, low = case.corpus, case.terms["R"], case.info["top"], case.info["low"]
    assert (c.n_docs + fx.BM_RANGE - 1) // fx.BM_RANGE == 64 == 2 * fx.MAX_GROUPS   # two ranges per group
    fs, ex, touched = fx.fixed_sums(c, [R])
    docs = np.nonzero(touched)[0]
    assert np.count_nonzero(docs < fx.BM_RANGE) == n_first and np.count_nonzero(docs >= 2 * fx.BM_RANGE) == 0
    assert n_first + np.count_nonzero(docs >= fx.BM_RANGE) > fx.CAND_CAP        # without compaction range 1 overflows
    wq4, fxs = fx.scales(1.5, 0.75, c.n_movies)
    m = fx.margin(fx.query_idf(c, [R]), fxs, wq4)
    assert fs[top].min() > fs[low].max() + m and len(np.unique(fs[low])) == 1
    assert (warp_of(top) == 0).all() and len(np.unique(warp_of(low[low < fx.BM_RANGE]))) >= case.info["k"]


def test_near_2p31_sum():
    case = cases.near_2p31()
    c, X, k1, b = case.corpus, case.terms["X"], case.info["k1"], case.info["b"]
    assert fx.eligible(10, 16, k1, b, c.n_movies) and not fx.eligible(10, 17, k1, b, c.n_movies)
    assert not fx.eligible(10, 16, k1 + 1e-6, b, c.n_movies)
    assert c.df[X] == 1 and fx.idf(1, c.n_movies) == fx.idf(c.df, c.n_movies).max()
    fs, _, _ = fx.fixed_sums(c, [X] * 16, k1, b)
    s = int(fs[case.info["x_doc"]])
    assert 2**31 - 2**27 <= s < 2**31


def test_parameter_edges_of_the_weight_word():
    c = cases.random_corpus(30_000, 20_000, seed=12)
    wq4, _ = fx.scales(0.0, 0.75, c.n_movies)
    w = fx.weights(c.tf, fx.normk(c.dl[c.doc], 0.0, 0.75, c.avgdl), 0.0)
    assert (w == 1.0).all() and (fx.wq(w, wq4) == fx.WQ_MAX).all()           # k1 = 0 clamps every weight
    df = c.df
    assert ((df >= 1) & (df <= 8)).sum() > 1000                              # enough rare terms for the queries


@pytest.mark.parametrize("n_docs", [2 * fx.BM_RANGE, 2 * fx.BM_RANGE + 1])
def test_range_edges_hold_the_edge_documents(n_docs):
    case = cases.range_edges(n_docs)
    e = set(case.info["e_docs"].tolist())
    assert {0, fx.BM_RANGE - 1, fx.BM_RANGE, 2 * fx.BM_RANGE - 1, n_docs - 1} <= e
    assert case.corpus.df[case.terms["F"]] == 40


def test_chunk_queries():
    c0 = cases.random_corpus(30_000, 20_000, seed=12)
    c, M = cases.with_mass_tie(c0, np.arange(0, 3000))
    fs, _, _ = fx.fixed_sums(c, [M])
    assert (fs[:3000] == fs[0]).all() and np.count_nonzero(fs) == 3000 > fx.CAND_CAP
