"""Corpora and queries at the edges of the fixed-point BM25 argument (see helpers/bm25_fx.py).

Each builder returns the corpus and, where it aims at an edge, what the model says about it, so that
test_bm25_fx_model.py can check the claim on the CPU and test_gpu_bm25_fixed_point.py can run the case.
Positions inside a range matter to the kernel: bm25_fx_kernel<512> reads the 7168 accumulators of a range as
uint4 vectors, vector v going to thread v % 512, so documents 0..127 of a range belong to warp 0."""
from __future__ import annotations

from dataclasses import dataclass, field

import numpy as np

from helpers import bm25_fx as fx
from helpers.bm25_fx import BM_RANGE, MAX_DOCS, Corpus


def pack(queries):
    tok_indptr = np.cumsum([0] + [len(q) for q in queries]).astype(np.int32)
    terms = np.array([t for q in queries for t in q], np.int32)
    return tok_indptr, terms


@dataclass
class Case:
    corpus: Corpus
    terms: dict = field(default_factory=dict)     # name -> term row
    info: dict = field(default_factory=dict)


# ----------------------------------------------------------------------------- zero contributions
def zero_small(n_docs: int = 20_000, seed: int = 1) -> Case:
    """U in every document, R in 3; dl 5..15.  At k1 = 1000 a posting of U has wq = 512 and idfx * wq < 0.5."""
    rng = np.random.default_rng(seed)
    dl = rng.integers(5, 16, n_docs).astype(np.uint32)
    r_docs = np.array([17, BM_RANGE + 5, n_docs - 1])
    z = Corpus.from_terms(n_docs, dl, [(np.arange(n_docs), 1), (r_docs, [2, 1, 3])])
    return Case(z, {"U": 0, "R": 1}, {"r_docs": r_docs})


def zero_long_doc(n_docs: int = 1000) -> Case:
    """1000 documents of length 10 and one 666 times as long; R (df = 5, idf 5.2) is in it.  At k1 = 4000 that
    posting's weight rounds to wq = 0."""
    dl = np.full(n_docs, 10, np.uint32)
    long_doc = 500
    dl[long_doc] = 6660
    r_docs = np.array([3, 200, long_doc, 777, 998])
    z = Corpus.from_terms(n_docs, dl, [(np.arange(n_docs), 1), (r_docs, 1)])
    return Case(z, {"U": 0, "R": 1}, {"long_doc": long_doc, "r_docs": r_docs})


def zero_largest(n_docs: int = MAX_DOCS) -> Case:
    """The largest corpus rse_load_bm25 accepts, built directly in numpy: dl = 2 nearly everywhere, U in every
    document, R (df = 3) in a document of 1.3 M tokens, and S, a term every 99 991 documents with varied lengths,
    so that a range group (64 ranges: the group count is capped at 32) holds several of its postings."""
    dl = np.full(n_docs, 2, np.uint32)
    long_doc = 7_000_003
    dl[long_doc] = 1_300_000
    s_docs = np.arange(11, n_docs, 99_991)
    dl[s_docs] = 1 + (np.arange(len(s_docs)) % 5).astype(np.uint32)
    r_docs = np.array([5, long_doc, n_docs - 1])
    indptr = np.array([0, n_docs, n_docs + 3, n_docs + 3 + len(s_docs)], np.int64)
    doc = np.concatenate([np.arange(n_docs, dtype=np.uint32), r_docs.astype(np.uint32), s_docs.astype(np.uint32)])
    tf = np.ones(len(doc), np.uint32)
    tf[n_docs + 3:] = 1 + (np.arange(len(s_docs)) % 3).astype(np.uint32)
    avgdl = float(dl.astype(np.float64).sum()) / n_docs
    z = Corpus(indptr, doc, tf, dl, n_docs, avgdl)
    return Case(z, {"U": 0, "R": 1, "S": 2}, {"long_doc": long_doc, "r_docs": r_docs})


# ----------------------------------------------------------------------------- margin
def warp_slot(i: int, k: int) -> int:
    """Offset inside a range of the i-th of k documents meant to set the first range's threshold: one per warp for
    k <= 16 (one maximum per warp counts), two per warp (distinct threads) for k <= 32 (two count)."""
    return 128 * i if k <= 16 else 128 * (i // 2) + 64 * (i % 2)


def margin_case(k: int, ntok: int, same_group: bool = False, n_docs: int = 20_000, k1: float = 1.5, b: float = 0.75,
                seed: int = 3) -> Case:
    """The fixed-point order is the reverse of the exact order at place k, by far more than kFxMargin.

    Documents T hold the terms A_1..A_h, documents I the terms B_1..B_h, h = ntok / 2; df(A) = k < df(B) = k + 8
    (8 long filler documents in range 2 hold B too).  dl_T and dl_I are chosen so that every T has a higher exact score
    than every I while its fixed-point sum is lower by as much as the rounding allows.  The query is
    [A_1..A_h, B_1..B_h].
      * same_group=False: k documents T in range 0 and k documents I in range 1, i.e. in two range groups: only
        bm25_fx_finish_kernel sees both, and its margin decides.  The answer is the k documents T.
      * same_group=True: all in range 0, i.e. in one group, so bm25_fx_body's margin decides: k - 1 documents C that
        hold every term and are far above everything, one T (the document at place k) and one I.  C and I take k warp
        slots, so the k-th warp maximum of the first range is I's sum and the threshold is I's sum minus the margin;
        T shares thread 0 with slot 0.  T is beaten by k documents by more than 40 units but only by the k - 1
        documents C by more than the per-query margin.  The answer is C and T."""
    assert ntok % 2 == 0 and 1 <= k <= 32
    h = ntok // 2
    rng = np.random.default_rng(seed)
    # documents of ~10^6 tokens: one token more or less moves a score by ~1e-6 of itself, a few fixed-point units
    dl = rng.integers(900_000, 1_100_000, n_docs).astype(np.uint32)
    if same_group:
        c_docs = np.array([warp_slot(i, k) for i in range(k - 1)], np.int64)
        i_docs = np.array([warp_slot(k - 1, k)])
        t_docs = np.array([2048 + warp_slot(0, k)])
        dl[c_docs] = 1000
    else:
        c_docs = np.zeros(0, np.int64)
        t_docs = np.arange(k) * 3                          # range 0
        i_docs = BM_RANGE + np.arange(k) * 3               # range 1
    f_docs = 2 * BM_RANGE + np.arange(8) * 5               # range 2
    dl[f_docs] = 50_000_000
    nt, ni = len(t_docs), len(i_docs)
    wq4, fxs = fx.scales(k1, b, n_docs)
    idf_a = float(fx.idf(k, n_docs))
    idf_b = float(fx.idf(k + 8, n_docs))
    base = dl.astype(np.float64).sum() - dl[t_docs].sum() - dl[i_docs].sum()
    # dl_T where idf_a * w(dl_T) = idf_b * w(10^6), then +-200 tokens around both
    avg0 = base / (n_docs - nt - ni)
    w_target = idf_b / idf_a * float(fx.weights(1, fx.normk(1_000_000, k1, b, avg0), k1))
    d_star = avg0 / b * (((k1 + 1.0) / w_target - 1.0) / k1 - (1.0 - b))
    dT, dI = np.meshgrid(np.round(d_star) + np.arange(-200, 200.0), 1_000_000 + np.arange(-200, 200.0), indexing="ij")
    avgdl = (base + nt * dT + ni * dI) / n_docs
    wT = fx.weights(1, fx.normk(dT, k1, b, avgdl), k1)
    wI = fx.weights(1, fx.normk(dI, k1, b, avgdl), k1)
    eT = np.zeros_like(wT)
    eI = np.zeros_like(wI)
    for _ in range(h):                                     # the reference's sum in token order
        eT = eT + idf_a * wT
    for _ in range(h):
        eI = eI + idf_b * wI
    fT = h * fx.contribution(fx.idfx(idf_a, fxs, wq4), fx.wq(wT, wq4))
    fI = h * fx.contribution(fx.idfx(idf_b, fxs, wq4), fx.wq(wI, wq4))
    inv = np.where(eT > eI, fI - fT, np.iinfo(np.int64).min)
    i, j = np.unravel_index(np.argmax(inv), inv.shape)
    dl[t_docs] = int(dT[i, j])
    dl[i_docs] = int(dI[i, j])
    a_docs = np.sort(np.concatenate([c_docs, t_docs]))
    b_docs = np.sort(np.concatenate([c_docs, i_docs, f_docs]))
    post = [(a_docs, 1)] * h + [(b_docs, 1)] * h
    others = np.setdiff1d(np.arange(n_docs), np.concatenate([c_docs, t_docs, i_docs, f_docs]))
    post.append((others, 1))                               # Z: every other document, not in any query
    c = Corpus.from_terms(n_docs, dl, post)
    query = list(range(2 * h))
    return Case(c, {"Z": 2 * h}, {"query": query, "t_docs": t_docs, "i_docs": i_docs, "c_docs": c_docs,
                                  "answer": np.sort(np.concatenate([c_docs, t_docs])), "k": k, "k1": k1, "b": b})


# ----------------------------------------------------------------------------- capacities
def tie_group(n: int, splits, n_docs: int = 20_000, k: int = 10, seed: int = 4) -> Case:
    """n documents holding R whose fixed-point sums span just less than the per-query margin: half exact ties
    (dl = 10^7), half near-ties with distinct exact scores (dl from 10^7 + 1 up to the longest length that keeps the
    spread of the sums below the margin, on an average of ~10^7).  No document is beaten by another by more than the
    margin, so all n are finalists.  `splits` gives how many sit in each of the ranges 0, 1, 2.  Every other document
    holds Z."""
    assert sum(splits) == n
    rng = np.random.default_rng(seed)
    dl = rng.integers(9_900_000, 10_100_000, n_docs).astype(np.uint32)
    docs = np.concatenate([r * BM_RANGE + 1 + np.arange(m) * 11 for r, m in enumerate(splits)])
    others = np.setdiff1d(np.arange(n_docs), docs)
    near = docs[1::2]

    def build(span: int):
        d = dl.copy()
        d[docs[0::2]] = 10_000_000
        d[near] = 10_000_001 + np.round(np.linspace(0, span, len(near))).astype(np.uint32)
        c = Corpus.from_terms(n_docs, d, [(docs, 1), (others, 1)])
        fs, _, _ = fx.fixed_sums(c, [0])
        return c, int(fs[docs].max() - fs[docs].min())

    wq4, fxs = fx.scales(1.5, 0.75, n_docs)
    margin = fx.margin(fx.query_idf(build(0)[0], [0]), fxs, wq4)
    lo, hi = 0, 1_000_000                                  # largest span whose spread stays below the margin
    while hi - lo > 1:
        mid = (lo + hi) // 2
        lo, hi = (mid, hi) if build(mid)[1] < margin else (lo, mid)
    c, spread = build(lo)
    return Case(c, {"R": 0, "Z": 1}, {"docs": docs, "k": k, "spread": spread})


def candidate_range(n_cand: int, n_docs: int = 20_000, k: int = 10, seed: int = 5) -> Case:
    """Range 0 holds k top documents (exact and near ties) in warp 0's slots (offsets < 128) and n_cand - k low
    documents spread over the other warps, all holding R.  With m = 1 maximum per warp the threshold of the first
    range is the low sum minus the margin, so all n_cand documents become candidates: n_cand = 256 fits the
    candidate list, is compacted (>= 128) down to the top k and finished; 257 overflows it."""
    rng = np.random.default_rng(seed)
    dl = rng.integers(9_900_000, 10_100_000, n_docs).astype(np.uint32)
    top = np.arange(k) * 7                                   # offsets 0..63: warp 0
    low = 128 + np.arange(n_cand - k) * (1920 // (n_cand - k))   # offsets 128..2047: warps 1..15
    dl[top[0::2]] = 10_000_000
    dl[top[1::2]] = 10_000_001
    dl[low] = 300_000_000
    docs = np.sort(np.concatenate([top, low]))
    others = np.setdiff1d(np.arange(n_docs), docs)
    c = Corpus.from_terms(n_docs, dl, [(docs, 1), (others, 1)])
    return Case(c, {"R": 0, "Z": 1}, {"top": top, "low": low, "k": k})


def compaction_boundary(n_first: int, n_second: int = 150, k: int = 10, seed: int = 7) -> Case:
    """kBsCompactAt = 128 candidates after one range.  64 ranges: bm25_run caps the group count at 32, so a group
    holds two ranges and range 1 is scanned with the threshold range 0 left.  Range 0 holds k top documents in warp
    0 and n_first - k low ones over warps 1..15 (as in candidate_range); range 1 holds n_second more low ones.
    n_first = 128 is compacted after range 0, the threshold rises above the low sum and range 1 adds nothing: the query
    is finished.  n_first = 127 is not; range 1's low documents all join and overflow kBsCandCap = 256."""
    n_docs = 64 * BM_RANGE
    base = candidate_range(n_first, n_docs=n_docs, k=k, seed=seed)
    top, low = base.info["top"], base.info["low"]
    low2 = BM_RANGE + np.arange(n_second) * 13
    dl = base.corpus.dl.copy()
    dl[low2] = 300_000_000
    docs = np.sort(np.concatenate([top, low, low2]))
    others = np.setdiff1d(np.arange(n_docs), docs)
    c = Corpus.from_terms(n_docs, dl, [(docs, 1), (others, 1)])
    return Case(c, {"R": 0, "Z": 1}, {"top": top, "low": np.concatenate([low, low2]), "k": k})


# ----------------------------------------------------------------------------- format edges
def near_2p31(n_docs: int = 20_000) -> Case:
    """X (df = 1, the largest idf) in one document with tf = 2^31 and b = 0, so w is as close to k1 + 1 as a
    weight gets, at the largest k1 the path accepts for this N: 16 tokens of X sum to just below 2^31."""
    k1 = fx.largest_k1(n_docs)
    dl = np.full(n_docs, 40, np.uint32)
    x_doc = 4321
    dl[x_doc] = 2**31
    others = np.setdiff1d(np.arange(n_docs), [x_doc])
    c = Corpus.from_terms(n_docs, dl, [(np.array([x_doc]), 2**31), (others, 1)])
    return Case(c, {"X": 0, "Z": 1}, {"k1": k1, "b": 0.0, "x_doc": x_doc})


def range_edges(n_docs: int, seed: int = 6) -> Case:
    """E holds the documents at offsets 0 and 7167 of every range and the last document; F 40 random ones."""
    rng = np.random.default_rng(seed)
    dl = rng.integers(5, 60, n_docs).astype(np.uint32)
    nr = (n_docs + BM_RANGE - 1) // BM_RANGE
    e_docs = np.unique(np.concatenate([np.arange(nr) * BM_RANGE, np.arange(nr) * BM_RANGE + BM_RANGE - 1,
                                       [n_docs - 1]]))
    e_docs = e_docs[e_docs < n_docs]
    f_docs = np.sort(rng.choice(n_docs, 40, replace=False))               # few: no cap can trip
    c = Corpus.from_terms(n_docs, dl, [(e_docs, 1 + np.arange(len(e_docs)) % 4), (f_docs, 1 + np.arange(40) % 3)])
    return Case(c, {"E": 0, "F": 1}, {"e_docs": e_docs})


def random_corpus(n_docs: int, vocab: int, seed: int, mean_len: int = 30) -> Corpus:
    """Random documents over a Zipf-like vocabulary, tf from repeated draws."""
    rng = np.random.default_rng(seed)
    p = 1.0 / np.arange(1, vocab + 1) ** 1.1
    p /= p.sum()
    dl = np.maximum(1, rng.poisson(mean_len, n_docs)).astype(np.uint32)
    doc_of = np.repeat(np.arange(n_docs), dl)
    term_of = rng.choice(vocab, len(doc_of), p=p)
    key = np.unique(term_of.astype(np.int64) * n_docs + doc_of, return_counts=True)
    t, d = key[0] // n_docs, key[0] % n_docs
    indptr = np.zeros(vocab + 1, np.int64)
    np.add.at(indptr, t + 1, 1)
    return Corpus(np.cumsum(indptr), d.astype(np.uint32), key[1].astype(np.uint32), dl, n_docs,
                  float(dl.astype(np.float64).sum()) / n_docs)


def with_mass_tie(c: Corpus, docs) -> tuple[Corpus, int]:
    """c plus one term M in `docs`, whose lengths are set equal: identical exact scores for a query [M]."""
    dl = c.dl.copy()
    dl[docs] = 25
    indptr = np.concatenate([c.indptr, [c.indptr[-1] + len(docs)]])
    return (Corpus(indptr, np.concatenate([c.doc, np.asarray(docs, np.uint32)]),
                   np.concatenate([c.tf, np.ones(len(docs), np.uint32)]), dl, c.n_movies,
                   float(dl.astype(np.float64).sum()) / len(dl)), len(indptr) - 2)
