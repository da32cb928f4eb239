"""CPU model of the fixed-point BM25 arithmetic (csrc/bm25.cuh K6''/K7'', csrc/rse.cu bm25_stage / bm25_run).

It restates four pieces of the library, nothing of its control flow:
  * ``scales``: wq4_scale, fx_scale and whether the fixed-point path is eligible, as ``bm25_run`` decides them;
  * ``idf``: as ``bm25_stage`` computes it (keyword_search.py:224);
  * ``weights`` / ``wq`` / ``contribution``: the per-posting weight, its 19-bit word and the integer each posting adds,
    as ``bm25_weight_kernel`` and ``item_apply`` compute them;
  * ``margin``: the per-query margin of ``bm25_fx_body`` and ``bm25_fx_finish_kernel``.
The scales are powers of two and the sums are integers, so ``fixed_sums`` gives each document's fixed-point sum
exactly.  ``zero_floor=False`` models the arithmetic before a posting could no longer add 0: a weight word rounded
to nearest without a floor of 1, and a contribution rounded to nearest instead of up.
The tests use the model to build inputs at the edges of the exactness argument and to assert that they reach them.
"""
from __future__ import annotations

import math
from dataclasses import dataclass

import numpy as np

BM_RANGE = 7168                     # kBmRange: documents per range
MAX_RANGES = 2048                   # rse_load_bm25 refuses more
MAX_DOCS = MAX_RANGES * BM_RANGE    # 14 680 064
MAX_TOKENS = 16                     # kBsMaxTok
MAX_K = 32                          # the streaming path serves k <= 32
FX_MARGIN = 40                      # kFxMargin: floor of the per-query margin
FX_FINAL_CAP = 48                   # kFxFinalCap: finalists one range group hands over
FX_RESCORE_CAP = 96                 # kFxRescoreCap: documents the finish kernel re-scores
CAND_CAP = 256                      # kBsCandCap: candidates of one group
COMPACT_AT = 128                    # kBsCompactAt
MAX_GROUPS = 32                     # kBsMaxGroups
WQ_MAX = 0x7FFFF                    # 19-bit weight word
CHUNK = 4096                        # queries per launch in bm25_run


@dataclass
class Corpus:
    """CSR postings as ``Index.load_bm25`` and ``oracle.bm25_batch`` take them."""
    indptr: np.ndarray     # int64 [n_terms + 1]
    doc: np.ndarray        # uint32 [n_postings], ascending inside a term
    tf: np.ndarray         # uint32 [n_postings]
    dl: np.ndarray         # uint32 [n_docs]
    n_movies: int
    avgdl: float

    @property
    def df(self) -> np.ndarray:
        return np.diff(self.indptr).astype(np.int64)

    @property
    def n_docs(self) -> int:
        return len(self.dl)

    def args(self):
        return self.indptr, self.doc, self.tf, self.df, self.dl, self.n_movies, self.avgdl

    @staticmethod
    def from_terms(n_docs: int, dl, term_postings, n_movies: int | None = None, avgdl: float | None = None) -> "Corpus":
        """term_postings: one (docs, tfs) pair per term row (docs strictly ascending)."""
        dl = np.ascontiguousarray(dl, np.uint32)
        assert len(dl) == n_docs
        indptr = np.zeros(len(term_postings) + 1, np.int64)
        docs, tfs = [], []
        for t, (d, f) in enumerate(term_postings):
            d = np.asarray(d, np.uint32)
            f = np.broadcast_to(np.asarray(f, np.uint32), d.shape)
            assert (np.diff(d.astype(np.int64)) > 0).all()
            docs.append(d); tfs.append(np.ascontiguousarray(f))
            indptr[t + 1] = indptr[t] + len(d)
        if avgdl is None:
            avgdl = float(dl.astype(np.float64).sum()) / n_docs
        return Corpus(indptr, np.concatenate(docs) if docs else np.zeros(0, np.uint32),
                      np.concatenate(tfs) if tfs else np.zeros(0, np.uint32), dl,
                      n_docs if n_movies is None else n_movies, float(avgdl))


def scales(k1: float, b: float, n_movies: int) -> tuple[float, float]:
    """(wq4_scale, fx_scale) of bm25_run; 0.0 where the 4-byte stream / the fixed-point path does not exist."""
    k1p1 = k1 + 1.0
    wq4 = 0.0
    if k1 >= 0.0 and 0.0 <= b <= 1.0 and k1p1 < 1048576.0:
        m, e = math.frexp(k1p1)
        wq4 = math.ldexp(1.0, 20 - e if m == 0.5 else 19 - e)
    fx = 0.0
    if wq4 > 0.0:
        max_sum = (k1 + 1.0) * math.log(float(n_movies) + 2.0) * 16.0 + 1.0
        _, e = math.frexp(max_sum)
        if 31 - e >= 12:
            fx = math.ldexp(1.0, 31 - e)
    return wq4, fx


def eligible(k: int, ntok: int, k1: float, b: float, n_movies: int) -> bool:
    """Mode 0 runs the fixed-point kernel for this query (it may still hand it on at a cap)."""
    return k <= MAX_K and ntok <= MAX_TOKENS and scales(k1, b, n_movies)[1] > 0.0


def largest_k1(n_movies: int) -> float:
    """The largest k1 (to 1e-9) for which the fixed-point path exists at this N."""
    lo, hi = 0.0, 1048575.0
    assert scales(lo, 0.75, n_movies)[1] > 0.0
    while hi - lo > 1e-9:
        mid = (lo + hi) / 2
        if scales(mid, 0.75, n_movies)[1] > 0.0:
            lo = mid
        else:
            hi = mid
    return lo


def idf(df, n_movies: int):
    """bm25_stage: log((N - df + 0.5) / (df + 0.5) + 1) with the integer difference taken first."""
    df = np.asarray(df, np.int64)
    return np.log((np.asarray(n_movies - df, np.float64) + 0.5) / (df.astype(np.float64) + 0.5) + 1.0)


def normk(dl, k1: float, b: float, avgdl: float):
    """bm25_norm_kernel: k1 * ((1 - b) + b * (dl / avgdl))."""
    return k1 * ((1.0 - b) + b * (np.asarray(dl, np.float64) / avgdl))


def weights(tf, nk, k1: float):
    """bm25_weight_kernel: tf * (k1 + 1) / (tf + normk)."""
    tf = np.asarray(tf, np.float64)
    return (tf * (k1 + 1.0)) / (tf + nk)


def wq(w, wq4_scale: float, zero_floor: bool = True):
    """The 19-bit weight word: round half to even, clamped at the top; at least 1 for w > 0 (zero_floor)."""
    w = np.asarray(w, np.float64)
    q = np.minimum(np.rint(w * wq4_scale), WQ_MAX).astype(np.int64)
    if zero_floor:
        q = np.where((q == 0) & (w > 0.0), 1, q)
    return q


def idfx(idf_value, fx_scale: float, wq4_scale: float):
    return np.asarray(idf_value, np.float64) * (fx_scale / wq4_scale)


def contribution(idfx_value, wq_value, zero_floor: bool = True):
    """item_apply: ceil(idfx * wq) for a non-zero word, so at least 1 (zero_floor=False: rounded to nearest);
    0 for a zero word."""
    wq_value = np.asarray(wq_value, np.int64)
    prod = np.asarray(idfx_value, np.float64) * wq_value.astype(np.float64)
    c = (np.ceil(prod) if zero_floor else np.rint(prod)).astype(np.int64)
    return np.where(wq_value != 0, c, 0)


def margin(token_idf, fx_scale: float, wq4_scale: float) -> int:
    """Per-query margin: 2 * ceil(sum_t (idfx_t + 0.5)) + 8, at least kFxMargin.  A term moves a document's sum by
    [-idfx_t, idfx_t + 1) from its exact value, so two sums disagree with the exact order by less than
    sum_t (2 * idfx_t + 1)."""
    m = 0.0
    for v in token_idf:
        m += float(v) * (fx_scale / wq4_scale) + 0.5
    return max(2 * math.ceil(m) + 8, FX_MARGIN)


def query_idf(c: Corpus, terms) -> np.ndarray:
    """idf of each query token (0 for a token outside the vocabulary or with df = 0, as bm25_stage stages it)."""
    df = c.df
    return np.array([float(idf(df[t], c.n_movies)) if t >= 0 and df[t] > 0 else 0.0 for t in terms], np.float64)


def fixed_sums(c: Corpus, terms, k1: float = 1.5, b: float = 0.75, zero_floor: bool = True):
    """(fixed-point sum int64[n_docs], exact score float64[n_docs], touched bool[n_docs]) of one query.

    The exact score is the reference's sum in query-token order; the fixed sum is what bm25_fx_kernel accumulates."""
    wq4, fx = scales(k1, b, c.n_movies)
    assert fx > 0.0, "the fixed-point path does not exist for these parameters"
    nk = normk(c.dl, k1, b, c.avgdl)
    qidf = query_idf(c, terms)
    fsum = np.zeros(c.n_docs, np.int64)
    exact = np.zeros(c.n_docs, np.float64)
    touched = np.zeros(c.n_docs, bool)
    for t, term in enumerate(terms):
        if term < 0 or c.df[term] == 0:
            continue
        lo, hi = c.indptr[term], c.indptr[term + 1]
        d = c.doc[lo:hi].astype(np.int64)
        w = weights(c.tf[lo:hi], nk[d], k1)
        fsum[d] += contribution(idfx(qidf[t], fx, wq4), wq(w, wq4, zero_floor), zero_floor)
        exact[d] = exact[d] + qidf[t] * w
        touched[d] = True
    return fsum, exact, touched


def exact_order(exact, touched, first_token=None):
    """Documents in the reference's order: score desc, then first query token holding the document, then doc."""
    d = np.nonzero(touched)[0]
    ft = np.zeros(len(d), np.int64) if first_token is None else np.asarray(first_token)[d]
    return d[np.lexsort((d, ft, -exact[d]))]
