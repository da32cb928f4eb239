"""Exact movie-level KNN restated in numpy over oracle.all_distances (the contract of rse_knn_movies_exact).

Every competing row (valid, movie_idx >= 0) gets the vec0 key (orderable f32 distance << 32) | (pos ^ 1023), whose
ascending order is the emit order (distance asc, block asc, slot desc).  A movie's best chunk is its row with the
smallest key; movies are ordered by that key and the first k are the answer.
"""
import numpy as np

import oracle


def orderable(d: np.ndarray) -> np.ndarray:
    b = np.ascontiguousarray(d, np.float32).view(np.uint32).astype(np.uint64)
    return np.where(b & 0x80000000, ~b & 0xFFFFFFFF, b | 0x80000000).astype(np.uint64)


def keys(d: np.ndarray, pos: np.ndarray) -> np.ndarray:
    return (orderable(d) << np.uint64(32)) | (np.asarray(pos, np.uint64) ^ np.uint64(1023))


def exact_movies(emb, q, movie_of, k, valid=None, use_fma=False, pos=None, dist=None):
    """(dist f32[n], row i64[n], movie i32[n]) of the n = min(k, competing movies) nearest movies, best key first.
    ``dist`` may pass the precomputed oracle.all_distances(emb, q) to share it across several k."""
    movie_of = np.asarray(movie_of, np.int64)
    n = len(movie_of)
    d = oracle.all_distances(emb, q, use_fma) if dist is None else dist
    pos = np.arange(n, dtype=np.int64) if pos is None else np.asarray(pos, np.int64)
    ok = movie_of >= 0
    if valid is not None:
        ok &= np.asarray(valid, bool)
    rows = np.nonzero(ok)[0]
    if len(rows) == 0:
        return np.zeros(0, np.float32), np.zeros(0, np.int64), np.zeros(0, np.int32)
    kk = keys(d[rows], pos[rows])
    order = rows[np.argsort(kk, kind="stable")]
    _, first = np.unique(movie_of[order], return_index=True)      # the first row of each movie in key order
    best = order[np.sort(first)][:k]                               # np.sort(first): movies in key order
    return d[best].astype(np.float32), best.astype(np.int64), movie_of[best].astype(np.int32)
