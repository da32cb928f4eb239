"""CPU model of the tensor-core KNN filter (K4: knn_tc3.cuh + knn_refine.cuh) and of its error bound.

What the device computes, restated in numpy:

  * amag[r]  = the reference's sequential fp32 sum of squares (``oracle.sq_magnitudes``, either FMA mode)      exact
  * inv      = fp32(1 / sqrt((double) amag)), a^ = fp16_rn(fp32(a * inv))                                     exact
  * sb[q]    = sqrt((double) sum of squares of q), q^ = fp16_rn(fp32(q * fp32(1 / sb)))                        exact
  * cos~     = sum_i a^_i q^_i: every product of two halves is exact in fp64, so the fp64 sum is the value the
               tensor cores approximate; the fp32 accumulator adds at most acc_term() on top                   bounded
  * the reference distance, from ``oracle`` (``vec0_knn`` / ``all_distances``) and ``cosine_tail``.

``bound_terms`` restates the header of knn_tc3.cuh term by term; ``eps`` = kTcEps.  The constructions at the end
build the corpora tests/test_gpu_knn_tc_bound.py places at each cut of the filter (an inverted order of cos~
against the exact order), and tests/test_knn_tc_model.py checks that each reaches the edge it claims.
"""
from __future__ import annotations

import numpy as np

import oracle

EPS = 2.5e-3                                  # kTcEps
FLT_MIN = np.float32(2.0 ** -126)             # kT3MinSq: the smallest squared norm the shadow accepts
MIN_NORM = 2.0 ** -63                         # kT3MinNorm: the smallest query norm sb


# ----------------------------------------------------------------------------- the arithmetic
def amag(emb: np.ndarray, use_fma: bool = False) -> np.ndarray:
    return oracle.sq_magnitudes(np.ascontiguousarray(emb, np.float32), use_fma)


def query_norms(Q: np.ndarray, use_fma: bool = False) -> np.ndarray:
    """sb = sqrt((double) m), m the sequential fp32 sum of squares (knn_query_prep_kernel)."""
    return np.sqrt(amag(np.atleast_2d(Q), use_fma).astype(np.float64))


def row_usable(am: np.ndarray) -> np.ndarray:
    """t3_shadow_row: a row reaches the shadow iff FLT_MIN <= amag < inf (empty slots, amag < 0, are zero rows)."""
    am = np.asarray(am, np.float32)
    return (am >= FLT_MIN) & np.isfinite(am)


def shadow(emb: np.ndarray, use_fma: bool = False, am: np.ndarray | None = None, guard: bool = True) -> np.ndarray:
    """fp16 shadow rows exactly as tc3_shadow_kernel writes them (float16 [n, D]).

    guard=False keeps the rule before FLT_MIN was required (any positive finite amag): the shadow of a row whose
    squares underflow, which the kernel no longer builds.
    """
    emb = np.ascontiguousarray(emb, np.float32)
    if am is None:
        am = amag(emb, use_fma)
    ok = row_usable(am) if guard else ((am > 0) & np.isfinite(am))
    inv = np.zeros(len(emb), np.float32)
    with np.errstate(divide="ignore"):
        inv[ok] = (1.0 / np.sqrt(am[ok].astype(np.float64))).astype(np.float32)
    return (emb * inv[:, None]).astype(np.float32).astype(np.float16)


def query_shadow(Q: np.ndarray, use_fma: bool = False, guard: bool = True) -> np.ndarray:
    """tc3_query_prep_kernel: q^ = fp16_rn(fp32(q * fp32(1 / sb))); zero for an unusable norm."""
    Q = np.ascontiguousarray(np.atleast_2d(Q), np.float32)
    sb = query_norms(Q, use_fma)
    ok = (sb >= MIN_NORM) & (sb < 1e300) if guard else (sb > 0) & (sb < 1e300)
    inv = np.zeros(len(Q), np.float32)
    inv[ok] = (1.0 / sb[ok]).astype(np.float32)
    return (Q * inv[:, None]).astype(np.float32).astype(np.float16)


def cos_tilde(sh: np.ndarray, qh: np.ndarray) -> np.ndarray:
    """The exact value of sum_i a^_i q^_i (fp64; each product of two halves is exact there)."""
    return sh.astype(np.float64) @ qh.astype(np.float64).T


def abs_products(sh: np.ndarray, qh: np.ndarray) -> np.ndarray:
    """sum_i |a^_i q^_i| per (row, query): what the accumulator's rounding scales with."""
    return np.abs(sh.astype(np.float64)) @ np.abs(qh.astype(np.float64)).T


def acc_term(dim: int, abs_sum=1.0):
    """The header's accumulator term: dim fp32 adds, each truncating, of partial sums at most sum|a^ q^|."""
    return dim * 2.0 ** -23 * np.asarray(abs_sum, np.float64)


def cosine_tail(dot, am, sb) -> np.ndarray:
    """vec0's tail (knn_scan.cuh cosine_tail): fp32(1 - dot / (sqrt((double) amag) * sb))."""
    return (1.0 - np.asarray(dot, np.float32).astype(np.float64) /
            (np.sqrt(np.asarray(am, np.float32).astype(np.float64)) * np.asarray(sb, np.float64))).astype(np.float32)


def exact_cos(emb: np.ndarray, q: np.ndarray, use_fma: bool = False) -> np.ndarray:
    """1 - the reference's distance (the value the refine kernel re-computes), fp64 of the fp32 distance."""
    return 1.0 - oracle.all_distances(emb, q, use_fma).astype(np.float64)


def bound_terms(dim: int) -> dict:
    """The error bound of knn_tc3.cuh at width dim, term by term, for unit a^ and q^."""
    t = {
        "rounding": 2.0 ** -10 + 2.0 ** -22,                    # fp16_rn of both operands, times sum|a^ q^| <= 1
        "subnormal_halves": 2.0 ** -25 * 2.0 * np.sqrt(dim),     # absolute 2^-25 below 2^-14, sum|a^| <= sqrt(D)
        "accumulator": float(acc_term(dim)),
        "reference_dot": dim * 2.0 ** -24,
        "underflowed_squares": dim * 2.0 ** -24,                 # amag >= FLT_MIN: lost squares < 2^-149 each
    }
    t["total"] = sum(t.values())
    return t


# ----------------------------------------------------------------------------- constructions
def _support(dim: int):
    """(s, 2^e): s = 4^k - 1 support coordinates at about 2^e = 2^-k, so s (2^e)^2 is just below 1; coordinate s makes
    up the norm and at least one free coordinate follows it (D = 64: s = 15; D = 320..512: s = 255)."""
    k = 1
    while 4 ** (k + 1) - 1 + 2 <= dim:
        k += 1
    s = 4 ** k - 1
    return s, 2.0 ** -k


def inversion_rows(dim: int, eta: float = 2.0 ** -17, cx: float | None = None):
    """(q, A, B): A is exactly closer to q than B, but every support component of A's shadow rounds DOWN by about
    2^-11 relative and every one of B's rounds UP by as much, so cos~(B) > cos~(A).

    Support: s = 4^k - 1 coordinates at v = 2^e (1 + 2^-11 -+ eta) (just below / above the fp16 midpoint above 2^e),
    coordinate s carries the rest of the norm, w = sqrt(1 - s v^2).  q = (1, ..., 1, cx) on the same s + 1
    coordinates: with cx > w / v, raising v lowers the exact cosine, so B (larger v) sits just below A.
    """
    s, p = _support(dim)
    if cx is None:
        cx = 1.2 if s < 255 else 1.5                  # inversions of 9.03e-4 (D = 64) and 9.45e-4 (D >= 320)
    def row(sign):
        v = p * (1.0 + 2.0 ** -11 + sign * eta)
        r = np.zeros(dim, np.float64)
        r[:s] = v
        r[s] = np.sqrt(1.0 - s * v * v)
        return r.astype(np.float32)
    q = np.zeros(dim, np.float32)
    q[:s] = 1.0
    q[s] = cx
    return q, row(-1.0), row(+1.0)


def rows_near(q: np.ndarray, cos: float, n: int, rng) -> np.ndarray:
    """n distinct rows at cosine ~cos to q (q rotated towards random directions orthogonal to it), unit norm."""
    qh = q.astype(np.float64) / np.linalg.norm(q)
    r = rng.standard_normal((n, q.size))
    r -= np.outer(r @ qh, qh)
    r /= np.linalg.norm(r, axis=1, keepdims=True)
    return (cos * qh[None, :] + np.sqrt(1.0 - cos * cos) * r).astype(np.float32)


def unit_rows(rng, n: int, dim: int) -> np.ndarray:
    x = rng.standard_normal((n, dim)).astype(np.float32)
    return x / np.linalg.norm(x, axis=1, keepdims=True)


def underflow_row(dim: int, sign_seed: int = 0) -> np.ndarray:
    """The row whose squares underflow in the reference's fp32 sum: one component of 1.14e-22 and dim - 1 of
    +-2.6e-23 (squares 1.3e-44 and 6.8e-46: the first is subnormal, the others flush to zero)."""
    rng = np.random.default_rng(sign_seed)
    r = np.where(rng.random(dim) < 0.5, -2.6e-23, 2.6e-23).astype(np.float32)
    r[0] = np.float32(1.14e-22)
    return r
