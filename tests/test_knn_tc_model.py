"""CPU checks of tests/helpers/knn_tc_model.py, the numpy restatement of the tensor-core KNN filter (K4), and of the
error bound in the header of knn_tc3.cuh it rests on.  No GPU needed: the GPU side is tests/test_gpu_knn_tc_bound.py."""
import numpy as np
import pytest

from helpers import knn_tc_model as m

WIDTHS = (64, 128, 192, 256, 320, 384, 448, 512)


# ----------------------------------------------------------------------------- the model at hand-worked values
def test_shadow_rounds_to_nearest_even_at_midpoints():
    # 1 + 2^-11 is the midpoint between 1 and the next half 1 + 2^-10: ties go to the even mantissa (1);
    # 1 + 3 * 2^-11 sits between 1 + 2^-10 (odd) and 1 + 2^-9 (even): up.  The row is scaled so that amag = 4
    # exactly and inv = 0.5: a^ = a / 2 keeps the mantissas.
    row = np.zeros(64, np.float32)
    row[0] = 2.0 * (1 + 2.0 ** -11)
    row[1] = 2.0 * (1 + 3 * 2.0 ** -11)
    am = np.array([4.0], np.float32)                      # forced: the point is the rounding, not the norm
    sh = m.shadow(row[None], am=am)[0]
    assert float(sh[0]) == 1.0
    assert float(sh[1]) == 1 + 2.0 ** -9
    # just either side of the midpoint
    row[0] = np.nextafter(np.float32(2.0 * (1 + 2.0 ** -11)), np.float32(0))
    row[1] = np.nextafter(np.float32(2.0 * (1 + 2.0 ** -11)), np.float32(4))
    sh = m.shadow(row[None], am=am)[0]
    assert float(sh[0]) == 1.0 and float(sh[1]) == 1 + 2.0 ** -10


def test_shadow_subnormal_halves_and_below():
    # fp16 subnormals are multiples of 2^-24; below 2^-25 a component rounds to zero (the 2^-25 absolute term)
    row = np.zeros(64, np.float32)
    row[0] = 1.0
    row[1] = 3 * 2.0 ** -24                     # subnormal half, exact
    row[2] = 2.0 ** -25                         # the midpoint 0 | 2^-24: ties to even -> 0
    row[3] = 1.5 * 2.0 ** -25                   # above the midpoint -> 2^-24
    row[4] = 2.0 ** -30                         # far below -> 0
    sh = m.shadow(row[None])[0].astype(np.float64)
    assert m.amag(row[None])[0] == np.float32(1.0)
    assert sh[0] == 1.0 and sh[1] == 3 * 2.0 ** -24 and sh[2] == 0.0 and sh[3] == 2.0 ** -24 and sh[4] == 0.0


@pytest.mark.parametrize("use_fma", [False, True])
def test_amag_and_inverse_follow_the_reference_sum(use_fma):
    rng = np.random.default_rng(3)
    x = rng.standard_normal((4, 384)).astype(np.float32)
    am = m.amag(x, use_fma)
    for r in range(4):
        acc = np.float32(0)
        for v in x[r]:
            acc = np.float32(np.float64(acc) + np.float64(v) * np.float64(v)) if use_fma else \
                np.float32(acc + np.float32(v * v))
        assert am[r] == acc
    sh = m.shadow(x, use_fma)
    inv = (1.0 / np.sqrt(am.astype(np.float64))).astype(np.float32)
    assert (sh == (x * inv[:, None]).astype(np.float16)).all()


def test_underflowing_row_breaks_the_unit_norm_premise():
    """The hole: squares of 2.6e-23 flush to zero and 1.14e-22^2 is subnormal in the sequential fp32 sum, so amag is
    positive and finite but 21x too small, and the shadow row normalised with it has norm 4.64, not 1."""
    row = m.underflow_row(384)
    am = m.amag(row[None])[0]
    true = float((row.astype(np.float64) ** 2).sum())
    assert 0 < am < m.FLT_MIN and am == np.float32(1.3e-44)
    assert true == pytest.approx(2.7e-43, rel=0.01)
    nrm = np.linalg.norm(m.shadow(row[None], guard=False)[0].astype(np.float64))
    assert nrm == pytest.approx(4.64, abs=0.01)
    # the rounding term of the bound grows with ||a^||: sum|a^ q^| <= ||a^|| (Cauchy-Schwarz), past eps / 2
    assert (2.0 ** -10) * nrm > m.EPS / 2 and (2.0 ** -10) * nrm == pytest.approx(4.5e-3, abs=1e-4)
    # the kernel's rule: below FLT_MIN the row does not reach the shadow, the corpus stays on the exact scan
    assert not m.row_usable([am])[0]
    assert (m.shadow(row[None])[0] == 0).all()
    # the same for a query: sum of squares below FLT_MIN <=> sb below 2^-63
    sb = m.query_norms(row)[0]
    assert sb < m.MIN_NORM and (m.query_shadow(row)[0] == 0).all()
    assert m.query_norms(np.full(64, 2.0 ** -63 / 8, np.float32))[0] == m.MIN_NORM      # 64 x 2^-132 = 2^-126


def test_amag_just_below_flt_max_stays_usable():
    row = np.full(512, 8.1e17, np.float32)
    am = m.amag(row[None])[0]
    assert np.isfinite(am) and am > 3.3e38 and m.row_usable([am])[0]
    sh = m.shadow(row[None])[0].astype(np.float64)
    assert abs(np.linalg.norm(sh) - 1.0) < 2.0 ** -10


# ----------------------------------------------------------------------------- the bound
def test_bound_stays_below_half_eps_at_every_width():
    for d in WIDTHS:
        assert m.bound_terms(d)["total"] < m.EPS / 2, d
    t = m.bound_terms(512)
    assert t["total"] == pytest.approx(1.10e-3, abs=5e-6)
    assert t["accumulator"] == pytest.approx(6.10e-5, abs=1e-7)


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("use_fma", [False, True])
def test_bound_holds_on_random_rows(d, use_fma):
    """|cos~ - cos| with cos~ the fp64 value of the fp16 products (the accumulator then adds at most its own term)
    stays within the rounding terms of the header, and far below eps / 2."""
    rng = np.random.default_rng(d + use_fma)
    emb = m.unit_rows(rng, 2000, d) * rng.uniform(0.25, 4.0, (2000, 1)).astype(np.float32)
    Q = m.unit_rows(rng, 3, d)
    Q[1] = emb[7] + 0.01 * Q[1]                                 # one query with a near neighbour
    ct = m.cos_tilde(m.shadow(emb, use_fma), m.query_shadow(Q, use_fma))
    t = m.bound_terms(d)
    worst = 0.0
    for j in range(3):
        dev = np.abs(ct[:, j] - m.exact_cos(emb, Q[j], use_fma))
        worst = max(worst, float(dev.max()))
    assert worst <= t["total"] - t["accumulator"]
    assert worst < m.EPS / 2


# ----------------------------------------------------------------------------- constructions reach their edges
@pytest.mark.parametrize("d", [64, 320, 384, 512])
@pytest.mark.parametrize("kprime", [1, 10, 100, 256, 400])
def test_inversion_construction_reaches_its_edge(d, kprime):
    """The corpus of the inversion cases (tests/test_gpu_knn_tc_bound.py): K' - 1 rows far above, A at place K' of
    the exact order, K' rows B just below A.  In cos~ every B is at least 9e-4 above A, so s_K (the K'-th largest
    cos~) is a B and A sits 9e-4 below it: inside the 2 eps band, outside a band of eps / 4."""
    q, A, B = m.inversion_rows(d)
    far = m.rows_near(q, 0.9999, max(kprime - 1, 1), np.random.default_rng(kprime))[:kprime - 1]
    rows = np.concatenate([far, A[None], np.repeat(B[None], kprime, 0)])
    ex = m.exact_cos(rows, q)
    order = np.argsort(-ex, kind="stable")
    assert order[kprime - 1] == kprime - 1                               # A is the K'-th exact neighbour
    assert ex[kprime - 1] > ex[kprime]                                   # and strictly above every B
    ct = m.cos_tilde(m.shadow(rows), m.query_shadow(q))[:, 0]
    s_k = np.sort(ct)[::-1][kprime - 1]
    assert s_k == ct[kprime]                                             # the K'-th largest cos~ is a B
    gap = s_k - ct[kprime - 1]
    assert gap >= 9.0e-4, gap                                            # the inversion the tests rely on
    assert gap + 2 * m.bound_terms(d)["accumulator"] < 2 * m.EPS         # A survives the real band ...
    assert gap - 2 * m.bound_terms(d)["accumulator"] > m.EPS / 4         # ... and not a band of eps / 4
