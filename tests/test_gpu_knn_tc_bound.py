"""The tensor-core KNN path (K4: knn_tc3.cuh + knn_refine.cuh) at the edges of its fp16 error bound.

K4 decides nothing on approximate numbers only because |cos~ - cos| <= 1.10e-3 < eps / 2 (eps = kTcEps = 2.5e-3):
four cuts keep a band of 2 eps below an approximate K'-th value — the probe's threshold (tc3_probe_threshold_kernel,
tc3_threshold_kernel), the refine cut s_K - 2 eps, the second chance s' - 2 eps and the sampled probe's verification
s_K >= T.  On random or clustered corpora fp16 rounding moves cos~ by ~1e-5 and never comes near that band.  Here
every case is built with tests/helpers/knn_tc_model.py so that it does:

  * the accumulator: every survivor's cos~ is read back (rse_tc_last_pairs) and held to the model;
  * an inverted order at place K': A is the K'-th exact neighbour, K' rows B just below it read 9e-4 HIGHER in
    cos~, so A survives only if the band at the cut that decides is wide enough (a band of eps / 4 loses it);
  * capacity and radix edges, and rows whose norms sit at the ends of fp32.

Each case runs the exact scan (tc_mode 1) and K4 (tc_mode 2), compares positions and distance bits with each
other and with the oracle, and asserts through rse_stats which path answered."""
import os

import numpy as np
import pytest

import oracle
from helpers import knn_tc_model as m

pytestmark = pytest.mark.gpu

WIDTHS = (64, 320, 384, 512)
ACC_WORST = {}                               # width -> largest |cos~_dev - model| / accumulator term seen


class _env:
    """librse reads its RSE_* knobs when a handle is created."""
    def __init__(self, **kw):
        self.kw = {k: str(v) for k, v in kw.items()}

    def __enter__(self):
        self.old = {k: os.environ.get(k) for k in self.kw}
        os.environ.update(self.kw)

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


@pytest.fixture(scope="module", autouse=True)
def _cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    yield
    if ACC_WORST:
        print("\nlargest accumulator deviation / D * 2^-23 * sum|a^ q^|: " +
              ", ".join(f"D={d}: {v[0]:.3g} ({v[1]:.3g} absolute)" for d, v in sorted(ACC_WORST.items())))


def run(emb, Q, kprime, fma=False, env=None, inspect=None):
    """knn in tc_mode 1 and 2 on fresh handles; both equal bit for bit and equal the oracle.  Returns the K4 stats
    and whatever inspect(idx) returned right after the K4 call."""
    from rag_search_engine_b200 import _lib
    out, st, seen = {}, None, None
    for mode in (1, 2):
        with _env(**(env if (env and mode == 2) else {})):
            idx = _lib.Index(0)
        try:
            idx.set_tc_mode(mode)
            idx.set_fma(fma)
            idx.load_embeddings(emb)
            idx.stats_reset()
            out[mode] = idx.knn(Q, kprime)
            if mode == 2:
                st = idx.stats()
                seen = inspect(idx) if inspect else None
        finally:
            idx.close()
    for a, b in zip(out[1], out[2]):
        assert (a.view(np.uint8) == b.view(np.uint8)).all(), "K4 differs from the exact scan"
    dist, pos = out[2][0], out[2][1]
    for qi in range(len(Q)):
        od, orow = oracle.vec0_knn(emb, Q[qi], kprime, use_fma=fma, literal=False)
        assert pos[qi, :len(orow)].tolist() == orow.tolist(), f"query {qi}: rows differ from the oracle"
        assert dist[qi, :len(od)].view(np.uint32).tolist() == od.view(np.uint32).tolist(), f"query {qi}: distance bits"
    return st, seen


def pairs_of(q):
    return lambda idx: idx.tc_last_pairs(q)


def check_accumulator(emb, Q, rows, cos, qi, fma=False):
    """Every survivor's device cos~ against the model: within the header's accumulator term."""
    d = emb.shape[1]
    sh = m.shadow(emb[rows], fma)
    qh = m.query_shadow(Q[qi], fma)
    want = m.cos_tilde(sh, qh)[:, 0]
    term = m.acc_term(d, m.abs_products(sh, qh)[:, 0])
    dev = np.abs(cos.astype(np.float64) - want)
    assert (dev <= term).all(), f"D={d}: accumulator deviation {dev.max():.3g} exceeds D 2^-23 sum|p|"
    worst = ACC_WORST.get(d, (0.0, 0.0))
    ACC_WORST[d] = (max(worst[0], float((dev / term).max())), max(worst[1], float(dev.max())))
    return want


# ----------------------------------------------------------------------------- the accumulator
@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("fma", [False, True])
def test_accumulator_on_random_rows_matches_the_model(d, fma):
    rng = np.random.default_rng(d)
    emb = m.unit_rows(rng, 20_000, d) * rng.uniform(0.5, 2.0, (20_000, 1)).astype(np.float32)
    Q = m.unit_rows(rng, 4, d)
    st, seen = run(emb, Q, 1000, fma, inspect=lambda idx: [idx.tc_last_pairs(q) for q in range(4)])
    assert st.tc_queries == 4 and st.tc_fallback_queries == 0 and st.tc_second_chance_queries == 0
    for qi, (rows, cos, n) in enumerate(seen):
        assert n >= 1000 and len(rows) == n
        check_accumulator(emb, Q, rows, cos, qi, fma)


def test_accumulator_on_adversarial_rows_at_512():
    """One large product then 511 tiny ones of the same sign (each below 2^-24 of the running sum: a truncating
    accumulator drops them all), and large cancelling pairs followed by small terms."""
    d, rng = 512, np.random.default_rng(5)
    emb = m.unit_rows(rng, 20_000, d)
    Q = m.unit_rows(rng, 3, d)
    # query 0: q = (1, 2^-13 ...), rows = (1, 2^-12 (1 + r) ...): products of ~2^-25 after the first
    Q[0] = 2.0 ** -13
    Q[0, 0] = 1.0
    tiny = (2.0 ** -12 * (1 + rng.integers(0, 1024, (300, d - 1)) / 1024)).astype(np.float32)
    emb[:300, 1:] = tiny
    emb[:300, 0] = 1.0
    # query 1: (x, -x, y, small ...) against rows (x, x, y, small ...): the two large products cancel
    Q[1] = 2.0 ** -10
    Q[1, :3] = (0.6, -0.6, 0.5)
    small = (2.0 ** -9 * (1 + rng.integers(0, 1024, (300, d - 3)) / 1024)).astype(np.float32)
    emb[300:600, :3] = (0.6, 0.6, 0.5)
    emb[300:600, 3:] = small
    st, seen = run(emb, Q, 200, inspect=lambda idx: [idx.tc_last_pairs(q) for q in range(2)])
    assert st.tc_queries == 3 and st.tc_fallback_queries == 0
    for qi, lo in ((0, 0), (1, 300)):
        rows, cos, n = seen[qi]
        assert set(range(lo, lo + 300)) <= set(rows.tolist()), "the adversarial rows must all survive"
        check_accumulator(emb, Q, rows, cos, qi)


# ----------------------------------------------------------------------------- inverted order at place K'
def inversion_corpus(d, kprime, n, rng, where):
    """Background of random unit rows; K' - 1 rows far above; A (the K'-th exact neighbour) and K' rows B that read
    higher in cos~.  where = "spread" (evenly over the corpus, <= 8 per 128-row group: the probe sees all of them),
    "odd" (odd 256-row tiles only: a probe with tile stride 2 sees none), or an int (one contiguous block there)."""
    q, A, B = m.inversion_rows(d)
    far = m.rows_near(q, 0.9999, max(kprime - 1, 1), rng)[:kprime - 1]
    special = np.concatenate([far, A[None], np.repeat(B[None], kprime, 0)])
    emb = m.unit_rows(rng, n, d)
    ns = len(special)
    if where == "spread":
        at = np.linspace(0, n - 1, ns).astype(np.int64)
    elif where == "odd":
        odd = np.concatenate([np.arange(t * 256, (t + 1) * 256) for t in range(1, n // 256, 2)])
        at = odd[:ns]
    else:
        at = np.arange(where, where + ns)
    emb[at] = special
    Q = np.concatenate([q[None], m.unit_rows(rng, 3, d)]).astype(np.float32)
    return emb, Q, int(at[kprime - 1]), at


def check_inversion_on_device(emb, Q, kprime, seen, a_row):
    """The device values reach the edge: A survived, the K'-th largest cos~ is at least 8.5e-4 above A's (so a band
    of eps / 4 = 6.25e-4 cuts A), and every survivor agrees with the model."""
    rows, cos, n = seen
    check_accumulator(emb, Q, rows, cos, 0)
    assert a_row in rows.tolist(), "A did not survive the filter"
    s_k = np.sort(cos)[::-1][kprime - 1]
    gap = float(s_k) - float(cos[rows.tolist().index(a_row)])
    assert gap >= 8.5e-4, f"inversion on the device {gap:.3g}"
    return gap, rows, cos


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("kprime", [1, 10, 100, 256, 400])
def test_inversion_at_the_filter_cut(d, kprime):
    """Corpus below 32 768 rows: the probe's tile stride is 1, its K'-th value is the exact K'-th cos~ (400: the
    dense probe and tc3_threshold_kernel; the others: the sparse probe and tc3_probe_threshold_kernel), and the
    filter's threshold 1 - tau - 2 eps is what keeps A."""
    rng = np.random.default_rng(1000 * d + kprime)
    emb, Q, a_row, _ = inversion_corpus(d, kprime, 74 * 256, rng, "spread")
    st, seen = run(emb, Q, kprime, inspect=pairs_of(0))
    assert st.tc_queries == 4 and st.tc_fallback_queries == 0 and st.tc_second_chance_queries == 0
    gap, rows, cos = check_inversion_on_device(emb, Q, kprime, seen, a_row)
    # the filter's threshold was tight: no survivor more than 2 eps (+ slack) below s_K
    s_k = np.sort(cos)[::-1][kprime - 1]
    assert cos.min() >= s_k - 2 * m.EPS - 1e-5


@pytest.mark.parametrize("d,kprime", [(384, 1), (384, 10), (384, 100), (384, 256), (384, 400), (64, 100), (512, 100),
                                      (320, 10)])
def test_inversion_at_the_refine_cut(d, kprime):
    """128 tiles: the probe reads every second tile and none of the special rows, so the filter keeps far more than
    the band and the refine cut s_K - 2 eps alone decides whether A stays."""
    rng = np.random.default_rng(2000 * d + kprime)
    emb, Q, a_row, _ = inversion_corpus(d, kprime, 128 * 256, rng, "odd")
    st, seen = run(emb, Q, kprime, inspect=pairs_of(0))
    assert st.tc_queries == 4 and st.tc_fallback_queries == 0 and st.tc_second_chance_queries == 0
    gap, rows, cos = check_inversion_on_device(emb, Q, kprime, seen, a_row)
    s_k = np.sort(cos)[::-1][kprime - 1]
    assert cos.min() < s_k - 2 * m.EPS, "the filter was not looser than the refine cut"


@pytest.mark.parametrize("d", WIDTHS)
@pytest.mark.parametrize("kprime", [10, 100])
def test_inversion_at_the_second_chance(d, kprime):
    """Filler rows 8e-3 below A and the special rows in one block the sparse probe sees only 8 (16) of: the first
    threshold falls to the fillers, the survivor list overflows by 8 rows, and the second pass runs with s' - 2 eps
    from the 8192 kept survivors — s' is a B whichever 8 were dropped, so that band is what keeps A.  (The order of
    the appends is not fixed: with hundreds of rows dropped, the special block's tile could be the one that loses
    them.)"""
    rng = np.random.default_rng(3000 * d + kprime)
    emb, Q, a_row, at = inversion_corpus(d, kprime, 80 * 256, rng, 10 * 256)
    ex = m.exact_cos(emb[a_row:a_row + 1], Q[0])[0]
    fill = np.setdiff1d(np.arange(len(emb)), at)[::2][:8200 - len(at)]
    emb[fill] = m.rows_near(Q[0], ex - 8e-3, len(fill), rng)
    st, seen = run(emb, Q, kprime, inspect=pairs_of(0))
    assert st.tc_queries == 4 and st.tc_second_chance_queries == 1 and st.tc_fallback_queries == 0
    rows, cos, n = seen                                   # the second pass's survivors: the band around s' only
    assert n < 8192 and a_row in rows.tolist()
    check_inversion_on_device(emb, Q, kprime, seen, a_row)


def _sampled(i, stride, n):
    """t3_sample_source: the corpus row behind sample row i."""
    x = (i * 0x9E3779B1) & 0xFFFFFFFF
    x ^= x >> 15; x = (x * 0x85EBCA77) & 0xFFFFFFFF; x ^= x >> 13; x = (x * 0xC2B2AE3D) & 0xFFFFFFFF; x ^= x >> 16
    g = i * stride
    return g + x % min(stride, n - g)


@pytest.mark.parametrize("d", WIDTHS)
def test_sampled_probe_when_s_k_equals_t(d):
    """RSE_TC_SAMPLE_MIN_TILES=1: the probe reads the stratified row sample and its threshold is the j-th best sample
    value T.  Every B sits on a sampled row and nothing else near q does, so T is B's cos~ — exactly s_K.  The refine
    kernel's verification s_K >= T - 1e-7 uses s_K with its low byte dropped: it passes only when that byte of B's
    cos~ is zero, and the query otherwise takes the second pass with s_K - 2 eps.  Either way the answer is exact and
    the path is the one the device's own cos~ predicts."""
    kprime, stride, n = 10, 8, 80 * 256
    env = dict(RSE_TC_SAMPLE_MIN_TILES=1, RSE_TC_SAMPLE_STRIDE=stride)
    rng = np.random.default_rng(4000 + d)
    q, A, B = m.inversion_rows(d)
    emb = m.unit_rows(rng, n, d)
    samp = np.array([_sampled(i, stride, n) for i in range((n + stride - 1) // stride)])
    b_at = samp[5::200][:kprime]                        # one per 128-row group of the sample: all reach the probe
    other = np.setdiff1d(np.arange(n), samp)
    far_at, a_row = other[100:100 + kprime - 1], int(other[50])
    emb[b_at] = B
    emb[far_at] = m.rows_near(q, 0.9999, kprime - 1, rng)
    emb[a_row] = A
    Q = np.concatenate([q[None], m.unit_rows(rng, 3, d)]).astype(np.float32)
    st, seen = run(emb, Q, kprime, env=env, inspect=pairs_of(0))
    assert st.tc_queries == 4 and st.tc_fallback_queries == 0
    rows, cos, n_s = seen
    assert a_row in rows.tolist()
    c_b = np.float32(cos[rows.tolist().index(int(b_at[0]))])
    t = np.float32(1) - (np.float32(1) - c_b)                                # T as tc3_probe_threshold_kernel forms it
    s_k = np.uint32(c_b.view(np.uint32) & np.uint32(0xFFFFFF00)).view(np.float32)   # the refine's s_K, low byte dropped
    second = not (s_k >= np.float32(t - np.float32(1e-7)))
    print(f"D={d}: s_K = T = {float(c_b):.9g}, verification {'fails: second pass' if second else 'passes'}")
    assert st.tc_second_chance_queries == int(second)


# ----------------------------------------------------------------------------- capacity and radix edges
@pytest.mark.parametrize("n_band,fallback", [(4095, 0), (4096, 1)])
def test_refined_list_at_its_capacity(n_band, fallback):
    """K' = 1: one row equal to q and n_band copies of a row at cos 0.998, inside the refine band: the refined list
    holds 1 + n_band rows — 4096 (kTcRefineCap) is answered on the tensor cores, 4097 is handed to the exact scan."""
    d, rng = 384, np.random.default_rng(n_band)
    emb = m.unit_rows(rng, 20_000, d)
    Q = m.unit_rows(rng, 2, d)
    emb[3] = Q[0]
    emb[100:100 + n_band] = m.rows_near(Q[0], 0.998, 1, rng)[0]
    st, seen = run(emb, Q, 1, inspect=pairs_of(0))
    assert st.tc_queries == 2 and st.tc_fallback_queries == fallback and st.tc_second_chance_queries == 0
    assert seen[2] == 1 + n_band


@pytest.mark.parametrize("n_fill,survivors", [(8191, 8192), (8192, 8193)])
def test_survivor_list_at_its_capacity(n_fill, survivors):
    """K' = 1, 128 tiles (the probe reads the even ones): the one row equal to q sits in an odd tile, n_fill rows at
    cos 0.97 everywhere set the probe's threshold, so the filter keeps 1 + n_fill rows.  8192 (kTcCandCap) fit and
    the refine keeps one; 8193 overflow and the second pass (bound from the kept 8192) answers."""
    d, rng = 384, np.random.default_rng(n_fill)
    n = 128 * 256
    emb = m.unit_rows(rng, n, d)
    Q = m.unit_rows(rng, 2, d)
    emb[256 + 7] = Q[0]
    at = np.setdiff1d(np.arange(n), [256 + 7])[::3][:n_fill]
    emb[at] = m.rows_near(Q[0], 0.97, 1, rng)[0]
    st, seen = run(emb, Q, 1, inspect=lambda idx: idx.tc_last_survivors(2))
    assert st.tc_queries == 2
    if survivors <= 8192:
        assert seen[0] == survivors and st.tc_second_chance_queries == 0 and st.tc_fallback_queries == 0
    else:
        # the second pass recounts: 1 survivor if the exact neighbour was among the 8192 kept (s' = 1), else the
        # bound came from a filler and the list overflows again (exact scan); 1 in 8193
        assert st.tc_second_chance_queries + st.tc_fallback_queries == 1
        assert seen[0] == (1 if st.tc_second_chance_queries else survivors)


@pytest.mark.parametrize("kprime,tc", [(2048, True), (2049, False)])
def test_eligibility_limits(kprime, tc):
    """K4 needs K' * 4 <= 8192 survivors and K' * 2 <= 4096 refined rows: 2048 takes it, 2049 the exact scan."""
    d, rng = 384, np.random.default_rng(kprime)
    emb = m.unit_rows(rng, 20_000, d)
    Q = m.unit_rows(rng, 2, d)
    st, _ = run(emb, Q, kprime)
    assert st.tc_queries == (2 if tc else 0)
    if tc:
        assert st.tc_fallback_queries == 0


@pytest.mark.parametrize("d", [64, 384, 512])
def test_survivors_sharing_their_top_24_bits_around_s_k(d):
    """600 rows within ~1e-6 of each other in cosine: their cos~ agree in the top 24 bits, which is all the refine's
    radix select resolves of s_K.  The cut s_K - 2 eps must round down (keep more), never up."""
    rng = np.random.default_rng(6000 + d)
    emb = m.unit_rows(rng, 20_000, d)
    Q = m.unit_rows(rng, 2, d)
    base = m.rows_near(Q[0], 0.95, 1, rng)[0]
    emb[1000:1600] = base + (1e-7 * rng.standard_normal((600, d))).astype(np.float32)
    st, seen = run(emb, Q, 300, inspect=pairs_of(0))
    assert st.tc_queries == 2 and st.tc_fallback_queries == 0 and st.tc_second_chance_queries == 0
    rows, cos, n = seen
    near = cos[(rows >= 1000) & (rows < 1600)].view(np.uint32)
    assert len(near) == 600 and len(np.unique(near >> 8)) <= 4
    check_accumulator(emb, Q, rows, cos, 0)


# ----------------------------------------------------------------------------- norm edges
@pytest.mark.parametrize("d", WIDTHS)
def test_rows_whose_squares_underflow_keep_the_corpus_exact(d):
    """A row with amag below FLT_MIN (squares lost to underflow: ||a^|| = 4.6 on the shadow, the bound void) keeps
    the whole corpus on the exact scan, like a zero norm."""
    rng = np.random.default_rng(7000 + d)
    emb = m.unit_rows(rng, 20_000, d)
    emb[123] = m.underflow_row(d)
    emb[9000] = m.underflow_row(d, 1)
    assert m.amag(emb[[123, 9000]]).max() < m.FLT_MIN
    Q = m.unit_rows(rng, 3, d)
    Q[1] = np.sign(emb[123]) * 0.05
    st, _ = run(emb, Q, 50)
    assert st.tc_queries == 0


@pytest.mark.parametrize("d", WIDTHS)
def test_query_whose_squares_underflow_is_answered_exactly(d):
    rng = np.random.default_rng(7100 + d)
    emb = m.unit_rows(rng, 20_000, d)
    Q = m.unit_rows(rng, 3, d)
    Q[2] = m.underflow_row(d)
    assert m.query_norms(Q[2])[0] < m.MIN_NORM
    st, _ = run(emb, Q, 50)
    assert st.tc_queries == 3 and st.tc_fallback_queries == 1


@pytest.mark.parametrize("d", WIDTHS)
def test_rows_near_flt_max_and_below_the_fp16_range(d):
    """Rows scaled to amag just below FLT_MAX, and rows with most components below 2^-25 relative to their norm
    (zero in the shadow): K4 serves the corpus and every survivor matches the model."""
    rng = np.random.default_rng(7200 + d)
    emb = m.unit_rows(rng, 20_000, d)
    Q = m.unit_rows(rng, 2, d)
    big = m.rows_near(Q[0], 0.9, 50, rng)
    emb[:50] = big * np.float32(1.8e19)                                      # amag ~3.24e38 (FLT_MAX 3.40e38)
    assert np.isfinite(m.amag(emb[:50])).all() and m.amag(emb[:50]).min() > 3.2e38
    tiny = m.rows_near(Q[0], 0.85, 50, rng)
    tiny[:, 1:] *= np.float32(2.0 ** -27)                                     # below the fp16 subnormals after
    emb[100:150] = tiny                                                       # normalisation
    st, seen = run(emb, Q, 100, inspect=pairs_of(0))
    assert st.tc_queries == 2 and st.tc_fallback_queries == 0
    rows, cos, n = seen
    assert set(range(50)) <= set(rows.tolist())
    check_accumulator(emb, Q, rows, cos, 0)
