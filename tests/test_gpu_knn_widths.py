"""GPU: the tensor-core KNN path (K4: fp16 probe / filter on tcgen05, exact fp32 re-score) at every embedding width
D = 64 KB, KB = 1..8, and the batched image search built on it.

K4 is an exact method: every answer must be bit-identical to the exact scan (tc mode 1) at the same width, under both
FMA modes.  Widths outside 64..512 or not a multiple of 64, and corpora with zero-norm rows, stay on the scan."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


def unit_rows(rng, n, d):
    x = rng.standard_normal((n, d)).astype(np.float32)
    x /= np.linalg.norm(x, axis=1, keepdims=True)
    return x


def same(a, b):
    return len(a) == len(b) and all((np.asarray(x).view(np.uint8) == np.asarray(y).view(np.uint8)).all()
                                    for x, y in zip(a, b))


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


def _hard_corpus(rng, d, n=20_037):
    """A row count that is not a multiple of 256, empty vec0 slots, runs of duplicate rows across 1024-row block
    boundaries, and rows of tiny and huge norm."""
    emb = unit_rows(rng, n, d)
    emb[1015:1035] = emb[1015]                      # duplicates on both sides of row 1024
    emb[4090:4102] = emb[7]                         # ... of row 4096, equal to a row far away
    emb[9000:9050] *= np.float32(1e-15)
    emb[9050:9100] *= np.float32(1e15)
    valid = np.ones(n, np.uint8)
    valid[rng.choice(n, 300, replace=False)] = 0
    movie = (np.arange(n) // 7).astype(np.int32)
    return emb, valid, movie


def _hard_queries(rng, emb, nq):
    d = emb.shape[1]
    Q = emb[rng.integers(0, len(emb), nq)] + 0.3 * unit_rows(rng, nq, d)
    Q[0] = emb[1015]                                # sits exactly on the duplicate run
    if nq > 2:
        Q[1] = 0.0                                  # zero-norm query (handed to the exact scan)
        Q[2] *= np.float32(1e12)
    return np.ascontiguousarray(Q, np.float32)


# (nq, K') pairs: every nq of {2, 7, 256, 300, 2100} and every K' of {5, 100, 256, 1000}; 2100 queries span two groups
CASES = [(2, 5), (7, 100), (256, 256), (300, 1000), (2100, 100), (7, 1000)]


@pytest.mark.parametrize("fma", [False, True])
@pytest.mark.parametrize("kb", [1, 2, 3, 4, 5, 6, 7, 8])
def test_every_width_equals_exact_scan(kb, fma):
    import torch
    from rag_search_engine_b200 import _lib
    d = 64 * kb
    rng = np.random.default_rng(100 + kb)
    emb, valid, movie = _hard_corpus(rng, d)
    queries = {nq: _hard_queries(rng, emb, nq) for nq, _ in CASES}
    out, stats = {}, {}
    for mode in (1, 2):
        idx = _lib.Index(0)
        try:
            idx.set_fma(fma)
            idx.set_tc_mode(mode)
            idx.load_embeddings(emb, valid=valid, movie_idx=movie)
            r = []
            for nq, kp in CASES:
                r += list(idx.knn(queries[nq], kp))
            r += list(idx.knn_movies(queries[300], 10, 100))
            qd = torch.as_tensor(queries[256], device="cuda")
            cand = torch.empty((256, 100, 3), dtype=torch.int64, device="cuda")
            idx.knn_local_dev(qd.data_ptr(), 256, 100, cand.data_ptr())
            idx.synchronize()
            r.append(cand.cpu().numpy())
            out[mode], stats[mode] = r, idx.stats()
        finally:
            idx.close()
    n_total = sum(nq for nq, _ in CASES) + 300 + 256
    assert stats[1].tc_queries == 0
    assert stats[2].tc_queries == n_total, "the tensor-core path did not serve every query"
    assert stats[2].tc_filter_launches > 0
    assert same(out[1], out[2])


def test_sampled_probe_and_second_chance_at_512():
    """>= 262 144 rows: the probe runs over the stratified row sample.  A forced order statistic of 1 (or of 12 with
    every 8th row sampled, ~12.5 sample rows among the top 100) makes the verified bound fail for many queries: second
    chance or exact fallback.  The same on a clustered corpus.  The answers stay the exact scan's."""
    from rag_search_engine_b200 import _lib, synth
    rng = np.random.default_rng(7)
    iso = unit_rows(rng, 270_000, 512)
    se = synth.synth_embeddings(36_000, seed=8, dim=512, device="cpu", distribution="clustered", n_centres=400,
                                spread=0.06)
    clu = se.emb.numpy()
    assert len(clu) >= 262_144
    runs = [(iso, {}, False), (iso, dict(RSE_TC_PROBE_RANK=1), True),
            (iso, dict(RSE_TC_SAMPLE_STRIDE=8, RSE_TC_PROBE_RANK=12), True),
            (clu, dict(RSE_TC_SAMPLE_STRIDE=8, RSE_TC_PROBE_RANK=12), True)]
    for emb, knobs, expect_second in runs:
        Q = np.ascontiguousarray(emb[rng.integers(0, len(emb), 300)] + 0.05 * unit_rows(rng, 300, 512))
        idx = _lib.Index(0)
        try:
            idx.set_tc_mode(1)
            idx.load_embeddings(emb)
            want = idx.knn(Q, 100) + idx.knn(Q[:40], 10)
        finally:
            idx.close()
        with _env(**knobs):
            idx = _lib.Index(0)
        try:
            idx.load_embeddings(emb)                 # automatic mode: batches take K4 at this size
            got = idx.knn(Q, 100) + idx.knn(Q[:40], 10)
            st = idx.stats()
        finally:
            idx.close()
        assert st.tc_queries == 340
        print(f"{knobs} rows {len(emb)}: second chance {st.tc_second_chance_queries}, fallback {st.tc_fallback_queries}")
        if expect_second:
            assert st.tc_second_chance_queries > 0
        assert same(want, got)


@pytest.mark.parametrize("d", [100, 768, 1024])
def test_other_widths_stay_on_the_scan(d):
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(d)
    emb = unit_rows(rng, 12_000, d)
    Q = unit_rows(rng, 40, d)
    out = {}
    for mode in (1, 2):
        idx = _lib.Index(0)
        try:
            idx.set_tc_mode(mode)
            idx.load_embeddings(emb)
            out[mode] = idx.knn(Q, 100)
            assert idx.stats().tc_queries == 0
        finally:
            idx.close()
    assert same(out[1], out[2])


def test_zero_norm_rows_keep_512_on_the_scan():
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(3)
    emb = unit_rows(rng, 12_000, 512)
    emb[777] = 0.0
    Q = unit_rows(rng, 40, 512)
    out = {}
    for mode in (1, 2):
        idx = _lib.Index(0)
        try:
            idx.set_tc_mode(mode)
            idx.load_embeddings(emb)
            out[mode] = idx.knn(Q, 100)
            assert idx.stats().tc_queries == 0
        finally:
            idx.close()
    assert same(out[1], out[2])


def test_hybrid_batch_at_512():
    from rag_search_engine_b200 import HybridSearch, _lib, synth
    se = synth.synth_embeddings(4000, seed=31, dim=512, device="cpu")
    bm = synth.synth_bm25(4000, 3000, seed=31, mean_len=30, sd_len=10)
    nq = 64
    tp, tr = synth.synth_token_queries(bm, nq, seed=32)
    Q = synth.synth_query_vectors(se.emb, nq, seed=32).numpy()
    T = len(bm.df)
    names = np.array([f"t{i}" for i in range(T)], dtype=np.str_)
    toks = np.where(tr >= 0, names[np.clip(tr, 0, None)], "<oov>").tolist()
    token_lists = [toks[tp[i]:tp[i + 1]] for i in range(nq)]
    idx = _lib.Index(0)
    try:
        idx.load_embeddings(se.emb.numpy(), movie_idx=se.movie_of_chunk.numpy())
        idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
        idx.set_id_tables(se.movie_ids, se.movie_ids)
        hs = HybridSearch.from_loaded(idx, dict(zip(names.tolist(), range(T))), se.movie_ids, se.movie_ids,
                                      registry_key="knn-widths-hybrid-512")
        out = {}
        for mode in (1, 2):
            idx.set_tc_mode(mode)
            idx.stats_reset()
            out[mode] = (hs.rrf_search_batch(token_lists, Q, k=60, limit=10),
                         hs.rrf_search_batch(token_lists, Q, k=60, limit=10, as_arrays=True),
                         hs.weighted_search_batch(token_lists, Q, alpha=0.5, limit=5))
            assert (idx.stats().tc_queries > 0) == (mode == 2)
        assert out[1][0] == out[2][0] and out[1][2] == out[2][2]
        assert same(out[1][1], out[2][1])
    finally:
        idx.close()


# ----------------------------------------------------------------------------- MultimodalSearch batch entry points
class _TableModel:
    """encode(texts) -> the precomputed embedding of each document text (the documents' own vectors)."""
    def __init__(self, table):
        self.table = table

    def encode(self, texts, convert_to_numpy=True, show_progress_bar=False):
        return self.table[[int(t.split(":")[0][1:]) for t in texts]]


def _docs(n):
    return [{"id": 10 + i, "title": f"d{i}", "description": f"text {i}"} for i in range(n)]


@pytest.mark.parametrize("n_docs,mode", [(3000, 2), (270_000, 0)])
def test_search_with_vectors_equals_per_row(n_docs, mode):
    from rag_search_engine_b200.multimodal import MultimodalSearch
    rng = np.random.default_rng(n_docs)
    table = unit_rows(rng, n_docs, 512)
    ms = MultimodalSearch(_docs(n_docs), model=_TableModel(table))
    try:
        if mode:
            ms._index.set_tc_mode(mode)
        Q = table[rng.integers(0, n_docs, 64)] + 0.2 * unit_rows(rng, 64, 512)
        ms._index.stats_reset()
        got = ms.search_with_vectors(Q, top_k=20)
        assert ms._index.stats().tc_queries == 64
        want = [ms.search_with_vector(q, top_k=20) for q in Q]
        assert got == want
        assert all(len(r) == 20 and list(r[0]) == ["id", "title", "description", "similarity"] for r in got)
        assert ms.search_with_vectors(Q[:3], top_k=0) == [[], [], []]
        assert ms.search_with_vectors(np.zeros((0, 512), np.float32)) == []
    finally:
        ms.close()


def test_search_with_vectors_errors():
    from rag_search_engine_b200.multimodal import MultimodalSearch
    ms = MultimodalSearch(None, model=_TableModel(None))
    with pytest.raises(ValueError, match="without documents"):
        ms.search_with_vectors(np.zeros((2, 512), np.float32))
    with pytest.raises(ValueError, match="without documents"):
        ms.search_with_images(["nothing.png"])
    with pytest.raises(ValueError, match="without documents"):
        ms.search_with_vectors([])


def test_search_with_images_equals_per_image(tmp_path):
    transformers = pytest.importorskip("transformers")
    torch = pytest.importorskip("torch")
    from PIL import Image
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.clip import GpuClipModel, clip_configs_from_hf
    from rag_search_engine_b200.multimodal import MultimodalSearch
    EOS, BOS = 49407, 49406

    def word_tok(texts):
        import zlib
        return [[BOS] + [3 + zlib.crc32(w.encode()) % 49000 for w in t.lower().split()][:75] + [EOS] for t in texts]

    vc = dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512, image_size=64,
              patch_size=16)
    tc = dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512, vocab_size=49408,
              max_position_embeddings=77, eos_token_id=EOS, bos_token_id=BOS, pad_token_id=1)
    cfg = transformers.CLIPConfig(text_config=tc, vision_config=vc, projection_dim=128)   # 128 wide: K4 at KB = 2
    torch.manual_seed(5)
    model = transformers.CLIPModel(cfg).eval()
    proc = transformers.CLIPImageProcessor(size={"shortest_edge": 64}, crop_size={"height": 64, "width": 64})
    rng = np.random.default_rng(9)
    words = [f"w{i}" for i in range(300)]
    docs = [{"id": 3 * i, "title": " ".join(rng.choice(words, 2)),
             "description": " ".join(rng.choice(words, int(rng.integers(5, 30))))} for i in range(3000)]
    paths = []
    for i in range(6):
        p = tmp_path / f"q{i}.png"
        Image.fromarray(rng.integers(0, 256, (int(rng.integers(60, 200)), 150, 3), dtype=np.uint8)).save(p)
        paths.append(str(p))
    vision, text = clip_configs_from_hf(model.config)
    idx = _lib.Index(0)
    try:
        gm = GpuClipModel(idx, model.state_dict(), vision, text, tokenizer=word_tok,
                          image_processor=lambda ims: proc(ims, return_tensors="np")["pixel_values"])
        ms = MultimodalSearch(docs, model=gm)
        try:
            for mode in (0, 2):
                ms._index.set_tc_mode(mode)
                got = ms.search_with_images(paths, top_k=15)
                assert got == [ms.search_with_image(p, top_k=15) for p in paths]
                assert all(len(r) == 15 for r in got)
            assert ms.search_with_images([], top_k=5) == []
            assert ms.search_with_images(paths[:2], top_k=-1) == [[], []]
        finally:
            ms.close()
    finally:
        idx.close()


def test_reload_at_another_width_on_one_handle():
    """One handle, embeddings reloaded at 384, then 512, then 128: every load gets its own shadow and query map."""
    from rag_search_engine_b200 import _lib
    rng = np.random.default_rng(11)
    ref = _lib.Index(0)
    idx = _lib.Index(0)
    try:
        ref.set_tc_mode(1)
        idx.set_tc_mode(2)
        for d in (384, 512, 128):
            emb = unit_rows(rng, 9_000, d)
            Q = unit_rows(rng, 300, d)
            ref.load_embeddings(emb)
            idx.load_embeddings(emb)
            idx.stats_reset()
            assert same(ref.knn(Q, 50), idx.knn(Q, 50))
            assert idx.stats().tc_queries == 300
    finally:
        idx.close()
        ref.close()
