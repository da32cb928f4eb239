"""GPU: CLIP's byte-level BPE on the device (csrc/bpe.cuh) against the HuggingFace fast tokenizer, bit for bit, and
the text path built on it (GpuClipModel.encode through DeviceBPE, MultimodalSearch's constructor) against the same
calls fed with HF ids; the ABI's error paths."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
transformers = pytest.importorskip("transformers")

from helpers import bpe_corpus as corpus  # noqa: E402
from helpers import bpe_ref  # noqa: E402

N_TEXTS = 20000
CASES = ((False, None), (True, None), (True, 77), (True, 8), (False, 77))


def _utf8(texts):
    from rag_search_engine_b200.encoder import _utf8
    return _utf8(texts)


def _device_ids(idx, slot, texts, special, ml):
    ids, cu = idx.tokenize(slot, *_utf8(texts), special, ml or 0)
    ids = ids.tolist()
    return [ids[a:b] for a, b in zip(cu[:-1].tolist(), cu[1:].tolist())]


@pytest.mark.parametrize("vocab", ["trained", "tiny"])
def test_device_ids_equal_hf(gpu_index, vocab):
    from rag_search_engine_b200.bpe import build_bpe_tables
    tok = corpus.tokenizer(vocab)
    t = build_bpe_tables(tok)
    gpu_index.tokenizer_load_bpe(0, t)
    pool = corpus.texts(N_TEXTS + 8000, seed=17)
    for special, ml in CASES:
        # the texts the device takes at this cut (the restatement refuses exactly those it refuses)
        texts = [x for x in pool if bpe_ref.tokenize(t, x, special, ml) is not None][:N_TEXTS]
        assert len(texts) == N_TEXTS
        want = tok(texts, add_special_tokens=special, truncation=ml is not None, max_length=ml)["input_ids"]
        got = _device_ids(gpu_index, 0, texts, special, ml)
        bad = [i for i, (g, w) in enumerate(zip(got, want)) if g != w]
        assert not bad, (special, ml, len(bad), repr(texts[bad[0]]), got[bad[0]], want[bad[0]])


def test_batch_sizes_and_the_callable(gpu_index):
    from rag_search_engine_b200.clip import DeviceBPE
    tok = corpus.tokenizer("trained")
    db = DeviceBPE(gpu_index, tok, slot=1, max_length=77)
    big = corpus.texts(100000, seed=23)
    for n in (1, 256, 100000):
        texts = big[:n]
        before = db.host_texts
        assert db(texts) == tok(texts, truncation=True, max_length=77)["input_ids"], n
        if n == 100000:                                    # some long word before the cut: the wide route
            assert db.host_texts - before == len(db.host_routed(texts, True))
    # routed texts (a code point NFC joins, a piece past the word buffer) go to the host tokenizer and are counted
    mixed = ["e\u0301 x", "plain text", "\u1100\u1161", "ab" * 200, "movie " * 90 + "ab" * 200]
    before = db.host_texts
    assert db(mixed) == tok(mixed, truncation=True, max_length=77)["input_ids"]
    assert db.host_texts - before >= 3
    assert db([]) == []
    assert db(["", " 　 "], False, None) == [[], []]
    assert db(["<|endoftext|>", "<|ENDOFTEXT|>"], False, None) == tok(["<|endoftext|>", "<|ENDOFTEXT|>"],
                                                                      add_special_tokens=False)["input_ids"]


SMALL_TEXT = dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
                  vocab_size=6100, max_position_embeddings=77)
SMALL_VISION = dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
                    image_size=64, patch_size=16)


def _clip_model(tok):
    cfg = transformers.CLIPConfig(text_config=dict(SMALL_TEXT, eos_token_id=tok.eos_token_id,
                                                   bos_token_id=tok.bos_token_id, pad_token_id=tok.pad_token_id),
                                  vision_config=SMALL_VISION, projection_dim=96)
    torch.manual_seed(3)
    return transformers.CLIPModel(cfg).eval()


def test_clip_encode_through_device_bpe(fresh_index):
    from rag_search_engine_b200.clip import DeviceBPE, GpuClipModel, clip_configs_from_hf
    tok = corpus.tokenizer("trained")
    model = _clip_model(tok)
    vision, text = clip_configs_from_hf(model.config)
    db = DeviceBPE(fresh_index, tok, slot=0, max_length=77)
    gm = GpuClipModel(fresh_index, model.state_dict(), vision, text, tokenizer=db)
    texts = corpus.texts(4000, seed=31)               # > 65536 tokens: several slices of the text tower
    dev = [x for x in texts if not db.tables.needs_host(x) and not db.tables.may_overflow(x)]
    hf = lambda x: tok(x, truncation=True, max_length=77)["input_ids"]   # noqa: E731
    for batch in (dev, dev[:1], texts):
        before = db.host_texts
        got = gm.encode(batch)
        assert np.array_equal(got, gm.encode_ids(hf(batch))), len(batch)
        assert (db.host_texts == before) == (batch is not texts)
    assert np.array_equal(gm.encode(dev[0]), gm.encode_ids(hf(dev[:1]))[0])


def test_multimodal_search_constructor_either_way(fresh_index):
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.clip import DeviceBPE, GpuClipModel, clip_configs_from_hf
    from rag_search_engine_b200.multimodal import MultimodalSearch
    tok = corpus.tokenizer("trained")
    model = _clip_model(tok)
    vision, text = clip_configs_from_hf(model.config)
    rng = np.random.default_rng(4)
    docs = [{"id": 3 + i, "title": " ".join(rng.choice(corpus.WORDS, 2)).title(),
             "description": corpus.texts(1, seed=1000 + i)[0]} for i in range(3000)]
    hf = lambda x: tok(list(x), truncation=True, max_length=77)["input_ids"]   # noqa: E731
    gm_dev = GpuClipModel(fresh_index, model.state_dict(), vision, text,
                          tokenizer=DeviceBPE(fresh_index, tok, slot=0, max_length=77))
    ms_dev = MultimodalSearch(docs, model=gm_dev)
    other = _lib.Index(0)                                  # (a handle holds two encoder slots: one CLIP model)
    gm_host = GpuClipModel(other, model.state_dict(), vision, text, tokenizer=hf)
    ms_host = MultimodalSearch(docs, model=gm_host)
    try:
        assert np.array_equal(ms_dev.text_embeddings, ms_host.text_embeddings)
        q = rng.standard_normal((8, 96)).astype(np.float32)
        assert ms_dev.search_with_vectors(q, top_k=20) == ms_host.search_with_vectors(q, top_k=20)
        assert ms_dev.search_with_vector(q[0], top_k=7) == ms_host.search_with_vector(q[0], top_k=7)
    finally:
        ms_dev.close()
        ms_host.close()
        other.close()


def test_bpe_abi_error_paths(fresh_index):
    from rag_search_engine_b200._lib import RseError
    from rag_search_engine_b200.bpe import build_bpe_tables
    from rag_search_engine_b200.clip import clip_configs_from_hf
    from rag_search_engine_b200.encoder import DeviceWordPiece, GpuSentenceEncoder, random_state_dict
    from helpers import wp_corpus
    idx = fresh_index
    tok = corpus.tokenizer("trained")
    t = build_bpe_tables(tok)
    ok = _utf8(["a movie"])
    with pytest.raises(RseError, match="no tokenizer") as e:
        idx.tokenize(0, *ok, True, 77)
    assert e.value.code == -3
    idx.tokenizer_load_bpe(0, t)
    data, offs = _utf8(["fine", "also fine", "bad"])
    with pytest.raises(RseError, match="offsets") as e:
        idx.tokenize(0, data, offs[::-1].copy(), True, 77)
    assert e.value.code == -1
    bad = b"fine" + b"ok \xc3\x28" + b"x"
    with pytest.raises(RseError, match="text 1 is not well-formed UTF-8") as e:
        idx.tokenize(0, bad, np.array([0, 4, 8, 9]), True, 77)
    assert e.value.code == -1
    for text in ("e\u0301", "ab" * 200):
        with pytest.raises(RseError, match="text 1 needs the host tokenizer") as e:
            idx.tokenize(0, *_utf8(["ok", text]), True, 77)
        assert e.value.code == -4
    # the long word past the cut is never tokenized, so it is not refused
    assert len(idx.tokenize(0, *_utf8(["movie " * 90 + "ab" * 200]), True, 77)[0]) == 77
    bad_t = build_bpe_tables(tok)
    bad_t.merges = bad_t.merges[:-1]
    with pytest.raises(RseError, match="power of two") as e:
        idx.tokenizer_load_bpe(1, bad_t)
    assert e.value.code == -1
    # a BPE slot feeds a CLIP text tower only; a WordPiece slot does not feed one
    model = _clip_model(tok)
    vision, text = clip_configs_from_hf(model.config)
    from rag_search_engine_b200.clip import GpuClipModel
    GpuClipModel(idx, model.state_dict(), vision, text)
    out = idx.encode_texts(0, 1, *ok, 77)
    assert out.shape == (1, 96)
    with pytest.raises(RseError, match="max_length") as e:
        idx.encode_texts(0, 1, *ok, 78)
    assert e.value.code == -4
    with pytest.raises(RseError, match="CLIP text tower") as e:
        idx.encode_texts(0, 0, *ok, 64)                                       # the vision tower
    assert e.value.code == -1
    with pytest.raises(RseError, match="BPE tokenizer") as e:
        idx.rerank_docs_load_texts(0, [1], *ok)
    assert e.value.code == -1
    wtok = wp_corpus.tokenizer("uncased")
    DeviceWordPiece(idx, wtok, slot=1, max_length=128)
    with pytest.raises(RseError, match="not WordPiece") as e:
        idx.encode_texts(1, 1, *ok, 64)
    assert e.value.code == -1
    # a BERT encoder in slot 1 instead of the text tower: the BPE slot is refused, WordPiece runs as before
    cfg = dict(vocab_size=4000, hidden=64, layers=1, heads=2, intermediate=128, max_positions=128, type_vocab=2,
               ln_eps=1e-12)
    GpuSentenceEncoder(idx, random_state_dict(cfg, seed=5), cfg, None, slot=1, max_seq_length=128)
    with pytest.raises(RseError, match="CLIP text tower") as e:
        idx.encode_texts(0, 1, *ok, 64)
    assert e.value.code == -1
    assert idx.encode_texts(1, 1, *ok, 64).shape == (1, 64)


def test_from_sentence_transformer_puts_the_tokenizer_on_the_device(fresh_index):
    """The reference's model object (a SentenceTransformer whose module 0 holds the CLIPModel and its processor) gets
    a DeviceBPE; a tokenizer the device does not take stays on the host with a warning that says why."""
    import types
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.clip import DeviceBPE, GpuClipModel
    from helpers import wp_corpus
    tok = corpus.tokenizer("trained")
    model = _clip_model(tok)
    proc = types.SimpleNamespace(tokenizer=tok, image_processor=transformers.CLIPImageProcessor(
        size={"shortest_edge": 64}, crop_size={"height": 64, "width": 64}))
    st = [types.SimpleNamespace(model=model, processor=proc)]
    gm = GpuClipModel.from_sentence_transformer(fresh_index, st)
    assert isinstance(gm.tokenizer, DeviceBPE) and gm.tokenizer.slot == 0
    texts = corpus.texts(300, seed=41)
    assert np.array_equal(gm.encode(texts), gm.encode_ids(tok(texts, truncation=True, max_length=77)["input_ids"]))
    other = _lib.Index(0)
    try:
        proc.tokenizer = wp_corpus.tokenizer("uncased")
        with pytest.warns(UserWarning, match="stays on the host"):
            gm2 = GpuClipModel.from_sentence_transformer(other, st)
        assert not isinstance(gm2.tokenizer, DeviceBPE)
    finally:
        other.close()
