"""GPU: the CLIP towers of csrc/clip.cuh (§10 f4) against transformers' fp32 CLIP models.

The reference's clip-ViT-B-32 checkpoint cannot be downloaded here, so the oracle is transformers' own
CLIPVisionModelWithProjection / CLIPTextModelWithProjection / CLIPModel with the same architecture and seeded random
weights, perturbed away from the initialiser so LayerNorm gains, biases, the class embedding and the position tables
all matter.  The oracles run on the same GPU in fp32 with TF32 off (and in fp64 for the error budget).

Tolerance (floating point, stated here): normwise relative error of the embedding <= 1e-5 against fp32 PyTorch,
<= 5e-6 against fp64, the two GEMM modes <= 5e-6 apart.
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
transformers = pytest.importorskip("transformers")

EOS, BOS = 49407, 49406
B32_VISION = dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                  image_size=224, patch_size=32, projection_dim=512)
B32_TEXT = dict(hidden_size=512, num_hidden_layers=12, num_attention_heads=8, intermediate_size=2048,
                vocab_size=49408, max_position_embeddings=77, projection_dim=512)
SMALL_VISION = dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
                    image_size=64, patch_size=16, projection_dim=96)
SMALL_TEXT = dict(hidden_size=128, num_hidden_layers=2, num_attention_heads=2, intermediate_size=512,
                  vocab_size=49408, max_position_embeddings=77, projection_dim=96)


@pytest.fixture(autouse=True, scope="module")
def _no_tf32():
    old = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    yield
    torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = old


def _randomise(model, seed):
    g = torch.Generator().manual_seed(seed)
    with torch.no_grad():
        for name, p in model.named_parameters():
            if "norm" in name and name.endswith("weight"):
                p.copy_(1.0 + 0.1 * torch.randn(p.shape, generator=g))
            elif name.endswith("bias"):
                p.copy_(0.05 * torch.randn(p.shape, generator=g))
            elif "embedding" in name and "patch_embedding" not in name:
                p.copy_(0.5 * torch.randn(p.shape, generator=g))
            elif p.dim() >= 2:
                p.copy_(torch.randn(p.shape, generator=g) / (p[0].numel() ** 0.5))
    return model.eval()


def _vision_model(cfg, seed):
    c = transformers.CLIPVisionConfig(**cfg, attn_implementation="eager")
    return _randomise(transformers.CLIPVisionModelWithProjection(c), seed)


def _text_model(cfg, seed, eos=EOS):
    c = transformers.CLIPTextConfig(**cfg, eos_token_id=eos, bos_token_id=BOS, pad_token_id=1,
                                    attn_implementation="eager")
    return _randomise(transformers.CLIPTextModelWithProjection(c), seed)


def _relerr(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.linalg.norm(a - b, axis=-1).max() / max(1e-30, np.linalg.norm(b, axis=-1).min()))


def _ref_images(model, px, dtype):
    m = model.to("cuda", dtype)
    with torch.no_grad():
        out = m(pixel_values=torch.from_numpy(px).to("cuda", dtype)).image_embeds
    model.to("cpu", torch.float32)
    return out.double().cpu().numpy()


def _ref_texts(model, id_lists, dtype):
    S = max(len(x) for x in id_lists)
    ids = np.zeros((len(id_lists), S), np.int64)
    mask = np.zeros_like(ids)
    for i, x in enumerate(id_lists):
        ids[i, :len(x)] = x
        mask[i, :len(x)] = 1
    m = model.to("cuda", dtype)
    with torch.no_grad():
        out = m(input_ids=torch.from_numpy(ids).cuda(), attention_mask=torch.from_numpy(mask).cuda()).text_embeds
    model.to("cpu", torch.float32)
    return out.double().cpu().numpy()


def _load(index, slot, model, tower):
    from rag_search_engine_b200.clip import clip_configs_from_hf, tower_tensors
    cfg = clip_configs_from_hf(model.config)[tower]
    index.clip_create(slot, **cfg)
    for name, a in tower_tensors(model.state_dict(), tower):
        index.encoder_set_tensor(slot, name, a)
    index.encoder_finalize(slot)
    return cfg


def _texts(seed, n, lo, hi, eos=EOS):
    """BOS, random tokens, EOS somewhere (often not last: tokens after it), sometimes the largest id twice."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        L = int(rng.integers(lo, hi + 1))
        x = rng.integers(3, 49000, L).tolist()
        x[0] = BOS
        e = int(rng.integers(1, L)) if L > 1 else 0
        x[e] = eos if eos != 2 else 49407
        if eos == 2 and L > 3 and rng.random() < 0.5:
            x[int(rng.integers(e + 1, L)) if e + 1 < L else 0] = 49407       # a tie for the argmax: the first wins
        out.append(x)
    return out


@pytest.mark.parametrize("cfg", [B32_VISION, SMALL_VISION], ids=["vit_b32", "small"])
def test_vision_tower_matches_fp32_pytorch(cfg, fresh_index):
    model = _vision_model(cfg, 1)
    _load(fresh_index, 0, model, 0)
    rng = np.random.default_rng(2)
    S = cfg["image_size"]
    for n in (1, 7, 64):
        px = rng.standard_normal((n, 3, S, S)).astype(np.float32)
        ref32 = _ref_images(model, px, torch.float32)
        got = {}
        for mode in (0, 1):
            fresh_index.encoder_set_mode(0, mode)
            got[mode] = fresh_index.encode_images(0, px)
            assert got[mode].shape == (n, cfg["projection_dim"])
            e = _relerr(got[mode], ref32)
            assert e <= 1e-5, f"image_embeds differ from fp32 PyTorch by {e:.2e} (n={n}, mode {mode})"
        assert _relerr(got[0], got[1]) <= 5e-6
    ref64 = _ref_images(model, px, torch.float64)
    theirs = _relerr(ref32, ref64)
    for mode in (0, 1):
        ours = _relerr(got[mode], ref64)
        print(f"vision {cfg['hidden_size']}: error vs fp64: librse mode {mode} {ours:.2e}, PyTorch fp32 {theirs:.2e}")
        assert ours <= 5e-6
    fresh_index.encoder_set_mode(0, 0)
    # the device-pixel entry point gives the same bits
    pdev = torch.from_numpy(px).cuda()
    odev = torch.empty((px.shape[0], cfg["projection_dim"]), dtype=torch.float32, device="cuda")
    fresh_index.encode_images_dev(0, pdev.data_ptr(), px.shape[0], odev.data_ptr())
    fresh_index.synchronize()
    assert np.array_equal(odev.cpu().numpy(), got[0])


@pytest.mark.parametrize("cfg", [B32_TEXT, SMALL_TEXT], ids=["vit_b32", "small"])
@pytest.mark.parametrize("eos", [EOS, 2])
def test_text_tower_matches_fp32_pytorch(cfg, eos, fresh_index):
    from rag_search_engine_b200._lib import RseError
    model = _text_model(cfg, 3, eos)
    _load(fresh_index, 1, model, 1)
    ids = _texts(4, 64, 2, 77, eos)
    ref32 = _ref_texts(model, ids, torch.float32)
    got = {}
    for mode in (0, 1):
        fresh_index.encoder_set_mode(1, mode)
        from rag_search_engine_b200.encoder import pack
        flat, _, cu = pack(ids)
        got[mode] = fresh_index.encode(1, flat, cu)
        assert got[mode].shape == (64, cfg["projection_dim"])
        e = _relerr(got[mode], ref32)
        assert e <= 1e-5, f"text_embeds differ from fp32 PyTorch by {e:.2e} (mode {mode})"
    assert _relerr(got[0], got[1]) <= 5e-6
    ref64 = _ref_texts(model, ids, torch.float64)
    theirs = _relerr(ref32, ref64)
    for mode in (0, 1):
        ours = _relerr(got[mode], ref64)
        print(f"text {cfg['hidden_size']} eos {eos}: error vs fp64: librse mode {mode} {ours:.2e}, PyTorch fp32 {theirs:.2e}")
        assert ours <= 5e-6
    fresh_index.encoder_set_mode(1, 0)
    # GpuClipModel.encode_ids: over-long input is cut on the host, equal to encoding the cut ids; empty is refused
    from rag_search_engine_b200.clip import GpuClipModel
    gm = GpuClipModel.__new__(GpuClipModel)
    gm.index, gm.text_slot, gm.max_positions = fresh_index, 1, 77
    gm.text_config = dict(projection_dim=cfg["projection_dim"])
    long = _texts(5, 3, 90, 120, eos)
    assert np.array_equal(gm.encode_ids(long), gm.encode_ids([x[:77] for x in long]))
    assert np.array_equal(gm.encode_ids(ids, max_tokens_per_call=300), got[0])
    with pytest.raises(RseError, match="empty"):
        gm.encode_ids([[BOS, EOS], []])


class _StClip:
    """The reference's path on the CPU: sentence-transformers' CLIP encode = processor -> get_*_features."""

    def __init__(self, model, tok, proc):
        self.model, self.tok, self.proc = model, tok, proc

    def encode(self, items, convert_to_numpy=True, show_progress_bar=False, **_kw):
        from rag_search_engine_b200.clip import _is_image
        out = [None] * len(items)
        txt = [i for i, x in enumerate(items) if not _is_image(x)]
        img = [i for i, x in enumerate(items) if _is_image(x)]
        with torch.no_grad():
            for lo in range(0, len(txt), 256):
                part = txt[lo:lo + 256]
                ids = self.tok([items[i] for i in part])
                S = max(map(len, ids))
                a = torch.zeros((len(ids), S), dtype=torch.long)
                m = torch.zeros_like(a)
                for j, x in enumerate(ids):
                    a[j, :len(x)] = torch.tensor(x)
                    m[j, :len(x)] = 1
                r = self.model.get_text_features(input_ids=a, attention_mask=m)
                r = getattr(r, "pooler_output", r)
                for j, i in enumerate(part):
                    out[i] = r[j].numpy()
            if img:
                px = self.proc([items[i] for i in img], return_tensors="pt")["pixel_values"]
                r = self.model.get_image_features(pixel_values=px)
                r = getattr(r, "pooler_output", r)
                for j, i in enumerate(img):
                    out[i] = r[j].numpy()
        return np.stack(out).astype(np.float32)


def _word_tok(texts):
    import zlib
    return [[BOS] + [3 + zlib.crc32(w.encode()) % 49000 for w in t.lower().split()][:75] + [EOS] for t in texts]


def test_multimodal_search_drop_in(tmp_path):
    from PIL import Image
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.clip import GpuClipModel, clip_configs_from_hf
    from rag_search_engine_b200.multimodal import MultimodalSearch
    vc = {k: v for k, v in SMALL_VISION.items() if k != "projection_dim"}
    tc = {k: v for k, v in SMALL_TEXT.items() if k != "projection_dim"}
    cfg = transformers.CLIPConfig(text_config=dict(tc, eos_token_id=EOS, bos_token_id=BOS, pad_token_id=1),
                                  vision_config=vc, projection_dim=96)
    model = _randomise(transformers.CLIPModel(cfg), 7)
    proc = transformers.CLIPImageProcessor(size={"shortest_edge": 64}, crop_size={"height": 64, "width": 64})
    rng = np.random.default_rng(8)
    words = [f"w{i}" for i in range(300)]
    docs = [{"id": 5 + 2 * i, "title": " ".join(rng.choice(words, 2)),
             "description": " ".join(rng.choice(words, int(rng.integers(5, 40))))} for i in range(3000)]
    img = Image.fromarray(rng.integers(0, 256, (224, 224, 3), dtype=np.uint8))
    path = tmp_path / "query.png"
    img.save(path)
    vision, text = clip_configs_from_hf(model.config)
    idx = _lib.Index(0)
    try:
        gm = GpuClipModel(idx, model.state_dict(), vision, text, tokenizer=_word_tok,
                          image_processor=lambda ims: proc(ims, return_tensors="np")["pixel_values"])
        st = _StClip(model, _word_tok, proc)
        ms_gpu = MultimodalSearch(docs, model=gm)
        ms_cpu = MultimodalSearch(docs, model=st)
        try:
            assert _relerr(ms_gpu.text_embeddings, ms_cpu.text_embeddings) <= 1e-5
            a = ms_gpu.search_with_image(str(path), top_k=20)
            b = ms_cpu.search_with_image(str(path), top_k=20)
            assert len(a) == len(b) == 20
            assert all(list(x) == ["id", "title", "description", "similarity"] for x in a)
            sims = np.array([x["similarity"] for x in b])
            assert np.abs(np.array([x["similarity"] for x in a]) - sims).max() <= 1e-5
            tol = 2e-5
            for j in range(20):
                gap_prev = sims[j - 1] - sims[j] if j > 0 else np.inf
                gap_next = sims[j] - sims[j + 1] if j + 1 < 20 else np.inf
                if min(gap_prev, gap_next) > tol:
                    assert a[j]["id"] == b[j]["id"], f"rank {j}: {a[j]['id']} vs {b[j]['id']}"
            # a mixed list comes back in input order, equal to the single-kind encodes
            im2 = Image.fromarray(rng.integers(0, 256, (80, 100, 3), dtype=np.uint8))
            items = ["w1 w2 w3", img.convert("RGB"), "w9", im2]
            mixed = gm.encode(items)
            assert mixed.shape == (4, 96)
            assert np.array_equal(mixed[[0, 2]], gm.encode(["w1 w2 w3", "w9"]))
            assert np.array_equal(mixed[[1, 3]], gm.encode([img.convert("RGB"), im2]))
            assert _relerr(mixed, st.encode(items)) <= 1e-5
            assert gm.encode("w1 w2 w3").shape == (96,)
        finally:
            ms_gpu.close()
            ms_cpu.close()
    finally:
        idx.close()


def test_clip_abi_error_paths(fresh_index):
    from rag_search_engine_b200._lib import RseError
    idx = fresh_index
    text = _text_model(SMALL_TEXT, 11)
    vision = _vision_model(SMALL_VISION, 12)
    from rag_search_engine_b200.clip import clip_configs_from_hf, tower_tensors
    vcfg = clip_configs_from_hf(vision.config)[0]
    tcfg = clip_configs_from_hf(text.config)[1]
    for bad in (dict(hidden=100), dict(heads=1), dict(image_size=70), dict(image_size=1024, patch_size=8),
                dict(tower=3)):
        with pytest.raises(RseError, match="unsupported"):
            idx.clip_create(0, **{**vcfg, **bad})
    with pytest.raises(RseError, match="unsupported"):
        idx.clip_create(1, **{**tcfg, "max_positions": 5000})
    with pytest.raises(RseError, match="bad arguments"):
        idx.clip_create(2, **vcfg)
    idx.clip_create(0, **vcfg)
    idx.clip_create(1, **tcfg)
    vsd = dict(tower_tensors(vision.state_dict(), 0))
    tsd = dict(tower_tensors(text.state_dict(), 1))
    with pytest.raises(RseError, match="element count"):
        idx.encoder_set_tensor(0, "vision_model.pre_layrnorm.weight", np.zeros(64, np.float32))
    with pytest.raises(RseError, match="unknown tensor"):
        idx.encoder_set_tensor(0, "vision_model.encoder.layers.0.self_attn.nope.weight", np.zeros(4, np.float32))
    with pytest.raises(RseError, match="not a CLIP vision"):
        idx.encoder_set_tensor(0, "text_model.final_layer_norm.weight", np.zeros(128, np.float32))
    with pytest.raises(RseError, match="layer index"):
        idx.encoder_set_tensor(0, "vision_model.encoder.layers.7.mlp.fc1.bias", np.zeros(512, np.float32))
    names = list(vsd)
    for n in names[:-1]:
        idx.encoder_set_tensor(0, "model." + n, vsd[n])                 # a wrapper prefix is ignored
    with pytest.raises(RseError, match="tensors were set"):
        idx.encoder_finalize(0)
    px = np.zeros((2, 3, 64, 64), np.float32)
    with pytest.raises(RseError, match="not finalized"):
        idx.encode_images(0, px)
    idx.encoder_set_tensor(0, "0.model." + names[-1], vsd[names[-1]])
    idx.encoder_finalize(0)
    for n, a in tsd.items():
        idx.encoder_set_tensor(1, n, a)
    idx.encoder_finalize(1)
    assert idx.encode_images(0, px).shape == (2, 96)
    ids, cu = np.array([BOS, 5, EOS], np.int32), np.array([0, 3], np.int32)
    assert idx.encode(1, ids, cu).shape == (1, 96)
    with pytest.raises(RseError, match="type_ids"):
        idx.encode(1, ids, cu, type_ids=np.zeros(3, np.int32))
    with pytest.raises(RseError, match="vision tower"):
        idx.encode(0, ids, cu)
    with pytest.raises(RseError, match="does not hold a CLIP vision"):
        idx.encode_images(1, px)
    with pytest.raises(RseError, match="n < 1"):
        idx.encode_images(0, px[:0])
    with pytest.raises(RseError, match="max_positions"):
        idx.encode(1, np.arange(80, dtype=np.int32), np.array([0, 80], np.int32))
