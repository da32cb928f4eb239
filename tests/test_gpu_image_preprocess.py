"""CLIP image preprocessing on the device (csrc/imgproc.cuh, rse_image_preprocess / rse_encode_images_u8): pixel_values
bit-identical to transformers' CLIPImageProcessor (torchvision backend) and CLIPImageProcessorPil, for the default 224
configuration and the 64-pixel test configuration, over mixed sizes in one call; embeddings from uint8 pixels
bit-identical to encode_pixels of the processor's output; search_with_image(s) identical to the host route; oversize
images and unsupported processors on the host route."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")
transformers = pytest.importorskip("transformers")
Image = pytest.importorskip("PIL.Image")

from rag_search_engine_b200 import _lib  # noqa: E402
from rag_search_engine_b200.clip import DeviceImageProcessor, GpuClipModel, clip_configs_from_hf  # noqa: E402

SMALL = dict(hidden_size=64, num_hidden_layers=1, num_attention_heads=2, intermediate_size=128, patch_size=16)
TEXT = dict(hidden_size=64, num_hidden_layers=1, num_attention_heads=2, intermediate_size=128, vocab_size=1000,
            max_position_embeddings=16)

# (H, W): down- and upscales, an exact-224 image, 1 x N and N x 1, odd and prime sizes, both orientations
SIZES = [(256, 320), (320, 256), (224, 224), (224, 300), (1, 7), (250, 1), (1, 250), (97, 211), (211, 97),
         (1500, 2000), (37, 41), (64, 64), (63, 65), (3, 5), (5, 3), (2731, 1223), (700, 7), (7, 700)]


def _procs(se):
    kw = dict(size={"shortest_edge": se}, crop_size={"height": se, "width": se})
    return {"torchvision": transformers.CLIPImageProcessor(**kw), "pil": transformers.CLIPImageProcessorPil(**kw)}


def _images(seed, sizes):
    rng = np.random.default_rng(seed)
    out = []
    for k, (h, w) in enumerate(sizes):
        if k % 2:                                   # smooth content as well as noise
            y, x = np.mgrid[0:h, 0:w]
            a = np.stack([(x * 255 // max(w - 1, 1)), (y * 255 // max(h - 1, 1)), ((x + y) * 7) % 256], -1)
            a = np.clip(a + rng.integers(-20, 21, a.shape), 0, 255).astype(np.uint8)
        else:
            a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        out.append(Image.fromarray(a))
    return out


def _clip_model(image_size, seed=3):
    cfg = transformers.CLIPConfig(text_config=dict(TEXT, eos_token_id=999, bos_token_id=998, pad_token_id=1),
                                  vision_config=dict(SMALL, image_size=image_size), projection_dim=48)
    torch.manual_seed(seed)
    return transformers.CLIPModel(cfg).eval()


def _gm(idx, model, proc):
    vision, text = clip_configs_from_hf(model.config)
    gm = GpuClipModel(idx, model.state_dict(), vision, text, tokenizer=lambda t: [[998, 5, 999] for _ in t],
                      image_processor=lambda ims: proc(ims, return_tensors="np")["pixel_values"])
    gm.device_image_processor = DeviceImageProcessor.maybe(idx, proc, gm.vision_slot, vision["image_size"])
    return gm


@pytest.mark.parametrize("se", [224, 64])
@pytest.mark.parametrize("backend", ["torchvision", "pil"])
def test_pixel_values_bit_identical_mixed_sizes(se, backend, fresh_index):
    print("aten CPU capability of the reference:", torch.backends.cpu.get_cpu_capability())
    proc = _procs(se)[backend]
    model = _clip_model(se)
    vision, _ = clip_configs_from_hf(model.config)
    fresh_index.clip_create(0, **vision)
    dp = DeviceImageProcessor.maybe(fresh_index, proc, 0, se)
    assert dp is not None and dp.backend == (1 if backend == "pil" else 0)
    images = _images(11, SIZES)
    want = proc(images, return_tensors="np")["pixel_values"]
    got = fresh_index.image_preprocess(0, [np.asarray(im) for im in images])
    assert got.shape == want.shape == (len(SIZES), 3, se, se)
    bad = [SIZES[i] for i in range(len(SIZES)) if not np.array_equal(got[i].view(np.uint32), want[i].view(np.uint32))]
    assert not bad, f"{backend} {se}: differ for {bad}"
    # one image per call gives the same bits as the batch
    for i in (0, 4, 9):
        assert np.array_equal(fresh_index.image_preprocess(0, [np.asarray(images[i])])[0].view(np.uint32),
                              want[i].view(np.uint32))


def test_many_chunks_and_rescale_variants(fresh_index):
    """More than one 64 MB staging chunk in one call (the copy of chunk i + 1 overlapping chunk i's kernels), and the
    processors' rescale-only / normalise-only / neither arithmetic."""
    model = _clip_model(64)
    vision, _ = clip_configs_from_hf(model.config)
    fresh_index.clip_create(0, **vision)
    images = _images(5, [(2000, 1500), (1500, 2000)] * 6 + [(33, 47), (2048, 2048)])     # ~120 MB of pixels
    for backend in ("torchvision", "pil"):
        for flags in (dict(), dict(do_normalize=False), dict(do_rescale=False), dict(do_rescale=False, do_normalize=False)):
            cls = transformers.CLIPImageProcessorPil if backend == "pil" else transformers.CLIPImageProcessor
            proc = cls(size={"shortest_edge": 64}, crop_size={"height": 64, "width": 64}, **flags)
            assert DeviceImageProcessor.maybe(fresh_index, proc, 0, 64) is not None
            want = np.asarray(proc(images, return_tensors="np")["pixel_values"], np.float32)
            got = fresh_index.image_preprocess(0, [np.asarray(im) for im in images])
            assert np.array_equal(got.view(np.uint32), want.view(np.uint32)), (backend, flags)


@pytest.mark.parametrize("backend", ["torchvision", "pil"])
def test_embeddings_from_uint8_bit_identical(backend, fresh_index):
    proc = _procs(64)[backend]
    gm = _gm(fresh_index, _clip_model(64), proc)
    assert gm.device_image_processor is not None
    images = _images(21, SIZES)
    want = gm.encode_pixels(proc(images, return_tensors="np")["pixel_values"])
    got = gm.encode(images)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert gm.device_image_processor.host_images == 0
    # the device-output variant
    out = torch.empty((len(images), 48), dtype=torch.float32, device="cuda")
    fresh_index.encode_images_u8_dev(gm.vision_slot, [np.asarray(im) for im in images], out.data_ptr())
    torch.cuda.synchronize()
    assert np.array_equal(out.cpu().numpy().view(np.uint32), want.view(np.uint32))


def test_oversize_and_unsupported_take_the_host_route(fresh_index):
    proc = _procs(64)["torchvision"]
    gm = _gm(fresh_index, _clip_model(64), proc)
    big = Image.fromarray(np.random.default_rng(2).integers(0, 256, (4100, 4100, 3), dtype=np.uint8))
    tall = Image.fromarray(np.random.default_rng(3).integers(0, 256, (7000, 66, 3), dtype=np.uint8))   # shrinks to 6787
    small = _images(4, [(90, 120)])[0]
    items = [small, big, tall]
    want = gm.encode_pixels(proc(items, return_tensors="np")["pixel_values"])
    got = gm.encode(items)
    assert np.array_equal(got.view(np.uint32), want.view(np.uint32))
    assert gm.device_image_processor.host_images == 1                 # the big one; torchvision numerics take the tall one
    with pytest.raises(_lib.RseError, match="RSE_IMGPROC_MAX_PIXELS"):
        fresh_index.image_preprocess(gm.vision_slot, [np.asarray(big)])
    # Pillow shrinks an image over 100 times taller than wide vertically first: host route for the Pil numerics
    pil = _procs(64)["pil"]
    dp = DeviceImageProcessor.maybe(fresh_index, pil, gm.vision_slot, 64)
    assert dp.array(tall) is None and dp.array(small) is not None
    with pytest.raises(_lib.RseError, match="taller"):
        fresh_index.image_preprocess(gm.vision_slot, [np.asarray(tall)])
    # an unsupported processor leaves the host route exactly as before
    bil = transformers.CLIPImageProcessor(size={"shortest_edge": 64}, crop_size={"height": 64, "width": 64},
                                          resample=2)
    assert DeviceImageProcessor.maybe(fresh_index, bil, gm.vision_slot, 64) is None


def test_abi_errors(fresh_index):
    model = _clip_model(64)
    vision, text = clip_configs_from_hf(model.config)
    fresh_index.clip_create(0, **vision)
    fresh_index.clip_create(1, **text)
    a = [np.zeros((10, 10, 3), np.uint8)]
    with pytest.raises(_lib.RseError) as e:
        fresh_index.image_preprocess(0, a)
    assert e.value.code == -3                                         # no configuration
    with pytest.raises(_lib.RseError) as e:
        fresh_index.imgproc_set(1, backend=0, shortest_edge=64, crop_height=64, crop_width=64, rescale_factor=1 / 255,
                                mean=[0.5] * 3, std=[0.5] * 3)
    assert e.value.code == -1                                         # not a vision tower
    with pytest.raises(_lib.RseError) as e:
        fresh_index.imgproc_set(0, backend=0, shortest_edge=64, crop_height=32, crop_width=32, rescale_factor=1 / 255,
                                mean=[0.5] * 3, std=[0.5] * 3)
    assert e.value.code == -4                                         # crop is not the tower's image_size


@pytest.mark.parametrize("backend", ["torchvision", "pil"])
def test_search_with_images_identical_to_host_route(backend, tmp_path):
    from rag_search_engine_b200.multimodal import MultimodalSearch
    proc = _procs(64)[backend]
    model = _clip_model(64)
    rng = np.random.default_rng(8)
    docs = [{"id": i, "title": f"t{i}", "description": f"d{i}"} for i in range(500)]
    paths = []
    for k, im in enumerate(_images(9, [(256, 320), (300, 200), (64, 64), (1, 50), (500, 499)] * 3)):
        p = tmp_path / f"q{k}.png"
        im.save(p)
        paths.append(str(p))
    idx_d, idx_h = _lib.Index(0), _lib.Index(0)
    try:
        gd, gh = _gm(idx_d, model, proc), _gm(idx_h, model, proc)
        gh.device_image_processor = None
        emb = rng.standard_normal((500, 48)).astype(np.float32)

        class _Docs:                                     # the same document embeddings for both searches
            def __init__(self, gm):
                self.gm = gm

            def encode(self, items, convert_to_numpy=True, show_progress_bar=False, **kw):
                return emb if isinstance(items, list) and items and isinstance(items[0], str) else self.gm.encode(items)

        md, mh = MultimodalSearch(docs, model=_Docs(gd)), MultimodalSearch(docs, model=_Docs(gh))
        try:
            assert md.search_with_images(paths, top_k=10) == mh.search_with_images(paths, top_k=10)
            assert md.search_with_image(paths[0], top_k=10) == mh.search_with_image(paths[0], top_k=10)
            assert gd.device_image_processor.host_images == 0
        finally:
            md.close()
            mh.close()
    finally:
        idx_d.close()
        idx_h.close()
