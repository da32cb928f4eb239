"""CPU tests of the CLIP image preprocessing's host side: tests/helpers/resample_ref.py (what csrc/imgproc.cuh is
written from) bit for bit against Pillow's Image.resize(BICUBIC) and torchvision's uint8 antialiased bicubic over a
sweep of sizes; the whole restated pipeline (resize, center crop, rescale / normalise) bit for bit against both CLIP
image processors; and DeviceImageProcessor's acceptance rules, size limits and routing (against a fake index)."""
import numpy as np
import pytest

from helpers import resample_ref as R

transformers = pytest.importorskip("transformers")
torch = pytest.importorskip("torch")
Image = pytest.importorskip("PIL.Image")

from rag_search_engine_b200.clip import DeviceImageProcessor, GpuClipModel, resized_size  # noqa: E402

# (H, W) -> (out_h, out_w): downscales 1.01x .. 20x, upscales to 3x, 1-wide / 1-tall, odd and prime sizes, an unchanged
# 224 edge, both orientations, Pillow's vertical-first case (H > 100 W, shrinking vertically)
SWEEP = [((227, 230), (224, 227)), ((256, 320), (224, 280)), ((320, 256), (280, 224)), ((4480, 300), (224, 15)),
         ((300, 4480), (15, 224)), ((1500, 2000), (224, 298)), ((2000, 1500), (298, 224)), ((97, 211), (224, 487)),
         ((211, 97), (487, 224)), ((1, 7), (224, 1568)), ((7, 1), (1568, 224)), ((1, 1), (3, 3)), ((224, 300), (224, 300)),
         ((224, 600), (224, 300)), ((600, 224), (300, 224)), ((331, 7), (993, 21)), ((13, 4481), (3, 97)),
         ((4481, 13), (97, 3)), ((75, 75), (224, 224)), ((2731, 1223), (500, 224)), ((8000, 60), (64, 5)),
         ((8000, 60), (7000, 64)), ((5, 3), (224, 134))]


def _torch_resize(a, oh, ow):
    from torchvision.transforms import InterpolationMode
    from torchvision.transforms.v2 import functional as F
    t = torch.from_numpy(np.ascontiguousarray(a)).permute(2, 0, 1).contiguous()
    return F.resize(t, [oh, ow], interpolation=InterpolationMode.BICUBIC, antialias=True).permute(1, 2, 0).numpy()


def _img(seed, h, w):
    rng = np.random.default_rng(seed)
    a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
    if seed % 2:                                             # smooth ramps with noise: mid-range sums
        y, x = np.mgrid[0:h, 0:w]
        a = np.clip(np.stack([x * 255 // max(w - 1, 1), y * 255 // max(h - 1, 1), (x + y) % 256], -1)
                    + rng.integers(-8, 9, a.shape), 0, 255).astype(np.uint8)
    return a


@pytest.mark.parametrize("k", range(len(SWEEP)))
def test_pil_bicubic_matches_pillow(k):
    (h, w), (oh, ow) = SWEEP[k]
    for seed in (k * 2, k * 2 + 1):
        a = _img(seed, h, w)
        want = np.asarray(Image.fromarray(a).resize((ow, oh), Image.BICUBIC))
        assert np.array_equal(R.pil_bicubic(a, ow, oh), want)


@pytest.mark.parametrize("k", range(len(SWEEP)))
def test_torch_u8_aa_bicubic_matches_torchvision(k):
    # aten's scalar (DEFAULT) dispatch differs from its AVX2 / AVX512 kernel for outputs 1 pixel wide; the restatement
    # and the device follow the vectorised kernel, which every x86 host with AVX2 runs
    (h, w), (oh, ow) = SWEEP[k]
    if torch.backends.cpu.get_cpu_capability() == "DEFAULT" and ow == 1:
        pytest.skip("aten's scalar path for 1-wide outputs")
    for seed in (k * 2, k * 2 + 1):
        a = _img(seed, h, w)
        assert np.array_equal(R.torch_u8_aa_bicubic(a, ow, oh), _torch_resize(a, oh, ow))


def test_the_two_resizes_differ():
    """Separate targets: the two libraries' uint8 results disagree by a count or two."""
    diff = 0
    for k, ((h, w), (oh, ow)) in enumerate(SWEEP[:8]):
        a = _img(k, h, w)
        d = np.abs(R.pil_bicubic(a, ow, oh).astype(int) - R.torch_u8_aa_bicubic(a, ow, oh).astype(int))
        assert d.max() <= 2
        diff += int(d.sum())
    assert diff > 0


def pixel_values_ref(a, backend, se, crop, rescale=True, normalize=True, mean=None, std=None, factor=1 / 255):
    """The device's whole pipeline on the host: resize, center crop, then the float step of imgproc_vpass_kernel."""
    mean = np.float32(mean if mean is not None else transformers.image_utils.OPENAI_CLIP_MEAN)
    std = np.float32(std if std is not None else transformers.image_utils.OPENAI_CLIP_STD)
    h, w = a.shape[:2]
    nh, nw = resized_size(h, w, se)
    x = (R.pil_bicubic if backend == "pil" else R.torch_u8_aa_bicubic)(a, nw, nh)
    top, left = (nh - crop) // 2, (nw - crop) // 2
    x = x[top:top + crop, left:left + crop].transpose(2, 0, 1)
    v = x.astype(np.float32)
    m, s = mean[:, None, None], std[:, None, None]
    if backend == "pil":
        if rescale:
            v = (x.astype(np.float64) * factor).astype(np.float32)
        return (v - m) / s if normalize else v
    if rescale and normalize:
        inv = np.float32(1.0 / factor)
        return (v - m * inv) / (s * inv)
    if normalize:
        return (v - m) / s
    return v * np.float32(factor) if rescale else v


@pytest.mark.parametrize("backend", ["torchvision", "pil"])
@pytest.mark.parametrize("se", [224, 64])
def test_restated_pipeline_matches_the_processors(backend, se):
    sizes = [(256, 320), (320, 256), (224, 224), (1, 300), (300, 1), (97, 211), (1500, 2000), (3, 5), (5, 3), (65, 64)]
    cls = transformers.CLIPImageProcessorPil if backend == "pil" else transformers.CLIPImageProcessor
    for flags in (dict(), dict(do_normalize=False), dict(do_rescale=False), dict(do_rescale=False, do_normalize=False)):
        proc = cls(size={"shortest_edge": se}, crop_size={"height": se, "width": se}, **flags)
        arrays = [_img(i, h, w) for i, (h, w) in enumerate(sizes)]
        want = np.asarray(proc([Image.fromarray(a) for a in arrays], return_tensors="np")["pixel_values"], np.float32)
        for i, a in enumerate(arrays):
            got = pixel_values_ref(a, backend, se, se, rescale=flags.get("do_rescale", True),
                                   normalize=flags.get("do_normalize", True)).astype(np.float32)
            assert np.array_equal(got.view(np.uint32), want[i].view(np.uint32)), (backend, se, flags, sizes[i])


def test_resized_size_and_crop_offsets_follow_the_processor():
    from transformers.image_transforms import get_resize_output_image_size
    for h, w in [(256, 320), (320, 256), (1, 7), (7, 1), (224, 224), (1500, 2000), (2731, 1223), (225, 301)]:
        for se in (224, 64, 77):
            assert resized_size(h, w, se) == R.resized_size(h, w, se) == \
                tuple(get_resize_output_image_size(np.zeros((3, h, w)), se, default_to_square=False,
                                                   input_data_format="channels_first"))


class _FakeIndex:
    def __init__(self):
        self.cfg, self.u8_calls, self.px_calls = None, [], []

    def imgproc_set(self, slot, **kw):
        self.cfg = dict(kw, slot=slot)

    def encode_images_u8(self, slot, arrays):
        self.u8_calls.append([a.shape for a in arrays])
        return np.stack([np.full(4, a.shape[0] * 10000 + a.shape[1], np.float32) for a in arrays])


def test_maybe_accepts_both_default_clip_processors():
    for cls, backend in ((transformers.CLIPImageProcessor, 0), (transformers.CLIPImageProcessorPil, 1)):
        idx = _FakeIndex()
        dp = DeviceImageProcessor.maybe(idx, cls(), 0, 224)
        assert dp is not None and dp.backend == backend
        assert idx.cfg["backend"] == backend and idx.cfg["shortest_edge"] == 224 and idx.cfg["crop_height"] == 224
        assert idx.cfg["mean"] == list(transformers.image_utils.OPENAI_CLIP_MEAN)
        assert idx.cfg["rescale_factor"] == 1 / 255 and idx.cfg["do_rescale"] and idx.cfg["do_normalize"]


@pytest.mark.parametrize("kw", [dict(resample=2), dict(resample=1), dict(size={"height": 224, "width": 224}),
                                dict(size={"shortest_edge": 224, "longest_edge": 400}), dict(do_center_crop=False),
                                dict(crop_size={"height": 200, "width": 200}),
                                dict(crop_size={"height": 224, "width": 200}),
                                dict(size={"shortest_edge": 200}), dict(do_resize=False), dict(do_pad=True),
                                dict(image_mean=[0.5, 0.5]), dict(image_std=[0.5, 0.0, 0.5])])
def test_maybe_rejects_each_unsupported_setting(kw):
    for cls in (transformers.CLIPImageProcessor, transformers.CLIPImageProcessorPil):
        assert DeviceImageProcessor.maybe(_FakeIndex(), cls(**kw), 0, 224) is None
    assert DeviceImageProcessor.maybe(_FakeIndex(), transformers.CLIPImageProcessor(), 0, 64) is None  # crop != tower
    assert DeviceImageProcessor.maybe(_FakeIndex(), object(), 0, 224) is None
    assert DeviceImageProcessor.maybe(_FakeIndex(), transformers.ViTImageProcessor(), 0, 224) is None


def test_device_limits():
    dp = DeviceImageProcessor(_FakeIndex(), transformers.CLIPImageProcessor(), 0)
    dpp = DeviceImageProcessor(_FakeIndex(), transformers.CLIPImageProcessorPil(), 0)
    assert dp.device_ok(4096, 4096) and not dp.device_ok(4097, 4096)               # 2^24 pixels
    dp64 = DeviceImageProcessor(_FakeIndex(), transformers.CLIPImageProcessor(size={"shortest_edge": 64}), 0)
    assert dp64.device_ok(2048, 2048) and not dp64.device_ok(2049, 2049)            # downscale <= 32 per axis
    assert dp.device_ok(1, 292) and not dp.device_ok(1, 293)                         # resized side <= 65536
    assert dp.device_ok(23000, 229) and not dpp.device_ok(23000, 229)                # Pillow's vertical-first case
    assert dpp.device_ok(20000, 200) and dpp.device_ok(3000, 20)                     # 100:1 exactly / upscaling


def test_encode_routes_device_and_host_images_in_input_order():
    idx = _FakeIndex()
    host_calls = []

    def host(images):
        host_calls.append(len(images))
        return np.zeros((len(images), 3, 224, 224), np.float32)

    gm = GpuClipModel.__new__(GpuClipModel)
    gm.index, gm.vision_slot, gm.image_processor = idx, 0, host
    gm.text_config = {"projection_dim": 4}
    gm.encode_pixels = lambda px, n=256: np.full((px.shape[0], 4), -1.0, np.float32)
    gm.device_image_processor = DeviceImageProcessor(idx, transformers.CLIPImageProcessor(), 0)
    ims = [Image.fromarray(np.zeros((10, 20, 3), np.uint8)), Image.fromarray(np.zeros((5000, 5000, 3), np.uint8)),
           Image.fromarray(np.zeros((30, 40), np.uint8)), Image.fromarray(np.zeros((11, 12, 4), np.uint8))]
    out = gm.encode(ims)
    assert out[0, 0] == 10 * 10000 + 20 and out[1, 0] == -1.0
    assert out[2, 0] == 30 * 10000 + 40 and out[3, 0] == 11 * 10000 + 12           # L and RGBA converted to RGB
    assert gm.device_image_processor.host_images == 1 and host_calls == [1]
    gm.device_image_processor = None                                               # no device processor: host only
    assert np.all(gm.encode(ims) == -1.0) and host_calls == [1, 4]
