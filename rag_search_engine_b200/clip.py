"""The CLIP model of the image search on the GPU (§10 f4).

``GpuClipModel`` stands in for ``SentenceTransformer("clip-ViT-B-32")`` where ``MultimodalSearch`` uses it
(llm/multimodal.py:35-42 encodes every document text, :46-58 every query image): pass it as
``MultimodalSearch(documents, model=GpuClipModel(...))``.  Both towers run csrc/clip.cuh through the C-ABI
(``rse_clip_create``, ``rse_encode`` for text, ``rse_encode_images`` for images) in fp32; the output is what
sentence-transformers' CLIP ``encode`` returns: ``get_text_features`` / ``get_image_features``, not normalised.

The tokenizer is pluggable: ``DeviceBPE`` runs CLIP's byte-level BPE on the device (csrc/bpe.cuh, ids identical to
the HF fast tokenizer), and any callable ``texts -> token-id lists`` (or a HuggingFace tokenizer) runs on the host;
the image processor is any callable ``images -> pixel_values [n, 3, S, S]`` (or a HuggingFace image processor).
Image decoding stays on the host.  ``from_sentence_transformer`` takes the weights, the tokenizer and the image
processor from a loaded reference model; its tokenizer goes on the device when ``bpe.build_bpe_tables`` accepts it,
and when the image processor is a CLIP one ``DeviceImageProcessor`` accepts, the resize, crop and normalisation run
on the device (csrc/imgproc.cuh) from the decoded uint8 pixels, bit for bit what the processor returns.  No weights
are bundled and nothing is downloaded.
"""
from __future__ import annotations

import warnings
from typing import Iterator, List, Optional, Sequence, Tuple

import numpy as np

from ._lib import RSE_ERR_UNSUPPORTED, RseError
from .encoder import DeviceTokenizer, _utf8, pack

VISION_SLOT, TEXT_SLOT = 0, 1
_TOWER_KEYS = {0: ("vision_model.", "visual_projection."), 1: ("text_model.", "text_projection.")}


def _vision_config(v, projection_dim: int) -> dict:
    if getattr(v, "hidden_act", "quick_gelu") != "quick_gelu":
        raise ValueError(f"CLIP vision tower: only hidden_act='quick_gelu' is implemented, not {v.hidden_act!r}")
    if getattr(v, "num_channels", 3) != 3:
        raise ValueError("CLIP vision tower: only 3-channel images are implemented")
    if v.image_size % v.patch_size:
        raise ValueError("CLIP vision tower: image_size must be a multiple of patch_size")
    return dict(tower=0, hidden=v.hidden_size, layers=v.num_hidden_layers, heads=v.num_attention_heads,
                intermediate=v.intermediate_size, projection_dim=int(projection_dim), image_size=v.image_size,
                patch_size=v.patch_size, ln_eps=v.layer_norm_eps)


def _text_config(t, projection_dim: int) -> dict:
    if getattr(t, "hidden_act", "quick_gelu") != "quick_gelu":
        raise ValueError(f"CLIP text tower: only hidden_act='quick_gelu' is implemented, not {t.hidden_act!r}")
    return dict(tower=1, hidden=t.hidden_size, layers=t.num_hidden_layers, heads=t.num_attention_heads,
                intermediate=t.intermediate_size, projection_dim=int(projection_dim), vocab_size=t.vocab_size,
                max_positions=t.max_position_embeddings, eos_token_id=int(t.eos_token_id), ln_eps=t.layer_norm_eps)


def clip_configs_from_hf(cfg) -> Tuple[Optional[dict], Optional[dict]]:
    """transformers ``CLIPConfig`` -> ``(vision, text)`` keyword arguments of ``Index.clip_create``; a
    ``CLIPVisionConfig`` or ``CLIPTextConfig`` alone gives ``(vision, None)`` / ``(None, text)``.  A CLIPModel
    projects both towers to the top-level ``projection_dim``.  Raises ValueError for what is not implemented."""
    if hasattr(cfg, "vision_config") and hasattr(cfg, "text_config"):
        pd = cfg.projection_dim
        return _vision_config(cfg.vision_config, pd), _text_config(cfg.text_config, pd)
    model_type = getattr(cfg, "model_type", "")
    if model_type == "clip_vision_model":
        return _vision_config(cfg, cfg.projection_dim), None
    if model_type == "clip_text_model":
        return None, _text_config(cfg, cfg.projection_dim)
    raise ValueError(f"not a CLIP config: {type(cfg).__name__}")


def tower_tensors(state_dict, tower: int) -> Iterator[Tuple[str, np.ndarray]]:
    """The float tensors of one tower (0 = vision, 1 = text) of a CLIPModel / CLIP*ModelWithProjection state_dict,
    as float32 arrays; the other tower, ``logit_scale`` and the integer ``position_ids`` buffers are left out."""
    keys = _TOWER_KEYS[int(tower)]
    for name, t in state_dict.items():
        if not any(k in name for k in keys) or name.endswith("position_ids"):
            continue
        a = t.detach().cpu().numpy() if hasattr(t, "detach") else np.asarray(t)
        if a.dtype.kind != "f":
            continue
        yield name, a.astype(np.float32, copy=False)


# per-image limits of the device preprocessing (include/rse.h RSE_IMGPROC_*): beyond them an image takes the host
# processor.  2^24 pixels (48 MB of RGB, e.g. 4096 x 4096) keeps every image inside one 64 MB staging chunk; a
# downscale of at most 32 per axis bounds the taps per output (129) and so the coefficient table.
MAX_PIXELS = 1 << 24
MAX_EDGE = 65536
MAX_SCALE = 32


def resized_size(h: int, w: int, shortest_edge: int) -> Tuple[int, int]:
    """transformers' ``get_resize_output_image_size(default_to_square=False)``: (new_h, new_w)."""
    short, long = (w, h) if w <= h else (h, w)
    new_short, new_long = shortest_edge, int(shortest_edge * long / short)
    return (new_long, new_short) if w <= h else (new_short, new_long)


def _size_dict(size) -> dict:
    if size is None:
        return {}
    keys = ("height", "width", "shortest_edge", "longest_edge", "max_height", "max_width")
    d = dict(size) if isinstance(size, dict) else {k: getattr(size, k, None) for k in keys}
    return {k: v for k, v in d.items() if v is not None}


class DeviceImageProcessor:
    """CLIP's image processor on the device: ``CLIPImageProcessor`` (torchvision backend) or ``CLIPImageProcessorPil``
    numerics, chosen from the processor object, bound to the vision tower in ``slot`` (``rse_imgproc_set``).

    ``maybe`` returns None for any configuration the device does not implement: another resample filter than BICUBIC,
    a size other than ``{"shortest_edge": n}``, no center crop, a crop other than the tower's square image_size or
    larger than the resized image (the processor would pad), ``do_pad``.  Images whose size is outside the device's
    limits (``device_ok``) go through the host processor and are counted in ``host_images``."""

    def __init__(self, index, hf_image_processor, slot: int):
        p = hf_image_processor
        self.index, self.slot, self.hf = index, int(slot), p
        self.backend = 1 if getattr(p, "backend", "torchvision") == "pil" else 0
        self.shortest_edge = int(_size_dict(p.size)["shortest_edge"])
        crop = _size_dict(p.crop_size)
        self.crop = int(crop["height"])
        self.do_convert_rgb = bool(getattr(p, "do_convert_rgb", True))
        self.host_images = 0
        index.imgproc_set(self.slot, backend=self.backend, shortest_edge=self.shortest_edge, crop_height=self.crop,
                          crop_width=int(crop["width"]), rescale_factor=float(p.rescale_factor),
                          mean=list(p.image_mean), std=list(p.image_std), do_resize=True, do_center_crop=True,
                          do_rescale=bool(p.do_rescale), do_normalize=bool(p.do_normalize))

    @classmethod
    def supported(cls, hf_image_processor, image_size: int) -> bool:
        try:
            import transformers
        except ImportError:
            return False
        p = hf_image_processor
        kinds = tuple(getattr(transformers, n) for n in ("CLIPImageProcessor", "CLIPImageProcessorPil")
                      if hasattr(transformers, n))
        if not kinds or type(p) not in kinds:
            return False
        size, crop = _size_dict(getattr(p, "size", None)), _size_dict(getattr(p, "crop_size", None))
        mean, std = getattr(p, "image_mean", None), getattr(p, "image_std", None)
        return (int(getattr(p, "resample", -1)) == 3                                    # PILImageResampling.BICUBIC
                and bool(getattr(p, "do_resize", False)) and bool(getattr(p, "do_center_crop", False))
                and not getattr(p, "do_pad", False)
                and set(size) == {"shortest_edge"} and set(crop) == {"height", "width"}
                and crop["height"] == crop["width"] == int(image_size) <= int(size["shortest_edge"]) <= MAX_EDGE
                and mean is not None and std is not None and len(mean) == 3 and len(std) == 3
                and all(float(x) != 0.0 for x in std) and float(getattr(p, "rescale_factor", 0.0)) > 0.0)

    @classmethod
    def maybe(cls, index, hf_image_processor, slot: int, image_size: int) -> Optional["DeviceImageProcessor"]:
        """A DeviceImageProcessor for ``hf_image_processor`` on the vision tower of ``image_size`` in ``slot``, or None
        when the device does not implement its configuration."""
        return cls(index, hf_image_processor, slot) if cls.supported(hf_image_processor, image_size) else None

    def device_ok(self, h: int, w: int) -> bool:
        """Whether an h x w image is within the device's limits (else the host processor takes it)."""
        if h < 1 or w < 1 or h * w > MAX_PIXELS:
            return False
        nh, nw = resized_size(h, w, self.shortest_edge)
        if max(nh, nw) > MAX_EDGE or h > MAX_SCALE * nh or w > MAX_SCALE * nw:
            return False
        return not (self.backend == 1 and h > 100 * w and nh < h)     # Pillow shrinks such an image vertically first

    def array(self, image) -> Optional[np.ndarray]:
        """A PIL image -> its [H, W, 3] uint8 pixels as the processor sees them (after its RGB conversion), or None
        when the host processor must take it."""
        if image.mode != "RGB":
            if not self.do_convert_rgb:
                return None
            from transformers.image_transforms import convert_to_rgb
            image = convert_to_rgb(image)
        a = np.asarray(image)
        if a.dtype != np.uint8 or a.ndim != 3 or a.shape[2] != 3 or not self.device_ok(a.shape[0], a.shape[1]):
            return None
        return a


class DeviceBPE(DeviceTokenizer):
    """CLIP's byte-level BPE tokenizer on the device (csrc/bpe.cuh) in a tokenizer slot of ``index``.

    Called on texts it returns what ``hf_tok(texts, add_special_tokens=..., truncation=..., max_length=...)
    ["input_ids"]`` returns; ``add_special_tokens`` / ``max_length`` fix which call it stands for (``max_length=None``:
    no cut).  ``GpuClipModel`` uses its device path instead, where the ids never become Python lists.  A text the
    device refuses goes to ``hf_tok``'s own Rust tokenizer on the host and is counted in ``host_texts``: a text with a
    code point NFC could join with its neighbours (``host_routed``, known up front), and, once the device reports one,
    every text that could hold a piece longer than its word buffer.  ``UnsupportedTokenizer`` when ``hf_tok`` is not
    the CLIP BPE pipeline; ``maybe`` returns None then."""

    def __init__(self, index, hf_tok, *, slot: int = 0, add_special_tokens: bool = True,
                 max_length: Optional[int] = None):
        from .bpe import build_bpe_tables, plain_backend
        self.tables = build_bpe_tables(hf_tok)
        self.backend = plain_backend(hf_tok)
        self.index, self.slot = index, int(slot)
        self.add_special_tokens = bool(add_special_tokens)
        self.max_length = None if max_length is None else int(max_length)
        self.bos_id, self.eos_id = self.tables.bos_id, self.tables.eos_id
        self.host_texts = 0
        index.tokenizer_load_bpe(self.slot, self.tables)

    def host_ids(self, texts, add_special: bool, max_length: Optional[int]) -> List[List[int]]:
        """The host tokenizer's ids under the same rule (the route of the texts the device refuses)."""
        from .bpe import host_ids
        self.host_texts += len(texts)
        return host_ids(self.backend, texts, add_special, max_length, self.bos_id, self.eos_id)

    def host_routed(self, texts, long_pieces: bool = False) -> List[int]:
        """The texts that go to the host: those with a code point NFC could join with its neighbours, and with
        ``long_pieces`` also those that could hold a piece longer than the device's word buffer."""
        t = self.tables
        return [i for i, x in enumerate(texts) if t.needs_host(x) or (long_pieces and t.may_overflow(x))]

    def run(self, texts, device, host):
        """``device(texts)`` on the texts the device takes and ``host(texts)`` on the rest -> (the device's result or
        None, the device's text indices, the host's result, the host's text indices)."""
        routed = self.host_routed(texts)
        for long_pieces in (False, True):
            if long_pieces:
                routed = self.host_routed(texts, True)
            at = set(routed)
            keep = [i for i in range(len(texts)) if i not in at]
            try:
                dev = device([texts[i] for i in keep]) if keep else None
                break
            except RseError as e:
                if long_pieces or e.code != RSE_ERR_UNSUPPORTED:
                    raise
        return dev, keep, (host([texts[i] for i in routed]) if routed else []), routed

    def tokenize(self, texts, add_special: Optional[bool] = None, max_length: Optional[int] = -1):
        """-> (ids int32[total], cu_seqlens int32[n + 1]) on the host; defaults are this object's call rule."""
        sp = self.add_special_tokens if add_special is None else bool(add_special)
        ml = self.max_length if max_length == -1 else max_length
        texts = list(texts)
        if not texts:
            return np.zeros(0, np.int32), np.zeros(1, np.int32)
        dev, keep, hst, routed = self.run(texts, lambda x: self.index.tokenize(self.slot, *_utf8(x), sp, ml or 0),
                                          lambda x: self.host_ids(x, sp, ml))
        if not routed:
            return dev
        got = dict(zip(routed, hst))
        if dev is not None:
            ids, cu = dev
            ids = ids.tolist()
            got.update((i, ids[a:b]) for i, a, b in zip(keep, cu[:-1].tolist(), cu[1:].tolist()))
        return pack([got[i] for i in range(len(texts))])[::2]


def _is_image(x) -> bool:
    return not isinstance(x, (str, bytes)) and hasattr(x, "size") and hasattr(x, "mode")      # a PIL image


class GpuClipModel:
    """``encode(items) -> float32[n, projection_dim]`` like sentence-transformers' CLIP model: strings through the
    text tower, PIL images through the vision tower, a mixed list split and returned in input order."""

    def __init__(self, index, state_dict, vision_config: dict, text_config: dict, tokenizer=None,
                 image_processor=None, *, vision_slot: int = VISION_SLOT, text_slot: int = TEXT_SLOT):
        if vision_config["projection_dim"] != text_config["projection_dim"]:
            raise ValueError("the two towers must project to the same projection_dim")
        self.index, self.vision_slot, self.text_slot = index, int(vision_slot), int(text_slot)
        self.vision_config, self.text_config = dict(vision_config, tower=0), dict(text_config, tower=1)
        self.tokenizer, self.image_processor = tokenizer, image_processor
        self.device_image_processor: Optional[DeviceImageProcessor] = None
        self.max_positions = int(self.text_config["max_positions"])
        sd = dict(state_dict)
        for slot, cfg in ((self.vision_slot, self.vision_config), (self.text_slot, self.text_config)):
            index.clip_create(slot, **cfg)
            for name, a in tower_tensors(sd, cfg["tower"]):
                index.encoder_set_tensor(slot, name, a)
            index.encoder_finalize(slot)

    @classmethod
    def from_sentence_transformer(cls, index, st_model, tok_slot: int = 0, **kw) -> "GpuClipModel":
        """From a loaded ``SentenceTransformer("clip-ViT-B-32")`` (llm/multimodal.py:28): its transformers
        ``CLIPModel`` weights, its processor's tokenizer (truncating to the text tower's length, as the
        processor does; a ``DeviceBPE`` in tokenizer slot ``tok_slot`` of ``index`` when the device takes it, which
        replaces whatever that slot held; a warning names the reason when it does not) and its image processor."""
        mod = st_model[0]
        model, proc = mod.model, mod.processor
        vision, text = clip_configs_from_hf(model.config)
        ml = int(text["max_positions"])
        tok = lambda texts: proc.tokenizer(list(texts), truncation=True, max_length=ml)["input_ids"]   # noqa: E731
        img = lambda images: proc.image_processor(list(images), return_tensors="np")["pixel_values"]   # noqa: E731
        m = cls(index, model.state_dict(), vision, text, tok, img, **kw)
        from .bpe import UnsupportedTokenizer
        try:
            m.tokenizer = DeviceBPE(index, proc.tokenizer, slot=tok_slot, max_length=ml)
        except UnsupportedTokenizer as e:
            warnings.warn(f"GpuClipModel: the CLIP tokenizer stays on the host ({e})")
        m.device_image_processor = DeviceImageProcessor.maybe(index, proc.image_processor, m.vision_slot,
                                                              vision["image_size"])
        return m

    def get_sentence_embedding_dimension(self) -> int:
        return int(self.text_config["projection_dim"])

    def encode_ids(self, id_lists: Sequence[Sequence[int]], max_tokens_per_call: int = 1 << 16) -> np.ndarray:
        """Token-id lists -> text embeddings.  Sequences are cut to max_positions; a bulk input (the document texts
        of an index build) goes through in slices of at most ``max_tokens_per_call`` tokens."""
        mp = self.max_positions
        id_lists = [x if len(x) <= mp else list(x)[:mp] for x in id_lists]
        out = np.empty((len(id_lists), self.get_sentence_embedding_dimension()), np.float32)
        lo = 0
        while lo < len(id_lists):
            hi, tok = lo, 0
            while hi < len(id_lists) and (hi == lo or tok + len(id_lists[hi]) <= max_tokens_per_call):
                tok += len(id_lists[hi]); hi += 1
            ids, _, cu = pack(id_lists[lo:hi])
            out[lo:hi] = self.index.encode(self.text_slot, ids, cu)
            lo = hi
        return out

    def encode_pixels(self, pixel_values, max_images_per_call: int = 256) -> np.ndarray:
        """pixel_values [n, 3, S, S] (the image processor's output) -> image embeddings, in slices of
        ``max_images_per_call`` images."""
        px = np.ascontiguousarray(pixel_values, np.float32)
        out = np.empty((px.shape[0], self.get_sentence_embedding_dimension()), np.float32)
        for lo in range(0, px.shape[0], max_images_per_call):
            out[lo:lo + max_images_per_call] = self.index.encode_images(self.vision_slot, px[lo:lo + max_images_per_call])
        return out

    def encode_images(self, images, max_images_per_call: int = 256) -> np.ndarray:
        """PIL images -> image embeddings.  With a ``device_image_processor`` the uint8 pixels go to the device
        (``rse_encode_images_u8``) and the float pixel_values never exist on the host; an image outside its limits,
        and every image without one, goes through the host image processor and ``encode_pixels``."""
        images = list(images)
        out = np.empty((len(images), self.get_sentence_embedding_dimension()), np.float32)
        dp = self.device_image_processor
        arrays = [dp.array(im) for im in images] if dp is not None else [None] * len(images)
        dev_at = [i for i, a in enumerate(arrays) if a is not None]
        host_at = [i for i, a in enumerate(arrays) if a is None]
        for lo in range(0, len(dev_at), max_images_per_call):
            at = dev_at[lo:lo + max_images_per_call]
            out[at] = self.index.encode_images_u8(self.vision_slot, [arrays[i] for i in at])
        if host_at:
            if dp is not None:
                dp.host_images += len(host_at)
            out[host_at] = self.encode_pixels(self._preprocess([images[i] for i in host_at]), max_images_per_call)
        return out

    def encode_texts(self, texts: Sequence[str]) -> np.ndarray:
        """Texts -> text embeddings.  With a ``DeviceBPE`` the texts the device takes are tokenized and encoded on the
        device (``rse_encode_texts``: their ids never leave it, the tower runs on slices of them cut at their real
        lengths) and the texts it refuses go through the host tokenizer and ``encode_ids``; without one every text
        takes the host path.  A text's embedding does not depend on the slice it is encoded in, so the result is the
        same either way, bit for bit."""
        texts = list(texts)
        tok = self.tokenizer
        if not texts or not isinstance(tok, DeviceBPE):
            return self.encode_ids(self._tokenize(texts))
        mp = self.max_positions
        out = np.empty((len(texts), self.get_sentence_embedding_dimension()), np.float32)
        dev, keep, hst, routed = tok.run(
            texts, lambda x: self.index.encode_texts(tok.slot, self.text_slot, *_utf8(x), mp),
            lambda x: self.encode_ids(tok.host_ids(x, True, mp)))
        if dev is not None:
            out[keep] = dev
        if routed:
            out[routed] = hst
        return out

    def _tokenize(self, texts):
        if self.tokenizer is None:
            raise RuntimeError("GpuClipModel has no tokenizer: pass tokenizer=<texts -> token-id lists> "
                               "(e.g. the reference model's CLIP tokenizer) or call encode_ids")
        ids = self.tokenizer(list(texts))
        return ids["input_ids"] if hasattr(ids, "keys") else ids

    def _preprocess(self, images):
        if self.image_processor is None:
            raise RuntimeError("GpuClipModel has no image processor: pass image_processor=<images -> pixel_values> "
                               "(e.g. the reference model's CLIP image processor) or call encode_pixels")
        px = self.image_processor(list(images))
        return np.asarray(px["pixel_values"] if hasattr(px, "keys") else px, np.float32)

    def encode(self, items, convert_to_numpy: bool = True, show_progress_bar: bool = False, **_kw) -> np.ndarray:
        single = isinstance(items, str) or _is_image(items)
        items = [items] if single else list(items)
        out = np.empty((len(items), self.get_sentence_embedding_dimension()), np.float32)
        img_at = [i for i, x in enumerate(items) if _is_image(x)]
        txt_at = [i for i, x in enumerate(items) if not _is_image(x)]
        if txt_at:
            out[txt_at] = self.encode_texts([items[i] for i in txt_at])
        if img_at:
            out[img_at] = self.encode_images([items[i] for i in img_at])
        return out[0] if single else out
