"""CPU tests of the CLIP model's host side (rag_search_engine_b200.clip): the transformers config translation, the
state_dict filtering per tower, and the input-order handling of mixed text / image lists (against a fake index)."""
import numpy as np
import pytest

from rag_search_engine_b200.clip import GpuClipModel, clip_configs_from_hf, tower_tensors

transformers = pytest.importorskip("transformers")


def _clip_config(**text_kw):
    return transformers.CLIPConfig(
        text_config=dict(hidden_size=64, num_hidden_layers=1, num_attention_heads=2, intermediate_size=128,
                         vocab_size=100, max_position_embeddings=16, eos_token_id=99, **text_kw),
        vision_config=dict(hidden_size=64, num_hidden_layers=1, num_attention_heads=2, intermediate_size=128,
                           image_size=32, patch_size=8),
        projection_dim=48)


def test_configs_from_a_clip_config_and_from_each_tower():
    cfg = _clip_config()
    v, t = clip_configs_from_hf(cfg)
    assert v == dict(tower=0, hidden=64, layers=1, heads=2, intermediate=128, projection_dim=48, image_size=32,
                     patch_size=8, ln_eps=cfg.vision_config.layer_norm_eps)
    assert t == dict(tower=1, hidden=64, layers=1, heads=2, intermediate=128, projection_dim=48, vocab_size=100,
                     max_positions=16, eos_token_id=99, ln_eps=cfg.text_config.layer_norm_eps)
    vc = transformers.CLIPVisionConfig(hidden_size=64, num_attention_heads=2, image_size=32, patch_size=8,
                                       projection_dim=40)
    assert clip_configs_from_hf(vc)[1] is None and clip_configs_from_hf(vc)[0]["projection_dim"] == 40
    tc = transformers.CLIPTextConfig(hidden_size=64, num_attention_heads=2, eos_token_id=2)
    assert clip_configs_from_hf(tc)[0] is None and clip_configs_from_hf(tc)[1]["eos_token_id"] == 2


def test_configs_that_are_not_implemented_are_rejected():
    with pytest.raises(ValueError, match="quick_gelu"):
        clip_configs_from_hf(_clip_config(hidden_act="gelu"))
    with pytest.raises(ValueError, match="quick_gelu"):
        clip_configs_from_hf(transformers.CLIPVisionConfig(hidden_act="gelu_new"))
    with pytest.raises(ValueError, match="3-channel"):
        clip_configs_from_hf(transformers.CLIPVisionConfig(num_channels=1))
    with pytest.raises(ValueError, match="multiple of patch_size"):
        clip_configs_from_hf(transformers.CLIPVisionConfig(image_size=50, patch_size=16))
    with pytest.raises(ValueError, match="not a CLIP config"):
        clip_configs_from_hf(transformers.BertConfig.__new__(transformers.BertConfig))


def test_tower_tensors_split_a_clip_model_state_dict():
    torch = pytest.importorskip("torch")
    model = transformers.CLIPModel(_clip_config())
    sd = dict(model.state_dict())
    sd["text_model.embeddings.position_ids"] = torch.arange(16)            # integer buffers (older checkpoints)
    vis = dict(tower_tensors(sd, 0))
    txt = dict(tower_tensors(sd, 1))
    assert "visual_projection.weight" in vis and "vision_model.embeddings.class_embedding" in vis
    assert "text_projection.weight" in txt and "text_model.final_layer_norm.bias" in txt
    assert not any(k.startswith("text") for k in vis) and not any(k.startswith(("vision", "visual")) for k in txt)
    assert "logit_scale" not in vis and "logit_scale" not in txt
    assert not any("position_ids" in k for k in txt)
    assert len(vis) == 8 + 16 and len(txt) == 5 + 16                    # what rse_encoder_finalize counts
    assert all(a.dtype == np.float32 for a in vis.values())
    # a wrapper prefix is kept (the library ignores it)
    assert set(dict(tower_tensors({"0.model." + k: v for k, v in sd.items()}, 0))) == {"0.model." + k for k in vis}


class _FakeIndex:
    """Records what GpuClipModel asks of the library; a text of ids -> [len, sum, 0...], an image -> [-1, mean...]."""

    def __init__(self):
        self.calls = []

    def clip_create(self, slot, **cfg):
        self.calls.append(("create", slot, cfg["tower"]))

    def encoder_set_tensor(self, slot, name, a):
        pass

    def encoder_finalize(self, slot):
        self.calls.append(("finalize", slot))

    def encode(self, slot, ids, cu):
        self.calls.append(("encode", slot, len(cu) - 1))
        out = np.zeros((len(cu) - 1, 4), np.float32)
        for i in range(len(cu) - 1):
            seq = ids[cu[i]:cu[i + 1]]
            out[i, :2] = len(seq), seq.sum()
        return out

    def encode_images(self, slot, px):
        self.calls.append(("images", slot, px.shape[0]))
        out = np.zeros((px.shape[0], 4), np.float32)
        out[:, 0] = -1.0
        out[:, 1] = px.reshape(px.shape[0], -1).mean(1)
        return out


class _Img:
    """Stands in for a PIL image (size + mode); carries the value its fake pixels are filled with."""
    mode = "RGB"

    def __init__(self, v):
        self.v, self.size = v, (8, 8)


def _model(idx):
    v = dict(tower=0, hidden=64, layers=1, heads=2, intermediate=128, projection_dim=4, image_size=8, patch_size=4,
             ln_eps=1e-5)
    t = dict(tower=1, hidden=64, layers=1, heads=2, intermediate=128, projection_dim=4, vocab_size=100,
             max_positions=6, eos_token_id=99, ln_eps=1e-5)
    tok = lambda texts: [[1] + [len(w) for w in s.split()] + [99] for s in texts]                # noqa: E731
    img = lambda ims: {"pixel_values": np.stack([np.full((3, 8, 8), im.v, np.float32) for im in ims])}  # noqa: E731
    return GpuClipModel(idx, {}, v, t, tokenizer=tok, image_processor=img)


def test_mixed_lists_come_back_in_input_order():
    idx = _FakeIndex()
    m = _model(idx)
    assert idx.calls == [("create", 0, 0), ("finalize", 0), ("create", 1, 1), ("finalize", 1)]
    idx.calls.clear()
    out = m.encode(["ab c", _Img(0.5), "d", _Img(2.0), "eee ff g"])
    assert out.shape == (5, 4) and out.dtype == np.float32
    assert out[:, 0].tolist() == [4, -1, 3, -1, 5]                     # text: its length; image: -1
    assert out[1, 1] == 0.5 and out[3, 1] == 2.0
    assert out[0, 1] == 1 + 2 + 1 + 99 and out[2, 1] == 1 + 1 + 99
    assert idx.calls == [("encode", 1, 3), ("images", 0, 2)]          # one call per tower
    assert m.encode("ab c").shape == (4,) and m.encode(_Img(1.0))[1] == 1.0
    assert m.encode(["x"] * 3).shape == (3, 4) and m.encode([_Img(3.0)]).shape == (1, 4)


def test_text_is_cut_to_max_positions_and_bulk_input_is_sliced():
    idx = _FakeIndex()
    m = _model(idx)
    idx.calls.clear()
    out = m.encode_ids([[1, 2, 3, 4, 5, 6, 7, 8], [1, 2]])
    assert out[:, 0].tolist() == [6, 2] and out[0, 1] == 21           # cut to max_positions = 6
    idx.calls.clear()
    ids = [[1, 2, 3]] * 10
    assert np.array_equal(m.encode_ids(ids, max_tokens_per_call=7), m.encode_ids(ids))
    assert [c[2] for c in idx.calls[:5]] == [2, 2, 2, 2, 2]
    idx.calls.clear()
    m.encode_pixels(np.zeros((5, 3, 8, 8), np.float32), max_images_per_call=2)
    assert [c[2] for c in idx.calls] == [2, 2, 1]


def test_missing_tokenizer_or_processor_is_an_error():
    idx = _FakeIndex()
    v = dict(tower=0, projection_dim=4, image_size=8, patch_size=4)
    t = dict(tower=1, projection_dim=4, max_positions=6)
    m = GpuClipModel(idx, {}, v, t)
    with pytest.raises(RuntimeError, match="tokenizer"):
        m.encode(["a"])
    with pytest.raises(RuntimeError, match="image processor"):
        m.encode([_Img(1.0)])
    with pytest.raises(ValueError, match="projection_dim"):
        GpuClipModel(idx, {}, dict(v, projection_dim=5), t)
