"""CLIP towers on the device (§10 f4): throughput of the vision and text towers, search_with_image end to end, and
the same towers in PyTorch fp32 on the same GPU and on the host CPU.  Prints one JSON line.

    python scripts/clip_bench.py [--out FILE] [--cpu-reps N]

Seeded random weights of the ViT-B/32 shapes (the arithmetic does not depend on the values).  Times are host clocks
around work that ends in a device synchronise, medians over repetitions after a warm-up of every shape.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

VISION = dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072, image_size=224,
              patch_size=32)
TEXT = dict(hidden_size=512, num_hidden_layers=12, num_attention_heads=8, intermediate_size=2048, vocab_size=49408,
            max_position_embeddings=77, eos_token_id=49407, bos_token_id=49406, pad_token_id=1)
PROJ = 512


def layer_flop(L: int, H: int, I: int) -> float:
    """Multiply-adds x 2 of one pre-LN layer over a sequence of L tokens (QKV, scores + context, out-proj, MLP)."""
    return 2.0 * L * (3 * H * H + H * H + 2 * H * I) + 4.0 * L * L * H


def image_flop() -> float:
    G = VISION["image_size"] // VISION["patch_size"]
    L, H = G * G + 1, VISION["hidden_size"]
    return (2.0 * G * G * H * 3 * VISION["patch_size"] ** 2 + VISION["num_hidden_layers"] * layer_flop(L, H, VISION["intermediate_size"])
            + 2.0 * H * PROJ)


def text_flop(lens) -> float:
    H, I = TEXT["hidden_size"], TEXT["intermediate_size"]
    # causal attention does half the score / context work
    return float(sum(TEXT["num_hidden_layers"] * (layer_flop(L, H, I) - 2.0 * L * L * H) + 2.0 * H * PROJ for L in lens))


def timed(fn, sync, reps: int, warmup: int = 2) -> float:
    for _ in range(warmup):
        fn()
    sync()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:                                  # the numbers are still measured; say what is missing
        return dict(gpu="unknown", power_limit=f"not read ({e})")


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--cpu-reps", type=int, default=3)
    args = ap.parse_args()

    import torch
    import transformers
    from PIL import Image
    if not torch.cuda.is_available():
        raise SystemExit("clip_bench: no CUDA device (this measures the B200; there is no CPU fallback)")
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.clip import GpuClipModel, clip_configs_from_hf
    from rag_search_engine_b200.multimodal import MultimodalSearch

    res = dict(bench="clip_vit_b32", **gpu_identity(), torch=torch.__version__)
    torch.manual_seed(0)
    cfg = transformers.CLIPConfig(text_config=TEXT, vision_config=VISION, projection_dim=PROJ)
    model = transformers.CLIPModel(cfg).eval()
    vision, text = clip_configs_from_hf(model.config)
    proc = transformers.CLIPImageProcessor()                 # clip-ViT-B-32's preprocessing: 224 resize + crop
    idx = _lib.Index(0)
    gm = GpuClipModel(idx, model.state_dict(), vision, text,
                      image_processor=lambda ims: proc(ims, return_tensors="np")["pixel_values"])
    rng = np.random.default_rng(0)
    fl_img = image_flop()
    res["gflop_per_image"] = round(fl_img / 1e9, 3)

    # ---- vision tower: device pixels in, device embeddings out
    vis = {}
    for n in (1, 64, 256):
        px = torch.from_numpy(rng.standard_normal((n, 3, 224, 224)).astype(np.float32)).cuda()
        out = torch.empty((n, PROJ), dtype=torch.float32, device="cuda")
        for mode in (0, 1):
            idx.encoder_set_mode(gm.vision_slot, mode)
            t = timed(lambda: idx.encode_images_dev(gm.vision_slot, px.data_ptr(), n, out.data_ptr()), idx.synchronize,
                      reps=20 if n < 256 else 10)
            vis[f"b{n}_mode{mode}"] = dict(ms=round(t * 1e3, 3), images_per_s=round(n / t, 1),
                                           tflops_fp32_equiv=round(n * fl_img / t / 1e12, 2))
    idx.encoder_set_mode(gm.vision_slot, 0)
    res["vision"] = vis

    # ---- text tower, bulk: 2048 texts of 20-77 tokens per call (the MultimodalSearch constructor's shape)
    lens = rng.integers(20, 78, 2048)
    ids = [[49406] + rng.integers(3, 49000, int(L) - 2).tolist() + [49407] for L in lens]
    fl_txt = text_flop(lens)
    txt = dict(texts_per_call=2048, tokens=int(lens.sum()), mflop_per_token=round(fl_txt / lens.sum() / 1e6, 2))
    for mode in (0, 1):
        idx.encoder_set_mode(gm.text_slot, mode)
        t = timed(lambda: gm.encode_ids(ids), lambda: None, reps=10)
        txt[f"mode{mode}"] = dict(ms=round(t * 1e3, 2), texts_per_s=round(2048 / t, 1),
                                  tflops_fp32_equiv=round(fl_txt / t / 1e12, 2))
    idx.encoder_set_mode(gm.text_slot, 0)
    res["text_bulk"] = txt

    # ---- search_with_image end to end on a 600 k x 512 index: the document embeddings are seeded random vectors
    # (encoding 600 k texts is what text_bulk measures); the query image goes through the processor and the tower
    class DocsFrozen:
        def encode(self, items, convert_to_numpy=True, show_progress_bar=False, **kw):
            if isinstance(items[0], str):
                return np.random.default_rng(1).standard_normal((len(items), PROJ), dtype=np.float32)
            return gm.encode(items)
    n_docs = 600_000
    docs = [{"id": i, "title": f"t{i}", "description": "d"} for i in range(n_docs)]
    ms = MultimodalSearch(docs, model=DocsFrozen())
    with tempfile.TemporaryDirectory() as td:
        path = str(Path(td) / "query.png")
        Image.fromarray(np.random.default_rng(2).integers(0, 256, (224, 224, 3), dtype=np.uint8)).save(path)
        pre = timed(lambda: proc([Image.open(path).convert("RGB")], return_tensors="np"), lambda: None, reps=30)
        e2e = timed(lambda: ms.search_with_image(path, top_k=5), lambda: None, reps=30)
        vec = ms.embed_image(path)
        rank = timed(lambda: ms.search_with_vector(vec, top_k=5), lambda: None, reps=30)
    ms.close()
    res["search_with_image_600k"] = dict(end_to_end_ms=round(e2e * 1e3, 3), host_decode_preprocess_ms=round(pre * 1e3, 3),
                                         ranking_ms=round(rank * 1e3, 3),
                                         device_encode_and_rest_ms=round((e2e - pre - rank) * 1e3, 3))

    # ---- baselines: the same towers in PyTorch fp32 on this GPU (TF32 off) and on the host CPU
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.backends.cudnn.allow_tf32 = False
    tok = torch.zeros((2048, 77), dtype=torch.long)
    mask = torch.zeros_like(tok)
    for i, x in enumerate(ids):
        tok[i, :len(x)] = torch.tensor(x)
        mask[i, :len(x)] = 1
    base = {}
    with torch.no_grad():
        mg = model.cuda()
        for n in (1, 64, 256):
            px = torch.randn((n, 3, 224, 224), device="cuda")
            t = timed(lambda: mg.get_image_features(pixel_values=px), torch.cuda.synchronize, reps=10)
            base[f"gpu_fp32_vision_b{n}"] = dict(ms=round(t * 1e3, 3), images_per_s=round(n / t, 1))
        tg, mkg = tok.cuda(), mask.cuda()
        t = timed(lambda: mg.get_text_features(input_ids=tg, attention_mask=mkg), torch.cuda.synchronize, reps=5)
        base["gpu_fp32_text_2048"] = dict(ms=round(t * 1e3, 2), texts_per_s=round(2048 / t, 1))
        mc = model.cpu()
        px = torch.randn((1, 3, 224, 224))
        t = timed(lambda: mc.get_image_features(pixel_values=px), lambda: None, reps=args.cpu_reps, warmup=1)
        base["cpu_fp32_vision_b1"] = dict(ms=round(t * 1e3, 2), images_per_s=round(1 / t, 2))
        t64 = tok[:64, :40].clone()
        t64[:, 39] = 49407
        t = timed(lambda: mc.get_text_features(input_ids=t64, attention_mask=torch.ones_like(t64)), lambda: None,
                  reps=args.cpu_reps, warmup=1)
        base["cpu_fp32_text_64x40"] = dict(ms=round(t * 1e3, 2), texts_per_s=round(64 / t, 1))
    base["cpu_threads"] = torch.get_num_threads()
    res["baselines"] = base
    idx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
