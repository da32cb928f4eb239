"""CLIP image preprocessing on the device against the host processor (§10 f6): ``search_with_images`` on 256 images over
600 k x 512 text embeddings, the host-processor route and the device route alternated in one session, at 256 x 320
PNG and 2000 x 1500 JPEG; the host decode that remains, with and without the thread pool; the device preprocessing
alone per 256 images with its H2D bytes and the share of the copy.  Prints one JSON line.

    python scripts/image_preprocess_bench.py [--out FILE] [--rounds N]

Model: clip-ViT-B/32's shapes with seeded random weights (nothing is downloaded), the default CLIPImageProcessor
(torchvision backend, the default of transformers 5) and CLIPImageProcessorPil.  Times are host clocks around calls
that end in a device synchronise, medians over rounds; the two routes run in alternating order each round.  Both
routes' results are compared: they must be identical.  Images are seeded noise over smooth gradients, written to a
temporary directory.
"""
from __future__ import annotations

import argparse
import json
import sys
import tempfile
import time
from concurrent.futures import ThreadPoolExecutor
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "scripts"))

from image_batch_bench import D, N_ROWS, TEXT, VISION, gpu_identity  # noqa: E402


def _image(rng, h, w):
    y, x = np.mgrid[0:h, 0:w]
    a = np.stack([x * 255 // (w - 1), y * 255 // (h - 1), (x + y) % 256], -1)
    return np.clip(a + rng.integers(-30, 31, (h, w, 3)), 0, 255).astype(np.uint8)


def _med(ts):
    return round(float(np.median(ts)) * 1e3, 2)


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("image_preprocess_bench: no CUDA device (this measures the B200; there is no CPU fallback)")
    import transformers
    from PIL import Image
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.clip import DeviceImageProcessor, GpuClipModel, clip_configs_from_hf
    from rag_search_engine_b200.multimodal import MultimodalSearch

    res = dict(bench="image_preprocess_256", **gpu_identity(), rows=N_ROWS, dim=D, rounds=args.rounds,
               cpu_threads=__import__("os").cpu_count(), aten_cpu_capability=torch.backends.cpu.get_cpu_capability(),
               timing="host clock around calls ending in a device synchronise, median over rounds, routes alternated")
    rng = np.random.default_rng(0)
    g = torch.Generator(device="cuda").manual_seed(1)
    emb = torch.randn((N_ROWS, D), device="cuda", generator=g)
    emb /= emb.norm(dim=1, keepdim=True)
    table = emb.cpu().numpy()
    del emb

    class Frozen:                                    # the document embeddings; query images go through the model
        def __init__(self):
            self.gm = None

        def encode(self, items, convert_to_numpy=True, show_progress_bar=False, **kw):
            return table[:len(items)] if self.gm is None else self.gm.encode(items)

    docs = [{"id": i, "title": f"t{i}", "description": "d"} for i in range(N_ROWS)]
    fz = Frozen()
    ms = MultimodalSearch(docs, model=fz)
    torch.manual_seed(0)
    model = transformers.CLIPModel(transformers.CLIPConfig(text_config=TEXT, vision_config=VISION, projection_dim=D)).eval()
    vision, text = clip_configs_from_hf(model.config)
    eidx = _lib.Index(0)
    procs = {"torchvision": transformers.CLIPImageProcessor(), "pil": transformers.CLIPImageProcessorPil()}
    gm = GpuClipModel(eidx, model.state_dict(), vision, text)
    fz.gm = gm

    with tempfile.TemporaryDirectory() as td:
        for label, (h, w), ext in (("png_256x320", (256, 320), "png"), ("jpeg_2000x1500", (1500, 2000), "jpg")):
            paths = []
            for i in range(256):
                p = str(Path(td) / f"{label}_{i}.{ext}")
                Image.fromarray(_image(rng, h, w)).save(p, quality=90) if ext == "jpg" else \
                    Image.fromarray(_image(rng, h, w)).save(p)
                paths.append(p)
            load = lambda p: Image.open(p).convert("RGB")  # noqa: E731
            r = dict(file_bytes=int(sum(Path(p).stat().st_size for p in paths)))
            # host decode alone: one thread and the thread pool search_with_images uses
            t1, tp = [], []
            for _ in range(max(2, args.rounds // 2)):
                t0 = time.perf_counter(); [load(p) for p in paths]; t1.append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                with ThreadPoolExecutor(max_workers=min(256, __import__("os").cpu_count() or 1, 16)) as pool:
                    list(pool.map(load, paths))
                tp.append(time.perf_counter() - t0)
            r["decode_ms_per_image_1_thread"] = round(_med(t1) / 256, 3)
            r["decode_ms_per_image_pool"] = round(_med(tp) / 256, 3)
            images = [load(p) for p in paths]
            arrays = [np.asarray(im) for im in images]
            for name, proc in procs.items():
                gm.image_processor = lambda ims, proc=proc: proc(ims, return_tensors="np")["pixel_values"]
                dp = DeviceImageProcessor.maybe(eidx, proc, gm.vision_slot, vision["image_size"])
                ts = {"host": [], "device": []}
                out = {}
                for k in range(args.rounds + 1):                     # round 0 warms up both routes
                    for route in (("host", "device") if k % 2 else ("device", "host")):
                        gm.device_image_processor = dp if route == "device" else None
                        t0 = time.perf_counter()
                        out[route] = ms.search_with_images(paths, top_k=5)
                        if k:
                            ts[route].append(time.perf_counter() - t0)
                rr = dict(host_route_ms=_med(ts["host"]), device_route_ms=_med(ts["device"]),
                          identical_results=out["host"] == out["device"])
                rr["speedup"] = round(rr["host_route_ms"] / rr["device_route_ms"], 2)
                # the stages of each route
                th = []
                for _ in range(max(2, args.rounds // 2)):
                    t0 = time.perf_counter(); proc(images, return_tensors="np"); th.append(time.perf_counter() - t0)
                rr["host_processor_ms"] = _med(th)
                eidx.stats_reset()
                eidx.image_preprocess(gm.vision_slot, arrays)
                st = eidx.stats()
                rr["device_h2d_bytes"] = int(st.h2d_bytes)
                td_, tc_, tk_ = [], [], []
                out_dev = torch.empty((256, 3, 224, 224), dtype=torch.float32, device="cuda")
                packed, offs, hw = eidx._pack_images(arrays)
                stage = torch.from_numpy(packed).pin_memory()
                dst = torch.empty(packed.size, dtype=torch.uint8, device="cuda")
                for _ in range(args.rounds):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    eidx._check(eidx._L.rse_image_preprocess_dev(eidx._h, gm.vision_slot, packed.ctypes.data,
                                                                 offs.ctypes.data, hw.ctypes.data, 256,
                                                                 out_dev.data_ptr()))
                    eidx.synchronize()
                    td_.append(time.perf_counter() - t0)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter(); dst.copy_(stage, non_blocking=True); torch.cuda.synchronize()
                    tc_.append(time.perf_counter() - t0)
                    t0 = time.perf_counter(); gm.encode_pixels(np.zeros((256, 3, 224, 224), np.float32)); tk_.append(time.perf_counter() - t0)
                rr["device_preprocess_ms"] = _med(td_)
                rr["pinned_copy_of_the_pixels_ms"] = _med(tc_)
                rr["copy_share_of_device_preprocess"] = round(float(np.median(tc_) / np.median(td_)), 3)
                rr["tower_from_host_pixel_values_ms"] = _med(tk_)
                r[name] = rr
            res[label] = r
    ms.close()
    eidx.close()
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
