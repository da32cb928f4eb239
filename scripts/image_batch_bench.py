"""Batched image search on a 600 k x 512 corpus (§10 f4): the exact scan (tc mode 1) against the tensor-core path
(K4, automatic mode) for batches of 2..1024 image embeddings, the MultimodalSearch batch entry points end to end, and
optionally a 384-wide regression check of bench.py against another build.  Prints one JSON line.

    python scripts/image_batch_bench.py [--out FILE] [--parent-tree DIR]

Corpus: seeded unit-norm N(0, I) rows generated on the device; queries are corpus rows plus noise, passed from host
buffers (rse_knn).  Times are host clocks around calls that end in a device synchronise (rse_knn returns host
results), medians over repetitions after a warm-up of every shape.  The filter pass alone is timed with the library's
device events (rse_set_timing: an event pair around every filter launch).  --parent-tree DIR: a checkout of another
build with its librse.so built; bench.py's hybrid600k and bm25_10k run on both trees, alternating with the order
flipped every round: outputs dumped and compared bit for bit, ms per step recorded.
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

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

VISION = dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072, image_size=224,
              patch_size=32)
TEXT = dict(hidden_size=512, num_hidden_layers=12, num_attention_heads=8, intermediate_size=2048, vocab_size=49408,
            max_position_embeddings=77, eos_token_id=49407, bos_token_id=49406, pad_token_id=1)
D = 512
N_ROWS = 600_000


def gpu_identity():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clk = [s.strip() for s in q.split(",")]
        return dict(gpu=name, power_limit=power, max_sm_clock=clk)
    except Exception as e:                                  # the numbers are still measured; say what is missing
        return dict(gpu="unknown", power_limit=f"not read ({e})")


def timed(fn, min_reps: int = 5, min_s: float = 0.5, warmup: int = 2) -> float:
    for _ in range(warmup):
        fn()
    ts, t_all = [], time.perf_counter()
    while len(ts) < min_reps or time.perf_counter() - t_all < min_s:
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return float(np.median(ts))


def same(a, b):
    return all((np.asarray(x).view(np.uint8) == np.asarray(y).view(np.uint8)).all() for x, y in zip(a, b))


def ranking(idx, emb_dev, rng):
    """ms per rse_knn call, both modes, and the filter pass alone in the automatic mode."""
    import torch
    out = {}
    n_pad = (N_ROWS + 255) // 256 * 256
    for nq in (2, 16, 64, 256, 1024):
        rows = torch.from_numpy(rng.integers(0, N_ROWS, nq)).cuda()
        Q = (emb_dev[rows] + 0.05 * torch.randn((nq, D), device="cuda")).cpu().numpy()
        for k in (5, 100):
            r, res = {}, {}
            for name, mode in (("exact_scan", 1), ("k4_auto", 0)):
                idx.set_tc_mode(mode)
                res[name] = idx.knn(Q, k)
                t = timed(lambda: idx.knn(Q, k))
                r[name] = dict(ms=round(t * 1e3, 4), queries_per_s=round(nq / t, 1))
            # the filter pass alone (device events around each filter launch), automatic mode
            idx.set_tc_mode(0)
            idx.set_timing(True)
            idx.stats_reset()
            for _ in range(5):
                idx.knn(Q, k)
            st = idx.stats()
            idx.set_timing(False)
            if st.tc_queries == 5 * nq and st.scan_launches_timed > 0:
                nblk = (nq + 255) // 256
                ms = st.scan_ms_total / 5                 # every timed pair of a call: the filter launch(es)
                flop = 2.0 * n_pad * D * 256 * nblk        # the GEMM as issued: whole 256-query blocks
                r["k4_filter"] = dict(ms_per_call=round(ms, 4), tflops=round(flop / (ms * 1e-3) / 1e12, 1),
                                      tc_queries=int(st.tc_queries), second_chance=int(st.tc_second_chance_queries),
                                      fallback=int(st.tc_fallback_queries))
            else:
                r["k4_filter"] = dict(note=f"K4 did not serve every query ({st.tc_queries} of {5 * nq})")
            r["identical_outputs"] = bool(same(res["exact_scan"], res["k4_auto"]))
            r["speedup"] = round(r["exact_scan"]["ms"] / r["k4_auto"]["ms"], 2)
            out[f"nq{nq}_k{k}"] = r
    idx.set_tc_mode(0)
    return out


def bench_line(tree: Path, workload: str, dump: Path, steps: int) -> dict:
    cmd = [sys.executable, str(tree / "bench.py"), "--gpus", "1", "--steps", str(steps), "--warmup", "5",
           "--workload", workload, "--no-extras", "--no-cpu-baseline", "--no-knn1", "--no-e2e",
           "--dump-outputs", str(dump)]
    p = subprocess.run(cmd, cwd=str(tree), capture_output=True, text=True, timeout=1800)
    if p.returncode != 0:
        return dict(error=p.stderr[-2000:])
    d = json.loads(p.stdout.strip().splitlines()[-1])
    return dict(ms_per_step=d.get("ms_per_step"), value=d.get("value"))


def dumps_equal(a: Path, b: Path) -> bool:
    fa, fb = sorted(x.name for x in a.glob("*.npy")), sorted(x.name for x in b.glob("*.npy"))
    return bool(fa) and fa == fb and all(np.array_equal(np.load(a / f).view(np.uint8), np.load(b / f).view(np.uint8))
                                         for f in fa)


def regression_384(parent: Path, rounds: int = 4) -> dict:
    """bench.py on both trees, alternating, the order flipped every round; outputs of every round compared."""
    res = dict(parent_tree=parent.name, rounds=rounds)
    with tempfile.TemporaryDirectory() as td:
        td = Path(td)
        for workload, steps in (("hybrid600k", 50), ("bm25_10k", 10)):
            runs = {"new": [], "parent": []}
            for r in range(rounds):
                order = (("new", ROOT), ("parent", parent)) if r % 2 == 0 else (("parent", parent), ("new", ROOT))
                for name, tree in order:
                    runs[name].append(bench_line(tree, workload, td / f"{workload}_{name}_{r}", steps=steps))
            res[f"{workload}_runs"] = runs
            res[f"{workload}_ms_per_step_mean"] = {k: round(float(np.mean([x["ms_per_step"] for x in v])), 4)
                                                   for k, v in runs.items() if all("ms_per_step" in x for x in v)}
            res[f"{workload}_outputs_equal"] = all(dumps_equal(td / f"{workload}_new_{r}", td / f"{workload}_parent_{r}")
                                                   for r in range(rounds))
    return res


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--parent-tree", default=None)
    args = ap.parse_args()

    import torch
    if not torch.cuda.is_available():
        raise SystemExit("image_batch_bench: no CUDA device (this measures the B200; there is no CPU fallback)")
    from rag_search_engine_b200 import _lib
    res = dict(bench="image_batch_600k_x512", **gpu_identity(), rows=N_ROWS, dim=D, timing="host clock around "
               "synchronous calls, median; filter: device events")
    rng = np.random.default_rng(0)

    # ---- ranking from host buffers: exact scan vs K4 on a device-generated corpus
    g = torch.Generator(device="cuda").manual_seed(1)
    emb = torch.randn((N_ROWS, D), device="cuda", generator=g)
    emb /= emb.norm(dim=1, keepdim=True)
    idx = _lib.Index(0)
    idx.attach_embeddings_dev(emb.data_ptr(), N_ROWS, D, keepalive=emb)
    res["ranking"] = ranking(idx, emb, rng)
    idx.close()

    # ---- MultimodalSearch: search_with_vectors for 256 queries vs 256 search_with_vector calls; search_with_images
    import transformers
    from PIL import Image
    from rag_search_engine_b200.clip import GpuClipModel, clip_configs_from_hf
    from rag_search_engine_b200.multimodal import MultimodalSearch
    table = emb.cpu().numpy()
    del emb

    class Frozen:                                  # the document embeddings above (text_bulk of r03 measures encoding)
        def encode(self, items, convert_to_numpy=True, show_progress_bar=False, **kw):
            return table[:len(items)]
    docs = [{"id": i, "title": f"t{i}", "description": "d"} for i in range(N_ROWS)]
    ms = MultimodalSearch(docs, model=Frozen())
    Q = table[rng.integers(0, N_ROWS, 256)] + 0.05 * rng.standard_normal((256, D)).astype(np.float32)
    batch = ms.search_with_vectors(Q, top_k=5)
    assert batch == [ms.search_with_vector(q, top_k=5) for q in Q[:16]] + batch[16:]
    t_b = timed(lambda: ms.search_with_vectors(Q, top_k=5))
    t_1 = timed(lambda: [ms.search_with_vector(q, top_k=5) for q in Q], min_reps=3)
    res["search_with_vectors_256"] = dict(ms=round(t_b * 1e3, 3), per_row_search_with_vector_ms=round(t_1 * 1e3, 2),
                                          speedup=round(t_1 / t_b, 1))

    torch.manual_seed(0)
    cfg = transformers.CLIPConfig(text_config=TEXT, vision_config=VISION, projection_dim=D)
    model = transformers.CLIPModel(cfg).eval()
    vision, text = clip_configs_from_hf(model.config)
    proc = transformers.CLIPImageProcessor()                 # clip-ViT-B-32's preprocessing: 224 resize + crop
    eidx = _lib.Index(0)
    gm = GpuClipModel(eidx, model.state_dict(), vision, text,
                      image_processor=lambda ims: proc(ims, return_tensors="np")["pixel_values"])
    ms.model = gm                                  # query images through the device towers, ranking over the table
    with tempfile.TemporaryDirectory() as td:
        paths = []
        for i in range(256):
            p = str(Path(td) / f"q{i}.png")
            Image.fromarray(rng.integers(0, 256, (256, 320, 3), dtype=np.uint8)).save(p)
            paths.append(p)
        t_e2e = timed(lambda: ms.search_with_images(paths, top_k=5), min_reps=3)
        t_pre = timed(lambda: proc([Image.open(p).convert("RGB") for p in paths], return_tensors="np"), min_reps=3)
        px = proc([Image.open(p).convert("RGB") for p in paths], return_tensors="np")["pixel_values"]
        t_tow = timed(lambda: gm.encode_pixels(px), min_reps=3)
        embs = gm.encode_pixels(px)
        t_rank = timed(lambda: ms.search_with_vectors(embs, top_k=5))
        t_one = timed(lambda: [ms.search_with_image(p, top_k=5) for p in paths[:32]], min_reps=2) * 8
    res["search_with_images_256"] = dict(end_to_end_ms=round(t_e2e * 1e3, 2), host_decode_preprocess_ms=round(t_pre * 1e3, 2),
                                         tower_ms=round(t_tow * 1e3, 2), ranking_ms=round(t_rank * 1e3, 3),
                                         per_image_search_with_image_ms_est=round(t_one * 1e3, 1))
    ms.close()
    eidx.close()

    if args.parent_tree:
        res["regression_384"] = regression_384(Path(args.parent_tree).resolve())
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
