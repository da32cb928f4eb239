"""Deep result lists on S-600k (the movies_600k-shaped synthetic corpus of bench.py): what a hybrid call costs at
limit 10 / 128 / 200 / 256 / 409 (knn_multiplier 10) and 512 (multiplier 8), for 256-query resident batches and
single queries, rrf and weighted; and BM25 alone at k = 256 (the general kernel) against k = 257 / 409 / 512 (the
radix-selection kernel).

    python scripts/deep_limits_bench.py [--out profiles/r06_deep_limits.json] [--steps 10]

Per configuration: ms per step (host clock around rse_hybrid_run + a stream synchronise, staged batch, median of
--steps after two warm-up runs), ms per single-query rse_hybrid call, the KNN path that served the step (rse_stats:
tc_queries > 0 = the tensor-core path K4; K' above 2048 always takes the exact scan), and the device ms of each stage
run on its own (rse_bm25, rse_knn_movies, rse_fuse_* with timing on: event pairs around the call, copies included).
The GPU name and power limit are read in the same run.  Writes only the output file.
"""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parents[1]
sys.path.insert(0, str(ROOT))

CONFIGS = [(10, 10), (128, 10), (200, 10), (256, 10), (409, 10), (512, 8)]


def gpu_card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in out[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--movies", type=int, default=600_000)
    ap.add_argument("--vocab", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--singles", type=int, default=20)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r06_deep_limits.json"))
    args = ap.parse_args()

    import torch
    from rag_search_engine_b200 import _lib, synth
    if not torch.cuda.is_available():
        raise SystemExit("deep_limits_bench needs a CUDA device")
    card = gpu_card()
    se = synth.synth_embeddings(args.movies, seed=1234, device="cuda")
    bm = synth.synth_bm25(args.movies, args.vocab, seed=1234, device="cuda")
    tp, tr = synth.synth_token_queries(bm, 256, seed=99)
    Q = synth.synth_query_vectors(se.emb, 256, seed=99).cpu().numpy()
    torch.cuda.synchronize()
    idx = _lib.Index(0)
    mo = se.movie_of_chunk.contiguous()
    idx.attach_embeddings_dev(se.emb.data_ptr(), se.emb.shape[0], se.emb.shape[1], movie_idx_ptr=mo.data_ptr(),
                              keepalive=(se, mo))
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    idx.set_id_tables(se.movie_ids, se.movie_ids)
    ids = se.movie_ids

    def med(xs):
        return round(float(np.median(xs)), 3)

    rows = []
    for limit, mult in CONFIGS:
        kprime = max(limit * mult, limit)
        for mode, param in ((0, 60.0), (1, 0.5)):
            idx.hybrid_stage(Q, tp, tr)
            for _ in range(2):
                idx.hybrid_run(mode, param, limit, knn_multiplier=mult)
            idx.synchronize()
            tc0 = idx.stats().tc_queries
            ms = []
            for _ in range(args.steps):
                t0 = time.perf_counter()
                idx.hybrid_run(mode, param, limit, knn_multiplier=mult)
                idx.synchronize()
                ms.append((time.perf_counter() - t0) * 1e3)
            tc = idx.stats().tc_queries - tc0
            idx.hybrid_fetch(limit)
            single = []
            for i in range(args.singles + 2):
                t0 = time.perf_counter()
                idx.hybrid(mode, param, limit, Q[i:i + 1], tp[i:i + 2] - tp[i], tr[tp[i]:tp[i + 1]], knn_multiplier=mult)
                single.append((time.perf_counter() - t0) * 1e3)
            # each stage on its own, same batch
            idx.set_timing(True)
            bms, kms, fms = [], [], []
            for _ in range(3):
                score, doc, cnt = idx.bm25(tp, tr, limit)
                bms.append(idx.stats().last_bm25_ms)
                dist, _rowid, movie, kc = idx.knn_movies(Q, limit, kprime)
                kms.append(idx.stats().last_knn_total_ms)
                bid = np.where(doc >= 0, ids[np.clip(doc, 0, None)], -1)
                sid = np.where(movie >= 0, ids[np.clip(movie, 0, None)], -1)
                fuse = idx.fuse_rrf if mode == 0 else idx.fuse_weighted
                fuse(limit, param, bid, score, cnt, sid, dist.astype(np.float64), kc)
                fms.append(idx.stats().last_fuse_ms)
            idx.set_timing(False)
            rows.append({"limit": limit, "knn_multiplier": mult, "kprime": kprime, "mode": "rrf" if mode == 0 else "weighted",
                         "batch256_ms_per_step": med(ms), "batch256_ms_min": round(min(ms), 3),
                         "single_query_ms": med(single[2:]),
                         "knn_path": "tensor-core (K4)" if tc > 0 else "exact scan",
                         "stage_alone_device_ms": {"bm25": med(bms), "knn_movies": med(kms), "fusion": med(fms)}})
            print(json.dumps(rows[-1]), flush=True)

    bm25_rows = []
    idx.set_timing(True)
    for k in (256, 257, 409, 512):
        idx.bm25(tp, tr, k)
        ms = []
        for _ in range(args.steps):
            idx.bm25(tp, tr, k)
            ms.append(idx.stats().last_bm25_ms)
        bm25_rows.append({"k": k, "kernel": "bm25_score_kernel (k-round arg-min)" if k <= 256 else
                          "bm25_deep_score_kernel (radix selection)", "batch256_device_ms": med(ms)})
        print(json.dumps(bm25_rows[-1]), flush=True)
    idx.close()
    out = {"card": card, "workload": f"S-600k: {se.emb.shape[0]} chunks x {se.emb.shape[1]}, {args.movies} movies, "
                                     f"{len(bm.doc_idx)} postings; 256 queries (bench.py seeds)",
           "method": __doc__.split("\n\n")[2].strip().replace("\n", " "),
           "hybrid": rows, "bm25_alone": bm25_rows}
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(out, indent=1) + "\n")
    print(json.dumps({"card": card, "written": args.out}))


if __name__ == "__main__":
    main()
