"""Exact movie-level KNN (rse_knn_movies_exact, DESIGN §11) against the reference-truncated rse_knn_movies on S-600k
(synth.synth_embeddings(600_000), isotropic and the clustered corpus of bench.py --corpus clustered).

    python scripts/exact_movies_bench.py [--out profiles/r10_exact_movies.json] [--steps 5] [--check 2]

Per corpus, batch size (1 / 16 / 256 queries) and k (10: the staged side of the rule, 1000: straight to the scan):
ms per call of knn_movies (K' = min(10 k, 4096)) and of knn_movies_exact (host clock around the blocking call,
median of --steps after two warm-up calls), the share of queries that took the segmented scan, and how many queries
knn_movies left short of k.  For the calls where every query took the scan, the bytes the scan path needs, computed
from the shapes (movies_exact_bytes), over the call's time: an achieved rate for the whole call (copies, selection
and launches included) against the data sheet's 7.7 TB/s; and, in separate calls with rse_set_timing on, the call's
device time split into the scan kernels (event pairs) and everything after them (segmented minimum, selection,
output copies).  The first --check queries at k = 10 and 1000 are compared
with the numpy restatement of the contract (tests/helpers/exact_movies_ref.py over oracle.all_distances), bit for
bit.  The GPU name and power limit are read in the same run.  Writes only the output file.
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
sys.path.insert(0, str(ROOT / "tests"))

HBM_TBPS = 7.7
QB = 16                                                       # queries per scan pass (knn_scan.cuh kScanMaxQB)


def gpu_card() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = [x.strip() for x in out[0].split(",")]
    return {"name": name, "power_limit": power, "max_sm_clock": clock}


def movies_exact_bytes(n_rows: int, dim: int, n_slots: int, nq: int, k: int) -> int:
    """HBM bytes of the segmented-scan path for nq queries: per group of <= 16 queries the scan reads every row
    (dim * 4 B) and its squared norm (4 B) and writes one f32 distance per (row, query); the segmented minimum reads
    those distances and movie_idx (4 B per row and query: counted as HBM although repeated reads may hit L2) and
    initialises the [query, movie] u64 keys; the six radix passes and the collect read the keys of each query."""
    total = 0
    for g0 in range(0, nq, QB):
        ng = min(QB, nq - g0)
        total += n_rows * (dim * 4 + 4) + n_rows * ng * 4           # scan
        total += n_rows * ng * (4 + 4) + n_slots * ng * 8           # segmented minimum + key initialisation
    total += nq * n_slots * 8 * 7                                   # selection passes + collect
    total += nq * k * (8 * 2 + 24)                                  # selected keys, candidates
    return total


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--movies", type=int, default=600_000)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--check", type=int, default=2)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r10_exact_movies.json"))
    args = ap.parse_args()

    import torch
    import oracle
    from helpers.exact_movies_ref import exact_movies
    from rag_search_engine_b200 import _lib, synth
    if not torch.cuda.is_available():
        raise SystemExit("exact_movies_bench needs a CUDA device")
    card = gpu_card()
    result = {"gpu": card, "movies": args.movies, "steps": args.steps, "corpora": []}

    def med(xs):
        return round(float(np.median(xs)), 3)

    for corpus in ("isotropic", "clustered"):
        kw = {} if corpus == "isotropic" else dict(distribution="clustered", n_centres=max(2, args.movies // 300),
                                                   spread=0.15)
        se = synth.synth_embeddings(args.movies, seed=1234, device="cuda", **kw)
        Q = synth.synth_query_vectors(se.emb, 256, seed=99).cpu().numpy()
        mo = se.movie_of_chunk.contiguous()
        n_rows, dim = se.emb.shape
        torch.cuda.synchronize()
        idx = _lib.Index(0)
        idx.attach_embeddings_dev(se.emb.data_ptr(), n_rows, dim, movie_idx_ptr=mo.data_ptr(), keepalive=(se, mo))
        n_slots = int(mo.max().item()) + 1
        rows = []
        for k in (10, 1000):
            kprime = min(10 * k, _lib.RSE_MAX_KPRIME)
            for nq in (1, 16, 256):
                q = Q[:nq]
                for _ in range(2):
                    idx.knn_movies(q, k, kprime)
                    idx.knn_movies_exact(q, k)
                ms_ref, ms_ex, scanned, short = [], [], [], 0
                for _ in range(args.steps):
                    t0 = time.perf_counter()
                    _, _, _, cnt = idx.knn_movies(q, k, kprime)
                    ms_ref.append((time.perf_counter() - t0) * 1e3)
                    t0 = time.perf_counter()
                    _, _, _, cnt_ex, sc = idx.knn_movies_exact(q, k)
                    ms_ex.append((time.perf_counter() - t0) * 1e3)
                    scanned.append(sc)
                    short = int((cnt < k).sum())
                    assert (cnt_ex == k).all()
                row = {"k": k, "nq": nq, "knn_movies_kprime": kprime, "knn_movies_ms": med(ms_ref),
                       "knn_movies_short_queries": short, "knn_movies_exact_ms": med(ms_ex),
                       "scan_share": round(float(np.mean(scanned)) / nq, 4)}
                if min(scanned) == nq:
                    b = movies_exact_bytes(n_rows, dim, n_slots, nq, k)
                    gbs = b / (med(ms_ex) * 1e-3) / 1e9
                    row.update({"scan_bytes_model": b, "scan_call_GBps": round(gbs, 1),
                                "scan_call_share_of_7p7TBps": round(gbs / (HBM_TBPS * 1e3), 4)})
                    # device split with rse_set_timing (separate calls: the event pairs are not in the timed ones):
                    # the scan kernels' event pairs, and the rest of the call (segmented minimum, selection, copies)
                    tot, scan = [], []
                    idx.set_timing(True)
                    for _ in range(args.steps):
                        idx.stats_reset()
                        idx.knn_movies_exact(q, k)
                        st = idx.stats()
                        tot.append(st.last_knn_total_ms)
                        scan.append(st.scan_ms_total)
                    idx.set_timing(False)
                    row.update({"device_call_ms": med(tot), "scan_kernels_ms": med(scan),
                                "after_scan_ms": med(np.subtract(tot, scan))})
                rows.append(row)
                print(corpus, json.dumps(row), flush=True)
        # bit-for-bit against the numpy restatement on a sample
        checked = []
        if args.check > 0:
            emb = se.emb.cpu().numpy()
            movie_of = mo.cpu().numpy()
            ref_d = [oracle.all_distances(emb, Q[qi]) for qi in range(args.check)]
            for k in (10, 1000):
                dist, rowid, movie, cnt, _ = idx.knn_movies_exact(Q[:args.check], k)
                for qi in range(args.check):
                    od, orow, omov = exact_movies(emb, Q[qi], movie_of, k, dist=ref_d[qi])
                    c = int(cnt[qi])
                    ok = (c == len(orow) and rowid[qi, :c].tolist() == orow.tolist()
                          and movie[qi, :c].tolist() == omov.tolist()
                          and dist[qi, :c].view(np.uint32).tolist() == od.view(np.uint32).tolist())
                    checked.append({"k": k, "query": qi, "bit_identical": bool(ok)})
            del emb
        result["corpora"].append({"corpus": corpus, "n_rows": int(n_rows), "dim": int(dim), "n_movie_slots": n_slots,
                                  "rows": rows, "oracle_check": checked})
        idx.close()
        del se, mo
        torch.cuda.empty_cache()
    Path(args.out).parent.mkdir(parents=True, exist_ok=True)
    Path(args.out).write_text(json.dumps(result, indent=1) + "\n")
    print(json.dumps({"out": args.out, "gpu": card}))


if __name__ == "__main__":
    main()
