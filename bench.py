#!/usr/bin/env python
"""bench.py — hybrid queries/sec (RRF, top-10) on the movies_600k-shaped synthetic corpus.

    python bench.py --gpus N --steps K --warmup W            # this repo (librse on the B200)
    python bench.py --impl reference --gpus N --steps K ...   # the reference's CPU path (oracle port)

A "step" = one batch of hybrid queries through the whole hot path
(BM25 top-10 + exact vec0 KNN top-100 + best-chunk-per-movie + RRF fusion).
  value : whole-job queries/s with the query batches already resident in HBM (8 distinct batches staged once
          and parked with rse_hybrid_stash, then K x rse_hybrid_run rotating over them), CUDA events, max over ranks.
  e2e   : the same metric through the host-buffer C-ABI calls: every step uploads its query
          vectors/tokens (host -> pinned -> device) and reads its results back inside the timed
          region.  Headline = the serving loop (rse_hybrid_submit / rse_hybrid_collect, two batches
          in flight); e2e.blocking_call = rse_hybrid one batch at a time.
N > 1   : weak scaling by default — the corpus replicated, the query batch split by rank, no
          data-path collective (--parallelism rowshard: corpus row-sharded, one all_gather of the
          local top-K' candidates per step, BM25/fusion split by query slice).
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

import numpy as np  # noqa: E402

ROW_BYTES = 384 * 4 + 4          # algorithmic bytes per chunk row per pass: 1536 B vector + 4 B |a|^2 (SURVEY §8d)
ROW_BYTES_SHADOW = 384 * 2       # the fp16-shadow filter pass (knn_tc3) streams 768 B per row and nothing else


def tc_kind(args):
    """The K4 kernel (r01's two TF32 mappings were removed in r02: 2.6-3.5x slower on every measured shape)."""
    return "f16-shadow"


def scan_kernel_desc(args, tc_used, qb):
    if not tc_used:
        return (f"knn_scan384_kernel<QB={qb}> (one pass over the shard serves {qb} queries; FFMA2-pipe-bound above QB=4, "
                f"HBM-bound at QB=1: see knn_batch1)"), ROW_BYTES
    return ("knn_tc3_kernel<filter> (tcgen05 kind::f16 256x256x16 cta_group::2 over the fp16 normalised shadow, "
            "queries resident in shared memory, TMA 4-stage ring; one pass serves 256 queries; survivors re-scored "
            "exactly in fp32; in the hybrid step one bm25_fx_kernel CTA per SM runs underneath it on a second "
            "stream, which costs the pass ~8 %)"), ROW_BYTES_SHADOW


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--movies", type=int, default=600_000)
    ap.add_argument("--vocab", type=int, default=1_000_000)
    ap.add_argument("--batch", type=int, default=256, help="hybrid queries per step")
    ap.add_argument("--limit", type=int, default=10)
    ap.add_argument("--mode", default="rrf", choices=["rrf", "weighted"])
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the cpu_baseline sample (0 = 2 x cores)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-knn1", action="store_true", help="skip the batch-1 KNN micro-measurement")
    ap.add_argument("--workload", default="hybrid600k", choices=["hybrid600k", "bm25_10k", "knn100m"],
                    help="hybrid600k = configs[3] (the metric's configuration, default); bm25_10k = configs[1]; "
                         "knn100m = configs[4] alone (fixed 100M-row corpus row-sharded over the GPUs, top-100)")
    ap.add_argument("--shard-rows", type=int, default=0,
                    help="--workload knn100m only: rows per GPU of a SMALLER corpus for experiments (0 = configs[4] as specified)")
    ap.add_argument("--corpus", default="isotropic", choices=["isotropic", "clustered", "clustered_dense"],
                    help="embedding distribution of the main line (the default line also carries short measurements on "
                         "the two clustered corpora)")
    ap.add_argument("--no-extras", action="store_true",
                    help="main line only: skip the weighted / clustered / python-API / small-batch / rowshard / knn100m objects")
    ap.add_argument("--no-knn100m", action="store_true", help="skip the configs[4] object of the default line")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="N > 1: weak = --batch queries per GPU per step (global batch = batch x N; every rank scans its "
                         "row shard for all of them, so per-GPU work is constant); strong = the same --batch split over N")
    ap.add_argument("--parallelism", default="auto", choices=["auto", "replicate", "rowshard"],
                    help="N > 1: replicate = every GPU holds the corpus and serves its own slice of the query batch (hybrid "
                         "queries are independent units: no data-path collective); rowshard = the corpus is cut by row, "
                         "local top-K' + one all_gather + merge (what a corpus that does not fit one GPU needs: "
                         "--workload knn100m always uses it).  auto = replicate when corpus + shadow fit in 1/3 of HBM; "
                         "the JSON line then carries a shorter rowshard measurement of the same batch as well")
    ap.add_argument("--bm25-mode", type=int, default=-1, help="rse_set_bm25_mode override (see include/rse.h); -1 = library default")
    ap.add_argument("--tc-mode", type=int, default=-1, help="rse_set_tc_mode override (see include/rse.h); -1 = library default")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the timed path returned in its LAST step as DIR/<name>.npy "
                         "(float64; float32 where the path returns float32; integers are exact): hybrid600k = "
                         "id, score, bm25, semantic (rrf: ranks, -1 = none; weighted: normalised scores), count; "
                         "bm25_10k = score, doc, count; knn100m = dist, row, movie, count.  The inputs are seeded, so "
                         "two builds run with the same arguments can be compared output for output.  One process only")
    return ap.parse_args()


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region.  The timed region of the default run is tens
    of milliseconds, far below nvidia-smi's loop granularity, so NVML is polled from a thread every ~1 ms
    (nvidia-smi -lms is the fallback when the NVML binding is missing)."""
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.thread = None
        self.stop_flag = False
        self.sm, self.reasons = [], set()
        self.sm_max = None
        self.path = Path(os.environ.get("TMPDIR", "/tmp")) / f"rse_clocks_{os.getpid()}.csv"

    def _poll(self, nv, handle):
        names = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                 "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                 "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                 "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or \
            getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        def once():
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(handle, nv.NVML_CLOCK_SM)))
                mask = int(get_reasons(handle))
                for k, bit in names.items():
                    if mask & bit:
                        self.reasons.add(k)
            except Exception:
                pass
        period = float(os.environ.get("RSE_CLOCK_POLL_MS", "1")) * 1e-3
        while not self.stop_flag:
            once()
            time.sleep(period)

    def start(self):
        try:
            import pynvml as nv
            import threading
            nv.nvmlInit()
            # CUDA_VISIBLE_DEVICES may renumber devices: address the GPU by the PCI bus id torch reports
            handle = None
            try:
                import torch
                bus = torch.cuda.get_device_properties(self.gpu).pci_bus_id
                dom = torch.cuda.get_device_properties(self.gpu).pci_domain_id
                dev = torch.cuda.get_device_properties(self.gpu).pci_device_id
                handle = nv.nvmlDeviceGetHandleByPciBusId(f"{dom:08x}:{bus:02x}:{dev:02x}.0".encode())
            except Exception:
                handle = nv.nvmlDeviceGetHandleByIndex(self.gpu)
            self.sm_max = float(nv.nvmlDeviceGetMaxClockInfo(handle, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._poll, args=(nv, handle), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.fh = open(self.path, "w")
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.FIELDS}",
                                          "--format=csv,noheader,nounits", "-lms", "20"], stdout=self.fh,
                                         stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            if self.sm:
                out.update(sm_mhz=statistics.median(self.sm), sm_max_mhz=self.sm_max, reasons=sorted(self.reasons),
                           samples=len(self.sm), source="nvml polling thread (one query takes ~25 ms)")
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        self.fh.close()
        sm, mx, reasons = [], [], set()
        for line in self.path.read_text().splitlines():
            p = [x.strip() for x in line.split(",")]
            if len(p) < 8:
                continue
            try:
                sm.append(float(p[0])); mx.append(float(p[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), p[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if sm:
            out.update(sm_mhz=statistics.median(sm), sm_max_mhz=max(mx), reasons=sorted(reasons), samples=len(sm),
                       source="nvidia-smi -lms 20")
        try:
            self.path.unlink()
        except Exception:
            pass
        return out


# ----------------------------------------------------------------------------- workload
NB = 8          # distinct query batches rotated through every timed loop (data-dependent variance stays visible)


def sqlite_vec_status() -> str:
    try:
        import sqlite_vec  # noqa: F401
        return "present"
    except Exception:
        return "absent"


def build_corpus(args, device: str, corpus: str = "isotropic"):
    from rag_search_engine_b200 import synth
    if corpus == "isotropic":
        return synth.synth_embeddings(args.movies, seed=1234, device=device)
    if corpus == "clustered":      # 2000 "genres", ~2400 chunks each, ~4e2 rows within +-2 eps of the 100-th neighbour
        return synth.synth_embeddings(args.movies, seed=1234, device=device, distribution="clustered",
                                      n_centres=max(2, args.movies // 300), spread=0.15)
    if corpus == "clustered_dense":  # near-duplicate neighbourhoods: ~1e3 rows within +-2 eps of the 100-th neighbour
        return synth.synth_embeddings(args.movies, seed=1234, device=device, distribution="clustered",
                                      n_centres=max(2, args.movies // 300), spread=0.06)
    raise ValueError(corpus)


def build_workload(args, device: str, corpus: str = "isotropic", bm=None):
    """Seeded S-600k corpus + NB query batches (identical on every rank and in both arms)."""
    import torch
    from rag_search_engine_b200 import synth
    t0 = time.time()
    se = build_corpus(args, device, corpus)
    if bm is None:
        bm = synth.synth_bm25(args.movies, args.vocab, seed=1234, device=device)
    tok_indptr, terms = synth.synth_token_queries(bm, NB * args.batch, seed=99)
    Q = synth.synth_query_vectors(se.emb, NB * args.batch, seed=99)
    if device != "cpu":
        torch.cuda.synchronize()
    info = {"chunks": int(se.emb.shape[0]), "dim": int(se.emb.shape[1]), "movies": args.movies,
            "postings": int(len(bm.doc_idx)), "terms": int(len(bm.df)), "build_s": round(time.time() - t0, 1),
            "corpus": corpus}
    return se, bm, tok_indptr, terms, Q, info


def batch_slice(tok_indptr, terms, Qn, lo, hi):
    """Queries lo..hi of the flattened workload as (Q, tok_indptr, term_rows) with a zero-based indptr."""
    tp = (tok_indptr[lo:hi + 1] - tok_indptr[lo]).astype(np.int32)
    tr = np.ascontiguousarray(terms[tok_indptr[lo]:tok_indptr[hi]])
    return Qn[lo:hi], tp, tr


def postings_touched(bm, terms) -> int:
    t = terms[terms >= 0]
    return int(bm.df[t].sum())


DUMP_MAX_BYTES = 64 << 20


def dump_outputs(out_dir, arrays: dict):
    """--dump-outputs: every array (query-major, one row per query) as out_dir/<name>.npy in float32 (what already
    is float32) or float64.  Above DUMP_MAX_BYTES a fixed seeded sample of the queries is written, their indices
    as query_index.npy."""
    conv = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        if a.dtype.kind in "iu" and a.size and int(np.abs(a.astype(np.int64)).max()) >= 2 ** 53:
            raise ValueError(f"--dump-outputs: {name} holds integers that float64 cannot represent exactly")
        conv[name] = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
    nq = next(iter(conv.values())).shape[0]
    total = sum(a.nbytes for a in conv.values())
    if total > DUMP_MAX_BYTES:
        keep = int(DUMP_MAX_BYTES // (total / nq + 8))
        rows = np.sort(np.random.default_rng(0).choice(nq, keep, replace=False))
        conv = {name: a[rows] for name, a in conv.items()}
        conv["query_index"] = rows.astype(np.float64)
    out = Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    for name, a in conv.items():
        np.save(out / f"{name}.npy", a)


def config_dict(args, info, world, par="replicate"):
    return {"workload": "configs[3]: movies_600k-shaped synthetic (S-600k), hybrid rrf_search k=60 limit=10 "
                        "(BM25 top-10 + exact vec0 KNN top-100 + per-movie best chunk + RRF), Gemini disabled",
            "mode": args.mode, "limit": args.limit, "knn_kprime": max(args.limit * 10, args.limit),
            "queries_per_step": args.batch, "queries_per_gpu_per_step": args.batch // max(1, world) if getattr(args, "scaling", "weak") == "weak" else None,
            "distinct_query_batches": NB, "corpus": info.get("corpus", "isotropic"),
            "movies": info["movies"], "chunks": info["chunks"], "dim": info["dim"],
            "bm25_postings": info["postings"], "bm25_terms": info["terms"],
            "l2": "inputs larger than L2: every step streams the 3.7 GB fp16 shadow of the corpus (one pass per 256 "
                  "queries) and ~1.3 GB of postings against a 126 MB L2; no flush",
            "sqlite_vec": sqlite_vec_status(),
            "parallelism": ("1 GPU" if world == 1 else
                            (f"row-shard x{world} + candidate exchange (top-K') + query-slice BM25/fusion" if par == "rowshard" else
                             f"corpus replicated x{world}, query batch split by rank, no data-path collective"))}


# ----------------------------------------------------------------------------- CPU baseline (oracle port)
def cpu_hybrid_sample(se_emb_host, movie_of, bm, ids, Q, tok_indptr, terms, limit, mode, sample, threads):
    """The reference's CPU path restated (oracle/): literal vec0 scan + aggregation, BM25, fusion."""
    import oracle
    from oracle import pyref
    oracle.set_threads(threads)
    nq = sample
    tp = tok_indptr[: nq + 1].astype(np.int32)
    tr = terms[: tp[-1]]
    t0 = time.perf_counter()
    kd, krow, kc = oracle.knn_movies_batch(se_emb_host, Q[:nq], movie_of, limit, max(limit * 10, limit), literal=True)
    osc, odc, ocnt = oracle.bm25_batch(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl, tp, tr, limit)
    out = []
    for qi in range(nq):
        bmh = [(int(ids[odc[qi, j]]), float(osc[qi, j])) for j in range(ocnt[qi])]
        semh = [(int(ids[movie_of[krow[qi, j]]]), float(kd[qi, j])) for j in range(kc[qi])]
        out.append(pyref.rrf_fuse(bmh, semh, 60, limit) if mode == "rrf" else pyref.weighted_fuse(bmh, semh, 0.5, limit))
    dt = time.perf_counter() - t0
    return nq / dt, dt, out


def run_reference(args, rank, world):
    """--impl reference: the reference's CPU implementation of the path on the box's host cores.
    The reference is Python + un-vendored sqlite-vec and cannot travel to the GPU box, so this
    times the oracle port (oracle/oracle.c: literal vec0 scan; BM25 over CSR; fusion in Python)."""
    if rank != 0:
        return
    import torch
    dev = "cuda" if torch.cuda.is_available() else "cpu"   # data generation only
    se, bm, tok_indptr, terms, Q, info = build_workload(args, dev)
    emb_host = se.emb.cpu().numpy()
    movie_of = se.movie_of_chunk.cpu().numpy().astype(np.int64)
    Qh = Q.cpu().numpy()
    del se.emb
    cores = os.cpu_count() or 1
    sample = min(args.batch, args.cpu_sample or cores)
    import oracle
    oracle.build()
    times = []
    nq_all = NB * args.batch
    for step in range(args.warmup + args.steps):
        off = (step * sample) % max(1, nq_all - sample + 1)
        Qs, tp, tr = batch_slice(tok_indptr, terms, Qh, off, off + sample)
        qps, dt, _ = cpu_hybrid_sample(emb_host, movie_of, bm, se.movie_ids, Qs, tp, tr, args.limit, args.mode, sample, cores)
        if step >= args.warmup:
            times.append(dt)
    total = sum(times)
    value = sample * len(times) / total
    line = {"impl": "reference", "metric": "hybrid queries/sec", "value": value, "unit": "queries/s",
            "n_gpus": args.gpus, "steps": len(times), "steps_requested": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * total / len(times),
            "higher_is_better": True, "scaling": "replicas only (CPU path, rank 0)", "vs_baseline": None,
            "dtype": "f32 sequential scan + f64 tail/BM25/fusion (the reference's arithmetic)",
            "data": "synthetic", "config": config_dict(args, info, 1),
            "cpu_baseline": {"value": value, "unit": "queries/s", "cores": cores, "kind": "port",
                             "sample": f"{sample} hybrid queries per step over the full S-600k corpus "
                                       f"(OpenMP over queries, each query a single-threaded literal vec0 scan)"},
            "e2e": {"value": value, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- one handle, one mode: resident + e2e
class Timer:
    def __init__(self, stream, world, device):
        import torch
        self.torch, self.stream, self.world, self.device = torch, stream, world, device
        self.e0, self.e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def barrier(self):
        if self.world > 1:
            import torch.distributed as dist
            dist.barrier()

    def gather_ranks(self, x: float):
        """x of every rank (diagnostics: which rank the max-over-ranks time belongs to)."""
        if self.world > 1:
            import torch.distributed as dist
            t = self.torch.zeros(self.world, dtype=self.torch.float64, device=self.device)
            dist.all_gather_into_tensor(t, self.torch.tensor([x], dtype=self.torch.float64, device=self.device))
            return [float(v) for v in t.cpu().tolist()]
        return [x]

    def max_over_ranks(self, x: float) -> float:
        if self.world > 1:
            import torch.distributed as dist
            t = self.torch.tensor([x], dtype=self.torch.float64, device=self.device)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return x


def measure_hybrid(idx, tm: Timer, batches, mode, param, limit, steps, warmup, *, sample_clocks=None, e2e=True):
    """batches = NB x (Q pinned numpy [nq, dim], tok_indptr, term_rows) of THIS rank.  Returns the device-timed
    resident number, the host-buffer numbers (serving loop + blocking call) and the last results per batch."""
    torch = tm.torch
    nb = len(batches)
    nq = batches[0][0].shape[0]
    # resident: every batch staged once and parked in HBM; a step exchanges the staged batch with its stash slot
    for b, (Qb, tp, tr) in enumerate(batches):
        idx.hybrid_stage(Qb, tp, tr)
        idx.hybrid_stash(b)

    def step(i, park=True):
        idx.hybrid_stash(i % nb)
        idx.hybrid_run(mode, param, limit)
        if park:
            idx.hybrid_stash(i % nb)

    for i in range(max(warmup, 3)):
        step(i)
    torch.cuda.synchronize(); tm.barrier()
    idx.set_timing(True)
    idx.stats_reset()
    sampler = None
    if sample_clocks is not None:
        sampler = ClockSampler(sample_clocks)
        sampler.start()
    torch.cuda.synchronize(); tm.barrier()
    tm.e0.record(tm.stream)
    for i in range(steps):
        step(i, park=i + 1 < steps)           # the last batch stays staged: its results are fetched below
    tm.e1.record(tm.stream)                   # (no inline NVML sampling in the loop: one query costs the host ~25 ms and
    torch.cuda.synchronize(); tm.barrier()    #  the device would idle; the sampler thread polls concurrently instead)
    clocks = sampler.stop() if sampler else None
    ms_local = tm.e0.elapsed_time(tm.e1)
    st = idx.stats()
    idx.set_timing(False)
    last = None
    if steps > 0:
        last = idx.hybrid_fetch(limit)        # what the last timed step computed
        idx.hybrid_stash((steps - 1) % nb)
    out = {"ms": tm.max_over_ranks(ms_local), "ms_local": ms_local, "stats": st, "clocks": clocks, "nq": nq,
           "survivors": None, "e2e": None, "results": None, "ms_ranks": tm.gather_ranks(ms_local), "last": last}
    if int(st.tc_filter_launches) > 0:
        try:
            out["survivors"] = idx.tc_last_survivors(min(nq, 256))
        except Exception:
            pass
    if not e2e:
        return out
    # (1) the blocking call, one batch at a time: the device idles while the host stages and collects
    res = [None] * nb
    for i in range(2):
        idx.hybrid(mode, param, limit, *batches[i % nb])
    torch.cuda.synchronize(); tm.barrier()
    t0 = time.perf_counter()
    tm.e0.record(tm.stream)
    for i in range(steps):
        res[i % nb] = idx.hybrid(mode, param, limit, *batches[i % nb])
    tm.e1.record(tm.stream)
    torch.cuda.synchronize()
    wall_blocking = tm.max_over_ranks(time.perf_counter() - t0)
    dev_blocking = tm.e0.elapsed_time(tm.e1) / steps
    for i in range(steps, nb):                                   # results of every batch for the comparisons below
        res[i] = idx.hybrid(mode, param, limit, *batches[i])
    # (2) the serving loop: rse_hybrid_submit / rse_hybrid_collect, two batches in flight — every step still
    # uploads its own inputs from host buffers and reads its own results back inside the timed region
    for _ in range(2):                                           # warm both ticket slots (their buffers are allocated lazily)
        t_prev = idx.hybrid_submit(mode, param, limit, *batches[0])
        t_next = idx.hybrid_submit(mode, param, limit, *batches[1 % nb])
        idx.hybrid_collect(t_prev); idx.hybrid_collect(t_next)
    torch.cuda.synchronize(); tm.barrier()
    res_p = [None] * nb
    t0 = time.perf_counter()
    t_prev = idx.hybrid_submit(mode, param, limit, *batches[0])
    for i in range(1, steps):
        t_next = idx.hybrid_submit(mode, param, limit, *batches[i % nb])
        res_p[(i - 1) % nb] = idx.hybrid_collect(t_prev)
        t_prev = t_next
    res_p[(steps - 1) % nb] = idx.hybrid_collect(t_prev)
    torch.cuda.synchronize()
    wall = tm.max_over_ranks(time.perf_counter() - t0)
    same = all(all((a.view(np.uint8) == b.view(np.uint8)).all() for a, b in zip(res[i], res_p[i]))
               for i in range(nb) if res_p[i] is not None)
    ntok = int(np.mean([len(b[2]) for b in batches]))
    h2d = batches[0][0].nbytes + (nq + 1) * 4 + ntok * (4 + 8)
    d2h = nq * limit * (8 + 8 + 8 + 8) + nq * 4
    out["e2e"] = {"wall": wall, "wall_blocking": wall_blocking, "dev_blocking": dev_blocking, "same": bool(same),
                  "h2d": int(h2d), "d2h": int(d2h)}
    out["results"] = res
    return out


def e2e_dict(m, nq_global, steps, world):
    e = m["e2e"]
    return {"value": nq_global * steps / e["wall"], "unit": "queries/s", "h2d_bytes_per_step": e["h2d"] * world,
            "d2h_bytes_per_step": e["d2h"] * world, "wall_ms_per_step": 1e3 * e["wall"] / steps,
            "api": "rse_hybrid_submit / rse_hybrid_collect, host buffers, two batches in flight, "
                   f"{NB} distinct batches in rotation",
            "same_results_as_blocking_call": e["same"],
            "blocking_call": {"value": nq_global * steps / e["wall_blocking"], "unit": "queries/s",
                              "api": "rse_hybrid (one batch at a time)", "device_ms_per_step": e["dev_blocking"],
                              "wall_ms_per_step": 1e3 * e["wall_blocking"] / steps}}


def survivor_stats(surv):
    if surv is None or len(surv) == 0:
        return None
    s = np.sort(np.asarray(surv, np.int64))
    pick = lambda p: int(s[min(len(s) - 1, int(p * len(s)))])          # noqa: E731
    return {"p50": pick(0.5), "p90": pick(0.9), "p99": pick(0.99), "max": int(s[-1]), "cap": 8192,
            "note": "rows per query that passed the tcgen05 filter of the LAST timed batch (exact re-score decides)"}


def make_handle(args, local_rank, stream, se, bm, lo, hi, dim):
    from rag_search_engine_b200 import _lib
    idx = _lib.Index(local_rank)
    if args.tc_mode >= 0:
        idx.set_tc_mode(args.tc_mode)
    if args.bm25_mode >= 0:
        idx.set_bm25_mode(args.bm25_mode)
    idx.set_stream(stream.cuda_stream)
    shard = se.emb[lo:hi]
    mo = se.movie_of_chunk[lo:hi].contiguous()
    idx.attach_embeddings_dev(shard.data_ptr(), hi - lo, dim, movie_idx_ptr=mo.data_ptr(), pos_base=lo,
                              keepalive=(se, shard, mo))
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    idx.set_id_tables(se.movie_ids, se.movie_ids)
    return idx


def pinned_batches(torch, Q, tok_indptr, terms, batch, qlo_of, qhi_of):
    """NB batches; from global batch b this rank takes queries [qlo_of, qhi_of) (the whole batch when N = 1)."""
    Qh = torch.empty(tuple(Q.shape), dtype=torch.float32, pin_memory=True)
    Qh.copy_(Q.cpu())
    Qn = Qh.numpy()
    out = []
    for b in range(NB):
        out.append(batch_slice(tok_indptr, terms, Qn, b * batch + qlo_of, b * batch + qhi_of))
    return Qn, out


def measure_corpus_variant(args, local_rank, device, stream, bm, corpus, steps, tm):
    """The same hybrid step on a CLUSTERED corpus (VERDICT r01 weak #3): fallback rate, survivor counts, q/s, and
    the tensor-core path's results against the exact scan on a sample."""
    import torch
    se, _, tok_indptr, terms, Q, info = build_workload(args, f"cuda:{local_rank}", corpus=corpus, bm=bm)
    idx = make_handle(args, local_rank, stream, se, bm, 0, info["chunks"], info["dim"])
    Qn, batches = pinned_batches(torch, Q, tok_indptr, terms, args.batch, 0, args.batch)
    m = measure_hybrid(idx, tm, batches, 0, 60.0, args.limit, steps, 3, e2e=False)
    st = m["stats"]
    # parity of the filter path on this distribution: K4 (auto) vs the exact scan (tc_mode 1) on a whole batch
    kp = max(args.limit * 10, args.limit)
    nchk = min(256, args.batch)
    a = idx.knn(Qn[:nchk], kp)
    idx.set_tc_mode(1)
    b = idx.knn(Qn[:nchk], kp)
    same = all((x.view(np.uint8) == y.view(np.uint8)).all() for x, y in zip(a, b))
    out = {"corpus": corpus, "value": m["nq"] * steps / (m["ms"] / 1e3), "unit": "queries/s", "ms_per_step": m["ms"] / steps,
           "steps": steps, "tc_queries": int(st.tc_queries), "tc_fallback_queries": int(st.tc_fallback_queries),
           "tc_second_chance_queries": int(st.tc_second_chance_queries),
           "tc_fallback_rate": (int(st.tc_fallback_queries) / int(st.tc_queries)) if int(st.tc_queries) else None,
           "filter_pass_ms": st.scan_ms_total / max(1, st.scan_launches_timed),
           "survivors_per_query": survivor_stats(m["survivors"]),
           "tc_equals_exact_scan": {"queries": nchk, "kprime": kp, "identical_rows_order_and_distances": bool(same)},
           "build_s": info["build_s"]}
    idx.close()
    del se
    torch.cuda.empty_cache()
    return out


def measure_python_api(args, idx, bm, se, Qn, tok_indptr, terms, limit, steps):
    """e2e through the advertised Python drop-in (VERDICT r01 weak #5): text tokens in, Python result lists out —
    HybridSearch.rrf_search_stream over the resident handle, including the term lookup and the construction of
    the result dicts; and the same stream with flat numpy token arrays in / packed numpy arrays out."""
    from rag_search_engine_b200 import HybridSearch
    T = len(bm.df)
    names = np.array([f"t{i}" for i in range(T)], dtype=np.str_)
    term_row = dict(zip(names.tolist(), range(T)))
    hs = HybridSearch.from_loaded(idx, term_row, se.movie_ids, se.movie_ids, registry_key=f"bench-{os.getpid()}-{id(idx)}",
                                  device=idx.device)
    nb = NB
    B = args.batch
    tok_lists, flat = [], []
    for b in range(nb):
        Qb, tp, tr = batch_slice(tok_indptr, terms, Qn, b * B, (b + 1) * B)
        toks = np.where(tr >= 0, names[np.clip(tr, 0, None)], "<oov>")
        flat.append(((tp, toks), Qb))
        tl = toks.tolist()
        tok_lists.append(([tl[tp[i]:tp[i + 1]] for i in range(B)], Qb))

    def run(batches, as_arrays):
        gen = (batches[i % nb] for i in range(steps))
        n = 0
        t0 = time.perf_counter()
        for out in hs.rrf_search_stream(gen, k=60, limit=limit, as_arrays=as_arrays):
            n += 1
        return time.perf_counter() - t0, out

    run(tok_lists, False); run(flat, True)                        # warm (sorted vocabulary, ticket slots)
    w_dict, last = run(tok_lists, False)
    w_arr, last_arr = run(flat, True)
    return {"value": B * steps / w_dict, "unit": "queries/s", "wall_ms_per_step": 1e3 * w_dict / steps,
            "api": "HybridSearch.rrf_search_stream(token lists, frozen vectors) -> list of result dicts per query "
                   "(term lookup in a 1M-entry dict + ~2.5k dicts built per batch, on the host, per step)",
            "arrays": {"value": B * steps / w_arr, "unit": "queries/s", "wall_ms_per_step": 1e3 * w_arr / steps,
                       "api": "the same stream with (tok_indptr, numpy str tokens) in and as_arrays=True out"},
            "hits_in_last_batch": int(sum(len(x) for x in last))}


def measure_text_in(args, idx, bm, se, tok_indptr, terms, limit, steps):
    """§8(f2): TEXT in — the MiniLM-L6 query encoder runs on the same GPU (csrc/encoder.cuh, random weights of the
    all-MiniLM-L6-v2 architecture: the checkpoint is not downloadable here and the arithmetic does not depend on
    the values) and hands its vectors to the hybrid step on the device (rse_encode_dev -> rse_hybrid_stage_dev).
    Every step uploads the token ids of ITS batch and reads its fused results back."""
    import torch
    from rag_search_engine_b200 import HybridSearch
    from rag_search_engine_b200.encoder import MINILM_L6_CONFIG, GpuSentenceEncoder, pack, random_state_dict
    enc = GpuSentenceEncoder(idx, random_state_dict(MINILM_L6_CONFIG, seed=5), MINILM_L6_CONFIG)
    B = args.batch
    rng = np.random.default_rng(17)
    id_batches, tok_batches = [], []
    for b in range(NB):
        lens = rng.integers(4, 17, B)                       # [CLS] + 2..14 word pieces + [SEP]: short search queries
        ids = [[101] + rng.integers(1000, 30000, L - 2).tolist() + [102] for L in lens]
        id_batches.append(ids)
        lo, hi = b * B, (b + 1) * B
        tok_batches.append(((tok_indptr[lo:hi + 1] - tok_indptr[lo]).astype(np.int32), terms[tok_indptr[lo]:tok_indptr[hi]]))
    tokens_per_batch = float(np.mean([sum(len(x) for x in ids) for ids in id_batches]))
    dev = torch.device("cuda", idx.device)
    qbuf = torch.empty((B, 384), dtype=torch.float32, device=dev)
    packed = [pack(ids) for ids in id_batches]

    def step(i):
        ids, _, cu = packed[i % NB]
        idx.encode_dev(enc.slot, ids, cu, qbuf.data_ptr())
        tp, tr = tok_batches[i % NB]
        idx.hybrid_stage_dev(B, qbuf.data_ptr(), tp, tr)
        idx.hybrid_run(0, 60.0, limit)
        return idx.hybrid_fetch(limit)

    for i in range(3):
        step(i)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for i in range(steps):
        step(i)
    torch.cuda.synchronize()
    wall = (time.perf_counter() - t0) / steps
    # the encoder alone, device-timed
    stream = torch.cuda.current_stream(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for i in range(steps):
        ids, _, cu = packed[i % NB]
        idx.encode_dev(enc.slot, ids, cu, qbuf.data_ptr())
    e1.record(stream)
    torch.cuda.synchronize()
    enc_ms = e0.elapsed_time(e1) / steps
    # index-build shaped input (semantic_search.py:199-206 encodes every chunk text at build time): 2048 chunks of
    # 24-64 word pieces per call, device-timed
    bulk_ids = [[101] + rng.integers(1000, 30000, int(L) - 2).tolist() + [102] for L in rng.integers(24, 65, 2048)]
    bids, _, bcu = pack(bulk_ids)
    bbuf = torch.empty((2048, 384), dtype=torch.float32, device=dev)
    idx.encode_dev(enc.slot, bids, bcu, bbuf.data_ptr())
    torch.cuda.synchronize()
    e0.record(stream)
    for _ in range(3):
        idx.encode_dev(enc.slot, bids, bcu, bbuf.data_ptr())
    e1.record(stream)
    torch.cuda.synchronize()
    bulk_ms = e0.elapsed_time(e1) / 3
    c = MINILM_L6_CONFIG
    flop_per_token = 2.0 * c["layers"] * (4 * c["hidden"] ** 2 + 2 * c["hidden"] * c["intermediate"])
    rerank = None
    try:
        rerank = measure_rerank(idx, limit)
    except Exception as e:                               # a bench extra must not take the line down
        rerank = {"error": repr(e)[:200]}
    return {"rerank": rerank, "value": B / wall, "unit": "queries/s", "wall_ms_per_step": 1e3 * wall, "queries_per_step": B,
            "api": "rse_encode_dev (MiniLM-L6 architecture, fp32) -> rse_hybrid_stage_dev -> rse_hybrid_run -> rse_hybrid_fetch",
            "encoder_ms_per_batch": enc_ms, "tokens_per_batch": tokens_per_batch,
            "encoder_tokens_per_s": tokens_per_batch / (enc_ms * 1e-3),
            "encoder_gemm_tflops": flop_per_token * tokens_per_batch / (enc_ms * 1e-3) / 1e12,
            "bulk_embed": {"chunks_per_call": 2048, "tokens_per_call": int(bcu[-1]), "ms_per_call": bulk_ms,
                           "chunks_per_s": 2048 / (bulk_ms * 1e-3), "tokens_per_s": int(bcu[-1]) / (bulk_ms * 1e-3),
                           "gemm_tflops": flop_per_token * int(bcu[-1]) / (bulk_ms * 1e-3) / 1e12,
                           "note": "index-build shaped input: 2048 chunk texts of 24-64 word pieces per call"},
            "weights": "random (seeded), all-MiniLM-L6-v2 architecture",
            "reference_cpu_encoder": "5-20 ms PER QUERY (SURVEY §8 f2: torch CPU via sentence-transformers; not installable here)"}


def measure_rerank(idx, limit):
    """§8(f3): the cross-encoder rerank of hybrid_search.py:279-312 — CrossEncoder.predict over the (query, document)
    pairs of the fused union (<= 2 * limit per query) — on the device: the TinyBERT-L2 architecture of
    cross-encoder/ms-marco-TinyBERT-L2-v2 with seeded random weights, pairs of an 8-token query and a 100-200 token
    document.  One query's pairs per call (the reference's call shape), and 64 queries' pairs in one call."""
    from rag_search_engine_b200.encoder import TINYBERT_L2_CONFIG, GpuCrossEncoder, random_state_dict
    ce = GpuCrossEncoder(idx, random_state_dict(TINYBERT_L2_CONFIG, seed=9, head=1), TINYBERT_L2_CONFIG)
    rng = np.random.default_rng(23)

    def pairs(n):
        ids, tts = [], []
        for _ in range(n):
            qn, dn = 8, int(rng.integers(100, 201))
            # numpy rows, as a tokenizer called with return_tensors="np" hands them over (Python int lists cost the
            # host ~50 ns per token in pack(): 10 ms for the 200 k tokens of the 64-query call)
            ids.append(np.concatenate(([101], rng.integers(1000, 30000, qn), [102], rng.integers(1000, 30000, dn), [102])).astype(np.int32))
            tts.append(np.concatenate((np.zeros(qn + 2, np.int32), np.ones(dn + 1, np.int32))))
        return ids, tts
    out = {}
    for name, n_pairs, reps in (("one_query", 2 * limit, 20), ("batch_of_64_queries", 64 * 2 * limit, 5)):
        ids, tts = pairs(n_pairs)
        for _ in range(2):
            ce.predict_ids(ids, tts)
        t0 = time.perf_counter()
        for _ in range(reps):
            sc = ce.predict_ids(ids, tts)
        dt = (time.perf_counter() - t0) / reps
        out[name] = {"pairs": n_pairs, "tokens": int(sum(len(x) for x in ids)), "call_ms": 1e3 * dt, "pairs_per_s": n_pairs / dt,
                     "finite": bool(np.isfinite(sc).all())}
    out["api"] = "GpuCrossEncoder.predict_ids -> rse_encode (packed tokens, pooler + classifier head), host buffers in and out"
    out["weights"] = "random (seeded), ms-marco-TinyBERT-L2-v2 architecture"
    return out


def measure_cold_open(emb_host, local_rank):
    """§8(f1): how long does a query-only open take?  The frozen sidecar's embedding matrix (a raw .npy next to the
    database, store.emb_matrix_path) is memory-mapped and handed to rse_load_embeddings, which streams it to HBM
    through two pinned 64 MB buffers (staging copy on a few threads).  Measured with the file just written (page cache warm)."""
    import shutil
    import tempfile
    from rag_search_engine_b200 import _lib
    d = Path(os.environ.get("TMPDIR", tempfile.gettempdir()))
    try:
        if shutil.disk_usage(d).free < emb_host.nbytes * 1.3:
            return {"skipped": f"not enough free space under {d}"}
        f = d / f"rse_bench_emb_{os.getpid()}.npy"
        np.save(f, emb_host)
        t0 = time.perf_counter()
        m = np.load(f, mmap_mode="r")
        idx = _lib.Index(local_rank)
        idx.load_embeddings(m)
        idx.synchronize()
        dt = time.perf_counter() - t0
        idx.close()
        del m
        f.unlink()
        return {"seconds": dt, "gbytes": emb_host.nbytes / 1e9, "gb_per_s": emb_host.nbytes / dt / 1e9,
                "what": "np.load(mmap) of the sidecar matrix + rse_load_embeddings (2 x 64 MB pinned buffers filled by min(16, cores) threads, row norms "
                        "included), page cache warm"}
    except Exception as e:                               # a bench extra must not take the line down
        return {"skipped": f"{type(e).__name__}: {e}"}


def measure_image_search(args, local_rank):
    """§8(f4): the ranking step of the image search (llm/multimodal.py:86-95: cosine of one CLIP image embedding
    against every movie text embedding + argsort) — 600 k x 512 fp32 text embeddings resident in HBM, rse_knn top-5
    per query (the any-width streaming scan), host buffers."""
    import torch
    from rag_search_engine_b200 import _lib
    dev = torch.device("cuda", local_rank)
    n, dim = args.movies, 512
    g = torch.Generator(device=dev).manual_seed(77)
    emb = torch.randn((n, dim), generator=g, device=dev)
    idx = _lib.Index(local_rank)
    idx.set_tc_mode(1)
    idx.attach_embeddings_dev(emb.data_ptr(), n, dim, keepalive=(emb,))
    q = torch.randn((8, dim), generator=g, device=dev).cpu().numpy()
    for i in range(3):
        idx.knn(q[i:i + 1], 5)
    reps = 20
    t0 = time.perf_counter()
    for i in range(reps):
        d, pos, _r, _m, cnt = idx.knn(q[i % 8:i % 8 + 1], 5)
    dt = (time.perf_counter() - t0) / reps
    # the reference expression on the same data (numpy on the host), one query
    e = emb.cpu().numpy()
    t1 = time.perf_counter()
    iv = q[0] / (np.linalg.norm(q[0]) + 1e-12)
    tn = e / (np.linalg.norm(e, axis=1, keepdims=True) + 1e-12)
    sims = (tn @ iv).astype(float)
    top = np.argsort(sims)[::-1][:5]
    cpu_dt = time.perf_counter() - t1
    d0, pos0, _r, _m, _c = idx.knn(q[0:1], 5)
    idx.close()
    return {"call_ms": 1e3 * dt, "queries_per_s": 1.0 / dt, "docs": n, "dim": dim,
            "scan_gbs": n * dim * 4 / dt / 1e9, "numpy_reference_ms": 1e3 * cpu_dt,
            "same_top5_as_numpy": bool(pos0[0].tolist() == top.tolist()),
            "max_similarity_diff": float(np.abs((1.0 - d0[0].astype(np.float64)) - sims[top]).max())}


def measure_small_batches(idx, Qn, limit):
    """Where does the tensor-core path take over from the streaming scan?  rse_knn_movies (host buffers) for small
    batches with the exact scan forced, K4 forced, and the library's automatic choice (VERDICT r01 weak #9)."""
    kp = max(limit * 10, limit)
    table = []
    for nq in (1, 2, 3, 4, 8, 16, 32, 47, 64):
        row = {"nq": nq}
        for name, mode in (("scan_ms", 1), ("tc_ms", 2), ("auto_ms", 0)):
            idx.set_tc_mode(mode)
            for _ in range(2):
                idx.knn_movies(Qn[:nq], limit, kp)
            reps = 5
            t0 = time.perf_counter()
            for r in range(reps):
                idx.knn_movies(Qn[r * nq:(r + 1) * nq], limit, kp)
            row[name] = round(1e3 * (time.perf_counter() - t0) / reps, 4)
        table.append(row)
    idx.set_tc_mode(0)
    return {"call": "rse_knn_movies, host buffers, S-600k, top-10 of K'=100", "rows": table,
            "auto_threshold": "nq >= 2 (RSE_TC_MIN_BATCH); a single query as well once a batch has built the shadow"}


def measure_rowshard(args, rank, world, local_rank, se, bm, tok_indptr, terms, Q, Qn, info, mode, param, limit, steps):
    """The same global batch through the ROW-SHARDED path (north_star: local top-K' per shard + candidate exchange
    + merge; sharded.py): device-timed steps with the batch resident, max over ranks, checked against one handle."""
    import torch
    import torch.distributed as dist
    from rag_search_engine_b200 import _lib, sharded
    device = torch.device("cuda", local_rank)
    C = info["chunks"]
    nq = args.batch
    bounds = sharded.shard_bounds(C, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    stream = torch.cuda.current_stream(device)
    idx = make_handle(args, local_rank, stream, se, bm, lo, hi, info["dim"])
    Qb, tp, tr = batch_slice(tok_indptr, terms, Qn, 0, nq)
    sh = sharded.NcclShardedHybrid(idx, Qb, tp, tr, device, nq)
    Qd = Q[:nq].to(device).contiguous()
    for _ in range(3):
        sh.step(Qd, mode, param, limit)
    torch.cuda.synchronize(); dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        r = sh.step(Qd, mode, param, limit, check=False)       # no host round trip inside the timed steps ...
    e1.record(stream)
    flagged_last = int(r.flagged.item())                       # ... the last step's flag count is checked here
    torch.cuda.synchronize(); dist.barrier()
    t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=device)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    ok = None
    if rank == 0:
        chk = make_handle(args, local_rank, stream, se, bm, 0, C, info["dim"])
        oid, osc, oa, ob, oc = chk.hybrid(mode, param, limit, Qb, tp, tr)
        ok = bool((r.ids.cpu().numpy() == oid).all() and (r.score.cpu().numpy() == osc).all() and
                  (r.count.cpu().numpy() == oc).all())
        chk.close()
    idx.close()
    dist.barrier()
    return {"value": nq * steps / (ms / 1e3), "unit": "queries/s", "ms_per_step": ms / steps, "steps": steps,
            "queries_per_step": nq, "parallelism": f"row-shard x{world} + candidate exchange (top-K') + query-slice BM25/fusion",
            "exchange": sh.exchange_kind, "flagged_queries_last_step": flagged_last, "sharded_matches_single_gpu": ok}


# ----------------------------------------------------------------------------- B200 arm
def run_b200(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist
    from rag_search_engine_b200 import sharded

    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)
    if world > 1 and args.scaling == "weak":
        args.batch = args.batch * world          # global batch; every rank serves its slice of it
    se, bm, tok_indptr, terms, Q, info = build_workload(args, f"cuda:{local_rank}", corpus=args.corpus)
    C = info["chunks"]
    par = args.parallelism
    if par == "auto":
        fits = C * info["dim"] * 6 < torch.cuda.get_device_properties(device).total_memory / 3
        par = "replicate" if fits else "rowshard"
    rowshard = world > 1 and par == "rowshard"
    stream = torch.cuda.current_stream(device)
    tm = Timer(stream, world, device)
    mode = 0 if args.mode == "rrf" else 1
    param = 60.0 if mode == 0 else 0.5
    limit, nq = args.limit, args.batch
    qs = sharded.query_slices(nq, world)
    qlo, qhi = (qs[rank], qs[rank + 1]) if (world > 1 and not rowshard) else (0, nq)

    if rowshard:
        line = run_b200_rowshard(args, rank, world, local_rank, se, bm, tok_indptr, terms, Q, info, mode, param, tm)
        if rank == 0:
            print(json.dumps(line), flush=True)
        return

    idx = make_handle(args, local_rank, stream, se, bm, 0, C, info["dim"])
    Qn, batches = pinned_batches(torch, Q, tok_indptr, terms, nq, qlo, qhi)
    m = measure_hybrid(idx, tm, batches, mode, param, limit, args.steps, args.warmup, sample_clocks=local_rank,
                       e2e=not args.no_e2e)
    if args.dump_outputs:
        oid, osc, oa, ob, oc = m["last"]
        dump_outputs(args.dump_outputs, {"id": oid, "score": osc, "bm25": oa, "semantic": ob, "count": oc})
    ms, st, clocks = m["ms"], m["stats"], m["clocks"]
    launches = int(st.kernel_launches)
    scan_ms = st.scan_ms_total / max(1, st.scan_launches_timed)
    scan_share = st.scan_ms_total / m["ms_local"] if m["ms_local"] > 0 else None
    value = nq * args.steps / (ms / 1e3)
    e2e = e2e_dict(m, nq, args.steps, world) if m["e2e"] else None
    res = m["results"]

    # ---- the other fusion mode of configs[3] (weighted alpha = 0.5 next to rrf): same batches, fewer steps
    other = None
    if not args.no_extras:
        omode, oparam, oname = (1, 0.5, "weighted") if mode == 0 else (0, 60.0, "rrf")
        osteps = min(args.steps, 40)
        mo_ = measure_hybrid(idx, tm, batches, omode, oparam, limit, osteps, 3, e2e=not args.no_e2e)
        other = {"mode": oname, "param": oparam, "value": nq * osteps / (mo_["ms"] / 1e3), "unit": "queries/s",
                 "ms_per_step": mo_["ms"] / osteps, "steps": osteps,
                 "e2e": e2e_dict(mo_, nq, osteps, world) if mo_["e2e"] else None,
                 "note": "r01's 55.9 k q/s weighted-mode figure (gpurun_out/b_weighted.log) was an artefact of the "
                         "bench of that hour, which took an inline NVML sample (~25 ms of host time) every 8 steps "
                         "inside the device-resident loop; the kernels of the two modes differ only in fuse_kernel"}

    # ---- full-size parity of the tensor-core path: the whole of batch 0 through K4 and through the exact scan
    tc_same = None
    if world == 1 and not args.no_extras:
        kp_ = max(limit * 10, limit)
        a_ = idx.knn(Qn[:min(256, nq)], kp_)
        idx.set_tc_mode(1)
        b_ = idx.knn(Qn[:min(256, nq)], kp_)
        idx.set_tc_mode(args.tc_mode if args.tc_mode >= 0 else 0)
        tc_same = {"queries": min(256, nq), "kprime": kp_,
                   "identical_rows_order_and_distances": bool(all((x.view(np.uint8) == y.view(np.uint8)).all() for x, y in zip(a_, b_)))}

    # ---- batch-1 KNN (north_star: batch-1 kNN as a fraction of HBM peak): scan<QB=1> alone + whole call
    knn1 = knn1k = small = pyapi = textin = None
    if world == 1 and not args.no_knn1:
        kp = max(limit * 10, limit)
        idx.set_tc_mode(1)                     # the HBM-bound exact streaming scan (the north_star's batch-1 kernel)
        for _ in range(3):
            idx.knn_movies(Qn[:1], limit, kp)
        idx.set_timing(True); idx.stats_reset()
        reps = 20
        t0 = time.perf_counter()
        for i in range(reps):
            idx.knn_movies(Qn[i: i + 1], limit, kp)
        wall1 = (time.perf_counter() - t0) / reps
        s1 = idx.stats(); idx.set_timing(False)
        sm1 = s1.scan_ms_total / max(1, s1.scan_launches_timed)
        knn1 = {"scan_ms": sm1, "call_ms_host_buffers": 1e3 * wall1, "launches_per_query": s1.kernel_launches / reps}
        idx.set_tc_mode(0)                     # the library's own choice: K4 over the fp16 shadow once a batch has built it
        for _ in range(3):
            idx.knn_movies(Qn[:1], limit, kp)
        t0 = time.perf_counter()
        for i in range(reps):
            idx.knn_movies(Qn[i: i + 1], limit, kp)
        knn1["auto_call_ms_host_buffers"] = 1e3 * (time.perf_counter() - t0) / reps
        knn1["auto_path"] = "K4 (shadow built by the hybrid batches above): 768 B per row instead of 1536"
        # configs[2]: batch-1024 semantic search (KNN top-K' + per-movie best chunk) through the host-buffer call
        Q1k = Qn[:1024]
        for _ in range(2):
            idx.knn_movies(Q1k, limit, kp)
        idx.set_timing(True); idx.stats_reset()
        reps = 5
        t0 = time.perf_counter()
        for _ in range(reps):
            idx.knn_movies(Q1k, limit, kp)
        wall1k = (time.perf_counter() - t0) / reps
        s1k = idx.stats(); idx.set_timing(False)
        f_ms = s1k.scan_ms_total / max(1, s1k.scan_launches_timed)
        knn1k = {"call_ms_host_buffers": 1e3 * wall1k, "queries_per_s": 1024 / wall1k, "filter_pass_ms": f_ms,
                 "filter_tflops": 2.0 * 384 * C * 256 / (f_ms * 1e-3) / 1e12 if f_ms > 0 else None,
                 "tc_fallback_queries": int(s1k.tc_fallback_queries)}
        if not args.no_extras:
            small = measure_small_batches(idx, Qn, limit)
            pyapi = measure_python_api(args, idx, bm, se, Qn, tok_indptr, terms, limit, min(args.steps, 40))
            textin = measure_text_in(args, idx, bm, se, tok_indptr, terms, limit, min(args.steps, 20))

    replicas_ok = mismatch = corpora_identical = rowshard_extra = None
    if world > 1:
        # every rank generates the corpus on its own GPU from the same seeds: verify they really are the same bits
        def csum(t):
            t = t.contiguous().view(torch.int32) if t.dtype == torch.float32 else t.to(torch.int64)
            return int(t.to(torch.int64).sum().item())
        sig = [csum(se.emb), csum(se.movie_of_chunk), csum(torch.as_tensor(np.asarray(bm.doc_idx).astype(np.int64))),
               csum(torch.as_tensor(np.asarray(bm.tf).astype(np.int64))), int(np.asarray(tok_indptr).sum()),
               int(np.asarray(terms).astype(np.int64).sum()), csum(torch.as_tensor(Qn).view(torch.int32))]
        sigs = [None] * world
        dist.all_gather_object(sigs, sig)
        corpora_identical = all(x == sigs[0] for x in sigs)
        # rank 0 holds the whole corpus: the gathered slices of batch 0 must equal one handle's run of the whole batch
        mine = res[0] if res is not None else idx.hybrid(mode, param, limit, *batches[0])
        parts = [None] * world
        dist.all_gather_object(parts, (mine[0], mine[1], mine[4]))
        got = tuple(np.concatenate([p[i] for p in parts]) for i in range(3))
        if rank == 0:
            oid, osc, oa, ob, oc = idx.hybrid(mode, param, limit, *batch_slice(tok_indptr, terms, Qn, 0, nq))
            replicas_ok = bool((got[0] == oid).all() and (got[1] == osc).all() and (got[2] == oc).all())
            if not replicas_ok:
                badq = np.nonzero((got[0] != oid).any(axis=1) | (got[1] != osc).any(axis=1) | (got[2] != oc))[0]
                mismatch = {"queries": int(len(badq)), "first": [int(x) for x in badq[:8]]}
        if args.parallelism == "auto" and not args.no_extras:
            rowshard_extra = measure_rowshard(args, rank, world, local_rank, se, bm, tok_indptr, terms, Q, Qn, info, mode,
                                              param, limit, min(args.steps, 30))
        dist.barrier()

    # ---- CPU baseline + clustered corpora (rank 0 of a 1-GPU run), then configs[4]
    cpu = cold = None
    clustered = []
    if world == 1 and not args.no_cpu_baseline:
        cores = os.cpu_count() or 1
        sample = min(nq, args.cpu_sample or 2 * cores)
        emb_host = se.emb.cpu().numpy()
        movie_of = se.movie_of_chunk.cpu().numpy().astype(np.int64)
        Qb, tp, tr = batch_slice(tok_indptr, terms, Qn, 0, nq)
        qps, dt, cpu_out = cpu_hybrid_sample(emb_host, movie_of, bm, se.movie_ids, Qb, tp, tr, limit, args.mode, sample, cores)
        # the sample doubles as a full-size parity check of the GPU results
        oid, osc, oa, ob, oc = res[0] if res is not None else idx.hybrid(mode, param, limit, Qb, tp, tr)
        ok = all([int(x) for x in oid[q, :oc[q]]] == [r["id"] for r in cpu_out[q]] and
                 [float(x) for x in osc[q, :oc[q]]] == [r["score"] for r in cpu_out[q]] for q in range(sample))
        # the reference itself is single-threaded (SURVEY §8d): the same port on ONE core, two queries
        qps1, dt1, _ = cpu_hybrid_sample(emb_host, movie_of, bm, se.movie_ids, Qb, tp, tr, limit, args.mode, 2, 1)
        cpu = {"value": qps, "unit": "queries/s", "cores": cores, "kind": "port",
               "one_core": {"value": qps1, "unit": "queries/s", "sample": f"2 queries, {dt1:.1f} s"},
               "sample": f"{sample} hybrid queries of batch 0 over the full corpus, {dt:.1f} s (OpenMP over queries; "
                         f"literal vec0 scan per query)", "gpu_matches_cpu_on_sample": bool(ok)}
        if not args.no_extras:
            cold = measure_cold_open(emb_host, local_rank)
        del emb_host
    ptouched = postings_touched(bm, terms) // NB
    idx.close()
    if world == 1 and not args.no_extras and args.corpus == "isotropic":
        del se
        torch.cuda.empty_cache()
        for corpus in ("clustered", "clustered_dense"):
            clustered.append(measure_corpus_variant(args, local_rank, device, stream, bm, corpus, min(args.steps, 20), tm))
    image = None
    if world == 1 and not args.no_extras:
        try:
            image = measure_image_search(args, local_rank)
        except Exception as e:                            # a bench extra must not take the line down
            image = {"skipped": f"{type(e).__name__}: {e}"}
    knn100m = None
    if not args.no_extras and not args.no_knn100m:
        se = None
        torch.cuda.empty_cache()
        knn100m = knn100m_measure(args, rank, world, local_rank, steps=min(args.steps, 20), batch=256)
    if rank != 0:
        return

    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    peak = float(peaks.get("hbm_gbs", 6650.0))
    nq_loc = qhi - qlo
    qb = 16 if nq_loc >= 9 else (8 if nq_loc >= 5 else (4 if nq_loc >= 3 else nq_loc))
    tc_used = int(st.tc_filter_launches) > 0
    kname, row_bytes = scan_kernel_desc(args, tc_used, qb)
    alg_bytes = C * row_bytes
    # DRAM bytes per launch of the dominant kernel, from the committed ncu --set full capture (profiles/): only
    # quoted when this run has the shard size that was profiled
    traffic = None
    for tj in sorted((ROOT / "profiles").glob("r0*_dominant_kernel_traffic.json"), reverse=True):
        t = json.loads(tj.read_text())
        if t.get("rows") == C and t.get("tc_kind") == (tc_kind(args) if tc_used else "scan"):
            traffic = t.get("dram_bytes_read", 0) + t.get("dram_bytes_write", 0)
            break
    hbm_achieved = alg_bytes / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else None
    psrc = "MEASURED_PEAKS.json" if peaks else "fallback"
    if tc_used:
        # The batched filter pass is bound by the tensor pipe (+ TMEM reads), not by the stream (DESIGN.md §5).
        # Algorithmic work: 2*384 flop per (row, query) pair.  Peak: the BURST figure when the SM clock sampled
        # during the timed region sat at its maximum with no power cap (a short run), the SUSTAINED one otherwise.
        q_per_pass = min(nq_loc, 256)
        flops = 2.0 * 384 * C * q_per_pass
        burst = float(peaks.get("bf16_tflops", 1623.4))
        sustained = float(peaks.get("bf16_tflops_sustained", 1379.6))
        at_max = bool(clocks and clocks.get("sm_mhz") and clocks.get("sm_max_mhz") and
                      clocks["sm_mhz"] >= 0.97 * clocks["sm_max_mhz"] and "sw_power_cap" not in (clocks.get("reasons") or []))
        tpeak = burst if at_max else sustained
        tach = flops / (scan_ms * 1e-3) / 1e12 if scan_ms > 0 else None
        roofline = {"bound": "tensor", "kernel": kname, "achieved": tach, "peak": tpeak, "unit": "TFLOP/s",
                    "frac": (tach / tpeak) if tach else None,
                    "peak_source": f"{psrc} {'bf16_tflops (burst: SM clock at max, no power cap during the timed region)' if at_max else 'bf16_tflops_sustained (SM clock below max / power-capped during the timed region)'}; "
                                   f"f16 and bf16 share the tensor rate",
                    "frac_of_burst_peak": (tach / burst) if tach else None,
                    "frac_of_sustained_peak": (tach / sustained) if tach else None,
                    "traffic": traffic, "algorithmic_flops_per_launch": flops, "queries_per_pass": q_per_pass,
                    "avg_launch_ms": scan_ms,
                    "hbm": {"achieved": hbm_achieved, "peak": peak, "unit": "GB/s",
                            "frac": (hbm_achieved / peak) if hbm_achieved else None,
                            "algorithmic_bytes_per_launch": alg_bytes, "bytes_per_row": row_bytes},
                    "scan_launches": int(st.scan_launches_timed), "scan_share_of_step": scan_share,
                    "tc_queries": int(st.tc_queries), "tc_fallback_queries": int(st.tc_fallback_queries),
                    "tc_second_chance_queries": int(st.tc_second_chance_queries),
                    "survivors_per_query": survivor_stats(m["survivors"]), "tc_equals_exact_scan": tc_same}
    else:
        roofline = {"bound": "hbm", "kernel": kname,
                    "achieved": hbm_achieved, "peak": peak, "unit": "GB/s", "frac": (hbm_achieved / peak) if hbm_achieved else None,
                    "peak_source": f"{psrc} hbm_gbs", "traffic": traffic, "algorithmic_bytes_per_launch": alg_bytes,
                    "avg_launch_ms": scan_ms, "scan_launches": int(st.scan_launches_timed), "scan_share_of_step": scan_share,
                    "tc_queries": int(st.tc_queries), "tc_fallback_queries": int(st.tc_fallback_queries)}
    if knn1:
        g1 = C * ROW_BYTES / (knn1["scan_ms"] * 1e-3) / 1e9
        knn1.update(achieved_gbs=g1, frac_of_measured_peak=g1 / peak, queries_per_s=1e3 / knn1["call_ms_host_buffers"])
    line = {"metric": "hybrid queries/sec", "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "ms_per_step_ranks": [round(v / args.steps, 4) for v in m["ms_ranks"]],
            "scaling": (args.scaling if world > 1 else "weak"), "vs_baseline": None,
            "dtype": "f16 tensor-core filter + exact f32 re-score (f64 tail), f64 BM25/fusion", "data": "synthetic",
            "config": config_dict(args, info, world, par), "roofline": roofline, "clocks": clocks, "e2e": e2e,
            "gpu_launches": launches,
            "bm25": {"queries": int(st.bm25_queries), "fallback_queries": int(st.bm25_fallback_queries),
                     "finalists_rescored": int(st.bm25_finalists), "candidates_merged": int(st.bm25_candidates)},
            "bytes_moved_resident_loop": {"h2d": int(st.h2d_bytes), "d2h": int(st.d2h_bytes)},
            ("weighted" if mode == 0 else "rrf"): other, "clustered": clustered or None, "e2e_python": pyapi, "text_in": textin,
            "knn_small_batches": small, "knn100m": knn100m, "cold_open": cold, "image_search": image,
            "replicas_match_single_gpu": replicas_ok, "mismatch": mismatch,
            "corpora_identical_across_ranks": corpora_identical,
            "rowshard": rowshard_extra, "knn_batch1": knn1, "knn_batch1024": knn1k, "postings_touched_per_step": ptouched}
    if cpu:
        line["cpu_baseline"] = cpu
    print(json.dumps(line), flush=True)


def run_b200_rowshard(args, rank, world, local_rank, se, bm, tok_indptr, terms, Q, info, mode, param, tm):
    """--parallelism rowshard as the MAIN line (a corpus that does not fit one GPU takes this path)."""
    import torch
    import torch.distributed as dist
    from rag_search_engine_b200 import sharded
    device = torch.device("cuda", local_rank)
    stream = tm.stream
    C, nq, limit = info["chunks"], args.batch, args.limit
    bounds = sharded.shard_bounds(C, world)
    lo, hi = bounds[rank], bounds[rank + 1]
    idx = make_handle(args, local_rank, stream, se, bm, lo, hi, info["dim"])
    Qn = Q.cpu().numpy()
    Qb, tp, tr = batch_slice(tok_indptr, terms, Qn, 0, nq)
    sh = sharded.NcclShardedHybrid(idx, Qb, tp, tr, device, nq)
    Qd = Q[:nq].to(device).contiguous()
    for _ in range(max(args.warmup, 3)):
        sh.step(Qd, mode, param, limit)
    torch.cuda.synchronize(); dist.barrier()
    idx.set_timing(True); idx.stats_reset()
    sampler = ClockSampler(local_rank); sampler.start()
    tm.e0.record(stream)
    for _ in range(args.steps):
        r = sh.step(Qd, mode, param, limit, check=False)
    tm.e1.record(stream)
    torch.cuda.synchronize(); dist.barrier()
    clocks = sampler.stop()
    ms = tm.max_over_ranks(tm.e0.elapsed_time(tm.e1))
    st = idx.stats(); idx.set_timing(False)
    # e2e: stage (H2D of this rank's slice + the batch's query vectors) + step + D2H of the fused batch
    Qh = torch.empty((nq, info["dim"]), dtype=torch.float32, pin_memory=True); Qh.copy_(Q[:nq].cpu())
    torch.cuda.synchronize(); dist.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sh.stage_slice()
        Qd2 = Qh.to(device, non_blocking=True)
        r2 = sh.step(Qd2, mode, param, limit)
        _ = r2.ids.cpu(), r2.score.cpu(), r2.count.cpu()
    torch.cuda.synchronize(); dist.barrier()
    wall = tm.max_over_ranks(time.perf_counter() - t0)
    ok = None
    if rank == 0:
        chk = make_handle(args, local_rank, stream, se, bm, 0, C, info["dim"])
        oid, osc, oa, ob, oc = chk.hybrid(mode, param, limit, Qb, tp, tr)
        ok = bool((r.ids.cpu().numpy() == oid).all() and (r.score.cpu().numpy() == osc).all() and
                  (r.count.cpu().numpy() == oc).all())
        chk.close()
    dist.barrier()
    scan_ms = st.scan_ms_total / max(1, st.scan_launches_timed)
    line = {"metric": "hybrid queries/sec", "value": nq * args.steps / (ms / 1e3), "unit": "queries/s", "n_gpus": world,
            "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": args.scaling, "vs_baseline": None,
            "dtype": "f16 tensor-core filter + exact f32 re-score (f64 tail), f64 BM25/fusion", "data": "synthetic",
            "config": config_dict(args, info, world, "rowshard"),
            "roofline": {"bound": "tensor", "kernel": scan_kernel_desc(args, True, 16)[0], "avg_launch_ms": scan_ms,
                         "achieved": 2.0 * 384 * (hi - lo) * min(nq, 256) / (scan_ms * 1e-3) / 1e12 if scan_ms else None,
                         "unit": "TFLOP/s", "peak": None, "frac": None, "traffic": None,
                         "tc_queries": int(st.tc_queries), "tc_fallback_queries": int(st.tc_fallback_queries)},
            "clocks": clocks,
            "e2e": {"value": nq * args.steps / wall, "unit": "queries/s", "h2d_bytes_per_step": int(Qh.numpy().nbytes),
                    "d2h_bytes_per_step": int(nq * limit * 16 + nq * 4), "wall_ms_per_step": 1e3 * wall / args.steps},
            "gpu_launches": int(st.kernel_launches), "exchange": sh.exchange_kind, "sharded_matches_single_gpu": ok}
    idx.close()
    return line


def run_bm25_10k(args, local_rank):
    """configs[1]: key_search BM25 top-10, 10k-query batch over the GPU CSR postings (host-buffer call)."""
    import torch
    from rag_search_engine_b200 import _lib, synth
    torch.cuda.set_device(local_rank)
    bm = synth.synth_bm25(args.movies, args.vocab, seed=1234, device=f"cuda:{local_rank}")
    nq = 10_000
    tok_indptr, terms = synth.synth_token_queries(bm, nq, seed=99)
    idx = _lib.Index(local_rank)
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    for _ in range(max(args.warmup, 3)):
        sc, dc, cnt = idx.bm25(tok_indptr, terms, 10)
    idx.stats_reset()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        sc, dc, cnt = idx.bm25(tok_indptr, terms, 10)
    wall = (time.perf_counter() - t0) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"score": sc, "doc": dc, "count": cnt})
    launches = int(idx.stats().kernel_launches)
    touched = postings_touched(bm, terms)
    import oracle
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)
    ns = 512
    tp = tok_indptr[: ns + 1].astype(np.int32)
    t0 = time.perf_counter()
    osc, odc, ocnt = oracle.bm25_batch(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl, tp, terms[: tp[-1]], 10)
    cpu_dt = time.perf_counter() - t0
    ok = bool((odc == dc[:ns]).all() and (osc.view(np.uint64) == sc[:ns].view(np.uint64)).all() and (ocnt == cnt[:ns]).all())
    peak = 6546.6
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peak = float(json.loads(pk.read_text()).get("hbm_gbs", peak))
    ach = touched * 12 / wall / 1e9
    print(json.dumps({"metric": "BM25 top-10 queries/sec (10k-query batch)", "value": nq / wall, "unit": "queries/s",
                      "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": 1e3 * wall,
                      "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                      "config": {"workload": "configs[1]: movies_600k-shaped BM25 index, 10k-query batch, top-10",
                                 "docs": args.movies, "postings": int(len(bm.doc_idx)), "postings_touched": touched},
                      "roofline": {"bound": "hbm", "kernel": "bm25_score_kernel", "achieved": ach, "peak": peak, "unit": "GB/s",
                                   "frac": ach / peak, "traffic": None,
                                   "note": "12 B per touched posting over the whole host-buffer call (H2D/D2H included)"},
                      "e2e": {"value": nq / wall, "unit": "queries/s", "h2d_bytes_per_step": int(terms.nbytes * 3 + tok_indptr.nbytes),
                              "d2h_bytes_per_step": int(sc.nbytes + dc.nbytes + cnt.nbytes)},
                      "gpu_launches": launches,
                      "cpu_baseline": {"value": ns / cpu_dt, "unit": "queries/s", "cores": cores, "kind": "port",
                                       "sample": f"first {ns} queries of the batch (oracle.c BM25 over CSR, OpenMP)",
                                       "gpu_matches_cpu_on_sample": ok}}), flush=True)
    idx.close()




# ----------------------------------------------------------------------------- configs[4]: 100M-chunk corpus
KNN100M_UNIT = 313 * 1024            # rows per generation unit (a whole number of vec0 blocks); 39 units = 12 499 968 rows
KNN100M_TOTAL_UNITS = 312            # 99 999 744 rows ("100 M"): 8 shards of 39 units, each aligned to vec0 blocks


def knn100m_measure(args, rank, world, local_rank, steps, batch=256, total_units=None, keep_outputs=False):
    """configs[4] AS SPECIFIED: a FIXED synthetic 100M x 384 fp32 corpus (99 999 744 rows: 312 units of 313 vec0
    blocks, unit u generated from seed 1234+u whatever N is) sharded by row over N GPUs, top-100, candidate
    exchange + merge — STRONG scaling over N = 2, 4, 8 (rows per GPU = 100M / N; 256 queries per step in total).
    One GPU cannot hold 100M rows (153.6 GB fp32 + 76.8 GB fp16 shadow): N = 1 measures an ANCHOR, the first
    half of the same corpus (= the N = 2 shard, no exchange)."""
    import torch
    import torch.distributed as dist
    from rag_search_engine_b200 import _lib, sharded
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    units_total = total_units or KNN100M_TOTAL_UNITS
    anchor = world == 1
    n_shards = 2 if anchor else world
    if units_total % n_shards:
        return {"skipped": f"{units_total} units do not split over {n_shards} shards"}
    upg = units_total // n_shards                       # units per GPU
    rows = upg * KNN100M_UNIT
    need = rows * 384 * 6 + rows * 4 * 17 + (2 << 30)
    free, _total = torch.cuda.mem_get_info(dev)
    if need > free:
        return {"skipped": f"needs {need / 2**30:.0f} GiB per GPU, {free / 2**30:.0f} GiB free"}
    t0 = time.time()
    emb = torch.empty((rows, 384), dtype=torch.float32, device=dev)
    for u in range(upg):
        g = torch.Generator(device=dev).manual_seed(1234 + rank * upg + u)
        x = torch.randn((KNN100M_UNIT, 384), generator=g, device=dev)
        x /= x.norm(dim=1, keepdim=True)
        emb[u * KNN100M_UNIT:(u + 1) * KNN100M_UNIT] = x
        del x
    base = rank * rows
    movie = ((torch.arange(rows, device=dev, dtype=torch.int64) + base) // 8).to(torch.int32)   # 8 chunks per "movie"
    torch.cuda.synchronize()
    build_s = time.time() - t0
    idx = _lib.Index(local_rank)
    if args.tc_mode >= 0:
        idx.set_tc_mode(args.tc_mode)
    stream = torch.cuda.current_stream(dev)
    idx.set_stream(stream.cuda_stream)
    idx.attach_embeddings_dev(emb.data_ptr(), rows, 384, movie_idx_ptr=movie.data_ptr(), pos_base=base, keepalive=(emb, movie))
    nq, kp = batch, 100
    gq = torch.Generator(device=dev).manual_seed(99)
    Q = torch.randn((nq, 384), generator=gq, device=dev)
    Q /= Q.norm(dim=1, keepdim=True)
    if rank == 0:
        Q[: min(8, nq)] = emb[torch.arange(min(8, nq), device=dev) * 1000 + 5]       # known self-hits (rows of shard 0)
    if world > 1:
        dist.broadcast(Q, 0)
    qsl = sharded.query_slices(nq, world)
    ns = qsl[rank + 1] - qsl[rank]
    exchange_kind = "none (1 rank)"
    if world > 1:                                         # the handle owns the NCCL communicator (include/rse.h)
        ids = [idx.comm_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(ids, src=0)
        idx.comm_init(ids[0], world, rank)
        n_ranks, _r, ver = idx.comm_info()
        exchange_kind = f"library-owned NCCL {ver}: grouped ncclSend/ncclRecv all-to-all by query slice ({n_ranks} ranks)"
    cand = torch.empty((nq, kp, 3), dtype=torch.int64, device=dev)
    od = torch.empty((max(ns, 1), kp), dtype=torch.float32, device=dev)
    orow = torch.empty((max(ns, 1), kp), dtype=torch.int64, device=dev)
    om = torch.empty((max(ns, 1), kp), dtype=torch.int32, device=dev)
    oc = torch.empty((max(ns, 1),), dtype=torch.int32, device=dev)
    flags = torch.zeros((1,), dtype=torch.int32, device=dev)
    idx.set_defer_flags(True)

    def step():
        if world > 1:      # local top-K' of all queries -> all-to-all -> merge + aggregation of this rank's slice, one call
            idx.knn_sharded_dev(Q.data_ptr(), nq, kp, kp, od.data_ptr(), orow.data_ptr(), om.data_ptr(), oc.data_ptr(),
                                flags.data_ptr())
            return
        idx.knn_local_dev(Q.data_ptr(), nq, kp, cand.data_ptr())
        idx.knn_flags_dev(flags.data_ptr())                                            # += flagged queries (device)
        idx.knn_merge_movies_dev(cand.data_ptr(), 1, nq, kp, kp, od.data_ptr(), orow.data_ptr(), om.data_ptr(), oc.data_ptr())

    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    flags.zero_()
    idx.set_timing(True); idx.stats_reset()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(steps):
        step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1)
    st = idx.stats()
    idx.set_timing(False)
    # results: every rank holds its query slice; a checksum over all slices lets records of different N be compared
    sig = torch.stack([(orow[:ns].to(torch.float64)).sum(), od[:ns].view(torch.int32).to(torch.float64).sum(),
                       oc[:ns].to(torch.float64).sum(), flags.to(torch.float64).sum(),
                       (od[:ns, 0] <= 1e-6).to(torch.float64).sum()]) if ns > 0 else torch.zeros(5, dtype=torch.float64, device=dev)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(sig, op=dist.ReduceOp.SUM)
    ms = float(t.item())
    sig = sig.cpu().tolist()
    outputs = None
    if keep_outputs:                                      # this rank's query slice, as the last timed step left it
        outputs = {"dist": od[:ns].cpu().numpy(), "row": orow[:ns].cpu().numpy(), "movie": om[:ns].cpu().numpy(),
                   "count": oc[:ns].cpu().numpy()}
    scan_ms = st.scan_ms_total / max(1, st.scan_launches_timed)
    idx.close()
    del emb, movie
    torch.cuda.empty_cache()
    peaks = {}
    pk = ROOT / "MEASURED_PEAKS.json"
    if pk.exists():
        peaks = json.loads(pk.read_text())
    total_rows = rows * world
    qps = nq * steps / (ms / 1e3)
    tfl = 2.0 * 384 * rows * min(nq, 256) / (scan_ms * 1e-3) / 1e12 if scan_ms > 0 else None
    return {"workload": ("configs[4]: FIXED synthetic 99 999 744 x 384 fp32 corpus row-sharded over N GPUs, top-100, "
                         "candidate exchange + merge; strong scaling over N = 2, 4, 8" if not anchor else
                         "configs[4] ANCHOR: 100M rows do not fit one GPU — the first half of the corpus (the N = 2 shard) "
                         "on one GPU, no exchange"),
            "value": qps * total_rows, "unit": "query-chunks/s", "queries_per_s": qps, "ms_per_step": ms / steps, "steps": steps,
            "n_gpus": world, "scaling": "strong" if not anchor else "anchor", "rows_per_gpu": rows, "total_rows": total_rows,
            "queries_per_step": nq, "exchange": exchange_kind, "build_s": round(build_s, 1),
            "filter_pass_ms": scan_ms, "filter_tflops_per_gpu": tfl,
            "filter_frac_of_sustained_peak": (tfl / float(peaks.get("bf16_tflops_sustained", 1379.6))) if tfl else None,
            "shadow_stream_gbs_per_gpu": rows * ROW_BYTES_SHADOW / (scan_ms * 1e-3) / 1e9 if scan_ms > 0 else None,
            "flagged_queries_in_timed_steps": int(sig[3]), "self_hits_found": int(sig[4]), "full_k": bool(sig[2] == nq * kp),
            "result_checksum": {"rowid_sum": sig[0], "dist_bits_sum": sig[1]},
            "gpu_launches": int(st.kernel_launches), **({"outputs": outputs} if keep_outputs else {})}


def run_knn100m(args, rank, world, local_rank):
    """--workload knn100m: configs[4] alone (see knn100m_measure)."""
    units = None
    if args.shard_rows:                                   # a smaller corpus for experiments: units per GPU given
        units = max(1, args.shard_rows // KNN100M_UNIT) * (2 if world == 1 else world)
    r = knn100m_measure(args, rank, world, local_rank, args.steps, args.batch, total_units=units,
                        keep_outputs=bool(args.dump_outputs))
    if rank != 0:
        return
    outputs = r.pop("outputs", None)
    if args.dump_outputs:
        if outputs is None:
            raise SystemExit(f"--dump-outputs: nothing was measured ({r.get('skipped')})")
        dump_outputs(args.dump_outputs, outputs)
    line = {"metric": "kNN top-100 queries/sec x corpus chunks (row-sharded, candidate exchange + merge)",
            "value": r.get("value"), "unit": "query-chunks/s", "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": r.get("ms_per_step"), "higher_is_better": True,
            "scaling": r.get("scaling"), "vs_baseline": None, "dtype": "f16-shadow filter + f32 exact re-score",
            "data": "synthetic", "config": {"workload": r.get("workload"), "rows_per_gpu": r.get("rows_per_gpu"),
                                            "total_rows": r.get("total_rows"), "queries_per_step": r.get("queries_per_step")},
            "knn100m": r, "gpu_launches": r.get("gpu_launches")}
    print(json.dumps(line), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.dump_outputs and (world > 1 or args.impl == "reference"):
        raise SystemExit("--dump-outputs: the b200 arm in one process only")
    if args.dump_outputs and args.steps < 1:
        raise SystemExit("--dump-outputs: needs --steps >= 1 (it writes what the last timed step computed)")
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        if args.workload == "bm25_10k":
            if rank == 0:
                run_bm25_10k(args, local_rank)
        elif args.workload == "knn100m":
            run_knn100m(args, rank, world, local_rank)
        else:
            run_b200(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.barrier()
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
