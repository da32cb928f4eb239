"""The semantic index build on the device against the fallback build with the same encoder, per stage, on a seeded
movies_600k-shaped corpus (descriptions of 3-25 sentences of tests/helpers/wp_corpus.py text, a WordPieceTrainer
vocab, MiniLM-L6 shapes with seeded weights).  Writes profiles/r09_device_build.json (or --out) with the GPU's name
and power limit read in the same run.

    python scripts/device_build_bench.py --movies 600000
"""
import argparse
import json
import shutil
import subprocess
import sys
import tempfile
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path[:0] = [str(ROOT), str(ROOT / "tests")]


def gpu_info():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=60).stdout.strip().splitlines()[0]
        name, power = [x.strip() for x in out.split(",")]
        return name, power
    except Exception as e:                                     # noqa: BLE001
        return f"unknown ({e})", "not measured"


def movies(n, seed, needs_host):
    """Descriptions of 3-25 sentences drawn from wp_corpus text the device tokenizer takes (a movie the host
    tokenizer has to take is rare in real descriptions; the tests cover that route)."""
    import random
    from helpers import wp_corpus
    rnd = random.Random(seed)
    pool = [" ".join(t.split()[:14]) or "x" for t in wp_corpus.texts(40000, seed=seed)]
    pool = [t for t in pool if not needs_host(t)]
    return [(i + 1, rnd.choice(pool)[:40] or "t",
             " ".join(rnd.choice(pool) + rnd.choice(".!?") for _ in range(rnd.randint(3, 25)))) for i in range(n)]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--movies", type=int, default=600000)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r09_device_build.json"))
    a = ap.parse_args()
    import torch
    from helpers import wp_corpus
    from rag_search_engine_b200 import runtime, store
    from rag_search_engine_b200.encoder import MINILM_L6_CONFIG, DeviceWordPiece, GpuSentenceEncoder, random_state_dict
    from rag_search_engine_b200.semantic_search import SemanticSearch
    name, power = gpu_info()
    tmp = Path(tempfile.mkdtemp(prefix="devbuild-"))
    rec = {"gpu": name, "power_limit": power, "movies": a.movies, "max_chunk_size": 3, "overlap": 1}
    try:
        from rag_search_engine_b200.wordpiece import build_tables
        tok = wp_corpus.tokenizer("uncased")
        mv = movies(a.movies, seed=1, needs_host=build_tables(tok).needs_host)
        docs = tmp / "movies.json"
        docs.write_text(json.dumps({"movies": [{"id": i, "title": t, "description": d} for i, t, d in mv]}))
        cfg = dict(MINILM_L6_CONFIG, vocab_size=len(tok.get_vocab()))
        sd = random_state_dict(cfg, seed=3)
        t0 = time.perf_counter()
        _rows, texts = store.plan_chunks(mv, 3, 1)
        rec["host_plan_chunks_s"] = time.perf_counter() - t0
        rec["chunks"] = len(texts)
        del texts
        db_dev, db_host = tmp / "dev.db", tmp / "host.db"
        idx = runtime.acquire(db_dev, 0)
        enc = GpuSentenceEncoder(idx, sd, cfg, DeviceWordPiece(idx, tok, max_length=256), max_seq_length=256)
        enc.encode(["warm up the encoder"] * 64)
        # the device build: SemanticSearch's constructor, its stages in ss.build_timings (device stages end in a
        # synchronise)
        t0 = time.perf_counter()
        ss = SemanticSearch(docs_path=docs, db_path=db_dev, encoder=enc, device_build=True, fallback_build=True)
        rec["device_build_s"] = time.perf_counter() - t0
        rec["device_build_stages_s"] = dict(ss.build_timings)
        rec["host_movies"] = int(enc.tokenizer.host_texts)
        # the fallback build with the same encoder: its constructor is plan_chunks + encode + the shadow write, then
        # the first open's export of the matrix from SQLite, the upload and the sidecar write
        t0 = time.perf_counter()
        host = SemanticSearch(docs_path=docs, db_path=db_host, encoder=enc, fallback_build=True)
        rec["fallback_build_s"] = time.perf_counter() - t0
        got, want = np.asarray(ss._arr.emb), np.asarray(host._arr.emb)
        rec["matrices_bit_identical"] = bool(got.shape == want.shape and got.view(np.uint32).tobytes() ==
                                             want.view(np.uint32).tobytes())
        host.close(); ss.close(); runtime.release(db_dev, 0)
        rec["note"] = ("device_build_stages_s: upload = packing the rows, the host-route check and the copy to HBM; "
                       "chunk = the count and write passes; tokenize = both tokenizer passes; encode = the sentence "
                       "encoder into the matrix; host_route = movies tokenized on the host; device_to_host = the one "
                       "host copy; sqlite_chunks / sqlite_vec0 = the chunks rows and the vec0 writes; attach = serving "
                       "the matrix as the corpus; sidecar = the .rse-emb write.  fallback_build_s = the "
                       "fallback_build=True constructor: host plan_chunks + encode + vec0 shadow write, then the "
                       "first open's export from SQLite, upload and sidecar write.  host_plan_chunks_s = "
                       "store.plan_chunks alone.")
    finally:
        shutil.rmtree(tmp, ignore_errors=True)
    print(json.dumps(rec))
    Path(a.out).write_text(json.dumps(rec, indent=1) + "\n")


if __name__ == "__main__":
    main()
