"""The batched cross-encoder rerank (rse_hybrid_rerank_run) on an S-600k-shaped corpus, against the same ranking
composed on the host from the existing calls.  Prints one JSON line (and writes it to --out).

    python scripts/rerank_batch_bench.py [--movies 600000] [--steps 24] [--out FILE]

Workload: the bench's seeded S-600k corpus (isotropic chunk embeddings, synthetic BM25 postings), a document-token
store of one 100-200 token document per movie, a TinyBERT-L2 cross-encoder with seeded random weights (the
arithmetic does not depend on the values), 8 resident batches of 256 queries (8 cross-encoder tokens each) used in
rotation, limit 10, max_length 512.  Times:
  - step: host clock around rse_hybrid_rerank_run + _fetch (which ends in a device synchronise), median of --steps;
  - stages: device events of the same step (rse_set_timing; a separate pass) split into hybrid / assembly /
    encoder / order;
  - host composition: today's calls (BM25 + KNN + RRF over the whole union, fetched) -> numpy gather of the
    document tokens -> GpuCrossEncoder.predict_ids -> the reference's sort in Python, per batch;
  - per query: the same composition for one query at a time (the single-query mirror's shape, without its host
    tokenizer), over --sample queries.
"""
from __future__ import annotations

import argparse
import json
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))

NB, BATCH, LIMIT, QTOK, MAX_LEN = 8, 256, 10, 8, 512


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    name, power = (x.strip() for x in out[0].split(","))
    return {"gpu": name, "power_limit": power}


def host_composition(idx, ce, movie_ids, doc_indptr, doc_tok, Q, tok_indptr, terms, qids):
    """Today's API: every stage fetched to the host, pairs gathered with numpy, the reference's sort."""
    from rag_search_engine_b200._lib import pair_truncate
    L2 = 2 * LIMIT
    score, doc, bc = idx.bm25(tok_indptr, terms, LIMIT)
    dist, _rowid, movie, sc = idx.knn_movies(Q, LIMIT, LIMIT * 10)
    pad = lambda a, fill: np.concatenate([a, np.full((a.shape[0], LIMIT), fill, a.dtype)], 1)  # noqa: E731
    bid = pad(np.where(doc >= 0, movie_ids[np.clip(doc, 0, None)], -1), -1)
    sid = pad(np.where(movie >= 0, movie_ids[np.clip(movie, 0, None)], -1), -1)
    oid, osc, _orb, _ors, oc = idx.fuse_rrf(L2, 60.0, bid, pad(score, 0.0), bc, sid, pad(dist.astype(np.float64), 0.0), sc)
    rows = np.searchsorted(movie_ids, oid)
    ids, tts = [], []
    for q in range(oid.shape[0]):
        qi = qids[q]
        for j in range(int(oc[q])):
            r = int(rows[q, j])
            d = doc_tok[doc_indptr[r]:doc_indptr[r + 1]]
            a, b = pair_truncate(len(qi), len(d), MAX_LEN)
            ids.append(np.concatenate([[ce.cls_id], qi[:a], [ce.sep_id], d[:b], [ce.sep_id]]).astype(np.int32))
            tts.append(np.concatenate([np.zeros(a + 2, np.int32), np.ones(b + 1, np.int32)]))
    ce_scores = ce.predict_ids(ids, tts).tolist() if ids else []
    out, p = [], 0
    for q in range(oid.shape[0]):
        n = int(oc[q])
        hits = [(ce_scores[p + j], float(osc[q, j]), int(oid[q, j])) for j in range(n)]
        p += n
        hits.sort(key=lambda h: (h[0], h[1]), reverse=True)
        out.append([h[2] for h in hits[:LIMIT]])
    return out, len(ids), int(sum(len(x) for x in ids))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--movies", type=int, default=600_000)
    ap.add_argument("--vocab", type=int, default=1_000_000)
    ap.add_argument("--steps", type=int, default=24)
    ap.add_argument("--sample", type=int, default=32)
    ap.add_argument("--out", default="")
    args = ap.parse_args()
    import torch
    from rag_search_engine_b200 import _lib, synth
    from rag_search_engine_b200.encoder import TINYBERT_L2_CONFIG, GpuCrossEncoder, random_state_dict
    if not torch.cuda.is_available():
        raise SystemExit("rerank_batch_bench needs a CUDA device")
    res = {"workload": {"movies": args.movies, "batch": BATCH, "batches": NB, "limit": LIMIT, "query_tokens": QTOK,
                        "max_length": MAX_LEN, "doc_tokens": "100-200 uniform"}}
    res.update(gpu_info())
    se = synth.synth_embeddings(args.movies, seed=1234, device="cuda")
    bm = synth.synth_bm25(args.movies, args.vocab, seed=1234, device="cuda")
    tok_indptr, terms = synth.synth_token_queries(bm, NB * BATCH, seed=99)
    Q = synth.synth_query_vectors(se.emb, NB * BATCH, seed=99).cpu().numpy()
    idx = _lib.Index(0)
    movie_of = se.movie_of_chunk.to(device="cuda", dtype=torch.int32).contiguous()
    idx.attach_embeddings_dev(se.emb.data_ptr(), se.emb.shape[0], se.emb.shape[1], movie_idx_ptr=movie_of.data_ptr(),
                              keepalive=(se.emb, movie_of))
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    movie_ids = np.asarray(se.movie_ids, np.int64)
    idx.set_id_tables(movie_ids, movie_ids)
    rng = np.random.default_rng(7)
    lens = rng.integers(100, 201, args.movies)
    doc_indptr = np.zeros(args.movies + 1, np.int64)
    np.cumsum(lens, out=doc_indptr[1:])
    doc_tok = rng.integers(1000, 30522, int(doc_indptr[-1]), dtype=np.int32)
    t0 = time.time()
    idx.rerank_docs_load(movie_ids, doc_indptr, doc_tok)
    res["store"] = {"docs": args.movies, "tokens": int(doc_indptr[-1]), "bytes": int(4 * doc_indptr[-1] + 16 * args.movies),
                    "load_s": round(time.time() - t0, 2)}
    ce = GpuCrossEncoder(idx, random_state_dict(TINYBERT_L2_CONFIG, seed=5, head=1), TINYBERT_L2_CONFIG, slot=1,
                         max_length=MAX_LEN)
    qids = rng.integers(1000, 30522, (NB * BATCH, QTOK), dtype=np.int32)
    q_ptr = np.arange(0, (BATCH + 1) * QTOK, QTOK, dtype=np.int32)

    batches = []
    for i in range(NB):
        lo, hi = i * BATCH, (i + 1) * BATCH
        tp = (tok_indptr[lo:hi + 1] - tok_indptr[lo]).astype(np.int32)
        tr = np.ascontiguousarray(terms[tok_indptr[lo]:tok_indptr[hi]])
        batches.append((Q[lo:hi], tp, tr, qids[lo:hi]))
        idx.hybrid_stage(Q[lo:hi], tp, tr)
        idx.hybrid_stash(i)

    def step(i):
        idx.hybrid_stash(i)
        idx.hybrid_rerank_run(ce.slot, 60.0, LIMIT, q_ptr, batches[i][3].ravel(), cls_id=ce.cls_id, sep_id=ce.sep_id,
                              max_length=MAX_LEN, activation=0)
        out = idx.hybrid_rerank_fetch(LIMIT)
        idx.hybrid_stash(i)
        return out

    for i in range(NB):                                  # warm-up: every batch once
        step(i)
    times = []
    for s in range(args.steps):
        t = time.perf_counter()
        step(s % NB)
        times.append(1e3 * (time.perf_counter() - t))
    idx.set_timing(True)
    stages = []
    for s in range(NB):
        step(s)
        stages.append(idx.hybrid_rerank_timing())
    idx.set_timing(False)

    # the host composition on the same batches (exact pair / token counts come from it), and its agreement
    host_ms, pairs, tokens, agree = [], [], [], True
    for i in range(NB):
        Qb, tp, tr, qi = batches[i]
        t = time.perf_counter()
        ranked, npairs, ntok = host_composition(idx, ce, movie_ids, doc_indptr, doc_tok, Qb, tp, tr, list(qi))
        host_ms.append(1e3 * (time.perf_counter() - t))
        pairs.append(npairs); tokens.append(ntok)
        dev = step(i)
        agree &= all(ranked[q] == dev[0][q, :dev[6][q]].tolist() for q in range(BATCH))
    per_query = []
    Qb, tp, tr, qi = batches[0]
    for q in range(args.sample):
        t = time.perf_counter()
        host_composition(idx, ce, movie_ids, doc_indptr, doc_tok, Qb[q:q + 1],
                         (tp[q:q + 2] - tp[q]).astype(np.int32), tr[tp[q]:tp[q + 1]], [qi[q]])
        per_query.append(1e3 * (time.perf_counter() - t))

    step_ms = statistics.median(times)
    st = np.median(np.array(stages), axis=0).tolist()
    mean_pairs, mean_tok = float(np.mean(pairs)), float(np.mean(tokens))
    res.update({
        "step_ms_median": round(step_ms, 3), "step_ms_min": round(min(times), 3), "step_ms_max": round(max(times), 3),
        "stages_ms": {k: round(v, 3) for k, v in zip(("hybrid", "assembly", "encoder", "order"), st)},
        "pairs_per_step": mean_pairs, "tokens_per_step": mean_tok,
        "queries_per_s": round(BATCH / step_ms * 1e3, 1), "pairs_per_s": round(mean_pairs / step_ms * 1e3, 1),
        "tokens_per_s": round(mean_tok / step_ms * 1e3, 1),
        "host_composition_ms_per_batch_median": round(statistics.median(host_ms), 2),
        "host_composition_queries_per_s": round(BATCH / statistics.median(host_ms) * 1e3, 1),
        "per_query_ms_median": round(statistics.median(per_query), 3),
        "per_query_queries_per_s": round(1e3 / statistics.median(per_query), 1),
        "host_composition_ranks_equal": bool(agree),
    })
    line = json.dumps(res)
    print(line)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(line + "\n")
    idx.close()


if __name__ == "__main__":
    main()
