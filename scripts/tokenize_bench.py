"""BERT WordPiece on the device (csrc/wordpiece.cuh) against HuggingFace ``tokenizers`` on the same machine's host
cores.  Prints one JSON line (and writes it to --out).

    python scripts/tokenize_bench.py [--docs 600000] [--reps 20] [--out FILE]

Workload: a 30 522-piece uncased WordPiece vocab trained with WordPieceTrainer on seeded synthetic text (pseudo-words
with a Zipf frequency, punctuation, a few accented words); queries of 3-12 words, index chunks of ~120 words,
documents of 80-150 words.  HF runs its batch API (``BertTokenizerFast.__call__``, Rust, every host core).  Times are
host clocks around calls that end in a device synchronise (or return host lists), median of --reps:
  - 256 queries and 2048 chunks: ``rse_tokenize`` + ``rse_tokens_fetch`` (ids on the host, like the HF call) and
    HF; for the chunks also the bulk embedding (MiniLM-L6 shapes, seeded weights) from texts on the device against
    HF ids + ``encode_ids``;
  - the rerank store of --docs documents: ``rse_rerank_docs_load_texts`` against HF + ``rse_rerank_docs_load``,
    once each (texts -> UTF-8 included on both sides); the two stores are compared through ``rse_tokenize``;
  - ``rrf_search_texts`` for 256 query strings against the same call with ids prepared in advance (S-20k corpus).
Every device result is compared with HF's before it is timed.
"""
from __future__ import annotations

import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))


def gpu_info() -> dict:
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                         text=True).stdout.strip().splitlines()
    name, power = (x.strip() for x in out[0].split(","))
    return {"gpu": name, "power_limit": power}


class Words:
    """Seeded synthetic text: pseudo-words with a Zipf frequency; a word is capitalised at 5 %, followed by
    punctuation at 8 %, and a text starts with a capital."""

    def __init__(self, seed):
        rng = random.Random(seed)
        syl = [a + b for a in "bcdfghjklmnprstvwz" for b in "aeiou"] + ["th", "qu", "ch", "é", "ö"]
        words = ["".join(rng.choice(syl) for _ in range(rng.choice((1, 2, 2, 3, 3, 4)))) for _ in range(60000)]
        self.nw = len(words)
        # variants: plain | capitalised | followed by one of five punctuation marks
        self.table = np.asarray(words + [w.capitalize() for w in words] +
                                [w + p for p in (",", ".", ";", "'s", "-") for w in words], dtype=object)
        w = 1.0 / np.arange(1, self.nw + 1) ** 1.05
        self.cdf = np.cumsum(w / w.sum())
        self.rng = np.random.default_rng(seed)

    def texts(self, n, lo, hi):
        lens = self.rng.integers(lo, hi + 1, n)
        cu = np.zeros(n + 1, np.int64)
        np.cumsum(lens, out=cu[1:])
        N = int(cu[-1])
        idx = np.minimum(np.searchsorted(self.cdf, self.rng.random(N)), self.nw - 1)
        u = self.rng.random(N)
        var = np.where(u < 0.08, 2 + self.rng.integers(0, 5, N), np.where(u < 0.13, 1, 0))
        var[cu[:-1]] = np.where(var[cu[:-1]] == 0, 1, var[cu[:-1]])
        words = self.table[idx + self.nw * var]
        return [" ".join(words[a:b].tolist()) for a, b in zip(cu[:-1].tolist(), cu[1:].tolist())]


def med(f, reps):
    ts = []
    for _ in range(reps):
        t = time.perf_counter()
        f()
        ts.append(time.perf_counter() - t)
    return statistics.median(ts) * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs", type=int, default=600000)
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import transformers
    from tokenizers import Tokenizer, normalizers, pre_tokenizers
    from tokenizers.models import WordPiece
    from tokenizers.trainers import WordPieceTrainer
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.encoder import (MINILM_L6_CONFIG, DeviceWordPiece, GpuSentenceEncoder, _utf8,
                                                random_state_dict)
    res = {"host_cpus": os.cpu_count(), **gpu_info()}
    W = Words(1)
    t = Tokenizer(WordPiece(unk_token="[UNK]"))
    t.normalizer = normalizers.BertNormalizer()
    t.pre_tokenizer = pre_tokenizers.BertPreTokenizer()
    t.train_from_iterator(W.texts(30000, 20, 120), WordPieceTrainer(vocab_size=30522, special_tokens=[
        "[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"]))
    tok = transformers.BertTokenizerFast(vocab=t.get_vocab())
    res["vocab"] = len(tok.get_vocab())
    idx = _lib.Index(0)
    tb = time.perf_counter()
    dw = DeviceWordPiece(idx, tok, slot=0, max_length=256)
    res["tables_build_and_load_s"] = round(time.perf_counter() - tb, 2)
    R = a.reps

    def hf(texts, special=True, ml=256):
        return tok(texts, add_special_tokens=special, truncation=ml is not None, max_length=ml)["input_ids"]

    def dev(texts, special=True, ml=256):
        return idx.tokenize(0, *_utf8(texts), special, ml or 0)

    for name, texts in (("queries_256", W.texts(256, 3, 12)), ("chunks_2048", W.texts(2048, 100, 140))):
        want = hf(texts)
        ids, cu = dev(texts)
        assert [ids[x:y].tolist() for x, y in zip(cu[:-1], cu[1:])] == want, name
        hf(texts); dev(texts)
        r = {"tokens": int(cu[-1]), "device_ms": round(med(lambda: dev(texts), R), 3),
             "hf_ms": round(med(lambda: hf(texts), R), 3)}
        r["speedup"] = round(r["hf_ms"] / r["device_ms"], 1)
        res[name] = r
    # bulk embedding of the chunks: text in on the device vs HF ids + encode_ids
    cfg = MINILM_L6_CONFIG
    enc = GpuSentenceEncoder(idx, random_state_dict(cfg, seed=3), cfg, dw, slot=0, max_seq_length=256)
    chunks = W.texts(2048, 100, 140)
    v_dev = enc.encode(chunks)
    v_host = enc.encode_ids(hf(chunks))
    assert v_dev.tobytes() == v_host.tobytes()
    res["embed_chunks_2048"] = {"device_text_in_ms": round(med(lambda: enc.encode(chunks), max(3, R // 4)), 2),
                                "hf_ids_then_encode_ms": round(med(lambda: enc.encode_ids(hf(chunks)), max(3, R // 4)), 2)}
    e = res["embed_chunks_2048"]
    e["device_chunks_per_s"] = round(2048 / e["device_text_in_ms"] * 1e3)
    e["hf_chunks_per_s"] = round(2048 / e["hf_ids_then_encode_ms"] * 1e3)
    # the rerank store
    docs = W.texts(a.docs, 80, 150)
    ids = np.arange(1, a.docs + 1, dtype=np.int64) * 3
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    data, offs = _utf8(docs)
    idx.rerank_docs_load_texts(0, ids, data, offs)
    t_dev = time.perf_counter() - t0
    t0 = time.perf_counter()
    lists = hf(docs, special=False, ml=None)
    t_tok = time.perf_counter() - t0
    lens = np.fromiter(map(len, lists), np.int64, count=len(lists))
    indptr = np.zeros(len(lists) + 1, np.int64)
    np.cumsum(lens, out=indptr[1:])
    import itertools
    flat = np.fromiter(itertools.chain.from_iterable(lists), np.int32, count=int(indptr[-1]))
    idx.rerank_docs_load(ids, indptr, flat)
    t_host = time.perf_counter() - t0
    d_ids, d_cu = dev(docs, special=False, ml=None)
    assert np.array_equal(d_cu.astype(np.int64), indptr) and np.array_equal(d_ids, flat)
    res["store"] = {"docs": a.docs, "text_bytes": len(data), "tokens": int(indptr[-1]),
                    "device_load_s": round(t_dev, 3), "hf_tokenize_s": round(t_tok, 3),
                    "hf_tokenize_and_load_s": round(t_host, 3), "speedup": round(t_host / t_dev, 1)}
    del docs, lists, flat, data
    # rrf_search_texts from strings vs prepared ids
    from rag_search_engine_b200 import HybridSearch, synth
    se = synth.synth_embeddings(20000, seed=5, device="cpu")
    bm = synth.synth_bm25(20000, 5000, seed=5, mean_len=30, sd_len=10)
    idx.load_embeddings(se.emb.numpy(), movie_idx=se.movie_of_chunk.numpy())
    idx.load_bm25(bm.indptr, bm.doc_idx, bm.tf, bm.df, bm.dl, bm.n_movies, bm.avgdl)
    T = len(bm.df)
    names = [f"t{i}" for i in range(T)]
    hs = HybridSearch.from_loaded(idx, dict(zip(names, range(T))), se.movie_ids, se.movie_ids,
                                  registry_key="tokenize-bench")
    tp, terms = synth.synth_token_queries(bm, 256, seed=7)
    toks = [[names[x] for x in terms[tp[i]:tp[i + 1]] if x >= 0] for i in range(256)]
    qs = W.texts(256, 3, 12)
    qids = hf(qs)
    r_ids = hs.rrf_search_texts(toks, qids, enc, as_arrays=True)
    r_txt = hs.rrf_search_texts(toks, qs, enc, as_arrays=True)
    assert all((x.view(np.uint8) == y.view(np.uint8)).all() for x, y in zip(r_ids, r_txt))
    res["rrf_search_texts_256"] = {
        "from_strings_ms": round(med(lambda: hs.rrf_search_texts(toks, qs, enc, as_arrays=True), R), 3),
        "from_prepared_ids_ms": round(med(lambda: hs.rrf_search_texts(toks, qids, enc, as_arrays=True), R), 3),
        "hf_tokenize_then_ids_ms": round(med(lambda: hs.rrf_search_texts(toks, hf(qs), enc, as_arrays=True), R), 3)}
    hs.close()
    idx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
