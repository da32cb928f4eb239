"""CLIP's byte-level BPE on the device (csrc/bpe.cuh) against HuggingFace ``tokenizers`` on the same machine's host
cores, and the ``MultimodalSearch`` constructor end to end with each tokenizer.  Prints one JSON line (and writes it
to --out).

    python scripts/clip_tokenize_bench.py [--docs 600000] [--reps 5] [--out FILE]

Workload: a 49 408-piece CLIP vocab (the size of clip-ViT-B-32's) trained with BpeTrainer (``</w>`` suffix, the
ByteLevel alphabet) on seeded synthetic text (scripts/tokenize_bench.py's pseudo-words with a Zipf frequency and
punctuation), built into ``transformers.CLIPTokenizer``; --docs ``"title: description"`` texts of movie-description
length (2-5 title words, 40-120 description words).  HF runs its batch API (Rust, every host core), truncating at 77
as the CLIP processor does.  Times are host clocks around calls that end in a device synchronise (or return host
lists):
  - tokenize the --docs texts: ``rse_tokenize`` + ``rse_tokens_fetch`` (ids on the host, like the HF call), median
    of --reps, against one HF call (its ids are compared with the device's first);
  - ``MultimodalSearch(documents, model=GpuClipModel(...))`` with ViT-B/32 tower shapes (seeded weights) and the
    tokenizer on the device, then with the HF tokenizer; the two text-embedding matrices are compared bit for bit.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import time
from pathlib import Path

import numpy as np

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
sys.path.insert(0, str(Path(__file__).resolve().parent))

from tokenize_bench import Words, gpu_info, med  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--docs", type=int, default=600000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    import torch
    import transformers
    from tokenizers import Regex, Tokenizer, normalizers, pre_tokenizers
    from tokenizers.models import BPE
    from tokenizers.trainers import BpeTrainer
    from rag_search_engine_b200 import _lib
    from rag_search_engine_b200.bpe import CLIP_PATTERN
    from rag_search_engine_b200.clip import DeviceBPE, GpuClipModel, clip_configs_from_hf
    from rag_search_engine_b200.encoder import _utf8
    from rag_search_engine_b200.multimodal import MultimodalSearch
    res = {"host_cpus": os.cpu_count(), **gpu_info()}
    W = Words(1)
    t = Tokenizer(BPE(unk_token="<|endoftext|>", end_of_word_suffix="</w>", fuse_unk=False))
    t.normalizer = normalizers.Sequence([normalizers.NFC(), normalizers.Replace(Regex(r"\s+"), " "),
                                         normalizers.Lowercase()])
    t.pre_tokenizer = pre_tokenizers.Sequence([
        pre_tokenizers.Split(Regex(CLIP_PATTERN), behavior="removed", invert=True),
        pre_tokenizers.ByteLevel(add_prefix_space=False)])
    t.train_from_iterator(W.texts(60000, 20, 120), BpeTrainer(
        vocab_size=49408, special_tokens=["<|startoftext|>", "<|endoftext|>"], end_of_word_suffix="</w>",
        initial_alphabet=pre_tokenizers.ByteLevel.alphabet()))
    merges = [tuple(m) for m in json.loads(t.to_str())["model"]["merges"]]
    tok = transformers.CLIPTokenizer(vocab=t.get_vocab(), merges=merges)
    res["vocab"] = len(tok.get_vocab())
    res["merges"] = len(merges)
    titles = W.texts(a.docs, 2, 5)
    descs = W.texts(a.docs, 40, 120)
    docs = [{"id": i, "title": x, "description": y} for i, (x, y) in enumerate(zip(titles, descs))]
    texts = [f"{x}: {y}" for x, y in zip(titles, descs)]
    del titles, descs
    res["docs"] = a.docs
    res["text_bytes"] = sum(map(len, texts))

    def hf(x):
        return tok(x, truncation=True, max_length=77)["input_ids"]

    idx = _lib.Index(0)
    tb = time.perf_counter()
    db = DeviceBPE(idx, tok, slot=0, max_length=77)
    res["tables_build_and_load_s"] = round(time.perf_counter() - tb, 2)
    res["host_routed"] = len(db.host_routed(texts))

    def dev():
        return idx.tokenize(0, *_utf8(texts), True, 77)
    t0 = time.perf_counter()
    want = hf(texts)
    t_hf = time.perf_counter() - t0
    ids, cu = dev()
    got = ids.tolist()
    assert [got[x:y] for x, y in zip(cu[:-1].tolist(), cu[1:].tolist())] == want
    res["tokens"] = int(cu[-1])
    r = {"device_s": round(med(dev, a.reps) / 1e3, 3), "hf_s": round(t_hf, 3)}
    r["device_us_per_text"] = round(r["device_s"] / a.docs * 1e6, 3)
    r["hf_us_per_text"] = round(t_hf / a.docs * 1e6, 2)
    r["speedup"] = round(r["hf_s"] / r["device_s"], 1)
    res["tokenize"] = r
    del want, got, ids, cu
    # the MultimodalSearch constructor with ViT-B/32 shapes, each tokenizer
    tc = dict(hidden_size=512, num_hidden_layers=12, num_attention_heads=8, intermediate_size=2048,
              vocab_size=49408, max_position_embeddings=77, eos_token_id=tok.eos_token_id,
              bos_token_id=tok.bos_token_id, pad_token_id=tok.pad_token_id)
    vc = dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072, image_size=224,
              patch_size=32)
    torch.manual_seed(0)
    model = transformers.CLIPModel(transformers.CLIPConfig(text_config=tc, vision_config=vc, projection_dim=512))
    vision, text = clip_configs_from_hf(model.config)
    sd = model.state_dict()
    out = {}
    for name, tk in (("device_bpe", db), ("hf_tokenizer", lambda x: hf(list(x)))):
        gm = GpuClipModel(idx, sd, vision, text, tokenizer=tk)
        gm.encode(texts[:256])                                   # warm-up of every launch shape
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        ms = MultimodalSearch(docs, model=gm)
        torch.cuda.synchronize()
        out[name] = (time.perf_counter() - t0, ms.text_embeddings)
        ms.close()
    assert out["device_bpe"][1].tobytes() == out["hf_tokenizer"][1].tobytes()
    res["multimodal_init"] = {k: round(v[0], 2) for k, v in out.items()}
    res["multimodal_init"]["device_texts_per_s"] = round(a.docs / out["device_bpe"][0])
    res["multimodal_init"]["hf_texts_per_s"] = round(a.docs / out["hf_tokenizer"][0])
    idx.close()
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
