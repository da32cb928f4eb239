"""The chunk embeddings of a semantic index build, on the device (``SemanticSearch(..., device_build=True)``).

The reference's build (semantic_search.py:164-206) reads ``movies ORDER BY id``, splits every description into
sentence windows (``store.plan_chunks``), embeds every chunk text with ``model.encode`` and inserts the vectors into
vec0.  Here the movie rows go up once as one UTF-8 buffer; csrc/chunk.cuh cuts the chunk texts into HBM, the
WordPiece kernels tokenize them where they are and the sentence encoder writes each chunk's vector at its chunk id
into one ``[n_chunks, hidden]`` fp32 matrix in HBM, which the caller then serves as the handle's corpus.

The movies go through in parts of at most ``part_bytes`` bytes of chunk text (the chunk CSR, its ids and the
tokenizer's buffers of one part are what the build holds besides the matrix).  A movie whose title or description
holds a text the device tokenizer refuses (``DeviceWordPiece.host_routed``: two code points whose combining marks NFD
could reorder) is chunked and tokenized on the host (``store.plan_chunks``, the host tokenizer) and its chunks are
encoded from those ids into their rows; such movies are counted in the tokenizer's ``host_texts``.  No row depends on
the part or the slice it was encoded in, so the matrix is ``encoder.encode(texts)`` of ``plan_chunks``' texts bit for
bit.
"""
from __future__ import annotations

import time
from dataclasses import dataclass, field
from typing import Dict, List, Sequence

import numpy as np

from . import store
from .encoder import DeviceWordPiece, GpuSentenceEncoder, pack

PART_BYTES = 1 << 30                 # chunk text of one part: ~1 GB of CSR + ~1 GB of ids + the tokenizer's scratch
TOKENS_PER_CALL = 1 << 16            # GpuSentenceEncoder.encode's slice (the encoder's scratch is ~10 KB a token)
# ids of one tokenize call stay below 2^31: a text has at most one id per byte plus [CLS] / [SEP]
_MAX_PART_IDS = (1 << 31) - 1


@dataclass
class DeviceChunks:
    """Every chunk of a movie list as the device cut it, on the host (what ``chunk_movies`` returns)."""
    text: bytes                      # chunk texts back to back (UTF-8)
    offsets: np.ndarray              # int64 [n_chunks + 1]
    movie: np.ndarray                # int32 [n_chunks] row of the chunk's movie in the list
    chunk_index: np.ndarray          # int32 [n_chunks]


@dataclass
class DeviceBuild:
    emb: "object"                    # torch float32 [n_chunks, hidden] on the device
    chunks_per_movie: np.ndarray     # int64 [n_movies]
    movie_idx: np.ndarray            # int32 [n_chunks] row of the chunk's movie
    host_movies: int                 # movies chunked and tokenized on the host
    timings: Dict[str, float] = field(default_factory=dict)   # seconds per stage (device stages end in a synchronise)


def _check_size(max_chunk_size: int) -> None:
    if int(max_chunk_size) < 1:                     # window_chunks never terminates there
        raise ValueError(f"max_chunk_size must be >= 1 (got {max_chunk_size})")


def pack_movies(movies: Sequence[tuple]):
    """(id, title, description) rows -> (UTF-8 bytes, int64 offsets [2n + 1]): title m, then description m."""
    parts = []
    for _, title, desc in movies:
        parts.append(title.encode("utf-8"))
        parts.append(desc.encode("utf-8"))
    offs = np.zeros(len(parts) + 1, np.int64)
    np.cumsum(np.fromiter(map(len, parts), np.int64, count=len(parts)), out=offs[1:])
    return b"".join(parts), offs


def _upload(torch, data: bytes, offs: np.ndarray, dev):
    text = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8).to(dev)
    return text, torch.from_numpy(offs).to(dev)


def _count(index, text, n_bytes: int, offs_dev, m0: int, m1: int, size: int, overlap: int, torch, dev):
    chunk_cu = torch.empty(m1 - m0 + 1, dtype=torch.int64, device=dev)
    byte_cu = torch.empty(m1 - m0 + 1, dtype=torch.int64, device=dev)
    torch.cuda.synchronize(dev)
    nc, nb = index.chunk_count(text.data_ptr(), n_bytes, offs_dev.data_ptr() + 16 * m0, m1 - m0, size, overlap,
                               chunk_cu.data_ptr(), byte_cu.data_ptr())
    return chunk_cu, byte_cu, nc, nb


def _write(index, text, n_bytes: int, offs_dev, m0: int, m1: int, size: int, overlap: int, torch, dev):
    """Movies [m0, m1) -> their chunk CSR on the device: (text uint8, offsets int64, movie int32, index int32)."""
    chunk_cu, byte_cu, nc, nb = _count(index, text, n_bytes, offs_dev, m0, m1, size, overlap, torch, dev)
    out = torch.empty(max(nb, 1), dtype=torch.uint8, device=dev)
    o_offs = torch.empty(nc + 1, dtype=torch.int64, device=dev)
    o_movie = torch.empty(nc, dtype=torch.int32, device=dev)
    o_index = torch.empty(nc, dtype=torch.int32, device=dev)
    torch.cuda.synchronize(dev)
    index.chunk_write(text.data_ptr(), n_bytes, offs_dev.data_ptr() + 16 * m0, m1 - m0, size, overlap,
                      chunk_cu.data_ptr(), byte_cu.data_ptr(), m0, out.data_ptr(), o_offs.data_ptr(),
                      o_movie.data_ptr(), o_index.data_ptr())
    index.synchronize()                             # the write pass reads chunk_cu / byte_cu, freed on return
    return out, o_offs, o_movie, o_index, nb


def chunk_movies(index, movies: Sequence[tuple], max_chunk_size: int, overlap: int) -> DeviceChunks:
    """The chunk texts and (movie, chunk_index) of ``movies`` as the device cuts them, fetched to the host: the
    same texts and order as ``store.plan_chunks(movies, max_chunk_size, overlap)``."""
    import torch
    _check_size(max_chunk_size)
    dev = torch.device("cuda", index.device)
    data, offs = pack_movies(movies)
    text, offs_dev = _upload(torch, data, offs, dev)
    out, o_offs, o_movie, o_index, nb = _write(index, text, len(data), offs_dev, 0, len(movies), max_chunk_size,
                                               overlap, torch, dev)
    return DeviceChunks(text=out[:nb].cpu().numpy().tobytes(), offsets=o_offs.cpu().numpy(),
                        movie=o_movie.cpu().numpy(), chunk_index=o_index.cpu().numpy())


def _parts(routed: np.ndarray, byte_cu: np.ndarray, chunk_cu: np.ndarray, part_bytes: int) -> List[tuple]:
    """Runs of consecutive device-tokenized movies, each of at most part_bytes bytes of chunk text (a bigger movie
    alone) and fewer than 2^31 ids; routed movies are left out."""
    n = len(routed)
    out = []
    m = 0
    while m < n:
        if routed[m]:
            m += 1
            continue
        hi = m + 1
        while (hi < n and not routed[hi] and byte_cu[hi + 1] - byte_cu[m] <= part_bytes
               and (byte_cu[hi + 1] - byte_cu[m]) + 2 * (chunk_cu[hi + 1] - chunk_cu[m]) <= _MAX_PART_IDS):
            hi += 1
        out.append((m, hi))
        m = hi
    return out


def build_embeddings(encoder: GpuSentenceEncoder, movies: Sequence[tuple], max_chunk_size: int, overlap: int, *,
                     part_bytes: int = PART_BYTES, max_tokens_per_call: int = TOKENS_PER_CALL) -> DeviceBuild:
    """``encoder.encode(plan_chunks(movies, ...) texts)`` as a device matrix, built without host strings.
    ``movies`` = (id, title, description) rows in ``ORDER BY id`` order."""
    import torch
    _check_size(max_chunk_size)
    tok = encoder.tokenizer
    if not isinstance(tok, DeviceWordPiece):
        raise TypeError("the device build tokenizes on the device: the encoder needs a DeviceWordPiece tokenizer")
    index = encoder.index
    if tok.index is not index:
        raise ValueError("the encoder's DeviceWordPiece lives on another handle")
    dev = torch.device("cuda", index.device)
    hidden = int(encoder.config["hidden"])
    if not movies:                                  # an empty index, as plan_chunks + encode give for no movies
        return DeviceBuild(emb=torch.empty((0, hidden), dtype=torch.float32, device=dev),
                           chunks_per_movie=np.zeros(0, np.int64), movie_idx=np.zeros(0, np.int32), host_movies=0)
    msl = encoder.max_seq_length
    t = {}

    t0 = time.perf_counter()
    data, offs = pack_movies(movies)
    routed = np.fromiter((tok.tables.needs_host(ti) or tok.tables.needs_host(de) for _, ti, de in movies), bool,
                         count=len(movies))
    text, offs_dev = _upload(torch, data, offs, dev)
    torch.cuda.synchronize(dev)
    t["upload"] = time.perf_counter() - t0

    # every movie's chunk count (the chunk ids, the matrix's size) and chunk bytes (the parts)
    t0 = time.perf_counter()
    chunk_cu_d, byte_cu_d, n_chunks, _ = _count(index, text, len(data), offs_dev, 0, len(movies), max_chunk_size,
                                                overlap, torch, dev)
    chunk_cu = chunk_cu_d.cpu().numpy()
    byte_cu = byte_cu_d.cpu().numpy()
    del chunk_cu_d, byte_cu_d
    t["chunk"] = time.perf_counter() - t0
    per_movie = np.diff(chunk_cu)
    emb = torch.empty((max(n_chunks, 1), hidden), dtype=torch.float32, device=dev)[:n_chunks]
    torch.cuda.synchronize(dev)

    t["tokenize"] = t["encode"] = 0.0
    for m0, m1 in _parts(routed, byte_cu, chunk_cu, int(part_bytes)):
        ts = time.perf_counter()
        out, o_offs, _o_movie, _o_index, nb = _write(index, text, len(data), offs_dev, m0, m1, max_chunk_size,
                                                     overlap, torch, dev)
        n = int(chunk_cu[m1] - chunk_cu[m0])
        t["chunk"] += time.perf_counter() - ts
        ts = time.perf_counter()
        index.tokenize_device_texts(tok.slot, out.data_ptr(), nb, o_offs.data_ptr(), n, True, msl)
        index.synchronize()                         # the write pass of the tokenizer is part of this stage
        t["tokenize"] += time.perf_counter() - ts
        ts = time.perf_counter()
        index.encode_tokens_dev(encoder.slot, max_tokens_per_call,
                                emb.data_ptr() + 4 * hidden * int(chunk_cu[m0]))
        index.synchronize()
        t["encode"] += time.perf_counter() - ts
        del out, o_offs, _o_movie, _o_index

    # the movies the device tokenizer would refuse: host chunking, host ids, encoded into their rows
    ts = time.perf_counter()
    host_movies = np.nonzero(routed)[0]
    for m in host_movies.tolist():
        _, texts = store.plan_chunks([movies[m]], max_chunk_size, overlap)
        ids = [x[:msl] for x in tok.host_ids(texts, True, msl)]
        flat, _, cu = pack(ids)
        index.encode_dev(encoder.slot, flat, cu, emb.data_ptr() + 4 * hidden * int(chunk_cu[m]))
    index.synchronize()
    t["host_route"] = time.perf_counter() - ts
    movie_idx = np.repeat(np.arange(len(movies), dtype=np.int32), per_movie)
    return DeviceBuild(emb=emb, chunks_per_movie=per_movie.astype(np.int64), movie_idx=movie_idx,
                       host_movies=int(len(host_movies)), timings=t)
