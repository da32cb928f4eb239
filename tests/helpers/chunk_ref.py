"""A byte-level restatement of csrc/chunk.cuh: the sentence chunking of a semantic index build over UTF-8 bytes and
offsets, walked the way the kernel walks them (strip, whitespace runs after '.', '!' or '?', windows by index
arithmetic, chunk texts joined without a separator).  tests/test_chunk_ref.py holds it to store.plan_chunks."""
from __future__ import annotations

from typing import List, Tuple

# Python's whitespace (str.isspace / str.strip / re's \s): 29 code points
WHITESPACE = frozenset([*range(0x09, 0x0E), *range(0x1C, 0x21), 0x85, 0xA0, 0x1680, *range(0x2000, 0x200B), 0x2028,
                        0x2029, 0x202F, 0x205F, 0x3000])
PUNCT = frozenset(b".!?")


def _cp(t: bytes, p: int, e: int) -> Tuple[int, int]:
    """(code point, length) at p < e; a sequence cut by e reads as its lead byte."""
    b = t[p]
    need = 1 if b < 0x80 else 2 if b < 0xE0 else 3 if b < 0xF0 else 4
    if b < 0x80 or p + need > e:
        return b, 1
    if need == 2:
        return (b & 0x1F) << 6 | (t[p + 1] & 0x3F), 2
    if need == 3:
        return (b & 0x0F) << 12 | (t[p + 1] & 0x3F) << 6 | (t[p + 2] & 0x3F), 3
    return (b & 0x07) << 18 | (t[p + 1] & 0x3F) << 12 | (t[p + 2] & 0x3F) << 6 | (t[p + 3] & 0x3F), 4


def strip(t: bytes, a: int, b: int) -> Tuple[int, int]:
    while a < b:
        c, n = _cp(t, a, b)
        if c not in WHITESPACE:
            break
        a += n
    while b > a:
        q = b - 1
        while q > a and (t[q] & 0xC0) == 0x80:
            q -= 1
        if _cp(t, q, b)[0] not in WHITESPACE:
            break
        b = q
    return a, b


def sentences(t: bytes, s: int, e: int) -> List[Tuple[int, int]]:
    """Byte ranges of the sentences of the stripped description [s, e): [(s, s)] when it is empty."""
    if s == e:
        return [(s, s)]
    out = []
    p, prev, start = s, 0, s
    while p < e:
        c, n = _cp(t, p, e)
        if c in WHITESPACE and prev in PUNCT:
            out.append((start, p))
            while p < e and _cp(t, p, e)[0] in WHITESPACE:
                p += _cp(t, p, e)[1]
            start, prev = p, 0
            continue
        prev = c
        p += n
    out.append((start, e))
    return out


def windows(n: int, size: int, overlap: int) -> List[Tuple[int, int]]:
    carry = overlap if 0 < overlap < size else 0
    fresh = size - carry
    n_win = 1 + (n - size + fresh - 1) // fresh if n > size else 1
    return [(0, min(size, n))] + [(size + (w - 1) * fresh - carry, min(size + w * fresh, n)) for w in range(1, n_win)]


def chunk_movies(text: bytes, offsets, size: int, overlap: int):
    """Movie m = title text[offsets[2m]:offsets[2m+1]], description text[offsets[2m+1]:offsets[2m+2]] ->
    (chunk texts as bytes, their movie rows, their chunk indexes)."""
    if size < 1:
        raise ValueError("max_chunk_size must be >= 1")
    texts, movie, index = [], [], []
    for m in range((len(offsets) - 1) // 2):
        t0, t1, d1 = int(offsets[2 * m]), int(offsets[2 * m + 1]), int(offsets[2 * m + 2])
        texts.append(text[t0:t1]); movie.append(m); index.append(0)
        sent = sentences(text, *strip(text, t1, d1))
        for w, (a, b) in enumerate(windows(len(sent), size, overlap), start=1):
            texts.append(b"".join(text[x:y] for x, y in sent[a:b])); movie.append(m); index.append(w)
    return texts, movie, index


NEAR_MISSES = ("​", "᠎", "﻿")
SIZES = ((3, 1), (1, 0), (2, 5), (4, 3), (3, 0), (3, -1))


def adversarial_movies(seed: int, n: int):
    """(id, title, description) rows that exercise every rule: each whitespace code point and the near misses,
    punctuation runs with whitespace runs between them, leading / trailing whitespace, empty and whitespace-only
    descriptions, untrimmed titles, multi-byte UTF-8 and long descriptions."""
    import random
    rnd = random.Random(seed)
    ws = [chr(c) for c in sorted(WHITESPACE)]
    words = ["alpha", "Beta", "γάμμα", "δ", "日本語", "naïve", "🎬", "x", "é", "Zoë", "", "ok"]
    punct = [".", "!", "?", "?!.", "..", "!?", ",", ";", "...", ".!"]

    def gap():
        r = rnd.random()
        if r < 0.5:
            return " "
        if r < 0.8:
            return "".join(rnd.choice(ws) for _ in range(rnd.randint(1, 3)))
        return rnd.choice(NEAR_MISSES) + rnd.choice(["", " "])

    movies = []
    for i in range(n):
        kind = rnd.random()
        if kind < 0.04:
            desc = ""
        elif kind < 0.08:
            desc = "".join(rnd.choice(ws) for _ in range(rnd.randint(1, 5)))
        else:
            n_sent = rnd.randint(1, 300 if kind > 0.97 else 12)
            parts = []
            for _ in range(n_sent):
                sent = gap().join(rnd.choice(words) for _ in range(rnd.randint(1, 6)))
                parts.append(sent + rnd.choice(punct) if rnd.random() < 0.85 else sent)
                parts.append(gap())
            desc = "".join(parts)
            if rnd.random() < 0.3:
                desc = "".join(rnd.choice(ws) for _ in range(rnd.randint(1, 3))) + desc
        title = rnd.choice(["", " ", "  Padded Title ", "Title. Two!", "日本 ", "　T "]) + rnd.choice(words)
        movies.append((i * 3 + 1, title, desc))
    return movies
