"""A host restatement of csrc/bpe.cuh over the tables of rag_search_engine_b200.bpe, step for step: special tokens
split off the raw text (leftmost, longest), each code point mapped and classified through the tables, pieces cut by
the CLIP pattern's leftmost-first alternation (the two literals, the contractions, a letter run, one number, a run of
anything else), a literal piece cut again into "<|", word, "|>" as ByteLevel's pattern does, each piece's bytes mapped
to their initial symbols (``</w>`` on the last), then merged: the adjacent pair of lowest rank, leftmost on a tie,
until no pair has a merge.  Truncation stops the text at the cap; bos / eos around it.  Returns None for a text the
device refuses (a route code point, or a piece that has to be merged and is longer than the device's word buffer)."""
from __future__ import annotations

from rag_search_engine_b200.bpe import (CLASS_LETTER, CLASS_NUMBER, CLASS_OTHER, CLASS_SPACE, MAX_WORD_BYTES,
                                        ROUTE_BIT, hash_pair)

CONTRACTIONS = ("s", "t", "re", "ve", "m", "ll", "d")
LITERAL_WORDS = (("<|startoftext|>", ("<|", "startoftext", "|>")), ("<|endoftext|>", ("<|", "endoftext", "|>")))
INF = 1 << 62


class Refused(Exception):
    pass


def merge_lookup(t, a: int, b: int):
    mask = t.merges.shape[0] - 1
    s = int(hash_pair(a, b, mask))
    while True:
        left, right, rank, new = (int(x) for x in t.merges[s])
        if left == a and right == b:
            return rank, new
        if left < 0:
            return INF, -1
        s = (s + 1) & mask


def merge_word(t, data: bytes):
    """The ids of one piece: initial symbols, then the lowest-rank adjacent pair merged first, leftmost on ties."""
    if len(data) > MAX_WORD_BYTES:
        raise Refused
    sym = [int(t.byte_ids[b]) for b in data[:-1]] + [int(t.byte_ids[256 + data[-1]])]
    rk = [merge_lookup(t, sym[i], sym[i + 1])[0] for i in range(len(sym) - 1)]
    while rk:
        best = min(rk)
        if best == INF:
            break
        i = rk.index(best)                                   # leftmost on a tie
        sym[i] = merge_lookup(t, sym[i], sym[i + 1])[1]
        del sym[i + 1]
        del rk[i]
        if i > 0:
            rk[i - 1] = merge_lookup(t, sym[i - 1], sym[i])[0]
        if i < len(rk):
            rk[i] = merge_lookup(t, sym[i], sym[i + 1])[0]
    return sym


def _normalized(t, seg: str):
    out = []
    for ch in seg:
        m = int(t.cp_map[ord(ch)])
        if m & ROUTE_BIT:
            raise Refused
        n = (m >> 21) & 3
        out += [chr(m & 0x1FFFFF)] if n == 1 else [chr(int(x)) for x in t.extra[m & 0x1FFFFF][:n]]
    return "".join(out)


def pieces(t, seg: str):
    """The pieces (strings) of one normalized segment, in order."""
    cls = lambda c: int(t.cp_class[ord(c)])            # noqa: E731
    i, out = 0, []
    while i < len(seg):
        c = seg[i]
        k = cls(c)
        if k == CLASS_SPACE:
            i += 1
            continue
        if k == CLASS_LETTER:
            j = i
            while j < len(seg) and cls(seg[j]) == CLASS_LETTER:
                j += 1
            out.append(seg[i:j]); i = j
            continue
        if k == CLASS_NUMBER:
            out.append(c); i += 1
            continue
        lit = next((w for s, w in LITERAL_WORDS if seg.startswith(s, i)), None) if c == "<" else None
        if lit is not None:
            out += lit
            i += sum(map(len, lit))
            continue
        con = next((x for x in CONTRACTIONS if seg.startswith(x, i + 1)), None) if c == "'" else None
        if con is not None:
            out.append("'" + con); i += 1 + len(con)
            continue
        j = i
        while j < len(seg) and cls(seg[j]) == CLASS_OTHER:
            j += 1
        out.append(seg[i:j]); i = j
    return out


def tokenize(t, text: str, add_special: bool = False, max_length: int | None = None):
    cap = INF if max_length is None else max_length - (2 if add_special else 0)
    if any(ord(c) < 0x110000 and int(t.cp_map[ord(c)]) & ROUTE_BIT for c in text):
        return None
    ids, i, seg = [], 0, []
    try:
        def flush():
            for p in pieces(t, _normalized(t, "".join(seg))):
                if len(ids) >= cap:
                    return
                ids.extend(merge_word(t, p.encode("utf-8")))
            seg.clear()
        while i < len(text):
            hit = max(((c, tid) for c, tid in t.added if text.startswith(c, i)), key=lambda x: len(x[0]), default=None)
            if hit is None:
                seg.append(text[i]); i += 1
                continue
            flush()
            ids.append(hit[1])
            i += len(hit[0])
        flush()
    except Refused:
        return None
    ids = ids[:cap] if cap < INF else ids
    return [t.bos_id] + ids + [t.eos_id] if add_special else ids
