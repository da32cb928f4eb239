"""A host restatement of csrc/wordpiece.cuh over the tables of rag_search_engine_b200.wordpiece, step for step:
added tokens split off the raw text (leftmost, longest), each code point mapped and classified through the tables,
words cut at whitespace and around punctuation, greedy longest match through the two tries, truncation and
[CLS] / [SEP].  Returns None for a text the device refuses (two code points NFD could reorder)."""
from __future__ import annotations

from rag_search_engine_b200.wordpiece import CLASS_OTHER, CLASS_PUNCT, REORDER_BIT


def _child(t, node, cp):
    lo, hi = int(t.node_first[node]), int(t.node_first[node + 1])
    end = hi
    while lo < hi:
        mid = (lo + hi) >> 1
        if t.edge_cp[mid] < cp:
            lo = mid + 1
        else:
            hi = mid
    return int(t.edge_child[lo]) if lo < end and t.edge_cp[lo] == cp else -1


def _word(t, w):
    if len(w) > t.max_input_chars_per_word:
        return [t.unk_id]
    out, start = [], 0
    while start < len(w):
        node, best, bend = (0 if start == 0 else 1), -1, start
        for i in range(start, len(w)):
            node = _child(t, node, w[i])
            if node < 0:
                break
            if t.node_id[node] >= 0:
                best, bend = int(t.node_id[node]), i + 1
        if best < 0:
            return [t.unk_id]
        out.append(best)
        start = bend
    return out


def tokenize(t, text: str, add_special: bool = False, max_length: int | None = None):
    pieces, word, reorder = [], [], 0
    i = 0
    while i < len(text):
        hit = max(((c, tid) for c, tid in t.added if text.startswith(c, i)), key=lambda x: len(x[0]), default=None)
        if hit is not None:
            pieces += _word(t, word) if word else []
            word = []
            pieces.append(hit[1])
            i += len(hit[0])
            continue
        m = int(t.cp_map[ord(text[i])])
        i += 1
        reorder += bool(m & REORDER_BIT)
        n = (m >> 21) & 3
        outs = [m & 0x1FFFFF] if n == 1 else [int(x) for x in t.extra[m & 0x1FFFFF][:n]]
        for o in outs:
            c = int(t.cp_class[o])
            if c == CLASS_OTHER:
                word.append(o)
                continue
            pieces += _word(t, word) if word else []
            word = []
            if c == CLASS_PUNCT:
                pieces += _word(t, [o])
    pieces += _word(t, word) if word else []
    if reorder >= 2:
        return None
    if max_length is not None:
        pieces = pieces[:max_length - (2 if add_special else 0)]
    return [t.cls_id] + pieces + [t.sep_id] if add_special else pieces
