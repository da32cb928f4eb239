"""Seeded texts and CLIP BPE tokenizers for the byte-level BPE tests: a vocab trained offline with BpeTrainer
(``end_of_word_suffix="</w>"``, the ByteLevel alphabet) and a tiny hand-made vocab whose missing ``x</w>`` symbols
fall back to the unk token.  The texts mix English words and "title: description" lines with contractions (any
case), digit runs, literal and lowercased special tokens, İ, U+3000, NBSP, tabs and newlines, accented and combining
text, CJK, emoji, random code points from every plane, words longer than the device's word buffer, empty strings
and texts far past 77 ids."""
from __future__ import annotations

import functools
import random

SPECIALS = ["<|startoftext|>", "<|endoftext|>"]
WORDS = ("the movie a of and to in is that it for with as was on be by his at an are from this film story love life "
         "young man woman world family two new war friends time city finds must home school detective haunted "
         "spaceship unbelievable reconstruction").split()
PIECES = [
    "don't", "DON'T", "it's", "IT'S", "we're", "they've", "I'm", "you'll", "he'd", "'s", "'''s", "'re'", "rock'n'roll",
    "o'clock", "'", "''", "'S", "'LL",
    "1999", "2024-01-05", "3.14159", "007", "1,000,000", "٣٤", "²", "½", "Ⅻ", "①",
    "<|startoftext|>", "<|endoftext|>", "<|ENDOFTEXT|>", "<|StartOfText|>", "x<|endoftext|>y", "!<|endoftext|>!",
    "<|endoftext|>!", "<|endoftext", "<||>", "<|", "|>", "<<|endoftext|>>", "<|endoftext|><|startoftext|>",
    "İstanbul", "İ", "ǅemal", "ΣΊΣΥΦΟΣ", "straße", "ﬁne", "Ⅷ", "KelvinK", "Ångström",
    "　", "\xa0", "\t", "\n", "\r\n", " \t \n ", " ", "\x85", "​", "­", "\x00", "\x7f",
    "café", "naïve", "résumé", "ÉCOLE", "é", "ä́", "가", "각", "ཱི",
    "中文", "東京都", "한국어", "日本語テキスト", "𠀀𠀁", "😀", "👩‍👩‍👧", "🇫🇷", "Москва", "ПРИВЕТ",
    "---", "...", "$100", "C++", "e-mail", "#hashtag", "@user", "¿qué?", "«quote»", "—", "http://x.org/a?b=c",
]


def _random_cp(rng: random.Random) -> str:
    while True:
        plane = rng.choice([0, 0, 0, 1, 2, 3, 14, 15, 16])
        c = (plane << 16) | rng.randint(0, 0xFFFF)
        if not 0xD800 <= c < 0xE000:
            return chr(c)


def random_text(rng: random.Random) -> str:
    r = rng.random()
    if r < 0.02:
        return ""
    if r < 0.04:
        return rng.choice([" ", "\t\n ", "　 ", "\xa0"])
    if r < 0.07:                                                   # one long word: around and past the word buffer
        return "".join(rng.choice("abcdefghij") for _ in range(rng.randint(200, 300)))
    if r < 0.25:                                                   # "title: description" of movie-description length
        title = " ".join(rng.choice(WORDS).capitalize() for _ in range(rng.randint(1, 4)))
        return title + ": " + " ".join(rng.choice(WORDS) for _ in range(rng.randint(20, 120))) + "."
    parts = []
    for _ in range(rng.randint(1, 30)):
        x = rng.random()
        if x < 0.5:
            w = rng.choice(WORDS)
            parts.append(w.upper() if rng.random() < 0.1 else w.capitalize() if rng.random() < 0.2 else w)
        elif x < 0.85:
            parts.append(rng.choice(PIECES))
        elif x < 0.92:
            parts.append(str(rng.randint(0, 10 ** rng.randint(1, 8))))
        else:
            parts.append(_random_cp(rng))
        parts.append(rng.choice([" ", " ", " ", "", ", ", ". ", " ", "-", "\n", "'"]))
    return "".join(parts)


def texts(n: int, seed: int):
    rng = random.Random(seed)
    return [random_text(rng) for _ in range(n)]


@functools.lru_cache(maxsize=None)
def tokenizer(vocab: str = "trained"):
    """A transformers CLIP tokenizer: ``vocab="trained"`` (BpeTrainer on seeded text, ~6 k pieces) or ``"tiny"``."""
    import transformers
    from tokenizers import Regex, Tokenizer, normalizers, pre_tokenizers
    from tokenizers.models import BPE
    from tokenizers.trainers import BpeTrainer
    from rag_search_engine_b200.bpe import CLIP_PATTERN, bytes_to_unicode
    if vocab == "tiny":
        b2u = bytes_to_unicode()
        v = {s: i for i, s in enumerate(SPECIALS)}
        for b in range(256):
            v.setdefault(b2u[b], len(v))
            if chr(b) in "abcdehlnorst.,'!":                  # every other "x</w>" is missing: unk
                v.setdefault(b2u[b] + "</w>", len(v))
        merges = [("t", "h"), ("th", "e</w>"), ("a", "n"), ("an", "d</w>"), ("e", "r"), ("o", "n</w>"),
                  ("t", "h</w>"), ("s", "t"), ("st", "o"), ("sto", "r"), ("e", "e"), ("ee", "e"), ("l", "l</w>"),
                  ("'", "s</w>"), ("c", "a"), ("ca", "t</w>"), ("e", "e</w>"), ("h", "e"), ("he", "l"),
                  ("hel", "l"), ("hell", "o</w>")]
        for a, b in merges:
            v.setdefault(a + b, len(v))
        return transformers.CLIPTokenizer(vocab=v, merges=merges)
    t = Tokenizer(BPE(unk_token="<|endoftext|>", end_of_word_suffix="</w>", fuse_unk=False))
    t.normalizer = normalizers.Sequence([normalizers.NFC(), normalizers.Replace(Regex(r"\s+"), " "),
                                         normalizers.Lowercase()])
    t.pre_tokenizer = pre_tokenizers.Sequence([pre_tokenizers.Split(Regex(CLIP_PATTERN), behavior="removed",
                                                                    invert=True),
                                               pre_tokenizers.ByteLevel(add_prefix_space=False)])
    t.train_from_iterator(texts(6000, seed=99), BpeTrainer(vocab_size=6000, special_tokens=SPECIALS,
                                                           end_of_word_suffix="</w>",
                                                           initial_alphabet=pre_tokenizers.ByteLevel.alphabet()))
    m = t.get_vocab()
    import json
    merges = [tuple(x) for x in json.loads(t.to_str())["model"]["merges"]]
    return transformers.CLIPTokenizer(vocab=m, merges=merges)
