"""Seeded texts and BERT tokenizers for the WordPiece tests: vocabs trained offline with WordPieceTrainer, a tiny
hand-made vocab (mostly [UNK], long ## chains), the four BertNormalizer configurations, and texts that mix accented
Latin, Greek (final sigma), Cyrillic, CJK, emoji, control and format characters, Unicode spaces, combining marks,
literal special tokens, words over 100 characters and empty or whitespace-only strings."""
from __future__ import annotations

import functools
import random

SPECIALS = ["[PAD]", "[UNK]", "[CLS]", "[SEP]", "[MASK]"]
CONFIGS = {
    "uncased": dict(),
    "cased": dict(lowercase=False),
    "strip_cased": dict(lowercase=False, strip_accents=True),
    "raw_chinese": dict(handle_chinese_chars=False, clean_text=False),
}

ASCII_WORDS = ("the movie a of and to in is that it for with as was on be by his at an are from this film story "
               "love life young man woman world family two new war friends time city finds must home school "
               "tokenization unbelievable reconstruct").split()
PIECES = [
    "café", "naïve", "Ångström", "résumé", "ÉCOLE", "straße", "İstanbul", "ǅemal",
    "ΟΔΥΣΣΕΥΣ", "Σίσυφος", "ΣΣ", "όσος", "Москва", "ПРИВЕТ", "ёжик",
    "中文", "東京都", "한국어", "日本語テキスト", "𠀀𠀁", "😀", "👩‍👩‍👧", "🇫🇷",
    " ", " ", "　", "​", "‍", "﻿", "­", "\x00", "\x07", "\x1f", "\x7f", "\t", "\n",
    "\r\n", "�", "é", "ậ", "ȫ", "́", "x⃝", "𝄞", "\U0001d165\U0001d16d",
    "[SEP]", "[CLS]", "[MASK]", "[mask]", "[sep]", "x[CLS]y", "[UNK]", "[[SEP]]", "[SEP][SEP]",
    "---", "...", "$100", "C++", "e-mail", "#hashtag", "@user", "¿qué?", "«quote»", "—", "½", "²", "ﬁ", "Ⅻ",
]


def random_text(rng: random.Random) -> str:
    r = rng.random()
    if r < 0.03:
        return ""
    if r < 0.06:
        return rng.choice([" ", "\t\n ", "　 ", "​"])
    if r < 0.09:
        return "".join(rng.choice("abcdefghij") for _ in range(rng.randint(95, 140)))       # around max chars
    parts = []
    for _ in range(rng.randint(1, 20)):
        x = rng.random()
        if x < 0.55:
            w = rng.choice(ASCII_WORDS)
            parts.append(w.upper() if rng.random() < 0.1 else w.capitalize() if rng.random() < 0.2 else w)
        elif x < 0.85:
            parts.append(rng.choice(PIECES))
        else:
            parts.append(chr(rng.choice([rng.randint(0x20, 0x2FF), rng.randint(0x370, 0x52F), rng.randint(0x4E00, 0x9FFF),
                                         rng.randint(0x1F300, 0x1FAFF), rng.randint(0x2000, 0x206F),
                                         rng.randint(0x300, 0x36F)])))
        parts.append(rng.choice([" ", " ", " ", "", ", ", ". ", " ", "-"]))
    return "".join(parts)


def texts(n: int, seed: int):
    rng = random.Random(seed)
    return [random_text(rng) for _ in range(n)]


@functools.lru_cache(maxsize=None)
def tokenizer(config: str, vocab: str = "trained"):
    """A transformers fast BERT tokenizer: ``vocab="trained"`` (WordPieceTrainer on seeded text, ~4 k pieces) or
    ``"tiny"`` (a handful of pieces)."""
    import transformers
    from tokenizers import normalizers
    kw = CONFIGS[config]

    def fast(v):
        tok = transformers.BertTokenizerFast(vocab=v, clean_up_tokenization_spaces=False)
        tok.backend_tokenizer.normalizer = normalizers.BertNormalizer(**kw)   # clean_text has no constructor flag
        return tok
    if vocab == "tiny":
        v = {t: i for i, t in enumerate(SPECIALS)}
        for t in ["a", "b", "c", "the", "th", "##e", "##a", "##b", "##c", "##ab", "##abc", "##bc", ",", ".", "-",
                  "中", "σ", "ς", "é", "##é", "caf", "##é", "naive"]:
            v.setdefault(t, len(v))
        return fast(v)
    from tokenizers import Tokenizer, pre_tokenizers
    from tokenizers.models import WordPiece
    from tokenizers.trainers import WordPieceTrainer
    t = Tokenizer(WordPiece(unk_token="[UNK]"))
    t.normalizer = normalizers.BertNormalizer(**kw)
    t.pre_tokenizer = pre_tokenizers.BertPreTokenizer()
    t.train_from_iterator(texts(4000, seed=99), WordPieceTrainer(vocab_size=4000, special_tokens=SPECIALS))
    return fast(t.get_vocab())
