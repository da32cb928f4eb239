"""Import the UNMODIFIED reference (a checkout of rag-search-engine under ``oracle/_ref``,
or wherever ``RSE_REFERENCE_ROOT`` points) with stub modules for those of its third-party
packages that are not installed.

TEST INFRASTRUCTURE ONLY.  The checkout is not part of this repository (``oracle/_ref`` is
git-ignored).  Used by oracle/make_golden.py to generate the golden fixtures under
tests/golden/ and by tests that are skipped when the reference is not present.

Stubbed (never reached by the arithmetic under test): spacy, rapidfuzz,
sqlite_vec, sentence_transformers, google.genai.  ``preprocess`` is replaced by
a frozen whitespace tokenizer (the reference's spaCy pipeline is query/corpus
NLP, out of scope — SURVEY §2 #5).
"""
from __future__ import annotations

import os
import sys
import types
from pathlib import Path

REFERENCE_ROOT = Path(os.environ.get("RSE_REFERENCE_ROOT") or Path(__file__).resolve().parent / "_ref")


def available() -> bool:
    try:
        return (REFERENCE_ROOT / "rag_search_engine" / "utils" / "keyword_search.py").is_file()
    except OSError:                   # a path this user may not enter counts as absent
        return False


def frozen_preprocess(texts, n_process=1, batch_size=256):
    """Whitespace/lower-case stand-in for utils/utils.py:75-123 (same call shape)."""
    if isinstance(texts, str):
        texts = [texts]
    return [[t for t in s.lower().split()] for s in texts]


def _stub(name: str, **attrs) -> types.ModuleType:
    m = types.ModuleType(name)
    m.__dict__.update(attrs)
    sys.modules[name] = m
    return m


def install_stubs() -> None:
    if "spacy" not in sys.modules:
        try:
            import spacy  # noqa: F401
        except Exception:
            sp = _stub("spacy", load=lambda *a, **k: None)
            lang = _stub("spacy.lang")
            en = _stub("spacy.lang.en")
            sw = _stub("spacy.lang.en.stop_words", STOP_WORDS=set())
            sp.lang = lang
            lang.en = en
            en.stop_words = sw
    if "rapidfuzz" not in sys.modules:
        try:
            import rapidfuzz  # noqa: F401
        except Exception:
            fz = _stub("rapidfuzz.fuzz", partial_ratio=lambda *a, **k: 0.0)
            pr = _stub("rapidfuzz.process", extractOne=lambda *a, **k: None)
            _stub("rapidfuzz", fuzz=fz, process=pr)
    if "sqlite_vec" not in sys.modules:
        try:
            import sqlite_vec  # noqa: F401
        except Exception:
            def _load(conn):
                raise RuntimeError("sqlite_vec stub: extension not available in this image")
            _stub("sqlite_vec", load=_load)
    if "sentence_transformers" not in sys.modules:
        try:
            import sentence_transformers  # noqa: F401
        except Exception:
            class _NoModel:
                def __init__(self, *a, **k):
                    raise RuntimeError("sentence_transformers stub")
            _stub("sentence_transformers", SentenceTransformer=_NoModel, CrossEncoder=_NoModel)
    if "google.genai" not in sys.modules:
        try:
            from google import genai  # noqa: F401
        except Exception:
            g = sys.modules.get("google") or _stub("google")
            if not hasattr(g, "__path__"):
                g.__path__ = []
            ty = _stub("google.genai.types")
            er = _stub("google.genai.errors", APIError=Exception, ClientError=Exception)
            ge = _stub("google.genai", types=ty, errors=er, Client=object)
            g.genai = ge


def load():
    """Returns (keyword_search, hybrid_search, utils) reference modules, preprocess frozen."""
    if not available():
        raise RuntimeError(f"reference not found under {REFERENCE_ROOT}")
    install_stubs()
    if str(REFERENCE_ROOT) not in sys.path:
        sys.path.insert(0, str(REFERENCE_ROOT))
    import rag_search_engine.utils.utils as ref_utils
    import rag_search_engine.utils.keyword_search as ref_kw
    import rag_search_engine.utils.hybrid_search as ref_hs
    ref_kw.preprocess = frozen_preprocess
    ref_utils.preprocess = frozen_preprocess
    return ref_kw, ref_hs, ref_utils
