"""configs[0] — the reference's own published sample outputs on ``data/movies.json`` (README.md:137-151).

``movies.json`` is absent from the reference checkout (.MISSING_LARGE_BLOBS) and sentence-transformers / spaCy /
sqlite-vec are not installable in the build container, so this known-answer run SKIPS there.  It enables itself
the day the data and the reference's dependencies are present (set ``RSE_MOVIES_JSON`` or drop the file at
``data/movies.json`` or at ``data/movies.json`` of the reference checkout, see oracle/ref_import.py): the database
is built by the REFERENCE's own build, queried through this package's GPU classes, and compared with the 4-decimal
values the README prints.
"""
import os
from pathlib import Path

import pytest

from oracle import ref_import

ROOT = Path(__file__).resolve().parents[1]


def _movies_json():
    for p in (os.environ.get("RSE_MOVIES_JSON"), ROOT / "data" / "movies.json",
              ref_import.REFERENCE_ROOT / "data" / "movies.json"):
        try:
            if p and Path(p).is_file():
                return Path(p)
        except OSError:               # a path this user may not enter counts as absent
            pass
    return None


pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def built_db(tmp_path_factory):
    data = _movies_json()
    if data is None:
        pytest.skip("data/movies.json is not available (absent from the reference checkout)")
    pytest.importorskip("sqlite_vec")
    pytest.importorskip("sentence_transformers")
    pytest.importorskip("spacy")
    ref_ks = pytest.importorskip("rag_search_engine.utils.keyword_search")
    ref_ss = pytest.importorskip("rag_search_engine.utils.semantic_search")
    db = tmp_path_factory.mktemp("movies") / "movies.db"
    ref_ks.KeywordSearch.build_from_docs(docs_path=data, db_path=db).close()          # `rag-search build` (cli.py:410-423)
    ref_ss.SemanticSearch.build_from_docs(docs_path=data, db_path=db).close()
    return db


def test_semantic_search_vampire_comedy(built_db):
    """README.md:145-151: 0.2044 Vampire / 0.2323 The Vampire Lovers / 0.2764 Vampire Circus."""
    from rag_search_engine_b200 import SemanticSearch
    ss = SemanticSearch(docs_path=None, db_path=built_db)
    try:
        hits = ss.query_top_k("vampire comedy", k=5)
    finally:
        ss.close()
    got = [(f"{h['distance']:.4f}", h["title"]) for h in hits[:3]]
    assert got == [("0.2044", "Vampire"), ("0.2323", "The Vampire Lovers"), ("0.2764", "Vampire Circus")]


def test_key_search_toy(built_db):
    """README.md:137-144: 8.5075 The Christmas Toy / 8.0325 Silent Night, Deadly Night 5: The Toy Maker / 7.9301 Toys."""
    from rag_search_engine.utils.utils import preprocess  # the reference's spaCy tokenizer
    from rag_search_engine_b200 import KeywordSearch
    ks = KeywordSearch(docs_path=None, db_path=built_db, tokenizer=preprocess)
    try:
        hits = ks.search("Toy", k=5)
    finally:
        ks.close()
    got = [(f"{h['score']:.4f}", h["title"]) for h in hits[:3]]
    assert got == [("8.5075", "The Christmas Toy"), ("8.0325", "Silent Night, Deadly Night 5: The Toy Maker"),
                   ("7.9301", "Toys")]
