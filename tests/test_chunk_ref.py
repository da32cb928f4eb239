"""The byte-level restatement of the device chunking (tests/helpers/chunk_ref.py) against store.plan_chunks and
against the reference's pinned answers (tests/golden/live_ref.json)."""
import json
import re
import sys
from pathlib import Path

import numpy as np
import pytest

sys.path.insert(0, str(Path(__file__).resolve().parent))
from helpers import chunk_ref  # noqa: E402
from rag_search_engine_b200 import store  # noqa: E402
from rag_search_engine_b200.device_build import pack_movies  # noqa: E402

GOLDEN = Path(__file__).resolve().parent / "golden"


def test_whitespace_set_is_pythons():
    py = {c for c in range(0x110000) if chr(c).isspace()}
    assert py == set(chunk_ref.WHITESPACE) and len(py) == 29
    assert py == {c for c in range(0x110000) if re.fullmatch(r"\s", chr(c))}
    assert py == {c for c in range(0x110000) if not chr(c).strip()}
    assert not {ord(c) for c in chunk_ref.NEAR_MISSES} & py


@pytest.mark.parametrize("size,overlap", chunk_ref.SIZES)
def test_restatement_equals_plan_chunks(size, overlap):
    movies = chunk_ref.adversarial_movies(seed=size * 10 + overlap + 5, n=1500)
    data, offs = pack_movies(movies)
    texts, movie, index = chunk_ref.chunk_movies(data, offs, size, overlap)
    rows, want = store.plan_chunks(movies, size, overlap)
    assert [t.decode("utf-8") for t in texts] == want
    assert [(movies[m][0], i) for m, i in zip(movie, index)] == [(r[1], r[2]) for r in rows]


def test_adversarial_corpus_covers_the_rules():
    movies = chunk_ref.adversarial_movies(seed=1, n=1500)
    descs = "".join(d for _, _, d in movies)
    assert set(chunk_ref.WHITESPACE) <= {ord(c) for c in descs}
    assert all(c in descs for c in chunk_ref.NEAR_MISSES)
    assert "?!." in descs and any(d == "" for _, _, d in movies)
    assert any(d and not d.strip() for _, _, d in movies)
    assert any(d != d.lstrip() and d.strip() for _, _, d in movies)
    assert any(t != t.strip() for _, t, _ in movies)
    assert max(len(d) for _, _, d in movies) > 1000 and any(not d.isascii() for _, _, d in movies)


def test_restatement_equals_pinned_reference_answers():
    from oracle.make_golden import chunk_inputs
    pinned = json.loads((GOLDEN / "live_ref.json").read_text())["chunks"]
    for (_items, cs, ov, text), want in zip(chunk_inputs(), pinned):
        data, offs = pack_movies([(0, "T", text)])
        got, _, index = chunk_ref.chunk_movies(data, offs, cs, ov)
        assert [g.decode("utf-8") for g in got[1:]] == ["".join(w) for w in want[1]], (cs, ov, text)
        assert index == list(range(len(got)))


def test_max_chunk_size_below_one_is_refused():
    data, offs = pack_movies([(0, "T", "A. B.")])
    for size in (0, -1):
        with pytest.raises(ValueError):
            chunk_ref.chunk_movies(data, offs, size, 0)
        with pytest.raises(ValueError):
            from rag_search_engine_b200.device_build import chunk_movies
            chunk_movies(None, [(0, "T", "A. B.")], size, 0)


def test_parts_respect_the_budget_and_skip_host_routed_movies():
    from rag_search_engine_b200.device_build import _parts
    byte_cu = np.array([0, 10, 30, 35, 100, 110], np.int64)
    chunk_cu = np.array([0, 2, 5, 7, 9, 11], np.int64)
    routed = np.array([False, False, True, False, False])
    assert _parts(routed, byte_cu, chunk_cu, 30) == [(0, 2), (3, 4), (4, 5)]
    assert _parts(routed, byte_cu, chunk_cu, 1) == [(0, 1), (1, 2), (3, 4), (4, 5)]
