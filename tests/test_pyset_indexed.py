"""CPU check of the 16-bit index-slot variant of csrc/pyset.h, the set emulation of the deep fusion kernel (limits
above 128): its union order equals CPython's  set(a) | set(b)  for unions up to 2048 ids, like the 8-byte key-slot
variant beside it."""
import ctypes
import random
import subprocess
from pathlib import Path

import numpy as np
import pytest

ROOT = Path(__file__).resolve().parents[1]
P = ctypes.POINTER(ctypes.c_int64)


@pytest.fixture(scope="module")
def shim(tmp_path_factory):
    so = tmp_path_factory.mktemp("shim") / "pyset_indexed_shim.so"
    subprocess.run(["g++", "-O2", "-shared", "-fPIC", "-o", str(so),
                    str(ROOT / "tests" / "helpers" / "pyset_indexed_shim.cpp")], check=True)
    return ctypes.CDLL(str(so))


def _emu(fn, a, b):
    A, B = np.array(a, np.int64), np.array(b, np.int64)
    out = np.zeros(len(a) + len(b) + 1, np.int64)
    n = fn(A.ctypes.data_as(P), len(a), B.ctypes.data_as(P), len(b), out.ctypes.data_as(P))
    return out[:n].tolist()


def _real(a, b):
    da, db = {x: None for x in a}, {x: None for x in b}
    return list(set(da.keys()) | set(db.keys()))          # hybrid_search.py:148, :248


def test_indexed_union_order_matches_cpython(shim):
    rnd = random.Random(7)
    cases = 0
    for _ in range(600):
        na = rnd.randint(0, rnd.choice([10, 129, 409, 512, 1024]))
        nb = rnd.randint(0, rnd.choice([10, 129, 409, 512, 1024]))
        space = rnd.choice([64, 700, 2048, 10**6, 2**40, 2**62])
        lo = -space if rnd.random() < 0.2 else 0
        # duplicates inside one list are kept: the fusion entry points take plugged-in retrievers' lists as given
        a = [rnd.randrange(lo, space) for _ in range(na)]
        b = [(rnd.choice(a) if a and rnd.random() < 0.4 else rnd.randrange(lo, space)) for _ in range(nb)]
        want = _real(a, b)
        assert _emu(shim.pyset_shim_union_indexed, a, b) == want, (na, nb, space)
        assert _emu(shim.pyset_shim_union, a, b) == want, (na, nb, space)
        cases += len(want) > 1024
    assert cases > 5


def test_indexed_union_at_2048_distinct_ids(shim):
    """The widest union the deep kernel forms: two disjoint 1024-id lists, ids around 2^62 and below zero, and the
    hash-colliding values -1 / -2 (CPython maps hash(-1) to -2)."""
    rnd = random.Random(11)
    for space, lo in ((2**62, 2**62 - 10**7), (10**5, -10**5), (2048, -2)):
        ids = rnd.sample(range(lo, lo + space if lo < 0 else space), 2048) if space > 2048 else list(range(-2, 2046))
        rnd.shuffle(ids)
        a, b = ids[:1024], ids[1024:]
        assert _emu(shim.pyset_shim_union_indexed, a, b) == _real(a, b)
