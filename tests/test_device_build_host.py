"""The host side of the device build that needs no GPU: the check that a freshly filled vec0 table keeps rows
0 .. n-1 at positions 0 .. n-1 before the build serves its own matrix instead of the exported one."""
import sqlite3

import numpy as np

from rag_search_engine_b200 import store
from rag_search_engine_b200.semantic_search import _vec0_rows_in_order


def test_vec0_row_order_check(tmp_path):
    conn = sqlite3.connect(tmp_path / "v.db")
    n = 3 * 1024 + 17
    emb = np.random.default_rng(0).standard_normal((n, 8)).astype(np.float32)
    store.write_vec0_shadow(conn, np.arange(n, dtype=np.int64), emb)
    assert _vec0_rows_in_order(conn, n)
    got = store.export_embeddings(conn)
    assert (got.rowid == np.arange(n)).all() and (got.emb == emb).all()
    assert not _vec0_rows_in_order(conn, n + 1)
    conn.execute("UPDATE chunk_embeddings_rowids SET chunk_offset = 5 WHERE rowid = 7")
    assert not _vec0_rows_in_order(conn, n)
    conn.execute("UPDATE chunk_embeddings_rowids SET chunk_offset = 7 WHERE rowid = 7")
    conn.execute("UPDATE chunk_embeddings_chunks SET chunk_id = 9 WHERE chunk_id = 4")
    assert not _vec0_rows_in_order(conn, n)
    conn.close()
