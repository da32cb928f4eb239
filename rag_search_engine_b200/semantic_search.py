"""SemanticSearch — drop-in for rag_search_engine.utils.semantic_search.SemanticSearch whose
``query_top_k`` runs the vec0 KNN + best-chunk-per-movie aggregation on the B200.

Same constructor, method names, return dicts and error behaviour as the reference
(semantic_search.py:36-65, :211-340, :375-395).  The chunk embeddings are read once from the
vec0 shadow tables of the reference-built SQLite file (store.export_embeddings) and kept in HBM;
chunk text / titles for the ≤k hits still come from SQLite (:262-279, :321-328).
"""
from __future__ import annotations

import json
import sqlite3
import time
from pathlib import Path
from typing import Any, Dict, List, Optional

import numpy as np

from . import runtime, store
from .keyword_search import DEFAULT_DB_PATH
from .textutil import chunk_text

MAX_EXACT_K = 4096                                              # rse_knn_movies_exact's bound on k (include/rse.h)


def _default_encoder():
    try:
        from sentence_transformers import SentenceTransformer  # type: ignore
    except Exception:
        return None
    return SentenceTransformer("all-MiniLM-L6-v2")              # semantic_search.py:45


def _vec0_rows_in_order(conn: sqlite3.Connection, n: int) -> bool:
    """Rows 0 .. n-1 of a freshly filled vec0 table sit at positions 0 .. n-1 of store.export_embeddings: ceil(n /
    1024) consecutive blocks, and every rowid at (block - first block) * 1024 + its offset."""
    t = store.VEC_TABLE
    n_blocks, lo, hi = conn.execute(f"SELECT COUNT(*), MIN(chunk_id), MAX(chunk_id) FROM {t}_chunks").fetchone()
    if n_blocks != (n + store.VEC0_BLOCK - 1) // store.VEC0_BLOCK or hi - lo + 1 != n_blocks:
        return False
    (n_rows,) = conn.execute(f"SELECT COUNT(*) FROM {t}_rowids").fetchone()
    (bad,) = conn.execute(f"SELECT COUNT(*) FROM {t}_rowids WHERE (chunk_id - ?) * ? + chunk_offset != rowid",
                          (lo, store.VEC0_BLOCK)).fetchone()
    return n_rows == n and bad == 0


class SemanticSearch:
    def __init__(self, docs_path: Path | str | None = None, db_path: Path | str | None = None,
                 max_chunk_size: int = 3, overlap: int = 1, force: bool = False, *, encoder=None,
                 device: int = 0, fallback_build: bool = False, device_build: bool = False) -> None:
        self.model = encoder if encoder is not None else _default_encoder()
        self.max_chunk_size = max_chunk_size
        self.overlap = overlap
        self.db_path = Path(db_path) if db_path else Path(DEFAULT_DB_PATH)
        self.db_path.parent.mkdir(parents=True, exist_ok=True)
        self.docs_path = Path(docs_path) if docs_path else None
        self.device = device
        self.fallback_build = fallback_build
        self.device_build = device_build
        if self.docs_path is not None:
            self._build_device(force) if device_build else self._build(force)
        self.conn = sqlite3.connect(self.db_path)
        self.conn.execute("PRAGMA journal_mode=WAL")
        self.conn.execute("PRAGMA synchronous=NORMAL")
        store._init_schema(self.conn)                         # a fresh database opens empty, as the reference's does
        self._index = runtime.acquire(self.db_path, device)
        self._closed = False
        self._load()
        self.embedding_dim = (self.model.get_sentence_embedding_dimension() if self.model is not None
                              else self._arr.dim)

    # ------------------------------------------------------------------ build (stays on SQLite)
    def _build(self, force: bool) -> None:
        """Chunking + embedding + vec0 insert are NOT accelerated (SURVEY §2 #1): use the reference's
        build when it is importable, else freeze embeddings with the given encoder into the same
        tables (store.write_reference_db)."""
        try:
            from rag_search_engine.utils.semantic_search import SemanticSearch as RefSS  # type: ignore
            ref = RefSS(docs_path=self.docs_path, db_path=self.db_path, max_chunk_size=self.max_chunk_size,
                        overlap=self.overlap, force=force)
            ref.close()
            return
        except ImportError:
            pass
        if not self.fallback_build:
            raise RuntimeError("the index build stays on the reference (SQLite + sqlite-vec, north_star) and the "
                               "reference package is not importable here; pass fallback_build=True to freeze the "
                               "embeddings into a GPU-ONLY database (vec0 shadow tables without the virtual table: "
                               "sqlite-vec / the reference cannot open it)")
        if self.model is None:
            raise RuntimeError("SemanticSearch build needs an encoder (sentence-transformers is not installed): "
                               "pass encoder=<object with .encode(texts)>")
        conn = sqlite3.connect(self.db_path)
        try:
            store._init_schema(conn)
            self._sync_movies_json(conn)
            cur = conn.cursor()
            if force or not self._in_sync(conn):
                movies = cur.execute("SELECT id, title, description FROM movies ORDER BY id").fetchall()
                rows, texts = store.plan_chunks(movies, self.max_chunk_size, self.overlap)
                cur.execute("DELETE FROM chunks")
                cur.executemany("INSERT INTO chunks(id, movie_id, chunk_index, max_chunk_size, overlap) "
                                "VALUES (?,?,?,?,?)", rows)
                emb = np.asarray(self.model.encode(texts), np.float32)
                store.write_vec0_shadow(conn, np.array([r[0] for r in rows], np.int64), emb)
                conn.commit()
        finally:
            conn.close()

    def _sync_movies_json(self, conn: sqlite3.Connection) -> None:
        """The fallback build's movies sync: the JSON rows replace the table when the counts differ."""
        data = json.loads(Path(self.docs_path).read_text(encoding="utf-8"))["movies"]
        cur = conn.cursor()
        (n_movies,) = cur.execute("SELECT COUNT(*) FROM movies").fetchone()
        if n_movies != len(data):
            cur.execute("DELETE FROM movies")
            cur.executemany("INSERT INTO movies(id, title, description) VALUES (?, ?, ?)",
                            [(int(d["id"]), d["title"], d["description"]) for d in data])
            conn.commit()

    def _in_sync(self, conn: sqlite3.Connection) -> bool:
        """semantic_search.py:145-154: chunks exist, all of this (max_chunk_size, overlap), and vec0 exists."""
        cur = conn.cursor()
        (n_chunks,) = cur.execute("SELECT COUNT(*) FROM chunks").fetchone()
        params = cur.execute("SELECT DISTINCT max_chunk_size, overlap FROM chunks").fetchall()
        return (n_chunks > 0 and len(params) == 1 and params[0] == (self.max_chunk_size, self.overlap)
                and store._table_exists(conn, f"{store.VEC_TABLE}_chunks"))

    def _sync_movies(self, conn: sqlite3.Connection) -> None:
        """The movies table for the device build: the reference's own sync when the reference is importable — its
        BaseSearchDB, constructed like the reference's search classes (docs_path=, db_path=), loads the docs and
        syncs the table (basesearch_db.py:24-49, :81-92) and may fix the texts it stores, so the build reads the rows
        back from the table — else the fallback build's JSON sync."""
        try:
            from rag_search_engine.utils.basesearch_db import BaseSearchDB  # type: ignore
        except ImportError:
            self._sync_movies_json(conn)
            return
        BaseSearchDB(docs_path=self.docs_path, db_path=self.db_path).close()

    def _build_device(self, force: bool) -> None:
        """``device_build=True``: the chunk texts, their ids and their embeddings are made on the device
        (device_build.build_embeddings) and the matrix stays in HBM as this handle's corpus; the ``chunks`` rows, vec0
        and the ``.rse-emb`` sidecar are written from the one host copy.  vec0 goes through the real ``vec0`` virtual
        table when ``sqlite_vec`` is importable (the reference can open the file), else, under ``fallback_build=True``
        only, into the shadow tables ``store.write_vec0_shadow`` writes."""
        from . import device_build
        from .encoder import DeviceWordPiece, GpuSentenceEncoder
        if self.max_chunk_size < 1:
            raise ValueError(f"max_chunk_size must be >= 1 (got {self.max_chunk_size})")
        try:
            import sqlite_vec  # type: ignore
        except ImportError:
            sqlite_vec = None
        if sqlite_vec is None and not self.fallback_build:
            raise RuntimeError("device_build writes vec0 through sqlite-vec, which is not importable here; pass "
                               "fallback_build=True as well to write a GPU-ONLY database (vec0 shadow tables without the "
                               "virtual table: sqlite-vec / the reference cannot open it)")
        index = runtime.acquire(self.db_path, self.device)
        try:
            enc = self.model
            if not isinstance(enc, GpuSentenceEncoder) or not isinstance(enc.tokenizer, DeviceWordPiece):
                raise TypeError("device_build needs encoder=GpuSentenceEncoder(...) with a DeviceWordPiece tokenizer")
            if enc.index is not index or enc.tokenizer.index is not index:
                raise ValueError("device_build: the encoder (and its DeviceWordPiece) must live on this database's "
                                 "handle, runtime.acquire(db_path, device)")
            conn = sqlite3.connect(self.db_path)
            try:
                store._init_schema(conn)
                self._sync_movies(conn)
                cur = conn.cursor()
                if self._in_sync(conn) and not force:
                    return
                movies = cur.execute("SELECT id, title, description FROM movies ORDER BY id").fetchall()
                built = device_build.build_embeddings(enc, movies, self.max_chunk_size, self.overlap)
                self._write_device_build(conn, index, movies, built, sqlite_vec)
            finally:
                conn.close()
        finally:
            runtime.release(self.db_path, self.device)

    def _write_device_build(self, conn, index, movies, built, sqlite_vec) -> None:
        """The chunks rows, vec0 and (through _load) the sidecar from the one host copy; the device matrix becomes the
        handle's corpus.  ``self.build_timings``: seconds per stage, the device stages of build_embeddings first."""
        import torch
        t = self.build_timings = dict(built.timings)
        ts = time.perf_counter()
        emb = built.emb.cpu().numpy()                                    # the one host copy
        t["device_to_host"] = time.perf_counter() - ts
        ts = time.perf_counter()
        n = int(built.movie_idx.shape[0])
        movie_ids = np.array([m[0] for m in movies], np.int64)
        per = built.chunks_per_movie
        first = np.repeat(np.cumsum(per) - per, per)
        chunk_ids = np.arange(n, dtype=np.int64)
        rows = zip(chunk_ids.tolist(), np.repeat(movie_ids, per).tolist(), (chunk_ids - first).tolist(),
                   [self.max_chunk_size] * n, [self.overlap] * n)
        cur = conn.cursor()
        cur.execute("DELETE FROM chunks")
        cur.executemany("INSERT INTO chunks(id, movie_id, chunk_index, max_chunk_size, overlap) VALUES (?,?,?,?,?)",
                        rows)
        conn.commit()
        t["sqlite_chunks"] = time.perf_counter() - ts
        ts = time.perf_counter()
        if sqlite_vec is not None:
            conn.enable_load_extension(True)
            sqlite_vec.load(conn)                                        # semantic_search.py:68-72
            conn.enable_load_extension(False)
            for x in ("_chunks", "_vector_chunks00", "_rowids", "_info"):  # a shadow-only layout from an earlier build
                if not store._table_exists(conn, store.VEC_TABLE) and store._table_exists(conn, store.VEC_TABLE + x):
                    cur.execute(f"DROP TABLE {store.VEC_TABLE}{x}")
            if store._table_exists(conn, "rse_meta"):
                cur.execute("DELETE FROM rse_meta WHERE key = 'vec0_shadow_writer'")
            cur.execute(f"DROP TABLE IF EXISTS {store.VEC_TABLE}")
            cur.execute(f"CREATE VIRTUAL TABLE IF NOT EXISTS {store.VEC_TABLE} USING vec0("
                        f"embedding float[{emb.shape[1]}] distance_metric=cosine)")      # :94-101
            cur.executemany(f"INSERT INTO {store.VEC_TABLE}(rowid, embedding) VALUES (?, ?)",   # :203-206
                            ((i, emb[i]) for i in range(n)))
        else:
            store.write_vec0_shadow(conn, chunk_ids, emb)
        conn.commit()
        t["sqlite_vec0"] = time.perf_counter() - ts
        if n == 0:                                                        # an empty index: _load exports it as usual
            return
        ts = time.perf_counter()
        keep = None
        if not _vec0_rows_in_order(conn, n):
            # vec0 placed the rows elsewhere than positions 0 .. n-1: serve what the file holds, as a fresh open would
            arr = store.export_embeddings(conn)
            index.load_embeddings(arr.emb, valid=arr.valid, rowid=arr.rowid, movie_idx=arr.movie_idx)
        else:
            # rows inserted 0, 1, ... into a fresh table sit at positions 0, 1, ...: these are the arrays
            # store.export_embeddings reads back from the file
            arr = store.EmbArrays(emb=emb, valid=None, rowid=chunk_ids, movie_idx=built.movie_idx,
                                  movie_ids=movie_ids, dim=int(emb.shape[1]))
            rowid_dev = torch.from_numpy(chunk_ids).to(built.emb.device)
            midx_dev = torch.from_numpy(built.movie_idx).to(built.emb.device)
            torch.cuda.synchronize(built.emb.device)
            index.attach_embeddings_dev(built.emb.data_ptr(), n, int(emb.shape[1]), rowid_ptr=rowid_dev.data_ptr(),
                                        movie_idx_ptr=midx_dev.data_ptr(), keepalive=built.emb)
            index.synchronize()
            keep = built.emb                                             # the registry keeps the borrowed matrix
        t["attach"] = time.perf_counter() - ts
        # the sidecar is written by _load, with the fingerprint of the connection a later open compares against
        self._device_built = arr
        full = store._db_fingerprint(conn, self.db_path)
        reg = runtime.parts(self.db_path, self.device)
        reg["emb"], reg["emb_fp"] = arr, store.part_fingerprint(full, "emb")
        reg["emb_dev"] = keep
        reg.pop("ids", None)

    def _load(self) -> None:
        reg = runtime.parts(self.db_path, self.device)
        full = store._db_fingerprint(self.conn, self.db_path)
        fp = store.part_fingerprint(full, "emb")
        built = self.__dict__.pop("_device_built", None)
        if built is not None:                                     # the device build's host copy: no export
            ts = time.perf_counter()
            store.write_sidecar(self.db_path, "emb", built, json.dumps(full, sort_keys=True))
            self.build_timings["sidecar"] = time.perf_counter() - ts
        if "emb" not in reg or reg.get("emb_fp") != fp:          # first open, or re-embedded under a live handle
            arr = store.load_or_export(self.conn, self.db_path, "emb", fingerprint=full)
            if arr.emb.shape[0] > 0:
                self._index.load_embeddings(arr.emb, valid=arr.valid, rowid=arr.rowid, movie_idx=arr.movie_idx)
                reg.pop("emb_dev", None)                         # a device-built matrix this load replaced
            else:
                # no chunk embeddings (keyword-only / fresh database): query_top_k returns [] like the reference;
                # the handle still needs a dimension for the batch entry points' reshape
                self._index.dim = int(arr.dim) or (int(self.model.get_sentence_embedding_dimension())
                                                   if self.model is not None else 384)
                self._index.n_rows = 0
            reg["emb"], reg["emb_fp"] = arr, fp
            reg.pop("ids", None)

    @property
    def _arr(self) -> store.EmbArrays:
        own = self.__dict__.get("_arr_own")                      # set directly by from_loaded / tests
        return own if own is not None else runtime.parts(self.db_path, self.device)["emb"]

    @_arr.setter
    def _arr(self, value) -> None:
        self.__dict__["_arr_own"] = value

    # ------------------------------------------------------------------ BaseSearchDB helpers
    def count_movies(self) -> int:
        (count,) = self.conn.execute("SELECT COUNT(*) FROM movies").fetchone()
        return count

    def close(self) -> None:
        if not self._closed:
            self._closed = True
            self.conn.close()
            runtime.release(self.db_path, self.device)

    @classmethod
    def build_from_docs(cls, docs_path, db_path=None, force: bool = False, **kw) -> "SemanticSearch":
        return cls(docs_path=docs_path, db_path=db_path, force=force, **kw)

    @classmethod
    def open_existing(cls, db_path=None, **kw) -> "SemanticSearch":
        return cls(docs_path=None, db_path=db_path, **kw)

    # ------------------------------------------------------------------ embeddings (semantic_search.py:211-222)
    def generate_embedding(self, text):
        texts = [text] if isinstance(text, str) else text
        if any(len(t.strip()) == 0 for t in texts):
            raise ValueError("cannot embed empty text")
        if self.model is None:
            raise RuntimeError("no query encoder (sentence-transformers is not installed): pass encoder=... "
                               "or call query_top_k_vec with frozen query vectors")
        return np.asarray(self.model.encode(texts), dtype=np.float32)

    # ------------------------------------------------------------------ query
    def query_top_k_vec(self, query_vecs, k: int = 5, knn_multiplier: int = 10, *,
                        exact_movies: bool = False) -> List[List[Dict[str, Any]]]:
        """Batch entry point on frozen query vectors [B, dim] → one reference-shaped result list per query.

        exact_movies=True: the k nearest movies by best chunk over every chunk (rse_knn_movies_exact), not only
        over the top k * knn_multiplier chunks, so a query gets min(k, movies) hits; knn_multiplier is ignored
        and k may go up to 4096.  Where the default call returns k movies, the exact one returns the same list."""
        if exact_movies and not 1 <= int(k) <= MAX_EXACT_K:
            raise ValueError(f"exact_movies: k must be in [1, {MAX_EXACT_K}], got {k}")
        Q = np.atleast_2d(np.ascontiguousarray(query_vecs, np.float32))
        if self._arr.emb.shape[0] == 0:                         # no chunk embeddings: [] per query, like the reference
            return [[] for _ in range(Q.shape[0])]
        Q = Q.reshape(-1, self._arr.dim)
        if exact_movies:
            dist, rowid, movie, cnt, _ = self._index.knn_movies_exact(Q, int(k))
        else:
            internal_k = max(k * knn_multiplier, k)             # semantic_search.py:251
            dist, rowid, movie, cnt = self._index.knn_movies(Q, k, internal_k)
        # the two JOINs of semantic_search.py:262-279 for the <= k final hits of every query: ONE lookup per table
        # for the whole batch (a point query per hit costs more than the device call from ~100 hits on)
        movie_ids = self._arr.movie_ids
        live = np.arange(rowid.shape[1])[None, :] < np.asarray(cnt)[:, None]
        chunk_meta = self._fetch("SELECT id, chunk_index, max_chunk_size, overlap FROM chunks WHERE id IN ({})",
                                 np.unique(rowid[live]))
        movie_meta = self._fetch("SELECT id, title, description FROM movies WHERE id IN ({})",
                                 np.unique(movie_ids[movie[live]]))
        out = []
        for q in range(Q.shape[0]):
            hits = []
            for j in range(cnt[q]):
                cid = int(rowid[q, j])
                movie_id = int(movie_ids[movie[q, j]])
                ci, mcs, ov = chunk_meta[cid]
                title, desc = movie_meta[movie_id]
                hits.append({"chunk_id": cid, "distance": float(dist[q, j]),
                             "chunk": chunk_text(title, desc, int(ci), int(mcs), int(ov)),
                             "movie_id": movie_id, "title": title, "description": desc})
            out.append(hits)
        return out

    def _fetch(self, sql: str, ids) -> Dict[int, tuple]:
        """{id: rest of the row} for ``ids`` (int64 array), in slices below SQLite's bound-variable limit."""
        got: Dict[int, tuple] = {}
        cur = self.conn.cursor()
        ids = [int(i) for i in ids]
        for lo in range(0, len(ids), 900):
            part = ids[lo:lo + 900]
            for row in cur.execute(sql.format(",".join("?" * len(part))), part):
                got[row[0]] = row[1:]
        return got

    def query_top_k(self, query_text: str, k: int = 5, knn_multiplier: int = 10, *,
                    exact_movies: bool = False) -> List[Dict[str, Any]]:
        """semantic_search.py:225-340; exact_movies as in query_top_k_vec."""
        if exact_movies and not 1 <= int(k) <= MAX_EXACT_K:
            raise ValueError(f"exact_movies: k must be in [1, {MAX_EXACT_K}], got {k}")
        query_vec = self.generate_embedding(query_text)[0]
        return self.query_top_k_vec(query_vec[None, :], k=k, knn_multiplier=knn_multiplier,
                                    exact_movies=exact_movies)[0]

    def _reconstruct_chunk_text(self, title, description, chunk_index, max_chunk_size, overlap) -> str:
        return chunk_text(title, description, chunk_index, max_chunk_size, overlap)

    # ------------------------------------------------------------------ verify (semantic_search.py:368-395)
    def verify_model(self) -> None:
        print(f"Model loaded: {self.model}")
        print(f"Max sequence length: {getattr(self.model, 'max_seq_length', None)}")
        print(f"Embedding dim: {self.embedding_dim}")

    def verify_db(self) -> None:
        cur = self.conn.cursor()
        (movie_count,) = cur.execute("SELECT COUNT(*) FROM movies").fetchone()
        (chunk_count,) = cur.execute("SELECT COUNT(*) FROM chunks").fetchone()
        vec_count = int(self._arr.valid.sum()) if self._arr.valid is not None else int(self._arr.emb.shape[0])
        print(f"Vector DB path: {self.db_path}")
        print("sqlite-vec version: (not loaded: vec0 shadow tables read directly; KNN runs in librse on the GPU)")
        print(f"Movies count:            {movie_count}")
        print(f"Chunks table count:      {chunk_count}")
        print(f"Embeddings (vec0) count: {vec_count}")
        print(f"Embedding dim:           {self.embedding_dim}")
