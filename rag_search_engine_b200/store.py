"""Load-time exporter: reference SQLite file → the arrays librse keeps in HBM.

SQLite stays the build/storage layer (north_star); this module only READS a database that
the reference built (``rag-search build``) with the stdlib ``sqlite3`` — no sqlite-vec
extension needed, because vec0 keeps its data in ordinary shadow tables:

  chunk_embeddings_chunks(chunk_id, size, validity BLOB, rowids BLOB)
  chunk_embeddings_vector_chunks00(rowid = chunk_id, vectors BLOB)      (SURVEY App. C)

and the keyword index lives in terms / postings / doclen
(rag_search_engine/utils/keyword_search.py:43-78).  It also contains the writer for those
same tables (``write_reference_db``), used to freeze synthetic corpora / precomputed
embeddings to disk in the reference's on-disk format where the reference's own build
(spaCy + sentence-transformers + sqlite-vec) is not installable.
"""
from __future__ import annotations

import hashlib
import json
import logging
import os
import sqlite3
from dataclasses import dataclass, field
from pathlib import Path
from typing import Callable, Dict, List, Optional, Sequence

import numpy as np

from .textutil import Tokenizer, sentence_chunks

VEC0_BLOCK = 1024
TITLE_END_TOKEN = "[TITLE_END]"        # keyword_search.py:24
VEC_TABLE = "chunk_embeddings"         # semantic_search.py:94
EXPORT_SLICE_POSTINGS = 1 << 22        # export_bm25 reads the postings table in slices of about this many rows

logger = logging.getLogger(__name__)


# ----------------------------------------------------------------------------- BM25 export
@dataclass
class Bm25Arrays:
    indptr: np.ndarray          # [T+1] int64
    doc_idx: np.ndarray         # [P] uint32 dense index into doc_ids, ascending within a term
    tf: np.ndarray              # [P] uint32 = len(positions)
    df: np.ndarray              # [T] int64 = len(rows) as the reference counts it (:222)
    dl: np.ndarray              # [M] uint32
    doc_ids: np.ndarray         # [M] int64 ascending (doclen.doc_id)
    n_movies: int               # COUNT(*) FROM movies (:196)
    avgdl: float                # AVG(length) FROM doclen (:197-198); 0.0 when the table is empty
    term_row: Dict[str, int] = field(default_factory=dict)


def export_bm25(conn: sqlite3.Connection) -> Bm25Arrays:
    cur = conn.cursor()
    (n_movies,) = cur.execute("SELECT COUNT(*) FROM movies").fetchone()
    rows = cur.execute("SELECT doc_id, length FROM doclen ORDER BY doc_id").fetchall()
    doc_ids = np.array([r[0] for r in rows], np.int64)
    dl = np.array([r[1] for r in rows], np.uint32)
    (avgdl,) = cur.execute("SELECT AVG(length) FROM doclen").fetchone()
    terms = cur.execute("SELECT id, term FROM terms ORDER BY id").fetchall()
    term_ids = np.array([t[0] for t in terms], np.int64)
    term_row = {t[1]: i for i, t in enumerate(terms)}
    T = len(terms)
    # postings in (term_id, doc_id) order = the autoindex order the reference reads them in (:214-218).  One result
    # row per TERM (group_concat over the (term_id, doc_id) autoindex), parsed in bulk: a Python tuple per posting
    # costs ~1.3 us in sqlite3's row loop alone — minutes at 54 M postings — against ~0.5 us this way.
    t_list: List[np.ndarray] = []
    d_list: List[np.ndarray] = []
    f_list: List[np.ndarray] = []
    # slices of ~4 M postings, cut on the per-term counts (term ids are handed out by first appearance, so the low
    # ids hold most of a Zipfian index: equal-width id ranges would put nearly everything into the first slice)
    per_term = np.array(cur.execute("SELECT term_id, COUNT(*) FROM postings GROUP BY term_id ORDER BY term_id").fetchall(),
                        np.int64).reshape(-1, 2)
    if len(per_term):
        csum = np.cumsum(per_term[:, 1])
        cuts = np.searchsorted(csum, np.arange(EXPORT_SLICE_POSTINGS, int(csum[-1]), EXPORT_SLICE_POSTINGS), side="left") + 1
        starts = np.concatenate([[0], cuts]).astype(np.int64)
        ends = np.concatenate([cuts, [len(per_term)]]).astype(np.int64)
        for a, b in zip(starts.tolist(), ends.tolist()):
            if a >= b:
                continue
            lo, hi = int(per_term[a, 0]), int(per_term[b - 1, 0])
            grp = cur.execute("SELECT term_id, group_concat(doc_id), group_concat(json_array_length(positions)) "
                              "FROM postings WHERE term_id >= ? AND term_id <= ? GROUP BY term_id ORDER BY term_id",
                              (lo, hi)).fetchall()
            cnt = per_term[a:b, 1]
            if [g[0] for g in grp] != per_term[a:b, 0].tolist():
                raise RuntimeError("postings export: the table changed while it was being read")
            t_list.append(np.repeat(per_term[a:b, 0], cnt))
            d_list.append(np.fromstring(",".join(g[1] for g in grp), dtype=np.int64, sep=","))
            f_list.append(np.fromstring(",".join(g[2] for g in grp), dtype=np.int64, sep=","))
            if len(d_list[-1]) != cnt.sum() or len(f_list[-1]) != cnt.sum():
                raise RuntimeError("postings export: group_concat row count mismatch")
    if t_list:
        pt = np.concatenate(t_list); pd = np.concatenate(d_list); pf = np.concatenate(f_list)
        # SQL does not promise an order inside a group (in practice the autoindex gives doc_id ascending): check, and
        # sort when it is not the reference's read order
        if len(pt) > 1 and not (((pt[1:] > pt[:-1]) | ((pt[1:] == pt[:-1]) & (pd[1:] > pd[:-1]))).all()):
            order = np.lexsort((pd, pt))
            pt, pd, pf = pt[order], pd[order], pf[order]
    else:
        pt = pd = pf = np.zeros(0, np.int64)
    trow = np.searchsorted(term_ids, pt)
    known_t = (trow < T)
    known_t[known_t] &= term_ids[trow[known_t]] == pt[known_t]
    trow, pd, pf = trow[known_t], pd[known_t], pf[known_t]
    df = np.bincount(trow, minlength=T).astype(np.int64)                 # len(rows), before the doclen filter
    didx = np.searchsorted(doc_ids, pd)
    has_dl = didx < len(doc_ids)
    has_dl[has_dl] &= doc_ids[didx[has_dl]] == pd[has_dl]                # `if not dl_row: continue` (:235-236)
    trow, didx, pf = trow[has_dl], didx[has_dl], pf[has_dl]
    indptr = np.zeros(T + 1, np.int64)
    np.cumsum(np.bincount(trow, minlength=T), out=indptr[1:])
    return Bm25Arrays(indptr=indptr, doc_idx=didx.astype(np.uint32), tf=pf.astype(np.uint32), df=df, dl=dl,
                      doc_ids=doc_ids, n_movies=int(n_movies), avgdl=float(avgdl) if avgdl else 0.0,
                      term_row=term_row)


# ----------------------------------------------------------------------------- vec0 export
@dataclass
class EmbArrays:
    emb: np.ndarray                     # [n_phys, dim] float32, vec0 physical layout (block*1024 + slot)
    valid: Optional[np.ndarray]         # [n_phys] uint8, None = all valid
    rowid: np.ndarray                   # [n_phys] int64 (chunks.id)
    movie_idx: np.ndarray               # [n_phys] int32 dense index into movie_ids, -1 = dropped by the JOINs
    movie_ids: np.ndarray               # [Mm] int64 ascending (movies.id)
    dim: int


def _table_exists(conn: sqlite3.Connection, name: str) -> bool:
    return conn.execute("SELECT 1 FROM sqlite_master WHERE name = ?", (name,)).fetchone() is not None


def export_embeddings(conn: sqlite3.Connection, table: str = VEC_TABLE) -> EmbArrays:
    """Read the vec0 shadow tables in vec0's own scan order (chunk_id ascending, slot ascending)."""
    cur = conn.cursor()
    movie_ids = (np.array([r[0] for r in cur.execute("SELECT id FROM movies ORDER BY id")], np.int64)
                 if _table_exists(conn, "movies") else np.zeros(0, np.int64))
    if not _table_exists(conn, f"{table}_chunks") or not _table_exists(conn, f"{table}_vector_chunks00"):
        # a keyword-only or fresh database: the reference creates an EMPTY chunk_embeddings table at open time
        # (semantic_search.py:94-101) and query_top_k returns [] — same here: no rows, no error
        return EmbArrays(np.zeros((0, 1), np.float32), None, np.zeros(0, np.int64), np.zeros(0, np.int32), movie_ids, 0)
    empty = EmbArrays(np.zeros((0, 1), np.float32), None, np.zeros(0, np.int64), np.zeros(0, np.int32), movie_ids, 0)
    (n_blocks,) = cur.execute(f"SELECT COUNT(*) FROM {table}_chunks c JOIN {table}_vector_chunks00 v "
                              f"ON v.rowid = c.chunk_id").fetchone()
    if n_blocks == 0:
        return empty
    # one pass over the blobs straight into the final arrays (sized from the block count; blocks without live rows
    # are skipped and trimmed off below): peak memory is the matrix itself, not the matrix plus a list of its blobs
    emb = None
    valid = np.zeros(n_blocks * VEC0_BLOCK, np.uint8)
    rowid = np.zeros(n_blocks * VEC0_BLOCK, np.int64)
    dim = None
    n = 0
    for _cid, size, validity, rowid_blob, vectors in cur.execute(
            f"SELECT c.chunk_id, c.size, c.validity, c.rowids, v.vectors FROM {table}_chunks c "
            f"JOIN {table}_vector_chunks00 v ON v.rowid = c.chunk_id ORDER BY c.chunk_id"):
        if size != VEC0_BLOCK:
            raise RuntimeError(f"vec0 chunk_size {size} != 1024 (the reference never sets chunk_size)")
        v = np.unpackbits(np.frombuffer(validity, np.uint8), bitorder="little")[:size]
        if not v.any():
            continue                                    # a block without live rows never yields a candidate
        vec = np.frombuffer(vectors, np.float32)
        d = vec.size // size
        if dim is None:
            dim = d
            emb = np.empty((n_blocks * VEC0_BLOCK, dim), np.float32)
        elif d != dim:
            raise RuntimeError("inconsistent vector dimension across vec0 blocks")
        emb[n:n + size] = vec.reshape(size, d)
        valid[n:n + size] = v
        rowid[n:n + size] = np.frombuffer(rowid_blob, np.int64)[:size]
        n += size
    if emb is None:
        return empty
    # trailing empty slots of the last block carry no information
    last = int(np.nonzero(valid[:n])[0][-1]) + 1
    emb, valid, rowid = emb[:last], valid[:last], rowid[:last]
    # the two JOINs of semantic_search.py:262-279 as sorted-array lookups: chunks.id -> movie_id -> dense movie
    # index; a live row without a chunks row, or whose movie is gone, keeps -1 (it still occupies its place in
    # the KNN's top-K' and is dropped afterwards, as the inner JOINs drop it)
    movie_idx = np.full(last, -1, np.int32)
    if _table_exists(conn, "chunks"):
        cm = np.array(cur.execute("SELECT id, movie_id FROM chunks ORDER BY id").fetchall(), np.int64).reshape(-1, 2)
        if len(cm) and len(movie_ids):
            live = np.nonzero(valid)[0]
            cpos = np.searchsorted(cm[:, 0], rowid[live])
            ok = cpos < len(cm)
            ok[ok] &= cm[cpos[ok], 0] == rowid[live][ok]
            mids = cm[cpos[ok], 1]
            mpos = np.searchsorted(movie_ids, mids)
            okm = mpos < len(movie_ids)
            okm[okm] &= movie_ids[mpos[okm]] == mids[okm]
            movie_idx[live[ok]] = np.where(okm, mpos, -1).astype(np.int32)
    return EmbArrays(emb=emb, valid=None if valid.all() else valid, rowid=rowid, movie_idx=movie_idx,
                     movie_ids=movie_ids, dim=int(dim))


# ----------------------------------------------------------------------------- frozen sidecar (SURVEY §8f rank 1)
SIDECAR_VERSION = 3


def _md5(b: bytes) -> str:
    return hashlib.md5(b).hexdigest()


def _db_fingerprint(conn: sqlite3.Connection, db_path) -> dict:
    """What the reference's own sync-or-skip checks look at (basesearch_db.py:81-92,
    keyword_search.py:87-100, semantic_search.py:145-154) plus cheap CONTENT probes: both classes open the
    database in WAL mode, where an in-place rewrite by another connection (a forced re-embed with the same
    chunk count, not yet checkpointed) leaves the main file's size and mtime — and possibly the -wal size —
    unchanged.  So the fingerprint also carries the file header's change counter, the WAL header (its salts
    change at every WAL restart) and tail (any appended frame changes it), id / length sums, and a digest of
    the first and last vec0 vector blocks."""
    p = Path(db_path)
    st = p.stat()
    cur = conn.cursor()
    counts = {}
    for t in ("movies", "terms", "postings", "doclen", "chunks", f"{VEC_TABLE}_chunks"):
        counts[t] = cur.execute(f"SELECT COUNT(*) FROM {t}").fetchone()[0] if _table_exists(conn, t) else -1
    probes = {}
    if counts["movies"] > 0:
        probes["movies"] = list(cur.execute("SELECT MAX(id), SUM(id) FROM movies").fetchone())
    if counts["doclen"] > 0:
        probes["doclen"] = list(cur.execute("SELECT MAX(doc_id), SUM(length) FROM doclen").fetchone())
    if counts["postings"] > 0:
        probes["postings"] = list(cur.execute("SELECT MAX(rowid), SUM(length(positions)) FROM postings "
                                              "WHERE term_id = (SELECT MAX(term_id) FROM postings)").fetchone())
    if counts["chunks"] > 0:
        probes["chunks"] = list(cur.execute("SELECT MAX(id), SUM(movie_id) FROM chunks").fetchone())
    if counts[f"{VEC_TABLE}_chunks"] > 0 and _table_exists(conn, f"{VEC_TABLE}_vector_chunks00"):
        lo, hi = cur.execute(f"SELECT MIN(rowid), MAX(rowid) FROM {VEC_TABLE}_vector_chunks00").fetchone()
        dig = []
        for rid in sorted({lo, hi}):
            (blob,) = cur.execute(f"SELECT vectors FROM {VEC_TABLE}_vector_chunks00 WHERE rowid = ?", (rid,)).fetchone()
            dig.append(_md5(bytes(blob)))
        (val,) = cur.execute(f"SELECT group_concat(hex(validity)) FROM (SELECT validity FROM {VEC_TABLE}_chunks "
                             f"ORDER BY chunk_id DESC LIMIT 2)").fetchone()
        probes["vec0"] = dig + [_md5((val or "").encode())]
    header = b""
    try:
        with open(p, "rb") as fh:
            header = fh.read(100)
    except OSError:
        pass
    wal = Path(str(p) + "-wal")
    wal_sig = ""
    wal_size = 0
    if wal.exists():
        wal_size = wal.stat().st_size
        try:
            with open(wal, "rb") as fh:
                head = fh.read(32)
                fh.seek(max(0, wal_size - 8192))
                wal_sig = _md5(head + fh.read())
        except OSError:
            pass
    return {"version": SIDECAR_VERSION, "size": st.st_size, "mtime_ns": st.st_mtime_ns, "wal_size": wal_size,
            "wal_sig": wal_sig, "change_counter": header[24:28].hex(), "schema_cookie": header[40:44].hex(),
            "counts": counts, "probes": probes}


def part_fingerprint(full: dict, part: str) -> str:
    """What a LIVE handle's copy of ``part`` ('bm25' | 'emb') depends on: the row counts and content probes of
    that part's tables out of ``_db_fingerprint`` (the other part's build — HybridSearch builds the keyword tables,
    opens them, then builds the vectors — must not look like a change; file size / mtime / WAL state therefore
    stay out).  The mirrors compare it at every open: a database rebuilt in place while this process still holds
    its handle is re-exported and re-uploaded instead of being searched through the stale copy (the reference
    re-reads SQLite on every query and cannot go stale)."""
    tables = {"bm25": ("movies", "terms", "postings", "doclen"),
              "emb": ("movies", "chunks", f"{VEC_TABLE}_chunks")}[part]
    probes = {"bm25": ("movies", "doclen", "postings"), "emb": ("movies", "chunks", "vec0")}[part]
    return json.dumps({"counts": {t: full["counts"].get(t) for t in tables},
                       "probes": {k: full["probes"].get(k) for k in probes}}, sort_keys=True)


def sidecar_path(db_path, part: str) -> Path:
    return Path(str(db_path) + f".rse-{part}.npz")


def emb_matrix_path(db_path) -> Path:
    """The embedding matrix of the 'emb' sidecar: a raw .npy of its own, so a later open MEMORY-MAPS it
    (np.load(mmap_mode="r")) instead of reading gigabytes into anonymous memory — rse_load_embeddings then
    copies to the device straight out of the page cache."""
    return Path(str(db_path) + ".rse-emb.f32.npy")


def load_or_export(conn: sqlite3.Connection, db_path, part: str, use_cache: bool = True, fingerprint: dict | None = None):
    """part = 'bm25' | 'emb'.  Exports once and keeps an .npz next to the database (plus, for 'emb', the
    matrix as a memory-mappable .npy); a later open whose fingerprint matches loads the arrays without
    touching the big tables.  ``fingerprint`` = a ``_db_fingerprint`` the caller has just taken (it counts the
    big tables: once per open is enough)."""
    exporter = {"bm25": export_bm25, "emb": export_embeddings}[part]
    if not use_cache:
        return exporter(conn)
    fp = json.dumps(fingerprint if fingerprint is not None else _db_fingerprint(conn, db_path), sort_keys=True)
    sc = sidecar_path(db_path, part)
    if sc.exists():
        try:
            with np.load(sc, allow_pickle=False) as z:
                if str(z["fingerprint"]) == fp:
                    if part == "bm25":
                        terms = z["terms"].tolist()
                        return Bm25Arrays(indptr=z["indptr"], doc_idx=z["doc_idx"], tf=z["tf"], df=z["df"], dl=z["dl"],
                                          doc_ids=z["doc_ids"], n_movies=int(z["n_movies"]), avgdl=float(z["avgdl"]),
                                          term_row={t: i for i, t in enumerate(terms)})
                    valid = z["valid"] if int(z["has_valid"]) else None
                    emb = np.load(emb_matrix_path(db_path), mmap_mode="r")
                    if emb.dtype != np.float32 or list(emb.shape) != z["emb_shape"].tolist():
                        raise ValueError("embedding matrix does not belong to this sidecar")
                    return EmbArrays(emb=emb, valid=valid, rowid=z["rowid"], movie_idx=z["movie_idx"],
                                     movie_ids=z["movie_ids"], dim=int(z["dim"]))
                logger.info("sidecar %s is stale (the database changed): re-exporting", sc)
        except Exception as e:                        # unreadable sidecar → re-export, but say so
            logger.warning("sidecar %s rejected (%s: %s): re-exporting", sc, type(e).__name__, e)
    arr = exporter(conn)
    write_sidecar(db_path, part, arr, fp)
    return arr


def write_sidecar(db_path, part: str, arr, fp: str) -> None:
    """The sidecar of ``part`` for the arrays ``arr`` of the database whose fingerprint (json) is ``fp``."""
    sc = sidecar_path(db_path, part)

    def atomic(path: Path, write) -> None:
        # tmp + os.replace: a concurrent opener sees the old file or the new one, never a half-written one
        tmp = path.with_name(path.name + f".tmp{os.getpid()}")
        try:
            with open(tmp, "wb") as fh:
                write(fh)
            os.replace(tmp, path)
        finally:
            if tmp.exists():
                tmp.unlink()

    try:
        if part == "bm25":
            terms = np.array([t for t, _ in sorted(arr.term_row.items(), key=lambda kv: kv[1])], dtype=np.str_)
            atomic(sc, lambda fh: np.savez(fh, fingerprint=np.str_(fp), indptr=arr.indptr, doc_idx=arr.doc_idx, tf=arr.tf,
                                           df=arr.df, dl=arr.dl, doc_ids=arr.doc_ids, n_movies=np.int64(arr.n_movies),
                                           avgdl=np.float64(arr.avgdl), terms=terms))
        else:
            # the matrix first, the .npz (which carries the fingerprint) last: it is the commit marker.  The old
            # .npz goes first so that no opener can pair the OLD fingerprint with the NEW matrix.
            if sc.exists():
                sc.unlink()
            atomic(emb_matrix_path(db_path), lambda fh: np.save(fh, np.ascontiguousarray(arr.emb, dtype=np.float32)))
            atomic(sc, lambda fh: np.savez(fh, fingerprint=np.str_(fp), emb_shape=np.asarray(arr.emb.shape, np.int64),
                                           has_valid=np.int64(arr.valid is not None),
                                           valid=arr.valid if arr.valid is not None else np.zeros(0, np.uint8),
                                           rowid=arr.rowid, movie_idx=arr.movie_idx, movie_ids=arr.movie_ids,
                                           dim=np.int64(arr.dim)))
    except OSError as e:
        logger.info("sidecar for %s not written (%s): read-only location?", db_path, e)


# ----------------------------------------------------------------------------- writer (reference on-disk format)
def _init_schema(conn: sqlite3.Connection) -> None:
    cur = conn.cursor()
    cur.execute("CREATE TABLE IF NOT EXISTS movies (id INTEGER PRIMARY KEY, title TEXT NOT NULL, description TEXT NOT NULL)")
    cur.execute("CREATE TABLE IF NOT EXISTS terms (id INTEGER PRIMARY KEY, term TEXT UNIQUE NOT NULL)")
    cur.execute("CREATE TABLE IF NOT EXISTS postings (term_id INTEGER NOT NULL, doc_id INTEGER NOT NULL, "
                "positions TEXT NOT NULL, PRIMARY KEY (term_id, doc_id))")
    cur.execute("CREATE TABLE IF NOT EXISTS doclen (doc_id INTEGER PRIMARY KEY, length INTEGER NOT NULL)")
    cur.execute("CREATE TABLE IF NOT EXISTS chunks (id INTEGER PRIMARY KEY, movie_id INTEGER NOT NULL, "
                "chunk_index INTEGER NOT NULL, max_chunk_size INTEGER NOT NULL, overlap INTEGER NOT NULL)")
    conn.commit()


def write_keyword_index(conn: sqlite3.Connection, docs: Sequence[dict], tokenizer: Tokenizer) -> None:
    """The tables KeywordSearch._rebuild_index fills (keyword_search.py:102-177): tokens =
    title + ["[TITLE_END]"] + body (:132), doclen counts the sentinel (:133), positions JSON (:169)."""
    cur = conn.cursor()
    cur.execute("DELETE FROM postings"); cur.execute("DELETE FROM terms"); cur.execute("DELETE FROM doclen")
    t_toks = tokenizer([d["title"] for d in docs])
    b_toks = tokenizer([d["description"] for d in docs])
    term_id: Dict[str, int] = {}
    post_rows, dl_rows = [], []
    for d, tt, bt in zip(docs, t_toks, b_toks):
        doc_id = int(d["id"])
        toks = list(tt) + [TITLE_END_TOKEN] + list(bt)
        dl_rows.append((doc_id, len(toks)))
        positions: Dict[str, List[int]] = {}
        for pos, tok in enumerate(toks):
            positions.setdefault(tok, []).append(pos)
        for tok, ps in positions.items():
            tid = term_id.setdefault(tok, len(term_id) + 1)
            post_rows.append((tid, doc_id, json.dumps(ps)))
    cur.executemany("INSERT INTO terms(id, term) VALUES (?, ?)", [(i, t) for t, i in term_id.items()])
    cur.executemany("INSERT INTO doclen(doc_id, length) VALUES (?, ?)", dl_rows)
    cur.executemany("INSERT INTO postings(term_id, doc_id, positions) VALUES (?, ?, ?)", post_rows)
    conn.commit()


def plan_chunks(movies: Sequence[tuple], max_chunk_size: int, overlap: int):
    """semantic_search.py:164-188: movies ORDER BY id, chunk ids 0,1,2,… contiguous per movie,
    title first, description windows joined without a separator.  Returns (rows, texts)."""
    rows, texts = [], []
    cid = 0
    for movie_id, title, description in movies:
        rows.append((cid, int(movie_id), 0, max_chunk_size, overlap)); texts.append(title); cid += 1
        for li, sent in enumerate(sentence_chunks(description, max_chunk_size, overlap), start=1):
            rows.append((cid, int(movie_id), li, max_chunk_size, overlap)); texts.append("".join(sent)); cid += 1
    return rows, texts


def write_vec0_shadow(conn: sqlite3.Connection, rowids: np.ndarray, emb: np.ndarray, table: str = VEC_TABLE) -> None:
    """Store vectors exactly where vec0 would after inserting ``rowids`` in order into an empty
    table: block i // 1024, slot i % 1024 (SURVEY App. A.2 / C).

    NOT a sqlite-vec writer: only the three shadow tables this package reads are created — there is no
    ``chunk_embeddings`` virtual-table entry and no ``_info`` table, so the reference (whose
    ``CREATE VIRTUAL TABLE IF NOT EXISTS`` would collide with the existing shadow tables) cannot open the
    result.  It exists to freeze synthetic corpora / precomputed embeddings for tests and benches; the file is
    marked in ``rse_meta`` so tools can tell, and SemanticSearch only uses it for a build when asked
    explicitly (``fallback_build=True``)."""
    cur = conn.cursor()
    cur.execute("CREATE TABLE IF NOT EXISTS rse_meta (key TEXT PRIMARY KEY, value TEXT)")
    cur.execute("INSERT OR REPLACE INTO rse_meta(key, value) VALUES ('vec0_shadow_writer', "
                "'rag_search_engine_b200.store.write_vec0_shadow: GPU-only database, not openable by sqlite-vec')")
    cur.execute(f"DROP TABLE IF EXISTS {table}_chunks")
    cur.execute(f"DROP TABLE IF EXISTS {table}_vector_chunks00")
    cur.execute(f"DROP TABLE IF EXISTS {table}_rowids")
    cur.execute(f"CREATE TABLE {table}_chunks (chunk_id INTEGER PRIMARY KEY AUTOINCREMENT, size INTEGER NOT NULL, "
                f"validity BLOB NOT NULL, rowids BLOB NOT NULL)")
    cur.execute(f"CREATE TABLE {table}_vector_chunks00 (rowid INTEGER PRIMARY KEY, vectors BLOB NOT NULL)")
    cur.execute(f"CREATE TABLE {table}_rowids (rowid INTEGER PRIMARY KEY AUTOINCREMENT, id, chunk_id INTEGER, "
                f"chunk_offset INTEGER)")
    emb = np.ascontiguousarray(emb, np.float32)
    n, dim = emb.shape
    for b0 in range(0, n, VEC0_BLOCK):
        b1 = min(n, b0 + VEC0_BLOCK)
        cnt = b1 - b0
        vec = np.zeros((VEC0_BLOCK, dim), np.float32); vec[:cnt] = emb[b0:b1]
        rid = np.zeros(VEC0_BLOCK, np.int64); rid[:cnt] = rowids[b0:b1]
        bits = np.zeros(VEC0_BLOCK, np.uint8); bits[:cnt] = 1
        chunk_id = b0 // VEC0_BLOCK + 1
        cur.execute(f"INSERT INTO {table}_chunks(chunk_id, size, validity, rowids) VALUES (?, ?, ?, ?)",
                    (chunk_id, VEC0_BLOCK, np.packbits(bits, bitorder="little").tobytes(), rid.tobytes()))
        cur.execute(f"INSERT INTO {table}_vector_chunks00(rowid, vectors) VALUES (?, ?)", (chunk_id, vec.tobytes()))
        cur.executemany(f"INSERT INTO {table}_rowids(rowid, id, chunk_id, chunk_offset) VALUES (?, NULL, ?, ?)",
                        [(int(rowids[i]), chunk_id, i - b0) for i in range(b0, b1)])
    conn.commit()


def write_reference_db(db_path, docs: Sequence[dict], tokenizer: Tokenizer,
                       embed: Optional[Callable[[List[str]], np.ndarray]] = None, max_chunk_size: int = 3,
                       overlap: int = 1) -> Path:
    """Create a database in the reference's on-disk format from ``docs`` = [{id,title,description}].
    ``embed(texts) -> [n, dim] float32`` freezes the chunk embeddings (None: keyword tables only)."""
    db_path = Path(db_path)
    db_path.parent.mkdir(parents=True, exist_ok=True)
    conn = sqlite3.connect(db_path)
    try:
        _init_schema(conn)
        cur = conn.cursor()
        cur.execute("DELETE FROM movies")
        cur.executemany("INSERT INTO movies(id, title, description) VALUES (?, ?, ?)",
                        [(int(d["id"]), d["title"], d["description"]) for d in docs])
        conn.commit()
        write_keyword_index(conn, docs, tokenizer)
        if embed is not None:
            movies = cur.execute("SELECT id, title, description FROM movies ORDER BY id").fetchall()
            rows, texts = plan_chunks(movies, max_chunk_size, overlap)
            cur.execute("DELETE FROM chunks")
            cur.executemany("INSERT INTO chunks(id, movie_id, chunk_index, max_chunk_size, overlap) VALUES (?,?,?,?,?)", rows)
            emb = np.asarray(embed(texts), np.float32)
            write_vec0_shadow(conn, np.array([r[0] for r in rows], np.int64), emb)
        conn.commit()
    finally:
        conn.close()
    return db_path
