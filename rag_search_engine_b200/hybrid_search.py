"""HybridSearch — drop-in for rag_search_engine.utils.hybrid_search.HybridSearch with the
fusion step (and, through the retrievers, BM25 + KNN) on the B200.

The seam is the reference's own (hybrid_search.py:41-54, :70, :88): the two retrievers are
looked up by MODULE-GLOBAL name at construction time, only ``.search(query, k=)``,
``.query_top_k(query_text=, k=)`` and ``.close()`` are called on them, and the reference's unit
tests swap them with ``monkeypatch.setattr(module, "KeywordSearch", Dummy)``
(tests/test_hybrid_search.py:73-76) — which works on this module too.  Whatever the retrievers
return is fused by ``rse_fuse_weighted`` / ``rse_fuse_rrf`` (min-max / RRF arithmetic and the
CPython-set tie order reproduced on the device).  When both retrievers are the GPU ones,
``*_batch`` runs the whole pipeline on the device in one call (``rse_hybrid``).
"""
from __future__ import annotations

import itertools
import logging
import time
from pathlib import Path
from typing import Any, Dict, List, Optional, Sequence

import numpy as np

from . import _lib, runtime
from .encoder import DeviceWordPiece, _utf8
from .keyword_search import DEFAULT_DB_PATH, KeywordSearch
from .semantic_search import SemanticSearch

logger = logging.getLogger(__name__)


class HybridSearch:
    def __init__(self, docs_path: Path | str | None = None, db_path: Path | str | None = None, *, force: bool = False,
                 max_chunk_size: int = 3, overlap: int = 1, device: int = 0, tie_mode: str = "reference",
                 cross_encoder=None, **retriever_kwargs) -> None:
        self.db_path = Path(db_path) if db_path else Path(DEFAULT_DB_PATH)
        self.device = device
        # rerank_method="cross_encoder": an object with .predict(pairs) (encoder.GpuCrossEncoder runs the reference's
        # TinyBERT cross-encoder on the same GPU); None = the reference's own CPU CrossEncoder (hybrid_search.py:296)
        self.cross_encoder = cross_encoder
        self.tie_mode = {"reference": _lib.TIE_REFERENCE, "id": _lib.TIE_BY_ID}[tie_mode]
        kw_extra = {k: v for k, v in retriever_kwargs.items() if k in ("tokenizer",)}
        sem_extra = {k: v for k, v in retriever_kwargs.items() if k in ("encoder", "fallback_build", "device_build")}
        if KeywordSearch.__module__.startswith(__package__):
            kw_extra["device"] = device
        if SemanticSearch.__module__.startswith(__package__):
            sem_extra["device"] = device
        # module-global lookup, exactly like hybrid_search.py:41-54
        self.keyword = KeywordSearch(docs_path=docs_path, db_path=self.db_path, force=force, **kw_extra)
        self.semantic = SemanticSearch(docs_path=docs_path, db_path=self.db_path, max_chunk_size=max_chunk_size,
                                       overlap=overlap, force=force, **sem_extra)
        self._index = runtime.acquire(self.db_path, device)      # fusion kernels (+ shared with GPU retrievers)
        self._closed = False

    @classmethod
    def from_loaded(cls, index: "_lib.Index", term_row: Dict[str, int], doc_ids, movie_ids, *, registry_key,
                    device: int = 0, tie_mode: str = "reference", cross_encoder=None) -> "HybridSearch":
        """The batch / stream entry points over a handle whose indexes are ALREADY in HBM (rse_load_bm25 +
        rse_load_embeddings / rse_attach_embeddings_dev done by the caller): for corpora that never lived in a
        SQLite file — synthetic benchmarks, a shard of a larger service.  The single-query text methods, which
        read titles from SQLite, are not available on such an object.  ``registry_key`` names the handle in
        ``runtime`` (any path-like string unique to it)."""
        from types import SimpleNamespace
        self = cls.__new__(cls)
        self.db_path = Path(registry_key)
        self.device = device
        self.tie_mode = {"reference": _lib.TIE_REFERENCE, "id": _lib.TIE_BY_ID}[tie_mode]
        kw = KeywordSearch.__new__(KeywordSearch)
        kw._arr = SimpleNamespace(term_row=term_row, doc_ids=np.ascontiguousarray(doc_ids, np.int64))
        kw._closed = True
        sem = SemanticSearch.__new__(SemanticSearch)
        sem._arr = SimpleNamespace(movie_ids=np.ascontiguousarray(movie_ids, np.int64),
                                   emb=np.zeros((int(index.n_rows), 0), np.float32))
        sem._closed = True
        self.keyword, self.semantic, self._index = kw, sem, index
        self.cross_encoder = cross_encoder
        runtime.adopt(self.db_path, device, index)
        self._closed = False
        return self

    # ---------------- wrappers (hybrid_search.py:57-88) ---------------- #
    def _bm25_search(self, query: str, limit: int) -> List[Dict[str, Any]]:
        return self.keyword.search(query, k=limit)

    def _semantic_search(self, query: str, limit: int) -> List[Dict[str, Any]]:
        return self.semantic.query_top_k(query_text=query, k=limit)

    # ---------------- fusion on the device ---------------- #
    def _fuse_inputs(self, bm25_hits, sem_hits, limit):
        L = max(1, min(limit, _lib.RSE_MAX_HYBRID_LIMIT))
        if limit > _lib.RSE_MAX_HYBRID_LIMIT:
            raise ValueError(f"limit {limit} exceeds the hybrid limit of {_lib.RSE_MAX_HYBRID_LIMIT}")
        # the retrievers are asked for k=limit; a plugged-in retriever may return more — the reference
        # would fuse all of them, so size the device call to what actually came back
        L = max(L, len(bm25_hits), len(sem_hits))
        if L > _lib.RSE_MAX_FUSE_LIMIT:
            raise ValueError(f"retriever returned more hits than the fusion kernel supports ({_lib.RSE_MAX_FUSE_LIMIT})")
        bid = np.full((1, L), -1, np.int64); bsc = np.zeros((1, L)); sid = np.full((1, L), -1, np.int64)
        sds = np.zeros((1, L))
        for j, h in enumerate(bm25_hits):
            bid[0, j] = int(h["id"]); bsc[0, j] = float(h["score"])
        for j, h in enumerate(sem_hits):
            sid[0, j] = int(h["movie_id"]); sds[0, j] = float(h["distance"])
        return L, bid, bsc, np.array([len(bm25_hits)], np.int32), sid, sds, np.array([len(sem_hits)], np.int32)

    # ---------------- weighted (hybrid_search.py:91-180) ---------------- #
    def weighted_search(self, query: str, alpha: float, limit: int = 5) -> List[Dict[str, Any]]:
        bm25_hits = self._bm25_search(query=query, limit=limit)
        sem_hits = self._semantic_search(query=query, limit=limit)
        if not bm25_hits and not sem_hits:
            return []
        L, bid, bsc, bc, sid, sds, sc = self._fuse_inputs(bm25_hits, sem_hits, limit)
        oid, ob, osem, osc, oc = self._index.fuse_weighted(L, alpha, bid, bsc, bc, sid, sds, sc, tie_mode=self.tie_mode)
        bm25_by_id = {int(h["id"]): h for h in bm25_hits}
        sem_by_id = {int(h["movie_id"]): h for h in sem_hits}
        results = []
        for j in range(min(int(oc[0]), limit)):
            doc_id = int(oid[0, j])
            b, s = bm25_by_id.get(doc_id, {}), sem_by_id.get(doc_id, {})
            results.append({"id": doc_id,
                            "title": b.get("title") or s.get("title") or "<unknown>",          # :155
                            "description": b.get("description") or s.get("description") or "",  # :156-158
                            "bm25": float(ob[0, j]), "semantic": float(osem[0, j]), "score": float(osc[0, j])})
        return results

    # ---------------- RRF (hybrid_search.py:183-379) ---------------- #
    def rrf_search(self, query: str, k: int = 60, limit: int = 10, rerank_method: str | None = None) -> List[Dict[str, Any]]:
        logger.debug("RRF search starting: query=%r, k=%s, limit=%d, rerank_method=%r", query, k, limit, rerank_method)
        bm25_hits = sorted(self._bm25_search(query=query, limit=limit), key=lambda h: h["score"], reverse=True)   # :220-224
        sem_hits = sorted(self._semantic_search(query=query, limit=limit), key=lambda h: h["distance"])          # :235-238
        results: List[Dict[str, Any]] = []
        if bm25_hits or sem_hits:
            # the reference sorts the FULL union before any truncation (rerankers see all of it)
            L, bid, bsc, bc, sid, sds, sc = self._fuse_inputs(bm25_hits, sem_hits, limit)
            n_union = len({int(h["id"]) for h in bm25_hits} | {int(h["movie_id"]) for h in sem_hits})
            Lout = max(L, min(n_union, _lib.RSE_MAX_FUSE_LIMIT))
            if Lout != L:
                pad = lambda a, fill: np.concatenate([a, np.full((1, Lout - L), fill, a.dtype)], 1)  # noqa: E731
                bid, bsc, sid, sds = pad(bid, -1), pad(bsc, 0.0), pad(sid, -1), pad(sds, 0.0)
            if n_union > _lib.RSE_MAX_FUSE_LIMIT:
                raise ValueError(f"union of retriever hits exceeds the fusion kernel's limit ({_lib.RSE_MAX_FUSE_LIMIT})")
            oid, osc, orb, ors, oc = self._index.fuse_rrf(Lout, k, bid, bsc, bc, sid, sds, sc, tie_mode=self.tie_mode)
            bm25_meta = {int(h["id"]): h for h in bm25_hits}
            sem_meta = {int(h["movie_id"]): h for h in sem_hits}
            for j in range(int(oc[0])):
                doc_id = int(oid[0, j])
                meta = bm25_meta.get(doc_id) or sem_meta.get(doc_id) or {}                 # :257
                results.append({"id": doc_id, "title": meta.get("title", "<unknown>"),
                                "description": meta.get("description", ""), "score": float(osc[0, j]),
                                "bm25_rank": None if orb[0, j] < 0 else int(orb[0, j]),
                                "sem_rank": None if ors[0, j] < 0 else int(ors[0, j])})
        logger.debug("RRF base results (pre-rerank, top %d): %s", len(results), results)

        # ---- rerank branches run on the host on top of the GPU results (out of scope, SURVEY §2 #3) ----
        if rerank_method == "cross_encoder":                                               # :279-312
            pairs = []
            for idx, doc in enumerate(results, start=1):
                doc["rrf_rank"] = idx
                pairs.append([query, f"{doc.get('title', '')} - {doc.get('document') or doc.get('description', '')}"])
            if pairs:
                ce = getattr(self, "cross_encoder", None)
                if ce is None:
                    from sentence_transformers import CrossEncoder  # type: ignore
                    ce = CrossEncoder("cross-encoder/ms-marco-TinyBERT-L2-v2")
                scores = ce.predict(pairs)
                for doc, score in zip(results, scores):
                    doc["cross_encoder_score"] = float(score)
                results.sort(key=lambda d: (d.get("cross_encoder_score", 0.0), d["score"]), reverse=True)
            return results[:limit]
        if rerank_method in ("individual", "batch"):                                       # :315-367
            from rag_search_engine.llm.gemini import Gemini  # type: ignore  (network LLM: reference package)
            gi = Gemini()
            if rerank_method == "individual":
                for idx, doc in enumerate(results):
                    if idx > 0:
                        time.sleep(3)
                    doc["rerank_score"] = gi.rerank_document(query, doc, rerank_method)
                results.sort(key=lambda r: (r.get("rerank_score", 0.0), r["score"]), reverse=True)
            else:
                ranked_ids = gi.rerank_batch(query, results, rerank_method)
                rank_map = {doc_id: idx for idx, doc_id in enumerate(ranked_ids, start=1)}
                for doc in results:
                    doc["rerank_rank"] = rank_map.get(doc["id"])
                results.sort(key=lambda r: (r.get("rerank_rank") is None, r.get("rerank_rank") or 1e9))
            return results[:limit]
        if rerank_method is not None:                                                      # :370-373
            logger.warning("Unknown rerank_method=%r, using base RRF only", rerank_method)
        return results[:limit]                                                             # :379

    # ---------------- fully on-device batch path ---------------- #
    def _gpu_retrievers(self) -> bool:
        return isinstance(self.keyword, KeywordSearch) and isinstance(self.semantic, SemanticSearch) and \
            type(self.keyword).__module__.startswith(__package__) and type(self.semantic).__module__.startswith(__package__)

    def _ensure_id_tables(self):
        reg = runtime.parts(self.db_path, self.device)
        if "ids" not in reg:
            self._index.set_id_tables(self.keyword._arr.doc_ids, self.semantic._arr.movie_ids)
            reg["ids"] = True

    def _hybrid_batch(self, mode, param, token_lists, query_vecs, limit, knn_multiplier, k1, b):
        if not self._gpu_retrievers():
            raise RuntimeError("*_batch needs the GPU KeywordSearch and SemanticSearch of this package")
        kw, sem = self.keyword, self.semantic
        tok_indptr, rows = kw._term_rows(token_lists)
        nq = len(tok_indptr) - 1
        if sem._arr.emb.shape[0] == 0 or len(kw._arr.doc_ids) == 0:
            # one side has no index (keyword-only or embeddings-only database): the reference degrades to the
            # other retriever (tests/test_hybrid_search.py:94-124); same here, still on the device
            L = int(limit)
            bid = np.full((nq, L), -1, np.int64); bsc = np.zeros((nq, L)); bc = np.zeros(nq, np.int32)
            sid = np.full((nq, L), -1, np.int64); sds = np.zeros((nq, L)); sc = np.zeros(nq, np.int32)
            if len(kw._arr.doc_ids):
                score, doc, bc = self._index.bm25(tok_indptr, rows, L, k1, b)
                bid = np.where(doc >= 0, kw._arr.doc_ids[np.clip(doc, 0, None)], -1)
                bsc = score
            if sem._arr.emb.shape[0]:
                dist, _rowid, movie, sc = self._index.knn_movies(query_vecs, L, max(L * knn_multiplier, L))
                sid = np.where(movie >= 0, sem._arr.movie_ids[np.clip(movie, 0, None)], -1)
                sds = dist.astype(np.float64)
            if mode == 0:
                oid, osc, orb, ors, oc = self._index.fuse_rrf(L, param, bid, bsc, bc, sid, sds, sc, tie_mode=self.tie_mode)
                return oid, osc, orb.astype(np.float64), ors.astype(np.float64), oc
            oid, ob, osem, osc, oc = self._index.fuse_weighted(L, param, bid, bsc, bc, sid, sds, sc, tie_mode=self.tie_mode)
            return oid, osc, ob, osem, oc
        self._ensure_id_tables()
        return self._index.hybrid(mode, param, limit, query_vecs, tok_indptr, rows, knn_multiplier=knn_multiplier,
                                  k1=k1, b=b, tie_mode=self.tie_mode)

    @staticmethod
    def _unpack_rrf(res, nq):
        """[{id, score, bm25_rank, sem_rank}] per query from the packed arrays.  ONE flat comprehension over bulk
        ``tolist()`` columns and slicing afterwards: per-element numpy indexing cost 4x the device step for a
        256-query batch, nested per-query comprehensions 2x (bench.py e2e_python)."""
        oid, osc, oa, ob, oc = res
        ra = oa.astype(np.int64).astype(object); ra[oa < 0] = None
        rb = ob.astype(np.int64).astype(object); rb[ob < 0] = None
        flat = [{"id": i, "score": s, "bm25_rank": a, "sem_rank": b_}
                for i, s, a, b_ in zip(oid.ravel().tolist(), osc.ravel().tolist(), ra.ravel().tolist(), rb.ravel().tolist())]
        L = oid.shape[1] if oid.ndim == 2 else 0
        cnt = oc.tolist()
        return [flat[q * L:q * L + cnt[q]] for q in range(nq)]

    def rrf_search_batch(self, token_lists, query_vecs, k=60, limit: int = 10, knn_multiplier: int = 10,
                         k1: float = 1.5, b: float = 0.75, as_arrays: bool = False, rerank_method: str | None = None,
                         rerank_query_ids=None):
        """[{id, score, bm25_rank, sem_rank}] per query; BM25 + KNN + aggregation + RRF in one device call.
        ``as_arrays=True`` returns the packed result instead — (id int64, score, bm25_rank, sem_rank as float64
        with -1 = None, each [nq, limit]; count int32[nq]) — for callers that do not want Python objects.

        ``rerank_method="cross_encoder"`` ranks like ``rrf_search(q, rerank_method="cross_encoder")`` for the whole
        batch on the device (``self.cross_encoder``, a ``GpuCrossEncoder`` on this object's handle, after
        ``load_rerank_documents``): ``rerank_query_ids`` are the cross-encoder tokenizer's ids of each query without
        special tokens (``cross_encoder.tokenize(texts)``), or the query strings, which that tokenizer then
        tokenizes.  Hits are {id, score, bm25_rank, sem_rank, rrf_rank,
        cross_encoder_score}; ``as_arrays=True`` gives (id, score, bm25_rank, sem_rank, rrf_rank, cross_encoder_score,
        count) with int32 ranks (-1 = None)."""
        if rerank_method is not None:
            ce = self._rerank_encoder(rerank_method)
            if not self._gpu_retrievers():
                raise RuntimeError("*_batch needs the GPU KeywordSearch and SemanticSearch of this package")
            self._ensure_id_tables()
            tok_indptr, rows = self.keyword._term_rows(token_lists)
            if len(tok_indptr) == 1:
                if not as_arrays:
                    return []
                z = [np.zeros((0, limit), t) for t in (np.int64, np.float64, np.int32, np.int32, np.int32, np.float32)]
                return (*z, np.zeros(0, np.int32))
            self._index.hybrid_stage(query_vecs, tok_indptr, rows)
            return self._rerank_staged(ce, len(tok_indptr) - 1, rerank_query_ids, k, limit, knn_multiplier, k1, b,
                                       as_arrays)
        res = self._hybrid_batch(0, float(k), token_lists, query_vecs, limit, knn_multiplier, k1, b)
        return res if as_arrays else self._unpack_rrf(res, len(res[4]))

    def weighted_search_batch(self, token_lists: Sequence[Sequence[str]], query_vecs, alpha: float, limit: int = 5,
                              knn_multiplier: int = 10, k1: float = 1.5, b: float = 0.75):
        oid, osc, oa, ob, oc = self._hybrid_batch(1, float(alpha), token_lists, query_vecs, limit, knn_multiplier, k1, b)
        return [[{"id": int(oid[q, j]), "bm25": float(oa[q, j]), "semantic": float(ob[q, j]),
                  "score": float(osc[q, j])} for j in range(oc[q])] for q in range(len(oc))]

    def rrf_search_texts(self, token_lists, encoder_ids, encoder, k=60, limit: int = 10, knn_multiplier: int = 10,
                         k1: float = 1.5, b: float = 0.75, as_arrays: bool = False, rerank_method: str | None = None,
                         rerank_query_ids=None):
        """Text in: the query vectors are produced by ``encoder`` (encoder.GpuSentenceEncoder) ON THE DEVICE and
        handed to the hybrid step there (``rse_encode_dev`` -> ``rse_hybrid_stage_dev``): no host hop for the
        vectors.  ``token_lists`` are the BM25 tokens of the queries (the reference's ``preprocess`` output),
        ``encoder_ids`` the encoder's token ids ([CLS] ... [SEP]) of the same queries, or the query strings
        themselves (tokenized by the encoder's tokenizer; on the device with a ``DeviceWordPiece``).  ``rerank_method``
        / ``rerank_query_ids`` as in ``rrf_search_batch``; given query strings, ``rerank_query_ids`` may be omitted
        and the cross-encoder's tokenizer makes them from the strings."""
        import torch
        ce = self._rerank_encoder(rerank_method) if rerank_method is not None else None
        if not self._gpu_retrievers():
            raise RuntimeError("rrf_search_texts needs the GPU KeywordSearch and SemanticSearch of this package")
        self._ensure_id_tables()
        tok_indptr, rows = self.keyword._term_rows(token_lists)
        nq = len(tok_indptr) - 1
        buf = getattr(self, "_qvec_dev", None)
        if buf is None or buf.shape[0] < nq:
            buf = self._qvec_dev = torch.empty((max(nq, 256), self._index.dim), dtype=torch.float32,
                                               device=torch.device("cuda", self.device))
        texts = len(encoder_ids) > 0 and all(isinstance(x, str) for x in encoder_ids)
        if texts:
            n = encoder.encode_texts_dev(encoder_ids, buf.data_ptr())
            if ce is not None and rerank_query_ids is None:
                rerank_query_ids = list(encoder_ids)
        else:
            n = encoder.encode_ids_dev(encoder_ids, buf.data_ptr())
        if n != nq:
            raise ValueError("token_lists and encoder_ids describe different numbers of queries")
        self._index.hybrid_stage_dev(nq, buf.data_ptr(), tok_indptr, rows)
        if ce is not None:
            return self._rerank_staged(ce, nq, rerank_query_ids, k, limit, knn_multiplier, k1, b, as_arrays)
        self._index.hybrid_run(0, float(k), limit, knn_multiplier=knn_multiplier, k1=k1, b=b, tie_mode=self.tie_mode)
        res = self._index.hybrid_fetch(limit)
        return res if as_arrays else self._unpack_rrf(res, nq)

    # ---------------- cross-encoder rerank of a batch (hybrid_search.py:279-312) on the device ---------------- #
    def load_rerank_documents(self, ids=None, token_lists=None) -> int:
        """Upload the cross-encoder's token ids of every document text, ``f"{title} - {description}"``, the strings
        ``rrf_search`` pairs with the query (an id without a ``movies`` row is ``"<missing> - "``, what
        ``KeywordSearch.search`` reports for it).  Without arguments the texts are read from this object's SQLite
        database for every id the two retrievers can return and tokenised with ``self.cross_encoder.tokenize``;
        ``ids`` + ``token_lists`` (ids without special tokens, per id) upload a ready store instead — the only form
        an object made by ``from_loaded`` has.  Returns the number of documents."""
        if ids is None:
            ce = self._rerank_encoder("cross_encoder")
            universe = np.union1d(np.asarray(self.keyword._arr.doc_ids, np.int64),
                                  np.asarray(self.semantic._arr.movie_ids, np.int64))
            import sqlite3
            conn = sqlite3.connect(self.db_path)
            try:
                rows = {int(i): (t, d) for i, t, d in conn.execute("SELECT id, title, description FROM movies")}
            finally:
                conn.close()
            texts = []
            for i in universe.tolist():
                title, desc = rows.get(i, ("<missing>", ""))
                texts.append(f"{title} - {desc or ''}")
            tok = ce.tokenizer
            if isinstance(tok, DeviceWordPiece) and not tok.host_routed(texts):
                # tokenized on the device straight into the store (universe is ascending): no host id lists
                data, offs = _utf8(texts)
                self._index.rerank_docs_load_texts(tok.slot, universe, data, offs)
                return len(universe)
            ids, token_lists = universe, ce.tokenize(texts)
        ids = np.asarray(ids, np.int64)
        if len(token_lists) != len(ids):
            raise ValueError("ids and token_lists differ in length")
        order = np.argsort(ids, kind="stable")
        lens = np.fromiter((len(token_lists[i]) for i in order.tolist()), np.int64, count=len(ids))
        indptr = np.zeros(len(ids) + 1, np.int64)
        np.cumsum(lens, out=indptr[1:])
        tokens = np.fromiter(itertools.chain.from_iterable(token_lists[i] for i in order.tolist()), np.int32,
                             count=int(indptr[-1]))
        self._index.rerank_docs_load(ids[order], indptr, tokens)
        return len(ids)

    def _rerank_encoder(self, rerank_method):
        if rerank_method != "cross_encoder":
            raise ValueError(f"rerank_method must be None or 'cross_encoder' for a batch, not {rerank_method!r}")
        ce = getattr(self, "cross_encoder", None)
        if ce is None or not hasattr(ce, "index") or not hasattr(ce, "cls_id"):
            raise RuntimeError("the batched rerank needs HybridSearch(cross_encoder=GpuCrossEncoder(...))")
        if ce.index is not self._index:
            raise ValueError("the cross-encoder lives on another handle than the hybrid index: create it on "
                             "runtime.acquire(db_path, device) (or the index given to from_loaded)")
        if ce.activation not in (None, "sigmoid"):
            raise ValueError(f"unsupported cross-encoder activation {ce.activation!r}")
        return ce

    def _rerank_staged(self, ce, nq, rerank_query_ids, k, limit, knn_multiplier, k1, b, as_arrays):
        if rerank_query_ids is None or len(rerank_query_ids) != nq:
            raise ValueError("rerank_query_ids must hold the cross-encoder token ids of every query")
        if all(isinstance(x, str) for x in rerank_query_ids):
            rerank_query_ids = ce.tokenize(rerank_query_ids)
        q_ptr = np.zeros(nq + 1, np.int32)
        np.cumsum([len(x) for x in rerank_query_ids], out=q_ptr[1:])
        q_ids = np.fromiter(itertools.chain.from_iterable(rerank_query_ids), np.int32, count=int(q_ptr[-1]))
        self._index.hybrid_rerank_run(ce.slot, float(k), limit, q_ptr, q_ids, cls_id=ce.cls_id, sep_id=ce.sep_id,
                                      max_length=ce.max_length, activation=int(ce.activation == "sigmoid"),
                                      knn_multiplier=knn_multiplier, k1=k1, b=b, tie_mode=self.tie_mode)
        res = self._index.hybrid_rerank_fetch(limit)
        return res if as_arrays else self._unpack_rerank(res, nq)

    @staticmethod
    def _unpack_rerank(res, nq):
        """[{id, score, bm25_rank, sem_rank, rrf_rank, cross_encoder_score}] per query (as _unpack_rrf)."""
        oid, osc, orb, ors, orr, oce, oc = res
        ra = orb.astype(object); ra[orb < 0] = None
        rb = ors.astype(object); rb[ors < 0] = None
        flat = [{"id": i, "score": s, "bm25_rank": a, "sem_rank": b_, "rrf_rank": r, "cross_encoder_score": c}
                for i, s, a, b_, r, c in zip(oid.ravel().tolist(), osc.ravel().tolist(), ra.ravel().tolist(),
                                             rb.ravel().tolist(), orr.ravel().tolist(), oce.ravel().tolist())]
        L = oid.shape[1] if oid.ndim == 2 else 0
        cnt = oc.tolist()
        return [flat[q * L:q * L + cnt[q]] for q in range(nq)]

    def rrf_search_stream(self, batches, k=60, limit: int = 10, knn_multiplier: int = 10, k1: float = 1.5,
                          b: float = 0.75, as_arrays: bool = False):
        """Serving loop over an iterable of ``(token_lists, query_vecs)`` batches: yields what ``rrf_search_batch``
        returns for each batch, in order, while the NEXT batch is already enqueued on the device
        (``rse_hybrid_submit`` / ``rse_hybrid_collect``, two batches in flight) — the device never waits for the host
        to stage inputs or unpack results.  ``token_lists`` may be the pre-flattened ``(tok_indptr, tokens)`` pair
        ``KeywordSearch._term_rows`` accepts; ``as_arrays`` as in ``rrf_search_batch``."""
        if not self._gpu_retrievers():
            raise RuntimeError("*_stream needs the GPU KeywordSearch and SemanticSearch of this package")
        kw = self.keyword
        self._ensure_id_tables()

        def unpack(res, nq):
            return res if as_arrays else self._unpack_rrf(res, nq)

        def n_queries(tl):
            return len(tl[0]) - 1 if isinstance(tl, tuple) else len(tl)

        pending = None                                           # (ticket, nq) of the batch in flight
        try:
            for token_lists, query_vecs in batches:
                if n_queries(token_lists) == 0:
                    if pending is not None:
                        done, pending = pending, None
                        yield unpack(self._index.hybrid_collect(done[0]), done[1])
                    yield []
                    continue
                tok_indptr, rows = kw._term_rows(token_lists)
                ticket = self._index.hybrid_submit(0, float(k), limit, query_vecs, tok_indptr, rows,
                                                   knn_multiplier=knn_multiplier, k1=k1, b=b, tie_mode=self.tie_mode)
                done, pending = pending, (ticket, n_queries(token_lists))
                if done is not None:
                    yield unpack(self._index.hybrid_collect(done[0]), done[1])
            if pending is not None:
                done, pending = pending, None
                yield unpack(self._index.hybrid_collect(done[0]), done[1])
        finally:
            # a consumer that stops iterating early (GeneratorExit) or an exception between a submit and its
            # collect must not leave tickets in flight: the handle is shared per (db, device) and collects in
            # submission order, so a stale ticket would wedge every later stream call
            self._index.hybrid_drain()

    # ---------------- cleanup (hybrid_search.py:382-384) ---------------- #
    def close(self) -> None:
        self.keyword.close()
        self.semantic.close()
        if not self._closed:
            self._closed = True
            runtime.release(self.db_path, self.device)
