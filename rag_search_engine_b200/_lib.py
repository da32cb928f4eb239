"""ctypes binding of librse.so (include/rse.h).

This is exactly the stub a reference maintainer would add (INTEGRATION.md).  It
fails loudly when the CUDA library is missing or when no GPU is present — there
is no CPU fallback anywhere in this package.
"""
from __future__ import annotations

import ctypes
from ctypes import POINTER, c_char_p, c_double, c_float, c_int32, c_int64, c_uint8, c_uint32, c_void_p
from pathlib import Path

import numpy as np

_HERE = Path(__file__).resolve().parent
LIB_PATH = _HERE / "csrc" / "librse.so"

RSE_OK = 0
RSE_ERR_UNSUPPORTED = -4
RSE_MAX_KPRIME = 4096
RSE_MAX_BM25_K = 512
RSE_MAX_FUSE_LIMIT = 1024
RSE_MAX_HYBRID_LIMIT = 512
RSE_MAX_RERANK_LIMIT = 128
RSE_MAX_QUERY_TOKENS = 255
TIE_REFERENCE = 0
TIE_BY_ID = 1


class RseError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"librse error {code}: {msg}")
        self.code = code


class RseStats(ctypes.Structure):
    _fields_ = [
        ("kernel_launches", c_int64),
        ("knn_scan_launches", c_int64),
        ("scan_ms_total", c_double),
        ("scan_launches_timed", c_int64),
        ("last_knn_total_ms", c_double),
        ("last_bm25_ms", c_double),
        ("last_fuse_ms", c_double),
        ("emb_rows", c_int64),
        ("emb_dim", c_int32),
        ("bm25_postings", c_int64),
        ("bm25_docs", c_int64),
        ("tc_filter_launches", c_int64),
        ("tc_queries", c_int64),
        ("tc_fallback_queries", c_int64),
        ("tc_second_chance_queries", c_int64),
        ("bm25_queries", c_int64),
        ("bm25_fallback_queries", c_int64),
        ("bm25_finalists", c_int64),
        ("bm25_candidates", c_int64),
        ("h2d_bytes", c_int64),
        ("d2h_bytes", c_int64),
    ]


class RseEncoderConfig(ctypes.Structure):
    """include/rse.h rse_encoder_config."""
    _fields_ = [("vocab_size", c_int32), ("hidden", c_int32), ("layers", c_int32), ("heads", c_int32),
                ("intermediate", c_int32), ("max_positions", c_int32), ("type_vocab", c_int32),
                ("ln_eps", c_float), ("head", c_int32)]


class RseClipConfig(ctypes.Structure):
    """include/rse.h rse_clip_config."""
    _fields_ = [("tower", c_int32), ("hidden", c_int32), ("layers", c_int32), ("heads", c_int32),
                ("intermediate", c_int32), ("projection_dim", c_int32), ("vocab_size", c_int32),
                ("max_positions", c_int32), ("image_size", c_int32), ("patch_size", c_int32),
                ("eos_token_id", c_int32), ("ln_eps", c_float)]


class RseImgprocCfg(ctypes.Structure):
    """include/rse.h rse_imgproc_cfg."""
    _fields_ = [("backend", c_int32), ("shortest_edge", c_int32), ("crop_height", c_int32), ("crop_width", c_int32),
                ("do_resize", c_int32), ("do_center_crop", c_int32), ("do_rescale", c_int32),
                ("do_normalize", c_int32), ("rescale_factor", c_double), ("mean", c_double * 3),
                ("std", c_double * 3)]


class RseWordpieceDesc(ctypes.Structure):
    """include/rse.h rse_wordpiece_desc."""
    _fields_ = [("cp_map", c_void_p), ("extra", c_void_p), ("n_extra", c_int32), ("cp_class", c_void_p),
                ("node_first", c_void_p), ("node_id", c_void_p), ("n_nodes", c_int32), ("edge_cp", c_void_p),
                ("edge_child", c_void_p), ("added", c_void_p), ("added_offsets", c_void_p), ("added_ids", c_void_p),
                ("n_added", c_int32), ("unk_id", c_int32), ("cls_id", c_int32), ("sep_id", c_int32),
                ("max_input_chars_per_word", c_int32)]


class RseBpeDesc(ctypes.Structure):
    """include/rse.h rse_bpe_desc."""
    _fields_ = [("cp_map", c_void_p), ("extra", c_void_p), ("n_extra", c_int32), ("cp_class", c_void_p),
                ("byte_ids", c_void_p), ("merges", c_void_p), ("merge_slots", c_int32), ("added", c_void_p),
                ("added_offsets", c_void_p), ("added_ids", c_void_p), ("n_added", c_int32), ("bos_id", c_int32),
                ("eos_id", c_int32)]


_SIGNATURES = {
    "rse_abi_version": (ctypes.c_int, []),
    "rse_create": (ctypes.c_int, [c_int32, POINTER(c_void_p)]),
    "rse_destroy": (None, [c_void_p]),
    "rse_last_error": (c_char_p, [c_void_p]),
    "rse_set_stream": (ctypes.c_int, [c_void_p, c_void_p]),
    "rse_use_own_stream": (ctypes.c_int, [c_void_p]),
    "rse_synchronize": (ctypes.c_int, [c_void_p]),
    "rse_load_embeddings": (ctypes.c_int, [c_void_p, POINTER(c_float), c_int64, c_int32, POINTER(c_uint8),
                                           POINTER(c_int64), POINTER(c_int32), c_int64]),
    "rse_attach_embeddings_dev": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_int32, c_void_p, c_void_p,
                                                 c_void_p, c_int64]),
    "rse_set_fma": (ctypes.c_int, [c_void_p, c_int32]),
    "rse_set_tc_mode": (ctypes.c_int, [c_void_p, c_int32]),
    "rse_set_bm25_mode": (ctypes.c_int, [c_void_p, c_int32]),
    "rse_knn": (ctypes.c_int, [c_void_p, POINTER(c_float), c_int32, c_int32, POINTER(c_float), POINTER(c_int64),
                               POINTER(c_int64), POINTER(c_int32), POINTER(c_int32)]),
    "rse_knn_movies": (ctypes.c_int, [c_void_p, POINTER(c_float), c_int32, c_int32, c_int32, POINTER(c_float),
                                      POINTER(c_int64), POINTER(c_int32), POINTER(c_int32)]),
    "rse_knn_movies_exact": (ctypes.c_int, [c_void_p, POINTER(c_float), c_int32, c_int32, POINTER(c_float),
                                            POINTER(c_int64), POINTER(c_int32), POINTER(c_int32), POINTER(c_int32)]),
    "rse_knn_local_dev": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "rse_set_defer_flags": (ctypes.c_int, [c_void_p, c_int32]),
    "rse_knn_flags_dev": (ctypes.c_int, [c_void_p, c_void_p]),
    "rse_knn_merge_movies_dev": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                                c_void_p, c_void_p, c_void_p]),
    "rse_load_bm25": (ctypes.c_int, [c_void_p, POINTER(c_int64), POINTER(c_uint32), POINTER(c_uint32),
                                     POINTER(c_int64), c_int64, c_int64, POINTER(c_uint32), c_int64, c_int64,
                                     c_double]),
    "rse_bm25": (ctypes.c_int, [c_void_p, POINTER(c_int32), POINTER(c_int32), c_int32, c_int32, c_double, c_double,
                                POINTER(c_double), POINTER(c_int32), POINTER(c_int32)]),
    "rse_fuse_weighted": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_double, c_int32, POINTER(c_int64),
                                         POINTER(c_double), POINTER(c_int32), POINTER(c_int64), POINTER(c_double),
                                         POINTER(c_int32), POINTER(c_int64), POINTER(c_double), POINTER(c_double),
                                         POINTER(c_double), POINTER(c_int32)]),
    "rse_fuse_rrf": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_double, c_int32, POINTER(c_int64),
                                    POINTER(c_double), POINTER(c_int32), POINTER(c_int64), POINTER(c_double),
                                    POINTER(c_int32), POINTER(c_int64), POINTER(c_double), POINTER(c_int32),
                                    POINTER(c_int32), POINTER(c_int32)]),
    "rse_set_id_tables": (ctypes.c_int, [c_void_p, POINTER(c_int64), c_int64, POINTER(c_int64), c_int64]),
    "rse_hybrid": (ctypes.c_int, [c_void_p, c_int32, c_double, c_int32, c_int32, c_int32, c_int32, POINTER(c_float),
                                  POINTER(c_int32), POINTER(c_int32), c_double, c_double, POINTER(c_int64),
                                  POINTER(c_double), POINTER(c_double), POINTER(c_double), POINTER(c_int32)]),
    "rse_hybrid_stage": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "rse_hybrid_run": (ctypes.c_int, [c_void_p, c_int32, c_double, c_int32, c_int32, c_int32, c_double, c_double]),
    "rse_hybrid_run_merged_dev": (ctypes.c_int, [c_void_p, c_int32, c_double, c_int32, c_int32, c_int32, c_double,
                                                 c_double, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                                 c_void_p]),
    "rse_hybrid_fetch": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p]),
    "rse_hybrid_submit": (ctypes.c_int, [c_void_p, c_int32, c_double, c_int32, c_int32, c_int32, c_int32, c_void_p,
                                         c_void_p, c_void_p, c_double, c_double, POINTER(c_int64)]),
    "rse_hybrid_collect": (ctypes.c_int, [c_void_p, c_int64, POINTER(c_int32), POINTER(c_int32), c_void_p, c_void_p,
                                          c_void_p, c_void_p, c_void_p]),
    "rse_hybrid_drain": (ctypes.c_int, [c_void_p, POINTER(c_int32)]),
    "rse_hybrid_stash": (ctypes.c_int, [c_void_p, c_int32]),
    "rse_tc_last_survivors": (ctypes.c_int, [c_void_p, POINTER(c_int32), c_int32]),
    "rse_tc_last_pairs": (ctypes.c_int, [c_void_p, c_int32, POINTER(c_int64), POINTER(c_float), c_int32,
                                         POINTER(c_int32)]),
    "rse_tc_probe_rank": (ctypes.c_int, [c_int32, c_int32]),
    "rse_encoder_create": (ctypes.c_int, [c_void_p, c_int32, POINTER(RseEncoderConfig)]),
    "rse_encoder_set_tensor": (ctypes.c_int, [c_void_p, c_int32, c_char_p, POINTER(c_float), c_int64]),
    "rse_encoder_finalize": (ctypes.c_int, [c_void_p, c_int32]),
    "rse_encoder_set_mode": (ctypes.c_int, [c_void_p, c_int32, c_int32]),
    "rse_encode": (ctypes.c_int, [c_void_p, c_int32, POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_int32,
                                  POINTER(c_float)]),
    "rse_encode_dev": (ctypes.c_int, [c_void_p, c_int32, POINTER(c_int32), POINTER(c_int32), POINTER(c_int32), c_int32,
                                      c_void_p]),
    "rse_clip_create": (ctypes.c_int, [c_void_p, c_int32, POINTER(RseClipConfig)]),
    "rse_encode_images": (ctypes.c_int, [c_void_p, c_int32, POINTER(c_float), c_int32, POINTER(c_float)]),
    "rse_encode_images_dev": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_int32, c_void_p]),
    "rse_imgproc_set": (ctypes.c_int, [c_void_p, c_int32, POINTER(RseImgprocCfg)]),
    "rse_image_preprocess": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "rse_image_preprocess_dev": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "rse_encode_images_u8": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "rse_encode_images_u8_dev": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_int32, c_void_p]),
    "rse_hybrid_stage_dev": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p]),
    "rse_rerank_docs_load": (ctypes.c_int, [c_void_p, POINTER(c_int64), c_int64, POINTER(c_int64), POINTER(c_int32)]),
    "rse_hybrid_rerank_run": (ctypes.c_int, [c_void_p, c_int32, c_double, c_int32, c_int32, c_int32, c_double, c_double,
                                             POINTER(c_int32), POINTER(c_int32), c_int32, c_int32, c_int32, c_int32]),
    "rse_hybrid_rerank_fetch": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p,
                                               c_void_p, c_void_p]),
    "rse_set_rerank_token_budget": (ctypes.c_int, [c_void_p, c_int64]),
    "rse_hybrid_rerank_timing": (ctypes.c_int, [c_void_p, POINTER(c_float)]),
    "rse_pair_truncate": (ctypes.c_int, [c_int32, c_int32, c_int32, POINTER(c_int32), POINTER(c_int32)]),
    "rse_tokenizer_load": (ctypes.c_int, [c_void_p, c_int32, POINTER(RseWordpieceDesc)]),
    "rse_tokenize": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_int32, POINTER(c_int64),
                                    POINTER(c_int32)]),
    "rse_tokens_fetch": (ctypes.c_int, [c_void_p, c_void_p, c_void_p]),
    "rse_tokens_fetch_dev": (ctypes.c_int, [c_void_p, c_void_p, c_void_p]),
    "rse_encode_texts": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "rse_encode_texts_dev": (ctypes.c_int, [c_void_p, c_int32, c_int32, c_void_p, c_void_p, c_int32, c_int32,
                                            c_void_p]),
    "rse_rerank_docs_load_texts": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_int64, c_void_p, c_void_p]),
    "rse_tokenizer_load_bpe": (ctypes.c_int, [c_void_p, c_int32, POINTER(RseBpeDesc)]),
    "rse_chunk_count": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_int32, c_int32, c_void_p,
                                       c_void_p, POINTER(c_int64), POINTER(c_int64)]),
    "rse_chunk_write": (ctypes.c_int, [c_void_p, c_void_p, c_int64, c_void_p, c_int32, c_int32, c_int32, c_void_p,
                                       c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p]),
    "rse_tokenize_dev": (ctypes.c_int, [c_void_p, c_int32, c_void_p, c_int64, c_void_p, c_int32, c_int32, c_int32,
                                        POINTER(c_int64), POINTER(c_int32)]),
    "rse_encode_tokens_dev": (ctypes.c_int, [c_void_p, c_int32, c_int64, c_void_p]),
    "rse_comm_unique_id": (ctypes.c_int, [c_void_p]),
    "rse_comm_init": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32]),
    "rse_comm_destroy": (ctypes.c_int, [c_void_p]),
    "rse_comm_info": (ctypes.c_int, [c_void_p, POINTER(c_int32), POINTER(c_int32), POINTER(c_int32)]),
    "rse_comm_exchange_candidates_dev": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_void_p]),
    "rse_comm_allgather_dev": (ctypes.c_int, [c_void_p, c_void_p, c_void_p, c_int64]),
    "rse_knn_sharded_dev": (ctypes.c_int, [c_void_p, c_void_p, c_int32, c_int32, c_int32, c_void_p, c_void_p, c_void_p,
                                           c_void_p, c_void_p]),
    "rse_hybrid_sharded_run_dev": (ctypes.c_int, [c_void_p, c_int32, c_double, c_int32, c_int32, c_int32, c_double,
                                                  c_double, c_void_p, c_int32, c_void_p, c_void_p, c_void_p, c_void_p,
                                                  c_void_p, c_void_p]),
    "rse_get_stats": (ctypes.c_int, [c_void_p, POINTER(RseStats)]),
    "rse_stats_reset": (ctypes.c_int, [c_void_p]),
    "rse_set_timing": (ctypes.c_int, [c_void_p, c_int32]),
}

EXPORTED_SYMBOLS = tuple(_SIGNATURES)

_lib = None


def load_library() -> ctypes.CDLL:
    """dlopen librse.so and bind every symbol include/rse.h declares.  No compute, no GPU needed."""
    global _lib
    if _lib is None:
        if not LIB_PATH.exists():
            raise RseError(-100, f"{LIB_PATH} is missing — build it with "
                                 f"`python -m rag_search_engine_b200.build` (nvcc, sm_100a). "
                                 f"There is no CPU fallback.")
        L = ctypes.CDLL(str(LIB_PATH))
        for name, (res, args) in _SIGNATURES.items():
            fn = getattr(L, name)          # AttributeError here = header/library drift
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def pair_truncate(n1: int, n2: int, max_length: int):
    """(a, b): how many of n1 query and n2 document tokens a cross-encoder pair of max_length keeps (rse_pair_truncate,
    the HF fast tokenizers' longest_first rule)."""
    a, b = c_int32(0), c_int32(0)
    rc = load_library().rse_pair_truncate(int(n1), int(n2), int(max_length), ctypes.byref(a), ctypes.byref(b))
    if rc != RSE_OK:
        raise RseError(rc, "rse_pair_truncate: n1, n2 >= 0 and max_length >= 4")
    return int(a.value), int(b.value)


def _ptr(a, ty):
    if a is None:
        return None
    return a.ctypes.data_as(POINTER(ty))


def _c(a, dtype):
    return np.ascontiguousarray(a, dtype=dtype)


class Index:
    """Thin RAII wrapper of an ``rse_index*`` handle."""

    def __init__(self, device: int = 0):
        self._L = load_library()
        self._h = c_void_p()
        rc = self._L.rse_create(int(device), ctypes.byref(self._h))
        if rc != RSE_OK:
            msg = self._L.rse_last_error(None)
            self._h = c_void_p()
            raise RseError(rc, msg.decode() if msg else "rse_create failed")
        self.device = int(device)
        self.n_rows, self.dim, self.n_docs = 0, 0, 0
        self._keepalive = []
        self._tickets = {}

    # ------------------------------------------------------------------ plumbing
    def _check(self, rc: int):
        if rc != RSE_OK:
            msg = self._L.rse_last_error(self._h)
            raise RseError(rc, msg.decode() if msg else "")

    def close(self):
        if getattr(self, "_h", None) is not None and self._h:
            self._L.rse_destroy(self._h)
            self._h = c_void_p()
        self._keepalive = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream_ptr: int):
        """cuda_stream_ptr = cudaStream_t as int; 0 is the legacy default stream (torch's default)."""
        self._check(self._L.rse_set_stream(self._h, c_void_p(int(cuda_stream_ptr))))

    def use_own_stream(self):
        self._check(self._L.rse_use_own_stream(self._h))

    def synchronize(self):
        self._check(self._L.rse_synchronize(self._h))

    def set_timing(self, on: bool):
        self._check(self._L.rse_set_timing(self._h, int(bool(on))))

    def set_tc_mode(self, mode: int):
        """0 = auto (batches of >= 2 queries on >= 256 k rows), 1 = exact scan only, 2 = tensor-core path
        whenever the shape allows it.  Results are identical in every mode."""
        self._check(self._L.rse_set_tc_mode(self._h, int(mode)))

    def set_bm25_mode(self, mode: int):
        """0 = fixed-point streaming BM25 + exact re-score of the finalists (default), 1 = exact-order streaming
        kernel, 2 = general kernel only.  Results are identical in every mode."""
        self._check(self._L.rse_set_bm25_mode(self._h, int(mode)))

    def set_fma(self, on: bool):
        self._check(self._L.rse_set_fma(self._h, int(bool(on))))

    def stats(self) -> RseStats:
        s = RseStats()
        self._check(self._L.rse_get_stats(self._h, ctypes.byref(s)))
        return s

    def stats_reset(self):
        self._check(self._L.rse_stats_reset(self._h))

    # ------------------------------------------------------------------ embeddings / KNN
    def load_embeddings(self, emb, valid=None, rowid=None, movie_idx=None, pos_base: int = 0):
        emb = _c(emb, np.float32)
        if emb.ndim != 2:
            raise ValueError("emb must be [n_rows, dim]")
        n, d = emb.shape
        valid = None if valid is None else _c(valid, np.uint8)
        rowid = None if rowid is None else _c(rowid, np.int64)
        movie_idx = None if movie_idx is None else _c(movie_idx, np.int32)
        self._check(self._L.rse_load_embeddings(self._h, _ptr(emb, c_float), n, d, _ptr(valid, c_uint8),
                                                _ptr(rowid, c_int64), _ptr(movie_idx, c_int32), int(pos_base)))
        self.n_rows, self.dim = n, d

    def attach_embeddings_dev(self, emb_ptr: int, n_rows: int, dim: int, valid_ptr: int = 0, rowid_ptr: int = 0,
                              movie_idx_ptr: int = 0, pos_base: int = 0, keepalive=None):
        self._check(self._L.rse_attach_embeddings_dev(self._h, c_void_p(emb_ptr), int(n_rows), int(dim),
                                                      c_void_p(valid_ptr or 0), c_void_p(rowid_ptr or 0),
                                                      c_void_p(movie_idx_ptr or 0), int(pos_base)))
        self.n_rows, self.dim = int(n_rows), int(dim)
        self._keepalive = [keepalive]

    def knn(self, Q, kprime: int):
        Q = _c(Q, np.float32).reshape(-1, self.dim)
        nq = Q.shape[0]
        dist = np.zeros((nq, kprime), np.float32)
        pos = np.zeros((nq, kprime), np.int64)
        rowid = np.zeros((nq, kprime), np.int64)
        movie = np.zeros((nq, kprime), np.int32)
        cnt = np.zeros(nq, np.int32)
        self._check(self._L.rse_knn(self._h, _ptr(Q, c_float), nq, int(kprime), _ptr(dist, c_float),
                                    _ptr(pos, c_int64), _ptr(rowid, c_int64), _ptr(movie, c_int32),
                                    _ptr(cnt, c_int32)))
        return dist, pos, rowid, movie, cnt

    def knn_movies(self, Q, k: int, kprime: int):
        Q = _c(Q, np.float32).reshape(-1, self.dim)
        nq = Q.shape[0]
        dist = np.zeros((nq, k), np.float32)
        rowid = np.zeros((nq, k), np.int64)
        movie = np.zeros((nq, k), np.int32)
        cnt = np.zeros(nq, np.int32)
        self._check(self._L.rse_knn_movies(self._h, _ptr(Q, c_float), nq, int(k), int(kprime), _ptr(dist, c_float),
                                           _ptr(rowid, c_int64), _ptr(movie, c_int32), _ptr(cnt, c_int32)))
        return dist, rowid, movie, cnt

    def knn_movies_exact(self, Q, k: int):
        """The k nearest movies by best chunk over every row (rse_knn_movies_exact) →
        (dist, rowid, movie, count, scanned); scanned = queries that took the full segmented scan."""
        Q = _c(Q, np.float32)
        Q = Q.reshape(-1, self.dim or Q.shape[-1])
        nq = Q.shape[0]
        kk = max(int(k), 1)
        dist = np.zeros((nq, kk), np.float32)
        rowid = np.zeros((nq, kk), np.int64)
        movie = np.zeros((nq, kk), np.int32)
        cnt = np.zeros(nq, np.int32)
        scanned = c_int32(0)
        self._check(self._L.rse_knn_movies_exact(self._h, _ptr(Q, c_float), nq, int(k), _ptr(dist, c_float),
                                                 _ptr(rowid, c_int64), _ptr(movie, c_int32), _ptr(cnt, c_int32),
                                                 ctypes.byref(scanned)))
        return dist, rowid, movie, cnt, int(scanned.value)

    def knn_local_dev(self, q_ptr: int, nq: int, kprime: int, cand_ptr: int):
        self._check(self._L.rse_knn_local_dev(self._h, c_void_p(q_ptr), int(nq), int(kprime), c_void_p(cand_ptr)))

    def set_defer_flags(self, on: bool):
        """rse_knn_local_dev without the host round trip for the overflow flags (see include/rse.h)."""
        self._check(self._L.rse_set_defer_flags(self._h, int(bool(on))))

    def knn_flags_dev(self, flagged_ptr: int):
        self._check(self._L.rse_knn_flags_dev(self._h, c_void_p(flagged_ptr)))

    def knn_merge_movies_dev(self, gathered_ptr: int, n_lists: int, nq: int, k: int, kprime: int, dist_ptr: int,
                             rowid_ptr: int, movie_ptr: int, count_ptr: int):
        self._check(self._L.rse_knn_merge_movies_dev(self._h, c_void_p(gathered_ptr), int(n_lists), int(nq), int(k),
                                                     int(kprime), c_void_p(dist_ptr), c_void_p(rowid_ptr),
                                                     c_void_p(movie_ptr), c_void_p(count_ptr)))

    # ------------------------------------------------------------------ BM25
    def load_bm25(self, indptr, doc_idx, tf, df, dl, n_movies: int, avgdl: float):
        indptr = _c(indptr, np.int64)
        doc_idx = _c(doc_idx, np.uint32)
        tf = _c(tf, np.uint32)
        df = _c(df, np.int64)
        dl = _c(dl, np.uint32)
        self._check(self._L.rse_load_bm25(self._h, _ptr(indptr, c_int64), _ptr(doc_idx, c_uint32),
                                          _ptr(tf, c_uint32), _ptr(df, c_int64), len(indptr) - 1, len(doc_idx),
                                          _ptr(dl, c_uint32), len(dl), int(n_movies), float(avgdl)))
        self.n_docs = len(dl)

    def bm25(self, tok_indptr, term_rows, k: int, k1: float = 1.5, b: float = 0.75):
        tok_indptr = _c(tok_indptr, np.int32)
        term_rows = _c(term_rows, np.int32)
        if term_rows.size == 0:
            term_rows = np.zeros(1, np.int32)
        nq = len(tok_indptr) - 1
        score = np.zeros((nq, k), np.float64)
        doc = np.full((nq, k), -1, np.int32)
        cnt = np.zeros(nq, np.int32)
        self._check(self._L.rse_bm25(self._h, _ptr(tok_indptr, c_int32), _ptr(term_rows, c_int32), nq, int(k),
                                     float(k1), float(b), _ptr(score, c_double), _ptr(doc, c_int32),
                                     _ptr(cnt, c_int32)))
        return score, doc, cnt

    # ------------------------------------------------------------------ fusion
    def _fuse_inputs(self, limit, bm25_id, bm25_score, bm25_count, sem_id, sem_dist, sem_count):
        bm25_id = _c(bm25_id, np.int64).reshape(-1, limit)
        nq = bm25_id.shape[0]
        return (nq, bm25_id, _c(bm25_score, np.float64).reshape(nq, limit), _c(bm25_count, np.int32).reshape(nq),
                _c(sem_id, np.int64).reshape(nq, limit), _c(sem_dist, np.float64).reshape(nq, limit),
                _c(sem_count, np.int32).reshape(nq))

    def fuse_weighted(self, limit, alpha, bm25_id, bm25_score, bm25_count, sem_id, sem_dist, sem_count,
                      tie_mode: int = TIE_REFERENCE):
        nq, bid, bsc, bc, sid, sds, scn = self._fuse_inputs(limit, bm25_id, bm25_score, bm25_count, sem_id,
                                                            sem_dist, sem_count)
        oid = np.zeros((nq, limit), np.int64)
        ob = np.zeros((nq, limit), np.float64)
        osem = np.zeros((nq, limit), np.float64)
        osc = np.zeros((nq, limit), np.float64)
        oc = np.zeros(nq, np.int32)
        self._check(self._L.rse_fuse_weighted(self._h, nq, int(limit), float(alpha), int(tie_mode),
                                              _ptr(bid, c_int64), _ptr(bsc, c_double), _ptr(bc, c_int32),
                                              _ptr(sid, c_int64), _ptr(sds, c_double), _ptr(scn, c_int32),
                                              _ptr(oid, c_int64), _ptr(ob, c_double), _ptr(osem, c_double),
                                              _ptr(osc, c_double), _ptr(oc, c_int32)))
        return oid, ob, osem, osc, oc

    def fuse_rrf(self, limit, k, bm25_id, bm25_score, bm25_count, sem_id, sem_dist, sem_count,
                 tie_mode: int = TIE_REFERENCE):
        nq, bid, bsc, bc, sid, sds, scn = self._fuse_inputs(limit, bm25_id, bm25_score, bm25_count, sem_id,
                                                            sem_dist, sem_count)
        oid = np.zeros((nq, limit), np.int64)
        osc = np.zeros((nq, limit), np.float64)
        orb = np.zeros((nq, limit), np.int32)
        ors = np.zeros((nq, limit), np.int32)
        oc = np.zeros(nq, np.int32)
        self._check(self._L.rse_fuse_rrf(self._h, nq, int(limit), float(k), int(tie_mode), _ptr(bid, c_int64),
                                         _ptr(bsc, c_double), _ptr(bc, c_int32), _ptr(sid, c_int64),
                                         _ptr(sds, c_double), _ptr(scn, c_int32), _ptr(oid, c_int64),
                                         _ptr(osc, c_double), _ptr(orb, c_int32), _ptr(ors, c_int32),
                                         _ptr(oc, c_int32)))
        return oid, osc, orb, ors, oc

    # ------------------------------------------------------------------ hybrid
    def set_id_tables(self, doc_ids, movie_ids):
        doc_ids = _c(doc_ids, np.int64)
        movie_ids = _c(movie_ids, np.int64)
        self._check(self._L.rse_set_id_tables(self._h, _ptr(doc_ids, c_int64), len(doc_ids),
                                              _ptr(movie_ids, c_int64), len(movie_ids)))

    def hybrid(self, mode: int, param: float, limit: int, Q, tok_indptr, term_rows, knn_multiplier: int = 10,
               k1: float = 1.5, b: float = 0.75, tie_mode: int = TIE_REFERENCE):
        Q = _c(Q, np.float32).reshape(-1, self.dim)
        nq = Q.shape[0]
        tok_indptr = _c(tok_indptr, np.int32)
        term_rows = _c(term_rows, np.int32)
        if term_rows.size == 0:
            term_rows = np.zeros(1, np.int32)
        if len(tok_indptr) != nq + 1:
            raise ValueError("tok_indptr must have nq+1 entries")
        oid = np.zeros((nq, limit), np.int64)
        osc = np.zeros((nq, limit), np.float64)
        oa = np.zeros((nq, limit), np.float64)
        ob = np.zeros((nq, limit), np.float64)
        oc = np.zeros(nq, np.int32)
        self._check(self._L.rse_hybrid(self._h, int(mode), float(param), int(tie_mode), int(limit),
                                       int(knn_multiplier), nq, _ptr(Q, c_float), _ptr(tok_indptr, c_int32),
                                       _ptr(term_rows, c_int32), float(k1), float(b), _ptr(oid, c_int64),
                                       _ptr(osc, c_double), _ptr(oa, c_double), _ptr(ob, c_double),
                                       _ptr(oc, c_int32)))
        return oid, osc, oa, ob, oc

    # split form (inputs resident in HBM between run() calls); pointers are raw host addresses
    def hybrid_stage(self, Q, tok_indptr, term_rows):
        Q = _c(Q, np.float32).reshape(-1, self.dim)
        tok_indptr = _c(tok_indptr, np.int32)
        term_rows = _c(term_rows, np.int32)
        if term_rows.size == 0:
            term_rows = np.zeros(1, np.int32)
        self._check(self._L.rse_hybrid_stage(self._h, Q.shape[0], c_void_p(Q.ctypes.data),
                                             c_void_p(tok_indptr.ctypes.data), c_void_p(term_rows.ctypes.data)))
        self._staged_nq = Q.shape[0]

    def hybrid_run(self, mode: int, param: float, limit: int, knn_multiplier: int = 10, k1: float = 1.5,
                   b: float = 0.75, tie_mode: int = TIE_REFERENCE):
        self._check(self._L.rse_hybrid_run(self._h, int(mode), float(param), int(tie_mode), int(limit),
                                           int(knn_multiplier), float(k1), float(b)))

    def hybrid_fetch(self, limit: int):
        nq = self._staged_nq
        oid = np.zeros((nq, limit), np.int64)
        osc = np.zeros((nq, limit), np.float64)
        oa = np.zeros((nq, limit), np.float64)
        ob = np.zeros((nq, limit), np.float64)
        oc = np.zeros(nq, np.int32)
        self._check(self._L.rse_hybrid_fetch(self._h, int(limit), c_void_p(oid.ctypes.data), c_void_p(osc.ctypes.data),
                                             c_void_p(oa.ctypes.data), c_void_p(ob.ctypes.data),
                                             c_void_p(oc.ctypes.data)))
        return oid, osc, oa, ob, oc

    # pipelined form: two batches in flight (rse_hybrid_submit / rse_hybrid_collect)
    def hybrid_submit(self, mode: int, param: float, limit: int, Q, tok_indptr, term_rows, knn_multiplier: int = 10,
                      k1: float = 1.5, b: float = 0.75, tie_mode: int = TIE_REFERENCE) -> int:
        Q = _c(Q, np.float32).reshape(-1, self.dim)
        nq = Q.shape[0]
        tok_indptr = _c(tok_indptr, np.int32)
        term_rows = _c(term_rows, np.int32)
        if term_rows.size == 0:
            term_rows = np.zeros(1, np.int32)
        if len(tok_indptr) != nq + 1:
            raise ValueError("tok_indptr must have nq+1 entries")
        ticket = c_int64(-1)
        self._check(self._L.rse_hybrid_submit(self._h, int(mode), float(param), int(tie_mode), int(limit),
                                              int(knn_multiplier), nq, c_void_p(Q.ctypes.data),
                                              c_void_p(tok_indptr.ctypes.data), c_void_p(term_rows.ctypes.data),
                                              float(k1), float(b), ctypes.byref(ticket)))
        self._tickets[ticket.value] = (nq, int(limit))
        return ticket.value

    def hybrid_collect(self, ticket: int):
        if ticket not in self._tickets:
            raise KeyError(f"unknown ticket {ticket}")
        nq, limit = self._tickets[ticket]
        oid = np.zeros((nq, limit), np.int64)
        osc = np.zeros((nq, limit), np.float64)
        oa = np.zeros((nq, limit), np.float64)
        ob = np.zeros((nq, limit), np.float64)
        oc = np.zeros(nq, np.int32)
        self._check(self._L.rse_hybrid_collect(self._h, int(ticket), None, None, c_void_p(oid.ctypes.data),
                                               c_void_p(osc.ctypes.data), c_void_p(oa.ctypes.data),
                                               c_void_p(ob.ctypes.data), c_void_p(oc.ctypes.data)))
        del self._tickets[ticket]
        return oid, osc, oa, ob, oc

    def hybrid_stash(self, slot: int):
        """Exchange the staged batch with stash slot ``slot`` (several batches resident in HBM)."""
        self._check(self._L.rse_hybrid_stash(self._h, int(slot)))
        stash = self.__dict__.setdefault("_stash_nq", {})
        stash[slot], self._staged_nq = getattr(self, "_staged_nq", 0), stash.get(slot, 0)

    def tc_last_survivors(self, n: int = 256):
        out = np.zeros(int(n), np.int32)
        self._check(self._L.rse_tc_last_survivors(self._h, _ptr(out, c_int32), int(n)))
        return out

    def tc_last_pairs(self, query: int, cap: int = 8192):
        """(rows int64[m], cos~ float32[m], count) of one query's survivors in the last K4 filter pass."""
        rows = np.zeros(int(cap), np.int64)
        cos = np.zeros(int(cap), np.float32)
        n = c_int32(0)
        self._check(self._L.rse_tc_last_pairs(self._h, int(query), _ptr(rows, c_int64), _ptr(cos, c_float), int(cap),
                                              ctypes.byref(n)))
        m = min(n.value, int(cap), 8192)
        return rows[:m], cos[:m], n.value

    def hybrid_drain(self) -> int:
        """Wait for and discard every ticket still in flight; the handle accepts submits again afterwards."""
        n = c_int32(0)
        self._check(self._L.rse_hybrid_drain(self._h, ctypes.byref(n)))
        self._tickets.clear()
        return int(n.value)

    # ------------------------------------------------------------------ text encoders (§8 f2 / f3)
    def encoder_create(self, slot: int, *, vocab_size: int, hidden: int, layers: int, heads: int, intermediate: int,
                       max_positions: int, type_vocab: int, ln_eps: float, head: int):
        cfg = RseEncoderConfig(int(vocab_size), int(hidden), int(layers), int(heads), int(intermediate),
                               int(max_positions), int(type_vocab), float(ln_eps), int(head))
        self._check(self._L.rse_encoder_create(self._h, int(slot), ctypes.byref(cfg)))
        self.__dict__.setdefault("_enc_cfg", {})[int(slot)] = cfg

    def clip_create(self, slot: int, *, tower: int, hidden: int, layers: int, heads: int, intermediate: int,
                    projection_dim: int, ln_eps: float, vocab_size: int = 0, max_positions: int = 0,
                    image_size: int = 0, patch_size: int = 0, eos_token_id: int = 0):
        """A CLIP tower (0 = vision, 1 = text) in encoder slot ``slot``; weights then go through encoder_set_tensor /
        encoder_finalize like a BERT slot's."""
        cfg = RseClipConfig(int(tower), int(hidden), int(layers), int(heads), int(intermediate), int(projection_dim),
                            int(vocab_size), int(max_positions), int(image_size), int(patch_size), int(eos_token_id),
                            float(ln_eps))
        self._check(self._L.rse_clip_create(self._h, int(slot), ctypes.byref(cfg)))
        self.__dict__.setdefault("_enc_cfg", {})[int(slot)] = cfg

    def encode_images(self, slot: int, pixel_values):
        """pixel_values [n, 3, S, S] float32 (NCHW, the image processor's output) -> [n, projection_dim] float32."""
        px = _c(pixel_values, np.float32)
        if px.ndim != 4 or px.shape[1] != 3:
            raise ValueError("pixel_values must be [n, 3, image_size, image_size]")
        cfg = self._enc_cfg.get(int(slot))
        if isinstance(cfg, RseClipConfig) and cfg.tower == 0 and px.shape[2:] != (cfg.image_size, cfg.image_size):
            raise ValueError(f"pixel_values must be {cfg.image_size} x {cfg.image_size} (the tower's image_size)")
        n = px.shape[0]
        out = np.zeros((n, cfg.projection_dim if isinstance(cfg, RseClipConfig) else 1), np.float32)
        self._check(self._L.rse_encode_images(self._h, int(slot), _ptr(px, c_float), n, _ptr(out, c_float)))
        return out

    def encode_images_dev(self, slot: int, pixels_ptr: int, n: int, out_ptr: int):
        """Same with the pixels on the device and the result left there (asynchronous on the handle's stream)."""
        self._check(self._L.rse_encode_images_dev(self._h, int(slot), c_void_p(pixels_ptr), int(n), c_void_p(out_ptr)))

    def imgproc_set(self, slot: int, *, backend: int, shortest_edge: int, crop_height: int, crop_width: int,
                    rescale_factor: float, mean, std, do_resize: bool = True, do_center_crop: bool = True,
                    do_rescale: bool = True, do_normalize: bool = True):
        """Bind a CLIP image-preprocessing configuration (0 = CLIPImageProcessor, 1 = CLIPImageProcessorPil numerics)
        to the vision tower in ``slot`` (rse_imgproc_set)."""
        cfg = RseImgprocCfg(int(backend), int(shortest_edge), int(crop_height), int(crop_width), int(bool(do_resize)),
                            int(bool(do_center_crop)), int(bool(do_rescale)), int(bool(do_normalize)),
                            float(rescale_factor), (c_double * 3)(*map(float, mean)), (c_double * 3)(*map(float, std)))
        self._check(self._L.rse_imgproc_set(self._h, int(slot), ctypes.byref(cfg)))

    @staticmethod
    def _pack_images(images):
        """[H, W, 3] uint8 arrays -> (packed bytes, int64 offsets [n], int32 hw [n, 2])."""
        arrs = [np.ascontiguousarray(a, np.uint8) for a in images]
        for a in arrs:
            if a.ndim != 3 or a.shape[2] != 3:
                raise ValueError("images must be [H, W, 3] uint8 (RGB)")
        sizes = np.array([a.size for a in arrs], np.int64)
        offs = np.zeros(len(arrs), np.int64)
        np.cumsum(sizes[:-1], out=offs[1:])
        packed = np.empty(int(sizes.sum()), np.uint8)
        for a, o, n in zip(arrs, offs, sizes):
            packed[o:o + n] = a.reshape(-1)
        hw = np.array([a.shape[:2] for a in arrs], np.int32).reshape(-1, 2)
        return packed, offs, hw

    def image_preprocess(self, slot: int, images) -> np.ndarray:
        """[H, W, 3] uint8 RGB images (any sizes) -> pixel_values [n, 3, S, S] float32 through the slot's
        preprocessing configuration, on the device."""
        packed, offs, hw = self._pack_images(images)
        cfg = self._enc_cfg[int(slot)]
        out = np.zeros((len(offs), 3, cfg.image_size, cfg.image_size), np.float32)
        self._check(self._L.rse_image_preprocess(self._h, int(slot), packed.ctypes.data, offs.ctypes.data,
                                                 hw.ctypes.data, len(offs), out.ctypes.data))
        return out

    def encode_images_u8(self, slot: int, images) -> np.ndarray:
        """[H, W, 3] uint8 RGB images -> [n, projection_dim] float32: preprocessing and the vision tower on the device."""
        packed, offs, hw = self._pack_images(images)
        out = np.zeros((len(offs), self._enc_cfg[int(slot)].projection_dim), np.float32)
        self._check(self._L.rse_encode_images_u8(self._h, int(slot), packed.ctypes.data, offs.ctypes.data,
                                                 hw.ctypes.data, len(offs), out.ctypes.data))
        return out

    def encode_images_u8_dev(self, slot: int, images, out_ptr: int):
        """Same with the embeddings left on the device at ``out_ptr`` (asynchronous on the handle's stream once the
        pixels are staged)."""
        packed, offs, hw = self._pack_images(images)
        self._check(self._L.rse_encode_images_u8_dev(self._h, int(slot), packed.ctypes.data, offs.ctypes.data,
                                                     hw.ctypes.data, len(offs), c_void_p(out_ptr)))

    def encoder_set_tensor(self, slot: int, name: str, data):
        a = _c(data, np.float32).reshape(-1)
        self._check(self._L.rse_encoder_set_tensor(self._h, int(slot), name.encode(), _ptr(a, c_float), a.size))

    def encoder_finalize(self, slot: int):
        self._check(self._L.rse_encoder_finalize(self._h, int(slot)))

    def encoder_set_mode(self, slot: int, mode: int):
        """0 = tcgen05 3xTF32 GEMMs (default), 1 = fp32 SIMT GEMMs."""
        self._check(self._L.rse_encoder_set_mode(self._h, int(slot), int(mode)))

    def _enc_inputs(self, ids, type_ids, cu_seqlens):
        ids = _c(ids, np.int32).reshape(-1)
        cu = _c(cu_seqlens, np.int32).reshape(-1)
        tt = None if type_ids is None else _c(type_ids, np.int32).reshape(-1)
        if cu[-1] != ids.size or (tt is not None and tt.size != ids.size):
            raise ValueError("cu_seqlens[-1] must equal the number of token ids (and of token type ids)")
        return ids, tt, cu

    def encode(self, slot: int, ids, cu_seqlens, type_ids=None):
        """Packed token ids -> [n_seq, hidden] float32 (head 0), [n_seq] logits (head 1) or [n_seq, projection_dim]
        (CLIP text tower), on the host."""
        ids, tt, cu = self._enc_inputs(ids, type_ids, cu_seqlens)
        cfg = self._enc_cfg[int(slot)]
        n_seq = cu.size - 1
        if isinstance(cfg, RseClipConfig):
            out = np.zeros((n_seq, cfg.projection_dim), np.float32)
        else:
            out = np.zeros((n_seq, cfg.hidden) if cfg.head == 0 else (n_seq,), np.float32)
        self._check(self._L.rse_encode(self._h, int(slot), _ptr(ids, c_int32), _ptr(tt, c_int32), _ptr(cu, c_int32),
                                       n_seq, _ptr(out, c_float)))
        return out

    def encode_dev(self, slot: int, ids, cu_seqlens, out_ptr: int, type_ids=None):
        """Same, result left on the device at ``out_ptr`` (asynchronous on the handle's stream)."""
        ids, tt, cu = self._enc_inputs(ids, type_ids, cu_seqlens)
        self._check(self._L.rse_encode_dev(self._h, int(slot), _ptr(ids, c_int32), _ptr(tt, c_int32), _ptr(cu, c_int32),
                                           cu.size - 1, c_void_p(out_ptr)))

    def hybrid_stage_dev(self, nq: int, q_ptr: int, tok_indptr, term_rows):
        """rse_hybrid_stage with the query vectors already on the device (e.g. encode_dev's output)."""
        tok_indptr = _c(tok_indptr, np.int32)
        term_rows = _c(term_rows, np.int32)
        if term_rows.size == 0:
            term_rows = np.zeros(1, np.int32)
        if len(tok_indptr) != nq + 1:
            raise ValueError("tok_indptr must have nq+1 entries")
        self._check(self._L.rse_hybrid_stage_dev(self._h, int(nq), c_void_p(q_ptr), c_void_p(tok_indptr.ctypes.data),
                                                 c_void_p(term_rows.ctypes.data)))
        self._staged_nq = int(nq)

    # ------------------------------------------------------------------ cross-encoder rerank of a fused batch
    def rerank_docs_load(self, ids, tok_indptr, tokens):
        """The document-token store: ids strictly ascending, CSR token ids (no special tokens) per document."""
        ids = _c(ids, np.int64)
        tok_indptr = _c(tok_indptr, np.int64)
        tokens = _c(tokens, np.int32)
        if len(tok_indptr) != len(ids) + 1:
            raise ValueError("tok_indptr must have len(ids) + 1 entries")
        if tokens.size == 0:
            tokens = np.zeros(1, np.int32)
        self._check(self._L.rse_rerank_docs_load(self._h, _ptr(ids, c_int64), len(ids), _ptr(tok_indptr, c_int64),
                                                 _ptr(tokens, c_int32)))

    def set_rerank_token_budget(self, tokens: int):
        self._check(self._L.rse_set_rerank_token_budget(self._h, int(tokens)))

    def hybrid_rerank_run(self, slot: int, k: float, limit: int, q_tok_indptr, q_tok_ids, *, cls_id: int, sep_id: int,
                          max_length: int, activation: int = 0, knn_multiplier: int = 10, k1: float = 1.5,
                          b: float = 0.75, tie_mode: int = TIE_REFERENCE):
        """RRF over the whole union + cross-encoder rerank of the staged batch (include/rse.h); the query token ids
        come without special tokens."""
        q_tok_indptr = _c(q_tok_indptr, np.int32)
        q_tok_ids = _c(q_tok_ids, np.int32)
        nq = getattr(self, "_staged_nq", 0)
        if nq and len(q_tok_indptr) != nq + 1:               # (nothing staged: the library reports the state)
            raise ValueError("q_tok_indptr must have (staged queries) + 1 entries")
        if q_tok_ids.size == 0:
            q_tok_ids = np.zeros(1, np.int32)
        self._check(self._L.rse_hybrid_rerank_run(self._h, int(slot), float(k), int(tie_mode), int(limit),
                                                  int(knn_multiplier), float(k1), float(b), _ptr(q_tok_indptr, c_int32),
                                                  _ptr(q_tok_ids, c_int32), int(cls_id), int(sep_id), int(max_length),
                                                  int(activation)))
        self._rerank_nq = self._staged_nq

    def hybrid_rerank_fetch(self, limit: int):
        """-> (id int64, rrf score float64, bm25_rank, sem_rank (-1 = None), rrf_rank int32, each [nq, limit];
        cross-encoder score float32 [nq, limit]; count int32 [nq])."""
        nq = getattr(self, "_rerank_nq", 0)
        oid = np.zeros((nq, limit), np.int64)
        osc = np.zeros((nq, limit), np.float64)
        orb = np.zeros((nq, limit), np.int32)
        ors = np.zeros((nq, limit), np.int32)
        orr = np.zeros((nq, limit), np.int32)
        oce = np.zeros((nq, limit), np.float32)
        oc = np.zeros(nq, np.int32)
        self._check(self._L.rse_hybrid_rerank_fetch(self._h, int(limit), c_void_p(oid.ctypes.data),
                                                    c_void_p(osc.ctypes.data), c_void_p(orb.ctypes.data),
                                                    c_void_p(ors.ctypes.data), c_void_p(orr.ctypes.data),
                                                    c_void_p(oce.ctypes.data), c_void_p(oc.ctypes.data)))
        return oid, osc, orb, ors, orr, oce, oc

    # ------------------------------------------------------------------ BERT WordPiece on the device
    def tokenizer_load(self, slot: int, tables):
        """A ``wordpiece.WordPieceTables`` into a tokenizer slot."""
        arrs = dict(cp_map=_c(tables.cp_map, np.uint32), extra=_c(tables.extra, np.uint32).reshape(-1),
                    cp_class=_c(tables.cp_class, np.uint8), node_first=_c(tables.node_first, np.int32),
                    node_id=_c(tables.node_id, np.int32), edge_cp=_c(tables.edge_cp, np.int32),
                    edge_child=_c(tables.edge_child, np.int32))
        raw = [c.encode() for c, _ in tables.added]
        added = np.frombuffer(b"".join(raw) or b"\0", np.uint8)
        aoff = np.zeros(len(raw) + 1, np.int32)
        np.cumsum([len(r) for r in raw], out=aoff[1:])
        aid = np.asarray([i for _, i in tables.added] or [0], np.int32)
        d = RseWordpieceDesc(n_extra=arrs["extra"].size // 3, n_nodes=arrs["node_id"].size, n_added=len(raw),
                             unk_id=tables.unk_id, cls_id=tables.cls_id, sep_id=tables.sep_id,
                             max_input_chars_per_word=tables.max_input_chars_per_word,
                             added=added.ctypes.data, added_offsets=aoff.ctypes.data, added_ids=aid.ctypes.data,
                             **{k: v.ctypes.data for k, v in arrs.items()})
        self._check(self._L.rse_tokenizer_load(self._h, int(slot), ctypes.byref(d)))

    @staticmethod
    def _added(added):
        raw = [c.encode() for c, _ in added]
        blob = np.frombuffer(b"".join(raw) or b"\0", np.uint8)
        offs = np.zeros(len(raw) + 1, np.int32)
        np.cumsum([len(r) for r in raw], out=offs[1:])
        return blob, offs, np.asarray([i for _, i in added] or [0], np.int32)

    def tokenizer_load_bpe(self, slot: int, tables):
        """A ``bpe.BpeTables`` (CLIP's byte-level BPE) into a tokenizer slot."""
        arrs = dict(cp_map=_c(tables.cp_map, np.uint32), extra=_c(tables.extra, np.uint32).reshape(-1),
                    cp_class=_c(tables.cp_class, np.uint8), byte_ids=_c(tables.byte_ids, np.int32),
                    merges=_c(tables.merges, np.int32).reshape(-1))
        added, aoff, aid = self._added(tables.added)
        d = RseBpeDesc(n_extra=arrs["extra"].size // 3, merge_slots=arrs["merges"].size // 4, n_added=len(tables.added),
                       bos_id=tables.bos_id, eos_id=tables.eos_id, added=added.ctypes.data,
                       added_offsets=aoff.ctypes.data, added_ids=aid.ctypes.data,
                       **{k: v.ctypes.data for k, v in arrs.items()})
        self._check(self._L.rse_tokenizer_load_bpe(self._h, int(slot), ctypes.byref(d)))

    @staticmethod
    def _texts(data: bytes, offsets):
        offsets = _c(offsets, np.int64)
        return c_char_p(data), offsets, len(offsets) - 1

    def tokenize(self, slot: int, data: bytes, offsets, add_special: bool, max_length: int = 0):
        """UTF-8 texts (``data`` delimited by ``offsets[n + 1]``) -> (ids int32[total], cu_seqlens int32[n + 1])."""
        txt, offs, n = self._texts(data, offsets)
        total, ml = c_int64(0), c_int32(0)
        self._check(self._L.rse_tokenize(self._h, int(slot), txt, c_void_p(offs.ctypes.data), n, int(bool(add_special)),
                                         int(max_length), ctypes.byref(total), ctypes.byref(ml)))
        ids = np.empty(max(total.value, 1), np.int32)
        cu = np.empty(n + 1, np.int32)
        self._check(self._L.rse_tokens_fetch(self._h, c_void_p(ids.ctypes.data), c_void_p(cu.ctypes.data)))
        return ids[:total.value], cu

    def tokenize_dev(self, slot: int, data: bytes, offsets, add_special: bool, max_length: int = 0):
        """Same, ids left in the handle's buffers: -> (total, longest); then ``tokens_fetch_dev``."""
        txt, offs, n = self._texts(data, offsets)
        total, ml = c_int64(0), c_int32(0)
        self._check(self._L.rse_tokenize(self._h, int(slot), txt, c_void_p(offs.ctypes.data), n, int(bool(add_special)),
                                         int(max_length), ctypes.byref(total), ctypes.byref(ml)))
        return int(total.value), int(ml.value)

    def tokens_fetch_dev(self, ids_ptr: int, cu_ptr: int):
        self._check(self._L.rse_tokens_fetch_dev(self._h, c_void_p(ids_ptr), c_void_p(cu_ptr)))

    def tokenize_device_texts(self, slot: int, text_ptr: int, text_bytes: int, offsets_ptr: int, n: int,
                              add_special: bool, max_length: int = 0):
        """``tokenize_dev`` over n texts already in device memory (bytes at ``text_ptr``, int64 offsets[n + 1] at
        ``offsets_ptr``), read in place: -> (total, longest); then ``tokens_fetch_dev`` / ``encode_tokens_dev``."""
        total, ml = c_int64(0), c_int32(0)
        self._check(self._L.rse_tokenize_dev(self._h, int(slot), c_void_p(text_ptr or 0), int(text_bytes),
                                             c_void_p(offsets_ptr), int(n), int(bool(add_special)), int(max_length),
                                             ctypes.byref(total), ctypes.byref(ml)))
        return int(total.value), int(ml.value)

    def encode_tokens_dev(self, enc_slot: int, max_tokens_per_call: int, out_ptr: int):
        """The sentence encoder on the last tokenization's ids, on the device -> [n, hidden] fp32 at ``out_ptr``."""
        self._check(self._L.rse_encode_tokens_dev(self._h, int(enc_slot), int(max_tokens_per_call), c_void_p(out_ptr)))

    def chunk_count(self, text_ptr: int, text_bytes: int, offsets_ptr: int, n_movies: int, max_chunk_size: int,
                    overlap: int, chunk_cu_ptr: int, byte_cu_ptr: int):
        """Sentence chunking, count pass (device buffers): -> (chunks, chunk-text bytes) of the n_movies movies."""
        nc, nb = c_int64(0), c_int64(0)
        self._check(self._L.rse_chunk_count(self._h, c_void_p(text_ptr or 0), int(text_bytes), c_void_p(offsets_ptr),
                                            int(n_movies), int(max_chunk_size), int(overlap), c_void_p(chunk_cu_ptr),
                                            c_void_p(byte_cu_ptr), ctypes.byref(nc), ctypes.byref(nb)))
        return int(nc.value), int(nb.value)

    def chunk_write(self, text_ptr: int, text_bytes: int, offsets_ptr: int, n_movies: int, max_chunk_size: int,
                    overlap: int, chunk_cu_ptr: int, byte_cu_ptr: int, movie_base: int, out_text_ptr: int,
                    out_offsets_ptr: int, out_movie_ptr: int, out_index_ptr: int):
        """Sentence chunking, write pass into the chunk CSR (device buffers; asynchronous)."""
        self._check(self._L.rse_chunk_write(self._h, c_void_p(text_ptr or 0), int(text_bytes), c_void_p(offsets_ptr),
                                            int(n_movies), int(max_chunk_size), int(overlap), c_void_p(chunk_cu_ptr),
                                            c_void_p(byte_cu_ptr), int(movie_base), c_void_p(out_text_ptr),
                                            c_void_p(out_offsets_ptr), c_void_p(out_movie_ptr), c_void_p(out_index_ptr)))

    def encode_texts(self, tok_slot: int, enc_slot: int, data: bytes, offsets, max_length: int):
        """Texts -> [n, hidden] float32 (head 0) / [n] logits (head 1) / [n, projection_dim] (a CLIP text tower with a
        BPE tokenizer): tokenized and encoded on the device."""
        txt, offs, n = self._texts(data, offsets)
        cfg = self._enc_cfg[int(enc_slot)]
        shape = (n, cfg.projection_dim) if isinstance(cfg, RseClipConfig) else (n, cfg.hidden) if cfg.head == 0 else (n,)
        out = np.zeros(shape, np.float32)
        self._check(self._L.rse_encode_texts(self._h, int(tok_slot), int(enc_slot), txt, c_void_p(offs.ctypes.data), n,
                                             int(max_length), c_void_p(out.ctypes.data)))
        return out

    def encode_texts_dev(self, tok_slot: int, enc_slot: int, data: bytes, offsets, max_length: int, out_ptr: int):
        txt, offs, n = self._texts(data, offsets)
        self._check(self._L.rse_encode_texts_dev(self._h, int(tok_slot), int(enc_slot), txt, c_void_p(offs.ctypes.data),
                                                 n, int(max_length), c_void_p(out_ptr)))

    def rerank_docs_load_texts(self, tok_slot: int, ids, data: bytes, offsets):
        """The rerank store from UTF-8 document texts, tokenized on the device (ids strictly ascending)."""
        ids = _c(ids, np.int64)
        txt, offs, n = self._texts(data, offsets)
        if n != len(ids):
            raise ValueError("offsets must have len(ids) + 1 entries")
        self._check(self._L.rse_rerank_docs_load_texts(self._h, int(tok_slot), c_void_p(ids.ctypes.data), len(ids), txt,
                                                       c_void_p(offs.ctypes.data)))

    def hybrid_rerank_timing(self):
        """Device ms of the last timed rerank run: (hybrid, assembly, encoder, order)."""
        out = (c_float * 4)()
        self._check(self._L.rse_hybrid_rerank_timing(self._h, out))
        return tuple(float(x) for x in out)

    # ------------------------------------------------------------------ multi-GPU (library-owned NCCL communicator)
    @staticmethod
    def comm_unique_id() -> bytes:
        """128-byte NCCL id; rank 0 creates it and hands it to the other ranks (any transport)."""
        L = load_library()
        buf = ctypes.create_string_buffer(128)
        rc = L.rse_comm_unique_id(buf)
        if rc != RSE_OK:
            msg = L.rse_last_error(None)
            raise RseError(rc, msg.decode() if msg else "rse_comm_unique_id failed")
        return bytes(buf.raw)

    def comm_init(self, id_bytes: bytes, n_ranks: int, rank: int):
        if len(id_bytes) != 128:
            raise ValueError("the NCCL unique id is 128 bytes")
        buf = ctypes.create_string_buffer(id_bytes, 128)
        self._check(self._L.rse_comm_init(self._h, buf, int(n_ranks), int(rank)))
        self.comm_ranks, self.comm_rank = int(n_ranks), int(rank)

    def comm_destroy(self):
        self._check(self._L.rse_comm_destroy(self._h))

    def comm_info(self):
        n, r, v = c_int32(0), c_int32(0), c_int32(0)
        self._check(self._L.rse_comm_info(self._h, ctypes.byref(n), ctypes.byref(r), ctypes.byref(v)))
        return int(n.value), int(r.value), int(v.value)

    def comm_exchange_candidates_dev(self, cand_ptr: int, nq: int, kprime: int, mine_ptr: int):
        self._check(self._L.rse_comm_exchange_candidates_dev(self._h, c_void_p(cand_ptr), int(nq), int(kprime),
                                                             c_void_p(mine_ptr)))

    def comm_allgather_dev(self, send_ptr: int, recv_ptr: int, bytes_per_rank: int):
        self._check(self._L.rse_comm_allgather_dev(self._h, c_void_p(send_ptr), c_void_p(recv_ptr), int(bytes_per_rank)))

    def knn_sharded_dev(self, q_all_ptr: int, nq_all: int, k: int, kprime: int, dist_ptr: int, rowid_ptr: int,
                        movie_ptr: int, count_ptr: int, flagged_ptr: int = 0):
        self._check(self._L.rse_knn_sharded_dev(self._h, c_void_p(q_all_ptr), int(nq_all), int(k), int(kprime),
                                                c_void_p(dist_ptr), c_void_p(rowid_ptr), c_void_p(movie_ptr),
                                                c_void_p(count_ptr), c_void_p(flagged_ptr or 0)))

    def hybrid_sharded_run_dev(self, mode: int, param: float, limit: int, q_all_ptr: int, nq_all: int, out_id_ptr: int,
                               out_score_ptr: int, out_a_ptr: int, out_b_ptr: int, out_count_ptr: int,
                               flagged_ptr: int = 0, knn_multiplier: int = 10, k1: float = 1.5, b: float = 0.75,
                               tie_mode: int = TIE_REFERENCE):
        self._check(self._L.rse_hybrid_sharded_run_dev(self._h, int(mode), float(param), int(tie_mode), int(limit),
                                                       int(knn_multiplier), float(k1), float(b), c_void_p(q_all_ptr),
                                                       int(nq_all), c_void_p(out_id_ptr), c_void_p(out_score_ptr),
                                                       c_void_p(out_a_ptr), c_void_p(out_b_ptr), c_void_p(out_count_ptr),
                                                       c_void_p(flagged_ptr or 0)))

    def hybrid_run_merged_dev(self, mode: int, param: float, limit: int, gathered_ptr: int, n_lists: int,
                              out_id_ptr: int, out_score_ptr: int, out_a_ptr: int, out_b_ptr: int, out_count_ptr: int,
                              knn_multiplier: int = 10, k1: float = 1.5, b: float = 0.75,
                              tie_mode: int = TIE_REFERENCE):
        self._check(self._L.rse_hybrid_run_merged_dev(self._h, int(mode), float(param), int(tie_mode), int(limit),
                                                      int(knn_multiplier), float(k1), float(b),
                                                      c_void_p(gathered_ptr), int(n_lists), c_void_p(out_id_ptr),
                                                      c_void_p(out_score_ptr), c_void_p(out_a_ptr),
                                                      c_void_p(out_b_ptr), c_void_p(out_count_ptr)))
