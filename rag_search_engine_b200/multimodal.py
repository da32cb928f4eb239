"""MultimodalSearch — drop-in for rag_search_engine.llm.multimodal.MultimodalSearch (SURVEY §8 f4) whose
image -> text search ranks on the B200.

The reference encodes every movie text with CLIP once, then per query image computes the cosine similarity to
ALL text embeddings in numpy and sorts them (llm/multimodal.py:86-95: normalise, ``text_normed @ image_vec``,
``np.argsort(...)[::-1][:top_k]``).  Here the text embeddings live in HBM and the ranking is the same cosine
top-k kernel the semantic path uses (``rse_knn``: exact fp32 cosine distance per row + radix top-k), so a search
is one scan instead of an O(N log N) host sort.  The CLIP model itself (image / text encoder) is NOT rewritten: it
is the pluggable ``model`` (``SentenceTransformer(model_name)`` when sentence-transformers is installed).

Same constructor arguments, method names, result dict keys and error behaviour as the reference.  Beyond the
reference: ``search_with_vectors`` / ``search_with_images`` rank a whole batch of image embeddings in one ``rse_knn``
call; a batch of two or more queries takes the tensor-core path (fp16 filter + exact fp32 re-score), whose results
are bit-identical to the exact scan, so row i equals ``search_with_vector`` of that row.
``similarity`` = 1 - cosine distance; it agrees with the reference's fp32 BLAS dot product to ~1e-7 (different
summation order), so two documents closer than that may swap places — numpy's argsort gives no tie guarantee
either.
"""
from __future__ import annotations

import os
from concurrent.futures import ThreadPoolExecutor
from typing import Dict, List, Optional, Sequence

import numpy as np

from . import _lib


class MultimodalSearch:
    def __init__(self, documents: Optional[List[Dict[str, object]]] = None, model_name: str = "clip-ViT-B-32", *,
                 model=None, device: int = 0) -> None:
        if model is None:
            from sentence_transformers import SentenceTransformer  # type: ignore  (llm/multimodal.py:28)
            model = SentenceTransformer(model_name)
        self.model = model
        self.documents: List[Dict[str, object]] = documents or []
        self.texts: List[str] = []
        self.text_embeddings: Optional[np.ndarray] = None
        self._index: Optional[_lib.Index] = None
        if self.documents:
            for doc in self.documents:                                           # llm/multimodal.py:35-38
                title = str(doc.get("title", "")).strip()
                desc = str(doc.get("description", doc.get("document", ""))).strip()
                self.texts.append(f"{title}: {desc}")
            self.text_embeddings = np.asarray(self.model.encode(self.texts, convert_to_numpy=True,
                                                                show_progress_bar=True), np.float32)
            self._index = _lib.Index(device)
            # automatic mode: batches take the tensor-core path at widths 64..512 (CLIP: 512), a single query keeps
            # the exact streaming scan at every width but 384
            self._index.load_embeddings(self.text_embeddings)

    def embed_image(self, image_path: str) -> np.ndarray:                        # llm/multimodal.py:46-58
        from PIL import Image  # type: ignore
        image = Image.open(image_path).convert("RGB")
        return self.model.encode([image], convert_to_numpy=True)[0]

    def search_with_vector(self, image_emb, top_k: int = 5) -> List[Dict[str, object]]:
        """The ranking step alone, for a precomputed (e.g. frozen) image embedding."""
        self._check_documents()
        q = np.ascontiguousarray(image_emb, np.float32).reshape(1, -1)
        return self._rank(q, top_k)[0]

    def search_with_vectors(self, image_embs, top_k: int = 5) -> List[List[Dict[str, object]]]:
        """The ranking step for a batch: ``image_embs`` [n, dim] in one device call; row i of the result equals
        ``search_with_vector(image_embs[i], top_k)``."""
        q = np.ascontiguousarray(image_embs, np.float32)
        if q.size == 0:
            self._check_documents()
            return []
        return self._rank(q.reshape(-1, q.shape[-1]), top_k)

    def search_with_images(self, image_paths: Sequence[str], top_k: int = 5) -> List[List[Dict[str, object]]]:
        """``search_with_image`` for a list of image files: every image is opened the way ``embed_image`` opens
        it (on a thread pool), the vision tower encodes them in one ``model.encode`` call and the batch is ranked in
        one device call."""
        self._check_documents()
        paths = list(image_paths)
        if not paths:
            return []
        from PIL import Image  # type: ignore

        def load(p):
            return Image.open(p).convert("RGB")
        # Pillow releases the GIL while it decodes: with the preprocessing on the device, decoding is the host's
        # whole share of the call, so the files are decoded in parallel (map keeps the input order)
        if len(paths) > 1:
            with ThreadPoolExecutor(max_workers=min(len(paths), os.cpu_count() or 1, 16)) as pool:
                images = list(pool.map(load, paths))
        else:
            images = [load(p) for p in paths]
        embs = np.asarray(self.model.encode(images, convert_to_numpy=True), np.float32)
        return self.search_with_vectors(embs, top_k=top_k)

    def _check_documents(self) -> None:
        if not self.documents or self.text_embeddings is None:
            raise ValueError("MultimodalSearch was initialized without documents; cannot run search_with_image.")

    def _rank(self, q: np.ndarray, top_k: int) -> List[List[Dict[str, object]]]:
        self._check_documents()
        top_k = min(int(top_k), len(self.documents))                             # llm/multimodal.py:93
        if top_k <= 0:
            return [[] for _ in range(q.shape[0])]
        if top_k > _lib.RSE_MAX_KPRIME:
            raise ValueError(f"top_k above {_lib.RSE_MAX_KPRIME} is not supported")
        dist, pos, _rowid, _movie, cnt = self._index.knn(q, top_k)
        out: List[List[Dict[str, object]]] = []
        for i in range(q.shape[0]):
            results: List[Dict[str, object]] = []
            for j in range(int(cnt[i])):
                idx = int(pos[i, j])
                doc = self.documents[idx]
                results.append({"id": doc.get("id", idx), "title": doc.get("title", ""),
                                "description": doc.get("description", doc.get("document", "")),
                                "similarity": float(1.0 - np.float64(dist[i, j]))})
            out.append(results)
        return out

    def search_with_image(self, image_path: str, top_k: int = 5) -> List[Dict[str, object]]:
        if not self.documents or self.text_embeddings is None:
            raise ValueError("MultimodalSearch was initialized without documents; cannot run search_with_image.")
        return self.search_with_vector(self.embed_image(image_path), top_k=top_k)

    def close(self) -> None:
        if self._index is not None:
            self._index.close()
            self._index = None
