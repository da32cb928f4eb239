/*
 * rse.h — C-ABI of librse.so, the B200-native retrieval core that replaces the
 * query hot path of JWSch4fer/rag-search-engine.
 *
 * Plain C: opaque handle, raw pointers and sizes, int status codes, no
 * exceptions and no torch/numpy types across the boundary.  The reference is
 * pure Python, so the reference-side binding is a ctypes stub (INTEGRATION.md);
 * each entry point names the reference interface it replaces (file:line are
 * relative to /root/reference/rag_search_engine/).
 *
 * Conventions
 *   - every function returns RSE_OK (0) or a negative RSE_ERR_* code;
 *     rse_last_error(h) gives the message (h may be NULL for rse_create).
 *   - "host" pointers are caller-owned CPU buffers; "dev" pointers are
 *     caller-owned device buffers on the handle's device (the *_dev entry
 *     points are what the torch.distributed host plumbing uses; they enqueue
 *     on the handle's stream and do not synchronise).
 *   - one handle = one device + one CUDA stream; calls on a handle are
 *     synchronous unless stated and not re-entrant (the reference objects are
 *     single-threaded too: utils/basesearch_db.py:40).
 *   - there is NO CPU fallback: without a CUDA device rse_create fails.
 */
#ifndef RSE_H_
#define RSE_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RSE_ABI_VERSION 2

#define RSE_OK 0
#define RSE_ERR_INVALID -1     /* bad argument */
#define RSE_ERR_CUDA -2        /* CUDA runtime error (message has the call) */
#define RSE_ERR_STATE -3       /* e.g. query before load */
#define RSE_ERR_UNSUPPORTED -4 /* outside documented limits */
#define RSE_ERR_NOMEM -5

/* Limits (documented in DESIGN.md §limits) */
#define RSE_VEC0_BLOCK 1024     /* sqlite-vec default chunk_size (semantic_search.py:96-99 passes none) */
#define RSE_MAX_KPRIME 4096     /* sqlite-vec caps k at 4096 */
#define RSE_MAX_BM25_K 512      /* rse_bm25 k; covers the k = 409 of a hybrid call at limit 409 */
#define RSE_MAX_FUSE_LIMIT 1024 /* rse_fuse_weighted / rse_fuse_rrf: a padded union of two 409-deep lists has 818 ids */
#define RSE_MAX_HYBRID_LIMIT 512 /* rse_hybrid*: also limit * knn_multiplier <= RSE_MAX_KPRIME (409 at multiplier 10) */
#define RSE_MAX_RERANK_LIMIT 128 /* rse_hybrid_rerank_run */
#define RSE_MAX_QUERY_TOKENS 255
#define RSE_RRF_NOT_FOUND 99999 /* hybrid_search.py:247 */
#define RSE_MAX_STASH 16        /* staged batches that can be parked in HBM (rse_hybrid_stash) */

/* tie_mode for the fusion entry points */
#define RSE_TIE_REFERENCE 0 /* CPython set iteration order of the id union (hybrid_search.py:148,248) */
#define RSE_TIE_BY_ID 1     /* deterministic by ascending id (north_star wording) */

typedef struct rse_index rse_index;

int rse_abi_version(void);

/* Create a handle bound to CUDA device `device`.  Fails (RSE_ERR_CUDA) when no
 * device is present.  Replaces the object construction at
 * utils/hybrid_search.py:41-54 (one KeywordSearch + one SemanticSearch). */
int rse_create(int32_t device, rse_index **out);
void rse_destroy(rse_index *h);
const char *rse_last_error(const rse_index *h);

/* Use an externally owned CUDA stream (cudaStream_t as void*), e.g. torch's current
 * stream.  NULL is the legacy default stream (what torch uses by default), NOT "unset";
 * rse_use_own_stream goes back to the handle's private non-blocking stream. */
int rse_set_stream(rse_index *h, void *cuda_stream);
int rse_use_own_stream(rse_index *h);
/* Block until everything enqueued on the handle's stream has finished. */
int rse_synchronize(rse_index *h);

/* ------------------------------------------------------------------ a1: vec0 store
 * Replaces the vec0 virtual table `chunk_embeddings` (semantic_search.py:94-101)
 * as the thing the KNN scans.  Rows are given in vec0 PHYSICAL layout: row i of
 * `emb` is (block pos_base/1024 + i/1024, slot i%1024); `valid[i]==0` marks an
 * empty slot (NULL: all valid).  `rowid` (NULL: rowid = pos_base + i) is
 * chunks.id; `movie_idx` (NULL: aggregation unavailable) is the dense index of
 * chunks.movie_id in the caller's sorted id universe, or -1 when the JOIN at
 * semantic_search.py:262-276 would drop the row.  pos_base must be a multiple of
 * 1024 (row shards are aligned to vec0 blocks).  use_fma selects the aarch64
 * (contracted) arithmetic of sqlite-vec instead of the x86-64 one.
 * The host variant copies; the dev variant BORROWS emb_dev (caller keeps it
 * alive) and copies the small side arrays. */
int rse_load_embeddings(rse_index *h, const float *emb_host, int64_t n_rows, int32_t dim,
                        const uint8_t *valid_host, const int64_t *rowid_host,
                        const int32_t *movie_idx_host, int64_t pos_base);
int rse_attach_embeddings_dev(rse_index *h, const float *emb_dev, int64_t n_rows, int32_t dim,
                              const uint8_t *valid_dev, const int64_t *rowid_dev,
                              const int32_t *movie_idx_dev, int64_t pos_base);
int rse_set_fma(rse_index *h, int32_t use_fma);
/* K4, the tcgen05 path for query batches (probe -> filter -> EXACT re-score, results identical to the
 * streaming scan): 0 = auto (batches of >= RSE_TC_MIN_BATCH queries on >= 256 k rows), 1 = never,
 * 2 = whenever the shape allows it.  K4 serves embedding widths dim = 64 KB, KB = 1..8 (64..512, e.g. 384 for
 * MiniLM, 512 for CLIP); any other width always takes the exact scan.  The probe/filter GEMM runs over an fp16
 * normalised shadow of the corpus (knn_tc3.cuh; built once at the first batch that needs it, +2 * dim B per row
 * of device memory: 768 B at 384).  Measured on
 * S-600k (bench.py knn_small_batches, r02): the K4 chain costs 0.75-0.82 ms per call for 1..64 queries, the exact
 * scan 1.21 / 1.41 / 1.65 / 1.72 / 2.32 / 3.98 ms for 1 / 2 / 3 / 4 / 8 / 16 — K4 wins from the first query on.  A
 * single query takes the exact streaming scan (north_star: batch-1 = the HBM-bound kernel; no shadow needed) until
 * a batch has built the shadow, and K4 from then on at dim 384 (the width that was measured; at any other width a
 * single query stays on the exact scan in auto mode); mode 2 sends it through K4 from the start. */
#define RSE_TC_MIN_BATCH 2
int rse_set_tc_mode(rse_index *h, int32_t mode);

/* Which BM25 kernels serve rse_bm25 / rse_hybrid for k <= 32 (results are bit-identical in every mode):
 * 0 = fixed-point streaming kernel + exact re-score of the finalists (default), 1 = streaming kernel that
 * keeps the reference's summation order with one barrier per (range, token) slice, 2 = general kernel only
 * (one CTA per range and query; what k > 32, > 16 tokens and flagged queries always use). */
int rse_set_bm25_mode(rse_index *h, int32_t mode);

/* KNN: `embedding MATCH :q AND k = :k ... ORDER BY knn.distance`
 * (semantic_search.py:254-279).  Q is [nq, dim] fp32.  Outputs are [nq, kprime]
 * in vec0 emit order (distance asc, block asc, slot desc); out_count[q] <= kprime
 * rows are valid.  out_pos / out_rowid / out_movie_idx may be NULL. */
int rse_knn(rse_index *h, const float *q_host, int32_t nq, int32_t kprime, float *out_dist,
            int64_t *out_pos, int64_t *out_rowid, int32_t *out_movie_idx, int32_t *out_count);

/* KNN + best-chunk-per-movie aggregation = SemanticSearch.query_top_k numerics
 * (semantic_search.py:250-317): top-kprime chunks, first row per movie, first k.
 * Outputs [nq, k]. */
int rse_knn_movies(rse_index *h, const float *q_host, int32_t nq, int32_t k, int32_t kprime,
                   float *out_dist, int64_t *out_chunk_rowid, int32_t *out_movie_idx,
                   int32_t *out_count);

/* Exact movie-level KNN: the k nearest movies by best chunk over EVERY row (DESIGN §11).  Outputs [nq, k] as
 * rse_knn_movies; out_scanned (may be NULL) = queries that needed the full segmented scan.  1 <= k <= 4096.
 * A movie's best chunk is its row with the smallest (distance, block asc, slot desc) key; rows with valid = 0 or
 * movie_idx = -1 never compete; movies are ordered by their best key and the first min(k, movies) are returned,
 * each distance bit-identical to rse_knn's for that row (rse_set_fma honoured).  Prefix property: where
 * rse_knn_movies(k, K') returns k movies for a query the two results are identical, and where it returns fewer its
 * list is a prefix of this one.  RSE_ERR_UNSUPPORTED for k > 4096; RSE_ERR_STATE without a corpus or movie_idx.
 * RSE_MOVIES_EXACT_BUDGET (bytes, read by rse_create; default 512 MB) bounds the [queries, movies] u64 key buffer
 * of the segmented scan, i.e. how many queries one pass over the corpus serves.  With rse_set_timing on, the call's
 * H2D → D2H time lands in last_knn_total_ms and its scan launches in scan_ms_total. */
int rse_knn_movies_exact(rse_index *h, const float *q_host, int32_t nq, int32_t k, float *out_dist,
                         int64_t *out_chunk_rowid, int32_t *out_movie_idx, int32_t *out_count,
                         int32_t *out_scanned);

/* Device-pointer building blocks for the row-sharded multi-GPU path (SURVEY §8e).
 * Local top-kprime as packed candidates: cand_dev is [nq, kprime, 3] int64 =
 * {key, rowid, movie_idx}; key = (orderable(distance) << 32) | (global_pos ^ 1023),
 * so ascending key IS the vec0 emit order; unused tail entries have key = -1
 * (all ones).  q_dev is [nq, dim] fp32 on the device.  Asynchronous on the handle's stream when
 * the exact scan serves the batch; the tensor-core path (rse_set_tc_mode) synchronises once to
 * read its per-query overflow flags. */
int rse_knn_local_dev(rse_index *h, const float *q_dev, int32_t nq, int32_t kprime,
                      int64_t *cand_dev);
/* Keep a row-sharded step free of host round trips: with deferral enabled rse_knn_local_dev never
 * synchronises — a query the tensor-core path could not finish (survivor overflow: a mass tie at the K'-th
 * distance) keeps key = -1 candidates and is only COUNTED: rse_knn_flags_dev enqueues `*flagged_dev +=
 * (flagged queries of the last rse_knn_local_dev)` on the handle's stream.  The caller lets that counter travel
 * with the step's results and repeats a step whose global count is non-zero with deferral off. */
int rse_set_defer_flags(rse_index *h, int32_t enabled);
int rse_knn_flags_dev(rse_index *h, int32_t *flagged_dev);
/* Merge n_lists candidate lists per query (gathered_dev is [n_lists, nq, kprime, 3],
 * the layout all_gather produces), keep the first kprime under the key order, then
 * aggregate per movie like rse_knn_movies.  Outputs are DEVICE buffers [nq, k]. */
int rse_knn_merge_movies_dev(rse_index *h, const int64_t *gathered_dev, int32_t n_lists,
                             int32_t nq, int32_t k, int32_t kprime, float *out_dist_dev,
                             int64_t *out_chunk_rowid_dev, int32_t *out_movie_idx_dev,
                             int32_t *out_count_dev);

/* ------------------------------------------------------------------ a6: BM25 index
 * Replaces the SQLite tables terms/postings/doclen as the thing
 * KeywordSearch.search (keyword_search.py:180-250) scores against.
 *   indptr[T+1], doc_idx[P] (dense doc index, ascending within a term — the
 *   order the (term_id, doc_id) autoindex yields, :214-218), tf[P] =
 *   len(positions) (:227-228), df[T] = len(rows) (:222; may exceed the CSR
 *   length when postings without a doclen row were dropped, :235-236),
 *   dl[M] = doclen.length, n_movies = COUNT(movies) (:196), avgdl = AVG(length)
 *   (:197-198). */
int rse_load_bm25(rse_index *h, const int64_t *indptr, const uint32_t *doc_idx, const uint32_t *tf,
                  const int64_t *df, int64_t n_terms, int64_t n_postings, const uint32_t *dl,
                  int64_t n_docs, int64_t n_movies, double avgdl);

/* BM25 top-k for a batch of tokenised queries.  tok_indptr[nq+1] delimits each
 * query's tokens in `term_rows` (CSR term row per token in query order,
 * duplicates kept, -1 = unknown term, skipped: keyword_search.py:205-210).
 * Outputs [nq, k]: scores (fp64, bit-exact reference arithmetic :224,:241-244),
 * dense doc indices, and per-query counts.  Order = sorted(..., reverse=True)
 * with dict-insertion tie order (:250).  1 <= k <= RSE_MAX_BM25_K (512); above 256 the
 * candidate lists of one call are held to 256 MB by scoring the batch in query chunks. */
int rse_bm25(rse_index *h, const int32_t *tok_indptr, const int32_t *term_rows, int32_t nq,
             int32_t k, double k1, double b, double *out_score, int32_t *out_doc_idx,
             int32_t *out_count);

/* ------------------------------------------------------------------ a8-a10: fusion
 * ids are the caller's document ids (movies.id).  Inputs [nq, limit] with
 * per-query counts; BM25 lists are score-descending, semantic lists
 * distance-ascending (what the retrievers return).  Distances are doubles: the
 * reference does float(hit["distance"]) on whatever the plugged-in retriever
 * returns (hybrid_search.py:134); vec0 distances are f32 values widened.  Outputs [nq, limit].
 * weighted: hybrid_search.py:117-180 (min_max_norm utils.py:182-191,
 *           alpha*b + (1-alpha)*s :163).
 * rrf:      hybrid_search.py:217-272,379 (0-based ranks, NOT_FOUND=99999 :247,
 *           1/(k+r_b) + 1/(k+r_s) :255); out ranks are -1 for None.
 * 1 <= limit <= RSE_MAX_FUSE_LIMIT (1024). */
int rse_fuse_weighted(rse_index *h, int32_t nq, int32_t limit, double alpha, int32_t tie_mode,
                      const int64_t *bm25_id, const double *bm25_score, const int32_t *bm25_count,
                      const int64_t *sem_id, const double *sem_dist, const int32_t *sem_count,
                      int64_t *out_id, double *out_bm25, double *out_sem, double *out_score,
                      int32_t *out_count);
int rse_fuse_rrf(rse_index *h, int32_t nq, int32_t limit, double k, int32_t tie_mode,
                 const int64_t *bm25_id, const double *bm25_score, const int32_t *bm25_count,
                 const int64_t *sem_id, const double *sem_dist, const int32_t *sem_count,
                 int64_t *out_id, double *out_score, int32_t *out_bm25_rank, int32_t *out_sem_rank,
                 int32_t *out_count);

/* ------------------------------------------------------------------ hybrid, end to end
 * HybridSearch.rrf_search / weighted_search numerics for a batch (hybrid_search.py:91-180,
 * 183-272): BM25(k=limit) + KNN(k=limit, kprime=max(limit*knn_multiplier, limit),
 * semantic_search.py:251) + fusion, all on the device, one host round trip.
 * doc_ids[n_docs] / movie_ids[n_movies_uni] map dense indices to movies.id (set with
 * rse_set_id_tables).  mode: 0 = rrf (param = k), 1 = weighted (param = alpha).
 * Outputs [nq, limit]; out_a/out_b = (bm25_rank, sem_rank) as doubles for rrf
 * (-1 = None) or (bm25_norm, sem_norm) for weighted.  Every hybrid entry point takes
 * 1 <= limit <= RSE_MAX_HYBRID_LIMIT (512) with max(limit * knn_multiplier, limit) <= RSE_MAX_KPRIME:
 * the reference's own ceiling at its multiplier 10 is limit 409 (sqlite-vec refuses k > 4096). */
int rse_set_id_tables(rse_index *h, const int64_t *doc_ids, int64_t n_docs, const int64_t *movie_ids,
                      int64_t n_movie_ids);
int rse_hybrid(rse_index *h, int32_t mode, double param, int32_t tie_mode, int32_t limit,
               int32_t knn_multiplier, int32_t nq, const float *q_host, const int32_t *tok_indptr,
               const int32_t *term_rows, double k1, double b, int64_t *out_id, double *out_score,
               double *out_a, double *out_b, int32_t *out_count);
/* The same call split in three, for callers that keep a query batch resident in HBM
 * (rse_hybrid == stage + run + fetch):
 *   stage: upload query vectors + tokens (+ host-computed idf, keyword_search.py:224);
 *   run:   BM25 + KNN + aggregation + fusion on the staged batch; asynchronous on the
 *          handle's stream, results stay on the device; may be repeated;
 *   fetch: copy the [nq, limit] results to the host and synchronise. */
int rse_hybrid_stage(rse_index *h, int32_t nq, const float *q_host, const int32_t *tok_indptr,
                     const int32_t *term_rows);
int rse_hybrid_run(rse_index *h, int32_t mode, double param, int32_t tie_mode, int32_t limit,
                   int32_t knn_multiplier, double k1, double b);
/* Row-sharded variant of `run` (SURVEY §8e): the KNN stage is replaced by the merge of
 * n_lists gathered candidate lists ([n_lists, nq, kprime, 3] from rse_knn_local_dev on every
 * shard + all_gather); the staged batch is this rank's query slice.  Outputs are DEVICE
 * buffers [nq, limit] (they feed the final all_gather).  Asynchronous on the handle's stream. */
int rse_hybrid_run_merged_dev(rse_index *h, int32_t mode, double param, int32_t tie_mode, int32_t limit,
                              int32_t knn_multiplier, double k1, double b, const int64_t *gathered_dev,
                              int32_t n_lists, int64_t *out_id_dev, double *out_score_dev,
                              double *out_a_dev, double *out_b_dev, int32_t *out_count_dev);
int rse_hybrid_fetch(rse_index *h, int32_t limit, int64_t *out_id, double *out_score, double *out_a,
                     double *out_b, int32_t *out_count);
/* EXCHANGE the staged batch with stash slot `slot` (0 .. RSE_MAX_STASH-1); pointer swaps on the host, no device
 * work.  stage(A); stash(0); stage(B); stash(1) parks two batches in HBM; a later stash(0) makes A the staged
 * batch again (and parks whatever was staged).  For callers that rotate over several RESIDENT batches. */
int rse_hybrid_stash(rse_index *h, int32_t slot);
/* Pipelined form of rse_hybrid for a serving loop: at most TWO batches in flight per handle.
 *   submit : stage (host buffers -> pinned -> device, asynchronous) + run + an asynchronous copy of
 *            the results into a pinned slot owned by the handle; returns a ticket.  It returns as
 *            soon as the batch is ENQUEUED — it never waits for the device — so the caller submits
 *            batch i+1 before collecting batch i and the device does not idle between batches.
 *            Caller buffers may be reused as soon as submit returns.
 *   collect: wait for the ticket's results and copy them out; tickets are collected in submission
 *            order.  out_nq / out_limit (optional) report the batch's shape.  The tensor-core
 *            path's per-query overflow flags (a mass tie at the K'-th distance; rse_hybrid waits
 *            for them in mid-batch) are checked HERE: a batch with a flagged query is re-run
 *            through rse_hybrid from the handle's copies of its inputs before collect returns.
 * Results are those of rse_hybrid on the same inputs.  A third submit before a collect returns
 * RSE_ERR_STATE.  Not to be interleaved with stage/run/fetch between a submit and its collect. */
int rse_hybrid_submit(rse_index *h, int32_t mode, double param, int32_t tie_mode, int32_t limit,
                      int32_t knn_multiplier, int32_t nq, const float *q_host,
                      const int32_t *tok_indptr, const int32_t *term_rows, double k1, double b,
                      int64_t *ticket);
int rse_hybrid_collect(rse_index *h, int64_t ticket, int32_t *out_nq, int32_t *out_limit,
                       int64_t *out_id, double *out_score, double *out_a, double *out_b,
                       int32_t *out_count);
/* Wait for and DISCARD every ticket still in flight (a consumer that stops early, an error between a
 * submit and its collect): afterwards the handle accepts submits again.  out_dropped (optional) = how many. */
int rse_hybrid_drain(rse_index *h, int32_t *out_dropped);

/* ------------------------------------------------------------------ §8(f2)/(f3): the text encoders on the device
 * The reference encodes every query text with SentenceTransformer("all-MiniLM-L6-v2") on the CPU
 * (utils/semantic_search.py:45, :211-222: model.encode -> float32[1, 384]) and reranks the fused hits with
 * CrossEncoder("cross-encoder/ms-marco-TinyBERT-L2-v2").predict(pairs) (utils/hybrid_search.py:279-312).  Both are
 * HuggingFace BertModels; here one implementation runs either next to the index (csrc/encoder.cuh):
 *   head 0 : BertModel -> mean pooling over the tokens -> L2 normalise  (the sentence-transformers pipeline);
 *            output [n_seq, hidden]
 *   head 1 : BertModel -> pooler (tanh(dense([CLS]))) -> classifier (num_labels = 1); output [n_seq] logits
 * Weights are handed over tensor by tensor under their HuggingFace state_dict names (any prefix such as "bert." or
 * "0.auto_model." is ignored).  rse_encode takes token ids (any tokenizer, run by the caller) and rse_encode_texts
 * takes the texts themselves (BERT WordPiece on the device, see "BERT WordPiece on the device" below).  The ids come
 * PACKED — ids[T] (+ optional token_type_ids[T], NULL = all 0) and cu_seqlens[n_seq + 1]
 * (sequence s owns tokens cu[s] .. cu[s+1]; what attention_mask == 1 selects).  fp32 throughout.
 * rse_encode_dev leaves the result on the device (out_dev on the handle's device, asynchronous on its stream), so
 * rse_hybrid_stage_dev can take the query vectors from there: text in, no host hop for the vectors. */
#define RSE_MAX_ENCODERS 2
typedef struct rse_encoder_config {
  int32_t vocab_size, hidden, layers, heads, intermediate, max_positions, type_vocab;
  float ln_eps;
  int32_t head; /* 0 = mean pool + L2 normalise, 1 = BERT pooler + 1-logit classifier */
} rse_encoder_config;
int rse_encoder_create(rse_index *h, int32_t slot, const rse_encoder_config *cfg);
int rse_encoder_set_tensor(rse_index *h, int32_t slot, const char *name, const float *data, int64_t n_elem);
int rse_encoder_finalize(rse_index *h, int32_t slot);
/* Which GEMM the encoder's linear layers run on (results agree to ~1e-6 relative; both meet the 1e-5 bar):
 * 0 = tcgen05 kind::tf32 tensor cores with a 3-pass hi/lo split of both operands (fp32-class accuracy; default
 * when every GEMM dimension is a multiple of 128), 1 = fp32 SIMT (fmaf). */
int rse_encoder_set_mode(rse_index *h, int32_t slot, int32_t mode);
int rse_encode(rse_index *h, int32_t slot, const int32_t *ids, const int32_t *type_ids, const int32_t *cu_seqlens,
               int32_t n_seq, float *out_host);
int rse_encode_dev(rse_index *h, int32_t slot, const int32_t *ids, const int32_t *type_ids,
                   const int32_t *cu_seqlens, int32_t n_seq, float *out_dev);

/* ------------------------------------------------------------------ §10 f4: the CLIP towers of the image search
 * The reference's MultimodalSearch runs SentenceTransformer("clip-ViT-B-32") (llm/multimodal.py:35-42 encodes every
 * document text, :46-58 every query image): HuggingFace CLIPTextModelWithProjection / CLIPVisionModelWithProjection,
 * fp32, output not normalised.  rse_clip_create puts one tower into an encoder slot (csrc/clip.cuh); the slot then
 * takes rse_encoder_set_tensor (names "vision_model.*" + "visual_projection.weight", or "text_model.*" +
 * "text_projection.weight"; q / k / v projections are fused on the device; a prefix such as "model." is ignored),
 * rse_encoder_finalize (fails while a tensor is missing) and rse_encoder_set_mode like a BERT slot.
 *   text tower   : rse_encode / rse_encode_dev with type_ids = NULL -> [n_seq, projection_dim]; sequences of
 *                  1 .. max_positions tokens (truncate on the host).  The pooled token follows transformers:
 *                  eos_token_id == 2 -> first argmax of the ids, else first position of eos_token_id (0 if none).
 *   vision tower : rse_encode_images(_dev) with the image processor's pixel_values [n, 3, image_size, image_size]
 *                  (NCHW fp32) -> [n, projection_dim].
 * Shapes: hidden % 32 == 0 and <= 1024, head_dim 32 or 64, image_size % patch_size == 0, at most RSE_CLIP_MAX_TOKENS
 * tokens per sequence (text max_positions, vision (image_size / patch_size)^2 + 1); else RSE_ERR_UNSUPPORTED. */
#define RSE_CLIP_MAX_TOKENS 1024
typedef struct rse_clip_config {
  int32_t tower; /* 0 = vision, 1 = text */
  int32_t hidden, layers, heads, intermediate, projection_dim;
  int32_t vocab_size, max_positions;  /* text */
  int32_t image_size, patch_size;     /* vision */
  int32_t eos_token_id;               /* text */
  float ln_eps;
} rse_clip_config;
int rse_clip_create(rse_index *h, int32_t slot, const rse_clip_config *cfg);
int rse_encode_images(rse_index *h, int32_t slot, const float *pixels_host, int32_t n, float *out_host);
int rse_encode_images_dev(rse_index *h, int32_t slot, const float *pixels_dev, int32_t n, float *out_dev);

/* ------------------------------------------------------------------ CLIP image preprocessing on the device
 * transformers' CLIPImageProcessor (backend 0: torchvision, aten's uint8 antialiased bicubic) or
 * CLIPImageProcessorPil (backend 1: Pillow's bicubic) from decoded RGB pixels, bit for bit (csrc/imgproc.cuh):
 * resize to shortest_edge, center crop, rescale / normalise, CHW.  rse_imgproc_set binds a configuration to a CLIP
 * vision slot (a new one replaces it); it requires do_resize and do_center_crop, crop_height == crop_width == the
 * tower's image_size <= shortest_edge (so the processor never pads), rescale_factor > 0 and std != 0.
 * Images: n packed HWC uint8 RGB in host memory, image i at byte offsets[i] with height hw[2i], width hw[2i + 1]:
 *   rse_image_preprocess(_dev)  -> pixel_values [n, 3, image_size, image_size] fp32, host or device memory;
 *   rse_encode_images_u8(_dev)  -> the vision tower's [n, projection_dim], host or device memory.
 * The pixels go up in chunks of at most RSE_IMGPROC_CHUNK_BYTES through pinned staging, the copy of one chunk
 * overlapping the kernels of the previous.  Per image, outside these limits RSE_ERR_UNSUPPORTED (the message names
 * the image): H * W <= RSE_IMGPROC_MAX_PIXELS, each resized side <= RSE_IMGPROC_MAX_EDGE, a downscale of at most
 * RSE_IMGPROC_MAX_SCALE per axis, and (backend 1) not more than 100 times taller than wide while shrinking vertically
 * (Pillow then runs the vertical pass first).  A slot that is not a CLIP vision tower: RSE_ERR_INVALID; one without
 * a configuration: RSE_ERR_STATE. */
#define RSE_IMGPROC_MAX_PIXELS (1 << 24)
#define RSE_IMGPROC_MAX_EDGE 65536
#define RSE_IMGPROC_MAX_SCALE 32
#define RSE_IMGPROC_CHUNK_BYTES (64 << 20)
typedef struct rse_imgproc_cfg {
  int32_t backend;                   /* 0 = CLIPImageProcessor (torchvision), 1 = CLIPImageProcessorPil */
  int32_t shortest_edge;
  int32_t crop_height, crop_width;
  int32_t do_resize, do_center_crop, do_rescale, do_normalize;
  double rescale_factor;
  double mean[3], std[3];
} rse_imgproc_cfg;
int rse_imgproc_set(rse_index *h, int32_t vision_slot, const rse_imgproc_cfg *cfg);
int rse_image_preprocess(rse_index *h, int32_t slot, const uint8_t *pixels, const int64_t *offsets,
                         const int32_t *hw, int32_t n, float *out_host);
int rse_image_preprocess_dev(rse_index *h, int32_t slot, const uint8_t *pixels, const int64_t *offsets,
                             const int32_t *hw, int32_t n, float *out_dev);
int rse_encode_images_u8(rse_index *h, int32_t slot, const uint8_t *pixels, const int64_t *offsets,
                         const int32_t *hw, int32_t n, float *out_host);
int rse_encode_images_u8_dev(rse_index *h, int32_t slot, const uint8_t *pixels, const int64_t *offsets,
                             const int32_t *hw, int32_t n, float *out_dev);

/* rse_hybrid_stage with the query vectors already ON THE DEVICE ([nq, dim] fp32, e.g. rse_encode_dev's output);
 * tokens still come from the host.  Followed by rse_hybrid_run / rse_hybrid_fetch as usual. */
int rse_hybrid_stage_dev(rse_index *h, int32_t nq, const float *q_dev, const int32_t *tok_indptr,
                         const int32_t *term_rows);

/* ------------------------------------------------------------------ cross-encoder rerank of a fused batch
 * HybridSearch.rrf_search(..., rerank_method="cross_encoder") (hybrid_search.py:279-312) for a whole staged batch, on
 * the device (csrc/rerank.cuh): RRF over the WHOLE union of the two hit lists (up to 2 * limit ids per query), one
 * (query, document) pair per union member scored by the cross-encoder of an encoder slot, a stable descending sort on
 * (cross_encoder_score, rrf_score), the first `limit`.
 *   rse_rerank_docs_load : the document-token store.  ids[n_docs] strictly ascending (the movies.id universe);
 *                          tok_indptr[n_docs + 1] (from 0, non-decreasing) / tokens = the cross-encoder tokenizer's
 *                          ids of each document's text f"{title} - {description}" WITHOUT special tokens.  4 B per
 *                          token in HBM.  A new load replaces the store.
 *   rse_hybrid_rerank_run: on the batch staged by rse_hybrid_stage / rse_hybrid_stage_dev.  q_tok_indptr[nq + 1] /
 *                          q_tok_ids = the cross-encoder tokenizer's ids of each query (no special tokens); cls_id /
 *                          sep_id its [CLS] / [SEP].  A pair is [CLS] q[:a] [SEP] d[:b] [SEP] with token types 0 for
 *                          the first a + 2 tokens and 1 for the rest, (a, b) by the HF fast tokenizers' longest_first
 *                          truncation to max_length (rse_pair_truncate).  activation 0 = the classifier logit, 1 =
 *                          float32(1 / (1 + exp(-logit))) in fp64.  Synchronises ONCE, after the pairs are assembled,
 *                          to cut them into encoder slices (rse_set_rerank_token_budget) — besides the wait for the
 *                          tensor-core KNN's overflow flags that every hybrid step has.  The plain hybrid results of
 *                          the staged batch (rse_hybrid_fetch) are not touched.
 *                          RSE_ERR_STATE: no store, nothing staged, submit tickets in flight, or a fused id missing
 *                          from the store (the message names the first).  RSE_ERR_INVALID: the slot is not a finalized
 *                          head-1 BERT, activation not 0 / 1, a query / store / cls / sep token >= vocab_size.
 *                          RSE_ERR_UNSUPPORTED: limit outside [1, 128], max_length < 4 or > max_positions.
 *   rse_hybrid_rerank_fetch: [nq, limit] id, rrf score, bm25_rank / sem_rank (0-based, -1 = None), rrf_rank (1-based
 *                          fused position), cross-encoder score; count[nq].  Synchronises.
 *   rse_set_rerank_token_budget: most tokens per encoder slice (default 131072: the TinyBERT encoder's scratch is
 *                          ~9 KB per token); a pair longer than the budget is a slice of its own.  Results do not
 *                          depend on it.
 *   rse_hybrid_rerank_timing: with rse_set_timing on, device ms of the last run's hybrid / assembly / encoder / order
 *                          stages (out_ms[4]).  Synchronises.
 *   rse_pair_truncate    : the truncation rule alone (host arithmetic, no handle): n1 query and n2 document tokens
 *                          -> the (a, b) kept for max_length (>= 4). */
int rse_rerank_docs_load(rse_index *h, const int64_t *ids, int64_t n_docs, const int64_t *tok_indptr,
                         const int32_t *tokens);
int rse_hybrid_rerank_run(rse_index *h, int32_t slot, double k, int32_t tie_mode, int32_t limit,
                          int32_t knn_multiplier, double k1, double b, const int32_t *q_tok_indptr,
                          const int32_t *q_tok_ids, int32_t cls_id, int32_t sep_id, int32_t max_length,
                          int32_t activation);
int rse_hybrid_rerank_fetch(rse_index *h, int32_t limit, int64_t *out_id, double *out_score,
                            int32_t *out_bm25_rank, int32_t *out_sem_rank, int32_t *out_rrf_rank,
                            float *out_ce_score, int32_t *out_count);
int rse_set_rerank_token_budget(rse_index *h, int64_t tokens);
int rse_hybrid_rerank_timing(rse_index *h, float *out_ms);
int rse_pair_truncate(int32_t n1, int32_t n2, int32_t max_length, int32_t *a, int32_t *b);

/* ------------------------------------------------------------------ BERT WordPiece on the device
 * The tokenizers of both reference models (all-MiniLM-L6-v2, ms-marco-TinyBERT-L2-v2: HF BertTokenizerFast, the
 * uncased BERT WordPiece vocab) run on the device (csrc/wordpiece.cuh) with ids identical to the HF fast tokenizer:
 * the special tokens split off the raw text (literal, leftmost-longest), BertNormalizer, BertPreTokenizer, greedy
 * longest-match WordPiece, optional [CLS] ... [SEP] and truncation.  Texts are UTF-8, back to back in `text`;
 * offsets[n + 1] (from 0, non-decreasing) delimit them in bytes.  They go up through a pinned buffer.
 *   rse_tokenizer_load : a tokenizer into a slot (a new load replaces it).  The description is built from the HF object
 *                        by rag_search_engine_b200/wordpiece.py: cp_map / cp_class for every code point (what the
 *                        normaliser makes of it, how the pre-tokenizer classes it), the two tries of word-initial and
 *                        "##" pieces, the special ids and the added-token strings.  Every index is checked here.
 *   rse_tokenize       : tokenize n texts into the handle's buffers.  add_special 1 = [CLS] pieces[:max_length - 2]
 *                        [SEP] (the sentence encoder's input), 0 = pieces[:max_length] (the cross-encoder's single
 *                        texts); max_length <= 0 keeps every piece.  out_total / out_max_len (may be NULL): ids in all,
 *                        the longest sequence.  Synchronises once, for those two numbers.
 *   rse_tokens_fetch   : the last rse_tokenize's ids[total] and cu_seqlens[n + 1] to host memory (synchronises), or
 *   rse_tokens_fetch_dev : to device memory (asynchronous on the handle's stream).
 *   rse_encode_texts(_dev): tokenize with [CLS] / [SEP] at max_length (2 .. max_positions) and run the BERT slot
 *                        enc_slot on the ids where they are: rse_encode's output without host id lists.  One small
 *                        device-to-host copy per call (the token total and the longest sequence the encoder launch needs).
 *   rse_rerank_docs_load_texts: the store rse_rerank_docs_load would hold for the same ids and the tokenizer's ids of
 *                        each text (no special tokens, no cut), built on the device.  ids[n_docs] strictly ascending.
 * Errors: an unloaded slot RSE_ERR_STATE; bad offsets and malformed UTF-8 (the message names the first text)
 * RSE_ERR_INVALID.  NFD (accent stripping) reorders combining marks by canonical class; the tables map each code point
 * on its own, so a text with two code points whose marks survive the stripping (spacing marks of a non-zero class:
 * the Mc viramas of Javanese, Balinese, Sundanese, Batak, Tagalog, Grantha and a few other scripts, the musical
 * symbol stems) is refused with RSE_ERR_UNSUPPORTED, never tokenized differently, even when a starter separates the
 * two; the Python layer hands those texts to the host tokenizer.  Without accent stripping nothing is refused.  Limits: max_input_chars_per_word <= 256, <= 32 added tokens, < 2^31
 * ids per call. */
#define RSE_MAX_TOKENIZERS 2
typedef struct rse_wordpiece_desc {
  const uint32_t *cp_map;       /* [0x110000]: bits 0-20 code point or extra row, 21-22 count (0-3), 23 reorder flag */
  const uint32_t *extra;        /* [n_extra][3] code points of the 2- and 3-code-point outputs */
  int32_t n_extra;
  const uint8_t *cp_class;      /* [0x110000]: 0 other, 1 whitespace, 2 punctuation */
  const int32_t *node_first;    /* [n_nodes + 1]: node 0 = word-initial root, node 1 = continuation root */
  const int32_t *node_id;       /* [n_nodes]: vocab id of the piece ending at the node, -1 none */
  int32_t n_nodes;
  const int32_t *edge_cp;       /* [node_first[n_nodes]], ascending within a node */
  const int32_t *edge_child;
  const char *added;            /* added-token strings (UTF-8) back to back */
  const int32_t *added_offsets; /* [n_added + 1] */
  const int32_t *added_ids;     /* [n_added] */
  int32_t n_added;
  int32_t unk_id, cls_id, sep_id, max_input_chars_per_word;
} rse_wordpiece_desc;
int rse_tokenizer_load(rse_index *h, int32_t slot, const rse_wordpiece_desc *desc);
int rse_tokenize(rse_index *h, int32_t slot, const char *text, const int64_t *offsets, int32_t n, int32_t add_special,
                 int32_t max_length, int64_t *out_total, int32_t *out_max_len);
int rse_tokens_fetch(rse_index *h, int32_t *ids_host, int32_t *cu_seqlens_host);
int rse_tokens_fetch_dev(rse_index *h, int32_t *ids_dev, int32_t *cu_seqlens_dev);
int rse_encode_texts(rse_index *h, int32_t tok_slot, int32_t enc_slot, const char *text, const int64_t *offsets,
                     int32_t n, int32_t max_length, float *out_host);
int rse_encode_texts_dev(rse_index *h, int32_t tok_slot, int32_t enc_slot, const char *text, const int64_t *offsets,
                         int32_t n, int32_t max_length, float *out_dev);
int rse_rerank_docs_load_texts(rse_index *h, int32_t tok_slot, const int64_t *ids, int64_t n_docs, const char *text,
                               const int64_t *offsets);

/* ------------------------------------------------------------------ the semantic index build on the device
 * The chunk texts of SemanticSearch's build (semantic_search.py:164-188, store.plan_chunks) and their embeddings,
 * without host strings (csrc/chunk.cuh).  Movie m of n_movies is two texts of the device buffer text_dev
 * (text_bytes bytes, UTF-8): its title text_dev[offsets[2m], offsets[2m+1]) and its description
 * text_dev[offsets[2m+1], offsets[2m+2]); offsets_dev[2 n_movies + 1] must lie in [0, text_bytes] and not decrease
 * (checked on the device: RSE_ERR_INVALID names the first bad entry); they need not start at 0, so a slice of the
 * offsets addresses a part of the movies in the same buffer.  Chunk 0 of a movie is its title,
 * verbatim; chunk w + 1 is window w of the stripped description's sentences (Python's 29 whitespace code points; split
 * at every whitespace run that follows '.', '!' or '?'; windows of max_chunk_size sentences, the next one carrying
 * the last `overlap` of the previous when 0 < overlap < max_chunk_size) joined without a separator.
 *   rse_chunk_count : chunk_cu_dev[n_movies + 1] / byte_cu_dev[n_movies + 1] (int64, device) = exclusive prefix
 *                     sums of each movie's chunks and chunk-text bytes; out_n_chunks / out_n_bytes the totals.
 *                     Synchronises once.  max_chunk_size < 1: RSE_ERR_INVALID.
 *   rse_chunk_write : with the same movies and the scans rse_chunk_count wrote, every chunk text back to back at
 *                     out_text_dev (out_n_bytes bytes), out_offsets_dev[n_chunks + 1] their byte offsets (from 0), out_movie_dev /
 *                     out_index_dev[n_chunks] its movie row (movie_base + m) and chunk_index.  Asynchronous after the
 *                     offsets check.
 *   rse_tokenize_dev: rse_tokenize over n texts that are already on the device (text_dev / offsets_dev[n + 1] as
 *                     above, e.g. rse_chunk_write's output), read in place; then rse_tokens_fetch(_dev) as usual.
 *   rse_encode_tokens_dev: the sentence encoder (head 0) of enc_slot on the last rse_tokenize(_dev)'s ids where they
 *                     are -> out_dev [n, hidden], in slices of at most max_tokens_per_call tokens cut greedily in text
 *                     order at their real lengths (a longer text alone).  cu_seqlens (4 bytes a text) is the one copy
 *                     to the host.  Every sequence needs 1 .. max_positions ids (tokenize with add_special 1 and
 *                     max_length). */
int rse_chunk_count(rse_index *h, const char *text_dev, int64_t text_bytes, const int64_t *offsets_dev, int32_t n_movies,
                    int32_t max_chunk_size, int32_t overlap, int64_t *chunk_cu_dev, int64_t *byte_cu_dev,
                    int64_t *out_n_chunks, int64_t *out_n_bytes);
int rse_chunk_write(rse_index *h, const char *text_dev, int64_t text_bytes, const int64_t *offsets_dev, int32_t n_movies,
                    int32_t max_chunk_size, int32_t overlap, const int64_t *chunk_cu_dev, const int64_t *byte_cu_dev,
                    int32_t movie_base, char *out_text_dev, int64_t *out_offsets_dev, int32_t *out_movie_dev,
                    int32_t *out_index_dev);
int rse_tokenize_dev(rse_index *h, int32_t slot, const char *text_dev, int64_t text_bytes, const int64_t *offsets_dev,
                     int32_t n, int32_t add_special, int32_t max_length, int64_t *out_total, int32_t *out_max_len);
int rse_encode_tokens_dev(rse_index *h, int32_t enc_slot, int64_t max_tokens_per_call, float *out_dev);

/* ------------------------------------------------------------------ CLIP byte-level BPE on the device
 * The image search's CLIP tokenizer (clip-ViT-B-32's CLIPTokenizerFast: NFC / \s+ -> " " / lowercase, the CLIP split
 * pattern, ByteLevel, BPE with the "</w>" suffix, <|startoftext|> ... <|endoftext|>) runs on the device
 * (csrc/bpe.cuh) with ids identical to the HF fast tokenizer.  A tokenizer slot holds either kind; the last load
 * decides.  rse_tokenize, rse_tokens_fetch(_dev) and rse_encode_texts(_dev) dispatch on it:
 *   rse_tokenizer_load_bpe : the description built from the HF object by rag_search_engine_b200/bpe.py: cp_map /
 *                        cp_class for every code point, the symbol of every byte (inside a piece and as its last byte),
 *                        the merge table, the special ids and the added-token strings.  Every index is checked here.
 *   rse_tokenize       : add_special 1 = <|startoftext|> ids[:max_length - 2] <|endoftext|>, 0 = ids[:max_length].
 *                        A text stops at the cut; its tail is validated, never tokenized.
 *   rse_encode_texts(_dev): enc_slot must hold a CLIP text tower (type ids none, max_length 2 .. max_positions); the
 *                        tower runs on the ids where they are, in slices of at most 65536 tokens cut greedily in text
 *                        order at their real lengths.  cu_seqlens (4 bytes a text) is the only copy to the host.
 * Errors: an unloaded slot RSE_ERR_STATE; bad offsets and malformed UTF-8 RSE_ERR_INVALID (the message names the
 * first text); a BPE slot with a BERT encoder or the rerank store, or a WordPiece slot with a CLIP tower,
 * RSE_ERR_INVALID.  RSE_ERR_UNSUPPORTED refuses, never tokenizes differently, a text that holds a code point NFC
 * could join or reorder with its neighbours (cp_map bit 23: non-zero combining class, a decomposition that starts
 * with one, the starters a canonical composition can take as second member) or a piece longer than 256 bytes that
 * is needed before the cut; the Python layer hands those texts to the host tokenizer.  Limits: <= 32 added tokens,
 * < 2^31 ids per call. */
typedef struct rse_bpe_desc {
  const uint32_t *cp_map;       /* [0x110000]: bits 0-20 code point or extra row, 21-22 count (0-3), 23 host route */
  const uint32_t *extra;        /* [n_extra][3] code points of the 2- and 3-code-point outputs */
  int32_t n_extra;
  const uint8_t *cp_class;      /* [0x110000]: 0 other, 1 whitespace, 2 letter (\p{L}), 3 number (\p{N}) */
  const int32_t *byte_ids;      /* [512]: symbol of byte b inside a piece at [b], as its last byte at [256 + b] */
  const int32_t *merges;        /* [merge_slots][4] {left, right, rank, merged}, left -1 = empty; linear probing from
                                   the high 32 bits of ((uint64)left << 32 | right) * 0x9E3779B97F4A7C15, masked */
  int32_t merge_slots;          /* a power of two, with at least one empty slot */
  const char *added;            /* added-token strings (UTF-8) back to back */
  const int32_t *added_offsets; /* [n_added + 1] */
  const int32_t *added_ids;     /* [n_added] */
  int32_t n_added;
  int32_t bos_id, eos_id;
} rse_bpe_desc;
int rse_tokenizer_load_bpe(rse_index *h, int32_t slot, const rse_bpe_desc *desc);

/* ------------------------------------------------------------------ multi-GPU: row shards over one box (SURVEY §8e)
 * One process per GPU, one handle per process; the HANDLE owns the NCCL communicator (NCCL is bound at run time:
 * libnccl.so.2, or $RSE_NCCL_LIB).  The chunk-embedding matrix is cut by row into contiguous shards aligned to
 * vec0 blocks (rse_load_embeddings / rse_attach_embeddings_dev with pos_base = the shard's first global position);
 * the BM25 index is replicated; rank r owns the contiguous query slice [r*nq/N ...) of every batch (the split of
 * sharded.query_slices).  The reference has no counterpart (single process, semantic_search.py:254-261 scans one
 * table); results equal those of one handle holding the whole corpus.
 *   rse_comm_unique_id : rank 0 creates the 128-byte id and hands it to the other ranks by any means
 *                        (torch.distributed broadcast, a file, an environment variable);
 *   rse_comm_init      : every rank, collectively (ncclCommInitRank on the handle's device). */
#define RSE_COMM_ID_BYTES 128
int rse_comm_unique_id(uint8_t *out_id);
int rse_comm_init(rse_index *h, const uint8_t *id_bytes, int32_t n_ranks, int32_t rank);
int rse_comm_destroy(rse_index *h);
int rse_comm_info(rse_index *h, int32_t *n_ranks, int32_t *rank, int32_t *nccl_version);
/* The exchange step alone: cand_dev [nq, kprime, 3] (this shard's local top-K' of ALL queries, rse_knn_local_dev)
 * -> mine_dev [n_ranks, ns, kprime, 3] (every shard's candidates for THIS rank's ns queries): an all-to-all by
 * query slice (grouped ncclSend / ncclRecv) on the handle's stream. */
int rse_comm_exchange_candidates_dev(rse_index *h, const int64_t *cand_dev, int32_t nq, int32_t kprime,
                                     int64_t *mine_dev);
int rse_comm_allgather_dev(rse_index *h, const void *send_dev, void *recv_dev, int64_t bytes_per_rank);
/* configs[4]: sharded KNN + per-movie aggregation in one call — local top-K' of all nq_all queries on this
 * shard, candidate exchange, merge + aggregation of this rank's query slice.  Outputs [ns, k] DEVICE buffers.
 * flagged_dev (optional, int32 on the device): never wait for the host; *flagged_dev += the queries this shard
 * could not finish (see rse_set_defer_flags).  NULL: blocking and always exact.  Collective: every rank calls. */
int rse_knn_sharded_dev(rse_index *h, const float *q_all_dev, int32_t nq_all, int32_t k, int32_t kprime,
                        float *out_dist_dev, int64_t *out_chunk_rowid_dev, int32_t *out_movie_idx_dev,
                        int32_t *out_count_dev, int32_t *flagged_dev);
/* The hybrid step, row-sharded: the staged batch (rse_hybrid_stage) is THIS rank's query slice (its tokens; the
 * staged vectors are not used), q_all_dev holds the vectors of the whole batch.  KNN local top-K' of all queries
 * (the slice's BM25 runs underneath the filter pass) -> exchange -> merge + aggregation + fusion of the slice.
 * Outputs [ns, limit] DEVICE buffers; flagged_dev as above.  Collective. */
int rse_hybrid_sharded_run_dev(rse_index *h, int32_t mode, double param, int32_t tie_mode, int32_t limit,
                               int32_t knn_multiplier, double k1, double b, const float *q_all_dev, int32_t nq_all,
                               int64_t *out_id_dev, double *out_score_dev, double *out_a_dev, double *out_b_dev,
                               int32_t *out_count_dev, int32_t *flagged_dev);

/* ------------------------------------------------------------------ introspection
 * Counters since the last rse_stats_reset: kernels launched by this library,
 * device ms of the last call per stage (CUDA events on the handle's stream). */
typedef struct rse_stats {
  int64_t kernel_launches;
  int64_t knn_scan_launches;
  double scan_ms_total;        /* Σ device time of the K1 scan launches (event pairs, resolved in rse_get_stats) */
  int64_t scan_launches_timed; /* how many scan launches that sum covers */
  double last_knn_total_ms;    /* last rse_knn / rse_knn_movies call, H2D → D2H */
  double last_bm25_ms;
  double last_fuse_ms;
  int64_t emb_rows;
  int32_t emb_dim;
  int64_t bm25_postings;
  int64_t bm25_docs;
  int64_t tc_filter_launches;   /* K4 tensor-core filter passes (each serves ≤ 256 queries) */
  int64_t tc_queries;           /* queries answered through K4 */
  int64_t tc_fallback_queries;  /* of those, re-run through the exact scan (survivor overflow) */
  int64_t tc_second_chance_queries; /* of tc_queries, answered by the second filter pass with a tightened bound */
  int64_t bm25_queries;           /* queries scored by the BM25 kernels */
  int64_t bm25_fallback_queries;  /* of those, handed to the general kernel by the streaming path (device-side flag) */
  int64_t bm25_finalists;         /* documents re-scored exactly by the fixed-point path's finish kernel */
  int64_t bm25_candidates;        /* candidates the fixed-point kernel handed to the finish kernel */
  int64_t h2d_bytes;              /* bytes moved host -> device by the query entry points (not the index loads) */
  int64_t d2h_bytes;              /* bytes moved device -> host by the query entry points */
} rse_stats;
int rse_get_stats(rse_index *h, rse_stats *out);
/* Survivor counts of the most recent K4 filter pass (one per query of its 256-query block; a count above the
 * survivor cap of 8192 means the query overflowed and was re-run).  Synchronises.  n <= 256. */
int rse_tc_last_survivors(rse_index *h, int32_t *out_counts, int32_t n);
/* The survivors of query `query` (an index into the most recent K4 group, 0 .. 2047) as the last filter pass left
 * them: corpus row (local) and cos~, the tensor-core value the filter compared with its threshold.  Copies
 * min(count, 8192, cap) pairs in the order they were appended; *out_n = the survivor count (above 8192: the list
 * overflowed).  Read-only; synchronises. */
int rse_tc_last_pairs(rse_index *h, int32_t query, int64_t *out_rows, float *out_cos, int32_t cap, int32_t *out_n);
/* The order statistic j of the K4 probe's row sample (DESIGN.md §5 "The probe's sample"): the smallest j with
 * P(Binomial(kprime, 1 / stride) >= j) <= 1e-7, capped at kprime.  Pure host arithmetic — exported so that the claim
 * can be checked against an independent binomial tail (tests/test_host_cpu.py). */
int rse_tc_probe_rank(int32_t kprime, int32_t stride);
int rse_stats_reset(rse_index *h);
/* Enable CUDA-event timing: an event pair around every scan launch (no extra syncs). */
int rse_set_timing(rse_index *h, int32_t enabled);

#ifdef __cplusplus
}
#endif
#endif /* RSE_H_ */
