// rse.cu — the C-ABI of librse.so (see include/rse.h).  Host-side orchestration of
// the sm_100a kernels; no torch, no CPU fallback.
#include "../../include/rse.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <set>
#include <string>
#include <thread>
#include <vector>

#include "bm25.cuh"
#include "clip.cuh"
#include "comm.h"
#include "common.cuh"
#include "encoder.cuh"
#include "fusion.cuh"
#include "imgproc.cuh"
#include "knn_scan.cuh"
#include "select.cuh"
#include "knn_tc3.cuh"
#include "rerank.cuh"
#include "wordpiece.cuh"
#include "bpe.cuh"
#include "chunk.cuh"
#include "knn_movies_exact.cuh"

using namespace rse;

namespace {

thread_local std::string g_create_error;

struct DevBuf {
  void* p = nullptr;
  size_t bytes = 0;
};

// the device inputs of one hybrid batch: query vectors and the BM25 tokens bm25_stage derives (token pointer, term
// rows, idf)
struct Batch {
  DevBuf q, tokptr, terms, idf;
  int nq = 0;
};

// pinned host landing buffer of the tensor-core path's per-query overflow flags
struct PinnedFlags {
  int* p = nullptr;
  size_t n = 0;
};

// what knn_local_begin leaves for knn_local_finish.  flags != nullptr: the tensor-core path ran, its per-query
// overflow flags are in tc_status and on their way into pinned memory (ready at ev)
struct PendingKnn {
  const float* q = nullptr;
  int nq = 0, kprime = 0;
  long long* cand = nullptr;
  const int* flags = nullptr;
  cudaEvent_t ev = nullptr;
};

// ---- §8(f2)/(f3): a BERT-family encoder resident next to the index (encoder.cuh)
struct EncLayer {
  float *wqkv = nullptr, *bqkv = nullptr, *wo = nullptr, *bo = nullptr, *ln1g = nullptr, *ln1b = nullptr;
  float *wi = nullptr, *bi = nullptr, *wo2 = nullptr, *bo2 = nullptr, *ln2g = nullptr, *ln2b = nullptr;
  // tf32 hi / lo halves of the four weight matrices (the tensor-core GEMM, encoder.cuh), written by finalize
  float *wqkv_h = nullptr, *wqkv_l = nullptr, *wo_h = nullptr, *wo_l = nullptr;
  float *wi_h = nullptr, *wi_l = nullptr, *wo2_h = nullptr, *wo2_l = nullptr;
};
struct Encoder {
  rse_encoder_config cfg{};
  bool created = false, finalized = false;
  float *word = nullptr, *pos = nullptr, *type = nullptr, *elng = nullptr, *elnb = nullptr;
  float *poolw = nullptr, *poolb = nullptr, *clsw = nullptr, *clsb = nullptr;
  std::vector<EncLayer> layers;
  std::set<std::string> seen;
  DevBuf ids, type_ids, cu, posidx, x, qkv, ctx, tmp, ff, out;
  DevBuf x_h, x_l, ctx_l, ff_l;       // hi / lo activations of the tensor-core path (ctx / ff hold the hi halves there)
  int mode = 0;                       // 0 = tcgen05 3xTF32 GEMMs (when every GEMM dimension is a multiple of 128 / 32),
                                      // 1 = fp32 SIMT GEMMs
  bool tc_ok = false;
  // pinned staging of ids | type_ids | cu_seqlens: two buffers used alternately, each guarded by an event, so a call
  // never waits for the device unless the upload two calls ago is still in flight
  int32_t* pin_in[2] = {nullptr, nullptr};
  size_t pin_in_n[2] = {0, 0};
  cudaEvent_t pin_ev[2] = {nullptr, nullptr};
  int pin_next = 0;
  int max_len = 128;                  // longest sequence of the batch being encoded (sizes the attention CTA)
  // ---- §10 f4: a CLIP tower in this slot (rse_clip_create, clip.cuh).  word = token_embedding, pos =
  // position_embedding, elng / elnb = pre_layrnorm; layer ln1 / ln2 = layer_norm1 / layer_norm2 (pre-LN), wi / wo2 =
  // mlp.fc1 / fc2.  The patch weight is [hidden, patch_k] with its columns zero-padded to a multiple of 128.
  bool clip = false;
  rse_clip_config ccfg{};
  int patch_k = 0;
  float *cls_emb = nullptr, *patch_w = nullptr, *patch_w_h = nullptr, *patch_w_l = nullptr;
  float *flng = nullptr, *flnb = nullptr, *proj = nullptr, *zero_bias = nullptr;
  DevBuf y, pix, patch, patch_l;      // LayerNorm output (the GEMM operand), device pixels, patch rows (+ lo half)
  float* pin_px[2] = {nullptr, nullptr};
  size_t pin_px_n[2] = {0, 0};
  // ---- the image preprocessing bound to this vision slot (rse_imgproc_set, imgproc.cuh).  A chunk's image table
  // and pixels are staged into ip_pin[b] and go up on the copy stream into ip_in[b], b alternating per chunk:
  // ip_ev_up[b] = that upload is done (pinned buffer free, kernels may start), ip_ev_read[b] = the kernels that
  // read ip_in[b] are done (the buffer may be overwritten)
  bool ip_set = false;
  rse_imgproc_cfg ipcfg{};
  IpNorm ipnorm{};
  char* ip_pin[2] = {nullptr, nullptr};
  size_t ip_pin_n[2] = {0, 0};
  DevBuf ip_in[2], ip_axes, ip_span, ip_w, ip_mid;
  cudaEvent_t ip_ev_up[2] = {nullptr, nullptr}, ip_ev_read[2] = {nullptr, nullptr};
  cudaStream_t ip_copy = nullptr;
};

}  // namespace

struct rse_index {
  int device = 0;
  int sm_count = 148;
  cudaStream_t own_stream = nullptr;
  cudaStream_t stream = nullptr;
  std::string err;
  bool fma = false;
  bool timing = false;
  cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
  // scan-kernel timing: event pairs recorded around every scan launch without
  // synchronising; resolved lazily in rse_get_stats (after the caller's sync).
  std::vector<cudaEvent_t> scan_ev;   // 2 per timed launch
  size_t scan_ev_used = 0;
  std::vector<int> scan_ev_passes;    // K4: how many 256-query passes each timed filter launch covered (else 1)
  // staged hybrid query batch (rse_hybrid_stage); rse_knn and rse_bm25 upload their inputs into its buffers too
  Batch staged;
  // rse_hybrid_stash: staged batches parked in HBM (a bench / server rotating over several resident batches)
  Batch stash[RSE_MAX_STASH];
  // K4 tensor-core path
  int tc_mode = 0;                 // 0 auto, 1 off (exact scan only), 2 force on
  int survivor_div = 5;            // probe sample density: expected first-pass survivors ~ cap / survivor_div (RSE_TC_SURVIVOR_DIV).
                                   // r02 sweep, ms per 256-query step, isotropic / clustered / dense-clustered S-600k:
                                   // 3: 1.155 / 1.460 / 2.336   5: 1.146 / 1.223 / 1.785   8: 1.174 / 1.240 / 1.454
  // rse_set_defer_flags: rse_knn_local_dev does not wait for the tensor-core path's overflow flags; they stay on
  // the device (tc_status) and rse_knn_flags_dev adds their count into a caller-owned device counter
  bool defer_flags_dev = false;
  int last_flags_n = 0;
  DevBuf f_pack;                   // rse_hybrid_run results: id | score | a | b | count, back to back
  size_t pack_n = 0;
  int pack_nq = 0;
  char* pin_out = nullptr;         // pinned landing buffer of rse_hybrid_fetch
  size_t pin_out_bytes = 0;
  // rse_hybrid_submit / rse_hybrid_collect: two batches in flight.  Inputs of batch i+1 are staged through their
  // own pinned buffer and uploaded in stream order behind batch i's kernels; each batch's results land in its own
  // pinned slot (copy enqueued by submit right behind the fusion kernel, event per slot).
  struct OutSlot {
    char* pin = nullptr; size_t bytes = 0; cudaEvent_t ev = nullptr;
    size_t n = 0; int nq = 0; long long ticket = -1;
    // the tensor-core path's per-query overflow flags are NOT waited for by submit (that wait is what would keep
    // the host one KNN stage behind the device): they land in `flags` and `knn` keeps them for collect; a batch with
    // a flagged query (rare: a mass tie at the K'-th distance) is re-run through the blocking call from the copies below
    PinnedFlags flags;
    PendingKnn knn;
    std::vector<int32_t> tok_indptr, term_rows;
    int mode = 0, tie_mode = 0, limit = 0, knn_multiplier = 0; double param = 0.0, k1 = 0.0, b = 0.0;
    // the slot's own device inputs and packed results: batch i+1's uploads (copy stream) overlap batch i's kernels,
    // batch i's result copy (third stream) overlaps batch i+1's first kernels — the main stream carries kernels only
    Batch in;
    DevBuf f_pack;
  } out_slot[2];
  cudaStream_t stream_h2d = nullptr, stream_d2h = nullptr;
  cudaEvent_t ev_fused = nullptr;
  long long pipeline_reruns = 0;
  long long next_ticket = 0, next_collect = 0;
  float* pin_q[2] = {nullptr, nullptr};   // pinned staging of the query vectors, alternating with the tickets
  size_t pin_q_bytes[2] = {0, 0};
  cudaEvent_t ev_q[2] = {nullptr, nullptr};
  char* pin_stage = nullptr;       // pinned staging for the token / idf upload of a hybrid or BM25 batch
  size_t pin_stage_bytes = 0;
  PinnedFlags pin_status;          // pinned host copy of the per-query overflow flags
  cudaEvent_t ev_status = nullptr;
  cudaEvent_t ev_stage = nullptr;  // the uploads out of pin_stage have completed
  // hybrid step: BM25 runs on a second, lowest-priority stream UNDER the tensor-core filter pass (one BM25 CTA fits
  // next to the filter's CTA on every SM); see hybrid_local / knn_tc3_group
  cudaStream_t stream_b = nullptr;
  cudaEvent_t ev_prefilter = nullptr, ev_bm25_done = nullptr;
  // RSE_TIMELINE=1: timed events at the stage boundaries of a hybrid step on both streams, printed (ms since the
  // step's first event) to stderr by rse_hybrid_fetch — a development aid, off by default
  bool timeline = false;
  cudaEvent_t tl[8] = {};
  bool tl_set[8] = {};
  DevBuf tc_thr, tc_rows, tc_cnt, tc_status;
  DevBuf fb_list, fb_q, fb_sb, fb_cand;       // exact-scan fallback of flagged queries, gathered (knn_local_finish)
  // fp16 normalised shadow of the corpus for knn_tc3 (built lazily at the first tensor-core batch)
  DevBuf tc_shadow, tc_q16;
  // the probe's stratified row sample (knn_tc3.cuh tc3_sample_kernel): one row of every sample_stride, own small shadow
  DevBuf tc_sample;
  CUtensorMap tmap_s16{};
  int64_t sample_tiles = 0;        // 0 = no sample (small corpus): the probe strides over the main shadow
  int sample_stride = 64;          // RSE_TC_SAMPLE_STRIDE (r02 sweep on S-600k: 16 -> 1.137, 32 -> 1.106, 64 -> 1.091 ms per step)
  int probe_rank = 0;              // RSE_TC_PROBE_RANK: force the probe's order statistic j (tests: 1 = always too tight)
  int sample_min_tiles = 16;       // RSE_TC_SAMPLE_MIN_TILES: 262 k rows at stride 64 (tests lower it for small corpora)
  int shadow_state = 0;            // 0 = not built, 1 = usable, -1 = corpus has non-finite norms: exact scan only
  CUtensorMap tmap_a16{};          // the tiled shadow as [n_pad * KB][64] f16 lines, box {64, 128}, SWIZZLE_128B
  CUtensorMap tmap_q16{};          // [nq_pad][dim] f16, box {64, 128}
  bool tmap_q16_ok = false;
  int tmap_q16_rows = 0;
  int tmap_q16_dim = 0;            // the map is [nq_pad][dim]: a reload at another width needs a new one
  const void* tmap_q16_base = nullptr;

  // ---- a1: embeddings (vec0 physical layout)
  const float* emb = nullptr;
  float* emb_owned = nullptr;
  int64_t n_rows = 0;
  int dim = 0;
  uint64_t pos_base = 0;
  float* amag = nullptr;
  int64_t* rowid = nullptr;
  int32_t* movie_idx = nullptr;

  // ---- knn scratch (grow-only)
  DevBuf sb, sel, hist, selkeys, cand, dist, o_dist, o_pos, o_rowid, o_movie, o_count;
  int64_t dist_ld = 0;

  // ---- rse_knn_movies_exact (knn_movies_exact.cuh): the corpus's movie layout, checked once per load (-1 = not
  // yet), and the per-(query, movie) key buffer's budget, which sets how many queries one segmented scan serves
  int movies_sorted = -1;
  int64_t movie_slots = 0;
  size_t mx_budget = size_t(512) << 20;   // RSE_MOVIES_EXACT_BUDGET (bytes)
  DevBuf mx_span, mx_meta, mx_best, mx_list, mx_q, mx_sb, mx_keys, mx_cand, mx_dist, mx_rowid, mx_movie, mx_count;

  // ---- a6: BM25
  int64_t n_terms = 0, n_postings = 0, n_docs = 0, n_movies = 0;
  double avgdl = 0.0;
  int nr = 0;
  int64_t* indptr = nullptr;
  uint2* post = nullptr;
  uint32_t* dl = nullptr;
  uint32_t* roff = nullptr;
  double* normk = nullptr;
  double normk_k1 = NAN, normk_b = NAN;
  Post16* post16 = nullptr;        // {doc, tf, w}: postings with the (k1, b)-dependent weight precomputed (bm25_stream_kernel)
  uint32_t* post4 = nullptr;       // (doc % range) | round(w * wq4_scale) << 13: the stream of bm25_fx_kernel (padded by one quad)
  double w_k1 = NAN, w_b = NAN;
  DevBuf b_shi, b_slo, b_scnt, b_status, b_flagged;
  int bm25_mode = 0;               // 0 = fixed-point streaming kernel (default), 1 = exact-order streaming kernel, 2 = general kernel only
  std::vector<int64_t> df_host;
  DevBuf b_chi, b_clo, b_ccnt, b_score, b_doc, b_count;

  // ---- fusion scratch + id tables
  DevBuf f_bid, f_bsc, f_bcnt, f_sid, f_sds, f_scnt, f_oid, f_osc, f_oa, f_ob, f_ocnt;
  long long* doc_ids = nullptr;
  int64_t n_doc_ids = 0;
  long long* movie_ids = nullptr;
  int64_t n_movie_ids = 0;

  // ---- cross-encoder rerank of a fused batch (rerank.cuh): the document-token store (CSR over ascending ids) ...
  long long* rr_doc_ids = nullptr;
  long long* rr_doc_indptr = nullptr;
  int32_t* rr_doc_tok = nullptr;
  int64_t rr_n_docs = 0;
  int32_t rr_max_tok = -1;
  int64_t rr_max_doc_len = 0;      // longest document: bounds a pair's length together with the queries and max_length
  int64_t rr_budget = 1 << 17;     // tokens per encoder slice: the encoder's scratch is ~9 KB per TinyBERT token
  // ... the whole fused union [nq, 2 * limit], the packed pairs, and the [nq, limit] results back to back
  DevBuf rr_fid, rr_fsc, rr_fa, rr_fb, rr_fcnt, rr_row, rr_ab, rr_qnp, rr_qnt, rr_qpb, rr_qtb, rr_meta, rr_qptr, rr_qtok;
  DevBuf rr_ids, rr_types, rr_cus, rr_logit, rr_pack;
  int* rr_pin_meta = nullptr;
  size_t rr_pin_meta_n = 0;
  char* rr_pin_out = nullptr;
  size_t rr_pin_out_bytes = 0;
  int rr_nq = 0, rr_limit = 0;
  cudaEvent_t rr_ev[5] = {};       // rse_set_timing: hybrid | assembly | encoder | order boundaries of the last run
  bool rr_timed = false;

  // ---- tokenizers on the device: each slot's tables in one allocation, BERT WordPiece (wordpiece.cuh) or CLIP's
  // byte-level BPE (bpe.cuh) ...
  struct TokSlot {
    bool loaded = false;
    bool bpe = false;
    void* blob = nullptr;
    WpTables t{};
    BpeTables bt{};
  } tok[RSE_MAX_TOKENIZERS];
  // ... and the last tokenisation: texts, offsets, per-text counts, cu_seqlens (int64 | int32), ids, meta (kWpMeta)
  DevBuf tk_text, tk_offs, tk_count, tk_cu64, tk_cu32, tk_ids, tk_meta;
  char* tk_pin = nullptr;          // pinned staging of texts | offsets
  size_t tk_pin_bytes = 0;
  unsigned long long* tk_pin_meta = nullptr;
  int tk_n = 0;                    // texts of the last rse_tokenize (0: nothing to fetch)
  int64_t tk_total = 0;
  unsigned long long tk_max_id = 0;  // the largest id of the last rse_tokenize(_dev)
  const uint8_t* tk_src_text = nullptr;  // the texts the write pass reads: tk_text, or the caller's (rse_tokenize_dev)
  const int64_t* tk_src_offs = nullptr;
  // ---- sentence chunking (chunk.cuh): per-movie counts, the int32 scan output nobody reads, meta
  DevBuf ck_chunks, ck_bytes, ck_cu32, ck_meta;

  // cudaFuncSetAttribute is per device: remember per HANDLE which kernels were configured (a process-wide static
  // flag would leave the second device of a multi-GPU process unconfigured)
  Encoder enc[RSE_MAX_ENCODERS];

  // ---- row-sharded multi-GPU path: the handle owns the communicator (comm.h)
  ncclComm_t comm = nullptr;
  int comm_ranks = 1, comm_rank = 0;
  DevBuf sh_cand, sh_mine;

  uint32_t attr_mask = 0;
  uint32_t attr_mask_wide = 0;     // knn_scan_wide_kernel instantiations
  uint32_t attr_mask_tc = 0;       // bit KB-1: knn_tc3_kernel<*, KB>; bit 8 + KB-1: knn_refine_kernel<*, KB>
  rse_stats stats{};
  // device-side counters read back by rse_get_stats: [0] BM25 queries handed to the general kernel, [1] BM25
  // finalists re-scored exactly, [2] BM25 candidates merged by the finish kernel
  unsigned long long* dev_counters = nullptr;
};

namespace {

int fail(rse_index* h, int code, const std::string& msg) {
  if (h) h->err = msg; else g_create_error = msg;
  return code;
}

#define CK(call)                                                                              \
  do {                                                                                        \
    cudaError_t e__ = (call);                                                                 \
    if (e__ != cudaSuccess)                                                                   \
      return fail(h, RSE_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e__));      \
  } while (0)

#define LAUNCHED(h)                                                                           \
  do {                                                                                        \
    (h)->stats.kernel_launches++;                                                             \
    cudaError_t e__ = cudaGetLastError();                                                     \
    if (e__ != cudaSuccess)                                                                   \
      return fail(h, RSE_ERR_CUDA, std::string("kernel launch: ") + cudaGetErrorString(e__)); \
  } while (0)

int ensure(rse_index* h, DevBuf& b, size_t bytes) {
  if (bytes <= b.bytes) return RSE_OK;
  if (b.p) CK(cudaFree(b.p));
  b.p = nullptr; b.bytes = 0;
  size_t want = bytes + bytes / 4 + 256;
  CK(cudaMalloc(&b.p, want));
  b.bytes = want;
  return RSE_OK;
}
#define ENSURE(buf, bytes)                         \
  do {                                             \
    int rc__ = ensure(h, (buf), (bytes));          \
    if (rc__ != RSE_OK) return rc__;               \
  } while (0)

void free_buf(DevBuf& b) {
  if (b.p) cudaFree(b.p);
  b.p = nullptr; b.bytes = 0;
}

template <typename T>
void free_ptr(T*& p) {
  if (p) cudaFree(p);
  p = nullptr;
}

void free_batch(Batch& b) {
  for (DevBuf* d : {&b.q, &b.tokptr, &b.terms, &b.idf}) free_buf(*d);
  b.nq = 0;
}

void release_embeddings(rse_index* h) {
  free_ptr(h->emb_owned);
  h->emb = nullptr;
  free_ptr(h->amag);
  free_ptr(h->rowid);
  free_ptr(h->movie_idx);
  h->n_rows = 0; h->dim = 0;
  free_buf(h->tc_shadow);
  free_buf(h->tc_sample);
  h->sample_tiles = 0;
  h->shadow_state = 0;
  h->movies_sorted = -1;
  h->movie_slots = 0;
}

void release_bm25(rse_index* h) {
  free_ptr(h->indptr); free_ptr(h->post); free_ptr(h->dl); free_ptr(h->roff); free_ptr(h->normk); free_ptr(h->post16); free_ptr(h->post4);
  h->w_k1 = NAN; h->w_b = NAN;
  h->df_host.clear();
  h->n_terms = h->n_postings = h->n_docs = h->n_movies = 0;
  h->normk_k1 = NAN; h->normk_b = NAN;
}

void enc_release(Encoder& e) {
  for (float** p : {&e.word, &e.pos, &e.type, &e.elng, &e.elnb, &e.poolw, &e.poolb, &e.clsw, &e.clsb}) free_ptr(*p);
  for (float** p : {&e.cls_emb, &e.patch_w, &e.patch_w_h, &e.patch_w_l, &e.flng, &e.flnb, &e.proj, &e.zero_bias}) free_ptr(*p);
  for (DevBuf* b : {&e.y, &e.pix, &e.patch, &e.patch_l}) free_buf(*b);
  for (auto& l : e.layers)
    for (float** p : {&l.wqkv, &l.bqkv, &l.wo, &l.bo, &l.ln1g, &l.ln1b, &l.wi, &l.bi, &l.wo2, &l.bo2, &l.ln2g, &l.ln2b,
                      &l.wqkv_h, &l.wqkv_l, &l.wo_h, &l.wo_l, &l.wi_h, &l.wi_l, &l.wo2_h, &l.wo2_l}) free_ptr(*p);
  e.layers.clear();
  e.seen.clear();
  for (DevBuf* b : {&e.ids, &e.type_ids, &e.cu, &e.posidx, &e.x, &e.qkv, &e.ctx, &e.tmp, &e.ff, &e.out, &e.x_h, &e.x_l,
                    &e.ctx_l, &e.ff_l}) free_buf(*b);
  for (int i = 0; i < 2; ++i) {
    if (e.pin_in[i]) cudaFreeHost(e.pin_in[i]);
    if (e.pin_ev[i]) cudaEventDestroy(e.pin_ev[i]);
    e.pin_in[i] = nullptr; e.pin_in_n[i] = 0; e.pin_ev[i] = nullptr;
    if (e.pin_px[i]) cudaFreeHost(e.pin_px[i]);
    e.pin_px[i] = nullptr; e.pin_px_n[i] = 0;
    if (e.ip_pin[i]) cudaFreeHost(e.ip_pin[i]);
    e.ip_pin[i] = nullptr; e.ip_pin_n[i] = 0;
    for (cudaEvent_t* ev : {&e.ip_ev_up[i], &e.ip_ev_read[i]}) { if (*ev) cudaEventDestroy(*ev); *ev = nullptr; }
    free_buf(e.ip_in[i]);
  }
  for (DevBuf* b : {&e.ip_axes, &e.ip_span, &e.ip_w, &e.ip_mid}) free_buf(*b);
  if (e.ip_copy) { cudaStreamSynchronize(e.ip_copy); cudaStreamDestroy(e.ip_copy); }
  e.ip_copy = nullptr;
  e.ip_set = false;
  e.created = e.finalized = e.clip = false;
}

// ------------------------------------------------------------------ scan launch
template <int QB, bool FMA>
int launch_scan384(rse_index* h, const float* q, const double* sb, int nq, float* dist) {
  const int smem = scan_smem_bytes(QB);
  constexpr uint32_t bit = 1u << ((QB == 1 ? 0 : QB == 2 ? 1 : QB == 4 ? 2 : QB == 8 ? 3 : 4) + (FMA ? 5 : 0));
  if (!(h->attr_mask & bit)) {
    CK(cudaFuncSetAttribute(knn_scan384_kernel<QB, FMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    h->attr_mask |= bit;
  }
  const int64_t n_tiles = (h->n_rows + kScanTileRows - 1) / kScanTileRows;
  int grid = static_cast<int>(std::min<int64_t>(h->sm_count, (n_tiles + kScanWarps - 1) / kScanWarps));
  if (grid < 1) grid = 1;
  // -0.0f / 1.0f pairs for the packed unfused step: run-time values on purpose (see knn_scan.cuh)
  const unsigned long long negz2 = 0x8000000080000000ull, one2 = 0x3F8000003F800000ull;
  knn_scan384_kernel<QB, FMA><<<grid, kScanWarps * 32, smem, h->stream>>>(h->emb, h->amag, h->n_rows, q, sb, nq,
                                                                         dist, h->dist_ld, negz2, one2);
  LAUNCHED(h);
  h->stats.knn_scan_launches++;
  return RSE_OK;
}

template <int QB, bool FMA>
int launch_scan_wide(rse_index* h, const float* q, const double* sb, int nq, float* dist) {
  const int smem = wide_smem_bytes(QB, h->dim);
  // (the opt-in is per function and per device; the size depends on dim, so it is simply raised to the cap once)
  constexpr uint32_t bit = 1u << ((QB == 1 ? 0 : QB == 2 ? 1 : QB == 4 ? 2 : QB == 8 ? 3 : 4) + (FMA ? 5 : 0));
  if (!(h->attr_mask_wide & bit)) {
    CK(cudaFuncSetAttribute(knn_scan_wide_kernel<QB, FMA>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
    h->attr_mask_wide |= bit;
  }
  const int64_t n_tiles = (h->n_rows + 31) / 32;
  const int per_sm = std::max(1, std::min(4, (220 * 1024) / (smem + 1024)));
  int grid = static_cast<int>(std::min<int64_t>(static_cast<int64_t>(h->sm_count) * per_sm, (n_tiles + kWideWarps - 1) / kWideWarps));
  if (grid < 1) grid = 1;
  knn_scan_wide_kernel<QB, FMA><<<grid, kWideWarps * 32, smem, h->stream>>>(h->emb, h->amag, h->n_rows, h->dim, q, sb, nq,
                                                                           dist, h->dist_ld);
  LAUNCHED(h);
  h->stats.knn_scan_launches++;
  return RSE_OK;
}

template <bool FMA>
int launch_scan(rse_index* h, const float* q, const double* sb, int nq, float* dist) {
  if (h->dim == kScanD) {
    if (nq <= 1) return launch_scan384<1, FMA>(h, q, sb, nq, dist);
    if (nq <= 2) return launch_scan384<2, FMA>(h, q, sb, nq, dist);
    if (nq <= 4) return launch_scan384<4, FMA>(h, q, sb, nq, dist);
    if (nq <= 8) return launch_scan384<8, FMA>(h, q, sb, nq, dist);
    return launch_scan384<16, FMA>(h, q, sb, nq, dist);
  }
  // any width that keeps the rows 16-byte aligned: the staged kernel (queries must fit beside the stages)
  if (h->dim % 4 == 0 && wide_smem_bytes(16, h->dim) <= 200 * 1024) {
    if (nq <= 1) return launch_scan_wide<1, FMA>(h, q, sb, nq, dist);
    if (nq <= 2) return launch_scan_wide<2, FMA>(h, q, sb, nq, dist);
    if (nq <= 4) return launch_scan_wide<4, FMA>(h, q, sb, nq, dist);
    if (nq <= 8) return launch_scan_wide<8, FMA>(h, q, sb, nq, dist);
    return launch_scan_wide<16, FMA>(h, q, sb, nq, dist);
  }
  const int threads = kGenWarps * 32;
  const int grid = static_cast<int>((h->n_rows + threads - 1) / threads);
  knn_scan_generic_kernel<FMA><<<grid, threads, 0, h->stream>>>(h->emb, h->amag, h->n_rows, h->dim, q, sb, nq,
                                                                dist, h->dist_ld);
  LAUNCHED(h);
  h->stats.knn_scan_launches++;
  return RSE_OK;
}

// ---- exact path (K1 + K2 + K3) for queries [0, nq) whose |q| factors sb[] are ready
int knn_exact_groups(rse_index* h, const float* q_dev, const double* sb, int nq, int kprime, long long* cand_dev) {
  const int QB = kScanMaxQB;
  ENSURE(h->sel, sizeof(SelState) * std::max(nq, kTcBN));
  ENSURE(h->selkeys, sizeof(unsigned long long) * static_cast<size_t>(nq) * kprime);
  ENSURE(h->dist, sizeof(float) * static_cast<size_t>(QB) * h->dist_ld);
  SelState* sel = static_cast<SelState*>(h->sel.p);
  unsigned int* hist = static_cast<unsigned int*>(h->hist.p);
  unsigned long long* selkeys = static_cast<unsigned long long*>(h->selkeys.p);
  float* dist = static_cast<float*>(h->dist.p);
  select_init_kernel<<<(nq + 127) / 128, 128, 0, h->stream>>>(sel, nq, static_cast<unsigned int>(kprime));
  LAUNCHED(h);
  static const int shifts[6] = {53, 42, 32, 21, 10, 0};
  static const int widths[6] = {11, 11, 10, 11, 11, 10};
  int sel_blocks = static_cast<int>(std::min<int64_t>((h->n_rows + 4095) / 4096, h->sm_count * 2));
  if (sel_blocks < 1) sel_blocks = 1;
  for (int g0 = 0; g0 < nq; g0 += QB) {
    const int ng = std::min(QB, nq - g0);
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    if (h->timing && h->scan_ev_used + 2 <= (1u << 16)) {
      while (h->scan_ev.size() < h->scan_ev_used + 2) {
        cudaEvent_t e;
        CK(cudaEventCreate(&e));
        h->scan_ev.push_back(e);
      }
      e0 = h->scan_ev[h->scan_ev_used];
      e1 = h->scan_ev[h->scan_ev_used + 1];
      h->scan_ev_used += 2;
      h->scan_ev_passes.push_back(1);
      CK(cudaEventRecord(e0, h->stream));
    }
    int rc = h->fma ? launch_scan<true>(h, q_dev + static_cast<int64_t>(g0) * h->dim, sb + g0, ng, dist)
                    : launch_scan<false>(h, q_dev + static_cast<int64_t>(g0) * h->dim, sb + g0, ng, dist);
    if (rc != RSE_OK) return rc;
    if (e1) CK(cudaEventRecord(e1, h->stream));
    dim3 grid(sel_blocks, ng);
    for (int p = 0; p < 6; ++p) {
      select_pass_kernel<<<grid, kSelThreads, 0, h->stream>>>(reinterpret_cast<const uint32_t*>(dist), h->dist_ld, h->n_rows, h->pos_base, sel + g0, hist,
                                                              shifts[p], widths[p]);
      LAUNCHED(h);
    }
    select_collect_kernel<<<grid, kSelThreads, 0, h->stream>>>(reinterpret_cast<const uint32_t*>(dist), h->dist_ld, h->n_rows, h->pos_base, sel + g0,
                                                               selkeys + static_cast<int64_t>(g0) * kprime, kprime);
    LAUNCHED(h);
  }
  const int kp2 = next_pow2(kprime);
  const size_t fsmem = static_cast<size_t>(kp2) * 12;
  if (fsmem > 48 * 1024) CK(cudaFuncSetAttribute(select_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  select_finish_kernel<<<nq, kSelThreads, fsmem, h->stream>>>(selkeys, sel, kprime, kp2, h->pos_base, h->rowid,
                                                             h->movie_idx, cand_dev);
  LAUNCHED(h);
  return RSE_OK;
}

// ---- K4: tensor-core path for one block of ≤ 256 queries (see knn_tc.cuh)
typedef CUresult (*PFN_tmapEncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

// [rows][cols] row-major matrix of f32 (elem_bytes 4) or f16 (2); box = one 128-byte swizzle atom x box_rows
int make_tmap_any(rse_index* h, CUtensorMap* out, const void* base, int64_t rows, int64_t cols, int box_rows,
                  int elem_bytes) {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (!p || qres != cudaDriverEntryPointSuccess) return fail(h, RSE_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
    fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
  const cuuint64_t gstr[1] = {static_cast<cuuint64_t>(cols) * elem_bytes};
  const cuuint32_t box[2] = {static_cast<cuuint32_t>(128 / elem_bytes), static_cast<cuuint32_t>(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, elem_bytes == 4 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2,
                  const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(h, RSE_ERR_CUDA, "cuTensorMapEncodeTiled failed: " + std::to_string(static_cast<int>(r)));
  return RSE_OK;
}

// [lines][64] f16 array of contiguous 128-byte lines, box {64, box_lines}, SWIZZLE_128B
int make_tmap_lines(rse_index* h, CUtensorMap* out, const void* base, int64_t lines, int box_lines) {
  PFN_tmapEncodeTiled fn = nullptr;
  {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (!p || qres != cudaDriverEntryPointSuccess) return fail(h, RSE_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
    fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  const cuuint64_t gdim[2] = {64, static_cast<cuuint64_t>(lines)};
  const cuuint64_t gstr[1] = {128};
  const cuuint32_t box[2] = {64, static_cast<cuuint32_t>(box_lines)};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(h, RSE_ERR_CUDA, "cuTensorMapEncodeTiled (lines) failed: " + std::to_string(static_cast<int>(r)));
  return RSE_OK;
}

// refine + exact re-score + emit for one block of queries whose survivors are in tc_rows / tc_cnt.
// thr2 / gate != NULL: the second-chance pass (only the queries tc3_second_threshold_kernel re-armed).
template <int KB>
int knn_tc_refine(rse_index* h, const float* q_dev, const double* sb, int nqb, int kprime, long long* cand_dev,
                  int* status_dev, const float* thr2, const unsigned int* gate, float* thr2_out, unsigned int* gate_out,
                  const float* tverify) {
  if (!(h->attr_mask_tc & (1u << (8 + KB - 1)))) {
    CK(cudaFuncSetAttribute(knn_refine_kernel<false, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRefineSmemBytes));
    CK(cudaFuncSetAttribute(knn_refine_kernel<true, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, kRefineSmemBytes));
    h->attr_mask_tc |= 1u << (8 + KB - 1);
  }
  if (h->fma)
    knn_refine_kernel<true, KB><<<nqb, kSelThreads, kRefineSmemBytes, h->stream>>>(
        h->emb, h->amag, q_dev, sb, static_cast<const uint2*>(h->tc_rows.p),
        static_cast<unsigned int*>(h->tc_cnt.p), kTcCandCap, kprime, h->pos_base, h->rowid, h->movie_idx,
        cand_dev, status_dev, 1, thr2, gate, h->dev_counters, thr2_out, gate_out, tverify);
  else
    knn_refine_kernel<false, KB><<<nqb, kSelThreads, kRefineSmemBytes, h->stream>>>(
        h->emb, h->amag, q_dev, sb, static_cast<const uint2*>(h->tc_rows.p),
        static_cast<unsigned int*>(h->tc_cnt.p), kTcCandCap, kprime, h->pos_base, h->rowid, h->movie_idx,
        cand_dev, status_dev, 1, thr2, gate, h->dev_counters, thr2_out, gate_out, tverify);
  LAUNCHED(h);
  return RSE_OK;
}

// record a CUDA-event pair around the dominant kernel of a pass (resolved lazily in rse_get_stats)
int scan_event(rse_index* h, cudaEvent_t* out) {
  *out = nullptr;
  if (!h->timing || h->scan_ev_used + 1 > (1u << 16)) return RSE_OK;
  while (h->scan_ev.size() < h->scan_ev_used + 1) {
    cudaEvent_t e;
    CK(cudaEventCreate(&e));
    h->scan_ev.push_back(e);
  }
  *out = h->scan_ev[h->scan_ev_used++];
  CK(cudaEventRecord(*out, h->stream));
  return RSE_OK;
}

// Build the fp16 normalised shadow (knn_tc3.cuh) once per corpus.  Returns RSE_OK with shadow_state = -1
// when the corpus holds rows whose squared norm is not finite (the error bound needs a finite norm).
// KB = dim / 64.
template <int KB>
int ensure_shadow(rse_index* h) {
  if (h->shadow_state != 0) return RSE_OK;
  const int64_t n_pad = (h->n_rows + kT3TileRows - 1) / kT3TileRows * kT3TileRows;     // zero rows up to a whole tile
  const size_t shadow_bytes = sizeof(__half) * static_cast<size_t>(n_pad) * h->dim;
  ENSURE(h->tc_shadow, shadow_bytes);
  ENSURE(h->tc_cnt, sizeof(unsigned int) * kTcBN);
  {
    // the last (partial) tile pair: zero it before the rows that exist are written
    const size_t tail0 = sizeof(__half) * static_cast<size_t>(n_pad - kT3TileRows) * h->dim;
    CK(cudaMemsetAsync(static_cast<char*>(h->tc_shadow.p) + tail0, 0, shadow_bytes - tail0, h->stream));
  }
  unsigned int* bad = static_cast<unsigned int*>(h->tc_cnt.p);
  CK(cudaMemsetAsync(bad, 0, sizeof(unsigned int), h->stream));
  const int grid = h->sm_count * 8;
  tc3_shadow_kernel<KB><<<grid, 256, 0, h->stream>>>(h->emb, h->amag, h->n_rows, static_cast<__half*>(h->tc_shadow.p), bad);
  LAUNCHED(h);
  unsigned int nbad = 0;
  CK(cudaMemcpyAsync(&nbad, bad, sizeof(unsigned int), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (nbad) {
    free_buf(h->tc_shadow);
    h->shadow_state = -1;
    return RSE_OK;
  }
  // the tiled shadow as a 2-D array of 128-byte lines: [n_pad * KB lines][64 halves], box = 128 lines = one stage
  int rc = make_tmap_lines(h, &h->tmap_a16, h->tc_shadow.p, n_pad * KB, kT3HalfRows);
  if (rc != RSE_OK) return rc;
  // the probe's sample: its own small matrix from sample_min_tiles tiles on (262 k corpus rows, the automatic K4
  // threshold); smaller corpora keep the strided-tile probe over the main shadow
  h->sample_tiles = 0;
  const int64_t n_sample = (h->n_rows + h->sample_stride - 1) / h->sample_stride;
  if (n_sample >= static_cast<int64_t>(h->sample_min_tiles) * kT3TileRows) {
    const int64_t s_pad = (n_sample + kT3TileRows - 1) / kT3TileRows * kT3TileRows;
    const size_t s_bytes = sizeof(__half) * static_cast<size_t>(s_pad) * h->dim;
    ENSURE(h->tc_sample, s_bytes);
    const size_t s_tail0 = sizeof(__half) * static_cast<size_t>(s_pad - kT3TileRows) * h->dim;
    CK(cudaMemsetAsync(static_cast<char*>(h->tc_sample.p) + s_tail0, 0, s_bytes - s_tail0, h->stream));
    tc3_sample_kernel<KB><<<grid, 256, 0, h->stream>>>(h->emb, h->amag, h->n_rows, h->sample_stride, n_sample,
                                                   static_cast<__half*>(h->tc_sample.p));
    LAUNCHED(h);
    rc = make_tmap_lines(h, &h->tmap_s16, h->tc_sample.p, s_pad * KB, kT3HalfRows);
    if (rc != RSE_OK) return rc;
    h->sample_tiles = s_pad / kT3TileRows;
  }
  h->shadow_state = 1;
  return RSE_OK;
}

// The probe's order statistic on the sample path: the smallest j with P(Binomial(K', 1/stride) >= j) <= 1e-7.  The
// sample's j-th best value exceeds the true K'-th best only if at least j of the (at most K' - 1) rows above it were
// drawn; the draw is independent of the data (tc3_sample_kernel), so that probability is bounded by the binomial tail
// whatever the corpus looks like.  j <= K' (the sample's K'-th best is always a valid bound).
int sample_probe_rank(int kprime, int stride) {
  const double p = 1.0 / stride, q = 1.0 - p;
  // tail(j) = sum_{i >= j} C(K', i) p^i q^(K'-i); walk the pmf up from i = 0
  double pmf = std::pow(q, kprime), cdf = 0.0;
  for (int j = 0; j < kprime; ++j) {
    // here pmf = P(X = j), cdf = P(X < j)
    if (1.0 - cdf <= 1e-7) return std::max(1, j);
    cdf += pmf;
    pmf *= static_cast<double>(kprime - j) / (j + 1) * p / q;
  }
  return kprime;
}

// defined with the BM25 entry points further down, inside the ABI's extern "C" block
extern "C" int bm25_run(rse_index* h, const Batch& in, int nq, int k, double k1, double b, cudaStream_t s,
                        bool under_filter);

// the BM25 batch a hybrid step hands to the KNN, to be enqueued underneath the tensor-core filter pass; `enqueued`
// reports whether that happened (the exact path has no filter pass: the caller then runs it itself)
struct Bm25Job {
  const Batch* in;
  int k;
  double k1, b;
  bool enqueued = false;
};

enum { kTlStart = 0, kTlPrefilter, kTlFilterEnd, kTlKnnEnd, kTlBm25Start, kTlBm25End, kTlStepEnd, kTlCount };

void tl_mark(rse_index* h, int which, cudaStream_t s) {
  if (!h->timeline) return;
  if (!h->tl[which] && cudaEventCreate(&h->tl[which]) != cudaSuccess) return;
  h->tl_set[which] = cudaEventRecord(h->tl[which], s) == cudaSuccess;
}

void tl_print(rse_index* h) {
  if (!h->timeline || !h->tl_set[kTlStart]) return;
  static const char* names[kTlCount] = {"start", "prefilter", "filter_end", "knn_end", "bm25_start", "bm25_end", "step_end"};
  std::fprintf(stderr, "[rse timeline]");
  for (int i = 1; i < kTlCount; ++i) {
    float ms = 0.f;
    if (h->tl_set[i] && cudaEventSynchronize(h->tl[i]) == cudaSuccess &&
        cudaEventElapsedTime(&ms, h->tl[kTlStart], h->tl[i]) == cudaSuccess)
      std::fprintf(stderr, " %s=%.3f", names[i], ms);
    h->tl_set[i] = false;
  }
  std::fprintf(stderr, "\n");
  h->tl_set[kTlStart] = false;
}

// Enqueue the BM25 batch of a hybrid step on the second stream, ordered behind `after` (an event on the main stream).
// Called right after the filter kernel has been launched, so the filter's CTAs are placed first and BM25 fills what
// is left of every SM.
int enqueue_bm25_overlapped(rse_index* h, Bm25Job& job, cudaEvent_t after) {
  job.enqueued = true;
  if (!h->stream_b) {
    int lo = 0, hi = 0;
    CK(cudaDeviceGetStreamPriorityRange(&lo, &hi));          // lo = numerically largest = lowest priority
    CK(cudaStreamCreateWithPriority(&h->stream_b, cudaStreamNonBlocking, lo));
    CK(cudaEventCreateWithFlags(&h->ev_bm25_done, cudaEventDisableTiming));
  }
  CK(cudaStreamWaitEvent(h->stream_b, after, 0));
  tl_mark(h, kTlBm25Start, h->stream_b);
  const int rc = bm25_run(h, *job.in, job.in->nq, job.k, job.k1, job.b, h->stream_b, true);
  if (rc != RSE_OK) return rc;
  tl_mark(h, kTlBm25End, h->stream_b);
  CK(cudaEventRecord(h->ev_bm25_done, h->stream_b));
  return RSE_OK;
}

// ---- K4 over the fp16 shadow (knn_tc3.cuh) for a GROUP of up to kTcGroupBlocks blocks of 256 queries: one launch
// per stage (query prep, probe, thresholds, filter, refine, gated second filter + refine) whatever the number of
// blocks — r01 ran the whole chain once per block from a host loop.  KB = dim / 64 selects the instantiation.
constexpr int kTcGroupBlocks = 8;                 // 2048 queries per group: 134 MB of survivor lists

template <int KB>
int knn_tc3_group(rse_index* h, const float* q_dev, const double* sb, int nqg, int kprime, long long* cand_dev,
                  int* status_dev, Bm25Job* bm25) {
  constexpr int kT3SmemBytes = t3_smem_bytes(KB);
  if (!(h->attr_mask_tc & (1u << (KB - 1)))) {
    CK(cudaFuncSetAttribute(knn_tc3_kernel<0, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, kT3SmemBytes));
    CK(cudaFuncSetAttribute(knn_tc3_kernel<1, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, kT3SmemBytes));
    CK(cudaFuncSetAttribute(knn_tc3_kernel<2, KB>, cudaFuncAttributeMaxDynamicSharedMemorySize, kT3SmemBytes));
    // the filter shares its SMs with BM25 CTAs (hybrid step): ask for the full shared-memory carve-out, otherwise the
    // driver picks the smallest configuration that fits the filter alone and nothing else can become resident
    // (at KB = 8 the filter's 210 KB leave no room for a BM25 CTA of the hybrid step: BM25 then runs after it)
    CK(cudaFuncSetAttribute(knn_tc3_kernel<1, KB>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    h->attr_mask_tc |= 1u << (KB - 1);
  }
  const int64_t n_tiles = (h->n_rows + kT3TileRows - 1) / kT3TileRows;
  const int max_clusters = std::max(1, h->sm_count / 2);
  // Probe sample: every tile_stride-th 256-row tile.  Expected survivors per query ≈ K' * tile_stride
  // (+ the 2*eps band), so the stride is as large as a fifth (survivor_div) of the survivor cap allows, while the
  // sample keeps at least 64 tiles (and 8 K' rows) so its K'-th value is a meaningful bound.
  int64_t tile_stride = std::max<int64_t>(1, std::min<int64_t>(kTcCandCap / (static_cast<int64_t>(h->survivor_div) * kprime), n_tiles / 64));
  int64_t n_probe = (n_tiles + tile_stride - 1) / tile_stride;
  while (n_probe * kT3TileRows < 8ll * kprime && tile_stride > 1) { tile_stride /= 2; n_probe = (n_tiles + tile_stride - 1) / tile_stride; }
  // Sample path (r02): the probe runs over the stratified row sample instead of a strided subset of tiles, and the
  // threshold is the sample's j-th best value, j = sample_probe_rank << K' — a few hundred survivors per query
  // instead of K' * tile_stride; the refine kernel verifies the bound and re-arms the second chance when it was too
  // tight (1e-7 per query by construction).
  int kth = kprime;
  bool sampled = false;
  if (h->sample_tiles > 0 && kprime <= 256) {
    const int clusters_s = static_cast<int>(std::min<int64_t>(max_clusters, h->sample_tiles));
    const int j = h->probe_rank > 0 ? std::min(h->probe_rank, kprime) : sample_probe_rank(kprime, h->sample_stride);
    if (static_cast<int64_t>(clusters_s) * 2 * kT3ProbeTop >= 8ll * j &&
        static_cast<int64_t>(clusters_s) * 2 * kT3ProbeTop <= kT3SelMax) {
      sampled = true; kth = j; tile_stride = 1; n_probe = h->sample_tiles;
    }
  }
  const int64_t ld_probe = n_probe * kT3TileRows;
  const int probe_clusters = static_cast<int>(std::min<int64_t>(max_clusters, n_probe));
  const int grid_p = 2 * probe_clusters;
  const bool sparse_probe = sampled ||
                            (kprime <= 256 && static_cast<int64_t>(probe_clusters) * 2 * kT3ProbeTop >= 4ll * kprime &&
                             static_cast<int64_t>(probe_clusters) * 2 * kT3ProbeTop <= kT3SelMax);
  // the dense probe (K' > 256, tiny corpora) keeps its per-query sample matrix and radix select: one block at a time
  if (!sparse_probe && nqg > kTcBN) {
    for (int b0 = 0; b0 < nqg; b0 += kTcBN) {
      const int nqb = std::min(kTcBN, nqg - b0);
      int rc = knn_tc3_group<KB>(h, q_dev + static_cast<int64_t>(b0) * h->dim, sb + b0, nqb, kprime,
                                 cand_dev + static_cast<int64_t>(b0) * kprime * 3, status_dev + b0, bm25);
      if (rc != RSE_OK) return rc;
    }
    return RSE_OK;
  }
  const int nblk = (nqg + kTcBN - 1) / kTcBN;
  const int nq_pad = nblk * kTcBN;
  ENSURE(h->tc_q16, sizeof(__half) * static_cast<size_t>(nq_pad) * h->dim);
  if (!h->tmap_q16_ok || h->tmap_q16_rows != nq_pad || h->tmap_q16_base != h->tc_q16.p || h->tmap_q16_dim != h->dim) {
    int rc = make_tmap_any(h, &h->tmap_q16, h->tc_q16.p, nq_pad, h->dim, kT3HalfRows, 2);
    if (rc != RSE_OK) return rc;
    h->tmap_q16_ok = true; h->tmap_q16_rows = nq_pad; h->tmap_q16_base = h->tc_q16.p; h->tmap_q16_dim = h->dim;
  }
  ENSURE(h->tc_thr, sizeof(float) * 3 * nq_pad);              // first-pass cuts, the second chance's, the bounds to verify
  ENSURE(h->tc_rows, sizeof(uint2) * static_cast<size_t>(nq_pad) * kTcCandCap);
  ENSURE(h->tc_cnt, sizeof(unsigned int) * (nq_pad + kTcGroupBlocks + 4));   // [nq_pad ...): one second-chance gate per block
  ENSURE(h->sel, sizeof(SelState) * kTcBN);
  int64_t ld_sel = sparse_probe ? static_cast<int64_t>(probe_clusters) * 2 * kT3ProbeTop : ld_probe;
  ENSURE(h->dist, std::max(sizeof(float) * static_cast<size_t>(kScanMaxQB) * h->dist_ld,
                           sizeof(uint32_t) * static_cast<size_t>(nq_pad) * ld_sel));
  uint32_t* dist = static_cast<uint32_t*>(h->dist.p);
  SelState* sel = static_cast<SelState*>(h->sel.p);
  unsigned int* hist = static_cast<unsigned int*>(h->hist.p);
  __half* q16 = static_cast<__half*>(h->tc_q16.p);
  float* thr = static_cast<float*>(h->tc_thr.p);

  tc3_query_prep_kernel<KB><<<nq_pad, 16 * KB, 0, h->stream>>>(q_dev, sb, nqg, q16);
  LAUNCHED(h);

  // 1. probe: approximate distances of a strided sample of tiles → K'-th smallest per query
  if (sparse_probe) {
    knn_tc3_kernel<2, KB><<<grid_p, kT3Threads, kT3SmemBytes, h->stream>>>(
        sampled ? h->tmap_s16 : h->tmap_a16, h->tmap_q16, n_probe, tile_stride, nqg, nblk, nullptr, dist, ld_sel, nullptr,
        nullptr, 0, nullptr);
    LAUNCHED(h);
    tc3_probe_threshold_kernel<<<nq_pad, 256, 0, h->stream>>>(dist, ld_sel, nqg, kth, sb, thr,
                                                              sampled ? thr + 2 * nq_pad : nullptr);
    LAUNCHED(h);
  } else {
    knn_tc3_kernel<0, KB><<<grid_p, kT3Threads, kT3SmemBytes, h->stream>>>(
        h->tmap_a16, h->tmap_q16, n_probe, tile_stride, nqg, 1, nullptr, dist, ld_probe, nullptr, nullptr, 0, nullptr);
    LAUNCHED(h);
    select_init_kernel<<<(nqg + 127) / 128, 128, 0, h->stream>>>(sel, nqg, static_cast<unsigned int>(kprime));
    LAUNCHED(h);
    int blocks = static_cast<int>(std::min<int64_t>((ld_sel + 4095) / 4096, h->sm_count));
    if (blocks < 1) blocks = 1;
    dim3 grid(blocks, nqg);
    static const int shifts[3] = {53, 42, 32};
    static const int widths[3] = {11, 11, 10};
    for (int p = 0; p < 3; ++p) {
      select_pass_kernel<<<grid, kSelThreads, 0, h->stream>>>(dist, ld_sel, ld_sel, 0ull, sel, hist, shifts[p], widths[p]);
      LAUNCHED(h);
    }
    tc3_threshold_kernel<<<2, 128, 0, h->stream>>>(sel, sb, nqg, thr);
    LAUNCHED(h);
  }

  // 2. filter pass over all rows (nblk passes in one launch)
  CK(cudaMemsetAsync(h->tc_cnt.p, 0, sizeof(unsigned int) * (nq_pad + kTcGroupBlocks + 4), h->stream));
  const int grid_f = 2 * static_cast<int>(std::min<int64_t>(max_clusters, n_tiles));
  cudaEvent_t e0 = nullptr, e1 = nullptr;
  if (h->timing && h->scan_ev_used + 2 <= (1u << 16)) {
    int rc = scan_event(h, &e0);
    if (rc != RSE_OK) return rc;
  }
  const bool overlap = bm25 && !bm25->enqueued;
  if (overlap) {
    if (!h->ev_prefilter) CK(cudaEventCreateWithFlags(&h->ev_prefilter, cudaEventDisableTiming));
    CK(cudaEventRecord(h->ev_prefilter, h->stream));
  }
  tl_mark(h, kTlPrefilter, h->stream);
  knn_tc3_kernel<1, KB><<<grid_f, kT3Threads, kT3SmemBytes, h->stream>>>(
      h->tmap_a16, h->tmap_q16, n_tiles, 1, nqg, nblk, thr, nullptr, 0, static_cast<uint2*>(h->tc_rows.p),
      static_cast<unsigned int*>(h->tc_cnt.p), kTcCandCap, nullptr);
  LAUNCHED(h);
  tl_mark(h, kTlFilterEnd, h->stream);
  if (overlap) {
    int rc = enqueue_bm25_overlapped(h, *bm25, h->ev_prefilter);
    if (rc != RSE_OK) return rc;
  }
  if (e0) {
    int rc = scan_event(h, &e1);
    if (rc != RSE_OK) return rc;
    h->scan_ev_passes.push_back(nblk);                        // this event pair covers nblk 256-query passes
  }
  h->stats.knn_scan_launches++;
  h->stats.tc_filter_launches += nblk;

  // 3. refine on the approximate values, 4. exact re-score + sort + emit (one CTA per query); a query whose
  //    survivor list overflowed arms the second chance instead (thr2 from the survivors that were kept)
  float* thr2 = thr + nq_pad;
  unsigned int* gate = static_cast<unsigned int*>(h->tc_cnt.p) + nq_pad;
  {
    int rc = knn_tc_refine<KB>(h, q_dev, sb, nqg, kprime, cand_dev, status_dev, nullptr, nullptr, thr2, gate,
                           sampled ? thr + 2 * nq_pad : nullptr);
    if (rc != RSE_OK) return rc;
  }
  // 5. second chance: one more filter pass + refine for the armed queries only (blocks without one are skipped).
  //    Enqueued unconditionally, gated on the device: two near-empty launches when no query needs it.
  knn_tc3_kernel<1, KB><<<grid_f, kT3Threads, kT3SmemBytes, h->stream>>>(
      h->tmap_a16, h->tmap_q16, n_tiles, 1, nqg, nblk, thr2, nullptr, 0, static_cast<uint2*>(h->tc_rows.p),
      static_cast<unsigned int*>(h->tc_cnt.p), kTcCandCap, gate);
  LAUNCHED(h);
  return knn_tc_refine<KB>(h, q_dev, sb, nqg, kprime, cand_dev, status_dev, thr2, gate, nullptr, nullptr, nullptr);
}

// K4 serves every width D = 64 KB, KB = 1..8 (knn_tc3_kernel<MODE, KB>); any other width keeps the exact scan
bool tc_width_ok(int dim) { return dim % kT3BK == 0 && dim >= kT3BK && dim <= kT3MaxKBlocks * kT3BK; }

bool tc_eligible(const rse_index* h, int nq, int kprime) {
  if (h->tc_mode == 1 || !tc_width_ok(h->dim)) return false;
  if (((h->n_rows + 127) / 128) * 128 < 8ll * kprime || h->n_rows < 1024) return false;   // the probe needs a usable sample
  if (kprime * 4 > kTcCandCap || kprime * 2 > kTcRefineCap) return false;
  if (h->tc_mode == 2) return true;
  // a single query joins the batches once the shadow exists (K4 reads 768 B per row instead of 1536: 0.76 against
  // 1.18 ms per call on S-600k) — but it never makes the library build the shadow.  That was measured at 384 only:
  // at any other width a single query keeps the exact scan.
  return (nq >= RSE_TC_MIN_BATCH || (h->shadow_state == 1 && h->dim == kScanD)) && h->n_rows >= 262144;
}

// the shadow (built once) and every group of up to kTcGroupBlocks x 256 queries; leaves shadow_state = -1 and enqueues
// nothing when the corpus cannot use K4
template <int KB>
int knn_tc3_run(rse_index* h, const float* q_dev, const double* sb, int nq, int kprime, long long* cand_dev,
                int* status, Bm25Job* bm25) {
  int rc = ensure_shadow<KB>(h);
  if (rc != RSE_OK || h->shadow_state < 0) return rc;
  for (int b0 = 0; b0 < nq; b0 += kTcGroupBlocks * kTcBN) {
    const int nqg = std::min(kTcGroupBlocks * kTcBN, nq - b0);
    rc = knn_tc3_group<KB>(h, q_dev + static_cast<int64_t>(b0) * h->dim, sb + b0, nqg, kprime,
                           cand_dev + static_cast<int64_t>(b0) * kprime * 3, status + b0, bm25);
    if (rc != RSE_OK) return rc;
  }
  return RSE_OK;
}

// Local top-kprime for nq device-resident queries → packed candidates (device), in two halves: _begin enqueues
// everything and, on the tensor-core path, an asynchronous read-back of the per-query overflow flags; _finish
// waits for that read-back only (an event, not the stream) and re-runs flagged queries through the exact scan.
// The hybrid step enqueues its BM25 kernels between the two, so the device never idles on the host round trip, and
// hands `bm25` down to be enqueued underneath the filter pass when the tensor-core path runs.  The flags land in `pin`.
int knn_local_begin(rse_index* h, const float* q_dev, int nq, int kprime, long long* cand_dev, PinnedFlags& pin,
                    Bm25Job* bm25, PendingKnn& pend) {
  pend = PendingKnn{};
  if (!h->emb) return fail(h, RSE_ERR_STATE, "rse_knn: no embeddings loaded");
  if (nq <= 0) return RSE_OK;
  if (kprime < 1 || kprime > RSE_MAX_KPRIME)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_knn: kprime must be in [1, 4096] (sqlite-vec caps k at 4096)");
  ENSURE(h->sb, sizeof(double) * nq);
  if (h->hist.bytes < sizeof(unsigned int) * kSelBins * kTcBN) {
    ENSURE(h->hist, sizeof(unsigned int) * kSelBins * kTcBN);
    CK(cudaMemsetAsync(h->hist.p, 0, h->hist.bytes, h->stream));
  }
  double* sb = static_cast<double*>(h->sb.p);
  if (h->fma) knn_query_prep_kernel<true><<<(nq + 3) / 4, 128, 0, h->stream>>>(q_dev, nq, h->dim, sb);
  else knn_query_prep_kernel<false><<<(nq + 3) / 4, 128, 0, h->stream>>>(q_dev, nq, h->dim, sb);
  LAUNCHED(h);

  if (!tc_eligible(h, nq, kprime)) return knn_exact_groups(h, q_dev, sb, nq, kprime, cand_dev);

  // ---- tensor-core path in blocks of 256 queries, exact fallback for overflowed queries
  ENSURE(h->tc_status, sizeof(int) * nq);
  int* status = static_cast<int*>(h->tc_status.p);
  {
    int rc = RSE_OK;
    switch (h->dim / kT3BK) {                      // tc_eligible: dim = 64 KB, KB = 1..8
      case 1: rc = knn_tc3_run<1>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      case 2: rc = knn_tc3_run<2>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      case 3: rc = knn_tc3_run<3>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      case 4: rc = knn_tc3_run<4>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      case 5: rc = knn_tc3_run<5>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      case 6: rc = knn_tc3_run<6>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      case 7: rc = knn_tc3_run<7>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      case 8: rc = knn_tc3_run<8>(h, q_dev, sb, nq, kprime, cand_dev, status, bm25); break;
      default: return fail(h, RSE_ERR_STATE, "rse_knn: no tensor-core instantiation for this width");
    }
    if (rc != RSE_OK) return rc;
    if (h->shadow_state < 0) return knn_exact_groups(h, q_dev, sb, nq, kprime, cand_dev);
  }
  h->stats.tc_queries += nq;
  if (pin.n < static_cast<size_t>(nq)) {
    if (pin.p) CK(cudaFreeHost(pin.p));
    pin = PinnedFlags{};
    CK(cudaMallocHost(reinterpret_cast<void**>(&pin.p), sizeof(int) * (static_cast<size_t>(nq) + 256)));
    pin.n = static_cast<size_t>(nq) + 256;
  }
  if (!h->ev_status) CK(cudaEventCreateWithFlags(&h->ev_status, cudaEventDisableTiming));
  CK(cudaMemcpyAsync(pin.p, status, sizeof(int) * nq, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaEventRecord(h->ev_status, h->stream));
  pend = PendingKnn{q_dev, nq, kprime, cand_dev, pin.p, h->ev_status};
  return RSE_OK;
}

int knn_local_finish(rse_index* h, const PendingKnn& pend) {
  if (!pend.flags) return RSE_OK;
  CK(cudaEventSynchronize(pend.ev));
  const int kprime = pend.kprime;
  const double* sb = static_cast<const double*>(h->sb.p);
  std::vector<int> flagged;
  for (int q = 0; q < pend.nq; ++q)
    if (pend.flags[q]) flagged.push_back(q);
  if (flagged.empty()) return RSE_OK;
  // the flagged queries (a mass tie at the K'-th distance; second chance already tried) go through the exact scan,
  // gathered into one contiguous group: one pass serves up to 16 of them wherever they sat in the batch
  const int nf = static_cast<int>(flagged.size());
  h->stats.tc_fallback_queries += nf;
  ENSURE(h->fb_list, sizeof(int) * nf);
  ENSURE(h->fb_q, sizeof(float) * static_cast<size_t>(nf) * h->dim);
  ENSURE(h->fb_sb, sizeof(double) * nf);
  ENSURE(h->fb_cand, sizeof(long long) * static_cast<size_t>(nf) * kprime * 3);
  CK(cudaMemcpyAsync(h->fb_list.p, flagged.data(), sizeof(int) * nf, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));                      // `flagged` is a pageable temporary
  knn_gather_queries_kernel<<<nf, 128, 0, h->stream>>>(pend.q, sb, static_cast<const int*>(h->fb_list.p), h->dim,
                                                      static_cast<float*>(h->fb_q.p), static_cast<double*>(h->fb_sb.p));
  LAUNCHED(h);
  int rc = knn_exact_groups(h, static_cast<const float*>(h->fb_q.p), static_cast<const double*>(h->fb_sb.p), nf, kprime,
                            static_cast<long long*>(h->fb_cand.p));
  if (rc != RSE_OK) return rc;
  knn_scatter_cand_kernel<<<nf, 128, 0, h->stream>>>(static_cast<const long long*>(h->fb_cand.p),
                                                    static_cast<const int*>(h->fb_list.p), kprime * 3, pend.cand);
  LAUNCHED(h);
  return RSE_OK;
}

int knn_local(rse_index* h, const float* q_dev, int nq, int kprime, long long* cand_dev) {
  PendingKnn pend;
  int rc = knn_local_begin(h, q_dev, nq, kprime, cand_dev, h->pin_status, nullptr, pend);
  if (rc != RSE_OK) return rc;
  return knn_local_finish(h, pend);
}

int aggregate(rse_index* h, const long long* cand, int nq, int k, int kprime, float* o_dist, long long* o_rowid,
              int* o_movie, int* o_count) {
  const size_t smem = static_cast<size_t>(kprime) * 8;
  knn_aggregate_kernel<<<nq, kSelThreads, smem, h->stream>>>(cand, nq, kprime, k, o_dist, o_rowid, o_movie, o_count);
  LAUNCHED(h);
  return RSE_OK;
}

// the n_lists candidate lists of K' per query gathered from the shards of one corpus → one merged list in h->cand
int merge_candidates(rse_index* h, const long long* gathered, int n_lists, int nq, int kprime) {
  const int n2 = next_pow2(n_lists * kprime);
  const size_t smem = static_cast<size_t>(n2) * 12;
  if (smem > 200 * 1024)
    return fail(h, RSE_ERR_UNSUPPORTED, "knn merge: n_lists*kprime too large for the merge kernel");
  if (smem > 48 * 1024) CK(cudaFuncSetAttribute(knn_merge_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
  ENSURE(h->cand, sizeof(long long) * static_cast<size_t>(nq) * kprime * 3);
  knn_merge_kernel<<<nq, kSelThreads, smem, h->stream>>>(gathered, n_lists, nq, kprime, n2,
                                                         static_cast<long long*>(h->cand.p));
  LAUNCHED(h);
  return RSE_OK;
}

// ---- exact movie-level KNN (knn_movies_exact.cuh, DESIGN §11)
// The corpus's movie layout, once per load: n_movie_slots and whether the competing rows are sorted by movie_idx.
int movies_layout(rse_index* h) {
  if (h->movies_sorted >= 0) return RSE_OK;
  const int n_spans = static_cast<int>(std::max<int64_t>(1, (h->n_rows + kLayoutRowsPerThread - 1) / kLayoutRowsPerThread));
  ENSURE(h->mx_span, sizeof(int4) * n_spans);
  ENSURE(h->mx_meta, sizeof(unsigned int) * 2);
  unsigned int* meta = static_cast<unsigned int*>(h->mx_meta.p);   // [0] n_movie_slots, [1] sorted
  CK(cudaMemsetAsync(meta, 0, sizeof(unsigned int) * 2, h->stream));
  if (h->n_rows > 0) {
    movies_layout_kernel<<<(n_spans + 127) / 128, 128, 0, h->stream>>>(h->movie_idx, h->amag, h->n_rows, n_spans,
                                                                      static_cast<int4*>(h->mx_span.p), meta);
    LAUNCHED(h);
    movies_layout_join_kernel<<<1, 1, 0, h->stream>>>(static_cast<const int4*>(h->mx_span.p), n_spans,
                                                      reinterpret_cast<int*>(meta + 1));
    LAUNCHED(h);
  }
  unsigned int host[2] = {0u, 0u};
  CK(cudaMemcpyAsync(host, meta, sizeof(host), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->movie_slots = host[0];
  h->movies_sorted = (h->n_rows == 0 || host[1]) ? 1 : 0;
  return RSE_OK;
}

// The k nearest movies of nq device-resident queries (|q| factors sb ready) over every row: the exact scan of
// knn_scan.cuh per group of 16 queries, the segmented minimum into best[query][movie], then the radix select over
// the movie keys per group of <= 256 queries.  Outputs are device [nq, k] in rse_knn_movies' layout.  Queries go in
// chunks whose best buffer fits mx_budget.
int movies_exact_scan(rse_index* h, const float* q, const double* sb, int nq, int k, float* o_dist,
                      long long* o_rowid, int* o_movie, int* o_count) {
  const int QB = kScanMaxQB;
  const int64_t n_slots = std::max<int64_t>(h->movie_slots, 1);   // no movie at all: one empty slot, nothing found
  const size_t per_q = sizeof(unsigned long long) * static_cast<size_t>(n_slots);
  int64_t chunk = std::max<int64_t>(1, static_cast<int64_t>(h->mx_budget / per_q));
  if (chunk >= QB) chunk -= chunk % QB;
  chunk = std::min<int64_t>(chunk, nq);
  const int sel_q = std::min(nq, kTcBN);
  ENSURE(h->mx_best, per_q * static_cast<size_t>(chunk));
  ENSURE(h->dist, sizeof(float) * static_cast<size_t>(QB) * h->dist_ld);
  ENSURE(h->sel, sizeof(SelState) * std::max(nq, kTcBN));
  ENSURE(h->mx_keys, sizeof(unsigned long long) * static_cast<size_t>(sel_q) * k);
  ENSURE(h->mx_cand, sizeof(long long) * static_cast<size_t>(sel_q) * k * 3);
  if (h->hist.bytes < sizeof(unsigned int) * kSelBins * kTcBN) {
    ENSURE(h->hist, sizeof(unsigned int) * kSelBins * kTcBN);
    CK(cudaMemsetAsync(h->hist.p, 0, h->hist.bytes, h->stream));
  }
  unsigned long long* best = static_cast<unsigned long long*>(h->mx_best.p);
  float* dist = static_cast<float*>(h->dist.p);
  SelState* sel = static_cast<SelState*>(h->sel.p);
  unsigned int* hist = static_cast<unsigned int*>(h->hist.p);
  unsigned long long* keys = static_cast<unsigned long long*>(h->mx_keys.p);
  long long* cand = static_cast<long long*>(h->mx_cand.p);
  static const int shifts[6] = {53, 42, 32, 21, 10, 0};
  static const int widths[6] = {11, 11, 10, 11, 11, 10};
  const int sel_blocks = static_cast<int>(std::min<int64_t>((n_slots + 4095) / 4096, h->sm_count * 2));
  const int kp2 = next_pow2(k);
  const size_t fsmem = static_cast<size_t>(kp2) * 12;
  if (fsmem > 48 * 1024) CK(cudaFuncSetAttribute(select_finish_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  for (int c0 = 0; c0 < nq; c0 += static_cast<int>(chunk)) {
    const int nc = std::min(static_cast<int>(chunk), nq - c0);
    CK(cudaMemsetAsync(best, 0xFF, per_q * nc, h->stream));
    for (int g0 = c0; g0 < c0 + nc; g0 += QB) {
      const int ng = std::min(QB, c0 + nc - g0);
      cudaEvent_t e0 = nullptr, e1 = nullptr;                    // rse_set_timing: the scan's share of the call
      if (h->timing && h->scan_ev_used + 2 <= (1u << 16)) {
        int rc = scan_event(h, &e0);
        if (rc != RSE_OK) return rc;
      }
      int rc = h->fma ? launch_scan<true>(h, q + static_cast<int64_t>(g0) * h->dim, sb + g0, ng, dist)
                      : launch_scan<false>(h, q + static_cast<int64_t>(g0) * h->dim, sb + g0, ng, dist);
      if (rc != RSE_OK) return rc;
      if (e0) {
        rc = scan_event(h, &e1);
        if (rc != RSE_OK) return rc;
        h->scan_ev_passes.push_back(1);
      }
      const int seg_blocks = static_cast<int>(std::max<int64_t>(1, std::min<int64_t>(
          (h->n_rows + kSegThreads - 1) / kSegThreads, std::max(1, h->sm_count * 16 / ng))));
      unsigned long long* bg = best + static_cast<int64_t>(g0 - c0) * n_slots;
      const uint32_t* d32 = reinterpret_cast<const uint32_t*>(dist);
      if (h->movies_sorted)
        movies_segmin_kernel<true><<<dim3(seg_blocks, ng), kSegThreads, 0, h->stream>>>(
            d32, h->dist_ld, h->n_rows, h->pos_base, h->movie_idx, n_slots, bg);
      else
        movies_segmin_kernel<false><<<dim3(seg_blocks, ng), kSegThreads, 0, h->stream>>>(
            d32, h->dist_ld, h->n_rows, h->pos_base, h->movie_idx, n_slots, bg);
      LAUNCHED(h);
    }
    for (int s0 = c0; s0 < c0 + nc; s0 += kTcBN) {
      const int ns = std::min(kTcBN, c0 + nc - s0);
      const unsigned long long* bs = best + static_cast<int64_t>(s0 - c0) * n_slots;
      select_init_kernel<<<(ns + 127) / 128, 128, 0, h->stream>>>(sel, ns, static_cast<unsigned int>(k));
      LAUNCHED(h);
      const dim3 grid(std::max(sel_blocks, 1), ns);
      for (int p = 0; p < 6; ++p) {
        select_keys_pass_kernel<<<grid, kSelThreads, 0, h->stream>>>(bs, n_slots, n_slots, sel, hist, shifts[p], widths[p]);
        LAUNCHED(h);
      }
      select_keys_collect_kernel<<<grid, kSelThreads, 0, h->stream>>>(bs, n_slots, n_slots, sel, keys, k);
      LAUNCHED(h);
      select_finish_kernel<<<ns, kSelThreads, fsmem, h->stream>>>(keys, sel, k, kp2, h->pos_base, h->rowid,
                                                                 h->movie_idx, cand);
      LAUNCHED(h);
      const int64_t o = static_cast<int64_t>(s0) * k;
      knn_unpack_kernel<<<ns, 128, 0, h->stream>>>(cand, ns, k, o_dist + o, nullptr, o_rowid + o, o_movie + o,
                                                   o_count + s0);
      LAUNCHED(h);
    }
  }
  return RSE_OK;
}

int upload_queries(rse_index* h, const float* q_host, int nq) {
  ENSURE(h->staged.q, sizeof(float) * static_cast<size_t>(nq) * h->dim);
  CK(cudaMemcpyAsync(h->staged.q.p, q_host, sizeof(float) * static_cast<size_t>(nq) * h->dim, cudaMemcpyHostToDevice,
                     h->stream));
  h->stats.h2d_bytes += static_cast<int64_t>(sizeof(float)) * nq * h->dim;
  return RSE_OK;
}

int finish_embeddings(rse_index* h, const uint8_t* valid_dev) {
  CK(cudaMalloc(&h->amag, sizeof(float) * std::max<int64_t>(h->n_rows, 1)));
  if (h->n_rows > 0) {
    const int threads = 128;
    const int grid = static_cast<int>((h->n_rows + threads - 1) / threads);
    if (h->fma) knn_row_sqmag_kernel<true><<<grid, threads, 0, h->stream>>>(h->emb, h->n_rows, h->dim, valid_dev, h->amag);
    else knn_row_sqmag_kernel<false><<<grid, threads, 0, h->stream>>>(h->emb, h->n_rows, h->dim, valid_dev, h->amag);
    LAUNCHED(h);
  }
  h->dist_ld = ((h->n_rows + 31) / 32) * 32;
  if (h->dist_ld < 32) h->dist_ld = 32;
  CK(cudaStreamSynchronize(h->stream));
  h->stats.emb_rows = h->n_rows;
  h->stats.emb_dim = h->dim;
  return RSE_OK;
}

int check_emb_args(rse_index* h, const float* emb, int64_t n_rows, int32_t dim, int64_t pos_base) {
  if (!h) return RSE_ERR_INVALID;
  if ((!emb && n_rows > 0) || n_rows < 0 || dim < 1 || dim > 65536)
    return fail(h, RSE_ERR_INVALID, "rse_load_embeddings: bad emb/n_rows/dim");
  if (pos_base < 0 || (pos_base % RSE_VEC0_BLOCK) != 0)
    return fail(h, RSE_ERR_INVALID, "rse_load_embeddings: pos_base must be a non-negative multiple of 1024");
  if (static_cast<uint64_t>(pos_base) + static_cast<uint64_t>(n_rows) >= 0xFFFFFFFFull)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_load_embeddings: global position must fit 32 bits");
  return RSE_OK;
}

}  // namespace

// =================================================================== C-ABI
extern "C" {

int rse_abi_version(void) { return RSE_ABI_VERSION; }

const char* rse_last_error(const rse_index* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

int rse_create(int32_t device, rse_index** out) {
  rse_index* h = nullptr;
  if (!out) return fail(nullptr, RSE_ERR_INVALID, "rse_create: out is NULL");
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n <= 0)
    return fail(nullptr, RSE_ERR_CUDA,
                std::string("rse_create: no CUDA device (") + cudaGetErrorString(e) + "); librse has no CPU fallback");
  if (device < 0 || device >= n) return fail(nullptr, RSE_ERR_INVALID, "rse_create: device ordinal out of range");
  e = cudaSetDevice(device);
  if (e != cudaSuccess) return fail(nullptr, RSE_ERR_CUDA, std::string("cudaSetDevice: ") + cudaGetErrorString(e));
  cudaDeviceProp prop;
  e = cudaGetDeviceProperties(&prop, device);
  if (e != cudaSuccess) return fail(nullptr, RSE_ERR_CUDA, std::string("cudaGetDeviceProperties: ") + cudaGetErrorString(e));
  if (prop.major != 10)
    return fail(nullptr, RSE_ERR_UNSUPPORTED, "rse_create: librse is built for sm_100a (B200) only");
  h = new rse_index();
  h->device = device;
  h->sm_count = prop.multiProcessorCount;
  e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    delete h;
    return fail(nullptr, RSE_ERR_CUDA, std::string("cudaStreamCreate: ") + cudaGetErrorString(e));
  }
  h->stream = h->own_stream;
  for (auto& ev : h->ev) cudaEventCreate(&ev);
  if (cudaMalloc(&h->dev_counters, sizeof(unsigned long long) * 8) == cudaSuccess)
    cudaMemset(h->dev_counters, 0, sizeof(unsigned long long) * 8);
  else
    h->dev_counters = nullptr;
  if (const char* ev = std::getenv("RSE_TIMELINE")) h->timeline = ev[0] == '1';
  if (const char* ev = std::getenv("RSE_TC_SAMPLE_STRIDE")) { const int v = std::atoi(ev); if (v >= 2 && v <= 256) h->sample_stride = v; }
  if (const char* ev = std::getenv("RSE_TC_SAMPLE_MIN_TILES")) { const int v = std::atoi(ev); if (v >= 1) h->sample_min_tiles = v; }
  if (const char* ev = std::getenv("RSE_TC_PROBE_RANK")) { const int v = std::atoi(ev); if (v >= 1) h->probe_rank = v; }
  if (const char* ev = std::getenv("RSE_MOVIES_EXACT_BUDGET")) { const long long v = std::atoll(ev); if (v >= 1) h->mx_budget = static_cast<size_t>(v); }
  if (const char* ev = std::getenv("RSE_TC_SURVIVOR_DIV")) { const int v = std::atoi(ev); if (v >= 1 && v <= 64) h->survivor_div = v; }
  *out = h;
  return RSE_OK;
}

void rse_destroy(rse_index* h) {
  if (!h) return;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (cudaStream_t st : {h->stream_b, h->stream_h2d, h->stream_d2h})   // tickets may still be in flight
    if (st) cudaStreamSynchronize(st);
  release_embeddings(h);
  release_bm25(h);
  for (DevBuf* b : {&h->sb, &h->sel, &h->hist, &h->selkeys, &h->cand, &h->dist, &h->o_dist, &h->o_pos, &h->o_rowid,
                    &h->o_movie, &h->o_count, &h->b_chi, &h->b_clo, &h->b_ccnt, &h->b_score, &h->b_doc, &h->b_count,
                    &h->f_bid, &h->f_bsc, &h->f_bcnt, &h->f_sid, &h->f_sds, &h->f_scnt, &h->f_oid, &h->f_osc, &h->f_oa,
                    &h->f_ob, &h->f_ocnt, &h->tc_thr,
                    &h->tc_rows, &h->tc_cnt, &h->tc_status, &h->fb_list, &h->fb_q, &h->fb_sb, &h->fb_cand, &h->tc_q16, &h->b_shi, &h->b_slo, &h->b_scnt,
                    &h->b_status, &h->b_flagged, &h->mx_span, &h->mx_meta, &h->mx_best, &h->mx_list, &h->mx_q,
                    &h->mx_sb, &h->mx_keys, &h->mx_cand, &h->mx_dist, &h->mx_rowid, &h->mx_movie, &h->mx_count})
    free_buf(*b);
  if (h->pin_status.p) cudaFreeHost(h->pin_status.p);
  if (h->pin_stage) cudaFreeHost(h->pin_stage);
  if (h->pin_out) cudaFreeHost(h->pin_out);
  for (auto& sl : h->out_slot) {
    if (sl.pin) cudaFreeHost(sl.pin);
    if (sl.flags.p) cudaFreeHost(sl.flags.p);
    if (sl.ev) cudaEventDestroy(sl.ev);
    free_batch(sl.in);
    free_buf(sl.f_pack);
  }
  if (h->stream_h2d) cudaStreamDestroy(h->stream_h2d);
  if (h->stream_d2h) cudaStreamDestroy(h->stream_d2h);
  if (h->ev_fused) cudaEventDestroy(h->ev_fused);
  for (int i = 0; i < 2; ++i) { if (h->pin_q[i]) cudaFreeHost(h->pin_q[i]); if (h->ev_q[i]) cudaEventDestroy(h->ev_q[i]); }
  free_buf(h->f_pack);
  free_batch(h->staged);
  for (Batch& st : h->stash) free_batch(st);
  if (h->ev_status) cudaEventDestroy(h->ev_status);
  if (h->ev_stage) cudaEventDestroy(h->ev_stage);
  for (cudaEvent_t e : h->tl) if (e) cudaEventDestroy(e);
  if (h->ev_prefilter) cudaEventDestroy(h->ev_prefilter);
  if (h->ev_bm25_done) cudaEventDestroy(h->ev_bm25_done);
  if (h->stream_b) cudaStreamDestroy(h->stream_b);
  free_ptr(h->doc_ids);
  free_ptr(h->movie_ids);
  free_ptr(h->rr_doc_ids); free_ptr(h->rr_doc_indptr); free_ptr(h->rr_doc_tok);
  for (DevBuf* b : {&h->rr_fid, &h->rr_fsc, &h->rr_fa, &h->rr_fb, &h->rr_fcnt, &h->rr_row, &h->rr_ab, &h->rr_qnp,
                    &h->rr_qnt, &h->rr_qpb, &h->rr_qtb, &h->rr_meta, &h->rr_qptr, &h->rr_qtok, &h->rr_ids, &h->rr_types,
                    &h->rr_cus, &h->rr_logit, &h->rr_pack})
    free_buf(*b);
  if (h->rr_pin_meta) cudaFreeHost(h->rr_pin_meta);
  if (h->rr_pin_out) cudaFreeHost(h->rr_pin_out);
  for (cudaEvent_t e : h->rr_ev) if (e) cudaEventDestroy(e);
  for (auto& t : h->tok) if (t.blob) cudaFree(t.blob);
  for (DevBuf* b : {&h->tk_text, &h->tk_offs, &h->tk_count, &h->tk_cu64, &h->tk_cu32, &h->tk_ids, &h->tk_meta}) free_buf(*b);
  if (h->tk_pin) cudaFreeHost(h->tk_pin);
  for (DevBuf* b : {&h->ck_chunks, &h->ck_bytes, &h->ck_cu32, &h->ck_meta}) free_buf(*b);
  if (h->tk_pin_meta) cudaFreeHost(h->tk_pin_meta);
  for (auto& e : h->enc) enc_release(e);
  free_ptr(h->dev_counters);
  if (h->comm) { if (NcclApi* n = nccl_api()) n->CommDestroy(h->comm); h->comm = nullptr; }
  free_buf(h->sh_cand); free_buf(h->sh_mine);
  for (auto& ev : h->ev) if (ev) cudaEventDestroy(ev);
  for (auto& ev : h->scan_ev) cudaEventDestroy(ev);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
}

int rse_set_stream(rse_index* h, void* s) {
  if (!h) return RSE_ERR_INVALID;
  CK(cudaStreamSynchronize(h->stream));
  h->stream = static_cast<cudaStream_t>(s);   // 0 is a real stream: the legacy default stream (torch's default)
  return RSE_OK;
}

int rse_use_own_stream(rse_index* h) {
  if (!h) return RSE_ERR_INVALID;
  CK(cudaStreamSynchronize(h->stream));
  h->stream = h->own_stream;
  return RSE_OK;
}

int rse_synchronize(rse_index* h) {
  if (!h) return RSE_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  return RSE_OK;
}

int rse_set_fma(rse_index* h, int32_t use_fma) {
  if (!h) return RSE_ERR_INVALID;
  if (h->emb) return fail(h, RSE_ERR_STATE, "rse_set_fma: set before loading embeddings");
  h->fma = use_fma != 0;
  return RSE_OK;
}

int rse_set_tc_mode(rse_index* h, int32_t mode) {
  if (!h) return RSE_ERR_INVALID;
  if (mode < 0 || mode > 2) return fail(h, RSE_ERR_INVALID, "rse_set_tc_mode: mode must be 0..2");
  h->tc_mode = mode;
  return RSE_OK;
}

int rse_set_bm25_mode(rse_index* h, int32_t mode) {
  if (!h) return RSE_ERR_INVALID;
  if (mode < 0 || mode > 2) return fail(h, RSE_ERR_INVALID, "rse_set_bm25_mode: mode must be 0..2");
  h->bm25_mode = mode;
  return RSE_OK;
}

int rse_set_timing(rse_index* h, int32_t enabled) {
  if (!h) return RSE_ERR_INVALID;
  h->timing = enabled != 0;
  return RSE_OK;
}

int rse_get_stats(rse_index* h, rse_stats* out) {
  if (!h || !out) return RSE_ERR_INVALID;
  // resolve pending scan event pairs (the caller has synchronised; if not, do it)
  if (h->scan_ev_used) {
    CK(cudaStreamSynchronize(h->stream));
    for (size_t i = 0; i + 1 < h->scan_ev_used; i += 2) {
      float ms = 0.f;
      CK(cudaEventElapsedTime(&ms, h->scan_ev[i], h->scan_ev[i + 1]));
      h->stats.scan_ms_total += ms;
      // a multi-block K4 launch counts as that many passes, so scan_ms_total / scan_launches_timed stays "per pass"
      h->stats.scan_launches_timed += (i / 2 < h->scan_ev_passes.size()) ? h->scan_ev_passes[i / 2] : 1;
    }
    h->scan_ev_used = 0;
    h->scan_ev_passes.clear();
  }
  if (h->dev_counters) {
    unsigned long long c[4] = {0, 0, 0, 0};
    CK(cudaStreamSynchronize(h->stream));
    if (h->stream_b) CK(cudaStreamSynchronize(h->stream_b));
    CK(cudaMemcpy(c, h->dev_counters, sizeof(c), cudaMemcpyDeviceToHost));
    h->stats.bm25_fallback_queries = static_cast<int64_t>(c[0]);
    h->stats.bm25_finalists = static_cast<int64_t>(c[1]);
    h->stats.bm25_candidates = static_cast<int64_t>(c[2]);
    h->stats.tc_second_chance_queries = static_cast<int64_t>(c[3]);
  }
  *out = h->stats;
  return RSE_OK;
}

int rse_stats_reset(rse_index* h) {
  if (!h) return RSE_ERR_INVALID;
  const int64_t rows = h->stats.emb_rows, post = h->stats.bm25_postings, docs = h->stats.bm25_docs;
  const int dim = h->stats.emb_dim;
  h->stats = rse_stats{};
  h->scan_ev_used = 0;
  h->scan_ev_passes.clear();
  if (h->dev_counters) {
    CK(cudaStreamSynchronize(h->stream));
    if (h->stream_b) CK(cudaStreamSynchronize(h->stream_b));
    CK(cudaMemset(h->dev_counters, 0, sizeof(unsigned long long) * 8));
  }
  h->stats.emb_rows = rows; h->stats.emb_dim = dim; h->stats.bm25_postings = post; h->stats.bm25_docs = docs;
  return RSE_OK;
}

// ------------------------------------------------------------------ embeddings
int rse_load_embeddings(rse_index* h, const float* emb_host, int64_t n_rows, int32_t dim, const uint8_t* valid_host,
                        const int64_t* rowid_host, const int32_t* movie_idx_host, int64_t pos_base) {
  int rc = check_emb_args(h, emb_host, n_rows, dim, pos_base);
  if (rc != RSE_OK) return rc;
  CK(cudaSetDevice(h->device));
  release_embeddings(h);
  const size_t bytes = sizeof(float) * static_cast<size_t>(std::max<int64_t>(n_rows, 1)) * dim;
  CK(cudaMalloc(&h->emb_owned, bytes));
  if (n_rows > 0) {
    // The matrix usually arrives as a memory-mapped sidecar (store.load_or_export): gigabytes of PAGEABLE memory,
    // possibly not yet in the page cache.  One cudaMemcpy of that stages through the driver's small bounce
    // buffer and serialises page-in and transfer; here the host side is cut into 64 MB pieces that are copied
    // into two pinned buffers alternately (the memcpy faults the next pages in) while the previous piece is on
    // its way to the device.
    const size_t total = sizeof(float) * static_cast<size_t>(n_rows) * dim;
    const size_t piece = size_t(64) << 20;
    if (total <= 2 * piece) {
      CK(cudaMemcpyAsync(h->emb_owned, emb_host, total, cudaMemcpyHostToDevice, h->stream));
    } else {
      char* pin[2] = {nullptr, nullptr};
      cudaEvent_t ev[2] = {nullptr, nullptr};
      cudaError_t ce = cudaSuccess;
      for (int i = 0; i < 2 && ce == cudaSuccess; ++i) {
        ce = cudaMallocHost(reinterpret_cast<void**>(&pin[i]), piece);
        if (ce == cudaSuccess) ce = cudaEventCreateWithFlags(&ev[i], cudaEventDisableTiming);
      }
      const char* src = reinterpret_cast<const char*>(emb_host);
      char* dst = reinterpret_cast<char*>(h->emb_owned);
      // the staging copy is the slow side (one thread moves ~10 GB/s out of the page cache, the link takes 25+):
      // a few threads share every piece (RSE_UPLOAD_THREADS, default min(16, cores); S-600k, 7.4 GB, page cache warm:
      // 1 / 2 / 8 / 16 threads -> 0.64 / 0.41 / 0.32 / 0.29 s)
      int n_threads = static_cast<int>(std::min(16u, std::max(1u, std::thread::hardware_concurrency())));
      if (const char* ev_t = std::getenv("RSE_UPLOAD_THREADS")) { const int v = std::atoi(ev_t); if (v >= 1 && v <= 64) n_threads = v; }
      auto par_copy = [n_threads](char* d, const char* s, size_t n) {
        if (n_threads <= 1 || n < (size_t(8) << 20)) { std::memcpy(d, s, n); return; }
        const size_t per = ((n / n_threads) + 4095) & ~size_t(4095);
        std::vector<std::thread> workers;
        for (int t = 1; t < n_threads; ++t) {
          const size_t o = per * t;
          if (o >= n) break;
          workers.emplace_back([=] { std::memcpy(d + o, s + o, std::min(per, n - o)); });
        }
        std::memcpy(d, s, std::min(per, n));
        for (auto& w : workers) w.join();
      };
      int b = 0;
      for (size_t off = 0; off < total && ce == cudaSuccess; off += piece, b ^= 1) {
        const size_t n = std::min(piece, total - off);
        ce = cudaEventSynchronize(ev[b]);                       // this buffer's previous piece has left
        if (ce != cudaSuccess) break;
        par_copy(pin[b], src + off, n);
        ce = cudaMemcpyAsync(dst + off, pin[b], n, cudaMemcpyHostToDevice, h->stream);
        if (ce == cudaSuccess) ce = cudaEventRecord(ev[b], h->stream);
      }
      if (ce == cudaSuccess) ce = cudaStreamSynchronize(h->stream);
      for (int i = 0; i < 2; ++i) { if (pin[i]) cudaFreeHost(pin[i]); if (ev[i]) cudaEventDestroy(ev[i]); }
      if (ce != cudaSuccess) return fail(h, RSE_ERR_CUDA, std::string("rse_load_embeddings (chunked upload): ") + cudaGetErrorString(ce));
    }
  }
  h->emb = h->emb_owned;
  h->n_rows = n_rows; h->dim = dim; h->pos_base = static_cast<uint64_t>(pos_base);
  uint8_t* valid_dev = nullptr;
  if (valid_host && n_rows > 0) {
    CK(cudaMalloc(&valid_dev, n_rows));
    CK(cudaMemcpyAsync(valid_dev, valid_host, n_rows, cudaMemcpyHostToDevice, h->stream));
  }
  if (rowid_host && n_rows > 0) {
    CK(cudaMalloc(&h->rowid, sizeof(int64_t) * n_rows));
    CK(cudaMemcpyAsync(h->rowid, rowid_host, sizeof(int64_t) * n_rows, cudaMemcpyHostToDevice, h->stream));
  }
  if (movie_idx_host && n_rows > 0) {
    CK(cudaMalloc(&h->movie_idx, sizeof(int32_t) * n_rows));
    CK(cudaMemcpyAsync(h->movie_idx, movie_idx_host, sizeof(int32_t) * n_rows, cudaMemcpyHostToDevice, h->stream));
  }
  rc = finish_embeddings(h, valid_dev);
  if (valid_dev) cudaFree(valid_dev);
  return rc;
}

int rse_attach_embeddings_dev(rse_index* h, const float* emb_dev, int64_t n_rows, int32_t dim,
                              const uint8_t* valid_dev, const int64_t* rowid_dev, const int32_t* movie_idx_dev,
                              int64_t pos_base) {
  int rc = check_emb_args(h, emb_dev, n_rows, dim, pos_base);
  if (rc != RSE_OK) return rc;
  if ((reinterpret_cast<uintptr_t>(emb_dev) & 15u) != 0)
    return fail(h, RSE_ERR_INVALID, "rse_attach_embeddings_dev: emb_dev must be 16-byte aligned");
  CK(cudaSetDevice(h->device));
  release_embeddings(h);
  h->emb = emb_dev;
  h->n_rows = n_rows; h->dim = dim; h->pos_base = static_cast<uint64_t>(pos_base);
  if (rowid_dev && n_rows > 0) {
    CK(cudaMalloc(&h->rowid, sizeof(int64_t) * n_rows));
    CK(cudaMemcpyAsync(h->rowid, rowid_dev, sizeof(int64_t) * n_rows, cudaMemcpyDeviceToDevice, h->stream));
  }
  if (movie_idx_dev && n_rows > 0) {
    CK(cudaMalloc(&h->movie_idx, sizeof(int32_t) * n_rows));
    CK(cudaMemcpyAsync(h->movie_idx, movie_idx_dev, sizeof(int32_t) * n_rows, cudaMemcpyDeviceToDevice, h->stream));
  }
  return finish_embeddings(h, valid_dev);
}

int rse_knn_local_dev(rse_index* h, const float* q_dev, int32_t nq, int32_t kprime, int64_t* cand_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!q_dev || !cand_dev || nq < 0) return fail(h, RSE_ERR_INVALID, "rse_knn_local_dev: bad arguments");
  CK(cudaSetDevice(h->device));
  h->last_flags_n = 0;
  if (!h->defer_flags_dev) return knn_local(h, q_dev, nq, kprime, reinterpret_cast<long long*>(cand_dev));
  PendingKnn pend;
  int rc = knn_local_begin(h, q_dev, nq, kprime, reinterpret_cast<long long*>(cand_dev), h->pin_status, nullptr, pend);
  if (rc != RSE_OK) return rc;
  if (pend.flags) h->last_flags_n = nq;  // tensor-core path: the flags are in tc_status; nobody waits for them here
  return RSE_OK;
}

int rse_set_defer_flags(rse_index* h, int32_t enabled) {
  if (!h) return RSE_ERR_INVALID;
  h->defer_flags_dev = enabled != 0;
  return RSE_OK;
}

int rse_knn_flags_dev(rse_index* h, int32_t* flagged_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!flagged_dev) return fail(h, RSE_ERR_INVALID, "rse_knn_flags_dev: flagged_dev is NULL");
  if (h->last_flags_n <= 0) return RSE_OK;
  CK(cudaSetDevice(h->device));
  knn_flag_count_kernel<<<1, 256, 0, h->stream>>>(static_cast<const int*>(h->tc_status.p), h->last_flags_n, flagged_dev);
  LAUNCHED(h);
  return RSE_OK;
}

int rse_knn(rse_index* h, const float* q_host, int32_t nq, int32_t kprime, float* out_dist, int64_t* out_pos,
            int64_t* out_rowid, int32_t* out_movie_idx, int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  if (nq < 0 || (nq > 0 && (!q_host || !out_dist || !out_count)))
    return fail(h, RSE_ERR_INVALID, "rse_knn: bad arguments");
  if (!h->emb) return fail(h, RSE_ERR_STATE, "rse_knn: no embeddings loaded");
  if (nq == 0) return RSE_OK;
  CK(cudaSetDevice(h->device));
  if (h->timing) CK(cudaEventRecord(h->ev[2], h->stream));
  int rc = upload_queries(h, q_host, nq);
  if (rc != RSE_OK) return rc;
  const size_t n = static_cast<size_t>(nq) * kprime;
  ENSURE(h->cand, sizeof(long long) * n * 3);
  ENSURE(h->o_dist, sizeof(float) * n);
  ENSURE(h->o_pos, sizeof(long long) * n);
  ENSURE(h->o_rowid, sizeof(long long) * n);
  ENSURE(h->o_movie, sizeof(int) * n);
  ENSURE(h->o_count, sizeof(int) * nq);
  rc = knn_local(h, static_cast<const float*>(h->staged.q.p), nq, kprime, static_cast<long long*>(h->cand.p));
  if (rc != RSE_OK) return rc;
  knn_unpack_kernel<<<nq, 128, 0, h->stream>>>(static_cast<const long long*>(h->cand.p), nq, kprime,
                                               static_cast<float*>(h->o_dist.p), static_cast<long long*>(h->o_pos.p),
                                               static_cast<long long*>(h->o_rowid.p), static_cast<int*>(h->o_movie.p),
                                               static_cast<int*>(h->o_count.p));
  LAUNCHED(h);
  CK(cudaMemcpyAsync(out_dist, h->o_dist.p, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
  if (out_pos) CK(cudaMemcpyAsync(out_pos, h->o_pos.p, sizeof(long long) * n, cudaMemcpyDeviceToHost, h->stream));
  if (out_rowid) CK(cudaMemcpyAsync(out_rowid, h->o_rowid.p, sizeof(long long) * n, cudaMemcpyDeviceToHost, h->stream));
  if (out_movie_idx) CK(cudaMemcpyAsync(out_movie_idx, h->o_movie.p, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_count, h->o_count.p, sizeof(int) * nq, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(n) * 16 + static_cast<int64_t>(nq) * 4;
  if (h->timing) CK(cudaEventRecord(h->ev[3], h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (h->timing) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]));
    h->stats.last_knn_total_ms = ms;
  }
  return RSE_OK;
}

int rse_knn_movies(rse_index* h, const float* q_host, int32_t nq, int32_t k, int32_t kprime, float* out_dist,
                   int64_t* out_chunk_rowid, int32_t* out_movie_idx, int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  if (nq < 0 || k < 1 || (nq > 0 && (!q_host || !out_dist || !out_chunk_rowid || !out_movie_idx || !out_count)))
    return fail(h, RSE_ERR_INVALID, "rse_knn_movies: bad arguments");
  if (!h->emb) return fail(h, RSE_ERR_STATE, "rse_knn_movies: no embeddings loaded");
  if (!h->movie_idx) return fail(h, RSE_ERR_STATE, "rse_knn_movies: embeddings were loaded without movie_idx");
  if (nq == 0) return RSE_OK;
  CK(cudaSetDevice(h->device));
  if (h->timing) CK(cudaEventRecord(h->ev[2], h->stream));
  int rc = upload_queries(h, q_host, nq);
  if (rc != RSE_OK) return rc;
  const size_t n = static_cast<size_t>(nq) * k;
  ENSURE(h->cand, sizeof(long long) * static_cast<size_t>(nq) * kprime * 3);
  ENSURE(h->o_dist, sizeof(float) * n);
  ENSURE(h->o_rowid, sizeof(long long) * n);
  ENSURE(h->o_movie, sizeof(int) * n);
  ENSURE(h->o_count, sizeof(int) * nq);
  rc = knn_local(h, static_cast<const float*>(h->staged.q.p), nq, kprime, static_cast<long long*>(h->cand.p));
  if (rc != RSE_OK) return rc;
  rc = aggregate(h, static_cast<const long long*>(h->cand.p), nq, k, kprime, static_cast<float*>(h->o_dist.p),
                 static_cast<long long*>(h->o_rowid.p), static_cast<int*>(h->o_movie.p),
                 static_cast<int*>(h->o_count.p));
  if (rc != RSE_OK) return rc;
  CK(cudaMemcpyAsync(out_dist, h->o_dist.p, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_chunk_rowid, h->o_rowid.p, sizeof(long long) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_movie_idx, h->o_movie.p, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_count, h->o_count.p, sizeof(int) * nq, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(n) * 16 + static_cast<int64_t>(nq) * 4;
  if (h->timing) CK(cudaEventRecord(h->ev[3], h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (h->timing) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]));
    h->stats.last_knn_total_ms = ms;
  }
  return RSE_OK;
}

int rse_knn_movies_exact(rse_index* h, const float* q_host, int32_t nq, int32_t k, float* out_dist,
                         int64_t* out_chunk_rowid, int32_t* out_movie_idx, int32_t* out_count, int32_t* out_scanned) {
  if (!h) return RSE_ERR_INVALID;
  if (nq < 0 || k < 1 || (nq > 0 && (!q_host || !out_dist || !out_chunk_rowid || !out_movie_idx || !out_count)))
    return fail(h, RSE_ERR_INVALID, "rse_knn_movies_exact: bad arguments");
  if (k > RSE_MAX_KPRIME) return fail(h, RSE_ERR_UNSUPPORTED, "rse_knn_movies_exact: k must be in [1, 4096]");
  if (!h->emb) return fail(h, RSE_ERR_STATE, "rse_knn_movies_exact: no embeddings loaded");
  if (!h->movie_idx) return fail(h, RSE_ERR_STATE, "rse_knn_movies_exact: embeddings were loaded without movie_idx");
  if (out_scanned) *out_scanned = 0;
  if (nq == 0) return RSE_OK;
  CK(cudaSetDevice(h->device));
  if (h->timing) CK(cudaEventRecord(h->ev[2], h->stream));
  int rc = upload_queries(h, q_host, nq);
  if (rc != RSE_OK) return rc;
  rc = movies_layout(h);
  if (rc != RSE_OK) return rc;
  const size_t n = static_cast<size_t>(nq) * k;
  ENSURE(h->o_dist, sizeof(float) * n);
  ENSURE(h->o_rowid, sizeof(long long) * n);
  ENSURE(h->o_movie, sizeof(int) * n);
  ENSURE(h->o_count, sizeof(int) * nq);
  float* o_dist = static_cast<float*>(h->o_dist.p);
  long long* o_rowid = static_cast<long long*>(h->o_rowid.p);
  int* o_movie = static_cast<int*>(h->o_movie.p);
  int* o_count = static_cast<int*>(h->o_count.p);
  const float* q = static_cast<const float*>(h->staged.q.p);
  // Staging (DESIGN §11): where the tensor-core filter serves K' = kMoviesExactStageMult * k, rse_knn_movies runs
  // first; a query it gives k movies is final (prefix property), and only the short ones take the segmented scan.
  // A corpus whose fp16 shadow cannot be built (shadow_state -1) would answer the first stage with the exact scan:
  // it goes straight to the segmented scan instead
  const int kprime = kMoviesExactStageMult * k;
  int n_scan = nq;
  if (kprime <= RSE_MAX_KPRIME && h->shadow_state >= 0 && tc_eligible(h, nq, kprime)) {
    ENSURE(h->cand, sizeof(long long) * static_cast<size_t>(nq) * kprime * 3);
    rc = knn_local(h, q, nq, kprime, static_cast<long long*>(h->cand.p));
    if (rc == RSE_OK) rc = aggregate(h, static_cast<const long long*>(h->cand.p), nq, k, kprime, o_dist, o_rowid, o_movie, o_count);
    if (rc != RSE_OK) return rc;
    std::vector<int> cnt(nq), list;
    CK(cudaMemcpyAsync(cnt.data(), o_count, sizeof(int) * nq, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int i = 0; i < nq; ++i)
      if (cnt[i] < k) list.push_back(i);
    n_scan = static_cast<int>(list.size());
    if (n_scan > 0) {
      const size_t ns = static_cast<size_t>(n_scan);
      ENSURE(h->mx_list, sizeof(int) * ns);
      ENSURE(h->mx_q, sizeof(float) * ns * h->dim);
      ENSURE(h->mx_sb, sizeof(double) * ns);
      ENSURE(h->mx_dist, sizeof(float) * ns * k);
      ENSURE(h->mx_rowid, sizeof(long long) * ns * k);
      ENSURE(h->mx_movie, sizeof(int) * ns * k);
      ENSURE(h->mx_count, sizeof(int) * ns);
      CK(cudaMemcpyAsync(h->mx_list.p, list.data(), sizeof(int) * ns, cudaMemcpyHostToDevice, h->stream));
      CK(cudaStreamSynchronize(h->stream));                      // `list` is a pageable temporary
      const int* dl = static_cast<const int*>(h->mx_list.p);
      knn_gather_queries_kernel<<<n_scan, 128, 0, h->stream>>>(q, static_cast<const double*>(h->sb.p), dl, h->dim,
                                                              static_cast<float*>(h->mx_q.p), static_cast<double*>(h->mx_sb.p));
      LAUNCHED(h);
      float* s_dist = static_cast<float*>(h->mx_dist.p);
      long long* s_rowid = static_cast<long long*>(h->mx_rowid.p);
      int* s_movie = static_cast<int*>(h->mx_movie.p);
      int* s_count = static_cast<int*>(h->mx_count.p);
      rc = movies_exact_scan(h, static_cast<const float*>(h->mx_q.p), static_cast<const double*>(h->mx_sb.p), n_scan, k,
                             s_dist, s_rowid, s_movie, s_count);
      if (rc != RSE_OK) return rc;
      movies_scatter_kernel<<<n_scan, 128, 0, h->stream>>>(s_dist, s_rowid, s_movie, s_count, dl, k, o_dist, o_rowid,
                                                          o_movie, o_count);
      LAUNCHED(h);
    }
  } else {
    ENSURE(h->sb, sizeof(double) * nq);
    double* sb = static_cast<double*>(h->sb.p);
    if (h->fma) knn_query_prep_kernel<true><<<(nq + 3) / 4, 128, 0, h->stream>>>(q, nq, h->dim, sb);
    else knn_query_prep_kernel<false><<<(nq + 3) / 4, 128, 0, h->stream>>>(q, nq, h->dim, sb);
    LAUNCHED(h);
    rc = movies_exact_scan(h, q, sb, nq, k, o_dist, o_rowid, o_movie, o_count);
    if (rc != RSE_OK) return rc;
  }
  CK(cudaMemcpyAsync(out_dist, o_dist, sizeof(float) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_chunk_rowid, o_rowid, sizeof(long long) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_movie_idx, o_movie, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_count, o_count, sizeof(int) * nq, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(n) * 16 + static_cast<int64_t>(nq) * 4;
  if (h->timing) CK(cudaEventRecord(h->ev[3], h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (h->timing) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]));
    h->stats.last_knn_total_ms = ms;
  }
  if (out_scanned) *out_scanned = n_scan;
  return RSE_OK;
}

int rse_knn_merge_movies_dev(rse_index* h, const int64_t* gathered_dev, int32_t n_lists, int32_t nq, int32_t k,
                             int32_t kprime, float* out_dist_dev, int64_t* out_chunk_rowid_dev,
                             int32_t* out_movie_idx_dev, int32_t* out_count_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!gathered_dev || n_lists < 1 || nq < 0 || k < 1 || kprime < 1 || !out_dist_dev || !out_chunk_rowid_dev ||
      !out_movie_idx_dev || !out_count_dev)
    return fail(h, RSE_ERR_INVALID, "rse_knn_merge_movies_dev: bad arguments");
  if (nq == 0) return RSE_OK;
  CK(cudaSetDevice(h->device));
  int rc = merge_candidates(h, reinterpret_cast<const long long*>(gathered_dev), n_lists, nq, kprime);
  if (rc != RSE_OK) return rc;
  return aggregate(h, static_cast<const long long*>(h->cand.p), nq, k, kprime, out_dist_dev,
                   reinterpret_cast<long long*>(out_chunk_rowid_dev), out_movie_idx_dev, out_count_dev);
}

// ------------------------------------------------------------------ BM25
int rse_load_bm25(rse_index* h, const int64_t* indptr, const uint32_t* doc_idx, const uint32_t* tf, const int64_t* df,
                  int64_t n_terms, int64_t n_postings, const uint32_t* dl, int64_t n_docs, int64_t n_movies,
                  double avgdl) {
  if (!h) return RSE_ERR_INVALID;
  if (n_terms < 0 || n_postings < 0 || n_docs < 0 || !indptr || (n_postings > 0 && (!doc_idx || !tf)) ||
      (n_terms > 0 && !df) || (n_docs > 0 && !dl))
    return fail(h, RSE_ERR_INVALID, "rse_load_bm25: bad arguments");
  if (n_docs >= 0xFFFFFFFFll || n_postings >= (1ll << 40))
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_load_bm25: index too large");
  if (indptr[0] != 0 || indptr[n_terms] != n_postings)
    return fail(h, RSE_ERR_INVALID, "rse_load_bm25: indptr must start at 0 and end at n_postings");
  CK(cudaSetDevice(h->device));
  release_bm25(h);
  h->n_terms = n_terms; h->n_postings = n_postings; h->n_docs = n_docs; h->n_movies = n_movies; h->avgdl = avgdl;
  h->nr = static_cast<int>((n_docs + kBmRange - 1) / kBmRange);
  if (h->nr < 1) h->nr = 1;
  if (h->nr > 2048) return fail(h, RSE_ERR_UNSUPPORTED, "rse_load_bm25: more than 14,680,064 documents (2048 ranges of 7168)");
  h->df_host.assign(df, df + n_terms);

  CK(cudaMalloc(&h->indptr, sizeof(int64_t) * (n_terms + 1)));
  CK(cudaMemcpyAsync(h->indptr, indptr, sizeof(int64_t) * (n_terms + 1), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMalloc(&h->post, sizeof(uint2) * std::max<int64_t>(n_postings, 1)));
  if (n_postings > 0) {
    // strided 2D copies interleave (doc, tf) into uint2 without a host temporary
    CK(cudaMemcpy2DAsync(reinterpret_cast<char*>(h->post), sizeof(uint2), doc_idx, sizeof(uint32_t), sizeof(uint32_t),
                         n_postings, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpy2DAsync(reinterpret_cast<char*>(h->post) + 4, sizeof(uint2), tf, sizeof(uint32_t), sizeof(uint32_t),
                         n_postings, cudaMemcpyHostToDevice, h->stream));
  }
  CK(cudaMalloc(&h->dl, sizeof(uint32_t) * std::max<int64_t>(n_docs, 1)));
  if (n_docs > 0) CK(cudaMemcpyAsync(h->dl, dl, sizeof(uint32_t) * n_docs, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMalloc(&h->normk, sizeof(double) * std::max<int64_t>(n_docs, 1)));
  const int64_t roff_n = std::max<int64_t>(n_terms, 1) * (h->nr + 1);
  CK(cudaMalloc(&h->roff, sizeof(uint32_t) * roff_n));
  if (n_terms > 0) {
    const int threads = 256;
    const int64_t total = n_terms * (h->nr + 1);
    const int64_t grid = (total + threads - 1) / threads;
    if (grid > 0x7FFFFFFFll) return fail(h, RSE_ERR_UNSUPPORTED, "rse_load_bm25: range table too large");
    bm25_range_offsets_by_term_kernel<<<static_cast<unsigned int>(grid), threads, 0, h->stream>>>(
        h->indptr, h->post, n_terms, h->nr, h->roff);
    LAUNCHED(h);
  }
  CK(cudaStreamSynchronize(h->stream));
  h->stats.bm25_postings = n_postings;
  h->stats.bm25_docs = n_docs;
  if (!(h->attr_mask & (1u << 14))) {
    CK(cudaFuncSetAttribute(bm25_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBmRange * 9));
    CK(cudaFuncSetAttribute(bm25_deep_score_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kBmRange * 9));
    CK(cudaFuncSetAttribute(bm25_stream_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bs_smem_bytes()));
    CK(cudaFuncSetAttribute(bm25_fx_kernel<kBsThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, fx_smem_bytes(kBsMaxRpg)));
    CK(cudaFuncSetAttribute(bm25_fx_kernel<kBsThreads>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    CK(cudaFuncSetAttribute(bm25_fx_kernel<kBsWideThreads>, cudaFuncAttributeMaxDynamicSharedMemorySize, fx_smem_bytes(kBsMaxRpg)));
    CK(cudaFuncSetAttribute(bm25_fx_kernel<kBsWideThreads>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    h->attr_mask |= 1u << 14;
  }
  return RSE_OK;
}

namespace {

// tokens → device, with host-computed idf (keyword_search.py:224, same libm `log` as CPython).
int bm25_stage(rse_index* h, Batch& in, const int32_t* tok_indptr, const int32_t* term_rows, int nq,
               cudaStream_t s) {
  if (!h->indptr) return fail(h, RSE_ERR_STATE, "rse_bm25: no BM25 index loaded");
  const int64_t ntok = tok_indptr[nq];
  if (tok_indptr[0] != 0 || ntok < 0) return fail(h, RSE_ERR_INVALID, "rse_bm25: bad tok_indptr");
  // The token table goes through a pinned staging buffer owned by the handle, so the three uploads are truly
  // asynchronous (a pageable source makes cudaMemcpyAsync synchronise the stream first).  Every entry point that
  // stages ends in a stream synchronisation before it returns (fetch / result copy), so the buffer is free again
  // by the next call; a stage-only caller (rse_hybrid_stage) is covered by the synchronisation below.
  const size_t nt = static_cast<size_t>(std::max<int64_t>(ntok, 1));
  const size_t bytes_idf = sizeof(double) * nt, bytes_terms = sizeof(int32_t) * nt, bytes_ptr = sizeof(int32_t) * (nq + 1);
  const size_t need = bytes_idf + ((bytes_terms + 7) & ~size_t(7)) + bytes_ptr;
  if (!h->ev_stage) CK(cudaEventCreateWithFlags(&h->ev_stage, cudaEventDisableTiming));
  else CK(cudaEventSynchronize(h->ev_stage));               // the previous batch's uploads are out of the buffer
  if (h->pin_stage_bytes < need) {
    CK(cudaStreamSynchronize(s));
    if (h->pin_stage) CK(cudaFreeHost(h->pin_stage));
    h->pin_stage = nullptr; h->pin_stage_bytes = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&h->pin_stage), need + need / 2 + 4096));
    h->pin_stage_bytes = need + need / 2 + 4096;
  }
  double* idf = reinterpret_cast<double*>(h->pin_stage);
  int32_t* terms = reinterpret_cast<int32_t*>(h->pin_stage + bytes_idf);
  int32_t* ptr = reinterpret_cast<int32_t*>(h->pin_stage + bytes_idf + ((bytes_terms + 7) & ~size_t(7)));
  for (size_t i = 0; i < nt; ++i) { idf[i] = 0.0; terms[i] = -1; }
  const bool dead = (h->n_docs == 0) || !(h->avgdl != 0.0);   // avgdl None/0 → [] (:199-200)
  for (int q = 0; q < nq; ++q) {
    const int n = tok_indptr[q + 1] - tok_indptr[q];
    if (n < 0) return fail(h, RSE_ERR_INVALID, "rse_bm25: tok_indptr not monotone");
    if (n > RSE_MAX_QUERY_TOKENS) return fail(h, RSE_ERR_UNSUPPORTED, "rse_bm25: more than 255 tokens in a query");
    for (int t = tok_indptr[q]; t < tok_indptr[q + 1]; ++t) {
      const int32_t term = term_rows[t];
      if (term >= h->n_terms) return fail(h, RSE_ERR_INVALID, "rse_bm25: term row out of range");
      if (term < 0 || dead) continue;
      const int64_t df = h->df_host[term];
      if (df <= 0) continue;                                   // `if not rows: continue` (:219-220)
      terms[t] = term;
      const double N = static_cast<double>(h->n_movies - df);  // int arithmetic first, as Python does
      idf[t] = std::log((N + 0.5) / (static_cast<double>(df) + 0.5) + 1.0);
    }
  }
  std::memcpy(ptr, tok_indptr, bytes_ptr);
  ENSURE(in.tokptr, sizeof(int32_t) * (nq + 1));
  ENSURE(in.terms, sizeof(int32_t) * std::max<int64_t>(ntok, 1));
  ENSURE(in.idf, sizeof(double) * std::max<int64_t>(ntok, 1));
  CK(cudaMemcpyAsync(in.tokptr.p, ptr, bytes_ptr, cudaMemcpyHostToDevice, s));
  if (ntok > 0) {
    CK(cudaMemcpyAsync(in.terms.p, terms, sizeof(int32_t) * ntok, cudaMemcpyHostToDevice, s));
    CK(cudaMemcpyAsync(in.idf.p, idf, sizeof(double) * ntok, cudaMemcpyHostToDevice, s));
  }
  CK(cudaEventRecord(h->ev_stage, s));
  h->stats.h2d_bytes += static_cast<int64_t>(bytes_ptr) + (ntok > 0 ? static_cast<int64_t>(ntok) * 12 : 0);
  return RSE_OK;
}

// scoring + top-k on the first nq queries of the staged tokens, on stream s; results stay on the device in
// h->b_score / b_doc / b_count ([nq][k]).  under_filter: the batch shares the SMs with the tensor-core filter pass.
int bm25_run(rse_index* h, const Batch& in, int nq, int k, double k1, double b, cudaStream_t s, bool under_filter) {
  if (!h->indptr) return fail(h, RSE_ERR_STATE, "rse_bm25: no BM25 index loaded");
  if (k < 1 || k > RSE_MAX_BM25_K) return fail(h, RSE_ERR_UNSUPPORTED, "rse_bm25: k must be in [1, 512]");
  ENSURE(h->b_score, sizeof(double) * static_cast<size_t>(nq) * k);
  ENSURE(h->b_doc, sizeof(int) * static_cast<size_t>(nq) * k);
  ENSURE(h->b_count, sizeof(int) * nq);
  if (!(h->normk_k1 == k1 && h->normk_b == b) && h->n_docs > 0) {
    const int threads = 256;
    bm25_norm_kernel<<<static_cast<unsigned int>((h->n_docs + threads - 1) / threads), threads, 0, s>>>(
        h->dl, h->n_docs, k1, b, h->avgdl, h->normk);
    LAUNCHED(h);
    h->normk_k1 = k1; h->normk_b = b;
  }
  // Queries per launch.  Above kBmGeneralMaxK the per-range candidate lists (16 B per candidate, nr * k per query:
  // 688 KB at k = 512 over the 84 ranges of 600 k documents, 16 MB over 2048 ranges) are held within 256 MB by
  // scoring the batch in chunks: 390 queries at k = 512 on 600 k documents, so a 256-query batch is one launch.
  constexpr size_t kDeepCandBudget = size_t(256) << 20;
  const bool deep = k > kBmGeneralMaxK;
  const int chunk = deep ? static_cast<int>(std::max<size_t>(1, std::min<size_t>(4096, kDeepCandBudget /
                                                             (static_cast<size_t>(h->nr) * k * 16))))
                         : 4096;
  const size_t per_q = static_cast<size_t>(h->nr) * k;
  ENSURE(h->b_chi, sizeof(unsigned long long) * per_q * std::min(nq, chunk));
  ENSURE(h->b_clo, sizeof(unsigned long long) * per_q * std::min(nq, chunk));
  ENSURE(h->b_ccnt, sizeof(int) * static_cast<size_t>(h->nr) * std::min(nq, chunk));
  const double k1p1 = k1 + 1.0;
  const int32_t* tokptr = static_cast<const int32_t*>(in.tokptr.p);
  const int32_t* terms = static_cast<const int32_t*>(in.terms.p);
  const double* idf = static_cast<const double*>(in.idf.p);

  // streaming path (bm25_stream_kernel): k <= 32; needs the weighted postings of this (k1, b)
  const bool stream = k <= 32 && h->n_postings > 0 && h->bm25_mode != 2;
  // the 4-byte posting stream of the fixed-point kernel: wq4_scale = largest power of two with
  // (k1 + 1) * wq4_scale <= 2^19; 0 = no stream (0 < w <= k1 + 1 needs normk >= 0)
  double wq4_scale = 0.0;
  if (k1 >= 0.0 && b >= 0.0 && b <= 1.0 && k1p1 < 1048576.0) {
    int e = 0;
    const double m = std::frexp(k1p1, &e);                 // k1p1 = m * 2^e, 0.5 <= m < 1
    wq4_scale = std::ldexp(1.0, m == 0.5 ? 20 - e : 19 - e);
  }
  // fixed-point sums must stay below 2^31: idf <= log(N + 2), w < k1 + 1, <= 16 tokens; the scale is the largest
  // power of two that allows (2^21 for the default k1), and the path needs at least 2^12 and the 4-byte stream (a
  // scale of 2^12 bounds k1 + 1 below 2^15 / ln 2 < 2^20, so the stream always exists when the scale does)
  double fx_scale = 0.0;
  if (stream && h->bm25_mode == 0 && wq4_scale > 0.0) {
    const double max_sum = (k1 + 1.0) * std::log(static_cast<double>(h->n_movies) + 2.0) * 16.0 + 1.0;
    int e = 0;
    std::frexp(max_sum, &e);                               // max_sum < 2^e
    if (31 - e >= 12) fx_scale = std::ldexp(1.0, 31 - e);
  }
  const bool fx = fx_scale > 0.0;
  int ng = 1, rpg = h->nr;
  if (stream) {
    if (!(h->w_k1 == k1 && h->w_b == b)) {
      if (!h->post16) CK(cudaMalloc(&h->post16, sizeof(Post16) * static_cast<size_t>(h->n_postings)));
      if (wq4_scale > 0.0 && !h->post4) CK(cudaMalloc(&h->post4, sizeof(uint32_t) * (static_cast<size_t>(h->n_postings) + 8)));
      const int threads = 256;
      bm25_weight_kernel<<<static_cast<unsigned int>((h->n_postings + threads - 1) / threads), threads, 0, s>>>(
          h->post, h->normk, h->n_postings, k1p1, h->post16, wq4_scale > 0.0 ? h->post4 : nullptr, wq4_scale);
      LAUNCHED(h);
      h->w_k1 = k1; h->w_b = b;
    }
    // one CTA per (query, group of consecutive ranges), 3 CTAs per SM: at least ~4 waves, and among the next
    // few group counts the one whose last wave is fullest (256 queries x 4 groups was 2.3 waves: a third of
    // the kernel ran at 30 % occupancy)
    {
      const int nqc = std::min(nq, chunk);
      const double conc = (fx ? 4.0 : 3.0) * h->sm_count;   // resident CTAs: the fixed-point kernel fits 4 per SM
      const int g_lo = std::max(1, static_cast<int>((4.0 * conc + nqc - 1) / nqc));
      double best_eff = -1.0;
      for (int cand = g_lo; cand <= g_lo + 10; ++cand) {
        int c_rpg = (h->nr + std::min(cand, h->nr) - 1) / std::min(cand, h->nr);
        if (c_rpg > kBsMaxRpg) c_rpg = kBsMaxRpg;
        const int c_ng = (h->nr + c_rpg - 1) / c_rpg;
        if (fx && c_ng > kBsMaxGroups && best_eff >= 0.0) continue;
        const double waves = nqc * static_cast<double>(c_ng) / conc;
        const double eff = waves / std::ceil(waves);
        if (eff > best_eff + 1e-9) { best_eff = eff; ng = c_ng; rpg = c_rpg; }
      }
    }
    if (fx && ng > kBsMaxGroups) { rpg = (h->nr + kBsMaxGroups - 1) / kBsMaxGroups; ng = (h->nr + rpg - 1) / rpg; }
    const size_t per_qs = static_cast<size_t>(ng) * std::max(k, 2 * kFxFinalCap);
    ENSURE(h->b_shi, sizeof(unsigned long long) * per_qs * std::min(nq, chunk));
    ENSURE(h->b_slo, sizeof(unsigned long long) * per_qs * std::min(nq, chunk));
    ENSURE(h->b_scnt, sizeof(int) * static_cast<size_t>(ng) * std::min(nq, chunk));
    ENSURE(h->b_status, sizeof(int) * nq);
    ENSURE(h->b_flagged, sizeof(int) * (std::min(nq, chunk) + 1));
    CK(cudaMemsetAsync(h->b_status.p, 0, sizeof(int) * nq, s));
  }
  h->stats.bm25_queries += nq;
  for (int q0 = 0; q0 < nq; q0 += chunk) {
    const int nc = std::min(chunk, nq - q0);
    // candidate buffers are indexed by absolute q inside the kernels → offset the base pointers
    unsigned long long* chi = static_cast<unsigned long long*>(h->b_chi.p) - static_cast<int64_t>(q0) * per_q;
    unsigned long long* clo = static_cast<unsigned long long*>(h->b_clo.p) - static_cast<int64_t>(q0) * per_q;
    int* ccnt = static_cast<int*>(h->b_ccnt.p) - static_cast<int64_t>(q0) * h->nr;
    unsigned long long* shi = nullptr;
    unsigned long long* slo = nullptr;
    int* scnt = nullptr;
    int* status = nullptr;
    if (fx) {
      uint2* fin = static_cast<uint2*>(h->b_shi.p) - static_cast<int64_t>(q0) * ng * kFxFinalCap;
      int* fcnt = static_cast<int*>(h->b_scnt.p) - static_cast<int64_t>(q0) * ng;
      status = static_cast<int*>(h->b_status.p);
      const double idfx_scale = fx_scale / wq4_scale;
      // underneath the tensor-core filter (hybrid step, second stream): wide CTAs (bm25.cuh: 28 warps beside the
      // filter's CTA).  Alone the 512-thread shape is the faster one (4 CTAs per SM: 284 against 318 us).  Splitting
      // the groups between the two shapes loses (r02, 25 / 40 / 60 / 100 % wide -> 1.064 / 1.071 / 1.087 / 1.050 ms
      // per step): a second launch waits for the first.
      const int threads = under_filter ? kBsWideThreads : kBsThreads;
      const auto kernel = under_filter ? bm25_fx_kernel<kBsWideThreads> : bm25_fx_kernel<kBsThreads>;
      kernel<<<dim3(nc, ng), threads, fx_smem_bytes(rpg), s>>>(h->indptr, h->post4, h->roff, h->nr, tokptr, terms, idf,
                                                               idfx_scale, q0, k, rpg, ng, fin, fcnt, status);
      LAUNCHED(h);
      bm25_fx_finish_kernel<<<nc, kBmThreads, 0, s>>>(
          fin, fcnt, ng, status, h->indptr, h->post16, h->roff, h->nr, tokptr, terms, idf, q0, k,
          static_cast<double*>(h->b_score.p), static_cast<int*>(h->b_doc.p), static_cast<int*>(h->b_count.p),
          h->dev_counters, idfx_scale);
      LAUNCHED(h);
    } else if (stream) {
      // bm25_stream_kernel and bm25_merge_kernel index these lists as [q][ng][k]: offset by that stride (the buffers
      // are sized for the larger fixed-point lists)
      const int64_t per_qs = static_cast<int64_t>(ng) * k;
      shi = static_cast<unsigned long long*>(h->b_shi.p) - static_cast<int64_t>(q0) * per_qs;
      slo = static_cast<unsigned long long*>(h->b_slo.p) - static_cast<int64_t>(q0) * per_qs;
      scnt = static_cast<int*>(h->b_scnt.p) - static_cast<int64_t>(q0) * ng;
      status = static_cast<int*>(h->b_status.p);
      dim3 sgrid(ng, nc);
      bm25_stream_kernel<<<sgrid, kBsThreads, bs_smem_bytes(), s>>>(h->indptr, h->post16, h->roff, h->nr, tokptr, terms,
                                                                    idf, q0, k, rpg, ng, shi, slo, scnt, status);
      LAUNCHED(h);
    }
    // general kernel: every query when the streaming path does not apply, else only the flagged ones
    // (compacted on the device; the launch is then a small grid that usually finds an empty list)
    int* flagged = nullptr;
    if (stream) {
      flagged = static_cast<int*>(h->b_flagged.p);
      bm25_flag_compact_kernel<<<1, 256, 0, s>>>(status, q0, nc, flagged, h->dev_counters);
      LAUNCHED(h);
    }
    dim3 grid(h->nr, stream ? std::min(nc, 16) : nc);
    if (deep)
      bm25_deep_score_kernel<<<grid, kBmThreads, kBmRange * 9, s>>>(
          h->indptr, h->post, h->roff, h->normk, h->nr, h->n_docs, tokptr, terms, idf, q0, k, k1p1, chi, clo, ccnt);
    else
      bm25_score_kernel<<<grid, kBmThreads, kBmRange * 9, s>>>(
          h->indptr, h->post, h->roff, h->normk, h->nr, h->n_docs, tokptr, terms, idf, q0, k, k1p1, chi, clo, ccnt,
          flagged);
    LAUNCHED(h);
    bm25_merge_kernel<<<nc, kBmThreads, 0, s>>>(chi, clo, ccnt, h->nr, q0, k, static_cast<double*>(h->b_score.p),
                                                static_cast<int*>(h->b_doc.p), static_cast<int*>(h->b_count.p), shi, slo,
                                                scnt, ng, status);
    LAUNCHED(h);
  }
  return RSE_OK;
}

int bm25_device(rse_index* h, const int32_t* tok_indptr, const int32_t* term_rows, int nq, int k, double k1, double b) {
  if (k < 1 || k > RSE_MAX_BM25_K) return fail(h, RSE_ERR_UNSUPPORTED, "rse_bm25: k must be in [1, 512]");
  int rc = bm25_stage(h, h->staged, tok_indptr, term_rows, nq, h->stream);
  if (rc != RSE_OK) return rc;
  return bm25_run(h, h->staged, nq, k, k1, b, h->stream, false);
}

}  // namespace

int rse_bm25(rse_index* h, const int32_t* tok_indptr, const int32_t* term_rows, int32_t nq, int32_t k, double k1,
             double b, double* out_score, int32_t* out_doc_idx, int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  if (nq < 0 || !tok_indptr || (nq > 0 && (!out_score || !out_doc_idx || !out_count)))
    return fail(h, RSE_ERR_INVALID, "rse_bm25: bad arguments");
  if (nq == 0) return RSE_OK;
  if (tok_indptr[nq] > 0 && !term_rows) return fail(h, RSE_ERR_INVALID, "rse_bm25: term_rows is NULL");
  CK(cudaSetDevice(h->device));
  if (h->timing) CK(cudaEventRecord(h->ev[2], h->stream));
  int rc = bm25_device(h, tok_indptr, term_rows, nq, k, k1, b);
  if (rc != RSE_OK) return rc;
  const size_t n = static_cast<size_t>(nq) * k;
  CK(cudaMemcpyAsync(out_score, h->b_score.p, sizeof(double) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_doc_idx, h->b_doc.p, sizeof(int) * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_count, h->b_count.p, sizeof(int) * nq, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(n) * 12 + static_cast<int64_t>(nq) * 4;
  if (h->timing) CK(cudaEventRecord(h->ev[3], h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (h->timing) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]));
    h->stats.last_bm25_ms = ms;
  }
  return RSE_OK;
}

// ------------------------------------------------------------------ fusion
namespace {

// inputs [nq, limit]; outputs [nq, out_w] (fuse_kernel: limit <= out_w <= 2 * limit)
int fuse_launch(rse_index* h, int mode, double param, int tie_mode, int nq, int limit, int out_w, const FuseIn& in,
                long long* o_id, double* o_sc, double* o_a, double* o_b, int* o_cnt) {
  if (limit < 1 || limit > RSE_MAX_FUSE_LIMIT) return fail(h, RSE_ERR_UNSUPPORTED, "fusion: limit must be in [1, 1024]");
  if (tie_mode != RSE_TIE_REFERENCE && tie_mode != RSE_TIE_BY_ID) return fail(h, RSE_ERR_INVALID, "fusion: bad tie_mode");
  if (limit > kFuseMaxLimit) {
    if (!(h->attr_mask & (1u << 16))) {
      CK(cudaFuncSetAttribute(fuse_kernel<kFuseDeepLimit>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                              static_cast<int>(fuse_deep_smem_bytes(kFuseDeepLimit))));
      h->attr_mask |= 1u << 16;
    }
    fuse_kernel<kFuseDeepLimit><<<nq, kFuseDeepThreads, fuse_deep_smem_bytes(limit), h->stream>>>(
        in, nq, limit, out_w, mode, param, tie_mode, o_id, o_sc, o_a, o_b, o_cnt);
    LAUNCHED(h);
    return RSE_OK;
  }
  const size_t smem = fuse_smem_bytes(limit);
  if (smem > 48 * 1024 && !(h->attr_mask & (1u << 15))) {     // per handle: the attribute is per device (ADVICE r01)
    CK(cudaFuncSetAttribute(fuse_kernel<kFuseMaxLimit>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            static_cast<int>(fuse_smem_bytes(kFuseMaxLimit))));
    h->attr_mask |= 1u << 15;
  }
  fuse_kernel<kFuseMaxLimit><<<nq, 32, smem, h->stream>>>(in, nq, limit, out_w, mode, param, tie_mode, o_id, o_sc, o_a,
                                                          o_b, o_cnt);
  LAUNCHED(h);
  return RSE_OK;
}

int fuse_host(rse_index* h, int mode, double param, int tie_mode, int nq, int limit, const int64_t* bm25_id,
              const double* bm25_score, const int32_t* bm25_count, const int64_t* sem_id, const double* sem_dist,
              const int32_t* sem_count, int64_t* out_id, double* out_score, double* out_a, double* out_b,
              int32_t* out_count) {
  if (nq < 0 || (nq > 0 && (!bm25_id || !bm25_score || !bm25_count || !sem_id || !sem_dist || !sem_count || !out_id ||
                            !out_score || !out_a || !out_b || !out_count)))
    return fail(h, RSE_ERR_INVALID, "fusion: bad arguments");
  if (nq == 0) return RSE_OK;
  if (limit < 1 || limit > RSE_MAX_FUSE_LIMIT) return fail(h, RSE_ERR_UNSUPPORTED, "fusion: limit must be in [1, 1024]");
  CK(cudaSetDevice(h->device));
  const size_t n = static_cast<size_t>(nq) * limit;
  ENSURE(h->f_bid, 8 * n); ENSURE(h->f_bsc, 8 * n); ENSURE(h->f_bcnt, 4 * static_cast<size_t>(nq));
  ENSURE(h->f_sid, 8 * n); ENSURE(h->f_sds, 8 * n); ENSURE(h->f_scnt, 4 * static_cast<size_t>(nq));
  ENSURE(h->f_oid, 8 * n); ENSURE(h->f_osc, 8 * n); ENSURE(h->f_oa, 8 * n); ENSURE(h->f_ob, 8 * n);
  ENSURE(h->f_ocnt, 4 * static_cast<size_t>(nq));
  if (h->timing) CK(cudaEventRecord(h->ev[2], h->stream));
  CK(cudaMemcpyAsync(h->f_bid.p, bm25_id, 8 * n, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->f_bsc.p, bm25_score, 8 * n, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->f_bcnt.p, bm25_count, 4 * static_cast<size_t>(nq), cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->f_sid.p, sem_id, 8 * n, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->f_sds.p, sem_dist, 8 * n, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(h->f_scnt.p, sem_count, 4 * static_cast<size_t>(nq), cudaMemcpyHostToDevice, h->stream));
  FuseIn in{static_cast<const long long*>(h->f_bid.p), static_cast<const double*>(h->f_bsc.p),
            static_cast<const int*>(h->f_bcnt.p),      static_cast<const long long*>(h->f_sid.p),
            nullptr,                                   static_cast<const int*>(h->f_scnt.p),
            static_cast<const double*>(h->f_sds.p)};
  int rc = fuse_launch(h, mode, param, tie_mode, nq, limit, limit, in, static_cast<long long*>(h->f_oid.p),
                       static_cast<double*>(h->f_osc.p), static_cast<double*>(h->f_oa.p),
                       static_cast<double*>(h->f_ob.p), static_cast<int*>(h->f_ocnt.p));
  if (rc != RSE_OK) return rc;
  CK(cudaMemcpyAsync(out_id, h->f_oid.p, 8 * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_score, h->f_osc.p, 8 * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_a, h->f_oa.p, 8 * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_b, h->f_ob.p, 8 * n, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaMemcpyAsync(out_count, h->f_ocnt.p, 4 * static_cast<size_t>(nq), cudaMemcpyDeviceToHost, h->stream));
  if (h->timing) CK(cudaEventRecord(h->ev[3], h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (h->timing) {
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, h->ev[2], h->ev[3]));
    h->stats.last_fuse_ms = ms;
  }
  return RSE_OK;
}

}  // namespace

int rse_fuse_weighted(rse_index* h, int32_t nq, int32_t limit, double alpha, int32_t tie_mode, const int64_t* bm25_id,
                      const double* bm25_score, const int32_t* bm25_count, const int64_t* sem_id, const double* sem_dist,
                      const int32_t* sem_count, int64_t* out_id, double* out_bm25, double* out_sem, double* out_score,
                      int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  return fuse_host(h, 1, alpha, tie_mode, nq, limit, bm25_id, bm25_score, bm25_count, sem_id, sem_dist, sem_count,
                   out_id, out_score, out_bm25, out_sem, out_count);
}

int rse_fuse_rrf(rse_index* h, int32_t nq, int32_t limit, double k, int32_t tie_mode, const int64_t* bm25_id,
                 const double* bm25_score, const int32_t* bm25_count, const int64_t* sem_id, const double* sem_dist,
                 const int32_t* sem_count, int64_t* out_id, double* out_score, int32_t* out_bm25_rank,
                 int32_t* out_sem_rank, int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  if (nq > 0 && (!out_bm25_rank || !out_sem_rank)) return fail(h, RSE_ERR_INVALID, "rse_fuse_rrf: bad arguments");
  const size_t n = static_cast<size_t>(std::max(nq, 0)) * std::max(limit, 0);
  std::vector<double> a(std::max<size_t>(n, 1)), b(std::max<size_t>(n, 1));
  int rc = fuse_host(h, 0, k, tie_mode, nq, limit, bm25_id, bm25_score, bm25_count, sem_id, sem_dist, sem_count, out_id,
                     out_score, a.data(), b.data(), out_count);
  if (rc != RSE_OK) return rc;
  for (size_t i = 0; i < n; ++i) {
    out_bm25_rank[i] = static_cast<int32_t>(a[i]);
    out_sem_rank[i] = static_cast<int32_t>(b[i]);
  }
  return RSE_OK;
}

// ------------------------------------------------------------------ hybrid
int rse_set_id_tables(rse_index* h, const int64_t* doc_ids, int64_t n_docs, const int64_t* movie_ids,
                      int64_t n_movie_ids) {
  if (!h) return RSE_ERR_INVALID;
  if (n_docs < 0 || n_movie_ids < 0 || (n_docs > 0 && !doc_ids) || (n_movie_ids > 0 && !movie_ids))
    return fail(h, RSE_ERR_INVALID, "rse_set_id_tables: bad arguments");
  CK(cudaSetDevice(h->device));
  free_ptr(h->doc_ids); free_ptr(h->movie_ids);
  CK(cudaMalloc(&h->doc_ids, 8 * std::max<int64_t>(n_docs, 1)));
  CK(cudaMalloc(&h->movie_ids, 8 * std::max<int64_t>(n_movie_ids, 1)));
  if (n_docs) CK(cudaMemcpyAsync(h->doc_ids, doc_ids, 8 * n_docs, cudaMemcpyHostToDevice, h->stream));
  if (n_movie_ids) CK(cudaMemcpyAsync(h->movie_ids, movie_ids, 8 * n_movie_ids, cudaMemcpyHostToDevice, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->n_doc_ids = n_docs; h->n_movie_ids = n_movie_ids;
  return RSE_OK;
}

namespace {

int check_hybrid_state(rse_index* h) {
  if (!h->emb || !h->movie_idx || !h->indptr || !h->doc_ids || !h->movie_ids)
    return fail(h, RSE_ERR_STATE, "rse_hybrid: needs embeddings (with movie_idx), a BM25 index and id tables");
  return RSE_OK;
}

// the arguments every hybrid entry point shares, and the state a step needs → K' (semantic_search.py:251), or an error
int hybrid_kprime(rse_index* h, int mode, int limit, int knn_multiplier) {
  if (mode != 0 && mode != 1) return fail(h, RSE_ERR_INVALID, "rse_hybrid: mode must be 0 (rrf) or 1 (weighted)");
  if (limit < 1 || limit > RSE_MAX_HYBRID_LIMIT) return fail(h, RSE_ERR_UNSUPPORTED, "rse_hybrid: limit must be in [1, 512]");
  if (knn_multiplier < 0) return fail(h, RSE_ERR_INVALID, "rse_hybrid: knn_multiplier < 0");
  const int kprime = std::max(limit * knn_multiplier, limit);
  if (kprime > RSE_MAX_KPRIME) return fail(h, RSE_ERR_UNSUPPORTED, "rse_hybrid: limit*knn_multiplier exceeds 4096");
  const int rc = check_hybrid_state(h);
  return rc != RSE_OK ? rc : kprime;
}

// The inputs of one hybrid batch → `in`, on stream s: the tokens through bm25_stage, then the query vectors (`kind`:
// from host or device memory).  `in` holds no batch unless this succeeds.
int stage_batch(rse_index* h, Batch& in, int nq, const float* q, cudaMemcpyKind kind, const int32_t* tok_indptr,
                const int32_t* term_rows, cudaStream_t s) {
  int rc = check_hybrid_state(h);
  if (rc != RSE_OK) return rc;
  in.nq = 0;
  if (nq == 0) return RSE_OK;
  if (tok_indptr[nq] > 0 && !term_rows) return fail(h, RSE_ERR_INVALID, "rse_hybrid_stage: term_rows is NULL");
  CK(cudaSetDevice(h->device));
  rc = bm25_stage(h, in, tok_indptr, term_rows, nq, s);
  if (rc != RSE_OK) return rc;
  const size_t bytes = sizeof(float) * static_cast<size_t>(nq) * h->dim;
  ENSURE(in.q, bytes);
  CK(cudaMemcpyAsync(in.q.p, q, bytes, kind, s));
  if (kind == cudaMemcpyHostToDevice) h->stats.h2d_bytes += static_cast<int64_t>(bytes);
  in.nq = nq;
  return RSE_OK;
}

// Where a hybrid step writes its results: [nq, w] each (w = limit is the reference's [:limit], 2 * limit the whole
// fused union the cross-encoder rerank scores).
struct Fused {
  long long* id;
  double *score, *a, *b;
  int* count;
  int w;
};

// the five result arrays back to back in one buffer, so rse_hybrid_fetch / _collect is ONE device-to-host copy into
// pinned memory (five copies into pageable caller buffers were five synchronous staging round trips)
int packed_results(rse_index* h, DevBuf& pack, int nq, int limit, Fused* out) {
  const size_t n = static_cast<size_t>(nq) * limit;
  ENSURE(pack, 32 * n + 4 * static_cast<size_t>(nq));
  char* pk = static_cast<char*>(pack.p);
  *out = Fused{reinterpret_cast<long long*>(pk), reinterpret_cast<double*>(pk + 8 * n),
               reinterpret_cast<double*>(pk + 16 * n), reinterpret_cast<double*>(pk + 24 * n),
               reinterpret_cast<int*>(pk + 32 * n), limit};
  return RSE_OK;
}

// The end of every hybrid step, for nq queries whose BM25 lists are in b_score / b_doc / b_count: [merge of the
// n_lists gathered shard lists into h->cand →] per-movie aggregation of the KNN candidates in h->cand → join of BM25
// on the second stream (join_bm25) → fusion.
int hybrid_tail(rse_index* h, int mode, double param, int tie_mode, int nq, int limit, int kprime,
                const long long* gathered, int n_lists, bool join_bm25, const Fused& out) {
  const size_t n = static_cast<size_t>(nq) * limit;
  ENSURE(h->o_dist, sizeof(float) * n);
  ENSURE(h->o_rowid, sizeof(long long) * n);
  ENSURE(h->o_movie, sizeof(int) * n);
  ENSURE(h->o_count, sizeof(int) * nq);
  int rc = gathered ? merge_candidates(h, gathered, n_lists, nq, kprime) : RSE_OK;
  if (rc != RSE_OK) return rc;
  rc = aggregate(h, static_cast<const long long*>(h->cand.p), nq, limit, kprime, static_cast<float*>(h->o_dist.p),
                 static_cast<long long*>(h->o_rowid.p), static_cast<int*>(h->o_movie.p), static_cast<int*>(h->o_count.p));
  if (rc != RSE_OK) return rc;
  // the per-movie aggregation needs the KNN candidates only: BM25 (usually the last to finish) is joined after it
  if (join_bm25) CK(cudaStreamWaitEvent(h->stream, h->ev_bm25_done, 0));
  // dense index → movies.id happens inside the fusion kernel (two gather launches less)
  FuseIn in{nullptr, static_cast<const double*>(h->b_score.p), static_cast<const int*>(h->b_count.p), nullptr,
            static_cast<const float*>(h->o_dist.p), static_cast<const int*>(h->o_count.p), nullptr};
  in.bm25_idx = static_cast<const int*>(h->b_doc.p); in.bm25_table = h->doc_ids; in.bm25_table_n = h->n_doc_ids;
  in.sem_idx = static_cast<const int*>(h->o_movie.p); in.sem_table = h->movie_ids; in.sem_table_n = h->n_movie_ids;
  rc = fuse_launch(h, mode, param, tie_mode, nq, limit, out.w, in, out.id, out.score, out.a, out.b, out.count);
  tl_mark(h, kTlStepEnd, h->stream);
  return rc;
}

// BM25 + local KNN + aggregation + fusion on the batch `in`.  The tensor-core path's overflow flags land in `pin`;
// with `keep` the flagged queries are left to the caller (rse_hybrid_submit: collect checks them), else they are
// re-run through the exact scan before the aggregation.
int hybrid_local(rse_index* h, int mode, double param, int tie_mode, int limit, int kprime, double k1, double b,
                 const Batch& in, PinnedFlags& pin, PendingKnn* keep, const Fused& out) {
  const int nq = in.nq;
  ENSURE(h->cand, sizeof(long long) * static_cast<size_t>(nq) * kprime * 3);
  // KNN (k = limit, hybrid_search.py:88) is enqueued first; BM25 (hybrid_search.py:70) goes in behind it while
  // the tensor-core path's overflow flags travel back, so the host round trip costs the device nothing
  // ... and when the KNN takes the tensor-core path, on a second stream UNDERNEATH the filter pass: the filter
  // kernel keeps one 178 KB CTA per SM busy on the tensor pipe at ~20 % issue utilisation, and one BM25 CTA
  // (38 KB, 512 threads) fits beside it.
  tl_mark(h, kTlStart, h->stream);
  Bm25Job bm25{&in, limit, k1, b};
  PendingKnn pend;
  int rc = knn_local_begin(h, static_cast<const float*>(in.q.p), nq, kprime, static_cast<long long*>(h->cand.p), pin,
                           &bm25, pend);
  if (rc != RSE_OK) return rc;
  if (!bm25.enqueued) {
    tl_mark(h, kTlBm25Start, h->stream);
    rc = bm25_run(h, in, nq, limit, k1, b, h->stream, false);
    if (rc != RSE_OK) return rc;
    tl_mark(h, kTlBm25End, h->stream);
  }
  if (keep) {
    *keep = pend;
  } else {
    rc = knn_local_finish(h, pend);
    if (rc != RSE_OK) return rc;
  }
  tl_mark(h, kTlKnnEnd, h->stream);
  return hybrid_tail(h, mode, param, tie_mode, nq, limit, kprime, nullptr, 0, bm25.enqueued, out);
}

}  // namespace

int rse_hybrid_stage(rse_index* h, int32_t nq, const float* q_host, const int32_t* tok_indptr,
                     const int32_t* term_rows) {
  if (!h) return RSE_ERR_INVALID;
  if (nq < 0 || (nq > 0 && (!q_host || !tok_indptr))) return fail(h, RSE_ERR_INVALID, "rse_hybrid_stage: bad arguments");
  // asynchronous: rse_hybrid_run / _fetch (or rse_synchronize) order behind it
  return stage_batch(h, h->staged, nq, q_host, cudaMemcpyHostToDevice, tok_indptr, term_rows, h->stream);
}

int rse_hybrid_run(rse_index* h, int32_t mode, double param, int32_t tie_mode, int32_t limit, int32_t knn_multiplier,
                   double k1, double b) {
  if (!h) return RSE_ERR_INVALID;
  const int nq = h->staged.nq;
  if (nq <= 0) return fail(h, RSE_ERR_STATE, "rse_hybrid_run: nothing staged");
  const int kprime = hybrid_kprime(h, mode, limit, knn_multiplier);
  if (kprime < 0) return kprime;
  CK(cudaSetDevice(h->device));
  Fused out;
  int rc = packed_results(h, h->f_pack, nq, limit, &out);
  if (rc != RSE_OK) return rc;
  h->pack_n = static_cast<size_t>(nq) * limit; h->pack_nq = nq;
  return hybrid_local(h, mode, param, tie_mode, limit, kprime, k1, b, h->staged, h->pin_status, nullptr, out);
}

int rse_hybrid_run_merged_dev(rse_index* h, int32_t mode, double param, int32_t tie_mode, int32_t limit,
                              int32_t knn_multiplier, double k1, double b, const int64_t* gathered_dev,
                              int32_t n_lists, int64_t* out_id_dev, double* out_score_dev, double* out_a_dev,
                              double* out_b_dev, int32_t* out_count_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!gathered_dev || n_lists < 1 || !out_id_dev || !out_score_dev || !out_a_dev || !out_b_dev || !out_count_dev)
    return fail(h, RSE_ERR_INVALID, "rse_hybrid_run_merged_dev: bad arguments");
  const int nq = h->staged.nq;
  if (nq <= 0) return fail(h, RSE_ERR_STATE, "rse_hybrid_run: nothing staged");
  const int kprime = hybrid_kprime(h, mode, limit, knn_multiplier);
  if (kprime < 0) return kprime;
  CK(cudaSetDevice(h->device));
  // BM25 (k = limit, hybrid_search.py:70), then the merge of the gathered KNN candidates
  int rc = bm25_run(h, h->staged, nq, limit, k1, b, h->stream, false);
  if (rc != RSE_OK) return rc;
  return hybrid_tail(h, mode, param, tie_mode, nq, limit, kprime, reinterpret_cast<const long long*>(gathered_dev),
                     n_lists, false,
                     Fused{reinterpret_cast<long long*>(out_id_dev), out_score_dev, out_a_dev, out_b_dev, out_count_dev,
                           limit});
}

int rse_hybrid_fetch(rse_index* h, int32_t limit, int64_t* out_id, double* out_score, double* out_a, double* out_b,
                     int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  const int nq = h->staged.nq;
  if (nq <= 0) return fail(h, RSE_ERR_STATE, "rse_hybrid_fetch: nothing staged");
  if (!out_id || !out_score || !out_a || !out_b || !out_count) return fail(h, RSE_ERR_INVALID, "rse_hybrid_fetch: bad arguments");
  const size_t n = static_cast<size_t>(nq) * limit;
  if (h->pack_n != n || h->pack_nq != nq) return fail(h, RSE_ERR_STATE, "rse_hybrid_fetch: limit differs from the last rse_hybrid_run");
  const size_t bytes = 32 * n + 4 * static_cast<size_t>(nq);
  if (h->pin_out_bytes < bytes) {
    if (h->pin_out) CK(cudaFreeHost(h->pin_out));
    h->pin_out = nullptr; h->pin_out_bytes = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&h->pin_out), bytes + bytes / 2));
    h->pin_out_bytes = bytes + bytes / 2;
  }
  CK(cudaMemcpyAsync(h->pin_out, h->f_pack.p, bytes, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(bytes);
  CK(cudaStreamSynchronize(h->stream));
  tl_print(h);
  std::memcpy(out_id, h->pin_out, 8 * n);
  std::memcpy(out_score, h->pin_out + 8 * n, 8 * n);
  std::memcpy(out_a, h->pin_out + 16 * n, 8 * n);
  std::memcpy(out_b, h->pin_out + 24 * n, 8 * n);
  std::memcpy(out_count, h->pin_out + 32 * n, 4 * static_cast<size_t>(nq));
  return RSE_OK;
}

int rse_hybrid(rse_index* h, int32_t mode, double param, int32_t tie_mode, int32_t limit, int32_t knn_multiplier,
               int32_t nq, const float* q_host, const int32_t* tok_indptr, const int32_t* term_rows, double k1,
               double b, int64_t* out_id, double* out_score, double* out_a, double* out_b, int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  if (nq < 0 || (nq > 0 && (!out_id || !out_score || !out_a || !out_b || !out_count)))
    return fail(h, RSE_ERR_INVALID, "rse_hybrid: bad arguments");
  if (nq == 0) return RSE_OK;
  int rc = rse_hybrid_stage(h, nq, q_host, tok_indptr, term_rows);
  if (rc != RSE_OK) return rc;
  rc = rse_hybrid_run(h, mode, param, tie_mode, limit, knn_multiplier, k1, b);
  if (rc != RSE_OK) return rc;
  return rse_hybrid_fetch(h, limit, out_id, out_score, out_a, out_b, out_count);
}

int rse_hybrid_submit(rse_index* h, int32_t mode, double param, int32_t tie_mode, int32_t limit, int32_t knn_multiplier,
                      int32_t nq, const float* q_host, const int32_t* tok_indptr, const int32_t* term_rows, double k1,
                      double b, int64_t* ticket) {
  if (!h) return RSE_ERR_INVALID;
  if (!ticket || nq < 1 || !q_host || !tok_indptr) return fail(h, RSE_ERR_INVALID, "rse_hybrid_submit: bad arguments");
  const int kprime = hybrid_kprime(h, mode, limit, knn_multiplier);
  if (kprime < 0) return kprime;
  if (h->next_ticket - h->next_collect >= 2)
    return fail(h, RSE_ERR_STATE, "rse_hybrid_submit: two batches already in flight, collect one first");
  CK(cudaSetDevice(h->device));
  if (!h->stream_h2d) {
    CK(cudaStreamCreateWithFlags(&h->stream_h2d, cudaStreamNonBlocking));
    CK(cudaStreamCreateWithFlags(&h->stream_d2h, cudaStreamNonBlocking));
    CK(cudaEventCreateWithFlags(&h->ev_fused, cudaEventDisableTiming));
  }
  const int s = static_cast<int>(h->next_ticket & 1);
  rse_index::OutSlot& sl = h->out_slot[s];
  // query vectors through a pinned buffer of this slot: the upload is then truly asynchronous (a pageable source
  // makes cudaMemcpyAsync wait for the stream before it returns)
  const size_t qbytes = sizeof(float) * static_cast<size_t>(nq) * h->dim;
  if (!h->ev_q[s]) CK(cudaEventCreateWithFlags(&h->ev_q[s], cudaEventDisableTiming));
  else CK(cudaEventSynchronize(h->ev_q[s]));                 // the upload two tickets ago has left the buffer
  if (h->pin_q_bytes[s] < qbytes) {
    if (h->pin_q[s]) CK(cudaFreeHost(h->pin_q[s]));
    h->pin_q[s] = nullptr; h->pin_q_bytes[s] = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&h->pin_q[s]), qbytes + qbytes / 2));
    h->pin_q_bytes[s] = qbytes + qbytes / 2;
  }
  std::memcpy(h->pin_q[s], q_host, qbytes);

  // the batch is staged into the SLOT's buffers (uploads on the copy stream) and runs from there: whatever the handle
  // had staged is given up, so a later rse_hybrid_run / _fetch without a fresh rse_hybrid_stage fails
  h->staged.nq = 0; h->pack_n = 0; h->pack_nq = 0;
  int rc = stage_batch(h, sl.in, nq, h->pin_q[s], cudaMemcpyHostToDevice, tok_indptr, term_rows, h->stream_h2d);
  if (rc != RSE_OK) return rc;
  CK(cudaEventRecord(h->ev_q[s], h->stream_h2d));
  CK(cudaStreamWaitEvent(h->stream, h->ev_q[s], 0));
  Fused out;
  rc = packed_results(h, sl.f_pack, nq, limit, &out);
  if (rc != RSE_OK) return rc;
  rc = hybrid_local(h, mode, param, tie_mode, limit, kprime, k1, b, sl.in, sl.flags, &sl.knn, out);
  if (rc != RSE_OK) return rc;
  const size_t n = static_cast<size_t>(nq) * limit;
  const size_t bytes = 32 * n + 4 * static_cast<size_t>(nq);
  if (sl.bytes < bytes) {                                     // the slot is free: its previous ticket was collected
    if (sl.pin) CK(cudaFreeHost(sl.pin));
    sl.pin = nullptr; sl.bytes = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&sl.pin), bytes + bytes / 2));
    sl.bytes = bytes + bytes / 2;
  }
  if (!sl.ev) CK(cudaEventCreateWithFlags(&sl.ev, cudaEventDisableTiming));
  // results: third stream, behind the fusion kernel
  CK(cudaEventRecord(h->ev_fused, h->stream));
  CK(cudaStreamWaitEvent(h->stream_d2h, h->ev_fused, 0));
  CK(cudaMemcpyAsync(sl.pin, sl.f_pack.p, bytes, cudaMemcpyDeviceToHost, h->stream_d2h));
  CK(cudaEventRecord(sl.ev, h->stream_d2h));
  h->stats.d2h_bytes += static_cast<int64_t>(bytes);
  if (sl.knn.flags) {
    sl.tok_indptr.assign(tok_indptr, tok_indptr + nq + 1);
    sl.term_rows.assign(term_rows, term_rows + (term_rows ? tok_indptr[nq] : 0));
    sl.mode = mode; sl.tie_mode = tie_mode; sl.limit = limit; sl.knn_multiplier = knn_multiplier;
    sl.param = param; sl.k1 = k1; sl.b = b;
  }
  sl.n = n; sl.nq = nq; sl.ticket = h->next_ticket;
  *ticket = h->next_ticket++;
  return RSE_OK;
}

int rse_hybrid_collect(rse_index* h, int64_t ticket, int32_t* out_nq, int32_t* out_limit, int64_t* out_id,
                       double* out_score, double* out_a, double* out_b, int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  if (!out_id || !out_score || !out_a || !out_b || !out_count) return fail(h, RSE_ERR_INVALID, "rse_hybrid_collect: bad arguments");
  if (ticket != h->next_collect || ticket >= h->next_ticket)
    return fail(h, RSE_ERR_STATE, "rse_hybrid_collect: tickets are collected in submission order");
  rse_index::OutSlot& sl = h->out_slot[ticket & 1];
  CK(cudaEventSynchronize(sl.ev));
  tl_print(h);
  const size_t n = sl.n;
  if (out_nq) *out_nq = sl.nq;
  if (out_limit) *out_limit = sl.nq ? static_cast<int32_t>(n / sl.nq) : 0;
  if (sl.knn.flags) {
    bool flagged = false;
    for (int q = 0; q < sl.nq && !flagged; ++q) flagged = sl.knn.flags[q] != 0;
    if (flagged) {
      // the query vectors are still in this ticket's pinned staging buffer (the next ticket uses the other one);
      // the blocking call handles the flagged queries through the exact scan.  The batch submitted after this one
      // is complete and parked in its own pinned slot once the stream has drained.
      CK(cudaStreamSynchronize(h->stream));
      ++h->pipeline_reruns;
      // the ticket stays collectable until the re-run has succeeded (a failed re-run can be retried or drained)
      const int rc = rse_hybrid(h, sl.mode, sl.param, sl.tie_mode, sl.limit, sl.knn_multiplier, sl.nq, h->pin_q[ticket & 1],
                                sl.tok_indptr.data(), sl.term_rows.empty() ? nullptr : sl.term_rows.data(), sl.k1, sl.b,
                                out_id, out_score, out_a, out_b, out_count);
      h->staged.nq = 0; h->pack_n = 0; h->pack_nq = 0;
      if (rc != RSE_OK) return rc;
      sl.knn = PendingKnn{};
      ++h->next_collect;
      return RSE_OK;
    }
  }
  std::memcpy(out_id, sl.pin, 8 * n);
  std::memcpy(out_score, sl.pin + 8 * n, 8 * n);
  std::memcpy(out_a, sl.pin + 16 * n, 8 * n);
  std::memcpy(out_b, sl.pin + 24 * n, 8 * n);
  std::memcpy(out_count, sl.pin + 32 * n, 4 * static_cast<size_t>(sl.nq));
  ++h->next_collect;
  return RSE_OK;
}

// ------------------------------------------------------------------ §8(f2)/(f3): text encoders on the device
namespace {

int enc_alloc(rse_index* h, float** p, size_t n) {
  CK(cudaMalloc(p, sizeof(float) * std::max<size_t>(n, 1)));
  return RSE_OK;
}

extern "C++" {
template <int EPI>
int enc_gemm(rse_index* h, const float* A, const float* W, const float* bias, float* C, int M, int N, int K) {
  dim3 grid((N + kGemmBN - 1) / kGemmBN, (M + kGemmBM - 1) / kGemmBM);
  enc_gemm_kernel<EPI><<<grid, 256, 0, h->stream>>>(A, W, bias, C, M, N, K);
  LAUNCHED(h);
  return RSE_OK;
}
}

// [rows][K] row-major fp32 matrix, box = 32 floats (one 128-byte swizzle atom) x 128 rows
int make_tmap_f32(rse_index* h, CUtensorMap* out, const float* base, int64_t rows, int64_t K, int box_rows) {
  static PFN_tmapEncodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    CK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres));
    if (!p || qres != cudaDriverEntryPointSuccess) return fail(h, RSE_ERR_CUDA, "cuTensorMapEncodeTiled unavailable");
    fn = reinterpret_cast<PFN_tmapEncodeTiled>(p);
  }
  const cuuint64_t gdim[2] = {static_cast<cuuint64_t>(K), static_cast<cuuint64_t>(rows)};
  const cuuint64_t gstr[1] = {static_cast<cuuint64_t>(K) * 4};
  const cuuint32_t box[2] = {kEgBK, static_cast<cuuint32_t>(box_rows)};
  const cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(out, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, const_cast<float*>(base), gdim, gstr, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(h, RSE_ERR_CUDA, "cuTensorMapEncodeTiled (encoder) failed: " + std::to_string(static_cast<int>(r)));
  return RSE_OK;
}

// tensor-core GEMM: C[M, N] = (A_hi + A_lo)[M, K] . (W_hi + W_lo)[N, K]^T + bias; EPI 1 / 2: GELU / quick_gelu -> C (hi), C_lo
extern "C++" {
template <int EPI>
int enc_gemm_tc(rse_index* h, const float* A_hi, const float* A_lo, const float* W_hi, const float* W_lo, const float* bias,
                float* C, float* C_lo, int M, int N, int K) {
  if (!(h->attr_mask & (1u << 17))) {
    CK(cudaFuncSetAttribute(enc_gemm_tc_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEgSmemBytes));
    CK(cudaFuncSetAttribute(enc_gemm_tc_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEgSmemBytes));
    CK(cudaFuncSetAttribute(enc_gemm_tc_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, kEgSmemBytes));
    h->attr_mask |= 1u << 17;
  }
  // 64-wide tiles, two CTAs per SM (r02, 256 queries / 2.5 k tokens, ms per host-buffer encode call: 64-wide
  // everywhere 1.35, 128-wide everywhere 1.46, 128-wide unless that leaves SMs idle 1.49): the kernel is bound by
  // the latency of its operand ring and by wave quantisation, so more, smaller tiles in flight win
  const int m_tiles = (M + kEgBM - 1) / kEgBM;
  CUtensorMap ta_h, ta_l, tw_h, tw_l;
  int rc = make_tmap_f32(h, &ta_h, A_hi, M, K, kEgBM);
  if (rc == RSE_OK) rc = make_tmap_f32(h, &ta_l, A_lo, M, K, kEgBM);
  if (rc == RSE_OK) rc = make_tmap_f32(h, &tw_h, W_hi, N, K, kEgBN);
  if (rc == RSE_OK) rc = make_tmap_f32(h, &tw_l, W_lo, N, K, kEgBN);
  if (rc != RSE_OK) return rc;
  dim3 grid((N + kEgBN - 1) / kEgBN, m_tiles);
  enc_gemm_tc_kernel<EPI><<<grid, kEgThreads, kEgSmemBytes, h->stream>>>(ta_h, ta_l, tw_h, tw_l, bias, C, C_lo, M, N, K);
  LAUNCHED(h);
  return RSE_OK;
}
}

// A BERT slot on device inputs: ids / type_ids (NULL = all 0) [T] and cu_seqlens [n_seq + 1] (starting at 0) are on the
// handle's device, max_len is the longest sequence; x <- encoder output [T, hidden]; out <- head output.  The host
// entry points (enc_run) and the batched rerank (rse_hybrid_rerank_run) both end here.
int enc_forward(rse_index* h, Encoder& e, const int32_t* ids, const int32_t* type_ids, const int32_t* cu, int n_seq,
                int T, int max_len, float* out_dev) {
  const rse_encoder_config& c = e.cfg;
  e.max_len = max_len;
  const int H = c.hidden, I = c.intermediate;
  const bool tc = e.mode == 0 && e.tc_ok;
  ENSURE(e.posidx, sizeof(int32_t) * T);
  ENSURE(e.x, sizeof(float) * static_cast<size_t>(T) * H);
  ENSURE(e.qkv, sizeof(float) * static_cast<size_t>(T) * 3 * H);
  ENSURE(e.ctx, sizeof(float) * static_cast<size_t>(T) * H);
  ENSURE(e.tmp, sizeof(float) * static_cast<size_t>(T) * H);
  ENSURE(e.ff, sizeof(float) * static_cast<size_t>(T) * I);
  if (tc) {
    ENSURE(e.x_h, sizeof(float) * static_cast<size_t>(T) * H);
    ENSURE(e.x_l, sizeof(float) * static_cast<size_t>(T) * H);
    ENSURE(e.ctx_l, sizeof(float) * static_cast<size_t>(T) * H);
    ENSURE(e.ff_l, sizeof(float) * static_cast<size_t>(T) * I);
  }
  float* x = static_cast<float*>(e.x.p);
  float* qkv = static_cast<float*>(e.qkv.p);
  float* ctx = static_cast<float*>(e.ctx.p);
  float* tmp = static_cast<float*>(e.tmp.p);
  float* ff = static_cast<float*>(e.ff.p);
  float* x_h = tc ? static_cast<float*>(e.x_h.p) : nullptr;
  float* x_l = tc ? static_cast<float*>(e.x_l.p) : nullptr;
  float* ctx_l = tc ? static_cast<float*>(e.ctx_l.p) : nullptr;
  float* ff_l = tc ? static_cast<float*>(e.ff_l.p) : nullptr;
  enc_positions_kernel<<<(T + 255) / 256, 256, 0, h->stream>>>(cu, n_seq, T, static_cast<int32_t*>(e.posidx.p));
  LAUNCHED(h);
  const int tok_grid = (T + 3) / 4;
  enc_embed_ln_kernel<<<tok_grid, 128, 0, h->stream>>>(
      ids, type_ids,
      static_cast<const int32_t*>(e.posidx.p), T, H, c.vocab_size, c.max_positions, c.type_vocab, e.word, e.pos, e.type,
      e.elng, e.elnb, c.ln_eps, x, x_h, x_l);
  LAUNCHED(h);
  const int hd = H / c.heads;
  for (const EncLayer& l : e.layers) {
    int rc = tc ? enc_gemm_tc<0>(h, x_h, x_l, l.wqkv_h, l.wqkv_l, l.bqkv, qkv, nullptr, T, 3 * H, H)
                : enc_gemm<0>(h, x, l.wqkv, l.bqkv, qkv, T, 3 * H, H);
    if (rc != RSE_OK) return rc;
    dim3 agrid(n_seq, c.heads);
    // one thread per query row: a CTA as wide as the longest sequence of the batch (32 .. 256 threads) — search
    // queries of 4-16 tokens used to idle 7 of 8 lanes of a 128-thread CTA, 160-token rerank pairs took two rounds
    // (above 128 threads only when the grid leaves SMs idle anyway: 216 registers x 256 threads is one CTA per SM)
    const int acap = static_cast<int64_t>(n_seq) * c.heads < 2ll * h->sm_count ? 256 : 128;
    const int athreads = std::min(acap, std::max(32, (e.max_len + 31) / 32 * 32));
    if (hd == 32) enc_attention_kernel<32><<<agrid, athreads, 0, h->stream>>>(qkv, cu, H, ctx, ctx_l);
    else enc_attention_kernel<64><<<agrid, athreads, 0, h->stream>>>(qkv, cu, H, ctx, ctx_l);
    LAUNCHED(h);
    rc = tc ? enc_gemm_tc<0>(h, ctx, ctx_l, l.wo_h, l.wo_l, l.bo, tmp, nullptr, T, H, H)
            : enc_gemm<0>(h, ctx, l.wo, l.bo, tmp, T, H, H);
    if (rc != RSE_OK) return rc;
    enc_add_ln_kernel<<<tok_grid, 128, 0, h->stream>>>(tmp, x, T, H, l.ln1g, l.ln1b, c.ln_eps, x, x_h, x_l);
    LAUNCHED(h);
    rc = tc ? enc_gemm_tc<1>(h, x_h, x_l, l.wi_h, l.wi_l, l.bi, ff, ff_l, T, I, H)
            : enc_gemm<1>(h, x, l.wi, l.bi, ff, T, I, H);
    if (rc != RSE_OK) return rc;
    rc = tc ? enc_gemm_tc<0>(h, ff, ff_l, l.wo2_h, l.wo2_l, l.bo2, tmp, nullptr, T, H, I)
            : enc_gemm<0>(h, ff, l.wo2, l.bo2, tmp, T, H, I);
    if (rc != RSE_OK) return rc;
    enc_add_ln_kernel<<<tok_grid, 128, 0, h->stream>>>(tmp, x, T, H, l.ln2g, l.ln2b, c.ln_eps, x, x_h, x_l);
    LAUNCHED(h);
  }
  if (c.head == 0) {
    enc_pool_mean_norm_kernel<<<n_seq, 128, 0, h->stream>>>(x, cu, H, out_dev);
  } else {
    enc_cls_head_kernel<<<n_seq, 128, sizeof(float) * (H + 32), h->stream>>>(x, cu, H, e.poolw, e.poolb, e.clsw, e.clsb, out_dev);
  }
  LAUNCHED(h);
  return RSE_OK;
}

// ---- §10 f4: the CLIP towers (clip.cuh).  Scratch for T tokens; y_h / y_l live in x_h / x_l.
int clip_buffers(rse_index* h, Encoder& e, int T, bool tc) {
  const size_t H = e.ccfg.hidden, I = e.ccfg.intermediate, t = static_cast<size_t>(T);
  ENSURE(e.x, sizeof(float) * t * H);
  ENSURE(e.y, sizeof(float) * t * H);
  ENSURE(e.qkv, sizeof(float) * t * 3 * H);
  ENSURE(e.ctx, sizeof(float) * t * H);
  ENSURE(e.tmp, sizeof(float) * t * H);
  ENSURE(e.ff, sizeof(float) * t * I);
  if (tc) {
    ENSURE(e.x_h, sizeof(float) * t * H);
    ENSURE(e.x_l, sizeof(float) * t * H);
    ENSURE(e.ctx_l, sizeof(float) * t * H);
    ENSURE(e.ff_l, sizeof(float) * t * I);
  }
  return RSE_OK;
}

// the pre-LN layers: on entry x = the embeddings and y = layer 0's layer_norm1(x); on exit x = the last hidden state
int clip_layers(rse_index* h, Encoder& e, int n_seq, int T, bool tc, bool causal) {
  const rse_clip_config& c = e.ccfg;
  const int H = c.hidden, I = c.intermediate, hd = H / c.heads;
  float* x = static_cast<float*>(e.x.p);
  float* y = static_cast<float*>(e.y.p);
  float* qkv = static_cast<float*>(e.qkv.p);
  float* ctx = static_cast<float*>(e.ctx.p);
  float* tmp = static_cast<float*>(e.tmp.p);
  float* ff = static_cast<float*>(e.ff.p);
  float* y_h = tc ? static_cast<float*>(e.x_h.p) : nullptr;
  float* y_l = tc ? static_cast<float*>(e.x_l.p) : nullptr;
  float* ctx_l = tc ? static_cast<float*>(e.ctx_l.p) : nullptr;
  float* ff_l = tc ? static_cast<float*>(e.ff_l.p) : nullptr;
  const int32_t* cu = static_cast<const int32_t*>(e.cu.p);
  const int tok_grid = (T + 3) / 4;
  for (size_t li = 0; li < e.layers.size(); ++li) {
    const EncLayer& l = e.layers[li];
    int rc = tc ? enc_gemm_tc<0>(h, y_h, y_l, l.wqkv_h, l.wqkv_l, l.bqkv, qkv, nullptr, T, 3 * H, H)
                : enc_gemm<0>(h, y, l.wqkv, l.bqkv, qkv, T, 3 * H, H);
    if (rc != RSE_OK) return rc;
    dim3 agrid(n_seq, c.heads);
    const int acap = static_cast<int64_t>(n_seq) * c.heads < 2ll * h->sm_count ? 256 : 128;   // as enc_forward
    const int athreads = std::min(acap, std::max(32, (e.max_len + 31) / 32 * 32));
    if (hd == 32) {
      if (causal) enc_attention_kernel<32, true><<<agrid, athreads, 0, h->stream>>>(qkv, cu, H, ctx, ctx_l);
      else enc_attention_kernel<32><<<agrid, athreads, 0, h->stream>>>(qkv, cu, H, ctx, ctx_l);
    } else {
      if (causal) enc_attention_kernel<64, true><<<agrid, athreads, 0, h->stream>>>(qkv, cu, H, ctx, ctx_l);
      else enc_attention_kernel<64><<<agrid, athreads, 0, h->stream>>>(qkv, cu, H, ctx, ctx_l);
    }
    LAUNCHED(h);
    rc = tc ? enc_gemm_tc<0>(h, ctx, ctx_l, l.wo_h, l.wo_l, l.bo, tmp, nullptr, T, H, H)
            : enc_gemm<0>(h, ctx, l.wo, l.bo, tmp, T, H, H);
    if (rc != RSE_OK) return rc;
    clip_residual_ln_kernel<<<tok_grid, 128, 0, h->stream>>>(x, tmp, T, H, l.ln2g, l.ln2b, c.ln_eps, y, y_h, y_l);
    LAUNCHED(h);
    rc = tc ? enc_gemm_tc<2>(h, y_h, y_l, l.wi_h, l.wi_l, l.bi, ff, ff_l, T, I, H)
            : enc_gemm<2>(h, y, l.wi, l.bi, ff, T, I, H);
    if (rc != RSE_OK) return rc;
    rc = tc ? enc_gemm_tc<0>(h, ff, ff_l, l.wo2_h, l.wo2_l, l.bo2, tmp, nullptr, T, H, I)
            : enc_gemm<0>(h, ff, l.wo2, l.bo2, tmp, T, H, I);
    if (rc != RSE_OK) return rc;
    const EncLayer* nx = li + 1 < e.layers.size() ? &e.layers[li + 1] : nullptr;    // the next layer's layer_norm1
    clip_residual_ln_kernel<<<tok_grid, 128, 0, h->stream>>>(x, tmp, T, H, nx ? nx->ln1g : nullptr,
                                                             nx ? nx->ln1b : nullptr, c.ln_eps, y, y_h, y_l);
    LAUNCHED(h);
  }
  return RSE_OK;
}

// pixels_dev [n, 3, S, S] on the device -> out_dev [n, projection_dim]
int clip_vision_forward(rse_index* h, Encoder& e, int n, const float* pixels_dev, float* out_dev) {
  const rse_clip_config& c = e.ccfg;
  const int H = c.hidden, S = c.image_size, P = c.patch_size, G = S / P, L = G * G + 1, Kp = e.patch_k;
  const int T = n * L, Mp = n * G * G;
  const bool tc = e.mode == 0 && e.tc_ok;
  int rc = clip_buffers(h, e, T, tc);
  if (rc != RSE_OK) return rc;
  ENSURE(e.cu, sizeof(int32_t) * (n + 1));
  ENSURE(e.patch, sizeof(float) * static_cast<size_t>(Mp) * Kp);
  if (tc) ENSURE(e.patch_l, sizeof(float) * static_cast<size_t>(Mp) * Kp);
  int32_t* cu = static_cast<int32_t*>(e.cu.p);
  float* patch = static_cast<float*>(e.patch.p);
  float* tmp = static_cast<float*>(e.tmp.p);
  clip_fixed_cu_kernel<<<(n + 256) / 256, 256, 0, h->stream>>>(n, L, cu);
  LAUNCHED(h);
  const int64_t n_elem = static_cast<int64_t>(Mp) * Kp;
  clip_patchify_kernel<<<static_cast<unsigned int>((n_elem + 255) / 256), 256, 0, h->stream>>>(
      pixels_dev, n_elem, S, P, G, Kp, tc ? nullptr : patch, tc ? patch : nullptr,
      tc ? static_cast<float*>(e.patch_l.p) : nullptr);
  LAUNCHED(h);
  // the patch conv (no bias) as one GEMM: [n*G*G, Kp] . [hidden, Kp]^T -> tmp
  rc = tc ? enc_gemm_tc<0>(h, patch, static_cast<float*>(e.patch_l.p), e.patch_w_h, e.patch_w_l, e.zero_bias, tmp,
                           nullptr, Mp, H, Kp)
          : enc_gemm<0>(h, patch, e.patch_w, e.zero_bias, tmp, Mp, H, Kp);
  if (rc != RSE_OK) return rc;
  const EncLayer& l0 = e.layers[0];
  clip_vision_embed_kernel<<<(T + 3) / 4, 128, 0, h->stream>>>(
      tmp, T, L, H, e.cls_emb, e.pos, e.elng, e.elnb, l0.ln1g, l0.ln1b, c.ln_eps, static_cast<float*>(e.x.p),
      static_cast<float*>(e.y.p), tc ? static_cast<float*>(e.x_h.p) : nullptr, tc ? static_cast<float*>(e.x_l.p) : nullptr);
  LAUNCHED(h);
  e.max_len = L;
  rc = clip_layers(h, e, n, T, tc, false);
  if (rc != RSE_OK) return rc;
  clip_head_kernel<<<n, 128, 0, h->stream>>>(static_cast<const float*>(e.x.p), cu, nullptr, 0, H, e.flng, e.flnb,
                                             c.ln_eps, e.proj, c.projection_dim, out_dev);
  LAUNCHED(h);
  return RSE_OK;
}

// ids / cu_seqlens on the device already (enc_run) -> out_dev [n_seq, projection_dim]
int clip_text_forward(rse_index* h, Encoder& e, int n_seq, int T, float* out_dev) {
  const rse_clip_config& c = e.ccfg;
  const int H = c.hidden;
  const bool tc = e.mode == 0 && e.tc_ok;
  int rc = clip_buffers(h, e, T, tc);
  if (rc != RSE_OK) return rc;
  ENSURE(e.posidx, sizeof(int32_t) * T);
  const int32_t* cu = static_cast<const int32_t*>(e.cu.p);
  const int32_t* ids = static_cast<const int32_t*>(e.ids.p);
  enc_positions_kernel<<<(T + 255) / 256, 256, 0, h->stream>>>(cu, n_seq, T, static_cast<int32_t*>(e.posidx.p));
  LAUNCHED(h);
  const EncLayer& l0 = e.layers[0];
  clip_text_embed_kernel<<<(T + 3) / 4, 128, 0, h->stream>>>(
      ids, static_cast<const int32_t*>(e.posidx.p), T, H, c.vocab_size, c.max_positions, e.word, e.pos, l0.ln1g,
      l0.ln1b, c.ln_eps, static_cast<float*>(e.x.p), static_cast<float*>(e.y.p),
      tc ? static_cast<float*>(e.x_h.p) : nullptr, tc ? static_cast<float*>(e.x_l.p) : nullptr);
  LAUNCHED(h);
  rc = clip_layers(h, e, n_seq, T, tc, true);
  if (rc != RSE_OK) return rc;
  clip_head_kernel<<<n_seq, 128, 0, h->stream>>>(static_cast<const float*>(e.x.p), cu, ids, c.eos_token_id, H, e.flng,
                                                 e.flnb, c.ln_eps, e.proj, c.projection_dim, out_dev);
  LAUNCHED(h);
  return RSE_OK;
}

int enc_check(rse_index* h, int32_t slot, bool need_final) {
  if (slot < 0 || slot >= RSE_MAX_ENCODERS) return fail(h, RSE_ERR_INVALID, "encoder: slot out of range");
  if (!h->enc[slot].created) return fail(h, RSE_ERR_STATE, "encoder: rse_encoder_create has not been called for this slot");
  if (need_final && !h->enc[slot].finalized) return fail(h, RSE_ERR_STATE, "encoder: not finalized (tensors missing?)");
  return RSE_OK;
}

// host inputs -> pinned -> device, then forward; out_dev [n_seq, hidden] (head 0) or [n_seq] (head 1)
int enc_run(rse_index* h, int32_t slot, const int32_t* ids, const int32_t* type_ids, const int32_t* cu, int32_t n_seq,
            float* out_dev) {
  int rc = enc_check(h, slot, true);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[slot];
  if (e.clip && e.ccfg.tower != 1)
    return fail(h, RSE_ERR_INVALID, "rse_encode: the slot holds a CLIP vision tower (use rse_encode_images)");
  if (e.clip && type_ids) return fail(h, RSE_ERR_INVALID, "rse_encode: type_ids must be NULL for a CLIP text tower");
  if (n_seq < 1 || !ids || !cu || !out_dev) return fail(h, RSE_ERR_INVALID, "rse_encode: bad arguments");
  if (cu[0] != 0) return fail(h, RSE_ERR_INVALID, "rse_encode: cu_seqlens must start at 0");
  int max_len = 1;
  for (int s = 0; s < n_seq; ++s) {
    const int len = cu[s + 1] - cu[s];
    max_len = std::max(max_len, len);
    if (len < 1) return fail(h, RSE_ERR_INVALID, "rse_encode: empty sequence (the reference raises 'cannot embed empty text', semantic_search.py:218-219)");
    if (len > e.cfg.max_positions) return fail(h, RSE_ERR_UNSUPPORTED, "rse_encode: sequence longer than max_positions (truncate on the host like the tokenizer does)");
  }
  const int T = cu[n_seq];
  CK(cudaSetDevice(h->device));
  const size_t n_in = static_cast<size_t>(T) * 2 + n_seq + 1;
  const int pb = e.pin_next;
  e.pin_next ^= 1;
  if (!e.pin_ev[pb]) CK(cudaEventCreateWithFlags(&e.pin_ev[pb], cudaEventDisableTiming));
  else CK(cudaEventSynchronize(e.pin_ev[pb]));            // the uploads out of this buffer (two calls ago) have finished
  if (e.pin_in_n[pb] < n_in) {
    if (e.pin_in[pb]) CK(cudaFreeHost(e.pin_in[pb]));
    e.pin_in[pb] = nullptr; e.pin_in_n[pb] = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&e.pin_in[pb]), sizeof(int32_t) * (n_in + n_in / 2 + 64)));
    e.pin_in_n[pb] = n_in + n_in / 2 + 64;
  }
  int32_t* pin = e.pin_in[pb];
  std::memcpy(pin, ids, sizeof(int32_t) * T);
  if (type_ids) std::memcpy(pin + T, type_ids, sizeof(int32_t) * T);
  std::memcpy(pin + 2 * static_cast<size_t>(T), cu, sizeof(int32_t) * (n_seq + 1));
  ENSURE(e.ids, sizeof(int32_t) * T);
  ENSURE(e.type_ids, sizeof(int32_t) * T);
  ENSURE(e.cu, sizeof(int32_t) * (n_seq + 1));
  CK(cudaMemcpyAsync(e.ids.p, pin, sizeof(int32_t) * T, cudaMemcpyHostToDevice, h->stream));
  if (type_ids) CK(cudaMemcpyAsync(e.type_ids.p, pin + T, sizeof(int32_t) * T, cudaMemcpyHostToDevice, h->stream));
  CK(cudaMemcpyAsync(e.cu.p, pin + 2 * static_cast<size_t>(T), sizeof(int32_t) * (n_seq + 1), cudaMemcpyHostToDevice, h->stream));
  CK(cudaEventRecord(e.pin_ev[pb], h->stream));
  h->stats.h2d_bytes += static_cast<int64_t>(sizeof(int32_t)) * (static_cast<int64_t>(T) * (type_ids ? 2 : 1) + n_seq + 1);
  if (e.clip) {
    e.max_len = max_len;
    return clip_text_forward(h, e, n_seq, T, out_dev);
  }
  return enc_forward(h, e, static_cast<const int32_t*>(e.ids.p),
                     type_ids ? static_cast<const int32_t*>(e.type_ids.p) : nullptr, static_cast<const int32_t*>(e.cu.p),
                     n_seq, T, max_len, out_dev);
}

}  // namespace

int rse_encoder_create(rse_index* h, int32_t slot, const rse_encoder_config* cfg) {
  if (!h) return RSE_ERR_INVALID;
  if (slot < 0 || slot >= RSE_MAX_ENCODERS || !cfg) return fail(h, RSE_ERR_INVALID, "rse_encoder_create: bad arguments");
  const rse_encoder_config& c = *cfg;
  if (c.hidden < 32 || c.hidden > kEncMaxHidden || c.hidden % 32 || c.heads < 1 || c.hidden % c.heads ||
      (c.hidden / c.heads != 32 && c.hidden / c.heads != 64) || c.layers < 1 || c.layers > 48 || c.intermediate < 16 ||
      c.intermediate % 16 || c.hidden % 16 || c.vocab_size < 1 || c.max_positions < 1 || c.type_vocab < 1 ||
      (c.head != 0 && c.head != 1) || !(c.ln_eps > 0.0f))
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_encoder_create: unsupported shape (hidden % 32, head_dim 32 or 64, intermediate % 16)");
  CK(cudaSetDevice(h->device));
  Encoder& e = h->enc[slot];
  enc_release(e);
  e.cfg = c;
  const size_t H = c.hidden, I = c.intermediate;
  int rc = RSE_OK;
  auto A = [&](float** p, size_t n) { if (rc == RSE_OK) rc = enc_alloc(h, p, n); };
  A(&e.word, c.vocab_size * H); A(&e.pos, c.max_positions * H); A(&e.type, c.type_vocab * H); A(&e.elng, H); A(&e.elnb, H);
  if (c.head == 1) { A(&e.poolw, H * H); A(&e.poolb, H); A(&e.clsw, H); A(&e.clsb, 1); }
  e.layers.resize(c.layers);
  for (auto& l : e.layers) {
    A(&l.wqkv, 3 * H * H); A(&l.bqkv, 3 * H); A(&l.wo, H * H); A(&l.bo, H); A(&l.ln1g, H); A(&l.ln1b, H);
    A(&l.wi, I * H); A(&l.bi, I); A(&l.wo2, H * I); A(&l.bo2, H); A(&l.ln2g, H); A(&l.ln2b, H);
  }
  if (rc != RSE_OK) { enc_release(e); return rc; }
  e.created = true;
  return RSE_OK;
}

int rse_clip_create(rse_index* h, int32_t slot, const rse_clip_config* cfg) {
  if (!h) return RSE_ERR_INVALID;
  if (slot < 0 || slot >= RSE_MAX_ENCODERS || !cfg) return fail(h, RSE_ERR_INVALID, "rse_clip_create: bad arguments");
  const rse_clip_config& c = *cfg;
  const bool vision = c.tower == 0;
  bool ok = (c.tower == 0 || c.tower == 1) && c.hidden >= 32 && c.hidden <= kEncMaxHidden && c.hidden % 32 == 0 &&
            c.heads >= 1 && c.hidden % c.heads == 0 && (c.hidden / c.heads == 32 || c.hidden / c.heads == 64) &&
            c.layers >= 1 && c.layers <= 48 && c.intermediate >= 16 && c.intermediate % 16 == 0 &&
            c.projection_dim >= 1 && c.projection_dim <= 65536 && c.ln_eps > 0.0f;
  if (ok && vision)
    ok = c.patch_size >= 1 && c.image_size >= c.patch_size && c.image_size % c.patch_size == 0 &&
         c.image_size <= 8192 && static_cast<int64_t>(c.image_size / c.patch_size) * (c.image_size / c.patch_size) + 1 <= RSE_CLIP_MAX_TOKENS;
  if (ok && !vision) ok = c.vocab_size >= 1 && c.max_positions >= 1 && c.max_positions <= RSE_CLIP_MAX_TOKENS;
  if (!ok)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_clip_create: unsupported shape (tower 0 / 1, hidden % 32 and <= 1024, head_dim 32 or 64, "
                                        "intermediate % 16, image_size % patch_size == 0, at most " +
                                        std::to_string(RSE_CLIP_MAX_TOKENS) + " tokens per sequence)");
  CK(cudaSetDevice(h->device));
  Encoder& e = h->enc[slot];
  enc_release(e);
  e.clip = true;
  e.ccfg = c;
  const int G = vision ? c.image_size / c.patch_size : 0;
  e.patch_k = vision ? (3 * c.patch_size * c.patch_size + 127) / 128 * 128 : 0;
  // the BERT view of the shape (finalize's tensor-core check, enc_run's length check)
  e.cfg = rse_encoder_config{};
  e.cfg.vocab_size = c.vocab_size; e.cfg.hidden = c.hidden; e.cfg.layers = c.layers; e.cfg.heads = c.heads;
  e.cfg.intermediate = c.intermediate; e.cfg.max_positions = vision ? G * G + 1 : c.max_positions; e.cfg.ln_eps = c.ln_eps;
  const size_t H = c.hidden, I = c.intermediate;
  int rc = RSE_OK;
  auto A = [&](float** p, size_t n) { if (rc == RSE_OK) rc = enc_alloc(h, p, n); };
  A(&e.pos, static_cast<size_t>(e.cfg.max_positions) * H);
  A(&e.flng, H); A(&e.flnb, H); A(&e.proj, static_cast<size_t>(c.projection_dim) * H);
  if (vision) {
    A(&e.cls_emb, H); A(&e.elng, H); A(&e.elnb, H); A(&e.patch_w, H * e.patch_k); A(&e.zero_bias, H);
  } else {
    A(&e.word, static_cast<size_t>(c.vocab_size) * H);
  }
  e.layers.resize(c.layers);
  for (auto& l : e.layers) {
    A(&l.wqkv, 3 * H * H); A(&l.bqkv, 3 * H); A(&l.wo, H * H); A(&l.bo, H); A(&l.ln1g, H); A(&l.ln1b, H);
    A(&l.wi, I * H); A(&l.bi, I); A(&l.wo2, H * I); A(&l.bo2, H); A(&l.ln2g, H); A(&l.ln2b, H);
  }
  if (rc == RSE_OK && vision) {
    if (cudaMemset(e.patch_w, 0, sizeof(float) * H * e.patch_k) != cudaSuccess ||
        cudaMemset(e.zero_bias, 0, sizeof(float) * H) != cudaSuccess)
      rc = fail(h, RSE_ERR_CUDA, "rse_clip_create: cudaMemset failed");
  }
  if (rc != RSE_OK) { enc_release(e); return rc; }
  e.created = true;
  return RSE_OK;
}

namespace {
// HuggingFace CLIP state_dict name -> destination in a CLIP slot
int clip_set_tensor(rse_index* h, Encoder& e, const std::string& full, const float* data, int64_t n_elem) {
  const rse_clip_config& c = e.ccfg;
  const bool vision = c.tower == 0;
  const int64_t H = c.hidden, I = c.intermediate;
  const char* tower = vision ? "vision_model." : "text_model.";
  const char* projn = vision ? "visual_projection." : "text_projection.";
  size_t at = std::string::npos;
  for (const char* key : {tower, projn}) {
    const size_t p = full.find(key);
    if (p != std::string::npos && (at == std::string::npos || p < at)) at = p;
  }
  if (at == std::string::npos)
    return fail(h, RSE_ERR_INVALID, std::string("rse_encoder_set_tensor: not a CLIP ") + (vision ? "vision" : "text") +
                                         " tower tensor name: " + full);
  const std::string nm = full.substr(at);
  const std::string tw(tower);
  float* dst = nullptr;
  int64_t want = 0;
  bool patch = false;
  auto is = [&](const char* s_) { return nm == s_; };
  if (is(vision ? "visual_projection.weight" : "text_projection.weight")) { dst = e.proj; want = c.projection_dim * H; }
  else if (nm == tw + "embeddings.position_embedding.weight") { dst = e.pos; want = e.cfg.max_positions * H; }
  else if (nm == tw + (vision ? "post_layernorm.weight" : "final_layer_norm.weight")) { dst = e.flng; want = H; }
  else if (nm == tw + (vision ? "post_layernorm.bias" : "final_layer_norm.bias")) { dst = e.flnb; want = H; }
  else if (!vision && is("text_model.embeddings.token_embedding.weight")) { dst = e.word; want = c.vocab_size * H; }
  else if (vision && is("vision_model.embeddings.class_embedding")) { dst = e.cls_emb; want = H; }
  else if (vision && is("vision_model.embeddings.patch_embedding.weight")) {
    dst = e.patch_w; want = H * 3 * c.patch_size * c.patch_size; patch = true;
  }
  else if (vision && is("vision_model.pre_layrnorm.weight")) { dst = e.elng; want = H; }
  else if (vision && is("vision_model.pre_layrnorm.bias")) { dst = e.elnb; want = H; }
  else if (nm.rfind(tw + "encoder.layers.", 0) == 0) {
    const size_t b = tw.size() + 15, dot = nm.find('.', b);
    if (dot == std::string::npos) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: bad layer name: " + full);
    const int li = std::atoi(nm.substr(b, dot - b).c_str());
    if (li < 0 || li >= c.layers) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: layer index out of range: " + full);
    EncLayer& l = e.layers[li];
    const std::string t = nm.substr(dot + 1);
    if (t == "self_attn.q_proj.weight") { dst = l.wqkv; want = H * H; }
    else if (t == "self_attn.k_proj.weight") { dst = l.wqkv + H * H; want = H * H; }
    else if (t == "self_attn.v_proj.weight") { dst = l.wqkv + 2 * H * H; want = H * H; }
    else if (t == "self_attn.q_proj.bias") { dst = l.bqkv; want = H; }
    else if (t == "self_attn.k_proj.bias") { dst = l.bqkv + H; want = H; }
    else if (t == "self_attn.v_proj.bias") { dst = l.bqkv + 2 * H; want = H; }
    else if (t == "self_attn.out_proj.weight") { dst = l.wo; want = H * H; }
    else if (t == "self_attn.out_proj.bias") { dst = l.bo; want = H; }
    else if (t == "layer_norm1.weight") { dst = l.ln1g; want = H; }
    else if (t == "layer_norm1.bias") { dst = l.ln1b; want = H; }
    else if (t == "mlp.fc1.weight") { dst = l.wi; want = I * H; }
    else if (t == "mlp.fc1.bias") { dst = l.bi; want = I; }
    else if (t == "mlp.fc2.weight") { dst = l.wo2; want = H * I; }
    else if (t == "mlp.fc2.bias") { dst = l.bo2; want = H; }
    else if (t == "layer_norm2.weight") { dst = l.ln2g; want = H; }
    else if (t == "layer_norm2.bias") { dst = l.ln2b; want = H; }
  }
  if (!dst) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: unknown tensor: " + full);
  if (n_elem != want) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: wrong element count for " + full);
  CK(cudaSetDevice(h->device));
  if (patch) {      // [hidden, 3*P*P] into the zero-padded [hidden, patch_k]
    const size_t k = 3 * static_cast<size_t>(c.patch_size) * c.patch_size;
    CK(cudaMemcpy2D(dst, sizeof(float) * e.patch_k, data, sizeof(float) * k, sizeof(float) * k, H, cudaMemcpyHostToDevice));
  } else {
    CK(cudaMemcpy(dst, data, sizeof(float) * n_elem, cudaMemcpyHostToDevice));
  }
  e.seen.insert(nm);
  e.finalized = false;
  return RSE_OK;
}
}  // namespace

int rse_encoder_set_tensor(rse_index* h, int32_t slot, const char* name, const float* data, int64_t n_elem) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, false);
  if (rc != RSE_OK) return rc;
  if (!name || !data || n_elem < 1) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: bad arguments");
  Encoder& e = h->enc[slot];
  if (e.clip) return clip_set_tensor(h, e, name, data, n_elem);
  const rse_encoder_config& c = e.cfg;
  const int64_t H = c.hidden, I = c.intermediate;
  // HuggingFace state_dict names, with whatever prefix the wrapper adds ("bert.", "0.auto_model.", ...)
  std::string full(name);
  size_t at = std::string::npos;
  for (const char* key : {"embeddings.", "encoder.layer.", "pooler.", "classifier."}) {
    const size_t p = full.find(key);
    if (p != std::string::npos && (at == std::string::npos || p < at)) at = p;
  }
  if (at == std::string::npos) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: not a BERT tensor name: " + full);
  const std::string nm = full.substr(at);
  float* dst = nullptr;
  int64_t want = 0;
  auto is = [&](const char* s_) { return nm == s_; };
  if (is("embeddings.word_embeddings.weight")) { dst = e.word; want = c.vocab_size * H; }
  else if (is("embeddings.position_embeddings.weight")) { dst = e.pos; want = c.max_positions * H; }
  else if (is("embeddings.token_type_embeddings.weight")) { dst = e.type; want = c.type_vocab * H; }
  else if (is("embeddings.LayerNorm.weight")) { dst = e.elng; want = H; }
  else if (is("embeddings.LayerNorm.bias")) { dst = e.elnb; want = H; }
  else if (is("pooler.dense.weight")) { dst = e.poolw; want = H * H; }
  else if (is("pooler.dense.bias")) { dst = e.poolb; want = H; }
  else if (is("classifier.weight")) { dst = e.clsw; want = H; }
  else if (is("classifier.bias")) { dst = e.clsb; want = 1; }
  else if (nm.rfind("encoder.layer.", 0) == 0) {
    const size_t dot = nm.find('.', 14);
    if (dot == std::string::npos) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: bad layer name: " + full);
    const int li = std::atoi(nm.substr(14, dot - 14).c_str());
    if (li < 0 || li >= c.layers) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: layer index out of range: " + full);
    EncLayer& l = e.layers[li];
    const std::string t = nm.substr(dot + 1);
    if (t == "attention.self.query.weight") { dst = l.wqkv; want = H * H; }
    else if (t == "attention.self.key.weight") { dst = l.wqkv + H * H; want = H * H; }
    else if (t == "attention.self.value.weight") { dst = l.wqkv + 2 * H * H; want = H * H; }
    else if (t == "attention.self.query.bias") { dst = l.bqkv; want = H; }
    else if (t == "attention.self.key.bias") { dst = l.bqkv + H; want = H; }
    else if (t == "attention.self.value.bias") { dst = l.bqkv + 2 * H; want = H; }
    else if (t == "attention.output.dense.weight") { dst = l.wo; want = H * H; }
    else if (t == "attention.output.dense.bias") { dst = l.bo; want = H; }
    else if (t == "attention.output.LayerNorm.weight") { dst = l.ln1g; want = H; }
    else if (t == "attention.output.LayerNorm.bias") { dst = l.ln1b; want = H; }
    else if (t == "intermediate.dense.weight") { dst = l.wi; want = I * H; }
    else if (t == "intermediate.dense.bias") { dst = l.bi; want = I; }
    else if (t == "output.dense.weight") { dst = l.wo2; want = H * I; }
    else if (t == "output.dense.bias") { dst = l.bo2; want = H; }
    else if (t == "output.LayerNorm.weight") { dst = l.ln2g; want = H; }
    else if (t == "output.LayerNorm.bias") { dst = l.ln2b; want = H; }
  }
  if (!dst) {
    if (c.head == 0 && (nm.rfind("pooler.", 0) == 0 || nm.rfind("classifier.", 0) == 0)) return RSE_OK;   // unused by this head
    return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: unknown tensor: " + full);
  }
  if (n_elem != want) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_tensor: wrong element count for " + full);
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpy(dst, data, sizeof(float) * n_elem, cudaMemcpyHostToDevice));
  e.seen.insert(nm);
  e.finalized = false;
  return RSE_OK;
}

int rse_encoder_finalize(rse_index* h, int32_t slot) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, false);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[slot];
  const size_t want = e.clip ? (e.ccfg.tower == 0 ? 8 : 5) + 16 * static_cast<size_t>(e.cfg.layers)
                             : 5 + 16 * static_cast<size_t>(e.cfg.layers) + (e.cfg.head == 1 ? 4 : 0);
  if (e.seen.size() != want)
    return fail(h, RSE_ERR_STATE, "rse_encoder_finalize: " + std::to_string(e.seen.size()) + " of " + std::to_string(want) +
                                      " tensors were set");
  // tf32 hi / lo halves of the weight matrices for the tensor-core GEMMs (every GEMM dimension must tile)
  const int64_t H = e.cfg.hidden, I = e.cfg.intermediate;
  e.tc_ok = (H % kEgBN == 0) && (I % kEgBN == 0) && (H % (kEgBK * kEgChunkKB) == 0) && (I % (kEgBK * kEgChunkKB) == 0);
  if (e.tc_ok) {
    CK(cudaSetDevice(h->device));
    for (EncLayer& l : e.layers) {
      struct { const float* w; float** hi; float** lo; int64_t n; } parts[4] = {
          {l.wqkv, &l.wqkv_h, &l.wqkv_l, 3 * H * H}, {l.wo, &l.wo_h, &l.wo_l, H * H},
          {l.wi, &l.wi_h, &l.wi_l, I * H}, {l.wo2, &l.wo2_h, &l.wo2_l, H * I}};
      for (auto& p : parts) {
        if (!*p.hi) { rc = enc_alloc(h, p.hi, p.n); if (rc != RSE_OK) return rc; }
        if (!*p.lo) { rc = enc_alloc(h, p.lo, p.n); if (rc != RSE_OK) return rc; }
        enc_split_kernel<<<static_cast<unsigned int>((p.n + 255) / 256), 256, 0, h->stream>>>(p.w, p.n, *p.hi, *p.lo);
        LAUNCHED(h);
      }
    }
    if (e.clip && e.ccfg.tower == 0) {          // the patch conv's weight (its K is padded to a multiple of 128)
      const int64_t n = H * e.patch_k;
      if (!e.patch_w_h) { rc = enc_alloc(h, &e.patch_w_h, n); if (rc != RSE_OK) return rc; }
      if (!e.patch_w_l) { rc = enc_alloc(h, &e.patch_w_l, n); if (rc != RSE_OK) return rc; }
      enc_split_kernel<<<static_cast<unsigned int>((n + 255) / 256), 256, 0, h->stream>>>(e.patch_w, n, e.patch_w_h, e.patch_w_l);
      LAUNCHED(h);
    }
    CK(cudaStreamSynchronize(h->stream));
  }
  e.finalized = true;
  return RSE_OK;
}

int rse_encoder_set_mode(rse_index* h, int32_t slot, int32_t mode) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, false);
  if (rc != RSE_OK) return rc;
  if (mode != 0 && mode != 1) return fail(h, RSE_ERR_INVALID, "rse_encoder_set_mode: mode must be 0 or 1");
  h->enc[slot].mode = mode;
  return RSE_OK;
}

int rse_encode_dev(rse_index* h, int32_t slot, const int32_t* ids, const int32_t* type_ids, const int32_t* cu_seqlens,
                   int32_t n_seq, float* out_dev) {
  if (!h) return RSE_ERR_INVALID;
  return enc_run(h, slot, ids, type_ids, cu_seqlens, n_seq, out_dev);
}

int rse_encode(rse_index* h, int32_t slot, const int32_t* ids, const int32_t* type_ids, const int32_t* cu_seqlens,
               int32_t n_seq, float* out_host) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, true);
  if (rc != RSE_OK) return rc;
  if (!out_host || n_seq < 1) return fail(h, RSE_ERR_INVALID, "rse_encode: bad arguments");
  Encoder& e = h->enc[slot];
  const size_t n_out = static_cast<size_t>(n_seq) * (e.clip ? e.ccfg.projection_dim : e.cfg.head == 0 ? e.cfg.hidden : 1);
  CK(cudaSetDevice(h->device));
  ENSURE(e.out, sizeof(float) * n_out);
  rc = enc_run(h, slot, ids, type_ids, cu_seqlens, n_seq, static_cast<float*>(e.out.p));
  if (rc != RSE_OK) return rc;
  CK(cudaMemcpyAsync(out_host, e.out.p, sizeof(float) * n_out, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(sizeof(float) * n_out);
  CK(cudaStreamSynchronize(h->stream));
  return RSE_OK;
}

namespace {
// checks, then (host pixels) pinned staging + upload on the handle's stream, then the vision tower
int clip_images(rse_index* h, int32_t slot, const float* pixels, int32_t n, float* out_dev, bool host) {
  int rc = enc_check(h, slot, true);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[slot];
  if (!e.clip || e.ccfg.tower != 0)
    return fail(h, RSE_ERR_INVALID, "rse_encode_images: the slot does not hold a CLIP vision tower");
  if (n < 1 || !pixels || !out_dev) return fail(h, RSE_ERR_INVALID, "rse_encode_images: bad arguments (n < 1 or NULL)");
  const int64_t per = 3ll * e.ccfg.image_size * e.ccfg.image_size;
  if (static_cast<int64_t>(n) * e.cfg.max_positions > (1ll << 24))
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_encode_images: more than 2^24 tokens in one call (split the batch)");
  CK(cudaSetDevice(h->device));
  if (!host) return clip_vision_forward(h, e, n, pixels, out_dev);
  const size_t n_px = static_cast<size_t>(n) * per;
  const int pb = e.pin_next;
  e.pin_next ^= 1;
  if (!e.pin_ev[pb]) CK(cudaEventCreateWithFlags(&e.pin_ev[pb], cudaEventDisableTiming));
  else CK(cudaEventSynchronize(e.pin_ev[pb]));              // the upload out of this buffer (two calls ago) is done
  if (e.pin_px_n[pb] < n_px) {
    if (e.pin_px[pb]) CK(cudaFreeHost(e.pin_px[pb]));
    e.pin_px[pb] = nullptr; e.pin_px_n[pb] = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&e.pin_px[pb]), sizeof(float) * n_px));
    e.pin_px_n[pb] = n_px;
  }
  std::memcpy(e.pin_px[pb], pixels, sizeof(float) * n_px);
  ENSURE(e.pix, sizeof(float) * n_px);
  CK(cudaMemcpyAsync(e.pix.p, e.pin_px[pb], sizeof(float) * n_px, cudaMemcpyHostToDevice, h->stream));
  CK(cudaEventRecord(e.pin_ev[pb], h->stream));
  h->stats.h2d_bytes += static_cast<int64_t>(sizeof(float) * n_px);
  return clip_vision_forward(h, e, n, static_cast<const float*>(e.pix.p), out_dev);
}
}  // namespace

int rse_encode_images_dev(rse_index* h, int32_t slot, const float* pixels_dev, int32_t n, float* out_dev) {
  if (!h) return RSE_ERR_INVALID;
  return clip_images(h, slot, pixels_dev, n, out_dev, false);
}

int rse_encode_images(rse_index* h, int32_t slot, const float* pixels_host, int32_t n, float* out_host) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, true);
  if (rc != RSE_OK) return rc;
  if (!out_host || n < 1) return fail(h, RSE_ERR_INVALID, "rse_encode_images: bad arguments (n < 1 or NULL)");
  Encoder& e = h->enc[slot];
  const size_t n_out = static_cast<size_t>(n) * (e.clip ? e.ccfg.projection_dim : 1);
  CK(cudaSetDevice(h->device));
  ENSURE(e.out, sizeof(float) * n_out);
  rc = clip_images(h, slot, pixels_host, n, static_cast<float*>(e.out.p), true);
  if (rc != RSE_OK) return rc;
  CK(cudaMemcpyAsync(out_host, e.out.p, sizeof(float) * n_out, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(sizeof(float) * n_out);
  CK(cudaStreamSynchronize(h->stream));
  return RSE_OK;
}

// ------------------------------------------------------------------ CLIP image preprocessing (imgproc.cuh)
int rse_imgproc_set(rse_index* h, int32_t slot, const rse_imgproc_cfg* cfg) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, false);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[slot];
  if (!e.clip || e.ccfg.tower != 0) return fail(h, RSE_ERR_INVALID, "rse_imgproc_set: the slot does not hold a CLIP vision tower");
  if (!cfg) return fail(h, RSE_ERR_INVALID, "rse_imgproc_set: cfg is NULL");
  const rse_imgproc_cfg& c = *cfg;
  if (c.backend != 0 && c.backend != 1) return fail(h, RSE_ERR_INVALID, "rse_imgproc_set: backend must be 0 or 1");
  const int S = e.ccfg.image_size;
  if (!c.do_resize || !c.do_center_crop || c.crop_height != S || c.crop_width != S || c.shortest_edge < S ||
      c.shortest_edge > RSE_IMGPROC_MAX_EDGE)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_imgproc_set: needs do_resize, do_center_crop and crop_height == crop_width == "
                                        "the tower's image_size (" + std::to_string(S) + ") <= shortest_edge");
  if (c.do_rescale && !(c.rescale_factor > 0.0 && std::isfinite(c.rescale_factor)))
    return fail(h, RSE_ERR_INVALID, "rse_imgproc_set: rescale_factor must be finite and > 0");
  IpNorm nm{};
  nm.normalize = c.do_normalize ? 1 : 0;
  for (int i = 0; i < 3; ++i) {
    if (c.do_normalize && static_cast<float>(c.std[i]) == 0.0f) return fail(h, RSE_ERR_INVALID, "rse_imgproc_set: std must not be 0");
    nm.m[i] = static_cast<float>(c.mean[i]);
    nm.s[i] = static_cast<float>(c.std[i]);
  }
  if (c.backend == 0) {
    if (c.do_rescale && c.do_normalize) {           // the fused form: float32 mean / std times float32(1 / rescale)
      const float inv = static_cast<float>(1.0 / c.rescale_factor);
      for (int i = 0; i < 3; ++i) { nm.m[i] = nm.m[i] * inv; nm.s[i] = nm.s[i] * inv; }
    } else if (c.do_rescale) {
      nm.rescale_mode = 1;
      nm.rf = static_cast<float>(c.rescale_factor);
    }
  } else if (c.do_rescale) {
    nm.rescale_mode = 2;
    nm.rd = c.rescale_factor;
  }
  e.ipcfg = c;
  e.ipnorm = nm;
  e.ip_set = true;
  return RSE_OK;
}

namespace {
constexpr size_t kIpTable = size_t(64) << 10;     // the image table in front of a chunk's pixels
constexpr int kIpChunkImages = static_cast<int>(kIpTable / sizeof(IpImage));

// first input index / end of the taps of output i of an axis n_in -> n_out (imgproc.cuh ip_taps, host side)
void ip_bounds(int i, int n_in, int n_out, int& lo, int& hi) {
  const double scale = static_cast<double>(n_in) / n_out;
  const double support = 2.0 * (scale > 1.0 ? scale : 1.0);
  const double center = (i + 0.5) * scale;
  lo = std::max(static_cast<int>(center - support + 0.5), 0);
  hi = std::min(static_cast<int>(center + support + 0.5), n_in);
}

int ip_taps_max(int n_in, int n_out) {
  if (n_in == n_out) return 1;
  const double scale = static_cast<double>(n_in) / n_out;
  return static_cast<int>(std::ceil(2.0 * (scale > 1.0 ? scale : 1.0))) * 2 + 1;
}

// checks every image, then chunk by chunk: stage -> upload (copy stream) -> coefficients, horizontal pass, vertical
// pass (handle's stream) into out_dev [n, 3, S, S]
int ip_run(rse_index* h, int32_t slot, const uint8_t* px, const int64_t* offs, const int32_t* hw, int32_t n,
           float* out_dev) {
  int rc = enc_check(h, slot, false);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[slot];
  if (!e.clip || e.ccfg.tower != 0) return fail(h, RSE_ERR_INVALID, "rse_image_preprocess: the slot does not hold a CLIP vision tower");
  if (!e.ip_set) return fail(h, RSE_ERR_STATE, "rse_image_preprocess: no rse_imgproc_set configuration for this slot");
  if (n < 1 || !px || !offs || !hw || !out_dev) return fail(h, RSE_ERR_INVALID, "rse_image_preprocess: bad arguments (n < 1 or NULL)");
  const rse_imgproc_cfg& c = e.ipcfg;
  const int S = e.ccfg.image_size, se = c.shortest_edge;
  std::vector<IpImage> im(n);
  std::vector<int> taps(n);
  for (int i = 0; i < n; ++i) {
    const int H = hw[2 * i], W = hw[2 * i + 1];
    const std::string at = "rse_image_preprocess: image " + std::to_string(i);
    if (H < 1 || W < 1 || offs[i] < 0) return fail(h, RSE_ERR_INVALID, at + ": bad size or offset");
    if (static_cast<int64_t>(H) * W > RSE_IMGPROC_MAX_PIXELS)
      return fail(h, RSE_ERR_UNSUPPORTED, at + ": more than RSE_IMGPROC_MAX_PIXELS pixels");
    IpImage& m = im[i];
    m.off = offs[i]; m.H = H; m.W = W; m.out = i;
    // transformers' get_resize_output_image_size(default_to_square=False): int(size * long / short)
    const int sh = std::min(H, W), lg = std::max(H, W);
    const int64_t nl = static_cast<int64_t>(static_cast<double>(static_cast<int64_t>(se) * lg) / sh);
    if (nl > RSE_IMGPROC_MAX_EDGE) return fail(h, RSE_ERR_UNSUPPORTED, at + ": a resized side above RSE_IMGPROC_MAX_EDGE");
    if (W <= H) { m.nw = se; m.nh = static_cast<int>(nl); } else { m.nh = se; m.nw = static_cast<int>(nl); }
    if (H > static_cast<int64_t>(RSE_IMGPROC_MAX_SCALE) * m.nh || W > static_cast<int64_t>(RSE_IMGPROC_MAX_SCALE) * m.nw)
      return fail(h, RSE_ERR_UNSUPPORTED, at + ": a downscale above RSE_IMGPROC_MAX_SCALE");
    if (c.backend == 1 && H > 100ll * W && m.nh < H)
      return fail(h, RSE_ERR_UNSUPPORTED, at + ": Pillow shrinks an image over 100 times taller than wide vertically first");
    m.top = (m.nh - S) / 2;
    m.left = (m.nw - S) / 2;
    if (m.nh == H) {
      m.ylo = m.top; m.rows = S;
    } else {                                        // one row of slack on each side: the device computes the taps
      int lo0, hi0, lo1, hi1;
      ip_bounds(m.top, H, m.nh, lo0, hi0);
      ip_bounds(m.top + S - 1, H, m.nh, lo1, hi1);
      m.ylo = std::max(lo0 - 1, 0);
      m.rows = std::min(hi1 + 1, H) - m.ylo;
    }
    taps[i] = std::max(ip_taps_max(W, m.nw), ip_taps_max(H, m.nh));
  }
  // chunks: consecutive images up to RSE_IMGPROC_CHUNK_BYTES of pixels (one image is at most 3 * 2^24 bytes)
  std::vector<int> starts{0};
  {
    size_t bytes = 0;
    for (int i = 0; i < n; ++i) {
      const size_t b = static_cast<size_t>(im[i].H) * im[i].W * 3;
      if (i > starts.back() && (bytes + b > size_t(RSE_IMGPROC_CHUNK_BYTES) || i - starts.back() >= kIpChunkImages)) {
        starts.push_back(i);
        bytes = 0;
      }
      bytes += b;
    }
    starts.push_back(n);
  }
  // scratch for the largest chunk (shared by all chunks: they run in order on one stream)
  size_t max_px = 0, max_mid = 0, max_w = 0;
  int max_cnt = 0;
  for (size_t ci = 0; ci + 1 < starts.size(); ++ci) {
    size_t pxb = 0, mid = 0;
    int K = 1;
    for (int i = starts[ci]; i < starts[ci + 1]; ++i) {
      im[i].mid_off = static_cast<long long>(mid);
      pxb += static_cast<size_t>(im[i].H) * im[i].W * 3;
      mid += static_cast<size_t>(im[i].rows) * S * 3;
      K = std::max(K, taps[i]);
    }
    const int cnt = starts[ci + 1] - starts[ci];
    max_px = std::max(max_px, pxb); max_mid = std::max(max_mid, mid); max_cnt = std::max(max_cnt, cnt);
    max_w = std::max(max_w, static_cast<size_t>(cnt) * 2 * S * K);
  }
  CK(cudaSetDevice(h->device));
  ENSURE(e.ip_axes, sizeof(IpAxis) * 2 * max_cnt);
  ENSURE(e.ip_span, sizeof(int2) * 2 * max_cnt * S);
  ENSURE(e.ip_w, sizeof(int) * max_w);
  ENSURE(e.ip_mid, std::max<size_t>(max_mid, 1));
  if (!e.ip_copy) CK(cudaStreamCreateWithFlags(&e.ip_copy, cudaStreamNonBlocking));
  const size_t need = kIpTable + max_px;
  for (int b = 0; b < 2; ++b) {
    if (!e.ip_ev_up[b]) CK(cudaEventCreateWithFlags(&e.ip_ev_up[b], cudaEventDisableTiming));
    if (!e.ip_ev_read[b]) CK(cudaEventCreateWithFlags(&e.ip_ev_read[b], cudaEventDisableTiming));
    if (e.ip_pin_n[b] < need) {
      CK(cudaEventSynchronize(e.ip_ev_up[b]));
      if (e.ip_pin[b]) CK(cudaFreeHost(e.ip_pin[b]));
      e.ip_pin[b] = nullptr; e.ip_pin_n[b] = 0;
      CK(cudaMallocHost(reinterpret_cast<void**>(&e.ip_pin[b]), need));
      e.ip_pin_n[b] = need;
    }
    ENSURE(e.ip_in[b], need);
  }
  IpAxis* axes = static_cast<IpAxis*>(e.ip_axes.p);
  int2* span = static_cast<int2*>(e.ip_span.p);
  int* wq = static_cast<int*>(e.ip_w.p);
  uint8_t* mid = static_cast<uint8_t*>(e.ip_mid.p);
  for (size_t ci = 0; ci + 1 < starts.size(); ++ci) {
    const int b = static_cast<int>(ci & 1), i0 = starts[ci], cnt = starts[ci + 1] - i0;
    CK(cudaEventSynchronize(e.ip_ev_up[b]));        // the upload out of this pinned buffer (two chunks ago) is done
    IpImage* tab = reinterpret_cast<IpImage*>(e.ip_pin[b]);
    uint8_t* dst = reinterpret_cast<uint8_t*>(e.ip_pin[b] + kIpTable);
    size_t pxb = 0;
    int K = 1, rows_w = 0;
    for (int j = 0; j < cnt; ++j) {
      IpImage m = im[i0 + j];
      const size_t bytes = static_cast<size_t>(m.H) * m.W * 3;
      std::memcpy(dst + pxb, px + m.off, bytes);
      m.off = static_cast<long long>(pxb);
      tab[j] = m;
      pxb += bytes;
      K = std::max(K, taps[i0 + j]);
      rows_w = std::max(rows_w, m.rows * S);
    }
    char* din = static_cast<char*>(e.ip_in[b].p);
    CK(cudaStreamWaitEvent(e.ip_copy, e.ip_ev_read[b], 0));
    CK(cudaMemcpyAsync(din, tab, sizeof(IpImage) * cnt, cudaMemcpyHostToDevice, e.ip_copy));
    CK(cudaMemcpyAsync(din + kIpTable, dst, pxb, cudaMemcpyHostToDevice, e.ip_copy));
    CK(cudaEventRecord(e.ip_ev_up[b], e.ip_copy));
    h->stats.h2d_bytes += static_cast<int64_t>(sizeof(IpImage) * cnt + pxb);
    CK(cudaStreamWaitEvent(h->stream, e.ip_ev_up[b], 0));
    const IpImage* dtab = reinterpret_cast<const IpImage*>(din);
    imgproc_bits_kernel<<<dim3(cnt, 2), kIpThreads, 0, h->stream>>>(dtab, c.backend, K, axes);
    LAUNCHED(h);
    imgproc_coeff_kernel<<<dim3(cnt, 2), kIpThreads, 0, h->stream>>>(dtab, c.backend, S, S, S, K, axes, span, wq);
    LAUNCHED(h);
    imgproc_hpass_kernel<<<dim3((rows_w + kIpThreads - 1) / kIpThreads, cnt), kIpThreads, 0, h->stream>>>(
        dtab, reinterpret_cast<const uint8_t*>(din + kIpTable), S, S, K, axes, span, wq, mid);
    LAUNCHED(h);
    imgproc_vpass_kernel<<<dim3((S * S + kIpThreads - 1) / kIpThreads, cnt), kIpThreads, 0, h->stream>>>(
        dtab, S, S, S, K, axes, span, wq, mid, e.ipnorm, out_dev);                  // IpImage::out is the call's index
    LAUNCHED(h);
    CK(cudaEventRecord(e.ip_ev_read[b], h->stream));
  }
  return RSE_OK;
}

// preprocess into the slot's pixel buffer, then the vision tower
int ip_encode(rse_index* h, int32_t slot, const uint8_t* px, const int64_t* offs, const int32_t* hw, int32_t n,
              float* out_dev) {
  int rc = enc_check(h, slot, true);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[slot];
  if (!e.clip || e.ccfg.tower != 0) return fail(h, RSE_ERR_INVALID, "rse_encode_images_u8: the slot does not hold a CLIP vision tower");
  if (n < 1 || !out_dev) return fail(h, RSE_ERR_INVALID, "rse_encode_images_u8: bad arguments (n < 1 or NULL)");
  if (static_cast<int64_t>(n) * e.cfg.max_positions > (1ll << 24))
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_encode_images_u8: more than 2^24 tokens in one call (split the batch)");
  CK(cudaSetDevice(h->device));
  ENSURE(e.pix, sizeof(float) * static_cast<size_t>(n) * 3 * e.ccfg.image_size * e.ccfg.image_size);
  rc = ip_run(h, slot, px, offs, hw, n, static_cast<float*>(e.pix.p));
  if (rc != RSE_OK) return rc;
  return clip_vision_forward(h, e, n, static_cast<const float*>(e.pix.p), out_dev);
}
}  // namespace

int rse_image_preprocess_dev(rse_index* h, int32_t slot, const uint8_t* px, const int64_t* offs, const int32_t* hw,
                             int32_t n, float* out_dev) {
  if (!h) return RSE_ERR_INVALID;
  return ip_run(h, slot, px, offs, hw, n, out_dev);
}

int rse_image_preprocess(rse_index* h, int32_t slot, const uint8_t* px, const int64_t* offs, const int32_t* hw,
                         int32_t n, float* out_host) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, false);
  if (rc != RSE_OK) return rc;
  if (!out_host || n < 1) return fail(h, RSE_ERR_INVALID, "rse_image_preprocess: bad arguments (n < 1 or NULL)");
  Encoder& e = h->enc[slot];
  const size_t n_out = static_cast<size_t>(n) * 3 * e.ccfg.image_size * e.ccfg.image_size;
  CK(cudaSetDevice(h->device));
  ENSURE(e.out, sizeof(float) * n_out);
  rc = ip_run(h, slot, px, offs, hw, n, static_cast<float*>(e.out.p));
  if (rc != RSE_OK) return rc;
  CK(cudaMemcpyAsync(out_host, e.out.p, sizeof(float) * n_out, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(sizeof(float) * n_out);
  CK(cudaStreamSynchronize(h->stream));
  return RSE_OK;
}

int rse_encode_images_u8_dev(rse_index* h, int32_t slot, const uint8_t* px, const int64_t* offs, const int32_t* hw,
                             int32_t n, float* out_dev) {
  if (!h) return RSE_ERR_INVALID;
  return ip_encode(h, slot, px, offs, hw, n, out_dev);
}

int rse_encode_images_u8(rse_index* h, int32_t slot, const uint8_t* px, const int64_t* offs, const int32_t* hw,
                         int32_t n, float* out_host) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, slot, true);
  if (rc != RSE_OK) return rc;
  if (!out_host || n < 1) return fail(h, RSE_ERR_INVALID, "rse_encode_images_u8: bad arguments (n < 1 or NULL)");
  Encoder& e = h->enc[slot];
  const size_t n_out = static_cast<size_t>(n) * (e.clip ? e.ccfg.projection_dim : 1);
  CK(cudaSetDevice(h->device));
  ENSURE(e.out, sizeof(float) * n_out);
  rc = ip_encode(h, slot, px, offs, hw, n, static_cast<float*>(e.out.p));
  if (rc != RSE_OK) return rc;
  CK(cudaMemcpyAsync(out_host, e.out.p, sizeof(float) * n_out, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(sizeof(float) * n_out);
  CK(cudaStreamSynchronize(h->stream));
  return RSE_OK;
}

int rse_hybrid_stage_dev(rse_index* h, int32_t nq, const float* q_dev, const int32_t* tok_indptr, const int32_t* term_rows) {
  if (!h) return RSE_ERR_INVALID;
  if (nq < 1 || !q_dev || !tok_indptr) return fail(h, RSE_ERR_INVALID, "rse_hybrid_stage_dev: bad arguments");
  return stage_batch(h, h->staged, nq, q_dev, cudaMemcpyDeviceToDevice, tok_indptr, term_rows, h->stream);
}

// ------------------------------------------------------------------ cross-encoder rerank of a fused batch (rerank.cuh)
int rse_rerank_docs_load(rse_index* h, const int64_t* ids, int64_t n_docs, const int64_t* tok_indptr,
                         const int32_t* tokens) {
  if (!h) return RSE_ERR_INVALID;
  if (n_docs < 1 || !ids || !tok_indptr) return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load: bad arguments");
  if (tok_indptr[0] != 0) return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load: tok_indptr must start at 0");
  for (int64_t i = 0; i < n_docs; ++i) {
    if (i > 0 && ids[i] <= ids[i - 1])
      return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load: ids must be strictly ascending (at " + std::to_string(i) + ")");
    if (tok_indptr[i + 1] < tok_indptr[i])
      return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load: tok_indptr must not decrease (at " + std::to_string(i) + ")");
  }
  const int64_t n_tok = tok_indptr[n_docs];
  if (n_tok > 0 && !tokens) return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load: tokens is NULL");
  int32_t max_tok = -1;
  int64_t max_len = 0;
  for (int64_t i = 0; i < n_docs; ++i) max_len = std::max(max_len, tok_indptr[i + 1] - tok_indptr[i]);
  for (int64_t i = 0; i < n_tok; ++i) {
    if (tokens[i] < 0) return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load: negative token id");
    max_tok = std::max(max_tok, tokens[i]);
  }
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));                       // a rerank run may still read the old store
  free_ptr(h->rr_doc_ids); free_ptr(h->rr_doc_indptr); free_ptr(h->rr_doc_tok);
  h->rr_n_docs = 0; h->rr_max_tok = -1;
  CK(cudaMalloc(&h->rr_doc_ids, 8 * n_docs));
  CK(cudaMalloc(&h->rr_doc_indptr, 8 * (n_docs + 1)));
  CK(cudaMalloc(&h->rr_doc_tok, 4 * std::max<int64_t>(n_tok, 1)));
  CK(cudaMemcpy(h->rr_doc_ids, ids, 8 * n_docs, cudaMemcpyHostToDevice));
  CK(cudaMemcpy(h->rr_doc_indptr, tok_indptr, 8 * (n_docs + 1), cudaMemcpyHostToDevice));
  if (n_tok > 0) CK(cudaMemcpy(h->rr_doc_tok, tokens, 4 * n_tok, cudaMemcpyHostToDevice));
  h->rr_n_docs = n_docs; h->rr_max_tok = max_tok; h->rr_max_doc_len = max_len;
  return RSE_OK;
}

int rse_set_rerank_token_budget(rse_index* h, int64_t tokens) {
  if (!h) return RSE_ERR_INVALID;
  if (tokens < 1 || tokens > INT_MAX) return fail(h, RSE_ERR_INVALID, "rse_set_rerank_token_budget: tokens must be in [1, 2^31)");
  h->rr_budget = tokens;
  return RSE_OK;
}

int rse_pair_truncate(int32_t n1, int32_t n2, int32_t max_length, int32_t* a, int32_t* b) {
  if (n1 < 0 || n2 < 0 || max_length < 4 || !a || !b) return RSE_ERR_INVALID;
  int x = 0, y = 0;
  pair_truncate(n1, n2, max_length - 3, &x, &y);
  *a = x; *b = y;
  return RSE_OK;
}

namespace {
void rr_mark(rse_index* h, int i) {
  if (h->timing && h->rr_ev[i]) cudaEventRecord(h->rr_ev[i], h->stream);
}
}  // namespace

int rse_hybrid_rerank_run(rse_index* h, int32_t slot, double k, int32_t tie_mode, int32_t limit,
                          int32_t knn_multiplier, double k1, double b, const int32_t* q_tok_indptr,
                          const int32_t* q_tok_ids, int32_t cls_id, int32_t sep_id, int32_t max_length,
                          int32_t activation) {
  if (!h) return RSE_ERR_INVALID;
  h->rr_nq = 0;
  if (limit < 1 || limit > RSE_MAX_RERANK_LIMIT) return fail(h, RSE_ERR_UNSUPPORTED, "rse_hybrid_rerank_run: limit must be in [1, 128]");
  if (activation != 0 && activation != 1) return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: activation must be 0 (logit) or 1 (sigmoid)");
  if (h->rr_n_docs < 1) return fail(h, RSE_ERR_STATE, "rse_hybrid_rerank_run: no document store (rse_rerank_docs_load)");
  const int nq = h->staged.nq;
  if (nq <= 0) return fail(h, RSE_ERR_STATE, "rse_hybrid_rerank_run: nothing staged");
  if (h->next_ticket != h->next_collect)
    return fail(h, RSE_ERR_STATE, "rse_hybrid_rerank_run: rse_hybrid_submit tickets are in flight (collect or drain them)");
  const int kprime = hybrid_kprime(h, 0, limit, knn_multiplier);
  if (kprime < 0) return kprime;
  if (slot < 0 || slot >= RSE_MAX_ENCODERS) return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: slot out of range");
  Encoder& e = h->enc[slot];
  if (!e.created || !e.finalized || e.clip || e.cfg.head != 1)
    return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: the slot does not hold a finalized head-1 (cross-encoder) BERT");
  if (max_length < 4 || max_length > e.cfg.max_positions)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_hybrid_rerank_run: max_length must be in [4, max_positions]");
  const int vocab = e.cfg.vocab_size;
  if (!q_tok_indptr || q_tok_indptr[0] != 0) return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: q_tok_indptr must start at 0");
  for (int q = 0; q < nq; ++q)
    if (q_tok_indptr[q + 1] < q_tok_indptr[q]) return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: q_tok_indptr must not decrease");
  const int n_qtok = q_tok_indptr[nq];
  if (n_qtok > 0 && !q_tok_ids) return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: q_tok_ids is NULL");
  int max_q = 0;
  for (int q = 0; q < nq; ++q) max_q = std::max(max_q, q_tok_indptr[q + 1] - q_tok_indptr[q]);
  for (int i = 0; i < n_qtok; ++i)
    if (q_tok_ids[i] < 0 || q_tok_ids[i] >= vocab)
      return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: query token id " + std::to_string(q_tok_ids[i]) + " outside the vocabulary");
  if (cls_id < 0 || cls_id >= vocab || sep_id < 0 || sep_id >= vocab)
    return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: cls_id / sep_id outside the vocabulary");
  if (h->rr_max_tok >= vocab)
    return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_run: the document store holds token id " + std::to_string(h->rr_max_tok) +
                                        " >= the encoder's vocab_size " + std::to_string(vocab));
  const int W = 2 * limit;
  const int64_t P = static_cast<int64_t>(nq) * W;
  if (P * max_length > INT_MAX) return fail(h, RSE_ERR_UNSUPPORTED, "rse_hybrid_rerank_run: nq * 2 * limit * max_length exceeds 2^31 tokens (split the batch)");
  CK(cudaSetDevice(h->device));
  if (h->timing)
    for (cudaEvent_t& ev : h->rr_ev) if (!ev) CK(cudaEventCreate(&ev));
  h->rr_timed = h->timing;
  ENSURE(h->rr_fid, 8 * P); ENSURE(h->rr_fsc, 8 * P); ENSURE(h->rr_fa, 8 * P); ENSURE(h->rr_fb, 8 * P);
  ENSURE(h->rr_fcnt, 4 * static_cast<size_t>(nq));
  ENSURE(h->rr_row, 4 * P); ENSURE(h->rr_ab, 8 * P);
  ENSURE(h->rr_qnp, 4 * static_cast<size_t>(nq)); ENSURE(h->rr_qnt, 4 * static_cast<size_t>(nq));
  ENSURE(h->rr_qpb, 4 * static_cast<size_t>(nq + 1)); ENSURE(h->rr_qtb, 4 * static_cast<size_t>(nq + 1));
  const size_t meta_n = kRrMetaHead + static_cast<size_t>(P) + 1;
  ENSURE(h->rr_meta, 4 * meta_n);
  ENSURE(h->rr_qptr, 4 * static_cast<size_t>(nq + 1)); ENSURE(h->rr_qtok, 4 * static_cast<size_t>(std::max(n_qtok, 1)));
  if (h->rr_pin_meta_n < meta_n) {
    if (h->rr_pin_meta) CK(cudaFreeHost(h->rr_pin_meta));
    h->rr_pin_meta = nullptr; h->rr_pin_meta_n = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&h->rr_pin_meta), 4 * (meta_n + meta_n / 2)));
    h->rr_pin_meta_n = meta_n + meta_n / 2;
  }
  CK(cudaMemcpyAsync(h->rr_qptr.p, q_tok_indptr, 4 * static_cast<size_t>(nq + 1), cudaMemcpyHostToDevice, h->stream));
  if (n_qtok > 0) CK(cudaMemcpyAsync(h->rr_qtok.p, q_tok_ids, 4 * static_cast<size_t>(n_qtok), cudaMemcpyHostToDevice, h->stream));
  h->stats.h2d_bytes += 4 * static_cast<int64_t>(nq + 1 + n_qtok);
  int* meta = static_cast<int*>(h->rr_meta.p);
  CK(cudaMemsetAsync(meta, 0, 4, h->stream));
  CK(cudaMemsetAsync(meta + 1, 0xFF, 4, h->stream));

  // 1. the hybrid step, with the whole union (2 * limit) in fused order into the rerank's own buffers
  rr_mark(h, 0);
  long long* fid = static_cast<long long*>(h->rr_fid.p);
  double* fsc = static_cast<double*>(h->rr_fsc.p);
  double* fa = static_cast<double*>(h->rr_fa.p);
  double* fb = static_cast<double*>(h->rr_fb.p);
  int* fcnt = static_cast<int*>(h->rr_fcnt.p);
  int rc = hybrid_local(h, 0, k, tie_mode, limit, kprime, k1, b, h->staged, h->pin_status, nullptr,
                        Fused{fid, fsc, fa, fb, fcnt, W});
  if (rc != RSE_OK) return rc;
  rr_mark(h, 1);

  // 2. pair assembly
  const int* qptr = static_cast<const int*>(h->rr_qptr.p);
  int* row = static_cast<int*>(h->rr_row.p);
  int2* ab = static_cast<int2*>(h->rr_ab.p);
  int* qpb = static_cast<int*>(h->rr_qpb.p);
  int* qtb = static_cast<int*>(h->rr_qtb.p);
  rerank_len_kernel<<<nq, kRrThreads, 0, h->stream>>>(fid, fcnt, W, h->rr_doc_ids, h->rr_n_docs, h->rr_doc_indptr, qptr,
                                                      max_length - 3, row, ab, static_cast<int*>(h->rr_qnp.p),
                                                      static_cast<int*>(h->rr_qnt.p), meta);
  LAUNCHED(h);
  rerank_scan_kernel<<<1, kRrScanThreads, 0, h->stream>>>(static_cast<const int*>(h->rr_qnp.p),
                                                          static_cast<const int*>(h->rr_qnt.p), nq, qpb, qtb, meta);
  LAUNCHED(h);
  // ids / type_ids are sized for the worst case of the batch (every union full, every pair as long as the longest
  // query and the longest document allow): their size is known before the step's one host round trip
  const size_t t_cap = static_cast<size_t>(P) * std::min<int64_t>(max_length, max_q + h->rr_max_doc_len + 3);
  ENSURE(h->rr_ids, 4 * t_cap); ENSURE(h->rr_types, 4 * t_cap);
  int* cu = meta + kRrMetaHead;
  int* ids = static_cast<int*>(h->rr_ids.p);
  int* types = static_cast<int*>(h->rr_types.p);
  rerank_pack_kernel<<<nq, kRrThreads, 0, h->stream>>>(fcnt, W, row, ab, qpb, qtb, qptr,
                                                       static_cast<const int*>(h->rr_qtok.p), h->rr_doc_indptr,
                                                       h->rr_doc_tok, cls_id, sep_id, cu, ids, types);
  LAUNCHED(h);
  rr_mark(h, 2);
  // THE host round trip of the step: the pair count, the missing-id flag and cu_seqlens, which the host needs to cut
  // the pairs into encoder slices of at most rr_budget tokens
  CK(cudaMemcpyAsync(h->rr_pin_meta, meta, 4 * meta_n, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(4 * meta_n);
  CK(cudaStreamSynchronize(h->stream));
  const int* hm = h->rr_pin_meta;
  if (hm[0] != 0) {
    const unsigned first = static_cast<unsigned>(hm[1]);
    long long id = -1;
    CK(cudaMemcpy(&id, fid + first, 8, cudaMemcpyDeviceToHost));
    return fail(h, RSE_ERR_STATE, "rse_hybrid_rerank_run: " + std::to_string(hm[0]) + " fused id(s) not in the document store, first " +
                                      std::to_string(id) + " (query " + std::to_string(first / W) + ")");
  }
  const int n_pairs = hm[2];
  const int* hcu = hm + kRrMetaHead;

  // 3. the cross-encoder, in slices of the token budget
  ENSURE(h->rr_logit, 4 * static_cast<size_t>(std::max(n_pairs, 1)));
  ENSURE(h->rr_cus, 4 * (static_cast<size_t>(n_pairs) + 1));
  float* logit = static_cast<float*>(h->rr_logit.p);
  int* cus = static_cast<int*>(h->rr_cus.p);
  for (int p0 = 0; p0 < n_pairs;) {
    int p1 = p0 + 1, max_len = hcu[p0 + 1] - hcu[p0];
    while (p1 < n_pairs && hcu[p1 + 1] - hcu[p0] <= h->rr_budget) {
      max_len = std::max(max_len, hcu[p1 + 1] - hcu[p1]);
      ++p1;
    }
    const int n = p1 - p0, T = hcu[p1] - hcu[p0];
    rerank_rebase_kernel<<<(n + 256) / 256, 256, 0, h->stream>>>(cu, p0, n, cus);
    LAUNCHED(h);
    rc = enc_forward(h, e, ids + hcu[p0], types + hcu[p0], cus, n, T, max_len, logit + p0);
    if (rc != RSE_OK) return rc;
    p0 = p1;
  }
  rr_mark(h, 3);

  // 4. the reference's reorder, [:limit], into one buffer for a single copy back
  const size_t n = static_cast<size_t>(nq) * limit;
  ENSURE(h->rr_pack, 32 * n + 4 * static_cast<size_t>(nq));
  char* pk = static_cast<char*>(h->rr_pack.p);
  rerank_order_kernel<<<nq, kRrThreads, 0, h->stream>>>(
      fid, fsc, fa, fb, fcnt, W, qpb, logit, activation, limit, reinterpret_cast<long long*>(pk),
      reinterpret_cast<double*>(pk + 8 * n), reinterpret_cast<float*>(pk + 16 * n), reinterpret_cast<int*>(pk + 20 * n),
      reinterpret_cast<int*>(pk + 24 * n), reinterpret_cast<int*>(pk + 28 * n), reinterpret_cast<int*>(pk + 32 * n));
  LAUNCHED(h);
  rr_mark(h, 4);
  h->rr_nq = nq; h->rr_limit = limit;
  return RSE_OK;
}

int rse_hybrid_rerank_fetch(rse_index* h, int32_t limit, int64_t* out_id, double* out_score, int32_t* out_bm25_rank,
                            int32_t* out_sem_rank, int32_t* out_rrf_rank, float* out_ce_score, int32_t* out_count) {
  if (!h) return RSE_ERR_INVALID;
  const int nq = h->rr_nq;
  if (nq <= 0) return fail(h, RSE_ERR_STATE, "rse_hybrid_rerank_fetch: no rerank run to fetch");
  if (limit != h->rr_limit) return fail(h, RSE_ERR_STATE, "rse_hybrid_rerank_fetch: limit differs from the last rse_hybrid_rerank_run");
  if (!out_id || !out_score || !out_bm25_rank || !out_sem_rank || !out_rrf_rank || !out_ce_score || !out_count)
    return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_fetch: bad arguments");
  const size_t n = static_cast<size_t>(nq) * limit;
  const size_t bytes = 32 * n + 4 * static_cast<size_t>(nq);
  CK(cudaSetDevice(h->device));
  if (h->rr_pin_out_bytes < bytes) {
    if (h->rr_pin_out) CK(cudaFreeHost(h->rr_pin_out));
    h->rr_pin_out = nullptr; h->rr_pin_out_bytes = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&h->rr_pin_out), bytes + bytes / 2));
    h->rr_pin_out_bytes = bytes + bytes / 2;
  }
  CK(cudaMemcpyAsync(h->rr_pin_out, h->rr_pack.p, bytes, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(bytes);
  CK(cudaStreamSynchronize(h->stream));
  const char* p = h->rr_pin_out;
  std::memcpy(out_id, p, 8 * n);
  std::memcpy(out_score, p + 8 * n, 8 * n);
  std::memcpy(out_ce_score, p + 16 * n, 4 * n);
  std::memcpy(out_bm25_rank, p + 20 * n, 4 * n);
  std::memcpy(out_sem_rank, p + 24 * n, 4 * n);
  std::memcpy(out_rrf_rank, p + 28 * n, 4 * n);
  std::memcpy(out_count, p + 32 * n, 4 * static_cast<size_t>(nq));
  return RSE_OK;
}

int rse_hybrid_rerank_timing(rse_index* h, float* out_ms) {
  if (!h) return RSE_ERR_INVALID;
  if (!out_ms) return fail(h, RSE_ERR_INVALID, "rse_hybrid_rerank_timing: bad arguments");
  if (!h->rr_timed || h->rr_nq <= 0)
    return fail(h, RSE_ERR_STATE, "rse_hybrid_rerank_timing: the last rerank run was not timed (rse_set_timing)");
  CK(cudaEventSynchronize(h->rr_ev[4]));
  for (int i = 0; i < 4; ++i) CK(cudaEventElapsedTime(&out_ms[i], h->rr_ev[i], h->rr_ev[i + 1]));
  return RSE_OK;
}

// ------------------------------------------------------------------ BERT WordPiece on the device (wordpiece.cuh)
int rse_tokenizer_load(rse_index* h, int32_t slot, const rse_wordpiece_desc* d) {
  if (!h) return RSE_ERR_INVALID;
  if (slot < 0 || slot >= RSE_MAX_TOKENIZERS || !d) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: bad arguments");
  const rse_wordpiece_desc& x = *d;
  if (!x.cp_map || !x.cp_class || !x.extra || x.n_extra < 1 || !x.node_first || !x.node_id || x.n_nodes < 2 ||
      x.n_added < 0 || (x.n_added > 0 && (!x.added || !x.added_offsets || !x.added_ids)))
    return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: a table is missing");
  if (x.n_added > kWpMaxAdded) return fail(h, RSE_ERR_UNSUPPORTED, "rse_tokenizer_load: more than 32 added tokens");
  if (x.max_input_chars_per_word < 1 || x.max_input_chars_per_word > kWpMaxWordChars)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_tokenizer_load: max_input_chars_per_word must be in [1, 256]");
  // every index the kernels follow is checked here, once
  const int n_nodes = x.n_nodes;
  if (x.node_first[0] != 0) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: node_first must start at 0");
  for (int i = 0; i < n_nodes; ++i)
    if (x.node_first[i + 1] < x.node_first[i]) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: node_first must not decrease");
  const int n_edges = x.node_first[n_nodes];
  if (n_edges > 0 && (!x.edge_cp || !x.edge_child)) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: edges missing");
  for (int i = 0; i < n_nodes; ++i)
    for (int j = x.node_first[i]; j < x.node_first[i + 1]; ++j)
      if (x.edge_child[j] < 2 || x.edge_child[j] >= n_nodes || (j > x.node_first[i] && x.edge_cp[j] <= x.edge_cp[j - 1]))
        return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: a trie edge is out of range or out of order");
  if (std::min({x.unk_id, x.cls_id, x.sep_id}) < 0) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: negative special id");
  for (int i = 0; i < n_nodes; ++i) {
    if (x.node_id[i] < -1) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: node_id below -1");
  }
  for (int i = 0; i < kWpCodePoints; ++i) {
    const uint32_t m = x.cp_map[i], c = (m >> 21) & 3, v = m & kWpCpMask;
    if ((m >> 24) || (c == 1 && v >= static_cast<uint32_t>(kWpCodePoints)) || (c > 1 && v >= static_cast<uint32_t>(x.n_extra)) ||
        x.cp_class[i] > kWpPunct)
      return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: code point map entry " + std::to_string(i) + " is out of range");
  }
  for (int64_t i = 0; i < 3ll * x.n_extra; ++i)
    if (x.extra[i] >= static_cast<uint32_t>(kWpCodePoints)) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: extra code point out of range");
  uint32_t first[8] = {};
  if (x.n_added > 0 && x.added_offsets[0] != 0) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: added_offsets must start at 0");
  for (int a = 0; a < x.n_added; ++a) {
    if (x.added_offsets[a + 1] <= x.added_offsets[a] || x.added_ids[a] < 0)
      return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load: an added token is empty or has a negative id");
    const uint8_t b = static_cast<uint8_t>(x.added[x.added_offsets[a]]);
    first[b >> 5] |= 1u << (b & 31);
  }
  const int n_added_bytes = x.n_added > 0 ? x.added_offsets[x.n_added] : 0;
  // one allocation: map | extra | cls | node_first | node_id | edge_cp | edge_child | added bytes | offsets | ids
  size_t off[11], at = 0;
  const size_t sz[10] = {4ull * kWpCodePoints, 12ull * x.n_extra, 1ull * kWpCodePoints, 4ull * (n_nodes + 1),
                         4ull * n_nodes, 4ull * n_edges, 4ull * n_edges, 1ull * n_added_bytes,
                         4ull * (x.n_added + 1), 4ull * x.n_added};
  for (int i = 0; i < 10; ++i) { off[i] = at; at += (sz[i] + 255) / 256 * 256; }
  off[10] = at;
  std::vector<char> host(at);
  const void* src[10] = {x.cp_map, x.extra, x.cp_class, x.node_first, x.node_id, x.edge_cp, x.edge_child, x.added,
                         x.added_offsets, x.added_ids};
  for (int i = 0; i < 10; ++i) if (sz[i] && src[i]) std::memcpy(host.data() + off[i], src[i], sz[i]);
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));                       // a tokenisation may still read the old tables
  auto& ts = h->tok[slot];
  if (ts.blob) CK(cudaFree(ts.blob));
  ts.blob = nullptr;
  ts.loaded = false;
  CK(cudaMalloc(&ts.blob, at));
  CK(cudaMemcpy(ts.blob, host.data(), at, cudaMemcpyHostToDevice));
  char* b = static_cast<char*>(ts.blob);
  WpTables& t = ts.t;
  t.map = reinterpret_cast<const uint32_t*>(b + off[0]);
  t.extra = reinterpret_cast<const uint32_t*>(b + off[1]);
  t.cls = reinterpret_cast<const uint8_t*>(b + off[2]);
  t.node_first = reinterpret_cast<const int32_t*>(b + off[3]);
  t.node_id = reinterpret_cast<const int32_t*>(b + off[4]);
  t.edge_cp = reinterpret_cast<const int32_t*>(b + off[5]);
  t.edge_child = reinterpret_cast<const int32_t*>(b + off[6]);
  t.added_bytes = reinterpret_cast<const uint8_t*>(b + off[7]);
  t.added_off = reinterpret_cast<const int32_t*>(b + off[8]);
  t.added_id = reinterpret_cast<const int32_t*>(b + off[9]);
  t.n_added = x.n_added;
  std::memcpy(t.added_first, first, sizeof(first));
  t.unk = x.unk_id; t.cls_id = x.cls_id; t.sep_id = x.sep_id; t.max_chars = x.max_input_chars_per_word;
  ts.bpe = false;
  ts.loaded = true;
  return RSE_OK;
}

// ------------------------------------------------------------------ CLIP byte-level BPE on the device (bpe.cuh)
int rse_tokenizer_load_bpe(rse_index* h, int32_t slot, const rse_bpe_desc* d) {
  if (!h) return RSE_ERR_INVALID;
  if (slot < 0 || slot >= RSE_MAX_TOKENIZERS || !d) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: bad arguments");
  const rse_bpe_desc& x = *d;
  if (!x.cp_map || !x.cp_class || !x.extra || x.n_extra < 1 || !x.byte_ids || !x.merges || x.n_added < 0 ||
      (x.n_added > 0 && (!x.added || !x.added_offsets || !x.added_ids)))
    return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: a table is missing");
  if (x.n_added > kWpMaxAdded) return fail(h, RSE_ERR_UNSUPPORTED, "rse_tokenizer_load_bpe: more than 32 added tokens");
  // every index the kernels follow is checked here, once
  if (x.merge_slots < 2 || (x.merge_slots & (x.merge_slots - 1)))
    return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: merge_slots must be a power of two >= 2");
  if (std::min(x.bos_id, x.eos_id) < 0) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: negative special id");
  for (int i = 0; i < 512; ++i)
    if (x.byte_ids[i] < 0) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: negative byte symbol id");
  int64_t empty = 0;
  for (int64_t i = 0; i < x.merge_slots; ++i) {
    const int32_t* m = x.merges + 4 * i;
    if (m[0] < 0) { ++empty; continue; }
    if (m[1] < 0 || m[2] < 0 || m[3] < 0)
      return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: merge slot " + std::to_string(i) + " holds a negative id or rank");
  }
  if (empty == 0) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: the merge table has no empty slot");
  for (int i = 0; i < kWpCodePoints; ++i) {
    const uint32_t m = x.cp_map[i], c = (m >> 21) & 3, v = m & kWpCpMask;
    if ((m >> 24) || (c == 1 && v >= static_cast<uint32_t>(kWpCodePoints)) || (c > 1 && v >= static_cast<uint32_t>(x.n_extra)) ||
        x.cp_class[i] > kBpeNumber)
      return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: code point map entry " + std::to_string(i) + " is out of range");
  }
  for (int64_t i = 0; i < 3ll * x.n_extra; ++i)
    if (x.extra[i] >= static_cast<uint32_t>(kWpCodePoints)) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: extra code point out of range");
  uint32_t first[8] = {};
  if (x.n_added > 0 && x.added_offsets[0] != 0) return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: added_offsets must start at 0");
  for (int a = 0; a < x.n_added; ++a) {
    if (x.added_offsets[a + 1] <= x.added_offsets[a] || x.added_ids[a] < 0)
      return fail(h, RSE_ERR_INVALID, "rse_tokenizer_load_bpe: an added token is empty or has a negative id");
    const uint8_t b = static_cast<uint8_t>(x.added[x.added_offsets[a]]);
    first[b >> 5] |= 1u << (b & 31);
  }
  const int n_added_bytes = x.n_added > 0 ? x.added_offsets[x.n_added] : 0;
  // one allocation: map | extra | cls | byte ids | merges | added bytes | offsets | ids
  size_t off[9], at = 0;
  const size_t sz[8] = {4ull * kWpCodePoints, 12ull * x.n_extra, 1ull * kWpCodePoints, 4ull * 512,
                        16ull * x.merge_slots, 1ull * n_added_bytes, 4ull * (x.n_added + 1), 4ull * x.n_added};
  for (int i = 0; i < 8; ++i) { off[i] = at; at += (sz[i] + 255) / 256 * 256; }
  off[8] = at;
  std::vector<char> host(at);
  const void* src[8] = {x.cp_map, x.extra, x.cp_class, x.byte_ids, x.merges, x.added, x.added_offsets, x.added_ids};
  for (int i = 0; i < 8; ++i) if (sz[i] && src[i]) std::memcpy(host.data() + off[i], src[i], sz[i]);
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));                       // a tokenisation may still read the old tables
  auto& ts = h->tok[slot];
  if (ts.blob) CK(cudaFree(ts.blob));
  ts.blob = nullptr;
  ts.loaded = false;
  CK(cudaMalloc(&ts.blob, at));
  CK(cudaMemcpy(ts.blob, host.data(), at, cudaMemcpyHostToDevice));
  char* b = static_cast<char*>(ts.blob);
  BpeTables& t = ts.bt;
  t.map = reinterpret_cast<const uint32_t*>(b + off[0]);
  t.extra = reinterpret_cast<const uint32_t*>(b + off[1]);
  t.cls = reinterpret_cast<const uint8_t*>(b + off[2]);
  t.byte_id = reinterpret_cast<const int32_t*>(b + off[3]);
  t.merges = reinterpret_cast<const int4*>(b + off[4]);
  t.merge_mask = static_cast<uint32_t>(x.merge_slots - 1);
  t.added_bytes = reinterpret_cast<const uint8_t*>(b + off[5]);
  t.added_off = reinterpret_cast<const int32_t*>(b + off[6]);
  t.added_id = reinterpret_cast<const int32_t*>(b + off[7]);
  t.n_added = x.n_added;
  std::memcpy(t.added_first, first, sizeof(first));
  t.bos_id = x.bos_id; t.eos_id = x.eos_id;
  ts.bpe = true;
  ts.loaded = true;
  return RSE_OK;
}

namespace {
// texts -> pinned -> device, the count pass and the scan, then THE small copy back of the call (meta, synchronises).
// Leaves the counts in tk_count and cu_seqlens in tk_cu64 / tk_cu32; *cap = pieces kept per text.
int tok_count_dev(rse_index* h, int32_t slot, int64_t n, int special, int cap, const std::string& w,
                  unsigned long long* meta);

int tok_count(rse_index* h, int32_t slot, const char* text, const int64_t* offs, int64_t n, int special, int max_length,
              const char* who, unsigned long long* meta, int* cap) {
  const std::string w(who);
  if (slot < 0 || slot >= RSE_MAX_TOKENIZERS) return fail(h, RSE_ERR_INVALID, w + ": tokenizer slot out of range");
  if (!h->tok[slot].loaded) return fail(h, RSE_ERR_STATE, w + ": no tokenizer in this slot (rse_tokenizer_load)");
  if (n < 1 || n > INT_MAX || !offs) return fail(h, RSE_ERR_INVALID, w + ": bad arguments (n < 1 or offsets NULL)");
  if (offs[0] != 0) return fail(h, RSE_ERR_INVALID, w + ": offsets must start at 0");
  for (int64_t i = 0; i < n; ++i)
    if (offs[i + 1] < offs[i]) return fail(h, RSE_ERR_INVALID, w + ": offsets must not decrease (at " + std::to_string(i) + ")");
  const int64_t bytes = offs[n];
  if (bytes > 0 && !text) return fail(h, RSE_ERR_INVALID, w + ": text is NULL");
  if (special && max_length > 0 && max_length < 2)
    return fail(h, RSE_ERR_UNSUPPORTED, w + ": max_length must be >= 2 with [CLS] / [SEP]");
  *cap = max_length > 0 ? max_length - 2 * special : INT_MAX;
  CK(cudaSetDevice(h->device));
  // every call ends in a synchronise after its uploads, so the pinned buffer is free again here
  const size_t ob = 8 * static_cast<size_t>(n + 1), need = ob + static_cast<size_t>(bytes);
  if (h->tk_pin_bytes < need) {
    if (h->tk_pin) CK(cudaFreeHost(h->tk_pin));
    h->tk_pin = nullptr; h->tk_pin_bytes = 0;
    CK(cudaMallocHost(reinterpret_cast<void**>(&h->tk_pin), need + need / 4 + 256));
    h->tk_pin_bytes = need + need / 4 + 256;
  }
  std::memcpy(h->tk_pin, offs, ob);
  if (bytes > 0) std::memcpy(h->tk_pin + ob, text, bytes);
  ENSURE(h->tk_offs, ob);
  ENSURE(h->tk_text, std::max<size_t>(bytes, 1));
  CK(cudaMemcpyAsync(h->tk_offs.p, h->tk_pin, ob, cudaMemcpyHostToDevice, h->stream));
  if (bytes > 0) CK(cudaMemcpyAsync(h->tk_text.p, h->tk_pin + ob, bytes, cudaMemcpyHostToDevice, h->stream));
  h->stats.h2d_bytes += static_cast<int64_t>(need);
  h->tk_src_text = static_cast<const uint8_t*>(h->tk_text.p);
  h->tk_src_offs = static_cast<const int64_t*>(h->tk_offs.p);
  return tok_count_dev(h, slot, n, special, *cap, w, meta);
}

// the count pass and the scan over the texts at tk_src_text / tk_src_offs (device), then THE small copy back of the
// call (meta, synchronises)
int tok_count_dev(rse_index* h, int32_t slot, int64_t n, int special, int cap, const std::string& w,
                  unsigned long long* meta) {
  ENSURE(h->tk_count, 4 * static_cast<size_t>(n));
  ENSURE(h->tk_cu64, 8 * static_cast<size_t>(n + 1));
  ENSURE(h->tk_cu32, 4 * static_cast<size_t>(n + 1));
  ENSURE(h->tk_meta, 8 * kWpMeta);
  if (!h->tk_pin_meta) CK(cudaMallocHost(reinterpret_cast<void**>(&h->tk_pin_meta), 8 * (kWpMeta + 1)));
  auto* dm = static_cast<unsigned long long*>(h->tk_meta.p);
  CK(cudaMemsetAsync(dm, 0, 8 * kWpMeta, h->stream));
  CK(cudaMemsetAsync(dm + 1, 0xFF, 8, h->stream));
  CK(cudaMemsetAsync(dm + 3, 0xFF, 8, h->stream));
  const int ni = static_cast<int>(n);
  const bool bpe = h->tok[slot].bpe;
  if (bpe)
    bpe_count_kernel<<<(ni + kWpThreads - 1) / kWpThreads, kWpThreads, 0, h->stream>>>(
        h->tok[slot].bt, h->tk_src_text, h->tk_src_offs, ni, special, cap, static_cast<int32_t*>(h->tk_count.p), dm);
  else
    wp_count_kernel<<<(ni + kWpThreads - 1) / kWpThreads, kWpThreads, 0, h->stream>>>(
        h->tok[slot].t, h->tk_src_text, h->tk_src_offs, ni, special, cap, static_cast<int32_t*>(h->tk_count.p), dm);
  LAUNCHED(h);
  wp_scan_kernel<<<1, kWpScanThreads, 0, h->stream>>>(static_cast<const int32_t*>(h->tk_count.p), ni,
                                                      static_cast<int64_t*>(h->tk_cu64.p),
                                                      static_cast<int32_t*>(h->tk_cu32.p), dm);
  LAUNCHED(h);
  CK(cudaMemcpyAsync(h->tk_pin_meta, dm, 8 * kWpMeta, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += 8 * kWpMeta;
  CK(cudaStreamSynchronize(h->stream));
  std::memcpy(meta, h->tk_pin_meta, 8 * kWpMeta);
  if (meta[0])
    return fail(h, RSE_ERR_INVALID, w + ": text " + std::to_string(meta[1]) + " is not well-formed UTF-8 (" +
                                        std::to_string(meta[0]) + " text(s))");
  if (meta[2] && bpe)
    return fail(h, RSE_ERR_UNSUPPORTED, w + ": text " + std::to_string(meta[3]) + " needs the host tokenizer (a code point "
                                        "NFC could join with its neighbours, or a piece longer than " +
                                        std::to_string(kBpeMaxWord) + " bytes before the cut; " + std::to_string(meta[2]) +
                                        " text(s))");
  if (meta[2])
    return fail(h, RSE_ERR_UNSUPPORTED, w + ": text " + std::to_string(meta[3]) + " holds combining marks of two code points "
                                        "that NFD's canonical reordering could move (" + std::to_string(meta[2]) +
                                        " text(s)); tokenize such texts on the host");
  if (meta[4] > static_cast<unsigned long long>(INT_MAX))
    return fail(h, RSE_ERR_UNSUPPORTED, w + ": more than 2^31 token ids in one call (split the batch)");
  h->tk_max_id = meta[6];
  return RSE_OK;
}

// the write pass of the texts tok_count uploaded, into ids (device, tk_cu64 positions)
int tok_write(rse_index* h, int32_t slot, int n, int special, int cap, int32_t* ids) {
  if (h->tok[slot].bpe)
    bpe_write_kernel<<<(n + kWpThreads - 1) / kWpThreads, kWpThreads, 0, h->stream>>>(
        h->tok[slot].bt, h->tk_src_text, h->tk_src_offs, n, special, cap, static_cast<const int64_t*>(h->tk_cu64.p), ids);
  else
    wp_write_kernel<<<(n + kWpThreads - 1) / kWpThreads, kWpThreads, 0, h->stream>>>(
        h->tok[slot].t, h->tk_src_text, h->tk_src_offs, n, special, cap, static_cast<const int64_t*>(h->tk_cu64.p), ids);
  LAUNCHED(h);
  return RSE_OK;
}

// tokenize ([CLS] ... [SEP], cut at max_length) into tk_ids, then the BERT slot on them: out_dev [n, hidden] / [n]
bool tok_is_bpe(const rse_index* h, int32_t slot) {
  return slot >= 0 && slot < RSE_MAX_TOKENIZERS && h->tok[slot].loaded && h->tok[slot].bpe;
}

// A CLIP text batch runs the tower in slices of at most this many tokens, greedy in text order (a text alone when it
// is longer): the slices GpuClipModel.encode_ids cuts by default, so both paths make the same launches.
constexpr int kClipTextTokensPerCall = 1 << 16;

// tokenize (bos ... eos, cut at max_length) into tk_ids, then the CLIP text tower on them, slice by slice:
// out_dev [n, projection_dim].  Only cu_seqlens comes to the host (the slices' bounds); the ids stay on the device.
int clip_enc_texts(rse_index* h, int32_t tok_slot, Encoder& e, const char* text, const int64_t* offs, int32_t n,
                   int32_t max_length, float* out_dev) {
  if (!e.clip || e.ccfg.tower != 1)
    return fail(h, RSE_ERR_INVALID, "rse_encode_texts: a BPE tokenizer feeds a CLIP text tower; the slot holds another encoder");
  if (!out_dev) return fail(h, RSE_ERR_INVALID, "rse_encode_texts: out is NULL");
  if (max_length < 2 || max_length > e.ccfg.max_positions)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_encode_texts: max_length must be in [2, max_positions]");
  unsigned long long m[kWpMeta];
  int cap = 0;
  int rc = tok_count(h, tok_slot, text, offs, n, 1, max_length, "rse_encode_texts", m, &cap);
  if (rc != RSE_OK) return rc;
  if (m[6] >= static_cast<unsigned long long>(e.ccfg.vocab_size))
    return fail(h, RSE_ERR_INVALID, "rse_encode_texts: token id " + std::to_string(m[6]) + " >= the encoder's vocab_size " +
                                        std::to_string(e.ccfg.vocab_size));
  const int T = static_cast<int>(m[4]);
  std::vector<int32_t> cu(static_cast<size_t>(n) + 1);
  CK(cudaMemcpy(cu.data(), h->tk_cu32.p, 4 * (static_cast<size_t>(n) + 1), cudaMemcpyDeviceToHost));   // (tok_count synchronised)
  h->stats.d2h_bytes += 4 * (static_cast<int64_t>(n) + 1);
  ENSURE(h->tk_ids, 4 * static_cast<size_t>(T));
  rc = tok_write(h, tok_slot, n, 1, cap, static_cast<int32_t*>(h->tk_ids.p));
  if (rc != RSE_OK) return rc;
  h->tk_n = n; h->tk_total = T;
  std::vector<int> bound{0};
  int t_max = 0, n_max = 0;
  for (int lo = 0; lo < n;) {
    int hi = lo + 1;
    while (hi < n && cu[hi + 1] - cu[lo] <= kClipTextTokensPerCall) ++hi;
    bound.push_back(hi);
    t_max = std::max(t_max, cu[hi] - cu[lo]);
    n_max = std::max(n_max, hi - lo);
    lo = hi;
  }
  rc = clip_buffers(h, e, t_max, e.mode == 0 && e.tc_ok);     // sized once for the largest slice
  if (rc != RSE_OK) return rc;
  ENSURE(e.ids, sizeof(int32_t) * t_max);
  ENSURE(e.cu, sizeof(int32_t) * (n_max + 1));
  const int proj = e.ccfg.projection_dim;
  for (size_t k = 0; k + 1 < bound.size(); ++k) {
    const int lo = bound[k], hi = bound[k + 1], ns = hi - lo, Ts = cu[hi] - cu[lo];
    int max_len = 1;
    for (int s = lo; s < hi; ++s) max_len = std::max(max_len, cu[s + 1] - cu[s]);
    CK(cudaMemcpyAsync(e.ids.p, static_cast<const int32_t*>(h->tk_ids.p) + cu[lo], sizeof(int32_t) * Ts,
                       cudaMemcpyDeviceToDevice, h->stream));
    bpe_rebase_kernel<<<(ns + 256) / 256, 256, 0, h->stream>>>(static_cast<const int32_t*>(h->tk_cu32.p) + lo, ns,
                                                               static_cast<int32_t*>(e.cu.p));
    LAUNCHED(h);
    e.max_len = max_len;
    rc = clip_text_forward(h, e, ns, Ts, out_dev + static_cast<size_t>(lo) * proj);
    if (rc != RSE_OK) return rc;
  }
  return RSE_OK;
}

int enc_texts(rse_index* h, int32_t tok_slot, int32_t enc_slot, const char* text, const int64_t* offs, int32_t n,
              int32_t max_length, float* out_dev) {
  h->tk_n = 0;
  int rc = enc_check(h, enc_slot, true);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[enc_slot];
  if (tok_is_bpe(h, tok_slot)) return clip_enc_texts(h, tok_slot, e, text, offs, n, max_length, out_dev);
  if (e.clip) return fail(h, RSE_ERR_INVALID, "rse_encode_texts: the slot holds a CLIP tower (its tokenizer is not WordPiece)");
  if (!out_dev) return fail(h, RSE_ERR_INVALID, "rse_encode_texts: out is NULL");
  if (max_length < 2 || max_length > e.cfg.max_positions)
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_encode_texts: max_length must be in [2, max_positions]");
  unsigned long long m[kWpMeta];
  int cap = 0;
  rc = tok_count(h, tok_slot, text, offs, n, 1, max_length, "rse_encode_texts", m, &cap);
  if (rc != RSE_OK) return rc;
  if (m[6] >= static_cast<unsigned long long>(e.cfg.vocab_size))
    return fail(h, RSE_ERR_INVALID, "rse_encode_texts: token id " + std::to_string(m[6]) + " >= the encoder's vocab_size " +
                                        std::to_string(e.cfg.vocab_size));
  const int T = static_cast<int>(m[4]);
  ENSURE(h->tk_ids, 4 * static_cast<size_t>(T));
  rc = tok_write(h, tok_slot, n, 1, cap, static_cast<int32_t*>(h->tk_ids.p));
  if (rc != RSE_OK) return rc;
  h->tk_n = n; h->tk_total = T;
  return enc_forward(h, e, static_cast<const int32_t*>(h->tk_ids.p), nullptr, static_cast<const int32_t*>(h->tk_cu32.p), n,
                     T, static_cast<int>(m[5]), out_dev);
}
}  // namespace

int rse_tokenize(rse_index* h, int32_t slot, const char* text, const int64_t* offsets, int32_t n, int32_t add_special,
                 int32_t max_length, int64_t* out_total, int32_t* out_max_len) {
  if (!h) return RSE_ERR_INVALID;
  h->tk_n = 0;
  if (add_special != 0 && add_special != 1) return fail(h, RSE_ERR_INVALID, "rse_tokenize: add_special must be 0 or 1");
  unsigned long long m[kWpMeta];
  int cap = 0;
  int rc = tok_count(h, slot, text, offsets, n, add_special, max_length, "rse_tokenize", m, &cap);
  if (rc != RSE_OK) return rc;
  ENSURE(h->tk_ids, 4 * std::max<size_t>(m[4], 1));
  rc = tok_write(h, slot, n, add_special, cap, static_cast<int32_t*>(h->tk_ids.p));
  if (rc != RSE_OK) return rc;
  h->tk_n = n; h->tk_total = static_cast<int64_t>(m[4]);
  if (out_total) *out_total = h->tk_total;
  if (out_max_len) *out_max_len = static_cast<int32_t>(m[5]);
  return RSE_OK;
}

int rse_tokens_fetch(rse_index* h, int32_t* ids_host, int32_t* cu_seqlens_host) {
  if (!h) return RSE_ERR_INVALID;
  if (h->tk_n < 1) return fail(h, RSE_ERR_STATE, "rse_tokens_fetch: nothing tokenized (rse_tokenize)");
  if (!cu_seqlens_host || (h->tk_total > 0 && !ids_host)) return fail(h, RSE_ERR_INVALID, "rse_tokens_fetch: bad arguments");
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(cu_seqlens_host, h->tk_cu32.p, 4 * static_cast<size_t>(h->tk_n + 1), cudaMemcpyDeviceToHost, h->stream));
  if (h->tk_total > 0)
    CK(cudaMemcpyAsync(ids_host, h->tk_ids.p, 4 * static_cast<size_t>(h->tk_total), cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += 4 * static_cast<int64_t>(h->tk_n + 1 + h->tk_total);
  CK(cudaStreamSynchronize(h->stream));
  return RSE_OK;
}

int rse_tokens_fetch_dev(rse_index* h, int32_t* ids_dev, int32_t* cu_seqlens_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (h->tk_n < 1) return fail(h, RSE_ERR_STATE, "rse_tokens_fetch_dev: nothing tokenized (rse_tokenize)");
  if (!cu_seqlens_dev || (h->tk_total > 0 && !ids_dev)) return fail(h, RSE_ERR_INVALID, "rse_tokens_fetch_dev: bad arguments");
  CK(cudaSetDevice(h->device));
  CK(cudaMemcpyAsync(cu_seqlens_dev, h->tk_cu32.p, 4 * static_cast<size_t>(h->tk_n + 1), cudaMemcpyDeviceToDevice, h->stream));
  if (h->tk_total > 0)
    CK(cudaMemcpyAsync(ids_dev, h->tk_ids.p, 4 * static_cast<size_t>(h->tk_total), cudaMemcpyDeviceToDevice, h->stream));
  return RSE_OK;
}

namespace {
// offsets_dev[0 .. n] of a device text of text_bytes bytes, checked on the device (one small copy back, synchronises)
int check_dev_offsets(rse_index* h, const std::string& w, const int64_t* offsets_dev, int64_t n, int64_t text_bytes) {
  ENSURE(h->ck_meta, 8);
  if (!h->tk_pin_meta) CK(cudaMallocHost(reinterpret_cast<void**>(&h->tk_pin_meta), 8 * (kWpMeta + 1)));
  auto* bad = static_cast<unsigned long long*>(h->ck_meta.p);
  CK(cudaMemsetAsync(bad, 0xFF, 8, h->stream));
  dev_offsets_check_kernel<<<static_cast<unsigned>((n + 256) / 256), 256, 0, h->stream>>>(offsets_dev, n, text_bytes, bad);
  LAUNCHED(h);
  CK(cudaMemcpyAsync(h->tk_pin_meta, bad, 8, cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  if (h->tk_pin_meta[0] != ~0ull)
    return fail(h, RSE_ERR_INVALID, w + ": offsets[" + std::to_string(h->tk_pin_meta[0]) + "] is out of order or outside "
                                        "the text (offsets must go from 0 up to at most text_bytes)");
  return RSE_OK;
}

int chunk_args(rse_index* h, const std::string& w, const char* text_dev, int64_t text_bytes, const int64_t* offsets_dev,
               int32_t n_movies, int32_t max_chunk_size) {
  if (max_chunk_size < 1) return fail(h, RSE_ERR_INVALID, w + ": max_chunk_size must be >= 1");
  if (n_movies < 1 || !offsets_dev || text_bytes < 0 || (text_bytes > 0 && !text_dev))
    return fail(h, RSE_ERR_INVALID, w + ": bad arguments (n_movies < 1, offsets or text NULL, or text_bytes < 0)");
  CK(cudaSetDevice(h->device));
  return check_dev_offsets(h, w, offsets_dev, 2 * static_cast<int64_t>(n_movies), text_bytes);
}

int chunk_carry(int32_t size, int32_t overlap) { return overlap > 0 && overlap < size ? overlap : 0; }
}  // namespace

int rse_tokenize_dev(rse_index* h, int32_t slot, const char* text_dev, int64_t text_bytes, const int64_t* offsets_dev,
                     int32_t n, int32_t add_special, int32_t max_length, int64_t* out_total, int32_t* out_max_len) {
  if (!h) return RSE_ERR_INVALID;
  h->tk_n = 0;
  const std::string w("rse_tokenize_dev");
  if (add_special != 0 && add_special != 1) return fail(h, RSE_ERR_INVALID, w + ": add_special must be 0 or 1");
  if (slot < 0 || slot >= RSE_MAX_TOKENIZERS) return fail(h, RSE_ERR_INVALID, w + ": tokenizer slot out of range");
  if (!h->tok[slot].loaded) return fail(h, RSE_ERR_STATE, w + ": no tokenizer in this slot (rse_tokenizer_load)");
  if (n < 1 || !offsets_dev || text_bytes < 0 || (text_bytes > 0 && !text_dev))
    return fail(h, RSE_ERR_INVALID, w + ": bad arguments (n < 1, offsets or text NULL, or text_bytes < 0)");
  if (add_special && max_length > 0 && max_length < 2)
    return fail(h, RSE_ERR_UNSUPPORTED, w + ": max_length must be >= 2 with [CLS] / [SEP]");
  const int cap = max_length > 0 ? max_length - 2 * add_special : INT_MAX;
  CK(cudaSetDevice(h->device));
  int rc = check_dev_offsets(h, w, offsets_dev, n, text_bytes);
  if (rc != RSE_OK) return rc;
  h->tk_src_text = reinterpret_cast<const uint8_t*>(text_dev);
  h->tk_src_offs = offsets_dev;
  unsigned long long m[kWpMeta];
  rc = tok_count_dev(h, slot, n, add_special, cap, w, m);
  if (rc != RSE_OK) return rc;
  ENSURE(h->tk_ids, 4 * std::max<size_t>(m[4], 1));
  rc = tok_write(h, slot, n, add_special, cap, static_cast<int32_t*>(h->tk_ids.p));
  if (rc != RSE_OK) return rc;
  h->tk_n = n; h->tk_total = static_cast<int64_t>(m[4]);
  if (out_total) *out_total = h->tk_total;
  if (out_max_len) *out_max_len = static_cast<int32_t>(m[5]);
  return RSE_OK;
}

int rse_encode_tokens_dev(rse_index* h, int32_t enc_slot, int64_t max_tokens_per_call, float* out_dev) {
  if (!h) return RSE_ERR_INVALID;
  const std::string w("rse_encode_tokens_dev");
  int rc = enc_check(h, enc_slot, true);
  if (rc != RSE_OK) return rc;
  Encoder& e = h->enc[enc_slot];
  if (e.clip || e.cfg.head != 0) return fail(h, RSE_ERR_INVALID, w + ": the slot does not hold a sentence encoder (head 0)");
  if (h->tk_n < 1) return fail(h, RSE_ERR_STATE, w + ": nothing tokenized (rse_tokenize / rse_tokenize_dev)");
  if (!out_dev || max_tokens_per_call < 1) return fail(h, RSE_ERR_INVALID, w + ": bad arguments");
  if (h->tk_max_id >= static_cast<unsigned long long>(e.cfg.vocab_size))
    return fail(h, RSE_ERR_INVALID, w + ": token id " + std::to_string(h->tk_max_id) + " >= the encoder's vocab_size " +
                                        std::to_string(e.cfg.vocab_size));
  const int n = h->tk_n;
  CK(cudaSetDevice(h->device));
  std::vector<int32_t> cu(static_cast<size_t>(n) + 1);
  CK(cudaMemcpyAsync(cu.data(), h->tk_cu32.p, 4 * (static_cast<size_t>(n) + 1), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->stats.d2h_bytes += 4 * (static_cast<int64_t>(n) + 1);
  for (int s = 0; s < n; ++s) {
    const int len = cu[s + 1] - cu[s];
    if (len < 1) return fail(h, RSE_ERR_INVALID, w + ": text " + std::to_string(s) + " has no ids (tokenize with add_special 1)");
    if (len > e.cfg.max_positions)
      return fail(h, RSE_ERR_UNSUPPORTED, w + ": text " + std::to_string(s) + " is longer than max_positions (tokenize with max_length)");
  }
  // slices of at most max_tokens_per_call tokens, greedy in text order at the real lengths (a text alone when it is
  // longer): GpuSentenceEncoder.encode's cut, which does not change any row (every kernel of the encoder works per
  // token or per sequence)
  int n_max = 0;
  std::vector<int> bound{0};
  for (int lo = 0; lo < n;) {
    int hi = lo + 1;
    while (hi < n && static_cast<int64_t>(cu[hi + 1]) - cu[lo] <= max_tokens_per_call) ++hi;
    bound.push_back(hi);
    n_max = std::max(n_max, hi - lo);
    lo = hi;
  }
  ENSURE(e.cu, sizeof(int32_t) * (n_max + 1));
  const int H = e.cfg.hidden;
  for (size_t k = 0; k + 1 < bound.size(); ++k) {
    const int lo = bound[k], hi = bound[k + 1], ns = hi - lo, Ts = cu[hi] - cu[lo];
    int max_len = 1;
    for (int s = lo; s < hi; ++s) max_len = std::max(max_len, cu[s + 1] - cu[s]);
    bpe_rebase_kernel<<<(ns + 256) / 256, 256, 0, h->stream>>>(static_cast<const int32_t*>(h->tk_cu32.p) + lo, ns,
                                                               static_cast<int32_t*>(e.cu.p));
    LAUNCHED(h);
    rc = enc_forward(h, e, static_cast<const int32_t*>(h->tk_ids.p) + cu[lo], nullptr, static_cast<const int32_t*>(e.cu.p),
                     ns, Ts, max_len, out_dev + static_cast<size_t>(lo) * H);
    if (rc != RSE_OK) return rc;
  }
  return RSE_OK;
}

int rse_chunk_count(rse_index* h, const char* text_dev, int64_t text_bytes, const int64_t* offsets_dev, int32_t n_movies,
                    int32_t max_chunk_size, int32_t overlap, int64_t* chunk_cu_dev, int64_t* byte_cu_dev,
                    int64_t* out_n_chunks, int64_t* out_n_bytes) {
  if (!h) return RSE_ERR_INVALID;
  int rc = chunk_args(h, "rse_chunk_count", text_dev, text_bytes, offsets_dev, n_movies, max_chunk_size);
  if (rc != RSE_OK) return rc;
  if (!chunk_cu_dev || !byte_cu_dev) return fail(h, RSE_ERR_INVALID, "rse_chunk_count: chunk_cu / byte_cu NULL");
  const int64_t n = n_movies;
  ENSURE(h->ck_chunks, 4 * static_cast<size_t>(n));
  ENSURE(h->ck_bytes, 4 * static_cast<size_t>(n));
  ENSURE(h->ck_cu32, 4 * static_cast<size_t>(n + 1));
  ENSURE(h->ck_meta, 8 * (kChunkMeta + 2 * kWpMeta));
  auto* dm = static_cast<unsigned long long*>(h->ck_meta.p);
  CK(cudaMemsetAsync(dm, 0, 8 * (kChunkMeta + 2 * kWpMeta), h->stream));
  CK(cudaMemsetAsync(dm + 1, 0xFF, 8, h->stream));
  const auto* t = reinterpret_cast<const uint8_t*>(text_dev);
  const int grid = static_cast<int>((n + kChunkThreads - 1) / kChunkThreads);
  chunk_count_kernel<<<grid, kChunkThreads, 0, h->stream>>>(t, offsets_dev, n_movies, max_chunk_size,
                                                            chunk_carry(max_chunk_size, overlap),
                                                            static_cast<int32_t*>(h->ck_chunks.p),
                                                            static_cast<int32_t*>(h->ck_bytes.p), dm);
  LAUNCHED(h);
  wp_scan_kernel<<<1, kWpScanThreads, 0, h->stream>>>(static_cast<const int32_t*>(h->ck_chunks.p), n_movies, chunk_cu_dev,
                                                      static_cast<int32_t*>(h->ck_cu32.p), dm + kChunkMeta);
  LAUNCHED(h);
  wp_scan_kernel<<<1, kWpScanThreads, 0, h->stream>>>(static_cast<const int32_t*>(h->ck_bytes.p), n_movies, byte_cu_dev,
                                                      static_cast<int32_t*>(h->ck_cu32.p), dm + kChunkMeta + kWpMeta);
  LAUNCHED(h);
  unsigned long long m[kChunkMeta + 2 * kWpMeta];
  CK(cudaMemcpyAsync(m, dm, sizeof(m), cudaMemcpyDeviceToHost, h->stream));
  CK(cudaStreamSynchronize(h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(sizeof(m));
  if (m[0])
    return fail(h, RSE_ERR_UNSUPPORTED, "rse_chunk_count: movie " + std::to_string(m[1]) + " has more than 2^31 bytes of "
                                        "chunk text (" + std::to_string(m[0]) + " movie(s))");
  if (out_n_chunks) *out_n_chunks = static_cast<int64_t>(m[kChunkMeta + 4]);
  if (out_n_bytes) *out_n_bytes = static_cast<int64_t>(m[kChunkMeta + kWpMeta + 4]);
  return RSE_OK;
}

int rse_chunk_write(rse_index* h, const char* text_dev, int64_t text_bytes, const int64_t* offsets_dev, int32_t n_movies,
                    int32_t max_chunk_size, int32_t overlap, const int64_t* chunk_cu_dev, const int64_t* byte_cu_dev,
                    int32_t movie_base, char* out_text_dev, int64_t* out_offsets_dev, int32_t* out_movie_dev,
                    int32_t* out_index_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!chunk_cu_dev || !byte_cu_dev || !out_offsets_dev || !out_movie_dev || !out_index_dev || !out_text_dev)
    return fail(h, RSE_ERR_INVALID, "rse_chunk_write: an output or a scan is NULL");
  if (movie_base < 0 || static_cast<int64_t>(movie_base) + n_movies > INT_MAX)
    return fail(h, RSE_ERR_INVALID, "rse_chunk_write: movie_base + n_movies must fit 31 bits");
  int rc = chunk_args(h, "rse_chunk_write", text_dev, text_bytes, offsets_dev, n_movies, max_chunk_size);
  if (rc != RSE_OK) return rc;
  const int grid = (n_movies + kChunkThreads - 1) / kChunkThreads;
  chunk_write_kernel<<<grid, kChunkThreads, 0, h->stream>>>(
      reinterpret_cast<const uint8_t*>(text_dev), offsets_dev, n_movies, max_chunk_size, chunk_carry(max_chunk_size, overlap),
      chunk_cu_dev, byte_cu_dev, movie_base, reinterpret_cast<uint8_t*>(out_text_dev), out_offsets_dev, out_movie_dev,
      out_index_dev);
  LAUNCHED(h);
  return RSE_OK;
}

int rse_encode_texts_dev(rse_index* h, int32_t tok_slot, int32_t enc_slot, const char* text, const int64_t* offsets,
                         int32_t n, int32_t max_length, float* out_dev) {
  if (!h) return RSE_ERR_INVALID;
  return enc_texts(h, tok_slot, enc_slot, text, offsets, n, max_length, out_dev);
}

int rse_encode_texts(rse_index* h, int32_t tok_slot, int32_t enc_slot, const char* text, const int64_t* offsets,
                     int32_t n, int32_t max_length, float* out_host) {
  if (!h) return RSE_ERR_INVALID;
  int rc = enc_check(h, enc_slot, true);
  if (rc != RSE_OK) return rc;
  if (!out_host || n < 1) return fail(h, RSE_ERR_INVALID, "rse_encode_texts: bad arguments");
  Encoder& e = h->enc[enc_slot];
  const bool bpe = tok_is_bpe(h, tok_slot);
  if (bpe && (!e.clip || e.ccfg.tower != 1))
    return fail(h, RSE_ERR_INVALID, "rse_encode_texts: a BPE tokenizer feeds a CLIP text tower; the slot holds another encoder");
  if (!bpe && e.clip) return fail(h, RSE_ERR_INVALID, "rse_encode_texts: the slot holds a CLIP tower (its tokenizer is not WordPiece)");
  const size_t n_out = static_cast<size_t>(n) * (bpe ? e.ccfg.projection_dim : e.cfg.head == 0 ? e.cfg.hidden : 1);
  CK(cudaSetDevice(h->device));
  ENSURE(e.out, sizeof(float) * n_out);
  rc = enc_texts(h, tok_slot, enc_slot, text, offsets, n, max_length, static_cast<float*>(e.out.p));
  if (rc != RSE_OK) return rc;
  CK(cudaMemcpyAsync(out_host, e.out.p, sizeof(float) * n_out, cudaMemcpyDeviceToHost, h->stream));
  h->stats.d2h_bytes += static_cast<int64_t>(sizeof(float) * n_out);
  CK(cudaStreamSynchronize(h->stream));
  return RSE_OK;
}

int rse_rerank_docs_load_texts(rse_index* h, int32_t tok_slot, const int64_t* ids, int64_t n_docs, const char* text,
                               const int64_t* offsets) {
  if (!h) return RSE_ERR_INVALID;
  h->tk_n = 0;
  if (n_docs < 1 || n_docs > INT_MAX || !ids) return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load_texts: bad arguments");
  for (int64_t i = 1; i < n_docs; ++i)
    if (ids[i] <= ids[i - 1])
      return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load_texts: ids must be strictly ascending (at " + std::to_string(i) + ")");
  if (tok_is_bpe(h, tok_slot))
    return fail(h, RSE_ERR_INVALID, "rse_rerank_docs_load_texts: the slot holds a BPE tokenizer (the cross-encoder's is WordPiece)");
  unsigned long long m[kWpMeta];
  int cap = 0;
  int rc = tok_count(h, tok_slot, text, offsets, n_docs, 0, 0, "rse_rerank_docs_load_texts", m, &cap);
  if (rc != RSE_OK) return rc;
  const int64_t n_tok = static_cast<int64_t>(m[4]);
  free_ptr(h->rr_doc_ids); free_ptr(h->rr_doc_indptr); free_ptr(h->rr_doc_tok);   // (tok_count synchronised)
  h->rr_n_docs = 0; h->rr_max_tok = -1;
  CK(cudaMalloc(&h->rr_doc_ids, 8 * n_docs));
  CK(cudaMalloc(&h->rr_doc_indptr, 8 * (n_docs + 1)));
  CK(cudaMalloc(&h->rr_doc_tok, 4 * std::max<int64_t>(n_tok, 1)));
  CK(cudaMemcpy(h->rr_doc_ids, ids, 8 * n_docs, cudaMemcpyHostToDevice));
  CK(cudaMemcpyAsync(h->rr_doc_indptr, h->tk_cu64.p, 8 * (n_docs + 1), cudaMemcpyDeviceToDevice, h->stream));
  rc = tok_write(h, tok_slot, static_cast<int>(n_docs), 0, cap, h->rr_doc_tok);
  if (rc != RSE_OK) return rc;
  CK(cudaStreamSynchronize(h->stream));
  h->rr_n_docs = n_docs; h->rr_max_tok = n_tok > 0 ? static_cast<int32_t>(m[6]) : -1;
  h->rr_max_doc_len = static_cast<int64_t>(m[5]);
  // a store load is a one-off bulk upload: give its staging back instead of keeping ~1 KB per document in HBM and
  // pinned memory
  for (DevBuf* b : {&h->tk_text, &h->tk_offs, &h->tk_count, &h->tk_cu64, &h->tk_cu32}) free_buf(*b);
  if (h->tk_pin) CK(cudaFreeHost(h->tk_pin));
  h->tk_pin = nullptr; h->tk_pin_bytes = 0;
  return RSE_OK;
}

// ------------------------------------------------------------------ multi-GPU (library-owned NCCL communicator)
#define NCK(call)                                                                                     \
  do {                                                                                                \
    ncclResult_t r__ = (call);                                                                        \
    if (r__ != ncclSuccess)                                                                           \
      return fail(h, RSE_ERR_CUDA, std::string(#call) + ": " + nccl_api()->GetErrorString(r__));      \
  } while (0)

int rse_comm_unique_id(uint8_t* out_id) {
  rse_index* h = nullptr;
  if (!out_id) return fail(h, RSE_ERR_INVALID, "rse_comm_unique_id: out_id is NULL");
  NcclApi* n = nccl_api();
  if (!n) return fail(h, RSE_ERR_UNSUPPORTED, "NCCL unavailable (set RSE_NCCL_LIB to libnccl.so.2)");
  ncclUniqueId id;
  NCK(n->GetUniqueId(&id));
  static_assert(sizeof(id) == RSE_COMM_ID_BYTES, "ncclUniqueId size");
  std::memcpy(out_id, &id, sizeof(id));
  return RSE_OK;
}

int rse_comm_init(rse_index* h, const uint8_t* id_bytes, int32_t n_ranks, int32_t rank) {
  if (!h) return RSE_ERR_INVALID;
  if (!id_bytes || n_ranks < 1 || rank < 0 || rank >= n_ranks) return fail(h, RSE_ERR_INVALID, "rse_comm_init: bad arguments");
  NcclApi* n = nccl_api();
  if (!n) return fail(h, RSE_ERR_UNSUPPORTED, "NCCL unavailable (set RSE_NCCL_LIB to libnccl.so.2)");
  CK(cudaSetDevice(h->device));
  if (h->comm) { n->CommDestroy(h->comm); h->comm = nullptr; }
  ncclUniqueId id;
  std::memcpy(&id, id_bytes, sizeof(id));
  NCK(n->CommInitRank(&h->comm, n_ranks, id, rank));
  h->comm_ranks = n_ranks; h->comm_rank = rank;
  return RSE_OK;
}

int rse_comm_destroy(rse_index* h) {
  if (!h) return RSE_ERR_INVALID;
  if (h->comm) {
    CK(cudaSetDevice(h->device));
    CK(cudaStreamSynchronize(h->stream));
    NCK(nccl_api()->CommDestroy(h->comm));
    h->comm = nullptr;
  }
  h->comm_ranks = 1; h->comm_rank = 0;
  return RSE_OK;
}

int rse_comm_info(rse_index* h, int32_t* n_ranks, int32_t* rank, int32_t* nccl_version) {
  if (!h) return RSE_ERR_INVALID;
  if (n_ranks) *n_ranks = h->comm ? h->comm_ranks : 0;
  if (rank) *rank = h->comm ? h->comm_rank : 0;
  if (nccl_version) {
    *nccl_version = 0;
    if (NcclApi* n = nccl_api()) { int v = 0; if (n->GetVersion(&v) == ncclSuccess) *nccl_version = v; }
  }
  return RSE_OK;
}

namespace {

// all-to-all by query slice: rank r receives, from every shard, the candidates of ITS queries.
// cand [nq, kprime, 3] (this shard, all queries) -> mine [n_ranks, ns, kprime, 3]
int comm_exchange(rse_index* h, const long long* cand, int nq, int kprime, long long* mine) {
  if (!h->comm) return fail(h, RSE_ERR_STATE, "no communicator: call rse_comm_init first");
  NcclApi* n = nccl_api();
  const int R = h->comm_ranks, me = h->comm_rank;
  const size_t per = static_cast<size_t>(kprime) * 3;
  const int ns = query_slice(nq, R, me + 1) - query_slice(nq, R, me);
  NCK(n->GroupStart());
  for (int r = 0; r < R; ++r) {
    const int lo = query_slice(nq, R, r), hi = query_slice(nq, R, r + 1);
    if (hi > lo) NCK(n->Send(cand + static_cast<size_t>(lo) * per, static_cast<size_t>(hi - lo) * per, ncclInt64, r, h->comm, h->stream));
    if (ns > 0) NCK(n->Recv(mine + static_cast<size_t>(r) * ns * per, static_cast<size_t>(ns) * per, ncclInt64, r, h->comm, h->stream));
  }
  NCK(n->GroupEnd());
  return RSE_OK;
}

}  // namespace

int rse_comm_exchange_candidates_dev(rse_index* h, const int64_t* cand_dev, int32_t nq, int32_t kprime, int64_t* mine_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!cand_dev || !mine_dev || nq < 1 || kprime < 1) return fail(h, RSE_ERR_INVALID, "rse_comm_exchange_candidates_dev: bad arguments");
  CK(cudaSetDevice(h->device));
  return comm_exchange(h, reinterpret_cast<const long long*>(cand_dev), nq, kprime, reinterpret_cast<long long*>(mine_dev));
}

int rse_comm_allgather_dev(rse_index* h, const void* send_dev, void* recv_dev, int64_t bytes_per_rank) {
  if (!h) return RSE_ERR_INVALID;
  if (!send_dev || !recv_dev || bytes_per_rank < 0) return fail(h, RSE_ERR_INVALID, "rse_comm_allgather_dev: bad arguments");
  if (!h->comm) return fail(h, RSE_ERR_STATE, "no communicator: call rse_comm_init first");
  CK(cudaSetDevice(h->device));
  NCK(nccl_api()->AllGather(send_dev, recv_dev, static_cast<size_t>(bytes_per_rank), ncclUint8, h->comm, h->stream));
  return RSE_OK;
}

namespace {

// local top-K' of ALL queries on this shard (+ deferred flag count or blocking exact fallback) + exchange:
// leaves [n_ranks, ns, kprime, 3] in h->sh_mine.  `bm25`: the slice's BM25, started underneath the filter pass when
// the tensor-core path runs, else on the main stream behind the KNN.
int sharded_knn_exchange(rse_index* h, const float* q_all_dev, int nq_all, int kprime, int32_t* flagged_dev,
                         Bm25Job* bm25) {
  if (!h->comm) return fail(h, RSE_ERR_STATE, "no communicator: call rse_comm_init first");
  const int R = h->comm_ranks, me = h->comm_rank;
  const int ns = query_slice(nq_all, R, me + 1) - query_slice(nq_all, R, me);
  const size_t per = static_cast<size_t>(kprime) * 3;
  ENSURE(h->sh_cand, sizeof(long long) * static_cast<size_t>(nq_all) * per);
  ENSURE(h->sh_mine, sizeof(long long) * static_cast<size_t>(R) * std::max(ns, 1) * per);
  PendingKnn pend;
  int rc = knn_local_begin(h, q_all_dev, nq_all, kprime, static_cast<long long*>(h->sh_cand.p), h->pin_status, bm25,
                           pend);
  if (rc != RSE_OK) return rc;
  if (bm25 && !bm25->enqueued) {
    rc = bm25_run(h, *bm25->in, bm25->in->nq, bm25->k, bm25->k1, bm25->b, h->stream, false);
    if (rc != RSE_OK) return rc;
  }
  if (pend.flags && flagged_dev) {                           // no host round trip: count the unfinished queries
    knn_flag_count_kernel<<<1, 256, 0, h->stream>>>(static_cast<const int*>(h->tc_status.p), pend.nq, flagged_dev);
    LAUNCHED(h);
  } else {
    rc = knn_local_finish(h, pend);                          // blocking, exact (flagged queries -> exact scan)
    if (rc != RSE_OK) return rc;
  }
  return comm_exchange(h, static_cast<const long long*>(h->sh_cand.p), nq_all, kprime, static_cast<long long*>(h->sh_mine.p));
}

}  // namespace

int rse_knn_sharded_dev(rse_index* h, const float* q_all_dev, int32_t nq_all, int32_t k, int32_t kprime, float* out_dist_dev,
                        int64_t* out_chunk_rowid_dev, int32_t* out_movie_idx_dev, int32_t* out_count_dev,
                        int32_t* flagged_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!q_all_dev || nq_all < 1 || k < 1 || kprime < 1) return fail(h, RSE_ERR_INVALID, "rse_knn_sharded_dev: bad arguments");
  if (!h->emb || !h->movie_idx) return fail(h, RSE_ERR_STATE, "rse_knn_sharded_dev: needs embeddings with movie_idx");
  CK(cudaSetDevice(h->device));
  int rc = sharded_knn_exchange(h, q_all_dev, nq_all, kprime, flagged_dev, nullptr);
  if (rc != RSE_OK) return rc;
  const int ns = query_slice(nq_all, h->comm_ranks, h->comm_rank + 1) - query_slice(nq_all, h->comm_ranks, h->comm_rank);
  if (ns == 0) return RSE_OK;
  if (!out_dist_dev || !out_chunk_rowid_dev || !out_movie_idx_dev || !out_count_dev)
    return fail(h, RSE_ERR_INVALID, "rse_knn_sharded_dev: output buffers are NULL");
  return rse_knn_merge_movies_dev(h, static_cast<const int64_t*>(h->sh_mine.p), h->comm_ranks, ns, k, kprime, out_dist_dev,
                                  out_chunk_rowid_dev, out_movie_idx_dev, out_count_dev);
}

int rse_hybrid_sharded_run_dev(rse_index* h, int32_t mode, double param, int32_t tie_mode, int32_t limit,
                               int32_t knn_multiplier, double k1, double b, const float* q_all_dev, int32_t nq_all,
                               int64_t* out_id_dev, double* out_score_dev, double* out_a_dev, double* out_b_dev,
                               int32_t* out_count_dev, int32_t* flagged_dev) {
  if (!h) return RSE_ERR_INVALID;
  if (!q_all_dev || nq_all < 1) return fail(h, RSE_ERR_INVALID, "rse_hybrid_sharded_run_dev: bad arguments");
  if (!h->comm) return fail(h, RSE_ERR_STATE, "no communicator: call rse_comm_init first");
  const int kprime = hybrid_kprime(h, mode, limit, knn_multiplier);
  if (kprime < 0) return kprime;
  const int ns = query_slice(nq_all, h->comm_ranks, h->comm_rank + 1) - query_slice(nq_all, h->comm_ranks, h->comm_rank);
  if (h->staged.nq != ns)
    return fail(h, RSE_ERR_STATE, "rse_hybrid_sharded_run_dev: the staged batch must be this rank's query slice (tokens)");
  CK(cudaSetDevice(h->device));
  Bm25Job bm25{&h->staged, limit, k1, b};
  int rc = sharded_knn_exchange(h, q_all_dev, nq_all, kprime, flagged_dev, ns > 0 ? &bm25 : nullptr);
  if (rc != RSE_OK) return rc;
  if (ns == 0) return RSE_OK;
  if (!out_id_dev || !out_score_dev || !out_a_dev || !out_b_dev || !out_count_dev)
    return fail(h, RSE_ERR_INVALID, "rse_hybrid_sharded_run_dev: output buffers are NULL");
  return hybrid_tail(h, mode, param, tie_mode, ns, limit, kprime, static_cast<const long long*>(h->sh_mine.p),
                     h->comm_ranks, bm25.enqueued,
                     Fused{reinterpret_cast<long long*>(out_id_dev), out_score_dev, out_a_dev, out_b_dev, out_count_dev,
                           limit});
}

int rse_hybrid_stash(rse_index* h, int32_t slot) {
  if (!h) return RSE_ERR_INVALID;
  if (slot < 0 || slot >= RSE_MAX_STASH) return fail(h, RSE_ERR_INVALID, "rse_hybrid_stash: slot out of range");
  if (h->next_collect < h->next_ticket)
    return fail(h, RSE_ERR_STATE, "rse_hybrid_stash: tickets in flight (collect or drain them first)");
  std::swap(h->staged, h->stash[slot]);
  h->pack_n = 0; h->pack_nq = 0;
  return RSE_OK;
}

int rse_tc_probe_rank(int32_t kprime, int32_t stride) {
  if (kprime < 1 || stride < 2) return kprime < 1 ? 0 : kprime;
  return sample_probe_rank(kprime, stride);
}

int rse_tc_last_survivors(rse_index* h, int32_t* out_counts, int32_t n) {
  if (!h) return RSE_ERR_INVALID;
  if (!out_counts || n < 0 || n > kTcBN) return fail(h, RSE_ERR_INVALID, "rse_tc_last_survivors: bad arguments");
  if (!h->tc_cnt.p) return fail(h, RSE_ERR_STATE, "rse_tc_last_survivors: the tensor-core path has not run");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  CK(cudaMemcpy(out_counts, h->tc_cnt.p, sizeof(int32_t) * n, cudaMemcpyDeviceToHost));
  return RSE_OK;
}

int rse_tc_last_pairs(rse_index* h, int32_t query, int64_t* out_rows, float* out_cos, int32_t cap, int32_t* out_n) {
  if (!h) return RSE_ERR_INVALID;
  if (!out_rows || !out_cos || !out_n || cap < 0) return fail(h, RSE_ERR_INVALID, "rse_tc_last_pairs: bad arguments");
  if (!h->tc_cnt.p || !h->tc_rows.p) return fail(h, RSE_ERR_STATE, "rse_tc_last_pairs: the tensor-core path has not run");
  const int64_t n_lists = static_cast<int64_t>(h->tc_rows.bytes / (sizeof(uint2) * kTcCandCap));
  if (query < 0 || query >= n_lists) return fail(h, RSE_ERR_INVALID, "rse_tc_last_pairs: query outside the last group");
  CK(cudaSetDevice(h->device));
  CK(cudaStreamSynchronize(h->stream));
  unsigned int cnt = 0;
  CK(cudaMemcpy(&cnt, static_cast<const unsigned int*>(h->tc_cnt.p) + query, sizeof(cnt), cudaMemcpyDeviceToHost));
  // the list keeps the first kTcCandCap survivors; a larger count is an overflow (reported, not copied)
  const int n = static_cast<int>(std::min<unsigned int>({cnt, static_cast<unsigned int>(kTcCandCap),
                                                         static_cast<unsigned int>(cap)}));
  std::vector<uint2> pairs(static_cast<size_t>(n));
  if (n > 0)
    CK(cudaMemcpy(pairs.data(), static_cast<const uint2*>(h->tc_rows.p) + static_cast<int64_t>(query) * kTcCandCap,
                  sizeof(uint2) * n, cudaMemcpyDeviceToHost));
  for (int i = 0; i < n; ++i) {
    out_rows[i] = static_cast<int64_t>(pairs[i].x);
    std::memcpy(&out_cos[i], &pairs[i].y, sizeof(float));
  }
  *out_n = static_cast<int32_t>(std::min<unsigned int>(cnt, 0x7FFFFFFFu));
  return RSE_OK;
}

int rse_hybrid_drain(rse_index* h, int32_t* out_dropped) {
  if (!h) return RSE_ERR_INVALID;
  CK(cudaSetDevice(h->device));
  int dropped = 0;
  while (h->next_collect < h->next_ticket) {
    rse_index::OutSlot& sl = h->out_slot[h->next_collect & 1];
    if (sl.ev) CK(cudaEventSynchronize(sl.ev));
    sl.knn = PendingKnn{};
    ++h->next_collect;
    ++dropped;
  }
  if (out_dropped) *out_dropped = dropped;
  return RSE_OK;
}

#ifdef RSE_REFINE_TIMING
// debug build only (-DRSE_REFINE_TIMING): per-CTA globaltimer stamps of the last knn_refine_kernel launch
int rse_debug_refine_ns(unsigned long long* out, int n_words) {
  return cudaMemcpyFromSymbol(out, rse::g_refine_ns, sizeof(unsigned long long) * n_words) == cudaSuccess ? 0 : -2;
}
#endif

}  // extern "C"
