/*
 * ccr_b200.h -- C ABI of the B200-native candidate score-and-rank path.
 *
 * The reference (awslabs/crowd-coachable-recommendations) has no FFI: its "operator API"
 * for this path is three Python call sites that run stock torch ops.  Each entry point
 * below replaces one of those torch call sites; the Python host layer
 * (crowd-coachable-recommendations_b200/ccr_b200) binds them with ctypes and keeps the
 * reference's Python signatures.  Reference paths are relative to /root/reference.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host;
 *   - the caller owns every buffer, including the workspace; the library allocates no
 *     persistent device memory and never synchronises the stream;
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*; NULL = legacy
 *     default stream);
 *   - return value: 0 on success, negative CCR_E* on failure; ccr_last_error_string()
 *     returns a thread-local description of the last failure;
 *   - re-entrant and stream-ordered.  Process-wide state is limited to: a per-device cache of
 *     immutable device attributes; the CCR_* environment test levers, parsed once on first
 *     use (ccr_debug_reload_env re-reads them); the optional watchdog record pointer
 *     (ccr_set_status_record).  The measurement hook (ccr_set_profile_events) is per host thread.
 *     Calls that share a workspace must be ordered on one stream.
 */
#ifndef CCR_B200_H_
#define CCR_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CCR_ABI_VERSION 6

/* error codes */
#define CCR_OK 0
#define CCR_EINVAL (-1)       /* bad argument (null pointer, misalignment, negative size...) */
#define CCR_EUNSUPPORTED (-2) /* shape outside what the kernels implement (k too large, D...) */
#define CCR_EWORKSPACE (-3)   /* workspace_bytes smaller than ccr_score_topk_workspace_bytes() */
#define CCR_ECUDA (-4)        /* a CUDA runtime / driver call failed                          */
#define CCR_EK_RANGE (-5)     /* k > number of items ("selected index k out of range")         */

/* mask_mode */
#define CCR_MASK_NONE 0
#define CCR_MASK_SET 1 /* score[row, col] = val   -- ranking(): scores[block_ind] = -1e6,
                          scripts/ms_marco_eval.py:227                                         */
#define CCR_MASK_ADD 2 /* score[row, col] += val in float64 -- rime_lite prior_score:
                          src/rime_lite/dataset/base.py:234,279-282 added at
                          src/ccrec/models/bert_mt.py:376 / score_array.py:120-121,291-293     */

/* flags for ccr_score_topk_bf16 */
#define CCR_ALGO_AUTO 0
#define CCR_ALGO_SIMT 1   /* CUDA-core streaming kernel (128-bit coalesced loads); any B, meant
                             for the bandwidth-bound B <= 8 regime                              */
#define CCR_ALGO_TCGEN05 2 /* TMA + tcgen05/TMEM bf16 GEMM fused with mask + top-k epilogue    */
#define CCR_ALGO_MASK 0xF
#define CCR_FLAG_ALLOW_SHORT 0x10 /* k > n_items allowed: tail padded with (-inf, id -1); used for
                                     row shards smaller than k                                  */

#define CCR_FLAG_PACKED_KEYS 0x20 /* out_scores64 receives uint64 sort keys instead of doubles:
                                       (ord32(float32 score) << 32) | (0xFFFFFFFF - uint32 global id),
                                       ord32(f) = bits(f) ^ (f < 0 ? 0xFFFFFFFF : 0x80000000); a larger key
                                       ranks first (score descending, then id ascending), 0 = padding.  The
                                       8-byte exchange format of the row-sharded path (ccr_merge_topk_keys);
                                       needs id_offset + n_items <= 2^32 and no CCR_MASK_ADD (float64
                                       priors do not fit a float32 key)                           */

#define CCR_MAX_K 2048

int ccr_abi_version(void);
const char* ccr_last_error_string(void);

/*
 * Fused  scores = Q . items^T  ->  sparse mask  ->  per-row top-k, sorted descending,
 * ties broken by lowest item id.  The B x N score matrix is never written to memory.
 *
 * Replaces, in one call:
 *   scripts/ms_marco_eval.py:206-218  (tile GEMM loop + D2H scatter into the host matrix)
 *   scripts/ms_marco_eval.py:221-230  (host mask, H2D of the row, full sort, [:1001])
 *   src/rime_lite/util/__init__.py:135-141 (as_tensor of MatMul+prior, topk(k).indices)
 *   src/ccrec/models/bbpr.py:528-545  (BertBPR.transform tile loop)
 *
 *   q        [B, ldq]  bf16 row-major queries / user embeddings (ldq >= D, ldq % 8 == 0)
 *   items    [n_items, ldi] bf16 row-major item / passage table shard (ldi >= D, ldi % 8 == 0,
 *            base 16-byte aligned)
 *   D        embedding dim (768 in the reference: ms_marco_eval.py:190), D % 8 == 0, D <= 4096
 *   k        1 .. CCR_MAX_K
 *   mask_*   CSR over the LOCAL item columns of this shard: indptr[B+1] (int64), cols sorted
 *            and unique per row (int32, < n_items), vals float64, mask_nnz == indptr[B];
 *            (mask_nnz may also be an UPPER BOUND of indptr[B] -- the capacity of cols / vals -- when
 *            the CSR was produced on the device, e.g. by ccr_mask_column_shard; the kernels read the
 *            true count from indptr, the bound sizes the workspace);
 *            mask_max_row_nnz = largest number of entries in one row, or an upper bound (lets the kernel stream masked
 *            items through and drop them at the end instead of testing every candidate; pass -1 if
 *            unknown); all NULL / 0 when mask_mode == CCR_MASK_NONE
 *   id_offset added to local item ids on output (row-sharded tables)
 *   out_scores   [B, k] float32, descending           (may be NULL)
 *   out_scores64 [B, k] float64 exact value the order was decided on (may be NULL)
 *   out_ids      [B, k] int64 global item ids
 */
int ccr_score_topk_bf16(const void* q, int64_t B, int64_t ldq,
                        const void* items, int64_t n_items, int64_t ldi,
                        int D, int k,
                        const int64_t* mask_indptr, const int32_t* mask_cols,
                        const double* mask_vals, int64_t mask_nnz, int64_t mask_max_row_nnz,
                        int mask_mode, int64_t id_offset,
                        float* out_scores, double* out_scores64, int64_t* out_ids,
                        void* workspace, size_t workspace_bytes,
                        int flags, void* stream);

/* Bytes of workspace ccr_score_topk_bf16 needs for these arguments (same flags!).
 * Returns 0 on invalid arguments. */
size_t ccr_score_topk_workspace_bytes(int64_t B, int64_t n_items, int D, int k,
                                      int64_t mask_nnz, int64_t mask_max_row_nnz, int flags);

/*
 * G-way merge of per-shard top-k lists after the all-gather (multi-GPU exchange step; no
 * reference counterpart -- the reference scores on one GPU, ms_marco_eval.py:205).
 *   scores64 [G, B, k_in] float64 each run sorted descending, ids [G, B, k_in] int64
 *   (id < 0 = padding).  Output: the k_out best of the union per row, descending,
 *   ties -> lowest id.  Missing entries are padded with (-inf, -1).
 */
int ccr_merge_topk(const double* scores64, const int64_t* ids, int G, int64_t B, int k_in,
                   int k_out, float* out_scores, double* out_scores64, int64_t* out_ids,
                   void* stream);

/*
 * The same merge for runs in the packed exchange format of CCR_FLAG_PACKED_KEYS:
 *   keys [G, B, k_in] uint64, each run sorted descending (0 = padding).  Outputs (each may be NULL, not
 *   both of out_ids / out_keys): out_scores float32 [B, k_out], out_ids int64 [B, k_out] (global ids;
 *   -1 / -inf padding), out_keys uint64 [B, k_out] the merged run still packed (for a further exchange).
 * 8 bytes per entry on the wire instead of 16 (SURVEY section 8e); merge-path merges in shared
 * memory.  G * k_in keys must fit shared memory (CCR_EUNSUPPORTED otherwise: G * k_in <= ~16 K).
 * ccr_unpack_topk_keys turns n packed keys into (float32 score, int64 id) pairs.
 */
int ccr_merge_topk_keys(const uint64_t* keys, int G, int64_t B, int k_in, int k_out, float* out_scores,
                        int64_t* out_ids, uint64_t* out_keys, void* stream);
int ccr_unpack_topk_keys(const uint64_t* keys, int64_t n, float* out_scores, int64_t* out_ids, void* stream);

/*
 * Column shard of a device mask CSR for a row-sharded table: entries with col_lo <= col < col_hi,
 * re-based to local columns (col - col_lo).  out_indptr [B+1]; out_cols / out_vals need room for
 * every entry of the input (the shard's count is only known on the device: pass the input's nnz as
 * mask_nnz upper bound to ccr_score_topk_bf16).  Replaces a host-side numpy pass per step.
 */
int ccr_mask_column_shard(const int64_t* indptr, const int32_t* cols, const double* vals, int64_t B, int64_t col_lo,
                          int64_t col_hi, int64_t* out_indptr, int32_t* out_cols, double* out_vals, void* stream);

/*
 * Embedding-table ingest: fp32 rows -> bf16 table rows, optionally L2-normalised first
 * (F.normalize(p=2, dim=1, eps=1e-12) in fp32, then round) for CCREC_SIM_TYPE=cos.
 * Replaces `.to("cpu")` in scripts/ms_marco_eval.py:140-145 and cos_sim's normalisation
 * (scripts/ms_marco_eval.py:160-161, src/ccrec/models/bbpr.py:490-491).
 *   src [n, ld_src] float32, dst [n, ld_dst] bf16; columns D..ld_dst-1 of dst are zeroed.
 */
int ccr_ingest_rows_f32(const float* src, int64_t n, int D, int64_t ld_src,
                        void* dst, int64_t ld_dst, int normalize, void* stream);

/* Same for rows that are already bf16 (normalisation computed in fp32). */
int ccr_normalize_rows_bf16(const void* src, int64_t n, int D, int64_t ld_src,
                            void* dst, int64_t ld_dst, void* stream);

/*
 * Dense score tile  out[B, n] = Q . items^T  (fp32) for callers that really want the matrix
 * (LazyScore.as_tensor / _argsort on reranking sets: score_array.py:291-293).  Tiles of at least
 * 2^20 scores run on the TMA + tcgen05 pipeline of the fused kernel with a store epilogue, smaller
 * ones on a CUDA-core kernel.
 */
int ccr_score_dense_f32(const void* q, int64_t B, int64_t ldq, const void* items, int64_t n_items,
                        int64_t ldi, int D, float* out, int64_t ld_out, void* stream);

/*
 * Whole-matrix argsort: rime_lite `_argsort` (src/rime_lite/util/__init__.py:158-184), which flattens
 * the evaluated score matrix and sorts ALL of it, best first.  scores [B, ld] float32 on the device
 * (e.g. written by ccr_score_dense_f32), optional mask CSR as in ccr_topk_dense_f32 (ADD ranks
 * double(score) + value, SET the value: the reference's float64 promotion).  Output: out_rows /
 * out_cols int64 [B * n_cols], score descending, equal scores in flat (row-major) order -- the
 * reference breaks ties with unseeded jitter.  LSD radix sort over ~ord64(double) keys, 8 passes;
 * B * n_cols <= 2^31.  Workspace from ccr_argsort_workspace_bytes(B * n_cols).
 */
size_t ccr_argsort_workspace_bytes(int64_t n_elements);
int ccr_argsort_scores_f32(const float* scores, int64_t B, int64_t n_cols, int64_t ld, const int64_t* mask_indptr,
                           const int32_t* mask_cols, const double* mask_vals, int64_t mask_nnz, int mask_mode,
                           int64_t* out_rows, int64_t* out_cols, void* workspace, size_t workspace_bytes,
                           void* stream);

/*
 * MRR core (scripts/al_0_rank.py:130-133: BEIR evaluate_custom(..., metric="mrr") over the ranking):
 * per query row the 1-based rank of the first relevant id in its ranked list, 0 if none.
 *   ids [B, k] int64 ranked best first (as written by ccr_score_topk_bf16; < 0 = padding);
 *   rel_indptr int64[B+1], rel_ids int64 sorted ascending inside a row (the qrels with score > 0).
 * MRR@c = sum over rows with 0 < rank <= c of 1 / rank, divided by the number of qrels queries.
 */
int ccr_first_hit_rank(const int64_t* ids, int64_t B, int k, const int64_t* rel_indptr, const int64_t* rel_ids,
                       int32_t* out_rank, void* stream);

/*
 * Top-k of an ALREADY MATERIALISED dense float32 score matrix plus an optional sparse prior: the
 * `_assign_topk` call the reference makes when `BertBPR.transform` hands it the dense users x items
 * host matrix (src/rime_lite/util/__init__.py:135-141 on the tensor built by
 * src/rime_lite/util/score_array.py:226-227 [+ :173-174 for the float64 CSR]).
 *   scores [B, ld] float32 on the device; mask as in ccr_score_topk_bf16 (CSR over columns, float64
 *   values): CCR_MASK_ADD ranks double(score) + value, CCR_MASK_SET ranks the value itself -- the
 *   float64 promotion of the reference; columns without an entry rank by their float32 score.
 *   Output: descending, ties -> lowest column.  B <= 65535, k + mask_max_row_nnz <= CCR_MAX_K.
 */
size_t ccr_topk_dense_workspace_bytes(int64_t B, int64_t n_cols, int k, int64_t mask_nnz, int64_t mask_max_row_nnz);
int ccr_topk_dense_f32(const float* scores, int64_t B, int64_t n_cols, int64_t ld, int k, const int64_t* mask_indptr,
                       const int32_t* mask_cols, const double* mask_vals, int64_t mask_nnz, int64_t mask_max_row_nnz,
                       int mask_mode, float* out_scores, double* out_scores64, int64_t* out_ids, void* workspace,
                       size_t workspace_bytes, void* stream);

/*
 * BM25 -- the lexical sibling of the dense path.  Replaces BM25.transform (scripts/bm_25.py:27-45)
 * and the per-query loop of ranking_bm25 (scripts/ms_marco_eval.py:165-186: one scipy transform,
 * one FULL sort of n_docs float32 scores and a [0:1001] slice per query).
 *
 * Index, resident on the device (CSC of the doc-term count matrix the reference caches,
 * bm_25.py:22-25):  post_indptr int64[n_terms+1], post_docs int32[nnz] ascending inside a term,
 * post_tf float32[nnz].
 *
 * ccr_bm25_build_impacts (once per fit / cache): per posting of term t in doc d
 *     post_val = ((tf * idf[t]) * (k1 + 1)) * (1 / (tf + doc_norm[d]))      float64, bm_25.py:39-45
 * (scipy evaluates the reference's sparse / dense division as a multiplication by the reciprocal)
 * with idf[t] = log(n/df_t) (sklearn idf_ - 1) and doc_norm[d] = k1 * (1 - b + b * len_d / avdl)
 * supplied by the host.  The expression does not depend on the query, so it is hoisted out of it.
 *
 * Queries: CSR of DISTINCT vocabulary term ids (q_indptr int64[Bq+1], q_terms int32; the
 * reference uses q.indices only, bm_25.py:38, so query term counts do not matter);
 * max_query_terms = longest row (<= 512).  score[q, d] = sum of post_val over the query's terms
 * present in d, summed in q_terms order in float64.
 *
 * ccr_bm25_topk: per query the k best docs RANKED AS FLOAT32 (the reference sorts
 * torch.Tensor(solution), ms_marco_eval.py:179-181), descending, ties -> lowest doc position
 * (reference: unspecified); out_scores float32 [Bq,k], out_ids int64 [Bq,k].  The n_docs-long
 * score vector only ever exists chunk-wise in shared memory.  k > n_docs -> CCR_EK_RANGE.
 * ccr_bm25_scores_f64: the dense float64 score rows themselves (BM25.transform drop-in).
 *
 * Head terms (optional, hybrid index).  A few vocabulary terms occur in a large share of the documents
 * (stop words); their posting lists dominate the postings a query batch touches.  For such terms the
 * caller may additionally keep a DENSE float64 row (post_val at the docs that contain the term, 0
 * elsewhere; x + 0.0 == x bit for bit, so the sums do not change): the kernels then add the row with
 * independent coalesced loads instead of walking the list (8 bytes per doc instead of 12 per posting, no
 * cursor, no searches).  ccr_bm25_build_head_rows fills head_slot int32[n_terms] (slot of a head term,
 * -1 for every other term) and head_rows float64[n_head, pitch] with pitch = ccr_bm25_head_row_pitch(n_docs)
 * (n_docs rounded up to the kernel's 512-doc chunk) from the postings of head_terms int32[n_head] (device;
 * distinct term ids chosen by the caller, e.g. every term with df >= n_docs / 4; ids outside [0, n_terms)
 * are ignored).  The posting lists stay
 * complete, so head_slot = head_rows = NULL is always valid.
 */
int64_t ccr_bm25_head_row_pitch(int64_t n_docs);
int ccr_bm25_build_head_rows(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                             const int32_t* head_terms, int n_head, int64_t n_terms, int64_t n_docs,
                             int32_t* head_slot, double* head_rows, void* stream);
int ccr_bm25_build_impacts(const int64_t* post_indptr, const int32_t* post_docs, const float* post_tf,
                           const double* idf, const double* doc_norm, double k1, int64_t n_terms, int64_t nnz,
                           double* post_val, void* stream);
size_t ccr_bm25_topk_workspace_bytes(int64_t Bq, int64_t n_docs, int k);
int ccr_bm25_topk(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                  const int32_t* head_slot, const double* head_rows, const int64_t* q_indptr,
                  const int32_t* q_terms, int64_t max_query_terms, int64_t Bq,
                  int64_t n_docs, int k, float* out_scores, int64_t* out_ids, void* workspace,
                  size_t workspace_bytes, void* stream);
int ccr_bm25_scores_f64(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                        const int32_t* head_slot, const double* head_rows, const int64_t* q_indptr,
                        const int32_t* q_terms, int64_t max_query_terms, int64_t Bq,
                        int64_t n_docs, double* scores, int64_t ld, void* stream);

/* Which kernel ccr_score_topk_bf16 picks under CCR_ALGO_AUTO: CCR_ALGO_SIMT or CCR_ALGO_TCGEN05. */
int ccr_choose_algo(int64_t B, int64_t n_items, int D, int k);

/*
 * Measurement hook: when both are non-NULL (cudaEvent_t passed as void*), every later
 * ccr_score_topk_bf16 call on this host thread records `start_event` immediately before and
 * `stop_event` immediately after its dominant kernel (the fused score+select kernel) on the
 * call's stream, so a benchmark can time that kernel alone without a profiler.  Pass NULLs to
 * switch it off.
 */
void ccr_set_profile_events(void* start_event, void* stop_event);

/* Launch plan ccr_score_topk_bf16 would use for these arguments, for benchmarks / DESIGN.md
 * bookkeeping.  Fills info8 = { n_q_tiles (units of 128 query rows, or 256 for CTA pairs), n_splits
 * (item splits), cand_capacity (keys per candidate buffer), algo (CCR_ALGO_*), two_cta (0/1),
 * seed_items (sampled items of the threshold-seeding pre-pass, 0 = none), n_kernel_launches (kernels
 * one call launches), lead_tiles (bounded drift of the units sharing an item split) }.  Returns 0 or
 * CCR_E*. */
int ccr_plan_info(int64_t B, int64_t n_items, int D, int k, int64_t mask_nnz, int64_t mask_max_row_nnz,
                  int flags, int32_t* info8);

/*
 * Watchdog record.  Every barrier wait of the tensor-core kernel is bounded (10 s); on expiry the
 * kernel writes { code = 1, where (role / barrier id), block, extra } and traps, which poisons the
 * CUDA context -- device memory can no longer be read back.  A caller that wants the record passes a
 * 16-byte HOST buffer that the device can write (cudaHostAlloc / pinned memory under UVA), zeroed;
 * after a failed synchronisation it reads the four int32 from host memory.  NULL (default): the
 * record goes to a slot inside the workspace.  Process-wide.
 */
void ccr_set_status_record(void* host_mapped_ptr);

/* Tests: re-read the CCR_* environment test levers (DESIGN.md section 7b).  They are parsed once on
 * first use; a test that changes the environment of a live process calls this afterwards.
 * Not thread-safe against concurrent ccr_* calls. */
void ccr_debug_reload_env(void);

#ifdef __cplusplus
}
#endif
#endif /* CCR_B200_H_ */
