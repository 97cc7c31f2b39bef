// Kernel parameter blocks and launcher prototypes shared by the .cu translation units.
#pragma once
#include "ccr_common.cuh"

namespace ccr {

// One "unit" = (query tile, item split).  Each unit owns, per query row, a private candidate
// buffer of `C` 64-bit keys in the workspace:  cand[(row * S + split) * C + i],
// counts[row * S + split].  rows are padded to a multiple of the row-tile of the kernel.
struct SelectParams {
  const __nv_bfloat16* q;
  long long ldq;
  int B;
  int q_rows;     // rows the query tensor map may address (>= B; > B when the caller padded q)
  const __nv_bfloat16* items;
  long long ldi;
  long long n_items;
  int D;
  int k;
  int k_keep;     // upper bound of the candidates one row must keep (k + mask_max_row_nnz in include
                  // mode, else k): the candidate buffers are sized for it, so per-row counts derived from
                  // the CSR are clamped to it (a caller that under-reports mask_max_row_nnz must not be
                  // able to overrun a buffer)
  int C;          // candidate capacity per (row, split)
  int S;          // item splits
  int n_q_tiles;  // query tiles (tensor-core kernel: 128 rows, or 256 when two_cta) or groups of 8 (SIMT)
  int two_cta;    // tensor-core kernel: units are CTA pairs (cta_group::2, UMMA M = 256)
  const long long* mask_indptr;  // null when no mask
  const int* mask_cols;          // null in 'include' mode (masked items are NOT excluded while
                                 // streaming: each row keeps k + nnz(row) candidates instead and
                                 // finalize drops the masked ones); set in 'exclude' mode
  u64* cand;
  int* counts;
  // cross-stream threshold sharing (tensor-core kernel; null/0 = off).  A "stream" is one
  // (row, split, half) candidate list.  Every stream publishes the score of its share_j-th best
  // candidate (g_q, monotone); the share_m-th largest published value over the row's streams is a
  // lower bound of the row's global k-th best (share_m * share_j >= k distinct unmasked items
  // score at least that much) and is max-reduced into g_tau[row].
  u32* g_tau;   // [rows_pad]            ord32(score), 0 = nothing known
  u32* g_q;     // [rows_pad][S_row]     ord32(score), 0 = not published
  int S_row;    // streams per row
  int share_j;
  int share_m;
  // early threshold sharing through a per-row score histogram (tensor-core kernel, no exclude-mode
  // mask; null = off).  Row r owns kHistBins counters over ord32(score) buckets of width 2^shift
  // starting at the row's seed bound (g_hpar[r] = {base, shift + 1}; .y == 0: row disabled).
  // Every appended candidate group adds its best item to its bucket; whoever finds >= k_row items
  // counted at or above a bucket's lower edge has a valid lower bound of the row's k-th best --
  // long before any stream has filled a buffer and pruned.
  u32* g_hist;        // [rows_pad][kHistBins]
  const uint2* g_hpar;  // [rows_pad]
  DeviceStatus* status;
  // bounded drift between the CTAs that stream the same item split (keeps their shared item
  // tiles L2-resident so the table is read from HBM once): tiles issued so far, per unit
  int* progress;  // [n_units], zeroed per call; null = off
  int lead_tiles; // max lead (item tiles) of a producer over the slowest unit on the same split
  int lead_every; // inline throttle: progress is published / checked every lead_every tiles (power of two)
  int throttle_poller;  // 1: a dedicated warp watches the peers (tile-granular), 0: the producer polls inline
  // store mode: write fp32 scores instead of selecting (dense score tiles for as_tensor / _argsort).
  // With store_max8 (threshold seeding pre-pass) only the best score of every 8 consecutive items is
  // written: the k-th largest of those group maxima is a lower bound of the k-th largest item score,
  // carried by k distinct items -- 1/8 of the bytes, and the selection pass over them is 8x shorter.
  float* dense_out;      // [rows_pad][ld_out], null in select mode
  long long ld_out;      // floats per row: >= n_items rounded up to 256 (full) or / 8 (store_max8)
  int store_max8;
};

struct FinalizeParams {
  int B;
  int k;
  int C;
  int S;
  const u64* cand;
  const int* counts;
  const u32* g_tau;  // per-row lower bound of the k-th best dense score (ord32), or null: prefilter
  const int* drop_cols;  // include mode: the mask's column array; dense candidates found in the row's
                         // list are dropped here (their override record carries the final value)
  // mask overrides (null when no mask): per mask entry e, value and ~col
  const long long* mask_indptr;
  const u64* ovr_hi;
  const u32* ovr_lo;
  long long id_offset;
  float* out_scores;
  double* out_scores64;
  u64* out_keys;   // CCR_FLAG_PACKED_KEYS: [ord32(float32 score) : ~uint32 global id] instead of out_scores64
  long long* out_ids;
};

struct OverrideParams {
  const __nv_bfloat16* q;
  long long ldq;
  int B;
  const __nv_bfloat16* items;
  long long ldi;
  long long n_items;
  int D;
  const long long* mask_indptr;
  const int* mask_cols;
  const double* mask_vals;
  long long nnz;
  int mode;
  u64* ovr_hi;
  u32* ovr_lo;
};

// launchers (return cudaError_t as int)
int launch_select_simt(const SelectParams& p, cudaStream_t st);
int launch_select_tc(const SelectParams& p, cudaStream_t st, int num_sms);
constexpr int kHistBins = 128;
int launch_seed_tau(const float* scores, long long ld, int m, int B, int k, const long long* mask_indptr,
                    u32* g_tau, uint2* g_hpar, cudaStream_t st);
int launch_overrides(const OverrideParams& p, cudaStream_t st);
int launch_finalize(const FinalizeParams& p, cudaStream_t st);
int launch_merge_topk(const double* s, const long long* ids, int G, long long B, int k_in, int k_out,
                      float* os, double* os64, long long* oi, cudaStream_t st);
int launch_merge_keys(const u64* keys, int G, long long B, int k_in, int k_out, float* os, long long* oi, u64* ok,
                      cudaStream_t st);
int launch_unpack_keys(const u64* keys, long long n, float* os, long long* oi, cudaStream_t st);
int launch_mask_shard(const long long* indptr, const int* cols, const double* vals, long long B, int lo, int hi,
                      long long* out_indptr, int* out_cols, double* out_vals, cudaStream_t st);
int launch_ingest_f32(const float* src, long long n, int D, long long ld_src, __nv_bfloat16* dst,
                      long long ld_dst, int normalize, cudaStream_t st);
int launch_normalize_bf16(const __nv_bfloat16* src, long long n, int D, long long ld_src,
                          __nv_bfloat16* dst, long long ld_dst, cudaStream_t st);
int launch_dense_f32(const __nv_bfloat16* q, long long B, long long ldq, const __nv_bfloat16* items,
                     long long n, long long ldi, int D, float* out, long long ld_out, cudaStream_t st);

// whole-matrix argsort and MRR first-hit scan (ccr_sort.cu)
size_t argsort_workspace_bytes(long long n);
int launch_argsort(const float* scores, long long B, long long N, long long ld, const long long* indptr, const int* cols,
                   const double* vals, long long nnz, int mode, long long* out_rows, long long* out_cols, void* ws,
                   cudaStream_t st);
int launch_first_hit_rank(const long long* ids, long long B, int k, const long long* rel_indptr, const long long* rel_ids,
                          int* out_rank, cudaStream_t st);

// dense top-k (ccr_kernels.cu)
constexpr int kDenseSlack = 4096;  // columns one block scans between two prune checks (16 per thread)
int launch_select_dense(const float* scores, long long ld, long long B, long long N, int k, int k_keep,
                        const long long* mask_indptr, int C, int S, u64* cand, int* counts, cudaStream_t st);
int launch_override_dense(const float* scores, long long ld, int B, long long N, const long long* mask_indptr,
                          const int* mask_cols, const double* mask_vals, long long nnz, int mode, u64* ovr_hi,
                          u32* ovr_lo, cudaStream_t st);

// BM25 (ccr_kernels.cu)
// block shape, measured at the NQ shape (profiles/r01_bm25_bench.json): 4096 docs x 256 threads x 5 blocks
// per SM 45.3 ms per 3,452 queries; 8192 x 512 x 2: 56.7 ms; 4096 x 512 x 2: 70.9; 8192 x 256 x 3: 65.7
#ifndef CCR_BM_CHUNK
#define CCR_BM_CHUNK 4096
#define CCR_BM_THREADS 256
#define CCR_BM_BLOCKS_PER_SM 5
#endif
constexpr int kBmChunk = CCR_BM_CHUNK;     // docs per shared-memory accumulator pass (8 bytes each)
constexpr int kBmThreads = CCR_BM_THREADS;
constexpr int kBmBlocksPerSm = CCR_BM_BLOCKS_PER_SM;
constexpr int kBmMaxTerms = 512;   // distinct vocabulary terms per query
constexpr int kBmSlack = 1024;     // accumulators ranked between two prune checks
// warp-private variant: 8 independent warps per block, 512-doc mini-chunks, <= 32 distinct query terms
constexpr int kBmwWarps = 8;
constexpr int kBmwMini = 512;
constexpr int kBmwMaxTerms = 32;   // one lane per term
constexpr int kBmwSketchM = 5;       // query bound = the 5th largest of the streams' ceil(k/5)-th best scores (7, 8: same speed)
constexpr int kBmwDepth = 4;         // batches of 32 postings in flight per warp on a dense term
#ifndef CCR_BMW_BLOCKS_PER_SM
#define CCR_BMW_BLOCKS_PER_SM 4
#endif
constexpr int kBmwBlocksPerSm = CCR_BMW_BLOCKS_PER_SM;   // 42.5 KB of static shared memory per block; 64 registers per
                                                         // thread (5 blocks = 48 registers spill: 46.7 vs 39.1 ms, r02_bm25.md)
int launch_bm25_topk_warp(const long long* post_indptr, const int* post_docs, const double* post_val,
                          const int* head_slot, const double* head_rows, long long ld_head,
                          const long long* q_indptr, const int* q_terms, long long Bq, long long N, int k, int C, int S,
                          u64* cand, int* counts, u32* row_tau, double* dense_out, long long ld_out, cudaStream_t st);
int launch_bm25_head_slots(const int* head_terms, int n_head, long long n_terms, int* head_slot, cudaStream_t st);
int launch_bm25_head_rows(const long long* post_indptr, const int* post_docs, const double* post_val,
                          const int* head_terms, int n_head, long long n_terms, long long ld_head, double* rows,
                          cudaStream_t st);
int launch_bm25_impacts(const long long* post_indptr, const int* post_docs, const float* post_tf, const double* idf,
                        const double* doc_norm, double k1p1, long long V, long long nnz, double* val,
                        cudaStream_t st);
int launch_bm25_topk(const long long* post_indptr, const int* post_docs, const double* post_val,
                     const int* head_slot, const double* head_rows, long long ld_head, const long long* q_indptr, const int* q_terms, long long Bq, long long N, int k, int C, int S,
                     u64* cand, int* counts, double* dense_out, long long ld_out, cudaStream_t st);

}  // namespace ccr
