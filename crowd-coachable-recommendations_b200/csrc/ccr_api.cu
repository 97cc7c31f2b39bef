// C ABI (include/ccr_b200.h): argument validation, launch planning, workspace carving.
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>

#include "../../include/ccr_b200.h"
#include "ccr_params.cuh"

using namespace ccr;

static thread_local char g_err[512] = "";
static void* g_status_record = nullptr;  // see ccr_set_status_record
static thread_local cudaEvent_t g_prof_start = nullptr, g_prof_stop = nullptr;  // see ccr_set_profile_events

// Test levers (DESIGN.md §7b): each forces a choice the planner otherwise makes itself, so that the
// tests can check that results do not depend on it.  The environment is parsed ONCE, on first use; a
// test that changes it inside a live process calls ccr_debug_reload_env().  None is needed in production.
namespace {
struct Knobs {
  int two_cta = -1, lead = 0, no_hist = 0, bm25_blockwide = 0, exact_fallback = 0;
};
Knobs g_knobs;
std::once_flag g_knobs_once;

int env_int(const char* name, int dflt) { const char* v = getenv(name); return v ? atoi(v) : dflt; }
void load_knobs() {
  Knobs k;
  k.two_cta = env_int("CCR_2CTA", -1);
  k.lead = env_int("CCR_LEAD", 0);
  k.no_hist = getenv("CCR_NO_HIST") != nullptr;
  k.bm25_blockwide = getenv("CCR_BM25_BLOCKWIDE") != nullptr;
  k.exact_fallback = env_int("CCR_EXACT_FALLBACK", 0) != 0;
  g_knobs = k;
}
const Knobs& knobs() {
  std::call_once(g_knobs_once, load_knobs);
  return g_knobs;
}
}  // namespace

static int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return code;
}

// The return code of a launcher or CUDA call: 0 is success, a cudaError_t becomes CCR_ECUDA with its text, and a
// negative code is a tensor map that could not be encoded (launch_select_tc).
static int cuda_rc(int rc, const char* what) {
  if (rc == 0) return CCR_OK;
  if (rc < 0) return fail(CCR_ECUDA, "%s failed: tensor map encode error %d", what, rc);
  return fail(CCR_ECUDA, "%s failed: %s", what, cudaGetErrorString((cudaError_t)rc));
}

static int device_sm_count() {
  static int cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); return 148; }
  if (!cached[dev]) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) {
      cudaGetLastError();
      n = 148;
    }
    cached[dev] = n;
  }
  return cached[dev];
}

namespace {
// Workspace layout: regions taken one after another, each starting at a 256-byte boundary
struct Carve {
  size_t off = 0;
  size_t take(size_t bytes) {
    const size_t at = off;
    off = (off + bytes + 255) / 256 * 256;
    return at;
  }
};

struct Plan {
  int sms;        // SMs of the device the plan is made for; every launch of the call uses the same count
  int algo;
  int n_q_tiles;  // TC: query tiles of 128; SIMT: groups of 8
  int rows_pad;
  int S;        // item splits
  int halves;   // candidate buffers per (row, split): 2 for the tensor-core kernel
  int C;
  int share_j, share_m;  // threshold sharing level (0 = off)
  int two_cta;           // tensor-core kernel variant: CTA pairs (cta_group::2)
  int include_mask;      // 1: masked items stream through and are dropped in finalize (k + h candidates/row)
  int k_keep;            // k + h_max in include mode, else k
  int seed_m;            // sampled items of the threshold-seeding pre-pass (0 = no pre-pass)
  long long seed_stride; // item-row stride of the sample
  long long seed_ld;     // row pitch of the sampled score matrix (floats)
  int use_hist;          // the pre-pass also sets up the per-row score histograms (histogram sharing)
  int throttle;          // bounded-drift throttle between the units of one item split (tensor-core kernel)
  int lead_tiles;        // throttle: max lead (item tiles) of a producer over its slowest peer
  int lead_every;        // throttle: progress is published / checked every lead_every tiles (power of two)
  int throttle_poller;   // throttle: 1 a dedicated warp watches the peers, 0 the producer polls inline
  int k_cand;            // exact ranking: candidates the scan stage returns per row (k' >= k, <= n_items)
  size_t off_cand, off_counts, off_rec_hi, off_rec_lo;
  // [zero_begin, zero_end) is cleared by ONE memset per call: status, throttle counters, sharing state
  size_t zero_begin, off_status, off_progress, off_gtau, off_gq, off_hist, off_hpar, zero_end;
  size_t off_qpad;       // zero-padded copy of a short query batch (B < 128): every TMA box in bounds
  size_t off_seed, total;
};

// item splits of the tensor-core pipeline: nq query tiles against the item tiles of n_items rows on `sms` units
int splits_tc(int nq, long long n_items, int sms) {
  const long long tiles = (n_items + kITile - 1) / kITile;
  long long smax = tiles < 1 ? 1 : tiles;
  long long s0 = sms / nq;  // from the largest split count that still fits ONE wave
  if (s0 < 1) s0 = 1;
  if (s0 >= smax) return (int)smax;
  long long best = s0;
  double best_waste = 2.0;
  long long send = s0 * 4 + 40;
  if (send > smax) send = smax;
  for (long long s = s0; s <= send; ++s) {
    long long units = (long long)nq * s;
    long long waves = (units + sms - 1) / sms;
    double waste = (double)(waves * sms - units) / (double)(waves * sms);
    if (waste < best_waste - 1e-12) { best_waste = waste; best = s; }
    if (waste <= 0.03) break;
  }
  return (int)best;
}

// h_max: largest number of mask entries in one row, or < 0 when unknown / no mask
bool make_plan(long long B, long long n_items, int D, int k, long long nnz, long long h_max, int flags, Plan* pl) {
  int algo = flags & CCR_ALGO_MASK;
  if (algo == CCR_ALGO_AUTO) algo = ccr_choose_algo(B, n_items, D, k);
  const int sms = device_sm_count();
  const Knobs& kn = knobs();
  pl->sms = sms;
  pl->algo = algo;
  {
    // Exact ranking (DESIGN.md section 6b): a row is certified when its k-th exact value beats the scan
    // score of the k'-th candidate by the error bound E of the scan format.  E is ~8x smaller for fp16
    // (u = 2^-11) than for bf16 (2^-8), so fp16 needs far fewer extra candidates for the same share of
    // certified rows.  See DESIGN.md section 6b for the measured shares behind the two rules.
    long long kc = (flags & CCR_FLAG_F16) ? k + k / 4 + 32 : 3LL * k + 32;
    if (kc > CCR_MAX_K) kc = CCR_MAX_K;
    if (kc < k) kc = k;
    if (kc > n_items) kc = n_items;
    pl->k_cand = (int)kc;
  }
  pl->include_mask = (algo == CCR_ALGO_TCGEN05 && nnz > 0 && h_max >= 0 && h_max <= 256 && k + h_max <= CCR_MAX_K) ? 1 : 0;
  pl->k_keep = pl->include_mask ? (int)(k + h_max) : k;
  if (algo == CCR_ALGO_TCGEN05) {
    // CTA pairs (cta_group::2, 256 query rows per unit) stream each item tile once for 256 queries:
    // a third less operand traffic from L2 into the SMs and a GEMM pipeline that is ~9 % faster on its
    // own.  With the bounded-drift throttle (below) they win at every batch size
    // measured on B200 (8.84M x 768, k=100, same box, profiles/r01_pairs_throttle_ab.txt): B=256 2.95 vs
    // 3.27 ms, 512 5.7 vs 6.05, 1024 11.2-11.7 vs 12.2, 2048 21.7 vs 23.4, 4096 43.3 vs 46.8, 8192 90.0 vs
    // 92.6; bench.py's sustained loop 94.3-95.0 k vs 87.1-87.4 k queries/s.  A pair pads the batch to 256
    // rows, so a small odd number of 128-row tiles stays on single CTAs (B=384: 4.72 vs 5.48 ms); the
    // margin shrinks with the number of query tiles per split (8192: 3 %), beyond that single CTAs.
    {
      const long long tiles128 = (B + kQTile - 1) / kQTile;
      pl->two_cta = (B > kQTile && B <= 8192 && (tiles128 % 2 == 0 || tiles128 >= 17)) ? 1 : 0;
    }
    if (kn.two_cta >= 0) pl->two_cta = (B > kQTile && kn.two_cta != 0) ? 1 : 0;
    const int unit_rows = kQTile * (pl->two_cta ? 2 : 1);
    pl->n_q_tiles = (int)((B + unit_rows - 1) / unit_rows);
    if (pl->n_q_tiles < 1) pl->n_q_tiles = 1;
    pl->rows_pad = pl->n_q_tiles * unit_rows;
    pl->S = splits_tc(pl->n_q_tiles, n_items, pl->two_cta ? sms / 2 : sms);
    pl->halves = 2;
    pl->C = cand_capacity(pl->k_keep, 128);
    {
      // streams of one row that run in the first wave; use half of them for the bound so a few
      // late streams do not hold it back
      int s_row = pl->S * pl->halves;
      const int workers = pl->two_cta ? sms / 2 : sms;
      int conc_splits = (workers + pl->n_q_tiles - 1) / pl->n_q_tiles;
      if (conc_splits > pl->S) conc_splits = pl->S;
      int s_conc = conc_splits * pl->halves;
      if (s_conc > 256) s_conc = 256;
      int use = s_conc / 2 > 1 ? s_conc / 2 : 1;
      int j = 1;
      const int kk = pl->k_keep;  // m * j distinct items must cover k plus every possibly-masked one
      while ((kk + j - 1) / j > use) j <<= 1;
      if (j > k) j = k;
      pl->share_j = s_row > 1 ? j : 0;
      pl->share_m = (kk + j - 1) / j;
      if (pl->share_m > 256 || pl->share_m > s_row) pl->share_j = 0;
    }
    // Bounded-drift throttle of the units that stream one item split (they only share its tiles through
    // L2 while they stay close; without it a leader runs away from its followers and every follower
    // misses L2 too: 99 GB instead of 15 GB of DRAM reads were measured for CTA pairs at B=4096).
    // Same-box A/B on B200, 8.84M x 768 (profiles/r02_throttle_ab.md):
    //  * lead: 16 tiles below 4 units per split (no throttle needed at 2: 6.27 vs 6.30 ms), 8 tiles from
    //    4 units per split on (B=1024 11.71 vs 11.75, 2048 21.6 vs 22.0, 4096 42.6 vs 42.9 ms); leads of
    //    2-4 tiles stall the producers on the polling itself and lose 10-30 %.
    //  * who polls: the producer itself every lead/2 tiles ("inline") is fastest up to 16 units per split
    //    (B <= 4096: 42.6 vs 46.0 ms at B=4096, 21.6 vs 28.0 at 2048); from 32 units per split on, reading
    //    32 counters serially stalls the producer and a dedicated poller warp that keeps
    //    "slowest + lead" in shared memory wins (B=8192: 84.9 vs 89.2 ms).
    //  * single CTAs (odd tile counts, B > 8192) gain from the same throttle: B=640 8.63 vs 9.16 ms, 1152
    //    13.8 vs 14.9, 16384 (poller) 183.1 vs 186.8.
    pl->throttle = pl->n_q_tiles > 1 ? 1 : 0;
    pl->lead_tiles = pl->n_q_tiles >= 4 ? 8 : 16;
    pl->throttle_poller = pl->n_q_tiles >= 32 ? 1 : 0;
  } else {
    pl->n_q_tiles = (int)((B + kSimtRows - 1) / kSimtRows);
    if (pl->n_q_tiles < 1) pl->n_q_tiles = 1;
    pl->rows_pad = pl->n_q_tiles * kSimtRows;
    long long chunks = (n_items + kSimtChunk - 1) / kSimtChunk;
    long long s = (2LL * sms + pl->n_q_tiles - 1) / pl->n_q_tiles;
    if (s > chunks) s = chunks;
    if (s < 1) s = 1;
    pl->S = (int)s;
    pl->halves = 1;
    pl->two_cta = 0;
    pl->C = cand_capacity(k, kSimtChunk);
    pl->share_j = 0; pl->share_m = 0;
    pl->throttle = 0; pl->lead_tiles = 0; pl->throttle_poller = 0;
  }
  if (kn.lead >= 1 && kn.lead <= 4096) pl->lead_tiles = kn.lead;
  pl->lead_every = 1;
  while (pl->lead_every * 2 <= pl->lead_tiles && pl->lead_every < 8) pl->lead_every *= 2;  // 16 -> 8, 8 -> 8, 4 -> 4
  Carve c;
  pl->off_cand = c.take((size_t)pl->rows_pad * pl->S * pl->halves * pl->C * sizeof(u64));
  pl->off_counts = c.take((size_t)pl->rows_pad * pl->S * pl->halves * sizeof(int));
  pl->off_rec_hi = c.take((size_t)(nnz > 0 ? nnz : 0) * sizeof(u64));
  pl->off_rec_lo = c.take((size_t)(nnz > 0 ? nnz : 0) * sizeof(u32));
  pl->zero_begin = c.off;
  pl->off_status = c.take(sizeof(DeviceStatus));
  pl->off_progress = c.take((size_t)pl->n_q_tiles * pl->S * sizeof(int));
  pl->off_gtau = c.take((size_t)pl->rows_pad * sizeof(u32));
  pl->off_gq = c.take((size_t)pl->rows_pad * pl->S * pl->halves * sizeof(u32));
  pl->off_hist = c.take((size_t)pl->rows_pad * kHistBins * sizeof(u32));
  pl->off_hpar = c.take((size_t)pl->rows_pad * sizeof(uint2));
  pl->zero_end = c.off;
  pl->off_qpad = c.take((size_t)kQTile * 4096 * sizeof(__nv_bfloat16));
  pl->seed_m = 0; pl->seed_stride = 1; pl->seed_ld = 0; pl->use_hist = 0;
  if (algo == CCR_ALGO_TCGEN05 && n_items >= (1 << 18)) {
    // strided sample of max(N/256, 64k) items (4096..131072, <= N/8); the pre-pass keeps one fp32 value
    // per 8 sampled items (their best score), capped so that matrix stays <= 512 MB
    // With histogram sharing (no mask / include mode) the seed only has to be a sensible origin for the
    // row histograms, which take over within a few tiles: a sample of N/512 (>= 8 k) is enough and
    // measurably faster (B=4096: 43.5 -> 43.0 ms, NQ k=1001: 12.4 -> 11.8 ms).  Without it (exclude-mode
    // masks) the seed is all a stream has until its first prune: N/256 and >= 64 k, so that the
    // (k+h)-th best of the sample sits in its top ~1.5 %.
    const bool hist_ok = !(nnz > 0 && !pl->include_mask);
    long long m = hist_ok ? n_items / 512 : n_items / 256;
    const long long floor_m = (hist_ok ? 16LL : 64LL) * pl->k_keep;  // >= 2 k_keep groups of 8
    if (m < floor_m) m = floor_m;
    if (m < 4096) m = 4096;
    m = (m + 255) / 256 * 256;  // whole tiles; rounding UP keeps m >= floor_m
    if (m > 131072) m = 131072;
    if (m > n_items / 8) m = n_items / 8;
    long long cap = 8LL * (512LL << 20) / (4LL * pl->rows_pad);
    if (m > cap) m = cap;
    m = m / 256 * 256;
    if (m >= 1024 && 16LL * pl->k_keep <= m) {
      pl->seed_m = (int)m;
      pl->seed_stride = n_items / m;
      pl->seed_ld = m / 8;
      // the histogram needs the seed bound as its origin and counts every streamed item, so it is
      // off in exclude-mask mode (masked items must not be counted)
      pl->use_hist = hist_ok && !kn.no_hist;
    }
  }
  // the pre-pass's score matrix (seed_ld = 0 without a pre-pass)
  pl->off_seed = c.take((size_t)pl->rows_pad * (size_t)pl->seed_ld * sizeof(float));
  pl->total = c.off;
  return true;
}

// k of a top-k over n columns: in [1, CCR_MAX_K] and, unless short rows are allowed, <= n (torch.topk's error)
int check_k(int k, long long n, bool allow_short) {
  if (k < 1 || k > CCR_MAX_K) return fail(CCR_EUNSUPPORTED, "k=%d outside [1,%d]", k, CCR_MAX_K);
  if (k > n && !allow_short) return fail(CCR_EK_RANGE, "selected index k out of range (k=%d > n=%lld)", k, n);
  return CCR_OK;
}

int check_shape(long long B, long long n_items, int D, int k, int flags) {
  if (B < 0 || n_items < 0) return fail(CCR_EINVAL, "negative size B=%lld n_items=%lld", B, n_items);
  if (B > (1LL << 24)) return fail(CCR_EUNSUPPORTED, "B=%lld > 2^24", B);
  if (n_items > (1LL << 31) - 512) return fail(CCR_EUNSUPPORTED, "n_items=%lld per shard must be < 2^31", n_items);
  if (D <= 0 || D % 8 != 0 || D > 4096) return fail(CCR_EUNSUPPORTED, "D=%d must be a multiple of 8 in [8,4096]", D);
  if (int rc = check_k(k, n_items, flags & CCR_FLAG_ALLOW_SHORT)) return rc;
  int algo = flags & CCR_ALGO_MASK;
  if (algo != CCR_ALGO_AUTO && algo != CCR_ALGO_SIMT && algo != CCR_ALGO_TCGEN05)
    return fail(CCR_EINVAL, "unknown algo flag %d", algo);
  return CCR_OK;
}

// q [B, ldq] and items [n, ldi] of the fused and exact entries: whole 16-byte rows, 16-byte aligned (TMA boxes)
int check_rows(const void* q, int64_t ldq, const void* items, int64_t ldi, int D) {
  if (ldq < D || ldi < D || ldq % 8 || ldi % 8) return fail(CCR_EINVAL, "ldq/ldi must be >= D and multiples of 8");
  if (((uintptr_t)q & 15) || ((uintptr_t)items & 15)) return fail(CCR_EINVAL, "q/items must be 16-byte aligned");
  return CCR_OK;
}

// h_max of a plan: the largest number of mask entries in one row (or a bound), < 0 when unknown or no mask
long long mask_h_max(long long nnz, long long max_row_nnz) { return nnz > 0 ? max_row_nnz : -1; }

// The mask CSR of an entry point.  A mask is present exactly when mode != CCR_MASK_NONE, indptr is set and
// nnz > 0; otherwise every field is the empty mask (null pointers, nnz 0, h_max -1, CCR_MASK_NONE).
struct MaskArgs { const long long* indptr; const int* cols; const double* vals; long long nnz, h_max; int mode; };

int parse_mask(const int64_t* indptr, const int32_t* cols, const double* vals, int64_t nnz, int64_t max_row_nnz,
               int mode, MaskArgs* m) {
  *m = {nullptr, nullptr, nullptr, 0, -1, CCR_MASK_NONE};
  if (mode != CCR_MASK_NONE && mode != CCR_MASK_SET && mode != CCR_MASK_ADD)
    return fail(CCR_EINVAL, "bad mask_mode %d", mode);
  if (mode != CCR_MASK_NONE && nnz < 0) return fail(CCR_EINVAL, "mask_nnz = %lld", (long long)nnz);
  if (mode == CCR_MASK_NONE || !indptr || nnz == 0) return CCR_OK;
  if (!cols || !vals) return fail(CCR_EINVAL, "mask_cols / mask_vals null");
  *m = {(const long long*)indptr, cols, vals, nnz, mask_h_max(nnz, max_row_nnz), mode};
  return CCR_OK;
}

// The operand fields of SelectParams: queries q [B, ldq] against table rows items [n_items, ldi], D wide (fp16 when
// f16, else bf16), in n_q_tiles query tiles and S item splits
void set_operands(SelectParams* p, const void* q, long long ldq, long long B, const void* items, long long ldi,
                  long long n_items, int D, int f16, int n_q_tiles, int S) {
  p->q = (const __nv_bfloat16*)q; p->ldq = ldq; p->B = (int)B; p->q_rows = (int)B;
  p->items = (const __nv_bfloat16*)items; p->ldi = ldi; p->n_items = n_items; p->D = D; p->f16 = f16;
  p->n_q_tiles = n_q_tiles; p->S = S;
}

// The candidate lists of a top-k call: per row, `streams` lists of C keys (cand[(row * streams + s) * C + i]) and
// their counts.  The exact re-rank has none (streams = 0).
struct Cands { int C, streams; u64* cand; int* counts; };
// finalize's entry records: the record CSR and one (hi, lo) pair per record; all null when there are none
struct Records { const long long* indptr; u64* hi; u32* lo; };

// The fields every entry-record launch shares: B rows of mask `m`, columns [0, n_cols), records written to `rec`.
// The caller adds the fields of its score source and, for the re-rank, its candidates.
RecordParams record_params(int B, RecordSource src, long long n_cols, const MaskArgs& m, const Records& rec) {
  RecordParams rp = {};
  rp.B = B; rp.src = src; rp.n_cols = n_cols;
  rp.mask_indptr = m.indptr; rp.mask_cols = m.cols; rp.mask_vals = m.vals; rp.mode = m.mode;
  rp.max_entries = m.nnz; rp.rec_hi = rec.hi; rp.rec_lo = rec.lo;
  return rp;
}

// One record per mask entry: the record CSR is the mask CSR.  Nothing to launch without a mask.
int mask_records(const RecordParams& rp, cudaStream_t st) {
  return rp.mask_indptr ? cuda_rc(launch_entry_records(rp, st), "mask record kernel launch") : CCR_OK;
}

// The last step of every top-k entry: the best k per row of the candidate lists and the entry records.  g_tau: a
// per-row lower bound of the k-th best for the prefilter, or null.  drop_cols (include mode: the mask's column
// array): a stream candidate is dropped when found in its row of the RECORD CSR, which is right because there the
// records are the mask entries (their record carries the final value).  packed_keys: out_scores64 receives
// CCR_FLAG_PACKED_KEYS keys instead of float64 values.
int finalize(int B, int k, const Cands& cb, const u32* g_tau, const Records& rec, const int* drop_cols,
             long long id_offset, float* out_scores, double* out_scores64, long long* out_ids, bool packed_keys,
             cudaStream_t st) {
  FinalizeParams fp = {};
  fp.B = B; fp.k = k; fp.C = cb.C; fp.S = cb.streams; fp.cand = cb.cand; fp.counts = cb.counts; fp.g_tau = g_tau;
  fp.rec_indptr = rec.indptr; fp.rec_hi = rec.hi; fp.rec_lo = rec.lo; fp.drop_cols = drop_cols;
  fp.id_offset = id_offset; fp.out_scores = out_scores; fp.out_ids = out_ids;
  if (packed_keys) fp.out_keys = (u64*)out_scores64;
  else fp.out_scores64 = out_scores64;
  return cuda_rc(launch_finalize(fp, st), "finalize kernel launch");
}

// The ingest / normalize entries: rows src [n, ld_src] -> dst [n, ld_dst]; `job` names the entry in the shape error
template <typename SrcT, typename DstT>
int ingest_rows(const char* job, const void* src, int64_t n, int D, int64_t ld_src, void* dst, int64_t ld_dst,
                int normalize, int* overflow, void* stream) {
  if (n < 0 || D <= 0 || ld_src < D || ld_dst < D) return fail(CCR_EINVAL, "bad %s shape", job);
  if (n == 0) return CCR_OK;
  if (!src || !dst) return fail(CCR_EINVAL, "null pointer");
  return cuda_rc(launch_ingest((const SrcT*)src, n, D, ld_src, (DstT*)dst, ld_dst, normalize, overflow,
                               (cudaStream_t)stream), "ingest kernel launch");
}
}  // namespace

extern "C" {

int ccr_abi_version(void) { return CCR_ABI_VERSION; }
const char* ccr_last_error_string(void) { return g_err; }

void ccr_set_status_record(void* host_mapped_ptr) { g_status_record = host_mapped_ptr; }
void ccr_debug_reload_env(void) { knobs(); load_knobs(); }

void ccr_set_profile_events(void* start_event, void* stop_event) {
  g_prof_start = (cudaEvent_t)start_event;
  g_prof_stop = (cudaEvent_t)stop_event;
}

int ccr_choose_algo(int64_t B, int64_t n_items, int D, int k) {
  (void)D; (void)k;
  // Measured on B200 (8.84M x 768, k=100): the TMA + tcgen05 kernel streams the table faster than
  // the CUDA-core kernel at every batch size (B=1: 3.0 vs 4.9 ms, B=8: 3.3 vs 5.2 ms) because TMA keeps
  // far more bytes in flight per SM; the 128 padded MMA rows are free in the HBM-bound regime.  The
  // CUDA-core kernel remains the choice for tiny tables with a handful of rows, where its launch is
  // cheaper than building tensor maps and running the persistent pipeline.
  return (B <= kSimtRows && n_items < 65536) ? CCR_ALGO_SIMT : CCR_ALGO_TCGEN05;
}

size_t ccr_score_topk_workspace_bytes(int64_t B, int64_t n_items, int D, int k, int64_t mask_nnz,
                                      int64_t mask_max_row_nnz, int flags) {
  if (check_shape(B, n_items, D, k, flags | CCR_FLAG_ALLOW_SHORT) != CCR_OK) return 0;
  Plan pl;
  make_plan(B, n_items, D, k, mask_nnz, mask_h_max(mask_nnz, mask_max_row_nnz), flags, &pl);
  return pl.total;
}

int ccr_plan_info(int64_t B, int64_t n_items, int D, int k, int64_t mask_nnz, int64_t mask_max_row_nnz, int flags,
                  int32_t* info8) {
  int rc = check_shape(B, n_items, D, k, flags | CCR_FLAG_ALLOW_SHORT);
  if (rc) return rc;
  if (!info8) return fail(CCR_EINVAL, "info8 is null");
  Plan pl;
  make_plan(B, n_items, D, k, mask_nnz, mask_h_max(mask_nnz, mask_max_row_nnz), flags, &pl);
  info8[0] = pl.n_q_tiles;
  info8[1] = pl.S;
  info8[2] = pl.C;
  info8[3] = pl.algo;
  info8[4] = pl.two_cta;
  info8[5] = pl.seed_m;
  // kernels one ccr_score_topk_bf16 call launches: [seeding GEMM, seed select,] fused score+select,
  // [mask-entry records,] finalize  (memsets / the short-batch query copy are not kernels of this library)
  info8[6] = (B > 0) ? (pl.seed_m > 0 ? 2 : 0) + (n_items > 0 ? 1 : 0) + (mask_nnz > 0 ? 1 : 0) + 1 : 0;
  info8[7] = pl.lead_tiles;
  return CCR_OK;
}

int ccr_score_topk_bf16(const void* q, int64_t B, int64_t ldq, const void* items, int64_t n_items,
                        int64_t ldi, int D, int k, const int64_t* mask_indptr, const int32_t* mask_cols,
                        const double* mask_vals, int64_t mask_nnz, int64_t mask_max_row_nnz, int mask_mode,
                        int64_t id_offset, float* out_scores,
                        double* out_scores64, int64_t* out_ids, void* workspace, size_t workspace_bytes,
                        int flags, void* stream) {
  int rc = check_shape(B, n_items, D, k, flags);
  if (rc) return rc;
  if (B == 0) return CCR_OK;
  if (!q || !out_ids) return fail(CCR_EINVAL, "null q / out_ids");
  if (n_items > 0 && !items) return fail(CCR_EINVAL, "null items");
  if ((rc = check_rows(q, ldq, items, ldi, D))) return rc;
  MaskArgs m;
  if ((rc = parse_mask(mask_indptr, mask_cols, mask_vals, mask_nnz, mask_max_row_nnz, mask_mode, &m))) return rc;
  if (flags & CCR_FLAG_PACKED_KEYS) {
    if (m.mode == CCR_MASK_ADD) return fail(CCR_EINVAL, "CCR_FLAG_PACKED_KEYS: float64 priors do not fit a float32 key");
    if (id_offset < 0 || id_offset + n_items > (1LL << 32)) return fail(CCR_EUNSUPPORTED, "CCR_FLAG_PACKED_KEYS: global ids must be < 2^32");
  }
  cudaStream_t st = (cudaStream_t)stream;

  Plan pl;
  make_plan(B, n_items, D, k, m.nnz, m.h_max, flags, &pl);
  if (!workspace || workspace_bytes < pl.total)
    return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, pl.total);
  unsigned char* ws = (unsigned char*)workspace;
  // watchdog record: the caller's host-mapped one (readable after a device trap) or a workspace slot
  DeviceStatus* status = g_status_record ? (DeviceStatus*)g_status_record : (DeviceStatus*)(ws + pl.off_status);
  // one memset for everything that must start from zero: status slot, throttle counters, thresholds,
  // published quantiles, histograms and their parameters
  if ((rc = cuda_rc(cudaMemsetAsync(ws + pl.zero_begin, 0, pl.zero_end - pl.zero_begin, st), "memset call state")))
    return rc;

  const Cands cb = {pl.C, pl.S * pl.halves, (u64*)(ws + pl.off_cand), (int*)(ws + pl.off_counts)};
  SelectParams sp = {};
  set_operands(&sp, q, ldq, B, items, ldi, n_items, D, (flags & CCR_FLAG_F16) ? 1 : 0, pl.n_q_tiles, pl.S);
  sp.k = k; sp.k_keep = pl.k_keep; sp.C = pl.C; sp.two_cta = pl.two_cta;
  sp.mask_indptr = m.indptr;
  sp.mask_cols = pl.include_mask ? nullptr : m.cols;
  sp.cand = cb.cand;
  sp.counts = cb.counts;
  sp.status = status;
  sp.S_row = cb.streams; sp.share_j = pl.share_j; sp.share_m = pl.share_m;
  sp.progress = pl.throttle ? (int*)(ws + pl.off_progress) : nullptr;
  sp.lead_tiles = pl.lead_tiles; sp.lead_every = pl.lead_every; sp.throttle_poller = pl.throttle_poller;
  if (pl.share_j > 0 || pl.seed_m > 0) {
    sp.g_tau = (u32*)(ws + pl.off_gtau);
    sp.g_q = (u32*)(ws + pl.off_gq);
  }
  if (pl.seed_m > 0) {
    // threshold seeding pre-pass: scores of a strided item sample -> per-row lower bound in g_tau
    SelectParams ss = sp;
    const int nqt = pl.rows_pad / kQTile;
    set_operands(&ss, q, ldq, B, items, ldi * pl.seed_stride, pl.seed_m, D, sp.f16, nqt,
                 splits_tc(nqt, pl.seed_m, pl.sms));
    ss.mask_indptr = nullptr; ss.mask_cols = nullptr;
    ss.dense_out = (float*)(ws + pl.off_seed); ss.ld_out = pl.seed_ld; ss.store_max8 = 1;
    ss.g_tau = nullptr; ss.g_q = nullptr; ss.share_j = 0; ss.progress = nullptr; ss.two_cta = 0;
    if (pl.use_hist) { sp.g_hist = (u32*)(ws + pl.off_hist); sp.g_hpar = (const uint2*)(ws + pl.off_hpar); }
    if ((rc = cuda_rc(launch_select_tc(ss, st, pl.sms), "seed GEMM launch"))) return rc;
    // per row: the (k + h)-th largest of the seed_m / 8 group maxima
    rc = cuda_rc(launch_seed_tau(ss.dense_out, pl.seed_ld, (int)pl.seed_ld, (int)B, k, m.indptr, sp.g_tau,
                                 pl.use_hist ? (uint2*)(ws + pl.off_hpar) : nullptr, st), "seed select launch");
    if (rc) return rc;
  }

  if (pl.algo == CCR_ALGO_TCGEN05 && B < kQTile && n_items > 0) {
    // short batch: stage the queries in a [128, D] block so that no TMA box of the query operand is
    // out of bounds (measurably faster than hardware zero-fill of 120+ rows); only the padding rows
    // are zeroed.  A plain copy of 2-byte elements: the same for fp16, whose +0 has bf16's bits
    __nv_bfloat16* qp = (__nv_bfloat16*)(ws + pl.off_qpad);
    cudaError_t e = cudaMemsetAsync(qp + (size_t)B * D, 0, (size_t)(kQTile - B) * D * sizeof(__nv_bfloat16), st);
    if (e == cudaSuccess)
      e = cudaMemcpy2DAsync(qp, (size_t)D * 2, q, (size_t)ldq * 2, (size_t)D * 2, (size_t)B, cudaMemcpyDeviceToDevice, st);
    if ((rc = cuda_rc(e, "query padding"))) return rc;
    sp.q = qp; sp.ldq = D; sp.q_rows = kQTile;
  }
  if (n_items == 0) {
    rc = cuda_rc(cudaMemsetAsync(cb.counts, 0, (size_t)pl.rows_pad * cb.streams * sizeof(int), st), "memset counts");
  } else {
    if (g_prof_start) cudaEventRecord(g_prof_start, st);
    const int lr = pl.algo == CCR_ALGO_TCGEN05 ? launch_select_tc(sp, st, pl.sms) : launch_select_simt(sp, st);
    if (g_prof_stop) cudaEventRecord(g_prof_stop, st);
    rc = cuda_rc(lr, "select kernel launch");
  }
  if (rc) return rc;

  const Records rec = {m.indptr, (u64*)(ws + pl.off_rec_hi), (u32*)(ws + pl.off_rec_lo)};
  RecordParams rp = record_params((int)B, sp.f16 ? kRecF16Dot : kRecBf16Dot, n_items, m, rec);
  // sp.q may be the padded staging block of a short batch: use ITS pitch (sp.ldq), not the caller's
  rp.q = sp.q; rp.ldq = sp.ldq; rp.items = sp.items; rp.ldi = ldi; rp.D = D;
  if ((rc = mask_records(rp, st))) return rc;
  return finalize((int)B, k, cb, sp.g_tau, rec, pl.include_mask ? m.cols : nullptr, id_offset, out_scores,
                  out_scores64, (long long*)out_ids, flags & CCR_FLAG_PACKED_KEYS, st);
}

int ccr_merge_topk(const double* scores64, const int64_t* ids, int G, int64_t B, int k_in, int k_out,
                   float* out_scores, double* out_scores64, int64_t* out_ids, void* stream) {
  if (G < 1 || B < 0 || k_in < 1 || k_out < 1) return fail(CCR_EINVAL, "bad merge shape G=%d B=%lld k_in=%d k_out=%d", G, (long long)B, k_in, k_out);
  if (B == 0) return CCR_OK;
  if (!scores64 || !ids || !out_ids) return fail(CCR_EINVAL, "null pointer");
  return cuda_rc(launch_merge_topk(scores64, (const long long*)ids, G, B, k_in, k_out, out_scores, out_scores64,
                                   (long long*)out_ids, (cudaStream_t)stream), "merge kernel launch");
}

int ccr_merge_topk_keys(const uint64_t* keys, int G, int64_t B, int k_in, int k_out, float* out_scores,
                        int64_t* out_ids, uint64_t* out_keys, void* stream) {
  if (G < 1 || B < 0 || k_in < 1 || k_out < 1) return fail(CCR_EINVAL, "bad merge shape G=%d B=%lld k_in=%d k_out=%d", G, (long long)B, k_in, k_out);
  if (B == 0) return CCR_OK;
  if (!keys || (!out_ids && !out_keys)) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_merge_keys((const u64*)keys, G, B, k_in, k_out, out_scores, (long long*)out_ids, (u64*)out_keys,
                             (cudaStream_t)stream);
  if (lr == (int)cudaErrorInvalidValue) return fail(CCR_EUNSUPPORTED, "merge: G * k_in = %lld keys do not fit shared memory", (long long)G * k_in);
  return cuda_rc(lr, "key merge kernel launch");
}

int ccr_unpack_topk_keys(const uint64_t* keys, int64_t n, float* out_scores, int64_t* out_ids, void* stream) {
  if (n < 0) return fail(CCR_EINVAL, "bad key count");
  if (n == 0) return CCR_OK;
  if (!keys) return fail(CCR_EINVAL, "null pointer");
  return cuda_rc(launch_unpack_keys((const u64*)keys, n, out_scores, (long long*)out_ids, (cudaStream_t)stream),
                 "key unpack kernel launch");
}

int ccr_mask_column_shard(const int64_t* indptr, const int32_t* cols, const double* vals, int64_t B, int64_t col_lo,
                          int64_t col_hi, int64_t* out_indptr, int32_t* out_cols, double* out_vals, void* stream) {
  if (B < 0 || col_lo < 0 || col_hi < col_lo || col_hi > (1LL << 31) - 1) return fail(CCR_EINVAL, "bad mask shard range");
  if (!indptr || !out_indptr) return fail(CCR_EINVAL, "null pointer");
  return cuda_rc(launch_mask_shard((const long long*)indptr, cols, vals, B, (int)col_lo, (int)col_hi,
                                   (long long*)out_indptr, out_cols, out_vals, (cudaStream_t)stream),
                 "mask shard kernel launch");
}

int ccr_ingest_rows_f32(const float* src, int64_t n, int D, int64_t ld_src, void* dst, int64_t ld_dst,
                        int normalize, void* stream) {
  return ingest_rows<float, __nv_bfloat16>("ingest", src, n, D, ld_src, dst, ld_dst, normalize, nullptr, stream);
}

int ccr_ingest_rows_f32_f16(const float* src, int64_t n, int D, int64_t ld_src, void* dst, int64_t ld_dst,
                            int normalize, int32_t* overflow_count, void* stream) {
  return ingest_rows<float, __half>("ingest", src, n, D, ld_src, dst, ld_dst, normalize, (int*)overflow_count, stream);
}

int ccr_normalize_rows_bf16(const void* src, int64_t n, int D, int64_t ld_src, void* dst, int64_t ld_dst,
                            void* stream) {
  return ingest_rows<__nv_bfloat16, __nv_bfloat16>("normalize", src, n, D, ld_src, dst, ld_dst, 1, nullptr, stream);
}

int ccr_normalize_rows_f16(const void* src, int64_t n, int D, int64_t ld_src, void* dst, int64_t ld_dst,
                           void* stream) {
  return ingest_rows<__half, __half>("normalize", src, n, D, ld_src, dst, ld_dst, 1, nullptr, stream);
}

}  // extern "C"

// ccr_score_dense_f32 / ccr_score_dense_f16: f16 selects the operand format
static int score_dense(const void* q, int64_t B, int64_t ldq, const void* items, int64_t n_items, int64_t ldi, int D,
                       float* out, int64_t ld_out, int f16, void* stream) {
  if (B < 0 || n_items < 0 || D <= 0 || D % 8 || ldq < D || ldi < D || ldq % 8 || ldi % 8 || ld_out < n_items)
    return fail(CCR_EINVAL, "bad dense shape");
  if (B == 0 || n_items == 0) return CCR_OK;
  if (!q || !items || !out) return fail(CCR_EINVAL, "null pointer");
  if (B > 65535) return fail(CCR_EUNSUPPORTED, "dense B > 65535");
  if (B * n_items >= (1LL << 20) && n_items >= kITile && n_items <= (1LL << 31) - 512 && D <= 4096 &&
      !(((uintptr_t)q | (uintptr_t)items) & 15)) {
    // large tiles: the TMA + tcgen05 pipeline of the fused kernel with a store epilogue
    const int sms = device_sm_count(), n_q_tiles = (int)((B + kQTile - 1) / kQTile);
    SelectParams sp = {};
    set_operands(&sp, q, ldq, B, items, ldi, n_items, D, f16, n_q_tiles, splits_tc(n_q_tiles, n_items, sms));
    sp.k = 1; sp.k_keep = 1; sp.C = 0;
    sp.status = (DeviceStatus*)g_status_record;
    sp.dense_out = out; sp.ld_out = ld_out; sp.store_max8 = 0;
    sp.lead_tiles = 16; sp.lead_every = 8;
    return cuda_rc(launch_select_tc(sp, (cudaStream_t)stream, sms), "dense tile launch");
  }
  const int lr = f16 ? launch_dense((const __half*)q, B, ldq, (const __half*)items, n_items, ldi, D, out, ld_out,
                                    (cudaStream_t)stream)
                     : launch_dense((const __nv_bfloat16*)q, B, ldq, (const __nv_bfloat16*)items, n_items, ldi, D,
                                    out, ld_out, (cudaStream_t)stream);
  return cuda_rc(lr, "dense kernel launch");
}

extern "C" {

int ccr_score_dense_f32(const void* q, int64_t B, int64_t ldq, const void* items, int64_t n_items,
                        int64_t ldi, int D, float* out, int64_t ld_out, void* stream) {
  return score_dense(q, B, ldq, items, n_items, ldi, D, out, ld_out, 0, stream);
}

int ccr_score_dense_f16(const void* q, int64_t B, int64_t ldq, const void* items, int64_t n_items,
                        int64_t ldi, int D, float* out, int64_t ld_out, void* stream) {
  return score_dense(q, B, ldq, items, n_items, ldi, D, out, ld_out, 1, stream);
}

size_t ccr_argsort_workspace_bytes(int64_t n_elements) {
  if (n_elements < 0 || n_elements > (1LL << 31)) return 0;
  return argsort_workspace_bytes(n_elements);
}

int ccr_argsort_scores_f32(const float* scores, int64_t B, int64_t n_cols, int64_t ld, const int64_t* mask_indptr,
                           const int32_t* mask_cols, const double* mask_vals, int64_t mask_nnz, int mask_mode,
                           int64_t* out_rows, int64_t* out_cols, void* workspace, size_t workspace_bytes, void* stream) {
  if (B < 0 || n_cols < 0 || ld < n_cols) return fail(CCR_EINVAL, "bad argsort shape");
  if (B * n_cols > (1LL << 31)) return fail(CCR_EUNSUPPORTED, "argsort: more than 2^31 matrix elements");
  MaskArgs m;
  if (int rc = parse_mask(mask_indptr, mask_cols, mask_vals, mask_nnz, -1, mask_mode, &m)) return rc;
  if (B * n_cols == 0) return CCR_OK;
  if (!scores || !out_rows || !out_cols) return fail(CCR_EINVAL, "null pointer");
  const size_t need = argsort_workspace_bytes(B * n_cols);
  if (!workspace || workspace_bytes < need) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, need);
  return cuda_rc(launch_argsort(scores, B, n_cols, ld, m.indptr, m.cols, m.vals, m.nnz, m.mode, (long long*)out_rows,
                                (long long*)out_cols, workspace, (cudaStream_t)stream), "argsort launch");
}

int ccr_first_hit_rank(const int64_t* ids, int64_t B, int k, const int64_t* rel_indptr, const int64_t* rel_ids,
                       int32_t* out_rank, void* stream) {
  if (B < 0 || k < 1) return fail(CCR_EINVAL, "bad first-hit shape");
  if (B == 0) return CCR_OK;
  if (!ids || !rel_indptr || !out_rank) return fail(CCR_EINVAL, "null pointer");
  return cuda_rc(launch_first_hit_rank((const long long*)ids, B, k, (const long long*)rel_indptr,
                                       (const long long*)rel_ids, out_rank, (cudaStream_t)stream),
                 "first-hit kernel launch");
}

// ---- top-k of a materialised dense score matrix ----
struct DensePlanC { int S, C; size_t off_cand, off_counts, off_rec_hi, off_rec_lo, total; };
static void dense_plan(long long B, long long N, int k_keep, long long nnz, DensePlanC* pl) {
  const int sms = device_sm_count();
  const long long rows = B > 0 ? B : 1;
  long long s = (8LL * sms + rows - 1) / rows;  // 8 blocks of 256 threads per SM
  const long long chunks = (N + kDenseSlack - 1) / kDenseSlack;
  if (s > chunks) s = chunks;
  if (s > 1024) s = 1024;  // finalize: kFinMaxStreams
  if (s < 1) s = 1;
  pl->S = (int)s;
  pl->C = cand_capacity(k_keep, kDenseSlack);
  Carve c;
  pl->off_cand = c.take((size_t)rows * s * pl->C * sizeof(u64));
  pl->off_counts = c.take((size_t)rows * s * sizeof(int));
  pl->off_rec_hi = c.take((size_t)(nnz > 0 ? nnz : 0) * sizeof(u64));
  pl->off_rec_lo = c.take((size_t)(nnz > 0 ? nnz : 0) * sizeof(u32));
  pl->total = c.off;
}

size_t ccr_topk_dense_workspace_bytes(int64_t B, int64_t n_cols, int k, int64_t mask_nnz, int64_t mask_max_row_nnz) {
  if (B < 0 || n_cols < 0 || k < 1 || k > CCR_MAX_K || mask_nnz < 0) return 0;
  const long long h = mask_nnz > 0 ? mask_max_row_nnz : 0;
  if (h < 0 || k + h > CCR_MAX_K) return 0;
  DensePlanC pl;
  dense_plan(B, n_cols, (int)(k + h), mask_nnz, &pl);
  return pl.total;
}

int ccr_topk_dense_f32(const float* scores, int64_t B, int64_t n_cols, int64_t ld, int k, const int64_t* mask_indptr,
                       const int32_t* mask_cols, const double* mask_vals, int64_t mask_nnz, int64_t mask_max_row_nnz,
                       int mask_mode, float* out_scores, double* out_scores64, int64_t* out_ids, void* workspace,
                       size_t workspace_bytes, void* stream) {
  if (B < 0 || n_cols < 0 || ld < n_cols) return fail(CCR_EINVAL, "bad dense top-k shape");
  if (B > 65535) return fail(CCR_EUNSUPPORTED, "dense top-k: more than 65535 rows per call");
  int rc = check_k(k, n_cols, false);
  if (rc) return rc;
  if (n_cols > (1LL << 31) - 512) return fail(CCR_EUNSUPPORTED, "n_cols must be < 2^31");
  MaskArgs m;
  if ((rc = parse_mask(mask_indptr, mask_cols, mask_vals, mask_nnz, mask_max_row_nnz, mask_mode, &m))) return rc;
  if (B == 0) return CCR_OK;
  if (!scores || !out_ids) return fail(CCR_EINVAL, "null pointer");
  // masked columns are dropped at the end: k + h candidates per row, h a bound of the mask entries in one row
  if (m.indptr && m.h_max < 0)
    return fail(CCR_EUNSUPPORTED, "dense top-k: a mask needs a known mask_max_row_nnz (got %lld)",
                (long long)mask_max_row_nnz);
  const long long h = m.indptr ? m.h_max : 0;
  if (k + h > CCR_MAX_K)
    return fail(CCR_EUNSUPPORTED, "dense top-k: k + max row nnz = %lld > %d", (long long)(k + h), CCR_MAX_K);
  DensePlanC pl;
  dense_plan(B, n_cols, (int)(k + h), m.nnz, &pl);
  if (!workspace || workspace_bytes < pl.total) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, pl.total);
  unsigned char* ws = (unsigned char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const Cands cb = {pl.C, pl.S, (u64*)(ws + pl.off_cand), (int*)(ws + pl.off_counts)};
  rc = cuda_rc(launch_select_dense(scores, ld, B, n_cols, k, (int)(k + h), m.indptr, pl.C, pl.S, cb.cand, cb.counts, st),
               "dense select launch");
  if (rc) return rc;
  const Records rec = {m.indptr, (u64*)(ws + pl.off_rec_hi), (u32*)(ws + pl.off_rec_lo)};
  RecordParams rp = record_params((int)B, kRecMatrix, n_cols, m, rec);
  rp.scores = scores; rp.ld = ld;
  if ((rc = mask_records(rp, st))) return rc;
  return finalize((int)B, k, cb, nullptr, rec, m.cols, 0, out_scores, out_scores64, (long long*)out_ids, false, st);
}

// ---- BM25 (lexical sibling of the dense path) ----
// warp = true: the warp-private kernel (S doc splits per query x kBmwWarps independent streams each);
// false: the block-wide kernel (queries with more than kBmwMaxTerms distinct terms).  streams = candidate
// lists per query handed to finalize.
struct Bm25Plan {
  int S, C, streams;
  size_t off_cand, off_counts, off_tau, total;
};

static Bm25Plan bm25_plan(long long Bq, long long N, int k, bool warp) {
  const int sms = device_sm_count();
  const long long rows = Bq > 0 ? Bq : 1;
  long long s, per_block = 1;
  Bm25Plan pl = {};
  if (warp) {
    // one resident set of blocks; finer doc splits were measured slower (more streams for finalize to
    // merge and more cursor searches than the better balance across Zipf queries buys: 42.9 ms at 1x,
    // 49.0 at 8x, 92.8 at 32x, profiles/r02_bm25.md)
    s = ((long long)kBmwBlocksPerSm * sms + rows - 1) / rows;
    const long long minis = (N + kBmwMini - 1) / kBmwMini;
    if (s * kBmwWarps > minis) s = (minis + kBmwWarps - 1) / kBmwWarps;
    if (s > 1024 / kBmwWarps) s = 1024 / kBmwWarps;  // finalize: kFinMaxStreams
    per_block = kBmwWarps;
    pl.C = cand_capacity(k, kBmwMini);   // larger buffers (fewer, longer prunes) measured slower: 34.1 ms at 2x, 36.1 at 4x
  } else {
    s = ((long long)kBmBlocksPerSm * sms + rows - 1) / rows;  // blocks resident per SM
    const long long chunks = (N + kBmChunk - 1) / kBmChunk;
    if (s > chunks) s = chunks;
    if (s > 1024) s = 1024;  // finalize: kFinMaxStreams
    pl.C = cand_capacity(k, kBmSlack);
  }
  if (s < 1) s = 1;
  pl.S = (int)s;
  pl.streams = (int)(s * per_block);
  Carve c;
  pl.off_cand = c.take((size_t)rows * (size_t)pl.streams * pl.C * sizeof(u64));
  pl.off_counts = c.take((size_t)rows * (size_t)pl.streams * sizeof(int));
  // then one u32 per query: the best stream threshold (row-level bound for finalize's prefilter)
  pl.off_tau = c.take((size_t)rows * sizeof(u32));
  pl.total = c.off;
  return pl;
}

int ccr_bm25_build_impacts(const int64_t* post_indptr, const int32_t* post_docs, const float* post_tf,
                           const double* idf, const double* doc_norm, double k1, int64_t n_terms, int64_t nnz,
                           double* post_val, void* stream) {
  if (n_terms < 0 || nnz < 0) return fail(CCR_EINVAL, "bad bm25 index shape");
  if (nnz == 0) return CCR_OK;
  if (!post_indptr || !post_docs || !post_tf || !idf || !doc_norm || !post_val) return fail(CCR_EINVAL, "null pointer");
  return cuda_rc(launch_bm25_impacts((const long long*)post_indptr, post_docs, post_tf, idf, doc_norm, k1 + 1.0,
                                     n_terms, nnz, post_val, (cudaStream_t)stream), "bm25 impacts launch");
}

size_t ccr_bm25_topk_workspace_bytes(int64_t Bq, int64_t n_docs, int k) {
  if (Bq < 0 || n_docs < 0 || k < 1 || k > CCR_MAX_K) return 0;
  // the caller does not say how long the queries are: room for either kernel
  const size_t tw = bm25_plan(Bq, n_docs, k, true).total, tb = bm25_plan(Bq, n_docs, k, false).total;
  return tw > tb ? tw : tb;
}

// The arguments both BM25 scoring entries share, checked and put in one parameter block.  The kernel is the
// warp-private one unless a query has more than kBmwMaxTerms distinct terms or CCR_BM25_BLOCKWIDE is set; k, C, S
// and the outputs are the caller's to set.
static int bm25_args(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                     const int32_t* head_slot, const double* head_rows, const int64_t* q_indptr,
                     const int32_t* q_terms, int64_t max_query_terms, int64_t Bq, int64_t n_docs, Bm25Params* p) {
  if (Bq < 0 || n_docs < 0) return fail(CCR_EINVAL, "bad bm25 shape");
  if (Bq > 65535) return fail(CCR_EUNSUPPORTED, "bm25: more than 65535 queries per call");
  if (n_docs > (1LL << 31) - 512) return fail(CCR_EUNSUPPORTED, "n_docs must be < 2^31");
  if (max_query_terms < 0 || max_query_terms > kBmMaxTerms)
    return fail(CCR_EUNSUPPORTED, "bm25: %lld distinct terms in one query (limit %d)", (long long)max_query_terms,
                kBmMaxTerms);
  if (Bq > 0 && (!q_indptr || (max_query_terms > 0 && (!q_terms || !post_indptr))))
    return fail(CCR_EINVAL, "null pointer");
  if ((head_slot == nullptr) != (head_rows == nullptr)) return fail(CCR_EINVAL, "head_slot and head_rows go together");
  *p = {};
  p->post_indptr = (const long long*)post_indptr; p->post_docs = post_docs; p->post_val = post_val;
  p->head_slot = head_slot; p->head_rows = head_rows; p->ld_head = ccr_bm25_head_row_pitch(n_docs);
  p->q_indptr = (const long long*)q_indptr; p->q_terms = q_terms; p->Bq = Bq; p->N = n_docs;
  p->warp = max_query_terms <= kBmwMaxTerms && !knobs().bm25_blockwide;
  return CCR_OK;
}

int64_t ccr_bm25_head_row_pitch(int64_t n_docs) {  // whole mini-chunks of the warp-private kernel
  return n_docs < 0 ? 0 : (n_docs + kBmwMini - 1) / kBmwMini * kBmwMini;
}

int ccr_bm25_build_head_rows(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                             const int32_t* head_terms, int n_head, int64_t n_terms, int64_t n_docs,
                             int32_t* head_slot, double* head_rows, void* stream) {
  if (n_head < 0 || n_terms < 0 || n_docs < 0) return fail(CCR_EINVAL, "bad bm25 head-row shape");
  if (n_terms > 0 && !head_slot) return fail(CCR_EINVAL, "null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  int rc = n_terms > 0 ? cuda_rc(cudaMemsetAsync(head_slot, 0xFF, (size_t)n_terms * sizeof(int32_t), st),  // all -1
                                 "memset bm25 head slots") : CCR_OK;
  if (rc || n_head == 0) return rc;
  if (!post_indptr || !post_docs || !post_val || !head_terms || !head_rows) return fail(CCR_EINVAL, "null pointer");
  if ((rc = cuda_rc(launch_bm25_head_slots(head_terms, n_head, n_terms, head_slot, st), "bm25 head slots launch")))
    return rc;
  return cuda_rc(launch_bm25_head_rows((const long long*)post_indptr, post_docs, post_val, head_terms, n_head, n_terms,
                                       ccr_bm25_head_row_pitch(n_docs), head_rows, st), "bm25 head rows launch");
}

int ccr_bm25_topk(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                  const int32_t* head_slot, const double* head_rows,
                  const int64_t* q_indptr, const int32_t* q_terms, int64_t max_query_terms, int64_t Bq,
                  int64_t n_docs, int k, float* out_scores, int64_t* out_ids, void* workspace,
                  size_t workspace_bytes, void* stream) {
  Bm25Params p;
  int rc = bm25_args(post_indptr, post_docs, post_val, head_slot, head_rows, q_indptr, q_terms, max_query_terms, Bq,
                     n_docs, &p);
  if (rc || (rc = check_k(k, n_docs, false))) return rc;
  if (Bq == 0) return CCR_OK;
  if (!out_scores || !out_ids) return fail(CCR_EINVAL, "null pointer");
  const Bm25Plan pl = bm25_plan(Bq, n_docs, k, p.warp);
  if (!workspace || workspace_bytes < pl.total) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, pl.total);
  unsigned char* ws = (unsigned char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const Cands cb = {pl.C, pl.streams, (u64*)(ws + pl.off_cand), (int*)(ws + pl.off_counts)};
  p.k = k; p.C = pl.C; p.S = pl.S; p.cand = cb.cand; p.counts = cb.counts;
  // per query: max over its streams of the stream's k-th best score (every stream that pruned holds >= k
  // docs at or above its threshold, so the row's k-th best is at least the largest of them)
  p.row_tau = (u32*)(ws + pl.off_tau);
  if ((rc = cuda_rc(cudaMemsetAsync(p.row_tau, 0, (size_t)Bq * sizeof(u32), st), "memset bm25 bounds"))) return rc;
  if ((rc = cuda_rc(launch_bm25(p, st), "bm25 top-k launch"))) return rc;
  return finalize((int)Bq, k, cb, p.warp ? p.row_tau : nullptr, {}, nullptr, 0, out_scores, nullptr,
                  (long long*)out_ids, false, st);
}

int ccr_bm25_scores_f64(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                        const int32_t* head_slot, const double* head_rows,
                        const int64_t* q_indptr, const int32_t* q_terms, int64_t max_query_terms, int64_t Bq,
                        int64_t n_docs, double* scores, int64_t ld, void* stream) {
  Bm25Params p;
  int rc = bm25_args(post_indptr, post_docs, post_val, head_slot, head_rows, q_indptr, q_terms, max_query_terms, Bq,
                     n_docs, &p);
  if (rc) return rc;
  if (ld < n_docs) return fail(CCR_EINVAL, "ld < n_docs");
  if (Bq == 0 || n_docs == 0) return CCR_OK;
  if (!scores) return fail(CCR_EINVAL, "null pointer");
  const Bm25Plan pl = bm25_plan(Bq, n_docs, 1, p.warp);
  p.k = 1; p.C = pl.C; p.S = pl.S; p.dense_out = scores; p.ld_out = ld;
  return cuda_rc(launch_bm25(p, (cudaStream_t)stream), "bm25 scores launch");
}

}  // extern "C"

// ---- exact fp32 ranking (DESIGN.md section 6b) ----
namespace {
// Exact ranking workspace: the scan stage's own (the fused call's for kc candidates per row), its [B, kc] outputs and
// the -inf values of its SET mask, then the entry records: the record CSR (B + 1 row offsets) and 12 bytes per entry.
// The re-rank alone has the records only.
struct ExactLayout {
  int kc;
  size_t scan_bytes, off_scores, off_ids, off_neg, off_rec_ip, off_rec_hi, off_rec_lo, total;
};

// L with the entry records of n_entries entries taken after c
ExactLayout add_records(ExactLayout L, Carve c, long long B, long long n_entries) {
  L.off_rec_ip = c.take((size_t)(B + 1) * sizeof(long long));
  L.off_rec_hi = c.take((size_t)(n_entries > 0 ? n_entries : 0) * sizeof(u64));
  L.off_rec_lo = c.take((size_t)(n_entries > 0 ? n_entries : 0) * sizeof(u32));
  L.total = c.off;
  return L;
}

ExactLayout exact_layout(long long B, long long n_items, int D, int k, long long nnz, long long h_max, int flags) {
  ExactLayout L = {};
  Plan pl;
  make_plan(B, n_items, D, k, 0, -1, flags, &pl);
  L.kc = pl.k_cand;
  if (L.kc > 0) {
    make_plan(B, n_items, D, L.kc, nnz, h_max, flags, &pl);
    L.scan_bytes = pl.total;
  }
  Carve c;
  c.take(L.scan_bytes);
  L.off_scores = c.take((size_t)B * L.kc * sizeof(float));
  L.off_ids = c.take((size_t)B * L.kc * sizeof(long long));
  L.off_neg = c.take((size_t)(nnz > 0 ? nnz : 0) * sizeof(double));
  return add_records(L, c, B, B * (long long)L.kc + (nnz > 0 ? nnz : 0));
}

// entry records of (candidates U mask entries) -> exact values -> finalize_kernel with no stream candidates
int rerank(const float* q, long long B, long long ldq, const float* items, long long n_items, long long ldi, int D,
           int k, const long long* cand_indptr, const long long* cand_ids, long long cand_stride, long long cand_nnz,
           const MaskArgs& m, long long id_offset, float* out_scores, double* out_scores64, long long* out_ids,
           unsigned char* ws, const ExactLayout& L, cudaStream_t st) {
  long long* rec_indptr = (long long*)(ws + L.off_rec_ip);
  const Records rec = {rec_indptr, (u64*)(ws + L.off_rec_hi), (u32*)(ws + L.off_rec_lo)};
  RecordParams rp = record_params((int)B, kRecExactDot, n_items, m, rec);
  rp.q = q; rp.ldq = ldq; rp.items = items; rp.ldi = ldi; rp.D = D;
  rp.cand_indptr = cand_indptr; rp.cand_ids = cand_ids; rp.cand_stride = cand_stride;
  rp.rec_indptr = rec_indptr; rp.max_entries = cand_nnz + m.nnz;
  int rc = cuda_rc(launch_entry_records(rp, st), "exact value kernel launch");
  if (rc) return rc;
  return finalize((int)B, k, {}, nullptr, rec, nullptr, id_offset, out_scores, out_scores64, out_ids, false, st);
}
}  // namespace

extern "C" {

double ccr_exact_error_bound(double q_norm, double max_row_norm, int D, int flags) {
  return exact_error_bound(q_norm, max_row_norm, D, (flags & CCR_FLAG_F16) ? 1 : 0);
}

int ccr_exact_k_candidates(int64_t B, int64_t n_items, int D, int k, int flags) {
  int rc = check_shape(B, n_items, D, k, flags | CCR_FLAG_ALLOW_SHORT);
  if (rc) return rc;
  Plan pl;
  make_plan(B, n_items, D, k, 0, -1, flags, &pl);
  return pl.k_cand;
}

int ccr_ingest_rows_f32_f32(const float* src, int64_t n, int D, int64_t ld_src, float* dst, int64_t ld_dst,
                            int normalize, double* max_row_norm, void* stream) {
  int rc = ingest_rows<float, float>("ingest", src, n, D, ld_src, dst, ld_dst, normalize, nullptr, stream);
  if (rc || !max_row_norm) return rc;
  return cuda_rc(launch_row_norm_max(dst, n, D, ld_dst, max_row_norm, (cudaStream_t)stream), "row norm kernel launch");
}

size_t ccr_score_topk_exact_workspace_bytes(int64_t B, int64_t n_items, int D, int k, int64_t mask_nnz,
                                            int64_t mask_max_row_nnz, int flags) {
  if (check_shape(B, n_items, D, k, flags | CCR_FLAG_ALLOW_SHORT) != CCR_OK || mask_nnz < 0) return 0;
  return exact_layout(B, n_items, D, k, mask_nnz, mask_h_max(mask_nnz, mask_max_row_nnz), flags).total;
}

int ccr_score_topk_exact(const float* q, const void* q_scan, int64_t B, int64_t ldq, const float* items,
                         const void* items_scan, int64_t n_items, int64_t ldi, int D, int k,
                         const double* max_row_norm, const int64_t* mask_indptr, const int32_t* mask_cols,
                         const double* mask_vals, int64_t mask_nnz, int64_t mask_max_row_nnz, int mask_mode,
                         int64_t id_offset, float* out_scores, double* out_scores64, int64_t* out_ids,
                         int32_t* out_uncertified, double* out_tau, int32_t* uncertified_count, void* workspace,
                         size_t workspace_bytes, int flags, void* stream) {
  int rc = check_shape(B, n_items, D, k, flags);
  if (rc) return rc;
  if (flags & CCR_FLAG_PACKED_KEYS) return fail(CCR_EINVAL, "exact ranking returns float64 values, not packed keys");
  if (B == 0) return CCR_OK;
  if (!q || !q_scan || !out_ids || !out_scores64 || !out_uncertified || !out_tau || !uncertified_count || !max_row_norm)
    return fail(CCR_EINVAL, "null q / q_scan / out_ids / out_scores64 / certificate outputs / max_row_norm");
  if (n_items > 0 && (!items || !items_scan)) return fail(CCR_EINVAL, "null items");
  if ((rc = check_rows(q, ldq, items, ldi, D)) || (rc = check_rows(q_scan, ldq, items_scan, ldi, D))) return rc;
  MaskArgs m;
  if ((rc = parse_mask(mask_indptr, mask_cols, mask_vals, mask_nnz, mask_max_row_nnz, mask_mode, &m))) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const ExactLayout L = exact_layout(B, n_items, D, k, m.nnz, m.h_max, flags);
  const int kc = L.kc;
  if (!workspace || workspace_bytes < L.total) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, L.total);
  unsigned char* ws = (unsigned char*)workspace;
  float* s1_scores = (float*)(ws + L.off_scores);
  long long* s1_ids = (long long*)(ws + L.off_ids);
  if (kc > 0) {
    // stage 1: the unchanged scan on the scan copies, every mask entry ranked last (SET -inf) so that none
    // takes a candidate slot; the re-rank below gives each its true value
    double* neg = (double*)(ws + L.off_neg);
    if ((rc = cuda_rc(launch_fill_f64(neg, m.nnz, -INFINITY, st), "fill launch"))) return rc;
    rc = ccr_score_topk_bf16(q_scan, B, ldq, items_scan, n_items, ldi, D, kc, (const int64_t*)m.indptr, m.cols, neg,
                             m.nnz, m.h_max, CCR_MASK_SET, 0, s1_scores, nullptr, (int64_t*)s1_ids, ws, L.scan_bytes,
                             flags & (CCR_ALGO_MASK | CCR_FLAG_F16), stream);
    if (rc) return rc;
  }
  rc = rerank(q, B, ldq, items, n_items, ldi, D, k, nullptr, s1_ids, kc, B * (long long)kc, m, id_offset, out_scores,
              out_scores64, (long long*)out_ids, ws, L, st);
  if (rc) return rc;
  return cuda_rc(launch_exact_certify(q, ldq, (int)B, D, (flags & CCR_FLAG_F16) ? 1 : 0, max_row_norm, k, kc, n_items,
                                      s1_scores, s1_ids, m.indptr, m.cols, out_scores64, knobs().exact_fallback,
                                      out_uncertified, out_tau, uncertified_count, st), "certify kernel launch");
}

size_t ccr_rerank_exact_workspace_bytes(int64_t B, int64_t cand_nnz, int64_t mask_nnz) {
  if (B < 0 || cand_nnz < 0 || mask_nnz < 0) return 0;
  return add_records({}, {}, B, cand_nnz + mask_nnz).total;
}

int ccr_rerank_exact(const float* q, int64_t B, int64_t ldq, const float* items, int64_t n_items, int64_t ldi, int D,
                     int k, const int64_t* cand_indptr, const int64_t* cand_ids, int64_t cand_nnz,
                     const int64_t* mask_indptr, const int32_t* mask_cols, const double* mask_vals, int64_t mask_nnz,
                     int mask_mode, int64_t id_offset, float* out_scores, double* out_scores64, int64_t* out_ids,
                     void* workspace, size_t workspace_bytes, int flags, void* stream) {
  int rc = check_shape(B, n_items, D, k, flags);
  if (rc) return rc;
  if (B == 0) return CCR_OK;
  if (!q || !out_ids || !cand_indptr || (cand_nnz > 0 && !cand_ids)) return fail(CCR_EINVAL, "null q / out_ids / candidates");
  if (cand_nnz < 0) return fail(CCR_EINVAL, "cand_nnz = %lld", (long long)cand_nnz);
  if (n_items > 0 && !items) return fail(CCR_EINVAL, "null items");
  if ((rc = check_rows(q, ldq, items, ldi, D))) return rc;
  MaskArgs m;
  if ((rc = parse_mask(mask_indptr, mask_cols, mask_vals, mask_nnz, -1, mask_mode, &m))) return rc;
  const ExactLayout L = add_records({}, {}, B, cand_nnz + m.nnz);
  if (!workspace || workspace_bytes < L.total) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, L.total);
  return rerank(q, B, ldq, items, n_items, ldi, D, k, (const long long*)cand_indptr, (const long long*)cand_ids, 0,
                cand_nnz, m, id_offset, out_scores, out_scores64, (long long*)out_ids, (unsigned char*)workspace, L,
                (cudaStream_t)stream);
}

int ccr_score_dense_exact(const float* q, int64_t B, int64_t ldq, const float* items, int64_t n_items, int64_t ldi,
                          int D, float* out, int64_t ld_out, void* stream) {
  if (B < 0 || n_items < 0 || ld_out < n_items) return fail(CCR_EINVAL, "bad exact dense shape");
  if (D <= 0 || D % 8) return fail(CCR_EINVAL, "D=%d must be a positive multiple of 8", D);
  if (D > 4096) return fail(CCR_EUNSUPPORTED, "D=%d > 4096", D);
  if (ldq < D || ldi < D || ldq % 8 || ldi % 8) return fail(CCR_EINVAL, "ldq/ldi must be >= D and multiples of 8");
  if (B == 0 || n_items == 0) return CCR_OK;
  if (!q || !items || !out) return fail(CCR_EINVAL, "null pointer");
  if (int rc = check_rows(q, ldq, items, ldi, D)) return rc;
  return cuda_rc(launch_dense_exact(q, B, ldq, items, n_items, ldi, D, out, ld_out, (cudaStream_t)stream),
                 "exact dense kernel launch");
}

int ccr_threshold_compact(const float* scores, int64_t R, int64_t N, int64_t ld, const double* tau,
                          int64_t* out_indptr, int64_t* out_ids, void* stream) {
  if (R < 0 || N < 0 || ld < N) return fail(CCR_EINVAL, "bad compaction shape");
  if (R == 0) return CCR_OK;
  if (!tau || !out_indptr || (N > 0 && !scores)) return fail(CCR_EINVAL, "null pointer");
  return cuda_rc(launch_threshold_compact(scores, R, N, ld, tau, (long long*)out_indptr, (long long*)out_ids,
                                          (cudaStream_t)stream), "compaction launch");
}

}  // extern "C"
