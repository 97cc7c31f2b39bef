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
  int two_cta = -1, lead = 0, no_hist = 0, bm25_blockwide = 0;
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
struct Plan {
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
  size_t off_seed;
  size_t off_progress;
  size_t off_qpad;       // zero-padded copy of a short query batch (B < 128): every TMA box in bounds
  size_t off_cand, off_counts, off_ovr_hi, off_ovr_lo, off_status, off_gtau, off_gq, off_hist, off_hpar, total;
};

size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

int splits_tc(int nq, long long tiles, int sms) {
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
  pl->algo = algo;
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
    long long tiles = (n_items + kITile - 1) / kITile;
    pl->S = splits_tc(pl->n_q_tiles, tiles, pl->two_cta ? sms / 2 : sms);
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
  size_t off = 0;
  pl->off_cand = off;   off = align_up(off + (size_t)pl->rows_pad * pl->S * pl->halves * pl->C * sizeof(u64), 256);
  pl->off_counts = off; off = align_up(off + (size_t)pl->rows_pad * pl->S * pl->halves * sizeof(int), 256);
  pl->off_ovr_hi = off; off = align_up(off + (size_t)(nnz > 0 ? nnz : 0) * sizeof(u64), 256);
  pl->off_ovr_lo = off; off = align_up(off + (size_t)(nnz > 0 ? nnz : 0) * sizeof(u32), 256);
  // [off_status, off_qpad) is zeroed by ONE memset per call: status, throttle counters, sharing state
  pl->off_status = off; off = align_up(off + sizeof(DeviceStatus), 256);
  pl->off_progress = off; off = align_up(off + (size_t)pl->n_q_tiles * pl->S * sizeof(int), 256);
  pl->off_gtau = off;   off = align_up(off + (size_t)pl->rows_pad * sizeof(u32), 256);
  pl->off_gq = off;     off = align_up(off + (size_t)pl->rows_pad * pl->S * pl->halves * sizeof(u32), 256);
  pl->off_hist = off;   off = align_up(off + (size_t)pl->rows_pad * kHistBins * sizeof(u32), 256);
  pl->off_hpar = off;   off = align_up(off + (size_t)pl->rows_pad * sizeof(uint2), 256);
  pl->off_qpad = off;     off = align_up(off + (size_t)kQTile * 4096 * sizeof(__nv_bfloat16), 256);
  pl->seed_m = 0; pl->seed_stride = 1; pl->seed_ld = 0; pl->off_seed = off; pl->use_hist = 0;
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
      off = align_up(off + (size_t)pl->rows_pad * (size_t)pl->seed_ld * sizeof(float), 256);
    }
  }
  pl->total = off;
  return true;
}

int check_shape(long long B, long long n_items, int D, int k, int flags) {
  if (B < 0 || n_items < 0) return fail(CCR_EINVAL, "negative size B=%lld n_items=%lld", B, n_items);
  if (B > (1LL << 24)) return fail(CCR_EUNSUPPORTED, "B=%lld > 2^24", B);
  if (n_items > (1LL << 31) - 512) return fail(CCR_EUNSUPPORTED, "n_items=%lld per shard must be < 2^31", n_items);
  if (D <= 0 || D % 8 != 0 || D > 4096) return fail(CCR_EUNSUPPORTED, "D=%d must be a multiple of 8 in [8,4096]", D);
  if (k < 1 || k > CCR_MAX_K) return fail(CCR_EUNSUPPORTED, "k=%d outside [1,%d]", k, CCR_MAX_K);
  if (k > n_items && !(flags & CCR_FLAG_ALLOW_SHORT))
    return fail(CCR_EK_RANGE, "selected index k out of range (k=%d > n_items=%lld)", k, n_items);
  int algo = flags & CCR_ALGO_MASK;
  if (algo != CCR_ALGO_AUTO && algo != CCR_ALGO_SIMT && algo != CCR_ALGO_TCGEN05)
    return fail(CCR_EINVAL, "unknown algo flag %d", algo);
  return CCR_OK;
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
  make_plan(B, n_items, D, k, mask_nnz, mask_nnz > 0 ? mask_max_row_nnz : -1, flags, &pl);
  return pl.total;
}

int ccr_plan_info(int64_t B, int64_t n_items, int D, int k, int64_t mask_nnz, int64_t mask_max_row_nnz, int flags,
                  int32_t* info8) {
  int rc = check_shape(B, n_items, D, k, flags | CCR_FLAG_ALLOW_SHORT);
  if (rc) return rc;
  if (!info8) return fail(CCR_EINVAL, "info8 is null");
  Plan pl;
  make_plan(B, n_items, D, k, mask_nnz, mask_nnz > 0 ? mask_max_row_nnz : -1, flags, &pl);
  info8[0] = pl.n_q_tiles;
  info8[1] = pl.S;
  info8[2] = pl.C;
  info8[3] = pl.algo;
  info8[4] = pl.two_cta;
  info8[5] = pl.seed_m;
  // kernels one ccr_score_topk_bf16 call launches: [seeding GEMM, seed select,] fused score+select,
  // [mask overrides,] finalize  (memsets / the short-batch query copy are not kernels of this library)
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
  if (ldq < D || ldi < D || ldq % 8 || ldi % 8) return fail(CCR_EINVAL, "ldq/ldi must be >= D and multiples of 8");
  if (((uintptr_t)q & 15) || ((uintptr_t)items & 15)) return fail(CCR_EINVAL, "q/items must be 16-byte aligned");
  if (mask_mode != CCR_MASK_NONE && mask_mode != CCR_MASK_SET && mask_mode != CCR_MASK_ADD)
    return fail(CCR_EINVAL, "bad mask_mode %d", mask_mode);
  const bool has_mask = mask_mode != CCR_MASK_NONE && mask_indptr != nullptr;
  if (has_mask && (!mask_cols || !mask_vals)) return fail(CCR_EINVAL, "mask_cols / mask_vals null");
  if (flags & CCR_FLAG_PACKED_KEYS) {
    if (mask_mode == CCR_MASK_ADD) return fail(CCR_EINVAL, "CCR_FLAG_PACKED_KEYS: float64 priors do not fit a float32 key");
    if (id_offset < 0 || id_offset + n_items > (1LL << 32)) return fail(CCR_EUNSUPPORTED, "CCR_FLAG_PACKED_KEYS: global ids must be < 2^32");
  }
  cudaStream_t st = (cudaStream_t)stream;

  const long long nnz = has_mask ? mask_nnz : 0;
  if (nnz < 0) return fail(CCR_EINVAL, "mask_nnz = %lld", nnz);
  Plan pl;
  make_plan(B, n_items, D, k, nnz, nnz > 0 ? mask_max_row_nnz : -1, flags, &pl);
  if (!workspace || workspace_bytes < pl.total)
    return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, pl.total);
  unsigned char* ws = (unsigned char*)workspace;
  // watchdog record: the caller's host-mapped one (readable after a device trap) or a workspace slot
  DeviceStatus* status = g_status_record ? (DeviceStatus*)g_status_record : (DeviceStatus*)(ws + pl.off_status);
  // one memset for everything that must start from zero: status slot, throttle counters, thresholds,
  // published quantiles, histograms and their parameters
  cudaError_t e = cudaMemsetAsync(ws + pl.off_status, 0, pl.off_qpad - pl.off_status, st);
  if (e != cudaSuccess) return fail(CCR_ECUDA, "memset call state: %s", cudaGetErrorString(e));

  SelectParams sp = {};
  sp.q = (const __nv_bfloat16*)q; sp.ldq = ldq; sp.B = (int)B; sp.q_rows = (int)B;
  sp.items = (const __nv_bfloat16*)items; sp.ldi = ldi; sp.n_items = n_items; sp.D = D;
  sp.k = k; sp.k_keep = pl.k_keep; sp.C = pl.C; sp.S = pl.S; sp.n_q_tiles = pl.n_q_tiles; sp.two_cta = pl.two_cta;
  sp.mask_indptr = has_mask ? (const long long*)mask_indptr : nullptr;
  sp.mask_cols = (has_mask && !pl.include_mask) ? mask_cols : nullptr;
  sp.cand = (u64*)(ws + pl.off_cand);
  sp.counts = (int*)(ws + pl.off_counts);
  sp.status = status;
  sp.g_tau = nullptr; sp.g_q = nullptr; sp.S_row = pl.S * pl.halves; sp.share_j = pl.share_j; sp.share_m = pl.share_m;
  sp.dense_out = nullptr; sp.ld_out = 0; sp.store_max8 = 0;
  sp.g_hist = nullptr; sp.g_hpar = nullptr;
  sp.progress = pl.throttle ? (int*)(ws + pl.off_progress) : nullptr;
  sp.lead_tiles = pl.lead_tiles; sp.lead_every = pl.lead_every; sp.throttle_poller = pl.throttle_poller;
  if (pl.share_j > 0 || pl.seed_m > 0) {
    sp.g_tau = (u32*)(ws + pl.off_gtau);
    sp.g_q = (u32*)(ws + pl.off_gq);
  }
  if (pl.seed_m > 0) {
    // threshold seeding pre-pass: scores of a strided item sample -> per-row lower bound in g_tau
    SelectParams ss = sp;
    ss.n_items = pl.seed_m; ss.ldi = ldi * pl.seed_stride;
    ss.mask_indptr = nullptr; ss.mask_cols = nullptr;
    ss.dense_out = (float*)(ws + pl.off_seed); ss.ld_out = pl.seed_ld; ss.store_max8 = 1;
    ss.g_tau = nullptr; ss.g_q = nullptr; ss.share_j = 0; ss.progress = nullptr;
    if (pl.use_hist) { sp.g_hist = (u32*)(ws + pl.off_hist); sp.g_hpar = (const uint2*)(ws + pl.off_hpar); }
    ss.two_cta = 0; ss.n_q_tiles = pl.rows_pad / kQTile;
    long long tiles = (pl.seed_m + kITile - 1) / kITile;
    ss.S = splits_tc(ss.n_q_tiles, tiles, device_sm_count());
    int lr0 = launch_select_tc(ss, st, device_sm_count());
    if (lr0) return fail(CCR_ECUDA, "seed GEMM launch failed (%d)", lr0);
    // per row: the (k + h)-th largest of the seed_m / 8 group maxima
    lr0 = launch_seed_tau(ss.dense_out, pl.seed_ld, (int)pl.seed_ld, (int)B, k, has_mask ? (const long long*)mask_indptr : nullptr,
                          sp.g_tau, pl.use_hist ? (uint2*)(ws + pl.off_hpar) : nullptr, st);
    if (lr0) return fail(CCR_ECUDA, "seed select launch failed: %s", cudaGetErrorString((cudaError_t)lr0));
  }

  if (pl.algo == CCR_ALGO_TCGEN05 && B < kQTile && n_items > 0) {
    // short batch: stage the queries in a [128, D] block so that no TMA box of the query operand is
    // out of bounds (measurably faster than hardware zero-fill of 120+ rows); only the padding rows
    // are zeroed
    __nv_bfloat16* qp = (__nv_bfloat16*)(ws + pl.off_qpad);
    e = cudaMemsetAsync(qp + (size_t)B * D, 0, (size_t)(kQTile - B) * D * sizeof(__nv_bfloat16), st);
    if (e == cudaSuccess)
      e = cudaMemcpy2DAsync(qp, (size_t)D * 2, q, (size_t)ldq * 2, (size_t)D * 2, (size_t)B, cudaMemcpyDeviceToDevice, st);
    if (e != cudaSuccess) return fail(CCR_ECUDA, "query padding: %s", cudaGetErrorString(e));
    sp.q = qp; sp.ldq = D; sp.q_rows = kQTile;
  }
  int lr = 0;
  if (n_items == 0) {
    e = cudaMemsetAsync(sp.counts, 0, (size_t)pl.rows_pad * pl.S * pl.halves * sizeof(int), st);
    if (e != cudaSuccess) return fail(CCR_ECUDA, "memset counts: %s", cudaGetErrorString(e));
  } else {
    if (g_prof_start) cudaEventRecord(g_prof_start, st);
    if (pl.algo == CCR_ALGO_TCGEN05) lr = launch_select_tc(sp, st, device_sm_count());
    else lr = launch_select_simt(sp, st);
    if (g_prof_stop) cudaEventRecord(g_prof_stop, st);
  }
  if (lr) return fail(CCR_ECUDA, "select kernel launch failed (%d: %s)", lr, lr > 0 ? cudaGetErrorString((cudaError_t)lr) : "tensor map");

  if (has_mask && nnz > 0) {
    OverrideParams op = {};
    // sp.q may be the padded staging block of a short batch: use ITS pitch (sp.ldq), not the caller's
    op.q = sp.q; op.ldq = sp.ldq; op.B = (int)B; op.items = sp.items; op.ldi = ldi; op.n_items = n_items; op.D = D;
    op.mask_indptr = sp.mask_indptr; op.mask_cols = mask_cols; op.mask_vals = mask_vals; op.nnz = nnz;
    op.mode = mask_mode; op.ovr_hi = (u64*)(ws + pl.off_ovr_hi); op.ovr_lo = (u32*)(ws + pl.off_ovr_lo);
    lr = launch_overrides(op, st);
    if (lr) return fail(CCR_ECUDA, "override kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  }

  FinalizeParams fp = {};
  fp.B = (int)B; fp.k = k; fp.C = pl.C; fp.S = pl.S * pl.halves; fp.cand = sp.cand; fp.counts = sp.counts;
  fp.g_tau = sp.g_tau;
  fp.drop_cols = (has_mask && nnz > 0 && pl.include_mask) ? mask_cols : nullptr;
  fp.mask_indptr = (has_mask && nnz > 0) ? sp.mask_indptr : nullptr;
  fp.ovr_hi = (u64*)(ws + pl.off_ovr_hi); fp.ovr_lo = (u32*)(ws + pl.off_ovr_lo);
  fp.id_offset = id_offset; fp.out_scores = out_scores; fp.out_scores64 = out_scores64;
  fp.out_keys = nullptr;
  if (flags & CCR_FLAG_PACKED_KEYS) { fp.out_keys = (u64*)out_scores64; fp.out_scores64 = nullptr; }
  fp.out_ids = (long long*)out_ids;
  lr = launch_finalize(fp, st);
  if (lr) return fail(CCR_ECUDA, "finalize kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_merge_topk(const double* scores64, const int64_t* ids, int G, int64_t B, int k_in, int k_out,
                   float* out_scores, double* out_scores64, int64_t* out_ids, void* stream) {
  if (G < 1 || B < 0 || k_in < 1 || k_out < 1) return fail(CCR_EINVAL, "bad merge shape G=%d B=%lld k_in=%d k_out=%d", G, (long long)B, k_in, k_out);
  if (B == 0) return CCR_OK;
  if (!scores64 || !ids || !out_ids) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_merge_topk(scores64, (const long long*)ids, G, B, k_in, k_out, out_scores, out_scores64,
                             (long long*)out_ids, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "merge kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_merge_topk_keys(const uint64_t* keys, int G, int64_t B, int k_in, int k_out, float* out_scores,
                        int64_t* out_ids, uint64_t* out_keys, void* stream) {
  if (G < 1 || B < 0 || k_in < 1 || k_out < 1) return fail(CCR_EINVAL, "bad merge shape G=%d B=%lld k_in=%d k_out=%d", G, (long long)B, k_in, k_out);
  if (B == 0) return CCR_OK;
  if (!keys || (!out_ids && !out_keys)) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_merge_keys((const u64*)keys, G, B, k_in, k_out, out_scores, (long long*)out_ids, (u64*)out_keys,
                             (cudaStream_t)stream);
  if (lr == (int)cudaErrorInvalidValue) return fail(CCR_EUNSUPPORTED, "merge: G * k_in = %lld keys do not fit shared memory", (long long)G * k_in);
  if (lr) return fail(CCR_ECUDA, "key merge kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_unpack_topk_keys(const uint64_t* keys, int64_t n, float* out_scores, int64_t* out_ids, void* stream) {
  if (n < 0) return fail(CCR_EINVAL, "bad key count");
  if (n == 0) return CCR_OK;
  if (!keys) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_unpack_keys((const u64*)keys, n, out_scores, (long long*)out_ids, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "key unpack kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_mask_column_shard(const int64_t* indptr, const int32_t* cols, const double* vals, int64_t B, int64_t col_lo,
                          int64_t col_hi, int64_t* out_indptr, int32_t* out_cols, double* out_vals, void* stream) {
  if (B < 0 || col_lo < 0 || col_hi < col_lo || col_hi > (1LL << 31) - 1) return fail(CCR_EINVAL, "bad mask shard range");
  if (!indptr || !out_indptr) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_mask_shard((const long long*)indptr, cols, vals, B, (int)col_lo, (int)col_hi, (long long*)out_indptr,
                             out_cols, out_vals, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "mask shard kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_ingest_rows_f32(const float* src, int64_t n, int D, int64_t ld_src, void* dst, int64_t ld_dst,
                        int normalize, void* stream) {
  if (n < 0 || D <= 0 || ld_src < D || ld_dst < D) return fail(CCR_EINVAL, "bad ingest shape");
  if (n == 0) return CCR_OK;
  if (!src || !dst) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_ingest_f32(src, n, D, ld_src, (__nv_bfloat16*)dst, ld_dst, normalize, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "ingest kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_normalize_rows_bf16(const void* src, int64_t n, int D, int64_t ld_src, void* dst, int64_t ld_dst,
                            void* stream) {
  if (n < 0 || D <= 0 || ld_src < D || ld_dst < D) return fail(CCR_EINVAL, "bad normalize shape");
  if (n == 0) return CCR_OK;
  if (!src || !dst) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_normalize_bf16((const __nv_bfloat16*)src, n, D, ld_src, (__nv_bfloat16*)dst, ld_dst,
                                 (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "normalize kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_score_dense_f32(const void* q, int64_t B, int64_t ldq, const void* items, int64_t n_items,
                        int64_t ldi, int D, float* out, int64_t ld_out, void* stream) {
  if (B < 0 || n_items < 0 || D <= 0 || D % 8 || ldq < D || ldi < D || ldq % 8 || ldi % 8 || ld_out < n_items)
    return fail(CCR_EINVAL, "bad dense shape");
  if (B == 0 || n_items == 0) return CCR_OK;
  if (!q || !items || !out) return fail(CCR_EINVAL, "null pointer");
  if (B > 65535) return fail(CCR_EUNSUPPORTED, "dense B > 65535");
  if (B * n_items >= (1LL << 20) && n_items >= kITile && n_items <= (1LL << 31) - 512 && D <= 4096 &&
      !(((uintptr_t)q | (uintptr_t)items) & 15)) {
    // large tiles: the TMA + tcgen05 pipeline of the fused kernel with a store epilogue
    SelectParams sp = {};
    sp.q = (const __nv_bfloat16*)q; sp.ldq = ldq; sp.B = (int)B; sp.q_rows = (int)B;
    sp.items = (const __nv_bfloat16*)items; sp.ldi = ldi; sp.n_items = n_items; sp.D = D;
    sp.k = 1; sp.k_keep = 1; sp.C = 0;
    sp.n_q_tiles = (int)((B + kQTile - 1) / kQTile);
    sp.S = splits_tc(sp.n_q_tiles, (n_items + kITile - 1) / kITile, device_sm_count());
    sp.status = (DeviceStatus*)g_status_record;
    sp.dense_out = out; sp.ld_out = ld_out; sp.store_max8 = 0;
    sp.lead_tiles = 16; sp.lead_every = 8;
    int lr = launch_select_tc(sp, (cudaStream_t)stream, device_sm_count());
    if (lr) return fail(CCR_ECUDA, "dense tile launch failed (%d)", lr);
    return CCR_OK;
  }
  int lr = launch_dense_f32((const __nv_bfloat16*)q, B, ldq, (const __nv_bfloat16*)items, n_items, ldi, D, out,
                            ld_out, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "dense kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
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
  if (mask_mode != CCR_MASK_NONE && mask_mode != CCR_MASK_SET && mask_mode != CCR_MASK_ADD)
    return fail(CCR_EINVAL, "bad mask_mode %d", mask_mode);
  if (B * n_cols == 0) return CCR_OK;
  if (!scores || !out_rows || !out_cols) return fail(CCR_EINVAL, "null pointer");
  const bool has_mask = mask_mode != CCR_MASK_NONE && mask_indptr != nullptr && mask_nnz > 0;
  if (has_mask && (!mask_cols || !mask_vals)) return fail(CCR_EINVAL, "mask_cols / mask_vals null");
  const size_t need = argsort_workspace_bytes(B * n_cols);
  if (!workspace || workspace_bytes < need) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, need);
  int lr = launch_argsort(scores, B, n_cols, ld, has_mask ? (const long long*)mask_indptr : nullptr, mask_cols, mask_vals,
                          has_mask ? mask_nnz : 0, mask_mode, (long long*)out_rows, (long long*)out_cols, workspace,
                          (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "argsort launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_first_hit_rank(const int64_t* ids, int64_t B, int k, const int64_t* rel_indptr, const int64_t* rel_ids,
                       int32_t* out_rank, void* stream) {
  if (B < 0 || k < 1) return fail(CCR_EINVAL, "bad first-hit shape");
  if (B == 0) return CCR_OK;
  if (!ids || !rel_indptr || !out_rank) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_first_hit_rank((const long long*)ids, B, k, (const long long*)rel_indptr, (const long long*)rel_ids,
                                 out_rank, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "first-hit kernel launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

// ---- top-k of a materialised dense score matrix ----
struct DensePlanC { int S, C; size_t off_counts, off_ovr_hi, off_ovr_lo, total; };
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
  size_t off = align_up((size_t)rows * s * pl->C * sizeof(u64), 256);
  pl->off_counts = off; off = align_up(off + (size_t)rows * s * sizeof(int), 256);
  pl->off_ovr_hi = off; off = align_up(off + (size_t)(nnz > 0 ? nnz : 0) * sizeof(u64), 256);
  pl->off_ovr_lo = off; off = align_up(off + (size_t)(nnz > 0 ? nnz : 0) * sizeof(u32), 256);
  pl->total = off;
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
  if (k < 1 || k > CCR_MAX_K) return fail(CCR_EUNSUPPORTED, "k=%d outside [1,%d]", k, CCR_MAX_K);
  if (k > n_cols) return fail(CCR_EK_RANGE, "selected index k out of range (k=%d > n=%lld)", k, (long long)n_cols);
  if (n_cols > (1LL << 31) - 512) return fail(CCR_EUNSUPPORTED, "n_cols must be < 2^31");
  if (mask_mode != CCR_MASK_NONE && mask_mode != CCR_MASK_SET && mask_mode != CCR_MASK_ADD)
    return fail(CCR_EINVAL, "bad mask_mode %d", mask_mode);
  if (B == 0) return CCR_OK;
  if (!scores || !out_ids) return fail(CCR_EINVAL, "null pointer");
  const bool has_mask = mask_mode != CCR_MASK_NONE && mask_indptr != nullptr && mask_nnz > 0;
  if (has_mask && (!mask_cols || !mask_vals)) return fail(CCR_EINVAL, "mask_cols / mask_vals null");
  const long long nnz = has_mask ? mask_nnz : 0;
  const long long h = has_mask ? mask_max_row_nnz : 0;
  if (h < 0 || k + h > CCR_MAX_K)
    return fail(CCR_EUNSUPPORTED, "dense top-k: k + max row nnz = %lld outside [1,%d]", (long long)(k + h), CCR_MAX_K);
  DensePlanC pl;
  dense_plan(B, n_cols, (int)(k + h), nnz, &pl);
  if (!workspace || workspace_bytes < pl.total) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, pl.total);
  unsigned char* ws = (unsigned char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const long long* indptr = has_mask ? (const long long*)mask_indptr : nullptr;
  int lr = launch_select_dense(scores, ld, B, n_cols, k, (int)(k + h), indptr, pl.C, pl.S, (u64*)ws, (int*)(ws + pl.off_counts), st);
  if (lr) return fail(CCR_ECUDA, "dense select launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  if (has_mask) {
    lr = launch_override_dense(scores, ld, (int)B, n_cols, indptr, mask_cols, mask_vals, nnz, mask_mode,
                               (u64*)(ws + pl.off_ovr_hi), (u32*)(ws + pl.off_ovr_lo), st);
    if (lr) return fail(CCR_ECUDA, "dense override launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  }
  FinalizeParams fp = {};
  fp.B = (int)B; fp.k = k; fp.C = pl.C; fp.S = pl.S; fp.cand = (u64*)ws; fp.counts = (int*)(ws + pl.off_counts);
  fp.g_tau = nullptr;
  fp.drop_cols = has_mask ? mask_cols : nullptr;
  fp.mask_indptr = indptr;
  fp.ovr_hi = (u64*)(ws + pl.off_ovr_hi); fp.ovr_lo = (u32*)(ws + pl.off_ovr_lo);
  fp.id_offset = 0; fp.out_keys = nullptr; fp.out_scores = out_scores; fp.out_scores64 = out_scores64; fp.out_ids = (long long*)out_ids;
  lr = launch_finalize(fp, st);
  if (lr) return fail(CCR_ECUDA, "finalize launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

// ---- BM25 (lexical sibling of the dense path) ----
// warp = true: the warp-private kernel (S doc splits per query x kBmwWarps independent streams each);
// false: the block-wide kernel (queries with more than kBmwMaxTerms distinct terms).  streams = candidate
// lists per query handed to finalize.
struct Bm25Plan {
  int S, C, streams;
  size_t off_counts, off_tau, total;
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
  pl.off_counts = align_up((size_t)rows * (size_t)pl.streams * pl.C * sizeof(u64), 256);
  // counts, then one u32 per query: the best stream threshold (row-level bound for finalize's prefilter)
  pl.off_tau = align_up(pl.off_counts + (size_t)rows * (size_t)pl.streams * sizeof(int), 256);
  pl.total = align_up(pl.off_tau + (size_t)rows * sizeof(u32), 256);
  return pl;
}

int ccr_bm25_build_impacts(const int64_t* post_indptr, const int32_t* post_docs, const float* post_tf,
                           const double* idf, const double* doc_norm, double k1, int64_t n_terms, int64_t nnz,
                           double* post_val, void* stream) {
  if (n_terms < 0 || nnz < 0) return fail(CCR_EINVAL, "bad bm25 index shape");
  if (nnz == 0) return CCR_OK;
  if (!post_indptr || !post_docs || !post_tf || !idf || !doc_norm || !post_val) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_bm25_impacts((const long long*)post_indptr, post_docs, post_tf, idf, doc_norm, k1 + 1.0, n_terms,
                               nnz, post_val, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "bm25 impacts launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

size_t ccr_bm25_topk_workspace_bytes(int64_t Bq, int64_t n_docs, int k) {
  if (Bq < 0 || n_docs < 0 || k < 1 || k > CCR_MAX_K) return 0;
  // the caller does not say how long the queries are: room for either kernel
  const size_t tw = bm25_plan(Bq, n_docs, k, true).total, tb = bm25_plan(Bq, n_docs, k, false).total;
  return tw > tb ? tw : tb;
}

static int bm25_check(const int64_t* post_indptr, const int64_t* q_indptr, const int32_t* q_terms, int64_t Bq,
                      int64_t n_docs, int64_t max_query_terms) {
  if (Bq < 0 || n_docs < 0) return fail(CCR_EINVAL, "bad bm25 shape");
  if (Bq > 65535) return fail(CCR_EUNSUPPORTED, "bm25: more than 65535 queries per call");
  if (n_docs > (1LL << 31) - 512) return fail(CCR_EUNSUPPORTED, "n_docs must be < 2^31");
  if (max_query_terms < 0 || max_query_terms > kBmMaxTerms)
    return fail(CCR_EUNSUPPORTED, "bm25: %lld distinct terms in one query (limit %d)", (long long)max_query_terms,
                kBmMaxTerms);
  if (Bq > 0 && (!q_indptr || (max_query_terms > 0 && (!q_terms || !post_indptr))))
    return fail(CCR_EINVAL, "null pointer");
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
  if (n_terms > 0 && cudaMemsetAsync(head_slot, 0xFF, (size_t)n_terms * sizeof(int32_t), st) != cudaSuccess)  // all -1
    return fail(CCR_ECUDA, "memset bm25 head slots");
  if (n_head == 0) return CCR_OK;
  if (!post_indptr || !post_docs || !post_val || !head_terms || !head_rows) return fail(CCR_EINVAL, "null pointer");
  int lr = launch_bm25_head_slots(head_terms, n_head, n_terms, head_slot, st);
  if (lr) return fail(CCR_ECUDA, "bm25 head slots launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  lr = launch_bm25_head_rows((const long long*)post_indptr, post_docs, post_val, head_terms, n_head, n_terms,
                             ccr_bm25_head_row_pitch(n_docs), head_rows, st);
  if (lr) return fail(CCR_ECUDA, "bm25 head rows launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_bm25_topk(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                  const int32_t* head_slot, const double* head_rows,
                  const int64_t* q_indptr, const int32_t* q_terms, int64_t max_query_terms, int64_t Bq,
                  int64_t n_docs, int k, float* out_scores, int64_t* out_ids, void* workspace,
                  size_t workspace_bytes, void* stream) {
  int rc = bm25_check(post_indptr, q_indptr, q_terms, Bq, n_docs, max_query_terms);
  if (rc) return rc;
  if ((head_slot == nullptr) != (head_rows == nullptr)) return fail(CCR_EINVAL, "head_slot and head_rows go together");
  if (k < 1 || k > CCR_MAX_K) return fail(CCR_EUNSUPPORTED, "k=%d outside [1,%d]", k, CCR_MAX_K);
  if (k > n_docs) return fail(CCR_EK_RANGE, "selected index k out of range (k=%d > n=%lld)", k, (long long)n_docs);
  if (Bq == 0) return CCR_OK;
  if (!out_scores || !out_ids) return fail(CCR_EINVAL, "null pointer");
  const bool warp = max_query_terms <= kBmwMaxTerms && !knobs().bm25_blockwide;
  const Bm25Plan pl = bm25_plan(Bq, n_docs, k, warp);
  if (!workspace || workspace_bytes < pl.total) return fail(CCR_EWORKSPACE, "workspace %zu < %zu", workspace_bytes, pl.total);
  unsigned char* ws = (unsigned char*)workspace;
  cudaStream_t st = (cudaStream_t)stream;
  const long long* pi = (const long long*)post_indptr;
  const long long* qi = (const long long*)q_indptr;
  u64* cand = (u64*)ws;
  int* counts = (int*)(ws + pl.off_counts);
  // per query: max over its streams of the stream's k-th best score (every stream that pruned holds >= k
  // docs at or above its threshold, so the row's k-th best is at least the largest of them)
  u32* row_tau = (u32*)(ws + pl.off_tau);
  if (cudaMemsetAsync(row_tau, 0, (size_t)Bq * sizeof(u32), st) != cudaSuccess) return fail(CCR_ECUDA, "memset bm25 bounds");
  int lr = warp ? launch_bm25_topk_warp(pi, post_docs, post_val, head_slot, head_rows, ccr_bm25_head_row_pitch(n_docs), qi,
                                        q_terms, Bq, n_docs, k, pl.C, pl.S, cand, counts, row_tau, nullptr, 0, st)
                : launch_bm25_topk(pi, post_docs, post_val, head_slot, head_rows, ccr_bm25_head_row_pitch(n_docs), qi, q_terms,
                                   Bq, n_docs, k, pl.C, pl.S, cand, counts, nullptr, 0, st);
  if (lr) return fail(CCR_ECUDA, "bm25 top-k launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  FinalizeParams fp = {};
  fp.B = (int)Bq; fp.k = k; fp.C = pl.C; fp.S = pl.streams; fp.cand = cand; fp.counts = counts;
  fp.g_tau = warp ? row_tau : nullptr; fp.drop_cols = nullptr; fp.mask_indptr = nullptr; fp.ovr_hi = nullptr; fp.ovr_lo = nullptr;
  fp.id_offset = 0; fp.out_keys = nullptr; fp.out_scores = out_scores; fp.out_scores64 = nullptr; fp.out_ids = (long long*)out_ids;
  lr = launch_finalize(fp, st);
  if (lr) return fail(CCR_ECUDA, "finalize launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

int ccr_bm25_scores_f64(const int64_t* post_indptr, const int32_t* post_docs, const double* post_val,
                        const int32_t* head_slot, const double* head_rows,
                        const int64_t* q_indptr, const int32_t* q_terms, int64_t max_query_terms, int64_t Bq,
                        int64_t n_docs, double* scores, int64_t ld, void* stream) {
  int rc = bm25_check(post_indptr, q_indptr, q_terms, Bq, n_docs, max_query_terms);
  if (rc) return rc;
  if ((head_slot == nullptr) != (head_rows == nullptr)) return fail(CCR_EINVAL, "head_slot and head_rows go together");
  if (ld < n_docs) return fail(CCR_EINVAL, "ld < n_docs");
  if (Bq == 0 || n_docs == 0) return CCR_OK;
  if (!scores) return fail(CCR_EINVAL, "null pointer");
  const bool warp = max_query_terms <= kBmwMaxTerms && !knobs().bm25_blockwide;
  const Bm25Plan pl = bm25_plan(Bq, n_docs, 1, warp);
  int lr = warp ? launch_bm25_topk_warp((const long long*)post_indptr, post_docs, post_val, head_slot, head_rows,
                                        ccr_bm25_head_row_pitch(n_docs), (const long long*)q_indptr,
                                        q_terms, Bq, n_docs, 1, pl.C, pl.S, nullptr, nullptr, nullptr, scores, ld, (cudaStream_t)stream)
                : launch_bm25_topk((const long long*)post_indptr, post_docs, post_val, head_slot, head_rows,
                                   ccr_bm25_head_row_pitch(n_docs), (const long long*)q_indptr, q_terms,
                                   Bq, n_docs, 1, pl.C, pl.S, nullptr, nullptr, scores, ld, (cudaStream_t)stream);
  if (lr) return fail(CCR_ECUDA, "bm25 scores launch failed: %s", cudaGetErrorString((cudaError_t)lr));
  return CCR_OK;
}

}  // extern "C"
