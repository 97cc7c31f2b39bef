// Tensor-core score + select kernel for sm_100a.
//
//   scores[128 queries x 256 items] per tile = Q_tile[128 x D] . Items_tile[256 x D]^T
//
// * operands staged by TMA (cp.async.bulk.tensor.2d, 128-byte swizzle) into a 4-stage
//   shared-memory ring of (16 KB Q block + 32 KB item block), K advanced 64 elements a stage;
// * one elected thread issues tcgen05.mma.cta_group::1.kind::f16 (bf16 x bf16 -> fp32,
//   M=128, N=256, K=16) into one of two 256-column TMEM accumulators;
// * four epilogue warps read the other accumulator with tcgen05.ld (thread == query row),
//   compare against the row's running threshold and append survivors to the row's candidate
//   buffer; a nearly full buffer is pruned in place to its exact top-k (warp radix select),
//   which raises the threshold.  The B x N score matrix never leaves the SM.
//
// Persistent: grid = #SMs, each CTA walks units (query tile, item split) round-robin with the
// query tile varying fastest so CTAs running concurrently share item tiles through L2.
#include <cuda.h>
#include <stddef.h>

#include "ccr_params.cuh"

namespace ccr {

constexpr int kMaxStages = 6;
constexpr int kBytesA = kQTile * kKBlock * 2;   // 16384: 128 query rows x 64 K-elements
constexpr int kBytesB = kITile * kKBlock * 2;   // 32768: 256 item rows x 64 K-elements
// kCta = 1: one CTA owns a 128-query tile, loads the whole item block: 48 KB / stage, 4 stages.
// kCta = 2: a CTA pair (cta_group::2, UMMA M = 256) owns 256 queries; each CTA loads its 128 query
//           rows and HALF of the item block: 32 KB / stage, 6 stages -> more bytes in flight per SM
//           and half the item traffic from L2.
template <int kCta> struct TcGeom {
  static constexpr int kStages = kCta == 2 ? 6 : 4;
  static constexpr int kItemBytes = kBytesB / kCta;
  static constexpr int kStageBytes = kBytesA + kItemBytes;
  static constexpr int kItemRows = kITile / kCta;
};
constexpr int kEpiWarps = 8;                    // 2 per TMEM lane quadrant, one per column half
constexpr int kTcThreads = 384;                 // 3 warpgroups: warps 0..7 selection, warp 8 TMA, warp 9 MMA,
                                                // warps 10..11 idle (whole warpgroups so that setmaxnreg can
                                                // move registers from the feeders to the selection warps)
constexpr int kSelRegs = 216, kFeedRegs = 56;
constexpr int kTmaWarp = kEpiWarps, kMmaWarp = kEpiWarps + 1, kPollWarp = kEpiWarps + 2;
constexpr unsigned long long kThrottleGiveUpNs = 2ull * 1000ull * 1000ull;  // 2 ms
constexpr int kStageKeys = 384;                 // candidate buffers up to this size are pruned in smem
constexpr int kTmemCols = 512;
constexpr unsigned long long kWaitLimitNs = 10ull * 1000ull * 1000ull * 1000ull;  // 10 s

struct __align__(8) TcShared {
  u64 full[kMaxStages];
  u64 empty[kMaxStages];
  u64 tmem_full[2];
  u64 tmem_empty[2];
  u32 tmem_base;
  int thr_unit;      // throttle: unit the producer is streaming (-1 none yet, -2 all done); written by the producer
  u64 thr_pack;      // throttle: (unit << 32) | tiles the producer may have issued; written by the poller warp
  u32 hist[kEpiWarps][256];
  u64 stage[kEpiWarps][kStageKeys];
};
// the store epilogue (kMode 2) carves 4 KB per warp out of hist + stage, which it does not use otherwise
static_assert(offsetof(TcShared, stage) == offsetof(TcShared, hist) + sizeof(u32) * kEpiWarps * 256 &&
                  sizeof(u32) * kEpiWarps * 256 + sizeof(u64) * kEpiWarps * kStageKeys >= (size_t)kEpiWarps * 4096,
              "TcShared: hist and stage must form one block of >= 4 KB per selection warp");
constexpr size_t kTcSmemBytes = (size_t)4 * (kBytesA + kBytesB) + sizeof(TcShared) + 1024;  // same for both geometries

// ---------------------------------------------------------------------------------------
// PTX wrappers
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_u32(const void* p) { return (u32)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(u64* bar, u32 count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(u64* bar, u32 bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(u64* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// relaxed arrive: the TMEM reads it publishes are already complete (tcgen05.wait::ld); a release
// arrive would additionally wait for this thread's outstanding candidate stores to global memory
__device__ __forceinline__ void mbar_arrive_relaxed(u64* bar) {
  asm volatile("mbarrier.arrive.relaxed.cta.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(u64* bar, u32 parity) {
  u32 ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
  return ok != 0;
}
// bounded wait: a pipeline bug must end in a trap + error record, never in a hung GPU
__device__ __forceinline__ void mbar_wait(u64* bar, u32 parity, DeviceStatus* st, int where) {
  u32 spins = 0;
  unsigned long long t0 = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 1023u) == 0) {
      unsigned long long now;
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
      if (t0 == 0) t0 = now;
      else if (now - t0 > kWaitLimitNs) {
        if (st) { st->code = 1; st->where = where; st->block = blockIdx.x; st->extra = (int)parity; }
        __threadfence_system();
        __trap();
      }
    }
  }
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* map, int c0, int c1, u64* bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// ---- cta_group::2 (CTA pair) variants ----
__device__ __forceinline__ u32 cluster_ctarank() { u32 r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// shared::cluster address of `p`'s offset inside CTA `rank` of this cluster
__device__ __forceinline__ u32 mapa_u32(const void* p, u32 rank) {
  u32 r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(smem_u32(p)), "r"(rank));
  return r;
}
// TMA load into OWN shared memory whose bytes are accounted on the LEADER CTA's mbarrier
__device__ __forceinline__ void tma_load_2d_2cta(void* dst, const CUtensorMap* map, int c0, int c1, u32 leader_bar) {
  asm volatile(
      "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(leader_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_commit_2cta(u64* bar) {  // arrives on `bar`'s offset in BOTH CTAs
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((unsigned short)3) : "memory");
}
__device__ __forceinline__ void tc_mma_bf16_2cta(u32 tmem_d, u64 adesc, u64 bdesc, u32 idesc, u32 accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void mbar_arrive_remote(u32 cluster_bar_addr) {
  asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(cluster_bar_addr) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(u64* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void tc_mma_bf16(u32 tmem_d, u64 adesc, u64 bdesc, u32 idesc, u32 accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32b_x32(u32 taddr, u32 (&v)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7]),
        "=r"(v[8]), "=r"(v[9]), "=r"(v[10]), "=r"(v[11]), "=r"(v[12]), "=r"(v[13]), "=r"(v[14]), "=r"(v[15]),
        "=r"(v[16]), "=r"(v[17]), "=r"(v[18]), "=r"(v[19]), "=r"(v[20]), "=r"(v[21]), "=r"(v[22]), "=r"(v[23]),
        "=r"(v[24]), "=r"(v[25]), "=r"(v[26]), "=r"(v[27]), "=r"(v[28]), "=r"(v[29]), "=r"(v[30]), "=r"(v[31])
      : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128-byte-swizzled operand tile (rows x 64 bf16, row pitch 128 B, 8-row atoms 1024 B
// apart).  Field layout per the sm_100 shared-memory matrix descriptor: start address [0,14)
// (>>4), LBO [16,30) (ignored for swizzled K-major; 1 like CUTLASS), SBO [32,46) = 1024>>4,
// version [46,48) = 1, layout [61,64) = 2 (SWIZZLE_128B).
__device__ __forceinline__ u64 make_sw128_desc(u32 saddr) {
  u64 d = 0;
  d |= (u64)((saddr & 0x3FFFFu) >> 4);
  d |= (u64)1 << 16;
  d |= (u64)(1024 >> 4) << 32;
  d |= (u64)1 << 46;
  d |= (u64)2 << 61;
  return d;
}
// instruction descriptor, kind::f16: c_format f32 (bit 4), a/b format bf16 (bits 7, 10),
// both K-major (bits 15,16 = 0), N>>3 at [17,23), M>>4 at [24,29)
template <int kCta> struct TcIdesc {
  static constexpr u32 value = (1u << 4) | (1u << 7) | (1u << 10) | ((u32)(kITile >> 3) << 17) | ((u32)((kQTile * kCta) >> 4) << 24);
};

// ---------------------------------------------------------------------------------------
// per-thread selection state, the per-chunk filter (32 columns of one query row) and the
// deferred prune
// ---------------------------------------------------------------------------------------
struct SelState {
  u64* buf;        // this (row, split, half)'s candidate buffer
  int cnt;         // keys currently in buf
  float tau_f;     // pass iff score >= tau_f: max(next_up(local k-th best), shared row bound),
                   // -inf before the first prune, +inf for padding rows
  long long mbeg, mend;  // the row's slice of the mask CSR
  u64 sig;         // signature of the row's masked columns: bit (col & 63) ...
  u64 sig2;        // ... and bit ((col >> 6) & 63): both must be set before the exact search runs
  int row;         // global query row
  int k_row;       // candidates this row must keep: k (+ the row's mask entries in include mode)
  int stream;      // index of this stream among the row's streams
  u32* hist;       // the row's score histogram (null: off for this row)
  u32 hbase, hshift;  // bucket b covers ord32 scores [hbase + (b << hshift), hbase + ((b + 1) << hshift))
};

__device__ __forceinline__ float max8(const u32 (&v)[32], int g) {
  const float a = fmaxf(fmaxf(__uint_as_float(v[g * 8 + 0]), __uint_as_float(v[g * 8 + 1])), __uint_as_float(v[g * 8 + 2]));
  const float b = fmaxf(fmaxf(__uint_as_float(v[g * 8 + 3]), __uint_as_float(v[g * 8 + 4])), __uint_as_float(v[g * 8 + 5]));
  const float c = fmaxf(__uint_as_float(v[g * 8 + 6]), __uint_as_float(v[g * 8 + 7]));
  return fmaxf(fmaxf(a, b), c);
}

// exact membership test for a column whose signature bit is set (rare)
static __device__ __noinline__ bool masked_slow(const int* mask_cols, long long mbeg, long long mend, int col) {
  return mask_contains(mask_cols, mbeg, mend, col);
}

// Branch-free conditional append: if (s >= tau) { buf[cnt] = make_key(s, ~nlo); ++cnt; }
// written as predicated PTX so that a group of 8 columns costs a fixed, short, straight-line
// sequence whatever the number of hits.
template <int J>
__device__ __forceinline__ void append_if_ge(u32 sbits, float tau, u32 nlo0, u64* buf, int& cnt) {
  if (__uint_as_float(sbits) >= tau) {
    const u32 hi = sbits ^ ((u32)((int)sbits >> 31) | 0x80000000u);
    buf[cnt] = ((u64)hi << 32) | (u64)(nlo0 - (u32)J);
    cnt += 1;
  }
}

// One more distinct item of this row scores `s` (>= the row's seed bound): count it in the row's
// histogram (fire-and-forget RED to L2).
__device__ __forceinline__ void hist_count(const SelState& st, float s) {
  const u32 o = ord32(s);
  if (o >= st.hbase) {
    u32 b = (o - st.hbase) >> st.hshift;
    b = b < (u32)(kHistBins - 1) ? b : (u32)(kHistBins - 1);
    asm volatile("red.relaxed.gpu.global.add.u32 [%0], 1;" ::"l"(st.hist + b) : "memory");
  }
}

// Lower bound of the row's k-th best from its histogram: the lower edge of the highest bucket with
// at least `need` items counted at or above it (0: not yet).  Counters only grow, so a stale
// read gives a weaker but still valid bound.  Per-thread code (lane == row): 4 batches of 8
// independent 16-byte loads from the top bucket down.
static __device__ __noinline__ u32 hist_bound(const u32* hist, int need, u32 hbase, u32 hshift) {
  u32 acc = 0u;
  const uint4* h4 = reinterpret_cast<const uint4*>(hist);
#pragma unroll 1
  for (int q4 = kHistBins / 4 - 8; q4 >= 0; q4 -= 8) {
    uint4 c[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) c[i] = __ldcg(h4 + q4 + i);
#pragma unroll
    for (int i = 7; i >= 0; --i) {
      const int b = (q4 + i) * 4;
      acc += c[i].w; if (acc >= (u32)need) return hbase + ((u32)(b + 3) << hshift);
      acc += c[i].z; if (acc >= (u32)need) return hbase + ((u32)(b + 2) << hshift);
      acc += c[i].y; if (acc >= (u32)need) return hbase + ((u32)(b + 1) << hshift);
      acc += c[i].x; if (acc >= (u32)need) return hbase + ((u32)b << hshift);
    }
  }
  return 0u;
}

// Append every score >= tau_f of this 32-column chunk to the row's buffer.  Warp-uniform votes
// decide whether a group of 8 columns is looked at; inside a group the appends are predicated
// (no branches, no calls, no key compares): the strict local threshold already encodes the
// lowest-id tie rule because a stream sees its items in ascending id order.
template <bool kMask>
__device__ __forceinline__ void filter_chunk(const u32 (&v)[32], u32 col0, SelState& st, const SelectParams& p) {
  float m8[4];
#pragma unroll
  for (int g = 0; g < 4; ++g) m8[g] = max8(v, g);
  const float m = fmaxf(fmaxf(m8[0], m8[1]), fmaxf(m8[2], m8[3]));
  if (!__any_sync(0xffffffffu, m >= st.tau_f)) return;
  const u32 nlo0 = 0xFFFFFFFFu - col0;  // low key word of column col0; column col0+j -> nlo0 - j
#define CCR_APPEND(J)                                                                            \
  if (kMask) {                                                                                   \
    u32 sb = v[J];                                                                               \
    const u32 col = col0 + (u32)(J);                                                             \
    if (__uint_as_float(sb) >= st.tau_f && ((st.sig >> (col & 63u)) & (st.sig2 >> ((col >> 6) & 63u)) & 1ull)) { \
      if (masked_slow(p.mask_cols, st.mbeg, st.mend, (int)col)) sb = 0x7fc00000u;                \
    }                                                                                            \
    append_if_ge<J>(sb, st.tau_f, nlo0, st.buf, st.cnt);                                         \
  } else {                                                                                       \
    append_if_ge<J>(v[J], st.tau_f, nlo0, st.buf, st.cnt);                                       \
  }
#define CCR_GROUP(G)                                                                             \
  if (__any_sync(0xffffffffu, m8[G] >= st.tau_f)) {                                              \
    if (!kMask && st.hist && m8[G] >= st.tau_f) hist_count(st, m8[G]);                           \
    CCR_APPEND(G * 8 + 0) CCR_APPEND(G * 8 + 1) CCR_APPEND(G * 8 + 2) CCR_APPEND(G * 8 + 3)      \
    CCR_APPEND(G * 8 + 4) CCR_APPEND(G * 8 + 5) CCR_APPEND(G * 8 + 6) CCR_APPEND(G * 8 + 7)      \
  }
  CCR_GROUP(0) CCR_GROUP(1) CCR_GROUP(2) CCR_GROUP(3)
#undef CCR_GROUP
#undef CCR_APPEND
  asm volatile("" ::: "memory");  // appended keys are read back by the prune
}

// columns at or beyond n_items (zero-filled by TMA) must never be selected
__device__ __forceinline__ void clamp_ragged(u32 (&v)[32], long long col0, long long n_items) {
#pragma unroll
  for (int j = 0; j < 32; ++j)
    if (col0 + j >= n_items) v[j] = 0x7fc00000u;  // NaN: ignored by fmaxf, fails every >= test
}

// Everything below the per-chunk filter is deliberately kept OUT of line (one copy each): the
// epilogue's common path must stay resident in the instruction caches.
struct ShareArgs {
  u32* g_tau;
  u32* g_q;
  int S_row, share_j, share_m;
};

// m-th largest of the row's published stream values (0 = unpublished) -- the shared lower bound.
static __device__ __noinline__ u32 sketch_bound(const u32* gq, int S_row, int m, int own_stream, u32 own_val,
                                                u32 hist_s, u32 stage_s) {
  const int lane = threadIdx.x & 31;
  if (S_row <= 32) {
    u32 v = 0u;
    if (lane < S_row) v = (lane == own_stream) ? own_val : __ldcg(gq + lane);
    int gt = 0, ge = 0;
#pragma unroll 4
    for (int i = 0; i < 32; ++i) {
      const u32 o = __shfl_sync(0xffffffffu, v, i);
      gt += (o > v);
      ge += (o >= v);
    }
    const unsigned who = __ballot_sync(0xffffffffu, gt < m && m <= ge);
    return who ? __shfl_sync(0xffffffffu, v, __ffs(who) - 1) : 0u;
  }
  const int ns = S_row < kStageKeys ? S_row : kStageKeys;
  for (int i = lane; i < ns; i += 32) {
    const u32 qv = (i == own_stream) ? own_val : __ldcg(gq + i);
    sm_st64(stage_s + (u32)i * 8u, ((u64)qv << 32) | (u64)(u32)(ns - i));
  }
  __syncwarp();
  return (u32)(warp_select_kth(SharedKeys{stage_s}, ns, m, hist_s) >> 32);
}

static __device__ __noinline__ u64 exact_prune(u64* b, int n, int k, int j, bool staged, u32 hist_s, u32 stage_s,
                                               u32* j_ord) {
  const u64 pivot = warp_prune(b, n, k, hist_s, staged ? stage_s : 0u);
  if (j > 0) {
    u64 kj;
    if (staged) kj = warp_select_kth(SharedKeys{stage_s}, n, j, hist_s);
    else kj = warp_select_kth(GlobalKeys{b}, k, j, hist_s);
    *j_ord = (u32)(kj >> 32);
  }
  return pivot;
}

// Prune one stream's buffer (all 32 lanes cooperate), publish its share_j-th best, refresh the
// row's shared bound.  Returns (kept << 32) | float bits of the stream's new threshold.
static __device__ __noinline__ u64 prune_stream(u64* b, int n, int k, int C, int row_s, int stream_s, ShareArgs sh,
                                                u32 hist_s, u32 stage_s) {
  const int lane = threadIdx.x & 31;
  const bool staged = C <= kStageKeys;
  const int jj = sh.share_j > 0 ? sh.share_j : k;
  float new_tau;
  int kept = k;
  u32 j_ord = 0u, pivot_ord = 0u;
  // fast path: one histogram pass; leaves between k and (k + C-128)/2 survivors
  const bool fast =
      staged ? warp_prune_hist<true>(b, n, k, jj, (k + C - 128) / 2, hist_s, stage_s, &pivot_ord, &kept, &j_ord)
             : warp_prune_hist<false>(b, n, k, jj, (k + C - 128) / 2, hist_s, stage_s, &pivot_ord, &kept, &j_ord);
  if (fast) {
    new_tau = unord32(pivot_ord);  // ">=": every key at or above the pivot bucket was kept
  } else {
    const u64 pivot = exact_prune(b, n, k, sh.share_j, staged, hist_s, stage_s, &j_ord);
    new_tau = next_up(key_score(pivot));
    kept = k;
  }
  if (sh.share_j > 0) {
    u32* gq = sh.g_q + (long long)row_s * sh.S_row;
    if (lane == 0) gq[stream_s] = j_ord;
    const u32 bound = sketch_bound(gq, sh.S_row, sh.share_m, stream_s, j_ord, hist_s, stage_s);
    if (bound != 0u) {
      if (lane == 0) atomicMax(sh.g_tau + row_s, bound);  // no return value needed: RED
      if (bound > ord32(new_tau)) new_tau = unord32(bound);
    }
  }
  return ((u64)(u32)kept << 32) | (u64)__float_as_uint(new_tau);
}

// Prune every stream of this warp whose buffer could overflow during the next half tile.  Runs
// after the accumulator has been handed back, i.e. off the MMA critical path.
__device__ __forceinline__ void prune_pending(SelState& st, const ShareArgs& sh, int C, u32 hist_s, u32 stage_s) {
  const int lane = threadIdx.x & 31;
  unsigned need = __ballot_sync(0xffffffffu, st.cnt > C - 128);
  while (need) {
    const int src = __ffs(need) - 1;
    need &= need - 1;
    u64* b = reinterpret_cast<u64*>(__shfl_sync(0xffffffffu, (u64)(uintptr_t)st.buf, src));
    const int n = __shfl_sync(0xffffffffu, st.cnt, src);
    const int row_s = __shfl_sync(0xffffffffu, st.row, src);
    const int stream_s = __shfl_sync(0xffffffffu, st.stream, src);
    const int k_s = __shfl_sync(0xffffffffu, st.k_row, src);
    const u64 r = prune_stream(b, n, k_s, C, row_s, stream_s, sh, hist_s, stage_s);
    if (lane == src) { st.cnt = (int)(r >> 32); st.tau_f = __uint_as_float((u32)r); }
  }
}

// ---------------------------------------------------------------------------------------
// the kernel
// ---------------------------------------------------------------------------------------
// kMode: 0 select (no mask), 1 select (mask CSR), 2 store fp32 scores (seeding pre-pass)
template <int kMode, int kCta>
__global__ void __launch_bounds__(kTcThreads, 1)
select_tc_kernel(const __grid_constant__ CUtensorMap tmap_q, const __grid_constant__ CUtensorMap tmap_items,
                 SelectParams p) {
  using G = TcGeom<kCta>;
  constexpr int kStages = G::kStages;
  constexpr int kStageBytes = G::kStageBytes;
  constexpr int kQRows = kQTile * kCta;   // query rows per unit
  extern __shared__ unsigned char smem_dyn[];
  // 1024-byte alignment for the swizzled tiles (identical offsets in both CTAs of a pair)
  unsigned char* smem = reinterpret_cast<unsigned char*>(((uintptr_t)smem_dyn + 1023) & ~(uintptr_t)1023);
  TcShared* sh = reinterpret_cast<TcShared*>(smem + (size_t)kStages * kStageBytes);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int num_kb = (p.D + kKBlock - 1) / kKBlock;
  const long long tiles_total = (p.n_items + kITile - 1) / kITile;
  const int n_units = p.n_q_tiles * p.S;
  const int crank = kCta == 2 ? (int)cluster_ctarank() : 0;   // 0 = leader (issues the MMAs)
  const int cid = (int)blockIdx.x / kCta, n_cl = (int)gridDim.x / kCta;  // persistent workers = clusters

  if (threadIdx.x == 0) {
    sh->thr_unit = -1;
    sh->thr_pack = ~0ull;  // unit tag that matches no unit
    for (int s = 0; s < kStages; ++s) { mbar_init(&sh->full[s], 1); mbar_init(&sh->empty[s], 1); }
    for (int s = 0; s < 2; ++s) { mbar_init(&sh->tmem_full[s], 1); mbar_init(&sh->tmem_empty[s], kEpiWarps * kCta); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_q) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&tmap_items) : "memory");
  }
  if (warp == kMmaWarp) {
    if (kCta == 2) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "r"((u32)kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&sh->tmem_base)),
                   "r"((u32)kTmemCols) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (kCta == 2) cluster_sync_all();  // the peer's barriers exist before anything is signalled on them
  tc_fence_after();
  const u32 tmem_base = sh->tmem_base;

  if (warp >= kEpiWarps) {
   // ---- feeder warpgroup: give registers away, then TMA producer / MMA issuer / idle ----
   asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(kFeedRegs));
   if (warp == kTmaWarp) {
    // ================= TMA producer =================
    if (lane == 0) {
      int stage = 0; u32 phase = 0;
      for (int unit = cid; unit < n_units; unit += n_cl) {
        const int qt = unit % p.n_q_tiles, u = unit / p.n_q_tiles;
        const long long t0 = (long long)u * tiles_total / p.S, t1 = (long long)(u + 1) * tiles_total / p.S;
        // peers: units of the same item split scheduled in the same persistent iteration
        int peer_lo = u * p.n_q_tiles, peer_hi = peer_lo + p.n_q_tiles;
        {
          const int it_lo = (unit / n_cl) * n_cl, it_hi = it_lo + n_cl;
          peer_lo = peer_lo > it_lo ? peer_lo : it_lo;
          peer_hi = peer_hi < it_hi ? peer_hi : it_hi;
        }
        // Units that stream the same split only share its tiles through L2 while they stay close
        // together.  A leader that is not slowed down by its own L2 misses (the 6-stage pair
        // pipeline hides them) runs away and every follower then misses too: DRAM reads of 7x the
        // table were measured for CTA pairs at B=4096.  So a producer never leads the slowest peer by
        // more than lead_tiles.  The lead is chosen by the host so that (splits in flight) x (lead) item
        // tiles stay well inside L2; the peers' counters are watched by the poller warp below.  Peers
        // run concurrently because the grid has at most one CTA per SM;
        // should one not be running (shared GPU), the wait gives up after 2 ms and throttling is
        // dropped for the rest of the unit.
        bool throttle = p.progress != nullptr && (peer_hi - peer_lo) > 1;
        if (p.progress != nullptr) {  // tell the poller warp which unit is being streamed
          asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"(smem_u32(&sh->thr_unit)),
                       "r"((throttle && p.throttle_poller) ? unit : -1) : "memory");
        }
        const int n_peers_inline = peer_hi - peer_lo;
        for (long long t = t0; t < t1; ++t) {
          if (throttle && !p.throttle_poller) {
            // inline variant: every lead_every tiles publish my position and read the peers' myself
            if (((t - t0) & (long long)(p.lead_every - 1)) == 0) {
              const int mine = (int)(t - t0);
              asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p.progress + unit), "r"(mine) : "memory");
              unsigned long long w0 = 0;
              for (;;) {
                int mn = 0x7fffffff;
                for (int v = 0; v < n_peers_inline; ++v) {
                  int pv;
                  asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(pv) : "l"(p.progress + peer_lo + v) : "memory");
                  mn = pv < mn ? pv : mn;
                }
                if (mine - mn <= p.lead_tiles) break;
                __nanosleep(500);
                unsigned long long now;
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
                if (w0 == 0) w0 = now;
                else if (now - w0 > kThrottleGiveUpNs) { throttle = false; break; }  // never depend on a peer
              }
            }
          } else if (throttle) {
            // publish my position (fire and forget), then make sure I am not more than lead_tiles ahead
            // of the slowest peer: the poller warp keeps (unit, slowest + lead) in shared memory, so this
            // thread never waits for a global load
            const int mine = (int)(t - t0);
            asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p.progress + unit), "r"(mine) : "memory");
            unsigned long long w0 = 0;
            for (;;) {
              u64 a;
              asm volatile("ld.volatile.shared.u64 %0, [%1];" : "=l"(a) : "r"(smem_u32(&sh->thr_pack)) : "memory");
              const int allowed = ((int)(a >> 32) == unit) ? (int)(u32)a : p.lead_tiles;  // no report yet: head start
              if (mine <= allowed) break;
              __nanosleep(100);
              unsigned long long now;
              asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(now));
              if (w0 == 0) w0 = now;
              else if (now - w0 > kThrottleGiveUpNs) { throttle = false; break; }  // never depend on a peer
            }
          }
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(&sh->empty[stage], phase ^ 1u, p.status, 100 + stage);
            unsigned char* sa = smem + (size_t)stage * kStageBytes;
            if (kCta == 2) {
              // both CTAs' bytes are accounted on the leader's barrier; only the leader arms it
              if (crank == 0) mbar_expect_tx(&sh->full[stage], 2 * kStageBytes);
              const u32 lbar = mapa_u32(&sh->full[stage], 0);
              tma_load_2d_2cta(sa, &tmap_q, kb * kKBlock, qt * kQRows + crank * kQTile, lbar);
              tma_load_2d_2cta(sa + kBytesA, &tmap_items, kb * kKBlock, (int)(t * kITile) + crank * G::kItemRows, lbar);
            } else {
              mbar_expect_tx(&sh->full[stage], kStageBytes);
              tma_load_2d(sa, &tmap_q, kb * kKBlock, qt * kQTile, &sh->full[stage]);
              tma_load_2d(sa + kBytesA, &tmap_items, kb * kKBlock, (int)(t * kITile), &sh->full[stage]);
            }
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
        }
        if (p.progress != nullptr && (peer_hi - peer_lo) > 1)  // finished: never hold a peer back
          asm volatile("st.relaxed.gpu.global.s32 [%0], %1;" ::"l"(p.progress + unit), "r"(0x3fffffff) : "memory");
      }
      if (p.progress != nullptr)
        asm volatile("st.volatile.shared.s32 [%0], %1;" ::"r"(smem_u32(&sh->thr_unit)), "r"(-2) : "memory");
    }
  } else if (warp == kPollWarp) {
    // ================= throttle poller =================
    // Units that stream the same item split only share its tiles through L2 while they stay close.  This
    // warp watches the progress counters of the producer's peers (one lane per peer, in parallel) and
    // keeps "slowest peer + lead" in shared memory for the producer, which therefore throttles at tile
    // granularity without ever waiting for a global load itself.
    if (p.progress != nullptr) {
      for (;;) {
        int unit;
        asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(unit) : "r"(smem_u32(&sh->thr_unit)) : "memory");
        if (unit == -2) break;
        if (unit >= 0) {
          const int u = unit / p.n_q_tiles;
          int peer_lo = u * p.n_q_tiles, peer_hi = peer_lo + p.n_q_tiles;
          const int it_lo = (unit / n_cl) * n_cl, it_hi = it_lo + n_cl;
          peer_lo = peer_lo > it_lo ? peer_lo : it_lo;
          peer_hi = peer_hi < it_hi ? peer_hi : it_hi;
          int mn = 0x7fffffff;
          for (int v = peer_lo + lane; v < peer_hi; v += 32) {
            int pv;
            asm volatile("ld.relaxed.gpu.global.s32 %0, [%1];" : "=r"(pv) : "l"(p.progress + v) : "memory");
            mn = pv < mn ? pv : mn;
          }
#pragma unroll
          for (int off = 16; off; off >>= 1) { const int o = __shfl_xor_sync(0xffffffffu, mn, off); mn = o < mn ? o : mn; }
          if (lane == 0) {
            const long long allowed = (long long)mn + p.lead_tiles;
            const u64 pack = ((u64)(u32)unit << 32) | (u64)(u32)(allowed > 0x3fffffff ? 0x3fffffff : (int)allowed);
            asm volatile("st.volatile.shared.u64 [%0], %1;" ::"r"(smem_u32(&sh->thr_pack)), "l"(pack) : "memory");
          }
        }
        __nanosleep(400);
      }
    }
  } else if (warp == kMmaWarp) {
    // ================= MMA issuer (leader CTA only in a pair) =================
    if (lane == 0 && crank == 0) {
      int stage = 0; u32 phase = 0;
      int acc = 0; u32 acc_phase = 0;
      for (int unit = cid; unit < n_units; unit += n_cl) {
        const int u = unit / p.n_q_tiles;
        const long long t0 = (long long)u * tiles_total / p.S, t1 = (long long)(u + 1) * tiles_total / p.S;
        for (long long t = t0; t < t1; ++t) {
          mbar_wait(&sh->tmem_empty[acc], acc_phase ^ 1u, p.status, 200 + acc);
          tc_fence_after();
          const u32 d_tmem = tmem_base + (u32)(acc * kITile);
          for (int kb = 0; kb < num_kb; ++kb) {
            mbar_wait(&sh->full[stage], phase, p.status, 300 + stage);
            tc_fence_after();
            const u32 sa = smem_u32(smem + (size_t)stage * kStageBytes);
            const u64 adesc = make_sw128_desc(sa);
            const u64 bdesc = make_sw128_desc(sa + kBytesA);
#pragma unroll
            for (int kk = 0; kk < kKBlock / 16; ++kk) {
              // +32 bytes (16 bf16) along K inside the 128-byte swizzle row: +2 in 16-byte units
              if (kCta == 2)
                tc_mma_bf16_2cta(d_tmem, adesc + (u64)(kk * 2), bdesc + (u64)(kk * 2), TcIdesc<2>::value, (kb | kk) ? 1u : 0u);
              else
                tc_mma_bf16(d_tmem, adesc + (u64)(kk * 2), bdesc + (u64)(kk * 2), TcIdesc<1>::value, (kb | kk) ? 1u : 0u);
            }
            // frees the smem slot (in both CTAs of a pair) once these MMAs retire
            if (kCta == 2) tc_commit_2cta(&sh->empty[stage]); else tc_commit(&sh->empty[stage]);
            if (++stage == kStages) { stage = 0; phase ^= 1u; }
          }
          // accumulator complete (both CTAs' selection warps wake up)
          if (kCta == 2) tc_commit_2cta(&sh->tmem_full[acc]); else tc_commit(&sh->tmem_full[acc]);
          if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
        }
      }
    }
   }
  } else {
   // ---- selection warpgroups: take the registers the feeders released ----
   asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(kSelRegs));
   if (kMode >= 2) {
    // ===== store epilogue: thread == query row; writes its 128 columns of the tile as fp32 (kMode 2)
    //       or the best score of every 8 columns (kMode 3, threshold seeding) =====
    const int quad = warp & 3, half = warp >> 2;
    const int row_in_tile = quad * 32 + lane;
    int acc = 0; u32 acc_phase = 0;
    const bool vec_ok = (p.ld_out & 3) == 0 && ((uintptr_t)p.dense_out & 15) == 0;
    for (int unit = cid; unit < n_units; unit += n_cl) {
      const int qt = unit % p.n_q_tiles, u = unit / p.n_q_tiles;
      const long long t0 = (long long)u * tiles_total / p.S, t1 = (long long)(u + 1) * tiles_total / p.S;
      const int row = qt * kQRows + crank * kQTile + row_in_tile;
      const bool valid_row = row < p.B;
      float* orow = p.dense_out + (long long)row * p.ld_out;
      for (long long t = t0; t < t1; ++t) {
        mbar_wait(&sh->tmem_full[acc], acc_phase, p.status, 400 + acc);
        tc_fence_after();
        const u32 taddr0 = tmem_base + ((u32)(quad * 32) << 16) + (u32)(acc * kITile + half * 128);
        const long long col0 = t * kITile + half * 128;
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
          u32 v[32];
          tmem_ld_32x32b_x32(taddr0 + (u32)(32 * c), v);
          tmem_ld_wait();
          const long long cc = col0 + 32 * c;
          if (kMode == 3) {
            // sampled items beyond n_items are zero rows (TMA fill): a 0 score may only raise a group
            // maximum that is negative, so such groups are written as -inf instead
            if (valid_row) {
              float m8[4];
#pragma unroll
              for (int g = 0; g < 4; ++g) m8[g] = (cc + 8 * g + 8 <= p.n_items) ? max8(v, g) : -INFINITY;
              *reinterpret_cast<float4*>(orow + (cc >> 3)) = make_float4(m8[0], m8[1], m8[2], m8[3]);
            }
          } else if (vec_ok && cc + 32 <= p.n_items) {   // warp-uniform
            // The lane holds 32 columns of ITS row: stored as they are, one instruction would touch 32 rows
            // (0.5 TB/s measured).  Transpose the 32 x 32 block through this warp's 4 KB of shared memory
            // (16-byte chunks XOR-swizzled by the row: conflict-free both ways) so that one instruction
            // writes 4 rows x 128 contiguous bytes.
            float* ts = reinterpret_cast<float*>(reinterpret_cast<unsigned char*>(sh->hist) + warp * 4096);
#pragma unroll
            for (int q = 0; q < 8; ++q)
              *reinterpret_cast<float4*>(ts + lane * 32 + ((q ^ (lane & 7)) << 2)) =
                  make_float4(__uint_as_float(v[4 * q]), __uint_as_float(v[4 * q + 1]), __uint_as_float(v[4 * q + 2]),
                              __uint_as_float(v[4 * q + 3]));
            __syncwarp();
            const int q = lane & 7;
#pragma unroll
            for (int i = 0; i < 8; ++i) {
              const int rr = 4 * i + (lane >> 3);
              const float4 x = *reinterpret_cast<const float4*>(ts + rr * 32 + ((q ^ (rr & 7)) << 2));
              const int grow = qt * kQRows + crank * kQTile + quad * 32 + rr;
              if (grow < p.B) *reinterpret_cast<float4*>(p.dense_out + (long long)grow * p.ld_out + cc + q * 4) = x;
            }
            __syncwarp();
          } else if (valid_row) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (cc + j < p.n_items) orow[cc + j] = __uint_as_float(v[j]);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCta == 2) mbar_arrive_remote(mapa_u32(&sh->tmem_empty[acc], 0));
          else mbar_arrive_relaxed(&sh->tmem_empty[acc]);
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
    }
  } else {
    constexpr bool kMask = (kMode == 1);
    // ===== epilogue / selection: 8 warps; thread == (query row, 128-column half of the tile) =====
    const int ew = warp;
    const int quad = warp & 3;   // TMEM lane quadrant this warp may access
    const int half = ew >> 2;    // 0: tile columns [0,128), 1: [128,256)
    const int row_in_tile = quad * 32 + lane;
    const u32 hist_s = smem_addr(sh->hist[ew]);
    const u32 stage_s = smem_addr(sh->stage[ew]);
    const int k = p.k, C = p.C;
    ShareArgs sa;
    sa.g_tau = p.g_tau; sa.g_q = p.g_q; sa.S_row = p.S_row; sa.share_j = p.share_j; sa.share_m = p.share_m;
    int acc = 0; u32 acc_phase = 0;
    for (int unit = cid; unit < n_units; unit += n_cl) {
      const int qt = unit % p.n_q_tiles, u = unit / p.n_q_tiles;
      const long long t0 = (long long)u * tiles_total / p.S, t1 = (long long)(u + 1) * tiles_total / p.S;
      const int row = qt * kQRows + crank * kQTile + row_in_tile;
      const bool valid_row = row < p.B;
      SelState st;
      st.buf = p.cand + (((long long)row * p.S + u) * 2 + half) * C;
      st.cnt = 0;
      st.tau_f = valid_row ? -INFINITY : INFINITY;
      st.mbeg = 0; st.mend = 0; st.sig = 0ull; st.sig2 = 0ull;
      st.row = row; st.stream = u * 2 + half;
      st.hist = nullptr; st.hbase = 0u; st.hshift = 0u;
      if (!kMask && p.g_hist && valid_row) {
        const uint2 hp = __ldg(p.g_hpar + row);
        if (hp.y) { st.hist = p.g_hist + (long long)row * kHistBins; st.hbase = hp.x; st.hshift = hp.y - 1u; }
      }
      st.k_row = k;
      if (!kMask && p.mask_indptr && valid_row) {
        const long long kr = (long long)k + (p.mask_indptr[row + 1] - p.mask_indptr[row]);
        st.k_row = kr < (long long)p.k_keep ? (int)kr : p.k_keep;  // buffers are sized for k_keep
      }
      if (kMask && valid_row) {
        st.mbeg = p.mask_indptr[row]; st.mend = p.mask_indptr[row + 1];
        for (long long e = st.mbeg; e < st.mend; ++e) {
          const u32 mc = (u32)__ldg(p.mask_cols + e);
          st.sig |= 1ull << (mc & 63u);
          st.sig2 |= 1ull << ((mc >> 6) & 63u);
        }
      }

      for (long long t = t0; t < t1; ++t) {
        u32 gt = 0u;
        if (p.g_tau && valid_row) gt = __ldcg(p.g_tau + row);  // issued before the wait
        mbar_wait(&sh->tmem_full[acc], acc_phase, p.status, 400 + acc);
        tc_fence_after();
        if (gt > ord32(st.tau_f)) st.tau_f = unord32(gt);
        const u32 taddr0 = tmem_base + ((u32)(quad * 32) << 16) + (u32)(acc * kITile + half * 128);
        const long long col0 = t * kITile + half * 128;
        const bool ragged = col0 + 128 > p.n_items;
        // all 128 columns of this half go to registers first, the accumulator is handed back to the
        // MMA warp (of the leader CTA when two CTAs share the MMA) immediately, and only then is
        // anything filtered: the MMA never waits for selection work, only for these four loads
        u32 v[32], w1[32], w2[32], w3[32];
        tmem_ld_32x32b_x32(taddr0, v);
        tmem_ld_32x32b_x32(taddr0 + 32u, w1);
        tmem_ld_32x32b_x32(taddr0 + 64u, w2);
        tmem_ld_32x32b_x32(taddr0 + 96u, w3);
        tmem_ld_wait();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) {
          if (kCta == 2) mbar_arrive_remote(mapa_u32(&sh->tmem_empty[acc], 0));
          else mbar_arrive_relaxed(&sh->tmem_empty[acc]);
        }
        // two filter call sites (instruction-cache footprint vs register moves): chunks 0,1 are
        // filtered from v,w1; then chunks 2,3 move into those registers and take the same code
#pragma unroll 1
        for (int c = 0; c < 4; c += 2) {
          if (ragged) { clamp_ragged(v, col0 + 32 * c, p.n_items); clamp_ragged(w1, col0 + 32 * c + 32, p.n_items); }
          filter_chunk<kMask>(v, (u32)col0 + (u32)(32 * c), st, p);
          filter_chunk<kMask>(w1, (u32)col0 + (u32)(32 * c + 32), st, p);
          if (c == 0) {
#pragma unroll
            for (int j = 0; j < 32; ++j) { v[j] = w2[j]; w1[j] = w3[j]; }
          }
        }
        prune_pending(st, sa, C, hist_s, stage_s);
        if (!kMask && p.g_hist) {
          // refresh the row bound from the histogram at tiles 4, 8, 16, ... 256 and every 256 after
          const long long ti = t - t0 + 1;
          if (ti >= 4 && ((ti & (ti - 1)) == 0 || (ti & 255) == 0) && st.hist) {
            const u32 hb = hist_bound(st.hist, st.k_row, st.hbase, st.hshift);
            if (hb > ord32(st.tau_f)) {
              st.tau_f = unord32(hb);
              atomicMax(p.g_tau + row, hb);
            }
          }
        }
        if (++acc == 2) { acc = 0; acc_phase ^= 1u; }
      }
      p.counts[((long long)row * p.S + u) * 2 + half] = st.cnt;
    }
   }
  }

  tc_fence_before();
  __syncthreads();
  if (kCta == 2) cluster_sync_all();  // the leader's MMAs read the peer's shared memory until the very end
  if (warp == kMmaWarp) {
    tc_fence_after();
    if (kCta == 2)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((u32)kTmemCols) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((u32)kTmemCols) : "memory");
  }
}

// ---------------------------------------------------------------------------------------
// Threshold seeding: per row, the (k + h)-th largest of the m sampled scores (h = number of
// mask entries of the row, so that even if every masked item were in the sample at least k
// unmasked sampled items score that much) is a valid lower bound of the row's k-th best.
// One block per row, MSB-first radix select over ord32(score).
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) seed_tau_kernel(const float* __restrict__ scores, long long ld, int m, int B,
                                                       int k, const long long* __restrict__ mask_indptr,
                                                       u32* __restrict__ g_tau, uint2* __restrict__ g_hpar) {
  __shared__ u32 hist[256];
  __shared__ u32 s_d, s_need, s_max;
  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31;
  long long h = mask_indptr ? (mask_indptr[row + 1] - mask_indptr[row]) : 0;
  long long kth = (long long)k + h;
  if (kth > m) return;  // no bound for this row (its histogram stays disabled: g_hpar zeroed)
  const float* r = scores + (long long)row * ld;
  u32 prefix = 0, pmask = 0;
  int need = (int)kth;
  if (tid == 0) s_max = 0u;
  u32 mx = 0u;  // best finite sampled score (upper end of the row's histogram range): found in pass 1
  for (int shift = 24; shift >= 0; shift -= 8) {
    hist[tid] = 0;
    __syncthreads();
    for (int i = tid; i < m; i += 256) {
      const u32 o = ord32(r[i]);
      if (shift == 24 && o <= 0xFF7FFFFFu && o > mx) mx = o;
      if ((o & pmask) == prefix) atomicAdd(&hist[(o >> shift) & 255u], 1u);
    }
    if (shift == 24) {
#pragma unroll
      for (int off = 16; off; off >>= 1) { const u32 a = __shfl_xor_sync(0xffffffffu, mx, off); mx = a > mx ? a : mx; }
      if (lane == 0) atomicMax(&s_max, mx);
    }
    __syncthreads();
    if (tid < 32) {
      u32 c[8], lane_sum = 0;
#pragma unroll
      for (int t = 0; t < 8; ++t) { c[t] = hist[lane * 8 + t]; lane_sum += c[t]; }
      u32 incl = lane_sum;
#pragma unroll
      for (int off = 1; off < 32; off <<= 1) {
        const u32 t = __shfl_down_sync(0xffffffffu, incl, off);
        if (lane + off < 32) incl += t;
      }
      const u32 above = incl - lane_sum;
      if (above < (u32)need && (u32)need <= incl) {
        u32 run = above;
        bool done = false;
#pragma unroll
        for (int t = 7; t >= 0; --t) {
          if (!done) {
            if (run + c[t] >= (u32)need) { s_d = lane * 8 + t; s_need = need - run; done = true; }
            else run += c[t];
          }
        }
      }
    }
    __syncthreads();
    prefix |= s_d << shift;
    pmask |= 0xFFu << shift;
    need = (int)s_need;
    __syncthreads();
  }
  if (tid == 0 && prefix >= 0x00800000u && prefix <= 0xFF7FFFFFu) {  // finite scores only
    g_tau[row] = prefix;
    if (g_hpar && s_max >= prefix) {
      // kHistBins buckets of width 2^shift from the seed bound to a little beyond the best sampled
      // score (the final k-th best of a row lies around the sample's best when k ~ N / m)
      const u32 span = s_max - prefix;
      const unsigned long long want = (unsigned long long)span + (span >> 3) + 1ull;
      u32 shift = 0;
      while (((unsigned long long)kHistBins << shift) < want) ++shift;
      g_hpar[row] = make_uint2(prefix, shift + 1u);
    }
  }
}

int launch_seed_tau(const float* scores, long long ld, int m, int B, int k, const long long* mask_indptr, u32* g_tau,
                    uint2* g_hpar, cudaStream_t st) {
  if (B <= 0) return 0;
  seed_tau_kernel<<<B, 256, 0, st>>>(scores, ld, m, B, k, mask_indptr, g_tau, g_hpar);
  return (int)cudaGetLastError();
}

// ---------------------------------------------------------------------------------------
// host side: tensor maps + launch
// ---------------------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(ptr);
  }
  return fn;
}

// 2-D bf16 row-major [rows, D] with row pitch ld elements; box = 64 x box_rows, 128B swizzle
static int make_tmap(CUtensorMap* m, const void* base, long long rows, int D, long long ld, int box_rows) {
  EncodeTiledFn fn = get_encode_fn();
  if (!fn) return -1;
  cuuint64_t dims[2] = {(cuuint64_t)D, (cuuint64_t)rows};
  cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
  cuuint32_t box[2] = {(cuuint32_t)kKBlock, (cuuint32_t)box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = fn(m, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS ? 0 : -(int)r - 1000;
}

template <int kMode, int kCta>
static int launch_variant(const CUtensorMap& tq, const CUtensorMap& ti, const SelectParams& p, cudaStream_t st,
                          int num_sms) {
  auto kern = select_tc_kernel<kMode, kCta>;
  cudaError_t e = cudaSuccess;
  {
    // the attribute is per function and device: set it once, not on every launch
    static bool attr_done[64];
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); dev = -1; }
    if (dev < 0 || !attr_done[dev]) {
      e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kTcSmemBytes);
      if (e != cudaSuccess) return (int)e;
      if (dev >= 0) attr_done[dev] = true;
    }
  }
  const int n_units = p.n_q_tiles * p.S;
  int workers = num_sms / kCta;  // persistent CTAs (kCta = 1) or CTA pairs (kCta = 2)
  if (n_units < workers) workers = n_units;
  if (workers < 1) workers = 1;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)(workers * kCta));
  cfg.blockDim = dim3(kTcThreads);
  cfg.dynamicSmemBytes = kTcSmemBytes;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCta; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr; cfg.numAttrs = 1;
  e = cudaLaunchKernelEx(&cfg, kern, tq, ti, p);
  return (int)e;
}

// p.n_q_tiles counts 128-row tiles for one-CTA units and 256-row tiles when p.two_cta is set
int launch_select_tc(const SelectParams& p, cudaStream_t st, int num_sms) {
  CUtensorMap tq, ti;
  int r = make_tmap(&tq, p.q, p.q_rows > p.B ? p.q_rows : p.B, p.D, p.ldq, kQTile);
  if (r) return r;
  r = make_tmap(&ti, p.items, p.n_items, p.D, p.ldi, p.two_cta ? kITile / 2 : kITile);
  if (r) return r;
  if (p.dense_out) return p.store_max8 ? launch_variant<3, 1>(tq, ti, p, st, num_sms) : launch_variant<2, 1>(tq, ti, p, st, num_sms);
  if (p.two_cta) return p.mask_cols ? launch_variant<1, 2>(tq, ti, p, st, num_sms) : launch_variant<0, 2>(tq, ti, p, st, num_sms);
  return p.mask_cols ? launch_variant<1, 1>(tq, ti, p, st, num_sms) : launch_variant<0, 1>(tq, ti, p, st, num_sms);
}

}  // namespace ccr
