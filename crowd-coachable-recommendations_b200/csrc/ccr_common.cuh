// Shared device helpers: sortable keys; mask lookup, CSR row lookup and the mask value rule; the
// 256-bin histogram select steps every top-k path uses; warp-cooperative selection on candidate
// buffers (exact radix select, in-place compaction, approximate histogram prune); small PTX wrappers.
#pragma once
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/ccr_b200.h"
namespace ccr {

typedef unsigned long long u64;
typedef unsigned int u32;

constexpr int kQTile = 128;   // query rows per tensor-core tile (UMMA M)
constexpr int kITile = 256;   // item rows per tensor-core tile (UMMA N)
constexpr int kKBlock = 64;   // K elements per pipeline stage (= one 128-byte swizzle row)
constexpr int kSimtRows = 8;  // query rows per SIMT pass
constexpr int kSimtChunk = 32;  // items per SIMT block iteration

// ---------------------------------------------------------------------------------------
// Sortable keys.  Larger key == better rank (score descending, then item id ascending).
//   dense candidates: 64-bit  [ ord32(score) : ~local_id ]
// ---------------------------------------------------------------------------------------
__host__ __device__ __forceinline__ u32 ord32(float f) {
#ifdef __CUDA_ARCH__
  u32 b = __float_as_uint(f);
#else
  union { float f; u32 u; } c; c.f = f; u32 b = c.u;
#endif
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__host__ __device__ __forceinline__ float unord32(u32 o) {
  u32 b = (o & 0x80000000u) ? (o & 0x7fffffffu) : ~o;
#ifdef __CUDA_ARCH__
  return __uint_as_float(b);
#else
  union { float f; u32 u; } c; c.u = b; return c.f;
#endif
}
__host__ __device__ __forceinline__ u64 ord64(double d) {
#ifdef __CUDA_ARCH__
  u64 b = (u64)__double_as_longlong(d);
#else
  union { double d; u64 u; } c; c.d = d; u64 b = c.u;
#endif
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__host__ __device__ __forceinline__ double unord64(u64 o) {
  u64 b = (o >> 63) ? (o & 0x7fffffffffffffffull) : ~o;
#ifdef __CUDA_ARCH__
  return __longlong_as_double((long long)b);
#else
  union { double d; u64 u; } c; c.u = b; return c.d;
#endif
}
__host__ __device__ __forceinline__ u64 make_key(float s, u32 id) {
  return ((u64)ord32(s) << 32) | (u64)(0xFFFFFFFFu - id);
}
__host__ __device__ __forceinline__ float key_score(u64 k) { return unord32((u32)(k >> 32)); }
__host__ __device__ __forceinline__ u32 key_id(u64 k) { return 0xFFFFFFFFu - (u32)k; }

// candidate-buffer capacity for a given k: room for >= k fresh inserts between prunes plus
// `slack` columns that may be appended before the next prune opportunity (32 for the SIMT
// kernel: one block iteration; 128 for the tensor-core kernel: one half tile), multiple of 64
__host__ __device__ __forceinline__ int cand_capacity(int k, int slack) { return ((2 * k + slack + 63) / 64) * 64; }

// smallest float strictly greater than x (x finite): "s > x"  <=>  "s >= next_up(x)"
__device__ __forceinline__ float next_up(float x) {
  if (!(x == x) || x == INFINITY) return x;
  if (x == 0.f) return __uint_as_float(1u);
  u32 b = __float_as_uint(x);
  return __uint_as_float(x > 0.f ? b + 1u : b - 1u);
}

// ---------------------------------------------------------------------------------------
// mask lookup: is `col` present in the sorted list cols[beg, end) ?
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ bool mask_contains(const int* __restrict__ cols, long long beg, long long end,
                                              int col) {
  while (beg < end) {
    long long mid = (beg + end) >> 1;
    int c = __ldg(cols + mid);
    if (c == col) return true;
    if (c < col) beg = mid + 1; else end = mid;
  }
  return false;
}

// ---------------------------------------------------------------------------------------
// explicit shared-memory accessors (32-bit shared addresses): keeps the selection code on
// LDS / STS / ATOMS instead of generic LD / ST / ATOM when pointers lose their address space
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ u32 smem_addr(const void* p) { return (u32)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void sm_red_inc(u32 a) { asm volatile("red.shared.add.u32 [%0], 1;" ::"r"(a) : "memory"); }
__device__ __forceinline__ u32 sm_ld32(u32 a) { u32 v; asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sm_st32(u32 a, u32 v) { asm volatile("st.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ u64 sm_ld64(u32 a) { u64 v; asm volatile("ld.shared.u64 %0, [%1];" : "=l"(v) : "r"(a) : "memory"); return v; }
__device__ __forceinline__ void sm_st64(u32 a, u64 v) { asm volatile("st.shared.u64 [%0], %1;" ::"r"(a), "l"(v) : "memory"); }

struct GlobalKeys {
  u64* p;
  __device__ __forceinline__ u64 get(int i) const { return p[i]; }
  __device__ __forceinline__ void set(int i, u64 v) const { p[i] = v; }
};
struct SharedKeys {
  u32 s;
  __device__ __forceinline__ u64 get(int i) const { return sm_ld64(s + (u32)i * 8u); }
  __device__ __forceinline__ void set(int i, u64 v) const { sm_st64(s + (u32)i * 8u, v); }
};

// ---------------------------------------------------------------------------------------
// 256-bin histogram select, shared by every prune, seed and finalize step.  Lane L owns bins
// [8L, 8L+8), so higher lanes hold higher bins.  warp_hist_scan loads the lane's bins into c
// and returns the count in the bins of the lanes above it; warp_hist_locate then finds the bin
// where the count from the top reaches `need` (1-based).  All 32 lanes call both.
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ u32 warp_hist_scan(u32 hist_s, u32 (&c)[8]) {
  const int lane = threadIdx.x & 31;
  u32 lane_sum = 0;
#pragma unroll
  for (int t = 0; t < 8; ++t) { c[t] = sm_ld32(hist_s + (u32)(lane * 8 + t) * 4u); lane_sum += c[t]; }
  u32 incl = lane_sum;  // keys in bins owned by lanes >= lane
#pragma unroll
  for (int off = 1; off < 32; off <<= 1) {
    const u32 t = __shfl_down_sync(0xffffffffu, incl, off);
    if (lane + off < 32) incl += t;
  }
  return incl - lane_sum;
}

struct HistBin {
  u32 bin;    // the bin where the count from the top reaches `need`
  u32 above;  // keys in the bins above it
  u32 count;  // keys in it
};

// Every lane gets the same answer.  When need exceeds the total, no lane owns it and the result
// is lane 31's {0, 0, 0}.
__device__ __forceinline__ HistBin warp_hist_locate(const u32 (&c)[8], u32 above, u32 need) {
  const int lane = threadIdx.x & 31;
  u32 lane_sum = 0;
#pragma unroll
  for (int t = 0; t < 8; ++t) lane_sum += c[t];
  const bool mine = above < need && need <= above + lane_sum;
  HistBin r = {0u, 0u, 0u};
  u32 run = above;
  bool done = !mine;
#pragma unroll
  for (int t = 7; t >= 0; --t) {
    const u32 prev = run;
    run += c[t];
    if (!done && run >= need) { r.bin = lane * 8 + t; r.above = prev; r.count = c[t]; done = true; }
  }
  const int src = __ffs(__ballot_sync(0xffffffffu, mine)) - 1;
  r.bin = __shfl_sync(0xffffffffu, r.bin, src);
  r.above = __shfl_sync(0xffffffffu, r.above, src);
  r.count = __shfl_sync(0xffffffffu, r.count, src);
  return r;
}

// m-th largest (1-based, repeats counted) of the nonzero values the 32 lanes hold; 0 when fewer
// than m are nonzero.  Lanes without a value pass 0.
__device__ __forceinline__ u32 warp_mth_largest(u32 v, int m) {
  int gt = 0, ge = 0;
#pragma unroll 4
  for (int i = 0; i < 32; ++i) {
    const u32 o = __shfl_sync(0xffffffffu, v, i);
    gt += (o > v);
    ge += (o >= v);
  }
  const unsigned who = __ballot_sync(0xffffffffu, v != 0u && gt < m && m <= ge);
  return who ? __shfl_sync(0xffffffffu, v, __ffs(who) - 1) : 0u;
}

// ---------------------------------------------------------------------------------------
// Warp-cooperative exact selection on n unique 64-bit keys.  Returns the `kth` largest key
// (1-based).  hist_s: shared address of 256 x u32 private to the warp.  MSB-first 8-bit radix
// select with early exit once the target bin holds one key.  All 32 lanes call it with
// identical arguments.
// ---------------------------------------------------------------------------------------
template <class Keys>
__device__ __forceinline__ u64 warp_select_kth(Keys keys, int n, int kth, u32 hist_s) {
  const int lane = threadIdx.x & 31;
  u64 prefix = 0, pmask = 0;
  int need = kth;
  for (int shift = 56; shift >= 0; shift -= 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) sm_st32(hist_s + (u32)(lane * 8 + j) * 4u, 0u);
    __syncwarp();
    for (int i = lane; i < n; i += 32) {
      u64 key = keys.get(i);
      if ((key & pmask) == prefix) sm_red_inc(hist_s + ((u32)(key >> shift) & 255u) * 4u);
    }
    __syncwarp();
    u32 c[8];
    const u32 above = warp_hist_scan(hist_s, c);
    const HistBin b = warp_hist_locate(c, above, (u32)need);  // kth <= n: found
    prefix |= (u64)b.bin << shift;
    pmask |= 0xFFull << shift;
    need -= (int)b.above;
    __syncwarp();
    if (b.count == 1 && shift > 0) {
      // unique key with this prefix: find it
      u64 found = 0;
      for (int i = lane; i < n; i += 32) {
        u64 key = keys.get(i);
        if ((key & pmask) == prefix) found = key;
      }
#pragma unroll
      for (int off = 16; off; off >>= 1) {
        u64 o = __shfl_xor_sync(0xffffffffu, found, off);
        found = found > o ? found : o;
      }
      return found;
    }
  }
  return prefix;
}

// Keep only keys >= pivot: src[0,n) -> dst[0, kept), stable.  dst may alias src (in place).
template <class Src, class Dst>
__device__ __forceinline__ int warp_compact_ge(Src src, Dst dst, int n, u64 pivot) {
  const int lane = threadIdx.x & 31;
  int base = 0;
  for (int i0 = 0; i0 < n; i0 += 32) {
    int i = i0 + lane;
    u64 key = (i < n) ? src.get(i) : 0ull;
    bool keep = (i < n) && (key >= pivot);
    unsigned m = __ballot_sync(0xffffffffu, keep);
    __syncwarp();
    if (keep) dst.set(base + __popc(m & ((1u << lane) - 1u)), key);
    base += __popc(m);
    __syncwarp();
  }
  return base;
}

// Prune a candidate buffer in global memory down to its exact top-k; returns the pivot (k-th
// largest key).  With stage_s != 0 the keys are first copied to that shared-memory staging area
// (>= n keys) so the radix passes run at shared-memory latency.
__device__ __forceinline__ u64 warp_prune(u64* buf, int n, int k, u32 hist_s, u32 stage_s) {
  const int lane = threadIdx.x & 31;
  __syncwarp();
  u64 pivot;
  if (stage_s) {
    for (int i = lane; i < n; i += 32) sm_st64(stage_s + (u32)i * 8u, buf[i]);
    __syncwarp();
    pivot = warp_select_kth(SharedKeys{stage_s}, n, k, hist_s);
    warp_compact_ge(SharedKeys{stage_s}, GlobalKeys{buf}, n, pivot);
  } else {
    pivot = warp_select_kth(GlobalKeys{buf}, n, k, hist_s);
    warp_compact_ge(GlobalKeys{buf}, GlobalKeys{buf}, n, pivot);
  }
  __syncwarp();
  return pivot;
}

// The outcome of one prune step (warp_prune_stream below): a later candidate (s, id) of the
// stream passes when s >= tau_f and make_key(s, id) > tau_key.
struct PruneResult {
  int kept;      // keys left in buf[0, kept)
  float tau_f;
  u64 tau_key;
  u32 j_ord;     // histogram path: ord32 score with >= j kept keys at or above it
  bool hist;     // the histogram path ran
};

// ---------------------------------------------------------------------------------------
// Approximate histogram prune (the common case).  Keys are bucketed by the 8 score bits just
// below the bits all n keys share, and everything at or above the bucket where the running count
// from the top reaches k is kept: between k and k + (that bucket's population - 1) survivors,
// which is all a *threshold* needs (any value with >= k candidates at or above it is a valid lower
// bound of the k-th best).  The same histogram gives, for free, a value with >= j candidates at or
// above it (the stream's contribution to the shared row bound).
// kLevels = 2 refines once: when the boundary bucket is too crowded to keep whole, that bucket
// alone is split into 256 finer ones by one more pass (BM25 scores of a young stream span many
// binades, so its boundary bucket often is).
// Returns false (nothing modified) when the keys do not spread over buckets (ties) or the
// boundary bucket is still too crowded; the caller then falls back to the exact radix select.
// Otherwise the survivors, exactly the keys with ord32 score >= pivot_ord, are compacted to
// buf[0, r.kept), and r.tau_f = unord32(pivot_ord).
// kStaged: keys are first copied to shared memory (stage_s) and the later passes read them there;
// otherwise (buffers larger than the staging area) every pass streams the keys from global memory.
// ---------------------------------------------------------------------------------------
template <bool kStaged, int kLevels>
__device__ __forceinline__ bool warp_prune_hist(u64* buf, int n, int k, int j, int max_keep, u32 hist_s,
                                                u32 stage_s, PruneResult& r) {
  const int lane = threadIdx.x & 31;
  __syncwarp();
  u32 mx = 0u, mn = 0xFFFFFFFFu;
  for (int i = lane; i < n; i += 32) {
    const u64 key = buf[i];
    if (kStaged) sm_st64(stage_s + (u32)i * 8u, key);
    const u32 o = (u32)(key >> 32);
    mx = o > mx ? o : mx;
    mn = o < mn ? o : mn;
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) {
    const u32 a = __shfl_xor_sync(0xffffffffu, mx, off), b = __shfl_xor_sync(0xffffffffu, mn, off);
    mx = a > mx ? a : mx;
    mn = b < mn ? b : mn;
  }
  const u32 d = mx ^ mn;
  if (d == 0u) return false;
  const int hb = 31 - __clz(d);
  int shift = hb > 7 ? hb - 7 : 0;
  u32 edge = (mn >> shift) << shift;  // ord of bucket 0's lower edge; bucket = (ord - edge) >> shift in [0, 255]
  u32 width = 0u;                     // level 1: ord span of the crowded bucket it splits
  u32 need = (u32)k, kept_above = 0u;  // still to find inside the current range / keys kept above it
  u32 pivot_ord = 0u, j_ord = 0u;
#pragma unroll
  for (int level = 0; level < kLevels; ++level) {
#pragma unroll
    for (int t = 0; t < 8; ++t) sm_st32(hist_s + (u32)(lane * 8 + t) * 4u, 0u);
    __syncwarp();
    for (int i = lane; i < n; i += 32) {
      const u32 o = kStaged ? (u32)(sm_ld64(stage_s + (u32)i * 8u) >> 32) : (u32)(buf[i] >> 32);
      if (level == 0 || o - edge < width) sm_red_inc(hist_s + ((o - edge) >> shift) * 4u);  // unsigned: o < edge fails too
    }
    __syncwarp();
    u32 c[8];
    const u32 above = warp_hist_scan(hist_s, c);
    const HistBin bk = warp_hist_locate(c, above, need);
    if (level == 0) j_ord = edge + (warp_hist_locate(c, above, (u32)j).bin << shift);  // level 0 sees every key
    pivot_ord = edge + (bk.bin << shift);
    if ((int)(kept_above + bk.above + bk.count) <= max_keep) break;  // keep the boundary bucket whole
    if (level == kLevels - 1 || shift == 0) return false;
    // split the boundary bucket: the keys above it are kept anyway
    kept_above += bk.above;
    need -= bk.above;
    edge = pivot_ord;
    width = 1u << shift;
    shift = shift > 8 ? shift - 8 : 0;
    __syncwarp();
  }
  if (pivot_ord < 0x00800000u) pivot_ord = 0x00800000u;  // never below ord32(-FLT_MAX): stays a finite float
  if (j_ord < 0x00800000u) j_ord = 0x00800000u;
  // (u32)(key >> 32) >= pivot_ord  <=>  key >= (u64)pivot_ord << 32
  const u64 pivot = (u64)pivot_ord << 32;
  const int kept = kStaged ? warp_compact_ge(SharedKeys{stage_s}, GlobalKeys{buf}, n, pivot)
                           : warp_compact_ge(GlobalKeys{buf}, GlobalKeys{buf}, n, pivot);
  r = {kept, unord32(pivot_ord), 0ull, j_ord, true};
  return true;
}

// ---------------------------------------------------------------------------------------
// One prune step of a streaming top-k: shrink a candidate buffer and raise the bound later
// candidates of the stream must pass (PruneResult).  Both forms keep every key that can still
// rank in the top k:
//   exact path (warp_prune): buf keeps the k largest keys and the k-th, `pivot`, becomes a *strict*
//     key bound: tau_f = key_score(pivot), tau_key = pivot.  Keys are unique, so a new key ranks
//     in the top k only if it is larger than the pivot -- including a score tied with the pivot's
//     whose id is lower.  A stream that visits ids in ascending order can drop the key compare: a
//     later id never beats a tied pivot, so s >= next_up(key_score(pivot)) is the same bound.
//   histogram path (warp_prune_hist): buf keeps every key whose score is >= unord32(pivot_ord),
//     at least k of them, so tau_f = unord32(pivot_ord) and tau_key = 0.  A score equal to that
//     edge may tie a kept key and still rank, so it passes (>=) and no key compare applies.
// kLevels = 0: exact path only.  Otherwise the histogram prune is tried first with that refinement
// depth; ties or a boundary bucket too crowded for max_keep fall back to the exact path.  j and
// max_keep are read by the histogram path only.  All 32 lanes call it with identical arguments.
// ---------------------------------------------------------------------------------------
template <bool kStaged, int kLevels>
__device__ __forceinline__ PruneResult warp_prune_stream(u64* buf, int n, int k, int j, int max_keep, u32 hist_s,
                                                         u32 stage_s) {
  PruneResult r;
  if constexpr (kLevels > 0) {
    if (warp_prune_hist<kStaged, kLevels>(buf, n, k, j, max_keep, hist_s, stage_s, r)) return r;
  }
  const u64 pivot = warp_prune(buf, n, k, hist_s, kStaged ? stage_s : 0u);
  return {k, key_score(pivot), pivot, 0u, false};
}

// The state of one candidate stream that every thread of a block appends to, in shared memory.
// One thread calls init; one warp prunes with warp_prune_stream and hands the result to apply.
struct BlockStream {
  int cnt;        // keys in the stream's buffer
  float tau_f;    // the PruneResult bound: -inf before the first prune
  u64 tau_key;
  u32 hist[256];  // the pruning warp's histogram

  __device__ __forceinline__ void init() { cnt = 0; tau_f = -INFINITY; tau_key = 0ull; }
  // Append (s, id) when it passes the bound (tf, tk): the record's own, or a copy of it read
  // before a block vote.
  __device__ __forceinline__ void append(u64* buf, float s, u32 id, float tf, u64 tk) {
    if (s >= tf) {
      const u64 key = make_key(s, id);
      if (key > tk) buf[atomicAdd(&cnt, 1)] = key;
    }
  }
  // lane 0 of the pruning warp publishes the new count and bound
  __device__ __forceinline__ void apply(const PruneResult& r) {
    if ((threadIdx.x & 31) == 0) { cnt = r.kept; tau_f = r.tau_f; tau_key = r.tau_key; }
  }
};

// ---------------------------------------------------------------------------------------
// misc
// ---------------------------------------------------------------------------------------
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ float bf16_lo(u32 w) { return __uint_as_float(w << 16); }
__device__ __forceinline__ float bf16_hi(u32 w) { return __uint_as_float(w & 0xffff0000u); }
__device__ __forceinline__ float f16_lo(u32 w) { return __half2float(__ushort_as_half((unsigned short)(w & 0xffffu))); }
__device__ __forceinline__ float f16_hi(u32 w) { return __half2float(__ushort_as_half((unsigned short)(w >> 16))); }

// Stored table / query element (2 bytes): bf16 (default) or IEEE binary16 (CCR_FLAG_F16).  lo / hi
// widen the low / high element of a packed pair exactly; from_float rounds to nearest even.
template <typename T> struct Elem;
template <> struct Elem<__nv_bfloat16> {
  static __device__ __forceinline__ float lo(u32 w) { return bf16_lo(w); }
  static __device__ __forceinline__ float hi(u32 w) { return bf16_hi(w); }
  static __device__ __forceinline__ float to_float(__nv_bfloat16 v) { return __bfloat162float(v); }
  static __device__ __forceinline__ __nv_bfloat16 from_float(float v) { return __float2bfloat16_rn(v); }
};
template <> struct Elem<__half> {
  static __device__ __forceinline__ float lo(u32 w) { return f16_lo(w); }
  static __device__ __forceinline__ float hi(u32 w) { return f16_hi(w); }
  static __device__ __forceinline__ float to_float(__half v) { return __half2float(v); }
  static __device__ __forceinline__ __half from_float(float v) { return __float2half_rn(v); }
};
// fp32 rows of an exact table (ingest only)
template <> struct Elem<float> {
  static __device__ __forceinline__ float to_float(float v) { return v; }
  static __device__ __forceinline__ float from_float(float v) { return v; }
};

// Exact ranking (DESIGN.md section 6b): a bound E on |s^ - s| for one query row, where s^ is the fp32
// score any scan kernel computes from the scan-format copies (bf16, or fp16 when f16) of the fp32 rows q
// and v, and s = fp32(sum q_i v_i summed in float64) is the exact value.  q_norm = ||q||_2, v_max = the
// largest ||v||_2 of the table (both of the fp32 rows, rounded up).  Terms, with u the unit roundoff of
// the scan format and eta its largest absolute rounding error below the normal range (gradual underflow):
//   operand rounding        (2u + u^2) ||q|| V + (1 + u) eta sqrt(D) (||q|| + V) + D eta^2
//   fp32 accumulation       D 2^-22 A, A >= sum |q^_i v^_i|: ASSUMED for the tensor cores (undocumented;
//                           4x the round-to-nearest bound D 2^-24 of the CUDA-core kernels)
//   fp32 underflow          D 2^-149 (bf16 products and partial sums below fp32's normal range)
//   rounding of s itself    (2^-24 + D 2^-53) ||q|| V
// times (1 + 2^-20) for the round-to-nearest arithmetic of this function.  The one implementation: the
// certify kernel calls it, ccr_exact_error_bound exports it, ccr_b200.engine.exact_error_bound mirrors
// it for the tests.
__host__ __device__ inline double exact_error_bound(double q_norm, double v_max, int D, int f16) {
  const double u = f16 ? 0x1p-11 : 0x1p-8;
  const double eta = f16 ? 0x1p-25 : 0x1p-134;
  const double d = (double)D;
  const double qv = q_norm * v_max;
  const double under = (1.0 + u) * eta * sqrt(d) * (q_norm + v_max) + d * eta * eta;
  const double a = (1.0 + u) * (1.0 + u) * qv + under;
  const double e = (2.0 * u + u * u) * qv + under + d * 0x1p-22 * a + d * 0x1p-149 + (0x1p-24 + d * 0x1p-53) * qv;
  return e * (1.0 + 0x1p-20);
}

// error slots written by device-side watchdogs (workspace tail)
struct DeviceStatus {
  int code;     // 0 ok
  int where;    // role / barrier id
  int block;
  int extra;
};

// ---------------------------------------------------------------------------------------
// sparse rows: CSR row lookup and the value rule of mask entries
// ---------------------------------------------------------------------------------------
// row of flat entry e of a CSR with n_rows rows: the largest r with indptr[r] <= e (indptr[0] <= e < indptr[n_rows])
template <typename I>
__device__ __forceinline__ I csr_row_of(const long long* __restrict__ indptr, I n_rows, long long e) {
  I lo = 0, hi = n_rows;  // invariant: indptr[lo] <= e < indptr[hi]
  while (hi - lo > 1) { const I mid = (lo + hi) >> 1; if (indptr[mid] <= e) lo = mid; else hi = mid; }
  return lo;
}

// the value a mask entry ranks by: CCR_MASK_SET the mask value, CCR_MASK_ADD double(score) + value
__device__ __forceinline__ double mask_value(int mode, float score, double v) {
  return mode == CCR_MASK_SET ? v : (double)score + v;
}

}  // namespace ccr
