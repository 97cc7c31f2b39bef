// CUDA-core kernels of the score-and-rank path:
//   select_simt_kernel  : streaming score + mask-exclusion + running top-k, B <= 8 rows per pass
//                         (bandwidth-bound small-query-batch regime; 128-bit coalesced loads)
//   entry_records_kernel: finalize's records of mask entries (and exact-path candidates), float64 values
//   finalize_kernel     : per row, exact top-k of (unit candidates U entry records), sorted
//   merge_topk_kernel   : G-way merge of per-shard sorted lists (multi-GPU exchange step)
//   ingest / normalize / dense helpers
#include "ccr_params.cuh"

namespace ccr {

// =======================================================================================
// SIMT streaming select.  grid = (S, n_groups), block = 256 (8 warps).
// Each block owns one item split and one group of 8 query rows.  Per block iteration it
// scores 32 items x 8 rows: warp w takes items [4w, 4w+4), every lane accumulates a 1/32
// slice of D for 4 items x 8 rows, a 5-step transpose-reduce leaves lane L holding the
// complete dot product of (item L>>3, row L&7), which is then threshold-tested and
// appended to the row's candidate buffer.  A row whose buffer is nearly full is pruned to
// its exact top-k by one warp (radix select in place), raising the row's threshold.
// =======================================================================================
template <typename T>
__global__ void __launch_bounds__(256, 2) select_simt_kernel(SelectParams p) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int D = p.D;
  const T* __restrict__ pq = reinterpret_cast<const T*>(p.q);
  const T* __restrict__ pitems = reinterpret_cast<const T*>(p.items);
  float* qs = reinterpret_cast<float*>(smem_raw);  // [8][D]
  // one stream per row, kept as separate arrays rather than BlockStream records: with the records
  // ptxas holds a row address across the dot-product loop (127 instead of 122 registers)
  __shared__ int s_cnt[kSimtRows];
  __shared__ float s_tau_f[kSimtRows];
  __shared__ u64 s_tau_key[kSimtRows];
  __shared__ u32 s_hist[kSimtRows][256];

  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int split = blockIdx.x, group = blockIdx.y;
  const int row0 = group * kSimtRows;

  // stage the 8 query rows as fp32, laid out [row][half][chunk][4] so that the two float4
  // reads of a lane's 8-element chunk are each contiguous across lanes (no bank conflicts)
  const int chunks = D >> 3;
  for (int i = tid; i < kSimtRows * D; i += 256) {
    int r = i / D, d = i - r * D;
    int row = row0 + r;
    int c = d >> 3, h = (d >> 2) & 1, e = d & 3;
    qs[((r * 2 + h) * chunks + c) * 4 + e] =
        (row < p.B) ? Elem<T>::to_float(pq[(long long)row * p.ldq + d]) : 0.f;
  }
  if (tid < kSimtRows) {
    s_cnt[tid] = 0;
    s_tau_f[tid] = (row0 + tid < p.B) ? -INFINITY : INFINITY;
    s_tau_key[tid] = 0ull;
  }
  __syncthreads();

  long long per = (p.n_items + p.S - 1) / p.S;
  per = (per + kSimtChunk - 1) / kSimtChunk * kSimtChunk;
  const long long i0 = (long long)split * per;
  long long i1 = i0 + per;
  if (i1 > p.n_items) i1 = p.n_items;

  const int my_item = lane >> 3, my_row = lane & 7;
  const int grow = row0 + my_row;
  u64* my_buf = p.cand + ((long long)grow * p.S + split) * p.C;
  long long mbeg = 0, mend = 0;
  if (p.mask_indptr && grow < p.B) { mbeg = p.mask_indptr[grow]; mend = p.mask_indptr[grow + 1]; }

  for (long long base = i0; base < i1; base += kSimtChunk) {
    float acc[32];
#pragma unroll
    for (int i = 0; i < 32; ++i) acc[i] = 0.f;
    const long long it0 = base + warp * 4;
    for (int c = lane; c < chunks; c += 32) {
      uint4 w[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        long long it = it0 + j;
        if (it < i1) w[j] = ldg_nc_v4(pitems + it * p.ldi + c * 8);
        else w[j] = make_uint4(0, 0, 0, 0);
      }
#pragma unroll
      for (int r = 0; r < kSimtRows; ++r) {
        const float4 qa = *reinterpret_cast<const float4*>(qs + ((r * 2 + 0) * chunks + c) * 4);
        const float4 qb = *reinterpret_cast<const float4*>(qs + ((r * 2 + 1) * chunks + c) * 4);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float a = acc[j * 8 + r];
          a = fmaf(Elem<T>::lo(w[j].x), qa.x, a);
          a = fmaf(Elem<T>::hi(w[j].x), qa.y, a);
          a = fmaf(Elem<T>::lo(w[j].y), qa.z, a);
          a = fmaf(Elem<T>::hi(w[j].y), qa.w, a);
          a = fmaf(Elem<T>::lo(w[j].z), qb.x, a);
          a = fmaf(Elem<T>::hi(w[j].z), qb.y, a);
          a = fmaf(Elem<T>::lo(w[j].w), qb.z, a);
          a = fmaf(Elem<T>::hi(w[j].w), qb.w, a);
          acc[j * 8 + r] = a;
        }
      }
    }
    // transpose-reduce: after step with offset o, lanes with bit o keep the upper half
#pragma unroll
    for (int o = 16, n = 16; o >= 1; o >>= 1, n >>= 1) {
      const bool upper = (lane & o) != 0;
#pragma unroll
      for (int i = 0; i < n; ++i) {
        float send = upper ? acc[i] : acc[i + n];
        float keep = upper ? acc[i + n] : acc[i];
        acc[i] = keep + __shfl_xor_sync(0xffffffffu, send, o);
      }
    }
    const float s = acc[0];
    const long long item = it0 + my_item;
    if (item < i1 && s >= s_tau_f[my_row]) {
      u64 key = make_key(s, (u32)item);
      if (key > s_tau_key[my_row] &&
          !(p.mask_cols && mask_contains(p.mask_cols, mbeg, mend, (int)item))) {
        int pos = atomicAdd(&s_cnt[my_row], 1);
        my_buf[pos] = key;  // pos < C: every row has >= 32 free slots at iteration start
      }
    }
    int near_full = 0;
    if (tid < kSimtRows) near_full = s_cnt[tid] > p.C - kSimtChunk;
    if (__syncthreads_or(near_full)) {
      if (warp < kSimtRows) {
        int n = s_cnt[warp];
        if (n > p.C - kSimtChunk) {
          u64* b = p.cand + ((long long)(row0 + warp) * p.S + split) * p.C;
          const PruneResult r = warp_prune_stream<false, 0>(b, n, p.k, 0, 0, smem_addr(s_hist[warp]), 0u);
          if (lane == 0) {
            s_cnt[warp] = r.kept;
            s_tau_key[warp] = r.tau_key;
            s_tau_f[warp] = r.tau_f;
          }
        }
      }
      __syncthreads();
    }
  }
  __syncthreads();
  if (tid < kSimtRows) p.counts[(long long)(row0 + tid) * p.S + split] = s_cnt[tid];
}

template <typename T>
static int launch_select_simt_t(const SelectParams& p, cudaStream_t st) {
  size_t smem = (size_t)kSimtRows * p.D * sizeof(float);
  cudaError_t e = cudaFuncSetAttribute(select_simt_kernel<T>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem);
  if (e != cudaSuccess) return (int)e;
  dim3 grid(p.S, p.n_q_tiles);
  select_simt_kernel<T><<<grid, 256, smem, st>>>(p);
  return (int)cudaGetLastError();
}

int launch_select_simt(const SelectParams& p, cudaStream_t st) {
  return p.f16 ? launch_select_simt_t<__half>(p, st) : launch_select_simt_t<__nv_bfloat16>(p, st);
}

// =======================================================================================
// Entry records (RecordParams): finalize's 96-bit records of the mask entries of the fused and
// dense paths, and of the candidates and mask entries of the exact re-rank.  The kernel owns the
// row lookup, the skip rules, the value rule and the record format; a score source supplies only
// the fp32 score of (row, col) and how many lanes compute it together (kLanes, 1 or 32).
// =======================================================================================
// 2-byte table rows, one warp per entry: lane-strided 8-element chunks, fmaf in element order, then
// the xor butterfly (tests/select_oracle.py: override_values repeats this order bit for bit)
template <typename T>
struct TableDot {
  static constexpr int kLanes = 32;
  static __device__ __forceinline__ float score(const RecordParams& p, int row, long long col, int lane) {
    const T* qr = reinterpret_cast<const T*>(p.q) + (long long)row * p.ldq;
    const T* ir = reinterpret_cast<const T*>(p.items) + col * p.ldi;
    float acc = 0.f;
    for (int c = lane; c < (p.D >> 3); c += 32) {
      uint4 a = *reinterpret_cast<const uint4*>(qr + c * 8);
      uint4 b = ldg_nc_v4(ir + c * 8);
      acc = fmaf(Elem<T>::lo(a.x), Elem<T>::lo(b.x), acc); acc = fmaf(Elem<T>::hi(a.x), Elem<T>::hi(b.x), acc);
      acc = fmaf(Elem<T>::lo(a.y), Elem<T>::lo(b.y), acc); acc = fmaf(Elem<T>::hi(a.y), Elem<T>::hi(b.y), acc);
      acc = fmaf(Elem<T>::lo(a.z), Elem<T>::lo(b.z), acc); acc = fmaf(Elem<T>::hi(a.z), Elem<T>::hi(b.z), acc);
      acc = fmaf(Elem<T>::lo(a.w), Elem<T>::lo(b.w), acc); acc = fmaf(Elem<T>::hi(a.w), Elem<T>::hi(b.w), acc);
    }
#pragma unroll
    for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
    return acc;
  }
};

// sum of a[i] * b[i] over i < D in float64; the order depends on D only (lane-strided float4 chunks, then
// a butterfly that leaves the same sum in every lane).  Products of two fp32 values are exact in float64.
__device__ __forceinline__ double dot_f64(const float* __restrict__ a, const float* __restrict__ b, int D, int lane) {
  double acc = 0.0;
  for (int c = lane; c < (D >> 2); c += 32) {
    const float4 x = *reinterpret_cast<const float4*>(a + c * 4);
    const float4 y = __ldg(reinterpret_cast<const float4*>(b + c * 4));
    acc = fma((double)x.x, (double)y.x, acc);
    acc = fma((double)x.y, (double)y.y, acc);
    acc = fma((double)x.z, (double)y.z, acc);
    acc = fma((double)x.w, (double)y.w, acc);
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  return acc;
}

// fp32 rows of an exact table, one warp per entry: fp32(q . v summed in float64)
struct ExactDot {
  static constexpr int kLanes = 32;
  static __device__ __forceinline__ float score(const RecordParams& p, int row, long long col, int lane) {
    return (float)dot_f64(reinterpret_cast<const float*>(p.q) + (long long)row * p.ldq,
                          reinterpret_cast<const float*>(p.items) + col * p.ldi, p.D, lane);
  }
};

// materialised score matrix, one thread per entry
struct ScoreMatrix {
  static constexpr int kLanes = 1;
  static __device__ __forceinline__ float score(const RecordParams& p, int row, long long col, int) {
    return __ldg(p.scores + (long long)row * p.ld + col);
  }
};

// at least 8 blocks of 256 per SM: <= 32 registers, so all 64 warps of an SM gather rows (ptxas would give
// ExactDot 40 registers and 48 warps otherwise)
template <class Src>
__global__ void __launch_bounds__(256, 8) entry_records_kernel(RecordParams p) {
  const int lane = threadIdx.x % Src::kLanes;
  const long long e = (long long)blockIdx.x * (256 / Src::kLanes) + threadIdx.x / Src::kLanes;
  const long long* ip = p.rec_indptr ? p.rec_indptr : p.mask_indptr;
  if (e >= p.max_entries || e >= ip[p.B]) return;  // max_entries may be an upper bound of ip[B]
  const int row = csr_row_of(ip, p.B, e);
  const long long j = e - ip[row];
  long long c0 = 0, nc = 0;  // the row's candidates: cand_ids[c0, c0 + nc)
  if (p.rec_indptr) {
    c0 = p.cand_indptr ? p.cand_indptr[row] : row * p.cand_stride;
    nc = (p.cand_indptr ? p.cand_indptr[row + 1] : (row + 1) * p.cand_stride) - c0;
  }
  const long long m0 = p.mask_indptr ? p.mask_indptr[row] : 0;
  const long long me = j < nc ? -1 : m0 + (j - nc);  // mask entry, or -1 for a candidate
  const long long col = me < 0 ? p.cand_ids[c0 + j] : p.mask_cols[me];
  bool skip = col < 0 || col >= p.n_cols;
  if (!skip && me < 0 && p.mask_indptr) skip = mask_contains(p.mask_cols, m0, p.mask_indptr[row + 1], (int)col);
  if (skip) {
    if (lane == 0) { p.rec_hi[e] = 0ull; p.rec_lo[e] = 0u; }  // ignored by finalize (hi == 0)
    return;
  }
  const float s = (me >= 0 && p.mode == CCR_MASK_SET) ? 0.f : Src::score(p, row, col, lane);
  const double val = me < 0 ? (double)s : mask_value(p.mode, s, p.mask_vals[me]);
  if (lane == 0) {
    // a NaN value never ranks, like a NaN score in the streams (its ord64 would rank it above +inf): the
    // skipped record, and a masked column's stream candidate is dropped by finalize, so the column is not returned
    const u64 h = ord64(val);
    p.rec_hi[e] = isnan(val) ? 0ull : h ? h : 1ull;  // 0 is reserved for "skipped"
    p.rec_lo[e] = 0xFFFFFFFFu - (u32)col;
  }
}

// the record CSR of rows with candidates: c(r) + m(r)
__global__ void entry_indptr_kernel(RecordParams p) {
  const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (r > p.B) return;
  const long long c = p.cand_indptr ? p.cand_indptr[r] : r * p.cand_stride;
  p.rec_indptr[r] = c + (p.mask_indptr ? p.mask_indptr[r] : 0);
}

template <class Src>
static void launch_entry_records_t(const RecordParams& p, cudaStream_t st) {
  constexpr int kPerBlock = 256 / Src::kLanes;
  entry_records_kernel<Src><<<(unsigned)((p.max_entries + kPerBlock - 1) / kPerBlock), 256, 0, st>>>(p);
}

int launch_entry_records(const RecordParams& p, cudaStream_t st) {
  if (p.B <= 0) return 0;
  if (p.rec_indptr) {
    entry_indptr_kernel<<<(unsigned)((p.B + 256) / 256), 256, 0, st>>>(p);
    const cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return (int)e;
  }
  if (p.max_entries <= 0) return 0;
  switch (p.src) {
    case kRecBf16Dot: launch_entry_records_t<TableDot<__nv_bfloat16>>(p, st); break;
    case kRecF16Dot: launch_entry_records_t<TableDot<__half>>(p, st); break;
    case kRecExactDot: launch_entry_records_t<ExactDot>(p, st); break;
    case kRecMatrix: launch_entry_records_t<ScoreMatrix>(p, st); break;
    default: return (int)cudaErrorInvalidValue;
  }
  return (int)cudaGetLastError();
}

// =======================================================================================
// Finalize: one block (256 threads) per query row.
// Entries: dense candidates of every stream (64-bit keys) and the row's entry records, unified
// as 96-bit sort keys (hi = ord64(double value), lo = ~id).
//   1. prefix-sum the stream counts so the candidates can be walked as one flat, fully parallel
//      index space (one independent global load per entry instead of a serial loop over streams);
//   2. gather into shared memory every dense candidate at or above the row's shared lower bound
//      g_tau (the global top-k is a subset of those) plus all records;
//   3. exact k-th largest by MSB-first radix select (<= 12 passes, early exit) in shared memory,
//      winners compacted, bitonic sorted, written out.
// If the gathered list does not fit (loose bound), the select runs over global memory instead.
// =======================================================================================
constexpr int kFinList = 4096;     // shared-memory entry list capacity
constexpr int kFinMaxStreams = 1024;

struct RowEntries {
  const u64* cand; const int* prefix; int S, C, total;
  const u64* rec_hi; const u32* rec_lo; long long rbeg, rend;
  const u64* l_hi; const u32* l_lo; int l_n;  // shared-memory list (when l_n >= 0)
  const int* drop_cols;                        // include mode: skip dense candidates in the row's mask
  template <class F> __device__ __forceinline__ void for_each(F f) const {
    if (l_n >= 0) {
      for (int i = threadIdx.x; i < l_n; i += blockDim.x) f(l_hi[i], l_lo[i]);
      return;
    }
    for (int i = threadIdx.x; i < total; i += blockDim.x) {
      int lo = 0, hi = S;  // stream u with prefix[u] <= i < prefix[u+1]
      while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (prefix[mid] <= i) lo = mid; else hi = mid; }
      const u64 key = cand[(long long)lo * C + (i - prefix[lo])];
      if (drop_cols && mask_contains(drop_cols, rbeg, rend, (int)key_id(key))) continue;
      f(ord64((double)key_score(key)), (u32)key);
    }
    for (long long e = rbeg + threadIdx.x; e < rend; e += blockDim.x) {
      u64 h = rec_hi[e];
      if (h) f(h, rec_lo[e]);
    }
  }
};

constexpr int kFinMaxThreads = 1024;

__global__ void __launch_bounds__(kFinMaxThreads) finalize_kernel(FinalizeParams p, int P /*pow2 >= k*/) {
  const int NT = blockDim.x;  // 1024 for small batches (latency-bound gather), 256 otherwise
  extern __shared__ __align__(16) unsigned char smem_raw[];
  u64* s_hi = reinterpret_cast<u64*>(smem_raw);                 // [kFinList]
  u32* s_lo = reinterpret_cast<u32*>(s_hi + kFinList);          // [kFinList]
  int* s_prefix = reinterpret_cast<int*>(s_lo + kFinList);      // [kFinMaxStreams + 1]
  __shared__ u32 hist[256];
  __shared__ int s_nwin, s_nlist, s_warp_sums[32];
  __shared__ u32 s_d, s_need, s_binc;

  const int row = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int S = p.S;
  // ---- 1. exclusive prefix sums of the stream counts (<= 4 streams per thread, S <= 1024) ----
  {
    const int per = (S + NT - 1) / NT;
    int loc[4], mine = 0;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int u = tid * per + t;
      loc[t] = (t < per && u < S) ? p.counts[(long long)row * S + u] : 0;
      mine += loc[t];
    }
    int incl = mine;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { int v = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += v; }
    if (lane == 31) s_warp_sums[warp] = incl;
    __syncthreads();
    int base = 0;
    for (int w = 0; w < warp; ++w) base += s_warp_sums[w];
    int run = base + incl - mine;
#pragma unroll
    for (int t = 0; t < 4; ++t) {
      const int u = tid * per + t;
      if (t < per && u < S) { s_prefix[u] = run; run += loc[t]; }
    }
    if (tid == NT - 1) s_prefix[S] = base + incl;
    if (tid == 0) { s_nwin = 0; s_nlist = 0; }
    __syncthreads();
  }
  RowEntries E;
  E.cand = p.cand + (long long)row * S * p.C;
  E.prefix = s_prefix; E.S = S; E.C = p.C; E.total = s_prefix[S];
  E.rec_hi = p.rec_hi; E.rec_lo = p.rec_lo;
  E.rbeg = p.rec_indptr ? p.rec_indptr[row] : 0;
  E.rend = p.rec_indptr ? p.rec_indptr[row + 1] : 0;
  E.l_hi = s_hi; E.l_lo = s_lo; E.l_n = -1;
  E.drop_cols = p.drop_cols;
  const int k = p.k;

  // ---- 2. gather (prefiltered) into shared memory ----
  {
    const u32 tau = p.g_tau ? p.g_tau[row] : 0u;  // ord32 lower bound of the k-th best DENSE score
    // 4 independent loads in flight per thread: the entries live in L2/HBM, latency-bound otherwise
    for (int i0 = tid; i0 < E.total; i0 += 4 * NT) {
      u64 key[4];
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        const int i = i0 + b * NT;
        key[b] = 0ull;
        if (i < E.total) {
          int lo = 0, hi = S;
          while (hi - lo > 1) { int mid = (lo + hi) >> 1; if (s_prefix[mid] <= i) lo = mid; else hi = mid; }
          key[b] = __ldcg(E.cand + (long long)lo * p.C + (i - s_prefix[lo]));
        }
      }
#pragma unroll
      for (int b = 0; b < 4; ++b) {
        bool take = i0 + b * NT < E.total && (u32)(key[b] >> 32) >= tau;
        if (take && p.drop_cols) take = !mask_contains(p.drop_cols, E.rbeg, E.rend, (int)key_id(key[b]));
        if (take) {
          int pos = atomicAdd(&s_nlist, 1);
          if (pos < kFinList) { s_hi[pos] = ord64((double)key_score(key[b])); s_lo[pos] = (u32)key[b]; }
        }
      }
    }
    for (long long e = E.rbeg + tid; e < E.rend; e += NT) {  // records are never filtered
      const u64 h = p.rec_hi[e];
      if (h) {
        int pos = atomicAdd(&s_nlist, 1);
        if (pos < kFinList) { s_hi[pos] = h; s_lo[pos] = p.rec_lo[e]; }
      }
    }
    __syncthreads();
    if (s_nlist <= kFinList) E.l_n = s_nlist;  // fits: everything below runs on shared memory
    __syncthreads();
  }
  if (E.l_n < 0) {  // list overflow: count the surviving entries over global memory
    if (tid == 0) s_nlist = 0;
    __syncthreads();
    int local = 0;
    E.for_each([&](u64, u32) { ++local; });
    atomicAdd(&s_nlist, local);
    __syncthreads();
  }
  const int total = E.l_n >= 0 ? E.l_n : s_nlist;

  u64 phi = 0, mhi = 0;  // prefix over hi
  u32 plo = 0, mlo = 0;  // prefix over lo
  bool select_all = total <= k;
  if (!select_all) {
    int need = k;
    for (int pass = 0; pass < 12; ++pass) {
      if (tid < 256) hist[tid] = 0;
      __syncthreads();
      const int sh = pass < 8 ? 56 - 8 * pass : 24 - 8 * (pass - 8);
      E.for_each([&](u64 hi, u32 lo) {
        if ((hi & mhi) == phi && (lo & mlo) == plo) {
          u32 d = pass < 8 ? (u32)(hi >> sh) & 255u : (lo >> sh) & 255u;
          atomicAdd(&hist[d], 1u);
        }
      });
      __syncthreads();
      if (warp == 0) {
        u32 c[8];
        const u32 above = warp_hist_scan(smem_addr(hist), c);
        const HistBin b = warp_hist_locate(c, above, (u32)need);  // need <= entries with the prefix: found
        if (lane == 0) { s_d = b.bin; s_need = need - b.above; s_binc = b.count; }
      }
      __syncthreads();
      const u32 d = s_d;
      need = (int)s_need;
      if (pass < 8) { phi |= (u64)d << sh; mhi |= 0xFFull << sh; }
      else { plo |= d << sh; mlo |= 0xFFu << sh; }
      if (s_binc == (u32)need) break;  // every key in the bin is a winner: prefix is enough
      __syncthreads();
    }
  }
  __syncthreads();
  // winners: masked key bits >= prefix.  They are compacted into a second region so the source
  // list is not overwritten while it is still being read.
  u64* w_hi = reinterpret_cast<u64*>(s_prefix + kFinMaxStreams + 2);  // [P], 8-byte aligned (see launcher)
  u32* w_lo = reinterpret_cast<u32*>(w_hi + P);
  for (int i = tid; i < P; i += NT) { w_hi[i] = 0ull; w_lo[i] = 0u; }
  __syncthreads();
  E.for_each([&](u64 hi, u32 lo) {
    bool win;
    if (select_all) win = true;
    else {
      u64 a = hi & mhi;
      win = (a > phi) || (a == phi && (lo & mlo) >= plo);
    }
    if (win) {
      int pos = atomicAdd(&s_nwin, 1);
      if (pos < P) { w_hi[pos] = hi; w_lo[pos] = lo; }
    }
  });
  __syncthreads();
  // bitonic sort, descending by (hi, lo); padding entries are (0,0) = smallest
  for (int size = 2; size <= P; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int t = tid; t < (P >> 1); t += NT) {
        int i = 2 * t - (t & (stride - 1));
        int j = i + stride;
        bool desc = ((i & size) == 0);
        u64 hi_i = w_hi[i], hi_j = w_hi[j];
        u32 lo_i = w_lo[i], lo_j = w_lo[j];
        bool i_lt_j = (hi_i < hi_j) || (hi_i == hi_j && lo_i < lo_j);
        if (i_lt_j == desc) { w_hi[i] = hi_j; w_hi[j] = hi_i; w_lo[i] = lo_j; w_lo[j] = lo_i; }
      }
      __syncthreads();
    }
  }
  const int nwin = min(s_nwin, k);
  for (int i = tid; i < k; i += NT) {
    long long o = (long long)row * k + i;
    if (i < nwin) {
      double v = unord64(w_hi[i]);
      const long long gid = (long long)(0xFFFFFFFFu - w_lo[i]) + p.id_offset;
      if (p.out_scores) p.out_scores[o] = (float)v;
      if (p.out_keys) p.out_keys[o] = make_key((float)v, (u32)gid);  // exchange format: [ord32 : ~global id]
      else if (p.out_scores64) p.out_scores64[o] = v;
      p.out_ids[o] = gid;
    } else {
      if (p.out_scores) p.out_scores[o] = -INFINITY;
      if (p.out_keys) p.out_keys[o] = 0ull;  // padding: below every real key
      else if (p.out_scores64) p.out_scores64[o] = -INFINITY;
      p.out_ids[o] = -1;
    }
  }
}

int launch_finalize(const FinalizeParams& p, cudaStream_t st) {
  if (p.S > kFinMaxStreams) return (int)cudaErrorInvalidValue;
  int P = 32;
  while (P < p.k) P <<= 1;
  // list (12 B/entry) + prefix (kFinMaxStreams + 2 ints, keeps the winner region 8-byte aligned) + winners
  size_t smem = (size_t)kFinList * 12 + (size_t)(kFinMaxStreams + 2) * 4 + (size_t)P * 12;
  cudaError_t e = cudaFuncSetAttribute(finalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return (int)e;
  // the gather is latency-bound: few rows -> wide blocks (2 x 1024 threads per SM keep 64 warps of loads
  // in flight); many rows -> 256-thread blocks fill the SMs on their own
  finalize_kernel<<<p.B, p.B <= 1536 ? kFinMaxThreads : 256, smem, st>>>(p, P);
  return (int)cudaGetLastError();
}

// =======================================================================================
// G-way merge of sorted runs (multi-GPU exchange step).  One block per row; every entry
// finds its output rank by binary-searching each of the G runs.
// order: score descending, then id ascending; id < 0 = padding (ignored).
// =======================================================================================
__device__ __forceinline__ bool precedes(double sa, long long ia, double sb, long long ib) {
  return (sa > sb) || (sa == sb && ia < ib);
}

// kStaged: the row's G runs are first copied to shared memory (16 bytes per entry) so that the
// ~G * log2(k) probes of every entry are shared-memory reads; otherwise they go to global memory.
template <bool kStaged>
__global__ void __launch_bounds__(1024) merge_topk_kernel(const double* __restrict__ s,
                                                          const long long* __restrict__ ids, int G,
                                                          long long B, int k_in, int k_out, float* os,
                                                          double* os64, long long* oi) {
  extern __shared__ __align__(16) unsigned char merge_smem[];
  const long long row = blockIdx.x;
  const int n = G * k_in;
  double* l_s = reinterpret_cast<double*>(merge_smem);            // [G][k_in] (staged only)
  long long* l_id = reinterpret_cast<long long*>(l_s + n);        // [G][k_in]
  __shared__ int s_valid;
  if (threadIdx.x == 0) s_valid = 0;
  if (kStaged) {
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
      const int g = e / k_in, i = e - g * k_in;
      const long long off = ((long long)g * B + row) * k_in + i;
      l_s[e] = s[off];
      l_id[e] = ids[off];
    }
  }
  __syncthreads();
  int local_valid = 0;
  for (int e = threadIdx.x; e < n; e += blockDim.x) {
    const int g = e / k_in, i = e - g * k_in;
    const long long off = ((long long)g * B + row) * k_in;
    const long long id = kStaged ? l_id[e] : ids[off + i];
    if (id < 0) continue;
    ++local_valid;
    const double sc = kStaged ? l_s[e] : s[off + i];
    int rank = 0;
    for (int h = 0; h < G && rank < k_out; ++h) {
      const long long oh = ((long long)h * B + row) * k_in;
      // number of valid entries of run h that precede (sc, id); more than k_out - rank of them
      // would push the entry out of the result anyway, so the search stops there
      int lo = 0, hi = k_in < k_out - rank ? k_in : k_out - rank;
      while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const long long mid_id = kStaged ? l_id[h * k_in + mid] : ids[oh + mid];
        const double mid_s = kStaged ? l_s[h * k_in + mid] : s[oh + mid];
        const bool before = (mid_id >= 0) && precedes(mid_s, mid_id, sc, id);
        if (before) lo = mid + 1; else hi = mid;
      }
      rank += lo;
    }
    if (rank < k_out) {
      long long o = row * k_out + rank;
      if (os) os[o] = (float)sc;
      if (os64) os64[o] = sc;
      oi[o] = id;
    }
  }
  atomicAdd(&s_valid, local_valid);
  __syncthreads();
  for (int r = s_valid + threadIdx.x; r < k_out; r += blockDim.x) {
    long long o = row * k_out + r;
    if (os) os[o] = -INFINITY;
    if (os64) os64[o] = -INFINITY;
    oi[o] = -1;
  }
}

int launch_merge_topk(const double* s, const long long* ids, int G, long long B, int k_in, int k_out,
                      float* os, double* os64, long long* oi, cudaStream_t st) {
  if (B == 0) return 0;
  const size_t smem = (size_t)G * k_in * 16;
  if (smem <= 200 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(merge_topk_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
    const int threads = G * k_in >= 4096 ? 1024 : 256;
    merge_topk_kernel<true><<<(unsigned)B, threads, smem, st>>>(s, ids, G, B, k_in, k_out, os, os64, oi);
  } else {
    merge_topk_kernel<false><<<(unsigned)B, 256, 0, st>>>(s, ids, G, B, k_in, k_out, os, os64, oi);
  }
  return (int)cudaGetLastError();
}

// =======================================================================================
// G-way merge of packed 64-bit keys ([ord32(score) : ~global id], larger = better, 0 = padding):
// the 8-byte-per-entry exchange format of the row-sharded path when the order is decided in
// float32.  One block per query row; the G sorted runs are staged in shared memory and merged
// pairwise, log2(G) rounds of merge-path merges: every thread finds the start of its output
// segment with one co-rank binary search (~log2 k probes) and then merges kMergeSeg keys
// sequentially.  Runs are truncated to k_out after every round, so the rounds produce
// (G/2 + G/4 + ... + 1) * k_out keys in total -- against ~G log2(k) probes for EVERY entry in the
// rank-by-search kernel above.
// =======================================================================================
constexpr int kMergeSeg = 4;

__global__ void __launch_bounds__(1024) merge_keys_kernel(const u64* __restrict__ keys, int G, long long B, int k_in,
                                                          int k_out, int n0, float* os, long long* oi, u64* ok) {
  extern __shared__ __align__(16) unsigned char merge_smem[];
  u64* buf0 = reinterpret_cast<u64*>(merge_smem);   // n0 keys: the G input runs, later the even rounds' outputs
  u64* buf1 = buf0 + n0;                            // the odd rounds' outputs
  const long long row = blockIdx.x;
  for (int e = threadIdx.x; e < G * k_in; e += blockDim.x) {
    const int g = e / k_in, i = e - g * k_in;
    buf0[e] = keys[((long long)g * B + row) * k_in + i];
  }
  __syncthreads();
  u64* src = buf0;
  u64* dst = buf1;
  int runs = G, len = k_in;
  while (runs > 1) {
    const int pairs = runs >> 1, odd = runs & 1;
    const int out_len = 2 * len < k_out ? 2 * len : k_out;
    const int segs = (out_len + kMergeSeg - 1) / kMergeSeg;
    for (int w = threadIdx.x; w < pairs * segs; w += blockDim.x) {
      const int pr = w / segs, sg = w - pr * segs;
      const u64* a = src + (size_t)(2 * pr) * len;
      const u64* b = a + len;
      const int d = sg * kMergeSeg;  // diagonal: outputs [d, d + kMergeSeg)
      // co-rank: i keys of a and d - i keys of b precede output d (keys are distinct except padding
      // zeros, whose relative order does not matter)
      int lo = d > len ? d - len : 0, hi = d < len ? d : len;
      while (lo < hi) {
        const int i = (lo + hi) >> 1;
        if (a[i] > b[d - i - 1]) lo = i + 1; else hi = i;
      }
      int i = lo, j = d - lo;
      u64* o = dst + (size_t)pr * out_len + d;
      const int n = out_len - d < kMergeSeg ? out_len - d : kMergeSeg;
      for (int t = 0; t < n; ++t) {
        const bool take_a = (j >= len) || (i < len && a[i] > b[j]);
        o[t] = take_a ? a[i++] : b[j++];
      }
    }
    if (odd) {  // the unpaired run moves on unchanged (truncated)
      const u64* a = src + (size_t)(2 * pairs) * len;
      const int n = len < out_len ? len : out_len;
      for (int t = threadIdx.x; t < out_len; t += blockDim.x) dst[(size_t)pairs * out_len + t] = t < n ? a[t] : 0ull;
    }
    __syncthreads();
    u64* tmp = src; src = dst; dst = tmp;
    runs = pairs + odd;
    len = out_len;
  }
  for (int r = threadIdx.x; r < k_out; r += blockDim.x) {
    const u64 key = r < len ? src[r] : 0ull;
    const long long o = row * k_out + r;
    if (ok) ok[o] = key;
    if (key) { if (os) os[o] = key_score(key); if (oi) oi[o] = (long long)key_id(key); }
    else { if (os) os[o] = -INFINITY; if (oi) oi[o] = -1; }
  }
}

int launch_merge_keys(const u64* keys, int G, long long B, int k_in, int k_out, float* os, long long* oi, u64* ok,
                      cudaStream_t st) {
  if (B == 0) return 0;
  const int ol = 2 * k_in < k_out ? 2 * k_in : k_out;
  // ping-pong buffers sized by replaying the rounds: round r reads buf[(r-1)&1], writes buf[r&1]
  size_t need[2] = {(size_t)G * k_in, 0};
  {
    int runs = G, len = k_in, r = 1;
    while (runs > 1) {
      const int out_len = 2 * len < k_out ? 2 * len : k_out;
      runs = (runs >> 1) + (runs & 1);
      const size_t n = (size_t)runs * out_len;
      if (n > need[r & 1]) need[r & 1] = n;
      len = out_len;
      ++r;
    }
  }
  const size_t n0 = need[0], n1 = need[1];
  const size_t smem = (n0 + n1) * sizeof(u64);
  if (smem > 220 * 1024) return (int)cudaErrorInvalidValue;
  static bool attr_done[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); dev = -1; }
  if (dev < 0 || !attr_done[dev]) {
    cudaError_t e = cudaFuncSetAttribute(merge_keys_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 220 * 1024);
    if (e != cudaSuccess) return (int)e;
    if (dev >= 0) attr_done[dev] = true;
  }
  int threads = (int)(((size_t)(G / 2) * ((ol + kMergeSeg - 1) / kMergeSeg) + 31) / 32 * 32);
  if (threads < 128) threads = 128;
  if (threads > 1024) threads = 1024;
  merge_keys_kernel<<<(unsigned)B, threads, smem, st>>>(keys, G, B, k_in, k_out, (int)n0, os, oi, ok);
  return (int)cudaGetLastError();
}

// packed exchange keys -> (float32 score, int64 global id); key 0 = padding -> (-inf, -1)
__global__ void __launch_bounds__(256) unpack_keys_kernel(const u64* __restrict__ keys, long long n, float* os,
                                                          long long* oi) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const u64 key = keys[i];
  if (os) os[i] = key ? key_score(key) : -INFINITY;
  if (oi) oi[i] = key ? (long long)key_id(key) : -1;
}

int launch_unpack_keys(const u64* keys, long long n, float* os, long long* oi, cudaStream_t st) {
  if (n <= 0) return 0;
  unpack_keys_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(keys, n, os, oi);
  return (int)cudaGetLastError();
}

// =======================================================================================
// Column shard of a mask CSR on the device (row-sharded tables): keep the entries with
// lo <= col < hi, re-based to local columns.  Columns are sorted inside a row, so the kept entries
// of a row are one contiguous range found by two binary searches; one block scans the row counts
// (B is a query batch: a few thousand rows) and copies the ranges.
// =======================================================================================
__global__ void __launch_bounds__(1024) mask_shard_kernel(const long long* __restrict__ indptr,
                                                          const int* __restrict__ cols,
                                                          const double* __restrict__ vals, long long B, int lo, int hi,
                                                          long long* __restrict__ out_indptr, int* __restrict__ out_cols,
                                                          double* __restrict__ out_vals) {
  __shared__ long long s_warp[32];
  __shared__ long long s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid == 0) { s_carry = 0; out_indptr[0] = 0; }
  __syncthreads();
  for (long long r0 = 0; r0 < B; r0 += blockDim.x) {
    const long long r = r0 + tid;
    long long a = 0, b = 0;
    if (r < B) {
      const long long beg = indptr[r], end = indptr[r + 1];
      long long x = beg, y = end;
      while (x < y) { const long long m = (x + y) >> 1; if (cols[m] < lo) x = m + 1; else y = m; }
      a = x; y = end;
      while (x < y) { const long long m = (x + y) >> 1; if (cols[m] < hi) x = m + 1; else y = m; }
      b = x;
    }
    const long long cnt = b - a;
    long long incl = cnt;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const long long v = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += v; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    long long base = s_carry;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    const long long start = base + incl - cnt;
    if (r < B) {
      out_indptr[r + 1] = start + cnt;
      for (long long e = 0; e < cnt; ++e) { out_cols[start + e] = cols[a + e] - lo; out_vals[start + e] = vals[a + e]; }
    }
    __syncthreads();
    if (tid == blockDim.x - 1) s_carry = base + incl;
    __syncthreads();
  }
}

int launch_mask_shard(const long long* indptr, const int* cols, const double* vals, long long B, int lo, int hi,
                      long long* out_indptr, int* out_cols, double* out_vals, cudaStream_t st) {
  if (B < 0) return (int)cudaErrorInvalidValue;
  mask_shard_kernel<<<1, 1024, 0, st>>>(indptr, cols, vals, B, lo, hi, out_indptr, out_cols, out_vals);
  return (int)cudaGetLastError();
}

// =======================================================================================
// Table ingest / normalisation: one warp per row.  DstT = __nv_bfloat16 or __half (round to nearest
// even; fp16 keeps subnormals).  overflow (fp16 tables, may be null): += number of stored values that
// are not finite -- |x| >= 65520 after normalisation rounds to inf, and non-finite inputs stay so;
// one atomic per warp that saw any.
// =======================================================================================
template <typename SrcT, typename DstT>
__global__ void __launch_bounds__(256) ingest_kernel(const SrcT* __restrict__ src, long long n, int D,
                                                     long long ld_src, DstT* __restrict__ dst,
                                                     long long ld_dst, int normalize, int* __restrict__ overflow) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= n) return;
  const SrcT* s = src + row * ld_src;
  float scale = 1.f;
  if (normalize) {
    float ss = 0.f;
    for (int d = lane; d < D; d += 32) { float v = (float)s[d]; ss = fmaf(v, v, ss); }
#pragma unroll
    for (int off = 16; off; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
    scale = fmaxf(sqrtf(ss), 1e-12f);  // F.normalize: x / max(||x||, eps) -- a true division, like torch
  }
  DstT* o = dst + row * ld_dst;
  int bad = 0;
  for (int d = lane; d < ld_dst; d += 32) {
    float v = d < D ? (normalize ? (float)s[d] / scale : (float)s[d]) : 0.f;
    const DstT r = Elem<DstT>::from_float(v);
    if (overflow) bad += isfinite(Elem<DstT>::to_float(r)) ? 0 : 1;
    o[d] = r;
  }
  if (overflow) {
#pragma unroll
    for (int off = 16; off; off >>= 1) bad += __shfl_xor_sync(0xffffffffu, bad, off);
    if (lane == 0 && bad) atomicAdd(overflow, bad);
  }
}

template <typename SrcT, typename DstT>
int launch_ingest(const SrcT* src, long long n, int D, long long ld_src, DstT* dst, long long ld_dst, int normalize,
                  int* overflow, cudaStream_t st) {
  if (n == 0) return 0;
  ingest_kernel<SrcT, DstT><<<(unsigned)((n + 7) / 8), 256, 0, st>>>(src, n, D, ld_src, dst, ld_dst, normalize,
                                                                     overflow);
  return (int)cudaGetLastError();
}
template int launch_ingest(const float*, long long, int, long long, __nv_bfloat16*, long long, int, int*, cudaStream_t);
template int launch_ingest(const float*, long long, int, long long, __half*, long long, int, int*, cudaStream_t);
template int launch_ingest(const float*, long long, int, long long, float*, long long, int, int*, cudaStream_t);
template int launch_ingest(const __nv_bfloat16*, long long, int, long long, __nv_bfloat16*, long long, int, int*,
                           cudaStream_t);
template int launch_ingest(const __half*, long long, int, long long, __half*, long long, int, int*, cudaStream_t);

// =======================================================================================
// Dense fp32 score tile (not a hot path): one warp per (row, item).
// =======================================================================================
template <typename T>
__global__ void __launch_bounds__(256) dense_kernel(const T* __restrict__ q, long long B,
                                                    long long ldq, const T* __restrict__ items,
                                                    long long n, long long ldi, int D,
                                                    float* __restrict__ out, long long ld_out) {
  const int lane = threadIdx.x & 31;
  const long long item = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const long long row = blockIdx.y;
  if (item >= n) return;
  const T* qr = q + row * ldq;
  const T* ir = items + item * ldi;
  float acc = 0.f;
  for (int c = lane; c < (D >> 3); c += 32) {
    uint4 a = *reinterpret_cast<const uint4*>(qr + c * 8);
    uint4 b = *reinterpret_cast<const uint4*>(ir + c * 8);
    acc = fmaf(Elem<T>::lo(a.x), Elem<T>::lo(b.x), acc); acc = fmaf(Elem<T>::hi(a.x), Elem<T>::hi(b.x), acc);
    acc = fmaf(Elem<T>::lo(a.y), Elem<T>::lo(b.y), acc); acc = fmaf(Elem<T>::hi(a.y), Elem<T>::hi(b.y), acc);
    acc = fmaf(Elem<T>::lo(a.z), Elem<T>::lo(b.z), acc); acc = fmaf(Elem<T>::hi(a.z), Elem<T>::hi(b.z), acc);
    acc = fmaf(Elem<T>::lo(a.w), Elem<T>::lo(b.w), acc); acc = fmaf(Elem<T>::hi(a.w), Elem<T>::hi(b.w), acc);
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, off);
  if (lane == 0) out[row * ld_out + item] = acc;
}

template <typename T>
int launch_dense(const T* q, long long B, long long ldq, const T* items, long long n, long long ldi, int D, float* out,
                 long long ld_out, cudaStream_t st) {
  if (B == 0 || n == 0) return 0;
  dim3 grid((unsigned)((n + 7) / 8), (unsigned)B);
  dense_kernel<T><<<grid, 256, 0, st>>>(q, B, ldq, items, n, ldi, D, out, ld_out);
  return (int)cudaGetLastError();
}
template int launch_dense(const __nv_bfloat16*, long long, long long, const __nv_bfloat16*, long long, long long, int,
                          float*, long long, cudaStream_t);
template int launch_dense(const __half*, long long, long long, const __half*, long long, long long, int, float*,
                          long long, cudaStream_t);

// =======================================================================================
// BM25 (lexical sibling of the dense path; reference: scripts/bm_25.py:27-45 scored per query by
// ranking_bm25, scripts/ms_marco_eval.py:165-186, which full-sorts N scores for 1001 outputs).
//   bm25_impacts_kernel : at fit time, per posting (term t, doc d, tf):
//                           val = ((tf * idf_t) * (k1 + 1)) * (1 / (tf + norm[d]))  (float64; scipy
//                         evaluates sparse / dense as a multiplication by the reciprocal)
//                         -- the reference's per-query arithmetic does not depend on the query, so
//                         it is done once; a query then only sums its terms' posting values.
//   bm25_topk_kernel    : block = (doc split, query), 256 threads, 5 blocks per SM (independent barrier
//                         domains hide each other's latency).  The split is walked in chunks of kBmChunk
//                         docs whose float64 score accumulators live in shared memory; the query's
//                         terms are applied one after the other (fixed order -> deterministic sums),
//                         each by streaming the term's postings from a per-term cursor until the
//                         chunk's end (postings are doc-sorted, so no searches in the loop).  The
//                         finished chunk is either ranked -- as float32, like the reference's
//                         torch.Tensor(solution).sort -- through the same candidate / prune /
//                         finalize protocol as the dense kernels (the N-vector never reaches HBM),
//                         or stored (BM25.transform drop-in).
// =======================================================================================
__global__ void __launch_bounds__(256) bm25_impacts_kernel(const long long* __restrict__ post_indptr,
                                                           const int* __restrict__ post_docs,
                                                           const float* __restrict__ post_tf,
                                                           const double* __restrict__ idf,
                                                           const double* __restrict__ doc_norm, double k1p1,
                                                           long long V, long long nnz, double* __restrict__ val) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= nnz) return;
  const long long t = csr_row_of(post_indptr, V, e);  // term of posting e
  const double tf = (double)post_tf[e];
  val[e] = ((tf * idf[t]) * k1p1) * (1.0 / (tf + doc_norm[post_docs[e]]));
}

int launch_bm25_impacts(const long long* post_indptr, const int* post_docs, const float* post_tf, const double* idf,
                        const double* doc_norm, double k1p1, long long V, long long nnz, double* val,
                        cudaStream_t st) {
  if (nnz <= 0) return 0;
  bm25_impacts_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(post_indptr, post_docs, post_tf, idf, doc_norm,
                                                                    k1p1, V, nnz, val);
  return (int)cudaGetLastError();
}

constexpr int kBmUnroll = 4;      // postings per thread and iteration (memory-level parallelism)

// dynamic shared memory: double acc[kBmChunk]; long long cur[kBmMaxTerms], pend[kBmMaxTerms]; int nxt[kBmMaxTerms]
constexpr size_t kBmSmem = (size_t)kBmChunk * 8 + (size_t)kBmMaxTerms * (8 + 8 + 4);

__global__ void __launch_bounds__(kBmThreads) bm25_topk_kernel(const long long* __restrict__ post_indptr,
                                                               const int* __restrict__ post_docs,
                                                               const double* __restrict__ post_val,
                                                               const int* __restrict__ head_slot,
                                                               const double* __restrict__ head_rows, long long ld_head,
                                                               const long long* __restrict__ q_indptr,
                                                               const int* __restrict__ q_terms, long long N, int k,
                                                               int C, int S, u64* cand, int* counts,
                                                               double* dense_out, long long ld_out) {
  extern __shared__ __align__(16) unsigned char bm_smem[];
  double* acc = reinterpret_cast<double*>(bm_smem);
  long long* cur = reinterpret_cast<long long*>(acc + kBmChunk);
  long long* pend = cur + kBmMaxTerms;
  int* nxt = reinterpret_cast<int*>(pend + kBmMaxTerms);
  __shared__ BlockStream s_st;

  const int tid = threadIdx.x, split = blockIdx.x;
  const long long row = blockIdx.y;
  const long long n_chunks = (N + kBmChunk - 1) / kBmChunk;
  const long long per = (n_chunks + S - 1) / S;
  const long long d0 = (long long)split * per * kBmChunk;
  long long d1 = d0 + per * kBmChunk;
  if (d1 > N) d1 = N;
  const long long tb = q_indptr[row];
  const int T = (int)(q_indptr[row + 1] - tb);
  u64* buf = cand ? cand + ((long long)row * S + split) * C : nullptr;

  // per-term cursor = first posting with doc >= d0 (one binary search per block and term)
  for (int t = tid; t < T; t += kBmThreads) {
    const int term = q_terms[tb + t];
    const int slot = head_slot ? __ldg(head_slot + term) : -1;
    if (slot >= 0) {  // head term: a dense float64 row instead of the list (a passage used as query is full of them)
      cur[t] = 0; pend[t] = 0; nxt[t] = -(slot + 1);
      continue;
    }
    long long lo = post_indptr[term];
    const long long end = post_indptr[term + 1];
    long long hi = end;
    while (lo < hi) { const long long mid = (lo + hi) >> 1; if ((long long)post_docs[mid] < d0) lo = mid + 1; else hi = mid; }
    cur[t] = lo;
    pend[t] = end;
    nxt[t] = lo < end ? post_docs[lo] : 0x7fffffff;
  }
  if (tid == 0) s_st.init();
  __syncthreads();

  for (long long c0 = d0; c0 < d1; c0 += kBmChunk) {
    const long long c1 = c0 + kBmChunk < d1 ? c0 + kBmChunk : d1;
    const int len = (int)(c1 - c0);
    for (int j = tid; j < kBmChunk; j += kBmThreads) acc[j] = 0.0;
    __syncthreads();
    for (int t = 0; t < T; ++t) {
      const int nx = nxt[t];
      if ((long long)nx >= c1) continue;  // uniform: shared-memory value
      if (nx < 0) {   // head term: coalesced adds of its dense row (x + 0.0 == x where the doc lacks the term)
        const double* r = head_rows + (long long)(-nx - 1) * ld_head + c0;
        for (int j = tid; j < len; j += kBmThreads) acc[j] += __ldg(r + j);
        __syncthreads();
        continue;
      }
      long long e = cur[t];
      const long long end = pend[t];
      bool more = true;
      {  // first 512 postings on their own: most terms have fewer than that in a chunk
        const long long i = e + tid;
        const int doc = i < end ? __ldg(post_docs + i) : 0x7fffffff;
        const bool in = (long long)doc < c1;  // doc-sorted: the in-chunk postings are a prefix
        if (in) acc[doc - (int)c0] += __ldg(post_val + i);
        const int n_in = __syncthreads_count(in);
        if (n_in < kBmThreads) {
          if (tid == n_in) { cur[t] = e + n_in; nxt[t] = doc; }  // first posting beyond the chunk
          more = false;
        }
        e += kBmThreads;
      }
      if (more) {
        // long list: kBmUnroll x 512 postings per iteration, double buffered -- the loads of the
        // next batch are issued (speculatively: harmless beyond the chunk, guarded by `end`) before
        // the current batch is applied, so their latency overlaps the accumulate + barrier steps
        int doc[kBmUnroll], ndoc[kBmUnroll];
        double v[kBmUnroll], nv[kBmUnroll];
#pragma unroll
        for (int u = 0; u < kBmUnroll; ++u) {
          const long long i = e + u * kBmThreads + tid;
          const bool live = i < end;
          doc[u] = live ? __ldg(post_docs + i) : 0x7fffffff;
          v[u] = live ? __ldg(post_val + i) : 0.0;
        }
        while (more) {  // a doc occurs at most once per term: no conflicts inside an iteration
          const long long en = e + (long long)kBmUnroll * kBmThreads;
#pragma unroll
          for (int u = 0; u < kBmUnroll; ++u) {
            const long long i = en + u * kBmThreads + tid;
            const bool live = i < end;
            ndoc[u] = live ? __ldg(post_docs + i) : 0x7fffffff;
            nv[u] = live ? __ldg(post_val + i) : 0.0;
          }
#pragma unroll
          for (int u = 0; u < kBmUnroll; ++u) {
            if (more) {  // uniform
              const bool in = (long long)doc[u] < c1;
              if (in) acc[doc[u] - (int)c0] += v[u];
              const int n_in = __syncthreads_count(in);
              if (n_in < kBmThreads) {
                if (tid == n_in) { cur[t] = e + u * kBmThreads + n_in; nxt[t] = doc[u]; }  // first posting beyond
                more = false;
              }
            }
          }
#pragma unroll
          for (int u = 0; u < kBmUnroll; ++u) { doc[u] = ndoc[u]; v[u] = nv[u]; }
          e = en;
        }
      }
    }
    __syncthreads();
    if (dense_out) {
      double* o = dense_out + row * ld_out + c0;
      for (int j = tid; j < len; j += kBmThreads) o[j] = acc[j];
    } else {
      for (int base = 0; base < len; base += kBmSlack) {
#pragma unroll
        for (int u = 0; u < kBmSlack / kBmThreads; ++u) {
          const int j = base + u * kBmThreads + tid;
          if (j < len) s_st.append(buf, (float)acc[j], (u32)(c0 + j), s_st.tau_f, s_st.tau_key);
        }
        __syncthreads();
        if (s_st.cnt > C - kBmSlack) {  // uniform: read after the barrier
          if (tid < 32) s_st.apply(warp_prune_stream<false, 0>(buf, s_st.cnt, k, 0, 0, smem_addr(s_st.hist), 0u));
        }
        __syncthreads();
      }
    }
    __syncthreads();
  }
  if (counts && tid == 0) counts[(long long)row * S + split] = s_st.cnt;
}

// =======================================================================================
// BM25, warp-private variant (queries of <= kBmwMaxTerms distinct terms -- every realistic query).
// The block-wide kernel above pays one block barrier per 256 postings.  Here every WARP is an
// independent worker: it owns a contiguous doc range (1/8 of the block's split), walks it in
// mini-chunks of 512 docs whose float64 accumulators are private to the warp (4 KB of shared memory),
// keeps its own per-term cursors, streams 32 postings per step (a ring of 4 x 32 in flight once a term
// turns out to be dense in the mini-chunk), and ranks into its own candidate buffer -- no block barrier anywhere, only warp votes.  Terms are
// still applied in q_terms order and a doc has at most one posting per term, so every float64 sum is
// bit-identical to the block-wide kernel's and to the reference's.
// =======================================================================================
__global__ void __launch_bounds__(kBmwWarps * 32, kBmwBlocksPerSm) bm25_topk_warp_kernel(
    const long long* __restrict__ post_indptr, const int* __restrict__ post_docs, const double* __restrict__ post_val,
    const int* __restrict__ head_slot, const double* __restrict__ head_rows, long long ld_head,
    const long long* __restrict__ q_indptr, const int* __restrict__ q_terms, long long N, int k, int C, int S,
    u64* cand, int* counts, u32* row_tau, double* dense_out, long long ld_out) {
  __shared__ __align__(16) double s_acc[kBmwWarps][kBmwMini];
  __shared__ long long s_cur[kBmwWarps][kBmwMaxTerms];
  __shared__ long long s_end[kBmwWarps][kBmwMaxTerms];
  __shared__ int s_nxt[kBmwWarps][kBmwMaxTerms];   // head terms: -(slot + 1)
  __shared__ u32 s_hist[kBmwWarps][256];
  __shared__ u32 s_tau_blk;  // ord32 of the best lower bound of the query's k-th best any of the block's streams knows
  __shared__ u32 s_jth[kBmwWarps];  // per stream: ord32 of a score with >= ceil(k / kBmwSketchM) of its docs at or above it
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const long long row = blockIdx.y;
  if (threadIdx.x == 0) s_tau_blk = 0u;
  if (threadIdx.x < kBmwWarps) s_jth[threadIdx.x] = 0u;
  __syncthreads();  // the only block barrier: from here on every warp runs on its own
  const int stream = blockIdx.x * kBmwWarps + warp, n_streams = S * kBmwWarps;
  const long long n_mini = (N + kBmwMini - 1) / kBmwMini;
  const long long per = (n_mini + n_streams - 1) / n_streams;
  const long long d0 = (long long)stream * per * kBmwMini;
  long long d1 = d0 + per * kBmwMini;
  if (d1 > N) d1 = N;
  const long long tb = q_indptr[row];
  const int T = (int)(q_indptr[row + 1] - tb);
  double* acc = s_acc[warp];
  long long* cur = s_cur[warp];
  long long* pend = s_end[warp];
  int* nxt = s_nxt[warp];
  u64* buf = cand ? cand + ((long long)row * n_streams + stream) * C : nullptr;
  if (lane < T && d0 < d1) {
    const int term = q_terms[tb + lane];
    const int slot = head_slot ? __ldg(head_slot + term) : -1;
    if (slot >= 0) {
      // head term: its values are read from a dense row (no cursor, no doc ids)
      cur[lane] = 0; pend[lane] = 0; nxt[lane] = -(slot + 1);
    } else {  // cursor of term `lane`: first posting with doc >= d0
      long long lo = post_indptr[term];
      const long long end = post_indptr[term + 1];
      long long hi = end;
      while (lo < hi) { const long long mid = (lo + hi) >> 1; if ((long long)post_docs[mid] < d0) lo = mid + 1; else hi = mid; }
      cur[lane] = lo;
      pend[lane] = end;
      nxt[lane] = lo < end ? post_docs[lo] : 0x7fffffff;
    }
  }
  __syncwarp();
  int cnt = 0;             // warp-uniform
  float tau_f = -INFINITY;
  u64 tau_key = 0ull;
  bool pruned = false;
  for (long long c0 = d0; c0 < d1; c0 += kBmwMini) {
    const long long c1 = c0 + kBmwMini < d1 ? c0 + kBmwMini : d1;
    const int len = (int)(c1 - c0);
#pragma unroll
    for (int j = 0; j < kBmwMini / 32; ++j) acc[j * 32 + lane] = 0.0;
    __syncwarp();
    for (int t = 0; t < T; ++t) {
      const int nx = nxt[t];
      if ((long long)nx >= c1) continue;  // warp-uniform: shared-memory value
      if (nx < 0) {
        // head term: 512 consecutive float64 values of its dense row (zero where the doc lacks the term:
        // x + 0.0 == x bit for bit, scores being sums of positive values from +0.0) -- independent,
        // fully coalesced 16-byte loads, nothing to search and nothing to vote on
        const double2* r = reinterpret_cast<const double2*>(head_rows + (long long)(-nx - 1) * ld_head + c0);
        double2* a2 = reinterpret_cast<double2*>(acc);
        double2 x[kBmwMini / 64];   // the whole 4 KB segment in flight at once (two half-segment trips: 28.2 vs 27.5 ms)
#pragma unroll
        for (int j = 0; j < kBmwMini / 64; ++j) x[j] = __ldg(r + j * 32 + lane);
#pragma unroll
        for (int j = 0; j < kBmwMini / 64; ++j) {
          double2 a = a2[j * 32 + lane];
          a.x += x[j].x; a.y += x[j].y;
          a2[j * 32 + lane] = a;
        }
        __syncwarp();
        continue;
      }
      long long e = cur[t];
      const long long end = pend[t];
      bool more = true;
      {  // first 32 postings on their own: most (term, mini-chunk) visits end inside them
        const int doc = e + lane < end ? __ldg(post_docs + e + lane) : 0x7fffffff;
        const double v = e + lane < end ? __ldg(post_val + e + lane) : 0.0;
        const bool in = (long long)doc < c1;  // doc-sorted: the in-range postings are a prefix
        if (in) acc[doc - (int)c0] += v;
        const int n_in = __popc(__ballot_sync(0xffffffffu, in));
        if (n_in < 32) {
          const int first_out = __shfl_sync(0xffffffffu, doc, n_in);
          if (lane == 0) { cur[t] = e + n_in; nxt[t] = first_out; }
          more = false;
        }
        e += 32;
      }
      if (more) {
        // dense term: a ring of kBmwDepth x 32 postings in flight per warp; a slot is refilled as soon
        // as it has been applied (speculative beyond the range: harmless, guarded by `end`)
        int doc[kBmwDepth];
        double v[kBmwDepth];
#pragma unroll
        for (int u = 0; u < kBmwDepth; ++u) {
          const long long i = e + u * 32 + lane;
          doc[u] = i < end ? __ldg(post_docs + i) : 0x7fffffff;
          v[u] = i < end ? __ldg(post_val + i) : 0.0;
        }
        while (more) {
#pragma unroll
          for (int u = 0; u < kBmwDepth; ++u) {
            if (more) {  // warp-uniform
              const bool in = (long long)doc[u] < c1;
              if (in) acc[doc[u] - (int)c0] += v[u];
              const int n_in = __popc(__ballot_sync(0xffffffffu, in));
              if (n_in < 32) {
                const int first_out = __shfl_sync(0xffffffffu, doc[u], n_in);
                if (lane == 0) { cur[t] = e + u * 32 + n_in; nxt[t] = first_out; }
                more = false;
              } else {
                const long long i = e + (u + kBmwDepth) * 32 + lane;
                doc[u] = i < end ? __ldg(post_docs + i) : 0x7fffffff;
                v[u] = i < end ? __ldg(post_val + i) : 0.0;
              }
            }
          }
          e += kBmwDepth * 32;
        }
      }
      __syncwarp();
    }
    __syncwarp();
    if (dense_out) {
      double* o = dense_out + row * ld_out + c0;
      for (int j = lane; j < len; j += 32) o[j] = acc[j];
    } else {
      // A stream that has pruned holds >= k docs at or above its threshold, so that threshold bounds the
      // QUERY's k-th best from below: the block's streams share the best one (fewer candidates, fewer
      // prunes).  Scores equal to a foreign bound are kept (>=); the own exact pivot stays a strict key bound.
      float tau_eff = tau_f;
      u64 key_eff = tau_key;
      {
        u32 tb;
        asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(tb) : "r"(smem_addr(&s_tau_blk)) : "memory");
        if (tb > ord32(tau_f)) { tau_eff = unord32(tb); key_eff = 0ull; }
      }
      // one compare per doc, one warp-wide OR: which of the 16 rows of 32 docs hold a candidate at all?
      // (once the threshold has matured: none, or one or two)
      unsigned bits = 0u;
#pragma unroll
      for (int j = 0; j < kBmwMini / 32; ++j) bits |= ((float)acc[j * 32 + lane] >= tau_eff ? 1u : 0u) << j;
      unsigned rows = __reduce_or_sync(0xffffffffu, bits);
      while (rows) {
        const int j = __ffs(rows) - 1;
        rows &= rows - 1u;
        const int idx = j * 32 + lane;
        bool pass = false;
        u64 key = 0ull;
        if (((bits >> j) & 1u) && idx < len) {   // docs beyond N score 0: never candidates
          key = make_key((float)acc[idx], (u32)(c0 + idx));
          pass = key > key_eff;
        }
        const unsigned m = __ballot_sync(0xffffffffu, pass);
        if (pass) buf[cnt + __popc(m & ((1u << lane) - 1u))] = key;
        cnt += __popc(m);
      }
      __syncwarp();
      if (cnt > C - kBmwMini) {  // C >= 2k + kBmwMini: room for the next mini-chunk after a prune
        // one histogram pass over the keys, and a second one over a crowded boundary bucket; tie-heavy or
        // still crowded buffers fall back to the exact radix select
        const PruneResult r = warp_prune_stream<false, 2>(buf, cnt, k, (k + kBmwSketchM - 1) / kBmwSketchM,
                                                          (k + C - kBmwMini) / 2, smem_addr(s_hist[warp]), 0u);
        cnt = r.kept; tau_f = r.tau_f; tau_key = r.tau_key;
        if (r.hist) {
          // sketch bound: this stream has >= ceil(k/M) docs at or above j_ord; the M-th largest of the block's
          // published values therefore has >= k docs of the query at or above it
          if (lane == 0) atomicMax(&s_jth[warp], r.j_ord);
          __syncwarp();
          u32 v = 0u;
          if (lane < kBmwWarps) asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(smem_addr(&s_jth[lane])) : "memory");
          const u32 bound = warp_mth_largest(v, kBmwSketchM);
          if (bound != 0u && lane == 0) atomicMax(&s_tau_blk, bound);
        }
        pruned = true;
        if (lane == 0) atomicMax(&s_tau_blk, ord32(tau_f));
      }
    }
    __syncwarp();
  }
  if (counts && lane == 0) {
    counts[(long long)row * n_streams + stream] = cnt;
    // this stream holds >= k docs scoring >= tau_f once it has pruned: a lower bound of the row's k-th best
    if (row_tau && pruned) atomicMax(row_tau + row, ord32(tau_f));
  }
  // A tighter row bound for finalize's prefilter from the block's 8 streams together: every stream
  // publishes its j-th best score (j = ceil(k / 5)); the 5th largest of those has >= 5 j >= k docs at or
  // above it.  With it the entries finalize has to look at (~3 k instead of ~8 k for k = 1001) fit its
  // shared-memory list.
  if (row_tau) {   // top-k mode (uniform)
    const int j = (k + kBmwSketchM - 1) / kBmwSketchM;
    u32 jv = 0u;
    if (cnt >= j && j >= 1) {
      __syncwarp();
      jv = (u32)(warp_select_kth(GlobalKeys{buf}, cnt, j, smem_addr(s_hist[warp])) >> 32);
    }
    __syncthreads();   // (every stream is past its last in-loop use of s_jth)
    if (lane == 0) s_jth[warp] = jv;
    __syncthreads();
    if (warp == 0) {
      const u32 bound = warp_mth_largest(lane < kBmwWarps ? s_jth[lane] : 0u, kBmwSketchM);
      if (bound != 0u && lane == 0) atomicMax(row_tau + row, bound);
    }
  }
}

int launch_bm25(const Bm25Params& p, cudaStream_t st) {
  if (p.Bq <= 0 || p.N <= 0) return 0;
  dim3 grid((unsigned)p.S, (unsigned)p.Bq);
  if (p.warp) {
    bm25_topk_warp_kernel<<<grid, kBmwWarps * 32, 0, st>>>(p.post_indptr, p.post_docs, p.post_val, p.head_slot,
                                                          p.head_rows, p.ld_head, p.q_indptr, p.q_terms, p.N, p.k, p.C,
                                                          p.S, p.cand, p.counts, p.row_tau, p.dense_out, p.ld_out);
  } else {
    cudaError_t e = cudaFuncSetAttribute(bm25_topk_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kBmSmem);
    if (e != cudaSuccess) return (int)e;
    bm25_topk_kernel<<<grid, kBmThreads, kBmSmem, st>>>(p.post_indptr, p.post_docs, p.post_val, p.head_slot,
                                                       p.head_rows, p.ld_head, p.q_indptr, p.q_terms, p.N, p.k, p.C,
                                                       p.S, p.cand, p.counts, p.dense_out, p.ld_out);
  }
  return (int)cudaGetLastError();
}

// Dense float64 rows of the head terms (built once per fit / cache): rows[slot, doc] = post_val of
// (head_terms[slot], doc), 0 elsewhere.  One block per head term.
__global__ void __launch_bounds__(256) bm25_head_rows_kernel(const long long* __restrict__ post_indptr,
                                                             const int* __restrict__ post_docs,
                                                             const double* __restrict__ post_val,
                                                             const int* __restrict__ head_terms, long long n_terms,
                                                             long long ld_head, double* __restrict__ rows) {
  const int term = head_terms[blockIdx.x];
  if (term < 0 || (long long)term >= n_terms) return;  // never trust a caller-supplied id: the row stays zero
  double* r = rows + (long long)blockIdx.x * ld_head;
  const long long e0 = post_indptr[term], e1 = post_indptr[term + 1];
  for (long long e = e0 + threadIdx.x; e < e1; e += 256) r[post_docs[e]] = post_val[e];
}

__global__ void bm25_head_slots_kernel(const int* __restrict__ head_terms, int n_head, long long n_terms,
                                       int* __restrict__ head_slot) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n_head) return;
  const int term = head_terms[i];
  if (term >= 0 && (long long)term < n_terms) head_slot[term] = i;
}

int launch_bm25_head_slots(const int* head_terms, int n_head, long long n_terms, int* head_slot, cudaStream_t st) {
  if (n_head <= 0) return 0;
  bm25_head_slots_kernel<<<(n_head + 127) / 128, 128, 0, st>>>(head_terms, n_head, n_terms, head_slot);
  return (int)cudaGetLastError();
}

int launch_bm25_head_rows(const long long* post_indptr, const int* post_docs, const double* post_val,
                          const int* head_terms, int n_head, long long n_terms, long long ld_head, double* rows,
                          cudaStream_t st) {
  if (n_head <= 0) return 0;
  cudaError_t e = cudaMemsetAsync(rows, 0, (size_t)n_head * (size_t)ld_head * sizeof(double), st);
  if (e != cudaSuccess) return (int)e;
  bm25_head_rows_kernel<<<(unsigned)n_head, 256, 0, st>>>(post_indptr, post_docs, post_val, head_terms, n_terms, ld_head,
                                                          rows);
  return (int)cudaGetLastError();
}

// =======================================================================================
// Top-k of an already materialised dense float32 score matrix (+ sparse priors): what the
// reference's `_assign_topk` receives when `BertBPR.transform` hands it the dense host matrix
// (src/rime_lite/util/__init__.py:135-141 after score_array.py:226-227 [+ :173-174]).
//   select_dense_kernel  : block = (column split, row); streams the row, threshold filter,
//                          candidate buffer, exact radix prune -- the protocol of the fused kernels.
//                          Rows with priors keep k + nnz(row) candidates (include mode) ...
//   entry_records_kernel : ... and every prior entry gets its exact float64 value (ScoreMatrix source)
//                          double(score) + prior (or the prior itself in SET mode), merged and the
//                          plain candidates of those columns dropped by finalize_kernel.
// =======================================================================================
constexpr int kDenseThreads = 256;

__global__ void __launch_bounds__(kDenseThreads) select_dense_kernel(const float* __restrict__ scores, long long ld,
                                                                     long long N, int k, int k_keep,
                                                                     const long long* __restrict__ mask_indptr, int C,
                                                                     int S, u64* cand, int* counts) {
  __shared__ BlockStream s_st;
  const int tid = threadIdx.x, split = blockIdx.x;
  const long long row = blockIdx.y;
  // buffers are sized for k_keep = k + mask_max_row_nnz: never trust the CSR beyond that
  const long long k_csr = (long long)k + (mask_indptr ? (mask_indptr[row + 1] - mask_indptr[row]) : 0);
  const int k_row = k_csr < (long long)k_keep ? (int)k_csr : k_keep;
  long long per = (N + S - 1) / S;
  per = (per + kDenseSlack - 1) / kDenseSlack * kDenseSlack;
  const long long i0 = (long long)split * per;
  long long i1 = i0 + per;
  if (i1 > N) i1 = N;
  u64* buf = cand + ((long long)row * S + split) * C;
  const float* r = scores + row * ld;
  if (tid == 0) s_st.init();
  __syncthreads();
  // kDenseSlack columns per iteration: 16 per thread as four 16-byte loads in flight (scalar loads at a
  // ragged end or an unaligned row), one max + ONE block vote, and only an iteration that holds a
  // candidate pays for the appends, the second barrier and the prune check.
  const bool vec = ((uintptr_t)r & 15) == 0;
  constexpr int kPer = kDenseSlack / kDenseThreads;   // 16
  for (long long base = i0; base < i1; base += kDenseSlack) {
    float v[kPer];
    if (vec && base + kDenseSlack <= i1) {
#pragma unroll
      for (int q = 0; q < kPer / 4; ++q) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(r + base) + q * kDenseThreads + tid);
        v[4 * q] = x.x; v[4 * q + 1] = x.y; v[4 * q + 2] = x.z; v[4 * q + 3] = x.w;
      }
    } else {
#pragma unroll
      for (int j = 0; j < kPer; ++j) {
        const long long i = base + ((j >> 2) * kDenseThreads + tid) * 4 + (j & 3);
        v[j] = i < i1 ? __ldg(r + i) : __uint_as_float(0x7fc00000u);   // NaN: fails every >= test
      }
    }
    float mx = v[0];
#pragma unroll
    for (int j = 1; j < kPer; ++j) mx = fmaxf(mx, v[j]);   // NaN scores never rank (torch would put them first; the reference has none)
    const float tau_f = s_st.tau_f;
    const u64 tau_key = s_st.tau_key;
    if (!__syncthreads_or(mx >= tau_f)) continue;
#pragma unroll
    for (int j = 0; j < kPer; ++j) {
      const long long i = base + ((j >> 2) * kDenseThreads + tid) * 4 + (j & 3);
      s_st.append(buf, v[j], (u32)i, tau_f, tau_key);
    }
    __syncthreads();
    if (s_st.cnt > C - kDenseSlack) {  // uniform: read after the barrier; C >= 2 * k_row + slack
      // one histogram pass first; the exact radix select only for tie-heavy or crowded buffers
      if (tid < 32)
        s_st.apply(warp_prune_stream<false, 1>(buf, s_st.cnt, k_row, k_row, (k_row + C - kDenseSlack) / 2,
                                               smem_addr(s_st.hist), 0u));
    }
    __syncthreads();
  }
  if (tid == 0) counts[(long long)row * S + split] = s_st.cnt;
}

int launch_select_dense(const float* scores, long long ld, long long B, long long N, int k, int k_keep,
                        const long long* mask_indptr, int C, int S, u64* cand, int* counts, cudaStream_t st) {
  if (B <= 0) return 0;
  dim3 grid((unsigned)S, (unsigned)B);
  select_dense_kernel<<<grid, kDenseThreads, 0, st>>>(scores, ld, N, k, k_keep, mask_indptr, C, S, cand, counts);
  return (int)cudaGetLastError();
}

}  // namespace ccr
