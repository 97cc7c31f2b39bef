// Whole-matrix argsort (rime_lite `_argsort`, src/rime_lite/util/__init__.py:158-184) and the MRR
// first-hit scan (scripts/al_0_rank.py:130-133) -- HBM-bound integer work, CUDA cores only.
//
//   argsort : keys = ~ord64(double(score) [+ prior | := value]) per matrix element (~ord32(score) when no prior
//             is given: the same order in half the bytes and passes), payload = flat
//             index; LSD radix sort, 8 passes of 8 bits, each pass = per-tile digit histogram ->
//             exclusive scan over (digit, tile) -> stable scatter (skipped on the device when every key
//             carries the same digit).  Ascending ~ord64 == descending
//             score; stability keeps equal scores in flat-index order (the reference adds unseeded
//             jitter instead).  Algorithmic bytes: 8 passes x 2 x 12 B per element.
//   first-hit rank : one warp per query row scans its ranked ids against the row's sorted list of
//             relevant ids (binary search per id), first lane that hits wins.
#include "ccr_params.cuh"

namespace ccr {

constexpr int kSortThreads = 256;
constexpr int kSortPerThread = 16;
constexpr int kSortTile = kSortThreads * kSortPerThread;  // keys per block and pass

// Bit p set = pass p (digit = key bits [8p, 8p+8)) can change the order: some key's digit is not the one its
// top bit alone implies (top bit set: 0x00, clear: 0xFF -- the low bytes of ~ord64(double(float32))).  A pass
// without such a key is a no-op for the final order: two keys that agree in all the higher digits (which
// include the top bit) agree in this one as well.
__device__ __forceinline__ u32 sort_needed_passes(u64 key) {
  const u64 implied = (key >> 63) ? 0ull : ~0ull;
  const u64 diff = key ^ implied;
  u32 m = 0;
#pragma unroll
  for (int p = 0; p < 8; ++p) m |= (((diff >> (8 * p)) & 255ull) != 0ull ? 1u : 0u) << p;
  return m | 0x80u;   // the top pass always runs
}

template <typename K>
__global__ void __launch_bounds__(256) sort_build_keys_kernel(const float* __restrict__ scores, long long B, long long N,
                                                              long long ld, K* __restrict__ keys,
                                                              u32* __restrict__ payload, int* __restrict__ state) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  u32 need = 0;
  if (i < B * N) {
    const long long r = i / N, c = i - r * N;
    const float sc = scores[r * ld + c];
    payload[i] = (u32)i;
    if (sizeof(K) == 4) {   // no float64 prior anywhere: the float32 order is the order
      keys[i] = (K)~ord32(sc);
      need = 0xFu;
    } else {
      const u64 key = ~ord64((double)sc);
      keys[i] = (K)key;
      need = sort_needed_passes(key);
    }
  }
  need = __reduce_or_sync(0xffffffffu, need);
  if ((threadIdx.x & 31) == 0 && (need & ~(u32)state[3])) atomicOr(state + 3, (int)need);
}

// mask entries overwrite their element's key with ~ord64(mask_value)
__global__ void __launch_bounds__(256) sort_override_keys_kernel(const float* __restrict__ scores, long long B,
                                                                 long long N, long long ld,
                                                                 const long long* __restrict__ indptr,
                                                                 const int* __restrict__ cols,
                                                                 const double* __restrict__ vals, int mode,
                                                                 u64* __restrict__ keys, int* __restrict__ state) {
  const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= indptr[B]) return;
  const long long row = csr_row_of(indptr, B, e);
  const int col = cols[e];
  if (col < 0 || (long long)col >= N) return;
  const u64 key = ~ord64(mask_value(mode, scores[row * ld + col], vals[e]));
  keys[row * N + col] = key;
  const u32 need = sort_needed_passes(key);
  if (need & ~(u32)state[3]) atomicOr(state + 3, (int)need);
}

// Pass state on the device (no host round trip): state[0] = which buffer holds the current order (0: a,
// 1: b), state[1] = skip flag of the pass in flight, state[3] = mask of the passes that can change the
// order (sort_needed_passes; 3 of the 8 passes are no-ops when no float64 prior is involved).
template <typename K> struct SortBufs {
  K* k[2];
  u32* p[2];
};

// per-tile digit counts, stored digit-major: hist[d * n_tiles + tile]
template <typename K>
__global__ void __launch_bounds__(kSortThreads) sort_hist_kernel(SortBufs<K> bufs, const int* __restrict__ state,
                                                                 long long n, int shift, u32* __restrict__ hist,
                                                                 int n_tiles) {
  if (!((state[3] >> (shift >> 3)) & 1)) return;   // pass not needed: nobody reads its counts
  __shared__ u32 s_cnt[256];
  const int tid = threadIdx.x;
  const K* __restrict__ keys = bufs.k[state[0]];
  s_cnt[tid] = 0;
  __syncthreads();
  const long long base = (long long)blockIdx.x * kSortTile;
#pragma unroll
  for (int j = 0; j < kSortPerThread; ++j) {
    const long long i = base + j * kSortThreads + tid;
    if (i < n) atomicAdd(&s_cnt[(u32)(keys[i] >> shift) & 255u], 1u);
  }
  __syncthreads();
  hist[(long long)tid * n_tiles + blockIdx.x] = s_cnt[tid];
}

// exclusive scan of one digit's row of tile counts in place (block d = digit d), row total -> totals[d]
__global__ void __launch_bounds__(1024) sort_scan_rows_kernel(u32* __restrict__ hist, int n_tiles,
                                                              u32* __restrict__ totals) {
  __shared__ u32 s_warp[32];
  __shared__ u32 s_carry;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  u32* row = hist + (long long)blockIdx.x * n_tiles;
  if (tid == 0) s_carry = 0;
  __syncthreads();
  for (int i0 = 0; i0 < n_tiles; i0 += 1024) {
    const int i = i0 + tid;
    const u32 v = i < n_tiles ? row[i] : 0u;
    u32 incl = v;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += t; }
    if (lane == 31) s_warp[warp] = incl;
    __syncthreads();
    u32 base = s_carry;
    for (int w = 0; w < warp; ++w) base += s_warp[w];
    if (i < n_tiles) row[i] = base + incl - v;
    __syncthreads();
    if (tid == 1023) s_carry = base + incl;
    __syncthreads();
  }
  if (tid == 0) totals[blockIdx.x] = s_carry;
}

// exclusive scan of the 256 digit totals -> dbase; sets the skip flag of a pass that is not needed
__global__ void __launch_bounds__(256) sort_scan_digits_kernel(const u32* __restrict__ totals, int pass,
                                                               u32* __restrict__ dbase, int* __restrict__ state) {
  __shared__ u32 s_tot[256];
  const int tid = threadIdx.x;
  s_tot[tid] = totals[tid];
  __syncthreads();
  u32 before = 0;
  for (int d = 0; d < tid; ++d) before += s_tot[d];
  dbase[tid] = before;
  if (tid == 0) state[1] = ((state[3] >> pass) & 1) ? 0 : 1;
}

__global__ void sort_flip_kernel(int* __restrict__ state) {
  if (state[1] == 0) state[0] ^= 1;
}

// Stable scatter.  Warp w owns the 512 consecutive keys [512 w, 512 w + 512) of the tile and walks them in
// 16 rounds of 32 (lane = consecutive key: coalesced loads).  Stable rank of a key inside the tile = keys
// of the same digit in earlier warps + earlier in this warp's chunk; the last term needs no block
// barrier: `match.any` groups the lanes of a round by digit and a per-warp running digit count in shared
// memory carries over the rounds.  The tile is then REORDERED IN SHARED MEMORY (digit-major, stable) and
// written out position by position, so that consecutive threads write consecutive addresses inside every
// digit's run (a random digit scatters 32 lanes to 32 runs otherwise: 2x DRAM write amplification and
// 1.98 ms per pass for 67 M keys instead of the 0.8 ms measured with the reorder).
template <typename K> constexpr size_t sort_scatter_smem() { return (size_t)kSortTile * (sizeof(K) + sizeof(u32)); }

template <typename K>
__global__ void __launch_bounds__(kSortThreads) sort_scatter_kernel(SortBufs<K> bufs, const int* __restrict__ state,
                                                                    long long n, int shift,
                                                                    const u32* __restrict__ hist,
                                                                    const u32* __restrict__ dbase, int n_tiles) {
  if (state[1]) return;   // the pass cannot change the order (see sort_scan_digits_kernel)
  const int src = state[0];
  const K* __restrict__ keys_in = bufs.k[src];
  const u32* __restrict__ pay_in = bufs.p[src];
  K* __restrict__ keys_out = bufs.k[src ^ 1];
  u32* __restrict__ pay_out = bufs.p[src ^ 1];
  extern __shared__ __align__(16) unsigned char sort_smem[];
  K* s_key = reinterpret_cast<K*>(sort_smem);                     // [kSortTile] the tile, digit-major
  u32* s_pay = reinterpret_cast<u32*>(s_key + kSortTile);         // [kSortTile]
  __shared__ u32 s_base[256];                      // global offset of this tile's first key of each digit
  __shared__ u32 s_toff[256];                      // tile-local offset of each digit's run
  __shared__ u32 s_wcnt[kSortThreads / 32][256];   // per-warp running digit counts, then exclusive warp bases
  __shared__ u32 s_wsum[kSortThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  s_base[tid] = dbase[tid] + hist[(long long)tid * n_tiles + blockIdx.x];
#pragma unroll
  for (int w = 0; w < kSortThreads / 32; ++w) s_wcnt[w][tid] = 0;
  __syncthreads();
  const long long tile0 = (long long)blockIdx.x * kSortTile;
  const long long base = tile0 + (long long)warp * (32 * kSortPerThread);
  K key[kSortPerThread];
  u32 pay[kSortPerThread], rank[kSortPerThread];
#pragma unroll
  for (int j = 0; j < kSortPerThread; ++j) {
    const long long i = base + j * 32 + lane;
    const bool live = i < n;
    key[j] = live ? keys_in[i] : (K)0;
    pay[j] = live ? pay_in[i] : 0u;
  }
#pragma unroll
  for (int j = 0; j < kSortPerThread; ++j) {
    const bool live = base + j * 32 + lane < n;
    const u32 d = (u32)(key[j] >> shift) & 255u;
    // lanes of this round with the same digit (dead lanes form their own group and count nothing)
    const unsigned peers = __match_any_sync(0xffffffffu, live ? d : 0xFFFFFFFFu);
    const u32 r = (u32)__popc(peers & ((1u << lane) - 1u));
    const u32 prev = s_wcnt[warp][d];
    __syncwarp();
    if (live && r == 0) s_wcnt[warp][d] = prev + (u32)__popc(peers);
    __syncwarp();
    rank[j] = prev + r;
  }
  __syncthreads();
  {  // thread d: exclusive prefix of digit d's counts over the warps; then of the digit totals over the digits
    u32 run = 0;
#pragma unroll
    for (int w = 0; w < kSortThreads / 32; ++w) { const u32 t = s_wcnt[w][tid]; s_wcnt[w][tid] = run; run += t; }
    u32 incl = run;
#pragma unroll
    for (int off = 1; off < 32; off <<= 1) { const u32 t = __shfl_up_sync(0xffffffffu, incl, off); if (lane >= off) incl += t; }
    if (lane == 31) s_wsum[warp] = incl;
    __syncthreads();
    u32 before = 0;
    for (int w = 0; w < warp; ++w) before += s_wsum[w];
    s_toff[tid] = before + incl - run;
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < kSortPerThread; ++j) {
    if (base + j * 32 + lane < n) {
      const u32 d = (u32)(key[j] >> shift) & 255u;
      const u32 loc = s_toff[d] + s_wcnt[warp][d] + rank[j];
      s_key[loc] = key[j];
      s_pay[loc] = pay[j];
    }
  }
  __syncthreads();
  const int tile_n = (int)((n - tile0 < (long long)kSortTile) ? (n - tile0) : (long long)kSortTile);
  for (int i = tid; i < tile_n; i += kSortThreads) {
    const K k2 = s_key[i];
    const u32 d = (u32)(k2 >> shift) & 255u;
    const u32 pos = s_base[d] + ((u32)i - s_toff[d]);
    keys_out[pos] = k2;
    pay_out[pos] = s_pay[i];
  }
}

__global__ void __launch_bounds__(256) sort_unravel_kernel(const u32* __restrict__ pay0, const u32* __restrict__ pay1,
                                                           const int* __restrict__ state, long long n,
                                                           long long N, long long* __restrict__ out_rows,
                                                           long long* __restrict__ out_cols) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const u32 flat = (state[0] ? pay1 : pay0)[i];   // n = B * N < 2^32 (checked by the caller), so N fits 32 bits too
  const u32 r = flat / (u32)N;
  out_rows[i] = (long long)r;
  out_cols[i] = (long long)(flat - r * (u32)N);
}

size_t argsort_workspace_bytes(long long n) {
  const long long tiles = (n + kSortTile - 1) / kSortTile;
  size_t off = 0;
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  off = up(off + (size_t)n * 8);   // keys a
  off = up(off + (size_t)n * 8);   // keys b
  off = up(off + (size_t)n * 4);   // payload a
  off = up(off + (size_t)n * 4);   // payload b
  off = up(off + (size_t)256 * (size_t)(tiles > 0 ? tiles : 1) * 4);   // per-tile digit counts
  off = up(off + (size_t)(256 + 256 + 4) * 4);                          // digit totals, digit bases, pass state
  return off;
}

template <typename K>
static int sort_passes(SortBufs<K> bufs, long long n, int tiles, u32* hist, u32* totals, u32* dbase, int* state,
                       cudaStream_t st) {
  {
    static bool attr_done[64];  // per function and device: dynamic + 10 KB of static shared memory exceed 48 KB
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) { cudaGetLastError(); dev = -1; }
    if (dev < 0 || !attr_done[dev]) {
      cudaError_t e = cudaFuncSetAttribute(sort_scatter_kernel<K>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           (int)sort_scatter_smem<K>());
      if (e != cudaSuccess) return (int)e;
      if (dev >= 0) attr_done[dev] = true;
    }
  }
  for (int pass = 0; pass < (int)sizeof(K); ++pass) {
    const int shift = pass * 8;
    sort_hist_kernel<K><<<tiles, kSortThreads, 0, st>>>(bufs, state, n, shift, hist, tiles);
    sort_scan_rows_kernel<<<256, 1024, 0, st>>>(hist, tiles, totals);
    sort_scan_digits_kernel<<<1, 256, 0, st>>>(totals, pass, dbase, state);
    sort_scatter_kernel<K><<<tiles, kSortThreads, sort_scatter_smem<K>(), st>>>(bufs, state, n, shift, hist, dbase, tiles);
    sort_flip_kernel<<<1, 1, 0, st>>>(state);
  }
  return (int)cudaGetLastError();
}

int launch_argsort(const float* scores, long long B, long long N, long long ld, const long long* indptr, const int* cols,
                   const double* vals, long long nnz, int mode, long long* out_rows, long long* out_cols, void* ws,
                   cudaStream_t st) {
  const long long n = B * N;
  if (n <= 0) return 0;
  const int tiles = (int)((n + kSortTile - 1) / kSortTile);
  auto up = [](size_t x) { return (x + 255) / 256 * 256; };
  unsigned char* w = (unsigned char*)ws;
  size_t off = 0;
  u64* ka = (u64*)(w + off); off = up(off + (size_t)n * 8);
  u64* kb = (u64*)(w + off); off = up(off + (size_t)n * 8);
  u32* pa = (u32*)(w + off); off = up(off + (size_t)n * 4);
  u32* pb = (u32*)(w + off); off = up(off + (size_t)n * 4);
  u32* hist = (u32*)(w + off); off = up(off + (size_t)256 * (size_t)tiles * 4);
  u32* totals = (u32*)(w + off);
  u32* dbase = totals + 256;
  int* state = (int*)(dbase + 256);
  const unsigned gb = (unsigned)((n + 255) / 256);
  if (cudaMemsetAsync(state, 0, 4 * sizeof(int), st) != cudaSuccess) return (int)cudaGetLastError();
  if (nnz > 0 && indptr) {   // float64 priors decide: 64-bit keys, 8 passes
    SortBufs<u64> bufs;
    bufs.k[0] = ka; bufs.k[1] = kb; bufs.p[0] = pa; bufs.p[1] = pb;
    sort_build_keys_kernel<u64><<<gb, 256, 0, st>>>(scores, B, N, ld, ka, pa, state);
    sort_override_keys_kernel<<<(unsigned)((nnz + 255) / 256), 256, 0, st>>>(scores, B, N, ld, indptr, cols, vals, mode, ka,
                                                                          state);
    const int rc = sort_passes<u64>(bufs, n, tiles, hist, totals, dbase, state, st);
    if (rc) return rc;
  } else {   // the float32 order is the order: 32-bit keys (in the first halves of the key buffers), 4 passes
    SortBufs<u32> bufs;
    bufs.k[0] = reinterpret_cast<u32*>(ka); bufs.k[1] = reinterpret_cast<u32*>(kb); bufs.p[0] = pa; bufs.p[1] = pb;
    sort_build_keys_kernel<u32><<<gb, 256, 0, st>>>(scores, B, N, ld, bufs.k[0], pa, state);
    const int rc = sort_passes<u32>(bufs, n, tiles, hist, totals, dbase, state, st);
    if (rc) return rc;
  }
  sort_unravel_kernel<<<gb, 256, 0, st>>>(pa, pb, state, n, N, out_rows, out_cols);
  return (int)cudaGetLastError();
}

// =======================================================================================
// MRR core: rank (1-based) of the first relevant id in each row's ranked list, 0 = none.
//   ids [B, k] int64 (ranked, best first; < 0 = padding), rel CSR: rel_indptr int64[B+1], rel_ids
//   int64 sorted ascending inside a row.
// =======================================================================================
__global__ void __launch_bounds__(256) first_hit_rank_kernel(const long long* __restrict__ ids, long long B, int k,
                                                             const long long* __restrict__ rel_indptr,
                                                             const long long* __restrict__ rel_ids,
                                                             int* __restrict__ out_rank) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= B) return;
  const long long beg = rel_indptr[row], end = rel_indptr[row + 1];
  int rank = 0;
  if (end > beg) {
    for (int j0 = 0; j0 < k && rank == 0; j0 += 32) {
      const int j = j0 + lane;
      bool hit = false;
      if (j < k) {
        const long long id = ids[row * k + j];
        long long lo = beg, hi = end;
        while (lo < hi) { const long long mid = (lo + hi) >> 1; const long long v = rel_ids[mid]; if (v == id) { hit = true; break; } if (v < id) lo = mid + 1; else hi = mid; }
      }
      const unsigned m = __ballot_sync(0xffffffffu, hit);
      if (m) rank = j0 + __ffs(m);
    }
  }
  if (lane == 0) out_rank[row] = rank;
}

int launch_first_hit_rank(const long long* ids, long long B, int k, const long long* rel_indptr, const long long* rel_ids,
                          int* out_rank, cudaStream_t st) {
  if (B <= 0) return 0;
  first_hit_rank_kernel<<<(unsigned)((B + 7) / 8), 256, 0, st>>>(ids, B, k, rel_indptr, rel_ids, out_rank);
  return (int)cudaGetLastError();
}

}  // namespace ccr
