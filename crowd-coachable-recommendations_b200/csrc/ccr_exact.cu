// Exact fp32 ranking (DESIGN.md section 6b): the stages around the unchanged scan kernels and the
// exact re-rank (entry_records_kernel with the ExactDot source + finalize_kernel, ccr_kernels.cu).
//   certify_kernel       : per row, does the k-th exact value beat every item the scan stage left out?
//   compact_kernel       : columns of a dense scan-score block at or above a per-row threshold, as a CSR
//   row_norm_max_kernel  : largest fp32 row norm of an appended batch (the V of the error bound)
//   dense_exact_kernel   : the exact value of every (query, item) pair of a [B, N] block
#include "ccr_params.cuh"

namespace ccr {

// One warp per row.  Certified when the scan stage returned every item (k_cand == n_items), fewer than
// k_cand unmasked items (every unmasked item), or when the k-th exact value L_k beats RU(t + E) strictly,
// t being the scan score of the k_cand-th candidate: no item left out can reach L_k, and no tie with it
// can displace a winner.  tau = RD(L_k - E) bounds the scan score of every item whose exact value is >= L_k.
__global__ void __launch_bounds__(256) certify_kernel(const float* __restrict__ q, long long ldq, int B, int D,
                                                      int f16, const double* __restrict__ v_max, int k, int k_cand,
                                                      long long n_items, const float* __restrict__ s1_scores,
                                                      const long long* __restrict__ s1_ids,
                                                      const long long* __restrict__ mask_indptr,
                                                      const int* __restrict__ mask_cols,
                                                      const double* __restrict__ out_scores64, int force_fallback,
                                                      int* __restrict__ uncert, double* __restrict__ tau,
                                                      int* __restrict__ count) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= B) return;
  double ss = 0.0;
  for (int d = lane; d < D; d += 32) { const double x = (double)q[row * ldq + d]; ss = fma(x, x, ss); }
#pragma unroll
  for (int off = 16; off; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
  const double err = exact_error_bound(__dsqrt_ru(ss), *v_max, D, f16);
  const long long m0 = mask_indptr ? mask_indptr[row] : 0, m1 = mask_indptr ? mask_indptr[row + 1] : 0;
  int unmasked = 0;
  for (int j = lane; j < k_cand; j += 32) {
    const long long id = s1_ids[row * k_cand + j];
    unmasked += (id >= 0 && !(mask_indptr && mask_contains(mask_cols, m0, m1, (int)id))) ? 1 : 0;
  }
#pragma unroll
  for (int off = 16; off; off >>= 1) unmasked += __shfl_xor_sync(0xffffffffu, unmasked, off);
  if (lane) return;
  const double lk = out_scores64[row * k + k - 1];
  bool ok = k_cand >= n_items || unmasked < k_cand;
  if (!ok) ok = lk > __dadd_ru((double)s1_scores[row * k_cand + k_cand - 1], err);
  if (force_fallback) ok = false;
  uncert[row] = ok ? 0 : 1;
  tau[row] = __dsub_rd(lk, err);
  if (!ok) atomicAdd(count, 1);
}

int launch_exact_certify(const float* q, long long ldq, int B, int D, int f16, const double* v_max, int k, int k_cand,
                         long long n_items, const float* s1_scores, const long long* s1_ids,
                         const long long* mask_indptr, const int* mask_cols, const double* out_scores64,
                         int force_fallback, int* uncert, double* tau, int* count, cudaStream_t st) {
  if (B <= 0) return 0;
  certify_kernel<<<(unsigned)((B + 7) / 8), 256, 0, st>>>(q, ldq, B, D, f16, v_max, k, k_cand, n_items, s1_scores,
                                                          s1_ids, mask_indptr, mask_cols, out_scores64,
                                                          force_fallback, uncert, tau, count);
  return (int)cudaGetLastError();
}

// One block per row.  kWrite = false: indptr[r + 1] = number of columns with double(score) >= tau[r];
// kWrite = true: their column ids, written from indptr[r] on (warp-aggregated, in no particular order).
template <bool kWrite>
__global__ void __launch_bounds__(256) compact_kernel(const float* __restrict__ scores, long long N, long long ld,
                                                      const double* __restrict__ tau, long long* __restrict__ indptr,
                                                      long long* __restrict__ ids) {
  __shared__ unsigned long long s_n;
  const int lane = threadIdx.x & 31;
  const long long r = blockIdx.x;
  const float* s = scores + r * ld;
  const double t = tau[r];
  if (threadIdx.x == 0) s_n = 0ull;
  __syncthreads();
  const long long base = kWrite ? indptr[r] : 0;
  unsigned long long mine = 0;
  for (long long j0 = 0; j0 < N; j0 += blockDim.x) {
    const long long j = j0 + threadIdx.x;
    const bool keep = j < N && (double)s[j] >= t;
    if (!kWrite) { mine += keep ? 1 : 0; continue; }
    const unsigned bal = __ballot_sync(0xffffffffu, keep);
    if (!bal) continue;
    unsigned long long wbase = 0;
    if (lane == 0) wbase = atomicAdd(&s_n, (unsigned long long)__popc(bal));
    wbase = __shfl_sync(0xffffffffu, wbase, 0);
    if (keep) ids[base + (long long)wbase + __popc(bal & ((1u << lane) - 1u))] = j;
  }
  if (!kWrite) {
    atomicAdd(&s_n, mine);
    __syncthreads();
    if (threadIdx.x == 0) indptr[r + 1] = (long long)s_n;
  }
}

// indptr[0] = 0, indptr[r + 1] += indptr[r]: a short serial scan (R is one chunk of fallback rows)
__global__ void indptr_scan_kernel(long long R, long long* indptr) {
  indptr[0] = 0;
  for (long long r = 0; r < R; ++r) indptr[r + 1] += indptr[r];
}

int launch_threshold_compact(const float* scores, long long R, long long N, long long ld, const double* tau,
                             long long* indptr, long long* ids, cudaStream_t st) {
  if (R <= 0) return 0;
  if (ids) {
    compact_kernel<true><<<(unsigned)R, 256, 0, st>>>(scores, N, ld, tau, indptr, ids);
    return (int)cudaGetLastError();
  }
  compact_kernel<false><<<(unsigned)R, 256, 0, st>>>(scores, N, ld, tau, indptr, nullptr);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return (int)e;
  indptr_scan_kernel<<<1, 1, 0, st>>>(R, indptr);
  return (int)cudaGetLastError();
}

// One warp per row: *v_max = max(*v_max, RU(||row||_2)), the norm summed in float64.  Non-negative
// doubles order like their bit patterns, so the maximum is an integer atomicMax.
__global__ void __launch_bounds__(256) row_norm_max_kernel(const float* __restrict__ rows, long long n, int D,
                                                           long long ld, double* v_max) {
  const int lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= n) return;
  double ss = 0.0;
  for (int d = lane; d < D; d += 32) { const double x = (double)rows[row * ld + d]; ss = fma(x, x, ss); }
#pragma unroll
  for (int off = 16; off; off >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, off);
  if (lane == 0)
    atomicMax(reinterpret_cast<unsigned long long*>(v_max),
              (unsigned long long)__double_as_longlong(__dsqrt_ru(ss) * (1.0 + 0x1p-40)));
}

int launch_row_norm_max(const float* rows, long long n, int D, long long ld, double* v_max, cudaStream_t st) {
  if (n <= 0) return 0;
  row_norm_max_kernel<<<(unsigned)((n + 7) / 8), 256, 0, st>>>(rows, n, D, ld, v_max);
  return (int)cudaGetLastError();
}

__global__ void fill_f64_kernel(double* dst, long long n, double v) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = v;
}

int launch_fill_f64(double* dst, long long n, double v, cudaStream_t st) {
  if (n <= 0) return 0;
  fill_f64_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(dst, n, v);
  return (int)cudaGetLastError();
}

// Exact dense scores.  dot_f64 (ccr_kernels.cu) fixes the value of a pair: lane l of a warp sums
// fma(double(q_e), double(v_e), acc) over the float4 chunks c = l, l + 32, ... < D/4 (elements in order), then
// an xor butterfly with offsets 16 .. 1.  Here one warp owns an 8 x 8 tile of pairs and lane l runs lane l's
// chain for all 64 of them, so every sum is formed in that order by construction.  A block of 8 warps (2 x 4)
// covers 16 queries x 32 items; per K-slice of 128 elements (one chunk per lane) its 48 rows are converted to
// double once and staged in shared memory as [row][element of the chunk][lane], which makes every warp load
// conflict-free.  The slice after the current one is read from global memory into registers during the FMAs.
constexpr int kDxQ = 16, kDxI = 32, kDxRows = kDxQ + kDxI;
constexpr int kDxSlice = 128;                                   // elements per stage: 32 chunks of 4
constexpr int kDxLoads = kDxRows * kDxSlice / 4 / 256;          // float4 loads per thread and stage
constexpr size_t kDxSmem = 2ull * kDxRows * kDxSlice * sizeof(double);  // two stages

__global__ void __launch_bounds__(256, 1) dense_exact_kernel(const float* __restrict__ q, long long B, long long ldq,
                                                             const float* __restrict__ items, long long N,
                                                             long long ldi, int D, float* __restrict__ out,
                                                             long long ld_out, long long n_qt, long long tile0) {
  extern __shared__ double s_rows[];
  const long long t = tile0 + blockIdx.x;  // query tiles vary fastest: the blocks in flight share item rows
  const long long q0 = (t % n_qt) * kDxQ, i0 = (t / n_qt) * kDxI;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int n_chunks = D >> 2, n_slices = (n_chunks + 31) >> 5;

  // chunks past D/4 and rows past B / N stage as zeros: fma(0, 0, acc) == acc for every acc but -0.0, and a
  // sum that starts at +0.0 never becomes -0.0 in round-to-nearest (x + -x is +0.0), so they change no sum
  float4 nxt[kDxLoads];
  auto load = [&](int slice) {
#pragma unroll
    for (int u = 0; u < kDxLoads; ++u) {
      const int f = threadIdx.x + 256 * u, row = f >> 5, c = (slice << 5) + (f & 31);
      const long long r = row < kDxQ ? q0 + row : i0 + (row - kDxQ);
      const bool ok = c < n_chunks && (row < kDxQ ? r < B : r < N);
      const float* src = row < kDxQ ? q + r * ldq : items + r * ldi;
      nxt[u] = ok ? __ldg(reinterpret_cast<const float4*>(src) + c) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
  };
  auto stage = [&](int buf) {
#pragma unroll
    for (int u = 0; u < kDxLoads; ++u) {
      const int f = threadIdx.x + 256 * u;
      double* d = s_rows + ((size_t)buf * kDxRows + (f >> 5)) * kDxSlice + (f & 31);
      d[0] = (double)nxt[u].x; d[32] = (double)nxt[u].y; d[64] = (double)nxt[u].z; d[96] = (double)nxt[u].w;
    }
  };

  double acc[64];  // acc[a * 8 + b]: query wq * 8 + a, item wi * 8 + b of the block tile
#pragma unroll
  for (int o = 0; o < 64; ++o) acc[o] = 0.0;
  const int wq = warp >> 2, wi = warp & 3;
  load(0);
  stage(0);
  __syncthreads();
  for (int sl = 0; sl < n_slices; ++sl) {
    if (sl + 1 < n_slices) load(sl + 1);
    const double* sq = s_rows + ((size_t)(sl & 1) * kDxRows + wq * 8) * kDxSlice + lane;
    const double* si = s_rows + ((size_t)(sl & 1) * kDxRows + kDxQ + wi * 8) * kDxSlice + lane;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      double x[8], y[8];
#pragma unroll
      for (int a = 0; a < 8; ++a) x[a] = sq[a * kDxSlice + j * 32];
#pragma unroll
      for (int b = 0; b < 8; ++b) y[b] = si[b * kDxSlice + j * 32];
#pragma unroll
      for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a * 8 + b] = fma(x[a], y[b], acc[a * 8 + b]);
    }
    if (sl + 1 < n_slices) stage((sl + 1) & 1);  // that buffer was last read before the previous barrier
    __syncthreads();
  }

  // The butterfly as a reduce-scatter: at offset `off` each lane keeps one half of its h sums and adds the
  // partner's value of it, the partner the other half.  Each sum is the butterfly's own a_l + a_(l^off) (the
  // two lanes of a pair compute the same value, fp add being commutative), so after 5 steps lane l holds the
  // butterfly result of pairs 2l and 2l + 1, with 62 shuffles instead of 320.
#pragma unroll
  for (int h = 32, off = 16; h >= 2; h >>= 1, off >>= 1) {
    const bool upper = lane & off;
#pragma unroll
    for (int i = 0; i < h; ++i) {
      const double send = upper ? acc[i] : acc[i + h];
      const double mine = upper ? acc[i + h] : acc[i];
      acc[i] = mine + __shfl_xor_sync(0xffffffffu, send, off);
    }
  }
  const long long r = q0 + wq * 8 + (lane >> 2), c = i0 + wi * 8 + 2 * (lane & 3);
  if (r < B) {
    if (c < N) out[r * ld_out + c] = (float)acc[0];
    if (c + 1 < N) out[r * ld_out + c + 1] = (float)acc[1];
  }
}

int launch_dense_exact(const float* q, long long B, long long ldq, const float* items, long long n, long long ldi,
                       int D, float* out, long long ld_out, cudaStream_t st) {
  if (B <= 0 || n <= 0) return 0;
  cudaError_t e = cudaFuncSetAttribute(dense_exact_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kDxSmem);
  if (e != cudaSuccess) return (int)e;
  const long long n_qt = (B + kDxQ - 1) / kDxQ, tiles = n_qt * ((n + kDxI - 1) / kDxI);
  for (long long t0 = 0; t0 < tiles; t0 += 1LL << 30) {
    const long long nb = tiles - t0 < (1LL << 30) ? tiles - t0 : (1LL << 30);
    dense_exact_kernel<<<(unsigned)nb, 256, kDxSmem, st>>>(q, B, ldq, items, n, ldi, D, out, ld_out, n_qt, t0);
    if ((e = cudaGetLastError()) != cudaSuccess) return (int)e;
  }
  return 0;
}

}  // namespace ccr
