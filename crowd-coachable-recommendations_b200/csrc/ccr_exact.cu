// Exact fp32 ranking (DESIGN.md section 6b): the stages around the unchanged scan kernels and the
// exact re-rank (entry_records_kernel with the ExactDot source + finalize_kernel, ccr_kernels.cu).
//   certify_kernel       : per row, does the k-th exact value beat every item the scan stage left out?
//   compact_kernel       : columns of a dense scan-score block at or above a per-row threshold, as a CSR
//   row_norm_max_kernel  : largest fp32 row norm of an appended batch (the V of the error bound)
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

}  // namespace ccr
