// Leave-one-out sweep on the resident correlation matrix (mcd_loo_sweep, include/macrodna_b200.h; SURVEY.md section 8
// row f1).
//
// Replaces the per-cell loop of the reference's leave-one-out experiment
// (Resampling_stability_analyses/BE_data_analyses/run_loo_experiment.py:201-319): replicate r deletes RNA row
// q = cells[r] of C (`np.delete(corrs, q, 0)`, :224), runs the step loop on the rest, and gives q the DNA cell of
// highest C[q, j] among those matched at most k_steps - 1 times (:296-309).  The solves run through the replicate
// sweep engine of api.cu; this file holds the two kernels of its own:
//
//   loo_gather_kernel  sub[i, :] = C[i + (i >= q), :]  -- the replicate's cost block without an index array
//   loo_place_kernel   one CTA per replicate: matches per DNA column, masked arg-max of row q, FP64 total
#include "mcd_internal.cuh"

namespace {

constexpr int LOO_NT = 256;

inline unsigned grid_rows(int64_t rows) { return (unsigned)(rows < 65535 ? (rows < 1 ? 1 : rows) : 65535); }

// order-preserving map double -> uint64; -0.0 and +0.0 compare equal as doubles and get the same key, so that they
// tie like any other pair of equal values
__device__ __forceinline__ unsigned long long loo_key(double v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v == 0.0 ? 0.0 : v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}

// (key, index) order of the placement: larger value first, among exact ties the larger column index -- the column
// a stable ascending sort, reversed, visits first
__device__ __forceinline__ bool loo_better(unsigned long long ka, int ia, unsigned long long kb, int ib) {
  return ka > kb || (ka == kb && ia > ib);
}

// float(sum(obj_scores)) of the reference's leave_one_out (run_loo_experiment.py:201-319): the step objectives, then
// -- if `with_last` -- the test cell's value, summed as CPython's builtin sum() sums floats since 3.12: the first term
// is added to the int 0, the rest with Neumaier's compensation, and the compensation is added at the end.  A plain
// left-to-right sum differs from it in the last bit for about a third of the replicates.
__device__ double py_float_sum(const double* x, int64_t n, bool with_last, double last) {
  const int64_t terms = n + (with_last ? 1 : 0);
  if (terms == 0) return 0.0;
  double f = 0.0 + (n > 0 ? x[0] : last);
  double c = 0.0;
  for (int64_t k = 1; k < terms; ++k) {
    const double v = k < n ? x[k] : last;
    const double t = f + v;
    c += fabs(f) >= fabs(v) ? (f - t) + v : (v - t) + f;
    f = t;
  }
  if (c != 0.0 && isfinite(c)) f += c;
  return f;
}

__global__ void loo_gather_kernel(const double* __restrict__ C, int64_t ldc, int64_t q, int64_t m, int64_t n,
                                  double* __restrict__ sub, int64_t lds) {
  for (int64_t i = blockIdx.y; i < m; i += gridDim.y) {
    const double* src = C + (i + (i >= q ? 1 : 0)) * ldc;
    double* dst = sub + i * lds;
    for (int64_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x) dst[j] = src[j];
  }
}

__global__ void __launch_bounds__(LOO_NT) loo_place_kernel(const double* __restrict__ C, int64_t ldc,
                                                           const int* __restrict__ cells, int64_t m_sub, int N,
                                                           int64_t nsteps, int64_t k_steps, char* __restrict__ base,
                                                           mcd_loo_layout L) {
  char* rep = base + (size_t)blockIdx.x * L.stride;
  const int* assign = reinterpret_cast<const int*>(rep + L.assign);
  const double* obj = reinterpret_cast<const double*>(rep + L.obj);
  int* cnt = reinterpret_cast<int*>(rep + L.cnt);
  const int64_t q = cells[blockIdx.x];
  const double* crow = C + q * ldc;
  // matches per DNA column (np.count_nonzero(tagged, axis=0), run_loo_experiment.py:296); the block is
  // per-replicate global scratch, L2-resident at these sizes
  for (int j = threadIdx.x; j < N; j += LOO_NT) cnt[j] = 0;
  __syncthreads();
  for (int64_t i = threadIdx.x; i < m_sub; i += LOO_NT) {
    const int j = assign[i];
    if (j >= 0) atomicAdd(cnt + j, 1);
  }
  if (L.match != 0) {  // corr_val of the remaining rows: C[row, assign[row]] (run_loo_experiment.py:285)
    double* mc = reinterpret_cast<double*>(rep + L.match);
    for (int64_t i = threadIdx.x; i < m_sub; i += LOO_NT) {
      const int j = assign[i];
      mc[i] = j >= 0 ? C[(i + (i >= q ? 1 : 0)) * ldc + j] : 0.0;
    }
  }
  __syncthreads();
  // masked arg-max over the eligible columns (count <= k_steps - 1, :298-309)
  unsigned long long bk = 0;  // below the key of every finite value
  int bi = -1;
  for (int j = threadIdx.x; j < N; j += LOO_NT) {
    if ((int64_t)__ldcg(cnt + j) <= k_steps - 1) {
      const unsigned long long k = loo_key(crow[j]);
      if (k >= bk) {  // j grows within a thread: an equal key is a later (larger) column
        bk = k;
        bi = j;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (loo_better(ok, oi, bk, bi)) {
      bk = ok;
      bi = oi;
    }
  }
  __shared__ unsigned long long sk[LOO_NT / 32];
  __shared__ int si[LOO_NT / 32];
  if ((threadIdx.x & 31) == 0) {
    sk[threadIdx.x >> 5] = bk;
    si[threadIdx.x >> 5] = bi;
  }
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int w = 1; w < LOO_NT / 32; ++w)
      if (loo_better(sk[w], si[w], bk, bi)) {
        bk = sk[w];
        bi = si[w];
      }
    const double tc = bi >= 0 ? crow[bi] : 0.0;
    double* res = reinterpret_cast<double*>(rep + L.res);
    res[0] = tc;
    res[1] = py_float_sum(obj, nsteps, bi >= 0, tc);
    reinterpret_cast<int*>(res + 2)[0] = bi;
  }
}

}  // namespace

int mcd_launch_loo_gather(mcd_context* h, const double* C, int64_t ldc, int64_t q, int64_t m, int64_t n, double* sub,
                          int64_t lds) {
  dim3 grid((unsigned)((n + 1023) / 1024 < 64 ? (n + 1023) / 1024 : 64), grid_rows(m));
  loo_gather_kernel<<<grid, 256, 0, h->stream>>>(C, ldc, q, m, n, sub, lds);
  MCD_LAUNCH_CHECK(h, "loo_gather_kernel");
  return MCD_OK;
}

int mcd_launch_loo_place(mcd_context* h, const double* C, int64_t ldc, const int* d_cells, int64_t nrep, int64_t m_sub,
                         int64_t N, int64_t nsteps, int64_t k_steps, char* base, const mcd_loo_layout& L) {
  if (nrep < 1) return MCD_OK;
  loo_place_kernel<<<(unsigned)nrep, LOO_NT, 0, h->stream>>>(C, ldc, d_cells, m_sub, (int)N, nsteps, k_steps, base, L);
  MCD_LAUNCH_CHECK(h, "loo_place_kernel");
  return MCD_OK;
}
