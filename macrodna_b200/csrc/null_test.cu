// Random-assignment null test on the resident correlation matrix (SURVEY.md section 8 row f3).
//
// Replaces `random_test.assign` of the reference
// (Resampling_stability_analyses/BE_data_analyses/random_assignment_test.py:233-258, 1e8 trials per biopsy):
// per trial, every step pairs a uniformly random N-subset of the still-unassigned RNA cells with the DNA cells
// (a random bijection), the last step maps the remaining r <= N RNA cells injectively onto a random r-subset of
// the DNA cells; the statistic is the sum (random_assignment_test.py) or the median
// (random_assignment_test_median.py) of the matched correlations.
//
// A trial is the draw defined in include/macrodna_b200.h (mcd_null_assignments) and restated in
// oracle/restatement.py (null_draw): a uniformly random permutation of the RNA cells is the ascending order of M
// hash keys (hash bits above the b index bits, the index below); position p of the permutation belongs to step
// p / N and, in the full steps, takes DNA cell p % N; the last partial step takes the first r entries of a second
// random permutation (of the DNA cells).  That is the same distribution as the reference's
// `np.random.choice(..., replace=False)` chain -- NOT the same random stream (NumPy's Mersenne Twister is not
// reproduced), so results are compared as distributions.  The matched values are gathered from C, summed in FP64
// and, when asked for, sorted once more for the median.
//
// Two kernels compute that draw, one CTA per trial, selected by the shape:
//   - up to NULL_MAX cells a side, null_assign_kernel: bitonic sorts in shared memory (the gather reads C from L2);
//   - above, null_assign_large_kernel: the keys live in a per-CTA slab of global scratch and are ordered by a
//     CTA-wide stable LSD radix sort (cta_radix_sort), which also orders the DNA keys and the matched values.
#include "mcd_internal.cuh"

namespace {

constexpr int NT = 256;
constexpr int NULL_MAX = 4096;  // cells per side that fit the shared-memory sort
constexpr int64_t NULL_LARGE_MAX = 1 << 24;  // cells per side: at least 40 hash bits stay above the index bits

__device__ __forceinline__ unsigned long long mix64(unsigned long long z) {  // splitmix64 finaliser
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

// ascending bitonic sort of n (power of two) 64-bit words in shared memory
__device__ void bitonic_sort_u64(unsigned long long* a, int n) {
  for (int k = 2; k <= n; k <<= 1) {
    for (int j = k >> 1; j > 0; j >>= 1) {
      for (int idx = threadIdx.x; idx < n; idx += NT) {
        const int ixj = idx ^ j;
        if (ixj > idx) {
          const unsigned long long x = a[idx], y = a[ixj];
          const bool up = (idx & k) == 0;
          if (up ? x > y : x < y) {
            a[idx] = y;
            a[ixj] = x;
          }
        }
      }
      __syncthreads();
    }
  }
}

// order-preserving map double -> uint64 (for sorting the matched values)
__device__ __forceinline__ unsigned long long f64_key(double v) {
  const unsigned long long b = (unsigned long long)__double_as_longlong(v);
  return (b >> 63) ? ~b : (b | 0x8000000000000000ull);
}
__device__ __forceinline__ double key_f64(unsigned long long k) {
  const unsigned long long b = (k >> 63) ? (k & 0x7fffffffffffffffull) : ~k;
  return __longlong_as_double((long long)b);
}

__global__ void __launch_bounds__(NT) null_assign_kernel(const double* __restrict__ C, int64_t ldc, int M, int N, int Mp,
                                                          int Np, long long t0, long long trials,
                                                          unsigned long long seed, double* __restrict__ sums,
                                                          double* __restrict__ medians) {
  extern __shared__ unsigned long long nsm[];
  unsigned long long* rk = nsm;        // [Mp] RNA keys -> permutation -> matched values
  unsigned long long* dk = nsm + Mp;   // [Np] DNA keys (last partial step)
  __shared__ double red[NT / 32];
  const int q = M / N, r = M - q * N;
  for (long long trial = blockIdx.x; trial < trials; trial += gridDim.x) {  // trial t0 + trial, written at [trial]
    const unsigned long long base = mix64(seed ^ mix64((unsigned long long)(t0 + trial)));
    for (int i = threadIdx.x; i < Mp; i += NT)
      rk[i] = i < M ? ((mix64(base + 2ull * (unsigned long long)i) >> 13) << 13) | (unsigned long long)i : ~0ull;
    if (r > 0)
      for (int j = threadIdx.x; j < Np; j += NT)
        dk[j] = j < N ? ((mix64(base + 2ull * (unsigned long long)j + 1ull) >> 13) << 13) | (unsigned long long)j : ~0ull;
    __syncthreads();
    bitonic_sort_u64(rk, Mp);
    if (r > 0) bitonic_sort_u64(dk, Np);
    double acc = 0.0;
    for (int p = threadIdx.x; p < M; p += NT) {
      const int row = (int)(rk[p] & 8191ull);
      const int col = p < q * N ? p % N : (int)(dk[p - q * N] & 8191ull);
      const double v = C[(int64_t)row * ldc + col];
      acc += v;
      if (medians != nullptr) rk[p] = f64_key(v);  // each thread overwrites only the slots it just read
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double s = 0.0;
      for (int w = 0; w < NT / 32; ++w) s += red[w];
      sums[trial] = s;
    }
    if (medians != nullptr) {
      for (int i = M + threadIdx.x; i < Mp; i += NT) rk[i] = ~0ull;
      __syncthreads();
      bitonic_sort_u64(rk, Mp);
      if (threadIdx.x == 0) medians[trial] = 0.5 * (key_f64(rk[(M - 1) / 2]) + key_f64(rk[M / 2]));  // numpy.median
    }
    __syncthreads();
  }
}

// ---- instances with more than NULL_MAX cells on a side --------------------------------------------------------
constexpr int LNT = 512;  // threads of a large-path CTA
constexpr int LWARPS = LNT / 32;
constexpr int RADIX = 256;  // 8-bit digits
constexpr int ITEMS = 6;    // keys per thread per tile (8 spill at two CTAs an SM)
constexpr int TILE = LNT * ITEMS;
constexpr int MAX_PASSES = 8;

struct RadixSmem {
  unsigned hist[MAX_PASSES][RADIX];  // digit counts of every pass, taken while the keys are written (radix_count)
  unsigned base[RADIX];              // start of each digit's next key in the destination
  unsigned wh[LWARPS][RADIX];        // per-warp digit counts of a tile, then the per-warp start offsets
  unsigned wsum[RADIX / 32];
  double red[LWARPS];
};

__device__ void radix_clear(RadixSmem& s) {
  for (int i = threadIdx.x; i < MAX_PASSES * RADIX; i += LNT) (&s.hist[0][0])[i] = 0u;
  __syncthreads();
}

// counts `key` in the digit histograms of passes [0, passes), pass p sorting on bits [lo + 8p, lo + 8p + 8)
__device__ __forceinline__ void radix_count(RadixSmem& s, unsigned long long key, int lo, int passes) {
  for (int p = 0; p < passes; ++p) atomicAdd(&s.hist[p][(unsigned)(key >> (lo + 8 * p)) & (RADIX - 1)], 1u);
}

// Stable ascending LSD radix sort of the n keys in `a` on bits [lo, min(64, lo + 8 * passes)), ping-ponging with
// `t`; s.hist must hold the digit counts of the n keys (radix_clear, then radix_count of every key).  Keys equal on
// those bits keep their order.  Returns the buffer that holds the result (a if passes is even, t if odd).
// A tile of TILE keys is ranked warp by warp: warp w holds the tile's keys [w * 32 * ITEMS, (w + 1) * 32 * ITEMS) in
// ITEMS rounds of 32, and a key's place is the digit's start + the counts of the earlier warps + its rank among the
// warp's earlier keys of that digit -- the source order, hence stability.
__device__ __forceinline__ unsigned long long* cta_radix_sort(RadixSmem& s, unsigned long long* a,
                                                              unsigned long long* t, int n, int lo, int passes) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  const unsigned lt = (1u << lane) - 1u;
  for (int p = 0; p < passes; ++p) {
    const int shift = lo + 8 * p;
    __syncthreads();  // the counts are complete, the previous pass's scatter is visible
    if (threadIdx.x < RADIX) {  // exclusive scan of the pass's digit counts
      const unsigned c = s.hist[p][threadIdx.x];
      unsigned x = c;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(0xffffffffu, x, o);
        if (lane >= o) x += y;
      }
      if (lane == 31) s.wsum[w] = x;
      s.base[threadIdx.x] = x - c;
    }
    __syncthreads();
    if (threadIdx.x < RADIX)
      for (int k = 0; k < w; ++k) s.base[threadIdx.x] += s.wsum[k];
    for (int t0 = 0; t0 < n; t0 += TILE) {
      for (int i = threadIdx.x; i < LWARPS * RADIX; i += LNT) (&s.wh[0][0])[i] = 0u;
      unsigned long long k[ITEMS];
      int d[ITEMS];
      unsigned rk[ITEMS];
#pragma unroll
      for (int it = 0; it < ITEMS; ++it) {
        const int idx = t0 + (w * ITEMS + it) * 32 + lane;
        k[it] = idx < n ? a[idx] : 0ull;
        d[it] = idx < n ? (int)((unsigned)(k[it] >> shift) & (RADIX - 1)) : RADIX;  // RADIX: past the end
      }
      __syncthreads();  // wh is zero
#pragma unroll
      for (int it = 0; it < ITEMS; ++it) {
        const unsigned peers = __match_any_sync(0xffffffffu, d[it]);
        const int leader = __ffs(peers) - 1;
        unsigned prior = 0u;
        if (lane == leader && d[it] < RADIX) {
          prior = s.wh[w][d[it]];
          s.wh[w][d[it]] = prior + __popc(peers);
        }
        rk[it] = __shfl_sync(0xffffffffu, prior, leader) + __popc(peers & lt);
        __syncwarp();
      }
      __syncthreads();
      if (threadIdx.x < RADIX) {
        unsigned run = s.base[threadIdx.x];
        for (int ww = 0; ww < LWARPS; ++ww) {
          const unsigned c = s.wh[ww][threadIdx.x];
          s.wh[ww][threadIdx.x] = run;
          run += c;
        }
        s.base[threadIdx.x] = run;
      }
      __syncthreads();
#pragma unroll
      for (int it = 0; it < ITEMS; ++it)
        if (d[it] < RADIX) t[s.wh[w][d[it]] + rk[it]] = k[it];
      __syncthreads();  // the scatter has read wh
    }
    unsigned long long* x = a;
    a = t;
    t = x;
  }
  __syncthreads();
  return a;
}

// One trial at a time per CTA; the CTA's slab of `scratch` holds 2 M keys (+ 2 N when r > 0).  b = index bits.
__global__ void __launch_bounds__(LNT, 2) null_assign_large_kernel(const double* __restrict__ C, int64_t ldc, int M, int N,
                                                                int b, long long t0, long long trials,
                                                                unsigned long long seed,
                                                                unsigned long long* __restrict__ scratch, size_t slab,
                                                                double* __restrict__ sums, double* __restrict__ medians) {
  __shared__ RadixSmem s;
  unsigned long long* ra = scratch + (size_t)blockIdx.x * slab;
  unsigned long long* rb = ra + M;
  unsigned long long* da = rb + M;
  unsigned long long* db = da + N;
  const int q = M / N, r = M - q * N;
  const unsigned long long imask = (1ull << b) - 1ull;
  const int kpass = (64 - b + 7) / 8;  // passes over the hash bits [b, 64)
  for (long long trial = blockIdx.x; trial < trials; trial += gridDim.x) {  // trial t0 + trial, written at [trial]
    const unsigned long long base = mix64(seed ^ mix64((unsigned long long)(t0 + trial)));
    radix_clear(s);
    for (int i = threadIdx.x; i < M; i += LNT) {
      const unsigned long long key = ((mix64(base + 2ull * (unsigned long long)i) >> b) << b) | (unsigned long long)i;
      ra[i] = key;
      radix_count(s, key, b, kpass);
    }
    unsigned long long* rows = cta_radix_sort(s, ra, rb, M, b, kpass);
    const unsigned long long* cols = nullptr;
    if (r > 0) {
      radix_clear(s);
      for (int j = threadIdx.x; j < N; j += LNT) {
        const unsigned long long key =
            ((mix64(base + 2ull * (unsigned long long)j + 1ull) >> b) << b) | (unsigned long long)j;
        da[j] = key;
        radix_count(s, key, b, kpass);
      }
      cols = cta_radix_sort(s, da, db, N, b, kpass);
    }
    if (medians != nullptr) radix_clear(s);
    double acc = 0.0;
    for (int p = threadIdx.x; p < M; p += LNT) {
      const int row = (int)(rows[p] & imask);
      const int col = p < q * N ? p % N : (int)(cols[p - q * N] & imask);
      const double v = C[(int64_t)row * ldc + col];
      acc += v;
      if (medians != nullptr) {  // each thread overwrites only the slots it just read
        const unsigned long long key = f64_key(v);
        rows[p] = key;
        radix_count(s, key, 0, 8);
      }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) s.red[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
      double t = 0.0;
      for (int w = 0; w < LWARPS; ++w) t += s.red[w];
      sums[trial] = t;
    }
    if (medians != nullptr) {
      const unsigned long long* v = cta_radix_sort(s, rows, rows == ra ? rb : ra, M, 0, 8);
      if (threadIdx.x == 0) medians[trial] = 0.5 * (key_f64(v[(M - 1) / 2]) + key_f64(v[M / 2]));  // numpy.median
    }
    __syncthreads();
  }
}

int pow2_at_least(int64_t n) {
  int p = 1;
  while (p < n) p <<= 1;
  return p;
}

int launch_null_large(mcd_context* h, const double* C, int64_t ldc, int64_t M, int64_t N, int64_t t0, int64_t trials,
                      uint64_t seed, double* d_sums, double* d_medians) {
  int b = 13;  // index bits: max(13, bit_length(max(M, N) - 1))
  while (((int64_t)1 << b) < (M > N ? M : N)) ++b;
  const int64_t r = M % N;
  const size_t slab = ((size_t)(2 * M + (r > 0 ? 2 * N : 0)) + 3) / 4 * 4;  // keys per CTA, 32-byte aligned
  int per_sm = 1;
  MCD_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, null_assign_large_kernel, LNT, 0));
  if (per_sm < 1) per_sm = 1;
  int64_t grid = (int64_t)h->sm_count * per_sm;
  const int64_t cap = (int64_t)(((size_t)1 << 30) / (slab * 8));  // scratch <= 1 GiB
  if (grid > cap) grid = cap;
  if (grid > trials) grid = trials;
  if (grid < 1) grid = 1;
  void* scratch = nullptr;
  int st;
  if ((st = mcd_ws(h, WS_NULL, (size_t)grid * slab * 8, &scratch))) return st;
  null_assign_large_kernel<<<(unsigned)grid, LNT, 0, h->stream>>>(C, ldc, (int)M, (int)N, b, (long long)t0,
                                                                 (long long)trials,
                                                                 (unsigned long long)seed,
                                                                 static_cast<unsigned long long*>(scratch), slab,
                                                                 d_sums, d_medians);
  MCD_LAUNCH_CHECK(h, "null_assign_large_kernel");
  return MCD_OK;
}

}  // namespace

int mcd_launch_null_assignments(mcd_context* h, const double* C, int64_t ldc, int64_t M, int64_t N, int64_t t0,
                                int64_t trials, uint64_t seed, double* d_sums, double* d_medians) {
  if (M > NULL_LARGE_MAX || N > NULL_LARGE_MAX)
    return mcd_fail(h, MCD_ERR_UNSUPPORTED,
                    "null test: more than 2^24 cells on a side (fewer than 40 hash bits would remain above the index)");
  if (M > NULL_MAX || N > NULL_MAX) return launch_null_large(h, C, ldc, M, N, t0, trials, seed, d_sums, d_medians);
  const int Mp = pow2_at_least(M), Np = pow2_at_least(N);
  const size_t smem = (size_t)(Mp + Np) * 8;
  MCD_CUDA(h, cudaFuncSetAttribute(null_assign_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int per_sm = 1;
  MCD_CUDA(h, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, null_assign_kernel, NT, smem));
  if (per_sm < 1) per_sm = 1;
  int64_t grid = (int64_t)h->sm_count * per_sm;
  if (grid > trials) grid = trials;
  null_assign_kernel<<<(unsigned)grid, NT, smem, h->stream>>>(C, ldc, (int)M, (int)N, Mp, Np, (long long)t0,
                                                              (long long)trials, (unsigned long long)seed, d_sums,
                                                              d_medians);
  MCD_LAUNCH_CHECK(h, "null_assign_kernel");
  return MCD_OK;
}
