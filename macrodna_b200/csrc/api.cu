// C ABI of the hot path (include/macrodna_b200.h): context, workspace, step loop (K4), fused driver.
#include <cstdio>
#include <cstdlib>
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cstddef>
#include <cstring>
#include <functional>
#include <new>
#include <thread>

#include "mcd_internal.cuh"

// ------------------------------------------------------------------------------------------------
// context plumbing
// ------------------------------------------------------------------------------------------------
int mcd_fail(mcd_context* h, int status, const char* what, cudaError_t e) {
  if (h != nullptr) {
    char buf[512];
    if (e != cudaSuccess)
      snprintf(buf, sizeof buf, "%s: %s (%s)", mcd_strerror(status), what, cudaGetErrorString(e));
    else
      snprintf(buf, sizeof buf, "%s: %s", mcd_strerror(status), what);
    h->err = buf;
  }
  return status;
}

int mcd_ws(mcd_context* h, int slot, size_t bytes, void** out) {
  mcd_buffer& b = h->ws[slot];
  if (bytes == 0) bytes = 256;
  if (b.bytes < bytes) {
    if (b.ptr != nullptr) {
      cudaStreamSynchronize(h->stream);
      cudaFree(b.ptr);
      b.ptr = nullptr;
      b.bytes = 0;
    }
    cudaError_t e = cudaMalloc(&b.ptr, bytes);
    if (e != cudaSuccess) {
      b.ptr = nullptr;
      return mcd_fail(h, MCD_ERR_NOMEM, "cudaMalloc workspace", e);
    }
    b.bytes = bytes;
  }
  *out = b.ptr;
  return MCD_OK;
}

// ------------------------------------------------------------------------------------------------
// resident matrix: the correlation matrix of a handle's last run (with its assignment), or a copy of another handle's
// (without one).  Generation ids are unique in the process, so equal ids mean "the same run's matrix".
// ------------------------------------------------------------------------------------------------
static std::atomic<uint64_t> g_generation(0);

static bool has_matrix(const mcd_context* h) { return h->gen != 0 && h->last_M >= 1; }
static bool has_assignment(const mcd_context* h) { return has_matrix(h) && h->last_assign != nullptr; }
static void drop_resident(mcd_context* h) {
  h->last_M = 0;
  h->last_assign = nullptr;
  h->gen = 0;
}
static void set_resident(mcd_context* h, int64_t M, int64_t N, int64_t ldc, const int* assign) {
  h->last_M = M;
  h->last_N = N;
  h->last_ldc = ldc;
  h->last_assign = assign;
  h->gen = ++g_generation;
}

extern "C" {

int mcd_abi_version(void) { return MCD_ABI_VERSION; }

const char* mcd_strerror(int status) {
  switch (status) {
    case MCD_OK: return "ok";
    case MCD_ERR_INVALID: return "invalid argument";
    case MCD_ERR_CUDA: return "CUDA error";
    case MCD_ERR_NOMEM: return "out of memory";
    case MCD_ERR_NONFINITE: return "non-finite value in input";
    case MCD_ERR_UNSUPPORTED: return "unsupported";
    case MCD_ERR_NOT_CONVERGED: return "assignment solver did not converge";
    default: return "unknown status";
  }
}

int mcd_create(mcd_handle* out, int device) {
  if (out == nullptr) return MCD_ERR_INVALID;
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return MCD_ERR_CUDA;
  if (device < 0 || device >= ndev) return MCD_ERR_INVALID;
  mcd_context* h = new (std::nothrow) mcd_context();
  if (h == nullptr) return MCD_ERR_NOMEM;
  h->device = device;
  cudaError_t e = cudaSetDevice(device);
  cudaDeviceProp prop;
  if (e == cudaSuccess) e = cudaGetDeviceProperties(&prop, device);
  if (e == cudaSuccess && prop.major < 10) {
    delete h;
    return MCD_ERR_UNSUPPORTED;  // sm_100a-only build
  }
  if (e == cudaSuccess) h->sm_count = prop.multiProcessorCount;
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaStreamCreateWithFlags(&h->copy_stream, cudaStreamNonBlocking);
  if (e == cudaSuccess) e = cudaMalloc(&h->d_flags, 64);
  if (e == cudaSuccess) e = cudaMemsetAsync(h->d_flags, 0, 64, h->stream);
  if (e != cudaSuccess) {
    delete h;
    return MCD_ERR_CUDA;
  }
  *out = h;
  return MCD_OK;
}

int mcd_destroy(mcd_handle h) {
  if (h == nullptr) return MCD_OK;
  cudaSetDevice(h->device);
  cudaStreamSynchronize(h->stream);
  for (mcd_context* w : h->workers) mcd_destroy(w);
  h->workers.clear();
  for (auto& b : h->ws)
    if (b.ptr) cudaFree(b.ptr);
  for (auto ev : h->ev) cudaEventDestroy(ev);
  for (int i = 0; i < 2; ++i) {
    if (h->h_stage[i]) cudaFreeHost(h->h_stage[i]);
    if (h->stage_ev[i]) cudaEventDestroy(h->stage_ev[i]);
  }
  if (h->stager) mcd_stager_destroy(h->stager);
  if (h->d_flags) cudaFree(h->d_flags);
  if (h->stream) cudaStreamDestroy(h->stream);
  if (h->copy_stream) cudaStreamDestroy(h->copy_stream);
  delete h;
  return MCD_OK;
}

const char* mcd_last_error(mcd_handle h) { return h ? h->err.c_str() : "null handle"; }
int mcd_device_sm_count(mcd_handle h) { return h ? h->sm_count : 0; }
void* mcd_stream(mcd_handle h) { return h ? (void*)h->stream : nullptr; }

int mcd_synchronize(mcd_handle h) {
  if (!h) return MCD_ERR_INVALID;
  MCD_CUDA(h, cudaSetDevice(h->device));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  return MCD_OK;
}

int64_t mcd_padded_k(int64_t G) { return (G + 15) / 16 * 16; }
int64_t mcd_padded_k_split(int64_t G) { return (G + 63) / 64 * 64; }
int64_t mcd_num_steps(int64_t M, int64_t N) { return N > 0 ? (M + N - 1) / N : 0; }

int mcd_standardize(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx, double* centred,
                    double* norms) {
  if (!h) return MCD_ERR_INVALID;
  if (!X || !centred || !norms || ncells < 0 || G < 1 || ldx < G || G > 0x7fffffff)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_standardize arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  return mcd_launch_standardize(h, X, ncells, G, ldx, centred, mcd_padded_k(G), nullptr, nullptr, 0, norms);
}

int mcd_standardize_split(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx, uint16_t* slices,
                           double* norms) {
  if (!h) return MCD_ERR_INVALID;
  if (!X || !slices || !norms || ncells < 0 || G < 1 || ldx < G || G > 0x7fffffff)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_standardize_split arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  const int64_t ldk16 = mcd_padded_k_split(G);
  return mcd_launch_standardize(h, X, ncells, G, ldx, nullptr, 0, slices, slices + ncells * ldk16, ldk16, norms);
}

int mcd_ozaki_default_slices(void) { return 6; }

int mcd_ozaki_format(mcd_handle h, int64_t M, int64_t N, int64_t G, int* nsl, int* radix_bits) {
  if (!nsl || !radix_bits) return MCD_ERR_INVALID;
  const int64_t ldk8 = mcd_padded_k_split(G);
  const int slices = h != nullptr ? h->opt.ozaki_slices : 0;
  const int radix = h != nullptr ? h->opt.ozaki_radix : 0;  // 128 / 256 forced, anything else automatic
  const bool cheap = (double)M * (double)N * (double)G <= 2.0e11;
  int n, rb;
  if (slices >= 2) {
    // an explicit slice count keeps radix 128 unless the radix is forced too (radix 256 carries at most 7 slices)
    rb = radix == 256 ? 8 : 7;
    n = slices > (rb == 8 ? 7 : MCD_OZAKI_MAX_SLICES) ? (rb == 8 ? 7 : MCD_OZAKI_MAX_SLICES) : slices;
  } else if (radix == 256) {
    rb = 8, n = 5;
  } else if (cheap || radix == 128) {
    // 8 slices (36 products, error at the level of an FP64 GEMM's own rounding) while the contraction is cheap
    // anyway; 6 slices (21 products, ~1e-12 absolute) above
    rb = 7, n = cheap ? 8 : 6;
  } else if (mcd_ozaki_exact(5, 8, ldk8)) {
    // the large-instance bottleneck: 5 radix-256 slices (15 products, ~5e-12 absolute) up to ldk8 = 32 704
    rb = 8, n = 5;
  } else {
    rb = 7, n = 6;
  }
  *nsl = n;
  *radix_bits = rb;
  return mcd_ozaki_exact(n, rb, ldk8) ? 1 : 0;
}

int mcd_ozaki_slices_for(int64_t M, int64_t N, int64_t G) {
  int nsl = 0, rb = 0;
  mcd_ozaki_format(nullptr, M, N, G, &nsl, &rb);
  return nsl;
}

int mcd_ozaki_slices(mcd_handle h, int64_t M, int64_t N, int64_t G) {
  int nsl = 0, rb = 0;
  mcd_ozaki_format(h, M, N, G, &nsl, &rb);
  return nsl;
}

namespace {
struct OptEntry {
  const char* name;
  int is_double;
  size_t off;
};
#define MCD_OPT_I(n, f) {n, 0, offsetof(mcd_options, f)}
#define MCD_OPT_D(n, f) {n, 1, offsetof(mcd_options, f)}
const OptEntry kOptions[] = {
    MCD_OPT_I("certify", certify),
    MCD_OPT_I("debug", debug),
    MCD_OPT_I("corr_only", corr_only),
    MCD_OPT_I("deterministic", deterministic),
    MCD_OPT_I("ozaki.slices", ozaki_slices),
    MCD_OPT_I("ozaki.radix", ozaki_radix),
    MCD_OPT_I("ozaki.align", ozaki_align),
    MCD_OPT_I("ozaki.plan", ozaki_plan),
    MCD_OPT_I("k1.generic", k1_generic),
    MCD_OPT_I("k1.no_stream", k1_no_stream),
    MCD_OPT_D("lap.theta", lap_theta),
    MCD_OPT_D("lap.eps_min", lap_eps_min),
    MCD_OPT_D("lap.eps0", lap_eps0),
    MCD_OPT_I("lap.scaling", lap_scaling),
    MCD_OPT_D("lap.max_rounds", lap_max_rounds),
    MCD_OPT_D("lap.tail_budget", lap_tail_budget),
    MCD_OPT_I("lap.blocks_per_sm", lap_blocks_per_sm),
    MCD_OPT_I("lap.grid_blocks", lap_grid_blocks),
    MCD_OPT_I("lap.list_max_m", lap_list_max_m),
    MCD_OPT_I("lap.lists", lap_lists),
    MCD_OPT_I("lap.list_min_nu", lap_list_min_nu),
    MCD_OPT_I("lap.tail_cluster", lap_tail_cluster),
    MCD_OPT_I("lap.tail_mh", lap_tail_mh),
    MCD_OPT_I("lap.tail_sym", lap_tail_sym),
    MCD_OPT_I("lap.async", lap_async),
    MCD_OPT_I("lap.async_nu", lap_async_nu),
    MCD_OPT_I("lap.async_threads", lap_async_threads),
    MCD_OPT_I("lap.async_blocks_per_sm", lap_async_blocks_per_sm),
    MCD_OPT_I("lap.async_stop", lap_async_stop),
    MCD_OPT_I("lap.sap", lap_sap),
    MCD_OPT_I("lap.sap_nu", lap_sap_nu),
    MCD_OPT_I("lap.prefetch_rows", lap_prefetch_rows),
    MCD_OPT_I("lap.tail_nu", lap_tail_nu),
    MCD_OPT_I("lap.mh_nu", lap_mh_nu),
    MCD_OPT_I("lap.scale_cut", lap_scale_cut),
    MCD_OPT_I("lap.scale_full_phases", lap_scale_full_phases),
    MCD_OPT_D("lap.scale_tail_rounds", lap_scale_tail_rounds),
    MCD_OPT_I("lap.aug_nu", lap_aug_nu),
    MCD_OPT_I("lap.aug_nu_square", lap_aug_nu_square),
    MCD_OPT_I("lap.rank_select", lap_rank_select),
    MCD_OPT_I("lap.min_chunk", lap_min_chunk),
    MCD_OPT_I("lap.chunk_waves", lap_chunk_waves),
};
const OptEntry* find_option(const char* name) {
  if (name == nullptr) return nullptr;
  for (const OptEntry& e : kOptions)
    if (strcmp(e.name, name) == 0) return &e;
  return nullptr;
}
}  // namespace

int mcd_set_option(mcd_handle h, const char* name, double value) {
  if (!h) return MCD_ERR_INVALID;
  const OptEntry* e = find_option(name);
  if (e == nullptr || !(value == value)) return mcd_fail(h, MCD_ERR_INVALID, "mcd_set_option: unknown option or NaN value");
  char* base = reinterpret_cast<char*>(&h->opt);
  if (e->is_double)
    *reinterpret_cast<double*>(base + e->off) = value;
  else
    *reinterpret_cast<int*>(base + e->off) = (int)value;
  return MCD_OK;
}

int mcd_get_option(mcd_handle h, const char* name, double* value) {
  if (!h || !value) return MCD_ERR_INVALID;
  const OptEntry* e = find_option(name);
  if (e == nullptr) return mcd_fail(h, MCD_ERR_INVALID, "mcd_get_option: unknown option");
  const char* base = reinterpret_cast<const char*>(&h->opt);
  *value = e->is_double ? *reinterpret_cast<const double*>(base + e->off)
                        : (double)*reinterpret_cast<const int*>(base + e->off);
  return MCD_OK;
}

int mcd_standardize_ozaki_radix(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx, int8_t* digits,
                                int nsl, int radix_bits, double* scale, double* norms) {
  if (!h) return MCD_ERR_INVALID;
  if (!X || !digits || !scale || !norms || ncells < 0 || G < 1 || ldx < G || G > 0x7fffffff || nsl < 2 ||
      (radix_bits != 7 && radix_bits != 8) || nsl > (radix_bits == 8 ? 7 : MCD_OZAKI_MAX_SLICES))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_standardize_ozaki arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  mcd_ozaki_out oz;
  oz.digits = digits;
  oz.ldk8 = mcd_padded_k_split(G);
  oz.slice_stride = ncells * oz.ldk8;
  oz.nsl = nsl;
  oz.rb = radix_bits;
  oz.scale = scale;
  return mcd_launch_standardize(h, X, ncells, G, ldx, nullptr, 0, nullptr, nullptr, 0, norms, nullptr, &oz);
}

int mcd_standardize_ozaki(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx, int8_t* digits,
                          int nsl, double* scale, double* norms) {
  return mcd_standardize_ozaki_radix(h, X, ncells, G, ldx, digits, nsl, 7, scale, norms);
}

int mcd_corr_ozaki_radix(mcd_handle h, const int8_t* A8, int64_t M, const int8_t* B8, int64_t N, int64_t G,
                         int64_t ldk8, int nsl, int radix_bits, const double* sA, const double* sB, const double* nA,
                         const double* nB, double* C, int64_t ldc, double* Ct, int64_t ldct) {
  if (!h) return MCD_ERR_INVALID;
  if (!A8 || !B8 || !sA || !sB || !nA || !nB || (!C && !Ct) || M < 0 || N < 0 || G < 1 || ldk8 < G ||
      (ldk8 % 64) != 0 || (C && ldc < N) || (Ct && ldct < M))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_corr_ozaki arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  return mcd_launch_corr_ozaki(h, A8, M * ldk8, M, B8, N * ldk8, N, ldk8, nsl, radix_bits, sA, sB, nA, nB, C, ldc, Ct,
                               ldct);
}

int mcd_corr_ozaki(mcd_handle h, const int8_t* A8, int64_t M, const int8_t* B8, int64_t N, int64_t G, int64_t ldk8,
                   int nsl, const double* sA, const double* sB, const double* nA, const double* nB, double* C,
                   int64_t ldc, double* Ct, int64_t ldct) {
  return mcd_corr_ozaki_radix(h, A8, M, B8, N, G, ldk8, nsl, 7, sA, sB, nA, nB, C, ldc, Ct, ldct);
}

int mcd_check_finite(mcd_handle h) {
  if (!h) return MCD_ERR_INVALID;
  MCD_CUDA(h, cudaSetDevice(h->device));
  int flag = 0;
  MCD_CUDA(h, cudaMemcpyAsync(&flag, h->d_flags, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemsetAsync(h->d_flags, 0, sizeof(int), h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  if (flag) return mcd_fail(h, MCD_ERR_NONFINITE, "NaN or Inf in the expression / copy-number matrix");
  return MCD_OK;
}

int mcd_corr_fp64(mcd_handle h, const double* A, int64_t M, const double* B, int64_t N, int64_t G, int64_t ldk,
                  const double* nA, const double* nB, double* C, int64_t ldc, double* Ct, int64_t ldct) {
  if (!h) return MCD_ERR_INVALID;
  if (!A || !B || !nA || !nB || (!C && !Ct) || M < 0 || N < 0 || G < 1 || ldk < G || (ldk % 16) != 0 ||
      (C && ldc < N) || (Ct && ldct < M))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_corr_fp64 arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  return mcd_launch_corr_fp64(h, A, M, B, N, ldk, nA, nB, C, ldc, Ct, ldct);
}

int mcd_corr_split(mcd_handle h, const uint16_t* A3, int64_t M, const uint16_t* B3, int64_t N, int64_t G,
                    int64_t ldk16, const double* nA, const double* nB, double* C, int64_t ldc, double* Ct,
                    int64_t ldct) {
  if (!h) return MCD_ERR_INVALID;
  if (!A3 || !B3 || !nA || !nB || (!C && !Ct) || M < 0 || N < 0 || G < 1 || ldk16 < G || (ldk16 % 64) != 0 ||
      (C && ldc < N) || (Ct && ldct < M))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_corr_split arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  return mcd_launch_corr_split(h, A3, A3 + M * ldk16, M, B3, B3 + N * ldk16, N, ldk16, nA, nB, C, ldc, Ct, ldct);
}

static int lap_max_impl(mcd_handle h, const double* W, int64_t n, int64_t m, int64_t ldw, int32_t* col4row,
                        double* objective, double* prices, double* cert_out) {
  if (!h) return MCD_ERR_INVALID;
  if (!W || !col4row || n < 0 || m < n || ldw < m) return mcd_fail(h, MCD_ERR_INVALID, "mcd_lap_max arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  void* work = nullptr;
  int st = mcd_ws(h, WS_LAP, mcd_lap_workspace_bytes(n, m) + 512, &work);
  if (st) return st;
  // counters and certificate live in the first 512 bytes of the slot
  mcd_lap_counters* cnt = static_cast<mcd_lap_counters*>(work);
  mcd_lap_cert* cert = reinterpret_cast<mcd_lap_cert*>(static_cast<char*>(work) + 256);
  MCD_CUDA(h, cudaMemsetAsync(work, 0, 512, h->stream));
  int st2 = mcd_launch_lap(h, W, n, m, ldw, col4row, objective, static_cast<char*>(work) + 512, cnt, true, cert, prices);
  if (st2) return st2;
  mcd_lap_counters hc;
  mcd_lap_cert hcert;
  MCD_CUDA(h, cudaMemcpyAsync(&hc, cnt, sizeof hc, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(&hcert, cert, sizeof hcert, cudaMemcpyDeviceToHost, h->stream));
  if ((st = mcd_check_finite(h))) return st;  // synchronises
  if (cert_out) {
    cert_out[0] = hcert.rel_gap;
    cert_out[1] = hcert.gap;
    cert_out[2] = hcert.max_violation;
    cert_out[3] = (double)hcert.n_bad;
  }
  if (n > 0 && (hc.status & 1)) return mcd_fail(h, MCD_ERR_NOT_CONVERGED, "a person was left unassigned");
  if (n > 0 && (hc.status & 2)) return mcd_fail(h, MCD_ERR_NOT_CONVERGED, "the dual certificate of the assignment failed");
  return MCD_OK;
}

int mcd_lap_certify(mcd_handle h, const double* W, int64_t n, int64_t m, int64_t ldw, const int32_t* col4row,
                    const double* prices, double* cert_out) {
  if (!h) return MCD_ERR_INVALID;
  if (!W || !col4row || !prices || !cert_out || n < 1 || m < n || ldw < m || m > 0x3fffffff)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_lap_certify arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  void* work = nullptr;
  int st = mcd_ws(h, WS_LAP, 512 + (size_t)m * 4 + (size_t)n * 8 + 1024, &work);
  if (st) return st;
  mcd_lap_counters* cnt = static_cast<mcd_lap_counters*>(work);
  mcd_lap_cert* cert = reinterpret_cast<mcd_lap_cert*>(static_cast<char*>(work) + 256);
  MCD_CUDA(h, cudaMemsetAsync(work, 0, 512, h->stream));
  if ((st = mcd_launch_lap_certify(h, W, n, m, ldw, col4row, prices, static_cast<char*>(work) + 512, cert, cnt)))
    return st;
  mcd_lap_cert hcert;
  MCD_CUDA(h, cudaMemcpyAsync(&hcert, cert, sizeof hcert, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  cert_out[0] = hcert.rel_gap;
  cert_out[1] = hcert.gap;
  cert_out[2] = hcert.max_violation;
  cert_out[3] = (double)hcert.n_bad;
  return MCD_OK;
}

int mcd_lap_max(mcd_handle h, const double* W, int64_t n, int64_t m, int64_t ldw, int32_t* col4row,
                double* objective) {
  return lap_max_impl(h, W, n, m, ldw, col4row, objective, nullptr, nullptr);
}

int mcd_lap_max_certified(mcd_handle h, const double* W, int64_t n, int64_t m, int64_t ldw, int32_t* col4row,
                          double* objective, double* prices, double* cert) {
  return lap_max_impl(h, W, n, m, ldw, col4row, objective, prices, cert);
}

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// K4: step-loop bookkeeping kernels (reference macrodna.py:110-145, O(M) instead of dense M x N)
// ------------------------------------------------------------------------------------------------
namespace {

__global__ void iota_flags_kernel(int* act, int* flag, int* assign, int* step, int M) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) {
    act[i] = i;
    flag[i] = 1;
    assign[i] = -1;
    step[i] = 0;
  }
}

// W[j, k] = Ct[j, act[k]]  (persons = DNA rows of Ct, objects = still-unassigned RNA cells)
__global__ void gather_cols_kernel(const double* __restrict__ Ct, int64_t ldct, const int* __restrict__ act, int R,
                                   double* __restrict__ W, int64_t ldw, int64_t nrows) {
  for (int64_t j = blockIdx.y; j < nrows; j += gridDim.y) {  // gridDim.y is capped at 65535
    const double* src = Ct + j * ldct;
    double* dst = W + j * ldw;
    for (int k = blockIdx.x * blockDim.x + threadIdx.x; k < R; k += gridDim.x * blockDim.x) dst[k] = src[act[k]];
  }
}

// W[k, :] = C[act[k], :]  (persons = still-unassigned RNA cells, objects = DNA cells)
__global__ void gather_rows_kernel(const double* __restrict__ C, int64_t ldc, const int* __restrict__ act, int N,
                                   double* __restrict__ W, int64_t ldw, int64_t nrows) {
  for (int64_t k = blockIdx.y; k < nrows; k += gridDim.y) {
    const double* src = C + (int64_t)act[k] * ldc;
    double* dst = W + k * ldw;
    for (int j = blockIdx.x * blockDim.x + threadIdx.x; j < N; j += gridDim.x * blockDim.x) dst[j] = src[j];
  }
}

// persons were DNA cells: col4row[j] = index into act
__global__ void record_dna_major_kernel(const int* __restrict__ col4row, int N, const int* __restrict__ act,
                                        int* assign, int* step, int* flag, int tag) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j < N) {
    const int k = col4row[j];
    if (k >= 0) {
      const int g = act[k];
      assign[g] = j;
      step[g] = tag;
      flag[g] = 0;
    }
  }
}
// persons were RNA cells: col4row[k] = DNA column
__global__ void record_rna_major_kernel(const int* __restrict__ col4row, int R, const int* __restrict__ act,
                                        int* assign, int* step, int* flag, int tag) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k < R) {
    const int j = col4row[k];
    if (j >= 0) {
      const int g = act[k];
      assign[g] = j;
      step[g] = tag;
      flag[g] = 0;
    }
  }
}

// Ordered stream compaction of the still-unassigned RNA rows (ascending, macrodna.py:141-145). One CTA.
__global__ void __launch_bounds__(1024) compact_active_kernel(const int* __restrict__ flag, int M, int* act_out) {
  __shared__ int sums[1024];
  const int t = threadIdx.x;
  const int per = (M + 1023) / 1024;
  const int lo = min(M, t * per), hi = min(M, lo + per);
  int c = 0;
  for (int i = lo; i < hi; ++i) c += flag[i];
  sums[t] = c;
  __syncthreads();
  for (int o = 1; o < 1024; o <<= 1) {  // Hillis-Steele inclusive scan
    const int v = t >= o ? sums[t - o] : 0;
    __syncthreads();
    sums[t] += v;
    __syncthreads();
  }
  int pos = sums[t] - c;
  for (int i = lo; i < hi; ++i)
    if (flag[i]) act_out[pos++] = i;
}

// dst[c, r] = src[r, c] through a padded 32x32 shared tile (coalesced on both sides)
__global__ void transpose_f64_kernel(const double* __restrict__ src, int64_t rows, int64_t cols, int64_t lds,
                                     double* __restrict__ dst, int64_t ldd) {
  __shared__ double tile[32][33];
  const int64_t c0 = (int64_t)blockIdx.x * 32, r0 = (int64_t)blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t r = r0 + i, c = c0 + threadIdx.x;
    tile[i][threadIdx.x] = (r < rows && c < cols) ? src[r * lds + c] : 0.0;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int64_t c = c0 + i, r = r0 + threadIdx.x;
    if (c < cols && r < rows) dst[c * ldd + r] = tile[threadIdx.x][i];
  }
}

__global__ void gather_match_kernel(const double* __restrict__ C, int64_t ldc, const int* __restrict__ assign, int64_t M,
                                    double* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < M) {
    const int j = assign[i];
    out[i] = j >= 0 ? C[i * ldc + j] : 0.0;
  }
}

// sub[i, j] = C[rows[i], cols[j]]  (rows / cols may repeat: resampled replicates carry duplicate DNA cells)
__global__ void gather_sub_kernel(const double* __restrict__ C, int64_t ldc, const int* __restrict__ rows,
                                  const int* __restrict__ cols, int64_t m, int64_t n, double* __restrict__ sub,
                                  int64_t lds) {
  for (int64_t i = blockIdx.y; i < m; i += gridDim.y) {
    const double* src = C + (int64_t)(rows ? rows[i] : i) * ldc;
    double* dst = sub + i * lds;
    for (int64_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x)
      dst[j] = src[cols ? cols[j] : j];
  }
}

__global__ void gather_rows_out_kernel(const double* __restrict__ C, int64_t ldc, const int* __restrict__ rows,
                                       int64_t nrows, int64_t n, double* __restrict__ out) {
  for (int64_t i = blockIdx.y; i < nrows; i += gridDim.y) {
    const double* src = C + (int64_t)rows[i] * ldc;
    for (int64_t j = blockIdx.x * blockDim.x + threadIdx.x; j < n; j += (int64_t)gridDim.x * blockDim.x)
      out[i * n + j] = src[j];
  }
}

__global__ void gather_pairs_kernel(const double* __restrict__ C, int64_t ldc, const int* __restrict__ rows,
                                    const int* __restrict__ cols, int64_t n, double* __restrict__ out) {
  const int64_t k = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (k < n) out[k] = C[(int64_t)rows[k] * ldc + cols[k]];
}

// cls[j] = first position of cols that holds the same cell as position j (copies of a cell share an id < n); returns
// the number of extra copies.  O(n log n).
int64_t duplicate_classes(const int32_t* cols, int64_t n, std::vector<int>& cls) {
  std::vector<int64_t> order((size_t)n);
  for (int64_t j = 0; j < n; ++j) order[(size_t)j] = j;
  std::stable_sort(order.begin(), order.end(), [&](int64_t a, int64_t b) { return cols[a] < cols[b]; });
  cls.assign((size_t)n, 0);
  int64_t extra = 0;
  for (int64_t q = 0; q < n; ++q) {
    const int64_t j = order[(size_t)q];
    if (q > 0 && cols[j] == cols[order[(size_t)q - 1]]) {
      cls[(size_t)j] = cls[(size_t)order[(size_t)q - 1]];
      ++extra;
    } else {
      cls[(size_t)j] = (int)j;
    }
  }
  return extra;
}

// rows of a gather go to gridDim.y, which the hardware caps at 65535: the kernels loop over the rest
inline unsigned grid_rows(int64_t rows) { return (unsigned)(rows < 65535 ? (rows < 1 ? 1 : rows) : 65535); }

cudaEvent_t get_event(mcd_context* h, size_t idx) {
  while (h->ev.size() <= idx) {
    cudaEvent_t e;
    cudaEventCreate(&e);
    h->ev.push_back(e);
  }
  return h->ev[idx];
}

struct StepPlan {
  int64_t nsteps;
  size_t w_bytes;
  size_t lap_bytes;
};

StepPlan plan_steps(int64_t M, int64_t N) {
  StepPlan p;
  p.nsteps = mcd_num_steps(M, N);
  p.w_bytes = 0;
  p.lap_bytes = 0;
  int64_t R = M;
  for (int64_t s = 0; s < p.nsteps; ++s, R -= N) {
    const int64_t n = R > N ? N : R;
    const int64_t m = R > N ? R : N;
    const size_t lb = mcd_lap_workspace_bytes(n, m);
    if (lb > p.lap_bytes) p.lap_bytes = lb;
    if (s > 0) {
      const size_t wb = (size_t)n * (size_t)((m + 1) & ~1LL) * 8;
      if (wb > p.w_bytes) p.w_bytes = wb;
    }
  }
  return p;
}

// Device-side outputs of one step loop, carved out of one block: assign[M], step[M], obj[nsteps], one counter
// block and one dual certificate per step.
struct StepOut {
  int* assign;
  int* step;
  double* obj;
  mcd_lap_counters* cnt;
  mcd_lap_cert* cert;
};
size_t step_out_bytes(int64_t M, int64_t nsteps) {
  const size_t mi = ((size_t)M * 4 + 255) / 256 * 256;
  const size_t ob = ((size_t)nsteps * 8 + 255) / 256 * 256;
  return 2 * mi + ob + (sizeof(mcd_lap_counters) + sizeof(mcd_lap_cert)) * (size_t)nsteps;
}
StepOut carve_step_out(void* base, int64_t M, int64_t nsteps) {
  const size_t mi = ((size_t)M * 4 + 255) / 256 * 256;
  const size_t ob = ((size_t)nsteps * 8 + 255) / 256 * 256;
  char* mb = static_cast<char*>(base);
  StepOut o;
  o.assign = reinterpret_cast<int*>(mb);
  o.step = reinterpret_cast<int*>(mb + mi);
  o.obj = reinterpret_cast<double*>(mb + 2 * mi);
  o.cnt = reinterpret_cast<mcd_lap_counters*>(mb + 2 * mi + ob);
  o.cert = reinterpret_cast<mcd_lap_cert*>(mb + 2 * mi + ob + sizeof(mcd_lap_counters) * (size_t)nsteps);
  return o;
}

// Host side of the per-step records: fills the solver part of `stats`, prints the debug lines, returns the OR of
// the steps' status bits (1 = a cell left unassigned, 2 = dual certificate failed).
int fold_step_records(mcd_context* h, int64_t M, int64_t N, int64_t nsteps, const mcd_lap_counters* hc,
                      const mcd_lap_cert* hcert, mcd_stats* stats, size_t ev_lap, bool have_events) {
  int bad = 0;
  if (h->opt.debug) {
    int64_t R = M;
    for (int64_t s = 0; s < nsteps; ++s, R -= N) {
      const int64_t mm = R > N ? R : N;
      fprintf(stderr, "[lap step %lld] n=%lld m=%lld rounds=%lld bids=%lld sweeps=%lld aug=%lld/%lld cert_gap=%.3e cyc=",
              (long long)s, (long long)(R > N ? N : R), (long long)mm, hc[s].rounds, hc[s].bids, hc[s].bytes / (mm * 8),
              hc[s].aug_rows, hc[s].aug_steps, hcert[s].rel_gap);
      for (int q = 0; q < 8; ++q) fprintf(stderr, "%lld ", hc[s].t_phase[q]);
      fprintf(stderr, " async_us=");
      for (int q = 0; q < 8; ++q) fprintf(stderr, "%lld ", hc[s].a_ts[q] / 1000);
      fprintf(stderr, " async_kbids=");
      for (int q = 0; q < 8; ++q) fprintf(stderr, "%lld ", hc[s].a_hops[q] / 1000);
      fprintf(stderr, "\n");
    }
  }
  for (int64_t s = 0; s < nsteps; ++s) {
    bad |= hc[s].status;
    if (!stats) continue;
    stats->lap_rounds += hc[s].rounds;
    stats->lap_bids += hc[s].bids;
    stats->lap_bytes += hc[s].bytes;
    stats->lap_aug_rows += hc[s].aug_rows;
    stats->lap_aug_steps += hc[s].aug_steps;
    for (int q = 0; q < 8; ++q) stats->lap_cycles[q] += hc[s].t_phase[q];
    if (h->opt.certify) {
      if (hcert[s].rel_gap > stats->cert_rel_gap) stats->cert_rel_gap = hcert[s].rel_gap;
      if (hcert[s].max_violation > stats->cert_max_violation) stats->cert_max_violation = hcert[s].max_violation;
      stats->cert_bad += hcert[s].n_bad;
      stats->cert_steps += 1;
    }
    if (s < MCD_MAX_STEP_STATS) {
      if (have_events) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, get_event(h, ev_lap + s), get_event(h, ev_lap + s + 1));
        stats->step_ms[s] = ms;
      }
      stats->step_rounds[s] = hc[s].rounds;
      stats->step_bids[s] = hc[s].bids;
      stats->step_cert_gap[s] = h->opt.certify ? hcert[s].rel_gap : -1.0;
    }
  }
  return bad;
}

int step_status(mcd_context* h, int bad) {
  if (bad & 1) return mcd_fail(h, MCD_ERR_NOT_CONVERGED, "a step left an RNA/DNA cell unassigned");
  if (bad & 2) return mcd_fail(h, MCD_ERR_NOT_CONVERGED, "the dual certificate of a step's assignment failed");
  return MCD_OK;
}

// Enqueue the whole step loop on h->stream (no host synchronisation: every step's shape is known
// up front because each non-final step matches exactly N RNA cells).
// Device outputs: d_assign[M], d_step[M], d_obj[nsteps], d_counters[nsteps].
// dna_class: optional DEVICE int [N], equal ids = DNA cells that are copies of one another (identical columns of C):
// in the steps where the DNA cells are the solver's persons they bid as a class (see mcd_launch_lap).
int enqueue_step_loop(mcd_context* h, const double* C, int64_t ldc, const double* Ct, int64_t ldct, int64_t M,
                      int64_t N, const StepOut& out, size_t ev_base, bool check_finite, bool record_events = true,
                      const int* dna_class = nullptr) {
  int* d_assign = out.assign;
  int* d_step = out.step;
  double* d_obj = out.obj;
  mcd_lap_counters* d_counters = out.cnt;
  const StepPlan plan = plan_steps(M, N);
  void* wbuf = nullptr;
  void* lapbuf = nullptr;
  void* stepbuf = nullptr;
  int st;
  if ((st = mcd_ws(h, WS_W, plan.w_bytes, &wbuf))) return st;
  if ((st = mcd_ws(h, WS_LAP, plan.lap_bytes, &lapbuf))) return st;
  const size_t mi = ((size_t)M * 4 + 255) / 256 * 256;
  const size_t ci = ((size_t)(M > N ? M : N) * 4 + 255) / 256 * 256;
  if ((st = mcd_ws(h, WS_STEP, 3 * mi + ci, &stepbuf))) return st;
  char* sb = static_cast<char*>(stepbuf);
  int* act[2] = {reinterpret_cast<int*>(sb), reinterpret_cast<int*>(sb + mi)};
  int* flag = reinterpret_cast<int*>(sb + 2 * mi);
  int* col4row = reinterpret_cast<int*>(sb + 3 * mi);
  double* W = static_cast<double*>(wbuf);

  MCD_CUDA(h, cudaMemsetAsync(d_counters, 0, (sizeof(mcd_lap_counters) + sizeof(mcd_lap_cert)) * plan.nsteps, h->stream));
  iota_flags_kernel<<<(unsigned)((M + 255) / 256), 256, 0, h->stream>>>(act[0], flag, d_assign, d_step, (int)M);
  MCD_LAUNCH_CHECK(h, "iota_flags_kernel");

  int64_t R = M;
  int cur = 0;
  for (int64_t s = 0; s < plan.nsteps; ++s) {
    if (record_events && s < MCD_MAX_STEP_STATS) MCD_CUDA(h, cudaEventRecord(get_event(h, ev_base + s), h->stream));
    if (R > N) {
      // all N DNA cells take one RNA cell each (macrodna.py:29,53 with n_min = N)
      const double* Wp;
      int64_t ldw;
      if (s == 0) {
        Wp = Ct;
        ldw = ldct;
      } else {
        ldw = (R + 1) & ~1LL;
        dim3 grid((unsigned)((R + 1023) / 1024 < 64 ? (R + 1023) / 1024 : 64), grid_rows(N));
        gather_cols_kernel<<<grid, 256, 0, h->stream>>>(Ct, ldct, act[cur], (int)R, W, ldw, N);
        MCD_LAUNCH_CHECK(h, "gather_cols_kernel");
        Wp = W;
      }
      if ((st = mcd_launch_lap(h, Wp, N, R, ldw, col4row, d_obj + s, lapbuf, d_counters + s, check_finite && s == 0,
                               out.cert + s, nullptr, dna_class)))
        return st;
      record_dna_major_kernel<<<(unsigned)((N + 255) / 256), 256, 0, h->stream>>>(col4row, (int)N, act[cur], d_assign,
                                                                                 d_step, flag, (int)(s + 1));
      MCD_LAUNCH_CHECK(h, "record_dna_major_kernel");
      if (s + 1 < plan.nsteps) {
        compact_active_kernel<<<1, 1024, 0, h->stream>>>(flag, (int)M, act[cur ^ 1]);
        MCD_LAUNCH_CHECK(h, "compact_active_kernel");
        cur ^= 1;
      }
    } else {
      // last step: every remaining RNA cell takes a DNA cell (n_min = |R|)
      const double* Wp;
      int64_t ldw;
      if (s == 0) {
        Wp = C;
        ldw = ldc;
      } else {
        ldw = (N + 1) & ~1LL;
        dim3 grid((unsigned)((N + 1023) / 1024 < 64 ? (N + 1023) / 1024 : 64), grid_rows(R));
        gather_rows_kernel<<<grid, 256, 0, h->stream>>>(C, ldc, act[cur], (int)N, W, ldw, R);
        MCD_LAUNCH_CHECK(h, "gather_rows_kernel");
        Wp = W;
      }
      if ((st = mcd_launch_lap(h, Wp, R, N, ldw, col4row, d_obj + s, lapbuf, d_counters + s, check_finite && s == 0,
                               out.cert + s)))
        return st;
      record_rna_major_kernel<<<(unsigned)((R + 255) / 256), 256, 0, h->stream>>>(col4row, (int)R, act[cur], d_assign,
                                                                                 d_step, flag, (int)(s + 1));
      MCD_LAUNCH_CHECK(h, "record_rna_major_kernel");
    }
    R -= N;
  }
  if (record_events)
    MCD_CUDA(h, cudaEventRecord(
        get_event(h, ev_base + (plan.nsteps < MCD_MAX_STEP_STATS ? plan.nsteps : MCD_MAX_STEP_STATS)), h->stream));
  return MCD_OK;
}

}  // namespace

extern "C" {

int mcd_transpose_f64(mcd_handle h, const double* src, int64_t rows, int64_t cols, int64_t lds, double* dst,
                      int64_t ldd) {
  if (!h) return MCD_ERR_INVALID;
  if (!src || !dst || rows < 0 || cols < 0 || lds < cols || ldd < rows)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_transpose_f64 arguments");
  if (rows == 0 || cols == 0) return MCD_OK;
  MCD_CUDA(h, cudaSetDevice(h->device));
  const int64_t gy = (rows + 31) / 32;
  if (gy > 65535) {
    // split the row range so gridDim.y stays legal
    for (int64_t r0 = 0; r0 < rows; r0 += 65535LL * 32) {
      const int64_t nr = rows - r0 < 65535LL * 32 ? rows - r0 : 65535LL * 32;
      dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((nr + 31) / 32));
      transpose_f64_kernel<<<grid, dim3(32, 8), 0, h->stream>>>(src + r0 * lds, nr, cols, lds, dst + r0, ldd);
      MCD_LAUNCH_CHECK(h, "transpose_f64_kernel");
    }
    return MCD_OK;
  }
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)gy);
  transpose_f64_kernel<<<grid, dim3(32, 8), 0, h->stream>>>(src, rows, cols, lds, dst, ldd);
  MCD_LAUNCH_CHECK(h, "transpose_f64_kernel");
  return MCD_OK;
}

int mcd_last_match_values(mcd_handle h, double* out, int64_t M, int out_space) {
  if (!h) return MCD_ERR_INVALID;
  if (!out || M < 1 || M != h->last_M || !has_assignment(h))
    return mcd_fail(h, MCD_ERR_INVALID,
                    "mcd_last_match_values: no matching mcd_cell2cell result is resident (a copy made by "
                    "mcd_share_resident carries no assignment)");
  MCD_CUDA(h, cudaSetDevice(h->device));
  const double* C = static_cast<const double*>(h->ws[WS_C].ptr);
  double* tmp = out;
  void* scratch = nullptr;
  if (out_space != MCD_MEM_DEVICE) {
    int st = mcd_ws(h, WS_W, (size_t)M * 8, &scratch);  // the step-loop block buffer is free between calls
    if (st) return st;
    tmp = static_cast<double*>(scratch);
  }
  gather_match_kernel<<<(unsigned)((M + 255) / 256), 256, 0, h->stream>>>(C, h->last_ldc, h->last_assign, M, tmp);
  MCD_LAUNCH_CHECK(h, "gather_match_kernel");
  if (out_space != MCD_MEM_DEVICE)
    MCD_CUDA(h, cudaMemcpyAsync(out, tmp, (size_t)M * 8, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  return MCD_OK;
}

int mcd_lap_steps(mcd_handle h, const double* C, int64_t ldc, const double* Ct, int64_t ldct, int64_t M, int64_t N,
                  int32_t* assign, int32_t* step, double* step_obj, int out_space, mcd_stats* stats) {
  if (!h) return MCD_ERR_INVALID;
  if (!C || !Ct || !assign || !step || M < 1 || N < 1 || ldc < N || ldct < M || M > 0x3fffffff || N > 0x3fffffff)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_lap_steps arguments");
  MCD_CUDA(h, cudaSetDevice(h->device));
  drop_resident(h);  // the resident cell2cell result (if any) is about to be overwritten
  const int64_t nsteps = mcd_num_steps(M, N);
  void* misc = nullptr;
  int st = mcd_ws(h, WS_MISC, step_out_bytes(M, nsteps), &misc);
  if (st) return st;
  const StepOut out = carve_step_out(misc, M, nsteps);
  const int64_t launches0 = h->launches;
  const size_t EV_LAP = 8;
  MCD_CUDA(h, cudaEventRecord(get_event(h, 6), h->stream));
  if ((st = enqueue_step_loop(h, C, ldc, Ct, ldct, M, N, out, EV_LAP, true))) return st;
  MCD_CUDA(h, cudaEventRecord(get_event(h, 7), h->stream));

  const cudaMemcpyKind kind = out_space == MCD_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  MCD_CUDA(h, cudaMemcpyAsync(assign, out.assign, (size_t)M * 4, kind, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(step, out.step, (size_t)M * 4, kind, h->stream));
  if (step_obj) MCD_CUDA(h, cudaMemcpyAsync(step_obj, out.obj, (size_t)nsteps * 8, kind, h->stream));
  std::vector<mcd_lap_counters> hc((size_t)nsteps);
  std::vector<mcd_lap_cert> hcert((size_t)nsteps);
  int flag = 0;
  MCD_CUDA(h, cudaMemcpyAsync(hc.data(), out.cnt, sizeof(mcd_lap_counters) * nsteps, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(hcert.data(), out.cert, sizeof(mcd_lap_cert) * nsteps, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(&flag, h->d_flags, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemsetAsync(h->d_flags, 0, sizeof(int), h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  if (flag) return mcd_fail(h, MCD_ERR_NONFINITE, "NaN or Inf in the correlation matrix");
  if (stats) memset(stats, 0, sizeof *stats);
  const int bad = fold_step_records(h, M, N, nsteps, hc.data(), hcert.data(), stats, EV_LAP, true);
  if (stats) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, get_event(h, 6), get_event(h, 7));
    stats->ms_lap = ms;
    stats->ms_total = ms;
    stats->n_steps = nsteps;
    stats->kernel_launches = h->launches - launches0;
  }
  return step_status(h, bad);
}

int mcd_cell2cell(mcd_handle h, const double* rna, int64_t ld_rna, const double* dna, int64_t ld_dna, int64_t M,
                  int64_t N, int64_t G, int in_space, int precision, int32_t* assign, int32_t* step, double* step_obj,
                  double* corr_out, int out_space, mcd_stats* stats) {
  return mcd_cell2cell_gather(h, rna, ld_rna, nullptr, dna, ld_dna, nullptr, M, N, G, in_space, precision, assign, step,
                              step_obj, corr_out, out_space, stats);
}

int mcd_cell2cell_gather(mcd_handle h, const double* rna, int64_t ld_rna, const int32_t* rna_gene_idx,
                         const double* dna, int64_t ld_dna, const int32_t* dna_gene_idx, int64_t M, int64_t N,
                         int64_t G, int in_space, int precision, int32_t* assign, int32_t* step, double* step_obj,
                         double* corr_out, int out_space, mcd_stats* stats) {
  if (!h) return MCD_ERR_INVALID;
  if (!rna || !dna || !assign || !step || M < 1 || N < 1 || G < 1 || (!rna_gene_idx && ld_rna < G) ||
      (!dna_gene_idx && ld_dna < G) || ld_rna < 1 || ld_dna < 1 || M > 0x3fffffff || N > 0x3fffffff || G > 0x7fffffff)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_cell2cell arguments");
  for (int64_t g = 0; g < G; ++g) {
    if ((rna_gene_idx && (rna_gene_idx[g] < 0 || rna_gene_idx[g] >= ld_rna)) ||
        (dna_gene_idx && (dna_gene_idx[g] < 0 || dna_gene_idx[g] >= ld_dna)))
      return mcd_fail(h, MCD_ERR_INVALID, "mcd_cell2cell_gather: gene index out of range");
  }
  if (precision != MCD_PREC_FP64 && precision != MCD_PREC_SPLIT_FP16 && precision != MCD_PREC_OZAKI_INT8)
    return mcd_fail(h, MCD_ERR_INVALID, "unknown precision");
  int nsl = 0, rb = 0;
  // exact int32 accumulation bounds the gene count of the integer path; longer rows use the FP64 pipe
  if (mcd_ozaki_format(h, M, N, G, &nsl, &rb) != 1 && precision == MCD_PREC_OZAKI_INT8) precision = MCD_PREC_FP64;
  MCD_CUDA(h, cudaSetDevice(h->device));
  drop_resident(h);  // whatever was resident is about to be overwritten (also on an early error return)
  const int64_t launches0 = h->launches;
  enum { EV_T0 = 0, EV_H2D, EV_STD, EV_CORR, EV_LAPEND, EV_D2H, EV_LAP = 8 };
  const size_t EV_DNA_K1 = 90;  // 2 events around the DNA operand's K1 launch
  int st;
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_T0), h->stream));

  // ---- outputs of K1/K2
  const int64_t ldc = (N + 1) & ~1LL, ldct = (M + 1) & ~1LL;
  void *pC = nullptr, *pCt = nullptr, *pnA = nullptr, *pnB = nullptr;
  if ((st = mcd_ws(h, WS_C, (size_t)M * ldc * 8, &pC))) return st;
  if ((st = mcd_ws(h, WS_CT, (size_t)N * ldct * 8, &pCt))) return st;
  if ((st = mcd_ws(h, WS_NORM_A, (size_t)M * 8, &pnA))) return st;
  if ((st = mcd_ws(h, WS_NORM_B, (size_t)N * 8, &pnB))) return st;
  double* C = static_cast<double*>(pC);
  double* Ct = static_cast<double*>(pCt);
  double* nA = static_cast<double*>(pnA);
  double* nB = static_cast<double*>(pnB);
  const int64_t ldk = precision == MCD_PREC_FP64 ? mcd_padded_k(G) : mcd_padded_k_split(G);
  void *pa = nullptr, *pb = nullptr;
  double *sA = nullptr, *sB = nullptr;
  if (precision == MCD_PREC_FP64) {
    if ((st = mcd_ws(h, WS_RNA_C, (size_t)M * ldk * 8, &pa))) return st;
    if ((st = mcd_ws(h, WS_DNA_C, (size_t)N * ldk * 8, &pb))) return st;
  } else if (precision == MCD_PREC_OZAKI_INT8) {
    void* ps = nullptr;
    if ((st = mcd_ws(h, WS_SLICES_A, (size_t)nsl * M * ldk, &pa))) return st;
    if ((st = mcd_ws(h, WS_SLICES_B, (size_t)nsl * N * ldk, &pb))) return st;
    if ((st = mcd_ws(h, WS_SCALE, (size_t)(M + N) * 8, &ps))) return st;
    sA = static_cast<double*>(ps);
    sB = sA + M;
  } else {
    if ((st = mcd_ws(h, WS_SLICES_A, (size_t)2 * M * ldk * 2, &pa))) return st;
    if ((st = mcd_ws(h, WS_SLICES_B, (size_t)2 * N * ldk * 2, &pb))) return st;
  }
  uint16_t* a_hi = static_cast<uint16_t*>(pa);
  uint16_t* a_lo = a_hi + M * ldk;
  uint16_t* b_hi = static_cast<uint16_t*>(pb);
  uint16_t* b_lo = b_hi + N * ldk;

  // ---- stage inputs.  Host inputs: the DNA operand first, then the RNA rows in chunks on the copy stream,
  //      so K1 + K2 of chunk c overlap the H2D copy of chunk c+1 (chunks are tile aligned: same results).
  const double* d_rna = rna;
  const double* d_dna = dna;
  int64_t ldr = ld_rna, ldd = ld_dna;
  int nchunk = 1;
  bool pageable_in = false;
  // gene gather indices (device copies); with a gather the staged rows keep all ld columns of the host block
  const int* d_ridx = nullptr;
  const int* d_didx = nullptr;
  if (rna_gene_idx || dna_gene_idx) {
    void* pg = nullptr;
    if ((st = mcd_ws(h, WS_GIDX, (size_t)2 * G * 4, &pg))) return st;
    int* gi = static_cast<int*>(pg);
    if (rna_gene_idx) {
      MCD_CUDA(h, cudaMemcpyAsync(gi, rna_gene_idx, (size_t)G * 4, cudaMemcpyHostToDevice, h->stream));
      d_ridx = gi;
    }
    if (dna_gene_idx) {
      MCD_CUDA(h, cudaMemcpyAsync(gi + G, dna_gene_idx, (size_t)G * 4, cudaMemcpyHostToDevice, h->stream));
      d_didx = gi + G;
    }
  }
  const int64_t wr = rna_gene_idx ? ld_rna : G;  // columns staged per RNA row
  const int64_t wd = dna_gene_idx ? ld_dna : G;
  if (in_space == MCD_MEM_HOST) {
    void *pr = nullptr, *pd = nullptr;
    if ((st = mcd_ws(h, WS_RNA_IN, (size_t)M * wr * 8, &pr))) return st;
    if ((st = mcd_ws(h, WS_DNA_IN, (size_t)N * wd * 8, &pd))) return st;
    pageable_in = mcd_is_pageable(rna) || mcd_is_pageable(dna);
    if (pageable_in) {
      if ((st = mcd_staged_h2d(h, static_cast<double*>(pd), wd, dna, ld_dna, wd, N, h->stream))) return st;
    } else {
      MCD_CUDA(h, cudaMemcpy2DAsync(pd, (size_t)wd * 8, dna, (size_t)ld_dna * 8, (size_t)wd * 8, (size_t)N,
                                    cudaMemcpyHostToDevice, h->stream));
    }
    d_rna = static_cast<const double*>(pr);
    d_dna = static_cast<const double*>(pd);
    ldr = wr;
    ldd = wd;
    const double bytes = (double)M * wr * 8;
    nchunk = (int)(bytes / (768.0 * 1024 * 1024)) + 1;
    if (nchunk > 16) nchunk = 16;
  }
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_H2D), h->stream));  // DNA operand resident
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_DNA_K1), h->stream));
  // DNA operand: K1 once
  mcd_ozaki_out ozb, oza;
  ozb.digits = static_cast<int8_t*>(pb);
  ozb.ldk8 = ldk;
  ozb.slice_stride = N * ldk;
  ozb.nsl = nsl;
  ozb.rb = rb;
  ozb.scale = sB;
  oza = ozb;
  oza.slice_stride = M * ldk;
  if (precision == MCD_PREC_FP64)
    st = mcd_launch_standardize(h, d_dna, N, G, ldd, (double*)pb, ldk, nullptr, nullptr, 0, nB, d_didx);
  else if (precision == MCD_PREC_OZAKI_INT8)
    st = mcd_launch_standardize(h, d_dna, N, G, ldd, nullptr, 0, nullptr, nullptr, 0, nB, d_didx, &ozb);
  else
    st = mcd_launch_standardize(h, d_dna, N, G, ldd, nullptr, 0, b_hi, b_lo, ldk, nB, d_didx);
  if (st) return st;
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_DNA_K1 + 1), h->stream));
  int64_t rows_per = ((M + nchunk - 1) / nchunk + 127) / 128 * 128;
  if (rows_per < 128) rows_per = 128;
  const size_t EV_CHUNK = 100;  // 4 events per chunk: copy done, K1 start, K1 end, K2 end
  int nchunk_used = 0;
  if (in_space == MCD_MEM_HOST) MCD_CUDA(h, cudaStreamWaitEvent(h->copy_stream, get_event(h, EV_T0), 0));
  for (int64_t r0 = 0; r0 < M; r0 += rows_per, ++nchunk_used) {
    const int64_t mr = (M - r0 < rows_per) ? (M - r0) : rows_per;
    const int c = nchunk_used;
    if (in_space == MCD_MEM_HOST) {
      double* dst = const_cast<double*>(d_rna) + r0 * wr;
      if (pageable_in) {
        if ((st = mcd_staged_h2d(h, dst, wr, rna + r0 * ld_rna, ld_rna, wr, mr, h->copy_stream))) return st;
      } else {
        MCD_CUDA(h, cudaMemcpy2DAsync(dst, (size_t)wr * 8, rna + r0 * ld_rna, (size_t)ld_rna * 8, (size_t)wr * 8,
                                      (size_t)mr, cudaMemcpyHostToDevice, h->copy_stream));
      }
      MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CHUNK + 4 * c), h->copy_stream));
      MCD_CUDA(h, cudaStreamWaitEvent(h->stream, get_event(h, EV_CHUNK + 4 * c), 0));
    } else {
      MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CHUNK + 4 * c), h->stream));
    }
    MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CHUNK + 4 * c + 1), h->stream));
    const double* xr = d_rna + r0 * ldr;
    if (precision == MCD_PREC_FP64) {
      double* ac = (double*)pa + r0 * ldk;
      if ((st = mcd_launch_standardize(h, xr, mr, G, ldr, ac, ldk, nullptr, nullptr, 0, nA + r0, d_ridx))) return st;
      MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CHUNK + 4 * c + 2), h->stream));
      if ((st = mcd_launch_corr_fp64(h, ac, mr, (double*)pb, N, ldk, nA + r0, nB, C + r0 * ldc, ldc, Ct + r0, ldct)))
        return st;
    } else if (precision == MCD_PREC_OZAKI_INT8) {
      oza.digits = static_cast<int8_t*>(pa) + r0 * ldk;
      oza.scale = sA + r0;
      if ((st = mcd_launch_standardize(h, xr, mr, G, ldr, nullptr, 0, nullptr, nullptr, 0, nA + r0, d_ridx, &oza)))
        return st;
      MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CHUNK + 4 * c + 2), h->stream));
      if ((st = mcd_launch_corr_ozaki(h, oza.digits, oza.slice_stride, mr, ozb.digits, ozb.slice_stride, N, ldk, nsl, rb,
                                      sA + r0, sB, nA + r0, nB, C + r0 * ldc, ldc, Ct + r0, ldct)))
        return st;
    } else {
      if ((st = mcd_launch_standardize(h, xr, mr, G, ldr, nullptr, 0, a_hi + r0 * ldk, a_lo + r0 * ldk, ldk, nA + r0,
                                       d_ridx)))
        return st;
      MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CHUNK + 4 * c + 2), h->stream));
      if ((st = mcd_launch_corr_split(h, a_hi + r0 * ldk, a_lo + r0 * ldk, mr, b_hi, b_lo, N, ldk, nA + r0, nB,
                                      C + r0 * ldc, ldc, Ct + r0, ldct)))
        return st;
    }
    MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CHUNK + 4 * c + 3), h->stream));
  }
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_STD), h->stream));
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_CORR), h->stream));

  // ---- K3 + K4
  const int64_t nsteps = mcd_num_steps(M, N);
  void* misc = nullptr;
  if ((st = mcd_ws(h, WS_MISC, step_out_bytes(M, nsteps), &misc))) return st;
  const StepOut out = carve_step_out(misc, M, nsteps);
  if (h->opt.corr_only) {
    // the caller only wants the correlation matrix resident (it will solve views of it): no step loop
    MCD_CUDA(h, cudaMemsetAsync(misc, 0, step_out_bytes(M, nsteps), h->stream));
    MCD_CUDA(h, cudaMemsetAsync(out.assign, 0xFF, (size_t)M * 4, h->stream));
    for (size_t e = 0; e <= (size_t)(nsteps < MCD_MAX_STEP_STATS ? nsteps : MCD_MAX_STEP_STATS); ++e)
      MCD_CUDA(h, cudaEventRecord(get_event(h, EV_LAP + e), h->stream));
  } else if ((st = enqueue_step_loop(h, C, ldc, Ct, ldct, M, N, out, EV_LAP, false))) {
    return st;
  }
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_LAPEND), h->stream));

  // ---- outputs
  const cudaMemcpyKind kind = out_space == MCD_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  MCD_CUDA(h, cudaMemcpyAsync(assign, out.assign, (size_t)M * 4, kind, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(step, out.step, (size_t)M * 4, kind, h->stream));
  if (step_obj) MCD_CUDA(h, cudaMemcpyAsync(step_obj, out.obj, (size_t)nsteps * 8, kind, h->stream));
  if (corr_out)
    MCD_CUDA(h, cudaMemcpy2DAsync(corr_out, (size_t)N * 8, C, (size_t)ldc * 8, (size_t)N * 8, (size_t)M, kind,
                                  h->stream));
  std::vector<mcd_lap_counters> hc((size_t)nsteps);
  std::vector<mcd_lap_cert> hcert((size_t)nsteps);
  int flag = 0;
  MCD_CUDA(h, cudaMemcpyAsync(hc.data(), out.cnt, sizeof(mcd_lap_counters) * nsteps, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(hcert.data(), out.cert, sizeof(mcd_lap_cert) * nsteps, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(&flag, h->d_flags, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemsetAsync(h->d_flags, 0, sizeof(int), h->stream));
  MCD_CUDA(h, cudaEventRecord(get_event(h, EV_D2H), h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));

  if (stats) memset(stats, 0, sizeof *stats);
  const int bad = h->opt.corr_only ? 0 : fold_step_records(h, M, N, nsteps, hc.data(), hcert.data(), stats, EV_LAP, true);
  if (stats) {
    auto el = [&](int a, int b) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, get_event(h, a), get_event(h, b));
      return (double)ms;
    };
    // K1 / K2 run per RNA chunk (interleaved with the H2D copies of the next chunk): sum the chunk spans, plus the
    // DNA operand's K1 launch.  ms_h2d is the EXPOSED copy time: everything of [T0, last K2] that is neither K1 nor K2.
    double k1 = el((int)EV_DNA_K1, (int)EV_DNA_K1 + 1), k2 = 0.0;
    for (int c = 0; c < nchunk_used; ++c) {
      k1 += el((int)EV_CHUNK + 4 * c + 1, (int)EV_CHUNK + 4 * c + 2);
      k2 += el((int)EV_CHUNK + 4 * c + 2, (int)EV_CHUNK + 4 * c + 3);
    }
    const double span = el(EV_T0, EV_CORR);
    stats->ms_standardize = k1;
    stats->ms_corr = k2;
    stats->ms_h2d = span - k1 - k2 > 0.0 ? span - k1 - k2 : 0.0;
    stats->ms_lap = el(EV_CORR, EV_LAPEND);
    stats->ms_d2h = el(EV_LAPEND, EV_D2H);
    stats->ms_total = el(EV_T0, EV_D2H);
    stats->n_steps = nsteps;
    stats->kernel_launches = h->launches - launches0;
  }
  if (flag) return mcd_fail(h, MCD_ERR_NONFINITE, "NaN or Inf in the expression / copy-number matrix");
  if ((st = step_status(h, bad))) return st;
  set_resident(h, M, N, ldc, out.assign);
  return MCD_OK;
}

// ------------------------------------------------------------------------------------------------
// Several GPUs, one caller.  SURVEY.md section 8e: K1 + K2 shard by RNA rows with no exchange inside the contraction;
// the correlation shards travel once to the first device (peer copies over NVLink), which runs the step loop.
// ------------------------------------------------------------------------------------------------
namespace {
struct ShardOperands {
  void* pa = nullptr;
  void* pb = nullptr;
  double* sA = nullptr;
  double* sB = nullptr;
  double* nA = nullptr;
  double* nB = nullptr;
};

// K1 of both operands + K2 of `rows` RNA rows on handle h; C_loc [rows, ldc] (no transpose).  All on h->stream.
int shard_standardize_correlate(mcd_context* h, const double* d_rna, int64_t ldr, const int* d_ridx, const double* d_dna,
                                int64_t ldd, const int* d_didx, int64_t rows, int64_t N, int64_t G, int precision, int nsl,
                                int rb, double* C_loc, int64_t ldc) {
  int st;
  ShardOperands o;
  void *pnA = nullptr, *pnB = nullptr;
  const int64_t ldk = precision == MCD_PREC_FP64 ? mcd_padded_k(G) : mcd_padded_k_split(G);
  if ((st = mcd_ws(h, WS_NORM_A, (size_t)(rows > 0 ? rows : 1) * 8, &pnA))) return st;
  if ((st = mcd_ws(h, WS_NORM_B, (size_t)N * 8, &pnB))) return st;
  o.nA = static_cast<double*>(pnA);
  o.nB = static_cast<double*>(pnB);
  const int64_t mr = rows > 0 ? rows : 1;
  if (precision == MCD_PREC_FP64) {
    if ((st = mcd_ws(h, WS_RNA_C, (size_t)mr * ldk * 8, &o.pa))) return st;
    if ((st = mcd_ws(h, WS_DNA_C, (size_t)N * ldk * 8, &o.pb))) return st;
    if ((st = mcd_launch_standardize(h, d_dna, N, G, ldd, (double*)o.pb, ldk, nullptr, nullptr, 0, o.nB, d_didx))) return st;
    if (rows > 0) {
      if ((st = mcd_launch_standardize(h, d_rna, rows, G, ldr, (double*)o.pa, ldk, nullptr, nullptr, 0, o.nA, d_ridx))) return st;
      st = mcd_launch_corr_fp64(h, (double*)o.pa, rows, (double*)o.pb, N, ldk, o.nA, o.nB, C_loc, ldc, nullptr, 0);
    }
  } else if (precision == MCD_PREC_OZAKI_INT8) {
    void* ps = nullptr;
    if ((st = mcd_ws(h, WS_SLICES_A, (size_t)nsl * mr * ldk, &o.pa))) return st;
    if ((st = mcd_ws(h, WS_SLICES_B, (size_t)nsl * N * ldk, &o.pb))) return st;
    if ((st = mcd_ws(h, WS_SCALE, (size_t)(mr + N) * 8, &ps))) return st;
    o.sA = static_cast<double*>(ps);
    o.sB = o.sA + mr;
    mcd_ozaki_out oza, ozb;
    ozb.digits = static_cast<int8_t*>(o.pb);
    ozb.ldk8 = ldk;
    ozb.slice_stride = N * ldk;
    ozb.nsl = nsl;
    ozb.rb = rb;
    ozb.scale = o.sB;
    oza = ozb;
    oza.digits = static_cast<int8_t*>(o.pa);
    oza.slice_stride = mr * ldk;
    oza.scale = o.sA;
    if ((st = mcd_launch_standardize(h, d_dna, N, G, ldd, nullptr, 0, nullptr, nullptr, 0, o.nB, d_didx, &ozb))) return st;
    if (rows > 0) {
      if ((st = mcd_launch_standardize(h, d_rna, rows, G, ldr, nullptr, 0, nullptr, nullptr, 0, o.nA, d_ridx, &oza))) return st;
      st = mcd_launch_corr_ozaki(h, oza.digits, oza.slice_stride, rows, ozb.digits, ozb.slice_stride, N, ldk, nsl, rb, o.sA, o.sB,
                                 o.nA, o.nB, C_loc, ldc, nullptr, 0);
    }
  } else {
    if ((st = mcd_ws(h, WS_SLICES_A, (size_t)2 * mr * ldk * 2, &o.pa))) return st;
    if ((st = mcd_ws(h, WS_SLICES_B, (size_t)2 * N * ldk * 2, &o.pb))) return st;
    uint16_t* a_hi = static_cast<uint16_t*>(o.pa);
    uint16_t* b_hi = static_cast<uint16_t*>(o.pb);
    if ((st = mcd_launch_standardize(h, d_dna, N, G, ldd, nullptr, 0, b_hi, b_hi + N * ldk, ldk, o.nB, d_didx))) return st;
    if (rows > 0) {
      if ((st = mcd_launch_standardize(h, d_rna, rows, G, ldr, nullptr, 0, a_hi, a_hi + mr * ldk, ldk, o.nA, d_ridx))) return st;
      st = mcd_launch_corr_split(h, a_hi, a_hi + mr * ldk, rows, b_hi, b_hi + N * ldk, N, ldk, o.nA, o.nB, C_loc, ldc, nullptr, 0);
    }
  }
  return st;
}
}  // namespace

int mcd_cell2cell_multi(mcd_handle* hs, int ndev, const double* rna, int64_t ld_rna, const int32_t* rna_gene_idx,
                        const double* dna, int64_t ld_dna, const int32_t* dna_gene_idx, int64_t M, int64_t N, int64_t G,
                        int precision, int32_t* assign, int32_t* step, double* step_obj, mcd_stats* stats) {
  if (!hs || ndev < 1 || !hs[0]) return MCD_ERR_INVALID;
  mcd_context* h0 = hs[0];
  if (ndev == 1)
    return mcd_cell2cell_gather(h0, rna, ld_rna, rna_gene_idx, dna, ld_dna, dna_gene_idx, M, N, G, MCD_MEM_HOST, precision,
                                assign, step, step_obj, nullptr, MCD_MEM_HOST, stats);
  for (int d = 0; d < ndev; ++d)
    if (!hs[d]) return mcd_fail(h0, MCD_ERR_INVALID, "mcd_cell2cell_multi: NULL handle");
  if (!rna || !dna || !assign || !step || M < 1 || N < 1 || G < 1 || (!rna_gene_idx && ld_rna < G) ||
      (!dna_gene_idx && ld_dna < G) || M > 0x3fffffff || N > 0x3fffffff || G > 0x7fffffff)
    return mcd_fail(h0, MCD_ERR_INVALID, "mcd_cell2cell_multi arguments");
  if (precision != MCD_PREC_FP64 && precision != MCD_PREC_SPLIT_FP16 && precision != MCD_PREC_OZAKI_INT8)
    return mcd_fail(h0, MCD_ERR_INVALID, "unknown precision");
  for (int64_t g = 0; g < G; ++g)
    if ((rna_gene_idx && (rna_gene_idx[g] < 0 || rna_gene_idx[g] >= ld_rna)) ||
        (dna_gene_idx && (dna_gene_idx[g] < 0 || dna_gene_idx[g] >= ld_dna)))
      return mcd_fail(h0, MCD_ERR_INVALID, "mcd_cell2cell_multi: gene index out of range");
  int nsl = 0, rb = 0;
  if (mcd_ozaki_format(h0, M, N, G, &nsl, &rb) != 1 && precision == MCD_PREC_OZAKI_INT8) precision = MCD_PREC_FP64;
  // hs[0]'s matrix is about to be overwritten; the other handles' WS_C slots hold shards from now on
  for (int d = 0; d < ndev; ++d) drop_resident(hs[d]);
  const int64_t ldc = (N + 1) & ~1LL, ldct = (M + 1) & ~1LL;
  const int64_t per = (M + ndev - 1) / ndev;
  const int64_t wr = rna_gene_idx ? ld_rna : G, wd = dna_gene_idx ? ld_dna : G;
  int st;
  // the whole matrix lives on the first device
  MCD_CUDA(h0, cudaSetDevice(h0->device));
  void *pC = nullptr, *pCt = nullptr;
  if ((st = mcd_ws(h0, WS_C, (size_t)M * ldc * 8, &pC))) return st;
  if ((st = mcd_ws(h0, WS_CT, (size_t)N * ldct * 8, &pCt))) return st;
  double* C = static_cast<double*>(pC);
  double* Ct = static_cast<double*>(pCt);
  const int64_t launches0 = h0->launches;
  MCD_CUDA(h0, cudaEventRecord(get_event(h0, 0), h0->stream));
  for (int d = 0; d < ndev; ++d) {
    mcd_context* h = hs[d];
    const int64_t lo = d * per < M ? d * per : M, hi = lo + per < M ? lo + per : M;
    const int64_t rows = hi - lo;
    MCD_CUDA(h0, cudaSetDevice(h->device));
    if (d > 0) {
      int can = 0;
      if (h->device != h0->device && cudaDeviceCanAccessPeer(&can, h->device, h0->device) == cudaSuccess && can) {
        cudaError_t pe = cudaDeviceEnablePeerAccess(h0->device, 0);
        if (pe != cudaSuccess) cudaGetLastError();  // already enabled
      }
    }
    void *pr = nullptr, *pd = nullptr, *pg = nullptr, *pcl = nullptr;
    if ((st = mcd_ws(h, WS_RNA_IN, (size_t)(rows > 0 ? rows : 1) * wr * 8, &pr))) return mcd_fail(h0, st, h->err.c_str());
    if ((st = mcd_ws(h, WS_DNA_IN, (size_t)N * wd * 8, &pd))) return mcd_fail(h0, st, h->err.c_str());
    const int* d_ridx = nullptr;
    const int* d_didx = nullptr;
    if (rna_gene_idx || dna_gene_idx) {
      if ((st = mcd_ws(h, WS_GIDX, (size_t)2 * G * 4, &pg))) return mcd_fail(h0, st, h->err.c_str());
      int* gi = static_cast<int*>(pg);
      if (rna_gene_idx) {
        MCD_CUDA(h0, cudaMemcpyAsync(gi, rna_gene_idx, (size_t)G * 4, cudaMemcpyHostToDevice, h->stream));
        d_ridx = gi;
      }
      if (dna_gene_idx) {
        MCD_CUDA(h0, cudaMemcpyAsync(gi + G, dna_gene_idx, (size_t)G * 4, cudaMemcpyHostToDevice, h->stream));
        d_didx = gi + G;
      }
    }
    // every device copies its RNA rows and the (small) DNA operand over its own PCIe link
    MCD_CUDA(h0, cudaMemcpy2DAsync(pd, (size_t)wd * 8, dna, (size_t)ld_dna * 8, (size_t)wd * 8, (size_t)N,
                                   cudaMemcpyHostToDevice, h->stream));
    if (rows > 0)
      MCD_CUDA(h0, cudaMemcpy2DAsync(pr, (size_t)wr * 8, rna + lo * ld_rna, (size_t)ld_rna * 8, (size_t)wr * 8, (size_t)rows,
                                     cudaMemcpyHostToDevice, h->stream));
    double* C_loc = C + lo * ldc;  // device 0 writes its shard in place
    if (d > 0) {
      if ((st = mcd_ws(h, WS_C, (size_t)(rows > 0 ? rows : 1) * ldc * 8, &pcl))) return mcd_fail(h0, st, h->err.c_str());
      C_loc = static_cast<double*>(pcl);
    } else {
      MCD_CUDA(h0, cudaStreamWaitEvent(h->stream, get_event(h0, 0), 0));
    }
    if ((st = shard_standardize_correlate(h, static_cast<const double*>(pr), wr, d_ridx, static_cast<const double*>(pd), wd,
                                          d_didx, rows, N, G, precision, nsl, rb, C_loc, ldc)))
      return mcd_fail(h0, st, h->err.c_str());
    if (d > 0 && rows > 0)
      MCD_CUDA(h0, cudaMemcpyPeerAsync(C + lo * ldc, h0->device, C_loc, h->device, (size_t)rows * ldc * 8, h->stream));
    if (d > 0) MCD_CUDA(h0, cudaEventRecord(get_event(h, 0), h->stream));
  }
  MCD_CUDA(h0, cudaSetDevice(h0->device));
  for (int d = 1; d < ndev; ++d) MCD_CUDA(h0, cudaStreamWaitEvent(h0->stream, get_event(hs[d], 0), 0));
  MCD_CUDA(h0, cudaEventRecord(get_event(h0, 3), h0->stream));
  if ((st = mcd_transpose_f64(h0, C, M, N, ldc, Ct, ldct))) return st;
  const int64_t nsteps = mcd_num_steps(M, N);
  void* misc = nullptr;
  if ((st = mcd_ws(h0, WS_MISC, step_out_bytes(M, nsteps), &misc))) return st;
  const StepOut out = carve_step_out(misc, M, nsteps);
  const size_t EV_LAP = 8;
  // check_finite: the non-finite flag K1 raises lives on the device that saw the bad value; the first solve
  // re-scans the assembled matrix so that hs[0]'s solver kernels no-op on NaN / Inf instead of iterating on them
  if ((st = enqueue_step_loop(h0, C, ldc, Ct, ldct, M, N, out, EV_LAP, true))) return st;
  MCD_CUDA(h0, cudaEventRecord(get_event(h0, 4), h0->stream));
  MCD_CUDA(h0, cudaMemcpyAsync(assign, out.assign, (size_t)M * 4, cudaMemcpyDeviceToHost, h0->stream));
  MCD_CUDA(h0, cudaMemcpyAsync(step, out.step, (size_t)M * 4, cudaMemcpyDeviceToHost, h0->stream));
  if (step_obj) MCD_CUDA(h0, cudaMemcpyAsync(step_obj, out.obj, (size_t)nsteps * 8, cudaMemcpyDeviceToHost, h0->stream));
  std::vector<mcd_lap_counters> hc((size_t)nsteps);
  std::vector<mcd_lap_cert> hcert((size_t)nsteps);
  MCD_CUDA(h0, cudaMemcpyAsync(hc.data(), out.cnt, sizeof(mcd_lap_counters) * nsteps, cudaMemcpyDeviceToHost, h0->stream));
  MCD_CUDA(h0, cudaMemcpyAsync(hcert.data(), out.cert, sizeof(mcd_lap_cert) * nsteps, cudaMemcpyDeviceToHost, h0->stream));
  MCD_CUDA(h0, cudaEventRecord(get_event(h0, 5), h0->stream));
  MCD_CUDA(h0, cudaStreamSynchronize(h0->stream));
  int flag = 0;
  for (int d = 0; d < ndev; ++d) {  // non-finite input is flagged by K1 on the device that saw it
    int f = 0;
    MCD_CUDA(h0, cudaSetDevice(hs[d]->device));
    MCD_CUDA(h0, cudaMemcpy(&f, hs[d]->d_flags, sizeof(int), cudaMemcpyDeviceToHost));
    MCD_CUDA(h0, cudaMemset(hs[d]->d_flags, 0, sizeof(int)));
    flag |= f;
  }
  MCD_CUDA(h0, cudaSetDevice(h0->device));
  if (stats) memset(stats, 0, sizeof *stats);
  const int bad = fold_step_records(h0, M, N, nsteps, hc.data(), hcert.data(), stats, EV_LAP, true);
  if (stats) {
    auto el = [&](int a, int b) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, get_event(h0, a), get_event(h0, b));
      return (double)ms;
    };
    stats->ms_corr = el(0, 3);  // H2D + K1 + K2 + shard transfer, all devices (overlapped)
    stats->ms_lap = el(3, 4);
    stats->ms_d2h = el(4, 5);
    stats->ms_total = el(0, 5);
    stats->n_steps = nsteps;
    int64_t launches = h0->launches - launches0;
    stats->kernel_launches = launches;
  }
  if (flag) return mcd_fail(h0, MCD_ERR_NONFINITE, "NaN or Inf in the expression / copy-number matrix");
  if ((st = step_status(h0, bad))) return st;
  set_resident(h0, M, N, ldc, out.assign);
  return MCD_OK;
}

int mcd_corr_rows(mcd_handle h, const int32_t* rows, int64_t nrows, double* out, int out_space) {
  if (!h) return MCD_ERR_INVALID;
  if (!rows || !out || nrows < 1 || !has_matrix(h))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_corr_rows: no mcd_cell2cell result is resident");
  for (int64_t i = 0; i < nrows; ++i)
    if (rows[i] < 0 || rows[i] >= h->last_M) return mcd_fail(h, MCD_ERR_INVALID, "mcd_corr_rows: row out of range");
  MCD_CUDA(h, cudaSetDevice(h->device));
  const int64_t N = h->last_N;
  void* pi = nullptr;
  void* po = nullptr;
  int st;
  if ((st = mcd_ws(h, WS_SUB_IDX, (size_t)nrows * 4, &pi))) return st;
  MCD_CUDA(h, cudaMemcpyAsync(pi, rows, (size_t)nrows * 4, cudaMemcpyHostToDevice, h->stream));
  double* dst = out;
  if (out_space != MCD_MEM_DEVICE) {
    if ((st = mcd_ws(h, WS_SUB_C, (size_t)nrows * N * 8, &po))) return st;
    dst = static_cast<double*>(po);
  }
  dim3 grid((unsigned)((N + 1023) / 1024 < 64 ? (N + 1023) / 1024 : 64), grid_rows(nrows));
  gather_rows_out_kernel<<<grid, 256, 0, h->stream>>>(static_cast<const double*>(h->ws[WS_C].ptr), h->last_ldc,
                                                      static_cast<const int*>(pi), nrows, N, dst);
  MCD_LAUNCH_CHECK(h, "gather_rows_out_kernel");
  if (out_space != MCD_MEM_DEVICE)
    MCD_CUDA(h, cudaMemcpyAsync(out, dst, (size_t)nrows * N * 8, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  return MCD_OK;
}

int mcd_corr_pairs(mcd_handle h, const int32_t* rows, const int32_t* cols, int64_t n, double* out) {
  if (!h) return MCD_ERR_INVALID;
  if (!rows || !cols || !out || n < 1 || !has_matrix(h))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_corr_pairs: no mcd_cell2cell result is resident");
  for (int64_t k = 0; k < n; ++k)
    if (rows[k] < 0 || rows[k] >= h->last_M || cols[k] < 0 || cols[k] >= h->last_N)
      return mcd_fail(h, MCD_ERR_INVALID, "mcd_corr_pairs: index out of range");
  MCD_CUDA(h, cudaSetDevice(h->device));
  void* pi = nullptr;
  void* po = nullptr;
  int st;
  if ((st = mcd_ws(h, WS_SUB_IDX, (size_t)n * 8, &pi))) return st;
  if ((st = mcd_ws(h, WS_SUB_MISC, (size_t)n * 8, &po))) return st;
  int* d_r = static_cast<int*>(pi);
  int* d_c = d_r + n;
  MCD_CUDA(h, cudaMemcpyAsync(d_r, rows, (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(d_c, cols, (size_t)n * 4, cudaMemcpyHostToDevice, h->stream));
  gather_pairs_kernel<<<(unsigned)((n + 255) / 256), 256, 0, h->stream>>>(static_cast<const double*>(h->ws[WS_C].ptr),
                                                                        h->last_ldc, d_r, d_c, n,
                                                                        static_cast<double*>(po));
  MCD_LAUNCH_CHECK(h, "gather_pairs_kernel");
  MCD_CUDA(h, cudaMemcpyAsync(out, po, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  return MCD_OK;
}

static int subinstance_steps_impl(mcd_handle h, const int32_t* rna_rows, int64_t m_sub, const int32_t* dna_cols,
                                  int64_t n_sub, int32_t* assign, int32_t* step, double* step_obj, int out_space,
                                  mcd_stats* stats, bool use_classes, int* bad_out);

int mcd_subinstance_steps(mcd_handle h, const int32_t* rna_rows, int64_t m_sub, const int32_t* dna_cols, int64_t n_sub,
                          int32_t* assign, int32_t* step, double* step_obj, int out_space, mcd_stats* stats) {
  int bad = 0;
  int st = subinstance_steps_impl(h, rna_rows, m_sub, dna_cols, n_sub, assign, step, step_obj, out_space, stats, true, &bad);
  if (st == MCD_ERR_NOT_CONVERGED && (bad & 4)) {
    // The class treatment of duplicated cells leaves one window open (two copies settling at different levels in the
    // very round a third party buys the dearer copy's object); the certificate catches it.  Such a replicate is
    // solved again with every copy as a person of its own: exact ties then stall the auction and the
    // augmenting-path kernel finishes them -- slower, never wrong.
    st = subinstance_steps_impl(h, rna_rows, m_sub, dna_cols, n_sub, assign, step, step_obj, out_space, stats, false, &bad);
  }
  return st;
}

static int subinstance_steps_impl(mcd_handle h, const int32_t* rna_rows, int64_t m_sub, const int32_t* dna_cols,
                                  int64_t n_sub, int32_t* assign, int32_t* step, double* step_obj, int out_space,
                                  mcd_stats* stats, bool use_classes, int* bad_out) {
  if (!h) return MCD_ERR_INVALID;
  if (!assign || !step || m_sub < 1 || n_sub < 1 || !has_matrix(h))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_steps: no mcd_cell2cell result is resident");
  if ((!rna_rows && m_sub != h->last_M) || (!dna_cols && n_sub != h->last_N))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_steps: NULL index means all rows / columns");
  for (int64_t i = 0; rna_rows && i < m_sub; ++i)
    if (rna_rows[i] < 0 || rna_rows[i] >= h->last_M)
      return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_steps: RNA row out of range");
  for (int64_t j = 0; dna_cols && j < n_sub; ++j)
    if (dna_cols[j] < 0 || dna_cols[j] >= h->last_N)
      return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_steps: DNA column out of range");
  MCD_CUDA(h, cudaSetDevice(h->device));
  int st;
  const int64_t lds = (n_sub + 1) & ~1LL, ldst = (m_sub + 1) & ~1LL;
  void *pc = nullptr, *pct = nullptr, *pi = nullptr, *misc = nullptr;
  if ((st = mcd_ws(h, WS_SUB_C, (size_t)m_sub * lds * 8, &pc))) return st;
  if ((st = mcd_ws(h, WS_SUB_CT, (size_t)n_sub * ldst * 8, &pct))) return st;
  if ((st = mcd_ws(h, WS_SUB_IDX, (size_t)(m_sub + 2 * n_sub) * 4, &pi))) return st;
  int* d_rows = rna_rows ? static_cast<int*>(pi) : nullptr;
  int* d_cols = dna_cols ? static_cast<int*>(pi) + m_sub : nullptr;
  int* d_cls = nullptr;
  if (rna_rows) MCD_CUDA(h, cudaMemcpyAsync(d_rows, rna_rows, (size_t)m_sub * 4, cudaMemcpyHostToDevice, h->stream));
  if (dna_cols) MCD_CUDA(h, cudaMemcpyAsync(d_cols, dna_cols, (size_t)n_sub * 4, cudaMemcpyHostToDevice, h->stream));
  // copies of a DNA cell (resampling with replacement): identical columns, i.e. exact ties by construction.  They
  // are told to the solver as classes of similar persons.
  std::vector<int> cls;
  if (use_classes && dna_cols && duplicate_classes(dna_cols, n_sub, cls) > 0) {
    d_cls = static_cast<int*>(pi) + m_sub + n_sub;
    MCD_CUDA(h, cudaMemcpyAsync(d_cls, cls.data(), (size_t)n_sub * 4, cudaMemcpyHostToDevice, h->stream));
  }
  const int64_t launches0 = h->launches;
  const size_t EV_LAP = 8;
  MCD_CUDA(h, cudaEventRecord(get_event(h, 6), h->stream));
  double* subC = static_cast<double*>(pc);
  double* subCt = static_cast<double*>(pct);
  {
    dim3 grid((unsigned)((n_sub + 1023) / 1024 < 64 ? (n_sub + 1023) / 1024 : 64), grid_rows(m_sub));
    gather_sub_kernel<<<grid, 256, 0, h->stream>>>(static_cast<const double*>(h->ws[WS_C].ptr), h->last_ldc, d_rows,
                                                   d_cols, m_sub, n_sub, subC, lds);
    MCD_LAUNCH_CHECK(h, "gather_sub_kernel");
  }
  if ((st = mcd_transpose_f64(h, subC, m_sub, n_sub, lds, subCt, ldst))) return st;
  const int64_t nsteps = mcd_num_steps(m_sub, n_sub);
  if ((st = mcd_ws(h, WS_SUB_MISC, step_out_bytes(m_sub, nsteps), &misc))) return st;
  const StepOut out = carve_step_out(misc, m_sub, nsteps);
  if ((st = enqueue_step_loop(h, subC, lds, subCt, ldst, m_sub, n_sub, out, EV_LAP, false, true, d_cls))) return st;
  MCD_CUDA(h, cudaEventRecord(get_event(h, 7), h->stream));
  const cudaMemcpyKind kind = out_space == MCD_MEM_DEVICE ? cudaMemcpyDeviceToDevice : cudaMemcpyDeviceToHost;
  MCD_CUDA(h, cudaMemcpyAsync(assign, out.assign, (size_t)m_sub * 4, kind, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(step, out.step, (size_t)m_sub * 4, kind, h->stream));
  if (step_obj) MCD_CUDA(h, cudaMemcpyAsync(step_obj, out.obj, (size_t)nsteps * 8, kind, h->stream));
  std::vector<mcd_lap_counters> hc((size_t)nsteps);
  std::vector<mcd_lap_cert> hcert((size_t)nsteps);
  MCD_CUDA(h, cudaMemcpyAsync(hc.data(), out.cnt, sizeof(mcd_lap_counters) * nsteps, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpyAsync(hcert.data(), out.cert, sizeof(mcd_lap_cert) * nsteps, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  if (stats) memset(stats, 0, sizeof *stats);
  const int bad = fold_step_records(h, m_sub, n_sub, nsteps, hc.data(), hcert.data(), stats, EV_LAP, true);
  if (stats) {
    float ms = 0.f;
    cudaEventElapsedTime(&ms, get_event(h, 6), get_event(h, 7));
    stats->ms_lap = ms;
    stats->ms_total = ms;
    stats->n_steps = nsteps;
    stats->kernel_launches = h->launches - launches0;
  }
  if (bad_out) *bad_out = bad | ((bad & 2) && d_cls != nullptr ? 4 : 0);  // bit 2: certificate failed WITH classes in use
  return step_status(h, bad);
}

// worker k of a handle (created on first use)
static int sweep_worker(mcd_context* h, size_t k, mcd_context** out) {
  while (h->workers.size() <= k) {
    mcd_context* w = new (std::nothrow) mcd_context();
    if (w == nullptr) return mcd_fail(h, MCD_ERR_NOMEM, "worker context");
    w->device = h->device;
    w->sm_count = h->sm_count;
    cudaError_t e = cudaStreamCreateWithFlags(&w->stream, cudaStreamNonBlocking);
    if (e == cudaSuccess) e = cudaMalloc(&w->d_flags, 64);
    if (e == cudaSuccess) e = cudaMemsetAsync(w->d_flags, 0, 64, w->stream);
    if (e != cudaSuccess) {
      mcd_destroy(w);
      return mcd_fail(h, MCD_ERR_CUDA, "worker context", e);
    }
    h->workers.push_back(w);
  }
  *out = h->workers[k];
  return MCD_OK;
}

// The replicate sweep engine shared by mcd_subinstance_sweep and mcd_loo_sweep and their _multi forms.  Replicates are
// independent step loops of one shape (m_sub rows, n_sub columns); what makes one replicate differ from the next comes
// in as hooks.
struct SweepPlan {
  int K;              // worker contexts (replicates in flight) per handle
  int64_t nsteps;     // steps of every replicate
  int64_t batch;      // replicates per batch
  size_t step_bytes;  // the replicate's StepOut block (256-byte aligned)
  size_t rep_bytes;   // step_bytes + the caller's extra bytes per replicate
};

static SweepPlan sweep_plan(int64_t nrep, int64_t m_sub, int64_t n_sub, size_t extra_rep_bytes, int concurrency) {
  SweepPlan p;
  p.K = concurrency < 1 ? 8 : concurrency;
  if (p.K > 32) p.K = 32;
  if ((int64_t)p.K > nrep) p.K = (int)nrep;
  p.nsteps = mcd_num_steps(m_sub, n_sub);
  p.step_bytes = (step_out_bytes(m_sub, p.nsteps) + 255) / 256 * 256;
  p.rep_bytes = p.step_bytes + (extra_rep_bytes + 255) / 256 * 256;
  p.batch = (int64_t)((size_t)1 << 30) / (int64_t)p.rep_bytes;  // <= 1 GiB of per-replicate outputs at a time
  if (p.batch < p.K) p.batch = p.K;
  if (p.batch > nrep) p.batch = nrep;
  return p;
}

// Every hook is called with the handle that owns the batch, h = hs[d], and its index d: a hook reads that handle's
// resident matrix (its own copy) and that handle's uploads, never another handle's.
struct SweepHooks {
  // on h->stream before the replicates of the batch [r0, r0 + nb) are dealt (uploads of the batch's indices); optional
  std::function<int(mcd_context* h, int d, int64_t r0, int64_t nb)> prepare;
  // on worker w's stream, from w's host thread: cost block subC [m_sub, lds] and its transpose subCt [n_sub, ldst] of
  // replicate r0 + b; *dna_class = DEVICE classes of duplicated DNA cells (see enqueue_step_loop) or NULL
  std::function<int(mcd_context* h, int d, mcd_context* w, int64_t r0, int64_t b, double* subC, int64_t lds,
                    double* subCt, int64_t ldst, const int** dna_class)>
      build;
  // on h->stream after the workers joined, before the outputs go to the host: replicate b of the batch has its block
  // at out + b * rep_bytes (StepOut first, the caller's extra bytes from step_bytes on); optional
  std::function<int(mcd_context* h, int d, int64_t r0, int64_t nb, char* out)> after;
  // on the host once the batch synchronised, per replicate r = r0 + b: status bits and certificate gap in / out (a
  // replicate may be solved again, on h); stats = h's share of the call's stats or NULL; optional
  std::function<int(mcd_context* h, int d, int64_t r, int64_t b, int& bad, double& gap, mcd_stats* stats)> redo;
};

// What one handle did in a sweep.
struct SweepShare {
  int bad = 0;                 // OR of the replicates' status bits
  double enqueue_ms = 0.0;     // wall time of the enqueuing phases of its batches
  int64_t launches = 0;        // kernels launched by the handle and its workers
  int64_t last_r0 = -1;        // first replicate of the last batch it solved
};

// The batch loop of handle hs[d]: batches [r0, r0 + batch) are claimed from `next_batch` until none is left or `stop`
// is raised.  With one handle it runs on the caller's thread; with several, each handle has a host thread of its own.
static int sweep_handle(mcd_context* const* hs, int d, const SweepPlan& P, int64_t batch, int64_t nrep, int64_t m_sub,
                        int64_t n_sub, int32_t* assign, int32_t* step, double* step_obj, double* cert_gap,
                        mcd_stats* stats, const SweepHooks& hk, std::atomic<int64_t>& next_batch,
                        std::atomic<bool>& stop, SweepShare& share) {
  mcd_context* h = hs[d];
  const int K = P.K;
  const int64_t nsteps = P.nsteps;
  const size_t rep_bytes = P.rep_bytes;
  int st;
  MCD_CUDA(h, cudaSetDevice(h->device));
  void* p_out = nullptr;
  if ((st = mcd_ws(h, WS_SWEEP_OUT, (size_t)batch * rep_bytes, &p_out))) return st;
  const int64_t lds = (n_sub + 1) & ~1LL, ldst = (m_sub + 1) & ~1LL;
  // every worker solves on a slice of the chip: the cooperative grid of the wide rounds is capped so that K of them
  // are co-resident (the narrow rounds run on one 8- or 16-CTA cluster per solve anyway).  That slice depends on the
  // device's SM count and K alone, so a replicate gets the same grid on every device of the same kind.
  std::vector<mcd_context*> ws((size_t)K);
  const int total_blocks = h->sm_count * (h->opt.lap_blocks_per_sm < 1 ? 1 : h->opt.lap_blocks_per_sm);
  for (int k = 0; k < K; ++k) {
    if ((st = sweep_worker(h, (size_t)k, &ws[k]))) return st;
    ws[k]->opt = h->opt;
    ws[k]->launches = 0;
    if (h->opt.lap_grid_blocks <= 0) {
      int gb = total_blocks / K;
      ws[k]->opt.lap_grid_blocks = gb < 16 ? 16 : gb;
    }
  }
  const int64_t launches0 = h->launches;
  std::vector<mcd_lap_counters> hc((size_t)(nsteps * batch));
  std::vector<mcd_lap_cert> hcert((size_t)(nsteps * batch));
  for (;;) {
    if (stop.load()) break;
    const int64_t r0 = next_batch.fetch_add(1) * batch;
    if (r0 >= nrep) break;
    const int64_t nb = nrep - r0 < batch ? nrep - r0 : batch;
    if (hk.prepare && (st = hk.prepare(h, d, r0, nb))) return st;
    MCD_CUDA(h, cudaEventRecord(get_event(h, 5), h->stream));
    for (int k = 0; k < K; ++k) MCD_CUDA(h, cudaStreamWaitEvent(ws[k]->stream, get_event(h, 5), 0));
    // Replicates differ a lot in cost (a resampled replicate with a starved clone needs 10x the rounds of a balanced
    // one), so they are dealt dynamically from a shared counter.  Every worker has its own HOST thread: a cooperative /
    // cluster launch may block its caller until the stream's earlier work has drained (measured: with one enqueuing
    // thread 75 % of the sweep's wall time was spent inside launch calls and the workers starved), and the runtime is
    // thread-safe.  A thread keeps at most two replicates queued on its stream.
    const auto host_t0 = std::chrono::steady_clock::now();
    std::atomic<int64_t> next_rep(0);
    std::vector<int> wstatus((size_t)K, 0);
    auto worker_main = [&](int k) {
      mcd_context* w = ws[(size_t)k];
      if (cudaSetDevice(h->device) != cudaSuccess) {
        wstatus[(size_t)k] = MCD_ERR_CUDA;
        return;
      }
      int issued = 0;
      for (;;) {
        const int64_t b = next_rep.fetch_add(1);
        if (b >= nb) break;
        if (issued >= 2) cudaEventSynchronize(get_event(w, 1 + (size_t)(issued & 1)));  // replicate issued - 2 is done
        int stw;
        void *pc = nullptr, *pct = nullptr;
        if ((stw = mcd_ws(w, WS_SUB_C, (size_t)m_sub * lds * 8, &pc)) ||
            (stw = mcd_ws(w, WS_SUB_CT, (size_t)n_sub * ldst * 8, &pct))) {
          wstatus[(size_t)k] = stw;
          return;
        }
        double* subC = static_cast<double*>(pc);
        double* subCt = static_cast<double*>(pct);
        const int* dna_class = nullptr;
        const StepOut out = carve_step_out(static_cast<char*>(p_out) + (size_t)b * rep_bytes, m_sub, nsteps);
        if ((stw = hk.build(h, d, w, r0, b, subC, lds, subCt, ldst, &dna_class)) ||
            (stw = enqueue_step_loop(w, subC, lds, subCt, ldst, m_sub, n_sub, out, 0, false, false, dna_class))) {
          wstatus[(size_t)k] = stw;
          return;
        }
        cudaEventRecord(get_event(w, 1 + (size_t)(issued & 1)), w->stream);
        issued++;
      }
    };
    for (int k = 0; k < K; ++k) {  // events are created on the calling thread (get_event grows a vector)
      get_event(ws[(size_t)k], 0);
      get_event(ws[(size_t)k], 1);
      get_event(ws[(size_t)k], 2);
    }
    {
      std::vector<std::thread> threads;
      for (int k = 1; k < K; ++k) threads.emplace_back(worker_main, k);
      worker_main(0);
      for (auto& t : threads) t.join();
    }
    for (int k = 0; k < K; ++k)
      if (wstatus[(size_t)k]) return mcd_fail(h, wstatus[(size_t)k], ws[(size_t)k]->err.c_str());
    share.enqueue_ms += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - host_t0).count();
    for (int k = 0; k < K; ++k) {
      MCD_CUDA(h, cudaEventRecord(get_event(ws[k], 0), ws[k]->stream));
      MCD_CUDA(h, cudaStreamWaitEvent(h->stream, get_event(ws[k], 0), 0));
    }
    if (hk.after && (st = hk.after(h, d, r0, nb, static_cast<char*>(p_out)))) return st;
    // results of the batch: strided device block -> dense host arrays
    const StepOut o0 = carve_step_out(p_out, m_sub, nsteps);
    if (assign)
      MCD_CUDA(h, cudaMemcpy2DAsync(assign + r0 * m_sub, (size_t)m_sub * 4, o0.assign, rep_bytes, (size_t)m_sub * 4,
                                    (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
    if (step)
      MCD_CUDA(h, cudaMemcpy2DAsync(step + r0 * m_sub, (size_t)m_sub * 4, o0.step, rep_bytes, (size_t)m_sub * 4,
                                    (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
    if (step_obj)
      MCD_CUDA(h, cudaMemcpy2DAsync(step_obj + r0 * nsteps, (size_t)nsteps * 8, o0.obj, rep_bytes, (size_t)nsteps * 8,
                                    (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
    MCD_CUDA(h, cudaMemcpy2DAsync(hc.data(), sizeof(mcd_lap_counters) * nsteps, o0.cnt, rep_bytes,
                                  sizeof(mcd_lap_counters) * nsteps, (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
    MCD_CUDA(h, cudaMemcpy2DAsync(hcert.data(), sizeof(mcd_lap_cert) * nsteps, o0.cert, rep_bytes,
                                  sizeof(mcd_lap_cert) * nsteps, (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
    MCD_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int64_t b = 0; b < nb; ++b) {
      const mcd_lap_cert* rc = hcert.data() + b * nsteps;
      int bad_b = fold_step_records(h, m_sub, n_sub, nsteps, hc.data() + b * nsteps, rc, stats, 0, false);
      double g = 0.0;
      for (int64_t s2 = 0; s2 < nsteps; ++s2) g = rc[s2].rel_gap > g ? rc[s2].rel_gap : g;
      if (hk.redo && (st = hk.redo(h, d, r0 + b, b, bad_b, g, stats))) return st;
      share.bad |= bad_b;
      if (cert_gap) cert_gap[r0 + b] = h->opt.certify ? g : -1.0;
    }
    if (r0 > share.last_r0) share.last_r0 = r0;
  }
  share.launches = h->launches - launches0;
  for (int k = 0; k < K; ++k) share.launches += ws[k]->launches;
  return MCD_OK;
}

// Replicates [0, nrep) over the handles hs[0..ndev).  One handle: its batch loop on the calling thread, timed with its
// events.  Several: one host thread per handle, batches claimed from one counter, the solver options of hs[0] on every
// handle for the duration of the call, stats merged (counters summed, certificate figures the maximum, per-step
// figures those of the handle that solved the last batch, times the host wall clock of the whole call).
static int sweep_replicates(mcd_context* const* hs, int ndev, const SweepPlan& P, int64_t nrep, int64_t m_sub,
                            int64_t n_sub, int32_t* assign, int32_t* step, double* step_obj, double* cert_gap,
                            mcd_stats* stats, const SweepHooks& hk) {
  mcd_context* h0 = hs[0];
  std::atomic<int64_t> next_batch(0);
  std::atomic<bool> stop(false);
  if (stats) memset(stats, 0, sizeof *stats);
  if (ndev == 1) {
    SweepShare share;
    MCD_CUDA(h0, cudaSetDevice(h0->device));
    // (events 6 / 7 and 8 .. 8 + steps belong to mcd_subinstance_steps, which the class-free re-solve of a replicate
    //  runs on this handle: the sweep times itself with events of its own)
    MCD_CUDA(h0, cudaEventRecord(get_event(h0, 96), h0->stream));
    int st = sweep_handle(hs, 0, P, P.batch, nrep, m_sub, n_sub, assign, step, step_obj, cert_gap, stats, hk, next_batch,
                          stop, share);
    if (st) return st;
    MCD_CUDA(h0, cudaEventRecord(get_event(h0, 97), h0->stream));
    MCD_CUDA(h0, cudaStreamSynchronize(h0->stream));
    if (stats) {
      float ms = 0.f;
      cudaEventElapsedTime(&ms, get_event(h0, 96), get_event(h0, 97));
      stats->ms_lap = ms;
      stats->ms_total = ms;
      stats->ms_h2d = share.enqueue_ms;  // wall time of the enqueuing phase of every batch
      stats->n_steps = P.nsteps;
      stats->kernel_launches = share.launches;
    }
    return step_status(h0, share.bad);
  }
  // Batches small enough that the last ones do not run on one device alone: about four per device
  // (ceil(nrep / (4 ndev)) replicates), never fewer than the K workers of the device that claims one, never more than
  // the 1 GiB cap of the plan.
  int64_t batch = (nrep + 4 * (int64_t)ndev - 1) / (4 * (int64_t)ndev);
  if (batch < P.K) batch = P.K;
  if (batch > P.batch) batch = P.batch;
  std::vector<SweepShare> share((size_t)ndev);
  std::vector<mcd_stats> dstats((size_t)ndev);
  std::vector<int> dst((size_t)ndev, MCD_OK);
  std::vector<mcd_options> saved((size_t)ndev);
  for (int d = 0; d < ndev; ++d) {
    memset(&dstats[(size_t)d], 0, sizeof(mcd_stats));
    saved[(size_t)d] = hs[d]->opt;
    hs[d]->opt = h0->opt;
  }
  const auto t0 = std::chrono::steady_clock::now();
  auto run = [&](int d) {
    int st = sweep_handle(hs, d, P, batch, nrep, m_sub, n_sub, assign, step, step_obj, cert_gap,
                          stats ? &dstats[(size_t)d] : nullptr, hk, next_batch, stop, share[(size_t)d]);
    if (st == MCD_OK) {
      const cudaError_t e = cudaStreamSynchronize(hs[d]->stream);
      if (e != cudaSuccess) st = mcd_fail(hs[d], MCD_ERR_CUDA, "cudaStreamSynchronize", e);
    }
    if (st != MCD_OK) stop = true;  // the other handles claim no further batch
    dst[(size_t)d] = st;
  };
  {
    std::vector<std::thread> threads;
    for (int d = 1; d < ndev; ++d) threads.emplace_back(run, d);
    run(0);
    for (auto& t : threads) t.join();
  }
  const double wall_ms = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
  for (int d = 0; d < ndev; ++d) hs[d]->opt = saved[(size_t)d];
  cudaSetDevice(h0->device);
  for (int d = 0; d < ndev; ++d)
    if (dst[(size_t)d] != MCD_OK) return d == 0 ? dst[0] : mcd_fail(h0, dst[(size_t)d], hs[d]->err.c_str());
  int bad = 0;
  int last = 0;
  for (int d = 0; d < ndev; ++d) {
    bad |= share[(size_t)d].bad;
    if (share[(size_t)d].last_r0 > share[(size_t)last].last_r0) last = d;
  }
  if (stats) {
    const mcd_stats& L = dstats[(size_t)last];
    memcpy(stats->step_rounds, L.step_rounds, sizeof L.step_rounds);
    memcpy(stats->step_bids, L.step_bids, sizeof L.step_bids);
    memcpy(stats->step_cert_gap, L.step_cert_gap, sizeof L.step_cert_gap);
    for (int d = 0; d < ndev; ++d) {
      const mcd_stats& s = dstats[(size_t)d];
      stats->lap_rounds += s.lap_rounds;
      stats->lap_bids += s.lap_bids;
      stats->lap_bytes += s.lap_bytes;
      stats->lap_aug_rows += s.lap_aug_rows;
      stats->lap_aug_steps += s.lap_aug_steps;
      for (int q = 0; q < 8; ++q) stats->lap_cycles[q] += s.lap_cycles[q];
      stats->cert_bad += s.cert_bad;
      stats->cert_steps += s.cert_steps;
      stats->sweep_fallbacks += s.sweep_fallbacks;
      if (s.cert_rel_gap > stats->cert_rel_gap) stats->cert_rel_gap = s.cert_rel_gap;
      if (s.cert_max_violation > stats->cert_max_violation) stats->cert_max_violation = s.cert_max_violation;
      if (share[(size_t)d].enqueue_ms > stats->ms_h2d) stats->ms_h2d = share[(size_t)d].enqueue_ms;
      stats->kernel_launches += share[(size_t)d].launches;
    }
    stats->ms_lap = wall_ms;
    stats->ms_total = wall_ms;
    stats->n_steps = P.nsteps;
  }
  return step_status(h0, bad);
}

// Handles of a call: hs[0..ndev) non-NULL and pairwise distinct (one context named twice would be driven by two host
// threads at once).  Separate contexts on one device are fine.
static int check_distinct_handles(mcd_context* const* hs, int ndev, const char* what) {
  char buf[256];
  for (int d = 0; d < ndev; ++d) {
    if (!hs[d]) {
      snprintf(buf, sizeof buf, "%s: handle %d is NULL", what, d);
      return mcd_fail(hs[0], MCD_ERR_INVALID, buf);
    }
    for (int e = 0; e < d; ++e)
      if (hs[e] == hs[d]) {
        snprintf(buf, sizeof buf, "%s: handles %d and %d are the same context (a handle may be listed once)", what, e, d);
        return mcd_fail(hs[0], MCD_ERR_INVALID, buf);
      }
  }
  return MCD_OK;
}

// Handles of a multi-device view call: distinct, hs[0] holds a resident matrix and every other handle a copy of that
// same run's matrix (mcd_share_resident since hs[0]'s last run).
static int check_view_handles(mcd_context* const* hs, int ndev, const char* what) {
  int st;
  if ((st = check_distinct_handles(hs, ndev, what))) return st;
  char buf[320];
  if (!has_matrix(hs[0])) {
    snprintf(buf, sizeof buf, "%s: no mcd_cell2cell result is resident on handle 0", what);
    return mcd_fail(hs[0], MCD_ERR_INVALID, buf);
  }
  for (int d = 1; d < ndev; ++d)
    if (hs[d]->gen != hs[0]->gen || hs[d]->last_M != hs[0]->last_M || hs[d]->last_N != hs[0]->last_N) {
      snprintf(buf, sizeof buf,
               "%s: handle %d holds no copy of handle 0's current resident matrix (call mcd_share_resident after "
               "every run on handle 0)", what, d);
      return mcd_fail(hs[0], MCD_ERR_INVALID, buf);
    }
  return MCD_OK;
}

static int subinstance_sweep_impl(mcd_context* const* hs, int ndev, int64_t nrep, const int32_t* rna_rows,
                                  int64_t m_sub, const int32_t* dna_cols, int64_t n_sub, int32_t* assign, int32_t* step,
                                  double* step_obj, double* cert_gap, int concurrency, mcd_stats* stats) {
  mcd_context* h = hs[0];
  if (!assign || !step || !dna_cols || nrep < 1 || m_sub < 1 || n_sub < 1 || !has_matrix(h))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_sweep: no mcd_cell2cell result is resident / bad arguments");
  if (!rna_rows && m_sub != h->last_M)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_sweep: NULL rna_rows means all rows");
  for (int64_t i = 0; rna_rows && i < m_sub; ++i)
    if (rna_rows[i] < 0 || rna_rows[i] >= h->last_M)
      return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_sweep: RNA row out of range");
  for (int64_t j = 0; j < nrep * n_sub; ++j)
    if (dna_cols[j] < 0 || dna_cols[j] >= h->last_N)
      return mcd_fail(h, MCD_ERR_INVALID, "mcd_subinstance_sweep: DNA column out of range");
  const SweepPlan P = sweep_plan(nrep, m_sub, n_sub, 0, concurrency);
  const int64_t batch = P.batch, nsteps = P.nsteps;
  // per handle: the shared RNA rows, the batch's DNA columns and their duplicate classes (device and host)
  struct Dev {
    int* d_rows;
    int* d_cols;
    int* d_clss;
    std::vector<int> clss, cls1;
    std::vector<int64_t> n_extra;
  };
  std::vector<Dev> dev((size_t)ndev);
  for (int d = 0; d < ndev; ++d) {
    mcd_context* hd = hs[d];
    Dev& v = dev[(size_t)d];
    int st;
    MCD_CUDA(h, cudaSetDevice(hd->device));
    void* p_idx = nullptr;
    if ((st = mcd_ws(hd, WS_SWEEP_IDX, (size_t)(m_sub + 2 * batch * n_sub) * 4, &p_idx)))
      return d == 0 ? st : mcd_fail(h, st, hd->err.c_str());
    v.d_rows = rna_rows ? static_cast<int*>(p_idx) : nullptr;
    v.d_cols = static_cast<int*>(p_idx) + m_sub;
    v.d_clss = v.d_cols + batch * n_sub;
    v.clss.resize((size_t)(batch * n_sub));
    v.n_extra.resize((size_t)batch);
    if (rna_rows)
      MCD_CUDA(h, cudaMemcpyAsync(v.d_rows, rna_rows, (size_t)m_sub * 4, cudaMemcpyHostToDevice, hd->stream));
  }
  SweepHooks hk;
  hk.prepare = [&](mcd_context* hd, int d, int64_t r0, int64_t nb) -> int {
    Dev& v = dev[(size_t)d];
    MCD_CUDA(hd, cudaMemcpyAsync(v.d_cols, dna_cols + r0 * n_sub, (size_t)nb * n_sub * 4, cudaMemcpyHostToDevice,
                                 hd->stream));
    for (int64_t b = 0; b < nb; ++b) {
      v.n_extra[(size_t)b] = duplicate_classes(dna_cols + (r0 + b) * n_sub, n_sub, v.cls1);
      std::copy(v.cls1.begin(), v.cls1.end(), v.clss.begin() + b * n_sub);
    }
    MCD_CUDA(hd, cudaMemcpyAsync(v.d_clss, v.clss.data(), (size_t)nb * n_sub * 4, cudaMemcpyHostToDevice, hd->stream));
    return MCD_OK;
  };
  hk.build = [&](mcd_context* hd, int d, mcd_context* w, int64_t, int64_t b, double* subC, int64_t lds, double* subCt,
                 int64_t ldst, const int** dna_class) -> int {
    const Dev& v = dev[(size_t)d];
    dim3 grid((unsigned)((n_sub + 1023) / 1024 < 64 ? (n_sub + 1023) / 1024 : 64), grid_rows(m_sub));
    gather_sub_kernel<<<grid, 256, 0, w->stream>>>(static_cast<const double*>(hd->ws[WS_C].ptr), hd->last_ldc, v.d_rows,
                                                   v.d_cols + b * n_sub, m_sub, n_sub, subC, lds);
    MCD_LAUNCH_CHECK(w, "gather_sub_kernel");
    *dna_class = v.n_extra[(size_t)b] > 0 ? v.d_clss + b * n_sub : nullptr;
    return mcd_transpose_f64(w, subC, m_sub, n_sub, lds, subCt, ldst);
  };
  hk.redo = [&](mcd_context* hd, int d, int64_t r, int64_t b, int& bad_b, double& g, mcd_stats* st) -> int {
    if (!((bad_b & 2) && dev[(size_t)d].n_extra[(size_t)b] > 0)) return MCD_OK;
    // certificate failed with the class treatment of duplicated cells: solve this replicate again without it
    // (see mcd_subinstance_steps)
    mcd_stats st2;
    const int rc2 = subinstance_steps_impl(hd, rna_rows, m_sub, dna_cols + r * n_sub, n_sub, assign + r * m_sub,
                                           step + r * m_sub, step_obj ? step_obj + r * nsteps : nullptr, MCD_MEM_HOST,
                                           &st2, false, &bad_b);
    if (rc2 != MCD_OK && rc2 != MCD_ERR_NOT_CONVERGED) return rc2;
    g = st2.cert_rel_gap;
    if (st) st->sweep_fallbacks += 1;
    return MCD_OK;
  };
  return sweep_replicates(hs, ndev, P, nrep, m_sub, n_sub, assign, step, step_obj, cert_gap, stats, hk);
}

int mcd_subinstance_sweep(mcd_handle h, int64_t nrep, const int32_t* rna_rows, int64_t m_sub, const int32_t* dna_cols,
                          int64_t n_sub, int32_t* assign, int32_t* step, double* step_obj, double* cert_gap,
                          int concurrency, mcd_stats* stats) {
  if (!h) return MCD_ERR_INVALID;
  return subinstance_sweep_impl(&h, 1, nrep, rna_rows, m_sub, dna_cols, n_sub, assign, step, step_obj, cert_gap,
                                concurrency, stats);
}

int mcd_subinstance_sweep_multi(mcd_handle* hs, int ndev, int64_t nrep, const int32_t* rna_rows, int64_t m_sub,
                                const int32_t* dna_cols, int64_t n_sub, int32_t* assign, int32_t* step,
                                double* step_obj, double* cert_gap, int concurrency, mcd_stats* stats) {
  if (!hs || ndev < 1 || !hs[0]) return MCD_ERR_INVALID;
  if (ndev == 1)
    return mcd_subinstance_sweep(hs[0], nrep, rna_rows, m_sub, dna_cols, n_sub, assign, step, step_obj, cert_gap,
                                 concurrency, stats);
  int st;
  if ((st = check_view_handles(hs, ndev, "mcd_subinstance_sweep_multi"))) return st;
  return subinstance_sweep_impl(hs, ndev, nrep, rna_rows, m_sub, dna_cols, n_sub, assign, step, step_obj, cert_gap,
                                concurrency, stats);
}

// Placement of the left-out cells of the replicates [r0, r0 + nb) (blocks at `out`, layout L) and the copies of
// their results into the dense host outputs, on h (its resident matrix, its stream).
static int loo_place_batch(mcd_context* h, const int* d_cells, int64_t r0, int64_t nb, int64_t m_sub, int64_t nsteps,
                           int64_t k_steps, char* out, const mcd_loo_layout& L, int32_t* test_col, double* test_corr,
                           double* total, double* match_corr) {
  int st;
  if ((st = mcd_launch_loo_place(h, static_cast<const double*>(h->ws[WS_C].ptr), h->last_ldc, d_cells + r0, nb, m_sub,
                                 h->last_N, nsteps, k_steps, out, L)))
    return st;
  MCD_CUDA(h, cudaMemcpy2DAsync(test_corr + r0, 8, out + L.res, L.stride, 8, (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpy2DAsync(total + r0, 8, out + L.res + 8, L.stride, 8, (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
  MCD_CUDA(h, cudaMemcpy2DAsync(test_col + r0, 4, out + L.res + 16, L.stride, 4, (size_t)nb, cudaMemcpyDeviceToHost,
                                h->stream));
  if (match_corr && m_sub > 0)
    MCD_CUDA(h, cudaMemcpy2DAsync(match_corr + r0 * m_sub, (size_t)m_sub * 8, out + L.match, L.stride, (size_t)m_sub * 8,
                                  (size_t)nb, cudaMemcpyDeviceToHost, h->stream));
  return MCD_OK;
}

static int loo_sweep_impl(mcd_context* const* hs, int ndev, const int32_t* cells, int64_t ncells, int64_t k_steps,
                          int32_t* test_col, double* test_corr, double* total, int32_t* assign, int32_t* step,
                          double* step_obj, double* match_corr, double* cert_gap, int concurrency, mcd_stats* stats) {
  mcd_context* h = hs[0];
  if (!has_matrix(h)) return mcd_fail(h, MCD_ERR_INVALID, "mcd_loo_sweep: no mcd_cell2cell result is resident");
  if (!cells || ncells < 1) return mcd_fail(h, MCD_ERR_INVALID, "mcd_loo_sweep: no cells to leave out");
  if (k_steps < 1) return mcd_fail(h, MCD_ERR_INVALID, "mcd_loo_sweep: k_steps must be >= 1");
  if (!test_col || !test_corr || !total)
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_loo_sweep: test_col, test_corr and total are required");
  for (int64_t r = 0; r < ncells; ++r)
    if (cells[r] < 0 || cells[r] >= h->last_M) return mcd_fail(h, MCD_ERR_INVALID, "mcd_loo_sweep: cell out of range");
  const int64_t N = h->last_N, m_sub = h->last_M - 1;
  const int64_t ldc = h->last_ldc;
  if (m_sub == 0) ndev = 1;  // M == 1: no replicate has a solve; hs[0] places every left-out cell in one launch
  // per handle: the left-out cells on its device
  std::vector<const int*> d_cells((size_t)ndev);
  int st;
  for (int d = 0; d < ndev; ++d) {
    mcd_context* hd = hs[d];
    MCD_CUDA(h, cudaSetDevice(hd->device));
    void* p_idx = nullptr;
    if ((st = mcd_ws(hd, WS_SWEEP_IDX, (size_t)ncells * 4, &p_idx))) return d == 0 ? st : mcd_fail(h, st, hd->err.c_str());
    d_cells[(size_t)d] = static_cast<const int*>(p_idx);
    MCD_CUDA(h, cudaMemcpyAsync(p_idx, cells, (size_t)ncells * 4, cudaMemcpyHostToDevice, hd->stream));
  }
  MCD_CUDA(h, cudaSetDevice(h->device));
  // the replicate's extra bytes after its StepOut block: match counts [N], results, matched correlations [m_sub]
  const size_t cnt_bytes = ((size_t)N * 4 + 255) / 256 * 256, res_bytes = 256;
  const size_t mc_bytes = match_corr ? ((size_t)m_sub * 8 + 255) / 256 * 256 : 0;
  mcd_loo_layout L;
  if (m_sub == 0) {
    // M == 1: every replicate is empty, no solve runs; the placement sees no matches at all
    L.stride = cnt_bytes + res_bytes;
    L.assign = L.obj = L.cnt = 0;
    L.res = cnt_bytes;
    L.match = 0;
    void* p_out = nullptr;
    if ((st = mcd_ws(h, WS_SWEEP_OUT, (size_t)ncells * L.stride, &p_out))) return st;
    const int64_t launches0 = h->launches;
    MCD_CUDA(h, cudaEventRecord(get_event(h, 96), h->stream));
    if ((st = loo_place_batch(h, d_cells[0], 0, ncells, 0, 0, k_steps, static_cast<char*>(p_out), L, test_col, test_corr,
                              total, nullptr)))
      return st;
    MCD_CUDA(h, cudaEventRecord(get_event(h, 97), h->stream));
    MCD_CUDA(h, cudaStreamSynchronize(h->stream));
    for (int64_t r = 0; cert_gap && r < ncells; ++r) cert_gap[r] = h->opt.certify ? 0.0 : -1.0;
    if (stats) {
      memset(stats, 0, sizeof *stats);
      float ms = 0.f;
      cudaEventElapsedTime(&ms, get_event(h, 96), get_event(h, 97));
      stats->ms_lap = ms;
      stats->ms_total = ms;
      stats->kernel_launches = h->launches - launches0;
    }
    return MCD_OK;
  }
  const SweepPlan P = sweep_plan(ncells, m_sub, N, cnt_bytes + res_bytes + mc_bytes, concurrency);
  L.stride = P.rep_bytes;
  L.cnt = P.step_bytes;
  L.res = P.step_bytes + cnt_bytes;
  L.match = match_corr ? P.step_bytes + cnt_bytes + res_bytes : 0;
  SweepHooks hk;
  hk.build = [&](mcd_context* hd, int, mcd_context* w, int64_t r0, int64_t b, double* subC, int64_t lds, double* subCt,
                 int64_t ldst, const int** dna_class) -> int {
    *dna_class = nullptr;  // no DNA cell is repeated: the asynchronous solver path
    int stw = mcd_launch_loo_gather(w, static_cast<const double*>(hd->ws[WS_C].ptr), ldc, cells[r0 + b], m_sub, N, subC,
                                    lds);
    return stw ? stw : mcd_transpose_f64(w, subC, m_sub, N, lds, subCt, ldst);
  };
  hk.after = [&](mcd_context* hd, int d, int64_t r0, int64_t nb, char* out) -> int {
    mcd_loo_layout Lb = L;  // a copy per call: the handles' threads run this hook concurrently
    const StepOut o = carve_step_out(out, m_sub, P.nsteps);  // the step loop's outputs inside a replicate's block
    Lb.assign = (size_t)(reinterpret_cast<char*>(o.assign) - out);
    Lb.obj = (size_t)(reinterpret_cast<char*>(o.obj) - out);
    return loo_place_batch(hd, d_cells[(size_t)d], r0, nb, m_sub, P.nsteps, k_steps, out, Lb, test_col, test_corr,
                           total, match_corr);
  };
  return sweep_replicates(hs, ndev, P, ncells, m_sub, N, assign, step, step_obj, cert_gap, stats, hk);
}

int mcd_loo_sweep(mcd_handle h, const int32_t* cells, int64_t ncells, int64_t k_steps, int32_t* test_col,
                  double* test_corr, double* total, int32_t* assign, int32_t* step, double* step_obj, double* match_corr,
                  double* cert_gap, int concurrency, mcd_stats* stats) {
  if (!h) return MCD_ERR_INVALID;
  return loo_sweep_impl(&h, 1, cells, ncells, k_steps, test_col, test_corr, total, assign, step, step_obj, match_corr,
                        cert_gap, concurrency, stats);
}

int mcd_loo_sweep_multi(mcd_handle* hs, int ndev, const int32_t* cells, int64_t ncells, int64_t k_steps,
                        int32_t* test_col, double* test_corr, double* total, int32_t* assign, int32_t* step,
                        double* step_obj, double* match_corr, double* cert_gap, int concurrency, mcd_stats* stats) {
  if (!hs || ndev < 1 || !hs[0]) return MCD_ERR_INVALID;
  if (ndev == 1)
    return mcd_loo_sweep(hs[0], cells, ncells, k_steps, test_col, test_corr, total, assign, step, step_obj, match_corr,
                         cert_gap, concurrency, stats);
  int st;
  if ((st = check_view_handles(hs, ndev, "mcd_loo_sweep_multi"))) return st;
  return loo_sweep_impl(hs, ndev, cells, ncells, k_steps, test_col, test_corr, total, assign, step, step_obj,
                        match_corr, cert_gap, concurrency, stats);
}

int mcd_null_assignments(mcd_handle h, int64_t trials, uint64_t seed, double* sums, double* medians, int out_space) {
  if (!h) return MCD_ERR_INVALID;
  if (!sums || trials < 1 || !has_matrix(h))
    return mcd_fail(h, MCD_ERR_INVALID, "mcd_null_assignments: no mcd_cell2cell result is resident");
  MCD_CUDA(h, cudaSetDevice(h->device));
  double* d_s = sums;
  double* d_m = medians;
  int st;
  if (out_space != MCD_MEM_DEVICE) {
    void* p = nullptr;
    if ((st = mcd_ws(h, WS_SUB_MISC, (size_t)trials * 16, &p))) return st;
    d_s = static_cast<double*>(p);
    d_m = medians ? d_s + trials : nullptr;
  }
  if ((st = mcd_launch_null_assignments(h, static_cast<const double*>(h->ws[WS_C].ptr), h->last_ldc, h->last_M,
                                        h->last_N, 0, trials, seed, d_s, d_m)))
    return st;
  if (out_space != MCD_MEM_DEVICE) {
    MCD_CUDA(h, cudaMemcpyAsync(sums, d_s, (size_t)trials * 8, cudaMemcpyDeviceToHost, h->stream));
    if (medians) MCD_CUDA(h, cudaMemcpyAsync(medians, d_m, (size_t)trials * 8, cudaMemcpyDeviceToHost, h->stream));
  }
  MCD_CUDA(h, cudaStreamSynchronize(h->stream));
  return MCD_OK;
}

int mcd_share_resident(mcd_handle* hs, int ndev) {
  if (!hs || ndev < 1 || !hs[0]) return MCD_ERR_INVALID;
  mcd_context* h0 = hs[0];
  int st;
  if ((st = check_distinct_handles(hs, ndev, "mcd_share_resident"))) return st;
  if (!has_matrix(h0)) return mcd_fail(h0, MCD_ERR_INVALID, "mcd_share_resident: no mcd_cell2cell result is resident on handle 0");
  const size_t bytes = (size_t)h0->last_M * (size_t)h0->last_ldc * 8;
  const void* src = h0->ws[WS_C].ptr;
  MCD_CUDA(h0, cudaSetDevice(h0->device));
  MCD_CUDA(h0, cudaEventRecord(get_event(h0, 95), h0->stream));  // the matrix is complete once this event has passed
  for (int d = 1; d < ndev; ++d) {
    mcd_context* h = hs[d];
    drop_resident(h);  // also if a copy below fails
    MCD_CUDA(h0, cudaSetDevice(h->device));
    if (h->device != h0->device) {
      int can = 0;
      if (cudaDeviceCanAccessPeer(&can, h->device, h0->device) == cudaSuccess && can) {
        cudaError_t pe = cudaDeviceEnablePeerAccess(h0->device, 0);
        if (pe != cudaSuccess) cudaGetLastError();  // already enabled
      }
    }
    void* dst = nullptr;
    if ((st = mcd_ws(h, WS_C, bytes, &dst))) return mcd_fail(h0, st, h->err.c_str());
    MCD_CUDA(h0, cudaStreamWaitEvent(h->stream, get_event(h0, 95), 0));
    if (h->device == h0->device)
      MCD_CUDA(h0, cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, h->stream));
    else
      MCD_CUDA(h0, cudaMemcpyPeerAsync(dst, h->device, src, h0->device, bytes, h->stream));
  }
  for (int d = 1; d < ndev; ++d) {
    MCD_CUDA(h0, cudaSetDevice(hs[d]->device));
    MCD_CUDA(h0, cudaStreamSynchronize(hs[d]->stream));
  }
  MCD_CUDA(h0, cudaSetDevice(h0->device));
  for (int d = 1; d < ndev; ++d) {
    mcd_context* h = hs[d];
    h->last_M = h0->last_M;
    h->last_N = h0->last_N;
    h->last_ldc = h0->last_ldc;
    h->last_assign = nullptr;
    h->gen = h0->gen;
  }
  return MCD_OK;
}

int mcd_null_assignments_multi(mcd_handle* hs, int ndev, int64_t trials, uint64_t seed, double* sums, double* medians) {
  if (!hs || ndev < 1 || !hs[0]) return MCD_ERR_INVALID;
  if (ndev == 1) return mcd_null_assignments(hs[0], trials, seed, sums, medians, MCD_MEM_HOST);
  mcd_context* h0 = hs[0];
  int st;
  if ((st = check_view_handles(hs, ndev, "mcd_null_assignments_multi"))) return st;
  if (!sums || trials < 1) return mcd_fail(h0, MCD_ERR_INVALID, "mcd_null_assignments_multi: bad arguments");
  // every trial costs the same: handle d takes the contiguous range [lo[d], lo[d + 1]), in proportion to its SMs
  int64_t sm_total = 0;
  for (int d = 0; d < ndev; ++d) sm_total += hs[d]->sm_count > 0 ? hs[d]->sm_count : 1;
  std::vector<int64_t> lo((size_t)ndev + 1);
  int64_t cum = 0;
  for (int d = 0; d < ndev; ++d) {
    lo[(size_t)d] = (int64_t)((__int128)trials * cum / sm_total);
    cum += hs[d]->sm_count > 0 ? hs[d]->sm_count : 1;
  }
  lo[(size_t)ndev] = trials;
  std::vector<double*> d_s((size_t)ndev, nullptr);
  for (int d = 0; d < ndev; ++d) {
    const int64_t n = lo[(size_t)d + 1] - lo[(size_t)d];
    if (n == 0) continue;
    mcd_context* h = hs[d];
    MCD_CUDA(h0, cudaSetDevice(h->device));
    void* p = nullptr;
    if ((st = mcd_ws(h, WS_SUB_MISC, (size_t)n * 16, &p))) return d == 0 ? st : mcd_fail(h0, st, h->err.c_str());
    d_s[(size_t)d] = static_cast<double*>(p);
    if ((st = mcd_launch_null_assignments(h, static_cast<const double*>(h->ws[WS_C].ptr), h->last_ldc, h->last_M,
                                          h->last_N, lo[(size_t)d], n, seed, d_s[(size_t)d],
                                          medians ? d_s[(size_t)d] + n : nullptr)))
      return d == 0 ? st : mcd_fail(h0, st, h->err.c_str());
  }
  // the copies only after every launch: a copy into pageable host memory returns once it is complete
  for (int d = 0; d < ndev; ++d) {
    const int64_t n = lo[(size_t)d + 1] - lo[(size_t)d];
    if (n == 0) continue;
    mcd_context* h = hs[d];
    MCD_CUDA(h0, cudaSetDevice(h->device));
    MCD_CUDA(h0, cudaMemcpyAsync(sums + lo[(size_t)d], d_s[(size_t)d], (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    if (medians)
      MCD_CUDA(h0, cudaMemcpyAsync(medians + lo[(size_t)d], d_s[(size_t)d] + n, (size_t)n * 8, cudaMemcpyDeviceToHost,
                                   h->stream));
  }
  for (int d = 0; d < ndev; ++d) {
    MCD_CUDA(h0, cudaSetDevice(hs[d]->device));
    MCD_CUDA(h0, cudaStreamSynchronize(hs[d]->stream));
  }
  MCD_CUDA(h0, cudaSetDevice(h0->device));
  return MCD_OK;
}

}  // extern "C"
