// Internal declarations shared by the kernels and the C ABI (include/macrodna_b200.h).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <string>
#include <vector>

#include "../../include/macrodna_b200.h"

struct mcd_stager;  // stage.cu: host threads + pinned buffers for pageable inputs
void mcd_stager_destroy(mcd_stager* s);

struct mcd_buffer {
  void* ptr = nullptr;
  size_t bytes = 0;
};

// Tuning / behaviour switches of a handle (mcd_set_option / mcd_get_option, include/macrodna_b200.h).  Every knob
// that used to be an environment variable read per solve lives here: tests and sweeps set them on the handle.
struct mcd_options {
  int certify = 1;            // "certify": dual certificate sweep after every assignment solve
  int debug = 0;              // "debug": per-step solver counters on stderr
  int corr_only = 0;          // "corr_only": mcd_cell2cell stops after K2 (matrix resident for the view calls)
  int deterministic = 0;      // "deterministic": round-synchronous solver kernels only (fixed bid order; see lap.async)
  int ozaki_slices = 0;       // "ozaki.slices": 0 = automatic (mcd_ozaki_slices_for)
  int ozaki_radix = 0;        // "ozaki.radix": 128 or 256 forces the digit radix, 0 = automatic (mcd_ozaki_format)
  int ozaki_align = 1;        // "ozaki.align": wave alignment of the K2c producers
  int ozaki_plan = 1;         // "ozaki.plan": unit order of a K2c pass
  int k1_generic = 0;         // "k1.generic": force the generic digit kernel
  int k1_no_stream = 0;       // "k1.no_stream": one-row-per-CTA digit kernel instead of the persistent streaming one
  double lap_theta = 3.0;     // "lap.theta": eps-scaling factor of the square phases
  double lap_eps_min = 1e-7;  // "lap.eps_min": smallest relative eps of the scaling phases
  double lap_eps0 = 0.0;      // "lap.eps0": relative eps of the first scaling phase (0 = 1 / lap.theta)
  int lap_scaling = 1;        // "lap.scaling": eps-scaling phases for n == m
  double lap_max_rounds = 0;  // "lap.max_rounds": 0 = 200000 + 64 n
  double lap_tail_budget = 0; // "lap.tail_budget": narrow rounds before a long price war goes to augmenting paths (0 = 4096 + m)
  int lap_blocks_per_sm = 4;  // "lap.blocks_per_sm": cooperative grid of the wide rounds
  int lap_grid_blocks = 0;    // "lap.grid_blocks": cap on that grid (0 = none); concurrent solves use a slice of the chip
  int lap_list_max_m = 0;     // "lap.list_max_m": single-CTA list tail up to this many objects
  int lap_lists = -1;         // "lap.lists": -1 = automatic (n < m)
  int lap_list_min_nu = 0;    // "lap.list_min_nu"
  int lap_tail_cluster = 0;   // "lap.tail_cluster": 0 = automatic (8, or 16 from 32768 objects)
  int lap_tail_mh = -1;       // "lap.tail_mh": -1 = automatic (n < m)
  int lap_tail_sym = 1;       // "lap.tail_sym": symmetric cluster tail (every CTA resolves the round); 0 = CTA-0-resolves form
  int lap_prefetch_rows = 1;  // "lap.prefetch_rows": symmetric tail prefetches the likely next bidder's row into L2
  int lap_async = 1;          // "lap.async": asynchronous (round-free) wide kernel for the rectangular steps
  int lap_async_nu = 0;       // "lap.async_nu": rounds with more bidders than this stay round-synchronous (0 = none)
  int lap_async_threads = 128;  // "lap.async_threads": threads per worker CTA (128 or 256)
  int lap_async_blocks_per_sm = 0;  // "lap.async_blocks_per_sm": 0 = as many as fit
  int lap_async_stop = 8;     // "lap.async_stop": unassigned persons at which the master/helper tail takes over
  int lap_sap = 1;            // "lap.sap": the asynchronous kernel's last persons go to grid-parallel augmenting paths
  int lap_sap_nu = 16;        // "lap.sap_nu": ... from this many unassigned persons on (replaces lap.async_stop)
  int lap_tail_nu = -1;       // "lap.tail_nu": -1 = kernel default
  int lap_mh_nu = 32;         // "lap.mh_nu": bidder count at which the master/helper kernel takes over from the wide rounds
  int lap_scale_cut = 0;      // "lap.scale_cut": eps-scaling phases end once at most this many persons still bid
  double lap_scale_tail_rounds = -1;  // "lap.scale_tail_rounds": narrow rounds a scaling phase may run (-1 = no limit)
  int lap_scale_full_phases = 0;  // "lap.scale_full_phases": the last this-many scaling phases are never cut short
  int lap_aug_nu = 0;         // "lap.aug_nu"
  int lap_aug_nu_square = -1; // "lap.aug_nu_square": -1 = lap.aug_nu
  int lap_rank_select = 1;    // "lap.rank_select"
  int lap_min_chunk = 4096;   // "lap.min_chunk"
  int lap_chunk_waves = 1;    // "lap.chunk_waves"
};

struct mcd_context {
  int device = 0;
  mcd_options opt;
  int sm_count = 0;
  cudaStream_t stream = nullptr;
  cudaStream_t copy_stream = nullptr;
  std::string err;
  int* d_flags = nullptr;  // [0] non-finite input seen, [1..] spare
  int64_t launches = 0;
  // grow-only device workspace slots (reused across calls)
  mcd_buffer ws[24];
  // pinned host staging
  void* h_stage[2] = {nullptr, nullptr};
  cudaEvent_t stage_ev[2] = {nullptr, nullptr};
  int stage_next = 0;
  mcd_stager* stager = nullptr;
  std::vector<cudaEvent_t> ev;
  // shape of the last mcd_cell2cell call whose correlation matrix / assignment are still resident
  int64_t last_M = 0, last_N = 0, last_ldc = 0;
  const int* last_assign = nullptr;  // NULL on a copy (mcd_share_resident): a matrix without an assignment
  // generation of the resident matrix: a process-wide id given to each successful mcd_cell2cell* run (0 = none); a
  // copy carries the id of the run it copied, so a multi-device call can tell a current copy from a stale one
  uint64_t gen = 0;
  // worker contexts of the replicate sweep (own stream + workspace each; same device): replicates are independent
  // problems, and most rounds of a solve keep a handful of SMs busy, so several are kept in flight
  std::vector<mcd_context*> workers;
};

enum {
  WS_RNA_IN = 0,   // staged raw RNA rows (host input path)
  WS_DNA_IN,       // staged raw DNA rows
  WS_RNA_C,        // centred RNA
  WS_DNA_C,        // centred DNA
  WS_NORM_A,
  WS_NORM_B,
  WS_C,            // corr [M,N]
  WS_CT,           // corr^T [N,M]
  WS_W,            // compacted per-step cost block
  WS_LAP,          // solver state
  WS_STEP,         // step-loop state (assign, step, active lists, objectives)
  WS_SLICES_A,
  WS_SLICES_B,
  WS_MISC,
  WS_GIDX,  // gene gather indices (rna, dna)
  WS_SCALE, // Ozaki row scales (rna then dna)
  WS_SUB_C,    // sub-instance views of the resident correlation matrix (replicate sweeps / leave-one-out)
  WS_SUB_CT,
  WS_SUB_IDX,
  WS_SUB_MISC,
  WS_SWEEP_IDX,  // replicate sweep: RNA rows + the batch's DNA columns
  WS_SWEEP_OUT,  // replicate sweep: per-replicate step-loop outputs of the batch
  WS_NULL,       // null test above 4096 cells a side: per-CTA key slabs (<= 1 GiB)
};

int mcd_fail(mcd_context* h, int status, const char* what, cudaError_t e = cudaSuccess);
// true if p is ordinary (unregistered) host memory
bool mcd_is_pageable(const void* p);
// host -> device copy of a [rows, width] float64 block (host pitch src_ld, device pitch dst_ld, elements) from
// PAGEABLE memory through the handle's pinned staging buffers, asynchronous on `stream` after each block's host copy
int mcd_staged_h2d(mcd_context* h, double* dst, int64_t dst_ld, const double* src, int64_t src_ld, int64_t width,
                   int64_t rows, cudaStream_t stream);
int mcd_ws(mcd_context* h, int slot, size_t bytes, void** out);

#define MCD_CUDA(h, call)                                      \
  do {                                                         \
    cudaError_t e__ = (call);                                  \
    if (e__ != cudaSuccess) return mcd_fail((h), MCD_ERR_CUDA, #call, e__); \
  } while (0)

#define MCD_LAUNCH_CHECK(h, name)                              \
  do {                                                         \
    (h)->launches++;                                           \
    cudaError_t e__ = cudaGetLastError();                      \
    if (e__ != cudaSuccess) return mcd_fail((h), MCD_ERR_CUDA, name, e__); \
  } while (0)

// int8 digit-slice operand of the Ozaki path (K1 output, K2c input):
//   digits [nsl, ncells(+), ldk8] int8 -- slice t of row r starts at digits + t*slice_stride + r*ldk8
//   scale  [ncells] double           -- 2^-e of the per-row power-of-two scaling
//   rb     radix bits: 7 = balanced radix-128 digits in [-64, 63], 8 = balanced radix-256 digits in [-128, 127]
//          (nsl <= 7: the fixed-point integer of 8 nsl - 1 bits must stay exact in a double's rounding)
#define MCD_OZAKI_MAX_SLICES 8
struct mcd_ozaki_out {
  int8_t* digits = nullptr;
  int64_t ldk8 = 0;
  int64_t slice_stride = 0;
  int nsl = 0;
  int rb = 7;
  double* scale = nullptr;
};
// True if every significance-group sum of nsl slices over ldk8 genes is exact in K2c's int32 accumulators.
// Radix 128: a group holds at most nsl products of |d d'| <= 4096.  Radix 256: the leading digit lies in [-64, 64]
// (|q| <= 2^(8 nsl - 2)), the others in [-128, 127]; the heaviest group (g = nsl - 1) holds two products with the
// leading digit (<= 64 * 128) and nsl - 2 others (<= 128 * 128): 16384 (nsl - 1) per gene.
inline bool mcd_ozaki_exact(int nsl, int rb, int64_t ldk8) {
  const double per_gene = rb == 8 ? 16384.0 * (nsl - 1) : 4096.0 * nsl;
  return per_gene * (double)ldk8 < 2147483648.0;
}

// ---- kernel launchers (each returns an mcd_status) -------------------------------------------
// slices_hi / slices_lo: the two fp16 slices (each [ncells, ldk16]); both NULL for the FP64 path
int mcd_launch_standardize(mcd_context* h, const double* X, int64_t ncells, int64_t G, int64_t ldx,
                           double* centred, int64_t ldk, uint16_t* slices_hi, uint16_t* slices_lo, int64_t ldk16,
                           double* norms, const int* gidx = nullptr, const mcd_ozaki_out* ozaki = nullptr);
// K2c: C = sum over genes of the digit-slice products (exact int32 accumulation in TMEM), FP64 epilogue.
// A: nsl slices of [M, ldk8] int8 (slice stride a_stride elements), B likewise; sA/sB the row scales; rb radix bits.
int mcd_launch_corr_ozaki(mcd_context* h, const int8_t* A, int64_t a_stride, int64_t M, const int8_t* B,
                          int64_t b_stride, int64_t N, int64_t ldk8, int nsl, int rb, const double* sA, const double* sB,
                          const double* nA, const double* nB, double* C, int64_t ldc, double* Ct, int64_t ldct);
int mcd_launch_corr_fp64(mcd_context* h, const double* A, int64_t M, const double* B, int64_t N, int64_t ldk,
                         const double* nA, const double* nB, double* C, int64_t ldc, double* Ct, int64_t ldct);
int mcd_launch_corr_split(mcd_context* h, const uint16_t* A_hi, const uint16_t* A_lo, int64_t M,
                          const uint16_t* B_hi, const uint16_t* B_lo, int64_t N, int64_t ldk16, const double* nA,
                          const double* nB, double* C, int64_t ldc, double* Ct, int64_t ldct);

// Random-assignment null test on a resident correlation matrix (null_test.cu): trials t0 .. t0 + trials - 1, trial
// t0 + t written at d_sums[t] / d_medians[t].
int mcd_launch_null_assignments(mcd_context* h, const double* C, int64_t ldc, int64_t M, int64_t N, int64_t t0,
                                int64_t trials, uint64_t seed, double* d_sums, double* d_medians);

// Leave-one-out sweep (loo.cu).  Byte offsets inside one replicate's block of the sweep's output buffer.
struct mcd_loo_layout {
  size_t stride;  // bytes per replicate
  size_t assign;  // int32 [m_sub]: DNA column of each remaining row (the replicate's step-loop output)
  size_t obj;     // double [nsteps]: its step objectives
  size_t cnt;     // int32 [N]: scratch, matches per DNA column
  size_t res;     // double test_corr, double total, int32 test_col
  size_t match;   // double [m_sub]: C[row, assign] of the remaining rows; 0 = not wanted
};
// sub [m, lds] = C [M, ldc] with row q deleted (rows in ascending order, columns [0, n))
int mcd_launch_loo_gather(mcd_context* h, const double* C, int64_t ldc, int64_t q, int64_t m, int64_t n, double* sub,
                          int64_t lds);
// one CTA per replicate r < nrep (block at base + r * L.stride, left-out row d_cells[r]): placement of the left-out
// cell, its correlation, the replicate's total and (L.match) the matched correlations
int mcd_launch_loo_place(mcd_context* h, const double* C, int64_t ldc, const int* d_cells, int64_t nrep, int64_t m_sub,
                         int64_t N, int64_t nsteps, int64_t k_steps, char* base, const mcd_loo_layout& L);

struct mcd_lap_counters {  // device-resident, one per solve
  long long rounds;
  long long bids;
  long long bytes;
  long long aug_rows;
  long long aug_steps;
  int status;  // 0 ok, 1 = guard hit
  int pad;
  long long t_phase[8];  // SM cycles seen by CTA 0. wide kernel: bidding, barrier 1, resolution, barrier 2;
                         // cluster kernel: scan, wait partials, resolve+send, wait packet
  long long a_ts[8];     // asynchronous wide kernel (debug): ns from its start until <= 4096, 2048, 1024, 512, 256, 128, 64,
                         // stop_nu persons were left unassigned
  long long a_hops[8];   // ... and the bids made until then
};
struct mcd_lap_cert {  // device-resident, one per solve: the dual certificate (lap.cu, lap_cert_* kernels)
  double lambda;         // min price over the assigned objects
  double gap;            // dual objective - primal objective >= 0 (0 to rounding <=> optimal)
  double rel_gap;        // gap / |primal|
  double max_violation;  // largest single term of the gap
  double primal;
  int n_bad;             // persons without an object + objects used twice
  int pad;
};
size_t mcd_lap_workspace_bytes(int64_t n, int64_t m);
// Solve one rectangular max-assignment (n <= m).  `work` is mcd_lap_workspace_bytes(n, m) of device memory.
// check_finite: also scan W for NaN/Inf (raises the context's non-finite flag; the solver kernels then no-op)
// d_cert: optional; when non-NULL (and the handle's "certify" option is on) the dual certificate of the solve is
// written there and a failed certificate raises d_counters->status bit 1.  prices_out: optional [m] device copy of
// the final object prices.  person_class: optional DEVICE int [n], ids in [0, n), equal ids = persons with identical
// cost rows (copies of one resampled cell): they bid as a class of similar persons (lap.cu, LapState::pcls).
int mcd_launch_lap(mcd_context* h, const double* W, int64_t n, int64_t m, int64_t ldw, int32_t* col4row,
                   double* objective, void* work, mcd_lap_counters* d_counters, bool check_finite,
                   mcd_lap_cert* d_cert = nullptr, double* prices_out = nullptr, const int* person_class = nullptr);
// certificate of an arbitrary (col4row, prices) pair; work: >= 4 m + 8 n + 1024 bytes of device scratch
int mcd_launch_lap_certify(mcd_context* h, const double* W, int64_t n, int64_t m, int64_t ldw, const int32_t* col4row,
                           const double* prices, void* work, mcd_lap_cert* d_cert, mcd_lap_counters* d_counters);
#define MCD_CERT_TOL_REL 1.0e-9  // north-star objective tolerance; observed gaps are ~1e-15
