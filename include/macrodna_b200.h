/*
 * macrodna_b200 -- C ABI of the B200-native cell-matching hot path.
 *
 * The reference (NakhlehLab/MaCroDNA) is pure Python and has no FFI of its own;
 * each entry point below replaces a span of src/MaCroDNA/macrodna.py and is what
 * a ctypes binding on the reference side would bind (see INTEGRATION.md).
 * Plain pointers and sizes only; no torch / numpy types.  All matrices are
 * row-major float64 "cells x genes" (what `df.T.to_numpy()` yields,
 * macrodna.py:93-94) unless stated otherwise.
 *
 * Conventions: every call returns 0 (MCD_OK) or a negative mcd_status;
 * mcd_last_error(h) gives the detail string of the last failure on a handle.
 * The caller owns every buffer it passes.  A handle is bound to one CUDA device
 * and one stream; calls on one handle are serialised by the caller; distinct
 * handles are independent (the only process-wide state is the counter that
 * numbers the runs, see mcd_share_resident).
 */
#ifndef MACRODNA_B200_H
#define MACRODNA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MCD_ABI_VERSION 2

typedef struct mcd_context* mcd_handle;

typedef enum {
  MCD_OK = 0,
  MCD_ERR_INVALID = -1,      /* bad argument (NULL, negative size, ld too small ...)     */
  MCD_ERR_CUDA = -2,         /* a CUDA runtime call or kernel failed                      */
  MCD_ERR_NOMEM = -3,        /* device or host allocation failed                          */
  MCD_ERR_NONFINITE = -4,    /* NaN/Inf in the input data (cf. SURVEY appendix B)         */
  MCD_ERR_UNSUPPORTED = -5,  /* precision / shape not supported by this build             */
  MCD_ERR_NOT_CONVERGED = -6 /* assignment solver hit its iteration guard                 */
} mcd_status;

/* Arithmetic of the correlation contraction (macrodna.py:103-107). */
typedef enum {
  MCD_PREC_FP64 = 0,  /* FP64 tensor-core (DMMA) contraction of centred rows: parity mode   */
  MCD_PREC_SPLIT_FP16 = 1, /* tcgen05 split precision: fp16 hi+lo slices, 3 products, FP32 in TMEM */
  MCD_PREC_OZAKI_INT8 = 2  /* tcgen05 int8 digit slices (Ozaki scheme), exact int32 accumulation in TMEM,
                              FP64 combination: FP64-class results from the integer tensor pipe          */
} mcd_precision;

/* Where a caller buffer lives. */
typedef enum { MCD_MEM_HOST = 0, MCD_MEM_DEVICE = 1 } mcd_memspace;

#define MCD_MAX_STEP_STATS 64

/* Per-call measurements, filled when a non-NULL pointer is passed. Times are CUDA-event ms. */
typedef struct {
  double ms_h2d;          /* host->device staging of the inputs                          */
  double ms_standardize;  /* K1 (both operands)                                           */
  double ms_corr;         /* K2                                                           */
  double ms_lap;          /* K3+K4, all steps                                             */
  double ms_d2h;          /* device->host of assign/step/objective                        */
  double ms_total;        /* first to last event                                          */
  int64_t n_steps;        /* ceil(M/N), macrodna.py:118-123                               */
  int64_t kernel_launches; /* kernels launched by this call                               */
  int64_t lap_rounds;     /* Jacobi bidding rounds, all steps                             */
  int64_t lap_bids;       /* row scans (one per bidder per round), all steps              */
  int64_t lap_bytes;      /* cost bytes scanned by bidding + augmentation, all steps      */
  int64_t lap_aug_rows;   /* persons finished by shortest-augmenting-path instead of bids */
  int64_t lap_aug_steps;  /* Dijkstra steps of those augmentations                        */
  int64_t lap_cycles[8];  /* [0..3] synchronous wide kernel, SM cycles of CTA 0: bidding, barrier 1, resolution,
                             barrier 2; steps run by the asynchronous wide kernel add ns instead: bidding until CTA 0
                             ran out of work, drain of the other workers, epilogue, and the persons parked on ties.
                             [4..7] narrow-round kernels, SM cycles of the resolving CTA: scan / bidding, wait for
                             partials / list rebuilds, resolution, (first cluster kernel only) wait for the packet */
  double step_ms[MCD_MAX_STEP_STATS];
  int64_t step_rounds[MCD_MAX_STEP_STATS];
  int64_t step_bids[MCD_MAX_STEP_STATS];
  /* Dual certificate of the assignment solves (handle option "certify", on by default): for every step the
   * solver's final object prices are turned into a feasible point of the dual of the reference's ILP
   * (macrodna.py:27-84) whose objective D bounds every feasible assignment from above; gap = D - objective >= 0
   * is 0 to rounding iff the step's assignment is optimal.  A relative gap above 1e-9 (the north-star objective
   * tolerance) fails the call with MCD_ERR_NOT_CONVERGED. */
  double cert_rel_gap;       /* max over the steps of gap / |objective|                              */
  double cert_max_violation; /* largest single dual-feasibility violation of a matched edge, any step */
  int64_t cert_bad;          /* unassigned persons + doubly used objects found by the checker (0)     */
  int64_t cert_steps;        /* steps certified                                                       */
  double step_cert_gap[MCD_MAX_STEP_STATS]; /* per-step relative gap (-1: not certified)              */
  int64_t sweep_fallbacks;   /* mcd_subinstance_sweep: replicates re-solved without the class treatment of
                                duplicated cells because their certificate failed with it             */
} mcd_stats;

int mcd_abi_version(void);
const char* mcd_strerror(int status);

/* Create / destroy a context on CUDA device `device` (owns a stream + workspace). */
int mcd_create(mcd_handle* out, int device);
int mcd_destroy(mcd_handle h);
const char* mcd_last_error(mcd_handle h);
int mcd_device_sm_count(mcd_handle h);
/* Block until everything queued on the handle's stream has finished. */
int mcd_synchronize(mcd_handle h);
/* The handle's cudaStream_t (as void*), for callers that record events on it. */
void* mcd_stream(mcd_handle h);

/*
 * Behaviour / tuning switches of a handle (all have working defaults; nothing on the product path reads the
 * environment).  Names: "certify" (1), "debug" (0: per-step solver counters on stderr), "corr_only" (0; 1 = the
 * fused driver stops after the correlation matrix, which stays resident for the view calls; assign comes back
 * as -1), "deterministic" (0; 1 = round-synchronous solver kernels only: the bid order, and with it the optimum
 * picked on inputs with exact ties, is then fixed; the default asynchronous kernel of the rectangular steps gives the
 * same unique optimum on tie-free inputs and redoes a step synchronously when it meets exact ties), "ozaki.slices" (0 = auto),
 * "ozaki.radix" (0 = auto; 128 or 256 forces the digit radix, see mcd_ozaki_format), "ozaki.align", "ozaki.plan", "k1.generic", "k1.no_stream", and the solver knobs "lap.theta", "lap.eps_min", "lap.eps0", "lap.scaling",
 * "lap.max_rounds", "lap.tail_budget", "lap.blocks_per_sm", "lap.grid_blocks", "lap.list_max_m", "lap.lists", "lap.list_min_nu",
 * "lap.tail_cluster", "lap.tail_mh", "lap.tail_sym", "lap.async", "lap.async_nu", "lap.async_threads", "lap.async_blocks_per_sm", "lap.async_stop", "lap.sap", "lap.sap_nu", "lap.prefetch_rows", "lap.tail_nu", "lap.mh_nu", "lap.scale_cut", "lap.scale_tail_rounds", "lap.scale_full_phases", "lap.aug_nu", "lap.aug_nu_square", "lap.rank_select",
 * "lap.min_chunk", "lap.chunk_waves".  Unknown names return MCD_ERR_INVALID.
 */
int mcd_set_option(mcd_handle h, const char* name, double value);
int mcd_get_option(mcd_handle h, const char* name, double* value);

/*
 * K1 -- per-cell standardisation.  Replaces the per-operand half of
 * cosine_similarity_np (macrodna.py:24-25): mean, x - mean, ||x - mean||_2.
 *   X        [ncells, G] row-major float64, leading dimension ldx (elements), DEVICE
 *   centred  [ncells, ldk] float64 centred rows, DEVICE; ldk = mcd_padded_k(G);
 *            columns [G, ldk) are written as zeros (K padding of the contraction)
 *   norms    [ncells] float64 ||x - mean||, DEVICE
 * Non-finite input is reported as MCD_ERR_NONFINITE at the next synchronising call
 * (mcd_check_finite) -- the kernel only raises a device flag.
 */
int64_t mcd_padded_k(int64_t G);
int mcd_standardize(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx,
                    double* centred, double* norms);
/* Same pass, but emits the split-precision operand of MCD_PREC_SPLIT_FP16: two fp16 slices (hi, lo) of
 * 256 * (x - mean)/||x - mean||:  slices [2, ncells, ldk16] uint16 (fp16 bits), ldk16 = mcd_padded_k_split(G),
 * zero padded. */
int64_t mcd_padded_k_split(int64_t G);
int mcd_standardize_split(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx,
                           uint16_t* slices, double* norms);
/* Same pass, but emits the integer operand of MCD_PREC_OZAKI_INT8: every unit-norm centred row, scaled by a
 * per-row power of two so that max|.| lies in [0.25, 0.5), as `nsl` balanced radix-128 digit slices:
 *   digits [nsl, ncells, ldk8] int8, ldk8 = mcd_padded_k_split(G), zero padded;  scale [ncells] = 2^-e (the
 *   factor that undoes the row scaling);  nsl in [2, 8] (mcd_ozaki_default_slices(): 6). */
int mcd_ozaki_default_slices(void);
/* Digit format the drivers use for an M x N x G instance on handle h (NULL: no handle options), ldk8 =
 * mcd_padded_k_split(G):
 *   "ozaki.slices" set: that many radix-128 slices (radix 256 if "ozaki.radix" is 256 too; at most 7 slices then);
 *   else "ozaki.radix" 256: 5 radix-256 slices;  else M*N*G <= 2e11 (or "ozaki.radix" 128): 8 radix-128 slices
 *   (FP64-GEMM-level error), 6 above M*N*G > 2e11;
 *   else ldk8 <= 32 704: 5 radix-256 slices (15 products, ~5e-12 absolute);  else 6 radix-128 slices (21 products).
 * Writes *nsl and *radix_bits (7 = radix 128, 8 = radix 256).  Returns 1 if the int32 accumulators of
 * mcd_corr_ozaki_radix are exact at this ldk8 in that format, 0 if the drivers take the FP64 pipe instead. */
int mcd_ozaki_format(mcd_handle h, int64_t M, int64_t N, int64_t G, int* nsl, int* radix_bits);
/* The slice count of mcd_ozaki_format without handle options (5 at radix-256 shapes). */
int mcd_ozaki_slices_for(int64_t M, int64_t N, int64_t G);
/* The slice count of mcd_ozaki_format for a given handle. */
int mcd_ozaki_slices(mcd_handle h, int64_t M, int64_t N, int64_t G);
int mcd_standardize_ozaki(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx, int8_t* digits,
                          int nsl, double* scale, double* norms);
/* Same with digits of radix_bits bits: 7 = the radix-128 digits above; 8 = balanced radix-256 digits in
 * [-128, 127] of rint(u * 2^(8 nsl - 1)) (the leading one in [-64, 64]), nsl in [2, 7]. */
int mcd_standardize_ozaki_radix(mcd_handle h, const double* X, int64_t ncells, int64_t G, int64_t ldx, int8_t* digits,
                                int nsl, int radix_bits, double* scale, double* norms);
/* Synchronise and return MCD_ERR_NONFINITE if any standardise call since the last check saw NaN/Inf. */
int mcd_check_finite(mcd_handle h);

/*
 * K2 -- correlation matrix.  Replaces the double loop macrodna.py:103-107:
 *   C[i, j] = dot(a_i, b_j) / (1e-10 + na_i * nb_j)
 *   A [M, ldk] centred RNA rows, B [N, ldk] centred DNA rows (outputs of mcd_standardize), DEVICE
 *   C  [M, ldc]  float64 row-major (rows = RNA, columns = DNA, macrodna.py:102), DEVICE, may be NULL
 *   Ct [N, ldct] float64, the transpose, DEVICE, may be NULL (at least one of C, Ct)
 */
int mcd_corr_fp64(mcd_handle h, const double* A, int64_t M, const double* B, int64_t N, int64_t G,
                  int64_t ldk, const double* nA, const double* nB, double* C, int64_t ldc,
                  double* Ct, int64_t ldct);
/* tcgen05 / TMEM split-precision variant on the fp16 slices of mcd_standardize_split (hi*hi + hi*lo + lo*hi). */
int mcd_corr_split(mcd_handle h, const uint16_t* A3, int64_t M, const uint16_t* B3, int64_t N,
                    int64_t G, int64_t ldk16, const double* nA, const double* nB, double* C,
                    int64_t ldc, double* Ct, int64_t ldct);

/* tcgen05 int8 variant on the digit slices of mcd_standardize_ozaki: all slice products with t + t' < nsl,
 * exact int32 accumulation per significance group in TMEM (cta_group::2, 256 x 256 tiles), FP64 epilogue.
 * MCD_ERR_UNSUPPORTED if nsl * 4096 * ldk8 >= 2^31 (the int32 accumulators could overflow). */
int mcd_corr_ozaki(mcd_handle h, const int8_t* A8, int64_t M, const int8_t* B8, int64_t N, int64_t G, int64_t ldk8,
                   int nsl, const double* sA, const double* sB, const double* nA, const double* nB, double* C,
                   int64_t ldc, double* Ct, int64_t ldct);
/* Same on the digits of mcd_standardize_ozaki_radix.  radix_bits 8: MCD_ERR_UNSUPPORTED if
 * 16384 (nsl - 1) ldk8 >= 2^31 (5 slices: ldk8 <= 32 704). */
int mcd_corr_ozaki_radix(mcd_handle h, const int8_t* A8, int64_t M, const int8_t* B8, int64_t N, int64_t G,
                         int64_t ldk8, int nsl, int radix_bits, const double* sA, const double* sB, const double* nA,
                         const double* nB, double* C, int64_t ldc, double* Ct, int64_t ldct);

/*
 * K3 -- one rectangular assignment.  Replaces one `ilp` call (macrodna.py:27-84):
 * maximise sum W[i, col4row[i]] over injective maps of the n rows into the m >= n columns.
 *   W [n, ldw] float64 DEVICE; col4row [n] int32 DEVICE out; objective: DEVICE double out (may be NULL)
 */
int mcd_lap_max(mcd_handle h, const double* W, int64_t n, int64_t m, int64_t ldw, int32_t* col4row,
                double* objective);
/* Same solve, also returning the proof of optimality: prices [m] float64 DEVICE out (the final object prices =
 * dual variables v_j, may be NULL) and cert [4] float64 HOST out = {relative duality gap, absolute gap, largest
 * single violation, #invalid entries} as described at mcd_stats (may be NULL).  The gap is recomputed from W, the
 * prices and col4row alone, so it does not depend on how the solver got there. */
int mcd_lap_max_certified(mcd_handle h, const double* W, int64_t n, int64_t m, int64_t ldw, int32_t* col4row,
                          double* objective, double* prices, double* cert);
/* The checker alone, on ANY assignment / price vector for W (all DEVICE; cert [4] HOST as above): lets a caller
 * certify a result obtained elsewhere, and lets the tests show that a damaged assignment or damaged prices are
 * caught.  Always returns MCD_OK when it ran; the verdict is in cert. */
int mcd_lap_certify(mcd_handle h, const double* W, int64_t n, int64_t m, int64_t ldw, const int32_t* col4row,
                    const double* prices, double* cert);

/*
 * K3+K4 -- the whole step loop (macrodna.py:110-145) on a resident correlation matrix.
 *   C [M, ldc], Ct [N, ldct] DEVICE (both required);
 *   assign [M] int32: DNA column of each RNA row; step [M] int32: 1-based step tag (macrodna.py:139);
 *   step_obj [ceil(M/N)] float64: per-step objective (`m.objVal`, cf. random_assignment_test.py:91);
 *   outputs live in `out_space` (host or device).
 */
int mcd_lap_steps(mcd_handle h, const double* C, int64_t ldc, const double* Ct, int64_t ldct,
                  int64_t M, int64_t N, int32_t* assign, int32_t* step, double* step_obj,
                  int out_space, mcd_stats* stats);

/*
 * The fused driver: everything between macrodna.py:93 and :145.
 *   rna [M, G] (ld = ld_rna), dna [N, G] (ld = ld_dna) float64 row-major in `in_space`
 *   (host buffers are staged through pinned chunks with async copies);
 *   assign/step/step_obj as above, in `out_space`;
 *   corr_out: optional [M, N] float64 copy of the correlation matrix in `out_space` (NULL to skip).
 */
int mcd_cell2cell(mcd_handle h, const double* rna, int64_t ld_rna, const double* dna, int64_t ld_dna,
                  int64_t M, int64_t N, int64_t G, int in_space, int precision, int32_t* assign,
                  int32_t* step, double* step_obj, double* corr_out, int out_space, mcd_stats* stats);

/*
 * Out-of-place transpose of a row-major float64 matrix: dst[c, r] = src[r, c], src [rows, lds],
 * dst [cols, ldd], both DEVICE.  Used by the multi-GPU driver to rebuild C^T after the NCCL
 * all-gather of the row-sharded correlation matrix.
 */
int mcd_transpose_f64(mcd_handle h, const double* src, int64_t rows, int64_t cols, int64_t lds, double* dst,
                      int64_t ldd);

/*
 * Same as mcd_cell2cell, with the gene intersection applied on the device: the host passes the frames' value
 * blocks as they are (rna [M, ld_rna], dna [N, ld_dna], any gene order, extra genes allowed) plus, per operand,
 * the column index of each of the G shared genes (int32 [G], HOST; NULL = identity).  This is the reference's
 * `.loc[genes, :]` re-indexing (macrodna.py:90-91) without the host copy of the matrices.
 */
int mcd_cell2cell_gather(mcd_handle h, const double* rna, int64_t ld_rna, const int32_t* rna_gene_idx,
                         const double* dna, int64_t ld_dna, const int32_t* dna_gene_idx, int64_t M, int64_t N,
                         int64_t G, int in_space, int precision, int32_t* assign, int32_t* step, double* step_obj,
                         double* corr_out, int out_space, mcd_stats* stats);

/*
 * The fused driver on several GPUs of one node, one caller (HOST inputs and outputs; gene indices as in
 * mcd_cell2cell_gather, NULL = identity).  hs[0..ndev): one handle per device.  RNA rows are sharded: device d
 * standardises rows [d*ceil(M/ndev), ...) and the DNA operand and contracts its row block -- no exchange inside the
 * contraction --, the correlation shards go to hs[0]'s device by peer copies (NVLink), which runs the step loop.
 * The matrix stays resident on hs[0] for the view calls.  Results are bit-identical to the single-device call.
 */
int mcd_cell2cell_multi(mcd_handle* hs, int ndev, const double* rna, int64_t ld_rna, const int32_t* rna_gene_idx,
                        const double* dna, int64_t ld_dna, const int32_t* dna_gene_idx, int64_t M, int64_t N, int64_t G,
                        int precision, int32_t* assign, int32_t* step, double* step_obj, mcd_stats* stats);

/*
 * Matched correlation of every RNA cell, corr[i, assign[i]], of the LAST mcd_cell2cell call on this handle
 * (its correlation matrix is still resident).  This is the `corr_val` column of the leave-one-out variant
 * (Resampling_stability_analyses/BE_data_analyses/run_loo_experiment.py:194) and the operand of the median
 * variant (random_assignment_test_median.py:196-199).  out [M] float64 in `out_space`.
 */
int mcd_last_match_values(mcd_handle h, double* out, int64_t M, int out_space);

/*
 * Views of the RESIDENT correlation matrix -- the reference's replicate sweeps and its leave-one-out test re-run
 * the whole class on frames that only gather or delete cells (clonal_proportions_resampling.py:177-190,
 * run_dna_batch_removal_exp.py, run_loo_experiment.py:217-226 `np.delete(corrs, cell_idx, 0)`): the genes are
 * untouched, so every such replicate is an index gather of the matrix the last mcd_cell2cell call left on the
 * device.  These calls keep that matrix (and mcd_last_match_values) valid.
 *
 * Duplicated DNA cells: when dna_cols repeats a cell (resampling WITH replacement, clonal_proportions_resampling.py
 * :184-187) the replicate has exact ties by construction and any of the tied optima answers the reference's ILP.
 * The copies of a cell are handled as a class of similar persons of the auction (they never bid against each
 * other; their duals are equalised before the certificate), so such replicates solve -- exactly -- as fast as
 * tie-free ones.
 *
 * mcd_subinstance_steps: the step loop (macrodna.py:110-145) on C[rna_rows][:, dna_cols].
 *   rna_rows [m_sub], dna_cols [n_sub]: HOST int32 indices into the resident matrix (NULL = all, in order;
 *   repeats allowed -- resampled replicates carry duplicate DNA cells);
 *   assign [m_sub]: POSITION in dna_cols matched to each listed RNA row; step, step_obj as in mcd_lap_steps.
 * mcd_corr_rows: rows of the resident matrix, out [nrows, N] row-major (the left-out cell's correlations,
 *   run_loo_experiment.py:226).
 */
int mcd_subinstance_steps(mcd_handle h, const int32_t* rna_rows, int64_t m_sub, const int32_t* dna_cols, int64_t n_sub,
                          int32_t* assign, int32_t* step, double* step_obj, int out_space, mcd_stats* stats);
/*
 * mcd_subinstance_sweep: `nrep` replicates of mcd_subinstance_steps in one call -- the reference's resampling
 * sweeps (clonal_proportions_resampling.py:172-201 under multiprocessing.Pool, :297-306; run_dna_batch_removal_exp.py
 * :275-287).  Replicate r is the step loop on C[rna_rows][:, dna_cols[r]]; rna_rows [m_sub] is shared (NULL = all),
 * dna_cols [nrep, n_sub] row-major HOST int32.  Replicates are independent problems and most rounds of a solve keep
 * only a few SMs busy, so `concurrency` of them (<= 32; 0 = 8) are kept in flight on worker streams with their own
 * workspaces, each on a slice of the chip.  Outputs (HOST): assign [nrep, m_sub], step [nrep, m_sub],
 * step_obj [nrep, ceil(m_sub/n_sub)] (may be NULL), cert_gap [nrep] = the replicate's largest per-step relative
 * duality gap (may be NULL).  Every replicate is solved to optimality (and certified) like a separate
 * mcd_subinstance_steps call: same objectives, same assignments except where exact ties (duplicated DNA cells) leave
 * several optima -- the trajectory of the solver depends on its grid size.
 */
int mcd_subinstance_sweep(mcd_handle h, int64_t nrep, const int32_t* rna_rows, int64_t m_sub, const int32_t* dna_cols,
                          int64_t n_sub, int32_t* assign, int32_t* step, double* step_obj, double* cert_gap,
                          int concurrency, mcd_stats* stats);
/*
 * mcd_loo_sweep: the reference's leave-one-out experiment (run_loo_experiment.py:201-319), `ncells` replicates in one
 * call on the resident M x N matrix, kept `concurrency` at a time in flight like mcd_subinstance_sweep.  Replicate r
 * leaves out RNA row q = cells[r] (HOST int32 in [0, M); repeats allowed):
 *   - the step loop runs on C with row q deleted (the M-1 other rows in ascending order, `np.delete(corrs, q, 0)`,
 *     all N columns; mcd_num_steps(M-1, N) steps); M == 1 leaves an empty replicate and no solve runs;
 *   - q takes the column of highest C[q, j] among those matched at most k_steps - 1 times by the replicate (:296-309);
 *     among exact ties the highest column index (the order a stable ascending sort, reversed, visits);
 *   - total = the step objectives, then the test cell's correlation if a column was found, summed in FP64 exactly as
 *     the reference's `float(sum(obj_scores))` sums them under CPython >= 3.12 (first term added to 0, the rest with
 *     Neumaier's compensation), so that it is bit-equal to the total of MaCroDNA.leave_one_out.
 * Required HOST outputs [ncells]: test_col (-1 if no column is eligible), test_corr (0 then), total.  Optional HOST
 * outputs (NULL to skip; a whole-biopsy sweep need not move O(M^2) data): assign / step [ncells, M-1], step_obj
 * [ncells, nsteps], match_corr [ncells, M-1] = C[row, assign] (the `corr_val` column), cert_gap [ncells] = the
 * replicate's largest per-step relative duality gap.  stats as mcd_subinstance_sweep fills it.
 * Measured throughput: not measured yet (see DESIGN.md section 5b).
 */
int mcd_loo_sweep(mcd_handle h, const int32_t* cells, int64_t ncells, int64_t k_steps, int32_t* test_col,
                  double* test_corr, double* total, int32_t* assign, int32_t* step, double* step_obj, double* match_corr,
                  double* cert_gap, int concurrency, mcd_stats* stats);
int mcd_corr_rows(mcd_handle h, const int32_t* rows, int64_t nrows, double* out, int out_space);

/*
 * Views on several GPUs of one node, from one caller.  hs[0..ndev) are distinct handles (one context named twice
 * returns MCD_ERR_INVALID; separate contexts on one device are allowed).
 *
 * mcd_share_resident: copies the correlation matrix resident on hs[0] into hs[1..ndev) -- peer copies between devices
 * (NVLink), a device-to-device copy for a handle on hs[0]'s device.  A copy is a resident matrix WITHOUT an
 * assignment: the view calls above (mcd_subinstance_steps, the sweeps, the null test, mcd_corr_rows, mcd_corr_pairs)
 * run on it, mcd_last_match_values refuses it.  Generations: every successful mcd_cell2cell / mcd_cell2cell_gather /
 * mcd_cell2cell_multi run gives the handle's matrix a new id, unique in the process; a copy carries the id of the run
 * it copied.  Every _multi call below requires that hs[1..) hold a copy of hs[0]'s CURRENT generation with the same
 * M and N, and returns MCD_ERR_INVALID otherwise: call mcd_share_resident again after every run on hs[0] (a run on
 * any of the handles, mcd_cell2cell_multi included, drops the copies it overwrites).  hs[0]'s matrix, its
 * assignment and mcd_last_match_values are unchanged by all of these calls.
 *
 * mcd_subinstance_sweep_multi / mcd_loo_sweep_multi: arguments after the handle list and outputs (HOST) as
 * mcd_subinstance_sweep / mcd_loo_sweep; ndev == 1 is exactly the single-handle call.  Replicates are dealt in
 * contiguous batches over the handles (one host thread per handle, `concurrency` workers on each), with hs[0]'s
 * solver options on every handle.  Each worker gets the cooperative grid of a single-handle call with the same
 * `concurrency` on its own device, so a replicate follows the same solver trajectory whichever device (of one kind)
 * solves it: every output is bit-identical to the single-handle call where the replicate's optimum is unique (no
 * duplicated DNA cells); with exact ties the objectives agree and the assignment is one of the optima.  A replicate
 * re-solved without the class treatment of duplicated cells is re-solved on the handle that owned it.  stats: counters
 * and sweep_fallbacks summed over the handles, cert_rel_gap / cert_max_violation the maximum, kernel_launches over
 * every handle and worker, the per-step arrays those of the handle that solved the last batch, ms_total / ms_lap the
 * host wall time from the first enqueue to the last synchronise (events of different devices are not comparable).
 *
 * mcd_null_assignments_multi: the trials are split into contiguous ranges, one per handle in proportion to its SM
 * count (a handle may get none); each device computes trials [t0, t0 + n) of the draw defined at
 * mcd_null_assignments.  A trial depends only on (seed, t, C), so sums / medians (HOST, medians may be NULL) are
 * bit-identical to mcd_null_assignments on hs[0].
 * Measured throughput: DESIGN.md section 5b (over several GPUs: not measured).
 */
int mcd_share_resident(mcd_handle* hs, int ndev);
int mcd_subinstance_sweep_multi(mcd_handle* hs, int ndev, int64_t nrep, const int32_t* rna_rows, int64_t m_sub,
                                const int32_t* dna_cols, int64_t n_sub, int32_t* assign, int32_t* step,
                                double* step_obj, double* cert_gap, int concurrency, mcd_stats* stats);
int mcd_loo_sweep_multi(mcd_handle* hs, int ndev, const int32_t* cells, int64_t ncells, int64_t k_steps,
                        int32_t* test_col, double* test_corr, double* total, int32_t* assign, int32_t* step,
                        double* step_obj, double* match_corr, double* cert_gap, int concurrency, mcd_stats* stats);
int mcd_null_assignments_multi(mcd_handle* hs, int ndev, int64_t trials, uint64_t seed, double* sums,
                               double* medians);
/* out[k] = C[rows[k], cols[k]] of the resident matrix (HOST indices, HOST out): the `corr_val` of a sub-instance's
 * matched pairs (run_loo_experiment.py:285). */
int mcd_corr_pairs(mcd_handle h, const int32_t* rows, const int32_t* cols, int64_t n, double* out);

/*
 * Random-assignment null test on the resident correlation matrix (random_assignment_test.py:233-258,
 * random_assignment_test_median.py): `trials` independent random step-wise injective assignments; sums [trials]
 * = sum of the matched correlations, medians [trials] = their median (NULL to skip).  Same distribution as the
 * reference's np.random.choice chain, not the same random stream.
 *
 * The draw of trial t (0 <= t < trials) of `seed` on the resident M x N matrix C, with mix64 the splitmix64
 * finaliser and all arithmetic in wrapping uint64:
 *   base = mix64(seed ^ mix64(t));  b = max(13, bit_length(max(M, N) - 1)) index bits;
 *   RNA key of row i    = ((mix64(base + 2i)     >> b) << b) | i,
 *   DNA key of column j = ((mix64(base + 2j + 1) >> b) << b) | j;
 *   q, r = divmod(M, N).  The RNA rows are taken in ascending key order; position p < q N takes DNA column p mod N,
 *   position p >= q N the DNA column with the (p - q N)-th smallest DNA key.
 *   sums[t] = the FP64 sum of the M matched values C[row, col]; medians[t] = 0.5 (v[(M-1)/2] + v[M/2]) of the sorted
 *   values (numpy.median).
 * A trial depends only on (seed, t, C): not on `trials`, the launch or the kernel that computes it.  The one
 * deviation from a uniformly random permutation: two keys with equal hash bits are ordered by index; the chance of
 * such a tie in a trial is about M^2 / 2^(65-b) (4e-6 at 50 000 x 10 000).  More than 2^24 cells on a side (fewer
 * than 40 hash bits) returns MCD_ERR_UNSUPPORTED.  Up to 4096 cells a side the keys are sorted in shared memory;
 * above, in per-CTA global scratch of its own (<= 1 GiB), so the resident matrix and the last run's outputs are
 * untouched.  Measured throughput: DESIGN.md section 4, "Views of the resident matrix".
 */
int mcd_null_assignments(mcd_handle h, int64_t trials, uint64_t seed, double* sums, double* medians, int out_space);

/* Number of steps ceil(M/N) (macrodna.py:118-123). */
int64_t mcd_num_steps(int64_t M, int64_t N);

#ifdef __cplusplus
}
#endif
#endif /* MACRODNA_B200_H */
