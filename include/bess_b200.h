/* bess_b200 -- C ABI of the B200-native BeSS primal-dual active-set (PDAS) hot path.
 *
 * One shared library (bess_b200/libbess_b200.so) exports two layers:
 *
 *  1. The drop-in boundary: `pywrap_bess`, argument for argument what the reference exports from
 *     /root/reference/src/bess.h:35-51 (implemented there in bess.cpp:218-281 on top of bessCpp, bess.cpp:37-214).
 *     It is exported twice: with C linkage (this header) and with the reference's own C++ linkage
 *     (_Z11pywrap_bessPdiiS_iiS_ibiiiiibibiPiiS_iS0_iS_iiiidddibiiS0_idS_iS_iS_iS_iS_S_iS_iS_iS0_iS0_), so that a SWIG
 *     wrapper generated from the reference's python/src/bess.i links against it unchanged.
 *     `bess_b200_fit` is the same call with a status code and the extensions a GPU build needs (explicit CV folds,
 *     device-resident x, per-level trace, counters).
 *
 *  2. `bessgpu_*`: the thin device shim the host path driver itself sits on (north_star: "C++ host code calls CUDA
 *     through a thin C-ABI shim").  One handle = one design matrix resident in HBM + its chain state.  Used directly by
 *     the parity tests and by bench.py's roofline probe.
 *
 * Everything computes on the GPU (sm_100a kernels); there is NO CPU fallback: without a CUDA device every compute entry
 * point returns a non-zero status and bess_b200_last_error() says why.
 *
 * Layout conventions (identical to the reference): x is ROW-major n x p (x[i*p + j], utilities.cpp:13-25), fp64; indices
 * are 0-based int32; all output buffers are caller-allocated.
 */
#ifndef BESS_B200_H
#define BESS_B200_H

#ifndef __cplusplus
#include <stdbool.h>
#endif

#ifdef __cplusplus
extern "C" {
#endif

#define BESS_B200_VERSION 100

/* ---- 1. drop-in boundary ------------------------------------------------------------------------------------- */

/* Replaces /root/reference/src/bess.h:35-51 `pywrap_bess` (bess.cpp:218-281).  Writes beta_out[0..x_col), *coef0_out,
 * *train_loss_out, *ic_out -- exactly the four outputs the reference writes (bess.cpp:277-280); nullloss/aic/bic/gic/
 * A_out/l_out are accepted and left untouched, as in the reference (SURVEY Q7).  Arguments the reference ignores on this
 * path (state, exchange_num, K_max, epsilon, tao; SURVEY Q6) are ignored here too.  On failure the three scalars are
 * set to NaN and bess_b200_last_error() holds the message (the reference would dereference null, SURVEY Q19).
 * CV folds are drawn like Metric.h:49-106 from seed $BESS_CV_SEED (default 123) -- the reference seeds from
 * std::random_device and is not reproducible under CV. */
void pywrap_bess(double *x, int x_row, int x_col, double *y, int y_len, int data_type, double *weight, int weight_len,
                 bool is_normal, int algorithm_type, int model_type, int max_iter, int exchange_num, int path_type,
                 bool is_warm_start, int ic_type, bool is_cv, int K, int *gindex, int gindex_len, double *state,
                 int state_len, int *sequence, int sequence_len, double *lambda_sequence, int lambda_sequence_len,
                 int s_min, int s_max, int K_max, double epsilon, double lambda_min, double lambda_max, int n_lambda,
                 bool is_screening, int screening_size, int powell_path, int *always_select, int always_select_len,
                 double tao, double *beta_out, int beta_out_len, double *coef0_out, int coef0_out_len,
                 double *train_loss_out, int train_loss_out_len, double *ic_out, int ic_out_len, double *nullloss_out,
                 double *aic_out, int aic_out_len, double *bic_out, int bic_out_len, double *gic_out, int gic_out_len,
                 int *A_out, int A_out_len, int *l_out);

/* A sparse design in compressed sparse column (CSC) form: column j holds the rows rowidx[colptr[j] .. colptr[j+1]) with
 * the values values[colptr[j] .. colptr[j+1]); every other entry is 0.  Offsets are 64-bit, so nnz may exceed 2^31.
 * bess_b200_fit checks the input and returns 1 with a message rather than repairing it:
 *   colptr[0] == 0, colptr non-decreasing, colptr[p] == nnz  (O(p), on the host; on the device for device arrays);
 *   0 <= rowidx[k] < n and rowidx strictly increasing inside every column (no duplicates)  (one O(nnz) device pass).
 * The values are used as given (fp64, lossless): the fit sees exactly the matrix a dense call with the same entries sees. */
typedef struct bess_b200_csc {
    const long long *colptr;  /* [p + 1] column offsets                                                                  */
    const int *rowidx;        /* [nnz] row of every stored entry                                                          */
    const double *values;     /* [nnz] value of every stored entry (explicit zeros allowed)                               */
    long long nnz;
} bess_b200_csc;

/* Extensions for bess_b200_fit (all optional; zero-initialise the struct for defaults). */
typedef struct bess_b200_ext {
    const int *fold_of_row;   /* explicit CV fold of every row (length n, values 0..K-1); NULL = draw from cv_seed   */
    unsigned cv_seed;         /* used when fold_of_row == NULL; 0 = $BESS_CV_SEED or 123                              */
    int x_on_device;          /* x is a device pointer (row-major, same layout)                                       */
    int device;               /* CUDA device ordinal, -1 = current                                                    */
    int *screening_A_out;     /* [screening_size] kept columns, ascending (List key "screening_A", bess.cpp:199)     */
    int *chosen_s_out;        /* sparsity level of the returned model                                                 */
    double *stats_out;        /* [32]: 0 n_fits, 1 n_pdas_iters, 2 n_sweeps, 3 n_batches, 4 n_boundary_ties,          */
                              /*  5 PDAS dual-sweep algorithmic bytes (8np + vectors per sweep; sweeps on the CSC      */
                              /*  arrays: 12 nnz + 8 (p + 1) + the column statistics + the n-vectors read + the        */
                              /*  partials written), 6 kernel_launches, 7 trace_len,                                   */
                              /*  8..15 device ms per kernel category (profile != 0): screening sweep, PDAS dual      */
                              /*  sweeps, finish, top-k, chain kernels, other, normalisation passes, H2D upload;      */
                              /*  16..23 launches per category; 24 algorithmic bytes of the screening sweep (8np;     */
                              /*  sparse design: 12 nnz + 8 (p + 1) + the n-vectors it reads); 7 covers a CSC copy;   */
                              /*  25 sweep row splits; 26 algorithmic bytes of the normalisation / x_j.x_j passes;    */
                              /*  27..31 host wall-clock ms by phase: load, screening, normalisation, fold / chain    */
                              /*  set-up, path                                                                        */
    int profile;              /* record CUDA events around every kernel category on the engine's stream               */
    /* ---- multi-GPU, columns of x sharded over `world` processes (one per GPU); world <= 1: single GPU.            */
    /* x then holds columns [col_lo, col_lo + x_col) = bess_b200_shard_range(p_total, world, rank) of the design,      */
    /* gindex is ignored, always_select / beta_out (length p_total) / screening_A_out use GLOBAL column numbers, and   */
    /* every rank must make the same call with the same non-x arguments.  Candidates and active columns travel over   */
    /* NCCL (all-gather / all-reduce on the library's own communicator).                                              */
    int world, rank;
    long long col_lo, p_total;
    const void *nccl_unique_id; /* 128 bytes from bess_b200_nccl_unique_id() on rank 0, broadcast by the caller       */
    double *chosen_lambda_out;  /* ridge level of the returned model (List key "lambda", path.cpp:129)                 */
    int beta_out_zeroed;        /* beta_out already holds zeros (e.g. calloc): only the non-zero coefficients are written */
    int cv_reduce_over_ranks;   /* world > 1, sequential path, CV + screening: REPEATED K-fold CV -- every rank passes its  */
                                /* own folds (cv_seed / fold_of_row), the per-level CV losses are averaged over the ranks   */
                                /* (one ncclAllReduce) before the level is chosen; all ranks return the same model          */
    int cv_seed_set;            /* non-zero: cv_seed is taken as given, INCLUDING 0 (cv_seed == 0 alone means "default")     */
    int *tie_exact_out;         /* bit 0: the call met a boundary tie of a top-k selection and was repeated with the tied     */
                                /* selections resolved by the reference's own std::nth_element (utilities.cpp:179-188);        */
                                /* bit 1: the fast pass met a numerically dependent active column (or a non-finite result)     */
                                /* and the call was repeated with the rank-revealing solver; bit 2: at least one normal-      */
                                /* equation solve was truncated the way colPivHouseholderQr / pivoted ldlt truncate            */
                                /* (Algorithm.h:1134, 1171; an exactly duplicated column inside the active set)                */
    double *resident_out;       /* [152] counters of the resident-path kernel (gaussian family, design resident in L2: the   */
                                /* whole PDAS path is ONE cooperative launch): 0 launches, 1 PDAS iterations, 2 full-vector */
                                /* select fallbacks, 3 path steps, 8..15 clock ticks by phase of chain owner 0, 16..18 of    */
                                /* sweeper 0; 24 + 4 i ..: chain owner i: busy ticks, longest phase, ticks in fallback        */
                                /* selects, fits solved; all zero when the multi-kernel path ran                             */
    int fold_shard;             /* world > 1 with the WHOLE design on every rank (col_lo / p_total unused), CV: the K fold    */
                                /* chains of Metric::test_loss (Metric.h:150-195) are dealt over the ranks (chain c on rank   */
                                /* c % world, bess_b200_chain_owner), every rank runs the full-data chain, and only the       */
                                /* per-fold test losses are all-reduced -- SURVEY 8e axis A inside ONE call; every rank       */
                                /* returns the same model, bit-identical to the single-GPU call                               */
    const bess_b200_csc *x_csc; /* non-NULL: the design is sparse (see bess_b200_csc); x must then be NULL, x_row / x_col give */
                                /* n and p, and x_on_device = 1 means the three arrays are device pointers (read in place,   */
                                /* never written).  Screening densifies only the kept columns.  Without screening and groups, */
                                /* a design whose dense form is over 1 GiB and at least 24 times its CSC bytes (12 nnz +      */
                                /* 8 (p + 1)), or larger than the device's memory, is swept on its non-zeros and only the     */
                                /* active columns are expanded; any other is densified on the device (n * p * 8 bytes must    */
                                /* fit).  Single GPU only (world <= 1); screening together with groups is refused as for      */
                                /* dense designs                                                                              */
    int *sparse_sweeps_out;     /* 1 when the call's PDAS sweeps ran on the CSC arrays of x_csc, else 0; may be NULL          */
} bess_b200_ext;

/* Same arguments and outputs as pywrap_bess, returns 0 on success.  The per-level trace of the call (what the reference's
 * R build returns as beta_all/coef0_all/train_loss_all/ic_all, path.cpp:116-123, 376-380) is kept until the next call
 * on this thread; fetch it with bess_b200_trace. */
int bess_b200_fit(double *x, int x_row, int x_col, double *y, int y_len, int data_type, double *weight, int weight_len,
                  bool is_normal, int algorithm_type, int model_type, int max_iter, int exchange_num, int path_type,
                  bool is_warm_start, int ic_type, bool is_cv, int K, int *gindex, int gindex_len, double *state,
                  int state_len, int *sequence, int sequence_len, double *lambda_sequence, int lambda_sequence_len,
                  int s_min, int s_max, int K_max, double epsilon, double lambda_min, double lambda_max, int n_lambda,
                  bool is_screening, int screening_size, int powell_path, int *always_select, int always_select_len,
                  double tao, double *beta_out, int beta_out_len, double *coef0_out, double *train_loss_out,
                  double *ic_out, const bess_b200_ext *ext);

/* Trace of the last bess_b200_fit/pywrap_bess on this thread.  Any pointer may be NULL.  beta_all is [len][p] and only
 * filled for the sequential path.  Returns the trace length. */
int bess_b200_trace(int *s_all, int *l_all, double *coef0_all, double *train_loss_all, double *ic_all, double *beta_all,
                    int p);

/* Metric.h:49-106 with the seed pinned: fold index of every row. */
/* lambda of every evaluated (s, lambda) pair of the last call, in evaluation order (same order as bess_b200_trace). */
int bess_b200_trace_lambda(double *lambda_all);
int bess_b200_cv_fold_ids(int n, int K, unsigned seed, int *fold_of_row_out);

/* ncclGetUniqueId through the library's run-time-loaded NCCL: call on rank 0, broadcast the 128 bytes to all ranks. */
int bess_b200_nccl_unique_id(void *out128);

/* Device-side design generator (R/R/gen.data.R:110-118, cortype 1): fills the DEVICE buffer x_dev (row-major n x p, leading
 * dimension ld >= p) with rows ~ MVN(0, Sigma), Sigma_jk = rho^|j-k| (rho = 0: iid N(0,1)); counter-based (Philox4x32-10 +
 * Box-Muller), so x[i][j] is a pure function of (seed, i, j).  For benchmarks whose design must not cross PCIe. */
int bess_b200_gen_design(double *x_dev, int n, long long p, long long ld, double rho, unsigned long long seed, int device);

/* The same for every correlation type of gen.data (R/R/gen.data.R:110-118, 167-181): cortype 1 = the call above; 2 =
 * exchangeable, Sigma = rho + (1 - rho) I (one common factor per row, rho in [0, 1)); 3 = the banded design of gen.data
 * cortype 3 and of python/bess/gen_data.py:25-30 (iid columns centred and scaled to norm sqrt(n), then
 * x_j = X_j + rho (X_{j-1} + X_{j+1}) inside, x_j = X_j at both ends). */
int bess_b200_gen_design_cortype(double *x_dev, int n, long long p, long long ld, double rho, unsigned long long seed, int cortype,
                                 int device);

const char *bess_b200_last_error(void);
int bess_b200_version(void);
/* number of CUDA devices visible (0 = no GPU: every compute call will fail) */
int bess_b200_device_count(void);

/* ---- 2. device shim ------------------------------------------------------------------------------------------ */
typedef struct bessgpu_handle bessgpu_handle;

int bessgpu_create(bessgpu_handle **h, int device);
int bessgpu_destroy(bessgpu_handle *h);
/* upload (or device-to-device copy) the design; replaces the by-value copies of bess.cpp:233/61 and Algorithm.h:58 */
int bessgpu_load(bessgpu_handle *h, const double *x, int n, int p, int x_on_device, const double *y,
                 const double *weight, int model_type);
/* the same for a CSC design (bess_b200_csc, same validation); it stays sparse until bessgpu_screen keeps its columns */
int bessgpu_load_csc(bessgpu_handle *h, const long long *colptr, const int *rowidx, const double *values, int n, int p,
                     long long nnz, int on_device, const double *y, const double *weight, int model_type);
/* screening.cpp:26-105; out: screening_size kept columns, ascending */
int bessgpu_screen(bessgpu_handle *h, int screening_size, const int *always_select, int n_always, int *screening_A_out);
/* column-sharded screening (multi-GPU): the local top-`size` candidates of this handle's columns as (utility, local
 * column index) pairs, ascending index; the design stays untouched.  count_out = min(size, p_local). */
int bessgpu_screen_local(bessgpu_handle *h, int screening_size, const int *always_select, int n_always,
                         double *vals_out, int *idx_out, int *count_out);
/* dst_dev[i*ld + pos[q]] = x[i][cols[q]], q < m: copies chosen columns into a DEVICE buffer (row-major, leading dim ld) */
int bessgpu_gather_columns(bessgpu_handle *h, const int *cols, const int *pos, int m, double *dst_dev, long long ld);
/* Data.h:41-77 + normalize.cpp:20-86 */
int bessgpu_normalize(bessgpu_handle *h, int data_type, int is_normal);
/* group selection (Data.h:53-61: g_index = first column of every group, ascending from 0; at most 64 variables per
 * group).  Call after bessgpu_normalize and before bessgpu_setup_chains; sparsity levels, kcap and always_select then
 * count groups (Algorithm.h:1097-1129, 1206-1263, 1324-1367, 1497-1568; utilities.cpp:113-177). */
int bessgpu_set_groups(bessgpu_handle *h, const int *g_index, int n_groups);
int bessgpu_get_norm(bessgpu_handle *h, double *x_mean_out, double *x_norm_out, double *y_mean_out);
/* the engine's current dense design (after screening: the kept columns; after normalize: normalised), row-major
 * n x p into host memory */
int bessgpu_design(bessgpu_handle *h, double *x_out);
/* Metric.h:49-129 (fold row lists, per-fold x_j.x_j) + workspace for supports up to kcap */
int bessgpu_setup_chains(bessgpu_handle *h, int K, const int *fold_of_row, int kcap, int max_iter, int warm_start,
                         const int *always_select, int n_always);
/* Algorithm::fit (Algorithm.h:113-171) for `nch` chains at sparsity T in lock-step.  Outputs are [nch] / [nch][T]. */
int bessgpu_run_batch(bessgpu_handle *h, int T, const int *chains, int nch, int new_path_step, int *l_out,
                      double *coef0_out, int *A_out, double *beta_A_out);
/* the same with a ridge level and supports of different width per chain (group selection): ks_out[i] columns of chain
 * i's support are written to A_out / beta_A_out rows of leading dimension ld */
int bessgpu_run_batch_groups(bessgpu_handle *h, int T, const int *chains, int nch, int new_path_step, double lambda,
                             int *l_out, double *coef0_out, int *ks_out, int *A_out, double *beta_A_out, int ld);
/* Metric::train_loss (kind 0) / fold test loss (kind 1) of a chain's current model */
int bessgpu_losses(bessgpu_handle *h, const int *chain, const int *kind, const int *fold, int njobs, double *out);
/* roofline probe: mean device time (ms) of one dual-sweep launch over all chain slots and its algorithmic bytes */
int bessgpu_time_dual_sweep(bessgpu_handle *h, int reps, float *ms_out, double *bytes_out);
/* test probe, after a batch returned: the sacrifice of every chain of `chains` for its current model (gradient vectors
 * published again from the chain's support, coefficients and intercept), through the dispatch a fit of this batch uses,
 * at ridge level `lambda`.  bd_out: [nch][p], or [nch][number of groups] with groups.  info_out[8]: [0] what ran (1
 * streaming column sweep, 2 bulk-TMA column sweep, 3 group kernels, 4 the sweep over a sparse design's CSC arrays),
 * [1] chain slots FS, [2] columns per thread (4: lanes per column), [3] row splits, [4] rows per split, [5] group kernels
 * launched (bits: 1 serial, 2 warp, 4 / 8 / 16 batched for widths <= 2 / 4 / 8, 32 wide; 4: columns swept by a CTA each) */
int bessgpu_sacrifice(bessgpu_handle *h, const int *chains, int nch, double lambda, double *bd_out, int *info_out);
int bessgpu_stats(bessgpu_handle *h, double *out8);
/* stand-alone exact top-k (utilities.cpp:179-188 max_k): host vals[n] -> ascending indices; tie_out = 1 when keys equal to
 * the k-th straddle the boundary */
int bessgpu_topk(const double *vals, int n, int k, int *idx_out, int *tie_out);
/* the same by the screening's select (a device-wide radix select when n > 16384): same indices, order and tie flag */
int bessgpu_screen_select(const double *vals, int n, int k, int *idx_out, int *tie_out);

/* pgs_path geometry (path.cpp:414-577, pure host code): the points where the search line p + t*u leaves the box
 * [s_min, s_max] x [log_lambda_min, log_lambda_max]; a2_out / b2_out receive the first two in the reference's edge order.
 * Returns the number of crossings found (the Powell search needs 2). */
int bess_b200_pgs_line_box(const double *p2, const double *u2, int s_min, int s_max, double log_lambda_min, double log_lambda_max,
                           double *a2_out, double *b2_out);

/* ---- 3. multi-GPU host helpers (pure host code, no CUDA) ------------------------------------------------------ */
/* contiguous column shard [lo, hi) of rank r out of `world` (SURVEY 8e axis B) */
void bess_b200_shard_range(long long p, int world, int rank, long long *lo, long long *hi);
/* chain -> rank assignment for fold sharding (SURVEY 8e axis A): round-robin, chain 0 on rank 0 */
int bess_b200_chain_owner(int chain, int world);
/* The chains rank `rank` runs in a fold-sharded call (ext.fold_shard) with K folds: chains_out[0] = 0 (full data), then its
 * fold chains (c % world == rank; on every rank also chain K when path_type != 1, path.cpp:314-319); counts_out[i] = 1
 * when the rank contributes the test loss of chains_out[i].  Both arrays need K + 1 entries.  Returns the number of
 * chains, -1 on bad arguments.  Host only. */
int bess_b200_fold_shard_chains(int K, int world, int rank, int path_type, int *chains_out, int *counts_out);
/* merge per-rank local top-k candidate lists (value, global index) into the global top-k, ascending indices.
 * Total order: larger value first, lower index first.  vals/idx: [count]. */
int bess_b200_merge_candidates(const double *vals, const int *idx, int count, int k, int *idx_out);

#ifdef __cplusplus
}
#endif
#endif /* BESS_B200_H */
