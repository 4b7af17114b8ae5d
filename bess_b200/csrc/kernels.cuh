// Kernel-side declarations shared by kernels.cu (device code + launchers) and engine.cu (orchestration).
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include "engine.h"

namespace bess {

constexpr int NVEC = 8;          // per-chain scratch vectors of length n
constexpr int SWEEP_NT = 128;    // threads per dual-sweep CTA
constexpr int SWEEP_RC = 64;     // rows per TMA-staged chunk of the gradient vectors
constexpr int FIT_NT = 512;      // threads per chain_fit CTA (one CTA per chain)
constexpr int TOPK_NT = 1024;
constexpr int TOPK_LMAX = 16384; // keys per top-k slice held in shared memory (128 KB)
// one-launch normalisation: columns per CTA (a warp load covers 4 rows x 64 bytes; p / 8 CTAs keep every SM streaming), and
// the most rows whose n x NR_TC slab the gather-fused variant stages in shared memory (227 KB less 1 KB for its static arrays)
constexpr int NR_TC = 8;
constexpr int NR_SLAB_ROWS = (227 * 1024 - 1024) / (NR_TC * 8);
constexpr int CLMAX = 16;        // max thread-block cluster size of chain_fit_kernel (8 = the portable limit; 16-CTA
                                 // clusters, one per GPC, are used when a batch has few chains: single-chain paths, fold shards)

// sweep modes
enum { MODE_D = 0, MODE_DH = 1, MODE_COX = 2 };
// finish epilogues
enum { EPI_RAW = 0, EPI_SACR_LM = 1, EPI_SACR_GLM = 2, EPI_SACR_COX = 3, EPI_SCREEN_LM = 4 };

// Everything the kernels need, passed by value.
struct Dev {
    // design (row-major n x ldx, ldx even, zero padded)
    double *X;
    long long ldx;
    int n, p;
    int family;
    int FS;      // chain-slot stride of the sweep vectors (compile-time FT of the sweep kernel)
    int kcap;    // max support size
    int ldA;     // leading dim of gathered active columns: kcap + 2 rounded to even
    int max_iter;
    int warm;
    double lambda;      // ridge level of the running batch (Algorithm::lambda_level; 0 for best-subset selection)
    // per-chain tables (index with chain id c)
    int *rows;          // [MAXC][n] train rows (ascending) of the chain's mask
    int *ntrain;        // [MAXC]
    double *ytr, *wtr;  // [MAXC][n] compacted response / weights
    int *ks;            // [MAXC] current support size
    int *A;             // [MAXC][kcap] current support
    double *bA;         // [MAXC][kcap] coefficients on the support
    double *coef0;      // [MAXC]
    double *coef0_level;// [1]  Algorithm::coef0_init of the current path step (path.cpp:57)
    int *Anew;          // [MAXC][kcap] output of top-k
    int *hist;          // [MAXC][hist_rows][kcap]  A_list (Algorithm.h:141-143)
    int hist_rows;      // max_iter + 2
    int *l;             // [MAXC]
    int *done;          // [MAXC]
    int *tie;           // [MAXC] boundary-tie flag of the last top-k
    int *tie_acc;       // [MAXC] boundary ties consumed by the chain's fits since chain_begin
    int *n_active;      // chains of the running batch that have not met the stopping rule yet (one of two alternating
                        // counters: consecutive batches use different ones)
    const int *prev_active; // the counter of the batch enqueued before this one.  A batch may be enqueued BEHIND an
                        // unfinished one (the next path step, speculatively, while the host still waits for the current
                        // one): chain_begin_kernel then finds *prev_active != 0, zeroes its own counter and the whole
                        // batch falls through its gates without touching any state; the host re-enqueues it later.
    const int *gate;    // == n_active while a batch runs: every per-iteration kernel returns at once when *gate == 0,
                        // so iterations can be enqueued speculatively without a host round trip; nullptr = no gate
    double *betaD;      // [MAXC][p] dense beta (for the sacrifice)
    double *XA;         // [MAXC][n][ldA] gathered active columns (+ intercept / working response columns)
    double *XB;         // [MAXC][n][ldA] cox: risk-set means
    double *vec;        // [MAXC][NVEC][n]
    double *Smat;       // [MAXC][2][ldA*ldA] normal equations (when they do not fit in smem) / Cox second Gram
    double *Spart;      // [MAXC][CLcap][nmat][ldA*ldA] per-CTA partial Grams of a cluster (nullptr when CLcap == 1)
    double *cw;         // [MAXC][CLMAX][4][ldA] cluster exchange vectors
    // column-sharded mode (multi-GPU axis B): X holds columns [col_lo, col_lo + p) of a wider design; supports (A, Anew,
    // hist) carry GLOBAL column indices, betaD / bd / xtx are local
    // group selection (group.cu): columns [gidx[g], gidx[g] + gsz[g]) form group g.  Anew / hist / the top-k work on
    // group ids, A / bA / ks / AnewCols on columns; kcap is the COLUMN capacity of a support.
    int grouped;        // 0: every column is its own group, the fields below are unused
    int N;              // number of groups
    int gmax;           // widest group
    const int *glist;   // narrow groups (<= GMAX variables) ordered by width class <= 2 | <= 4 | <= 8
    int gcls_off[4];    // class k = glist[gcls_off[k] .. gcls_off[k + 1])
    const int *gidx;    // [N]
    const int *gsz;     // [N]
    int *Tc;            // [MAXC] number of columns of the groups chosen by the last top-k
    int *AnewCols;      // [MAXC][kcap] those columns (find_ind, utilities.cpp:113-130)
    int sharded;
    int col_lo;
    int ax_ext;         // X_A comes from AXr (column-sharded mode, sparse design): chain_fit gathers its train rows from
                        // there and keeps AXk; the loss kernel reads AXk
    // sparse design swept on its non-zeros (ccp != nullptr; X unused): the design the fits see is the implicit
    // x~_ij = ((x_ij - cmean[j]) * cmul[j]) * crm[i] (crm == nullptr: 1), an unstored x_ij reading 0
    const long long *ccp;
    const int *cri;
    const double *ccv;
    const double *cmean, *cmul, *crm;
    double *csum;       // [2][FS] per-iteration sums of the CSC sweep: 0 = sum_i G'_i (G' = crm o G in MODE_D), 1 = sum_i W_i
    double *cpre;       // [n][FS] cox: prefix sums of C2 over the rows (inclusive)
    int csc_g;          // lanes per column of the CSC sweep (2, 8 or 32)
    long long clong_thr;// columns with more entries are swept by a CTA each ...
    const int *clong;   // ... these [nlong]
    int nlong;
    long long csc_nnz;
    double *AXr;        // [MAXC][n][ldXr] active columns of this iteration for ALL rows, summed over ranks (ldXr = T)
    double *AXk;        // [MAXC][n][ldXk] all-row active columns of each chain's CURRENT support (losses)
    int ldXr, ldXk;
    int fit_smem_doubles; // dynamic shared memory of the chain kernels, in doubles (fit_smem_doubles())
    int CLcap;          // largest cluster size the workspaces were sized for
    int nmat;           // Gram matrices per fit step: 2 for cox, else 1
    double *xtx;        // [MAXC][p] x_j.x_j over the chain's train rows (gaussian only)
    // sweep vectors [n][FS]
    double *G, *W, *TH, *C2;
    // sweep outputs
    double *part;       // [S][NQ][FS][pstride]
    double *c2sum;      // [S][FS]
    double *bd;         // [FS][pstride]
    long long pstride;
    int S;              // row splits
    int rows_per_split; // multiple of 2
};

struct BatchDesc {
    int nch;
    int chain[MAXC];
    int T;
    int new_path_step;
    int CL;  // cluster size of chain_fit_kernel for this batch
};

struct LossDesc {
    int njobs;
    int chain[2 * MAXC];
    int kind[2 * MAXC];
    int fold[2 * MAXC];
};

// ---- launchers (kernels.cu) ----
void launch_dual_sweep(const Dev &d, int mode, cudaStream_t st);
// bulk-TMA pipelined variant for batched chains (sweep_tma.cu); launch_dual_sweep dispatches to it when FS >= 2
bool sweep_uses_tma(const Dev &d);
void launch_dual_sweep_tma(const Dev &d, int mode, cudaStream_t st);
// columns per thread of the sweep launch_dual_sweep runs for d.FS and `mode` (sweep_tma_cpt: of the bulk-TMA kernel)
int sweep_cpt(const Dev &d, int mode);
int sweep_tma_cpt(int FS, int mode);
void launch_finish(const Dev &d, int mode, int epi, const BatchDesc &b, double *raw_out, cudaStream_t st);
void launch_pin(const Dev &d, double *vals, long long stride, int nch, const int *idx, int nidx, cudaStream_t st);
// `gate`: see Dev::gate
// exact top-k of `vals` ([nch][stride], first n_in of each row) -> out_idx [nch][out_ld] ascending; uses ping-pong scratch
// idx0: optional explicit index of every input key ([nch][stride], ascending inside each row); default = position
int launch_topk(const double *vals, long long stride, int n_in, int k, int nch, int *out_idx, int out_ld, int *tie,
                double *ck0, int *ci0, double *ck1, int *ci1, long long cstride, cudaStream_t st,
                const int *gate = nullptr, const int *idx0 = nullptr);
// the exact top-k of the screening (ascending indices, larger key first then lower index, the tie flag of launch_topk) by a
// device-wide radix select when p > TOPK_LMAX; otherwise, or when the boundary bin is too large, launch_topk.  scratch:
// screen_select_scratch_bytes(p) device bytes; ck*/ci*/cstride as for launch_topk.  Returns the number of launches.
size_t screen_select_scratch_bytes(int p);
int launch_screen_select(const double *vals, int p, int k, int *out_idx, int *tie, void *scratch, double *ck0, int *ci0,
                         double *ck1, int *ci1, long long cstride, cudaStream_t st);
// finish + pin + top-k in one kernel (p <= TOPK_LMAX): reads the sweep partials, writes d.Anew / d.tie for chains
// cmin .. cmin + nspan - 1 that have not met the stopping rule
void launch_topk_fused(const Dev &d, int mode, int epi, int cmin, int nspan, int k, const int *always, int n_always,
                       cudaStream_t st);
// ---- column-sharded mode
struct Cand {
    double v;
    long long idx;
};
// out[f][a] = (vals[f][sel[f][a]], sel[f][a] + offset) for a < kloc, padded with (-1, INT_MAX) up to kpad
void launch_pack_candidates(const double *vals, long long stride, const int *sel, int sel_ld, int kloc, int kpad,
                            long long offset, int nch, Cand *out, int out_ld, const int *gate, cudaStream_t st);
// in [world][nch][in_ld] -> mv/mi [nch][world * k] (rank-major, so index-ascending)
void launch_unpack_candidates(const Cand *in, int world, int nch, int in_ld, int k, double *mv, int *mi, long long mstride,
                              const int *gate, cudaStream_t st);
// AXs[c][i][a] = X[i][Anew[c][a] - col_lo] when this rank owns the column, else 0   (ld = T)
void launch_gather_active(const Dev &d, const BatchDesc &b, double *AXs, cudaStream_t st);
// Xn[i][q] = X[i][sel[q] - col_lo] when owned else 0
void launch_gather_owned_cols(const double *X, long long ldx, int n, int p_local, long long col_lo, const int *sel, int m,
                              double *Xn, long long ldn, cudaStream_t st);
void launch_chain_begin(const Dev &d, const BatchDesc &b, cudaStream_t st);
// ---- group selection (group.cu): sweep + group sacrifice in one kernel -> d.bd[chain][group]; selected groups -> columns
// returns the GSAC_* bits of the kernels it launched
enum { GSAC_SERIAL = 1, GSAC_WARP = 2, GSAC_BATCHED2 = 4, GSAC_BATCHED4 = 8, GSAC_BATCHED8 = 16, GSAC_WIDE = 32 };
int launch_group_sacrifice(const Dev &d, const BatchDesc &b, cudaStream_t st);
void launch_group_expand(const Dev &d, const BatchDesc &b, cudaStream_t st);
// ---- explicit warm-start state of a chain.  pgs_path re-seeds Algorithm::beta_init / coef0_init by hand (zeros at the
// start of every line search, path.cpp:590-592; the snapshot after the first fit for the backward walk of seq_search,
// path.cpp:1040-1041, 1084-1085; a stale value for its last fit, path.cpp:1212-1217), so the driver needs to save,
// restore and clear what a chain would otherwise simply carry forward.
struct StateSlots {
    int *A;         // [NSLOT][kcap]
    double *bA;     // [NSLOT][kcap]
    int *ks;        // [NSLOT]
    double *coef0;  // [NSLOT]
};
// SAVE: slot_beta <- (A, beta_A, ks) and slot_coef0 <- coef0 of `chain`.  LOAD: the reverse (also rewrites the dense beta
// and re-gathers X_A).  ZERO: beta = 0, coef0 = 0.  A negative slot leaves that half untouched.
void launch_chain_state(const Dev &d, int chain, int op, int slot_beta, int slot_coef0, const StateSlots &s, cudaStream_t st);
void launch_chain_fit(const Dev &d, const BatchDesc &b, cudaStream_t st);
// test hook: the gradient vectors (G, W, TH, C2) of every chain of the batch from its stored state (A, beta_A, coef0), X_A
// re-gathered first -- what chain_begin_kernel publishes, without touching the chains' iteration state
void launch_chain_gradient(const Dev &d, const BatchDesc &b, cudaStream_t st);
void launch_losses(const Dev &d, const LossDesc &jobs, const int *testrows, const int *ntest, const double *y,
                   const double *w, const double *lfact, double *scratch, double *out, cudaStream_t st);
void launch_norm_factors(const double *h, int p, double sn, double *norm_out, double *mul_out, cudaStream_t st);
// one-launch normalisation of an L2-resident design (gmean = w / n or nullptr for no centring, wnorm = w, rowmul or nullptr)
void launch_normalize_resident(double *X, long long ldx, int n, int p, const double *gmean, const double *wnorm,
                               const double *rowmul, double sn, double *mean_out, double *norm_out, cudaStream_t st);
// the same with screening's gather of the kept columns fused in: Xn[:, q] <- normalised X[:, cols[q]], q < p (n <= NR_SLAB_ROWS)
void launch_gather_normalize(const double *X, long long ldx, const int *cols, double *Xn, long long ldn, int n, int p,
                             const double *gmean, const double *wnorm, const double *rowmul, double sn, double *mean_out,
                             double *norm_out, cudaStream_t st);
void launch_center_scale(double *X, long long ldx, int n, int p, const double *sub, const double *mul,
                         const double *rowmul, cudaStream_t st);
void launch_gather_cols(const double *X, long long ldx, int n, const int *cols, int pnew, double *Xn, long long ldn,
                        cudaStream_t st);
void launch_gather_cols_pos(const double *X, long long ldx, int n, const int *cols, const int *pos, int m, double *dst,
                            long long ld, cudaStream_t st);
void launch_screen_glm(const double *X, long long ldx, int n, int p, const double *y, const double *w, int family,
                       double *util, cudaStream_t st);
// ---- sparse (CSC) designs: colptr [p + 1] 64-bit offsets, rowidx / values [nnz]
// flag |= CSC_BAD_COLPTR / CSC_BAD_ROW / CSC_UNSORTED (one O(nnz) pass; a column whose offsets are bad is not read)
enum { CSC_BAD_COLPTR = 1, CSC_BAD_ROW = 2, CSC_UNSORTED = 4 };
void launch_csc_check(const long long *colptr, const int *rowidx, int n, int p, long long nnz, int *flag, cudaStream_t st);
// Xn[rowidx[k]][q] = values[k] for the entries of column cols[q] (cols == nullptr: column q), q < m; Xn zero-filled
void launch_csc_densify(const long long *colptr, const int *rowidx, const double *values, const int *cols, int m, double *Xn,
                        long long ldn, cudaStream_t st);
// gaussian screening utility (x_j.y / x_j.x_j)^2 of every column over its non-zeros
void launch_screen_csc_lm(const long long *colptr, const int *rowidx, const double *values, int p, long long nnz,
                          const double *y, double *util, cudaStream_t st);
// screen_glm_kernel with a CSC column reader (absent rows read as 0.0): the same arithmetic in the same order
void launch_screen_glm_csc(const long long *colptr, const int *rowidx, const double *values, int n, int p, const double *y,
                           const double *w, int family, double *util, cudaStream_t st);
// ---- sparse design swept on its non-zeros (Dev::ccp; DESIGN 3.12 "without screening")
// column statistics of normalize.cpp:20-86 over the stored entries: mean_j = sum_stored x g (g = w / n; nullptr: no centring,
// mean 0), norm_j = sqrt(sum_stored w (x - m)^2 + m^2 (sumw - sum_stored w)), mul_j = sn / norm_j
void launch_csc_stats(const long long *colptr, const int *rowidx, const double *values, int p, const double *g,
                      const double *w, double sumw, double sn, double *mean_out, double *norm_out, double *mul_out,
                      cudaStream_t st);
// the sums of the sweep vectors (Dev::csum, Dev::cpre) and the sweep itself: the partials of dual_sweep_kernel with S = 1
void launch_csc_sweep(const Dev &d, int mode, cudaStream_t st);
// list[0, *count) <- the columns with more than thr entries (any order); *count must be zero on entry
void launch_csc_long_list(const long long *colptr, int p, long long thr, int *list, int *count, cudaStream_t st);
// which 0: AXr[c] <- x~ of the columns Anew[c][0, T) for all rows (gated; chains that are done skip);
// which 1: AXk[c] <- x~ of the columns A[c][0, ks[c]) (the chain's stored support)
void launch_csc_gather(const Dev &d, const BatchDesc &b, int which, cudaStream_t st);
// out[i * ld + q] = x~_{i, q} for every column q < p (the normalised dense design)
void launch_csc_expand(const Dev &d, double *out, long long ld, cudaStream_t st);
// device-side gen.data design (gen_design.cu): X[i][j], row-major n x p with leading dimension ld
void launch_gen_design(double *X, long long ld, int n, long long p, double rho, unsigned long long seed, cudaStream_t st);
void launch_gen_design_cortype(double *X, long long ld, int n, long long p, double rho, unsigned long long seed, int cortype,
                               double *scratch, cudaStream_t st);
size_t fit_smem_bytes(const Dev &d);
int fit_smem_doubles(int ldA, int kcap);
int chain_cluster_size(const Dev &d, int T, int nch);
void configure_kernels();
void debug_set(int key, int val);
void debug_get(unsigned long long *out32);
// truncated (rank-deficient) normal-equation solves of the chain kernels since the last call (synchronises the device)
long long debug_take_rankdef();
// singular normal-equation systems of more than 63 unknowns (solution returned as NaN) since the last call
long long take_wide_singular();
void debug_solve(const double *S, int lds, int mm, double *x_out, int impl, int reps, double *ticks_out);
void debug_gram(const double *V, int ldv, int nrows, int mm, const double *wt, double *S_out, int impl, int reps,
                double *ticks_out);
// path_out[0] = solver that finished (chain_fit.cu SOLVE_*), [1] = truncated solves, [2] = wide singular solves
void debug_solve_path(const double *S, int lds, int mm, int kcap, double *x_out, int *path_out);
void debug_gram_rows(const double *V, int ldv, int r0, int r1, int mm, const double *wt, double *S_io, int kcap, int impl);


}  // namespace bess
