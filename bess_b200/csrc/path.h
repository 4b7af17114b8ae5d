// Host-side driver of the BeSS PDAS path: the B200-native counterpart of bessCpp
// (/root/reference/src/bess.cpp:37-214), sequential_path (/root/reference/src/path.cpp:25-132),
// gs_path (path.cpp:134-389) and the Metric family (/root/reference/src/Metric.h).
// Control flow (which sparsity level next, argmin of the criterion) stays on the host; every fit,
// sweep, selection and loss runs on the device through bess::Engine.
#pragma once
#include <string>
#include <vector>

#include "engine.h"

namespace bess {

struct BessArgs {
    // --- the 30 bessCpp arguments (bess.h:20-33); x is row-major n x p as in pywrap_bess
    const double *x = nullptr;
    int n = 0, p = 0;
    const double *y = nullptr;
    int data_type = 1;
    const double *weight = nullptr;
    bool is_normal = true;
    int algorithm_type = 1, model_type = 1, max_iter = 20, exchange_num = 2;
    int path_type = 1;
    bool is_warm_start = true;
    int ic_type = 1;
    bool is_cv = false;
    int K = 5;
    std::vector<double> state;        // accepted and ignored (SURVEY Q6)
    std::vector<int> sequence;
    std::vector<double> lambda_seq;
    int s_min = 1, s_max = 1, K_max = 10;
    double epsilon = 10.0, lambda_min = 0.0, lambda_max = 0.0;
    int nlambda = 1;
    bool is_screening = false;
    int screening_size = 1, powell_path = 1;
    std::vector<int> g_index;
    std::vector<int> always_select;
    double tao = 1.1;
    // --- extensions (not in the reference)
    const int *fold_of_row = nullptr;  // explicit CV folds (length n); else drawn like Metric.h:49-106 from cv_seed
    unsigned cv_seed = 123;
    bool x_on_device = false;          // x is a device pointer (bench "resident" mode)
    int device = -1;
    bool profile = false;              // CUDA-event timing per kernel category
    // multi-GPU, columns sharded (SURVEY 8e axis B): x holds columns [col_lo, col_lo + p) of a p_total-column design,
    // always_select / the returned beta use GLOBAL column numbers; nccl_id = the 128-byte ncclUniqueId of the job
    int world = 1, rank = 0;
    long long col_lo = 0, p_total = 0;
    const void *nccl_id = nullptr;
    // repeated K-fold CV over the ranks: each rank passes its own folds (cv_seed / fold_of_row); the per-level CV losses
    // are averaged over the ranks before the level is chosen, so every rank returns the same model.  Sequential path with
    // CV and screening only (the ranks then share the screened design but not the folds).
    bool cv_reduce_over_ranks = false;
    // SURVEY 8e axis A inside ONE call: every rank holds the WHOLE design and makes the same call; the K fold chains of
    // Metric::test_loss (Metric.h:150-195) are dealt over the ranks (bess_b200_chain_owner), every rank runs the full-data
    // chain, and only the per-fold test losses are reduced (one NCCL all-reduce of K numbers per evaluated level; the
    // sequential path reduces its whole levels x K matrix once).  world / rank / nccl_id as above, col_lo / p_total unused.
    bool fold_shard = false;
    // sparse design (bess_b200_csc): x is then null and the three arrays (device pointers when x_on_device) give n x p
    bool csc = false;
    const long long *csc_colptr = nullptr;
    const int *csc_rowidx = nullptr;
    const double *csc_values = nullptr;
    long long csc_nnz = 0;
};

struct BessResult {
    // the returned model, sparse: de-normalised coefficients on its support (ORIGINAL, un-screened column numbers,
    // ascending); p_out = length of the dense beta vector the caller sees
    std::vector<int> beta_idx;
    std::vector<double> beta_val;
    long long p_out = 0;
    double coef0 = 0.0, train_loss = 0.0, ic = 0.0, lambda = 0.0;
    std::vector<int> screening_A;
    int chosen_s = 0;
    // per-level trace (sequential path; normalised scale like beta_all before de-normalisation is NOT kept:
    // these are de-normalised, as the R build returns them, path.cpp:76-123)
    // kept sparse: support (ORIGINAL column numbering, ascending) + de-normalised coefficients per level; expanded
    // to dense rows only on request (bess_b200_trace)
    std::vector<std::vector<int>> A_all;
    std::vector<std::vector<double>> bA_all;
    std::vector<double> coef0_all, train_loss_all, ic_all;
    std::vector<int> s_all, l_all;
    std::vector<double> lambda_all;
    EngineStats stats;
    double prof_ms[PROF_NCAT] = {};
    long long prof_n[PROF_NCAT] = {};
    int sweep_splits = 1;
    bool sparse_sweeps = false;   // the PDAS sweeps ran on the CSC arrays of a sparse design (keep_sparse)
    bool tie_exact_pass = false;  // the call met a boundary tie and was repeated with host-resolved selections
    bool robust_pass = false;     // the fast pass met a dependent active column (or a non-finite result) and the call was
                                  // repeated on the multi-kernel path, whose solver is rank-revealing
    double resident[24 + 4 * MAXC] = {};  // Engine::resident_counters (24) + resident_owner_counters (4 per chain)
    // host wall-clock of the call by phase (ms): 0 engine + load (+ upload), 1 screening, 2 normalisation, 3 fold / chain
    // set-up, 4 the path itself
    double host_ms[5] = {};
};

// Metric.h:49-106 with the seed pinned (same std::mt19937 + std::shuffle + chunking)
std::vector<int> cv_fold_ids(int n, int K, unsigned seed);

// pgs_path geometry (path.cpp:414-577), host only: where the line p + t*u leaves the (s, log lambda) box
int pgs_line_box(const double p[2], const double u[2], int s_min, int s_max, double lmin, double lmax, double a[2], double b[2]);

// Fold-sharded calls (BessArgs::fold_shard): the chains rank `rank` of `world` runs -- chain 0 (full data) always, fold chain
// c (1..K) when c % world == rank, and on every rank the last fold chain K when `last_fold_everywhere` (gs_path reads its
// model at the end, path.cpp:314-319).  counts[i] = 1 when this rank contributes the test loss of chains[i] (every fold
// loss is contributed by exactly one rank; chain 0 has no test loss: counts[0] = 0).
void fold_shard_chains(int K, int world, int rank, bool last_fold_everywhere, std::vector<int> &chains, std::vector<char> &counts);

// throws EngineError
void bess_run(const BessArgs &a, BessResult &out);
// a sparse design without screening (and without groups) keeps its CSC form for the PDAS sweeps (DESIGN 3.12)
bool keep_sparse(long long n, long long p, long long nnz, size_t device_total);

}  // namespace bess
