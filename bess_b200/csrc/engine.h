// bess_b200 device engine -- internal C++ interface between the host path driver (path.cpp)
// and the CUDA kernels (kernels.cu / engine.cu).  Not installed; the public boundary is
// include/bess_b200.h.
//
// Vocabulary (follows the reference, /root/reference/src):
//   chain   one warm-start lineage: chain 0 = the full-data fit of sequential_path/gs_path
//           (path.cpp:48-74), chain 1+k = CV fold k (Metric.h:163-191).  A chain owns its train-row
//           list, its current support A / beta_A / coef0 and its gathered active columns X_A.
//   batch   all chains that run one sparsity level T concurrently (Algorithm::fit, Algorithm.h:113-171,
//           advanced in lock-step: one dual sweep over X serves every chain of the batch).
#pragma once
#include <cstddef>
#include <cstdint>
#include <string>
#include <vector>

namespace bess {

constexpr int MAXC = 32;      // max chains = 1 + K folds (K <= 31)
constexpr int PROF_NCAT = 8;
constexpr int MAX_ITER_CAP = 100000;  // A_list (Algorithm.h:142) is sized max_iter + 2 per problem; this only bounds the argument
constexpr int GMAX = 8;       // widest group of variables the register kernels of group selection take (gsize > 1)
constexpr int GWIDE = 64;     // widest group at all (shared-memory kernel, group.cu)
constexpr int NSLOT = 4;      // snapshot slots of Engine::chain_state
enum { STATE_ZERO = 0, STATE_SAVE = 1, STATE_LOAD = 2 };

enum Family { FAM_LM = 1, FAM_LOGIT = 2, FAM_POISSON = 3, FAM_COX = 4 };

struct BatchResult {
    int T = 0;
    int nchains = 0;
    int chain_ids[MAXC];
    int l[MAXC];                 // PDAS iterations used (Algorithm::l)
    double coef0[MAXC];
    std::vector<int> A[MAXC];     // support, ascending
    std::vector<double> bA[MAXC]; // coefficients on the support (normalised scale)
};

// one step of a path segment: sparsity level + ridge level (path.cpp:48-74 walks these in a fixed order)
struct PathStep {
    int T;
    double lambda;
};

struct LossJob {
    int chain;   // whose beta/coef0
    int kind;    // 0 = train_loss formula on ALL rows (Metric::train_loss); 1 = fold test loss on fold `fold`
    int fold;    // for kind 1
};

struct EngineStats {
    long long n_fits = 0, n_pdas_iters = 0, n_sweeps = 0, n_batches = 0, n_boundary_ties = 0;
    long long n_suspect_pivots = 0;   // resident path: fits whose Cholesky met a (numerically) dependent column
    long long n_rank_deficient = 0;   // multi-kernel path: normal-equation solves truncated by the rank-revealing fallback
    long long n_wide_singular = 0;    // multi-kernel path: singular systems of more than 63 unknowns (no truncating solver)
    int max_cluster = 0;              // largest cluster size of a chain_fit_kernel launch since load
    double sweep_bytes = 0.0;     // algorithmic bytes of the PDAS dual sweeps (8*n*p per launch + vectors)
    double big_sweep_bytes = 0.0; // algorithmic bytes of the screening sweep(s) over the raw design (8*n*p each)
    double norm_bytes = 0.0;      // algorithmic bytes of the normalisation / x_j.x_j passes
    long long kernel_launches = 0;
};

class Engine {
public:
    explicit Engine(int device = -1);
    ~Engine();

    // ---- multi-GPU, columns of X sharded over `world` ranks (SURVEY 8e axis B).  Call before load().
    // unique_id: the 128-byte ncclUniqueId every rank received from rank 0 (bess_b200_nccl_unique_id); the
    // communicator is cached per device for the life of the process.
    // This rank will load columns [col_lo, col_lo + p_local) = shard_range(p_total, world, rank) of a p_total-column design.
    void init_shard(int world, int rank, const void *unique_id, long long col_lo, long long p_total);
    // the communicator alone (fold-sharded mode: the design is replicated, only fold losses travel)
    void init_comm(int world, int rank, const void *unique_id);
    bool sharded() const { return sharded_; }
    // element-wise mean of `v` over the ranks of the job's communicator (one ncclAllReduce on the engine's stream); every
    // rank gets the same result.  Used for repeated K-fold CV: the ranks hold different fold assignments and average
    // their per-level CV losses before the level is chosen.  Needs init_shard().
    void allreduce_mean(std::vector<double> &v);
    void allreduce_sum(std::vector<double> &v);
    bool has_comm() const;
    // column count the model sees (IC penalties, validation): p_total while sharded, else p
    long long p_model() const { return sharded_ ? p_total_ : p_; }
    double x_mean_at(long long j) const { ensure_stats(); return sharded_ ? g_xmean_[(size_t)j] : h_xmean_[(size_t)j]; }
    double x_norm_at(long long j) const { ensure_stats(); return sharded_ ? g_xnorm_[(size_t)j] : h_xnorm_[(size_t)j]; }
    // ---- boundary ties of the top-k selections.  max_k (utilities.cpp:179-188) leaves a tie between the k-th and the
    // (k+1)-th value to std::nth_element; the device select takes the lower index and only COUNTS such ties
    // (stats().n_boundary_ties).  In exact mode every selection that meets a boundary tie is repeated on the host with the
    // reference's own index-array nth_element + sort, at the price of one host round trip per PDAS iteration (no
    // speculative iterations, no resident path).  bess_run repeats a call in this mode when the fast pass saw a tie.
    // Call before load().  Not available in column-sharded mode (ties are then only counted).
    void set_tie_exact(bool on);
    // fold-sharded calls: size the chain clusters as if every batch had `nch` chains (the most any rank runs), so that
    // every rank -- whatever its share of the fold chains -- fits the full-data chain with the same cluster size and the
    // ranks return bit-identical models.  0 = use each batch's own chain count.
    void set_cluster_chains(int nch);
    bool tie_exact() const;
    Engine(const Engine &) = delete;
    Engine &operator=(const Engine &) = delete;

    // ---- design upload.  x: row-major n x p (pywrap_bess layout, utilities.cpp:13-25).
    // x_on_device: x already lives in device memory (bench "resident" mode); it is still copied
    // into engine-owned storage because normalisation is in place.
    // borrow: a device-resident x may be used in place (no copy) until something needs to write to it.
    void load(const double *x, int n, int p, bool x_on_device, const double *y, const double *weight, int family,
              bool borrow = false);
    // ---- sparse design in CSC form (include/bess_b200.h, bess_b200_csc): the three arrays are copied to the device
    // (device arrays are read in place) and checked; a malformed input throws.  The design stays sparse until screening
    // keeps its columns (screen / screen_enqueue densify them) or densify() expands all of it; screen_local reads it as is.
    void load_csc(const long long *colptr, const int *rowidx, const double *values, int n, int p, long long nnz,
                  bool on_device, const double *y, const double *weight, int family);
    // the whole CSC design -> the dense row-major n x ldx design a load() of the same matrix holds
    void densify();
    bool sparse() const;
    // normalize() kept the design sparse: the PDAS sweeps run on the CSC arrays (DESIGN 3.12, "without screening")
    bool sparse_sweeps() const;
    size_t device_total_bytes() const;  // cudaDeviceProp::totalGlobalMem of the engine's device
    // per-category device time (CUDA events on the engine's stream): 0 screening sweep (the pass over the raw design),
    // 1 PDAS dual sweeps, 2 finish, 3 top-k, 4 chain kernels, 5 other, 6 normalisation / x_j.x_j passes, 7 host->device upload
    void set_profiling(bool on);
    void profile(double *ms_out8, long long *n_out8) const;

    // ---- screening.cpp:26-105: marginal utilities on RAW x, top `size`, X <- X[:, A].  Returns A ascending.
    std::vector<int> screen(int size, const std::vector<int> &always_select);
    // the same in two halves: screen_enqueue only enqueues device work (the path can start behind it), screen_result waits
    // for the kept-column list
    void screen_enqueue(int size, const std::vector<int> &always_select);
    std::vector<int> screen_result();

    // ---- column-sharded screening (multi-GPU axis B): local top-`size` candidates, X untouched
    void screen_local(int size, const std::vector<int> &always_select, std::vector<double> &vals, std::vector<int> &idx);
    // dst_dev[i*ld + pos[q]] = X[i][cols[q]]  (dst_dev: device buffer)
    void gather_columns(const int *cols, const int *pos, int m, double *dst_dev, long long ld);

    // ---- Data ctor normalisation (Data.h:41-68, normalize.cpp) + add_weight for gaussian (Data.h:70-77).
    void normalize(int data_type, bool is_normal);
    // the current dense design (n x p_model(), row-major, without the row padding) -> host; waits for the device.  A sparse
    // design normalised in place of densifying is expanded to its normalised dense form.
    void copy_design(double *host_out);

    // ---- group selection (R: group.index, Python: GroupPdas*).  g_index: first column of every group, ascending from 0
    // (Data.h:53-61); call after normalize() and before setup_chains().  From then on sparsity levels, top-k results and
    // always_select count GROUPS; supports / coefficients reported by run_batch are still per column.
    void set_groups(const std::vector<int> &g_index);
    int n_groups() const { return n_groups_; }

    // ---- CV folds (Metric.h:49-129).  fold_of_row[i] in [0,K) or K == 0 for no CV.  Also (re)allocates all
    // chain workspaces for supports up to kcap.
    void setup_chains(int K, const int *fold_of_row, int kcap, int max_iter, bool warm_start,
                      const std::vector<int> &always_select);

    // ---- one sparsity level for a set of chains (ascending chain ids).  with_full: the batch starts a new
    // path step (update_coef0_init, path.cpp:57) -- chain 0 must then be in the set.
    // jobs/loss_out: optional Metric losses evaluated right behind the fits (same stream, one host synchronisation).
    // lambda: ridge level of the fits (Algorithm::lambda_level, the L0L2 / "bsrr" penalty); 0 = best-subset selection.
    void run_batch(int T, const std::vector<int> &chains, bool new_path_step, BatchResult &out,
                   const std::vector<LossJob> *jobs = nullptr, std::vector<double> *loss_out = nullptr, double lambda = 0.0);

    // ---- the same in two halves, so that the NEXT path step can be enqueued while the host still waits for this one
    // (sequential_path knows its order of evaluation in advance).  enqueue returns a ticket (two may be pending);
    // collect waits for the batch, enqueues more PDAS iterations if the first speculative group did not finish every
    // chain, and returns true when the first group sufficed.  When it returns false, a batch enqueued behind this one
    // found it unfinished and skipped itself on the device (Dev::prev_active): discard that ticket and enqueue it again.
    int run_batch_enqueue(int T, const std::vector<int> &chains, bool new_path_step, const std::vector<LossJob> *jobs,
                          double lambda);
    bool run_batch_collect(int ticket, BatchResult &out, std::vector<double> *loss_out);
    void run_batch_discard(int ticket);

    // ---- resident path (gaussian family, lm_path.cu): a whole path segment -- `steps` in evaluation order, every chain of
    // `chains` fitted at every step, warm-started from its own previous step -- in ONE cooperative launch with the PDAS
    // iteration loop on the device.  out[t] = the batch result of step t; loss_all / loss_test [t * chains.size() + i] =
    // the Lm train-loss formula over all rows (Metric.h:145-148) / the fold loss over chain i's held-out rows (:190).
    // Only when resident_path() (decided by setup_chains: family, shapes, shared-memory budget); run_batch uses the same
    // kernel for single steps.
    bool resident_path() const;
    const std::string &resident_path_why() const;
    void run_steps(const std::vector<PathStep> &steps, const std::vector<int> &chains, std::vector<BatchResult> &out,
                   std::vector<double> &loss_all, std::vector<double> &loss_test);
    // counters of the resident kernel since load(): 0 launches, 1 PDAS iterations (sweeps), 2 full-vector select fallbacks,
    // 3 path steps, 8..15 clock ticks by phase of chain owner 0 (begin, wait, select, load columns, gram, solve, residual +
    // cycle test, publish), 16..18 of sweeper 0 (wait, stream X, reduce + sacrifice)
    void resident_counters(double *out24) const;
    // per chain owner i (position in the batch): [4 * i + 0] busy ticks, [1] longest phase, [2] ticks in fallback selects,
    // [3] fits actually solved
    void resident_owner_counters(double *out4c) const;  // [4 * MAXC]

    // ---- explicit warm-start state of a chain (STATE_ZERO / STATE_SAVE / STATE_LOAD on NSLOT slots; the
    // (A, beta_A) half and the coef0 half are addressed separately, a negative slot skips that half).  Used by pgs_path.
    void chain_state(int chain, int op, int slot_beta, int slot_coef0);

    // ---- Metric::train_loss / fold test losses for the chains' current beta.
    void losses(const std::vector<LossJob> &jobs, std::vector<double> &out);

    // ---- primitives exposed for tests / roofline benchmarking through the C-ABI
    // Dual sweep + sacrifice for `nch` chains (chain slots f0..f0+nch) -> bd on device; returns kernel ms if timed.
    float time_dual_sweep(int nch, int reps);
    // algorithmic bytes of one such sweep: 8np, or for a sparse design swept on its non-zeros those of launch_csc_sweep
    double dual_sweep_bytes() const;
    // after run_batch: bd of `chains` for their current model ([nch][p], or [nch][n_groups]); info_out[8] as
    // bessgpu_sacrifice (include/bess_b200.h)
    void debug_sacrifice(const std::vector<int> &chains, double lambda, std::vector<double> &bd_out, int *info_out);

    int n() const { return n_; }
    int p() const { return p_; }
    bool grouped() const { return n_groups_ > 0; }
    int family() const { return family_; }
    const std::vector<double> &x_mean() const { ensure_stats(); return h_xmean_; }
    const std::vector<double> &x_norm() const { ensure_stats(); return h_xnorm_; }
    // the column statistics travel to the host asynchronously; the first reader waits for them
    void ensure_stats() const;
    double y_mean() const { return y_mean_; }
    EngineStats &stats() { return stats_; }
    int sweep_splits() const { return S_; }

    struct Impl;
private:
    void begin_load(int n, int p, int family);
    void normalize_csc(int data_type, bool is_normal);
    void end_load(const double *y, const double *weight, int family);
    Impl *d_ = nullptr;
    int n_ = 0, p_ = 0, family_ = 0;
    int S_ = 1;
    int n_groups_ = 0;
    std::vector<int> g_index_, g_size_;
    std::vector<double> h_xmean_, h_xnorm_;
    double y_mean_ = 0.0;
    // sharded mode
    bool sharded_ = false;
    int world_ = 1, rank_ = 0;
    long long col_lo_ = 0, p_total_ = 0;
    std::vector<double> g_xmean_, g_xnorm_;  // column statistics of the WHOLE design (all-gathered)
    EngineStats stats_;
};

// contiguous, even-aligned column shards (16-byte loads need even column offsets), remainder spread over the first ranks
inline void shard_range(long long p, int world, int rank, long long *lo, long long *hi)
{
    const long long pairs = (p + 1) / 2;
    const long long base = pairs / world, rem = pairs % world;
    const long long b = rank * base + (rank < rem ? rank : rem);
    const long long e = b + base + (rank < rem ? 1 : 0);
    *lo = 2 * b < p ? 2 * b : p;
    *hi = 2 * e < p ? 2 * e : p;
}

// test knob (bess_b200_debug_set(3, n)): how many PDAS iterations run_batch_enqueue enqueues before the host first looks.
// 1 forces the "needs more iterations" path at almost every step, i.e. the next path step skips itself and is re-enqueued.
void engine_debug_first_group(int n);

// thrown by the engine on CUDA errors / misuse; the C-ABI turns it into an error code + message
struct EngineError {
    std::string msg;
};

}  // namespace bess
