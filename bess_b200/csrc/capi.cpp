// extern "C" surface of libbess_b200.so (declared in include/bess_b200.h).
#include "../../include/bess_b200.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <limits>
#include <string>

#include "kernels.cuh"
#include "nccl_dl.h"
#include "path.h"

using namespace bess;

namespace {
thread_local std::string g_err;
thread_local BessResult g_last;

unsigned env_seed()
{
    const char *s = std::getenv("BESS_CV_SEED");
    return s ? (unsigned)std::strtoul(s, nullptr, 10) : 123u;
}

template <class F>
int guarded(F &&f)
{
    try {
        g_err.clear();
        f();
        return 0;
    } catch (const EngineError &e) {
        g_err = e.msg;
    } catch (const std::exception &e) {
        g_err = e.what();
    } catch (...) {
        g_err = "unknown error";
    }
    return 1;
}
}  // namespace

struct bessgpu_handle {
    Engine *eng = nullptr;
};

// shared by both linkages of pywrap_bess and by bess_b200_fit
int bess_b200_fit_impl(double *x, int x_row, int x_col, double *y, int y_len, int data_type, double *weight,
                       int weight_len, bool is_normal, int algorithm_type, int model_type, int max_iter,
                       int exchange_num, int path_type, bool is_warm_start, int ic_type, bool is_cv, int K, int *gindex,
                       int gindex_len, double *state, int state_len, int *sequence, int sequence_len,
                       double *lambda_sequence, int lambda_sequence_len, int s_min, int s_max, int K_max, double epsilon,
                       double lambda_min, double lambda_max, int n_lambda, bool is_screening, int screening_size,
                       int powell_path, int *always_select, int always_select_len, double tao, double *beta_out,
                       int beta_out_len, double *coef0_out, double *train_loss_out, double *ic_out,
                       const bess_b200_ext *ext)
{
    return guarded([&] {
        if (y_len != x_row || weight_len != x_row) throw EngineError{"y/weight length must equal the number of rows of x"};
        const bool fshard = ext && ext->world > 1 && ext->fold_shard != 0;  // folds over the ranks, design replicated
        const bool shard = ext && ext->world > 1 && !fshard;                // columns over the ranks
        if (beta_out && beta_out_len < (shard ? ext->p_total : (long long)x_col)) throw EngineError{"beta_out shorter than p"};
        BessArgs a;
        a.x = x; a.n = x_row; a.p = x_col; a.y = y; a.data_type = data_type; a.weight = weight;
        a.is_normal = is_normal; a.algorithm_type = algorithm_type; a.model_type = model_type; a.max_iter = max_iter;
        a.exchange_num = exchange_num; a.path_type = path_type; a.is_warm_start = is_warm_start; a.ic_type = ic_type;
        a.is_cv = is_cv; a.K = K;
        if (state && state_len > 0) a.state.assign(state, state + state_len);
        if (sequence && sequence_len > 0) a.sequence.assign(sequence, sequence + sequence_len);
        if (lambda_sequence && lambda_sequence_len > 0) a.lambda_seq.assign(lambda_sequence, lambda_sequence + lambda_sequence_len);
        a.s_min = s_min; a.s_max = s_max; a.K_max = K_max; a.epsilon = epsilon; a.lambda_min = lambda_min;
        a.lambda_max = lambda_max; a.nlambda = n_lambda; a.is_screening = is_screening;
        a.screening_size = screening_size; a.powell_path = powell_path;
        // (in column-sharded mode a real group structure is refused by bess_run; a trivial gindex -- one entry per local
        // column, 0..x_col-1 -- carries no information and is dropped)
        if (gindex && gindex_len > 0 && !(shard && gindex_len == x_col)) a.g_index.assign(gindex, gindex + gindex_len);
        if (always_select && always_select_len > 0) a.always_select.assign(always_select, always_select + always_select_len);
        a.tao = tao;
        a.cv_seed = env_seed();
        if (ext) {
            a.fold_of_row = ext->fold_of_row;
            if (ext->cv_seed || ext->cv_seed_set) a.cv_seed = ext->cv_seed;
            a.x_on_device = ext->x_on_device != 0;
            a.device = ext->device;
            a.profile = ext->profile != 0;
            if (ext->x_csc) {
                a.csc = true;
                a.csc_colptr = ext->x_csc->colptr;
                a.csc_rowidx = ext->x_csc->rowidx;
                a.csc_values = ext->x_csc->values;
                a.csc_nnz = ext->x_csc->nnz;
            }
            if (shard) {
                a.world = ext->world;
                a.rank = ext->rank;
                a.col_lo = ext->col_lo;
                a.p_total = ext->p_total;
                a.nccl_id = ext->nccl_unique_id;
                a.cv_reduce_over_ranks = ext->cv_reduce_over_ranks != 0;
            }
            if (fshard) {
                a.world = ext->world;
                a.rank = ext->rank;
                a.nccl_id = ext->nccl_unique_id;
                a.fold_shard = true;
            }
        }
        BessResult r;
        bess_run(a, r);
        if (beta_out) {
            // dense beta by contract (bess.cpp:277); a caller that hands in a zero-filled buffer can say so and spare the
            // p-sized pass (at p = 500000 zeroing 4 MB of fresh pages costs more than a PDAS iteration)
            if (!(ext && ext->beta_out_zeroed)) std::fill(beta_out, beta_out + r.p_out, 0.0);
            for (size_t i = 0; i < r.beta_idx.size(); i++) beta_out[r.beta_idx[i]] = r.beta_val[i];
        }
        if (coef0_out) *coef0_out = r.coef0;
        if (train_loss_out) *train_loss_out = r.train_loss;
        if (ic_out) *ic_out = r.ic;
        if (ext) {
            if (ext->screening_A_out && !r.screening_A.empty())
                std::copy(r.screening_A.begin(), r.screening_A.end(), ext->screening_A_out);
            if (ext->chosen_s_out) *ext->chosen_s_out = r.chosen_s;
            if (ext->sparse_sweeps_out) *ext->sparse_sweeps_out = r.sparse_sweeps ? 1 : 0;
            if (ext->chosen_lambda_out) *ext->chosen_lambda_out = r.lambda;
            if (ext->resident_out) std::copy(r.resident, r.resident + 24 + 4 * MAXC, ext->resident_out);
            if (ext->tie_exact_out)
                *ext->tie_exact_out = (r.tie_exact_pass ? 1 : 0) | (r.robust_pass ? 2 : 0) | (r.stats.n_rank_deficient > 0 ? 4 : 0);
            if (ext->stats_out) {
                ext->stats_out[0] = (double)r.stats.n_fits;
                ext->stats_out[1] = (double)r.stats.n_pdas_iters;
                ext->stats_out[2] = (double)r.stats.n_sweeps;
                ext->stats_out[3] = (double)r.stats.n_batches;
                ext->stats_out[4] = (double)r.stats.n_boundary_ties;
                ext->stats_out[5] = r.stats.sweep_bytes;
                ext->stats_out[6] = (double)r.stats.kernel_launches;
                ext->stats_out[7] = (double)r.s_all.size();
                for (int q = 0; q < PROF_NCAT; q++) {
                    ext->stats_out[8 + q] = r.prof_ms[q];
                    ext->stats_out[16 + q] = (double)r.prof_n[q];
                }
                ext->stats_out[24] = r.stats.big_sweep_bytes;
                ext->stats_out[25] = (double)r.sweep_splits;
                ext->stats_out[26] = r.stats.norm_bytes;
                for (int q = 0; q < 5; q++) ext->stats_out[27 + q] = r.host_ms[q];
            }
        }
        g_last = std::move(r);
    });
}

void bess_b200_pywrap_impl(double *x, int x_row, int x_col, double *y, int y_len, int data_type, double *weight,
                           int weight_len, bool is_normal, int algorithm_type, int model_type, int max_iter,
                           int exchange_num, int path_type, bool is_warm_start, int ic_type, bool is_cv, int K,
                           int *gindex, int gindex_len, double *state, int state_len, int *sequence, int sequence_len,
                           double *lambda_sequence, int lambda_sequence_len, int s_min, int s_max, int K_max,
                           double epsilon, double lambda_min, double lambda_max, int n_lambda, bool is_screening,
                           int screening_size, int powell_path, int *always_select, int always_select_len, double tao,
                           double *beta_out, int beta_out_len, double *coef0_out, double *train_loss_out, double *ic_out)
{
    const int rc = bess_b200_fit_impl(x, x_row, x_col, y, y_len, data_type, weight, weight_len, is_normal, algorithm_type,
                                      model_type, max_iter, exchange_num, path_type, is_warm_start, ic_type, is_cv, K,
                                      gindex, gindex_len, state, state_len, sequence, sequence_len, lambda_sequence,
                                      lambda_sequence_len, s_min, s_max, K_max, epsilon, lambda_min, lambda_max, n_lambda,
                                      is_screening, screening_size, powell_path, always_select, always_select_len, tao,
                                      beta_out, beta_out_len, coef0_out, train_loss_out, ic_out, nullptr);
    if (rc != 0) {
        std::fprintf(stderr, "bess_b200: pywrap_bess failed: %s\n", g_err.c_str());
        const double nan = std::numeric_limits<double>::quiet_NaN();
        if (coef0_out) *coef0_out = nan;
        if (train_loss_out) *train_loss_out = nan;
        if (ic_out) *ic_out = nan;
    }
}

extern "C" {

void pywrap_bess(double *x, int x_row, int x_col, double *y, int y_len, int data_type, double *weight, int weight_len,
                 bool is_normal, int algorithm_type, int model_type, int max_iter, int exchange_num, int path_type,
                 bool is_warm_start, int ic_type, bool is_cv, int K, int *gindex, int gindex_len, double *state,
                 int state_len, int *sequence, int sequence_len, double *lambda_sequence, int lambda_sequence_len,
                 int s_min, int s_max, int K_max, double epsilon, double lambda_min, double lambda_max, int n_lambda,
                 bool is_screening, int screening_size, int powell_path, int *always_select, int always_select_len,
                 double tao, double *beta_out, int beta_out_len, double *coef0_out, int, double *train_loss_out, int,
                 double *ic_out, int, double *, double *, int, double *, int, double *, int, int *, int, int *)
{
    bess_b200_pywrap_impl(x, x_row, x_col, y, y_len, data_type, weight, weight_len, is_normal, algorithm_type, model_type,
                          max_iter, exchange_num, path_type, is_warm_start, ic_type, is_cv, K, gindex, gindex_len, state,
                          state_len, sequence, sequence_len, lambda_sequence, lambda_sequence_len, s_min, s_max, K_max,
                          epsilon, lambda_min, lambda_max, n_lambda, is_screening, screening_size, powell_path,
                          always_select, always_select_len, tao, beta_out, beta_out_len, coef0_out, train_loss_out, ic_out);
}

int bess_b200_fit(double *x, int x_row, int x_col, double *y, int y_len, int data_type, double *weight, int weight_len,
                  bool is_normal, int algorithm_type, int model_type, int max_iter, int exchange_num, int path_type,
                  bool is_warm_start, int ic_type, bool is_cv, int K, int *gindex, int gindex_len, double *state,
                  int state_len, int *sequence, int sequence_len, double *lambda_sequence, int lambda_sequence_len,
                  int s_min, int s_max, int K_max, double epsilon, double lambda_min, double lambda_max, int n_lambda,
                  bool is_screening, int screening_size, int powell_path, int *always_select, int always_select_len,
                  double tao, double *beta_out, int beta_out_len, double *coef0_out, double *train_loss_out,
                  double *ic_out, const bess_b200_ext *ext)
{
    return bess_b200_fit_impl(x, x_row, x_col, y, y_len, data_type, weight, weight_len, is_normal, algorithm_type,
                              model_type, max_iter, exchange_num, path_type, is_warm_start, ic_type, is_cv, K, gindex,
                              gindex_len, state, state_len, sequence, sequence_len, lambda_sequence, lambda_sequence_len,
                              s_min, s_max, K_max, epsilon, lambda_min, lambda_max, n_lambda, is_screening,
                              screening_size, powell_path, always_select, always_select_len, tao, beta_out, beta_out_len,
                              coef0_out, train_loss_out, ic_out, ext);
}

int bess_b200_trace(int *s_all, int *l_all, double *coef0_all, double *train_loss_all, double *ic_all, double *beta_all,
                    int p)
{
    const BessResult &r = g_last;
    const size_t L = r.s_all.size();
    if (s_all) std::copy(r.s_all.begin(), r.s_all.end(), s_all);
    if (l_all) std::copy(r.l_all.begin(), r.l_all.end(), l_all);
    if (coef0_all) std::copy(r.coef0_all.begin(), r.coef0_all.end(), coef0_all);
    if (train_loss_all) std::copy(r.train_loss_all.begin(), r.train_loss_all.end(), train_loss_all);
    if (ic_all) std::copy(r.ic_all.begin(), r.ic_all.end(), ic_all);
    if (beta_all)
        for (size_t i = 0; i < r.A_all.size(); i++) {
            double *row = beta_all + i * (size_t)p;
            std::fill(row, row + p, 0.0);
            for (size_t q = 0; q < r.A_all[i].size(); q++)
                if (r.A_all[i][q] < p) row[r.A_all[i][q]] = r.bA_all[i][q];
        }
    return (int)L;
}

int bess_b200_trace_lambda(double *lambda_all)
{
    const BessResult &r = g_last;
    if (lambda_all) std::copy(r.lambda_all.begin(), r.lambda_all.end(), lambda_all);
    return (int)r.lambda_all.size();
}

int bess_b200_cv_fold_ids(int n, int K, unsigned seed, int *out)
{
    return guarded([&] {
        if (n < 1 || K < 1 || K > n) throw EngineError{"cv_fold_ids: need 1 <= K <= n"};
        std::vector<int> f = cv_fold_ids(n, K, seed);
        std::copy(f.begin(), f.end(), out);
    });
}

int bess_b200_nccl_unique_id(void *out128)
{
    return guarded([&] {
        ncclUniqueId id;
        ncclResult_t r = nccl_api().GetUniqueId(&id);
        if (r != ncclSuccess) throw EngineError{std::string("ncclGetUniqueId: ") + nccl_api().GetErrorString(r)};
        std::memcpy(out128, id.internal, NCCL_UNIQUE_ID_BYTES);
    });
}

int bess_b200_gen_design(double *x_dev, int n, long long p, long long ld, double rho, unsigned long long seed, int device)
{
    return guarded([&] {
        if (!x_dev || n < 1 || p < 1 || ld < p) throw EngineError{"gen_design: need a device buffer, n >= 1, 1 <= p <= ld"};
        if (device >= 0 && cudaSetDevice(device) != cudaSuccess) throw EngineError{"gen_design: cudaSetDevice failed"};
        launch_gen_design(x_dev, ld, n, p, rho, seed, nullptr);
        const cudaError_t e = cudaStreamSynchronize(nullptr);
        if (e != cudaSuccess) throw EngineError{std::string("gen_design: ") + cudaGetErrorString(e)};
    });
}

int bess_b200_gen_design_cortype(double *x_dev, int n, long long p, long long ld, double rho, unsigned long long seed, int cortype,
                                 int device)
{
    return guarded([&] {
        if (!x_dev || n < 1 || p < 1 || ld < p) throw EngineError{"gen_design: need a device buffer, n >= 1, 1 <= p <= ld"};
        if (device >= 0 && cudaSetDevice(device) != cudaSuccess) throw EngineError{"gen_design: cudaSetDevice failed"};
        double *scratch = nullptr;
        if (cortype == 3 && cudaMalloc((void **)&scratch, (size_t)2 * p * sizeof(double)) != cudaSuccess)
            throw EngineError{"gen_design: out of device memory"};
        try {
            launch_gen_design_cortype(x_dev, ld, n, p, rho, seed, cortype, scratch, nullptr);
        } catch (...) {
            cudaFree(scratch);
            throw;
        }
        const cudaError_t e = cudaStreamSynchronize(nullptr);
        cudaFree(scratch);
        if (e != cudaSuccess) throw EngineError{std::string("gen_design: ") + cudaGetErrorString(e)};
    });
}

int bess_b200_pgs_line_box(const double *p2, const double *u2, int s_min, int s_max, double log_lambda_min, double log_lambda_max,
                           double *a2_out, double *b2_out)
{
    return pgs_line_box(p2, u2, s_min, s_max, log_lambda_min, log_lambda_max, a2_out, b2_out);
}

const char *bess_b200_last_error(void) { return g_err.c_str(); }
int bess_b200_version(void) { return BESS_B200_VERSION; }
int bess_b200_device_count(void)
{
    int c = 0;
    if (cudaGetDeviceCount(&c) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return c;
}

// ---- device shim -------------------------------------------------------------------------------------------------
int bessgpu_create(bessgpu_handle **h, int device)
{
    return guarded([&] {
        bessgpu_handle *hh = new bessgpu_handle();
        try {
            hh->eng = new Engine(device);
        } catch (...) {
            delete hh;
            throw;
        }
        *h = hh;
    });
}
int bessgpu_destroy(bessgpu_handle *h)
{
    return guarded([&] {
        if (h) {
            delete h->eng;
            delete h;
        }
    });
}
int bessgpu_load(bessgpu_handle *h, const double *x, int n, int p, int x_on_device, const double *y,
                 const double *weight, int model_type)
{
    return guarded([&] { h->eng->load(x, n, p, x_on_device != 0, y, weight, model_type); });
}
int bessgpu_load_csc(bessgpu_handle *h, const long long *colptr, const int *rowidx, const double *values, int n, int p,
                     long long nnz, int on_device, const double *y, const double *weight, int model_type)
{
    return guarded([&] { h->eng->load_csc(colptr, rowidx, values, n, p, nnz, on_device != 0, y, weight, model_type); });
}
int bessgpu_screen(bessgpu_handle *h, int size, const int *always, int n_always, int *out)
{
    return guarded([&] {
        std::vector<int> al(always, always + (always ? n_always : 0));
        std::vector<int> r = h->eng->screen(size, al);
        std::copy(r.begin(), r.end(), out);
    });
}
int bessgpu_screen_local(bessgpu_handle *h, int size, const int *always, int n_always, double *vals_out, int *idx_out,
                         int *count_out)
{
    return guarded([&] {
        std::vector<int> al(always, always + (always ? n_always : 0));
        std::vector<double> v;
        std::vector<int> ix;
        h->eng->screen_local(size, al, v, ix);
        std::copy(v.begin(), v.end(), vals_out);
        std::copy(ix.begin(), ix.end(), idx_out);
        *count_out = (int)ix.size();
    });
}
int bessgpu_gather_columns(bessgpu_handle *h, const int *cols, const int *pos, int m, double *dst_dev, long long ld)
{
    return guarded([&] { h->eng->gather_columns(cols, pos, m, dst_dev, ld); });
}
int bessgpu_set_groups(bessgpu_handle *h, const int *g_index, int n_groups)
{
    return guarded([&] { h->eng->set_groups(std::vector<int>(g_index, g_index + n_groups)); });
}
int bessgpu_normalize(bessgpu_handle *h, int data_type, int is_normal)
{
    return guarded([&] { h->eng->normalize(data_type, is_normal != 0); });
}
int bessgpu_design(bessgpu_handle *h, double *x_out)
{
    return guarded([&] { h->eng->copy_design(x_out); });
}
int bessgpu_get_norm(bessgpu_handle *h, double *xm, double *xn, double *ym)
{
    return guarded([&] {
        if (xm) std::copy(h->eng->x_mean().begin(), h->eng->x_mean().end(), xm);
        if (xn) std::copy(h->eng->x_norm().begin(), h->eng->x_norm().end(), xn);
        if (ym) *ym = h->eng->y_mean();
    });
}
int bessgpu_setup_chains(bessgpu_handle *h, int K, const int *fold_of_row, int kcap, int max_iter, int warm,
                         const int *always, int n_always)
{
    return guarded([&] {
        std::vector<int> al(always, always + (always ? n_always : 0));
        h->eng->setup_chains(K, fold_of_row, kcap, max_iter, warm != 0, al);
    });
}
int bessgpu_run_batch(bessgpu_handle *h, int T, const int *chains, int nch, int new_path_step, int *l_out,
                      double *coef0_out, int *A_out, double *bA_out)
{
    return guarded([&] {
        std::vector<int> ch(chains, chains + nch);
        BatchResult br;
        h->eng->run_batch(T, ch, new_path_step != 0, br);
        for (int i = 0; i < nch; i++) {
            if (l_out) l_out[i] = br.l[i];
            if (coef0_out) coef0_out[i] = br.coef0[i];
            if (A_out) std::copy(br.A[i].begin(), br.A[i].end(), A_out + (size_t)i * T);
            if (bA_out) std::copy(br.bA[i].begin(), br.bA[i].end(), bA_out + (size_t)i * T);
        }
    });
}
int bessgpu_run_batch_groups(bessgpu_handle *h, int T, const int *chains, int nch, int new_path_step, double lambda,
                             int *l_out, double *coef0_out, int *ks_out, int *A_out, double *bA_out, int ld)
{
    return guarded([&] {
        std::vector<int> ch(chains, chains + nch);
        BatchResult br;
        h->eng->run_batch(T, ch, new_path_step != 0, br, nullptr, nullptr, lambda);
        for (int i = 0; i < nch; i++) {
            if ((int)br.A[i].size() > ld) throw EngineError{"run_batch_groups: ld is smaller than a support"};
            if (l_out) l_out[i] = br.l[i];
            if (coef0_out) coef0_out[i] = br.coef0[i];
            if (ks_out) ks_out[i] = (int)br.A[i].size();
            if (A_out) std::copy(br.A[i].begin(), br.A[i].end(), A_out + (size_t)i * ld);
            if (bA_out) std::copy(br.bA[i].begin(), br.bA[i].end(), bA_out + (size_t)i * ld);
        }
    });
}
int bessgpu_losses(bessgpu_handle *h, const int *chain, const int *kind, const int *fold, int njobs, double *out)
{
    return guarded([&] {
        std::vector<LossJob> jobs;
        for (int i = 0; i < njobs; i++) jobs.push_back({chain[i], kind[i], fold[i]});
        std::vector<double> v;
        h->eng->losses(jobs, v);
        std::copy(v.begin(), v.end(), out);
    });
}
int bessgpu_time_dual_sweep(bessgpu_handle *h, int reps, float *ms_out, double *bytes_out)
{
    return guarded([&] {
        *ms_out = h->eng->time_dual_sweep(0, reps);
        if (bytes_out) *bytes_out = h->eng->dual_sweep_bytes();
    });
}
int bessgpu_sacrifice(bessgpu_handle *h, const int *chains, int nch, double lambda, double *bd_out, int *info_out)
{
    return guarded([&] {
        std::vector<double> bd;
        h->eng->debug_sacrifice(std::vector<int>(chains, chains + nch), lambda, bd, info_out);
        std::copy(bd.begin(), bd.end(), bd_out);
    });
}
int bessgpu_stats(bessgpu_handle *h, double *o)
{
    return guarded([&] {
        const EngineStats &s = h->eng->stats();
        o[0] = (double)s.n_fits; o[1] = (double)s.n_pdas_iters; o[2] = (double)s.n_sweeps; o[3] = (double)s.n_batches;
        o[4] = (double)s.n_boundary_ties; o[5] = s.sweep_bytes; o[6] = (double)s.kernel_launches;
        o[7] = (double)s.max_cluster;
    });
}
int bessgpu_topk(const double *vals, int n, int k, int *idx_out, int *tie_out)
{
    return guarded([&] {
        if (k < 1 || k > n) throw EngineError{"topk: need 1 <= k <= n"};
        auto ck = [](cudaError_t e) { if (e != cudaSuccess) throw EngineError{cudaGetErrorString(e)}; };
        configure_kernels();
        double *dv = nullptr, *ck0 = nullptr, *ck1 = nullptr;
        int *ci0 = nullptr, *ci1 = nullptr, *dout = nullptr, *dtie = nullptr;
        const long long cs = std::max<long long>(2LL * k + 16, ((long long)n / 8192 + 2) * std::min(k, TOPK_LMAX));
        ck(cudaMalloc(&dv, (size_t)n * 8));
        ck(cudaMalloc(&ck0, (size_t)cs * 8)); ck(cudaMalloc(&ck1, (size_t)cs * 8));
        ck(cudaMalloc(&ci0, (size_t)cs * 4)); ck(cudaMalloc(&ci1, (size_t)cs * 4));
        ck(cudaMalloc(&dout, (size_t)k * 4)); ck(cudaMalloc(&dtie, 4));
        ck(cudaMemcpy(dv, vals, (size_t)n * 8, cudaMemcpyHostToDevice));
        ck(cudaMemset(dtie, 0, 4));
        launch_topk(dv, n, n, k, 1, dout, k, dtie, ck0, ci0, ck1, ci1, cs, 0);
        ck(cudaMemcpy(idx_out, dout, (size_t)k * 4, cudaMemcpyDeviceToHost));
        if (tie_out) ck(cudaMemcpy(tie_out, dtie, 4, cudaMemcpyDeviceToHost));
        cudaFree(dv); cudaFree(ck0); cudaFree(ck1); cudaFree(ci0); cudaFree(ci1); cudaFree(dout); cudaFree(dtie);
    });
}

int bessgpu_screen_select(const double *vals, int n, int k, int *idx_out, int *tie_out)
{
    return guarded([&] {
        if (k < 1 || k > n) throw EngineError{"screen_select: need 1 <= k <= n"};
        auto ck = [](cudaError_t e) { if (e != cudaSuccess) throw EngineError{cudaGetErrorString(e)}; };
        configure_kernels();
        double *dv = nullptr, *ck0 = nullptr, *ck1 = nullptr;
        int *ci0 = nullptr, *ci1 = nullptr, *dout = nullptr, *dtie = nullptr;
        void *scratch = nullptr;
        const long long cs = std::max<long long>(2LL * k + 16, ((long long)n / 8192 + 2) * std::min(k, TOPK_LMAX));
        ck(cudaMalloc(&dv, (size_t)n * 8));
        ck(cudaMalloc(&ck0, (size_t)cs * 8)); ck(cudaMalloc(&ck1, (size_t)cs * 8));
        ck(cudaMalloc(&ci0, (size_t)cs * 4)); ck(cudaMalloc(&ci1, (size_t)cs * 4));
        ck(cudaMalloc(&dout, (size_t)k * 4)); ck(cudaMalloc(&dtie, 4));
        ck(cudaMalloc(&scratch, screen_select_scratch_bytes(n)));
        ck(cudaMemcpy(dv, vals, (size_t)n * 8, cudaMemcpyHostToDevice));
        ck(cudaMemset(dtie, 0, 4));
        launch_screen_select(dv, n, k, dout, dtie, scratch, ck0, ci0, ck1, ci1, cs, 0);
        ck(cudaMemcpy(idx_out, dout, (size_t)k * 4, cudaMemcpyDeviceToHost));
        if (tie_out) ck(cudaMemcpy(tie_out, dtie, 4, cudaMemcpyDeviceToHost));
        cudaFree(dv); cudaFree(ck0); cudaFree(ck1); cudaFree(ci0); cudaFree(ci1); cudaFree(dout); cudaFree(dtie);
        cudaFree(scratch);
    });
}

int bess_b200_debug_set(int key, int val)
{
    return guarded([&] {
        if (key == 3) engine_debug_first_group(val);  // size of the first speculative group of PDAS iterations (default 3)
        else debug_set(key, val);
    });
}

int bess_b200_debug_get(unsigned long long *out32)
{
    return guarded([&] { debug_get(out32); });
}
// probes of the chain kernels' building blocks (tools / tests; not part of the public header)
int bess_b200_debug_gram(const double *V, int ldv, int nrows, int mm, const double *wt, double *S_out, int impl, int reps,
                         double *ticks_out)
{
    return guarded([&] { debug_gram(V, ldv, nrows, mm, wt, S_out, impl, reps, ticks_out); });
}
int bess_b200_debug_solve(const double *S, int lds, int mm, double *x_out, int impl, int reps, double *ticks_out)
{
    return guarded([&] { debug_solve(S, lds, mm, x_out, impl, reps, ticks_out); });
}
// S: (mm + 1) x lds bordered system, placed and solved as a fit with support cap kcap would; path_out: int[3]
int bess_b200_debug_solve_path(const double *S, int lds, int mm, int kcap, double *x_out, int *path_out)
{
    return guarded([&] { debug_solve_path(S, lds, mm, kcap, x_out, path_out); });
}
// Gram of rows [r0, r1) of V; S_io: ldo x ldo (ldo = 64 when mm <= 64, else ldv), initial contents in, result out
int bess_b200_debug_gram_rows(const double *V, int ldv, int r0, int r1, int mm, const double *wt, double *S_io, int kcap,
                              int impl)
{
    return guarded([&] { debug_gram_rows(V, ldv, r0, r1, mm, wt, S_io, kcap, impl); });
}

// ---- multi-GPU host helpers ------------------------------------------------------------------------------------------
void bess_b200_shard_range(long long p, int world, int rank, long long *lo, long long *hi)
{
    shard_range(p, world, rank, lo, hi);
}
int bess_b200_chain_owner(int chain, int world) { return world > 0 ? chain % world : 0; }
int bess_b200_fold_shard_chains(int K, int world, int rank, int path_type, int *chains_out, int *counts_out)
{
    int n = -1;
    const int rc = guarded([&] {
        if (K < 0 || world < 1 || rank < 0 || rank >= world) throw EngineError{"fold_shard_chains: need K >= 0, 0 <= rank < world"};
        std::vector<int> ch;
        std::vector<char> cnt;
        fold_shard_chains(K, world, rank, path_type != 1, ch, cnt);
        for (size_t i = 0; i < ch.size(); i++) {
            if (chains_out) chains_out[i] = ch[i];
            if (counts_out) counts_out[i] = cnt[i];
        }
        n = (int)ch.size();
    });
    return rc == 0 ? n : -1;
}
int bess_b200_merge_candidates(const double *vals, const int *idx, int count, int k, int *idx_out)
{
    return guarded([&] {
        if (k < 0 || k > count) throw EngineError{"merge_candidates: need 0 <= k <= count"};
        std::vector<int> ord((size_t)count);
        for (int i = 0; i < count; i++) ord[(size_t)i] = i;
        std::sort(ord.begin(), ord.end(), [&](int a, int b) {
            if (vals[a] != vals[b]) return vals[a] > vals[b];
            return idx[a] < idx[b];
        });
        std::vector<int> sel((size_t)k);
        for (int i = 0; i < k; i++) sel[(size_t)i] = idx[ord[(size_t)i]];
        std::sort(sel.begin(), sel.end());
        std::copy(sel.begin(), sel.end(), idx_out);
    });
}

}  // extern "C"
