// Host path driver.  See path.h.  Every numerical step runs on the GPU through bess::Engine; this file only
// decides which sparsity level to evaluate next and applies the scalar criterion / de-normalisation formulas.
#include "path.h"
#include "kernels.cuh"

#include <algorithm>
#include <chrono>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <numeric>
#include <random>

namespace bess {

// Metric::set_cv_train_test_mask (Metric.h:49-106): shuffle 0..n-1 with mt19937, folds are consecutive chunks of
// floor(n/K), the last fold takes the remainder.  The reference seeds from std::random_device (Metric.h:57-58);
// here the seed is an argument (SURVEY 8c: parity on CV-chosen s needs the split pinned).
std::vector<int> cv_fold_ids(int n, int K, unsigned seed)
{
    std::vector<int> index_vec((size_t)n);
    std::iota(index_vec.begin(), index_vec.end(), 0);
    std::mt19937 g(seed);
    std::shuffle(index_vec.begin(), index_vec.end(), g);
    std::vector<int> fold((size_t)n, 0);
    const int group_size = n / K;
    for (int k = 0; k < K; k++) {
        const int b = k * group_size;
        const int e = (k == K - 1) ? n : b + group_size;
        for (int i = b; i < e; i++) fold[(size_t)index_vec[(size_t)i]] = k;
    }
    return fold;
}

// path.cpp:414-577 (line_intersection + cal_intersections): the points where the line p + t*u leaves the box
// [s_min, s_max] x [lmin, lmax]; a <- first, b <- second (in the reference's edge order); returns how many were found.
int pgs_line_box(const double p[2], const double u[2], int s_min, int s_max, double lmin, double lmax, double a[2], double b[2])
{
    auto det = [](const double x[2], const double y[2]) { return x[0] * y[1] - x[1] * y[0]; };
    auto line_intersection = [&](double l1[2][2], double l2[2][2], double x[2], bool &need) {
        double xdiff[2] = {l1[0][0] - l1[1][0], l2[0][0] - l2[1][0]};
        double ydiff[2] = {l1[0][1] - l1[1][1], l2[0][1] - l2[1][1]};
        const double div = det(xdiff, ydiff);
        if (div == 0) {
            need = false;
            return;
        }
        double d[2] = {det(l1[0], l1[1]), det(l2[0], l2[1])};
        x[0] = det(d, xdiff) / div;
        x[1] = det(d, ydiff) / div;
        need = true;
    };
    double line0[2][2] = {{p[0], p[1]}, {p[0] + u[0], p[1] + u[1]}};
    double ls[4][2][2] = {{{(double)s_min, lmin}, {(double)s_min, lmax}},
                          {{(double)s_max, lmin}, {(double)s_max, lmax}},
                          {{(double)s_min, lmin}, {(double)s_max, lmin}},
                          {{(double)s_min, lmax}, {(double)s_max, lmax}}};
    double x[4][2] = {};
    bool need[4];
    for (int i = 0; i < 4; i++) line_intersection(line0, ls[i], x[i], need[i]);
    for (int i = 0; i < 4; i++)
        if (need[i] && ((x[i][0] < s_min - 0.0001) | (x[i][0] > s_max + 0.0001) | (x[i][1] < lmin - 0.001) |
                        (x[i][1] > lmax + 0.001)))
            need[i] = false;
    for (int i = 0; i < 4; i++)
        if (need[i])
            for (int j = i + 1; j < 4; j++)
                if (need[j] && std::fabs(x[i][0] - x[j][0]) < 0.0001 && std::fabs(x[i][1] - x[j][1]) < 0.0001)
                    need[j] = false;
    int j = 0;
    for (int i = 0; i < 4; i++)
        if (need[i]) {
            if (j == 2) j += 1;
            if (j == 1) {
                b[0] = x[i][0];
                b[1] = x[i][1];
                j += 1;
            }
            if (j == 0) {
                a[0] = x[i][0];
                a[1] = x[i][1];
                j += 1;
            }
        }
    return j;
}

namespace {

struct Eval {
    int T = 0, l = 0;
    std::vector<int> A;
    std::vector<double> bA;
    double coef0 = 0.0, train_loss = 0.0, ic = 0.0, lambda = 0.0;
    std::vector<double> fold_part;  // fold-sharded sequential path: this rank's fold losses (K entries, 0 elsewhere)
};

struct Driver {
    Engine &eng;
    const BessArgs &a;
    int n, p, K;  // p: columns after screening; K: folds (0 when !is_cv)
    int kcap = 0;  // largest sparsity level the chain workspaces were sized for
    std::vector<int> all_chains, fold_chains;
    // Fold-sharded mode (SURVEY 8e axis A inside one call): this rank runs the full-data chain and the fold chains it
    // owns (chain c belongs to rank c % world, bess_b200_chain_owner); the per-fold test losses are all-reduced (x + 0 is
    // exact, so every rank -- and a single GPU -- sums the same K numbers in the same order).  gs_path reads the LAST
    // fold's model at the end (path.cpp:314-319): there every rank runs chain K as well, its loss counted once.
    bool fshard = false;
    std::vector<char> counts;  // per entry of fold_chains: does this rank contribute that fold's loss

    Driver(Engine &e, const BessArgs &args) : eng(e), a(args)
    {
        n = eng.n();
        p = (int)eng.p_model();
        K = a.is_cv ? a.K : 0;
        fshard = a.fold_shard && a.world > 1 && K > 0;
        std::vector<char> cnt;
        fold_shard_chains(K, fshard ? a.world : 1, fshard ? a.rank : 0, a.path_type != 1, all_chains, cnt);
        fold_chains.assign(all_chains.begin() + 1, all_chains.end());
        counts.assign(cnt.begin() + 1, cnt.end());
    }
    int nfc() const { return (int)fold_chains.size(); }
    // the most chains any rank of a fold-sharded call runs in one batch (cluster sizing must not depend on the rank)
    int max_chains_per_rank() const
    {
        size_t most = 0;
        for (int r = 0; r < a.world; r++) {
            std::vector<int> ch;
            std::vector<char> cnt;
            fold_shard_chains(K, a.world, r, a.path_type != 1, ch, cnt);
            most = std::max(most, ch.size());
        }
        return (int)most;
    }
    // loss jobs of a batch: [full-data train loss] + the test loss of every fold chain this rank runs
    std::vector<LossJob> make_jobs(bool with_full) const
    {
        std::vector<LossJob> jobs;
        if (with_full) jobs.push_back({0, 0, 0});
        for (int c : fold_chains) jobs.push_back({c, 1, c - 1});
        return jobs;
    }
    // this rank's share of the K fold losses (v[off + i] = loss of fold_chains[i])
    std::vector<double> fold_losses(const std::vector<double> &v, size_t off) const
    {
        std::vector<double> fl((size_t)K, 0.0);
        for (int i = 0; i < nfc(); i++)
            if (counts[(size_t)i]) fl[(size_t)fold_chains[(size_t)i] - 1] = v[off + (size_t)i];
        return fl;
    }
    // the CV criterion of one evaluated level (Metric.h:150-195: mean of the K fold losses)
    double cv_ic(const std::vector<double> &v, size_t off)
    {
        if (!fshard) return mean_of(v, off, off + (size_t)K);
        std::vector<double> fl = fold_losses(v, off);
        eng.allreduce_sum(fl);
        return mean_of(fl, 0, (size_t)K);
    }

    // Metric::ic without CV (Metric.h:205-229 gaussian: n*log(loss) + pen; :365-388 etc. GLMs: loss + pen).
    // The penalty uses the full sample size and the POST-screening column count (SURVEY Q15).
    double ic_formula(double train_loss, int T) const
    {
        double pen;
        // algorithm_type 2 / 3: log(g_num) and group_df = sparsity level (Metric.h:230-254); equal to p and s without groups
        const double dn = (double)n, dp = (double)((a.algorithm_type == 2 || a.algorithm_type == 3) && eng.grouped() ? eng.n_groups() : p);
        switch (a.ic_type) {
            case 1: pen = 2.0 * T; break;
            case 2: pen = std::log(dn) * T; break;
            case 3: pen = std::log(dp) * std::log(std::log(dn)) * T; break;
            case 4: pen = (std::log(dn) + 2 * std::log(dp)) * T; break;
            default: return 0.0;
        }
        if (a.model_type == 1) return dn * std::log(train_loss) + pen;
        return train_loss + pen;
    }

    static double mean_of(const std::vector<double> &v, size_t b, size_t e)
    {
        double s = 0.0;
        for (size_t i = b; i < e; i++) s += v[i];
        return s / (double)(e - b);
    }

    // One path step: full-data fit at level T (path.cpp:52-64) + train_loss + ic (path.cpp:71-72).  Under CV the K
    // fold fits of Metric::test_loss run in the same batch as the full fit (they never read its result; their
    // coef0_init is the one the path set BEFORE this step, SURVEY Q3).
    // last_fold: also return the last fold's beta and ITS full-data loss (gs_path final sweep, path.cpp:314-319).
    Eval step(int T, Eval *last_fold = nullptr, double lambda = 0.0)
    {
        BatchResult br;
        std::vector<LossJob> jobs = make_jobs(true);
        if (last_fold && K > 0) jobs.push_back({K, 0, 0});
        std::vector<double> v;
        eng.run_batch(T, all_chains, /*new_path_step=*/true, br, &jobs, &v, lambda);
        const size_t posK = all_chains.size() - 1;  // chain K is the last chain of the batch whenever last_fold is asked for
        Eval e;
        e.T = T;
        e.lambda = lambda;
        e.l = br.l[0];
        e.A = br.A[0];
        e.bA = br.bA[0];
        e.coef0 = br.coef0[0];
        e.train_loss = v[0];
        e.ic = K > 0 ? cv_ic(v, 1) : ic_formula(e.train_loss, T);
        if (last_fold) {
            if (K > 0) {
                last_fold->T = T;
                last_fold->l = br.l[posK];
                last_fold->A = br.A[posK];
                last_fold->bA = br.bA[posK];
                last_fold->coef0 = br.coef0[posK];
                last_fold->train_loss = v[1 + (size_t)nfc()];
                last_fold->ic = e.ic;
            } else {
                *last_fold = e;
            }
        }
        return e;
    }

    // step() in two halves for paths whose order of evaluation is known in advance (Engine::run_batch_enqueue)
    int step_enqueue(int T, double lambda)
    {
        std::vector<LossJob> jobs = make_jobs(true);
        return eng.run_batch_enqueue(T, all_chains, /*new_path_step=*/true, &jobs, lambda);
    }
    bool step_collect(int ticket, int T, double lambda, Eval &e)
    {
        BatchResult br;
        std::vector<double> v;
        const bool in_one_go = eng.run_batch_collect(ticket, br, &v);
        e.T = T;
        e.lambda = lambda;
        e.l = br.l[0];
        e.A = br.A[0];
        e.bA = br.bA[0];
        e.coef0 = br.coef0[0];
        e.train_loss = v[0];
        if (fshard) e.fold_part = fold_losses(v, 1);  // reduced over the ranks once, at the end of the walk
        else e.ic = K > 0 ? mean_of(v, 1, 1 + (size_t)K) : ic_formula(e.train_loss, T);
        return in_one_go;
    }

    // A repeated metric->ic() on the same level (gs_path evaluates every fresh point twice, SURVEY Q4): under CV
    // that is a second K-fold pass warm-started by the first; without CV the value is unchanged.
    double ic_again(const Eval &e)
    {
        if (K == 0) return e.ic;
        BatchResult br;
        std::vector<LossJob> jobs = make_jobs(false);
        std::vector<double> v;
        // (a rank of a fold-sharded call with more ranks than folds may own no fold chain: it only takes part in the reduce)
        if (!fold_chains.empty()) eng.run_batch(e.T, fold_chains, /*new_path_step=*/false, br, &jobs, &v);
        return cv_ic(v, 0);
    }

    // path.cpp:76-110 / :330-343.  bA_out: de-normalised coefficients on the support e.A
    void denormalise(const Eval &e, std::vector<double> &bA_out, double &coef0) const
    {
        bA_out.assign(e.bA.begin(), e.bA.end());
        coef0 = e.coef0;
        if (!a.is_normal) return;
        const double sn = std::sqrt((double)n);
        double dot = 0.0;
        for (size_t i = 0; i < e.A.size(); i++) {
            const int j = e.A[i];
            const double b = sn * e.bA[i] / eng.x_norm_at(j);
            bA_out[i] = b;
            dot += b * eng.x_mean_at(j);
        }
        if (a.data_type == 1) coef0 = eng.y_mean() - dot;
        else if (a.data_type == 2) coef0 = e.coef0 - dot;
        // data_type 3: x_mean == 0, coef0 unchanged in both path functions
    }
};

void sequential_path(Driver &dr, BessResult &out, Eval &best)
{
    // path.cpp:48-74: for every sparsity level the lambda grid is walked zig-zag (:50), the warm start follows the walk.
    const BessArgs &a = dr.a;
    std::vector<double> lams = a.lambda_seq.empty() ? std::vector<double>{0.0} : a.lambda_seq;
    const int S = (int)a.sequence.size(), L = (int)lams.size();
    std::vector<Eval> evs((size_t)S * L);  // [lambda][s]
    std::vector<int> order;
    for (int i = 0; i < S; i++)
        for (int q = 0; q < L; q++) {
            const int j = (i % 2 == 0) ? q : L - 1 - q;
            order.push_back(j * S + i);
        }
    // The order of evaluation is fixed in advance and every warm start lives on the device, so step t+1 is enqueued
    // before the host waits for step t: the GPU never idles through a host round trip.  If step t needs more PDAS
    // iterations than its first speculative group, step t+1 skips itself on the device and is enqueued again.
    auto level = [&](int idx) { return a.sequence[(size_t)(order[(size_t)idx] % S)]; };
    auto ridge = [&](int idx) { return lams[(size_t)(order[(size_t)idx] / S)]; };
    const int n_steps = (int)order.size();
    const bool pipelined = !dr.eng.sharded();
    if (dr.eng.resident_path()) {
        // gaussian family on an L2-resident design: the whole walk is one cooperative launch (Engine::run_steps); every
        // chain advances from step to step on the device, the host only reads the per-step results
        std::vector<PathStep> steps;
        for (int t = 0; t < n_steps; t++) steps.push_back({level(t), ridge(t)});
        std::vector<BatchResult> brs;
        std::vector<double> la, lt;
        dr.eng.run_steps(steps, dr.all_chains, brs, la, lt);
        const size_t nch = dr.all_chains.size();
        for (int t = 0; t < n_steps; t++) {
            Eval &e = evs[(size_t)order[(size_t)t]];
            const BatchResult &br = brs[(size_t)t];
            e.T = level(t);
            e.lambda = ridge(t);
            e.l = br.l[0];
            e.A = br.A[0];
            e.bA = br.bA[0];
            e.coef0 = br.coef0[0];
            e.train_loss = la[(size_t)t * nch];
            if (dr.fshard) e.fold_part = dr.fold_losses(lt, (size_t)t * nch + 1);
            else e.ic = dr.K > 0 ? Driver::mean_of(lt, (size_t)t * nch + 1, (size_t)t * nch + 1 + (size_t)dr.K)
                                 : dr.ic_formula(e.train_loss, e.T);
        }
    } else if (!pipelined) {
        for (int t = 0; t < n_steps; t++) evs[(size_t)order[(size_t)t]] = dr.step(level(t), nullptr, ridge(t));
    } else {
        int cur = dr.step_enqueue(level(0), ridge(0));
        for (int t = 0; t < n_steps; t++) {
            int next = t + 1 < n_steps ? dr.step_enqueue(level(t + 1), ridge(t + 1)) : -1;
            const bool in_one_go = dr.step_collect(cur, level(t), ridge(t), evs[(size_t)order[(size_t)t]]);
            if (!in_one_go && next >= 0) {
                dr.eng.run_batch_discard(next);
                next = dr.step_enqueue(level(t + 1), ridge(t + 1));
            }
            cur = next;
        }
    }
    if (dr.fshard) {
        // fold-sharded call: one all-reduce of the levels x K matrix of fold losses; then Metric.h:150-195's mean per level
        const size_t K = (size_t)dr.K;
        std::vector<double> mat(evs.size() * K, 0.0);
        for (size_t i = 0; i < evs.size(); i++)
            if (evs[i].fold_part.size() == K) std::copy(evs[i].fold_part.begin(), evs[i].fold_part.end(), mat.begin() + i * K);
        dr.eng.allreduce_sum(mat);
        for (size_t i = 0; i < evs.size(); i++) evs[i].ic = Driver::mean_of(mat, i * K, (i + 1) * K);
    }
    if (a.cv_reduce_over_ranks && a.world > 1) {
        // repeated CV: every rank ran its own fold assignment on the shared screened design; average the CV curves
        std::vector<double> curve(evs.size());
        for (size_t i = 0; i < evs.size(); i++) curve[i] = evs[i].ic;
        dr.eng.allreduce_mean(curve);
        for (size_t i = 0; i < evs.size(); i++) evs[i].ic = curve[i];
    }
    // ic_sequence.minCoeff (path.cpp:113): Eigen visits the column-major matrix ic(s, lambda) column by column, i.e.
    // lambda outer / s inner, and keeps the first minimum
    size_t bi = 0;
    for (size_t i = 1; i < evs.size(); i++)
        if (evs[i].ic < evs[bi].ic) bi = i;
    best = evs[bi];
    for (int idx : order) {  // trace in evaluation order
        const Eval &e = evs[(size_t)idx];
        std::vector<double> b;
        double c0;
        dr.denormalise(e, b, c0);
        out.A_all.push_back(e.A);
        out.bA_all.push_back(std::move(b));
        out.coef0_all.push_back(c0);
        out.train_loss_all.push_back(e.train_loss);
        out.ic_all.push_back(e.ic);
        out.s_all.push_back(e.T);
        out.l_all.push_back(e.l);
        out.lambda_all.push_back(e.lambda);
    }
}

inline int c_round(double v) { return (int)std::round(v); }

// path.cpp:134-389, including its stateful quirks (SURVEY Q4, Q5).
void gs_path(Driver &dr, BessResult &out, Eval &best)
{
    const BessArgs &a = dr.a;
    int Tmin = a.s_min, Tmax = a.s_max;
    int T1 = c_round(0.618 * Tmin + 0.382 * Tmax);
    int T2 = c_round(0.382 * Tmin + 0.618 * Tmax);
    double ic_seq[4] = {0, 0, 0, 0};
    double icT1, icT2;
    auto record = [&](const Eval &e) {
        out.s_all.push_back(e.T);
        out.ic_all.push_back(e.ic);
        out.train_loss_all.push_back(e.train_loss);
        out.l_all.push_back(e.l);
    };
    Eval e1 = dr.step(T1);  // :174-187 -- the very first point is scored once
    ic_seq[1] = e1.ic;
    icT1 = ic_seq[1];
    record(e1);
    Eval e2 = dr.step(T2);  // :189-210 -- ic() twice
    ic_seq[2] = e2.ic;
    icT2 = dr.ic_again(e2);
    record(e2);
    while (T1 != T2) {
        if (icT1 < icT2) {
            Tmax = T2;
            ic_seq[3] = ic_seq[2];
            T2 = T1;
            ic_seq[2] = ic_seq[1];
            icT2 = ic_seq[1];
            T1 = c_round(0.618 * Tmin + 0.382 * Tmax);
            Eval e = dr.step(T1);
            ic_seq[1] = e.ic;
            icT1 = dr.ic_again(e);
            record(e);
        } else {
            Tmin = T1;
            ic_seq[0] = ic_seq[1];
            T1 = T2;
            ic_seq[1] = ic_seq[2];
            icT1 = ic_seq[2];
            T2 = c_round(0.382 * Tmin + 0.618 * Tmax);
            Eval e = dr.step(T2);
            ic_seq[2] = e.ic;
            icT2 = dr.ic_again(e);
            record(e);
        }
    }
    double best_ic = DBL_MAX;
    bool have = false;
    for (int T = Tmin; T <= Tmax; T++) {
        Eval lf;
        Eval e = dr.step(T, &lf);
        if (e.ic < best_ic) {
            // algorithm->get_beta() is read AFTER ic(): under CV it is the last fold's fit, and train_loss is that
            // beta's full-data loss (path.cpp:314-319)
            best = lf;
            best.ic = e.ic;
            best_ic = e.ic;
            have = true;
            record(best);
        }
    }
    if (!have) throw EngineError{"gs_path: no finite criterion value in the final sweep"};
}

// ======================================================================================================================
// pgs_path (path.cpp:1138-1309): Powell's conjugate-direction search over (sparsity level, log lambda) -- the default
// method of R's type = "bsrr" and of the Python L0L2* classes with path_type = "pgs".  Line searches are either
// golden-section (powell_path == 1, path.cpp:579-935) or exhaustive walks on the lambda grid (seq_search, :954-1137).
// Everything below is control flow on scalars; each evaluation is one Driver::step on the device.  The reference's
// statefulness is kept literally (stale "temp" records after a bracket swap, the warm start of the closing fit, ...):
// those decide which model is returned.
// ======================================================================================================================
enum { SLOT_WARM = 0, SLOT_PREV = 1, SLOT_PREV_FOLD = 2 };

struct Pgs {
    Driver &dr;
    BessResult &out;
    int s_min, s_max;
    double lmin, lmax;  // log(lambda) bounds (bess.cpp:171-172)
    bool warm;

    static int sign(double a) { return a > 0 ? 1 : (a < 0 ? -1 : 0); }  // path.cpp:391-405
    void cal_intersections(const double p[2], const double u[2], double a[2], double b[2]) const
    {
        // the reference prints a diagnostic and carries on with uninitialised end points (path.cpp:539-574)
        if (pgs_line_box(p, u, s_min, s_max, lmin, lmax, a, b) < 2)
            throw EngineError{"pgs_path: search line does not cross the (s, lambda) box twice"};
    }

    // One evaluation: full-data fit at (T, exp(loglam)) then metric->ic() and metric->train_loss() in the order every
    // call site uses (path.cpp:633-650).  Under CV the recorded model is what Algorithm holds AFTER ic(): the last
    // fold's fit, with that beta's full-data loss.
    Eval eval(double Td, double loglam)
    {
        const int T = (int)Td;  // update_sparsity_level(int) truncates
        if (T < 1 || T > dr.kcap) throw EngineError{"pgs_path: sparsity level left [1, s_max]"};
        if (warm) {
            dr.eng.chain_state(0, STATE_SAVE, SLOT_PREV, SLOT_PREV);
            if (dr.K > 0) dr.eng.chain_state(dr.K, STATE_SAVE, SLOT_PREV_FOLD, -1);
        }
        Eval lf;
        Eval e = dr.step(T, &lf, std::exp(loglam));
        std::vector<double> b;
        double c0;
        dr.denormalise(lf, b, c0);
        out.A_all.push_back(lf.A);
        out.bA_all.push_back(std::move(b));
        out.coef0_all.push_back(c0);
        out.train_loss_all.push_back(lf.train_loss);
        out.ic_all.push_back(lf.ic);
        out.s_all.push_back(T);
        out.l_all.push_back(e.l);
        out.lambda_all.push_back(e.lambda);
        lf.lambda = e.lambda;
        return lf;
    }
    void zero_start()
    {
        if (warm) dr.eng.chain_state(0, STATE_ZERO, -1, -1);  // beta_init = 0, coef0_init = 0 (path.cpp:590-592, 966-967)
    }

    // path.cpp:579-935.  p may alias best_arg (P[0] -> P[0]).
    void golden_section_search(const double p[2], const double u[2], double best_arg[2], Eval &best)
    {
        zero_start();
        const double s_tol = 2;
        const double log_lambda_tol = (lmax - lmin) / 200;
        const double invphi = (std::pow(5.0, 0.5) - 1.0) / 2.0;
        const double invphi2 = (3.0 - std::pow(5.0, 0.5)) / 2.0;
        double a[2], b[2], c[2], d[2], h[2];
        cal_intersections(p, u, a, b);
        h[0] = b[0] - a[0];
        h[1] = b[1] - a[1];
        c[0] = a[0] + invphi2 * h[0];
        c[1] = a[1] + invphi2 * h[1];
        d[0] = a[0] + invphi * h[0];
        d[1] = a[1] + invphi * h[1];
        if (h[0] > 0.0001) {
            c[0] = (int)c[0];
            d[0] = std::ceil(d[0]);
        } else if (h[0] < -0.0001) {
            c[0] = std::ceil(c[0]);
            d[0] = (int)d[0];
        } else {
            c[0] = std::round(c[0]);
            d[0] = std::round(d[0]);
        }
        // temp1 / temp2 are only refreshed when c / d is EVALUATED; a bracket swap moves closs / dloss but not them
        Eval temp1 = eval(c[0], c[1]);
        double closs = temp1.ic;
        Eval temp2 = eval(d[0], d[1]);
        double dloss = temp2.ic;
        auto small = [&] {
            return std::fabs((invphi2 - invphi) * h[0]) <= s_tol && std::fabs((invphi2 - invphi) * h[1]) < log_lambda_tol;
        };
        auto finish = [&] {
            double min_loss;
            const double c0 = c[0], c1 = c[1];
            if (closs < dloss) {
                best_arg[0] = c[0];
                best_arg[1] = c[1];
                min_loss = closs;
                best = temp1;
                best.ic = closs;
            } else {
                best_arg[0] = d[0];
                best_arg[1] = d[1];
                min_loss = dloss;
                best = temp2;
                best.ic = dloss;
            }
            for (int i = 1; i < std::fabs((invphi2 - invphi) * h[0]); i++) {
                Eval e = eval((double)(int)(c0 + sign(h[0]) * i), c1);
                if (e.ic < min_loss) {
                    best_arg[0] = c0 + sign(h[0]) * i;
                    best_arg[1] = c1;
                    min_loss = e.ic;
                    best = e;
                }
            }
        };
        if (small()) {
            finish();
            return;
        }
        int tt = 0;
        while (tt < 100) {
            tt++;
            if (closs < dloss) {
                b[0] = d[0];
                b[1] = d[1];
                d[0] = c[0];
                d[1] = c[1];
                dloss = closs;
                h[0] = b[0] - a[0];
                h[1] = b[1] - a[1];
                c[0] = a[0] + invphi2 * h[0];
                c[1] = a[1] + invphi2 * h[1];
                if (h[0] > 0.0001) c[0] = (int)c[0];
                else if (h[0] < -0.0001) c[0] = std::ceil(c[0]);
                else c[0] = std::round(c[0]);
                temp1 = eval(c[0], c[1]);
                closs = temp1.ic;
            } else {
                a[0] = c[0];
                a[1] = c[1];
                c[0] = d[0];
                c[1] = d[1];
                closs = dloss;
                h[0] = b[0] - a[0];
                h[1] = b[1] - a[1];
                d[0] = a[0] + invphi * h[0];
                d[1] = a[1] + invphi * h[1];
                if (h[0] > 0.0001) d[0] = std::ceil(d[0]);
                else if (h[0] < -0.0001) d[0] = (int)d[0];
                else d[0] = std::round(d[0]);
                temp2 = eval(d[0], d[1]);
                dloss = temp2.ic;
            }
            if (small() || tt == 50) {
                finish();
                return;
            }
        }
    }

    static int GDC(int a, int b)  // path.cpp:937-953
    {
        int Max = a > b ? a : b;
        int Min = (a == Max) ? b : a;
        if (Min == 0) throw EngineError{"pgs_path: degenerate search direction (the reference divides by zero here)"};
        int z = Min;
        while (Max % Min != 0) {
            z = Max % Min;
            Max = Min;
            Min = z;
        }
        return z;
    }

    // path.cpp:954-1137.  u is rescaled IN PLACE to a primitive grid step; p may alias best_arg.
    void seq_search(const double p[2], double u[2], double best_arg[2], Eval &best, int nlambda)
    {
        zero_start();
        const double d_lambda = (lmax - lmin) / (nlambda - 1);
        const int k_lambda = (int)std::fabs(std::round(u[1] / d_lambda));
        if (std::fabs(u[0]) != 1 && k_lambda != 1) {
            if (k_lambda == 0 && u[0] != 0) {
                u[0] = u[0] / std::fabs(u[0]);
            } else if (u[0] == 0 && k_lambda != 0) {
                u[1] = u[1] / k_lambda;
            } else {
                const int gdc = GDC(k_lambda, std::abs((int)u[0]));
                if (gdc) {
                    u[0] = std::round(u[0] / gdc);
                    u[1] = u[1] / gdc;
                }
            }
        }
        const double p0 = p[0], p1 = p[1];
        auto inside = [&](double s, double l) {
            return (s <= s_max) && (l <= lmax + d_lambda * 1e-4) && (s >= s_min) && (l >= lmin - d_lambda * 1e-4);
        };
        std::vector<Eval> fwd, bwd;
        fwd.push_back(eval(p0, p1));
        bwd.push_back(fwd[0]);
        if (warm) dr.eng.chain_state(0, STATE_SAVE, SLOT_WARM, SLOT_WARM);  // beta_warm / coef0_warm (:1040-1041)
        const size_t cap = (size_t)(s_max - s_min + 1) * (size_t)nlambda;    // rows of beta_all_1 / _2 (:999-1006)
        for (int i = 1; inside(p0 + i * u[0], p1 + i * u[1]); i++) {
            if (fwd.size() >= cap) throw EngineError{"pgs_path: seq_search walk longer than the (s, lambda) grid"};
            fwd.push_back(eval(p0 + i * u[0], p1 + i * u[1]));
        }
        if (warm) dr.eng.chain_state(0, STATE_LOAD, SLOT_WARM, SLOT_WARM);  // :1084-1085
        for (int j = 1; inside(p0 - j * u[0], p1 - j * u[1]); j++) {
            if (bwd.size() >= cap) throw EngineError{"pgs_path: seq_search walk longer than the (s, lambda) grid"};
            bwd.push_back(eval(p0 - j * u[0], p1 - j * u[1]));
        }
        size_t m1 = 0, m2 = 0;  // Eigen minCoeff: first minimum
        for (size_t i = 1; i < fwd.size(); i++)
            if (fwd[i].ic < fwd[m1].ic) m1 = i;
        for (size_t j = 1; j < bwd.size(); j++)
            if (bwd[j].ic < bwd[m2].ic) m2 = j;
        int min_position;
        if (fwd[m1].ic < bwd[m2].ic) {
            min_position = (int)m1;
            best = fwd[m1];
        } else {
            min_position = -(int)m2;
            best = bwd[m2];
        }
        best_arg[0] = p0 + min_position * u[0];
        best_arg[1] = p1 + min_position * u[1];
    }

    void run(Eval &best, double &best_lambda)
    {
        const BessArgs &a = dr.a;
        const int powell_path = a.powell_path;
        const int nlambda = powell_path == 1 ? 100 : a.nlambda;
        if (nlambda < 2) throw EngineError{"pgs_path: nlambda must be >= 2"};
        double P[3][2], U[2][2];
        P[0][0] = (double)s_min;
        P[0][1] = lmin;
        U[1][0] = 1.;
        U[1][1] = 0.;
        U[0][0] = 0.;
        U[0][1] = (lmax - lmin) / (nlambda - 1);
        std::vector<Eval> rec(16);
        std::vector<double> lam(16, 0.0);
        auto search = [&](double *p, double *u, double *arg, Eval &e) {
            if (powell_path == 1) golden_section_search(p, u, arg, e);
            else seq_search(p, u, arg, e, nlambda);
        };
        int ttt = 0;
        search(P[0], U[1], P[0], rec[0]);
        lam[0] = std::exp(P[0][1]);
        while (ttt < 11) {
            ttt++;
            for (int i = 0; i < 2; i++) {
                search(P[i], U[i], P[i + 1], rec[(size_t)ttt]);
                lam[(size_t)ttt] = std::exp(P[i + 1][1]);
                ttt++;
            }
            U[0][0] = U[1][0];
            U[0][1] = U[1][1];
            U[1][0] = P[2][0] - P[0][0];
            U[1][1] = P[2][1] - P[0][1];
            if ((!(std::fabs(U[1][0]) <= 0.0001 && std::fabs(U[1][1]) <= 0.0001)) && ttt < 11) {
                search(P[0], U[1], P[0], rec[(size_t)ttt]);
                lam[(size_t)ttt] = std::exp(P[0][1]);
            } else {
                // the closing fit at P[0] (:1212-1225).  Neither update_beta_init nor update_coef0_init is called, so it
                // starts from whatever Algorithm was last handed: coef0_init of the search's last fit, and beta_init of
                // that fit -- or, under CV, of the last fold fitted by the ic() behind it (Metric.h:179).
                const int T = (int)P[0][0];
                if (T < 1 || T > dr.kcap) throw EngineError{"pgs_path: sparsity level left [1, s_max]"};
                if (warm) dr.eng.chain_state(0, STATE_LOAD, dr.K > 0 ? SLOT_PREV_FOLD : SLOT_PREV, SLOT_PREV);
                Eval e = dr.step(T, nullptr, std::exp(P[0][1]));
                rec[(size_t)ttt] = e;
                lam[(size_t)ttt] = std::exp(P[0][1]);
                std::vector<double> b;
                double c0;
                dr.denormalise(e, b, c0);
                out.A_all.push_back(e.A);
                out.bA_all.push_back(std::move(b));
                out.coef0_all.push_back(c0);
                out.train_loss_all.push_back(e.train_loss);
                out.ic_all.push_back(e.ic);
                out.s_all.push_back(T);
                out.l_all.push_back(e.l);
                out.lambda_all.push_back(e.lambda);
                ttt++;
                size_t mi = 0;  // ic_all.minCoeff (:1262), ties go to the closing fit (:1263-1266)
                for (size_t i = 1; i < (size_t)ttt; i++)
                    if (rec[i].ic < rec[mi].ic) mi = i;
                if (rec[mi].ic == rec[(size_t)ttt - 1].ic) mi = (size_t)ttt - 1;
                best = rec[mi];
                best_lambda = lam[mi];
                return;
            }
        }
        throw EngineError{"pgs_path: no result (the reference returns an empty list here)"};
    }
};

void pgs_path(Driver &dr, BessResult &out, Eval &best)
{
    const BessArgs &a = dr.a;
    Pgs g{dr, out, a.s_min, a.s_max, std::log(std::max(a.lambda_min, 1e-5)), std::log(std::max(a.lambda_max, 1e-5)),
          a.is_warm_start};
    if (!(g.lmax > g.lmin)) throw EngineError{"pgs_path needs lambda_max > max(lambda_min, 1e-5)"};
    double lam = 0.0;
    g.run(best, lam);
    best.lambda = lam;  // lambda_chosen (:1176, 1192, 1207): the line search's end point, not the record's own level
}

}  // namespace

void fold_shard_chains(int K, int world, int rank, bool last_fold_everywhere, std::vector<int> &chains, std::vector<char> &counts)
{
    chains.assign(1, 0);
    counts.assign(1, 0);
    for (int c = 1; c <= K; c++) {
        const bool mine = world <= 1 || c % world == rank;
        const bool everyone = world > 1 && c == K && last_fold_everywhere;
        if (mine || everyone) {
            chains.push_back(c);
            counts.push_back(mine ? 1 : 0);
        }
    }
}

// Where a sparse design without screening is swept: on its CSC arrays (the dual sweep reads 12 bytes per stored entry, the
// fits read the active columns expanded from them) or densified (8 bytes per entry, stored or not, read by every sweep).
// Small designs stay dense: every one up to 1 GiB, which includes every design of the resident path (64 MB).  Larger
// ones keep the CSC form when it is at most 1 / KEEP_SPARSE_RATIO of the dense bytes -- the crossover measured in
// DESIGN 3.12 -- or when the dense form could not fit the device at all.  The device's total memory decides, not its
// free memory, so that a call's numerics never depend on what other jobs hold.
constexpr double KEEP_SPARSE_RATIO = 24.0;
bool keep_sparse(long long n, long long p, long long nnz, size_t device_total)
{
    const double dense = 8.0 * (double)n * (double)(((p + 1) & ~1LL));
    const double sparse = 12.0 * (double)nnz + 8.0 * ((double)p + 1);
    return (dense > (double)(1LL << 30) && sparse * KEEP_SPARSE_RATIO <= dense) || dense > (double)device_total;
}

static void bess_run_once(const BessArgs &a, BessResult &out, bool tie_exact)
{
    // ---- argument validation (the reference validates in its R/Python front-ends and dereferences null otherwise,
    // SURVEY Q19; here bad arguments are reported)
    if ((!a.x && !a.csc) || !a.y || !a.weight) throw EngineError{"x, y and weight must be non-null"};
    if (a.csc && a.x) throw EngineError{"x and x_csc are both given: pass the design one way"};
    if (a.csc && a.world > 1) throw EngineError{"a sparse design (x_csc) is single-GPU only (world must be <= 1)"};
    if (a.n < 2 || a.p < 1) throw EngineError{"need n >= 2 and p >= 1"};
    if (!(a.algorithm_type == 1 || a.algorithm_type == 2 || a.algorithm_type == 3 || a.algorithm_type == 5))
        throw EngineError{"algorithm_type must be 1 (PDAS), 2, 3 or 5 (bess.cpp:93)"};
    if (a.model_type < 1 || a.model_type > 4) throw EngineError{"model_type must be 1..4"};
    if (a.data_type < 1 || a.data_type > 3) throw EngineError{"data_type must be 1..3"};
    // bess.cpp:167-180: path_type != 1 runs pgs_path for the L0L2 algorithm types and gs_path otherwise
    const bool pgs = a.path_type != 1 && (a.algorithm_type == 5 || a.algorithm_type == 3);
    if (pgs && a.world > 1) throw EngineError{"pgs_path is not available in column-sharded / fold-sharded mode"};
    if (a.fold_shard && a.world > 1 && a.cv_reduce_over_ranks) throw EngineError{"fold_shard and cv_reduce_over_ranks exclude each other"};
    if (a.cv_reduce_over_ranks && a.world > 1 && !(a.path_type == 1 && a.is_cv && a.is_screening))
        throw EngineError{"cv_reduce_over_ranks needs the sequential path with CV and screening (ranks share the screened "
                          "design and differ only in their folds)"};
    if (pgs && !(a.lambda_min >= 0.0 && a.lambda_max >= 0.0)) throw EngineError{"lambda_min / lambda_max must be >= 0"};
    if (pgs && a.powell_path != 1 && a.powell_path != 2) throw EngineError{"powell_path must be 1 (golden section) or 2 (sequential)"};
    if (a.path_type == 1)
        for (double l : a.lambda_seq)
            if (!(l >= 0.0)) throw EngineError{"lambda_seq entries must be >= 0"};
    // g_index: first column of every group (bess.R:540, linear.py:238-254).  p entries = no group structure.
    const bool grouped = !a.g_index.empty() && (int)a.g_index.size() != a.p;
    if (!a.g_index.empty() && !grouped)
        for (int j = 0; j < a.p; j++)
            if (a.g_index[(size_t)j] != j) throw EngineError{"g_index with p entries must be 0..p-1"};
    if (grouped) {
        if (a.algorithm_type != 2 && a.algorithm_type != 3)
            throw EngineError{"group selection needs algorithm_type 2 (GPDAS) or 3 (GL0L2)"};
        // the reference un-screens a grouped fit by group number (bess.cpp:186-209 writes beta(screening_A(i))), which
        // scrambles the coefficients; there is no defined behaviour to reproduce
        if (a.is_screening) throw EngineError{"screening together with group selection is not supported"};
        if (a.world > 1 && !a.fold_shard) throw EngineError{"group selection is not available in column-sharded mode"};
    }
    if (a.is_cv && (a.K < 2 || a.K > MAXC - 1)) throw EngineError{"K (nfolds) must be in [2, 31]"};
    const bool shard = a.world > 1 && !a.fold_shard;  // columns sharded (axis B); fold_shard: the design is replicated
    const long long p_all = shard ? a.p_total : a.p;
    if (shard && a.x_on_device == false && a.x == nullptr) throw EngineError{"sharded fit: x shard is null"};
    const long long n_units = grouped ? (long long)a.g_index.size() : p_all;  // what s.list / always_select count
    for (int j : a.always_select)
        if (j < 0 || j >= n_units) throw EngineError{"always_select index out of range"};

    using clk = std::chrono::steady_clock;
    auto t_last = clk::now();
    auto lap = [&](int phase) {
        const auto now = clk::now();
        out.host_ms[phase] += std::chrono::duration<double, std::milli>(now - t_last).count();
        t_last = now;
    };
    Engine eng(a.device);
    eng.set_tie_exact(tie_exact);
    eng.set_profiling(a.profile);
    if (shard) eng.init_shard(a.world, a.rank, a.nccl_id, a.col_lo, a.p_total);
    else if (a.fold_shard && a.world > 1 && a.is_cv) eng.init_comm(a.world, a.rank, a.nccl_id);
    if (a.csc) {
        eng.load_csc(a.csc_colptr, a.csc_rowidx, a.csc_values, a.n, a.p, a.csc_nnz, a.x_on_device, a.y, a.weight, a.model_type);
        // screening densifies only the columns it keeps; without it the design is densified unless the sweeps run on the
        // CSC arrays (keep_sparse)
        if (!a.is_screening && (grouped || !keep_sparse(a.n, a.p, a.csc_nnz, eng.device_total_bytes()))) eng.densify();
    } else {
        eng.load(a.x, a.n, a.p, a.x_on_device, a.y, a.weight, a.model_type, /*borrow=*/a.is_screening);
    }

    lap(0);
    std::vector<int> always = a.always_select;
    std::sort(always.begin(), always.end());
    if (a.is_screening) {
        if (a.screening_size < 1 || a.screening_size > p_all) throw EngineError{"screening_size must be in [1, p]"};
        // only device work is enqueued here; the kept-column list is read when it is first needed -- for the remap of
        // always_select right away, else at the end of the call (the normalisation and the path queue up behind it)
        eng.screen_enqueue(a.screening_size, always);
        if (!always.empty()) out.screening_A = eng.screen_result();
        // screening.cpp:91-102: always_select -> positions inside the screened matrix
        for (int &j : always) {
            auto it = std::lower_bound(out.screening_A.begin(), out.screening_A.end(), j);
            if (it == out.screening_A.end() || *it != j) throw EngineError{"always_select column lost in screening"};
            j = (int)(it - out.screening_A.begin());
        }
    }
    lap(1);
    eng.normalize(a.data_type, a.is_normal);
    if (grouped) eng.set_groups(a.g_index);
    lap(2);

    const long long p = grouped ? (long long)eng.n_groups() : eng.p_model();
    int kcap;
    if (a.path_type == 1) {
        if (a.sequence.empty()) throw EngineError{"sequence (s.list) is empty"};
        kcap = *std::max_element(a.sequence.begin(), a.sequence.end());
        if (*std::min_element(a.sequence.begin(), a.sequence.end()) < 1) throw EngineError{"s.list entries must be >= 1"};
    } else {
        if (a.s_min < 1 || a.s_max < a.s_min) throw EngineError{"need 1 <= s_min <= s_max"};
        kcap = a.s_max;
    }
    if (kcap > p) throw EngineError{"sparsity level exceeds the number of (screened) columns / groups"};

    std::vector<int> folds;
    if (a.is_cv) {
        if (a.fold_of_row) folds.assign(a.fold_of_row, a.fold_of_row + a.n);
        else folds = cv_fold_ids(a.n, a.K, a.cv_seed);
    }
    eng.setup_chains(a.is_cv ? a.K : 0, folds.data(), kcap, a.max_iter, a.is_warm_start, always);

    lap(3);
    Driver dr(eng, a);
    dr.kcap = kcap;
    if (dr.fshard) eng.set_cluster_chains(dr.max_chains_per_rank());
    Eval best;
    if (a.path_type == 1) sequential_path(dr, out, best);
    else if (pgs) pgs_path(dr, out, best);
    else gs_path(dr, out, best);

    lap(4);
    if (a.is_screening && out.screening_A.empty()) out.screening_A = eng.screen_result();
    std::vector<double> bA;
    double coef0;
    dr.denormalise(best, bA, coef0);
    out.coef0 = coef0;
    out.train_loss = best.train_loss;
    out.ic = best.ic;
    out.lambda = best.lambda;
    out.chosen_s = best.T;
    // scatter to the ORIGINAL column numbering (un-screen: bess.cpp:186-209)
    out.p_out = p_all;
    out.beta_idx.clear();
    out.beta_val.clear();
    auto orig = [&](int j) { return a.is_screening ? out.screening_A[(size_t)j] : j; };
    for (size_t i = 0; i < best.A.size(); i++) {
        out.beta_idx.push_back(orig(best.A[i]));
        out.beta_val.push_back(bA[i]);
    }
    for (auto &A : out.A_all)
        for (int &j : A) j = orig(j);
    out.sparse_sweeps = eng.sparse_sweeps();
    out.stats = eng.stats();
    out.stats.n_rank_deficient += debug_take_rankdef();
    out.stats.n_wide_singular += take_wide_singular();
    eng.profile(out.prof_ms, out.prof_n);
    out.sweep_splits = eng.sweep_splits();
    eng.resident_counters(out.resident);
    eng.resident_owner_counters(out.resident + 24);
}

// bessCpp (bess.cpp:37-214) on the device.  The fast pass resolves a boundary tie of a top-k selection -- the k-th and the
// (k+1)-th sacrifice / screening utility exactly equal, e.g. duplicated columns -- towards the lower index and counts it;
// the reference leaves such a tie to std::nth_element (utilities.cpp:179-188, SURVEY a-5).  When the fast pass met one,
// the whole call is repeated in exact mode, where every tied selection is redone on the host with the reference's own
// index-array nth_element + sort (Engine::set_tie_exact).  Continuous designs never take the second pass.
void bess_run(const BessArgs &a, BessResult &out)
{
    bess_run_once(a, out, false);
    static const bool redo = [] {
        const char *e = std::getenv("BESS_B200_TIE_EXACT");
        return !(e && e[0] == '0');
    }();
    // A dependent column inside an active set (an exact duplicate both of whose copies were selected, e.g. by a cold
    // start): the resident kernel flags it (its plain Cholesky has no answer), and a non-finite result says the same of a
    // wide system.  The exact mode runs on the multi-kernel path, whose small-system solver falls back to a rank-revealing
    // LDL^T that truncates like the reference's colPivHouseholderQr / pivoted ldlt (chain_fit.cu: ldlt_pivoted_small).
    // Its wide-system solver (more than 63 unknowns, e.g. a sparsity level above the number of training rows) has no such
    // fallback: it returns NaN and counts the system, and any level of the path -- chosen or not -- may carry it.
    auto all_finite = [](const std::vector<double> &v) {
        for (double x : v)
            if (!std::isfinite(x)) return false;
        return true;
    };
    auto finite_result = [&](const BessResult &r) {
        bool f = std::isfinite(r.train_loss) && std::isfinite(r.ic) && std::isfinite(r.coef0);
        return f && all_finite(r.beta_val) && all_finite(r.ic_all) && all_finite(r.train_loss_all);
    };
    const bool suspect = out.stats.n_suspect_pivots > 0 || out.stats.n_wide_singular > 0 || !finite_result(out);
    if (redo && (out.stats.n_boundary_ties > 0 || suspect) && a.world <= 1) {
        const bool ties = out.stats.n_boundary_ties > 0;
        BessResult exact;
        bess_run_once(a, exact, true);
        out = std::move(exact);
        out.tie_exact_pass = ties;
        out.robust_pass = suspect;
    }
    if (out.stats.n_wide_singular > 0)
        throw EngineError{"rank-deficient wide system: the normal equations of a support with more than 63 unknowns are "
                          "singular (is the sparsity level above the number of training rows?); only systems of up to 63 "
                          "unknowns are solved rank-revealingly"};
    if (!finite_result(out)) throw EngineError{"non-finite criterion, loss or coefficient on the path"};
}

}  // namespace bess
