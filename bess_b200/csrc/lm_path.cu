// Resident PDAS path for the gaussian family: Algorithm::fit (/root/reference/src/Algorithm.h:113-171) with
// GroupPdasLm::get_A / primary_model_fit (:1097-1135), max_k (utilities.cpp:179-199), the warm-started level loop of
// sequential_path (path.cpp:48-74) and the Lm losses of Metric.h:145-148 / 190 -- for ALL chains of a batch (full-data
// fit + CV folds) and ALL steps of a path segment in ONE cooperative launch.
//
// Why: after screening (BASELINE config 5: 1000 x 5000, 11 chains, s = 1..20) the design is L2-resident and a PDAS
// iteration is a few microseconds of work; launched as sweep / top-k / fit kernels the path was ~55 dependent iterations
// of three 11-to-300-CTA launches each (profiles/r01g_small_kernels_full.md: 1-2 % SM throughput).  Here the iteration
// loop lives on the device:
//
//   * SWEEPER CTAs (all but one CTA per chain) each own a slice of ~p/137 adjacent columns for the whole launch.  Per
//     iteration a sweeper stages the residual vectors of all chains ([n][FT], one bulk-TMA copy into shared memory), walks
//     all n rows of its slice once (the leading rows from a copy it keeps in the shared memory the owners' budget leaves
//     it, the others as 16-byte loads of X from L2; 2*FT fp64 FMAs per 16 bytes), reduces its row phases in a
//     fixed order, applies the splicing sacrifice (Algorithm.h:1112-1123) and writes bd; values above the chain's
//     published threshold are appended to a short candidate list.  No row splits, no partial vectors in memory.
//   * one OWNER CTA per chain keeps the chain's state in shared memory for the whole launch: the active columns X_A (all
//     n rows, column-major, in reusable slots), their Gram matrix and X_A^T y (cached per slot pair -- a PDAS iteration
//     typically exchanges 0-3 columns, only those rows of the Gram are recomputed), the response, the fold mask and
//     A_list.  Per iteration it ranks the best candidates (exact top-k: larger value first, lower index first; falls back to a
//     radix select over the whole bd vector when the list is short or overflows), loads the new columns, solves the
//     bordered normal equations by Cholesky, publishes the residual of the next sweep and runs the cycle test
//     (Algorithm.h:164-170).  A chain that has met the stopping rule writes its result (support, coefficients, l, train /
//     held-out loss) and moves on to ITS next path step at once -- the chains of a batch are independent lineages
//     (SURVEY 7.2), so nobody waits for the slowest chain of a level.
//   * two counters in global memory order the phases: sweepers arrive at B1, owners wait for it; owners arrive at B2,
//     everybody waits for it.  The launch is cooperative (all CTAs co-resident), a watchdog turns a lost arrival into an
//     error instead of a hang.
//
// The results are bitwise reproducible from run to run (fixed summation orders; the candidate list is unordered but its
// ranking is a total order) and equal to the multi-kernel path up to fp64 re-association (supports identical).
#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>
#include <type_traits>

#include "device_utils.cuh"
#include "lm_path.cuh"

namespace bess {

namespace {

// ---------------------------------------------------------------------------------------------------------------------
// small PTX helpers
// ---------------------------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t lp_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void lp_mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(lp_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void lp_mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(lp_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void lp_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     lp_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(lp_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ bool lp_mbar_try(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%1], %2;\n"
        "selp.u32 %0, 1, 0, P1;\n"
        "}"
        : "=r"(ok)
        : "r"(lp_smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void lp_mbar_wait(uint64_t *bar, uint32_t parity)
{
    while (!lp_mbar_try(bar, parity)) {
    }
}
__device__ __forceinline__ unsigned ld_acquire_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void red_release_add_u32(unsigned *p, unsigned v)
{
    asm volatile("red.release.gpu.global.add.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ double2 ldg_stream_v2(const double *p)
{
    double2 v;
    asm("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "l"(p));
    return v;
}
__device__ __forceinline__ double ldg_stream(const double *p)
{
    double v;
    asm("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(v) : "l"(p));
    return v;
}
__device__ __forceinline__ unsigned long long lp_globaltimer()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}

// ---------------------------------------------------------------------------------------------------------------------
// phase barriers: monotonic counters in global memory
// ---------------------------------------------------------------------------------------------------------------------
constexpr unsigned long long LP_WATCHDOG_NS = 4000000000ull;  // a lost arrival becomes an error after 4 s

__device__ __forceinline__ unsigned ld_relaxed_u32(const unsigned *p)
{
    unsigned v;
    asm volatile("ld.relaxed.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void fence_acq_rel_gpu() { asm volatile("fence.acq_rel.gpu;" ::: "memory"); }

// The CTA's writes so far (ordered before thread 0's release by the block barrier) become visible to whoever acquires
// the counter afterwards.
__device__ __forceinline__ void cta_arrive(unsigned *ctr, unsigned add = 1u)
{
    __syncthreads();
    if (threadIdx.x == 0) red_release_add_u32(ctr, add);
}
// The owner that sets LP_SYNC_TERM adds this flag with its next arrival at B2.  A waiter that reads no flag in the counters
// of its decision point knows, without reading the termination word, that no phase up to that point has set it.
constexpr unsigned LP_TERM_FLAG = 1u << 31;
// Thread 0 polls counters with RELAXED loads (an acquire load invalidates the L1 on every poll) and fences once when all
// have reached their targets.  The abort word is loaded with the counters, not after them: one L2 round trip per poll.
// *flags <- LP_TERM_FLAG when a counter carried it.  Returns false when the launch was aborted (by this or another CTA's
// watchdog).
__device__ __forceinline__ bool poll_until(unsigned *sync, int w0, unsigned t0, int w1, unsigned t1, unsigned *flags)
{
    unsigned spins = 0;
    unsigned long long ts = 0;
    for (;;) {
        const unsigned v0 = ld_relaxed_u32(sync + w0);
        const unsigned v1 = w1 < 0 ? t1 : ld_relaxed_u32(sync + w1);
        if (ld_relaxed_u32(sync + LP_SYNC_ABORT) != 0u) return false;
        if ((v0 & ~LP_TERM_FLAG) >= t0 && (v1 & ~LP_TERM_FLAG) >= t1) {
            *flags = (v0 | v1) & LP_TERM_FLAG;
            break;
        }
        if ((++spins & 0x3ffu) == 0u) {
            if (ts == 0) ts = lp_globaltimer();
            if (lp_globaltimer() - ts > LP_WATCHDOG_NS) {
                atomicExch(sync + LP_SYNC_ABORT, 1u);
                return false;
            }
        }
    }
    fence_acq_rel_gpu();
    return true;
}
// The CTA waits for counters w0 / w1 (w1 < 0: none), then decides: LP_WAIT_TERM when the termination word holds a phase
// index at or below `decision` (see sweeper_main); else, when wb >= 0, it waits for counter wb as well.  Every phase up to
// `decision` has arrived on w0 / w1 by then (the owner that sets the word arrives with LP_TERM_FLAG), or on a counter of an
// earlier decision point of this CTA, at which it would have left; so the word is read only when a counter carries the
// flag.  Thread 0 does all of it and hands the outcome to the CTA through one block barrier pair.
enum { LP_WAIT_ABORT = 0, LP_WAIT_GO = 1, LP_WAIT_TERM = 2 };
__device__ __forceinline__ int cta_wait_term(unsigned *sync, int w0, unsigned t0, int w1, unsigned t1, unsigned decision,
                                             int wb, unsigned tb, int *flag_sh)
{
    if (threadIdx.x == 0) {
        int res = LP_WAIT_ABORT;
        unsigned flags = 0u, fb;
        if (poll_until(sync, w0, t0, w1, t1, &flags)) {
            const unsigned term = flags ? ld_acquire_u32(sync + LP_SYNC_TERM) : 0u;
            if (term != 0u && term - 1u <= decision) res = LP_WAIT_TERM;
            else if (wb < 0 || poll_until(sync, wb, tb, -1, 0u, &fb)) res = LP_WAIT_GO;
        }
        *flag_sh = res;
    }
    __syncthreads();
    const int res = *flag_sh;
    __syncthreads();
    return res;
}

// Phase-timer and counter width of a kernel instantiation.  Per launch the sums stay far below 2^32 clocks, and 32-bit
// sums leave registers to the owner's hot code: at FT = 6 the kernel's spills fall from 130 to 64 bytes and the slowest
// owner phase of a C5 round from 18.7 to 16.5 us.  The widest residual stages keep 64 bits; there the narrower sums only
// move the spills into the sweep.
template <int FT>
using LpTick = typename std::conditional<(FT >= 12), unsigned long long, unsigned>::type;

// Phase timers of ONE thread (clock ticks).  The sums stay in that thread's registers and are flushed to global memory
// once, when the CTA leaves -- a read-modify-write of global memory per mark stalls the timing warp (and everybody
// behind the next barrier) for an L2 round trip, which at 13 marks per fit distorted what it measured.
template <int NSLOT, typename Tick>
struct Timer {
    long long t;
    bool on;
    Tick acc[NSLOT];
    __device__ __forceinline__ void start(bool enable)
    {
        on = enable;
#pragma unroll
        for (int q = 0; q < NSLOT; q++) acc[q] = 0;
        if (on) t = clock64();
    }
    __device__ __forceinline__ void mark(int id)
    {
        if (on) {
            const long long now = clock64();
            const Tick dt = (Tick)(now - t);
#pragma unroll
            for (int q = 0; q < NSLOT; q++)
                if (q == id) acc[q] += dt;
            t = now;
        }
    }
    __device__ __forceinline__ void flush(unsigned long long *dst)
    {
        if (on) {
#pragma unroll
            for (int q = 0; q < NSLOT; q++) dst[q] += acc[q];
        }
    }
};

// =====================================================================================================================
// SWEEPER
// =====================================================================================================================
struct SweepSm {
    double *R;        // [npad][FT] residual vectors of all chain slots; aliased by the row-phase scratch [RP][FT][W2]
    double *tau;      // [16]
    double *lam;      // [16]
    uint64_t *mbar;
    int *flag;
};

__host__ __device__ inline size_t sweeper_smem_doubles(int npad, int FT)
{
    const size_t r = (size_t)npad * FT;
    const size_t scr = (size_t)2 * LP_NT * FT;  // RP * Wp <= LP_NT
    return (r > scr ? r : scr) + 16 + 16 + 2 + 2;
}

// Slice width in column pairs, rounded to even: a row segment of an even number of pairs is a whole number of 32-byte
// sectors (measured: 18-pair slices stream 15 % faster than 17- or 19-pair ones)
__host__ __device__ inline int sweeper_pairs(int p, int nsweep)
{
    const int P2 = (p + 1) >> 1;
    int WpA = (P2 + nsweep - 1) / nsweep;
    if (WpA > 1 && (WpA & 1) && WpA < LP_WPMAX) WpA++;
    return WpA;
}

template <int FT>
__device__ void sweeper_main(const Dev &d, const LpDesc &L, unsigned char *raw)
{
    SweepSm sm;
    {
        double *p = reinterpret_cast<double *>(raw);
        const size_t r = (size_t)((d.n + 1) & ~1) * FT, scr = (size_t)2 * LP_NT * FT;
        sm.R = p;
        p += (r > scr ? r : scr);
        sm.tau = p;
        p += 16;
        sm.lam = p;
        p += 16;
        sm.mbar = reinterpret_cast<uint64_t *>(p);
        p += 2;
        sm.flag = reinterpret_cast<int *>(p);
    }
    const int tid = threadIdx.x;
    const int n = d.n, npad = (n + 1) & ~1;
    const int sidx = (int)blockIdx.x - L.nch;
    const int P2 = (d.p + 1) >> 1;
    const int WpA = sweeper_pairs(d.p, L.nsweep);
    const int q0 = min(P2, sidx * WpA), q1 = min(P2, q0 + WpA);
    const int Wp = q1 - q0;
    const int RP = Wp > 0 ? min(LP_NT / Wp, LP_RPMAX) : 0;
    const int cp = Wp > 0 ? tid % Wp : 0, rp = Wp > 0 ? tid / Wp : 0;
    const bool active = Wp > 0 && rp < RP;
    const int W2 = 2 * Wp, nout = W2 * FT;
    const uint32_t rbytes = (uint32_t)((size_t)npad * FT * sizeof(double));
    // The launch sizes its shared memory for the owners; what the residual stage leaves free keeps the first nres rows of
    // the slice on chip for the whole launch, [nres][W2] (a warp's double2 reads are consecutive: conflict-free).  Each sweep
    // reads those rows from shared memory and streams only rows nres.. from L2.
    double2 *Xs = reinterpret_cast<double2 *>(raw + sweeper_smem_doubles(npad, FT) * sizeof(double));
    int nres = 0;
    if (Wp > 0) {
        unsigned dyn;
        asm("mov.u32 %0, %%dynamic_smem_size;" : "=r"(dyn));
        const size_t used = sweeper_smem_doubles(npad, FT) * sizeof(double);
        if (dyn > used) nres = (int)min((size_t)n, (dyn - used) / (sizeof(double2) * Wp));
    }
#pragma unroll 4
    for (int e = tid; e < nres * Wp; e += LP_NT) {
        const int i = e / Wp, q = e - i * Wp;
        Xs[e] = ldg_stream_v2(d.X + (size_t)i * d.ldx + 2 * (size_t)(q0 + q));
    }
    if (tid == 0) {
        lp_mbar_init(sm.mbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    Timer<3, LpTick<FT>> tm;
    tm.start(tid == 0 && sidx == 0);
    uint32_t parity = 0;
    // step s sweeps group g = s % ng for the r-th time (r = s / ng + 1) once that group's owners have finished their
    // phase r - 1.  Owner phase O_g(r) has index ng * r + g; LP_SYNC_TERM holds 1 + the index of the phase in which the
    // last chain finished its last step, and everybody leaves at the first decision point at or past it.
    for (unsigned st = 0;; st++) {
        const int g = (int)(st % (unsigned)L.ng);
        const unsigned r = st / (unsigned)L.ng + 1u;
        if (cta_wait_term(L.sync, LP_SYNC_B2 + g, (unsigned)L.gcount[g] * r, -1, 0u, st, -1, 0u, sm.flag) != LP_WAIT_GO) break;
        tm.mark(0);
        if (L.trace && tid == 0 && sidx == 0 && st < LP_TRACE) L.trace[((size_t)MAXC * LP_TRACE + st) * 2] = lp_globaltimer();
        const double *Rsrc = L.Rg[g];
        const int nslot = L.gcount[g];
        if (Wp > 0) {
            if (tid == 0) {
                asm volatile("fence.proxy.async;" ::: "memory");
                lp_mbar_expect_tx(sm.mbar, rbytes);
                uint32_t off = 0;
                while (off < rbytes) {
                    const uint32_t chunk = min(rbytes - off, 32768u);
                    lp_bulk_g2s(reinterpret_cast<unsigned char *>(sm.R) + off, reinterpret_cast<const unsigned char *>(Rsrc) + off,
                                chunk, sm.mbar);
                    off += chunk;
                }
            }
            if (tid < 16) {
                const int cc = tid < nslot ? L.gchain[g][tid] : 0;
                sm.tau[tid] = tid < nslot ? __ldcg(L.pub + 2 * cc) : 0.0;
                sm.lam[tid] = tid < nslot ? __ldcg(L.pub + 2 * cc + 1) : 0.0;
            }
            double a0[FT], a1[FT];
#pragma unroll
            for (int f = 0; f < FT; f++) a0[f] = a1[f] = 0.0;
            if (active) {
                // row i of this thread's column pair into the sums; every thread adds its rows in ascending order
                auto row_fma = [&](const double2 xv, int i) {
                    const double *r = sm.R + (size_t)i * FT;
                    if constexpr (FT == 1) {
                        const double g = r[0];
                        a0[0] = fma(xv.x, g, a0[0]);
                        a1[0] = fma(xv.y, g, a1[0]);
                    } else {
#pragma unroll
                        for (int f = 0; f < FT; f += 2) {
                            const double2 g = *reinterpret_cast<const double2 *>(r + f);
                            a0[f] = fma(xv.x, g.x, a0[f]);
                            a1[f] = fma(xv.y, g.x, a1[f]);
                            a0[f + 1] = fma(xv.x, g.y, a0[f + 1]);
                            a1[f + 1] = fma(xv.y, g.y, a1[f + 1]);
                        }
                    }
                };
                // software pipeline: the x loads of row group g + 1 are in flight while group g is multiplied; the first
                // streamed group is in flight while the on-chip rows are multiplied
                constexpr int U = 4;
                const double *xp = d.X + 2 * (size_t)(q0 + cp);
                const int is = rp + (nres > rp ? (nres - rp + RP - 1) / RP : 0) * RP;  // first row of this thread from L2
                double2 xn[U];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int i = is + u * RP;
                    xn[u] = i < n ? ldg_stream_v2(xp + (size_t)i * d.ldx) : make_double2(0.0, 0.0);
                }
                lp_mbar_wait(sm.mbar, parity);
#pragma unroll 4
                for (int i = rp; i < nres; i += RP) row_fma(Xs[(size_t)i * Wp + cp], i);
                for (int i0 = is; i0 < n; i0 += RP * U) {
                    double2 xv[U];
#pragma unroll
                    for (int u = 0; u < U; u++) xv[u] = xn[u];
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const int i = i0 + (U + u) * RP;
                        xn[u] = i < n ? ldg_stream_v2(xp + (size_t)i * d.ldx) : make_double2(0.0, 0.0);
                    }
#pragma unroll
                    for (int u = 0; u < U; u++) {
                        const int i = i0 + u * RP;
                        if (i < n) row_fma(xv[u], i);
                    }
                }
            } else {
                lp_mbar_wait(sm.mbar, parity);
            }
            parity ^= 1u;
            tm.mark(1);
            __syncthreads();  // every thread is done with R: the scratch may overwrite it
            double *scr = sm.R;
            if (active) {
#pragma unroll
                for (int f = 0; f < FT; f++)
                    *reinterpret_cast<double2 *>(scr + ((size_t)rp * FT + f) * W2 + 2 * cp) = make_double2(a0[f], a1[f]);
            }
            __syncthreads();
            for (int o = tid; o < nout; o += LP_NT) {
                const int f = o / W2, col = o - f * W2;
                const long long j = 2LL * q0 + col;
                if (f >= nslot || j >= d.p) continue;
                const int cc = L.gchain[g][f];  // chain id: row of betaD / xtx / bd, candidate list
                double dsum = 0.0;
                for (int r2 = 0; r2 < RP; r2++) dsum += scr[((size_t)r2 * FT + f) * W2 + col];
                // splicing sacrifice, Algorithm.h:1112-1123 with the L0L2 ridge term (:1109) -- same formula as
                // finish_epilogue<EPI_SACR_LM> of the multi-kernel path
                const double beta = __ldcg(d.betaD + (size_t)cc * d.pstride + j);
                const double lam2 = 2.0 * sm.lam[f];
                const double phi = sqrt(lam2 + __ldg(d.xtx + (size_t)cc * d.pstride + j) / (double)__ldg(d.ntrain + cc));
                const double t = phi * beta + (1.0 / phi) * (dsum - lam2 * beta);
                double v = t * t;
                if (!(v == v)) v = 0.0;  // a NaN sacrifice ranks last (topk_key of the multi-kernel path)
                for (int q = 0; q < L.n_always; q++)
                    if (__ldg(L.always + q) == (int)j) v = DBL_MAX;  // utilities.cpp:190-199
                __stcg(d.bd + (size_t)cc * d.pstride + j, v);
                if (v >= sm.tau[f]) {
                    const int pos = atomicAdd(L.ncand + cc, 1);
                    if (pos < LP_CAP) {
                        LpCand cnd;
                        cnd.v = v;
                        cnd.idx = (int)j;
                        cnd.pad = 0;
                        __stcg(reinterpret_cast<int4 *>(L.cand + (size_t)cc * LP_CAP + pos), *reinterpret_cast<int4 *>(&cnd));
                    }
                }
            }
            tm.mark(2);
        }
        if (L.trace && tid == 0 && sidx == 0 && st < LP_TRACE) L.trace[((size_t)MAXC * LP_TRACE + st) * 2 + 1] = lp_globaltimer();
        cta_arrive(L.sync + LP_SYNC_B1 + g);  // its leading __syncthreads also protects the scratch from the next TMA copy
    }
    tm.flush(L.dbg + 16);
}

// =====================================================================================================================
// OWNER
// =====================================================================================================================
struct OwnSm {
    double *XA;    // [ns][npad] active columns, one per slot, all n rows
    double *y, *m, *my;  // [npad] response, train mask (1/0), their product
    double *Gc;    // [ns][ns] sum_i m_i x_s x_t per slot pair
    double *bc;    // [ns] sum_i m_i y_i x_s
    double *S;     // [(kcap+1)][ldS] bordered normal equations
    double *beta;  // [kcap]
    double *dg;    // [kcap+1]
    double *cv;    // [LP_CAP] candidate values
    double *selv;  // [2*kcap+8] candidate values by rank
    double *bage;  // [kcap+1] solution in factor (age) order
    double *red;   // [40]
    int *ci;       // [LP_CAP]
    int *A, *slotA, *Anew, *slotNew, *newlist;  // [kcap]
    int *seli;     // [2*kcap+8] candidate indices by rank
    int *ord, *ordNew;  // [kcap] slot of the t-th column of the Cholesky factor (columns are kept in order of arrival)
    int *pos;      // [ns] position of a slot's column in that order, -1 when the column is not part of the factor
    int *freel;    // [ns] scratch: free slots
    int *slot_col, *keep;  // [ns]
    int *hist;     // [hist_rows][kcap]
    int *hbin;     // [256]
    int *misc;     // [16]
    int ldS;
};
enum { MI_FLAG = 0, MI_CNT = 1, MI_NNEW = 2, MI_SEEN = 3, MI_TIE = 4, MI_KREM = 5, MI_NEQ = 6, MI_COUNT = 7, MI_Q = 8, MI_RANKN = 9,
       MI_B2ADD = 10 };

__host__ __device__ inline size_t owner_smem_bytes(int npad, int kcap, int ns, int hist_rows)
{
    const int ldS = (kcap + 2) | 1;
    size_t dbl = (size_t)ns * npad + 3 * (size_t)npad + (size_t)ns * ns + ns + (size_t)(kcap + 1) * ldS + kcap + (kcap + 1) +
                 LP_CAP + (2 * kcap + 8) + (kcap + 1) + 40 + 2 /* prefix/scratch */;
    size_t ints = LP_CAP + 7 * (size_t)kcap + (2 * kcap + 8) + 4 * (size_t)ns + (size_t)hist_rows * kcap + 256 + 16 + 64 /* scan */;
    return dbl * 8 + ((ints + 1) & ~(size_t)1) * 4;
}

__device__ __forceinline__ OwnSm carve_owner(unsigned char *raw, int npad, int kcap, int ns, int hist_rows, double **pre_out,
                                             int **scan_out)
{
    OwnSm s;
    double *p = reinterpret_cast<double *>(raw);
    s.ldS = (kcap + 2) | 1;
    s.XA = p; p += (size_t)ns * npad;
    s.y = p; p += npad;
    s.m = p; p += npad;
    s.my = p; p += npad;
    s.Gc = p; p += (size_t)ns * ns;
    s.bc = p; p += ns;
    s.S = p; p += (size_t)(kcap + 1) * s.ldS;
    s.beta = p; p += kcap;
    s.dg = p; p += kcap + 1;
    s.cv = p; p += LP_CAP;
    s.selv = p; p += 2 * kcap + 8;
    s.bage = p; p += kcap + 1;
    s.red = p; p += 40;
    *pre_out = p; p += 2;
    int *q = reinterpret_cast<int *>(p);
    s.ci = q; q += LP_CAP;
    s.A = q; q += kcap;
    s.slotA = q; q += kcap;
    s.Anew = q; q += kcap;
    s.slotNew = q; q += kcap;
    s.newlist = q; q += kcap;
    s.seli = q; q += 2 * kcap + 8;
    s.ord = q; q += kcap;
    s.ordNew = q; q += kcap;
    s.pos = q; q += ns;
    s.freel = q; q += ns;
    s.slot_col = q; q += ns;
    s.keep = q; q += ns;
    s.hist = q; q += (size_t)hist_rows * kcap;
    s.hbin = q; q += 256;
    s.misc = q; q += 16;
    *scan_out = q;
    return s;
}

// exclusive block scan of one int per thread; scan_sh: 64 ints
__device__ __forceinline__ int block_excl_scan_int(int v, int *scan_sh, int *total)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    int inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    __syncthreads();
    if (lane == 31) scan_sh[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const int w = lane < LP_NT / 32 ? scan_sh[lane] : 0;
        int winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < LP_NT / 32) scan_sh[lane] = winc - w;
        if (lane == 31) scan_sh[32] = winc;
    }
    __syncthreads();
    const int r = scan_sh[wid] + inc - v;
    *total = scan_sh[32];
    __syncthreads();
    return r;
}

// Exact top-kk of the whole sacrifice vector bd[0..p) (global memory, L2-resident), for the iterations whose candidate
// list is unusable: MSB-first radix select on the fp64 bit patterns (values are >= 0), then the kk winners -- every key
// above the boundary bin plus the lowest-index keys of the bin -- go to (cv, ci) in any order; rank_select orders them.
// p <= LP_NT * FB_PER: the keys stay in registers between the passes (strided, coalesced), else they are re-read from L2.
constexpr int FB_PER = 12;
__device__ void fallback_select(const double *bd, int p, int kk, OwnSm &s, int *scan_sh)
{
    const int tid = threadIdx.x;
    unsigned long long prefix = 0ull, mask = 0ull;
    int krem = kk, neq = p;
    bool whole_bin = false;
    unsigned long long *pre_sh = reinterpret_cast<unsigned long long *>(s.red);  // red[0] as a 64-bit scratch word
    const bool inreg = p <= LP_NT * FB_PER;
    unsigned long long key[FB_PER];
    if (inreg) {
#pragma unroll
        for (int q = 0; q < FB_PER; q++) {
            const int i = tid + q * LP_NT;
            key[q] = i < p ? (unsigned long long)__double_as_longlong(__ldcg(bd + i)) : 0ull;
        }
    }
    if (kk < p) {
        for (int pass = 7; pass >= 0; pass--) {
            const int shift = pass * 8;
            if (tid < 256) s.hbin[tid] = 0;
            __syncthreads();
            if (inreg) {
#pragma unroll
                for (int q = 0; q < FB_PER; q++)
                    if (tid + q * LP_NT < p && (key[q] & mask) == prefix) atomicAdd(&s.hbin[(int)((key[q] >> shift) & 255ull)], 1);
            } else {
                for (int i = tid; i < p; i += LP_NT) {
                    const unsigned long long u = (unsigned long long)__double_as_longlong(__ldcg(bd + i));
                    if ((u & mask) == prefix) atomicAdd(&s.hbin[(int)((u >> shift) & 255ull)], 1);
                }
            }
            __syncthreads();
            if (tid < 32) {
                int loc[8], tot = 0;
#pragma unroll
                for (int q = 0; q < 8; q++) {
                    loc[q] = s.hbin[tid * 8 + q];
                    tot += loc[q];
                }
                int suf = tot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const int t = __shfl_down_sync(0xffffffffu, suf, o);
                    if (tid + o < 32) suf += t;
                }
                const int above = suf - tot;
                if (above < krem && suf >= krem) {
                    int acc = above;
                    for (int q = 7; q >= 0; q--) {
                        if (acc + loc[q] >= krem) {
                            *pre_sh = prefix | ((unsigned long long)(tid * 8 + q) << shift);
                            s.misc[MI_KREM] = krem - acc;
                            s.misc[MI_NEQ] = loc[q];
                            break;
                        }
                        acc += loc[q];
                    }
                }
            }
            __syncthreads();
            prefix = *pre_sh;
            krem = s.misc[MI_KREM];
            neq = s.misc[MI_NEQ];
            mask |= 255ull << shift;
            __syncthreads();
            if (neq == krem) break;  // every key of the boundary bin is wanted: lower digits cannot change the set
            if ((kk - krem) + neq <= LP_CAP / 2) {
                // the keys above the bin plus the WHOLE bin fit the candidate list: hand them all over, the ranking that
                // follows picks the exact winners (usually after two or three digits instead of eight)
                whole_bin = true;
                break;
            }
        }
    } else {
        krem = p;  // kk == p: everything matches the empty prefix and is taken
        neq = p;
    }
    if (tid == 0) s.misc[MI_CNT] = 0;
    __syncthreads();
    if (whole_bin) krem = neq;
    if (inreg && neq == krem) {
        // the usual case: the boundary bin is wanted as a whole
#pragma unroll
        for (int q = 0; q < FB_PER; q++) {
            const int i = tid + q * LP_NT;
            if (i < p && (key[q] & mask) >= prefix) {
                const int pos = atomicAdd(&s.misc[MI_CNT], 1);
                if (pos < LP_CAP) {
                    s.cv[pos] = __longlong_as_double((long long)key[q]);
                    s.ci[pos] = i;
                }
            }
        }
        __syncthreads();
        return;
    }
    // keys above the boundary bin, and the first krem keys of the bin in index order (contiguous chunk per thread)
    const int per = (p + LP_NT - 1) / LP_NT;
    const int cb = min(p, tid * per), ce = min(p, cb + per);
    int ceq = 0;
    for (int i = cb; i < ce; i++) {
        const unsigned long long u = (unsigned long long)__double_as_longlong(__ldcg(bd + i));
        ceq += ((u & mask) == prefix);
    }
    int tot_eq;
    int eq_before = block_excl_scan_int(ceq, scan_sh, &tot_eq);
    for (int i = cb; i < ce; i++) {
        const double v = __ldcg(bd + i);
        const unsigned long long u = (unsigned long long)__double_as_longlong(v), mu = u & mask;
        bool take = mu > prefix;
        if (mu == prefix) {
            take = eq_before < krem;
            eq_before++;
        }
        if (take) {
            const int pos = atomicAdd(&s.misc[MI_CNT], 1);
            if (pos < LP_CAP) {
                s.cv[pos] = v;
                s.ci[pos] = i;
            }
        }
    }
    __syncthreads();
}

// Rank the `count` <= LP_CAP candidates once (larger value first, lower index first -- a total order; the values are
// non-negative doubles, so their bit patterns order like the values and the comparisons stay off the FP64 pipe) and file
// the best 2 * kcap + 8 of them by rank: every select of this phase (the closing cycle test of a fit, then the first
// iteration of the next path step) reads its winners, its boundary and its next threshold from that table.
constexpr int RANK_DIRECT = 128;  // lists up to this size are ranked by direct comparison alone (P = 4)
__device__ void rank_candidates(OwnSm &s, int count, int rmax)
{
    const int tid = threadIdx.x;
    if (count > RANK_DIRECT && count > rmax) {
        // Only ranks below rmax are read.  Narrow the list to the keys that can hold one: MSB-first radix digits of the bit
        // patterns, from the highest bit in which the keys differ, until the keys above the boundary digit plus that
        // digit's whole bin are at most RANK_DIRECT (or every bit is decided: exact ties).  Every dropped key ranks below
        // every kept one, so the kept keys ranked among themselves get their ranks in the whole list.
        const int lane = tid & 31, wid = tid >> 5;
        const bool have = tid < count;
        const unsigned long long key = have ? (unsigned long long)__double_as_longlong(s.cv[tid]) : 0ull;
        const int idx = have ? s.ci[tid] : 0;
        const unsigned long long dx = have ? key ^ (unsigned long long)__double_as_longlong(s.cv[0]) : 0ull;
        const unsigned ohi = __reduce_or_sync(0xffffffffu, (unsigned)(dx >> 32)), olo = __reduce_or_sync(0xffffffffu, (unsigned)dx);
        if (lane == 0) {
            s.hbin[2 * wid] = (int)ohi;
            s.hbin[2 * wid + 1] = (int)olo;
        }
        if (tid == 0) s.misc[MI_RANKN] = 0;
        __syncthreads();
        unsigned long long dall = 0ull;
        for (int w = 0; w < LP_NT / 32; w++)
            dall |= ((unsigned long long)(unsigned)s.hbin[2 * w] << 32) | (unsigned)s.hbin[2 * w + 1];
        unsigned long long *pre_sh = reinterpret_cast<unsigned long long *>(s.red);
        if (dall != 0ull) {
            int hb = 63 - __clzll((long long)dall), lb = max(hb - 7, 0);
            unsigned long long mask = hb == 63 ? 0ull : ~0ull << (hb + 1);  // the bits above hb are equal in all keys
            unsigned long long prefix;
            if (tid == 0) *pre_sh = (unsigned long long)__double_as_longlong(s.cv[0]) & mask;
            int krem = rmax;
            for (;;) {
                __syncthreads();
                prefix = *pre_sh;
                if (tid < 256) s.hbin[tid] = 0;
                __syncthreads();
                const unsigned long long dmask = (2ull << (hb - lb)) - 1ull;
                if (have && (key & mask) == prefix) atomicAdd(&s.hbin[(int)((key >> lb) & dmask)], 1);
                __syncthreads();
                if (tid < 32) {
                    int loc[8], tot = 0;
#pragma unroll
                    for (int q = 0; q < 8; q++) {
                        loc[q] = s.hbin[tid * 8 + q];
                        tot += loc[q];
                    }
                    int suf = tot;
#pragma unroll
                    for (int o = 1; o < 32; o <<= 1) {
                        const int t = __shfl_down_sync(0xffffffffu, suf, o);
                        if (tid + o < 32) suf += t;
                    }
                    const int above = suf - tot;
                    if (above < krem && suf >= krem) {
                        int acc = above;
                        for (int q = 7; q >= 0; q--) {
                            if (acc + loc[q] >= krem) {
                                *pre_sh = prefix | ((unsigned long long)(tid * 8 + q) << lb);
                                s.misc[MI_KREM] = krem - acc;
                                s.misc[MI_NEQ] = loc[q];
                                break;
                            }
                            acc += loc[q];
                        }
                    }
                }
                __syncthreads();
                prefix = *pre_sh;
                krem = s.misc[MI_KREM];
                mask |= dmask << lb;
                if ((rmax - krem) + s.misc[MI_NEQ] <= RANK_DIRECT || lb == 0) break;
                hb = lb - 1;
                lb = max(hb - 7, 0);
            }
            if (have && (key & mask) >= prefix) {
                const int pos = atomicAdd(&s.misc[MI_RANKN], 1);
                s.cv[pos] = __longlong_as_double((long long)key);
                s.ci[pos] = idx;
            }
            __syncthreads();
            count = s.misc[MI_RANKN];
        }
    }
    // P threads per candidate split the comparison loop (P = 4 while 4 * count fits the CTA): the loop is a chain of
    // shared-memory loads and integer compares that a thread cannot overlap with anything, so its length is the cost
    const int P = count * 4 <= LP_NT ? 4 : (count * 2 <= LP_NT ? 2 : 1);
    const int t = tid / P, h = tid - t * P;
    int r = 0;
    unsigned long long v = 0ull;
    int id = 0;
    if (t < count) {
        v = (unsigned long long)__double_as_longlong(s.cv[t]);
        id = s.ci[t];
        for (int u = h; u < count; u += P) {
            const unsigned long long vu = (unsigned long long)__double_as_longlong(s.cv[u]);
            const int iu = s.ci[u];
            r += (vu > v) || (vu == v && iu < id);
        }
    }
    // the P partial counts of a candidate sit in adjacent lanes of one warp (P divides 32)
    if (P >= 2) r += __shfl_xor_sync(0xffffffffu, r, 1);
    if (P >= 4) r += __shfl_xor_sync(0xffffffffu, r, 2);
    if (t < count && h == 0 && r < rmax) {
        s.seli[r] = id;
        s.selv[r] = s.cv[t];
    }
    __syncthreads();
}
// The k best of the ranked candidates in ascending index order -> Anew.  MI_TIE <- the k-th and (k+1)-th values are equal
// (a boundary tie: utilities.cpp:179-188 leaves its resolution to std::nth_element).  *vdeep <- value of rank min(count, deep).
__device__ void pick_topk(OwnSm &s, int count, int k, int deep, double *vdeep)
{
    const int tid = threadIdx.x;
    if (tid < k) {
        const int id = s.seli[tid];
        int pos = 0;
        for (int u = 0; u < k; u++) pos += (s.seli[u] < id);
        s.Anew[pos] = id;
    }
    if (tid == 0) s.misc[MI_TIE] = (count > k && s.selv[k] == s.selv[k - 1]) ? 1 : 0;
    *vdeep = s.selv[min(count, deep) - 1];
    __syncthreads();
}

// XA[slot][i] = X[i][slot_col[slot]] for the nnew slots of newlist, all n rows; up to 8 loads in flight per thread
__device__ void gather_new(const Dev &d, OwnSm &s, int nnew, int npad)
{
    const int n = d.n;
    if (nnew == 0) return;
    for (int q0 = 0; q0 < nnew; q0 += 4) {
        for (int i0 = threadIdx.x; i0 < n; i0 += 2 * LP_NT) {
            double v[4][2];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (q0 + u < nnew) {
                    const double *col = d.X + s.slot_col[s.newlist[q0 + u]];
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        const int i = i0 + r * LP_NT;
                        if (i < n) v[u][r] = ldg_stream(col + (size_t)i * d.ldx);
                    }
                }
            }
#pragma unroll
            for (int u = 0; u < 4; u++) {
                if (q0 + u < nnew) {
                    double *dst = s.XA + (size_t)s.newlist[q0 + u] * npad;
#pragma unroll
                    for (int r = 0; r < 2; r++) {
                        const int i = i0 + r * LP_NT;
                        if (i < n) dst[i] = v[u][r];
                    }
                }
            }
        }
    }
    __syncthreads();
}

// sum_i a_i * b_i * w_i, lanes stride the rows, four running sums per lane, fixed combination order
__device__ __forceinline__ double warp_dot3(const double *a, const double *b, const double *w, int n)
{
    const int lane = threadIdx.x & 31;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    int i = lane;
    for (; i + 96 < n; i += 128) {
#pragma unroll
        for (int u = 0; u < 4; u++) acc[u] = fma(a[i + 32 * u] * w[i + 32 * u], b[i + 32 * u], acc[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; u++)
        if (i + 32 * u < n) acc[u] = fma(a[i + 32 * u] * w[i + 32 * u], b[i + 32 * u], acc[u]);
    return warp_sum((acc[0] + acc[1]) + (acc[2] + acc[3]));
}
__device__ __forceinline__ double warp_dot2(const double *a, const double *b, int n)
{
    const int lane = threadIdx.x & 31;
    double acc[4] = {0.0, 0.0, 0.0, 0.0};
    int i = lane;
    for (; i + 96 < n; i += 128) {
#pragma unroll
        for (int u = 0; u < 4; u++) acc[u] = fma(a[i + 32 * u], b[i + 32 * u], acc[u]);
    }
#pragma unroll
    for (int u = 0; u < 4; u++)
        if (i + 32 * u < n) acc[u] = fma(a[i + 32 * u], b[i + 32 * u], acc[u]);
    return warp_sum((acc[0] + acc[1]) + (acc[2] + acc[3]));
}

// Gram rows / columns and X^T y entries of the freshly loaded slots against every occupied slot
__device__ void gram_new(const Dev &d, OwnSm &s, int nnew, int ns, int npad)
{
    const int wid = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int items = nnew * (ns + 1);
    for (int item = wid; item < items; item += LP_NT / 32) {
        const int q = item / (ns + 1), o = item - q * (ns + 1);
        const int sn = s.newlist[q];
        if (o == ns) {
            const double v = warp_dot2(s.XA + (size_t)sn * npad, s.my, d.n);
            if (lane == 0) s.bc[sn] = v;
        } else if (s.slot_col[o] >= 0) {
            const int lo = min(sn, o), hi = max(sn, o);
            const double v = warp_dot3(s.XA + (size_t)lo * npad, s.XA + (size_t)hi * npad, s.m, d.n);
            if (lane == 0) {
                s.Gc[(size_t)sn * ns + o] = v;
                s.Gc[(size_t)o * ns + sn] = v;
            }
        }
    }
    __syncthreads();
}

// Bordered Cholesky solve, incremental.  S (shared memory, row-major, leading dimension ldS) keeps the factor of the
// previous fit: rows 0..q-1 (columns in order of arrival; a PDAS iteration typically appends or exchanges the youngest
// columns) are still valid, dg[j] = 1 / L_jj.  Rows q..k-1 hold fresh Gram rows (lower triangle) and row k the right-hand
// side X_A^T y; on return rows q..k hold L (row k: L^{-1} rhs) and out[0..k) the solution of the normal equations.
// (The reference solves with colPivHouseholderQr, Algorithm.h:1134; on these SPD systems the solutions agree to ~1e-13.)
//
// All variants are compact rolled loops: a fully unrolled register version (one lane per row) was tried and lost -- 40 KB
// of straight-line code executed once per fit by one warp is bound by instruction fetch, not by its dependency chain.
constexpr int CHOL_NR = 4;  // new rows (incl. the right-hand side) the append variant carries in registers

// k <= 32 and k - q + 1 == NR <= CHOL_NR.  Lane c owns COLUMN c of the NR new rows (the last one is the right-hand side).
// Per column j: the entries of the new rows at column j travel by shuffle, are scaled by 1 / L_jj (stored for an old
// column, one rsqrt for a new one) and eliminated from the lanes to the right -- L_cj of an old row c comes from shared
// memory, of a new row from the scaled values.  One warp runs this alone, so what counts is the number of dependent
// instructions per column: NR is a template parameter (no run-time row selects), the old and the new columns have their
// own loops, all addresses are hoisted.
template <int NR>
__device__ __forceinline__ void chol_append_warp(double *S, int ldS, double *dg, int k, int q)
{
    const int lane = threadIdx.x & 31;
    double row[NR];
#pragma unroll
    for (int r = 0; r < NR; r++) row[r] = (lane < k && lane <= q + r) ? S[(q + r) * ldS + lane] : 0.0;
    // ---- old columns: every new row lies below them
    const double *Lc = S + lane * ldS;  // row `lane` of the old factor (lanes < q)
    const bool old_lane = lane < q;
    const int rl = lane - q;            // lanes >= q: the new row that sits at this column
    for (int j = 0; j < q; j++) {
        const double inv = dg[j];
        double l[NR];
#pragma unroll
        for (int r = 0; r < NR; r++) l[r] = __shfl_sync(0xffffffffu, row[r], j) * inv;
        double lcj = old_lane ? Lc[j] : 0.0;
#pragma unroll
        for (int r = 0; r < NR - 1; r++)
            if (rl == r) lcj = l[r];
        if (lane == j) {
#pragma unroll
            for (int r = 0; r < NR; r++) row[r] = l[r];
        } else if (lane > j) {
#pragma unroll
            for (int r = 0; r < NR; r++) row[r] = fma(-l[r], lcj, row[r]);
        }
    }
    // ---- new columns j = q + rj: pivot = diagonal entry of new row rj
#pragma unroll
    for (int rj = 0; rj < NR - 1; rj++) {
        const int j = q + rj;
        double l[NR];
#pragma unroll
        for (int r = 0; r < NR; r++) l[r] = __shfl_sync(0xffffffffu, row[r], j);
        const double inv = rsqrt(l[rj]);
        if (lane == 0) dg[j] = inv;
#pragma unroll
        for (int r = 0; r < NR; r++) l[r] = r < rj ? 0.0 : l[r] * inv;  // rows above the diagonal are not part of L
        double lcj = 0.0;
#pragma unroll
        for (int r = 0; r < NR - 1; r++)
            if (rl == r) lcj = l[r];
        if (lane == j) {
#pragma unroll
            for (int r = 0; r < NR; r++) row[r] = l[r];
        } else if (lane > j) {
#pragma unroll
            for (int r = 0; r < NR; r++) row[r] = fma(-l[r], lcj, row[r]);
        }
    }
#pragma unroll
    for (int r = 0; r < NR; r++)
        if (lane < k && lane <= q + r) S[(q + r) * ldS + lane] = row[r];
    __syncwarp();
}

// k + 1 <= 32 rows: one warp, lane t owns ROW t (in shared memory), every row from q on is factored
__device__ __forceinline__ void chol_rows_warp(double *S, int ldS, double *dg, int k, int q)
{
    const int lane = threadIdx.x & 31;
    const bool mine = lane >= q && lane <= k;
    for (int j = 0; j < k; j++) {
        double inv;
        if (j < q) {
            inv = dg[j];
        } else {
            inv = rsqrt(S[j * ldS + j]);
            if (lane == 0) dg[j] = inv;
        }
        double lij = 0.0;
        if (mine && lane >= j) {
            lij = S[lane * ldS + j] * inv;
            S[lane * ldS + j] = lij;
        }
        __syncwarp();
        if (mine && lane > j) {
            const int cend = min(lane, k - 1);
            for (int c = j + 1; c <= cend; c++) S[lane * ldS + c] = fma(-lij, S[c * ldS + j], S[lane * ldS + c]);
        }
        __syncwarp();
    }
}

// L^T x = z (z = row k of S), lane c owns x_c; k <= 32
__device__ __forceinline__ void chol_backsub_warp(const double *S, int ldS, const double *dg, double *out, int k)
{
    const int lane = threadIdx.x & 31;
    double z = lane < k ? S[k * ldS + lane] : 0.0;
    const double *Lj = S + (k - 1) * ldS + lane;  // L_jc for j = k-1, c = lane; one row up per step
    for (int j = k - 1; j >= 0; j--, Lj -= ldS) {
        const double xj = __shfl_sync(0xffffffffu, z, j) * dg[j];
        const double ljc = lane < j ? *Lj : 0.0;
        z = lane == j ? xj : fma(-ljc, xj, z);
    }
    if (lane < k) out[lane] = z;
}

// chol[0..3] (shared memory, owner 0 only): factor ticks, back-substitution ticks, warp solves, their summed k
__device__ __forceinline__ void chol_solve(OwnSm &s, int k, int q, unsigned long long *chol)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ldS = s.ldS;
    double *S = s.S;
    if (k <= 31) {
        if (wid == 0) {
            const long long t0 = clock64();
            const int nr = k - q + 1;
            if (nr == 2) chol_append_warp<2>(S, ldS, s.dg, k, q);
            else if (nr == 3) chol_append_warp<3>(S, ldS, s.dg, k, q);
            else if (nr == 4) chol_append_warp<4>(S, ldS, s.dg, k, q);
            else chol_rows_warp(S, ldS, s.dg, k, q);
            const long long t1 = clock64();
            chol_backsub_warp(S, ldS, s.dg, s.bage, k);
            const long long t2 = clock64();
            if (tid == 0 && blockIdx.x == 0) {
                chol[0] += (unsigned long long)(t1 - t0);
                chol[1] += (unsigned long long)(t2 - t1);
                chol[2] += 1ull;
                chol[3] += (unsigned long long)k;
            }
        }
        __syncthreads();
        return;
    }
    // q == 0 here (the caller assembles every row for systems this large)
    for (int j = 0; j < k; j++) {
        __syncthreads();
        const double inv = rsqrt(S[j * ldS + j]);
        __syncthreads();
        if (tid == 0) {
            s.dg[j] = inv;
            S[j * ldS + j] *= inv;
        }
        for (int i = j + 1 + tid; i <= k; i += LP_NT) S[i * ldS + j] *= inv;
        __syncthreads();
        for (int i = j + 1 + wid; i <= k; i += LP_NT / 32) {
            const double lij = S[i * ldS + j];
            const int cend = min(i, k - 1);
            for (int c = j + 1 + lane; c <= cend; c += 32) S[i * ldS + c] -= lij * S[c * ldS + j];
        }
    }
    __syncthreads();
    if (wid == 0) {
        for (int c = lane; c < k; c += 32) s.bage[c] = S[k * ldS + c];
        __syncwarp();
        for (int j = k - 1; j >= 0; j--) {
            const double xj = s.bage[j] * s.dg[j];
            __syncwarp();
            if (lane == 0) s.bage[j] = xj;
            for (int c = lane; c < j; c += 32) s.bage[c] -= S[j * ldS + c] * xj;
            __syncwarp();
        }
    }
    __syncthreads();
}

// Residual of the next sweep, G[i][c] = (y_i - x_i,A beta_A) / n_train on the chain's train rows, 0 elsewhere
// (Algorithm.h:1109), and on request the Lm losses of Metric.h:145-148 (all rows, / n) and :190 (held-out rows, / 2 n_t).
__device__ void residual(const Dev &d, OwnSm &s, double *Rcol, int fh, int ks, int nt, int npad, bool want_loss,
                         double *loss_all, double *loss_test)
{
    // Rcol: this chain's column of its group's residual matrix [npad][fh] (what the sweepers stage)
    const int n = d.n;
    double sa = 0.0, st = 0.0;
    for (int i0 = threadIdx.x; i0 < n; i0 += 2 * LP_NT) {
        const int i1 = i0 + LP_NT;
        const bool two = i1 < n;
        double eta0 = 0.0, eta1 = 0.0;
        for (int a = 0; a < ks; a++) {
            const double *col = s.XA + (size_t)s.slotA[a] * npad;
            const double b = s.beta[a];
            eta0 = fma(col[i0], b, eta0);
            if (two) eta1 = fma(col[i1], b, eta1);
        }
        {
            const double e = s.y[i0] - eta0;
            const bool train = s.m[i0] != 0.0;
            const double gv = train ? e / (double)nt : 0.0;
            __stcg(Rcol + (size_t)i0 * fh, gv);
            sa += e * e;
            if (!train) st += e * e;
        }
        if (two) {
            const double e = s.y[i1] - eta1;
            const bool train = s.m[i1] != 0.0;
            const double gv = train ? e / (double)nt : 0.0;
            __stcg(Rcol + (size_t)i1 * fh, gv);
            sa += e * e;
            if (!train) st += e * e;
        }
    }
    if (want_loss) {
        // both sums through one deterministic block reduction
        const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
        sa = warp_sum(sa);
        st = warp_sum(st);
        __syncthreads();
        if (lane == 0) {
            s.red[2 + wid] = sa;
            s.red[20 + wid] = st;
        }
        __syncthreads();
        double ta = 0.0, tt = 0.0;
        for (int w = 0; w < LP_NT / 32; w++) {
            ta += s.red[2 + w];
            tt += s.red[20 + w];
        }
        *loss_all = ta / (double)n;
        *loss_test = n > nt ? tt / (double)(2 * (n - nt)) : 0.0;
    }
    __syncthreads();
}

template <int FT>
__device__ void owner_main(const Dev &d, const LpDesc &L, unsigned char *raw)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ci = blockIdx.x, c = L.chain[ci];
    const int n = d.n, npad = (n + 1) & ~1, kcap = d.kcap, ns = L.ns, p = d.p;
    double *pre_sh;
    int *scan_sh;
    OwnSm s = carve_owner(raw, npad, kcap, ns, L.hist_rows, &pre_sh, &scan_sh);
    (void)pre_sh;
    const int nt = d.ntrain[c];
    const int g = L.ogroup[ci], og = 1 - g;
    double *Rcol = L.Rg[g] + L.oslot[ci];
    const int *rows = d.rows + (size_t)c * n;
    double *bD = d.betaD + (size_t)c * d.pstride;
    Timer<13, LpTick<FT>> tm;
    tm.start(tid == 0 && ci == 0);
    LpTick<FT> own_busy = 0, own_max = 0, own_fb = 0, own_fits = 0;  // thread 0: flushed at exit
    // solver timers of owner 0 (chol_solve) in the spare tail of s.red: an array in registers would live on the stack
    unsigned long long *chol = reinterpret_cast<unsigned long long *>(s.red + 36);

    // ---- phase O(0): Algorithm::fit prologue from the chain's stored state (Algorithm.h:141-148)
    for (int i = tid; i < npad; i += LP_NT) {
        s.m[i] = 0.0;
        s.y[i] = i < n ? L.y[i] : 0.0;
    }
    for (int q = tid; q < ns; q += LP_NT) {
        s.slot_col[q] = -1;
        s.pos[q] = -1;
    }
    if (tid < 4) chol[tid] = 0ull;
    if (tid == 0) s.misc[MI_B2ADD] = 1;  // what this owner's arrivals add to B2 (LP_TERM_FLAG too after it sets the word)
    __syncthreads();
    for (int r = tid; r < nt; r += LP_NT) s.m[rows[r]] = 1.0;
    __syncthreads();
    for (int i = tid; i < npad; i += LP_NT) s.my[i] = s.m[i] * s.y[i];
    int ks = d.ks[c];
    if (!d.warm) {  // cold start: beta_init = 0
        for (int a = tid; a < ks; a += LP_NT) __stcg(bD + d.A[(size_t)c * kcap + a], 0.0);
        ks = 0;
    }
    for (int a = tid; a < ks; a += LP_NT) {
        s.A[a] = d.A[(size_t)c * kcap + a];
        s.beta[a] = d.bA[(size_t)c * kcap + a];
        s.slotA[a] = a;
        s.slot_col[a] = s.A[a];
        s.newlist[a] = a;
    }
    __syncthreads();
    gather_new(d, s, ks, npad);
    gram_new(d, s, ks, ns, npad);
    int step = 0, T = L.T[0], l = 0, tie_acc = 0;
    int kfac = 0;  // columns of the Cholesky factor in s.S that are valid (in the order s.ord)
    double lam = L.lam[0], lam_fact = L.lam[0];
    for (int a = tid; a < T; a += LP_NT) s.hist[a] = 0;  // A_list.col(0) = 0 (Algorithm.h:143)
    double la = 0.0, lt = 0.0;
    residual(d, s, Rcol, L.fh, ks, nt, npad, false, &la, &lt);
    double tau = L.tau[c];
    if (tid == 0) {
        __stcg(L.pub + 2 * c, tau);
        __stcg(L.pub + 2 * c + 1, lam);
    }
    bool complete = false;
    tm.mark(0);
    cta_arrive(L.sync + LP_SYNC_B2 + g);

    // Owner phase O_g(it) has index ng * it + g (see sweeper_main).  Before reading the termination word the owner has
    // seen every owner phase up to its decision index complete (its own group's phase it - 1 and the other group's phase
    // just before it), so the word can no longer change below that index: every CTA leaves at the same point.
    for (unsigned it = 1;; it++) {
        // (B1 only after the termination word: once the last chain has finished, the sweepers leave and that counter
        // never moves again)
        if (cta_wait_term(L.sync, LP_SYNC_B2 + g, (unsigned)L.gcount[g] * it, L.ng == 2 ? LP_SYNC_B2 + og : -1,
                          (unsigned)L.gcount[og] * (g == 0 ? it - 1u : it), (unsigned)L.ng * (it - 1u) + (unsigned)g,
                          LP_SYNC_B1 + g, (unsigned)L.nsweep * it, &s.misc[MI_FLAG]) != LP_WAIT_GO)
            break;
        tm.mark(1);
        const long long t_phase = clock64();
        if (L.trace && tid == 0 && it < LP_TRACE) L.trace[((size_t)ci * LP_TRACE + it) * 2] = lp_globaltimer();
        if (!complete) {
            // ---- the candidates the sweepers published for this chain; the count and the (possibly stale) slots are
            // fetched together: one L2 round trip
            {
                int4 raw4 = make_int4(0, 0, 0, 0);
                if (tid < LP_CAP) raw4 = __ldcg(reinterpret_cast<const int4 *>(L.cand + (size_t)c * LP_CAP + tid));
                if (tid == 0) s.misc[MI_COUNT] = __ldcg(L.ncand + c);
                const LpCand cnd = *reinterpret_cast<const LpCand *>(&raw4);
                if (tid < LP_CAP) {
                    s.cv[tid] = cnd.v;
                    s.ci[tid] = cnd.idx;
                }
            }
            __syncthreads();
            int count = s.misc[MI_COUNT];
            tm.mark(9);
            // One sweep can serve two fits: when a fit ends because its active set repeats the previous one, beta has not
            // moved since the sweep, and the first get_A of the NEXT path step (warm start, same ridge level) would
            // recompute exactly this sacrifice vector -- the owner selects again from the same candidates at once.
            bool again = true, ranked = false;
            const int rmax = 2 * kcap + 8;
            while (again) {
                again = false;
                const int k = T;
                // ---- exact top-k (max_k, utilities.cpp:179-188)
                const int deep = min(p, 2 * k + 4);  // how far down the order statistics the next threshold looks
                if (count < k || count > LP_CAP) {
                    __syncthreads();
                    const long long t_fb = clock64();
                    fallback_select(d.bd + (size_t)c * d.pstride, p, deep, s, scan_sh);
                    count = min(s.misc[MI_CNT], LP_CAP);
                    ranked = false;
                    if (tid == 0) {
                        atomicAdd(L.sync + LP_SYNC_FALLBACKS, 1u);
                        (void)t_fb;
                    }
                }
                if (!ranked) {
                    rank_candidates(s, count, rmax);
                    ranked = true;
                }
                double vdeep = 0.0;
                pick_topk(s, count, k, deep, &vdeep);
                // candidate threshold of the next iteration: well below the `deep`-th largest sacrifice, so that the next
                // level (k + 1) and moderately changed sacrifices still find their k winners in the list
                tau = 0.7 * vdeep;
                tm.mark(2);
                // ---- same active set as the previous iteration of this fit: the fit would reproduce beta bit for bit
                // and the cycle test (Algorithm.h:164-170) ends the fit -- nothing to recompute
                int same = (l >= 1 && ks == k) ? 1 : 0;
                if (same)
                    for (int a2 = tid; a2 < k; a2 += LP_NT) same &= (s.A[a2] == s.Anew[a2]);
                same = __syncthreads_and(same);
                bool seen = same != 0;
                if (!same) {
                    // ---- which of the selected columns are already resident
                    for (int q2 = tid; q2 < ns; q2 += LP_NT) s.keep[q2] = 0;
                    __syncthreads();
                    if (tid < k) {
                        const int j = s.Anew[tid];
                        int sl = -1;
                        for (int q2 = 0; q2 < ns; q2++)
                            if (s.slot_col[q2] == j) sl = q2;
                        s.slotNew[tid] = sl;
                        if (sl >= 0) s.keep[sl] = 1;
                    }
                    __syncthreads();
                    // ---- one warp, ballots instead of serial loops: (a) how much of the Cholesky factor survives -- its
                    // columns are kept in order of arrival, the longest prefix whose columns are all still selected stays
                    // valid; (b) the new column order: that prefix, the other survivors, the newcomers; (c) the newcomers
                    // take free slots, empty ones first, then slots of columns that are not selected now
                    if (wid == 0) {
                        const unsigned lt = (1u << lane) - 1u;
                        int q = kfac;
                        for (int t0 = 0; t0 < kfac; t0 += 32) {
                            const int t = t0 + lane;
                            const bool okk = t < kfac && s.keep[s.ord[t]] != 0;
                            const unsigned mk = __ballot_sync(0xffffffffu, okk || t >= kfac);
                            if (mk != 0xffffffffu) {
                                q = t0 + __ffs(~mk) - 1;
                                break;
                            }
                        }
                        if (lam != lam_fact || k > 31) q = 0;  // another ridge level / a system the CTA refactors as a whole
                        for (int t = lane; t < q; t += 32) s.ordNew[t] = s.ord[t];
                        int n_out = q;
                        for (int t0 = q; t0 < kfac; t0 += 32) {
                            const int t = t0 + lane;
                            const bool okk = t < kfac && s.keep[s.ord[t]] != 0;
                            const unsigned mk = __ballot_sync(0xffffffffu, okk);
                            if (okk) s.ordNew[n_out + __popc(mk & lt)] = s.ord[t];
                            n_out += __popc(mk);
                        }
                        // selected columns that are resident but not part of the factor (loaded by the prologue, or
                        // dropped by an earlier fit and still cached in their slot)
                        for (int a0 = 0; a0 < k; a0 += 32) {
                            const int a2 = a0 + lane;
                            const int sl = a2 < k ? s.slotNew[a2] : -1;
                            const bool okk = sl >= 0 && (s.pos[sl] < 0 || s.pos[sl] >= kfac);
                            const unsigned mk = __ballot_sync(0xffffffffu, okk);
                            if (okk) s.ordNew[n_out + __popc(mk & lt)] = sl;
                            n_out += __popc(mk);
                        }
                        int nfree = 0;
                        for (int pass = 0; pass < 2; pass++)
                            for (int q0 = 0; q0 < ns; q0 += 32) {
                                const int sl = q0 + lane;
                                const bool okk = sl < ns && s.keep[sl] == 0 && ((s.slot_col[sl] < 0) == (pass == 0));
                                const unsigned mk = __ballot_sync(0xffffffffu, okk);
                                if (okk) s.freel[nfree + __popc(mk & lt)] = sl;
                                nfree += __popc(mk);
                            }
                        __syncwarp();
                        int nnew = 0;
                        for (int a0 = 0; a0 < k; a0 += 32) {
                            const int a2 = a0 + lane;
                            const bool need = a2 < k && s.slotNew[a2] < 0;
                            const unsigned mk = __ballot_sync(0xffffffffu, need);
                            if (need) {
                                const int r2 = nnew + __popc(mk & lt);
                                const int sl = s.freel[r2];
                                s.slotNew[a2] = sl;
                                s.slot_col[sl] = s.Anew[a2];
                                s.newlist[r2] = sl;
                                s.ordNew[n_out + r2] = sl;
                            }
                            nnew += __popc(mk);
                        }
                        __syncwarp();
                        for (int sl = lane; sl < ns; sl += 32) s.pos[sl] = -1;
                        __syncwarp();
                        for (int t = lane; t < k; t += 32) {
                            const int sl = s.ordNew[t];
                            s.ord[t] = sl;
                            s.pos[sl] = t;
                        }
                        if (lane == 0) {
                            s.misc[MI_NNEW] = nnew;
                            s.misc[MI_Q] = q;
                        }
                    }
                    __syncthreads();
                    const int nnew = s.misc[MI_NNEW], q = s.misc[MI_Q];
                    tm.mark(10);
                    gather_new(d, s, nnew, npad);
                    tm.mark(3);
                    gram_new(d, s, nnew, ns, npad);
                    tm.mark(4);
                    // ---- rows q..k-1 of X_A^T X_A + lambda I (Algorithm.h:1134) in factor order, X_A^T y as row k
                    for (int e = tid; e < (k + 1 - q) * k; e += LP_NT) {
                        const int t = q + e / k, u = e - (t - q) * k;
                        if (t < k) {
                            if (u <= t) s.S[t * s.ldS + u] = s.Gc[(size_t)s.ord[t] * ns + s.ord[u]] + (t == u ? lam : 0.0);
                        } else {
                            s.S[k * s.ldS + u] = s.bc[s.ord[u]];
                        }
                    }
                    __syncthreads();
                    tm.mark(8);
                    own_fb += (LpTick<FT>)(k - q) * 1965u;  // DEBUG: new rows per fit (x1965 so the us conversion shows the count)
                    chol_solve(s, k, q, chol);
                    // A pivot at or below 1e-13 of its column's own squared norm (or a NaN) is a numerically dependent
                    // active column (e.g. an exact duplicate): this kernel's plain Cholesky has no answer for it.  Flag
                    // the launch; the host repeats the call on the multi-kernel path, whose solver truncates the way the
                    // reference's colPivHouseholderQr does (chain_fit.cu: ldlt_pivoted_small).
                    for (int t2 = tid; t2 < k; t2 += LP_NT) {
                        const double gjj = s.Gc[(size_t)s.ord[t2] * ns + s.ord[t2]] + lam, dv = s.dg[t2];
                        if (!(dv * dv * gjj * 1e-13 < 1.0)) atomicAdd(L.sync + LP_SYNC_RANKDEF, 1u);
                    }
                    kfac = k;
                    lam_fact = lam;
                    for (int a2 = tid; a2 < k; a2 += LP_NT) s.beta[a2] = s.bage[s.pos[s.slotNew[a2]]];  // back to ascending column order
                    __syncthreads();
                    tm.mark(5);
                    // ---- scatter (Algorithm.h:159-163), cycle test against A_list[0..l] (Algorithm.h:164-170)
                    for (int a2 = tid; a2 < ks; a2 += LP_NT) __stcg(bD + s.A[a2], 0.0);
                    if (tid == 0) s.misc[MI_SEEN] = 0;
                    __syncthreads();
                    for (int a2 = tid; a2 < k; a2 += LP_NT) {
                        s.A[a2] = s.Anew[a2];
                        s.slotA[a2] = s.slotNew[a2];
                        __stcg(bD + s.Anew[a2], s.beta[a2]);
                    }
                    ks = k;
                    for (int ll = wid; ll <= l; ll += LP_NT / 32) {
                        const int *hp = s.hist + (size_t)ll * kcap;
                        int eq = 1;
                        for (int a2 = lane; a2 < k; a2 += 32) eq &= (hp[a2] == s.Anew[a2]);
                        if (__all_sync(0xffffffffu, eq) && lane == 0) s.misc[MI_SEEN] = 1;
                    }
                    __syncthreads();
                    seen = s.misc[MI_SEEN] != 0;
                    tm.mark(11);
                    // the losses ride along with every residual: a fit that ends on a repeated set needs them without a pass
                    residual(d, s, Rcol, L.fh, ks, nt, npad, true, &la, &lt);
                    tm.mark(6);
                    own_fits += 1;
                }
                l += 1;
                tie_acc += s.misc[MI_TIE];
                if (l < L.hist_rows)
                    for (int a2 = tid; a2 < k; a2 += LP_NT) s.hist[(size_t)l * kcap + a2] = s.Anew[a2];
                const bool finished = seen || l >= d.max_iter;
                if (finished) {
                    int *ri = L.res_i + ((size_t)step * L.nch + ci) * (2 + kcap);
                    double *rd = L.res_d + ((size_t)step * L.nch + ci) * (2 + kcap);
                    const int l_out = seen ? l : d.max_iter + 1;
                    if (tid == 0) {
                        ri[0] = l_out;
                        ri[1] = tie_acc;
                        rd[0] = la;
                        rd[1] = lt;
                    }
                    for (int a2 = tid; a2 < k; a2 += LP_NT) {
                        ri[2 + a2] = s.A[a2];
                        rd[2 + a2] = s.beta[a2];
                    }
                    step += 1;
                    if (step == L.nsteps) {
                        complete = true;
                        // hand the chain back to the engine's tables (chain_state / the multi-kernel path read them)
                        for (int a2 = tid; a2 < k; a2 += LP_NT) {
                            d.A[(size_t)c * kcap + a2] = s.A[a2];
                            d.bA[(size_t)c * kcap + a2] = s.beta[a2];
                        }
                        // the chain's last residual into d.G, where the multi-kernel helpers (debug_sacrifice,
                        // time_dual_sweep) read a chain's current state after the launch
                        for (int i = tid; i < n; i += LP_NT) d.G[(size_t)i * d.FS + c] = __ldcg(Rcol + (size_t)i * L.fh);
                        if (tid == 0) {
                            d.ks[c] = ks;
                            d.l[c] = l_out;
                            d.done[c] = 1;
                            d.coef0[c] = 0.0;
                            d.tie_acc[c] = tie_acc;
                            L.tau[c] = tau;
                            const unsigned old = atomicAdd(L.sync + LP_SYNC_NCOMPLETE, 1u);
                            if (old + 1u == (unsigned)L.nch) {
                                atomicExch(L.sync + LP_SYNC_TERM, (unsigned)L.ng * it + (unsigned)g + 1u);
                                s.misc[MI_B2ADD] = (int)(1u + LP_TERM_FLAG);
                                atomicExch(L.sync + LP_SYNC_ITERS, (unsigned)L.ng * (it - 1u) + (unsigned)g + 1u);  // sweeps that fed a fit
                            }
                        }
                    } else {
                        const double lam_prev = lam;
                        T = L.T[step];
                        lam = L.lam[step];
                        l = 0;
                        tie_acc = 0;
                        __syncthreads();
                        for (int a2 = tid; a2 < T; a2 += LP_NT) s.hist[a2] = 0;
                        if (!d.warm) {
                            for (int a2 = tid; a2 < ks; a2 += LP_NT) __stcg(bD + s.A[a2], 0.0);
                            ks = 0;  // (the factor stays: its leading columns are reused if the next fit selects them again)
                            residual(d, s, Rcol, L.fh, 0, nt, npad, true, &la, &lt);
                        } else if (same && lam == lam_prev) {
                            again = true;  // the sweep this phase consumed was computed from exactly the state the next step starts in
                            if (tid == 0) atomicAdd(L.sync + LP_SYNC_MERGED, 1u);
                        }
                        __syncthreads();
                    }
                }
            }
            tm.mark(12);
            if (tid == 0) {
                __stcg(L.pub + 2 * c, complete ? (double)INFINITY : tau);
                __stcg(L.pub + 2 * c + 1, lam);
                __stcg(L.ncand + c, 0);
            }
            tm.mark(7);
        }
        if (tid == 0) {
            const LpTick<FT> dt = (LpTick<FT>)(clock64() - t_phase);
            own_busy += dt;
            if (dt > own_max) own_max = dt;
            if (L.trace && it < LP_TRACE) L.trace[((size_t)ci * LP_TRACE + it) * 2 + 1] = lp_globaltimer();
        }
        cta_arrive(L.sync + LP_SYNC_B2 + g, (unsigned)s.misc[MI_B2ADD]);
    }
    tm.flush(L.dbg);
    if (tid == 0 && ci == 0) {
        L.dbg[13] += chol[0];
        L.dbg[14] += chol[1];
        L.dbg[15] = chol[3] * 1965ull / (chol[2] ? chol[2] : 1ull);
    }
    if (tid == 0) {
        unsigned long long *od = L.dbg + 32 + 4 * ci;
        od[0] += own_busy;
        if (own_max > od[1]) od[1] = own_max;
        od[2] += own_fb;
        od[3] += own_fits;
    }
}

template <int FT>
__global__ void __launch_bounds__(LP_NT, 1) lm_path_kernel(const Dev d, const LpDesc L)
{
    extern __shared__ __align__(128) unsigned char lp_smem[];
    if ((int)blockIdx.x < L.nch) owner_main<FT>(d, L, lp_smem);
    else sweeper_main<FT>(d, L, lp_smem);
}

bool env_enabled()
{
    static const bool on = [] {
        const char *e = std::getenv("BESS_B200_RESIDENT");
        return !(e && e[0] == '0');
    }();
    return on;
}

}  // namespace

int lm_path_slots(const Dev &d, int max_iter)
{
    const int npad = (d.n + 1) & ~1;
    const size_t budget = 232448 - 2048;
    int ns = d.kcap + 8;
    while (ns > d.kcap && owner_smem_bytes(npad, d.kcap, ns, max_iter + 2) > budget) ns--;
    return ns;
}

int lm_path_groups(int nch) { return nch >= 4 ? 2 : 1; }
int lm_path_fh(int nch, int ng)
{
    const int per = (nch + ng - 1) / ng;
    const int opts[] = {1, 2, 4, 6, 8, 12, 16};
    for (int o : opts)
        if (o >= per) return o;
    return 16;
}

size_t lm_path_smem_bytes(const Dev &d, int max_iter, int sm_count)
{
    (void)sm_count;
    const int npad = (d.n + 1) & ~1;
    const size_t own = owner_smem_bytes(npad, d.kcap, lm_path_slots(d, max_iter), max_iter + 2);
    int fhmax = 1;  // the widest chain group any batch of this problem (at most d.FS chains) can have
    for (int nch = 1; nch <= d.FS; nch++) fhmax = std::max(fhmax, lm_path_fh(nch, lm_path_groups(nch)));
    const size_t swp = sweeper_smem_doubles(npad, fhmax) * 8;
    return ((own > swp ? own : swp) + 127) & ~(size_t)127;
}

bool lm_path_eligible(const Dev &d, int max_iter, int sm_count, std::string *why)
{
    auto no = [&](const char *m) {
        if (why) *why = m;
        return false;
    };
    if (!env_enabled()) return no("disabled by BESS_B200_RESIDENT=0");
    if (d.family != FAM_LM) return no("family is not gaussian");
    if (d.grouped) return no("group selection");
    if (d.sharded) return no("column-sharded mode");
    if (d.ccp) return no("sparse design (swept on its non-zeros)");
    if (d.kcap > LP_KMAX) return no("support larger than 64");
    if (d.kcap > d.p) return no("support larger than p");
    if (sm_count < MAXC + 8) return no("too few SMs");
    const int nsweep = sm_count - MAXC;  // the fewest sweepers any batch of this problem can have
    const int P2 = (d.p + 1) >> 1;
    if ((P2 + nsweep - 1) / nsweep > LP_WPMAX) return no("too many columns per sweeper CTA");
    if (lm_path_smem_bytes(d, max_iter, sm_count) > 232448 - 2048) return no("shared-memory budget");
    if (owner_smem_bytes((d.n + 1) & ~1, d.kcap, d.kcap, max_iter + 2) > 232448 - 2048) return no("shared-memory budget");
    return true;
}

void launch_lm_path(const Dev &d, const LpDesc &desc, int sm_count, int max_iter, cudaStream_t st)
{
    // CTAs run one per SM whatever they request: when the owners need less than the whole budget, ask for enough to keep
    // each sweeper's whole slice on chip (sweeper_main), up to the budget
    const size_t slice = (size_t)d.n * sweeper_pairs(d.p, desc.nsweep) * 2 * sizeof(double);
    const size_t want = std::min(sweeper_smem_doubles((d.n + 1) & ~1, desc.fh) * sizeof(double) + slice, (size_t)(232448 - 2048));
    const size_t smem = std::max(lm_path_smem_bytes(d, max_iter, sm_count), (want + 127) & ~(size_t)127);
    void (*fn)(const Dev, const LpDesc) = nullptr;
    switch (desc.fh) {
        case 1: fn = lm_path_kernel<1>; break;
        case 2: fn = lm_path_kernel<2>; break;
        case 4: fn = lm_path_kernel<4>; break;
        case 6: fn = lm_path_kernel<6>; break;
        case 8: fn = lm_path_kernel<8>; break;
        case 12: fn = lm_path_kernel<12>; break;
        case 16: fn = lm_path_kernel<16>; break;
        default: throw EngineError{"resident path: unsupported chain-slot count"};
    }
    CUDA_CHECK(cudaFuncSetAttribute((const void *)fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    void *args[2] = {(void *)&d, (void *)&desc};
    CUDA_CHECK(cudaLaunchCooperativeKernel((const void *)fn, dim3((unsigned)(desc.nch + desc.nsweep)), dim3(LP_NT), args, smem, st));
}

}  // namespace bess
