// Hand-written sm_100a kernels for the BeSS primal-dual active-set hot path.
//
//   dual_sweep_kernel   d = X^T g, h = (X.X)^T w (+ Cox risk-set suffix term) for every chain of a batch in ONE
//                       pass over X.  X is row-major n x p (the layout pywrap_bess hands over,
//                       /root/reference/src/utilities.cpp:13-25), so a thread owns 1-2 adjacent columns, walks the
//                       rows with coalesced 16-byte loads and needs no cross-lane reduction; the per-row gradient
//                       vectors of all chains are staged into shared memory with 1-D bulk TMA copies
//                       (cp.async.bulk + mbarrier), double buffered.
//                       Replaces the GEMVs + per-column 1x1 sqrt()/ldlt() objects of
//                       Algorithm.h:1097-1129 (Lm), :1206-1263 (Logistic), :1324-1367 (Poisson), :1569-1640 (Cox).
//   finish_kernel       reduces the row-split partials and applies the splicing sacrifice (same citations).
//   topk_slices_kernel  exact top-k by MSB-first radix select on the fp64 bit patterns held in shared memory,
//                       ordered compaction => ascending indices (utilities.cpp:179-199 max_k + slice_assignment).
//   chain_begin/chain_fit  one CTA per chain: gather X_A (utilities.cpp:132-140), active-set fit
//                       (Algorithm.h:1131-1135 / 1148-1204 / 1273-1322 / 1377-1490), cycle test (Algorithm.h:164-170),
//                       and the gradient vectors of the next sweep.
//   loss_kernel         Metric.h train_loss / fold test losses.
#include "kernels.cuh"
#include "device_utils.cuh"

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdio>

namespace bess {

// =====================================================================================================
// mbarrier + 1-D bulk TMA (cp.async.bulk) helpers
// =====================================================================================================
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "LAB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra DONE;\n"
        "bra LAB_WAIT;\n"
        "DONE:\n"
        "}" ::"r"(smem_u32(bar)),
        "r"(parity)
        : "memory");
}

// =====================================================================================================
// dual sweep
// =====================================================================================================
template <int MODE>
struct SweepTraits {
    static constexpr int NV = MODE == MODE_D ? 1 : (MODE == MODE_DH ? 2 : 4);  // staged vectors
    static constexpr int NQ = MODE == MODE_D ? 1 : (MODE == MODE_DH ? 2 : 5);  // partial outputs per column
};

template <int FT, int MODE, int CPT>
__global__ void __launch_bounds__(SWEEP_NT) dual_sweep_kernel(const Dev d)
{
    constexpr int NV = SweepTraits<MODE>::NV;
    constexpr int NQ = SweepTraits<MODE>::NQ;
    constexpr bool REV = (MODE == MODE_COX);  // risk-set suffix sums: walk rows from the last to the first
    constexpr int RC = SWEEP_RC;
    constexpr int U = 8;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *tile = reinterpret_cast<double *>(smem_raw);  // [2][NV][RC][FT]
    __shared__ __align__(8) uint64_t bar[2];
    if (d.gate && *d.gate == 0) return;  // every chain of the batch already stopped (speculative launch)

    const int tid = threadIdx.x;
    const int s = blockIdx.y;
    const int r0 = s * d.rows_per_split;
    const int r1 = min(d.n, r0 + d.rows_per_split);
    const int nrows = r1 - r0;
    const int nchunks = (nrows + RC - 1) / RC;
    const long long j0 = ((long long)blockIdx.x * SWEEP_NT + tid) * CPT;
    const bool active = j0 < d.p;

    double accd[CPT][FT];
    double acch[MODE >= MODE_DH ? CPT : 1][MODE >= MODE_DH ? FT : 1];
    double s1[MODE == MODE_COX ? CPT : 1][MODE == MODE_COX ? FT : 1];
    double accA[MODE == MODE_COX ? CPT : 1][MODE == MODE_COX ? FT : 1];
    double accB[MODE == MODE_COX ? CPT : 1][MODE == MODE_COX ? FT : 1];
#pragma unroll
    for (int c = 0; c < CPT; c++)
#pragma unroll
        for (int f = 0; f < FT; f++) {
            accd[c][f] = 0.0;
            if constexpr (MODE >= MODE_DH) acch[c][f] = 0.0;
            if constexpr (MODE == MODE_COX) { s1[c][f] = 0.0; accA[c][f] = 0.0; accB[c][f] = 0.0; }
        }
    double c2acc = 0.0;

    if (tid == 0) {
        mbar_init(&bar[0], 1);
        mbar_init(&bar[1], 1);
        mbar_fence_init();
    }
    __syncthreads();

    const double *vecs[4] = {d.G, d.W, d.TH, d.C2};
    auto issue = [&](int q, int stage) {
        const int c = REV ? (nchunks - 1 - q) : q;
        const int cr0 = r0 + c * RC;
        const int crows = min(RC, r1 - cr0);
        const uint32_t bytes = (uint32_t)(((crows + 1) & ~1) * FT * 8);  // vectors are padded to an even row count
        mbar_expect_tx(&bar[stage], bytes * NV);
#pragma unroll
        for (int v = 0; v < NV; v++)
            bulk_g2s(tile + (size_t)(stage * NV + v) * RC * FT, vecs[v] + (size_t)cr0 * FT, bytes, &bar[stage]);
    };
    if (tid == 0 && nchunks > 0) {
        issue(0, 0);
        if (nchunks > 1) issue(1, 1);
    }

    for (int q = 0; q < nchunks; q++) {
        const int stage = q & 1;
        mbar_wait(&bar[stage], (q >> 1) & 1);
        const int c = REV ? (nchunks - 1 - q) : q;
        const int cr0 = r0 + c * RC;
        const int crows = min(RC, r1 - cr0);
        const double *tg = tile + (size_t)(stage * NV + 0) * RC * FT;
        const double *tw = tile + (size_t)(stage * NV + (NV > 1 ? 1 : 0)) * RC * FT;
        const double *tt = tile + (size_t)(stage * NV + (NV > 2 ? 2 : 0)) * RC * FT;
        const double *tc = tile + (size_t)(stage * NV + (NV > 3 ? 3 : 0)) * RC * FT;
        if (active) {
            for (int rr = 0; rr < crows; rr += U) {
                double xv[U][CPT];
#pragma unroll
                for (int u = 0; u < U; u++) {
                    const int lr = REV ? (crows - 1 - (rr + u)) : (rr + u);
                    if (rr + u < crows) {
                        const double *xp = d.X + (size_t)(cr0 + lr) * d.ldx + j0;
                        if constexpr (CPT == 2) {
                            const double2 t = __ldg(reinterpret_cast<const double2 *>(xp));
                            xv[u][0] = t.x;
                            xv[u][CPT - 1] = t.y;
                        } else {
                            xv[u][0] = __ldg(xp);
                        }
                    } else {
#pragma unroll
                        for (int cc = 0; cc < CPT; cc++) xv[u][cc] = 0.0;
                    }
                }
#pragma unroll
                for (int u = 0; u < U; u++) {
                    if (rr + u < crows) {
                        const int lr = REV ? (crows - 1 - (rr + u)) : (rr + u);
                        double xx[CPT];
#pragma unroll
                        for (int cc = 0; cc < CPT; cc++) xx[cc] = xv[u][cc] * xv[u][cc];
#pragma unroll
                        for (int f = 0; f < FT; f++) {
                            const double g = tg[lr * FT + f];
#pragma unroll
                            for (int cc = 0; cc < CPT; cc++) accd[cc][f] = fma(xv[u][cc], g, accd[cc][f]);
                            if constexpr (MODE >= MODE_DH) {
                                const double w = tw[lr * FT + f];
#pragma unroll
                                for (int cc = 0; cc < CPT; cc++) acch[cc][f] = fma(xx[cc], w, acch[cc][f]);
                            }
                            if constexpr (MODE == MODE_COX) {
                                const double th = tt[lr * FT + f];
                                const double c2 = tc[lr * FT + f];
#pragma unroll
                                for (int cc = 0; cc < CPT; cc++) {
                                    s1[cc][f] = fma(xv[u][cc], th, s1[cc][f]);
                                    const double t = c2 * s1[cc][f];
                                    accA[cc][f] = fma(t, s1[cc][f], accA[cc][f]);
                                    accB[cc][f] += t;
                                }
                            }
                        }
                    }
                }
            }
        }
        if (MODE == MODE_COX && blockIdx.x == 0 && tid < FT) {
            for (int lr = 0; lr < crows; lr++) c2acc += tc[lr * FT + tid];
        }
        __syncthreads();
        if (tid == 0 && q + 2 < nchunks) issue(q + 2, stage);
    }

    if (MODE == MODE_COX && blockIdx.x == 0 && tid < FT) d.c2sum[s * FT + tid] = c2acc;
    if (!active) return;
    // partials: part[((s*NQ + q)*FT + f) * pstride + j]
#pragma unroll
    for (int f = 0; f < FT; f++) {
        auto put = [&](int q, double v0, double v1) {
            double *dst = d.part + ((size_t)(s * NQ + q) * FT + f) * d.pstride + j0;
            if (CPT == 2)
                *reinterpret_cast<double2 *>(dst) = make_double2(v0, v1);
            else
                *dst = v0;
        };
        put(0, accd[0][f], accd[CPT - 1][f]);
        if constexpr (MODE >= MODE_DH) put(1, acch[0][f], acch[CPT - 1][f]);
        if constexpr (MODE == MODE_COX) {
            put(2, s1[0][f], s1[CPT - 1][f]);
            put(3, accA[0][f], accA[CPT - 1][f]);
            put(4, accB[0][f], accB[CPT - 1][f]);
        }
    }
}

template <int FT, int MODE, int CPT>
static void launch_sweep_t(const Dev &d, cudaStream_t st)
{
    constexpr int NV = SweepTraits<MODE>::NV;
    const size_t smem = (size_t)2 * NV * SWEEP_RC * FT * sizeof(double);
    static bool configured = false;
    if (!configured) {
        CUDA_CHECK(cudaFuncSetAttribute(dual_sweep_kernel<FT, MODE, CPT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem));
        configured = true;
    }
    const long long cols_per_cta = (long long)SWEEP_NT * CPT;
    dim3 grid((unsigned)((d.p + cols_per_cta - 1) / cols_per_cta), (unsigned)d.S);
    dual_sweep_kernel<FT, MODE, CPT><<<grid, SWEEP_NT, smem, st>>>(d);
    CUDA_CHECK(cudaGetLastError());
}

// columns per thread of dual_sweep_kernel: 2 (16-byte loads) unless the accumulator set would not fit in registers
constexpr int stream_cpt(int FT, int MODE)
{
    return FT <= 2 ? 2 : (FT <= 6 ? (MODE == MODE_COX ? 1 : 2) : (FT <= 12 ? (MODE == MODE_D ? 2 : 1) : 1));
}

template <int MODE>
static void launch_sweep_m(const Dev &d, cudaStream_t st)
{
    switch (d.FS) {
        case 1: launch_sweep_t<1, MODE, stream_cpt(1, MODE)>(d, st); break;
        case 2: launch_sweep_t<2, MODE, stream_cpt(2, MODE)>(d, st); break;
        case 4: launch_sweep_t<4, MODE, stream_cpt(4, MODE)>(d, st); break;
        case 6: launch_sweep_t<6, MODE, stream_cpt(6, MODE)>(d, st); break;
        case 8: launch_sweep_t<8, MODE, stream_cpt(8, MODE)>(d, st); break;
        case 12: launch_sweep_t<12, MODE, stream_cpt(12, MODE)>(d, st); break;
        case 16: launch_sweep_t<16, MODE, stream_cpt(16, MODE)>(d, st); break;
        case 24: launch_sweep_t<24, MODE, stream_cpt(24, MODE)>(d, st); break;
        case 32: launch_sweep_t<32, MODE, stream_cpt(32, MODE)>(d, st); break;
        default: throw EngineError{"dual sweep: unsupported chain tile FS=" + std::to_string(d.FS)};
    }
}

int sweep_cpt(const Dev &d, int mode)
{
    return sweep_uses_tma(d) ? sweep_tma_cpt(d.FS, mode) : stream_cpt(d.FS, mode);
}

void launch_dual_sweep(const Dev &d, int mode, cudaStream_t st)
{
    if (sweep_uses_tma(d)) {
        launch_dual_sweep_tma(d, mode, st);
        return;
    }
    if (mode == MODE_D) launch_sweep_m<MODE_D>(d, st);
    else if (mode == MODE_DH) launch_sweep_m<MODE_DH>(d, st);
    else launch_sweep_m<MODE_COX>(d, st);
}

// =====================================================================================================
// finish: reduce row-split partials, apply the sacrifice
// =====================================================================================================
// sacrifice / screening utility from the reduced sums (the tail of the finish epilogue)
template <int EPI>
__device__ __forceinline__ double finish_epilogue(const Dev &d, int c, long long j, double dsum, double hsum, double R)
{
    double out;
    if (EPI == EPI_SCREEN_LM) {
        const double bq = dsum / hsum;  // one-column least squares (screening.cpp:46)
        out = bq * bq;
    } else {
        const double beta = d.betaD[(size_t)c * d.pstride + j];
        const double lam2 = 2.0 * d.lambda;  // L0L2 ridge term (Algorithm.h:1109, 1236/1246, 1341/1350, 1629-1630)
        if (EPI == EPI_SACR_LM) {
            // Phi = sqrt(2*lambda + x_j.x_j / n) (utilities.cpp:142-151), invPhi = 1/Phi (:167-177); Algorithm.h:1116-1122
            const double phi = sqrt(lam2 + d.xtx[(size_t)c * d.pstride + j] / (double)d.ntrain[c]);
            const double t = phi * beta + (1.0 / phi) * (dsum - lam2 * beta);
            out = t * t;
        } else if (EPI == EPI_SACR_GLM) {
            const double phi = sqrt(hsum + lam2);  // Algorithm.h:1238-1257 / 1342-1361
            const double t = phi * beta + (1.0 / phi) * (dsum - lam2 * beta);
            out = t * t;
        } else {
            // Algorithm.h:1626-1634: l1 = -dsum + 2*lambda*beta, l2 = hsum - R + 2*lambda, d = -l1/l2, bd = |beta + d| * sqrt(l2)
            const double l2 = hsum - R + lam2;
            out = fabs(beta + (dsum - lam2 * beta) / l2) * sqrt(l2);
        }
    }
    return out;
}

// value of the finish epilogue EPI for chain c, column j: reduces the row-split partials in a fixed order and applies the
// sacrifice / screening formula.  EPI_RAW writes the reduced sums to raw_out and returns 0.
template <int EPI>
__device__ __forceinline__ double finish_value(const Dev &d, int mode, int c, long long j, double *raw_out)
{
    const int NQ = mode == MODE_D ? 1 : (mode == MODE_DH ? 2 : 5);
    const int FT = d.FS;
    double dsum = 0.0, hsum = 0.0, R = 0.0;
    if (mode != MODE_COX) {
        for (int s = 0; s < d.S; s++) {
            dsum += d.part[((size_t)(s * NQ + 0) * FT + c) * d.pstride + j];
            if (mode == MODE_DH) hsum += d.part[((size_t)(s * NQ + 1) * FT + c) * d.pstride + j];
        }
    } else {
        double carry = 0.0;
        for (int s = d.S - 1; s >= 0; s--) {
            const size_t base = ((size_t)(s * NQ) * FT + c) * d.pstride + j;
            const size_t qs = (size_t)FT * d.pstride;
            dsum += d.part[base];
            hsum += d.part[base + qs];
            const double Ts = d.part[base + 2 * qs], As = d.part[base + 3 * qs], Bs = d.part[base + 4 * qs];
            R += As + 2.0 * carry * Bs + carry * carry * d.c2sum[s * FT + c];
            carry += Ts;
        }
    }
    if (EPI == EPI_RAW) {
        raw_out[(size_t)(0 * FT + c) * d.pstride + j] = dsum;
        if (mode >= MODE_DH) raw_out[(size_t)(1 * FT + c) * d.pstride + j] = hsum;
        return 0.0;
    }
    return finish_epilogue<EPI>(d, c, j, dsum, hsum, R);
}

// The same for NB columns j0, j0 + jstep, ... of one thread at once (gaussian / GLM sweeps): the partials of all NB columns
// are in flight together instead of one dependent chain of S loads per column.  Per column the partials are still added
// in the order s = 0 .. S-1, so the result is bit-identical to finish_value.
template <int EPI, int NB>
__device__ __forceinline__ void finish_batch(const Dev &d, int mode, int c, long long j0, long long jstep, int nb, double (&out)[NB])
{
    const int NQ = mode == MODE_D ? 1 : 2;
    const int FT = d.FS;
    double ds[NB], hs[NB];
#pragma unroll
    for (int q = 0; q < NB; q++) ds[q] = 0.0, hs[q] = 0.0;
#pragma unroll 2
    for (int s = 0; s < d.S; s++) {
        const double *pd = d.part + ((size_t)(s * NQ + 0) * FT + c) * d.pstride + j0;
        const double *ph = d.part + ((size_t)(s * NQ + (NQ - 1)) * FT + c) * d.pstride + j0;
        double vd[NB], vh[NB];
#pragma unroll
        for (int q = 0; q < NB; q++) {
            vd[q] = q < nb ? pd[q * jstep] : 0.0;
            vh[q] = (q < nb && mode == MODE_DH) ? ph[q * jstep] : 0.0;
        }
#pragma unroll
        for (int q = 0; q < NB; q++) {
            ds[q] += vd[q];
            hs[q] += vh[q];
        }
    }
#pragma unroll
    for (int q = 0; q < NB; q++)
        if (q < nb) out[q] = finish_epilogue<EPI>(d, c, j0 + q * jstep, ds[q], hs[q], 0.0);
}


template <int EPI>
__global__ void __launch_bounds__(256) finish_kernel(const Dev d, int mode, const BatchDesc b, double *raw_out)
{
    const long long j = (long long)blockIdx.x * 256 + threadIdx.x;
    if (j >= d.p) return;
    if (d.gate && *d.gate == 0) return;
    const int c = b.chain[blockIdx.y];  // chain id == slot in the sweep vectors
    const double out = finish_value<EPI>(d, mode, c, j, raw_out);
    if (EPI != EPI_RAW) d.bd[(size_t)c * d.pstride + j] = out;
}

void launch_finish(const Dev &d, int mode, int epi, const BatchDesc &b, double *raw_out, cudaStream_t st)
{
    dim3 grid((unsigned)((d.p + 255) / 256), (unsigned)b.nch);
    switch (epi) {
        case EPI_RAW: finish_kernel<EPI_RAW><<<grid, 256, 0, st>>>(d, mode, b, raw_out); break;
        case EPI_SACR_LM: finish_kernel<EPI_SACR_LM><<<grid, 256, 0, st>>>(d, mode, b, raw_out); break;
        case EPI_SACR_GLM: finish_kernel<EPI_SACR_GLM><<<grid, 256, 0, st>>>(d, mode, b, raw_out); break;
        case EPI_SACR_COX: finish_kernel<EPI_SACR_COX><<<grid, 256, 0, st>>>(d, mode, b, raw_out); break;
        default: finish_kernel<EPI_SCREEN_LM><<<grid, 256, 0, st>>>(d, mode, b, raw_out); break;
    }
    CUDA_CHECK(cudaGetLastError());
}

// always_select -> DBL_MAX (utilities.cpp:190-199)
__global__ void pin_kernel(double *vals, long long stride, int nch, const int *idx, int nidx, const int *gate)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nidx * nch) return;
    if (gate && *gate == 0) return;
    vals[(size_t)(i / nidx) * stride + idx[i % nidx]] = DBL_MAX;
}
void launch_pin(const Dev &d, double *vals, long long stride, int nch, const int *idx, int nidx, cudaStream_t st)
{
    if (nidx <= 0) return;
    const int tot = nidx * nch;
    pin_kernel<<<(tot + 255) / 256, 256, 0, st>>>(vals, stride, nch, idx, nidx, d.gate);
    CUDA_CHECK(cudaGetLastError());
}

// =====================================================================================================
// exact top-k: radix select in shared memory + ordered compaction
// =====================================================================================================
// One CTA selects the top min(k, len) keys of its slice and writes them IN INPUT ORDER (so candidate lists stay
// index-ascending through every stage and the final list needs no sort).  Total order: larger key first, then
// lower index first.  grid = (nslices, nchains).
__device__ __forceinline__ unsigned long long topk_key(double v)
{
    unsigned long long u = (unsigned long long)__double_as_longlong(v);
    if (!(v == v) || v < 0.0) u = 0ull;  // NaN / negative never happen for a sacrifice; rank them last
    return u;
}

// The select half of topk_body over `len` keys already in shared memory (block-synchronised by its first barrier):
// every key > thr is taken, plus the first krem keys equal to thr; neq keys equal thr (a boundary tie when neq > krem).
// Block-wide: every thread returns the same values.  blockDim = TOPK_NT.
__device__ __forceinline__ void topk_threshold(const unsigned long long *keys, int len, int kk, unsigned long long &thr_out,
                                               int &krem_out, int &neq_out)
{
    __shared__ int hist[256];
    __shared__ unsigned long long sh_prefix;
    __shared__ int sh_krem, sh_neq, sh_cnt;
    __shared__ unsigned long long small_bin[32];
    const int tid = threadIdx.x;
    unsigned long long thr = 0ull;
    int krem = kk, neq = len;
    if (kk < len) {
        unsigned long long prefix = 0ull, mask = 0ull;
        bool early = false;
        for (int pass = 7; pass >= 0; pass--) {
            const int shift = pass * 8;
            if (tid < 256) hist[tid] = 0;
            __syncthreads();
            // (a warp-aggregated variant -- __match_any_sync on the digit, one atomicAdd per distinct digit -- was measured
            // and lost: 0.135 -> 0.247 ms for the four stages of the screening's top-5000; match.any costs more than the
            // same-address shared atomics it saves; so did a single-ballot variant that counts the lanes sharing the digit
            // of the warp's first candidate with one add: 0.134 -> 0.160 ms -- the hardware already merges same-address
            // shared atomics of a warp)
            for (int i = tid; i < len; i += TOPK_NT) {
                const unsigned long long u = keys[i];
                if ((u & mask) == prefix) atomicAdd(&hist[(int)((u >> shift) & 255ull)], 1);
            }
            __syncthreads();
            if (tid < 32) {
                // lane owns bins [8*lane, 8*lane+8); find the digit where the count from the top reaches krem
                int loc[8], tot = 0;
#pragma unroll
                for (int q = 0; q < 8; q++) { loc[q] = hist[tid * 8 + q]; tot += loc[q]; }
                // suffix sums over lanes (higher lanes = larger digits)
                int suf = tot;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    int t = __shfl_down_sync(0xffffffffu, suf, o);
                    if (tid + o < 32) suf += t;
                }
                const int above = suf - tot;  // keys with a digit in a higher lane
                if (above < krem && suf >= krem) {
                    int acc = above;
                    for (int q = 7; q >= 0; q--) {
                        if (acc + loc[q] >= krem) {
                            sh_prefix = prefix | ((unsigned long long)(tid * 8 + q) << shift);
                            sh_krem = krem - acc;
                            sh_neq = loc[q];
                            break;
                        }
                        acc += loc[q];
                    }
                }
            }
            __syncthreads();
            prefix = sh_prefix;
            krem = sh_krem;
            neq = sh_neq;
            mask |= 255ull << shift;
            __syncthreads();
            // every key of the boundary bin is wanted: the select is decided, the remaining digits cannot change it
            if (neq == krem && pass > 0 && prefix > 0ull) {
                early = true;
                break;
            }
            // few keys left in the boundary bin (the usual case after two digits: the largest sacrifices are spread over
            // orders of magnitude): rank them in one warp instead of walking the remaining digits
            if (neq <= 32 && pass > 0) {
                if (tid == 0) sh_cnt = 0;
                __syncthreads();
                for (int i = tid; i < len; i += TOPK_NT) {
                    const unsigned long long u = keys[i];
                    if ((u & mask) == prefix) small_bin[atomicAdd(&sh_cnt, 1)] = u;
                }
                __syncthreads();
                if (tid < 32 && tid < neq) {
                    const unsigned long long u = small_bin[tid];
                    int gt = 0, ge = 0;
                    for (int j = 0; j < neq; j++) {
                        const unsigned long long v = small_bin[j];
                        gt += (v > u);
                        ge += (v >= u);
                    }
                    if (gt < krem && krem <= ge) {  // u is the krem-th largest of the bin (all its duplicates agree)
                        sh_prefix = u;
                        sh_krem = krem - gt;
                        sh_neq = ge - gt;
                    }
                }
                __syncthreads();
                prefix = sh_prefix;
                krem = sh_krem;
                neq = sh_neq;
                __syncthreads();
                break;
            }
        }
        if (early) {
            thr = prefix - 1ull;  // u > thr  <=>  u >= prefix (lower digits zero): all of the boundary bin and above
            krem = 0;             // nothing is taken from keys equal to thr (they sit in a lower bin)
            neq = 0;
        } else {
            thr = prefix;
        }
    } else {
        __syncthreads();
    }
    thr_out = thr;
    krem_out = krem;
    neq_out = neq;
}

// Select + ordered compaction over `len` keys already in shared memory (block-synchronised by the caller's first barrier
// inside).  Outputs as in topk_slices_kernel.
__device__ __forceinline__ void topk_body(unsigned long long *keys, int len, int k, int slice_len, const int *iin, int b0, int s,
                                          int f, double *keys_out, int *idx_out, long long out_stride, int *final_out,
                                          int final_ld, int *tie)
{
    __shared__ unsigned long long scan_sh[34];
    const int tid = threadIdx.x;
    const int kk = min(k, len);
    const int out_per_slice = min(k, slice_len);
    unsigned long long thr;
    int krem, neq;
    topk_threshold(keys, len, kk, thr, krem, neq);
    // ordered compaction.  thread owns a contiguous chunk.
    const int per = (len + TOPK_NT - 1) / TOPK_NT;
    const int cb = min(len, tid * per), ce = min(len, cb + per);
    unsigned int cgt = 0, ceq = 0;
    if (kk < len) {
        for (int i = cb; i < ce; i++) {
            const unsigned long long u = keys[i];
            cgt += (u > thr);
            ceq += (u == thr);
        }
    } else {
        cgt = ce - cb;
    }
    // exclusive scan of (gt, eq) packed in 64 bits
    unsigned long long v = ((unsigned long long)cgt << 32) | ceq, inc = v;
    const int lane = tid & 31, wid = tid >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) scan_sh[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        unsigned long long w = scan_sh[lane], winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            unsigned long long t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        scan_sh[lane] = winc - w;
    }
    __syncthreads();
    const unsigned long long ex = scan_sh[wid] + (inc - v);
    int gt_before = (int)(ex >> 32), eq_before = (int)(ex & 0xffffffffull);
    for (int i = cb; i < ce; i++) {
        const unsigned long long u = keys[i];
        bool sel;
        if (kk >= len) sel = true;
        else if (u > thr) sel = true;
        else if (u == thr) sel = eq_before < krem;
        else sel = false;
        if (sel) {
            const int pos = gt_before + min(eq_before, kk < len ? krem : 0);
            const int id = iin ? iin[i] : (b0 + i);
            if (final_out) {
                final_out[(size_t)f * final_ld + pos] = id;
            } else {
                keys_out[(size_t)f * out_stride + (size_t)s * out_per_slice + pos] = __longlong_as_double((long long)u);
                idx_out[(size_t)f * out_stride + (size_t)s * out_per_slice + pos] = id;
            }
        }
        if (kk < len) {
            gt_before += (u > thr);
            eq_before += (u == thr);
        } else {
            gt_before++;
        }
    }
    if (final_out && tie && tid == 0) tie[f] = (kk < len && neq > krem) ? 1 : 0;
}


// One CTA selects the top min(k, len) keys of its slice and writes them IN INPUT ORDER (so candidate lists stay
// index-ascending through every stage and the final list needs no sort).  Total order: larger key first, then
// lower index first.  grid = (nslices, nchains).
__global__ void __launch_bounds__(TOPK_NT) topk_slices_kernel(const double *__restrict__ keys_in,
                                                              const int *__restrict__ idx_in, long long in_stride,
                                                              int n_in, int k, int slice_len, double *keys_out,
                                                              int *idx_out, long long out_stride, int *final_out,
                                                              int final_ld, int *tie, const int *gate)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned long long *keys = reinterpret_cast<unsigned long long *>(smem_raw);
    if (gate && *gate == 0) return;
    const int tid = threadIdx.x;
    const int s = blockIdx.x, f = blockIdx.y;
    const int b0 = s * slice_len;
    const int len = min(slice_len, n_in - b0);
    if (len <= 0) return;
    const double *kin = keys_in + (size_t)f * in_stride + b0;
    const int *iin = idx_in ? idx_in + (size_t)f * in_stride + b0 : nullptr;
    for (int i = tid; i < len; i += TOPK_NT) keys[i] = topk_key(kin[i]);
    topk_body(keys, len, k, slice_len, iin, b0, s, f, keys_out, idx_out, out_stride, final_out, final_ld, tie);
}

// Fused finish + pin + top-k for designs of at most TOPK_LMAX columns: the CTA of chain c reduces the sweep partials and
// applies the sacrifice itself (finish_value), pins the always-include columns to DBL_MAX (utilities.cpp:190-199) and
// selects -- the sacrifice vector never goes to memory.  grid = (1, chains cmin..cmax); chains that already met the
// stopping rule are skipped.
template <int EPI>
__global__ void __launch_bounds__(TOPK_NT) topk_fused_kernel(const Dev d, int mode, int cmin, int k, const int *always,
                                                             int n_always)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned long long *keys = reinterpret_cast<unsigned long long *>(smem_raw);
    if (d.gate && *d.gate == 0) return;
    const int tid = threadIdx.x;
    const int c = cmin + blockIdx.y;
    if (d.done[c]) return;
    const int len = d.p;
    if (mode != MODE_COX) {
        constexpr int NB = 8;
        for (int i0 = tid; i0 < len; i0 += NB * TOPK_NT) {
            const int nb = min(NB, (len - i0 + TOPK_NT - 1) / TOPK_NT);
            double v[NB];
            finish_batch<EPI, NB>(d, mode, c, i0, TOPK_NT, nb, v);
#pragma unroll
            for (int q = 0; q < NB; q++)
                if (q < nb) keys[i0 + q * TOPK_NT] = topk_key(v[q]);
        }
    } else {
        for (int i = tid; i < len; i += TOPK_NT) keys[i] = topk_key(finish_value<EPI>(d, mode, c, i, nullptr));
    }
    if (n_always > 0) {
        __syncthreads();
        for (int q = tid; q < n_always; q += TOPK_NT) keys[always[q]] = (unsigned long long)__double_as_longlong(DBL_MAX);
    }
    topk_body(keys, len, k, len, nullptr, 0, 0, 0, nullptr, nullptr, 0, d.Anew + (size_t)c * d.kcap, d.kcap, d.tie + c);
}
void launch_topk_fused(const Dev &d, int mode, int epi, int cmin, int nspan, int k, const int *always, int n_always,
                       cudaStream_t st)
{
    if (k > d.p) throw EngineError{"top-k: k > number of candidates"};
    if (d.p > TOPK_LMAX) throw EngineError{"fused top-k: too many columns"};
    const size_t smem = (size_t)d.p * 8;
    dim3 grid(1, nspan);
    static bool configured = false;
    if (!configured) {
        CUDA_CHECK(cudaFuncSetAttribute(topk_fused_kernel<EPI_SACR_LM>, cudaFuncAttributeMaxDynamicSharedMemorySize, TOPK_LMAX * 8));
        CUDA_CHECK(cudaFuncSetAttribute(topk_fused_kernel<EPI_SACR_GLM>, cudaFuncAttributeMaxDynamicSharedMemorySize, TOPK_LMAX * 8));
        CUDA_CHECK(cudaFuncSetAttribute(topk_fused_kernel<EPI_SACR_COX>, cudaFuncAttributeMaxDynamicSharedMemorySize, TOPK_LMAX * 8));
        configured = true;
    }
    if (epi == EPI_SACR_LM) topk_fused_kernel<EPI_SACR_LM><<<grid, TOPK_NT, smem, st>>>(d, mode, cmin, k, always, n_always);
    else if (epi == EPI_SACR_GLM) topk_fused_kernel<EPI_SACR_GLM><<<grid, TOPK_NT, smem, st>>>(d, mode, cmin, k, always, n_always);
    else topk_fused_kernel<EPI_SACR_COX><<<grid, TOPK_NT, smem, st>>>(d, mode, cmin, k, always, n_always);
    CUDA_CHECK(cudaGetLastError());
}

int launch_topk(const double *vals, long long stride, int n_in, int k, int nch, int *out_idx, int out_ld, int *tie,
                double *ck0, int *ci0, double *ck1, int *ci1, long long cstride, cudaStream_t st, const int *gate,
                const int *idx0)
{
    if (k > n_in) throw EngineError{"top-k: k > number of candidates"};
    const double *kin = vals;
    const int *iin = idx0;
    long long in_stride = stride;
    int cur_n = n_in;
    int pp = 0;
    for (int guard = 0; guard < 16; guard++) {
        if (cur_n <= TOPK_LMAX) {
            const size_t smem = (size_t)cur_n * 8;
            dim3 grid(1, nch);
            topk_slices_kernel<<<grid, TOPK_NT, smem, st>>>(kin, iin, in_stride, cur_n, k, cur_n, nullptr, nullptr, 0,
                                                            out_idx, out_ld, tie, gate);
            CUDA_CHECK(cudaGetLastError());
            return guard + 1;
        }
        // slice length: keep >= ~600 CTAs busy but never so short that nothing is filtered
        int slice = 8192;
        while (slice < TOPK_LMAX && k * 2 > slice) slice *= 2;
        if (k * 2 > slice)
            throw EngineError{"top-k: k=" + std::to_string(k) + " too large for the shared-memory radix select (max " +
                              std::to_string(TOPK_LMAX / 2) + " when p > " + std::to_string(TOPK_LMAX) + ")"};
        const int nsl = (cur_n + slice - 1) / slice;
        const int per = k < slice ? k : slice;
        // the last slice may be shorter than `per`: its candidates are packed at s*per; we compact counts on the host
        // side by making the stage output dense: slice s writes min(k, len_s) entries; only the LAST slice can be
        // short, so the dense length is (nsl-1)*per + min(k, len_last).
        const int len_last = cur_n - (nsl - 1) * slice;
        const int out_n = (nsl - 1) * per + (k < len_last ? k : len_last);
        double *ko = pp ? ck1 : ck0;
        int *io = pp ? ci1 : ci0;
        if ((long long)out_n > cstride) throw EngineError{"top-k: candidate scratch too small"};
        dim3 grid(nsl, nch);
        topk_slices_kernel<<<grid, TOPK_NT, (size_t)slice * 8, st>>>(kin, iin, in_stride, cur_n, k, slice, ko, io,
                                                                    cstride, nullptr, 0, nullptr, gate);
        CUDA_CHECK(cudaGetLastError());
        kin = ko;
        iin = io;
        in_stride = cstride;
        cur_n = out_n;
        pp ^= 1;
    }
    throw EngineError{"top-k: did not converge"};
}

// =====================================================================================================
// device-wide exact select of the screening list (p > TOPK_LMAX): the same list, order and tie flag as launch_topk
// =====================================================================================================
// launch_topk at p = 500 000, k = 5000 is four dependent stages of 31, 10, 4 and 1 CTAs, each an 8-pass radix select in one
// CTA's shared memory: latency-bound with most SMs idle.  Here every pass spreads over the machine:
//   ss_hist_kernel (pass 0)  histogram of the top 12 key bits (sign + exponent); the last CTA finds the boundary bin
//   ss_hist_kernel (pass 1)  histogram of the next 12 bits inside that bin; the last CTA finds the boundary sub-bin
//   ss_collect_kernel        the keys of the boundary sub-bin -> scratch (at most TOPK_LMAX, else the fallback flag)
//   ss_resolve_kernel        one CTA: topk_threshold over them -> thr, krem (keys == thr taken), the tie flag
//   ss_count_kernel          per-chunk counts of (key > thr, key == thr)
//   ss_write_kernel          chunk base by summing the counts before it, block scan, ordered compaction (ascending)
// A boundary sub-bin larger than TOPK_LMAX (all-zero or massively tied utilities) sets the fallback flag: the kernels above
// stop and launch_topk, enqueued behind them and gated on that flag, decides -- no host round trip.
constexpr int SS_NT = 512;
constexpr int SS_BINS = 4096;        // 12-bit digits
constexpr int SS_CHUNK = SS_NT * 8;  // keys per CTA of the ordered compaction
struct SsState {                     // zeroed before every select
    int hist[2][SS_BINS];
    int done[2];
    int bin[2];    // boundary digit of pass 0 / pass 1
    int above[2];  // keys above the boundary bin / sub-bin
    int fallback;
    int ncand;
    int krem, neq;
    unsigned long long thr;
};

__global__ void __launch_bounds__(SS_NT) ss_hist_kernel(const double *__restrict__ vals, int p, int k, int pass, SsState *s)
{
    __shared__ int h[SS_BINS];
    __shared__ int suf[SS_NT];
    __shared__ bool last;
    const int tid = threadIdx.x;
    for (int i = tid; i < SS_BINS; i += SS_NT) h[i] = 0;
    __syncthreads();
    const int b0 = pass ? s->bin[0] : 0;
    for (long long i = (long long)blockIdx.x * SS_NT + tid; i < p; i += (long long)gridDim.x * SS_NT) {
        const unsigned long long u = topk_key(vals[i]);
        if (pass == 0) atomicAdd(&h[(int)(u >> 52)], 1);
        else if ((int)(u >> 52) == b0) atomicAdd(&h[(int)((u >> 40) & (SS_BINS - 1))], 1);
    }
    __syncthreads();
    for (int i = tid; i < SS_BINS; i += SS_NT)
        if (h[i]) atomicAdd(&s->hist[pass][i], h[i]);
    __threadfence();
    __syncthreads();
    if (tid == 0) last = atomicAdd(&s->done[pass], 1) == (int)gridDim.x - 1;
    __syncthreads();
    if (!last) return;
    __threadfence();
    // the last CTA: the digit at which the count from the top reaches krem (thread t owns bins [8t, 8t + 8))
    const int above0 = pass ? __ldcg(&s->above[0]) : 0;
    const int krem = k - above0;
    int loc[8], tot = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        loc[q] = __ldcg(&s->hist[pass][tid * 8 + q]);
        tot += loc[q];
    }
    suf[tid] = tot;
    __syncthreads();
    for (int o = 1; o < SS_NT; o <<= 1) {
        const int v = tid + o < SS_NT ? suf[tid + o] : 0;
        __syncthreads();
        suf[tid] += v;
        __syncthreads();
    }
    int acc = suf[tid] - tot;  // keys in the bins of higher threads
    if (acc < krem && suf[tid] >= krem) {
        for (int q = 7; q >= 0; q--) {
            if (acc + loc[q] >= krem) {
                s->bin[pass] = tid * 8 + q;
                s->above[pass] = above0 + acc;
                if (pass == 1) s->fallback = loc[q] > TOPK_LMAX;
                break;
            }
            acc += loc[q];
        }
    }
}

__global__ void __launch_bounds__(SS_NT) ss_collect_kernel(const double *__restrict__ vals, int p, SsState *s,
                                                           unsigned long long *cand)
{
    if (s->fallback) return;
    const unsigned long long pb = ((unsigned long long)s->bin[0] << 12) | (unsigned long long)s->bin[1];  // key >> 40
    for (long long i = (long long)blockIdx.x * SS_NT + threadIdx.x; i < p; i += (long long)gridDim.x * SS_NT) {
        const unsigned long long u = topk_key(vals[i]);
        if ((u >> 40) == pb) cand[atomicAdd(&s->ncand, 1)] = u;
    }
}

__global__ void __launch_bounds__(TOPK_NT) ss_resolve_kernel(int k, SsState *s, const unsigned long long *cand, int *tie)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    unsigned long long *keys = reinterpret_cast<unsigned long long *>(smem_raw);
    __shared__ unsigned long long mn;
    __shared__ int cmin;
    if (s->fallback) return;
    const int tid = threadIdx.x;
    const int nb = s->ncand;
    const int krem = k - s->above[1];  // 1 <= krem <= nb
    for (int i = tid; i < nb; i += TOPK_NT) keys[i] = cand[i];
    unsigned long long thr;
    int kr, neq;
    if (krem < nb) {
        topk_threshold(keys, nb, krem, thr, kr, neq);
    } else {  // the whole sub-bin is taken: the threshold is its smallest key, and every copy of it is taken
        if (tid == 0) { mn = ~0ull; cmin = 0; }
        __syncthreads();
        for (int i = tid; i < nb; i += TOPK_NT) atomicMin(&mn, keys[i]);
        __syncthreads();
        for (int i = tid; i < nb; i += TOPK_NT)
            if (keys[i] == mn) atomicAdd(&cmin, 1);
        __syncthreads();
        thr = mn;
        kr = neq = cmin;
    }
    if (tid == 0) {
        s->thr = thr;
        s->krem = kr;
        s->neq = neq;
        *tie = neq > kr ? 1 : 0;
    }
}

// (key > thr, key == thr) packed as (gt << 32) | eq
__device__ __forceinline__ unsigned long long ss_block_sum(unsigned long long v, unsigned long long *red)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if (lane == 0) red[wid] = v;
    __syncthreads();
    unsigned long long t = 0;
    if (wid == 0) {
        t = lane < SS_NT / 32 ? red[lane] : 0ull;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) t += __shfl_xor_sync(0xffffffffu, t, o);
    }
    return t;  // valid on thread 0
}

__global__ void __launch_bounds__(SS_NT) ss_count_kernel(const double *__restrict__ vals, int p, const SsState *s,
                                                         unsigned long long *cnt)
{
    __shared__ unsigned long long red[SS_NT / 32];
    if (s->fallback) return;
    const unsigned long long thr = s->thr;
    const long long c0 = (long long)blockIdx.x * SS_CHUNK;
    unsigned long long c = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        const long long i = c0 + q * SS_NT + threadIdx.x;
        if (i < p) {
            const unsigned long long u = topk_key(vals[i]);
            c += (u > thr ? (1ull << 32) : 0ull) + (u == thr ? 1ull : 0ull);
        }
    }
    const unsigned long long t = ss_block_sum(c, red);
    if (threadIdx.x == 0) cnt[blockIdx.x] = t;
}

__global__ void __launch_bounds__(SS_NT) ss_write_kernel(const double *__restrict__ vals, int p, const SsState *s,
                                                         const unsigned long long *cnt, int *out_idx)
{
    __shared__ unsigned long long red[SS_NT / 32];
    __shared__ unsigned long long base_sh;
    __shared__ unsigned long long scan_sh[SS_NT / 32];
    if (s->fallback) return;
    const unsigned long long thr = s->thr;
    const int krem = s->krem;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    // counts of the chunks before this one
    unsigned long long b = 0;
    for (int q = tid; q < (int)blockIdx.x; q += SS_NT) b += cnt[q];
    b = ss_block_sum(b, red);
    if (tid == 0) base_sh = b;
    // this thread's 8 contiguous keys
    const long long i0 = (long long)blockIdx.x * SS_CHUNK + (long long)tid * 8;
    unsigned long long u[8];
    unsigned long long v = 0;
#pragma unroll
    for (int q = 0; q < 8; q++) {
        u[q] = i0 + q < p ? topk_key(vals[i0 + q]) : 0ull;
        if (i0 + q < p) v += (u[q] > thr ? (1ull << 32) : 0ull) + (u[q] == thr ? 1ull : 0ull);
    }
    // exclusive block scan of v
    unsigned long long inc = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const unsigned long long t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += t;
    }
    if (lane == 31) scan_sh[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        const unsigned long long w = lane < SS_NT / 32 ? scan_sh[lane] : 0ull;
        unsigned long long winc = w;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long t = __shfl_up_sync(0xffffffffu, winc, o);
            if (lane >= o) winc += t;
        }
        if (lane < SS_NT / 32) scan_sh[lane] = winc - w;
    }
    __syncthreads();
    const unsigned long long ex = base_sh + scan_sh[wid] + (inc - v);
    int gt_before = (int)(ex >> 32), eq_before = (int)(ex & 0xffffffffull);
#pragma unroll
    for (int q = 0; q < 8; q++) {
        if (i0 + q >= p) break;
        const bool sel = u[q] > thr || (u[q] == thr && eq_before < krem);
        if (sel) out_idx[gt_before + min(eq_before, krem)] = (int)(i0 + q);
        gt_before += u[q] > thr;
        eq_before += u[q] == thr;
    }
}

size_t screen_select_scratch_bytes(int p)
{
    return sizeof(SsState) + (size_t)TOPK_LMAX * 8 + (size_t)((p + SS_CHUNK - 1) / SS_CHUNK) * 8;
}

int launch_screen_select(const double *vals, int p, int k, int *out_idx, int *tie, void *scratch, double *ck0, int *ci0,
                         double *ck1, int *ci1, long long cstride, cudaStream_t st)
{
    if (k < 1 || k > p) throw EngineError{"screen select: need 1 <= k <= p"};
    // one CTA holds every key (p <= TOPK_LMAX), or a k the fallback could not take: launch_topk as it is
    if (p <= TOPK_LMAX || 2LL * k > TOPK_LMAX) return launch_topk(vals, p, p, k, 1, out_idx, k, tie, ck0, ci0, ck1, ci1, cstride, st);
    SsState *s = static_cast<SsState *>(scratch);
    unsigned long long *cand = reinterpret_cast<unsigned long long *>(s + 1);
    unsigned long long *cnt = cand + TOPK_LMAX;
    CUDA_CHECK(cudaMemsetAsync(s, 0, sizeof(SsState), st));
    const int gh = (int)std::min<long long>(1184, ((long long)p + SS_NT * 8 - 1) / (SS_NT * 8));
    const int nchunk = (p + SS_CHUNK - 1) / SS_CHUNK;
    ss_hist_kernel<<<gh, SS_NT, 0, st>>>(vals, p, k, 0, s);
    ss_hist_kernel<<<gh, SS_NT, 0, st>>>(vals, p, k, 1, s);
    ss_collect_kernel<<<gh, SS_NT, 0, st>>>(vals, p, s, cand);
    ss_resolve_kernel<<<1, TOPK_NT, (size_t)TOPK_LMAX * 8, st>>>(k, s, cand, tie);
    ss_count_kernel<<<nchunk, SS_NT, 0, st>>>(vals, p, s, cnt);
    ss_write_kernel<<<nchunk, SS_NT, 0, st>>>(vals, p, s, cnt, out_idx);
    CUDA_CHECK(cudaGetLastError());
    return 6 + launch_topk(vals, p, p, k, 1, out_idx, k, tie, ck0, ci0, ck1, ci1, cstride, st, &s->fallback);
}

// =====================================================================================================
// column-sharded mode: candidate exchange and active-column exchange (the collectives themselves are NCCL calls in
// engine.cu; these kernels pack / unpack their payloads)
// =====================================================================================================
__global__ void pack_candidates_kernel(const double *vals, long long stride, const int *sel, int sel_ld, int kloc, int kpad,
                                       long long offset, Cand *out, int out_ld, const int *gate)
{
    if (gate && *gate == 0) return;
    const int f = blockIdx.y;
    const int a = blockIdx.x * blockDim.x + threadIdx.x;
    if (a >= kpad) return;
    Cand cnd;
    if (a < kloc) {
        const int j = sel[(size_t)f * sel_ld + a];
        cnd.v = vals[(size_t)f * stride + j];
        cnd.idx = (long long)j + offset;
    } else {
        cnd.v = -1.0;
        cnd.idx = 2147483647LL;
    }
    out[(size_t)f * out_ld + a] = cnd;
}
void launch_pack_candidates(const double *vals, long long stride, const int *sel, int sel_ld, int kloc, int kpad,
                            long long offset, int nch, Cand *out, int out_ld, const int *gate, cudaStream_t st)
{
    dim3 grid((kpad + 127) / 128, nch);
    pack_candidates_kernel<<<grid, 128, 0, st>>>(vals, stride, sel, sel_ld, kloc, kpad, offset, out, out_ld, gate);
    CUDA_CHECK(cudaGetLastError());
}
__global__ void unpack_candidates_kernel(const Cand *in, int world, int nch, int in_ld, int k, double *mv, int *mi,
                                         long long mstride, const int *gate)
{
    if (gate && *gate == 0) return;
    const int f = blockIdx.y;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= world * k) return;
    const int q = e / k, a = e - q * k;
    const Cand cnd = in[((size_t)q * nch + f) * in_ld + a];
    mv[(size_t)f * mstride + e] = cnd.v;
    mi[(size_t)f * mstride + e] = (int)cnd.idx;
}
void launch_unpack_candidates(const Cand *in, int world, int nch, int in_ld, int k, double *mv, int *mi, long long mstride,
                              const int *gate, cudaStream_t st)
{
    dim3 grid((world * k + 127) / 128, nch);
    unpack_candidates_kernel<<<grid, 128, 0, st>>>(in, world, nch, in_ld, k, mv, mi, mstride, gate);
    CUDA_CHECK(cudaGetLastError());
}
__global__ void gather_active_kernel(const Dev d, const BatchDesc b, double *AXs)
{
    if (d.gate && *d.gate == 0) return;
    const int c = b.chain[blockIdx.y];
    if (d.done[c]) return;
    const int T = b.T;
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= d.n * T) return;
    const int i = e / T, a = e - i * T;
    const int j = d.Anew[(size_t)c * d.kcap + a] - d.col_lo;
    AXs[((size_t)c * d.n + i) * T + a] = (j >= 0 && j < d.p) ? __ldg(d.X + (size_t)i * d.ldx + j) : 0.0;
}
void launch_gather_active(const Dev &d, const BatchDesc &b, double *AXs, cudaStream_t st)
{
    dim3 grid((d.n * b.T + 255) / 256, b.nch);
    gather_active_kernel<<<grid, 256, 0, st>>>(d, b, AXs);
    CUDA_CHECK(cudaGetLastError());
}
__global__ void gather_owned_cols_kernel(const double *X, long long ldx, int n, int p_local, long long col_lo, const int *sel,
                                         int m, double *Xn, long long ldn)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const long long j = (long long)sel[q] - col_lo;
    const bool own = j >= 0 && j < p_local;
    const int r0 = blockIdx.y * 32, r1 = min(n, r0 + 32);
    for (int i = r0; i < r1; i++) Xn[(size_t)i * ldn + q] = own ? X[(size_t)i * ldx + j] : 0.0;
}
void launch_gather_owned_cols(const double *X, long long ldx, int n, int p_local, long long col_lo, const int *sel, int m,
                              double *Xn, long long ldn, cudaStream_t st)
{
    dim3 grid((m + 127) / 128, (n + 31) / 32);
    gather_owned_cols_kernel<<<grid, 128, 0, st>>>(X, ldx, n, p_local, col_lo, sel, m, Xn, ldn);
    CUDA_CHECK(cudaGetLastError());
}

__global__ void gather_normalize_kernel(const double *__restrict__ X, long long ldx, const int *__restrict__ cols, double *Xn,
                                        long long ldn, int n, int p, const double *gmean, const double *wnorm,
                                        const double *rowmul, double sn, double *mean_out, double *norm_out);

void configure_kernels()
{
    CUDA_CHECK(cudaFuncSetAttribute(topk_slices_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TOPK_LMAX * 8));
    CUDA_CHECK(cudaFuncSetAttribute(ss_resolve_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TOPK_LMAX * 8));
    CUDA_CHECK(cudaFuncSetAttribute(gather_normalize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, NR_SLAB_ROWS * NR_TC * 8));
}

// =====================================================================================================
// losses: Metric.h:145-148/190 (lm), :266-290/336-351 (logistic), :426-440/489 (poisson), :565-568/609 (cox)
// =====================================================================================================
__global__ void __launch_bounds__(FIT_NT) loss_kernel(const Dev d, const LossDesc jobs, const int *testrows,
                                                      const int *ntest, const double *y, const double *w,
                                                      const double *lfact, double *scratch, double *out)
{
    __shared__ double red[40];
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *bsl = reinterpret_cast<double *>(smem_raw);           // [kcap]
    int *As = reinterpret_cast<int *>(bsl + d.kcap);              // [kcap]
    const int job = blockIdx.x;
    const int c = jobs.chain[job], kind = jobs.kind[job], fold = jobs.fold[job];
    const int ks = d.ks[c];
    const double coef0 = d.coef0[c];
    for (int a = threadIdx.x; a < ks; a += FIT_NT) {
        bsl[a] = d.bA[(size_t)c * d.kcap + a];
        As[a] = d.A[(size_t)c * d.kcap + a];
    }
    __syncthreads();
    const int nr = kind == 0 ? d.n : ntest[fold];
    const int *rl = kind == 0 ? nullptr : testrows + (size_t)fold * d.n;
    double *e_s = scratch + (size_t)job * 2 * d.n;
    double *c_s = e_s + d.n;
    double acc = 0.0;
    for (int r = threadIdx.x; r < nr; r += FIT_NT) {
        const int i = rl ? rl[r] : r;
        double eta = d.family == FAM_LM || d.family == FAM_COX ? 0.0 : coef0;
        if (d.ax_ext) {
            const double *row = d.AXk + ((size_t)c * d.n + i) * d.ldXk;
            for (int a = 0; a < ks; a++) eta = fma(row[a], bsl[a], eta);
        } else {
            const double *row = d.X + (size_t)i * d.ldx;
            for (int a = 0; a < ks; a++) eta = fma(row[As[a]], bsl[a], eta);
        }
        if (d.family == FAM_LM) {
            const double t = y[i] - eta;
            acc += t * t;
        } else if (d.family == FAM_LOGIT) {
            const double e = exp(clampd(eta, kind == 0 ? 30.0 : 25.0));
            const double pr = e / (e + 1.0);
            acc += w[i] * (y[i] * log(pr) + (1.0 - y[i]) * log(1.0 - pr));
        } else if (d.family == FAM_POISSON) {
            const double ec = clampd(eta, 30.0);
            acc += (y[i] * ec - exp(ec) - lfact[i]) * w[i];
        } else {
            const double ec = clampd(eta, 30.0);
            e_s[r] = exp(ec);
            c_s[r] = e_s[r];
        }
    }
    double res;
    if (d.family == FAM_COX) {
        __syncthreads();
        block_suffix_scan<FIT_NT>(c_s, nr, red);
        for (int r = threadIdx.x; r < nr; r += FIT_NT) {
            const int i = rl ? rl[r] : r;
            acc += log(e_s[r] / c_s[r]) * y[i] * w[i];
        }
        res = -2.0 * block_sum<FIT_NT>(acc, red);
    } else {
        const double s = block_sum<FIT_NT>(acc, red);
        if (d.family == FAM_LM) res = kind == 0 ? s / (double)d.n : s / (double)(2 * nr);
        else if (d.family == FAM_LOGIT) res = -2.0 * s;
        else res = kind == 0 ? -2.0 * s : -s;
    }
    if (threadIdx.x == 0) out[job] = res;
}

void launch_losses(const Dev &d, const LossDesc &jobs, const int *testrows, const int *ntest, const double *y,
                   const double *w, const double *lfact, double *scratch, double *out, cudaStream_t st)
{
    // + 16: nvcc reads the index list two entries at a time (LDS.64) in the loop remainder, i.e. up to one int past the end
    const size_t smem = (size_t)d.kcap * (sizeof(double) + sizeof(int)) + 16;
    loss_kernel<<<jobs.njobs, FIT_NT, smem, st>>>(d, jobs, testrows, ntest, y, w, lfact, scratch, out);
    CUDA_CHECK(cudaGetLastError());
}

// =====================================================================================================
// normalisation / screening helpers
// =====================================================================================================
// X[i][j] = (X[i][j] - sub[j]) * mul[j] * rowmul[i]     (normalize.cpp:30-45 + Data.h:70-77)
__global__ void center_scale_kernel(double *X, long long ldx, int n, int p, const double *sub, const double *mul,
                                    const double *rowmul)
{
    const long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 2;
    if (j >= p) return;
    const bool two = j + 1 < p;
    const double s0 = sub ? sub[j] : 0.0, s1 = (sub && two) ? sub[j + 1] : 0.0;
    const double m0 = mul ? mul[j] : 1.0, m1 = (mul && two) ? mul[j + 1] : 1.0;
    const int r0 = blockIdx.y * 64, r1 = min(n, r0 + 64);
    // eight rows in flight per thread: the pass is a pure stream (40 MB in, 40 MB out on a screened design), a dependent
    // load -> store per row left the memory system idle most of the time (39 us measured for 80 MB)
    for (int i0 = r0; i0 < r1; i0 += 8) {
        double2 v[8];
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (i0 + u < r1) v[u] = *reinterpret_cast<const double2 *>(X + (size_t)(i0 + u) * ldx + j);
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (i0 + u < r1) {
                const double rm = rowmul ? rowmul[i0 + u] : 1.0;
                double2 o;
                o.x = (v[u].x - s0) * m0 * rm;
                o.y = two ? (v[u].y - s1) * m1 * rm : 0.0;
                *reinterpret_cast<double2 *>(X + (size_t)(i0 + u) * ldx + j) = o;
            }
    }
}
// normx_j = sqrt(h_j), mul_j = sqrt(n) / normx_j  (normalize.cpp:36-45; IEEE sqrt and division: the same bits as the host)
__global__ void norm_factors_kernel(const double *h, int p, double sn, double *norm_out, double *mul_out)
{
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p) return;
    const double nx = sqrt(h[j]);
    norm_out[j] = nx;
    mul_out[j] = sn / nx;
}
void launch_norm_factors(const double *h, int p, double sn, double *norm_out, double *mul_out, cudaStream_t st)
{
    norm_factors_kernel<<<(p + 255) / 256, 256, 0, st>>>(h, p, sn, norm_out, mul_out);
    CUDA_CHECK(cudaGetLastError());
}

// Normalisation of a design that fits L2 (the screened design of config 5: 40 MB) in ONE launch: a CTA owns 8 adjacent
// columns for all rows and makes the three passes of normalize.cpp:20-86 over its own slab (64 KB at n = 1000, re-read
// from L2 / L1) -- weighted column means, norms of the CENTRED columns, scaling (+ the sqrt(w) row factors of add_weight,
// Data.h:70-77).  Per element the arithmetic is that of center_scale_kernel ((x - mean) rounded once, then * mul * rm);
// only the summation order of the two column sums differs from the sweep kernels (fixed: rows warp-strided, warps added
// in order).  Replaces 7 launches and 6 passes over X by 1 launch and 4.
constexpr int NR_NT = 256;
// The three passes over one tile of NR_TC columns; ld(i) reads element i of this thread's column (only called for live
// columns and rows < n), st(i, v) writes it.  Shared by the in-place kernel (ld / st on X itself) and the gather-fused
// kernel (ld from a shared-memory slab, st to Xn): the rows each thread sums, the shuffles, the order in which warps are
// added and the per-element arithmetic are the same for both, so they agree bit for bit.
template <class Ld, class St>
__device__ __forceinline__ void normalize_tile(Ld ld, St st, int n, int p, const double *gmean, const double *wnorm,
                                               const double *rowmul, double sn, double *mean_out, double *norm_out)
{
    __shared__ double red[NR_NT / 32][NR_TC];
    __shared__ double cmean[NR_TC], cmul[NR_TC];
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    constexpr int NW = NR_NT / 32, RS = NW * 4;  // rows per CTA step
    const int c = lane & (NR_TC - 1), rg = lane >> 3;
    const long long j = (long long)blockIdx.x * NR_TC + c;
    const bool live = j < p;
    const int ifirst = wid * 4 + rg;
    // column sum of f(x_i, i) over this thread's rows, 8 loads in flight; then lanes of the same column, then warps
    auto column_sum = [&](auto f) {
        double s = 0.0;
        for (int i0 = ifirst; i0 < n; i0 += 8 * RS) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) v[u] = (live && i0 + u * RS < n) ? ld(i0 + u * RS) : 0.0;
#pragma unroll
            for (int u = 0; u < 8; u++)
                if (i0 + u * RS < n) s = f(v[u], i0 + u * RS, s);
        }
        s += __shfl_xor_sync(0xffffffffu, s, 8);
        s += __shfl_xor_sync(0xffffffffu, s, 16);
        __syncthreads();
        if (lane < NR_TC) red[wid][lane] = s;
        __syncthreads();
        double t = 0.0;
        if (threadIdx.x < NR_TC) {
#pragma unroll
            for (int q = 0; q < NW; q++) t += red[q][threadIdx.x];
        }
        return t;  // valid on threads < NR_TC (thread = column of the tile)
    };
    // pass 1: mean_j = sum_i gmean_i x_ij  (gmean = w / n; nullptr: no centring, cox)
    double mean = 0.0;
    if (gmean) {
        const double t = column_sum([&](double v, int i, double s) { return fma(v, gmean[i], s); });
        if (threadIdx.x < NR_TC) {
            cmean[threadIdx.x] = t;
            if (live) mean_out[j] = t;
        }
        __syncthreads();
        mean = cmean[c];
    }
    // pass 2: h_j = sum_i wnorm_i (x_ij - mean_j)^2
    {
        const double t = column_sum([&](double v, int i, double s) {
            const double d = v - mean;
            return fma(d * d, wnorm[i], s);
        });
        if (threadIdx.x < NR_TC) {
            const double nx = sqrt(t);
            cmul[threadIdx.x] = sn / nx;
            if (live) norm_out[j] = nx;
        }
        __syncthreads();
    }
    // pass 3: x_ij <- (x_ij - mean_j) * mul_j * rowmul_i
    const double mul = cmul[c];
    for (int i0 = ifirst; i0 < n; i0 += 8 * RS) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; u++) v[u] = (live && i0 + u * RS < n) ? ld(i0 + u * RS) : 0.0;
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (live && i0 + u * RS < n) {
                const double rm = rowmul ? rowmul[i0 + u * RS] : 1.0;
                st(i0 + u * RS, (v[u] - mean) * mul * rm);
            }
    }
}
__global__ void __launch_bounds__(NR_NT) normalize_resident_kernel(double *X, long long ldx, int n, int p, const double *gmean,
                                                                   const double *wnorm, const double *rowmul, double sn,
                                                                   double *mean_out, double *norm_out)
{
    const long long j = (long long)blockIdx.x * NR_TC + (threadIdx.x & (NR_TC - 1));
    double *col = X + (j < p ? j : 0);
    normalize_tile([&](int i) { return col[(size_t)i * ldx]; }, [&](int i, double v) { col[(size_t)i * ldx] = v; }, n, p,
                   gmean, wnorm, rowmul, sn, mean_out, norm_out);
}
void launch_normalize_resident(double *X, long long ldx, int n, int p, const double *gmean, const double *wnorm,
                               const double *rowmul, double sn, double *mean_out, double *norm_out, cudaStream_t st)
{
    normalize_resident_kernel<<<(p + NR_TC - 1) / NR_TC, NR_NT, 0, st>>>(X, ldx, n, p, gmean, wnorm, rowmul, sn, mean_out, norm_out);
    CUDA_CHECK(cudaGetLastError());
}

// Screening's gather fused into the one-launch normalisation: the CTA of tile b copies the n x NR_TC slab of its kept
// columns cols[8b .. 8b+8) from the RAW design into shared memory, runs the three passes over the slab and writes Xn
// once.  Every element is its own 32-byte sector of a multi-GB design, so the copy is latency-bound: it goes global ->
// shared by cp.async, with no register round trip, and all n x 8 copies of the CTA are in flight at once.  The raw
// sectors are read with an L2 evict-first policy so that they do not push the screened design, which the path reads
// next, out of L2.  Replaces gather_cols (one write of Xn) + normalize_resident (three reads and one write of Xn).
__global__ void __launch_bounds__(NR_NT) gather_normalize_kernel(const double *__restrict__ X, long long ldx,
                                                                 const int *__restrict__ cols, double *Xn, long long ldn,
                                                                 int n, int p, const double *gmean, const double *wnorm,
                                                                 const double *rowmul, double sn, double *mean_out,
                                                                 double *norm_out)
{
    extern __shared__ __align__(16) double slab[];  // [n][NR_TC]
    {
        constexpr int RR = NR_NT / NR_TC;  // rows per round of the copy
        const int tc = threadIdx.x & (NR_TC - 1), tr = threadIdx.x / NR_TC;
        const long long jt = (long long)blockIdx.x * NR_TC + tc;
        if (jt < p) {
            const double *src = X + cols[jt];
            unsigned long long pol;
            asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(pol));
            for (int i = tr; i < n; i += RR) {
                const unsigned dst = (unsigned)__cvta_generic_to_shared(slab + i * NR_TC + tc);
                asm volatile("cp.async.ca.shared.global.L2::cache_hint [%0], [%1], 8, %2;" ::"r"(dst),
                             "l"(src + (size_t)i * ldx), "l"(pol)
                             : "memory");
            }
            asm volatile("cp.async.wait_all;" ::: "memory");
        } else {
            for (int i = tr; i < n; i += RR) slab[i * NR_TC + tc] = 0.0;
        }
        __syncthreads();
    }
    const int c = threadIdx.x & (NR_TC - 1);
    const long long j = (long long)blockIdx.x * NR_TC + c;
    double *out = Xn + (j < p ? j : 0);
    normalize_tile([&](int i) { return slab[i * NR_TC + c]; }, [&](int i, double v) { out[(size_t)i * ldn] = v; }, n, p,
                   gmean, wnorm, rowmul, sn, mean_out, norm_out);
}
void launch_gather_normalize(const double *X, long long ldx, const int *cols, double *Xn, long long ldn, int n, int p,
                             const double *gmean, const double *wnorm, const double *rowmul, double sn, double *mean_out,
                             double *norm_out, cudaStream_t st)
{
    if (n > NR_SLAB_ROWS) throw EngineError{"gather_normalize: the n x 8 slab does not fit shared memory"};
    gather_normalize_kernel<<<(p + NR_TC - 1) / NR_TC, NR_NT, (size_t)n * NR_TC * 8, st>>>(X, ldx, cols, Xn, ldn, n, p, gmean,
                                                                                         wnorm, rowmul, sn, mean_out, norm_out);
    CUDA_CHECK(cudaGetLastError());
}

void launch_center_scale(double *X, long long ldx, int n, int p, const double *sub, const double *mul,
                         const double *rowmul, cudaStream_t st)
{
    dim3 grid((unsigned)(((long long)(p + 1) / 2 + 127) / 128), (unsigned)((n + 63) / 64));
    center_scale_kernel<<<grid, 128, 0, st>>>(X, ldx, n, p, sub, mul, rowmul);
    CUDA_CHECK(cudaGetLastError());
}

// Xn[i][jn] = X[i][cols[jn]]   (screening.cpp:83-88)
__global__ void gather_cols_kernel(const double *X, long long ldx, int n, const int *cols, int pnew, double *Xn,
                                   long long ldn)
{
    const int jn = blockIdx.x * blockDim.x + threadIdx.x;
    if (jn >= pnew) return;
    const int src = cols[jn];
    const int r0 = blockIdx.y * 32, r1 = min(n, r0 + 32);
    // every element is its own 32-byte sector somewhere in a multi-GB design: what matters is how many of these reads are
    // in flight, so a thread issues eight before it stores any
    for (int i0 = r0; i0 < r1; i0 += 8) {
        double v[8];
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (i0 + u < r1) v[u] = __ldg(X + (size_t)(i0 + u) * ldx + src);
#pragma unroll
        for (int u = 0; u < 8; u++)
            if (i0 + u < r1) Xn[(size_t)(i0 + u) * ldn + jn] = v[u];
    }
}
void launch_gather_cols(const double *X, long long ldx, int n, const int *cols, int pnew, double *Xn, long long ldn,
                        cudaStream_t st)
{
    dim3 grid((pnew + 127) / 128, (n + 31) / 32);
    gather_cols_kernel<<<grid, 128, 0, st>>>(X, ldx, n, cols, pnew, Xn, ldn);
    CUDA_CHECK(cudaGetLastError());
}

__global__ void gather_cols_pos_kernel(const double *X, long long ldx, int n, const int *cols, const int *pos, int m,
                                       double *dst, long long ld)
{
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const int src = cols[q], dp = pos[q];
    const int r0 = blockIdx.y * 32, r1 = min(n, r0 + 32);
    for (int i = r0; i < r1; i++) dst[(size_t)i * ld + dp] = X[(size_t)i * ldx + src];
}
void launch_gather_cols_pos(const double *X, long long ldx, int n, const int *cols, const int *pos, int m, double *dst,
                            long long ld, cudaStream_t st)
{
    dim3 grid((m + 127) / 128, (n + 31) / 32);
    gather_cols_pos_kernel<<<grid, 128, 0, st>>>(X, ldx, n, cols, pos, m, dst, ld);
    CUDA_CHECK(cudaGetLastError());
}

// Marginal GLM utilities for screening (screening.cpp:48-61): one thread per column, the column is re-read from
// L2/HBM each Newton/IRLS step (coalesced across the warp because X is row-major).
//   binomial: logit_fit, logistic.cpp:61-157 (2-parameter IRLS, no W floor, returns the previous iterate)
//   poisson : poisson_fit, poisson.cpp:84-137, restated LITERALLY incl. the vector*vector product that evaluates to
//             X.col(i)*expeta_w(0) with asserts off (:117) and the wrong-sign step (:122,:128)
//   cox     : cox_fit, coxph.cpp:42-109 (1-parameter damped Newton, clamp +-50)
__device__ __forceinline__ void solve2(double a, double b, double c, double r0, double r1, double &x0, double &x1)
{
    // [[a b][b c]] x = r  (2x2 symmetric)
    const double det = a * c - b * b;
    x0 = (c * r0 - b * r1) / det;
    x1 = (a * r1 - b * r0) / det;
}

// Column readers of screen_glm_kernel.  start(rev) begins a pass over the rows (ascending, or descending when rev); at(i)
// then returns x[i][j] for the rows of that pass in order.  The dense reader is the strided load of a row-major design;
// the CSC reader walks the column's stored entries with a cursor and returns 0.0 for absent rows, so both feed the same
// arithmetic the same values in the same order.
struct DenseColumn {
    const double *__restrict__ xc;
    long long ldx;
    static __device__ __forceinline__ DenseColumn make(const double *X, long long ldx, const long long *, const int *, int j)
    {
        return DenseColumn{X + j, ldx};
    }
    __device__ __forceinline__ void start(bool) {}
    __device__ __forceinline__ double at(int i) { return __ldg(xc + (size_t)i * ldx); }
};
struct CscColumn {
    const int *ri;
    const double *v;
    long long b, e, k;
    int next;  // row of entry k, -1 once the pass has used every entry
    int step;
    // values = the CSC value array (passed where the dense reader takes X)
    static __device__ __forceinline__ CscColumn make(const double *values, long long, const long long *colptr,
                                                     const int *rowidx, int j)
    {
        CscColumn c;
        c.ri = rowidx;
        c.v = values;
        c.b = __ldg(colptr + j);
        c.e = __ldg(colptr + j + 1);
        c.k = c.b;
        c.next = -1;
        c.step = 1;
        return c;
    }
    __device__ __forceinline__ void start(bool rev)
    {
        step = rev ? -1 : 1;
        k = rev ? e - 1 : b;
        next = (k >= b && k < e) ? __ldg(ri + k) : -1;
    }
    __device__ __forceinline__ double at(int i)
    {
        if (i != next) return 0.0;
        const double x = __ldg(v + k);
        k += step;
        next = (k >= b && k < e) ? __ldg(ri + k) : -1;
        return x;
    }
};

template <class Column>
__global__ void __launch_bounds__(128) screen_glm_kernel(const double *__restrict__ X, long long ldx,
                                                         const long long *__restrict__ colptr, const int *__restrict__ rowidx,
                                                         int n, int p, const double *__restrict__ y,
                                                         const double *__restrict__ w, int family, double *util)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *ys = reinterpret_cast<double *>(smem_raw);
    double *ws = ys + n;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        ys[i] = y[i];
        ws[i] = w[i];
    }
    __syncthreads();
    const int j = blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= p) return;
    Column xc = Column::make(X, ldx, colptr, rowidx, j);
    if (family == FAM_LOGIT) {
        double b00 = 0.0, b01 = 0.0;  // beta0
        double b10, b11;              // beta1
        // step 0 at beta0 = 0: Pi = 0.5
        double ll0 = 0.0, s00 = 0, s01 = 0, s11 = 0, r0 = 0, r1 = 0;
        xc.start(false);
        for (int i = 0; i < n; i++) {
            const double x = xc.at(i);
            const double pi = 0.5;
            ll0 += (ys[i] * log(pi) + (1.0 - ys[i]) * log(1.0 - pi)) * ws[i];
            const double W = pi * (1.0 - pi);
            const double Z = (ys[i] - pi) / W;
            const double ww = W * ws[i];
            s00 += ww; s01 += ww * x; s11 += ww * x * x; r0 += ww * Z; r1 += ww * x * Z;
        }
        solve2(s00, s01, s11, r0, r1, b10, b11);
        for (int it = 0; it < 30; it++) {
            double ll1 = 0.0;
            s00 = s01 = s11 = r0 = r1 = 0.0;
            xc.start(false);
            for (int i = 0; i < n; i++) {
                const double x = xc.at(i);
                const double eu = b10 + b11 * x;
                const double e = exp(clampd(eu, 30.0));
                const double pi = e / (1.0 + e);
                ll1 += (ys[i] * log(pi) + (1.0 - ys[i]) * log(1.0 - pi)) * ws[i];
                const double W = pi * (1.0 - pi);
                const double Z = eu + (ys[i] - pi) / W;
                const double ww = W * ws[i];
                s00 += ww; s01 += ww * x; s11 += ww * x * x; r0 += ww * Z; r1 += ww * x * Z;
            }
            if (fabs(ll0 - ll1) / (0.1 + fabs(ll1)) < 1e-6) break;
            b00 = b10; b01 = b11; ll0 = ll1;
            solve2(s00, s01, s11, r0, r1, b10, b11);
        }
        (void)b00;
        util[j] = b01 * b01;
    } else if (family == FAM_POISSON) {
        double b0 = 0.0, b1 = 0.0;
        for (int it = 0; it < 100; it++) {
            double g0 = 0, g1 = 0, h00 = 0, h01 = 0, h11 = 0, ll0 = 0, ew0 = 0;
            xc.start(false);
            for (int i = 0; i < n; i++) {
                const double x = xc.at(i);
                const double eta = clampd(b0 + b1 * x, 30.0);
                const double e = exp(eta);
                if (i == 0) ew0 = e * ws[0];
                const double r = (ys[i] - e) * ws[i];
                g0 += r; g1 += x * r;
                h00 += 1.0; h01 += x; h11 += x * x;  // scaled by ew0 below (poisson.cpp:117 as evaluated)
                ll0 += (ys[i] * eta - e) * ws[i];
            }
            h00 *= ew0; h01 *= ew0; h11 *= ew0;
            double d0, d1;
            solve2(h00, h01, h11, g0, g1, d0, d1);
            int m = 0;
            double step = 1.0;
            double n0 = b0 - d0, n1 = b1 - d1, ll1 = 0.0;
            for (;;) {
                ll1 = 0.0;
                xc.start(false);
                for (int i = 0; i < n; i++) {
                    const double x = xc.at(i);
                    const double eta = clampd(n0 + n1 * x, 30.0);
                    ll1 += (ys[i] * eta - exp(eta)) * ws[i];
                }
                if (!(ll0 >= ll1 && m < 10)) break;
                m++;
                step *= 0.2;
                n0 = b0 - step * d0;
                n1 = b1 - step * d1;
            }
            b0 = n0; b1 = n1;
            if (fabs(ll0 - ll1) / fabs(ll0) < 1e-8) break;
        }
        util[j] = b1 * b1;
    } else {  // cox, one parameter
        double b0 = 0.0, ll0 = 1e5;
        for (int l = 1; l <= 30; l++) {
            // one backward pass: S0, S1, S2 running suffix sums
            double S0 = 0, S1 = 0, S2 = 0, g = 0, hneg = 0;
            xc.start(true);
            for (int i = n - 1; i >= 0; i--) {
                const double x = xc.at(i);
                const double th = exp(clampd(b0 * x, 50.0));
                S0 += th; S1 += th * x; S2 += th * x * x;
                const double e = ws[i] * ys[i];
                const double xb = S1 / S0;
                g += (x - xb) * e;
                hneg += (S2 / S0 - xb * xb) * e;  // = -h
            }
            const double d = -g / hneg;  // h d = g
            int m = 1;
            double step = 0.5;
            double b1 = b0 - step * d, ll1;
            for (;;) {
                double S = 0, acc = 0;
                xc.start(true);
                for (int i = n - 1; i >= 0; i--) {
                    const double x = xc.at(i);
                    const double th = exp(clampd(b1 * x, 30.0));
                    S += th;
                    acc += log(th / S) * ys[i] * ws[i];
                }
                ll1 = acc;
                if (!(ll0 > ll1 && m < 5)) break;
                m++;
                step *= 0.5;
                b1 = b0 - step * d;
            }
            if (fabs(ll0 - ll1) / fabs(0.1 + ll0) < 1e-5) break;
            b0 = b1;
            ll0 = ll1;
        }
        util[j] = b0 * b0;
    }
}
void launch_screen_glm(const double *X, long long ldx, int n, int p, const double *y, const double *w, int family,
                       double *util, cudaStream_t st)
{
    const size_t smem = (size_t)2 * n * sizeof(double);
    CUDA_CHECK(cudaFuncSetAttribute(screen_glm_kernel<DenseColumn>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    screen_glm_kernel<DenseColumn><<<(p + 127) / 128, 128, smem, st>>>(X, ldx, nullptr, nullptr, n, p, y, w, family, util);
    CUDA_CHECK(cudaGetLastError());
}
void launch_screen_glm_csc(const long long *colptr, const int *rowidx, const double *values, int n, int p, const double *y,
                           const double *w, int family, double *util, cudaStream_t st)
{
    const size_t smem = (size_t)2 * n * sizeof(double);
    CUDA_CHECK(cudaFuncSetAttribute(screen_glm_kernel<CscColumn>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    screen_glm_kernel<CscColumn><<<(p + 127) / 128, 128, smem, st>>>(values, 0, colptr, rowidx, n, p, y, w, family, util);
    CUDA_CHECK(cudaGetLastError());
}

// ---- sparse (CSC) designs.  A warp (or, for the gaussian utility, a sub-warp sized to the mean column length) owns a
// column and walks its stored entries; offsets into rowidx / values are 64-bit.
static unsigned csc_grid(long long items_per_block, long long count)
{
    return (unsigned)std::max<long long>(1, std::min<long long>((count + items_per_block - 1) / items_per_block, 148LL * 64));
}

// Validation of the caller's arrays: colptr[0] == 0, non-decreasing, colptr[p] == nnz; rows in [0, n) and strictly
// increasing inside every column.  A column whose offsets are out of range is flagged and not read.
__global__ void __launch_bounds__(256) csc_check_kernel(const long long *__restrict__ colptr, const int *__restrict__ rowidx,
                                                        int n, int p, long long nnz, int *flag)
{
    const int lane = threadIdx.x & 31;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    int bad = 0;
    for (long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < p; j += nw) {
        const long long b = __ldg(colptr + j), e = __ldg(colptr + j + 1);
        if (b < 0 || e < b || e > nnz || (j == 0 && b != 0) || (j == p - 1 && e != nnz)) {
            bad |= CSC_BAD_COLPTR;
            continue;
        }
        for (long long k = b + lane; k < e; k += 32) {
            const int r = __ldg(rowidx + k);
            if (r < 0 || r >= n) bad |= CSC_BAD_ROW;
            if (k > b && __ldg(rowidx + k - 1) >= r) bad |= CSC_UNSORTED;
        }
    }
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (lane == 0 && bad) atomicOr(flag, bad);
}
void launch_csc_check(const long long *colptr, const int *rowidx, int n, int p, long long nnz, int *flag, cudaStream_t st)
{
    csc_check_kernel<<<csc_grid(8, p), 256, 0, st>>>(colptr, rowidx, n, p, nnz, flag);
    CUDA_CHECK(cudaGetLastError());
}

// Xn[rowidx[k]][q] = values[k] over the entries of column cols[q] (the columns screening keeps, or all of them)
__global__ void __launch_bounds__(256) csc_densify_kernel(const long long *__restrict__ colptr, const int *__restrict__ rowidx,
                                                          const double *__restrict__ values, const int *__restrict__ cols,
                                                          int m, double *Xn, long long ldn)
{
    const int lane = threadIdx.x & 31;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long q = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; q < m; q += nw) {
        const int j = cols ? __ldg(cols + q) : (int)q;
        const long long b = __ldg(colptr + j), e = __ldg(colptr + j + 1);
        for (long long k = b + lane; k < e; k += 32) Xn[(size_t)__ldg(rowidx + k) * ldn + q] = __ldg(values + k);
    }
}
void launch_csc_densify(const long long *colptr, const int *rowidx, const double *values, const int *cols, int m, double *Xn,
                        long long ldn, cudaStream_t st)
{
    if (m <= 0) return;
    csc_densify_kernel<<<csc_grid(8, m), 256, 0, st>>>(colptr, rowidx, values, cols, m, Xn, ldn);
    CUDA_CHECK(cudaGetLastError());
}

// One-column least squares on the raw column (screening.cpp:46), (x_j.y / x_j.x_j)^2, over the non-zeros only: G lanes per
// column, G the power of two nearest below the mean column length.  An all-zero column gives 0 / 0 as in the dense sweep.
template <int G>
__global__ void __launch_bounds__(256) screen_csc_lm_kernel(const long long *__restrict__ colptr,
                                                            const int *__restrict__ rowidx,
                                                            const double *__restrict__ values, int p,
                                                            const double *__restrict__ y, double *util)
{
    const int lane = threadIdx.x % G;
    const long long per_pass = ((long long)gridDim.x * blockDim.x) / G;
    for (long long j0 = ((long long)blockIdx.x * blockDim.x) / G; j0 < p; j0 += per_pass) {
        const long long j = j0 + threadIdx.x / G;
        double ds = 0.0, hs = 0.0;
        if (j < p) {
            const long long b = __ldg(colptr + j), e = __ldg(colptr + j + 1);
            for (long long k = b + lane; k < e; k += G) {
                const double x = __ldg(values + k);
                ds = fma(x, __ldg(y + __ldg(rowidx + k)), ds);
                hs = fma(x, x, hs);
            }
        }
#pragma unroll
        for (int o = G / 2; o > 0; o >>= 1) {
            ds += __shfl_xor_sync(0xffffffffu, ds, o, G);
            hs += __shfl_xor_sync(0xffffffffu, hs, o, G);
        }
        if (j < p && lane == 0) {
            const double bq = ds / hs;
            util[j] = bq * bq;
        }
    }
}
void launch_screen_csc_lm(const long long *colptr, const int *rowidx, const double *values, int p, long long nnz,
                          const double *y, double *util, cudaStream_t st)
{
    const double mean = (double)nnz / (double)p;
    int g = 1;
    while (g < 32 && 2 * g <= mean) g *= 2;
    const unsigned grid = csc_grid(256 / g, p);
    switch (g) {
        case 1: screen_csc_lm_kernel<1><<<grid, 256, 0, st>>>(colptr, rowidx, values, p, y, util); break;
        case 2: screen_csc_lm_kernel<2><<<grid, 256, 0, st>>>(colptr, rowidx, values, p, y, util); break;
        case 4: screen_csc_lm_kernel<4><<<grid, 256, 0, st>>>(colptr, rowidx, values, p, y, util); break;
        case 8: screen_csc_lm_kernel<8><<<grid, 256, 0, st>>>(colptr, rowidx, values, p, y, util); break;
        case 16: screen_csc_lm_kernel<16><<<grid, 256, 0, st>>>(colptr, rowidx, values, p, y, util); break;
        default: screen_csc_lm_kernel<32><<<grid, 256, 0, st>>>(colptr, rowidx, values, p, y, util); break;
    }
    CUDA_CHECK(cudaGetLastError());
}

// ---- sparse design swept on its non-zeros (Dev::ccp).  The design stays in CSC form; the centring and scaling of
// normalize.cpp are applied implicitly, with the unstored rows' terms summed in closed form.  Every sum is a per-lane
// sequential sum followed by a fixed shuffle tree: a call is bitwise reproducible.

// mask of the G-lane group of this thread inside its warp (sub-warp shuffles of groups that loop independently)
template <int G>
__device__ __forceinline__ unsigned group_mask()
{
    if constexpr (G == 32) return 0xffffffffu;
    else return ((1u << G) - 1u) << ((threadIdx.x & 31) & ~(G - 1));
}
template <int G>
__device__ __forceinline__ double group_sum(double v, unsigned mask)
{
#pragma unroll
    for (int o = G / 2; o > 0; o >>= 1) v += __shfl_xor_sync(mask, v, o, G);
    return v;
}

__global__ void __launch_bounds__(256) csc_stats_kernel(const long long *__restrict__ colptr, const int *__restrict__ rowidx,
                                                        const double *__restrict__ values, int p, const double *g,
                                                        const double *w, double sumw, double sn, double *mean_out,
                                                        double *norm_out, double *mul_out)
{
    const int lane = threadIdx.x & 31;
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < p; j += nw) {
        const long long b = __ldg(colptr + j), e = __ldg(colptr + j + 1);
        double m = 0.0;
        if (g) {
            for (long long k = b + lane; k < e; k += 32) m = fma(__ldg(values + k), __ldg(g + __ldg(rowidx + k)), m);
            m = warp_sum(m);
        }
        double h = 0.0, ws = 0.0;
        for (long long k = b + lane; k < e; k += 32) {
            const double wi = __ldg(w + __ldg(rowidx + k));
            const double xc = __ldg(values + k) - m;
            h = fma(xc * xc, wi, h);
            ws += wi;
        }
        h = warp_sum(h);
        ws = warp_sum(ws);
        h += m * m * (sumw - ws);
        if (lane == 0) {
            const double nx = sqrt(h);
            mean_out[j] = m;
            norm_out[j] = nx;
            mul_out[j] = sn / nx;
        }
    }
}
void launch_csc_stats(const long long *colptr, const int *rowidx, const double *values, int p, const double *g,
                      const double *w, double sumw, double sn, double *mean_out, double *norm_out, double *mul_out,
                      cudaStream_t st)
{
    csc_stats_kernel<<<csc_grid(8, p), 256, 0, st>>>(colptr, rowidx, values, p, g, w, sumw, sn, mean_out, norm_out, mul_out);
    CUDA_CHECK(cudaGetLastError());
}

// The per-iteration sums the implicit centring needs, one CTA per chain slot: csum[0][f] = sum_i G'_i[f], csum[1][f] =
// sum_i W_i[f] (gaussian / GLM); cox (no centring): cpre[i][f] = sum_{k <= i} C2_k[f], c2sum[f] = its total.  Each thread
// owns a contiguous row chunk, so the order of every sum is fixed.
constexpr int CSUM_NT = 512;
__global__ void __launch_bounds__(CSUM_NT) csc_sums_kernel(const Dev d, int mode)
{
    __shared__ double red[40];
    if (d.gate && *d.gate == 0) return;
    const int f = blockIdx.x, FS = d.FS, n = d.n;
    const int per = (n + CSUM_NT - 1) / CSUM_NT;
    const int r0 = min(n, (int)threadIdx.x * per), r1 = min(n, r0 + per);
    if (mode == MODE_COX) {
        double s = 0.0;
        for (int i = r0; i < r1; i++) s += d.C2[(size_t)i * FS + f];
        double tot;
        double run = block_excl_scan<CSUM_NT>(s, red, &tot);
        for (int i = r0; i < r1; i++) {
            run += d.C2[(size_t)i * FS + f];
            d.cpre[(size_t)i * FS + f] = run;
        }
        if (threadIdx.x == 0) d.c2sum[f] = tot;
        return;
    }
    const double *rm = mode == MODE_D ? d.crm : nullptr;
    double sg = 0.0, sw = 0.0;
    for (int i = r0; i < r1; i++) {
        const double gi = d.G[(size_t)i * FS + f];
        sg += rm ? rm[i] * gi : gi;
        if (mode == MODE_DH) sw += d.W[(size_t)i * FS + f];
    }
    sg = block_sum<CSUM_NT>(sg, red);
    sw = block_sum<CSUM_NT>(sw, red);
    if (threadIdx.x == 0) {
        d.csum[f] = sg;
        d.csum[FS + f] = sw;
    }
}

// The dual sweep over the CSC arrays.  With x~ = (x - m) mul rm and G' = rm o G, per column j and chain slot f:
//   MODE_D   d = mul (sum_stored x G' - m sum_i G'_i)
//   MODE_DH  d as in MODE_D (rm = 1), h = mul^2 (sum_stored (x - m)^2 W + m^2 (sum_i W_i - sum_stored W))
//   MODE_COX (m = 0) d, h as above; s1 = mul sum_stored TH x; R = mul^2 sum_t (P_{i_t} - P_{i_{t-1}}) S_t^2 with S_t the
//            suffix of TH x over the column's entries from t and P the row prefix of C2 (s1_k is constant between stored
//            rows); B = mul sum_t (P_{i_t} - P_{i_{t-1}}) S_t
// The partials land where dual_sweep_kernel writes them with S = 1: part[(q * FT + f) * pstride + j].
// Work split: columns of at most Dev::clong_thr entries are walked by G lanes each (csc_sweep_kernel, G from the mean
// column length); longer ones -- the frequent terms of a power-law design -- by a whole CTA each (csc_sweep_long_kernel),
// its warps owning fixed consecutive segments whose sums are combined in a fixed order.
template <int FT, int MODE>
__host__ __device__ constexpr int csc_fc() { return MODE == MODE_COX ? (FT < 4 ? FT : 4) : (FT < 8 ? FT : 8); }

// The sums of the entries [k0, k1) of a column that starts at entry b (the Cox dP of entry k reads row k - 1 when k > b),
// for chain slots fb .. fb + FC - 1, by the G lanes of `mask`.  Cox: the entries are walked in chunks of G from k1 down,
// carry[f] enters as the suffix of the entries after k1 and leaves as the suffix from k0.  Per-lane partials: the caller
// reduces them.
template <int FT, int MODE, int G>
__device__ __forceinline__ void csc_range(const Dev &d, long long b, long long k0, long long k1, int fb, double mj, int lane,
                                          unsigned mask, double (&ad)[csc_fc<FT, MODE>()], double (&ah)[csc_fc<FT, MODE>()],
                                          double (&aw)[csc_fc<FT, MODE>()], double (&aR)[csc_fc<FT, MODE>()],
                                          double (&aB)[csc_fc<FT, MODE>()], double (&carry)[csc_fc<FT, MODE>()])
{
    constexpr int FC = csc_fc<FT, MODE>();
    const double *rm = MODE == MODE_D ? d.crm : nullptr;
    if constexpr (MODE != MODE_COX) {
        for (long long k = k0 + lane; k < k1; k += G) {
            const int i = __ldg(d.cri + k);
            const double x = __ldg(d.ccv + k);
            const double r = rm ? __ldg(rm + i) : 1.0;
            const double xc = x - mj;
#pragma unroll
            for (int f = 0; f < FC; f++) {
                if (fb + f < FT) {
                    const double gi = __ldg(d.G + (size_t)i * FT + fb + f);
                    ad[f] = fma(x, rm ? r * gi : gi, ad[f]);
                    if constexpr (MODE == MODE_DH) {
                        const double wi = __ldg(d.W + (size_t)i * FT + fb + f);
                        ah[f] = fma(xc * xc, wi, ah[f]);
                        aw[f] += wi;
                    }
                }
            }
        }
    } else {
        const long long nck = (k1 - k0 + G - 1) / G;
        for (long long q = nck - 1; q >= 0; q--) {
            const long long k = k0 + q * G + lane;
            const bool valid = k < k1;
            const int i = valid ? __ldg(d.cri + k) : 0;
            const int ip = (valid && k > b) ? __ldg(d.cri + k - 1) : -1;
            const double x = valid ? __ldg(d.ccv + k) : 0.0;
#pragma unroll
            for (int f = 0; f < FC; f++) {
                if (fb + f < FT) {
                    const size_t o = (size_t)i * FT + fb + f;
                    const double v = valid ? x * __ldg(d.TH + o) : 0.0;
                    double s = v;
#pragma unroll
                    for (int sh = 1; sh < G; sh <<= 1) {
                        const double t = __shfl_down_sync(mask, s, sh, G);
                        if (lane + sh < G) s += t;
                    }
                    const double S = s + carry[f];
                    carry[f] += __shfl_sync(mask, s, 0, G);
                    if (valid) {
                        const double dP = d.cpre[o] - (ip >= 0 ? d.cpre[(size_t)ip * FT + fb + f] : 0.0);
                        aR[f] = fma(dP * S, S, aR[f]);
                        aB[f] = fma(dP, S, aB[f]);
                        ad[f] = fma(x, __ldg(d.G + o), ad[f]);
                        ah[f] = fma(x * x, __ldg(d.W + o), ah[f]);
                    }
                }
            }
        }
    }
}

// the partials of column j, slot ff from its reduced sums
template <int FT, int MODE>
__device__ __forceinline__ void csc_put(const Dev &d, long long j, int ff, double mj, double mu, double ad, double ah,
                                        double aw, double aR, double aB, double s1)
{
    auto put = [&](int qq, double v) { d.part[((size_t)qq * FT + ff) * d.pstride + j] = v; };
    if constexpr (MODE == MODE_COX) {
        put(0, mu * ad);
        put(1, mu * mu * ah);
        put(2, mu * s1);
        put(3, mu * mu * aR);
        put(4, mu * aB);
    } else {
        put(0, mu * (ad - mj * d.csum[ff]));
        if constexpr (MODE == MODE_DH) put(1, mu * mu * (ah + mj * mj * (d.csum[FT + ff] - aw)));
    }
}

template <int FT, int MODE, int G>
__global__ void __launch_bounds__(256, 1) csc_sweep_kernel(const Dev d)
{
    constexpr int FC = csc_fc<FT, MODE>();
    if (d.gate && *d.gate == 0) return;
    const int lane = threadIdx.x & (G - 1);
    const unsigned mask = group_mask<G>();
    const long long per_pass = ((long long)gridDim.x * blockDim.x) / G;
    for (long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) / G; j < d.p; j += per_pass) {
        const long long b = __ldg(d.ccp + j), e = __ldg(d.ccp + j + 1);
        if (e - b > d.clong_thr) continue;  // csc_sweep_long_kernel's column
        const double mj = MODE == MODE_COX ? 0.0 : d.cmean[j];
        const double mu = d.cmul[j];
#pragma unroll 1
        for (int fb = 0; fb < FT; fb += FC) {
            double ad[FC], ah[FC], aw[FC], aR[FC], aB[FC], carry[FC];
#pragma unroll
            for (int f = 0; f < FC; f++) ad[f] = ah[f] = aw[f] = aR[f] = aB[f] = carry[f] = 0.0;
            csc_range<FT, MODE, G>(d, b, b, e, fb, mj, lane, mask, ad, ah, aw, aR, aB, carry);
#pragma unroll
            for (int f = 0; f < FC; f++) {
                if (fb + f >= FT) continue;
                ad[f] = group_sum<G>(ad[f], mask);
                if constexpr (MODE >= MODE_DH) ah[f] = group_sum<G>(ah[f], mask);
                if constexpr (MODE == MODE_DH) aw[f] = group_sum<G>(aw[f], mask);
                if constexpr (MODE == MODE_COX) {
                    aR[f] = group_sum<G>(aR[f], mask);
                    aB[f] = group_sum<G>(aB[f], mask);
                }
                if (lane == 0) csc_put<FT, MODE>(d, j, fb + f, mj, mu, ad[f], ah[f], aw[f], aR[f], aB[f], carry[f]);
            }
        }
    }
}

// One CTA per long column (Dev::clong): warp w owns the entries [b + w seg, b + (w + 1) seg).  The warps' sums are added
// in warp order; for Cox a first pass gives every segment's suffix total, so that each warp starts its scan with the
// suffix of the segments after it (added from the last segment down).
constexpr int CSC_LONG_NT = 256;
template <int FT, int MODE>
__global__ void __launch_bounds__(CSC_LONG_NT, 1) csc_sweep_long_kernel(const Dev d)
{
    constexpr int FC = csc_fc<FT, MODE>();
    constexpr int NW = CSC_LONG_NT / 32;
    __shared__ double red[4][FC][NW];
    __shared__ double cin[FC][NW];
    if (d.gate && *d.gate == 0) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const long long j = d.clong[blockIdx.x];
    const long long b = __ldg(d.ccp + j), e = __ldg(d.ccp + j + 1);
    const long long seg = (e - b + NW - 1) / NW;
    const long long k0 = min(e, b + wid * seg), k1 = min(e, k0 + seg);
    const double mj = MODE == MODE_COX ? 0.0 : d.cmean[j];
    const double mu = d.cmul[j];
#pragma unroll 1
    for (int fb = 0; fb < FT; fb += FC) {
        double ad[FC], ah[FC], aw[FC], aR[FC], aB[FC], carry[FC];
#pragma unroll
        for (int f = 0; f < FC; f++) ad[f] = ah[f] = aw[f] = aR[f] = aB[f] = carry[f] = 0.0;
        if constexpr (MODE == MODE_COX) {
            // pass 1: the segment's own suffix total
            csc_range<FT, MODE, 32>(d, b, k0, k1, fb, mj, lane, 0xffffffffu, ad, ah, aw, aR, aB, carry);
            if (lane == 0)
#pragma unroll
                for (int f = 0; f < FC; f++) cin[f][wid] = carry[f];
            __syncthreads();
#pragma unroll
            for (int f = 0; f < FC; f++) {
                double c = 0.0;
                for (int w2 = NW - 1; w2 > wid; w2--) c += cin[f][w2];
                ad[f] = ah[f] = aR[f] = aB[f] = 0.0;
                carry[f] = c;
            }
            __syncthreads();
        }
        csc_range<FT, MODE, 32>(d, b, k0, k1, fb, mj, lane, 0xffffffffu, ad, ah, aw, aR, aB, carry);
#pragma unroll
        for (int f = 0; f < FC; f++) {
            if (fb + f >= FT) continue;
            const double v[4] = {warp_sum(ad[f]), warp_sum(ah[f]), warp_sum(MODE == MODE_COX ? aR[f] : aw[f]),
                                 warp_sum(aB[f])};
            if (lane == 0)
#pragma unroll
                for (int q = 0; q < 4; q++) red[q][f][wid] = v[q];
            if (MODE == MODE_COX && wid == 0 && lane == 0) cin[f][0] = carry[f];  // suffix from the column's first entry
        }
        __syncthreads();
        if (threadIdx.x < FC && fb + (int)threadIdx.x < FT) {
            const int f = threadIdx.x;
            double t[4] = {0.0, 0.0, 0.0, 0.0};
            for (int w2 = 0; w2 < NW; w2++)
#pragma unroll
                for (int q = 0; q < 4; q++) t[q] += red[q][f][w2];
            if constexpr (MODE == MODE_COX) csc_put<FT, MODE>(d, j, fb + f, mj, mu, t[0], t[1], 0.0, t[2], t[3], cin[f][0]);
            else csc_put<FT, MODE>(d, j, fb + f, mj, mu, t[0], t[1], t[2], 0.0, 0.0, 0.0);
        }
        __syncthreads();
    }
}

template <int FT, int MODE>
static void launch_csc_sweep_t(const Dev &d, cudaStream_t st)
{
    switch (d.csc_g) {
        case 2: csc_sweep_kernel<FT, MODE, 2><<<csc_grid(128, d.p), 256, 0, st>>>(d); break;
        case 8: csc_sweep_kernel<FT, MODE, 8><<<csc_grid(32, d.p), 256, 0, st>>>(d); break;
        default: csc_sweep_kernel<FT, MODE, 32><<<csc_grid(8, d.p), 256, 0, st>>>(d); break;
    }
    if (d.nlong > 0) csc_sweep_long_kernel<FT, MODE><<<d.nlong, CSC_LONG_NT, 0, st>>>(d);
}
template <int MODE>
static void launch_csc_sweep_m(const Dev &d, cudaStream_t st)
{
    switch (d.FS) {
        case 1: launch_csc_sweep_t<1, MODE>(d, st); break;
        case 2: launch_csc_sweep_t<2, MODE>(d, st); break;
        case 4: launch_csc_sweep_t<4, MODE>(d, st); break;
        case 6: launch_csc_sweep_t<6, MODE>(d, st); break;
        case 8: launch_csc_sweep_t<8, MODE>(d, st); break;
        case 12: launch_csc_sweep_t<12, MODE>(d, st); break;
        case 16: launch_csc_sweep_t<16, MODE>(d, st); break;
        case 24: launch_csc_sweep_t<24, MODE>(d, st); break;
        case 32: launch_csc_sweep_t<32, MODE>(d, st); break;
        default: throw EngineError{"csc sweep: unsupported chain tile FS=" + std::to_string(d.FS)};
    }
}
void launch_csc_sweep(const Dev &d, int mode, cudaStream_t st)
{
    csc_sums_kernel<<<d.FS, CSUM_NT, 0, st>>>(d, mode);
    CUDA_CHECK(cudaGetLastError());
    if (mode == MODE_D) launch_csc_sweep_m<MODE_D>(d, st);
    else if (mode == MODE_DH) launch_csc_sweep_m<MODE_DH>(d, st);
    else launch_csc_sweep_m<MODE_COX>(d, st);
    CUDA_CHECK(cudaGetLastError());
}

// the columns with more than thr entries (their order does not matter: each is summed by its own CTA)
__global__ void __launch_bounds__(256) csc_long_list_kernel(const long long *__restrict__ colptr, int p, long long thr,
                                                            int *list, int *count)
{
    for (long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x; j < p; j += (long long)gridDim.x * blockDim.x)
        if (__ldg(colptr + j + 1) - __ldg(colptr + j) > thr) list[atomicAdd(count, 1)] = (int)j;
}
void launch_csc_long_list(const long long *colptr, int p, long long thr, int *list, int *count, cudaStream_t st)
{
    csc_long_list_kernel<<<csc_grid(256, p), 256, 0, st>>>(colptr, p, thr, list, count);
    CUDA_CHECK(cudaGetLastError());
}

// column j of the implicit normalised design into out[i * ld] for all n rows: every row first gets the value of an unstored
// entry, then the stored rows theirs; per element the expression of center_scale_kernel's two passes, ((x - m) mul) rm
__device__ __forceinline__ void csc_column_out(const Dev &d, int j, double *out, long long ld, int lane)
{
    const double mj = d.cmean[j], mu = d.cmul[j];
    const double z = (0.0 - mj) * mu;
    for (int i = lane; i < d.n; i += 32) out[(size_t)i * ld] = z * (d.crm ? d.crm[i] : 1.0);
    __syncwarp();
    const long long b = __ldg(d.ccp + j), e = __ldg(d.ccp + j + 1);
    for (long long k = b + lane; k < e; k += 32) {
        const int i = __ldg(d.cri + k);
        out[(size_t)i * ld] = ((__ldg(d.ccv + k) - mj) * mu) * (d.crm ? d.crm[i] : 1.0);
    }
}
__global__ void __launch_bounds__(256) csc_gather_kernel(const Dev d, const BatchDesc b, int which)
{
    const int c = b.chain[blockIdx.y];
    if (which == 0) {
        if (d.gate && *d.gate == 0) return;
        if (d.done[c]) return;
    }
    const int cnt = which == 0 ? b.T : d.ks[c];
    const int a = blockIdx.x * 8 + (threadIdx.x >> 5);
    if (a >= cnt) return;
    const int j = (which == 0 ? d.Anew : d.A)[(size_t)c * d.kcap + a];
    const long long ld = which == 0 ? d.ldXr : d.ldXk;
    double *out = (which == 0 ? d.AXr : d.AXk) + (size_t)c * d.n * ld + a;
    csc_column_out(d, j, out, ld, threadIdx.x & 31);
}
void launch_csc_gather(const Dev &d, const BatchDesc &b, int which, cudaStream_t st)
{
    const int cols = which == 0 ? b.T : d.kcap;
    if (cols <= 0) return;
    dim3 grid((unsigned)((cols + 7) / 8), (unsigned)b.nch);
    csc_gather_kernel<<<grid, 256, 0, st>>>(d, b, which);
    CUDA_CHECK(cudaGetLastError());
}
__global__ void __launch_bounds__(256) csc_expand_kernel(const Dev d, double *out, long long ld)
{
    const long long nw = ((long long)gridDim.x * blockDim.x) >> 5;
    for (long long j = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5; j < d.p; j += nw)
        csc_column_out(d, (int)j, out + j, ld, threadIdx.x & 31);
}
void launch_csc_expand(const Dev &d, double *out, long long ld, cudaStream_t st)
{
    csc_expand_kernel<<<csc_grid(8, d.p), 256, 0, st>>>(d, out, ld);
    CUDA_CHECK(cudaGetLastError());
}

}  // namespace bess
