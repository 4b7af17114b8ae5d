// dual_sweep_tma_kernel -- the batched dual sweep (F >= 2 chains per pass over X) as a bulk-TMA pipeline.
//
//   d_j = sum_i x_ij g_if,   h_j = sum_i x_ij^2 w_if   (+ the Cox risk-set recurrences)   for FT chain slots f
//   (Algorithm.h:1109 Lm, :1236-1252 Logistic, :1341-1356 Poisson, :1593-1630 Cox; /root/reference/src)
//
// Why a second kernel: the register-streaming dual_sweep_kernel (kernels.cu) keeps 8 rows of loads in flight per thread
// and reaches the HBM roofline for ONE chain, but with 12 chains each warp alternates between a load phase and ~300
// FP64 instructions, its 24-48 accumulators cap occupancy at 4 CTAs/SM and ncu shows 59 % DRAM throughput with
// long-scoreboard stalls (profiles/r01c_dual_sweep_F12_full.md).  Here the loads are decoupled from the math:
//   * one producer thread per CTA streams X as row segments (COLS columns x 8 rows per stage) and the matching rows of
//     the gradient vectors into an NS-stage shared-memory ring with cp.async.bulk (SASS UBLKCP), completion on
//     full[stage] mbarriers (expect_tx byte counts);
//   * four consumer warps read x (conflict-free 16-byte LDS) and the chain values (broadcast LDS), do the FMAs and
//     release the stage through empty[stage] mbarriers -- no __syncthreads in the main loop;
//   * bytes in flight per SM = resident CTAs x (NS-1) x 16 KB, independent of register pressure.
// Output format (row-split partials reduced by finish_kernel) is identical to dual_sweep_kernel.
#include <cstdlib>

#include "device_utils.cuh"
#include "kernels.cuh"

namespace bess {

namespace {

constexpr int TNT = 128;       // consumer threads
constexpr int TRS = 8;         // rows per stage
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
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
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

template <int MODE>
struct TmaTraits {
    static constexpr int NV = MODE == MODE_D ? 1 : (MODE == MODE_DH ? 2 : 4);  // staged vectors
    static constexpr int NQ = MODE == MODE_D ? 1 : (MODE == MODE_DH ? 2 : 5);  // partial outputs per column
};

template <int FT, int MODE, int CPT, int NS>
__global__ void __launch_bounds__(TNT + 32) dual_sweep_tma_kernel(const Dev d)
{
    constexpr int NV = TmaTraits<MODE>::NV;
    constexpr int NQ = TmaTraits<MODE>::NQ;
    constexpr bool REV = (MODE == MODE_COX);  // risk-set suffix sums: walk rows from the last to the first
    constexpr int COLS = TNT * CPT;
    constexpr int XS = TRS * COLS;            // doubles of X per stage
    constexpr int VS = TRS * FT;              // doubles per vector per stage
    constexpr int STAGE = XS + NV * VS;

    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *ring = reinterpret_cast<double *>(smem_raw);  // [NS][STAGE]
    __shared__ __align__(8) uint64_t full[NS], empty[NS];
    if (d.gate && *d.gate == 0) return;  // every chain of the batch already stopped (speculative launch)

    const int tid = threadIdx.x;
    const int s = blockIdx.y;
    const int r0 = s * d.rows_per_split;
    const int r1 = min(d.n, r0 + d.rows_per_split);
    const int nrows = r1 - r0;
    const int nchunks = (nrows + TRS - 1) / TRS;
    const long long jb = (long long)blockIdx.x * COLS;        // first column of the CTA
    const int ncols = (int)min((long long)COLS, d.ldx - jb);   // ldx is even and zero padded
    const uint32_t seg_bytes = (uint32_t)ncols * 8u;

    if (tid == 0) {
#pragma unroll
        for (int q = 0; q < NS; q++) {
            mbar_init(&full[q], 1);
            mbar_init(&empty[q], TNT / 32);
        }
        mbar_fence_init();
    }
    __syncthreads();

    if (tid >= TNT) {
        // ---------------- producer: one thread streams the stages ----------------
        if (tid == TNT) {
            const double *vecs[4] = {d.G, d.W, d.TH, d.C2};
            for (int q = 0; q < nchunks; q++) {
                const int st = q % NS;
                if (q >= NS) mbar_wait(&empty[st], (uint32_t)(((q / NS) - 1) & 1));
                const int c = REV ? (nchunks - 1 - q) : q;
                const int cr0 = r0 + c * TRS;
                const int crows = min(TRS, r1 - cr0);
                const uint32_t vbytes = (uint32_t)(((crows + 1) & ~1) * FT * 8);  // vectors are padded to an even row count
                double *stg = ring + (size_t)st * STAGE;
                mbar_expect_tx(&full[st], seg_bytes * (uint32_t)crows + vbytes * NV);
                for (int r = 0; r < crows; r++)
                    bulk_g2s(stg + r * COLS, d.X + (size_t)(cr0 + r) * d.ldx + jb, seg_bytes, &full[st]);
#pragma unroll
                for (int v = 0; v < NV; v++) bulk_g2s(stg + XS + v * VS, vecs[v] + (size_t)cr0 * FT, vbytes, &full[st]);
            }
        }
        return;
    }

    // ---------------- consumers ----------------
    const long long j0 = jb + (long long)tid * CPT;
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

    for (int q = 0; q < nchunks; q++) {
        const int st = q % NS;
        mbar_wait(&full[st], (uint32_t)((q / NS) & 1));
        const int c = REV ? (nchunks - 1 - q) : q;
        const int cr0 = r0 + c * TRS;
        const int crows = min(TRS, r1 - cr0);
        const double *stg = ring + (size_t)st * STAGE;
        const double *tg = stg + XS;
        const double *tw = stg + XS + (NV > 1 ? 1 : 0) * VS;
        const double *tt = stg + XS + (NV > 2 ? 2 : 0) * VS;
        const double *tc = stg + XS + (NV > 3 ? 3 : 0) * VS;
        if (active) {
#pragma unroll
            for (int rr = 0; rr < TRS; rr++) {
                if (rr < crows) {
                    const int lr = REV ? (crows - 1 - rr) : rr;
                    double xv[CPT], xx[CPT];
                    if constexpr (CPT == 2) {
                        const double2 t = *reinterpret_cast<const double2 *>(stg + lr * COLS + tid * 2);
                        xv[0] = t.x;
                        xv[CPT - 1] = t.y;
                    } else {
                        xv[0] = stg[lr * COLS + tid];
                    }
#pragma unroll
                    for (int cc = 0; cc < CPT; cc++) xx[cc] = xv[cc] * xv[cc];
#pragma unroll
                    for (int f = 0; f < FT; f += 2) {
                        // FT is even: two chains per 16-byte broadcast load
                        const double2 g2 = *reinterpret_cast<const double2 *>(tg + lr * FT + f);
                        const double gq[2] = {g2.x, g2.y};
                        double wq[2] = {0.0, 0.0}, thq[2] = {0.0, 0.0}, c2q[2] = {0.0, 0.0};
                        if constexpr (MODE >= MODE_DH) {
                            const double2 w2 = *reinterpret_cast<const double2 *>(tw + lr * FT + f);
                            wq[0] = w2.x;
                            wq[1] = w2.y;
                        }
                        if constexpr (MODE == MODE_COX) {
                            const double2 t2 = *reinterpret_cast<const double2 *>(tt + lr * FT + f);
                            const double2 k2 = *reinterpret_cast<const double2 *>(tc + lr * FT + f);
                            thq[0] = t2.x; thq[1] = t2.y;
                            c2q[0] = k2.x; c2q[1] = k2.y;
                        }
#pragma unroll
                        for (int u = 0; u < 2; u++) {
#pragma unroll
                            for (int cc = 0; cc < CPT; cc++) {
                                accd[cc][f + u] = fma(xv[cc], gq[u], accd[cc][f + u]);
                                if constexpr (MODE >= MODE_DH) acch[cc][f + u] = fma(xx[cc], wq[u], acch[cc][f + u]);
                                if constexpr (MODE == MODE_COX) {
                                    s1[cc][f + u] = fma(xv[cc], thq[u], s1[cc][f + u]);
                                    const double t = c2q[u] * s1[cc][f + u];
                                    accA[cc][f + u] = fma(t, s1[cc][f + u], accA[cc][f + u]);
                                    accB[cc][f + u] += t;
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
        __syncwarp();
        if ((tid & 31) == 0) mbar_arrive(&empty[st]);
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
void launch_tma_t(const Dev &d, cudaStream_t st)
{
    constexpr int NV = TmaTraits<MODE>::NV;
    constexpr int NS = 4;
    constexpr size_t smem = (size_t)NS * (TRS * TNT * CPT + NV * TRS * FT) * sizeof(double);
    static bool configured = false;
    if (!configured) {
        CUDA_CHECK(cudaFuncSetAttribute(dual_sweep_tma_kernel<FT, MODE, CPT, NS>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)smem));
        configured = true;
    }
    const long long cols_per_cta = (long long)TNT * CPT;
    dim3 grid((unsigned)((d.p + cols_per_cta - 1) / cols_per_cta), (unsigned)d.S);
    dual_sweep_tma_kernel<FT, MODE, CPT, NS><<<grid, TNT + 32, smem, st>>>(d);
    CUDA_CHECK(cudaGetLastError());
}

// columns per thread: 2 (16-byte shared loads) unless the accumulator set would not fit in registers
constexpr int tma_cpt(int FT, int MODE)
{
    return FT <= 6 ? 2 : (FT <= 12 ? (MODE == MODE_COX ? 1 : 2) : (FT == 16 ? (MODE == MODE_D ? 2 : 1) : 1));
}

template <int MODE>
void launch_tma_m(const Dev &d, cudaStream_t st)
{
    switch (d.FS) {
        case 2: launch_tma_t<2, MODE, tma_cpt(2, MODE)>(d, st); break;
        case 4: launch_tma_t<4, MODE, tma_cpt(4, MODE)>(d, st); break;
        case 6: launch_tma_t<6, MODE, tma_cpt(6, MODE)>(d, st); break;
        case 8: launch_tma_t<8, MODE, tma_cpt(8, MODE)>(d, st); break;
        case 12: launch_tma_t<12, MODE, tma_cpt(12, MODE)>(d, st); break;
        case 16: launch_tma_t<16, MODE, tma_cpt(16, MODE)>(d, st); break;
        case 24: launch_tma_t<24, MODE, tma_cpt(24, MODE)>(d, st); break;
        case 32: launch_tma_t<32, MODE, tma_cpt(32, MODE)>(d, st); break;
        default: throw EngineError{"dual sweep: unsupported chain tile FS=" + std::to_string(d.FS)};
    }
}

}  // namespace

bool sweep_uses_tma(const Dev &d)
{
    static int force = -1;
    if (force < 0) {
        const char *e = std::getenv("BESS_B200_SWEEP");
        force = (e && std::string(e) == "stream") ? 0 : 1;
    }
    return force == 1 && d.FS >= 2;
}

int sweep_tma_cpt(int FS, int mode)
{
    return tma_cpt(FS, mode);
}

void launch_dual_sweep_tma(const Dev &d, int mode, cudaStream_t st)
{
    if (mode == MODE_D) launch_tma_m<MODE_D>(d, st);
    else if (mode == MODE_DH) launch_tma_m<MODE_DH>(d, st);
    else launch_tma_m<MODE_COX>(d, st);
}

}  // namespace bess
