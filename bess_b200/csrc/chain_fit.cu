// Chain kernels: the active-set side of one PDAS iteration (Algorithm::fit, /root/reference/src/Algorithm.h:154-170).
//
//   chain_begin_kernel   Algorithm::fit prologue (Algorithm.h:141-148) + gradient vectors of the first dual sweep.
//   chain_fit_kernel     after the top-k: gather X_A (utilities.cpp:132-140), the family's primary_model_fit
//                        (Algorithm.h:1131-1135 Lm / 1148-1204 Logistic / 1273-1322 Poisson / 1377-1490 Cox, iteration-exact),
//                        scatter + cycle test (Algorithm.h:159-170) and the gradient vectors of the next sweep
//                        (get_A prologues, Algorithm.h:1109 / 1223-1236 / 1338-1341 / 1579-1630).
//
// One thread-block CLUSTER of CL in {1,2,4,8} CTAs works on one chain.  The train rows are cut into CL contiguous
// slices; everything per-row (gather, linear predictor, IRLS weights, gradient vectors) is slice-local, Gram/Hessian
// matrices are accumulated per slice and reduced in a fixed order (bitwise reproducible), scalars are exchanged through
// distributed shared memory, the risk-set scans of the Cox model carry their totals from slice to slice.  Rank 0 of the
// cluster factors the (small) normal equations and broadcasts the solution.  CL = 1 (the k <= 20 configs) runs the very
// same code with every cluster operation compiled to a no-op branch.
#include <cooperative_groups.h>
#include <cuda_pipeline.h>

#include <algorithm>
#include <cfloat>
#include <cmath>
#include <cstdlib>

#include "device_utils.cuh"
#include "kernels.cuh"

namespace cg = cooperative_groups;

namespace bess {

constexpr int FIT_TILE_DOUBLES = 8192;  // 64 KB row tile for the Gram / panel of the blocked Cholesky
constexpr int FIT_SMEM_MS = 64;         // normal equations up to 64 x 64 are factored in shared memory
constexpr int CHOL_NB = 16;             // panel width of the blocked Cholesky (systems larger than FIT_SMEM_MS)

struct FitSmem {
    double *b0, *b1, *rhs, *dg;  // ldA each
    double *red;      // 40
    double *xch;      // 2 * CLMAX: cluster scalar exchange (written remotely through DSMEM)
    // the arena: tile | scratch | Ssm are its first three regions; the packed in-smem Cholesky uses all of it
    double *tile;     // FIT_TILE_DOUBLES
    double *scratch;  // FIT_NT * 16
    double *Ssm;      // FIT_SMEM_MS^2
    int arena_len;    // doubles from `tile` to the end of the dynamic shared memory
};
constexpr int FIT_ARENA_MIN = FIT_TILE_DOUBLES + FIT_NT * 16 + FIT_SMEM_MS * FIT_SMEM_MS;
// The FitSmem pointers travel through structs, references and (for the big solvers) real calls, where the compiler's
// address-space inference loses track of them and falls back to GENERIC loads / stores (LD.E / ST.E, 64-bit address
// arithmetic, no LDS.128) -- the hot loops re-derive them from the kernel's dynamic shared array with as_shared().
__device__ __forceinline__ double *as_shared(const double *p)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *const sbase = reinterpret_cast<double *>(smem_raw);
    return sbase + (p - sbase);
}
__device__ __forceinline__ FitSmem sm_shared(const FitSmem &a)
{
    FitSmem s;
    s.b0 = as_shared(a.b0);
    s.b1 = as_shared(a.b1);
    s.rhs = as_shared(a.rhs);
    s.dg = as_shared(a.dg);
    s.red = as_shared(a.red);
    s.xch = as_shared(a.xch);
    s.tile = as_shared(a.tile);
    s.scratch = as_shared(a.scratch);
    s.Ssm = as_shared(a.Ssm);
    s.arena_len = a.arena_len;
    return s;
}
__device__ __forceinline__ FitSmem carve_fit_smem(unsigned char *raw, int ldA, int total_doubles)
{
    FitSmem s;
    double *p = reinterpret_cast<double *>(raw);
    double *const base = p;
    s.b0 = p; p += ldA;
    s.b1 = p; p += ldA;
    s.rhs = p; p += ldA;
    s.dg = p; p += ldA;
    s.red = p; p += 40;
    s.xch = p; p += 2 * CLMAX;
    s.tile = p;
    s.scratch = p + FIT_TILE_DOUBLES;
    s.Ssm = p + FIT_TILE_DOUBLES + FIT_NT * 16;
    s.arena_len = total_doubles - (int)(p - base);
    return s;
}
// Dynamic shared memory of the chain kernels, in doubles: the minimum layout for small supports, everything the SM has
// (227 KB) when the normal equations may exceed FIT_SMEM_MS (so systems up to ~230 unknowns are factored in smem).
int fit_smem_doubles(int ldA, int kcap)
{
    const int fixed = 4 * ldA + 40 + 2 * CLMAX;
    const int maxd = (232448 - 1024) / 8;
    if (kcap + 3 <= FIT_SMEM_MS) return fixed + FIT_ARENA_MIN;
    return std::max(fixed + FIT_ARENA_MIN, maxd);
}
size_t fit_smem_bytes(const Dev &d) { return sizeof(double) * (size_t)d.fit_smem_doubles; }

// =====================================================================================================
// cluster plumbing
// =====================================================================================================
// ---- debug phase timers (bess_b200_debug_set(2, 1) enables; bess_b200_debug_get reads): clock64 ticks spent by thread 0
// of rank 0 between consecutive PH() markers, accumulated per phase id, plus a hit counter per phase
__device__ int g_dbg_phase_on = 0;
__device__ unsigned long long g_dbg_phase[2][16];
struct PhaseTimer {
    long long t;
    bool on;
    __device__ __forceinline__ void start(bool leader)
    {
        on = leader && g_dbg_phase_on;
        if (on) t = clock64();
    }
    __device__ __forceinline__ void mark(int id)
    {
        if (on) {
            const long long now = clock64();
            atomicAdd(&g_dbg_phase[0][id], (unsigned long long)(now - t));
            atomicAdd(&g_dbg_phase[1][id], 1ull);
            t = now;
        }
    }
};
enum { PH_GATHER = 0, PH_EVAL = 1, PH_WZ = 2, PH_SYRK = 3, PH_REDUCE = 4, PH_CHOL = 5, PH_BCAST = 6, PH_GRAD = 7,
       PH_CYCLE = 8, PH_OTHER = 9 };

struct Clu {
    int CL, rank;
    double *xch;
    int phase;
    PhaseTimer pt;
};
__device__ __forceinline__ void clu_sync(const Clu &cl)
{
    if (cl.CL > 1) cg::this_cluster().sync();
    else __syncthreads();
}
// Every thread of every CTA passes its CTA's value `local` (uniform inside a CTA); on return out[q] = value of rank q.
// Two alternating slot sets: a CTA can only reach exchange t+2 after every CTA has passed the barrier of exchange t+1,
// i.e. after everybody has finished reading the slots of exchange t.
__device__ __forceinline__ void clu_allgather(Clu &cl, double local, double (&out)[CLMAX])
{
#pragma unroll
    for (int q = 0; q < CLMAX; q++) out[q] = 0.0;
    if (cl.CL == 1) {
        out[0] = local;
        return;
    }
    cg::cluster_group cluster = cg::this_cluster();
    double *slot = cl.xch + cl.phase * CLMAX;
    if ((int)threadIdx.x < cl.CL) {
        double *remote = cluster.map_shared_rank(slot, threadIdx.x);
        remote[cl.rank] = local;
    }
    cluster.sync();
#pragma unroll
    for (int q = 0; q < CLMAX; q++)
        if (q < cl.CL) out[q] = slot[q];
    cl.phase ^= 1;
}
__device__ __forceinline__ double clu_allsum(Clu &cl, double local)
{
    if (cl.CL == 1) return local;
    double t[CLMAX];
    clu_allgather(cl, local, t);
    double s = 0.0;
#pragma unroll
    for (int q = 0; q < CLMAX; q++)
        if (q < cl.CL) s += t[q];
    return s;
}

struct ChainCtx {
    int c, nt, T, off, m;  // m = number of columns of the design incl. intercept
    int rb, re;            // this CTA's slice of the chain's (compacted) train rows
    double *XA;
    const double *y, *w;
    double *v[NVEC];
    double *S;             // where rank 0 factors the normal equations (smem or global), leading dim lds
    int lds;
    double *Sp0;           // cluster mode: partial-Gram buffers of the chain, rank q at Sp0 + q * sp_stride, [nmat][ldA*ldA]
    size_t sp_stride;
    double *Sfin;          // the chain's global matrices [2][ldA*ldA] (reduced normal equations / Cox second Gram)
    double *cw;            // exchange vectors of the chain [CLMAX][4][ldA]
    int ldA;
};
__device__ __forceinline__ double *cw_slot(const ChainCtx &cx, int rank, int s) { return cx.cw + (size_t)(rank * 4 + s) * cx.ldA; }

// =====================================================================================================
// Gram: S (mm x mm, both triangles) = sum_{r in [r0,r1)} wt[r] * V[r][a] * V[r][b]; V row-major, ld ldv, global memory
// =====================================================================================================
__device__ void block_syrk(const double *V, int ldv, int r0, int r1, int mm, const double *wt, double *S, int lds,
                           const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    const int tid = threadIdx.x;
    const int mb = (mm + 3) >> 2, mp = mb * 4;
    const int nblk = mb * (mb + 1) / 2;
    int R = FIT_TILE_DOUBLES / (mp + 1);
    if (R > 512) R = 512;
    double *tile = as_shared(sm.tile);
    double *tw = tile + (size_t)R * mp;
    double *scratch = as_shared(sm.scratch);
    const int nsl = nblk >= FIT_NT ? 1 : FIT_NT / nblk;
    const int nbatch = nsl > 1 ? 1 : (nblk + FIT_NT - 1) / FIT_NT;
    for (int batch = 0; batch < nbatch; batch++) {
        int blk, sl;
        bool valid;
        if (nsl > 1) {
            blk = tid % nblk;
            sl = tid / nblk;
            valid = sl < nsl;
        } else {
            blk = batch * FIT_NT + tid;
            sl = 0;
            valid = blk < nblk;
        }
        int bi = 0, bj = 0;
        if (valid) {
            bi = (int)((sqrt(8.0 * (double)blk + 1.0) - 1.0) * 0.5);
            while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
            while (bi * (bi + 1) / 2 > blk) bi--;
            bj = blk - bi * (bi + 1) / 2;
        }
        double acc[16];
#pragma unroll
        for (int e = 0; e < 16; e++) acc[e] = 0.0;
        auto fma_rows = [&](const double *tl, const double *twt, int rc) {
            for (int r = sl; r < rc; r += nsl) {
                const double w = twt[r];
                const double *ta = tl + r * mp + 4 * bi;
                const double *tb = tl + r * mp + 4 * bj;
                const double2 a01 = *reinterpret_cast<const double2 *>(ta);
                const double2 a23 = *reinterpret_cast<const double2 *>(ta + 2);
                const double2 b01 = *reinterpret_cast<const double2 *>(tb);
                const double2 b23 = *reinterpret_cast<const double2 *>(tb + 2);
                const double a[4] = {a01.x * w, a01.y * w, a23.x * w, a23.y * w};
                const double bb[4] = {b01.x, b01.y, b23.x, b23.y};
#pragma unroll
                for (int qa = 0; qa < 4; qa++)
#pragma unroll
                    for (int qb = 0; qb < 4; qb++) acc[qa * 4 + qb] = fma(a[qa], bb[qb], acc[qa * 4 + qb]);
            }
        };
        if (nsl == 1) {
            // Large systems (>= 512 tiles): the slice-reduction scratch is free, so it serves as a second row-tile buffer
            // and the staging of tile t+1 (cp.async, 16-byte chunks, no register round trip) overlaps the FMAs of tile t.
            // Columns in [mm, mp) receive whatever follows in the row (or stale shared memory past the row end): they only
            // feed accumulators that are never stored.
            double *const buf0 = as_shared(sm.tile), *const buf1 = as_shared(sm.scratch);
            const int ntile = (r1 - r0 + R - 1) / R;
            const int cpr = mp >> 1;  // 16-byte chunks per row
            auto issue = [&](int t) {
                const int rb = r0 + t * R;
                const int rc = min(R, r1 - rb);
                double *dst = (t & 1) ? buf1 : buf0;
                for (int e = tid; e < rc * cpr; e += FIT_NT) {
                    const int r = e / cpr, cidx = (e - r * cpr) * 2;
                    if (cidx < ldv) __pipeline_memcpy_async(dst + r * mp + cidx, V + (size_t)(rb + r) * ldv + cidx, 16);
                }
                double *twd = dst + (size_t)R * mp;
                for (int r = tid; r < rc; r += FIT_NT) twd[r] = wt ? wt[rb + r] : 1.0;
                __pipeline_commit();
            };
            __syncthreads();
            if (ntile > 0) issue(0);
            for (int t = 0; t < ntile; t++) {
                if (t + 1 < ntile) {
                    issue(t + 1);
                    __pipeline_wait_prior(1);
                } else {
                    __pipeline_wait_prior(0);
                }
                __syncthreads();
                if (valid) fma_rows((t & 1) ? buf1 : buf0, ((t & 1) ? buf1 : buf0) + (size_t)R * mp, min(R, r1 - (r0 + t * R)));
                __syncthreads();
            }
        } else {
            for (int rb = r0; rb < r1; rb += R) {
                const int rc = min(R, r1 - rb);
                const int tot = rc * mp;
                __syncthreads();
                // stage rc rows (zero-padded to mp columns): flattened and unrolled so 4 loads are in flight per thread
                for (int e0 = tid; e0 < tot; e0 += 4 * FIT_NT) {
                    double val[4];
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int e = e0 + q * FIT_NT;
                        val[q] = 0.0;
                        if (e < tot) {
                            const int r = e / mp, cidx = e - r * mp;
                            if (cidx < mm) val[q] = V[(size_t)(rb + r) * ldv + cidx];
                        }
                    }
#pragma unroll
                    for (int q = 0; q < 4; q++) {
                        const int e = e0 + q * FIT_NT;
                        if (e < tot) tile[e] = val[q];
                    }
                }
                for (int r = tid; r < rc; r += FIT_NT) tw[r] = wt ? wt[rb + r] : 1.0;
                __syncthreads();
                if (valid) fma_rows(tile, tw, rc);
            }
        }
        if (nsl > 1) {
            __syncthreads();
            if (valid) {
#pragma unroll
                for (int e = 0; e < 16; e++) scratch[(size_t)(sl * nblk + blk) * 16 + e] = acc[e];
            }
            __syncthreads();
            for (int idx = tid; idx < nblk * 16; idx += FIT_NT) {
                const int bk = idx >> 4, e = idx & 15;
                double v = 0.0;
                for (int q = 0; q < nsl; q++) v += scratch[(size_t)(q * nblk + bk) * 16 + e];
                int ci = (int)((sqrt(8.0 * (double)bk + 1.0) - 1.0) * 0.5);
                while ((ci + 1) * (ci + 2) / 2 <= bk) ci++;
                while (ci * (ci + 1) / 2 > bk) ci--;
                const int cj = bk - ci * (ci + 1) / 2;
                const int a = 4 * ci + (e >> 2), bcol = 4 * cj + (e & 3);
                if (a < mm && bcol < mm && a >= bcol) {
                    S[(size_t)a * lds + bcol] = v;
                    S[(size_t)bcol * lds + a] = v;
                }
            }
        } else if (valid) {
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const int a = 4 * bi + (e >> 2), bcol = 4 * bj + (e & 3);
                if (a < mm && bcol < mm && a >= bcol) {
                    S[(size_t)a * lds + bcol] = acc[e];
                    S[(size_t)bcol * lds + a] = acc[e];
                }
            }
        }
    }
    __syncthreads();
}

// =====================================================================================================
// Gram on the FP64 tensor cores (DMMA, mma.sync.m8n8k4.f64) for systems wide enough to be a real dense contraction
// (mm > 96): same contract as block_syrk.
//   * Work: the lower triangle in 16 x 16 tiles (m = 203: 91 tiles, 13 % more entries than the triangle itself; the
//     32 x 16 warp blocks of round 1 issued 39 % more and ran 3.5 rounds on 16 warps).  The tiles are dealt round robin
//     to the 16 warps; a warp accumulates up to GT = 3 tiles at once (12 DMMAs per 4-row step, 24 accumulator registers),
//     so the whole Gram is ceil(tiles / 48) passes over the row slice (2 at m = 203).
//   * Data: rows travel global -> shared memory as 1-D bulk-TMA copies (cp.async.bulk, one per row, issued by the lanes
//     of warp 0, completion on a `full` mbarrier per stage with expect-tx byte counts) into a 3-stage ring of row tiles
//     whose row stride is == 4 (mod 8) doubles (fragment loads hit every bank exactly twice: the minimum for 256 bytes).
//     A stage is released through an `empty` mbarrier (one arrival per warp) -- no block barrier and no per-thread
//     staging instructions in the main loop (the cp.async staging of round 1 spent a fifth of the issue slots on address
//     arithmetic with every warp staging at the same time, the tensor pipe idle meanwhile).
//   * The weight enters through the B operand (2 multiplies per tile and 4-row step).
// =====================================================================================================
__device__ __forceinline__ void dmma_m8n8k4(double (&c)[2], double a, double b)
{
    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                 : "+d"(c[0]), "+d"(c[1])
                 : "d"(a), "d"(b));
}
__device__ __forceinline__ uint32_t cf_smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void cf_mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(cf_smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void cf_mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(cf_smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void cf_mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(cf_smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void cf_bulk_g2s(void *dst, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     cf_smem_u32(dst)),
                 "l"(src), "r"(bytes), "r"(cf_smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void cf_mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred P1;\n"
        "CF_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 P1, [%0], %1;\n"
        "@P1 bra CF_DONE;\n"
        "bra CF_WAIT;\n"
        "CF_DONE:\n"
        "}" ::"r"(cf_smem_u32(bar)),
        "r"(parity)
        : "memory");
}
constexpr int GRAM_DMMA_MIN = 56;  // systems wider than this take the tensor-core path (probe: FMA path 11 us vs 16 us at 32, 44 vs 26 at 97)
constexpr int GRAM_NS = 3;  // ring stages
constexpr int GRAM_GT = 3;  // 16 x 16 tiles a warp accumulates at once
__device__ __noinline__ void block_syrk_dmma(const double *V, int ldv, int r0, int r1, int mm, const double *wt, double *S, int lds,
                                const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    constexpr int NW = FIT_NT / 32;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int g = lane >> 2, t4 = lane & 3;
    const int mp = ((mm + 3) >> 2) << 2;
    const int ts = (mp & 7) == 4 ? mp : mp + 4;       // tile row stride == 4 (mod 8) doubles
    const int ncopy = min(mp, ldv);                   // doubles copied per row (even: 16-byte multiples)
    const int nt16 = (mm + 15) >> 4;
    const int ntiles = nt16 * (nt16 + 1) / 2;
    const int npass = (ntiles + NW * GRAM_GT - 1) / (NW * GRAM_GT);
    // ring: GRAM_NS stages of R rows (+ R weights each) in the arena
    // (systems of up to FIT_SMEM_MS rows may have their output S in the Ssm region of the arena: keep the ring off it)
    const int ring_len = mm <= FIT_SMEM_MS ? FIT_TILE_DOUBLES + FIT_NT * 16 - 16 : sm.arena_len - 16;
    int R = (ring_len / GRAM_NS / (ts + 1)) & ~3;
    if (R > 64) R = 64;
    double *ring = sm.tile;
    const int stage_len = R * (ts + 1);               // rows, then the R weights of the stage
    uint64_t *full = reinterpret_cast<uint64_t *>(sm.red);  // [GRAM_NS], empty = full + GRAM_NS
    uint64_t *empty = full + GRAM_NS;
    const int nrow = r1 - r0;
    if (nrow <= 0) {  // an empty row slice contributes a zero matrix (cluster sizing never produces one; kept for safety)
        for (int e = tid; e < mm * mm; e += FIT_NT) S[(size_t)(e / mm) * lds + e % mm] = 0.0;
        __syncthreads();
        return;
    }
    const int ntile = (nrow + R - 1) / R;
    const int nstep = ntile * npass;
    __syncthreads();  // the arena and sm.red are free
    if (tid == 0) {
        for (int q = 0; q < GRAM_NS; q++) {
            cf_mbar_init(&full[q], 1);
            cf_mbar_init(&empty[q], NW);
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    // rows that only pad the last 4-row step of the last tile must be finite (their weight is 0): clear them in the stage
    // that will hold the last tile if no earlier tile overwrites them with data first
    {
        const int rc_last = nrow - (ntile - 1) * R, rc4 = (rc_last + 3) & ~3;
        for (int q = 0; q < GRAM_NS; q++)
            for (int e = tid; e < (rc4 - rc_last) * ts; e += FIT_NT) ring[q * stage_len + rc_last * ts + e] = 0.0;
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    __syncthreads();
    // producer (warp 0): tile step q -> stage q % NS
    // weights of tile step q for rows lane, lane + 32 (R <= 64), fetched one step ahead of their use by the producer
    double wpre[2] = {0.0, 0.0};
    auto fetch_w = [&](int q) {
        const int t = q % ntile;
        const int rb = r0 + t * R, rc = min(R, r1 - rb);
#pragma unroll
        for (int h = 0; h < 2; h++) wpre[h] = lane + 32 * h < rc ? (wt ? wt[rb + lane + 32 * h] : 1.0) : 0.0;
    };
    auto produce = [&](int q) {
        const int st = q % GRAM_NS;
        const int t = q % ntile;
        const int rb = r0 + t * R, rc = min(R, r1 - rb);
        double *dst = ring + st * stage_len;
        if (q >= GRAM_NS) cf_mbar_wait(&empty[st], (uint32_t)(((q / GRAM_NS) - 1) & 1));
        // weights of the stage (generic stores, published by the arrive below), zero for the padding rows
#pragma unroll
        for (int h = 0; h < 2; h++)
            if (lane + 32 * h < R) dst[R * ts + lane + 32 * h] = wpre[h];
        if (q + 1 < nstep) fetch_w(q + 1);
        __syncwarp();
        if (lane == 0) cf_mbar_expect_tx(&full[st], (uint32_t)(rc * ncopy * 8));
        __syncwarp();
        for (int r = lane; r < rc; r += 32) cf_bulk_g2s(dst + r * ts, V + (size_t)(rb + r) * ldv, (uint32_t)(ncopy * 8), &full[st]);
    };
    if (wid == 0) {
        fetch_w(0);
        for (int q = 0; q < GRAM_NS - 1 && q < nstep; q++) produce(q);
    }
    // this warp's tiles of the current pass
    int ti[GRAM_GT], tj[GRAM_GT];
    bool tv[GRAM_GT];
    double acc[GRAM_GT][2][2][2];
    auto start_pass = [&](int pass) {
#pragma unroll
        for (int u = 0; u < GRAM_GT; u++) {
            const int t = (pass * GRAM_GT + u) * NW + wid;
            tv[u] = t < ntiles;
            int bi = 0, bj = 0;
            if (tv[u]) {
                bi = (int)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
                while ((bi + 1) * (bi + 2) / 2 <= t) bi++;
                while (bi * (bi + 1) / 2 > t) bi--;
                bj = t - bi * (bi + 1) / 2;
            }
            ti[u] = bi;
            tj[u] = bj;
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int nt = 0; nt < 2; nt++) acc[u][mt][nt][0] = acc[u][mt][nt][1] = 0.0;
        }
    };
    auto store_pass = [&]() {
#pragma unroll
        for (int u = 0; u < GRAM_GT; u++) {
            if (!tv[u]) continue;
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int nt = 0; nt < 2; nt++)
#pragma unroll
                    for (int w = 0; w < 2; w++) {
                        const int a = ti[u] * 16 + mt * 8 + g, b = tj[u] * 16 + nt * 8 + t4 * 2 + w;
                        // lower triangle only: a diagonal tile holds (a, b) and (b, a), rounded differently (the weight
                        // scales the B operand), and both would be stored to both places
                        if (a < mm && b < mm && a >= b) {
                            S[(size_t)a * lds + b] = acc[u][mt][nt][w];
                            S[(size_t)b * lds + a] = acc[u][mt][nt][w];
                        }
                    }
        }
    };
    start_pass(0);
    for (int q = 0; q < nstep; q++) {
        const int st = q % GRAM_NS;
        const int t = q % ntile;
        if (wid == 0 && q + GRAM_NS - 1 < nstep) produce(q + GRAM_NS - 1);
        cf_mbar_wait(&full[st], (uint32_t)((q / GRAM_NS) & 1));
        const double *tl = ring + st * stage_len;
        const double *twt = tl + R * ts;
        const int rc4 = (min(R, nrow - t * R) + 3) & ~3;
        const double *pk = tl + t4 * ts + g;
#pragma unroll 2
        for (int k0 = 0; k0 < rc4; k0 += 4) {
            const double w = twt[k0 + t4];
#pragma unroll
            for (int u = 0; u < GRAM_GT; u++) {
                if (tv[u]) {
                    const double *pa = pk + (size_t)k0 * ts + ti[u] * 16;
                    const double *pb = pk + (size_t)k0 * ts + tj[u] * 16;
                    const double a0 = pa[0], a1 = pa[8];
                    const double b0 = pb[0] * w, b1 = pb[8] * w;
                    dmma_m8n8k4(acc[u][0][0], a0, b0);
                    dmma_m8n8k4(acc[u][0][1], a0, b1);
                    dmma_m8n8k4(acc[u][1][0], a1, b0);
                    dmma_m8n8k4(acc[u][1][1], a1, b1);
                }
            }
        }
        __syncwarp();
        if (lane == 0) cf_mbar_arrive(&empty[st]);
        if (t == ntile - 1) {
            store_pass();
            if (q + 1 < nstep) start_pass(q / ntile + 1);
        }
    }
    __syncthreads();
    if (tid == 0) {  // sm.red goes back to being plain scratch
        for (int q = 0; q < 2 * GRAM_NS; q++) asm volatile("mbarrier.inval.shared::cta.b64 [%0];" ::"r"(cf_smem_u32(&full[q])) : "memory");
    }
    __syncthreads();
}
// dispatcher: tensor cores when the system is wide, register-blocked FMAs otherwise
__device__ __forceinline__ void gram(const double *V, int ldv, int r0, int r1, int mm, const double *wt, double *S, int lds,
                                     const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    if (mm > GRAM_DMMA_MIN) block_syrk_dmma(V, ldv, r0, r1, mm, wt, S, lds, sm);
    else block_syrk(V, ldv, r0, r1, mm, wt, S, lds, sm);
}

// =====================================================================================================
// Cholesky solves.  The systems are "bordered": rows 0..mm-1 hold the SPD matrix (lower triangle used), row mm holds the
// right-hand side.  Factoring the bordered matrix leaves z = L^{-1} rhs in row mm (forward substitution for free);
// a back substitution then gives x = S^{-1} rhs.
// (The reference uses Eigen's pivoted ldlt()/colPivHouseholderQr(); for the SPD, well-conditioned active-set systems of
//  this path the solutions agree to ~1e-13 relative.)
// =====================================================================================================
// unblocked, for systems resident in shared memory
// A pivot at or below PIVOT_TOL times the column's own diagonal entry (its squared norm) is a numerically dependent column.
constexpr double PIVOT_TOL = 1e-13;
__device__ unsigned long long g_rankdef_count = 0ull;  // truncated (rank-deficient) solves since the last debug_take_rankdef()
// singular systems of more than FIT_SMEM_MS unknowns (chol_panel_major: x <- NaN) since the last take_wide_singular()
__device__ unsigned long long g_wide_singular_count = 0ull;
// S0: pristine copy of the system (same layout).  Returns false -- S is then garbage -- when a pivot fails the test above.
__device__ bool block_chol_solve_small(double *S, int lds, int mm, double *x, double *dg, const double *S0)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    for (int j = 0; j < mm; j++) {
        __syncthreads();
        const double sjj = S[(size_t)j * lds + j];
        if (!(sjj > PIVOT_TOL * S0[(size_t)j * lds + j])) return false;  // uniform over the CTA (NaN fails too)
        const double djj = sqrt(sjj);
        if (tid == 0) dg[j] = djj;
        const double inv = 1.0 / djj;
        for (int i = j + 1 + tid; i <= mm; i += FIT_NT) S[(size_t)i * lds + j] *= inv;
        __syncthreads();
        for (int i = j + 1 + wid; i <= mm; i += FIT_NT / 32) {
            const double lij = S[(size_t)i * lds + j];
            const int cend = min(i, mm - 1);
            for (int c = j + 1 + lane; c <= cend; c += 32) S[(size_t)i * lds + c] -= lij * S[(size_t)c * lds + j];
        }
    }
    __syncthreads();
    if (wid == 0) {
        for (int c = lane; c < mm; c += 32) x[c] = S[(size_t)mm * lds + c];  // z
        __syncwarp();
        for (int j = mm - 1; j >= 0; j--) {  // L^T x = z, column oriented
            const double xj = x[j] / dg[j];
            __syncwarp();
            if (lane == 0) x[j] = xj;
            for (int c = lane; c < j; c += 32) x[c] -= S[(size_t)j * lds + c] * xj;
            __syncwarp();
        }
    }
    __syncthreads();
    return true;
}

// Rank-revealing fallback for the systems above (<= FIT_SMEM_MS unknowns, both triangles of S valid, border row mm = right-
// hand side): LDL^T with Eigen's diagonal pivoting -- at step k the FIRST largest diagonal entry in the current positional
// order of the remaining unknowns, swapped into position k, the unknown that sat there moving back to where the pivot came
// from (Eigen/src/Cholesky/LDLT.h:300-330) -- that STOPS when no remaining pivot passes the PIVOT_TOL test; the unknowns
// left over get 0.  This is what the reference's solvers return on a singular system with an exactly duplicated column:
// the pivoted ldlt() meets an exactly zero pivot and its solve() skips it (LDLT.h:558-592), colPivHouseholderQr()
// truncates at its rank threshold (Algorithm.h:1134) -- one copy keeps the whole coefficient, the other gets 0.  (Which
// copy: the one met first in the positional order, as in the LDLT; the QR's own order can differ -- the two models are
// the same function of the data.)  work: >= 3 * (mm + 1) doubles.
__device__ void ldlt_pivoted_small(double *S, int lds, int mm, double *x, const double *S0, double *work)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    double *lcol = work;                                       // [mm + 1] multipliers of the running step
    int *perm = reinterpret_cast<int *>(work + mm + 1);        // [mm] unknown at position q; then perm[mm] = step's pivot position
    int *posof = perm + mm + 1;                                // [mm] position of unknown i
    for (int i = tid; i < mm; i += FIT_NT) {
        perm[i] = i;
        posof[i] = i;
        x[i] = 0.0;
    }
    __syncthreads();
    int rank = 0;
    for (; rank < mm; rank++) {
        const int k = rank;
        if (wid == 0) {
            double best = -1.0;
            int bpos = -1;
            for (int pos = k + lane; pos < mm; pos += 32) {
                const int p = perm[pos];
                const double v = S[(size_t)p * lds + p];
                if (v > PIVOT_TOL * S0[(size_t)p * lds + p] && v > best) {
                    best = v;
                    bpos = pos;
                }
            }
#pragma unroll
            for (int o = 16; o > 0; o >>= 1) {
                const double ov = __shfl_xor_sync(0xffffffffu, best, o);
                const int op = __shfl_xor_sync(0xffffffffu, bpos, o);
                if (op >= 0 && (bpos < 0 || ov > best || (ov == best && op < bpos))) {
                    best = ov;
                    bpos = op;
                }
            }
            if (lane == 0) {
                perm[mm] = bpos;
                if (bpos >= 0) {
                    const int pk = perm[k], pb = perm[bpos];
                    perm[k] = pb;
                    perm[bpos] = pk;
                    posof[pb] = k;
                    posof[pk] = bpos;
                }
            }
        }
        __syncthreads();
        if (perm[mm] < 0) break;
        const int p = perm[k];
        const double dinv = 1.0 / S[(size_t)p * lds + p];
        for (int i = tid; i <= mm; i += FIT_NT)
            if (i == mm || posof[i] > k) lcol[i] = S[(size_t)i * lds + p] * dinv;
        __syncthreads();
        for (int e = tid; e < (mm + 1) * mm; e += FIT_NT) {
            const int i = e / mm, c = e - i * mm;
            if ((i == mm || posof[i] > k) && posof[c] > k) S[(size_t)i * lds + c] -= lcol[i] * S[(size_t)p * lds + c];
        }
        __syncthreads();
        for (int i = tid; i < mm; i += FIT_NT)
            if (posof[i] > k) S[(size_t)i * lds + p] = lcol[i];  // kept for the back substitution
        __syncthreads();
    }
    // back substitution in reverse pivot order: x_p = y_p / d_p - sum over later pivots q of l_qp x_q
    if (wid == 0) {
        for (int k = rank - 1; k >= 0; k--) {
            const int p = perm[k];
            double acc = 0.0;
            for (int t = k + 1 + lane; t < rank; t += 32) {
                const int q = perm[t];
                acc = fma(S[(size_t)q * lds + p], x[q], acc);
            }
            acc = warp_sum(acc);
            if (lane == 0) x[p] = S[(size_t)mm * lds + p] / S[(size_t)p * lds + p] - acc;
            __syncwarp();
        }
        if (lane == 0 && rank < mm) atomicAdd(&g_rankdef_count, 1ull);
    }
    __syncthreads();
}

// Factor one CHOL_NB-column panel of a bordered lower-triangular system held in shared memory.  Thread i owns panel row i
// (i < mr <= FIT_NT) in registers; rowp(i) points at its first panel column.  Per column q one block barrier: the rows of the
// diagonal block publish their (unscaled) column-q entry, every thread derives the pivot and L[c][q] itself and updates
// its own row.  On exit rows hold L (diagonal block: lower part only, `lower_only(i)` tells how many columns row i has).
template <class RowPtr>
__device__ __forceinline__ void panel_factor(RowPtr rowp, int mr, int nb, double *colbuf /* 2 * CHOL_NB */)
{
    constexpr int NB = CHOL_NB;
    const int i = threadIdx.x;
    const bool own = i < mr;
    double row[NB];
    double *rp = own ? rowp(i) : nullptr;
#pragma unroll
    for (int c = 0; c < NB; c++) row[c] = (own && c < nb && (i >= nb || c <= i)) ? rp[c] : 0.0;
#pragma unroll
    for (int q = 0; q < NB; q++) {
        if (q < nb) {
            double *cb = colbuf + (q & 1) * NB;
            if (own && i >= q && i < nb) cb[i] = row[q];
            __syncthreads();
            const double inv = rsqrt(cb[q]);
            if (i == q) row[q] = cb[q] * inv;
            else if (i > q) row[q] *= inv;
            if (i > q) {
#pragma unroll
                for (int c = 0; c < NB; c++)
                    if (c > q && c < nb) row[c] -= row[q] * (cb[c] * inv);
            }
        }
    }
#pragma unroll
    for (int c = 0; c < NB; c++)
        if (own && c < nb && (i >= nb || c <= i)) rp[c] = row[c];
    __syncthreads();
}

// Bordered Cholesky solve entirely in shared memory (one CTA) for systems of 65 .. ~230 unknowns: the lower triangle is
// copied from the global matrix into PACKED row-major storage in the arena, factored right-looking in CHOL_NB-column
// panels (panel_factor + register-blocked 4x4 trailing update) and back-substituted in place.  x (smem) <- solution.
__device__ __forceinline__ int tri(int i) { return (i * (i + 1)) >> 1; }
__device__ __forceinline__ bool packed_fits(int mm, int arena_len) { return tri(mm + 1) + FIT_NT <= arena_len; }
__device__ __noinline__ void chol_packed_smem(const double *Sg, int lds, int mm, double *x, const FitSmem &sm_, PhaseTimer &pt)
{
    const FitSmem sm = sm_shared(sm_);
    constexpr int NB = CHOL_NB;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    double *Lp = sm.tile;                 // packed: row i at tri(i), columns 0..min(i, mm-1)
    double *red = sm.tile + tri(mm + 1);  // FIT_NT doubles of reduction scratch behind the matrix
    __syncthreads();
    for (int i0 = wid * 8; i0 <= mm; i0 += (FIT_NT / 32) * 8) {
        for (int c = lane; c < mm; c += 32) {
            double v[8];
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int i = i0 + u;
                if (i <= mm && c <= i) v[u] = Sg[(size_t)i * lds + c];
            }
#pragma unroll
            for (int u = 0; u < 8; u++) {
                const int i = i0 + u;
                if (i <= mm && c <= i) Lp[tri(i) + c] = v[u];
            }
        }
    }
    __syncthreads();
    pt.mark(10);
    for (int j0 = 0; j0 < mm; j0 += NB) {
        const int nb = min(NB, mm - j0);
        const int mr = mm + 1 - j0;
        panel_factor([&](int i) { return Lp + tri(j0 + i) + j0; }, mr, nb, sm.dg);
        const int t0 = j0 + nb;
        const int mt = mm - t0;
        if (mt <= 0) break;
        // trailing update: S[a][b] -= sum_q L[a][j0+q] L[b][j0+q] for a in [t0, mm], b in [t0, min(a, mm-1)]
        const int rbk = (mt + 1 + 3) >> 2;
        const int nblk = rbk * (rbk + 1) / 2;
        for (int blk = tid; blk < nblk; blk += FIT_NT) {
            int bi = (int)((sqrt(8.0 * (double)blk + 1.0) - 1.0) * 0.5);
            while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
            while (bi * (bi + 1) / 2 > blk) bi--;
            const int bj = blk - bi * (bi + 1) / 2;
            double acc[16];
#pragma unroll
            for (int e = 0; e < 16; e++) acc[e] = 0.0;
            const double *pa[4], *pb[4];
#pragma unroll
            for (int u = 0; u < 4; u++) {
                const int ra = min(t0 + 4 * bi + u, mm), rb = min(t0 + 4 * bj + u, mm);
                pa[u] = Lp + tri(ra) + j0;
                pb[u] = Lp + tri(rb) + j0;
            }
            for (int q = 0; q < nb; q++) {
                double a[4], bb[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    a[u] = pa[u][q];
                    bb[u] = pb[u][q];
                }
#pragma unroll
                for (int qa = 0; qa < 4; qa++)
#pragma unroll
                    for (int qb = 0; qb < 4; qb++) acc[qa * 4 + qb] = fma(a[qa], bb[qb], acc[qa * 4 + qb]);
            }
#pragma unroll
            for (int e = 0; e < 16; e++) {
                const int a = t0 + 4 * bi + (e >> 2), b = t0 + 4 * bj + (e & 3);
                if (a <= mm && b < mm && b <= a) Lp[tri(a) + b] -= acc[e];
            }
        }
        __syncthreads();
    }
    __syncthreads();
    pt.mark(11);
    // back substitution L^T x = z, z = row mm
    for (int c = tid; c < mm; c += FIT_NT) x[c] = Lp[tri(mm) + c];
    __syncthreads();
    const int jlast = ((mm - 1) / NB) * NB;
    for (int j0 = jlast; j0 >= 0; j0 -= NB) {
        const int nb = min(NB, mm - j0);
        const int t0 = j0 + nb;
        // v[q] = sum_{i in [t0, mm)} L[i][j0+q] x[i]: thread (q = tid & 15, g = tid >> 4) sums the rows i == g (mod 32)
        {
            const int q = tid & (NB - 1), g = tid >> 4;
            double acc = 0.0;
            if (q < nb)
                for (int i = t0 + g; i < mm; i += FIT_NT / NB) acc = fma(Lp[tri(i) + j0 + q], x[i], acc);
            red[g * NB + q] = acc;
        }
        __syncthreads();
        if (wid == 0) {
            double t = 0.0;
            if (lane < nb) {
                double vsum = 0.0;
                for (int g2 = 0; g2 < FIT_NT / NB; g2++) vsum += red[g2 * NB + lane];
                t = x[j0 + lane] - vsum;
            }
            for (int q = nb - 1; q >= 0; q--) {
                const double yq = __shfl_sync(0xffffffffu, t, q) / Lp[tri(j0 + q) + j0 + q];
                if (lane == q) t = yq;
                if (lane < q) t -= Lp[tri(j0 + q) + j0 + lane] * yq;
            }
            if (lane < nb) x[j0 + lane] = t;
        }
        __syncthreads();
    }
    pt.mark(12);
}

// =====================================================================================================
// Panel-major Cholesky: the solver of the wide systems (65 .. 511 unknowns; C2: every IRLS step factors a ~200 x 200
// Hessian).  One CTA, the matrix in shared memory in PANEL-MAJOR storage: panel pb holds columns [16 pb, 16 pb + 16) for
// the rows from its own first column down to the border row mm, COLUMN-major inside the panel with a leading dimension
// == 4 (mod 8) doubles.  That layout makes every access of the factorisation conflict-free:
//   * panel factor: thread i owns panel row i, a column is contiguous over the threads;
//   * trailing update on the FP64 tensor cores (mma.sync.m8n8k4.f64, SASS DMMA): an A / B fragment is 8 consecutive rows
//     x 4 consecutive panel columns -- 8 contiguous doubles per column, the four columns 4 (mod 8) doubles apart, i.e.
//     two shared-memory wavefronts, the minimum for 256 bytes; a warp owns a 32 x 16 block of the trailing matrix
//     (8 accumulator tiles), 6 loads per 8 DMMAs.  (The packed row-major layout this replaces had every lane of a warp
//     in a different row at an irregular offset: 4-8-way bank conflicts, 137 us per factorisation at 200 unknowns.)
//   * back substitution: warp q reduces panel column q against x with contiguous loads.
// Systems that do not fit the arena (~225 unknowns at 227 KB) run in STAGES: as many leading panels as fit are factored in
// shared memory at their full height, the Schur complement of the remaining columns is updated in place in the global
// matrix by DMMA blocks with the stage as the k dimension, the factored panels are written back, and the next stage loads
// what is left; the back substitution reloads the stages in reverse order.
// =====================================================================================================
constexpr int PNB = 16;
constexpr int PM_MAX_STAGES = 12;
__device__ int g_dbg_solver = 0;  // debug knob (bess_b200_debug_set key 4): 1 = the round-1 solvers (packed / cluster-blocked)
__device__ __forceinline__ int pm_ld(int h) { return (((h + 3) >> 3) << 3) + 4; }  // >= h and == 4 (mod 8)
// number of 16-column panels from column c0 on (at their full height mm + 1 - c) that fit `cap` doubles
__device__ __forceinline__ int pm_plan(int c0, int mm, int cap)
{
    int used = 0, np = 0;
    for (int c = c0; c < mm; c += PNB) {
        const int need = PNB * pm_ld(mm + 1 - c);
        if (used + need > cap) break;
        used += need;
        np++;
    }
    return np;
}
__device__ __forceinline__ int pm_capacity(int arena_len) { return arena_len - 96; }  // 64-double header in front, slack behind
__device__ __forceinline__ int pm_stage_count(int mm, int arena_len)
{
    const int cap = pm_capacity(arena_len);
    int ns = 0;
    for (int c0 = 0; c0 < mm;) {
        const int np = pm_plan(c0, mm, cap);
        if (np == 0) return PM_MAX_STAGES + 1;
        c0 += np * PNB;
        ns++;
    }
    return ns;
}
// poff[pb] = offset of panel pb of the stage that starts at column c0
__device__ __forceinline__ void pm_offsets(int *poff, int mm, int c0, int np)
{
    __syncthreads();
    if ((int)threadIdx.x < np) {
        int off = 0;
        for (int q = 0; q < (int)threadIdx.x; q++) off += PNB * pm_ld(mm + 1 - (c0 + q * PNB));
        poff[threadIdx.x] = off;
    }
    __syncthreads();
}
// global (row-major, lower triangle) -> panels.  A warp moves 4-row x 8-column patches: 64-byte row segments on the
// global side, 16 distinct banks x 2 on the shared side.  Columns past the last one are zero-filled.
template <bool TO_GLOBAL>
__device__ void pm_copy(double *L, const int *poff, double *Sg, int lds, int mm, int c0, int np)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int il = lane >> 3, cl = lane & 7;
    constexpr int NW = FIT_NT / 32;
    for (int pb = 0; pb < np; pb++) {
        const int r0 = c0 + pb * PNB;
        const int h = mm + 1 - r0, ld = pm_ld(h);
        const int nb = min(PNB, mm - r0);
        double *P = L + poff[pb];
        const int npatch = 2 * ((h + 3) >> 2);
        if (TO_GLOBAL) {
            for (int pa = wid; pa < npatch; pa += NW) {
                const int i = (pa >> 1) * 4 + il, c = (pa & 1) * 8 + cl;
                if (i < h && c < nb && c <= i) Sg[(size_t)(r0 + i) * lds + r0 + c] = P[c * ld + i];
            }
        } else {
            for (int pa0 = wid; pa0 < npatch; pa0 += 4 * NW) {
                double v[4];
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int pa = pa0 + u * NW;
                    const int i = (pa >> 1) * 4 + il, c = (pa & 1) * 8 + cl;
                    v[u] = (pa < npatch && i < h && c < nb) ? Sg[(size_t)(r0 + i) * lds + r0 + c] : 0.0;
                }
#pragma unroll
                for (int u = 0; u < 4; u++) {
                    const int pa = pa0 + u * NW;
                    const int i = (pa >> 1) * 4 + il, c = (pa & 1) * 8 + cl;
                    if (pa < npatch && i < h) P[c * ld + i] = v[u];
                }
            }
        }
    }
    __syncthreads();
}
// 1 / sqrt(d) for the pivots: hardware approximation (2^-22) + two Newton steps (full double precision for normal d; a
// non-positive pivot gives NaN like the library call, which is how a non-SPD system shows up).
__device__ __forceinline__ double pm_rsqrt(double d)
{
    double y;
    asm("rsqrt.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(d));
#pragma unroll
    for (int it = 0; it < 2; it++) {
        const double t = d * y;
        const double e = fma(-t, y, 1.0);
        y = fma(0.5 * y, e, y);
    }
    return y;
}
// Diagonal block of a panel (nb x nb, in place), ONE warp: lane r holds row r in registers; per column the scaled pivot
// column goes through a 16-double shared buffer (one store, broadcast loads) -- no block barrier in the serial part of
// the factorisation.  dinv[q] <- 1 / L[q][q] (the rsqrt itself: neither the row solve below nor the back substitution
// ever divides).  colbuf: 2 * PNB doubles.
__device__ __forceinline__ void pm_diag_factor(double *P, int ld, int nb, double *dinv, double *colbuf)
{
    const int lane = threadIdx.x & 31, r = lane & 15;
    double a[PNB];
#pragma unroll
    for (int c = 0; c < PNB; c++) a[c] = (r < nb && c <= r) ? P[c * ld + r] : (c == r ? 1.0 : 0.0);
#pragma unroll
    for (int q = 0; q < PNB; q++) {
        const double d = __shfl_sync(0xffffffffu, a[q], q);
        const double inv = pm_rsqrt(d);
        const double lq = (r == q) ? d * inv : a[q] * inv;
        a[q] = lq;
        if (lane == q && q < nb) dinv[q] = inv;
        if (q + 1 < PNB) {
            double *cb = colbuf + (q & 1) * PNB;
            if (lane < PNB) cb[lane] = lq;
            __syncwarp();
#pragma unroll
            for (int c = q + 1; c < PNB; c++) a[c] = fma(-lq, cb[c], a[c]);
        }
    }
    if (lane < nb) {
#pragma unroll
        for (int c = 0; c < PNB; c++)
            if (c <= lane) P[c * ld + lane] = a[c];
    }
}
// Rows below the diagonal block: thread i solves its own row against L11 (x L11^T = a, forward substitution in registers,
// L11 broadcast from shared memory): 136 fp64 instructions per row, no barrier, no rsqrt.
template <bool FULL>
__device__ __forceinline__ void pm_row_solve_one(double *P, int ld, int i, int nb, const double *dinv)
{
    double a[PNB];
#pragma unroll
    for (int c = 0; c < PNB; c++) a[c] = (FULL || c < nb) ? P[c * ld + i] : 0.0;
#pragma unroll
    for (int c = 0; c < PNB; c++) {
        if (FULL || c < nb) {
            const double xc = a[c] * dinv[c];
            a[c] = xc;
#pragma unroll
            for (int q = c + 1; q < PNB; q++)
                if (FULL || q < nb) a[q] = fma(-xc, P[c * ld + q], a[q]);
        }
    }
#pragma unroll
    for (int c = 0; c < PNB; c++)
        if (FULL || c < nb) P[c * ld + i] = a[c];
}
// Phase A of a panel step: warp 0 solves the 16 rows right below the diagonal block (the rows of the NEXT diagonal block:
// its own critical path), warps 1 .. 15 the rows beyond.
template <bool FULL>
__device__ __forceinline__ void pm_row_solve(double *P, int ld, int h, int nb, const double *dinv)
{
    const int tid = threadIdx.x;
    const int i = tid < 32 ? (tid < PNB ? nb + tid : h) : nb + PNB + (tid - 32);
    if (i < h) pm_row_solve_one<FULL>(P, ld, i, nb, dinv);
    __syncthreads();
}
// acc (32 rows from a0 x 16 rows from b0, as 4 x 2 mma tiles) += L[a][q] L[b][q] over the 16 columns q of panel Pq
// (first row / column cq, leading dimension ldq, hq rows).  Rows past the border are clamped to the border row: they only
// reach accumulators that are never stored, and the loads stay inside the (read-only) source panel.
__device__ __forceinline__ void pm_mma_panel(double (&acc)[4][2][2], const double *Pq, int ldq, int cq, int hq, int a0, int b0,
                                             int g, int t4)
{
    const double *pk = Pq + t4 * ldq;
    int ra[4], rb[2];
#pragma unroll
    for (int mt = 0; mt < 4; mt++) ra[mt] = min(a0 - cq + 8 * mt + g, hq - 1);
#pragma unroll
    for (int nt = 0; nt < 2; nt++) rb[nt] = min(b0 - cq + 8 * nt + g, hq - 1);
#pragma unroll
    for (int q0 = 0; q0 < PNB; q0 += 4) {
        double a[4], b[2];
#pragma unroll
        for (int mt = 0; mt < 4; mt++) a[mt] = pk[q0 * ldq + ra[mt]];
#pragma unroll
        for (int nt = 0; nt < 2; nt++) b[nt] = pk[q0 * ldq + rb[nt]];
#pragma unroll
        for (int mt = 0; mt < 4; mt++)
#pragma unroll
            for (int nt = 0; nt < 2; nt++) dmma_m8n8k4(acc[mt][nt], a[mt], b[nt]);
    }
}
// Phase B of a panel step.  Warps 1 .. 15: right-looking update of the stage's later panels with factored panel pb,
// S[a][b] -= sum_q L[a][q] L[b][q], work units (target panel, 32-row block) dealt round robin -- everything except the
// 16 x 16 diagonal block of the NEXT panel.  Warp 0: that block (4 mma tiles), then its factorisation (look-ahead): the
// serial part of the next panel step runs underneath the update.
__device__ void pm_trailing(double *L, const int *poff, int mm, int c0, int np, int pb, double *dinv_stage, double *colbuf)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int g = lane >> 2, t4 = lane & 3;
    constexpr int NW = FIT_NT / 32 - 1;
    const int cq = c0 + pb * PNB;
    const int ldq = pm_ld(mm + 1 - cq);
    const double *Pq = L + poff[pb];
    if (wid == 0) {
        const int cj = cq + PNB;
        const int ldj = pm_ld(mm + 1 - cj);
        const int nbj = min(PNB, mm - cj);
        double *Pj = L + poff[pb + 1];
        double acc[2][2][2];
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int nt = 0; nt < 2; nt++) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
        const int hq = mm + 1 - cq;
        const double *pa = Pq + t4 * ldq;  // rows cj + g (+ 8) of panel pb, clamped to its border row
        const int r0 = min(PNB + g, hq - 1), r1 = min(PNB + 8 + g, hq - 1);
#pragma unroll
        for (int q0 = 0; q0 < PNB; q0 += 4) {
            const double f0 = pa[q0 * ldq + r0], f1 = pa[q0 * ldq + r1];
            dmma_m8n8k4(acc[0][0], f0, f0);
            dmma_m8n8k4(acc[0][1], f0, f1);
            dmma_m8n8k4(acc[1][0], f1, f0);
            dmma_m8n8k4(acc[1][1], f1, f1);
        }
#pragma unroll
        for (int mt = 0; mt < 2; mt++)
#pragma unroll
            for (int nt = 0; nt < 2; nt++)
#pragma unroll
                for (int w = 0; w < 2; w++) {
                    const int al = 8 * mt + g, bl = 8 * nt + 2 * t4 + w;
                    if (al < nbj && bl <= al) Pj[bl * ldj + al] -= acc[mt][nt][w];
                }
        __syncwarp();
        pm_diag_factor(Pj, ldj, nbj, dinv_stage + (pb + 1) * PNB, colbuf);
    } else {
        int u = 0;
        for (int pj = pb + 1; pj < np; pj++) {
            const int cj = c0 + pj * PNB;
            const int hj = mm + 1 - cj, ldj = pm_ld(hj);
            const int nbj = min(PNB, mm - cj);
            const int nrb = (hj + 31) >> 5;
            const int alo = pj == pb + 1 ? cj + nbj : cj;  // the next diagonal block is warp 0's
            double *Pj = L + poff[pj];
            for (int rb = (wid - 1 - u % NW + NW) % NW; rb < nrb; rb += NW) {
                const int a0 = cj + 32 * rb;
                double acc[4][2][2];
#pragma unroll
                for (int mt = 0; mt < 4; mt++)
#pragma unroll
                    for (int nt = 0; nt < 2; nt++) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
                pm_mma_panel(acc, Pq, ldq, cq, mm + 1 - cq, a0, cj, g, t4);
#pragma unroll
                for (int mt = 0; mt < 4; mt++)
#pragma unroll
                    for (int nt = 0; nt < 2; nt++)
#pragma unroll
                        for (int w = 0; w < 2; w++) {
                            const int a = a0 + 8 * mt + g, bl = 8 * nt + 2 * t4 + w;
                            if (a >= alo && a <= mm && bl < nbj) Pj[bl * ldj + (a - cj)] -= acc[mt][nt][w];
                        }
            }
            u += nrb;
        }
    }
    __syncthreads();
}
// Schur complement of the columns behind a stage, in place in the global matrix: S[a][b] -= sum over ALL columns q of the
// stage of L[a][q] L[b][q] for b >= c1, a >= b's block.
__device__ void pm_update_global(const double *L, const int *poff, double *Sg, int lds, int mm, int c0, int np)
{
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int g = lane >> 2, t4 = lane & 3;
    constexpr int NW = FIT_NT / 32;
    const int c1 = c0 + np * PNB;
    int u = 0;
    for (int cj = c1; cj < mm; cj += PNB) {
        const int nrb = (mm + 1 - cj + 31) >> 5;
        const int first = (wid - u % NW + NW) % NW;
        for (int rb = first; rb < nrb; rb += NW) {
            const int a0 = cj + 32 * rb;
            double acc[4][2][2];
#pragma unroll
            for (int mt = 0; mt < 4; mt++)
#pragma unroll
                for (int nt = 0; nt < 2; nt++) acc[mt][nt][0] = acc[mt][nt][1] = 0.0;
            for (int pb = 0; pb < np; pb++) {
                const int cq = c0 + pb * PNB;
                pm_mma_panel(acc, L + poff[pb], pm_ld(mm + 1 - cq), cq, mm + 1 - cq, a0, cj, g, t4);
            }
#pragma unroll
            for (int mt = 0; mt < 4; mt++)
#pragma unroll
                for (int nt = 0; nt < 2; nt++) {
                    const int a = a0 + 8 * mt + g, b = cj + 8 * nt + 2 * t4;
                    if (a <= mm) {
                        if (b < mm) Sg[(size_t)a * lds + b] -= acc[mt][nt][0];
                        if (b + 1 < mm) Sg[(size_t)a * lds + b + 1] -= acc[mt][nt][1];
                    }
                }
        }
        u += nrb;
    }
    __syncthreads();
}
// L^T x = z over the columns of the stage in shared memory; x[c] of the later columns is final.
__device__ void pm_backsub(const double *L, const int *poff, int mm, int c0, int np, double *x, double *red /* PNB */,
                           const double *dinv_stage)
{
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ncol = min(np * PNB, mm - c0);
    for (int e = tid; e < ncol; e += FIT_NT) {
        const int pb = e >> 4, q = e & 15, r0 = c0 + pb * PNB;
        x[c0 + e] = L[poff[pb] + q * pm_ld(mm + 1 - r0) + (mm - r0)];  // z = the border row
    }
    __syncthreads();
    for (int pb = np - 1; pb >= 0; pb--) {
        const int r0 = c0 + pb * PNB;
        const int h = mm + 1 - r0, ld = pm_ld(h);
        const int nb = min(PNB, mm - r0);
        const double *P = L + poff[pb];
        if (wid < nb) {  // warp q: v_q = sum_{i > block} L[i][r0 + q] x[i]
            double acc = 0.0;
            for (int i = nb + lane; i < h - 1; i += 32) acc = fma(P[wid * ld + i], x[r0 + i], acc);
            acc = warp_sum(acc);
            if (lane == 0) red[wid] = acc;
        }
        __syncthreads();
        if (wid == 0) {
            double t = 0.0, dinv = 0.0, lrow[PNB];  // lrow[q] = L[r0 + q][r0 + lane] (q > lane)
#pragma unroll
            for (int q = 0; q < PNB; q++) lrow[q] = (lane < q && q < nb) ? P[lane * ld + q] : 0.0;
            if (lane < nb) {
                t = x[r0 + lane] - red[lane];
                dinv = dinv_stage[pb * PNB + lane];
            }
#pragma unroll
            for (int q = PNB - 1; q >= 0; q--) {
                const double yq = __shfl_sync(0xffffffffu, t, q) * __shfl_sync(0xffffffffu, dinv, q);
                if (lane == q) t = yq;
                t = fma(-lrow[q], yq, t);  // lrow[q] == 0 for lane >= q and for q >= nb (then yq == 0 as well)
            }
            if (lane < nb) x[r0 + lane] = t;
        }
        __syncthreads();
    }
}
// Sg: bordered system in global memory (row-major, lower triangle + border row mm); multi-stage runs overwrite it.
// x (shared memory) <- solution.  There is no rank-revealing fallback at this size: a pivot at or below PIVOT_TOL times
// its column's original diagonal entry (tested after the factorisation on dinv = 1 / L_jj, a NaN dinv -- a non-positive
// pivot -- failing too) makes the whole x NaN and counts in g_wide_singular_count, so a singular system never returns a
// finite solution.  The original diagonal is kept in sm.b1, which no caller uses across a solve.
__device__ __noinline__ void chol_panel_major(double *Sg, int lds, int mm, double *x, const FitSmem &sm_, PhaseTimer &pt,
                                              bool preloaded = false)
{
    const FitSmem sm = sm_shared(sm_);
    // Re-derive every shared-memory pointer from the kernel's dynamic shared array: behind the call boundary of this
    // (not inlined) function the compiler would otherwise address them generically (LD.E / ST.E instead of LDS / STS,
    // 64-bit address arithmetic) -- measured 5x slower per DMMA block.
    int *poff = reinterpret_cast<int *>(as_shared(sm.tile));  // header: up to 64 panel offsets | pivot-column buffer
    double *colbuf = as_shared(sm.tile) + 32;                 // 2 * PNB doubles
    double *L = as_shared(sm.tile) + 64;
    double *dg = as_shared(sm.dg);
    double *red = as_shared(sm.red);
    double *diag0 = as_shared(sm.b1);
    x = as_shared(x);
    const int cap = pm_capacity(sm.arena_len);
    int sc0[PM_MAX_STAGES], snp[PM_MAX_STAGES], ns = 0;
    for (int c0 = 0; c0 < mm && ns < PM_MAX_STAGES;) {
        const int np = pm_plan(c0, mm, cap);
        sc0[ns] = c0;
        snp[ns] = np;
        ns++;
        c0 += np * PNB;
    }
    for (int s = 0; s < ns; s++) {
        const int c0 = sc0[s], np = snp[s];
        pm_offsets(poff, mm, c0, np);
        if (!(preloaded && s == 0)) pm_copy<false>(L, poff, Sg, lds, mm, c0, np);  // (reduce_to_panels filled stage 0)
        if (s == 0) {  // stage 0's columns from its panels, the later ones from Sg before the first Schur update
            for (int j = threadIdx.x; j < mm; j += FIT_NT) {
                const int pb = j >> 4, q = j & (PNB - 1);
                diag0[j] = pb < np ? L[poff[pb] + q * pm_ld(mm + 1 - pb * PNB) + q] : Sg[(size_t)j * lds + j];
            }
            __syncthreads();
        }
        pt.mark(10);
        if (threadIdx.x < 32) pm_diag_factor(L + poff[0], pm_ld(mm + 1 - c0), min(PNB, mm - c0), dg + c0, colbuf);
        __syncthreads();
        for (int pb = 0; pb < np; pb++) {
            const int r0 = c0 + pb * PNB;
            const int nb = min(PNB, mm - r0);
            if (nb == PNB) pm_row_solve<true>(L + poff[pb], pm_ld(mm + 1 - r0), mm + 1 - r0, nb, dg + r0);
            else pm_row_solve<false>(L + poff[pb], pm_ld(mm + 1 - r0), mm + 1 - r0, nb, dg + r0);
            pt.mark(13);
            if (pb + 1 < np) pm_trailing(L, poff, mm, c0, np, pb, dg + c0, colbuf);
            pt.mark(14);
        }
        if (s + 1 < ns) {
            pm_update_global(L, poff, Sg, lds, mm, c0, np);
            pm_copy<true>(L, poff, Sg, lds, mm, c0, np);
            pt.mark(11);
        }
    }
    for (int s = ns - 1; s >= 0; s--) {
        const int c0 = sc0[s], np = snp[s];
        if (s != ns - 1) {
            pm_offsets(poff, mm, c0, np);
            pm_copy<false>(L, poff, Sg, lds, mm, c0, np);
        }
        pm_backsub(L, poff, mm, c0, np, x, red, dg + c0);
    }
    // pivot_j = 1 / dinv_j^2 > PIVOT_TOL * diag0_j, written so that a NaN dinv fails
    bool bad = false;
    for (int j = threadIdx.x; j < mm; j += FIT_NT) bad |= !(dg[j] * dg[j] * (PIVOT_TOL * diag0[j]) < 1.0);
    if (__syncthreads_or(bad)) {
        for (int j = threadIdx.x; j < mm; j += FIT_NT) x[j] = __longlong_as_double(0x7ff8000000000000ll);
        if (threadIdx.x == 0) atomicAdd(&g_wide_singular_count, 1ull);
        __syncthreads();
    }
    pt.mark(12);
}

// P[i][q] = S[j0 + i][j0 + q] for i in [i0, i1), q < nb: 8 independent loads in flight per thread
__device__ __forceinline__ void panel_load(double *P, const double *S, int lds, int j0, int i0, int i1, int nb)
{
    constexpr int PS = CHOL_NB + 1;
    const int tot = (i1 - i0) * nb;
    for (int e0 = threadIdx.x; e0 < tot; e0 += 8 * FIT_NT) {
        double val[8];
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int e = e0 + u * FIT_NT;
            if (e < tot) {
                const int i = i0 + e / nb, q = e % nb;
                val[u] = S[(size_t)(j0 + i) * lds + j0 + q];
            }
        }
#pragma unroll
        for (int u = 0; u < 8; u++) {
            const int e = e0 + u * FIT_NT;
            if (e < tot) {
                const int i = i0 + e / nb, q = e % nb;
                P[i * PS + q] = val[u];
            }
        }
    }
}

// Blocked right-looking version for systems that live in global memory (L2), run by the WHOLE cluster: rank 0 factors
// each CHOL_NB-column panel in shared memory (diagonal block by one warp, rows below by one thread each) and writes it
// back; after a cluster barrier every CTA loads the panel and updates its share of the trailing matrix with
// register-blocked 4x4 tiles (read-modify-write in L2); a second barrier publishes the update.  Back substitution on
// rank 0.  x (rank 0's shared memory) <- solution.  With CL == 1 the barriers degenerate to __syncthreads.
__device__ __noinline__ void chol_blocked_cluster(double *S, int lds, int mm, double *x, const FitSmem &sm_, Clu &cl)
{
    const FitSmem sm = sm_shared(sm_);
    constexpr int NB = CHOL_NB, PS = NB + 1;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    double *P = sm.tile;  // panel rows j0..mm, PS doubles each: (mm + 1) * 17 <= FIT_TILE_DOUBLES for mm <= 480
    for (int j0 = 0; j0 < mm; j0 += NB) {
        const int nb = min(NB, mm - j0);
        const int mr = mm + 1 - j0;
        __syncthreads();
        if (cl.rank == 0) {
            panel_load(P, S, lds, j0, 0, mr, nb);
            __syncthreads();
            cl.pt.mark(10);
            panel_factor([&](int i) { return P + i * PS; }, mr, nb, sm.dg);
            cl.pt.mark(12);
            // L panel back to global (the other CTAs and the back substitution read it there)
            for (int e = tid; e < mr * nb; e += FIT_NT) {
                const int i = e / nb, q = e - i * nb;
                if (i >= nb || q <= i) S[(size_t)(j0 + i) * lds + j0 + q] = P[i * PS + q];
            }
        }
        const int t0 = j0 + nb;
        const int mt = mm - t0;  // trailing columns
        if (mt <= 0) break;      // uniform over the cluster
        clu_sync(cl);
        cl.pt.mark(13);
        if (cl.rank != 0) {
            panel_load(P, S, lds, j0, nb, mr, nb);
            __syncthreads();
        }
        // trailing update: S[a][b] -= sum_q P[a][q] P[b][q] for a in [t0, mm], b in [t0, min(a, mm-1)]
        {
            const int rbk = (mt + 1 + 3) >> 2;  // row blocks (incl. the rhs row)
            const int nblk = rbk * (rbk + 1) / 2;
            for (int blk = cl.rank * FIT_NT + tid; blk < nblk; blk += cl.CL * FIT_NT) {
                int bi = (int)((sqrt(8.0 * (double)blk + 1.0) - 1.0) * 0.5);
                while ((bi + 1) * (bi + 2) / 2 <= blk) bi++;
                while (bi * (bi + 1) / 2 > blk) bi--;
                const int bj = blk - bi * (bi + 1) / 2;
                double acc[16];
#pragma unroll
                for (int e = 0; e < 16; e++) acc[e] = 0.0;
                const double *pa = P + (size_t)(nb + 4 * bi) * PS;
                const double *pb = P + (size_t)(nb + 4 * bj) * PS;
                for (int q = 0; q < nb; q++) {
                    double a[4], bb[4];
#pragma unroll
                    for (int u = 0; u < 4; u++) {
                        a[u] = (4 * bi + u <= mt) ? pa[u * PS + q] : 0.0;
                        bb[u] = (4 * bj + u <= mt) ? pb[u * PS + q] : 0.0;
                    }
#pragma unroll
                    for (int qa = 0; qa < 4; qa++)
#pragma unroll
                        for (int qb = 0; qb < 4; qb++) acc[qa * 4 + qb] = fma(a[qa], bb[qb], acc[qa * 4 + qb]);
                }
#pragma unroll
                for (int e = 0; e < 16; e++) {
                    const int a = t0 + 4 * bi + (e >> 2), b = t0 + 4 * bj + (e & 3);
                    if (a <= mm && b < mm && b <= a) S[(size_t)a * lds + b] -= acc[e];
                }
            }
        }
        clu_sync(cl);
        cl.pt.mark(14);
    }
    if (cl.rank != 0) return;
    __syncthreads();
    // back substitution L^T x = z, z = row mm
    for (int c = tid; c < mm; c += FIT_NT) x[c] = S[(size_t)mm * lds + c];
    __syncthreads();
    const int jlast = ((mm - 1) / NB) * NB;
    for (int j0 = jlast; j0 >= 0; j0 -= NB) {
        const int nb = min(NB, mm - j0);
        const int t0 = j0 + nb;
        // v[q] = sum_{i in [t0, mm)} L[i][j0+q] x[i]: thread (q = tid & 15, g = tid >> 4) sums the rows i == g (mod 32)
        __syncthreads();
        {
            const int q = tid & (NB - 1), g = tid >> 4;
            double acc = 0.0;
            if (q < nb)
                for (int i = t0 + g; i < mm; i += FIT_NT / NB) acc = fma(S[(size_t)i * lds + j0 + q], x[i], acc);
            sm.scratch[g * NB + q] = acc;
        }
        // diagonal block to smem
        for (int e = tid; e < nb * nb; e += FIT_NT) {
            const int i = e / nb, q = e - i * nb;
            P[i * PS + q] = q <= i ? S[(size_t)(j0 + i) * lds + j0 + q] : 0.0;
        }
        __syncthreads();
        if (wid == 0) {
            double t = 0.0;
            if (lane < nb) {
                double vsum = 0.0;
                for (int g2 = 0; g2 < FIT_NT / NB; g2++) vsum += sm.scratch[g2 * NB + lane];
                t = x[j0 + lane] - vsum;
            }
            for (int q = nb - 1; q >= 0; q--) {
                const double yq = __shfl_sync(0xffffffffu, t, q) / P[q * PS + q];
                if (lane == q) t = yq;
                if (lane < q) t -= P[q * PS + lane] * yq;
            }
            if (lane < nb) x[j0 + lane] = t;
        }
        __syncthreads();
    }
}

// Systems of up to 31 unknowns (most fits of the path: config 3's poisson levels, config 4's Cox Newton steps, every small
// gaussian support): ONE warp, lane r holds row r of the bordered system in registers (row nu = right-hand side).  Per
// column: the pivot by shuffle, rsqrt (hardware approximation + two Newton steps), the scaled column published through 32
// shared doubles, every lane updates its own row -- no block barrier anywhere (the CTA-wide unblocked version this replaces
// paid two per column: 16 us at 40 unknowns, measured 4 us here).  The pivots are tested against PIVOT_TOL of the
// column's own diagonal entry; S itself is never written (the factor lives in a side buffer), so
// a rank-deficient system goes to the rank-revealing fallback untouched.  work: 32 * 33 + 32 doubles of shared scratch.
__device__ __noinline__ bool warp_chol_solve32(const double *S, int lds, int nu, double *x, double *work)
{
    constexpr int LS = 33;  // row stride of the factor buffer: a lane reading its own row never shares a bank
    const int lane = threadIdx.x & 31;
    S = as_shared(S);
    x = as_shared(x);
    double *Lb = as_shared(work);      // [32][LS] the factor (row nu: z = L^{-1} rhs)
    double *cb = Lb + 32 * LS;         // [2][16] pivot column of the running step
    const double diag0 = lane < nu ? S[lane * lds + lane] : 1.0;
    double dinv = 0.0;  // lane j: 1 / L_jj
    bool ok = true;
    // two panels of 16 columns: 16 doubles of a row in registers at a time (a whole 32-column row per lane spilled)
    for (int c0 = 0; c0 < nu; c0 += PNB) {
        const int nb = min(PNB, nu - c0);
        double a[PNB];
#pragma unroll
        for (int c = 0; c < PNB; c++) a[c] = (lane <= nu && c < nb && c0 + c <= lane) ? S[lane * lds + c0 + c] : 0.0;
        // left-looking update with the columns factored so far: a[c] -= sum_q L[lane][q] L[c0 + c][q]
        for (int q = 0; q < c0; q++) {
            const double lrq = Lb[lane * LS + q];
#pragma unroll
            for (int c = 0; c < PNB; c++) a[c] = fma(-lrq, Lb[(c0 + c) * LS + q], a[c]);
        }
#pragma unroll
        for (int q = 0; q < PNB; q++) {
            if (q < nb) {  // uniform
                const int j = c0 + q;
                const double d = __shfl_sync(0xffffffffu, a[q], j);
                if (!(d > PIVOT_TOL * __shfl_sync(0xffffffffu, diag0, j))) ok = false;  // the same on every lane
                const double inv = pm_rsqrt(d);
                const double lq = lane == j ? d * inv : a[q] * inv;
                a[q] = lq;
                if (lane == j) dinv = inv;
                double *cq = cb + (q & 1) * PNB;
                if (lane >= c0 && lane < c0 + PNB) cq[lane - c0] = lq;  // L[c0 + c][j] for the rows of this diagonal block
                __syncwarp();
#pragma unroll
                for (int c = q + 1; c < PNB; c++) a[c] = fma(-lq, cq[c], a[c]);  // (only rows >= c0 + c use the result)
            }
        }
#pragma unroll
        for (int c = 0; c < PNB; c++) Lb[lane * LS + c0 + c] = a[c];
        __syncwarp();
    }
    if (!ok) return false;
    // L^T x = z with lane c owning x_c
    double z = lane < nu ? Lb[nu * LS + lane] : 0.0;
    for (int j = nu - 1; j >= 0; j--) {
        const double xj = __shfl_sync(0xffffffffu, z, j) * __shfl_sync(0xffffffffu, dinv, j);
        const double ljc = lane < j ? Lb[j * LS + lane] : 0.0;
        z = lane == j ? xj : fma(-ljc, xj, z);
    }
    if (lane < nu) x[lane] = z;
    __syncwarp();
    return true;
}

// Which solver finished a normal-equation solve (solve_on_rank0's return value, reported by the solve probe).
enum {
    SOLVE_WARP = 1, SOLVE_WARP_LDLT = 2,   // warp_chol_solve32, and its rank-revealing fallback
    SOLVE_SMEM = 3, SOLVE_SMEM_LDLT = 4,   // block_chol_solve_small, and its rank-revealing fallback
    SOLVE_PANEL = 10,                      // + the stage count: chol_panel_major in 1 .. PM_MAX_STAGES stages
    SOLVE_PACKED = 30,                     // chol_packed_smem
    SOLVE_CLUSTER = 40                     // chol_blocked_cluster (the whole cluster; never from solve_on_rank0)
};
// Every solver except chol_blocked_cluster runs on rank 0 alone.
__device__ __forceinline__ bool solved_on_rank0(const double *S, int nu, const FitSmem &sm)
{
    return S == sm.Ssm || (g_dbg_solver == 0 && nu < FIT_NT && pm_stage_count(nu, sm.arena_len) <= PM_MAX_STAGES) ||
           packed_fits(nu, sm.arena_len);
}
// The solve of a bordered system (nu unknowns) at S when solved_on_rank0(): x -> sm.rhs.  Run by every thread of rank 0.
__device__ __forceinline__ int solve_on_rank0(double *S, int lds, int nu, const FitSmem &sm_, PhaseTimer &pt, bool preloaded)
{
    const FitSmem sm = sm_shared(sm_);
    if (S == sm.Ssm) {
        if (nu <= 31 && g_dbg_solver == 0) {
            // one warp, rows in registers; S stays intact unless every pivot passes
            int *okf = reinterpret_cast<int *>(sm.red);
            __syncthreads();
            if (threadIdx.x < 32) {
                const bool ok = warp_chol_solve32(S, lds, nu, sm.rhs, sm.tile);
                if (threadIdx.x == 0) *okf = ok ? 1 : 0;
            }
            __syncthreads();
            if (!*okf) {
                double *S0 = sm.scratch;
                for (int e = threadIdx.x; e < (nu + 1) * lds; e += FIT_NT) S0[e] = S[e];
                __syncthreads();
                ldlt_pivoted_small(S, lds, nu, sm.rhs, S0, sm.tile);
                return SOLVE_WARP_LDLT;
            }
            return SOLVE_WARP;
        }
        // pristine copy (the scratch region is free here): the pivot test of the factorisation compares against it,
        // and a rank-deficient system is solved again from it by the rank-revealing fallback
        double *S0 = sm.scratch;
        __syncthreads();
        for (int e = threadIdx.x; e < (nu + 1) * lds; e += FIT_NT) S0[e] = S[e];
        __syncthreads();
        if (!block_chol_solve_small(S, lds, nu, sm.rhs, sm.dg, S0)) {
            __syncthreads();
            for (int e = threadIdx.x; e < (nu + 1) * lds; e += FIT_NT) S[e] = S0[e];
            __syncthreads();
            ldlt_pivoted_small(S, lds, nu, sm.rhs, S0, sm.tile);
            return SOLVE_SMEM_LDLT;
        }
        return SOLVE_SMEM;
    }
    if (g_dbg_solver == 0 && nu < FIT_NT) {
        const int ns = pm_stage_count(nu, sm.arena_len);
        if (ns <= PM_MAX_STAGES) {
            chol_panel_major(S, lds, nu, sm.rhs, sm, pt, preloaded);
            return SOLVE_PANEL + ns;
        }
    }
    chol_packed_smem(S, lds, nu, sm.rhs, sm, pt);
    return SOLVE_PACKED;
}

// Rank 0 holds a bordered system (nu unknowns) at S -- its own shared memory (small systems) or the chain's global matrix
// (large systems, then every CTA of the cluster takes part in the factorisation): solve it and hand the solution to
// every CTA of the cluster (out: smem).
__device__ void solve_broadcast(const ChainCtx &cx, Clu &cl, double *S, int lds, int nu, double *out, const FitSmem &sm_,
                                bool preloaded = false)
{
    const FitSmem sm = sm_shared(sm_);
    out = as_shared(out);
    if (solved_on_rank0(S, nu, sm)) {
        if (cl.rank == 0) solve_on_rank0(S, lds, nu, sm, cl.pt, preloaded);
    } else {
        chol_blocked_cluster(S, lds, nu, sm.rhs, sm, cl);
    }
    cl.pt.mark(PH_CHOL);  // small systems: the whole solve; blocked: the back substitution (phases 10-14 = panels)
    if (cl.rank == 0 && cl.CL > 1) {
        double *bc = cw_slot(cx, 0, 2);
        for (int a = threadIdx.x; a < nu; a += FIT_NT) bc[a] = sm.rhs[a];
    }
    if (cl.CL > 1) {
        clu_sync(cl);
        const double *bc = cw_slot(cx, 0, 2);
        for (int a = threadIdx.x; a < nu; a += FIT_NT) out[a] = bc[a];
    } else {
        for (int a = threadIdx.x; a < nu; a += FIT_NT) out[a] = sm.rhs[a];
    }
    __syncthreads();
    cl.pt.mark(PH_BCAST);
}

// Cluster mode: Sfin[a][b] = sum_q P_q[0][a][b] (- sum_q P_q[1][a][b] when nmat == 2) for a < rows, b < cols, each CTA
// reducing a slab of rows, ranks summed in a fixed order; optional extra row `rows` = sum_q cw_slot(q, 1) (Cox gradient).
// Ends with a cluster barrier; afterwards rank 0 stages the system where it will factor it and returns that pointer.
// Cluster mode, wide systems that the panel-major solver factors in ONE stage: the per-CTA partial Grams are reduced
// straight into rank 0's shared memory, already in panel-major layout -- every CTA of the cluster sums its share of the
// lower triangle (4-row x 8-column patches dealt round robin over all warps of the cluster, ranks added in a fixed
// order) and stores the results through distributed shared memory.  Replaces a full-square reduction into global memory
// plus rank 0's load of the result (12.5 + 10 us per IRLS step at 200 unknowns).  Ends with a cluster barrier.
__device__ void reduce_to_panels(const ChainCtx &cx, Clu &cl, int rows, int nmat, bool extra_row, const FitSmem &sm,
                                 double diag_add, int diag_from, int diag_to)
{
    const int ldA = cx.ldA;
    const int brows = rows + (extra_row ? 1 : 0), nu = brows - 1;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int il = lane >> 3, cl8 = lane & 7;
    constexpr int NWC = FIT_NT / 32;
    const int np = (nu + PNB - 1) / PNB;
    int *poff = reinterpret_cast<int *>(sm.tile);
    pm_offsets(poff, nu, 0, np);
    double *L0 = cg::this_cluster().map_shared_rank(sm.tile + 64, 0);  // rank 0's panel storage (same carve in every CTA)
    const int nwarps = cl.CL * NWC, gw = cl.rank * NWC + wid;
    int u = 0;
    for (int pb = 0; pb < np; pb++) {
        const int r0 = pb * PNB;
        const int h = nu + 1 - r0, ld = pm_ld(h);
        const int nb = min(PNB, nu - r0);
        double *P = L0 + poff[pb];
        const int npatch = 2 * ((h + 3) >> 2);
        for (int pa = (gw - u % nwarps + nwarps) % nwarps; pa < npatch; pa += nwarps) {
            const int i = (pa >> 1) * 4 + il, c = (pa & 1) * 8 + cl8;
            if (i >= h) continue;
            double v = 0.0;
            if (c < nb) {
                const int a = r0 + i, b = r0 + c;
                if (a < rows) {
                    const size_t o = (size_t)a * ldA + b;
                    for (int q = 0; q < cl.CL; q++) v += cx.Sp0[q * cx.sp_stride + o];
                    if (nmat == 2) {
                        double s2 = 0.0;
                        for (int q = 0; q < cl.CL; q++) s2 += cx.Sp0[q * cx.sp_stride + (size_t)ldA * ldA + o];
                        v -= s2;
                    }
                    if (a == b && a >= diag_from && a < diag_to) v += diag_add;
                } else {  // the extra border row (cox gradient)
                    for (int q = 0; q < cl.CL; q++) v += cw_slot(cx, q, 1)[b];
                }
            }
            P[c * ld + i] = v;
        }
        u += npatch;
    }
    clu_sync(cl);
}

__device__ double *reduce_partials(const ChainCtx &cx, Clu &cl, int rows, int cols, int nmat, bool extra_row, int *lds_out,
                                   const FitSmem &sm_, double diag_add = 0.0, int diag_from = 0, int diag_to = 0,
                                   bool *preloaded = nullptr)
{
    const FitSmem sm = sm_shared(sm_);
    const int ldA = cx.ldA;
    {
        const int nu = rows + (extra_row ? 1 : 0) - 1;
        if (preloaded) *preloaded = false;
        if (preloaded && nu + 1 > FIT_SMEM_MS && g_dbg_solver == 0 && nu < FIT_NT && pm_stage_count(nu, sm.arena_len) == 1) {
            reduce_to_panels(cx, cl, rows, nmat, extra_row, sm, diag_add, diag_from, diag_to);
            *preloaded = true;
            *lds_out = ldA;
            return cx.Sfin;
        }
    }
    const int per = (rows + cl.CL - 1) / cl.CL;
    const int a0 = cl.rank * per, a1 = min(rows, a0 + per);
    const int cnt = max(0, a1 - a0) * cols;
    for (int e = threadIdx.x; e < cnt; e += FIT_NT) {
        const int a = a0 + e / cols, b = e % cols;
        const size_t o = (size_t)a * ldA + b;
        double s = 0.0;
        for (int q = 0; q < cl.CL; q++) s += cx.Sp0[q * cx.sp_stride + o];
        if (nmat == 2) {
            double s2 = 0.0;
            for (int q = 0; q < cl.CL; q++) s2 += cx.Sp0[q * cx.sp_stride + (size_t)ldA * ldA + o];
            s -= s2;
        }
        if (a == b && a >= diag_from && a < diag_to) s += diag_add;
        cx.Sfin[o] = s;
    }
    if (extra_row && cl.rank == cl.CL - 1) {
        for (int b = threadIdx.x; b < cols; b += FIT_NT) {
            double s = 0.0;
            for (int q = 0; q < cl.CL; q++) s += cw_slot(cx, q, 1)[b];
            cx.Sfin[(size_t)rows * ldA + b] = s;
        }
    }
    clu_sync(cl);
    const int brows = rows + (extra_row ? 1 : 0);  // bordered system: brows rows, brows - 1 unknowns
    if (brows <= FIT_SMEM_MS) {
        if (cl.rank == 0) {
            for (int e = threadIdx.x; e < brows * cols; e += FIT_NT) {
                const int a = e / cols, b = e % cols;
                sm.Ssm[a * FIT_SMEM_MS + b] = cx.Sfin[(size_t)a * ldA + b];
            }
            __syncthreads();
        }
        *lds_out = FIT_SMEM_MS;
        return sm.Ssm;
    }
    *lds_out = ldA;
    return cx.Sfin;
}

// Weighted Gram of columns [0, mm) of V over ALL train rows of the chain, then solve for the first mm-1 unknowns with
// row mm-1 as right-hand side:  S = sum_r wt[r] V[r][a] V[r][b];  S[0:mm-1, 0:mm-1] x = S[mm-1, 0:mm-1].
// out (shared memory of every CTA) <- x.
__device__ void gram_solve(const ChainCtx &cx, Clu &cl, const double *V, int ldv, int mm, const double *wt, double *out,
                           const FitSmem &sm_, double diag_add = 0.0, int diag_from = 0)
{
    const FitSmem sm = sm_shared(sm_);
    out = as_shared(out);
    cl.pt.mark(PH_OTHER);
    if (cl.CL == 1) {
        gram(V, ldv, cx.rb, cx.re, mm, wt, cx.S, cx.lds, sm);
        if (diag_add != 0.0) {  // ridge term on the unknowns [diag_from, mm - 1)
            for (int a = diag_from + threadIdx.x; a < mm - 1; a += FIT_NT) cx.S[(size_t)a * cx.lds + a] += diag_add;
            __syncthreads();
        }
        cl.pt.mark(PH_SYRK);
        solve_broadcast(cx, cl, cx.S, cx.lds, mm - 1, out, sm);
        return;
    }
    gram(V, ldv, cx.rb, cx.re, mm, wt, cx.Sp0 + cl.rank * cx.sp_stride, cx.ldA, sm);
    clu_sync(cl);
    cl.pt.mark(PH_SYRK);
    int lds;
    bool preloaded;
    double *S = reduce_partials(cx, cl, mm, mm, 1, false, &lds, sm, diag_add, diag_from, mm - 1, &preloaded);
    cl.pt.mark(PH_REDUCE);
    solve_broadcast(cx, cl, S, lds, mm - 1, out, sm, preloaded);
}

__device__ __forceinline__ double row_dot(const double *row, const double *b, int m)
{
    double s = 0.0;
    for (int a = 0; a < m; a++) s = fma(row[a], b[a], s);
    return s;
}
// Linear predictor of the CTA's row slice: f(r, X_A[r] . beta) for every row r, called by the lane that owns the row.
// Groups of 8 consecutive rows are dealt round robin to the 16 warps; a warp walks its 8 rows with coalesced loads
// (lane = column mod 32, 16 loads in flight per lane), a butterfly sum per row, and parks the results on distinct lanes
// until 32 rows are ready for f -- the thread-per-row walk this replaces read every row as a serial chain of 32-byte
// sectors (26 us per IRLS step at 225 rows x 203 columns; fixed summation order either way).
template <class F>
__device__ __forceinline__ void rows_dot(const ChainCtx &cx, const double *beta, int m, F f)
{
    constexpr int GR = 8;
    if (m < 64) {  // narrow supports: a thread per row, the row's few sectors stay in L1 between its loads
        for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) f(r, row_dot(cx.XA + (size_t)r * cx.ldA, beta, m));
        return;
    }
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int ngroups = (cx.re - cx.rb + GR - 1) / GR;
    double mine = 0.0;
    int myrow = -1, slot = 0;
    for (int gi = wid; gi < ngroups; gi += FIT_NT / 32) {
        const int rbase = cx.rb + gi * GR;
        const int nr = min(GR, cx.re - rbase);
        const double *row = cx.XA + (size_t)rbase * cx.ldA;
        double sacc[GR];
#pragma unroll
        for (int u = 0; u < GR; u++) sacc[u] = 0.0;
#pragma unroll 4
        for (int a = lane; a < m; a += 32) {
            const double bv = beta[a];
#pragma unroll
            for (int u = 0; u < GR; u++)
                if (u < nr) sacc[u] = fma(row[(size_t)u * cx.ldA + a], bv, sacc[u]);
        }
#pragma unroll
        for (int u = 0; u < GR; u++) {
            const double t = warp_sum(sacc[u]);
            if (lane == slot * GR + u && u < nr) {
                mine = t;
                myrow = rbase + u;
            }
        }
        if (++slot == 32 / GR) {
            if (myrow >= 0) f(myrow, mine);
            slot = 0;
            myrow = -1;
        }
    }
    if (myrow >= 0) f(myrow, mine);
}

// ---- gaussian: Algorithm.h:1131-1135
__device__ void fit_lm(const ChainCtx &cx, Clu &cl, const FitSmem &sm_, double *beta_out, double lambda)
{
    const FitSmem sm = sm_shared(sm_);
    beta_out = as_shared(beta_out);
    const int T = cx.T, ldA = cx.ldA;
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) cx.XA[(size_t)r * ldA + T] = cx.y[r];
    __syncthreads();
    gram_solve(cx, cl, cx.XA, ldA, T + 1, nullptr, beta_out, sm, lambda, 0);  // X'X + lambda*I (Algorithm.h:1134)
}

// ---- binomial: Algorithm.h:1148-1204.  Design columns: [1 | X_A | z]
__device__ double logit_eval(const ChainCtx &cx, Clu &cl, const double *beta, const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    beta = as_shared(beta);
    double ll = 0.0;
    rows_dot(cx, beta, cx.m, [&](int r, double eu) {
        const double e = exp(clampd(eu, 30.0));
        const double pi = e / (1.0 + e);
        cx.v[0][r] = eu;
        cx.v[1][r] = pi;
        ll += (cx.y[r] * log(pi) + (1.0 - cx.y[r]) * log(1.0 - pi)) * cx.w[r];
    });
    const double r = clu_allsum(cl, block_sum<FIT_NT>(ll, sm.red));
    cl.pt.mark(PH_EVAL);
    return r;
}
__device__ void logit_wz(const ChainCtx &cx, bool floor_w)
{
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) {
        const double pi = cx.v[1][r];
        double W = pi * (1.0 - pi);
        if (floor_w && W < 0.001) W = 0.001;
        cx.XA[(size_t)r * cx.ldA + cx.m] = cx.v[0][r] + (cx.y[r] - pi) / W;
        cx.v[2][r] = W * cx.w[r];
    }
    __syncthreads();
}
__device__ void fit_logistic(const ChainCtx &cx, Clu &cl, const FitSmem &sm_, double lambda)
{
    const FitSmem sm = sm_shared(sm_);
    double *b0 = sm.b0, *b1 = sm.b1;
    for (int a = threadIdx.x; a < cx.m; a += FIT_NT) b0[a] = 0.0;
    __syncthreads();
    double ll0 = logit_eval(cx, cl, b0, sm);
    logit_wz(cx, false);
    cl.pt.mark(PH_WZ);
    gram_solve(cx, cl, cx.XA, cx.ldA, cx.m + 1, cx.v[2], b1, sm, 2.0 * lambda, 1);  // + 2*lambda*lambdamat, intercept free
    for (int j = 0; j < 30; j++) {
        const double ll1 = logit_eval(cx, cl, b1, sm);
        if (fabs(ll0 - ll1) / (0.1 + fabs(ll1)) < 1e-6) break;
        for (int a = threadIdx.x; a < cx.m; a += FIT_NT) b0[a] = b1[a];
        ll0 = ll1;
        __syncthreads();
        logit_wz(cx, true);
        cl.pt.mark(PH_WZ);
        gram_solve(cx, cl, cx.XA, cx.ldA, cx.m + 1, cx.v[2], b1, sm, 2.0 * lambda, 1);  // + 2*lambda*lambdamat, intercept free
    }
    // result: b0 (the iterate before the last solve)
}

// ---- poisson: Algorithm.h:1273-1322
__device__ void fit_poisson(const ChainCtx &cx, Clu &cl, double coef0_in, const FitSmem &sm_, double lambda)
{
    const FitSmem sm = sm_shared(sm_);
    double *b0 = sm.b0;
    const int ldA = cx.ldA;
    for (int a = threadIdx.x; a < cx.m; a += FIT_NT) b0[a] = a == 0 ? coef0_in : 0.0;
    __syncthreads();
    rows_dot(cx, b0, cx.m, [&](int r, double eta) {
        cx.v[0][r] = eta;
        cx.v[1][r] = exp(eta);
    });
    __syncthreads();
    double ll0 = 1e5;
    for (int j = 0; j < 50; j++) {
        for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) {
            const double e = cx.v[1][r];
            cx.v[2][r] = e * cx.w[r];
            cx.XA[(size_t)r * ldA + cx.m] = cx.v[0][r] + (cx.y[r] - e) / e;
        }
        __syncthreads();
        gram_solve(cx, cl, cx.XA, ldA, cx.m + 1, cx.v[2], b0, sm, 2.0 * lambda, 1);
        double ll = 0.0;
        rows_dot(cx, b0, cx.m, [&](int r, double dot) {
            const double eta = clampd(dot, 30.0);
            double e = exp(eta);
            if (e < 0.001) e = 0.001;
            cx.v[0][r] = eta;
            cx.v[1][r] = e;
            ll += (cx.y[r] * eta - e) * cx.w[r];
        });
        const double ll1 = clu_allsum(cl, block_sum<FIT_NT>(ll, sm.red));
        if (fabs(ll0 - ll1) / fabs(0.1 + ll0) < 1e-6) break;
        ll0 = ll1;
    }
}

// ---- scans over the chain's rows, cut into the cluster's contiguous slices.  v is global, indexed by absolute row.
// suffix: v[r] <- sum_{k >= r} v[k];  prefix: v[r] <- sum_{k <= r} v[k].  The slice total is carried from rank to rank by
// ADDITION only (risk sets span e^+-30: never subtract, see block_excl_scan).
__device__ void clu_suffix_scan(const ChainCtx &cx, Clu &cl, double *v, const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    const int nr = cx.re - cx.rb;
    block_suffix_scan<FIT_NT>(v + cx.rb, nr, sm.red);
    if (cl.CL == 1) return;
    double tot[CLMAX];
    clu_allgather(cl, nr > 0 ? v[cx.rb] : 0.0, tot);
    double carry = 0.0;
#pragma unroll
    for (int q = CLMAX - 1; q >= 0; q--)
        if (q < cl.CL && q > cl.rank) carry += tot[q];
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) v[r] += carry;
    __syncthreads();
}
__device__ void clu_prefix_scan(const ChainCtx &cx, Clu &cl, double *v, const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    const int nr = cx.re - cx.rb;
    block_prefix_scan<FIT_NT>(v + cx.rb, nr, sm.red);
    if (cl.CL == 1) return;
    double tot[CLMAX];
    clu_allgather(cl, nr > 0 ? v[cx.re - 1] : 0.0, tot);
    double carry = 0.0;
#pragma unroll
    for (int q = 0; q < CLMAX; q++)
        if (q < cl.rank) carry += tot[q];
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) v[r] += carry;
    __syncthreads();
}

// ---- cox: Algorithm.h:1377-1490 (+ loglik_cox, coxph.cpp:16-40)
// loglik at beta: theta = exp(clip(X_A beta)), S0 = suffix(theta); sum status*w*log(theta/S0)
__device__ double cox_loglik(const ChainCtx &cx, Clu &cl, const double *beta, double *th, double *s0, const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    beta = as_shared(beta);
    rows_dot(cx, beta, cx.m, [&](int r, double dot) {
        const double t = exp(clampd(dot, 30.0));
        th[r] = t;
        s0[r] = t;
    });
    __syncthreads();
    clu_suffix_scan(cx, cl, s0, sm);
    double ll = 0.0;
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) ll += log(th[r] / s0[r]) * cx.y[r] * cx.w[r];
    return clu_allsum(cl, block_sum<FIT_NT>(ll, sm.red));
}
// XB[r][a] = suffix_r(theta * XA[.][a]) / S0[r]   (risk-set means), chunked two-pass scan over the slice's rows with the
// column totals of the later slices carried in
__device__ void cox_riskset_means(const ChainCtx &cx, Clu &cl, double *XB, const double *th, const double *s0,
                                  const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    const int m = cx.m, ldA = cx.ldA;
    const int nr = cx.re - cx.rb;
    // rows per chunk: chunk sums [nch][m] must fit the scratch region (FIT_NT*16 doubles)
    const int nch_max = max(1, (FIT_NT * 16) / m);
    const int CH = max(32, (nr + nch_max - 1) / nch_max);
    const int nch = (nr + CH - 1) / CH;
    double *csum = sm.scratch;  // [nch][m]
    for (int it = threadIdx.x; it < nch * m; it += FIT_NT) {
        const int ch = it / m, a = it % m;
        const int rb = cx.rb + ch * CH, re = min(cx.re, rb + CH);
        double s = 0.0;
        for (int r = re - 1; r >= rb; r--) s += th[r] * cx.XA[(size_t)r * ldA + a];
        csum[it] = s;
    }
    __syncthreads();
    if (cl.CL > 1) {  // publish this slice's column totals
        double *mine = cw_slot(cx, cl.rank, 0);
        for (int a = threadIdx.x; a < m; a += FIT_NT) {
            double s = 0.0;
            for (int ch = nch - 1; ch >= 0; ch--) s += csum[ch * m + a];
            mine[a] = s;
        }
        clu_sync(cl);
    }
    // exclusive suffix over chunks per column (sequential over nch, parallel over columns)
    for (int a = threadIdx.x; a < m; a += FIT_NT) {
        double run = 0.0;
        for (int q = cl.CL - 1; q > cl.rank; q--) run += cw_slot(cx, q, 0)[a];
        for (int ch = nch - 1; ch >= 0; ch--) {
            const double t = csum[ch * m + a];
            csum[ch * m + a] = run;
            run += t;
        }
    }
    __syncthreads();
    for (int it = threadIdx.x; it < nch * m; it += FIT_NT) {
        const int ch = it / m, a = it % m;
        const int rb = cx.rb + ch * CH, re = min(cx.re, rb + CH);
        double s = csum[it];
        for (int r = re - 1; r >= rb; r--) {
            s += th[r] * cx.XA[(size_t)r * ldA + a];
            XB[(size_t)r * ldA + a] = s / s0[r];
        }
    }
    __syncthreads();
}
__device__ int g_dbg_cox_iters = 30;  // debug knob (bess_b200_debug_set key 1); 30 = reference behaviour
__device__ void fit_cox(const ChainCtx &cx, Clu &cl, double *XB, const FitSmem &sm_, double lambda)
{
    const FitSmem sm = sm_shared(sm_);
    const int max_newton = g_dbg_cox_iters;
    const int m = cx.m, ldA = cx.ldA;
    double *b0 = sm.b0, *b1 = sm.b1;
    double *th = cx.v[0], *s0 = cx.v[1], *ev = cx.v[2], *om = cx.v[3], *gv = cx.v[4];
    for (int a = threadIdx.x; a < m; a += FIT_NT) b0[a] = 0.0;
    __syncthreads();
    double ll0 = 1e5;
    for (int l = 1; l <= max_newton; l++) {
        // theta (no weights here, Algorithm.h:1423), S0
        rows_dot(cx, b0, m, [&](int r, double dot) {
            const double t = exp(clampd(dot, 30.0));
            th[r] = t;
            s0[r] = t;
        });
        __syncthreads();
        clu_suffix_scan(cx, cl, s0, sm);
        // e = w*status; C = prefix(e/S0); omega = theta*C; gvec = e - omega
        for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) {
            ev[r] = cx.w[r] * cx.y[r];
            om[r] = ev[r] / s0[r];
        }
        __syncthreads();
        clu_prefix_scan(cx, cl, om, sm);
        for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) {
            om[r] *= th[r];
            gv[r] = ev[r] - om[r];
        }
        __syncthreads();
        cox_riskset_means(cx, cl, XB, th, s0, sm);
        // -h = P1 - P2,  P1 = X_A^T diag(omega) X_A,  P2 = XB^T diag(e) XB;  g = X_A^T gv
        double *P1 = cl.CL == 1 ? cx.S : cx.Sp0 + cl.rank * cx.sp_stride;
        double *P2 = cl.CL == 1 ? cx.Sfin + (size_t)ldA * ldA : P1 + (size_t)ldA * ldA;
        const int ld1 = cl.CL == 1 ? cx.lds : ldA;
        gram(cx.XA, ldA, cx.rb, cx.re, m, om, P1, ld1, sm);
        gram(XB, ldA, cx.rb, cx.re, m, ev, P2, ldA, sm);
        {
            // g_a = sum_r XA[r][a]*gv[r] over the slice: (a, sub-slice) decomposition, deterministic reduction
            const int nsl = max(1, FIT_NT / m);
            for (int it = threadIdx.x; it < m * nsl; it += FIT_NT) {
                const int a = it % m, sl = it / m;
                double s = 0.0;
                for (int r = cx.rb + sl; r < cx.re; r += nsl) s = fma(cx.XA[(size_t)r * ldA + a], gv[r], s);
                sm.scratch[it] = s;
            }
            __syncthreads();
            double *gdst = cl.CL == 1 ? cx.S + (size_t)m * cx.lds : cw_slot(cx, cl.rank, 1);
            for (int a = threadIdx.x; a < m; a += FIT_NT) {
                double s = 0.0;
                for (int sl = 0; sl < nsl; sl++)
                    if (a + sl * m < m * nsl) s += sm.scratch[sl * m + a];
                // + 2*lambda*beta0 (Algorithm.h:1429); in cluster mode rank 0's share carries it
                if (cl.rank == 0) s += 2.0 * lambda * b0[a];
                gdst[a] = s;  // CL == 1: row m of the bordered system
            }
            __syncthreads();
        }
        double *S;
        int lds;
        bool preloaded = false;
        if (cl.CL == 1) {
            for (int it = threadIdx.x; it < m * m; it += FIT_NT) {
                const int a = it / m, bcol = it % m;
                cx.S[(size_t)a * cx.lds + bcol] -= P2[(size_t)a * ldA + bcol];
                // h + 2*lambda*I on the reference's negative-definite h (Algorithm.h:1472)  <=>  P - 2*lambda*I here
                if (a == bcol) cx.S[(size_t)a * cx.lds + bcol] -= 2.0 * lambda;
            }
            __syncthreads();
            S = cx.S;
            lds = cx.lds;
        } else {
            clu_sync(cl);
            S = reduce_partials(cx, cl, m, m, 2, true, &lds, sm, -2.0 * lambda, 0, m, &preloaded);
        }
        // P d' = g  (d' = -d of Algorithm.h:1472)
        solve_broadcast(cx, cl, S, lds, m, sm.rhs, sm, preloaded);
        // line search (Algorithm.h:1474-1481): beta1 = beta0 - 0.5^mm * d = beta0 + 0.5^mm * rhs
        int mm = 1;
        double step = 0.5;
        for (int a = threadIdx.x; a < m; a += FIT_NT) b1[a] = b0[a] + step * sm.rhs[a];
        __syncthreads();
        double ll1 = cox_loglik(cx, cl, b1, cx.v[5], cx.v[6], sm);
        while (ll0 > ll1 && mm < 5) {
            mm++;
            step *= 0.5;
            __syncthreads();
            for (int a = threadIdx.x; a < m; a += FIT_NT) b1[a] = b0[a] + step * sm.rhs[a];
            __syncthreads();
            ll1 = cox_loglik(cx, cl, b1, cx.v[5], cx.v[6], sm);
        }
        if (fabs(ll0 - ll1) / fabs(0.1 + ll0) < 1e-5) break;
        __syncthreads();
        for (int a = threadIdx.x; a < m; a += FIT_NT) b0[a] = b1[a];
        ll0 = ll1;
        __syncthreads();
    }
}

// Gradient vectors of the next dual sweep from the chain's current (A, beta_A, coef0); X_A is in cx.XA.
__device__ void chain_gradient(const Dev &d, const ChainCtx &cx, Clu &cl, const double *bsl /*smem slopes*/, int ks,
                               double coef0, const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    bsl = as_shared(bsl);
    const int c = cx.c, FS = d.FS, nt = cx.nt;
    const int *rows = d.rows + (size_t)c * d.n;
    const int fam = d.family;
    if (fam != FAM_COX) {
        for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) {
            double eta = coef0;
            const double *row = cx.XA + (size_t)r * d.ldA + cx.off;
            for (int a = 0; a < ks; a++) eta = fma(row[a], bsl[a], eta);
            const size_t o = (size_t)rows[r] * FS + c;
            if (fam == FAM_LM) {
                d.G[o] = (cx.y[r] - eta) / (double)nt;  // Algorithm.h:1109 (coef0 == 0 for gaussian)
            } else if (fam == FAM_LOGIT) {
                const double e = exp(clampd(eta, 30.0));  // Algorithm.h:1223-1236
                const double pr = e / (e + 1.0);
                d.G[o] = cx.w[r] * (cx.y[r] - pr);
                d.W[o] = cx.w[r] * pr * (1.0 - pr);
            } else {
                const double e = exp(eta);  // Algorithm.h:1338-1341 (not clamped)
                d.G[o] = (cx.y[r] - e) * cx.w[r];
                d.W[o] = e * cx.w[r];
            }
        }
        __syncthreads();
        return;
    }
    // cox, Algorithm.h:1579-1630 restated with prefix/suffix sums (SURVEY 8a-4)
    double *th = cx.v[0], *s0 = cx.v[1], *cc = cx.v[2];
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) {
        double eta = 0.0;
        const double *row = cx.XA + (size_t)r * d.ldA + cx.off;
        for (int a = 0; a < ks; a++) eta = fma(row[a], bsl[a], eta);
        const double t = cx.w[r] * exp(clampd(eta, 30.0));
        th[r] = t;
        s0[r] = t;
    }
    __syncthreads();
    clu_suffix_scan(cx, cl, s0, sm);
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) cc[r] = (cx.y[r] != 0.0 ? cx.w[r] : 0.0) / s0[r];
    __syncthreads();
    clu_prefix_scan(cx, cl, cc, sm);
    for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) {
        const double e = cx.y[r] != 0.0 ? cx.w[r] : 0.0;
        const double om = th[r] * cc[r];
        const size_t o = (size_t)rows[r] * FS + c;
        d.G[o] = e - om;
        d.W[o] = om;
        d.TH[o] = th[r];
        d.C2[o] = e / (s0[r] * s0[r]);
    }
    __syncthreads();
}

__device__ __forceinline__ ChainCtx make_ctx(const Dev &d, int c, int T, const Clu &cl, const FitSmem &sm_)
{
    const FitSmem sm = sm_shared(sm_);
    ChainCtx cx;
    cx.c = c;
    cx.nt = d.ntrain[c];
    cx.T = T;
    cx.off = (d.family == FAM_LOGIT || d.family == FAM_POISSON) ? 1 : 0;
    cx.m = T + cx.off;
    cx.ldA = d.ldA;
    const int per = (cx.nt + cl.CL - 1) / cl.CL;
    cx.rb = min(cx.nt, cl.rank * per);
    cx.re = min(cx.nt, cx.rb + per);
    cx.XA = d.XA + (size_t)c * d.n * d.ldA;
    cx.y = d.ytr + (size_t)c * d.n;
    cx.w = d.wtr + (size_t)c * d.n;
    for (int q = 0; q < NVEC; q++) cx.v[q] = d.vec + ((size_t)c * NVEC + q) * d.n;
    cx.Sfin = d.Smat + (size_t)c * 2 * d.ldA * d.ldA;
    const int mmax = cx.m + 1;
    if (mmax <= FIT_SMEM_MS) {
        cx.S = sm.Ssm;
        cx.lds = FIT_SMEM_MS;
    } else {
        cx.S = cx.Sfin;
        cx.lds = d.ldA;
    }
    cx.sp_stride = (size_t)d.nmat * d.ldA * d.ldA;
    cx.Sp0 = d.Spart ? d.Spart + (size_t)c * d.CLcap * cx.sp_stride : nullptr;
    cx.cw = d.cw + (size_t)c * CLMAX * 4 * d.ldA;
    return cx;
}

__device__ __forceinline__ Clu make_clu(const FitSmem &sm_, int CL)
{
    const FitSmem sm = sm_shared(sm_);
    Clu cl;
    cl.CL = CL;
    cl.rank = CL > 1 ? (int)cg::this_cluster().block_rank() : 0;
    cl.xch = sm.xch;
    cl.phase = 0;
    cl.pt.start(threadIdx.x == 0 && cl.rank == 0);
    return cl;
}

// Start of a batch (Algorithm::fit prologue, Algorithm.h:141-148): coef0 <- coef0_init, l <- 0, A_list.col(0) <- 0,
// gradient vectors from beta_init.  One CTA per chain (the gradient is a single pass over the rows).
__global__ void __launch_bounds__(FIT_NT, 1) chain_begin_kernel(const Dev d, const BatchDesc b)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FitSmem sm = carve_fit_smem(smem_raw, d.ldA, d.fit_smem_doubles);
    if (d.prev_active && *d.prev_active != 0) {
        // speculatively enqueued behind a batch that has not finished: close this batch's gate, touch nothing
        if (blockIdx.x == 0 && threadIdx.x == 0) *d.n_active = 0;
        return;
    }
    const int c = b.chain[blockIdx.x];
    // Algorithm::coef0_init is only refreshed when the path starts a new step (path.cpp:57); CV folds of the same
    // step inherit it (SURVEY quirk Q3).
    double level;
    if (!d.warm) level = 0.0;
    else if (b.new_path_step) level = d.coef0[0];
    else level = *d.coef0_level;
    __syncthreads();
    int ks = d.ks[c];
    if (!d.warm) {
        // cold start: beta_init = 0
        for (int a = threadIdx.x; a < ks; a += FIT_NT) {
            const int j = d.A[(size_t)c * d.kcap + a] - d.col_lo;
            if (j >= 0 && j < d.p) d.betaD[(size_t)c * d.pstride + j] = 0.0;
        }
        ks = 0;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        if (blockIdx.x == 0 && b.new_path_step) *d.coef0_level = level;
        if (blockIdx.x == 0) *d.n_active = b.nch;
        d.tie_acc[c] = 0;
        if (!(c == 0 && b.new_path_step && d.warm)) d.coef0[c] = level;
        d.ks[c] = ks;
        d.l[c] = 0;
        d.done[c] = 0;
    }
    int *h0 = d.hist + (size_t)c * d.hist_rows * d.kcap;
    for (int a = threadIdx.x; a < b.T; a += FIT_NT) h0[a] = 0;
    for (int a = threadIdx.x; a < ks; a += FIT_NT) sm.b0[a] = d.bA[(size_t)c * d.kcap + a];
    __syncthreads();
    Clu cl = make_clu(sm, 1);
    ChainCtx cx = make_ctx(d, c, ks, cl, sm);
    chain_gradient(d, cx, cl, sm.b0, ks, level, sm);
}

// One PDAS iteration after the top-k (Algorithm.h:154-170) + gradient vectors for the next one.
// grid = nch * CL CTAs, cluster dimension CL (launch attribute); CTA rank inside the cluster = row slice.
__global__ void __launch_bounds__(FIT_NT, 1) chain_fit_kernel(const Dev d, const BatchDesc b)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FitSmem sm = carve_fit_smem(smem_raw, d.ldA, d.fit_smem_doubles);
    if (d.gate && *d.gate == 0) return;  // whole batch already finished (speculative launch)
    const int CL = b.CL;
    const int c = b.chain[blockIdx.x / CL];
    if (d.done[c]) return;  // uniform over the cluster
    Clu cl = make_clu(sm, CL);
    if (CL > 1) cg::this_cluster().sync();  // every CTA of the cluster is running before any DSMEM traffic
    // group selection: the top-k chose T0 GROUPS (Ag), the fit works on their T columns (Anew); without groups they coincide
    const int T0 = b.T;
    const int T = d.grouped ? d.Tc[c] : T0;
    const int *Ag = d.Anew + (size_t)c * d.kcap;
    ChainCtx cx = make_ctx(d, c, T, cl, sm);
    const int ldA = d.ldA;
    const int *Anew = d.grouped ? d.AnewCols + (size_t)c * d.kcap : Ag;
    const int *rows = d.rows + (size_t)c * d.n;
    int *Acur = d.A + (size_t)c * d.kcap;
    const int ks_old = d.ks[c];
    const double coef0_in = d.coef0[c];
    const int l = d.l[c] + 1;

    // clear the dense beta on the old support (Algorithm.h:159)
    if (cl.rank == 0)
        for (int a = threadIdx.x; a < ks_old; a += FIT_NT) {
            const int j = Acur[a] - d.col_lo;
            if (j >= 0 && j < d.p) d.betaD[(size_t)c * d.pstride + j] = 0.0;
        }
    // gather X_A (utilities.cpp:132-140): XA[r][off + a] = X[rows[r]][A[a]], this CTA's row slice, 8 loads in flight
    {
        const int nloc = cx.re - cx.rb;
        const int tot = nloc * T;
        for (int it0 = threadIdx.x; it0 < tot; it0 += 8 * FIT_NT) {
            double val[8];
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int it = it0 + q * FIT_NT;
                if (it < tot) {
                    const int r = it / T, a = it - r * T;
                    val[q] = d.ax_ext ? d.AXr[((size_t)c * d.n + rows[cx.rb + r]) * d.ldXr + a]
                                       : __ldg(d.X + (size_t)rows[cx.rb + r] * d.ldx + Anew[a]);
                }
            }
#pragma unroll
            for (int q = 0; q < 8; q++) {
                const int it = it0 + q * FIT_NT;
                if (it < tot) {
                    const int r = it / T, a = it - r * T;
                    cx.XA[(size_t)(cx.rb + r) * ldA + cx.off + a] = val[q];
                }
            }
        }
        if (cx.off)
            for (int r = cx.rb + threadIdx.x; r < cx.re; r += FIT_NT) cx.XA[(size_t)r * ldA] = 1.0;
        if (d.ax_ext) {  // keep the all-row columns of this support for the loss kernel
            const double *src = d.AXr + (size_t)c * d.n * d.ldXr;
            double *dst = d.AXk + (size_t)c * d.n * d.ldXk;
            for (int e = cl.rank * FIT_NT + threadIdx.x; e < d.n * T; e += cl.CL * FIT_NT) {
                const int i = e / T, a = e - i * T;
                dst[(size_t)i * d.ldXk + a] = src[(size_t)i * d.ldXr + a];
            }
        }
    }
    __syncthreads();
    cl.pt.mark(PH_GATHER);

    double coef0 = coef0_in;
    const double *slopes;
    if (d.family == FAM_LM) {
        fit_lm(cx, cl, sm, sm.b0, d.lambda);
        slopes = sm.b0;
    } else if (d.family == FAM_LOGIT) {
        fit_logistic(cx, cl, sm, d.lambda);
        coef0 = sm.b0[0];
        slopes = sm.b0 + 1;
    } else if (d.family == FAM_POISSON) {
        fit_poisson(cx, cl, coef0_in, sm, d.lambda);
        coef0 = sm.b0[0];
        slopes = sm.b0 + 1;
    } else {
        fit_cox(cx, cl, d.XB + (size_t)c * d.n * ldA, sm, d.lambda);
        slopes = sm.b0;
    }
    __syncthreads();
    // cycle test (Algorithm.h:164-170) against A_list[0..l-1]; every CTA of the cluster evaluates it identically
    int seen = 0;
    for (int ll = 0; ll < l && !seen; ll++) {
        const int *hp = d.hist + ((size_t)c * d.hist_rows + ll) * d.kcap;
        int same = 1;
        for (int a = threadIdx.x; a < T0; a += FIT_NT) same &= (hp[a] == Ag[a]);
        seen = __syncthreads_and(same);
    }
    const int finished = seen || l >= d.max_iter;
    clu_sync(cl);  // every CTA has read the chain state it needs; rank 0 may now overwrite it
    cl.pt.mark(PH_CYCLE);
    // scatter (Algorithm.h:159-163), record A
    if (cl.rank == 0) {
        int *hl = d.hist + ((size_t)c * d.hist_rows + l) * d.kcap;
        for (int a = threadIdx.x; a < T0; a += FIT_NT) hl[a] = Ag[a];
        for (int a = threadIdx.x; a < T; a += FIT_NT) {
            const int j = Anew[a];
            Acur[a] = j;
            d.bA[(size_t)c * d.kcap + a] = slopes[a];
            const int jl = j - d.col_lo;
            if (jl >= 0 && jl < d.p) d.betaD[(size_t)c * d.pstride + jl] = slopes[a];
        }
        if (threadIdx.x == 0) {
            d.l[c] = seen ? l : (l >= d.max_iter ? d.max_iter + 1 : l);
            d.ks[c] = T;
            d.coef0[c] = coef0;
            d.done[c] = finished;
            d.tie_acc[c] += d.tie[c];
            if (finished) atomicSub(d.n_active, 1);
        }
    }
    if (finished) return;
    chain_gradient(d, cx, cl, slopes, T, coef0, sm);
    cl.pt.mark(PH_GRAD);
}

// ---- explicit chain state (see kernels.cuh).  One CTA rewrites the small tables; a second, wide launch re-gathers the
// active columns of the restored support for the chain's train rows (chain_begin_kernel computes the linear predictor
// from XA and never re-gathers).
__global__ void __launch_bounds__(FIT_NT, 1)
chain_state_kernel(const Dev d, int c, int op, int slot_beta, int slot_coef0, const StateSlots s)
{
    int *A = d.A + (size_t)c * d.kcap;
    double *bA = d.bA + (size_t)c * d.kcap;
    double *bD = d.betaD + (size_t)c * d.pstride;
    if (op == STATE_SAVE) {
        if (slot_beta >= 0) {
            const int ks = d.ks[c];
            for (int a = threadIdx.x; a < ks; a += FIT_NT) {
                s.A[(size_t)slot_beta * d.kcap + a] = A[a];
                s.bA[(size_t)slot_beta * d.kcap + a] = bA[a];
            }
            if (threadIdx.x == 0) s.ks[slot_beta] = ks;
        }
        if (slot_coef0 >= 0 && threadIdx.x == 0) s.coef0[slot_coef0] = d.coef0[c];
        return;
    }
    if (op == STATE_ZERO || slot_beta >= 0) {
        const int ks_old = d.ks[c];
        for (int a = threadIdx.x; a < ks_old; a += FIT_NT) {
            const int j = A[a] - d.col_lo;
            if (j >= 0 && j < d.p) bD[j] = 0.0;
        }
        __syncthreads();
        const int ks_new = op == STATE_LOAD ? s.ks[slot_beta] : 0;
        for (int a = threadIdx.x; a < ks_new; a += FIT_NT) {
            const int j = s.A[(size_t)slot_beta * d.kcap + a];
            const double v = s.bA[(size_t)slot_beta * d.kcap + a];
            A[a] = j;
            bA[a] = v;
            const int jl = j - d.col_lo;
            if (jl >= 0 && jl < d.p) bD[jl] = v;
        }
        if (threadIdx.x == 0) d.ks[c] = ks_new;
    }
    if (threadIdx.x == 0) {
        if (op == STATE_ZERO) d.coef0[c] = 0.0;
        else if (slot_coef0 >= 0) d.coef0[c] = s.coef0[slot_coef0];
    }
}
__global__ void __launch_bounds__(256) chain_state_gather_kernel(const Dev d, int c)
{
    const int ks = d.ks[c], nt = d.ntrain[c];
    const int off = (d.family == FAM_LOGIT || d.family == FAM_POISSON) ? 1 : 0;
    const int *rows = d.rows + (size_t)c * d.n;
    const int *A = d.A + (size_t)c * d.kcap;
    double *XA = d.XA + (size_t)c * d.n * d.ldA;
    const long long tot = (long long)nt * ks;
    for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < tot; e += (long long)gridDim.x * blockDim.x) {
        const int r = (int)(e / ks), a = (int)(e - (long long)r * ks);
        XA[(size_t)r * d.ldA + off + a] = d.ax_ext ? d.AXk[((size_t)c * d.n + rows[r]) * d.ldXk + a]
                                                   : __ldg(d.X + (size_t)rows[r] * d.ldx + A[a]);
    }
    if (off)
        for (int r = blockIdx.x * blockDim.x + threadIdx.x; r < nt; r += gridDim.x * blockDim.x) XA[(size_t)r * d.ldA] = 1.0;
}
// A chain that meets the stopping rule returns from chain_fit_kernel before chain_gradient, so the vectors it last published
// belong to the beta before its last fit; this kernel publishes them for the stored (A, beta_A, coef0) (kernels.cuh).
__global__ void __launch_bounds__(FIT_NT, 1) chain_gradient_kernel(const Dev d, const BatchDesc b)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FitSmem sm = carve_fit_smem(smem_raw, d.ldA, d.fit_smem_doubles);
    const int c = b.chain[blockIdx.x];
    const int ks = d.ks[c];
    for (int a = threadIdx.x; a < ks; a += FIT_NT) sm.b0[a] = d.bA[(size_t)c * d.kcap + a];
    __syncthreads();
    Clu cl = make_clu(sm, 1);
    ChainCtx cx = make_ctx(d, c, ks, cl, sm);
    chain_gradient(d, cx, cl, sm.b0, ks, d.coef0[c], sm);
}
void launch_chain_gradient(const Dev &d, const BatchDesc &b, cudaStream_t st)
{
    if (d.ccp) launch_csc_gather(d, b, 1, st);  // AXk <- the stored supports, re-expanded from the CSC arrays
    for (int i = 0; i < b.nch; i++) {
        chain_state_gather_kernel<<<148, 256, 0, st>>>(d, b.chain[i]);
        CUDA_CHECK(cudaGetLastError());
    }
    const size_t smem = fit_smem_bytes(d);
    CUDA_CHECK(cudaFuncSetAttribute(chain_gradient_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    chain_gradient_kernel<<<b.nch, FIT_NT, smem, st>>>(d, b);
    CUDA_CHECK(cudaGetLastError());
}

void launch_chain_state(const Dev &d, int chain, int op, int slot_beta, int slot_coef0, const StateSlots &s, cudaStream_t st)
{
    chain_state_kernel<<<1, FIT_NT, 0, st>>>(d, chain, op, slot_beta, slot_coef0, s);
    CUDA_CHECK(cudaGetLastError());
    if (op == STATE_LOAD && slot_beta >= 0) {
        if (d.ccp) {  // AXk (losses) <- the restored support from the CSC arrays; XA's train rows follow from it
            BatchDesc b{};
            b.nch = 1;
            b.chain[0] = chain;
            launch_csc_gather(d, b, 1, st);
        }
        chain_state_gather_kernel<<<148, 256, 0, st>>>(d, chain);
        CUDA_CHECK(cudaGetLastError());
    }
}

// ---- solver probe (tools / tests): one CTA factors and solves a bordered system given in global memory, `reps` times from
// a pristine copy; ticks[0] = clock64 ticks of the last repetition.  impl 0 = chol_panel_major, 1 = chol_packed_smem.
__global__ void __launch_bounds__(FIT_NT, 1)
solve_probe_kernel(const double *S0, double *Sw, int lds, int mm, double *xout, int impl, int reps, unsigned long long *ticks,
                   int smem_doubles)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FitSmem sm = carve_fit_smem(smem_raw, lds, smem_doubles);
    PhaseTimer pt;
    for (int rep = 0; rep < reps; rep++) {
        for (int e = threadIdx.x; e < (mm + 1) * lds; e += FIT_NT) Sw[e] = S0[e];
        pt.start(threadIdx.x == 0 && rep == reps - 1);
        __syncthreads();
        const long long t0 = clock64();
        if (impl != 1) chol_panel_major(Sw, lds, mm, sm.rhs, sm, pt);
        else chol_packed_smem(Sw, lds, mm, sm.rhs, sm, pt);
        __syncthreads();
        if (threadIdx.x == 0) ticks[0] = (unsigned long long)(clock64() - t0);
    }
    for (int a = threadIdx.x; a < mm; a += FIT_NT) xout[a] = sm.rhs[a];
}
void debug_solve(const double *S, int lds, int mm, double *x_out, int impl, int reps, double *ticks_out)
{
    if (mm < 1 || mm >= FIT_NT || lds < mm || (lds & 1)) throw EngineError{"debug_solve: need 1 <= mm < 512, even lds >= mm"};
    const int smd = fit_smem_doubles(lds, 400);
    double *dS0, *dSw, *dx;
    unsigned long long *dt, ht = 0;
    const size_t nb = sizeof(double) * (size_t)(mm + 1) * lds;
    CUDA_CHECK(cudaMalloc(&dS0, nb));
    CUDA_CHECK(cudaMalloc(&dSw, nb));
    CUDA_CHECK(cudaMalloc(&dx, sizeof(double) * mm));
    CUDA_CHECK(cudaMalloc(&dt, 8));
    CUDA_CHECK(cudaMemcpy(dS0, S, nb, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaFuncSetAttribute(solve_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smd * 8));
    solve_probe_kernel<<<1, FIT_NT, (size_t)smd * 8>>>(dS0, dSw, lds, mm, dx, impl, reps, dt, smd);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(x_out, dx, sizeof(double) * mm, cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(&ht, dt, 8, cudaMemcpyDeviceToHost));
    if (ticks_out) *ticks_out = (double)ht;
    cudaFree(dS0); cudaFree(dSw); cudaFree(dx); cudaFree(dt);
}

// ---- Gram probe: one CTA computes S = V^T diag(wt) V over `nrows` rows (V in global memory, as in the chain kernels).
// impl 0 = gram() dispatcher, 1 = register-blocked FMA path, 2 = DMMA path
__global__ void __launch_bounds__(FIT_NT, 1)
gram_probe_kernel(const double *V, int ldv, int nrows, int mm, const double *wt, double *S, int impl, int reps,
                  unsigned long long *ticks, int smem_doubles)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FitSmem sm = carve_fit_smem(smem_raw, ldv, smem_doubles);
    for (int rep = 0; rep < reps; rep++) {
        __syncthreads();
        const long long t0 = clock64();
        if (impl == 1) block_syrk(V, ldv, 0, nrows, mm, wt, S, ldv, sm);
        else if (impl == 2) block_syrk_dmma(V, ldv, 0, nrows, mm, wt, S, ldv, sm);
        else gram(V, ldv, 0, nrows, mm, wt, S, ldv, sm);
        __syncthreads();
        if (threadIdx.x == 0) ticks[0] = (unsigned long long)(clock64() - t0);
    }
}
void debug_gram(const double *V, int ldv, int nrows, int mm, const double *wt, double *S_out, int impl, int reps,
                double *ticks_out)
{
    if (mm < 1 || mm > ldv || (ldv & 1) || nrows < 1) throw EngineError{"debug_gram: need 1 <= mm <= ldv, even ldv, nrows >= 1"};
    const int smd = fit_smem_doubles(ldv, 400);
    double *dV, *dw, *dS;
    unsigned long long *dt, ht = 0;
    CUDA_CHECK(cudaMalloc(&dV, sizeof(double) * (size_t)nrows * ldv));
    CUDA_CHECK(cudaMalloc(&dw, sizeof(double) * nrows));
    CUDA_CHECK(cudaMalloc(&dS, sizeof(double) * (size_t)ldv * ldv));
    CUDA_CHECK(cudaMalloc(&dt, 8));
    CUDA_CHECK(cudaMemcpy(dV, V, sizeof(double) * (size_t)nrows * ldv, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemcpy(dw, wt, sizeof(double) * nrows, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaMemset(dS, 0, sizeof(double) * (size_t)ldv * ldv));
    CUDA_CHECK(cudaFuncSetAttribute(gram_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smd * 8));
    gram_probe_kernel<<<1, FIT_NT, (size_t)smd * 8>>>(dV, ldv, nrows, mm, dw, dS, impl, reps, dt, smd);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(S_out, dS, sizeof(double) * (size_t)ldv * ldv, cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(&ht, dt, 8, cudaMemcpyDeviceToHost));
    if (ticks_out) *ticks_out = (double)ht;
    cudaFree(dV); cudaFree(dw); cudaFree(dS); cudaFree(dt);
}

// ---- production-placement probes (tests).  The solve probe places a bordered system where make_ctx puts it for a support
// cap kcap -- in sm.Ssm at ld FIT_SMEM_MS when it has at most FIT_SMEM_MS rows, else in global memory at ldA = (kcap + 3) & ~1
// with the arena of fit_smem_doubles(ldA, kcap) -- and solves it with solve_on_rank0, the code a CL = 1 fit runs.
__global__ void __launch_bounds__(FIT_NT, 1)
solve_path_probe_kernel(const double *Sin, int ldin, double *Sg, int ldA, int mm, double *xout, int *path, int smem_doubles)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FitSmem sm = carve_fit_smem(smem_raw, ldA, smem_doubles);
    const bool small = mm + 1 <= FIT_SMEM_MS;
    double *S = small ? sm.Ssm : Sg;
    const int lds = small ? FIT_SMEM_MS : ldA;
    for (int e = threadIdx.x; e < (mm + 1) * (mm + 1); e += FIT_NT) S[(size_t)(e / (mm + 1)) * lds + e % (mm + 1)] = Sin[(size_t)(e / (mm + 1)) * ldin + e % (mm + 1)];
    __syncthreads();
    PhaseTimer pt;
    pt.start(false);
    // a fit hands such a system to chol_blocked_cluster, which needs the whole cluster: reported, not solved
    const bool rank0 = solved_on_rank0(S, mm, sm);
    const int code = rank0 ? solve_on_rank0(S, lds, mm, sm, pt, false) : SOLVE_CLUSTER;
    __syncthreads();
    for (int a = threadIdx.x; a < mm; a += FIT_NT) xout[a] = rank0 ? sm.rhs[a] : __longlong_as_double(0x7ff8000000000000ll);
    if (threadIdx.x == 0) *path = code;
}
static unsigned long long take_counter(const unsigned long long &sym)
{
    unsigned long long v = 0ull, z = 0ull;
    CUDA_CHECK(cudaMemcpyFromSymbol(&v, sym, sizeof(v)));
    if (v) CUDA_CHECK(cudaMemcpyToSymbol(sym, &z, sizeof(z)));
    return v;
}
void debug_solve_path(const double *S, int lds, int mm, int kcap, double *x_out, int *path_out)
{
    const int ldA = (kcap + 3) & ~1;
    if (mm < 1 || mm >= FIT_NT || mm > kcap + 1 || lds < mm + 1)
        throw EngineError{"debug_solve_path: need 1 <= mm < 512, mm <= kcap + 1, lds >= mm + 1"};
    const int smd = fit_smem_doubles(ldA, kcap);
    double *dS, *dSg, *dx;
    int *dp;
    const size_t nb = sizeof(double) * (size_t)(mm + 1) * lds;
    CUDA_CHECK(cudaMalloc(&dS, nb));
    CUDA_CHECK(cudaMalloc(&dSg, sizeof(double) * (size_t)(mm + 1) * ldA));
    CUDA_CHECK(cudaMalloc(&dx, sizeof(double) * mm));
    CUDA_CHECK(cudaMalloc(&dp, sizeof(int)));
    CUDA_CHECK(cudaMemcpy(dS, S, nb, cudaMemcpyHostToDevice));
    const unsigned long long rd0 = take_counter(g_rankdef_count), ws0 = take_counter(g_wide_singular_count);
    CUDA_CHECK(cudaFuncSetAttribute(solve_path_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smd * 8));
    solve_path_probe_kernel<<<1, FIT_NT, (size_t)smd * 8>>>(dS, lds, dSg, ldA, mm, dx, dp, smd);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(x_out, dx, sizeof(double) * mm, cudaMemcpyDeviceToHost));
    CUDA_CHECK(cudaMemcpy(path_out, dp, sizeof(int), cudaMemcpyDeviceToHost));
    path_out[1] = (int)take_counter(g_rankdef_count);
    path_out[2] = (int)take_counter(g_wide_singular_count);
    // give back what a fit running before the probe had counted
    if (rd0) CUDA_CHECK(cudaMemcpyToSymbol(g_rankdef_count, &rd0, sizeof(rd0)));
    if (ws0) CUDA_CHECK(cudaMemcpyToSymbol(g_wide_singular_count, &ws0, sizeof(ws0)));
    cudaFree(dS); cudaFree(dSg); cudaFree(dx); cudaFree(dp);
}

// The Gram probe over the rows [r0, r1) of V (r0 > 0: a cluster's row slice), wt may be null.  The output lands where
// gram_solve puts it: in sm.Ssm at ld FIT_SMEM_MS when mm <= FIT_SMEM_MS (the DMMA ring then shares the arena with it),
// else in global memory at ld ldv; the arena is fit_smem_doubles(ldv, kcap).  S_io (ldo x ldo, ldo = FIT_SMEM_MS or ldv)
// is loaded as the output region's initial contents and read back whole, so stray writes show.
__global__ void __launch_bounds__(FIT_NT, 1)
gram_rows_probe_kernel(const double *V, int ldv, int r0, int r1, int mm, const double *wt, double *Sg, int impl, int smem_doubles)
{
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const FitSmem sm = carve_fit_smem(smem_raw, ldv, smem_doubles);
    const bool small = mm <= FIT_SMEM_MS;
    double *S = small ? sm.Ssm : Sg;
    const int lds = small ? FIT_SMEM_MS : ldv;
    if (small)
        for (int e = threadIdx.x; e < FIT_SMEM_MS * FIT_SMEM_MS; e += FIT_NT) S[e] = Sg[e];
    __syncthreads();
    if (impl == 1) block_syrk(V, ldv, r0, r1, mm, wt, S, lds, sm);
    else if (impl == 2) block_syrk_dmma(V, ldv, r0, r1, mm, wt, S, lds, sm);
    else gram(V, ldv, r0, r1, mm, wt, S, lds, sm);
    __syncthreads();
    if (small)
        for (int e = threadIdx.x; e < FIT_SMEM_MS * FIT_SMEM_MS; e += FIT_NT) Sg[e] = S[e];
}
void debug_gram_rows(const double *V, int ldv, int r0, int r1, int mm, const double *wt, double *S_io, int kcap, int impl)
{
    if (mm < 1 || mm > ldv || (ldv & 1) || r0 < 0 || r1 <= r0 || mm > kcap + 2 || impl < 0 || impl > 2)
        throw EngineError{"debug_gram_rows: need 1 <= mm <= min(ldv, kcap + 2), even ldv, 0 <= r0 < r1, impl 0..2"};
    const int smd = fit_smem_doubles(ldv, kcap);
    const int ldo = mm <= FIT_SMEM_MS ? FIT_SMEM_MS : ldv;
    double *dV, *dw = nullptr, *dS;
    CUDA_CHECK(cudaMalloc(&dV, sizeof(double) * (size_t)r1 * ldv));
    CUDA_CHECK(cudaMalloc(&dS, sizeof(double) * (size_t)ldo * ldo));
    CUDA_CHECK(cudaMemcpy(dV, V, sizeof(double) * (size_t)r1 * ldv, cudaMemcpyHostToDevice));
    if (wt) {
        CUDA_CHECK(cudaMalloc(&dw, sizeof(double) * r1));
        CUDA_CHECK(cudaMemcpy(dw, wt, sizeof(double) * r1, cudaMemcpyHostToDevice));
    }
    CUDA_CHECK(cudaMemcpy(dS, S_io, sizeof(double) * (size_t)ldo * ldo, cudaMemcpyHostToDevice));
    CUDA_CHECK(cudaFuncSetAttribute(gram_rows_probe_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smd * 8));
    gram_rows_probe_kernel<<<1, FIT_NT, (size_t)smd * 8>>>(dV, ldv, r0, r1, mm, dw, dS, impl, smd);
    CUDA_CHECK(cudaGetLastError());
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpy(S_io, dS, sizeof(double) * (size_t)ldo * ldo, cudaMemcpyDeviceToHost));
    cudaFree(dV); cudaFree(dS);
    if (dw) cudaFree(dw);
}

long long debug_take_rankdef() { return (long long)take_counter(g_rankdef_count); }
long long take_wide_singular() { return (long long)take_counter(g_wide_singular_count); }

void debug_set(int key, int val)
{
    if (key == 1) CUDA_CHECK(cudaMemcpyToSymbol(g_dbg_cox_iters, &val, sizeof(int)));
    if (key == 4) CUDA_CHECK(cudaMemcpyToSymbol(g_dbg_solver, &val, sizeof(int)));
    if (key == 2) {
        CUDA_CHECK(cudaMemcpyToSymbol(g_dbg_phase_on, &val, sizeof(int)));
        unsigned long long z[2][16] = {};
        CUDA_CHECK(cudaMemcpyToSymbol(g_dbg_phase, z, sizeof(z)));
    }
}
void debug_get(unsigned long long *out32)
{
    CUDA_CHECK(cudaDeviceSynchronize());
    CUDA_CHECK(cudaMemcpyFromSymbol(out32, g_dbg_phase, sizeof(unsigned long long) * 32));
}

// cluster size for sparsity level T: enough work per CTA to amortise the cluster barriers, all clusters co-resident.
// work ~ rows x columns^2 of one Gram (x2 for cox: two Grams per Newton step).  Even the small gaussian fits of config 5
// (900 x 21) gain from 4 CTAs: gather, Gram and gradient are row-parallel and a cluster barrier costs ~0.2 us.
// how many 16-CTA clusters of chain_fit_kernel the device can hold at once (0: not schedulable); queried once
static int g_cl16_chains = -1;
static void query_cl16(size_t smem)
{
    if (g_cl16_chains >= 0) return;
    g_cl16_chains = 0;
    if (cudaFuncSetAttribute(chain_fit_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) != cudaSuccess) {
        cudaGetLastError();
        return;
    }
    cudaFuncSetAttribute(chain_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(16);
    cfg.blockDim = dim3(FIT_NT);
    cfg.dynamicSmemBytes = smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 16;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int ncl = 0;
    if (cudaOccupancyMaxActiveClusters(&ncl, chain_fit_kernel, &cfg) == cudaSuccess) g_cl16_chains = std::max(0, ncl);
    else cudaGetLastError();
    if (const char *e = std::getenv("BESS_B200_CL16_CHAINS")) g_cl16_chains = std::min(g_cl16_chains, std::max(0, std::atoi(e)));
}
int chain_cluster_size(const Dev &d, int T, int nch)
{
    query_cl16(fit_smem_bytes(d));
    static double thr = -1.0;
    static int clmax = CLMAX;
    if (thr < 0.0) {
        const char *e = std::getenv("BESS_B200_CL_WORK");
        thr = e ? std::atof(e) : 1.25e4;  // swept on configs 3 / 4: 1e5 -> 121 / 81 ms of chain kernels, 2.5e4 -> 108 / 75, 1.25e4 -> 106 / 74
        const char *e2 = std::getenv("BESS_B200_CL_MAX");
        if (e2) clmax = std::max(1, std::min(CLMAX, std::atoi(e2)));
    }
    const double m = T + 2.0;
    const double work = (double)d.n * m * m * (d.family == FAM_COX ? 2.0 : 1.0);
    int CL = 1;
    while (CL < std::min(clmax, 8) && CL < d.CLcap && work / CL > thr && nch * CL * 2 <= 148 && d.n / (CL * 2) >= 128) CL *= 2;
    // 16-CTA (non-portable) clusters: one fits a GPC, so at most 8 can run at once -- for batches of few chains with a
    // lot of work per chain (a single IC chain at n = 5000; the 3-4 chains a rank keeps of a fold-sharded call)
    if (CL == 8 && clmax >= 16 && d.CLcap >= 16 && nch <= g_cl16_chains && work / 16.0 > 3.0 * thr && d.n / 16 >= 96) CL = 16;
    return CL;
}

void launch_chain_begin(const Dev &d, const BatchDesc &b, cudaStream_t st)
{
    const size_t smem = fit_smem_bytes(d);
    CUDA_CHECK(cudaFuncSetAttribute(chain_begin_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    chain_begin_kernel<<<b.nch, FIT_NT, smem, st>>>(d, b);
    CUDA_CHECK(cudaGetLastError());
}
void launch_chain_fit(const Dev &d, const BatchDesc &b, cudaStream_t st)
{
    const size_t smem = fit_smem_bytes(d);
    CUDA_CHECK(cudaFuncSetAttribute(chain_fit_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    if (b.CL > 8) CUDA_CHECK(cudaFuncSetAttribute(chain_fit_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)(b.nch * b.CL));
    cfg.blockDim = dim3(FIT_NT);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = (unsigned)b.CL;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    CUDA_CHECK(cudaLaunchKernelEx(&cfg, chain_fit_kernel, d, b));
}

}  // namespace bess
