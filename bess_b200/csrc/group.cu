// Group selection (gsize > 1): R bess(..., group.index =), Python GroupPdas* -- algorithm_type 2 (GPDAS) / 3 (GL0L2).
//
// A sparsity level counts GROUPS.  get_A (Algorithm.h:1097-1129 lm, :1206-1263 logistic, :1324-1367 poisson,
// :1497-1568 cox) scores group g by
//     bd_g = || Phi_g beta_g + Phi_g^{-1} d_g ||^2 / gsize_g,   Phi_g = (M_g + 2 lambda I)^{1/2},
// with d = X^T (gradient vector) - 2 lambda beta and M_g the k_g x k_g block of the model's curvature on the group's
// columns:  lm  X_g^T X_g / n  (utilities.cpp:142-165);  logistic / poisson  X_g^T diag(h) X_g;  cox  X_g^T H X_g with the
// dense n x n partial-likelihood Hessian H, which in risk-set form is
//     sum_i omega_i x_ia x_ib  -  sum_{k: event} (e_k / S_k^2) s_a(k) s_b(k),    s_a(k) = sum_{i >= k} theta_i x_ia.
// The matrix square root (Eigen's Schur-based sqrt(), utilities.cpp:147) of an SPD block is U diag(sqrt(ev)) U^T, so with
// M_g + 2 lambda I = U diag(ev) U^T:   bd_g = sum_i ( sqrt(ev_i) (U^T beta_g)_i + (U^T d_g)_i / sqrt(ev_i) )^2 / gsize_g.
//
// group_sacrifice_kernel fuses sweep and epilogue: one thread per (group, chain) walks all rows once (neighbouring
// threads own neighbouring column ranges of the row-major design, so the loads coalesce), accumulating d_g, the packed
// block M_g and -- for cox, walking the rows from the last to the first -- the running risk-set sums, then diagonalises
// the block with cyclic Jacobi rotations.  The gradient vectors (G, W, TH, C2; zero on rows outside the chain's train
// mask) are the ones chain_begin / chain_fit already publish for the column-wise sweep.
// group_expand_kernel turns the T selected groups into the column list the active-set fit works on (find_ind,
// utilities.cpp:113-130).
#include <cfloat>
#include <cmath>
#include <cstdlib>

#include "device_utils.cuh"
#include "kernels.cuh"

namespace bess {

constexpr int GS_NT = 128;

// cyclic Jacobi on a symmetric g x g matrix (g <= GMAX): A -> diag(ev), U = eigenvectors in columns
__device__ void jacobi_eig(double (*A)[GMAX], double (*U)[GMAX], int g)
{
    for (int i = 0; i < g; i++)
        for (int j = 0; j < g; j++) U[i][j] = i == j ? 1.0 : 0.0;
    for (int sweep = 0; sweep < 60; sweep++) {
        int rotated = 0;
        for (int p = 0; p < g - 1; p++)
            for (int q = p + 1; q < g; q++) {
                const double apq = A[p][q];
                // a rotation that cannot change the diagonal any more is skipped
                if (fabs(apq) <= 1e-18 * sqrt(fabs(A[p][p] * A[q][q])) || apq == 0.0) continue;
                rotated = 1;
                const double theta = (A[q][q] - A[p][p]) / (2.0 * apq);
                const double t = (theta >= 0.0 ? 1.0 : -1.0) / (fabs(theta) + sqrt(theta * theta + 1.0));
                const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
                for (int k = 0; k < g; k++) {
                    const double akp = A[k][p], akq = A[k][q];
                    A[k][p] = c * akp - s * akq;
                    A[k][q] = s * akp + c * akq;
                }
                for (int k = 0; k < g; k++) {
                    const double apk = A[p][k], aqk = A[q][k];
                    A[p][k] = c * apk - s * aqk;
                    A[q][k] = s * apk + c * aqk;
                }
                for (int k = 0; k < g; k++) {
                    const double ukp = U[k][p], ukq = U[k][q];
                    U[k][p] = c * ukp - s * ukq;
                    U[k][q] = s * ukp + c * ukq;
                }
            }
        if (!rotated) break;
    }
}

// block + gradient of one group -> its sacrifice (shared by the two sweep kernels below)
__device__ void group_epilogue(const Dev &d, int c, int g, int j0, int gs, double (&dv)[GMAX], const double (&M)[GMAX * (GMAX + 1) / 2])
{
    // M_g + 2 lambda I, d_g - 2 lambda beta_g
    double A[GMAX][GMAX], U[GMAX][GMAX], bg[GMAX];
    {
        int e = 0;
        for (int a = 0; a < GMAX; a++)
            for (int bb = a; bb < GMAX; bb++, e++)
                if (bb < gs) A[a][bb] = A[bb][a] = M[e] + (a == bb ? 2.0 * d.lambda : 0.0);
    }
    for (int a = 0; a < gs; a++) {
        bg[a] = d.betaD[(size_t)c * d.pstride + j0 + a];
        dv[a] -= 2.0 * d.lambda * bg[a];
    }
    double bd;
    if (gs == 1) {
        const double phi = sqrt(A[0][0]);
        const double t = phi * bg[0] + dv[0] / phi;
        bd = t * t;
    } else {
        jacobi_eig(A, U, gs);
        bd = 0.0;
        for (int q = 0; q < gs; q++) {
            double ub = 0.0, ud = 0.0;
            for (int a = 0; a < gs; a++) {
                ub = fma(U[a][q], bg[a], ub);
                ud = fma(U[a][q], dv[a], ud);
            }
            const double r = sqrt(A[q][q]);
            const double t = r * ub + ud / r;
            bd = fma(t, t, bd);
        }
        bd /= (double)gs;
    }
    d.bd[(size_t)c * d.pstride + g] = bd;
}

// Row-parallel variant for the gaussian / logistic / poisson blocks (no risk-set recurrence): one WARP per (group, chain),
// lane l takes rows l, l + 32, ..., the 8 + 36 partial sums meet in a butterfly reduction (fixed lane order => bitwise
// reproducible), lane 0 diagonalises.  32 x the threads of the serial kernel: the row walk is no longer a serial chain of
// n dependent steps per thread.
__global__ void __launch_bounds__(GS_NT) group_sacrifice_warp_kernel(const Dev d, const BatchDesc b)
{
    if (d.gate && *d.gate == 0) return;
    const int c = b.chain[blockIdx.y];
    if (d.done[c]) return;
    const int lane = threadIdx.x & 31;
    const int g = blockIdx.x * (GS_NT / 32) + (threadIdx.x >> 5);
    if (g >= d.N) return;  // warp-uniform
    const int j0 = d.gidx[g], gs = d.gsz[g];
    if (gs > GMAX) return;  // wide groups: group_sacrifice_wide_kernel
    const int FS = d.FS;
    double dv[GMAX], M[GMAX * (GMAX + 1) / 2];
#pragma unroll
    for (int a = 0; a < GMAX; a++) dv[a] = 0.0;
#pragma unroll
    for (int e = 0; e < GMAX * (GMAX + 1) / 2; e++) M[e] = 0.0;
    for (int i = lane; i < d.n; i += 32) {
        const double gi = d.G[(size_t)i * FS + c], wi = d.W[(size_t)i * FS + c];
        if (gi == 0.0 && wi == 0.0) continue;  // row outside the chain's train mask
        const double *xr = d.X + (size_t)i * d.ldx + j0;
        double x[GMAX];
#pragma unroll
        for (int a = 0; a < GMAX; a++) x[a] = a < gs ? __ldg(xr + a) : 0.0;
#pragma unroll
        for (int a = 0; a < GMAX; a++) dv[a] = fma(x[a], gi, dv[a]);
        int e = 0;
#pragma unroll
        for (int a = 0; a < GMAX; a++) {
            const double wa = wi * x[a];
#pragma unroll
            for (int bb = a; bb < GMAX; bb++, e++) M[e] = fma(wa, x[bb], M[e]);
        }
    }
#pragma unroll
    for (int off = 16; off >= 1; off >>= 1) {
#pragma unroll
        for (int a = 0; a < GMAX; a++) dv[a] += __shfl_xor_sync(0xffffffffu, dv[a], off);
#pragma unroll
        for (int e = 0; e < GMAX * (GMAX + 1) / 2; e++) M[e] += __shfl_xor_sync(0xffffffffu, M[e], off);
    }
    if (lane == 0) group_epilogue(d, c, g, j0, gs, dv, M);
}

// Chain-batched variant for the gaussian / logistic / poisson blocks: ONE pass over X serves every chain of the batch (the
// warp kernel above re-reads the group's columns once per chain).  A CTA takes 8 groups (one per warp); the gradient
// vectors G, W of a 64-row tile -- [row][chain slot], the layout chain_begin / chain_fit publish -- are staged in shared
// memory once per CTA and shared by its warps.  Inside a warp lane = (row phase, chain slot): with FS <= 8 chain slots four
// rows are in flight per step (two with FS <= 16, eight with FS <= 4), the x values of a row are the same address for all its lanes (one broadcast load), and
// every lane carries the d_g / M_g accumulators of ITS chain (compact, sized by the padded group width GSP in {2, 4, 8}:
// a group of 4 pays 10 block entries per row, not the 36 of the widest group).  The row phases meet in one shuffle, then
// the lanes of all chains run the eigen-solve epilogue side by side.
constexpr int GB_NT = 256;  // 8 warps = 8 groups per CTA share one staged tile of the gradient vectors (4 per CTA measured slower)
constexpr int GB_RT = 64;
template <int GSP>
__global__ void __launch_bounds__(GB_NT) group_sacrifice_batched_kernel(const Dev d, const BatchDesc b, int lo, int hi)
{
    __shared__ double sG[GB_RT][32], sW[GB_RT][32];
    if (d.gate && *d.gate == 0) return;
    const int lane = threadIdx.x & 31, wid = threadIdx.x >> 5;
    const int FS = d.FS;
    int CS = 2;  // lanes per row phase: the chain slots rounded up to a power of two
    while (CS < FS) CS <<= 1;
    const int nrp = 32 / CS;  // row phases in flight per warp step (FS = 6 or 8: 4, FS = 12 or 16: 2)
    const int c = lane & (CS - 1), rp = lane / CS;
    const int li = lo + blockIdx.x * (GB_NT / 32) + wid;  // position in the class's group list
    const bool have = li < hi;
    const int g = have ? d.glist[li] : 0;
    const int j0 = d.gidx[g], gs = d.gsz[g];
    bool live = false;  // is chain slot c part of this batch and still iterating?
    for (int q = 0; q < b.nch; q++) live = live || (b.chain[q] == c && !d.done[c]);
    double dv[GSP], M[GSP * (GSP + 1) / 2];
#pragma unroll
    for (int a = 0; a < GSP; a++) dv[a] = 0.0;
#pragma unroll
    for (int e = 0; e < GSP * (GSP + 1) / 2; e++) M[e] = 0.0;
    constexpr int RU = GSP == GMAX ? 2 : (GSP == 4 ? 4 : 8);  // rows in flight per lane
    for (int e = threadIdx.x; e < GB_RT * 32; e += GB_NT) {  // chain slots >= FS stay zero
        sG[e >> 5][e & 31] = 0.0;
        sW[e >> 5][e & 31] = 0.0;
    }
    for (int t0 = 0; t0 < d.n; t0 += GB_RT) {
        const int rows = min(GB_RT, d.n - t0);
        __syncthreads();
        for (int e = threadIdx.x; e < rows * FS; e += GB_NT) {  // the tile is one contiguous block of both vectors
            const int r = e / FS, cc = e - r * FS;
            sG[r][cc] = d.G[(size_t)t0 * FS + e];
            sW[r][cc] = d.W[(size_t)t0 * FS + e];
        }
        __syncthreads();
        if (!have) continue;  // warp-uniform
        for (int r0 = rp; r0 < rows; r0 += RU * nrp) {
            double x[RU][GSP];
#pragma unroll
            for (int u = 0; u < RU; u++) {
                const int r = r0 + u * nrp;
                const double *xr = d.X + (size_t)(t0 + min(r, rows - 1)) * d.ldx + j0;
#pragma unroll
                for (int a = 0; a < GSP; a++) x[u][a] = a < gs ? __ldg(xr + a) : 0.0;
            }
#pragma unroll
            for (int u = 0; u < RU; u++) {
                const int r = r0 + u * nrp;
                if (r < rows) {
                    const double gi = sG[r][c], wi = sW[r][c];
#pragma unroll
                    for (int a = 0; a < GSP; a++) dv[a] = fma(x[u][a], gi, dv[a]);
                    int e = 0;
#pragma unroll
                    for (int a = 0; a < GSP; a++) {
                        const double wa = wi * x[u][a];
#pragma unroll
                        for (int bb = a; bb < GSP; bb++, e++) M[e] = fma(wa, x[u][bb], M[e]);
                    }
                }
            }
        }
    }
    if (!have) return;
    for (int off = CS; off < 32; off <<= 1) {  // the row phases meet (fixed order)
#pragma unroll
        for (int a = 0; a < GSP; a++) dv[a] += __shfl_xor_sync(0xffffffffu, dv[a], off);
#pragma unroll
        for (int e = 0; e < GSP * (GSP + 1) / 2; e++) M[e] += __shfl_xor_sync(0xffffffffu, M[e], off);
    }
    if (rp == 0 && live) {
        // compact accumulators -> the GMAX-packed layout of the epilogue
        double dvf[GMAX], Mf[GMAX * (GMAX + 1) / 2];
#pragma unroll
        for (int a = 0; a < GMAX; a++) dvf[a] = 0.0;
#pragma unroll
        for (int e = 0; e < GMAX * (GMAX + 1) / 2; e++) Mf[e] = 0.0;
        int e = 0;
#pragma unroll
        for (int a = 0; a < GSP; a++) {
            dvf[a] = dv[a];
#pragma unroll
            for (int bb = a; bb < GSP; bb++, e++) Mf[a * GMAX - a * (a - 1) / 2 + (bb - a)] = M[e];
        }
        group_epilogue(d, c, g, j0, gs, dvf, Mf);
    }
}

template <bool COX>
__global__ void __launch_bounds__(GS_NT) group_sacrifice_kernel(const Dev d, const BatchDesc b)
{
    if (d.gate && *d.gate == 0) return;
    const int c = b.chain[blockIdx.y];
    if (d.done[c]) return;
    const int g = blockIdx.x * GS_NT + threadIdx.x;
    if (g >= d.N) return;
    const int j0 = d.gidx[g], gs = d.gsz[g];
    if (gs > GMAX) return;  // wide groups: group_sacrifice_wide_kernel
    const int FS = d.FS;
    double dv[GMAX], sv[GMAX], M[GMAX * (GMAX + 1) / 2];
#pragma unroll
    for (int a = 0; a < GMAX; a++) dv[a] = 0.0, sv[a] = 0.0;
#pragma unroll
    for (int e = 0; e < GMAX * (GMAX + 1) / 2; e++) M[e] = 0.0;
    for (int ii = 0; ii < d.n; ii++) {
        const int i = COX ? d.n - 1 - ii : ii;
        const double gi = d.G[(size_t)i * FS + c], wi = d.W[(size_t)i * FS + c];
        double th = 0.0, c2 = 0.0;
        if (COX) {
            th = d.TH[(size_t)i * FS + c];
            c2 = d.C2[(size_t)i * FS + c];
        }
        if (gi == 0.0 && wi == 0.0 && th == 0.0) continue;  // row outside the chain's train mask
        const double *xr = d.X + (size_t)i * d.ldx + j0;
        double x[GMAX];
#pragma unroll
        for (int a = 0; a < GMAX; a++) x[a] = a < gs ? __ldg(xr + a) : 0.0;
#pragma unroll
        for (int a = 0; a < GMAX; a++) {
            dv[a] = fma(x[a], gi, dv[a]);
            if (COX) sv[a] = fma(x[a], th, sv[a]);
        }
        int e = 0;
#pragma unroll
        for (int a = 0; a < GMAX; a++) {
            const double wa = wi * x[a];
#pragma unroll
            for (int bb = a; bb < GMAX; bb++, e++) {
                double v = fma(wa, x[bb], M[e]);
                if (COX) v = fma(-c2 * sv[a], sv[bb], v);
                M[e] = v;
            }
        }
    }
    group_epilogue(d, c, g, j0, gs, dv, M);
}

// Groups of GMAX + 1 .. GWIDE variables: one CTA per (group, chain), the k_g x k_g block in shared memory.  Rows travel
// in tiles of GW_RT (for cox from the last row to the first: the risk-set sums s_a(k) of a tile are formed first, one
// thread per column, then the block update is a tile contraction like the weighted one); thread t owns the block entries
// t, t + GW_NT, ...  No eigen-decomposition here: with A = M_g + 2 lambda I = Phi^2,
//     || Phi beta + Phi^{-1} d ||^2 = beta' A beta + 2 beta' d + d' A^{-1} d,
// and d' A^{-1} d = || L^{-1} d ||^2 with the Cholesky factor A = L L' (an in-place unblocked factorisation by the CTA and
// one forward substitution) -- the same number as the reference's Schur-based sqrt() / inverse route (utilities.cpp:147,
// Algorithm.h:1112-1123) up to rounding.
constexpr int GW_NT = 256;
constexpr int GW_RT = 32;
constexpr int GW_EPT = (GWIDE * GWIDE + GW_NT - 1) / GW_NT;  // block entries per thread
template <bool COX>
__global__ void __launch_bounds__(GW_NT) group_sacrifice_wide_kernel(const Dev d, const BatchDesc b)
{
    extern __shared__ __align__(16) double gw_smem[];
    if (d.gate && *d.gate == 0) return;
    const int c = b.chain[blockIdx.y];
    if (d.done[c]) return;
    const int g = blockIdx.x;
    const int gs = d.gsz[g];
    if (gs <= GMAX) return;  // CTA-uniform: the register kernels own the narrow groups
    const int j0 = d.gidx[g], FS = d.FS, tid = threadIdx.x;
    double *A = gw_smem;                 // [gs][gs]
    double *xt = A + GWIDE * GWIDE;      // [GW_RT][gs] x tile
    double *stl = xt + GW_RT * GWIDE;    // [GW_RT][gs] cox: risk-set sums after each row of the tile
    double *rv = stl + GW_RT * GWIDE;    // [4][GW_RT] g, w, theta, c2 of the tile's rows
    double *vec = rv + 4 * GW_RT;        // [4][GWIDE] d, beta, L^{-1} d, scratch
    double *red = vec + 4 * GWIDE;       // [40] block_sum scratch
    double macc[GW_EPT];
#pragma unroll
    for (int q = 0; q < GW_EPT; q++) macc[q] = 0.0;
    double dacc = 0.0, sacc = 0.0;  // threads < gs: d_a, running risk-set sum s_a
    const int ne = gs * gs;
    for (int t0 = 0; t0 < d.n; t0 += GW_RT) {
        const int rc = min(GW_RT, d.n - t0);
        // tile row r is design row i(r): ascending, or for cox descending from the last row
        __syncthreads();
        for (int e = tid; e < rc * gs; e += GW_NT) {
            const int r = e / gs, a = e - r * gs;
            const int i = COX ? d.n - 1 - (t0 + r) : t0 + r;
            xt[r * GWIDE + a] = __ldg(d.X + (size_t)i * d.ldx + j0 + a);
        }
        if (tid < rc) {
            const int i = COX ? d.n - 1 - (t0 + tid) : t0 + tid;
            const double gi = d.G[(size_t)i * FS + c], wi = d.W[(size_t)i * FS + c];
            const double th = COX ? d.TH[(size_t)i * FS + c] : 0.0;
            const bool off = gi == 0.0 && wi == 0.0 && th == 0.0;  // row outside the chain's train mask
            rv[tid] = gi;
            rv[GW_RT + tid] = wi;
            rv[2 * GW_RT + tid] = th;
            rv[3 * GW_RT + tid] = (COX && !off) ? d.C2[(size_t)i * FS + c] : 0.0;
        }
        __syncthreads();
        if (tid < gs) {
            for (int r = 0; r < rc; r++) {
                const double x = xt[r * GWIDE + tid];
                dacc = fma(x, rv[r], dacc);
                if (COX) {
                    sacc = fma(x, rv[2 * GW_RT + r], sacc);
                    stl[r * GWIDE + tid] = sacc;
                }
            }
        }
        if (COX) __syncthreads();
#pragma unroll
        for (int q = 0; q < GW_EPT; q++) {
            const int e = tid + q * GW_NT;
            if (e < ne) {
                const int a = e / gs, bb = e - a * gs;
                double m = macc[q];
                for (int r = 0; r < rc; r++) {
                    m = fma(rv[GW_RT + r] * xt[r * GWIDE + a], xt[r * GWIDE + bb], m);
                    if (COX) m = fma(-rv[3 * GW_RT + r] * stl[r * GWIDE + a], stl[r * GWIDE + bb], m);
                }
                macc[q] = m;
            }
        }
    }
    __syncthreads();
#pragma unroll
    for (int q = 0; q < GW_EPT; q++) {
        const int e = tid + q * GW_NT;
        if (e < ne) {
            const int a = e / gs, bb = e - a * gs;
            A[a * GWIDE + bb] = macc[q] + (a == bb ? 2.0 * d.lambda : 0.0);
        }
    }
    if (tid < gs) {
        const double bg = d.betaD[(size_t)c * d.pstride + j0 + tid];
        vec[tid] = dacc - 2.0 * d.lambda * bg;  // d_g - 2 lambda beta_g
        vec[GWIDE + tid] = bg;
    }
    __syncthreads();
    // beta' A beta + 2 beta' d
    double part = 0.0;
    for (int e = tid; e < ne; e += GW_NT) {
        const int a = e / gs, bb = e - a * gs;
        part = fma(vec[GWIDE + a] * A[a * GWIDE + bb], vec[GWIDE + bb], part);
    }
    if (tid < gs) part = fma(2.0 * vec[GWIDE + tid], vec[tid], part);
    const double quad = block_sum<GW_NT>(part, red);
    // A = L L' in place (lower triangle), then y = L^{-1} d
    for (int j = 0; j < gs; j++) {
        __syncthreads();
        const double djj = sqrt(A[j * GWIDE + j]);
        __syncthreads();
        if (tid == 0) A[j * GWIDE + j] = djj;
        for (int i = j + 1 + tid; i < gs; i += GW_NT) A[i * GWIDE + j] /= djj;
        __syncthreads();
        const int rem = gs - j - 1;
        for (int e = tid; e < rem * rem; e += GW_NT) {
            const int i = j + 1 + e / rem, cc = j + 1 + e % rem;
            if (cc <= i) A[i * GWIDE + cc] -= A[i * GWIDE + j] * A[cc * GWIDE + j];
        }
    }
    __syncthreads();
    if (tid < 32) {
        for (int a = tid; a < gs; a += 32) vec[2 * GWIDE + a] = vec[a];
        __syncwarp();
        for (int j = 0; j < gs; j++) {
            const double yj = vec[2 * GWIDE + j] / A[j * GWIDE + j];
            __syncwarp();
            if (tid == 0) vec[2 * GWIDE + j] = yj;
            for (int i = j + 1 + tid; i < gs; i += 32) vec[2 * GWIDE + i] -= A[i * GWIDE + j] * yj;
            __syncwarp();
        }
        double s2 = 0.0;
        for (int a = tid; a < gs; a += 32) s2 = fma(vec[2 * GWIDE + a], vec[2 * GWIDE + a], s2);
        s2 = warp_sum(s2);
        if (tid == 0) d.bd[(size_t)c * d.pstride + g] = (quad + s2) / (double)gs;
    }
}
static size_t gw_smem_bytes() { return sizeof(double) * (size_t)(GWIDE * GWIDE + 2 * GW_RT * GWIDE + 4 * GW_RT + 4 * GWIDE + 40); }

// find_ind (utilities.cpp:113-130): the T selected groups (ascending) -> their columns, in order
__global__ void group_expand_kernel(const Dev d, const BatchDesc b)
{
    if (d.gate && *d.gate == 0) return;
    const int c = b.chain[blockIdx.x];
    if (d.done[c]) return;
    if (threadIdx.x != 0) return;
    const int *An = d.Anew + (size_t)c * d.kcap;
    int *out = d.AnewCols + (size_t)c * d.kcap;
    int cnt = 0;
    for (int a = 0; a < b.T; a++) {
        const int g = An[a];
        const int j0 = d.gidx[g], gs = d.gsz[g];
        for (int q = 0; q < gs && cnt < d.kcap; q++) out[cnt++] = j0 + q;
    }
    d.Tc[c] = cnt;
}

int launch_group_sacrifice(const Dev &d, const BatchDesc &b, cudaStream_t st)
{
    int ran = 0;
    static const bool serial = [] {
        const char *e = std::getenv("BESS_B200_GROUP_SERIAL");
        return e && e[0] == '1';
    }();
    if (d.family == FAM_COX || serial) {
        const dim3 grid((unsigned)((d.N + GS_NT - 1) / GS_NT), (unsigned)b.nch);
        if (d.family == FAM_COX) group_sacrifice_kernel<true><<<grid, GS_NT, 0, st>>>(d, b);
        else group_sacrifice_kernel<false><<<grid, GS_NT, 0, st>>>(d, b);
        ran |= GSAC_SERIAL;
    } else {
        static const bool per_chain = [] {
            const char *e = std::getenv("BESS_B200_GROUP_PER_CHAIN");
            return e && e[0] == '1';
        }();
        if (per_chain || b.nch == 1) {  // a single chain: the warp-per-(group, chain) kernel spreads the rows over 32 lanes
            const int wpb = GS_NT / 32;
            const dim3 grid((unsigned)((d.N + wpb - 1) / wpb), (unsigned)b.nch);
            group_sacrifice_warp_kernel<<<grid, GS_NT, 0, st>>>(d, b);
            ran |= GSAC_WARP;
        } else {
            const int wpb = GB_NT / 32;
            for (int k = 0; k < 3; k++) {  // one instantiation per width class of the narrow groups
                const int lo = d.gcls_off[k], hi = d.gcls_off[k + 1];
                if (hi <= lo) continue;
                const unsigned grid = (unsigned)((hi - lo + wpb - 1) / wpb);
                if (k == 0) group_sacrifice_batched_kernel<2><<<grid, GB_NT, 0, st>>>(d, b, lo, hi);
                else if (k == 1) group_sacrifice_batched_kernel<4><<<grid, GB_NT, 0, st>>>(d, b, lo, hi);
                else group_sacrifice_batched_kernel<GMAX><<<grid, GB_NT, 0, st>>>(d, b, lo, hi);
                ran |= GSAC_BATCHED2 << k;
            }
        }
    }
    CUDA_CHECK(cudaGetLastError());
    if (d.gmax > GMAX) {  // some groups are wider than the register kernels take
        const dim3 grid((unsigned)d.N, (unsigned)b.nch);
        const size_t smem = gw_smem_bytes();
        if (d.family == FAM_COX) {
            CUDA_CHECK(cudaFuncSetAttribute(group_sacrifice_wide_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            group_sacrifice_wide_kernel<true><<<grid, GW_NT, smem, st>>>(d, b);
        } else {
            CUDA_CHECK(cudaFuncSetAttribute(group_sacrifice_wide_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            group_sacrifice_wide_kernel<false><<<grid, GW_NT, smem, st>>>(d, b);
        }
        CUDA_CHECK(cudaGetLastError());
        ran |= GSAC_WIDE;
    }
    return ran;
}
void launch_group_expand(const Dev &d, const BatchDesc &b, cudaStream_t st)
{
    group_expand_kernel<<<b.nch, 32, 0, st>>>(d, b);
    CUDA_CHECK(cudaGetLastError());
}

}  // namespace bess
