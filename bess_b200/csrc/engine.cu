// Device engine: owns the design matrix and all chain state in HBM and drives the kernels of kernels.cu.
// See engine.h for the vocabulary.  All compute is on the GPU; there is no CPU fallback anywhere in this file.
#include "kernels.cuh"
#include "lm_path.cuh"
#include "device_utils.cuh"
#include "nccl_dl.h"

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <mutex>
#include <numeric>
#include <thread>
#include <utility>

namespace bess {

#define NCCL_CHECK(x)                                                                              \
    do {                                                                                           \
        ncclResult_t r_ = (x);                                                                     \
        if (r_ != ncclSuccess) {                                                                   \
            throw EngineError{std::string(#x) + ": " + nccl_api().GetErrorString(r_)};             \
        }                                                                                          \
    } while (0)

namespace {
// Stream-ordered allocation from the device's default memory pool (release threshold raised to "never" in
// DeviceContext): after the first call every alloc/free is a pool hit, no cudaMalloc/cudaFree (and no implicit
// device synchronisation) on the hot path.  All engine work is on ONE stream, so stream order == program order.
template <class T>
T *dalloc(cudaStream_t st, size_t count)
{
    T *p = nullptr;
    if (count == 0) count = 1;
    CUDA_CHECK(cudaMallocAsync((void **)&p, count * sizeof(T), st));
    return p;
}
template <class T>
void dfree(cudaStream_t st, T *&p)
{
    if (p) cudaFreeAsync((void *)p, st);
    p = nullptr;
}

// Workspaces cached per device for the life of the process.  A call on a 1000 x 5000 screened design is a few hundred
// microseconds of kernels; dozens of cudaMallocAsync / cudaMemsetAsync / pageable cudaMemcpyAsync calls (3-20 us of host
// time each) used to cost more than the kernels.  All small buffers are therefore bump-allocated from chunks that are
// created once and reused by every later call:
//   * DevArena     device-only scratch and state (stack discipline: mark / release; one stream, so stream order == program
//                  order and a released block can be handed out again at once);
//   * MirrorArena  host-to-device payloads: a pinned chunk and its device twin; the host fills the pinned side, flush()
//                  moves everything filled since the last flush with ONE truly asynchronous copy;
//   * pinned read-back blocks for results that the host only needs at the end of the call.
// Chunks never move, so pointers stay valid; a chunk that is too small is left in place and a larger one is appended
// (cudaMalloc -- only while the process warms up).
struct DevArena {
    struct Chunk {
        char *base = nullptr;
        size_t cap = 0, used = 0;
    };
    struct Mark {
        size_t chunk = 0, used = 0;
    };
    std::vector<Chunk> chunks;
    size_t cur = 0;
    void *alloc_bytes(size_t bytes)
    {
        bytes = (bytes + 255) & ~(size_t)255;
        if (bytes == 0) bytes = 256;
        for (;;) {
            if (cur < chunks.size()) {
                Chunk &c = chunks[cur];
                if (c.used + bytes <= c.cap) {
                    void *p = c.base + c.used;
                    c.used += bytes;
                    return p;
                }
                if (cur + 1 < chunks.size()) {
                    cur++;
                    chunks[cur].used = 0;
                    continue;
                }
            }
            Chunk c;
            c.cap = std::max<size_t>(bytes, (size_t)32 << 20);
            CUDA_CHECK(cudaMalloc((void **)&c.base, c.cap));
            chunks.push_back(c);
            cur = chunks.size() - 1;
        }
    }
    template <class T>
    T *alloc(size_t count)
    {
        return reinterpret_cast<T *>(alloc_bytes(count * sizeof(T)));
    }
    Mark mark() const { return Mark{cur, cur < chunks.size() ? chunks[cur].used : 0}; }
    void release(const Mark &mk)
    {
        if (chunks.empty()) return;
        cur = std::min(mk.chunk, chunks.size() - 1);
        chunks[cur].used = std::min(mk.used, chunks[cur].cap);
    }
    void reset()
    {
        cur = 0;
        if (!chunks.empty()) chunks[0].used = 0;
    }
};

struct MirrorArena {
    struct Chunk {
        char *pin = nullptr, *dev = nullptr;
        size_t cap = 0, used = 0, flushed = 0;
    };
    std::vector<Chunk> chunks;
    size_t cur = 0;
    // host <- where to write, returns the device address the bytes will have after flush()
    void *alloc_bytes(size_t bytes, void **host)
    {
        bytes = (bytes + 255) & ~(size_t)255;
        if (bytes == 0) bytes = 256;
        for (;;) {
            if (cur < chunks.size()) {
                Chunk &c = chunks[cur];
                if (c.used + bytes <= c.cap) {
                    *host = c.pin + c.used;
                    void *p = c.dev + c.used;
                    c.used += bytes;
                    return p;
                }
                if (cur + 1 < chunks.size()) {
                    cur++;
                    chunks[cur].used = chunks[cur].flushed = 0;
                    continue;
                }
            }
            Chunk c;
            c.cap = std::max<size_t>(bytes, (size_t)4 << 20);
            CUDA_CHECK(cudaMallocHost((void **)&c.pin, c.cap));
            CUDA_CHECK(cudaMalloc((void **)&c.dev, c.cap));
            chunks.push_back(c);
            cur = chunks.size() - 1;
        }
    }
    template <class T>
    T *alloc(size_t count, T **host)
    {
        void *h = nullptr;
        T *d = reinterpret_cast<T *>(alloc_bytes(count * sizeof(T), &h));
        *host = reinterpret_cast<T *>(h);
        return d;
    }
    void flush(cudaStream_t st)
    {
        for (size_t i = 0; i <= cur && i < chunks.size(); i++) {
            Chunk &c = chunks[i];
            if (c.used > c.flushed) {
                CUDA_CHECK(cudaMemcpyAsync(c.dev + c.flushed, c.pin + c.flushed, c.used - c.flushed, cudaMemcpyHostToDevice, st));
                c.flushed = c.used;
            }
        }
    }
    void reset()
    {
        cur = 0;
        if (!chunks.empty()) chunks[0].used = chunks[0].flushed = 0;
    }
};

// pinned host blocks for deferred read-backs (bump, reset per load())
struct PinnedArena {
    struct Chunk {
        char *pin = nullptr;
        size_t cap = 0, used = 0;
    };
    std::vector<Chunk> chunks;
    size_t cur = 0;
    void *alloc_bytes(size_t bytes)
    {
        bytes = (bytes + 63) & ~(size_t)63;
        if (bytes == 0) bytes = 64;
        for (;;) {
            if (cur < chunks.size()) {
                Chunk &c = chunks[cur];
                if (c.used + bytes <= c.cap) {
                    void *p = c.pin + c.used;
                    c.used += bytes;
                    return p;
                }
                if (cur + 1 < chunks.size()) {
                    cur++;
                    chunks[cur].used = 0;
                    continue;
                }
            }
            Chunk c;
            c.cap = std::max<size_t>(bytes, (size_t)1 << 20);
            CUDA_CHECK(cudaMallocHost((void **)&c.pin, c.cap));
            chunks.push_back(c);
            cur = chunks.size() - 1;
        }
    }
    template <class T>
    T *alloc(size_t count)
    {
        return reinterpret_cast<T *>(alloc_bytes(count * sizeof(T)));
    }
    void reset()
    {
        cur = 0;
        if (!chunks.empty()) chunks[0].used = 0;
    }
};

// Per-device resources that are expensive to create (stream, pinned mirrors) are cached for the life of the process
// and lent to one Engine at a time.
struct DeviceContext {
    DevArena ar;
    MirrorArena mir;
    PinnedArena rb;
    int coop_launch = -1;  // cudaDevAttrCooperativeLaunch, queried once
    int device = 0;
    int sm_count = 148;
    cudaStream_t st = nullptr;
    // pinned result mirrors, two of each (one per batch slot, Engine::Impl::Mirror)
    int *h_int = nullptr;        // [2][5][MAXC] done, l, tie, ks, gate
    double *h_dbl = nullptr;     // [2]([MAXC] coef0 + [2*MAXC] losses)
    int *h_A = nullptr;          // grow-only: [2][MAXC][kcap]
    double *h_bA = nullptr;
    size_t cap_A = 0;
    // resident path (lm_path.cu): result mirrors, two slots each, grow-only
    int *h_lp_i = nullptr;
    double *h_lp_d = nullptr;
    unsigned *h_lp_sync = nullptr;           // [2][LP_SYNC_WORDS]
    unsigned long long *h_lp_dbg = nullptr;  // [2][LP_NDBG]
    size_t cap_lp = 0;                        // entries per slot
    bool in_use = false;
    // pinned staging ring of the pageable-design upload (Engine::load), grow-only
    char *h_stage[2] = {nullptr, nullptr};
    size_t cap_stage = 0;
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};
    void reserve_stage(size_t bytes)
    {
        if (!ev_stage[0])
            for (int q = 0; q < 2; q++) CUDA_CHECK(cudaEventCreateWithFlags(&ev_stage[q], cudaEventDisableTiming));
        if (bytes <= cap_stage) return;
        for (int q = 0; q < 2; q++) {
            if (h_stage[q]) cudaFreeHost(h_stage[q]);
            h_stage[q] = nullptr;
        }
        cap_stage = 0;
        for (int q = 0; q < 2; q++) CUDA_CHECK(cudaMallocHost(&h_stage[q], bytes));
        cap_stage = bytes;
    }
    // NCCL communicator of the column-sharded mode, created once per (world, rank, unique id)
    ncclComm_t comm = nullptr;
    int comm_world = 0, comm_rank = -1;
    char comm_id[NCCL_UNIQUE_ID_BYTES] = {};
    void reserve_resident(size_t count)
    {
        if (!h_lp_sync) {
            CUDA_CHECK(cudaMallocHost(&h_lp_sync, 2 * LP_SYNC_WORDS * sizeof(unsigned)));
            CUDA_CHECK(cudaMallocHost(&h_lp_dbg, 2 * LP_NDBG * sizeof(unsigned long long)));
        }
        if (count <= cap_lp) return;
        if (h_lp_i) cudaFreeHost(h_lp_i);
        if (h_lp_d) cudaFreeHost(h_lp_d);
        h_lp_i = nullptr; h_lp_d = nullptr; cap_lp = 0;
        CUDA_CHECK(cudaMallocHost(&h_lp_i, 2 * count * sizeof(int)));
        CUDA_CHECK(cudaMallocHost(&h_lp_d, 2 * count * sizeof(double)));
        cap_lp = count;
    }
    void reserve_support(size_t count)
    {
        if (count <= cap_A) return;
        if (h_A) cudaFreeHost(h_A);
        if (h_bA) cudaFreeHost(h_bA);
        h_A = nullptr; h_bA = nullptr; cap_A = 0;
        CUDA_CHECK(cudaMallocHost(&h_A, 2 * count * sizeof(int)));
        CUDA_CHECK(cudaMallocHost(&h_bA, 2 * count * sizeof(double)));
        cap_A = count;
    }
};
std::mutex g_ctx_mu;
std::vector<DeviceContext *> g_ctx;

DeviceContext *acquire_context(int device)
{
    if (device >= 0) CUDA_CHECK(cudaSetDevice(device));
    int dev = 0;
    CUDA_CHECK(cudaGetDevice(&dev));
    {
        std::lock_guard<std::mutex> lk(g_ctx_mu);
        for (DeviceContext *c : g_ctx)
            if (c->device == dev && !c->in_use) {
                c->in_use = true;
                return c;
            }
    }
    cudaDeviceProp prop;
    CUDA_CHECK(cudaGetDeviceProperties(&prop, dev));
    if (prop.major < 10) throw EngineError{"bess_b200 needs an sm_100a (Blackwell) device"};
    DeviceContext *c = new DeviceContext();
    c->device = dev;
    c->sm_count = prop.multiProcessorCount;
    CUDA_CHECK(cudaStreamCreateWithFlags(&c->st, cudaStreamNonBlocking));
    cudaMemPool_t pool;
    CUDA_CHECK(cudaDeviceGetDefaultMemPool(&pool, dev));
    unsigned long long keep = ~0ULL;
    CUDA_CHECK(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    CUDA_CHECK(cudaMallocHost(&c->h_int, 2 * 5 * MAXC * sizeof(int)));
    CUDA_CHECK(cudaMallocHost(&c->h_dbl, 2 * 3 * MAXC * sizeof(double)));
    configure_kernels();
    c->in_use = true;
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    g_ctx.push_back(c);
    return c;
}
void release_context(DeviceContext *c)
{
    std::lock_guard<std::mutex> lk(g_ctx_mu);
    c->in_use = false;
}
int pick_fs(int nch)
{
    const int opts[] = {1, 2, 4, 6, 8, 12, 16, 24, 32};
    for (int o : opts)
        if (o >= nch) return o;
    throw EngineError{"too many chains (K must be <= 31)"};
}
}  // namespace

struct Engine::Impl {
    DeviceContext *ctx = nullptr;
    cudaStream_t st = nullptr;
    int sm_count = 148;
    Dev d{};
    // design
    double *X = nullptr;
    long long ldx = 0;
    // sparse design (Engine::load_csc) until screening or densify() makes it dense; csc_owned: the arrays are ours
    bool csc = false, csc_owned = false;
    long long *cp = nullptr;
    int *ri = nullptr;
    double *cv = nullptr;
    long long nnz = 0;
    // a sparse design normalised in place of densifying it (normalize of a CSC engine): the path sweeps the CSC arrays and
    // sees x~_ij = ((x_ij - cmean[j]) * cmul[j]) * crm[i] (Dev::ccp)
    bool csc_norm = false;
    double *cmean = nullptr, *cmul = nullptr, *crm = nullptr;
    void free_csc()
    {
        if (csc_owned) {
            dfree(st, cp);
            dfree(st, ri);
            dfree(st, cv);
        }
        dfree(st, cmean);
        dfree(st, cmul);
        dfree(st, crm);
        cp = nullptr; ri = nullptr; cv = nullptr;
        csc = csc_owned = csc_norm = false;
        nnz = 0;
    }
    int n = 0, p = 0, npad = 0;
    double *y = nullptr, *w = nullptr;  // [npad] device
    std::vector<double> hy, hw;          // host copies (current, i.e. after normalisation)
    // sweep scratch for the setup phases (screening / normalisation), FS = 1
    double *raw = nullptr;  // [2][FS][pstride]
    // chain setup
    int K = 0, nchains = 1;
    int *testrows = nullptr, *ntest = nullptr;
    double *lfact = nullptr;
    double *loss_scratch = nullptr, *loss_out = nullptr;
    int *always = nullptr;
    int n_always = 0;
    StateSlots slots{};
    // ---- batches in flight.  Two slots alternate: a batch's kernels carry a private copy of the descriptor (ridge level,
    // gate counter), its results land in the slot's pinned mirror, so the next path step can be enqueued before the
    // host has read the current one.
    struct Ticket {
        Dev d{};
        BatchDesc b{};
        LossDesc ld{};
        bool has_jobs = false, fused = false, pending = false;
        bool resident = false, loss_kernel = false;  // resident: one lm_path launch; loss_kernel: jobs it cannot express
        LpDesc lp{};
        int T = 0, slot = 0, enq = 0, cmin = 0, cmax = 0;
        long long launches = 0;
        cudaEvent_t ev = nullptr;
    };
    struct Mirror {
        int *done = nullptr, *l = nullptr, *tie = nullptr, *ks = nullptr, *gate = nullptr, *A = nullptr;
        double *coef0 = nullptr, *loss = nullptr, *bA = nullptr;
    };
    Ticket tk[2];
    Mirror mir[2];
    unsigned long long seq = 0;
    int *n_active2 = nullptr;  // device [2]: the alternating gate counters (Dev::n_active / Dev::prev_active)
    double *ck0 = nullptr, *ck1 = nullptr;
    int *ci0 = nullptr, *ci1 = nullptr;
    long long cstride = 0;
    // pinned host mirrors (owned by the DeviceContext)
    int *h_A = nullptr;
    int *gidx = nullptr, *gsz = nullptr;  // group selection: device copies of Engine::g_index_ / g_size_
    int *glist = nullptr;                 // the narrow groups (<= GMAX variables) ordered by width class <= 2 | <= 4 | <= 8
    int gcls_off[4] = {0, 0, 0, 0};       // class k = glist[gcls_off[k] .. gcls_off[k + 1])
    int Tmax = 0;                          // largest sparsity level (in groups when grouped) the workspaces hold
    double *h_bA = nullptr;
    bool chains_ready = false;
    bool x_owned = true;
    bool tie_exact = false;  // Engine::set_tie_exact
    int cl_chains = 0;       // Engine::set_cluster_chains
    // column-sharded mode
    ncclComm_t comm = nullptr;
    int world = 1, rank = 0;
    Cand *cand_s = nullptr, *cand_r = nullptr;  // [C][kcap] local candidates, [world][C][kcap] gathered
    double *mv = nullptr;                        // [C][world * kcap] merged candidate values
    int *mi = nullptr;                           // ... and global indices
    long long mstride = 0;
    int *Aloc = nullptr;                         // [C][kcap] local top-k (local column indices)
    double *AXs = nullptr;                       // [C][n][T] this rank's contribution to the active columns
    // ---- resident path (lm_path.cu)
    bool lp_ok = false;
    std::string lp_why = "chains not set up";
    int lp_ns = 0;
    size_t lp_res_count = 0;               // result entries per slot
    unsigned *lp_sync = nullptr;           // device [2][LP_SYNC_WORDS]
    LpCand *lp_cand = nullptr;
    int *lp_ncand = nullptr;
    double *lp_pub = nullptr, *lp_tau = nullptr;
    int *lp_res_i = nullptr;               // device [2][lp_res_count]
    double *lp_res_d = nullptr;
    unsigned long long *lp_dbg = nullptr;  // device [LP_NDBG]
    double *lp_R = nullptr;                // device [2][npad][MAXC] residual matrices of the two chain groups
    unsigned long long *lp_trace = nullptr;  // device, only with $BESS_B200_TRACE: phase time stamps of the resident kernel
    double lp_counters[24] = {};
    double lp_owner[4 * MAXC] = {};
    // ---- per-category device timing (CUDA events on the engine stream), enabled by Engine::set_profiling
    bool prof = false;
    struct Span { cudaEvent_t a, b; int cat; };
    std::vector<Span> spans;
    std::vector<cudaEvent_t> pool;
    double cat_ms[PROF_NCAT] = {};
    long long cat_n[PROF_NCAT] = {};
    cudaEvent_t get_event()
    {
        if (!pool.empty()) { cudaEvent_t e = pool.back(); pool.pop_back(); return e; }
        cudaEvent_t e;
        CUDA_CHECK(cudaEventCreate(&e));
        return e;
    }
    int span_begin(int cat)
    {
        if (!prof) return -1;
        Span sp{get_event(), get_event(), cat};
        CUDA_CHECK(cudaEventRecord(sp.a, st));
        spans.push_back(sp);
        return (int)spans.size() - 1;
    }
    void span_end(int id)
    {
        if (id >= 0) CUDA_CHECK(cudaEventRecord(spans[id].b, st));
    }
    // call only after a stream synchronize
    void collect_spans()
    {
        for (Span &sp : spans) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, sp.a, sp.b) == cudaSuccess) {
                cat_ms[sp.cat] += ms;
                cat_n[sp.cat]++;
            }
            pool.push_back(sp.a);
            pool.push_back(sp.b);
        }
        spans.clear();
    }

    // ---- workspace bookkeeping (DeviceContext arenas).  Stack order in the device arena: [load] [sweep buffers]
    // [phase scratch | chain state].  config_sweep releases everything above the load mark, so it ends the life of the
    // chain state as well (setup_chains re-creates it right afterwards).
    DevArena::Mark mk_load{}, mk_sweep_end{};
    bool have_sweep = false;
    // read-backs that are only awaited when somebody asks for them
    int *h_sel = nullptr;          // pinned: kept columns of the last screening
    int *h_sel_tie = nullptr;
    int sel_count = 0;
    bool sel_pending = false;
    // screening's gather of the kept columns (dense, unsharded), deferred so that normalize() can fuse it into its one
    // launch: X (the screened design, allocated but not yet written) <- gsrc[:, gsel].  gsel is the arena list of
    // screen_select, alive until the next config_sweep; gsrc is the raw design, freed with the gather when owned.
    const int *gsel = nullptr;
    double *gsrc = nullptr;
    long long gsrc_ld = 0;
    bool gsrc_owned = false;
    void drop_gather_source()
    {
        if (gsrc_owned) dfree(st, gsrc);
        gsel = nullptr;
        gsrc = nullptr;
        gsrc_owned = false;
    }
    double *h_mean = nullptr, *h_norm = nullptr;  // pinned: column statistics of the last normalisation
    bool stats_pending = false;
    bool stats_have_mean = false;

    void free_sweep_buffers()
    {
        d.G = d.W = d.TH = d.C2 = nullptr;
        d.part = d.c2sum = d.bd = nullptr;
        raw = nullptr;
        have_sweep = false;
    }
    void free_chain_buffers()
    {
        Impl &m = *this;
        // everything of the chain state lives in the arenas and dies with the next config_sweep / load; only the
        // column-sharded exchange buffers are stream-ordered allocations
        d.rows = nullptr; d.ntrain = nullptr; d.ytr = d.wtr = nullptr; d.ks = nullptr; d.A = nullptr; d.bA = nullptr;
        d.coef0 = d.coef0_level = nullptr; d.Anew = nullptr; d.hist = nullptr; d.l = d.done = d.tie = d.tie_acc = nullptr;
        n_active2 = nullptr;
        d.n_active = nullptr;
        d.betaD = d.XA = d.XB = d.vec = d.Smat = d.Spart = d.cw = d.xtx = nullptr;
        testrows = ntest = nullptr; lfact = loss_scratch = loss_out = nullptr; always = nullptr;
        ck0 = ck1 = nullptr; ci0 = ci1 = nullptr;
        dfree(m.st, cand_s); dfree(m.st, cand_r); dfree(m.st, mv); dfree(m.st, mi); dfree(m.st, Aloc); dfree(m.st, AXs);
        dfree(m.st, d.AXr); dfree(m.st, d.AXk);
        slots = StateSlots{};
        d.Tc = nullptr; d.AnewCols = nullptr;
        lp_sync = nullptr; lp_cand = nullptr; lp_ncand = nullptr; lp_pub = lp_tau = nullptr;
        lp_res_i = nullptr; lp_res_d = nullptr; lp_dbg = nullptr; lp_R = nullptr;
        lp_ok = false;
        chains_ready = false;
    }
    // (re)allocate the sweep vectors / partial buffers for FS chain slots over the current (n, p)
    void config_sweep(int FS)
    {
        Impl &m = *this;
        free_chain_buffers();
        free_sweep_buffers();
        ctx->ar.release(mk_load);
        d.gate = nullptr;
        d.X = X; d.ldx = ldx; d.n = n; d.p = p; d.FS = FS;
        d.pstride = (p + 1) & ~1LL;
        // row splits.  One chain (streaming kernel): enough CTAs to fill the machine several times over.
        // Batched chains (bulk-TMA kernel, 3 CTAs of 256 columns per SM): every extra split costs a set of partial
        // vectors (written by the sweep, re-read by finish), so pick the split count that balances whole waves of
        // CTAs against that traffic: score = wave efficiency / (1 + partial bytes / X bytes).
        const long long ntiles = (p + 2LL * SWEEP_NT - 1) / (2LL * SWEEP_NT);
        long long smax = std::max<long long>(1, n / SWEEP_RC);
        long long S;
        const double part_bytes_per_split = 8.0 * FS * (d.family == FAM_LM ? 1 : (d.family == FAM_COX ? 5 : 2)) * (double)p;
        if (FS == 1 || part_bytes_per_split < 16.0e6) {
            // partial vectors stay in L2: splits are free, fill the machine several times over
            const long long want = (6LL * sm_count + ntiles - 1) / ntiles;
            S = std::max<long long>(1, std::min(want, smax));
        } else {
            const double slots = 3.0 * sm_count;
            const int nq = d.family == FAM_LM ? 1 : (d.family == FAM_COX ? 5 : 2);
            double best = -1.0;
            S = 1;
            for (long long cand = 1; cand <= smax; cand++) {
                const double waves = (double)(ntiles * cand) / slots;
                const double eff = waves >= 1.0 ? waves / std::ceil(waves) : waves;
                const double extra = (double)cand * FS * nq * 16.0 / (8.0 * n);
                const double score = eff / (1.0 + extra);
                if (score > best * 1.0001) {
                    best = score;
                    S = cand;
                }
            }
        }
        if (csc_norm) S = 1;  // the CSC sweep reduces each column over all rows itself
        int rps = (int)((n + S - 1) / S);
        rps = (rps + 1) & ~1;
        d.rows_per_split = rps;
        d.S = (n + rps - 1) / rps;
        const size_t vsz = ((size_t)npad * FS + 31) & ~(size_t)31;  // keeps the four vectors 256-byte aligned
        double *vecs = ctx->ar.alloc<double>(4 * vsz);  // one block, one memset
        d.G = vecs; d.W = vecs + vsz; d.TH = vecs + 2 * vsz; d.C2 = vecs + 3 * vsz;
        CUDA_CHECK(cudaMemsetAsync(vecs, 0, 4 * vsz * 8, st));
        d.part = ctx->ar.alloc<double>((size_t)d.S * 5 * FS * d.pstride);
        d.c2sum = ctx->ar.alloc<double>((size_t)d.S * FS);
        d.bd = ctx->ar.alloc<double>((size_t)FS * d.pstride);
        raw = ctx->ar.alloc<double>((size_t)2 * FS * d.pstride);
        d.ccp = nullptr; d.cri = nullptr; d.ccv = nullptr;
        d.clong = nullptr; d.nlong = 0;
        d.cmean = d.cmul = d.crm = nullptr;
        d.csum = d.cpre = nullptr;
        if (csc_norm) {
            d.ccp = cp; d.cri = ri; d.ccv = cv;
            d.cmean = cmean; d.cmul = cmul; d.crm = crm;
            d.csum = ctx->ar.alloc<double>((size_t)2 * FS);
            d.cpre = d.family == FAM_COX ? ctx->ar.alloc<double>((size_t)npad * FS) : nullptr;
            const double mean_len = (double)nnz / (double)p;
            d.csc_g = mean_len < 4.0 ? 2 : (mean_len < 16.0 ? 8 : 32);
            d.csc_nnz = nnz;
            // a column longer than 16 steps of its G lanes (the frequent terms of a power-law design) is swept by a CTA of
            // its own, so that it does not hold the rest of the grid up
            d.clong_thr = 16LL * d.csc_g;
            int *list = ctx->ar.alloc<int>((size_t)p);
            int *cnt = ctx->ar.alloc<int>(1);
            int *h_cnt = ctx->rb.alloc<int>(1);
            CUDA_CHECK(cudaMemsetAsync(cnt, 0, sizeof(int), st));
            launch_csc_long_list(cp, p, d.clong_thr, list, cnt, st);
            CUDA_CHECK(cudaMemcpyAsync(h_cnt, cnt, sizeof(int), cudaMemcpyDeviceToHost, st));
            CUDA_CHECK(cudaStreamSynchronize(st));
            d.clong = list;
            d.nlong = *h_cnt;
        }
        mk_sweep_end = ctx->ar.mark();
        have_sweep = true;
    }
    // Stage a host vector for the device: the returned device pointer is valid after the next mirror flush.
    // pad: number of doubles of the device block (>= v.size(), the tail is zero)
    double *stage_vec(const double *v, size_t count, size_t pad)
    {
        double *h = nullptr;
        double *dv = ctx->mir.alloc<double>(pad, &h);
        std::memcpy(h, v, count * 8);
        if (pad > count) std::memset(h + count, 0, (pad - count) * 8);
        return dv;
    }
    // slot f of a [npad][FS] sweep vector <- host vector (FS == 1: the staged block itself becomes the vector)
    void put_vec(double *&dst, int f, const std::vector<double> &v)
    {
        if (d.FS == 1 && f == 0) {
            dst = stage_vec(v.data(), v.size(), (size_t)npad);
            ctx->mir.flush(st);
            return;
        }
        double *sv = stage_vec(v.data(), v.size(), v.size());
        ctx->mir.flush(st);
        CUDA_CHECK(cudaMemcpy2DAsync(dst + f, (size_t)d.FS * 8, sv, 8, 8, v.size(), cudaMemcpyDeviceToDevice, st));
    }
    void await_stream() { CUDA_CHECK(cudaStreamSynchronize(st)); }
};

Engine::Engine(int device)
{
    d_ = new Impl();
    try {
        d_->ctx = acquire_context(device);
    } catch (...) {
        delete d_;
        d_ = nullptr;
        throw;
    }
    DeviceContext *c = d_->ctx;
    d_->st = c->st;
    d_->sm_count = c->sm_count;
    for (int q = 0; q < 2; q++) {
        Impl::Mirror &h = d_->mir[q];
        int *hi = c->h_int + (size_t)q * 5 * MAXC;
        h.done = hi;
        h.l = hi + MAXC;
        h.tie = hi + 2 * MAXC;
        h.ks = hi + 3 * MAXC;
        h.gate = hi + 4 * MAXC;
        h.coef0 = c->h_dbl + (size_t)q * 3 * MAXC;
        h.loss = h.coef0 + MAXC;
    }
}

Engine::~Engine()
{
    if (!d_) return;
    Impl &m = *d_;
    cudaSetDevice(m.ctx->device);
    cudaStreamSynchronize(m.st);
    m.collect_spans();
    for (cudaEvent_t e : m.pool) cudaEventDestroy(e);
    m.free_chain_buffers();
    m.free_sweep_buffers();
    m.drop_gather_source();
    if (m.x_owned) dfree(m.st, m.X);
    m.free_csc();
    dfree(m.st, m.gidx); dfree(m.st, m.gsz); dfree(m.st, m.glist);
    cudaStreamSynchronize(m.st);
    m.ctx->ar.reset();
    m.ctx->mir.reset();
    m.ctx->rb.reset();
    release_context(m.ctx);
    delete d_;
}

void Engine::set_profiling(bool on) { d_->prof = on; }
void Engine::set_tie_exact(bool on) { d_->tie_exact = on; }
void Engine::set_cluster_chains(int nch) { d_->cl_chains = nch; }
bool Engine::tie_exact() const { return d_->tie_exact; }

// max_k of the reference, statement for statement (utilities.cpp:179-188): an index array 0..N-1, std::nth_element with
// the comparator vec(i) > vec(j), std::sort of the first k.  Which of several equal values at the boundary survive is
// whatever libstdc++'s introselect leaves in front -- reproduced by running the same algorithm on the same ordering.
static void host_max_k(const double *vec, int N, int k, int *out)
{
    std::vector<int> ind((size_t)N);
    std::iota(ind.begin(), ind.end(), 0);
    auto rule = [vec](int i, int j) -> bool { return vec[i] > vec[j]; };
    std::nth_element(ind.data(), ind.data() + k, ind.data() + ind.size(), rule);
    std::sort(ind.data(), ind.data() + k);
    std::copy(ind.data(), ind.data() + k, out);
}

bool Engine::has_comm() const { return d_->comm != nullptr && d_->world > 1; }

void Engine::allreduce_mean(std::vector<double> &v)
{
    allreduce_sum(v);
    // the sum is reduced in the same order on every rank (one collective), the division is exact arithmetic on equal
    // inputs: all ranks hold bit-identical means
    for (double &x : v) x /= (double)d_->world;
}
void Engine::allreduce_sum(std::vector<double> &v)
{
    Impl &m = *d_;
    if (!has_comm()) throw EngineError{"allreduce: no communicator (call init_shard / init_comm first)"};
    if (v.empty()) return;
    const NcclApi &api = nccl_api();
    double *buf = dalloc<double>(m.st, v.size());
    CUDA_CHECK(cudaMemcpyAsync(buf, v.data(), v.size() * 8, cudaMemcpyHostToDevice, m.st));
    NCCL_CHECK(api.AllReduce(buf, buf, v.size(), ncclDouble, ncclSum, m.comm, m.st));
    CUDA_CHECK(cudaMemcpyAsync(v.data(), buf, v.size() * 8, cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    dfree(m.st, buf);
}

void Engine::init_shard(int world, int rank, const void *unique_id, long long col_lo, long long p_total)
{
    if (p_total > 2147483646LL) throw EngineError{"init_shard: p_total must fit a 32-bit index"};
    long long lo, hi;
    if (world < 2) throw EngineError{"init_shard: world must be >= 2"};
    shard_range(p_total, world, rank, &lo, &hi);
    if (lo != col_lo) throw EngineError{"init_shard: col_lo does not match bess_b200_shard_range(p_total, world, rank)"};
    init_comm(world, rank, unique_id);
    sharded_ = true;
    world_ = world;
    rank_ = rank;
    col_lo_ = col_lo;
    p_total_ = p_total;
}
void Engine::init_comm(int world, int rank, const void *unique_id)
{
    Impl &m = *d_;
    if (world < 2) throw EngineError{"init_comm: world must be >= 2"};
    if (rank < 0 || rank >= world) throw EngineError{"init_comm: rank out of range"};
    if (!unique_id) throw EngineError{"init_comm: the NCCL unique id is missing"};
    DeviceContext *c = m.ctx;
    if (!(c->comm && c->comm_world == world && c->comm_rank == rank &&
          std::memcmp(c->comm_id, unique_id, NCCL_UNIQUE_ID_BYTES) == 0)) {
        const NcclApi &api = nccl_api();
        if (c->comm) {
            api.CommDestroy(c->comm);
            c->comm = nullptr;
        }
        ncclUniqueId id;
        std::memcpy(id.internal, unique_id, NCCL_UNIQUE_ID_BYTES);
        NCCL_CHECK(api.CommInitRank(&c->comm, world, id, rank));
        c->comm_world = world;
        c->comm_rank = rank;
        std::memcpy(c->comm_id, unique_id, NCCL_UNIQUE_ID_BYTES);
    }
    m.comm = c->comm;
    m.world = world;
    m.rank = rank;
}
void Engine::profile(double *ms_out, long long *n_out) const
{
    if (d_->prof && !d_->spans.empty()) {  // pipelined batches leave their spans for the end of the path
        cudaStreamSynchronize(d_->st);
        d_->collect_spans();
    }
    for (int i = 0; i < PROF_NCAT; i++) {
        ms_out[i] = d_->cat_ms[i];
        n_out[i] = d_->cat_n[i];
    }
}

// Host -> device copy of a design that sits in PAGEABLE host memory (what pywrap_bess gets from R / numpy): the driver's
// own pageable path stages through one thread's memcpy (measured 11 GB/s: 183 of the 357 ms of a config-3 call).  Here a
// few host threads fill a two-buffer pinned ring in parallel while the previous buffer's DMA runs: the copy approaches
// the PCIe rate of a pinned source.  Row chunks keep the 2-D pitch conversion (p -> ldx columns) inside the DMA.
// The ring itself: chunk(k) gives the host bytes of chunk k (at most buf_bytes), dma(k, stage, bytes) enqueues the copy of
// the staged chunk.
template <class Chunk, class Dma>
static void staged_upload(DeviceContext *c, cudaStream_t st, size_t buf_bytes, int nchunks, Chunk chunk, Dma dma)
{
    c->reserve_stage(buf_bytes);
    static const int T = [] {
        const char *e = std::getenv("BESS_B200_UPLOAD_THREADS");
        // measured on the 16-core box, 2 GB design: 1 thread 147 ms, 4: 90, 8: 72, 12: 41 (49 GB/s; the driver's own path 183)
        int t = e ? std::atoi(e) : (int)std::min(12u, std::max(1u, std::thread::hardware_concurrency() * 3 / 4));
        return std::max(1, std::min(t, 32));
    }();
    std::atomic<int> go{-1};
    std::atomic<long long> done{0};
    auto worker = [&](int t) {
        for (int k = 0; k < nchunks; k++) {
            while (go.load(std::memory_order_acquire) < k) std::this_thread::yield();
            const std::pair<const char *, size_t> ck = chunk(k);
            const size_t b0 = ck.second * (size_t)t / (size_t)T, b1 = ck.second * (size_t)(t + 1) / (size_t)T;
            std::memcpy(c->h_stage[k & 1] + b0, ck.first + b0, b1 - b0);
            done.fetch_add(1, std::memory_order_release);
        }
    };
    std::vector<std::thread> pool;
    for (int t = 1; t < T; t++) pool.emplace_back(worker, t);
    try {
        for (int k = 0; k < nchunks; k++) {
            if (k >= 2) CUDA_CHECK(cudaEventSynchronize(c->ev_stage[k & 1]));  // the DMA that read this buffer last
            go.store(k, std::memory_order_release);
            const std::pair<const char *, size_t> ck = chunk(k);
            std::memcpy(c->h_stage[k & 1], ck.first, ck.second / (size_t)T);  // the calling thread is worker 0
            done.fetch_add(1, std::memory_order_release);
            while (done.load(std::memory_order_acquire) < (long long)T * (k + 1)) std::this_thread::yield();
            dma(k, c->h_stage[k & 1], ck.second);
            CUDA_CHECK(cudaEventRecord(c->ev_stage[k & 1], st));
        }
    } catch (...) {
        go.store(nchunks, std::memory_order_release);  // let the workers run out (they copy into a live buffer: harmless)
        for (auto &th : pool) th.join();
        throw;
    }
    for (auto &th : pool) th.join();
    // the ring may be refilled by the next call only after these DMAs: the next upload's k < 2 chunks do not wait on the
    // events, so drain them here (the caller synchronises the stream soon anyway)
    CUDA_CHECK(cudaEventSynchronize(c->ev_stage[(nchunks - 1) & 1]));
    if (nchunks > 1) CUDA_CHECK(cudaEventSynchronize(c->ev_stage[(nchunks - 2) & 1]));
}

static void upload_pageable(DeviceContext *c, cudaStream_t st, double *dX, size_t ldx, const double *x, int n, int p)
{
    const size_t row_bytes = (size_t)p * 8;
    const size_t buf_bytes = std::max<size_t>((size_t)32 << 20, row_bytes);
    const size_t rows_per = std::max<size_t>(1, buf_bytes / row_bytes);
    const int nchunks = (int)(((size_t)n + rows_per - 1) / rows_per);
    auto chunk = [&](int k) {
        const size_t r0 = (size_t)k * rows_per, rows = std::min(rows_per, (size_t)n - r0);
        return std::make_pair(reinterpret_cast<const char *>(x) + r0 * row_bytes, rows * row_bytes);
    };
    auto dma = [&](int k, const char *stage, size_t bytes) {
        const size_t r0 = (size_t)k * rows_per;
        CUDA_CHECK(cudaMemcpy2DAsync(dX + r0 * ldx, ldx * 8, stage, row_bytes, row_bytes, bytes / row_bytes,
                                     cudaMemcpyHostToDevice, st));
    };
    staged_upload(c, st, buf_bytes, nchunks, chunk, dma);
}

// Host -> device copy of a 1-D host array (the CSC arrays of load_csc): pageable memory of 64 MB or more goes through the
// same ring in 32 MB chunks, pinned memory (and small arrays) with one direct copy.
static void upload_1d(DeviceContext *c, cudaStream_t st, void *dst, const void *src, size_t bytes)
{
    if (bytes == 0) return;
    bool pageable = false;
    if (bytes >= ((size_t)64 << 20)) {
        cudaPointerAttributes pa;
        const cudaError_t e = cudaPointerGetAttributes(&pa, src);
        if (e != cudaSuccess) cudaGetLastError();
        pageable = e != cudaSuccess || pa.type == cudaMemoryTypeUnregistered;
    }
    if (!pageable) {
        CUDA_CHECK(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyHostToDevice, st));
        return;
    }
    const size_t buf_bytes = (size_t)32 << 20;
    const int nchunks = (int)((bytes + buf_bytes - 1) / buf_bytes);
    auto chunk = [&](int k) {
        const size_t b0 = (size_t)k * buf_bytes;
        return std::make_pair(reinterpret_cast<const char *>(src) + b0, std::min(buf_bytes, bytes - b0));
    };
    auto dma = [&](int k, const char *stage, size_t nb) {
        CUDA_CHECK(cudaMemcpyAsync(reinterpret_cast<char *>(dst) + (size_t)k * buf_bytes, stage, nb, cudaMemcpyHostToDevice, st));
    };
    staged_upload(c, st, buf_bytes, nchunks, chunk, dma);
}

void Engine::load(const double *x, int n, int p, bool x_on_device, const double *y, const double *weight, int family,
                  bool borrow)
{
    Impl &m = *d_;
    begin_load(n, p, family);
    // A device-resident design with an even column count can be used in place while it is only READ (screening
    // replaces it by the gathered columns); normalize() takes a private copy otherwise.
    if (borrow && x_on_device && (p % 2 == 0) && ((uintptr_t)x % 16 == 0)) {
        m.X = const_cast<double *>(x);
        m.x_owned = false;
    } else {
        m.x_owned = true;
        m.X = dalloc<double>(m.st, (size_t)n * m.ldx);
        if (m.ldx != p) CUDA_CHECK(cudaMemsetAsync(m.X, 0, (size_t)n * m.ldx * 8, m.st));
        const int sp = m.span_begin(7);
        bool pageable = false;
        if (!x_on_device && (size_t)n * p * 8 >= ((size_t)64 << 20)) {
            cudaPointerAttributes pa;
            const cudaError_t e = cudaPointerGetAttributes(&pa, x);
            if (e != cudaSuccess) cudaGetLastError();  // (older drivers report an unregistered pointer as an error)
            pageable = e != cudaSuccess || pa.type == cudaMemoryTypeUnregistered;
        }
        if (pageable)
            upload_pageable(m.ctx, m.st, m.X, (size_t)m.ldx, x, n, p);
        else
            CUDA_CHECK(cudaMemcpy2DAsync(m.X, (size_t)m.ldx * 8, x, (size_t)p * 8, (size_t)p * 8, n,
                                         x_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, m.st));
        m.span_end(sp);
    }
    end_load(y, weight, family);
}

// what every load shares: the previous problem's buffers go, the shapes are set
void Engine::begin_load(int n, int p, int family)
{
    Impl &m = *d_;
    if (n < 2 || p < 1) throw EngineError{"load: need n >= 2 and p >= 1"};
    stats_.max_cluster = 0;
    if (family < 1 || family > 4) throw EngineError{"load: model_type must be 1..4"};
    if (sharded_) {
        long long lo, hi;
        shard_range(p_total_, world_, rank_, &lo, &hi);
        if (hi - lo != p) throw EngineError{"load: the shard must hold exactly the columns of bess_b200_shard_range"};
    }
    m.free_chain_buffers();
    m.free_sweep_buffers();
    m.drop_gather_source();
    if (m.x_owned) dfree(m.st, m.X);
    m.free_csc();
    m.X = nullptr;
    m.x_owned = true;
    // a new problem: every arena block of the previous one is dead once the stream has drained
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    m.ctx->ar.reset();
    m.ctx->mir.reset();
    m.ctx->rb.reset();
    m.sel_pending = m.stats_pending = false;
    n_ = n; p_ = p; family_ = family;
    m.n = n; m.p = p; m.npad = (n + 1) & ~1;
    m.ldx = (p + 1) & ~1LL;
}

// the response and weights, and the kernel descriptor of the new problem
void Engine::end_load(const double *y, const double *weight, int family)
{
    Impl &m = *d_;
    const int n = m.n;
    m.hy.assign(y, y + n);
    m.hw.assign(weight, weight + n);
    m.y = m.stage_vec(y, (size_t)n, (size_t)m.npad);
    m.w = m.stage_vec(weight, (size_t)n, (size_t)m.npad);
    m.ctx->mir.flush(m.st);
    m.mk_load = m.ctx->ar.mark();
    m.d = Dev{};
    m.d.family = family;
    m.d.sharded = sharded_ ? 1 : 0;
    m.d.col_lo = sharded_ ? (int)col_lo_ : 0;
    // (the column statistics are p-sized host vectors: at p = 500000 zero-filling them costs more than the whole path of
    // a screened call, so they are only materialised when somebody reads them -- ensure_stats)
    h_xmean_.clear();
    h_xnorm_.clear();
    y_mean_ = 0.0;
}

void Engine::load_csc(const long long *colptr, const int *rowidx, const double *values, int n, int p, long long nnz,
                      bool on_device, const double *y, const double *weight, int family)
{
    Impl &m = *d_;
    if (n < 2 || p < 1) throw EngineError{"load_csc: need n >= 2 and p >= 1"};
    if (family < 1 || family > 4) throw EngineError{"load_csc: model_type must be 1..4"};
    if (sharded_) throw EngineError{"load_csc: a sparse design is single-GPU only"};
    if (nnz < 0 || !colptr || (nnz > 0 && (!rowidx || !values))) throw EngineError{"x_csc: colptr, rowidx and values must be given"};
    if (!on_device) {  // O(p) on the host; device arrays are checked by csc_check_kernel
        if (colptr[0] != 0) throw EngineError{"x_csc: colptr[0] must be 0"};
        for (long long j = 0; j < p; j++)
            if (colptr[j + 1] < colptr[j])
                throw EngineError{"x_csc: colptr must be non-decreasing (colptr[" + std::to_string(j + 1) + "] < colptr[" +
                                  std::to_string(j) + "])"};
        if (colptr[p] != nnz) throw EngineError{"x_csc: colptr[p] must equal nnz"};
    }
    begin_load(n, p, family);
    const int sp = m.span_begin(7);
    if (on_device) {  // only ever read: used in place
        m.cp = const_cast<long long *>(colptr);
        m.ri = const_cast<int *>(rowidx);
        m.cv = const_cast<double *>(values);
        m.csc_owned = false;
    } else {
        m.csc_owned = true;
        m.cp = dalloc<long long>(m.st, (size_t)p + 1);
        m.ri = dalloc<int>(m.st, (size_t)nnz);
        m.cv = dalloc<double>(m.st, (size_t)nnz);
        upload_1d(m.ctx, m.st, m.cp, colptr, ((size_t)p + 1) * 8);
        upload_1d(m.ctx, m.st, m.ri, rowidx, (size_t)nnz * 4);
        upload_1d(m.ctx, m.st, m.cv, values, (size_t)nnz * 8);
    }
    m.span_end(sp);
    m.csc = true;
    m.nnz = nnz;
    end_load(y, weight, family);
    int *h_flag = m.ctx->rb.alloc<int>(1);
    int *d_flag = m.ctx->ar.alloc<int>(1);
    CUDA_CHECK(cudaMemsetAsync(d_flag, 0, 4, m.st));
    launch_csc_check(m.cp, m.ri, n, p, nnz, d_flag, m.st);
    CUDA_CHECK(cudaMemcpyAsync(h_flag, d_flag, 4, cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    stats_.kernel_launches += 1;
    m.mk_load = m.ctx->ar.mark();
    const int bad = *h_flag;
    if (bad) {
        m.free_csc();
        std::string why;
        if (bad & CSC_BAD_COLPTR) why += " colptr must start at 0, be non-decreasing and end at nnz;";
        if (bad & CSC_BAD_ROW) why += " a row index is outside [0, n);";
        if (bad & CSC_UNSORTED) why += " row indices must be strictly increasing inside every column (unsorted or duplicate);";
        why.pop_back();
        throw EngineError{"x_csc:" + why};
    }
}

bool Engine::sparse() const { return d_->csc; }

void Engine::densify()
{
    Impl &m = *d_;
    if (!m.csc) return;
    const long long ldx = ((long long)m.p + 1) & ~1LL;
    const size_t bytes = (size_t)m.n * (size_t)ldx * 8;
    size_t free_b = 0, total_b = 0;
    CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    if (bytes > free_b)
        throw EngineError{"sparse design without screening: its dense form (" + std::to_string(bytes >> 20) + " MB) does not fit "
                          "the device (" + std::to_string(free_b >> 20) + " MB free); screen it (is_screening) instead"};
    double *X = dalloc<double>(m.st, (size_t)m.n * ldx);
    CUDA_CHECK(cudaMemsetAsync(X, 0, bytes, m.st));
    const int sp = m.span_begin(5);
    launch_csc_densify(m.cp, m.ri, m.cv, nullptr, m.p, X, ldx, m.st);
    m.span_end(sp);
    stats_.kernel_launches += 1;
    m.free_csc();  // stream-ordered: the arrays live until the densify kernel is done
    m.X = X;
    m.x_owned = true;
    m.ldx = ldx;
}

static int *screen_select(Engine::Impl &m, EngineStats &st, int family, int size, const std::vector<int> &always_select,
                          std::vector<double> *vals_out, std::vector<int> *sel_out, bool to_pinned);

// The deferred gather of screen_enqueue, for every reader of X other than normalize()'s fused launch
static void materialise_gather(Engine::Impl &m, EngineStats &st)
{
    if (!m.gsel) return;
    const int sp = m.span_begin(5);
    launch_gather_cols(m.gsrc, m.gsrc_ld, m.n, m.gsel, m.p, m.X, m.ldx, m.st);
    m.span_end(sp);
    st.kernel_launches += 1;
    m.drop_gather_source();
}

std::vector<int> Engine::screen(int size, const std::vector<int> &always_select)
{
    screen_enqueue(size, always_select);
    return screen_result();
}

// The kept columns of the last screen_enqueue(), ascending (waits for the device only here).
std::vector<int> Engine::screen_result()
{
    Impl &m = *d_;
    if (!m.h_sel) throw EngineError{"screen_result: no screening has run"};
    if (m.sel_pending) {
        CUDA_CHECK(cudaStreamSynchronize(m.st));
        m.sel_pending = false;
        stats_.n_boundary_ties += *m.h_sel_tie;
    }
    return std::vector<int>(m.h_sel, m.h_sel + m.sel_count);
}

void Engine::screen_enqueue(int size, const std::vector<int> &always_select)
{
    Impl &m = *d_;
    if (size < 1 || size > p_model()) throw EngineError{"screening_size must be in [1, p]"};
    materialise_gather(m, stats_);  // a second screening reads the first one's kept columns
    const long long ldn = (size + 1) & ~1LL;
    double *Xn = dalloc<double>(m.st, (size_t)m.n * ldn);
    if (ldn != size || m.csc) CUDA_CHECK(cudaMemsetAsync(Xn, 0, (size_t)m.n * ldn * 8, m.st));
    m.h_sel = m.ctx->rb.alloc<int>((size_t)size);
    m.h_sel_tie = m.ctx->rb.alloc<int>(1);
    *m.h_sel_tie = 0;
    m.sel_count = size;
    if (!sharded_) {
        const int *d_sel = screen_select(m, stats_, family_, size, always_select, nullptr, nullptr, /*to_pinned=*/true);
        // X <- X[:, sel]  (screening.cpp:83-88).  A dense design's gather waits for normalize(), which fuses it into its
        // one launch, or for the first other reader of X (materialise_gather).
        if (m.csc) {
            const int spk = m.span_begin(5);
            launch_csc_densify(m.cp, m.ri, m.cv, d_sel, size, Xn, ldn, m.st);
            m.span_end(spk);
            stats_.kernel_launches += 1;
        } else {
            m.gsel = d_sel;
            m.gsrc = m.X;
            m.gsrc_ld = m.ldx;
            m.gsrc_owned = m.x_owned;
            m.x_owned = false;  // ownership of the raw design moved to the pending gather
        }
        m.sel_pending = true;  // the index list and the tie flag are on their way to the pinned block
    } else {
        // Column-sharded screening (SURVEY 8e axis B): marginal utilities of the local columns, exact local top-`size`,
        // NCCL all-gather of the (utility, global index) candidates, identical merge on every rank, then every rank
        // contributes the kept columns it owns and an all-reduce(sum) over NVLink hands the n x size screened design
        // to everybody (adding zeros is exact, so all ranks hold bit-identical copies).
        const NcclApi &api = nccl_api();
        const int kloc = std::min<long long>(size, m.p);
        std::vector<int> alw_local;
        for (int j : always_select)
            if (j >= col_lo_ && j < col_lo_ + m.p) alw_local.push_back((int)(j - col_lo_));
        const int *d_sel = screen_select(m, stats_, family_, kloc, alw_local, nullptr, nullptr, /*to_pinned=*/false);
        Cand *cs = dalloc<Cand>(m.st, size), *cr = dalloc<Cand>(m.st, (size_t)m.world * size);
        const long long n_in = (long long)m.world * size;
        double *mv = dalloc<double>(m.st, n_in);
        int *mi = dalloc<int>(m.st, n_in), *d_gsel = dalloc<int>(m.st, size), *d_tie = dalloc<int>(m.st, 1);
        const long long cstride = std::max<long long>(2LL * size + 16, (n_in / 8192 + 2) * std::min(size, TOPK_LMAX));
        double *ck0 = dalloc<double>(m.st, cstride), *ck1 = dalloc<double>(m.st, cstride);
        int *ci0 = dalloc<int>(m.st, cstride), *ci1 = dalloc<int>(m.st, cstride);
        const int spx = m.span_begin(5);
        launch_pack_candidates(m.d.bd, m.d.pstride, d_sel, size, kloc, size, col_lo_, 1, cs, size, nullptr, m.st);
        NCCL_CHECK(api.AllGather(cs, cr, (size_t)size * sizeof(Cand), ncclChar, m.comm, m.st));
        launch_unpack_candidates(cr, m.world, 1, size, size, mv, mi, n_in, nullptr, m.st);
        launch_topk(mv, n_in, (int)n_in, size, 1, d_gsel, size, d_tie, ck0, ci0, ck1, ci1, cstride, m.st, nullptr, mi);
        launch_gather_owned_cols(m.X, m.ldx, m.n, m.p, col_lo_, d_gsel, size, Xn, ldn, m.st);
        NCCL_CHECK(api.AllReduce(Xn, Xn, (size_t)m.n * ldn, ncclDouble, ncclSum, m.comm, m.st));
        m.span_end(spx);
        CUDA_CHECK(cudaMemcpyAsync(m.h_sel, d_gsel, (size_t)size * 4, cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaMemcpyAsync(m.h_sel_tie, d_tie, 4, cudaMemcpyDeviceToHost, m.st));
        m.sel_pending = true;
        stats_.kernel_launches += 4;
        dfree(m.st, cs); dfree(m.st, cr); dfree(m.st, mv); dfree(m.st, mi); dfree(m.st, d_gsel);
        dfree(m.st, d_tie); dfree(m.st, ck0); dfree(m.st, ck1); dfree(m.st, ci0); dfree(m.st, ci1);
        // from here on every rank holds the whole (screened) design: the path runs replicated
        sharded_ = false;
        col_lo_ = 0;
    }
    if (m.x_owned) dfree(m.st, m.X);  // stream-ordered: the gather above has the old design until it is done
    m.free_csc();
    m.x_owned = true;
    m.X = Xn;
    m.ldx = ldn;
    m.p = size;
    p_ = size;
    m.free_sweep_buffers();
    m.d.sharded = 0;
    m.d.col_lo = 0;
    h_xmean_.clear();
    h_xnorm_.clear();
}

// Column-sharded screening (SURVEY 8e axis B): the local top-`size` candidates (utility, local column index) of this
// rank's columns; X is left untouched.
void Engine::screen_local(int size, const std::vector<int> &always_select, std::vector<double> &vals,
                          std::vector<int> &idx)
{
    Impl &m = *d_;
    size = std::min(size, m.p);
    materialise_gather(m, stats_);
    screen_select(m, stats_, family_, size, always_select, &vals, &idx, /*to_pinned=*/false);
    m.free_sweep_buffers();
}

// dst[i*ld + pos[q]] = X[i][cols[q]] for q < m  (dst is a device buffer shared by all ranks' selections)
void Engine::gather_columns(const int *cols, const int *pos, int mcols, double *dst_dev, long long ld)
{
    Impl &m = *d_;
    if (m.csc) throw EngineError{"gather_columns: the design is sparse"};
    if (mcols <= 0) return;
    materialise_gather(m, stats_);
    int *d_cols = dalloc<int>(m.st, mcols), *d_pos = dalloc<int>(m.st, mcols);
    CUDA_CHECK(cudaMemcpyAsync(d_cols, cols, (size_t)mcols * 4, cudaMemcpyHostToDevice, m.st));
    CUDA_CHECK(cudaMemcpyAsync(d_pos, pos, (size_t)mcols * 4, cudaMemcpyHostToDevice, m.st));
    launch_gather_cols_pos(m.X, m.ldx, m.n, d_cols, d_pos, mcols, dst_dev, ld, m.st);
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    stats_.kernel_launches += 1;
    dfree(m.st, d_cols);
    dfree(m.st, d_pos);
}

// Marginal utilities (screening.cpp:26-61) on RAW x -> m.d.bd, always_select pinned, exact top-`size` (ascending) into a
// device list that is returned (arena memory, alive until the next config_sweep).  Host copies:
//   sel_out / vals_out   synchronous (screen_local);
//   to_pinned            the list and the boundary-tie flag go to m.h_sel / m.h_sel_tie asynchronously.
static int *screen_select(Engine::Impl &m, EngineStats &stats_, int family_, int size,
                          const std::vector<int> &always_select, std::vector<double> *vals_out,
                          std::vector<int> *sel_out, bool to_pinned)
{
    m.config_sweep(1);
    DevArena &ar = m.ctx->ar;
    BatchDesc b{};
    b.nch = 1;
    b.chain[0] = 0;
    if (m.csc) {
        // the same utilities over the stored entries of a sparse design; algorithmic bytes: the three CSC arrays and the
        // n-vectors the kernel reads (y; y and w for the GLM families)
        const int sp = m.span_begin(0);
        if (family_ == FAM_LM) launch_screen_csc_lm(m.cp, m.ri, m.cv, m.p, m.nnz, m.y, m.d.bd, m.st);
        else launch_screen_glm_csc(m.cp, m.ri, m.cv, m.n, m.p, m.y, m.w, family_, m.d.bd, m.st);
        m.span_end(sp);
        stats_.big_sweep_bytes += 12.0 * (double)m.nnz + 8.0 * ((double)m.p + 1) + (family_ == FAM_LM ? 8.0 : 16.0) * m.n;
        stats_.kernel_launches += 1;
    } else if (family_ == FAM_LM) {
        // one-column least squares on RAW x (screening.cpp:46): (x_j.y / x_j.x_j)^2
        std::vector<double> ones(m.n, 1.0);
        m.put_vec(m.d.G, 0, m.hy);
        m.put_vec(m.d.W, 0, ones);
        int sp = m.span_begin(0);
        launch_dual_sweep(m.d, MODE_DH, m.st);
        m.span_end(sp);
        sp = m.span_begin(2);
        launch_finish(m.d, MODE_DH, EPI_SCREEN_LM, b, nullptr, m.st);
        m.span_end(sp);
        stats_.big_sweep_bytes += 8.0 * m.n * m.p;
        stats_.n_sweeps++;
        stats_.kernel_launches += 2;
    } else {
        const int sp = m.span_begin(0);
        launch_screen_glm(m.X, m.ldx, m.n, m.p, m.y, m.w, family_, m.d.bd, m.st);
        m.span_end(sp);
        stats_.big_sweep_bytes += 8.0 * m.n * m.p;  // algorithmic: one pass (the marginal fits re-read the column from L2)
        stats_.kernel_launches += 1;
    }
    if (!always_select.empty()) {
        int *h_alw = nullptr;
        int *d_alw = m.ctx->mir.alloc<int>(always_select.size(), &h_alw);
        std::copy(always_select.begin(), always_select.end(), h_alw);
        m.ctx->mir.flush(m.st);
        launch_pin(m.d, m.d.bd, m.d.pstride, 1, d_alw, (int)always_select.size(), m.st);
    }
    int *d_sel = ar.alloc<int>((size_t)size);
    const long long cstride = std::max<long long>(2LL * size + 16, ((long long)m.p / 8192 + 2) * std::min(size, TOPK_LMAX));
    double *ck0 = ar.alloc<double>((size_t)cstride), *ck1 = ar.alloc<double>((size_t)cstride);
    int *ci0 = ar.alloc<int>((size_t)cstride), *ci1 = ar.alloc<int>((size_t)cstride);
    int *d_tie = ar.alloc<int>(1);
    void *scratch = ar.alloc<unsigned char>(screen_select_scratch_bytes(m.p));
    const int spk = m.span_begin(3);
    stats_.kernel_launches += launch_screen_select(m.d.bd, m.p, size, d_sel, d_tie, scratch, ck0, ci0, ck1, ci1, cstride, m.st);
    m.span_end(spk);
    if (m.tie_exact && !m.d.sharded) {
        int tie = 0;
        CUDA_CHECK(cudaMemcpyAsync(&tie, d_tie, 4, cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaStreamSynchronize(m.st));
        if (tie) {  // the reference's own resolution of the tie (max_k on the utilities, screening.cpp:66)
            std::vector<double> all((size_t)m.p);
            std::vector<int> hs((size_t)size);
            CUDA_CHECK(cudaMemcpyAsync(all.data(), m.d.bd, (size_t)m.p * 8, cudaMemcpyDeviceToHost, m.st));
            CUDA_CHECK(cudaStreamSynchronize(m.st));
            host_max_k(all.data(), m.p, size, hs.data());
            CUDA_CHECK(cudaMemcpyAsync(d_sel, hs.data(), (size_t)size * 4, cudaMemcpyHostToDevice, m.st));
            CUDA_CHECK(cudaStreamSynchronize(m.st));
        }
    }
    if (to_pinned) {
        CUDA_CHECK(cudaMemcpyAsync(m.h_sel, d_sel, (size_t)size * 4, cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaMemcpyAsync(m.h_sel_tie, d_tie, 4, cudaMemcpyDeviceToHost, m.st));
    }
    if (sel_out) {
        int tie = 0;
        sel_out->resize(size);
        CUDA_CHECK(cudaMemcpyAsync(sel_out->data(), d_sel, (size_t)size * 4, cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaMemcpyAsync(&tie, d_tie, 4, cudaMemcpyDeviceToHost, m.st));  // a LOCAL boundary tie only matters
        CUDA_CHECK(cudaStreamSynchronize(m.st));                                    // when the local list is the result
        stats_.n_boundary_ties += tie;
        if (vals_out) {
            std::vector<double> all((size_t)m.p);
            CUDA_CHECK(cudaMemcpyAsync(all.data(), m.d.bd, (size_t)m.p * 8, cudaMemcpyDeviceToHost, m.st));
            CUDA_CHECK(cudaStreamSynchronize(m.st));
            vals_out->resize(size);
            for (int q = 0; q < size; q++) (*vals_out)[q] = all[(size_t)(*sel_out)[q]];
        }
    }
    return d_sel;
}

void Engine::copy_design(double *host_out)
{
    Impl &m = *d_;
    if (m.csc && !m.csc_norm) throw EngineError{"copy_design: the design is sparse (normalise it first)"};
    if (m.csc) {  // the normalised design, expanded on the device
        if (!m.have_sweep) m.config_sweep(1);
        double *buf = dalloc<double>(m.st, (size_t)m.n * m.p);
        launch_csc_expand(m.d, buf, m.p, m.st);
        CUDA_CHECK(cudaMemcpyAsync(host_out, buf, (size_t)m.n * m.p * 8, cudaMemcpyDeviceToHost, m.st));
        dfree(m.st, buf);
        CUDA_CHECK(cudaStreamSynchronize(m.st));
        stats_.kernel_launches += 1;
        return;
    }
    if (!m.X) throw EngineError{"copy_design: no design is loaded"};
    materialise_gather(m, stats_);
    CUDA_CHECK(cudaMemcpy2DAsync(host_out, (size_t)m.p * 8, m.X, (size_t)m.ldx * 8, (size_t)m.p * 8, m.n,
                                 cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaStreamSynchronize(m.st));
}

// Data ctor (Data.h:41-68) + normalize.cpp + add_weight (Data.h:70-77, bess.cpp:97)
void Engine::normalize(int data_type, bool is_normal)
{
    Impl &m = *d_;
    if (m.csc) {
        normalize_csc(data_type, is_normal);
        return;
    }
    const int n = m.n, p = m.p;
    // ---- a design that fits L2 (after screening: config 5's 40 MB): the whole normalisation is ONE launch, which also
    // gathers the kept columns of a pending screening when their n x 8 slabs fit shared memory
    static const bool one_launch = [] {
        const char *e = std::getenv("BESS_B200_NORM_FUSED");
        return !(e && e[0] == '0');
    }();
    const bool resident = one_launch && is_normal && !sharded_ && (size_t)n * m.ldx * 8 <= ((size_t)64 << 20);
    const bool fuse_gather = resident && m.gsel && n <= NR_SLAB_ROWS;
    if (!fuse_gather) materialise_gather(m, stats_);
    if (!m.x_owned) {  // normalisation is in place: take a private copy of a borrowed design
        double *Xc = dalloc<double>(m.st, (size_t)n * m.ldx);
        CUDA_CHECK(cudaMemcpyAsync(Xc, m.X, (size_t)n * m.ldx * 8, cudaMemcpyDeviceToDevice, m.st));
        m.X = Xc;
        m.x_owned = true;
    }
    DevArena &ar = m.ctx->ar;
    m.stats_have_mean = false;
    m.stats_pending = false;
    if (resident) {
        const int sp = m.span_begin(6);
        m.h_mean = m.ctx->rb.alloc<double>((size_t)p);
        m.h_norm = m.ctx->rb.alloc<double>((size_t)p);
        const bool centre = data_type == 1 || data_type == 2;
        std::vector<double> g(n), rm(n);
        for (int i = 0; i < n; i++) g[i] = m.hw[i] / (double)n;  // meanx_j = w.x_j / n (normalize.cpp:25-28, 52-55)
        if (data_type == 1) {
            double s = 0.0;
            for (int i = 0; i < n; i++) s += m.hy[i] * m.hw[i];  // normalize.cpp:29
            y_mean_ = s / (double)n;
            for (int i = 0; i < n; i++) m.hy[i] -= y_mean_;
        }
        double *d_g = centre ? m.stage_vec(g.data(), (size_t)n, (size_t)n) : nullptr;
        double *d_w = m.stage_vec(m.hw.data(), (size_t)n, (size_t)n);
        double *d_rm = nullptr;
        if (family_ == FAM_LM) {  // add_weight: rows scaled by sqrt(w) (Data.h:70-77)
            for (int i = 0; i < n; i++) {
                rm[i] = std::sqrt(m.hw[i]);
                m.hy[i] *= rm[i];
            }
            d_rm = m.stage_vec(rm.data(), (size_t)n, (size_t)n);
        }
        m.y = m.stage_vec(m.hy.data(), (size_t)n, (size_t)m.npad);  // the response as the fits see it
        m.ctx->mir.flush(m.st);
        double *d_mean = ar.alloc<double>((size_t)p + 2), *d_norm = ar.alloc<double>((size_t)p + 2);
        if (fuse_gather) {
            launch_gather_normalize(m.gsrc, m.gsrc_ld, m.gsel, m.X, m.ldx, n, p, d_g, d_w, d_rm, std::sqrt((double)n), d_mean,
                                    d_norm, m.st);
            m.drop_gather_source();  // stream-ordered: an owned raw design lives until the launch above is done
            stats_.norm_bytes += 16.0 * n * p;  // one read of the kept elements (each its own sector) and one write
        } else {
            launch_normalize_resident(m.X, m.ldx, n, p, d_g, d_w, d_rm, std::sqrt((double)n), d_mean, d_norm, m.st);
            stats_.norm_bytes += 32.0 * n * p;  // three reads and one write of X
        }
        if (centre) CUDA_CHECK(cudaMemcpyAsync(m.h_mean, d_mean, (size_t)p * 8, cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaMemcpyAsync(m.h_norm, d_norm, (size_t)p * 8, cudaMemcpyDeviceToHost, m.st));
        m.stats_have_mean = centre;
        m.stats_pending = true;
        m.span_end(sp);
        stats_.kernel_launches += 1;
        h_xmean_.clear();
        h_xnorm_.clear();
        return;
    }
    m.config_sweep(1);
    BatchDesc b{};
    b.nch = 1;
    b.chain[0] = 0;
    double *d_mul = nullptr, *d_rowmul = nullptr;
    const int sp_all = m.span_begin(6);
    // No host round trip in here: the column statistics stay on the device (the scale factors are derived there) and
    // travel to pinned memory for the de-normalisation at the end of the call (ensure_stats).
    if (is_normal) {
        m.h_mean = m.ctx->rb.alloc<double>((size_t)p);
        m.h_norm = m.ctx->rb.alloc<double>((size_t)p);
        if (data_type == 1 || data_type == 2) {
            // meanx_j = w.x_j / n  (normalize.cpp:25-28, 52-55)
            std::vector<double> g(n);
            for (int i = 0; i < n; i++) g[i] = m.hw[i] / (double)n;
            m.put_vec(m.d.G, 0, g);
            launch_dual_sweep(m.d, MODE_D, m.st);
            launch_finish(m.d, MODE_D, EPI_RAW, b, m.raw, m.st);
            double *d_mean = ar.alloc<double>((size_t)m.d.pstride);
            CUDA_CHECK(cudaMemcpyAsync(d_mean, m.raw, (size_t)p * 8, cudaMemcpyDeviceToDevice, m.st));
            CUDA_CHECK(cudaMemcpyAsync(m.h_mean, m.raw, (size_t)p * 8, cudaMemcpyDeviceToHost, m.st));
            launch_center_scale(m.X, m.ldx, n, p, d_mean, nullptr, nullptr, m.st);
            m.stats_have_mean = true;
            stats_.kernel_launches += 3;
        }
        if (data_type == 1) {
            double s = 0.0;
            for (int i = 0; i < n; i++) s += m.hy[i] * m.hw[i];  // normalize.cpp:29
            y_mean_ = s / (double)n;
            for (int i = 0; i < n; i++) m.hy[i] -= y_mean_;
        }
        // normx_j = sqrt(w.(x_j)^2) on the centred column (normalize.cpp:36-41)
        std::vector<double> zero(n, 0.0);
        m.put_vec(m.d.G, 0, zero);
        m.put_vec(m.d.W, 0, m.hw);
        launch_dual_sweep(m.d, MODE_DH, m.st);
        launch_finish(m.d, MODE_DH, EPI_RAW, b, m.raw, m.st);
        // x_j <- sqrt(n) * x_j / normx_j  (normalize.cpp:42-45): norms and factors from the sums, on the device
        d_mul = ar.alloc<double>((size_t)m.d.pstride);
        double *d_norm = ar.alloc<double>((size_t)m.d.pstride);
        launch_norm_factors(m.raw + (size_t)m.d.FS * m.d.pstride, p, std::sqrt((double)n), d_norm, d_mul, m.st);
        CUDA_CHECK(cudaMemcpyAsync(m.h_norm, d_norm, (size_t)p * 8, cudaMemcpyDeviceToHost, m.st));
        m.stats_pending = true;
        stats_.kernel_launches += 3;
        stats_.n_sweeps += 2;
    }
    if (family_ == FAM_LM) {
        // add_weight: rows scaled by sqrt(w) (Data.h:70-77)
        std::vector<double> rm(n);
        for (int i = 0; i < n; i++) {
            rm[i] = std::sqrt(m.hw[i]);
            m.hy[i] *= rm[i];
        }
        d_rowmul = m.stage_vec(rm.data(), (size_t)n, (size_t)n);
    }
    m.y = m.stage_vec(m.hy.data(), (size_t)n, (size_t)m.npad);  // the response as the fits see it
    m.ctx->mir.flush(m.st);
    if (d_mul || d_rowmul) {
        launch_center_scale(m.X, m.ldx, n, p, nullptr, d_mul, d_rowmul, m.st);
        stats_.kernel_launches += 1;
    }
    m.span_end(sp_all);
    // passes over X: [mean sweep 8np + centre 16np] (data_type 1,2) + norm sweep 8np + scale 16np
    if (is_normal) stats_.norm_bytes += (data_type == 3 ? 24.0 : 48.0) * n * p;
    else if (family_ == FAM_LM) stats_.norm_bytes += 16.0 * n * p;
    m.free_sweep_buffers();
    if (sharded_) {
        // column statistics are shard-local; de-normalisation (path.cpp:76-110) needs those of the selected columns,
        // whoever owns them: all-gather both vectors once (2 * p_total doubles)
        ensure_stats();
        const NcclApi &api = nccl_api();
        long long lo0, hi0;
        shard_range(p_total_, world_, 0, &lo0, &hi0);
        const size_t pmax = (size_t)(hi0 - lo0);
        std::vector<double> send(2 * pmax, 0.0), recv((size_t)world_ * 2 * pmax);
        std::copy(h_xmean_.begin(), h_xmean_.end(), send.begin());
        std::copy(h_xnorm_.begin(), h_xnorm_.end(), send.begin() + pmax);
        double *ds = dalloc<double>(m.st, 2 * pmax), *dr = dalloc<double>(m.st, (size_t)world_ * 2 * pmax);
        CUDA_CHECK(cudaMemcpyAsync(ds, send.data(), send.size() * 8, cudaMemcpyHostToDevice, m.st));
        NCCL_CHECK(api.AllGather(ds, dr, 2 * pmax, ncclDouble, m.comm, m.st));
        CUDA_CHECK(cudaMemcpyAsync(recv.data(), dr, recv.size() * 8, cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaStreamSynchronize(m.st));
        dfree(m.st, ds); dfree(m.st, dr);
        g_xmean_.assign((size_t)p_total_, 0.0);
        g_xnorm_.assign((size_t)p_total_, 0.0);
        for (int q = 0; q < world_; q++) {
            long long lo, hi;
            shard_range(p_total_, world_, q, &lo, &hi);
            const double *blk = recv.data() + (size_t)q * 2 * pmax;
            std::copy(blk, blk + (hi - lo), g_xmean_.begin() + lo);
            std::copy(blk + pmax, blk + pmax + (hi - lo), g_xnorm_.begin() + lo);
        }
    }
}

// normalize() of a sparse design: the arrays stay as they are and only the column statistics and the row factors are
// computed (normalize.cpp:20-86, add_weight of Data.h:70-77); the design the path sees is the implicit
// x~_ij = ((x_ij - mean_j) * mul_j) * rowmul_i, swept on its non-zeros.  Equal to the dense statistics up to summation order.
void Engine::normalize_csc(int data_type, bool is_normal)
{
    Impl &m = *d_;
    if (m.csc_norm) throw EngineError{"normalize: the sparse design is already normalised"};
    const int n = m.n, p = m.p;
    const int sp = m.span_begin(6);
    const bool centre = is_normal && (data_type == 1 || data_type == 2);
    m.free_sweep_buffers();
    m.cmean = dalloc<double>(m.st, (size_t)p);
    m.cmul = dalloc<double>(m.st, (size_t)p);
    m.stats_have_mean = false;
    m.stats_pending = false;
    if (is_normal) {
        std::vector<double> g(n);
        double sumw = 0.0;
        for (int i = 0; i < n; i++) {
            g[i] = m.hw[i] / (double)n;  // meanx_j = w.x_j / n (normalize.cpp:25-28, 52-55)
            sumw += m.hw[i];
        }
        double *d_g = centre ? m.stage_vec(g.data(), (size_t)n, (size_t)n) : nullptr;
        m.ctx->mir.flush(m.st);
        m.h_mean = m.ctx->rb.alloc<double>((size_t)p);
        m.h_norm = m.ctx->rb.alloc<double>((size_t)p);
        double *d_norm = m.ctx->ar.alloc<double>((size_t)p);
        launch_csc_stats(m.cp, m.ri, m.cv, p, d_g, m.w, sumw, std::sqrt((double)n), m.cmean, d_norm, m.cmul, m.st);
        if (centre) CUDA_CHECK(cudaMemcpyAsync(m.h_mean, m.cmean, (size_t)p * 8, cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaMemcpyAsync(m.h_norm, d_norm, (size_t)p * 8, cudaMemcpyDeviceToHost, m.st));
        m.stats_have_mean = centre;
        m.stats_pending = true;
        stats_.kernel_launches += 1;
        stats_.norm_bytes += 2.0 * (12.0 * (double)m.nnz + 8.0 * ((double)p + 1)) + 16.0 * n + 24.0 * p;
    } else {
        std::vector<double> zero((size_t)p, 0.0), one((size_t)p, 1.0);
        CUDA_CHECK(cudaMemcpyAsync(m.cmean, zero.data(), (size_t)p * 8, cudaMemcpyHostToDevice, m.st));
        CUDA_CHECK(cudaMemcpyAsync(m.cmul, one.data(), (size_t)p * 8, cudaMemcpyHostToDevice, m.st));
        CUDA_CHECK(cudaStreamSynchronize(m.st));  // the host vectors die here
    }
    if (data_type == 1 && is_normal) {
        double s = 0.0;
        for (int i = 0; i < n; i++) s += m.hy[i] * m.hw[i];  // normalize.cpp:29
        y_mean_ = s / (double)n;
        for (int i = 0; i < n; i++) m.hy[i] -= y_mean_;
    }
    if (family_ == FAM_LM) {  // add_weight: rows scaled by sqrt(w) (Data.h:70-77)
        std::vector<double> rm(n);
        for (int i = 0; i < n; i++) {
            rm[i] = std::sqrt(m.hw[i]);
            m.hy[i] *= rm[i];
        }
        m.crm = dalloc<double>(m.st, (size_t)n);
        CUDA_CHECK(cudaMemcpyAsync(m.crm, rm.data(), (size_t)n * 8, cudaMemcpyHostToDevice, m.st));
        CUDA_CHECK(cudaStreamSynchronize(m.st));
    }
    m.y = m.stage_vec(m.hy.data(), (size_t)n, (size_t)m.npad);  // the response as the fits see it
    m.ctx->mir.flush(m.st);
    m.csc_norm = true;
    m.span_end(sp);
    h_xmean_.clear();
    h_xnorm_.clear();
}

bool Engine::sparse_sweeps() const { return d_->csc_norm; }
size_t Engine::device_total_bytes() const
{
    size_t free_b = 0, total_b = 0;
    CUDA_CHECK(cudaMemGetInfo(&free_b, &total_b));
    return total_b;
}

// The column statistics of the last normalize() on the host (h_xmean_, h_xnorm_): waits for the device only here.
void Engine::ensure_stats() const
{
    Impl &m = *d_;
    Engine *self = const_cast<Engine *>(this);
    if ((int)h_xmean_.size() != m.p) {
        self->h_xmean_.assign((size_t)m.p, 0.0);
        self->h_xnorm_.assign((size_t)m.p, 0.0);
    }
    if (!m.stats_pending) return;
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    if (m.stats_have_mean) std::copy(m.h_mean, m.h_mean + m.p, self->h_xmean_.begin());
    std::copy(m.h_norm, m.h_norm + m.p, self->h_xnorm_.begin());
    m.stats_pending = false;
}

void Engine::set_groups(const std::vector<int> &g_index)
{
    Impl &m = *d_;
    if (sharded_) throw EngineError{"group selection is not available in column-sharded mode"};
    if (m.csc) throw EngineError{"group selection needs a dense design (densify or screen the sparse one)"};
    const int p = m.p, N = (int)g_index.size();
    if (N < 1 || N > p) throw EngineError{"g_index must hold between 1 and p group starts"};
    if (g_index[0] != 0) throw EngineError{"g_index must start at column 0"};
    g_index_ = g_index;
    g_size_.assign((size_t)N, 0);
    for (int g = 0; g < N; g++) {
        const int next = g + 1 < N ? g_index[(size_t)g + 1] : p;  // Data.h:53-61
        if (next <= g_index[(size_t)g]) throw EngineError{"g_index must be strictly ascending"};
        g_size_[(size_t)g] = next - g_index[(size_t)g];
        if (g_size_[(size_t)g] > GWIDE) throw EngineError{"groups of more than 64 variables are not supported"};
    }
    n_groups_ = N;
    dfree(m.st, m.gidx);
    dfree(m.st, m.gsz);
    m.gidx = dalloc<int>(m.st, (size_t)N);
    m.gsz = dalloc<int>(m.st, (size_t)N);
    CUDA_CHECK(cudaMemcpyAsync(m.gidx, g_index_.data(), (size_t)N * 4, cudaMemcpyHostToDevice, m.st));
    CUDA_CHECK(cudaMemcpyAsync(m.gsz, g_size_.data(), (size_t)N * 4, cudaMemcpyHostToDevice, m.st));
    // narrow groups by width class, for the chain-batched sacrifice kernels (one instantiation per class)
    std::vector<int> order;
    const int bound[3] = {2, 4, GMAX};
    for (int k = 0; k < 3; k++) {
        m.gcls_off[k] = (int)order.size();
        for (int g = 0; g < N; g++)
            if (g_size_[(size_t)g] <= bound[k] && (k == 0 || g_size_[(size_t)g] > bound[k - 1])) order.push_back(g);
    }
    m.gcls_off[3] = (int)order.size();
    dfree(m.st, m.glist);
    m.glist = dalloc<int>(m.st, (size_t)std::max<size_t>(order.size(), 1));
    if (!order.empty()) CUDA_CHECK(cudaMemcpyAsync(m.glist, order.data(), order.size() * 4, cudaMemcpyHostToDevice, m.st));
    CUDA_CHECK(cudaStreamSynchronize(m.st));
}

void Engine::setup_chains(int K, const int *fold_of_row, int kcap, int max_iter, bool warm_start,
                          const std::vector<int> &always_select)
{
    Impl &m = *d_;
    const int n = m.n, p = m.p;
    if (K < 0 || K > MAXC - 1) throw EngineError{"K (nfolds) must be in [0, 31]"};
    if (m.csc && !m.csc_norm) throw EngineError{"setup_chains: a sparse design must be normalised (or densified) first"};
    if (max_iter < 1 || max_iter > MAX_ITER_CAP) throw EngineError{"max_iter must be in [1, 100000]"};
    const bool grp = grouped();
    if (kcap < 1 || kcap > (grp ? n_groups_ : p_model())) throw EngineError{"support size must be in [1, p]"};
    m.Tmax = kcap;
    if (grp) {
        // sparsity levels count groups; the column capacity of a support is the size of the kcap widest groups
        std::vector<int> sz = g_size_;
        std::sort(sz.begin(), sz.end(), [](int a, int b) { return a > b; });
        int cols = 0;
        for (int g = 0; g < kcap; g++) cols += sz[(size_t)g];
        kcap = cols;
        for (int j : always_select)
            if (j < 0 || j >= n_groups_) throw EngineError{"always_select must hold group numbers in [0, number of groups)"};
    }
    m.free_chain_buffers();
    m.K = K;
    m.nchains = 1 + K;
    const int C = m.nchains;
    materialise_gather(m, stats_);
    m.config_sweep(pick_fs(C));
    DevArena &ar = m.ctx->ar;
    MirrorArena &mir = m.ctx->mir;
    Dev &d = m.d;
    d.kcap = kcap;
    d.ldA = (kcap + 2 + 1) & ~1;
    d.fit_smem_doubles = fit_smem_doubles(d.ldA, kcap);
    d.max_iter = max_iter;
    d.warm = warm_start ? 1 : 0;
    d.sharded = sharded_ ? 1 : 0;
    d.col_lo = sharded_ ? (int)col_lo_ : 0;
    d.ax_ext = (sharded_ || m.csc_norm) ? 1 : 0;
    d.nmat = family_ == FAM_COX ? 2 : 1;
    d.grouped = grp ? 1 : 0;
    d.N = n_groups_;
    d.gmax = grp ? *std::max_element(g_size_.begin(), g_size_.end()) : 1;
    d.gidx = m.gidx;
    d.gsz = m.gsz;
    d.glist = m.glist;
    for (int k = 0; k < 4; k++) d.gcls_off[k] = m.gcls_off[k];

    // ---- host tables, written straight into the pinned half of the mirror arena: ONE copy moves them all.
    // Row lists (Metric.h:80-103: train masks are the sorted complement of each fold), compacted response / weights.
    int *h_rows, *h_ntrain, *h_testrows, *h_ntest;
    double *h_ytr, *h_wtr, *h_lfact;
    d.rows = mir.alloc<int>((size_t)MAXC * n, &h_rows);
    d.ntrain = mir.alloc<int>(MAXC, &h_ntrain);
    m.testrows = mir.alloc<int>((size_t)MAXC * n, &h_testrows);
    m.ntest = mir.alloc<int>(MAXC, &h_ntest);
    d.ytr = mir.alloc<double>((size_t)MAXC * n, &h_ytr);
    d.wtr = mir.alloc<double>((size_t)MAXC * n, &h_wtr);
    m.lfact = mir.alloc<double>((size_t)n, &h_lfact);
    std::memset(h_ntrain, 0, MAXC * sizeof(int));
    std::memset(h_ntest, 0, MAXC * sizeof(int));
    for (int i = 0; i < n; i++) h_rows[i] = i;
    h_ntrain[0] = n;
    for (int k = 0; k < K; k++) {
        int a = 0, t = 0;
        for (int i = 0; i < n; i++) {
            if (fold_of_row[i] < 0 || fold_of_row[i] >= K) throw EngineError{"fold_of_row out of range"};
            if (fold_of_row[i] == k) h_testrows[(size_t)k * n + t++] = i;
            else h_rows[(size_t)(1 + k) * n + a++] = i;
        }
        h_ntrain[1 + k] = a;
        h_ntest[k] = t;
        if (a < 2) throw EngineError{"a CV fold leaves fewer than 2 training rows"};
    }
    for (int c = 0; c < C; c++)
        for (int r = 0; r < h_ntrain[c]; r++) {
            h_ytr[(size_t)c * n + r] = m.hy[h_rows[(size_t)c * n + r]];
            h_wtr[(size_t)c * n + r] = m.hw[h_rows[(size_t)c * n + r]];
        }
    // poisson: sum_{j<=y} log j (poisson.cpp:29-44), same summation order as the reference
    std::memset(h_lfact, 0, (size_t)n * 8);
    if (family_ == FAM_POISSON) {
        double ymax = 0.0;
        for (int i = 0; i < n; i++) ymax = std::max(ymax, m.hy[i]);
        if (ymax <= 5.0e7) {
            std::vector<double> cum((size_t)ymax + 2, 0.0);
            for (size_t j = 1; j < cum.size(); j++) cum[j] = cum[j - 1] + std::log((double)j);
            for (int i = 0; i < n; i++) {
                const double yi = m.hy[i];
                h_lfact[i] = (yi == 1.0 || yi < 1.0) ? 0.0 : cum[(size_t)std::floor(yi)];
            }
        } else {
            for (int i = 0; i < n; i++) h_lfact[i] = m.hy[i] < 1.0 ? 0.0 : std::lgamma(std::floor(m.hy[i]) + 1.0);
        }
    }
    std::vector<int> alw_local;  // pins are applied to the local sacrifice vector
    for (int j : always_select)
        if (!sharded_) alw_local.push_back(j);
        else if (j >= col_lo_ && j < col_lo_ + p) alw_local.push_back((int)(j - col_lo_));
    m.n_always = (int)alw_local.size();
    if (m.n_always) {
        int *h_alw;
        m.always = mir.alloc<int>((size_t)m.n_always, &h_alw);
        std::copy(alw_local.begin(), alw_local.end(), h_alw);
    }
    // the train-row indicators of every chain as a [npad][FS] sweep vector: x_j.x_j over each chain's train rows in one
    // pass (utilities.cpp:153-165, Metric.h:108-129; gaussian only).  With groups the blocks X_g^T X_g / n are
    // accumulated by group_sacrifice_kernel itself: W = 1/n_train on the chain's train rows, for the life of the chains.
    double *d_ind = nullptr;
    const size_t vsz = (size_t)m.npad * d.FS;
    if (family_ == FAM_LM) {
        double *h_ind;
        d_ind = mir.alloc<double>(vsz, &h_ind);
        std::memset(h_ind, 0, vsz * 8);
        for (int c = 0; c < C; c++) {
            const double v = grp ? 1.0 / (double)h_ntrain[c] : 1.0;
            for (int r = 0; r < h_ntrain[c]; r++) {
                const int i = h_rows[(size_t)c * n + r];
                // the sparse sweep sees the raw column: the row factors of add_weight enter as rowmul^2
                h_ind[(size_t)i * d.FS + c] = m.csc_norm ? std::sqrt(m.hw[i]) * std::sqrt(m.hw[i]) : v;
            }
        }
    }
    // resident path (lm_path.cu): one cooperative launch per path segment when the problem fits
    m.lp_why.clear();
    m.lp_ok = lm_path_eligible(d, max_iter, m.sm_count, &m.lp_why);
    if (m.lp_ok && m.tie_exact) {
        m.lp_ok = false;
        m.lp_why = "exact boundary-tie mode (selections may need the host)";
    }
    if (m.lp_ok) {
        if (m.ctx->coop_launch < 0) CUDA_CHECK(cudaDeviceGetAttribute(&m.ctx->coop_launch, cudaDevAttrCooperativeLaunch, m.ctx->device));
        if (!m.ctx->coop_launch) {
            m.lp_ok = false;
            m.lp_why = "device without cooperative launch";
        }
    }
    if (m.lp_ok) {
        double *h_tau;
        m.lp_tau = mir.alloc<double>(MAXC, &h_tau);
        for (int q = 0; q < MAXC; q++) h_tau[q] = INFINITY;  // no candidate threshold yet: the first select reads the whole vector
    }
    mir.flush(m.st);

    // ---- chain state that starts from zero: one block, one memset
    auto z_bytes = [](size_t b) { return (b + 255) & ~(size_t)255; };
    const size_t zb_ks = z_bytes(MAXC * 4), zb_A = z_bytes((size_t)MAXC * kcap * 4), zb_bA = z_bytes((size_t)MAXC * kcap * 8),
                 zb_c0 = z_bytes(MAXC * 8), zb_lvl = z_bytes(8), zb_act = z_bytes(8), zb_slot = z_bytes(NSLOT * 8),
                 zb_beta = z_bytes((size_t)C * d.pstride * 8), zb_XA = z_bytes((size_t)C * n * d.ldA * 8),
                 zb_grp = grp ? z_bytes((size_t)MAXC * kcap * 4) : 0,
                 zb_lp = m.lp_ok ? z_bytes(2 * MAXC * 8) + z_bytes(LP_NDBG * 8) + z_bytes((size_t)2 * m.npad * MAXC * 8) : 0;
    const size_t ztotal = 5 * zb_ks + zb_A + zb_bA + zb_c0 + zb_lvl + zb_act + 2 * zb_slot + zb_beta + zb_XA +
                          (grp ? zb_ks + zb_grp : 0) + zb_lp;
    char *zp = ar.alloc<char>(ztotal);
    CUDA_CHECK(cudaMemsetAsync(zp, 0, ztotal, m.st));
    auto take = [&](size_t b) {
        char *r = zp;
        zp += b;
        return r;
    };
    d.ks = (int *)take(zb_ks);
    d.l = (int *)take(zb_ks);
    d.done = (int *)take(zb_ks);
    d.tie = (int *)take(zb_ks);
    d.tie_acc = (int *)take(zb_ks);
    d.A = (int *)take(zb_A);
    d.bA = (double *)take(zb_bA);
    d.coef0 = (double *)take(zb_c0);
    d.coef0_level = (double *)take(zb_lvl);
    m.n_active2 = (int *)take(zb_act);
    m.slots.ks = (int *)take(zb_slot);
    m.slots.coef0 = (double *)take(zb_slot);
    d.betaD = (double *)take(zb_beta);
    d.XA = (double *)take(zb_XA);
    if (grp) {
        d.Tc = (int *)take(zb_ks);
        d.AnewCols = (int *)take(zb_grp);
    }
    if (m.lp_ok) {
        m.lp_pub = (double *)take(z_bytes(2 * MAXC * 8));
        m.lp_dbg = (unsigned long long *)take(z_bytes(LP_NDBG * 8));
        m.lp_R = (double *)take(z_bytes((size_t)2 * m.npad * MAXC * 8));
    }
    d.n_active = m.n_active2;
    d.prev_active = nullptr;
    // ---- the rest needs no initial value
    d.Anew = ar.alloc<int>((size_t)MAXC * kcap);
    d.hist_rows = max_iter + 2;
    d.hist = ar.alloc<int>((size_t)C * d.hist_rows * kcap);
    d.XB = family_ == FAM_COX ? ar.alloc<double>((size_t)C * n * d.ldA) : nullptr;
    d.vec = ar.alloc<double>((size_t)C * NVEC * n);
    d.Smat = ar.alloc<double>((size_t)C * 2 * d.ldA * d.ldA);
    d.cw = ar.alloc<double>((size_t)C * CLMAX * 4 * d.ldA);
    d.CLcap = CLMAX;
    d.CLcap = chain_cluster_size(d, kcap, 1);  // the largest cluster any batch of this problem can ask for
    d.Spart = d.CLcap > 1 ? ar.alloc<double>((size_t)C * d.CLcap * d.nmat * d.ldA * d.ldA) : nullptr;
    m.slots.A = ar.alloc<int>((size_t)NSLOT * kcap);
    m.slots.bA = ar.alloc<double>((size_t)NSLOT * kcap);
    m.loss_scratch = ar.alloc<double>((size_t)2 * MAXC * 2 * n);
    m.loss_out = ar.alloc<double>(2 * MAXC);
    if (m.lp_ok) {
        if (std::getenv("BESS_B200_TRACE")) {
            m.lp_trace = ar.alloc<unsigned long long>((size_t)(MAXC + 1) * LP_TRACE * 2);
            CUDA_CHECK(cudaMemsetAsync(m.lp_trace, 0, (size_t)(MAXC + 1) * LP_TRACE * 2 * 8, m.st));
        } else {
            m.lp_trace = nullptr;
        }
        m.lp_ns = lm_path_slots(d, max_iter);
        m.lp_res_count = (size_t)LP_MAXSTEP * MAXC * (2 + kcap);
        m.lp_sync = ar.alloc<unsigned>(2 * LP_SYNC_WORDS);
        m.lp_cand = ar.alloc<LpCand>((size_t)MAXC * LP_CAP);
        m.lp_ncand = ar.alloc<int>(MAXC);
        m.lp_res_i = ar.alloc<int>(2 * m.lp_res_count);
        m.lp_res_d = ar.alloc<double>(2 * m.lp_res_count);
        m.ctx->reserve_resident(m.lp_res_count);
    }

    // ---- x_j.x_j over each chain's train rows
    if (family_ == FAM_LM && grp) {
        CUDA_CHECK(cudaMemcpyAsync(d.W, d_ind, vsz * 8, cudaMemcpyDeviceToDevice, m.st));
    } else if (family_ == FAM_LM) {
        double *Wkeep = d.W;
        d.W = d_ind;  // the staged indicators ARE the weight vector of this one pass
        BatchDesc b{};
        b.nch = C;
        for (int c = 0; c < C; c++) b.chain[c] = c;
        const int spx = m.span_begin(6);
        if (m.csc_norm) launch_csc_sweep(d, MODE_DH, m.st);
        else launch_dual_sweep(d, MODE_DH, m.st);
        launch_finish(d, MODE_DH, EPI_RAW, b, m.raw, m.st);
        m.span_end(spx);
        d.W = Wkeep;
        // finish wrote the reduced sums as raw[1][chain][pstride]: exactly the layout of xtx (raw is not used again while
        // these chains live)
        d.xtx = m.raw + (size_t)d.FS * d.pstride;
        stats_.n_sweeps++;
        stats_.norm_bytes += m.csc_norm ? 12.0 * (double)m.nnz + 8.0 * ((double)p + 1) + 16.0 * n * d.FS : 8.0 * n * p;
        stats_.kernel_launches += m.csc_norm ? 3 + (d.nlong ? 1 : 0) : 2;
    }
    if (m.csc_norm) {  // the active columns are expanded from the CSC arrays into AXr every iteration (launch_csc_gather)
        d.AXr = dalloc<double>(m.st, (size_t)C * n * kcap);
        d.ldXk = kcap;
        d.AXk = dalloc<double>(m.st, (size_t)C * n * d.ldXk);
        CUDA_CHECK(cudaMemsetAsync(d.AXk, 0, (size_t)C * n * d.ldXk * 8, m.st));
    }
    if (sharded_) {
        m.cand_s = dalloc<Cand>(m.st, (size_t)C * kcap);
        m.cand_r = dalloc<Cand>(m.st, (size_t)m.world * C * kcap);
        m.mstride = (long long)m.world * kcap;
        m.mv = dalloc<double>(m.st, (size_t)C * m.mstride);
        m.mi = dalloc<int>(m.st, (size_t)C * m.mstride);
        m.Aloc = dalloc<int>(m.st, (size_t)C * kcap);
        m.AXs = dalloc<double>(m.st, (size_t)C * n * kcap);
        d.AXr = dalloc<double>(m.st, (size_t)C * n * kcap);
        d.ldXk = kcap;
        d.AXk = dalloc<double>(m.st, (size_t)C * n * d.ldXk);
        CUDA_CHECK(cudaMemsetAsync(m.cand_s, 0, (size_t)C * kcap * sizeof(Cand), m.st));
        CUDA_CHECK(cudaMemsetAsync(m.AXs, 0, (size_t)C * n * kcap * 8, m.st));
        CUDA_CHECK(cudaMemsetAsync(d.AXk, 0, (size_t)C * n * d.ldXk * 8, m.st));
    }
    m.cstride = std::max<long long>(2LL * kcap + 16, ((long long)p / 8192 + 2) * std::min(kcap, TOPK_LMAX));
    if (sharded_) m.cstride = std::max<long long>(m.cstride, (long long)m.world * kcap + 16);
    m.ck0 = ar.alloc<double>((size_t)C * m.cstride);
    m.ck1 = ar.alloc<double>((size_t)C * m.cstride);
    m.ci0 = ar.alloc<int>((size_t)C * m.cstride);
    m.ci1 = ar.alloc<int>((size_t)C * m.cstride);
    m.ctx->reserve_support((size_t)MAXC * kcap);
    for (int q = 0; q < 2; q++) {
        m.mir[q].A = m.ctx->h_A + (size_t)q * MAXC * kcap;
        m.mir[q].bA = m.ctx->h_bA + (size_t)q * MAXC * kcap;
        m.tk[q].pending = false;
    }
    S_ = d.S;
    m.chains_ready = true;
}

bool Engine::resident_path() const { return d_->lp_ok; }
const std::string &Engine::resident_path_why() const { return d_->lp_why; }
void Engine::resident_counters(double *out24) const
{
    for (int i = 0; i < 24; i++) out24[i] = d_->lp_counters[i];
}
void Engine::resident_owner_counters(double *out4c) const
{
    for (int i = 0; i < 4 * MAXC; i++) out4c[i] = d_->lp_owner[i];
}

// Enqueue one launch of the resident kernel for the batch in t.b: memsets, kernel, result copies into the slot's pinned
// mirrors.  The caller records the ticket's event.
static void lp_launch(Engine::Impl &m, Engine::Impl::Ticket &t, const PathStep *steps, int nsteps)
{
    const Dev &d = t.d;
    if (nsteps < 1 || nsteps > LP_MAXSTEP) throw EngineError{"resident path: bad step count"};
    LpDesc &L = t.lp;
    L = LpDesc{};
    L.nsteps = nsteps;
    L.nch = t.b.nch;
    L.n_always = m.n_always;
    L.nsweep = m.sm_count - t.b.nch;
    L.ns = m.lp_ns;
    L.hist_rows = d.max_iter + 2;
    for (int q = 0; q < nsteps; q++) {
        if (steps[q].T < 1 || steps[q].T > m.Tmax) throw EngineError{"sparsity level outside [1, kcap]"};
        if (!(steps[q].lambda >= 0.0)) throw EngineError{"lambda must be >= 0"};
        L.T[q] = steps[q].T;
        L.lam[q] = steps[q].lambda;
    }
    for (int i = 0; i < t.b.nch; i++) L.chain[i] = t.b.chain[i];
    // two chain groups (alternate chains, so the full-data chain and the folds spread evenly): one group's owners work
    // while the other group is swept
    L.ng = lm_path_groups(L.nch);
    L.gcount[0] = L.gcount[1] = 0;
    for (int i = 0; i < L.nch; i++) {
        const int g = L.ng == 2 ? (i & 1) : 0;
        L.ogroup[i] = g;
        L.oslot[i] = L.gcount[g];
        L.gchain[g][L.gcount[g]++] = L.chain[i];
    }
    L.fh = lm_path_fh(L.nch, L.ng);
    L.Rg[0] = m.lp_R;
    L.Rg[1] = m.lp_R + (size_t)m.npad * MAXC;
    L.always = m.always;
    L.y = m.y;
    L.sync = m.lp_sync + (size_t)t.slot * LP_SYNC_WORDS;
    L.cand = m.lp_cand;
    L.ncand = m.lp_ncand;
    L.pub = m.lp_pub;
    L.tau = m.lp_tau;
    L.res_i = m.lp_res_i + (size_t)t.slot * m.lp_res_count;
    L.res_d = m.lp_res_d + (size_t)t.slot * m.lp_res_count;
    L.dbg = m.lp_dbg;
    L.trace = m.lp_trace;
    CUDA_CHECK(cudaMemsetAsync(L.sync, 0, LP_SYNC_WORDS * sizeof(unsigned), m.st));
    CUDA_CHECK(cudaMemsetAsync(m.lp_ncand, 0, MAXC * sizeof(int), m.st));
    const int sp = m.span_begin(4);
    launch_lm_path(d, L, m.sm_count, d.max_iter, m.st);
    m.span_end(sp);
    const size_t cnt = (size_t)nsteps * t.b.nch * (2 + d.kcap);
    DeviceContext *c = m.ctx;
    CUDA_CHECK(cudaMemcpyAsync(c->h_lp_i + (size_t)t.slot * c->cap_lp, L.res_i, cnt * sizeof(int), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(c->h_lp_d + (size_t)t.slot * c->cap_lp, L.res_d, cnt * sizeof(double), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(c->h_lp_sync + (size_t)t.slot * LP_SYNC_WORDS, L.sync, LP_SYNC_WORDS * sizeof(unsigned),
                               cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(c->h_lp_dbg + (size_t)t.slot * LP_NDBG, m.lp_dbg, LP_NDBG * sizeof(unsigned long long),
                               cudaMemcpyDeviceToHost, m.st));
}

// After the ticket's event: unpack the slot's mirrors.  outs[q] <- batch result of step q; la / lt [q * nch + i].
static void lp_parse(Engine::Impl &m, const Engine::Impl::Ticket &t, EngineStats &stats, BatchResult *outs, double *la, double *lt)
{
    const Dev &d = t.d;
    const LpDesc &L = t.lp;
    DeviceContext *c = m.ctx;
    const unsigned *sy = c->h_lp_sync + (size_t)t.slot * LP_SYNC_WORDS;
    if (sy[LP_SYNC_ABORT] != 0u || sy[LP_SYNC_TERM] == 0u)
        throw EngineError{"resident path: the kernel did not finish (phase barrier watchdog)"};
    const int *ri0 = c->h_lp_i + (size_t)t.slot * c->cap_lp;
    const double *rd0 = c->h_lp_d + (size_t)t.slot * c->cap_lp;
    const int nch = L.nch, kc = d.kcap;
    for (int q = 0; q < L.nsteps; q++) {
        BatchResult &o = outs[q];
        o.T = L.T[q];
        o.nchains = nch;
        for (int i = 0; i < nch; i++) {
            const int *ri = ri0 + ((size_t)q * nch + i) * (2 + kc);
            const double *rd = rd0 + ((size_t)q * nch + i) * (2 + kc);
            o.chain_ids[i] = L.chain[i];
            o.l[i] = ri[0];
            o.coef0[i] = 0.0;  // the gaussian fit leaves coef0 at coef0_init = 0 (Algorithm.h:1131-1135)
            o.A[i].assign(ri + 2, ri + 2 + L.T[q]);
            o.bA[i].assign(rd + 2, rd + 2 + L.T[q]);
            la[(size_t)q * nch + i] = rd[0];
            lt[(size_t)q * nch + i] = rd[1];
            stats.n_pdas_iters += std::min(ri[0], d.max_iter);
            stats.n_boundary_ties += ri[1];
        }
    }
    stats.n_suspect_pivots += sy[LP_SYNC_RANKDEF];
    if (m.lp_trace) {  // developer aid: time line of the owner phases and of sweeper 0 ($BESS_B200_TRACE = output file)
        std::vector<unsigned long long> tr((size_t)(MAXC + 1) * LP_TRACE * 2);
        CUDA_CHECK(cudaMemcpy(tr.data(), m.lp_trace, tr.size() * 8, cudaMemcpyDeviceToHost));
        if (FILE *f = std::fopen(std::getenv("BESS_B200_TRACE"), "w")) {
            for (int c2 = 0; c2 <= MAXC; c2++)
                for (int q = 0; q < LP_TRACE; q++) {
                    const unsigned long long a = tr[((size_t)c2 * LP_TRACE + q) * 2], b2 = tr[((size_t)c2 * LP_TRACE + q) * 2 + 1];
                    if (a || b2) std::fprintf(f, "%d %d %llu %llu\n", c2, q, a, b2);
                }
            std::fclose(f);
        }
        CUDA_CHECK(cudaMemset(m.lp_trace, 0, tr.size() * 8));
    }
    const double iters = (double)sy[LP_SYNC_ITERS];
    stats.n_sweeps += (long long)iters;
    stats.sweep_bytes += iters * (8.0 * d.n * d.p + 8.0 * d.n * nch + 8.0 * d.p * nch);
    stats.kernel_launches += 1;
    stats.n_fits += (long long)nch * L.nsteps;
    stats.n_batches += L.nsteps;
    m.lp_counters[0] += 1.0;
    m.lp_counters[1] += iters;
    m.lp_counters[2] += (double)sy[LP_SYNC_FALLBACKS];
    m.lp_counters[3] += (double)L.nsteps;
    m.lp_counters[4] += (double)sy[LP_SYNC_MERGED];
    const unsigned long long *dbg = c->h_lp_dbg + (size_t)t.slot * LP_NDBG;  // cumulative since setup_chains
    for (int q = 0; q < 8; q++) m.lp_counters[8 + q] = (double)dbg[q];
    for (int q = 0; q < 3; q++) m.lp_counters[16 + q] = (double)dbg[16 + q];
    for (int q = 0; q < 5; q++) m.lp_counters[19 + q] = (double)dbg[8 + q];
    for (int q = 0; q < 3; q++) m.lp_counters[5 + q] = (double)dbg[13 + q];  // DEBUG chol  // assemble, candidate load, slot assignment, scatter + cycle test, level bookkeeping
    for (int q = 0; q < 4 * MAXC; q++) m.lp_owner[q] = (double)dbg[32 + q];  // assembling the normal equations (part of `solve` when added to slot 13)
}

void Engine::run_steps(const std::vector<PathStep> &steps, const std::vector<int> &chains, std::vector<BatchResult> &out,
                       std::vector<double> &loss_all, std::vector<double> &loss_test)
{
    Impl &m = *d_;
    if (!m.chains_ready || !m.lp_ok) throw EngineError{"run_steps: the resident path is not available (" + m.lp_why + ")"};
    if (m.tk[0].pending || m.tk[1].pending) throw EngineError{"run_steps: a batch is still pending"};
    if (chains.empty() || (int)chains.size() > m.nchains) throw EngineError{"bad chain set"};
    const int nch = (int)chains.size();
    out.assign(steps.size(), BatchResult{});
    loss_all.assign(steps.size() * nch, 0.0);
    loss_test.assign(steps.size() * nch, 0.0);
    for (size_t s0 = 0; s0 < steps.size(); s0 += LP_MAXSTEP) {
        const int cnt = (int)std::min<size_t>(LP_MAXSTEP, steps.size() - s0);
        const int slot = (int)(m.seq++ & 1);
        Impl::Ticket &t = m.tk[slot];
        t.b = BatchDesc{};
        t.b.nch = nch;
        for (int i = 0; i < nch; i++) {
            if (chains[i] < 0 || chains[i] >= m.nchains) throw EngineError{"chain id out of range"};
            t.b.chain[i] = chains[i];
        }
        t.d = m.d;
        t.slot = slot;
        t.resident = true;
        if (!t.ev) CUDA_CHECK(cudaEventCreateWithFlags(&t.ev, cudaEventDisableTiming));
        lp_launch(m, t, steps.data() + s0, cnt);
        CUDA_CHECK(cudaEventRecord(t.ev, m.st));
        CUDA_CHECK(cudaEventSynchronize(t.ev));
        lp_parse(m, t, stats_, out.data() + s0, loss_all.data() + s0 * nch, loss_test.data() + s0 * nch);
    }
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    m.collect_spans();
}

// Algorithmic bytes of one CSC sweep (launch_csc_sweep): the three CSC arrays, the statistics of every column, the
// n-vectors of every chain slot (read by the sums kernel and, for cox, the prefix written and read), the partials written.
static double csc_sweep_bytes(const Dev &d, int mode)
{
    const int nv = mode == MODE_D ? 1 : (mode == MODE_DH ? 2 : 4), nq = mode == MODE_D ? 1 : (mode == MODE_DH ? 2 : 5);
    return 12.0 * (double)d.csc_nnz + 8.0 * ((double)d.p + 1) + 16.0 * d.p + 8.0 * d.n * d.FS * (nv + (mode == MODE_COX ? 2 : 0)) +
           8.0 * (double)d.p * d.FS * nq;
}
static inline int sweep_mode(int family) { return family == FAM_LM ? MODE_D : (family == FAM_COX ? MODE_COX : MODE_DH); }
static inline int sweep_epi(int family)
{
    return family == FAM_LM ? EPI_SACR_LM : (family == FAM_COX ? EPI_SACR_COX : EPI_SACR_GLM);
}

static int g_first_group = 3;
void engine_debug_first_group(int n) { g_first_group = n < 1 ? 1 : n; }

// One group of PDAS iterations for the batch described by ticket `t` (enqueue only).
static void enqueue_iterations(Engine::Impl &m, Engine::Impl::Ticket &t, int count, bool sharded, long long col_lo);

static void enqueue_results(Engine::Impl &m, Engine::Impl::Ticket &t);

// One batch in exact boundary-tie mode (Engine::set_tie_exact): the PDAS iterations run one at a time; after every device
// select the host reads the tie flags and repeats the selection of a tied chain with the reference's max_k on the chain's
// sacrifice vector.  Synchronous: the batch is finished when this returns.
static void run_batch_exact(Engine::Impl &m, Engine::Impl::Ticket &t, EngineStats &stats)
{
    Dev &d = t.d;
    const BatchDesc &b = t.b;
    d.prev_active = nullptr;  // no speculative batch behind this one
    t.fused = false;
    const int T = t.T, cmin = t.cmin, cmax = t.cmax, nspan = cmax - cmin + 1;
    const int mode = sweep_mode(d.family), epi = sweep_epi(d.family);
    const int N = d.grouped ? d.N : d.p;
    launch_chain_begin(d, b, m.st);
    std::vector<int> tie(MAXC), done(MAXC), hsel((size_t)T);
    std::vector<double> row((size_t)N);
    for (int it = 0; it <= d.max_iter; it++) {
        int active = 0;
        CUDA_CHECK(cudaMemcpyAsync(&active, d.n_active, sizeof(int), cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaStreamSynchronize(m.st));
        if (active == 0) break;
        if (d.grouped) {
            launch_group_sacrifice(d, b, m.st);
        } else {
            if (d.ccp) launch_csc_sweep(d, mode, m.st);
            else launch_dual_sweep(d, mode, m.st);
            launch_finish(d, mode, epi, b, nullptr, m.st);
        }
        if (m.n_always) launch_pin(d, d.bd + (size_t)cmin * d.pstride, d.pstride, nspan, m.always, m.n_always, m.st);
        launch_topk(d.bd + (size_t)cmin * d.pstride, d.pstride, N, T, nspan, d.Anew + (size_t)cmin * d.kcap, d.kcap, d.tie + cmin,
                    m.ck0, m.ci0, m.ck1, m.ci1, m.cstride, m.st, d.gate);
        CUDA_CHECK(cudaMemcpyAsync(tie.data(), d.tie, MAXC * sizeof(int), cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaMemcpyAsync(done.data(), d.done, MAXC * sizeof(int), cudaMemcpyDeviceToHost, m.st));
        CUDA_CHECK(cudaStreamSynchronize(m.st));
        for (int i = 0; i < b.nch; i++) {
            const int c = b.chain[i];
            if (done[c] || !tie[c]) continue;
            CUDA_CHECK(cudaMemcpyAsync(row.data(), d.bd + (size_t)c * d.pstride, (size_t)N * 8, cudaMemcpyDeviceToHost, m.st));
            CUDA_CHECK(cudaStreamSynchronize(m.st));
            host_max_k(row.data(), N, T, hsel.data());
            CUDA_CHECK(cudaMemcpyAsync(d.Anew + (size_t)c * d.kcap, hsel.data(), (size_t)T * sizeof(int), cudaMemcpyHostToDevice, m.st));
            CUDA_CHECK(cudaStreamSynchronize(m.st));  // hsel is reused
        }
        if (d.grouped) launch_group_expand(d, b, m.st);
        if (d.ccp) launch_csc_gather(d, b, 0, m.st);
        launch_chain_fit(d, b, m.st);
        t.enq++;
        stats.kernel_launches += d.grouped ? 4 : (d.ccp ? 7 + (d.nlong ? 1 : 0) : 5);
    }
    enqueue_results(m, t);
}

int Engine::run_batch_enqueue(int T, const std::vector<int> &chains, bool new_path_step, const std::vector<LossJob> *jobs,
                              double lambda)
{
    Impl &m = *d_;
    if (!m.chains_ready) throw EngineError{"run_batch before setup_chains"};
    Dev &d = m.d;
    if (T < 1 || T > m.Tmax) throw EngineError{"sparsity level outside [1, kcap]"};
    if (chains.empty() || (int)chains.size() > m.nchains) throw EngineError{"bad chain set"};
    if (!(lambda >= 0.0)) throw EngineError{"lambda must be >= 0"};
    const int slot = (int)(m.seq++ & 1);
    Impl::Ticket &t = m.tk[slot];
    if (t.pending) throw EngineError{"run_batch_enqueue: the ticket of this slot has not been collected"};
    BatchDesc &b = t.b;
    b = BatchDesc{};
    b.nch = (int)chains.size();
    b.T = T;
    b.new_path_step = new_path_step ? 1 : 0;
    b.CL = chain_cluster_size(d, d.grouped ? std::min(d.kcap, T * d.gmax) : T, m.cl_chains > 0 ? std::max(m.cl_chains, b.nch) : b.nch);
    stats_.max_cluster = std::max(stats_.max_cluster, b.CL);
    t.cmin = MAXC;
    t.cmax = -1;
    for (int i = 0; i < b.nch; i++) {
        if (chains[i] < 0 || chains[i] >= m.nchains) throw EngineError{"chain id out of range"};
        b.chain[i] = chains[i];
        t.cmin = std::min(t.cmin, chains[i]);
        t.cmax = std::max(t.cmax, chains[i]);
    }
    if (new_path_step && chains[0] != 0) throw EngineError{"a new path step must include the full-data chain"};
    t.ld = LossDesc{};
    t.has_jobs = jobs != nullptr;
    if (jobs) {
        if ((int)jobs->size() > 2 * MAXC) throw EngineError{"too many loss jobs"};
        t.ld.njobs = (int)jobs->size();
        for (int i = 0; i < t.ld.njobs; i++) {
            t.ld.chain[i] = (*jobs)[i].chain;
            t.ld.kind[i] = (*jobs)[i].kind;
            t.ld.fold[i] = (*jobs)[i].fold;
        }
    }
    // the kernels of this batch carry their own copy of the descriptor: ridge level, gate counter of this slot and the
    // counter of the batch enqueued before it (Dev::prev_active)
    t.d = d;
    t.d.ldXr = T;
    t.d.lambda = lambda;
    t.d.n_active = m.n_active2 + slot;
    t.d.prev_active = m.n_active2 + (slot ^ 1);
    t.d.gate = t.d.n_active;
    t.T = T;
    t.slot = slot;
    t.enq = 0;
    t.launches = 1;
    static const bool fuse_topk = [] {
        const char *e = std::getenv("BESS_B200_FUSE_TOPK");
        return !(e && e[0] == '0');
    }();
    t.fused = fuse_topk && !sharded_ && !d.grouped && d.p <= TOPK_LMAX;
    if (!t.ev) CUDA_CHECK(cudaEventCreateWithFlags(&t.ev, cudaEventDisableTiming));
    t.resident = m.lp_ok;
    if (t.resident) {
        // gaussian family, L2-resident design: the whole batch (prologue, every PDAS iteration, losses) is one launch
        const PathStep st1{T, lambda};
        lp_launch(m, t, &st1, 1);
        t.loss_kernel = false;
        for (int i = 0; i < t.ld.njobs; i++) {
            bool in_batch = false;
            for (int q = 0; q < b.nch; q++) in_batch = in_batch || b.chain[q] == t.ld.chain[i];
            const bool ok = in_batch && (t.ld.kind[i] == 0 || (t.ld.kind[i] == 1 && t.ld.fold[i] == t.ld.chain[i] - 1));
            if (!ok) t.loss_kernel = true;
        }
        if (t.loss_kernel) {
            Engine::Impl::Mirror &h = m.mir[t.slot];
            const int sp2 = m.span_begin(5);
            launch_losses(t.d, t.ld, m.testrows, m.ntest, m.y, m.w, m.lfact, m.loss_scratch, m.loss_out, m.st);
            m.span_end(sp2);
            CUDA_CHECK(cudaMemcpyAsync(h.loss, m.loss_out, t.ld.njobs * sizeof(double), cudaMemcpyDeviceToHost, m.st));
        }
        CUDA_CHECK(cudaEventRecord(t.ev, m.st));
        t.pending = true;
        return slot;
    }

    if (m.tie_exact && !sharded_) {
        run_batch_exact(m, t, stats_);
        t.pending = true;
        return slot;
    }
    int sp = m.span_begin(4);
    launch_chain_begin(t.d, b, m.st);
    m.span_end(sp);
    // PDAS iterations are enqueued speculatively: the kernels of an iteration return at once when every chain of the
    // batch has already met the stopping rule (Dev::gate), so the host only synchronises once per group.  PDAS needs
    // 2-4 iterations per warm-started fit; the first group covers that, later groups are shorter.
    enqueue_iterations(m, t, std::min(g_first_group, d.max_iter), sharded_, col_lo_);
    t.pending = true;
    return slot;
}

static void enqueue_iterations(Engine::Impl &m, Engine::Impl::Ticket &t, int count, bool sharded, long long col_lo)
{
    const Dev &d = t.d;
    const BatchDesc &b = t.b;
    const int T = t.T, cmin = t.cmin, cmax = t.cmax;
    const int mode = sweep_mode(d.family), epi = sweep_epi(d.family);
    int sp;
    for (int q = 0; q < count; q++) {
        if (d.grouped) {
            // group selection: sweep + group sacrifice in one kernel, top-k over the groups, groups -> columns
            sp = m.span_begin(1);
            launch_group_sacrifice(d, b, m.st);
            m.span_end(sp);
            if (m.n_always)
                launch_pin(d, d.bd + (size_t)cmin * d.pstride, d.pstride, cmax - cmin + 1, m.always, m.n_always, m.st);
            sp = m.span_begin(3);
            launch_topk(d.bd + (size_t)cmin * d.pstride, d.pstride, d.N, T, cmax - cmin + 1, d.Anew + (size_t)cmin * d.kcap,
                        d.kcap, d.tie + cmin, m.ck0, m.ci0, m.ck1, m.ci1, m.cstride, m.st, d.gate);
            launch_group_expand(d, b, m.st);
            m.span_end(sp);
            sp = m.span_begin(4);
            launch_chain_fit(d, b, m.st);
            m.span_end(sp);
            continue;
        }
        sp = m.span_begin(1);
        if (d.ccp) launch_csc_sweep(d, mode, m.st);
        else launch_dual_sweep(d, mode, m.st);
        m.span_end(sp);
        if (!t.fused) {
            sp = m.span_begin(2);
            launch_finish(d, mode, epi, b, nullptr, m.st);
            m.span_end(sp);
            if (m.n_always)
                launch_pin(d, d.bd + (size_t)cmin * d.pstride, d.pstride, cmax - cmin + 1, m.always, m.n_always, m.st);
        }
        sp = m.span_begin(3);
        if (t.fused) {
            launch_topk_fused(d, mode, epi, cmin, cmax - cmin + 1, T, m.always, m.n_always, m.st);
        } else if (!sharded) {
            launch_topk(d.bd + (size_t)cmin * d.pstride, d.pstride, d.p, T, cmax - cmin + 1, d.Anew + (size_t)cmin * d.kcap,
                        d.kcap, d.tie + cmin, m.ck0, m.ci0, m.ck1, m.ci1, m.cstride, m.st, d.gate);
        } else {
            // exact local top-k -> all-gather of (sacrifice, global index) candidates -> identical merge on every
            // rank (rank-major concatenation of ascending lists is ascending, so the ordered compaction of the
            // select keeps the reference's ascending-index output and the lower-index tie rule)
            const NcclApi &api = nccl_api();
            const int nspan = cmax - cmin + 1;
            const int kloc = std::min(T, d.p);
            launch_topk(d.bd + (size_t)cmin * d.pstride, d.pstride, d.p, kloc, nspan, m.Aloc + (size_t)cmin * d.kcap, d.kcap,
                        d.tie + cmin, m.ck0, m.ci0, m.ck1, m.ci1, m.cstride, m.st, d.gate);
            launch_pack_candidates(d.bd + (size_t)cmin * d.pstride, d.pstride, m.Aloc + (size_t)cmin * d.kcap, d.kcap, kloc, T,
                                   col_lo, nspan, m.cand_s + (size_t)cmin * d.kcap, d.kcap, d.gate, m.st);
            NCCL_CHECK(api.AllGather(m.cand_s, m.cand_r, (size_t)m.nchains * d.kcap * sizeof(Cand), ncclChar, m.comm, m.st));
            launch_unpack_candidates(m.cand_r + (size_t)cmin * d.kcap, m.world, m.nchains, d.kcap, T,
                                     m.mv + (size_t)cmin * m.mstride, m.mi + (size_t)cmin * m.mstride, m.mstride, d.gate, m.st);
            launch_topk(m.mv + (size_t)cmin * m.mstride, m.mstride, m.world * T, T, nspan, d.Anew + (size_t)cmin * d.kcap,
                        d.kcap, d.tie + cmin, m.ck0, m.ci0, m.ck1, m.ci1, m.cstride, m.st, d.gate,
                        m.mi + (size_t)cmin * m.mstride);
            // the k active columns, all rows: owners write them, everybody sums (x + 0 is exact)
            launch_gather_active(d, b, m.AXs, m.st);
            NCCL_CHECK(api.AllReduce(m.AXs, d.AXr, (size_t)m.nchains * d.n * T, ncclDouble, ncclSum, m.comm, m.st));
        }
        m.span_end(sp);
        sp = m.span_begin(4);
        if (d.ccp) launch_csc_gather(d, b, 0, m.st);
        launch_chain_fit(d, b, m.st);
        m.span_end(sp);
    }
    t.enq += count;
    enqueue_results(m, t);
}

// results are enqueued behind a group of iterations; they are only used if the batch turns out to be finished
static void enqueue_results(Engine::Impl &m, Engine::Impl::Ticket &t)
{
    const Dev &d = t.d;
    int sp;
    Engine::Impl::Mirror &h = m.mir[t.slot];
    if (t.has_jobs) {
        sp = m.span_begin(5);
        launch_losses(d, t.ld, m.testrows, m.ntest, m.y, m.w, m.lfact, m.loss_scratch, m.loss_out, m.st);
        m.span_end(sp);
        CUDA_CHECK(cudaMemcpyAsync(h.loss, m.loss_out, t.ld.njobs * sizeof(double), cudaMemcpyDeviceToHost, m.st));
    }
    CUDA_CHECK(cudaMemcpyAsync(h.done, d.done, MAXC * sizeof(int), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(h.l, d.l, MAXC * sizeof(int), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(h.tie, d.tie_acc, MAXC * sizeof(int), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(h.ks, d.ks, MAXC * sizeof(int), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(h.gate, d.n_active, sizeof(int), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(h.coef0, d.coef0, MAXC * sizeof(double), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(h.A, d.A, (size_t)MAXC * d.kcap * sizeof(int), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaMemcpyAsync(h.bA, d.bA, (size_t)MAXC * d.kcap * sizeof(double), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaEventRecord(t.ev, m.st));
}

bool Engine::run_batch_collect(int ticket, BatchResult &out, std::vector<double> *loss_out)
{
    Impl &m = *d_;
    if (ticket < 0 || ticket > 1 || !m.tk[ticket].pending) throw EngineError{"run_batch_collect: no such pending batch"};
    Impl::Ticket &t = m.tk[ticket];
    Impl::Mirror &h = m.mir[t.slot];
    const Dev &d = t.d;
    const BatchDesc &b = t.b;
    CUDA_CHECK(cudaEventSynchronize(t.ev));
    if (t.resident) {
        t.pending = false;
        double la[MAXC], lt[MAXC];
        lp_parse(m, t, stats_, &out, la, lt);
        if (t.has_jobs && loss_out) {
            if (t.loss_kernel) {
                stats_.kernel_launches++;
                loss_out->assign(h.loss, h.loss + t.ld.njobs);
            } else {
                loss_out->resize((size_t)t.ld.njobs);
                for (int i = 0; i < t.ld.njobs; i++) {
                    int q = 0;
                    while (b.chain[q] != t.ld.chain[i]) q++;
                    (*loss_out)[(size_t)i] = t.ld.kind[i] == 0 ? la[q] : lt[q];
                }
            }
        }
        return true;
    }
    auto finished = [&] {
        bool all = true;
        for (int i = 0; i < b.nch; i++) all = all && h.done[b.chain[i]];
        return all;
    };
    const bool in_one_go = finished();
    // a batch that was itself enqueued behind an unfinished one never started (its gate counter reads 0 while its chains
    // are not done): the caller collects the earlier batch first, so this cannot happen here
    while (!finished() && t.enq < d.max_iter) {
        enqueue_iterations(m, t, std::min(2, d.max_iter - t.enq), sharded_, col_lo_);
        CUDA_CHECK(cudaEventSynchronize(t.ev));
    }
    t.pending = false;
    const int T = t.T;
    out.T = T;
    out.nchains = b.nch;
    int executed = 0;  // iterations that actually ran (the rest of the last group returned at the gate)
    for (int i = 0; i < b.nch; i++) {
        const int c = b.chain[i];
        out.chain_ids[i] = c;
        out.l[i] = h.l[c];
        out.coef0[i] = h.coef0[c];
        const int ks = d.grouped ? h.ks[c] : T;  // columns in the support (== T without group structure)
        out.A[i].assign(h.A + (size_t)c * d.kcap, h.A + (size_t)c * d.kcap + ks);
        out.bA[i].assign(h.bA + (size_t)c * d.kcap, h.bA + (size_t)c * d.kcap + ks);
        const int iters = std::min(h.l[c], d.max_iter);
        stats_.n_pdas_iters += iters;
        stats_.n_boundary_ties += h.tie[c];
        executed = std::max(executed, iters);
    }
    const int mode = sweep_mode(family_);
    const double vec_bytes = 8.0 * d.n * b.nch * (mode == MODE_D ? 1 : (mode == MODE_DH ? 2 : 4)) + 8.0 * d.p * b.nch;
    const long long per_iter = d.grouped ? 4 + (m.n_always ? 1 : 0)
                                         : (t.fused ? 3 : 4 + (m.n_always ? 1 : 0) + (sharded_ ? 4 : 0)) + (d.ccp ? 2 + (d.nlong ? 1 : 0) : 0);
    stats_.n_sweeps += executed;
    stats_.sweep_bytes += executed * (d.ccp ? csc_sweep_bytes(d, mode) : 8.0 * d.n * d.p * (d.grouped ? b.nch : 1) + vec_bytes);
    stats_.kernel_launches += 1 + (long long)executed * per_iter + (t.has_jobs ? 1 : 0);  // gated no-op launches are not counted
    stats_.n_fits += b.nch;
    stats_.n_batches++;
    if (t.has_jobs && loss_out) loss_out->assign(h.loss, h.loss + t.ld.njobs);
    return in_one_go;
}

void Engine::run_batch(int T, const std::vector<int> &chains, bool new_path_step, BatchResult &out,
                       const std::vector<LossJob> *jobs, std::vector<double> *loss_out, double lambda)
{
    const int tk = run_batch_enqueue(T, chains, new_path_step, jobs, lambda);
    run_batch_collect(tk, out, loss_out);
    Impl &m = *d_;
    if (!m.tk[tk ^ 1].pending) {
        CUDA_CHECK(cudaStreamSynchronize(m.st));
        m.collect_spans();
    }
}

void Engine::run_batch_discard(int ticket)
{
    Impl &m = *d_;
    if (ticket < 0 || ticket > 1 || !m.tk[ticket].pending) return;
    CUDA_CHECK(cudaEventSynchronize(m.tk[ticket].ev));
    m.tk[ticket].pending = false;
}

void Engine::chain_state(int chain, int op, int slot_beta, int slot_coef0)
{
    Impl &m = *d_;
    if (!m.chains_ready) throw EngineError{"chain_state before setup_chains"};
    if (sharded_) throw EngineError{"chain_state is not available in column-sharded mode"};
    if (chain < 0 || chain >= m.nchains || slot_beta >= NSLOT || slot_coef0 >= NSLOT) throw EngineError{"bad chain_state call"};
    if (op != STATE_ZERO && op != STATE_SAVE && op != STATE_LOAD) throw EngineError{"bad chain_state op"};
    const int sp = m.span_begin(5);
    launch_chain_state(m.d, chain, op, slot_beta, slot_coef0, m.slots, m.st);
    m.span_end(sp);
    stats_.kernel_launches += (op == STATE_LOAD && slot_beta >= 0) ? 2 : 1;
}

void Engine::losses(const std::vector<LossJob> &jobs, std::vector<double> &out)
{
    Impl &m = *d_;
    if (jobs.empty()) { out.clear(); return; }
    if ((int)jobs.size() > 2 * MAXC) throw EngineError{"too many loss jobs"};
    LossDesc ld{};
    ld.njobs = (int)jobs.size();
    for (int i = 0; i < ld.njobs; i++) {
        ld.chain[i] = jobs[i].chain;
        ld.kind[i] = jobs[i].kind;
        ld.fold[i] = jobs[i].fold;
    }
    const int sp = m.span_begin(5);
    launch_losses(m.d, ld, m.testrows, m.ntest, m.y, m.w, m.lfact, m.loss_scratch, m.loss_out, m.st);
    m.span_end(sp);
    CUDA_CHECK(cudaMemcpyAsync(m.mir[0].loss, m.loss_out, ld.njobs * sizeof(double), cudaMemcpyDeviceToHost, m.st));
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    stats_.kernel_launches++;
    out.assign(m.mir[0].loss, m.mir[0].loss + ld.njobs);
}

// Roofline probe: `reps` back-to-back dual sweeps (+ finish) for all chain slots; returns mean ms per sweep kernel.
float Engine::time_dual_sweep(int nch, int reps)
{
    Impl &m = *d_;
    if (!m.chains_ready) throw EngineError{"time_dual_sweep before setup_chains"};
    (void)nch;
    const int mode = sweep_mode(family_);
    cudaEvent_t e0, e1;
    CUDA_CHECK(cudaEventCreate(&e0));
    CUDA_CHECK(cudaEventCreate(&e1));
    auto sweep = [&] {
        if (m.d.ccp) launch_csc_sweep(m.d, mode, m.st);
        else launch_dual_sweep(m.d, mode, m.st);
    };
    sweep();
    CUDA_CHECK(cudaEventRecord(e0, m.st));
    for (int r = 0; r < reps; r++) sweep();
    CUDA_CHECK(cudaEventRecord(e1, m.st));
    CUDA_CHECK(cudaStreamSynchronize(m.st));
    float ms = 0.f;
    CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    stats_.kernel_launches += (long long)(reps + 1) * (m.d.ccp ? 2 + (m.d.nlong ? 1 : 0) : 1);
    return ms / (float)reps;
}

double Engine::dual_sweep_bytes() const
{
    const Dev &d = d_->d;
    return d.ccp ? csc_sweep_bytes(d, sweep_mode(family_)) : 8.0 * (double)n_ * (double)p_;
}

// Test hook: recompute the sacrifice of every chain of `chains` for the state the last batch returned, through the
// dispatch a fit of this batch uses.  The gradient vectors are published again from the stored (A, beta_A, coef0) first
// (see launch_chain_gradient); the launches run on a copy of the descriptor without gate, at ridge level `lambda`, with
// every chain marked as iterating (the group kernels skip chains that are done).
void Engine::debug_sacrifice(const std::vector<int> &chains, double lambda, std::vector<double> &bd_out, int *info_out)
{
    Impl &m = *d_;
    if (!m.chains_ready) throw EngineError{"debug_sacrifice before setup_chains"};
    if (sharded_) throw EngineError{"debug_sacrifice is not available in column-sharded mode"};
    if (m.tk[0].pending || m.tk[1].pending) throw EngineError{"debug_sacrifice: a batch is still pending"};
    if (chains.empty() || (int)chains.size() > m.nchains) throw EngineError{"bad chain set"};
    if (!(lambda >= 0.0)) throw EngineError{"lambda must be >= 0"};
    Dev d = m.d;
    d.gate = nullptr;
    d.prev_active = nullptr;
    d.lambda = lambda;
    BatchDesc b{};
    b.nch = (int)chains.size();
    b.CL = 1;
    for (int i = 0; i < b.nch; i++) {
        if (chains[i] < 0 || chains[i] >= m.nchains) throw EngineError{"chain id out of range"};
        b.chain[i] = chains[i];
    }
    int *done0 = dalloc<int>(m.st, MAXC);
    CUDA_CHECK(cudaMemsetAsync(done0, 0, MAXC * sizeof(int), m.st));
    d.done = done0;
    launch_chain_gradient(d, b, m.st);
    const int mode = sweep_mode(family_), epi = sweep_epi(family_);
    for (int q = 0; q < 8; q++) info_out[q] = 0;
    info_out[1] = d.FS;
    if (d.grouped) {
        info_out[0] = 3;
        info_out[5] = launch_group_sacrifice(d, b, m.st);
    } else if (d.ccp) {
        info_out[0] = 4;  // the sweep over the CSC arrays
        info_out[2] = d.csc_g;
        info_out[5] = d.nlong;  // columns swept by a CTA each
        info_out[3] = d.S;
        info_out[4] = d.rows_per_split;
        launch_csc_sweep(d, mode, m.st);
        launch_finish(d, mode, epi, b, nullptr, m.st);
    } else {
        info_out[0] = sweep_uses_tma(d) ? 2 : 1;
        info_out[2] = sweep_cpt(d, mode);
        info_out[3] = d.S;
        info_out[4] = d.rows_per_split;
        launch_dual_sweep(d, mode, m.st);
        launch_finish(d, mode, epi, b, nullptr, m.st);
    }
    const int N = d.grouped ? d.N : d.p;
    bd_out.resize((size_t)b.nch * N);
    for (int i = 0; i < b.nch; i++)
        CUDA_CHECK(cudaMemcpyAsync(bd_out.data() + (size_t)i * N, d.bd + (size_t)b.chain[i] * d.pstride, (size_t)N * 8,
                                   cudaMemcpyDeviceToHost, m.st));
    dfree(m.st, done0);
    CUDA_CHECK(cudaStreamSynchronize(m.st));
}

}  // namespace bess
