// capi.cu -- the C ABI of include/cgb200.h: context management, the CG iteration schedule
// (CUDA-graph replay, device-side convergence, batched host polling) and the NCCL gather.
//
// Multi-GPU design (replaces MPI_Allgatherv + 2 x MPI_Allreduce per iteration,
// code/MPI/cg.cc:105-136): A is row-sharded by the reference's partition rule; the O(N) vectors
// x, r, p are REPLICATED and updated redundantly by every rank, so the only exchange per
// iteration is ONE all-gather of the Ap rows after the mat-vec.  The
// scalars (alpha, beta, r'r, the stop test) are then computed by every rank from identical
// data in an identical order: bitwise equal on all ranks without any all-reduce.
// Two implementations of that exchange (option "exchange"):
//   1 (default once cgb_exchange_import was called)  FUSED: the mat-vec kernel stores every
//     finished row straight into all ranks' gather buffers over NVLink (peer-mapped memory,
//     cudaIpc across processes) as self-flagging 16-byte LL entries {lo, tag, hi, tag}; the
//     x/r update kernel polls exactly the entries it reads.  No fence, no flag, no collective
//     kernel, nothing between the two launches.
//   0  ncclAllGather (in place) between the two kernels -- the baseline to beat.
#include "../../include/cgb200.h"
#include "cgb_kernels.h"

#include <cmath>
#include <cstdarg>
#include <cstddef>
#include <cstdio>
#include <cstring>
#include <dlfcn.h>
#include <mutex>
#include <new>
#include <string>
#include <unistd.h>
#include <unordered_map>
#include <vector>

using namespace cgb;

// ------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";

static int fail(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return fail(e_ == cudaErrorNoDevice || e_ == cudaErrorInsufficientDriver               \
                            ? CGB_ERR_NO_DEVICE                                                    \
                            : CGB_ERR_CUDA,                                                        \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

// ------------------------------------------------------------------ NCCL, loaded on demand
// (dlopen keeps libnccl out of DT_NEEDED: inside a torch process we bind to the copy torch
// already loaded, in the C++ host program to the system one.)
namespace {
typedef struct ncclComm *ncclComm_t;
typedef struct { char internal[CGB_UNIQUE_ID_BYTES]; } ncclUniqueId;
enum { kNcclDouble = 8 };
struct Nccl {
    void *h = nullptr;
    int (*GetUniqueId)(ncclUniqueId *) = nullptr;
    int (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    int (*CommDestroy)(ncclComm_t) = nullptr;
    int (*AllGather)(const void *, void *, size_t, int, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(int) = nullptr;
    int (*GetVersion)(int *) = nullptr;
};
Nccl g_nccl;
std::mutex g_nccl_mu; // ranks may be threads of one process

int load_nccl()
{
    std::lock_guard<std::mutex> lock(g_nccl_mu);
    if (g_nccl.h) return CGB_OK;
    const char *names[] = {"libnccl.so.2", "libnccl.so"};
    void *h = nullptr;
    for (const char *nm : names) {
        h = dlopen(nm, RTLD_NOW | RTLD_GLOBAL);
        if (h) break;
    }
    if (!h) return fail(CGB_ERR_NCCL, "cannot dlopen libnccl.so.2: %s", dlerror());
    Nccl n;
    n.h = h;
    n.GetUniqueId = (decltype(n.GetUniqueId))dlsym(h, "ncclGetUniqueId");
    n.CommInitRank = (decltype(n.CommInitRank))dlsym(h, "ncclCommInitRank");
    n.CommDestroy = (decltype(n.CommDestroy))dlsym(h, "ncclCommDestroy");
    n.AllGather = (decltype(n.AllGather))dlsym(h, "ncclAllGather");
    n.GetErrorString = (decltype(n.GetErrorString))dlsym(h, "ncclGetErrorString");
    n.GetVersion = (decltype(n.GetVersion))dlsym(h, "ncclGetVersion");
    if (!n.GetUniqueId || !n.CommInitRank || !n.CommDestroy || !n.AllGather || !n.GetErrorString)
        return fail(CGB_ERR_NCCL, "libnccl lacks a required symbol");
    g_nccl = n;
    return CGB_OK;
}
} // namespace

#define NK(call)                                                                                   \
    do {                                                                                           \
        int r_ = (call);                                                                           \
        if (r_ != 0)                                                                               \
            return fail(CGB_ERR_NCCL, "%s failed: %s", #call, g_nccl.GetErrorString(r_));          \
    } while (0)

// ------------------------------------------------------------------ context
static_assert(kMaxRhs == CGB_MAX_RHS, "one limit of columns");

// One solve in progress: the single solve's (cgb_ctx::run) or the block solve's (BlockSolve::run)
struct SolveRun {
    int nrhs = 1;
    long long max_iter = 0, launched = 0;
    double tol = 1e-10, loop_ms = 0.0;
    State *st = nullptr;            // [nrhs]
    double *hist = nullptr;         // column j's r'r history at hist + j * hist_ld; null: not kept
    long long hist_ld = 0;
};

// A loop graph and what its captured kernel arguments bake in.  A context caches four: the host loops
// of the single and the block solve (cgb_iterate) and the device loops of both (cgb_solve_device,
// cgb_solve_block_device).  `gen` is cgb_ctx::graph_gen at capture.
struct GraphKey {
    int len = 0, nrhs = 0, pdl = 0;
    double tol = 0.0;
    const double *hist = nullptr;
    long long gen = -1;
};
struct CachedGraph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    GraphKey key;
    int pdl_used = -1;              // device loops: 1 the bodies keep the programmatic dependent launches, 0 not
};

// Block solve (cgb_solve_block_begin): its own buffers and States, allocated on the first block solve
// and never shared with the single solve.
struct BlockSolve {
    int cap = 0;                    // columns the vector buffers hold
    double *x = nullptr, *r = nullptr, *p = nullptr, *b = nullptr; // [cap][ld]
    double *ap = nullptr;           // [cap][slot]
    double *rrpart = nullptr, *papart = nullptr; // [cap][nchunks]
    unsigned int *arrive = nullptr; // [cap][2] arrival counters, then the count of converged columns
    double *hist_buf = nullptr;     // [cap][hist_cap]
    long long hist_cap = 0;
    bool active = false;
    SolveRun run;                   // st: [cap]
};

struct cgb_ctx {
    long long n = 0, ld = 0, rows = 0, row0 = 0, n_loc = 0, maxrows = 0, nchunks = 0;
    int rank = 0, world = 1, device = 0, sm_count = 0;
    int variant = 0, nblk = 0;
    long long slot = 0, slot_cap = 0;
    int opt_graph = 1, opt_profile = 0, opt_num_threads = 0, opt_block_width = 0, opt_transposed = 1;
    int opt_compat = 0;            // 1: the reference's mat-vec topologies (compat.cu)
    double *compat_part = nullptr; // chunk partials of the compat mat-vec
    size_t compat_part_cap = 0;
    int poll_every = 16, graph_unroll = 16, opt_pdl = 1, opt_l2_prefetch = 4, opt_l2_ramp = 2;
    long long graph_replays = 0;   // graph launches since creation ("graph_replays", read-only option)
    long long graph_captures = 0;  // loop graphs captured and instantiated ("graph_captures", read-only option)
    int opt_balance = 1;           // persistent kernel: re-balance the rows between the CTAs from measured speeds
    long long aux_stride = 0;      // entries of one parity of the local LL side buffer
    int opt_schedule = 1;          // 1: persistent cooperative kernel (persist.cu) when usable, 0: CUDA graph of 4 kernels per iteration
    long long spin_timeout_ms = 20000; // bound of the device-side waits on other CTAs / ranks
    PersistSync *psync = nullptr;
    uint4 *rr_ll = nullptr;        // [2][nchunks] LL entries of the r'r chunk partials
    int smem_optin = 0;            // cudaDevAttrMaxSharedMemoryPerBlockOptin
    long long persist_launches = 0;
    int opt_loopback = 0;          // profiling: this rank plays every rank of the exchange (see "loopback")
    // diagnostic timelines (option "trace"): 0 = mat-vec, 1 = update_xr, 2 = update_p
    unsigned long long *trace_buf[3] = {nullptr, nullptr, nullptr};
    unsigned int *trace_cnt[3] = {nullptr, nullptr, nullptr};
    int trace_blocks[3] = {0, 0, 0}; // capacity in blocks per launch
    int trace_cap = 0;

    int storage = 0;               // 0: dense rows x ld shard `A`, 1: CSR shard `csr` (cgb_create_csr)
    CsrShard csr;
    AsmPlan plan;                  // the last cgb_assemble_coo's, while its matrix is the context's (start: null)
    unsigned int *arrive = nullptr; // CSR: arrival counters of the once-per-iteration vector phase
    double *A = nullptr, *p = nullptr, *r = nullptr, *x = nullptr, *b = nullptr;
    int2 *env = nullptr;           // dense: [first, last + 1) of the non-zero columns of every local row,
                                   // rebuilt after every write of A (the mat-vecs stream only these windows)
    double *apx = nullptr, *rrpart = nullptr, *papart = nullptr, *scratch = nullptr, *sink = nullptr;
    // apx: plain gather buffer [world][slot_cap] doubles.  ll: fused-mode LL buffers
    // [2][world][slot_cap] x 16 B, the allocation peers map; ctl: local control words.
    long long bufstride = 0;
    size_t ll_bytes = 0;
    uint4 *ll = nullptr;
    Ctl *ctl = nullptr;
    uint4 *peer_ll[kMaxWorld] = {};
    void *ipc_opened[kMaxWorld] = {};
    bool p2p_ready = false;
    int opt_exchange = 0; // 0 = ncclAllGather, 1 = fused peer stores
    long long hist_cap = 0;        // doubles at run.hist
    // mapped pinned flag: [0] the stop test fired (raised by the solve in progress, single or block) or,
    // negative, a device-side wait timed out; [1..6] context of a timeout report
    int *h_done = nullptr, *d_hdone = nullptr;
    double *h_pin = nullptr;                   // pinned staging for small D2H reads

    cudaStream_t stream = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev_batch[2] = {nullptr, nullptr};
    std::vector<cudaEvent_t> prof_ev;
    ncclComm_t comm = nullptr;

    bool matrix_set = false, rhs_set = false;
    bool in_solve = false;         // a single or (blk.active) a block solve is between begin and end
    long long kernel_launches = 0;
    SolveRun run;                  // the single solve; run.hist is the host API's history (null: not kept)
    double prof_gemv_ms = 0.0;
    long long prof_gemv_n = 0;
    BlockSolve blk;

    // Bumped whenever something a captured loop graph bakes in, other than its key's own fields, may have
    // changed: an option, a buffer that moved, a CSR matrix build (it reallocates col / val)
    long long graph_gen = 0;
    CachedGraph graph_single, graph_block, loop_single, loop_block; // host loops, device loops

    // device solves (cgb_solve_device, cgb_solve_block_device); allocated on the first one
    LoopCtl *loopctl = nullptr;    // the loop's body limit, bodies issued, start stamp
    double *dev_hist = nullptr;    // cgb_solve_device's r'r history (the host solve's stays its own)
    long long dev_hist_cap = 0;
    cudaEvent_t ev_dev[2] = {nullptr, nullptr}; // caller's stream -> ctx stream, and back
};

namespace {

// How a solve's loop kernels launch: the r'r history they write (nullable), the mapped host flag they
// raise when the stop test fires (null in a device solve: nobody polls it, and a host solve queued
// behind it resets it from the host) and whether they chain by programmatic dependent launch.
struct Mode {
    double *hist;
    int *host_done;
    int pdl;
};

// the host API's single solve ("profile" times each mat-vec between events: no PDL)
Mode host_mode(const cgb_ctx *c) { return {c->run.hist, c->d_hdone, (c->opt_pdl && !c->opt_profile) ? 1 : 0}; }

int use_device(cgb_ctx *c)
{
    if (!c) return fail(CGB_ERR_INVALID, "null context");
    CK(cudaSetDevice(c->device));
    return CGB_OK;
}

// Entries that arrive in every slot of the gather buffer: the largest shard's -- or, in "loopback" (this rank
// plays every rank of the exchange with its OWN rows: cgb_autotune, profiling), this rank's row count; reads
// past them are clamped, else a rank with fewer rows than the last one would wait for entries nobody stores
long long loopback_cap(const cgb_ctx *c)
{
    if (!c->opt_loopback) return c->maxrows > 0 ? c->maxrows : 1;
    return c->rows > 0 ? c->rows : 1;
}

// the fused exchange's peer buffers; in "loopback" every "peer" is this rank's own buffer, shifted so
// that slot g is hit
void peer_pointers(const cgb_ctx *c, uint4 **peer)
{
    for (int g = 0; g < kMaxWorld; ++g) peer[g] = c->peer_ll[g];
    if (c->opt_loopback)
        for (int g = 0; g < c->world; ++g) peer[g] = c->ll + ((long long)g - c->rank) * c->slot;
}

Gather make_gather(const cgb_ctx *c)
{
    Gather g;
    g.n_loc = c->n_loc > 0 ? c->n_loc : 1;
    g.slot = c->slot;
    g.maxrows = c->maxrows;
    g.loc_cap = loopback_cap(c);
    g.world = c->world;
    g.nblk = c->nblk;
    g.bufstride = c->bufstride;
    g.ll = c->ll;
    g.ctl = c->ctl;
    g.p2p = (c->world > 1 && c->opt_exchange == 1) ? 1 : 0;
    g.spin_ns = (unsigned long long)c->spin_timeout_ms * 1000000ULL;
    g.host_err = c->d_hdone;
    return g;
}

Trace make_trace(const cgb_ctx *c, int which, int blocks)
{
    Trace t;
    t.buf = c->trace_buf[which];
    t.cnt = c->trace_cnt[which];
    t.cap = c->trace_cap;
    t.nblk = blocks;
    if (blocks > c->trace_blocks[which]) t.buf = nullptr; // cannot happen: sized for the largest grid
    return t;
}

GemvArgs make_gemv_args(const cgb_ctx *c, const double *v, int advance, const Mode &m)
{
    GemvArgs a;
    memset(&a, 0, sizeof a);
    a.A = c->A;
    a.env = c->env;
    a.csr_rp = c->csr.rp;
    a.csr_col = c->csr.col;
    a.csr_val = c->csr.val;
    a.v = v;
    a.base = c->apx;
    a.ctl = c->ctl;
    a.bufstride = c->bufstride;
    a.slot_off = (long long)c->rank * c->slot;
    a.rank = c->rank;
    a.world = c->world;
    a.p2p = (c->world > 1 && c->opt_exchange == 1) ? 1 : 0;
    peer_pointers(c, a.peer_ll);
    a.ld = c->ld;
    a.rows = c->rows;
    a.row0 = c->row0;
    a.maxrows = c->maxrows;
    a.st = c->run.st;
    a.rrpart = c->rrpart;
    a.nchunks = c->nchunks;
    a.hist = m.hist;
    a.advance = advance;
    a.pdl = (advance && m.pdl) ? 1 : 0; // only inside the CG loop
    a.l2_prefetch = a.pdl ? c->opt_l2_prefetch : 0;
    if (c->trace_cap > 0 && advance) a.trace = make_trace(c, 0, c->nblk);
    return a;
}

VecArgs make_vec_args(const cgb_ctx *c, const Mode &m)
{
    VecArgs a;
    memset(&a, 0, sizeof a);
    a.x = c->x;
    a.r = c->r;
    a.p = c->p;
    a.b = c->b;
    a.apx = c->apx;
    a.rrpart = c->rrpart;
    a.papart = c->papart;
    a.st = c->run.st;
    a.host_done = m.host_done;
    a.hist = m.hist;
    a.g = make_gather(c);
    a.n = c->n;
    a.tol = c->run.tol;
    a.pdl = m.pdl;
    a.arrive = c->arrive;
    if (c->trace_cap > 0) {
        a.trace_xr = make_trace(c, 1, (int)c->nchunks);
        a.trace_p = make_trace(c, 2, (int)c->nchunks);
    }
    return a;
}

void set_variant(cgb_ctx *c, int v)
{
    c->variant = v;
    c->nblk = c->sm_count * gemv_variant(v).ctas_per_sm;
    c->slot = (c->maxrows + 1) & ~1LL;
}

void free_trace(cgb_ctx *c)
{
    for (int w = 0; w < 3; ++w) {
        if (c->trace_buf[w]) cudaFree(c->trace_buf[w]);
        if (c->trace_cnt[w]) cudaFree(c->trace_cnt[w]);
        c->trace_buf[w] = nullptr;
        c->trace_cnt[w] = nullptr;
        c->trace_blocks[w] = 0;
    }
    c->trace_cap = 0;
}

// `n` States as a solve starts them: zero, iter = -1
int reset_states(cgb_ctx *c, State *st, int n)
{
    State s0[kMaxRhs];
    memset(s0, 0, sizeof s0);
    for (State &s : s0) s.iter = -1;
    CK(cudaMemcpyAsync(st, s0, (size_t)n * sizeof(State), cudaMemcpyHostToDevice, c->stream));
    return CGB_OK;
}

// ---- cached loop graphs ---------------------------------------------------------------------
// Loop bodies in a loop graph: a batch between two looks at the stop flag is poll_every bodies, and a
// longer graph could never be replayed
int graph_len_wanted(const cgb_ctx *c) { return c->graph_unroll < c->poll_every ? c->graph_unroll : c->poll_every; }

GraphKey graph_key(const cgb_ctx *c, int nrhs, double tol, const double *hist)
{
    return GraphKey{graph_len_wanted(c), nrhs, c->opt_pdl, tol, hist, c->graph_gen};
}

bool holds(const CachedGraph &g, const GraphKey &k)
{
    return g.exec && g.key.len == k.len && g.key.nrhs == k.nrhs && g.key.pdl == k.pdl && g.key.tol == k.tol &&
           g.key.hist == k.hist && g.key.gen == k.gen;
}

void drop(CachedGraph &g)
{
    if (g.exec) cudaGraphExecDestroy(g.exec);
    if (g.graph) cudaGraphDestroy(g.graph);
    g.exec = nullptr;
    g.graph = nullptr;
}

void drop_graphs(cgb_ctx *c)
{
    for (CachedGraph *g : {&c->graph_single, &c->graph_block, &c->loop_single, &c->loop_block}) drop(*g);
}

// Captures into `g` the launches `enqueue` makes on c->stream, after the node `dep` (nullable);
// *tail (nullable) = the last node captured.  The capture always ends, whatever fails.
template <class F>
int capture_into(cgb_ctx *c, cudaGraph_t g, cudaGraphNode_t dep, F enqueue, cudaGraphNode_t *tail)
{
    CK(cudaStreamBeginCaptureToGraph(c->stream, g, dep ? &dep : nullptr, nullptr, dep ? 1 : 0,
                                     cudaStreamCaptureModeThreadLocal));
    int rc = enqueue();
    if (rc == CGB_OK && tail) {
        cudaStreamCaptureStatus cs;
        const cudaGraphNode_t *deps = nullptr;
        size_t nd = 0;
        cudaError_t e = cudaStreamGetCaptureInfo(c->stream, &cs, nullptr, nullptr, &deps, &nd);
        if (e != cudaSuccess) rc = fail(CGB_ERR_CUDA, "cudaStreamGetCaptureInfo: %s", cudaGetErrorString(e));
        else if (nd != 1) rc = fail(CGB_ERR_CUDA, "a captured loop control kernel left %zu tail nodes", nd);
        else *tail = deps[0];
    }
    cudaGraph_t out = nullptr;
    cudaError_t e = cudaStreamEndCapture(c->stream, &out);
    if (rc) return rc;
    CK(e);
    return CGB_OK;
}

// `g` captured anew by `build(graph)` into a created graph, instantiated, and keyed with `key`
template <class F>
int rebuild(cgb_ctx *c, CachedGraph &g, const GraphKey &key, F build)
{
    drop(g);
    CK(cudaGraphCreate(&g.graph, 0));
    const long long before = c->kernel_launches;
    int rc = build(g.graph);
    c->kernel_launches = before; // capture launches nothing
    if (rc == CGB_OK) {
        const cudaError_t e = cudaGraphInstantiate(&g.exec, g.graph, 0);
        if (e != cudaSuccess) rc = fail(CGB_ERR_CUDA, "instantiating a loop graph failed: %s", cudaGetErrorString(e));
    }
    if (rc) {
        drop(g);
        return rc;
    }
    g.key = key;
    c->graph_captures += 1;
    return CGB_OK;
}

// the mat-vec and, for world > 1, the gather of its result
int launch_matvec(cgb_ctx *c, const double *v, int advance, int variant, const Mode &m)
{
    if (c->opt_compat) { // reference topologies, NUM_THREADS / BLOCK_WIDTH literal (single GPU)
        GemvArgs a = make_gemv_args(c, v, advance, m);
        a.pdl = 0;
        CK(launch_compat_matvec(a, c->nblk, c->opt_num_threads, c->opt_block_width, c->opt_transposed,
                                c->compat_part, c->stream));
        c->kernel_launches += 2;
        return CGB_OK;
    }
    const GemvArgs a = make_gemv_args(c, v, advance, m);
    if (c->storage == 1) CK(launch_spmv(a, c->sm_count, c->stream));
    else CK(gemv_variant(variant).launch(a, c->sm_count * gemv_variant(variant).ctas_per_sm, c->stream));
    c->kernel_launches += 1;
    return CGB_OK;
}

int launch_gather(cgb_ctx *c)
{
    if (c->world == 1) return CGB_OK;
    if (c->opt_exchange == 1) return CGB_OK; // fused into the mat-vec kernel (peer stores + flags)
    if (!c->comm) return fail(CGB_ERR_STATE, "world > 1 but neither cgb_comm_init nor cgb_exchange_import was called");
    NK(g_nccl.AllGather(c->apx + (long long)c->rank * c->slot, c->apx, (size_t)c->slot, kNcclDouble,
                        c->comm, c->stream));
    return CGB_OK;
}

// the three vector kernels of one iteration; CSR contexts compute every scalar once per iteration
int launch_vector_phase(cgb_ctx *c, const Mode &m)
{
    const VecArgs va = make_vec_args(c, m);
    if (c->storage == 1) {
        CK(launch_pap_alpha(va, c->stream));
        CK(launch_update_xr_once(va, c->stream));
        CK(launch_update_p_once(va, c->stream));
    } else {
        CK(launch_pap_partials(va, c->stream));                             // cg.cc:105
        CK(launch_update_xr(va, c->stream));                                // cg.cc:106-117
        CK(launch_update_p(va, c->stream));                                 // cg.cc:120-132
    }
    c->kernel_launches += 3;
    return CGB_OK;
}

int launch_iteration(cgb_ctx *c, const Mode &m)
{
    int rc = launch_matvec(c, c->p, 1, c->variant, m);                     // cg.cc:100-102
    if (rc) return rc;
    if ((rc = launch_gather(c))) return rc;                                 // cg.cc:135-136 (moved)
    return launch_vector_phase(c, m);
}

// ---- persistent schedule (persist.cu) ------------------------------------------------
// The persistent kernel exists for the tile shapes listed in persist.cu; it needs one CTA per SM,
// the fused exchange (or one rank), at most persist_max_chunks() vector chunks per CTA and the
// scratch for the block / chunk partials next to the tile ring in shared memory.
int persist_index(const cgb_ctx *c)
{
    const char *name = gemv_variant(c->variant).name;
    for (int i = 0; i < persist_variant_count(); ++i)
        if (strcmp(persist_variant(i).name, name) == 0) return i;
    return -1;
}

void persist_scratch(const cgb_ctx *c, int *scr_n)
{
    const long long scr = c->nchunks > c->nblk ? c->nchunks : c->nblk; // chunk partials / per-CTA timings
    *scr_n = (int)((scr + 1) & ~1LL);
}

// nullptr when the persistent schedule can run this context as configured, else the reason; `profile`:
// "profile" is in force (a device solve runs as if it were 0)
const char *persist_unusable(const cgb_ctx *c, bool profile)
{
    if (c->storage == 1) return "CSR storage";
    if (c->opt_compat) return "compat mat-vec";
    if (profile) return "profile mode (per-launch events)";
    if (c->world > 1 && c->opt_exchange != 1) return "ncclAllGather exchange";
    if (gemv_variant(c->variant).ctas_per_sm != 1) return "variant runs 2 CTAs per SM";
    const int pi = persist_index(c);
    if (pi < 0) return "no persistent instantiation of this tile shape";
    if (c->nchunks > (long long)persist_max_chunks() * c->nblk) return "N too large for the per-CTA vector chunks";
    int scr_n;
    persist_scratch(c, &scr_n);
    if (persist_variant(pi).smem_fixed() + (size_t)scr_n * 8 + 4096 > (size_t)c->smem_optin) // + static
        return "tile ring + scratch exceed shared memory";
    return nullptr;
}

int launch_persist(cgb_ctx *c, long long iters, const Mode &m)
{
    PersistArgs a;
    memset(&a, 0, sizeof a);
    a.A = c->A;
    a.env = c->env;
    a.x = c->x;
    a.r = c->r;
    a.p = c->p;
    a.rrpart = c->rrpart;
    peer_pointers(c, a.peer_ll);
    a.ll = c->ll;
    a.rr_ll = c->rr_ll;
    a.rr_stride = c->aux_stride;
    a.sync = c->psync;
    a.st = c->run.st;
    a.ctl = c->ctl;
    a.hist = m.hist;
    a.host_done = m.host_done;
    a.ld = c->ld;
    a.rows = c->rows;
    a.row0 = c->row0;
    a.n = c->n;
    a.maxrows = c->maxrows;
    a.n_loc = c->n_loc > 0 ? c->n_loc : 1;
    a.loc_cap = loopback_cap(c);
    a.slot = c->slot;
    a.bufstride = c->bufstride;
    a.slot_off = (long long)c->rank * c->slot;
    a.nchunks = c->nchunks;
    a.rank = c->rank;
    a.world = c->world;
    a.iters = (int)iters;
    a.l2_prefetch = c->opt_l2_prefetch;
    a.l2_ramp = c->opt_l2_ramp;
    a.balance = c->opt_balance;
    persist_scratch(c, &a.scr_n);
    a.tol = c->run.tol;
    a.spin_ns = (unsigned long long)c->spin_timeout_ms * 1000000ULL;
    if (c->trace_cap > 0) a.trace = make_trace(c, 0, c->nblk);
    CK(cudaMemsetAsync(c->psync, 0, sizeof(PersistSync), c->stream));
    CK(persist_variant(persist_index(c)).launch(a, c->nblk, c->stream));
    c->kernel_launches += 1;
    c->persist_launches += 1;
    return CGB_OK;
}

// ONE cooperative launch per 2^30 loop bodies (its count is an int); it leaves the loop on convergence by itself
int launch_persist_bodies(cgb_ctx *c, long long todo, const Mode &m)
{
    while (todo > 0) {
        const long long part = std::min<long long>(todo, 1 << 30);
        const int rc = launch_persist(c, part, m);
        if (rc) return rc;
        todo -= part;
    }
    return CGB_OK;
}

bool exchange_configured(const cgb_ctx *c)
{
    return c->world == 1 || (c->opt_exchange == 1 ? c->p2p_ready : c->comm != nullptr);
}

// Hooks that read the gathered result with memcpys: in fused mode first consume the running
// exchange into the plain buffer (this also advances the epoch, like every consumer kernel).
int collect_for_host(cgb_ctx *c)
{
    const Gather g = make_gather(c);
    if (g.p2p) {
        CK(launch_exchange_collect(c->apx, g, c->stream));
        c->kernel_launches += 1;
    }
    return CGB_OK;
}

// ---- the host loop (cgb_iterate) -------------------------------------------------------------
// Ends cgb_iterate's timed window: ev1, the wait for it -- a device-side wait that timed out is
// reported as such -- and the window's time added to the solve's
int end_window(cgb_ctx *c, SolveRun &run, float *ms)
{
    CK(cudaEventRecord(c->ev1, c->stream));
    cudaError_t e = cudaEventSynchronize(c->ev1);
    if (e != cudaSuccess) {
        const int code = *(volatile int *)c->h_done;
        if (code < 0)
            return fail(CGB_ERR_TIMEOUT, "a device-side wait (kind %d: 1 = an LL entry -- a peer rank's mat-vec rows or a chunk "
                        "partial, 4 = p chunks, 5 = tile for the consumers, 6 / 9 = row partition hand-over, 7 = free "
                        "pipeline stage, 8 = drain, 10 = column-window table) exceeded spin_timeout_ms = %lld: a rank is "
                        "missing or stuck (%s) [cta %d thread %d: %d %d %d %d]", -code, c->spin_timeout_ms,
                        cudaGetErrorString(e), c->h_done[1], c->h_done[2], c->h_done[3], c->h_done[4], c->h_done[5],
                        c->h_done[6]);
        CK(e);
    }
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, c->ev0, c->ev1));
    run.loop_ms += t;
    if (ms) *ms = t;
    return CGB_OK;
}

// Up to `todo` loop bodies of the solve in progress on the graph schedule, timed.  `body()` enqueues
// one body of `per_body` kernels.  Batches of poll_every bodies, each a replay of the cached graph `g`
// (when `graph` and its L bodies fit the batch) or single bodies; the mapped flag is read between
// batches, and the host keeps at most two batches in flight so that it never runs far ahead of it.
template <class F>
int host_loop(cgb_ctx *c, SolveRun &run, long long todo, bool graph, CachedGraph &g, int per_body, F body, float *ms)
{
    int rc;
    const GraphKey key = graph_key(c, run.nrhs, run.tol, run.hist);
    const bool replay = graph && todo >= key.len;
    if (replay && !holds(g, key)) {
        rc = rebuild(c, g, key, [&](cudaGraph_t gr) {
            return capture_into(c, gr, nullptr, [&]() -> int {
                int r = CGB_OK;
                for (int u = 0; u < key.len && r == CGB_OK; ++u) r = body();
                return r;
            }, nullptr);
        });
        if (rc) return rc;
    }
    // ncclAllGather mode: the collectives of a batch run on every rank or on none, so all
    // ranks must take the same stop decision -- wait for the batch just issued (the flag is
    // then the same on every rank) instead of looking one batch back.  The fused exchange
    // needs no such lockstep: launches after convergence communicate nothing.
    const bool lockstep = c->world > 1 && c->opt_exchange == 0;
    CK(cudaEventRecord(c->ev0, c->stream));
    long long issued = 0;
    int batch_idx = 0;
    while (issued < todo) {
        if (*(volatile int *)c->h_done) break; // converged: later launches would be no-ops
        const long long batch = std::min<long long>(c->poll_every, todo - issued);
        long long i = 0;
        while (i < batch) {
            if (replay && batch - i >= key.len) {
                CK(cudaGraphLaunch(g.exec, c->stream));
                c->kernel_launches += (long long)per_body * key.len;
                c->graph_replays += 1;
                i += key.len;
            } else {
                if ((rc = body())) return rc;
                i += 1;
            }
        }
        issued += batch;
        CK(cudaEventRecord(c->ev_batch[batch_idx & 1], c->stream));
        if (lockstep) CK(cudaEventSynchronize(c->ev_batch[batch_idx & 1]));
        else if (batch_idx >= 1) CK(cudaEventSynchronize(c->ev_batch[(batch_idx - 1) & 1]));
        ++batch_idx;
    }
    run.launched += issued;
    return end_window(c, run, ms);
}

// cgb_solve_end / cgb_solve_block_end after the finalize kernel: the States, each column's executed
// r'r history (to resid_hist + j * max_iter) and its cgb_solve_info
int collect_solve(cgb_ctx *c, const SolveRun &run, double *resid_hist, cgb_solve_info *info)
{
    State s[kMaxRhs];
    CK(cudaMemcpyAsync(s, run.st, (size_t)run.nrhs * sizeof(State), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    for (int j = 0; j < run.nrhs; ++j) {
        const long long executed = s[j].done ? s[j].iter + 1 : s[j].iter;
        if (resid_hist && executed > 0)
            CK(cudaMemcpyAsync(resid_hist + (size_t)j * run.max_iter, run.hist + (size_t)j * run.hist_ld,
                               (size_t)executed * 8, cudaMemcpyDeviceToHost, c->stream));
        if (info) {
            info[j].k = s[j].iter;
            info[j].converged = s[j].done;
            info[j].rsold = s[j].rsold;
            info[j].rsnew = s[j].rsnew;
            info[j].seconds = run.loop_ms * 1e-3;
            info[j].iterations = executed;
        }
    }
    CK(cudaStreamSynchronize(c->stream));
    return CGB_OK;
}

// ---- block solve ---------------------------------------------------------------------------
void free_block_vectors(cgb_ctx *c)
{
    BlockSolve &k = c->blk;
    double *bufs[] = {k.x, k.r, k.p, k.b, k.ap, k.rrpart, k.papart};
    for (double *p : bufs)
        if (p) cudaFree(p);
    if (k.run.st) cudaFree(k.run.st);
    if (k.arrive) cudaFree(k.arrive);
    k.x = k.r = k.p = k.b = k.ap = k.rrpart = k.papart = nullptr;
    k.run.st = nullptr;
    k.arrive = nullptr;
    k.cap = 0;
}

// buffers for nrhs columns and, with a history, max(max_iter, 1) entries per column; grows only
int size_block(cgb_ctx *c, int nrhs, long long max_iter, bool history)
{
    BlockSolve &k = c->blk;
    auto alloc = [&](void **p, size_t bytes) -> int {
        cudaError_t e = cudaMalloc(p, bytes);
        if (e == cudaSuccess) e = cudaMemsetAsync(*p, 0, bytes, c->stream);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return fail(e == cudaErrorMemoryAllocation ? CGB_ERR_NOMEM : CGB_ERR_CUDA, "block solve buffers: %s",
                        cudaGetErrorString(e));
        }
        return CGB_OK;
    };
    int rc = CGB_OK;
    const long long hist_need = max_iter > 0 ? max_iter : 1;
    if (nrhs > k.cap) {
        if (k.cap == 0) { // first block solve of this context
            CK(preload_spmv_block_kernels());
            CK(preload_vec_block_kernels());
        }
        c->graph_gen += 1; // the block graphs bake in the buffers
        free_block_vectors(c);
        const size_t vec = (size_t)nrhs * c->ld * sizeof(double);
        const size_t part = (size_t)nrhs * c->nchunks * sizeof(double);
        if ((rc = alloc((void **)&k.x, vec)) || (rc = alloc((void **)&k.r, vec)) || (rc = alloc((void **)&k.p, vec)) ||
            (rc = alloc((void **)&k.b, vec)) || (rc = alloc((void **)&k.ap, (size_t)nrhs * c->slot_cap * sizeof(double))) ||
            (rc = alloc((void **)&k.rrpart, part)) || (rc = alloc((void **)&k.papart, part)) ||
            (rc = alloc((void **)&k.run.st, (size_t)nrhs * sizeof(State))) ||
            (rc = alloc((void **)&k.arrive, (size_t)(2 * nrhs + 1) * sizeof(unsigned int)))) {
            free_block_vectors(c);
            return rc;
        }
        k.cap = nrhs;
        if (k.hist_buf) cudaFree(k.hist_buf); // its column stride follows from the new capacity
        k.hist_buf = nullptr;
        k.hist_cap = 0;
    }
    if (history && hist_need > k.hist_cap) {
        c->graph_gen += 1;
        if (k.hist_buf) cudaFree(k.hist_buf);
        k.hist_buf = nullptr;
        k.hist_cap = 0;
        if ((rc = alloc((void **)&k.hist_buf, (size_t)k.cap * hist_need * sizeof(double)))) return rc;
        k.hist_cap = hist_need;
    }
    return CGB_OK;
}

// the block solve's run for nrhs columns, after size_block
void start_block_run(cgb_ctx *c, int nrhs, long long max_iter, double tol, bool history)
{
    SolveRun &run = c->blk.run;
    run.nrhs = nrhs;
    run.max_iter = max_iter;
    run.tol = tol;
    run.launched = 0;
    run.loop_ms = 0.0;
    run.hist = history ? c->blk.hist_buf : nullptr;
    run.hist_ld = c->blk.hist_cap;
}

BlockArgs make_block_args(const cgb_ctx *c, const double *v, int advance, const Mode &m)
{
    const BlockSolve &k = c->blk;
    BlockArgs a;
    memset(&a, 0, sizeof a);
    a.rp = c->csr.rp;
    a.col = c->csr.col;
    a.val = c->csr.val;
    a.v = v;
    a.x = k.x;
    a.r = k.r;
    a.p = k.p;
    a.b = k.b;
    a.ap = k.ap;
    a.rrpart = k.rrpart;
    a.papart = k.papart;
    a.st = k.run.st;
    a.arrive = k.arrive;
    a.ndone = k.arrive + 2 * k.cap;
    a.host_done = m.host_done;
    a.hist = m.hist;
    a.n = c->n;
    a.ld = c->ld;
    a.rows = c->rows;
    a.slot = c->slot_cap;
    a.nchunks = c->nchunks;
    a.hist_ld = k.run.hist_ld;
    a.nrhs = k.run.nrhs;
    a.advance = advance;
    a.pdl = (advance && m.pdl) ? 1 : 0; // only inside the CG loop
    a.tol = k.run.tol;
    return a;
}

// mat-vec + the three vector kernels of one block iteration
int launch_block_iteration(cgb_ctx *c, const Mode &m)
{
    const BlockArgs a = make_block_args(c, c->blk.p, 1, m);
    CK(launch_spmv_block(a, c->sm_count, c->stream));
    CK(launch_pap_alpha_block(a, c->stream));
    CK(launch_update_xr_block(a, c->stream));
    CK(launch_update_p_block(a, c->stream));
    c->kernel_launches += 4;
    return CGB_OK;
}

// ---- device solves -------------------------------------------------------------------------
// Pointers a device solve takes: device memory of the context's GPU (or managed memory)
int check_device_ptr(const cgb_ctx *c, const void *p, const char *what)
{
    if (!p) return fail(CGB_ERR_INVALID, "null %s", what);
    cudaPointerAttributes a;
    cudaError_t e = cudaPointerGetAttributes(&a, p);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(CGB_ERR_INVALID, "%s is not a pointer CUDA knows (%s)", what, cudaGetErrorString(e));
    }
    if (a.type == cudaMemoryTypeManaged) return CGB_OK;
    if (a.type != cudaMemoryTypeDevice)
        return fail(CGB_ERR_INVALID, "%s is host memory: this call takes device pointers", what);
    if (a.device != c->device)
        return fail(CGB_ERR_INVALID, "%s lives on device %d, the context on device %d", what, a.device, c->device);
    return CGB_OK;
}

// The two events that order the context's stream after a caller's stream and back (device solves,
// cgb_set_matrix_csr, cgb_update_matrix_values); created on first use
int stream_events(cgb_ctx *c)
{
    for (cudaEvent_t &e : c->ev_dev)
        if (!e) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    return CGB_OK;
}

// The loop of a device solve as one graph (DESIGN 3.9), captured into `g`:
//   head -> WHILE { len loop bodies ; ctl } -> mid -> WHILE { 1 loop body ; ctl }
// head, mid and ctl are loop_ctl_kernel: each sets the condition of the WHILE node it precedes or
// runs in -- the stop test has not fired and the bodies issued so far leave room for the next
// body under max_iter.  So no loop body starts past max_iter, and the count of bodies issued is the
// host loop's (whole graphs of `len`, then single iterations), short of the no-op bodies the host
// issues after the stop test fired.  `body()` enqueues one loop body on c->stream.
template <class F>
int capture_loop(cgb_ctx *c, cudaGraph_t g, int len, const int *done, const unsigned int *ndone, int nrhs, F body)
{
    int rc = CGB_OK;
    cudaGraphNode_t tail = nullptr;
    for (int part = 0; part < 2 && rc == CGB_OK; ++part) {
        const int step = part == 0 ? len : 1;
        cudaGraphConditionalHandle h;
        CK(cudaGraphConditionalHandleCreate(&h, g, 0, cudaGraphCondAssignDefault));
        cudaGraphNode_t ctl = nullptr;
        rc = capture_into(c, g, tail, [&]() -> int {
            CK(launch_loop_ctl(c->loopctl, done, ndone, nrhs, h, 1, step, 0, part == 0 ? 1 : 0, c->stream));
            return CGB_OK;
        }, &ctl);
        if (rc) break;
        cudaGraphNodeParams p = {cudaGraphNodeTypeConditional};
        p.conditional.handle = h;
        p.conditional.type = cudaGraphCondTypeWhile;
        p.conditional.size = 1;
        CK(cudaGraphAddNode(&tail, g, &ctl, 1, &p));
        rc = capture_into(c, p.conditional.phGraph_out[0], nullptr, [&]() -> int {
            int r = CGB_OK;
            for (int u = 0; u < step && r == CGB_OK; ++u) r = body();
            if (r == CGB_OK) CK(launch_loop_ctl(c->loopctl, done, ndone, nrhs, h, 1, step, step, 0, c->stream));
            return r;
        }, nullptr);
    }
    return rc;
}

// A device solve's loop on the graph schedule, launched: the cached loop graph `d` when its key still
// holds, else a new capture.  The bodies (`body(mode)`, `per_body` kernels) are captured with
// programmatic dependent launches when "pdl" asks for them; should the driver refuse them inside a
// conditional body, they are captured without (CachedGraph::pdl_used, option "device_loop_pdl").
// Its kernels count as if the loop ran to max_iter: the host does not learn where it stops.
template <class F>
int launch_loop_graph(cgb_ctx *c, CachedGraph &d, const GraphKey &key, Mode m, const int *done,
                      const unsigned int *ndone, int per_body, long long max_iter, F body)
{
    if (!holds(d, key)) {
        auto build = [&](cudaGraph_t g) {
            return capture_loop(c, g, key.len, done, ndone, key.nrhs, [&]() { return body(m); });
        };
        int rc = rebuild(c, d, key, build);
        d.pdl_used = m.pdl;
        if (rc && m.pdl) {
            cudaGetLastError();
            m.pdl = 0;
            rc = rebuild(c, d, key, build);
            d.pdl_used = 0;
        }
        if (rc) return rc;
    }
    CK(cudaGraphLaunch(d.exec, c->stream));
    c->graph_replays += 1;
    c->kernel_launches += per_body * max_iter + 2 + max_iter / key.len + max_iter % key.len;
    return CGB_OK;
}

} // namespace

// ------------------------------------------------------------------ library
extern "C" int cgb_abi_version(void) { return CGB_ABI_VERSION; }
extern "C" const char *cgb_last_error(void) { return g_err; }

extern "C" int cgb_device_count(int *count)
{
    if (!count) return fail(CGB_ERR_INVALID, "null count");
    *count = 0;
    CK(cudaGetDeviceCount(count));
    return CGB_OK;
}

extern "C" int cgb_partition(int64_t n, int psize, int64_t *start_rows, int64_t *num_rows)
{
    if (n < 0 || psize < 1 || !start_rows || !num_rows) return fail(CGB_ERR_INVALID, "bad partition arguments");
    // partition_matrix, code/MPI/cg.cc:236-268
    const int64_t n_loc = n / psize;
    int64_t i0 = 0;
    for (int r = 0; r < psize - 1; ++r) {
        start_rows[r] = i0;
        num_rows[r] = n_loc;
        i0 += n_loc;
    }
    start_rows[psize - 1] = i0;
    num_rows[psize - 1] = n - i0;
    return CGB_OK;
}

extern "C" int cgb_gemv_variant_count(void) { return gemv_variant_count(); }
extern "C" const char *cgb_gemv_variant_name(int v)
{
    return (v >= 0 && v < gemv_variant_count()) ? gemv_variant(v).name : nullptr;
}

// ------------------------------------------------------------------ context
// cgb_create / cgb_create_csr: everything but the shard is the same
static int create_ctx(int64_t n, int rank, int world, int device, int storage, cgb_ctx **out)
{
    if (!out) return fail(CGB_ERR_INVALID, "null out");
    *out = nullptr;
    if (n < 1) return fail(CGB_ERR_INVALID, "n must be >= 1 (got %lld)", (long long)n);
    if (world < 1 || world > kMaxWorld || rank < 0 || rank >= world)
        return fail(CGB_ERR_INVALID, "bad rank/world %d/%d (world <= %d)", rank, world, kMaxWorld);
    if (n < world) return fail(CGB_ERR_INVALID, "n (%lld) < world (%d)", (long long)n, world);
    if (storage == 1 && n > INT32_MAX)
        return fail(CGB_ERR_INVALID, "CSR storage keeps 32-bit column indices: n must be <= %d", INT32_MAX);
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (ndev == 0) return fail(CGB_ERR_NO_DEVICE, "no CUDA device");
    if (device < 0 || device >= ndev) return fail(CGB_ERR_INVALID, "device %d out of range (%d)", device, ndev);
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10 || prop.minor != 0) // sm_100a SASS only: arch-specific, no forward-compatible PTX
        return fail(CGB_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a (B200) only",
                    device, prop.major, prop.minor);

    cgb_ctx *c = new (std::nothrow) cgb_ctx;
    if (!c) return fail(CGB_ERR_NOMEM, "out of host memory");
    c->n = n;
    c->ld = (n + 15) & ~15LL;
    c->rank = rank;
    c->world = world;
    c->device = device;
    c->storage = storage;
    c->sm_count = prop.multiProcessorCount;
    if (const char *e = getenv("CGB_SPIN_TIMEOUT_MS")) { // default of the option "spin_timeout_ms"
        const long long v = atoll(e);
        if (v >= 1 && v <= 3600000) c->spin_timeout_ms = v;
    }
    std::vector<int64_t> start(world), num(world);
    cgb_partition(n, world, start.data(), num.data());
    c->row0 = start[rank];
    c->rows = num[rank];
    c->n_loc = n / world;
    c->maxrows = num[world - 1];
    c->nchunks = (n + kChunk - 1) / kChunk;
    c->slot_cap = (c->maxrows + 1) & ~1LL;
    set_variant(c, 0);

    auto bail = [&](int code) {
        cgb_destroy(c);
        return code;
    };
#define CKB(call)                                                                                  \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess)                                                                     \
            return bail(fail(e_ == cudaErrorMemoryAllocation ? CGB_ERR_NOMEM : CGB_ERR_CUDA,       \
                             "%s failed: %s", #call, cudaGetErrorString(e_)));                     \
    } while (0)
    CKB(cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking));
    CKB(cudaEventCreate(&c->ev0));
    CKB(cudaEventCreate(&c->ev1));
    CKB(cudaEventCreateWithFlags(&c->ev_batch[0], cudaEventDisableTiming));
    CKB(cudaEventCreateWithFlags(&c->ev_batch[1], cudaEventDisableTiming));
    const size_t vec_bytes = (size_t)c->ld * sizeof(double);
    if (storage == 1) {
        CKB(cudaMalloc(&c->csr.rp, (size_t)(c->rows + 1) * sizeof(long long)));
        CKB(cudaMemsetAsync(c->csr.rp, 0, (size_t)(c->rows + 1) * sizeof(long long), c->stream));
        CKB(cudaMalloc(&c->arrive, 2 * sizeof(unsigned int)));
        CKB(cudaMemsetAsync(c->arrive, 0, 2 * sizeof(unsigned int), c->stream));
    } else {
        CKB(cudaMalloc(&c->A, (size_t)c->rows * c->ld * sizeof(double)));
        CKB(cudaMemsetAsync(c->A, 0, (size_t)c->rows * c->ld * sizeof(double), c->stream));
        CKB(cudaMalloc(&c->env, (size_t)(c->rows > 0 ? c->rows : 1) * sizeof(int2)));
        CKB(cudaMemsetAsync(c->env, 0, (size_t)(c->rows > 0 ? c->rows : 1) * sizeof(int2), c->stream)); // all rows empty
    }
    CKB(cudaMalloc(&c->p, vec_bytes));
    CKB(cudaMalloc(&c->r, vec_bytes));
    CKB(cudaMalloc(&c->x, vec_bytes));
    CKB(cudaMalloc(&c->b, vec_bytes));
    c->bufstride = (long long)c->world * c->slot_cap;
    CKB(cudaMalloc(&c->apx, (size_t)c->bufstride * sizeof(double)));
    CKB(cudaMalloc(&c->ctl, sizeof(Ctl)));
    {   // LL gather buffers: the fused exchange (world > 1) and the persistent schedule (any world)
        c->ll_bytes = (size_t)2 * c->bufstride * sizeof(uint4);
        CKB(cudaMalloc(&c->ll, c->ll_bytes));
        CKB(cudaMemsetAsync(c->ll, 0, c->ll_bytes, c->stream)); // tag 0 is never used
        c->peer_ll[rank] = c->ll;
    }
    c->aux_stride = 2 * c->nchunks + 2LL * c->sm_count; // [r'r | p'Ap chunk partials | per-CTA times]
    CKB(cudaMalloc(&c->rr_ll, (size_t)2 * c->aux_stride * sizeof(uint4)));
    CKB(cudaMemsetAsync(c->rr_ll, 0, (size_t)2 * c->aux_stride * sizeof(uint4), c->stream));
    CKB(cudaMalloc(&c->psync, sizeof(PersistSync)));
    CKB(cudaMemsetAsync(c->psync, 0, sizeof(PersistSync), c->stream));
    CKB(cudaDeviceGetAttribute(&c->smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
    CKB(cudaMemsetAsync(c->ctl, 0, sizeof(Ctl), c->stream));
    CKB(cudaMalloc(&c->rrpart, (size_t)c->nchunks * sizeof(double)));
    CKB(cudaMalloc(&c->papart, (size_t)c->nchunks * sizeof(double)));
    CKB(cudaMemsetAsync(c->papart, 0, (size_t)c->nchunks * sizeof(double), c->stream));
    CKB(cudaMalloc(&c->scratch, (size_t)(3 * c->nchunks + 8) * sizeof(double)));
    CKB(cudaMalloc(&c->sink, 64));
    CKB(cudaMalloc(&c->run.st, sizeof(State)));
    CKB(cudaHostAlloc(&c->h_done, 8 * sizeof(int), cudaHostAllocMapped)); // [0] flag, [1..6] context of a timeout report
    CKB(cudaHostGetDevicePointer(&c->d_hdone, c->h_done, 0));
    CKB(cudaHostAlloc(&c->h_pin, 64 * sizeof(double), cudaHostAllocDefault));
    *c->h_done = 0;
    CKB(cudaMemsetAsync(c->p, 0, vec_bytes, c->stream));
    CKB(cudaMemsetAsync(c->r, 0, vec_bytes, c->stream));
    CKB(cudaMemsetAsync(c->x, 0, vec_bytes, c->stream));
    CKB(cudaMemsetAsync(c->b, 0, vec_bytes, c->stream));
    CKB(cudaMemsetAsync(c->apx, 0, (size_t)c->bufstride * sizeof(double), c->stream));
    CKB(cudaMemsetAsync(c->rrpart, 0, (size_t)c->nchunks * sizeof(double), c->stream));
    CKB(cudaMemsetAsync(c->run.st, 0, sizeof(State), c->stream));
    CKB(cudaStreamSynchronize(c->stream));
    CKB(preload_vec_kernels());
    if (storage == 1) {
        CKB(preload_spmv_kernels());
    } else {
        CKB(gemv_variant(c->variant).preload());
        if (persist_index(c) >= 0) CKB(persist_variant(persist_index(c)).preload());
    }
#undef CKB
    *out = c;
    return CGB_OK;
}

extern "C" int cgb_create(int64_t n, int rank, int world, int device, cgb_ctx **out)
{
    return create_ctx(n, rank, world, device, 0, out);
}

extern "C" int cgb_create_csr(int64_t n, int rank, int world, int device, cgb_ctx **out)
{
    return create_ctx(n, rank, world, device, 1, out);
}

extern "C" int cgb_destroy(cgb_ctx *c)
{
    if (!c) return CGB_OK;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    drop_graphs(c);
    if (c->comm && g_nccl.CommDestroy) g_nccl.CommDestroy(c->comm);
    for (cudaEvent_t e : c->prof_ev) cudaEventDestroy(e);
    for (void *p : c->ipc_opened)
        if (p) cudaIpcCloseMemHandle(p);
    double *bufs[] = {c->A, c->p, c->r, c->x, c->b, c->apx, c->rrpart, c->papart, c->scratch, c->run.hist, c->sink};
    for (double *p : bufs)
        if (p) cudaFree(p);
    if (c->run.st) cudaFree(c->run.st);
    if (c->env) cudaFree(c->env);
    if (c->csr.rp) cudaFree(c->csr.rp);
    if (c->csr.col) cudaFree(c->csr.col);
    if (c->csr.val) cudaFree(c->csr.val);
    asm_plan_free(&c->plan);
    if (c->arrive) cudaFree(c->arrive);
    if (c->compat_part) cudaFree(c->compat_part);
    free_trace(c);
    if (c->ll) cudaFree(c->ll);
    if (c->psync) cudaFree(c->psync);
    if (c->rr_ll) cudaFree(c->rr_ll);
    if (c->ctl) cudaFree(c->ctl);
    if (c->h_done) cudaFreeHost(c->h_done);
    if (c->h_pin) cudaFreeHost(c->h_pin);
    free_block_vectors(c);
    if (c->blk.hist_buf) cudaFree(c->blk.hist_buf);
    if (c->loopctl) cudaFree(c->loopctl);
    if (c->dev_hist) cudaFree(c->dev_hist);
    for (cudaEvent_t e : c->ev_dev)
        if (e) cudaEventDestroy(e);
    if (c->ev0) cudaEventDestroy(c->ev0);
    if (c->ev1) cudaEventDestroy(c->ev1);
    for (cudaEvent_t e : c->ev_batch)
        if (e) cudaEventDestroy(e);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
    return CGB_OK;
}

extern "C" int cgb_comm_unique_id(void *id_out)
{
    if (!id_out) return fail(CGB_ERR_INVALID, "null id");
    int rc = load_nccl();
    if (rc) return rc;
    ncclUniqueId id;
    NK(g_nccl.GetUniqueId(&id));
    memcpy(id_out, &id, sizeof id);
    return CGB_OK;
}

extern "C" int cgb_comm_init(cgb_ctx *c, const void *id_in)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->world == 1) return CGB_OK;
    if (!id_in) return fail(CGB_ERR_INVALID, "null id");
    if (c->comm) return fail(CGB_ERR_STATE, "communicator already initialised");
    if ((rc = load_nccl())) return rc;
    ncclUniqueId id;
    memcpy(&id, id_in, sizeof id);
    NK(g_nccl.CommInitRank(&c->comm, c->world, id, c->rank));
    return CGB_OK;
}

// ---- fused exchange wiring -------------------------------------------------------------
namespace {
struct XchBlob {
    uint64_t magic;
    int32_t pid, device, rank, world;
    uint64_t ptr, bytes;
    cudaIpcMemHandle_t handle;
};
static_assert(sizeof(XchBlob) <= CGB_EXCHANGE_BLOB_BYTES, "exchange blob too large");
constexpr uint64_t kXchMagic = 0x6367623230307832ULL;
} // namespace

extern "C" int cgb_exchange_export(cgb_ctx *c, void *blob_out)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (!blob_out) return fail(CGB_ERR_INVALID, "null blob");
    XchBlob b;
    memset(&b, 0, sizeof b);
    b.magic = kXchMagic;
    b.pid = (int32_t)getpid();
    b.device = c->device;
    b.rank = c->rank;
    b.world = c->world;
    b.ptr = (uint64_t)(uintptr_t)c->ll;
    b.bytes = c->ll_bytes;
    if (c->ll) CK(cudaIpcGetMemHandle(&b.handle, c->ll));
    memset(blob_out, 0, CGB_EXCHANGE_BLOB_BYTES);
    memcpy(blob_out, &b, sizeof b);
    return CGB_OK;
}

extern "C" int cgb_exchange_import(cgb_ctx *c, const void *blobs)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->world == 1) return CGB_OK;
    if (!blobs) return fail(CGB_ERR_INVALID, "null blobs");
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (c->p2p_ready) return fail(CGB_ERR_STATE, "exchange already imported");
    const char *base = static_cast<const char *>(blobs);
    for (int g = 0; g < c->world; ++g) {
        XchBlob b;
        memcpy(&b, base + (size_t)g * CGB_EXCHANGE_BLOB_BYTES, sizeof b);
        if (b.magic != kXchMagic || b.rank != g || b.world != c->world || b.bytes != c->ll_bytes)
            return fail(CGB_ERR_INVALID, "exchange blob %d does not match this context "
                        "(rank %d world %d bytes %llu)", g, b.rank, b.world, (unsigned long long)b.bytes);
        if (g == c->rank) continue;
        void *ptr = nullptr;
        if (b.pid == (int32_t)getpid()) { // same process (threads): plain peer access
            if (b.device != c->device) {
                int can = 0;
                CK(cudaDeviceCanAccessPeer(&can, c->device, b.device));
                if (!can) return fail(CGB_ERR_CUDA, "device %d cannot access peer %d", c->device, b.device);
                cudaError_t e = cudaDeviceEnablePeerAccess(b.device, 0);
                if (e == cudaErrorPeerAccessAlreadyEnabled) cudaGetLastError();
                else CK(e);
            }
            ptr = (void *)(uintptr_t)b.ptr;
        } else {
            CK(cudaIpcOpenMemHandle(&ptr, b.handle, cudaIpcMemLazyEnablePeerAccess));
            c->ipc_opened[g] = ptr;
        }
        c->peer_ll[g] = static_cast<uint4 *>(ptr);
    }
    c->p2p_ready = true;
    c->opt_exchange = 1;
    c->graph_gen += 1;
    return CGB_OK;
}

// ------------------------------------------------------------------ inputs
namespace {

// A local CSR a builder stages for install_matrix.  What it holds when it goes out of scope is freed: the
// staged arrays after a refusal or an error, the context's previous ones after an install that adopted it.
struct StagedCsr : CsrShard {
    ~StagedCsr()
    {
        cudaFree(rp);
        cudaFree(col);
        cudaFree(val);
    }
};

// cgb_assemble_coo's plan until install_matrix adopts it
struct StagedPlan : AsmPlan {
    ~StagedPlan() { asm_plan_free(this); }
};

// The one place a built matrix becomes the context's.  `m` is this rank's validated local CSR in device
// memory: rp rebased to 0, columns ascending and unique per row, explicit zeros kept.  A CSR context adopts
// it: a builder's staging (`staged`) is swapped in, a caller's arrays are copied.  The loop graphs bake in
// col / val, which move, so the generation is bumped.  A dense context densifies it into A (the whole
// rows x ld block is zeroed first) and rebuilds every row's envelope; its graphs bake in A and env, which
// stay where they are, so its generation is not bumped.  The previous matrix's assembly plan goes; `plan`
// (cgb_assemble_coo's, of `m`) becomes the context's, on a dense context with m's rp / col to find A's cells.
int install_matrix(cgb_ctx *c, CsrShard &m, bool staged, AsmPlan *plan = nullptr)
{
    c->matrix_set = false; // until the install completes
    asm_plan_free(&c->plan);
    if (c->storage == 1) {
        StagedCsr copy;
        if (!staged) {
            CK(cudaMalloc(&copy.rp, (size_t)(c->rows + 1) * sizeof(long long)));
            CK(csr_alloc_entries(&copy, m.nnz));
            CK(cudaMemcpyAsync(copy.rp, m.rp, (size_t)(c->rows + 1) * sizeof(long long), cudaMemcpyDeviceToDevice,
                               c->stream));
            if (m.nnz > 0) {
                CK(cudaMemcpyAsync(copy.col, m.col, (size_t)m.nnz * sizeof(int), cudaMemcpyDeviceToDevice, c->stream));
                CK(cudaMemcpyAsync(copy.val, m.val, (size_t)m.nnz * sizeof(double), cudaMemcpyDeviceToDevice,
                                   c->stream));
            }
        }
        std::swap(c->csr, staged ? m : copy);
        c->graph_gen += 1;
    } else {
        CK(csr_densify(m.rp, m.col, m.val, 0, c->rows, c->ld, c->A, c->stream));
        CK(launch_row_envelope(c->A, c->ld, 0, c->rows, c->env, c->stream));
        c->kernel_launches += 2;
    }
    CK(cudaStreamSynchronize(c->stream));
    if (plan) {
        if (c->storage == 0) {
            std::swap(plan->rp, m.rp);
            std::swap(plan->col, m.col);
        }
        std::swap(c->plan, *plan);
    }
    c->matrix_set = true;
    return CGB_OK;
}

// Stages this rank's rows of COO triples in device memory, each cell's writes folded by `fold`, and installs
// them.  Nothing of the context, its matrix or its plan, is touched before every triple has been checked.  A
// non-null `plan` (cgb_assemble_coo's) receives the assembly plan, which becomes the context's.
int install_coo(cgb_ctx *c, int64_t nz, const int32_t *irn, const int32_t *jcn, const double *val, int symmetric,
                AsmFold fold, AsmPlan *plan)
{
    StagedCsr m;
    int bad = 0;
    CK(csr_assemble_coo(&m, plan, fold, c->n, c->row0, c->rows, irn, jcn, val, nz, symmetric ? 1 : 0, &bad,
                        c->stream));
    // keys, runs, rows, cols, fold (CUB's sort and selects not counted); of the two COO builders only
    // cgb_assemble_coo promises its kernels to cgb_launch_count
    if (plan) c->kernel_launches += nz > 0 ? 5 : 2;
    if (bad) return fail(CGB_ERR_INVALID, "a COO entry lies outside %lld x %lld", (long long)c->n, (long long)c->n);
    return install_matrix(c, m, true, plan);
}

} // namespace

extern "C" int cgb_generate_lap2d(cgb_ctx *c)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    StagedCsr m;
    CK(csr_generate_lap2d(&m, c->n, c->row0, c->rows, c->stream));
    c->kernel_launches += 3;
    return install_matrix(c, m, true);
}

extern "C" int cgb_set_matrix_rows(cgb_ctx *c, const double *rows_host, int64_t first_row,
                                   int64_t nrows, int64_t ld_host)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (c->storage == 1) return fail(CGB_ERR_STATE, "dense rows cannot be set on a CSR context (use cgb_set_matrix_coo)");
    if (!rows_host || nrows < 0 || first_row < 0 || first_row + nrows > c->n || ld_host < c->n)
        return fail(CGB_ERR_INVALID, "bad row block [%lld, +%lld) ld %lld", (long long)first_row,
                    (long long)nrows, (long long)ld_host);
    const long long lo = std::max<long long>(first_row, c->row0);
    const long long hi = std::min<long long>(first_row + nrows, c->row0 + c->rows);
    asm_plan_free(&c->plan); // the rows may overwrite assembled cells
    if (hi > lo) {
        CK(cudaMemcpy2DAsync(c->A + (lo - c->row0) * c->ld, (size_t)c->ld * 8,
                             rows_host + (lo - first_row) * ld_host, (size_t)ld_host * 8,
                             (size_t)c->n * 8, (size_t)(hi - lo), cudaMemcpyHostToDevice, c->stream));
        CK(launch_row_envelope(c->A, c->ld, lo - c->row0, hi - lo, c->env, c->stream)); // the rows written
        c->kernel_launches += 1;
        CK(cudaStreamSynchronize(c->stream));
    }
    c->matrix_set = true;
    return CGB_OK;
}

extern "C" int cgb_set_matrix_coo(cgb_ctx *c, int64_t nz, const int32_t *irn, const int32_t *jcn,
                                  const double *val, int symmetric)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (nz < 0 || (nz > 0 && (!irn || !jcn || !val))) return fail(CGB_ERR_INVALID, "bad COO arguments");
    // Matrix::read's sequential "later entries overwrite" (matrix.cc:12-21) on the device: the writes as
    // sequence 2z (direct) / 2z+1 (mirror), stable-sorted by (row, column), the last of every run kept (spmv.cu)
    DevBuf i, j, v;
    CK(i.alloc((size_t)nz * sizeof(int)));
    CK(j.alloc((size_t)nz * sizeof(int)));
    CK(v.alloc((size_t)nz * sizeof(double)));
    if (nz > 0) {
        CK(cudaMemcpyAsync(i.p, irn, (size_t)nz * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        CK(cudaMemcpyAsync(j.p, jcn, (size_t)nz * sizeof(int), cudaMemcpyHostToDevice, c->stream));
        CK(cudaMemcpyAsync(v.p, val, (size_t)nz * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    }
    return install_coo(c, nz, i.as<int32_t>(), j.as<int32_t>(), v.as<double>(), symmetric, kFoldLast, nullptr);
}

extern "C" int cgb_get_matrix_rows(cgb_ctx *c, double *rows_host, int64_t first_row, int64_t nrows,
                                   int64_t ld_host)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (!rows_host || nrows < 0 || first_row < c->row0 || first_row + nrows > c->row0 + c->rows ||
        ld_host < c->n)
        return fail(CGB_ERR_INVALID, "rows [%lld, +%lld) are not inside this rank's shard",
                    (long long)first_row, (long long)nrows);
    if (nrows > 0 && c->storage == 1) { // densified through a device buffer (a test hook)
        double *dense = nullptr;
        CK(cudaMalloc(&dense, (size_t)nrows * c->n * sizeof(double)));
        cudaError_t e = csr_densify(c->csr.rp, c->csr.col, c->csr.val, first_row - c->row0, nrows, c->n, dense, c->stream);
        if (e == cudaSuccess)
            e = cudaMemcpy2DAsync(rows_host, (size_t)ld_host * 8, dense, (size_t)c->n * 8, (size_t)c->n * 8,
                                  (size_t)nrows, cudaMemcpyDeviceToHost, c->stream);
        if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
        cudaFree(dense);
        CK(e);
    } else if (nrows > 0) {
        CK(cudaMemcpy2DAsync(rows_host, (size_t)ld_host * 8, c->A + (first_row - c->row0) * c->ld,
                             (size_t)c->ld * 8, (size_t)c->n * 8, (size_t)nrows,
                             cudaMemcpyDeviceToHost, c->stream));
        CK(cudaStreamSynchronize(c->stream));
    }
    return CGB_OK;
}

extern "C" int cgb_init_source_term(int64_t n, double h, double *b_host)
{
    if (n < 0 || (n > 0 && !b_host)) return fail(CGB_ERR_INVALID, "bad source-term arguments");
    for (int64_t i = 0; i < n; ++i) { // cg.cc:222-233
        const double s = std::sin(10. * M_PI * i * h);
        b_host[i] = -2. * i * M_PI * M_PI * s * s;
    }
    return CGB_OK;
}

extern "C" int cgb_set_rhs(cgb_ctx *c, const double *b_host)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (!b_host) return fail(CGB_ERR_INVALID, "null b");
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    CK(cudaMemcpyAsync(c->b, b_host, (size_t)c->n * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    c->rhs_set = true;
    return CGB_OK;
}

// ------------------------------------------------------------------ options
extern "C" int cgb_set_option(cgb_ctx *c, const char *key, int64_t value)
{
    if (!c || !key) return fail(CGB_ERR_INVALID, "null argument");
    const std::string k(key);
    // the schedules hand the complete state over between launches, so this one may change mid-solve
    if (c->in_solve && k != "schedule") return fail(CGB_ERR_STATE, "options cannot change during a solve");
    // CSR contexts have one mat-vec: the dense-only modes are refused, the launch-shape knobs
    // (set by the CUDA-form command line) are kept but change nothing
    if (c->storage == 1 && ((k == "compat" && value == 1) || ((k == "loopback" || k == "trace") && value > 0)))
        return fail(CGB_ERR_STATE, "option '%s' = %lld is not available with CSR storage", key, (long long)value);
    if (k == "gemv_variant") {
        if (value < 0 || value >= gemv_variant_count())
            return fail(CGB_ERR_INVALID, "gemv_variant %lld out of range", (long long)value);
        set_variant(c, (int)value);
        c->graph_gen += 1;
        if (use_device(c) == CGB_OK) {
            gemv_variant(c->variant).preload();
            if (persist_index(c) >= 0) persist_variant(persist_index(c)).preload();
        }
    } else if (k == "graph") {
        c->opt_graph = value != 0;
    } else if (k == "profile") {
        c->opt_profile = value != 0;
    } else if (k == "poll_every") {
        if (value < 1) return fail(CGB_ERR_INVALID, "poll_every must be >= 1");
        c->poll_every = (int)value;
    } else if (k == "graph_unroll") {
        if (value < 1 || value > 64) return fail(CGB_ERR_INVALID, "graph_unroll must be in [1, 64]");
        c->graph_unroll = (int)value;
        c->graph_gen += 1;
    } else if (k == "compat") {
        if (value != 0) {
            if (c->world != 1) return fail(CGB_ERR_INVALID, "compat mat-vec is single-GPU (like the reference CUDA program)");
            if (c->opt_num_threads < 1 || c->opt_num_threads > 1024 || c->opt_block_width < 1)
                return fail(CGB_ERR_INVALID, "compat needs num_threads in [1, 1024] and block_width >= 1 set first");
            int rc = use_device(c);
            if (rc) return rc;
            const size_t need = compat_part_doubles(c->n, c->opt_block_width);
            if (need > c->compat_part_cap) {
                if (c->compat_part) cudaFree(c->compat_part);
                c->compat_part = nullptr;
                c->compat_part_cap = 0;
                cudaError_t e = cudaMalloc(&c->compat_part, need * sizeof(double));
                if (e != cudaSuccess)
                    return fail(CGB_ERR_NOMEM, "compat partial buffer (%zu MB): %s", need * 8 >> 20,
                                cudaGetErrorString(e));
                c->compat_part_cap = need;
            }
        }
        c->opt_compat = value != 0;
        c->graph_gen += 1;
    } else if (k == "pdl") {
        c->opt_pdl = value != 0;
        c->graph_gen += 1;
    } else if (k == "l2_ramp") {
        if (value < 0 || value > 64) return fail(CGB_ERR_INVALID, "l2_ramp must be in [0, 64] pipeline steps");
        c->opt_l2_ramp = (int)value;
    } else if (k == "l2_prefetch") {
        if (value < 0 || value > 64) return fail(CGB_ERR_INVALID, "l2_prefetch must be in [0, 64] pipeline steps");
        c->opt_l2_prefetch = (int)value;
        c->graph_gen += 1;
    } else if (k == "balance") {
        c->opt_balance = value != 0;
    } else if (k == "schedule") {
        if (value != 0 && value != 1) return fail(CGB_ERR_INVALID, "schedule must be 0 (CUDA graph of 4 kernels per iteration) or 1 (persistent kernel)");
        c->opt_schedule = (int)value;
    } else if (k == "spin_timeout_ms") {
        if (value < 1 || value > 3600000) return fail(CGB_ERR_INVALID, "spin_timeout_ms must be in [1, 3600000]");
        c->spin_timeout_ms = value;
    } else if (k == "trace") {
        // keep %globaltimer timelines of the last `value` launches of the loop kernels (0 = off)
        if (value < 0 || value > 4096) return fail(CGB_ERR_INVALID, "trace must be in [0, 4096] launches");
        int rc = use_device(c);
        if (rc) return rc;
        CK(cudaStreamSynchronize(c->stream));
        free_trace(c);
        c->graph_gen += 1;
        if (value > 0) {
            int max_cps = 1;
            for (int v = 0; v < gemv_variant_count(); ++v)
                if (gemv_variant(v).ctas_per_sm > max_cps) max_cps = gemv_variant(v).ctas_per_sm;
            const int blocks[3] = {c->sm_count * max_cps, (int)c->nchunks, (int)c->nchunks};
            for (int w = 0; w < 3; ++w) {
                const size_t words = (size_t)value * blocks[w] * kTraceWords;
                CK(cudaMalloc(&c->trace_buf[w], words * sizeof(unsigned long long)));
                CK(cudaMalloc(&c->trace_cnt[w], (size_t)blocks[w] * sizeof(unsigned int)));
                CK(cudaMemset(c->trace_buf[w], 0, words * sizeof(unsigned long long)));
                CK(cudaMemset(c->trace_cnt[w], 0, (size_t)blocks[w] * sizeof(unsigned int)));
                c->trace_blocks[w] = blocks[w];
            }
            c->trace_cap = (int)value;
        }
    } else if (k == "loopback") {
        // Profiling aid: one GPU runs ONE rank's shard of a `world`-way split under the production
        // schedule, with every peer pointer of the fused exchange aimed at its own buffer (it
        // fills all `world` slots itself).  Timing and traffic of that rank are real; the
        // numbers it iterates on are not a CG solve.
        if (value != 0) {
            if (c->world < 2) return fail(CGB_ERR_INVALID, "loopback needs world > 1");
            if (c->p2p_ready && !c->opt_loopback) return fail(CGB_ERR_STATE, "a real exchange is already imported");
            c->opt_loopback = 1;
            c->p2p_ready = true;
            c->opt_exchange = 1;
        } else if (c->opt_loopback) {
            c->opt_loopback = 0;
            c->p2p_ready = false;
            c->opt_exchange = 0;
        }
        c->graph_gen += 1;
    } else if (k == "exchange") {
        if (value != 0 && value != 1) return fail(CGB_ERR_INVALID, "exchange must be 0 (nccl) or 1 (fused p2p)");
        if (c->world > 1 && value == 1 && !c->p2p_ready)
            return fail(CGB_ERR_STATE, "exchange = 1 needs cgb_exchange_import first");
        if (c->world > 1 && value == 0 && !c->comm)
            return fail(CGB_ERR_STATE, "exchange = 0 needs cgb_comm_init first");
        c->opt_exchange = (int)value;
        c->graph_gen += 1;
    } else if (k == "num_threads") {
        c->opt_num_threads = (int)value;
        c->opt_compat = 0; // re-enable with "compat" = 1 (re-validates, re-sizes the partial buffer)
        c->graph_gen += 1;
    } else if (k == "block_width") {
        c->opt_block_width = (int)value;
        c->opt_compat = 0;
        c->graph_gen += 1;
    } else if (k == "transposed") {
        c->opt_transposed = value != 0;
        c->graph_gen += 1;
    } else {
        return fail(CGB_ERR_INVALID, "unknown option '%s'", key);
    }
    return CGB_OK;
}

extern "C" int cgb_get_option(cgb_ctx *c, const char *key, int64_t *value)
{
    if (!c || !key || !value) return fail(CGB_ERR_INVALID, "null argument");
    const std::string k(key);
    if (k == "gemv_variant") *value = c->variant;
    else if (k == "graph") *value = c->opt_graph;
    else if (k == "profile") *value = c->opt_profile;
    else if (k == "poll_every") *value = c->poll_every;
    else if (k == "graph_unroll") *value = c->graph_unroll;
    else if (k == "graph_replays") *value = c->graph_replays;
    else if (k == "graph_captures") *value = c->graph_captures;
    else if (k == "device_loop_pdl") *value = c->loop_single.pdl_used >= 0 ? c->loop_single.pdl_used : c->loop_block.pdl_used;
    else if (k == "compat") *value = c->opt_compat;
    else if (k == "pdl") *value = c->opt_pdl;
    else if (k == "l2_prefetch") *value = c->opt_l2_prefetch;
    else if (k == "l2_ramp") *value = c->opt_l2_ramp;
    else if (k == "exchange") *value = c->opt_exchange;
    else if (k == "trace") *value = c->trace_cap;
    else if (k == "schedule") *value = c->opt_schedule;
    else if (k == "balance") *value = c->opt_balance;
    else if (k == "schedule_in_use") *value = (c->opt_schedule == 1 && !persist_unusable(c, c->opt_profile)) ? 1 : 0;
    else if (k == "spin_timeout_ms") *value = c->spin_timeout_ms;
    else if (k == "loopback") *value = c->opt_loopback;
    else if (k == "num_threads") *value = c->opt_num_threads;
    else if (k == "block_width") *value = c->opt_block_width;
    else if (k == "transposed") *value = c->opt_transposed;
    else if (k == "storage") *value = c->storage;
    else if (k == "nnz") *value = c->storage == 1 ? c->csr.nnz : 0;
    else if (k == "envelope_doubles") { // sum over this rank's rows of (last + 1 - first); 0 on a CSR context
        *value = 0;
        if (c->storage == 0 && c->rows > 0) {
            CK(cudaSetDevice(c->device));
            std::vector<int2> env((size_t)c->rows);
            CK(cudaMemcpyAsync(env.data(), c->env, (size_t)c->rows * sizeof(int2), cudaMemcpyDeviceToHost, c->stream));
            CK(cudaStreamSynchronize(c->stream));
            for (const int2 &e : env)
                if (e.y > e.x) *value += e.y - e.x;
        }
    }
    else return fail(CGB_ERR_INVALID, "unknown option '%s'", key);
    return CGB_OK;
}

extern "C" int cgb_get_layout(cgb_ctx *c, cgb_layout *out)
{
    if (!c || !out) return fail(CGB_ERR_INVALID, "null argument");
    out->n = c->n;
    out->ld = c->ld;
    out->rows = c->rows;
    out->row0 = c->row0;
    out->rank = c->rank;
    out->world = c->world;
    out->device = c->device;
    out->nblk = c->nblk;
    out->sm_count = c->sm_count;
    out->nchunks = c->nchunks;
    return CGB_OK;
}

// ------------------------------------------------------------------ solve
extern "C" int cgb_solve_begin(cgb_ctx *c, const double *x0_host, int64_t max_iter, double tol,
                               int keep_history)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (!c->matrix_set) return fail(CGB_ERR_STATE, "matrix not set");
    if (!c->rhs_set) return fail(CGB_ERR_STATE, "right-hand side not set");
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve already in progress");
    if (max_iter < 0) return fail(CGB_ERR_INVALID, "max_iter < 0");
    if (!exchange_configured(c))
        return fail(CGB_ERR_STATE, "world > 1 but neither cgb_comm_init nor cgb_exchange_import was called");
    SolveRun &run = c->run;
    run.max_iter = max_iter;
    run.tol = tol;
    run.launched = 0;
    run.loop_ms = 0.0;
    c->prof_gemv_ms = 0.0;
    c->prof_gemv_n = 0;
    if (keep_history) {
        const long long need = max_iter > 0 ? max_iter : 1;
        if (need > c->hist_cap) {
            if (run.hist) cudaFree(run.hist);
            run.hist = nullptr;
            c->hist_cap = 0;
            CK(cudaMalloc(&run.hist, (size_t)need * sizeof(double)));
            c->hist_cap = need;
            c->graph_gen += 1;
        }
        CK(cudaMemsetAsync(run.hist, 0, (size_t)c->hist_cap * sizeof(double), c->stream));
    } else if (run.hist) {
        cudaFree(run.hist);
        run.hist = nullptr;
        c->hist_cap = 0;
        c->graph_gen += 1;
    }
    *c->h_done = 0;
    if ((rc = reset_states(c, run.st, 1))) return rc;
    if (x0_host) CK(cudaMemcpyAsync(c->x, x0_host, (size_t)c->n * 8, cudaMemcpyHostToDevice, c->stream));
    else CK(cudaMemsetAsync(c->x, 0, (size_t)c->ld * 8, c->stream));
    // r = b - A x0 ; p = r ; partials of r.p                          cg.cc:77-92
    const Mode m = host_mode(c);
    if ((rc = launch_matvec(c, c->x, 0, c->variant, m))) return rc;
    if ((rc = launch_gather(c))) return rc;
    CK(launch_init_residual(make_vec_args(c, m), c->stream));
    c->kernel_launches += 1;
    CK(cudaStreamSynchronize(c->stream));
    c->in_solve = true;
    return CGB_OK;
}

extern "C" int cgb_iterate(cgb_ctx *c, int64_t iters, float *ms)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (!c->in_solve) return fail(CGB_ERR_STATE, "cgb_solve_begin was not called");
    if (iters < 0) return fail(CGB_ERR_INVALID, "iters < 0");
    SolveRun &run = c->blk.active ? c->blk.run : c->run;
    long long todo = std::min<long long>(iters, run.max_iter - run.launched);
    if (todo < 0) todo = 0;
    if (c->blk.active) {
        const Mode m = {run.hist, c->d_hdone, c->opt_pdl};
        return host_loop(c, run, todo, c->opt_graph != 0, c->graph_block, 4,
                         [&]() { return launch_block_iteration(c, m); }, ms);
    }
    const Mode m = host_mode(c);
    if (c->opt_schedule == 1 && !persist_unusable(c, c->opt_profile) && todo > 0) {
        // no graph, no per-iteration launch, no host polling
        CK(cudaEventRecord(c->ev0, c->stream));
        if ((rc = launch_persist_bodies(c, todo, m))) return rc;
        run.launched += todo;
        return end_window(c, run, ms);
    }
    const bool profile = c->opt_profile != 0;
    if (profile) {
        while ((long long)c->prof_ev.size() < 2 * todo) {
            cudaEvent_t e;
            CK(cudaEventCreate(&e));
            c->prof_ev.push_back(e);
        }
    }
    long long profiled = 0; // "profile": each body's mat-vec between two events
    rc = host_loop(c, run, todo, c->opt_graph != 0 && !profile, c->graph_single, c->opt_compat ? 5 : 4, [&]() -> int {
        if (!profile) return launch_iteration(c, m);
        const long long slot = 2 * profiled++;
        CK(cudaEventRecord(c->prof_ev[slot], c->stream));
        int r = launch_matvec(c, c->p, 1, c->variant, m);
        if (r) return r;
        CK(cudaEventRecord(c->prof_ev[slot + 1], c->stream));
        if ((r = launch_gather(c))) return r;
        return launch_vector_phase(c, m);
    }, ms);
    if (rc) return rc;
    for (long long k = 0; k < profiled; ++k) {
        float g = 0.f;
        CK(cudaEventElapsedTime(&g, c->prof_ev[2 * k], c->prof_ev[2 * k + 1]));
        c->prof_gemv_ms += g;
    }
    c->prof_gemv_n += profiled;
    return CGB_OK;
}

extern "C" int cgb_solve_end(cgb_ctx *c, double *x_host, double *resid_hist, cgb_solve_info *info)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (!c->in_solve) return fail(CGB_ERR_STATE, "no solve in progress");
    if (c->blk.active) return fail(CGB_ERR_STATE, "a block solve is in progress (cgb_solve_block_end)");
    if (resid_hist && !c->run.hist) return fail(CGB_ERR_STATE, "history was not requested in cgb_solve_begin");
    CK(launch_finalize(make_vec_args(c, host_mode(c)), c->stream));
    c->kernel_launches += 1;
    if (x_host) CK(cudaMemcpyAsync(x_host, c->x, (size_t)c->n * 8, cudaMemcpyDeviceToHost, c->stream));
    if ((rc = collect_solve(c, c->run, resid_hist, info))) return rc;
    c->in_solve = false;
    return CGB_OK;
}

extern "C" int cgb_solve(cgb_ctx *c, double *x_host, int64_t max_iter, double tol, double *resid_hist,
                         cgb_solve_info *info)
{
    if (!x_host) return fail(CGB_ERR_INVALID, "null x");
    int rc = cgb_solve_begin(c, x_host, max_iter, tol, resid_hist != nullptr);
    if (rc) return rc;
    rc = cgb_iterate(c, max_iter, nullptr);
    if (rc) {
        c->in_solve = false;
        return rc;
    }
    return cgb_solve_end(c, x_host, resid_hist, info);
}

// ------------------------------------------------------------------ block solve
// A null context on a machine without a device is reported as the missing device, like the
// context creation it stands for.
static int null_context()
{
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return fail(CGB_ERR_NO_DEVICE, "no CUDA device");
    }
    return fail(CGB_ERR_INVALID, "null context");
}

extern "C" int cgb_solve_block_begin(cgb_ctx *c, int nrhs, const double *b_host, const double *x0_host,
                                     int64_t max_iter, double tol, int keep_history)
{
    if (!c) return null_context();
    if (nrhs < 1 || nrhs > CGB_MAX_RHS) return fail(CGB_ERR_INVALID, "nrhs must be in [1, %d] (got %d)", CGB_MAX_RHS, nrhs);
    if (!b_host) return fail(CGB_ERR_INVALID, "null b");
    if (max_iter < 0) return fail(CGB_ERR_INVALID, "max_iter < 0");
    int rc = use_device(c);
    if (rc) return rc;
    if (c->storage != 1)
        return fail(CGB_ERR_STATE, "block solves need CSR storage: the dense mat-vec streams one p per tile pipeline");
    if (c->world > 1)
        return fail(CGB_ERR_STATE, "block solves run on one rank: the exchange carries one vector per row");
    if (!c->matrix_set) return fail(CGB_ERR_STATE, "matrix not set");
    if (c->in_solve) return fail(CGB_ERR_STATE, c->blk.active ? "block solve already in progress" : "a single solve is in progress");
    BlockSolve &k = c->blk;
    if ((rc = size_block(c, nrhs, max_iter, keep_history != 0))) return rc;
    start_block_run(c, nrhs, max_iter, tol, keep_history != 0);
    if (k.run.hist) CK(cudaMemsetAsync(k.run.hist, 0, (size_t)k.cap * k.hist_cap * sizeof(double), c->stream));
    *c->h_done = 0;
    if ((rc = reset_states(c, k.run.st, nrhs))) return rc;
    CK(cudaMemsetAsync(k.arrive, 0, (size_t)(2 * k.cap + 1) * sizeof(unsigned int), c->stream));
    const size_t row = (size_t)c->n * 8, pitch = (size_t)c->ld * 8;
    CK(cudaMemcpy2DAsync(k.b, pitch, b_host, row, row, (size_t)nrhs, cudaMemcpyHostToDevice, c->stream));
    if (x0_host) CK(cudaMemcpy2DAsync(k.x, pitch, x0_host, row, row, (size_t)nrhs, cudaMemcpyHostToDevice, c->stream));
    else CK(cudaMemsetAsync(k.x, 0, (size_t)nrhs * pitch, c->stream));
    // r = b - A x0 ; p = r ; partials of r.p, per column                cg.cc:77-92
    const BlockArgs a = make_block_args(c, k.x, 0, {k.run.hist, c->d_hdone, c->opt_pdl});
    CK(launch_spmv_block(a, c->sm_count, c->stream));
    CK(launch_init_residual_block(a, c->stream));
    c->kernel_launches += 2;
    CK(cudaStreamSynchronize(c->stream));
    k.active = true;
    c->in_solve = true;
    return CGB_OK;
}

extern "C" int cgb_solve_block_end(cgb_ctx *c, double *x_host, double *resid_hist, cgb_solve_info *info)
{
    if (!c) return null_context();
    int rc = use_device(c);
    if (rc) return rc;
    BlockSolve &k = c->blk;
    if (!k.active) return fail(CGB_ERR_STATE, "no block solve in progress");
    if (resid_hist && !k.run.hist) return fail(CGB_ERR_STATE, "history was not requested in cgb_solve_block_begin");
    CK(launch_finalize_block(make_block_args(c, k.p, 0, {k.run.hist, c->d_hdone, c->opt_pdl}), c->stream));
    c->kernel_launches += 1;
    const size_t row = (size_t)c->n * 8, pitch = (size_t)c->ld * 8;
    if (x_host) CK(cudaMemcpy2DAsync(x_host, row, k.x, pitch, row, (size_t)k.run.nrhs, cudaMemcpyDeviceToHost, c->stream));
    if ((rc = collect_solve(c, k.run, resid_hist, info))) return rc;
    k.active = false;
    c->in_solve = false;
    return CGB_OK;
}

extern "C" int cgb_solve_block(cgb_ctx *c, int nrhs, const double *b_host, double *x_host, int64_t max_iter,
                               double tol, double *resid_hist, cgb_solve_info *info)
{
    if (!c) return null_context();
    if (!x_host) return fail(CGB_ERR_INVALID, "null x");
    int rc = cgb_solve_block_begin(c, nrhs, b_host, x_host, max_iter, tol, resid_hist != nullptr);
    if (rc) return rc;
    rc = cgb_iterate(c, max_iter, nullptr);
    if (rc) {
        c->blk.active = false;
        c->in_solve = false;
        return rc;
    }
    return cgb_solve_block_end(c, x_host, resid_hist, info);
}

// ------------------------------------------------------------------ device solves
// The refusals both device solves share, and what a context's first device solve allocates
static int device_solve_check(cgb_ctx *c, const double *B, const double *X, const double *hist_dev,
                              const cgb_solve_info *info, const char *bname, const char *xname)
{
    if (c->world > 1)
        return fail(CGB_ERR_STATE, "device solves run on one rank: the exchange of a world > 1 needs the host in lockstep");
    if (c->in_solve)
        return fail(CGB_ERR_STATE, c->blk.active ? "a block solve is in progress" : "a single solve is in progress");
    if (!c->matrix_set) return fail(CGB_ERR_STATE, "matrix not set");
    int rc;
    if ((rc = check_device_ptr(c, B, bname)) || (rc = check_device_ptr(c, X, xname)) ||
        (rc = check_device_ptr(c, info, "info")) || (hist_dev && (rc = check_device_ptr(c, hist_dev, "history"))))
        return rc;
    if (c->loopctl) return CGB_OK;
    CK(preload_loop_kernels());
    if ((rc = stream_events(c))) return rc;
    CK(cudaMalloc(&c->loopctl, sizeof(LoopCtl)));
    CK(cudaMemsetAsync(c->loopctl, 0, sizeof(LoopCtl), c->stream));
    return CGB_OK;
}

// The start of both device solves: the caller's stream gates the context's (the solve sees everything
// enqueued on `us` before the call), b and x0 go into the solve's ld-padded buffers, and device_begin
// sets the States and the loop's body limit from kernel arguments
static int device_solve_enter(cgb_ctx *c, cudaStream_t us, int nrhs, long long max_iter, const double *B,
                              const double *X, double *b, double *x, State *st)
{
    CK(cudaEventRecord(c->ev_dev[0], us));
    CK(cudaStreamWaitEvent(c->stream, c->ev_dev[0], 0));
    const size_t row = (size_t)c->n * 8, pitch = (size_t)c->ld * 8;
    CK(cudaMemcpy2DAsync(b, pitch, B, row, row, (size_t)nrhs, cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaMemcpy2DAsync(x, pitch, X, row, row, (size_t)nrhs, cudaMemcpyDeviceToDevice, c->stream));
    CK(launch_device_begin(st, nrhs, c->loopctl, max_iter, c->stream));
    c->kernel_launches += 1;
    return CGB_OK;
}

// ... and its end, after the finalize kernel: the info and the executed history into the caller's
// memory, x back, and the context's stream gates the caller's (work enqueued on `us` after the call
// sees them)
static int device_solve_leave(cgb_ctx *c, cudaStream_t us, int nrhs, long long max_iter, const State *st,
                              const double *hist, long long hist_ld, double *hist_dev, cgb_solve_info *info,
                              const double *x, double *X)
{
    CK(launch_device_info(st, nrhs, c->loopctl, info, hist, hist_ld, hist_dev, max_iter, c->stream));
    c->kernel_launches += 2; // and finalize
    const size_t row = (size_t)c->n * 8, pitch = (size_t)c->ld * 8;
    CK(cudaMemcpy2DAsync(X, row, x, pitch, row, (size_t)nrhs, cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev_dev[1], c->stream));
    CK(cudaStreamWaitEvent(us, c->ev_dev[1], 0));
    return CGB_OK;
}

extern "C" int cgb_solve_device(cgb_ctx *c, const double *b_dev, double *x_dev, int64_t max_iter, double tol,
                                double *hist_dev, cgb_solve_info *info_dev, void *stream)
{
    if (!c) return null_context();
    int rc = use_device(c);
    if (rc) return rc;
    if (max_iter < 0) return fail(CGB_ERR_INVALID, "max_iter < 0");
    if ((rc = device_solve_check(c, b_dev, x_dev, hist_dev, info_dev, "b", "x"))) return rc;
    const long long hist_need = max_iter > 0 ? max_iter : 1;
    if (hist_dev && hist_need > c->dev_hist_cap) { // grows only; the loop graph is keyed on the pointer
        CK(cudaStreamSynchronize(c->stream));
        if (c->dev_hist) cudaFree(c->dev_hist);
        c->dev_hist = nullptr;
        c->dev_hist_cap = 0;
        CK(cudaMalloc(&c->dev_hist, (size_t)hist_need * sizeof(double)));
        c->dev_hist_cap = hist_need;
    }
    const cudaStream_t us = static_cast<cudaStream_t>(stream);
    const Mode m = {hist_dev ? c->dev_hist : nullptr, nullptr, c->opt_pdl};
    c->run.tol = tol;
    if ((rc = device_solve_enter(c, us, 1, max_iter, b_dev, x_dev, c->b, c->x, c->run.st))) return rc;
    // cgb_solve_begin's r = b - A x0 ; p = r ; rsold = r.p, then cgb_iterate's loop
    if ((rc = launch_matvec(c, c->x, 0, c->variant, m))) return rc;
    CK(launch_init_residual(make_vec_args(c, m), c->stream));
    c->kernel_launches += 1;
    if (c->opt_schedule == 1 && !persist_unusable(c, false)) {
        if (max_iter > 0) {
            CK(launch_loop_ctl(c->loopctl, nullptr, nullptr, 0, 0, 0, 1, 0, 1, c->stream)); // start stamp
            c->kernel_launches += 1;
        }
        if ((rc = launch_persist_bodies(c, max_iter, m))) return rc;
    } else {
        rc = launch_loop_graph(c, c->loop_single, graph_key(c, 1, tol, m.hist), m, &c->run.st->done, nullptr,
                               c->opt_compat ? 5 : 4, max_iter, [&](const Mode &bm) { return launch_iteration(c, bm); });
        if (rc) return rc;
    }
    CK(launch_finalize(make_vec_args(c, m), c->stream));
    if ((rc = device_solve_leave(c, us, 1, 0, c->run.st, m.hist, 0, hist_dev, info_dev, c->x, x_dev))) return rc;
    c->rhs_set = true;
    return CGB_OK;
}

extern "C" int cgb_solve_block_device(cgb_ctx *c, int nrhs, const double *B_dev, double *X_dev, int64_t max_iter,
                                      double tol, double *hist_dev, cgb_solve_info *info_dev, void *stream)
{
    if (!c) return null_context();
    if (nrhs < 1 || nrhs > CGB_MAX_RHS) return fail(CGB_ERR_INVALID, "nrhs must be in [1, %d] (got %d)", CGB_MAX_RHS, nrhs);
    if (max_iter < 0) return fail(CGB_ERR_INVALID, "max_iter < 0");
    int rc = use_device(c);
    if (rc) return rc;
    if (c->storage != 1)
        return fail(CGB_ERR_STATE, "block solves need CSR storage: the dense mat-vec streams one p per tile pipeline");
    if ((rc = device_solve_check(c, B_dev, X_dev, hist_dev, info_dev, "B", "X"))) return rc;
    BlockSolve &k = c->blk;
    if ((rc = size_block(c, nrhs, max_iter, hist_dev != nullptr))) return rc;
    start_block_run(c, nrhs, max_iter, tol, hist_dev != nullptr);
    const cudaStream_t us = static_cast<cudaStream_t>(stream);
    const Mode m = {k.run.hist, nullptr, c->opt_pdl};
    if ((rc = device_solve_enter(c, us, nrhs, max_iter, B_dev, X_dev, k.b, k.x, k.run.st))) return rc;
    // cgb_solve_block_begin's initial residuals, then cgb_iterate's loop
    CK(cudaMemsetAsync(k.arrive, 0, (size_t)(2 * k.cap + 1) * sizeof(unsigned int), c->stream));
    const BlockArgs a = make_block_args(c, k.x, 0, m);
    CK(launch_spmv_block(a, c->sm_count, c->stream));
    CK(launch_init_residual_block(a, c->stream));
    c->kernel_launches += 2;
    rc = launch_loop_graph(c, c->loop_block, graph_key(c, nrhs, tol, m.hist), m, nullptr, k.arrive + 2 * k.cap, 4,
                           max_iter, [&](const Mode &bm) { return launch_block_iteration(c, bm); });
    if (rc) return rc;
    CK(launch_finalize_block(make_block_args(c, k.p, 0, m), c->stream));
    return device_solve_leave(c, us, nrhs, max_iter, k.run.st, m.hist, k.run.hist_ld, hist_dev, info_dev, k.x, X_dev);
}

// ------------------------------------------------------------------ matrix from device memory (DESIGN 3.10)
extern "C" int cgb_set_matrix_csr(cgb_ctx *c, const int64_t *rp_dev, const int32_t *col_dev, const double *val_dev,
                                  int64_t nnz, void *stream)
{
    if (!c) return null_context();
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, c->blk.active ? "a block solve is in progress" : "a single solve is in progress");
    if (nnz < 0) return fail(CGB_ERR_INVALID, "nnz < 0 (got %lld)", (long long)nnz);
    if ((rc = check_device_ptr(c, rp_dev, "rp")) ||
        (nnz > 0 && ((rc = check_device_ptr(c, col_dev, "col")) || (rc = check_device_ptr(c, val_dev, "val")))))
        return rc;
    if ((rc = stream_events(c))) return rc;
    CK(cudaEventRecord(c->ev_dev[0], static_cast<cudaStream_t>(stream)));
    CK(cudaStreamWaitEvent(c->stream, c->ev_dev[0], 0));
    DevBuf rp, err_dev;
    CK(rp.alloc((size_t)(c->rows + 1) * sizeof(long long)));
    CK(err_dev.alloc(sizeof(unsigned long long)));
    // nothing of the context is touched before the input has been checked
    CK(launch_validate_csr(reinterpret_cast<const long long *>(rp_dev), col_dev, nnz, c->n, c->rows,
                           rp.as<long long>(), err_dev.as<unsigned long long>(), c->stream));
    c->kernel_launches += 1;
    CK(cudaMemcpyAsync(c->h_pin, err_dev.p, sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    unsigned long long err;
    memcpy(&err, c->h_pin, sizeof err);
    if (err != ~0ULL) {
        static const char *const what[kCsrFaultKinds] = {
            "rp[0] is negative", "rp decreases (row pointers must be monotone)",
            "its entries reach past rp[0] + nnz", "a column lies outside [0, n)",
            "columns are not strictly ascending (a duplicate or a descending pair)", "rp[rows] - rp[0] != nnz"};
        return fail(CGB_ERR_INVALID, "CSR refused at local row %llu: %s (n %lld, rows %lld, nnz %lld)",
                    err / kCsrFaultKinds, what[err % kCsrFaultKinds], c->n, c->rows, (long long)nnz);
    }
    CsrShard m{rp.as<long long>(), const_cast<int *>(col_dev), const_cast<double *>(val_dev), nnz};
    return install_matrix(c, m, false);
}

extern "C" int cgb_update_matrix_values(cgb_ctx *c, const double *val_dev, void *stream)
{
    if (!c) return null_context();
    int rc = use_device(c);
    if (rc) return rc;
    if (c->storage != 1) return fail(CGB_ERR_STATE, "values can only be updated on a CSR context: a dense shard keeps no pattern");
    if (!c->matrix_set) return fail(CGB_ERR_STATE, "matrix not set");
    if (c->in_solve) return fail(CGB_ERR_STATE, c->blk.active ? "a block solve is in progress" : "a single solve is in progress");
    if (c->csr.nnz > 0 && (rc = check_device_ptr(c, val_dev, "val"))) return rc;
    if ((rc = stream_events(c))) return rc;
    // col / val stay where they are: every cached loop graph stays valid, no generation bump
    const cudaStream_t us = static_cast<cudaStream_t>(stream);
    CK(cudaEventRecord(c->ev_dev[0], us));
    CK(cudaStreamWaitEvent(c->stream, c->ev_dev[0], 0));
    if (c->csr.nnz > 0)
        CK(cudaMemcpyAsync(c->csr.val, val_dev, (size_t)c->csr.nnz * sizeof(double), cudaMemcpyDeviceToDevice, c->stream));
    CK(cudaEventRecord(c->ev_dev[1], c->stream));
    CK(cudaStreamWaitEvent(us, c->ev_dev[1], 0));
    return CGB_OK;
}

// ------------------------------------------------------------------ sum-assembly from device COO (DESIGN 3.11)
extern "C" int cgb_assemble_coo(cgb_ctx *c, int64_t nz, const int32_t *irn_dev, const int32_t *jcn_dev,
                                const double *val_dev, int symmetric, void *stream)
{
    if (!c) return null_context();
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, c->blk.active ? "a block solve is in progress" : "a single solve is in progress");
    if (nz < 0) return fail(CGB_ERR_INVALID, "nz < 0 (got %lld)", (long long)nz);
    if (nz > 0 && ((rc = check_device_ptr(c, irn_dev, "irn")) || (rc = check_device_ptr(c, jcn_dev, "jcn")) ||
                   (rc = check_device_ptr(c, val_dev, "val"))))
        return rc;
    if ((rc = stream_events(c))) return rc;
    CK(cudaEventRecord(c->ev_dev[0], static_cast<cudaStream_t>(stream)));
    CK(cudaStreamWaitEvent(c->stream, c->ev_dev[0], 0));
    StagedPlan plan;
    return install_coo(c, nz, irn_dev, jcn_dev, val_dev, symmetric, kFoldSum, &plan);
}

extern "C" int cgb_assemble_values(cgb_ctx *c, const double *val_dev, void *stream)
{
    if (!c) return null_context();
    int rc = use_device(c);
    if (rc) return rc;
    if (!c->plan.start || !c->matrix_set)
        return fail(CGB_ERR_STATE, "no assembly plan: the matrix was not built by cgb_assemble_coo, or another builder replaced it");
    if (c->in_solve) return fail(CGB_ERR_STATE, c->blk.active ? "a block solve is in progress" : "a single solve is in progress");
    if (c->plan.nz > 0 && (rc = check_device_ptr(c, val_dev, "val"))) return rc;
    if ((rc = stream_events(c))) return rc;
    // the values are written where they are (CSR: csr.val, dense: A): every cached loop graph stays valid
    const cudaStream_t us = static_cast<cudaStream_t>(stream);
    CK(cudaEventRecord(c->ev_dev[0], us));
    CK(cudaStreamWaitEvent(c->stream, c->ev_dev[0], 0));
    if (c->storage == 1) {
        CK(launch_assemble_csr(c->plan, kFoldSum, val_dev, c->csr.val, c->stream));
        c->kernel_launches += 1;
    } else {
        // a cell stored as 0 at assembly lies outside its row's envelope and may have become non-zero
        CK(launch_assemble_dense(c->plan, val_dev, c->ld, c->A, c->stream));
        CK(launch_row_envelope(c->A, c->ld, 0, c->rows, c->env, c->stream));
        c->kernel_launches += 2;
    }
    CK(cudaEventRecord(c->ev_dev[1], c->stream));
    CK(cudaStreamWaitEvent(us, c->ev_dev[1], 0));
    return CGB_OK;
}

extern "C" int cgb_residual_check(cgb_ctx *c, double *norm_x, double *rel_resid)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (!c->matrix_set || !c->rhs_set) return fail(CGB_ERR_STATE, "matrix / right-hand side not set");
    // `done` may still be raised from the solve: the DEBUG mat-vec must run regardless
    CK(cudaMemsetAsync(&c->run.st->done, 0, sizeof(int), c->stream));
    const Mode m = host_mode(c);
    if ((rc = launch_matvec(c, c->x, 0, c->variant, m))) return rc;   // cg.cc:146-147
    if ((rc = launch_gather(c))) return rc;
    double *out = c->scratch + 3 * c->nchunks;
    CK(launch_debug_norms(make_vec_args(c, m), c->scratch, out, c->stream));
    c->kernel_launches += 2;
    CK(cudaMemcpyAsync(c->h_pin, out, 2 * sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    if (norm_x) *norm_x = c->h_pin[0];
    if (rel_resid) *rel_resid = c->h_pin[1];
    return CGB_OK;
}

// ------------------------------------------------------------------ kernel-level hooks
extern "C" int cgb_gemv(cgb_ctx *c, const double *v_host, double *y_host, double *chunk_partials,
                        double *pAp)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (!c->matrix_set) return fail(CGB_ERR_STATE, "matrix not set");
    if (!v_host) return fail(CGB_ERR_INVALID, "null v");
    CK(cudaMemsetAsync(&c->run.st->done, 0, sizeof(int), c->stream));
    CK(cudaMemcpyAsync(c->p, v_host, (size_t)c->n * 8, cudaMemcpyHostToDevice, c->stream));
    if (!exchange_configured(c)) return fail(CGB_ERR_STATE, "world > 1 but no exchange is configured");
    if ((rc = launch_matvec(c, c->p, 0, c->variant, host_mode(c)))) return rc;
    if ((rc = launch_gather(c))) return rc;
    if ((rc = collect_for_host(c))) return rc;
    const Gather gth = make_gather(c);
    const double *mine = c->apx + (long long)c->rank * c->slot;
    if (y_host) CK(cudaMemcpyAsync(y_host, mine, (size_t)c->rows * 8, cudaMemcpyDeviceToHost, c->stream));
    if (chunk_partials || pAp) {
        double *out = c->scratch + 3 * c->nchunks;
        CK(launch_pap_plain(c->p, c->apx, gth, c->n, c->papart, out, c->stream));
        c->kernel_launches += 2;
        if (chunk_partials)
            CK(cudaMemcpyAsync(chunk_partials, c->papart, (size_t)c->nchunks * 8, cudaMemcpyDeviceToHost, c->stream));
        CK(cudaMemcpyAsync(c->h_pin, out, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    }
    CK(cudaStreamSynchronize(c->stream));
    if (pAp) *pAp = c->h_pin[0];
    return CGB_OK;
}

extern "C" int cgb_dot(cgb_ctx *c, const double *a_host, const double *b_host, double *result)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (!a_host || !b_host || !result) return fail(CGB_ERR_INVALID, "null argument");
    CK(cudaMemcpyAsync(c->p, a_host, (size_t)c->n * 8, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemcpyAsync(c->r, b_host, (size_t)c->n * 8, cudaMemcpyHostToDevice, c->stream));
    double *out = c->scratch + 3 * c->nchunks;
    CK(launch_dot(c->p, c->r, c->n, c->scratch, out, c->stream));
    c->kernel_launches += 2;
    CK(cudaMemcpyAsync(c->h_pin, out, sizeof(double), cudaMemcpyDeviceToHost, c->stream));
    CK(cudaStreamSynchronize(c->stream));
    *result = c->h_pin[0];
    return CGB_OK;
}

extern "C" int cgb_bench_gemv(cgb_ctx *c, int variant, int reps, float *ms_avg)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (!c->matrix_set) return fail(CGB_ERR_STATE, "matrix not set");
    if (variant < 0) variant = c->variant;
    if (variant >= gemv_variant_count() || reps < 1) return fail(CGB_ERR_INVALID, "bad variant / reps");
    // A rank of a world > 1 without a configured exchange times its shard with local stores
    // only (shape tuning on one GPU).  The gather geometry follows the timed variant.
    const int keep_variant = c->variant;
    if (variant != keep_variant && c->storage == 0) {
        set_variant(c, variant);
        c->graph_gen += 1;
        CK(gemv_variant(variant).preload()); // loads the kernel and sets its shared-memory limit
    }
    CK(cudaMemsetAsync(&c->run.st->done, 0, sizeof(int), c->stream));
    const Mode m = host_mode(c);
    if ((rc = launch_matvec(c, c->p, 0, variant, m))) return rc; // warm-up
    CK(cudaEventRecord(c->ev0, c->stream));
    for (int i = 0; i < reps; ++i)
        if ((rc = launch_matvec(c, c->p, 0, variant, m))) return rc;
    CK(cudaEventRecord(c->ev1, c->stream));
    // fused mode: the launches above all carried the same tag; consume it so that the next
    // exchange starts from a fresh tag on every rank
    if ((rc = collect_for_host(c))) return rc;
    CK(cudaEventSynchronize(c->ev1));
    CK(cudaStreamSynchronize(c->stream));
    if (variant != keep_variant) set_variant(c, keep_variant);
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, c->ev0, c->ev1));
    if (ms_avg) *ms_avg = t / reps;
    return CGB_OK;
}

extern "C" int cgb_bench_read(cgb_ctx *c, int reps, float *ms_avg)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (reps < 1) return fail(CGB_ERR_INVALID, "reps < 1");
    const long long nd = c->rows * c->ld;
    auto read_once = [&]() {
        return c->storage == 1 ? launch_read_csr(c->csr, c->rows, c->sink, c->sm_count, c->stream)
                               : launch_read_stream(c->A, nd, c->sink, c->sm_count, c->stream);
    };
    CK(read_once());
    CK(cudaEventRecord(c->ev0, c->stream));
    for (int i = 0; i < reps; ++i) CK(read_once());
    CK(cudaEventRecord(c->ev1, c->stream));
    CK(cudaEventSynchronize(c->ev1));
    c->kernel_launches += reps + 1;
    float t = 0.f;
    CK(cudaEventElapsedTime(&t, c->ev0, c->ev1));
    if (ms_avg) *ms_avg = t / reps;
    return CGB_OK;
}

extern "C" int cgb_last_gemv_timing(cgb_ctx *c, float *ms_avg, int64_t *launches)
{
    if (!c) return fail(CGB_ERR_INVALID, "null context");
    if (ms_avg) *ms_avg = c->prof_gemv_n ? (float)(c->prof_gemv_ms / (double)c->prof_gemv_n) : 0.f;
    if (launches) *launches = c->prof_gemv_n;
    return CGB_OK;
}

extern "C" int cgb_launch_count(cgb_ctx *c, int64_t *launches)
{
    if (!c || !launches) return fail(CGB_ERR_INVALID, "null argument");
    *launches = c->kernel_launches;
    return CGB_OK;
}

extern "C" int cgb_trace_read(cgb_ctx *c, int which, uint64_t *out, int64_t capacity_words,
                              int64_t *launches, int64_t *blocks)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (which < 0 || which > 2) return fail(CGB_ERR_INVALID, "which must be 0 (mat-vec), 1 (update_xr) or 2 (update_p)");
    if (c->trace_cap <= 0) return fail(CGB_ERR_STATE, "option \"trace\" is off");
    const int nb = which == 0 ? c->nblk : (int)c->nchunks;
    const int64_t words = (int64_t)c->trace_cap * nb * kTraceWords;
    if (!out || capacity_words < words)
        return fail(CGB_ERR_INVALID, "trace buffer too small: need %lld words", (long long)words);
    CK(cudaStreamSynchronize(c->stream));
    CK(cudaMemcpy(out, c->trace_buf[which], (size_t)words * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    unsigned int seen = 0;
    CK(cudaMemcpy(&seen, c->trace_cnt[which], sizeof seen, cudaMemcpyDeviceToHost));
    if (launches) *launches = seen;
    if (blocks) *blocks = nb;
    return CGB_OK;
}

// One-off selection of the mat-vec tile shape for THIS shard shape on THIS GPU (outside any timed
// region): every candidate runs a few loop bodies of the schedule in use on the resident matrix,
// the fastest is kept.  Box-to-box and shape-to-shape the best shape moves by several percent
// (profiles/r02/tune_*), a static table does not hold.  Ranks of a world > 1 tune alone, with the
// exchange looped back to themselves, so no peer has to take part; all tile shapes share one
// summation order, so the choice never changes a result bit.
extern "C" int cgb_autotune(cgb_ctx *c, int iters, int *chosen, float *us_per_iter)
{
    int rc = use_device(c);
    if (rc) return rc;
    if (c->in_solve) return fail(CGB_ERR_STATE, "solve in progress");
    if (!c->matrix_set) return fail(CGB_ERR_STATE, "matrix not set");
    if (iters < 1) iters = 32; // long enough for the row re-balancing to act on every shape alike
    const int nv = gemv_variant_count();
    if (us_per_iter)
        for (int v = 0; v < nv; ++v) us_per_iter[v] = -1.f;
    if (c->storage == 1) { // one CSR mat-vec: nothing to choose
        if (chosen) *chosen = c->variant;
        return CGB_OK;
    }
    const int keep_variant = c->variant, keep_loopback = c->opt_loopback, keep_exchange = c->opt_exchange;
    const bool keep_ready = c->p2p_ready;
    const double keep_tol = c->run.tol;
    const bool want_persist = c->opt_schedule == 1 && !c->opt_compat && !(c->world > 1 && keep_exchange == 0 && c->comm);
    Ctl ctl0;
    CK(cudaMemcpy(&ctl0, c->ctl, sizeof ctl0, cudaMemcpyDeviceToHost));
    // Tune alone, on SCRATCH gather buffers: every peer pointer aims at the scratch copy, so the
    // real buffers -- which a peer that has already left its own tuning may be writing -- stay untouched
    uint4 *const real_ll = c->ll, *const real_rr = c->rr_ll;
    uint4 *tune_ll = nullptr, *tune_rr = nullptr;
    CK(cudaMalloc(&tune_ll, c->ll_bytes));
    if (cudaMalloc(&tune_rr, (size_t)2 * c->aux_stride * sizeof(uint4)) != cudaSuccess) {
        cudaFree(tune_ll);
        return fail(CGB_ERR_NOMEM, "autotune scratch");
    }
    cudaMemsetAsync(tune_ll, 0, c->ll_bytes, c->stream);
    cudaMemsetAsync(tune_rr, 0, (size_t)2 * c->aux_stride * sizeof(uint4), c->stream);
    c->ll = tune_ll;
    c->rr_ll = tune_rr;
    c->peer_ll[c->rank] = tune_ll;
    if (c->world > 1) {
        c->opt_loopback = 1;
        c->p2p_ready = true;
        c->opt_exchange = 1;
    }
    c->run.tol = 0.0; // never converges
    c->graph_gen += 1;
    int best = keep_variant;
    float best_us = -1.f, default_us = -1.f;
    // the timed runs; a lambda so that a failing CUDA call still reaches the restore below
    auto tune = [&]() -> int {
    int rc = CGB_OK;
    for (int v = 0; v < nv && rc == CGB_OK; ++v) {
        if (strncmp(gemv_variant(v).name, "tma", 3) != 0 || strstr(gemv_variant(v).name, "nohint")) continue;
        set_variant(c, v);
        // only shapes with a persistent instantiation, on either schedule (DESIGN.md 3.3): the
        // choice stays a shape both schedules run when the schedule is switched after tuning
        if (persist_index(c) < 0) continue;
        const bool persist = want_persist && !persist_unusable(c, c->opt_profile);
        if (want_persist && !persist) continue; // compare like with like
        if (gemv_variant(v).preload() != cudaSuccess) { cudaGetLastError(); continue; }
        if (persist && persist_variant(persist_index(c)).preload() != cudaSuccess) { cudaGetLastError(); continue; }
        float t_best = -1.f;
        for (int rep = 0; rep < 3 && rc == CGB_OK; ++rep) { // rep 0 warms up
            if ((rc = reset_states(c, c->run.st, 1))) break;
            CK(cudaEventRecord(c->ev0, c->stream));
            if (persist) {
                rc = launch_persist(c, iters, host_mode(c));
            } else {
                for (int i = 0; i < iters && rc == CGB_OK; ++i) rc = launch_iteration(c, host_mode(c));
            }
            if (rc) break;
            CK(cudaEventRecord(c->ev1, c->stream));
            CK(cudaEventSynchronize(c->ev1));
            float t = 0.f;
            CK(cudaEventElapsedTime(&t, c->ev0, c->ev1));
            if (rep > 0 && (t_best < 0.f || t < t_best)) t_best = t;
        }
        if (rc) break;
        const float us = t_best * 1e3f / (float)iters;
        if (us_per_iter) us_per_iter[v] = us;
        if (v == keep_variant) default_us = us;
        if (best_us < 0.f || us < best_us) {
            best_us = us;
            best = v;
        }
    }
    return rc;
    };
    rc = tune();
    // a candidate must beat the configured shape by more than the run-to-run noise
    if (default_us > 0.f && best_us > default_us * 0.997f) best = keep_variant;
    // leave no trace: state, exchange epoch; the LL entries of the looped-back runs go with the scratch
    cudaStreamSynchronize(c->stream);
    c->ll = real_ll;
    c->rr_ll = real_rr;
    c->peer_ll[c->rank] = real_ll;
    cudaFree(tune_ll);
    cudaFree(tune_rr);
    c->opt_loopback = keep_loopback;
    c->p2p_ready = keep_ready;
    c->opt_exchange = keep_exchange;
    c->run.tol = keep_tol;
    set_variant(c, best);
    c->graph_gen += 1;
    if (rc) return rc;
    gemv_variant(best).preload();
    if (persist_index(c) >= 0) persist_variant(persist_index(c)).preload();
    CK(cudaMemcpyAsync(c->ctl, &ctl0, sizeof ctl0, cudaMemcpyHostToDevice, c->stream));
    CK(cudaMemsetAsync(c->run.st, 0, sizeof(State), c->stream));
    *c->h_done = 0;
    CK(cudaStreamSynchronize(c->stream));
    if (chosen) *chosen = best;
    return CGB_OK;
}
