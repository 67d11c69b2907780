// cgb_device.cuh -- device-side building blocks shared by the sm_100a kernels:
// mbarrier / bulk-copy (TMA) PTX wrappers, the deterministic reduction primitives whose
// order oracle/cg_oracle.c mirrors, and the structs passed to the kernels.
#pragma once

#include <cstdint>
#include <cuda_runtime.h>

namespace cgb {

constexpr double kNearZero = 1.0e-14; // NEARZERO, code/MPI/cg.cc:8, code/CUDA/cg.cu:11
constexpr int kChunk = 256;           // elements per r'r chunk partial
constexpr int kMaxWorld = 8;

// Scalars that live on the device for the whole solve (no host round trip per iteration;
// the reference computes alpha/beta on the host after blocking copies, cg.cu:231-269).
struct State {
    double rsold;   // reference's rsold (stale after a convergence break, as the DEBUG line prints)
    double rsnew;   // last r'r
    double conj;    // last p'Ap          (diagnostic)
    double alpha;   // last step length   (diagnostic)
    long long iter; // loop bodies completed without breaking == the reference's k
    int done;       // sqrt(rsnew) < tol fired
    int pad;
};

// Control words of the fused exchange (P2P mode), local to each rank.
struct Ctl {
    unsigned long long epoch; // exchanges consumed so far; the running one carries tag epoch + 1
    unsigned int arrive;      // blocks of the running consumer kernel that have finished reading
    unsigned int pad;
};

// Geometry of the gathered mat-vec result: rank g owns slot g of `slot` entries,
// [0, rows_g) = its Ap rows.
//   plain buffer (`apx`, doubles)  : 1 GPU, ncclAllGather mode, staging for the test hooks
//   LL buffers (`ll`, 16 B entries): fused mode.  An entry is {lo32, tag, hi32, tag}: the value
//       carries its own arrival flag (the tag of the exchange), so the producer needs no fence
//       and no separate flag store, and the consumer polls exactly the data it needs -- the
//       LL protocol of NCCL, applied to fp64.  Two buffers (tag parity): ranks can be at most
//       one exchange apart.
struct Gather {
    long long n_loc;   // rows of every rank but the last (N / world)
    long long slot;    // entries per rank slot
    long long maxrows; // rows of the last rank (the largest shard)
    long long loc_cap;   // entries that really arrive per slot: maxrows -- or, "loopback", this rank's own
                         // row count (it plays every rank with its own rows; reads past them are clamped)
    long long bufstride; // entries per LL buffer (world * slot capacity)
    const uint4 *ll;   // this rank's LL buffers (peers write into them over NVLink)
    Ctl *ctl;
    int world;
    int nblk;
    int p2p;           // 1: fused mode
    unsigned long long spin_ns; // bound of a wait for a peer's entry (option "spin_timeout_ms")
    int *host_err;     // mapped pinned flag: set to -1 before the launch is faulted on a timeout
};

// Diagnostic timeline (option "trace" = launches kept): every CTA of a traced kernel stamps
// %globaltimer at fixed points of its life into rec[(launch % cap) * nblk + cta][kTraceWords];
// `cnt[cta]` counts the launches that CTA index has seen.  This is how the production schedule
// (CUDA graph + programmatic dependent launch, where CUDA events cannot be placed between the
// kernels) is timed: profiles/trace_iter.py, bench.py "production_launch_ms".
constexpr int kTraceWords = 8;
struct Trace {
    unsigned long long *buf; // nullptr: tracing off
    unsigned int *cnt;       // one launch counter per CTA index
    int cap;                 // launches kept (ring)
    int nblk;                // CTAs per launch
};

// ---- column windows of the dense mat-vec --------------------------------------------------
// env[i] = [first, last + 1) of the non-zero (not +-0) columns of local row i; first >= end: the row
// is all zero (the zeroed shard of a new context is {0, 0} everywhere).  A row block is streamed over
// the hull of its rows' envelopes only: every column outside it holds +-0 in every row of the block,
// and a lane-order accumulator (which starts at +0 and is never -0) is unchanged by fma(+-0, p, acc)
// for finite p -- the result is the full-row stream's, bit for bit.
//   c_begin is rounded DOWN to a multiple of 64: lane l owns the columns c % 64 = 2l, 2l + 1 of every
//           tile, which holds only if every tile starts at a multiple of 64
//   c_end   is rounded up to a multiple of 16 and clipped to ld: every bulk copy stays a whole number
//           of 16-byte units at a 16-byte-aligned address
// A block table entry packs (c_begin / 16) | (c_end / 16) << 16, which covers ld <= kWinMaxLd (a dense
// shard that wide holds 8 TB per 1000 rows); a wider ld streams full rows.
constexpr int kWinBlocks = 128;                  // blocks of a CTA with a table entry; later ones stream full rows
constexpr long long kWinMaxLd = 16LL * 0xffff;
__device__ __forceinline__ unsigned block_window(const int2 *env, long long rb0, int nr, long long ld)
{
    int lo = 0x7fffffff, hi = 0;
#pragma unroll 4
    for (int j = 0; j < nr; ++j) {
        const int2 e = env[rb0 + j];
        if (e.x < e.y) {
            lo = e.x < lo ? e.x : lo;
            hi = e.y > hi ? e.y : hi;
        }
    }
    if (lo >= hi) return 0u; // no non-zero in the block: an empty window
    const long long cb = (long long)(lo & ~63), ce0 = ((long long)hi + 15) & ~15LL;
    const long long ce = ce0 < ld ? ce0 : ld;
    return (unsigned)(cb >> 4) | ((unsigned)(ce >> 4) << 16);
}
// the window of block b from a CTA's table `tab` (filled with block_window for b < kWinBlocks)
__device__ __forceinline__ void window_of(const unsigned *tab, int b, long long ld, long long &cb, long long &ce)
{
    if (b < kWinBlocks && ld <= kWinMaxLd) {
        const unsigned w = tab[b];
        cb = (long long)(w & 0xffffu) << 4;
        ce = (long long)(w >> 16) << 4;
    } else {
        cb = 0;
        ce = ld;
    }
}
// tiles of width wd (a multiple of 64) that cover [cb, ce)
__device__ __forceinline__ int window_tiles(long long cb, long long ce, int wd)
{
    return ce > cb ? (int)((ce - cb + wd - 1) / wd) : 0;
}

struct GemvArgs {
    const double *A;      // rows x ld shard, zero-padded columns
    const int2 *env;      // rows envelopes of A (see block_window)
    const double *v;      // input vector, ld doubles, zero-padded
    double *base;         // local plain gather buffer
    uint4 *peer_ll[kMaxWorld]; // fused mode: every rank's LL buffers (self included), peer-mapped
    const Ctl *ctl;
    long long bufstride;
    long long slot_off;   // rank * slot: where this rank's slot starts inside a buffer
    int rank;
    int world;
    int p2p;              // 1: store rows + partials straight into every rank's LL buffer
    long long ld;
    long long rows;
    long long row0;       // global index of the shard's first row (index into v)
    long long maxrows;
    // bookkeeping done by block 0 before streaming (see kernels.cu: advance_state)
    State *st;
    const double *rrpart;
    long long nchunks;
    double *hist;         // nullable
    int advance;          // 1 inside the CG loop, 0 for the init / DEBUG mat-vecs
    int pdl;              // host side: launch with the programmatic-dependent-launch attribute
    int l2_prefetch;      // pipeline steps of A prefetched into L2 before the dependency wait
    Trace trace;          // diagnostic timeline (option "trace"); buf == nullptr: off
    // CSR storage (spmv.cu; A is then nullptr): rows + 1 row pointers, global column indices
    // ascending and unique within a row, values
    const long long *csr_rp;
    const int *csr_col;
    const double *csr_val;
};

// ---- persistent schedule (persist.cu): the whole CG loop in one cooperative launch ----
// Arrival counters of one launch (zeroed by the host before it): CTAs of THIS GPU that finished
// their mat-vec rows, chunk partials of r'r published, chunks of p published.
struct PersistSync {
    unsigned int arrive_mv, arrive_rr, arrive_p, pad;
};
struct PersistArgs {
    const double *A;           // rows x ld shard
    const int2 *env;           // rows envelopes of A (see block_window)
    double *x, *r, *p;         // full-length replicated vectors (ld doubles)
    double *rrpart;            // nchunks chunk partials of r'r (also the hand-over to the next launch)
    uint4 *peer_ll[kMaxWorld]; // every rank's LL gather buffers (self included)
    const uint4 *ll;           // this rank's own LL buffers
    uint4 *rr_ll;              // [2][rr_stride] LL entries local to this GPU: [r'r | p'Ap chunk partials | CTA times]
    long long rr_stride;
    PersistSync *sync;
    State *st;
    Ctl *ctl;
    double *hist;              // nullable
    int *host_done;            // mapped pinned flag: 1 = converged, < 0 = a wait timed out
    long long ld, rows, row0, n, maxrows, n_loc, loc_cap, slot, bufstride, slot_off, nchunks;
    int rank, world, iters, l2_prefetch, l2_ramp, balance;
    int scr_n;                 // shared-memory scratch: doubles for the chunk partials being summed
    double tol;
    unsigned long long spin_ns; // bound of every cross-CTA / cross-rank wait
    Trace trace;
};

// ------------------------------------------------------------------ reductions
__device__ __forceinline__ double shfl_xor_f64(double v, int m)
{
    return __shfl_xor_sync(0xffffffffu, v, m);
}

// butterfly over the 32 lanes: every lane ends with the same, order-specified sum
__device__ __forceinline__ double warp_butterfly(double v)
{
    v = __dadd_rn(v, shfl_xor_f64(v, 16));
    v = __dadd_rn(v, shfl_xor_f64(v, 8));
    v = __dadd_rn(v, shfl_xor_f64(v, 4));
    v = __dadd_rn(v, shfl_xor_f64(v, 2));
    v = __dadd_rn(v, shfl_xor_f64(v, 1));
    return v;
}

// det_sum: lane l adds v[l], v[l+32], ... in ascending order, then the butterfly.
// Must be called by one full warp; `v` may be shared or global memory.
__device__ __forceinline__ double warp_det_sum(const double *v, long long n, int lane)
{
    double s = 0.0;
    for (long long t = lane; t < n; t += 32) s = __dadd_rn(s, v[t]);
    return warp_butterfly(s);
}

// chunk256: perfect xor tree over the 256 per-thread values of a 256-thread block.
// Returns the total in every thread of warp 0; `wsum` is 8 doubles of shared memory.
__device__ __forceinline__ double block_chunk256(double v, double *wsum, int tid)
{
    v = warp_butterfly(v);
    if ((tid & 31) == 0) wsum[tid >> 5] = v;
    __syncthreads();
    double t = 0.0;
    if (tid < 32) {
        t = (tid < 8) ? wsum[tid] : 0.0;
        t = __dadd_rn(t, shfl_xor_f64(t, 4));
        t = __dadd_rn(t, shfl_xor_f64(t, 2));
        t = __dadd_rn(t, shfl_xor_f64(t, 1));
    }
    return t;
}

// ------------------------------------------------------------------ exchange (fused mode)
__device__ __forceinline__ unsigned long long globaltimer_ns()
{
    unsigned long long t;
    asm volatile("mov.u64 %0, %globaltimer;" : "=l"(t));
    return t;
}
// trace helpers: slot of this launch for CTA `cta` (one thread per CTA calls it once) ...
__device__ __forceinline__ unsigned long long *trace_slot(const Trace &t, int cta)
{
    const unsigned k = atomicAdd(&t.cnt[cta], 1u);
    return t.buf + ((size_t)(k % (unsigned)t.cap) * (size_t)t.nblk + (size_t)cta) * kTraceWords;
}
// ... and one stamp into it
__device__ __forceinline__ void trace_stamp(unsigned long long *rec, int word)
{
    if (rec) rec[word] = globaltimer_ns();
}
__device__ __forceinline__ unsigned smid()
{
    unsigned r;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(r));
    return r;
}

// producer: one 16-byte store {lo, tag, hi, tag}; correct even if it tears into two 8-byte halves
__device__ __forceinline__ void ll_store(uint4 *dst, double v, unsigned tag)
{
    const unsigned lo = (unsigned)__double2loint(v), hi = (unsigned)__double2hiint(v);
    asm volatile("st.volatile.global.v4.u32 [%0], {%1, %2, %3, %4};" ::"l"(dst), "r"(lo), "r"(tag), "r"(hi),
                 "r"(tag)
                 : "memory");
}
// consumer: poll the entry until both halves carry the tag.  Bounded (option "spin_timeout_ms"):
// a dead or missing peer is reported through the mapped host flag, then the launch is faulted
// (trap) instead of hanging the GPU -- the C ABI returns CGB_ERR_TIMEOUT.
__device__ __forceinline__ double ll_load(const uint4 *src, unsigned tag, unsigned long long spin_ns, int *host_err)
{
    unsigned lo, f0, hi, f1;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(f0), "=r"(hi), "=r"(f1) : "l"(src) : "memory");
    if (f0 != tag || f1 != tag) {
        const unsigned long long t0 = globaltimer_ns();
        do {
            asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(lo), "=r"(f0), "=r"(hi), "=r"(f1) : "l"(src) : "memory");
            if (globaltimer_ns() - t0 > spin_ns) {
                if (host_err) {
                    *host_err = -1;
                    __threadfence_system();
                }
                __trap();
            }
        } while (f0 != tag || f1 != tag);
    }
    return __hiloint2double((int)hi, (int)lo);
}
// tag of the exchange the running mat-vec produces / the running consumer kernel reads.
// ctl->epoch only changes in exchange_consumed(), never while either of them is reading it.
__device__ __forceinline__ unsigned exchange_tag(const Ctl *ctl) { return (unsigned)(ctl->epoch + 1ULL); }

// The consumers' view of the gathered result.
struct GatherView {
    const double *plain;
    const uint4 *ll;
    unsigned tag;
    int p2p;
    unsigned long long spin_ns;
    int *host_err;
};
__device__ __forceinline__ GatherView gather_view(const double *apx, const Gather &g)
{
    GatherView v;
    v.plain = apx;
    v.p2p = g.p2p;
    v.tag = g.p2p ? exchange_tag(g.ctl) : 0u;
    v.ll = g.ll + (long long)(v.tag & 1u) * g.bufstride;
    v.spin_ns = g.spin_ns;
    v.host_err = g.host_err;
    return v;
}
__device__ __forceinline__ double gather_read(const GatherView &v, long long idx)
{
    return v.p2p ? ll_load(v.ll + idx, v.tag, v.spin_ns, v.host_err) : v.plain[idx];
}
// Called by ALL threads of every block of a consumer kernel after its last gather_read: the
// last block to finish advances the epoch, so the next mat-vec tags (and double-buffers) anew.
__device__ __forceinline__ void exchange_consumed(const Gather &g, int tid)
{
    if (g.p2p) {
        __syncthreads();
        if (tid == 0) {
            const unsigned t = atomicAdd(&g.ctl->arrive, 1u);
            if (t == gridDim.x - 1) {
                g.ctl->arrive = 0;
                g.ctl->epoch = g.ctl->epoch + 1ULL;
            }
        }
    }
}

__device__ __forceinline__ long long gather_index_raw(long long n_loc, int world, long long slot, long long loc_cap,
                                                      long long i)
{
    long long r = i / n_loc;
    if (r > world - 1) r = world - 1;
    long long l = i - r * n_loc;
    if (l >= loc_cap) l = loc_cap - 1; // only in "loopback" (see Gather::loc_cap)
    return r * slot + l;
}
__device__ __forceinline__ long long gather_index(const Gather &g, long long i)
{
    return gather_index_raw(g.n_loc, g.world, g.slot, g.loc_cap, i);
}

// Called by one full warp of block 0 before it starts streaming: nobody else touches these
// scalars while a mat-vec is running, so rsold / iter advance without a race.
__device__ __forceinline__ void advance_state(const GemvArgs &a, int lane)
{
    const double s = warp_det_sum(a.rrpart, a.nchunks, lane);
    if (lane == 0) {
        State *st = a.st;
        const long long it = st->iter;
        if (it >= 0 && a.hist) a.hist[it] = s; // r'r of loop index `it`
        st->rsold = s;                          // cg.cc:132 rsold = rsnew (cg.cc:91 when it == -1)
        st->rsnew = s;
        st->iter = it + 1;
    }
}

// One result (a row of Ap) into the gather buffer: locally, or --
// fused exchange -- as a self-flagging LL entry straight into every rank's buffer over NVLink
// (peer stores).  That store IS the all-gather: no fence, no flag, no collective kernel.
// Called by ALL lanes of a warp with the same value: in fused mode lane g stores to rank g -- one
// store instruction with `world` transactions in flight (a loop in one lane serialises the
// strong.sys stores: ~0.35 us each on the local GPU, a NVLink round trip each to a peer).
__device__ __forceinline__ void store_out(const GemvArgs &a, long long plain_off, long long ll_off,
                                          unsigned tag, double v, int lane)
{
    if (!a.p2p) {
        if (lane == 0) a.base[plain_off] = v;
    } else if (lane < a.world) {
        ll_store(a.peer_ll[lane] + ll_off, v, tag);
    }
}

// ------------------------------------------------------------------ programmatic dependent launch
// A kernel launched with the programmatic-stream-serialization attribute may become resident
// before its predecessor has finished; everything it reads from the predecessor must come
// after griddep_wait().  Both are no-ops in a kernel launched the ordinary way.
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch_dependents()
{
    asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
}

// ------------------------------------------------------------------ mbarrier / TMA
__device__ __forceinline__ uint32_t smem_u32(const void *p)
{
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init()
{
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes)
                 : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t *bar, uint32_t parity)
{
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity)
        : "memory");
    return ok != 0;
}
// Bounded wait: a pipeline bug must fault the launch (trap), never hang the GPU.
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    if (mbar_try_wait(bar, parity)) return;
    const long long t0 = clock64();
    while (!mbar_try_wait(bar, parity)) {
        if (clock64() - t0 > 8000000000LL) __trap();
    }
}
__device__ __forceinline__ uint64_t l2_policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t l2_policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
// 1-D bulk copy global -> shared through the TMA unit, completion on an mbarrier.
// dst/src 16-byte aligned, bytes a multiple of 16.
__device__ __forceinline__ void bulk_g2s(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar,
                                         uint64_t policy)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint "
        "[%0], [%1], %2, [%3], %4;" ::"r"(smem_u32(dst_smem)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar)), "l"(policy)
        : "memory");
}
__device__ __forceinline__ void bulk_g2s_nohint(void *dst_smem, const void *src, uint32_t bytes, uint64_t *bar)
{
    asm volatile(
        "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
            smem_u32(dst_smem)),
        "l"(src), "r"(bytes), "r"(smem_u32(bar))
        : "memory");
}
// Asynchronous prefetch of `bytes` (multiple of 16) into L2 through the TMA unit; no completion.
__device__ __forceinline__ void bulk_prefetch_l2(const void *src, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(src), "r"(bytes) : "memory");
}
__device__ __forceinline__ void named_bar_sync(int id, int nthreads)
{
    asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory");
}
// streaming 128-bit load that does not allocate in L1 (direct-load mat-vec variant)
__device__ __forceinline__ double2 ldg_stream_f64x2(const double *p)
{
    double2 r;
    asm volatile("ld.global.nc.L1::no_allocate.v2.f64 {%0, %1}, [%2];" : "=d"(r.x), "=d"(r.y) : "l"(p));
    return r;
}

} // namespace cgb
