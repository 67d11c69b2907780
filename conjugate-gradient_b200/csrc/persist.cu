// persist.cu -- the whole CG loop (code/MPI/cg.cc:96-137) as ONE persistent cooperative kernel.
//
// The graph schedule (gemv.cu + vec.cu: four kernels per iteration from a CUDA graph, chained
// with programmatic dependent launch) serialises, every iteration, mat-vec -> vector updates ->
// mat-vec through kernel boundaries; its %globaltimer timeline (profiles/r02/README.md) shows
// ~11 us of such chain plus ~5 us of start skew per iteration on the 8-way shard (5000 x 40000,
// 230 us of streaming).  Here one CTA per SM stays resident for all iterations; the iteration's
// data dependencies -- the reference's MPI_Allgatherv + 2 x MPI_Allreduce (cg.cc:105-136) --
// are data-flow waits inside the kernel, and the producer warp never stops streaming A:
//
//   phase M  mat-vec of this CTA's rows (the tile pipeline of gemv.cu, same summation order, but
//            with full stages for any rows-per-CTA ratio); every finished row goes straight into
//            EVERY rank's gather buffer as a self-flagging LL entry (NVLink peer stores; the
//            same entries are the intra-GPU synchronisation, so also on 1 GPU).
//   phase U  the CTA owns the 256-element chunks c, c + grid, ... of the replicated vectors and
//            keeps their x, r, p IN REGISTERS for the whole launch.  It polls the Ap entries of
//            its chunks (rows of any CTA of any rank), publishes the chunk partials of p'Ap as LL
//            entries, polls all of them -> p'Ap, alpha; x += alpha p, r -= alpha Ap; publishes the
//            chunk partials of r'r.
//   phase B  polls all r'r partials -> stop test, beta; p = r + beta p for the own chunks, stored
//            to the global p vector, red.release on a counter.
//   producer warp: meanwhile already has the first A tiles of the next mat-vec in the shared-
//            memory ring (A never changes) and a few more prefetched into L2; ld.acquire on the p
//            counter, fence.proxy.async, then the p slices.
//   re-balancing: no reduction depends on which CTA computed a row, so the rows are
//            re-partitioned between the CTAs from the mat-vec-phase times they publish (SMs differ
//            persistently in the HBM bandwidth they obtain) -- without changing a result bit.
//
// Every reduction has the order of oracle/cg_oracle.c (lane-order row dot; chunk256 partials of
// the GLOBAL vector + det_sum for p'Ap and r'r alike), so the result is bitwise equal to the graph
// schedule, to the CPU oracle, and the same for 1, 2, 4, 8 GPUs.  All scalars are computed
// redundantly by every CTA of every rank from identical data: no all-reduce, no host round trip,
// no launch per iteration; the kernel leaves the loop by itself on sqrt(r'r) < tol (cg.cc:120-121).
//
// CTAs wait on one another, so the launch is cooperative (co-residency is guaranteed or the
// launch fails).  Ranks on other GPUs are waited for through the LL entries they write, exactly
// as in the fused exchange of the graph schedule; every wait is bounded (spin_timeout_ms).
#include "cgb_device.cuh"
#include "cgb_kernels.h"

namespace cgb {

namespace {

// doubles of p a pipeline stage can hold = the widest tile a CTA may choose: an eighth of the
// A slot (a 16-row x 512 slot may be used as 8 rows x 1024), never less than the nominal width
__host__ __device__ constexpr int persist_pmax(int slot, int tc) { return slot / 8 > tc ? slot / 8 : tc; }
// 256-chunks of the replicated vectors one CTA can own (their x, r, p live in registers: 9 warps
// leave 168 registers per thread): N <= 2 * 148 * 256 = 75776; larger systems take the graph schedule
constexpr int kPersistMaxChunks = 2;

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
__device__ __forceinline__ void fence_proxy_async_global()
{
    asm volatile("fence.proxy.async.global;" ::: "memory");
}
__device__ __forceinline__ uint4 ld_volatile_v4(const uint4 *p)
{
    uint4 v;
    asm volatile("ld.volatile.global.v4.u32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w)
                 : "l"(p)
                 : "memory");
    return v;
}

// A wait that can only end badly is reported before it faults the launch: the host finds the
// code in the mapped flag and returns CGB_ERR_TIMEOUT instead of a bare "unspecified failure".
__device__ __noinline__ void spin_timeout(const PersistArgs &a, int what, int d0 = 0, int d1 = 0, int d2 = 0,
                                          int d3 = 0)
{
    if (a.host_done) {
        if (*(volatile int *)a.host_done >= 0) { // (racy on purpose) an early report; context for the message
            a.host_done[1] = (int)blockIdx.x;
            a.host_done[2] = (int)threadIdx.x;
            a.host_done[3] = d0;
            a.host_done[4] = d1;
            a.host_done[5] = d2;
            a.host_done[6] = d3;
            __threadfence_system();
            *a.host_done = -(what);
        }
        __threadfence_system();
    }
    __trap();
}

// PB LL entries at once: all pending loads are in flight together in every round (polling them
// one after the other costs a round trip per late entry)
template <int PB>
__device__ __forceinline__ void ll_wait_batch(const PersistArgs &a, const uint4 *const (&src)[PB], unsigned pending,
                                              unsigned tag, double (&out)[PB])
{
    uint4 v[PB];
#pragma unroll
    for (int u = 0; u < PB; ++u)
        if ((pending >> u) & 1u) v[u] = ld_volatile_v4(src[u]);
    unsigned long long t0 = 0;
    unsigned ns = 20;
    for (;;) {
#pragma unroll
        for (int u = 0; u < PB; ++u)
            if (((pending >> u) & 1u) && v[u].y == tag && v[u].w == tag) {
                out[u] = __hiloint2double((int)v[u].z, (int)v[u].x);
                pending &= ~(1u << u);
            }
        if (!pending) return;
        if (t0 == 0) t0 = globaltimer_ns();
        __nanosleep(ns);
        if (ns < 320) ns += ns; // early CTAs must not hammer L2 while the others still stream
        if (globaltimer_ns() - t0 > a.spin_ns) spin_timeout(a, 1);
#pragma unroll
        for (int u = 0; u < PB; ++u)
            if ((pending >> u) & 1u) v[u] = ld_volatile_v4(src[u]);
    }
}

// det_sum over shared memory with the loads of 8 terms in flight (the adds keep their order)
__device__ __forceinline__ double warp_det_sum_smem(const double *v, int n, int lane)
{
    double s = 0.0;
    int t = lane;
    for (; t + 7 * 32 < n; t += 8 * 32) {
        double x[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) x[k] = v[t + 32 * k];
#pragma unroll
        for (int k = 0; k < 8; ++k) s = __dadd_rn(s, x[k]);
    }
    for (; t < n; t += 32) s = __dadd_rn(s, v[t]);
    return warp_butterfly(s);
}

__device__ __forceinline__ void prefetch_l2_line(const void *p)
{
    asm volatile("prefetch.global.L2 [%0];" ::"l"(p));
}

// mbarrier wait with the configurable bound (a peer rank may legitimately be seconds late)
__device__ __forceinline__ void mbar_wait_ns(const PersistArgs &a, uint64_t *bar, uint32_t parity, int what,
                                             int d0 = 0, int d1 = 0, int d2 = 0, int d3 = 0)
{
    if (mbar_try_wait(bar, parity)) return;
    const unsigned long long t0 = globaltimer_ns();
    while (!mbar_try_wait(bar, parity)) {
        if (globaltimer_ns() - t0 > a.spin_ns) spin_timeout(a, what, d0, d1, d2, d3);
    }
}

} // namespace

// Geometry of one CTA's mat-vec for a given row range: balanced row blocks of at most TR rows,
// tile width per block as wide as the stage allows (a full stage keeps the bytes in flight -- and
// with them this SM's share of the saturated HBM stream -- independent of the rows-per-CTA ratio).
// Block b streams the columns of its window (block_window) from the table s_win[par][b] in tiles of
// that width; T, the pipeline steps of the mat-vec, is summed from the table by the producer.
struct Geo {
    long long r0;
    int nrows, nb, lo, n_hi, w_lo, w_hi, par;
    unsigned T;
};
template <int TR, int SLOT, int PMAX>
__device__ __forceinline__ Geo make_geo(long long r0, long long r1, int par)
{
    Geo g;
    g.r0 = r0;
    g.par = par;
    g.T = 0;
    g.nrows = (int)(r1 - r0);
    g.nb = (g.nrows + TR - 1) / TR;
    g.lo = g.nb ? g.nrows / g.nb : 1; // the balanced split gives blocks of lo or lo + 1 rows
    g.n_hi = g.nb ? g.nrows - g.lo * g.nb : 0;
    int w = (SLOT / g.lo) & ~63;
    g.w_lo = w > PMAX ? PMAX : w;
    w = (SLOT / (g.lo + 1)) & ~63;
    g.w_hi = w > PMAX ? PMAX : w;
    return g;
}

constexpr int kMaxGrid = 160; // CTAs of the persistent grid (one per SM) the re-balancing handles

template <int CW, int RPW, int TC, int STAGES, int MAXC>
__global__ void __launch_bounds__((CW + 1) * 32, 1) cg_persist_kernel(const PersistArgs a)
{
    constexpr int TR = CW * RPW;            // most rows of a row block
    constexpr int SLOT = TR * TC;           // doubles of A per pipeline stage
    constexpr int PMAX = persist_pmax(SLOT, TC); // doubles of p per pipeline stage = widest tile
    constexpr int NCT = CW * 32;            // consumer threads
    constexpr int EPT = kChunk / NCT;       // elements of a 256-chunk per consumer thread
    static_assert(CW == 4 || CW == 8, "chunk256 mapping is written for 4 or 8 consumer warps");
    static_assert(TC % 64 == 0, "tile width must be a multiple of 64 doubles");
    static_assert(STAGES <= 8, "stage metadata");
    extern __shared__ __align__(128) unsigned char smem_raw[];
    double *sA = reinterpret_cast<double *>(smem_raw);            // [STAGES][SLOT]
    double *sP = sA + (size_t)STAGES * SLOT;                      // [STAGES][PMAX]
    uint64_t *full = reinterpret_cast<uint64_t *>(sP + (size_t)STAGES * PMAX);
    uint64_t *empty = full + STAGES;
    double *wsum = reinterpret_cast<double *>(empty + STAGES);    // [MAXC][8]
    double *s_sc = wsum + MAXC * 8;                               // [4] broadcast scalars
    double *scr = s_sc + 4;                                       // [nchunks] chunk partials being summed
    __shared__ volatile int s_stop;          // consumers -> producer: loop left
    __shared__ volatile int s_part_seq;      // highest iteration whose row partition is in s_bnd
    __shared__ volatile int s_prod_geo;      // highest iteration whose row partition the producer has read
                                             // and whose window table it has written
    __shared__ unsigned s_win[2][kWinBlocks]; // column window of every row block, iteration parity
    __shared__ int s_bnd[2][kMaxGrid + 1];   // row boundaries of all CTAs, iteration parity
    __shared__ double s_tm[kMaxGrid];        // mat-vec-phase times of all CTAs (re-balancing)
    __shared__ long long s_c0[8];            // per stage: first column and width of the tile in flight
    __shared__ int s_w[8];

    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int nblk = gridDim.x, c = blockIdx.x;
    // re-balancing moves whole rows: worth it from ~64 rows per CTA on (one row = 1.5 % of a CTA's work);
    // below that its granularity is coarser than the imbalance it removes (measured: -0.5 % at 34 rows)
    const bool balance = a.balance != 0 && nblk <= kMaxGrid && a.rows >= 64LL * nblk;

    if (tid == 0) {
        for (int s = 0; s < STAGES; ++s) {
            mbar_init(&full[s], 1);
            mbar_init(&empty[s], CW);
        }
        fence_mbar_init();
        s_stop = 0;
        s_part_seq = 1;
        s_prod_geo = -1;
    }
    if (nblk <= kMaxGrid)
        for (int k = tid; k <= nblk; k += blockDim.x) { // static start: the balanced split of gemv.cu
            const int bk = (int)((long long)k * a.rows / nblk);
            s_bnd[0][k] = bk;
            s_bnd[1][k] = bk;
        }
    __syncthreads();
    if (a.st->done) return; // converged in an earlier launch: nothing to do (uniform)

    const unsigned nchunks = (unsigned)a.nchunks;
    auto geo_of = [&](int m) {
        if (nblk <= kMaxGrid) return make_geo<TR, SLOT, PMAX>(s_bnd[m & 1][c], s_bnd[m & 1][c + 1], m & 1);
        return make_geo<TR, SLOT, PMAX>((long long)c * a.rows / nblk, (long long)(c + 1) * a.rows / nblk, m & 1);
    };

    if (warp == CW) {
        // ================= producer: streams A, never waits for the vector phases =================
        const uint64_t pol_a = l2_policy_evict_first();
        const uint64_t pol_p = l2_policy_evict_last();
        // the window table of a mat-vec (its slot is free: see the wait for s_part_seq) and its steps T
        auto take_windows = [&](Geo &ge) {
            unsigned T = 0;
            for (int b = lane; b < ge.nb; b += 32) {
                const long long rb0 = ge.r0 + (long long)b * ge.nrows / ge.nb;
                const int nr = (int)(ge.r0 + (long long)(b + 1) * ge.nrows / ge.nb - rb0);
                if (b < kWinBlocks && a.ld <= kWinMaxLd) s_win[ge.par][b] = block_window(a.env, rb0, nr, a.ld);
                long long cb, ce;
                window_of(s_win[ge.par], b, a.ld, cb, ce);
                T += (unsigned)window_tiles(cb, ce, (nr == ge.lo) ? ge.w_lo : ge.w_hi);
            }
            ge.T = __reduce_add_sync(0xffffffffu, T);
            __syncwarp(); // the table is read by every lane from here on
        };
        // cursor over the pipeline steps (row block b, column tile t) of one mat-vec
        struct Cur {
            int b, t, nr, wdb, ntb;
            long long rb0, cb, ce;
        };
        // the first block from b on (wrapping around) with a tile to stream; none (T == 0): ntb = 0
        auto cur_block = [&](Cur &k, const Geo &ge, int b) {
            k.t = 0;
            k.nr = 0; k.wdb = 64; k.ntb = 0; k.rb0 = ge.r0; k.cb = 0; k.ce = 0; k.b = 0;
            for (int n = 0; n < ge.nb; ++n, ++b) {
                if (b >= ge.nb) b = 0;
                k.b = b;
                k.rb0 = ge.r0 + (long long)b * ge.nrows / ge.nb;
                k.nr = (int)(ge.r0 + (long long)(b + 1) * ge.nrows / ge.nb - k.rb0);
                k.wdb = (k.nr == ge.lo) ? ge.w_lo : ge.w_hi;
                window_of(s_win[ge.par], b, a.ld, k.cb, k.ce);
                k.ntb = window_tiles(k.cb, k.ce, k.wdb);
                if (k.ntb > 0) return;
            }
        };
        auto cur_next = [&](Cur &k, const Geo &ge) {
            if (++k.t >= k.ntb) cur_block(k, ge, k.b + 1);
        };
        // first column and width of the tile under the cursor
        auto cur_tile = [&](const Cur &k, long long &c0, int &w) {
            c0 = k.cb + (long long)k.t * k.wdb;
            w = (int)((k.ce - c0 < k.wdb) ? (k.ce - c0) : k.wdb);
        };
        auto issueA = [&](unsigned g, const Cur &k) {
            long long c0;
            int w;
            cur_tile(k, c0, w);
            const int stage = g % STAGES;
            if (lane == 0) {
                s_c0[stage] = c0;
                s_w[stage] = w;
                mbar_arrive_expect_tx(&full[stage], (unsigned)((k.nr + 1) * w * 8));
            }
            __syncwarp();
            double *dstA = sA + (size_t)stage * SLOT;
            for (int j = lane; j < k.nr; j += 32)
                bulk_g2s(dstA + (size_t)j * k.wdb, a.A + (k.rb0 + j) * a.ld + c0, (unsigned)(w * 8), &full[stage], pol_a);
        };
        auto issueP = [&](unsigned g) {
            const int stage = g % STAGES;
            if (lane == 0)
                bulk_g2s(sP + (size_t)stage * PMAX, a.p + s_c0[stage], (unsigned)(s_w[stage] * 8), &full[stage], pol_p);
        };
        auto wait_empty = [&](unsigned g) {
            if (g >= (unsigned)STAGES) mbar_wait_ns(a, &empty[g % STAGES], ((g / STAGES) & 1u) ^ 1u, 7, (int)g);
        };
        Geo ge = geo_of(0);
        take_windows(ge);
        Cur cur;
        cur_block(cur, ge, 0);
        if (lane == 0) {
            __threadfence_block();
            s_prod_geo = 0;
        }
        unsigned gbase = 0; // global step index of the first tile of mat-vec m
        unsigned pre = 0;   // steps of the coming mat-vec whose A part is already in flight
        for (int m = 0; m < a.iters; ++m) {
            if (m > 0 && (ge.T > 0 || pre > 0)) {
                // p of this mat-vec is final once every chunk owner has published it -- or the
                // loop was left (converged): then only the copies in flight must still land
                int stop = 0;
                if (lane == 0) {
                    const unsigned target = nchunks * (unsigned)m;
                    const unsigned long long t0 = globaltimer_ns();
                    while (ld_acquire_u32(&a.sync->arrive_p) < target) {
                        if (s_stop) {
                            stop = 1;
                            break;
                        }
                        if (globaltimer_ns() - t0 > a.spin_ns) spin_timeout(a, 4);
                    }
                    fence_proxy_async_global(); // the chunk owners' stores to p are read through the async proxy (TMA)
                }
                stop = __shfl_sync(0xffffffffu, stop, 0);
                if (stop) {
                    for (unsigned u = 0; u < pre; ++u) issueP(gbase + u);
                    for (unsigned u = 0; u < pre; ++u)
                        mbar_wait_ns(a, &full[(gbase + u) % STAGES], ((gbase + u) / STAGES) & 1u, 8, m, (int)gbase, (int)pre,
                                     (int)ge.T);
                    return;
                }
            }
            for (unsigned u = 0; u < pre; ++u) issueP(gbase + u);
            if (a.l2_ramp > 0 && m > 0) {
                // the steps already on chip (ring + L2) are consumed faster than HBM delivers: keep HBM
                // busy meanwhile with the steps after them
                Cur pf = cur;
                unsigned u = pre;
                for (int q = 0; q < a.l2_prefetch && u < ge.T; ++q, ++u) cur_next(pf, ge);
                for (int q = 0; q < a.l2_ramp && u < ge.T; ++q, ++u) {
                    long long c0;
                    int w;
                    cur_tile(pf, c0, w);
                    for (int j = lane; j < pf.nr; j += 32)
                        bulk_prefetch_l2(a.A + (pf.rb0 + j) * a.ld + c0, (unsigned)(w * 8));
                    cur_next(pf, ge);
                }
            }
            for (unsigned g = gbase + pre; g < gbase + ge.T; ++g) {
                wait_empty(g);
                issueA(g, cur);
                cur_next(cur, ge);
                issueP(g);
            }
            gbase += ge.T;
            pre = 0;
            if (m + 1 < a.iters) {
                // the row range of the next mat-vec (re-balanced two iterations ago; s_part_seq is also
                // raised without re-balancing: the consumers are then past mat-vec m - 1, so the slot
                // of its window table can take the next one) ...
                int stop = 0;
                if (lane == 0) {
                    const unsigned long long t0 = globaltimer_ns();
                    while (s_part_seq < m + 1 && !s_stop) {
                        __nanosleep(64);
                        if (globaltimer_ns() - t0 > a.spin_ns) spin_timeout(a, 6);
                    }
                    stop = s_stop;
                }
                // ONE lane decides for the warp: s_stop may be raised at this very moment, and lanes that
                // read it themselves could disagree -- part of the warp (lane 0, which arms the barriers,
                // perhaps among them) would leave while the rest went on issuing copies
                stop = __shfl_sync(0xffffffffu, stop, 0);
                __threadfence_block();
                if (stop) return; // nothing in flight: all steps of mat-vec m were consumed or the loop never reached it
                ge = geo_of(m + 1);
                take_windows(ge);
                cur_block(cur, ge, 0);
                __syncwarp();
                if (lane == 0) {
                    __threadfence_block();
                    s_prod_geo = m + 1; // its slot may be re-used for mat-vec m + 3 from now on
                }
                // ... run ahead into it: A tiles into the ring as its stages drain (A never changes),
                // the steps after them into L2, while the vector phases of this iteration run
                const unsigned npre = ge.T < (unsigned)STAGES ? ge.T : (unsigned)STAGES;
                for (; pre < npre; ++pre) {
                    wait_empty(gbase + pre);
                    issueA(gbase + pre, cur);
                    cur_next(cur, ge);
                }
                Cur pf = cur;
                for (int u = 0; u < a.l2_prefetch && (unsigned)u + pre < ge.T; ++u) {
                    long long c0;
                    int w;
                    cur_tile(pf, c0, w);
                    for (int j = lane; j < pf.nr; j += 32)
                        bulk_prefetch_l2(a.A + (pf.rb0 + j) * a.ld + c0, (unsigned)(w * 8));
                    cur_next(pf, ge);
                }
            }
        }
        return;
    }

    // ======================================= consumers =======================================
    const long long it0 = a.st->iter;                       // loop bodies book-kept so far - 1 ...
    const unsigned epoch0 = (unsigned)a.ctl->epoch;         // exchanges consumed so far
    unsigned long long *const trace = a.trace.buf;
    const unsigned tr0 = (trace && tid == 0) ? a.trace.cnt[c] : 0u; // iterations traced before this launch

    // chunks of the replicated vectors this CTA owns: c, c + grid, ...; element el of a chunk
    // belongs to consumer thread el % NCT (32-group el / 32 = warp + e * CW)
    double xs[MAXC][EPT], rs[MAXC][EPT], ps[MAXC][EPT];
    unsigned mychunks = 0;
#pragma unroll
    for (int cc = 0; cc < MAXC; ++cc) {
        const long long j = (long long)c + (long long)cc * nblk;
        if (j < a.nchunks) ++mychunks;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const long long i = j * kChunk + tid + e * NCT;
            const bool ok = j < a.nchunks && i < a.n;
            xs[cc][e] = ok ? a.x[i] : 0.0;
            rs[cc][e] = ok ? a.r[i] : 0.0;
            ps[cc][e] = ok ? a.p[i] : 0.0;
        }
    }
    // deferred book-keeping of the previous loop body (advance_state of the graph schedule):
    // rsold = r'r from the chunk partials the previous kernel left in rrpart
    for (unsigned t = tid; t < nchunks; t += NCT) scr[t] = a.rrpart[t];
    named_bar_sync(1, NCT);
    if (warp == 0) {
        const double s = warp_det_sum_smem(scr, (int)nchunks, lane);
        if (lane == 0) {
            s_sc[0] = s;
            if (c == 0 && it0 >= 0 && a.hist) a.hist[it0] = s;
        }
    }
    named_bar_sync(1, NCT);
    double rsold = s_sc[0];
    double rsnew = rsold, alpha = 0.0, conj = 0.0;
    int converged = 0, executed = 0;

    // chunk256 of one value per owned element: butterfly inside the 32-groups, group g + group g + 4
    // inside the thread (CW == 4), the rest of the perfect tree across the warps by warp 0, which
    // publishes every partial as a self-flagging LL entry (no fence, no counter) -- and, for r'r,
    // also plainly in rrpart for the hand-over to the next launch.
    auto publish_chunk_partials = [&](const double (&val)[MAXC][EPT], uint4 *dst_ll, unsigned tag, double *plain) {
#pragma unroll
        for (int cc = 0; cc < MAXC; ++cc) {
            double v = 0.0;
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const double bf = warp_butterfly(val[cc][e]);
                v = (e == 0) ? bf : __dadd_rn(v, bf);
            }
            if (lane == 0) wsum[cc * 8 + warp] = v;
        }
        named_bar_sync(1, NCT);
        if (warp == 0) {
#pragma unroll
            for (int cc = 0; cc < MAXC; ++cc) {
                const long long j = (long long)c + (long long)cc * nblk;
                if (j < a.nchunks) {
                    double t = (lane < CW) ? wsum[cc * 8 + lane] : 0.0;
                    if (CW == 8) t = __dadd_rn(t, shfl_xor_f64(t, 4));
                    t = __dadd_rn(t, shfl_xor_f64(t, 2));
                    t = __dadd_rn(t, shfl_xor_f64(t, 1));
                    if (lane == 0) {
                        ll_store(dst_ll + j, t, tag);
                        if (plain) plain[j] = t;
                    }
                }
            }
        }
        named_bar_sync(1, NCT); // wsum may be reused
    };
    // all chunk partials of one reduction -> their det_sum, in every consumer thread
    auto collect_chunk_partials = [&](const uint4 *src_ll, unsigned tag, int slot_sc) {
        constexpr int PB = 3;
        for (unsigned t0 = tid; t0 < nchunks; t0 += PB * NCT) {
            const uint4 *src[PB];
            double val[PB];
            unsigned pending = 0;
#pragma unroll
            for (int u = 0; u < PB; ++u) {
                src[u] = src_ll + t0 + u * NCT;
                if (t0 + u * NCT < nchunks) pending |= 1u << u;
            }
            ll_wait_batch<PB>(a, src, pending, tag, val);
#pragma unroll
            for (int u = 0; u < PB; ++u)
                if (t0 + u * NCT < nchunks) scr[t0 + u * NCT] = val[u];
        }
        named_bar_sync(1, NCT);
        if (warp == 0) {
            const double s = warp_det_sum_smem(scr, (int)nchunks, lane);
            if (lane == 0) s_sc[slot_sc] = s;
        }
        named_bar_sync(1, NCT);
        return s_sc[slot_sc];
    };

    unsigned g = 0; // pipeline step counter, never reset (mbarrier parities)
    for (int m = 0; m < a.iters; ++m) {
        const long long jloop = it0 + 1 + m;             // the reference's k of this loop body
        const unsigned tag = epoch0 + 1u + (unsigned)m;  // tag + buffer of this exchange
        const long long lbase = (long long)(tag & 1u) * a.bufstride + a.slot_off;
        const uint4 *const view = a.ll + (long long)(tag & 1u) * a.bufstride;
        uint4 *const aux = a.rr_ll + (long long)(tag & 1u) * a.rr_stride; // [r'r | p'Ap | times]
        uint4 *const rrview = aux, *const papview = aux + a.nchunks, *const tmview = aux + 2 * a.nchunks;
        const Geo ge = geo_of(m);
        if (s_prod_geo < m) { // the window table of this mat-vec (normally written an iteration ago)
            const unsigned long long t0 = globaltimer_ns();
            while (s_prod_geo < m)
                if (globaltimer_ns() - t0 > a.spin_ns) spin_timeout(a, 10, m);
        }
        __threadfence_block();
        // the two parities of the partition are re-balanced in turn, two iterations out of eight
        const bool rebalance_now = balance && (m & 7) < 2 && m + 2 < a.iters;
        unsigned long long *rec = nullptr;
        if (trace && tid == 0) {
            rec = trace + ((size_t)((tr0 + (unsigned)m) % (unsigned)a.trace.cap) * (size_t)nblk + (size_t)c) * kTraceWords;
            rec[0] = globaltimer_ns();
            rec[7] = (unsigned long long)smid() | ((unsigned long long)ge.nrows << 32);
        }

        // ------------------------------------------------ phase M: Ap rows of this CTA (cg.cc:100-102)
        unsigned long long tm0 = 0;
        const unsigned g_mv = g; // first step of this mat-vec
        for (int b = 0; b < ge.nb; ++b) {
            const long long rb0 = ge.r0 + (long long)b * ge.nrows / ge.nb;
            const int nr = (int)(ge.r0 + (long long)(b + 1) * ge.nrows / ge.nb - rb0);
            const int nv = (nr > warp) ? ((nr - warp + CW - 1) / CW) : 0;
            const int wd = (nr == ge.lo) ? ge.w_lo : ge.w_hi;
            long long cb, ce;
            window_of(s_win[ge.par], b, a.ld, cb, ce);
            const int ntc = window_tiles(cb, ce, wd); // 0: the block's rows are +0
            double acc0[RPW], acc1[RPW];
#pragma unroll
            for (int s = 0; s < RPW; ++s) {
                acc0[s] = 0.0;
                acc1[s] = 0.0;
            }
            for (int t = 0; t < ntc; ++t, ++g) {
                const int stage = g % STAGES;
                const unsigned ph = (g / STAGES) & 1u;
                const long long c0 = cb + (long long)t * wd;
                const int w = (int)((ce - c0 < wd) ? (ce - c0) : wd);
                mbar_wait_ns(a, &full[stage], ph, 5, m, (int)g, b, t);
                if (tid == 0 && g == g_mv) {
                    tm0 = globaltimer_ns();
                    if (rec) rec[3] = tm0;
                }
                const double2 *sa2 = reinterpret_cast<const double2 *>(sA + (size_t)stage * SLOT);
                const double2 *sp2 = reinterpret_cast<const double2 *>(sP + (size_t)stage * PMAX);
                const int pitch2 = wd >> 1; // tile row pitch in 16-byte chunks
                if (nv == RPW) {
                    const int full_it = w >> 6; // 64 columns per warp pass
#pragma unroll 4
                    for (int i = 0; i < full_it; ++i) {
                        const int q = lane + 32 * i;
                        const double2 pv = sp2[q];
#pragma unroll
                        for (int s = 0; s < RPW; ++s) {
                            const double2 av = sa2[(warp + s * CW) * pitch2 + q];
                            acc0[s] = __fma_rn(av.x, pv.x, acc0[s]);
                            acc1[s] = __fma_rn(av.y, pv.y, acc1[s]);
                        }
                    }
                    const int q = lane + 32 * full_it; // ragged end of the last tile (ld is a multiple of 16)
                    if (q < (w >> 1)) {
                        const double2 pv = sp2[q];
#pragma unroll
                        for (int s = 0; s < RPW; ++s) {
                            const double2 av = sa2[(warp + s * CW) * pitch2 + q];
                            acc0[s] = __fma_rn(av.x, pv.x, acc0[s]);
                            acc1[s] = __fma_rn(av.y, pv.y, acc1[s]);
                        }
                    }
                } else {
                    const int nq = w >> 1;
                    for (int q = lane; q < nq; q += 32) {
                        const double2 pv = sp2[q];
#pragma unroll
                        for (int s = 0; s < RPW; ++s) {
                            if (s < nv) {
                                const double2 av = sa2[(warp + s * CW) * pitch2 + q];
                                acc0[s] = __fma_rn(av.x, pv.x, acc0[s]);
                                acc1[s] = __fma_rn(av.y, pv.y, acc1[s]);
                            }
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[stage]);
            }
            // row epilogue: butterfly, Ap_row straight to every rank (lane g -> rank g: ONE store
            // instruction, `world` transactions in flight)
#pragma unroll
            for (int s = 0; s < RPW; ++s) {
                if (s < nv) {
                    const double y = warp_butterfly(__dadd_rn(acc0[s], acc1[s])); // every lane holds y
                    const long long li = rb0 + warp + s * CW;
                    if (lane < a.world) ll_store(a.peer_ll[lane] + lbase + li, y, tag);
                }
            }
        }
        const bool streamed = g != g_mv;
        if (tid == 0 && !streamed && ge.nb > 0) { // rows, but no block had a column to stream
            tm0 = globaltimer_ns();
            if (rec) rec[3] = tm0;
        }
        if (rebalance_now || trace) { // uniform over the CTA
            named_bar_sync(1, NCT); // all rows of this CTA are stored
            if (tid == 0) {
                const unsigned long long t1 = globaltimer_ns();
                if (rec) rec[5] = t1;
                // the time this CTA streamed its rows in: the input of the re-balancing (no reading
                // without a streamed tile: such a CTA gets the mean speed)
                if (rebalance_now) ll_store(tmview + c, streamed ? (double)(t1 - tm0) : 0.0, tag);
            }
        }

        // ------------------------------------------------ phase U: p'Ap, alpha, x, r, r'r (cg.cc:105-116)
        // The Ap values of the own chunks, polled straight from the LL entries the owning CTAs (of
        // any rank) stored; they serve both p'Ap and the r update.
        double apv[MAXC * EPT];
        {
            const uint4 *esrc[MAXC * EPT];
            unsigned pending = 0;
#pragma unroll
            for (int cc = 0; cc < MAXC; ++cc) {
                const long long j = (long long)c + (long long)cc * nblk;
#pragma unroll
                for (int e = 0; e < EPT; ++e) {
                    const long long i = j * kChunk + tid + e * NCT;
                    const bool ok = j < a.nchunks && i < a.n;
                    esrc[cc * EPT + e] = view + gather_index_raw(a.n_loc, a.world, a.slot, a.loc_cap, ok ? i : 0);
                    if (ok) pending |= 1u << (cc * EPT + e);
                }
            }
            ll_wait_batch<MAXC * EPT>(a, esrc, pending, tag, apv);
        }
        {
            double q[MAXC][EPT];
#pragma unroll
            for (int cc = 0; cc < MAXC; ++cc)
#pragma unroll
                for (int e = 0; e < EPT; ++e) {
                    const long long j = (long long)c + (long long)cc * nblk;
                    const long long i = j * kChunk + tid + e * NCT;
                    q[cc][e] = (j < a.nchunks && i < a.n) ? __dmul_rn(ps[cc][e], apv[cc * EPT + e]) : 0.0; // cg.cc:105
                }
            publish_chunk_partials(q, papview, tag, nullptr);
        }
        conj = collect_chunk_partials(papview, tag, 3);                               // cg.cc:105-106
        {
            const double clamp = __dmul_rn(rsold, kNearZero);
            alpha = __ddiv_rn(rsold, (conj < clamp) ? clamp : conj);                  // cg.cc:107
        }
        if (rec) rec[1] = globaltimer_ns();
        {
            double sq[MAXC][EPT];
#pragma unroll
            for (int cc = 0; cc < MAXC; ++cc)
#pragma unroll
                for (int e = 0; e < EPT; ++e) {
                    const long long j = (long long)c + (long long)cc * nblk;
                    const long long i = j * kChunk + tid + e * NCT;
                    sq[cc][e] = 0.0;
                    if (j < a.nchunks && i < a.n) {
                        xs[cc][e] = __fma_rn(alpha, ps[cc][e], xs[cc][e]);             // cg.cc:110
                        rs[cc][e] = __fma_rn(-alpha, apv[cc * EPT + e], rs[cc][e]);    // cg.cc:113
                        sq[cc][e] = __dmul_rn(rs[cc][e], rs[cc][e]);                   // cg.cc:116
                    }
                }
            publish_chunk_partials(sq, rrview, tag, a.rrpart);
        }
        if (rec) rec[2] = globaltimer_ns();

        // ---- re-balancing (off the critical path: the r'r partials of the other CTAs are still on
        // their way): rows for mat-vec m + 2 in proportion to the speed every CTA showed in this one.
        // Every CTA computes the same boundaries from the same 148 numbers; no result bit depends on them.
        if (warp == CW - 1) {
            const int par = m & 1;
            if (rebalance_now) {
                // this parity's slot still holds the partition of mat-vec m: the producer must have
                // taken it (it normally did an iteration ago; a CTA without rows can run ahead of it)
                if (lane == 0) {
                    const unsigned long long t0 = globaltimer_ns();
                    while (s_prod_geo < m) {
                        __nanosleep(64);
                        if (globaltimer_ns() - t0 > a.spin_ns) spin_timeout(a, 9);
                    }
                }
                __syncwarp();
                constexpr int PER = kMaxGrid / 32;
                const uint4 *src[PER];
                double tmv[PER];
                unsigned pending = 0;
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    src[u] = tmview + lane * PER + u;
                    if (lane * PER + u < nblk) pending |= 1u << u;
                }
                ll_wait_batch<PER>(a, src, pending, tag, tmv);
                // speed of CTA k = rows / time; CTAs without rows (or a zero reading) get the mean speed
                double sp[PER], ssum = 0.0;
                int nz = 0;
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    const int k = lane * PER + u;
                    sp[u] = 0.0;
                    if (k < nblk) {
                        const int rk = s_bnd[par][k + 1] - s_bnd[par][k];
                        if (rk > 0 && tmv[u] > 0.0) {
                            sp[u] = (double)rk / tmv[u];
                            ssum += sp[u];
                            ++nz;
                        }
                    }
                }
#pragma unroll
                for (int off = 16; off >= 1; off >>= 1) {
                    ssum += __shfl_xor_sync(0xffffffffu, ssum, off);
                    nz += __shfl_xor_sync(0xffffffffu, nz, off);
                }
                const double mean = nz > 0 ? ssum / nz : 1.0;
                double lsum = 0.0;
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    if (lane * PER + u < nblk && sp[u] == 0.0) sp[u] = mean;
                    if (lane * PER + u < nblk) lsum += sp[u];
                }
                // exclusive prefix of the speeds over the CTAs (lane-major), total in every lane
                double incl = lsum;
#pragma unroll
                for (int off = 1; off < 32; off <<= 1) {
                    const double up = __shfl_up_sync(0xffffffffu, incl, off);
                    if (lane >= off) incl += up;
                }
                const double total = __shfl_sync(0xffffffffu, incl, 31);
                double run = incl - lsum;
                int nbv[PER];
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    const int k = lane * PER + u;
                    nbv[u] = 0;
                    if (k < nblk) {
                        // boundary k of the speed-proportional split, blended 1:1 with the current one:
                        // floor of a sum of two non-decreasing sequences -- stays non-decreasing
                        const double target = (double)a.rows * (run / total);
                        nbv[u] = (int)(0.5 * (target + (double)s_bnd[par][k]) + 0.5);
                        if (nbv[u] > (int)a.rows) nbv[u] = (int)a.rows;
                        run += sp[u];
                    }
                }
                __syncwarp(); // all reads of the old boundaries are done
#pragma unroll
                for (int u = 0; u < PER; ++u) {
                    const int k = lane * PER + u;
                    if (k > 0 && k < nblk) s_bnd[par][k] = nbv[u]; // ends stay 0 and rows
                }
            }
            __syncwarp();
            if (lane == 0) {
                __threadfence_block();
                s_part_seq = m + 2; // partition of mat-vec m + 2 = this parity's slot, updated or not
            }
        }

        // ------------------------------------------------ phase B: r'r, stop test, beta (cg.cc:116-124)
        rsnew = collect_chunk_partials(rrview, tag, 2);
        executed = m + 1;
        if (rec) rec[4] = globaltimer_ns();
        if (c == 0 && tid == 0 && a.hist) a.hist[jloop] = rsnew;
        if (sqrt(rsnew) < a.tol) { // cg.cc:120-121: leave BEFORE p and rsold are updated
            converged = 1;
            if (tid == 0) s_stop = 1;
            break;
        }
        const double beta = __ddiv_rn(rsnew, rsold); // cg.cc:124
        rsold = rsnew;                               // cg.cc:132
#pragma unroll
        for (int cc = 0; cc < MAXC; ++cc) {
            const long long j = (long long)c + (long long)cc * nblk;
#pragma unroll
            for (int e = 0; e < EPT; ++e) {
                const long long i = j * kChunk + tid + e * NCT;
                if (j < a.nchunks && i < a.n) {
                    ps[cc][e] = __fma_rn(beta, ps[cc][e], rs[cc][e]); // cg.cc:127-129
                    a.p[i] = ps[cc][e];
                }
            }
        }
        if (mychunks) {
            named_bar_sync(1, NCT);
            if (tid == 0) {
                red_release_add_u32(&a.sync->arrive_p, mychunks); // release p[own chunks] to every CTA's producer
                if (rec) rec[6] = globaltimer_ns();
            }
        } else if (rec) {
            rec[6] = globaltimer_ns();
        }
    }
    if (tid == 0) s_stop = 1; // the producer may be waiting for a partition that will never come

    // ---- hand the state back: x, r of the own chunks (p is already in place), scalars by CTA 0
#pragma unroll
    for (int cc = 0; cc < MAXC; ++cc) {
        const long long j = (long long)c + (long long)cc * nblk;
#pragma unroll
        for (int e = 0; e < EPT; ++e) {
            const long long i = j * kChunk + tid + e * NCT;
            if (j < a.nchunks && i < a.n) {
                a.x[i] = xs[cc][e];
                a.r[i] = rs[cc][e];
            }
        }
    }
    if (trace && tid == 0) a.trace.cnt[c] += (unsigned)executed;
    if (c == 0 && tid == 0) {
        State *st = a.st;
        st->conj = conj;
        st->alpha = alpha;
        st->rsnew = rsnew;
        st->rsold = rsold; // converged: the STALE rsold the reference prints (cg.cc:152-153)
        // not converged: "inside loop body it0 + executed" -- rrpart holds its r'r partials; the next
        // launch (or cgb_solve_end) does the deferred rsold = rsnew / iter + 1, as in vec.cu.
        // converged: k = loop index at the break.  Both are it0 + executed.
        st->iter = it0 + executed;
        if (converged) {
            st->done = 1;
            if (a.host_done) *a.host_done = 1;
            __threadfence_system();
        }
        a.ctl->epoch = a.ctl->epoch + (unsigned long long)executed;
    }
}

// --------------------------------------------------------------------------------- host side
namespace {

template <int CW, int RPW, int TC, int STAGES>
size_t persist_smem(const PersistArgs &a)
{
    return (size_t)STAGES * CW * RPW * TC * 8 + (size_t)STAGES * persist_pmax(CW * RPW * TC, TC) * 8 + 2 * STAGES * 8 +
           (kPersistMaxChunks * 8 + 4) * 8 + (size_t)a.scr_n * 8;
}

template <int CW, int RPW, int TC, int STAGES>
cudaError_t persist_launch(const PersistArgs &a, int nblk, cudaStream_t s)
{
    auto k = cg_persist_kernel<CW, RPW, TC, STAGES, kPersistMaxChunks>;
    const size_t smem = persist_smem<CW, RPW, TC, STAGES>(a);
    cudaError_t e = cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)nblk, 1, 1);
    cfg.blockDim = dim3((unsigned)((CW + 1) * 32), 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeCooperative; // CTAs wait on one another: co-residency or failure
    attr[0].val.cooperative = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, k, a);
}

template <int CW, int RPW, int TC, int STAGES>
size_t persist_smem_fixed()
{
    PersistArgs z;
    memset(&z, 0, sizeof z);
    return persist_smem<CW, RPW, TC, STAGES>(z);
}

template <int CW, int RPW, int TC, int STAGES>
cudaError_t persist_preload()
{
    cudaFuncAttributes fa;
    return cudaFuncGetAttributes(&fa, cg_persist_kernel<CW, RPW, TC, STAGES, kPersistMaxChunks>);
}

const PersistVariant kPersist[] = {
    // the tile shapes of the gemv.cu variants of the same name (1 CTA per SM, 4 or 8 consumer warps)
    {"tma_w8r2c512s3", persist_launch<8, 2, 512, 3>, persist_preload<8, 2, 512, 3>, persist_smem_fixed<8, 2, 512, 3>},
    {"tma_w4r4c512s3", persist_launch<4, 4, 512, 3>, persist_preload<4, 4, 512, 3>, persist_smem_fixed<4, 4, 512, 3>},
    {"tma_w8r1c1024s3", persist_launch<8, 1, 1024, 3>, persist_preload<8, 1, 1024, 3>, persist_smem_fixed<8, 1, 1024, 3>},
    {"tma_w4r2c1024s3", persist_launch<4, 2, 1024, 3>, persist_preload<4, 2, 1024, 3>, persist_smem_fixed<4, 2, 1024, 3>},
    {"tma_w4r1c2048s2", persist_launch<4, 1, 2048, 2>, persist_preload<4, 1, 2048, 2>, persist_smem_fixed<4, 1, 2048, 2>},
};

} // namespace

int persist_variant_count() { return (int)(sizeof(kPersist) / sizeof(kPersist[0])); }
const PersistVariant &persist_variant(int i) { return kPersist[i]; }
int persist_max_chunks() { return kPersistMaxChunks; }

} // namespace cgb
