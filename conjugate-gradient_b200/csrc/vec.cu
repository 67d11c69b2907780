// vec.cu -- the O(N) part of the CG iteration for the graph schedule: one iteration is four launches
// (mat-vec, pap_partials, update_xr, update_p) with every scalar (alpha, beta, the stop test) on the device.
// Replaces cblas_daxpy x3 + cblas_ddot x2 + MPI_Allreduce x2 (code/MPI/cg.cc:105-132) and
// sumVec / fill / copy / cublasDdot + cudaMemcpy + cudaDeviceSynchronize (code/CUDA/cg.cu:
// 112-164, 231-269).  All ranks hold the full-length x, r, p and run these kernels redundantly
// on identical data, so no scalar ever crosses NVLink; the only exchange per iteration is the
// gather of the mat-vec result (see capi.cu).
//
// Reduction order (mirrored by oracle/cg_oracle.c): 256-element chunk partials (perfect xor
// tree) of the GLOBAL vector -> det_sum over the chunk partials, for p'Ap and r'r alike.  Nothing
// depends on which CTA / SM / GPU computed a row of Ap.
#include "cgb_device.cuh"
#include "cgb_kernels.h"

namespace cgb {

namespace {

// cooperative copy of `n` doubles into shared memory, then det_sum by warp 0, result broadcast
__device__ __forceinline__ double block_det_sum(const double *src, long long n, double *buf,
                                                double *bcast, int tid)
{
    for (long long t = tid; t < n; t += blockDim.x) buf[t] = src[t];
    __syncthreads();
    if (tid < 32) {
        const double s = warp_det_sum(buf, n, tid);
        if (tid == 0) *bcast = s;
    }
    __syncthreads();
    return *bcast;
}

__global__ void __launch_bounds__(kChunk) init_residual_kernel(const VecArgs a)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x;
    const long long i = (long long)blockIdx.x * kChunk + tid;
    const GatherView gv = gather_view(a.apx, a.g);
    double v = 0.0;
    if (i < a.n) {
        const double ap = gather_read(gv, gather_index(a.g, i));
        const double rr = __fma_rn(-1.0, ap, a.b[i]); // daxpy(-1, Ap, r = b)   cg.cc:82
        a.r[i] = rr;
        a.p[i] = rr;                                  // p = r                  cg.cc:85
        v = __dmul_rn(rr, rr);                        // ddot(r, p)             cg.cc:91
    }
    const double t = block_chunk256(v, wsum, tid);
    if (tid == 0) a.rrpart[blockIdx.x] = t;
    exchange_consumed(a.g, tid);
}

// chunk partials of p'Ap from the gathered rows (cg.cc:105): level 1 of the two-level reduction
__global__ void __launch_bounds__(kChunk) pap_partials_kernel(const VecArgs a)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x;
    griddep_launch_dependents(); // let update_xr become resident
    griddep_wait();              // ... but read nothing before the mat-vec has completed
    if (a.st->done) return;
    // fused exchange: every read polls its own LL entry until the owning rank's mat-vec has
    // delivered it over NVLink -- this kernel may start while peers are still streaming A
    const GatherView gv = gather_view(a.apx, a.g);
    const long long i = (long long)blockIdx.x * kChunk + tid;
    const double v = (i < a.n) ? __dmul_rn(a.p[i], gather_read(gv, gather_index(a.g, i))) : 0.0;
    const double t = block_chunk256(v, wsum, tid);
    if (tid == 0) a.papart[blockIdx.x] = t;
    // the exchange stays open: update_xr reads the same rows again and closes it
}

__global__ void __launch_bounds__(kChunk) update_xr_kernel(const VecArgs a, long long nchunks)
{
    extern __shared__ double sh_part[]; // nchunks chunk partials of p'Ap
    __shared__ double wsum[8];
    __shared__ double sh_alpha;
    const int tid = threadIdx.x;
    // diagnostic timeline: thread 0 of every block stamps entry / dependency met / alpha known / exit
    unsigned long long *rec = nullptr;
    if (a.trace_xr.buf && tid == 0) {
        rec = trace_slot(a.trace_xr, blockIdx.x);
        trace_stamp(rec, 0);
    }
    griddep_launch_dependents(); // let update_p (and, behind it, the next mat-vec) become resident
    griddep_wait();              // pap_partials has completed
    trace_stamp(rec, 1);
    if (a.st->done) return;
    const GatherView gv = gather_view(a.apx, a.g);
    for (long long t = tid; t < nchunks; t += kChunk) sh_part[t] = a.papart[t];
    __syncthreads();
    if (tid < 32) {
        const double conj = warp_det_sum(sh_part, nchunks, tid);      // p'Ap     cg.cc:105-106
        const double rsold = a.st->rsold;
        const double clamp = __dmul_rn(rsold, kNearZero);
        const double alpha = __ddiv_rn(rsold, (conj < clamp) ? clamp : conj); // cg.cc:107
        if (tid == 0) {
            sh_alpha = alpha;
            if (blockIdx.x == 0) {
                a.st->conj = conj;
                a.st->alpha = alpha;
            }
        }
    }
    __syncthreads();
    trace_stamp(rec, 2);
    const double alpha = sh_alpha;
    const long long i = (long long)blockIdx.x * kChunk + tid;
    double v = 0.0;
    if (i < a.n) {
        const double pi = a.p[i];
        a.x[i] = __fma_rn(alpha, pi, a.x[i]);                          // cg.cc:110
        const double rn = __fma_rn(-alpha, gather_read(gv, gather_index(a.g, i)), a.r[i]); // cg.cc:113
        a.r[i] = rn;
        v = __dmul_rn(rn, rn);                                         // cg.cc:116
    }
    const double t = block_chunk256(v, wsum, tid);
    if (tid == 0) a.rrpart[blockIdx.x] = t;
    exchange_consumed(a.g, tid);
    trace_stamp(rec, 3);
}

__global__ void __launch_bounds__(kChunk) update_p_kernel(const VecArgs a, long long nchunks)
{
    extern __shared__ double sh_rr[]; // nchunks chunk partials
    __shared__ double sh_bcast;
    __shared__ int sh_done;
    const int tid = threadIdx.x;
    unsigned long long *rec = nullptr;
    if (a.trace_p.buf && tid == 0) {
        rec = trace_slot(a.trace_p, blockIdx.x);
        trace_stamp(rec, 0);
    }
    griddep_launch_dependents(); // the next mat-vec may start prefetching A now
    griddep_wait();              // update_xr has completed: rrpart and r are final
    trace_stamp(rec, 1);
    // block 0 may raise `done` while this launch is still running: sample it once per block
    if (tid == 0) sh_done = a.st->done;
    __syncthreads();
    if (sh_done) return;
    const double rsnew = block_det_sum(a.rrpart, nchunks, sh_rr, &sh_bcast, tid); // cg.cc:116-117
    if (sqrt(rsnew) < a.tol) {                                                    // cg.cc:120-121
        // break BEFORE p / rsold are updated: rsold stays stale, x stops here
        if (blockIdx.x == 0 && tid == 0) {
            a.st->rsnew = rsnew;
            if (a.hist) a.hist[a.st->iter] = rsnew;
            a.st->done = 1;
            if (a.host_done) *a.host_done = 1;
            __threadfence_system();
        }
        return;
    }
    const double beta = __ddiv_rn(rsnew, a.st->rsold);                            // cg.cc:124
    const long long i = (long long)blockIdx.x * kChunk + tid;
    if (i < a.n) a.p[i] = __fma_rn(beta, a.p[i], a.r[i]);                         // cg.cc:127-129
    trace_stamp(rec, 3);
}

// ---- the once-per-iteration vector phase (CSR contexts) ----------------------------------
// Every block publishes its chunk partial; the last block to arrive (threadfence + arrival
// counter, reset by that block) reduces all of them with the same warp_det_sum as the kernels
// above.  Returns true in warp 0 of the last block, after which the partials are visible.
__device__ __forceinline__ bool publish_partial(double *part, double t, unsigned int *arrive, int tid)
{
    __shared__ int sh_last;
    if (tid == 0) {
        part[blockIdx.x] = t;
        __threadfence();
        sh_last = atomicAdd(arrive, 1u) == gridDim.x - 1;
    }
    __syncthreads();
    if (!sh_last || tid >= 32) return false;
    __threadfence();
    return true;
}
// warp_det_sum over partials other blocks wrote during this launch (read from L2)
__device__ __forceinline__ double warp_det_sum_l2(const double *v, long long n, int lane)
{
    double s = 0.0;
    for (long long t = lane; t < n; t += 32) s = __dadd_rn(s, __ldcg(v + t));
    return warp_butterfly(s);
}

__global__ void __launch_bounds__(kChunk) pap_alpha_kernel(const VecArgs a)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x;
    griddep_launch_dependents();
    griddep_wait();
    if (a.st->done) return;
    const GatherView gv = gather_view(a.apx, a.g);
    const long long i = (long long)blockIdx.x * kChunk + tid;
    const double v = (i < a.n) ? __dmul_rn(a.p[i], gather_read(gv, gather_index(a.g, i))) : 0.0;
    const double t = block_chunk256(v, wsum, tid);
    if (!publish_partial(a.papart, t, &a.arrive[0], tid)) return;
    const double conj = warp_det_sum_l2(a.papart, gridDim.x, tid);        // p'Ap     cg.cc:105-106
    if (tid == 0) {
        const double rsold = a.st->rsold;
        const double clamp = __dmul_rn(rsold, kNearZero);
        a.st->conj = conj;
        a.st->alpha = __ddiv_rn(rsold, (conj < clamp) ? clamp : conj);   // cg.cc:107
        a.arrive[0] = 0;
    }
}

__global__ void __launch_bounds__(kChunk) update_xr_once_kernel(const VecArgs a)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x;
    griddep_launch_dependents();
    griddep_wait();                      // pap_alpha has completed: st->alpha is final
    if (a.st->done) return;
    const double alpha = a.st->alpha;
    const GatherView gv = gather_view(a.apx, a.g);
    const long long i = (long long)blockIdx.x * kChunk + tid;
    double v = 0.0;
    if (i < a.n) {
        const double pi = a.p[i];
        a.x[i] = __fma_rn(alpha, pi, a.x[i]);                          // cg.cc:110
        const double rn = __fma_rn(-alpha, gather_read(gv, gather_index(a.g, i)), a.r[i]); // cg.cc:113
        a.r[i] = rn;
        v = __dmul_rn(rn, rn);                                         // cg.cc:116
    }
    const double t = block_chunk256(v, wsum, tid);
    exchange_consumed(a.g, tid);
    if (!publish_partial(a.rrpart, t, &a.arrive[1], tid)) return;
    const double rsnew = warp_det_sum_l2(a.rrpart, gridDim.x, tid);      // cg.cc:116-117
    if (tid == 0) {
        a.st->rsnew = rsnew;
        if (sqrt(rsnew) < a.tol) {                                      // cg.cc:120-121
            // break BEFORE p / rsold are updated: rsold stays stale, x stops here
            if (a.hist) a.hist[a.st->iter] = rsnew;
            a.st->done = 1;
            if (a.host_done) *a.host_done = 1;
            __threadfence_system();
        }
        a.arrive[1] = 0;
    }
}

__global__ void __launch_bounds__(kChunk) update_p_once_kernel(const VecArgs a)
{
    griddep_launch_dependents(); // the next mat-vec may start now
    griddep_wait();              // update_xr_once has completed: r, st->rsnew and the stop test are final
    if (a.st->done) return;
    const double beta = __ddiv_rn(a.st->rsnew, a.st->rsold);                      // cg.cc:124
    const long long i = (long long)blockIdx.x * kChunk + threadIdx.x;
    if (i < a.n) a.p[i] = __fma_rn(beta, a.p[i], a.r[i]);                         // cg.cc:127-129
}

// ---- block solve: the kernels above per column (blockIdx.y = column j) ---------------------------
// Same chunks, same last-block reductions, same FMAs as the CSR single solve; column j has its own
// State and arrival counters, and a column that is done returns like a single solve after its break.
__global__ void __launch_bounds__(kChunk) init_residual_block_kernel(const BlockArgs a)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x, j = blockIdx.y;
    const long long i = (long long)blockIdx.x * kChunk + tid, o = j * a.ld + i;
    double v = 0.0;
    if (i < a.n) {
        const double rr = __fma_rn(-1.0, a.ap[j * a.slot + i], a.b[o]); // cg.cc:82
        a.r[o] = rr;
        a.p[o] = rr;                                                    // cg.cc:85
        v = __dmul_rn(rr, rr);                                          // cg.cc:91
    }
    const double t = block_chunk256(v, wsum, tid);
    if (tid == 0) a.rrpart[j * a.nchunks + blockIdx.x] = t;
}

__global__ void __launch_bounds__(kChunk) pap_alpha_block_kernel(const BlockArgs a)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x, j = blockIdx.y;
    griddep_launch_dependents();
    griddep_wait();
    State *st = a.st + j;
    if (st->done) return;
    const long long i = (long long)blockIdx.x * kChunk + tid;
    const double v = (i < a.n) ? __dmul_rn(a.p[j * a.ld + i], a.ap[j * a.slot + i]) : 0.0;
    const double t = block_chunk256(v, wsum, tid);
    double *part = a.papart + j * a.nchunks;
    if (!publish_partial(part, t, &a.arrive[2 * j], tid)) return;
    const double conj = warp_det_sum_l2(part, gridDim.x, tid);        // p'Ap     cg.cc:105-106
    if (tid == 0) {
        const double rsold = st->rsold;
        const double clamp = __dmul_rn(rsold, kNearZero);
        st->conj = conj;
        st->alpha = __ddiv_rn(rsold, (conj < clamp) ? clamp : conj);   // cg.cc:107
        a.arrive[2 * j] = 0;
    }
}

__global__ void __launch_bounds__(kChunk) update_xr_block_kernel(const BlockArgs a)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x, j = blockIdx.y;
    griddep_launch_dependents();
    griddep_wait();
    State *st = a.st + j;
    if (st->done) return;
    const double alpha = st->alpha;
    const long long i = (long long)blockIdx.x * kChunk + tid, o = j * a.ld + i;
    double v = 0.0;
    if (i < a.n) {
        const double pi = a.p[o];
        a.x[o] = __fma_rn(alpha, pi, a.x[o]);                                   // cg.cc:110
        const double rn = __fma_rn(-alpha, a.ap[j * a.slot + i], a.r[o]);       // cg.cc:113
        a.r[o] = rn;
        v = __dmul_rn(rn, rn);                                                  // cg.cc:116
    }
    const double t = block_chunk256(v, wsum, tid);
    double *part = a.rrpart + j * a.nchunks;
    if (!publish_partial(part, t, &a.arrive[2 * j + 1], tid)) return;
    const double rsnew = warp_det_sum_l2(part, gridDim.x, tid);        // cg.cc:116-117
    if (tid == 0) {
        st->rsnew = rsnew;
        if (sqrt(rsnew) < a.tol) {                                      // cg.cc:120-121
            if (a.hist) a.hist[j * a.hist_ld + st->iter] = rsnew;
            st->done = 1;
            // the last column to converge tells the host that every later launch is a no-op
            if (atomicAdd(a.ndone, 1u) == (unsigned)a.nrhs - 1u && a.host_done) *a.host_done = 1;
            __threadfence_system();
        }
        a.arrive[2 * j + 1] = 0;
    }
}

__global__ void __launch_bounds__(kChunk) update_p_block_kernel(const BlockArgs a)
{
    const int j = blockIdx.y;
    griddep_launch_dependents();
    griddep_wait();
    const State *st = a.st + j;
    if (st->done) return;
    const double beta = __ddiv_rn(st->rsnew, st->rsold);                          // cg.cc:124
    const long long i = (long long)blockIdx.x * kChunk + threadIdx.x, o = j * a.ld + i;
    if (i < a.n) a.p[o] = __fma_rn(beta, a.p[o], a.r[o]);                         // cg.cc:127-129
}

// one warp per column
__global__ void __launch_bounds__(32) finalize_block_kernel(const BlockArgs a)
{
    const int j = blockIdx.x, lane = threadIdx.x;
    State *st = a.st + j;
    if (st->done) return;
    const double s = warp_det_sum(a.rrpart + j * a.nchunks, a.nchunks, lane);
    if (lane == 0) {
        const long long it = st->iter;
        if (it >= 0 && a.hist) a.hist[j * a.hist_ld + it] = s;
        st->rsold = s; // cg.cc:132
        st->rsnew = s;
        st->iter = it + 1;
    }
}

__global__ void __launch_bounds__(32) finalize_kernel(const VecArgs a, long long nchunks)
{
    if (a.st->done) return;
    const int lane = threadIdx.x;
    const double s = warp_det_sum(a.rrpart, nchunks, lane);
    if (lane == 0) {
        const long long it = a.st->iter;
        if (it >= 0 && a.hist) a.hist[it] = s;
        a.st->rsold = s; // cg.cc:132
        a.st->rsnew = s;
        a.st->iter = it + 1;
    }
}

// DEBUG block (cg.cc:144-154), chunk partials: d = A x - b ; d.d, b.b, x.x per chunk
__global__ void __launch_bounds__(kChunk) debug_partials_kernel(const VecArgs a, double *scratch,
                                                                 long long nchunks)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x;
    const long long i = (long long)blockIdx.x * kChunk + tid;
    const GatherView gv = gather_view(a.apx, a.g);
    double dd = 0.0, bb = 0.0, xx = 0.0;
    if (i < a.n) {
        const double bi = a.b[i], xi = a.x[i];
        const double d = __fma_rn(-1.0, bi, gather_read(gv, gather_index(a.g, i))); // cg.cc:146-148
        dd = __dmul_rn(d, d);
        bb = __dmul_rn(bi, bi);
        xx = __dmul_rn(xi, xi);
    }
    double t = block_chunk256(dd, wsum, tid);
    if (tid == 0) scratch[blockIdx.x] = t;
    __syncthreads();
    t = block_chunk256(bb, wsum, tid);
    if (tid == 0) scratch[nchunks + blockIdx.x] = t;
    __syncthreads();
    t = block_chunk256(xx, wsum, tid);
    if (tid == 0) scratch[2 * nchunks + blockIdx.x] = t;
    exchange_consumed(a.g, tid);
}

__global__ void __launch_bounds__(32) debug_final_kernel(const double *scratch, long long nchunks,
                                                          double *out)
{
    const int lane = threadIdx.x;
    const double dd = warp_det_sum(scratch, nchunks, lane);
    const double bb = warp_det_sum(scratch + nchunks, nchunks, lane);
    const double xx = warp_det_sum(scratch + 2 * nchunks, nchunks, lane);
    if (lane == 0) {
        out[0] = sqrt(xx);                         // cg.cc:151
        out[1] = __ddiv_rn(sqrt(dd), sqrt(bb));    // cg.cc:149-150
    }
}

__global__ void __launch_bounds__(kChunk) dot_partials_kernel(const double *x, const double *y,
                                                               long long n, double *scratch)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x;
    const long long i = (long long)blockIdx.x * kChunk + tid;
    const double v = (i < n) ? __dmul_rn(x[i], y[i]) : 0.0;
    const double t = block_chunk256(v, wsum, tid);
    if (tid == 0) scratch[blockIdx.x] = t;
}

__global__ void __launch_bounds__(32) sum_kernel(const double *v, long long n, double *out)
{
    const double s = warp_det_sum(v, n, threadIdx.x);
    if (threadIdx.x == 0) out[0] = s;
}

// hooks: chunk partials of v.(A v) from the PLAIN gather buffer (after exchange_collect)
__global__ void __launch_bounds__(kChunk) pap_plain_kernel(const double *v, const double *apx, const Gather g,
                                                            long long n, double *papart)
{
    __shared__ double wsum[8];
    const int tid = threadIdx.x;
    const long long i = (long long)blockIdx.x * kChunk + tid;
    const double q = (i < n) ? __dmul_rn(v[i], apx[gather_index(g, i)]) : 0.0;
    const double t = block_chunk256(q, wsum, tid);
    if (tid == 0) papart[blockIdx.x] = t;
}

// Fused mode, test hooks only: consume the running exchange into the plain buffer (every rank's
// rows), so that memcpys and pap_plain_kernel can read it.
__global__ void __launch_bounds__(kChunk) exchange_collect_kernel(double *apx, const Gather g)
{
    const int tid = threadIdx.x;
    const GatherView gv = gather_view(apx, g);
    const long long per = g.maxrows;
    const long long total = (long long)g.world * per;
    for (long long t = (long long)blockIdx.x * kChunk + tid; t < total; t += (long long)gridDim.x * kChunk) {
        const int r = (int)(t / per);
        const long long e = t - (long long)r * per;
        const long long rows_r = (r == g.world - 1) ? g.maxrows : g.n_loc;
        if (e < rows_r && e < g.loc_cap) { // loc_cap < rows_r only in "loopback"
            const long long idx = (long long)r * g.slot + e;
            apx[idx] = gather_read(gv, idx);
        }
    }
    exchange_consumed(g, tid);
}

// Envelope of every row of [lr0, lr0 + nrows) (see block_window): one warp per row, 128-bit loads,
// lane l sees the columns 2(l + 32 i), +1; "non-zero" is any bit pattern but +-0 (NaN and Inf count).
__global__ void __launch_bounds__(256) row_envelope_kernel(const double *A, long long ld, long long lr0,
                                                            long long nrows, int2 *env)
{
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= nrows) return;
    const unsigned long long *a = reinterpret_cast<const unsigned long long *>(A + (lr0 + row) * ld);
    const long long nq = ld >> 1;
    constexpr unsigned long long kMag = 0x7fffffffffffffffULL;
    int first = 0x7fffffff, last = -1;
    long long q = lane;
    for (; q + 3 * 32 < nq; q += 4 * 32) {
        ulonglong2 v[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) v[u] = __ldcs(reinterpret_cast<const ulonglong2 *>(a) + q + 32 * u);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int j = (int)(2 * (q + 32 * u));
            if (v[u].x & kMag) { first = min(first, j); last = j; }
            if (v[u].y & kMag) { first = min(first, j + 1); last = j + 1; }
        }
    }
    for (; q < nq; q += 32) {
        const ulonglong2 v = __ldcs(reinterpret_cast<const ulonglong2 *>(a) + q);
        const int j = (int)(2 * q);
        if (v.x & kMag) { first = min(first, j); last = j; }
        if (v.y & kMag) { first = min(first, j + 1); last = j + 1; }
    }
    first = __reduce_min_sync(0xffffffffu, first);
    last = __reduce_max_sync(0xffffffffu, last);
    if (lane == 0) env[lr0 + row] = last >= 0 ? make_int2(first, last + 1) : make_int2(0, 0);
}

inline int grid_for(long long n) { return (int)((n + kChunk - 1) / kChunk); }

} // namespace

cudaError_t launch_row_envelope(const double *A, long long ld, long long lr0, long long nrows, int2 *env,
                                cudaStream_t s)
{
    if (nrows <= 0) return cudaSuccess;
    row_envelope_kernel<<<(unsigned)((nrows + 7) / 8), 256, 0, s>>>(A, ld, lr0, nrows, env);
    return cudaGetLastError();
}

cudaError_t preload_vec_kernels()
{
    cudaFuncAttributes fa;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&fa, init_residual_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, pap_partials_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, update_xr_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, update_p_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, pap_alpha_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, update_xr_once_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, update_p_once_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, finalize_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, debug_partials_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, debug_final_kernel)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&fa, exchange_collect_kernel);
}

cudaError_t launch_init_residual(const VecArgs &a, cudaStream_t s)
{
    init_residual_kernel<<<grid_for(a.n), kChunk, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pap_partials(const VecArgs &a, cudaStream_t s)
{
    return launch_kernel(pap_partials_kernel, grid_for(a.n), kChunk, 0, s, a.pdl != 0, a);
}

cudaError_t launch_update_xr(const VecArgs &a, cudaStream_t s)
{
    const long long nchunks = grid_for(a.n);
    return launch_kernel(update_xr_kernel, (int)nchunks, kChunk, (size_t)nchunks * sizeof(double), s, a.pdl != 0,
                         a, nchunks);
}

cudaError_t launch_update_p(const VecArgs &a, cudaStream_t s)
{
    const long long nchunks = grid_for(a.n);
    return launch_kernel(update_p_kernel, (int)nchunks, kChunk, (size_t)nchunks * sizeof(double), s,
                         a.pdl != 0, a, nchunks);
}

cudaError_t launch_pap_alpha(const VecArgs &a, cudaStream_t s)
{
    return launch_kernel(pap_alpha_kernel, grid_for(a.n), kChunk, 0, s, a.pdl != 0, a);
}

cudaError_t launch_update_xr_once(const VecArgs &a, cudaStream_t s)
{
    return launch_kernel(update_xr_once_kernel, grid_for(a.n), kChunk, 0, s, a.pdl != 0, a);
}

cudaError_t launch_update_p_once(const VecArgs &a, cudaStream_t s)
{
    return launch_kernel(update_p_once_kernel, grid_for(a.n), kChunk, 0, s, a.pdl != 0, a);
}

cudaError_t preload_vec_block_kernels()
{
    cudaFuncAttributes fa;
    cudaError_t e;
    if ((e = cudaFuncGetAttributes(&fa, init_residual_block_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, pap_alpha_block_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, update_xr_block_kernel)) != cudaSuccess) return e;
    if ((e = cudaFuncGetAttributes(&fa, update_p_block_kernel)) != cudaSuccess) return e;
    return cudaFuncGetAttributes(&fa, finalize_block_kernel);
}

cudaError_t launch_init_residual_block(const BlockArgs &a, cudaStream_t s)
{
    init_residual_block_kernel<<<dim3((unsigned)a.nchunks, (unsigned)a.nrhs), kChunk, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_pap_alpha_block(const BlockArgs &a, cudaStream_t s)
{
    return launch_kernel_xy(pap_alpha_block_kernel, dim3((unsigned)a.nchunks, (unsigned)a.nrhs), kChunk, s, a.pdl != 0, a);
}

cudaError_t launch_update_xr_block(const BlockArgs &a, cudaStream_t s)
{
    return launch_kernel_xy(update_xr_block_kernel, dim3((unsigned)a.nchunks, (unsigned)a.nrhs), kChunk, s, a.pdl != 0, a);
}

cudaError_t launch_update_p_block(const BlockArgs &a, cudaStream_t s)
{
    return launch_kernel_xy(update_p_block_kernel, dim3((unsigned)a.nchunks, (unsigned)a.nrhs), kChunk, s, a.pdl != 0, a);
}

cudaError_t launch_finalize_block(const BlockArgs &a, cudaStream_t s)
{
    finalize_block_kernel<<<a.nrhs, 32, 0, s>>>(a);
    return cudaGetLastError();
}

cudaError_t launch_finalize(const VecArgs &a, cudaStream_t s)
{
    finalize_kernel<<<1, 32, 0, s>>>(a, grid_for(a.n));
    return cudaGetLastError();
}

cudaError_t launch_debug_norms(const VecArgs &a, double *scratch, double *out, cudaStream_t s)
{
    const long long nchunks = grid_for(a.n);
    debug_partials_kernel<<<(int)nchunks, kChunk, 0, s>>>(a, scratch, nchunks);
    debug_final_kernel<<<1, 32, 0, s>>>(scratch, nchunks, out);
    return cudaGetLastError();
}

cudaError_t launch_dot(const double *a, const double *b, long long n, double *scratch, double *out,
                       cudaStream_t s)
{
    const long long nchunks = grid_for(n);
    dot_partials_kernel<<<(int)nchunks, kChunk, 0, s>>>(a, b, n, scratch);
    sum_kernel<<<1, 32, 0, s>>>(scratch, nchunks, out);
    return cudaGetLastError();
}

cudaError_t launch_pap_plain(const double *v, const double *apx, const Gather &g, long long n, double *papart,
                             double *out, cudaStream_t s)
{
    const long long nchunks = grid_for(n);
    pap_plain_kernel<<<(int)nchunks, kChunk, 0, s>>>(v, apx, g, n, papart);
    sum_kernel<<<1, 32, 0, s>>>(papart, nchunks, out);
    return cudaGetLastError();
}

cudaError_t launch_exchange_collect(double *apx, const Gather &g, cudaStream_t s)
{
    const long long total = (long long)g.world * g.maxrows;
    long long blocks = (total + kChunk - 1) / kChunk;
    if (blocks > 296) blocks = 296;
    exchange_collect_kernel<<<(int)blocks, kChunk, 0, s>>>(apx, g);
    return cudaGetLastError();
}

} // namespace cgb
