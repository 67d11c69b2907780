// spmv.cu -- CSR storage of the row shard: the mat-vec in lane order and the builders of the shard
// (generate_lap2d_matrix, COO writes folded by Matrix::read's last write or summed) on the device.
//
// Exactness.  The dense mat-vec (gemv.cu, oracle/cg_oracle.h "lane order") keeps 64 accumulators
// acc[c % 64] = fma(A[i][c], p[c], acc[c % 64]) over ascending c from +0, adds acc[2l] + acc[2l+1]
// per lane and finishes with the butterfly ^16, ^8, ^4, ^2, ^1.  An accumulator is never -0 (it
// starts at +0 and an exactly-zero sum rounds to +0 unless both operands are -0), so for a finite
// p[c] an entry A[i][c] = +-0 leaves it unchanged, and so does adding an all-zero partner in the
// lane sum or the butterfly.  Touching the stored entries only -- each bucket's fma chain over its
// entries in ascending column order, absent buckets and partners skipped -- therefore gives the
// dense result bit for bit.  (A NaN / Inf of p at a column where A is zero makes the dense row
// NaN and leaves this one alone; only a solve that has already diverged gets there.)
//
// Layout: one warp per 32 consecutive rows.  A row of at most kShortRow entries (the 2-D stencil
// has 3 to 5) is done by its own lane: bucket sums, then the merge tree above with absent
// entries skipped.  Longer rows are taken by the whole warp one after the other, lane l owning
// buckets 2l and 2l+1 exactly like the dense consumers; entries reach their owner in column order
// in 32-entry slabs broadcast by shuffle.
#include "cgb_device.cuh"
#include "cgb_kernels.h"

#include <cub/device/device_radix_sort.cuh>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_select.cuh>
#include <thrust/iterator/counting_iterator.h>

namespace cgb {

namespace {

constexpr int kShortRow = 8;    // entries a single lane handles (the merge tree is kShortRow^2 / 2 per level)
constexpr int kSpmvThreads = 256;

// lane order for a row of at most kShortRow entries, by one thread
__device__ __forceinline__ double row_short(const int *col, const double *val, int len, const double *v)
{
    double s[kShortRow];
    int key[kShortRow];
    bool live[kShortRow];
#pragma unroll
    for (int e = 0; e < kShortRow; ++e) {
        live[e] = false;
        key[e] = 0;
        s[e] = 0.0;
        if (e < len) {
            const int c = __ldcs(col + e);
            const double prod_a = __ldcs(val + e), pv = __ldg(v + c);
            const int b = c & 63;
            bool merged = false;
#pragma unroll
            for (int f = 0; f < e; ++f)
                if (live[f] && key[f] == b) { // same bucket, earlier column: continue its chain
                    s[f] = __fma_rn(prod_a, pv, s[f]);
                    merged = true;
                }
            key[e] = b;
            live[e] = !merged;
            s[e] = merged ? 0.0 : __fma_rn(prod_a, pv, 0.0);
        }
    }
    // bucket 2l + j: lane sum (bit 0), then the butterfly over the lane index l = bits 5..1
    const int bits[6] = {1, 32, 16, 8, 4, 2};
#pragma unroll
    for (int lv = 0; lv < 6; ++lv) {
#pragma unroll
        for (int e = 0; e < kShortRow; ++e) key[e] &= ~bits[lv];
#pragma unroll
        for (int e = 1; e < kShortRow; ++e)
#pragma unroll
            for (int f = 0; f < e; ++f)
                if (live[f] && live[e] && key[f] == key[e]) {
                    s[f] = __dadd_rn(s[f], s[e]);
                    live[e] = false;
                }
    }
    double y = 0.0;
#pragma unroll
    for (int e = 0; e < kShortRow; ++e)
        if (live[e]) y = s[e];
    return y;
}

// lane order for a row of any length, by the whole warp (every lane returns the row's value)
__device__ __forceinline__ double row_warp(const int *col, const double *val, long long len, const double *v, int lane)
{
    double acc0 = 0.0, acc1 = 0.0;
    for (long long k0 = 0; k0 < len; k0 += 32) {
        const long long k = k0 + lane;
        int c = 0;
        double av = 0.0, pv = 0.0;
        if (k < len) {
            c = __ldcs(col + k);
            av = __ldcs(val + k);
            pv = __ldg(v + c);
        }
        const int m = (len - k0 < 32) ? (int)(len - k0) : 32;
        for (int j = 0; j < m; ++j) {
            const int cj = __shfl_sync(0xffffffffu, c, j);
            const double aj = __shfl_sync(0xffffffffu, av, j);
            const double pj = __shfl_sync(0xffffffffu, pv, j);
            if (((cj & 63) >> 1) == lane) {
                if (cj & 1) acc1 = __fma_rn(aj, pj, acc1);
                else acc0 = __fma_rn(aj, pj, acc0);
            }
        }
    }
    return warp_butterfly(__dadd_rn(acc0, acc1));
}

__global__ void __launch_bounds__(kSpmvThreads) spmv_csr_kernel(const GemvArgs a)
{
    griddep_launch_dependents();
    griddep_wait();
    if (a.st->done) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (a.advance && blockIdx.x == 0 && warp == 0) advance_state(a, lane);
    const unsigned tag = a.p2p ? exchange_tag(a.ctl) : 0u;
    const long long obase = a.slot_off;
    const long long lbase = (long long)(tag & 1u) * a.bufstride + a.slot_off;
    const long long nwarps = (long long)gridDim.x * (kSpmvThreads / 32);
    for (long long w = (long long)blockIdx.x * (kSpmvThreads / 32) + warp; w * 32 < a.rows; w += nwarps) {
        const long long li = w * 32 + lane;
        long long beg = 0, len = 0;
        if (li < a.rows) {
            beg = __ldcs(a.csr_rp + li);
            len = __ldcs(a.csr_rp + li + 1) - beg;
        }
        const bool is_long = len > kShortRow;
        if (li < a.rows && !is_long) {
            const double y = row_short(a.csr_col + beg, a.csr_val + beg, (int)len, a.v);
            if (!a.p2p) {
                a.base[obase + li] = y;
            } else {
                for (int g = 0; g < a.world; ++g) ll_store(a.peer_ll[g] + lbase + li, y, tag);
            }
        }
        unsigned todo = __ballot_sync(0xffffffffu, is_long);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const long long b = __shfl_sync(0xffffffffu, beg, src), l = __shfl_sync(0xffffffffu, len, src);
            const double y = row_warp(a.csr_col + b, a.csr_val + b, l, a.v, lane);
            store_out(a, obase + w * 32 + src, lbase + w * 32 + src, tag, y, lane);
        }
    }
}

// ---- block mat-vec (block solve) ----------------------------------------------------------
// Every column is spmv_csr_kernel's arithmetic on that column alone: row_short's bucket chains and
// merge tree over the row's entries, row_warp's lane-owned accumulators and butterfly.  Only the
// loads are shared: a row's rp / col / val come from memory once for all columns.

// row_short for one column, the row's (at most kShortRow) entries already in registers
__device__ __forceinline__ double row_short_regs(const int (&col)[kShortRow], const double (&val)[kShortRow], int len,
                                                 const double *v)
{
    double s[kShortRow];
    int key[kShortRow];
    bool live[kShortRow];
#pragma unroll
    for (int e = 0; e < kShortRow; ++e) {
        live[e] = false;
        key[e] = 0;
        s[e] = 0.0;
        if (e < len) {
            const double prod_a = val[e], pv = __ldg(v + col[e]);
            const int b = col[e] & 63;
            bool merged = false;
#pragma unroll
            for (int f = 0; f < e; ++f)
                if (live[f] && key[f] == b) {
                    s[f] = __fma_rn(prod_a, pv, s[f]);
                    merged = true;
                }
            key[e] = b;
            live[e] = !merged;
            s[e] = merged ? 0.0 : __fma_rn(prod_a, pv, 0.0);
        }
    }
    const int bits[6] = {1, 32, 16, 8, 4, 2};
#pragma unroll
    for (int lv = 0; lv < 6; ++lv) {
#pragma unroll
        for (int e = 0; e < kShortRow; ++e) key[e] &= ~bits[lv];
#pragma unroll
        for (int e = 1; e < kShortRow; ++e)
#pragma unroll
            for (int f = 0; f < e; ++f)
                if (live[f] && live[e] && key[f] == key[e]) {
                    s[f] = __dadd_rn(s[f], s[e]);
                    live[e] = false;
                }
    }
    double y = 0.0;
#pragma unroll
    for (int e = 0; e < kShortRow; ++e)
        if (live[e]) y = s[e];
    return y;
}

// row_warp for the live columns of `mask` (y[j] in every lane); each 32-entry slab is loaded once
template <int NC>
__device__ __forceinline__ void row_warp_block(const int *col, const double *val, long long len, const double *v,
                                               long long ld, unsigned mask, int lane, double (&y)[NC])
{
    double acc0[NC], acc1[NC];
#pragma unroll
    for (int j = 0; j < NC; ++j) acc0[j] = acc1[j] = 0.0;
    for (long long k0 = 0; k0 < len; k0 += 32) {
        const long long k = k0 + lane;
        int c = 0;
        double av = 0.0, pv[NC];
#pragma unroll
        for (int j = 0; j < NC; ++j) pv[j] = 0.0;
        if (k < len) {
            c = __ldcs(col + k);
            av = __ldcs(val + k);
#pragma unroll
            for (int j = 0; j < NC; ++j)
                if (mask >> j & 1u) pv[j] = __ldg(v + j * ld + c);
        }
        const int m = (len - k0 < 32) ? (int)(len - k0) : 32;
        for (int i = 0; i < m; ++i) {
            const int ci = __shfl_sync(0xffffffffu, c, i);
            const double ai = __shfl_sync(0xffffffffu, av, i);
            const bool mine = ((ci & 63) >> 1) == lane;
#pragma unroll
            for (int j = 0; j < NC; ++j) {
                if (!(mask >> j & 1u)) continue; // warp-uniform
                const double pj = __shfl_sync(0xffffffffu, pv[j], i);
                if (mine) {
                    if (ci & 1) acc1[j] = __fma_rn(ai, pj, acc1[j]);
                    else acc0[j] = __fma_rn(ai, pj, acc0[j]);
                }
            }
        }
    }
#pragma unroll
    for (int j = 0; j < NC; ++j) y[j] = (mask >> j & 1u) ? warp_butterfly(__dadd_rn(acc0[j], acc1[j])) : 0.0;
}

// advance_state of column j (one full warp)
__device__ __forceinline__ void advance_column(const BlockArgs &a, int j, int lane)
{
    const double s = warp_det_sum(a.rrpart + j * a.nchunks, a.nchunks, lane);
    if (lane == 0) {
        State *st = a.st + j;
        const long long it = st->iter;
        if (it >= 0 && a.hist) a.hist[j * a.hist_ld + it] = s;
        st->rsold = s;
        st->rsnew = s;
        st->iter = it + 1;
    }
}

template <int NC>
__global__ void __launch_bounds__(kSpmvThreads) spmv_csr_block_kernel(const BlockArgs a)
{
    griddep_launch_dependents();
    griddep_wait();
    unsigned mask = 0; // live columns; no kernel of this iteration changes a `done` before this one ends
#pragma unroll
    for (int j = 0; j < NC; ++j)
        if (!a.st[j].done) mask |= 1u << j;
    if (!mask) return;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    if (a.advance && blockIdx.x == 0 && warp == 0)
        for (int j = 0; j < NC; ++j)
            if (mask >> j & 1u) advance_column(a, j, lane);
    const long long nwarps = (long long)gridDim.x * (kSpmvThreads / 32);
    for (long long w = (long long)blockIdx.x * (kSpmvThreads / 32) + warp; w * 32 < a.rows; w += nwarps) {
        const long long li = w * 32 + lane;
        long long beg = 0, len = 0;
        if (li < a.rows) {
            beg = __ldcs(a.rp + li);
            len = __ldcs(a.rp + li + 1) - beg;
        }
        const bool is_long = len > kShortRow;
        if (li < a.rows && !is_long) {
            int c[kShortRow];
            double av[kShortRow];
#pragma unroll
            for (int e = 0; e < kShortRow; ++e) {
                c[e] = 0;
                av[e] = 0.0;
                if (e < len) {
                    c[e] = __ldcs(a.col + beg + e);
                    av[e] = __ldcs(a.val + beg + e);
                }
            }
#pragma unroll
            for (int j = 0; j < NC; ++j)
                if (mask >> j & 1u) a.ap[j * a.slot + li] = row_short_regs(c, av, (int)len, a.v + j * a.ld);
        }
        unsigned todo = __ballot_sync(0xffffffffu, is_long);
        while (todo) {
            const int src = __ffs(todo) - 1;
            todo &= todo - 1;
            const long long b = __shfl_sync(0xffffffffu, beg, src), l = __shfl_sync(0xffffffffu, len, src);
            double y[NC];
            row_warp_block<NC>(a.col + b, a.val + b, l, a.v, a.ld, mask, lane, y);
            if (lane == 0)
#pragma unroll
                for (int j = 0; j < NC; ++j)
                    if (mask >> j & 1u) a.ap[j * a.slot + w * 32 + src] = y[j];
        }
    }
}

// ---- builders ---------------------------------------------------------------------------
// generate_lap2d_matrix (cg.cc:159-188), the one statement of the stencil (dense shards are densified
// from it): the non-zeros of row i in ascending column order i-1-inc, i-1, i, i+1, i+1+inc;
// emit(column, value) for each
template <class Emit>
__device__ __forceinline__ void lap2d_row(long long n, long long inc, long long i, Emit emit)
{
    if (i > inc) emit(i - 1 - inc, -1.0);
    if (i > 0) emit(i - 1, -1.0);
    emit(i, 4.0);
    if (i < n - 1) emit(i + 1, -1.0);
    if (i < n - 1 - inc) emit(i + 1 + inc, -1.0);
}

__global__ void lap2d_count_kernel(long long n, long long inc, long long row0, long long rows, long long *cnt)
{
    const long long li = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= rows) return;
    long long k = 0;
    lap2d_row(n, inc, row0 + li, [&](long long, double) { ++k; });
    cnt[li] = k;
}

__global__ void lap2d_fill_kernel(long long n, long long inc, long long row0, long long rows, const long long *rp,
                                  int *col, double *val)
{
    const long long li = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (li >= rows) return;
    long long o = rp[li];
    lap2d_row(n, inc, row0 + li, [&](long long c, double v) {
        col[o] = (int)c;
        val[o++] = v;
    });
}

// COO triples as a write sequence: triple z makes write 2z at (i, j) and, symmetric and off the diagonal, write
// 2z+1 at (j, i).  A mirrored diagonal would count twice in a sum; under Matrix::read's "later entries
// overwrite" it would only repeat write 2z's value in the same cell.  So neither fold needs it.  A write
// outside this shard's rows gets the key that sorts last.  The sort payload is the write id, so that the
// sorted order doubles as the plan every fold gathers by.
constexpr unsigned long long kNoKey = ~0ULL;
__global__ void asm_keys_kernel(long long n, long long row0, long long rows, const int *irn, const int *jcn,
                                long long nz, int symmetric, unsigned long long *key, long long *wid, long long *bad)
{
    const long long z = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (z >= nz) return;
    const long long i = irn[z], j = jcn[z];
    unsigned long long k0 = kNoKey, k1 = kNoKey;
    if (i < 0 || j < 0 || i >= n || j >= n) {
        *bad = 1;
    } else {
        if (i >= row0 && i < row0 + rows) k0 = ((unsigned long long)(i - row0) << 32) | (unsigned long long)j;
        if (symmetric && i != j && j >= row0 && j < row0 + rows)
            k1 = ((unsigned long long)(j - row0) << 32) | (unsigned long long)i;
    }
    key[2 * z] = k0;
    key[2 * z + 1] = k1;
    wid[2 * z] = 2 * z;
    wid[2 * z + 1] = 2 * z + 1;
}

// after the stable sort: flag the first write of every (row, column) run; *nw = the writes this shard keeps
__global__ void asm_runs_kernel(const unsigned long long *key, long long m, unsigned char *first, long long *nw)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= m) return;
    const bool kept = key[k] != kNoKey;
    first[k] = (kept && (k == 0 || key[k - 1] != key[k])) ? 1 : 0;
    if (kept && (k == m - 1 || key[k + 1] == kNoKey)) *nw = k + 1;
}

// The one statement of the fold: stored entry e is its run of writes in write order, folded by F.
//   kFoldSum   left fold from the first write (not from +0, which would turn a lone -0 into +0), serial per
//              cell by definition;
//   kFoldLast  the run's last write, verbatim (Matrix::read, matrix.cc:12-21: later entries overwrite).
template <AsmFold F> __device__ __forceinline__ double fold_run(const AsmPlan &p, const double *val, long long e)
{
    const long long end = p.start[e + 1];
    if (F == kFoldLast) return val[p.wid[end - 1] >> 1];
    long long k = p.start[e];
    double v = val[p.wid[k] >> 1];
    for (++k; k < end; ++k) v = __dadd_rn(v, val[p.wid[k] >> 1]);
    return v;
}

// CSR shard: the values in stored order, one thread per entry
template <AsmFold F> __global__ void assemble_csr_kernel(const AsmPlan p, const double *val, double *out)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e < p.nnz) out[e] = fold_run<F>(p, val, e);
}

// dense shard (re-assembly, a sum): one warp per row (its row from the plan's rp), lanes striding over the row's
// entries
__global__ void __launch_bounds__(256) assemble_dense_kernel(const AsmPlan p, const double *val, long long ld,
                                                              double *A)
{
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    if (row >= p.rows) return;
    const long long end = p.rp[row + 1];
    for (long long e = p.rp[row] + (threadIdx.x & 31); e < end; e += 32)
        A[row * ld + p.col[e]] = fold_run<kFoldSum>(p, val, e);
}

// row pointers and columns from the surviving keys (sorted by row, then column)
__global__ void csr_rows_kernel(const unsigned long long *key, long long nnz, long long rows, long long *rp)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r > rows) return;
    const unsigned long long want = (unsigned long long)r << 32;
    long long lo = 0, hi = nnz; // first key >= want
    while (lo < hi) {
        const long long mid = (lo + hi) >> 1;
        if (key[mid] < want) lo = mid + 1;
        else hi = mid;
    }
    rp[r] = lo;
}
__global__ void csr_cols_kernel(const unsigned long long *key, long long nnz, int *col)
{
    const long long k = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (k < nnz) col[k] = (int)(key[k] & 0xffffffffULL);
}

// rows [lr0, lr0 + nrows) of a CSR into a dense nrows x ld buffer (zeroed by the caller)
__global__ void csr_densify_kernel(const long long *rp, const int *col, const double *val, long long lr0,
                                   long long nrows, long long ld, double *dst)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= nrows) return;
    for (long long k = rp[lr0 + r]; k < rp[lr0 + r + 1]; ++k) dst[r * ld + col[k]] = val[k];
}

// A caller's CSR (cgb_set_matrix_csr) checked against the stored format, one warp per row.  The row's
// rp pair is checked first, and its columns are read only when the pair lies inside [rp[0], rp[0] + nnz]:
// a bad rp is refused and never leads to a read outside the caller's nnz entries.  Then the lanes stride
// over the row's entries for the range and the strict ascent.  The first fault lands in *err as
// row * kCsrFaultKinds + kind (atomicMin: the smallest row, and the first failed check of that row);
// rp_local receives rp - rp[0].
__global__ void __launch_bounds__(256) validate_csr_kernel(const long long *rp, const int *col, long long nnz,
                                                            long long n, long long rows, long long *rp_local,
                                                            unsigned long long *err)
{
    const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= rows) return;
    const long long base = rp[0], beg = rp[row], end = rp[row + 1]; // warp-uniform
    const unsigned long long here = (unsigned long long)row * kCsrFaultKinds;
    int kind = -1;
    if (base < 0) kind = kCsrNegativeBase;
    else if (end < beg) kind = kCsrNotMonotone;
    else if (beg < base || end - base > nnz) kind = kCsrPastNnz;
    if (kind >= 0) {
        if (lane == 0) atomicMin(err, here + kind);
        return;
    }
    bool range = false, order = false;
    for (long long k = beg - base + lane; k < end - base; k += 32) {
        const int c = col[k];
        if (c < 0 || c >= n) range = true;
        else if (k > beg - base && col[k - 1] >= c) order = true;
    }
    range = __any_sync(0xffffffffu, range);
    order = __any_sync(0xffffffffu, order);
    if (lane != 0) return;
    if (range) atomicMin(err, here + kCsrColumnRange);
    else if (order) atomicMin(err, here + kCsrNotAscending);
    else if (row == rows - 1 && end - base != nnz) atomicMin(err, here + kCsrCount);
    rp_local[row + 1] = end - base;
    if (row == 0) rp_local[0] = 0;
}

inline unsigned blocks_for(long long n, int t) { return (unsigned)((n + t - 1) / t > 0 ? (n + t - 1) / t : 1); }

#define CU(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) return e_;                                                          \
    } while (0)

} // namespace

cudaError_t csr_alloc_entries(CsrShard *m, long long nnz)
{
    CU(cudaMalloc(&m->col, (size_t)(nnz > 0 ? nnz : 1) * sizeof(int)));
    CU(cudaMalloc(&m->val, (size_t)(nnz > 0 ? nnz : 1) * sizeof(double)));
    m->nnz = nnz;
    return cudaSuccess;
}

cudaError_t preload_spmv_kernels()
{
    cudaFuncAttributes fa;
    return cudaFuncGetAttributes(&fa, spmv_csr_kernel);
}

cudaError_t launch_spmv(const GemvArgs &a, int sm_count, cudaStream_t s)
{
    // enough warps to cover every row once, capped at 32 resident blocks per SM (grid-stride beyond)
    long long blocks = (a.rows + kSpmvThreads - 1) / kSpmvThreads;
    if (blocks > 32LL * sm_count) blocks = 32LL * sm_count;
    if (blocks < 1) blocks = 1;
    return launch_kernel(spmv_csr_kernel, (int)blocks, kSpmvThreads, 0, s, a.pdl != 0, a);
}

namespace {
template <int NC> cudaError_t launch_spmv_block_nc(const BlockArgs &a, int sm_count, cudaStream_t s)
{
    long long blocks = (a.rows + kSpmvThreads - 1) / kSpmvThreads; // the grid of launch_spmv
    if (blocks > 32LL * sm_count) blocks = 32LL * sm_count;
    if (blocks < 1) blocks = 1;
    return launch_kernel(spmv_csr_block_kernel<NC>, (int)blocks, kSpmvThreads, 0, s, a.pdl != 0, a);
}
template <int NC> cudaError_t preload_spmv_block_nc()
{
    cudaFuncAttributes fa;
    return cudaFuncGetAttributes(&fa, spmv_csr_block_kernel<NC>);
}
} // namespace

cudaError_t launch_spmv_block(const BlockArgs &a, int sm_count, cudaStream_t s)
{
    static_assert(kMaxRhs == 8, "one instantiation per column count");
    switch (a.nrhs) {
    case 1: return launch_spmv_block_nc<1>(a, sm_count, s);
    case 2: return launch_spmv_block_nc<2>(a, sm_count, s);
    case 3: return launch_spmv_block_nc<3>(a, sm_count, s);
    case 4: return launch_spmv_block_nc<4>(a, sm_count, s);
    case 5: return launch_spmv_block_nc<5>(a, sm_count, s);
    case 6: return launch_spmv_block_nc<6>(a, sm_count, s);
    case 7: return launch_spmv_block_nc<7>(a, sm_count, s);
    case 8: return launch_spmv_block_nc<8>(a, sm_count, s);
    default: return cudaErrorInvalidValue;
    }
}

cudaError_t preload_spmv_block_kernels()
{
    cudaError_t e;
    if ((e = preload_spmv_block_nc<1>()) != cudaSuccess) return e;
    if ((e = preload_spmv_block_nc<2>()) != cudaSuccess) return e;
    if ((e = preload_spmv_block_nc<3>()) != cudaSuccess) return e;
    if ((e = preload_spmv_block_nc<4>()) != cudaSuccess) return e;
    if ((e = preload_spmv_block_nc<5>()) != cudaSuccess) return e;
    if ((e = preload_spmv_block_nc<6>()) != cudaSuccess) return e;
    if ((e = preload_spmv_block_nc<7>()) != cudaSuccess) return e;
    return preload_spmv_block_nc<8>();
}

cudaError_t csr_generate_lap2d(CsrShard *m, long long n, long long row0, long long rows, cudaStream_t s)
{
    const long long inc = (long long)floor(sqrt((double)n)); // cg.cc:175
    DevBuf cnt, tmp;
    CU(cudaMalloc(&m->rp, (size_t)(rows + 1) * sizeof(long long)));
    CU(cnt.alloc((size_t)rows * sizeof(long long)));
    lap2d_count_kernel<<<blocks_for(rows, 256), 256, 0, s>>>(n, inc, row0, rows, cnt.as<long long>());
    CU(cudaGetLastError());
    size_t tmp_bytes = 0;
    CU(cub::DeviceScan::InclusiveSum(nullptr, tmp_bytes, cnt.as<long long>(), m->rp + 1, rows, s));
    CU(tmp.alloc(tmp_bytes));
    CU(cudaMemsetAsync(m->rp, 0, sizeof(long long), s));
    CU(cub::DeviceScan::InclusiveSum(tmp.p, tmp_bytes, cnt.as<long long>(), m->rp + 1, rows, s));
    long long nnz = 0;
    CU(cudaMemcpyAsync(&nnz, m->rp + rows, sizeof nnz, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    CU(csr_alloc_entries(m, nnz));
    lap2d_fill_kernel<<<blocks_for(rows, 256), 256, 0, s>>>(n, inc, row0, rows, m->rp, m->col, m->val);
    CU(cudaGetLastError());
    return cudaStreamSynchronize(s);
}

void asm_plan_free(AsmPlan *p)
{
    cudaFree(p->wid);
    cudaFree(p->start);
    cudaFree(p->rp);
    cudaFree(p->col);
    *p = AsmPlan();
}

cudaError_t csr_assemble_coo(CsrShard *m, AsmPlan *p, AsmFold fold, long long n, long long row0, long long rows,
                             const int *irn, const int *jcn, const double *val, long long nz, int symmetric,
                             int *bad_host, cudaStream_t s)
{
    *bad_host = 0;
    const long long m2 = 2 * nz;
    // 66 B per triple: 2 writes x (8 B key + 8 B write id) x (unsorted, sorted) + 2 flag bytes.  key / wid are
    // dead after the sort and receive the unique keys and the run starts (wid one longer, for the sentinel
    // start[nnz]).  cnt: [0] entries, [1] writes kept, [2] non-zero when an entry lies outside n x n.
    DevBuf key, wid, key_s, wid_s, first, cnt, tmp;
    CU(key.alloc((size_t)m2 * 8));
    CU(wid.alloc((size_t)(m2 + 1) * 8));
    CU(key_s.alloc((size_t)m2 * 8));
    CU(wid_s.alloc((size_t)m2 * 8));
    CU(first.alloc((size_t)m2));
    CU(cnt.alloc(3 * sizeof(long long)));
    CU(cudaMemsetAsync(cnt.p, 0, 3 * sizeof(long long), s));
    if (nz > 0) {
        asm_keys_kernel<<<blocks_for(nz, 256), 256, 0, s>>>(n, row0, rows, irn, jcn, nz, symmetric, key.as<unsigned long long>(),
                                                            wid.as<long long>(), cnt.as<long long>() + 2);
        CU(cudaGetLastError());
        // radix sort is stable: equal (row, column) keys keep their write order
        const thrust::counting_iterator<long long> pos(0);
        size_t b_sort = 0, b_sel = 0, b_sel2 = 0;
        CU(cub::DeviceRadixSort::SortPairs(nullptr, b_sort, key.as<unsigned long long>(), key_s.as<unsigned long long>(),
                                           wid.as<long long>(), wid_s.as<long long>(), m2, 0, 64, s));
        CU(cub::DeviceSelect::Flagged(nullptr, b_sel, key_s.as<unsigned long long>(), first.as<unsigned char>(),
                                      key.as<unsigned long long>(), cnt.as<long long>(), m2, s));
        CU(cub::DeviceSelect::Flagged(nullptr, b_sel2, pos, first.as<unsigned char>(), wid.as<long long>(),
                                      cnt.as<long long>(), m2, s));
        size_t b = b_sort > b_sel ? b_sort : b_sel;
        if (b_sel2 > b) b = b_sel2;
        CU(tmp.alloc(b));
        CU(cub::DeviceRadixSort::SortPairs(tmp.p, b_sort, key.as<unsigned long long>(), key_s.as<unsigned long long>(),
                                           wid.as<long long>(), wid_s.as<long long>(), m2, 0, 64, s));
        asm_runs_kernel<<<blocks_for(m2, 256), 256, 0, s>>>(key_s.as<unsigned long long>(), m2, first.as<unsigned char>(),
                                                            cnt.as<long long>() + 1);
        CU(cudaGetLastError());
        CU(cub::DeviceSelect::Flagged(tmp.p, b_sel, key_s.as<unsigned long long>(), first.as<unsigned char>(),
                                      key.as<unsigned long long>(), cnt.as<long long>(), m2, s));
        CU(cub::DeviceSelect::Flagged(tmp.p, b_sel2, pos, first.as<unsigned char>(), wid.as<long long>(),
                                      cnt.as<long long>(), m2, s));
    }
    long long counts[3] = {0, 0, 0};
    CU(cudaMemcpyAsync(counts, cnt.p, sizeof counts, cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    *bad_host = counts[2] != 0;
    if (*bad_host) return cudaSuccess;
    const long long nnz = counts[0], nw = counts[1];
    // the staging buffers as a plan: the sorted write ids and the run starts where the selects left them
    const AsmPlan run{wid_s.as<long long>(), wid.as<long long>(), nullptr, nullptr, nz, nnz, nw, rows};
    CU(cudaMemcpyAsync(run.start + nnz, cnt.as<long long>() + 1, sizeof(long long), cudaMemcpyDeviceToDevice, s));
    CU(cudaMalloc(&m->rp, (size_t)(rows + 1) * sizeof(long long)));
    CU(csr_alloc_entries(m, nnz));
    if (p) {
        CU(cudaMalloc(&p->wid, (size_t)(nw > 0 ? nw : 1) * sizeof(long long)));
        CU(cudaMalloc(&p->start, (size_t)(nnz + 1) * sizeof(long long)));
        p->nz = nz;
        p->nnz = nnz;
        p->nwrites = nw;
        p->rows = rows;
        if (nw > 0) CU(cudaMemcpyAsync(p->wid, run.wid, (size_t)nw * 8, cudaMemcpyDeviceToDevice, s));
        CU(cudaMemcpyAsync(p->start, run.start, (size_t)(nnz + 1) * 8, cudaMemcpyDeviceToDevice, s));
    }
    csr_rows_kernel<<<blocks_for(rows + 1, 256), 256, 0, s>>>(key.as<unsigned long long>(), nnz, rows, m->rp);
    csr_cols_kernel<<<blocks_for(nnz, 256), 256, 0, s>>>(key.as<unsigned long long>(), nnz, m->col);
    CU(cudaGetLastError());
    CU(launch_assemble_csr(run, fold, val, m->val, s));
    return cudaStreamSynchronize(s);
}

cudaError_t launch_assemble_csr(const AsmPlan &p, AsmFold fold, const double *val, double *out, cudaStream_t s)
{
    if (p.nnz == 0) return cudaSuccess;
    if (fold == kFoldLast) assemble_csr_kernel<kFoldLast><<<blocks_for(p.nnz, 256), 256, 0, s>>>(p, val, out);
    else assemble_csr_kernel<kFoldSum><<<blocks_for(p.nnz, 256), 256, 0, s>>>(p, val, out);
    return cudaGetLastError();
}

cudaError_t launch_assemble_dense(const AsmPlan &p, const double *val, long long ld, double *A, cudaStream_t s)
{
    if (p.nnz == 0) return cudaSuccess;
    assemble_dense_kernel<<<blocks_for(p.rows, 8), 256, 0, s>>>(p, val, ld, A);
    return cudaGetLastError();
}

cudaError_t csr_densify(const long long *rp, const int *col, const double *val, long long lr0, long long nrows,
                        long long ld, double *dst, cudaStream_t s)
{
    CU(cudaMemsetAsync(dst, 0, (size_t)nrows * ld * sizeof(double), s));
    csr_densify_kernel<<<blocks_for(nrows, 256), 256, 0, s>>>(rp, col, val, lr0, nrows, ld, dst);
    return cudaGetLastError();
}

cudaError_t launch_validate_csr(const long long *rp, const int *col, long long nnz, long long n, long long rows,
                                long long *rp_local, unsigned long long *err, cudaStream_t s)
{
    CU(cudaMemsetAsync(err, 0xff, sizeof *err, s));
    validate_csr_kernel<<<blocks_for(rows, 8), 256, 0, s>>>(rp, col, nnz, n, rows, rp_local, err);
    return cudaGetLastError();
}

cudaError_t launch_read_csr(const CsrShard &m, long long rows, double *sink, int sm_count, cudaStream_t s)
{
    CU(launch_read_stream(m.val, m.nnz, sink, sm_count, s));
    CU(launch_read_stream(reinterpret_cast<const double *>(m.col), m.nnz / 2, sink, sm_count, s));
    return launch_read_stream(reinterpret_cast<const double *>(m.rp), rows + 1, sink, sm_count, s);
}

#undef CU

} // namespace cgb
