// cgb_kernels.h -- host-callable launchers of the sm_100a kernels (gemv.cu, spmv.cu, vec.cu).
#pragma once

#include "cgb_device.cuh"

#include <cstring>

#include <utility>

struct cgb_solve_info; // include/cgb200.h

namespace cgb {

// Launch with (pdl = true) or without the programmatic-stream-serialization attribute: the
// kernels of the CG loop are chained with programmatic dependent launches so that the next
// kernel is already resident (and the mat-vec already prefetching A) when its predecessor ends.
template <class... KArgs, class... Args>
inline cudaError_t launch_kernel(void (*kernel)(KArgs...), int grid, int block, size_t smem,
                                 cudaStream_t stream, bool pdl, Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3((unsigned)grid, 1, 1);
    cfg.blockDim = dim3((unsigned)block, 1, 1);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
// the same with a 2-D grid (block solve: x = chunk, y = column)
template <class... KArgs, class... Args>
inline cudaError_t launch_kernel_xy(void (*kernel)(KArgs...), dim3 grid, int block, cudaStream_t stream, bool pdl,
                                    Args &&...args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid;
    cfg.blockDim = dim3((unsigned)block, 1, 1);
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}

// ---- mat-vec (gemv.cu) --------------------------------------------------------------
struct GemvVariant {
    const char *name;
    int ctas_per_sm; // grid = sm_count * ctas_per_sm persistent CTAs
    int threads;
    cudaError_t (*launch)(const GemvArgs &a, int nblk, cudaStream_t s);
    cudaError_t (*preload)(); // load the kernel now (lazy module loading), not at its first launch
};
int gemv_variant_count();
const GemvVariant &gemv_variant(int i);
cudaError_t launch_read_stream(const double *A, long long ndoubles, double *sink, int sm_count,
                               cudaStream_t s);

// ---- persistent schedule (persist.cu): the CG loop as one cooperative launch --------------
struct PersistVariant {
    const char *name; // = the gemv.cu variant with the same tile shape
    cudaError_t (*launch)(const PersistArgs &a, int nblk, cudaStream_t s);
    cudaError_t (*preload)();
    size_t (*smem_fixed)(); // shared memory without the size-dependent scratch (qs_n + scr_n doubles)
};
int persist_variant_count();
const PersistVariant &persist_variant(int i);
int persist_max_chunks(); // 256-element chunks of the vectors one CTA can own

// ---- reference-topology mat-vec (compat.cu): NUM_THREADS / BLOCK_WIDTH honoured literally ----
size_t compat_part_doubles(long long n, int block_width);
cudaError_t launch_compat_matvec(const GemvArgs &a, int nblk, int num_threads, int block_width,
                                 int transposed, double *part /* compat_part_doubles */, cudaStream_t s);

// ---- vector kernels (vec.cu) -------------------------------------------------------
// load every kernel of the solve path now instead of at first launch
cudaError_t preload_vec_kernels();
struct VecArgs {
    double *x, *r, *p;       // full-length (ld) replicated work vectors
    const double *b;
    const double *apx;       // gathered mat-vec result (see Gather)
    double *rrpart;          // nchunks chunk partials of r'r
    double *papart;          // nchunks chunk partials of p'Ap
    State *st;
    int *host_done;          // mapped pinned flag the host polls (nullable)
    double *hist;            // nullable
    Gather g;
    long long n;
    double tol;
    int pdl;                 // host side: chain update_xr / update_p with programmatic dependent launch
    Trace trace_xr, trace_p; // diagnostic timelines of update_xr / update_p (buf == nullptr: off)
    unsigned int *arrive;    // 2 zeroed arrival counters of the once-per-iteration phase (CSR contexts)
};
// r = b - A x0 ; p = r ; rrpart = chunk partials of r.p             (cg.cc:77-92)
cudaError_t launch_init_residual(const VecArgs &a, cudaStream_t s);
// chunk partials of p'Ap from the gathered rows                      (cg.cc:105)
cudaError_t launch_pap_partials(const VecArgs &a, cudaStream_t s);
// alpha = rsold / max(p'Ap, rsold*NEARZERO) ; x += alpha p ; r -= alpha Ap ; r'r partials
//                                                                   (cg.cc:106-117)
cudaError_t launch_update_xr(const VecArgs &a, cudaStream_t s);
// rsnew = sum(partials) ; stop test ; beta = rsnew/rsold ; p = r + beta p   (cg.cc:120-129)
cudaError_t launch_update_p(const VecArgs &a, cudaStream_t s);
// after the last iteration: rsold = rsnew, iter += 1 when the loop did not break (cg.cc:132)
cudaError_t launch_finalize(const VecArgs &a, cudaStream_t s);
// DEBUG block (cg.cc:144-154): out[0] = ||x||, out[1] = ||Ax-b|| / ||b||, given apx = A x
cudaError_t launch_debug_norms(const VecArgs &a, double *scratch /* 3*nchunks */, double *out,
                               cudaStream_t s);
// generic deterministic dot (tests): out[0] = a.b
cudaError_t launch_dot(const double *a, const double *b, long long n, double *scratch, double *out,
                       cudaStream_t s);
// hooks: chunk partials of v.(A v) from the plain gather buffer into papart, out[0] = their det_sum
cudaError_t launch_pap_plain(const double *v, const double *apx, const Gather &g, long long n, double *papart,
                             double *out, cudaStream_t s);

// The same three steps with every scalar computed ONCE per iteration (CSR contexts): the last
// block of pap_alpha reduces the p'Ap partials into alpha (st->conj, st->alpha), the last block of
// update_xr_once reduces the r'r partials into st->rsnew and takes the stop test, update_p_once
// reads both.  Per-iteration traffic is O(N) and nothing is sized by the chunk count; every State
// transition and every bit equals the kernels above.
cudaError_t launch_pap_alpha(const VecArgs &a, cudaStream_t s);
cudaError_t launch_update_xr_once(const VecArgs &a, cudaStream_t s);
cudaError_t launch_update_p_once(const VecArgs &a, cudaStream_t s);

// fused mode, hooks only: consume the running exchange into the plain gather buffer `apx`
// (the kernels of the iteration read the LL entries directly)
cudaError_t launch_exchange_collect(double *apx, const Gather &g, cudaStream_t s);

// ---- matrix construction ------------------------------------------------------------
// Every builder of a shard, dense or CSR, makes this rank's local CSR on the device (spmv.cu: lap2d_row
// is the one statement of generate_lap2d_matrix's stencil, csr_assemble_coo the one staging of COO triples,
// fold_run the one statement of how a cell's writes become its value: Matrix::read's last write or a sum),
// and capi.cu installs it: a CSR context adopts it, a dense one densifies it and rebuilds the envelopes.

// device scratch freed on every path
struct DevBuf {
    void *p = nullptr;
    ~DevBuf() { cudaFree(p); }
    cudaError_t alloc(size_t bytes) { return cudaMalloc(&p, bytes > 0 ? bytes : 1); }
    template <class T> T *as() const { return static_cast<T *>(p); }
};
// non-zero envelope of local rows [lr0, lr0 + nrows) of the dense shard into env (see block_window; vec.cu)
cudaError_t launch_row_envelope(const double *A, long long ld, long long lr0, long long nrows, int2 *env,
                                cudaStream_t s);

// ---- CSR storage (spmv.cu) ----------------------------------------------------------
// The shard: rp[rows + 1] (rebased to 0), col[nnz] (ascending and unique per row) / val[nnz]
struct CsrShard {
    long long *rp = nullptr;
    int *col = nullptr;
    double *val = nullptr;
    long long nnz = 0;
};
cudaError_t preload_spmv_kernels();
// the CSR mat-vec, lane order (bitwise the dense mat-vec); a.csr_* set
cudaError_t launch_spmv(const GemvArgs &a, int sm_count, cudaStream_t s);
// The builders fill an empty shard `m` (all of its arrays allocated here, freed by the caller on every
// path) and synchronise.
// generate_lap2d_matrix's non-zeros of rows [row0, row0 + rows)
cudaError_t csr_generate_lap2d(CsrShard *m, long long n, long long row0, long long rows, cudaStream_t s);
// COO triples in device memory (DESIGN 3.6, 3.11).  Triple z makes write 2z at (irn[z], jcn[z]) and, symmetric
// and off the diagonal, write 2z+1 at (jcn[z], irn[z]).  A stored entry folds its writes in write order: to the
// last (cgb_set_matrix_coo, Matrix::read) or to their left-fold sum (cgb_assemble_coo).  The plan lets every
// later set of values for the same triples be folded without a sort.
enum AsmFold { kFoldSum, kFoldLast };
struct AsmPlan {
    long long *wid = nullptr;   // [nwrites] the writes this shard keeps, sorted by (row, column, write id)
    long long *start = nullptr; // [nnz + 1] entry e (stored order) folds wid[start[e] .. start[e+1])
    long long *rp = nullptr;    // dense contexts: the staged row pointers and columns, to find A's cells
    int *col = nullptr;
    long long nz = 0, nnz = 0, nwrites = 0, rows = 0;
};
void asm_plan_free(AsmPlan *p);
// this rank's rows of the triples into an empty shard `m` and, if `p` is not null, plan `p` (wid / start; rp /
// col are left null), synchronised; *bad_host = 1 (and `m`, `p` left empty) when an entry lies outside n x n
cudaError_t csr_assemble_coo(CsrShard *m, AsmPlan *p, AsmFold fold, long long n, long long row0, long long rows,
                             const int *irn, const int *jcn, const double *val, long long nz, int symmetric,
                             int *bad_host, cudaStream_t s);
// the plan's fold of nz values: into a CSR shard's values (stored order), or by sum into the cells of the dense
// rows x ld shard A (p.rp / p.col set)
cudaError_t launch_assemble_csr(const AsmPlan &p, AsmFold fold, const double *val, double *out, cudaStream_t s);
cudaError_t launch_assemble_dense(const AsmPlan &p, const double *val, long long ld, double *A, cudaStream_t s);
// col / val of `nnz` entries for a shard without them
cudaError_t csr_alloc_entries(CsrShard *m, long long nnz);
// rows [lr0, lr0 + nrows) of a CSR (rp indexing col / val from 0) into a dense nrows x ld device buffer,
// zeroed first (padding columns included)
cudaError_t csr_densify(const long long *rp, const int *col, const double *val, long long lr0, long long nrows,
                        long long ld, double *dst, cudaStream_t s);
// A caller's CSR of `rows` rows against the stored format (cgb_set_matrix_csr): rp[0] >= 0, rp monotone,
// rp[rows] - rp[0] == nnz, columns in [0, n) and strictly ascending per row.  *err = ~0 when it holds,
// else the first fault as row * kCsrFaultKinds + kind; rp_local[rows + 1] = rp - rp[0]
enum { kCsrNegativeBase, kCsrNotMonotone, kCsrPastNnz, kCsrColumnRange, kCsrNotAscending, kCsrCount, kCsrFaultKinds };
cudaError_t launch_validate_csr(const long long *rp, const int *col, long long nnz, long long n, long long rows,
                                long long *rp_local, unsigned long long *err, cudaStream_t s);
// streams the three CSR arrays once (the read ceiling of the CSR mat-vec)
cudaError_t launch_read_csr(const CsrShard &m, long long rows, double *sink, int sm_count, cudaStream_t s);

// ---- block solve (CSR, one rank): nrhs right-hand sides against one matrix (spmv.cu, vec.cu) ----
// Column j of x, r, p, b starts at j * ld, of ap at j * slot, of the chunk partials at j * nchunks,
// of the history at j * hist_ld; st[j] is its State.  Every column runs the kernels of a single CSR
// solve with its own scalars and arrival counters, so its bits are that solve's; a column whose
// st[j].done is set is skipped by every kernel, like a single solve after its break.
constexpr int kMaxRhs = 8;
struct BlockArgs {
    const long long *rp;      // the CSR shard
    const int *col;
    const double *val;
    const double *v;          // mat-vec input: x (init) or p (loop)
    double *x, *r, *p;
    const double *b;
    double *ap;               // mat-vec result, [nrhs][slot]
    double *rrpart, *papart;  // [nrhs][nchunks]
    State *st;                // [nrhs]
    unsigned int *arrive;     // [nrhs][2] zeroed arrival counters of pap_alpha / update_xr
    unsigned int *ndone;      // columns that have converged
    int *host_done;           // mapped pinned flag, raised when ndone reaches nrhs
    double *hist;             // nullable, [nrhs][hist_ld]
    long long n, ld, rows, slot, nchunks, hist_ld;
    int nrhs;
    int advance;              // mat-vec: 1 inside the CG loop (block 0 advances every live State)
    int pdl;
    double tol;
};
cudaError_t preload_spmv_block_kernels();
cudaError_t preload_vec_block_kernels();
// ap[j] = A v[j] for the live columns: rp / col / val read once per row for all of them
cudaError_t launch_spmv_block(const BlockArgs &a, int sm_count, cudaStream_t s);
// r = b - A x0 ; p = r ; r'r chunk partials, per column
cudaError_t launch_init_residual_block(const BlockArgs &a, cudaStream_t s);
// pap_alpha / update_xr_once / update_p_once / finalize per column (grid y = column)
cudaError_t launch_pap_alpha_block(const BlockArgs &a, cudaStream_t s);
cudaError_t launch_update_xr_block(const BlockArgs &a, cudaStream_t s);
cudaError_t launch_update_p_block(const BlockArgs &a, cudaStream_t s);
cudaError_t launch_finalize_block(const BlockArgs &a, cudaStream_t s);

// ---- device solves (loop.cu): the loop's bookkeeping without the host --------------------------
// `limit` = max_iter of the solve, `bodies` = loop bodies issued so far, `t0` = %globaltimer at the
// loop's start (0: no loop ran)
struct LoopCtl {
    long long limit, bodies;
    unsigned long long t0, pad;
};
cudaError_t preload_loop_kernels();
// st[0 .. nst) = the State cgb_solve_begin uploads; ctl = {max_iter, 0, 0}
cudaError_t launch_device_begin(State *st, int nst, LoopCtl *ctl, long long max_iter, cudaStream_t s);
// bodies = reset ? 0 : bodies + add (reset also stamps t0); with `set`, the WHILE condition h = the stop
// test has not fired (*done, or *ndone == nrhs when done is null) and limit - bodies >= len
cudaError_t launch_loop_ctl(LoopCtl *ctl, const int *done, const unsigned int *ndone, int nrhs,
                            cudaGraphConditionalHandle h, int set, int len, int add, int reset, cudaStream_t s);
// info[j] from st[j] (as cgb_solve_end) and, hist_out non-null, the executed r'r history of column j
// from hist + j * hist_ld to hist_out + j * out_ld; seconds = %globaltimer now - ctl->t0
cudaError_t launch_device_info(const State *st, int nrhs, const LoopCtl *ctl, cgb_solve_info *info, const double *hist,
                               long long hist_ld, double *hist_out, long long out_ld, cudaStream_t s);

} // namespace cgb
