/*
 * cgb200.h -- C ABI of the B200-native conjugate-gradient hot path.
 *
 * The reference (federicobetti99/Conjugate-Gradient) has no plugin / FFI surface: its only
 * stable interfaces are the `cgsolver` command line + results file and the C++ class
 * `CGSolver` (code/MPI/cg.hh:11-57, code/CUDA/cg.hh:13-45).  This ABI sits directly UNDER
 * `CGSolver::solve`; every entry point below names the reference code it replaces.  The host
 * program `cgsolver` (conjugate-gradient_b200/host/) and the Python mirror bind exactly these
 * symbols; INTEGRATION.md shows the stub a maintainer of the reference would add.
 *
 * Conventions: plain pointers and sizes, no C++/torch types; every function returns a
 * cgb_status (0 = ok) and never throws or exits; cgb_last_error() gives the message of the
 * last failure on the calling thread.  Host buffers belong to the caller, device buffers to
 * the library.  One cgb_ctx = one rank = one GPU holding one contiguous row shard of A
 * (reference rule partition_matrix, code/MPI/cg.cc:236-268); a ctx is not thread-safe, but
 * different ctxs may be driven from different threads or processes.  There is no CPU
 * fallback: without a CUDA device every compute entry point fails with CGB_ERR_NO_DEVICE.
 */
#ifndef CGB200_H
#define CGB200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CGB_ABI_VERSION 1

typedef enum cgb_status {
    CGB_OK = 0,
    CGB_ERR_INVALID = 1,   /* bad argument */
    CGB_ERR_STATE = 2,     /* call out of order (e.g. solve before the matrix is set) */
    CGB_ERR_NO_DEVICE = 3, /* no CUDA device / driver */
    CGB_ERR_CUDA = 4,      /* a CUDA runtime call failed */
    CGB_ERR_NCCL = 5,      /* NCCL missing or a NCCL call failed */
    CGB_ERR_NOMEM = 6,
    CGB_ERR_TIMEOUT = 7    /* a device-side wait on another rank exceeded "spin_timeout_ms" */
} cgb_status;

typedef struct cgb_ctx cgb_ctx;

/* ---- library ------------------------------------------------------------------------- */
int cgb_abi_version(void);
const char *cgb_last_error(void);
int cgb_device_count(int *count);

/* CGSolver::partition_matrix (code/MPI/cg.cc:236-268) with 64-bit indices: ranks 0..P-2 get
 * N/P rows, the last rank the remainder. */
int cgb_partition(int64_t n, int psize, int64_t *start_rows, int64_t *num_rows);

/* ---- context ------------------------------------------------------------------------- */
/* One rank of `world` on CUDA device `device`, for an n x n system.  Allocates the row shard
 * (rows x ld doubles, ld = n rounded up to 16) and the work vectors -- the
 * std::vector / cudaMallocManaged temporaries of solve (cg.cc:55-75, cg.cu:179-193). */
int cgb_create(int64_t n, int rank, int world, int device, cgb_ctx **out);

/* The same rank with the shard held in CSR storage: no dense shard is allocated, so the system
 * size is bounded by the non-zeros, not by n^2 (n <= INT32_MAX: column indices are int32_t,
 * global; row pointers int64_t; values double; columns ascending and unique within a row).
 * The matrix comes from cgb_generate_lap2d, cgb_set_matrix_coo, cgb_set_matrix_csr or cgb_assemble_coo
 * (built on the device), its values may be refreshed with cgb_update_matrix_values or cgb_assemble_values;
 * cgb_set_matrix_rows returns CGB_ERR_STATE.  Vectors, exchange wiring and cgb_get_layout are
 * those of cgb_create; the solve runs on the graph schedule ("schedule_in_use" reads 0).
 * Exactness: the CSR mat-vec keeps the lane order of the dense one over the stored entries, and
 * a zero entry never changes a lane-order sum, so every result -- k, the r'r history, x, the
 * DEBUG numbers, the hooks -- is bitwise that of a dense context holding the same matrix as long
 * as the vector multiplied stays finite.  (A NaN / Inf of p at a column where A is zero makes the
 * dense row NaN and leaves the CSR row alone; only an already diverged solve gets there.)
 * Options: "compat" = 1, "loopback" > 0 and "trace" > 0 return CGB_ERR_STATE; "gemv_variant",
 * "num_threads", "block_width" and "transposed" are accepted and change nothing; cgb_autotune
 * changes nothing and reports every candidate as not run.  Read-only: "storage" (0 dense,
 * 1 CSR), "nnz" (entries stored in this rank's shard), "envelope_doubles" (dense: the sum over
 * this rank's rows of last + 1 - first non-zero column, the part of each row the mat-vecs stream;
 * 0 on a CSR context). */
int cgb_create_csr(int64_t n, int rank, int world, int device, cgb_ctx **out);
int cgb_destroy(cgb_ctx *ctx);

/* Replaces MPI_Init_thread / MPI_COMM_WORLD (code/MPI/cg_main.cc:15-20): rank 0 obtains an
 * id with cgb_comm_unique_id, ships it to the other ranks by any means, and every rank calls
 * cgb_comm_init (collective; wraps ncclCommInitRank).  Not needed when world == 1. */
#define CGB_UNIQUE_ID_BYTES 128
int cgb_comm_unique_id(void *id_out);
int cgb_comm_init(cgb_ctx *ctx, const void *id);

/* Fused exchange (the B200-native replacement of MPI_Allgatherv, cg.cc:135-136): the mat-vec
 * kernel stores its rows directly into every rank's gather buffer over NVLink and raises a
 * flag; no collective kernel runs.  Every rank exports a blob describing its buffer, the blobs
 * are shipped to all ranks by any means (world x CGB_EXCHANGE_BLOB_BYTES, rank order) and
 * imported; ranks may be threads of one process (peer access) or separate processes (CUDA
 * IPC).  After the import the option "exchange" is 1 (fused); 0 selects ncclAllGather, which
 * needs cgb_comm_init instead.  Like a collective, every rank must issue the same sequence of
 * solves / mat-vec hooks. */
#define CGB_EXCHANGE_BLOB_BYTES 128
int cgb_exchange_export(cgb_ctx *ctx, void *blob_out);
int cgb_exchange_import(cgb_ctx *ctx, const void *blobs);

/* ---- inputs -------------------------------------------------------------------------- */
/* CGSolver::generate_lap2d_matrix (code/MPI/cg.cc:159-188), this rank's rows built on the device
 * (values exactly 0, -1, 4; inc = floor(sqrt(n))): staged as CSR (5 non-zeros per row), then taken
 * over by a CSR context or densified into a dense one, padding columns zeroed. */
int cgb_generate_lap2d(cgb_ctx *ctx);

/* Dense rows from the host (what Matrix::read, matrix.cc:6-22, produces): `nrows` rows
 * starting at GLOBAL row `first_row`, row-major with leading dimension `ld_host`; the part
 * that falls inside this rank's shard is uploaded, the rest ignored. */
int cgb_set_matrix_rows(cgb_ctx *ctx, const double *rows_host, int64_t first_row, int64_t nrows,
                        int64_t ld_host);

/* Matrix::read's densification (matrix.cc:12-21) done on the device: the COO triples (0-based)
 * in file order, mirroring (j,i) when `symmetric`; later duplicates win, as in the reference, and
 * explicit zeros are stored.  The triples are uploaded once and this rank's rows staged as CSR (a
 * stable sort of the writes by row and column, the last of each run kept), which a CSR context takes
 * over and a dense one densifies, padding columns zeroed.  The staging takes about 82 bytes of device
 * memory per triple besides the shard and the sort's scratch, so a dense context loaded from a very
 * large COO (around 10^9 triples: some 82 GB) needs that much free next to its shard.  An entry
 * outside n x n returns CGB_ERR_INVALID before anything of the context is touched: the previous
 * matrix stays, and stays set. */
int cgb_set_matrix_coo(cgb_ctx *ctx, int64_t nz, const int32_t *irn, const int32_t *jcn,
                       const double *val, int symmetric);

/* This rank's rows [row0, row0 + rows) from a CSR matrix in device memory of the context's GPU:
 *   rp_dev   rows + 1 row pointers; local row i holds the entries rp[i] - rp[0] .. rp[i+1] - rp[0]
 *   col_dev  nnz = rp[rows] - rp[0] global columns, in [0, n) and strictly ascending within a row
 *   val_dev  nnz values (explicit zeros are stored, as by cgb_set_matrix_coo); empty rows are allowed
 * So a rank of a larger CSR passes rp + row0 and col / val + rp[row0], with nothing rebased.  col_dev and
 * val_dev may be null when nnz == 0.  The reads are ordered after the work enqueued on `stream` (a
 * cudaStream_t as void *, NULL = the legacy default stream) by an event; the call synchronises, like every
 * builder, and returns with the matrix built: the caller may overwrite its arrays afterwards.
 * The input is checked on the device before anything of the context is touched -- rp[0] >= 0, rp
 * monotone, rp[rows] - rp[0] == nnz, every column in range and strictly ascending; a row's columns are read
 * only after its rp pair has been checked.  A refusal returns CGB_ERR_INVALID with a message naming the
 * first offending local row, and the previous matrix stays as it was.
 * CSR context: the shard takes copies of the arrays (col / val are reallocated, so the next solve captures
 * its loop graph anew).  Dense context: the shard cgb_set_matrix_coo builds from the same triples.
 * CGB_ERR_STATE: a single or block solve between begin and end.  CGB_ERR_INVALID: nnz < 0, a null
 * pointer, a host pointer or one on another device.  Its kernels count in cgb_launch_count. */
int cgb_set_matrix_csr(cgb_ctx *ctx, const int64_t *rp_dev, const int32_t *col_dev, const double *val_dev,
                       int64_t nnz, void *stream);

/* New values for the matrix of a CSR context, its pattern kept: val_dev holds the context's "nnz" values
 * in stored order (rows ascending, columns ascending within a row -- cgb_set_matrix_csr's input order,
 * defined as well for a matrix from cgb_generate_lap2d or cgb_set_matrix_coo), in device memory of the
 * context's GPU (null allowed when nnz == 0).  Fully asynchronous: an event orders the copy after the work
 * enqueued on `stream` and after every solve already enqueued on the context from any stream, and work
 * enqueued on `stream` after the call sees the new values.  No host synchronisation, no allocation (the
 * first call of a context that has run no device solve creates two events), and the values array does
 * not move, so every cached loop graph stays valid: the next device solve is one graph launch, nothing
 * captured ("graph_captures" does not change).
 * CGB_ERR_STATE: a dense context (a dense shard keeps no pattern), the matrix not set, a single or block
 * solve between begin and end.  CGB_ERR_INVALID: a null pointer, a host pointer or one on another device. */
int cgb_update_matrix_values(cgb_ctx *ctx, const double *val_dev, void *stream);

/* Sum-assembly of COO contributions held in device memory of the context's GPU (finite-element or
 * finite-volume assembly: duplicates are added, as by scipy's coo_matrix.tocsr() or PETSc's ADD_VALUES).
 *   irn_dev, jcn_dev  nz 0-based global (row, column) pairs;  val_dev  nz values
 * Triple z makes write 2z at (i, j) and, with `symmetric` and i != j, write 2z+1 at (j, i).  A diagonal
 * triple is NOT mirrored -- in a sum that would double the diagonal.  This is the one deliberate difference
 * from the mirroring of cgb_set_matrix_coo (Matrix::read), which keeps the last write instead of adding.
 * Only writes whose row lies in this rank's shard are kept.  The value of a cell is the sequential left fold
 * of its writes in ascending write order, starting from the first write:
 *   v = w0;  v = v + w1;  v = v + w2; ...   (each + one IEEE double addition, rounded to nearest even)
 * This order is the contract: it makes the result reproducible and checkable bit for bit, and starting from
 * w0 rather than +0 keeps a lone -0 as -0.  The fold is serial per cell, so a cell that receives 10^5
 * writes is correct but slow; assembly gives a handful per cell.  Every cell that receives at least one
 * write is stored, explicit zeros and sums that cancel to zero included, so the pattern depends only on
 * (irn, jcn, symmetric), never on the values.  Dense and CSR contexts both work: this rank's rows are staged
 * as CSR and installed like cgb_set_matrix_csr's.  The reads are ordered after the work enqueued on `stream`
 * by an event; the call synchronises, like every builder.  Staging takes about 66 bytes of device memory per
 * triple besides the shard, the plan and the sort's scratch.
 * The call keeps an assembly plan in the context for cgb_assemble_values: 8 bytes per write kept in this
 * shard and 8 bytes per stored entry (+ 8), and on a dense context also the staged row pointers and columns
 * (8 bytes per row + 8, 4 bytes per stored entry).  Any other builder (cgb_generate_lap2d,
 * cgb_set_matrix_coo, cgb_set_matrix_csr, cgb_set_matrix_rows) frees it; cgb_update_matrix_values leaves it.
 * CGB_ERR_INVALID: nz < 0, a null, host or other-device pointer (nz > 0), or an entry outside n x n.  The
 * entries are checked on the device before anything of the context is touched, so after a refusal the
 * previous matrix and its plan stay.  CGB_ERR_STATE: a single or block solve between begin and end.
 * Its kernels count in cgb_launch_count. */
int cgb_assemble_coo(cgb_ctx *ctx, int64_t nz, const int32_t *irn_dev, const int32_t *jcn_dev,
                     const double *val_dev, int symmetric, void *stream);

/* Re-assembly: val_dev holds nz new values for the SAME triples as the last cgb_assemble_coo (same irn, jcn,
 * symmetric, nz; only the values differ), in device memory of the context's GPU (null allowed when nz == 0).
 * It writes the matrix cgb_assemble_coo would build from them, bit for bit, with the same fold order, by one
 * gather-and-fold kernel over the plan.  Fully asynchronous, like cgb_update_matrix_values: an event orders
 * it after the work enqueued on `stream` and after every solve already enqueued on the context, and work
 * enqueued on `stream` after the call sees the new matrix.  No host synchronisation, no allocation.  A CSR
 * context's values are written in place, so every cached loop graph stays valid ("graph_captures" does not
 * change).  A dense context's cells are written in A and then every row's envelope is rebuilt: a cell that
 * was an explicit zero at assembly may now be non-zero.
 * CGB_ERR_STATE: no plan (no cgb_assemble_coo yet, or another builder replaced its matrix), a single or
 * block solve between begin and end.  CGB_ERR_INVALID: a null pointer, a host pointer or one on another
 * device. */
int cgb_assemble_values(cgb_ctx *ctx, const double *val_dev, void *stream);

/* Read rows of the shard back (tests); a CSR shard is densified. */
int cgb_get_matrix_rows(cgb_ctx *ctx, double *rows_host, int64_t first_row, int64_t nrows,
                        int64_t ld_host);

/* CGSolver::init_source_term (code/MPI/cg.cc:218-234, code/CUDA/cg.cu:324-340):
 * b_i = -2 i pi^2 sin(10 pi i h)^2 into a caller-owned HOST buffer of n doubles.  Like the
 * reference this is a host loop over libm sin (the values feed cgb_set_rhs); it is the one
 * entry point that needs no GPU. */
int cgb_init_source_term(int64_t n, double h, double *b_host);

/* Right-hand side m_b (filled on the host by init_source_term, cg.cc:218-234, so that libm
 * sin is shared with the reference), full length n. */
int cgb_set_rhs(cgb_ctx *ctx, const double *b_host);

/* ---- tuning -------------------------------------------------------------------------- */
/* Integer options.  "gemv_variant": index into the table cgb_gemv_variant_name() lists;
 * "num_threads"/"block_width": the NUM_THREADS / BLOCK_WIDTH command-line knobs of the
 * reference CUDA program (code/CUDA/cg_main.cc:21-25), mapped onto threads per CTA and
 * column-tile width of the mat-vec; "graph": 0/1 CUDA-graph replay of the iteration;
 * "poll_every" / "graph_unroll": graph schedule only -- iterations between two looks at the stop flag and
 * iterations per graph (the instantiated graph holds min of the two; "graph_replays", read-only,
 * counts its launches, and those of the block solve's graph; "graph_captures", read-only, counts the
 * loop graphs -- host and device loops, single and block -- this context has captured and instantiated);
 * "pdl": 0/1 programmatic dependent launch between the kernels of the iteration (the next
 * mat-vec prefetches A while the vector updates still run); "l2_prefetch": pipeline steps of A
 * the mat-vec additionally pulls into L2 before that wait (0 = off); "l2_ramp": persistent
 * schedule only -- further steps pulled into L2 the moment p arrives, so that HBM keeps
 * streaming while the steps already on chip are consumed (default 2, 0 = off);
 * "exchange": 0 ncclAllGather / 1 fused peer stores (see cgb_exchange_import);
 * "schedule": 1 (default) = the whole loop of cgb_iterate as ONE persistent cooperative kernel
 * (one CTA per SM stays resident, the iteration's dependencies are data-flow waits inside the
 * kernel, A streams across iteration boundaries), 0 = a CUDA graph of four kernels per
 * iteration; bitwise identical results; "schedule_in_use" (read-only) tells which one the
 * current configuration gets (the persistent kernel needs the fused exchange, a 1-CTA-per-SM
 * variant, and is not used with "compat" / "profile");
 * "spin_timeout_ms": bound of the device-side waits on other ranks (default 20000); when it
 * expires the call returns CGB_ERR_TIMEOUT (the context is then unusable);
 * "balance": 1 (default) = the persistent kernel re-partitions the rows between its CTAs from the
 * mat-vec times they measure, when a CTA has at least 64 rows (no result bit depends on the partition);
 * "trace": launches kept by the diagnostic timeline (cgb_trace_read; 0 = off);
 * "loopback": profiling aid -- a rank of world > 1 with no peers aims every peer pointer of the
 * fused exchange at its own buffer, so ONE GPU runs one rank's shard under the production
 * schedule (timing and traffic are real, the numbers are not a CG solve);
 * "transposed": the reference's true/false kernel switch (accepted, A is symmetric);
 * "compat": 1 = run the mat-vec in the reference CUDA program's own topologies (MatVecT /
 * MatVec, code/CUDA/cg.cu:14-110) with num_threads / block_width / transposed honoured
 * literally but a deterministic chunk reduction instead of atomicAdd -- single GPU, for the
 * NUM_THREADS x BLOCK_WIDTH sweep of BASELINE.json config 5; set the three knobs first. */
int cgb_set_option(cgb_ctx *ctx, const char *key, int64_t value);
int cgb_get_option(cgb_ctx *ctx, const char *key, int64_t *value);
int cgb_gemv_variant_count(void);
const char *cgb_gemv_variant_name(int variant);

/* One-off choice of the mat-vec tile shape ("gemv_variant") for this rank's shard shape on this
 * GPU: every candidate shape runs `iters` (<= 0: 32) loop bodies of the schedule in use on the
 * resident matrix, the fastest becomes the configured variant.  Call it after the matrix is
 * set and OUTSIDE any timed region (the reference's timer brackets solve() only,
 * code/MPI/cg_main.cc:53-55).  A rank of world > 1 tunes alone (its exchange looped back to
 * itself on scratch buffers); peers need not take part or wait.  All shapes share one summation order:
 * the choice never changes a result bit.  us_per_iter (nullable, cgb_gemv_variant_count()
 * floats) receives the time of every candidate, < 0 for shapes that were not candidates. */
int cgb_autotune(cgb_ctx *ctx, int iters, int *chosen, float *us_per_iter);

typedef struct cgb_layout {
    int64_t n, ld, rows, row0; /* shard geometry */
    int rank, world, device;
    int nblk;                  /* mat-vec grid (CTAs); no reduction depends on it */
    int sm_count;
    int64_t nchunks;           /* 256-element chunks of the r'r reduction */
} cgb_layout;
int cgb_get_layout(cgb_ctx *ctx, cgb_layout *out);

/* ---- the hot path: CGSolver::solve (code/MPI/cg.cc:38-156, code/CUDA/cg.cu:166-305) ----- */
typedef struct cgb_solve_info {
    int64_t k;          /* the k of "[STEP k]": loop index at break, or max_iter */
    int converged;      /* loop left through sqrt(rsnew) < tol (cg.cc:120-121) */
    double rsold;       /* rsold at exit -- stale by one iteration after a break, as printed */
    double rsnew;       /* last r'r computed */
    double seconds;     /* device time of the iteration loop (CUDA events) */
    int64_t iterations; /* loop bodies executed on the device */
} cgb_solve_info;

/* Whole solve, host buffers in and out: x_host holds x0 on entry (n doubles), the solution
 * on return (every rank receives the full x -- MPI_Gatherv, cg.cc:140-142, delivered it to
 * rank 0 only).  resid_hist (nullable, capacity max_iter) receives r'r of every executed loop
 * index.  tol is the absolute tolerance on sqrt(r'r) (m_tolerance, cg.hh:56). */
int cgb_solve(cgb_ctx *ctx, double *x_host, int64_t max_iter, double tol, double *resid_hist,
              cgb_solve_info *info);

/* The same solve in three steps, for callers that keep the state on the device between
 * batches of iterations (bench.py's device-resident timing, the CLI's convergence polling):
 *   begin   : upload x0, r = b - A x0, p = r, rsold = r.p      (cg.cc:77-92)
 *   iterate : up to `iters` loop bodies (stops early on convergence); *ms = device time
 *   end     : download x, fill info                             (cg.cc:140-142) */
int cgb_solve_begin(cgb_ctx *ctx, const double *x0_host, int64_t max_iter, double tol,
                    int keep_history);
int cgb_iterate(cgb_ctx *ctx, int64_t iters, float *ms);
int cgb_solve_end(cgb_ctx *ctx, double *x_host, double *resid_hist, cgb_solve_info *info);

/* ---- block solve: up to CGB_MAX_RHS right-hand sides against one matrix ------------------
 * Column j of a block solve is, bit for bit, a single solve of A x = b_j from x0_j with the same
 * max_iter and tol: k, converged, rsold, rsnew, the r'r history and x.  The columns share every
 * read of the matrix (each row's CSR entries are loaded once per iteration for all of them) and
 * every launch, but no arithmetic.  A column that converges is frozen -- its x, r, p, scalars and
 * history stop changing -- while the others go on; the loop ends when every column has converged
 * or after max_iter loop bodies.
 * Layout: column j of b_host, x0_host and x_host is n contiguous doubles at offset j * n;
 * x0_host == NULL means zeros.  resid_hist (nullable) holds nrhs * max_iter doubles, column j's
 * r'r history at j * max_iter, filled like cgb_solve's for that column.  info is an array of
 * nrhs entries; `seconds` is the loop time all columns share.
 * Needs a CSR context of world == 1 with its matrix set (no cgb_set_rhs: the right-hand sides are
 * arguments).  CGB_ERR_STATE for a dense context (the tile pipeline of the dense mat-vec carries
 * one p), for world > 1 (the exchange carries one vector per row), before the matrix is set, and
 * while a single solve is in progress -- as cgb_solve_begin is refused during a block solve.
 * CGB_ERR_INVALID for nrhs outside [1, CGB_MAX_RHS] or a null b_host / x_host.
 * cgb_solve_block, like cgb_solve, takes the x0 columns in x_host and returns the solutions there.
 * Begin / iterate / end work as for the single solve; cgb_iterate advances whichever solve is in
 * progress and stops issuing launches once every column has converged.  The block solve has its
 * own device buffers (allocated on a context's first block solve, grown for a larger nrhs, freed
 * by cgb_destroy) and its own CUDA graph: it leaves the single solve's x, r, p, b, state, history
 * and graph untouched, so cgb_residual_check still reports the last single solve.
 * Options: "graph", "pdl", "poll_every" and "graph_unroll" apply as to a CSR single solve;
 * "profile" does not apply (the block loop runs as if it were 0), and cgb_last_gemv_timing keeps
 * describing single solves.  Block launches count in cgb_launch_count. */
#define CGB_MAX_RHS 8
int cgb_solve_block_begin(cgb_ctx *ctx, int nrhs, const double *b_host, const double *x0_host,
                          int64_t max_iter, double tol, int keep_history);
int cgb_solve_block_end(cgb_ctx *ctx, double *x_host, double *resid_hist, cgb_solve_info *info);
int cgb_solve_block(cgb_ctx *ctx, int nrhs, const double *b_host, double *x_host, int64_t max_iter,
                    double tol, double *resid_hist, cgb_solve_info *info);

/* ---- device solves: device memory in and out, ordered on the caller's stream ----------------
 * cgb_solve_device is cgb_set_rhs + cgb_solve on buffers that live on the context's GPU:
 *   b_dev     n doubles, the right-hand side
 *   x_dev     n doubles, x0 on entry, the solution once the stream reaches the end of the solve
 *   hist_dev  (nullable) max(max_iter, 1) doubles, receives r'r of every executed loop index
 *   info_dev  one cgb_solve_info in device memory
 *   stream    a cudaStream_t passed as void * (NULL = the legacy default stream)
 * Stream-ordered and asynchronous: the solve sees all work enqueued on `stream` before the call, and
 * work enqueued on `stream` after the call sees the finished x, history and info (an event recorded on
 * `stream` is waited on by the context's own stream, and the reverse at the end).  Nothing waits for
 * the host in between: the loop's stop test and its max_iter cap are decided on the device, and the
 * whole loop is one launch -- the persistent kernel, or on the graph schedule one CUDA graph whose
 * conditional WHILE nodes repeat the loop bodies.  Repeated solves of the same shape and options
 * return without any host synchronisation; the first device solve of a context, and one that needs
 * a larger history or block buffer than any before, allocate and may synchronise.
 * Bits: k, converged, rsold, rsnew, iterations, the r'r history and x equal those of cgb_set_rhs +
 * cgb_solve on the same context, on every schedule and storage.  info_dev->seconds is the device time
 * of the loop from %globaltimer stamps of its first and last kernel.  Like cgb_set_rhs + cgb_solve,
 * the solve leaves b and x in the context, so cgb_residual_check reports it.
 * cgb_solve_block_device is cgb_solve_block likewise: column j of B_dev / X_dev at j * n, hist_dev
 * (nullable) nrhs * max_iter doubles with column j at j * max_iter, info_dev nrhs entries; it keeps to
 * the block buffers and leaves the single solve alone, as cgb_solve_block does.
 * CGB_ERR_STATE: world > 1 (the fused exchange cannot be validated on one GPU, and the ncclAllGather
 * exchange needs the ranks in host lockstep), a host solve or block solve between begin and end, the
 * matrix not set, and for the block form whatever cgb_solve_block_begin refuses.
 * CGB_ERR_INVALID: a null pointer, a host pointer or one on another device (cudaPointerGetAttributes),
 * max_iter < 0, nrhs outside [1, CGB_MAX_RHS].
 * Options: the solve runs as if "profile" were 0, as the block solve does; its graph launches count in
 * "graph_replays" (one per solve on the graph schedule) and its kernels in cgb_launch_count, the loop
 * counted as if it ran to max_iter.  "device_loop_pdl" (read-only): 1 when the loop graph's bodies
 * keep the programmatic dependent launches, 0 when they are captured without, -1 before the first.
 * A device fault surfaces as CGB_ERR_CUDA at the next call on the context that synchronises. */
int cgb_solve_device(cgb_ctx *ctx, const double *b_dev, double *x_dev, int64_t max_iter, double tol,
                     double *hist_dev, cgb_solve_info *info_dev, void *stream);
int cgb_solve_block_device(cgb_ctx *ctx, int nrhs, const double *B_dev, double *X_dev, int64_t max_iter,
                           double tol, double *hist_dev, cgb_solve_info *info_dev, void *stream);

/* The DEBUG block at the end of solve (cg.cc:144-154, cg.cu:272-296): ||x|| and
 * ||A x - b|| / ||b|| for the x held on the device after a solve. */
int cgb_residual_check(cgb_ctx *ctx, double *norm_x, double *rel_resid);

/* ---- kernel-level hooks (tests, ncu, roofline) ------------------------------------------ */
/* y = A_shard . v through the production mat-vec: v_host has n doubles; y_host (nullable)
 * receives this rank's `rows` results, chunk_partials (nullable, `nchunks` of cgb_get_layout) the
 * partial sums of v_i * (A v)_i over the 256-element chunks of the GLOBAL vector (all ranks'
 * rows, after the exchange), pAp (nullable) their deterministic total -- level 1 and 2 of the
 * reduction that replaces cblas_ddot + MPI_Allreduce (cg.cc:105-106). */
int cgb_gemv(cgb_ctx *ctx, const double *v_host, double *y_host, double *chunk_partials,
             double *pAp);
/* Deterministic two-level dot of two host vectors (n doubles each) on the device. */
int cgb_dot(cgb_ctx *ctx, const double *a_host, const double *b_host, double *result);
/* `reps` back-to-back launches of mat-vec variant `variant` (-1 = the configured one) on the
 * resident shard and the resident p; *ms_avg = average device time per launch. */
int cgb_bench_gemv(cgb_ctx *ctx, int variant, int reps, float *ms_avg);
/* Streams the shard once with a plain read-only kernel: the read-bandwidth ceiling. */
int cgb_bench_read(cgb_ctx *ctx, int reps, float *ms_avg);
/* Average device time of the mat-vec launches inside the last cgb_iterate that ran with the
 * option "profile" = 1 (per-launch CUDA events). */
int cgb_last_gemv_timing(cgb_ctx *ctx, float *ms_avg, int64_t *launches);
/* Kernel launches issued by this ctx since creation (bench.py's gpu_launches). */
int cgb_launch_count(cgb_ctx *ctx, int64_t *launches);
/* Diagnostic timeline of the iteration under its PRODUCTION schedule (CUDA graph + programmatic
 * dependent launch, where no CUDA event can sit between the kernels).  With the option
 * "trace" = L every CTA of the loop kernels stamps %globaltimer (ns) into a ring of the last L
 * launches; this call copies the ring of kernel `which` (0 = mat-vec, 1 = x/r update, 2 = p
 * update) to `out` as [L][*blocks][8] words and reports how many launches were seen in total.
 * mat-vec words: 0 entry, 1 ring pre-filled, 2 dependency met (p final), 3 first tile
 * consumed, 4 last tile issued, 5 rows done, 6 exit, 7 = smid | rows << 32.  vector kernels:
 * 0 entry, 1 dependency met, 2 scalar known, 3 exit.  The replacement for what the reference
 * measures with one chrono pair around solve (code/MPI/cg_main.cc:53-55). */
int cgb_trace_read(cgb_ctx *ctx, int which, uint64_t *out, int64_t capacity_words,
                   int64_t *launches, int64_t *blocks);

#ifdef __cplusplus
}
#endif
#endif /* CGB200_H */
