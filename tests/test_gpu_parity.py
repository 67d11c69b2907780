"""GPU parity tests: the sm_100a path, called through the C ABI, against the CPU oracle
(bitwise -- the oracle restates the kernels' exact summation order) and against the golden
fixtures produced by the unmodified reference (tolerances of BASELINE.json's north_star:
iteration count +-1, residual norms 1e-10 relative, final x 1e-9 relative).

Every test here needs a B200:  python -m pytest tests -m gpu
"""
import glob
import os

import numpy as np
import pytest

from parity_util import check_against_reference, reference_k_set

pytestmark = pytest.mark.gpu


def _rng(seed):
    return np.random.default_rng(seed)


def _ctx(cgb, n, **kw):
    return cgb.Context(n, kw.get("rank", 0), kw.get("world", 1), kw.get("device", 0))


# --------------------------------------------------------------------------- inputs
@pytest.mark.parametrize("n", [1, 2, 17, 1000, 1024, 2050])
def test_generate_lap2d_matches_oracle(cgb, O, n):
    """cgb_generate_lap2d == generate_lap2d_matrix (cg.cc:159-188), every element."""
    with _ctx(cgb, n) as ctx:
        ctx.generate_lap2d()
        A = ctx.get_matrix_rows(0, n)
    assert np.array_equal(A, O.generate_lap2d(n))


def test_generator_known_answers(cgb, O):
    """Analytic checks of SURVEY.md 8(c): symmetry, nnz, row sums in {0, 1, 2}."""
    n = 4096
    inc = int(np.floor(np.sqrt(n)))
    with _ctx(cgb, n) as ctx:
        ctx.generate_lap2d()
        A = ctx.get_matrix_rows(0, n)
        y, _ = ctx.gemv(np.ones(n))
    assert np.array_equal(A, A.T)
    assert np.count_nonzero(A) == n + 2 * (n - 1) + 2 * (n - 1 - inc)
    assert np.array_equal(y, A.sum(axis=1))          # small integers: exact in any order
    assert set(np.unique(y)).issubset({0.0, 1.0, 2.0})


def test_set_matrix_rows_and_coo_roundtrip(cgb, O, tmp_path):
    """Dense upload and device-side COO densification (matrix.cc:6-22) give the same shard,
    including 'later duplicates overwrite' and symmetric mirroring."""
    path = str(tmp_path / "lap.mtx")
    O.write_lap2d_5pt_mtx(path, 12)
    A = O.read_mtx_dense(path)
    n = A.shape[0]
    tri = [(i, j, A[i, j]) for j in range(n) for i in range(j, n) if A[i, j] != 0]
    irn = np.array([t[0] for t in tri] + [5, 5], dtype=np.int32)
    jcn = np.array([t[1] for t in tri] + [3, 3], dtype=np.int32)
    val = np.array([t[2] for t in tri] + [7.0, 9.0])     # duplicate cell: 9.0 must win
    expect = A.copy()
    expect[5, 3] = expect[3, 5] = 9.0
    with _ctx(cgb, n) as ctx:
        ctx.set_matrix_rows(A)
        assert np.array_equal(ctx.get_matrix_rows(0, n), A)
        ctx.set_matrix_coo(irn, jcn, val, symmetric=True)
        assert np.array_equal(ctx.get_matrix_rows(0, n), expect)


@pytest.mark.parametrize("symmetric", [False, True])
def test_set_matrix_coo_million_random_duplicates(cgb, symmetric):
    """Device-side densification with heavy cell collisions: 10^6 random triples into a 1500 x 1500
    matrix (every cell is written ~0.4 / ~0.9 times on average, thousands of cells many times).  The
    result must be the SEQUENTIAL loop of matrix.cc:12-21 -- the last entry in file order wins, the
    mirror write of a symmetric entry included -- although the scatter runs in parallel."""
    n, nz = 1500, 1_000_000
    rng = _rng(11 + int(symmetric))
    irn = rng.integers(0, n, nz, dtype=np.int32)
    jcn = rng.integers(0, n, nz, dtype=np.int32)
    val = rng.standard_normal(nz)
    if symmetric:   # write order: (i, j) of entry 0, (j, i) of entry 0, (i, j) of entry 1, ...
        cells = np.stack([irn.astype(np.int64) * n + jcn, jcn.astype(np.int64) * n + irn], axis=1).ravel()
        vals = np.repeat(val, 2)
    else:
        cells, vals = irn.astype(np.int64) * n + jcn, val
    u, first_in_reversed = np.unique(cells[::-1], return_index=True)
    expect = np.zeros(n * n)
    expect[u] = vals[len(cells) - 1 - first_in_reversed]
    with _ctx(cgb, n) as ctx:
        ctx.set_matrix_coo(irn, jcn, val, symmetric=symmetric)
        assert np.array_equal(ctx.get_matrix_rows(0, n), expect.reshape(n, n))
        with pytest.raises(cgb.CgbError):                       # an entry outside the matrix
            ctx.set_matrix_coo(np.array([0, n], dtype=np.int32), np.array([0, 0], dtype=np.int32),
                               np.array([1.0, 2.0]), symmetric=False)


# --------------------------------------------------------------------------- kernels
@pytest.mark.parametrize("n", [64, 1000, 2050, 4097])
def test_gemv_every_variant_bitwise(cgb, O, n):
    """Every mat-vec variant == the oracle's lane-order row dot, bit for bit; chunk partials
    and their deterministic total likewise."""
    rng = _rng(n)
    A = rng.standard_normal((n, n))
    p = rng.standard_normal(n)
    y_ref = O.gemv(A, p)
    with _ctx(cgb, n) as ctx:
        ctx.set_matrix_rows(A)
        for v, name in enumerate(cgb.gemv_variants()):
            ctx.set_option("gemv_variant", v)
            y, cp, pap = ctx.gemv(p, want_partials=True)
            assert np.array_equal(y, y_ref), name
            cp_ref = O.chunk_partials(p, y_ref)     # chunk256 partials of p_i * (A p)_i, global vector
            assert np.array_equal(cp, cp_ref), name
            assert pap == O.det_sum(cp_ref) == O.dot(p, y_ref), name


def test_gemv_exactness_properties(cgb, O):
    """Size-independent properties on the generator matrix: A e_j = column j = row j
    (symmetry), A (2p) = 2 (A p) exactly."""
    n = 3000
    rng = _rng(7)
    p = rng.standard_normal(n)
    with _ctx(cgb, n) as ctx:
        ctx.generate_lap2d()
        A = O.generate_lap2d(n)
        for j in (0, 1, 54, 55, 56, n - 1):
            e = np.zeros(n)
            e[j] = 1.0
            y, _ = ctx.gemv(e)
            assert np.array_equal(y, A[j])
        y1, _ = ctx.gemv(p)
        y2, _ = ctx.gemv(2.0 * p)
        assert np.array_equal(y2, 2.0 * y1)


@pytest.mark.parametrize("n", [1, 255, 256, 257, 5000])
def test_dot_bitwise(cgb, O, n):
    rng = _rng(100 + n)
    a, b = rng.standard_normal(n), rng.standard_normal(n)
    with _ctx(cgb, n) as ctx:
        assert ctx.dot(a, b) == O.dot(a, b)


# --------------------------------------------------------------------------- solve
SCHEDULES = {"persistent": (1, 1), "graph": (0, 1), "launches": (0, 0)}   # (schedule, graph)


def _solve_gpu(cgb, n, setup, max_iter, variant=None, graph=1, x0=None, schedule=None):
    with _ctx(cgb, n) as ctx:
        if variant is not None:
            ctx.set_option("gemv_variant", variant)
        ctx.set_option("graph", graph)
        if schedule is not None:
            ctx.set_option("schedule", schedule)
        setup(ctx)
        x = np.zeros(n) if x0 is None else x0.copy()
        info, hist = ctx.solve(x, max_iter=max_iter, tol=1e-10, history=True)
        nx, rr = ctx.residual_check()
        nblk = ctx.layout().nblk
    return x, info, hist, nx, rr, nblk


@pytest.mark.parametrize("n,max_iter", [(1000, 50), (1024, 1024), (1448, 200), (2048, 2048)])
@pytest.mark.parametrize("sched", list(SCHEDULES))
def test_solve_generated_bitwise_vs_oracle(cgb, O, n, max_iter, sched):
    """Whole solve == oracle bit for bit: iteration count, every r'r, final x, DEBUG numbers --
    under every schedule of the loop: ONE persistent cooperative kernel (csrc/persist.cu, the
    default), a CUDA graph of four kernels per iteration, plain launches."""
    b = O.init_source_term(n)

    def setup(ctx):
        ctx.generate_lap2d()
        ctx.set_rhs(b)

    schedule, graph = SCHEDULES[sched]
    x, info, hist, nx, rr, nblk = _solve_gpu(cgb, n, setup, max_iter, graph=graph, schedule=schedule)
    ref = O.solve(O.generate_lap2d(n), b, max_iter=max_iter, nranks=1, nblk=nblk)
    assert info.k == ref.k and bool(info.converged) == ref.converged
    assert info.iterations == len(ref.hist)
    assert np.array_equal(hist, ref.hist)
    assert np.array_equal(x, ref.x)
    assert info.rsold == ref.rsold and info.rsnew == ref.rsnew
    assert nx == ref.norm_x and rr == ref.rel_resid


def test_solve_nonzero_x0_and_variants(cgb, O):
    """x0 != 0 exercises the init mat-vec (cg.cc:77-82); every variant -- whatever its grid and tile
    shape -- gives the oracle's bits (no reduction depends on how rows are spread over CTAs)."""
    n = 1536
    rng = _rng(3)
    A = O.generate_lap2d(n)
    b = O.init_source_term(n)
    x0 = rng.standard_normal(n)
    for v, name in enumerate(cgb.gemv_variants()):
        def setup(ctx):
            ctx.generate_lap2d()
            ctx.set_rhs(b)
        x, info, hist, _, _, nblk = _solve_gpu(cgb, n, setup, 120, variant=v, x0=x0)
        ref = O.solve(A, b, x0=x0, max_iter=120, nranks=1, nblk=nblk)
        assert info.k == ref.k, name
        assert np.array_equal(hist, ref.hist), name
        assert np.array_equal(x, ref.x), name


def _persist_variants(cgb, n):
    """Variants for which the persistent kernel is instantiated (option "schedule_in_use")."""
    out = []
    with _ctx(cgb, n) as ctx:
        for v, name in enumerate(cgb.gemv_variants()):
            ctx.set_option("gemv_variant", v)
            if ctx.get_option("schedule_in_use") == 1:
                out.append((v, name))
    return out


@pytest.mark.parametrize("n", [1, 2, 17, 255, 257, 1001, 4097])
def test_persistent_schedule_ragged_sizes_every_shape(cgb, O, n):
    """The persistent kernel on ragged sizes (CTAs without rows, a last chunk of 1 element,
    tiles narrower than the tile width), every instantiated tile shape, against the oracle."""
    b = O.init_source_term(n)
    A = O.generate_lap2d(n)
    max_iter = min(n, 90)
    variants = _persist_variants(cgb, n)
    assert len(variants) >= 4, variants
    ref = None
    for v, name in variants:
        def setup(ctx):
            ctx.generate_lap2d()
            ctx.set_rhs(b)
        x, info, hist, nx, rr, nblk = _solve_gpu(cgb, n, setup, max_iter, variant=v, schedule=1)
        if ref is None:
            ref = O.solve(A, b, max_iter=max_iter, nranks=1, nblk=nblk)
        assert info.k == ref.k and bool(info.converged) == ref.converged, name
        # n = 1: b = [0], so alpha = 0/0 -- the reference, the oracle and the kernels all carry NaN
        assert np.array_equal(hist, ref.hist, equal_nan=True), name
        assert np.array_equal(x, ref.x, equal_nan=True), name
        assert np.array_equal([nx, rr], [ref.norm_x, ref.rel_resid], equal_nan=True), name


def _interleave_schedules(cgb, O, graph, profile):
    n = 3000
    b = O.init_source_term(n)
    with _ctx(cgb, n) as ctx:
        ctx.generate_lap2d()
        ctx.set_rhs(b)
        ctx.set_option("graph", graph)
        ctx.set_option("profile", profile)
        nblk = ctx.layout().nblk
        ctx.solve_begin(np.zeros(n), 150, 1e-10, True)
        for sched, iters in ((1, 7), (0, 20), (1, 1), (1, 40), (0, 3), (1, 79)):
            ctx.set_option("schedule", sched)
            ctx.iterate(iters)
        x, hist = np.zeros(n), np.zeros(150)
        info = ctx.solve_end(x, hist)
    ref = O.solve(O.generate_lap2d(n), b, max_iter=150, nranks=1, nblk=nblk)
    assert info.k == ref.k == 150 and info.iterations == 150
    assert np.array_equal(hist, ref.hist) and np.array_equal(x, ref.x)


def test_schedules_interleave_bitwise(cgb, O):
    """cgb_iterate in pieces, alternating the persistent kernel and the graph schedule on the
    same solve: the state handed over between launches (x, r, p, r'r partials, k) is complete,
    so any split gives the bits of one uninterrupted solve."""
    _interleave_schedules(cgb, O, graph=1, profile=0)


@pytest.mark.parametrize("graph,profile", [(0, 0), (1, 1), (0, 1)])
def test_schedules_interleave_launch_modes(cgb, O, graph, profile):
    """The same split when the graph-schedule pieces run as plain launches (graph = 0) or in
    profile mode, which launches without programmatic dependent launch and, since the persistent
    kernel cannot run there, keeps the whole solve on the graph schedule's kernels."""
    _interleave_schedules(cgb, O, graph=graph, profile=profile)


def test_vector_kernel_timelines(cgb, O):
    """Option "trace" on the graph schedule: thread 0 of every block of update_xr stamps entry <=
    dependency met <= alpha known <= exit, of update_p entry <= dependency met <= exit, in each of
    the last 8 launches, and each kernel counts one launch per iteration.  Every update_p block
    passes its dependency after every update_xr block of the same iteration has exited, and every
    update_xr block of the next iteration after every update_p block: a block that skipped a launch
    would leave a stale slot out of this order."""
    n, iters, cap = 3000, 40, 8
    with _ctx(cgb, n) as ctx:
        ctx.generate_lap2d()
        ctx.set_rhs(O.init_source_term(n))
        ctx.set_option("schedule", 0)
        ctx.set_option("trace", cap)
        info, _ = ctx.solve(np.zeros(n), max_iter=iters, tol=1e-10, history=True)
        nchunks = ctx.layout().nchunks
        xr, n_xr = ctx.trace_read(1)
        p, n_p = ctx.trace_read(2)
    assert info.iterations == iters and not info.converged
    assert n_xr == n_p == iters
    assert xr.shape == p.shape == (cap, nchunks, 8)
    xr, p = xr.astype(np.int64), p.astype(np.int64)
    assert np.all(xr[:, :, 0] > 0) and np.all(np.diff(xr[:, :, :4], axis=2) >= 0)
    assert np.all(p[:, :, 0] > 0) and np.all(p[:, :, 1] >= p[:, :, 0]) and np.all(p[:, :, 3] >= p[:, :, 1])
    assert np.all(p[:, :, 1].min(axis=1) >= xr[:, :, 3].max(axis=1))
    assert np.all(xr[1:, :, 1].min(axis=1) >= p[:-1, :, 3].max(axis=1))


@pytest.mark.parametrize("case", list(SCHEDULES) + ["csr"])
def test_nearzero_clamp_bitwise_vs_oracle(cgb, O, case):
    """alpha = rsold / max(p'Ap, rsold * NEARZERO) (cg.cc:107).  On -lap2d every p'Ap is negative,
    so the clamp fires in every iteration: alpha = rsold / (rsold * 1e-14) and r'r grows by ~1e57 per
    iteration (it overflows in the fourth, so three keep every number finite).  Dense storage under
    every schedule (one-iteration graphs, so the graph is replayed) and CSR storage, bit for bit
    against the oracle."""
    n, iters = 1000, 3
    A = -O.generate_lap2d(n)
    b = O.init_source_term(n)
    schedule, graph = SCHEDULES.get(case, (0, 1))
    with cgb.Context(n, storage="csr" if case == "csr" else "dense") as ctx:
        if case == "csr":
            i, j = np.nonzero(A)
            ctx.set_matrix_coo(i.astype(np.int32), j.astype(np.int32), A[i, j], symmetric=False)
        else:
            ctx.set_matrix_rows(A)
        ctx.set_rhs(b)
        ctx.set_option("schedule", schedule)
        ctx.set_option("graph", graph)
        ctx.set_option("graph_unroll", 1)
        assert ctx.get_option("schedule_in_use") == schedule
        x = np.zeros(n)
        info, hist = ctx.solve(x, max_iter=iters, tol=1e-10, history=True)
        nx, rr = ctx.residual_check()
        nblk = ctx.layout().nblk
    ref = O.solve(A, b, max_iter=iters, nranks=1, nblk=nblk)
    assert np.all(np.isfinite(ref.hist)) and np.all(np.isfinite(ref.x))
    assert info.k == ref.k == iters and info.iterations == iters
    assert np.array_equal(hist, ref.hist, equal_nan=True)
    assert np.array_equal(x, ref.x, equal_nan=True)
    assert np.array_equal([info.rsold, info.rsnew, nx, rr],
                          [ref.rsold, ref.rsnew, ref.norm_x, ref.rel_resid], equal_nan=True)
    # the first iteration (p = r = b) took the clamped step, not rsold / p'Ap
    rs = O.dot(b, b)
    assert O.dot(b, A @ b) < rs * 1e-14
    r1 = b - rs / (rs * 1e-14) * (A @ b)
    assert abs(hist[0] - r1 @ r1) <= 1e-12 * hist[0]


def test_solve_mtx_bitwise_vs_oracle(cgb, O, tmp_path):
    """Config 1's input family (5-point Laplacian .mtx) through the COO path, to convergence."""
    path = str(tmp_path / "lap30.mtx")
    O.write_lap2d_5pt_mtx(path, 30)
    A = O.read_mtx_dense(path)
    n = A.shape[0]
    b = O.init_source_term(n)

    def setup(ctx):
        ctx.set_matrix_rows(A)
        ctx.set_rhs(b)

    x, info, hist, nx, rr, nblk = _solve_gpu(cgb, n, setup, n)
    ref = O.solve(A, b, max_iter=n, nranks=1, nblk=nblk)
    assert info.k == ref.k and info.converged == 1
    assert np.array_equal(hist, ref.hist) and np.array_equal(x, ref.x)


def test_max_iter_zero_and_early_stop_semantics(cgb, O):
    """max_iter = 0 leaves x = x0 and k = 0; a converged run leaves rsold stale (the value
    the reference prints, cg.cc:152-153) and x untouched after the break."""
    n = 1024
    b = O.init_source_term(n)

    def setup(ctx):
        ctx.generate_lap2d()
        ctx.set_rhs(b)

    x, info, hist, *_ = _solve_gpu(cgb, n, setup, 0)
    assert info.k == 0 and info.iterations == 0 and not info.converged
    assert np.array_equal(x, np.zeros(n)) and len(hist) == 0
    x, info, hist, *_ = _solve_gpu(cgb, n, setup, n)
    assert info.converged and info.iterations == info.k + 1
    assert np.sqrt(hist[-1]) < 1e-10 <= np.sqrt(hist[-2])
    assert info.rsold == hist[-2] and info.rsnew == hist[-1]


# --------------------------------------------------------------------------- vs the reference
def _golden_cases(golden_dir):
    return sorted(glob.glob(os.path.join(golden_dir, "*.npz")))


def test_solve_matches_reference_golden(cgb, O, golden_dir, tmp_path):
    """Against outputs of the UNMODIFIED reference (OpenBLAS 0.3.15 behind cblas_*):
    k within +-1, r'r history within 1e-10 relative on the segment before the rounding floor
    (SURVEY.md 7.3: below ~1e-9 of the peak residual every summation order diverges, the
    reference's own two BLAS providers included), final x within 1e-9 relative."""
    cases = _golden_cases(golden_dir)
    assert cases, "golden fixtures missing"
    for f in cases:
        g = np.load(f)
        if "ranks" in g:
            continue  # multi-rank runs of the reference: tests/test_gpu_multi.py
        n, max_iter = int(g["n"]), int(g["max_iter"])
        b = O.init_source_term(n)
        if str(g["kind"]) == "mtx":
            path = str(tmp_path / "g.mtx")
            O.write_lap2d_5pt_mtx(path, int(g["grid"]))
            A = O.read_mtx_dense(path)

            def setup(ctx, A=A):
                ctx.set_matrix_rows(A)
                ctx.set_rhs(b)
        else:
            def setup(ctx):
                ctx.generate_lap2d()
                ctx.set_rhs(b)
        x, info, hist, nx, rr, _ = _solve_gpu(cgb, n, setup, max_iter)
        # k within +-1 of a count the reference itself produces for this system (its BLAS providers
        # disagree in the rounding-noise tail: N = 4096 stops at 358 with OpenBLAS, 385 with plain loops)
        check_against_reference(info.k, hist, x, g, "openblas", os.path.basename(f),
                                k_refs=reference_k_set(golden_dir, g))
        assert abs(nx - float(g["openblas_norm_x"])) <= 1e-6 * nx


# --------------------------------------------------------------------------- beyond the reference
def test_n_beyond_int32_indexing(cgb, O):
    """N = 46400 > 46340: the reference's `int` index i*m_n+j overflows (matrix.hh:17,
    cg.cc:80; SURVEY.md 8c), so there is no reference run -- size-independent properties
    instead: A.1 = analytic row sums, A e_j = generator row j (symmetry) at both ends of the
    index range, and the recursive residual of 40 CG iterations equals the true residual
    ||A x - b|| recomputed by the DEBUG block."""
    n = 46400
    inc = int(np.floor(np.sqrt(n)))
    with _ctx(cgb, n) as ctx:
        ctx.generate_lap2d()
        y, _ = ctx.gemv(np.ones(n))
        i = np.arange(n)
        neigh = (i > 0).astype(float) + (i < n - 1) + (i > inc) + (i < n - 1 - inc)
        assert np.array_equal(y, 4.0 - neigh)
        for j in (0, inc, inc + 1, n // 2, n - 2 - inc, n - 1):
            e = np.zeros(n)
            e[j] = 1.0
            yj, _ = ctx.gemv(e)
            assert np.array_equal(yj, O.generate_lap2d_rows(n, j, 1)[0]), j
        b = cgb.init_source_term(n)
        ctx.set_rhs(b)
        x = np.zeros(n)
        info, hist = ctx.solve(x, max_iter=40, tol=1e-10, history=True)
        nx, rr = ctx.residual_check()
    assert info.k == 40 and len(hist) == 40 and np.all(np.diff(np.sqrt(hist[5:])) != 0)
    true_resid = rr * np.linalg.norm(b)
    assert abs(true_resid - np.sqrt(info.rsold)) <= 1e-9 * true_resid
    assert abs(nx - np.linalg.norm(x)) <= 1e-12 * nx


def test_row_rebalancing_changes_no_bit(cgb, O):
    """The persistent kernel re-partitions the rows between its CTAs from measured mat-vec times (from
    64 rows per CTA on: n >= 9472 on 148 SMs) -- a timing-dependent choice.  No reduction depends on
    row ownership, so the run with re-balancing, the run without and the oracle agree bit for bit."""
    n, iters = 9600, 48
    A, b = O.generate_lap2d(n), O.init_source_term(n)
    ref = O.solve(A, b, max_iter=iters, nranks=1, nblk=148)
    with _ctx(cgb, n) as ctx:
        ctx.generate_lap2d()
        ctx.set_rhs(b)
        ctx.set_option("schedule", 1)
        for balance in (1, 0, 1):
            ctx.set_option("balance", balance)
            x = np.zeros(n)
            info, hist = ctx.solve(x, max_iter=iters, tol=1e-10, history=True)
            assert info.k == ref.k == iters
            assert np.array_equal(hist, ref.hist) and np.array_equal(x, ref.x), balance


@pytest.mark.parametrize("rank", [0, 7])
def test_autotune_alone_on_a_ragged_shard(cgb, rank):
    """cgb_autotune times a rank ALONE, the exchange looped back to itself.  With n % world != 0 the last
    rank owns more rows than the others (cg.cc:236-268): a rank with fewer rows must not wait for gather
    entries only the last rank would store (found by profiles/sanitize_small.py: 8 ranks, n = 2311, rank 0
    sat in the wait until the spin time-out).  Both schedules, then a looped-back run of each: same bits."""
    n = 2311
    with cgb.Context(n, rank, 8, 0) as ctx:
        ctx.set_option("spin_timeout_ms", 4000)
        ctx.generate_lap2d()
        ctx.set_rhs(cgb.init_source_term(n))
        for schedule in (1, 0):
            ctx.set_option("schedule", schedule)
            res = ctx.autotune(4)
            assert res["chosen"].startswith("tma_") and len(res["us_per_iteration"]) >= 4, res
        ctx.set_option("loopback", 1)
        hists = []
        for schedule in (0, 1):
            ctx.set_option("schedule", schedule)
            ctx.solve_begin(None, 24, 0.0, True)
            ctx.iterate(24)
            hist = np.zeros(24)
            ctx.solve_end(None, hist)
            hists.append(hist)
        assert np.array_equal(hists[0], hists[1], equal_nan=True)


def test_persistent_schedule_size_limit_and_fallback(cgb, O):
    """The persistent kernel keeps the vector chunks of a CTA in registers: it takes N up to
    2 * 148 * 256 = 75776; one more and cgb_iterate falls back to the graph schedule by itself.  At
    the limit (46 GB of A, 64-bit indexing, two chunks per CTA) both schedules give the same bits,
    and the recursive residual equals the true residual the DEBUG block recomputes."""
    n = 75776
    b = cgb.init_source_term(n)
    out = {}
    with _ctx(cgb, n) as ctx:
        if ctx.layout().sm_count != 148:
            pytest.skip("limit is stated for 148 SMs")
        ctx.generate_lap2d()
        ctx.set_rhs(b)
        for sched in (1, 0):
            ctx.set_option("schedule", sched)
            assert ctx.get_option("schedule_in_use") == sched
            x = np.zeros(n)
            info, hist = ctx.solve(x, max_iter=24, tol=1e-10, history=True)
            nx, rr = ctx.residual_check()
            out[sched] = (x, hist, info.k, nx, rr)
    assert out[1][2] == out[0][2] == 24
    assert np.array_equal(out[1][1], out[0][1]) and np.array_equal(out[1][0], out[0][0])
    assert out[1][3:] == out[0][3:]
    true_resid = out[1][4] * np.linalg.norm(b)
    assert abs(true_resid - np.sqrt(out[1][1][-1])) <= 1e-9 * true_resid
    with _ctx(cgb, n + 1) as ctx:
        ctx.set_option("schedule", 1)
        assert ctx.get_option("schedule_in_use") == 0     # falls back: too many chunks per CTA


# --------------------------------------------------------------------------- reference topologies
@pytest.mark.parametrize("nt,bw", [(32, 1), (64, 16), (1000, 4096), (7, 5), (256, 1024)])
def test_compat_topologies_bitwise_vs_oracle(cgb, O, nt, bw):
    """Option "compat": the reference's column (MatVecT) and row (MatVec) launch topologies with
    NUM_THREADS / BLOCK_WIDTH literal (csrc/compat.cu).  Both give the oracle's chunked order
    bit for bit -- mat-vec, chunk partials and a whole solve -- for any launch shape, where the
    reference's atomicAdd version is run-to-run non-deterministic."""
    n = 1030
    rng = _rng(bw)
    A = O.generate_lap2d(n) + np.diag(rng.standard_normal(n) * 0.01)   # symmetric, non-trivial values
    p = rng.standard_normal(n)
    b = O.init_source_term(n)
    with O.gemv_chunk(bw):
        y_ref = O.gemv(A, p)
        ref = O.solve(A, b, max_iter=60, nranks=1, nblk=148)
    results = []
    for transposed in (1, 0):
        with _ctx(cgb, n) as ctx:
            ctx.set_matrix_rows(A)
            ctx.set_rhs(b)
            ctx.set_option("num_threads", nt)
            ctx.set_option("block_width", bw)
            ctx.set_option("transposed", transposed)
            ctx.set_option("compat", 1)
            y, cp, pap = ctx.gemv(p, want_partials=True)
            assert np.array_equal(y, y_ref), (transposed, nt, bw)
            cp_ref = O.chunk_partials(p, y_ref)
            assert np.array_equal(cp, cp_ref) and pap == O.det_sum(cp_ref)
            x = np.zeros(n)
            info, hist = ctx.solve(x, max_iter=60, tol=1e-10, history=True)
            assert info.k == ref.k and np.array_equal(hist, ref.hist) and np.array_equal(x, ref.x)
            results.append((x, hist))
    assert np.array_equal(results[0][0], results[1][0])     # column == row topology (A symmetric)


def test_compat_option_validation(cgb):
    with _ctx(cgb, 64) as ctx:
        with pytest.raises(cgb.CgbError):
            ctx.set_option("compat", 1)                      # knobs not set
        ctx.set_option("num_threads", 2048)
        ctx.set_option("block_width", 16)
        with pytest.raises(cgb.CgbError):
            ctx.set_option("compat", 1)                      # NUM_THREADS > 1024 cannot launch
        ctx.set_option("num_threads", 128)
        ctx.set_option("compat", 1)
        assert ctx.get_option("compat") == 1
        ctx.set_option("block_width", 4)                     # changing a knob drops compat
        assert ctx.get_option("compat") == 0
