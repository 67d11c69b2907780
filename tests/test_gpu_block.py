"""Block solves (cgb_solve_block*): several right-hand sides against one CSR matrix.  Column j of a
block solve must equal, bit for bit, both the CSR oracle's solve of A x = b_j from x0_j and a single
cgb_solve of that column on the same context: k, converged, rsold, rsnew, iterations, the r'r
history and x.  A NaN (the b = 0, x0 = 0 column, whose alpha is 0 / 0) is compared as "NaN at the
same places" against the oracle only, whose NaN payload is the host's; against the GPU's own
single solve every bit is compared."""
import ctypes

import numpy as np
import pytest

import csr_oracle


def _bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


def _eq(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _eq_nan(a, b):
    """bitwise, except that a NaN only has to meet a NaN"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(_bits(a[~na]), _bits(b[~nb]))


def _info_tuple(info):
    return (info.k, bool(info.converged), info.iterations)


def _check_block(ctx, m, B, X0, max_iter, tol=1e-10):
    """block solve == CSR oracle == single solve on the same context, column by column"""
    X, infos, hist = ctx.solve_block(B, X0, max_iter=max_iter, tol=tol, history=True)
    for j in range(B.shape[0]):
        x0 = np.zeros(ctx.n) if X0 is None else X0[j]
        ref = csr_oracle.solve_csr(m, B[j], x0, max_iter=max_iter, tol=tol)
        assert _info_tuple(infos[j]) == (ref.k, ref.converged, len(ref.hist)), j
        assert _eq_nan(hist[j], ref.hist) and _eq_nan(X[j], ref.x), j
        assert _eq_nan([infos[j].rsold, infos[j].rsnew], [ref.rsold, ref.rsnew]), j
        ctx.set_rhs(B[j])
        x = x0.copy()
        info, h = ctx.solve(x, max_iter=max_iter, tol=tol, history=True)
        assert _info_tuple(infos[j]) == _info_tuple(info), j
        assert _eq(hist[j], h) and _eq(X[j], x) and _eq([infos[j].rsold, infos[j].rsnew], [info.rsold, info.rsnew]), j
    assert len({i.seconds for i in infos}) == 1
    return X, infos, hist


def _csr_ctx(cgb, m, irn=None, jcn=None, val=None):
    ctx = cgb.Context(m.n, storage="csr")
    if irn is None:
        ctx.generate_lap2d()
    else:
        ctx.set_matrix_coo(irn, jcn, val, symmetric=False)
    return ctx


def _lap2d_inputs(O, n, nrhs):
    """distinct b_j (source terms with different h, seeded random vectors, scaled copies) and x0_j"""
    rng = np.random.default_rng(n)
    bs = [O.init_source_term(n), 1e-9 * O.init_source_term(n), rng.standard_normal(n), O.init_source_term(n, 0.37 / n),
          2.5 * O.init_source_term(n), 1e3 * rng.standard_normal(n), O.init_source_term(n, 0.11 / n),
          -0.5 * rng.standard_normal(n)]
    B = np.array(bs[:nrhs])
    X0 = np.array([1e-3 * (j + 1) * rng.standard_normal(n) for j in range(nrhs)])
    if nrhs > 1:
        X0[1] *= 1e-9   # the small column starts small too, and converges first
    return B, X0


# --------------------------------------------------------------------------- generated matrices
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("nrhs", [1, 2, 3, 8])
@pytest.mark.parametrize("n", [17, 1000, 4096, 4099])
def test_block_lap2d_columns_are_single_solves(cgb, O, n, nrhs):
    m = csr_oracle.generate_lap2d_csr(n)
    B, X0 = _lap2d_inputs(O, n, nrhs)
    with _csr_ctx(cgb, m) as ctx:
        _, infos, _ = _check_block(ctx, m, B, X0, max_iter=n)
    if nrhs > 1:   # one column's alpha / beta used for all of them could not pass
        assert len({i.k for i in infos}) > 1, [i.k for i in infos]


# --------------------------------------------------------------------------- ragged CSR
def _ragged_coo(n, seed):
    """symmetric, diagonally dominant: short rows, rows of 9 .. ~45 entries (the warp path), empty rows
    (and columns), colliding buckets, explicit zeros.  Returns COO triples and the empty rows."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 4, n)
    lens[rng.choice(n, n // 20, replace=False)] = rng.integers(9, 41, n // 20)
    A = np.zeros((n, n))
    for i in range(n):
        c = rng.choice(n, lens[i], replace=False)
        A[i, c] = 0.1 * rng.standard_normal(c.size)
    A = A + A.T
    empty = rng.choice(n, 12, replace=False)
    A[empty, :] = 0.0
    A[:, empty] = 0.0
    d = 1.0 + np.abs(A).sum(axis=1)
    d[empty] = 0.0
    A[np.arange(n), np.arange(n)] = d
    keep = np.zeros((n, n), dtype=bool)   # stored zeros
    zi, zj = rng.integers(0, n, 300), rng.integers(0, n, 300)
    ok = ~np.isin(zi, empty) & ~np.isin(zj, empty)
    keep[zi[ok], zj[ok]] = keep[zj[ok], zi[ok]] = True
    irn, jcn = np.nonzero((A != 0) | keep)
    return irn.astype(np.int32), jcn.astype(np.int32), np.ascontiguousarray(A[irn, jcn]), empty


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("nrhs", [3, 8])
def test_block_ragged_csr_with_long_and_empty_rows(cgb, nrhs):
    n = 3001
    irn, jcn, val, empty = _ragged_coo(n, 11)
    m = csr_oracle.csr_from_coo(n, irn, jcn, val, False)
    lens = np.diff(m.rp)
    assert (lens > 8).sum() > 100 and (lens == 0).sum() == 12 and (m.val == 0).sum() > 100
    rng = np.random.default_rng(12)
    B = rng.standard_normal((nrhs, n)) * np.logspace(0, 4, nrhs)[:, None]
    B[:, empty] = 0.0
    X0 = 1e-2 * rng.standard_normal((nrhs, n))
    with _csr_ctx(cgb, m, irn, jcn, val) as ctx:
        assert ctx.nnz() == m.col.size
        _check_block(ctx, m, B, X0, max_iter=120)


# --------------------------------------------------------------------------- columns that stop apart
def _stop_apart(O):
    """lap2d at N = 1000 with its last 8 rows and columns emptied, and five columns:
    0 converges at k = 2, 1 runs to max_iter (250), 2 has p'Ap = 0 < rsold * NEARZERO in every
    iteration (b lives on the empty rows), 3 is b = 0 from x0 = 0 (alpha = 0 / 0), 4 converges at 172"""
    n, cut = 1000, 992
    A = csr_oracle.generate_lap2d_csr(n).dense()
    A[cut:, :] = 0.0
    A[:, cut:] = 0.0
    irn, jcn = np.nonzero(A)
    val = np.ascontiguousarray(A[irn, jcn])
    irn, jcn = irn.astype(np.int32), jcn.astype(np.int32)
    src = O.init_source_term(n)
    src[cut:] = 0.0
    quick = np.zeros(n)
    quick[:cut] = 1e-11 * np.random.default_rng(5).standard_normal(cut)
    clamp = np.zeros(n)
    clamp[cut:] = 1.0
    B = np.array([quick, 1e12 * src, clamp, np.zeros(n), src])
    return n, (irn, jcn, val), csr_oracle.csr_from_coo(n, irn, jcn, val, False), B, 250


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_block_columns_stop_at_different_times(cgb, O):
    n, coo, m, B, max_iter = _stop_apart(O)
    with _csr_ctx(cgb, m, *coo) as ctx:
        X, infos, hist = _check_block(ctx, m, B, None, max_iter)
    assert [(i.k, bool(i.converged)) for i in infos] == [(2, True), (max_iter, False), (max_iter, False),
                                                         (max_iter, False), (172, True)]
    assert np.abs(X[2]).max() > 1e13                     # alpha = rsold / (rsold * NEARZERO) every time
    assert np.isnan(X[3]).all() and not np.isnan(X[[0, 1, 2, 4]]).any()
    # the column that stopped at k = 2 is the 3-iteration solve, though the block ran 250
    ref = csr_oracle.solve_csr(m, B[0], None, max_iter=3)
    assert _eq(X[0], ref.x) and _eq(hist[0], ref.hist)


# --------------------------------------------------------------------------- split iteration
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("opts", [{}, {"poll_every": 5, "graph_unroll": 3}, {"poll_every": 1, "graph_unroll": 1},
                                  {"graph": 0}, {"pdl": 0, "graph_unroll": 7}])
def test_block_split_iteration_equals_one_shot(cgb, O, opts):
    n, coo, m, B, max_iter = _stop_apart(O)   # from x0 = 0: columns stop at k = 2 and 172, inside a graph
    X0 = 1e-3 * np.random.default_rng(9).standard_normal(B.shape)
    with _csr_ctx(cgb, m, *coo) as ctx:
        for k, v in opts.items():
            ctx.set_option(k, v)
        X, infos, hist = ctx.solve_block(B, None, max_iter=max_iter, history=True)
        launches = ctx.launch_count()
        ctx.solve_block_begin(B, None, max_iter=max_iter, history=True)
        ctx.iterate(7)
        ctx.iterate(max_iter)
        X2, infos2, hist2 = ctx.solve_block_end()
        assert ctx.launch_count() > launches
        ctx.solve_block_begin(B, X0, max_iter=0, history=True)
        assert ctx.iterate(5) >= 0.0
        X3, infos3, hist3 = ctx.solve_block_end()
    assert [_info_tuple(i) for i in infos] == [_info_tuple(i) for i in infos2]
    assert _eq(X, X2) and all(_eq(a, b) for a, b in zip(hist, hist2))
    assert _eq([(i.rsold, i.rsnew) for i in infos], [(i.rsold, i.rsnew) for i in infos2])
    # max_iter = 0: nothing runs, x = x0, k = 0, rsold = rsnew = r'r of x0 (the oracle's)
    assert _eq(X3, X0) and all(len(h) == 0 for h in hist3)
    for j in range(B.shape[0]):
        ref = csr_oracle.solve_csr(m, B[j], X0[j], max_iter=0)
        assert _info_tuple(infos3[j]) == (0, False, 0) and _eq_nan([infos3[j].rsold], [ref.rsold])


# --------------------------------------------------------------------------- size
@pytest.mark.gpu
@pytest.mark.timeout(1800)
def test_block_two_million_four_columns(cgb, O):
    """Past L2: the CSR arrays and four columns of x, r, p, b, Ap stream from HBM."""
    n, nrhs, max_iter = 2_000_000, 4, 40
    m = csr_oracle.generate_lap2d_csr(n)
    B, X0 = _lap2d_inputs(O, n, nrhs)
    with _csr_ctx(cgb, m) as ctx:
        _check_block(ctx, m, B, X0, max_iter)


# --------------------------------------------------------------------------- refusals and isolation
@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_block_refusals(cgb, O):
    n = 1000
    B = np.array([O.init_source_term(n)] * 2)
    with cgb.Context(n) as d:
        d.generate_lap2d()
        with pytest.raises(cgb.CgbError) as ei:
            d.solve_block(B, max_iter=10)
        assert ei.value.code == 2 and "CSR" in str(ei.value)
    with cgb.Context(n, 0, 2, 0, storage="csr") as w:
        w.generate_lap2d()
        with pytest.raises(cgb.CgbError) as ei:
            w.solve_block(B, max_iter=10)
        assert ei.value.code == 2 and "rank" in str(ei.value)
    with cgb.Context(n, storage="csr") as c:
        with pytest.raises(cgb.CgbError) as ei:
            c.solve_block(B, max_iter=10)
        assert ei.value.code == 2 and "matrix" in str(ei.value)
        c.generate_lap2d()
        for bad in (np.zeros((0, n)), np.zeros((9, n))):
            with pytest.raises(cgb.CgbError) as ei:
                c.solve_block(bad, max_iter=10)
            assert ei.value.code == 1
        lib, x = c._lib, np.zeros(2 * n)
        dp = ctypes.POINTER(ctypes.c_double)
        assert lib.cgb_solve_block(c._h, 2, None, x.ctypes.data_as(dp), 10, 1e-10, None, None) == 1
        assert lib.cgb_solve_block(c._h, 2, B.ctypes.data_as(dp), None, 10, 1e-10, None, None) == 1
        assert lib.cgb_solve_block_begin(c._h, 2, None, None, 10, 1e-10, 0) == 1
        # one solve at a time, either way round
        c.set_rhs(B[0])
        c.solve_begin(np.zeros(n), 10)
        with pytest.raises(cgb.CgbError) as ei:
            c.solve_block_begin(B, max_iter=10)
        assert ei.value.code == 2
        c.solve_end()
        c.solve_block_begin(B, max_iter=10)
        for call in (lambda: c.solve_begin(np.zeros(n), 10), lambda: c.solve_end(), lambda: c.residual_check(),
                     lambda: c.solve_block_begin(B, max_iter=10)):
            with pytest.raises(cgb.CgbError) as ei:
                call()
            assert ei.value.code == 2
        c.iterate(10)
        c.solve_block_end()
        with pytest.raises(cgb.CgbError) as ei:
            c.solve_block_end()
        assert ei.value.code == 2


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_block_leaves_the_single_solve_alone(cgb, O):
    n = 4096
    m = csr_oracle.generate_lap2d_csr(n)
    b = O.init_source_term(n)
    B, X0 = _lap2d_inputs(O, n, 3)
    ref = csr_oracle.solve_csr(m, b, None, max_iter=n)
    nx_ref, rr_ref = csr_oracle.residual_check_csr(m, b, ref.x)

    def single(ctx):
        x = np.zeros(n)
        info, hist = ctx.solve(x, max_iter=n, history=True)
        assert (info.k, bool(info.converged)) == (ref.k, ref.converged)
        assert _eq(x, ref.x) and _eq(hist, ref.hist) and _eq([info.rsold, info.rsnew], [ref.rsold, ref.rsnew])

    with _csr_ctx(cgb, m) as ctx:
        ctx.set_rhs(b)
        single(ctx)
        assert _eq(ctx.residual_check(), [nx_ref, rr_ref])
        replays = ctx.get_option("graph_replays")
        X, infos, _ = ctx.solve_block(B, X0, max_iter=n, history=True)   # no set_rhs in between
        assert ctx.get_option("graph_replays") > replays
        assert _eq(ctx.residual_check(), [nx_ref, rr_ref])          # x, b of the single solve untouched
        single(ctx)
        ctx.solve_block(B[:1], X0[:1], max_iter=n)                  # fewer columns: the same buffers
        X8, infos8, _ = ctx.solve_block(np.vstack([B] * 3)[:8], np.vstack([X0] * 3)[:8], max_iter=n)  # grown
        single(ctx)
        assert _eq(ctx.residual_check(), [nx_ref, rr_ref])
    assert _eq(X8[:3], X) and _eq(X8[3:6], X) and [i.k for i in infos8[:3]] == [i.k for i in infos]


# --------------------------------------------------------------------------- without a GPU
def _no_gpu(cgb):
    try:
        return cgb.device_count() == 0
    except cgb.CgbError:
        return True


def test_block_solve_without_gpu_fails_loudly(cgb):
    if not _no_gpu(cgb):
        pytest.skip("a GPU is present")
    lib = cgb.load()
    n = 64
    b, x = np.ones(2 * n), np.zeros(2 * n)
    dp = ctypes.POINTER(ctypes.c_double)
    assert lib.cgb_solve_block(None, 2, b.ctypes.data_as(dp), x.ctypes.data_as(dp), 10, 1e-10, None, None) == 3
    assert lib.cgb_solve_block_begin(None, 2, b.ctypes.data_as(dp), None, 10, 1e-10, 0) == 3
    assert lib.cgb_solve_block_end(None, None, None, None) == 3
    assert np.all(x == 0.0)
