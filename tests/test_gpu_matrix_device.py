"""Matrices from device memory (cgb_set_matrix_csr) and value refreshes of a CSR context's matrix
(cgb_update_matrix_values).  A matrix set from a device CSR must be, bit for bit, the one
cgb_set_matrix_coo builds from the same triples -- the shard, its envelopes, every solve -- and a
context whose values were refreshed must solve exactly like a context built afresh with those values,
without capturing a loop graph again."""
import ctypes

import numpy as np
import pytest

import csr_oracle
from test_gpu_block import _lap2d_inputs, _ragged_coo


def _bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


def _eq(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _key(info):
    return (info.k, bool(info.converged), info.iterations)


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _gpu(torch, a, dtype=None):
    return torch.tensor(np.asarray(a), dtype=dtype or torch.float64, device="cuda:0")


def _coo(m):
    """the CSR's triples, in stored order"""
    return np.repeat(np.arange(m.rows), np.diff(m.rp)).astype(np.int32), m.col.copy(), m.val.copy()


def _torch_csr(torch, m, form, idx):
    dt = torch.int32 if idx == "int32" else torch.int64
    crow, col, val = _gpu(torch, m.rp, dt), _gpu(torch, m.col, dt), _gpu(torch, m.val)
    if form == "sparse":
        return torch.sparse_csr_tensor(crow, col, val, (m.n, m.n))
    return crow, col, val


def _ragged(n=3001):
    irn, jcn, val, empty = _ragged_coo(n, 11)
    return csr_oracle.csr_from_coo(n, irn, jcn, val, False), empty


MATRICES = ["lap2d_17", "lap2d_1000", "lap2d_4099", "ragged_3001"]


def _matrix(O, name):
    """(Csr, b, max_iter)"""
    kind, n = name.split("_")
    n = int(n)
    if kind == "lap2d":
        return csr_oracle.generate_lap2d_csr(n), O.init_source_term(n), n
    m, empty = _ragged(n)
    b = np.random.default_rng(12).standard_normal(n)
    b[empty] = 0.0
    return m, b, 120


def _host(ctx, b, x0, max_iter, tol=1e-10):
    ctx.set_rhs(b)
    x = np.array(x0, dtype=np.float64)
    info, hist = ctx.solve(x, max_iter=max_iter, tol=tol, history=True)
    return info, hist, x


def _device(torch, ctx, b, x0, max_iter, tol=1e-10):
    x = _gpu(torch, x0)
    info, hist = ctx.solve_device(x, _gpu(torch, b), max_iter, tol=tol, history=True).result()
    return info, hist, x.cpu().numpy()


def _like_oracle(d, ref):
    info, hist, x = d
    assert _key(info) == (ref.k, ref.converged, len(ref.hist))
    assert _eq(hist, ref.hist) and _eq(x, ref.x) and _eq([info.rsold, info.rsnew], [ref.rsold, ref.rsnew])


def _same(a, b):
    (ai, ah, ax), (bi, bh, bx) = a, b
    assert _key(ai) == _key(bi) and _eq([ai.rsold, ai.rsnew], [bi.rsold, bi.rsnew])
    assert _eq(ah, bh) and _eq(ax, bx)


# --------------------------------------------------------------------------- set == COO
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
@pytest.mark.parametrize("name", MATRICES)
def test_set_matrix_csr_equals_coo(cgb, O, torch, name, storage):
    m, b, max_iter = _matrix(O, name)
    n = m.n
    x0 = 1e-3 * np.random.default_rng(n).standard_normal(n)
    ref_solve = csr_oracle.solve_csr(m, b, x0, max_iter=max_iter)
    with cgb.Context(n, storage=storage) as ref, cgb.Context(n, storage=storage) as ctx:
        ref.set_matrix_coo(*_coo(m), symmetric=False)
        A_ref = ref.get_matrix_rows(0, n)
        assert _eq(A_ref, m.dense())
        if storage == "csr":
            B, X0 = _lap2d_inputs(O, n, 3)
            block_ref = ref.solve_block(B, X0, max_iter=max_iter, history=True)
        for form in ("sparse", "tuple"):
            for idx in ("int32", "int64"):
                ctx.generate_lap2d()   # a different matrix in between: the set has to replace it
                ctx.set_matrix_csr(_torch_csr(torch, m, form, idx))
                assert _eq(ctx.get_matrix_rows(0, n), A_ref), (form, idx)
                assert ctx.nnz() == ref.nnz() == (m.col.size if storage == "csr" else 0)
                assert ctx.get_option("envelope_doubles") == ref.get_option("envelope_doubles")
                _like_oracle(_host(ctx, b, x0, max_iter), ref_solve)
                _like_oracle(_device(torch, ctx, b, x0, max_iter), ref_solve)
                if storage == "csr":
                    X, infos, hist = ctx.solve_block(B, X0, max_iter=max_iter, history=True)
                    assert _eq(X, block_ref[0]) and [_key(i) for i in infos] == [_key(i) for i in block_ref[1]]
                    assert all(_eq(h, g) for h, g in zip(hist, block_ref[2]))


# --------------------------------------------------------------------------- shard slicing
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
def test_set_matrix_csr_takes_this_ranks_rows(cgb, torch, storage):
    m, _ = _ragged()
    n = m.n
    crow, col, val = _torch_csr(torch, m, "tuple", "int64")
    col32 = col.to(torch.int32)
    for rank in range(2):
        with cgb.Context(n, rank, 2, 0, storage=storage) as ref, \
                cgb.Context(n, rank, 2, 0, storage=storage) as py, \
                cgb.Context(n, rank, 2, 0, storage=storage) as c:
            lay = ref.layout()
            r0, rows = lay.row0, lay.rows
            ref.set_matrix_coo(*_coo(m), symmetric=False)
            py.set_matrix_csr((crow, col, val))
            base, end = int(m.rp[r0]), int(m.rp[r0 + rows])
            assert c._lib.cgb_set_matrix_csr(c._h, crow.data_ptr() + 8 * r0, col32.data_ptr() + 4 * base,
                                             val.data_ptr() + 8 * base, end - base, None) == 0
            want = ref.get_matrix_rows(r0, rows)
            assert _eq(want, m.dense()[r0:r0 + rows])
            for ctx in (py, c):
                assert _eq(ctx.get_matrix_rows(r0, rows), want)
                assert ctx.nnz() == ref.nnz()
                assert ctx.get_option("envelope_doubles") == ref.get_option("envelope_doubles")


# --------------------------------------------------------------------------- refusals of set
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
def test_set_matrix_csr_refusals(cgb, O, torch, storage):
    n = 1000
    old = csr_oracle.generate_lap2d_csr(n)
    b = O.init_source_term(n)
    ref = csr_oracle.solve_csr(old, b, None, max_iter=n)
    new = csr_oracle.Csr(n, old.rp, old.col, 1.5 * old.val)   # what a wrongly accepted set would leave
    rp, col, val = _gpu(torch, new.rp, torch.int64), _gpu(torch, new.col, torch.int32), _gpu(torch, new.val)
    nnz = new.col.size
    host = np.zeros(4 * nnz)
    pinned = torch.zeros(4 * nnz, dtype=torch.float64).pin_memory()

    def row_start(i):
        return int(new.rp[i])

    def with_rp(i, v):
        t = rp.clone()
        t[i] = v
        return t

    def with_col(k, v):
        t = col.clone()
        t[k] = v
        return t

    swapped = col.clone()
    swapped[row_start(401)], swapped[row_start(401) + 1] = col[row_start(401) + 1], col[row_start(401)]
    # (rp, col, nnz, the local row the message has to name)
    bad = [
        (with_rp(500, row_start(499) - 1), col, nnz, 499),               # rp decreases
        (rp, col, nnz + 1, n - 1),                                       # rp[rows] - rp[0] < nnz
        (rp, col, nnz - 1, n - 1),                                       # ... > nnz
        (rp - 5, col, nnz, 0),                                           # rp[0] < 0
        (rp, with_col(row_start(322) - 1, n), nnz, 321),                 # column = n (last entry of row 321)
        (rp, with_col(row_start(322), -1), nnz, 322),                    # column = -1
        (rp, with_col(row_start(400) + 1, int(new.col[row_start(400)])), nnz, 400),   # a duplicate
        (rp, swapped, nnz, 401),                                         # a descending pair
    ]
    with cgb.Context(n, storage=storage) as ctx:
        ctx.generate_lap2d()
        lib = ctx._lib

        def cset(r=rp.data_ptr(), c=col.data_ptr(), v=val.data_ptr(), z=nnz):
            return lib.cgb_set_matrix_csr(ctx._h, r, c, v, z, None)

        for r, c, z, row in bad:
            assert cset(r.data_ptr(), c.data_ptr(), z=z) == 1, row
            assert f"local row {row}:" in lib.cgb_last_error().decode(), (row, lib.cgb_last_error())
        hp = host.ctypes.data
        for args in ({"r": None}, {"c": None}, {"v": None}, {"r": hp}, {"c": hp}, {"v": hp},
                     {"r": pinned.data_ptr()}, {"v": pinned.data_ptr()}, {"z": -1}):
            assert cset(**args) == 1, args
        assert cset(v=pinned.data_ptr()) == 1 and b"host" in lib.cgb_last_error()
        with pytest.raises(TypeError):
            ctx.set_matrix_csr((rp.cpu(), col.cpu(), val.cpu()))
        with pytest.raises(TypeError):
            ctx.set_matrix_csr((rp, col, val))   # crow int64, col int32
        with pytest.raises(TypeError):
            ctx.set_matrix_csr((rp, col.to(torch.int64), val.float()))
        # nothing of the refused calls reached the context: the previous matrix, bit for bit
        assert _eq(ctx.get_matrix_rows(0, n), old.dense())
        _like_oracle(_host(ctx, b, np.zeros(n), n), ref)
        _like_oracle(_device(torch, ctx, b, np.zeros(n), n), ref)
        # one matrix build at a time with a solve
        ctx.set_rhs(b)
        ctx.solve_begin(np.zeros(n), 10)
        assert cset() == 2
        ctx.solve_end()
        if storage == "csr":
            ctx.solve_block_begin(np.array([b, b]), max_iter=10)
            assert cset() == 2
            ctx.iterate(10)
            ctx.solve_block_end()
        assert cset() == 0
        assert _eq(ctx.get_matrix_rows(0, n), new.dense())


# --------------------------------------------------------------------------- updates
def _values(m, t):
    """value set t on the pattern of lap2d m: diagonal 4 + sigma_t, odd t a seeded symmetric perturbation of
    the off-diagonals"""
    rows = np.repeat(np.arange(m.rows), np.diff(m.rp))
    v = m.val.copy()
    diag = rows == m.col
    v[diag] = 4.0 + [0.0, 0.5, 2.0, 1e-3, 7.25][t]
    if t % 2:
        lo, hi = np.minimum(rows, m.col), np.maximum(rows, m.col)
        v[~diag] += 0.05 * np.sin(1.3 * lo[~diag] + 0.7 * hi[~diag] + t)
    return csr_oracle.Csr(m.n, m.rp, m.col, np.ascontiguousarray(v))


def _fresh(cgb, torch, mt, b, x0, B, X0, max_iter):
    """host, device and block device solves of a context built afresh by set_matrix_coo"""
    with cgb.Context(mt.n, storage="csr") as f:
        f.set_matrix_coo(*_coo(mt), symmetric=False)
        h = _host(f, b, x0, max_iter)
        d = _device(torch, f, b, x0, max_iter)
        X = _gpu(torch, X0)
        infos, hist = f.solve_block_device(X, _gpu(torch, B), max_iter, history=True).result()
    return h, d, (X.cpu().numpy(), infos, hist)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_updates_equal_fresh_builds_without_recapture(cgb, O, torch):
    n = 4099
    m = csr_oracle.generate_lap2d_csr(n)
    b = O.init_source_term(n)
    x0 = 1e-3 * np.random.default_rng(1).standard_normal(n)
    B, X0 = _lap2d_inputs(O, n, 3)
    with cgb.Context(n, storage="csr") as c:
        c.generate_lap2d()
        # warm-up: the first host and block solves allocate their history and block buffers, which moves
        # what the graphs bake in; the second pass captures every loop graph for good
        for _ in range(2):
            _host(c, b, x0, n)
            c.solve_block_device(_gpu(torch, X0), _gpu(torch, B), n, history=True).result()
            _device(torch, c, b, x0, n)
        captures = c.get_option("graph_captures")
        assert captures >= 3
        x_prev = None
        for t in range(5):
            mt = _values(m, t)
            c.update_matrix_values(_gpu(torch, mt.val))
            if x_prev is not None:   # b and x of the last solve, the mat-vec on the new values
                assert _eq(c.residual_check(), csr_oracle.residual_check_csr(mt, b, x_prev))
            replays = c.get_option("graph_replays")
            d = _device(torch, c, b, x0, n)
            assert c.get_option("graph_replays") == replays + 1
            h = _host(c, b, x0, n)
            X = _gpu(torch, X0)
            replays = c.get_option("graph_replays")
            infos, hist = c.solve_block_device(X, _gpu(torch, B), n, history=True).result()
            assert c.get_option("graph_replays") == replays + 1
            assert c.get_option("graph_captures") == captures, t
            fh, fd, (fX, finfos, fhist) = _fresh(cgb, torch, mt, b, x0, B, X0, n)
            _same(d, fd)
            _same(h, fh)
            _like_oracle(d, csr_oracle.solve_csr(mt, b, x0, max_iter=n))
            assert _eq(X.cpu().numpy(), fX) and [_key(i) for i in infos] == [_key(i) for i in finfos]
            assert all(_eq(p, q) for p, q in zip(hist, fhist))
            assert _eq(c.residual_check(), csr_oracle.residual_check_csr(mt, b, h[2]))   # the host solve's x
            x_prev = h[2]
        # a set reallocates the arrays the graphs bake in: the next device solve captures anew
        c.set_matrix_csr(_torch_csr(torch, m, "tuple", "int64"))
        _like_oracle(_device(torch, c, b, x0, n), csr_oracle.solve_csr(m, b, x0, max_iter=n))
        assert c.get_option("graph_captures") == captures + 1


# --------------------------------------------------------------------------- stream order
@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_updates_are_ordered_on_the_stream_and_asynchronous(cgb, O, torch):
    n = 4099
    m = csr_oracle.generate_lap2d_csr(n)
    b_host = O.init_source_term(n)
    diag = torch.tensor(np.repeat(np.arange(n), np.diff(m.rp)) == m.col, device="cuda:0")
    with cgb.Context(n, storage="csr") as c:
        c.generate_lap2d()
        base = _gpu(torch, m.val)
        b = _gpu(torch, b_host)
        x = torch.zeros(n, dtype=torch.float64, device="cuda:0")
        c.update_matrix_values(base.clone())
        c.solve_device(x, b, n, history=True).result()                  # warm-up: graphs, buffers, events
        s = torch.cuda.current_stream()
        x1 = torch.zeros(n, dtype=torch.float64, device="cuda:0")
        x2 = torch.zeros(n, dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        torch.cuda._sleep(100_000_000)                                  # ~50 ms of GPU clock cycles
        v1 = torch.where(diag, base + 0.5, base)                        # values made by torch kernels, no sync
        c.update_matrix_values(v1)
        h1 = c.solve_device(x1, b, n, history=True)
        v2 = torch.where(diag, base + 2.0, base * 1.25)
        c.update_matrix_values(v2)
        h2 = c.solve_device(x2, b, n, history=True)
        ev = torch.cuda.Event()
        ev.record(s)
        assert not ev.query(), "a call waited for the stream"
        got = [(*h.result(), xx.cpu().numpy()) for h, xx in ((h1, x1), (h2, x2))]
        vals = [v1.cpu().numpy(), v2.cpu().numpy()]
    for d, v in zip(got, vals):
        mt = csr_oracle.Csr(n, m.rp, m.col, v)
        _like_oracle(d, csr_oracle.solve_csr(mt, b_host, None, max_iter=n))
        with cgb.Context(n, storage="csr") as f:
            f.set_matrix_coo(*_coo(mt), symmetric=False)
            _same(d, _device(torch, f, b_host, np.zeros(n), n))


# --------------------------------------------------------------------------- refusals of update
@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_update_matrix_values_refusals(cgb, O, torch):
    n = 1000
    m = csr_oracle.generate_lap2d_csr(n)
    b = O.init_source_term(n)
    val = _gpu(torch, 2.0 * m.val)
    host = np.zeros(2 * m.col.size)
    pinned = torch.zeros(m.col.size, dtype=torch.float64).pin_memory()

    def upd(ctx, p=val.data_ptr()):
        return ctx._lib.cgb_update_matrix_values(ctx._h, p, None)

    with cgb.Context(n) as d:
        d.generate_lap2d()
        assert upd(d) == 2 and b"pattern" in d._lib.cgb_last_error()
        with pytest.raises(cgb.CgbError) as ei:
            d.update_matrix_values(val)
        assert ei.value.code == 2
    with cgb.Context(n, storage="csr") as c:
        assert upd(c) == 2 and b"matrix" in c._lib.cgb_last_error()
        c.generate_lap2d()
        c.set_rhs(b)
        c.solve_begin(np.zeros(n), 10)
        assert upd(c) == 2
        c.solve_end()
        c.solve_block_begin(np.array([b, b]), max_iter=10)
        assert upd(c) == 2
        c.iterate(10)
        c.solve_block_end()
        for p in (None, host.ctypes.data, pinned.data_ptr()):
            assert upd(c, p) == 1, p
        with pytest.raises(ValueError):
            c.update_matrix_values(val[:-1])
        with pytest.raises(TypeError):
            c.update_matrix_values(val.cpu())
        with pytest.raises(TypeError):
            c.update_matrix_values(val.float())
        torch.cuda.synchronize()
        assert _eq(c.get_matrix_rows(0, n), m.dense())   # no refused call copied anything
        assert upd(c) == 0
        torch.cuda.synchronize()
        assert _eq(c.get_matrix_rows(0, n), 2.0 * m.dense())


# --------------------------------------------------------------------------- without a GPU
def test_matrix_from_device_without_gpu_fails_loudly(cgb):
    try:
        if cgb.device_count() > 0:
            pytest.skip("a GPU is present")
    except cgb.CgbError:
        pass
    lib = cgb.load()
    buf = np.zeros(64)
    p = buf.ctypes.data
    assert lib.cgb_set_matrix_csr(None, p, p, p, 4, None) == 3
    assert lib.cgb_update_matrix_values(None, p, None) == 3
    assert np.all(buf == 0.0)
