"""Sum-assembly of device COO contributions (cgb_assemble_coo) and re-assembly of new values for the same
triples (cgb_assemble_values).  The reference is a sequential loop: the writes stable-sorted by (row, column),
then added in write order from the first write -- no numpy reduction, which would sum pairwise.  Every stored
cell, every solve and every re-assembly is checked bit for bit against it."""
import numpy as np
import pytest

import csr_oracle
from test_gpu_envelope import envelope_doubles


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


# --------------------------------------------------------------------------- the reference
def _seq(ws):
    v = ws[0]
    for w in ws[1:]:
        v = v + w
    return v


def _reversed(ws):
    return _seq(ws[::-1])


def _pairwise(ws):
    if len(ws) == 1:
        return ws[0]
    h = len(ws) // 2
    return _pairwise(ws[:h]) + _pairwise(ws[h:])


def _from_zero(ws):
    return _seq([0.0] + list(ws))


def assemble(n, irn, jcn, val, symmetric, row0=0, rows=None, fold=_seq):
    """Csr of rows [row0, row0 + rows): triple z writes (i, j) and, symmetric and i != j, (j, i) right after it;
    every cell that receives a write is stored, its value fold(writes in write order)."""
    rows = n - row0 if rows is None else rows
    irn, jcn = np.asarray(irn, dtype=np.int64), np.asarray(jcn, dtype=np.int64)
    val = np.asarray(val, dtype=np.float64)
    if symmetric:
        off = irn != jcn
        r = np.stack([irn, np.where(off, jcn, -1)], axis=1).ravel()
        c = np.stack([jcn, irn], axis=1).ravel()
        v = np.repeat(val, 2)
    else:
        r, c, v = irn, jcn, val
    sel = (r >= row0) & (r < row0 + rows)
    key = (r[sel] - row0) * n + c[sel]
    order = np.argsort(key, kind="stable")
    keys, runs = [], []
    for k, w in zip(key[order].tolist(), v[sel][order].tolist()):
        if keys and keys[-1] == k:
            runs[-1].append(w)
        else:
            keys.append(k)
            runs.append([w])
    keys = np.array(keys, dtype=np.int64)
    rp = np.searchsorted(keys, np.arange(rows + 1) * n).astype(np.int64)
    return csr_oracle.Csr(n, rp, (keys % n).astype(np.int32), np.array([fold(ws) for ws in runs], dtype=np.float64))


# --------------------------------------------------------------------------- inputs
def quad_coo(m, seed=0, reaction=0.01):
    """A variable-coefficient 2-D Laplacian on an m x m grid of bilinear quads, (m + 1)^2 nodes: every element
    adds its 16 entries k_e K + reaction I (K the bilinear stiffness matrix), elements in a seeded order."""
    rng = np.random.default_rng(seed)
    K = np.array([[4, -1, -2, -1], [-1, 4, -1, -2], [-2, -1, 4, -1], [-1, -2, -1, 4]], dtype=np.float64) / 6.0
    K += reaction * np.eye(4)
    ex, ey = np.meshgrid(np.arange(m), np.arange(m), indexing="ij")
    ex, ey = ex.ravel(), ey.ravel()
    perm = rng.permutation(ex.size)
    ex, ey = ex[perm], ey[perm]
    nodes = np.stack([ey * (m + 1) + ex, ey * (m + 1) + ex + 1, (ey + 1) * (m + 1) + ex + 1, (ey + 1) * (m + 1) + ex],
                     axis=1)
    k = 1.0 + 0.9 * np.sin(0.37 * ex + 0.61 * ey) + 0.05 * rng.random(ex.size)
    irn = np.repeat(nodes, 4, axis=1).ravel()
    jcn = np.tile(nodes, (1, 4)).ravel()
    val = (k[:, None, None] * K[None]).reshape(-1)
    return (m + 1) ** 2, irn.astype(np.int32), jcn.astype(np.int32), np.ascontiguousarray(val)


def random_coo(n, nz, seed, width=12, empty=40):
    """heavy duplication: every row draws its columns from `width` candidates; `empty` rows receive nothing"""
    rng = np.random.default_rng(seed)
    live = np.setdiff1d(np.arange(n), rng.choice(n, empty, replace=False))
    irn = rng.choice(live, nz)
    jcn = (irn * 7 + rng.integers(0, width, nz) * 131) % n
    val = rng.standard_normal(nz) * 10.0 ** rng.integers(-3, 4, nz)
    return n, irn.astype(np.int32), jcn.astype(np.int32), val


def long_run_coo(n=500, dups=100_000, seed=3):
    """one cell with 10^5 writes among some scattered triples"""
    rng = np.random.default_rng(seed)
    _, irn, jcn, val = random_coo(n, 2000, seed, empty=5)
    pos = np.sort(rng.choice(2000 + dups, 2000, replace=False))
    I = np.full(2000 + dups, 7, dtype=np.int32)
    J = np.full(2000 + dups, 11, dtype=np.int32)
    V = rng.standard_normal(2000 + dups) * 1e3 + 0.1
    I[pos], J[pos], V[pos] = irn, jcn, val
    return n, I, J, V


def symmetric_coo(n=2000, seed=5):
    """symmetric contributions, diagonal triples among them (which must not be doubled)"""
    n, irn, jcn, val = random_coo(n, 30_000, seed, empty=20)
    rng = np.random.default_rng(seed + 1)
    d = rng.choice(np.unique(irn), 3000)
    irn, jcn = np.concatenate([irn, d]), np.concatenate([jcn, d])
    val = np.concatenate([val, 50.0 + rng.random(d.size)])
    p = rng.permutation(irn.size)
    return n, irn[p].astype(np.int32), jcn[p].astype(np.int32), np.ascontiguousarray(val[p])


# cells whose value depends on the fold order, and the signed zeros
ORDER_CELLS = [
    [1.0, 1e16, -1e16],          # 1 + 1e16 rounds to 1e16: the sum is 0 in write order, 1 reversed or pairwise
    [1e16, -1e16, 1.0],          # 1 in write order, 0 reversed or pairwise
    [-1e16, 1e16, 3.0],
    [2.0, 2.0 ** 54, -2.0 ** 54],
    [1e16, 1.0, -1e16],          # 0 in every order
    [-0.0],                      # a lone -0 stays -0 (+0 + -0 = +0 when the fold starts from +0)
    [-0.0, -0.0],
    [-0.0, -0.0, -0.0],
    [1.5, -1.5],                 # cancels to +0: stored all the same
    [0.0],
    [-0.0, 0.0],
    [3.25],
]
ORDER_WRONG = {"reversed": 4, "pairwise": 4, "from_zero": 3}   # cells each wrong fold changes


def order_coo(n=64, seed=9):
    """ORDER_CELLS at scattered cells, their writes interleaved with each other's"""
    rng = np.random.default_rng(seed)
    cells = rng.choice(n * n, len(ORDER_CELLS), replace=False)
    slots = [(c, w) for c, ws in zip(cells, ORDER_CELLS) for w in ws]
    owner = np.concatenate([np.full(len(ws), i) for i, ws in enumerate(ORDER_CELLS)])
    # a random interleaving that keeps every cell's own writes in order
    seq = rng.permutation(owner)
    nxt = [0] * len(ORDER_CELLS)
    irn, jcn, val = [], [], []
    for i in seq:
        irn.append(cells[i] // n)
        jcn.append(cells[i] % n)
        val.append(ORDER_CELLS[i][nxt[i]])
        nxt[i] += 1
    assert len(val) == len(slots)
    return n, np.array(irn, dtype=np.int32), np.array(jcn, dtype=np.int32), np.array(val, dtype=np.float64)


INPUTS = {
    "quad": lambda: (*quad_coo(30), False),
    "random": lambda: (*random_coo(3001, 200_000, 1), False),
    "long_run": lambda: (*long_run_coo(), False),
    "symmetric": lambda: (*symmetric_coo(), True),
    "order": lambda: (*order_coo(), False),
}


# --------------------------------------------------------------------------- the inputs can see a wrong order
def test_wrong_fold_orders_change_the_order_input():
    """A kernel that folds in reverse, pairwise or from +0 changes a known number of cells of the order
    input, so it cannot pass the bitwise checks below."""
    n, irn, jcn, val = order_coo()
    ref = assemble(n, irn, jcn, val, False)
    assert ref.col.size == len(ORDER_CELLS)
    got = {}
    for name, fold in (("reversed", _reversed), ("pairwise", _pairwise), ("from_zero", _from_zero)):
        m = assemble(n, irn, jcn, val, False, fold=fold)
        assert np.array_equal(m.rp, ref.rp) and np.array_equal(m.col, ref.col)
        got[name] = int(np.count_nonzero(_bits(m.val) != _bits(ref.val)))
    assert got == ORDER_WRONG
    # every cell got its own writes back in order; the signed zeros of the contract
    cells = {}
    for i, j, w in zip(irn.tolist(), jcn.tolist(), val.tolist()):
        cells.setdefault((i, j), []).append(w)
    assert sorted(map(str, cells.values())) == sorted(map(str, ORDER_CELLS))
    d = ref.dense()
    for (i, j), ws in cells.items():
        assert _eq(d[i, j], _seq(ws)), ws
        assert np.signbit(d[i, j]) == (str(ws) in ("[-0.0]", "[-0.0, -0.0]", "[-0.0, -0.0, -0.0]")), ws


def test_the_reference_does_not_mirror_the_diagonal():
    m = assemble(3, [0, 1, 2], [0, 2, 2], [1.0, 2.0, 4.0], True)
    assert _eq(m.dense(), [[1.0, 0, 0], [0, 0, 2.0], [0, 2.0, 4.0]])
    # a symmetric pair written as two triples is the sum of both, in write order
    m = assemble(2, [0, 1, 0], [1, 0, 0], [1e16, 1.0, 3.0], True)
    assert _eq(m.dense(), [[3.0, 1e16 + 1.0], [1e16 + 1.0, 0.0]])


# --------------------------------------------------------------------------- bits of the assembled matrix
def _check_shard(ctx, ref, r0=0):
    rows = ref.rows
    assert _eq(ctx.get_matrix_rows(r0, rows), ref.dense())
    if ctx.storage == "csr":
        assert ctx.nnz() == ref.col.size
        assert ctx.get_option("envelope_doubles") == 0
    else:
        assert ctx.nnz() == 0
        assert ctx.get_option("envelope_doubles") == envelope_doubles(ref.dense())


def _forms(torch, irn, jcn, val):
    """the same triples as an uncoalesced sparse tensor (int64) and as tuples with int32 and int64 indices"""
    I, J, V = _gpu(torch, irn, torch.int64), _gpu(torch, jcn, torch.int64), _gpu(torch, val)
    yield "sparse", lambda n: torch.sparse_coo_tensor(torch.stack([I, J]), V, (n, n))
    yield "tuple32", lambda n: (I.to(torch.int32), J.to(torch.int32), V)
    yield "tuple64", lambda n: (I, J, V)


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
@pytest.mark.parametrize("name", list(INPUTS))
def test_assembled_matrix_is_the_sequential_sum(cgb, torch, name, storage):
    n, irn, jcn, val, sym = INPUTS[name]()
    ref = assemble(n, irn, jcn, val, sym)
    if name == "long_run":
        assert np.diff(ref.rp).max() >= 1 and len(ref.val) < len(val) - 99_000
    with cgb.Context(n, storage=storage) as ctx:
        for form, make in _forms(torch, irn, jcn, val):
            ctx.generate_lap2d()   # a different matrix in between: the assembly has to replace it
            coo = make(n)
            if form == "sparse":
                assert not coo.is_coalesced()
            ctx.assemble_coo(coo, symmetric=sym)
            _check_shard(ctx, ref)


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
def test_assembly_takes_this_ranks_rows(cgb, torch, storage):
    n, irn, jcn, val = symmetric_coo(2001, 7)
    I, J, V = _gpu(torch, irn, torch.int32), _gpu(torch, jcn, torch.int32), _gpu(torch, val)
    for rank in range(2):
        with cgb.Context(n, rank, 2, 0, storage=storage) as ctx:
            lay = ctx.layout()
            ref = assemble(n, irn, jcn, val, True, lay.row0, lay.rows)
            ctx.assemble_coo((I, J, V), symmetric=True)
            _check_shard(ctx, ref, lay.row0)
            ctx.assemble_values(2.0 * V)
            torch.cuda.synchronize()
            _check_shard(ctx, assemble(n, irn, jcn, 2.0 * val, True, lay.row0, lay.rows), lay.row0)


# --------------------------------------------------------------------------- solves after assembly
def _host(ctx, b, x0, max_iter):
    ctx.set_rhs(b)
    x = np.array(x0, dtype=np.float64)
    info, hist = ctx.solve(x, max_iter=max_iter, tol=1e-10, history=True)
    return info, hist, x


def _device(torch, ctx, b, x0, max_iter):
    x = _gpu(torch, x0)
    info, hist = ctx.solve_device(x, _gpu(torch, b), max_iter, tol=1e-10, history=True).result()
    return info, hist, x.cpu().numpy()


def _like_oracle(d, ref):
    info, hist, x = d
    assert _key(info) == (ref.k, ref.converged, len(ref.hist))
    assert _eq(hist, ref.hist) and _eq(x, ref.x) and _eq([info.rsold, info.rsnew], [ref.rsold, ref.rsnew])


def _inputs(n, nrhs=3):
    rng = np.random.default_rng(n)
    B = rng.standard_normal((nrhs, n))
    X0 = 1e-3 * rng.standard_normal((nrhs, n))
    return B, X0


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
@pytest.mark.parametrize("sym", [False, True])
def test_solves_after_assembly_are_the_oracles(cgb, torch, storage, sym):
    n, irn, jcn, val = quad_coo(40, seed=2)
    if sym:   # the upper triangle and the diagonal, mirrored by the library
        up = irn <= jcn
        irn, jcn, val = irn[up], jcn[up], np.ascontiguousarray(val[up])
    m = assemble(n, irn, jcn, val, sym)
    assert _eq(m.dense(), m.dense().T)
    B, X0 = _inputs(n)
    max_iter = 300
    ref = csr_oracle.solve_csr(m, B[0], X0[0], max_iter=max_iter)
    with cgb.Context(n, storage=storage) as ctx:
        ctx.assemble_coo((_gpu(torch, irn, torch.int32), _gpu(torch, jcn, torch.int32), _gpu(torch, val)), sym)
        _check_shard(ctx, m)
        if storage == "csr":
            _like_oracle(_host(ctx, B[0], X0[0], max_iter), ref)
            _like_oracle(_device(torch, ctx, B[0], X0[0], max_iter), ref)
            X, infos, hist = ctx.solve_block(B, X0, max_iter=max_iter, history=True)
            for j in range(B.shape[0]):
                rj = csr_oracle.solve_csr(m, B[j], X0[j], max_iter=max_iter)
                _like_oracle((infos[j], hist[j], X[j]), rj)
        else:
            for schedule in (1, 0):
                ctx.set_option("schedule", schedule)
                _like_oracle(_host(ctx, B[0], X0[0], max_iter), ref)
                _like_oracle(_device(torch, ctx, B[0], X0[0], max_iter), ref)


# --------------------------------------------------------------------------- re-assembly
def _steps(val, k):
    """k value sets for the same triples: seeded scalings of every contribution"""
    rng = np.random.default_rng(17)
    return [np.ascontiguousarray(val * (1.0 + 0.5 * rng.random(val.size))) for _ in range(k)]


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
def test_reassembly_equals_fresh_assembly(cgb, torch, storage):
    n, irn, jcn, val = quad_coo(40, seed=4)
    I, J = _gpu(torch, irn, torch.int32), _gpu(torch, jcn, torch.int32)
    B, X0 = _inputs(n)
    max_iter = 300
    with cgb.Context(n, storage=storage) as c, cgb.Context(n, storage=storage) as f:
        c.assemble_coo((I, J, _gpu(torch, val)))
        # warm-up: the first solves allocate their buffers; the second pass captures every loop graph for good
        for _ in range(2):
            _host(c, B[0], X0[0], max_iter)
            _device(torch, c, B[0], X0[0], max_iter)
            if storage == "csr":
                c.solve_block_device(_gpu(torch, X0), _gpu(torch, B), max_iter, history=True).result()
        captures = c.get_option("graph_captures")
        for t, vt in enumerate(_steps(val, 4)):
            V = _gpu(torch, vt)
            c.assemble_values(V)
            f.assemble_coo((I, J, V))
            m = assemble(n, irn, jcn, vt, False)
            assert _eq(c.get_matrix_rows(0, n), f.get_matrix_rows(0, n))
            _check_shard(c, m)
            ref = csr_oracle.solve_csr(m, B[0], X0[0], max_iter=max_iter)
            for ctx in (c, f):
                _like_oracle(_device(torch, ctx, B[0], X0[0], max_iter), ref)
                _like_oracle(_host(ctx, B[0], X0[0], max_iter), ref)
            if storage == "csr":
                X = _gpu(torch, X0)
                infos, hist = c.solve_block_device(X, _gpu(torch, B), max_iter, history=True).result()
                Xf, finfos, fhist = f.solve_block(B, X0, max_iter=max_iter, history=True)
                assert _eq(X.cpu().numpy(), Xf) and [_key(i) for i in infos] == [_key(i) for i in finfos]
                assert all(_eq(p, q) for p, q in zip(hist, fhist))
                assert c.get_option("graph_captures") == captures, t
        if storage == "csr":   # an update of the values in stored order keeps the plan
            c.update_matrix_values(_gpu(torch, m.val * 3.0))
            c.assemble_values(_gpu(torch, val))
            torch.cuda.synchronize()
            _check_shard(c, assemble(n, irn, jcn, val, False))


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_dense_reassembly_rebuilds_the_envelopes(cgb, torch):
    """A cell that sums to 0.0 at assembly, beyond the last non-zero of its row (and, mirrored, before the
    first of its column's row), becomes non-zero: the dense mat-vec must stream it."""
    n, irn, jcn, val = quad_coo(30, seed=6)
    r, cfar = 5, n - 3
    irn = np.concatenate([irn, [r, r, cfar, cfar]]).astype(np.int32)
    jcn = np.concatenate([jcn, [cfar, cfar, r, r]]).astype(np.int32)
    v0 = np.concatenate([val, [0.25, -0.25, 0.25, -0.25]])
    v1 = np.concatenate([val, [0.25, -0.125, 0.25, -0.125]])
    m0, m1 = assemble(n, irn, jcn, v0, False), assemble(n, irn, jcn, v1, False)
    assert m0.dense()[r, cfar] == 0.0 and m1.dense()[r, cfar] == 0.125
    assert envelope_doubles(m1.dense()) > envelope_doubles(m0.dense())
    B, X0 = _inputs(n)
    with cgb.Context(n) as ctx:
        I, J = _gpu(torch, irn, torch.int32), _gpu(torch, jcn, torch.int32)
        ctx.assemble_coo((I, J, _gpu(torch, v0)))
        _check_shard(ctx, m0)
        _like_oracle(_device(torch, ctx, B[0], X0[0], 200), csr_oracle.solve_csr(m0, B[0], X0[0], max_iter=200))
        ctx.assemble_values(_gpu(torch, v1))
        _like_oracle(_device(torch, ctx, B[0], X0[0], 200), csr_oracle.solve_csr(m1, B[0], X0[0], max_iter=200))
        _check_shard(ctx, m1)
        for schedule in (1, 0):
            ctx.set_option("schedule", schedule)
            _like_oracle(_host(ctx, B[0], X0[0], 200), csr_oracle.solve_csr(m1, B[0], X0[0], max_iter=200))


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
def test_reassembly_is_ordered_on_the_stream_and_asynchronous(cgb, torch, storage):
    n, irn, jcn, val = quad_coo(40, seed=8)
    b_host = np.random.default_rng(3).standard_normal(n)
    with cgb.Context(n, storage=storage) as c:
        I, J, base = _gpu(torch, irn, torch.int32), _gpu(torch, jcn, torch.int32), _gpu(torch, val)
        b = _gpu(torch, b_host)
        c.assemble_coo((I, J, base))
        x = torch.zeros(n, dtype=torch.float64, device="cuda:0")
        c.assemble_values(base.clone())
        c.solve_device(x, b, 200).result()                             # warm-up: graphs, buffers, events
        s = torch.cuda.current_stream()
        x1 = torch.zeros(n, dtype=torch.float64, device="cuda:0")
        x2 = torch.zeros(n, dtype=torch.float64, device="cuda:0")
        torch.cuda.synchronize()
        torch.cuda._sleep(100_000_000)                                  # ~50 ms of GPU clock cycles
        v1 = base * 1.5 + 0.001                                         # values made by torch kernels, no sync
        c.assemble_values(v1)
        h1 = c.solve_device(x1, b, 200, history=True)
        v2 = torch.sin(base) + base
        c.assemble_values(v2)
        h2 = c.solve_device(x2, b, 200, history=True)
        ev = torch.cuda.Event()
        ev.record(s)
        assert not ev.query(), "a call waited for the stream"
        got = [(*h.result(), xx.cpu().numpy()) for h, xx in ((h1, x1), (h2, x2))]
        vals = [v1.cpu().numpy(), v2.cpu().numpy()]
    for d, v in zip(got, vals):
        m = assemble(n, irn, jcn, v, False)
        _like_oracle(d, csr_oracle.solve_csr(m, b_host, None, max_iter=200))


# --------------------------------------------------------------------------- refusals
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("storage", ["csr", "dense"])
def test_assembly_refusals(cgb, torch, storage):
    n, irn, jcn, val = quad_coo(20, seed=10)
    m = assemble(n, irn, jcn, val, False)
    I, J, V = _gpu(torch, irn, torch.int32), _gpu(torch, jcn, torch.int32), _gpu(torch, val)
    host = np.zeros(2 * val.size)
    pinned = torch.zeros(val.size, dtype=torch.float64).pin_memory()
    b = np.random.default_rng(0).standard_normal(n)

    with cgb.Context(n, storage=storage) as ctx:
        lib = ctx._lib

        def coo(i=I.data_ptr(), j=J.data_ptr(), v=V.data_ptr(), z=val.size):
            return lib.cgb_assemble_coo(ctx._h, z, i, j, v, 0, None)

        def again(p=V.data_ptr()):
            return lib.cgb_assemble_values(ctx._h, p, None)

        assert again() == 2 and b"assembly plan" in lib.cgb_last_error()   # nothing assembled yet
        ctx.assemble_coo((I, J, V))
        _check_shard(ctx, m)
        # an entry outside n x n, in each index and either sign: the matrix and the plan stay
        for t, k, bad in ((I, 17, n), (J, val.size - 1, n), (I, 0, -1), (J, 333, -5)):
            w = t.clone()
            w[k] = bad
            args = {"i": w.data_ptr()} if t is I else {"j": w.data_ptr()}
            assert coo(**args) == 1 and b"outside" in lib.cgb_last_error(), (k, bad)
        with pytest.raises(cgb.CgbError) as ei:
            ctx.assemble_coo((I.to(torch.int64) + 2 ** 32, J, V))   # wraps to an index in range when narrowed
        assert ei.value.code == 1
        _check_shard(ctx, m)
        assert again((2.0 * V).data_ptr()) == 0
        torch.cuda.synchronize()
        _check_shard(ctx, assemble(n, irn, jcn, 2.0 * val, False))
        hp = host.ctypes.data
        for args in ({"z": -1}, {"i": None}, {"j": None}, {"v": None}, {"i": hp}, {"v": hp},
                     {"j": pinned.data_ptr()}, {"v": pinned.data_ptr()}):
            assert coo(**args) == 1, args
        for p in (None, hp, pinned.data_ptr()):
            assert again(p) == 1, p
        assert again(pinned.data_ptr()) == 1 and b"host" in lib.cgb_last_error()
        with pytest.raises(TypeError):
            ctx.assemble_coo((I.cpu(), J.cpu(), V.cpu()))
        with pytest.raises(TypeError):
            ctx.assemble_coo((I, J, V.float()))
        with pytest.raises(ValueError):
            ctx.assemble_coo((I[:-1], J, V))
        with pytest.raises(ValueError):
            ctx.assemble_values(V[:-1])
        torch.cuda.synchronize()
        _check_shard(ctx, assemble(n, irn, jcn, 2.0 * val, False))   # no refused call wrote anything
        # one matrix build at a time with a solve
        ctx.set_rhs(b)
        ctx.solve_begin(np.zeros(n), 10)
        assert again() == 2 and coo() == 2
        ctx.solve_end()
        if storage == "csr":
            ctx.solve_block_begin(np.array([b, b]), max_iter=10)
            assert again() == 2 and coo() == 2
            ctx.iterate(10)
            ctx.solve_block_end()
        assert again() == 0
        # every other builder drops the plan
        T = csr_oracle.generate_lap2d_csr(n)
        builders = [ctx.generate_lap2d,
                    lambda: ctx.set_matrix_coo(*_coo(T), symmetric=False),
                    lambda: ctx.set_matrix_csr((_gpu(torch, T.rp, torch.int64), _gpu(torch, T.col, torch.int64),
                                                _gpu(torch, T.val)))]
        if storage == "dense":
            builders.append(lambda: ctx.set_matrix_rows(T.dense()[:3], first_row=0))
        for build in builders:
            assert coo() == 0 and again() == 0
            build()
            assert again() == 2, build
    with cgb.Context(n, storage=storage) as ctx:
        ctx.assemble_coo((I[:0], J[:0], V[:0]))   # nothing assembled: an empty matrix, and a plan of it
        assert ctx.nnz() == 0 and not ctx.get_matrix_rows(0, n).any()
        assert ctx._lib.cgb_assemble_values(ctx._h, None, None) == 0


def _coo(m):
    return np.repeat(np.arange(m.rows), np.diff(m.rp)).astype(np.int32), m.col.copy(), m.val.copy()


# --------------------------------------------------------------------------- without a GPU
def test_assembly_without_gpu_fails_loudly(cgb):
    try:
        if cgb.device_count() > 0:
            pytest.skip("a GPU is present")
    except cgb.CgbError:
        pass
    lib = cgb.load()
    buf = np.zeros(64)
    p = buf.ctypes.data
    assert lib.cgb_assemble_coo(None, 4, p, p, p, 0, None) == 3
    assert lib.cgb_assemble_values(None, p, None) == 3
    assert np.all(buf == 0.0)
