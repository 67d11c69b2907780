"""CSR storage on the B200: construction, the CSR mat-vec and whole solves, bit for bit against
dense contexts holding the same matrix and against the CSR oracle (which tests/test_sparse_cpu.py
ties to the dense oracle).  Multi-GPU cases skip on a machine with one GPU."""
import hashlib
import os
import subprocess
import threading

import numpy as np
import pytest

import csr_oracle

pytestmark = [pytest.mark.gpu, pytest.mark.timeout(900)]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CGSOLVER = os.path.join(ROOT, "conjugate-gradient_b200", "host", "cgsolver")


def _bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


def _eq(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _solve(cgb, n, storage, setup, max_iter, x0=None, tol=1e-10):
    with cgb.Context(n, storage=storage) as ctx:
        setup(ctx)
        x = np.zeros(n) if x0 is None else x0.copy()
        info, hist = ctx.solve(x, max_iter=max_iter, tol=tol, history=True)
        nx, rr = ctx.residual_check()
    return x, info, hist, nx, rr


def _same_as_oracle(got, ref):
    x, info, hist, nx, rr = got
    assert info.k == ref.k and bool(info.converged) == ref.converged
    assert info.iterations == len(ref.hist)
    assert _eq(hist, ref.hist) and _eq(x, ref.x)
    assert _eq([info.rsold, info.rsnew, nx, rr], [ref.rsold, ref.rsnew, ref.norm_x, ref.rel_resid])


def _lap2d(b):
    def setup(ctx):
        ctx.generate_lap2d()
        ctx.set_rhs(b)
    return setup


# --------------------------------------------------------------------------- construction
@pytest.mark.parametrize("n", [1, 2, 17, 1000, 2050])
def test_generate_lap2d_csr_rows(cgb, O, n):
    inc = int(np.floor(np.sqrt(n)))
    with cgb.Context(n, storage="csr") as ctx:
        ctx.generate_lap2d()
        assert ctx.get_option("storage") == 1
        assert ctx.nnz() == n + 2 * (n - 1) + 2 * max(0, n - 1 - inc)
        assert np.array_equal(ctx.get_matrix_rows(0, n), O.generate_lap2d(n))
    if n >= 3:   # the shard of every rank of a 3-way split
        s, c = cgb.partition(n, 3)
        for r in range(3):
            with cgb.Context(n, r, 3, 0, storage="csr") as ctx:
                ctx.generate_lap2d()
                assert np.array_equal(ctx.get_matrix_rows(s[r], c[r]), O.generate_lap2d_rows(n, s[r], c[r]))


@pytest.mark.parametrize("symmetric", [False, True])
def test_coo_million_duplicates_dense_and_csr_are_the_oracle(cgb, symmetric):
    n, nz = 1500, 1_000_000
    rng = np.random.default_rng(31 + int(symmetric))
    irn = rng.integers(0, n, nz, dtype=np.int32)
    jcn = rng.integers(0, n, nz, dtype=np.int32)
    val = rng.standard_normal(nz)
    val[::1000] = 0.0
    val[500::1000] = -0.0
    ref = csr_oracle.csr_from_coo(n, irn, jcn, val, symmetric)
    zero = ref.val == 0
    assert np.signbit(ref.val[zero]).any() and not np.signbit(ref.val[zero]).all()  # -0 and +0 last writers
    want = ref.dense()
    with cgb.Context(n) as d, cgb.Context(n, storage="csr") as c:
        d.set_matrix_coo(irn, jcn, val, symmetric=symmetric)
        c.set_matrix_coo(irn, jcn, val, symmetric=symmetric)
        assert _eq(d.get_matrix_rows(0, n), want)
        assert _eq(c.get_matrix_rows(0, n), want)
        assert c.nnz() == ref.col.size   # explicit zeros stored
        s, cnt = cgb.partition(n, 3)
        for r in range(3):   # every shard of a 3-way split
            part = csr_oracle.csr_from_coo(n, irn, jcn, val, symmetric, s[r], cnt[r])
            for storage in ("dense", "csr"):
                with cgb.Context(n, r, 3, 0, storage=storage) as ctx:
                    ctx.set_matrix_coo(irn, jcn, val, symmetric=symmetric)
                    assert _eq(ctx.get_matrix_rows(s[r], cnt[r]), part.dense())
                    if storage == "csr":
                        assert ctx.nnz() == part.col.size
        with pytest.raises(cgb.CgbError) as ei:
            c.set_matrix_coo(np.array([0, n], dtype=np.int32), np.array([0, 0], dtype=np.int32),
                             np.array([1.0, 2.0]), symmetric=False)
        assert ei.value.code == 1


@pytest.mark.parametrize("storage", ["dense", "csr"])
def test_refused_coo_keeps_the_previous_matrix(cgb, O, storage):
    """A COO load with an entry outside n x n is refused before the context is touched: the previous
    matrix stays, bit for bit, and still solves."""
    n = 1000
    b = O.init_source_term(n)
    x_ref, info_ref, hist_ref, _, _ = _solve(cgb, n, storage, _lap2d(b), n)
    with cgb.Context(n, storage=storage) as ctx:
        ctx.generate_lap2d()
        ctx.set_rhs(b)
        A = ctx.get_matrix_rows(0, n)
        with pytest.raises(cgb.CgbError) as ei:
            ctx.set_matrix_coo(np.array([0, n], dtype=np.int32), np.array([0, 0], dtype=np.int32),
                               np.array([1.0, 2.0]), symmetric=False)
        assert ei.value.code == 1 and "outside" in str(ei.value)
        assert _eq(ctx.get_matrix_rows(0, n), A)
        x = np.zeros(n)
        info, hist = ctx.solve(x, max_iter=n, history=True)
    assert (info.k, info.converged) == (info_ref.k, info_ref.converged)
    assert _eq(hist, hist_ref) and _eq(x, x_ref)


# --------------------------------------------------------------------------- mat-vec
def _ragged_matrix(n, seed):
    """row lengths 0 .. 2000, colliding buckets, explicit zeros; returned as sorted COO triples"""
    rng = np.random.default_rng(seed)
    lens = rng.integers(0, 7, n)
    lens[rng.choice(n, 60, replace=False)] = rng.integers(9, 2001, 60)
    lens[rng.choice(n, 20, replace=False)] = 0
    rows, cols = [], []
    for i in range(n):
        c = np.sort(rng.choice(n, lens[i], replace=False))
        rows.append(np.full(c.size, i))
        cols.append(c)
    irn, jcn = np.concatenate(rows), np.concatenate(cols)
    val = rng.standard_normal(irn.size)
    val[::53] = 0.0
    val[::59] = -0.0
    return irn.astype(np.int32), jcn.astype(np.int32), val


@pytest.mark.parametrize("n", [3000, 5000])
def test_csr_gemv_is_the_dense_gemv(cgb, O, n):
    irn, jcn, val = _ragged_matrix(n, n)
    v = np.random.default_rng(7).standard_normal(n)
    with cgb.Context(n) as d, cgb.Context(n, storage="csr") as c:
        d.set_matrix_coo(irn, jcn, val, symmetric=False)
        c.set_matrix_coo(irn, jcn, val, symmetric=False)
        assert c.nnz() == irn.size
        yd, pd, sd = d.gemv(v, want_partials=True)
        yc, pc, sc = c.gemv(v, want_partials=True)
    assert _eq(yc, yd) and _eq(pc, pd) and _eq(sc, sd)
    assert _eq(yc, csr_oracle.gemv_csr(csr_oracle.csr_from_coo(n, irn, jcn, val, False), v))


# --------------------------------------------------------------------------- solves
@pytest.mark.parametrize("n,max_iter", [(1000, 50), (1024, 1024), (1448, 200), (2048, 2048)])
def test_csr_solve_generated_bitwise(cgb, O, n, max_iter):
    b = O.init_source_term(n)
    got = _solve(cgb, n, "csr", _lap2d(b), max_iter)
    _same_as_oracle(got, O.solve(O.generate_lap2d(n), b, max_iter=max_iter))


def test_csr_solve_nonzero_x0_max_iter_zero_early_stop(cgb, O):
    n = 1536
    b = O.init_source_term(n)
    x0 = np.random.default_rng(3).standard_normal(n)
    A = O.generate_lap2d(n)
    _same_as_oracle(_solve(cgb, n, "csr", _lap2d(b), 120, x0=x0), O.solve(A, b, x0=x0, max_iter=120))
    x, info, hist, *_ = _solve(cgb, n, "csr", _lap2d(b), 0, x0=x0)
    assert info.k == 0 and info.iterations == 0 and not info.converged and _eq(x, x0) and len(hist) == 0
    got = _solve(cgb, n, "csr", _lap2d(b), n)
    _same_as_oracle(got, O.solve(A, b, max_iter=n))
    x, info, hist, *_ = got
    assert info.converged and info.iterations == info.k + 1 and info.rsold == hist[-2]


def test_csr_solve_mtx_fixture(cgb, O, tmp_path):
    path = str(tmp_path / "lap2D_5pt_n100.mtx")
    O.write_lap2d_5pt_mtx(path, 100)
    A = O.read_mtx_dense(path)
    n = A.shape[0]
    t = np.loadtxt(path, skiprows=3)
    irn, jcn = t[:, 0].astype(np.int32) - 1, t[:, 1].astype(np.int32) - 1
    b = O.init_source_term(n)

    def setup(ctx):
        ctx.set_matrix_coo(irn, jcn, t[:, 2], symmetric=True)
        ctx.set_rhs(b)

    got = _solve(cgb, n, "csr", setup, n)
    assert got[1].k == 488 and got[1].converged
    dense = _solve(cgb, n, "dense", setup, n)
    assert _eq(got[0], dense[0]) and _eq(got[2], dense[2]) and _eq(got[3:], dense[3:])
    _same_as_oracle(got, O.solve(A, b, max_iter=n))


def test_csr_reference_goldens(cgb, O):
    """N = 20000 converges at k = 875; N = 40000 x 200 gives the digest DESIGN.md records."""
    n = 20000
    x, info, *_ = _solve(cgb, n, "csr", _lap2d(O.init_source_term(n)), n)
    assert info.converged and info.k == 875
    n = 40000
    x, info, hist, nx, rr = _solve(cgb, n, "csr", _lap2d(O.init_source_term(n)), 200)
    digest = hashlib.sha256(x.tobytes() + hist.tobytes() + np.array([nx, rr]).tobytes()).hexdigest()
    assert digest[:16] == "1b58205beac19aa4"


@pytest.mark.parametrize("n", [2_000_000, 16_000_000])
def test_csr_large_n_vs_csr_oracle(cgb, O, n):
    """Past the chunk count at which the dense path's vector kernels run out of shared memory."""
    b = O.init_source_term(n)
    got = _solve(cgb, n, "csr", _lap2d(b), 50)
    _same_as_oracle(got, csr_oracle.solve_csr(csr_oracle.generate_lap2d_csr(n), b, max_iter=50))


def test_dense_past_the_int_limit_vs_csr_oracle(cgb, O):
    """The dense path at N = 46400 (N^2 > INT_MAX) against the O(nnz) CSR oracle, bit for bit."""
    n = 46400
    b = O.init_source_term(n)
    got = _solve(cgb, n, "dense", _lap2d(b), 50)
    _same_as_oracle(got, csr_oracle.solve_csr(csr_oracle.generate_lap2d_csr(n), b, max_iter=50))


@pytest.mark.parametrize("form", ["solve", "solve_block"])
def test_csr_graph_solve_after_matrix_reload(cgb, O, form):
    """Every CSR build reallocates col / val, which the captured loop graphs bake in.  A second solve with
    the same tol and history after loading a larger matrix must capture its graph anew: replaying the
    first one would run the mat-vec on the freed arrays of lap2d."""
    from test_gpu_block import _ragged_coo
    n, max_iter = 3001, 200
    irn, jcn, val, empty = _ragged_coo(n, 11)
    m = csr_oracle.csr_from_coo(n, irn, jcn, val, False)
    B = np.random.default_rng(12).standard_normal((3, n))
    B[0] = O.init_source_term(n)
    B[:, empty] = 0.0
    with cgb.Context(n, storage="csr") as ctx:
        assert max_iter >= min(ctx.get_option("graph_unroll"), ctx.get_option("poll_every"))

        def run():
            if form == "solve":
                ctx.set_rhs(B[0])
                x = np.zeros(n)
                info, hist = ctx.solve(x, max_iter=max_iter, history=True)
                return x[None], [info], hist[None]
            return ctx.solve_block(B, None, max_iter=max_iter, history=True)

        ctx.generate_lap2d()
        lap_nnz = ctx.nnz()
        run()
        replays = ctx.get_option("graph_replays")
        ctx.set_matrix_coo(irn, jcn, val, symmetric=False)
        assert ctx.nnz() == m.col.size > lap_nnz
        X, infos, hist = run()
        assert ctx.get_option("graph_replays") > replays
    for j in range(len(infos)):
        ref = csr_oracle.solve_csr(m, B[j], np.zeros(n), max_iter=max_iter)
        assert (infos[j].k, bool(infos[j].converged), infos[j].iterations) == (ref.k, ref.converged, len(ref.hist))
        assert _eq(hist[j], ref.hist) and _eq(X[j], ref.x)
        assert _eq([infos[j].rsold, infos[j].rsnew], [ref.rsold, ref.rsnew])


# --------------------------------------------------------------------------- options
def test_csr_options(cgb):
    n = 4096
    with cgb.Context(n, storage="csr") as c, cgb.Context(n) as d:
        c.generate_lap2d()
        assert c.get_option("storage") == 1 and d.get_option("storage") == 0
        assert c.get_option("nnz") == c.nnz() > 0 and d.get_option("nnz") == 0
        assert c.get_option("schedule_in_use") == 0
        for k in ("gemv_variant", "num_threads", "block_width", "transposed"):
            c.set_option(k, 1)
        for k, v in (("compat", 1), ("loopback", 1), ("trace", 4)):
            with pytest.raises(cgb.CgbError) as ei:
                c.set_option(k, v)
            assert ei.value.code == 2
        with pytest.raises(cgb.CgbError) as ei:
            c.set_matrix_rows(np.zeros((1, n)))
        assert ei.value.code == 2
        before = c.get_option("gemv_variant")
        r = c.autotune()
        assert r["us_per_iteration"] == {} and c.get_option("gemv_variant") == before
        assert c.bench_gemv(reps=3) > 0 and c.bench_read(reps=3) > 0


# --------------------------------------------------------------------------- multi-GPU
def _ngpu(cgb):
    try:
        return cgb.device_count()
    except cgb.CgbError:
        return 0


def _solve_ranks(cgb, n, world, exchange, max_iter, b):
    ctxs = [cgb.Context(n, r, world, r, storage="csr") for r in range(world)]
    try:
        if exchange == "fused":
            blobs = [c.exchange_export() for c in ctxs]
            for c in ctxs:
                c.exchange_import(blobs)
        else:
            uid = cgb.unique_id()
            th = [threading.Thread(target=c.comm_init, args=(uid,)) for c in ctxs]
            [t.start() for t in th]
            [t.join() for t in th]
        out, err = [None] * world, []

        def body(r):
            try:
                c = ctxs[r]
                c.generate_lap2d()
                c.set_rhs(b)
                x = np.zeros(n)
                info, hist = c.solve(x, max_iter=max_iter, history=True)
                out[r] = (x, info, hist, *c.residual_check())
            except BaseException as e:  # noqa: BLE001
                err.append(e)

        th = [threading.Thread(target=body, args=(r,)) for r in range(world)]
        [t.start() for t in th]
        [t.join() for t in th]
        assert not err, err
        return out
    finally:
        for c in ctxs:
            c.close()


@pytest.mark.parametrize("exchange", ["fused", "nccl"])
@pytest.mark.parametrize("n", [4096, 4099])
def test_csr_two_gpus_equal_one(cgb, O, exchange, n):
    if _ngpu(cgb) < 2:
        pytest.skip("needs 2 GPUs")
    b = O.init_source_term(n)
    one = _solve(cgb, n, "csr", _lap2d(b), 300)
    for x, info, hist, nx, rr in _solve_ranks(cgb, n, 2, exchange, 300, b):
        assert info.k == one[1].k and _eq(x, one[0]) and _eq(hist, one[2]) and _eq([nx, rr], one[3:])


# --------------------------------------------------------------------------- CLI
def _cli(tmp_path, env, *args):
    e = dict(os.environ, CGB_AUTOTUNE="0", **env)
    out = subprocess.run([CGSOLVER, *args], capture_output=True, text=True, timeout=600, cwd=str(tmp_path), env=e)
    assert out.returncode == 0, out.stderr
    return out.stdout


def _debug_line(stdout):
    return [ln for ln in stdout.splitlines() if "[STEP" in ln]


def test_cli_csr_prints_the_dense_debug_line(cgb, O, tmp_path):
    dense = _cli(tmp_path, {}, "40000", "d.txt", "200")
    csr = _cli(tmp_path, {"CGB_STORAGE": "csr", "CGB_JSON": str(tmp_path / "j.json")}, "40000", "c.txt", "200")
    assert _debug_line(csr) == _debug_line(dense) and len(_debug_line(csr)) == 1
    d, c = open(tmp_path / "d.txt").read().split(","), open(tmp_path / "c.txt").read().split(",")
    assert c[:2] == d[:2] == ["40000", "1"] and len(c) == len(d) == 3
    assert '"storage": "csr"' in open(tmp_path / "j.json").read()
    if _ngpu(cgb) >= 2:
        two = _cli(tmp_path, {"CGB_STORAGE": "csr", "CGB_GPUS": "2"}, "40000", "c2.txt", "200")
        assert _debug_line(two) == _debug_line(dense)
    path = str(tmp_path / "lap2D_5pt_n100.mtx")
    O.write_lap2d_5pt_mtx(path, 100)
    dense = _cli(tmp_path, {}, path, "64", "512", "true", "m_d.txt")
    csr = _cli(tmp_path, {"CGB_STORAGE": "csr"}, path, "64", "512", "true", "m_c.txt")
    assert _debug_line(csr) == _debug_line(dense)
    assert "Time for CG (dense solver)" in csr
    assert open(tmp_path / "m_c.txt").read().split(",")[:2] == ["64", "512"]
