"""CSR storage without a GPU: the CSR oracle (tests/csr_oracle.c) is the dense oracle bit for bit, the
COO -> CSR restatement keeps Matrix::read's semantics, and the CSR entry points of the library
and of `cgsolver` fail loudly without a device."""
import os
import subprocess

import numpy as np
import pytest

import csr_oracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CGSOLVER = os.path.join(ROOT, "conjugate-gradient_b200", "host", "cgsolver")


def _bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


def _same_solve(a, b):
    """bit for bit, NaNs included (n = 1 has b = 0)"""
    assert a.k == b.k and a.converged == b.converged
    assert np.array_equal(_bits(a.hist), _bits(b.hist))
    assert np.array_equal(_bits(a.x), _bits(b.x))
    assert np.array_equal(_bits([a.rsold, a.rsnew, a.norm_x, a.rel_resid]),
                          _bits([b.rsold, b.rsnew, b.norm_x, b.rel_resid]))


@pytest.mark.parametrize("n", [1, 2, 17, 255, 1000, 4096])
def test_lap2d_csr_oracle_is_the_dense_oracle(O, n):
    m = csr_oracle.generate_lap2d_csr(n)
    A = O.generate_lap2d(n)
    assert np.array_equal(m.dense(), A)
    inc = int(np.floor(np.sqrt(n)))
    assert m.col.size == n + 2 * (n - 1) + 2 * max(0, n - 1 - inc)
    assert all(np.all(np.diff(m.col[m.rp[i]:m.rp[i + 1]]) > 0) for i in range(0, n, max(1, n // 97)))
    b = O.init_source_term(n)
    it = n if n <= 1000 else 200
    _same_solve(csr_oracle.solve_csr(m, b, max_iter=it), O.solve(A, b, max_iter=it))


def test_lap2d_csr_rows_of_a_shard(O):
    n = 1000
    for row0, rows in [(0, 333), (333, 333), (666, 334)]:
        m = csr_oracle.generate_lap2d_csr(n, row0, rows)
        assert np.array_equal(m.dense(), O.generate_lap2d_rows(n, row0, rows))


def _random_spd(n, seed):
    """Symmetric, diagonally dominant where not empty: rows of 0 .. 1500 entries (bucket collisions
    c = c' mod 64 in every long row, a row > 1024), empty rows, stored +0 / -0 cells."""
    rng = np.random.default_rng(seed)
    A = np.zeros((n, n))
    lens = rng.integers(0, 6, n)
    lens[rng.choice(n, 40, replace=False)] = rng.integers(65, 300, 40)
    lens[rng.choice(n, 2, replace=False)] = 1500
    for i in range(n):
        cols = rng.choice(n, lens[i], replace=False)
        A[i, cols] = rng.standard_normal(lens[i])
    A[7, [3, 67, 131, 195]] = [1.0, 2.0, -3.0, 0.5]            # one bucket, a short row
    A = A + A.T
    empty = rng.choice(n, 5, replace=False)
    A[empty, :] = 0.0
    A[:, empty] = 0.0
    d = np.abs(A).sum(axis=1) + 1.0
    d[empty] = 0.0
    A[np.arange(n), np.arange(n)] += d
    keep = np.zeros((n, n), dtype=bool)
    zr, zc = rng.integers(0, n, 30), rng.integers(0, n, 30)
    ok = ~np.isin(zr, empty) & ~np.isin(zc, empty)
    zr, zc = zr[ok], zc[ok]
    A[zr, zc] = A[zc, zr] = np.where(np.arange(zr.size) % 2, 0.0, -0.0)
    keep[zr, zc] = keep[zc, zr] = True
    b = rng.standard_normal(n)
    b[empty] = 0.0
    return A, keep, b, empty


def test_random_spd_csr_oracle_is_the_dense_oracle(O):
    n = 3000
    A, keep, b, empty = _random_spd(n, 5)
    m = csr_oracle.csr_from_dense(A, keep)
    lens = np.diff(m.rp)
    assert lens.max() > 1024 and (lens[empty] == 0).all() and ((lens > 64) & (lens <= 1024)).any()
    assert (np.signbit(m.val) & (m.val == 0)).any() and (~np.signbit(m.val) & (m.val == 0)).any()
    p = np.random.default_rng(1).standard_normal(n)
    assert np.array_equal(csr_oracle.gemv_csr(m, p), O.gemv(A, p))
    x0 = np.random.default_rng(2).standard_normal(n)
    x0[empty] = 0.0
    r_csr, r_dense = csr_oracle.solve_csr(m, b, x0=x0, max_iter=60), O.solve(A, b, x0=x0, max_iter=60)
    assert np.isfinite(r_csr.x).all()
    _same_solve(r_csr, r_dense)


@pytest.mark.parametrize("symmetric", [False, True])
def test_csr_from_coo_keeps_matrix_read_semantics(O, symmetric):
    """Duplicates: the last write in file order wins, the mirror write of a symmetric entry
    included; explicit zeros are stored; a row range keeps only its rows."""
    n, nz = 300, 40000
    rng = np.random.default_rng(21 + int(symmetric))
    irn = rng.integers(0, n, nz)
    jcn = rng.integers(0, n, nz)
    val = rng.standard_normal(nz)
    val[::97] = 0.0
    A = np.zeros((n, n))
    for i, j, a in zip(irn, jcn, val):           # matrix.cc:12-21
        A[i, j] = a
        if symmetric:
            A[j, i] = a
    m = csr_oracle.csr_from_coo(n, irn, jcn, val, symmetric)
    assert np.array_equal(m.dense(), A)
    assert (m.val == 0).any()
    for row0, rows in [(0, 100), (100, 200)]:
        assert np.array_equal(csr_oracle.csr_from_coo(n, irn, jcn, val, symmetric, row0, rows).dense(), A[row0:row0 + rows])
    p = rng.standard_normal(n)
    assert np.array_equal(csr_oracle.gemv_csr(m, p), O.gemv(A, p))


def test_mtx_fixture_csr_solve_is_the_dense_solve(O, tmp_path):
    path = str(tmp_path / "lap.mtx")
    O.write_lap2d_5pt_mtx(path, 30)
    A = O.read_mtx_dense(path)
    n = A.shape[0]
    lines = open(path).read().split("\n")[3:]
    t = np.array([ln.split() for ln in lines if ln.strip()], dtype=float)
    m = csr_oracle.csr_from_coo(n, t[:, 0].astype(int) - 1, t[:, 1].astype(int) - 1, t[:, 2], True)
    b = O.init_source_term(n)
    _same_solve(csr_oracle.solve_csr(m, b, max_iter=n), O.solve(A, b, max_iter=n))


def _no_gpu(cgb):
    try:
        return cgb.device_count() == 0
    except cgb.CgbError:
        return True


def test_create_csr_without_gpu_fails_loudly(cgb):
    if not _no_gpu(cgb):
        pytest.skip("a GPU is present")
    import ctypes
    h = ctypes.c_void_p()
    assert cgb.load().cgb_create_csr(128, 0, 1, 0, ctypes.byref(h)) == 3   # CGB_ERR_NO_DEVICE
    with pytest.raises(cgb.CgbError) as ei:
        cgb.Context(128, storage="csr")
    assert ei.value.code == 3
    with pytest.raises(ValueError):
        cgb.Context(128, storage="coo")


def _cli(tmp_path, env, *args):
    e = dict(os.environ, **env)
    return subprocess.run([CGSOLVER, *args], capture_output=True, text=True, timeout=120, cwd=str(tmp_path), env=e)


def test_cgsolver_csr_storage_without_gpu(cgb, tmp_path):
    if not os.path.exists(CGSOLVER):
        pytest.skip("cgsolver not built")
    out = _cli(tmp_path, {"CGB_STORAGE": "csr", "CGB_KERNEL": "compat"}, "100", "out")
    assert out.returncode == 2 and "CGB_STORAGE=csr" in out.stderr and out.stdout == ""
    out = _cli(tmp_path, {"CGB_STORAGE": "sparse"}, "100", "out")
    assert out.returncode == 2 and "CGB_STORAGE" in out.stderr
    if not _no_gpu(cgb):
        return
    dense = _cli(tmp_path, {}, "100", "out")
    csr = _cli(tmp_path, {"CGB_STORAGE": "csr"}, "100", "out")
    assert dense.returncode == csr.returncode == 2
    assert csr.stdout == "" and "cgb_create_csr" in csr.stderr
    assert not (tmp_path / "out").exists()
