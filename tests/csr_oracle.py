"""ctypes front-end of the CSR oracle (tests/csr_oracle.c): CSR storage, its lane-order mat-vec and
the CG solve over it, O(nnz) per iteration.  TEST INFRASTRUCTURE ONLY.

csr_oracle.c includes the dense oracle's source (oracle/cg_oracle.c) unchanged, so every reduction
is the dense oracle's; tests/test_sparse_cpu.py checks the two bit for bit.  The library is compiled
on first use into a temporary directory (the repository may be read-only), keyed by the sources.
"""
from __future__ import annotations

import ctypes as C
import hashlib
import os
import subprocess
import tempfile
from dataclasses import dataclass

import numpy as np

import oracle

_HERE = os.path.dirname(os.path.abspath(__file__))
_SRC = os.path.join(_HERE, "csr_oracle.c")
_ORACLE_DIR = os.path.join(os.path.dirname(_HERE), "oracle")
_LIB = None
_p = oracle._p

_dp = C.POINTER(C.c_double)
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)


def build() -> str:
    h = hashlib.sha256()
    for f in (_SRC, os.path.join(_ORACLE_DIR, "cg_oracle.c"), os.path.join(_ORACLE_DIR, "cg_oracle.h")):
        h.update(open(f, "rb").read())
    so = os.path.join(tempfile.gettempdir(), f"cgb_csr_oracle_{os.getuid()}_{h.hexdigest()[:16]}.so")
    if not os.path.exists(so):
        fd, tmp = tempfile.mkstemp(suffix=".so", dir=tempfile.gettempdir())
        os.close(fd)
        subprocess.check_call(["gcc", "-O2", "-mfma", "-ffp-contract=off", "-fopenmp", "-shared", "-fPIC",
                               "-o", tmp, _SRC, "-lm"])
        os.replace(tmp, so)
    return so


def lib():
    global _LIB
    if _LIB is None:
        L = C.CDLL(build())
        L.cso_generate_lap2d.argtypes = [C.c_int64, C.c_int64, C.c_int64, _i64p, _i32p, _dp]
        L.cso_generate_lap2d.restype = C.c_int64
        L.cso_row_dot.argtypes = [_i32p, _dp, C.c_int64, _dp]
        L.cso_row_dot.restype = C.c_double
        L.cso_gemv.argtypes = [C.c_int64, _i64p, _i32p, _dp, _dp, _dp]
        L.cso_solve.argtypes = [C.c_int64, _i64p, _i32p, _dp, _dp, _dp, C.c_int64, C.c_double, _dp,
                                C.POINTER(oracle._Info)]
        L.cso_residual_check.argtypes = [C.c_int64, _i64p, _i32p, _dp, _dp, _dp, _dp, _dp]
        _LIB = L
    return _LIB


@dataclass
class Csr:
    """rows x n shard: rp[rows + 1] int64, col int32 (ascending, unique per row), val float64."""
    n: int
    rp: np.ndarray
    col: np.ndarray
    val: np.ndarray

    @property
    def rows(self) -> int:
        return self.rp.size - 1

    def dense(self) -> np.ndarray:
        A = np.zeros((self.rows, self.n), dtype=np.float64)
        A[np.repeat(np.arange(self.rows), np.diff(self.rp)), self.col] = self.val
        return A


def _ci(a, dt, ptr):
    assert a.dtype == dt and a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(ptr)


def generate_lap2d_csr(n: int, row0: int = 0, nrows: int | None = None) -> Csr:
    nrows = n - row0 if nrows is None else nrows
    rp = np.empty(nrows + 1, dtype=np.int64)
    nnz = lib().cso_generate_lap2d(n, row0, nrows, _ci(rp, np.int64, _i64p), None, None)
    col = np.empty(nnz, dtype=np.int32)
    val = np.empty(nnz, dtype=np.float64)
    lib().cso_generate_lap2d(n, row0, nrows, _ci(rp, np.int64, _i64p), _ci(col, np.int32, _i32p), _p(val))
    return Csr(n, rp, col, val)


def csr_from_dense(A: np.ndarray, keep=None) -> Csr:
    """The non-zeros of A (plus the cells where `keep` is True, stored even when zero)."""
    mask = A != 0 if keep is None else (A != 0) | keep
    rows, n = A.shape
    rp = np.zeros(rows + 1, dtype=np.int64)
    rp[1:] = np.cumsum(mask.sum(axis=1))
    r, c = np.nonzero(mask)
    return Csr(n, rp, c.astype(np.int32), np.ascontiguousarray(A[r, c], dtype=np.float64))


def csr_from_coo(n: int, irn, jcn, val, symmetric: bool, row0: int = 0, rows: int | None = None) -> Csr:
    """Matrix::read's semantics (file order, (j,i) mirrored when symmetric, later writes win) as
    CSR of rows [row0, row0+rows): every stored cell, explicit zeros included."""
    rows = n - row0 if rows is None else rows
    irn = np.asarray(irn, dtype=np.int64)
    jcn = np.asarray(jcn, dtype=np.int64)
    val = np.asarray(val, dtype=np.float64)
    if symmetric:   # write sequence 2z (A(i,j)), 2z+1 (A(j,i))
        ri = np.stack([irn, jcn], axis=1).ravel()
        ci = np.stack([jcn, irn], axis=1).ravel()
        vv = np.repeat(val, 2)
    else:
        ri, ci, vv = irn, jcn, val
    sel = (ri >= row0) & (ri < row0 + rows)
    ri, ci, vv = ri[sel] - row0, ci[sel], vv[sel]
    key = ri * n + ci
    order = np.argsort(key, kind="stable")
    key, vv = key[order], vv[order]
    last = np.ones(key.size, dtype=bool)
    last[:-1] = key[1:] != key[:-1]
    key, vv = key[last], vv[last]
    rp = np.searchsorted(key, np.arange(rows + 1) * n).astype(np.int64)
    return Csr(n, rp, (key % n).astype(np.int32), np.ascontiguousarray(vv))


def _mat(m: Csr):
    return _ci(m.rp, np.int64, _i64p), _ci(m.col, np.int32, _i32p), _p(m.val)


def gemv_csr(m: Csr, p: np.ndarray) -> np.ndarray:
    y = np.empty(m.rows, dtype=np.float64)
    lib().cso_gemv(m.rows, *_mat(m), _p(p), _p(y))
    return y


def solve_csr(m: Csr, b: np.ndarray, x0: np.ndarray | None = None, max_iter: int | None = None,
              tol: float = 1e-10) -> oracle.SolveResult:
    """oracle.solve over CSR storage: the same statements, O(nnz) per mat-vec."""
    n = m.n
    assert m.rows == n
    max_iter = n if max_iter is None else max_iter
    x = np.zeros(n, dtype=np.float64) if x0 is None else np.array(x0, dtype=np.float64)
    hist = np.zeros(max(max_iter, 1), dtype=np.float64)
    info = oracle._Info()
    lib().cso_solve(n, *_mat(m), _p(b), _p(x), max_iter, tol, _p(hist), C.byref(info))
    executed = min(info.k + (1 if info.converged else 0), max_iter)
    return oracle.SolveResult(x, info.k, bool(info.converged), info.rsold, info.rsnew, info.norm_x,
                              info.rel_resid, hist[:executed].copy())


def residual_check_csr(m: Csr, b: np.ndarray, x: np.ndarray):
    nx, rr = C.c_double(), C.c_double()
    lib().cso_residual_check(m.n, *_mat(m), _p(b), _p(x), C.byref(nx), C.byref(rr))
    return nx.value, rr.value
