"""ctypes binding of libcgb200.so (the C ABI declared in include/cgb200.h).

Plumbing only: every call goes straight to the sm_100a library.  There is no CPU fallback --
if the library is missing or no B200 is present the calls raise CgbError.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libcgb200.so")

UNIQUE_ID_BYTES = 128
EXCHANGE_BLOB_BYTES = 128
_dp = C.POINTER(C.c_double)
_i64p = C.POINTER(C.c_int64)
_i32p = C.POINTER(C.c_int32)


class CgbError(RuntimeError):
    def __init__(self, code: int, msg: str):
        super().__init__(f"cgb200 error {code}: {msg}")
        self.code = code


class Layout(C.Structure):
    _fields_ = [("n", C.c_int64), ("ld", C.c_int64), ("rows", C.c_int64), ("row0", C.c_int64),
                ("rank", C.c_int), ("world", C.c_int), ("device", C.c_int), ("nblk", C.c_int),
                ("sm_count", C.c_int), ("nchunks", C.c_int64)]


class SolveInfo(C.Structure):
    _fields_ = [("k", C.c_int64), ("converged", C.c_int), ("rsold", C.c_double),
                ("rsnew", C.c_double), ("seconds", C.c_double), ("iterations", C.c_int64)]


# every symbol include/cgb200.h declares: (name, restype, argtypes)
_CTX = C.c_void_p
SIGNATURES = [
    ("cgb_abi_version", C.c_int, []),
    ("cgb_last_error", C.c_char_p, []),
    ("cgb_device_count", C.c_int, [C.POINTER(C.c_int)]),
    ("cgb_partition", C.c_int, [C.c_int64, C.c_int, _i64p, _i64p]),
    ("cgb_create", C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(_CTX)]),
    ("cgb_create_csr", C.c_int, [C.c_int64, C.c_int, C.c_int, C.c_int, C.POINTER(_CTX)]),
    ("cgb_destroy", C.c_int, [_CTX]),
    ("cgb_comm_unique_id", C.c_int, [C.c_void_p]),
    ("cgb_comm_init", C.c_int, [_CTX, C.c_void_p]),
    ("cgb_exchange_export", C.c_int, [_CTX, C.c_void_p]),
    ("cgb_exchange_import", C.c_int, [_CTX, C.c_void_p]),
    ("cgb_generate_lap2d", C.c_int, [_CTX]),
    ("cgb_set_matrix_rows", C.c_int, [_CTX, _dp, C.c_int64, C.c_int64, C.c_int64]),
    ("cgb_set_matrix_coo", C.c_int, [_CTX, C.c_int64, _i32p, _i32p, _dp, C.c_int]),
    ("cgb_set_matrix_csr", C.c_int, [_CTX, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p]),
    ("cgb_update_matrix_values", C.c_int, [_CTX, C.c_void_p, C.c_void_p]),
    ("cgb_assemble_coo", C.c_int, [_CTX, C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_void_p]),
    ("cgb_assemble_values", C.c_int, [_CTX, C.c_void_p, C.c_void_p]),
    ("cgb_get_matrix_rows", C.c_int, [_CTX, _dp, C.c_int64, C.c_int64, C.c_int64]),
    ("cgb_init_source_term", C.c_int, [C.c_int64, C.c_double, _dp]),
    ("cgb_set_rhs", C.c_int, [_CTX, _dp]),
    ("cgb_set_option", C.c_int, [_CTX, C.c_char_p, C.c_int64]),
    ("cgb_get_option", C.c_int, [_CTX, C.c_char_p, _i64p]),
    ("cgb_gemv_variant_count", C.c_int, []),
    ("cgb_gemv_variant_name", C.c_char_p, [C.c_int]),
    ("cgb_autotune", C.c_int, [_CTX, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_float)]),
    ("cgb_get_layout", C.c_int, [_CTX, C.POINTER(Layout)]),
    ("cgb_solve", C.c_int, [_CTX, _dp, C.c_int64, C.c_double, _dp, C.POINTER(SolveInfo)]),
    ("cgb_solve_begin", C.c_int, [_CTX, _dp, C.c_int64, C.c_double, C.c_int]),
    ("cgb_iterate", C.c_int, [_CTX, C.c_int64, C.POINTER(C.c_float)]),
    ("cgb_solve_end", C.c_int, [_CTX, _dp, _dp, C.POINTER(SolveInfo)]),
    ("cgb_solve_block_begin", C.c_int, [_CTX, C.c_int, _dp, _dp, C.c_int64, C.c_double, C.c_int]),
    ("cgb_solve_block_end", C.c_int, [_CTX, _dp, _dp, C.POINTER(SolveInfo)]),
    ("cgb_solve_block", C.c_int, [_CTX, C.c_int, _dp, _dp, C.c_int64, C.c_double, _dp, C.POINTER(SolveInfo)]),
    ("cgb_solve_device", C.c_int, [_CTX, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p, C.c_void_p,
                                   C.c_void_p]),
    ("cgb_solve_block_device", C.c_int, [_CTX, C.c_int, C.c_void_p, C.c_void_p, C.c_int64, C.c_double, C.c_void_p,
                                         C.c_void_p, C.c_void_p]),
    ("cgb_residual_check", C.c_int, [_CTX, _dp, _dp]),
    ("cgb_gemv", C.c_int, [_CTX, _dp, _dp, _dp, _dp]),
    ("cgb_dot", C.c_int, [_CTX, _dp, _dp, _dp]),
    ("cgb_bench_gemv", C.c_int, [_CTX, C.c_int, C.c_int, C.POINTER(C.c_float)]),
    ("cgb_bench_read", C.c_int, [_CTX, C.c_int, C.POINTER(C.c_float)]),
    ("cgb_last_gemv_timing", C.c_int, [_CTX, C.POINTER(C.c_float), _i64p]),
    ("cgb_launch_count", C.c_int, [_CTX, _i64p]),
    ("cgb_trace_read", C.c_int, [_CTX, C.c_int, C.POINTER(C.c_uint64), C.c_int64, _i64p, _i64p]),
]

_lib = None


def load():
    """Load libcgb200.so (built in-tree by __graft_entry__.build()).  Fails loudly if absent."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise CgbError(-1, f"{LIB_PATH} is missing: run `python -c 'import __graft_entry__ as g; "
                               "g.build()'` (nvcc, sm_100a). There is no CPU fallback.")
        lib = C.CDLL(LIB_PATH, mode=C.RTLD_GLOBAL)
        for name, res, args in SIGNATURES:
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def _check(rc: int):
    if rc != 0:
        raise CgbError(rc, load().cgb_last_error().decode("utf-8", "replace"))


def _p(a):
    if a is None:
        return None
    assert isinstance(a, np.ndarray) and a.dtype == np.float64 and a.flags["C_CONTIGUOUS"], \
        "expected a C-contiguous float64 array"
    return a.ctypes.data_as(_dp)


def device_count() -> int:
    n = C.c_int(0)
    _check(load().cgb_device_count(C.byref(n)))
    return n.value


def partition(n: int, psize: int):
    s = (C.c_int64 * psize)()
    c = (C.c_int64 * psize)()
    _check(load().cgb_partition(n, psize, s, c))
    return list(s), list(c)


def init_source_term(n: int, h: float | None = None, out: np.ndarray | None = None) -> np.ndarray:
    """b of CGSolver::init_source_term (host libm loop inside the library, as in the reference)."""
    b = np.empty(n, dtype=np.float64) if out is None else out
    _check(load().cgb_init_source_term(n, (1.0 / n) if h is None else h, _p(b)))
    return b


def unique_id() -> bytes:
    buf = C.create_string_buffer(UNIQUE_ID_BYTES)
    _check(load().cgb_comm_unique_id(buf))
    return buf.raw


def gemv_variants():
    lib = load()
    return [lib.cgb_gemv_variant_name(i).decode() for i in range(lib.cgb_gemv_variant_count())]


class DeviceSolve:
    """A solve enqueued by Context.solve_device / solve_block_device.  The caller's x (X) tensor
    receives the solution when `stream` gets there; result() waits for that and decodes the device
    info (and history) the way the host methods return them."""

    def __init__(self, stream, info, hist, nrhs, block, keep):
        self.stream = stream
        self.info = info        # device tensor: nrhs cgb_solve_info records (uint8)
        self.hist = hist        # device tensor (nrhs, max(max_iter, 1)) or None
        self._nrhs, self._block = nrhs, block
        self._keep = keep       # the caller's tensors stay alive until result()

    def result(self):
        """single: (SolveInfo, hist or None); block: (list of SolveInfo, list of histories or None)"""
        self.stream.synchronize()
        infos = list((SolveInfo * self._nrhs).from_buffer_copy(self.info.cpu().numpy().tobytes()))
        hist = None
        if self.hist is not None:
            h = self.hist.cpu().numpy()
            hist = [h[j, :infos[j].iterations].copy() for j in range(self._nrhs)]
        self._keep = None
        if self._block:
            return infos, hist
        return infos[0], (hist[0] if hist is not None else None)


class Context:
    """One rank (= one GPU, one row shard).  Thin object wrapper over cgb_ctx*.

    storage="dense" holds the shard as rows x ld doubles (cgb_create), storage="csr" as CSR
    (cgb_create_csr): bitwise the same results, memory bounded by the non-zeros."""

    _CREATE = {"dense": "cgb_create", "csr": "cgb_create_csr"}

    def __init__(self, n: int, rank: int = 0, world: int = 1, device: int = 0, storage: str = "dense"):
        if storage not in self._CREATE:
            raise ValueError(f"storage must be 'dense' or 'csr', not {storage!r}")
        self._lib = load()
        self._h = _CTX()
        _check(getattr(self._lib, self._CREATE[storage])(n, rank, world, device, C.byref(self._h)))
        self.n = n
        self.storage = storage

    def close(self):
        if getattr(self, "_h", None):
            self._lib.cgb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def __enter__(self):
        return self

    def __exit__(self, *exc):
        self.close()

    # -- wiring
    def comm_init(self, uid: bytes):
        buf = C.create_string_buffer(uid, UNIQUE_ID_BYTES)
        _check(self._lib.cgb_comm_init(self._h, buf))

    def exchange_export(self) -> bytes:
        buf = C.create_string_buffer(EXCHANGE_BLOB_BYTES)
        _check(self._lib.cgb_exchange_export(self._h, buf))
        return buf.raw

    def exchange_import(self, blobs):
        """blobs: one exchange_export() result per rank, in rank order."""
        raw = b"".join(blobs)
        assert len(raw) == EXCHANGE_BLOB_BYTES * len(blobs)
        buf = C.create_string_buffer(raw, len(raw))
        _check(self._lib.cgb_exchange_import(self._h, buf))

    def layout(self) -> Layout:
        lay = Layout()
        _check(self._lib.cgb_get_layout(self._h, C.byref(lay)))
        return lay

    def set_option(self, key: str, value: int):
        _check(self._lib.cgb_set_option(self._h, key.encode(), int(value)))

    def get_option(self, key: str) -> int:
        v = C.c_int64()
        _check(self._lib.cgb_get_option(self._h, key.encode(), C.byref(v)))
        return v.value

    def nnz(self) -> int:
        """Entries stored in this rank's shard (CSR storage; 0 for a dense context)."""
        return self.get_option("nnz")

    def autotune(self, iters: int = 0) -> dict:
        """One-off tile-shape selection (cgb_autotune); returns the choice and every candidate's time."""
        names = gemv_variants()
        chosen = C.c_int(-1)
        us = (C.c_float * len(names))()
        _check(self._lib.cgb_autotune(self._h, iters, C.byref(chosen), us))
        return {"chosen": names[chosen.value],
                "us_per_iteration": {nm: round(float(t), 2) for nm, t in zip(names, us) if t >= 0}}

    # -- inputs
    def generate_lap2d(self):
        _check(self._lib.cgb_generate_lap2d(self._h))

    def set_matrix_rows(self, rows: np.ndarray, first_row: int = 0):
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        _check(self._lib.cgb_set_matrix_rows(self._h, _p(rows), first_row, rows.shape[0], rows.shape[1]))

    def set_matrix_coo(self, irn, jcn, val, symmetric: bool):
        irn = np.ascontiguousarray(irn, dtype=np.int32)
        jcn = np.ascontiguousarray(jcn, dtype=np.int32)
        val = np.ascontiguousarray(val, dtype=np.float64)
        _check(self._lib.cgb_set_matrix_coo(self._h, irn.size, irn.ctypes.data_as(_i32p),
                                            jcn.ctypes.data_as(_i32p), _p(val), int(bool(symmetric))))

    def set_matrix_csr(self, A, stream=None):
        """cgb_set_matrix_csr from the full n x n matrix on the GPU: a CUDA torch.sparse_csr_tensor of float64
        or a (crow, col, val) tuple of CUDA tensors, crow and col both int32 or both int64.  This rank's rows
        are passed on `stream` (default: the current torch stream); the call returns with the matrix built."""
        import torch
        if isinstance(A, torch.Tensor):
            if A.layout != torch.sparse_csr:
                raise TypeError("A must be a torch.sparse_csr_tensor or a (crow, col, val) tuple")
            if tuple(A.shape) != (self.n, self.n):
                raise ValueError(f"A is {tuple(A.shape)}, the context {self.n} x {self.n}")
            crow, col, val = A.crow_indices(), A.col_indices(), A.values()
        else:
            crow, col, val = A
        torch, dev, stream = self._device_args([("val", val)], stream)
        for nm, t in (("crow", crow), ("col", col)):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype in (torch.int32, torch.int64)
                    and t.is_contiguous()):
                raise TypeError(f"{nm} must be a contiguous int32 or int64 CUDA tensor")
            if t.device.index != dev:
                raise ValueError(f"{nm} is on cuda:{t.device.index}, the context on cuda:{dev}")
        if crow.dtype != col.dtype:
            raise TypeError("crow and col must share one index dtype")
        if crow.numel() != self.n + 1:
            raise ValueError(f"crow has {crow.numel()} entries, the full matrix n + 1 = {self.n + 1}")
        lay = self.layout()
        with torch.cuda.stream(stream):
            rp = crow[lay.row0:lay.row0 + lay.rows + 1].to(torch.int64)
            base, end = (int(v) for v in rp[[0, -1]].cpu())   # a synchronisation: the call makes one anyway
            if not 0 <= base <= end <= min(col.numel(), val.numel()):
                raise ValueError(f"crow[{lay.row0}] = {base} and crow[{lay.row0 + lay.rows}] = {end} do not "
                                 f"delimit this rank's entries of col / val")
            cols = col[base:end]
            if cols.dtype != torch.int32:
                cols = cols.clamp(-1, self.n).to(torch.int32)   # a column out of range stays out of range
            vals = val[base:end]
            _check(self._lib.cgb_set_matrix_csr(self._h, rp.data_ptr(), cols.data_ptr(), vals.data_ptr(),
                                                end - base, stream.cuda_stream))

    def update_matrix_values(self, val, stream=None):
        """cgb_update_matrix_values: new values (the first nnz() entries of the float64 CUDA tensor `val`, in
        stored order) for this CSR context's matrix, enqueued on `stream`; returns at once."""
        torch, dev, stream = self._device_args([("val", val)], stream)
        nnz = self.nnz()
        if val.numel() < nnz:
            raise ValueError(f"val has {val.numel()} entries, the matrix {nnz}")
        _check(self._lib.cgb_update_matrix_values(self._h, val.data_ptr(), stream.cuda_stream))
        val.record_stream(stream)   # its memory is not handed out again before `stream` has passed the copy

    def assemble_coo(self, coo, symmetric: bool = False, stream=None):
        """cgb_assemble_coo: the matrix as the sum of COO contributions on the GPU -- an uncoalesced CUDA
        torch.sparse_coo_tensor of float64 (its entries read in stored order; it is never coalesced, which would
        reorder them) or a (rows, cols, vals) tuple of CUDA tensors, indices int32 or int64.  Duplicates are
        added in entry order (see include/cgb200.h).  Runs on `stream` (default: the current torch stream) and
        returns with the matrix built."""
        import torch
        if isinstance(coo, torch.Tensor):
            if coo.layout != torch.sparse_coo:
                raise TypeError("coo must be a torch.sparse_coo_tensor or a (rows, cols, vals) tuple")
            if tuple(coo.shape) != (self.n, self.n):
                raise ValueError(f"coo is {tuple(coo.shape)}, the context {self.n} x {self.n}")
            idx = coo._indices()
            rows, cols, vals = idx[0], idx[1], coo._values()
        else:
            rows, cols, vals = coo
        torch, dev, stream = self._device_args([("vals", vals)], stream)
        nz = vals.numel()
        for nm, t in (("rows", rows), ("cols", cols)):
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype in (torch.int32, torch.int64)):
                raise TypeError(f"{nm} must be an int32 or int64 CUDA tensor")
            if t.device.index != dev:
                raise ValueError(f"{nm} is on cuda:{t.device.index}, the context on cuda:{dev}")
            if t.numel() != nz:
                raise ValueError(f"{nm} has {t.numel()} entries, vals {nz}")
        with torch.cuda.stream(stream):
            # an index out of range stays out of range, and is refused by the library
            irn, jcn = (t.contiguous() if t.dtype == torch.int32 else t.clamp(-1, self.n).to(torch.int32)
                        for t in (rows, cols))
            _check(self._lib.cgb_assemble_coo(self._h, nz, irn.data_ptr(), jcn.data_ptr(), vals.data_ptr(),
                                              int(bool(symmetric)), stream.cuda_stream))
        self._assembled_nz = nz

    def assemble_values(self, vals, stream=None):
        """cgb_assemble_values: new contributions (the float64 CUDA tensor `vals`, in the entry order of the last
        assemble_coo) folded into the matrix with its pattern and fold order, enqueued on `stream`; returns at
        once."""
        torch, dev, stream = self._device_args([("vals", vals)], stream)
        nz = getattr(self, "_assembled_nz", 0)
        if vals.numel() < nz:
            raise ValueError(f"vals has {vals.numel()} entries, the assembly {nz}")
        _check(self._lib.cgb_assemble_values(self._h, vals.data_ptr(), stream.cuda_stream))
        vals.record_stream(stream)   # its memory is not handed out again before `stream` has passed the fold

    def get_matrix_rows(self, first_row: int, nrows: int) -> np.ndarray:
        out = np.empty((nrows, self.n), dtype=np.float64)
        _check(self._lib.cgb_get_matrix_rows(self._h, _p(out), first_row, nrows, self.n))
        return out

    def set_rhs(self, b: np.ndarray):
        b = np.ascontiguousarray(b, dtype=np.float64)
        assert b.size == self.n
        _check(self._lib.cgb_set_rhs(self._h, _p(b)))

    # -- solve
    def solve(self, x: np.ndarray, max_iter: int, tol: float = 1e-10, history: bool = False):
        assert x.dtype == np.float64 and x.size == self.n and x.flags["C_CONTIGUOUS"]
        hist = np.zeros(max(max_iter, 1), dtype=np.float64) if history else None
        info = SolveInfo()
        _check(self._lib.cgb_solve(self._h, _p(x), max_iter, tol, _p(hist), C.byref(info)))
        return info, (hist[:info.iterations].copy() if history else None)

    def solve_begin(self, x0, max_iter: int, tol: float = 1e-10, history: bool = False):
        _check(self._lib.cgb_solve_begin(self._h, _p(x0), max_iter, tol, int(history)))

    def iterate(self, iters: int) -> float:
        ms = C.c_float()
        _check(self._lib.cgb_iterate(self._h, iters, C.byref(ms)))
        return ms.value

    def solve_end(self, x=None, hist=None) -> SolveInfo:
        info = SolveInfo()
        _check(self._lib.cgb_solve_end(self._h, _p(x), _p(hist), C.byref(info)))
        return info

    # -- block solve (CSR, one rank): column j bit for bit the single solve of A x = B[j] from X0[j]
    def _block_inputs(self, B, X0):
        B = np.ascontiguousarray(B, dtype=np.float64)
        assert B.ndim == 2 and B.shape[1] == self.n, "B must be (nrhs, n)"
        X = np.zeros_like(B) if X0 is None else np.array(X0, dtype=np.float64, order="C")
        assert X.shape == B.shape
        return B, X

    def solve_block(self, B, X0=None, max_iter: int = 0, tol: float = 1e-10, history: bool = False):
        """B: (nrhs, n) right-hand sides; returns (X, infos, hist) -- X (nrhs, n), one SolveInfo per
        column, and (history=True) a list of each column's r'r history, else None."""
        B, X = self._block_inputs(B, X0)
        nrhs = B.shape[0]
        hist = np.zeros((nrhs, max(max_iter, 1)), dtype=np.float64) if history else None
        infos = (SolveInfo * nrhs)()
        _check(self._lib.cgb_solve_block(self._h, nrhs, _p(B), _p(X), max_iter, tol, _p(hist), infos))
        return X, list(infos), self._block_hist(hist, infos)

    def solve_block_begin(self, B, X0=None, max_iter: int = 0, tol: float = 1e-10, history: bool = False):
        B, X0 = self._block_inputs(B, X0)
        self._block = (B.shape[0], max_iter, history)
        _check(self._lib.cgb_solve_block_begin(self._h, B.shape[0], _p(B), _p(X0), max_iter, tol, int(history)))

    def solve_block_end(self):
        """(X, infos, hist) of the block solve begun with solve_block_begin (advanced by iterate)."""
        nrhs, max_iter, history = self._block
        X = np.empty((nrhs, self.n), dtype=np.float64)
        hist = np.zeros((nrhs, max(max_iter, 1)), dtype=np.float64) if history else None
        infos = (SolveInfo * nrhs)()
        _check(self._lib.cgb_solve_block_end(self._h, _p(X), _p(hist), infos))
        return X, list(infos), self._block_hist(hist, infos)

    @staticmethod
    def _block_hist(hist, infos):
        return None if hist is None else [hist[j, :infos[j].iterations].copy() for j in range(len(infos))]

    # -- device solves: CUDA tensors in and out, ordered on a torch stream, no host round trip
    def _device_args(self, tensors, stream):
        import torch
        dev = self.layout().device
        for nm, t in tensors:
            if not (isinstance(t, torch.Tensor) and t.is_cuda and t.dtype == torch.float64 and t.is_contiguous()):
                raise TypeError(f"{nm} must be a contiguous float64 CUDA tensor")
            if t.device.index != dev:
                raise ValueError(f"{nm} is on cuda:{t.device.index}, the context on cuda:{dev}")
        stream = torch.cuda.current_stream(dev) if stream is None else stream
        return torch, dev, stream

    def solve_device(self, x, b, max_iter: int, tol: float = 1e-10, history: bool = False, stream=None):
        """cgb_solve_device: x (x0 in, the solution out) and b are (n,) float64 CUDA tensors; the solve
        is enqueued on `stream` (default: the current torch stream) and the call returns at once."""
        torch, dev, stream = self._device_args([("x", x), ("b", b)], stream)
        assert x.numel() == self.n and b.numel() == self.n
        info = torch.zeros(C.sizeof(SolveInfo), dtype=torch.uint8, device=f"cuda:{dev}")
        hist = torch.zeros((1, max(max_iter, 1)), dtype=torch.float64, device=f"cuda:{dev}") if history else None
        _check(self._lib.cgb_solve_device(self._h, b.data_ptr(), x.data_ptr(), max_iter, tol,
                                          hist.data_ptr() if history else None, info.data_ptr(),
                                          stream.cuda_stream))
        return DeviceSolve(stream, info, hist, 1, False, (x, b))

    def solve_block_device(self, X, B, max_iter: int = 0, tol: float = 1e-10, history: bool = False, stream=None):
        """cgb_solve_block_device: X (X0 in, the solutions out) and B are (nrhs, n) float64 CUDA tensors."""
        torch, dev, stream = self._device_args([("X", X), ("B", B)], stream)
        assert B.ndim == 2 and B.shape[1] == self.n and X.shape == B.shape, "B and X must be (nrhs, n)"
        nrhs = B.shape[0]
        info = torch.zeros(max(nrhs, 1) * C.sizeof(SolveInfo), dtype=torch.uint8, device=f"cuda:{dev}")
        hist = torch.zeros((max(nrhs, 1), max(max_iter, 1)), dtype=torch.float64, device=f"cuda:{dev}") \
            if history else None
        _check(self._lib.cgb_solve_block_device(self._h, nrhs, B.data_ptr(), X.data_ptr(), max_iter, tol,
                                                hist.data_ptr() if history else None, info.data_ptr(),
                                                stream.cuda_stream))
        return DeviceSolve(stream, info, hist, nrhs, True, (X, B))

    def residual_check(self):
        nx, rr = C.c_double(), C.c_double()
        _check(self._lib.cgb_residual_check(self._h, C.byref(nx), C.byref(rr)))
        return nx.value, rr.value

    # -- kernel-level hooks
    def gemv(self, v: np.ndarray, want_partials: bool = False):
        lay = self.layout()
        y = np.empty(lay.rows, dtype=np.float64)
        bp = np.empty(lay.nchunks, dtype=np.float64) if want_partials else None   # chunk partials of v.(A v)
        pap = C.c_double()
        v = np.ascontiguousarray(v, dtype=np.float64)
        _check(self._lib.cgb_gemv(self._h, _p(v), _p(y), _p(bp), C.byref(pap)))
        return (y, bp, pap.value) if want_partials else (y, pap.value)

    def dot(self, a: np.ndarray, b: np.ndarray) -> float:
        out = C.c_double()
        _check(self._lib.cgb_dot(self._h, _p(np.ascontiguousarray(a)), _p(np.ascontiguousarray(b)),
                                 C.byref(out)))
        return out.value

    def bench_gemv(self, variant: int = -1, reps: int = 10) -> float:
        ms = C.c_float()
        _check(self._lib.cgb_bench_gemv(self._h, variant, reps, C.byref(ms)))
        return ms.value

    def bench_read(self, reps: int = 10) -> float:
        ms = C.c_float()
        _check(self._lib.cgb_bench_read(self._h, reps, C.byref(ms)))
        return ms.value

    def last_gemv_timing(self):
        ms, n = C.c_float(), C.c_int64()
        _check(self._lib.cgb_last_gemv_timing(self._h, C.byref(ms), C.byref(n)))
        return ms.value, n.value

    def trace_read(self, which: int):
        """(records[L, blocks, 8] uint64 in launch order, launches seen) of the diagnostic
        timeline of kernel `which` (0 mat-vec, 1 update_xr, 2 update_p); option "trace" = L."""
        cap = self.get_option("trace")
        lay = self.layout()
        nb = lay.nblk if which == 0 else lay.nchunks
        buf = np.zeros(cap * nb * 8, dtype=np.uint64)
        seen, blocks = C.c_int64(), C.c_int64()
        _check(self._lib.cgb_trace_read(self._h, which, buf.ctypes.data_as(C.POINTER(C.c_uint64)),
                                        buf.size, C.byref(seen), C.byref(blocks)))
        rec = buf.reshape(cap, blocks.value, 8)
        n = seen.value
        if n >= cap:   # ring: oldest kept launch first
            rec = np.roll(rec, -(n % cap), axis=0)
        else:
            rec = rec[:n]
        return rec, n

    def launch_count(self) -> int:
        n = C.c_int64()
        _check(self._lib.cgb_launch_count(self._h, C.byref(n)))
        return n.value
