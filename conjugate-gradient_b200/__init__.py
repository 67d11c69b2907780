"""conjugate-gradient_b200 -- B200-native dense fp64 conjugate-gradient hot path.

The product is the sm_100a library `libcgb200.so` (csrc/, C ABI in include/cgb200.h) and the
C++ host program `cgsolver` (host/) that keeps the reference's command line, Matrix Market
reader and results-file format.  This Python package is a thin ctypes binding used by the
tests and bench.py; it never computes anything itself and has no CPU fallback.

The directory name contains a hyphen, so import it with
    importlib.import_module("conjugate-gradient_b200")
"""
from ._capi import (CgbError, Context, DeviceSolve, Layout, SolveInfo, SIGNATURES, LIB_PATH, UNIQUE_ID_BYTES, EXCHANGE_BLOB_BYTES,
                    device_count, gemv_variants, init_source_term, load, partition, unique_id)

__all__ = ["CgbError", "Context", "DeviceSolve", "Layout", "SolveInfo", "SIGNATURES", "LIB_PATH",
           "UNIQUE_ID_BYTES", "EXCHANGE_BLOB_BYTES", "device_count", "gemv_variants", "init_source_term", "load", "partition", "unique_id"]
