"""CSR storage on one GPU: the lap2d system at N in {40 000, 1 M, 4 M, 16 M}, one JSON line per N.

  it_per_s / ms_per_iter : cgb_iterate batches with the solve state resident on the device
                           (cgb_solve_begin outside the timed region, tol = 0 so that no batch stops
                           early), device-timed like bench.py's `value`
  bytes_per_iter         : algorithmic traffic from the shapes -- the CSR arrays once (8 B row
                           pointer, 4 B column, 8 B value) plus every vector read and write of the
                           four kernels of an iteration (see traffic())
  spmv_ms / read_ms      : the CSR mat-vec alone (cgb_bench_gemv) against a plain stream over the
                           same CSR arrays (cgb_bench_read)
  digest                 : N = 40 000 x 200 iterations (b = init_source_term(1/N), x0 = 0, tol 1e-10),
                           computed like bench.py's parity_check; DESIGN.md records 1b58205beac19aa4

The 4 M and 16 M inputs (CSR arrays of ~0.24 GB and ~0.96 GB, vectors of 32 / 128 MB each) exceed
the 126 MB L2, so their passes stream from HBM; the two smaller ones are partly L2-resident.

    python profiles/sparse_bench.py [--sizes 40000,1000000] [--out DIR]
"""
import argparse
import hashlib
import importlib
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
L2_BYTES = 126 * 2**20


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def traffic(n, nnz):
    """bytes one iteration moves at least: CSR arrays once + vectors (8 B each element)"""
    csr = 8 * (n + 1) + 4 * nnz + 8 * nnz
    spmv = csr + 8 * n + 8 * n                  # p gathered (each element at least once), Ap written
    pap = 16 * n                                # p, Ap
    xr = 48 * n                                 # read x p Ap r, write x r
    p = 24 * n                                  # read p r, write p
    return csr, spmv + pap + xr + p


def digest(cgb, n=40000, iters=200):
    b = cgb.init_source_term(n)
    with cgb.Context(n, storage="csr") as ctx:
        ctx.generate_lap2d()
        ctx.set_rhs(b)
        x = np.zeros(n)
        info, hist = ctx.solve(x, max_iter=iters, tol=1e-10, history=True)
        nx, rr = ctx.residual_check()
    return hashlib.sha256(x.tobytes() + hist.tobytes() + np.array([nx, rr]).tobytes()).hexdigest()[:16]


def measure(cgb, n, steps, batch, warmup):
    with cgb.Context(n, storage="csr") as ctx:
        ctx.generate_lap2d()
        ctx.set_rhs(cgb.init_source_term(n))
        nnz = ctx.nnz()
        ctx.solve_begin(None, (warmup + steps) * batch, 0.0, False)
        for _ in range(warmup):
            ctx.iterate(batch)
        ms = sum(ctx.iterate(batch) for _ in range(steps))
        ctx.solve_end(None, None)
        spmv_ms = ctx.bench_gemv(reps=50)
        read_ms = ctx.bench_read(reps=50)
    it = steps * batch
    csr_bytes, per_iter = traffic(n, nnz)
    return {
        "n": n, "nnz": nnz, "iterations_timed": it,
        "it_per_s": round(it / (ms * 1e-3), 2), "ms_per_iter": round(ms / it, 5),
        "bytes_per_iter": per_iter, "achieved_GBps": round(per_iter * it / (ms * 1e-3) / 1e9, 1),
        "csr_bytes": csr_bytes, "spmv_ms": round(spmv_ms, 5), "read_ms": round(read_ms, 5),
        "spmv_GBps_over_csr": round(csr_bytes / (spmv_ms * 1e-3) / 1e9, 1),
        "read_GBps_over_csr": round(csr_bytes / (read_ms * 1e-3) / 1e9, 1),
        "spmv_over_read_rate": round(read_ms / spmv_ms, 3),
        "exceeds_l2": csr_bytes + 4 * 8 * n > L2_BYTES,
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="40000,1000000,4000000,16000000")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="also append the lines to DIR/sparse_bench.jsonl")
    a = ap.parse_args()
    cgb = importlib.import_module("conjugate-gradient_b200")
    info = card()
    dg = digest(cgb)
    lines = []
    for n in [int(s) for s in a.sizes.split(",")]:
        r = measure(cgb, n, a.steps, a.batch, a.warmup)
        r.update(info)
        r["digest_n40000_it200"] = dg
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "sparse_bench.jsonl"), "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
