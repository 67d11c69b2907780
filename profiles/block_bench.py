"""Block solves against single solves on one GPU: lap2d (CSR storage) at N in {40 000, 1 M, 4 M, 16 M},
nrhs in {1, 2, 4, 8}, one context per N.  One JSON line per (N, nrhs).

  block_col_it_per_s  : column-iterations per second of the block solve (nrhs x loop bodies / time)
  single_it_per_s     : iterations per second of a single solve on the same context
  ratio               : median block / median single -- how much faster nrhs right-hand sides get
                        through as one block than one after another (1 / nrhs: no gain at all)
Both are cgb_iterate batches with the state resident on the device: begin outside the timed region,
tol = 0 so that no batch stops early, device time as cgb_iterate reports it.  Each repeat runs the
single solve and then every block size, so the two alternate in one process; every repeat is kept
(the lists give the spread).  The card's name and power limit are read in the same run.

    python profiles/block_bench.py [--sizes 40000,1000000] [--nrhs 1,2,4,8] [--out DIR]
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def timed(ctx, begin, end, steps, batch):
    """ms of `steps` batches of `batch` loop bodies after one warm-up batch"""
    begin((steps + 1) * batch)
    ctx.iterate(batch)
    ms = sum(ctx.iterate(batch) for _ in range(steps))
    end()
    return ms


def measure(cgb, n, nrhs_list, steps, batch, repeats):
    B = np.array([cgb.init_source_term(n, h / n) for h in (1.0, 0.37, 0.11, 0.73, 0.5, 0.29, 0.61, 0.83)])
    single, block = [], {r: [] for r in nrhs_list}
    with cgb.Context(n, storage="csr") as ctx:
        ctx.generate_lap2d()
        ctx.set_rhs(B[0])
        for _ in range(repeats):
            ms = timed(ctx, lambda it: ctx.solve_begin(None, it, 0.0), lambda: ctx.solve_end(), steps, batch)
            single.append(steps * batch / (ms * 1e-3))
            for r in nrhs_list:
                ms = timed(ctx, lambda it: ctx.solve_block_begin(B[:r], None, it, 0.0), ctx.solve_block_end,
                           steps, batch)
                block[r].append(r * steps * batch / (ms * 1e-3))
        nnz = ctx.nnz()
    s_med = statistics.median(single)
    for r in nrhs_list:
        b_med = statistics.median(block[r])
        yield {"n": n, "nnz": nnz, "nrhs": r, "iterations_per_run": steps * batch, "repeats": repeats,
               "block_col_it_per_s": round(b_med, 1), "single_it_per_s": round(s_med, 1),
               "ratio": round(b_med / s_med, 3),
               "block_col_it_per_s_all": [round(v, 1) for v in block[r]],
               "single_it_per_s_all": [round(v, 1) for v in single],
               "us_per_block_iteration": round(r / b_med * 1e6, 2), "us_per_single_iteration": round(1e6 / s_med, 2)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sizes", default="40000,1000000,4000000,16000000")
    ap.add_argument("--nrhs", default="1,2,4,8")
    ap.add_argument("--steps", type=int, default=8)
    ap.add_argument("--batch", type=int, default=64)
    ap.add_argument("--repeats", type=int, default=3)
    ap.add_argument("--out", default=None, help="also append the lines to DIR/block_bench.jsonl")
    a = ap.parse_args()
    cgb = importlib.import_module("conjugate-gradient_b200")
    info = card()
    nrhs_list = [int(s) for s in a.nrhs.split(",")]
    lines = []
    for n in [int(s) for s in a.sizes.split(",")]:
        for r in measure(cgb, n, nrhs_list, a.steps, a.batch, a.repeats):
            r.update(info)
            lines.append(json.dumps(r))
            print(lines[-1], flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "block_bench.jsonl"), "a") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
