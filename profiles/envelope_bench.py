"""Column-windowed dense mat-vec against the parent commit's full-row stream, one GPU.

The parent's libcgb200.so is cross-compiled from the parent commit into profiles/_parent/ (git-ignored):

    git archive <parent> conjugate-gradient_b200/csrc include | tar -x -C /tmp/p
    make -C /tmp/p/conjugate-gradient_b200/csrc && mkdir -p profiles/_parent
    cp /tmp/p/conjugate-gradient_b200/libcgb200.so profiles/_parent/

Every measurement runs in a process of its own (the library is bound once per process through
_capi.LIB_PATH); the builds alternate, case by case, round by round, so both see the same machine.

Cases (the persistent schedule unless --schedule 0 selects the graph schedule, tol = 0 so no batch
stops early, device-timed cgb_iterate batches with the solve state resident, as bench.py's `value`):
  lap40k / lap20k : generate_lap2d at N = 40 000 / 20 000 (bench.py's system and --workload weak)
  dense20k        : a seeded, diagonally dominant, symmetric matrix with every entry non-zero at
                    N = 20 000 through set_matrix_rows: every window is [0, ld), the windowed stream
                    must be today's stream -- new against parent within the spread of repeats
Per line: it/s, us per iteration, "envelope_doubles", the windowed bytes of one mat-vec from the block
geometry of the static partition (A rows + p slice per block, tma_w8r2c512s3, 148 CTAs; the
persistent kernel re-balances rows, which moves these by a few blocks' worth), that over the time,
and a digest of x + r'r history of a 200-iteration (dense: 50) solve, to show both builds agree.

    python profiles/envelope_bench.py [--rounds 3] [--schedule 1] [--out DIR]
"""
import argparse
import hashlib
import importlib
import json
import math
import os
import statistics
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARENT_LIB = os.path.join(ROOT, "profiles", "_parent", "libcgb200.so")
PEAK_BPS = 7.7e12   # HBM3e, HGX B200 data sheet, one GPU
CASES = {"lap40k": 40000, "lap20k": 20000, "dense20k": 20000}


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def lap2d_env(i, n):
    inc = int(math.floor(math.sqrt(n)))
    c = [i]
    if i > inc:
        c.append(i - 1 - inc)
    if i > 0:
        c.append(i - 1)
    if i < n - 1:
        c.append(i + 1)
    if i < n - 1 - inc:
        c.append(i + 1 + inc)
    return min(c), max(c) + 1


def windowed_bytes(n, env, nblk=148, TR=16):
    """A rows + p slice of every block window of one mat-vec (static partition, 1 GPU)."""
    ld = (n + 15) // 16 * 16
    tot = 0
    for c in range(nblk):
        r0, r1 = c * n // nblk, (c + 1) * n // nblk
        nb = (r1 - r0 + TR - 1) // TR
        for b in range(nb):
            a0, a1 = r0 + b * (r1 - r0) // nb, r0 + (b + 1) * (r1 - r0) // nb
            lo = min(env(i)[0] for i in range(a0, a1)) // 64 * 64
            hi = min(ld, (max(env(i)[1] for i in range(a0, a1)) + 15) // 16 * 16)
            tot += 8 * (a1 - a0 + 1) * (hi - lo)
    return tot


def dense_rows(n, r0, r1, seed=7):
    """rows [r0, r1) of a symmetric matrix with every entry non-zero, strictly diagonally dominant"""
    ph = np.random.default_rng(seed).uniform(0, 2 * np.pi)
    i = np.arange(r0, r1, dtype=np.float64)[:, None]
    j = np.arange(n, dtype=np.float64)[None, :]
    M = 1e-3 * (1.5 + np.sin(ph + 1e-4 * (i + j)) * np.cos(1e-3 * i * j))
    M[np.arange(r1 - r0), np.arange(r0, r1)] = 1.0 + 3e-3 * n
    return M


def setup(cgb, ctx, case, n):
    if case == "dense20k":
        for r0 in range(0, n, 2000):
            ctx.set_matrix_rows(dense_rows(n, r0, min(n, r0 + 2000)), first_row=r0)
    else:
        ctx.generate_lap2d()
    ctx.set_rhs(cgb.init_source_term(n))


def worker(case, batch, min_ms, schedule):
    cgb = importlib.import_module("conjugate-gradient_b200")
    n = CASES[case]
    with cgb.Context(n, 0, 1, 0) as ctx:
        setup(cgb, ctx, case, n)
        ctx.set_option("schedule", schedule)
        ctx_schedule = ctx.get_option("schedule_in_use")
        try:
            envd = ctx.get_option("envelope_doubles")
        except cgb.CgbError:                            # the parent build has no such option
            envd = None
        it_check = 50 if case == "dense20k" else 200
        x = np.zeros(n)
        info, hist = ctx.solve(x, max_iter=it_check, tol=1e-10, history=True)
        dg = hashlib.sha256(x.tobytes() + hist.tobytes()).hexdigest()[:16]
        ctx.solve_begin(None, 10**9, 0.0, False)
        ctx.iterate(batch)                              # warm-up (module load, first partition)
        ms = []
        while sum(ms) < min_ms or len(ms) < 3:
            ms.append(ctx.iterate(batch))
        ctx.solve_end(None, None)
    it = batch * len(ms)
    return {"case": case, "n": n, "iterations_timed": it, "ms_total": round(sum(ms), 3),
            "it_per_s": round(it / (sum(ms) * 1e-3), 1),
            "us_per_iter": round(1e3 * sum(ms) / it, 3),
            "batch_it_per_s": [round(batch / (m * 1e-3), 1) for m in ms],
            "envelope_doubles": envd, "schedule_in_use": ctx_schedule, "digest": dg}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cases", default=",".join(CASES))
    ap.add_argument("--batch", type=int, default=200)
    ap.add_argument("--min-ms", type=float, default=1000.0)
    ap.add_argument("--schedule", type=int, default=1, help="1 persistent kernel, 0 CUDA graph of 4 kernels per iteration")
    ap.add_argument("--out", default=None, help="also write DIR/envelope_bench.jsonl")
    ap.add_argument("--worker", default=None, help=argparse.SUPPRESS)
    ap.add_argument("--lib", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        sys.path.insert(0, ROOT)
        if a.lib:
            importlib.import_module("conjugate-gradient_b200._capi").LIB_PATH = a.lib
        print(json.dumps(worker(a.worker, a.batch, a.min_ms, a.schedule)), flush=True)
        return
    if not os.path.exists(PARENT_LIB):
        sys.exit(f"{PARENT_LIB} is missing (see the docstring)")
    info = card()
    cases = a.cases.split(",")
    runs = {(c, b): [] for c in cases for b in ("parent", "new")}
    for rnd in range(a.rounds):
        for c in cases:
            for build in (("parent", "new") if rnd % 2 == 0 else ("new", "parent")):
                cmd = [sys.executable, os.path.abspath(__file__), "--worker", c, "--batch", str(a.batch),
                       "--min-ms", str(a.min_ms), "--schedule", str(a.schedule)] + (["--lib", PARENT_LIB] if build == "parent" else [])
                out = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, check=True)
                r = json.loads(out.stdout.strip().splitlines()[-1])
                r.update(build=build, round=rnd)
                runs[(c, build)].append(r)
                print(json.dumps(r), flush=True)
    lines = []
    for c in cases:
        n = CASES[c]
        new, par = runs[(c, "new")], runs[(c, "parent")]
        rn, rp = [r["it_per_s"] for r in new], [r["it_per_s"] for r in par]
        if c == "dense20k":
            wb = windowed_bytes(n, lambda i: (0, n))
        else:
            wb = windowed_bytes(n, lambda i: lap2d_env(i, n))
        dense_b = 8 * n * ((n + 15) // 16 * 16)
        us = 1e6 / statistics.median(rn)
        s = {"case": c, "n": n, "schedule": a.schedule, **info,
             "new_it_per_s": rn, "parent_it_per_s": rp,
             "new_median": statistics.median(rn), "parent_median": statistics.median(rp),
             "speedup_median": round(statistics.median(rn) / statistics.median(rp), 3),
             "new_spread_pct": round(100 * (max(rn) - min(rn)) / statistics.median(rn), 2),
             "parent_spread_pct": round(100 * (max(rp) - min(rp)) / statistics.median(rp), 2),
             "us_per_iter_new": round(us, 3), "us_per_iter_parent": round(1e6 / statistics.median(rp), 3),
             "envelope_doubles": new[0]["envelope_doubles"],
             "dense_A_bytes_per_matvec": dense_b, "windowed_bytes_per_matvec": wb,
             "windowed_GBps_new": round(wb / (us * 1e-6) / 1e9, 1),
             "windowed_frac_of_7p7TBps": round(wb / (us * 1e-6) / PEAK_BPS, 3),
             "digests_equal": len({r["digest"] for r in new + par}) == 1, "digest": new[0]["digest"]}
        lines.append(json.dumps(s))
        print(lines[-1], flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "envelope_bench.jsonl"), "w") as f:
            f.write("\n".join(json.dumps(r) for v in runs.values() for r in v) + "\n")
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
