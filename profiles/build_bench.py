"""Time the matrix builders of this tree against the parent commit's, one GPU.

The parent's libcgb200.so is cross-compiled from the parent commit into profiles/_parent/ (git-ignored):

    git archive <parent> conjugate-gradient_b200/csrc include | tar -x -C /tmp/p
    make -C /tmp/p/conjugate-gradient_b200/csrc && mkdir -p profiles/_parent
    cp /tmp/p/conjugate-gradient_b200/libcgb200.so profiles/_parent/

Every build runs in a process of its own (the library is bound once per process through
_capi.LIB_PATH), and the builds alternate round by round, so both see the same machine.

Cases (each call synchronises before it returns, so a host clock around it is the call's time;
one untimed call first, then --repeats timed calls on the same context):
  lap2d_dense_40k : cgb_generate_lap2d on a dense context at N = 40 000 (bench.py's matrix)
  coo_dense_1m    : cgb_set_matrix_coo, 10^6 seeded random triples (heavy duplicates) into 1500 x 1500, dense
  coo_csr_1m      : the same triples on a CSR context
  coo_dense_1500  : 1500 seeded random triples into 1500 x 1500, dense
  coo_csr_1500    : the same on a CSR context
Per case a digest of what was built (the shard's rows for COO; x and the r'r history of a 50-iteration
solve for lap2d) shows that both builds agree.

    python profiles/build_bench.py [--rounds 4] [--repeats 5] [--out DIR]
"""
import argparse
import hashlib
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARENT_LIB = os.path.join(ROOT, "profiles", "_parent", "libcgb200.so")
CASES = ["lap2d_dense_40k", "coo_dense_1m", "coo_csr_1m", "coo_dense_1500", "coo_csr_1500"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True, timeout=60)
    name, power, clock = [s.strip() for s in q.stdout.splitlines()[0].split(",")]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def triples(nz, n=1500):
    rng = np.random.default_rng(nz)
    return (rng.integers(0, n, nz, dtype=np.int32), rng.integers(0, n, nz, dtype=np.int32),
            rng.standard_normal(nz))


def timed(fn, repeats):
    fn()                                   # module load, first allocations
    ms = []
    for _ in range(repeats):
        t0 = time.perf_counter()
        fn()
        ms.append(1e3 * (time.perf_counter() - t0))
    return ms


def run_case(cgb, case, repeats):
    if case == "lap2d_dense_40k":
        n = 40000
        with cgb.Context(n) as ctx:
            ms = timed(ctx.generate_lap2d, repeats)
            ctx.set_rhs(cgb.init_source_term(n))
            x = np.zeros(n)
            _, hist = ctx.solve(x, max_iter=50, tol=1e-10, history=True)
            digest = hashlib.sha256(x.tobytes() + hist.tobytes()).hexdigest()[:16]
        return ms, digest
    _, storage, size = case.split("_")
    n, nz = 1500, (10**6 if size == "1m" else 1500)
    irn, jcn, val = triples(nz, n)
    with cgb.Context(n, storage=storage) as ctx:
        ms = timed(lambda: ctx.set_matrix_coo(irn, jcn, val, symmetric=False), repeats)
        digest = hashlib.sha256(ctx.get_matrix_rows(0, n).tobytes()).hexdigest()[:16]
    return ms, digest


def worker(repeats):
    cgb = importlib.import_module("conjugate-gradient_b200")
    out = []
    for case in CASES:
        ms, digest = run_case(cgb, case, repeats)
        out.append({"case": case, "ms": [round(m, 3) for m in ms], "median_ms": round(statistics.median(ms), 3),
                    "digest": digest})
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--out", default=None, help="also write DIR/build_bench.jsonl")
    ap.add_argument("--worker", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--lib", default=None, help=argparse.SUPPRESS)
    a = ap.parse_args()
    if a.worker:
        sys.path.insert(0, ROOT)
        if a.lib:
            importlib.import_module("conjugate-gradient_b200._capi").LIB_PATH = a.lib
        print(json.dumps(worker(a.repeats)), flush=True)
        return
    if not os.path.exists(PARENT_LIB):
        sys.exit(f"{PARENT_LIB} is missing (see the docstring)")
    info = card()
    runs = {(c, b): [] for c in CASES for b in ("parent", "new")}
    for rnd in range(a.rounds):
        for build in (("parent", "new") if rnd % 2 == 0 else ("new", "parent")):
            cmd = [sys.executable, os.path.abspath(__file__), "--worker", "--repeats", str(a.repeats)]
            cmd += ["--lib", PARENT_LIB] if build == "parent" else []
            out = subprocess.run(cmd, capture_output=True, text=True, timeout=1800, check=True)
            for r in json.loads(out.stdout.strip().splitlines()[-1]):
                r.update(build=build, round=rnd)
                runs[(r["case"], build)].append(r)
                print(json.dumps(r), flush=True)
    lines = []
    for c in CASES:
        new, par = runs[(c, "new")], runs[(c, "parent")]
        mn, mp = [r["median_ms"] for r in new], [r["median_ms"] for r in par]
        lines.append(json.dumps({"case": c, **info, "new_median_ms": statistics.median(mn),
                                 "parent_median_ms": statistics.median(mp),
                                 "new_round_medians": mn, "parent_round_medians": mp,
                                 "digests_equal": len({r["digest"] for r in new + par}) == 1}))
        print(lines[-1], flush=True)
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "build_bench.jsonl"), "w") as f:
            f.write("\n".join(json.dumps(r) for v in runs.values() for r in v) + "\n")
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
