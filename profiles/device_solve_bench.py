"""Device solves against host solves on one context, for a caller whose b and x live on the GPU.

    python profiles/device_solve_bench.py [--out DIR] [--repeats R]

Per case (lap2d; dense N = 40 000 on the default persistent schedule, CSR at N = 1 M and 16 M):
  short  warm-started solves: `--short-iters` iterations (tol = 0) from the previous solve's x, back to
         back.  host: b and x to the host (.cpu()), cgb_set_rhs + cgb_solve, x back to the GPU -- the copies
         a GPU-resident caller pays with the host API.  device: solve_device on the current stream, one
         synchronisation after the whole batch.  Reported as solves per second, end to end.
  long   one solve of `--long-iters` iterations (tol = 0) from x = 0: iterations per second.
The host and device API alternate on one context in every repeat.  One JSON line per measurement goes to
stdout and to DIR/device_solve_bench.jsonl, after a line with the card's name, power limit and clocks.
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card():
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (s.strip() for s in out.stdout.strip().splitlines()[0].split(","))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--short-iters", type=int, default=20)
    ap.add_argument("--short-solves", type=int, default=50)
    ap.add_argument("--long-iters", type=int, default=1000)
    ap.add_argument("--cases", default="dense:40000,csr:1000000,csr:16000000")
    args = ap.parse_args()
    import torch
    cgb = importlib.import_module("conjugate-gradient_b200")
    if not torch.cuda.is_available() or cgb.device_count() == 0:
        raise SystemExit("no GPU: nothing to measure")
    sink = open(os.path.join(args.out, "device_solve_bench.jsonl"), "w") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if sink:
            sink.write(line + "\n")
            sink.flush()

    emit({"card": card()})
    for case in args.cases.split(","):
        storage, n = case.split(":")
        n = int(n)
        with cgb.Context(n, storage=storage) as ctx:
            ctx.generate_lap2d()
            b = torch.tensor(cgb.init_source_term(n), device="cuda:0")
            x = torch.zeros(n, dtype=torch.float64, device="cuda:0")
            info = {"case": case, "schedule_in_use": ctx.get_option("schedule_in_use")}

            def host(iters):
                bh = b.cpu().numpy()
                ctx.set_rhs(bh)
                xh = x.cpu().numpy()
                ctx.solve(xh, max_iter=iters, tol=0.0)
                x.copy_(torch.from_numpy(xh))

            def device(iters):
                ctx.solve_device(x, b, iters, tol=0.0)

            def timed(fn, iters, solves):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                for _ in range(solves):
                    fn(iters)
                torch.cuda.synchronize()
                return time.perf_counter() - t0

            for api in (host, device):   # warm-up: graphs, buffers, first launches
                timed(api, args.short_iters, 2)
                x.zero_()
                timed(api, args.long_iters, 1)
            info["device_loop_pdl"] = ctx.get_option("device_loop_pdl")
            short = {"host": [], "device": []}
            long_ = {"host": [], "device": []}
            for _ in range(args.repeats):
                for api in (host, device):
                    x.zero_()
                    timed(api, 50, 1)    # the warm-started solves start near the solution
                    short[api.__name__].append(args.short_solves / timed(api, args.short_iters, args.short_solves))
                    x.zero_()
                    long_[api.__name__].append(args.long_iters / timed(api, args.long_iters, 1))
            for kind, res, unit in (("short", short, "solves_per_s"), ("long", long_, "it_per_s")):
                rec = dict(info, kind=kind, unit=unit,
                           iters=args.short_iters if kind == "short" else args.long_iters)
                for api in ("host", "device"):
                    rec[api] = {"median": statistics.median(res[api]), "min": min(res[api]), "max": max(res[api]),
                                "all": [round(v, 2) for v in res[api]]}
                rec["device_over_host"] = rec["device"]["median"] / rec["host"]["median"]
                emit(rec)


if __name__ == "__main__":
    main()
