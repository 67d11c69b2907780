"""A time-step loop whose matrix changes every step, on a CSR context: what refreshing A costs.

    python profiles/matrix_update_bench.py [--out DIR] [--sizes 1000000,4000000] [--steps K] [--repeats R]

Workload: the lap2d pattern at each size; every step a torch kernel makes the step's values (diagonal
4 + sigma_t, off-diagonals kept) on the GPU, A is refreshed from them, and one device solve follows
(max_iter = `--iters`, tol = 0, so every solve runs the same loop).  Three arms, alternating inside every
repeat, K steps each between two CUDA events on the stream (ms per step = elapsed / K):
  update  cgb_update_matrix_values + cgb_solve_device: no host synchronisation, no recapture
  set     cgb_set_matrix_csr (device CSR, validated, copied; synchronises) + cgb_solve_device
  coo     the values downloaded (.cpu()), cgb_set_matrix_coo from the host triples + cgb_solve_device:
          what a caller with the matrix on the GPU paid before cgb_set_matrix_csr
Also the refresh alone: K back-to-back cgb_update_matrix_values against K device copies of nnz doubles
(torch copy_), same events.  After the loop, one step of each arm from the same x0 and values checks that
the three give the same x bit for bit.  One JSON line per measurement goes to stdout and to
DIR/matrix_update_bench.jsonl, after a line with the card's name, power limit and clocks.
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
    q = "name,power.limit,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader"], capture_output=True, text=True)
    return dict(zip(q.split(","), (s.strip() for s in out.stdout.strip().splitlines()[0].split(","))))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--sizes", default="1000000,4000000")
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    import torch
    cgb = importlib.import_module("conjugate-gradient_b200")
    if not torch.cuda.is_available() or cgb.device_count() == 0:
        raise SystemExit("no GPU: nothing to measure")
    sink = open(os.path.join(args.out, "matrix_update_bench.jsonl"), "w") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if sink:
            sink.write(line + "\n")
            sink.flush()

    emit({"card": card()})
    dev = "cuda:0"
    for n in (int(s) for s in args.sizes.split(",")):
        with cgb.Context(n, storage="csr") as ctx:
            ctx.generate_lap2d()
            # generate_lap2d's pattern in stored order: a set from it is the generated matrix again
            crow, col, val = lap2d_csr(torch, n, dev)
            ctx.set_matrix_csr((crow, col, val))
            nnz = ctx.nnz()
            assert nnz == val.numel()
            irn = np.repeat(np.arange(n, dtype=np.int32), np.diff(crow.cpu().numpy()))
            jcn = col.cpu().numpy().astype(np.int32)
            diag = torch.tensor(irn == jcn, device=dev)
            b = torch.tensor(cgb.init_source_term(n), device=dev)
            x = torch.zeros(n, dtype=torch.float64, device=dev)
            vals = torch.empty_like(val)
            step_no = [0]

            def values():
                t = step_no[0]
                step_no[0] += 1
                torch.where(diag, val + (0.5 + 0.01 * (t % 100)), val, out=vals)
                return vals

            def solve():
                ctx.solve_device(x, b, args.iters, tol=0.0)

            def update():
                ctx.update_matrix_values(values())
                solve()

            def set_csr():
                ctx.set_matrix_csr((crow, col, values()))
                solve()

            def coo():
                ctx.set_matrix_coo(irn, jcn, values().cpu().numpy(), symmetric=False)
                solve()

            def timed(fn, k):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize()
                e0.record()
                for _ in range(k):
                    fn()
                e1.record()
                torch.cuda.synchronize()
                return e0.elapsed_time(e1) / k

            arms = {"update": update, "set": set_csr, "coo": coo}
            for fn in arms.values():   # warm-up: graphs, buffers, first launches
                timed(fn, 2)
            res = {a: [] for a in arms}
            for _ in range(args.repeats):
                for a, fn in arms.items():
                    res[a].append(timed(fn, args.steps))
            info = {"n": n, "nnz": nnz, "iters": args.iters, "steps": args.steps,
                    "graph_captures_after": ctx.get_option("graph_captures")}
            rec = dict(info, kind="step", unit="ms_per_step")
            for a in arms:
                rec[a] = {"median": statistics.median(res[a]), "min": min(res[a]), "max": max(res[a]),
                          "all": [round(v, 4) for v in res[a]]}
            rec["set_over_update"] = rec["set"]["median"] / rec["update"]["median"]
            rec["coo_over_update"] = rec["coo"]["median"] / rec["update"]["median"]
            emit(rec)

            # the refresh alone, against a plain device copy of nnz doubles
            src, dst = val.clone(), torch.empty_like(val)
            alone = {"update": [], "copy": []}
            for _ in range(args.repeats):
                alone["update"].append(timed(lambda: ctx.update_matrix_values(src), 10 * args.steps))
                alone["copy"].append(timed(lambda: dst.copy_(src), 10 * args.steps))
            rec = dict(info, kind="refresh_alone", unit="ms_per_call", bytes=8 * nnz)
            for a, v in alone.items():
                rec[a] = {"median": statistics.median(v), "min": min(v), "max": max(v), "all": [round(t, 5) for t in v]}
                rec[a]["GB_per_s"] = 8 * nnz / (rec[a]["median"] * 1e-3) / 1e9
            emit(rec)

            # the three arms leave the same x for the same values from the same x0
            xs = {}
            for a, fn in arms.items():
                step_no[0] = 7
                x.zero_()
                fn()
                torch.cuda.synchronize()
                xs[a] = x.cpu().numpy().view(np.uint64).copy()
            emit(dict(info, kind="check", same_x_bits=bool(np.array_equal(xs["update"], xs["set"]) and
                                                           np.array_equal(xs["update"], xs["coo"]))))


def lap2d_csr(torch, n, dev):
    """generate_lap2d_matrix's non-zeros as CSR tensors (int64 crow, int64 col, float64 values)"""
    inc = int(np.floor(np.sqrt(n)))
    i = torch.arange(n, device=dev)
    cols = torch.stack([i - 1 - inc, i - 1, i, i + 1, i + 1 + inc], dim=1)
    vals = torch.tensor([-1.0, -1.0, 4.0, -1.0, -1.0], dtype=torch.float64, device=dev).expand(n, 5)
    keep = torch.stack([i > inc, i > 0, torch.ones_like(i, dtype=torch.bool), i < n - 1, i < n - 1 - inc], dim=1)
    crow = torch.zeros(n + 1, dtype=torch.int64, device=dev)
    crow[1:] = torch.cumsum(keep.sum(dim=1), 0)
    return crow, cols[keep].contiguous(), vals[keep].contiguous()


if __name__ == "__main__":
    main()
