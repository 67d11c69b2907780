"""A time-step loop whose matrix is assembled from finite-element contributions every step, on CSR contexts.

    python profiles/assemble_bench.py [--out DIR] [--grids 1000,2000] [--steps K] [--repeats R] [--iters I]

Workload: a variable-coefficient 2-D Laplacian (plus a small reaction term) on an m x m grid of bilinear quad
elements, N = (m + 1)^2 nodes (m = 1000: N = 1.0 M, m = 2000: N = 4.0 M).  Every element contributes its 16
entries, so an interior cell receives up to 4 writes.  Every step a torch kernel makes the step's contributions
on the GPU (the element coefficients change with the step), the matrix is rebuilt from them, and one device solve
follows (max_iter = `--iters`, tol = 0, so every solve runs the same loop).  Four arms, alternating inside every
repeat, K steps each between two CUDA events on the stream (ms per step = elapsed / K), each arm on its own
context so that no arm's rebuild invalidates another's loop graphs:
  values    cgb_assemble_values + cgb_solve_device: the plan's gather-and-fold, no sync, no recapture
  assemble  cgb_assemble_coo every step (sort, stage, install; synchronises) + cgb_solve_device
  torch     torch coalesce() + to_sparse_csr() + cgb_update_matrix_values + cgb_solve_device: what a caller
            had to do before cgb_assemble_values (torch's summation order is not the library's contract)
  alone     K back-to-back cgb_assemble_values against K device copies whose read + write traffic equals the
            re-assembly's compulsory traffic (write ids, run starts, the contributions, the values written)
After the loop, one step of each arm from the same x0 and contributions: `values` and `assemble` must leave the
same x bit for bit; whether `torch` does too is reported.  One JSON line per measurement goes to stdout and to
DIR/assemble_bench.jsonl, after a line with the card's name, power limit and clocks.
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


class QuadAssembly:
    """The triples of the m x m quad grid (fixed) and, per step, their values made by torch kernels."""

    def __init__(self, torch, m, dev):
        self.torch = torch
        K = np.array([[4, -1, -2, -1], [-1, 4, -1, -2], [-2, -1, 4, -1], [-1, -2, -1, 4]], dtype=np.float64) / 6.0
        K += 0.01 * np.eye(4)
        e = torch.arange(m * m, device=dev)
        ex, ey = e % m, e // m
        nodes = torch.stack([ey * (m + 1) + ex, ey * (m + 1) + ex + 1, (ey + 1) * (m + 1) + ex + 1,
                             (ey + 1) * (m + 1) + ex], dim=1)
        self.n = (m + 1) ** 2
        self.irn = nodes.repeat_interleave(4, dim=1).reshape(-1).to(torch.int32)
        self.jcn = nodes.repeat(1, 4).reshape(-1).to(torch.int32)
        self.phase = (0.37 * ex + 0.61 * ey).to(torch.float64)
        self.K = torch.tensor(K.reshape(1, 16), device=dev)
        self.k = torch.empty(m * m, dtype=torch.float64, device=dev)
        self.vals = torch.empty(m * m * 16, dtype=torch.float64, device=dev)

    def values(self, t):
        torch = self.torch
        torch.sin(self.phase + 0.01 * (t % 100), out=self.k)
        self.k.mul_(0.9).add_(1.0)
        torch.mul(self.k[:, None], self.K, out=self.vals.view(-1, 16))
        return self.vals


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--grids", default="1000,2000")
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--repeats", type=int, default=5)
    ap.add_argument("--iters", type=int, default=50)
    args = ap.parse_args()
    import torch
    cgb = importlib.import_module("conjugate-gradient_b200")
    if not torch.cuda.is_available() or cgb.device_count() == 0:
        raise SystemExit("no GPU: nothing to measure")
    sink = open(os.path.join(args.out, "assemble_bench.jsonl"), "w") if args.out else None

    def emit(rec):
        line = json.dumps(rec)
        print(line, flush=True)
        if sink:
            sink.write(line + "\n")
            sink.flush()

    emit({"card": card()})
    dev = "cuda:0"
    for m in (int(s) for s in args.grids.split(",")):
        q = QuadAssembly(torch, m, dev)
        n, nz = q.n, q.irn.numel()
        ctx = {a: cgb.Context(n, storage="csr") for a in ("values", "assemble", "torch")}
        for c in ctx.values():
            c.assemble_coo((q.irn, q.jcn, q.values(0)))
        nnz = ctx["values"].nnz()
        idx = torch.stack([q.irn.to(torch.int64), q.jcn.to(torch.int64)])
        b = torch.tensor(cgb.init_source_term(n), device=dev)
        x = torch.zeros(n, dtype=torch.float64, device=dev)
        step_no = [0]

        def vals():
            step_no[0] += 1
            return q.values(step_no[0])

        def values():
            ctx["values"].assemble_values(vals())
            ctx["values"].solve_device(x, b, args.iters, tol=0.0)

        def assemble():
            ctx["assemble"].assemble_coo((q.irn, q.jcn, vals()))
            ctx["assemble"].solve_device(x, b, args.iters, tol=0.0)

        def coalesce():
            A = torch.sparse_coo_tensor(idx, vals(), (n, n)).coalesce().to_sparse_csr()
            ctx["torch"].update_matrix_values(A.values())
            ctx["torch"].solve_device(x, b, args.iters, tol=0.0)

        def timed(fn, k):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            for _ in range(k):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / k

        arms = {"values": values, "assemble": assemble, "torch": coalesce}
        for fn in arms.values():   # warm-up: graphs, buffers, first launches, torch's allocator
            timed(fn, 2)
        captures = ctx["values"].get_option("graph_captures")
        res = {a: [] for a in arms}
        for _ in range(args.repeats):
            for a, fn in arms.items():
                res[a].append(timed(fn, args.steps))
        info = {"grid": m, "n": n, "triples": nz, "nnz": nnz, "iters": args.iters, "steps": args.steps}
        rec = dict(info, kind="step", unit="ms_per_step",
                   graph_captures_values_arm=[captures, ctx["values"].get_option("graph_captures")])
        for a in arms:
            rec[a] = {"median": statistics.median(res[a]), "min": min(res[a]), "max": max(res[a]),
                      "all": [round(v, 4) for v in res[a]]}
        rec["assemble_over_values"] = rec["assemble"]["median"] / rec["values"]["median"]
        rec["torch_over_values"] = rec["torch"]["median"] / rec["values"]["median"]
        emit(rec)

        # the re-assembly alone, against a device copy of the same traffic
        c = ctx["values"]
        src_vals = q.values(3).clone()
        nwrites = nz   # no write leaves the shard and nothing is mirrored: every triple is one kept write
        traffic = 8 * nwrites + 8 * (nnz + 1) + 8 * nz + 8 * nnz
        src = torch.empty(traffic // 16, dtype=torch.float64, device=dev)
        dst = torch.empty_like(src)
        alone = {"values": [], "copy": []}
        for _ in range(args.repeats):
            alone["values"].append(timed(lambda: c.assemble_values(src_vals), 10 * args.steps))
            alone["copy"].append(timed(lambda: dst.copy_(src), 10 * args.steps))
        rec = dict(info, kind="assemble_values_alone", unit="ms_per_call", traffic_bytes=traffic)
        for a, v in alone.items():
            rec[a] = {"median": statistics.median(v), "min": min(v), "max": max(v), "all": [round(t, 5) for t in v]}
            rec[a]["GB_per_s"] = traffic / (rec[a]["median"] * 1e-3) / 1e9
        emit(rec)

        # the same contributions from the same x0 through every arm
        xs = {}
        for a, fn in arms.items():
            step_no[0] = 6
            x.zero_()
            fn()
            torch.cuda.synchronize()
            xs[a] = x.cpu().numpy().view(np.uint64).copy()
        emit(dict(info, kind="check", values_equals_assemble_x_bits=bool(np.array_equal(xs["values"], xs["assemble"])),
                  torch_equals_values_x_bits=bool(np.array_equal(xs["torch"], xs["values"])),
                  torch_x_words_differing=int(np.count_nonzero(xs["torch"] != xs["values"]))))
        for c in ctx.values():
            c.close()


if __name__ == "__main__":
    main()
