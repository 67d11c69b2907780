"""GPU tests of the drop-in command line (conjugate-gradient_b200/host/cgsolver): both reference
forms, the DEBUG stdout line, the results-file rows (code/MPI/cg_main.cc:57-64,
code/CUDA/cg_main.cc:54-60) -- numbers checked against the CPU oracle."""
import json
import os
import re
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CGSOLVER = os.path.join(ROOT, "conjugate-gradient_b200", "host", "cgsolver")
LINE = re.compile(r"^\t\[STEP (\d+)\] residual = (\d\.\d{6}e[+-]\d\d), \|\|x\|\| = (\d\.\d{6}e[+-]\d\d), "
                  r"\|\|Ax - b\|\|/\|\|b\|\| = (\d\.\d{6}e[+-]\d\d)$")


def _run(args, env=None, timeout=300):
    return subprocess.run([CGSOLVER] + args, capture_output=True, text=True, timeout=timeout,
                          env=dict(os.environ, **(env or {})))


def _step_line(stdout):
    """The DEBUG line (NCCL may print its version banner on stdout when NCCL_DEBUG is set)."""
    hits = [ln for ln in stdout.splitlines() if ln.startswith("\t[STEP")]
    assert len(hits) == 1, stdout
    return hits[0]


def test_form1_generated(O, tmp_path):
    """cgsolver N outfile [max_iter]: DEBUG line identical to the oracle's, row `n,psize,seconds`
    appended (not truncated)."""
    out = tmp_path / "res.txt"
    out.write_text("1024,1,0.0610\n")                       # an earlier row must survive
    js = tmp_path / "side.jsonl"
    r = _run(["1024", str(out)], env={"CGB_JSON": str(js)})
    assert r.returncode == 0, r.stderr
    ref = O.solve(O.generate_lap2d(1024), O.init_source_term(1024), nranks=1, nblk=148)
    lines = r.stdout.splitlines()
    assert len(lines) == 1 and LINE.match(lines[0])
    assert lines[0] == O.debug_line(ref.k, ref.rsold, ref.norm_x, ref.rel_resid)
    rows = out.read_text().splitlines()
    assert rows[0] == "1024,1,0.0610" and len(rows) == 2
    n, psize, sec = rows[1].split(",")
    assert (int(n), int(psize)) == (1024, 1) and 0 < float(sec) < 60
    side = json.loads(js.read_text())
    assert side["k"] == ref.k and side["converged"] is True
    # weak-scaling form: max_iter caps the loop; k printed = max_iter
    r = _run(["1448", str(out), "200"])
    assert r.returncode == 0
    ref = O.solve(O.generate_lap2d(1448), O.init_source_term(1448), max_iter=200, nranks=1, nblk=148)
    assert r.stdout.splitlines()[0] == O.debug_line(200, ref.rsold, ref.norm_x, ref.rel_resid)
    assert len(out.read_text().splitlines()) == 3


def test_form2_matrix_market(O, tmp_path):
    """cgsolver file.mtx NUM_THREADS BLOCK_WIDTH true/false outfile, with cg.run's comma-
    terminated tokens ("64,"), the sticky-scientific time line and the plain results row."""
    mtx = str(tmp_path / "lap30.mtx")
    O.write_lap2d_5pt_mtx(mtx, 30)
    A = O.read_mtx_dense(mtx)
    n = A.shape[0]
    ref = O.solve(A, O.init_source_term(n), max_iter=n, nranks=1, nblk=148)
    out = tmp_path / "res2.txt"
    for nt, bw, t in (("64,", "16,", "true"), ("1024", "4096", "false")):
        r = _run([mtx, nt, bw, t, str(out)])
        assert r.returncode == 0, r.stderr
        lines = r.stdout.splitlines()
        assert lines[0] == O.debug_line(ref.k, ref.rsold, ref.norm_x, ref.rel_resid)
        assert re.match(r"^Time for CG \(dense solver\)  = \d\.\d{6}e[+-]\d\d \[s\]$", lines[1])
    rows = out.read_text().splitlines()
    assert [row.split(",")[:2] for row in rows] == [["64", "16"], ["1024", "4096"]]
    for row in rows:
        assert re.match(r"^\d+,\d+,\d*\.?\d+(e-\d+)?$", row)
        assert 0 < float(row.split(",")[2]) < 60


def test_form2_compat_kernel_mode(O, tmp_path):
    """CGB_KERNEL=compat: the reference's own launch topologies, NUM_THREADS / BLOCK_WIDTH
    literal; the printed numbers are the oracle's for that chunked order."""
    mtx = str(tmp_path / "lap30.mtx")
    O.write_lap2d_5pt_mtx(mtx, 30)
    A = O.read_mtx_dense(mtx)
    n = A.shape[0]
    out = tmp_path / "res.txt"
    for nt, bw, t in (("64", "16", "true"), ("8", "900", "false")):
        with O.gemv_chunk(int(bw)):
            ref = O.solve(A, O.init_source_term(n), max_iter=n, nranks=1, nblk=148)
        r = _run([mtx, nt, bw, t, str(out)], env={"CGB_KERNEL": "compat"})
        assert r.returncode == 0, r.stderr
        assert _step_line(r.stdout) == O.debug_line(ref.k, ref.rsold, ref.norm_x, ref.rel_resid)
    assert [row.split(",")[:2] for row in out.read_text().splitlines()] == [["64", "16"], ["8", "900"]]


def test_cli_prints_what_the_reference_printed(O, tmp_path, golden_dir):
    """Both command-line forms against the stored stdout of the unmodified reference's own cgsolver on
    the same command line (tests/golden/, make_golden.py): a run capped above the rounding floor prints
    its [STEP k] and, to the 7 printed digits, its three numbers; converged runs stop within +-1 of an
    iteration count the reference itself produces for the system."""
    from parity_util import reference_k_set

    def numbers(line):
        m = LINE.match(line if line.startswith("\t") else "\t" + line)
        assert m, line
        return int(m.group(1)), [float(m.group(i)) for i in (2, 3, 4)]

    out = tmp_path / "res.txt"
    g = np.load(os.path.join(golden_dir, "gen_n1000_it50.npz"))
    r = _run(["1000", str(out), "50"])
    assert r.returncode == 0, r.stderr
    (k, mine), (k_ref, ref) = numbers(_step_line(r.stdout)), numbers(str(g["openblas_stdout_line"]))
    assert k == k_ref == 50
    for a, b in zip(mine, ref):
        assert abs(a - b) <= 2e-6 * abs(b), (mine, ref)
    mtx = str(tmp_path / "lap30.mtx")
    O.write_lap2d_5pt_mtx(mtx, 30)
    for name, args in (("gen_n1024.npz", ["1024", str(out)]),
                       ("mtx_lap2d_5pt_n30.npz", [mtx, "64", "16", "true", str(out)])):
        g = np.load(os.path.join(golden_dir, name))
        r = _run(args)
        assert r.returncode == 0, r.stderr
        k, (_, nx, _) = numbers(_step_line(r.stdout))
        assert min(abs(k - kr) for kr in reference_k_set(golden_dir, g)) <= 1, (name, k)
        assert abs(nx - float(g["openblas_norm_x"])) <= 2e-6 * nx, name
    rows = out.read_text().splitlines()
    assert [row.split(",")[:2] for row in rows] == [["1000", "1"], ["1024", "1"], ["64", "16"]]


def test_multi_gpu_cli_psize_column(O, tmp_path, cgb):
    if cgb.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    out = tmp_path / "res.txt"
    for mode in ("fused", "nccl"):
        r = _run(["2048", str(out), "150"], env={"CGB_GPUS": "2", "CGB_EXCHANGE": mode})
        assert r.returncode == 0, r.stderr
        ref = O.solve(O.generate_lap2d(2048), O.init_source_term(2048), max_iter=150, nranks=2, nblk=148)
        assert _step_line(r.stdout) == O.debug_line(150, ref.rsold, ref.norm_x, ref.rel_resid)
    assert [row.split(",")[:2] for row in out.read_text().splitlines()] == [["2048", "2"]] * 2


def test_multi_gpu_cli_ragged_rows(O, tmp_path, cgb):
    """N not divisible by the GPU count: the last rank owns more rows (cg.cc:236-268).  The default path --
    cgb_autotune on every rank alone before the timed solve, fused exchange, persistent kernel -- must
    neither wait for rows a shorter rank never stores nor change a digit of the DEBUG line."""
    G = cgb.device_count()
    if G < 2:
        pytest.skip("needs 2 GPUs")
    n, iters = 2051, 120
    out = tmp_path / "res.txt"
    r = _run([str(n), str(out), str(iters)], env={"CGB_GPUS": str(G), "CGB_SPIN_TIMEOUT_MS": "5000"})
    assert r.returncode == 0, r.stderr
    ref = O.solve(O.generate_lap2d(n), O.init_source_term(n), max_iter=iters, nranks=G, nblk=148)
    assert _step_line(r.stdout) == O.debug_line(iters, ref.rsold, ref.norm_x, ref.rel_resid)
    assert out.read_text().splitlines()[0].split(",")[:2] == [str(n), str(G)]


# --------------------------------------------------------------------------- INTEGRATION.md section B, compiled
REF_DIR = os.path.join(ROOT, "oracle", "_ref")
REF_CGB = os.path.join(REF_DIR, "cgsolver_ref_cgb")   # the reference's main + reader + rest of cg.cc, solve -> libcgb200
REF_CPU = os.path.join(REF_DIR, "cgsolver_ref")       # the unmodified reference (CPU, OpenBLAS or naive loops)


def _run_ref(exe, args, np_ranks=1, timeout=600):
    env = dict(os.environ, CGREF_NP=str(np_ranks), CGREF_BLAS="auto", OPENBLAS_NUM_THREADS="8", OMP_NUM_THREADS="8")
    return subprocess.run([exe] + args, capture_output=True, text=True, timeout=timeout, env=env)


@pytest.mark.parametrize("ranks", [1, 2])
def test_reference_main_bound_to_libcgb200(O, cgb, tmp_path, ranks):
    """The binding stub of INTEGRATION.md B (oracle/ref_shim/cg_cgb.cc) under the reference's OWN,
    unmodified cg_main.cc / matrix / rest of cg.cc (oracle/Makefile: cgsolver_ref_cgb; fork shim for
    P = 2, one rank per GPU): stdout and the results row against the unmodified CPU program
    (cgsolver_ref) on the same command line -- and, digit for digit, against the oracle."""
    if not (os.path.exists(REF_CGB) and os.path.exists(REF_CPU)):
        pytest.skip("oracle/_ref not built (needs /root/reference at build time)")
    if cgb.device_count() < ranks:
        pytest.skip("needs %d GPUs" % ranks)
    n, cap = 1448, "60"      # still above the rounding floor: the printed digits of the two programs agree
    out_gpu, out_cpu = tmp_path / "gpu.txt", tmp_path / "cpu.txt"
    g = _run_ref(REF_CGB, [str(n), str(out_gpu), cap], np_ranks=ranks)
    assert g.returncode == 0, g.stdout + g.stderr
    c = _run_ref(REF_CPU, [str(n), str(out_cpu), cap])
    assert c.returncode == 0, c.stderr
    lg, lc = _step_line(g.stdout), _step_line(c.stdout)
    mg, mc = LINE.match(lg), LINE.match(lc)
    assert mg and mc, (lg, lc)
    assert mg.group(1) == mc.group(1) == cap                         # [STEP k]
    for i in (2, 3, 4):                                              # residual, ||x||, ||Ax-b||/||b||
        a, b = float(mg.group(i)), float(mc.group(i))
        assert abs(a - b) <= 2e-6 * abs(b), (i, lg, lc)              # 7 printed digits; orders differ in the last
    ref = O.solve(O.generate_lap2d(n), O.init_source_term(n), max_iter=int(cap), nranks=ranks, nblk=148)
    assert lg == O.debug_line(int(cap), ref.rsold, ref.norm_x, ref.rel_resid)
    rg, rc = out_gpu.read_text().split(","), out_cpu.read_text().split(",")
    assert rg[:2] == [str(n), str(ranks)] and rc[:2] == [str(n), "1"]   # n,psize,seconds (cg_main.cc:62)
    assert 0 < float(rg[2]) < 120
    # converged run: the iteration count the reference prints, within +-1
    g = _run_ref(REF_CGB, ["1024", str(out_gpu)], np_ranks=ranks)
    c = _run_ref(REF_CPU, ["1024", str(out_cpu)])
    assert g.returncode == 0 and c.returncode == 0, g.stderr + c.stderr
    kg, kc = int(LINE.match(_step_line(g.stdout)).group(1)), int(LINE.match(_step_line(c.stdout)).group(1))
    assert abs(kg - kc) <= 1, (kg, kc)
