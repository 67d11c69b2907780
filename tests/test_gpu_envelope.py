"""Column windows of the dense mat-vec: every row block streams only the hull of its rows' non-zero
envelopes (DESIGN.md 3.3).  For finite p the skipped columns hold +-0 in every row of the block, so
the results are the full-row stream's, bit for bit -- checked here against the CPU oracle on
matrices whose envelopes stress the windows, on every persistent tile shape and on the graph
schedule, after every kind of write of A.

Every test here needs a B200:  python -m pytest tests -m gpu
"""
import math

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SIZES = [17, 257, 1001, 4097]


def _variants(cgb, n):
    """(variant, name) of every tile shape the persistent kernel is instantiated for; the graph
    schedule runs the gemv.cu variant of the same name."""
    out = []
    with cgb.Context(n, 0, 1, 0) as ctx:
        for v, name in enumerate(cgb.gemv_variants()):
            ctx.set_option("gemv_variant", v)
            if ctx.get_option("schedule_in_use") == 1:
                out.append((v, name))
    assert len(out) >= 4, out
    return out


def envelope_doubles(A):
    """Sum over the rows of (last + 1 - first) of the entries that are not +-0."""
    nz = (A.view(np.uint64) & np.uint64(0x7FFFFFFFFFFFFFFF)) != 0
    tot = 0
    for row in nz:
        idx = np.flatnonzero(row)
        if idx.size:
            tot += int(idx[-1]) + 1 - int(idx[0])
    return tot


def stress_matrix(n, seed):
    """Random per-row half-bandwidths from 0 to n (full dense rows included), all-zero rows and a
    whole zero block, a row whose only entry is column n - 1, neighbouring rows with far-apart
    envelopes, -0.0 entries outside the envelopes.  Strictly diagonally dominant wherever the row has
    a diagonal entry (a zero row has its column zeroed with it; stress_rhs puts b = 0 in the rows
    without one), so the solves stay finite."""
    rng = np.random.default_rng(seed)
    A = np.zeros((n, n))
    h = rng.integers(0, 4, n)                        # mostly narrow ...
    wide = rng.random(n) < 0.08
    h[wide] = rng.integers(0, n + 1, int(wide.sum()))  # ... some up to full rows
    if n > 4:
        h[n // 3] = n
    for i in range(n):
        lo, hi = max(0, i - h[i]), min(n, i + h[i] + 1)
        A[i, lo:hi] = rng.uniform(-1.0, 1.0, hi - lo)
    if n >= 8:                                       # far-apart envelopes in neighbouring rows
        i = n // 2
        A[i, :] = 0.0
        A[i + 1, :] = 0.0
        A[i, :3] = rng.uniform(-1, 1, 3)
        A[i + 1, n - 3:] = rng.uniform(-1, 1, 3)
    zero = np.zeros(n, dtype=bool)
    zero[rng.random(n) < 0.05] = True
    if n >= 100:
        zero[n // 5:n // 5 + max(40, n // 60)] = True  # more rows than one CTA holds
    A[zero, :] = 0.0
    A[:, zero] = 0.0
    d = np.abs(A).sum(axis=1) + np.abs(A).sum(axis=0) + 1.0
    A[np.arange(n), np.arange(n)] = np.where(zero, 0.0, d)
    if n >= 8:                                       # a row whose only entry is column n - 1
        r = n // 4
        A[r, :] = 0.0
        A[:, r] = 0.0
        A[r, n - 1] = 1e-3
    # -0.0 outside the envelopes (and in zero rows): not a non-zero
    for i in rng.choice(n, size=max(1, n // 10), replace=False):
        nzc = np.flatnonzero(A[i])
        if nzc.size == 0:
            A[i, rng.integers(0, n)] = -0.0
        else:
            if nzc[0] > 0:
                A[i, 0] = -0.0
            if nzc[-1] < n - 1:
                A[i, n - 1] = -0.0
    return A


def stress_rhs(A, O):
    """b of the stress systems: 0 in the rows without a diagonal entry, so that r stays 0 there."""
    b = O.init_source_term(A.shape[0]) + 1.0
    b[np.diag(A) == 0.0] = 0.0
    return b


def to_coo(A):
    irn, jcn = np.nonzero(A.view(np.uint64) != 0)   # -0.0 cells included: they are written as such
    return irn.astype(np.int32), jcn.astype(np.int32), A[irn, jcn]


def _solve(ctx, b, max_iter, x0=None):
    x = np.zeros(b.size) if x0 is None else x0.copy()
    info, hist = ctx.solve(x, max_iter=max_iter, tol=1e-10, history=True)
    nx, rr = ctx.residual_check()
    return x, info, hist, nx, rr


def _assert_oracle(got, ref, label, equal_nan=False):
    x, info, hist, nx, rr = got
    assert info.k == ref.k and bool(info.converged) == ref.converged, label
    assert np.array_equal(hist, ref.hist, equal_nan=equal_nan), label
    assert np.array_equal(x, ref.x, equal_nan=equal_nan), label
    assert np.array_equal([info.rsold, info.rsnew], [ref.rsold, ref.rsnew], equal_nan=equal_nan), label
    assert np.array_equal([nx, rr], [ref.norm_x, ref.rel_resid], equal_nan=equal_nan), label


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("upload", ["rows", "coo"])
def test_windows_bitwise_every_shape(cgb, O, n, upload):
    """Stress envelopes through set_matrix_rows and set_matrix_coo: every persistent shape, the
    persistent kernel and the graph schedule, == the oracle (the dense full-row order) bit for bit."""
    A = stress_matrix(n, 100 + n)
    b = stress_rhs(A, O)
    max_iter = min(n, 60)
    ref = None
    for v, name in _variants(cgb, n):
        for sched in (1, 0):
            with cgb.Context(n, 0, 1, 0) as ctx:
                ctx.set_option("gemv_variant", v)
                ctx.set_option("schedule", sched)
                if upload == "rows":
                    ctx.set_matrix_rows(A)
                else:
                    ctx.set_matrix_coo(*to_coo(A), symmetric=False)
                assert np.array_equal(ctx.get_matrix_rows(0, n).view(np.uint64), A.view(np.uint64))
                assert ctx.get_option("envelope_doubles") == envelope_doubles(A)
                ctx.set_rhs(b)
                got = _solve(ctx, b, max_iter)
                nblk = ctx.layout().nblk
            if ref is None:
                ref = O.solve(A, b, max_iter=max_iter, nranks=1, nblk=nblk)
                assert np.all(np.isfinite(ref.x)) and np.all(np.isfinite(ref.hist))
            _assert_oracle(got, ref, (name, sched))


def test_windows_with_rebalancing(cgb, O):
    """A system large enough for the persistent kernel's row re-balancing (rows >= 64 per CTA),
    with a zero block wider than a CTA's rows (CTAs with rows but no tile to stream) and a few full
    rows: the re-balanced partition moves the blocks and with them the windows; same bits."""
    n = 12000
    A = O.generate_lap2d(n)
    A[3000:3400, :] = 0.0
    A[:, 3000:3400] = 0.0
    A[3000:3400, 3000:3400] = np.diag(np.full(400, 4.0))
    for i in (10, 7777):
        A[i, :] += 1e-3
        A[:, i] += 1e-3
        A[i, i] = 4.0 + 2e-3 * n
    b = O.init_source_term(n) + 1.0
    for sched in (1, 0):
        with cgb.Context(n, 0, 1, 0) as ctx:
            ctx.set_option("schedule", sched)
            ctx.set_matrix_rows(A)
            ctx.set_rhs(b)
            got = _solve(ctx, b, 64)
            nblk = ctx.layout().nblk
        if sched == 1:
            ref = O.solve(A, b, max_iter=64, nranks=1, nblk=nblk)
        _assert_oracle(got, ref, sched)


@pytest.mark.parametrize("sched", [1, 0])
def test_envelope_follows_every_write(cgb, O, sched):
    """Stale-envelope guard: solve, widen some rows, solve, narrow them again, solve; then a dense
    upload followed by generate_lap2d.  Each solve == the oracle for the matrix held then."""
    n = 4097
    b = O.init_source_term(n) + 1.0
    L = O.generate_lap2d(n)
    rows = [0, 5, 1000, 1001, 2048, n - 1]
    W = L.copy()
    for i in rows:                                   # widened: the whole row
        W[i, :] = np.where(W[i] == 0.0, 1e-4, W[i])
    N = L.copy()
    for i in rows:                                   # narrowed: the diagonal only
        N[i, :] = 0.0
        N[i, i] = 4.0
    with cgb.Context(n, 0, 1, 0) as ctx:
        ctx.set_option("schedule", sched)
        ctx.set_rhs(b)
        nblk = ctx.layout().nblk
        ctx.generate_lap2d()
        for label, M in (("lap2d", L), ("widened", W), ("narrowed", N)):
            if label != "lap2d":
                for i in rows:
                    ctx.set_matrix_rows(M[i:i + 1], first_row=i)
            assert ctx.get_option("envelope_doubles") == envelope_doubles(M), label
            _assert_oracle(_solve(ctx, b, 80), O.solve(M, b, max_iter=80, nranks=1, nblk=nblk), label)
        D = np.full((n, n), 1e-5)
        D[np.arange(n), np.arange(n)] = 2.0 * n
        ctx.set_matrix_rows(D)
        assert ctx.get_option("envelope_doubles") == n * n
        _assert_oracle(_solve(ctx, b, 20), O.solve(D, b, max_iter=20, nranks=1, nblk=nblk), "dense")
        ctx.generate_lap2d()
        assert ctx.get_option("envelope_doubles") == envelope_doubles(L)
        _assert_oracle(_solve(ctx, b, 80), O.solve(L, b, max_iter=80, nranks=1, nblk=nblk), "lap2d again")


def _lap2d_envelope_doubles(n):
    """generate_lap2d_matrix's row envelopes (cg.cc:159-188) in closed form."""
    inc = int(math.floor(math.sqrt(n)))
    tot = 0
    for i in range(n):
        lo = i - 1 - inc if i > inc else (i - 1 if i > 0 else i)
        hi = i + 1 + inc if i < n - 1 - inc else (i + 1 if i < n - 1 else i)
        tot += hi + 1 - lo
    return tot


def test_envelope_doubles_option(cgb, O):
    """"envelope_doubles" == the count numpy gives; lap2d at N = 40000 in closed form; 0 on CSR."""
    for n in (17, 1001):
        with cgb.Context(n, 0, 1, 0) as ctx:
            assert ctx.get_option("envelope_doubles") == 0         # a new context: every row empty
            ctx.generate_lap2d()
            assert ctx.get_option("envelope_doubles") == envelope_doubles(O.generate_lap2d(n))
            assert envelope_doubles(O.generate_lap2d(n)) == _lap2d_envelope_doubles(n)
    n = 40000
    with cgb.Context(n, 0, 1, 0) as ctx:
        ctx.generate_lap2d()
        assert ctx.get_option("envelope_doubles") == _lap2d_envelope_doubles(n) == 16_039_598
    with cgb.Context(1001, 0, 1, 0, storage="csr") as ctx:
        ctx.generate_lap2d()
        assert ctx.get_option("envelope_doubles") == 0


def test_non_finite_p_exception(cgb, O):
    """The one exception (DESIGN.md 3.7 for CSR, 3.3 here): an Inf of the input vector in a column a
    row block skips.  The dense stream makes every row with a 0 there NaN (0 x Inf); the windowed
    stream leaves the rows whose window excludes that column finite -- exactly those rows differ.
    A whole solve driven non-finite (x0 with +-1e308) gives the oracle's outputs (NaN where NaN):
    alpha is NaN after the first iteration either way, and nothing else reaches the outputs."""
    n = 4097
    A = O.generate_lap2d(n)
    b = O.init_source_term(n)
    c = 3000
    v = np.ones(n)
    v[c] = np.inf
    with cgb.Context(n, 0, 1, 0) as ctx:
        ctx.generate_lap2d()
        y, _ = ctx.gemv(v)
        nblk = ctx.layout().nblk
        x0 = np.zeros(n)
        x0[[100, 101, 2500]] = [1e308, -1e308, 1e308]
        ctx.set_rhs(b)
        got = _solve(ctx, b, 30, x0=x0)
    dense = O.gemv(A, v)
    v0 = v.copy()
    v0[c] = 0.0
    finite = O.gemv(A, v0)
    differ = ~np.isfinite(dense) & np.isfinite(y)
    # the rows that differ are rows without an entry in column c, and there they are the finite sum
    assert np.all(A[differ, c] == 0.0)
    assert np.array_equal(y[differ], finite[differ])
    assert np.array_equal(y[~differ], dense[~differ], equal_nan=True)
    assert differ.sum() > n // 2                    # most rows' windows are far from column c
    assert np.all(~np.isfinite(y[A[:, c] != 0.0]))   # the rows with an entry there are Inf in both
    ref = O.solve(A, b, x0=x0, max_iter=30, nranks=1, nblk=nblk)
    _assert_oracle(got, ref, "non-finite", equal_nan=True)
