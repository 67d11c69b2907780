"""The dense mat-vec's column windows and the CSR mat-vec's row paths at their structural edges.

Three groups of checks:
  * CPU (no marker): every input family used below is checked against *mutants* of the kernels'
    summation order -- a dropped tail chunk, a block hull taken from the first row only, an envelope
    that treats subnormals / NaN / Inf as zero, merge or butterfly levels in another order, one
    sequential chain instead of bucket chains.  Each mutant must change the bits of a stated number
    of rows, so a kernel with that bug cannot pass the GPU checks.  The lane order is also pinned to
    be invariant under an even rotation of the bucket index (why a window may start at any even
    column), and the oracle is checked against the exact dot product.
  * GPU, dense: every gemv variant on windows that start at every residue mod 64, end at every
    residue mod 16, run exactly k tiles (+ 16 columns), sit between empty blocks; special values;
    the graph-only tile shapes in whole solves; the kWinBlocks = 128 fallback (blocks of a CTA past
    the window table stream full rows) on the graph schedule and the persistent kernel, each test
    asserting that it reached it; the partial envelope rebuild of a rank's shard.
  * GPU, CSR: row lengths 0 .. 12 (the single-lane merge tree up to kShortRow = 8 and the warp path
    from 9), the 32-entry slab edges and 2000, with bucket patterns that exercise each merge level.

GPU tests:  python -m pytest tests/test_matvec_edges.py -m gpu
"""
from fractions import Fraction

import numpy as np
import pytest

import csr_oracle
import oracle
from test_gpu_envelope import envelope_doubles, stress_matrix, stress_rhs, to_coo

U = 2.0 ** -53
GRID = 148                                   # CTAs of a 1-CTA-per-SM tile shape on a B200
SHAPES = [(tr, nblk) for tr in (4, 8, 16, 32) for nblk in (GRID, 2 * GRID)]  # (rows of a tile, CTAs)
EDGE_SIZES = [17, 257, 1001, 4095, 4096, 4097, 4081]     # ld - n = 15, 15, 7, 1, 0, 15, 15
STRESS_SIZES = [17, 257, 1001, 4097]
WIN_BLOCKS = 128                             # kWinBlocks (cgb_device.cuh)
CSR_LENGTHS = list(range(13)) + [31, 32, 33, 34, 63, 64, 65, 66, 95, 96, 97, 2000]


# --------------------------------------------------------------------------- helpers
def _bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


def _differ(a, b):
    """rows whose bits differ (two NaNs count as equal)"""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    nan = np.isnan(a) & np.isnan(b)
    return (_bits(a) != _bits(b)) & ~nan


def _same(a, b):
    return not _differ(a, b).any()


def _spread(rng, k):
    """k values of magnitude 2^-30 .. 2^30 with random signs: a different association changes bits"""
    return rng.choice([-1.0, 1.0], k) * np.exp2(rng.uniform(-30.0, 30.0, k))


def edge_vector(n, seed):
    """input vector: |p| in [1, 2) with random signs (so 5e-324 * p is not 0)"""
    rng = np.random.default_rng(seed)
    return rng.choice([-1.0, 1.0], n) * rng.uniform(1.0, 2.0, n)


def block_bounds(rows, nblk, tr):
    """[start, end) of every row block of gemv.cu's graph kernel: CTA c owns rows c*rows/nblk ..,
    cut into nb = ceil(nrows / tr) balanced blocks.  (CTA, block index in the CTA, start, end)."""
    out = []
    for c in range(nblk):
        r0, r1 = c * rows // nblk, (c + 1) * rows // nblk
        nrows = r1 - r0
        nb = -(-nrows // tr)
        for b in range(nb):
            out.append((c, b, r0 + b * nrows // nb, r0 + (b + 1) * nrows // nb))
    return out


def _fill(A, rng, i, f, last, interior=40):
    """row i: non-zeros at f and `last` and up to `interior` random columns in between"""
    A[i, f] = _spread(rng, 1)[0]
    A[i, last] = _spread(rng, 1)[0]
    k = min(max(last - f - 1, 0), interior)
    if k:
        A[i, rng.choice(np.arange(f + 1, last), k, replace=False)] = _spread(rng, k)


def edge_matrix(n, seed):
    """Deterministic envelopes at the window edges, in row order (what does not fit in n rows is
    left out; edge_coverage states what is in):
      rows whose first non-zero has residue r = 0 .. 63 mod 64 and last non-zero r mod 16;
      single-entry rows at column 0 and n - 1;
      all-zero runs longer than 3 row blocks, so whole blocks without a window sit between others;
      alternating rows [0, 16) / [n - 16, n), so a block's hull is the full row;
      one full row;
      runs of rows with windows of exactly k*w and k*w + 16 columns from a 64-aligned start
      (w = 256, 512, 640, 704, 1024, 2048, the tile widths of the shapes; k = 1, 2), each run long
      enough to hold a whole row block;
      the rest narrow random rows and zero rows.
    Values 2^-30 .. 2^30 with random signs."""
    rng = np.random.default_rng(seed)
    A = np.zeros((n, n))
    bmax = max(1, min(32, -(-n // GRID)))      # most rows a row block of any shape has at this n
    i = 0
    for r in range(64):                        # first % 64 = r, last % 16 = r % 16
        if i >= n or r >= n:
            break
        f = r + 64 * ((7 * r) % max(1, (n - r) // 64))
        want = f + int(rng.integers(0, 300))
        last = want + ((r % 16) - want) % 16
        if last >= n:                          # the last column of that residue, if past f
            last = max(f, n - 1 - (n - 1 - r % 16) % 16)
        _fill(A, rng, i, f, last)
        i += 1
    for c in (0, n - 1):                       # single entries at the first and the last column
        if i < n:
            A[i, c] = _spread(rng, 1)[0]
            i += 1
    i += 3 * bmax + 1                          # zero run
    for j in range(2 * bmax + 2):              # [0, 16) and [n - 16, n) in turn
        if i >= n:
            break
        if j % 2 == 0:
            _fill(A, rng, i, 0, min(15, n - 1), interior=14)
        else:
            _fill(A, rng, i, max(0, n - 16), n - 1, interior=14)
        i += 1
    i += 3 * bmax + 1
    if i < n:                                  # one full row
        A[i, :] = _spread(rng, n)
        i += 1
    run = 2 * bmax + 1
    for w in (256, 512, 640, 704, 1024, 2048):
        for k in (1, 2):
            for extra in (0, 16):
                width = k * w + extra
                if width > n or i + run > n:
                    continue
                f = ((n - width) // 2) & ~63
                for _ in range(run):
                    _fill(A, rng, i, f, f + width - 1)
                    i += 1
        i += 1
    while i < n:                               # filler: narrow random envelopes, some zero rows
        if rng.random() < 0.8:
            f = int(rng.integers(0, n))
            _fill(A, rng, i, f, min(n - 1, f + int(rng.integers(0, 200))), interior=8)
        i += 1
    return A


def edge_coverage(A):
    """what edge_matrix put in: residues of first / last non-zeros, single entries, widths"""
    nz = _bits(A) & np.uint64(0x7FFFFFFFFFFFFFFF) != 0
    has = nz.any(axis=1)
    first = np.argmax(nz, axis=1)[has]
    last = (A.shape[1] - 1 - np.argmax(nz[:, ::-1], axis=1))[has]
    return set(first % 64), set(last % 16), set(last - first + 1), nz.sum(axis=1)


def add_special_rows(A):
    """Five rows near the end: only subnormals (1, 8, 64, 512 times 5e-324: whatever the signs of p,
    the largest product outweighs the others); a narrow row holding NaN; one holding +Inf; -0.0
    inside a window; only -0.0 (an empty envelope).  Returns their indices."""
    n = A.shape[0]
    rows = [n - 6 + j for j in range(5)]
    A[rows, :] = 0.0
    c = n // 2
    cols = [x for x in (c - 3, c, c + 5, c + 40) if 0 <= x < n]
    A[rows[0], cols] = 5e-324 * np.array([1.0, 8.0, 64.0, 512.0])[:len(cols)]  # no sum of them cancels
    A[rows[1], c:min(n, c + 6)] = 1.5
    A[rows[1], min(n - 1, c + 2)] = np.nan
    A[rows[2], max(0, c - 4):c + 1] = -2.5
    A[rows[2], max(0, c - 2)] = np.inf
    A[rows[3], 0:min(n, 70)] = 0.75
    A[rows[3], min(n - 1, 33)] = -0.0
    A[rows[3], min(n - 1, 1)] = -0.0
    A[rows[4], cols] = -0.0
    return rows


# ---- mutants of the summation order, built from the CSR oracle (tied bit for bit to the dense one)
def to_csr(A):
    """the entries that are not +-0 (NaN and Inf included); the lane order skips +-0 for finite p"""
    return csr_oracle.csr_from_dense(A)


def _rows_of(m):
    return np.repeat(np.arange(m.rows), np.diff(m.rp))


def _keep(m, mask):
    lens = np.bincount(_rows_of(m)[mask], minlength=m.rows)
    rp = np.zeros(m.rows + 1, dtype=np.int64)
    rp[1:] = np.cumsum(lens)
    return csr_oracle.Csr(m.n, rp, np.ascontiguousarray(m.col[mask]), np.ascontiguousarray(m.val[mask]))


def bucket_map(f):
    """column c -> (c & ~63) | f(c & 63), for a bijection f of 0 .. 63"""
    tab = np.array([f(b) for b in range(64)], dtype=np.int64)
    assert sorted(tab) == list(range(64))
    return lambda c: (c & ~63) | tab[c & 63]


def gemv_mapped(m, p, g):
    """the lane order of a column-mapped copy: a bucket permutation keeps every chain in its order
    (a bucket's entries keep their column order) but changes which lane and level meets which"""
    col = g(m.col.astype(np.int64))
    pp = np.zeros(-(-m.n // 64) * 64 + 64)
    pp[g(np.arange(m.n))] = p
    return csr_oracle.gemv_csr(csr_oracle.Csr(m.n, m.rp, col.astype(np.int32), m.val), pp)


def _bitperm(order):
    """bucket b = 2l + e: lane bit j of the new index is bit order[j] of l (the pair bit e kept)"""
    def f(b):
        l, e = b >> 1, b & 1
        return 2 * sum(((l >> order[j]) & 1) << j for j in range(5)) + e
    return f


PERMS = {
    "levels_reversed": _bitperm([4, 3, 2, 1, 0]),       # butterfly ^1 first instead of ^16
    "levels_16_8_swapped": _bitperm([0, 1, 2, 4, 3]),   # the first two levels exchanged
    "pair_with_lane_bit": lambda b: (b & 0b011110) | ((b & 1) << 5) | (b >> 5),  # even/odd pair split
}


def mutant_tail_dropped(m, p):
    """c_end rounded down to 16 instead of up: the last partial 16-column chunk of every row lost"""
    rows = _rows_of(m)
    hi = np.zeros(m.rows, dtype=np.int64)
    np.maximum.at(hi, rows, m.col.astype(np.int64) + 1)
    return csr_oracle.gemv_csr(_keep(m, m.col < (hi[rows] & ~15)), p)


def mutant_first_row_hull(m, p, ld, tr, nblk):
    """every block's window taken from its first row's envelope"""
    rows = _rows_of(m)
    lo_of = np.full(m.rows, 1 << 62, dtype=np.int64)
    hi_of = np.zeros(m.rows, dtype=np.int64)
    np.minimum.at(lo_of, rows, m.col.astype(np.int64))
    np.maximum.at(hi_of, rows, m.col.astype(np.int64) + 1)
    cb = np.zeros(m.rows, dtype=np.int64)
    ce = np.zeros(m.rows, dtype=np.int64)
    for _, _, s, e in block_bounds(m.rows, nblk, tr):
        if e > s and hi_of[s] > 0:
            cb[s:e] = lo_of[s] & ~63
            ce[s:e] = min(ld, (hi_of[s] + 15) & ~15)
    return csr_oracle.gemv_csr(_keep(m, (m.col >= cb[rows]) & (m.col < ce[rows])), p)


def mutant_special_as_zero(m, p):
    """an envelope that does not count subnormals, NaN or Inf: those entries skipped"""
    a = np.abs(m.val)
    return csr_oracle.gemv_csr(_keep(m, np.isfinite(a) & (a >= 2.2250738585072014e-308)), p)


def _fma(a, b, c):
    return float(Fraction(a) * Fraction(b) + Fraction(c))


def mutant_sequential(m, p):
    """one fma chain over the row in column order (rounded exactly like fma)"""
    y = np.empty(m.rows)
    for i in range(m.rows):
        s = 0.0
        for k in range(m.rp[i], m.rp[i + 1]):
            s = _fma(float(m.val[k]), float(p[m.col[k]]), s)
        y[i] = s
    return y


def _ld(n):
    return (n + 15) & ~15


# ---- input families: (name, CSR matrix, p, ld); every one is used by a GPU test below
def _family(name):
    kind, n = name.split(":")
    n = int(n)
    if kind == "edge":
        A = edge_matrix(n, 7 + n)
        return to_csr(A), edge_vector(n, n), _ld(n), A
    if kind == "special":
        A = edge_matrix(n, 7 + n)
        add_special_rows(A)
        return to_csr(A), edge_vector(n, n), _ld(n), A
    if kind == "stress":
        A = stress_matrix(n, 100 + n)
        return to_csr(A), edge_vector(n, n), _ld(n), A
    if kind == "lap2d":
        A = oracle.generate_lap2d(n)
        return to_csr(A), edge_vector(n, n), _ld(n), A
    if kind == "fallback":
        m, _ = lap2d_with_far_rows(n, fallback_rows(n))
        return m, edge_vector(n, n), _ld(n), None
    if kind == "csr_rows":
        m = csr_oracle.csr_from_coo(n, *csr_row_matrix(n), symmetric=False)
        return m, edge_vector(n, n), _ld(n), None
    raise AssertionError(name)


# --------------------------------------------------------------------------- C: the fallback inputs
def fallback_rows(n, nblk=GRID, tr=4):
    """Rows to widen in lap2d: in 3 CTAs, the first row of blocks 5, 127 (window table) and 128,
    nb - 1 (past it, full rows) -- for the graph kernel's split of tma_w4r1c2048s2."""
    bb = block_bounds(n, nblk, tr)
    out = []
    for c in (0, nblk // 2, nblk - 1):
        mine = [x for x in bb if x[0] == c]
        for b in (5, WIN_BLOCKS - 1, WIN_BLOCKS, len(mine) - 1):
            if b < len(mine):
                out.append(mine[b][2] + (1 if mine[b][3] - mine[b][2] > 1 else 0))
    return sorted(set(out))


def lap2d_with_far_rows(n, rows):
    """lap2d (CSR) with `rows` given small entries far from the diagonal, at column 0, mid-row and
    column n - 1, the diagonal raised by their sum (strictly diagonally dominant).  Returns the CSR
    matrix and {row: dense row}."""
    m = csr_oracle.generate_lap2d_csr(n)
    new = {}
    for i in rows:
        r = np.zeros(n)
        s, e = m.rp[i], m.rp[i + 1]
        r[m.col[s:e]] = m.val[s:e]
        extra = [0, 17, n // 3 + 5, (2 * n) // 3 + 38, n - 1]
        for k, c in enumerate(extra):
            if abs(c - i) > 300:
                r[c] = (1e-3 + 1e-5 * k) * (-1) ** k
        r[i] = 0.0
        r[i] = np.abs(r).sum() + 1e-3
        new[i] = r
    lens = np.diff(m.rp)
    cparts, vparts, prev = [], [], 0
    for i in sorted(new):
        cparts += [m.col[m.rp[prev]:m.rp[i]]]
        vparts += [m.val[m.rp[prev]:m.rp[i]]]
        nz = np.flatnonzero(new[i])
        cparts.append(nz.astype(np.int32))
        vparts.append(new[i][nz])
        lens[i] = nz.size
        prev = i + 1
    cparts.append(m.col[m.rp[prev]:])
    vparts.append(m.val[m.rp[prev]:])
    rp = np.zeros(n + 1, dtype=np.int64)
    rp[1:] = np.cumsum(lens)
    return csr_oracle.Csr(n, rp, np.concatenate(cparts), np.concatenate(vparts)), new


# --------------------------------------------------------------------------- D: CSR row patterns
def _row_cols(rng, n, L, kind):
    """L distinct columns of one pattern kind, or None when n cannot hold it"""
    nblocks = n // 64
    if kind == "one_bucket":                   # every entry in bucket b
        if L > nblocks:
            return None
        b = int(rng.integers(0, 64))
        return 64 * np.sort(rng.choice(nblocks, L, replace=False)) + b
    if kind == "pairs":                        # 2l and 2l + 1 of the same 64-block
        if L < 2 or (L + 1) // 2 > nblocks:
            return None
        l = int(rng.integers(0, 32))
        blocks = np.sort(rng.choice(nblocks, (L + 1) // 2, replace=False))
        cols = np.concatenate([[64 * k + 2 * l, 64 * k + 2 * l + 1] for k in blocks])[:L]
        return np.sort(cols)
    if kind.startswith("bit"):                 # buckets b and b ^ 2^j only: merges at level j
        j = int(kind[3:])
        if L < 2 or (L + 1) // 2 > nblocks:
            return None
        b = int(rng.integers(0, 64))
        blocks = np.sort(rng.choice(nblocks, (L + 1) // 2, replace=False))
        cols = np.concatenate([[64 * k + b, 64 * k + (b ^ (1 << j))] for k in blocks])[:L]
        return np.sort(cols)
    if kind == "descending":                   # the first column in a higher bucket than later ones
        if L < 2 or 64 + L - 1 > n:
            return None
        s = 64 * int(rng.integers(0, max(1, nblocks - 2))) + 63 - (L - 1) // 2
        return np.arange(max(0, s), max(0, s) + L)
    if kind == "spread":
        return np.sort(rng.choice(n, L, replace=False))
    raise AssertionError(kind)


CSR_KINDS = ["one_bucket", "pairs", "bit1", "bit2", "bit3", "bit4", "bit5", "descending", "spread"]


def csr_row_matrix(n, seed=5):
    """COO (row-major, ascending columns) with a row of every length in CSR_LENGTHS for every
    pattern kind that fits; rows of 8 non-zeros + a stored +0 or -0 (9 stored: the warp path) and
    of 7 + a stored zero (8: the single lane); the rest random lengths 0 .. 12.  Rows shuffled so
    short and long rows share warps."""
    rng = np.random.default_rng(seed)
    rows = []                                  # (cols, vals)
    for L in CSR_LENGTHS:
        for kind in CSR_KINDS if L else ["spread"]:
            c = _row_cols(rng, n, L, kind)
            if c is not None:
                rows.append((c, _spread(rng, c.size)))
    for base, z in ((8, 0.0), (8, -0.0), (7, 0.0), (7, -0.0)):
        c = np.sort(rng.choice(n, base + 1, replace=False))
        v = _spread(rng, base + 1)
        v[int(rng.integers(0, base + 1))] = z
        rows.append((c, v))
    assert len(rows) <= n
    while len(rows) < n:
        L = int(rng.integers(0, 13))
        rows.append((np.sort(rng.choice(n, L, replace=False)), _spread(rng, L)))
    order = rng.permutation(n)
    irn, jcn, val = [], [], []
    for i, k in enumerate(order):
        c, v = rows[k]
        irn.append(np.full(c.size, i))
        jcn.append(c)
        val.append(v)
    return (np.concatenate(irn).astype(np.int32), np.concatenate(jcn).astype(np.int32),
            np.concatenate(val))


def csr_solve_matrix(n, seed=11):
    """diagonally dominant rows of 7 .. 9 stored entries (the diagonal and 6 .. 8 others)"""
    rng = np.random.default_rng(seed)
    irn, jcn, val = [], [], []
    for i in range(n):
        k = int(rng.integers(6, 9))
        off = rng.choice(np.setdiff1d(np.arange(max(0, i - 200), min(n, i + 200)), [i]), k, replace=False)
        v = rng.uniform(-1.0, 1.0, k)
        c = np.append(off, i)
        v = np.append(v, np.abs(v).sum() + 0.5)
        o = np.argsort(c)
        irn.append(np.full(k + 1, i))
        jcn.append(c[o])
        val.append(v[o])
    return (np.concatenate(irn).astype(np.int32), np.concatenate(jcn).astype(np.int32),
            np.concatenate(val))


# ============================================================================ A: CPU
# Rows each mutant must change, per input family: about half of what the seeded inputs give.  0
# states that the family cannot see that mutant (lap2d's few buckets never meet at those levels;
# at n = 17 the rows are too short); the other families of the same GPU tests do.
MUTANTS = ["levels_reversed", "levels_16_8_swapped", "pair_with_lane_bit", "tail_dropped", "first_row_hull"]
MIN_CHANGED = {
    "edge:17": (1, 0, 0, 8, 0),
    "edge:257": (50, 10, 6, 85, 29),
    "edge:1001": (200, 45, 15, 300, 220),
    "edge:4095": (900, 200, 100, 900, 750),
    "edge:4096": (900, 200, 100, 900, 750),
    "edge:4097": (900, 200, 100, 900, 750),
    "edge:4081": (900, 200, 100, 900, 750),
    "special:257": (50, 10, 6, 85, 29),
    "special:4097": (900, 200, 100, 900, 750),
    "stress:17": (1, 0, 0, 7, 0),
    "stress:257": (17, 2, 2, 96, 10),
    "stress:1001": (65, 12, 10, 435, 65),
    "stress:4097": (300, 44, 45, 1800, 300),
    "fallback:75776": (14500, 0, 0, 35000, 11),
    "fallback:80000": (14800, 0, 0, 37000, 3800),
    "csr_rows:5000": (750, 38, 14, 2000, 1190),
}
FAMILIES = list(MIN_CHANGED)


def test_lap2d_4097_is_blind_to_the_level_order(O):
    """Why the families below exist: at n = 4097 (inc = 64) lap2d's five entries fall in three
    adjacent buckets and the merge tree has two leaves, so a reversed butterfly changes no row."""
    m, p, _, _ = _family("lap2d:4097")
    y = csr_oracle.gemv_csr(m, p)
    assert _differ(gemv_mapped(m, p, bucket_map(PERMS["levels_reversed"])), y).sum() == 0


@pytest.mark.parametrize("family", FAMILIES)
def test_mutants_change_rows(O, family):
    """Each mutant of the kernels' order changes at least MIN_CHANGED rows of the family's y.  The
    first-row hull is checked on every tile shape whose CTAs hold more than one row."""
    m, p, ld, A = _family(family)
    y = csr_oracle.gemv_csr(m, p)
    if A is not None:
        assert _same(y, O.gemv(A, p))         # the CSR form is the dense lane order, bit for bit
    got = [int(_differ(gemv_mapped(m, p, bucket_map(PERMS[k])), y).sum()) for k in MUTANTS[:3]]
    got.append(int(_differ(mutant_tail_dropped(m, p), y).sum()))
    got.append(min([int(_differ(mutant_first_row_hull(m, p, ld, tr, nblk), y).sum())
                    for tr, nblk in SHAPES if m.rows > nblk] or [0]))
    for name, k, need in zip(MUTANTS, got, MIN_CHANGED[family]):
        assert k >= need, (family, name, k, need)
    if family.startswith("special"):           # the subnormal, the NaN and the Inf row
        assert int(_differ(mutant_special_as_zero(m, p), y).sum()) == 3


@pytest.mark.parametrize("family", ["edge:4097", "stress:1001", "csr_rows:5000"])
def test_sequential_chain_mutant(family):
    """A CSR mat-vec that ran one fma chain per row in column order instead of bucket chains"""
    m, p, _, _ = _family(family)
    sel = np.flatnonzero(np.diff(m.rp) <= 2100)[:1500]   # a bounded number of exact evaluations
    sub = csr_oracle.Csr(m.n, np.concatenate([[0], np.cumsum(np.diff(m.rp)[sel])]).astype(np.int64),
                         np.concatenate([m.col[m.rp[i]:m.rp[i + 1]] for i in sel]).astype(np.int32),
                         np.concatenate([m.val[m.rp[i]:m.rp[i + 1]] for i in sel]))
    y = csr_oracle.gemv_csr(sub, p)
    multi = int((np.diff(sub.rp) > 1).sum())
    assert int(_differ(mutant_sequential(sub, p), y).sum()) >= max(1, multi // 10)


@pytest.mark.parametrize("family", ["edge:4097", "stress:4097", "fallback:80000", "csr_rows:5000"])
def test_even_bucket_rotation_is_invariant(family):
    """Rotating the bucket index by an even amount keeps the lane pairs (2l, 2l+1) and maps the
    butterfly's residue classes onto residue classes: no row changes.  So a window may start at any
    even column; 64-alignment is sufficient, not necessary.  An odd rotation splits the pairs."""
    m, p, _, _ = _family(family)
    y = csr_oracle.gemv_csr(m, p)
    for k in (2, 16, 48):
        assert _same(gemv_mapped(m, p, bucket_map(lambda b, k=k: (b + k) & 63)), y), k
    assert _differ(gemv_mapped(m, p, bucket_map(lambda b: (b + 1) & 63)), y).sum() > 0


@pytest.mark.parametrize("family", ["edge:4097", "stress:1001", "csr_rows:5000"])
def test_oracle_within_error_bound_of_exact(family):
    """|y - round(exact)| <= (L + 7) u sum |a p|: L + 6 roundings on the lane order's longest path
    (a bucket chain of L fmas, the pair sum, 5 butterfly levels), one more for rounding the exact
    dot.  Guards against the oracle and the kernels agreeing on nonsense."""
    m, p, _, _ = _family(family)
    y = csr_oracle.gemv_csr(m, p)
    for i in range(0, m.rows, max(1, m.rows // 600)):
        s, e = m.rp[i], m.rp[i + 1]
        if e == s:
            assert _bits(y[i]) == 0
            continue
        cols, vals = m.col[s:e], m.val[s:e]
        exact = sum(Fraction(float(a)) * Fraction(float(p[c])) for a, c in zip(vals, cols))
        L = int(np.bincount(cols & 63).max())
        mag = sum(abs(Fraction(float(a)) * Fraction(float(p[c]))) for a, c in zip(vals, cols))
        assert abs(Fraction(float(y[i])) - Fraction(float(exact))) <= (L + 7) * Fraction(U) * mag, i


@pytest.mark.parametrize("n", EDGE_SIZES)
def test_edge_matrix_reaches_its_edges(n):
    """the edge family holds what it promises (for the sizes that have room for it)"""
    A = edge_matrix(n, 7 + n)
    first, last, widths, _ = edge_coverage(A)
    assert last >= set(range(16))
    assert first >= set(range(min(64, n)))
    if n >= 257:
        assert np.count_nonzero(A[:, 0]) and np.count_nonzero(A[:, n - 1])
        nz = np.count_nonzero(A, axis=1)
        assert (nz == n).any()                 # the full row
        assert (nz == 0).sum() > 3 * max(1, min(32, -(-n // GRID)))
    for w in (256, 512, 640, 704, 1024, 2048):
        for k in (1, 2):
            for extra in (0, 16):
                if k * w + extra <= n and n >= 4000:
                    assert k * w + extra in widths, (w, k, extra)


def test_fallback_rows_straddle_the_table():
    """the edited rows of the kWinBlocks tests lie in blocks < 128 and >= 128 of one CTA"""
    for n in (75776, 80000):
        rows = set(fallback_rows(n))
        blocks = {(c, b) for c, b, s, e in block_bounds(n, GRID, 4) for r in rows if s <= r < e}
        if n == 80000:
            assert any(b >= WIN_BLOCKS for _, b in blocks)
        ctas = {c for c, _ in blocks}
        assert len(ctas) == 3


def test_csr_row_matrix_has_every_length():
    n = 5000
    irn, jcn, val = csr_row_matrix(n)
    lens = np.bincount(irn, minlength=n)
    assert set(CSR_LENGTHS) <= set(lens.tolist())
    m = csr_oracle.csr_from_coo(n, irn, jcn, val, symmetric=False)
    assert np.array_equal(np.diff(m.rp), lens)  # every entry stored, explicit zeros included
    zero = (val == 0.0)
    assert zero.any() and (np.signbit(val) & zero).any()
    for L in (8, 9):                           # rows that cross 8/9 only through a stored zero
        assert any(lens[r] == L and (val[irn == r] == 0.0).any() for r in np.unique(irn[zero]))


# ============================================================================ B: GPU, dense windows
def _gemv_all_variants(cgb, O, ctx, p, y_ref):
    """every gemv variant (tma, tensor map, ldg, no-hint) == y_ref, chunk partials likewise"""
    cp_ref = O.chunk_partials(p, y_ref)
    names = cgb.gemv_variants()
    for fam in ("tma_", "tma2_", "ldg_", "tm2d_", "_nohint"):
        assert any(fam in nm for nm in names), fam
    for v, name in enumerate(names):
        ctx.set_option("gemv_variant", v)
        y, cp, pap = ctx.gemv(p, want_partials=True)
        assert _same(y, y_ref), (name, np.flatnonzero(_differ(y, y_ref))[:8])
        assert _same(cp, cp_ref), name
        assert _same(pap, O.det_sum(cp_ref)), name


@pytest.mark.gpu
@pytest.mark.parametrize("special", [False, True])
@pytest.mark.parametrize("n", EDGE_SIZES)
def test_edge_windows_every_variant(cgb, O, n, special):
    A = edge_matrix(n, 7 + n)
    first, last, _, _ = edge_coverage(A)
    assert first >= set(range(min(64, n))) and last >= set(range(16))   # every residue present
    if special:
        rows = add_special_rows(A)
    p = edge_vector(n, n)
    y_ref = O.gemv(A, p)
    if special:
        assert np.isnan(y_ref[rows[1]]) and np.isinf(y_ref[rows[2]]) and y_ref[rows[0]] != 0.0
        assert _bits(y_ref[rows[4]]) == 0
    with cgb.Context(n, 0, 1, 0) as ctx:
        assert ctx.layout().ld - n == (-n) % 16
        ctx.set_matrix_rows(A)
        assert ctx.get_option("envelope_doubles") == envelope_doubles(A)
        _gemv_all_variants(cgb, O, ctx, p, y_ref)


@pytest.mark.gpu
@pytest.mark.parametrize("n", STRESS_SIZES)
def test_graph_only_shapes_solve_stress(cgb, O, n):
    """Whole solves on every tile shape the persistent kernel does not have (graph schedule only):
    2, 3 and 6 stages meet zero blocks, far-apart envelopes and partial last tiles."""
    A = stress_matrix(n, 100 + n)
    b = stress_rhs(A, O)
    max_iter = min(n, 60)
    graph_only = []
    with cgb.Context(n, 0, 1, 0) as ctx:
        for v, name in enumerate(cgb.gemv_variants()):
            ctx.set_option("gemv_variant", v)
            if ctx.get_option("schedule_in_use") != 1:
                graph_only.append((v, name))
    names = {nm for _, nm in graph_only}
    assert {"tma_w8r1c512s6", "tma_w8r2c256s6", "tma_w8r4c256s3", "tma_w4r8c256s3",
            "tma_w8r2c512s3_nohint"} <= names, names
    ref = None
    for v, name in graph_only:
        with cgb.Context(n, 0, 1, 0) as ctx:
            ctx.set_option("gemv_variant", v)
            ctx.set_option("schedule", 0)
            ctx.set_matrix_coo(*to_coo(A), symmetric=False)
            ctx.set_rhs(b)
            x = np.zeros(n)
            info, hist = ctx.solve(x, max_iter=max_iter, tol=1e-10, history=True)
            nx, rr = ctx.residual_check()
            nblk = ctx.layout().nblk
        if ref is None:
            ref = O.solve(A, b, max_iter=max_iter, nranks=1, nblk=nblk)
            assert np.all(np.isfinite(ref.x))
        assert info.k == ref.k and bool(info.converged) == ref.converged, name
        assert _same(hist, ref.hist) and _same(x, ref.x), name
        assert _same([info.rsold, info.rsnew, nx, rr], [ref.rsold, ref.rsnew, ref.norm_x, ref.rel_resid]), name


# ============================================================================ C: GPU, kWinBlocks
def _variant(cgb, name):
    return cgb.gemv_variants().index(name)


def _same_as_csr_oracle(ctx, m, b, max_iter):
    x = np.zeros(m.n)
    info, hist = ctx.solve(x, max_iter=max_iter, tol=1e-10, history=True)
    nx, rr = ctx.residual_check()
    ref = csr_oracle.solve_csr(m, b, max_iter=max_iter)
    assert np.all(np.isfinite(ref.x)) and info.k == ref.k == max_iter
    assert _same(hist, ref.hist) and _same(x, ref.x)
    assert _same([info.rsold, info.rsnew, nx, rr], [ref.rsold, ref.rsnew, ref.norm_x, ref.rel_resid])


def _upload_rows(ctx, new):
    for i, r in sorted(new.items()):
        ctx.set_matrix_rows(r[None, :], first_row=i)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_window_table_fallback_graph(cgb, O):
    """Graph schedule, tma_w4r1c2048s2 at N = 80000 (51 GB of A): a CTA has 540 rows in 135 blocks of
    4, so blocks 128 .. 134 are past the window table and stream full rows.  Rows widened with far
    entries in blocks on both sides of 128 in the same CTA; mat-vec and a 20-iteration solve ==
    the CSR oracle bit for bit."""
    n = 80000
    rows = fallback_rows(n)
    m, new = lap2d_with_far_rows(n, rows)
    b = O.init_source_term(n)
    p = edge_vector(n, n)
    with cgb.Context(n, 0, 1, 0) as ctx:
        lay = ctx.layout()
        if lay.sm_count != GRID:
            pytest.skip("the split is stated for 148 SMs")
        ctx.set_option("gemv_variant", _variant(cgb, "tma_w4r1c2048s2"))
        ctx.set_option("schedule", 0)
        assert ctx.get_option("schedule_in_use") == 0 and ctx.layout().nblk == GRID
        where = {(c, bk) for c, bk, s, e in block_bounds(n, ctx.layout().nblk, 4) for r in rows if s <= r < e}
        past = {c for c, bk in where if bk >= WIN_BLOCKS}
        assert any(bk < WIN_BLOCKS and c in past for c, bk in where), where
        ctx.generate_lap2d()
        _upload_rows(ctx, new)
        y, cp, pap = ctx.gemv(p, want_partials=True)
        y_ref = csr_oracle.gemv_csr(m, p)
        assert _same(y, y_ref), np.flatnonzero(_differ(y, y_ref))[:8]
        assert _same(cp, O.chunk_partials(p, y_ref))
        ctx.set_rhs(b)
        _same_as_csr_oracle(ctx, m, b, 20)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_window_table_fallback_persistent(cgb, O):
    """Persistent kernel, tma_w4r1c2048s2 at N = 75776 (the kernel's size limit): the static split
    gives every CTA exactly 512 rows = 128 blocks, so any row the re-balancing moves in crosses into
    the blocks past the window table.  A few widened rows make their CTAs slower, so others take
    rows.  64 iterations == the CSR oracle; the trace shows a CTA with more than 512 rows."""
    n = 75776
    m, new = lap2d_with_far_rows(n, fallback_rows(n))
    b = O.init_source_term(n)
    with cgb.Context(n, 0, 1, 0) as ctx:
        if ctx.layout().sm_count != GRID:
            pytest.skip("the persistent kernel's size limit is stated for 148 SMs")
        ctx.set_option("gemv_variant", _variant(cgb, "tma_w4r1c2048s2"))
        ctx.set_option("schedule", 1)
        ctx.set_option("balance", 1)
        ctx.set_option("trace", 64)
        assert ctx.get_option("schedule_in_use") == 1
        ctx.generate_lap2d()
        _upload_rows(ctx, new)
        ctx.set_rhs(b)
        _same_as_csr_oracle(ctx, m, b, 64)
        rec, seen = ctx.trace_read(0)
    nrows = (rec[..., 7] >> np.uint64(32)).astype(np.int64)
    tot = nrows.sum(axis=1)
    assert seen > 0 and (tot > 0).sum() >= 32 and (tot[tot > 0] == n).all()  # iterations, all rows
    assert nrows.max() > 4 * WIN_BLOCKS, nrows.max()      # some CTA ran blocks >= 128


# ============================================================================ D: GPU, CSR row paths
@pytest.mark.gpu
def test_csr_row_lengths_and_bucket_patterns(cgb, O):
    n = 5000
    irn, jcn, val = csr_row_matrix(n)
    lens = np.bincount(irn, minlength=n)
    assert set(CSR_LENGTHS) <= set(lens.tolist())
    m = csr_oracle.csr_from_coo(n, irn, jcn, val, symmetric=False)
    p = edge_vector(n, 3)
    y_ref = csr_oracle.gemv_csr(m, p)
    with cgb.Context(n) as d, cgb.Context(n, storage="csr") as c:
        d.set_matrix_coo(irn, jcn, val, symmetric=False)
        c.set_matrix_coo(irn, jcn, val, symmetric=False)
        assert c.nnz() == irn.size
        yd, pd, sd = d.gemv(p, want_partials=True)
        yc, pc, sc = c.gemv(p, want_partials=True)
    assert _same(yc, y_ref), np.flatnonzero(_differ(yc, y_ref))[:8]
    assert _same(yd, y_ref) and _same(pc, pd) and _same(sc, sd)
    assert _same(pc, O.chunk_partials(p, y_ref))


@pytest.mark.gpu
def test_csr_solve_rows_of_7_to_9(cgb, O):
    n = 3000
    irn, jcn, val = csr_solve_matrix(n)
    assert {7, 8, 9} == set(np.bincount(irn, minlength=n).tolist())
    m = csr_oracle.csr_from_coo(n, irn, jcn, val, symmetric=False)
    b = O.init_source_term(n) + 1.0
    with cgb.Context(n, storage="csr") as c:
        c.set_matrix_coo(irn, jcn, val, symmetric=False)
        c.set_rhs(b)
        _same_as_csr_oracle(c, m, b, 50)


# ============================================================================ E: GPU, rank shards
@pytest.mark.gpu
@pytest.mark.parametrize("rank", [0, 2])
def test_rank_shard_envelopes(cgb, O, rank):
    """A rank of 3 holds only its rows; their envelopes, then a 5-row write straddling the shard's
    first (rank 2) or last (rank 0) row: only the rows inside are written and re-enveloped."""
    n = 1001
    A = stress_matrix(n, 17)
    W = stress_matrix(n, 29)
    with cgb.Context(n, rank, 3, 0) as ctx:
        lay = ctx.layout()
        r0, rows = lay.row0, lay.rows
        assert (r0, rows) == (O.partition(n, 3)[0][rank], O.partition(n, 3)[1][rank])
        ctx.set_matrix_rows(A)
        assert ctx.get_option("envelope_doubles") == envelope_doubles(A[r0:r0 + rows])
        M = A.copy()
        for first in (r0 - 2, r0 + rows - 3):
            if first < 0 or first + 5 > n:
                continue
            ctx.set_matrix_rows(W[first:first + 5], first_row=first)
            M[first:first + 5] = W[first:first + 5]
            assert ctx.get_option("envelope_doubles") == envelope_doubles(M[r0:r0 + rows]), first
        assert _same(ctx.get_matrix_rows(r0, rows), M[r0:r0 + rows])
