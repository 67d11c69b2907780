"""Device solves (cgb_solve_device, cgb_solve_block_device): CUDA tensors in and out, ordered on the
caller's stream, the loop's stop decision taken on the device.  Every solve must equal, bit for bit,
the host API's solve on the same context -- k, converged, rsold, rsnew, iterations, the r'r history
and x -- and the CSR oracle's where the oracle applies (a NaN only has to meet a NaN there)."""
import ctypes

import numpy as np
import pytest

import csr_oracle
from test_gpu_block import _lap2d_inputs, _ragged_coo, _stop_apart


def _bits(v):
    return np.asarray(v, dtype=np.float64).view(np.uint64)


def _eq(a, b):
    return np.array_equal(_bits(a), _bits(b))


def _eq_nan(a, b):
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    na, nb = np.isnan(a), np.isnan(b)
    return a.shape == b.shape and np.array_equal(na, nb) and np.array_equal(_bits(a[~na]), _bits(b[~nb]))


def _key(info):
    return (info.k, bool(info.converged), info.iterations)


@pytest.fixture(scope="module")
def torch():
    import torch
    return torch


def _gpu(torch, a):
    return torch.tensor(np.asarray(a, dtype=np.float64), device="cuda:0")


def _device(torch, ctx, b, x0, max_iter, tol):
    x = _gpu(torch, x0)
    info, hist = ctx.solve_device(x, _gpu(torch, b), max_iter, tol=tol, history=True).result()
    return info, hist, x.cpu().numpy()


def _host(ctx, b, x0, max_iter, tol):
    ctx.set_rhs(b)
    x = np.array(x0, dtype=np.float64)
    info, hist = ctx.solve(x, max_iter=max_iter, tol=tol, history=True)
    return info, hist, x


def _same(d, h):
    (di, dh, dx), (hi, hh, hx) = d, h
    assert _key(di) == _key(hi)
    assert _eq([di.rsold, di.rsnew], [hi.rsold, hi.rsnew])
    assert _eq(dh, hh) and _eq(dx, hx)


def _like_oracle(d, ref):
    info, hist, x = d
    assert _key(info) == (ref.k, ref.converged, len(ref.hist))
    assert _eq_nan(hist, ref.hist) and _eq_nan(x, ref.x) and _eq_nan([info.rsold, info.rsnew], [ref.rsold, ref.rsnew])


# dense on the persistent kernel, dense on the graph schedule, CSR (graph schedule)
CONFIGS = {"dense_persist": ("dense", {}), "dense_graph": ("dense", {"schedule": 0}), "csr": ("csr", {})}


def _ctx(cgb, n, cfg, coo=None):
    storage, opts = CONFIGS[cfg]
    ctx = cgb.Context(n, storage=storage)
    if coo is None:
        ctx.generate_lap2d()
    else:
        ctx.set_matrix_coo(*coo, symmetric=False)
    for k, v in opts.items():
        ctx.set_option(k, v)
    assert ctx.get_option("schedule_in_use") == (1 if cfg == "dense_persist" else 0)
    return ctx


# --------------------------------------------------------------------------- bits
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("cfg", list(CONFIGS))
@pytest.mark.parametrize("n", [17, 1000, 4099])
def test_device_solve_equals_host_and_oracle(cgb, O, torch, n, cfg):
    m = csr_oracle.generate_lap2d_csr(n)
    b = O.init_source_term(n)
    x0 = 1e-3 * np.random.default_rng(n).standard_normal(n)
    with _ctx(cgb, n, cfg) as ctx:
        for start in (np.zeros(n), x0):
            d = _device(torch, ctx, b, start, n, 1e-10)   # first: nothing of the host solve is reused
            _same(d, _host(ctx, b, start, n, 1e-10))
            _like_oracle(d, csr_oracle.solve_csr(m, b, start, max_iter=n, tol=1e-10))
        assert d[0].seconds > 0.0


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_device_solve_ragged_csr_matrix(cgb, torch, cfg):
    n = 3001
    irn, jcn, val, empty = _ragged_coo(n, 11)
    m = csr_oracle.csr_from_coo(n, irn, jcn, val, False)
    rng = np.random.default_rng(12)
    b = rng.standard_normal(n)
    b[empty] = 0.0
    x0 = 1e-2 * rng.standard_normal(n)
    with _ctx(cgb, n, cfg, (irn, jcn, val)) as ctx:
        d = _device(torch, ctx, b, x0, 120, 1e-10)
        _same(d, _host(ctx, b, x0, 120, 1e-10))
    _like_oracle(d, csr_oracle.solve_csr(m, b, x0, max_iter=120, tol=1e-10))


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_device_solve_stop_apart_columns(cgb, O, torch, cfg):
    """k = 2, max_iter, the NEARZERO clamp every iteration, NaN (b = 0 from x0 = 0), k = 172"""
    n, coo, m, B, max_iter = _stop_apart(O)
    with _ctx(cgb, n, cfg, coo) as ctx:
        got = []
        for j in range(B.shape[0]):
            d = _device(torch, ctx, B[j], np.zeros(n), max_iter, 1e-10)
            _same(d, _host(ctx, B[j], np.zeros(n), max_iter, 1e-10))
            if cfg == "csr":   # a NaN p makes a dense row NaN where the CSR row stays finite (DESIGN 3.7)
                _like_oracle(d, csr_oracle.solve_csr(m, B[j], None, max_iter=max_iter, tol=1e-10))
            got.append((d[0].k, bool(d[0].converged)))
    assert got == [(2, True), (max_iter, False), (max_iter, False), (max_iter, False), (172, True)]


# --------------------------------------------------------------------------- loop length
GRAPH_OPTS = [{}, {"poll_every": 5, "graph_unroll": 3}, {"poll_every": 1, "graph_unroll": 1},
              {"graph_unroll": 7}, {"poll_every": 4, "pdl": 0}]


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("cfg", ["dense_graph", "csr"])
@pytest.mark.parametrize("opts", GRAPH_OPTS)
def test_device_loop_runs_exactly_max_iter_bodies(cgb, O, torch, cfg, opts):
    n = 1000
    b = O.init_source_term(n)
    with _ctx(cgb, n, cfg) as ctx:
        for k, v in opts.items():
            ctx.set_option(k, v)
        u = min(ctx.get_option("graph_unroll"), ctx.get_option("poll_every"))
        for max_iter in sorted({0, 1, max(u - 1, 0), u, u + 1, 2 * u + 3}):
            replays = ctx.get_option("graph_replays")
            d = _device(torch, ctx, b, np.zeros(n), max_iter, 0.0)   # tol = 0: never converges
            assert ctx.get_option("graph_replays") == replays + 1
            assert _key(d[0]) == (max_iter, False, max_iter) and len(d[1]) == max_iter
            _same(d, _host(ctx, b, np.zeros(n), max_iter, 0.0))
        # a solve that stops at every offset inside a body: tol just above sqrt(r'r) of loop index k
        _, h, _ = _host(ctx, b, np.zeros(n), 200, 0.0)
        norms = np.sqrt(h)
        offsets = set()
        for k in range(20, 200):
            tol = float(np.nextafter(norms[k], np.inf))
            if k % u in offsets or norms[:k].min() < tol:
                continue
            d = _device(torch, ctx, b, np.zeros(n), 200, tol)
            assert _key(d[0]) == (k, True, k + 1)
            _same(d, _host(ctx, b, np.zeros(n), 200, tol))
            offsets.add(k % u)
            if len(offsets) == u:
                break
        assert offsets == set(range(u))


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_persistent_device_solve_runs_no_graph(cgb, O, torch):
    n = 4096
    b = O.init_source_term(n)
    with _ctx(cgb, n, "dense_persist") as ctx:
        replays = ctx.get_option("graph_replays")
        for max_iter in (0, 1, 37):
            d = _device(torch, ctx, b, np.zeros(n), max_iter, 0.0)
            assert _key(d[0]) == (max_iter, False, max_iter)
            _same(d, _host(ctx, b, np.zeros(n), max_iter, 0.0))
        assert ctx.get_option("graph_replays") == replays


# --------------------------------------------------------------------------- asynchrony
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_device_solve_returns_before_the_stream_gets_there(cgb, O, torch, cfg):
    n = 4099
    b_host = O.init_source_term(n)
    with _ctx(cgb, n, cfg) as ctx:
        src = _gpu(torch, 0.5 * b_host)
        x = torch.zeros(n, dtype=torch.float64, device="cuda:0")
        ctx.solve_device(x, 2.0 * src, n, history=True).result()     # warm-up: same shape and options
        s = torch.cuda.current_stream()
        torch.cuda.synchronize()
        torch.cuda._sleep(100_000_000)                               # ~50 ms of GPU clock cycles
        b = src * 2.0                                                # b made by a torch kernel, no sync
        x.zero_()
        h = ctx.solve_device(x, b, n, history=True)
        ev = torch.cuda.Event()
        ev.record(s)
        assert not ev.query(), "the call waited for the stream"
        info, hist = h.result()
        d = (info, hist, x.cpu().numpy())
        _same(d, _host(ctx, b_host, np.zeros(n), n, 1e-10))


# --------------------------------------------------------------------------- block form
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("nrhs", [1, 3, 8])
def test_block_device_equals_block(cgb, O, torch, nrhs):
    n = 4099
    B, X0 = _lap2d_inputs(O, n, nrhs)
    with _ctx(cgb, n, "csr") as ctx:
        X = _gpu(torch, X0)
        replays = ctx.get_option("graph_replays")
        infos, hist = ctx.solve_block_device(X, _gpu(torch, B), n, history=True).result()
        assert ctx.get_option("graph_replays") == replays + 1
        Xh, infos_h, hist_h = ctx.solve_block(B, X0, max_iter=n, history=True)
    X = X.cpu().numpy()
    for j in range(nrhs):
        assert _key(infos[j]) == _key(infos_h[j]), j
        assert _eq([infos[j].rsold, infos[j].rsnew], [infos_h[j].rsold, infos_h[j].rsnew]), j
        assert _eq(hist[j], hist_h[j]) and _eq(X[j], Xh[j]), j
    assert len({i.seconds for i in infos}) == 1


@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("opts", [{}, {"poll_every": 5, "graph_unroll": 3}])
def test_block_device_stop_apart_columns(cgb, O, torch, opts):
    n, coo, m, B, max_iter = _stop_apart(O)
    with _ctx(cgb, n, "csr", coo) as ctx:
        for k, v in opts.items():
            ctx.set_option(k, v)
        X = torch.zeros((B.shape[0], n), dtype=torch.float64, device="cuda:0")
        infos, hist = ctx.solve_block_device(X, _gpu(torch, B), max_iter, history=True).result()
        Xh, infos_h, hist_h = ctx.solve_block(B, None, max_iter=max_iter, history=True)
    X = X.cpu().numpy()
    assert [_key(i) for i in infos] == [_key(i) for i in infos_h]
    assert _eq(X, Xh) and all(_eq(a, b) for a, b in zip(hist, hist_h))
    assert [(i.k, bool(i.converged)) for i in infos] == [(2, True), (max_iter, False), (max_iter, False),
                                                         (max_iter, False), (172, True)]


# --------------------------------------------------------------------------- interplay
@pytest.mark.gpu
@pytest.mark.timeout(900)
@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_device_and_host_solves_share_a_context(cgb, O, torch, cfg):
    n = 4096
    rng = np.random.default_rng(3)
    bs = [O.init_source_term(n), rng.standard_normal(n), O.init_source_term(n, 0.37 / n)]
    with _ctx(cgb, n, cfg) as ctx:
        refs = []
        for b in bs:
            h = _host(ctx, b, np.zeros(n), n, 1e-10)
            refs.append((h, ctx.residual_check()))
        for (h, check), b in zip(refs, bs):        # device, host, device, ... on one context
            d = _device(torch, ctx, b, np.zeros(n), n, 1e-10)
            _same(d, h)
            assert _eq(ctx.residual_check(), check)  # the device solve left its b and x in the context
            _same(_host(ctx, b, np.zeros(n), n, 1e-10), h)
            assert _eq(ctx.residual_check(), check)


@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_device_solves_keep_block_and_single_apart(cgb, O, torch):
    n = 4096
    b = O.init_source_term(n)
    B, X0 = _lap2d_inputs(O, n, 3)
    with _ctx(cgb, n, "csr") as ctx:
        single = _device(torch, ctx, b, np.zeros(n), n, 1e-10)
        check = ctx.residual_check()
        Xh, infos_h, hist_h = ctx.solve_block(B, X0, max_iter=n, history=True)
        X = _gpu(torch, X0)
        infos, hist = ctx.solve_block_device(X, _gpu(torch, B), n, history=True).result()
        assert _eq(ctx.residual_check(), check)          # neither block solve touched the single solve
        _same(_device(torch, ctx, b, np.zeros(n), n, 1e-10), single)
        X2 = _gpu(torch, X0)
        infos2, hist2 = ctx.solve_block_device(X2, _gpu(torch, B), n, history=True).result()
    for j in range(3):
        assert _key(infos[j]) == _key(infos_h[j]) == _key(infos2[j])
        assert _eq(hist[j], hist_h[j]) and _eq(hist2[j], hist_h[j])
    assert _eq(X.cpu().numpy(), Xh) and _eq(X2.cpu().numpy(), Xh)


# --------------------------------------------------------------------------- refusals
@pytest.mark.gpu
@pytest.mark.timeout(900)
def test_device_solve_refusals(cgb, O, torch):
    n = 1000
    dp = ctypes.c_void_p
    b = _gpu(torch, O.init_source_term(n))
    x = torch.zeros(n, dtype=torch.float64, device="cuda:0")
    B = torch.stack([b, b])
    X = torch.zeros_like(B)
    info = torch.zeros(8 * 48, dtype=torch.uint8, device="cuda:0")
    host = np.zeros(8 * n)

    def single(ctx, bp=b.data_ptr(), xp=x.data_ptr(), max_iter=10, ip=info.data_ptr(), hp=None):
        return ctx._lib.cgb_solve_device(ctx._h, bp, xp, max_iter, 1e-10, hp, ip, None)

    def block(ctx, nrhs=2, bp=B.data_ptr(), xp=X.data_ptr(), max_iter=10, ip=info.data_ptr()):
        return ctx._lib.cgb_solve_block_device(ctx._h, nrhs, bp, xp, max_iter, 1e-10, None, ip, None)

    for storage in ("dense", "csr"):
        with cgb.Context(n, 0, 2, 0, storage=storage) as w:
            w.generate_lap2d()
            assert single(w) == 2 and "rank" in w._lib.cgb_last_error().decode()
            assert block(w) == 2
    with cgb.Context(n) as d:
        assert single(d) == 2 and b"matrix" in d._lib.cgb_last_error()
        d.generate_lap2d()
        assert block(d) == 2 and b"CSR" in d._lib.cgb_last_error()
        d.set_rhs(O.init_source_term(n))
        d.solve_begin(np.zeros(n), 10)
        assert single(d) == 2
        d.solve_end()
    with cgb.Context(n, storage="csr") as c:
        assert block(c) == 2 and b"matrix" in c._lib.cgb_last_error()
        c.generate_lap2d()
        hp = host.ctypes.data
        for args in ({"bp": None}, {"xp": None}, {"ip": None}, {"bp": hp}, {"xp": hp}, {"ip": hp}, {"hp": hp},
                     {"max_iter": -1}):
            assert single(c, **args) == 1, args
        for args in ({"nrhs": 0}, {"nrhs": 9}, {"bp": None}, {"xp": hp}, {"ip": hp}, {"max_iter": -1}):
            assert block(c, **args) == 1, args
        pinned = torch.zeros(n, dtype=torch.float64).pin_memory()
        assert single(c, xp=pinned.data_ptr()) == 1 and b"host" in c._lib.cgb_last_error()
        with pytest.raises(TypeError):
            c.solve_device(x.cpu(), b, 10)
        c.solve_block_begin(B.cpu().numpy(), max_iter=10)
        assert single(c) == 2 and block(c) == 2
        c.iterate(10)
        c.solve_block_end()
        c.set_rhs(O.init_source_term(n))
        c.solve_begin(np.zeros(n), 10)
        assert single(c) == 2 and block(c) == 2
        c.solve_end()
        assert single(c) == 0 and block(c) == 0
        torch.cuda.synchronize()
        assert c.launch_count() > 0


# --------------------------------------------------------------------------- without a GPU
def test_device_solve_without_gpu_fails_loudly(cgb):
    try:
        if cgb.device_count() > 0:
            pytest.skip("a GPU is present")
    except cgb.CgbError:
        pass
    lib = cgb.load()
    buf = np.zeros(64)
    p = buf.ctypes.data
    assert lib.cgb_solve_device(None, p, p, 10, 1e-10, None, p, None) == 3
    assert lib.cgb_solve_block_device(None, 2, p, p, 10, 1e-10, None, p, None) == 3
    assert np.all(buf == 0.0)
