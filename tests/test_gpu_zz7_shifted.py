"""spmv_b200_spmv_shifted: y <- alpha (A - sigma I) x + beta y on square handles, with x . y and y . y, taken by the
kernel that stores each final y value.

y is compared by bits with the contract computed in numpy from spmv()'s bits on the same handle:
fl(fl(alpha fl(s - fl(sigma x))) + fl(beta y_old)), sigma == 0 without the shift term.  With sigma == 0, y and both dots
must equal spmv_b200_spmv_axpby's y and spmv_b200_spmv_axpby_dot's dot with w = x and w = y, bit for bit.  On integer
data the dots must equal the int64 sums exactly; on real data they must lie within the bound of the header (as in
test_gpu_zz6_axpby_dot).

The kernel-instance configurations use matrices that are not square.  Every configuration here keeps its matrix's rows
(row lengths, so the layouts and kernels spmv() picks) and makes it square: n = m, with columns taken modulo m where
n > m.
"""
import functools
import types

import numpy as np
import pytest

from conftest import bits_equal
from spmv_b200 import api
from test_gpu_kernel_instances import DTYPES, assert_same, matrix, normalise, options, spmv_instances
from test_gpu_zz5_axpby import ALL, BY_NAME, SCRATCH, old_y, tdtype
from test_gpu_zz6_axpby_dot import assert_within_bound, dot_table, int_dot, int_old_y

gpu = pytest.mark.gpu

FAMILIES = frozenset(["csr_vector_shift_kernel", "band_reduce_shift_kernel", "sell_shift_kernel",
                      "csr_tail_shift_kernel", "shift_kernel"])
INT_TRIPLES = [(1.0, 2.0, 0.0), (2.0, -3.0, -1.0), (-1.0, 1.0, 1.0), (2.0, 0.0, -3.0)]
REAL_TRIPLES = [(0.1, 0.3, -0.7), (2.0 / 3.0, -1.25, -1.0), (1.5, 0.0, 1.0), (-1.5, 0.5, 0.0)]


@functools.lru_cache(maxsize=None)
def square(name):
    """The kernel-instance matrix `name` with its rows kept and n = m."""
    A = matrix(name)
    m = A.m
    col = A.col % m if A.n > m else A.col.copy()
    x = np.zeros(m, dtype=np.int64)
    k = min(m, A.n)
    x[:k] = A.x[:k]
    x[k:] = np.random.default_rng(m).integers(-4, 5, m - k)
    return types.SimpleNamespace(name=name, m=m, n=m, rowptr=A.rowptr, col=col.astype(np.int32), a=A.a, x=x,
                                 nnz=A.nnz)


def make(cfg, dt):
    """The handle of `cfg` on the square matrix at precision dt, and s = spmv()'s y for its integer x."""
    import torch
    A = square(cfg.mat)
    xv = A.x.astype(dt)
    with options(cfg.opts):  # held through the first spmv: seg_ctas is read at the first band-segment launch
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(dt), cfg.method)
        try:
            if "kernel" in cfg.expect:
                assert h.info("kernel") == cfg.expect["kernel"], (cfg.name, h.kernel)
            if cfg.host:
                s = np.full(A.m, 0.5, dtype=dt)
                h.spmv(xv, s)
            else:
                yd = torch.full((A.m,), 0.5, dtype=tdtype(dt), device="cuda")
                h.spmv(torch.from_numpy(xv).cuda(), yd)
                h.sync()
                s = yd.cpu().numpy()
        except BaseException:
            h.destroy()
            raise
    return s, h, A


def formula(s, x, alpha, sigma, beta, y_old):
    """The contract in numpy: alpha, sigma and beta rounded to the precision first, every operation rounded once."""
    dt = y_old.dtype.type
    a, sg, b = dt(alpha), dt(sigma), dt(beta)
    with np.errstate(all="ignore"):
        if a == 0:
            return np.zeros_like(y_old) if b == 0 else b * y_old
        v = s if sg == 0 else s - sg * x
        return a * v if b == 0 else a * v + b * y_old


def call(h, alpha, sigma, x, beta, y_old, host, dots=True, dots_on_device=False):
    """One spmv_shifted with host or device x / y; returns (y, (x . y, y . y)), or (y, None) without dots."""
    import torch
    if host:
        y = y_old.copy()
        if not dots:  # (the Python wrapper always takes the dots: NULL dots through the C entry point)
            x = np.ascontiguousarray(x)
            assert api.lib().spmv_b200_spmv_shifted(h.h, alpha, sigma, x.ctypes.data, beta, y.ctypes.data, None) == 0
            return y, None
        return y, h.spmv_shifted(alpha, sigma, x, beta, y)
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    yd = torch.from_numpy(y_old.copy()).cuda()
    if not dots:
        assert api.lib().spmv_b200_spmv_shifted(h.h, alpha, sigma, xd.data_ptr(), beta, yd.data_ptr(), None) == 0
        h.sync()
        return yd.cpu().numpy(), None
    if dots_on_device:
        dd = torch.full((2,), 0.5, dtype=torch.float64, device="cuda")
        assert h.spmv_shifted(alpha, sigma, xd, beta, yd, dd) is None
        h.sync()
        return yd.cpu().numpy(), tuple(dd.cpu().numpy().tolist())
    d = h.spmv_shifted(alpha, sigma, xd, beta, yd)
    return yd.cpu().numpy(), d


def axpby_dot_ref(h, alpha, x, beta, y_old, w_is_x):
    """spmv_b200_spmv_axpby_dot's (y, dot) with w = x or w = y, device pointers."""
    import torch
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    yd = torch.from_numpy(y_old.copy()).cuda()
    d = h.spmv_axpby_dot(alpha, xd, beta, yd, xd if w_is_x else yd)
    return yd.cpu().numpy(), d


def same_double(a, b):
    return np.float64(a).tobytes() == np.float64(b).tobytes()


# ---------------------------------------------------------------------------------------------------------------------
# 1-3. every configuration: y bits against the formula, sigma == 0 against axpby / axpby_dot, exact and bounded dots
# ---------------------------------------------------------------------------------------------------------------------
def check_config(cfg, dt):
    import torch
    tag = f"{cfg.name}/{np.dtype(dt).name}"
    s, h, A = make(cfg, dt)
    try:
        xv = A.x.astype(dt)
        peers = None
        if cfg.peers:
            peers = [torch.full((A.m,), 0.25, dtype=tdtype(dt), device="cuda") for _ in range(2)]
            h.set_y_peers([p.data_ptr() for p in peers])
        assert h.info("dot_path") == dot_table(h, cfg.peers), (tag, h.info("dot_path"))
        for i, (alpha, sigma, beta) in enumerate(INT_TRIPLES):
            y_old = int_old_y(A.m, dt, seed=i)
            y, (xy, yy) = call(h, alpha, sigma, xv, beta, y_old, cfg.host)
            assert_same(y, formula(s, xv, alpha, sigma, beta, y_old), f"{tag} int ({alpha}, {sigma}, {beta})")
            assert xy == int_dot(xv, y) and yy == int_dot(y, y), (tag, alpha, sigma, beta, xy, yy)
        for i, (alpha, sigma, beta) in enumerate(REAL_TRIPLES):
            y_old = old_y(A.m, dt, seed=i)
            y, (xy, yy) = call(h, alpha, sigma, xv, beta, y_old, cfg.host, dots_on_device=not cfg.host and i % 2 == 1)
            assert_same(y, formula(s, xv, alpha, sigma, beta, y_old), f"{tag} ({alpha}, {sigma}, {beta})")
            assert_within_bound(xy, xv, y, f"{tag} x.y ({alpha}, {sigma}, {beta})")
            assert_within_bound(yy, y, y, f"{tag} y.y ({alpha}, {sigma}, {beta})")
            for k, p in enumerate(peers or []):
                assert bits_equal(p.cpu().numpy(), y), (tag, alpha, sigma, beta, k)
            y_nodots, _ = call(h, alpha, sigma, xv, beta, y_old, cfg.host, dots=False)
            assert bits_equal(y_nodots, y), (tag, "without dots", alpha, sigma, beta)
            if sigma == 0:
                for w_is_x, got in ((True, xy), (False, yy)):
                    y_ref, d_ref = axpby_dot_ref(h, alpha, xv, beta, y_old, w_is_x)
                    assert bits_equal(y, y_ref) and same_double(got, d_ref), (tag, "sigma 0", w_is_x, got, d_ref)
        return h.info("dot_path")
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("cfg", ALL, ids=[c.name for c in ALL])
def test_shifted_every_configuration(libpath, cfg, dt):
    check_config(cfg, DTYPES[dt])


# ---------------------------------------------------------------------------------------------------------------------
# 7. reproducible: call after call, on another stream; option "axpby_fused" = 0
# ---------------------------------------------------------------------------------------------------------------------
SOME = ["vector_tpr1", "banded", "bseg40_ctas3_bseg_small", "csr5_sigma8", "sell_v0_nocap", "bins"]


def real_inputs(A, dt, seed):
    rng = np.random.default_rng(seed)
    return rng.standard_normal(A.n).astype(dt), old_y(A.m, dt, seed)


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("name", SOME)
def test_shifted_is_reproducible_across_calls_and_streams(libpath, name, dt):
    import torch
    dt = DTYPES[dt]
    _, h, A = make(BY_NAME[name], dt)
    try:
        x, y_old = real_inputs(A, dt, 3)
        got = [call(h, 0.7, 0.4, x, -1.3, y_old, False) for _ in range(2)]
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        got.append(call(h, 0.7, 0.4, x, -1.3, y_old, False, dots_on_device=True))
        h.set_stream(0)
        for y, d in got[1:]:
            assert bits_equal(y, got[0][0]), name
            assert same_double(d[0], got[0][1][0]) and same_double(d[1], got[0][1][1]), name
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("name", ["vector_tpr1", "sell_v0_nocap", "banded", "bseg3_ctas2_bseg_small"])
def test_option_axpby_fused_0_gives_the_same_bits(libpath, name):
    cfg = BY_NAME[name]
    A = square(cfg.mat)
    x, y_old = real_inputs(A, np.float64, 4)
    out = {}
    for fused in (1, 0):
        with options({**cfg.opts, "axpby_fused": fused}):
            h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(np.float64), cfg.method)
        try:
            out[fused] = call(h, -1.5, 0.25, x, 0.75, y_old, False)
            assert h.info("dot_path") == (dot_table(h, False) if fused else SCRATCH), (name, fused)
        finally:
            h.destroy()
    assert bits_equal(out[0][0], out[1][0]), name
    for fused in (0, 1):
        assert_within_bound(out[fused][1][0], x, out[fused][0], f"{name} fused={fused} x.y")
        assert_within_bound(out[fused][1][1], out[fused][0], out[fused][0], f"{name} fused={fused} y.y")


# ---------------------------------------------------------------------------------------------------------------------
# 4. special cases; 5. argument errors
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "bseg3_ctas2_bseg_small", "csr5_sigma8", "sell_v0_nocap"])
def test_shifted_special_cases(libpath, name, dt):
    dt = DTYPES[dt]
    s, h, A = make(BY_NAME[name], dt)
    try:
        xv = A.x.astype(dt)
        poison = old_y(A.m, dt, seed=9)
        poison[::3], poison[1::3] = np.nan, np.inf
        # beta == 0: the old y is never read
        y, (xy, yy) = call(h, 2.0, -1.0, xv, 0.0, poison, False)
        assert bits_equal(y, formula(s, xv, 2.0, -1.0, 0.0, np.zeros(A.m, dtype=dt))), name
        assert xy == int_dot(xv, y) and yy == int_dot(y, y), name
        # alpha == 0: A is not read, and x only for dots[0]
        y_old = int_old_y(A.m, dt, seed=3)
        y, (xy, yy) = call(h, 0.0, 2.0, xv, -3.0, y_old, False)
        assert bits_equal(y, dt(-3.0) * y_old) and xy == int_dot(xv, y) and yy == int_dot(y, y), name
        xn = xv.copy()
        xn[::3] = np.nan
        y, _ = call(h, 0.0, 2.0, xn, -3.0, y_old, False, dots=False)
        assert bits_equal(y, dt(-3.0) * y_old), name
        # alpha == beta == 0: y = +0 without reading the old y; the dots over those zeros
        for beta in (0.0, -0.0):
            y, (xy, yy) = call(h, 0.0, 2.0, xv, beta, poison, False)
            assert bits_equal(y, np.zeros(A.m, dtype=dt)) and xy == 0.0 and yy == 0.0, name
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("method", [api.Method_Serial, api.Method_Parallel, api.Method_CSR5SPMV])
def test_shifted_empty_matrix_and_no_rows(libpath, method, dt):
    import torch
    dt = DTYPES[dt]
    m = 50
    h = api.Handle(m, m, np.zeros(m + 1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=dt), method)
    x = (np.arange(m) - 20).astype(dt)
    for alpha, sigma, beta in ((-2.0, 3.0, 3.0), (3.0, -1.0, 0.0), (0.0, 2.0, 2.0), (2.0, 0.0, 1.0)):
        y_old = int_old_y(m, dt, seed=4)
        y, (xy, yy) = call(h, alpha, sigma, x, beta, y_old, False)
        assert bits_equal(y, formula(np.zeros(m, dtype=dt), x, alpha, sigma, beta, y_old)), (alpha, sigma, beta)
        assert xy == int_dot(x, y) and yy == int_dot(y, y), (alpha, sigma, beta)
    h.destroy()
    h = api.Handle(0, 0, np.zeros(1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=dt), method)
    xd = torch.ones(1, dtype=tdtype(dt), device="cuda")
    y = torch.full((1,), 0.5, dtype=tdtype(dt), device="cuda")
    dd = torch.full((2,), 0.5, dtype=torch.float64, device="cuda")
    launches = api.launch_count()
    assert h.spmv_shifted(2.0, 1.0, xd, 3.0, y) == (0.0, 0.0)
    h.spmv_shifted(2.0, 1.0, xd, 3.0, y, dd)
    h.sync()
    assert api.launch_count() == launches and y.item() == 0.5
    assert dd.cpu().numpy().tobytes() == np.zeros(2).tobytes()
    h.destroy()


@gpu
def test_shifted_argument_errors_leave_y_and_dots_untouched(libpath):
    import torch
    L = api.lib()
    for name, square_handle in (("vector_tpr4", False), ("vector_tpr1", True)):
        cfg = BY_NAME[name]
        A = square(cfg.mat) if square_handle else matrix(cfg.mat)
        with options(cfg.opts):
            h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(np.float64), cfg.method)
        xd = torch.from_numpy(A.x.astype(np.float64)).cuda()
        y = torch.full((A.m,), 0.5, dtype=torch.float64, device="cuda")
        dd = torch.full((2,), 0.25, dtype=torch.float64, device="cuda")
        hd = np.full(2, 0.25)
        X, Y, D = xd.data_ptr(), y.data_ptr(), dd.data_ptr()
        if square_handle:
            cases = (((X, None, D), "y is NULL"), ((None, Y, D), "x is NULL"), ((Y, Y, D), "same array"),
                     ((X, None, hd.ctypes.data), "y is NULL"), ((None, Y, hd.ctypes.data), "x is NULL"))
        else:
            assert A.m != A.n
            cases = (((X, Y, D), "not square"), ((X, Y, None), "not square"), ((X, Y, hd.ctypes.data), "not square"))
        for args, what in cases:
            api.clear_error()
            assert L.spmv_b200_spmv_shifted(h.h, 1.0, 0.5, args[0], 0.0, args[1], args[2]) == -1, (name, what)
            assert what in api.last_error(), (name, what, api.last_error())
        h.sync()
        assert (y == 0.5).all() and (dd == 0.25).all() and (hd == 0.25).all(), name
        h.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# 6. host and device pointers
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("pin", [0, 1])
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "csr5_sigma8"])
def test_shifted_host_and_device_pointers(libpath, name, pin):
    """Every mix of host and device x, y and dots gives the same bits ("banded" has a 2 MiB y: pinned at the second call
    with "pin_host" = 1)."""
    import torch
    cfg = BY_NAME[name]
    A = square(cfg.mat)
    dt = np.float64
    with options({**cfg.opts, "pin_host": pin}):
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(dt), cfg.method)
    try:
        x, y_old = real_inputs(A, dt, 6)
        want_y, want_d = call(h, -1.5, 0.75, x, 0.75, y_old, False)
        dev = lambda a: torch.from_numpy(a.copy()).cuda()
        hx, hy = x.copy(), y_old.copy()  # one host x and y for the handle's life, as "pin_host" requires
        for xh in (True, False):
            for yh in (True, False):
                for dh in (True, False, None):  # None: no dots
                    xa = hx if xh else dev(x)
                    ya = hy if yh else dev(y_old)
                    dd = torch.zeros(2, dtype=torch.float64, device="cuda") if dh is False else None
                    for _ in range(2):  # the same host buffers again, as a client's loop passes them
                        if yh:
                            ya[:] = y_old
                        else:
                            ya.copy_(dev(y_old))
                        if dh is None:
                            assert api.lib().spmv_b200_spmv_shifted(h.h, -1.5, 0.75, api._addr(xa), 0.75, api._addr(ya),
                                                                    None) == 0
                        else:
                            d = h.spmv_shifted(-1.5, 0.75, xa, 0.75, ya, dd)
                    h.sync()
                    yv = ya if yh else ya.cpu().numpy()
                    tag = f"{name} pin={pin} x={xh} y={yh} dots_host={dh}"
                    assert bits_equal(yv, want_y), tag
                    if dh is not None:
                        d = d if dh else tuple(dd.cpu().numpy().tolist())
                        assert same_double(d[0], want_d[0]) and same_double(d[1], want_d[1]), (tag, d, want_d)
        if name == "banded":
            assert h.info("pinned_host_buffers") == 2 * pin
    finally:
        h.destroy()


@gpu
def test_device_dots_return_without_a_host_synchronisation(libpath):
    import torch
    _, h, A = make(BY_NAME["banded"], np.float64)
    try:
        x, y_old = (torch.from_numpy(a).cuda() for a in real_inputs(A, np.float64, 7))
        dd = torch.zeros(2, dtype=torch.float64, device="cuda")
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        h.spmv_shifted(1.0, 0.5, x, 2.0, y_old, dd)  # warm: allocates the partials
        side.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(2_000_000_000)  # ~1 s of spinning ahead of the call on the handle's stream
        h.spmv_shifted(1.0, 0.5, x, 2.0, y_old, dd)
        assert not side.query(), "the call waited for its stream"
        side.synchronize()
        h.set_stream(0)
    finally:
        h.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# 8. CUDA graphs, peers and spmv() afterwards, allocations
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "bseg3_ctas2_bseg_small", "csr5_sigma8", "sell_v0_nocap"])
def test_shifted_is_cuda_graph_capturable(libpath, name):
    import torch
    _, h, A = make(BY_NAME[name], np.float64)
    try:
        x, y0 = (torch.from_numpy(a).cuda() for a in real_inputs(A, np.float64, 8))
        dots = torch.zeros(3, 2, dtype=torch.float64, device="cuda")
        y = y0.clone()
        for k in range(3):
            h.spmv_shifted(-0.5, 0.25, x, 1.0, y, dots[k])
        h.sync()
        want_y, want_d = y.clone(), dots.clone()
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        g = torch.cuda.CUDAGraph()
        yg, dg = y0.clone(), torch.zeros(3, 2, dtype=torch.float64, device="cuda")
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
            for k in range(3):
                h.spmv_shifted(-0.5, 0.25, x, 1.0, yg, dg[k])
        for _ in range(2):
            yg.copy_(y0)
            dg.zero_()
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(yg.view(torch.int64), want_y.view(torch.int64)), name
            assert torch.equal(dg.view(torch.int64), want_d.view(torch.int64)), name
        h.set_stream(0)
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("name", ["vector_tpr1_peers", "banded", "bseg40_ctas3_bseg_small_peers", "csr5_peers",
                                  "sell_v2_nocap_peers"])
def test_peers_and_later_calls_after_shifted(libpath, name):
    """The peers receive the final y; spmv() afterwards keeps its bits and launches."""
    import torch
    s, h, A = make(BY_NAME[name], np.float64)
    try:
        peers = [torch.full((A.m,), 0.25, dtype=torch.float64, device="cuda") for _ in range(2)]
        h.set_y_peers([p.data_ptr() for p in peers])
        xv = A.x.astype(np.float64)
        x = torch.from_numpy(xv).cuda()
        yd = torch.full((A.m,), 0.5, dtype=torch.float64, device="cuda")
        l0 = api.launch_count()
        h.spmv(x, yd)
        h.sync()
        per_call = api.launch_count() - l0
        assert bits_equal(yd.cpu().numpy(), s), name
        y_old = old_y(A.m, np.float64, seed=1)
        for dots in (True, False):
            y, _ = call(h, 2.0, -0.5, xv, -3.0, y_old, False, dots=dots)
            assert bits_equal(y, formula(s, xv, 2.0, -0.5, -3.0, y_old)), (name, dots)
            for k, p in enumerate(peers):
                assert bits_equal(p.cpu().numpy(), y), (name, dots, k)
        yd.fill_(0.5)
        l0 = api.launch_count()
        h.spmv(x, yd)
        h.sync()
        assert api.launch_count() - l0 == per_call, name
        assert bits_equal(yd.cpu().numpy(), s), name
        for p in peers:
            assert bits_equal(p.cpu().numpy(), s), name
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("name", ["csr5_sigma8", "vector_tpr1", "banded", "bseg3_ctas2_bseg_small", "sell_v0_nocap",
                                  "sell_v2_nocap"])
def test_shifted_allocations(libpath, name):
    """No dots: the scratch array on the scratch pass only; dots: the two partial sets; host dots: the 2 device doubles;
    destroy returns the count to where it was before the handle."""
    import torch
    cfg = BY_NAME[name]
    A = square(cfg.mat)
    x = torch.from_numpy(A.x.astype(np.float64)).cuda()
    y = torch.zeros(A.m, dtype=torch.float64, device="cuda")
    dd = torch.zeros(2, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    base = api.live_allocations()
    with options(cfg.opts):
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(np.float64), cfg.method)
        h.spmv(x, y)
    h.sync()
    held = api.live_allocations()
    scratch = int(h.info("dot_path") == SCRATCH)
    assert api.lib().spmv_b200_spmv_shifted(h.h, 0.5, 0.25, x.data_ptr(), 2.0, y.data_ptr(), None) == 0
    h.sync()
    assert api.live_allocations() == held + scratch, name
    for k in range(2):
        h.spmv_shifted(0.5, 0.25, x, 2.0, y, dd)
        h.sync()
        assert api.live_allocations() == held + scratch + 2, (name, k)
    h.spmv_shifted(0.5, 0.25, x, 2.0, y)
    assert api.live_allocations() == held + scratch + 3, name
    h.destroy()
    assert api.live_allocations() == base, (name, api.live_allocations() - base)


# ---------------------------------------------------------------------------------------------------------------------
# 9. coverage of the shifted kernel instances
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_every_shifted_instance_is_launched(libpath, monkeypatch):
    import torch
    import test_gpu_kernel_instances
    from torch.profiler import ProfilerActivity, profile
    monkeypatch.setattr(test_gpu_kernel_instances, "FAMILIES", FAMILIES)
    want = spmv_instances(libpath)
    monkeypatch.undo()
    assert len(want) == 10, sorted(want)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for cfg in ALL:
            for dt in DTYPES.values():
                _, h, A = make(cfg, dt)
                try:
                    xv = A.x.astype(dt)
                    call(h, 1.5, 0.5, xv, -1.0, old_y(A.m, dt, 0), cfg.host)
                    call(h, 0.0, 0.5, xv, 2.0, old_y(A.m, dt, 0), cfg.host)
                finally:
                    h.destroy()
        torch.cuda.synchronize()
    raw = {e.name for e in prof.events() if "kernel" in e.name}
    if not raw:
        pytest.skip("torch.profiler recorded no CUDA kernels (no CUPTI activity on this machine)")
    seen = {k for k in map(normalise, raw) if k[0] in FAMILIES}
    missing = sorted(want - seen)
    assert not missing, f"{len(missing)} of {len(want)} instances never launched:\n" + \
        "\n".join(f"  {f}<{', '.join(a)}>" for f, a in missing)


# ---------------------------------------------------------------------------------------------------------------------
# 10. Chebyshev iteration and KPM moments on the device
# ---------------------------------------------------------------------------------------------------------------------
def chebyshev(h, b, lo, hi, tol, max_iters=2000, chunk=25):
    """Chebyshev iteration for A x = b (A SPD, spectrum in [lo, hi]), x0 = 0.  The residual obeys the three-term
    recurrence r_{k+1} = alpha_k (A - theta I) r_k + beta_k r_{k-1} (theta, delta the centre and half-width of the
    spectrum, c_k = T_k(theta / delta), alpha_k = -2 c_k / (delta c_{k+1}), beta_k = -c_{k-1} / c_{k+1}), one
    spmv_b200_spmv_shifted per step, which also returns |r_{k+1}|^2 in dots[1]; the iterate follows the same recurrence
    in torch.  The coefficients are host scalars and the dots stay on the device: the host reads |r| once every `chunk`
    steps."""
    import torch
    theta, delta = (hi + lo) / 2, (hi - lo) / 2
    dots = torch.zeros(2, dtype=torch.float64, device="cuda")
    bb = float(torch.dot(b, b))
    r_prev, x_prev = b.clone(), torch.zeros_like(b)
    r, x = torch.empty_like(b), b / theta
    h.spmv_shifted(-1.0 / theta, theta, r_prev, 0.0, r, dots)  # r_1 = (I - A / theta) r_0
    c_prev, c = 1.0, theta / delta
    for k in range(1, max_iters):
        c_next = 2 * theta / delta * c - c_prev
        alpha, beta = -2 * c / (delta * c_next), -c_prev / c_next
        omega, gamma = 2 * theta * c / (delta * c_next), 2 * c / (delta * c_next)
        h.spmv_shifted(alpha, theta, r, beta, r_prev, dots)  # r_prev <- r_{k+1}
        x_prev.mul_(1 - omega).add_(x, alpha=omega).add_(r, alpha=gamma)  # x_prev <- x_{k+1}
        r, r_prev, x, x_prev = r_prev, r, x_prev, x
        c_prev, c = c, c_next
        if k % chunk == 0 and float(dots[1]) <= tol * tol * bb:
            break
    return x


@gpu
def test_chebyshev_iteration_on_the_device(libpath):
    import scipy.sparse as sp
    import scipy.sparse.linalg as spl
    import torch
    from spmv_b200 import matrices as M
    A = M.laplacian2d(32)
    S = sp.csr_matrix((A.val, A.col, A.rowptr), shape=(A.m, A.n))
    ev = np.linalg.eigvalsh(S.toarray())
    lo, hi = 0.999 * ev[0], 1.001 * ev[-1]
    h = api.Handle(A.m, A.n, A.rowptr, A.col, A.val, api.Method_Parallel)
    try:
        b_np = np.random.default_rng(12).standard_normal(A.m)
        b = torch.from_numpy(b_np).cuda()
        xs = [chebyshev(h, b, lo, hi, 1e-12) for _ in range(2)]
        torch.cuda.synchronize()
        assert torch.equal(xs[0].view(torch.int64), xs[1].view(torch.int64))
        x = xs[0].cpu().numpy()
        assert np.linalg.norm(b_np - S @ x) / np.linalg.norm(b_np) < 1e-10
        ref = spl.spsolve(S.tocsc(), b_np)
        assert np.max(np.abs(x - ref)) <= 1e-8 * np.max(np.abs(ref))
    finally:
        h.destroy()


@gpu
def test_kpm_moments_match_a_dense_recurrence(libpath):
    """mu_n = v . T_n(H~) v, H~ = (A - c I) / e: two moments per step from t_k . t_{k+1} and |t_{k+1}|^2
    (mu_{2k+1} = 2 t_k . t_{k+1} - mu_1, mu_{2k+2} = 2 t_{k+1} . t_{k+1} - mu_0), against the dense recurrence in
    numpy."""
    import torch
    from spmv_b200 import matrices as M
    A = M.laplacian2d(12)
    D = np.zeros((A.m, A.m))
    for i in range(A.m):
        D[i, A.col[A.rowptr[i]:A.rowptr[i + 1]]] = A.val[A.rowptr[i]:A.rowptr[i + 1]]
    c, e = 4.0, 4.1
    Ht = (D - c * np.eye(A.m)) / e
    v = np.random.default_rng(13).standard_normal(A.m)
    v /= np.linalg.norm(v)
    K = 40
    mu_ref = np.zeros(2 * K + 2)
    t_prev, t = v, Ht @ v
    mu_ref[0], mu_ref[1] = v @ v, v @ t
    for n in range(2, 2 * K + 2):
        t_prev, t = t, 2 * Ht @ t - t_prev
        mu_ref[n] = v @ t
    h = api.Handle(A.m, A.n, A.rowptr, A.col, A.val, api.Method_Parallel)
    try:
        dots = torch.zeros(K + 1, 2, dtype=torch.float64, device="cuda")
        t_prev, t = torch.from_numpy(v).cuda(), torch.empty(A.m, dtype=torch.float64, device="cuda")
        h.spmv_shifted(1.0 / e, c, t_prev, 0.0, t, dots[0])  # t_1 = H~ t_0
        for k in range(1, K + 1):
            h.spmv_shifted(2.0 / e, c, t, -1.0, t_prev, dots[k])  # t_prev <- t_{k+1}
            t, t_prev = t_prev, t
        d = dots.cpu().numpy()
        mu0 = float(v @ v)
        mu1 = d[0, 0]
        mu = np.zeros(2 * K + 2)
        mu[0], mu[1], mu[2] = mu0, mu1, 2 * d[0, 1] - mu0
        for k in range(1, K + 1):
            mu[2 * k + 1] = 2 * d[k, 0] - mu1
            if 2 * k + 2 < 2 * K + 2:
                mu[2 * k + 2] = 2 * d[k, 1] - mu0
        tol = 1e-13 * np.arange(1, 2 * K + 3)
        assert (np.abs(mu - mu_ref) <= tol).all(), np.max(np.abs(mu - mu_ref) / tol)
    finally:
        h.destroy()
