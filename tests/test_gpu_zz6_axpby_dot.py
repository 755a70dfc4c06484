"""spmv_b200_spmv_axpby_dot: y <- alpha A x + beta y, bit for bit as spmv_b200_spmv_axpby writes it, and dot = w . y,
taken by the kernel that stores each final y value.

y is compared by bits with spmv_b200_spmv_axpby on the same handle.  The dot is checked two ways.  With integer data
(the integer matrices and x of test_gpu_kernel_instances, an integer old y and integer alpha, beta) every product and
every partial sum is exact in double, so the dot must equal the int64 sum of w_i y_i exactly: a dropped or doubled row
cannot hide behind a tolerance.  With real data the dot must lie within the bound the header states,
|dot - sum p_i| <= L 2^-53 sum |p_i| with L = 18 + ceil(P / 1024), P <= m + 2, where p_i is computed in numpy from the
returned y as the contract defines it and math.fsum rounds the exact sum once (hence one more 2^-53 |sum p_i|).
"""
import math

import numpy as np
import pytest

from conftest import bits_equal
from spmv_b200 import api
from test_gpu_kernel_instances import DTYPES, assert_same, matrix, normalise, options, run, spmv_instances
from test_gpu_zz5_axpby import ALL, BY_NAME, PAIRS, SCRATCH, formula, old_y, table_path, tdtype

gpu = pytest.mark.gpu

FAMILIES = frozenset(["csr_vector_axpby_dot_kernel", "band_reduce_axpby_dot_kernel", "sell_axpby_dot_kernel",
                      "csr_tail_axpby_dot_kernel", "axpby_dot_kernel", "dot_finish_kernel"])
INT_PAIRS = [(1.0, 0.0), (2.0, -3.0), (-1.0, 1.0)]


def products(w, y):
    """p_i as the contract defines them: fl(w_i y_i) in double (exact for two floats)."""
    with np.errstate(all="ignore"):
        return w.astype(np.float64) * y.astype(np.float64)


def assert_within_bound(dot, w, y, tag):
    p = products(w, y)
    L = 18 + -(-(len(y) + 2) // 1024)
    exact = math.fsum(p)
    bound = L * 2.0 ** -53 * float(np.sum(np.abs(p))) + 2.0 ** -53 * abs(exact)
    assert abs(dot - exact) <= bound, f"{tag}: dot {dot!r}, fsum {exact!r}, bound {bound!r}"


def int_dot(w, y):
    """The exact sum of integer-valued w_i y_i, asserting that every partial sum is exact in double."""
    wi, yi = w.astype(np.int64), y.astype(np.int64)
    assert (wi == w).all() and (yi == y).all()
    p = wi * yi
    assert int(np.sum(np.abs(p))) < (1 << 53)
    return float(int(np.sum(p)))


def dot_table(h, peers):
    """Where the dot is taken, as the documented table states it: axpby_path's table, but the scratch pass on band
    segments."""
    return SCRATCH if h.kernel == "band_seg" else table_path(h, peers)


def int_old_y(m, dt, seed):
    return np.random.default_rng(seed).integers(-4, 5, m).astype(dt)


def call(h, alpha, x, beta, y_old, w, host, dot_on_device=False):
    """One spmv_axpby_dot with host or device x / y / w ("y" as w: w is the new y); returns (y, dot)."""
    import torch
    if host:
        y = y_old.copy()
        d = h.spmv_axpby_dot(alpha, x, beta, y, y if isinstance(w, str) else w)
        return y, d
    xd = torch.from_numpy(np.ascontiguousarray(x)).cuda()
    yd = torch.from_numpy(y_old.copy()).cuda()
    wd = yd if isinstance(w, str) else xd if w is x else torch.from_numpy(np.ascontiguousarray(w)).cuda()
    if dot_on_device:
        dd = torch.full((1,), 0.5, dtype=torch.float64, device="cuda")
        assert h.spmv_axpby_dot(alpha, xd, beta, yd, wd, dd) is None
        h.sync()
        return yd.cpu().numpy(), dd.item()
    d = h.spmv_axpby_dot(alpha, xd, beta, yd, wd)
    return yd.cpu().numpy(), d


def axpby_ref(h, alpha, x, beta, y_old, host):
    import torch
    if host:
        y = y_old.copy()
        h.spmv_axpby(alpha, x, beta, y)
        return y
    yd = torch.from_numpy(y_old.copy()).cuda()
    h.spmv_axpby(alpha, torch.from_numpy(np.ascontiguousarray(x)).cuda(), beta, yd)
    h.sync()
    return yd.cpu().numpy()


def ws_of(A, dt, xv):
    """The w of each check: the new y, x (square handles), a separate integer vector."""
    out = [("y", "y")]
    if A.m == A.n:
        out.append(("x", xv))
    out.append(("w", np.random.default_rng(11).integers(-4, 5, A.m).astype(dt)))
    return out


# ---------------------------------------------------------------------------------------------------------------------
# errors without a device
# ---------------------------------------------------------------------------------------------------------------------
def test_null_and_failed_handles_return_an_error(libpath):
    L = api.lib()
    x, y, w = np.ones(4), np.full(4, 7.0), np.ones(4)
    dot = np.full(1, 5.0)
    api.clear_error()
    assert L.spmv_b200_spmv_axpby_dot(None, 1.0, x.ctypes.data, 0.0, y.ctypes.data, w.ctypes.data, dot.ctypes.data) == -1
    assert "NULL handle" in api.last_error()
    rowptr = np.array([1, 2, 3, 4, 5], dtype=np.int32)  # RowPtr[0] != 0: create fails, with or without a device
    h = api.spmv_create_handle_all_in_one(4, 4, rowptr, np.zeros(4, dtype=np.int32), np.ones(4), 1, api.Method_Parallel, 8)
    for args in ((x.ctypes.data, y.ctypes.data, w.ctypes.data, dot.ctypes.data), (None, None, None, None),
                 (x.ctypes.data, y.ctypes.data, y.ctypes.data, dot.ctypes.data)):
        api.clear_error()
        assert L.spmv_b200_spmv_axpby_dot(h, 1.0, args[0], 0.0, args[1], args[2], args[3]) == -1
        assert "create failed" in api.last_error()
    assert (y == 7.0).all() and dot[0] == 5.0
    api.spmv_destory_handle(h)


# ---------------------------------------------------------------------------------------------------------------------
# 1. every configuration: y bits, exact integer dots, the bound on real data, the path
# ---------------------------------------------------------------------------------------------------------------------
def check_config(cfg, dt):
    import torch
    tag = f"{cfg.name}/{np.dtype(dt).name}"
    s, _, h, A = run(cfg, dt)
    try:
        assert h.info("dot_path") == dot_table(h, cfg.peers), (tag, h.info("dot_path"))
        xv = A.x.astype(dt)
        peers = None
        if cfg.peers:
            peers = [torch.full((A.m,), 0.25, dtype=tdtype(dt), device="cuda") for _ in range(2)]
            h.set_y_peers([p.data_ptr() for p in peers])
        for wname, w in ws_of(A, dt, xv):
            for i, (alpha, beta) in enumerate(INT_PAIRS):
                y_old = int_old_y(A.m, dt, seed=i)
                y, d = call(h, alpha, xv, beta, y_old, w, cfg.host)
                assert_same(y, formula(s, alpha, beta, y_old), f"{tag} w={wname} int ({alpha}, {beta})")
                assert d == int_dot(y if wname == "y" else w, y), (tag, wname, alpha, beta, d)
            for i, (alpha, beta) in enumerate(PAIRS):
                y_old = old_y(A.m, dt, seed=i)
                y, d = call(h, alpha, xv, beta, y_old, w, cfg.host, dot_on_device=not cfg.host and i % 2 == 1)
                assert bits_equal(y, axpby_ref(h, alpha, xv, beta, y_old, cfg.host)), (tag, wname, alpha, beta)
                assert_within_bound(d, y if wname == "y" else w, y, f"{tag} w={wname} ({alpha}, {beta})")
                for k, p in enumerate(peers or []):
                    assert bits_equal(p.cpu().numpy(), y), (tag, wname, k)
        return h.info("dot_path")
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("cfg", ALL, ids=[c.name for c in ALL])
def test_dot_every_configuration(libpath, cfg, dt):
    check_config(cfg, DTYPES[dt])


# ---------------------------------------------------------------------------------------------------------------------
# 2. reproducible: call after call, on another stream; 3. option "axpby_fused" = 0
# ---------------------------------------------------------------------------------------------------------------------
SOME = ["vector_tpr1", "banded", "bseg40_ctas3_bseg_small", "csr5_sigma8", "sell_v0_nocap", "bins"]


def real_inputs(A, dt, seed):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal(A.n).astype(dt), old_y(A.m, dt, seed), rng.standard_normal(A.m).astype(dt))


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("name", SOME)
def test_dot_is_reproducible_across_calls_and_streams(libpath, name, dt):
    import torch
    dt = DTYPES[dt]
    _, _, h, A = run(BY_NAME[name], dt)
    try:
        x, y_old, w = real_inputs(A, dt, 3)
        got = [call(h, 0.7, x, -1.3, y_old, w, False) for _ in range(2)]
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        got.append(call(h, 0.7, x, -1.3, y_old, w, False))
        h.set_stream(0)
        for y, d in got[1:]:
            assert bits_equal(y, got[0][0]) and np.float64(d).tobytes() == np.float64(got[0][1]).tobytes(), name
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("name", ["vector_tpr1", "sell_v0_nocap", "banded", "bseg3_ctas2_bseg_small"])
def test_option_axpby_fused_0_takes_the_scratch_pass(libpath, name):
    cfg = BY_NAME[name]
    A = matrix(cfg.mat)
    x, y_old, w = real_inputs(A, np.float64, 4)
    out = {}
    for fused in (1, 0):
        with options({**cfg.opts, "axpby_fused": fused}):
            h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(np.float64), cfg.method)
        try:
            out[fused] = call(h, -1.5, x, 0.75, y_old, w, False)
            assert h.info("dot_path") == (dot_table(h, False) if fused else SCRATCH), (name, fused)
        finally:
            h.destroy()
    assert bits_equal(out[0][0], out[1][0]), name
    for fused in (0, 1):
        assert_within_bound(out[fused][1], w, out[fused][0], f"{name} fused={fused}")


# ---------------------------------------------------------------------------------------------------------------------
# 4. special cases
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "bseg3_ctas2_bseg_small", "csr5_sigma8", "sell_v0_nocap"])
def test_dot_special_cases(libpath, name, dt):
    dt = DTYPES[dt]
    s, _, h, A = run(BY_NAME[name], dt)
    try:
        xv = A.x.astype(dt)
        w = np.random.default_rng(5).integers(-4, 5, A.m).astype(dt)
        poison = old_y(A.m, dt, seed=9)
        poison[::3], poison[1::3] = np.nan, np.inf
        # beta == 0: the old y is never read
        y, d = call(h, 2.0, xv, 0.0, poison, w, False)
        assert bits_equal(y, (dt(2.0) * s).astype(dt)) and d == int_dot(w, y), name
        # alpha == 0: A and x are not read
        xn = xv.copy()
        xn[::3] = np.nan
        y_old = int_old_y(A.m, dt, seed=3)
        y, d = call(h, 0.0, xn, -3.0, y_old, w, False)
        assert bits_equal(y, dt(-3.0) * y_old) and d == int_dot(w, y), name
        y, d = call(h, 0.0, xn, -3.0, y_old, "y", False)
        assert d == int_dot(y, y), name
        # alpha == beta == 0: y = +0, the dot over those zeros; NaN if w holds a NaN or an Inf
        for beta in (0.0, -0.0):
            y, d = call(h, 0.0, xv, beta, poison, w, False)
            assert bits_equal(y, np.zeros(A.m, dtype=dt)) and d == 0.0, name
        wn = w.copy()
        wn[7] = np.inf
        y, d = call(h, 0.0, xv, 0.0, poison, wn, False)
        assert bits_equal(y, np.zeros(A.m, dtype=dt)) and math.isnan(d), name
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("method", [api.Method_Serial, api.Method_Parallel, api.Method_CSR5SPMV])
def test_dot_empty_matrix_and_no_rows(libpath, method, dt):
    import torch
    dt = DTYPES[dt]
    m, n = 50, 40
    h = api.Handle(m, n, np.zeros(m + 1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=dt), method)
    w = np.arange(m).astype(dt) - 20
    for alpha, beta in ((-2.0, 3.0), (3.0, 0.0), (0.0, 2.0)):
        y_old = int_old_y(m, dt, seed=4)
        y, d = call(h, alpha, np.ones(n, dtype=dt), beta, y_old, w, False)
        assert bits_equal(y, formula(np.zeros(m, dtype=dt), alpha, beta, y_old)) and d == int_dot(w, y), (alpha, beta)
    h.destroy()
    h = api.Handle(0, n, np.zeros(1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=dt), method)
    xd = torch.ones(n, dtype=tdtype(dt), device="cuda")
    y = torch.full((1,), 0.5, dtype=tdtype(dt), device="cuda")
    dd = torch.full((1,), 0.5, dtype=torch.float64, device="cuda")
    launches = api.launch_count()
    assert h.spmv_axpby_dot(2.0, xd, 3.0, y, y) == 0.0
    h.spmv_axpby_dot(2.0, xd, 3.0, y, y, dd)
    h.sync()
    assert api.launch_count() == launches and y.item() == 0.5 and dd.item() == 0.0
    assert np.float64(dd.item()).tobytes() == np.float64(0.0).tobytes()
    h.destroy()


@gpu
def test_dot_argument_errors_leave_y_and_dot_untouched(libpath):
    import torch
    _, _, h, A = run(BY_NAME["vector_tpr4"], np.float64)
    L = api.lib()
    assert A.m != A.n
    xd = torch.from_numpy(A.x.astype(np.float64)).cuda()
    big = torch.full((A.m + 8,), 0.5, dtype=torch.float64, device="cuda")
    y = big[:A.m]
    dd = torch.full((1,), 0.25, dtype=torch.float64, device="cuda")
    w = torch.ones(A.m, dtype=torch.float64, device="cuda")
    X, Y, W, D = xd.data_ptr(), y.data_ptr(), w.data_ptr(), dd.data_ptr()
    for args, what in (((X, None, W, D), "y is NULL"), ((X, Y, W, None), "dot is NULL"), ((X, Y, None, D), "w is NULL"),
                       ((None, Y, W, D), "x is NULL"), ((Y, Y, W, D), "same array"), ((X, Y, X, D), "not square"),
                       ((X, Y, big[4:].data_ptr(), D), "overlaps y"), ((X, Y, Y + 8, D), "overlaps y")):
        api.clear_error()
        assert L.spmv_b200_spmv_axpby_dot(h.h, 1.0, args[0], 0.0, args[1], args[2], args[3]) == -1, what
        assert what in api.last_error(), (what, api.last_error())
    h.sync()
    assert (big == 0.5).all() and dd.item() == 0.25
    h.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# 5. host and device pointers
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("pin", [0, 1])
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "csr5_sigma8"])
def test_dot_host_and_device_pointers(libpath, name, pin):
    """Every mix of host and device x, y, w and dot gives the same bits ("banded" has a 2 MiB y: pinned at the second
    call with "pin_host" = 1)."""
    import torch
    cfg = BY_NAME[name]
    A = matrix(cfg.mat)
    dt = np.float64
    with options({**cfg.opts, "pin_host": pin}):
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(dt), cfg.method)
    try:
        x, y_old, w = real_inputs(A, dt, 6)
        want_y, want_d = call(h, -1.5, x, 0.75, y_old, w, False)
        want_yy = call(h, -1.5, x, 0.75, y_old, "y", False)[1]
        dev = lambda a: torch.from_numpy(a.copy()).cuda()
        hy = y_old.copy()  # one host y for the handle's life, as "pin_host" requires of a buffer it may pin
        for xh in (True, False):
            for yh in (True, False):
                for wh in (True, False, None):  # None: w = y
                    for dh in (True, False):
                        xa = x if xh else dev(x)
                        ya = hy if yh else dev(y_old)
                        wa = ya if wh is None else w if wh else dev(w)
                        dd = None if dh else torch.zeros(1, dtype=torch.float64, device="cuda")
                        for _ in range(2):  # the same host buffers again, as a client's loop passes them
                            if yh:
                                ya[:] = y_old
                            else:
                                ya.copy_(dev(y_old))
                            d = h.spmv_axpby_dot(-1.5, xa, 0.75, ya, wa, dd)
                        h.sync()
                        d = d if dh else dd.item()
                        yv = ya if yh else ya.cpu().numpy()
                        tag = f"{name} pin={pin} x={xh} y={yh} w={wh} dot_host={dh}"
                        assert bits_equal(yv, want_y), tag
                        ref = want_yy if wh is None else want_d
                        assert np.float64(d).tobytes() == np.float64(ref).tobytes(), (tag, d, ref)
        if name == "banded":
            assert h.info("pinned_host_buffers") == pin
    finally:
        h.destroy()


@gpu
def test_device_dot_returns_without_a_host_synchronisation(libpath):
    import torch
    _, _, h, A = run(BY_NAME["banded"], np.float64)
    try:
        x, y_old, w = (torch.from_numpy(a).cuda() for a in real_inputs(A, np.float64, 7))
        dd = torch.zeros(1, dtype=torch.float64, device="cuda")
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        h.spmv_axpby_dot(1.0, x, 2.0, y_old, w, dd)  # warm: allocates the partials
        side.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(2_000_000_000)  # ~1 s of spinning ahead of the call on the handle's stream
        h.spmv_axpby_dot(1.0, x, 2.0, y_old, w, dd)
        assert not side.query(), "the call waited for its stream"
        side.synchronize()
        h.set_stream(0)
    finally:
        h.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# 6. CUDA graphs; 7. peers and spmv() afterwards; 8. allocations
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "bseg3_ctas2_bseg_small", "csr5_sigma8", "sell_v0_nocap"])
def test_dot_is_cuda_graph_capturable(libpath, name):
    import torch
    _, _, h, A = run(BY_NAME[name], np.float64)
    try:
        x, y0, w = (torch.from_numpy(a).cuda() for a in real_inputs(A, np.float64, 8))
        dots = torch.zeros(3, dtype=torch.float64, device="cuda")
        y = y0.clone()
        for k in range(3):
            h.spmv_axpby_dot(-1.0, x, 1.0, y, w, dots[k:k + 1])
        h.sync()
        want_y, want_d = y.clone(), dots.clone()
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        g = torch.cuda.CUDAGraph()
        yg, dg = y0.clone(), torch.zeros(3, dtype=torch.float64, device="cuda")
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
            for k in range(3):
                h.spmv_axpby_dot(-1.0, x, 1.0, yg, w, dg[k:k + 1])
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
def test_peers_and_later_calls_after_dot(libpath, name):
    """The peers receive the scaled y; spmv() and spmv_b200_spmv_axpby afterwards keep their bits and launches."""
    import torch
    s, _, h, A = run(BY_NAME[name], np.float64)
    try:
        peers = [torch.full((A.m,), 0.25, dtype=torch.float64, device="cuda") for _ in range(2)]
        h.set_y_peers([p.data_ptr() for p in peers])
        x = torch.from_numpy(A.x.astype(np.float64)).cuda()
        y_old = old_y(A.m, np.float64, seed=1)
        yd = torch.full((A.m,), 0.5, dtype=torch.float64, device="cuda")
        l0 = api.launch_count()
        h.spmv(x, yd)
        h.sync()
        per_call = api.launch_count() - l0
        ax = axpby_ref(h, 2.0, A.x.astype(np.float64), -3.0, y_old, False)
        y = torch.from_numpy(y_old.copy()).cuda()
        h.spmv_axpby_dot(2.0, x, -3.0, y, y)
        h.sync()
        for k, p in enumerate(peers):
            assert torch.equal(p.view(torch.int64), y.view(torch.int64)), (name, k)
        assert bits_equal(y.cpu().numpy(), ax), name
        assert bits_equal(axpby_ref(h, 2.0, A.x.astype(np.float64), -3.0, y_old, False), ax), name
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
def test_dot_allocations(libpath, name):
    """The partials from the first call on; a host dot adds the device double, a host w its staging array, the scratch
    pass its scratch array; destroy returns the count to where it was before the handle."""
    import torch
    cfg = BY_NAME[name]
    A = matrix(cfg.mat)
    x = torch.from_numpy(A.x.astype(np.float64)).cuda()
    y = torch.zeros(A.m, dtype=torch.float64, device="cuda")
    dd = torch.zeros(1, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    base = api.live_allocations()
    with options(cfg.opts):
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(np.float64), cfg.method)
        h.spmv(x, y)
    h.sync()
    held = api.live_allocations()
    scratch = int(h.info("dot_path") == SCRATCH)
    for k in range(2):
        h.spmv_axpby_dot(0.5, x, 2.0, y, y, dd)
        h.sync()
        assert api.live_allocations() == held + scratch + 1, (name, k)
    h.spmv_axpby_dot(0.5, x, 2.0, y, y)
    assert api.live_allocations() == held + scratch + 2, name
    h.spmv_axpby_dot(0.5, x, 2.0, y, np.ones(A.m))
    assert api.live_allocations() == held + scratch + 3, name
    h.destroy()
    assert api.live_allocations() == base, (name, api.live_allocations() - base)


# ---------------------------------------------------------------------------------------------------------------------
# 9. coverage of the dot kernel instances
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_every_dot_instance_is_launched(libpath, monkeypatch):
    import torch
    import test_gpu_kernel_instances
    from torch.profiler import ProfilerActivity, profile
    monkeypatch.setattr(test_gpu_kernel_instances, "FAMILIES", FAMILIES)
    want = spmv_instances(libpath)
    monkeypatch.undo()
    assert len(want) == 11, sorted(want)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for cfg in ALL:
            for dt in DTYPES.values():
                _, _, h, A = run(cfg, dt)
                try:
                    xv = A.x.astype(dt)
                    call(h, 1.5, xv, -1.0, old_y(A.m, dt, 0), "y", cfg.host)
                    call(h, 0.0, xv, 2.0, old_y(A.m, dt, 0), "y", cfg.host)
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
# 10. conjugate gradients on the device
# ---------------------------------------------------------------------------------------------------------------------
def cg(h, b, tol, max_iters=3000, chunk=25):
    """CG for A x = b, x0 = 0: r = b - A x by spmv_b200_spmv_axpby, q = A p with p . q by spmv_b200_spmv_axpby_dot, the
    vector updates in torch.  The scalars stay on the device; the host looks at |r| once every `chunk` steps."""
    import torch
    x = torch.zeros_like(b)
    r = b.clone()
    h.spmv_axpby(-1.0, x, 1.0, r)
    p = r.clone()
    rr = torch.dot(r, r).reshape(1)
    q = torch.empty_like(b)
    pq = torch.empty(1, dtype=torch.float64, device="cuda")
    bb = float(torch.dot(b, b))
    for k in range(max_iters):
        h.spmv_axpby_dot(1.0, p, 0.0, q, p, pq)
        a = rr / pq
        x.add_(a * p)
        r.sub_(a * q)
        rr_new = torch.dot(r, r).reshape(1)
        p.mul_(rr_new / rr).add_(r)
        rr = rr_new
        if k % chunk == chunk - 1 and float(rr) <= tol * tol * bb:
            break
    return x


@gpu
def test_conjugate_gradients_on_the_device(libpath):
    import scipy.sparse as sp
    import scipy.sparse.linalg as spl
    import torch
    from spmv_b200 import matrices as M
    A = M.laplacian2d(64)
    h = api.Handle(A.m, A.n, A.rowptr, A.col, A.val, api.Method_Parallel)
    try:
        b_np = np.random.default_rng(12).standard_normal(A.m)
        b = torch.from_numpy(b_np).cuda()
        xs = [cg(h, b, 1e-12) for _ in range(2)]
        torch.cuda.synchronize()
        assert torch.equal(xs[0].view(torch.int64), xs[1].view(torch.int64))
        x = xs[0].cpu().numpy()
        S = sp.csr_matrix((A.val, A.col, A.rowptr), shape=(A.m, A.n))
        assert np.linalg.norm(b_np - S @ x) / np.linalg.norm(b_np) < 1e-10
        ref = spl.spsolve(S.tocsc(), b_np)
        assert np.max(np.abs(x - ref)) <= 1e-8 * np.max(np.abs(ref))
    finally:
        h.destroy()
