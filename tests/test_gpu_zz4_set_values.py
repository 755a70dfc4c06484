"""spmv_b200_set_values: new values for a handle created with option "refresh", written into every device layout in
place through the source maps kept at create, stream-ordered on the handle's stream.

The yardstick is a handle newly created with the new values: after set_values(v) every spmv() result (and every value
array the structure interface exposes) must be bit for bit that handle's, for every method, precision and layout
option.  The fresh handle is created WITHOUT the option, which also shows that the option changes nothing else."""
import contextlib
import ctypes as C
import gc

import numpy as np
import pytest

from cases import EXTRA_CASES, all_cases
from conftest import bits_equal
from spmv_b200 import api, matrices as M

gpu = pytest.mark.gpu

METHODS = (api.Method_Serial, api.Method_Parallel, api.Method_Balanced, api.Method_Balanced2, api.Method_Balanced_Yid,
           api.Method_SellCSigma, api.Method_CSR5SPMV)
CASES = all_cases()


@contextlib.contextmanager
def options(**kw):
    old = {k: api.get_option(k) for k in kw}
    for k, v in kw.items():
        api.set_option(k, v)
    try:
        yield
    finally:
        for k, v in old.items():
            api.set_option(k, v)


def new_values(nnz, dtype, seed):
    """Seeded, signed, with explicit zeros."""
    rng = np.random.default_rng(seed)
    v = rng.standard_normal(nnz)
    v[rng.random(nnz) < 0.1] = 0.0
    return v.astype(dtype)


def make(a, vals, method, refresh, nthreads=4, **opts):
    with options(refresh=int(refresh), **opts):
        return api.Handle(a.m, a.n, a.rowptr, a.col, vals, method, nthreads=nthreads)


def host_y(h, a, x, index=None):
    """y = A x with host x and y; with option "reorder", x and y go through handle->index (test_spmv.c:95-101,130-137)."""
    y = np.full(a.m, np.nan, dtype=x.dtype)
    if index is None:
        h.spmv(x, y)
        return y
    yy = np.full(a.m, np.nan, dtype=x.dtype)
    h.spmv(x[index], yy)
    y[index] = yy
    return y


def handle_index(h, m):
    s = h.struct
    if not s.Level_3_opt_used:
        return None
    return np.ctypeslib.as_array(C.cast(s.index, C.POINTER(C.c_int)), shape=(m,)).copy()


def check_refresh(a, method, dtype, nthreads=4, **opts):
    """Create with v1 under "refresh", set_values(v2), compare with a handle created with v2 (option off), bitwise."""
    v1 = a.val.astype(dtype)
    v2 = new_values(a.nnz, dtype, seed=a.nnz + method)
    x = M.make_x(a.n, 1, dtype)
    h = make(a, v1.copy(), method, True, nthreads, **opts)
    assert h.info("refreshable") == 1
    if "reorder" in opts:
        assert h.struct.Level_3_opt_used == 1
    host_y(h, a, x, handle_index(h, a.m))
    h.set_values(v2)
    f = make(a, v2.copy(), method, False, nthreads, **opts)
    assert f.info("refreshable") == 0
    where = (a.name, api.METHOD_NAMES[method], np.dtype(dtype).name, opts, h.kernel)
    assert h.kernel == f.kernel and h.info("x_bands") == f.info("x_bands"), where
    index = handle_index(h, a.m)
    y = host_y(h, a, x, index)
    assert bits_equal(y, host_y(f, a, x, handle_index(f, a.m))), where
    for name in ("sell_val", "csr5_val"):
        assert bits_equal(h.structure(name, dtype), f.structure(name, dtype)), (name,) + where
    h.destroy()
    f.destroy()


@gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", list(CASES))
def test_set_values_is_bitwise_a_fresh_create(libpath, name, dtype):
    a = CASES[name]()
    for method in METHODS:
        check_refresh(a, method, dtype)


def _uni():
    return M.uniform_random(6000, 6000, 24, seed=9)


def _lap160_scrambled():
    g = M.laplacian2d(160)  # 25 600 rows, 127 360 non-zeros: above the reorder thresholds
    q = np.random.default_rng(11).permutation(g.m).astype(np.int32)
    return M.CSR(g.m, g.n, *api.permute_csr(g.rowptr, g.col, g.val, q), "lap160_scrambled")


LAYOUTS = [
    ("x_bands3", _uni, (api.Method_Parallel, api.Method_Balanced, api.Method_Balanced_Yid, api.Method_SellCSigma,
                        api.Method_CSR5SPMV), {"x_bands": 3}, ("x_bands", 3)),
    ("seg_bands5", _uni, (api.Method_Parallel, api.Method_Balanced2), {"seg_bands": 5}, ("kernel", 8)),
    ("seg_bands40", _uni, (api.Method_Parallel, api.Method_Balanced2), {"seg_bands": 40}, ("kernel", 8)),
    ("sell_cap64", EXTRA_CASES["hub"], (api.Method_SellCSigma,), {"sell_cap": 64}, ("long_rows", None)),
    ("row_bins", EXTRA_CASES["hub"], (api.Method_Parallel,), {}, ("binned", 1)),
    ("auto", lambda: M.uniform_random(20000, 20000, 32, seed=3), (api.Method_Parallel,), {"auto": 1},
     ("auto_method", api.Method_SellCSigma)),
    ("reorder", _lap160_scrambled, (api.Method_Parallel, api.Method_SellCSigma, api.Method_CSR5SPMV), {"reorder": 1},
     ("released_csr", 0)),
]


@gpu
@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("layout", [l[0] for l in LAYOUTS], ids=str)
def test_every_layout_option(libpath, layout, dtype):
    _, gen, methods, opts, (key, want) = next(l for l in LAYOUTS if l[0] == layout)
    a = gen()
    for method in methods:
        with options(refresh=1, **opts):
            h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val.astype(dtype), method, nthreads=4)
        got = h.info(key)
        h.destroy()
        assert got > 0 if want is None else got == want, (layout, api.METHOD_NAMES[method], key, got)
        check_refresh(a, method, dtype, **opts)


# ------------------------------------------------------------------------------------------------
# sources
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("method", [api.Method_Parallel, api.Method_SellCSigma, api.Method_CSR5SPMV])
def test_sources(libpath, method):
    import torch
    a = _uni()
    x = M.make_x(a.n, 2, np.float64)
    v2 = new_values(a.nnz, np.float64, 5)
    f = make(a, v2.copy(), method, False)
    want = host_y(f, a, x)
    f.destroy()
    for kind in ("numpy", "cpu_torch", "cuda_torch", "null"):
        create_time = a.val.copy()
        h = make(a, create_time, method, True)
        if kind == "numpy":
            h.set_values(v2.copy())
        elif kind == "cpu_torch":
            h.set_values(torch.from_numpy(v2.copy()))
        elif kind == "cuda_torch":
            h.set_values(torch.from_numpy(v2).cuda())
        else:
            create_time[:] = v2  # the reference's usage: change the create-time array in place, then call
            h.set_values()
        assert bits_equal(host_y(h, a, x), want), (kind, api.METHOD_NAMES[method])
        h.destroy()


@gpu
@pytest.mark.parametrize("method", [api.Method_Serial, api.Method_Parallel, api.Method_SellCSigma, api.Method_CSR5SPMV])
def test_adopted_device_csr(libpath, method):
    """Only NULL (or the adopted pointer itself) is accepted: the caller refreshes its own array in place."""
    import torch
    a = _uni()
    rp, ci = torch.from_numpy(a.rowptr).cuda(), torch.from_numpy(a.col).cuda()
    va = torch.from_numpy(a.val.copy()).cuda()
    v2 = new_values(a.nnz, np.float64, 6)
    dx = torch.from_numpy(M.make_x(a.n, 2, np.float64)).cuda()
    with options(refresh=1):
        h = api.Handle(a.m, a.n, rp, ci, va, method)
    assert h.info("owns_csr") == 0 and h.info("refreshable") == 1
    f = api.Handle(a.m, a.n, rp, ci, torch.from_numpy(v2).cuda(), method)
    want = torch.empty(a.m, dtype=torch.float64, device="cuda")
    f.spmv(dx, want)
    va.copy_(torch.from_numpy(v2))
    h.set_values()
    y = torch.empty(a.m, dtype=torch.float64, device="cuda")
    h.spmv(dx, y)
    torch.cuda.synchronize()
    assert bits_equal(y.cpu().numpy(), want.cpu().numpy()), api.METHOD_NAMES[method]
    h.set_values(va)  # the adopted pointer itself
    for other in (torch.from_numpy(a.val).cuda(), a.val.copy()):
        with pytest.raises(RuntimeError, match="adopted"):
            h.set_values(other)
    h.spmv(dx, y)
    torch.cuda.synchronize()
    assert bits_equal(y.cpu().numpy(), want.cpu().numpy()), api.METHOD_NAMES[method]
    h.destroy()
    f.destroy()


# ------------------------------------------------------------------------------------------------
# ordering
# ------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("method", [api.Method_Parallel, api.Method_SellCSigma, api.Method_CSR5SPMV])
@pytest.mark.parametrize("bands", [0, 3])
def test_stream_order_on_a_side_stream(libpath, method, bands):
    """spmv -> y1, set_values(d_v2), d_v2 <- NaN, spmv -> y2, all on one non-default stream with no host sync."""
    import torch
    a = M.uniform_random(100000, 100000, 16, seed=12)
    v1, v2 = a.val.copy(), new_values(a.nnz, np.float64, 7)
    x = M.make_x(a.n, 3, np.float64)
    opts = {"x_bands": bands} if bands else {}
    want1 = host_y(make(a, v1.copy(), method, False, **opts), a, x)
    want2 = host_y(make(a, v2.copy(), method, False, **opts), a, x)
    h = make(a, v1.copy(), method, True, **opts)
    dx = torch.from_numpy(x).cuda()
    y1 = torch.empty(a.m, dtype=torch.float64, device="cuda")
    y2 = torch.empty_like(y1)
    d_v2 = torch.from_numpy(v2).cuda()
    torch.cuda.synchronize()
    s = torch.cuda.Stream()
    h.set_stream(s.cuda_stream)
    with torch.cuda.stream(s):
        h.spmv(dx, y1)
        h.set_values(d_v2)
        d_v2.fill_(float("nan"))
        h.spmv(dx, y2)
    s.synchronize()
    assert bits_equal(y1.cpu().numpy(), want1) and bits_equal(y2.cpu().numpy(), want2), api.METHOD_NAMES[method]
    h.destroy()


@gpu
@pytest.mark.parametrize("pinned", [False, True])
def test_host_source_is_copied_out_on_return(libpath, pinned):
    import torch
    a = M.uniform_random(100000, 100000, 16, seed=12)
    v2 = new_values(a.nnz, np.float64, 8)
    x = M.make_x(a.n, 3, np.float64)
    for method, opts in ((api.Method_Parallel, {}), (api.Method_SellCSigma, {"x_bands": 3})):
        want = host_y(make(a, v2.copy(), method, False, **opts), a, x)
        h = make(a, a.val.copy(), method, True, **opts)
        src = torch.from_numpy(v2.copy())
        if pinned:
            src = src.pin_memory()
        h.set_values(src)
        src.fill_(float("nan"))
        assert bits_equal(host_y(h, a, x), want), (pinned, api.METHOD_NAMES[method])
        h.destroy()


@gpu
def test_pipelined_host_path_sees_new_values(libpath):
    a = M.uniform_random(1 << 16, 1 << 16, 8, seed=4)
    v2 = new_values(a.nnz, np.float64, 9)
    x = M.make_x(a.n, 3, np.float64)
    h = make(a, a.val.copy(), api.Method_Parallel, True)
    assert h.info("pipeline") == 1
    host_y(h, a, x)
    h.set_values(v2)
    f = make(a, v2.copy(), api.Method_Parallel, False)
    assert bits_equal(host_y(h, a, x), host_y(f, a, x))
    h.destroy()
    f.destroy()


@gpu
@pytest.mark.parametrize("opts", [{"x_bands": 3}, {"seg_bands": 5}], ids=str)
def test_column_stages_see_new_values(libpath, opts):
    import torch
    a = _uni()
    v2 = new_values(a.nnz, np.float64, 10)
    x = M.make_x(a.n, 3, np.float64)
    h = make(a, a.val.copy(), api.Method_Parallel, True, **opts)
    f = make(a, v2.copy(), api.Method_Parallel, False, **opts)
    K = h.bands()
    assert K > 1
    dx = torch.from_numpy(x).cuda()
    y = torch.empty(a.m, dtype=torch.float64, device="cuda")
    h.spmv_bands(0, K, dx)
    h.spmv_finish(y)
    h.set_values(torch.from_numpy(v2).cuda())
    for b in reversed(range(K)):
        h.spmv_bands(b, 1, dx)
    h.spmv_finish(y)
    h.sync()
    assert bits_equal(y.cpu().numpy(), host_y(f, a, x)), opts
    h.destroy()
    f.destroy()


# ------------------------------------------------------------------------------------------------
# errors
# ------------------------------------------------------------------------------------------------
def test_null_handle(libpath):
    """Needs no device."""
    assert api.lib().spmv_b200_set_values(None, None) == -1
    assert "NULL handle" in api.last_error()


@gpu
def test_without_the_option(libpath):
    a = _uni()
    x = M.make_x(a.n, 3, np.float64)
    for method in (api.Method_Parallel, api.Method_SellCSigma):
        h = make(a, a.val.copy(), method, False)
        assert h.info("refreshable") == 0 and h.info("values_snapshotted") == 1
        y0 = host_y(h, a, x)
        with pytest.raises(RuntimeError, match='"refresh"'):
            h.set_values(new_values(a.nnz, np.float64, 1))
        assert bits_equal(host_y(h, a, x), y0)
        h.destroy()


@gpu
def test_failed_create(libpath):
    a = _uni()
    rp = a.rowptr.copy()
    rp[0] = 1
    with options(refresh=1):
        h = api.spmv_create_handle_all_in_one(a.m, a.n, rp, a.col, a.val, 1, api.Method_Parallel, 8)
    assert api.lib().spmv_b200_set_values(h, None) == -1
    assert "create failed" in api.last_error()
    api.spmv_destory_handle(h)


@gpu
def test_python_checks_dtype_and_length(libpath):
    import torch
    a = _uni()
    h = make(a, a.val.copy(), api.Method_SellCSigma, True)
    for bad in (a.val.astype(np.float32), a.val.astype(np.int64), a.val[:-1].copy(),
                np.concatenate([a.val, a.val])[::2], torch.zeros(a.nnz, dtype=torch.float32)):
        with pytest.raises(ValueError):
            h.set_values(bad)
    h.destroy()


@gpu
def test_wrong_device(libpath):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    a = _uni()
    h = make(a, a.val.copy(), api.Method_SellCSigma, True)
    with pytest.raises(RuntimeError, match="device 1"):
        h.set_values(torch.from_numpy(a.val).to("cuda:1"))
    h.destroy()


# ------------------------------------------------------------------------------------------------
# allocations
# ------------------------------------------------------------------------------------------------
def _baseline():
    gc.collect()
    return api.live_allocations()


@gpu
def test_allocations(libpath):
    import torch
    a = _uni()
    r = _lap160_scrambled()
    # (matrix, method, options, maps the option adds, staging arrays a host source adds)
    configs = [
        (a, api.Method_Serial, {}, 0, 0),                 # the upload in the caller's order needs no map
        (a, api.Method_Parallel, {}, 0, 0),
        (a, api.Method_SellCSigma, {}, 1, 0),
        (a, api.Method_CSR5SPMV, {}, 1, 0),
        (a, api.Method_Parallel, {"x_bands": 3}, 1, 1),   # the upload is given back: a host source is staged
        (a, api.Method_SellCSigma, {"x_bands": 3}, 2, 1),
        (a, api.Method_Balanced2, {"seg_bands": 5}, 1, 1),
        (r, api.Method_SellCSigma, {"reorder": 1}, 2, 1),  # the permuted upload has a map
    ]
    for A, method, opts, maps, staging in configs:
        where = (api.METHOD_NAMES[method], opts)
        base = _baseline()
        f = make(A, A.val.copy(), method, False, **opts)
        plain = api.live_allocations() - base
        f.destroy()
        assert api.live_allocations() == base, where
        h = make(A, A.val.copy(), method, True, **opts)
        assert api.live_allocations() - base == plain + maps, where
        with_maps = api.live_allocations()
        h.set_values(torch.from_numpy(new_values(A.nnz, np.float64, 2)).cuda())
        assert api.live_allocations() == with_maps, where
        h.set_values(new_values(A.nnz, np.float64, 3))
        assert api.live_allocations() == with_maps + staging, where
        h.set_values(new_values(A.nnz, np.float64, 4))
        assert api.live_allocations() == with_maps + staging, where
        api.spmv_clear_handle(h.h)
        assert api.live_allocations() == base, where
        h.destroy()
        assert api.live_allocations() == base, where
