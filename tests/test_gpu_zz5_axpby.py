"""spmv_b200_spmv_axpby: y <- alpha A x + beta y, scaled by the kernel that stores each final y value.

The contract is exact: with s = the bits spmv() writes on the same handle for the same x, every row is
fl(fl(alpha s) + fl(beta y_old)) (beta == 0: fl(alpha s), old y never read; alpha == 0: fl(beta y_old), A and x never
read; both 0: +0.0), each product and sum rounded once in the handle's precision.  numpy computes exactly that, so
every comparison below is of bits.  The configurations are test_gpu_kernel_instances.CONFIGS -- every group of kernel
instances spmv() can launch -- plus SELL handles without long-row list (the only SELL layouts whose main kernel writes
every final value), so that every scaled kernel instance is launched; the coverage test checks that with
torch.profiler against the instances compiled into the library.
"""
import numpy as np
import pytest

from conftest import bits_equal
from spmv_b200 import api
from test_gpu_kernel_instances import (CONFIGS, DTYPES, Config, assert_same, exact_ref, matrix, normalise, options, run,
                                       spmv_instances)

gpu = pytest.mark.gpu

SCRATCH, MAIN, FOLD = 0, 1, 2
PAIRS = [(1.0, 0.0), (2.0, -3.0), (0.1, -0.7), (-1.5, 1.0)]
FAMILIES = frozenset(["csr_vector_axpby_kernel", "band_reduce_axpby_kernel", "bseg_merge_axpby_kernel",
                      "sell_axpby_kernel", "csr_tail_axpby_kernel", "axpby_kernel"])

SELL = api.Method_SellCSigma
K = {v: k for k, v in api.KERNEL_NAMES.items()}
# SELL without the slice-width cap has no long-row list: its main kernel and its CSR tail write every final value.  The
# scaled SELL kernel steps 8 columns, as spmv()'s variant 0 does (and any variant with peers and no CSR tail); variant
# 2's 4-column handles take the scratch pass.
EXTRA = [
    Config("sell_v0_nocap", "regions", SELL, {"sell_variant": 0, "sell_cap": 0},
           {"kernel": K["sell"], "sell_variant": 0, "long_rows": 0, "banner": 10752}),
    Config("sell_v2_nocap", "regions", SELL, {"sell_variant": 2, "sell_cap": 0},
           {"kernel": K["sell"], "sell_variant": 2, "long_rows": 0, "banner": 10752}),
    # with peers and no CSR tail spmv() runs the 8-column flavour whatever the variant: the scaled kernel must follow
    Config("sell_v2_nocap_peers", "bins256", SELL, {"sell_variant": 2, "sell_cap": 0},
           {"kernel": K["sell"], "sell_variant": 2, "long_rows": 0, "banner": 12032}, peers=True),
]
ALL = CONFIGS + EXTRA
BY_NAME = {c.name: c for c in ALL}


def table_path(h, peers):
    """Where the scaling happens, as the documented table states it, from the handle's public facts."""
    if h.kernel == "band_seg" or h.info("x_bands") > 1:
        return FOLD
    if h.info("long_rows") > 0:
        return SCRATCH
    if h.kernel == "csr_vector":
        return MAIN if h.info("tpr") == 1 and not h.info("binned") else SCRATCH
    if h.kernel == "sell":
        eight = h.info("sell_variant") != 2 or (peers and h.info("banner") == h.info("m"))
        return MAIN if eight else SCRATCH
    return SCRATCH


def formula(s, alpha, beta, y_old):
    """The contract in numpy: alpha and beta rounded to the precision first, every operation rounded once."""
    dt = y_old.dtype.type
    a, b = dt(alpha), dt(beta)
    with np.errstate(all="ignore"):
        if a == 0:
            return np.zeros_like(y_old) if b == 0 else b * y_old
        if b == 0:
            return a * s
        return a * s + b * y_old


def old_y(m, dt, seed):
    """Random signed values, exact zeros of both signs, and integers (so that a*s + b*y can cancel to zero)."""
    rng = np.random.default_rng(seed)
    y = rng.standard_normal(m)
    y[::7] = rng.integers(-4, 5, len(y[::7]))
    y = y.astype(dt)
    y[::5] = -0.0
    y[1::11] = 0.0
    return y


def tdtype(dt):
    import torch
    return torch.float64 if dt == np.float64 else torch.float32


def axpby_device(h, alpha, x, beta, y_old, peers=None):
    """One call with device x and y (and the peer buffers given); returns y and the peers' copies."""
    import torch
    yd = torch.from_numpy(y_old.copy()).cuda()
    h.spmv_axpby(alpha, x, beta, yd)
    h.sync()
    return yd.cpu().numpy(), [p.cpu().numpy() for p in (peers or [])]


def check_config(cfg, dt):
    """spmv() once, then every (alpha, beta) of PAIRS against the formula on spmv()'s bits; peers hold y's bits."""
    import torch
    tag = f"{cfg.name}/{np.dtype(dt).name}"
    s, _, h, A = run(cfg, dt)
    try:
        assert h.info("axpby_path") == table_path(h, cfg.peers), (tag, h.info("axpby_path"), table_path(h, cfg.peers))
        xv = A.x.astype(dt)
        peers = None
        if cfg.peers:
            peers = [torch.full((A.m,), 0.25, dtype=tdtype(dt), device="cuda") for _ in range(2)]
            h.set_y_peers([p.data_ptr() for p in peers])
        for i, (alpha, beta) in enumerate(PAIRS):
            y_old = old_y(A.m, dt, seed=i)
            want = formula(s, alpha, beta, y_old)
            if cfg.host:
                y = y_old.copy()
                h.spmv_axpby(alpha, xv, beta, y)
                got_peers = []
            else:
                y, got_peers = axpby_device(h, alpha, torch.from_numpy(xv).cuda(), beta, y_old, peers)
            assert_same(y, want, f"{tag} alpha={alpha} beta={beta}")
            for k, yp in enumerate(got_peers):
                assert bits_equal(yp, y), f"{tag} alpha={alpha} beta={beta}: peer {k} differs from y"
            if (alpha, beta) == (1.0, 0.0):
                assert bits_equal(y, s), f"{tag}: (1, 0) is not spmv()'s bits"
        return h.info("axpby_path")
    finally:
        h.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# 8. errors without a device
# ---------------------------------------------------------------------------------------------------------------------
def test_null_and_failed_handles_return_an_error(libpath):
    L = api.lib()
    x, y = np.ones(4), np.full(4, 7.0)
    api.clear_error()
    assert L.spmv_b200_spmv_axpby(None, 1.0, x.ctypes.data, 0.0, y.ctypes.data) == -1
    assert "NULL handle" in api.last_error()
    rowptr = np.array([1, 2, 3, 4, 5], dtype=np.int32)  # RowPtr[0] != 0: create fails, with or without a device
    col = np.zeros(4, dtype=np.int32)
    h = api.spmv_create_handle_all_in_one(4, 4, rowptr, col, np.ones(4), 1, api.Method_Parallel, 8)
    api.clear_error()
    assert L.spmv_b200_spmv_axpby(h, 1.0, x.ctypes.data, 0.0, y.ctypes.data) == -1
    assert "create failed" in api.last_error()
    assert (y == 7.0).all()
    api.spmv_destory_handle(h)


# ---------------------------------------------------------------------------------------------------------------------
# 1. bits on every configuration
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("cfg", ALL, ids=[c.name for c in ALL])
def test_axpby_bits_every_configuration(libpath, cfg, dt):
    path = check_config(cfg, DTYPES[dt])
    if cfg in EXTRA:
        assert path == (SCRATCH if cfg.name == "sell_v2_nocap" else MAIN), (cfg.name, path)


@gpu
def test_every_path_is_taken():
    """The table's three rows each serve some configuration (the per-configuration path is asserted above)."""
    paths = {}
    for name, want in (("vector_tpr1", MAIN), ("vector_tpr4", SCRATCH), ("row_blocks", SCRATCH),
                       ("sell_v0_nocap", MAIN), ("banded", FOLD),
                       ("bseg40_ctas3_bseg_small", FOLD), ("vector_tpr8_fused", FOLD), ("bins", SCRATCH),
                       ("csr5_sigma8", SCRATCH), ("serial", SCRATCH), ("merge_ipt4", SCRATCH), ("sell_v0", SCRATCH),
                       ("sell_v2_nocap", SCRATCH)):
        _, _, h, _ = run(BY_NAME[name], np.float64)
        paths[name] = h.info("axpby_path")
        h.destroy()
        assert paths[name] == want, (name, paths[name], want)


# ---------------------------------------------------------------------------------------------------------------------
# 2. special cases
# ---------------------------------------------------------------------------------------------------------------------
SPECIAL = ["vector_tpr1", "banded", "bseg3_ctas2_bseg_small", "csr5_sigma8", "sell_v0_nocap"]


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("name", SPECIAL)
def test_axpby_special_cases(libpath, name, dt):
    import torch
    dt = DTYPES[dt]
    cfg = BY_NAME[name]
    s, _, h, A = run(cfg, dt)
    try:
        xd = torch.from_numpy(A.x.astype(dt)).cuda()
        poison = old_y(A.m, dt, seed=9)
        poison[::3], poison[1::3] = np.nan, np.inf
        poison[2::6] = -np.inf
        # beta == 0: the old y is never read, NaN / Inf in it do not propagate
        y, _ = axpby_device(h, 2.5, xd, 0.0, poison)
        assert bits_equal(y, (dt(2.5) * s).astype(dt)), name
        # alpha == 0: A and x are not read, NaN in x changes nothing
        xn = A.x.astype(dt)
        xn[::3] = np.nan
        y_old = old_y(A.m, dt, seed=3)
        y, _ = axpby_device(h, 0.0, torch.from_numpy(xn).cuda(), -3.0, y_old)
        assert bits_equal(y, dt(-3.0) * y_old), name
        # alpha == beta == 0: +0.0 everywhere, whatever y held
        y, _ = axpby_device(h, 0.0, xd, 0.0, poison)
        assert bits_equal(y, np.zeros(A.m, dtype=dt)), name
        # (1, 0) is spmv()
        y, _ = axpby_device(h, 1.0, xd, 0.0, poison)
        assert bits_equal(y, s), name
        # fp32 handles round alpha and beta to float first
        alpha, beta = 1.0 + 2.0 ** -40, 3.0 ** 0.5
        y, _ = axpby_device(h, alpha, xd, beta, y_old)
        assert bits_equal(y, formula(s, alpha, beta, y_old)), name
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("method", [api.Method_Serial, api.Method_Parallel, api.Method_CSR5SPMV])
def test_axpby_empty_matrix_and_no_rows(libpath, method, dt):
    """nnz == 0: the formula with s = +0 (so fl(alpha 0) keeps the sign of alpha); m == 0: returns 0, writes nothing."""
    import torch
    dt = DTYPES[dt]
    m, n = 50, 40
    h = api.Handle(m, n, np.zeros(m + 1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=dt), method)
    xd = torch.from_numpy(np.ones(n, dtype=dt)).cuda()
    for alpha, beta in ((-2.0, 0.5), (3.0, 0.0), (-1.0, 0.0), (0.0, 2.0)):
        y_old = old_y(m, dt, seed=4)
        y, _ = axpby_device(h, alpha, xd, beta, y_old)
        assert bits_equal(y, formula(np.zeros(m, dtype=dt), alpha, beta, y_old)), (alpha, beta)
    h.destroy()
    h = api.Handle(0, n, np.zeros(1, dtype=np.int32), np.zeros(0, dtype=np.int32), np.zeros(0, dtype=dt), method)
    y = torch.full((1,), 0.5, dtype=tdtype(dt), device="cuda")
    launches = api.launch_count()
    h.spmv_axpby(2.0, xd, 3.0, y)
    h.sync()
    assert api.launch_count() == launches and y.item() == 0.5
    h.destroy()


@gpu
def test_axpby_argument_errors_leave_y_untouched(libpath):
    import torch
    _, _, h, A = run(BY_NAME["vector_tpr4"], np.float64)
    L = api.lib()
    xd = torch.from_numpy(A.x.astype(np.float64)).cuda()
    y = torch.full((A.m,), 0.5, dtype=torch.float64, device="cuda")
    for args, what in (((1.0, xd.data_ptr(), 0.0, None), "y is NULL"), ((1.0, None, 0.0, y.data_ptr()), "x is NULL"),
                       ((1.0, y.data_ptr(), 1.0, y.data_ptr()), "same array")):
        api.clear_error()
        assert L.spmv_b200_spmv_axpby(h.h, *args) == -1, what
        assert what in api.last_error(), (what, api.last_error())
    h.sync()
    assert (y == 0.5).all()
    h.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# 3. coverage of the scaled kernel instances
# ---------------------------------------------------------------------------------------------------------------------
@gpu
def test_every_axpby_instance_is_launched(libpath, monkeypatch):
    import torch
    import test_gpu_kernel_instances
    from torch.profiler import ProfilerActivity, profile
    # spmv_instances' listing (cuobjdump + cu++filt), filtered by the scaled families instead of spmv()'s
    monkeypatch.setattr(test_gpu_kernel_instances, "FAMILIES", FAMILIES)
    want = spmv_instances(libpath)
    monkeypatch.undo()
    assert len(want) == 14, sorted(want)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for cfg in ALL:
            for dt in DTYPES.values():
                check_config(cfg, dt)
        torch.cuda.synchronize()
    raw = {e.name for e in prof.events() if "kernel" in e.name}
    if not raw:
        pytest.skip("torch.profiler recorded no CUDA kernels (no CUPTI activity on this machine)")
    seen = {k for k in map(normalise, raw) if k[0] in FAMILIES}
    missing = sorted(want - seen)
    assert not missing, f"{len(missing)} of {len(want)} instances never launched:\n" + \
        "\n".join(f"  {f}<{', '.join(a)}>" for f, a in missing)


# ---------------------------------------------------------------------------------------------------------------------
# 4. host and device pointers
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("pin", [0, 1])
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "csr5_sigma8"])
def test_axpby_host_and_device_pointers(libpath, name, pin):
    """host x / host y, host x / device y and device x / device y give the same bits; a host y with beta != 0 is
    uploaded first.  The "fused" matrix of "banded" has a 2 MiB y: with "pin_host" = 1 it is page-locked at the second
    call."""
    import torch
    cfg = BY_NAME[name]
    A = matrix(cfg.mat)
    dt = np.float64
    with options({**cfg.opts, "pin_host": pin}):
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(dt), cfg.method)
    try:
        xv = A.x.astype(dt)
        s = exact_ref(A, A.a, A.x, dt)
        y_old = old_y(A.m, dt, seed=5)
        want = formula(s, -1.5, 0.75, y_old)
        hy = y_old.copy()
        for _ in range(3):  # the same host buffers each time, as a client's loop passes them
            hy[:] = y_old
            h.spmv_axpby(-1.5, xv, 0.75, hy)
            assert_same(hy, want, f"{name} host/host pin_host={pin}")
        if name == "banded":
            assert h.info("pinned_host_buffers") == pin
        yd = torch.from_numpy(y_old.copy()).cuda()
        h.spmv_axpby(-1.5, xv, 0.75, yd)
        h.sync()
        assert_same(yd.cpu().numpy(), want, f"{name} host x / device y")
        y, _ = axpby_device(h, -1.5, torch.from_numpy(xv).cuda(), 0.75, y_old)
        assert_same(y, want, f"{name} device/device")
        hy2 = y_old.copy()
        h.spmv_axpby(-1.5, torch.from_numpy(xv).cuda(), 0.75, hy2)
        assert_same(hy2, want, f"{name} device x / host y")
    finally:
        h.destroy()


# ---------------------------------------------------------------------------------------------------------------------
# 6. stream order: CUDA graphs, value refresh, spmv() afterwards
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name", ["vector_tpr1", "banded", "bseg3_ctas2_bseg_small", "csr5_sigma8", "sell_v0_nocap"])
def test_axpby_is_cuda_graph_capturable(libpath, name):
    """After one call outside the capture, three residual updates r <- b - A x_k recorded once replay to the bits of
    the direct calls."""
    import torch
    cfg = BY_NAME[name]
    _, _, h, A = run(cfg, np.float64)
    try:
        x = torch.from_numpy(A.x.astype(np.float64)).cuda()
        r0 = torch.from_numpy(old_y(A.m, np.float64, seed=6)).cuda()
        r = r0.clone()
        for _ in range(3):
            h.spmv_axpby(-1.0, x, 1.0, r)
        h.sync()
        want = r.clone()
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        g = torch.cuda.CUDAGraph()
        rg = r0.clone()
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
            for _ in range(3):
                h.spmv_axpby(-1.0, x, 1.0, rg)
        for _ in range(2):
            rg.copy_(r0)
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(rg.view(torch.int64), want.view(torch.int64)), name
        h.set_stream(0)
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("name", ["csr5_refresh", "sell_refresh", "serial_refresh"])
def test_axpby_after_set_values_uses_the_new_values(libpath, name):
    import torch
    cfg = BY_NAME[name]
    _, _, h, A = run(cfg, np.float64)
    try:
        x = torch.from_numpy(A.x.astype(np.float64)).cuda()
        y_old = old_y(A.m, np.float64, seed=7)
        y1 = torch.from_numpy(y_old.copy()).cuda()
        h.spmv_axpby(2.0, x, -1.0, y1)
        a2 = np.random.default_rng(8).integers(-4, 5, A.nnz).astype(np.int64)
        h.set_values(torch.from_numpy(a2.astype(np.float64)).cuda())
        y2 = torch.from_numpy(y_old.copy()).cuda()
        h.spmv_axpby(2.0, x, -1.0, y2)
        h.sync()
        assert_same(y1.cpu().numpy(), formula(exact_ref(A, A.a, A.x, np.float64), 2.0, -1.0, y_old), name + " before")
        assert_same(y2.cpu().numpy(), formula(exact_ref(A, a2, A.x, np.float64), 2.0, -1.0, y_old), name + " after")
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("name", ["vector_tpr1_peers", "banded", "bseg40_ctas3_bseg_small_peers", "csr5_peers",
                                  "sell_v2_nocap_peers"])
def test_spmv_after_axpby_is_unchanged(libpath, name):
    """spmv() after scaled products: its old bits and its old number of launches, and the peers (live buffers of this
    test, registered in place of run()'s) hold the bits of each call's y."""
    import torch
    cfg = BY_NAME[name]
    s, _, h, A = run(cfg, np.float64)
    try:
        peers = [torch.full((A.m,), 0.25, dtype=torch.float64, device="cuda") for _ in range(2)]
        h.set_y_peers([p.data_ptr() for p in peers])
        x = torch.from_numpy(A.x.astype(np.float64)).cuda()
        y = torch.full((A.m,), 0.5, dtype=torch.float64, device="cuda")
        l0 = api.launch_count()
        h.spmv(x, y)
        h.sync()
        per_call = api.launch_count() - l0
        for alpha, beta in PAIRS:
            yo = torch.from_numpy(old_y(A.m, np.float64, seed=1)).cuda()
            h.spmv_axpby(alpha, x, beta, yo)
            h.sync()
            for k, p in enumerate(peers):
                assert torch.equal(p.view(torch.int64), yo.view(torch.int64)), (name, alpha, beta, k)
        y.fill_(0.5)
        l0 = api.launch_count()
        h.spmv(x, y)
        h.sync()
        assert api.launch_count() - l0 == per_call
        assert bits_equal(y.cpu().numpy(), s), name
        for p in peers:
            assert bits_equal(p.cpu().numpy(), s), name
    finally:
        h.destroy()


@gpu
@pytest.mark.parametrize("name", ["vector_tpr1", "sell_v0_nocap", "banded", "bseg3_ctas2_bseg_small"])
def test_option_axpby_fused_0_takes_the_scratch_pass_with_the_same_bits(libpath, name):
    import torch
    cfg = BY_NAME[name]
    A = matrix(cfg.mat)
    x = torch.from_numpy(A.x.astype(np.float64)).cuda()
    y_old = old_y(A.m, np.float64, seed=2)
    out = {}
    for fused in (1, 0):
        with options({**cfg.opts, "axpby_fused": fused}):
            h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(np.float64), cfg.method)
            try:
                out[fused], _ = axpby_device(h, -1.5, x, 0.75, y_old)
                assert (h.info("axpby_path") == SCRATCH) == (fused == 0), (name, fused, h.info("axpby_path"))
            finally:
                h.destroy()
    assert bits_equal(out[0], out[1]), name
    assert_same(out[1], formula(exact_ref(A, A.a, A.x, np.float64), -1.5, 0.75, y_old), name)


# ---------------------------------------------------------------------------------------------------------------------
# 7. memory
# ---------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("name,extra", [("csr5_sigma8", 1), ("bins", 1), ("serial", 1), ("vector_tpr1", 0),
                                        ("vector_tpr4", 1), ("banded", 0), ("bseg3_ctas2_bseg_small", 0), ("row_blocks", 1),
                                        ("sell_v0_nocap", 0), ("sell_v2_nocap", 1)])
def test_axpby_allocations(libpath, name, extra):
    """The scratch pass holds exactly one more array (from its first call on), the fused paths none; destroy returns
    the count to where it was before the handle."""
    import torch
    cfg = BY_NAME[name]
    A = matrix(cfg.mat)
    x = torch.from_numpy(A.x.astype(np.float64)).cuda()
    y = torch.zeros(A.m, dtype=torch.float64, device="cuda")
    torch.cuda.synchronize()
    base = api.live_allocations()
    with options(cfg.opts):
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(np.float64), cfg.method)
        h.spmv(x, y)
    h.sync()
    held = api.live_allocations()
    for k in range(3):
        h.spmv_axpby(0.5, x, 2.0, y)
        h.sync()
        assert api.live_allocations() == held + extra, (name, k, api.live_allocations() - held)
    assert (h.info("axpby_path") == SCRATCH) == bool(extra), (name, h.info("axpby_path"))
    h.destroy()
    assert api.live_allocations() == base, (name, api.live_allocations() - base)
