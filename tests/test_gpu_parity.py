"""Parity of the CUDA path against the reference's Method_Serial, through the C-ABI.  Needs a B200.

The checker is oracle/_ref/libmv_l2.so (the unmodified reference, when its built .so travelled with the
repo) or the bit-identical port oracle/liboracle.so.  Bars (BASELINE.json north_star):
  * |y - y_ref| <= 8*eps*sum_j|a_ij x_j| per row for every SPMV_METHODS value, fp64 and fp32;
  * Method_Serial on the GPU is BITWISE equal to the reference's Method_Serial;
  * repeated runs are bitwise reproducible.
On rows longer than LONG_ROW the reference's own 4/8-lane chains carry ~sqrt(len)*eps of rounding error,
so there the bound is asserted against the extended-precision sum (oracle_spmv_exact) instead.
"""
import numpy as np
import pytest

from conftest import bits_equal
from cases import GOLDEN_CASES, all_cases, expected_band_segments
from spmv_b200 import api, matrices as M

pytestmark = pytest.mark.gpu

LONG_ROW = 1024
METHODS = list(range(7))
CASES = all_cases()


@pytest.fixture(scope="module")
def serial_ref(port):
    from oracle import oracle as O
    if O.have_reference():
        R = O.Reference()
        return lambda a, x: R.serial(a.rowptr, a.col, a.val, x)
    return lambda a, x: port.spmv_serial(a.rowptr, a.col, a.val, x)


def check_y(port, serial_ref, a, x, y, method, tag=""):
    eps = np.finfo(a.val.dtype).eps
    y_ref = serial_ref(a, x)
    S = port.row_abs_sum(a.rowptr, a.col, a.val, x)
    tol = 8 * eps * S
    lens = np.diff(a.rowptr)
    err = np.abs(y.astype(np.float64) - y_ref.astype(np.float64))
    short = lens <= LONG_ROW
    bad = np.nonzero(short & ~(err <= tol))[0]
    assert len(bad) == 0, f"{tag}: {len(bad)} rows off vs Method_Serial; first row {bad[0]} len {lens[bad[0]]} " \
                          f"y={y[bad[0]]!r} ref={y_ref[bad[0]]!r} tol={tol[bad[0]]:.3e}"
    if method != api.Method_Serial:
        y_ex = port.spmv_exact(a.rowptr, a.col, a.val, x)
        err2 = np.abs(y.astype(np.float64) - y_ex.astype(np.float64))
        # half an ulp of the result itself is unavoidable when rounding the exact sum to the value type
        bad = np.nonzero(~(err2 <= tol + 0.5 * eps * np.abs(y_ex)))[0]
        assert len(bad) == 0, f"{tag}: {len(bad)} rows off vs exact sum; first row {bad[0]} len {lens[bad[0]]} " \
                              f"y={y[bad[0]]!r} exact={y_ex[bad[0]]!r} tol={tol[bad[0]]:.3e}"
    if method == api.Method_Serial:
        assert bits_equal(y, y_ref), f"{tag}: Method_Serial is not bit-identical to the reference"


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
@pytest.mark.parametrize("name", list(CASES))
def test_all_methods_match_reference_serial(libpath, port, serial_ref, name, dt):
    a = CASES[name]().astype(dt)
    x = M.make_x(a.n, 4321, dt)
    for method in METHODS:
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method, nthreads=8)
        y = np.full(a.m, np.nan, dtype=dt)
        h.spmv(x, y)
        tag = f"{name}/{dt.__name__}/{api.METHOD_NAMES[method]}[{h.kernel}]"
        assert not np.isnan(y).any(), tag + ": rows left unwritten"
        check_y(port, serial_ref, a, x, y, method, tag)
        y2 = np.full(a.m, np.nan, dtype=dt)
        h.spmv(x, y2)
        assert bits_equal(y, y2), tag + ": not reproducible run to run"
        h.destroy()


@pytest.mark.parametrize("name", list(GOLDEN_CASES))
def test_all_methods_match_the_stored_reference_y(libpath, port, golden, name):
    """Every method against y of the reference's own Method_Serial as stored in tests/golden (Method_Serial bit for
    bit): the same bars as above with the reference's outputs, not the port's, on the other side."""
    A = GOLDEN_CASES[name]()
    for dt, tag in ((np.float64, "d"), (np.float32, "s")):
        a = A.astype(dt)
        x = M.make_x(a.n, 1234, dt)  # the x tests/golden/make_golden.py used
        stored = golden[f"{name}/y_serial_{tag}"]
        for method in METHODS:
            h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method, nthreads=8)
            y = np.full(a.m, np.nan, dtype=dt)
            h.spmv(x, y)
            check_y(port, lambda *_: stored, a, x, y, method, f"{name}/{dt.__name__}/{api.METHOD_NAMES[method]}[{h.kernel}]")
            h.destroy()


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
def test_merge_path_forced_on_every_case(libpath, port, serial_ref, dt):
    """Method_Balanced2 normally runs merge-path only when a row starves a row block (the reference's
    Balanced2 -> Balanced rule); force it everywhere so the kernel is covered on regular matrices too."""
    api.set_option("force_merge", 1)
    try:
        for name, make in CASES.items():
            a = make().astype(dt)
            x = M.make_x(a.n, 4321, dt)
            h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Balanced2)
            assert h.kernel in ("merge_path", "none"), name
            y = np.full(a.m, np.nan, dtype=dt)
            h.spmv(x, y)
            check_y(port, serial_ref, a, x, y, api.Method_Balanced2, f"force_merge/{name}")
            h.destroy()
    finally:
        api.set_option("force_merge", 0)


def test_balanced2_follows_reference_demotion(libpath):
    """No starved block -> row-block kernel; a long row -> merge-path (for Balanced and Balanced2 alike)."""
    for name, want in (("uni32", "row_blocks"), ("lap48", "row_blocks"), ("hub", "merge_path"), ("one_long_row", "merge_path")):
        a = CASES[name]()
        for method in (api.Method_Balanced, api.Method_Balanced2):
            h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
            assert h.kernel == want, (name, method, h.kernel)
            h.destroy()


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
def test_signed_data_with_cancellation(libpath, port, serial_ref, dt):
    """Mixed-sign values and x: the bound is relative to sum|a x|, not to |y|."""
    rng = np.random.default_rng(17)
    for name in ("skew", "uni32", "lap48", "hub"):
        a = CASES[name]().astype(dt)
        a.val[:] = rng.standard_normal(a.nnz).astype(dt) * (10.0 ** rng.integers(-3, 4, a.nnz)).astype(dt)
        x = rng.standard_normal(a.n).astype(dt)
        for method in METHODS:
            h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method, nthreads=4)
            y = np.full(a.m, np.nan, dtype=dt)
            h.spmv(x, y)
            check_y(port, serial_ref, a, x, y, method, f"signed/{name}/{api.METHOD_NAMES[method]}")
            h.destroy()


def test_device_pointers_and_adopted_device_csr(libpath, port, serial_ref):
    """x / y / CSR already resident in HBM (torch tensors): same bits as the staged host path."""
    import torch
    a = CASES["skew"]()
    x = M.make_x(a.n, 9, np.float64)
    dev = torch.device("cuda:0")
    rp, ci, va = (torch.from_numpy(t).to(dev) for t in (a.rowptr, a.col, a.val))
    xd = torch.from_numpy(x).to(dev)
    for method in METHODS:
        h_host = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
        y_host = np.empty(a.m)
        h_host.spmv(x, y_host)
        h_dev = api.Handle(a.m, a.n, rp, ci, va, method)
        assert h_dev.info("owns_csr") == 0 and h_host.info("owns_csr") == 1
        yd = torch.full((a.m,), float("nan"), dtype=torch.float64, device=dev)
        h_dev.spmv(xd, yd)
        h_dev.sync()
        assert bits_equal(yd.cpu().numpy(), y_host), api.METHOD_NAMES[method]
        # mixed: device x, host y
        y_mixed = np.empty(a.m)
        h_dev.spmv(xd, y_mixed)
        assert bits_equal(y_mixed, y_host)
        h_host.destroy()
        h_dev.destroy()
    # the caller's arrays are never modified (the reference's CSR5 transposes them in place)
    assert np.array_equal(ci.cpu().numpy(), a.col) and np.array_equal(va.cpu().numpy(), a.val)


def test_handle_semantics_follow_the_reference(libpath):
    a = CASES["lap48"]()
    x = M.make_x(a.n, 1, np.float64)
    # out-of-range method -> Method_Serial (common.c:136), Method_Numa included
    for bad in (-1, 7, 8, 99):
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, bad)
        assert h.struct.spmvMethod == api.Method_Serial and h.kernel == "csr_reforder"
        h.destroy()
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma, nthreads=12, vectorizedWay=api.VECTOR_AVX512)
    s = h.struct
    assert (s.nthreads, s.vectorizedWay, s.data_size, s.Level_3_opt_used) == (12, api.VECTOR_AVX512, 8, 0)
    assert s.RowPtr == a.rowptr.ctypes.data and s.ColIdx == a.col.ctypes.data and s.Matrix_Val == a.val.ctypes.data
    assert not s.index and not s.Y_temp
    # clear: handle reusable/inert afterwards, spmv is a no-op
    api.spmv_clear_handle(h.h)
    assert h.struct.spmvMethod == api.Method_Serial and not h.struct.extraHandle
    y = np.full(a.m, 7.0)
    h.spmv(x, y)
    assert (y == 7.0).all()
    h.destroy()
    # size other than sizeof(double) means float (serial_spmv.c:48-54)
    a32 = a.astype(np.float32)
    h = api.Handle(a.m, a.n, a32.rowptr, a32.col, a32.val, api.Method_Parallel, size=4)
    assert h.struct.data_size == 4
    h.destroy()


def test_balanced_demotion_rule_mirrors_reference(libpath, port):
    """handle->spmvMethod after create follows parallel_balanced2_spmv.c:72-94 with the caller's nthreads."""
    for name in ("lap48", "skew", "longrow0", "hub", "uni32"):
        a = CASES[name]()
        for T in (1, 4, 64):
            use_bal, _ = port.balanced2_yid(port.splitter(a.rowptr, T), a.m)
            for req in (api.Method_Balanced, api.Method_Balanced2):
                h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, req, nthreads=T)
                assert h.struct.spmvMethod == (api.Method_Balanced if use_bal else api.Method_Balanced2), (name, T, req)
                assert np.array_equal(h.structure("ref_splitter", np.int32), port.splitter(a.rowptr, T))
                h.destroy()


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
@pytest.mark.parametrize("bands", [2, 5])
def test_band_major_layout_keeps_parity(libpath, port, serial_ref, dt, bands):
    """The band-major (virtual-row) copy under every method: same bound, reproducible; Method_Serial is
    never banded and stays bit-identical to the reference."""
    for name in ("uni32", "skew", "hub", "lead_trail_empty", "lap48", "rmat12"):
        a = CASES[name]().astype(dt)
        x = M.make_x(a.n, 99, dt)
        for method in METHODS:
            api.set_option("x_bands", bands)
            try:
                h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
            finally:
                api.set_option("x_bands", 0)
            assert h.info("x_bands") == (1 if method == api.Method_Serial else bands)
            # the uploaded CSR is given back once every kernel of the handle reads the band-major copy
            assert h.info("released_csr") == (0 if method == api.Method_Serial else 1)
            y = np.full(a.m, np.nan, dtype=dt)
            h.spmv(x, y)
            tag = f"bands{bands}/{name}/{dt.__name__}/{api.METHOD_NAMES[method]}[{h.kernel}]"
            assert not np.isnan(y).any(), tag
            check_y(port, serial_ref, a, x, y, method, tag)
            y2 = np.full(a.m, np.nan, dtype=dt)
            h.spmv(x, y2)
            assert bits_equal(y, y2), tag
            h.destroy()


def test_fused_peer_scatter_single_gpu_emulation(libpath, port, serial_ref):
    """spmv_b200_set_y_peers: every y value also lands in the extra destinations (here: local buffers that
    stand in for the peers' next-x slices), for the fused kernels and for the copy fallback alike."""
    import torch
    dev = torch.device("cuda:0")
    for name, bands in (("uni32", 0), ("skew", 0), ("hub", 0), ("uni32", 3), ("lap48", 0)):
        a = CASES[name]()
        x = torch.from_numpy(M.make_x(a.n, 3, np.float64)).to(dev)
        for method in METHODS:
            api.set_option("x_bands", bands)
            try:
                h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
            finally:
                api.set_option("x_bands", 0)
            y = torch.full((a.m,), float("nan"), dtype=torch.float64, device=dev)
            big = torch.full((3, a.m + 10), float("nan"), dtype=torch.float64, device=dev)
            peers = [big[i, 5:].data_ptr() for i in range(3)]  # slices at a row offset inside larger buffers
            h.set_y_peers(peers)
            h.spmv(x, y)
            h.sync()
            yh = y.cpu().numpy()
            check_y(port, serial_ref, a, x.cpu().numpy(), yh, method, f"peers/{name}/{api.METHOD_NAMES[method]}")
            for i in range(3):
                assert bits_equal(big[i, 5:5 + a.m].cpu().numpy(), yh), (name, method, i)
                assert torch.isnan(big[i, :5]).all() and torch.isnan(big[i, 5 + a.m:]).all()
            h.set_y_peers([])
            y2 = torch.zeros_like(y)
            big.fill_(float("nan"))
            h.spmv(x, y2)
            h.sync()
            assert torch.isnan(big).all() and bits_equal(y2.cpu().numpy(), yh)
            h.destroy()


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
@pytest.mark.parametrize("case", ["lap_local", "uni_random", "uni_banded3", "tall", "wide_empty_tail"])
def test_pipelined_host_path_same_bits_as_device_path(libpath, port, serial_ref, dt, case):
    """Host x + host y on a Method_Parallel handle with >= 2^16 rows takes the PCIe-pipelined path (x in
    pieces, row chunks start when their prefix of x has arrived, y chunks return early): it must give exactly
    the bits of the one-shot device-pointer path, pinned or pageable memory, banded or not."""
    import torch
    bands = 0
    if case == "lap_local":
        a = M.laplacian2d(300, 260)                                   # chunk c needs only a prefix of x
    elif case == "uni_random":
        a = M.uniform_random(70000, 50000, 9, seed=31)                # every chunk needs all of x
    elif case == "uni_banded3":
        a, bands = M.uniform_random(66000, 90001, 24, seed=32), 3     # band b needs slice b of x
    elif case == "tall":
        a = M.uniform_random(200003, 1000, 3, seed=33)
    else:
        a = M.from_row_lengths([5] * 70000 + [0] * 3000, 300000)      # trailing empty rows, n >> m
    a = a.astype(dt)
    x = M.make_x(a.n, 77, dt)
    api.set_option("x_bands", bands)
    try:
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Parallel)
    finally:
        api.set_option("x_bands", 0)
    assert h.info("pipeline") == 1 and h.info("x_bands") == max(bands, 1)
    dev = torch.device("cuda:0")
    xd = torch.from_numpy(x).to(dev)
    yd = torch.full((a.m,), float("nan"), dtype=xd.dtype, device=dev)
    h.spmv(xd, yd)
    h.sync()
    y_dev = yd.cpu().numpy()
    check_y(port, serial_ref, a, x, y_dev, api.Method_Parallel, "pipeline/" + case)
    y_pageable = np.full(a.m, np.nan, dtype=dt)
    h.spmv(x, y_pageable)
    assert bits_equal(y_pageable, y_dev), case
    xp = torch.from_numpy(x).pin_memory()
    yp = torch.full((a.m,), float("nan"), dtype=xd.dtype).pin_memory()
    for _ in range(3):                                               # back to back: stage buffers are reused
        yp.fill_(float("nan"))
        h.spmv(xp, yp)
        assert bits_equal(yp.numpy(), y_dev), case
    api.set_option("pipeline", 0)
    api.set_option("x_bands", bands)
    try:
        h2 = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Parallel)
    finally:
        api.set_option("pipeline", 1)
        api.set_option("x_bands", 0)
    assert h2.info("pipeline") == 0
    y_plain = np.full(a.m, np.nan, dtype=dt)
    h2.spmv(x, y_plain)
    assert bits_equal(y_plain, y_dev), case
    h.destroy()
    h2.destroy()


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
@pytest.mark.parametrize("bands", [2, 7, 40])
def test_band_segment_layout_keeps_parity(libpath, port, serial_ref, dt, bands):
    """Hyper-sparse column bands as band segments (band_seg.cuh), forced on small matrices: every method but
    Method_Serial runs the two-pass band-segment kernels; same error bound, reproducible, and the layout is the
    stable bucketing of the CSR entries by col // band_cols with segment-end bits and per-row band masks
    (40 bands: 64-bit masks)."""
    for name in ("uni32", "uni5r", "skew", "hub", "lead_trail_empty", "lap48", "one_long_row", "one_row", "tiny_m3", "empties",
                 "exact2048"):
        a = CASES[name]().astype(dt)
        x = M.make_x(a.n, 5, dt)
        for method in METHODS:
            api.set_option("seg_bands", bands)
            try:
                h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
            finally:
                api.set_option("seg_bands", 0)
            tag = f"seg{bands}/{name}/{dt.__name__}/{api.METHOD_NAMES[method]}[{h.kernel}]"
            if method == api.Method_Serial:
                assert h.kernel == "csr_reforder" and h.info("seg_bands") == 0
            else:
                assert h.kernel == "band_seg" and h.info("seg_bands") == bands and h.info("x_bands") == bands, tag
                assert h.info("released_csr") == 1 and h.info("layout_fallbacks") == 0, tag
            y = np.full(a.m, np.nan, dtype=dt)
            h.spmv(x, y)
            assert not np.isnan(y).any(), tag
            check_y(port, serial_ref, a, x, y, method, tag)
            y2 = np.full(a.m, np.nan, dtype=dt)
            h.spmv(x, y2)
            assert bits_equal(y, y2), tag
            if method == api.Method_Parallel:
                bc, ptr, cnt, col, mask, nseg = expected_band_segments(a, bands)
                assert h.info("band_cols") == bc
                assert np.array_equal(h.structure("seg_ptr", np.int32), ptr), tag
                assert np.array_equal(h.structure("seg_cnt", np.int32), cnt), tag
                assert np.array_equal(h.structure("seg_col", np.uint32), col), tag
                got_mask = h.structure("seg_mask", np.uint64 if bands > 32 else np.uint32).astype(np.uint64)
                assert np.array_equal(got_mask, mask), tag
                assert h.info("segments") == nseg, tag
                # position of every 32-row group's first segment sum in every band's list: [group][band]
                groups = -(-a.m // 32)
                bits = ((mask[:, None] >> np.arange(bands, dtype=np.uint64)[None, :]) & np.uint64(1)).astype(np.int64)
                padded = np.zeros((groups * 32, bands), dtype=np.int64)
                padded[:a.m] = bits
                cnt_bg = padded.reshape(groups, 32, bands).sum(axis=1).T          # [band][group]
                base_bg = (np.cumsum(cnt_bg.reshape(-1)) - cnt_bg.reshape(-1)).reshape(bands, groups)
                assert np.array_equal(h.structure("seg_gbase", np.int32).reshape(groups, bands), base_bg.T.astype(np.int32)), tag
            h.destroy()
    # a Balanced / Balanced2 handle still mirrors the reference's demotion rule for clients that read it
    a = CASES["longrow0"]()
    api.set_option("seg_bands", 2)
    try:
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Balanced, nthreads=4)
    finally:
        api.set_option("seg_bands", 0)
    assert h.kernel == "band_seg" and h.struct.spmvMethod == api.Method_Balanced2
    h.destroy()


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
def test_mega_hub_rows_two_level_carries(libpath, port, serial_ref, dt):
    """Rows of 2.3 M and 0.4 M non-zeros: thousands of consecutive tiles carry into one row, which takes the
    two-level carry fix-up (carry_group_kernel) in the merge-path / equal-nnz / CSR5 kernels and the long-row
    path in Method_Parallel / SELL.  The 8*eps*sum|a x| bound must still hold against the exact sum."""
    a = M.from_row_lengths([5] * 200 + [2_300_000] + [0] * 5 + [7] * 300 + [400_000] + [2] * 100, 50_000).astype(dt)
    x = M.make_x(a.n, 13, dt)
    for method in METHODS:
        if method == api.Method_Serial:
            continue  # the reference-order chain is checked on the other cases; here it only costs time
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
        y = np.full(a.m, np.nan, dtype=dt)
        h.spmv(x, y)
        tag = f"mega_hub/{dt.__name__}/{api.METHOD_NAMES[method]}[{h.kernel}]"
        assert not np.isnan(y).any(), tag
        check_y(port, serial_ref, a, x, y, method, tag)
        y2 = np.full(a.m, np.nan, dtype=dt)
        h.spmv(x, y2)
        assert bits_equal(y, y2), tag
        if h.kernel in ("merge_path", "nnz_split", "csr5"):
            assert h.info("tiles") >= 1024, tag  # long enough for the two-level path
        h.destroy()


def test_pin_host_option_page_locks_recurring_buffers(libpath, port, serial_ref):
    """Option pin_host (on by default, 0 = off): pageable x / y that come back on consecutive calls are page-locked
    in place after the second sighting, released when the caller switches buffers; results do not change."""
    a = M.laplacian2d(400)  # x, y = 1.28 MB each (>= 1 MiB)
    x = M.make_x(a.n, 3, np.float64)
    api.set_option("pin_host", 0)
    try:
        h0 = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma)
    finally:
        api.set_option("pin_host", 1)
    y0 = np.empty(a.m)
    for _ in range(3):
        h0.spmv(x, y0)
    assert h0.info("pinned_host_buffers") == 0  # switched off: the caller's pages are never touched
    h0.destroy()
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma)
    y = np.full(a.m, np.nan)
    h.spmv(x, y)
    assert h.info("pinned_host_buffers") == 0 and bits_equal(y, y0)
    y.fill(np.nan)
    h.spmv(x, y)
    assert h.info("pinned_host_buffers") == 2 and bits_equal(y, y0)
    y.fill(np.nan)
    h.spmv(x, y)
    assert bits_equal(y, y0)
    y_other = np.full(a.m, np.nan)      # a different y: the old registration is dropped
    h.spmv(x, y_other)
    assert h.info("pinned_host_buffers") == 1 and bits_equal(y_other, y0)
    check_y(port, serial_ref, a, x, y_other, api.Method_SellCSigma, "pin_host")
    h.destroy()                         # unregisters x before the arrays go away


def test_spmv_is_cuda_graph_capturable(libpath):
    """Device-pointer spmv() is a pure sequence of stream-ordered launches on the handle's stream, so an iterated
    loop can be captured once and replayed (launch-bound small matrices): same bits as direct calls."""
    import torch
    dev = torch.device("cuda:0")
    for name, method, bands in (("lap48", api.Method_Parallel, 0), ("hub", api.Method_Balanced2, 0),
                                ("uni32", api.Method_SellCSigma, 3), ("skew", api.Method_CSR5SPMV, 0),
                                ("hub", api.Method_Parallel, 0), ("uni32", api.Method_Balanced_Yid, 0)):
        a = CASES[name]()
        if a.m != a.n:
            continue
        api.set_option("x_bands", bands)
        try:
            h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
        finally:
            api.set_option("x_bands", 0)
        x0 = torch.from_numpy(M.make_x(a.n, 8, np.float64) / 64.0).to(dev)
        # direct: three power iterations x <- A x (ping-pong buffers)
        xa, xb = x0.clone(), torch.empty_like(x0)
        for _ in range(3):
            h.spmv(xa, xb)
            xa, xb = xb, xa
        h.sync()
        want = xa.clone()
        # captured: the same three calls recorded once on a side stream, replayed twice from the same start
        side = torch.cuda.Stream()
        h.set_stream(side.cuda_stream)
        ga, gb = x0.clone(), torch.empty_like(x0)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g, stream=side, capture_error_mode="thread_local"):
            h.spmv(ga, gb)
            h.spmv(gb, ga)
            h.spmv(ga, gb)
        for _ in range(2):
            ga.copy_(x0)
            g.replay()
            torch.cuda.synchronize()
            assert torch.equal(gb, want), (name, api.METHOD_NAMES[method])
        h.set_stream(0)
        h.destroy()


def test_spmv_on_a_handle_whose_create_failed_leaves_y_untouched(libpath):
    """The API returns void: a failed create (here: RowPtr[0] != 0) latches an error, and spmv() on that handle is a
    no-op that must not write a single byte of y -- on the GPU box, with host and with device y."""
    import torch
    a = CASES["uni32"]()
    bad = a.rowptr.copy()
    bad[0] = 1
    api.clear_error()
    h = api.spmv_create_handle_all_in_one(a.m, a.n, bad, a.col, a.val, 1, api.Method_Parallel, 8)
    assert h and api.lib().spmv_b200_info(h, b"ok") == 0 and api.last_error() != ""
    x = M.make_x(a.n, 2, np.float64)
    y = np.full(a.m, 7.25)
    api.spmv(h, a.m, bad, a.col, a.val, x, y)
    assert (y == 7.25).all()
    yd = torch.full((a.m,), 7.25, dtype=torch.float64, device="cuda")
    xd = torch.as_tensor(x, device="cuda")
    api.spmv(h, a.m, bad, a.col, a.val, xd, yd)
    torch.cuda.synchronize()
    assert bool((yd == 7.25).all())
    api.spmv_destory_handle(h)
    api.clear_error()


@pytest.mark.parametrize("dt", [np.float64, np.float32], ids=["fp64", "fp32"])
def test_band_staged_spmv_is_bit_identical_in_any_band_order(libpath, dt):
    """spmv_b200_spmv_bands / spmv_b200_spmv_finish (the interface the pipelined multi-GPU loop is built on): bands
    staged one by one, in scrambled order and in runs, fold to exactly the y of spmv() -- for the band-major copy of
    Method_Parallel and for band segments; unbanded handles report one band."""
    import torch
    for name in ("uni32", "uni16", "hub", "lap48", "empties"):
        a = CASES[name]().astype(dt)
        x = torch.as_tensor(M.make_x(a.n, 9, dt), device="cuda")
        for opt, bands in (("x_bands", 5), ("seg_bands", 6), ("seg_bands", 37)):
            api.set_option(opt, bands)
            api.set_option("long_thr", -1)
            try:
                h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Parallel)
            finally:
                api.set_option(opt, 0)
                api.set_option("long_thr", 0)
            tag = f"{name}/{dt.__name__}/{opt}={bands}[{h.kernel}]"
            assert h.bands() == bands, tag
            cols = [h.band_columns(b) for b in range(bands)]
            assert cols[0][0] == 0 and cols[-1][1] == a.n and all(cols[i][1] == cols[i + 1][0] or cols[i + 1][0] >= a.n for i in range(bands - 1)), tag
            y = torch.full((a.m,), float("nan"), dtype=x.dtype, device="cuda")
            h.spmv(x, y)
            order = list(np.random.default_rng(3).permutation(bands))
            y2 = torch.full((a.m,), float("nan"), dtype=x.dtype, device="cuda")
            for b in order:
                h.spmv_bands(int(b), 1, x)
            h.spmv_finish(y2)
            y3 = torch.full((a.m,), float("nan"), dtype=x.dtype, device="cuda")
            h.spmv_bands(2, bands - 2, x)
            h.spmv_bands(0, 2, x)
            h.spmv_finish(y3)
            torch.cuda.synchronize()
            assert torch.equal(y, y2) and torch.equal(y, y3), tag
            h.destroy()
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma)
        assert h.bands() == 1 and h.band_columns(0) == (0, a.n)
        h.destroy()
