"""Every device array the library allocates for itself has one owner: destroying a handle, or finishing a generator
call, gives all of them back.  api.live_allocations() counts the arrays the library currently holds (generated matrices
and spmv_b200_malloc blocks belong to the caller and are not counted)."""
import gc

import numpy as np
import pytest

from cases import EXTRA_CASES, GOLDEN_CASES
from spmv_b200 import api, matrices as M

pytestmark = pytest.mark.gpu

METHODS = (api.Method_Serial, api.Method_Parallel, api.Method_Balanced, api.Method_Balanced2, api.Method_Balanced_Yid,
           api.Method_SellCSigma, api.Method_CSR5SPMV)
CASES = {"hub": EXTRA_CASES["hub"], "rmat12": EXTRA_CASES["rmat12"],
         "lead_trail_empty": EXTRA_CASES["lead_trail_empty"], "empties": GOLDEN_CASES["empties"]}


def _baseline():
    gc.collect()  # a handle of an earlier test collected in the middle of this one would move the count
    return api.live_allocations()


def _run(h, a, dtype):
    x = M.make_x(a.n, 1, dtype)
    y = np.full(a.m, np.nan, dtype=dtype)
    h.spmv(x, y)  # host x and y: the staging buffers are allocated on the first call
    return y


def _handle(a, method, dtype=np.float64, option=None, **kw):
    if option:
        api.set_option(*option)
    try:
        return api.Handle(a.m, a.n, a.rowptr, a.col, a.val.astype(dtype), method, **kw)
    finally:
        if option:
            api.set_option(option[0], 0)


@pytest.mark.parametrize("dtype", [np.float64, np.float32])
@pytest.mark.parametrize("name", list(CASES))
def test_destroy_gives_back_every_allocation(libpath, name, dtype):
    a = CASES[name]()
    base = _baseline()
    for method in METHODS:
        h = _handle(a, method, dtype, nthreads=4)
        _run(h, a, dtype)
        assert api.live_allocations() > base, (name, api.METHOD_NAMES[method])
        kernel = h.kernel
        h.destroy()
        assert api.live_allocations() == base, (name, api.METHOD_NAMES[method], kernel)


def test_band_major_copy_and_band_segments(libpath):
    a = M.uniform_random(6000, 6000, 24, seed=9)
    base = _baseline()
    h = _handle(a, api.Method_Parallel, option=("x_bands", 3))
    assert h.info("x_bands") == 3 and h.info("released_csr") == 1  # the upload was given back at create
    _run(h, a, np.float64)
    h.destroy()
    assert api.live_allocations() == base
    h = _handle(a, api.Method_Balanced, option=("seg_bands", 7), nthreads=4)
    assert h.kernel == "band_seg"
    assert len(h.structure("ref_splitter", np.int32)) == 5
    _run(h, a, np.float64)
    h.destroy()
    assert api.live_allocations() == base


def test_pipelined_host_path(libpath):
    a = M.uniform_random(1 << 16, 1 << 16, 8, seed=4)
    base = _baseline()
    h = _handle(a, api.Method_Parallel)
    assert h.info("pipeline") == 1
    _run(h, a, np.float64)
    _run(h, a, np.float64)
    h.destroy()
    assert api.live_allocations() == base


def test_adopted_csr_update_values_and_clear(libpath):
    import torch
    a = M.uniform_random(3000, 3000, 12, seed=2)
    base = _baseline()
    h = _handle(a, api.Method_Serial)
    assert api.live_allocations() - base == 3  # the upload: RowPtr, ColIdx, values
    h.destroy()
    rp, ci, va = (torch.from_numpy(v).cuda() for v in (a.rowptr, a.col, a.val))
    base = _baseline()
    h = api.Handle(a.m, a.n, rp, ci, va, api.Method_Serial)
    assert h.info("owns_csr") == 0 and api.live_allocations() == base  # adopted in place: nothing of ours
    h.destroy()
    for method in (api.Method_Parallel, api.Method_CSR5SPMV):
        h = api.Handle(a.m, a.n, rp, ci, va, method)
        h.update_values(va * 0.5)
        y = torch.empty(a.m, dtype=torch.float64, device="cuda")
        h.spmv(torch.ones(a.n, dtype=torch.float64, device="cuda"), y)
        torch.cuda.synchronize()
        h.destroy()
        assert api.live_allocations() == base, api.METHOD_NAMES[method]
    h = _handle(a, api.Method_SellCSigma)
    h.update_values(a.val * 2.0)
    api.spmv_clear_handle(h.h)
    assert api.live_allocations() == base
    h.destroy()
    assert api.live_allocations() == base


def test_reorder_and_auto_options(libpath):
    g = M.laplacian2d(160)  # 25 600 rows, 127 360 non-zeros: above the reorder thresholds
    q = np.random.default_rng(11).permutation(g.m).astype(np.int32)
    a = M.CSR(g.m, g.n, *api.permute_csr(g.rowptr, g.col, g.val, q), "lap160_scrambled")
    base = _baseline()
    for method in (api.Method_Parallel, api.Method_SellCSigma):
        h = _handle(a, method, option=("reorder", 1))
        assert h.struct.Level_3_opt_used == 1
        _run(h, a, np.float64)
        h.destroy()
        assert api.live_allocations() == base
    b = M.uniform_random(20000, 20000, 32, seed=3)
    h = _handle(b, api.Method_Parallel, option=("auto", 1))
    assert h.info("auto_method") == api.Method_SellCSigma
    _run(h, b, np.float64)
    h.destroy()
    assert api.live_allocations() == base


def test_rejected_create(libpath):
    a = M.uniform_random(3000, 3000, 12, seed=2)
    rp = a.rowptr.copy()
    rp[0] = 1
    base = _baseline()
    with pytest.raises(RuntimeError, match="RowPtr"):
        api.Handle(a.m, a.n, rp, a.col, a.val, api.Method_Parallel)
    assert api.live_allocations() == base


def test_generators(libpath):
    base = _baseline()
    for gen in (lambda: api.gen_uniform(20000, 30000, 16, 5), lambda: api.gen_rmat(14, 8, 7)):
        A = gen()
        assert A.nnz > 0
        assert api.live_allocations() == base  # the matrix is the caller's; the temporaries are gone
        A.destroy()
        assert api.live_allocations() == base
