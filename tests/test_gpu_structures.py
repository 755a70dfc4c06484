"""Bit-exactness of the device-built layouts against the reference's structures (SURVEY.md 8c):
splitters (a9), SELL permutation (a13), CSR5 tile_ptr / tile_desc / offsets / transpose (a16-a18)."""
import numpy as np
import pytest

from cases import GOLDEN_CASES, SELL_NT, all_cases
from spmv_b200 import api, matrices as M

pytestmark = pytest.mark.gpu
CASES = all_cases()
BIG = {k: v for k, v in CASES.items() if k not in ("all_empty",)}


@pytest.mark.parametrize("name", list(BIG))
def test_row_block_splitter_is_reference_a9(libpath, port, name):
    a = BIG[name]()
    for block_nnz in (512, 64):
        api.set_option("block_nnz", block_nnz)
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Balanced)
        parts = h.info("parts")
        assert parts == max(1, -(-a.nnz // block_nnz))
        assert np.array_equal(h.structure("splitter", np.int32), port.splitter(a.rowptr, parts))
        h.destroy()
    api.set_option("block_nnz", 512)


@pytest.mark.parametrize("name", list(BIG))
def test_tile_rows_and_merge_coords(libpath, port, name):
    a = BIG[name]()
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Balanced_Yid)
    tiles, per = h.info("tiles"), 256 * h.info("tile_items")
    tr = h.structure("tile_rows", np.int32)
    want = [port.lib.oracle_right_boundary(a.rowptr, min(t * per, a.nnz), a.m + 1) - 1 for t in range(tiles + 1)]
    assert np.array_equal(tr, np.array(want, np.int32))
    h.destroy()
    api.set_option("force_merge", 1)
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Balanced2)
    api.set_option("force_merge", 0)
    assert h.kernel == "merge_path"
    tiles = h.info("tiles")
    mc = h.structure("merge_coords", np.int32).reshape(-1, 2)
    d = np.minimum(np.arange(tiles + 1, dtype=np.int64) * per, a.m + a.nnz)
    assert np.array_equal(mc.sum(1), d)                      # on the diagonal
    rows, nz = mc[:, 0], mc[:, 1]
    ends = a.rowptr[1:]
    for r, z in zip(rows, nz):                                # a valid merge-path split point
        assert (r == 0 or ends[r - 1] <= z) and (r == a.m or z == 0 or ends[r] > z - 1)
    h.destroy()


@pytest.mark.parametrize("name", list(BIG))
def test_sell_permutation_is_reference_a13(libpath, port, name):
    a = BIG[name]()
    api.set_option("sell_cap", 0)  # the reference's widths: every slice as wide as its longest row
    for sigma in (256, 64):
        api.set_option("sell_sigma", sigma)
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma)
        assert h.info("sigma") == sigma and h.info("banner") == sigma * (a.m // sigma)
        perm = h.structure("sell_perm", np.int32)
        assert np.array_equal(perm, port.sell_perm(a.rowptr, sigma))
        if len(perm):
            w, f = port.sell_chunks(a.rowptr, perm, 32)
            assert np.array_equal(h.structure("sell_width", np.int32), w)
            assert np.array_equal(h.structure("sell_full", np.int32), f)
            sp = h.structure("sell_slice_ptr", np.int64)
            assert np.array_equal(sp, np.concatenate([[0], np.cumsum(w.astype(np.int64) * 32)]))
            scol = h.structure("sell_col", np.int32)
            # every stored entry is either padding or the right element of the right row
            lens = np.diff(a.rowptr)
            for s in range(0, len(w), max(1, len(w) // 7)):
                blk = scol[sp[s]:sp[s + 1]].reshape(-1, 32)
                for lane in (0, 13, 31):
                    r = perm[s * 32 + lane]
                    assert np.array_equal(blk[:lens[r], lane], a.col[a.rowptr[r]:a.rowptr[r + 1]])
                    assert (blk[lens[r]:, lane] == -1).all()
        h.destroy()
    api.set_option("sell_sigma", 256)
    api.set_option("sell_cap", 1024)


def _capped_widths(rowptr, perm, cap=1024):
    """numpy restatement of sell_width_kernel's rule (sell.cuh): slices that would be mostly padding take the
    row length that minimises 32*l + 2*overflow + 64*rows_over; ties -> the larger width; never wider than cap."""
    L = np.diff(rowptr)[perm].reshape(-1, 32).astype(np.int64)
    w = L.max(axis=1)
    for s in np.nonzero(32 * w > 2 * L.sum(axis=1))[0]:
        l = L[s]
        cost = np.array([32 * li + 2 * (l[l > li] - li).sum() + 64 * (l > li).sum() for li in l])
        w[s] = l[cost == cost.min()].max()
    return np.minimum(w, cap).astype(np.int32)


@pytest.mark.parametrize("name", ["skew", "rmat12", "hub"])
def test_sell_capped_slices_and_overflow(libpath, port, name):
    """Default SELL on skewed matrices: same permutation as the reference, slice widths by the documented
    cost rule, every row's first min(len, width) entries in its slice and the rest on the long-row list."""
    a = (BIG[name] if name in BIG else all_cases()[name])()
    api.set_option("sell_sigma", 64)
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma)
    perm = h.structure("sell_perm", np.int32)
    assert np.array_equal(perm, port.sell_perm(a.rowptr, 64))
    w = h.structure("sell_width", np.int32)
    assert np.array_equal(w, _capped_widths(a.rowptr, perm))
    w_ref, f_ref = port.sell_chunks(a.rowptr, perm, 32)
    assert (w <= w_ref).all() and (w < w_ref).any() and np.array_equal(h.structure("sell_full", np.int32), np.minimum(f_ref, w))
    lens = np.diff(a.rowptr)
    over = np.maximum(lens[perm] - np.repeat(w, 32), 0)
    tail = lens[len(perm):]
    n_long = int((over > 0).sum() + (tail > 4096).sum())
    n_segs = int(((over + 2047) // 2048).sum() + ((tail[tail > 4096] + 2047) // 2048).sum())
    assert (h.info("long_rows"), h.info("long_segs")) == (n_long, n_segs)
    sp = h.structure("sell_slice_ptr", np.int64)
    scol = h.structure("sell_col", np.int32)
    for s in range(0, len(w), max(1, len(w) // 9)):
        blk = scol[sp[s]:sp[s + 1]].reshape(-1, 32)
        for lane in (0, 17, 31):
            r = perm[s * 32 + lane]
            k = min(lens[r], w[s])
            assert np.array_equal(blk[:k, lane], a.col[a.rowptr[r]:a.rowptr[r] + k]) and (blk[k:, lane] == -1).all()
    h.destroy()
    api.set_option("sell_sigma", 256)


def test_parallel_hub_rows_go_to_the_long_row_path(libpath):
    a = all_cases()["hub"]()
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Parallel)
    lens = np.diff(a.rowptr)
    thr = h.info("long_thr")
    # short rows + hubs: rows binned by length class (<= 8 / <= 32 / <= 128), hubs beyond 128 on the long-row list
    assert thr == 128 and h.info("binned") == 1
    assert h.info("long_rows") == int((lens > thr).sum()) == 2
    assert h.info("long_segs") == int(((lens[lens > thr] + 2047) // 2048).sum())
    h.destroy()
    # a matrix without hubs keeps the plain rule: 256 * lanes-per-row clamped to [512, 4096], nothing on the list
    a = all_cases()["uni32"]()
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Parallel)
    assert h.info("long_thr") == 256 * h.info("tpr") == 2048 and h.info("long_rows") == 0 and h.info("binned") == 0
    h.destroy()


def test_sell_permutation_against_live_reference(libpath, ref):
    """m = 256*k rows and nthreads = k make the reference pick sigma = 4*floor(m/k/4) = 256."""
    a = M.skewed(256 * 9, 3000, max_len=700)
    sigma, banner, perm, _, _ = ref.sell(a.rowptr, a.col, a.val, 9)
    assert sigma == 256 and banner == a.m
    api.set_option("sell_sigma", 256)
    h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma)
    assert np.array_equal(h.structure("sell_perm", np.int32), perm)
    h.destroy()


def test_sell_permutation_matches_the_stored_reference(libpath, golden):
    """The device-built SELL permutation against the reference's own, as stored in tests/golden: every stored window
    (sigma = 4*floor(m/nthreads/4)) that is a whole number of 32-row slices."""
    checked = []
    try:
        for name, make in GOLDEN_CASES.items():
            a = make()
            for nt in SELL_NT:
                sigma, banner = (int(v) for v in golden[f"{name}/sell_nt{nt}_sigma"])
                if sigma == 0 or sigma % 32 or sigma > 4096:
                    continue
                api.set_option("sell_sigma", sigma)
                h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_SellCSigma)
                assert (h.info("sigma"), h.info("banner")) == (sigma, banner), (name, nt)
                assert np.array_equal(h.structure("sell_perm", np.int32), golden[f"{name}/sell_nt{nt}_perm"]), (name, nt)
                h.destroy()
                checked.append((name, nt))
    finally:
        api.set_option("sell_sigma", 256)
    assert checked == [("lap48", 1), ("lap48", 3), ("rmat10", 1), ("st27_9", 11)]


@pytest.mark.parametrize("name", list(BIG))
def test_csr5_descriptors_are_reference_a16_a18(libpath, port, name):
    a = BIG[name]()
    for sigma in (16, 4):
        api.set_option("csr5_sigma", sigma)
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_CSR5SPMV)
        want = port.csr5(a.rowptr, 32, sigma, a.col)
        assert h.info("csr5_p") == want["p"] and h.info("csr5_sigma") == sigma
        if want["p"]:
            assert h.info("csr5_bit_y_offset") == want["bit_y_offset"]
            assert h.info("csr5_bit_scansum_offset") == want["bit_scansum_offset"] and want["num_packet"] == 1
            assert h.info("csr5_tail_start") == want["tail_start"]
            assert np.array_equal(h.structure("csr5_tile_ptr", np.uint32), want["tile_ptr"])
            assert np.array_equal(h.structure("csr5_tile_desc", np.uint32), want["tile_desc"])
            assert np.array_equal(h.structure("csr5_offset_ptr", np.int32), want["offset_ptr"])
            assert np.array_equal(h.structure("csr5_offsets", np.int32), want["offsets"])
            assert np.array_equal(h.structure("csr5_col", np.int32), want["col_t"])
        h.destroy()
    api.set_option("csr5_sigma", 0)


def test_generators_match_numpy_bit_for_bit(libpath):
    from conftest import bits_equal
    pairs = [
        (lambda: api.gen_laplacian2d(37, 53, 8), lambda: M.laplacian2d(37, 53)),
        (lambda: api.gen_stencil27(7, 9, 11, 8), lambda: M.stencil27(7, 9, 11)),
        (lambda: api.gen_uniform(3000, 5000, 32, M.SEED_C2, 0, False, 8), lambda: M.uniform_random(3000, 5000, 32)),
        (lambda: api.gen_uniform(1000, 999, 16, M.SEED_C5, 12345, True, 4),
         lambda: M.uniform_random(1000, 999, 16, seed=M.SEED_C5, dtype=np.float32, row0=12345, eighths=True)),
        (lambda: api.gen_rmat(11, 16, M.SEED_C3, 4), lambda: M.rmat(11, 16)),
    ]
    for dev, host in pairs:
        d = dev()
        g, w = d.to_host(), host()
        assert (g.m, g.n, g.nnz) == (w.m, w.n, w.nnz), d.name
        assert np.array_equal(g.rowptr, w.rowptr) and np.array_equal(g.col, w.col), d.name
        assert bits_equal(g.val, w.val), d.name
        d.destroy()
    import torch
    for dt, size in ((torch.float64, 8), (torch.float32, 4)):
        x = torch.empty(5000, dtype=dt, device="cuda:0")
        api.gen_x(x, 5000, 77, False, size)
        assert bits_equal(x.cpu().numpy(), M.make_x(5000, 77, np.float64 if size == 8 else np.float32))


@pytest.mark.parametrize("name", ["uni32", "skew", "hub", "lap48", "lead_trail_empty"])
def test_band_major_copy_is_a_stable_column_bucketing(libpath, name):
    a = CASES[name]()
    for K in (2, 3, 7):
        api.set_option("x_bands", K)
        h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, api.Method_Parallel)
        api.set_option("x_bands", 0)
        assert h.info("x_bands") == K and h.info("active_rows") == K * a.m
        bc = h.info("band_cols")
        assert bc == -(-a.n // K)
        vr = h.structure("band_rowptr", np.int32)
        vc = h.structure("band_col", np.int32)
        rows = np.repeat(np.arange(a.m), np.diff(a.rowptr))
        band = np.minimum(a.col // bc, K - 1)
        order = np.lexsort((np.arange(a.nnz), rows, band))      # band-major, row, original order (stable)
        assert np.array_equal(vc, a.col[order])
        cnt = np.bincount(band.astype(np.int64) * a.m + rows, minlength=K * a.m)
        assert np.array_equal(vr, np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32))
        h.destroy()
