"""Create-time option values outside the documented ones: every create reads its options once and applies each key's
rule (clamped, rounded or taken as automatic).  Each test pins, through spmv_b200_info, what such a value stands for,
next to a value that shows the option is in effect on that matrix."""
import pytest

from cases import all_cases
from spmv_b200 import api, matrices as M

pytestmark = pytest.mark.gpu

CASES = all_cases()
INFO_KEYS = ("kernel", "requested", "ok", "m", "n", "nnz", "tpr", "parts", "ref_parts", "tiles", "tile_items", "sigma",
             "banner", "slices", "sell_variant", "padded_nnz", "csr5_p", "csr5_sigma", "csr5_bit_y_offset",
             "csr5_bit_scansum_offset", "csr5_num_offsets", "csr5_tail_start", "pipeline", "refreshable", "binned",
             "long_rows", "long_segs", "long_thr", "has_empty_rows", "x_bands", "auto_method", "seg_bands", "segments",
             "seg_cross", "layout_fallbacks", "band_cols", "far_permille", "active_rows", "owns_csr", "released_csr")


@pytest.fixture
def info(libpath):
    """info(a, method, **options): every INFO_KEYS value of a handle of `a` created under those options.  The options
    are set for that create only and restored afterwards, also when the create fails."""

    def create(a, method, **opts):
        old = {}
        try:
            for k, v in opts.items():
                old[k] = api.get_option(k)
                api.set_option(k, v)
            h = api.Handle(a.m, a.n, a.rowptr, a.col, a.val, method)
        finally:
            for k, v in old.items():
                api.set_option(k, v)
        try:
            got = {k: h.info(k) for k in INFO_KEYS}
        finally:
            h.destroy()
        assert got["ok"] == 1, (api.METHOD_NAMES[method], opts, api.last_error())
        return got

    return create


def test_tile_items_other_than_4_is_8(info):
    a = CASES["uni32"]()
    assert info(a, api.Method_Balanced_Yid, tile_items=4)["tile_items"] == 4
    for v in (5, 0):
        assert info(a, api.Method_Balanced_Yid, tile_items=v)["tile_items"] == 8, v


def test_sell_sigma_is_a_multiple_of_32_in_32_to_4096(info):
    a = CASES["uni32"]()
    for v, want in ((1, 32), (33, 32), (5000, 4096)):
        assert info(a, api.Method_SellCSigma, sell_sigma=v)["sigma"] == want, v


def test_sell_variant_other_than_0_or_2_is_automatic(info):
    a = CASES["uni32"]()
    auto = info(a, api.Method_SellCSigma, sell_variant=-1)
    assert auto["sell_variant"] in (0, 2)
    assert info(a, api.Method_SellCSigma, sell_variant=1) == auto
    assert info(a, api.Method_SellCSigma, sell_variant=2 - auto["sell_variant"])["sell_variant"] != auto["sell_variant"]


def test_csr5_sigma_other_than_4_8_16_is_automatic(info):
    a = CASES["uni32"]()  # below 2^25 non-zeros: the automatic sigma is 8
    assert info(a, api.Method_CSR5SPMV, csr5_sigma=4)["csr5_sigma"] == 4
    assert info(a, api.Method_CSR5SPMV, csr5_sigma=7)["csr5_sigma"] == 8


def test_block_nnz_is_at_least_32(info):
    a = CASES["uni32"]()
    at_32 = info(a, api.Method_Balanced, block_nnz=32)
    assert at_32["parts"] == -(-a.nnz // 32)
    assert info(a, api.Method_Balanced, block_nnz=1) == at_32


def test_sell_cap_is_at_least_32_and_negative_is_off(info):
    # slices of 32 rows of 100 entries (one with a hub row): a cap of 32 columns cuts every row, 1024 only the hub
    a = M.from_row_lengths([100] * 2047 + [6000], 8000)
    cap_32, cap_off, cap_1024 = (info(a, api.Method_SellCSigma, sell_cap=v) for v in (32, 0, 1024))
    assert len({cap_32["padded_nnz"], cap_off["padded_nnz"], cap_1024["padded_nnz"]}) == 3
    assert cap_off["long_rows"] == 0 and cap_32["long_rows"] > 0
    assert info(a, api.Method_SellCSigma, sell_cap=5) == cap_32
    assert info(a, api.Method_SellCSigma, sell_cap=-1) == cap_off


def test_negative_x_bands_is_off(info):
    a = CASES["uni32"]()
    assert info(a, api.Method_Parallel, x_bands=2)["x_bands"] == 2
    off = info(a, api.Method_Parallel, x_bands=-1)
    assert off["x_bands"] == 1 and off["active_rows"] == a.m


def test_seg_bands_1_is_never_and_above_64_is_64(info):
    a = CASES["uni16"]()
    band_seg, csr_vector = 8, 2  # spmv_b200_info "kernel": SPMV_B200_KERNEL_BAND_SEG, SPMV_B200_KERNEL_CSR_VECTOR
    assert info(a, api.Method_Parallel, seg_bands=2)["kernel"] == band_seg
    never = info(a, api.Method_Parallel, seg_bands=1)
    assert never["seg_bands"] == 0 and never["kernel"] == csr_vector
    most = info(a, api.Method_Parallel, seg_bands=100)
    assert most["seg_bands"] == 64 and most["x_bands"] == 64 and most["kernel"] == band_seg


def test_negative_long_thr_is_off(info):
    a = CASES["hub"]()
    assert info(a, api.Method_Parallel, long_thr=0)["long_rows"] > 0
    off = info(a, api.Method_Parallel, long_thr=-1)
    assert off["long_thr"] == 0x7FFFFFFF and off["long_rows"] == 0 and off["binned"] == 0


def test_tpr_not_a_power_of_two_takes_the_mean_but_no_row_bins(info):
    a = CASES["hub"]()  # short rows with hub rows: the automatic path bins the rows
    auto = info(a, api.Method_Parallel, tpr=0)
    assert auto["binned"] == 1
    odd = info(a, api.Method_Parallel, tpr=3)
    assert odd["tpr"] == auto["tpr"] and odd["binned"] == 0
