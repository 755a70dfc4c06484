"""Every SpMV kernel template instance the dispatcher can launch, against an exact reference.

Matrix values a_ij and vector entries x_j are integers in [-4, 4] (zeros included).  While every row has
sum_j |a_ij x_j| < 2^24 (fp32) or 2^53 (fp64), every partial sum in every summation order is exact, so every correct
kernel returns exactly y_ref = sum_j a_ij x_j computed in int64 -- a zero sum as +0.0, since every path accumulates
from +0.  The tests compare bits: a dropped, duplicated or misrouted entry, a carry added twice or to the wrong row,
or a band partial summed twice cannot hide behind a tolerance.  y is prefilled with 0.5, which no correct output can
be, so a row left unwritten shows too.

CONFIGS is one configuration (matrix, method, options, precision, peers, host or device x / y) per group of kernel
instances; each asserts through spmv_b200_info that it took the intended branch before it compares.  The non-finite
test puts +-Inf and NaN into x and NaN into a few values: rows that do not touch them must still be exact, which is
what catches padding or tail lanes that gather x[col] and multiply it by 0.  The coverage test runs every
configuration under torch.profiler and checks that every spmv-path instance compiled into libspmv_b200.so (listed
with cuobjdump) was launched: a new instance fails it until a configuration reaches it.
"""
import contextlib
import functools
import os
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import bits_equal
from spmv_b200 import api

# ---------------------------------------------------------------------------------------------------------------------
# kernel instances: names as cu++filt and the profiler print them, normalised to (family, template arguments)
# ---------------------------------------------------------------------------------------------------------------------
# the kernel families that spmv() (and spmv_b200_set_values) launch; builders, generators and cub are left out
FAMILIES = frozenset([
    "csr_reforder_kernel", "csr_vector_kernel", "csr_vector_list_kernel", "row_block_kernel", "merge_path_kernel",
    "nnz_split_kernel", "carry_fixup_kernel", "carry_group_kernel", "sell_kernel", "csr_tail_kernel",
    "long_seg_kernel", "long_final_kernel", "csr5_kernel", "csr5_tail_kernel", "bseg_kernel", "bseg_merge_kernel",
    "band_reduce_kernel", "peer_copy_kernel", "value_refresh_kernel"])

_CASTS = re.compile(r"^\((?:int|bool|unsigned int|long|long long|unsigned long|unsigned long long)\)")
_BOOLS = {"false": "0", "true": "1"}


def _template_arg(a):
    a = " ".join(a.split())
    a = _CASTS.sub("", a)  # cu++filt: (int)16, (bool)0
    a = _BOOLS.get(a, a)   # the profiler: false / true
    return {"uint32_t": "unsigned int", "unsigned": "unsigned int", "uint64_t": "unsigned long long"}.get(a, a)


def normalise(name):
    """(family, template arguments) of a demangled kernel name: 'void sb::csr_vector_kernel<double, (int)16, (int)4,
    (bool)0, (bool)0>(int, ...)' and 'void sb::csr_vector_kernel<double, 16, 4, false, false>(int, ...)' both give
    ('csr_vector_kernel', ('double', '16', '4', '0', '0'))."""
    s = name.strip()
    if s.startswith("void "):
        s = s[5:]
    lt, paren = s.find("<"), s.find("(")
    if lt < 0 or (0 <= paren < lt):
        return s[:paren if paren >= 0 else len(s)].split("::")[-1].strip(), ()
    family = s[:lt].split("::")[-1].strip()
    args, cur, depth = [], "", 0
    for ch in s[lt + 1:]:
        if ch == "<":
            depth += 1
        elif ch == ">":
            if depth == 0:
                break
            depth -= 1
        if ch == "," and depth == 0:
            args.append(cur)
            cur = ""
        else:
            cur += ch
    args.append(cur)
    return family, tuple(_template_arg(a) for a in args)


def spmv_instances(lib_path):
    """The spmv-path kernel instances compiled into the library: cuobjdump -symbols, demangled with cu++filt (both
    next to the nvcc that spmv_b200/build.py uses)."""
    from spmv_b200 import build
    bindir = os.path.dirname(build.NVCC)
    tools = [os.path.join(bindir, t) for t in ("cuobjdump", "cu++filt")]
    for t in tools:
        if not os.path.exists(t) and shutil.which(os.path.basename(t)) is None:
            pytest.skip(f"{os.path.basename(t)} not found next to {build.NVCC}")
    tools = [t if os.path.exists(t) else shutil.which(os.path.basename(t)) for t in tools]
    out = subprocess.run([tools[0], "-symbols", lib_path], capture_output=True, text=True, check=True).stdout
    mangled = sorted({line.split()[-1] for line in out.splitlines() if line.strip().startswith("STT_FUNC")})
    names = subprocess.run([tools[1]], input="\n".join(mangled), capture_output=True, text=True, check=True).stdout
    return {k for k in map(normalise, names.splitlines()) if k[0] in FAMILIES}


# recorded: cu++filt on libspmv_b200.so, and torch.profiler on one B200 run of this file
CUFILT_SAMPLES = {
    "void sb::csr_vector_kernel<double, (int)16, (int)4, (bool)0, (bool)0>(int, int, int, int, const int *, const int *, "
    "const T1 *, const T1 *, T1 *, sb::PeerList<T1>, int, int, const T1 *)":
        ("csr_vector_kernel", ("double", "16", "4", "0", "0")),
    "void sb::bseg_merge_kernel<float, unsigned long long, (bool)1>(int, int, int, const T2 *, const int *, "
    "const T1 *, T1 *, sb::PeerList<T1>)": ("bseg_merge_kernel", ("float", "unsigned long long", "1")),
    "void sb::carry_group_kernel<float>(int, const int *, const T1 *, T1 *, int *, T1 *)":
        ("carry_group_kernel", ("float",)),
}
PROFILER_SAMPLES = {
    "void sb::csr_vector_kernel<double, 1, 4, false, false>(int, int, int, int, int const*, int const*, "
    "double const*, double const*, double*, sb::PeerList<double>, int, int, double const*)":
        ("csr_vector_kernel", ("double", "1", "4", "0", "0")),
}


def test_normalise_kernel_names():
    for name, want in {**CUFILT_SAMPLES, **PROFILER_SAMPLES}.items():
        assert normalise(name) == want, name
    assert normalise("sb::peer_copy_kernel<double>") == ("peer_copy_kernel", ("double",))
    assert normalise("void sb::set_int_kernel(int *, int)") == ("set_int_kernel", ())


def test_library_lists_every_spmv_instance(libpath):
    """108 instances in 19 families at the time of writing; the per-family counts pin the dispatch table."""
    inst = spmv_instances(libpath)
    per_family = {}
    for fam, _ in inst:
        per_family[fam] = per_family.get(fam, 0) + 1
    assert set(per_family) == FAMILIES, sorted(FAMILIES - set(per_family))
    assert per_family["csr_vector_kernel"] == 36 and per_family["csr_vector_list_kernel"] == 12
    assert per_family["bseg_merge_kernel"] == 8 and per_family["sell_kernel"] == 6 and per_family["csr5_kernel"] == 6
    assert len(inst) == 108, len(inst)


# ---------------------------------------------------------------------------------------------------------------------
# integer matrices
# ---------------------------------------------------------------------------------------------------------------------
class IntCSR:
    def __init__(self, name, n, lens, rng, col_fn=None):
        lens = np.asarray(lens, dtype=np.int64)
        self.name, self.m, self.n = name, len(lens), int(n)
        self.rowptr = np.concatenate([[0], np.cumsum(lens)]).astype(np.int32)
        nnz = int(self.rowptr[-1])
        # unsorted columns, duplicates within a row wherever they happen to fall (n is small against some rows)
        self.col = rng.integers(0, self.n, nnz).astype(np.int32)
        if col_fn is not None:
            col_fn(self)
        self.a = rng.integers(-4, 5, nnz).astype(np.int64)
        self.x = rng.integers(-4, 5, self.n).astype(np.int64)
        self.x[::7] = 0

    @property
    def nnz(self):
        return int(self.rowptr[-1])

    def row_of_entry(self):
        return np.repeat(np.arange(self.m), np.diff(self.rowptr))


def _align(lens, q):
    """Append one row so that the next row starts on a multiple of q non-zeros."""
    pad = (-int(np.sum(lens))) % q
    return lens + [pad] if pad else lens


@functools.lru_cache(maxsize=None)
def matrix(name):
    rng = np.random.default_rng(sum(map(ord, name)) * 7919)
    if name == "edges":
        # row lengths 0..300 and around kLongSeg / 2 kLongSeg, runs of empty rows at row 0, across tile edges and at
        # row m-1, then rows of 128 starting on a multiple of 2048 (every CSR5 / tile / band-segment edge of 128..2048)
        lens = [0] * 40 + list(range(301)) + [2047, 2048, 2049, 4095, 4096, 4097] + list(rng.integers(0, 40, 600))
        lens = _align(lens, 2048) + [128] * 48 + [0] * 300 + list(rng.integers(0, 300, 200)) + [0] * 3
        return IntCSR(name, 10007, lens, rng)
    if name in ("bins", "bins256"):
        # short rows in all three length classes of the row bins plus hub rows of 1, 2 and 3 long-row segments; the
        # last rows (the CSR tail of SELL when m is not a multiple of sigma) hold hub rows past SELL's long_thr 4096
        m = 12000 if name == "bins" else 12032
        cls = rng.choice(3, size=m, p=[0.55, 0.3, 0.15])
        lens = np.where(cls == 0, rng.integers(0, 9, m), np.where(cls == 1, rng.integers(9, 33, m), rng.integers(33, 129, m)))
        hubs = {100: 600, 2000: 2047, 4000: 2048, 6000: 2049, m - 3: 4097, m - 2: 5000}
        for r, ln in hubs.items():
            lens[r] = ln
        return IntCSR(name, 49999, lens, rng)
    if name == "regions":
        # equal-length regions whose 512-nnz row blocks / 1024- and 2048-nnz tiles fall in every lane-width class
        lens = []
        for ln in (3, 6, 12, 24, 48, 100, 250):
            lens += [ln] * (16384 // ln)
        return IntCSR(name, 4099, lens, rng)
    if name == "big":
        # >= 1024 tiles for every tile kernel at its smallest tile; carry chains of a 70000-entry row cross many
        # 32-tile groups of the two-level fix-up
        lens = list(rng.integers(0, 22, 100000))
        lens[777], lens[50000], lens[99990] = 70000, 5000, 2049
        return IntCSR(name, 100003, lens, rng)
    if name in ("bseg_big", "bseg_small"):
        m, n = (30000, 100003) if name == "bseg_big" else (2000, 1009)

        def cols(A):
            row = A.row_of_entry()
            if name == "bseg_big":
                # one row with 5000 entries inside band 0 of 3 and of 40 bands (a segment over many chunks and tiles),
                # one with 600; band 7 of 40 left empty
                A.col[row == 5] = rng.integers(0, 2501, int(np.sum(row == 5)))
                A.col[row == 9] = rng.integers(40000, 42000, int(np.sum(row == 9)))
                in7 = (A.col >= 7 * 2501) & (A.col < 8 * 2501)
                A.col[in7] += 2501
        lens = list(rng.integers(0, 21, m))
        if name == "bseg_big":
            lens[5], lens[9] = 5000, 600
        return IntCSR(name, n, lens, rng, cols)
    if name == "fused":
        # 2^18 + 1 rows for the pipelined host path (m >= 2^16); a prime n, so the last of 3 bands is short
        return IntCSR(name, 1009, list(rng.integers(0, 6, (1 << 18) + 1)), rng)
    raise KeyError(name)


def exact_ref(A, a, x, dt):
    """y_i = sum_j a_ij x_j in int64, cast to dt; asserts the bound under which every summation order is exact."""
    prod = a * x[A.col]
    c = np.concatenate([[0], np.cumsum(prod)])
    cabs = np.concatenate([[0], np.cumsum(np.abs(prod))])
    bound = (1 << 24) if dt == np.float32 else (1 << 53)
    row_abs = cabs[A.rowptr[1:]] - cabs[A.rowptr[:-1]]
    assert row_abs.max(initial=0) < bound, (A.name, int(row_abs.max()))
    return (c[A.rowptr[1:]] - c[A.rowptr[:-1]]).astype(dt)


def nonfinite_ref(A, a, x, dt):
    """Reference for float a, x whose non-finite entries are +-Inf / NaN and the rest integers: NaN if a product is
    NaN (0 * Inf included) or the products hold both +Inf and -Inf, else +-Inf, else the exact finite sum.  Every
    summation order gives this."""
    with np.errstate(invalid="ignore"):
        prod = a * x[A.col]
    row = A.row_of_entry()
    hits = lambda mask: np.bincount(row, weights=mask, minlength=A.m) > 0
    nan, pinf, ninf = hits(np.isnan(prod)), hits(prod == np.inf), hits(prod == -np.inf)
    fin = np.where(np.isfinite(prod), prod, 0).astype(np.int64)
    c = np.concatenate([[0], np.cumsum(fin)])
    y = (c[A.rowptr[1:]] - c[A.rowptr[:-1]]).astype(dt)
    y[pinf] = np.inf
    y[ninf] = -np.inf
    y[nan | (pinf & ninf)] = np.nan
    return y


def assert_same(y, ref, tag):
    """Bits equal; NaN rows only need to be NaN (a NaN's sign and payload are not specified)."""
    ynan, rnan = np.isnan(y), np.isnan(ref)
    bad = np.nonzero(ynan != rnan)[0]
    assert len(bad) == 0, f"{tag}: NaN in {int(ynan.sum())} rows, expected {int(rnan.sum())}; first row {bad[0]}: " \
                          f"y={y[bad[0]]!r} ref={ref[bad[0]]!r}"
    ok = ~rnan
    if not bits_equal(y[ok], ref[ok]):
        rows = np.nonzero(ok)[0][y[ok].view(f"u{y.itemsize}") != ref[ok].view(f"u{y.itemsize}")]
        r = rows[0]
        raise AssertionError(f"{tag}: {len(rows)} rows differ; first row {r}: y={y[r]!r} ref={ref[r]!r}")


# ---------------------------------------------------------------------------------------------------------------------
# configurations
# ---------------------------------------------------------------------------------------------------------------------
@contextlib.contextmanager
def options(opts):
    """Set library options for the block and restore them afterwards, also when it fails."""
    old = {k: api.get_option(k) for k in opts}
    try:
        for k, v in opts.items():
            api.set_option(k, v)
        yield
    finally:
        for k, v in old.items():
            api.set_option(k, v)


class Config:
    def __init__(self, name, mat, method, opts=None, expect=None, peers=False, host=False, refresh=False, check=None):
        self.name, self.mat, self.method = name, mat, method
        self.opts, self.expect = dict(opts or {}), dict(expect or {})
        self.peers, self.host, self.refresh, self.check = peers, host, refresh, check


def _block_classes(h, A):
    """Lane-width class (0..5) of every row block of Method_Balanced, as row_block_kernel derives it."""
    sp = h.structure("splitter", np.int32)
    classes = set()
    for w in range(len(sp) - 1):
        r0, r1 = (0 if w == 0 else int(sp[w])), int(sp[w + 1])
        if r1 - r0 <= 0:
            continue
        avg = -(-int(A.rowptr[r1] - A.rowptr[r0]) // (r1 - r0))
        classes.add(next((k for k, lim in enumerate((7, 14, 28, 56, 112)) if avg <= lim), 5))
    return classes


def _tile_classes(h, A):
    """Lane-width class (0..5) of every equal-nnz tile of Method_Balanced_Yid, as nnz_split_kernel derives it."""
    tr = h.structure("tile_rows", np.int32)
    tile = 256 * h.info("tile_items")
    classes = set()
    for t in range(len(tr) - 1):
        r0, r_last = (0 if t == 0 else int(tr[t])), min(int(tr[t + 1]), A.m - 1)
        nrows = r_last - r0 + 1
        cnt = min(tile, A.nnz - t * tile)
        avg = -(-cnt // max(nrows, 1))
        classes.add(next((k for k, lim in enumerate((4, 8, 16, 32, 64)) if avg <= lim), 5))
    return classes


def _all_six(fn):
    def check(h, A):
        assert fn(h, A) == set(range(6)), fn(h, A)
    return check


def _tiles_at_least(k):
    def check(h, A):
        assert h.info("tiles") >= k, h.info("tiles")
    return check


def _tiles_below(k):
    def check(h, A):
        assert h.info("tiles") < k, h.info("tiles")
    return check


def _seg_carries(big):
    def check(h, A):  # one carry slot per 256-entry chunk: 8 per tile of 2048 entries
        assert h.info("seg_cross") == 1
        assert (h.info("tiles") * 8 >= 1024) == big, h.info("tiles")
    return check


S, P, B, B2, Y, SELL, C5 = (api.Method_Serial, api.Method_Parallel, api.Method_Balanced, api.Method_Balanced2,
                            api.Method_Balanced_Yid, api.Method_SellCSigma, api.Method_CSR5SPMV)
K = {v: k for k, v in api.KERNEL_NAMES.items()}


def _configs():
    c = []
    c.append(Config("serial", "edges", S, expect={"kernel": K["csr_reforder"]}))
    c.append(Config("serial_peers", "edges", S, peers=True))
    for t in (1, 2, 4, 8, 16, 32):
        o = {"tpr": t, "long_thr": -1}
        e = {"kernel": K["csr_vector"], "tpr": t, "x_bands": 1, "long_rows": 0}
        c.append(Config(f"vector_tpr{t}", "edges", P, o, e))
        c.append(Config(f"vector_tpr{t}_peers", "edges", P, o, e, peers=True))
        c.append(Config(f"vector_tpr{t}_fused", "fused", P, {**o, "x_bands": 3},
                        {"kernel": K["csr_vector"], "tpr": t, "x_bands": 3, "pipeline": 1}, host=True))
    for peers in (False, True):
        sfx = "_peers" if peers else ""
        c.append(Config("banded" + sfx, "fused", P, {"x_bands": 3, "long_thr": -1}, {"x_bands": 3}, peers=peers))
        c.append(Config("bins" + sfx, "bins", P, {}, {"kernel": K["csr_vector"], "binned": 1, "tpr": 4}, peers=peers))
        c.append(Config("row_blocks" + sfx, "regions", B, {}, {"kernel": K["row_blocks"]}, peers=peers,
                        check=_all_six(_block_classes)))
    for ipt in (4, 8):
        o = {"force_merge": 1, "tile_items": ipt}
        c.append(Config(f"merge_ipt{ipt}", "edges", B2, o, {"kernel": K["merge_path"], "tile_items": ipt},
                        check=_tiles_below(1024)))
        c.append(Config(f"nnz_split_ipt{ipt}", "regions", Y, {"tile_items": ipt},
                        {"kernel": K["nnz_split"], "tile_items": ipt}, check=_all_six(_tile_classes)))
    c.append(Config("merge_ipt4_groups", "big", B2, {"force_merge": 1, "tile_items": 4},
                    {"kernel": K["merge_path"], "tile_items": 4}, check=_tiles_at_least(1024)))
    c.append(Config("nnz_split_ipt4_groups", "big", Y, {"tile_items": 4}, {"kernel": K["nnz_split"], "tile_items": 4},
                    check=_tiles_at_least(1024)))
    c.append(Config("merge_ipt8_peers", "edges", B2, {"force_merge": 1}, {"kernel": K["merge_path"]}, peers=True))
    c.append(Config("nnz_split_ipt8_peers", "regions", Y, {}, {"kernel": K["nnz_split"]}, peers=True))
    for v in (0, 2):
        c.append(Config(f"sell_v{v}", "edges", SELL, {"sell_variant": v},
                        {"kernel": K["sell"], "sell_variant": v, "banner": 1280}))
        c.append(Config(f"sell_v{v}_tail_hubs", "bins", SELL, {"sell_variant": v},
                        {"kernel": K["sell"], "sell_variant": v, "banner": 11776}))
    c.append(Config("sell_peers", "bins256", SELL, {}, {"kernel": K["sell"], "banner": 12032}, peers=True))
    c.append(Config("sell_tail_peers", "bins", SELL, {}, {"kernel": K["sell"], "banner": 11776}, peers=True))
    for sg in (4, 8, 16):
        c.append(Config(f"csr5_sigma{sg}", "edges", C5, {"csr5_sigma": sg},
                        {"kernel": K["csr5"], "csr5_sigma": sg, "has_empty_rows": 1}))
        c.append(Config(f"csr5_sigma{sg}_groups", "big", C5, {"csr5_sigma": sg},
                        {"kernel": K["csr5"], "csr5_sigma": sg}, check=lambda h, A: h.info("csr5_p") >= 1024))
    c.append(Config("csr5_peers", "edges", C5, {}, {"kernel": K["csr5"]}, peers=True))
    c.append(Config("csr5_refresh", "edges", C5, {"refresh": 1}, {"kernel": K["csr5"], "refreshable": 1}, refresh=True))
    c.append(Config("sell_refresh", "bins", SELL, {"refresh": 1}, {"kernel": K["sell"], "refreshable": 1}, refresh=True))
    c.append(Config("serial_refresh", "edges", S, {"refresh": 1}, {"refreshable": 1}, refresh=True))
    for bands, ctas in ((3, 2), (40, 3)):
        for mat in ("bseg_big", "bseg_small"):
            for peers in (False, True):
                c.append(Config(f"bseg{bands}_ctas{ctas}_{mat}" + ("_peers" if peers else ""), mat, P,
                                {"seg_bands": bands, "seg_ctas": ctas},
                                {"kernel": K["band_seg"], "seg_bands": bands, "seg_ctas": ctas}, peers=peers,
                                check=_seg_carries(mat == "bseg_big") if not peers else None))
    return c


CONFIGS = _configs()
DTYPES = {"fp64": np.float64, "fp32": np.float32}


def run(cfg, dt, a=None, x=None):
    """Create the handle of `cfg` at precision dt, check its branch, run one SpMV (prefilled y, and peer buffers, of
    0.5) and return (y, [peer copies], handle, matrix).  a / x override the matrix values / x (floats)."""
    import torch
    A = matrix(cfg.mat)
    val = (A.a if a is None else a).astype(dt)
    xv = (A.x if x is None else x).astype(dt)
    with options(cfg.opts):  # held through the first spmv: seg_ctas is read at the first band-segment launch
        h = api.Handle(A.m, A.n, A.rowptr, A.col, val, cfg.method)
        try:
            peers_out = []
            if cfg.host:
                y = np.full(A.m, 0.5, dtype=dt)
                h.spmv(xv, y)
            else:
                tdt = torch.float64 if dt == np.float64 else torch.float32
                xd = torch.from_numpy(xv).cuda()
                yd = torch.full((A.m,), 0.5, dtype=tdt, device="cuda")
                big = torch.full((2, A.m + 3), 0.5, dtype=tdt, device="cuda")
                if cfg.peers:
                    h.set_y_peers([big[i, 3:].data_ptr() for i in range(2)])
                h.spmv(xd, yd)
                h.sync()
                y = yd.cpu().numpy()
                if cfg.peers:
                    peers_out = [big[i, 3:].cpu().numpy() for i in range(2)]
                    assert (big[:, :3].cpu().numpy() == 0.5).all(), "peer write before the slice"
            for key, want in cfg.expect.items():
                assert h.info(key) == want, f"{cfg.name}: info({key!r}) = {h.info(key)}, expected {want}"
            if cfg.check is not None:
                cfg.check(h, A)
        except BaseException:
            h.destroy()
            raise
    return y, peers_out, h, A


def run_exact(cfg, dt):
    tag = f"{cfg.name}/{np.dtype(dt).name}"
    y, peers_out, h, A = run(cfg, dt)
    try:
        ref = exact_ref(A, A.a, A.x, dt)
        assert_same(y, ref, tag)
        for i, yp in enumerate(peers_out):
            assert_same(yp, ref, f"{tag} peer {i}")
        if cfg.refresh:
            import torch
            a2 = np.random.default_rng(5).integers(-4, 5, A.nnz).astype(np.int64)
            h.set_values(torch.from_numpy(a2.astype(dt)).cuda())
            y2 = torch.full((A.m,), 0.5, dtype=torch.float64 if dt == np.float64 else torch.float32, device="cuda")
            h.spmv(torch.from_numpy(A.x.astype(dt)).cuda(), y2)
            h.sync()
            assert_same(y2.cpu().numpy(), exact_ref(A, a2, A.x, dt), tag + " after set_values")
    finally:
        h.destroy()


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("cfg", CONFIGS, ids=[c.name for c in CONFIGS])
def test_instance_exact(libpath, cfg, dt):
    run_exact(cfg, DTYPES[dt])


# one configuration per kernel family (and per SELL flavour), rerun with non-finite inputs
NONFINITE = ["serial", "vector_tpr4", "vector_tpr16_peers", "vector_tpr2_fused", "banded_peers", "bins_peers",
             "row_blocks", "merge_ipt4", "merge_ipt8_peers", "nnz_split_ipt8", "sell_v0", "sell_v2",
             "sell_v0_tail_hubs", "sell_peers", "csr5_sigma4", "csr5_sigma16", "bseg40_ctas3_bseg_small_peers",
             "bseg3_ctas2_bseg_big"]


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("name", NONFINITE)
def test_instance_nonfinite(libpath, name, dt):
    """+Inf at x[0] (where padding slots would gather), -Inf and NaN at two more columns, NaN in a few values: rows
    that touch none of them must stay exact, the others follow the IEEE rules."""
    dt = DTYPES[dt]
    cfg = next(c for c in CONFIGS if c.name == name)
    A = matrix(cfg.mat)
    x = A.x.astype(np.float64)
    x[0], x[A.n // 2], x[A.n // 3] = np.inf, -np.inf, np.nan
    a = A.a.astype(np.float64)
    a[::997] = np.nan
    y, peers_out, h, _ = run(cfg, dt, a=a, x=x)
    h.destroy()
    ref = nonfinite_ref(A, a, x, dt)
    clean = int(np.sum(np.isfinite(ref)))
    assert clean > A.m // 4 and clean < A.m, (name, clean, A.m)  # both kinds of rows are there
    assert_same(y, ref, f"nonfinite/{name}/{np.dtype(dt).name}")
    for i, yp in enumerate(peers_out):
        assert_same(yp, ref, f"nonfinite/{name}/{np.dtype(dt).name} peer {i}")


@pytest.mark.gpu
@pytest.mark.parametrize("dt", list(DTYPES), ids=list(DTYPES))
@pytest.mark.parametrize("m,n", [(1, 1), (31, 1), (32, 7), (33, 7), (33, 1)])
def test_tiny_shapes_every_method(libpath, m, n, dt):
    """m in {1, 31, 32, 33} and n = 1 (every gather hits x[0]), with an empty row and duplicated columns."""
    import torch
    dt = DTYPES[dt]
    rng = np.random.default_rng(m * 100 + n)
    lens = rng.integers(0, 70, m)
    lens[m // 2] = 0
    A = IntCSR(f"tiny{m}x{n}", n, lens, rng)
    ref = exact_ref(A, A.a, A.x, dt)
    tdt = torch.float64 if dt == np.float64 else torch.float32
    for method in range(7):
        h = api.Handle(A.m, A.n, A.rowptr, A.col, A.a.astype(dt), method)
        yd = torch.full((m,), 0.5, dtype=tdt, device="cuda")
        h.spmv(torch.from_numpy(A.x.astype(dt)).cuda(), yd)
        h.sync()
        tag = f"tiny {m}x{n} {api.METHOD_NAMES[method]}[{h.kernel}] {np.dtype(dt).name}"
        h.destroy()
        assert_same(yd.cpu().numpy(), ref, tag)


@pytest.mark.gpu
def test_every_instance_is_launched(libpath):
    """All configurations, fp64 and fp32, under torch.profiler: the launched kernels must include every spmv-path
    instance the library holds."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    want = spmv_instances(libpath)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for cfg in CONFIGS:
            for dt in DTYPES.values():
                run_exact(cfg, dt)
        torch.cuda.synchronize()
    raw = {e.name for e in prof.events() if "kernel" in e.name}
    if not raw:
        pytest.skip("torch.profiler recorded no CUDA kernels (no CUPTI activity on this machine)")
    seen = {k for k in map(normalise, raw) if k[0] in FAMILIES}
    print(f"launched {len(want & seen)} of {len(want)} spmv-path instances; e.g. "
          f"{next(n for n in sorted(raw) if 'csr_vector_kernel' in n)!r}")
    missing = sorted(want - seen)
    assert not missing, f"{len(missing)} of {len(want)} instances never launched:\n" + \
        "\n".join(f"  {f}<{', '.join(a)}>" for f, a in missing)
