"""Python mirror of the reference's C interface (include/spmv.h) over libspmv_b200.so via ctypes.

Same entry points, same argument order and meaning as the reference's API
(reference include/spmv.h:19,26,41-52,65-71): ``spmv_create_handle_all_in_one``, ``spmv``,
``spmv_clear_handle``, ``spmv_destory_handle`` (sic), plus the extension calls of include/spmv_b200.h.
Array arguments may be numpy arrays (host), torch tensors (host or CUDA), or raw integer addresses.

This module is plumbing only: every number comes out of the CUDA library.  If the library is missing it
raises -- there is no fallback of any kind.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libspmv_b200.so")

# SPMV_METHODS / VECTORIZED_WAY (reference include/spmv_Defines.h:18-35)
Method_Serial, Method_Parallel, Method_Balanced, Method_Balanced2, Method_Balanced_Yid, \
    Method_SellCSigma, Method_CSR5SPMV, Method_Total_Size, Method_Numa = range(9)
VECTOR_NONE, VECTOR_AVX2, VECTOR_AVX512, VECTOR_TOTAL_SIZE = range(4)
METHOD_NAMES = ["Method_Serial", "Method_Parallel", "Method_Balanced", "Method_Balanced2",
                "Method_BalancedYid", "Method_SellCSigma", "Method_Csr5Spmv"]

KERNEL_NAMES = {0: "none", 1: "csr_reforder", 2: "csr_vector", 3: "row_blocks", 4: "merge_path",
                5: "nnz_split", 6: "sell", 7: "csr5", 8: "band_seg"}

# every symbol include/spmv.h and include/spmv_b200.h declare
EXPORTED_FUNCTIONS = [
    "spmv_create_handle_all_in_one", "spmv", "spmv_clear_handle", "spmv_destory_handle",
    "spmv_b200_version", "spmv_b200_last_error", "spmv_b200_clear_error", "spmv_b200_set_stream",
    "spmv_b200_sync", "spmv_b200_set_option", "spmv_b200_get_option", "spmv_b200_info",
    "spmv_b200_structure", "spmv_b200_launch_count", "spmv_b200_partition_rows", "spmv_b200_malloc",
    "spmv_b200_free", "spmv_b200_memcpy", "spmv_b200_gen_laplacian2d", "spmv_b200_gen_stencil27",
    "spmv_b200_gen_uniform", "spmv_b200_gen_rmat", "spmv_b200_gen_x", "spmv_b200_csr_free",
    "spmv_b200_set_y_peers", "spmv_b200_ipc_export", "spmv_b200_ipc_open", "spmv_b200_ipc_close",
    "spmv_b200_recommend_method", "spmv_b200_bands", "spmv_b200_band_columns", "spmv_b200_spmv_bands",
    "spmv_b200_spmv_finish", "spmv_b200_memcpy_async", "spmv_b200_stream_write32", "spmv_b200_stream_wait32_geq",
    "spmv_b200_reorder", "spmv_b200_permute_csr", "spmv_b200_update_values", "spmv_b200_live_allocations",
    "spmv_b200_set_values"]
EXPORTED_DATA = ["Methods_names", "Vectorized_names", "funcNames"]


class spmv_Handle(C.Structure):
    """struct spmv_Handle, field for field (reference include/spmv_Defines.h:44-70)."""
    _fields_ = [("spmvMethod", C.c_int), ("data_size", C.c_ulong), ("nthreads", C.c_ulong),
                ("vectorizedWay", C.c_int), ("Level_3_opt_used", C.c_int),
                ("RowPtr", C.c_void_p), ("ColIdx", C.c_void_p), ("index", C.c_void_p),
                ("Matrix_Val", C.c_void_p), ("Y_temp", C.c_void_p), ("extraHandle", C.c_void_p)]


spmv_Handle_t = C.POINTER(spmv_Handle)


class DeviceCSR(C.Structure):
    """struct spmv_b200_csr (include/spmv_b200.h)."""
    _fields_ = [("m", C.c_int), ("n", C.c_int), ("nnz", C.c_longlong), ("RowPtr", C.c_void_p),
                ("ColIdx", C.c_void_p), ("Val", C.c_void_p), ("size", C.c_ulong)]


_lib = None


def lib() -> C.CDLL:
    """Load libspmv_b200.so (built in-tree by spmv_b200.build); fail loudly when absent."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} is missing: run `python -m spmv_b200.build` "
                          "(spmv_b200 has no CPU / PyTorch fallback)")
    L = C.CDLL(LIB_PATH)  # RTLD_LOCAL: the reference .so exports the same names
    vp, i, ul, ll = C.c_void_p, C.c_int, C.c_ulong, C.c_longlong
    L.spmv_create_handle_all_in_one.argtypes = [C.POINTER(spmv_Handle_t), i, i, vp, vp, vp, ul, i, ul, i, C.c_char_p]
    L.spmv_create_handle_all_in_one.restype = None
    L.spmv.argtypes = [spmv_Handle_t, i, vp, vp, vp, vp, vp]
    L.spmv.restype = None
    L.spmv_clear_handle.argtypes = [spmv_Handle_t]
    L.spmv_clear_handle.restype = None
    L.spmv_destory_handle.argtypes = [spmv_Handle_t]
    L.spmv_destory_handle.restype = None
    L.spmv_b200_version.restype = i
    L.spmv_b200_last_error.restype = C.c_char_p
    L.spmv_b200_clear_error.restype = None
    L.spmv_b200_set_stream.argtypes = [spmv_Handle_t, vp]
    L.spmv_b200_set_stream.restype = None
    L.spmv_b200_sync.argtypes = [spmv_Handle_t]
    L.spmv_b200_sync.restype = None
    L.spmv_b200_set_option.argtypes = [C.c_char_p, ll]
    L.spmv_b200_get_option.argtypes = [C.c_char_p]
    L.spmv_b200_get_option.restype = ll
    L.spmv_b200_info.argtypes = [spmv_Handle_t, C.c_char_p]
    L.spmv_b200_info.restype = ll
    L.spmv_b200_structure.argtypes = [spmv_Handle_t, C.c_char_p, vp, C.c_size_t]
    L.spmv_b200_structure.restype = ll
    L.spmv_b200_launch_count.restype = C.c_ulonglong
    L.spmv_b200_live_allocations.restype = ll
    L.spmv_b200_partition_rows.argtypes = [vp, i, i, vp]
    L.spmv_b200_recommend_method.argtypes = [i, vp]
    L.spmv_b200_malloc.argtypes = [C.c_size_t]
    L.spmv_b200_malloc.restype = vp
    L.spmv_b200_free.argtypes = [vp]
    L.spmv_b200_free.restype = None
    L.spmv_b200_memcpy.argtypes = [vp, vp, C.c_size_t, i]
    L.spmv_b200_set_y_peers.argtypes = [spmv_Handle_t, i, C.POINTER(vp)]
    L.spmv_b200_ipc_export.argtypes = [vp, C.c_char_p]
    L.spmv_b200_ipc_open.argtypes = [C.c_char_p]
    L.spmv_b200_ipc_open.restype = vp
    L.spmv_b200_ipc_close.argtypes = [vp]
    L.spmv_b200_bands.argtypes = [spmv_Handle_t]
    L.spmv_b200_band_columns.argtypes = [spmv_Handle_t, i, C.POINTER(ll), C.POINTER(ll)]
    L.spmv_b200_spmv_bands.argtypes = [spmv_Handle_t, i, i, vp]
    L.spmv_b200_spmv_finish.argtypes = [spmv_Handle_t, vp]
    L.spmv_b200_update_values.argtypes = [spmv_Handle_t, vp]
    L.spmv_b200_set_values.argtypes = [spmv_Handle_t, vp]
    L.spmv_b200_reorder.argtypes = [i, vp, vp, vp]
    L.spmv_b200_permute_csr.argtypes = [i, vp, vp, vp, ul, vp, vp, vp, vp]
    L.spmv_b200_memcpy_async.argtypes = [vp, vp, C.c_size_t, vp]
    L.spmv_b200_stream_write32.argtypes = [vp, vp, C.c_uint]
    L.spmv_b200_stream_wait32_geq.argtypes = [vp, vp, C.c_uint]
    P = C.POINTER(DeviceCSR)
    L.spmv_b200_gen_laplacian2d.argtypes = [i, i, ul, P]
    L.spmv_b200_gen_stencil27.argtypes = [i, i, i, ul, P]
    L.spmv_b200_gen_uniform.argtypes = [i, i, i, C.c_ulonglong, ll, i, ul, P]
    L.spmv_b200_gen_rmat.argtypes = [i, i, C.c_ulonglong, ul, P]
    L.spmv_b200_gen_x.argtypes = [vp, ll, C.c_ulonglong, i, ul]
    L.spmv_b200_csr_free.argtypes = [P]
    L.spmv_b200_csr_free.restype = None
    _lib = L
    return L


def _addr(a):
    """Raw address of a numpy array / torch tensor / int / None."""
    if a is None:
        return None
    if isinstance(a, int):
        return a
    if isinstance(a, np.ndarray):
        return a.ctypes.data
    if hasattr(a, "data_ptr"):
        return a.data_ptr()
    raise TypeError(f"cannot take the address of {type(a)}")


def last_error() -> str:
    return lib().spmv_b200_last_error().decode()


def clear_error() -> None:
    lib().spmv_b200_clear_error()


# ---------------------------------------------------------------------------------------------
# the four reference entry points
# ---------------------------------------------------------------------------------------------
def spmv_create_handle_all_in_one(m, n, RowPtr, ColIdx, Matrix_Val, nthreads, Function, size,
                                  vectorizedWay=VECTOR_AVX2, MtxToken=b""):
    """reference include/spmv.h:41-52.  Returns the spmv_Handle_t (the C API's out-parameter)."""
    h = spmv_Handle_t()
    lib().spmv_create_handle_all_in_one(C.byref(h), int(m), int(n), _addr(RowPtr), _addr(ColIdx),
                                        _addr(Matrix_Val), int(nthreads), int(Function), int(size),
                                        int(vectorizedWay), MtxToken if isinstance(MtxToken, bytes) else MtxToken.encode())
    return h


def spmv(handle, m, RowPtr, ColIdx, Matrix_Val, Vector_Val_X, Vector_Val_Y):
    """reference include/spmv.h:65-71.  y is written in place (host: complete on return)."""
    lib().spmv(handle, int(m), _addr(RowPtr), _addr(ColIdx), _addr(Matrix_Val), _addr(Vector_Val_X),
               _addr(Vector_Val_Y))


def spmv_clear_handle(handle):
    lib().spmv_clear_handle(handle)


def spmv_destory_handle(handle):
    lib().spmv_destory_handle(handle)


# ---------------------------------------------------------------------------------------------
# convenience wrapper used by tests / bench (keeps the borrowed arrays alive, like a C caller would)
# ---------------------------------------------------------------------------------------------
class Handle:
    def __init__(self, m, n, RowPtr, ColIdx, Matrix_Val, method, size=None, nthreads=1,
                 vectorizedWay=VECTOR_AVX2, token=b"spmv_b200"):
        if size is None:
            size = Matrix_Val.dtype.itemsize if isinstance(Matrix_Val, np.ndarray) else Matrix_Val.element_size()
        self.m, self.n, self.size = int(m), int(n), int(size)
        self.keep = (RowPtr, ColIdx, Matrix_Val)
        self.h = spmv_create_handle_all_in_one(m, n, RowPtr, ColIdx, Matrix_Val, nthreads, method, size,
                                               vectorizedWay, token)
        if not self.h or self.info("ok") != 1:
            err = last_error()
            self.destroy()
            raise RuntimeError("spmv_create_handle_all_in_one failed: " + err)

    @property
    def struct(self) -> spmv_Handle:
        return self.h.contents

    def spmv(self, x, y):
        rp, ci, va = self.keep
        spmv(self.h, self.m, rp, ci, va, x, y)
        return y

    def info(self, key: str) -> int:
        return int(lib().spmv_b200_info(self.h, key.encode()))

    @property
    def kernel(self) -> str:
        return KERNEL_NAMES.get(self.info("kernel"), "?")

    def structure(self, name: str, dtype) -> np.ndarray:
        nbytes = lib().spmv_b200_structure(self.h, name.encode(), None, 0)
        if nbytes < 0:
            raise KeyError(name)
        out = np.empty(nbytes // np.dtype(dtype).itemsize, dtype=dtype)
        if nbytes:
            got = lib().spmv_b200_structure(self.h, name.encode(), out.ctypes.data, out.nbytes)
            if got != nbytes:
                raise RuntimeError(last_error())
        return out

    def set_y_peers(self, ptrs):
        """Extra destinations of y (addresses); [] switches the fused scatter off."""
        arr = (C.c_void_p * max(len(ptrs), 1))(*[int(p) for p in ptrs])
        if lib().spmv_b200_set_y_peers(self.h, len(ptrs), arr) != 0:
            raise ValueError("set_y_peers: at most 8 destinations")

    def update_values(self, Matrix_Val=None):
        """Rebuild the device layout with new values on the same pattern (spmv_b200_update_values)."""
        if Matrix_Val is not None:
            self.keep = (self.keep[0], self.keep[1], Matrix_Val)
        if lib().spmv_b200_update_values(self.h, _addr(Matrix_Val) if Matrix_Val is not None else None) != 0:
            raise RuntimeError("spmv_b200_update_values failed: " + last_error())

    def set_values(self, Matrix_Val=None):
        """New values on the same pattern, in place and stream-ordered (spmv_b200_set_values; the handle must have been
        created with option "refresh").  Matrix_Val: nnz values of the handle's precision in the order of the ColIdx
        given at create, as numpy, CPU torch or CUDA torch; None re-reads the array given at create.  A CUDA source is
        kept alive here until the next set_values or destroy, since the refresh reads it on the stream."""
        addr = None
        if Matrix_Val is not None:
            if isinstance(Matrix_Val, np.ndarray):
                floating, itemsize = Matrix_Val.dtype.kind == "f", Matrix_Val.dtype.itemsize
                count, contiguous = Matrix_Val.size, Matrix_Val.flags.c_contiguous
            else:
                floating, itemsize = Matrix_Val.is_floating_point(), Matrix_Val.element_size()
                count, contiguous = Matrix_Val.numel(), Matrix_Val.is_contiguous()
            nnz = self.info("nnz")
            if not floating or itemsize != self.size:
                raise ValueError(f"set_values: the handle holds {8 * self.size}-bit floats, got {Matrix_Val.dtype}")
            if count != nnz or not contiguous:
                raise ValueError(f"set_values: need {nnz} contiguous values, got {count}")
            addr = _addr(Matrix_Val)
        if lib().spmv_b200_set_values(self.h, addr) != 0:
            raise RuntimeError(last_error())
        self.values_source = Matrix_Val if getattr(Matrix_Val, "is_cuda", False) else None

    def bands(self) -> int:
        """Column bands that can be staged one by one (1: use spmv())."""
        return int(lib().spmv_b200_bands(self.h))

    def band_columns(self, band: int):
        lo, hi = C.c_longlong(), C.c_longlong()
        if lib().spmv_b200_band_columns(self.h, band, C.byref(lo), C.byref(hi)) != 0:
            raise IndexError(band)
        return int(lo.value), int(hi.value)

    def spmv_bands(self, first: int, count: int, x):
        if lib().spmv_b200_spmv_bands(self.h, first, count, _addr(x)) != 0:
            raise RuntimeError("spmv_b200_spmv_bands: " + last_error())

    def spmv_finish(self, y):
        if lib().spmv_b200_spmv_finish(self.h, _addr(y)) != 0:
            raise RuntimeError("spmv_b200_spmv_finish: " + last_error())

    def set_stream(self, cuda_stream: int):
        lib().spmv_b200_set_stream(self.h, cuda_stream)

    def sync(self):
        lib().spmv_b200_sync(self.h)

    def destroy(self):
        if getattr(self, "h", None):
            spmv_destory_handle(self.h)
            self.h = None
        self.values_source = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def device_malloc(nbytes: int) -> int:
    p = lib().spmv_b200_malloc(nbytes)
    if not p:
        raise MemoryError(last_error())
    return int(p)


def device_free(ptr: int) -> None:
    lib().spmv_b200_free(ptr)


def device_memcpy(dst, src, nbytes: int, kind: int) -> None:
    """kind 0 H2D, 1 D2H, 2 D2D (synchronous)."""
    if lib().spmv_b200_memcpy(_addr(dst), _addr(src), nbytes, kind) != 0:
        raise RuntimeError(last_error())


def memcpy_async(dst, src, nbytes: int, stream: int) -> None:
    """Device-to-device copy (dst may be a peer mapping) enqueued on a CUDA stream (raw handle)."""
    if lib().spmv_b200_memcpy_async(_addr(dst), _addr(src), nbytes, stream) != 0:
        raise RuntimeError(last_error())


def stream_write32(stream: int, ptr: int, value: int) -> None:
    if lib().spmv_b200_stream_write32(stream, ptr, value) != 0:
        raise RuntimeError(last_error())


def stream_wait32_geq(stream: int, ptr: int, value: int) -> None:
    if lib().spmv_b200_stream_wait32_geq(stream, ptr, value) != 0:
        raise RuntimeError(last_error())


def ipc_export(ptr: int) -> bytes:
    buf = C.create_string_buffer(64)
    if lib().spmv_b200_ipc_export(ptr, buf) != 0:
        raise RuntimeError(last_error())
    return buf.raw


def ipc_open(handle: bytes) -> int:
    p = lib().spmv_b200_ipc_open(handle)
    if not p:
        raise RuntimeError(last_error())
    return int(p)


def ipc_close(ptr: int) -> None:
    lib().spmv_b200_ipc_close(ptr)


def set_option(key: str, value: int) -> None:
    if lib().spmv_b200_set_option(key.encode(), int(value)) != 0:
        raise KeyError(key)


def get_option(key: str) -> int:
    return int(lib().spmv_b200_get_option(key.encode()))


def launch_count() -> int:
    return int(lib().spmv_b200_launch_count())


def live_allocations() -> int:
    """Device allocations the library holds for its own use (handles, layouts, temporaries of a running call)."""
    return int(lib().spmv_b200_live_allocations())


def partition_rows(rowptr: np.ndarray, parts: int) -> np.ndarray:
    """Equal-nnz row partition = reference init_csrSplitter_balanced2 with nthreads=parts (host code)."""
    rp = np.ascontiguousarray(rowptr, dtype=np.int32)
    out = np.empty(parts + 1, dtype=np.int32)
    if lib().spmv_b200_partition_rows(rp.ctypes.data, len(rp) - 1, parts, out.ctypes.data) != 0:
        raise ValueError("bad partition arguments")
    return out


def reorder(rowptr: np.ndarray, col: np.ndarray) -> np.ndarray:
    """index[i] = original row placed at position i: the permutation create stores in handle->index with option
    "reorder" (reverse Cuthill-McKee; host code)."""
    rp = np.ascontiguousarray(rowptr, dtype=np.int32)
    ci = np.ascontiguousarray(col, dtype=np.int32)
    out = np.empty(len(rp) - 1, dtype=np.int32)
    if lib().spmv_b200_reorder(len(rp) - 1, rp.ctypes.data, ci.ctypes.data, out.ctypes.data) != 0:
        raise ValueError("bad reorder arguments")
    return out


def permute_csr(rowptr, col, val, index):
    """(rowptr', col', val') of A' = P A P^T (host code)."""
    rp = np.ascontiguousarray(rowptr, dtype=np.int32)
    ci = np.ascontiguousarray(col, dtype=np.int32)
    va = np.ascontiguousarray(val)
    ix = np.ascontiguousarray(index, dtype=np.int32)
    rp2, ci2, va2 = np.empty_like(rp), np.empty_like(ci), np.empty_like(va)
    if lib().spmv_b200_permute_csr(len(rp) - 1, rp.ctypes.data, ci.ctypes.data, va.ctypes.data, va.dtype.itemsize,
                                   ix.ctypes.data, rp2.ctypes.data, ci2.ctypes.data, va2.ctypes.data) != 0:
        raise ValueError("bad permute arguments (index must be a permutation, the pattern square)")
    return rp2, ci2, va2


def recommend_method(rowptr: np.ndarray) -> int:
    """SPMV_METHODS value this library runs fastest for a matrix with these row lengths (host code)."""
    rp = np.ascontiguousarray(rowptr, dtype=np.int32)
    r = lib().spmv_b200_recommend_method(len(rp) - 1, rp.ctypes.data)
    if r < 0:
        raise ValueError("bad arguments")
    return r


# ---------------------------------------------------------------------------------------------
# device generators
# ---------------------------------------------------------------------------------------------
class DeviceMatrix:
    """A generated device-resident CSR; frees its arrays on destroy()."""

    def __init__(self, csr: DeviceCSR, name: str):
        self.c, self.name = csr, name

    m = property(lambda s: s.c.m)
    n = property(lambda s: s.c.n)
    nnz = property(lambda s: int(s.c.nnz))
    size = property(lambda s: int(s.c.size))
    RowPtr = property(lambda s: s.c.RowPtr)
    ColIdx = property(lambda s: s.c.ColIdx)
    Val = property(lambda s: s.c.Val)

    def min_bytes(self) -> int:
        v = self.size
        return self.nnz * (v + 4) + (self.m + 1) * 4 + self.m * v + self.n * v

    def handle(self, method, nthreads=1) -> Handle:
        return Handle(self.m, self.n, self.RowPtr, self.ColIdx, self.Val, method, self.size, nthreads)

    def to_host(self):
        from .matrices import CSR
        dt = np.float64 if self.size == 8 else np.float32
        rp = np.empty(self.m + 1, np.int32)
        ci = np.empty(self.nnz, np.int32)
        va = np.empty(self.nnz, dt)
        L = lib()
        for dst, src in ((rp, self.RowPtr), (ci, self.ColIdx), (va, self.Val)):
            if dst.nbytes and L.spmv_b200_memcpy(dst.ctypes.data, src, dst.nbytes, 1) != 0:
                raise RuntimeError(last_error())
        return CSR(self.m, self.n, rp, ci, va, self.name)

    def destroy(self):
        if self.c is not None:
            lib().spmv_b200_csr_free(C.byref(self.c))
            self.c = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def _gen(fn, name, *args) -> DeviceMatrix:
    c = DeviceCSR()
    if fn(*args, C.byref(c)) != 0:
        raise RuntimeError(f"{name}: {last_error()}")
    return DeviceMatrix(c, name)


def gen_laplacian2d(nx, ny=None, size=8):
    ny = nx if ny is None else ny
    return _gen(lib().spmv_b200_gen_laplacian2d, f"laplacian2d_{nx}x{ny}", nx, ny, size)


def gen_stencil27(nx, ny=None, nz=None, size=8):
    ny = nx if ny is None else ny
    nz = nx if nz is None else nz
    return _gen(lib().spmv_b200_gen_stencil27, f"stencil27_{nx}x{ny}x{nz}", nx, ny, nz, size)


def gen_uniform(m, n, k, seed, row0=0, eighths=False, size=8):
    return _gen(lib().spmv_b200_gen_uniform, f"uniform_{m}x{n}_k{k}", m, n, k, seed, row0, int(eighths), size)


def gen_rmat(scale, edge_factor, seed, size=4):
    return _gen(lib().spmv_b200_gen_rmat, f"rmat_s{scale}_ef{edge_factor}", scale, edge_factor, seed, size)


def gen_x(dst, n, seed, ones=False, size=8):
    if lib().spmv_b200_gen_x(_addr(dst), n, seed, int(ones), size) != 0:
        raise RuntimeError(last_error())
