"""Python mirror of the C interface of libxsmm_b200.so (ctypes; no torch, no CPU compute path).

Every function below has the name, argument order and meaning of the reference's C entry point
(reference include/libxsmm_spmdm.h:74-132, include/libxsmm_fsspmdm.h:41-57) or of one of the
stream-ordered additions declared in include/libxsmm_b200.h.  The functions only marshal arguments;
all arithmetic happens in the CUDA kernels inside the shared library.  If the library is missing,
``load()`` raises -- there is no fallback of any kind.

Small conveniences on top (``DeviceBuffer``, ``Spmdm``, ``Fsspmdm``) keep the tests and bench.py short;
they still go through the C ABI for every operation.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "lib", "libxsmm_b200.so")

LIBXSMM_SPMDM_DATATYPE_F32 = 0
LIBXSMM_SPMDM_DATATYPE_BFLOAT16 = 1

# every symbol include/*.h declares (tests check that the library exports all of them)
REFERENCE_SYMBOLS = [
    "libxsmm_spmdm_init", "libxsmm_spmdm_destroy",
    "libxsmm_spmdm_get_num_createSparseSlice_blocks", "libxsmm_spmdm_get_num_compute_blocks",
    "libxsmm_spmdm_createSparseSlice_fp32_thread", "libxsmm_spmdm_createSparseSlice_bfloat16_thread",
    "libxsmm_spmdm_compute_fp32_thread", "libxsmm_spmdm_compute_bfloat16_thread",
    "libxsmm_dfsspmdm_create", "libxsmm_dfsspmdm_execute", "libxsmm_dfsspmdm_destroy",
    "libxsmm_sfsspmdm_create", "libxsmm_sfsspmdm_execute", "libxsmm_sfsspmdm_destroy",
]
ADDED_SYMBOLS = [
    "libxsmm_spmdm_createSparseSlice_fp32_stream", "libxsmm_spmdm_createSparseSlice_bfloat16_stream",
    "libxsmm_spmdm_createSparseSlice_csr_fp32_stream", "libxsmm_spmdm_createSparseSlice_csr_bfloat16_stream",
    "libxsmm_spmdm_createSparseSlice_csc_fp32_stream", "libxsmm_spmdm_createSparseSlice_csc_bfloat16_stream",
    "libxsmm_spmdm_compute_fp32_stream", "libxsmm_spmdm_compute_bfloat16_stream",
    "libxsmm_spmdm_exec_host", "libxsmm_spmdm_exec_stream",
    "libxsmm_dfsspmdm_execute_stream", "libxsmm_sfsspmdm_execute_stream",
    "libxsmm_dfsspmdm_is_sparse", "libxsmm_sfsspmdm_is_sparse",
    "libxsmm_dfsspmdm_is_baked", "libxsmm_sfsspmdm_is_baked", "libxsmm_sfsspmdm_is_tensor_core",
    "libxsmm_b200_last_error", "libxsmm_b200_last_error_string", "libxsmm_b200_clear_error",
    "libxsmm_b200_launch_count", "libxsmm_b200_last_compute_kernel",
    "libxsmm_b200_host_alloc", "libxsmm_b200_host_free",
    "libxsmm_b200_device_alloc", "libxsmm_b200_device_free",
    "libxsmm_b200_memcpy_h2d", "libxsmm_b200_memcpy_d2h", "libxsmm_b200_memset",
    "libxsmm_b200_synchronize", "libxsmm_b200_device_count", "libxsmm_b200_set_device",
    "libxsmm_b200_stream_create", "libxsmm_b200_stream_destroy", "libxsmm_b200_stream_synchronize",
    "libxsmm_b200_event_create", "libxsmm_b200_event_destroy", "libxsmm_b200_event_record",
    "libxsmm_b200_event_synchronize", "libxsmm_b200_event_elapsed_ms",
    "libxsmm_b200_memcpy_h2d_async", "libxsmm_b200_memcpy_d2h_async", "libxsmm_b200_memset_async",
    "libxsmm_b200_spmdm_geometry", "libxsmm_b200_fsspmdm_plan", "libxsmm_b200_fsspmdm_kernel_source",
    "libxsmm_b200_free_string",
    "libxsmm_b200_graph_begin", "libxsmm_b200_graph_end", "libxsmm_b200_graph_launch", "libxsmm_b200_graph_destroy",
    "libxsmm_b200_sparse_matmul", "libxsmm_b200_sparse_matmul_cache_entries", "libxsmm_b200_sparse_matmul_cache_clear",
    "libxsmm_b200_csr_read_mtx", "libxsmm_b200_csr_free", "libxsmm_b200_dfsspmdm_create_mtx", "libxsmm_b200_sfsspmdm_create_mtx",
    "libxsmm_b200_dcsr_soa_create", "libxsmm_b200_scsr_soa_create", "libxsmm_b200_csr_soa_execute", "libxsmm_b200_csr_soa_is_baked",
    "libxsmm_b200_csr_soa_destroy", "libxsmm_b200_dcsc_soa_create", "libxsmm_b200_scsc_soa_create",
    "libxsmm_b200_dmmdispatch", "libxsmm_b200_smmdispatch", "libxsmm_b200_mm_execute", "libxsmm_b200_mm_kernel", "libxsmm_b200_mm_release",
    "libxsmm_b200_drm_ac_soa_create", "libxsmm_b200_srm_ac_soa_create", "libxsmm_b200_drm_bc_soa_create", "libxsmm_b200_srm_bc_soa_create",
    "libxsmm_b200_rm_soa_execute", "libxsmm_b200_rm_soa_destroy",
    "libxsmm_b200_csr_soa_execute_indexed", "libxsmm_b200_rm_soa_execute_indexed",
    "libxsmm_b200_sp24_create_bfloat16", "libxsmm_b200_sp24_execute", "libxsmm_b200_sp24_destroy",
    "libxsmm_b200_sp24_create_fp8", "libxsmm_b200_sp24_execute_fp8",
    "libxsmm_b200_sp24_execute_bf16out", "libxsmm_b200_sp24_execute_fp8_bf16out",
]


class libxsmm_spmdm_handle(ctypes.Structure):
    """reference include/libxsmm_spmdm.h:42-60 (same field order; caller-owned storage)."""
    _fields_ = [("m", ctypes.c_int), ("n", ctypes.c_int), ("k", ctypes.c_int),
                ("bm", ctypes.c_int), ("bn", ctypes.c_int), ("bk", ctypes.c_int),
                ("mb", ctypes.c_int), ("nb", ctypes.c_int), ("kb", ctypes.c_int),
                ("datatype", ctypes.c_int),
                ("base_ptr_scratch_A", ctypes.c_void_p),
                ("base_ptr_scratch_B_scratch_C", ctypes.c_void_p),
                ("memory_for_scratch_per_thread", ctypes.c_int)]


class libxsmm_CSR_sparseslice(ctypes.Structure):
    """reference include/libxsmm_spmdm.h:66-71; the three pointers are DEVICE pointers."""
    _fields_ = [("rowidx", ctypes.c_void_p), ("colidx", ctypes.c_void_p), ("values", ctypes.c_void_p)]


_lib = None


def load():
    """dlopen the product library.  Raises if it has not been built (python libxsmm-1_b200/build.py)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError("libxsmm_b200.so is not built (%s): run `python libxsmm-1_b200/build.py`; "
                           "there is no CPU fallback" % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, ci, cc = ctypes.c_void_p, ctypes.c_int, ctypes.c_char
    H = ctypes.POINTER(libxsmm_spmdm_handle)
    S = ctypes.POINTER(libxsmm_CSR_sparseslice)
    L.libxsmm_spmdm_init.argtypes = [ci, ci, ci, ci, H, ctypes.POINTER(S)]
    L.libxsmm_spmdm_init.restype = None
    L.libxsmm_spmdm_destroy.argtypes = [H]
    L.libxsmm_spmdm_destroy.restype = None
    L.libxsmm_spmdm_get_num_createSparseSlice_blocks.argtypes = [H]
    L.libxsmm_spmdm_get_num_compute_blocks.argtypes = [H]
    for nm in ("fp32", "bfloat16"):
        f = getattr(L, "libxsmm_spmdm_createSparseSlice_%s_thread" % nm)
        f.argtypes = [H, cc, vp, S, ci, ci, ci]
        f.restype = None
        f = getattr(L, "libxsmm_spmdm_compute_%s_thread" % nm)
        f.argtypes = [H, cc, cc, vp, S, vp, cc, vp, vp, ci, ci, ci]
        f.restype = None
        f = getattr(L, "libxsmm_spmdm_createSparseSlice_%s_stream" % nm)
        f.argtypes = [H, cc, vp, S, vp]
        f.restype = None
        f = getattr(L, "libxsmm_spmdm_compute_%s_stream" % nm)
        f.argtypes = [H, cc, cc, vp, S, vp, cc, vp, vp, vp]
        f.restype = None
        for form in ("csr", "csc"):
            f = getattr(L, "libxsmm_spmdm_createSparseSlice_%s_%s_stream" % (form, nm))
            f.argtypes = [H, vp, vp, vp, ctypes.c_longlong, S, vp]
            f.restype = None
    L.libxsmm_spmdm_exec_host.argtypes = [H, S, ci, cc, cc, cc, vp, vp, vp, vp]
    L.libxsmm_spmdm_exec_host.restype = None
    L.libxsmm_spmdm_exec_stream.argtypes = [H, S, ci, cc, cc, cc, vp, vp, vp, vp, vp]
    L.libxsmm_spmdm_exec_stream.restype = None
    L.libxsmm_dfsspmdm_create.argtypes = [ci] * 6 + [ctypes.c_double, ctypes.c_double, vp]
    L.libxsmm_dfsspmdm_create.restype = vp
    L.libxsmm_sfsspmdm_create.argtypes = [ci] * 6 + [ctypes.c_float, ctypes.c_float, vp]
    L.libxsmm_sfsspmdm_create.restype = vp
    for p in ("d", "s"):
        f = getattr(L, "libxsmm_%sfsspmdm_execute" % p)
        f.argtypes = [vp, vp, vp]
        f.restype = None
        f = getattr(L, "libxsmm_%sfsspmdm_execute_stream" % p)
        f.argtypes = [vp, vp, vp, vp]
        f.restype = None
        f = getattr(L, "libxsmm_%sfsspmdm_destroy" % p)
        f.argtypes = [vp]
        f.restype = None
        getattr(L, "libxsmm_%sfsspmdm_is_sparse" % p).argtypes = [vp]
        getattr(L, "libxsmm_%sfsspmdm_is_baked" % p).argtypes = [vp]
    L.libxsmm_sfsspmdm_is_tensor_core.argtypes = [vp]
    L.libxsmm_b200_last_error_string.restype = ctypes.c_char_p
    L.libxsmm_b200_launch_count.restype = ctypes.c_ulonglong
    L.libxsmm_b200_last_compute_kernel.restype = ctypes.c_char_p
    L.libxsmm_b200_host_alloc.argtypes = [ctypes.c_size_t]
    L.libxsmm_b200_host_alloc.restype = vp
    L.libxsmm_b200_host_free.argtypes = [vp]
    L.libxsmm_b200_device_alloc.argtypes = [ctypes.c_size_t]
    L.libxsmm_b200_device_alloc.restype = vp
    L.libxsmm_b200_device_free.argtypes = [vp]
    L.libxsmm_b200_memcpy_h2d.argtypes = [vp, vp, ctypes.c_size_t]
    L.libxsmm_b200_memcpy_d2h.argtypes = [vp, vp, ctypes.c_size_t]
    L.libxsmm_b200_memset.argtypes = [vp, ci, ctypes.c_size_t]
    L.libxsmm_b200_set_device.argtypes = [ci]
    L.libxsmm_b200_stream_create.restype = vp
    L.libxsmm_b200_stream_destroy.argtypes = [vp]
    L.libxsmm_b200_stream_synchronize.argtypes = [vp]
    L.libxsmm_b200_event_create.restype = vp
    L.libxsmm_b200_event_destroy.argtypes = [vp]
    L.libxsmm_b200_event_record.argtypes = [vp, vp]
    L.libxsmm_b200_event_synchronize.argtypes = [vp]
    L.libxsmm_b200_event_elapsed_ms.argtypes = [vp, vp]
    L.libxsmm_b200_event_elapsed_ms.restype = ctypes.c_float
    L.libxsmm_b200_memcpy_h2d_async.argtypes = [vp, vp, ctypes.c_size_t, vp]
    L.libxsmm_b200_memcpy_d2h_async.argtypes = [vp, vp, ctypes.c_size_t, vp]
    L.libxsmm_b200_memset_async.argtypes = [vp, ci, ctypes.c_size_t, vp]
    L.libxsmm_b200_graph_begin.argtypes = [vp]
    L.libxsmm_b200_graph_end.argtypes = [vp]
    L.libxsmm_b200_graph_end.restype = vp
    L.libxsmm_b200_graph_launch.argtypes = [vp, vp]
    L.libxsmm_b200_graph_destroy.argtypes = [vp]
    L.libxsmm_b200_spmdm_geometry.argtypes = [ci] * 5 + [vp]
    L.libxsmm_b200_fsspmdm_plan.argtypes = [ci] * 7 + [ctypes.c_double, vp, vp]
    L.libxsmm_b200_fsspmdm_kernel_source.argtypes = [ci] * 7 + [ctypes.c_double, vp]
    L.libxsmm_b200_fsspmdm_kernel_source.restype = vp
    L.libxsmm_b200_free_string.argtypes = [vp]
    _lib = L
    return L


def device_count():
    return int(load().libxsmm_b200_device_count())


def require_gpu():
    if device_count() < 1:
        raise RuntimeError("libxsmm_b200: no CUDA device visible; this library has no CPU path")


def last_error():
    L = load()
    return int(L.libxsmm_b200_last_error()), (L.libxsmm_b200_last_error_string() or b"").decode()


def clear_error():
    load().libxsmm_b200_clear_error()


def check():
    code, msg = last_error()
    if code != 0:
        clear_error()
        raise RuntimeError("libxsmm_b200 error %d: %s" % (code, msg))


def launch_count():
    return int(load().libxsmm_b200_launch_count())


def last_compute_kernel():
    return load().libxsmm_b200_last_compute_kernel().decode()


def synchronize():
    load().libxsmm_b200_synchronize()
    check()


def _addr(x):
    """numpy array -> host address; DeviceBuffer/HostBuffer -> its address; int passes through."""
    if x is None:
        return None
    if isinstance(x, (DeviceBuffer, HostBuffer)):
        return x.ptr
    if isinstance(x, np.ndarray):
        assert x.flags.c_contiguous
        return x.ctypes.data
    return int(x)


class DeviceBuffer:
    """cudaMalloc'ed bytes obtained through the C ABI (libxsmm_b200_device_alloc)."""

    def __init__(self, nbytes):
        self.nbytes = int(nbytes)
        self.ptr = load().libxsmm_b200_device_alloc(self.nbytes)
        if not self.ptr:
            check()
            raise MemoryError("device_alloc(%d)" % self.nbytes)

    @classmethod
    def from_numpy(cls, a):
        a = np.ascontiguousarray(a)
        d = cls(max(a.nbytes, 1))
        if a.nbytes:
            load().libxsmm_b200_memcpy_h2d(d.ptr, a.ctypes.data, a.nbytes)
        check()
        return d

    def upload(self, a, offset=0):
        a = np.ascontiguousarray(a)
        assert offset + a.nbytes <= self.nbytes
        load().libxsmm_b200_memcpy_h2d(self.ptr + offset, a.ctypes.data, a.nbytes)
        check()

    def to_numpy(self, dtype, shape, offset=0):
        out = np.empty(shape, dtype)
        assert offset + out.nbytes <= self.nbytes
        if out.nbytes:
            load().libxsmm_b200_memcpy_d2h(out.ctypes.data, self.ptr + offset, out.nbytes)
        check()
        return out

    def fill(self, byte):
        load().libxsmm_b200_memset(self.ptr, int(byte), self.nbytes)

    def free(self):
        if self.ptr:
            load().libxsmm_b200_device_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class HostBuffer:
    """Page-locked host memory (libxsmm_b200_host_alloc) viewed as a numpy array."""

    def __init__(self, shape, dtype):
        self.shape = tuple(int(s) for s in np.atleast_1d(shape))
        self.dtype = np.dtype(dtype)
        self.nbytes = int(np.prod(self.shape)) * self.dtype.itemsize
        self.ptr = load().libxsmm_b200_host_alloc(max(self.nbytes, 1))
        if not self.ptr:
            check()
            raise MemoryError("host_alloc(%d)" % self.nbytes)
        buf = (ctypes.c_char * self.nbytes).from_address(self.ptr)
        self.array = np.frombuffer(buf, dtype=self.dtype).reshape(self.shape)

    def free(self):
        if self.ptr:
            self.array = None
            load().libxsmm_b200_host_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Stream:
    def __init__(self):
        self.ptr = load().libxsmm_b200_stream_create()
        check()

    def synchronize(self):
        load().libxsmm_b200_stream_synchronize(self.ptr)
        check()

    def destroy(self):
        if self.ptr:
            load().libxsmm_b200_stream_destroy(self.ptr)
            self.ptr = None


class Event:
    def __init__(self):
        self.ptr = load().libxsmm_b200_event_create()
        check()

    def record(self, stream):
        load().libxsmm_b200_event_record(self.ptr, stream.ptr if isinstance(stream, Stream) else stream)

    def synchronize(self):
        load().libxsmm_b200_event_synchronize(self.ptr)

    def elapsed_ms(self, later):
        return float(load().libxsmm_b200_event_elapsed_ms(self.ptr, later.ptr))

    def destroy(self):
        if self.ptr:
            load().libxsmm_b200_event_destroy(self.ptr)
            self.ptr = None


def _c(ch):
    return ch.encode() if isinstance(ch, str) else ch


def _sptr(stream):
    return stream.ptr if isinstance(stream, Stream) else stream


# ======================================================================================================
# SPMDM -- same names and argument order as reference include/libxsmm_spmdm.h:74-132
# ======================================================================================================
def libxsmm_spmdm_init(M, N, K, max_threads):
    """-> (handle, slices).  handle is caller storage filled by the library; slices points INTO the
    library-owned arena (reference src/libxsmm_spmdm.c:540-627)."""
    L = load()
    h = libxsmm_spmdm_handle()
    s = ctypes.POINTER(libxsmm_CSR_sparseslice)()
    L.libxsmm_spmdm_init(M, N, K, max_threads, ctypes.byref(h), ctypes.byref(s))
    return h, s


def libxsmm_spmdm_destroy(handle):
    load().libxsmm_spmdm_destroy(ctypes.byref(handle))


def libxsmm_spmdm_get_num_createSparseSlice_blocks(handle):
    return int(load().libxsmm_spmdm_get_num_createSparseSlice_blocks(ctypes.byref(handle)))


def libxsmm_spmdm_get_num_compute_blocks(handle):
    return int(load().libxsmm_spmdm_get_num_compute_blocks(ctypes.byref(handle)))


def libxsmm_spmdm_createSparseSlice_fp32_thread(handle, transa, a, slices, block_id, tid, nthreads):
    load().libxsmm_spmdm_createSparseSlice_fp32_thread(ctypes.byref(handle), _c(transa), _addr(a), slices, block_id, tid, nthreads)


def libxsmm_spmdm_createSparseSlice_bfloat16_thread(handle, transa, a, slices, block_id, tid, nthreads):
    load().libxsmm_spmdm_createSparseSlice_bfloat16_thread(ctypes.byref(handle), _c(transa), _addr(a), slices, block_id, tid, nthreads)


def libxsmm_spmdm_compute_fp32_thread(handle, transa, transb, alpha, slices, b, transc, beta, c, block_id, tid, nthreads):
    al = ctypes.c_float(alpha)
    be = ctypes.c_float(beta)
    load().libxsmm_spmdm_compute_fp32_thread(ctypes.byref(handle), _c(transa), _c(transb), ctypes.addressof(al), slices,
                                             _addr(b), _c(transc), ctypes.addressof(be), _addr(c), block_id, tid, nthreads)


def libxsmm_spmdm_compute_bfloat16_thread(handle, transa, transb, alpha_bits, slices, b, transc, beta_bits, c, block_id, tid, nthreads):
    """alpha_bits / beta_bits are raw 16-bit patterns, read by the library the way the reference reads
    them (as integers; reference bf16 compute template :91,113,164)."""
    al = ctypes.c_ushort(alpha_bits)
    be = ctypes.c_ushort(beta_bits)
    load().libxsmm_spmdm_compute_bfloat16_thread(ctypes.byref(handle), _c(transa), _c(transb), ctypes.addressof(al), slices,
                                                 _addr(b), _c(transc), ctypes.addressof(be), _addr(c), block_id, tid, nthreads)


# stream-ordered additions (include/libxsmm_b200.h)
def libxsmm_spmdm_createSparseSlice_fp32_stream(handle, transa, d_a, slices, stream=None):
    load().libxsmm_spmdm_createSparseSlice_fp32_stream(ctypes.byref(handle), _c(transa), _addr(d_a), slices, _sptr(stream))


def libxsmm_spmdm_createSparseSlice_bfloat16_stream(handle, transa, d_a, slices, stream=None):
    load().libxsmm_spmdm_createSparseSlice_bfloat16_stream(ctypes.byref(handle), _c(transa), _addr(d_a), slices, _sptr(stream))


def libxsmm_spmdm_createSparseSlice_csr_fp32_stream(handle, d_row_ptr, d_col_idx, d_values, nnz, slices, stream=None):
    load().libxsmm_spmdm_createSparseSlice_csr_fp32_stream(ctypes.byref(handle), _addr(d_row_ptr), _addr(d_col_idx), _addr(d_values),
                                                           int(nnz), slices, _sptr(stream))


def libxsmm_spmdm_createSparseSlice_csr_bfloat16_stream(handle, d_row_ptr, d_col_idx, d_values, nnz, slices, stream=None):
    load().libxsmm_spmdm_createSparseSlice_csr_bfloat16_stream(ctypes.byref(handle), _addr(d_row_ptr), _addr(d_col_idx), _addr(d_values),
                                                               int(nnz), slices, _sptr(stream))


def libxsmm_spmdm_createSparseSlice_csc_fp32_stream(handle, d_col_ptr, d_row_idx, d_values, nnz, slices, stream=None):
    load().libxsmm_spmdm_createSparseSlice_csc_fp32_stream(ctypes.byref(handle), _addr(d_col_ptr), _addr(d_row_idx), _addr(d_values),
                                                           int(nnz), slices, _sptr(stream))


def libxsmm_spmdm_createSparseSlice_csc_bfloat16_stream(handle, d_col_ptr, d_row_idx, d_values, nnz, slices, stream=None):
    load().libxsmm_spmdm_createSparseSlice_csc_bfloat16_stream(ctypes.byref(handle), _addr(d_col_ptr), _addr(d_row_idx), _addr(d_values),
                                                               int(nnz), slices, _sptr(stream))


def libxsmm_spmdm_compute_fp32_stream(handle, transa, transb, alpha, slices, d_b, transc, beta, d_c, stream=None):
    al = ctypes.c_float(alpha)
    be = ctypes.c_float(beta)
    load().libxsmm_spmdm_compute_fp32_stream(ctypes.byref(handle), _c(transa), _c(transb), ctypes.addressof(al), slices,
                                             _addr(d_b), _c(transc), ctypes.addressof(be), _addr(d_c), _sptr(stream))


def libxsmm_spmdm_compute_bfloat16_stream(handle, transa, transb, alpha_bits, slices, d_b, transc, beta_bits, d_c, stream=None):
    al = ctypes.c_ushort(alpha_bits)
    be = ctypes.c_ushort(beta_bits)
    load().libxsmm_spmdm_compute_bfloat16_stream(ctypes.byref(handle), _c(transa), _c(transb), ctypes.addressof(al), slices,
                                                 _addr(d_b), _c(transc), ctypes.addressof(be), _addr(d_c), _sptr(stream))


def _beta_box(datatype, beta):
    return ctypes.c_ushort(int(beta)) if datatype == LIBXSMM_SPMDM_DATATYPE_BFLOAT16 else ctypes.c_float(beta)


def libxsmm_spmdm_exec_host(handle, slices, datatype, transa, transb, transc, a, b, beta, c):
    """One whole multiply on HOST matrices (what one repetition of samples/spmdm/spmdm.c:88-111 does)."""
    be = _beta_box(datatype, beta)
    load().libxsmm_spmdm_exec_host(ctypes.byref(handle), slices, datatype, _c(transa), _c(transb), _c(transc),
                                   _addr(a), _addr(b), ctypes.addressof(be), _addr(c))


def libxsmm_spmdm_exec_stream(handle, slices, datatype, transa, transb, transc, d_a, d_b, beta, d_c, stream=None):
    """Slice creation followed by compute, both asynchronous on ``stream``, DEVICE matrices."""
    be = _beta_box(datatype, beta)
    load().libxsmm_spmdm_exec_stream(ctypes.byref(handle), slices, datatype, _c(transa), _c(transb), _c(transc),
                                     _addr(d_a), _addr(d_b), ctypes.addressof(be), _addr(d_c), _sptr(stream))


def libxsmm_b200_sparse_matmul(datatype, transa, transb, transc, M, N, K, max_threads, d_a, d_b, beta, d_c, stream=None):
    """Fused caller step (handle cache + slice creation + compute in one stream-ordered call); returns the error code."""
    be = _beta_box(datatype, beta)
    L = load()
    L.libxsmm_b200_sparse_matmul.restype = ctypes.c_int
    L.libxsmm_b200_sparse_matmul.argtypes = [ctypes.c_int, ctypes.c_char, ctypes.c_char, ctypes.c_char, ctypes.c_int, ctypes.c_int, ctypes.c_int,
                                             ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p]
    return int(L.libxsmm_b200_sparse_matmul(datatype, _c(transa), _c(transb), _c(transc), M, N, K, max_threads,
                                            _addr(d_a), _addr(d_b), ctypes.addressof(be), _addr(d_c), _sptr(stream)))


def sparse_matmul_cache_entries():
    return int(load().libxsmm_b200_sparse_matmul_cache_entries())


def sparse_matmul_cache_clear():
    load().libxsmm_b200_sparse_matmul_cache_clear()


def csr_read_mtx(path):
    """MatrixMarket coordinate file -> (row_ptr, col_idx, values, rows, cols) through the library's reader (host only).
    Raises ValueError with the library's message on a malformed file."""
    L = load()
    rp, ci, va = ctypes.POINTER(ctypes.c_uint)(), ctypes.POINTER(ctypes.c_uint)(), ctypes.POINTER(ctypes.c_double)()
    nr, nc, ne = ctypes.c_uint(0), ctypes.c_uint(0), ctypes.c_uint(0)
    L.libxsmm_b200_csr_read_mtx.restype = ctypes.c_int
    rc = L.libxsmm_b200_csr_read_mtx(os.fsencode(path), ctypes.byref(rp), ctypes.byref(ci), ctypes.byref(va),
                                     ctypes.byref(nr), ctypes.byref(nc), ctypes.byref(ne))
    if 0 != rc:
        code, msg = last_error()
        clear_error()
        raise ValueError("csr_read_mtx failed (%d): %s" % (rc, msg))
    try:
        row_ptr = np.ctypeslib.as_array(rp, shape=(nr.value + 1,)).copy()
        col_idx = np.ctypeslib.as_array(ci, shape=(ne.value,)).copy()
        values = np.ctypeslib.as_array(va, shape=(ne.value,)).copy()
    finally:
        L.libxsmm_b200_csr_free.restype = None
        L.libxsmm_b200_csr_free(rp, ci, va)
    return row_ptr, col_idx, values, int(nr.value), int(nc.value)


# ======================================================================================================
# FSSPMDM -- reference include/libxsmm_fsspmdm.h:41-57
# ======================================================================================================
def libxsmm_dfsspmdm_create(M, N, K, lda, ldb, ldc, alpha, beta, a_dense):
    a = np.ascontiguousarray(a_dense, np.float64)
    return load().libxsmm_dfsspmdm_create(M, N, K, lda, ldb, ldc, float(alpha), float(beta), a.ctypes.data)


def libxsmm_sfsspmdm_create(M, N, K, lda, ldb, ldc, alpha, beta, a_dense):
    a = np.ascontiguousarray(a_dense, np.float32)
    return load().libxsmm_sfsspmdm_create(M, N, K, lda, ldb, ldc, float(alpha), float(beta), a.ctypes.data)


def libxsmm_dfsspmdm_execute(handle, B, C):
    load().libxsmm_dfsspmdm_execute(handle, _addr(B), _addr(C))


def libxsmm_sfsspmdm_execute(handle, B, C):
    load().libxsmm_sfsspmdm_execute(handle, _addr(B), _addr(C))


def libxsmm_dfsspmdm_execute_stream(handle, d_B, d_C, stream=None):
    load().libxsmm_dfsspmdm_execute_stream(handle, _addr(d_B), _addr(d_C), _sptr(stream))


def libxsmm_sfsspmdm_execute_stream(handle, d_B, d_C, stream=None):
    load().libxsmm_sfsspmdm_execute_stream(handle, _addr(d_B), _addr(d_C), _sptr(stream))


def libxsmm_dfsspmdm_destroy(handle):
    load().libxsmm_dfsspmdm_destroy(handle)


def libxsmm_sfsspmdm_destroy(handle):
    load().libxsmm_sfsspmdm_destroy(handle)


# ======================================================================================================
# conveniences used by tests and bench.py
# ======================================================================================================
class Spmdm:
    """One spmdm problem: handle + slices, with helpers to read the slice arena back in the flat layout
    the oracle uses (slice s = kb*mb + mb owns rowidx[s, :bm+1], colidx[s, :bm*bk], values[s, :bm*bk])."""

    def __init__(self, M, N, K, max_threads=1):
        require_gpu()
        self.handle, self.slices = libxsmm_spmdm_init(M, N, K, max_threads)
        check()
        if not self.handle.base_ptr_scratch_A:
            raise RuntimeError("libxsmm_spmdm_init failed")

    @property
    def geometry(self):
        h = self.handle
        return dict(m=h.m, n=h.n, k=h.k, bm=h.bm, bn=h.bn, bk=h.bk, mb=h.mb, nb=h.nb, kb=h.kb)

    def create_slices(self, d_a, transa="N", bf16=False, stream=None):
        f = libxsmm_spmdm_createSparseSlice_bfloat16_stream if bf16 else libxsmm_spmdm_createSparseSlice_fp32_stream
        f(self.handle, transa, d_a, self.slices, stream)

    def create_slices_csr(self, d_row_ptr, d_col_idx, d_values, nnz, bf16=False, stream=None):
        """A in CSR form: device arrays row_ptr[M + 1], col_idx[nnz] (uint32, 0-based, ascending within a row) and values[nnz]
        (float32, or bf16 bit patterns as uint16); the same slices as create_slices() on the dense matrix (transa 'N')."""
        f = libxsmm_spmdm_createSparseSlice_csr_bfloat16_stream if bf16 else libxsmm_spmdm_createSparseSlice_csr_fp32_stream
        f(self.handle, d_row_ptr, d_col_idx, d_values, nnz, self.slices, stream)

    def create_slices_csc(self, d_col_ptr, d_row_idx, d_values, nnz, bf16=False, stream=None):
        """A in CSC form (equally: the CSR arrays of A stored K x M): device arrays col_ptr[K + 1], row_idx[nnz] (uint32, 0-based,
        ascending within a column) and values[nnz]; the same slices as create_slices() on the K x M array with transa 'T'."""
        f = libxsmm_spmdm_createSparseSlice_csc_bfloat16_stream if bf16 else libxsmm_spmdm_createSparseSlice_csc_fp32_stream
        f(self.handle, d_col_ptr, d_row_idx, d_values, nnz, self.slices, stream)

    def compute(self, d_b, d_c, transb="N", transc="N", beta=0.0, bf16=False, stream=None, transa="N"):
        if bf16:
            libxsmm_spmdm_compute_bfloat16_stream(self.handle, transa, transb, 0x3F80, self.slices, d_b, transc, int(beta), d_c, stream)
        else:
            libxsmm_spmdm_compute_fp32_stream(self.handle, transa, transb, 1.0, self.slices, d_b, transc, float(beta), d_c, stream)

    def read_slices(self):
        h = self.handle
        ns, cap = h.mb * h.kb, h.bm * h.bk
        L = load()
        L.libxsmm_b200_synchronize()
        ro = np.empty((ns, h.bm + 1), np.uint16)
        co = np.empty((ns, cap), np.uint16)
        va = np.empty((ns, cap), np.float32)
        # the table entries point into one arena with per-array strides; slice 0 is the base of each
        s0 = self.slices[0]
        L.libxsmm_b200_memcpy_d2h(ro.ctypes.data, s0.rowidx, ro.nbytes)
        L.libxsmm_b200_memcpy_d2h(co.ctypes.data, s0.colidx, co.nbytes)
        L.libxsmm_b200_memcpy_d2h(va.ctypes.data, s0.values, va.nbytes)
        check()
        return ro, co, va

    def destroy(self):
        if self.handle.base_ptr_scratch_A:
            libxsmm_spmdm_destroy(self.handle)


class Fsspmdm:
    """A fixed operator: create once, execute many times (reference src/libxsmm_fsspmdm.c)."""

    def __init__(self, a_dense, N, ldb=None, ldc=None, beta=0.0, alpha=1.0, lda=None):
        require_gpu()
        a = np.ascontiguousarray(a_dense)
        assert a.dtype in (np.float64, np.float32)
        self.double = a.dtype == np.float64
        self.M, self.K = a.shape
        self.N = N
        self.ldb = N if ldb is None else ldb
        self.ldc = N if ldc is None else ldc
        lda = self.K if lda is None else lda
        create = libxsmm_dfsspmdm_create if self.double else libxsmm_sfsspmdm_create
        self.handle = create(self.M, N, self.K, lda, self.ldb, self.ldc, alpha, beta, a)
        if not self.handle:
            code, msg = last_error()
            clear_error()
            raise ValueError("fsspmdm_create failed: %s" % msg)
        clear_error()   # a missing NVRTC is reported but not fatal (generic kernel)

    @classmethod
    def from_mtx(cls, path, N, ldb=None, ldc=None, beta=0.0, double=True):
        """the operator of a MatrixMarket file (libxsmm_b200_[sd]fsspmdm_create_mtx)."""
        require_gpu()
        L = load()
        self = cls.__new__(cls)
        self.double, self.N = bool(double), N
        self.ldb = N if ldb is None else ldb
        self.ldc = N if ldc is None else ldc
        m, k = ctypes.c_int(0), ctypes.c_int(0)
        f = L.libxsmm_b200_dfsspmdm_create_mtx if double else L.libxsmm_b200_sfsspmdm_create_mtx
        f.restype = ctypes.c_void_p
        f.argtypes = [ctypes.c_char_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double if double else ctypes.c_float,
                      ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int)]
        self.handle = f(os.fsencode(path), N, self.ldb, self.ldc, float(beta), ctypes.byref(m), ctypes.byref(k))
        if not self.handle:
            code, msg = last_error()
            clear_error()
            raise ValueError("fsspmdm_create_mtx failed: %s" % msg)
        clear_error()
        self.M, self.K = int(m.value), int(k.value)
        return self

    @property
    def is_sparse(self):
        L = load()
        return bool((L.libxsmm_dfsspmdm_is_sparse if self.double else L.libxsmm_sfsspmdm_is_sparse)(self.handle))

    @property
    def is_baked(self):
        L = load()
        return bool((L.libxsmm_dfsspmdm_is_baked if self.double else L.libxsmm_sfsspmdm_is_baked)(self.handle))

    @property
    def is_tensor_core(self):
        return (not self.double) and bool(load().libxsmm_sfsspmdm_is_tensor_core(self.handle))

    def execute(self, B, C):
        (libxsmm_dfsspmdm_execute if self.double else libxsmm_sfsspmdm_execute)(self.handle, B, C)

    def execute_stream(self, d_B, d_C, stream=None):
        (libxsmm_dfsspmdm_execute_stream if self.double else libxsmm_sfsspmdm_execute_stream)(self.handle, d_B, d_C, stream)

    def destroy(self):
        if self.handle:
            (libxsmm_dfsspmdm_destroy if self.double else libxsmm_sfsspmdm_destroy)(self.handle)
            self.handle = None


class MmDispatch:
    """libxsmm_b200_[sd]mmdispatch: column-major SMM handle used the way samples/pyfr/pyfr_gemm_rm.c:98-122 uses
    libxsmm_dmmdispatch (row-major operator applied to a panel with very many columns)."""

    def __init__(self, m, n, k, lda=None, ldb=None, ldc=None, alpha=None, beta=None, dtype=np.float64):
        require_gpu()
        L = load()
        self.double = np.dtype(dtype) == np.float64
        f = L.libxsmm_b200_dmmdispatch if self.double else L.libxsmm_b200_smmdispatch
        f.restype = ctypes.c_void_p
        f.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p] * 5
        sc = ctypes.c_double if self.double else ctypes.c_float
        box = lambda v, t: None if v is None else ctypes.cast(ctypes.pointer(t(v)), ctypes.c_void_p)   # noqa: E731
        self.handle = f(m, n, k, box(lda, ctypes.c_int), box(ldb, ctypes.c_int), box(ldc, ctypes.c_int), box(alpha, sc), box(beta, sc))
        if not self.handle:
            code, msg = last_error()
            clear_error()
            raise ValueError("mmdispatch failed: %s" % msg)

    def execute(self, d_a, b, d_c, m_total, stream=None):
        L = load()
        L.libxsmm_b200_mm_execute.restype = None
        L.libxsmm_b200_mm_execute.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_void_p]
        L.libxsmm_b200_mm_execute(self.handle, _addr(d_a), _addr(b), _addr(d_c), m_total, _sptr(stream))

    @property
    def kernel(self):
        L = load()
        L.libxsmm_b200_mm_kernel.restype = ctypes.c_char_p
        L.libxsmm_b200_mm_kernel.argtypes = [ctypes.c_void_p]
        return L.libxsmm_b200_mm_kernel(self.handle).decode()

    def release(self):
        if self.handle:
            L = load()
            L.libxsmm_b200_mm_release.argtypes = [ctypes.c_void_p]
            L.libxsmm_b200_mm_release(self.handle)
            self.handle = None


class CsrSoa:
    """CSR operand applied to [element][row][column][soa] tensors (libxsmm_b200_[sd]csr_soa_*; the batched GPU counterpart of
    libxsmm_create_xcsr_soa).  sparse="A": reference samples/edge/asparse_srsoa.c (the CSR matrix is M x K, the dense operand
    B is [K][ldb][soa]); sparse="B": samples/edge/bsparse_srsoa.c (the CSR matrix is K x N, the dense operand A is [M][lda][soa])."""

    def __init__(self, M, N, K, rowptr, colidx, values, soa_width, lda=None, ldb=None, ldc=None, beta=0.0, sparse="A", fmt="csr"):
        """fmt="csc" (sparse="B" only): rowptr / colidx are the column pointers / row indices of B (libxsmm_create_xcsc_soa,
        reference samples/edge/bsparse_scsoa.c)."""
        require_gpu()
        L = load()
        values = np.ascontiguousarray(values)
        assert values.dtype in (np.float64, np.float32) and sparse in ("A", "B") and fmt in ("csr", "csc") and (fmt == "csr" or sparse == "B")
        self.double = values.dtype == np.float64
        rowptr = np.ascontiguousarray(rowptr, np.uint32); colidx = np.ascontiguousarray(colidx, np.uint32)
        self.M, self.N, self.K, self.soa, self.sparse = M, N, K, soa_width, sparse
        self.lda = 0 if sparse == "A" else (K if lda is None else lda)
        self.ldb = 0 if sparse == "B" else (N if ldb is None else ldb)
        self.ldc = N if ldc is None else ldc
        if fmt == "csc":
            f = L.libxsmm_b200_dcsc_soa_create if self.double else L.libxsmm_b200_scsc_soa_create
            f.restype = ctypes.c_void_p
            f.argtypes = [ctypes.c_int] * 6 + [ctypes.c_double if self.double else ctypes.c_float] + [ctypes.c_void_p] * 3
            self.handle = f(M, N, K, self.lda, self.ldc, soa_width, float(beta), rowptr.ctypes.data, colidx.ctypes.data, values.ctypes.data)
        else:
            f = L.libxsmm_b200_dcsr_soa_create if self.double else L.libxsmm_b200_scsr_soa_create
            f.restype = ctypes.c_void_p
            f.argtypes = [ctypes.c_int] * 7 + [ctypes.c_double if self.double else ctypes.c_float] + [ctypes.c_void_p] * 3
            self.handle = f(M, N, K, self.lda, self.ldb, self.ldc, soa_width, float(beta), rowptr.ctypes.data, colidx.ctypes.data, values.ctypes.data)
        if not self.handle:
            code, msg = last_error()
            clear_error()
            raise ValueError("csr_soa_create failed: %s" % msg)
        clear_error()

    @property
    def is_baked(self):
        return bool(load().libxsmm_b200_csr_soa_is_baked(ctypes.c_void_p(self.handle)))

    def execute(self, d_X, d_C, n_elements, stride_x=None, stride_c=None, stream=None):
        L = load()
        L.libxsmm_b200_csr_soa_execute.restype = None
        L.libxsmm_b200_csr_soa_execute.argtypes = [ctypes.c_void_p, ctypes.c_void_p, ctypes.c_void_p, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_longlong, ctypes.c_void_p]
        dense = self.K * self.ldb if self.sparse == "A" else self.M * self.lda
        sx = dense * self.soa if stride_x is None else stride_x
        sc = self.M * self.ldc * self.soa if stride_c is None else stride_c
        L.libxsmm_b200_csr_soa_execute(self.handle, _addr(d_X), _addr(d_C), n_elements, sx, sc, _sptr(stream))

    def execute_indexed(self, d_X, d_C, n_elements, x_index=None, x_slots=0, c_index=None, c_slots=0, stride_x=None, stride_c=None, stream=None):
        """element e reads its dense operand at slot x_index[e] and writes its C at slot c_index[e] (DEVICE uint32 arrays; None:
        slot e); an element with a slot at or past x_slots / c_slots is skipped.  Strides as for execute()."""
        dense = self.K * self.ldb if self.sparse == "A" else self.M * self.lda
        sx = dense * self.soa if stride_x is None else stride_x
        sc = self.M * self.ldc * self.soa if stride_c is None else stride_c
        csr_soa_execute_indexed(self.handle, d_X, d_C, n_elements, sx, sc, x_index, x_slots, c_index, c_slots, stream)

    def destroy(self):
        if self.handle:
            L = load()
            L.libxsmm_b200_csr_soa_destroy.argtypes = [ctypes.c_void_p]
            L.libxsmm_b200_csr_soa_destroy(self.handle)
            self.handle = None


class RmSoa:
    """Dense operand applied to [element][row][column][soa] tensors (libxsmm_b200_[sd]rm_{ac,bc}_soa_*; the batched GPU counterpart of
    libxsmm_create_rm_ac_soa / libxsmm_create_rm_bc_soa).  form="ac": A [M][lda][soa] and C [M][ldc][soa] are SoA, b is K x N
    row-major; form="bc": B [K][ldb][soa] and C are SoA, a is M x K row-major.  Pitches default to the dense extents."""

    def __init__(self, form, M, N, K, soa, dtype, lda=None, ldb=None, ldc=None, beta=0.0):
        assert form in ("ac", "bc")
        self.double = np.dtype(dtype) == np.float64
        assert self.double or np.dtype(dtype) == np.float32
        self.form, self.M, self.N, self.K, self.soa = form, M, N, K, soa
        self.lda = K if lda is None else lda
        self.ldb = N if ldb is None else ldb
        self.ldc = N if ldc is None else ldc
        self.handle = rm_soa_create(form, self.double, M, N, K, self.lda, self.ldb, self.ldc, soa, beta)
        if not self.handle:
            code, msg = last_error()
            clear_error()
            raise ValueError("rm_soa_create failed (%d): %s" % (code, msg))

    @property
    def extents(self):
        """scalars of one element's (first operand, second operand, C) as they lie in memory"""
        a = ((self.M - 1) * self.lda + self.K) * (self.soa if self.form == "ac" else 1)
        b = ((self.K - 1) * self.ldb + self.N) * (self.soa if self.form == "bc" else 1)
        return a, b, ((self.M - 1) * self.ldc + self.N) * self.soa

    def execute(self, d_a, d_b, d_c, n_elements, stride_a=None, stride_b=None, stride_c=None, stream=None):
        """stride None: the dense extent of one element (M lda, K ldb or M ldc rows, times soa for an SoA operand)"""
        sa = self.M * self.lda * (self.soa if self.form == "ac" else 1) if stride_a is None else stride_a
        sb = self.K * self.ldb * (self.soa if self.form == "bc" else 1) if stride_b is None else stride_b
        sc = self.M * self.ldc * self.soa if stride_c is None else stride_c
        rm_soa_execute(self.handle, d_a, d_b, d_c, n_elements, sa, sb, sc, stream)

    def execute_indexed(self, d_a, d_b, d_c, n_elements, a_index=None, a_slots=0, b_index=None, b_slots=0, c_index=None, c_slots=0,
                        stride_a=None, stride_b=None, stride_c=None, stream=None):
        """element e reads a, b and writes C at slots a_index[e], b_index[e], c_index[e] (DEVICE uint32 arrays; None: slot e); an
        element with a slot at or past that operand's *_slots is skipped.  Strides as for execute()."""
        sa = self.M * self.lda * (self.soa if self.form == "ac" else 1) if stride_a is None else stride_a
        sb = self.K * self.ldb * (self.soa if self.form == "bc" else 1) if stride_b is None else stride_b
        sc = self.M * self.ldc * self.soa if stride_c is None else stride_c
        rm_soa_execute_indexed(self.handle, d_a, d_b, d_c, n_elements, sa, sb, sc, a_index, a_slots, b_index, b_slots, c_index, c_slots, stream)

    def destroy(self):
        if self.handle:
            rm_soa_destroy(self.handle)
            self.handle = None


def rm_soa_create(form, double, M, N, K, lda, ldb, ldc, soa, beta):
    """the raw create entry (host only): the handle or None"""
    L = load()
    f = getattr(L, "libxsmm_b200_%srm_%s_soa_create" % ("d" if double else "s", form))
    f.restype = ctypes.c_void_p
    f.argtypes = [ctypes.c_int] * 7 + [ctypes.c_double if double else ctypes.c_float]
    return f(M, N, K, lda, ldb, ldc, soa, float(beta))


def rm_soa_execute(handle, d_a, d_b, d_c, n_elements, stride_a, stride_b, stride_c, stream=None):
    L = load()
    L.libxsmm_b200_rm_soa_execute.restype = None
    L.libxsmm_b200_rm_soa_execute.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_longlong] * 4 + [ctypes.c_void_p]
    L.libxsmm_b200_rm_soa_execute(handle, _addr(d_a), _addr(d_b), _addr(d_c), n_elements, stride_a, stride_b, stride_c, _sptr(stream))


def rm_soa_execute_indexed(handle, d_a, d_b, d_c, n_elements, stride_a, stride_b, stride_c, a_index, a_slots, b_index, b_slots,
                           c_index, c_slots, stream=None):
    """the raw indexed entry: every pointer may be a DeviceBuffer, an address or None (checked by the library, error -84)"""
    L = load()
    f = L.libxsmm_b200_rm_soa_execute_indexed
    f.restype = None
    f.argtypes = [ctypes.c_void_p] * 4 + [ctypes.c_longlong] * 4 + [ctypes.c_void_p, ctypes.c_longlong] * 3 + [ctypes.c_void_p]
    f(handle, _addr(d_a), _addr(d_b), _addr(d_c), n_elements, stride_a, stride_b, stride_c,
      _addr(a_index), a_slots, _addr(b_index), b_slots, _addr(c_index), c_slots, _sptr(stream))


def csr_soa_execute_indexed(handle, d_X, d_C, n_elements, stride_x, stride_c, x_index, x_slots, c_index, c_slots, stream=None):
    """the raw indexed entry of a csr_soa handle (see rm_soa_execute_indexed)"""
    L = load()
    f = L.libxsmm_b200_csr_soa_execute_indexed
    f.restype = None
    f.argtypes = [ctypes.c_void_p] * 3 + [ctypes.c_longlong] * 3 + [ctypes.c_void_p, ctypes.c_longlong] * 2 + [ctypes.c_void_p]
    f(handle, _addr(d_X), _addr(d_C), n_elements, stride_x, stride_c, _addr(x_index), x_slots, _addr(c_index), c_slots, _sptr(stream))


def rm_soa_destroy(handle):
    L = load()
    L.libxsmm_b200_rm_soa_destroy.restype = None
    L.libxsmm_b200_rm_soa_destroy.argtypes = [ctypes.c_void_p]
    L.libxsmm_b200_rm_soa_destroy(handle)


FP8_FORMATS = {"e4m3": 0, "e5m2": 1}


def _fp8_format(x, fmt):
    """the library's format code (0 e4m3, 1 e5m2) of a torch float8 tensor, or of raw bytes given with fmt"""
    name = str(getattr(x, "dtype", ""))
    if name in ("torch.float8_e4m3fn", "torch.float8_e5m2"):
        code = 0 if name == "torch.float8_e4m3fn" else 1
        if fmt is not None and FP8_FORMATS.get(fmt) != code:
            raise ValueError("fmt=%r does not match the tensor's %s" % (fmt, name))
        return code
    if fmt not in FP8_FORMATS:
        raise ValueError("raw FP8 bytes need fmt='e4m3' or 'e5m2', got %r" % (fmt,))
    return FP8_FORMATS[fmt]


def _c_is_bf16(d_c, c_dtype):
    """True for bf16 C: a torch bfloat16 d_c, or c_dtype="bf16" for other buffers (default fp32)"""
    if c_dtype not in (None, "bf16", "fp32"):
        raise ValueError("c_dtype must be 'bf16' or 'fp32', got %r" % (c_dtype,))
    name = str(getattr(d_c, "dtype", ""))
    if name in ("torch.bfloat16", "torch.float32"):
        tensor_bf16 = name == "torch.bfloat16"
        if c_dtype is not None and (c_dtype == "bf16") != tensor_bf16:
            raise ValueError("c_dtype=%r does not match d_c's %s" % (c_dtype, name))
        return tensor_bf16
    return c_dtype == "bf16"


def _check_bias(bias, M):
    """a torch bias must hold M bf16 values; device buffers and addresses are the caller's responsibility"""
    if hasattr(bias, "dtype") and hasattr(bias, "numel"):
        if str(bias.dtype) != "torch.bfloat16" or bias.numel() != M or not bias.is_contiguous():
            raise ValueError("bias must be a contiguous bfloat16 tensor of M=%d elements, got %s of %d" % (M, bias.dtype, bias.numel()))


class Sp24:
    """A fixed 2:4-sparse operator (libxsmm_b200_sp24_*): every aligned group of four along k keeps at most two ordered
    nonzeros.  a: M x K, rows with unit stride, host or CUDA --
      bf16: a torch bfloat16 tensor or a numpy uint16 array of bf16 bit patterns;
      FP8:  a torch float8_e4m3fn / float8_e5m2 tensor, or a numpy uint8 array of FP8 bytes with fmt="e4m3" | "e5m2".
    lda defaults to a's row stride.  Create compresses A on the GPU once; a matrix that is not 2:4 raises ValueError naming
    the first offending row and group."""
    fp8, format = False, None       # FP8 operators set both in __init__

    def __init__(self, a, lda=None, fmt=None):
        if hasattr(a, "data_ptr"):
            assert a.dim() == 2 and a.stride(1) == 1
            esize = a.element_size()
            self.M, self.K = int(a.shape[0]), int(a.shape[1])
            self.lda = int(a.stride(0)) if lda is None else lda
            ptr = a.data_ptr()
        else:
            assert isinstance(a, np.ndarray) and a.dtype in (np.uint16, np.uint8) and a.ndim == 2 and a.strides[1] == a.itemsize
            esize = a.itemsize
            self.M, self.K = a.shape
            self.lda = a.strides[0] // esize if lda is None else lda
            ptr = a.ctypes.data
        self.fp8 = esize == 1
        assert esize in (1, 2)
        if self.fp8:
            self.format = _fp8_format(a, fmt)
            self.handle = sp24_create_fp8(self.M, self.K, self.lda, ptr, self.format)
        else:
            assert fmt is None, "fmt names an FP8 format; a holds bf16"
            self.format = None
            self.handle = sp24_create_bfloat16(self.M, self.K, self.lda, ptr)
        if not self.handle:
            code, msg = last_error()
            clear_error()
            raise ValueError("%s failed (%d): %s" % ("sp24_create_fp8" if self.fp8 else "sp24_create_bfloat16", code, msg))

    def execute(self, d_b, d_c, N, ldb=None, ldc=None, beta=0.0, transb="N", transc="N", stream=None, alpha=1.0, b_fmt=None,
                bias=None, c_dtype=None):
        """C = alpha . (A . op(B)) + beta C (alpha only for FP8 operators, where it carries the per-tensor scales).
        d_b, d_c: DEVICE memory (DeviceBuffer, torch CUDA tensor or address).  For an FP8 operator B is a torch float8 tensor,
        or device bytes with b_fmt="e4m3" | "e5m2".  transb 'N': B is K x N, 'T': B is stored N x K; transc 'N': C is M x N,
        'T': C is stored N x M.  Pitches default to the dense extents (in elements of C).
        C is fp32 unless d_c is a torch bfloat16 tensor or c_dtype="bf16": then C is bf16 and bias (NULL or a DEVICE array
        of M bf16 values) is added per row before beta C, as include/libxsmm_b200.h states.  A bias with fp32 C is refused."""
        tb, tc = transb in ("T", "t"), transc in ("T", "t")
        ldb = (self.K if tb else N) if ldb is None else ldb
        ldc = (self.M if tc else N) if ldc is None else ldc
        bf16_c = _c_is_bf16(d_c, c_dtype)
        if bias is not None and not bf16_c:
            raise ValueError("a bias needs bf16 C (a torch bfloat16 d_c or c_dtype='bf16'): the fp32-output entries have no bias")
        if bias is not None:
            _check_bias(bias, self.M)
        if self.fp8:
            b_code = _fp8_format(d_b, b_fmt)
            if bf16_c:
                sp24_execute_fp8_bf16out(self.handle, transb, transc, N, d_b, b_code, ldb, alpha, bias, beta, d_c, ldc, stream)
            else:
                sp24_execute_fp8(self.handle, transb, transc, N, d_b, b_code, ldb, alpha, beta, d_c, ldc, stream)
        else:
            assert alpha == 1.0 and b_fmt is None, "alpha and b_fmt belong to FP8 operators"
            if bf16_c:
                sp24_execute_bf16out(self.handle, transb, transc, N, d_b, ldb, bias, beta, d_c, ldc, stream)
            else:
                sp24_execute(self.handle, transb, transc, N, d_b, ldb, beta, d_c, ldc, stream)

    def linear(self, x, bias=None, alpha=1.0):
        """y = x . Aᵀ (+ bias), what torch.nn.functional.linear(x, W, bias) returns for the pruned weight W = A, in bf16.
        x: a contiguous CUDA tensor whose last dimension is K -- bfloat16 for a bf16 operator, float8_e4m3fn / float8_e5m2
        for an FP8 one, where alpha carries scale_x * scale_w.  bias: None or a CUDA bfloat16 tensor of M elements.
        Returns y of shape x.shape[:-1] + (M,), bfloat16, on x's device; runs on torch.cuda.current_stream() with
        transb = transc = 'T', N = x.numel() // K and ldb = K.  Inputs the library would refuse raise ValueError here,
        and x is never copied or padded."""
        import torch
        if not isinstance(x, torch.Tensor):
            raise ValueError("x must be a torch tensor, got %s" % type(x).__name__)
        if self.fp8:
            if x.dtype not in (torch.float8_e4m3fn, torch.float8_e5m2):
                raise ValueError("an FP8 operator takes x as float8_e4m3fn or float8_e5m2, got %s" % x.dtype)
        else:
            if x.dtype != torch.bfloat16:
                raise ValueError("a bf16 operator takes x as bfloat16, got %s" % x.dtype)
            if alpha != 1.0:
                raise ValueError("alpha=%r: alpha belongs to FP8 operators" % (alpha,))
        if x.dim() < 1 or x.shape[-1] != self.K:
            raise ValueError("x has shape %s: its last dimension must be K=%d" % (tuple(x.shape), self.K))
        if not x.is_contiguous():
            raise ValueError("x must be contiguous (its rows are read through TMA with pitch K)")
        unit = 16 if self.fp8 else 8
        if self.K % unit:
            raise ValueError("K=%d must be a multiple of %d: x is read through TMA with pitch K, in whole 16-byte units"
                             % (self.K, unit))
        if x.data_ptr() % 16:
            raise ValueError("x must start on a 16-byte boundary (it is read through TMA)")
        if bias is not None:
            if not isinstance(bias, torch.Tensor):
                raise ValueError("bias must be a torch tensor, got %s" % type(bias).__name__)
            _check_bias(bias, self.M)
        if x.device.type != "cuda":
            raise ValueError("x must be a CUDA tensor, got one on %s" % x.device)
        if bias is not None and bias.device != x.device:
            raise ValueError("bias is on %s, x on %s" % (bias.device, x.device))
        N = x.numel() // self.K
        y = torch.empty(tuple(x.shape[:-1]) + (self.M,), dtype=torch.bfloat16, device=x.device)
        if N == 0:
            return y
        self.execute(x, y, N, ldb=self.K, ldc=self.M, transb="T", transc="T", stream=torch.cuda.current_stream(x.device),
                     alpha=alpha, bias=bias)
        check()
        return y

    def destroy(self):
        if self.handle:
            sp24_destroy(self.handle)
            self.handle = None


def _dptr(x):
    return x.data_ptr() if hasattr(x, "data_ptr") else _addr(x)


def sp24_create_bfloat16(M, K, lda, a):
    """the raw create entry: a is an address (host or device) or None; the handle or None"""
    L = load()
    f = L.libxsmm_b200_sp24_create_bfloat16
    f.restype = ctypes.c_void_p
    f.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p]
    return f(M, K, lda, _dptr(a))


def sp24_execute(handle, transb, transc, N, d_b, ldb, beta, d_c, ldc, stream=None):
    """the raw execute entry (arguments checked by the library, error -97)"""
    L = load()
    f = L.libxsmm_b200_sp24_execute
    f.restype = None
    f.argtypes = [ctypes.c_void_p, ctypes.c_char, ctypes.c_char, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_float,
                  ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    s = stream.cuda_stream if hasattr(stream, "cuda_stream") else _sptr(stream)
    f(handle, _c(transb), _c(transc), N, _dptr(d_b), ldb, float(beta), _dptr(d_c), ldc, s)


def sp24_create_fp8(M, K, lda, a, fmt):
    """the raw FP8 create entry: a is an address (host or device) or None, fmt 0 (e4m3) / 1 (e5m2); the handle or None"""
    L = load()
    f = L.libxsmm_b200_sp24_create_fp8
    f.restype = ctypes.c_void_p
    f.argtypes = [ctypes.c_int] * 3 + [ctypes.c_void_p, ctypes.c_int]
    return f(M, K, lda, _dptr(a), fmt)


def sp24_execute_fp8(handle, transb, transc, N, d_b, b_fmt, ldb, alpha, beta, d_c, ldc, stream=None):
    """the raw FP8 execute entry (arguments checked by the library, error -97); b_fmt 0 (e4m3) / 1 (e5m2)"""
    L = load()
    f = L.libxsmm_b200_sp24_execute_fp8
    f.restype = None
    f.argtypes = [ctypes.c_void_p, ctypes.c_char, ctypes.c_char, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                  ctypes.c_float, ctypes.c_float, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    s = stream.cuda_stream if hasattr(stream, "cuda_stream") else _sptr(stream)
    f(handle, _c(transb), _c(transc), N, _dptr(d_b), b_fmt, ldb, float(alpha), float(beta), _dptr(d_c), ldc, s)


def sp24_execute_bf16out(handle, transb, transc, N, d_b, ldb, bias, beta, d_c, ldc, stream=None):
    """the raw bf16-output entry of a bf16 operator (arguments checked by the library, error -97); bias None or M bf16 values"""
    L = load()
    f = L.libxsmm_b200_sp24_execute_bf16out
    f.restype = None
    f.argtypes = [ctypes.c_void_p, ctypes.c_char, ctypes.c_char, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                  ctypes.c_float, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    s = stream.cuda_stream if hasattr(stream, "cuda_stream") else _sptr(stream)
    f(handle, _c(transb), _c(transc), N, _dptr(d_b), ldb, _dptr(bias), float(beta), _dptr(d_c), ldc, s)


def sp24_execute_fp8_bf16out(handle, transb, transc, N, d_b, b_fmt, ldb, alpha, bias, beta, d_c, ldc, stream=None):
    """the raw bf16-output entry of an FP8 operator (arguments checked by the library, error -97); b_fmt 0 (e4m3) / 1 (e5m2)"""
    L = load()
    f = L.libxsmm_b200_sp24_execute_fp8_bf16out
    f.restype = None
    f.argtypes = [ctypes.c_void_p, ctypes.c_char, ctypes.c_char, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_int,
                  ctypes.c_float, ctypes.c_void_p, ctypes.c_float, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    s = stream.cuda_stream if hasattr(stream, "cuda_stream") else _sptr(stream)
    f(handle, _c(transb), _c(transc), N, _dptr(d_b), b_fmt, ldb, float(alpha), _dptr(bias), float(beta), _dptr(d_c), ldc, s)


def sp24_destroy(handle):
    L = load()
    L.libxsmm_b200_sp24_destroy.restype = None
    L.libxsmm_b200_sp24_destroy.argtypes = [ctypes.c_void_p]
    L.libxsmm_b200_sp24_destroy(handle)


# ---- host-only planning (works without a GPU) ----------------------------------------------------------
def spmdm_geometry(M, N, K, max_threads=1, bn=48):
    vec = (ctypes.c_int * 9)()
    if 0 != load().libxsmm_b200_spmdm_geometry(M, N, K, max_threads, bn, ctypes.cast(vec, ctypes.c_void_p)):
        raise ValueError("spmdm_geometry(%d,%d,%d)" % (M, N, K))
    return dict(zip(("m", "n", "k", "bm", "bn", "bk", "mb", "nb", "kb"), [int(v) for v in vec]))


def fsspmdm_plan(a_dense, N=16, ldb=None, ldc=None, beta=0.0, lda=None):
    a = np.ascontiguousarray(a_dense)
    assert a.dtype in (np.float64, np.float32)
    M, K = a.shape
    info = (ctypes.c_longlong * 6)()
    rc = load().libxsmm_b200_fsspmdm_plan(int(a.dtype == np.float64), M, N, K, K if lda is None else lda,
                                          N if ldb is None else ldb, N if ldc is None else ldc, float(beta),
                                          a.ctypes.data, ctypes.cast(info, ctypes.c_void_p))
    if rc != 0:
        code, msg = last_error()
        clear_error()
        raise ValueError(msg)
    return dict(nnz=int(info[0]), n_unique=int(info[1]), sparse=bool(info[2]), x86_code_size=int(info[3]), chunk=int(info[4]),
                form={0: "generic", 1: "baked-registers", 2: "baked-strip"}[int(info[5])])


def fsspmdm_kernel_source(a_dense, N=16, ldb=None, ldc=None, beta=0.0):
    a = np.ascontiguousarray(a_dense)
    M, K = a.shape
    L = load()
    p = L.libxsmm_b200_fsspmdm_kernel_source(int(a.dtype == np.float64), M, N, K, K, N if ldb is None else ldb,
                                             N if ldc is None else ldc, float(beta), a.ctypes.data)
    if not p:
        return None
    src = ctypes.string_at(p).decode()
    L.libxsmm_b200_free_string(p)
    return src
