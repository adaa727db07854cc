"""ctypes bindings for libsparsex_b200.so.

Two layers are exposed, both straight through the C-ABI:

* ``CsxMatrix``  — the engine ABI of include/csx_b200.h (csxb_*): tune on the
  host, inspect the CSX arrays, upload, SpMV on raw device pointers (torch
  tensors are only used as device-memory owners).
* ``SpxApi``     — the SparseX drop-in API of include/sparsex/*.h (spx_*), the
  call a user of the reference makes (src/api/matvec.c).
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_LIB = None


class EngineError(RuntimeError):
    pass


def lib_path():
    # SPARSEX_B200_LIB: another build of the same library (kernel experiments, tools/variants.sh)
    return os.environ.get("SPARSEX_B200_LIB") or os.path.join(_HERE, "libsparsex_b200.so")


def lib():
    """Load the product library; there is no fallback."""
    global _LIB
    if _LIB is not None:
        return _LIB
    path = lib_path()
    if not os.path.exists(path):
        raise EngineError("%s is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(the engine has no CPU fallback)" % path)
    L = C.CDLL(path, mode=C.RTLD_GLOBAL)
    vp, i32, i64, dbl, cp = C.c_void_p, C.c_int, C.c_int64, C.c_double, C.c_char_p
    L.csxb_tune_csr.restype = vp
    L.csxb_tune_csr.argtypes = [vp, vp, vp, i64, i64, cp, i32, i32, cp, C.c_size_t]
    L.csxb_tune_csr_slab.restype = vp
    L.csxb_tune_csr_slab.argtypes = [vp, vp, vp, i64, i64, i64, i64, i32, cp, cp, C.c_size_t]
    L.csxb_tune_mmf.restype = vp
    L.csxb_tune_mmf.argtypes = [cp, cp, i32, i32, cp, C.c_size_t]
    L.csxb_destroy.argtypes = [vp]
    L.csxb_info.restype = i64
    L.csxb_info.argtypes = [vp, i32]
    L.csxb_part_info.restype = i64
    L.csxb_part_info.argtypes = [vp, i32, i32]
    L.csxb_part_copy.restype = i32
    L.csxb_part_copy.argtypes = [vp, i32, i32, vp]
    L.csxb_part_log.restype = cp
    L.csxb_part_log.argtypes = [vp, i32]
    L.csxb_upload.restype = i32
    L.csxb_upload.argtypes = [vp, i32, i32]
    L.csxb_last_error.restype = cp
    L.csxb_traffic.restype = i64
    L.csxb_traffic.argtypes = [vp, i32]
    L.csxb_spmv.restype = i32
    L.csxb_spmv.argtypes = [vp, dbl, vp, dbl, vp, i32, vp]
    L.csxb_spmv_host.restype = i32
    L.csxb_spmv_host.argtypes = [vp, dbl, vp, dbl, vp, i32]
    L.csxb_decode_coords.restype = i32
    L.csxb_decode_coords.argtypes = [vp, i32, vp, vp]
    L.csxb_transpose_prepare.restype = i32
    L.csxb_transpose_prepare.argtypes = [vp]
    L.csxb_spmv_t.restype = i32
    L.csxb_spmv_t.argtypes = [vp, dbl, vp, dbl, vp, i32, vp]
    L.csxb_spmv_t_host.restype = i32
    L.csxb_spmv_t_host.argtypes = [vp, dbl, vp, dbl, vp, i32]
    L.csxb_transpose_info.restype = i64
    L.csxb_transpose_info.argtypes = [vp, i32]
    L.csxb_decode_coords_t.restype = i32
    L.csxb_decode_coords_t.argtypes = [vp, vp, vp]
    L.csxb_save.restype = i32
    L.csxb_save.argtypes = [vp, cp]
    L.csxb_load.restype = vp
    L.csxb_load.argtypes = [cp, cp, C.c_size_t]
    L.csxb_get_entry.restype = i32
    L.csxb_get_entry.argtypes = [vp, i64, i64, C.POINTER(dbl)]
    L.csxb_set_entry.restype = i32
    L.csxb_set_entry.argtypes = [vp, i64, i64, dbl]
    L.csxb_rcm_csr.restype = i32
    L.csxb_rcm_csr.argtypes = [vp, vp, i64, i64, vp, vp]
    L.csxb_permute_csr.restype = i32
    L.csxb_permute_csr.argtypes = [vp, vp, vp, i64, vp, vp, vp, vp]
    L.csxb_set_perm.restype = i32
    L.csxb_set_perm.argtypes = [vp, vp, i64]
    L.csxb_get_perm.restype = i64
    L.csxb_get_perm.argtypes = [vp, vp]
    L.csxb_group_create.restype = vp
    L.csxb_group_create.argtypes = [vp, vp, i32, i32, cp, C.c_size_t]
    L.csxb_group_destroy.argtypes = [vp]
    L.csxb_group_size.restype = i32
    L.csxb_group_size.argtypes = [vp]
    L.csxb_group_member.restype = vp
    L.csxb_group_member.argtypes = [vp, i32]
    L.csxb_group_device.restype = i32
    L.csxb_group_device.argtypes = [vp, i32]
    L.csxb_group_spmv.restype = i32
    L.csxb_group_spmv.argtypes = [vp, dbl, vp, dbl, vp, i32]
    L.csxb_group_spmv_t.restype = i32
    L.csxb_group_spmv_t.argtypes = [vp, dbl, vp, dbl, vp, i32]
    L.csxb_group_save.restype = i32
    L.csxb_group_save.argtypes = [vp, cp]
    L.csxb_group_get_entry.restype = i32
    L.csxb_group_get_entry.argtypes = [vp, i64, i64, C.POINTER(dbl)]
    L.csxb_group_set_entry.restype = i32
    L.csxb_group_set_entry.argtypes = [vp, i64, i64, dbl]
    L.csxb_xchg_create.restype = vp
    L.csxb_xchg_create.argtypes = [vp, i32, i32]
    L.csxb_xchg_handle.restype = i32
    L.csxb_xchg_handle.argtypes = [vp, vp]
    L.csxb_xchg_connect.restype = i32
    L.csxb_xchg_connect.argtypes = [vp, vp, vp, vp, vp, vp]
    L.csxb_xchg_connect_ptr.restype = i32
    L.csxb_xchg_connect_ptr.argtypes = [vp, vp, vp, vp, vp, vp]
    L.csxb_xchg_base.restype = vp
    L.csxb_xchg_base.argtypes = [vp]
    L.csxb_xchg_vector.restype = vp
    L.csxb_xchg_vector.argtypes = [vp, i32]
    L.csxb_xchg_spmv.restype = i32
    L.csxb_xchg_spmv.argtypes = [vp, dbl, vp]
    L.csxb_xchg_status.restype = i64
    L.csxb_xchg_status.argtypes = [vp, i32]
    L.csxb_xchg_destroy.argtypes = [vp]
    _LIB = L
    return L


def rcm_csr(rowptr, colind, n):
    """csxb_rcm_csr: (perm, (bandwidth before, after)) with perm[old] = new, or (None, None) when the matrix has
    no off-diagonal element (Rcm.hpp:275-279)."""
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
    colind = np.ascontiguousarray(colind, dtype=np.int32)
    perm = np.empty(n, dtype=np.int32)
    bw = np.zeros(2, dtype=np.int64)
    rc = lib().csxb_rcm_csr(rowptr.ctypes.data, colind.ctypes.data, n, n, perm.ctypes.data, bw.ctypes.data)
    if rc == 1:
        return None, None
    if rc != 0:
        raise EngineError("csxb_rcm_csr: invalid arguments")
    return perm, (int(bw[0]), int(bw[1]))


def permute_csr(rowptr, colind, values, perm):
    """csxb_permute_csr: P A P^T as (rowptr, colind, values)."""
    rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
    colind = np.ascontiguousarray(colind, dtype=np.int32)
    values = np.ascontiguousarray(values, dtype=np.float64)
    perm = np.ascontiguousarray(perm, dtype=np.int32)
    n = len(rowptr) - 1
    orp, oci, ova = np.empty_like(rowptr), np.empty_like(colind), np.empty_like(values)
    if lib().csxb_permute_csr(rowptr.ctypes.data, colind.ctypes.data, values.ctypes.data, n, perm.ctypes.data,
                              orp.ctypes.data, oci.ctypes.data, ova.ctypes.data) != 0:
        raise EngineError("csxb_permute_csr: invalid arguments")
    return orp, oci, ova


def _opts(opts):
    return ";".join("%s=%s" % (k, v) for k, v in (opts or {}).items()).encode()


class Partition(object):
    """Fields of csx_matrix_t (+ CSX-Sym extras) for one row partition."""
    pass


class CsxMatrix(object):
    """A tuned matrix: csxb_matrix_t handle."""

    # csxb_info / csxb_part_info / csxb_part_copy / csxb_traffic selectors (include/csx_b200.h)
    NROWS, NCOLS, NNZ, SYMMETRIC, NPARTS, NPARTS_TOTAL, PART_LO, FULL_COLIND = range(8)
    B_VALUES, B_CTL, B_TABLES, B_X, B_Y, B_TOTAL, B_LAUNCHES = range(7)

    def __init__(self, handle, keepalive=None):
        self._h = handle
        self._keep = keepalive
        L = lib()
        self.nrows = L.csxb_info(handle, self.NROWS)
        self.ncols = L.csxb_info(handle, self.NCOLS)
        self.nnz = L.csxb_info(handle, self.NNZ)
        self.symmetric = bool(L.csxb_info(handle, self.SYMMETRIC))
        self.nparts = L.csxb_info(handle, self.NPARTS)
        self.nparts_total = L.csxb_info(handle, self.NPARTS_TOTAL)
        self.part_lo = L.csxb_info(handle, self.PART_LO)
        self.uploaded = False

    @classmethod
    def tune_csr(cls, rowptr, colind, values, nrows, ncols, opts=None, part_lo=0, part_hi=-1):
        rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
        colind = np.ascontiguousarray(colind, dtype=np.int32)
        values = np.ascontiguousarray(values, dtype=np.float64)
        err = C.create_string_buffer(1024)
        h = lib().csxb_tune_csr(rowptr.ctypes.data, colind.ctypes.data, values.ctypes.data, nrows, ncols,
                                _opts(opts), part_lo, part_hi, err, 1024)
        if not h:
            raise EngineError(err.value.decode())
        return cls(h)

    @classmethod
    def tune_csr_slab(cls, rowptr, colind, values, nrows_total, ncols, row_start, part, opts=None):
        """Partition `part` of the spx.rt.nr_threads-way split from its own rows only (csxb_tune_csr_slab):
        rowptr (relative to the slab), colind, values of rows [row_start, row_start + len(rowptr) - 1)."""
        rowptr = np.ascontiguousarray(rowptr, dtype=np.int32)
        colind = np.ascontiguousarray(colind, dtype=np.int32)
        values = np.ascontiguousarray(values, dtype=np.float64)
        err = C.create_string_buffer(1024)
        h = lib().csxb_tune_csr_slab(rowptr.ctypes.data, colind.ctypes.data, values.ctypes.data, rowptr.size - 1, nrows_total,
                                     ncols, row_start, part, _opts(opts), err, 1024)
        if not h:
            raise EngineError(err.value.decode())
        return cls(h)

    @classmethod
    def tune_mmf(cls, path, opts=None, part_lo=0, part_hi=-1):
        err = C.create_string_buffer(1024)
        h = lib().csxb_tune_mmf(path.encode(), _opts(opts), part_lo, part_hi, err, 1024)
        if not h:
            raise EngineError(err.value.decode())
        return cls(h)

    def partition(self, p):
        L = lib()
        P = Partition()
        info = [L.csxb_part_info(self._h, p, w) for w in range(11)]
        (P.nnz, P.nrows, P.ncols, P.row_start, P.ctl_size, P.row_jumps, idl, mapl, dvl, ril, P.sampling_undefined) = info

        def grab(what, n, dt):
            a = np.empty(n, dt)
            if n and L.csxb_part_copy(self._h, p, what, a.ctypes.data) != 0:
                raise EngineError(L.csxb_last_error().decode())
            return a
        P.values = grab(0, P.nnz, np.float64)
        P.ctl = grab(1, P.ctl_size, np.uint8)
        P.id_map = grab(2, idl, np.int64)
        ri = grab(3, ril * 3, np.int64).reshape(-1, 3)
        P.rows_info = np.stack([ri[:, 0], ri[:, 1], ri[:, 2] & 0xffffffff], axis=1) if ril else ri
        P.dvalues = grab(4, dvl, np.float64)
        P.map_cpus = grab(5, mapl, np.uint32)
        P.map_pos = grab(6, mapl, np.uint32)
        P.log = L.csxb_part_log(self._h, p).decode()
        return P

    def upload(self, device=0, free_host=False):
        if lib().csxb_upload(self._h, device, int(free_host)) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        self.uploaded = True
        return self

    def traffic(self):
        L = lib()
        keys = ["values", "ctl", "tables", "x", "y", "total", "launches"]
        return {k: L.csxb_traffic(self._h, i) for i, k in enumerate(keys)}

    def spmv_ptr(self, alpha, x_ptr, beta, y_ptr, overwrite, stream=0):
        if lib().csxb_spmv(self._h, alpha, x_ptr, beta, y_ptr, int(overwrite), stream) != 0:
            raise EngineError(lib().csxb_last_error().decode())

    def spmv(self, alpha, x, y, beta=0.0, overwrite=True, stream=None):
        """x, y: torch CUDA float64 tensors (device-memory owners only)."""
        import torch
        assert x.is_cuda and y.is_cuda and x.dtype == torch.float64 and y.dtype == torch.float64
        assert x.numel() == self.ncols and y.numel() == self.nrows and x.is_contiguous() and y.is_contiguous()
        s = torch.cuda.current_stream().cuda_stream if stream is None else stream
        self.spmv_ptr(alpha, x.data_ptr(), beta, y.data_ptr(), overwrite, s)
        return y

    def spmv_host(self, alpha, x, y, beta=0.0, overwrite=True):
        """x, y: numpy float64 arrays in host memory; copies happen inside the call."""
        assert x.dtype == np.float64 and y.dtype == np.float64 and x.flags.c_contiguous and y.flags.c_contiguous
        if lib().csxb_spmv_host(self._h, alpha, x.ctypes.data, beta, y.ctypes.data, int(overwrite)) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return y

    def prepare_transpose(self):
        """Build and upload the tables of the transposed product (csxb_transpose_prepare); idempotent."""
        if lib().csxb_transpose_prepare(self._h) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return self

    def spmv_t(self, alpha, x, y, beta=0.0, overwrite=True, stream=None):
        """y = alpha*A^T*x (+ beta*y): x (nrows) and y (ncols) are torch CUDA float64 tensors."""
        import torch
        assert x.is_cuda and y.is_cuda and x.dtype == torch.float64 and y.dtype == torch.float64
        assert x.numel() == self.nrows and y.numel() == self.ncols and x.is_contiguous() and y.is_contiguous()
        s = torch.cuda.current_stream().cuda_stream if stream is None else stream
        if lib().csxb_spmv_t(self._h, alpha, x.data_ptr(), beta, y.data_ptr(), int(overwrite), s) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return y

    def spmv_t_host(self, alpha, x, y, beta=0.0, overwrite=True):
        """y = alpha*A^T*x (+ beta*y) on numpy float64 host arrays (x: nrows, y: ncols)."""
        assert x.dtype == np.float64 and y.dtype == np.float64 and x.flags.c_contiguous and y.flags.c_contiguous
        assert x.size == self.nrows and y.size == self.ncols
        if lib().csxb_spmv_t_host(self._h, alpha, x.ctypes.data, beta, y.ctypes.data, int(overwrite)) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return y

    def transpose_info(self):
        """csxb_transpose_info after prepare_transpose(): column window, bytes, launches, heavy columns, build time."""
        keys = ["col_lo", "col_hi", "device_bytes", "alg_bytes", "launches", "heavy_cols", "segments", "build_us"]
        return {k: lib().csxb_transpose_info(self._h, i) for i, k in enumerate(keys)}

    def decode_coords_t(self):
        """(rows, cols) of A for every device-wide value index, as the transposed tables gather it (host only)."""
        n = sum(lib().csxb_part_info(self._h, p, 0) for p in range(self.nparts))
        r = np.empty(n, np.int32)
        c = np.empty(n, np.int32)
        if lib().csxb_decode_coords_t(self._h, r.ctypes.data, c.ctypes.data) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return r, c

    def save(self, path):
        if lib().csxb_save(self._h, path.encode()) != 0:
            raise EngineError(lib().csxb_last_error().decode())

    @classmethod
    def load(cls, path):
        err = C.create_string_buffer(1024)
        h = lib().csxb_load(path.encode(), err, 1024)
        if not h:
            raise EngineError(err.value.decode())
        return cls(h)

    def get_entry(self, row, col):
        """A(row, col), zero-based; None when the entry is not stored."""
        v = C.c_double()
        rc = lib().csxb_get_entry(self._h, row, col, C.byref(v))
        if rc < 0:
            raise EngineError(lib().csxb_last_error().decode())
        return v.value if rc == 0 else None

    def set_entry(self, row, col, value):
        rc = lib().csxb_set_entry(self._h, row, col, value)
        if rc < 0:
            raise EngineError(lib().csxb_last_error().decode())
        return rc == 0

    def decode_coords(self, p):
        n = lib().csxb_part_info(self._h, p, 0)
        r = np.empty(n, np.int32)
        c = np.empty(n, np.int32)
        if lib().csxb_decode_coords(self._h, p, r.ctypes.data, c.ctypes.data) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return r, c

    def close(self):
        if self._h:
            lib().csxb_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def _vec_ptr(v, n):
    """numpy float64 array (host buffer) or torch float64 tensor (device or pinned memory) of n entries."""
    if isinstance(v, np.ndarray):
        assert v.dtype == np.float64 and v.flags.c_contiguous and v.size == n
        return v.ctypes.data
    assert v.is_contiguous() and v.numel() == n
    return v.data_ptr()


class DeviceGroup(object):
    """csxb_group_* (include/csx_b200.h): the partitions of one tuned matrix spread over several GPUs of this process.
    Consumes `matrix` (which must hold all partitions and must not be uploaded)."""

    def __init__(self, matrix, devices, free_host=False):
        dev = np.ascontiguousarray(devices, dtype=np.int32)
        err = C.create_string_buffer(1024)
        self.nrows, self.ncols = matrix.nrows, matrix.ncols
        self._h = lib().csxb_group_create(matrix._h, dev.ctypes.data, len(dev), int(free_host), err, 1024)
        if not self._h:
            raise EngineError(err.value.decode())
        matrix._h = None   # consumed
        self.size = lib().csxb_group_size(self._h)

    def member_info(self, i, what):
        return lib().csxb_info(lib().csxb_group_member(self._h, i), what)

    def spmv(self, alpha, x, y, beta=0.0, overwrite=True):
        """x, y: numpy float64 arrays (host buffers) or torch float64 tensors (device or pinned memory)."""
        if lib().csxb_group_spmv(self._h, alpha, _vec_ptr(x, self.ncols), beta, _vec_ptr(y, self.nrows), int(overwrite)) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return y

    def spmv_t(self, alpha, x, y, beta=0.0, overwrite=True):
        """y = alpha*A^T*x (+ beta*y): x has nrows, y ncols entries; the memory kinds of spmv()."""
        if lib().csxb_group_spmv_t(self._h, alpha, _vec_ptr(x, self.nrows), beta, _vec_ptr(y, self.ncols), int(overwrite)) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return y

    def save(self, path):
        if lib().csxb_group_save(self._h, path.encode()) != 0:
            raise EngineError(lib().csxb_last_error().decode())

    def get_entry(self, row, col):
        v = C.c_double()
        rc = lib().csxb_group_get_entry(self._h, row, col, C.byref(v))
        if rc < 0:
            raise EngineError(lib().csxb_last_error().decode())
        return v.value if rc == 0 else None

    def set_entry(self, row, col, value):
        rc = lib().csxb_group_set_entry(self._h, row, col, value)
        if rc < 0:
            raise EngineError(lib().csxb_last_error().decode())
        return rc == 0

    def close(self):
        if self._h:
            lib().csxb_group_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _DevArray(object):
    """Device memory owned by the engine, exposed through __cuda_array_interface__ (float64 vector)."""

    def __init__(self, ptr, n):
        self.__cuda_array_interface__ = {"shape": (n,), "typestr": "<f8", "data": (ptr, False), "version": 2}


class PeerExchange(object):
    """csxb_xchg_* (include/csx_b200.h): repeated SpMV across GPUs with the exchange fused into the kernel."""

    def __init__(self, matrix, rank, world):
        self.A, self.rank, self.world = matrix, rank, world
        self._h = lib().csxb_xchg_create(matrix._h, rank, world)
        if not self._h:
            raise EngineError(lib().csxb_last_error().decode())

    def handle(self):
        buf = np.zeros(64, np.uint8)
        if lib().csxb_xchg_handle(self._h, buf.ctypes.data) != 0:
            raise EngineError(lib().csxb_last_error().decode())
        return buf

    def base(self):
        return lib().csxb_xchg_base(self._h)

    def _ranges(self, ranges, windows):
        a = [np.ascontiguousarray(v, np.int64) for v in ([r[0] for r in ranges], [r[1] for r in ranges],
                                                         [w[0] for w in windows], [w[1] for w in windows])]
        return a

    def connect(self, handles, ranges, windows):
        """handles: (world, 64) uint8 array of every rank's handle(); ranges: (row_lo, row_n); windows: (col_min, col_max)."""
        hb = np.ascontiguousarray(handles, np.uint8)
        a = self._ranges(ranges, windows)
        if lib().csxb_xchg_connect(self._h, hb.ctypes.data, *[v.ctypes.data for v in a]) != 0:
            raise EngineError(lib().csxb_last_error().decode())

    def connect_ptr(self, bases, ranges, windows):
        pb = (C.c_void_p * self.world)(*bases)
        a = self._ranges(ranges, windows)
        if lib().csxb_xchg_connect_ptr(self._h, pb, *[v.ctypes.data for v in a]) != 0:
            raise EngineError(lib().csxb_last_error().decode())

    def vector(self, which):
        """torch view of ping-pong vector `which` (0: the initial x)."""
        import torch
        return torch.as_tensor(_DevArray(lib().csxb_xchg_vector(self._h, which), self.A.nrows), device="cuda")

    def spmv(self, alpha, stream=None):
        import torch
        s = torch.cuda.current_stream().cuda_stream if stream is None else stream
        if lib().csxb_xchg_spmv(self._h, alpha, s) != 0:
            raise EngineError(lib().csxb_last_error().decode())

    def steps(self):
        return lib().csxb_xchg_status(self._h, 0)

    def error(self):
        return lib().csxb_xchg_status(self._h, 1)

    def protocol(self):
        """(mode, edge tiles): mode 1 = edge tiles first, 0 = sync kernel per step."""
        return lib().csxb_xchg_status(self._h, 2), lib().csxb_xchg_status(self._h, 3)

    def close(self):
        if self._h:
            lib().csxb_xchg_destroy(self._h)
            self._h = None


class SpxVector(C.Structure):
    """struct vector_struct (include/sparsex/common.h)."""
    _fields_ = [("elements", C.POINTER(C.c_double)), ("size", C.c_size_t), ("alloc_type", C.c_int),
                ("vec_mode", C.c_int)]


class SpxApi(object):
    """The spx_* functions with argument/return types declared."""

    def __init__(self):
        L = lib()
        self.L = L
        vp, i32, dbl, cp = C.c_void_p, C.c_int, C.c_double, C.c_char_p
        VP = C.POINTER(SpxVector)
        sig = {
            "spx_init": (None, []), "spx_finalize": (None, []),
            "spx_log_disable_all": (None, []), "spx_log_error_console": (None, []),
            "spx_input_load_csr": (vp, [vp, vp, vp, i32, i32]),
            "spx_input_load_mmf": (vp, [cp]),
            "spx_input_destroy": (i32, [vp]),
            "spx_mat_tune": (vp, [vp]),
            "spx_mat_destroy": (i32, [vp]),
            "spx_mat_get_nrows": (i32, [vp]), "spx_mat_get_ncols": (i32, [vp]), "spx_mat_get_nnz": (i32, [vp]),
            "spx_mat_get_partition": (vp, [vp]),
            "spx_mat_get_entry": (i32, [vp, i32, i32, C.POINTER(dbl)]),
            "spx_mat_get_engine": (vp, [vp]),
            "spx_mat_set_entry": (i32, [vp, i32, i32, dbl]),
            "spx_mat_get_perm": (C.POINTER(i32), [vp]),
            "spx_mat_save": (i32, [vp, cp]), "spx_mat_restore": (vp, [cp]),
            "spx_vec_reorder": (i32, [VP, C.POINTER(i32)]), "spx_vec_inv_reorder": (i32, [VP, C.POINTER(i32)]),
            "spx_partition_csr": (vp, [vp, i32, C.c_size_t]),
            "spx_partition_get_rs": (C.POINTER(i32), [vp]), "spx_partition_get_re": (C.POINTER(i32), [vp]),
            "spx_partition_destroy": (i32, [vp]),
            "spx_option_set": (None, [cp, cp]), "spx_options_set_from_env": (None, []),
            "spx_vec_create": (VP, [C.c_size_t, vp]),
            "spx_vec_create_from_buff": (VP, [vp, C.POINTER(vp), C.c_size_t, vp, C.c_uint]),
            "spx_vec_create_random": (VP, [C.c_size_t, vp]),
            "spx_vec_init": (None, [VP, dbl]),
            "spx_vec_init_rand_range": (None, [VP, dbl, dbl]),
            "spx_vec_set_entry": (i32, [VP, i32, dbl]),
            "spx_vec_scale": (None, [VP, VP, dbl]),
            "spx_vec_scale_add": (None, [VP, VP, VP, dbl]),
            "spx_vec_add": (None, [VP, VP, VP]), "spx_vec_sub": (None, [VP, VP, VP]),
            "spx_vec_mul": (dbl, [VP, VP]),
            "spx_vec_copy": (None, [VP, VP]), "spx_vec_compare": (i32, [VP, VP]),
            "spx_vec_destroy": (None, [VP]),
            "spx_matvec_mult": (i32, [dbl, vp, VP, VP]),
            "spx_matvec_kernel": (i32, [dbl, vp, VP, dbl, VP]),
            "spx_matvec_mult_trans": (i32, [dbl, vp, VP, VP]),
            "spx_matvec_kernel_trans": (i32, [dbl, vp, VP, dbl, VP]),
            "spx_matvec_kernel_csr": (i32, [C.POINTER(vp), i32, i32, vp, vp, vp, dbl, VP, dbl, VP]),
            "spx_device_synchronize": (None, []),
            "spx_err_set_handler": (None, [vp]),
        }
        for name, (res, args) in sig.items():
            f = getattr(L, name)
            f.restype = res
            f.argtypes = args
            setattr(self, name, f)
        tune = self.spx_mat_tune

        def spx_mat_tune(inp, option=0):
            # the optional argument is always passed: the callee reads the variadic slot unconditionally (matvec.c:268-272)
            return tune(inp, C.c_int(option))
        self.spx_mat_tune = spx_mat_tune

    @staticmethod
    def as_numpy(vec):
        v = vec.contents
        return np.ctypeslib.as_array(v.elements, shape=(v.size,))


def load_spx_api():
    return SpxApi()
