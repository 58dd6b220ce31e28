"""Host-side mirror of the reference's interface for the CSR / TJDS path, over the C ABI of
libsmvp_cuda (include/smvp_cuda.h).

The reference exposes the path as two C functions called from main() (main-cli.c:1457, :1469):

    double *smvp_csr_compute (MMRawData *mmImportData, int fInputRows, int fInputNonZeros, int compiter, struct _time_data_ *csr_time)
    double *smvp_tjds_compute(MMRawData *mmImportData, int fInputRows, int fInputColumns, int fInputNonZeros, int compiter, struct _time_data_ *tjds_time)

`smvp_csr_compute` / `smvp_tjds_compute` below keep those names and argument meanings (the time
struct is returned instead of filled through a pointer).  `CsrMatrix` / `TjdsMatrix` expose the split
build / multiply steps of the C ABI for callers that keep a matrix resident across calls.

There is NO CPU fallback: if the CUDA library is missing or no device is present every call raises.
Nothing in this package imports or executes anything under oracle/.
"""
import ctypes
import os

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SMVP_LIB_PATH") or os.path.join(HERE, "lib", "libsmvp_cuda.so")  # override: tuning builds only

# == MMRawData (main-cli.c:42-47)
COO_DT = np.dtype([("row", "<i4"), ("col", "<i4"), ("val", "<f8")])

CSR_AUTO, CSR_VECTOR, CSR_MERGE = 0, 1, 2
TJDS_ATOMIC, TJDS_DETERMINISTIC, TJDS_DETERMINISTIC_FAST = 0, 1, 2
VAL_STENCIL, VAL_HASH, VAL_ONES = 0, 1, 2

OK, E_ARG, E_ALLOC, E_CUDA, E_RANGE, E_TOOBIG = 0, -1, -2, -3, -4, -5


class SmvpError(RuntimeError):
    def __init__(self, code, where):
        L = lib()
        msg = L.smvp_strerror(code).decode()
        detail = L.smvp_last_cuda_error().decode()
        super().__init__("%s: %s (%d)%s" % (where, msg, code, (" -- " + detail) if detail and code == E_CUDA else ""))
        self.code = code


class _CsrInfo(ctypes.Structure):
    _fields_ = [("rows", ctypes.c_int32), ("cols", ctypes.c_int32), ("nnz", ctypes.c_int64),
                ("max_row_nnz", ctypes.c_int32), ("auto_variant", ctypes.c_int32), ("input_order", ctypes.c_int32),
                ("bytes_per_mult", ctypes.c_int64), ("device_bytes", ctypes.c_int64),
                ("launches_per_mult", ctypes.c_int32 * 3), ("x_relabel", ctypes.c_int32),
                ("row_patterns", ctypes.c_int32), ("value_bytes", ctypes.c_int32)]


class _TjdsInfo(ctypes.Structure):
    _fields_ = [("rows", ctypes.c_int32), ("cols", ctypes.c_int32), ("nnz", ctypes.c_int64), ("ndiag", ctypes.c_int32),
                ("ref_diag_limit", ctypes.c_int32), ("input_order", ctypes.c_int32), ("bytes_per_mult", ctypes.c_int64),
                ("device_bytes", ctypes.c_int64), ("launches_per_mult", ctypes.c_int32 * 3), ("y_relabel", ctypes.c_int32),
                ("skewed_walk", ctypes.c_int32), ("det_route", ctypes.c_int32)]


class _TimeStats(ctypes.Structure):
    _fields_ = [("time_total", ctypes.c_double), ("time_avg", ctypes.c_double), ("time_stdev", ctypes.c_double),
                ("time_min", ctypes.c_double), ("time_max", ctypes.c_double)]


# every symbol include/smvp_cuda.h and include/smvp_synth.h declare, with its ctypes signature
_vp, _i32, _i64, _int, _u64, _dbl = (ctypes.c_void_p, ctypes.c_int32, ctypes.c_int64, ctypes.c_int, ctypes.c_uint64,
                                     ctypes.c_double)
_pp = ctypes.POINTER(ctypes.c_void_p)
_pi64 = ctypes.POINTER(ctypes.c_int64)
SIGNATURES = {
    "smvp_time_stats": (_int, [_vp, _int, ctypes.POINTER(_TimeStats)]),
    "smvp_csr_build": (_int, [_vp, _i32, _i32, _i64, _pp]),
    "smvp_tjds_build": (_int, [_vp, _i32, _i32, _i64, _pp]),
    "smvp_csr_mult": (_int, [_vp, _vp, _vp, _int, _vp, _int]),
    "smvp_tjds_mult": (_int, [_vp, _vp, _vp, _int, _vp, _int, _i32]),
    "smvp_csr_build_device": (_int, [_vp, _vp, _vp, _i32, _i32, _i64, _pp]),
    "smvp_tjds_build_device": (_int, [_vp, _vp, _vp, _i32, _i32, _i64, _pp]),
    "smvp_csr_set_x_device": (_int, [_vp, _vp, _vp]),
    "smvp_csr_mult_device": (_int, [_vp, _vp, _vp, _int, _vp]),
    "smvp_csr_set_corunner_headroom": (_int, [_vp, _int]),
    "smvp_csr_mult_device_fanout": (_int, [_vp, _vp, _vp, _int, _int, _vp]),
    "smvp_tjds_set_x_device": (_int, [_vp, _vp, _vp]),
    "smvp_tjds_mult_device": (_int, [_vp, _vp, _int, _i32, _vp]),
    "smvp_csr_transpose": (_int, [_vp, _pp]),
    "smvp_tjds_mult_transpose_device": (_int, [_vp, _vp, _vp, _vp]),
    "smvp_tjds_mult_transpose": (_int, [_vp, _vp, _vp, _int, _vp]),
    "smvp_csr_mult_device_axpby": (_int, [_vp, _dbl, _vp, _dbl, _vp, _int, _vp]),
    "smvp_tjds_mult_device_axpby": (_int, [_vp, _dbl, _dbl, _vp, _int, _i32, _vp]),
    "smvp_tjds_mult_transpose_device_axpby": (_int, [_vp, _dbl, _vp, _dbl, _vp, _vp]),
    "smvp_csr_mult_device_axpby_dot": (_int, [_vp, _dbl, _vp, _dbl, _vp, _vp, _vp, _int, _vp]),
    "smvp_tjds_mult_device_axpby_dot": (_int, [_vp, _dbl, _dbl, _vp, _vp, _vp, _int, _i32, _vp]),
    "smvp_tjds_mult_transpose_device_axpby_dot": (_int, [_vp, _dbl, _vp, _dbl, _vp, _vp, _vp, _vp]),
    "smvp_csr_info": (_int, [_vp, ctypes.POINTER(_CsrInfo)]),
    "smvp_tjds_info": (_int, [_vp, ctypes.POINTER(_TjdsInfo)]),
    "smvp_csr_export": (_int, [_vp, _vp, _vp, _vp]),
    "smvp_tjds_export": (_int, [_vp, _vp, _vp, _vp, _vp]),
    "smvp_csr_arrays_device": (_int, [_vp, _pp, _pp, _pp]),
    "smvp_csr_free": (None, [_vp]),
    "smvp_tjds_free": (None, [_vp]),
    "smvp_host_alloc": (_vp, [_i64]),
    "smvp_host_free": (None, [_vp]),
    "smvp_strerror": (ctypes.c_char_p, [_int]),
    "smvp_last_cuda_error": (ctypes.c_char_p, []),
    "smvp_device_count": (_int, []),
    "smvp_launch_count": (_i64, []),
    # include/smvp_synth.h
    "smvp_synth_stencil27": (_int, [_i32, _i32, _i32, _i64, _i64, _int, _u64, _pp, _pp, _pp, _pi64]),
    "smvp_synth_stencil27_prefix": (_i64, [_i32, _i32, _i32, _i64]),
    "smvp_synth_rmat": (_int, [_int, _i64, _dbl, _dbl, _dbl, _int, _u64, _pp, _pp, _pp, _pi64]),
    "smvp_synth_vector": (_int, [_vp, _i64, _u64, _vp]),
    "smvp_coo_filter_device": (_int, [_vp, _vp, _vp, _i64, _i32, _i32, _i32, _i32, _i32, _i32, _pp, _pp, _pp, _pi64]),
    "smvp_coo_histogram_device": (_int, [_vp, _vp, _i64, _int, _i32, _vp]),
    "smvp_vector_add_device": (_int, [_vp, _vp, _i64, _vp]),
    "smvp_copy_device": (_int, [_vp, _vp, _i64, _vp]),
    "smvp_push_device": (_int, [_vp, _vp, _i64, _int, _vp]),
    "smvp_push_fanout_device": (_int, [_vp, _int, _vp, _i64, _int, _vp]),
    "smvp_push_tma_device": (_int, [_vp, _int, _vp, _i64, _int, _vp]),
    "smvp_sum_ordered_device": (_int, [_vp, _vp, _int, _i64, _i64, _vp]),
    "smvp_sum_ordered_ptrs_device": (_int, [_vp, _vp, _int, _i64, _vp]),
    "smvp_flush_l2": (_int, [_i64, _vp]),
    "smvp_device_free": (None, [_vp]),
}

_lib = None


def lib():
    """Load libsmvp_cuda.so.  Fails loudly when it has not been built: there is no other code path."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError("libsmvp_cuda.so is not built (%s missing): run `python smvp-toolkit_b200/build.py` or "
                               "__graft_entry__.build(); there is no CPU fallback" % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            f = getattr(L, name)  # AttributeError if the library does not export a declared symbol
            f.restype = res
            f.argtypes = args
        _lib = L
    return _lib


def _check(code, where):
    if code != OK:
        raise SmvpError(code, where)


def _ptr(a):
    if a is None:
        return None
    if isinstance(a, np.ndarray):
        return a.ctypes.data_as(ctypes.c_void_p)
    if isinstance(a, int):
        return ctypes.c_void_p(a)
    if hasattr(a, "data_ptr"):  # torch tensor
        return ctypes.c_void_p(a.data_ptr())
    if hasattr(a, "ptr"):  # DeviceArray
        return ctypes.c_void_p(a.ptr)
    raise TypeError("cannot take a pointer of %r" % type(a))


def _stream(stream):
    if stream is None:
        return None
    if isinstance(stream, int):
        return ctypes.c_void_p(stream)
    return ctypes.c_void_p(stream.cuda_stream)  # torch.cuda.Stream


def device_count():
    n = lib().smvp_device_count()
    if n < 0:
        raise SmvpError(n, "smvp_device_count")
    return n


def launch_count():
    return int(lib().smvp_launch_count())


class DeviceArray:
    """A device buffer returned by the library (owned here, freed with smvp_device_free).
    Exposes __cuda_array_interface__ so torch.as_tensor(arr, device="cuda") views it without a copy."""

    def __init__(self, ptr, n, dtype):
        self.ptr, self.n, self.dtype = int(ptr or 0), int(n), np.dtype(dtype)

    @property
    def __cuda_array_interface__(self):
        return {"shape": (self.n,), "typestr": self.dtype.str, "data": (self.ptr, False), "version": 2}

    def free(self):
        if self.ptr:
            lib().smvp_device_free(ctypes.c_void_p(self.ptr))
            self.ptr = 0

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class TimeData:
    """struct _time_data_ (main-cli.c:87-95)."""

    def __init__(self, time_each):
        self.time_each = np.ascontiguousarray(time_each, np.float64)
        st = _TimeStats()
        _check(lib().smvp_time_stats(_ptr(self.time_each), len(self.time_each), ctypes.byref(st)), "smvp_time_stats")
        self.time_total, self.time_avg, self.time_stdev = st.time_total, st.time_avg, st.time_stdev
        self.time_min, self.time_max = st.time_min, st.time_max


def _as_coo(coo):
    coo = np.ascontiguousarray(coo)
    if coo.dtype != COO_DT:
        raise TypeError("COO must be a numpy array of dtype %r (== MMRawData)" % (COO_DT,))
    return coo


class CsrMatrix:
    """CSRData (main-cli.c:61-66) resident in HBM behind an smvp_csr handle."""

    def __init__(self, handle):
        self._h = handle
        info = _CsrInfo()
        _check(lib().smvp_csr_info(self._h, ctypes.byref(info)), "smvp_csr_info")
        self.rows, self.cols, self.nnz = info.rows, info.cols, info.nnz
        self.max_row_nnz, self.auto_variant, self.input_order = info.max_row_nnz, info.auto_variant, info.input_order
        self.bytes_per_mult, self.device_bytes = info.bytes_per_mult, info.device_bytes
        self.launches_per_mult = list(info.launches_per_mult)

    @classmethod
    def build(cls, coo, rows, cols):
        """COO on the host -> CSR in HBM (smvp_csr_build; replaces main-cli.c:336-365)."""
        coo = _as_coo(coo)
        h = ctypes.c_void_p()
        _check(lib().smvp_csr_build(_ptr(coo), rows, cols, len(coo), ctypes.byref(h)), "smvp_csr_build")
        return cls(h)

    @classmethod
    def build_device(cls, d_row, d_col, d_val, rows, cols, nnz):
        h = ctypes.c_void_p()
        _check(lib().smvp_csr_build_device(_ptr(d_row), _ptr(d_col), _ptr(d_val), rows, cols, nnz, ctypes.byref(h)),
               "smvp_csr_build_device")
        return cls(h)

    def transpose(self):
        """A^T as a new, independent CsrMatrix built on the device (smvp_csr_transpose); this matrix is unchanged."""
        h = ctypes.c_void_p()
        _check(lib().smvp_csr_transpose(self._h, ctypes.byref(h)), "smvp_csr_transpose")
        return CsrMatrix(h)

    def mult(self, x, iters=1, variant=CSR_AUTO):
        """`iters` timed passes of y = A x with host vectors (smvp_csr_mult). Returns (y, TimeData)."""
        x = np.ascontiguousarray(x, np.float64)
        if x.shape != (self.cols,):
            raise ValueError("x must have %d entries" % self.cols)
        y = np.zeros(self.rows, np.float64)
        ms = np.zeros(iters, np.float64)
        _check(lib().smvp_csr_mult(self._h, _ptr(x), _ptr(y), iters, _ptr(ms), variant), "smvp_csr_mult")
        return y, TimeData(ms)

    def set_x_device(self, d_x, stream=None):
        """Declare the x of the following passes (smvp_csr_set_x_device); pass d_x=None to mult_device afterwards."""
        _check(lib().smvp_csr_set_x_device(self._h, _ptr(d_x), _stream(stream)), "smvp_csr_set_x_device")

    def set_corunner_headroom(self, ctas_per_sm):
        """Leave room for `ctas_per_sm` CTAs of another kernel per SM beside the persistent merge-path grid."""
        _check(lib().smvp_csr_set_corunner_headroom(self._h, ctas_per_sm), "smvp_csr_set_corunner_headroom")

    def mult_device(self, d_x, d_y, variant=CSR_AUTO, stream=None):
        """One pass y = A x; d_x=None uses the x last given to set_x_device."""
        _check(lib().smvp_csr_mult_device(self._h, _ptr(d_x), _ptr(d_y), variant, _stream(stream)), "smvp_csr_mult_device")

    def mult_device_axpby(self, alpha, d_x, beta, d_y, variant=CSR_AUTO, stream=None):
        """One pass y = alpha * A x + beta * y fused into the multiply (beta == 0: y is not read); d_x=None uses the x
        last given to set_x_device.  See smvp_csr_mult_device_axpby in include/smvp_cuda.h."""
        _check(lib().smvp_csr_mult_device_axpby(self._h, alpha, _ptr(d_x), beta, _ptr(d_y), variant, _stream(stream)),
               "smvp_csr_mult_device_axpby")

    def mult_device_axpby_dot(self, alpha, d_x, beta, d_y, d_w, d_dot, variant=CSR_AUTO, stream=None):
        """mult_device_axpby with d_dot[0] = sum of w[r] * y_new[r] formed in the same pass (d_w=None: w = y_new, the
        squared norm).  d_dot is a one-element device tensor, overwritten.  See smvp_csr_mult_device_axpby_dot in
        include/smvp_cuda.h for the order of the sum and its error bound."""
        _check(lib().smvp_csr_mult_device_axpby_dot(self._h, alpha, _ptr(d_x), beta, _ptr(d_y), _ptr(d_w), _ptr(d_dot), variant,
                                                    _stream(stream)), "smvp_csr_mult_device_axpby_dot")

    @property
    def x_relabel(self):
        """1: the multiply reads popularity-relabelled columns, -1: natural order, 0: not decided yet."""
        info = _CsrInfo()
        _check(lib().smvp_csr_info(self._h, ctypes.byref(info)), "smvp_csr_info")
        return info.x_relabel

    @property
    def row_patterns(self):
        """P > 0: the merge variant streams one of P row patterns per row instead of col_ind, -1: not used, 0: not decided yet."""
        info = _CsrInfo()
        _check(lib().smvp_csr_info(self._h, ctypes.byref(info)), "smvp_csr_info")
        return info.row_patterns

    @property
    def value_bytes(self):
        """With row_patterns > 0: 2 / 4 / 8 = the pattern kernel streams the values as fp16 / fp32 / fp64 (a narrow width
        only when every value converts to it and back exactly), 0: not decided yet."""
        info = _CsrInfo()
        _check(lib().smvp_csr_info(self._h, ctypes.byref(info)), "smvp_csr_info")
        return info.value_bytes

    def mult_device_fanout(self, d_x, y_ptrs, variant=CSR_AUTO, stream=None):
        """y = A x stored into every destination of y_ptrs (device addresses, possibly peer-mapped)."""
        arr = (ctypes.c_void_p * len(y_ptrs))(*[int(p) for p in y_ptrs])
        _check(lib().smvp_csr_mult_device_fanout(self._h, _ptr(d_x), arr, len(y_ptrs), variant, _stream(stream)),
               "smvp_csr_mult_device_fanout")

    def export(self):
        row_ptr = np.zeros(self.rows + 1, np.int32)
        col_ind = np.zeros(self.nnz, np.int32)
        val = np.zeros(self.nnz, np.float64)
        _check(lib().smvp_csr_export(self._h, _ptr(row_ptr), _ptr(col_ind), _ptr(val)), "smvp_csr_export")
        return row_ptr, col_ind, val

    def export_row_ptr(self):
        row_ptr = np.zeros(self.rows + 1, np.int32)
        _check(lib().smvp_csr_export(self._h, _ptr(row_ptr), None, None), "smvp_csr_export")
        return row_ptr

    def device_arrays(self):
        a, b, c = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        _check(lib().smvp_csr_arrays_device(self._h, ctypes.byref(a), ctypes.byref(b), ctypes.byref(c)),
               "smvp_csr_arrays_device")
        return a.value, b.value, c.value

    def free(self):
        if self._h:
            lib().smvp_csr_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class TjdsMatrix:
    """TJDSData (main-cli.c:70-75) + the column permutation, resident in HBM behind an smvp_tjds handle."""

    def __init__(self, handle):
        self._h = handle
        info = _TjdsInfo()
        _check(lib().smvp_tjds_info(self._h, ctypes.byref(info)), "smvp_tjds_info")
        self.rows, self.cols, self.nnz, self.ndiag = info.rows, info.cols, info.nnz, info.ndiag
        self.ref_diag_limit, self.input_order = info.ref_diag_limit, info.input_order
        self.bytes_per_mult, self.device_bytes = info.bytes_per_mult, info.device_bytes
        self.launches_per_mult = list(info.launches_per_mult)

    @property
    def y_relabel(self):
        """1: the multiply scatters through popularity-relabelled rows, -1: natural order, 0: not decided yet."""
        info = _TjdsInfo()
        _check(lib().smvp_tjds_info(self._h, ctypes.byref(info)), "smvp_tjds_info")
        return info.y_relabel

    def plan(self):
        """(skewed_walk, det_route) as smvp_tjds_info_t reports them now (see include/smvp_cuda.h)."""
        info = _TjdsInfo()
        _check(lib().smvp_tjds_info(self._h, ctypes.byref(info)), "smvp_tjds_info")
        return info.skewed_walk, info.det_route

    @classmethod
    def build(cls, coo, rows, cols):
        """COO on the host -> TJDS in HBM (smvp_tjds_build; replaces main-cli.c:755-967)."""
        coo = _as_coo(coo)
        h = ctypes.c_void_p()
        _check(lib().smvp_tjds_build(_ptr(coo), rows, cols, len(coo), ctypes.byref(h)), "smvp_tjds_build")
        return cls(h)

    @classmethod
    def build_device(cls, d_row, d_col, d_val, rows, cols, nnz):
        h = ctypes.c_void_p()
        _check(lib().smvp_tjds_build_device(_ptr(d_row), _ptr(d_col), _ptr(d_val), rows, cols, nnz, ctypes.byref(h)),
               "smvp_tjds_build_device")
        return cls(h)

    def mult(self, x, iters=1, variant=TJDS_ATOMIC, diag_limit=0):
        x = np.ascontiguousarray(x, np.float64)
        if x.shape != (self.cols,):
            raise ValueError("x must have %d entries" % self.cols)
        y = np.zeros(self.rows, np.float64)
        ms = np.zeros(iters, np.float64)
        _check(lib().smvp_tjds_mult(self._h, _ptr(x), _ptr(y), iters, _ptr(ms), variant, diag_limit), "smvp_tjds_mult")
        return y, TimeData(ms)

    def mult_transpose(self, x, iters=1):
        """`iters` timed passes of y = A^T x with host vectors (smvp_tjds_mult_transpose): x has `rows` entries, y `cols`.
        Returns (y, TimeData)."""
        x = np.ascontiguousarray(x, np.float64)
        if x.shape != (self.rows,):
            raise ValueError("x must have %d entries" % self.rows)
        y = np.zeros(self.cols, np.float64)
        ms = np.zeros(iters, np.float64)
        _check(lib().smvp_tjds_mult_transpose(self._h, _ptr(x), _ptr(y), iters, _ptr(ms)), "smvp_tjds_mult_transpose")
        return y, TimeData(ms)

    def mult_transpose_device(self, d_x, d_y, stream=None):
        """One pass y = A^T x on device vectors (d_x: `rows` entries, d_y: `cols`)."""
        _check(lib().smvp_tjds_mult_transpose_device(self._h, _ptr(d_x), _ptr(d_y), _stream(stream)),
               "smvp_tjds_mult_transpose_device")

    def mult_transpose_device_axpby(self, alpha, d_x, beta, d_y, stream=None):
        """One pass y = alpha * A^T x + beta * y (d_x: `rows` entries, d_y: `cols`; beta == 0: y is not read)."""
        _check(lib().smvp_tjds_mult_transpose_device_axpby(self._h, alpha, _ptr(d_x), beta, _ptr(d_y), _stream(stream)),
               "smvp_tjds_mult_transpose_device_axpby")

    def mult_transpose_device_axpby_dot(self, alpha, d_x, beta, d_y, d_w, d_dot, stream=None):
        """mult_transpose_device_axpby with d_dot[0] = sum over the `cols` entries of w[c] * y_new[c] (d_w=None: w = y_new)."""
        _check(lib().smvp_tjds_mult_transpose_device_axpby_dot(self._h, alpha, _ptr(d_x), beta, _ptr(d_y), _ptr(d_w), _ptr(d_dot),
                                                               _stream(stream)), "smvp_tjds_mult_transpose_device_axpby_dot")

    def set_x_device(self, d_x, stream=None):
        _check(lib().smvp_tjds_set_x_device(self._h, _ptr(d_x), _stream(stream)), "smvp_tjds_set_x_device")

    def mult_device(self, d_y, variant=TJDS_ATOMIC, diag_limit=0, stream=None):
        _check(lib().smvp_tjds_mult_device(self._h, _ptr(d_y), variant, diag_limit, _stream(stream)),
               "smvp_tjds_mult_device")

    def mult_device_axpby(self, alpha, beta, d_y, variant=TJDS_ATOMIC, diag_limit=0, stream=None):
        """One pass y = alpha * A x + beta * y with the x last given to set_x_device (beta == 0: y is not read)."""
        _check(lib().smvp_tjds_mult_device_axpby(self._h, alpha, beta, _ptr(d_y), variant, diag_limit, _stream(stream)),
               "smvp_tjds_mult_device_axpby")

    def mult_device_axpby_dot(self, alpha, beta, d_y, d_w, d_dot, variant=TJDS_ATOMIC, diag_limit=0, stream=None):
        """mult_device_axpby with d_dot[0] = sum of w[r] * y_new[r] formed in the same pass (d_w=None: w = y_new)."""
        _check(lib().smvp_tjds_mult_device_axpby_dot(self._h, alpha, beta, _ptr(d_y), _ptr(d_w), _ptr(d_dot), variant, diag_limit,
                                                     _stream(stream)), "smvp_tjds_mult_device_axpby_dot")

    def export(self):
        perm = np.zeros(self.cols, np.int32)
        start_pos = np.zeros(self.ndiag + 1, np.int32)
        row_ind = np.zeros(self.nnz, np.int32)
        val = np.zeros(self.nnz, np.float64)
        _check(lib().smvp_tjds_export(self._h, _ptr(perm), _ptr(start_pos), _ptr(row_ind), _ptr(val)), "smvp_tjds_export")
        return perm, start_pos, row_ind, val

    def free(self):
        if self._h:
            lib().smvp_tjds_free(self._h)
            self._h = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


# ------------------------------------------------------------------ the reference's two entry points
def smvp_csr_compute(mmImportData, fInputRows, fInputNonZeros, compiter, fInputColumns=None, x=None, variant=CSR_AUTO):
    """Mirror of smvp_csr_compute (main-cli.c:325): build CSR from the COO list, run `compiter` timed
    multiplies with the ones vector (main-cli.c:368-369) unless `x` is given, return (outputVector, time data).
    The reference sizes x by rows and indexes it by column (U14); here x has fInputColumns entries
    (default: fInputRows, the reference's assumption of a square matrix)."""
    coo = _as_coo(mmImportData)[:fInputNonZeros]
    cols = fInputRows if fInputColumns is None else fInputColumns
    A = CsrMatrix.build(coo, fInputRows, cols)
    try:
        xv = np.ones(cols, np.float64) if x is None else x
        return A.mult(xv, compiter, variant)
    finally:
        A.free()


def smvp_tjds_compute(mmImportData, fInputRows, fInputColumns, fInputNonZeros, compiter, x=None, variant=TJDS_ATOMIC,
                      ref_compat=False):
    """Mirror of smvp_tjds_compute (main-cli.c:734).  ref_compat=True walks only the diagonals the shipped
    loop walks (main-cli.c:865, :1013), which is what the reference's golden TJDS reports contain."""
    coo = _as_coo(mmImportData)[:fInputNonZeros]
    A = TjdsMatrix.build(coo, fInputRows, fInputColumns)
    try:
        xv = np.ones(fInputColumns, np.float64) if x is None else x
        return A.mult(xv, compiter, variant, A.ref_diag_limit if ref_compat else 0)
    finally:
        A.free()


# ------------------------------------------------------------------ synthetic inputs (include/smvp_synth.h)
def _three_out():
    return ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_int64(0)


def synth_stencil27(nx, ny, nz, row_begin=0, row_end=None, value_mode=VAL_STENCIL, seed=0):
    """Device COO (row, col, val DeviceArrays) of rows [row_begin,row_end) of the 27-point stencil matrix."""
    total = nx * ny * nz
    row_end = total if row_end is None else row_end
    r, c, v, n = _three_out()
    _check(lib().smvp_synth_stencil27(nx, ny, nz, row_begin, row_end, value_mode, seed, ctypes.byref(r), ctypes.byref(c),
                                      ctypes.byref(v), ctypes.byref(n)), "smvp_synth_stencil27")
    return DeviceArray(r.value, n.value, "<i4"), DeviceArray(c.value, n.value, "<i4"), DeviceArray(v.value, n.value, "<f8")


def synth_stencil27_prefix(nx, ny, nz, row):
    return int(lib().smvp_synth_stencil27_prefix(nx, ny, nz, row))


def synth_rmat(scale, nedges, a=0.57, b=0.19, c=0.19, value_mode=VAL_HASH, seed=42):
    r, cc, v, n = _three_out()
    _check(lib().smvp_synth_rmat(scale, nedges, a, b, c, value_mode, seed, ctypes.byref(r), ctypes.byref(cc),
                                 ctypes.byref(v), ctypes.byref(n)), "smvp_synth_rmat")
    return DeviceArray(r.value, n.value, "<i4"), DeviceArray(cc.value, n.value, "<i4"), DeviceArray(v.value, n.value, "<f8")


def synth_vector(d_x, n, seed, stream=None):
    _check(lib().smvp_synth_vector(_ptr(d_x), n, seed, _stream(stream)), "smvp_synth_vector")


def coo_filter_device(d_row, d_col, d_val, nnz, row_lo, row_hi, col_lo, col_hi, row_shift=0, col_shift=0):
    r, c, v, n = _three_out()
    _check(lib().smvp_coo_filter_device(_ptr(d_row), _ptr(d_col), _ptr(d_val), nnz, row_lo, row_hi, col_lo, col_hi,
                                        row_shift, col_shift, ctypes.byref(r), ctypes.byref(c), ctypes.byref(v),
                                        ctypes.byref(n)), "smvp_coo_filter_device")
    return DeviceArray(r.value, n.value, "<i4"), DeviceArray(c.value, n.value, "<i4"), DeviceArray(v.value, n.value, "<f8")


def coo_histogram_device(d_row, d_col, nnz, by_col, nkeys, d_counts):
    _check(lib().smvp_coo_histogram_device(_ptr(d_row), _ptr(d_col), nnz, int(by_col), nkeys, _ptr(d_counts)),
           "smvp_coo_histogram_device")


def vector_add_device(d_y, d_a, n, stream=None):
    _check(lib().smvp_vector_add_device(_ptr(d_y), _ptr(d_a), n, _stream(stream)), "smvp_vector_add_device")


def copy_device(d_dst, d_src, nbytes, stream=None):
    _check(lib().smvp_copy_device(_ptr(d_dst), _ptr(d_src), nbytes, _stream(stream)), "smvp_copy_device")


def push_device(d_dst, d_src, nbytes, ctas=16, stream=None):
    _check(lib().smvp_push_device(_ptr(d_dst), _ptr(d_src), nbytes, ctas, _stream(stream)), "smvp_push_device")


def push_fanout_device(dst_ptrs, d_src, nbytes, ctas=16, stream=None):
    arr = (ctypes.c_void_p * len(dst_ptrs))(*[int(p) for p in dst_ptrs])
    _check(lib().smvp_push_fanout_device(arr, len(dst_ptrs), _ptr(d_src), nbytes, ctas, _stream(stream)), "smvp_push_fanout_device")


def push_tma_device(dst_ptrs, d_src, nbytes, ctas=16, stream=None):
    arr = (ctypes.c_void_p * len(dst_ptrs))(*[int(p) for p in dst_ptrs])
    _check(lib().smvp_push_tma_device(arr, len(dst_ptrs), _ptr(d_src), nbytes, ctas, _stream(stream)), "smvp_push_tma_device")


def sum_ordered_device(d_out, d_parts, nparts, stride, n, stream=None):
    _check(lib().smvp_sum_ordered_device(_ptr(d_out), _ptr(d_parts), nparts, stride, n, _stream(stream)), "smvp_sum_ordered_device")


def sum_ordered_ptrs_device(d_out, part_ptrs, n, stream=None):
    arr = (ctypes.c_void_p * len(part_ptrs))(*[int(p) for p in part_ptrs])
    _check(lib().smvp_sum_ordered_ptrs_device(_ptr(d_out), arr, len(part_ptrs), n, _stream(stream)), "smvp_sum_ordered_ptrs_device")


def flush_l2(nbytes=256 << 20, stream=None):
    _check(lib().smvp_flush_l2(nbytes, _stream(stream)), "smvp_flush_l2")
