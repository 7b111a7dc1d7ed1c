"""basic_dsp_b200 - Python (ctypes) host binding of the B200-native basic_dsp hot path.

The product is `libbasic_dsp_b200.so` (hand-written sm_100a CUDA kernels behind the reference's
`interop` C ABI, see include/basic_dsp_b200.h).  This module is the thin host side used by the tests
and the benchmark, in the same style as the reference's own ctypes examples
(examples/basic_dsp_example.py): it declares the prototypes and wraps a handle in `DspVec`, whose
methods carry the names of the reference's vector traits (TimeToFrequencyDomainOperations::fft,
ConvolutionOps::convolve_signal, InterpolationOps::interpolatef, ...).

There is no CPU fallback: importing works everywhere (so that the symbol table can be checked on a
machine without a GPU), but every compute call needs a CUDA device and raises `DspError` otherwise.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import POINTER, Structure, c_char_p, c_double, c_float, c_int32, c_size_t, c_uint8, c_uint64, c_void_p

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("BASIC_DSP_B200_LIB", os.path.join(_HERE, "libbasic_dsp_b200.so"))

F_INVERSE, F_SHIFT, F_MAGNITUDE, F_REAL_INPUT = 1, 2, 4, 8
F_REAL_OUTPUT = 16   # bdsp_ifft_frames_*: the output holds the real parts of the synthesis as scalars
F_ONESIDED = 32         # bdsp_welch_*: real input only, points/2 + 1 bins, interior bins doubled
F_POWER_SPECTRUM = 64   # bdsp_welch_*: scaling 1/(sum w)^2 (power per bin) instead of the density 1/(fs sum w^2)


def F_WINDOW(kind):
    """bdsp_fft_rows_* flag: multiply every row by the built-in window `kind` while loading it (windowed_fft per row)."""
    return ((kind & 7) + 1) << 8
TIME, FREQ = 0, 1
SINC, RAISED_COSINE = 0, 1
TRIANGULAR, HAMMING, BLACKMAN_HARRIS, RECTANGULAR = 0, 1, 2, 3   # translate_to_window_function (interop/src/lib.rs:153-164)


class DspError(RuntimeError):
    """A C-ABI call returned a non-zero result code (see the table in include/basic_dsp_b200.h)."""

    def __init__(self, code, what):
        self.code = int(code)
        super().__init__("%s failed with result code %d%s" % (what, self.code, _last_error_suffix()))


class _VecResult(Structure):
    _fields_ = [("result_code", c_int32), ("vector", c_void_p)]


class _Complex32(Structure):
    _fields_ = [("re", c_float), ("im", c_float)]


class _Complex64(Structure):
    _fields_ = [("re", c_double), ("im", c_double)]


def _stats_struct(V):
    class _Stats(Structure):  # Statistics<T>, statistics.rs:11-31 (#[repr(C)])
        _fields_ = [("sum", V), ("count", c_size_t), ("average", V), ("rms", V), ("min", V), ("min_index", c_size_t),
                    ("max", V), ("max_index", c_size_t)]
    return _Stats


_Statistics32, _Statistics64 = _stats_struct(c_float), _stats_struct(c_double)
_ComplexStatistics32, _ComplexStatistics64 = _stats_struct(_Complex32), _stats_struct(_Complex64)


def _scalar_result(V):
    class _Scalar(Structure):  # ScalarInteropResult<T>, interop/src/lib.rs:229-242
        _fields_ = [("result_code", c_int32), ("result", V)]
    return _Scalar


_ScalarResult32, _ScalarResult64 = _scalar_result(c_float), _scalar_result(c_double)
_ComplexScalarResult32, _ComplexScalarResult64 = _scalar_result(_Complex32), _scalar_result(_Complex64)
_PointerResult = _scalar_result(c_void_p)

_lib = None


def _last_error_suffix():
    if _lib is None:
        return ""
    msg = _lib.bdsp_last_error()
    return " (%s)" % msg.decode() if msg else ""


def _declare(lib):
    H = c_void_p
    for s, T, CT in (("32", c_float, _Complex32), ("64", c_double, _Complex64)):
        RFN = ctypes.CFUNCTYPE(T, c_void_p, T)
        # ctypes cannot return structs from callbacks.  A {float, float} struct comes back in the low
        # 64 bits of xmm0 on SysV x86-64, i.e. exactly like a double with that bit pattern; the f64
        # variant ({double, double} in xmm0:xmm1) needs a native function pointer.
        CFN = ctypes.CFUNCTYPE(c_double, c_void_p, T) if s == "32" else c_void_p
        setattr(lib, "RealFn" + s, RFN)
        setattr(lib, "ComplexFn" + s, CFN)
        protos = {
            "new": (H, [c_int32, c_int32, T, c_size_t, T]),
            "new_with_performance_options": (H, [c_int32, c_int32, T, c_size_t, T, c_size_t]),
            "new_with_detailed_performance_options": (H, [c_int32, c_int32, T, c_size_t, T] + [c_size_t] * 5),
            "delete_vector": (None, [H]),
            "clone": (H, [H]),
            "get_value": (T, [H, c_size_t]),
            "set_value": (None, [H, c_size_t, T]),
            "is_complex": (c_int32, [H]),
            "get_domain": (c_int32, [H]),
            "get_len": (c_size_t, [H]),
            "set_len": (None, [H, c_size_t]),
            "get_points": (c_size_t, [H]),
            "get_delta": (T, [H]),
            "data": (POINTER(T), [H]),
            "complex_data": (POINTER(CT), [H]),
            "get_allocated_len": (c_size_t, [H]),
            "overwrite_data": (_VecResult, [H, POINTER(T), c_size_t]),
            "real_offset": (_VecResult, [H, T]),
            "real_scale": (_VecResult, [H, T]),
            "complex_offset": (_VecResult, [H, T, T]),
            "complex_scale": (_VecResult, [H, T, T]),
            "complex_divide": (_VecResult, [H, T, T]),
            "zero_pad": (_VecResult, [H, c_size_t, c_int32]),
            "zero_interleave": (_VecResult, [H, c_int32]),
            "convolve_signal": (_VecResult, [H, H]),
            "convolve": (_VecResult, [H, c_int32, T, T, c_size_t]),
            "convolve_real": (_VecResult, [H, RFN, c_void_p, c_uint8, T, c_size_t]),
            "convolve_complex": (_VecResult, [H, CFN, c_void_p, c_uint8, T, c_size_t]),
            "multiply_frequency_response": (_VecResult, [H, c_int32, T, T]),
            "multiply_frequency_response_real": (_VecResult, [H, RFN, c_void_p, c_uint8, T]),
            "multiply_frequency_response_complex": (_VecResult, [H, CFN, c_void_p, c_uint8, T]),
            "interpolatef": (_VecResult, [H, c_int32, T, T, T, c_size_t]),
            "interpolatef_custom": (_VecResult, [H, RFN, c_void_p, c_uint8, T, T, c_size_t]),
            "interpolate_lin": (_VecResult, [H, T, T]),
            "get_mag_phase": (c_int32, [H, H, H]),
        }
        for name in ("add", "sub", "div", "mul", "add_vector", "sub_vector", "div_vector", "mul_vector"):
            protos[name] = (_VecResult, [H, H])
        for name in ("apply_window", "unapply_window", "windowed_fft", "windowed_ifft"):
            protos[name] = (_VecResult, [H, c_int32])
        protos["correlate"] = (_VecResult, [H, H])
        protos["interpolatei"] = (_VecResult, [H, c_int32, T, c_int32])
        protos["interpolatei_custom"] = (_VecResult, [H, RFN, c_void_p, c_uint8, c_int32])
        protos["decimatei"] = (_VecResult, [H, ctypes.c_uint32, ctypes.c_uint32])
        protos["interpolate"] = (_VecResult, [H, c_int32, T, c_size_t, T])
        protos["interpolate_custom"] = (_VecResult, [H, RFN, c_void_p, c_uint8, c_size_t, T])
        protos["interpft"] = (_VecResult, [H, c_size_t])
        protos["multiply_complex_exponential"] = (_VecResult, [H, T, T])
        for name in ("windowed_sfft", "windowed_sifft"):
            protos[name] = (_VecResult, [H, c_int32])
        for name in ("mirror", "plain_sfft", "sfft", "plain_sifft", "sifft"):
            protos[name] = (_VecResult, [H])
        for name in ("prepare_argument", "prepare_argument_padded", "reverse"):
            protos[name] = (_VecResult, [H])
        # rest of the facade: elementwise math, reorganisation, reductions
        for name in ("sin", "cos", "tan", "asin", "acos", "atan", "sinh", "cosh", "tanh", "asinh", "acosh", "atanh", "sqrt",
                     "square", "ln", "exp", "abs", "ln_approx", "exp_approx", "sin_approx", "cos_approx", "diff",
                     "diff_with_start", "cum_sum"):
            protos[name] = (_VecResult, [H])
        for name in ("root", "powf", "log", "expf", "wrap", "unwrap", "log_approx", "expf_approx", "powf_approx"):
            protos[name] = (_VecResult, [H, T])
        for name in ("add_smaller_vector", "sub_smaller_vector", "mul_smaller_vector", "div_smaller_vector"):
            protos[name] = (_VecResult, [H, H])
        protos["get_real_imag"] = (c_int32, [H, H, H])
        protos["set_real_imag"] = (_VecResult, [H, H, H])
        protos["set_mag_phase"] = (_VecResult, [H, H, H])
        protos["split_into"] = (c_int32, [H, POINTER(c_void_p), c_size_t])
        protos["merge"] = (_VecResult, [H, POINTER(c_void_p), c_size_t])
        protos["interpolate_hermite"] = (_VecResult, [H, T, T])
        WFN = ctypes.CFUNCTYPE(T, c_void_p, c_size_t, c_size_t)
        setattr(lib, "WindowFn" + s, WFN)
        for name in ("apply_custom_window", "unapply_custom_window", "windowed_custom_fft", "windowed_custom_ifft",
                     "windowed_custom_sfft", "windowed_custom_sifft"):
            protos[name] = (_VecResult, [H, WFN, c_void_p, c_uint8])
        MAPR = ctypes.CFUNCTYPE(T, T, c_size_t)
        setattr(lib, "MapRealFn" + s, MAPR)
        protos["map_inplace_real"] = (_VecResult, [H, MAPR])
        protos["map_inplace_complex"] = (_VecResult, [H, c_void_p])      # struct-returning callback: native pointer only
        AGGM = ctypes.CFUNCTYPE(c_void_p, T, c_size_t)
        AGG = ctypes.CFUNCTYPE(c_void_p, c_void_p, c_void_p)
        setattr(lib, "MapAggregateRealFn" + s, AGGM)
        setattr(lib, "AggregateFn" + s, AGG)
        protos["map_aggregate_real"] = (_PointerResult, [H, AGGM, AGG])
        protos["map_aggregate_complex"] = (_PointerResult, [H, c_void_p, AGG])
        SR, CSR = (_ScalarResult32, _ComplexScalarResult32) if s == "32" else (_ScalarResult64, _ComplexScalarResult64)
        ST, CST = (_Statistics32, _ComplexStatistics32) if s == "32" else (_Statistics64, _ComplexStatistics64)
        protos["real_dot_product"] = (SR, [H, H])
        protos["real_dot_product_prec"] = (SR, [H, H])
        protos["complex_dot_product"] = (CSR, [H, H])
        protos["complex_dot_product_prec"] = (CSR, [H, H])
        protos["real_sum"] = (T, [H])
        protos["real_sum_sq"] = (T, [H])
        protos["complex_sum"] = (CT, [H])
        protos["complex_sum_sq"] = (CT, [H])
        protos["real_sum_prec"] = (c_double, [H])
        protos["real_sum_sq_prec"] = (c_double, [H])
        protos["complex_sum_prec"] = (_Complex64, [H])
        protos["complex_sum_sq_prec"] = (_Complex64, [H])
        protos["real_statistics"] = (ST, [H])
        protos["complex_statistics"] = (CST, [H])
        protos["real_statistics_prec"] = (_Statistics64, [H])
        protos["complex_statistics_prec"] = (_ComplexStatistics64, [H])
        protos["real_statistics_split"] = (c_int32, [H, POINTER(ST), c_size_t])
        protos["complex_statistics_split"] = (c_int32, [H, POINTER(CST), c_size_t])
        protos["real_statistics_split_prec"] = (c_int32, [H, POINTER(_Statistics64), c_size_t])
        protos["complex_statistics_split_prec"] = (c_int32, [H, POINTER(_ComplexStatistics64), c_size_t])
        for name in ("conj", "to_complex", "magnitude", "magnitude_squared", "phase", "to_real", "to_imag",
                     "plain_fft", "plain_ifft", "fft", "ifft", "swap_halves", "fft_shift", "ifft_shift"):
            protos[name] = (_VecResult, [H])
        for name in ("get_magnitude", "get_magnitude_squared", "get_phase", "get_real", "get_imag"):
            protos[name] = (c_int32, [H, H])
        for name, (res, args) in protos.items():
            fn = getattr(lib, name + s)
            fn.restype, fn.argtypes = res, args
        ext = {
            "bdsp_upload": (c_int32, [H, POINTER(T), c_size_t]),
            "bdsp_download": (c_int32, [H, POINTER(T), c_size_t]),
            "bdsp_download_async": (c_int32, [H, POINTER(T), c_size_t]),
            "bdsp_device_ptr": (c_void_p, [H]),
            "bdsp_scale_mul_mag_phase": (c_int32, [H, T, T, H, H, H, c_int32]),
            "bdsp_fft_magnitude": (_VecResult, [H]),
        }
        for name, (res, args) in ext.items():
            fn = getattr(lib, name + s)
            fn.restype, fn.argtypes = res, args
        for name in ("bdsp_fft_rows_c", "bdsp_convolve_signal_rows_c", "bdsp_conv_plan_create_c"):
            pass
    lib.bdsp_version.restype, lib.bdsp_version.argtypes = c_char_p, []
    lib.bdsp_last_error.restype, lib.bdsp_last_error.argtypes = c_char_p, []
    lib.bdsp_device_count.restype, lib.bdsp_device_count.argtypes = c_int32, []
    lib.bdsp_set_device.restype, lib.bdsp_set_device.argtypes = c_int32, [c_int32]
    lib.bdsp_sync.restype, lib.bdsp_sync.argtypes = c_int32, []
    lib.bdsp_set_stream.restype, lib.bdsp_set_stream.argtypes = None, [c_void_p]
    lib.bdsp_stream_create.restype, lib.bdsp_stream_create.argtypes = c_void_p, []
    lib.bdsp_stream_destroy.restype, lib.bdsp_stream_destroy.argtypes = None, [c_void_p]
    lib.bdsp_stream_sync.restype, lib.bdsp_stream_sync.argtypes = c_int32, [c_void_p]
    for s in ("32", "64"):
        f = getattr(lib, "bdsp_fft_rows_c" + s)
        f.restype, f.argtypes = c_int32, [c_void_p, c_void_p, c_size_t, c_size_t, c_int32]
        for name in ("bdsp_fft_frames_c", "bdsp_ifft_frames_c"):
            f = getattr(lib, name + s)
            f.restype, f.argtypes = c_int32, [c_void_p, c_void_p, c_size_t, c_size_t, c_size_t, c_int32]
        f = getattr(lib, "bdsp_welch_c" + s)
        f.restype, f.argtypes = c_int32, [c_void_p, c_void_p, c_size_t, c_size_t, c_size_t, c_int32, c_float if s == "32" else c_double]
        f = getattr(lib, "bdsp_conv_plan_create_c" + s)
        f.restype, f.argtypes = c_void_p, [c_void_p, c_size_t]
        f = getattr(lib, "bdsp_convolve_signal_rows_c" + s)
        f.restype, f.argtypes = c_int32, [c_void_p, c_void_p, c_size_t, c_size_t, c_void_p]
    lib.bdsp_conv_plan_destroy.restype, lib.bdsp_conv_plan_destroy.argtypes = None, [c_void_p]
    lib.bdsp_malloc.restype, lib.bdsp_malloc.argtypes = c_void_p, [c_size_t]
    lib.bdsp_free.restype, lib.bdsp_free.argtypes = None, [c_void_p]
    lib.bdsp_mem_free.restype, lib.bdsp_mem_free.argtypes = c_size_t, []
    for sfx, T in (("32", c_float), ("64", c_double)):
        for name in ("bdsp_magnitude_rows_c", "bdsp_magnitude_squared_rows_c", "bdsp_phase_rows_c"):
            fn = getattr(lib, name + sfx)
            fn.restype, fn.argtypes = c_int32, [c_void_p, c_void_p, c_size_t, c_size_t]
        fn = getattr(lib, "bdsp_scale_mul_mag_phase_rows_c" + sfx)
        fn.restype, fn.argtypes = c_int32, [c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_size_t, T, T, c_int32]
        fn = getattr(lib, "bdsp_interpolatef_rows" + sfx)
        fn.restype, fn.argtypes = c_int32, [c_void_p, c_void_p, c_size_t, c_size_t, c_int32, c_int32, T, T, T, c_size_t, POINTER(c_size_t)]
    lib.bdsp_malloc_host.restype, lib.bdsp_malloc_host.argtypes = c_void_p, [c_size_t]
    lib.bdsp_free_host.restype, lib.bdsp_free_host.argtypes = None, [c_void_p]
    lib.bdsp_memcpy_h2d.restype, lib.bdsp_memcpy_h2d.argtypes = c_int32, [c_void_p, c_void_p, c_size_t]
    lib.bdsp_memcpy_d2h.restype, lib.bdsp_memcpy_d2h.argtypes = c_int32, [c_void_p, c_void_p, c_size_t]
    lib.bdsp_memset.restype, lib.bdsp_memset.argtypes = c_int32, [c_void_p, c_int32, c_size_t]
    lib.bdsp_event_create.restype, lib.bdsp_event_create.argtypes = c_void_p, []
    lib.bdsp_event_destroy.restype, lib.bdsp_event_destroy.argtypes = None, [c_void_p]
    lib.bdsp_event_record.restype, lib.bdsp_event_record.argtypes = c_int32, [c_void_p]
    lib.bdsp_event_elapsed_ms.restype, lib.bdsp_event_elapsed_ms.argtypes = c_float, [c_void_p, c_void_p]
    lib.bdsp_kernel_launch_count.restype, lib.bdsp_kernel_launch_count.argtypes = c_uint64, []


def lib():
    """The loaded C-ABI library.  Raises if libbasic_dsp_b200.so has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                "basic_dsp_b200: %s is missing - build it with `python -m basic_dsp_b200.build` "
                "(there is no CPU fallback)" % LIB_PATH)
        loaded = ctypes.CDLL(LIB_PATH)
        _declare(loaded)
        _lib = loaded
    return _lib


def device_count():
    return int(lib().bdsp_device_count())


def require_device():
    if device_count() < 1:
        raise DspError(-1000, "basic_dsp_b200: no CUDA device available (no CPU fallback)")


def synchronize():
    rc = lib().bdsp_sync()
    if rc:
        raise DspError(rc, "bdsp_sync")


def kernel_launch_count():
    return int(lib().bdsp_kernel_launch_count())


def _check(res, what):
    if res.result_code != 0:
        raise DspError(res.result_code, what)
    return res.vector


class DspVec:
    """A device-resident vector behind an `InteropVec` handle (GenDspVec semantics: real/complex and
    time/frequency are run-time properties).  Methods mirror the reference's trait methods; the ones
    that consume `self` in Rust (fft, magnitude, ...) mutate this object in place and return it."""

    def __init__(self, data=None, *, is_complex=None, domain=TIME, delta=1.0, dtype=None, _handle=None, _suffix=None):
        L = lib()
        if _handle is not None:
            self._s = _suffix
            self._h = _handle
            return
        require_device()
        arr = np.asarray(data)
        if is_complex is None:
            is_complex = np.iscomplexobj(arr)
        if dtype is None:
            dtype = np.float64 if arr.dtype in (np.float64, np.complex128) else np.float32
        self._s = "64" if np.dtype(dtype) == np.float64 else "32"
        flat = self._flatten(arr, is_complex)
        self._h = getattr(L, "new" + self._s)(1 if is_complex else 0, domain, 0.0, flat.size, delta)
        self.upload(flat)

    # -- plumbing ---------------------------------------------------------------------------------
    @property
    def _T(self):
        return np.float64 if self._s == "64" else np.float32

    @property
    def _cT(self):
        return c_double if self._s == "64" else c_float

    def _fn(self, name):
        return getattr(lib(), name + self._s)

    def _flatten(self, arr, is_complex):
        T = self._T
        if np.iscomplexobj(arr):
            ct = np.complex128 if T == np.float64 else np.complex64
            return np.ascontiguousarray(arr.astype(ct)).view(T).ravel()
        return np.ascontiguousarray(arr.astype(T)).ravel()

    def _call(self, name, *args):
        res = self._fn(name)(self._h, *args)
        self._h = res.vector  # callers continue with the returned pointer (interop/src/lib.rs:203-212)
        if res.result_code != 0:
            raise DspError(res.result_code, name + self._s)
        return self

    def result_code_of(self, name, *args):
        """Runs a mutating C-ABI call and returns its result code instead of raising."""
        args = [a._h if isinstance(a, DspVec) else a for a in args]
        res = self._fn(name)(self._h, *args)
        self._h = res.vector
        return int(res.result_code)

    def __del__(self):
        try:
            if getattr(self, "_h", None):
                self._fn("delete_vector")(self._h)
                self._h = None
        except Exception:
            pass

    # -- host access -------------------------------------------------------------------------------
    def upload(self, flat):
        flat = np.ascontiguousarray(flat, dtype=self._T)
        rc = self._fn("bdsp_upload")(self._h, flat.ctypes.data_as(POINTER(self._cT)), flat.size)
        if rc:
            raise DspError(rc, "bdsp_upload" + self._s)
        return self

    def to_numpy(self):
        """Copy of the data: complex array (one element per point) or real array."""
        n = self.len()
        out = np.empty(n, dtype=self._T)
        rc = self._fn("bdsp_download")(self._h, out.ctypes.data_as(POINTER(self._cT)), n)
        if rc:
            raise DspError(rc, "bdsp_download" + self._s)
        if self.is_complex():
            return out.view(np.complex128 if self._s == "64" else np.complex64)
        return out

    def data_via_host_mirror(self):
        """data32()/data64(): pointer into the synchronised host mirror, copied out."""
        n = self.len()
        p = self._fn("data")(self._h)
        return np.ctypeslib.as_array(p, shape=(max(n, 1),))[:n].copy()

    # -- meta data (Vector<T>, MetaData) --------------------------------------------------------------
    def len(self):
        return int(self._fn("get_len")(self._h))

    def points(self):
        return int(self._fn("get_points")(self._h))

    def is_complex(self):
        return bool(self._fn("is_complex")(self._h))

    def domain(self):
        return int(self._fn("get_domain")(self._h))

    def delta(self):
        return float(self._fn("get_delta")(self._h))

    def alloc_len(self):
        return int(self._fn("get_allocated_len")(self._h))

    def set_len(self, n):
        self._fn("set_len")(self._h, n)

    def get_value(self, i):
        return float(self._fn("get_value")(self._h, i))

    def set_value(self, i, v):
        self._fn("set_value")(self._h, i, v)

    def clone(self):
        return DspVec(_handle=self._fn("clone")(self._h), _suffix=self._s)

    @classmethod
    def zeros(cls, length, *, is_complex=False, domain=TIME, delta=1.0, dtype=np.float32, init=0.0):
        require_device()
        s = "64" if np.dtype(dtype) == np.float64 else "32"
        h = getattr(lib(), "new" + s)(1 if is_complex else 0, domain, init, length, delta)
        return cls(_handle=h, _suffix=s)

    # -- TimeToFrequencyDomainOperations / FrequencyToTimeDomainOperations ------------------------------
    def plain_fft(self):
        return self._call("plain_fft")

    def fft(self):
        return self._call("fft")

    def plain_ifft(self):
        return self._call("plain_ifft")

    def ifft(self):
        return self._call("ifft")

    def fft_magnitude(self):
        """fft(&mut buffer).magnitude() in one kernel."""
        return self._call("bdsp_fft_magnitude")

    # -- FrequencyDomainOperations / ReorganizeDataOps ----------------------------------------------------
    def fft_shift(self):
        return self._call("fft_shift")

    def ifft_shift(self):
        return self._call("ifft_shift")

    def swap_halves(self):
        return self._call("swap_halves")

    def zero_pad(self, points, option=0):
        return self._call("zero_pad", points, option)

    def zero_interleave(self, factor):
        return self._call("zero_interleave", factor)

    def to_complex(self):
        return self._call("to_complex")

    # -- ConvolutionOps / Convolution / FrequencyMultiplication ---------------------------------------------
    def convolve_signal(self, impulse_response):
        return self._call("convolve_signal", impulse_response._h)

    def convolve(self, impulse_response, rolloff, ratio, length):
        """Built-in responses (SINC / RAISED_COSINE) or a Python callable x -> float."""
        if callable(impulse_response):
            cb = getattr(lib(), "RealFn" + self._s)(lambda _d, x: float(impulse_response(x)))
            return self._call("convolve_real", cb, None, 1, ratio, length)
        return self._call("convolve", impulse_response, rolloff, ratio, length)

    def convolve_complex(self, fn, ratio, length):
        """`fn`: Python callable x -> complex (f32 vectors only, see _declare) or a native function
        pointer (int / c_void_p) of type BdspComplexFn32/64."""
        if callable(fn):
            if self._s != "32":
                raise TypeError("Python complex callbacks are only supported for f32 vectors")

            pyfn = fn

            def _cb(_d, x):
                c = complex(pyfn(x))
                return float(np.array([c.real, c.imag], dtype=np.float32).view(np.float64)[0])
            native = getattr(lib(), "ComplexFn32")(_cb)
            return self._call("convolve_complex", native, None, 0, ratio, length)
        return self._call("convolve_complex", fn, None, 0, ratio, length)

    def multiply_frequency_response(self, frequency_response, rolloff, ratio):
        if callable(frequency_response):
            cb = getattr(lib(), "RealFn" + self._s)(lambda _d, x: float(frequency_response(x)))
            return self._call("multiply_frequency_response_real", cb, None, 1, ratio)
        return self._call("multiply_frequency_response", frequency_response, rolloff, ratio)

    # -- InterpolationOps / RealInterpolationOps --------------------------------------------------------------
    def interpolatef(self, impulse_response, rolloff, factor, delay, length):
        if callable(impulse_response):
            cb = getattr(lib(), "RealFn" + self._s)(lambda _d, x: float(impulse_response(x)))
            return self._call("interpolatef_custom", cb, None, 1, factor, delay, length)
        return self._call("interpolatef", impulse_response, rolloff, factor, delay, length)

    def interpolate_lin(self, factor, delay):
        return self._call("interpolate_lin", factor, delay)

    # -- next rows (SURVEY 8f): TimeDomainOperations, CrossCorrelation*Ops, reverse, decimatei ----------------------
    def apply_window(self, window):
        return self._call("apply_window", window)

    def unapply_window(self, window):
        return self._call("unapply_window", window)

    def windowed_fft(self, window):
        return self._call("windowed_fft", window)

    def windowed_ifft(self, window):
        return self._call("windowed_ifft", window)

    def prepare_argument(self):
        return self._call("prepare_argument")

    def prepare_argument_padded(self):
        return self._call("prepare_argument_padded")

    def correlate(self, prepared):
        return self._call("correlate", prepared._h)

    def interpolatei(self, frequency_response, rolloff, factor, is_symmetric=True):
        if callable(frequency_response):
            cb = getattr(lib(), "RealFn" + self._s)(lambda _d, x: float(frequency_response(x)))
            return self._call("interpolatei_custom", cb, None, 1 if is_symmetric else 0, factor)
        return self._call("interpolatei", frequency_response, rolloff, factor)

    def interpolate(self, frequency_response, rolloff, dest_points, delay, is_symmetric=True):
        """InterpolationOps::interpolate; frequency_response None = interpft."""
        if frequency_response is None:
            return self._call("interpft", dest_points)
        if callable(frequency_response):
            cb = getattr(lib(), "RealFn" + self._s)(lambda _d, x: float(frequency_response(x)))
            return self._call("interpolate_custom", cb, None, 1 if is_symmetric else 0, dest_points, delay)
        return self._call("interpolate", frequency_response, rolloff, dest_points, delay)

    def interpft(self, dest_points):
        return self._call("interpft", dest_points)

    def multiply_complex_exponential(self, a, b):
        return self._call("multiply_complex_exponential", a, b)

    # SymmetricTimeToFrequencyDomainOperations / SymmetricFrequencyToTimeDomainOperations / mirror
    def mirror(self):
        return self._call("mirror")

    def plain_sfft(self):
        return self._call("plain_sfft")

    def sfft(self):
        return self._call("sfft")

    def windowed_sfft(self, window):
        return self._call("windowed_sfft", window)

    def plain_sifft(self):
        return self._call("plain_sifft")

    def sifft(self):
        return self._call("sifft")

    def windowed_sifft(self, window):
        return self._call("windowed_sifft", window)

    def reverse(self):
        return self._call("reverse")

    # -- rest of the facade: TrigOps / PowerOps / RealOps / ModuloOps / ApproximatedOps / DiffSumOps ------------------
    def math(self, name, *args):
        """sin, cos, tan, asin, acos, atan, sinh, cosh, tanh, asinh, acosh, atanh, sqrt, square, ln, exp, abs,
        root(d), powf(e), log(base), expf(base), wrap(d), unwrap(d), *_approx, diff, diff_with_start, cum_sum."""
        return self._call(name, *args)

    def add_smaller(self, o):
        return self._call("add_smaller_vector", o._h)

    def sub_smaller(self, o):
        return self._call("sub_smaller_vector", o._h)

    def mul_smaller(self, o):
        return self._call("mul_smaller_vector", o._h)

    def div_smaller(self, o):
        return self._call("div_smaller_vector", o._h)

    def get_real_imag(self, real, imag):
        return self._fn("get_real_imag")(self._h, real._h, imag._h)

    def set_real_imag(self, real, imag):
        return self._call("set_real_imag", real._h, imag._h)

    def set_mag_phase(self, mag, phase):
        return self._call("set_mag_phase", mag._h, phase._h)

    def split_into(self, targets):
        arr = (c_void_p * len(targets))(*[t._h for t in targets])
        return int(self._fn("split_into")(self._h, arr, len(targets)))

    def merge(self, sources):
        arr = (c_void_p * len(sources))(*[t._h for t in sources])
        return self._call("merge", arr, len(sources))

    def interpolate_hermite(self, factor, delay):
        return self._call("interpolate_hermite", factor, delay)

    def custom_window(self, name, fn, is_symmetric=True):
        """apply_custom_window / unapply_custom_window / windowed_custom_{fft,ifft,sfft,sifft} with fn(i, points)."""
        cb = getattr(lib(), "WindowFn" + self._s)(lambda _d, i, p: float(fn(i, p)))
        return self._call(name, cb, None, 1 if is_symmetric else 0)

    def map_inplace(self, fn):
        cb = getattr(lib(), "MapRealFn" + self._s)(lambda v, i: float(fn(v, i)))
        return self._call("map_inplace_real", cb)

    # -- reductions: DotProductOps / SumOps / StatisticsOps (+ _prec, + _split) -----------------------------------------
    def _kind(self):
        return "complex" if self.is_complex() else "real"

    def dot_product(self, o, prec=False):
        r = self._fn(self._kind() + "_dot_product" + ("_prec" if prec else ""))(self._h, o._h)
        if r.result_code != 0:
            raise DspError(r.result_code, "dot_product" + self._s)
        return complex(r.result.re, r.result.im) if self.is_complex() else float(r.result)

    def sum(self, prec=False, squared=False):
        r = self._fn(self._kind() + ("_sum_sq" if squared else "_sum") + ("_prec" if prec else ""))(self._h)
        return complex(r.re, r.im) if self.is_complex() else float(r)

    @staticmethod
    def _stats_dict(st, cplx):
        conv = (lambda c: complex(c.re, c.im)) if cplx else float
        return dict(sum=conv(st.sum), count=int(st.count), average=conv(st.average), rms=conv(st.rms), min=conv(st.min),
                    min_index=int(st.min_index), max=conv(st.max), max_index=int(st.max_index))

    def statistics(self, prec=False):
        st = self._fn(self._kind() + "_statistics" + ("_prec" if prec else ""))(self._h)
        return self._stats_dict(st, self.is_complex())

    def statistics_split(self, parts, prec=False):
        fn = self._fn(self._kind() + "_statistics_split" + ("_prec" if prec else ""))
        arr = (fn.argtypes[1]._type_ * max(parts, 1))()
        rc = fn(self._h, arr, parts)
        if rc != 0:
            raise DspError(rc, "statistics_split" + self._s)
        return [self._stats_dict(arr[i], self.is_complex()) for i in range(parts)]

    def decimatei(self, factor, delay):
        return self._call("decimatei", factor, delay)

    # -- ScaleOps / OffsetOps / ElementaryOps -----------------------------------------------------------------
    def scale(self, c):
        if isinstance(c, complex):
            return self._call("complex_scale", c.real, c.imag)
        return self._call("real_scale", c)

    def offset(self, c):
        if isinstance(c, complex):
            return self._call("complex_offset", c.real, c.imag)
        return self._call("real_offset", c)

    def add(self, other):
        return self._call("add", other._h)

    def sub(self, other):
        return self._call("sub", other._h)

    def mul(self, other):
        return self._call("mul", other._h)

    def div(self, other):
        return self._call("div", other._h)

    def conj(self):
        return self._call("conj")

    # -- ComplexToRealTransformsOps / ComplexToRealGetterOps ----------------------------------------------------
    def magnitude(self):
        return self._call("magnitude")

    def magnitude_squared(self):
        return self._call("magnitude_squared")

    def phase(self):
        return self._call("phase")

    def to_real(self):
        return self._call("to_real")

    def to_imag(self):
        return self._call("to_imag")

    def get_magnitude(self, dest):
        return int(self._fn("get_magnitude")(self._h, dest._h))

    def get_phase(self, dest):
        return int(self._fn("get_phase")(self._h, dest._h))

    def get_mag_phase(self, mag, phase):
        return int(self._fn("get_mag_phase")(self._h, mag._h, phase._h))

    def scale_mul_mag_phase(self, c, w, mag, phase, write_back=False):
        """Fused scale(c) -> mul(&w) -> get_mag_phase in one pass over memory."""
        c = complex(c)
        rc = self._fn("bdsp_scale_mul_mag_phase")(self._h, c.real, c.imag, w._h, mag._h, phase._h, 1 if write_back else 0)
        if rc:
            raise DspError(rc, "bdsp_scale_mul_mag_phase" + self._s)
        return mag, phase
