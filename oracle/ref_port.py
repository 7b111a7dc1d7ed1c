"""ctypes loader for oracle/ref_port.c (C port of the reference's CPU convolve_signal path).
TEST / BASELINE INFRASTRUCTURE ONLY - never imported by basic_dsp_b200."""
import ctypes
import hashlib
import os
import subprocess
import tempfile

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
_BUILD = os.path.join(_HERE, "_build")
_lib = None


def _host_tag():
    try:
        with open("/proc/cpuinfo") as fh:
            for line in fh:
                if line.startswith("flags"):
                    return hashlib.sha256(line.encode()).hexdigest()[:16]
    except OSError:
        pass
    return "unknown"


def _current(out):
    """True when `out` holds a port built from the current source for this host's CPU."""
    so, tag_file = os.path.join(out, "libref_port.so"), os.path.join(out, "host_tag")
    if not os.path.exists(so) or not os.path.exists(tag_file):
        return False
    if os.path.getmtime(so) < os.path.getmtime(os.path.join(_HERE, "ref_port.c")):
        return False
    with open(tag_file) as fh:
        return fh.read() == _host_tag()


def build(force=False, out=_BUILD):
    """(Re)builds the port with -march=native into `out`; a tag file makes a box with another CPU rebuild it."""
    if force or not _current(out):
        subprocess.check_call(["make", "-C", _HERE, "-B", "OUT=" + out], stdout=subprocess.DEVNULL)
        with open(os.path.join(out, "host_tag"), "w") as fh:
            fh.write(_host_tag())
    return os.path.join(out, "libref_port.so")


def lib():
    """Loads the port built in oracle/_build, or, when that build is missing or stale, one built in a temporary
    directory: the source tree may be read-only."""
    global _lib
    if _lib is None:
        if _current(_BUILD):
            _lib = ctypes.CDLL(os.path.join(_BUILD, "libref_port.so"))
        else:
            with tempfile.TemporaryDirectory(prefix="ref_port-") as tmp:
                _lib = ctypes.CDLL(build(out=tmp))
        P = ctypes.c_void_p
        _lib.ref_convolve_signal_c32.restype = ctypes.c_int
        _lib.ref_convolve_signal_c32.argtypes = [P, ctypes.c_size_t, P, ctypes.c_size_t, P]
        _lib.ref_convolve_signal_rows_c32.restype = ctypes.c_int
        _lib.ref_convolve_signal_rows_c32.argtypes = [P, ctypes.c_size_t, ctypes.c_size_t, P, ctypes.c_size_t, ctypes.c_int]
        _lib.ref_convolve_signal_scalar_c32.restype = None
        _lib.ref_convolve_signal_scalar_c32.argtypes = [P, ctypes.c_size_t, P, ctypes.c_size_t, P]
        _lib.ref_overlap_discard_c32.restype = ctypes.c_int
        _lib.ref_overlap_discard_c32.argtypes = [P, ctypes.c_size_t, P, ctypes.c_size_t]
        _lib.ref_fft_rows_c32.restype = ctypes.c_int
        _lib.ref_fft_rows_c32.argtypes = [P, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_int, ctypes.c_int]
    return _lib


def convolve_signal_rows(x, h, threads=1):
    """x: (rows, n) complex64, h: (l,) complex64 -> centred circular convolution of every row,
    computed the way the reference's CPU path does (overlap_discard incl. its scalar head/tail)."""
    x = np.ascontiguousarray(x, dtype=np.complex64).copy()
    h = np.ascontiguousarray(h, dtype=np.complex64)
    rows, n = (1, x.shape[0]) if x.ndim == 1 else x.shape
    rc = lib().ref_convolve_signal_rows_c32(x.ctypes.data, n, rows, h.ctypes.data, len(h), threads)
    if rc:
        raise RuntimeError("ref_convolve_signal_rows_c32 -> %d" % rc)
    return x


def convolve_signal_rows_inplace(x, h, threads=1):
    rows, n = x.shape
    return lib().ref_convolve_signal_rows_c32(x.ctypes.data, n, rows, h.ctypes.data, len(h), threads)


def fft_rows(x, shift=True, threads=1):
    x = np.ascontiguousarray(x, dtype=np.complex64).copy()
    rows, n = x.shape
    rc = lib().ref_fft_rows_c32(x.ctypes.data, n, rows, 1 if shift else 0, threads)
    if rc:
        raise RuntimeError("ref_fft_rows_c32 -> %d" % rc)
    return x
