"""Per-element and exact-tap tests of every interpolation kernel (csrc/interp.cu) at its tile, edge and wrap-around shapes.

Every case names the kernel it targets and the condition in interp_poly / interpf_shape / interp_lin that selects it.
  * Exact taps (polyphase paths): the input is zeros plus impulses of small distinct integer amplitude, at least 2L + 4
    apart, so every output sees at most one nonzero sample and is one product of an impulse with a host-built tap: it
    must equal the float64 / long double reference cast to T value for value, and every output no impulse reaches must
    be zero.  A wrong table, window offset or wrap shows at the exact output where it happens.
  * Accuracy (all interpolatef paths): uniform input in [-10, 10), oracle.accuracy.check against the reference (taps
    in T, sums in float64 / long double) and the peer (the same sums in T, taps in ascending window order), then the
    4^k scaling of test_gpu_accuracy.py bit for bit.
  * Rows: bdsp_interpolatef_rows* on 1 and 3 rows equals the per-vector interpolatef byte for byte, leaves 64 sentinels
    on each side of the output intact, and does so with `in` and `out` one element past a 16-byte boundary as well.
  * interpolate_lin: the tail, clamp and tie shapes, bit for bit against the oracle.

Run with -s to see the records of profiles/r3_interp_accuracy.txt."""
import ctypes

import numpy as np
import pytest

import basic_dsp_b200 as bd
from basic_dsp_b200 import DspVec
from oracle import accuracy as acc
from oracle import dsp_oracle as o
from test_gpu_accuracy import Buf, assert_scaled_exact, check_rows, rand_c

pytestmark = pytest.mark.gpu

F32, F64 = np.float32, np.float64
RC = 0.25   # raised-cosine rolloff: with delay 0 a tap lands on the special point |x| = 1 / (2 rolloff) = 2


def poly_kernel(dtype, cplx, F):
    """(kernel, input positions per CTA or None, selecting condition) of interp_poly."""
    T = "float" if dtype == F32 else "double"
    if F > 8:
        return "interp_poly_generic_kernel<%s,%s>" % (T, str(cplx).lower()), None, "interp_poly: F > 8"
    if cplx:
        return (("interp_poly_tiled_kernel<%s,true,4,2>" % T, 512, "interp_poly: complex, F <= 4") if F <= 4 else
                ("interp_poly_tiled_kernel<%s,true,8,1>" % T, 256, "interp_poly: complex, 5 <= F <= 8"))
    if dtype == F32:
        return (("interp_poly_f32_kernel", 512, "interp_poly: real f32, F <= 4") if F <= 4 else
                ("interp_poly_tiled_kernel<float,false,8,2>", 512, "interp_poly: real f32, 5 <= F <= 8"))
    return (("interp_poly_tiled_kernel<double,false,4,4>", 1024, "interp_poly: real f64, F <= 4") if F <= 4 else
            ("interp_poly_tiled_kernel<double,false,8,2>", 512, "interp_poly: real f64, 5 <= F <= 8"))


# (dtype, complex, N, factor, conv_len, delay, kind, shape): polyphase cases (interpf_shape: L = min(conv_len, points/2)
# <= 202, new_len >= 2000, integer factor)
POLY = []


def pc(dtype, cplx, N, F, L, delay, kind, shape):
    POLY.append((dtype, cplx, N, float(F), L, delay, kind, shape))


for _dt in (F32, F64):
    for _cx in (False, True):
        for _F in ((1, 2, 3, 4, 5, 8) if not _cx else (1, 2, 4, 5, 8)):
            _tile = poly_kernel(_dt, _cx, _F)[1]
            _min = -(-2000 // (_F * (2 if _cx else 1)))            # new_len >= 2000
            if _F in (4, 5) or (_F == 8 and _cx):
                # the full shape list on the main factor of each kernel
                if _tile >= _min:
                    pc(_dt, _cx, _tile, _F, 12, 0.0, 0, "one tile, all edge")
                pc(_dt, _cx, 3 * _tile, _F, 12, 0.0, 1, "N = 3 tiles")
                pc(_dt, _cx, 3 * _tile + 1, _F, 12, 0.3, 0, "N = 3 tiles + 1")
                pc(_dt, _cx, 3 * _tile - 1, _F, 12, 0.0, 0, "N = 3 tiles - 1")
                pc(_dt, _cx, 3 * _tile + 12, _F, 12, -0.2, 1, "trailing edge straddles the last two tiles")
                for _L in (0, 1, 3):
                    pc(_dt, _cx, 2 * _tile + 3, _F, _L, 0.0, _L % 2, "L = %d (remainder taps, read-ahead clamp)" % _L)
                pc(_dt, _cx, 4 * _tile + 5, _F, 202, 0.0, 1, "L = 202" + (", leading edge longer than a tile" if 405 > _tile else ""))
                pc(_dt, _cx, 4 * _tile + 5, _F, 202, 0.45, 0, "L = 202, delay")
            else:
                pc(_dt, _cx, max(_min, 2 * _tile + 7), _F, 12, 0.0, 1, "F = %d" % _F)
    # windows longer than the vector (2L + 3 > N): the window wraps
    pc(_dt, False, 404, 5, 202, 0.0, 0, "window longer than the vector")
    pc(_dt, False, 405, 8, 202, 0.1, 1, "window longer than the vector")
    pc(_dt, True, 250, 4, 125, 0.0, 1, "window longer than the vector")
    pc(_dt, True, 128, 8, 64, 0.0, 0, "window longer than the vector")
    # real odd N, odd F: new_points = N F + 1, one output past N F
    pc(_dt, False, 1537, 3, 12, 0.0, 1, "odd N, odd F: output N F")
    pc(_dt, False, 1025, 5, 30, 0.2, 0, "odd N, odd F: output N F")
    pc(_dt, False, 1023, 7, 3, 0.0, 1, "odd N, odd F: output N F")
    # F > 8: one thread per output
    pc(_dt, False, 301, 9, 12, 0.0, 0, "F = 9")
    pc(_dt, False, 223, 9, 202, 0.0, 1, "F = 9, odd N, window longer than the vector")
    pc(_dt, True, 300, 16, 40, -0.3, 1, "F = 16")
    pc(_dt, False, 1000, 16, 202, 0.0, 0, "F = 16, L = 202")
    pc(_dt, True, 70, 16, 3, 0.0, 0, "F = 16, L = 3")

# (dtype, complex, N, factor, conv_len, delay, kind, shape): per-output cases (interp_frac_kernel)
FRAC = [
    (F32, False, 900, 2.5, 12, 0.0, 0, "non-integer factor"),
    (F32, True, 700, 13.0 / 6.0, 10, 0.25, 1, "non-integer factor"),
    (F32, False, 1500, 3.0, 250, 0.0, 0, "integer factor, conv_len > 202"),
    (F32, True, 300, 3.0, 12, 0.0, 1, "integer factor, new_len < 2000"),
    (F32, False, 3000, 0.5, 10, 0.0, 1, "factor < 1"),
    (F32, False, 1001, 2.5, 12, 0.0, 0, "tie: new_len = round(2502.5) = 2503 -> 2504"),
    (F32, True, 1001, 2.25, 12, 0.0, 1, "tie: new_len = round(4504.5) = 4505 -> 4506"),
    (F64, False, 900, 2.5, 12, 0.1, 0, "non-integer factor"),
    (F64, True, 700, 13.0 / 6.0, 10, 0.0, 1, "non-integer factor"),
    (F64, True, 1500, 2.0, 230, 0.0, 1, "integer factor, conv_len > 202"),
    (F64, False, 3000, 0.25, 10, 0.0, 0, "factor < 1"),
    (F64, False, 1001, 2.5, 12, 0.0, 1, "tie: new_len = round(2502.5) = 2503 -> 2504"),
    (F64, True, 1001, 2.25, 12, 0.0, 0, "tie: new_len = round(4504.5) = 4505 -> 4506"),
]

def _id(c):
    return "%s-%s-N%d-F%g-L%d-d%g-%s" % ("f32" if c[0] == F32 else "f64", "c" if c[1] else "r", c[2], c[3], c[4], c[5],
                                         "sinc" if c[6] == 0 else "rc")


def path_of(c):
    dtype, cplx, N, factor, L, _, _, shape = c
    if c in FRAC:
        return "interp_frac_kernel<%s,%s> (%s)" % ("float" if dtype == F32 else "double", str(cplx).lower(), shape), \
            "interpf_shape: not polyphase"
    k, _, cond = poly_kernel(dtype, cplx, int(factor))
    return "%s (%s)" % (k, shape), cond


def gpu_interpf(x, c):
    dtype, cplx, N, factor, L, delay, kind, _ = c
    return DspVec(x.astype(acc.ctype(dtype) if cplx else dtype)).interpolatef(kind, RC, factor, delay, L).to_numpy()


def rand_x(rng, c):
    return rand_c(rng, c[2], c[0]) if c[1] else rng.uniform(-10, 10, c[2]).astype(c[0])


EXACT = [c for c in POLY if c[2] >= 2 * min(c[4], c[2] // 2) + 4]


@pytest.mark.parametrize("case", EXACT, ids=[_id(c) for c in EXACT])
def test_poly_exact_taps(case):
    dtype, cplx, N, factor, conv_len, delay, kind, shape = case
    L = min(conv_len, N // 2)
    tile = poly_kernel(dtype, cplx, int(factor))[1] or N // 2
    pos = [0, 1, L, 2 * L + 1, tile - 1, tile, tile + 1, N - L - 1, N - 2, N - 1]
    for gi, group in enumerate(acc.impulse_groups(N, L, pos)):
        x = np.zeros(N, dtype=acc.ctype(dtype) if cplx else dtype)
        for k, p in enumerate(group):
            a = (k + 1 + gi) * (-1) ** k
            x[p] = complex(a, -(k + 2)) if cplx else a
        got = gpu_interpf(x, case)
        ref, _, poly = acc.interpf_pair(x, kind, RC, factor, delay, conv_len, dtype)
        assert poly
        want = ref.astype(got.dtype)
        bad = np.flatnonzero(got != want)
        assert bad.size == 0, "%s: impulses at %s: %d outputs differ, first %d: got %r want %r" % (
            path_of(case)[0], group, bad.size, bad[0], got[bad[0]], want[bad[0]])
    print("exact taps   %-80s ok" % path_of(case)[0])


@pytest.mark.parametrize("case", POLY + FRAC, ids=[_id(c) for c in POLY + FRAC])
def test_interpf_accuracy(case):
    dtype, cplx, N, factor, conv_len, delay, kind, shape = case
    rng = np.random.default_rng(N * 31 + int(factor * 8) + conv_len)
    x = rand_x(rng, case)
    got = gpu_interpf(x, case)
    ref, peer, poly = acc.interpf_pair(x, kind, RC, factor, delay, conv_len, dtype)
    assert poly == (case in POLY)
    assert len(got) == len(ref)
    # every path stays within the default K_rel = 4, K_el = 8 (worst measured ratio 1.5, profiles/r3_interp_accuracy.txt)
    check_rows(got, ref, peer, dtype, path_of(case)[0])
    assert_scaled_exact(lambda xs: gpu_interpf(xs, case), x, got, dtype)


# one case per kernel: (case, condition)
ROWS = []
_seen = set()
for _c in sorted(POLY + FRAC, key=lambda c: c[7] != "N = 3 tiles + 1"):   # the main factor of each kernel first
    _k = path_of(_c)[0].split(" (")[0]
    if _k not in _seen and _c[2] >= 2 * min(_c[4], _c[2] // 2) + 4:
        _seen.add(_k)
        ROWS.append(_c)


def gpu_rows(x, c, off, sentinel):
    """bdsp_interpolatef_rows* on the rows of x; returns (rows of output, the 64 elements before and after them)."""
    dtype, cplx, N, factor, conv_len, delay, kind, _ = c
    rows = x.shape[0]
    n = ctypes.c_size_t(0)
    fn = getattr(bd.lib(), "bdsp_interpolatef_rows" + ("32" if dtype == F32 else "64"))
    assert fn(None, None, N, 0, int(cplx), kind, RC, factor, delay, conv_len, ctypes.byref(n)) == 0
    npts = n.value
    pad = np.full(64, sentinel, dtype=x.dtype)
    xin = Buf(x, off, dtype)
    out = Buf(np.concatenate([pad, np.zeros(rows * npts, dtype=x.dtype), pad]), off, dtype)
    rc = fn(xin.ptr, out.ptr + 64 * out.esize, N, rows, int(cplx), kind, RC, factor, delay, conv_len, ctypes.byref(n))
    assert rc == 0 and n.value == npts, bd.lib().bdsp_last_error()
    full = out.get(-1)
    return full[64:-64].reshape(rows, npts), np.concatenate([full[:64], full[-64:]])


@pytest.mark.parametrize("off", [0, 1], ids=["aligned", "offset"])
@pytest.mark.parametrize("rows", [1, 3])
@pytest.mark.parametrize("case", ROWS, ids=[_id(c) for c in ROWS])
def test_interpf_rows(case, rows, off):
    rng = np.random.default_rng(case[2] + rows)
    x = np.stack([rand_x(rng, case) for _ in range(rows)])
    sentinel = x.dtype.type(complex(-1234.5, 777.25) if case[1] else -1234.5)
    got, pads = gpu_rows(x, case, off, sentinel)
    assert np.all(pads == sentinel), "%s: output sentinels overwritten" % path_of(case)[0]
    for r in range(rows):
        want = gpu_interpf(x[r], case)
        assert got[r].tobytes() == want.tobytes(), "%s row %d (offset %d)" % (path_of(case)[0], r, off)
    print("rows x%d %-7s %-80s ok" % (rows, "offset" if off else "aligned", path_of(case)[0]))


# (dtype, n, factor, delay, shape); f32 with a power-of-two factor and an aligned output (every DspVec) runs
# interp_lin_pow2_f32_kernel, everything else interp_lin_kernel.  Residues are of dest_len - 1 mod 4.
LIN = []
for _dt in (F32, F64):
    for _n in (101, 102, 103, 104):
        LIN.append((_dt, _n, 1.0, 0.0, "dest_len - 1 = %d (mod 4 = %d)" % (_n - 1, (_n - 1) % 4)))
        LIN.append((_dt, _n, 3.0, 0.25, "dest_len - 1 = %d (mod 4 = %d)" % (3 * (_n - 1), 3 * (_n - 1) % 4)))
    for _F in (4.0, 3.0, 1.0, 0.125, 0.3):
        LIN.append((_dt, 2, _F, 0.0, "n = 2"))
    LIN += [(_dt, 81, 0.125, 0.0, "factor 2^-3"), (_dt, 8001, 0.125, 0.0, "factor 2^-3"), (_dt, 1000, 0.3, 0.0, "factor < 1"),
            (_dt, 500, 2.0, -1.5, "delay clamps the read index at the start"), (_dt, 500, 3.0, -2.25, "delay clamps at the start"),
            (_dt, 500, 2.0, 2.5, "delay clamps the read index at the end"), (_dt, 500, 2.5, 3.75, "delay clamps at the end"),
            (_dt, 998, 2.5, 0.0, "tie: dest_len = round(2492.5) + 1 = 2494")]


def lin_kernel(dtype, factor):
    m, _ = np.frexp(np.float32(factor))
    return "interp_lin_pow2_f32_kernel" if dtype == F32 and m == 0.5 else "interp_lin_kernel<%s>" % np.dtype(dtype).name


@pytest.mark.parametrize("dtype,n,factor,delay,shape", LIN,
                         ids=["%s-n%d-F%g-d%g" % (np.dtype(c[0]).name, c[1], c[2], c[3]) for c in LIN])
def test_interpolate_lin_shapes(dtype, n, factor, delay, shape):
    rng = np.random.default_rng(n)
    x = rng.uniform(-10, 10, n).astype(dtype)
    got = DspVec(x).interpolate_lin(factor, delay).to_numpy()
    want = o.interpolate_lin(x, factor, delay, dtype)
    assert len(got) == len(want)
    bad = np.flatnonzero(got.view(dtype) != want)
    assert bad.size == 0, "%s %s: %d outputs differ, first %d" % (lin_kernel(dtype, factor), shape, bad.size, bad[0])
    print("lin bit-exact %-28s n=%-5d factor %-6g delay %-5g dest_len %-6d %s" % (lin_kernel(dtype, factor), n, factor, delay,
                                                                                   len(got), shape))
