"""The 4096-point fused overlap-save kernel on aligned rows (ols4096i_kernel<true>), whose input and output move
between global and shared memory through bulk asynchronous copies: a launch with fewer blocks than SMs, block counts
that are not a multiple of the resident CTA slots, blocks that wrap around the end of a vector at several N mod step,
many short rows, back-to-back calls on one stream and two streams sharing one plan.

Accuracy is checked as in test_gpu_accuracy.py: against the same-precision block overlap-save peer of oracle/accuracy.py
with the default factors, and bit for bit against the unscaled result on 4^+-10 scaled inputs."""
import threading

import numpy as np
import pytest

import basic_dsp_b200 as bd
from basic_dsp_b200 import DspVec
from oracle import accuracy as acc

pytestmark = pytest.mark.gpu

F32 = np.float32


def dptr(v):
    return v._fn("bdsp_device_ptr")(v._h)


def rand_c(rng, shape):
    return (rng.uniform(-10, 10, shape) + 1j * rng.uniform(-10, 10, shape)).astype(np.complex64)


class Plan:
    def __init__(self, h):
        self.L = bd.lib()
        self.hv = DspVec(h)
        self.p = self.L.bdsp_conv_plan_create_c32(dptr(self.hv), len(h))
        assert self.p, self.L.bdsp_last_error()

    def run(self, x, out=None):
        """bdsp_convolve_signal_rows_c32 on the rows of x (16-byte aligned device buffers) -> numpy rows."""
        rows, n = x.shape
        xin = DspVec(np.ascontiguousarray(x).ravel())
        out = DspVec.zeros(2 * rows * n, is_complex=True, dtype=F32) if out is None else out
        assert self.L.bdsp_convolve_signal_rows_c32(dptr(xin), dptr(out), n, rows, self.p) == 0, self.L.bdsp_last_error()
        return out.to_numpy().reshape(rows, n)

    def close(self):
        self.L.bdsp_conv_plan_destroy(self.p)


def blocks(n, rows, taps):
    return -(-n // acc.olsi_geometry(4096, taps)[2]) * rows


# (n, rows, taps, what the case covers); all take ols4096i<true> (even N, aligned buffers, L <= 2046, N >= 4096)
CASES = [
    (4096, 1, 1023, "2 blocks: fewer blocks than SMs"),
    (4098, 2, 1023, "N mod 3072 = 1026: first and last block wrap"),
    (6146, 1, 1023, "N mod 3072 = 2: the last block holds 2 outputs"),
    (9214, 1, 1023, "N mod 3072 = 3070"),
    (11000, 3, 1023, "N mod 3072 = 1784, rows"),
    (5000, 3, 511, "511 taps (step 3584), N mod step = 1416"),
    (20000, 2, 2046, "2046 taps (step 2048): the longest response of the 4096-point block"),
    (300000, 3, 1023, "294 blocks: not a multiple of the resident CTA slots"),
    (8192, 300, 1023, "300 short rows of 3 blocks: every row's first and last block wrap"),
    (150002, 9, 1023, "441 blocks, N mod 3072 = 2546"),
]


@pytest.mark.parametrize("n,rows,taps,what", CASES, ids=["%d-x%d-L%d" % c[:3] for c in CASES])
def test_ols4096_aligned_accuracy(n, rows, taps, what):
    rng = np.random.default_rng(n * 7 + rows * 3 + taps)
    x = rand_c(rng, (rows, n))
    h = (rand_c(rng, taps) / 10).astype(np.complex64)
    assert acc.ols_block(F32, taps, True, n, rows) == (4096, "olsi")
    plan = Plan(h)
    try:
        got = plan.run(x)
        ref = acc.conv_ref(x, h, F32)
        peer = acc.ols_peer(x, h, F32, 4096, "olsi")
        rec = acc.check(got, ref, peer, F32, path="ols4096i<true> %s (%d blocks)" % (what, blocks(n, rows, taps)), tol_n=n)
        for r in (0, rows - 1):
            acc.check(got[r], ref[r], peer[r], F32, path="row %d" % r, tol_n=n)
        print(acc.format_record(rec))
        for k in (10, -10):
            s = F32(4.0) ** k
            scaled = plan.run((x * s).astype(np.complex64))
            bad = np.flatnonzero(scaled.view(F32).ravel() != (got * s).view(F32).ravel())
            assert bad.size == 0, "4^%d scaling not exact at %d elements (first flat index %d)" % (k, bad.size, bad[0])
    finally:
        plan.close()


def test_back_to_back_calls_on_one_stream_are_identical():
    """Three calls in a row on one stream (each may start while the previous one drains), 1026 blocks each."""
    rng = np.random.default_rng(11)
    n, rows, taps = 1 << 19, 6, 1023
    x = rand_c(rng, (rows, n))
    h = (rand_c(rng, taps) / 10).astype(np.complex64)
    plan = Plan(h)
    try:
        L = bd.lib()
        xin = DspVec(x.ravel())
        outs = [DspVec.zeros(2 * rows * n, is_complex=True, dtype=F32) for _ in range(3)]
        for o in outs:
            assert L.bdsp_convolve_signal_rows_c32(dptr(xin), dptr(o), n, rows, plan.p) == 0, L.bdsp_last_error()
        got = [o.to_numpy() for o in outs]
        for g in got[1:]:
            assert np.array_equal(g.view(F32), got[0].view(F32))
        peer = acc.ols_peer(x[:1], h, F32, 4096, "olsi")
        acc.check(got[0][:n], acc.conv_ref(x[:1], h, F32)[0], peer[0], F32, path="back to back row 0", tol_n=n)
    finally:
        plan.close()


def test_two_streams_share_one_plan():
    """Two threads, each on its own stream, convolve different rows with ONE plan at the same time, three times each:
    every result equals the one computed alone."""
    L = bd.lib()
    rng = np.random.default_rng(12)
    n, rows, taps = 1 << 18, 4, 1023
    xs = [rand_c(rng, (rows, n)) for _ in range(2)]
    h = (rand_c(rng, taps) / 10).astype(np.complex64)
    plan = Plan(h)
    try:
        alone = [plan.run(x) for x in xs]
        errs = []
        start = threading.Barrier(2)

        def work(i):
            try:
                st = L.bdsp_stream_create()
                L.bdsp_set_stream(st)
                start.wait()
                for _ in range(3):
                    got = plan.run(xs[i])
                    if not np.array_equal(got.view(F32), alone[i].view(F32)):
                        errs.append(i)
                L.bdsp_set_stream(None)
                L.bdsp_stream_destroy(st)
            except Exception as exc:  # noqa: BLE001
                errs.append((i, repr(exc)))

        ts = [threading.Thread(target=work, args=(i,)) for i in range(2)]
        [t.start() for t in ts]
        [t.join() for t in ts]
        assert not errs, errs
    finally:
        plan.close()
