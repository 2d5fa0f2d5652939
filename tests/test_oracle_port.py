"""Pins the plain-C oracle port (oracle/port_*.c) against the real reference
(oracle/_ref/libdaala_ref.so = unmodified xiph/daala sources, or the outputs recorded from it:
tests/golden/pins.py), and against the reference's own self-consistency checks
(src/dct.c:8825-8906 check_transform, :8300-8328 ieee1180 round trip, src/filter.c:1624-1698 TEST main)."""
import ctypes

import numpy as np
import pytest

from tests.golden.pins import OUT
from tests.oracle_lib import addr

SIZES = [2, 3, 4, 5, 6]  # log2 n


def rand_blocks(rng, n, count, lo=-2048, hi=2047):
    return rng.integers(lo, hi + 1, size=(count, n, n), dtype=np.int32)


@pytest.mark.parametrize("ln", SIZES)
def test_fdct_idct_1d_port_matches_reference(port, reference, ln):
    n = 1 << ln
    rng = np.random.default_rng(ln)
    for t in range(200):
        x = rng.integers(-4096, 4096, size=n, dtype=np.int32)
        if t == 0:
            x[:] = 4095
        if t == 1:
            x[:] = np.where(np.arange(n) % 2, -4096, 4095)
        y_port = np.zeros(n, np.int32)
        port.port_bin_fdct(ln, addr(y_port), addr(x), 1)
        reference.out(y_port, "od_bin_fdct%d" % n, OUT, addr(x), 1)
        x_port = np.zeros(n, np.int32)
        port.port_bin_idct(ln, addr(x_port), 1, addr(y_port))
        reference.out(x_port, "od_bin_idct%d" % n, OUT, 1, addr(y_port))
        assert np.array_equal(x_port, x)  # reversible (dct.c:8825 check_transform)


@pytest.mark.parametrize("ln", SIZES)
def test_dct_2d_port_matches_reference(port, reference, ln):
    n = 1 << ln
    rng = np.random.default_rng(100 + ln)
    for x in rand_blocks(rng, n, 20):
        x = np.ascontiguousarray(x)
        y_port = np.zeros((n, n), np.int32)
        port.port_bin_fdct2d(ln, addr(y_port), n, addr(x), n)
        reference.out(y_port, "od_bin_fdct%dx%d" % (n, n), OUT, n, addr(x), n)
        x_port = np.zeros((n, n), np.int32)
        port.port_bin_idct2d(ln, addr(x_port), n, addr(y_port), n)
        reference.out(x_port, "od_bin_idct%dx%d" % (n, n), OUT, n, addr(y_port), n)
        assert np.array_equal(x_port, x)


@pytest.mark.parametrize("ln", [1, 2, 3, 4, 5, 6])
def test_haar_port_matches_reference_and_is_lossless(port, reference, ln):
    """od_haar / od_haar_inv (src/dct.c:4822/:4861), strided in and out; the wavelet is exactly invertible."""
    n = 1 << ln
    rng = np.random.default_rng(300 + ln)
    for t in range(10):
        x = np.zeros((n, n + 3), np.int32)
        x[:, :n] = rng.integers(-(1 << 14), 1 << 14, size=(n, n))
        y_port = np.zeros((n, n + 1), np.int32)
        port.port_haar(addr(y_port), n + 1, addr(x), n + 3, ln)
        reference.out(y_port, "od_haar", OUT, n + 1, addr(x), n + 3, ln)
        x_port = np.zeros((n, n + 2), np.int32)
        port.port_haar_inv(addr(x_port), n + 2, addr(y_port), n + 1, ln)
        reference.out(x_port, "od_haar_inv", OUT, n + 2, addr(y_port), n + 1, ln)
        assert np.array_equal(x_port[:, :n], x[:, :n])


def test_filter4_port_matches_reference_and_inverts(port, reference):
    rng = np.random.default_rng(7)
    for t in range(2000):
        x = rng.integers(-40000, 40000, size=4, dtype=np.int32)
        y_port = np.zeros(4, np.int32)
        port.port_pre_filter4(addr(y_port), addr(x))
        reference.out(y_port, "od_pre_filter4", OUT, addr(x))
        x_port = np.zeros(4, np.int32)
        port.port_post_filter4(addr(x_port), addr(y_port))
        reference.out(x_port, "od_post_filter4", OUT, addr(y_port))
        assert np.array_equal(x_port, x)  # filter.c:1624 TEST main: post(pre(x)) == x


@pytest.mark.parametrize("xdec", [0, 1])
def test_frame_sb_filters_port_matches_reference(port, reference, xdec):
    rng = np.random.default_rng(11 + xdec)
    nhsb, nvsb = 3, 2
    w, h = (nhsb * 64) >> xdec, (nvsb * 64) >> xdec
    c = rng.integers(-2048, 2048, size=(h, w), dtype=np.int32)
    b = c.copy()
    port.port_apply_prefilter_frame_sbs(addr(b), w, nhsb, nvsb, xdec, xdec)
    pre = b.copy()

    def ref_pre(lib):
        a = c.copy()
        lib.od_apply_prefilter_frame_sbs(addr(a), w, nhsb, nvsb, xdec, xdec)
        return a
    reference.check(b, ref_pre)
    assert not np.array_equal(b, c)
    port.port_apply_postfilter_frame_sbs(addr(b), w, nhsb, nvsb, xdec, xdec)

    def ref_post(lib):
        a = pre.copy()
        lib.od_apply_postfilter_frame_sbs(addr(a), w, nhsb, nvsb, xdec, xdec, 0, None, 0)
        return a
    reference.check(b, ref_post)
    assert np.array_equal(b, c)


@pytest.mark.parametrize("bs", [1, 2, 3, 4])
@pytest.mark.parametrize("hv", [(1, 1), (1, 0), (0, 1)])
def test_split_filters_port_matches_reference(port, reference, bs, hv):
    rng = np.random.default_rng(bs)
    n = 4 << bs
    stride = n + 8
    c = rng.integers(-2048, 2048, size=(n, stride), dtype=np.int32)
    b = c.copy()
    port.port_prefilter_split(addr(b), stride, bs, hv[0], hv[1])
    pre = b.copy()

    def ref_pre(lib):
        a = c.copy()
        lib.od_prefilter_split(addr(a), stride, bs, 0, hv[0], hv[1])
        return a
    reference.check(b, ref_pre)
    port.port_postfilter_split(addr(b), stride, bs, hv[0], hv[1])

    def ref_post(lib):
        a = pre.copy()
        lib.od_postfilter_split(addr(a), stride, bs, 0, 0, None, 0, hv[0], hv[1])
        return a
    reference.check(b, ref_post)
    assert np.array_equal(b, c)


@pytest.mark.parametrize("n", [8, 16, 32])
def test_large_filters_port_matches_reference_and_inverts(port, reference, n):
    """od_pre/post_filter8/16/32 (dead in the codec, exported for dcttest/tools)."""
    rng = np.random.default_rng(n)
    for t in range(500):
        x = rng.integers(-30000, 30000, size=n, dtype=np.int32)
        yb = np.zeros(n, np.int32)
        port.port_pre_filter_n(n, addr(yb), addr(x))
        reference.out(yb, "od_pre_filter%d" % n, OUT, addr(x))
        xb = np.zeros(n, np.int32)
        port.port_post_filter_n(n, addr(xb), addr(yb))
        reference.out(xb, "od_post_filter%d" % n, OUT, addr(yb))
        assert np.array_equal(xb, x)
