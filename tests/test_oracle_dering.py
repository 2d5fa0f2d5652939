"""Pins oracle/port_dering.c (the oracle of the NEXT hot-path row, SURVEY.md 8(f) rank 1 -- no CUDA
twin yet) against the reference's od_dering with its C vtable (src/dering.c:252), or the outputs recorded from it."""
import ctypes

import numpy as np
import pytest

from tests.oracle_lib import addr


def _image(rng, nvsb, nhsb, sb, kind):
    h, w = nvsb * sb, nhsb * sb
    yy, xx = np.mgrid[0:h, 0:w]
    if kind == "edges":
        img = 900 * np.sign(np.sin((xx * 0.9 + yy * 0.4) / 6.0)) + 300 * np.sin(yy / 3.0)
    elif kind == "noise":
        img = rng.integers(-1500, 1500, size=(h, w))
    else:
        img = 1200 * np.sin(xx / 9.0) * np.cos(yy / 7.0)
    img = img + rng.integers(-40, 41, size=(h, w))
    return np.clip(np.round(img), -2048, 2047).astype(np.int16)


@pytest.mark.parametrize("kind", ["edges", "noise", "smooth"])
def test_direction_search_matches_reference(port, kind):
    rng = np.random.default_rng(5)
    img = _image(rng, 2, 2, 64, kind)
    stride = img.shape[1]
    # od_dir_find8 is static: reach it through od_dering's `dir` output below; here the port's own
    # invariances: a constant block has no direction contrast, a pure horizontal ramp picks direction 2
    flat = np.full((8, 8), 100 << 4, np.int16)
    var = ctypes.c_int32(-1)
    assert port.port_dering_find_direction(addr(flat), 8, ctypes.byref(var), 4) == 0 and var.value == 0
    rows = (np.arange(8)[:, None] * np.ones((1, 8)) * 160).astype(np.int16)   # constant along each row
    assert port.port_dering_find_direction(addr(rows), 8, ctypes.byref(var), 4) == 2 and var.value > 0
    cols = np.ascontiguousarray(rows.T)
    assert port.port_dering_find_direction(addr(cols), 8, ctypes.byref(var), 4) == 6 and var.value > 0
    assert img.shape[1] == stride


@pytest.mark.parametrize("kind", ["edges", "noise", "smooth"])
@pytest.mark.parametrize("xdec", [0, 1])
def test_superblock_dering_port_matches_reference(port, reference, kind, xdec):
    rng = np.random.default_rng(11 + xdec)
    nhsb, nvsb = 3, 2
    sb = 64 >> xdec
    img = _image(rng, nvsb, nhsb, sb, kind)
    h, w = img.shape
    Dir = (ctypes.c_int * 8) * 8
    skip_stride = nhsb * 16
    for threshold in (0, 19, 64, 200):
        for overlap in (0, 1):
            bskip = (rng.random((nvsb * 16, skip_stride)) < 0.5).astype(np.uint8)
            if threshold == 64:
                bskip[:] = 0
            for sby in range(nvsb):
                for sbx in range(nhsb):
                    vals = rng.integers(0, 8, size=(8, 8)) if xdec else None   # chroma reads the directions luma found
                    x0 = addr(img, sby * sb * w + sbx * sb)
                    s0 = addr(bskip, (sby * 16) * skip_stride + sbx * 16)

                    def dering(fn, *vtbl):
                        d = Dir()
                        if vals is not None:
                            for r in range(8):
                                for c in range(8):
                                    d[r][c] = int(vals[r, c])
                        y = np.zeros((sb, sb), np.int16)
                        fn(*vtbl, addr(y), sb, x0, w, 8, 8, sbx, sby, nhsb, nvsb, xdec, d, 1 if xdec else 0, s0,
                           skip_stride, threshold, overlap, 4)
                        return y, [list(r) for r in d]
                    yb, db = dering(port.port_dering)
                    reference.check((yb, db), lambda ref: dering(ref.od_dering, ctypes.c_void_p(
                        ctypes.addressof(ctypes.c_void_p.in_dll(ref, "OD_DERING_VTBL_C")))),
                        (threshold, overlap, sbx, sby))
                    if threshold == 64 and kind != "smooth":
                        assert not np.array_equal(yb, img[sby * sb:(sby + 1) * sb, sbx * sb:(sbx + 1) * sb])


def ref_dist(ref, x, y, n, qm, masking, cq):
    ref.oracle_ref_compute_dist.restype = ctypes.c_double
    return ref.oracle_ref_compute_dist(addr(x), addr(y), n, qm, masking, cq)


@pytest.mark.parametrize("n", [8, 16, 32, 64])
def test_distortion_metric_port_matches_reference(port, reference, n):
    """od_compute_dist (static, reached through oracle/ref_hooks_encode.c): bit-identical doubles -- same
    libm, same operation order."""
    rng = np.random.default_rng(n)
    port.port_compute_dist.restype = ctypes.c_double
    for t in range(12):
        x = (rng.integers(-128, 128, size=(n, n)) * 16 + rng.integers(-8, 9, size=(n, n))).astype(np.int32)
        if t % 3 == 0:
            x[:] = (x // 64) * 64                       # flat-ish regions: small window variances
        y = (x + rng.integers(-60, 61, size=(n, n)) * (1 + t % 4)).astype(np.int32)
        for qm, masking, cq in ((1, 1, 20), (1, 0, 40), (1, 1, 60), (0, 1, 20)):
            b = port.port_compute_dist(addr(x), addr(y), n, 1 if qm == 0 else 0, masking, cq)
            reference.check(b, lambda ref: ref_dist(ref, x, y, n, qm, masking, cq), (t, qm, masking, cq))
            assert b > 0, (t, qm, masking, cq)
    assert port.port_compute_dist(addr(x), addr(x), n, 0, 1, 20) == 0.0
