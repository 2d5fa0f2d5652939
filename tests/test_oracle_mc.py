"""Pins the plain-C MC / block-matching port (oracle/port_mc.c) against the
real reference (src/mc.c, src/mcenc.c C kernels; the x86 SIMD twins are
bit-identical to those by the reference's own OD_CHECKASM) or the outputs recorded from it."""
import ctypes

import numpy as np
import pytest

from tests.golden.pins import OUT
from tests.oracle_lib import addr


def ref_frame(rng, h=160, w=192):
    y, x = np.mgrid[0:h, 0:w]
    img = 128 + 60 * np.sin(x / 7.0) + 40 * np.cos(y / 5.0) + rng.integers(-20, 21, size=(h, w))
    return np.clip(img, 0, 255).astype(np.uint8)


@pytest.mark.parametrize("lg", [(2, 2), (3, 3), (4, 4), (5, 5), (6, 6), (3, 2), (2, 4)])
def test_predict1fmv_port_matches_reference(port, reference, lg):
    rng = np.random.default_rng(sum(lg))
    img = ref_frame(rng)
    h, w = img.shape
    lx, ly = lg
    nx, ny = 1 << lx, 1 << ly
    for t in range(60):
        mvx, mvy = int(rng.integers(-60, 61)), int(rng.integers(-60, 61))
        if lx != ly and not (mvx & 7 or mvy & 7):
            mvx |= 1  # reference asserts square blocks on the full-pel copy path
        if t < 4:
            mvx, mvy = [(0, 0), (8, -16), (4, 0), (0, 3)][t]
            if lx != ly and t < 2:
                continue
        x0, y0 = 40 + int(rng.integers(0, 40)), 40 + int(rng.integers(0, 30))
        b = np.zeros(nx * ny, np.uint8)
        port.port_mc_predict1fmv8(addr(b), addr(img, y0 * w + x0), w, mvx, mvy, lx, ly)
        reference.out(b, "oracle_ref_mc_predict1fmv8", OUT, addr(img, y0 * w + x0), w, mvx, mvy, lx, ly, msg=(mvx, mvy))


@pytest.mark.parametrize("ln", [2, 3, 4, 5])
def test_obmc_predict_port_matches_reference(port, reference, ln):
    rng = np.random.default_rng(ln)
    img = ref_frame(rng)
    h, w = img.shape
    n = 1 << ln
    I4 = ctypes.c_int32 * 4
    for t in range(60):
        mvx = [int(v) for v in rng.integers(-40, 41, size=4)]
        mvy = [int(v) for v in rng.integers(-40, 41, size=4)]
        if t % 5 == 0:
            mvx[1], mvy[1] = mvx[0], mvy[0]
        if t % 7 == 0:
            mvx[3], mvy[3] = mvx[2], mvy[2]
        oc, s = int(rng.integers(0, 4)), int(rng.integers(0, 4))
        x0, y0 = 50, 45
        b = np.zeros((n, n + 4), np.uint8)
        port.port_mc_predict(addr(b), n + 4, addr(img, y0 * w + x0), w, I4(*mvx), I4(*mvy), oc, s, ln, ln)
        reference.out(b, "oracle_ref_mc_predict", OUT, n + 4, addr(img, y0 * w + x0), w, I4(*mvx), I4(*mvy), oc, s, ln,
                      ln, msg=(mvx, mvy, oc, s))


@pytest.mark.parametrize("ln", [2, 3, 4, 5, 6])
def test_sad_satd_port_matches_reference(port, reference, ln):
    rng = np.random.default_rng(10 + ln)
    n = 1 << ln
    for t in range(40):
        a = rng.integers(0, 256, size=(n, n + 8), dtype=np.uint8)
        b = np.clip(a.astype(int) + rng.integers(-30, 31, size=a.shape), 0, 255).astype(np.uint8)
        if t == 0:
            a[:], b[:] = 255, 0
        sad = port.port_mc_compute_sad8(addr(a), n + 8, addr(b), n + 8, n, n)
        reference.check(sad, lambda ref: getattr(ref, "od_mc_compute_sad8_%dx%d_c" % (n, n))(addr(a), n + 8, addr(b), n + 8))
        reference.check(sad, lambda ref: ref.od_mc_compute_sad8_c(addr(a), n + 8, addr(b), n + 8, n, n))
        satd = port.port_mc_compute_satd8(ln, addr(a), n + 8, addr(b), n + 8)
        reference.check(satd, lambda ref: getattr(ref, "od_mc_compute_satd8_%dx%d_c" % (n, n))(addr(a), n + 8, addr(b), n + 8))


def test_mv_grid_block_list_reproduces_reference_frame_prediction(port, reference):
    """Host logic of daala_b200/mvgrid.py (leaf walk, corner / split state, vertex selection, chroma MV
    scaling) checked on the CPU: predicting its block list with the plain-C OBMC port must give the planes
    od_state_mc_predict (src/state.c:932) produces on a real od_state."""
    from daala_b200 import mc, mvgrid
    from tests.test_gpu_mc import _frames, _random_mv_grid
    rng = np.random.default_rng(77)
    W, H = 192, 128
    _, ref_y = _frames(seed=3, h=H, w=W)
    ref_u = np.ascontiguousarray(ref_y[::2, ::2][:, ::-1])
    ref_v = np.ascontiguousarray(ref_y[1::2, 1::2])
    valid, mv = _random_mv_grid(rng, H // 8, W // 8)
    want = None
    if reference.lib is not None:
        want = [np.zeros((H, W), np.uint8), np.zeros((H // 2, W // 2), np.uint8), np.zeros((H // 2, W // 2), np.uint8)]
        rc = reference.lib.oracle_ref_state_mc_predict(W, H, addr(ref_y), addr(ref_u), addr(ref_v),
                                                       addr(np.ascontiguousarray(valid.astype(np.uint8))),
                                                       addr(np.ascontiguousarray(mv)), addr(want[0]), addr(want[1]),
                                                       addr(want[2]))
        assert rc == 0
    I4 = ctypes.c_int32 * 4
    pad = mc.OD_BUFFER_PADDING
    for pli, plane in enumerate((ref_y, ref_u, ref_v)):
        blocks = mvgrid.block_list(valid, mv, xdec=1 if pli else 0)
        src = np.pad(plane, pad, mode="edge")
        stride = src.shape[1]
        got = np.zeros_like(plane)
        w = plane.shape[1]
        for b in blocks:
            x0, y0 = int(b["x0"]), int(b["y0"])
            port.port_mc_predict(addr(got, y0 * w + x0), w, addr(src, (y0 + pad) * stride + x0 + pad), stride,
                                 I4(*[int(v) for v in b["mvx"]]), I4(*[int(v) for v in b["mvy"]]), int(b["oc"]),
                                 int(b["s"]), int(b["log_xblk"]), int(b["log_yblk"]))
        reference.check(got, want and want[pli], "plane %d" % pli)
