"""Pins oracle/port_tf.c (TF switching, H/V intra prediction, CfL resampling)
against the real reference (src/tf.c, src/intra.c) or the outputs recorded from it."""
import numpy as np
import pytest

from tests.golden.pins import OUT
from tests.oracle_lib import addr


@pytest.mark.parametrize("n", [4, 8, 16, 32])
def test_tf_port_matches_reference(port, reference, n):
    rng = np.random.default_rng(n)
    src = rng.integers(-3000, 3000, size=(2 * n, 2 * n + 3), dtype=np.int32)
    for name, args in (("tf_up_h_lp", (n, n)), ("tf_up_v_lp", (n, n)), ("tf_up_hv_lp", (n, n, n))):
        b = np.zeros((2 * n, 2 * n + 1), np.int32)
        getattr(port, "port_" + name)(addr(b), 2 * n + 1, addr(src), 2 * n + 3, *args)
        reference.out(b, "od_" + name, OUT, 2 * n + 1, addr(src), 2 * n + 3, *args, msg=name)
    b = np.zeros((2 * n, 2 * n), np.int32)
    port.port_tf_up_hv(addr(b), 2 * n, addr(src), 2 * n + 3, n)
    reference.out(b, "od_tf_up_hv", OUT, 2 * n, addr(src), 2 * n + 3, n)
    e = np.zeros((2 * n, 2 * n), np.int32)
    port.port_tf_down_hv(addr(e), 2 * n, addr(b), 2 * n, 2 * n)
    reference.out(e, "od_tf_down_hv", OUT, 2 * n, addr(b), 2 * n, 2 * n)
    assert np.array_equal(e, src[:2 * n, :2 * n])  # od_tf_down_hv inverts od_tf_up_hv exactly


def test_hv_intra_pred_and_cfl_resample_port_match_reference(port, reference):
    from daala_b200 import synth
    from daala_b200.frame import Geometry
    rng = np.random.default_rng(5)
    geom = Geometry(192, 128)
    bsize = synth.block_size_map(geom, "mixed", seed=1)
    w = geom.frame_w
    d = rng.integers(-2000, 2000, size=(geom.frame_h, w), dtype=np.int32)
    checked = 0
    for by4 in range(0, geom.frame_h // 4):
        for bx4 in range(0, w // 4):
            bs = int(bsize[by4 >> 1, bx4 >> 1])
            n4 = 1 << bs
            if bx4 % n4 or by4 % n4:
                continue
            n = 4 << bs
            b = np.zeros(n * n, np.int32)
            port.port_hv_intra_pred(addr(b), addr(d), w, bx4, by4, addr(bsize), bsize.shape[1], bs)
            reference.out(b, "od_hv_intra_pred", OUT, addr(d), w, bx4, by4, addr(bsize), bsize.shape[1], bs)
            checked += b.any()
    assert checked > 20
    for bs in (0, 1, 2, 3):
        n = 4 << bs
        for luma4 in ((1, 0) if bs == 0 else (0,)):
            b = np.zeros((n, n), np.int32)
            port.port_resample_luma_coeffs_420(addr(b), n, addr(d, 64 * w + 64), w, bs, luma4)
            # od_resample_luma_coeffs(chroma_pred, cpstride, decoded_luma, dlstride, xdec, ydec, bs, chroma_bs)
            reference.out(b, "od_resample_luma_coeffs", OUT, n, addr(d, 64 * w + 64), w, 1, 1, bs,
                          0 if luma4 else bs + 1, msg=(bs, luma4))
