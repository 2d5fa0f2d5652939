"""Pins the plain-C PVQ port (oracle/port_pvq.c) against the real reference
(static pvq_theta / pvq_search_rdo_double of src/pvq_encoder.c reached through
oracle/ref_hooks_pvq.c, and the exported src/pvq.c functions), or the outputs recorded from it."""
import ctypes

import numpy as np
import pytest

from tests import pvq_cases
from tests.golden.pins import OUT
from tests.oracle_lib import addr


def test_fixed_point_helpers_match_reference(port, reference):
    rng = np.random.default_rng(3)
    ref = reference.lib
    if ref is not None:
        for fn in (ref.od_pvq_cos, ref.od_pvq_sin):
            fn.restype = ctypes.c_int16  # od_val16
    for x in list(range(-70000, 70000, 997)) + [0, 32768, 65536, 98304, 131072]:
        reference.check(np.int16(port.port_pvq_cos(x)), lambda ref: np.int16(ref.od_pvq_cos(x)))
        reference.check(np.int16(port.port_pvq_sin(x)), lambda ref: np.int16(ref.od_pvq_sin(x)))
    for beta in (4096, 6144, 5000):
        for cg0 in [0, 1, 100, 256, 300, 1000, 5000, 20000]:
            for q0 in (8, 64, 400, 1100):
                reference.check(port.port_gain_expand(cg0, q0, beta), lambda ref: ref.od_gain_expand(cg0, q0, beta),
                                (cg0, q0, beta))
        for qcg in range(0, 5000, 37):
            reference.check(port.port_pvq_compute_max_theta(qcg, beta),
                            lambda ref: ref.od_pvq_compute_max_theta(qcg, beta))
        for n in (15, 8, 32, 128):
            for qcg in range(0, 6000, 101):
                reference.check(port.port_pvq_compute_k(qcg, -1, 1, n, beta),
                                lambda ref: ref.od_pvq_compute_k(qcg, -1, -1, 1, n, beta, 1))
            for it in range(0, 40):
                reference.check(port.port_pvq_compute_k(512, it, 0, n, beta),
                                lambda ref: ref.od_pvq_compute_k(512, it, 0, 0, n, beta, 1))
    for ts in range(0, 30):
        for t in range(0, 30):
            reference.check(port.port_pvq_compute_theta(t, ts), lambda ref: ref.od_pvq_compute_theta(t, ts))
    for n in (15, 8, 32, 128):
        for _ in range(50):
            x = rng.integers(-3000, 3000, size=n).astype(np.int16)
            for beta in (4096, 6144):
                for q0 in (8, 100, 900):
                    def gain(fn, *speed):
                        g = ctypes.c_int32(0)
                        return fn(addr(x), n, q0, ctypes.byref(g), beta, *speed), g.value
                    reference.check(gain(port.port_pvq_compute_gain, 2), lambda ref: gain(ref.od_pvq_compute_gain, 2))
            x32 = (x.astype(np.int32) * 37)
            reference.check(port.port_vector_log_mag(addr(x32), n), lambda ref: ref.od_vector_log_mag(addr(x32), n))
            r = rng.integers(-3000, 3000, size=n).astype(np.int16)
            gr = int(np.sqrt(float((r.astype(np.int64) ** 2).sum())))

            def householder(fn, *extra):
                rr, sgn = r.copy(), ctypes.c_int(0)
                return fn(addr(rr), n, gr, ctypes.byref(sgn), *extra), sgn.value, rr
            hb = householder(port.port_compute_householder, 0)
            reference.check(hb, lambda ref: householder(ref.od_compute_householder, 0))
            ob = np.zeros(n, np.int16)
            port.port_apply_householder(addr(ob), addr(x), addr(hb[2]), n)
            reference.out(ob, "od_apply_householder", OUT, addr(x), addr(hb[2]), n)


def test_pulse_search_matches_reference(port, reference):
    rng = np.random.default_rng(4)
    port.port_pvq_search_rdo_double.restype = ctypes.c_double
    if reference.lib is not None:
        reference.lib.oracle_ref_pvq_search_rdo_double.restype = ctypes.c_double
    for n in (15, 8, 32, 128, 14, 7, 31, 127):
        for t in range(40):
            x = np.round(rng.laplace(0, 400, size=n) * np.exp(-np.arange(n) / (n / 3))).astype(np.int16)
            ya, yb = np.zeros(n, np.int32), np.zeros(n, np.int32)
            prev = 0
            for k in sorted(set(int(v) for v in rng.integers(1, 40, size=3))):
                g2 = float(rng.uniform(0.5, 50))

                def ref_search(ref):
                    # the search continues from the pulses of the previous K (prev): ya holds the reference's
                    c = ref.oracle_ref_pvq_search_rdo_double(addr(x), n, k, addr(ya), ctypes.c_double(g2),
                                                            ctypes.c_double(0.147), prev)
                    return ya.copy(), c
                cb = port.port_pvq_search_rdo_double(addr(x), n, k, addr(yb), ctypes.c_double(g2),
                                                     ctypes.c_double(0.147), prev)
                reference.check((yb, cb), ref_search)
                assert np.abs(yb).sum() == k
                prev = k


def test_pvq_theta_port_matches_reference(port, reference):
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    count = 0
    nonskip = 0
    withref = 0
    for c in pvq_cases.cases(seed=1, per_combo=8):
        b = pvq_cases.run_theta(port, "port", c, qm, qm_inv)
        key = (c["n"], c["kind"], c["is_keyframe"], c["pli"], c["beta"], c["q0"])
        reference.check(b, lambda ref: pvq_cases.run_theta(ref, "ref", c, qm, qm_inv), key)
        count += 1
        nonskip += b["k"] > 0
        withref += b["itheta"] > 0
    assert count > 1000 and nonskip > 300 and withref > 100, (count, nonskip, withref)


def test_frame_pvq_driver_port_matches_reference(port, reference):
    """oracle/pipeline_driver.inc compiled against the port and against the
    real reference functions must quantise a whole plane identically."""
    from daala_b200 import synth
    from daala_b200.frame import Geometry
    from tests import frame_oracle
    geom = Geometry(192, 128)
    planes, _ = synth.frame(192, 128, f=1)
    planes = synth.pad_planes(planes, geom)
    prev, _ = synth.frame(192, 128, f=0, seed=99)
    prev = synth.pad_planes(prev, geom)
    bsize = synth.block_size_map(geom, "mixed", seed=2)
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    q4 = np.full((3, 30), 24, np.uint8)
    for is_keyframe in (1, 0):
        for pli in range(3):
            # the planes both drivers quantise: the reference's forward transform (the port's is pinned in
            # tests/test_oracle_port.py)
            d = frame_oracle.forward_plane(port, "port", planes[pli], geom, pli, bsize, is_keyframe)
            reference.check(d, lambda ref: frame_oracle.forward_plane(ref, "ref", planes[pli], geom, pli, bsize,
                                                                      is_keyframe))
            md = frame_oracle.forward_plane(port, "port", prev[pli], geom, pli, bsize, 0) if not is_keyframe else None
            if md is not None:
                reference.check(md, lambda ref: frame_oracle.forward_plane(ref, "ref", prev[pli], geom, pli, bsize, 0))
            b, sb = frame_oracle.pvq_plane(port, "port", d, md, geom, pli, bsize, 38, is_keyframe, 1, 0.147, qm, qm_inv, q4)
            reference.check((b, sb), lambda ref: frame_oracle.pvq_plane(ref, "ref", d, md, geom, pli, bsize, 38,
                                                                        is_keyframe, 1, 0.147, qm, qm_inv, q4))
            assert sb[0] > 0 and not np.array_equal(b, d)


def test_keyframe_prediction_driver_port_matches_reference(port, reference):
    """Luma H/V intra prediction + chroma CfL inside the frame PVQ driver."""
    from daala_b200 import synth
    from daala_b200.frame import Geometry
    from tests import frame_oracle
    geom = Geometry(192, 128)
    planes, _ = synth.frame(192, 128, f=1)
    planes = synth.pad_planes(planes, geom)
    bsize = synth.block_size_map(geom, "mixed", seed=2)
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    q4 = np.full((3, 30), 20, np.uint8)

    def luma(lib, prefix):
        d0 = frame_oracle.forward_plane(lib, prefix, planes[0], geom, 0, bsize, 1)
        return frame_oracle.pvq_plane_pred(lib, prefix, d0, geom, 0, bsize, 45, 1, 0.147, qm, qm_inv, q4)
    got = luma(port, "port")
    reference.check(got, lambda ref: luma(ref, "ref"))
    nopred = frame_oracle.pvq_plane(port, "port", frame_oracle.forward_plane(port, "port", planes[0], geom, 0, bsize, 1),
                                    None, geom, 0, bsize, 45, 1, 1, 0.147, qm, qm_inv, q4)
    assert not np.array_equal(nopred[0], got[0])  # the prediction changes decisions
    assert got[1][2] > -got[1][3]  # some bands chose a reference (itheta >= 0)
    for pli in (1, 2):
        def chroma(lib, prefix):
            # each driver predicts chroma from its own quantised luma (equal, as checked above)
            dc = frame_oracle.forward_plane(lib, prefix, planes[pli], geom, pli, bsize, 1)
            return frame_oracle.pvq_plane_pred(lib, prefix, dc, geom, pli, bsize, 45, 1, 0.147, qm, qm_inv, q4,
                                               luma_d=got[0])
        reference.check(chroma(port, "port"), lambda ref: chroma(ref, "ref"))


def test_full_4k_frame_port_matches_reference(port, reference):
    """BASELINE.json's frame size (3840x2160, padded to 3840x2176): the whole keyframe chain of the frame
    drivers -- forward, PVQ with intra / CfL prediction, inverse -- port vs reference, all three planes."""
    import zlib
    from daala_b200 import synth
    from daala_b200.frame import Geometry
    from tests import frame_oracle
    geom = Geometry(3840, 2160)
    planes, _ = synth.frame(3840, 2160, f=1)
    planes = synth.pad_planes(planes, geom)
    bsize = synth.block_size_map(geom, "mixed", seed=21)
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    q4 = np.full((3, 30), 16, np.uint8)

    def chain(lib, prefix):
        luma_q = None
        out = []
        for pli in range(3):
            d = frame_oracle.forward_plane(lib, prefix, planes[pli], geom, pli, bsize, 1)
            dq, stats = frame_oracle.pvq_plane_pred(lib, prefix, d, geom, pli, bsize, 72, 1, 0.147, qm, qm_inv, q4,
                                                    luma_d=luma_q)
            if pli == 0:
                luma_q = dq
            rec = frame_oracle.inverse_plane(lib, prefix, dq, geom, pli, bsize, 1)
            out += [zlib.crc32(d.tobytes()), zlib.crc32(dq.tobytes()), zlib.crc32(rec.tobytes()), int(stats[0])]
        return out
    got = chain(port, "port")
    reference.check(got, lambda ref: chain(ref, "ref"))
    assert got[3] > 100000     # coded pulses on the luma plane


@pytest.mark.parametrize("content", ["flat128", "noise", "black", "white"])
def test_edge_content_frames_port_matches_reference(port, reference, content):
    """SURVEY.md 8(d) edge cases: a flat-128 frame (every AC coefficient zero: all-skip paths), saturated
    frames and a pure-noise frame (large K everywhere) through the whole keyframe chain."""
    from daala_b200 import synth
    from daala_b200.frame import Geometry
    from tests import frame_oracle
    geom = Geometry(200, 136)
    rng = np.random.default_rng(3)
    planes = []
    for pli in range(3):
        h, w = (136, 200) if pli == 0 else (68, 100)
        if content == "flat128":
            p = np.full((h, w), 128, np.uint8)
        elif content == "black":
            p = np.zeros((h, w), np.uint8)
        elif content == "white":
            p = np.full((h, w), 255, np.uint8)
        else:
            p = rng.integers(0, 256, size=(h, w), dtype=np.uint8)
        planes.append(p)
    planes = synth.pad_planes(planes, geom)
    bsize = synth.block_size_map(geom, "mixed", seed=8)
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    q4 = np.full((3, 30), 16, np.uint8)

    def chain(lib, prefix):
        luma_q = None
        out = []
        for pli in range(3):
            d = frame_oracle.forward_plane(lib, prefix, planes[pli], geom, pli, bsize, 1)
            dq, stats = frame_oracle.pvq_plane_pred(lib, prefix, d, geom, pli, bsize, 30, 1, 0.147, qm, qm_inv, q4,
                                                    luma_d=luma_q)
            if pli == 0:
                luma_q = dq
            rec = frame_oracle.inverse_plane(lib, prefix, dq, geom, pli, bsize, 1)
            out.append((d, dq, rec, stats))
        return out
    res = {"port": chain(port, "port")}
    for pli in range(3):
        reference.check(res["port"][pli], lambda ref: chain(ref, "ref")[pli], pli)
    res["ref"] = res["port"]      # equal to the reference's, as checked
    pulses = sum(int(o[3][0]) for o in res["ref"])
    if content == "noise":
        assert pulses > 20000
    elif content == "flat128":
        assert pulses == 0
        for pli in range(3):        # mid-grey is the transform's zero: it survives the lossy chain exactly
            assert np.array_equal(res["ref"][pli][2], planes[pli])
    else:
        # saturated constants: the lapping filters are gated at the picture edge (src/filter.c:1459), which
        # leaves a little AC there; the reconstruction stays within the quantiser's reach
        assert pulses < 500
        for pli in range(3):
            assert np.abs(res["ref"][pli][2].astype(int) - planes[pli].astype(int)).max() <= 8


def test_real_encoder_block_sizes_through_the_frame_drivers(port, reference):
    """Block sizes decided by the WHOLE reference encoder (oracle_ref_encode_keyframe: public API, complexity 7
    RDO) instead of a synthetic quadtree: the list builders agree on that map and the frame drivers of the
    port and of the reference produce identical planes with it."""
    from daala_b200 import pvq, synth
    from daala_b200.frame import Geometry
    from tests import frame_oracle
    w, h = 960, 540
    geom = Geometry(w, h)
    src, _ = synth.frame(w, h, f=4)

    def encode(ref):
        bsize = np.zeros(geom.bsize_shape, np.uint8)
        dering = np.zeros((geom.nvsb, geom.nhsb), np.uint8)
        nbytes, csum = ctypes.c_long(0), ctypes.c_uint(0)
        quant = 20
        rc = ref.oracle_ref_encode_keyframe(w, h, addr(np.ascontiguousarray(src[0])), addr(np.ascontiguousarray(src[1])),
                                            addr(np.ascontiguousarray(src[2])), quant, 7, addr(bsize), addr(dering),
                                            ctypes.byref(nbytes), ctypes.byref(csum))
        assert rc == 0 and nbytes.value > 1000
        return bsize
    bsize = reference.value("bsize", encode)
    assert bsize.max() <= 4 and len(np.unique(bsize)) >= 2
    # quadtree consistency of the decided map: a block of size L covers units that all carry L
    blocks = pvq.block_list(bsize, geom)
    for pli in range(3):
        cover = np.zeros(geom.plane_shape(pli), np.int32)
        for b in blocks[blocks["pli"] == pli]:
            n = 4 << int(b["bs"])
            cover[b["y0"]:b["y0"] + n, b["x0"]:b["x0"] + n] += 1
        assert (cover == 1).all()
    nat = pvq.native_keyframe_lists([bsize], geom)
    luma, top, left, depth = pvq.sort_by_depth(pvq.raster_order(blocks[blocks["pli"] == 0]), [bsize], geom)
    assert np.array_equal(nat["dep_top"], top) and np.array_equal(nat["depth"], depth)
    planes = synth.pad_planes(src, geom)
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    q4 = np.full((3, 30), 16, np.uint8)

    def chain(lib, prefix):
        luma_q = None
        res = []
        for pli in range(3):
            d = frame_oracle.forward_plane(lib, prefix, planes[pli], geom, pli, bsize, 1)
            dq, stats = frame_oracle.pvq_plane_pred(lib, prefix, d, geom, pli, bsize, 72, 1, 0.147, qm, qm_inv, q4,
                                                    luma_d=luma_q)
            if pli == 0:
                luma_q = dq
            res += [d, dq, frame_oracle.inverse_plane(lib, prefix, dq, geom, pli, bsize, 1)]
        return res
    got = chain(port, "port")
    want = chain(reference.lib, "ref") if reference.lib is not None else [None] * len(got)
    for g, w_ in zip(got, want):
        reference.check(g, w_)
