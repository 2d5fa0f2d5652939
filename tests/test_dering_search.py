"""The deringing level search (reference src/encode.c:2680-2811; csrc/dering_search.cu).

CPU: the host decision daala_b200_dering_decide (context modelling, adaptive-CDF rate, strict-less choice, CDF
update) against the reference's own od_encode_cdf_cost / od_encode_cdf_adapt driven by
oracle/ref_hooks_encode.c::oracle_ref_dering_search, on the distortions the reference computed, over a chain
of frames long enough for the CDFs to go through their halving step.
GPU: the whole search (5 plane filters + 6 distortion passes on the device, decision on the host) against the
same reference driver: distortions to 1e-12 relative (CUDA pow vs glibc pow), levels identical wherever the
reference's two best scores are further apart than that tolerance (everywhere, on these inputs), CDFs identical.
"""
import ctypes

import numpy as np
import pytest

from tests.oracle_lib import addr

LEVELS = 6
DERING_LAMBDA_SCALE = 0.67 * 0.147      # src/rate.c:1086: 0.67 * OD_PVQ_LAMBDA * q^2


def synth_pair(rng, nhsb, nvsb, ring):
    """Source luma and a 'reconstruction' (od_coeff, x16 scale): smooth shapes plus edges, the reconstruction
    with edge-following ringing of a strength that varies across the frame, so different superblocks prefer
    different levels."""
    h, w = nvsb * 64, nhsb * 64
    yy, xx = np.mgrid[0:h, 0:w]
    img = 110 + 50 * np.sin(xx / 37.0) * np.cos(yy / 23.0)
    img += 60 * (((xx // 48) + (yy // 40)) % 2)
    img += 30 * ((xx + 2 * yy) % 97 < 30)
    src = np.clip(img + rng.normal(0, 1.5, img.shape), 0, 255).astype(np.uint8)
    strength = ring * (0.2 + 1.8 * (np.sin(xx / 211.0 + 1) ** 2) * (np.cos(yy / 173.0) ** 2))
    noise = rng.normal(0, 1, img.shape)
    noise = noise + np.roll(noise, 1, 1) - np.roll(noise, 2, 0)
    ctmp = ((src.astype(np.int32) - 128) << 4) + np.rint(16 * strength * noise).astype(np.int32)
    ctmp = np.clip(ctmp, -2048, 2047).astype(np.int32)
    return np.ascontiguousarray(src), np.ascontiguousarray(ctmp)


def ref_search(ref, src, ctmp, nhsb, nvsb, q, masking, keyframe, lam, bskip, cdf, increment=128, qm=1):
    nsb = nhsb * nvsb
    levels = np.zeros(nsb, np.uint8)
    dist = np.zeros((LEVELS, nsb), np.float64)
    ref.oracle_ref_dering_search.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p] + [ctypes.c_int] * 7 + [
        ctypes.c_double, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    r = ref.oracle_ref_dering_search(addr(src), src.shape[1], addr(ctmp), nhsb, nvsb, q, q, qm, masking, keyframe, lam,
                                     addr(bskip) if bskip is not None else None,
                                     bskip.shape[1] if bskip is not None else 0, addr(cdf), increment, addr(levels), addr(dist))
    assert r == 0
    return levels, dist


def lib_decide():
    from daala_b200 import _native
    L = _native.lib()
    L.daala_b200_dering_decide.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_double,
                                           ctypes.c_void_p, ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p]
    L.daala_b200_dering_cdf_init.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    return L


def coded_flags(bskip, nhsb, nvsb):
    return np.ascontiguousarray((bskip.reshape(nvsb, 16, nhsb, 16) == 0).any(axis=(1, 3)).astype(np.uint8).ravel())


@pytest.mark.parametrize("keyframe", [1, 0])
def test_decision_matches_reference_cdf_model(keyframe, reference):
    L = lib_decide()
    rng = np.random.default_rng(5 + keyframe)
    nhsb, nvsb = 7, 5
    cdf_ref = np.zeros((2 * LEVELS - 1, LEVELS), np.uint16)
    inc = ctypes.c_int(0)
    L.daala_b200_dering_cdf_init(addr(cdf_ref), ctypes.byref(inc))
    assert inc.value == 128 and cdf_ref[3].tolist() == [32, 64, 96, 128, 160, 192]     # src/state.c:573-574
    cdf_ours = cdf_ref.copy()
    seen = set()
    halved = False
    for frame in range(36 if keyframe else 12):
        q = [72, 38, 140, 20][frame % 4]
        src, ctmp = synth_pair(rng, nhsb, nvsb, ring=[0.6, 2.5, 1.2][frame % 3] * q / 72.0)
        bskip = None
        if frame % 3 == 2:
            bskip = (rng.random((nvsb * 16, nhsb * 16)) < 0.5).astype(np.uint8)
            bskip[16:32, 32:64] = 1            # two superblocks with every block skipped: not searched, not coded
            bskip = np.ascontiguousarray(bskip)
        lam = DERING_LAMBDA_SCALE * q * q
        before = cdf_ours[:, -1].copy()
        search = {}

        def ref_dist(ref):
            # the reference's search runs frame after frame on its own CDFs (cdf_ref)
            search["lv"], dist = ref_search(ref, src, ctmp, nhsb, nvsb, q, frame & 1, keyframe, lam, bskip, cdf_ref)
            return dist
        dist = np.ascontiguousarray(reference.value("dist%d" % frame, ref_dist))
        lv = np.zeros(nhsb * nvsb, np.uint8)
        coded = coded_flags(bskip, nhsb, nvsb) if bskip is not None else None
        r = L.daala_b200_dering_decide(addr(dist), nhsb, nvsb, keyframe, lam, addr(coded) if coded is not None else None,
                                       addr(cdf_ours), 128, addr(lv))
        assert r == 0
        reference.check(lv, search.get("lv"), frame)
        reference.check(cdf_ours, cdf_ref, frame)
        halved |= bool((cdf_ours[:, -1] < before).any())
        if bskip is not None:
            assert lv.reshape(nvsb, nhsb)[1, 2] == 0 and lv.reshape(nvsb, nhsb)[1, 3] == 0
        seen |= set(lv.tolist())
    assert len(seen) >= 4, seen              # the inputs exercise most of the level range
    assert halved                            # and the CDFs went through the halving branch
    if not keyframe:
        assert not cdf_ours[1:].any() or np.array_equal(cdf_ours[1:], np.tile(32 * np.arange(1, 7, dtype=np.uint16), (10, 1)))


@pytest.mark.gpu
@pytest.mark.parametrize("masking,keyframe,skips", [(0, 1, False), (1, 1, False), (1, 0, True)])
def test_search_on_device_matches_reference(masking, keyframe, skips, reference):
    import torch
    L = lib_decide()

    class P(ctypes.Structure):
        _fields_ = [("etmp", ctypes.c_void_p), ("src", ctypes.c_void_p), ("bskip", ctypes.c_void_p),
                    ("etmp_stride", ctypes.c_int), ("src_stride", ctypes.c_int), ("skip_stride", ctypes.c_int),
                    ("nhsb", ctypes.c_int), ("nvsb", ctypes.c_int), ("quantizer", ctypes.c_int),
                    ("coded_quantizer", ctypes.c_int), ("qm_is_flat", ctypes.c_int), ("use_activity_masking", ctypes.c_int),
                    ("is_keyframe", ctypes.c_int), ("dering_lambda", ctypes.c_double)]

    L.daala_b200_dering_search.argtypes = [ctypes.POINTER(P), ctypes.c_void_p, ctypes.c_int, ctypes.c_void_p,
                                           ctypes.c_void_p, ctypes.c_void_p]
    rng = np.random.default_rng(11 + masking + 2 * keyframe)
    nhsb, nvsb = 9, 6
    nsb = nhsb * nvsb
    cdf_ref = np.zeros((2 * LEVELS - 1, LEVELS), np.uint16)
    L.daala_b200_dering_cdf_init(addr(cdf_ref), None)
    cdf_ours = cdf_ref.copy()
    seen = set()
    for frame, q in enumerate([72, 30, 160]):
        src, ctmp = synth_pair(rng, nhsb, nvsb, ring=[1.0, 2.0, 0.5][frame] * q / 72.0)
        bskip = None
        if skips:
            bskip = (rng.random((nvsb * 16, nhsb * 16)) < 0.6).astype(np.uint8)
            bskip[32:48, 16:48] = 1
            bskip = np.ascontiguousarray(bskip)
        lam = DERING_LAMBDA_SCALE * q * q
        search = {}

        def ref_dist(ref):
            search["lv"], dist = ref_search(ref, src, ctmp, nhsb, nvsb, q, masking, keyframe, lam, bskip, cdf_ref)
            return dist
        dist_ref = reference.value("dist%d" % frame, ref_dist)
        d_etmp = torch.from_numpy(ctmp.astype(np.int16)).cuda()
        d_src = torch.from_numpy(src).cuda()
        d_skip = torch.from_numpy(bskip).cuda() if bskip is not None else None
        prm = P(d_etmp.data_ptr(), d_src.data_ptr(), d_skip.data_ptr() if d_skip is not None else None, nhsb * 64,
                nhsb * 64, nhsb * 16, nhsb, nvsb, q, q, 0, masking, keyframe, lam)
        lv = np.zeros(nsb, np.uint8)
        dist = np.zeros((LEVELS, nsb), np.float64)
        s = torch.cuda.current_stream().cuda_stream
        assert L.daala_b200_dering_search(ctypes.byref(prm), addr(cdf_ours), 128, addr(lv), addr(dist), s) == 0
        coded = coded_flags(bskip, nhsb, nvsb).astype(bool) if bskip is not None else np.ones(nsb, bool)
        np.testing.assert_allclose(dist[:, coded], dist_ref[:, coded], rtol=1e-12, atol=0)
        reference.check(lv, search.get("lv"), frame)
        reference.check(cdf_ours, cdf_ref, frame)
        seen |= set(lv.tolist())
    assert len(seen) >= 3, seen
