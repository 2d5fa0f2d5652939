"""GPU parity of the motion-compensation and block-matching kernels (through
the C ABI) against the CPU oracle: bit-exact pixels and integer SAD/SATD."""
import ctypes

import numpy as np
import pytest

from tests import oracle_lib
from tests.oracle_lib import addr

pytestmark = pytest.mark.gpu


def _oracle():
    ref = oracle_lib.load_ref()
    return (ref, "ref") if ref is not None else (oracle_lib.load_port(), "port")


def _frames(seed=0, h=256, w=320):
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    base = 128 + 60 * np.sin(x / 7.0) + 40 * np.cos(y / 5.0)
    ref = np.clip(base + rng.integers(-20, 21, size=(h, w)), 0, 255).astype(np.uint8)
    cur = np.clip(np.roll(base, (2, 3), (0, 1)) + rng.integers(-20, 21, size=(h, w)), 0, 255).astype(np.uint8)
    return cur, ref


def test_obmc_blocks_match_oracle():
    import torch
    from daala_b200 import mc
    lib, prefix = _oracle()
    cur, ref = _frames()
    h, w = ref.shape
    pad = mc.OD_BUFFER_PADDING
    refp = np.pad(ref, pad, mode="edge")
    rng = np.random.default_rng(2)
    blocks = []
    for ln in (2, 3, 4, 5, 6):
        n = 1 << ln
        for t in range(40):
            b = np.zeros(1, mc.MC_BLOCK_DTYPE)[0]
            b["x0"] = int(rng.integers(0, (w - n) // n + 1)) * n
            b["y0"] = int(rng.integers(0, (h - n) // n + 1)) * n
            mvx = rng.integers(-200, 201, size=4)
            mvy = rng.integers(-200, 201, size=4)
            if t % 4 == 0:
                mvx[1:3], mvy[1:3] = mvx[0], mvy[0]
            if t % 9 == 0:
                mvx[:] = (mvx // 8) * 8
                mvy[:] = (mvy // 8) * 8
            b["mvx"], b["mvy"] = mvx, mvy
            b["log_xblk"] = b["log_yblk"] = ln
            b["oc"], b["s"] = int(rng.integers(0, 4)), int(rng.integers(0, 4))
            blocks.append(b)
    blocks = np.array(blocks, mc.MC_BLOCK_DTYPE)
    # non-overlapping destinations are not required for the check: compare block by block
    rp = mc.PaddedPlane(ref)
    dev_blocks = mc.to_device(blocks)
    I4 = ctypes.c_int32 * 4
    fn = lib.oracle_ref_mc_predict if prefix == "ref" else lib.port_mc_predict
    stride = refp.shape[1]
    for i, b in enumerate(blocks):
        dst = torch.zeros((h, w), dtype=torch.uint8, device="cuda:0")
        mc.predict_blocks(rp, dst, dev_blocks[i * 40:(i + 1) * 40], 1)
        n = 1 << int(b["log_xblk"])
        x0, y0 = int(b["x0"]), int(b["y0"])
        exp = np.zeros((n, n), np.uint8)
        fn(addr(exp), n, addr(refp, (y0 + pad) * stride + x0 + pad), stride, I4(*[int(v) for v in b["mvx"]]),
           I4(*[int(v) for v in b["mvy"]]), int(b["oc"]), int(b["s"]), int(b["log_xblk"]), int(b["log_yblk"]))
        got = dst[y0:y0 + n, x0:x0 + n].cpu().numpy()
        assert np.array_equal(got, exp), (i, b)


@pytest.mark.parametrize("use_satd", [0, 1])
def test_match_candidates_match_oracle(use_satd):
    import torch
    from daala_b200 import mc
    lib, prefix = _oracle()
    cur, ref = _frames(seed=1)
    h, w = ref.shape
    pad = mc.OD_BUFFER_PADDING
    refp = np.pad(ref, pad, mode="edge")
    stride = refp.shape[1]
    rng = np.random.default_rng(3 + use_satd)
    jobs = []
    for ln in (2, 3, 4, 5, 6):
        n = 1 << ln
        for t in range(60):
            j = np.zeros(1, mc.MATCH_JOB_DTYPE)[0]
            j["x0"] = int(rng.integers(0, (w - n) // 4 + 1)) * 4
            j["y0"] = int(rng.integers(0, (h - n) // 4 + 1)) * 4
            j["mvx"], j["mvy"] = int(rng.integers(-300, 301)), int(rng.integers(-300, 301))
            if t % 3 == 0:
                j["mvx"], j["mvy"] = (int(j["mvx"]) // 8) * 8, (int(j["mvy"]) // 8) * 8
            j["log_blk"] = ln
            jobs.append(j)
    jobs = np.array(jobs, mc.MATCH_JOB_DTYPE)
    rp = mc.PaddedPlane(ref)
    cur_d = torch.from_numpy(cur).to("cuda:0")
    out = mc.match_candidates(cur_d, rp, mc.to_device(jobs), len(jobs), use_satd=bool(use_satd)).cpu().numpy()
    pfn = lib.oracle_ref_mc_predict1fmv8 if prefix == "ref" else lib.port_mc_predict1fmv8
    for i, j in enumerate(jobs):
        ln = int(j["log_blk"])
        n = 1 << ln
        x0, y0 = int(j["x0"]), int(j["y0"])
        pred = np.zeros((n, n), np.uint8)
        pfn(addr(pred), addr(refp, (y0 + pad) * stride + x0 + pad), stride, int(j["mvx"]), int(j["mvy"]), ln, ln)
        cblk = np.ascontiguousarray(cur[y0:y0 + n, x0:x0 + n])
        if use_satd:
            if prefix == "ref":
                exp = getattr(lib, "od_mc_compute_satd8_%dx%d_c" % (n, n))(addr(cblk), n, addr(pred), n)
            else:
                exp = lib.port_mc_compute_satd8(ln, addr(cblk), n, addr(pred), n)
        else:
            if prefix == "ref":
                exp = lib.od_mc_compute_sad8_c(addr(cblk), n, addr(pred), n, n, n)
            else:
                exp = lib.port_mc_compute_sad8(addr(cblk), n, addr(pred), n, n, n)
        assert out[i] == exp, (i, j, out[i], exp)


def test_dropin_mc_symbols_match_oracle():
    """Host-pointer vtable entries (od_mc_*_cuda) against the oracle."""
    from daala_b200 import _native
    L = _native.lib()
    lib, prefix = _oracle()
    cur, ref = _frames(seed=4, h=128, w=160)
    h, w = ref.shape
    rng = np.random.default_rng(8)
    pfn = lib.oracle_ref_mc_predict1fmv8 if prefix == "ref" else lib.port_mc_predict1fmv8
    for ln in (2, 3, 4, 5):
        n = 1 << ln
        for t in range(6):
            mvx, mvy = int(rng.integers(-80, 81)), int(rng.integers(-80, 81))
            if t == 0:
                mvx, mvy = 16, -8
            x0, y0 = 48, 40
            a = np.zeros(n * n, np.uint8)
            b = np.zeros(n * n, np.uint8)
            L.od_mc_predict1fmv8_cuda(None, addr(a), addr(ref, y0 * w + x0), w, mvx, mvy, ln, ln)
            pfn(addr(b), addr(ref, y0 * w + x0), w, mvx, mvy, ln, ln)
            assert np.array_equal(a, b), (ln, mvx, mvy)
        blk_c = np.ascontiguousarray(cur[8:8 + n, 16:16 + n + 3])
        blk_r = np.ascontiguousarray(ref[8:8 + n, 16:16 + n + 5])
        sad = getattr(L, "od_mc_compute_sad8_%dx%d_cuda" % (n, n))(addr(blk_c), n + 3, addr(blk_r), n + 5)
        satd = getattr(L, "od_mc_compute_satd8_%dx%d_cuda" % (n, n))(addr(blk_c), n + 3, addr(blk_r), n + 5)
        if prefix == "ref":
            assert sad == lib.od_mc_compute_sad8_c(addr(blk_c), n + 3, addr(blk_r), n + 5, n, n)
            assert satd == getattr(lib, "od_mc_compute_satd8_%dx%d_c" % (n, n))(addr(blk_c), n + 3, addr(blk_r), n + 5)
        else:
            assert sad == lib.port_mc_compute_sad8(addr(blk_c), n + 3, addr(blk_r), n + 5, n, n)
            assert satd == lib.port_mc_compute_satd8(ln, addr(blk_c), n + 3, addr(blk_r), n + 5)
        # blends
        P4 = ctypes.c_void_p * 4
        preds = [np.ascontiguousarray(rng.integers(0, 256, size=n * n, dtype=np.uint8)) for _ in range(4)]
        for oc, s in ((0, 3), (1, 0), (2, 1), (3, 2)):
            g = np.zeros((n, n + 2), np.uint8)
            e = np.zeros((n, n + 2), np.uint8)
            ptrs = P4(*[p.ctypes.data for p in preds])
            if s == 3:
                L.od_mc_blend_full8_cuda(addr(g), n + 2, ptrs, ln, ln)
                (lib.od_mc_blend_full8_c if prefix == "ref" else lib.port_mc_blend_full8)(addr(e), n + 2, ptrs, ln, ln)
            else:
                L.od_mc_blend_full_split8_cuda(addr(g), n + 2, ptrs, oc, s, ln, ln)
                (lib.od_mc_blend_full_split8_c if prefix == "ref" else lib.port_mc_blend_full_split8)(
                    addr(e), n + 2, ptrs, oc, s, ln, ln)
            assert np.array_equal(g, e), (ln, oc, s)


def _random_mv_grid(rng, nv, nh, max_mv=200):
    """Hierarchically consistent validity flags + random MVs (1/8 pel)."""
    valid = np.zeros((nv + 1, nh + 1), bool)
    valid[::8, ::8] = True

    def split(vx, vy, l):
        if l == 0:
            return
        h = (1 << l) >> 1
        if rng.random() < 0.6:
            valid[vy + h, vx + h] = True
            for dx, dy in ((h, 0), (0, h), (2 * h, h), (h, 2 * h)):
                if rng.random() < 0.7:
                    valid[vy + dy, vx + dx] = True
            for dx, dy in ((0, 0), (h, 0), (0, h), (h, h)):
                split(vx + dx, vy + dy, l - 1)

    for vy in range(0, nv, 8):
        for vx in range(0, nh, 8):
            split(vx, vy, 3)
    mv = rng.integers(-max_mv, max_mv + 1, size=(nv + 1, nh + 1, 2)).astype(np.int32)
    # smooth-ish field plus a few exact full-pel and identical-neighbour vectors
    mv[::2, ::2] = (mv[::2, ::2] // 8) * 8
    mv[1::4, :] = mv[0::4, :][:mv[1::4, :].shape[0]]
    return valid, mv


def _state_mc_predict(ref, W, H, ref_y, ref_u, ref_v, valid, mv):
    """The three planes od_state_mc_predict predicts on a real od_state (oracle/ref_hooks_mc.c); None per plane
    without the reference build."""
    if ref is None:
        return [None] * 3
    outs = [np.zeros((H, W), np.uint8), np.zeros((H // 2, W // 2), np.uint8), np.zeros((H // 2, W // 2), np.uint8)]
    rc = ref.oracle_ref_state_mc_predict(W, H, addr(ref_y), addr(ref_u), addr(ref_v),
                                         addr(np.ascontiguousarray(valid.astype(np.uint8))),
                                         addr(np.ascontiguousarray(mv)), addr(outs[0]), addr(outs[1]), addr(outs[2]))
    assert rc == 0
    return outs


def test_frame_obmc_prediction_matches_reference_state_mc_predict(reference):
    """MV grid -> block list (daala_b200/mvgrid.py) -> k_obmc_blocks for all three planes against
    the reference's od_state_mc_predict driven on a real od_state (oracle/ref_hooks_mc.c)."""
    import torch
    from daala_b200 import mc, mvgrid
    rng = np.random.default_rng(21)
    W, H = 256, 192
    cur, ref_y = _frames(seed=6, h=H, w=W)
    ref_u = np.ascontiguousarray(ref_y[::2, ::2][:, ::-1])
    ref_v = np.ascontiguousarray(ref_y[1::2, 1::2])
    nv, nh = H // 8, W // 8
    valid, mv = _random_mv_grid(rng, nv, nh)
    outs = _state_mc_predict(reference.lib, W, H, ref_y, ref_u, ref_v, valid, mv)
    for pli, refp in enumerate((ref_y, ref_u, ref_v)):
        xdec = 1 if pli else 0
        blocks = mvgrid.block_list(valid, mv, xdec=xdec)
        rp = mc.PaddedPlane(refp)
        dst = torch.zeros(refp.shape, dtype=torch.uint8, device="cuda:0")
        mc.predict_blocks(rp, dst, mc.to_device(blocks), len(blocks))
        got = dst.cpu().numpy()
        reference.check(got, outs[pli], "plane %d" % pli)


def test_inter_frame_chain_mv_grid_to_pvq_matches_reference(reference):
    """The inter-frame hot path end to end on the device: MV grid -> OBMC prediction of all planes
    (k_obmc_blocks) -> forward transform of the prediction (the reference's mdtmp planes,
    src/encode.c:2566-2573) -> forward transform of the source -> PVQ against that prediction ->
    inverse.  Oracle: od_state_mc_predict on a real od_state, then the reference's own transform /
    pvq_theta / inverse functions on the predicted planes."""
    import torch
    from daala_b200 import mc, mvgrid, pvq, synth
    from daala_b200.frame import FrameBuffers, Geometry
    from daala_b200.pipeline import HotPath
    from tests import frame_oracle
    lib, prefix = _oracle()
    rng = np.random.default_rng(33)
    W, H = 256, 192
    geom = Geometry(W, H)
    cur_y, ref_y = _frames(seed=9, h=H, w=W)
    ref_u = np.ascontiguousarray(ref_y[::2, ::2][:, ::-1])
    ref_v = np.ascontiguousarray(ref_y[1::2, 1::2])
    cur = [cur_y, np.ascontiguousarray(cur_y[::2, ::2][:, ::-1]), np.ascontiguousarray(cur_y[1::2, 1::2])]
    valid, mv = _random_mv_grid(rng, H // 8, W // 8)
    # reference prediction
    pred_ref = _state_mc_predict(reference.lib, W, H, ref_y, ref_u, ref_v, valid, mv)
    # device chain
    bsize = synth.block_size_map(geom, "mixed", seed=12)
    q4 = np.full((3, 30), 20, np.uint8)
    hp = HotPath(geom, q0=45, is_keyframe=0, pvq_qm_q4=q4)
    hp.fb.upload(cur, bsize)
    pred = FrameBuffers(geom)
    pred.upload(cur, bsize)      # block-size map; the pixel planes are overwritten by the prediction below
    pred.haar_dc = 0
    for pli, refp in enumerate((ref_y, ref_u, ref_v)):
        blocks = mvgrid.block_list(valid, mv, xdec=1 if pli else 0)
        dst = torch.zeros(refp.shape, dtype=torch.uint8, device="cuda:0")
        mc.predict_blocks(mc.PaddedPlane(refp), dst, mc.to_device(blocks), len(blocks))
        pred.pixels[pli][0].copy_(dst)
    pred.forward()
    hp.use_prediction(pred)
    hp.set_block_sizes([bsize])
    hp.run()
    torch.cuda.synchronize()
    qm, qm_inv = pvq.default_qm(True)
    coded = 0
    for pli in range(3):
        pred_dev = pred.pixels[pli][0].cpu().numpy()
        reference.check(pred_dev, pred_ref[pli], "prediction plane %d" % pli)
        d = frame_oracle.forward_plane(lib, prefix, cur[pli], geom, pli, bsize, 0)
        # the device's prediction, equal to the reference's as checked
        md = frame_oracle.forward_plane(lib, prefix, pred_dev, geom, pli, bsize, 0)
        dq, stats = frame_oracle.pvq_plane(lib, prefix, d, md, geom, pli, bsize, 45, 0, 1, 0.147, qm, qm_inv, q4)
        coded += int(stats[0])
        assert np.array_equal(hp.fb.coeffs[pli][0].cpu().numpy(), dq), "quantised plane %d" % pli
        rec = frame_oracle.inverse_plane(lib, prefix, dq, geom, pli, bsize, 0)
        assert np.array_equal(hp.fb.pixels_out[pli][0].cpu().numpy(), rec), "recon plane %d" % pli
    assert coded > 0


def test_bma_candidate_cost_matches_reference(reference):
    """daala_b200_mv_bma_sad against the reference's own od_mv_est_bma_sad (static, src/mcenc.c:2224) run on
    a real od_state: all three planes, chroma >> 2, blocks hanging over every picture edge (od_enc_sad's
    clipping, including the negative origins of centred BMA blocks), every block size, fractional and
    integer half-pel vectors."""
    import ctypes
    import torch
    from daala_b200 import _native, synth
    from daala_b200.frame import Geometry
    L = _native.lib()
    pic_w, pic_h = 200, 130
    geom = Geometry(pic_w, pic_h)
    cur, _ = synth.frame(pic_w, pic_h, f=3)
    prev, _ = synth.frame(pic_w, pic_h, f=2)
    cur = synth.pad_planes(cur, geom)
    prev = synth.pad_planes(prev, geom)
    rng = np.random.default_rng(11)
    jobs = []
    for log_sz in range(0, 4):                       # 8x8 .. 64x64 luma (OD_LOG_MVBSIZE_MIN = 3)
        n = 8 << log_sz
        for _ in range(40):
            bx = int(rng.integers(-n // 2, pic_w)) & ~1
            by = int(rng.integers(-n // 2, pic_h)) & ~1
            jobs.append((bx, by, int(rng.integers(-40, 41)), int(rng.integers(-40, 41)), log_sz))
        jobs.append((0, 0, 0, 0, log_sz))
        jobs.append((pic_w - n // 2 & ~1, pic_h - n // 2 & ~1, 6, -4, log_sz))
    jobs = np.array(jobs, np.int32)
    a = oracle_lib.addr
    for use_chroma in (1, 0):
        def bma_sad(ref):
            want = np.zeros(len(jobs), np.int32)
            rc = ref.oracle_ref_bma_sad(pic_w, pic_h, a(cur[0]), a(cur[1]), a(cur[2]), a(prev[0]), a(prev[1]), a(prev[2]),
                                        use_chroma, a(jobs), len(jobs), a(want))
            assert rc == 0
            return want
        pad = 96
        dev_cur, dev_ref, cs, rs, cptr, rptr = [], [], [], [], [], []
        for p in range(3):
            pd = pad >> (1 if p else 0)
            dev_cur.append(torch.from_numpy(cur[p]).cuda())
            padded = torch.from_numpy(np.pad(prev[p], pd, mode="edge")).cuda()   # od_img_edge_ext
            dev_ref.append(padded)
            cs.append(cur[p].shape[1])
            rs.append(padded.shape[1])
            cptr.append(dev_cur[p].data_ptr())
            rptr.append(padded.data_ptr() + pd * padded.shape[1] + pd)
        d_jobs = torch.from_numpy(jobs).cuda()
        d_out = torch.zeros(len(jobs), dtype=torch.int32, device="cuda")
        P3 = ctypes.c_void_p * 3
        I3 = ctypes.c_int * 3
        L.daala_b200_mv_bma_sad.argtypes = [P3, I3, P3, I3, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                            ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        rc = L.daala_b200_mv_bma_sad(P3(*cptr), I3(*cs), P3(*rptr), I3(*rs), pic_w, pic_h, 3 if use_chroma else 1,
                                     d_jobs.data_ptr(), len(jobs), d_out.data_ptr(), None)
        assert rc == 0
        torch.cuda.synchronize()
        reference.check(d_out.cpu().numpy(), bma_sad, use_chroma)


def test_obmc_candidate_cost_matches_reference(reference):
    """daala_b200_mv_est_sad against the reference's own od_mv_est_sad (static, src/mcenc.c:2267) on a real
    od_state with a random MV grid: OBMC prediction of all three planes from the grid (every outside corner /
    split state the grid produces, all block sizes) + od_enc_sad with clipping at the picture edge, chroma >> 2."""
    import ctypes
    import torch
    from daala_b200 import _native, mc, mvgrid, synth
    from daala_b200.frame import Geometry
    L = _native.lib()
    pic_w, pic_h = 200, 130
    geom = Geometry(pic_w, pic_h)
    W, H = geom.frame_w, geom.frame_h
    cur, _ = synth.frame(pic_w, pic_h, f=3)
    prev, _ = synth.frame(pic_w, pic_h, f=2)
    cur = synth.pad_planes(cur, geom)
    prev = synth.pad_planes(prev, geom)
    rng = np.random.default_rng(21)
    valid, mv = _random_mv_grid(rng, H // 8, W // 8)
    vx, vy, l, oc, s = mvgrid.leaves(valid)
    jobs = np.ascontiguousarray(np.stack([vx, vy, oc, s, l], axis=1).astype(np.int32))
    a = oracle_lib.addr
    vmap = np.ascontiguousarray(valid.astype(np.uint8))
    mvc = np.ascontiguousarray(mv)
    for use_chroma in (1, 0):
        def mv_est_sad(ref):
            want = np.zeros(len(jobs), np.int32)
            rc = ref.oracle_ref_mv_est_sad(pic_w, pic_h, a(cur[0]), a(cur[1]), a(cur[2]), a(prev[0]), a(prev[1]),
                                           a(prev[2]), a(vmap), a(mvc), use_chroma, a(jobs), len(jobs), a(want))
            assert rc == 0
            return want
        blocks = np.zeros((len(jobs), 3), mc.MC_BLOCK_DTYPE)
        for p in range(3):
            blocks[:, p] = mvgrid.blocks_for(vx, vy, l, oc, s, mv, xdec=1 if p else 0)
        pad = 96
        keep, cs, rs, cptr, rptr = [], [], [], [], []
        for p in range(3):
            pd = pad >> (1 if p else 0)
            dc = torch.from_numpy(cur[p]).cuda()
            dr = torch.from_numpy(np.pad(prev[p], pd, mode="edge")).cuda()   # od_img_edge_ext
            keep += [dc, dr]
            cs.append(cur[p].shape[1])
            rs.append(dr.shape[1])
            cptr.append(dc.data_ptr())
            rptr.append(dr.data_ptr() + pd * dr.shape[1] + pd)
        d_blocks = torch.from_numpy(np.ascontiguousarray(blocks).view(np.uint8).reshape(-1)).cuda()
        d_out = torch.zeros(len(jobs), dtype=torch.int32, device="cuda")
        P3 = ctypes.c_void_p * 3
        I3 = ctypes.c_int * 3
        L.daala_b200_mv_est_sad.argtypes = [P3, I3, P3, I3, ctypes.c_int, ctypes.c_int, ctypes.c_int, ctypes.c_void_p,
                                            ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
        rc = L.daala_b200_mv_est_sad(P3(*cptr), I3(*cs), P3(*rptr), I3(*rs), pic_w, pic_h, 3 if use_chroma else 1,
                                     d_blocks.data_ptr(), len(jobs), d_out.data_ptr(), None)
        assert rc == 0
        torch.cuda.synchronize()
        reference.check(d_out.cpu().numpy(), mv_est_sad, use_chroma)
    assert len(jobs) > 50 and len(np.unique(l)) >= 3
