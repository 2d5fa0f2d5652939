"""The keyframe engine (csrc/kf_engine.cu) through its host-buffer C ABI against the oracle: device-side
work lists, persistent intra wavefront, chroma CfL, reconstruction and every per-band decision."""
import os

import numpy as np
import pytest

from tests import frame_oracle, oracle_lib

pytestmark = [pytest.mark.gpu]
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _oracle():
    ref = oracle_lib.load_ref()
    return (ref, "ref") if ref is not None else (oracle_lib.load_port(), "port")


def _coding_tables():
    """Per block size: (rows, cols) of the coded prefix in coding order."""
    from daala_b200 import pvq
    inp = pvq.qm_inputs()
    scans = {m: inp["scan%d" % m].astype(np.int64) for m in (4, 8, 16, 32, 64)}
    tabs = {}
    for bs in range(5):
        n = 4 << bs
        idx = np.arange(n * n).reshape(n, n)
        order = pvq.raster_to_coding_order(idx, scans)[:min(n * n, 512)]
        tabs[bs] = (order // n, order % n)
    return tabs


def _y_plane(blocks, y16, geom, pli, frame, tabs):
    h, w = geom.plane_shape(pli)
    out = np.zeros((h, w), np.int32)
    sel = np.nonzero((blocks["pli"] == pli) & (blocks["frame"] == frame))[0]
    for bs in range(5):
        ids = sel[blocks["bs"][sel] == bs]
        if not len(ids):
            continue
        r, c = tabs[bs]
        off = blocks["coef_off"][ids].astype(np.int64)[:, None] + np.arange(len(r))[None, :]
        rows = blocks["y0"][ids].astype(np.int64)[:, None] + r[None, :]
        cols = blocks["x0"][ids].astype(np.int64)[:, None] + c[None, :]
        out[rows, cols] = y16[off]
    return out


def _check_batch(eng, geom, frames, q0, q4, use_masking=1, planes_checked=(0, 1, 2)):
    """frames: list of (padded planes, bsize).  Runs the engine end to end and compares everything."""
    from daala_b200 import engine
    lib, prefix = _oracle()
    F = len(frames)
    planes = [np.stack([f[0][p] for f in frames]) for p in range(3)]
    bsize = np.stack([f[1] for f in frames])
    out = eng.encode(planes, bsize)
    tabs = _coding_tables()
    for f in range(F):
        want = frame_oracle.keyframe_chain(lib, prefix, frames[f][0], geom, frames[f][1], q0, q4, use_masking)
        for pli in planes_checked:
            blocks = out["luma_blocks"] if pli == 0 else out["chroma_blocks"]
            res = out["luma_res"] if pli == 0 else out["chroma_res"]
            y16 = out["luma_y16"] if pli == 0 else out["chroma_y16"]
            got = engine.band_records(blocks, res, geom, pli, f)
            bad = np.argwhere(got != want[pli]["rec"])
            assert len(bad) == 0, ("band decisions", f, pli, len(bad), bad[:8].tolist(), got[tuple(bad[0][:3])].tolist(),
                                   want[pli]["rec"][tuple(bad[0][:3])].tolist())
            assert np.array_equal(_y_plane(blocks, y16, geom, pli, f, tabs), want[pli]["yplane"]), ("pulses", f, pli)
            assert np.array_equal(out["recon%d" % pli][f], want[pli]["recon"]), ("recon", f, pli)
        dq = [eng.coeff_plane(p)[f] for p in range(3)]
        for pli in planes_checked:
            assert np.array_equal(dq[pli], want[pli]["dq"]), ("quantised plane", f, pli)
    return out


def _frames(geom, n, q_seed=0, mode="mixed", pic=None):
    from daala_b200 import synth
    frames = []
    seed = 12345 + q_seed
    for f in range(n):
        planes, seed = synth.frame(geom.pic_w, geom.pic_h, f=f, seed=seed)
        frames.append((synth.pad_planes(planes, geom), synth.block_size_map(geom, mode, seed=50 + f + q_seed)))
    return frames


def test_engine_lists_are_consistent():
    """Descriptors partition the coding-order buffers; neighbours are the same-size top / left blocks;
    the item lists hold every dependency-free (block, band) once, the chain heads are the chain items without a
    neighbour to wait for."""
    from daala_b200 import engine
    from daala_b200.frame import Geometry
    geom = Geometry(328, 200)
    frames = _frames(geom, 3)
    eng = engine.KeyframeEngine(geom, nframes=3, q0=40)
    eng.upload([np.stack([f[0][p] for f in frames]) for p in range(3)], np.stack([f[1] for f in frames]))
    eng.run_device(engine.PH_LISTS, graph=False)
    cnt = eng.counts()
    tot = eng.count_blocks(np.stack([f[1] for f in frames]))
    assert cnt[0] == tot.n_luma and cnt[1] == tot.n_chroma and cnt[2] == tot.luma_coefs and cnt[3] == tot.chroma_coefs
    from daala_b200 import pvq
    nl = int(cnt[0])
    luma = eng.download(eng.buf.luma_blocks, (nl,), pvq.BLOCK_DTYPE)
    top = eng.download(eng.buf.dep_top, (nl,), np.int32)
    left = eng.download(eng.buf.dep_left, (nl,), np.int32)
    # same set of blocks as the numpy builder
    want = np.concatenate([pvq.block_list(frames[f][1], geom, frame=f) for f in range(3)])
    key = lambda b: (b["frame"].astype(np.int64) << 40) | (b["pli"].astype(np.int64) << 36) | (b["y0"].astype(np.int64) << 18) | b["x0"]  # noqa: E731
    wl = want[want["pli"] == 0]
    assert np.array_equal(np.sort(key(luma)), np.sort(key(wl)))
    o1, o2 = np.argsort(key(luma)), np.argsort(key(wl))
    assert np.array_equal(luma["bs"][o1], wl["bs"][o2])
    # coefficient ranges tile [0, total)
    length = np.minimum(16 << (2 * luma["bs"].astype(np.int64)), 512)
    o = np.argsort(luma["coef_off"])
    assert luma["coef_off"][o][0] == 0 and np.array_equal(luma["coef_off"][o][1:], np.cumsum(length[o])[:-1])
    # neighbours
    maps = np.stack([f[1] for f in frames])
    index = {}
    for i, b in enumerate(luma):
        index[(int(b["frame"]), int(b["y0"]), int(b["x0"]))] = i
    for i, b in enumerate(luma):
        n = 4 << int(b["bs"])
        f, y0, x0 = int(b["frame"]), int(b["y0"]), int(b["x0"])
        et = index[(f, y0 - n, x0)] if y0 > 0 and maps[f, (y0 - 1) >> 3, x0 >> 3] == b["bs"] else -1
        el = index[(f, y0, x0 - n)] if x0 > 0 and maps[f, y0 >> 3, (x0 - 1) >> 3] == b["bs"] else -1
        assert (top[i], left[i]) == (et, el), (i, b, top[i], left[i], et, el)
    # chroma descriptors
    nc = int(cnt[1])
    chroma = eng.download(eng.buf.chroma_blocks, (nc,), pvq.BLOCK_DTYPE)
    wc = pvq.mark_luma4x4(want[want["pli"] != 0].copy(), [f[1] for f in frames])
    assert np.array_equal(np.sort(key(chroma)), np.sort(key(wc)))
    o1, o2 = np.argsort(key(chroma)), np.argsort(key(wc))
    assert np.array_equal(chroma["bs"][o1], wc["bs"][o2]) and np.array_equal(chroma["xdec"][o1], wc["xdec"][o2])
    # inverse neighbours
    sb = eng.download(eng.buf.succ_bottom, (nl,), np.int32)
    sr = eng.download(eng.buf.succ_right, (nl,), np.int32)
    want_sb, want_sr = np.full(nl, -1, np.int32), np.full(nl, -1, np.int32)
    want_sb[top[top >= 0]] = np.nonzero(top >= 0)[0]
    want_sr[left[left >= 0]] = np.nonzero(left >= 0)[0]
    assert np.array_equal(sb, want_sb) and np.array_equal(sr, want_sr)
    # items: dependency-free bands 3 / 6 per class, chain heads, chain total
    nbands = np.array([1, 4, 7, 9, 9])
    nb = nbands[luma["bs"]]
    assert cnt[4] == 0
    for c, band in ((1, 3), (2, 6)):
        n = int(cnt[4 + c])
        items = eng.download(eng.buf.luma_items[c], (n,), np.uint32)
        assert ((items & 15) == band).all() and len(np.unique(items)) == n == int((nb > band).sum())
    heads = np.concatenate([eng.download(eng.buf.luma_heads, (int(cnt[engine.CNT["n_heads"]]),), np.uint32),
                            eng.download(eng.buf.luma_heads0, (int(cnt[engine.CNT["n_heads0"]]),), np.uint32)])
    assert ((heads[:int(cnt[engine.CNT["n_heads"]])] & 15) != 0).all() and ((heads[int(cnt[engine.CNT["n_heads"]]):] & 15) == 0).all()
    want_heads = set()
    for band in (0, 1, 2, 4, 5, 7, 8):
        r = band % 3
        waits = ((top >= 0) | (left >= 0)) if band == 0 else (top >= 0) if r == 1 else (left >= 0)
        for i in np.nonzero((nb > band) & ~waits)[0]:
            want_heads.add((int(i) << 4) | band)
    assert len(heads) == len(want_heads) and set(int(h) for h in heads) == want_heads
    assert cnt[engine.CNT["total_hi"]] == int((nb - (nb > 3) - (nb > 6)).sum())
    for c in range(3):
        n = int(cnt[7 + c])
        items = eng.download(eng.buf.chroma_items[c], (n,), np.uint32)
        assert len(np.unique(items)) == n == int((np.clip(nbands[chroma["bs"]] - 3 * c, 0, 3)).sum())
    eng.close()


@pytest.mark.parametrize("size,q0,nf", [((200, 130), 45, 1), ((384, 256), 38, 2), ((328, 200), 72, 3)])
def test_engine_keyframe_chain_matches_oracle(size, q0, nf):
    from daala_b200 import engine
    from daala_b200.frame import Geometry
    geom = Geometry(*size)
    q4 = np.full((3, 30), 16 if q0 != 45 else 20, np.uint8)
    eng = engine.KeyframeEngine(geom, nframes=nf, q0=q0, pvq_qm_q4=q4)
    frames = _frames(geom, nf)
    _check_batch(eng, geom, frames, q0, q4)
    # block sizes change every step: second batch with different maps and content on the same engine
    frames = _frames(geom, nf, q_seed=7)
    _check_batch(eng, geom, frames, q0, q4)
    eng.close()


def test_engine_noref_prepass_matches_oracle():
    """The no-reference searches of the luma chain bands ahead of the chains (daala_b200_kf_config.noref_prepass),
    imported by the persistent kernel: same results, on mixed and on uniform maps, two batches per engine."""
    from daala_b200 import engine
    from daala_b200.frame import Geometry
    geom = Geometry(328, 200)
    q4 = np.full((3, 30), 16, np.uint8)
    eng = engine.KeyframeEngine(geom, nframes=2, q0=72, pvq_qm_q4=q4, split_free=1, noref_prepass=1)
    _check_batch(eng, geom, _frames(geom, 2), 72, q4)
    _check_batch(eng, geom, _frames(geom, 2, q_seed=5, mode="32"), 72, q4)
    _check_batch(eng, geom, _frames(geom, 2, q_seed=6, mode="4"), 72, q4)
    eng.close()


@pytest.mark.parametrize("split", [1, 2, 3])
def test_engine_split_phase_kernels_match_oracle(split):
    """The dependency-free bands (chroma; with split = 2 also luma bands 3 / 6) through the three phase
    kernels with the band context parked in HBM records (daala_b200_kf_config.split_free) instead of the
    persistent kernel: same results, bit for bit."""
    from daala_b200 import engine
    from daala_b200.frame import Geometry
    geom = Geometry(328, 200)
    q4 = np.full((3, 30), 16, np.uint8)
    # split 3: additionally the luma intra chains level-synchronously (daala_b200_kf_config.level_chains)
    eng = engine.KeyframeEngine(geom, nframes=2, q0=72, pvq_qm_q4=q4, split_free=min(split, 2), level_chains=int(split == 3))
    _check_batch(eng, geom, _frames(geom, 2), 72, q4)
    _check_batch(eng, geom, _frames(geom, 2, q_seed=3, mode="64"), 72, q4)
    eng.close()


@pytest.mark.parametrize("mode", ["4", "8", "16", "32", "64"])
def test_engine_uniform_block_sizes(mode):
    from daala_b200 import engine
    from daala_b200.frame import Geometry
    geom = Geometry(256, 192)
    q4 = np.full((3, 30), 16, np.uint8)
    eng = engine.KeyframeEngine(geom, nframes=1, q0=50, pvq_qm_q4=q4)
    _check_batch(eng, geom, _frames(geom, 1, mode=mode), 50, q4)
    eng.close()


@pytest.mark.parametrize("content", ["flat128", "noise", "black", "white"])
def test_engine_edge_content(content):
    from daala_b200 import engine, synth
    from daala_b200.frame import Geometry
    geom = Geometry(200, 136)
    rng = np.random.default_rng(3)
    planes = []
    for pli in range(3):
        h, w = (136, 200) if pli == 0 else (68, 100)
        value = {"flat128": 128, "black": 0, "white": 255}.get(content)
        planes.append(np.full((h, w), value, np.uint8) if value is not None
                      else rng.integers(0, 256, size=(h, w), dtype=np.uint8))
    planes = synth.pad_planes(planes, geom)
    bsize = synth.block_size_map(geom, "mixed", seed=8)
    q4 = np.full((3, 30), 16, np.uint8)
    eng = engine.KeyframeEngine(geom, nframes=1, q0=30, pvq_qm_q4=q4)
    _check_batch(eng, geom, [(planes, bsize)], 30, q4)
    eng.close()


@pytest.mark.parametrize("size,maps", [((1920, 1080), "synthetic"), ((3840, 2160), "synthetic"),
                                       ((3840, 2160), "reference")])
def test_engine_baseline_sizes_q72_match_oracle(size, maps):
    """BASELINE.json's configurations at the bench's quantiser (q0 = 72): whole keyframe chain, every
    per-band index, against the reference build."""
    from daala_b200 import engine, synth
    from daala_b200.frame import Geometry
    geom = Geometry(*size)
    q4 = np.full((3, 30), 16, np.uint8)
    planes, _ = synth.frame(geom.pic_w, geom.pic_h, f=1, seed=4242)
    planes = synth.pad_planes(planes, geom)
    if maps == "reference":
        real = np.load(os.path.join(ROOT, "daala_b200", "data", "bench_bsize_4k.npz"))
        bsize = np.ascontiguousarray(real["bsize_1"])
    else:
        bsize = synth.block_size_map(geom, "mixed", seed=101)
    eng = engine.KeyframeEngine(geom, nframes=1, q0=72, pvq_qm_q4=q4)
    _check_batch(eng, geom, [(planes, bsize)], 72, q4)
    eng.close()


def test_engine_dering_stage_matches_oracle(reference):
    """daala_b200_kf_config.dering: the reconstruction through od_dering with caller-supplied per-superblock
    levels (the final application of src/encode.c:2812-2842 on keyframes: no block is marked skipped, luma
    directions re-used by chroma, chroma thresholds * 0.6, level 0 = untouched).  Oracle: the reference chain
    up to the lapped planes, the reference's SB-edge postfilter, the pinned deringing port per superblock."""
    import ctypes
    from daala_b200 import engine
    from daala_b200.frame import Geometry
    port = oracle_lib.load_port()
    geom = Geometry(328, 200)
    q0, q4 = 72, np.full((3, 30), 16, np.uint8)
    F = 2
    frames = _frames(geom, F)
    rng = np.random.default_rng(3)
    levels = rng.integers(0, 6, size=(F, geom.nvsb, geom.nhsb)).astype(np.uint8)
    levels[0, 0, 0] = 0
    eng = engine.KeyframeEngine(geom, nframes=F, q0=q0, pvq_qm_q4=q4, split_free=1, dering=1)
    out = eng.encode([np.stack([f[0][p] for f in frames]) for p in range(3)], np.stack([f[1] for f in frames]),
                     dering_levels=levels)
    gain = [0, 0.5, 0.707, 1, 1.41, 2]
    base = float(q0) ** 0.84182
    Dir = (ctypes.c_int * 8) * 8
    a = oracle_lib.addr

    def oracle(lib, f):
        """Per plane the reconstruction through the frame driver's od_dering, then per plane the same through the
        reference's SB-edge postfilter and the pinned deringing port."""
        prefix = "ref"
        want = frame_oracle.keyframe_chain(lib, prefix, frames[f][0], geom, frames[f][1], q0, q4, 1)
        # the same through the oracle's frame driver (the reference's own od_dering), which bench.py uses
        want_d = frame_oracle.keyframe_chain(lib, prefix, frames[f][0], geom, frames[f][1], q0, q4, 1, dering_levels=levels[f])
        recs = [want_d[pli]["recon"] for pli in range(3)]
        dirs = {}
        for pli in range(3):
            xdec = 1 if pli else 0
            c = frame_oracle.inverse_plane(lib, prefix, want[pli]["dq"], geom, pli, frames[f][1], 1, lapped_only=True)
            c = np.ascontiguousarray(c, np.int32)
            h, w = c.shape
            lib.od_apply_postfilter_frame_sbs(a(c), w, geom.nhsb, geom.nvsb, xdec, xdec)
            x16 = c.astype(np.int16)
            y16 = x16.copy()
            sb = 64 >> xdec
            units = 16 >> xdec
            skip_stride = geom.nhsb * units
            bskip = np.zeros((geom.nvsb * units, skip_stride), np.uint8)
            for sby in range(geom.nvsb):
                for sbx in range(geom.nhsb):
                    g = int(levels[f, sby, sbx])
                    if g == 0:
                        continue
                    thr = int(gain[g] * base * (0.6 if pli else 1))
                    d = dirs.setdefault((sby, sbx), Dir())
                    yb = np.zeros((sb, sb), np.int16)
                    port.port_dering(a(yb), sb, a(x16, sby * sb * w + sbx * sb), w, 8, 8, sbx, sby, geom.nhsb, geom.nvsb,
                                     xdec, d, pli, a(bskip, (sby * units) * skip_stride + sbx * units), skip_stride, thr, 1, 4)
                    y16[sby * sb:(sby + 1) * sb, sbx * sb:(sbx + 1) * sb] = yb
            recs.append(np.clip(((y16.astype(np.int32) + 8) >> 4) + 128, 0, 255).astype(np.uint8))
        return recs
    for f in range(F):
        want = oracle(reference.lib, f) if reference.lib is not None else [None] * 6
        for pli in range(3):
            reference.check(out["recon%d" % pli][f], want[pli], ("dering recon vs od_dering", f, pli))
        for pli in range(3):
            reference.check(out["recon%d" % pli][f], want[3 + pli], ("dering recon", f, pli))
    eng.close()


@pytest.mark.parametrize("q0", [72, 38])
def test_engine_dering_search_matches_reference(q0, reference):
    """daala_b200_kf_config.dering = 2: the engine searches the deringing levels itself (src/encode.c:2708-2811: five
    filtered candidates and the unfiltered reconstruction scored by od_compute_dist + lambda * adaptive-CDF rate, one
    decision thread per frame) and applies them.  Oracle: the reference chain up to the SB-edge postfilter (ctmp),
    then the reference's own loop (oracle/ref_hooks_encode.c::oracle_ref_dering_search) on ctmp and the source
    luma; the levels must be identical, and the reconstruction equal to the oracle's deringing application at
    those levels."""
    from daala_b200 import engine
    from daala_b200.frame import Geometry
    from tests import test_dering_search as ds
    geom = Geometry(328, 200)
    q4 = np.full((3, 30), 16, np.uint8)
    F = 3
    frames = _frames(geom, F, q_seed=q0)
    eng = engine.KeyframeEngine(geom, nframes=F, q0=q0, pvq_qm_q4=q4, split_free=1, dering=2, coded_quantizer=q0)
    out = eng.encode([np.stack([f[0][p] for f in frames]) for p in range(3)], np.stack([f[1] for f in frames]))
    got_levels = out["dering_levels"].copy()
    a = oracle_lib.addr
    seen = set()

    def levels(lib, f):
        prefix = "ref"
        want = frame_oracle.keyframe_chain(lib, prefix, frames[f][0], geom, frames[f][1], q0, q4, 1)
        c = frame_oracle.inverse_plane(lib, prefix, want[0]["dq"], geom, 0, frames[f][1], 1, lapped_only=True)
        c = np.ascontiguousarray(c, np.int32)
        lib.od_apply_postfilter_frame_sbs(a(c), c.shape[1], geom.nhsb, geom.nvsb, 0, 0)
        cdf = np.zeros((11, 6), np.uint16)
        cdf[:] = 32 * np.arange(1, 7, dtype=np.uint16)
        src = np.ascontiguousarray(frames[f][0][0], np.uint8)
        lv_ref, _ = ds.ref_search(lib, src, c, geom.nhsb, geom.nvsb, q0, 1, 1, eng.dering_lambda, None, cdf)
        return lv_ref.reshape(geom.nvsb, geom.nhsb)

    def recons(lib, f):
        want_d = frame_oracle.keyframe_chain(lib, "ref", frames[f][0], geom, frames[f][1], q0, q4, 1,
                                             dering_levels=got_levels[f])
        return [want_d[pli]["recon"] for pli in range(3)]
    for f in range(F):
        reference.check(got_levels[f], lambda lib: levels(lib, f), f)
        seen |= set(got_levels[f].ravel().tolist())
        want = recons(reference.lib, f) if reference.lib is not None else [None] * 3
        for pli in range(3):
            # the reconstruction at the levels the reference chose (equal to the engine's, as checked)
            reference.check(out["recon%d" % pli][f], want[pli], ("recon at the searched levels", f, pli))
    assert len(seen) >= 2, seen
    eng.close()
