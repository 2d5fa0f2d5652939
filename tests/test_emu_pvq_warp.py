"""The warp-per-band PVQ quantiser of the device (daala_b200/csrc/pvq_warp.cuh) compiled for the host
on a SIMT emulation (tests/emu/simt_emu.h: 32 fibres, warp collectives as rendezvous) and pinned
against the reference build's pvq_theta (or the outputs recorded from it) -- the same source the CUDA
kernels include, so the candidate parallelisation, the event order and the redux-screened pulse search are checked on the CPU."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from tests import pvq_cases
from tests.oracle_lib import addr

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
BUILD = os.path.join(HERE, "emu", "_build")


def _build(name, extra):
    os.makedirs(BUILD, exist_ok=True)
    out = os.path.join(BUILD, name)
    srcs = [os.path.join(HERE, "emu", "pvq_warp_emu.cpp"), os.path.join(HERE, "emu", "simt_emu.h"),
            os.path.join(ROOT, "daala_b200", "csrc", "pvq_warp.cuh"), os.path.join(ROOT, "daala_b200", "csrc", "pvq_math.cuh")]
    if not os.path.exists(out) or os.path.getmtime(out) < max(os.path.getmtime(s) for s in srcs):
        subprocess.run(["g++", "-O1", "-std=c++17", "-shared", "-fPIC", "-Wno-unknown-pragmas"] + extra +
                       ["-I", os.path.join(ROOT, "daala_b200", "csrc"), "-I", os.path.join(HERE, "emu"), srcs[0], "-o", out],
                       check=True)
    lib = ctypes.CDLL(out)
    lib.emu_quantise_band.restype = ctypes.c_int
    return lib


def _run(emu, c, qm, qm_inv):
    n = c["n"]
    out = np.zeros(n, np.int32)
    y = np.zeros(n, np.int32)
    it, mt, vk = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0)
    sd = ctypes.c_double(0.0)
    x0 = np.ascontiguousarray(c["x0"])
    r0 = np.ascontiguousarray(c["r0"])
    q = np.ascontiguousarray(qm[c["qm_off"]:c["qm_off"] + n])
    qi = np.ascontiguousarray(qm_inv[c["qm_off"]:c["qm_off"] + n])
    g = emu.emu_quantise_band(addr(out), addr(x0), addr(r0), n, c["q0"], addr(y), ctypes.byref(it), ctypes.byref(mt),
                              ctypes.byref(vk), c["beta"], ctypes.byref(sd), c["is_keyframe"], c["pli"], addr(q), addr(qi),
                              ctypes.c_double(c["lam"]))
    ny = n if it.value == -1 else n - 1
    return dict(gain=g, itheta=it.value, max_theta=mt.value, k=vk.value, y=y[:ny].copy(), out=out, skip_diff=sd.value)


# the second build lowers the "products are exact" bound so that the literal-scan path of the plain
# pulses (taken on the device only when a product could exceed 2^53) runs on ordinary inputs
# fourth run: keyframe luma with the no-reference half searched ahead of time (the engine's prepass);
# third run: the same bands through the three phases with the band context parked in a record in between
# (the split kernels of the engine), size-class specialised instantiations
@pytest.mark.parametrize("name,extra,seeds,split", [("libpvq_warp_emu.so", [], (1, 2, 3), False),
                                                    ("libpvq_warp_emu_scan.so", ["-DDAALA_B200_PVQ_EXACT_BOUND=1e12"], (1,), False),
                                                    ("libpvq_warp_emu.so", [], (4,), True),
                                                    ("libpvq_warp_emu.so", [], (5,), "prepass")])
def test_warp_quantiser_matches_reference(name, extra, seeds, split, monkeypatch, reference):
    emu = _build(name, extra)
    # "prepass": keyframe luma bands with their no-reference events searched ahead of time and imported
    monkeypatch.delenv("DAALA_B200_EMU_SPLIT", raising=False)
    monkeypatch.delenv("DAALA_B200_EMU_PREPASS", raising=False)
    if split == "prepass":
        monkeypatch.setenv("DAALA_B200_EMU_PREPASS", "1")
    elif split:
        monkeypatch.setenv("DAALA_B200_EMU_SPLIT", "1")
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    stats = (ctypes.c_longlong * 4).in_dll(emu, "daala_b200_pvq_warp_stats")
    n = 0
    for seed in seeds:
        for c in pvq_cases.cases(seed=seed, per_combo=3):
            got = _run(emu, c, qm, qm_inv)
            reference.check(got, lambda ref: pvq_cases.run_theta(ref, "ref", c, qm, qm_inv),
                            {k: c[k] for k in ("n", "kind", "is_keyframe", "pli", "beta", "q0", "lam")})
            n += 1
    # coverage: unique-contender fast path, both exact fallbacks, and (second build) the literal scan
    assert n >= 400 and stats[0] > 0 and stats[1] > 0 and stats[2] > 0
    if extra:
        assert stats[3] > 0


def test_warp_quantiser_large_k(reference):
    """Fine quantisers on large vectors: K in the hundreds to thousands (all-RDO searches, 64-bit sums)."""
    emu = _build("libpvq_warp_emu.so", [])
    qm, qm_inv = pvq_cases.reference_qm(reference.lib)
    rng = np.random.default_rng(7)
    kmax = 0
    for q0 in (16, 40, 500, 620):
        for n in (8, 15, 32, 128):
            for kf, pli in ((1, 0), (1, 1), (0, 0)):
                x0, r0 = pvq_cases.make_band(rng, n, "big")
                c = dict(n=n, kind="big", is_keyframe=kf, pli=pli, beta=4096, q0=q0, x0=x0, r0=r0, qm_off=5, lam=0.147)
                got = _run(emu, c, qm, qm_inv)
                reference.check(got, lambda ref: pvq_cases.run_theta(ref, "ref", c, qm, qm_inv), (q0, n, kf, pli))
                kmax = max(kmax, got["k"])
    assert kmax > 1000
