"""Seeded PVQ band test cases shared by the CPU pin tests and the GPU parity
tests (test infrastructure)."""
import ctypes

import numpy as np

from tests.oracle_lib import addr

BAND_SIZES = [15, 8, 8, 32, 32, 32, 128, 128, 128]  # src/partition.c:85-91
OD_QM_STRIDE = ((1 << 10) - 1) * 16 // 3              # OD_QM_OFFSET(OD_NBSIZES), src/pvq.h:71-72


def reference_qm(ref, hvs=True):
    """state->qm / qm_inv exactly as od_init_qm (src/pvq.c:322) fills them; without the reference build, the same
    tables as exported from it (daala_b200/data/qm_*.npy, checked against od_init_qm in tests/test_host_logic.py)."""
    if ref is None:
        from daala_b200 import pvq
        return pvq.default_qm(hvs)
    qm = np.zeros(2 * OD_QM_STRIDE, np.int16)
    qm_inv = np.zeros(2 * OD_QM_STRIDE, np.int16)
    tbl = (ctypes.c_int * 64).in_dll(ref, "OD_QM8_Q4_HVS" if hvs else "OD_QM8_Q4_FLAT")
    ref.od_init_qm(addr(qm), addr(qm_inv), tbl)
    return qm, qm_inv


def make_band(rng, n, kind):
    """(x0, r0) int32 vectors.  kind: 'pred' (good prediction), 'weak', 'zero_ref',
    'zero_x', 'big' (large magnitudes, exercises xshift/rshift), 'tiny', 'sparse'."""
    decay = np.exp(-np.arange(n) / max(4.0, n / 3.0))
    amp = {"pred": 600, "weak": 400, "zero_ref": 500, "zero_x": 300, "big": 60000, "tiny": 6,
           "sparse": 900}[kind]
    x = rng.laplace(0, amp, size=n) * decay
    if kind == "sparse":
        x *= rng.random(n) < 0.2
    if kind == "zero_x":
        x[:] = 0
    x0 = np.round(x).astype(np.int32)
    if kind == "zero_ref":
        r0 = np.zeros(n, np.int32)
    elif kind in ("pred", "big", "sparse"):
        r0 = np.round(x * rng.uniform(0.7, 1.2) + rng.laplace(0, amp * 0.15, size=n) * decay).astype(np.int32)
    elif kind == "zero_x":
        r0 = np.round(rng.laplace(0, amp, size=n) * decay).astype(np.int32)
    else:
        r0 = np.round(rng.laplace(0, amp, size=n) * decay + 0.3 * x).astype(np.int32)
    return x0, r0


def cases(seed=1, per_combo=3):
    """Yields dicts describing pvq_theta invocations."""
    rng = np.random.default_rng(seed)
    kinds = ["pred", "weak", "zero_ref", "zero_x", "big", "tiny", "sparse"]
    for n in (15, 8, 32, 128):
        for kind in kinds:
            for is_keyframe, pli in ((1, 0), (1, 1), (0, 0), (0, 2)):
                for beta in (4096, 6144):
                    if beta == 6144 and (pli != 0 or n == 15):
                        continue  # masking only on luma, never 4x4 (src/pvq.c:205-268)
                    for _ in range(per_combo):
                        x0, r0 = make_band(rng, n, kind)
                        q0 = int(rng.choice([8, 23, 64, 150, 400, 1100]))
                        yield dict(n=n, kind=kind, is_keyframe=is_keyframe, pli=pli, beta=beta, q0=q0,
                                   x0=x0, r0=r0, qm_off=int(rng.integers(1, 64)),
                                   lam=float(rng.choice([0.147, 0.05, 0.3])))


def run_theta(lib, prefix, c, qm, qm_inv):
    """Calls pvq_theta of `lib` ('ref': oracle_ref_pvq_theta with speed=1;
    'port': port_pvq_theta).  Returns a comparable dict."""
    n = c["n"]
    out = np.zeros(n, np.int32)
    y = np.zeros(n, np.int32)
    it, mt, vk = ctypes.c_int(0), ctypes.c_int(0), ctypes.c_int(0)
    sd = ctypes.c_double(0.0)
    x0 = np.ascontiguousarray(c["x0"])
    r0 = np.ascontiguousarray(c["r0"])
    q = np.ascontiguousarray(qm[c["qm_off"]:c["qm_off"] + n])
    qi = np.ascontiguousarray(qm_inv[c["qm_off"]:c["qm_off"] + n])
    if prefix == "ref":
        fn = lib.oracle_ref_pvq_theta
        fn.restype = ctypes.c_int
        g = fn(addr(out), addr(x0), addr(r0), n, c["q0"], addr(y), ctypes.byref(it), ctypes.byref(mt),
               ctypes.byref(vk), c["beta"], ctypes.byref(sd), 1, c["is_keyframe"], c["pli"], None,
               addr(q), addr(qi), ctypes.c_double(c["lam"]), 1)
    else:
        fn = lib.port_pvq_theta
        fn.restype = ctypes.c_int
        g = fn(addr(out), addr(x0), addr(r0), n, c["q0"], addr(y), ctypes.byref(it), ctypes.byref(mt),
               ctypes.byref(vk), c["beta"], ctypes.byref(sd), c["is_keyframe"], c["pli"],
               addr(q), addr(qi), ctypes.c_double(c["lam"]))
    ny = n if it.value == -1 else n - 1
    return dict(gain=g, itheta=it.value, max_theta=mt.value, k=vk.value, y=y[:ny].copy(), out=out,
                skip_diff=sd.value)
