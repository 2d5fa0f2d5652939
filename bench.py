#!/usr/bin/env python
"""bench.py -- Daala per-block encode hot path on B200: Mpixels/s on 4K 4:2:0 intra.

A "step" = one pass of the keyframe hot path over a batch of `--frames` synthetic
3840x2160 4:2:0 frames (SURVEY.md 8(d) content, seeded) through the keyframe engine
(include/daala_b200.h, csrc/kf_engine.cu):
    u8 planes + block-size maps -> work lists built on the device (every step)
      -> lapped prefilter + fDCT (4..64) -> PVQ (luma H/V intra wavefront, chroma CfL)
      -> iDCT + lapped postfilter -> u8 reconstruction + PVQ symbols

  value : luma picture pixels x frames / device time (CUDA events), inputs resident in HBM,
          one CUDA-graph replay per step
  e2e   : the same through the host-buffer C ABI (daala_b200_kf_submit / _wait): pinned host
          planes + block-size maps copied H2D, reconstruction + symbols copied D2H every step,
          two engines double-buffered, block-size maps differ from step to step
  --impl reference : the reference's own CPU code (oracle/_ref, SIMD build, one process per
          usable host core) on whole 4K frames of the same workload

Prints ONE JSON line (rank 0).  --dump-outputs DIR also writes what the last timed end-to-end step returned.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True      # the tree may be read-only: nothing is written into it
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "encoder Mpixels/s on 4K YUV420 intra"
UNIT = "Mpixels/s"
PIC_W, PIC_H = 3840, 2160
WORKLOAD = ("3840x2160 4:2:0 all-intra hot path: lapped prefilter + fDCT(4..64, quadtree map) + PVQ band "
            "quantisation (keyframe: luma H/V intra prediction, chroma CfL) + iDCT + lapped postfilter")


def workload_text():
    if DERING == 2:
        return WORKLOAD + (" + deringing with its level search (src/encode.c:2708-2842: od_dering at 5 thresholds + "
                           "od_compute_dist of the 6 candidates per 64x64 superblock, adaptive-CDF rate, decision, "
                           "application to the three planes)")
    return WORKLOAD + (" + deringing filter (od_dering of every superblock at the level the reference encoder chose "
                       "for it)" if DERING else "")
FWD_BYTES_PER_PX = 7.5   # SURVEY.md 8(d) K_fwd: 1.5 B in + 6 B out per padded luma pixel (4:2:0)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--frames", type=int, default=16, help="4K frames per step per rank")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch every kernel from the host instead of replaying a CUDA graph")
    ap.add_argument("--no-overlap", action="store_true", help="e2e: one engine, submit + wait per step")
    ap.add_argument("--block-sizes", default="reference", choices=["synthetic", "reference"],
                    help="reference (default): the maps the whole reference encoder decides for these frames at "
                         "OD_SET_QUANT 20, complexity 7 (daala_b200/data/bench_bsize_4k.npz); synthetic: seeded "
                         "quadtree maps with every size 4..64")
    ap.add_argument("--ctas-per-sm", type=int, default=0, help="persistent PVQ kernel CTAs per SM (0 = default)")
    ap.add_argument("--split-free", type=int, default=1, help="dependency-free PVQ bands as phase kernels: 0 no, 1 chroma, 2 chroma + luma")
    ap.add_argument("--dering", type=int, default=1,
                    help="config 4's 'PVQ + deringing': 1 = reconstruction through od_dering at the per-superblock levels "
                         "the whole reference encoder chose; 2 = the chain searches the levels itself (both arms); 0 = off")
    ap.add_argument("--prepass", type=int, default=0, help="luma no-reference searches ahead of the chains (1) or inside them (0)")
    ap.add_argument("--level-chains", type=int, default=0, help="luma intra chains level-synchronously (1) instead of the dependency queue (0)")
    ap.add_argument("--shard", default="frames", choices=["frames", "sbrow"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the arrays the last timed end-to-end step returned (reconstruction, PVQ symbols, "
                         "deringing levels) as DIR/<name>.npy, float32 or float64; arrays of more than %d values as "
                         "the same seeded sample of that many values" % DUMP_LIMIT)
    return ap.parse_args()


# --------------------------------------------------------------------------
# synthetic workload (host side)
# --------------------------------------------------------------------------
BLOCK_SIZES = "reference"   # --block-sizes: "synthetic" quadtree maps, or the "reference" encoder's decisions
DERING = 1                  # --dering


def make_host_frames(geom, nframes, distinct=4, rotate=0):
    """`distinct` different synthetic frames, cycled to `nframes` starting at frame `rotate`; padded
    planes + bsize maps."""
    import numpy as np
    from daala_b200 import synth
    frames = []
    seed = 12345
    real = None
    if BLOCK_SIZES == "reference":
        # maps the whole reference encoder decided for these frames (tools/make_real_bsize.py); a band
        # geometry (CPU sample) takes the top superblock rows of the same maps
        real = np.load(os.path.join(ROOT, "daala_b200", "data", "bench_bsize_4k.npz"))
        assert geom.pic_w == PIC_W and geom.bsize_shape[0] <= real["bsize_0"].shape[0]
    for f in range(min(distinct, nframes)):
        planes, seed = synth.frame(geom.pic_w, geom.pic_h, f=f, seed=seed)
        if real is not None:
            bsize = np.ascontiguousarray(real["bsize_%d" % (f % 4)][:geom.bsize_shape[0]])
            levels = np.ascontiguousarray(real["dering_%d" % (f % 4)][:geom.nvsb]).astype(np.uint8)
        else:
            bsize = synth.block_size_map(geom, "mixed", seed=100 + f)
            levels = np.random.default_rng(200 + f).integers(0, 6, size=(geom.nvsb, geom.nhsb)).astype(np.uint8)
        frames.append((synth.pad_planes(planes, geom), bsize, levels))
    return [frames[(i + rotate) % len(frames)] for i in range(nframes)]


# --------------------------------------------------------------------------
# clocks sampler
# --------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[1]))
                mx = float(parts[2])
            except ValueError:
                continue
            for n, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": mx,
                "reasons": sorted(reasons), "samples": len(sm)}


# --------------------------------------------------------------------------
# CPU reference pipeline (the reference's own functions via oracle/_ref)
# --------------------------------------------------------------------------
def cpu_pipeline_lib():
    """The reference build with its x86 SIMD paths (what a user of the reference runs), else the
    pure-C build, else the plain-C port."""
    import ctypes
    from tests import oracle_lib
    for name, build in (("libdaala_ref_simd.so", "unmodified reference sources, x86 SSE2/SSE4.1/AVX2 paths on"),
                        ("libdaala_ref.so", "unmodified reference sources, pure C")):
        path = os.path.join(ROOT, "oracle", "_ref", name)
        if os.path.exists(path):
            CPU_BUILD["build"] = build
            return ctypes.CDLL(path), "ref", "reference"
    CPU_BUILD["build"] = "plain-C port of the reference functions (oracle/port_*.c)"
    return oracle_lib.load_port(), "port", "port"


CPU_BUILD = {"build": None}
Q0 = 72            # state->quantizer for OD_SET_QUANT = 20 (coded quantizer 20 -> 0x48, src/quantizer.c:47)
CODED_Q = 20       # state->coded_quantizer (scale of od_compute_dist in the deringing search)
DERING_LAMBDA = 0.67 * 0.147 * Q0 * Q0    # enc->dering_lambda, src/rate.c:1086
PVQ_QM_Q4 = 16     # flat state->pvq_qm_q4 entries


def cpu_frame(lib, prefix, geom, planes, bsize, levels=None, record=False):
    """The same chain as the GPU step with the reference's own functions: forward transform ->
    per-block PVQ (od_hv_intra_pred / CfL prediction, pvq_theta with the closed-form rate) -> inverse."""
    import numpy as np
    from tests import frame_oracle
    q4 = np.full((3, 30), PVQ_QM_Q4, np.uint8)
    return frame_oracle.keyframe_chain(lib, prefix, planes, geom, bsize, Q0, q4, use_masking=1, record=record,
                                       dering_levels=levels if DERING == 1 else None,
                                       dering_search=dict(coded_quantizer=CODED_Q, dering_lambda=DERING_LAMBDA)
                                       if DERING == 2 else None)


_CPU_JOB = {}


def _cpu_worker(i):
    """Runs in a forked worker process: one frame of the CPU pipeline."""
    if "lib" not in _CPU_JOB:
        _CPU_JOB["lib"] = cpu_pipeline_lib()
    lib, prefix, _ = _CPU_JOB["lib"]
    frames = _CPU_JOB["frames"]
    planes, bsize, levels = frames[i % len(frames)]
    cpu_frame(lib, prefix, _CPU_JOB["geom"], planes, bsize, levels)
    return i


def cpu_pool(geom, host_frames, workers):
    """Worker processes (fork: they inherit the frames) -- the reference has no threading of its own,
    so its all-core throughput is N independent encoders, one per host core."""
    import multiprocessing
    _CPU_JOB.update(geom=geom, frames=host_frames)
    return multiprocessing.get_context("fork").Pool(workers)


def cgroup_cpu_quota():
    """CPU quota of this container in cores (cgroup v2 cpu.max / v1 cfs), or None when unlimited/unknown:
    sched_getaffinity can list far more CPUs than the container may actually use."""
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        return None if quota == "max" else round(int(quota) / int(period), 2)
    except (OSError, ValueError):
        pass
    try:
        q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        return None if q <= 0 else round(q / p, 2)
    except (OSError, ValueError):
        return None


def usable_cores():
    """Cores this process can really use: the affinity mask capped by the cgroup CPU quota."""
    aff = len(os.sched_getaffinity(0))
    quota = cgroup_cpu_quota()
    return max(1, min(aff, int(quota + 0.5))) if quota else aff, aff, quota


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from daala_b200.frame import Geometry
    geom = Geometry(PIC_W, PIC_H)
    cores, aff, quota = usable_cores()
    host_frames = make_host_frames(geom, 4, distinct=4)
    per_step = cores                       # one whole 4K frame per worker per step (~1 s of CPU each)
    pool = cpu_pool(geom, host_frames, cores) if cores > 1 else None
    lib, prefix, kind = cpu_pipeline_lib()

    def one_step():
        t0 = time.perf_counter()
        if pool is None:
            for i in range(per_step):
                cpu_frame(lib, prefix, geom, *host_frames[i % len(host_frames)])
        else:
            pool.map(_cpu_worker, range(per_step), chunksize=1)
        return time.perf_counter() - t0

    for _ in range(max(min(args.warmup, 2), 1)):
        one_step()
    times = [one_step() for _ in range(args.steps)]
    if pool is not None:
        pool.close()
    total = sum(times)
    value = geom.luma_pixels * per_step * args.steps / total / 1e6
    sample = ("%d whole 3840x2160 4:2:0 frames per step, one per worker process on %d processes (= usable cores: "
              "affinity %d, cgroup CPU quota %s); reference functions: prefilter + fDCT + pvq_theta(speed=1) + "
              "iDCT + postfilter%s; block sizes: %s" % (per_step, cores, aff, "none" if quota is None else "%.2f" % quota,
                                                          " + od_dering" + (" with its level search" if DERING == 2 else "")
                                                          if DERING else "", BLOCK_SIZES))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * total / args.steps, 3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": workload_text() + " (CPU reference functions)", "frames_per_step": per_step,
                   "block_sizes": block_sizes_text(), "quantizer": Q0},
        "cpu_baseline": {"value": round(value, 3), "unit": UNIT, "cores": cores, "kind": kind,
                         "build": CPU_BUILD["build"], "sample": sample},
        "e2e": {"value": round(value, 3), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


def block_sizes_text():
    return ("synthetic quadtree map, sizes 4..64" if BLOCK_SIZES == "synthetic" else
            "decided by the whole reference encoder for these frames (quant 20, complexity 7): mostly 32x32")


# --------------------------------------------------------------------------
# B200 arm
# --------------------------------------------------------------------------
def run_b200(args):
    import zlib
    import numpy as np
    import torch
    import torch.distributed as dist
    from daala_b200 import engine
    from daala_b200.frame import Geometry

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    geom = Geometry(PIC_W, PIC_H)
    F = args.frames
    q4 = np.full((3, 30), PVQ_QM_Q4, np.uint8)
    use_graph = not args.no_graph
    nslots = 1 if args.no_overlap else 2

    # two engines = two sets of device + pinned host buffers; slot s holds batch s of the synthetic
    # sequence (frames and block-size maps rotated by s), so consecutive e2e steps see different maps
    slots, batches = [], []
    for s in range(nslots):
        hf = make_host_frames(geom, F, rotate=s + 2 * rank)
        planes = [np.stack([f[0][p] for f in hf]) for p in range(3)]
        bsize = np.stack([f[1] for f in hf])
        eng = engine.KeyframeEngine(geom, nframes=F, q0=Q0, use_masking=1, pvq_qm_q4=q4, dering=DERING, coded_quantizer=CODED_Q,
                                    dering_lambda=DERING_LAMBDA,
                                    persist_ctas_per_sm=args.ctas_per_sm, split_free=args.split_free, level_chains=args.level_chains, noref_prepass=args.prepass,
                                    max_blocks_div=1 if BLOCK_SIZES == "synthetic" else 2)
        eng.stage_inputs(planes, bsize)
        if DERING == 1:
            eng.stage_dering_levels(np.stack([f[2] for f in hf]))
        eng.prepare_io(symbols=True, recon=True)
        slots.append(eng)
        batches.append(hf)
    eng0 = slots[0]

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        for e in slots:
            e.wait()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return float(t.item())
        return ms

    # first end-to-end pass (also uploads the inputs the device-resident timing uses) + parity check
    for e in slots:
        e.submit()
    out0 = slots[0].wait()
    for e in slots[1:]:
        e.wait()
    assert int(out0["counts"][engine.CNT["error"]]) == 0, "engine block capacity exceeded"
    total_k = int(out0["luma_res"][..., 3].clip(min=0).sum()) + int(out0["chroma_res"][..., 3].clip(min=0).sum())
    assert total_k > 0, "PVQ produced no pulses"
    dev_crc = {"recon%d" % p: zlib.crc32(np.ascontiguousarray(out0["recon%d" % p][0]).tobytes()) for p in range(3)}
    dev_levels = out0["dering_levels"][0].copy() if DERING else None
    dev_rec = [engine.band_records(out0["luma_blocks"] if p == 0 else out0["chroma_blocks"],
                                   out0["luma_res"] if p == 0 else out0["chroma_res"], geom, p, 0) for p in range(3)]

    # device-resident step time (CUDA events on the engine's stream)
    sampler = ClockSampler(local)
    eng0.time_device(engine.PH_ALL, use_graph, max(args.warmup, 3))
    barrier()
    if rank == 0:
        sampler.start()
    ms = max_over_ranks(eng0.time_device(engine.PH_ALL, use_graph, args.steps))
    # the same with both engines' graphs in flight (inputs resident, no copies): the tail of one batch's luma
    # dependency chains overlaps the next batch's work
    ms_pipelined = None
    if nslots == 2 and use_graph:
        for e in slots:
            e.run_device(engine.PH_ALL, True)
        for e in slots:
            e.wait()
        t0 = time.perf_counter()
        for i in range(2 * args.steps):
            slots[i % 2].run_device(engine.PH_ALL, True)
        for e in slots:
            e.wait()
        ms_pipelined = max_over_ranks((time.perf_counter() - t0) * 1e3) / 2

    # end to end through the host-buffer C ABI: H2D + step + D2H per batch, engines alternate
    def e2e_loop(steps):
        for i in range(steps):
            e = slots[i % nslots]
            if i >= nslots:
                e.wait()
            e.submit()
        for e in slots:
            e.wait()

    e2e_loop(2 * nslots)
    barrier()
    t0 = time.perf_counter()
    e2e_loop(args.steps)
    ms_e2e = max_over_ranks((time.perf_counter() - t0) * 1e3)
    barrier()
    if args.dump_outputs and rank == 0:
        dump_outputs(slots[(args.steps - 1) % nslots].wait(), args.dump_outputs)
    clocks = sampler.stop() if rank == 0 else None

    # per-phase device times
    reps = max(5, args.steps)
    phase_ms = {}
    chroma_kernels = "k_pvq_split<setup|search|finish>" if args.split_free > 0 else "k_pvq_persist"
    for name, ph in (("work_lists(5 kernels)", engine.PH_LISTS), ("k_forward_sb_tma", engine.PH_FORWARD),
                     ("pvq_luma(gather+k_pvq_persist<intra>+finish)", engine.PH_PVQ_LUMA),
                     ("pvq_chroma(cfl+gather+%s+finish)" % chroma_kernels, engine.PH_PVQ_CHROMA),
                     ("k_inverse_sb+k_sb_postfilter_store", engine.PH_INVERSE),
                     ("k_pvq_persist<intra> alone", engine.PH_PVQ_LUMA | engine.PH_SEARCH_ONLY),
                     ("chroma band kernels alone", engine.PH_PVQ_CHROMA | engine.PH_SEARCH_ONLY)):
        eng0.time_device(ph, False, 1)
        phase_ms[name] = eng0.time_device(ph, False, reps) / reps
    # leave the planes consistent again
    eng0.time_device(engine.PH_ALL, use_graph, 1)
    ms_fwd = phase_ms["k_forward_sb_tma"]
    ms_dom = phase_ms["k_pvq_persist<intra> alone"]

    px_job = geom.luma_pixels * F * world
    value = px_job / (ms / args.steps * 1e-3) / 1e6
    e2e = px_job / (ms_e2e / args.steps * 1e-3) / 1e6
    algo_bytes = FWD_BYTES_PER_PX * geom.frame_w * geom.frame_h * F
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = algo_bytes / (ms_fwd * 1e-3) / 1e9
    dom_bytes = 20.0 * float(eng0.totals.luma_coefs)    # K_pvq = 20 B per coded coefficient (SURVEY.md 8(d))

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    profiles = load_profile_notes()
    out = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms / args.steps, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
        "config": {"workload": workload_text(), "frames_per_step": F * world,
                   "parallelism": "frames%d (independent keyframes per rank, no data-path collective)" % world,
                   "l2": "inputs larger than L2 (%.0f MB of planes per step per rank)" % ((geom.padded_samples * F * 9) / 1e6),
                   "block_sizes": block_sizes_text(), "quantizer": Q0,
                   "work_lists": "rebuilt on the device from the block-size maps inside every step (timed region); "
                                 "e2e uploads different maps on consecutive steps",
                   "pvq": "one warp per band; luma intra chains in a persistent kernel with a dependency queue%s; "
                          "chroma%s as three phase kernels (setup / search / finish, band context in HBM)" % (
                              " (level-synchronous variant)" if args.level_chains else "",
                              " and luma bands 3/6" if args.split_free > 1 else "") if args.split_free > 0 else
                          "one warp per band, persistent kernels for luma (dependency queue) and chroma",
                   "pvq_pulses_first_batch": total_k},
        "e2e": {"value": round(e2e, 2), "unit": UNIT, "h2d_bytes_per_step": int(eng0.h2d_bytes),
                "d2h_bytes_per_step": int(eng0.d2h_bytes), "ms_per_step": round(ms_e2e / args.steps, 4),
                "api": "daala_b200_kf_submit / daala_b200_kf_wait (C ABI, pinned host buffers)",
                "pipeline": ("two engines alternate: copy-in / graph / copy-out of consecutive batches overlap"
                             if nslots == 2 else "one engine, serial copy-in, compute, copy-out")},
        "cuda_graph": bool(use_graph),
        "value_two_batches_in_flight": None if ms_pipelined is None else {
            "value": round(px_job / (ms_pipelined / args.steps * 1e-3) / 1e6, 2), "ms_per_step": round(ms_pipelined / args.steps, 4),
            "note": "both engines' graphs enqueued back to back on their own streams, inputs resident, wall clock"},
        "gpu_launches": eng0.launches_per_step() * args.steps,
        "clocks": clocks,
        # dominant kernel by time: the persistent luma PVQ kernel -- a greedy double-precision search bound by
        # dependency latency and FP64/integer issue, not HBM; its HBM fraction is reported as the contract asks
        "roofline": {"kernel": "k_pvq_persist<intra> (luma PVQ search + H/V intra prediction wavefront)", "bound": "hbm",
                     "achieved": round(dom_bytes / (ms_dom * 1e-3) / 1e9, 1), "peak": peak, "peak_source": peak_src,
                     "unit": "GB/s", "frac": round(dom_bytes / (ms_dom * 1e-3) / 1e9 / peak, 4),
                     "traffic": profiles.get("pvq_traffic"), "traffic_source": profiles.get("pvq_traffic_source"),
                     "algorithmic_bytes_per_launch": int(dom_bytes), "ms_per_launch": round(ms_dom, 4),
                     "note": "latency/issue-bound search; see roofline_transform for the HBM-bound kernel"},
        # the fused lapped-filter + DCT kernel the north star sets its HBM target on
        "roofline_transform": {"kernel": "k_forward_sb_tma", "bound": "hbm", "achieved": round(achieved, 1),
                               "peak": peak, "peak_source": peak_src, "unit": "GB/s", "frac": round(achieved / peak, 4),
                               "traffic": profiles.get("fwd_traffic"), "traffic_source": profiles.get("fwd_traffic_source"),
                               "algorithmic_bytes_per_launch": int(algo_bytes), "ms_per_launch": round(ms_fwd, 4)},
        "kernels_ms": {k: round(v, 4) for k, v in phase_ms.items()},
    }
    if world == 1 and not args.no_cpu_baseline:
        lib, prefix, kind = cpu_pipeline_lib()
        # parity: frame 0 of batch 0 through the reference chain, every plane and every band decision
        t0 = time.perf_counter()
        want = cpu_frame(lib, prefix, geom, *batches[0][0], record=True)
        mism = 0
        for p in range(3):
            mism += int(zlib.crc32(want[p]["recon"].tobytes()) != dev_crc["recon%d" % p])
            mism += int(np.count_nonzero(dev_rec[p] != want[p]["rec"]))
        if DERING == 2:
            mism += int(np.count_nonzero(dev_levels != want[0]["dering_levels"]))
        out["parity_checked"] = {"frames": 1, "against": kind, "what": "reconstruction CRC-32 of 3 planes + every per-band "
                                 "(gain, theta, max_theta, K) of frame 0" + (" + the deringing level of every superblock"
                                                                           if DERING == 2 else ""), "mismatches": mism}
        if mism:
            # still print the line (flagged) so that the failure is visible in the record, then exit non-zero
            out["parity_failed"] = True
            sys.stderr.write("bench.py: device results differ from the oracle (%d mismatches): the numbers of this run "
                             "do not count\n" % mism)
        n = 0
        while time.perf_counter() - t0 < 12.0:
            cpu_frame(lib, prefix, geom, *batches[0][(n + 1) % F])
            n += 1
        dt = time.perf_counter() - t0
        out["cpu_baseline"] = {"value": round(geom.luma_pixels * (n + 1) / dt / 1e6, 3), "unit": UNIT, "cores": 1, "kind": kind,
                               "build": CPU_BUILD["build"],
                               "sample": "%d whole 3840x2160 frames, same chain (reference functions, pvq_theta speed=1, od_dering%s), "
                                         "1 thread, %.1f s" % (n + 1, " + level search" if DERING == 2 else "", dt)}
    print(json.dumps(out), flush=True)
    if world > 1:
        dist.destroy_process_group()
    if out.get("parity_failed"):
        sys.exit(1)


DUMP_LIMIT = 1 << 19


def dump_outputs(out, dirname):
    """Writes one step's result arrays (KeyframeEngine.wait()) as <name>.npy: integers of up to 16 bits as float32,
    wider integers and doubles as float64, block descriptors as one float64 column per field.  An array of more than
    DUMP_LIMIT values is sampled at DUMP_LIMIT positions drawn with a fixed seed from its size alone, so that two
    builds given the same arguments write comparable samples.  `counts` holds the device queues' scheduling
    counters, which vary from run to run, and is left out."""
    import numpy as np
    os.makedirs(dirname, exist_ok=True)
    for name, a in sorted(out.items()):
        if name == "counts":
            continue
        if a.dtype.names:
            a = np.stack([a[f].astype(np.float64) for f in a.dtype.names], axis=-1)
        flat = a.reshape(-1)
        if flat.size > DUMP_LIMIT:
            flat = flat[np.sort(np.random.default_rng(flat.size).integers(0, flat.size, DUMP_LIMIT))]
        small = flat.dtype.kind in "iub" and flat.dtype.itemsize <= 2
        np.save(os.path.join(dirname, name + ".npy"), flat.astype(np.float32 if small else np.float64))


def load_profile_notes():
    """DRAM traffic per launch from the committed ncu captures (profiles/r2_traffic.json), if present."""
    path = os.path.join(ROOT, "profiles", "r2_traffic.json")
    if os.path.exists(path):
        try:
            return json.load(open(path))
        except ValueError:
            pass
    return {}


def main():
    global BLOCK_SIZES, DERING
    args = parse()
    BLOCK_SIZES = args.block_sizes
    DERING = int(args.dering)
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
