#!/usr/bin/env python
"""bench.py -- frame-pair alignments/sec @640x480x5-level (BASELINE.json metric) on N B200s.

A "step" = one pass of the hot path (DenseTracker::match, all levels, all iterations, 6x6 solves)
over one batch of synthetic frame pairs.  Workload at every N: 512 independent 640x480 pairs PER GPU
(configs[2]; configs[3] = 4096 pairs over 8 GPUs is the same per-GPU batch -> weak scaling).

  value  : alignments/s with the pyramids already resident in HBM (device time, CUDA events on the
           engine stream, max over ranks)
  e2e    : the same metric through the public C-ABI call sequence with HOST buffers: pinned host
           images (8-bit grey + 16-bit raw depth, as the reference's loader holds them) ->
           dvo_b200_pyramid_create_raw_batch (H2D + conversion + pyramid build) -> dvo_b200_match_batch ->
           results on the host (D2H), every step
  roofline: the persistent per-level kernel k_level_persistent (both stages of every Gauss-Newton iteration), algorithmic
           40 B per pixel-iteration (SURVEY.md 8d) / their device time measured with CUDA events
  cpu_baseline: the reference's CPU path, match-only, on the box's host cores (bounded sample).  kind
           "reference" = every per-point pass (warp/residual, weights, scale, LL, normal equations) executed by
           the reference's own SSE object code (oracle/_ref/libdvo_ref_O3.so: dense_tracking_impl.cpp,
           core/math_sse.cpp, core/intrinsic_matrix.cpp compiled unmodified at the reference's -O3 -msse3; the
           match() control flow around them is oracle/ref_driver.cpp).  kind "port" (fallback when oracle/_ref
           is absent) = the oracle's scalar FAITHFUL restatement.
  --impl reference: the same CPU implementation from host images (pyramid build + match), all host threads.
  --config 5: BASELINE.json configs[4] (1280x960, 6 levels, mu = 0.05, 32 pairs per GPU = 256 over 8 GPUs).
  --dump-outputs DIR: after the timed steps, the result records of the last timed step (every pair of the global batch,
           in pair order) as DIR/<field>.npy in float64, so that two builds can be compared output for output: the inputs
           are seeded and the same for the same arguments.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True     # the benchmark writes nothing into the tree it runs from

import numpy as np  # noqa: E402

W, H, LEVELS = 640, 480, 5
FIRST_LEVEL, LAST_LEVEL, MAX_IT, PRECISION = 4, 0, 50, 1e-4   # benchmark.yaml:3-4 values, 5 levels
MU = 0.0
ALGO_BYTES_PER_PIXEL_ITERATION = 40.0                         # SURVEY.md 8(d)
LEVEL_PIXELS = [(W >> l) * (H >> l) for l in range(LEVELS)]
METRIC = "frame-pair alignments/sec @640x480x5-level"
DEFAULT_BATCH = 512


def select_workload(config: int):
    """configs[2]/[3] (default) or configs[4] of BASELINE.json; sets the module-level workload constants."""
    global W, H, LEVELS, FIRST_LEVEL, MU, LEVEL_PIXELS, METRIC, DEFAULT_BATCH
    if config == 5:
        W, H, LEVELS, FIRST_LEVEL, MU, DEFAULT_BATCH = 1280, 960, 6, 5, 0.05, 32
        METRIC = "frame-pair alignments/sec @1280x960x6-level"
    elif config not in (0, 2, 3, 4):
        raise SystemExit(f"unknown --config {config} (2/3 = 640x480x5 batch 512 per GPU [default], 5 = 1280x960x6 mu=0.05 batch 32 per GPU)")
    LEVEL_PIXELS = [(W >> l) * (H >> l) for l in range(LEVELS)]


def scene_config():
    """640x480: fr1 intrinsics; 1280x960 = the same camera upsampled 2x (configs[4]: "upsampled TUM fr1")."""
    from dvo_slam_b200 import synth
    if W == 640:
        return synth.SceneConfig()
    f = W / 640.0
    fx, fy, ox, oy = synth.FR1_INTRINSICS
    return synth.SceneConfig(width=W, height=H, intrinsics=(fx * f, fy * f, ox * f + (f - 1) / 2, oy * f + (f - 1) / 2))


def source_stamp() -> str:
    """sha256 over the CUDA sources the level kernel is built from: ties a profile to a build."""
    import glob
    import hashlib
    h = hashlib.sha256()
    for p in sorted(glob.glob(os.path.join(ROOT, "dvo_slam_b200", "csrc", "*"))):
        if p.endswith((".cu", ".cuh", ".h")):
            h.update(os.path.basename(p).encode())
            h.update(open(p, "rb").read())
    return h.hexdigest()[:16]


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="frame pairs per GPU (0 = the workload's default: 512, or 32 for --config 5)")
    ap.add_argument("--config", type=int, default=2, help="BASELINE.json configs index + 1 style: 2/3 = 640x480x5 (default), 5 = 1280x960x6 mu=0.05")
    ap.add_argument("--cpu-sample", type=int, default=0, help="pairs in the CPU baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-consecutive", action="store_true", help="skip the consecutive-frames e2e leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the results of the last timed step as DIR/<field>.npy (float64)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def dump_outputs(directory: str, records: np.ndarray, num_levels: int):
    """records: dvo_b200_result records (numpy view with the dtype of engine.CResult), one per pair.  Writes every field a
    caller of dvo_b200_match_batch receives, as float64, the per-level statistics for the levels the configuration runs."""
    os.makedirs(directory, exist_ok=True)
    out = {name: records[name] for name in records.dtype.names if name != "levels"}
    out["transformation"] = out["transformation"].reshape(-1, 4, 4)
    out["information"] = out["information"].reshape(-1, 6, 6)
    levels = records["levels"][:, :num_levels]
    for name in levels.dtype.names:
        out["levels_" + name] = levels[name]
    for name, a in out.items():
        np.save(os.path.join(directory, name + ".npy"), np.ascontiguousarray(a, dtype=np.float64))


# ---------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    """Polls nvidia-smi every 200 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.stop_flag, self.thread = index, [], threading.Event(), None

    def _loop(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.splitlines()[0].split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def start(self):
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        self.stop_flag.set()
        if self.thread:
            self.thread.join(timeout=10)
        sm, mx, pw, reasons = [], [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1])); pw.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "reasons": sorted(reasons), "samples": len(sm)}


def usable_cores() -> int:
    """Host threads this process may really use: min(visible CPUs, cgroup CPU quota)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:
        pass
    return n


# ---------------------------------------------------------------------------------------------
# CPU arm (oracle = test infrastructure; only this leg of bench.py may execute it)
# ---------------------------------------------------------------------------------------------
def cpu_kind():
    """("reference", variant) when the reference's compiled translation units are present, else ("port", None)."""
    from oracle import oracle_py as orc
    for variant in ("_O3", ""):
        if orc.ref_available(variant):
            return "reference", variant
    return "port", None


def cpu_kind_text(kind, variant):
    if kind == "reference":
        return ("reference SSE object code (oracle/_ref/libdvo_ref%s.so = dense_tracking_impl.cpp + core/math_sse.cpp + "
                "core/intrinsic_matrix.cpp compiled unmodified, %s) for every per-point pass; match() control flow, LDLT and "
                "SE(3) from oracle/ref_driver.cpp; pyramids from the oracle port" % (variant, "-O3 -msse3" if variant == "_O3" else "-O2 -msse3"))
    return "oracle scalar FAITHFUL port (oracle/_ref absent)"


def cpu_alignments(pairs, include_pyramid: bool, threads: int):
    """Runs DenseTracker::match on `pairs` with `threads` host threads through the reference's object code
    (oracle/_ref) when present, else the oracle FAITHFUL port; returns (seconds, n)."""
    from oracle import oracle_py as orc
    orc.lib()
    K = pairs[0]["intrinsics"]
    cfg = orc.config(first_level=FIRST_LEVEL, last_level=LAST_LEVEL, max_iterations_per_level=MAX_IT, precision=PRECISION, mu=MU)
    mode = orc.mode("faithful")
    kind, variant = cpu_kind()

    def pyramids(p):
        r = orc.Pyramid(p["I_ref"], p["Z_ref"], K, LEVELS)
        c = orc.Pyramid(p["I_cur"], p["Z_cur"], K, LEVELS)
        if kind == "reference":
            return orc.RefPyramid(r, variant), orc.RefPyramid(c, variant)
        return r, c

    prebuilt = None
    if not include_pyramid:
        prebuilt = [pyramids(p) for p in pairs]
    idx = list(range(len(pairs)))
    lock = threading.Lock()

    def worker():
        while True:
            with lock:
                if not idx:
                    return
                i = idx.pop()
            r, c = pyramids(pairs[i]) if include_pyramid else prebuilt[i]
            if kind == "reference":
                orc.ref_match(r, c, cfg)
            else:
                orc.match(r, c, cfg, mode, max_iters=8)

    t0 = time.perf_counter()
    ths = [threading.Thread(target=worker) for _ in range(threads)]
    for t in ths:
        t.start()
    for t in ths:
        t.join()
    return time.perf_counter() - t0, len(pairs)


def host_pairs(seeds, device="cpu"):
    from dvo_slam_b200 import synth
    out = []
    for s in seeds:
        p = synth.make_pair(s, scene_config(), device=device)
        out.append({k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in p.items()})
    return out


def run_reference(args, rank, world):
    """Reference arm: the reference's CPU implementation of the path on the host cores (see cpu_kind_text)."""
    if rank != 0:
        return
    cores = usable_cores()
    per_step = args.cpu_sample or max(cores, min(4 * cores, 64))
    dev = "cpu"
    try:
        import torch
        if torch.cuda.is_available():
            dev = "cuda:0"
    except Exception:
        pass
    pairs = host_pairs(range(per_step), device=dev)
    for _ in range(min(args.warmup, 1)):
        cpu_alignments(pairs[:cores], True, cores)
    t_total, n_total = 0.0, 0
    for _ in range(args.steps):
        t, n = cpu_alignments(pairs, True, cores)
        t_total += t
        n_total += n
    value = n_total / t_total
    kind, variant = cpu_kind()
    sample = f"{per_step} pairs/step x {args.steps} steps, pyramid build + match from host images, {cores} threads; {cpu_kind_text(kind, variant)}"
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "alignments/s", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1e3 * t_total / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{per_step}-pair sample of the batch={args.batch or DEFAULT_BATCH}/GPU {W}x{H} {LEVELS}-level workload",
                       "first_level": FIRST_LEVEL, "last_level": LAST_LEVEL, "max_iterations_per_level": MAX_IT, "precision": PRECISION,
                       "mu": MU},
            "cpu_baseline": {"value": value, "unit": "alignments/s", "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "alignments/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "note": "the reference's build system needs Eigen3/OpenCV2/Sophus/ROS (absent here); its hot-path translation units "
                    "compile unmodified against header-only container shims (oracle/ref_shim) and are what this arm executes"
                    if kind == "reference" else "oracle/_ref absent: timed arm is the oracle's scalar FAITHFUL port"}
    emit(json.dumps(line))


# ---------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    from dvo_slam_b200 import synth
    from dvo_slam_b200.distributed import tensor_to_results
    from dvo_slam_b200.engine import Config, Engine, CResult

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    B = args.batch or DEFAULT_BATCH
    total = B * world
    eng = Engine(device=local_rank)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    cfg = Config(first_level=FIRST_LEVEL, last_level=LAST_LEVEL, max_iterations_per_level=MAX_IT, precision=PRECISION, mu=MU)
    scfg = scene_config()
    K = scfg.intrinsics

    # ---- synthetic batch: distinct seeded pairs, rendered on the GPU, kept in pinned host memory ----
    npx = W * H
    hI = torch.empty((2 * B, H, W), dtype=torch.float32).pin_memory()
    hZ = torch.empty((2 * B, H, W), dtype=torch.float32).pin_memory()
    for i in range(B):
        p = synth.make_pair(rank * B + i, scfg, device=dev)
        hI[i].copy_(p["I_ref"]); hZ[i].copy_(p["Z_ref"])
        hI[B + i].copy_(p["I_cur"]); hZ[B + i].copy_(p["Z_cur"])
    torch.cuda.synchronize()
    # The same images as the loader of the reference holds them before conversion (benchmark_slam.cpp:46-93):
    # 8-bit grey and 16-bit raw depth (1/5000 m, 0 = invalid).  The synthetic images are integer-valued and
    # quantised to 1/5000 m, so this representation is lossless; the e2e leg uploads these (N2 row).
    hG = hI.to(torch.uint8).pin_memory()
    raw = torch.where(torch.isnan(hZ), torch.zeros_like(hZ), torch.round(hZ * 5000.0)).to(torch.int32)
    hD = raw.to(torch.uint16).pin_memory()
    assert torch.equal(hG.to(torch.float32), hI)
    # float32 depth exactly as convertRawDepthImageSse produces it (u16 * (1/5000)f, 0 -> NaN), so that the
    # resident leg (float32 API) and the e2e leg (raw API) see bit-identical inputs
    hZ.copy_(torch.where(raw == 0, torch.full_like(hZ, float("nan")), raw.to(torch.float32) * torch.tensor(1.0 / 5000.0, dtype=torch.float32)))
    del raw
    h2d_per_step = (2 * B) * npx * 3
    d2h_per_step = B * C.sizeof(CResult)

    def build_pyramids():
        pyrs = eng.pyramid_batch(None, None, K, LEVELS, host_ptrs=(hI.data_ptr(), hZ.data_ptr(), 2 * B, H, W))
        return pyrs[:B], pyrs[B:]

    refs, curs = build_pyramids()
    eng.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(steps):
            fn()
        e1.record(stream)
        barrier()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    last = {}

    # N > 1: the one exchange of the path -- an all-gather of the fixed-size result records -- is part of every step:
    # results are written to device memory (dvo_b200_match_batch_device), gathered over NCCL on the engine's
    # stream, and the gathered table is read back to the host (what dvo_slam's single-process callers consume).
    if world > 1:
        d_local = torch.zeros((B, C.sizeof(CResult)), dtype=torch.uint8, device=dev)
        d_all = torch.zeros((total, C.sizeof(CResult)), dtype=torch.uint8, device=dev)
        h_all = torch.zeros((total, C.sizeof(CResult)), dtype=torch.uint8).pin_memory()

    def step_resident():
        if world == 1:
            last["res"] = eng.match_batch(refs, curs, cfg, raw=True)
            return
        eng.match_batch_device(refs, curs, cfg, d_local.data_ptr())
        with torch.cuda.stream(stream):
            dist.all_gather_into_tensor(d_all, d_local)
            h_all.copy_(d_all, non_blocking=True)
        eng.synchronize()
        last["gathered"] = h_all

    # e2e: every step goes host images (8-bit grey, 16-bit raw depth, pinned) -> dvo_b200_pyramid_create_raw_batch
    # -> dvo_b200_match_batch -> host results through the public C ABI.  A double-buffered front end on two host
    # threads, each with its own context/stream (the reference's one-tracker-per-thread model): the loader
    # thread uploads the 2B images of a step in one call and builds their pyramids while the tracker thread
    # aligns the previous step's pairs.  All copies of all timed steps lie inside the timed region.
    import queue
    engines = [eng, Engine(device=local_rank)]
    from concurrent.futures import ThreadPoolExecutor
    pool = ThreadPoolExecutor(2)

    def e2e_loader(steps, q):
        for _ in range(steps):
            # references then currents, contiguous in host memory: the whole upload is enqueued before the first
            # build kernel
            pyr = engines[1].pyramid_raw_batch((hG.data_ptr(), hD.data_ptr(), 2 * B, H, W), 1.0 / 5000.0, K, LEVELS)
            # hand the batch over only when its pyramids are complete: the tracker's persistent launch needs every SM at once, and
            # a loader that runs further ahead interleaves its build kernels with that launch (measured: 28.6 vs 24.0 ms per step)
            engines[1].synchronize()
            q.put(pyr)

    done_at = []

    def e2e_tracker(steps, q):
        out = None
        for _ in range(steps):
            pyr = q.get()
            out = engines[0].match_batch(pyr[:B], pyr[B:], cfg, raw=True)
            done_at.append(time.perf_counter())
            for p in pyr:
                p.release()
        return out

    def run_e2e(steps):
        q = queue.Queue(maxsize=1)    # the loader runs at most one finished step ahead
        f0 = pool.submit(e2e_loader, steps, q)
        f1 = pool.submit(e2e_tracker, steps, q)
        f0.result()
        last["res_e2e"] = f1.result()

    # ---- value: resident pyramids ----
    for _ in range(args.warmup):
        step_resident()
    eng.profile_read(reset=True)
    eng.profile_enable(True)
    launches0 = eng.kernel_launches()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    ms_total = timed(step_resident, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    launches = eng.kernel_launches() - launches0
    prof = eng.profile_read(reset=True)
    eng.profile_enable(False)
    ms_per_step = ms_total / args.steps
    value = total / (ms_per_step * 1e-3)

    # pixel-iterations actually executed in one step on this rank (from the results' statistics)
    if world > 1:
        assert last["gathered"].shape[0] == total
        res = tensor_to_results(last["gathered"][rank * B:(rank + 1) * B])
    else:
        res = last["res"]
    if args.dump_outputs and rank == 0:
        records = last["gathered"].numpy().view(np.dtype(CResult)).reshape(-1) if world > 1 else np.frombuffer(res, dtype=np.dtype(CResult))
        dump_outputs(args.dump_outputs, records, FIRST_LEVEL - LAST_LEVEL + 1)
    pix_iters = 0
    it_hist = [0] * LEVELS
    for i in range(B):
        for l in range(res[i].num_levels):
            ls = res[i].levels[l]
            pix_iters += LEVEL_PIXELS[ls.id] * ls.num_iterations
            it_hist[ls.id] += ls.num_iterations
    stage_ms = (prof["residual"]["ms"] + prof["normal"]["ms"]) / args.steps
    stage_launches = (prof["residual"]["launches"] + prof["normal"]["launches"]) / args.steps
    algo_bytes = ALGO_BYTES_PER_PIXEL_ITERATION * pix_iters
    peaks = {}
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            peaks = json.load(f)
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = algo_bytes / (stage_ms * 1e-3) / 1e9 if stage_ms > 0 else 0.0
    # DRAM traffic of the dominant launch from the committed `ncu --set full` capture of THIS build (profiles/,
    # regenerated by scripts/gpu_ncu.sh + scripts/make_traffic_json.py, which stamps the hash of the CUDA sources);
    # a capture of another build is reported as stale and not used
    traffic, traffic_note = None, None
    if W == 640 and B == 512:
        try:
            with open(os.path.join(ROOT, "profiles", "r02_traffic.json")) as f:
                tj = json.load(f)
            if tj.get("source_stamp") == source_stamp():
                traffic, traffic_note = tj["dram_bytes_per_step"] / tj["launches_per_step"], tj["note"]
            else:
                traffic_note = "stale: profiles/r02_traffic.json was captured from sources %s, this build is %s" % (tj.get("source_stamp"), source_stamp())
        except Exception as e:
            traffic_note = f"no capture: {e}"
    else:
        traffic_note = "capture exists for the default workload only"

    # ---- e2e: host buffers in, host results out, every step ----
    run_e2e(max(2, min(args.warmup, 4)))
    h2d0, d2h0 = sum(e.h2d_bytes() for e in engines), sum(e.d2h_bytes() for e in engines)
    barrier()
    t0 = time.perf_counter()          # two streams are involved: host clock between full device synchronisations
    del done_at[:]
    run_e2e(args.steps)
    barrier()
    ms_local = torch.tensor([(time.perf_counter() - t0) * 1e3 / args.steps], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(ms_local, op=dist.ReduceOp.MAX)
    ms_e2e = float(ms_local.item())
    h2d_meas = (sum(e.h2d_bytes() for e in engines) - h2d0) / args.steps
    d2h_meas = (sum(e.d2h_bytes() for e in engines) - d2h0) / args.steps
    e2e_value = total / (ms_e2e * 1e-3)
    # interval between the completions of consecutive steps once the two-stage pipeline is full (the timed region above also
    # contains the fill: the first upload has nothing to overlap with)
    gaps = [1e3 * (b_ - a_) for a_, b_ in zip(done_at[1:-1], done_at[2:])]
    ms_e2e_steady = statistics.median(gaps) if gaps else None
    # the e2e path must give the same answers as the resident path (identical inputs through the raw-input
    # entry point: agreement to the stated SE(3) tolerance, typically bit-identical)
    worst = 0.0
    for j in range(B):
        a_, b_ = np.array(last["res_e2e"][j].transformation), np.array(res[j].transformation)
        worst = max(worst, float(np.abs(a_ - b_).max()))
    if not worst < 2e-3:
        raise SystemExit(f"e2e leg disagrees with the resident leg: max |dT| = {worst}")

    # ---- e2e on CONSECUTIVE frames (dvo_slam's odometry workload, local_tracker.cpp:172-184: frame k is the current image of
    # alignment k-1 and the reference of alignment k): B alignments over sequences of 17 frames, every frame uploaded and its
    # pyramid built ONCE per step.  Reported next to the headline e2e (which uploads 2B images for B independent pairs).
    e2e_seq = None
    if not args.no_consecutive and W == 640:
        SEQ = 16                                   # alignments per sequence
        nseq = (B + SEQ - 1) // SEQ
        nfr = nseq * (SEQ + 1)
        sG = torch.empty((nfr, H, W), dtype=torch.uint8).pin_memory()
        sD = torch.empty((nfr, H, W), dtype=torch.uint16).pin_memory()
        for q in range(nseq):
            frames, _ = synth.make_sequence(10000 + rank * nseq + q, SEQ + 1, scfg, device=dev)
            for k, (fi, fz) in enumerate(frames):
                sG[q * (SEQ + 1) + k].copy_(fi.to(torch.uint8))
                sD[q * (SEQ + 1) + k].copy_(torch.where(torch.isnan(fz), torch.zeros_like(fz), torch.round(fz * 5000.0)).to(torch.int32).to(torch.uint16))
        torch.cuda.synchronize()
        ref_idx = [q * (SEQ + 1) + k for q in range(nseq) for k in range(SEQ)][:B]

        def seq_loader(steps, q):
            for _ in range(steps):
                pyr = engines[1].pyramid_raw_batch((sG.data_ptr(), sD.data_ptr(), nfr, H, W), 1.0 / 5000.0, K, LEVELS)
                engines[1].synchronize()
                q.put(pyr)

        def seq_tracker(steps, q):
            out = None
            for _ in range(steps):
                pyr = q.get()
                out = engines[0].match_batch([pyr[i] for i in ref_idx], [pyr[i + 1] for i in ref_idx], cfg, raw=True)
                for p in pyr:
                    p.release()
            return out

        def run_seq(steps):
            q = queue.Queue(maxsize=1)
            f0 = pool.submit(seq_loader, steps, q)
            f1 = pool.submit(seq_tracker, steps, q)
            f0.result()
            return f1.result()

        run_seq(2)
        barrier()
        t0 = time.perf_counter()
        res_seq = run_seq(args.steps)
        barrier()
        ms_seq = torch.tensor([(time.perf_counter() - t0) * 1e3 / args.steps], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms_seq, op=dist.ReduceOp.MAX)
        ms_seq = float(ms_seq.item())
        e2e_seq = {"value": total / (ms_seq * 1e-3), "unit": "alignments/s", "ms_per_step": ms_seq,
                   "h2d_bytes_per_step": nfr * npx * 3, "d2h_bytes_per_step": d2h_per_step,
                   "workload": f"{nseq} sequences of {SEQ + 1} consecutive frames per GPU = {B} alignments, each frame uploaded once",
                   "iterations_total_mean": float(np.mean([res_seq[i].num_iterations_total for i in range(B)]))}

    # ---- single-pair latency (configs[1]) ----
    lat_ms = None
    if rank == 0:
        for _ in range(3):
            eng.match_batch(refs[:1], curs[:1], cfg, raw=True)
        t0 = time.perf_counter()
        for _ in range(10):
            eng.match_batch(refs[:1], curs[:1], cfg, raw=True)
        lat_ms = (time.perf_counter() - t0) / 10 * 1e3

    # ---- CPU baseline: the reference's CPU path, match only, bounded sample (rank 0, N=1 only) ----
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cores = usable_cores()
        nsample = args.cpu_sample or max(cores, min(4 * cores, 64))
        hp = [{"I_ref": hI[i].numpy(), "Z_ref": hZ[i].numpy(), "I_cur": hI[B + i].numpy(), "Z_cur": hZ[B + i].numpy(),
               "intrinsics": K} for i in range(min(nsample, B))]
        t1, n1 = cpu_alignments(hp[: max(2, min(8, len(hp)))], False, 1)
        tc, nc = cpu_alignments(hp, False, cores)
        kind, variant = cpu_kind()
        cpu = {"value": nc / tc, "unit": "alignments/s", "cores": cores, "kind": kind,
               "sample": f"first {len(hp)} pairs of the batch, match() on prebuilt pyramids, {cores} threads; {cpu_kind_text(kind, variant)}",
               "value_1core": n1 / t1}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "alignments/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic",
                "config": {"workload": f"batch={B} independent {W}x{H} frame pairs per GPU, {LEVELS}-level pyramid (FirstLevel={FIRST_LEVEL}, LastLevel=0)",
                           "global_batch": total, "max_iterations_per_level": MAX_IT, "precision": PRECISION, "mu": MU,
                           "parallelism": f"pairs sharded over {world} GPU(s), no collective inside the alignments; one NCCL all-gather of the "
                                          f"result records per step" + (", inside the timed region" if world > 1 else " (N=1: none)"),
                           "l2": "inputs larger than L2: %.1f GB of pyramids per GPU" % (2 * B * sum(LEVEL_PIXELS) * 32 / 1e9),
                           "iterations_per_level_mean": [it_hist[l] / B for l in range(LEVELS)]},
                "e2e": {"value": e2e_value, "unit": "alignments/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d_per_step,
                        "d2h_bytes_per_step": d2h_per_step, "h2d_bytes_counted": h2d_meas, "d2h_bytes_counted": d2h_meas,
                        "pipeline": "loader thread/context uploads the images of step i+1 while the tracker thread/context aligns step i; their pyramids are built when "
                                    "the level kernel releases the SMs, and the batch is handed over once complete",
                        "timer": "host clock between device synchronisations, max over ranks",
                        "steady_state_ms_per_step": ms_e2e_steady,
                        "steady_state_note": "median interval between step completions on this rank after the pipeline fill (informative; value = whole timed region)"},
                "gpu_launches": int(launches),
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
                             "traffic": traffic, "traffic_note": traffic_note, "kernel": "k_level_persistent (persistent cooperative kernel; one launch per level group: coarse levels walked in one launch, "
                                       "fine levels in another; bulk-copy staged tiles, warp+residual+weight+scale, LL+J^T W J, on-device solve)",
                             "source_stamp": source_stamp(),
                             "algorithmic_bytes_per_step": algo_bytes, "kernel_ms_per_step": stage_ms,
                             "algorithmic_bytes_per_launch": algo_bytes / stage_launches if stage_launches else None,
                             "kernel_ms_per_launch": stage_ms / stage_launches if stage_launches else None,
                             "launches_per_step": stage_launches,
                             "peak_source": "MEASURED_PEAKS.json hbm_gbs (of measured)" if peaks else "fallback 6650 GB/s (of fallback)",
                             "kernel_share_of_step": stage_ms / ms_per_step if ms_per_step else None,
                             "pair_step_ms_per_step": prof["pair_step"]["ms"] / args.steps},
                "e2e_consecutive_frames": e2e_seq,
                "cpu_baseline": cpu, "clocks": clocks, "single_pair_latency_ms": lat_ms}
        emit(json.dumps(line))


def main():
    args = parse_args()
    select_workload(args.config)
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"      # rank 0 prints exactly one line on stdout: no NCCL version banner
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


_JSON_OUT = None


def emit(text):
    """The one JSON line of the contract, on the process's ORIGINAL stdout."""
    out = _JSON_OUT or sys.stdout
    out.write(text + "\n")
    out.flush()


def _reserve_stdout():
    """Rank 0 prints exactly one line on stdout.  Libraries write there too (NCCL prints its version banner at
    NCCL_DEBUG=VERSION and above, whatever this process sets later): keep a private handle on the original stdout for the JSON
    line and point file descriptor 1 at stderr for everything else."""
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


if __name__ == "__main__":
    _reserve_stdout()
    main()
