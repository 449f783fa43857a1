#!/usr/bin/env python
"""Device-fed alignment throughput: frames already in GPU memory -> pyramids -> alignments -> results on the device.

Workload: the default bench.py workload (512 seeded synthetic 640x480 pairs, 5 levels, FirstLevel 4, LastLevel 0, 50
iterations, precision 1e-4), held on the GPU as 8-bit grey + 16-bit raw depth (uploaded once, before timing).  A timed
step is dvo_b200_pyramid_create_device_batch over the 1 024 frames, then dvo_b200_match_batch_enqueue with the initial
estimates (identity, use_initial_estimate = 1) in device memory; the result records stay on the device.  Steps are timed
with CUDA events on the engine's stream; the host never waits inside the timed window.  Reported: alignments/s, ms per
step, the build's share of a step, the bytes that crossed the bus per step (only the pair descriptors), and the GPU's name
and power limit queried in the same run.  Before timing, the step's result records are checked byte for byte against the
host-input path (dvo_b200_pyramid_create_raw_batch from host memory + dvo_b200_match_batch) on the same seeds.

  python scripts/device_frames_bench.py [--steps 10] [--warmup 3] [--batch 512]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True

import numpy as np  # noqa: E402

W, H, LEVELS = 640, 480, 5
SCALE = 1.0 / 5000.0


def gpu_identity(index: int) -> dict:
    """name and power limit of the card, as nvidia-smi reports them"""
    try:
        out = subprocess.run(["nvidia-smi", f"--id={index}", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=20).stdout.strip().splitlines()[0]
        name, power, clock = [c.strip() for c in out.split(",")]
        return {"name": name, "power_limit": power, "sm_clock_max": clock}
    except Exception as e:  # the numbers are still reported, marked as unidentified
        import torch
        return {"name": torch.cuda.get_device_name(index), "power_limit": None, "query_error": str(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=512)
    args = ap.parse_args()

    import torch
    from dvo_slam_b200 import synth
    from dvo_slam_b200.engine import Config, CResult, Engine

    if not torch.cuda.is_available():
        raise SystemExit("device_frames_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    B = args.batch
    scfg = synth.SceneConfig()
    K = scfg.intrinsics
    cfg = Config(first_level=4, last_level=0, max_iterations_per_level=50, precision=1e-4, use_initial_estimate=1)

    # ---- the frames, once: references then currents, 8-bit grey + 16-bit raw depth, resident on the GPU ----
    G = torch.empty((2 * B, H, W), dtype=torch.uint8, device=dev)
    D = torch.empty((2 * B, H, W), dtype=torch.int16, device=dev)
    for i in range(B):
        p = synth.make_pair(i, scfg, device=dev)
        for k, (I, Z) in ((i, (p["I_ref"], p["Z_ref"])), (B + i, (p["I_cur"], p["Z_cur"]))):
            G[k] = I.to(torch.uint8)
            D[k] = torch.where(torch.isnan(Z), torch.zeros_like(Z), torch.round(Z * 5000.0)).to(torch.int32).to(torch.int16)
    T_init = torch.eye(4, dtype=torch.float64, device=dev).repeat(B, 1, 1).contiguous()
    torch.cuda.synchronize()

    eng = Engine(device=0)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)

    def step():
        pyr = eng.pyramid_from_tensors(G, D, K, LEVELS, depth_scale=SCALE)
        rec = eng.match_batch_enqueue(pyr[:B], pyr[B:], cfg, T_init=T_init)
        for p in pyr:          # the slabs return to the pool; the next step's build reuses them in stream order
            p.release()
        return rec

    # ---- parity with the host-input path on the same seeds ----
    rec = step()
    eng.synchronize()
    torch.cuda.synchronize()
    hG, hD = G.cpu().numpy(), D.cpu().numpy().view(np.uint16)
    hp = eng.pyramid_raw_batch((hG.ctypes.data, hD.ctypes.data, 2 * B, H, W), SCALE, K, LEVELS)
    eng.synchronize()
    host = eng.match_batch(hp[:B], hp[B:], cfg, T_init=np.tile(np.eye(4), (B, 1, 1)), raw=True)
    for p in hp:
        p.release()
    parity = rec.cpu().numpy().tobytes() == bytes(memoryview(host))
    if not parity:
        raise SystemExit("device-fed step disagrees with the host-input path")
    del hG, hD

    # ---- timed steps ----
    for _ in range(args.warmup):
        step()
    eng.synchronize()
    torch.cuda.synchronize()
    h2d0, d2h0 = eng.h2d_bytes(), eng.d2h_bytes()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(args.steps):
        rec = step()
    e1.record(stream)
    eng.synchronize()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    h2d = (eng.h2d_bytes() - h2d0) / args.steps
    d2h = (eng.d2h_bytes() - d2h0) / args.steps

    # ---- the build alone (same events, separate window) ----
    b0, b1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    b0.record(stream)
    for _ in range(args.steps):
        for p in eng.pyramid_from_tensors(G, D, K, LEVELS, depth_scale=SCALE):
            p.release()
    b1.record(stream)
    eng.synchronize()
    build_ms = b0.elapsed_time(b1) / args.steps

    line = {"metric": "device-fed frame-pair alignments/sec @640x480x5-level", "value": B / (ms * 1e-3), "unit": "alignments/s",
            "ms_per_step": ms, "build_ms_per_step": build_ms, "steps": args.steps, "warmup": args.warmup,
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "frame_bytes_per_step_avoided": 2 * B * W * H * 3,
            "result_record_bytes": C.sizeof(CResult),
            "parity_with_host_input_path": "byte-identical result records" if parity else "differs",
            "config": {"workload": f"batch={B} pairs, {2 * B} frames resident as u8 grey + u16 raw depth", "first_level": 4,
                       "last_level": 0, "max_iterations_per_level": 50, "precision": 1e-4, "use_initial_estimate": 1,
                       "T_init": "identity, device memory"},
            "gpu": gpu_identity(0), "timer": "CUDA events on the engine stream"}
    print(json.dumps(line))
    eng.close()


if __name__ == "__main__":
    main()
