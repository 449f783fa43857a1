#!/usr/bin/env python
"""Point selections on the device: the cost of building them, and the alignment step against them.

Workload: the default bench.py workload (512 seeded synthetic 640x480 pairs, 5 levels, FirstLevel 4, LastLevel 0, 50
iterations, precision 1e-4); the pyramids are built once, before timing.  Measured with CUDA events on the engine's stream:
  * build: dvo_b200_selection_create_device_batch of --selections selections (the 512 reference pyramids, cycled) with
    level-0 device masks (random blobs, GRADIENT_THRESHOLD(0, 0)), one call per step;
  * step: dvo_b200_match_batch_enqueue of the 512 pairs against the pyramids' own selections, and
    dvo_b200_match_batch_selected_enqueue of the same pairs against selections equal to them (no mask).  The result
    records of the two are checked byte for byte before timing.
Reported with the GPU's name and power limit queried in the same run.

  python scripts/selection_bench.py [--steps 10] [--warmup 3] [--batch 512] [--selections 1024]
"""
from __future__ import annotations

import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))
sys.dont_write_bytecode = True

from device_frames_bench import gpu_identity  # noqa: E402

W, H, LEVELS = 640, 480, 5


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batch", type=int, default=512)
    ap.add_argument("--selections", type=int, default=1024)
    args = ap.parse_args()

    import torch
    from dvo_slam_b200 import synth
    from dvo_slam_b200.engine import Config, Engine

    if not torch.cuda.is_available():
        raise SystemExit("selection_bench.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    B, NS = args.batch, args.selections
    scfg = synth.SceneConfig()
    K = scfg.intrinsics
    cfg = Config(first_level=4, last_level=0, max_iterations_per_level=50, precision=1e-4)

    I = torch.empty((2 * B, H, W), dtype=torch.float32, device=dev)
    Z = torch.empty((2 * B, H, W), dtype=torch.float32, device=dev)
    for i in range(B):
        p = synth.make_pair(i, scfg, device=dev)
        I[i], Z[i], I[B + i], Z[B + i] = p["I_ref"], p["Z_ref"], p["I_cur"], p["Z_cur"]
    # random blob masks, one per selection: about a third of every image excluded
    g = torch.Generator(device=dev).manual_seed(7)
    yy, xx = torch.meshgrid(torch.arange(H, device=dev), torch.arange(W, device=dev), indexing="ij")
    masks = torch.ones((NS, H, W), dtype=torch.uint8, device=dev)
    for _ in range(6):
        c = torch.rand((NS, 3), generator=g, device=dev) * torch.tensor([H, W, 0.12 * H], device=dev) + torch.tensor([0, 0, 0.08 * H], device=dev)
        masks[((yy[None] - c[:, 0, None, None]) ** 2 + (xx[None] - c[:, 1, None, None]) ** 2) < c[:, 2, None, None] ** 2] = 0
    torch.cuda.synchronize()

    eng = Engine(device=0)
    stream = torch.cuda.ExternalStream(eng.stream, device=dev)
    pyr = eng.pyramid_from_tensors(I, Z, K, LEVELS)
    refs, curs = pyr[:B], pyr[B:]
    sel_refs = [refs[i % B] for i in range(NS)]
    own = eng.selections_from_tensors(refs, None, 0, 0.0, 0.0)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        eng.synchronize()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(args.steps):
            fn()
        e1.record(stream)
        eng.synchronize()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / args.steps

    def build():
        for s in eng.selections_from_tensors(sel_refs, masks, 0, 0.0, 0.0):
            s.release()

    a = eng.match_batch_enqueue(refs, curs, cfg)
    b = eng.match_batch_enqueue(own, curs, cfg)
    eng.synchronize()
    torch.cuda.synchronize()
    parity = a.cpu().numpy().tobytes() == b.cpu().numpy().tobytes()
    if not parity:
        raise SystemExit("selected step disagrees with the pyramid step")

    build_ms = timed(build)
    step_pyr_ms = timed(lambda: eng.match_batch_enqueue(refs, curs, cfg))
    step_sel_ms = timed(lambda: eng.match_batch_enqueue(own, curs, cfg))
    rec_bytes = sum(((W >> l) + 127) // 128 * (((H >> l) + 6) // 7) for l in range(LEVELS)) * 14848
    line = {"metric": "selection build and selected alignment step @640x480x5-level",
            "build_ms": build_ms, "selections_per_build": NS, "build_us_per_selection": build_ms * 1e3 / NS,
            "record_bytes_per_selection": rec_bytes,
            "step_ms_pyramid_selection": step_pyr_ms, "step_ms_separate_selection": step_sel_ms,
            "step_ratio": step_sel_ms / step_pyr_ms, "batch": B, "steps": args.steps, "warmup": args.warmup,
            "parity": "byte-identical result records" if parity else "differs",
            "config": {"first_level": 4, "last_level": 0, "max_iterations_per_level": 50, "precision": 1e-4,
                       "masks": "random blobs, u8 [n,480,640] device tensor", "predicate": "GRADIENT_THRESHOLD(0, 0)"},
            "gpu": gpu_identity(0), "timer": "CUDA events on the engine stream"}
    print(json.dumps(line))
    del a, b, masks, I, Z    # marked as used on the engine's stream: freed before that stream goes away
    torch.cuda.synchronize()
    eng.close()


if __name__ == "__main__":
    main()
