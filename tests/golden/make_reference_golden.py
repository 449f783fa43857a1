"""Generates tests/golden/reference_pin.npz: what the original dvo_core's own SSE object code computes on the golden pairs.

oracle/_ref/libdvo_ref.so and libdvo_ref_O3.so are the original dense_tracking_impl.cpp, core/math_sse.cpp and
core/intrinsic_matrix.cpp compiled unmodified (`make -C oracle ref REF=<dvo_core source directory>`), driven by
oracle/ref_driver.cpp.  They can only be built where those sources are, so tests/test_reference_pin.py compares the oracle
with the numbers stored here.  Run from the repo root, after building them:  python tests/golden/make_reference_golden.py

Per-pixel records are stored as a digest (helpers.nan_digest) of the whole dense record planes, which pins them bit for
bit, plus the values at a seeded sample of valid pixels, which keeps a failure readable; everything else is stored whole.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))
from dvo_slam_b200 import synth  # noqa: E402
from helpers import GOLDEN_LEVELS, GOLDEN_SEEDS, REFERENCE_GOLDEN, golden_images, load_golden, nan_digest  # noqa: E402
from oracle import oracle_py as orc  # noqa: E402

SAMPLE = 128          # record samples per golden pair and level
THRESHOLDS = ((0.0, 0.0), (2.0, 0.02))


def dense(r, h, w):
    """scatter the reference's compacted records {point (4), i, z, idx, idy, zdx, zdy, -, -} into seven h*w planes"""
    d = np.full((7, h * w), np.nan, np.float32)
    d[0:6, r["index"]] = r["records"][:, 4:10].T
    d[6, r["index"]] = r["records"][:, 2]
    return d


def pyramids(im, K, levels):
    return orc.Pyramid(im["I_ref"], im["Z_ref"], K, levels), orc.Pyramid(im["I_cur"], im["Z_cur"], K, levels)


def match_cases():
    """Whole alignments: the golden pairs (3 levels), and two 640x480 five-level pairs, the second with mu and an initial
    estimate.  Returns (images, K, levels, config, T_init) per case."""
    cases = []
    for seed in GOLDEN_SEEDS:
        g = load_golden(seed)
        im = golden_images(g, orc)
        cases.append((im, g["K"], GOLDEN_LEVELS, dict(first_level=2, last_level=0, max_iterations_per_level=50, precision=1e-4), None))
    for seed, extra in ((3, {}), (5, dict(mu=0.05, use_initial_estimate=1))):
        p = synth.make_pair(seed)
        im = {k: p[k].numpy() for k in ("I_ref", "Z_ref", "I_cur", "Z_cur")}
        cfg = dict(first_level=4, last_level=0, max_iterations_per_level=50, precision=1e-4)
        cfg.update(extra)
        cases.append((im, p["intrinsics"], 5, cfg, synth.se3_exp(p["xi"] * 0.8) if extra else None))
    return cases


def odd_point_margin(g, im):
    """The first margin for which the masked reference frame selects an odd number of points whose last one is valid
    by itself (see test_intensity_error_image_walk_equals_reference_valid_flag_stream)."""
    for margin in range(4, 40):
        Z = im["Z_ref"].copy()
        Z[-margin:, :] = np.nan
        Z[:, -margin:] = np.nan
        oref = orc.Pyramid(im["I_ref"], Z, g["K"], 1)
        ocur = orc.Pyramid(im["I_ref"], im["Z_ref"], g["K"], 1)
        S, mask = orc.select(oref, 0, 0.0, 0.0, None)
        last = np.flatnonzero(mask.reshape(-1))[-1]
        _, planes_exact = orc.residual_image(oref, ocur, 0, np.eye(4), orc.mode("exact"))
        if S % 2 == 1 and not np.isnan(planes_exact[0].reshape(-1)[last]):
            return margin, oref, ocur
    raise RuntimeError("no margin gave an odd selection count with a valid last point")


def main():
    for variant in ("", "_O3"):
        if not orc.ref_available(variant):
            raise SystemExit(f"oracle/_ref/libdvo_ref{variant}.so is missing: make -C oracle ref REF=<dvo_core source directory>")
    out = {}
    for seed in GOLDEN_SEEDS:
        g = load_golden(seed)
        im = golden_images(g, orc)
        oref, ocur = pyramids(im, g["K"], GOLDEN_LEVELS)
        rref, rcur = orc.RefPyramid(oref), orc.RefPyramid(ocur)
        for lvl in range(GOLDEN_LEVELS):
            w, h, K = oref.level_info(lvl)
            key = f"lin_{seed}_l{lvl}"
            for uw in (0, 1):
                r = orc.ref_linearize(oref.planes(lvl), ocur.planes(lvl), K, g["kat_T"], bool(uw), g["kat_prev_precision"])
                for name in ("precision", "A", "b"):
                    out[f"{key}_w{uw}_{name}"] = r[name]
                out[f"{key}_w{uw}_ll"] = np.float32(r["ll"])
            # the records do not depend on the weights: the last call's stand for both
            d = dense(r, h, w)
            pix = np.sort(np.random.default_rng(1000 * seed + lvl).choice(r["index"], SAMPLE, replace=False)).astype(np.int32)
            out[f"{key}_n_selected"], out[f"{key}_n"] = np.int64(r["n_selected"]), np.int64(r["n"])
            out[f"{key}_records_digest"] = np.array(nan_digest(d))
            out[f"{key}_sample_pixels"], out[f"{key}_sample"] = pix, d[:, pix]
            # the original build's own -O3
            r3 = orc.ref_linearize(oref.planes(lvl), ocur.planes(lvl), K, g["kat_T"], True, g["kat_prev_precision"], variant="_O3")
            d3 = dense(r3, h, w)
            key3 = f"o3_{seed}_l{lvl}"
            out[f"{key3}_n"] = np.int64(r3["n"])
            out[f"{key3}_nan_digest"] = np.array(nan_digest(np.isnan(d3)))
            out[f"{key3}_sample"] = d3[:, pix]
            for name in ("precision", "A", "b"):
                out[f"{key3}_{name}"] = r3[name]
            # computeIntensityErrorImage fed by the original computeResidualsAndValidFlagsSse
            for j, (ti, td) in enumerate(THRESHOLDS):
                n, img = orc.ref_intensity_error_image(rref, rcur, lvl, g["kat_T"], ti, td)
                out[f"err_{seed}_l{lvl}_t{j}_n"], out[f"err_{seed}_l{lvl}_t{j}_digest"] = np.int64(n), np.array(nan_digest(img))
    # non-default selection thresholds and the identity pose, golden pair 12, level 1
    g = load_golden(12)
    im = golden_images(g, orc)
    oref, ocur = pyramids(im, g["K"], GOLDEN_LEVELS)
    w, h, K = oref.level_info(1)
    for k, (T, ti, td) in enumerate(((np.eye(4), 0.0, 0.0), (g["kat_T"], 4.0, 0.02))):
        r = orc.ref_linearize(oref.planes(1), ocur.planes(1), K, T, True, g["kat_prev_precision"], ti, td)
        out[f"thr_{k}_n_selected"], out[f"thr_{k}_n"], out[f"thr_{k}_ll"] = np.int64(r["n_selected"]), np.int64(r["n"]), np.float32(r["ll"])
        for name in ("precision", "A", "b"):
            out[f"thr_{k}_{name}"] = r[name]
    # the odd last point of the SSE loop
    g = load_golden(GOLDEN_SEEDS[0])
    margin, oref, ocur = odd_point_margin(g, golden_images(g, orc))
    n, img = orc.ref_intensity_error_image(orc.RefPyramid(oref), orc.RefPyramid(ocur), 0, np.eye(4))
    out["odd_margin"], out["odd_n"], out["odd_digest"] = np.int64(margin), np.int64(n), np.array(nan_digest(img))
    # DenseTracker::match() end to end
    for i, (im, K, levels, cfg, T0) in enumerate(match_cases()):
        oref, ocur = pyramids(im, K, levels)
        r = orc.ref_match(orc.RefPyramid(oref), orc.RefPyramid(ocur), orc.config(**cfg), T_init=T0)
        for name in ("termination", "num_iterations", "valid_pixels"):
            out[f"match_{i}_{name}"] = np.array([l[name] for l in r["levels"]], dtype=np.int64)
        out[f"match_{i}_T"], out[f"match_{i}_information"] = r["T"], r["information"]
        out[f"match_{i}_log_likelihood"] = np.float64(r["log_likelihood"])
    np.savez_compressed(REFERENCE_GOLDEN, **out)
    print("wrote", REFERENCE_GOLDEN, os.path.getsize(REFERENCE_GOLDEN), "bytes,", len(out), "arrays")


if __name__ == "__main__":
    main()
