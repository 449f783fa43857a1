import hashlib
import os

import numpy as np

GOLDEN_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
GOLDEN_SEEDS = (11, 12, 13)
GOLDEN_LEVELS = 3
# outputs of the original dvo_core's own SSE object code on the golden pairs (tests/golden/make_reference_golden.py)
REFERENCE_GOLDEN = os.path.join(GOLDEN_DIR, "reference_pin.npz")

# Stated SE(3) tolerance of the path (DESIGN.md "Parity").  Measured with scripts/oracle_spread.py over 96
# seeded 640x480 pairs: the reference's own numerical noise (_mm_rcp_ps, round-toward-zero, fp32 serial
# sums; FAITHFUL vs MIRROR oracle) moves the converged pose by median 1.3e-4 m / 3.0e-5 rad,
# p90 6.2e-4 m / 7.6e-5 rad, max 1.06e-3 m / 3.4e-4 rad -- the same order as the method's accuracy on
# this data (FAITHFUL vs ground truth: median 9.7e-4 m, max 2.3e-3 m).  Tolerance = ~2x the max spread.
POSE_TOL_T = 2e-3   # metres
POSE_TOL_R = 1e-3   # radians


def load_golden(seed):
    g = dict(np.load(os.path.join(GOLDEN_DIR, f"pair_{seed}.npz")))
    g["K"] = tuple(float(v) for v in g["intrinsics"])
    return g


def golden_images(g, orc):
    """float32 intensity/depth exactly as benchmark_slam.cpp:46-93 would hand them to the tracker."""
    out = {}
    for k in ("ref", "cur"):
        out[f"I_{k}"] = g[f"grey_{k}"].astype(np.float32)
        out[f"Z_{k}"] = orc.convert_raw_depth(g[f"depth_{k}"], 1.0 / 5000.0)
    return out


def pose_delta(Ta, Tb):
    """(max |translation|, max |rotation|) components of log(Ta^-1 Tb)."""
    from dvo_slam_b200 import synth
    d = synth.se3_log(np.linalg.inv(Ta) @ Tb)
    return float(np.abs(d[:3]).max()), float(np.abs(d[3:]).max())


def nan_equal(a, b):
    return np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~np.isnan(a)], b[~np.isnan(b)])


def nan_digest(a):
    """sha256 of a float32 array with every NaN made the same NaN and -0 made +0: two arrays have the same digest
    exactly when nan_equal(a, b) holds and their shapes agree."""
    a = np.asarray(a, dtype=np.float32)
    c = np.where(np.isnan(a), np.float32(np.nan), a + np.float32(0.0)).astype(np.float32)
    return hashlib.sha256(str(c.shape).encode() + np.ascontiguousarray(c).tobytes()).hexdigest()
