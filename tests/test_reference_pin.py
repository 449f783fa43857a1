"""Pins the oracle against the REFERENCE'S OWN OBJECT CODE.

tests/golden/reference_pin.npz holds what the original dvo_core's dense_tracking_impl.cpp, core/math_sse.cpp and
core/intrinsic_matrix.cpp, compiled unmodified (oracle/Makefile target `ref`; Eigen / OpenCV / Boost containers from
oracle/ref_shim/), compute on the golden pairs: oracle/ref_driver.cpp strings computeResidualsSse, computeWeightsSse,
computeScaleSse, computeCompleteDataLogLikelihood and OptimizedSelfAdjointMatrix6x6f::rankUpdate together exactly as
DenseTracker::match() does for one Gauss-Newton linearisation (dense_tracking.cpp:212-220, 271-343).  The oracle's FAITHFUL
mode must reproduce every number BIT FOR BIT: selected and valid point counts, which points are valid, all six
residual-record channels, the Student-t weights' effect on the scale (precision), the log-likelihood, A and b.

Per-pixel outputs are stored as digests of the whole images (helpers.nan_digest: equal digests <=> nan_equal) plus the
values at a seeded sample of pixels; tests/golden/make_reference_golden.py regenerates the file from the compiled sources."""
import numpy as np
import pytest

from helpers import GOLDEN_LEVELS, GOLDEN_SEEDS, REFERENCE_GOLDEN, golden_images, load_golden, nan_digest, nan_equal


@pytest.fixture(scope="module")
def ref():
    return dict(np.load(REFERENCE_GOLDEN))


def _cases(oracle):
    for seed in GOLDEN_SEEDS:
        g = load_golden(seed)
        im = golden_images(g, oracle)
        oref = oracle.Pyramid(im["I_ref"], im["Z_ref"], g["K"], GOLDEN_LEVELS)
        ocur = oracle.Pyramid(im["I_cur"], im["Z_cur"], g["K"], GOLDEN_LEVELS)
        for lvl in range(GOLDEN_LEVELS):
            yield seed, g, oref, ocur, lvl


def _linearisation_equal(ref, key, o):
    assert np.array_equal(ref[key + "_precision"], o["precision"])     # computeWeightsSse + computeScaleSse + inverse()
    assert float(ref[key + "_ll"]) == o["ll"]                          # computeCompleteDataLogLikelihood
    assert np.array_equal(ref[key + "_A"].astype(np.float64), o["A"])  # rankUpdate(2x6, 2x2) + toEigen, fp32 serial
    assert np.array_equal(ref[key + "_b"].astype(np.float64), o["b"])


def test_faithful_oracle_equals_reference_object_code_bit_for_bit(oracle, ref):
    fa = oracle.mode("faithful")
    checked = 0
    for seed, g, oref, ocur, lvl in _cases(oracle):
        key = f"lin_{seed}_l{lvl}"
        S, _ = oracle.select(oref, lvl, 0.0, 0.0, fa)
        n_img, img = oracle.residual_image(oref, ocur, lvl, g["kat_T"], fa)
        img = img.reshape(7, -1)
        assert int(ref[key + "_n_selected"]) == S                          # PointSelection::select
        assert int(ref[key + "_n"]) == n_img                               # valid constraints (bounds, NaN and occlusion tests)
        # computeResidualsSse: the same points are valid, every channel of every point is equal
        assert nan_equal(ref[key + "_sample"], img[:, ref[key + "_sample_pixels"]])
        assert ref[key + "_records_digest"] == nan_digest(img), (seed, lvl)
        for uw in (False, True):
            o = oracle.linearize(oref, ocur, lvl, g["kat_T"], fa, uw, g["kat_prev_precision"])
            assert o["n"] == n_img
            _linearisation_equal(ref, f"{key}_w{int(uw)}", o)
            checked += int((~np.isnan(img)).sum())
    assert checked > 500000


def test_nondefault_thresholds_and_identity_pose(oracle, ref):
    """selection thresholds (Config::Intensity/DepthDerivativeThreshold) and a second transform"""
    fa = oracle.mode("faithful")
    g = load_golden(12)
    im = golden_images(g, oracle)
    oref = oracle.Pyramid(im["I_ref"], im["Z_ref"], g["K"], GOLDEN_LEVELS)
    ocur = oracle.Pyramid(im["I_cur"], im["Z_cur"], g["K"], GOLDEN_LEVELS)
    for k, (T, ti, td) in enumerate(((np.eye(4), 0.0, 0.0), (g["kat_T"], 4.0, 0.02))):
        o = oracle.linearize(oref, ocur, 1, T, fa, True, g["kat_prev_precision"], ti, td)
        S, _ = oracle.select(oref, 1, ti, td, fa)
        assert int(ref[f"thr_{k}_n_selected"]) == S and int(ref[f"thr_{k}_n"]) == o["n"]
        _linearisation_equal(ref, f"thr_{k}", o)


def test_reference_built_at_its_own_O3_stays_within_the_stated_spread(oracle, ref):
    """At -O3 (dvo_core/CMakeLists.txt:36-40) GCC 13 schedules floating-point work across the MXCSR switch of
    dense_tracking_impl.cpp:165-167: the reference's own numbers then differ from the program-order build.  The same points
    stay valid; records move by < 5e-3 absolute (measured 2.7e-3), precision / A / b by < 5e-4 relative (measured 1.7e-4) -- the noise floor any comparison
    with 'the reference' has, and two orders of magnitude below the pose tolerance."""
    fa = oracle.mode("faithful")
    for seed, g, oref, ocur, lvl in _cases(oracle):
        key = f"o3_{seed}_l{lvl}"
        o = oracle.linearize(oref, ocur, lvl, g["kat_T"], fa, True, g["kat_prev_precision"])
        n_img, img = oracle.residual_image(oref, ocur, lvl, g["kat_T"], fa)
        img = img.reshape(7, -1)
        assert int(ref[key + "_n"]) == o["n"] and ref[key + "_nan_digest"] == nan_digest(np.isnan(img))
        d, want = ref[key + "_sample"], img[:, ref[f"lin_{seed}_l{lvl}_sample_pixels"]]
        m = ~np.isnan(d)
        assert np.array_equal(m, ~np.isnan(want)) and np.abs(d[m] - want[m]).max() < 5e-3
        assert np.allclose(ref[key + "_precision"], o["precision"], rtol=5e-4)
        assert np.abs(ref[key + "_A"] - o["A"]).max() <= 5e-4 * np.abs(o["A"]).max()
        assert np.abs(ref[key + "_b"] - o["b"]).max() <= 5e-4 * np.abs(o["b"]).max()


def test_whole_alignment_through_reference_object_code_equals_faithful_oracle(oracle, ref):
    """DenseTracker::match() end to end: oracle/ref_driver.cpp runs the coarse-to-fine loop (dense_tracking.cpp:131-376) with
    every per-point pass executed by the reference's own object code; the oracle's FAITHFUL match must take the same control
    flow on every level and return the same Result (the poses agree to the rounding of the 4x4 bookkeeping, Information and
    LogLikelihood exactly)."""
    from dvo_slam_b200 import synth
    fa = oracle.mode("faithful")
    cases = []
    for seed in GOLDEN_SEEDS:
        g = load_golden(seed)
        im = golden_images(g, oracle)
        cases.append((im["I_ref"], im["Z_ref"], im["I_cur"], im["Z_cur"], g["K"], GOLDEN_LEVELS,
                      dict(first_level=2, last_level=0, max_iterations_per_level=50, precision=1e-4), None))
    for seed, extra in ((3, {}), (5, dict(mu=0.05, use_initial_estimate=1))):     # 640x480, 5 levels (BASELINE configs[0])
        p = synth.make_pair(seed)
        a = {k: p[k].numpy() for k in ("I_ref", "Z_ref", "I_cur", "Z_cur")}
        cfg = dict(first_level=4, last_level=0, max_iterations_per_level=50, precision=1e-4)
        cfg.update(extra)
        T0 = synth.se3_exp(p["xi"] * 0.8) if extra else None
        cases.append((a["I_ref"], a["Z_ref"], a["I_cur"], a["Z_cur"], p["intrinsics"], 5, cfg, T0))
    for i, (Ir, Zr, Ic, Zc, K, levels, cfg, T0) in enumerate(cases):
        oref, ocur = oracle.Pyramid(Ir, Zr, K, levels), oracle.Pyramid(Ic, Zc, K, levels)
        o = oracle.match(oref, ocur, oracle.config(**cfg), fa, T_init=T0)
        assert ref[f"match_{i}_termination"].tolist() == [l["termination"] for l in o["levels"]]
        assert ref[f"match_{i}_num_iterations"].tolist() == [l["num_iterations"] for l in o["levels"]]
        assert ref[f"match_{i}_valid_pixels"].tolist() == [l["valid_pixels"] for l in o["levels"]]
        assert np.abs(ref[f"match_{i}_T"] - o["T"]).max() < 1e-12
        assert np.array_equal(ref[f"match_{i}_information"], o["information"])
        assert float(ref[f"match_{i}_log_likelihood"]) == o["log_likelihood"]


def test_intensity_error_image_walk_equals_reference_valid_flag_stream(oracle, ref):
    """DenseTracker::computeIntensityErrorImage (dense_tracking.cpp:378-444): the oracle's raster walk against the same
    walk fed by the reference's OWN computeResidualsAndValidFlagsSse (flags and residuals from the Debug instantiation of
    the SSE loop) -- bit for bit, including the odd last selected point, which the SSE loop never visits and which
    therefore stays 0 although its warp is valid."""
    fa = oracle.mode("faithful")
    for seed, g, oref, ocur, lvl in _cases(oracle):
        for j, (ti, td) in enumerate(((0.0, 0.0), (2.0, 0.02))):
            key = f"err_{seed}_l{lvl}_t{j}"
            n_o, img_o = oracle.intensity_error_image(oref, ocur, lvl, g["kat_T"], fa, ti, td)
            assert n_o == int(ref[key + "_n"]) and n_o > 0
            assert ref[key + "_digest"] == nan_digest(img_o), key
            # semantics, stated independently: |e.i| where the residual stage has a valid residual, 0 elsewhere
            n_img, planes = oracle.residual_image(oref, ocur, lvl, g["kat_T"], fa, ti, td)
            want = np.where(np.isnan(planes[0]), 0.0, np.abs(planes[0])).astype(np.float32)
            assert n_img == n_o and np.array_equal(img_o, want)
    # The odd-point drop made visible: reference = a frame with its bottom/right margin made invalid, current = the same
    # frame unmasked, identity transform -> every selected point maps onto itself and is valid, so the only selected pixel
    # the image may leave at 0 is the odd last one (which EXACT numerics, without the drop, would fill).
    g = load_golden(GOLDEN_SEEDS[0])
    im = golden_images(g, oracle)
    saw_odd = False
    for margin in range(4, 40):
        Z = im["Z_ref"].copy()
        Z[-margin:, :] = np.nan
        Z[:, -margin:] = np.nan
        oref = oracle.Pyramid(im["I_ref"], Z, g["K"], 1)
        ocur = oracle.Pyramid(im["I_ref"], im["Z_ref"], g["K"], 1)
        S, mask = oracle.select(oref, 0, 0.0, 0.0, None)
        last = np.flatnonzero(mask.reshape(-1))[-1]
        _, planes_exact = oracle.residual_image(oref, ocur, 0, np.eye(4), oracle.mode("exact"))
        if S % 2 == 0 or np.isnan(planes_exact[0].reshape(-1)[last]):   # need: odd count, last point valid by itself
            continue
        assert margin == int(ref["odd_margin"])                        # the margin the stored reference image was taken at
        n_o, img_o = oracle.intensity_error_image(oref, ocur, 0, np.eye(4), fa)
        assert ref["odd_digest"] == nan_digest(img_o) and n_o == int(ref["odd_n"]) <= S - 1
        assert img_o.reshape(-1)[last] == 0.0                      # the point itself is fine and still 0 in the reference's image
        saw_odd = True
        break
    assert saw_odd, "no margin gave an odd selection count with a valid last point"
