"""CPU tests of the point-selection surface: the ctypes mirrors match include/dvo_b200.h (predicate values, signatures), the
adapter headers compile with ValidPointPredicate, and the oracle's predicate- and mask-aware selection (orc_select_ex /
orc_match_ex) agrees with its plain thresholded selection where the two must coincide.  No compute calls on a GPU."""
import os
import re
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HEADER = os.path.join(ROOT, "include", "dvo_b200.h")
SELECTION_CALLS = ("dvo_b200_selection_create", "dvo_b200_selection_create_device_batch", "dvo_b200_selection_retain",
                   "dvo_b200_selection_release", "dvo_b200_selection_pyramid", "dvo_b200_selection_download",
                   "dvo_b200_match_batch_selected", "dvo_b200_match_batch_selected_enqueue")


@pytest.fixture(scope="module")
def engine_mod():
    import __graft_entry__ as ge
    ge.build_cuda()
    from dvo_slam_b200 import engine
    engine.load_library()
    return engine


def _declaration(name):
    src = re.sub(r"/\*.*?\*/", "", open(HEADER).read(), flags=re.S)
    m = re.search(r"\b" + name + r"\s*\(([^)]*)\)", src)
    assert m, name
    return [a.strip() for a in m.group(1).split(",")]


def test_predicate_values_match_header(engine_mod, tmp_path):
    prog = tmp_path / "pred.c"
    prog.write_text('#include <stdio.h>\n#include "dvo_b200.h"\nint main(){printf("%d %d %d",DVO_B200_PREDICATE_GRADIENT_THRESHOLD,'
                    'DVO_B200_PREDICATE_VALID_POINT,DVO_B200_PREDICATE_MASK_ONLY);return 0;}\n')
    exe = tmp_path / "pred"
    subprocess.check_call(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    assert got == [engine_mod.PREDICATE_GRADIENT_THRESHOLD, engine_mod.PREDICATE_VALID_POINT, engine_mod.PREDICATE_MASK_ONLY]
    import selection_oracle as so
    assert (so.PREDICATE_GRADIENT_THRESHOLD, so.PREDICATE_VALID_POINT, so.PREDICATE_MASK_ONLY) == tuple(got)


def test_selection_signatures_match_ctypes(engine_mod):
    L = engine_mod.load_library()
    for name in SELECTION_CALLS:
        assert name in engine_mod.ABI_SYMBOLS
        args = _declaration(name)
        assert len(getattr(L, name).argtypes) == len(args), (name, args)


def test_adapter_headers_compile_with_valid_point_predicate(tmp_path):
    src = tmp_path / "pred.cpp"
    src.write_text('#include "dvo/core/point_selection.h"\n'
                   'int main(){dvo::core::ValidPointPredicate v; dvo::core::ValidPointAndGradientThresholdPredicate g;\n'
                   'const dvo::core::PointSelectionPredicate& p = v; float n = NAN;\n'
                   'return (p.isPointOk(0,0,1.f,0.f,0.f,0.f,0.f) && !v.isPointOk(0,0,n,0.f,0.f,0.f,0.f) &&\n'
                   '        !g.isPointOk(0,0,1.f,0.f,0.f,0.f,0.f)) ? 0 : 1;}\n')
    # both type modes: the adapter's own types, and Eigen / OpenCV types (the container stand-ins of oracle/ref_shim)
    for flags in ([], ["-DDVO_B200_WITH_EIGEN_OPENCV", "-I", os.path.join(ROOT, "oracle", "ref_shim")]):
        exe = tmp_path / "pred"
        r = subprocess.run(["g++", "-std=c++17", "-Wall", "-I", os.path.join(ROOT, "include")] + flags + [str(src), "-o", str(exe)],
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stderr
        assert subprocess.run([str(exe)]).returncode == 0


@pytest.fixture(scope="module")
def so(oracle):
    import selection_oracle
    selection_oracle.lib()
    return selection_oracle


@pytest.fixture(scope="module")
def scene(so, small_scene):
    from dvo_slam_b200 import synth
    pair = synth.make_pair(21, small_scene)
    ref = so.Pyramid(pair["I_ref"].numpy(), pair["Z_ref"].numpy(), small_scene.intrinsics, 3)
    cur = so.Pyramid(pair["I_cur"].numpy(), pair["Z_cur"].numpy(), small_scene.intrinsics, 3)
    rng = np.random.default_rng(5)
    masks = [(rng.random(ref.level_info(l)[1::-1]) < 0.7).astype(np.uint8) for l in range(3)]
    return ref, cur, masks


def test_oracle_all_ones_mask_equals_no_mask(oracle, so, scene):
    ref, _, _ = scene
    for pred in (so.PREDICATE_GRADIENT_THRESHOLD, so.PREDICATE_VALID_POINT, so.PREDICATE_MASK_ONLY):
        for lvl in range(3):
            w, h, _ = ref.level_info(lvl)
            a = so.select_ex(ref, lvl, pred, 4.0, 0.02)
            b = so.select_ex(ref, lvl, pred, 4.0, 0.02, np.ones((h, w), np.uint8))
            assert a[0] == b[0] and np.array_equal(a[1], b[1]), (pred, lvl)
    for lvl in range(3):   # and the plain selection is the gradient predicate without mask
        assert so.select(ref, lvl, 4.0, 0.02)[0] == so.select_ex(ref, lvl, so.PREDICATE_GRADIENT_THRESHOLD, 4.0, 0.02)[0]


def test_oracle_gradient_and_mask_is_the_and_of_both(oracle, so, scene):
    ref, _, masks = scene
    for lvl in range(3):
        S, m = so.select_ex(ref, lvl, so.PREDICATE_GRADIENT_THRESHOLD, 4.0, 0.02, masks[lvl])
        _, g = so.select(ref, lvl, 4.0, 0.02)
        want = g & masks[lvl]
        assert np.array_equal(m, want) and S == int(want.sum()), lvl
        S0, m0 = so.select_ex(ref, lvl, so.PREDICATE_MASK_ONLY, level_mask=masks[lvl])
        assert np.array_equal(m0, masks[lvl]) and S0 == int(masks[lvl].sum())


def test_oracle_mask_only_with_the_gradient_mask_is_the_thresholded_match(oracle, so, scene):
    """The adapter's route for an arbitrary predicate: evaluate it on the host, pass the result as a MASK_ONLY mask."""
    ref, cur, _ = scene
    ti, td = 4.0, 0.02
    cfg = oracle.config(first_level=2, last_level=0, max_iterations_per_level=50, intensity_derivative_threshold=ti,
                        depth_derivative_threshold=td)
    m = oracle.mode("faithful")
    want = so.match(ref, cur, cfg, m)
    masks = [so.select(ref, lvl, ti, td)[1] for lvl in range(3)]
    got = so.match_ex(ref, cur, oracle.config(first_level=2, last_level=0, max_iterations_per_level=50), m,
                          so.PREDICATE_MASK_ONLY, masks=masks)
    assert np.array_equal(got["T"], want["T"]) and np.array_equal(got["information"], want["information"])
    assert got["log_likelihood"] == want["log_likelihood"] and got["levels"] == want["levels"]
    assert [it["n"] for it in got["iterations"]] == [it["n"] for it in want["iterations"]]


def test_extension_library_computes_what_the_oracle_computes(oracle, so, small_scene):
    """the selection oracle includes the oracle's source unchanged: its plain selection and match are the oracle's bits"""
    from dvo_slam_b200 import synth
    pair = synth.make_pair(22, small_scene)
    args = (pair["I_ref"].numpy(), pair["Z_ref"].numpy(), small_scene.intrinsics, 3)
    cargs = (pair["I_cur"].numpy(), pair["Z_cur"].numpy(), small_scene.intrinsics, 3)
    a, b = oracle.Pyramid(*args), so.Pyramid(*args)
    for lvl in range(3):
        sa, sb = oracle.select(a, lvl, 4.0, 0.02), so.select(b, lvl, 4.0, 0.02)
        assert sa[0] == sb[0] and np.array_equal(sa[1], sb[1])
    cfg = oracle.config(first_level=2, last_level=0, max_iterations_per_level=50)
    want = oracle.match(a, oracle.Pyramid(*cargs), cfg, oracle.mode("faithful"))
    got = so.match(b, so.Pyramid(*cargs), cfg, oracle.mode("faithful"))
    assert np.array_equal(got["T"], want["T"]) and got["log_likelihood"] == want["log_likelihood"]


def test_oracle_mask_only_keeps_invalid_points_in_the_list(oracle, so, scene):
    """MASK_ONLY: a point without valid depth counts in S (and in ValidPixels) but yields no constraint"""
    ref, cur, _ = scene
    m = oracle.mode("faithful")
    cfg = oracle.config(first_level=2, last_level=0, max_iterations_per_level=50)
    every = so.match_ex(ref, cur, cfg, m, so.PREDICATE_MASK_ONLY)
    valid = so.match_ex(ref, cur, cfg, m, so.PREDICATE_VALID_POINT)
    for lvl, (le, lv) in enumerate(zip(every["levels"], valid["levels"])):
        w, h, _ = ref.level_info(2 - lvl)
        assert le["valid_pixels"] == w * h and lv["valid_pixels"] < w * h
        assert le["valid_pixels"] == so.select_ex(ref, 2 - lvl, so.PREDICATE_MASK_ONLY)[0]
    assert np.isfinite(every["T"]).all()
