"""Reference point selections as device objects (dvo_b200_selection_*, dvo_b200_match_batch_selected[_enqueue]).

A selection owns its own copy of the reference tile records with Zsel from its predicate and mask, its own mask words and
{S, last}; the level kernel reads nothing else of it.  So a gradient-threshold selection without mask aligns byte for byte
like the pyramid's own selection with the same thresholds; masks and the other predicates select exactly the oracle's
points and align within the pose tolerance of the oracle with the same mask; and any number of selections of one pyramid
can be aligned at once without touching the pyramid's own selection."""
import ctypes as C
import math
import time

import numpy as np
import pytest

from helpers import POSE_TOL_R, POSE_TOL_T, pose_delta

pytestmark = pytest.mark.gpu

PREDICATES = (0, 1, 2)   # GRADIENT_THRESHOLD, VALID_POINT, MASK_ONLY
LEVELS = 3


def records_bytes(res):
    return bytes(memoryview(res).cast("B"))


def blob_mask(h, w, seed):
    """random blobs: about a third of the image excluded in round patches"""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    m = np.ones((h, w), np.uint8)
    for _ in range(6):
        cy, cx, r = rng.uniform(0, h), rng.uniform(0, w), rng.uniform(0.08, 0.2) * min(h, w)
        m[(yy - cy) ** 2 + (xx - cx) ** 2 < r * r] = 0
    return m


def box_mask(h, w):
    m = np.ones((h, w), np.uint8)
    m[h // 4: h // 2, w // 3: (2 * w) // 3] = 0
    return m


def scene_cfg(width):
    from dvo_slam_b200 import synth
    if width == 640:
        return synth.SceneConfig()
    return synth.SceneConfig(width=160, height=120, intrinsics=tuple(v / 4 for v in synth.FR1_INTRINSICS))


def pyramids(engine, pairs, K, levels):
    refs = engine.pyramid_batch(np.stack([p["I_ref"].numpy() for p in pairs]), np.stack([p["Z_ref"].numpy() for p in pairs]), K, levels)
    curs = engine.pyramid_batch(np.stack([p["I_cur"].numpy() for p in pairs]), np.stack([p["Z_cur"].numpy() for p in pairs]), K, levels)
    return refs, curs


@pytest.fixture(scope="module")
def small(engine, small_scene):
    from dvo_slam_b200 import synth
    pairs = [synth.make_pair(s, small_scene) for s in (31, 32, 33, 34)]
    refs, curs = pyramids(engine, pairs, small_scene.intrinsics, LEVELS)
    return pairs, refs, curs


# ---- 1. equivalence with the pyramid's own selection -----------------------------------------------------------------
@pytest.mark.parametrize("ti,td", [(0.0, 0.0), (4.0, 0.02)])
def test_gradient_selection_equals_pyramid_select(engine, small, ti, td):
    _, refs, _ = small
    for p in refs:
        s = engine.selection(p, 0, ti, td)
        for lvl in range(LEVELS):
            assert s.download(lvl)[0] == p.select(lvl, ti, td)[0]
            assert np.array_equal(s.download(lvl)[1], p.select(lvl, ti, td)[1]), lvl


@pytest.mark.parametrize("ti,td", [(0.0, 0.0), (4.0, 0.02)])
def test_selected_match_is_byte_equal_batch4(engine, small, ti, td):
    from dvo_slam_b200.engine import Config
    _, refs, curs = small
    cfg = Config(first_level=2, last_level=0, max_iterations_per_level=50, intensity_derivative_threshold=ti, depth_derivative_threshold=td)
    want = records_bytes(engine.match_batch(refs, curs, cfg, raw=True))
    sels = [engine.selection(p, 0, ti, td) for p in refs]
    # the selected entry point ignores cfg's thresholds: give it others
    got = records_bytes(engine.match_batch(sels, curs, Config(first_level=2, last_level=0, max_iterations_per_level=50,
                                                               intensity_derivative_threshold=9.0), raw=True))
    assert got == want


@pytest.mark.parametrize("ti,td", [(0.0, 0.0), (4.0, 0.02)])
def test_selected_match_is_byte_equal_batch512(engine, ti, td):
    from dvo_slam_b200 import synth
    from dvo_slam_b200.engine import Config
    sc = synth.SceneConfig()
    pairs = [synth.make_pair(s, sc) for s in range(100, 132)]
    refs, curs = pyramids(engine, pairs, sc.intrinsics, 5)
    refs, curs = refs * 16, curs * 16
    cfg = Config(intensity_derivative_threshold=ti, depth_derivative_threshold=td)
    want = records_bytes(engine.match_batch(refs, curs, cfg, raw=True))
    sels = engine.selections_from_tensors(refs[:32], None, 0, ti, td) * 16
    got = records_bytes(engine.match_batch(sels, curs, Config(), raw=True))
    assert got == want


# ---- 2. masks and predicates against the oracle ----------------------------------------------------------------------
@pytest.mark.parametrize("width", [160, 640])
@pytest.mark.parametrize("kind", ["blob", "box"])
def test_masks_and_predicates_match_the_oracle(engine, oracle, width, kind):
    import selection_oracle as so
    from dvo_slam_b200 import synth
    from dvo_slam_b200.engine import Config, level_masks
    sc = scene_cfg(width)
    levels = 3 if width == 160 else 5
    first, last = (2, 0) if width == 160 else (3, 1)
    pair = synth.make_pair(41, sc)
    m0 = blob_mask(sc.height, sc.width, 3) if kind == "blob" else box_mask(sc.height, sc.width)
    masks = level_masks(m0, levels)
    ref = engine.pyramid(pair["I_ref"].numpy(), pair["Z_ref"].numpy(), sc.intrinsics, levels)
    cur = engine.pyramid(pair["I_cur"].numpy(), pair["Z_cur"].numpy(), sc.intrinsics, levels)
    oref = so.Pyramid(pair["I_ref"].numpy(), pair["Z_ref"].numpy(), sc.intrinsics, levels)
    ocur = so.Pyramid(pair["I_cur"].numpy(), pair["Z_cur"].numpy(), sc.intrinsics, levels)
    ti, td = 4.0, 0.02
    for pred in PREDICATES:
        s = engine.selection(ref, pred, ti, td, masks)
        for lvl in range(levels):
            S, m = s.download(lvl)
            oS, om = so.select_ex(oref, lvl, pred, ti, td, masks[lvl])
            assert S == oS and np.array_equal(m, om), (pred, lvl)
        res = engine.match_batch([s], [cur], Config(first_level=first, last_level=last))[0]
        ores = so.match_ex(oref, ocur, oracle.config(first_level=first, last_level=last), oracle.mode("faithful"), pred, ti, td, masks)
        dt, dr = pose_delta(ores["T"], res.transformation)
        assert dt < POSE_TOL_T and dr < POSE_TOL_R, (pred, dt, dr)
        assert [l["valid_pixels"] for l in res.levels] == [l["valid_pixels"] for l in ores["levels"]]


def moving_box_pair(seed, cfg, shift):
    """make_pair with the box of the current frame moved by `shift` metres along x (independently of the camera)"""
    import torch
    from dvo_slam_b200 import synth
    rng = np.random.default_rng(seed)
    xi = np.concatenate([rng.uniform(-cfg.max_translation, cfg.max_translation, 3), rng.uniform(-cfg.max_rotation, cfg.max_rotation, 3)])
    T_true = synth.se3_exp(xi)
    lam = np.exp(rng.uniform(math.log(0.04), math.log(0.60), cfg.n_sinusoids))
    dirs = rng.standard_normal((cfg.n_sinusoids, 3))
    dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    freq = dirs / lam[:, None]
    phase = rng.uniform(0, 2 * math.pi, cfg.n_sinusoids)
    amp = lam / lam.sum() * 2.2
    tex = tuple(torch.tensor(v, dtype=torch.float64) for v in (freq, phase, amp))
    box = (1.2 + rng.uniform(-0.1, 0.1), rng.uniform(-0.2, 0.2), rng.uniform(-0.15, 0.15), 0.28, 0.22)
    I_ref, Z_ref = synth._render(cfg, np.eye(4), tex, box, rng, "cpu")
    moved = (box[0], box[1] + shift) + box[2:]
    I_cur, Z_cur = synth._render(cfg, T_true, tex, moved, rng, "cpu")
    return {"I_ref": I_ref, "Z_ref": Z_ref, "I_cur": I_cur, "Z_cur": Z_cur, "T_true": T_true, "box": box}


def test_masking_a_moving_box_does_not_hurt(engine):
    from dvo_slam_b200.engine import Config, level_masks
    sc = scene_cfg(640)
    pair = moving_box_pair(43, sc, 0.06)
    ref = engine.pyramid(pair["I_ref"].numpy(), pair["Z_ref"].numpy(), sc.intrinsics, 5)
    cur = engine.pyramid(pair["I_cur"].numpy(), pair["Z_cur"].numpy(), sc.intrinsics, 5)
    # the box in the reference image: the pixels whose depth is the box plane (closer than the background)
    zb = pair["box"][0]
    Z = pair["Z_ref"].numpy()
    m0 = ~(np.abs(Z - zb) < 0.05)
    m0 = np.where(np.isnan(Z), True, m0).astype(np.uint8)
    m0 = np.minimum(m0, np.roll(m0, 4, 0)) & np.roll(m0, -4, 0) & np.roll(m0, 4, 1) & np.roll(m0, -4, 1)   # a margin around it
    assert m0.mean() < 0.97
    plain = engine.selection(ref, 0)
    masked = engine.selection(ref, 0, masks=level_masks(m0, 5))
    a, b = engine.match_batch([plain, masked], [cur, cur], Config())
    ea = pose_delta(pair["T_true"], a.transformation)
    eb = pose_delta(pair["T_true"], b.transformation)
    print(f"moving box: error vs T_true unmasked |dt|={ea[0]:.3e} |dr|={ea[1]:.3e}, masked |dt|={eb[0]:.3e} |dr|={eb[1]:.3e}")
    assert eb[0] <= ea[0] and eb[1] <= ea[1]


# ---- 3. many selections of one pyramid -------------------------------------------------------------------------------
def test_one_pyramid_under_several_selections(engine, small):
    from dvo_slam_b200.engine import Config, level_masks
    pairs, refs, curs = small
    ref, cur = refs[0], curs[0]
    before = [ref.select(l, 0.0, 0.0) for l in range(LEVELS)]
    sels = [engine.selection(ref, 0), engine.selection(ref, 0, 4.0, 0.02), engine.selection(ref, 1),
            engine.selection(ref, 2, masks=level_masks(blob_mask(120, 160, 7), LEVELS))]
    cfg = Config(first_level=2, last_level=0, max_iterations_per_level=50)
    together = engine.match_batch(sels, [cur] * len(sels), cfg, raw=True)
    for i, s in enumerate(sels):
        alone = engine.match_batch([s], [cur], cfg, raw=True)
        assert records_bytes(alone) == bytes(memoryview(together).cast("B"))[i * C.sizeof(alone[0]):(i + 1) * C.sizeof(alone[0])]
    after = [ref.select(l, 0.0, 0.0) for l in range(LEVELS)]
    assert all(a[0] == b[0] and np.array_equal(a[1], b[1]) for a, b in zip(before, after))


def test_two_contexts_enqueue_against_one_pyramid(engine, small):
    import torch
    from dvo_slam_b200.engine import Config, Engine
    _, refs, curs = small
    cfg = Config(first_level=2, last_level=0, max_iterations_per_level=50)
    other = Engine(device=0)
    ra = rb = None
    try:
        sa = engine.selection(refs[1], 0, 4.0, 0.02)
        sb = other.selection(refs[1], 1)
        want_a = records_bytes(engine.match_batch([sa], [curs[1]], cfg, raw=True))
        want_b = records_bytes(other.match_batch([sb], [curs[1]], cfg, raw=True))
        ra = engine.match_batch_enqueue([sa] * 3, [curs[1]] * 3, cfg)
        rb = other.match_batch_enqueue([sb] * 3, [curs[1]] * 3, cfg)
        engine.synchronize(); other.synchronize()
        torch.cuda.synchronize()
        # the records are in use on `other`'s stream: copy them out and free them before that stream goes away
        ha, hb = ra.cpu().numpy(), rb.cpu().numpy()
        del sb
    finally:
        ra = rb = None
        torch.cuda.synchronize()
        other.close()
    for i in range(3):
        assert ha[i].tobytes() == want_a and hb[i].tobytes() == want_b


# ---- 4. device masks -------------------------------------------------------------------------------------------------
def test_device_masks_equal_host_level_masks(engine, small):
    import torch
    from dvo_slam_b200.engine import level_masks
    _, refs, _ = small
    n = len(refs)
    host = np.stack([blob_mask(120, 160, 10 + i) for i in range(n)])
    dev = torch.device("cuda", 0)
    dense = torch.from_numpy(host).to(dev)
    wide = torch.zeros((n, 120, 200), dtype=torch.uint8, device=dev)
    wide[:, :, 17:177] = dense
    every_other = torch.zeros((2 * n, 120, 160), dtype=torch.bool, device=dev)
    every_other[::2] = dense.bool()
    for t in (dense, wide[:, :, 17:177], every_other[::2]):
        for pred in PREDICATES:
            got = engine.selections_from_tensors(refs, t, pred, 4.0, 0.02)
            for i, s in enumerate(got):
                want = engine.selection(refs[i], pred, 4.0, 0.02, level_masks(host[i], LEVELS))
                for lvl in range(LEVELS):
                    a, b = s.download(lvl), want.download(lvl)
                    assert a[0] == b[0] and np.array_equal(a[1], b[1]), (pred, i, lvl)


def test_bad_device_masks_are_refused(engine, small):
    import torch
    _, refs, _ = small
    L = engine.lib
    n = len(refs)
    ph = (C.c_void_p * n)(*[p.handle for p in refs])
    out = (C.c_void_p * n)()
    host = np.ones((n, 120, 160), np.uint8)
    dense = torch.ones((n, 120, 160), dtype=torch.uint8, device="cuda:0")
    assert L.dvo_b200_selection_create_device_batch(engine.ctx, n, ph, 0, 0.0, 0.0, host.ctypes.data, 160, 120 * 160, out) == -1
    assert L.dvo_b200_selection_create_device_batch(engine.ctx, n, ph, 0, 0.0, 0.0, dense.data_ptr(), 159, 120 * 160, out) == -1
    assert L.dvo_b200_selection_create_device_batch(engine.ctx, n, ph, 0, 0.0, 0.0, dense.data_ptr(), 160, 119 * 160, out) == -1
    assert L.dvo_b200_selection_create_device_batch(engine.ctx, n, ph, 7, 0.0, 0.0, dense.data_ptr(), 160, 120 * 160, out) == -1
    assert not any(out[i] for i in range(n))
    if torch.cuda.device_count() > 1:
        other = torch.ones((n, 120, 160), dtype=torch.uint8, device="cuda:1")
        assert L.dvo_b200_selection_create_device_batch(engine.ctx, n, ph, 0, 0.0, 0.0, other.data_ptr(), 160, 120 * 160, out) == -1


# ---- 5. lifetime -----------------------------------------------------------------------------------------------------
def test_selection_outlives_its_pyramid_and_context(small_scene):
    from dvo_slam_b200 import synth
    from dvo_slam_b200.engine import Engine, load_library
    pair = synth.make_pair(51, small_scene)
    eng = Engine(device=0)
    p = eng.pyramid(pair["I_ref"].numpy(), pair["Z_ref"].numpy(), small_scene.intrinsics, LEVELS)
    want = p.select(1, 0.0, 0.0)
    s = eng.selection(p, 0)
    handle = s.handle
    s.handle = None          # keep the raw handle past the Python objects
    p.release()
    eng.close()
    L = load_library()
    cnt = C.c_int64()
    mask = np.zeros((60, 80), np.uint8)
    assert L.dvo_b200_selection_download(None, handle, 1, C.byref(cnt), mask.ctypes.data_as(C.POINTER(C.c_uint8))) == 0
    assert cnt.value == want[0] and np.array_equal(mask, want[1])
    assert L.dvo_b200_selection_pyramid(handle)
    assert L.dvo_b200_selection_release(handle) == 0


# ---- 6. enqueue ------------------------------------------------------------------------------------------------------
def test_selected_enqueue_returns_before_the_gpu_and_matches(engine, small):
    import torch
    from dvo_slam_b200.engine import Config
    _, refs, curs = small
    cfg = Config(first_level=2, last_level=0, max_iterations_per_level=50)
    sels = [engine.selection(p, 2, masks=None) for p in refs]
    want = records_bytes(engine.match_batch(sels, curs, cfg, raw=True))
    engine.match_batch_enqueue(sels, curs, cfg)   # warm
    torch.cuda.synchronize()
    engine.synchronize()
    torch.cuda._sleep(int(2.5e8))          # >= 0.1 s at the B200's clocks
    sleeping = torch.cuda.Event()
    sleeping.record()
    t0 = time.perf_counter()
    rec = engine.match_batch_enqueue(sels, curs, cfg)
    returned = time.perf_counter() - t0
    still_sleeping = not sleeping.query()
    assert still_sleeping, f"the call waited for the GPU ({returned * 1e3:.1f} ms)"
    engine.synchronize()
    torch.cuda.synchronize()
    assert rec.cpu().numpy().tobytes() == want


# ---- 7. the C++ adapter: match(PointSelection&, ...) honours the selection's predicate ------------------------------
def test_adapter_honours_point_selection_predicates(engine, small_scene, tmp_path):
    import json
    import os
    import subprocess
    from dvo_slam_b200 import synth
    from dvo_slam_b200.engine import Config
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "dvo_slam_b200", "host", "selection_selftest")
    pair = synth.make_pair(61, small_scene)
    path = tmp_path / "pair.bin"
    with open(path, "wb") as f:
        for k in ("I_ref", "Z_ref", "I_cur", "Z_cur"):
            f.write(np.ascontiguousarray(pair[k].numpy(), dtype=np.float32).tobytes())
    K = small_scene.intrinsics
    r = subprocess.run([exe, str(path), "160", "120"] + [repr(float(v)) for v in K] + ["2", "0"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr
    got = {k: np.array(v).reshape(4, 4) for k, v in json.loads(r.stdout).items()}

    cfg = Config(first_level=2, last_level=0, max_iterations_per_level=50)
    ref = engine.pyramid(pair["I_ref"].numpy(), pair["Z_ref"].numpy(), K, LEVELS)
    cur = engine.pyramid(pair["I_cur"].numpy(), pair["Z_cur"].numpy(), K, LEVELS)
    # own predicate {0, 0} under a tracker configured with (5, 0.05): the (0, 0) alignment
    assert np.array_equal(got["own"], engine.match(ref, cur, cfg).transformation)
    assert not np.array_equal(got["own"], engine.match(ref, cur, Config(first_level=2, last_level=0, max_iterations_per_level=50,
                                                                         intensity_derivative_threshold=5.0,
                                                                         depth_derivative_threshold=0.05)).transformation)
    # a predicate of its own: the MASK_ONLY selection with the predicate's mask (true depth of the level, device gradients)
    Z0 = pair["Z_ref"].numpy()
    masks = []
    for lvl in range(LEVELS):
        planes = ref.download(lvl)
        h, w = planes.shape[1:]
        z = Z0[::1 << lvl, ::1 << lvl][:h, :w]
        with np.errstate(invalid="ignore"):
            masks.append((~np.isnan(z) & ~np.isnan(planes[4]) & ~np.isnan(planes[5]) & (z < 2.0)).astype(np.uint8))
    custom = engine.selection(ref, 2, masks=masks)
    assert np.array_equal(got["custom"], engine.match_batch([custom], [cur], cfg)[0].transformation)
    # match(pyramid, pyramid) is unchanged
    assert np.array_equal(got["plain"], engine.match(ref, cur, cfg).transformation)
