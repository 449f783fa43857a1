"""Frames already in GPU memory (dvo_b200_pyramid_create_device_batch, dvo_b200_match_batch_enqueue).

The rule of the device-input path: a device-input call gives the same bits as the host-input call on the same pixels.
Pyramids built in place from device tensors -- dense, with padded rows, every other image of a batch, an odd crop -- equal
those of the host entry point of the same format plane for plane (NaN-aware byte equality) with the same selection; enqueued
alignments with device initial estimates return the records of dvo_b200_match_batch byte for byte, while the host does not
wait for the GPU and only the pair descriptors cross the bus."""
import ctypes as C
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SCALE = 1.0 / 5000.0
FORMATS = ("f32", "grey8", "bgr8")
FULL_LEVELS, SMALL_LEVELS = 5, 3


def same_bits(a, b):
    """byte equality with every NaN made the same NaN"""
    a = np.where(np.isnan(a), np.float32(np.nan), a).astype(np.float32)
    b = np.where(np.isnan(b), np.float32(np.nan), b).astype(np.float32)
    return a.shape == b.shape and np.array_equal(a.view(np.uint32), b.view(np.uint32))


def assert_same_pyramids(got, want, levels):
    assert len(got) == len(want)
    for i, (a, b) in enumerate(zip(got, want)):
        for lvl in range(levels):
            assert a.level_info(lvl) == b.level_info(lvl), (i, lvl)
            assert same_bits(a.download(lvl), b.download(lvl)), (i, lvl)
            sa, ma = a.select(lvl)
            sb, mb = b.select(lvl)
            assert sa == sb and np.array_equal(ma, mb), (i, lvl)


def make_frames(scene, seeds):
    """references then currents of the seeded pairs, on cuda:0: float32 intensity / depth, 8-bit grey, 16-bit raw depth
    (int16 holding the bits; the synthetic depth is quantised to 1/5000 m, so both representations hold the same pixels),
    an interleaved BGR image, and the true motions"""
    import torch
    from dvo_slam_b200 import synth
    dev = torch.device("cuda", 0)
    pairs = [synth.make_pair(s, scene, device=dev) for s in seeds]
    I = torch.stack([p["I_ref"] for p in pairs] + [p["I_cur"] for p in pairs]).float().contiguous()
    Z = torch.stack([p["Z_ref"] for p in pairs] + [p["Z_cur"] for p in pairs]).float()
    raw = torch.where(torch.isnan(Z), torch.zeros_like(Z), torch.round(Z * 5000.0)).to(torch.int32)
    Z = torch.where(raw == 0, torch.full_like(Z, float("nan")), raw.to(torch.float32) * torch.tensor(SCALE, dtype=torch.float32, device=dev))
    G = I.to(torch.uint8)
    assert torch.equal(G.float(), I)
    D = raw.to(torch.int16)
    g = G.to(torch.int32)
    BGR = torch.stack([g, (g * 7 + 13) % 256, 255 - g], -1).to(torch.uint8).contiguous()
    torch.cuda.synchronize()
    return {"I": I, "Z": Z.contiguous(), "G": G, "D": D, "BGR": BGR, "T_true": [p["T_true"] for p in pairs], "K": scene.intrinsics}


def device_inputs(fr, fmt):
    if fmt == "f32":
        return fr["I"], fr["Z"], None
    return (fr["G"] if fmt == "grey8" else fr["BGR"]), fr["D"], SCALE


def host_pyramids(engine, fmt, colour, depth, K, levels):
    """the host entry point of the format, from dense host copies of the given (device) images"""
    c = np.ascontiguousarray(colour.cpu().numpy())
    d = np.ascontiguousarray(depth.cpu().numpy())
    n, h, w = d.shape
    if fmt == "f32":
        return engine.pyramid_batch(c, d, K, levels)
    d = d.view(np.uint16)
    if fmt == "grey8":
        out = engine.pyramid_raw_batch((c.ctypes.data, d.ctypes.data, n, h, w), SCALE, K, levels)
    else:
        out = engine.pyramid_bgr_batch((c.ctypes.data, d.ctypes.data, n, h, w), SCALE, K, levels)
    engine.synchronize()
    return out


@pytest.fixture(scope="module")
def scenes(small_scene):
    from dvo_slam_b200 import synth
    return {"small": (make_frames(small_scene, [3]), SMALL_LEVELS), "full": (make_frames(synth.SceneConfig(), [5]), FULL_LEVELS)}


@pytest.mark.parametrize("scene", ["small", "full"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_dense_device_frames_equal_host_input(engine, scenes, scene, fmt):
    fr, levels = scenes[scene]
    colour, depth, scale = device_inputs(fr, fmt)
    h2d = engine.h2d_bytes()
    got = engine.pyramid_from_tensors(colour, depth, fr["K"], levels, depth_scale=scale)
    assert engine.h2d_bytes() == h2d            # no frame crosses the bus
    assert_same_pyramids(got, host_pyramids(engine, fmt, colour, depth, fr["K"], levels), levels)


def _padded(x, pad, fill):
    import torch
    shape = list(x.shape)
    shape[2] += pad
    big = torch.full(shape, fill, dtype=x.dtype, device=x.device)
    big[:, :, : x.shape[2]] = x
    return big[:, :, : x.shape[2]]


def _every_other(x, fill):
    import torch
    big = torch.full((2 * x.shape[0],) + tuple(x.shape[1:]), fill, dtype=x.dtype, device=x.device)
    big[::2] = x
    return big[::2]


@pytest.mark.parametrize("layout", ["padded_unaligned", "padded_aligned", "every_other", "odd_crop"])
@pytest.mark.parametrize("fmt", FORMATS)
def test_strided_device_frames_equal_host_input(engine, scenes, fmt, layout):
    fr, levels = scenes["small"]
    colour, depth, scale = device_inputs(fr, fmt)
    if layout == "padded_unaligned":      # pitch element-aligned, but not a multiple of two pixels: scalar 2x2 loads
        colour, depth = _padded(colour, 1, 77), _padded(depth, 1, 77)
    elif layout == "padded_aligned":      # pitch a multiple of two pixels: vector 2x2 loads
        colour, depth = _padded(colour, 6, 77), _padded(depth, 2, 77)
    elif layout == "every_other":
        colour, depth = _every_other(colour, 77), _every_other(depth, 77)
    else:                                 # 157 x 119 crop of the 160 x 120 frames, rows 160 pixels apart
        colour, depth = colour[:, :119, :157], depth[:, :119, :157]
    assert not (colour.is_contiguous() and depth.is_contiguous())
    got = engine.pyramid_from_tensors(colour, depth, fr["K"], levels, depth_scale=scale)
    assert_same_pyramids(got, host_pyramids(engine, fmt, colour, depth, fr["K"], levels), levels)


# ---- alignment ----------------------------------------------------------------------------------------------------------
def _cfg(use_init):
    from dvo_slam_b200.engine import Config
    return Config(first_level=4, last_level=0, max_iterations_per_level=50, precision=1e-4, use_initial_estimate=use_init)


def _t_init(fr):
    """a guess near the true Result.Transformation (inv(T_true)) of every pair"""
    from dvo_slam_b200 import synth
    rng = np.random.default_rng(17)
    return np.stack([np.linalg.inv(T) @ synth.se3_exp(0.003 * rng.standard_normal(6)) for T in fr["T_true"]]).astype(np.float64)


@pytest.fixture(scope="module")
def batches():
    from dvo_slam_b200 import synth
    return {4: make_frames(synth.SceneConfig(), range(4)), 512: make_frames(synth.SceneConfig(), range(512))}


def _host_records(engine, fr, cfg, T):
    B = len(fr["T_true"])
    pyr = host_pyramids(engine, "grey8", fr["G"], fr["D"], fr["K"], FULL_LEVELS)
    h2d = engine.h2d_bytes()
    res = engine.match_batch(pyr[:B], pyr[B:], cfg, T_init=T, raw=True)
    return bytes(memoryview(res)), engine.h2d_bytes() - h2d


@pytest.mark.parametrize("use_init", [0, 1])
@pytest.mark.parametrize("B", [4, 512])
def test_enqueue_equals_match_batch(engine, batches, B, use_init):
    import torch
    from dvo_slam_b200.engine import CResult, result_transformations
    fr = batches[B]
    cfg = _cfg(use_init)
    T = _t_init(fr)
    want, h2d_host = _host_records(engine, fr, cfg, T)
    T_dev = torch.from_numpy(T).cuda()
    pyr = engine.pyramid_from_tensors(fr["G"], fr["D"], fr["K"], FULL_LEVELS, depth_scale=SCALE)
    h2d, d2h = engine.h2d_bytes(), engine.d2h_bytes()
    rec = engine.match_batch_enqueue(pyr[:B], pyr[B:], cfg, T_init=T_dev)
    # only the pair descriptors went up (the host call also staged the n initial estimates), nothing came down
    assert engine.h2d_bytes() - h2d == h2d_host - (128 * B if use_init else 0)
    assert engine.d2h_bytes() == d2h
    engine.synchronize()
    torch.cuda.synchronize()
    assert rec.shape == (B, C.sizeof(CResult))
    assert rec.cpu().numpy().tobytes() == want
    assert np.array_equal(result_transformations(rec).cpu().numpy(), np.frombuffer(want, np.float64).reshape(B, -1)[:, :16].reshape(B, 4, 4))


def test_host_does_not_wait(batches):
    """Context on a torch stream, both calls warm at these shapes: with 0.1 s of sleep queued ahead of them on that stream,
    they return while the sleep is still running, and the results equal those of dvo_b200_match_batch."""
    import torch
    from dvo_slam_b200.engine import Engine
    fr = batches[4]
    B = len(fr["T_true"])
    cfg = _cfg(1)
    T = _t_init(fr)
    T_dev = torch.from_numpy(T).cuda()
    stream = torch.cuda.Stream()
    eng = Engine(device=0, stream=stream.cuda_stream)
    try:
        want, _ = _host_records(eng, fr, cfg, T)
        with torch.cuda.stream(stream):
            for _ in range(2):    # warm: slab pool, workspace, descriptor ring, the caching allocator's pool of this stream
                pyr = eng.pyramid_from_tensors(fr["G"], fr["D"], fr["K"], FULL_LEVELS, depth_scale=SCALE)
                rec = eng.match_batch_enqueue(pyr[:B], pyr[B:], cfg, T_init=T_dev)
                eng.synchronize()
                for p in pyr:
                    p.release()
                del rec
        torch.cuda.synchronize()
        with torch.cuda.stream(stream):
            torch.cuda._sleep(int(2.5e8))          # >= 0.1 s at the B200's clocks
            sleeping = torch.cuda.Event()
            sleeping.record(stream)
            t0 = time.perf_counter()
            pyr = eng.pyramid_from_tensors(fr["G"], fr["D"], fr["K"], FULL_LEVELS, depth_scale=SCALE)
            rec = eng.match_batch_enqueue(pyr[:B], pyr[B:], cfg, T_init=T_dev)
            returned = time.perf_counter() - t0
            still_sleeping = not sleeping.query()
        assert still_sleeping, f"the calls waited for the GPU ({returned * 1e3:.1f} ms)"
        eng.synchronize()
        torch.cuda.synchronize()
        assert rec.cpu().numpy().tobytes() == want
    finally:
        eng.close()


# ---- refusals -----------------------------------------------------------------------------------------------------------
def _create(engine, frames, n, K, levels=SMALL_LEVELS):
    out = (C.c_void_p * n)()
    rc = engine.lib.dvo_b200_pyramid_create_device_batch(engine.ctx, n, C.byref(frames), *[float(v) for v in K], levels, out)
    return rc, [out[i] for i in range(n)]


def test_refusals(engine, scenes):
    import torch
    from dvo_slam_b200.engine import device_frames
    fr, _ = scenes["small"]
    n, h, w = fr["Z"].shape
    K = fr["K"]
    host = fr["I"].cpu().numpy()
    pinned = fr["I"].cpu().pin_memory()

    def refused(**changes):
        f = device_frames(fr["I"], fr["Z"])
        for k, v in changes.items():
            setattr(f, k, v)
        rc, out = _create(engine, f, n, K)
        assert rc == -1 and all(p is None for p in out), changes          # DVO_B200_ERR_INVALID_ARGUMENT, no pyramid
        return engine.lib.dvo_b200_last_error(engine.ctx).decode()

    assert "host memory" in refused(colour=host.ctypes.data)
    assert "host memory" in refused(depth=pinned.data_ptr())
    assert "colour_row_bytes" in refused(colour_row_bytes=4 * w - 4)
    assert "colour_image_bytes" in refused(colour_image_bytes=4 * w * (h - 1))
    assert "depth_row_bytes" in refused(depth_row_bytes=4 * w + 2)                    # not a multiple of 4
    assert "format" in refused(format=7)
    raw = device_frames(fr["G"], fr["D"], SCALE)
    raw.depth_row_bytes = 2 * w + 1                                                   # 16-bit depth: odd pitch
    rc, out = _create(engine, raw, n, K)
    assert rc == -1 and all(p is None for p in out)
    with pytest.raises(ValueError):
        engine.pyramid_from_tensors(fr["I"].cpu(), fr["Z"].cpu(), K, SMALL_LEVELS)
    # enqueue: results must be device memory too
    pyr = engine.pyramid_from_tensors(fr["I"], fr["Z"], K, SMALL_LEVELS)
    from dvo_slam_b200.engine import CResult, Config
    res = np.zeros(C.sizeof(CResult), np.uint8)
    rh, ch = (C.c_void_p * 1)(pyr[0].handle), (C.c_void_p * 1)(pyr[1].handle)
    cfg = Config(first_level=2, last_level=0)
    assert engine.lib.dvo_b200_match_batch_enqueue(engine.ctx, C.byref(cfg), 1, rh, ch, None, res.ctypes.data) == -1
    if torch.cuda.device_count() < 2:
        pytest.skip("the pointer-on-another-device refusal needs two GPUs")
    other = fr["I"].to("cuda:1")
    torch.cuda.synchronize(1)
    assert "device 1" in refused(colour=other.data_ptr())
