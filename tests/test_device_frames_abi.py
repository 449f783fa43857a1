"""CPU tests of the device-frame surface: dvo_b200_device_frames has the layout the ctypes mirror assumes, and torch tensors
are described by their byte strides without a copy.  No compute calls (no GPU here)."""
import ctypes as C
import os
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
FIELDS = ("format", "width", "height", "reserved", "colour", "colour_row_bytes", "colour_image_bytes", "depth", "depth_row_bytes",
          "depth_image_bytes", "depth_scale")


@pytest.fixture(scope="module")
def engine_mod():
    import __graft_entry__ as ge
    ge.build_cuda()
    from dvo_slam_b200 import engine
    engine.load_library()
    return engine


def test_device_frames_layout_matches_header(engine_mod, tmp_path):
    prog = tmp_path / "frames_layout.c"
    offs = ",".join(f"offsetof(dvo_b200_device_frames,{f})" for f in FIELDS)
    prog.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "dvo_b200.h"\nint main(){size_t v[]={sizeof(dvo_b200_device_frames),'
                    f'{offs},DVO_B200_FRAME_F32,DVO_B200_FRAME_GREY8_RAW16,DVO_B200_FRAME_BGR8_RAW16}};'
                    'for(size_t i=0;i<sizeof(v)/sizeof(v[0]);++i)printf("%zu ",v[i]);return 0;}\n')
    exe = tmp_path / "frames_layout"
    subprocess.check_call(["gcc", "-I", os.path.join(ROOT, "include"), str(prog), "-o", str(exe)])
    got = [int(v) for v in subprocess.check_output([str(exe)]).split()]
    D = engine_mod.DeviceFrames
    want = [C.sizeof(D)] + [getattr(D, f).offset for f in FIELDS] + [engine_mod.FRAME_F32, engine_mod.FRAME_GREY8_RAW16,
                                                                     engine_mod.FRAME_BGR8_RAW16]
    assert got == want


def test_byte_strides_of_sliced_tensors(engine_mod):
    import torch
    n, h, w = 4, 10, 12
    wide = torch.zeros((2 * n, h, w + 3), dtype=torch.float32)
    depth = torch.zeros((n, h, w), dtype=torch.float32)
    f = engine_mod.device_frames(wide[::2, :, :w], depth)
    assert (f.format, f.width, f.height) == (engine_mod.FRAME_F32, w, h)
    assert f.colour == wide.data_ptr() and f.colour_row_bytes == 4 * (w + 3) and f.colour_image_bytes == 2 * 4 * h * (w + 3)
    assert f.depth == depth.data_ptr() and f.depth_row_bytes == 4 * w and f.depth_image_bytes == 4 * h * w

    grey = torch.zeros((n, h, w + 1), dtype=torch.uint8)[:, :, 1:]
    raw = torch.zeros((n, h, w), dtype=torch.int16)
    f = engine_mod.device_frames(grey, raw, 1.0 / 5000.0)
    assert f.format == engine_mod.FRAME_GREY8_RAW16 and f.colour == grey.data_ptr() and f.colour_row_bytes == w + 1
    assert f.depth_row_bytes == 2 * w and f.depth_image_bytes == 2 * h * w and f.depth_scale == pytest.approx(1.0 / 5000.0)

    bgr = torch.zeros((n, h, w + 2, 3), dtype=torch.uint8)[:, :, :w]
    f = engine_mod.device_frames(bgr, raw, 1.0 / 5000.0)
    assert f.format == engine_mod.FRAME_BGR8_RAW16 and f.colour_row_bytes == 3 * (w + 2) and f.colour_image_bytes == 3 * (w + 2) * h

    one = engine_mod.device_frames(wide[:1, :, :w], depth[:1])       # a single image: image stride = height x row stride
    assert one.colour_image_bytes == h * one.colour_row_bytes


def test_device_frames_refuses_what_it_cannot_describe(engine_mod):
    import torch
    z = torch.zeros((2, 8, 8), dtype=torch.float32)
    with pytest.raises(ValueError):
        engine_mod.device_frames(torch.zeros((2, 8, 8), dtype=torch.float64), z)                  # unknown format
    with pytest.raises(ValueError):
        engine_mod.device_frames(torch.zeros((2, 8, 8), dtype=torch.uint8), z, 1e-3)              # raw colour, float depth
    with pytest.raises(ValueError):
        engine_mod.device_frames(torch.zeros((2, 8, 8), dtype=torch.uint8), z.to(torch.int16))    # no depth scale
    with pytest.raises(ValueError):
        engine_mod.device_frames(torch.zeros((2, 8, 8)).transpose(1, 2), z)                       # no unit pixel stride
    with pytest.raises(ValueError):
        engine_mod.device_frames(torch.zeros((2, 8, 9)), z)                                       # shapes differ


def test_result_transformations_is_a_view(engine_mod):
    import torch
    n, rb = 3, C.sizeof(engine_mod.CResult)
    recs = (engine_mod.CResult * n)()
    for i in range(n):
        for k in range(16):
            recs[i].transformation[k] = 100 * i + k
        recs[i].log_likelihood = -1.0
    t = torch.frombuffer(bytearray(memoryview(recs)), dtype=torch.uint8).view(n, rb)
    T = engine_mod.result_transformations(t)
    assert T.shape == (n, 4, 4) and T.dtype == torch.float64 and T.data_ptr() == t.data_ptr()
    for i in range(n):
        assert torch.equal(T[i].reshape(16), torch.arange(16, dtype=torch.float64) + 100 * i)
