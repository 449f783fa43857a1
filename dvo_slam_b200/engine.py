"""ctypes binding of the C ABI in include/dvo_b200.h (dvo_slam_b200/libdvo_b200.so).

This is the harness-side view used by tests/ and bench.py; the product is the CUDA library and the
C++ adapter (include/dvo_b200/).  There is no CPU fallback: if the shared library is missing or no
CUDA device is present, construction raises.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("DVO_B200_LIB", os.path.join(_HERE, "libdvo_b200.so"))   # env override: developer A/B builds
MAX_LEVELS = 8

TERMINATION_NAMES = ["IterationsExceeded", "IncrementTooSmall", "LogLikelihoodDecreased", "TooFewConstraints"]

# every symbol include/dvo_b200.h declares (checked by tests/test_abi.py)
ABI_SYMBOLS = [
    "dvo_b200_abi_version", "dvo_b200_create", "dvo_b200_destroy", "dvo_b200_stream", "dvo_b200_synchronize",
    "dvo_b200_last_error", "dvo_b200_config_default", "dvo_b200_kernel_launches", "dvo_b200_h2d_bytes",
    "dvo_b200_d2h_bytes", "dvo_b200_pyramid_create", "dvo_b200_pyramid_create_batch", "dvo_b200_pyramid_create_raw",
    "dvo_b200_pyramid_create_raw_batch", "dvo_b200_pyramid_create_bgr_batch",
    "dvo_b200_pyramid_retain", "dvo_b200_pyramid_release", "dvo_b200_pyramid_num_levels", "dvo_b200_pyramid_level_info",
    "dvo_b200_pyramid_download", "dvo_b200_pyramid_select", "dvo_b200_match", "dvo_b200_match_batch",
    "dvo_b200_match_batch_device", "dvo_b200_residual_image", "dvo_b200_intensity_error_image", "dvo_b200_linearize", "dvo_b200_profile_enable",
    "dvo_b200_profile_read", "dvo_b200_pyramid_device", "dvo_b200_sharded_create", "dvo_b200_sharded_destroy",
    "dvo_b200_sharded_num_shards", "dvo_b200_sharded_ctx", "dvo_b200_sharded_last_error", "dvo_b200_shard_range",
    "dvo_b200_sharded_pyramid_create_batch", "dvo_b200_sharded_pyramid_create_raw_batch", "dvo_b200_match_batch_sharded",
    "dvo_b200_pyramid_create_device_batch", "dvo_b200_match_batch_enqueue",
    "dvo_b200_selection_create", "dvo_b200_selection_create_device_batch", "dvo_b200_selection_retain",
    "dvo_b200_selection_release", "dvo_b200_selection_pyramid", "dvo_b200_selection_download",
    "dvo_b200_match_batch_selected", "dvo_b200_match_batch_selected_enqueue",
]

# dvo_b200_frame_format
FRAME_F32, FRAME_GREY8_RAW16, FRAME_BGR8_RAW16 = 0, 1, 2
# dvo_b200_predicate
PREDICATE_GRADIENT_THRESHOLD, PREDICATE_VALID_POINT, PREDICATE_MASK_ONLY = 0, 1, 2


def level_masks(mask0, levels: int):
    """Per-level masks of a level-0 mask [h, w] by the subsample chain of the depth: M_l(y, x) = M_0(y << l, x << l) on the
    (w >> l) x (h >> l) grid of level l.  What Engine.selections_from_tensors computes on the device."""
    m = np.asarray(mask0)
    h, w = m.shape
    return [np.ascontiguousarray(m[::1 << l, ::1 << l][:h >> l, :w >> l] != 0).astype(np.uint8) for l in range(levels)]


class Config(C.Structure):
    """dvo_b200_config; defaults = DenseTracker::Config (dense_tracking_config.cpp:27-42)."""
    _fields_ = [("first_level", C.c_int32), ("last_level", C.c_int32), ("max_iterations_per_level", C.c_int32),
                ("use_initial_estimate", C.c_int32), ("precision", C.c_double), ("mu", C.c_double),
                ("intensity_derivative_threshold", C.c_float), ("depth_derivative_threshold", C.c_float)]

    def __init__(self, **kw):
        super().__init__()
        self.first_level, self.last_level, self.max_iterations_per_level, self.use_initial_estimate = 3, 1, 100, 0
        self.precision, self.mu = 5e-7, 0.0
        self.intensity_derivative_threshold = self.depth_derivative_threshold = 0.0
        for k, v in kw.items():
            if not hasattr(self, k):
                raise AttributeError(k)
            setattr(self, k, v)


class IterationStats(C.Structure):
    _fields_ = [("level", C.c_int32), ("id", C.c_int32), ("valid_constraints", C.c_int64),
                ("tdist_log_likelihood", C.c_double), ("tdist_precision", C.c_double * 4),
                ("prior_log_likelihood", C.c_double), ("increment", C.c_double * 6), ("information", C.c_double * 36)]


class LevelStats(C.Structure):
    _fields_ = [("id", C.c_int32), ("termination", C.c_int32), ("max_valid_pixels", C.c_int64),
                ("valid_pixels", C.c_int64), ("num_iterations", C.c_int32), ("has_iteration_with_increment", C.c_int32),
                ("last_valid_constraints", C.c_int64), ("last_increment_valid_constraints", C.c_int64),
                ("last_increment_log_likelihood", C.c_double)]


class CResult(C.Structure):
    _fields_ = [("transformation", C.c_double * 16), ("information", C.c_double * 36), ("log_likelihood", C.c_double),
                ("num_levels", C.c_int32), ("num_iterations_total", C.c_int32), ("levels", LevelStats * MAX_LEVELS)]


class DeviceFrames(C.Structure):
    """dvo_b200_device_frames: n images in device memory, strides in bytes."""
    _fields_ = [("format", C.c_int32), ("width", C.c_int32), ("height", C.c_int32), ("reserved", C.c_int32),
                ("colour", C.c_void_p), ("colour_row_bytes", C.c_int64), ("colour_image_bytes", C.c_int64),
                ("depth", C.c_void_p), ("depth_row_bytes", C.c_int64), ("depth_image_bytes", C.c_int64),
                ("depth_scale", C.c_float)]


def device_frames(colour, depth, depth_scale=None) -> DeviceFrames:
    """dvo_b200_device_frames describing two torch tensors in place (no copy).

    colour: [n,h,w] float32 (intensity) or uint8 (grey), or [n,h,w,3] uint8 (interleaved BGR); depth: [n,h,w] float32
    (metres, NaN = invalid) with float32 colour, else 16-bit raw depth (torch.uint16, or int16 holding the same bits) and
    depth_scale.  Unit stride is required along the pixels of a row; element strides become byte strides."""
    import torch
    u16 = tuple(t for t in (getattr(torch, "uint16", None), torch.int16) if t is not None)
    if colour.dtype == torch.float32:
        fmt = FRAME_F32
        if depth.dtype != torch.float32:
            raise ValueError("float32 colour takes float32 depth in metres")
    elif colour.dtype == torch.uint8:
        fmt = FRAME_BGR8_RAW16 if colour.dim() == 4 else FRAME_GREY8_RAW16
        if depth.dtype not in u16:
            raise ValueError("8-bit colour takes 16-bit raw depth (torch.uint16 or int16)")
        if depth_scale is None:
            raise ValueError("16-bit raw depth needs depth_scale")
    else:
        raise ValueError(f"colour dtype {colour.dtype}: float32, or uint8 grey / BGR")
    if depth.dim() != 3 or colour.dim() != (4 if fmt == FRAME_BGR8_RAW16 else 3) or tuple(colour.shape[:3]) != tuple(depth.shape):
        raise ValueError(f"shapes {tuple(colour.shape)} / {tuple(depth.shape)}: colour [n,h,w] or [n,h,w,3], depth [n,h,w]")
    if fmt == FRAME_BGR8_RAW16 and (colour.shape[3] != 3 or colour.stride(3) != 1 or colour.stride(2) != 3):
        raise ValueError("BGR colour needs 3 interleaved channels with unit stride, pixels 3 bytes apart")
    if fmt != FRAME_BGR8_RAW16 and colour.stride(2) != 1:
        raise ValueError("colour needs unit stride along a row")
    if depth.stride(2) != 1:
        raise ValueError("depth needs unit stride along a row")
    n, h, w = depth.shape

    def strides(t):
        row = t.stride(1) * t.element_size()
        return row, (t.stride(0) * t.element_size() if n > 1 else h * row)

    f = DeviceFrames()
    f.format, f.width, f.height, f.reserved = fmt, w, h, 0
    f.colour, (f.colour_row_bytes, f.colour_image_bytes) = colour.data_ptr(), strides(colour)
    f.depth, (f.depth_row_bytes, f.depth_image_bytes) = depth.data_ptr(), strides(depth)
    f.depth_scale = float(depth_scale) if depth_scale is not None else 0.0
    return f


def result_transformations(records):
    """[n, 4, 4] float64 view (no copy) of Result.Transformation in a uint8 tensor of n dvo_b200_result records, as
    Engine.match_batch_enqueue returns it: transformation is the first field of the record."""
    import torch
    return records.view(torch.float64)[:, :16].view(records.shape[0], 4, 4)


class Result:
    """Python view of dvo_b200_result (dvo::DenseTracker::Result, dense_tracking.h:125-140)."""

    def __init__(self, c: CResult, iterations=None):
        self.transformation = np.array(c.transformation).reshape(4, 4)
        self.information = np.array(c.information).reshape(6, 6)
        self.log_likelihood = c.log_likelihood
        self.num_iterations_total = c.num_iterations_total
        self.levels = []
        for i in range(c.num_levels):
            l = c.levels[i]
            self.levels.append({"id": l.id, "termination": l.termination, "max_valid_pixels": l.max_valid_pixels,
                                "valid_pixels": l.valid_pixels, "num_iterations": l.num_iterations,
                                "has_iteration_with_increment": bool(l.has_iteration_with_increment),
                                "last_valid_constraints": l.last_valid_constraints,
                                "last_increment_valid_constraints": l.last_increment_valid_constraints,
                                "last_increment_log_likelihood": l.last_increment_log_likelihood})
        self.iterations = iterations or []

    def is_nan(self) -> bool:  # Result::isNaN (dense_tracking_config.cpp:96-99)
        return not (np.isfinite(self.transformation.sum()) and np.isfinite(self.information.sum()))


_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(f"{LIB_PATH} is missing: run `python __graft_entry__.py` (nvcc, sm_100a). "
                           "There is no CPU fallback for the engine.")
    L = C.CDLL(LIB_PATH)
    vp, fp, dp, i32, i64 = C.c_void_p, C.POINTER(C.c_float), C.POINTER(C.c_double), C.c_int32, C.c_int64
    L.dvo_b200_abi_version.restype = C.c_int
    L.dvo_b200_create.argtypes = [C.c_int, vp, C.POINTER(vp)]
    L.dvo_b200_destroy.argtypes = [vp]
    L.dvo_b200_stream.restype = vp
    L.dvo_b200_stream.argtypes = [vp]
    L.dvo_b200_synchronize.argtypes = [vp]
    L.dvo_b200_last_error.restype = C.c_char_p
    L.dvo_b200_last_error.argtypes = [vp]
    L.dvo_b200_config_default.argtypes = [C.POINTER(Config)]
    L.dvo_b200_config_default.restype = None
    for f in (L.dvo_b200_kernel_launches, L.dvo_b200_h2d_bytes, L.dvo_b200_d2h_bytes):
        f.restype = i64
        f.argtypes = [vp]
    L.dvo_b200_pyramid_create.argtypes = [vp, vp, vp, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32, C.POINTER(vp)]
    L.dvo_b200_pyramid_create_batch.argtypes = [vp, i32, vp, vp, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32, C.POINTER(vp)]
    L.dvo_b200_pyramid_create_raw.argtypes = [vp, vp, vp, C.c_float, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32, C.POINTER(vp)]
    L.dvo_b200_pyramid_create_raw_batch.argtypes = [vp, i32, vp, vp, C.c_float, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32, C.POINTER(vp)]
    L.dvo_b200_pyramid_create_bgr_batch.argtypes = [vp, i32, vp, vp, C.c_float, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32, C.POINTER(vp)]
    L.dvo_b200_pyramid_device.argtypes = [vp]
    L.dvo_b200_pyramid_create_device_batch.argtypes = [vp, i32, C.POINTER(DeviceFrames), C.c_float, C.c_float, C.c_float, C.c_float, i32,
                                                       C.POINTER(vp)]
    L.dvo_b200_match_batch_enqueue.argtypes = [vp, C.POINTER(Config), i32, C.POINTER(vp), C.POINTER(vp), vp, vp]
    L.dvo_b200_selection_create.argtypes = [vp, vp, i32, C.c_float, C.c_float, C.POINTER(C.c_void_p), C.POINTER(vp)]
    L.dvo_b200_selection_create_device_batch.argtypes = [vp, i32, C.POINTER(vp), i32, C.c_float, C.c_float, vp, i64, i64, C.POINTER(vp)]
    L.dvo_b200_selection_retain.argtypes = [vp]
    L.dvo_b200_selection_release.argtypes = [vp]
    L.dvo_b200_selection_pyramid.restype = vp
    L.dvo_b200_selection_pyramid.argtypes = [vp]
    L.dvo_b200_selection_download.argtypes = [vp, vp, i32, C.POINTER(i64), C.POINTER(C.c_uint8)]
    L.dvo_b200_match_batch_selected.argtypes = [vp, C.POINTER(Config), i32, C.POINTER(vp), C.POINTER(vp), dp, C.POINTER(CResult),
                                                C.POINTER(IterationStats), i32]
    L.dvo_b200_match_batch_selected_enqueue.argtypes = [vp, C.POINTER(Config), i32, C.POINTER(vp), C.POINTER(vp), vp, vp]
    L.dvo_b200_sharded_create.argtypes = [i32, C.POINTER(i32), C.POINTER(vp)]
    L.dvo_b200_sharded_destroy.argtypes = [vp]
    L.dvo_b200_sharded_num_shards.argtypes = [vp]
    L.dvo_b200_sharded_ctx.restype = vp
    L.dvo_b200_sharded_ctx.argtypes = [vp, i32]
    L.dvo_b200_sharded_last_error.restype = C.c_char_p
    L.dvo_b200_sharded_last_error.argtypes = [vp]
    L.dvo_b200_shard_range.argtypes = [i64, i32, i32, C.POINTER(i64), C.POINTER(i64)]
    L.dvo_b200_sharded_pyramid_create_batch.argtypes = [vp, i32, vp, vp, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32, C.POINTER(vp)]
    L.dvo_b200_sharded_pyramid_create_raw_batch.argtypes = [vp, i32, vp, vp, C.c_float, i32, i32, C.c_float, C.c_float, C.c_float, C.c_float, i32,
                                                        C.POINTER(vp)]
    L.dvo_b200_match_batch_sharded.argtypes = [vp, C.POINTER(Config), i32, C.POINTER(vp), C.POINTER(vp), dp, C.POINTER(CResult),
                                               C.POINTER(IterationStats), i32]
    L.dvo_b200_pyramid_retain.argtypes = [vp]
    L.dvo_b200_pyramid_release.argtypes = [vp]
    L.dvo_b200_pyramid_num_levels.argtypes = [vp]
    L.dvo_b200_pyramid_level_info.argtypes = [vp, i32, C.POINTER(i32), C.POINTER(i32), fp]
    L.dvo_b200_pyramid_download.argtypes = [vp, vp, i32, fp]
    L.dvo_b200_pyramid_select.argtypes = [vp, vp, i32, C.c_float, C.c_float, C.POINTER(i64), C.POINTER(C.c_uint8)]
    L.dvo_b200_match.argtypes = [vp, C.POINTER(Config), vp, vp, dp, C.POINTER(CResult)]
    L.dvo_b200_match_batch.argtypes = [vp, C.POINTER(Config), i32, C.POINTER(vp), C.POINTER(vp), dp, C.POINTER(CResult),
                                       C.POINTER(IterationStats), i32]
    L.dvo_b200_match_batch_device.argtypes = [vp, C.POINTER(Config), i32, C.POINTER(vp), C.POINTER(vp), dp, vp]
    L.dvo_b200_residual_image.argtypes = [vp, C.POINTER(Config), vp, vp, i32, dp, fp, C.POINTER(i64)]
    L.dvo_b200_intensity_error_image.argtypes = [vp, C.POINTER(Config), vp, vp, i32, dp, fp, C.POINTER(i64)]
    L.dvo_b200_linearize.argtypes = [vp, C.POINTER(Config), vp, vp, i32, dp, i32, fp, C.POINTER(i64), fp, fp, dp, dp]
    L.dvo_b200_profile_enable.argtypes = [vp, i32]
    L.dvo_b200_profile_read.argtypes = [vp, dp, C.POINTER(i64), i32]
    _lib = L
    return L


class Pyramid:
    """Owning handle of a dvo_b200_pyramid (device mirror of dvo::core::RgbdImagePyramid)."""

    def __init__(self, engine: "Engine", handle: int):
        self.engine, self.handle = engine, handle

    @property
    def num_levels(self) -> int:
        return load_library().dvo_b200_pyramid_num_levels(self.handle)

    def level_info(self, level: int):
        w, h = C.c_int32(), C.c_int32()
        K = (C.c_float * 4)()
        self.engine._check(load_library().dvo_b200_pyramid_level_info(self.handle, level, C.byref(w), C.byref(h), K))
        return w.value, h.value, tuple(K)

    def download(self, level: int) -> np.ndarray:
        w, h, _ = self.level_info(level)
        out = np.empty((6, h, w), dtype=np.float32)
        self.engine._check(load_library().dvo_b200_pyramid_download(self.engine.ctx, self.handle, level,
                                                                    out.ctypes.data_as(C.POINTER(C.c_float))))
        return out

    def select(self, level: int, ti: float = 0.0, td: float = 0.0):
        w, h, _ = self.level_info(level)
        mask = np.zeros((h, w), dtype=np.uint8)
        cnt = C.c_int64()
        self.engine._check(load_library().dvo_b200_pyramid_select(self.engine.ctx, self.handle, level, ti, td, C.byref(cnt),
                                                                  mask.ctypes.data_as(C.POINTER(C.c_uint8))))
        return cnt.value, mask

    def release(self):
        if self.handle:
            load_library().dvo_b200_pyramid_release(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


class Selection:
    """Owning handle of a dvo_b200_selection (dvo::core::PointSelection with its own predicate and mask).  Keeps the Python
    Pyramid it was built from alive too, although the selection itself retains the device pyramid."""

    def __init__(self, engine: "Engine", handle: int, pyramid: Pyramid):
        self.engine, self.handle, self.pyramid = engine, handle, pyramid

    def download(self, level: int):
        """(S, mask[h, w] uint8): the number of selected points of the level and where they are."""
        w, h, _ = self.pyramid.level_info(level)
        mask = np.zeros((h, w), dtype=np.uint8)
        cnt = C.c_int64()
        ctx = self.engine.ctx if self.engine is not None else None
        rc = load_library().dvo_b200_selection_download(ctx, self.handle, level, C.byref(cnt), mask.ctypes.data_as(C.POINTER(C.c_uint8)))
        if rc != 0:
            raise RuntimeError(f"dvo_b200_selection_download: status {rc}")
        return cnt.value, mask

    def release(self):
        if self.handle:
            load_library().dvo_b200_selection_release(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass


def _reference_handles(refs):
    """(handles, selected): pyramids or selections as references of one batch, not mixed."""
    sel = [isinstance(r, Selection) for r in refs]
    if any(sel) and not all(sel):
        raise ValueError("references of one batch are all Pyramids or all Selections")
    return (C.c_void_p * len(refs))(*[r.handle for r in refs]), all(sel)


class Engine:
    """One dvo_b200_ctx (one CUDA stream on one device)."""

    def __init__(self, device: int = 0, stream: int | None = None):
        self.lib = load_library()
        ctx = C.c_void_p()
        rc = self.lib.dvo_b200_create(device, C.c_void_p(stream) if stream else None, C.byref(ctx))
        if rc != 0:
            raise RuntimeError(f"dvo_b200_create(device={device}) failed with status {rc}: no usable CUDA device "
                               "(the engine has no CPU fallback)")
        self.ctx = ctx
        self.device = device

    def close(self):
        if getattr(self, "ctx", None):
            self.lib.dvo_b200_destroy(self.ctx)
            self.ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc: int):
        if rc != 0:
            raise RuntimeError(f"dvo_b200 status {rc}: {self.lib.dvo_b200_last_error(self.ctx).decode()}")

    @property
    def stream(self) -> int:
        return self.lib.dvo_b200_stream(self.ctx)

    def synchronize(self):
        self._check(self.lib.dvo_b200_synchronize(self.ctx))

    def kernel_launches(self) -> int:
        return self.lib.dvo_b200_kernel_launches(self.ctx)

    def h2d_bytes(self) -> int:
        return self.lib.dvo_b200_h2d_bytes(self.ctx)

    def d2h_bytes(self) -> int:
        return self.lib.dvo_b200_d2h_bytes(self.ctx)

    # ---- pyramids ----
    def pyramid(self, intensity, depth, intrinsics, levels: int) -> Pyramid:
        I = np.ascontiguousarray(intensity, dtype=np.float32)
        Z = np.ascontiguousarray(depth, dtype=np.float32)
        assert I.ndim == 2 and I.shape == Z.shape
        h, w = I.shape
        fx, fy, ox, oy = intrinsics
        out = C.c_void_p()
        self._check(self.lib.dvo_b200_pyramid_create(self.ctx, I.ctypes.data, Z.ctypes.data, w, h, fx, fy, ox, oy, levels, C.byref(out)))
        self.synchronize()  # numpy temporaries may die
        return Pyramid(self, out.value)

    def pyramid_batch(self, intensity, depth, intrinsics, levels: int, host_ptrs=None) -> list[Pyramid]:
        """intensity/depth: [n,h,w] float32 arrays, or (ptr_I, ptr_Z, n, h, w) raw host pointers via host_ptrs."""
        if host_ptrs is not None:
            pI, pZ, n, h, w = host_ptrs
        else:
            I = np.ascontiguousarray(intensity, dtype=np.float32)
            Z = np.ascontiguousarray(depth, dtype=np.float32)
            assert I.ndim == 3 and I.shape == Z.shape
            n, h, w = I.shape
            pI, pZ = I.ctypes.data, Z.ctypes.data
        fx, fy, ox, oy = intrinsics
        out = (C.c_void_p * n)()
        self._check(self.lib.dvo_b200_pyramid_create_batch(self.ctx, n, pI, pZ, w, h, fx, fy, ox, oy, levels, out))
        if host_ptrs is None:
            self.synchronize()
        return [Pyramid(self, out[i]) for i in range(n)]

    def pyramid_raw_batch(self, host_ptrs, depth_scale, intrinsics, levels: int) -> list[Pyramid]:
        """host_ptrs = (ptr_grey_u8, ptr_depth_u16, n, h, w): n consecutive raw images in (pinned) host memory."""
        pG, pD, n, h, w = host_ptrs
        fx, fy, ox, oy = intrinsics
        out = (C.c_void_p * n)()
        self._check(self.lib.dvo_b200_pyramid_create_raw_batch(self.ctx, n, pG, pD, depth_scale, w, h, fx, fy, ox, oy, levels, out))
        return [Pyramid(self, out[i]) for i in range(n)]

    def pyramid_bgr_batch(self, host_ptrs, depth_scale, intrinsics, levels: int) -> list[Pyramid]:
        """host_ptrs = (ptr_bgr_u8x3, ptr_depth_u16, n, h, w): n consecutive interleaved-BGR images and raw depth images
        in (pinned) host memory; grey conversion (OpenCV BGR2GRAY) and depth scaling run on the device."""
        pC, pD, n, h, w = host_ptrs
        fx, fy, ox, oy = intrinsics
        out = (C.c_void_p * n)()
        self._check(self.lib.dvo_b200_pyramid_create_bgr_batch(self.ctx, n, pC, pD, depth_scale, w, h, fx, fy, ox, oy, levels, out))
        return [Pyramid(self, out[i]) for i in range(n)]

    def pyramid_raw(self, grey_u8, depth_u16, depth_scale, intrinsics, levels: int) -> Pyramid:
        G = np.ascontiguousarray(grey_u8, dtype=np.uint8)
        D = np.ascontiguousarray(depth_u16, dtype=np.uint16)
        assert G.ndim == 2 and G.shape == D.shape
        h, w = G.shape
        fx, fy, ox, oy = intrinsics
        out = C.c_void_p()
        self._check(self.lib.dvo_b200_pyramid_create_raw(self.ctx, G.ctypes.data, D.ctypes.data, depth_scale, w, h, fx, fy, ox, oy,
                                                         levels, C.byref(out)))
        self.synchronize()
        return Pyramid(self, out.value)

    # ---- point selections ----
    def selection(self, pyramid: Pyramid, predicate: int = PREDICATE_GRADIENT_THRESHOLD, ti: float = 0.0, td: float = 0.0,
                  masks=None) -> Selection:
        """dvo_b200_selection_create: a selection of `pyramid` by `predicate` (PREDICATE_*; ti / td for the gradient
        threshold), optionally restricted by host masks: one [h_l, w_l] array per level (nonzero = allowed) or None for a
        level without mask.  level_masks() derives them from a level-0 mask."""
        n = pyramid.num_levels
        keep, arr = [], None
        if masks is not None:
            if len(masks) != n:
                raise ValueError(f"masks: {n} levels expected, got {len(masks)}")
            arr = (C.c_void_p * n)()
            for l, m in enumerate(masks):
                if m is None:
                    continue
                w, h, _ = pyramid.level_info(l)
                a = np.ascontiguousarray(np.asarray(m) != 0, dtype=np.uint8)
                if a.shape != (h, w):
                    raise ValueError(f"mask of level {l}: shape {a.shape}, expected {(h, w)}")
                keep.append(a)
                arr[l] = a.ctypes.data
        out = C.c_void_p()
        self._check(self.lib.dvo_b200_selection_create(self.ctx, pyramid.handle, int(predicate), float(ti), float(td), arr, C.byref(out)))
        return Selection(self, out.value, pyramid)

    def selections_from_tensors(self, pyramids, masks=None, predicate: int = PREDICATE_GRADIENT_THRESHOLD, ti: float = 0.0,
                                td: float = 0.0) -> list[Selection]:
        """dvo_b200_selection_create_device_batch: one selection per pyramid in one build.  masks: None, or a CUDA
        uint8 / bool tensor [n, h, w] of level-0 masks (nonzero = allowed) at any strides with unit stride along a row,
        read in place; coarser levels subsample it like the depth.  Ordered after the current torch stream; the masks are
        marked as used on the context's stream."""
        import torch
        n = len(pyramids)
        ph = (C.c_void_p * n)(*[p.handle for p in pyramids])
        ptr, row, img = None, 0, 0
        ext = self._torch_stream()
        if masks is not None:
            self._check_on_device(masks, "masks")
            if masks.dtype not in (torch.uint8, torch.bool) or masks.dim() != 3 or masks.shape[0] != n:
                raise ValueError(f"masks: uint8 / bool [{n},h,w] expected, got {masks.dtype} {tuple(masks.shape)}")
            if masks.stride(2) != 1:
                raise ValueError("masks need unit stride along a row")
            ptr, row = masks.data_ptr(), masks.stride(1)
            img = masks.stride(0) if n > 1 else masks.shape[1] * row
            ext.wait_stream(torch.cuda.current_stream(masks.device))
        out = (C.c_void_p * n)()
        self._check(self.lib.dvo_b200_selection_create_device_batch(self.ctx, n, ph, int(predicate), float(ti), float(td), ptr, row, img, out))
        if masks is not None:
            masks.record_stream(ext)
        return [Selection(self, out[i], pyramids[i]) for i in range(n)]

    # ---- alignment ----
    def match(self, ref: Pyramid, cur: Pyramid, cfg: Config, T_init=None, with_iterations: bool = False) -> Result:
        return self.match_batch([ref], [cur], cfg, None if T_init is None else [T_init], with_iterations)[0]

    def match_batch(self, refs, curs, cfg: Config, T_init=None, with_iterations: bool = False, raw: bool = False):
        """refs: Pyramids (their built-in selection with cfg's thresholds) or Selections (their own predicate and mask)."""
        n = len(refs)
        assert n == len(curs) and n > 0
        rh, selected = _reference_handles(refs)
        ch = (C.c_void_p * n)(*[p.handle for p in curs])
        T = None
        if T_init is not None:
            T = np.ascontiguousarray(np.asarray(T_init, dtype=np.float64).reshape(n, 16))
        res = (CResult * n)()
        max_log = 0
        log = None
        if with_iterations:
            max_log = (cfg.first_level - cfg.last_level + 1) * (cfg.max_iterations_per_level + 1)
            log = (IterationStats * (n * max_log))()
        fn = self.lib.dvo_b200_match_batch_selected if selected else self.lib.dvo_b200_match_batch
        self._check(fn(self.ctx, C.byref(cfg), n, rh, ch, T.ctypes.data_as(C.POINTER(C.c_double)) if T is not None else None,
                       res, log, max_log))
        if raw:
            return res
        out = []
        for i in range(n):
            its = []
            if with_iterations:
                for k in range(res[i].num_iterations_total):
                    s = log[i * max_log + k]
                    its.append({"level": s.level, "id": s.id, "n": s.valid_constraints, "nll": s.tdist_log_likelihood,
                                "precision": np.array(s.tdist_precision).reshape(2, 2), "prior": s.prior_log_likelihood,
                                "x": np.array(s.increment), "A": np.array(s.information).reshape(6, 6)})
            out.append(Result(res[i], its))
        return out

    def match_batch_device(self, refs, curs, cfg: Config, d_results_ptr: int, T_init=None):
        n = len(refs)
        rh = (C.c_void_p * n)(*[p.handle for p in refs])
        ch = (C.c_void_p * n)(*[p.handle for p in curs])
        T = None
        if T_init is not None:
            T = np.ascontiguousarray(np.asarray(T_init, dtype=np.float64).reshape(n, 16))
        self._check(self.lib.dvo_b200_match_batch_device(self.ctx, C.byref(cfg), n, rh, ch,
                                                         T.ctypes.data_as(C.POINTER(C.c_double)) if T is not None else None,
                                                         C.c_void_p(d_results_ptr)))

    # ---- frames and results in GPU memory (torch tensors) ----
    def _torch_stream(self):
        """The context's stream as a torch stream (for ordering against torch work)."""
        import torch
        if getattr(self, "_ext_stream", None) is None:
            self._ext_stream = torch.cuda.ExternalStream(self.stream, device=torch.device("cuda", self.device))
        return self._ext_stream

    def _check_on_device(self, t, name):
        if not t.is_cuda or t.device.index != self.device:
            raise ValueError(f"{name} must be a CUDA tensor on cuda:{self.device} (got {t.device})")

    def pyramid_from_tensors(self, colour, depth, intrinsics, levels: int, depth_scale=None) -> list[Pyramid]:
        """Pyramids of n frames already in GPU memory, read in place (dvo_b200_pyramid_create_device_batch).

        colour: [n,h,w] float32 or uint8, or [n,h,w,3] uint8 BGR; depth: [n,h,w] float32 metres, or 16-bit raw depth
        (torch.uint16 / int16) with depth_scale.  Any row / image strides with unit stride along a row.  The context's stream
        waits for the work already queued on the current torch stream, and the inputs are marked as used on the context's
        stream, so the caching allocator does not reuse their memory before the build has read them.  Equal bit for bit to
        the host entry point of the same format on the same pixels."""
        import torch
        self._check_on_device(colour, "colour")
        self._check_on_device(depth, "depth")
        frames = device_frames(colour, depth, depth_scale)
        n = depth.shape[0]
        ext = self._torch_stream()
        ext.wait_stream(torch.cuda.current_stream(colour.device))
        fx, fy, ox, oy = intrinsics
        out = (C.c_void_p * n)()
        self._check(self.lib.dvo_b200_pyramid_create_device_batch(self.ctx, n, C.byref(frames), fx, fy, ox, oy, levels, out))
        colour.record_stream(ext)
        depth.record_stream(ext)
        return [Pyramid(self, out[i]) for i in range(n)]

    def match_batch_enqueue(self, refs, curs, cfg: Config, T_init=None):
        """dvo_b200_match_batch_enqueue: returns a uint8 CUDA tensor [n, sizeof(dvo_b200_result)] of result records,
        ordered onto the current torch stream; the host does not wait for the GPU.  T_init: CUDA float64 [n,4,4]
        (Result.Transformation on entry, read iff cfg.use_initial_estimate).  result_transformations() views the poses.
        refs: Pyramids or Selections, as for match_batch."""
        import torch
        n = len(refs)
        assert n == len(curs) and n > 0
        dev = torch.device("cuda", self.device)
        cur = torch.cuda.current_stream(dev)
        T = None
        if T_init is not None:
            self._check_on_device(T_init, "T_init")
            if T_init.dtype != torch.float64 or tuple(T_init.shape) != (n, 4, 4):
                raise ValueError(f"T_init: float64 [{n},4,4] expected, got {T_init.dtype} {tuple(T_init.shape)}")
            T = T_init.contiguous()
        records = torch.empty((n, C.sizeof(CResult)), dtype=torch.uint8, device=dev)
        rh, selected = _reference_handles(refs)
        ch = (C.c_void_p * n)(*[p.handle for p in curs])
        ext = self._torch_stream()
        ext.wait_stream(cur)
        fn = self.lib.dvo_b200_match_batch_selected_enqueue if selected else self.lib.dvo_b200_match_batch_enqueue
        self._check(fn(self.ctx, C.byref(cfg), n, rh, ch, T.data_ptr() if T is not None else None, records.data_ptr()))
        records.record_stream(ext)
        if T is not None:
            T.record_stream(ext)
        cur.wait_stream(ext)
        return records

    def residual_image(self, ref: Pyramid, cur: Pyramid, level: int, T, cfg: Config | None = None):
        cfg = cfg or Config()
        w, h, _ = ref.level_info(level)
        out = np.empty((7, h, w), dtype=np.float32)
        T = np.ascontiguousarray(np.asarray(T, dtype=np.float64).reshape(16))
        cnt = C.c_int64()
        self._check(self.lib.dvo_b200_residual_image(self.ctx, C.byref(cfg), ref.handle, cur.handle, level,
                                                     T.ctypes.data_as(C.POINTER(C.c_double)),
                                                     out.ctypes.data_as(C.POINTER(C.c_float)), C.byref(cnt)))
        return cnt.value, out

    def intensity_error_image(self, ref: Pyramid, cur: Pyramid, level: int, T, cfg: Config | None = None):
        """DenseTracker::computeIntensityErrorImage (dense_tracking.cpp:378-444) -> (n_written, image[h, w])."""
        cfg = cfg or Config()
        w, h, _ = ref.level_info(level)
        out = np.empty((h, w), dtype=np.float32)
        T = np.ascontiguousarray(np.asarray(T, dtype=np.float64).reshape(16))
        cnt = C.c_int64()
        self._check(self.lib.dvo_b200_intensity_error_image(self.ctx, C.byref(cfg), ref.handle, cur.handle, level,
                                                            T.ctypes.data_as(C.POINTER(C.c_double)),
                                                            out.ctypes.data_as(C.POINTER(C.c_float)), C.byref(cnt)))
        return int(cnt.value), out

    def linearize(self, ref: Pyramid, cur: Pyramid, level: int, T, use_weights=False, prev_precision=None, cfg: Config | None = None):
        cfg = cfg or Config()
        T = np.ascontiguousarray(np.asarray(T, dtype=np.float64).reshape(16))
        pp = np.ascontiguousarray(np.asarray(prev_precision if prev_precision is not None else np.zeros(4), dtype=np.float32).reshape(4))
        P = np.zeros(4, dtype=np.float32)
        ll = C.c_float()
        A = np.zeros(36)
        b = np.zeros(6)
        cnt = C.c_int64()
        self._check(self.lib.dvo_b200_linearize(self.ctx, C.byref(cfg), ref.handle, cur.handle, level,
                                                T.ctypes.data_as(C.POINTER(C.c_double)), int(use_weights),
                                                pp.ctypes.data_as(C.POINTER(C.c_float)), C.byref(cnt),
                                                P.ctypes.data_as(C.POINTER(C.c_float)), C.byref(ll),
                                                A.ctypes.data_as(C.POINTER(C.c_double)), b.ctypes.data_as(C.POINTER(C.c_double))))
        return {"n": cnt.value, "precision": P.reshape(2, 2), "ll": ll.value, "A": A.reshape(6, 6), "b": b}

    # ---- profiling ----
    def profile_enable(self, on: bool = True):
        self._check(self.lib.dvo_b200_profile_enable(self.ctx, int(on)))

    def profile_read(self, reset: bool = True):
        ms = (C.c_double * 8)()
        ln = (C.c_int64 * 8)()
        self._check(self.lib.dvo_b200_profile_read(self.ctx, ms, ln, int(reset)))
        names = ["residual", "normal", "pair_step", "pyramid", "select"]
        return {names[i]: {"ms": ms[i], "launches": ln[i]} for i in range(len(names))}


class ShardedEngine:
    """dvo_b200_sharded: one process, one context + host thread per device, contiguous shards of pair indices
    (the C-ABI form of the multi-GPU path; the multi-process form is dvo_slam_b200/distributed.py)."""

    def __init__(self, devices):
        self.lib = load_library()
        devs = (C.c_int32 * len(devices))(*devices)
        h = C.c_void_p()
        rc = self.lib.dvo_b200_sharded_create(len(devices), devs, C.byref(h))
        if rc != 0:
            raise RuntimeError(f"dvo_b200_sharded_create({list(devices)}) failed with status {rc}: no usable CUDA device "
                               "(the engine has no CPU fallback)")
        self.h = h
        self.devices = list(devices)

    def close(self):
        if getattr(self, "h", None):
            self.lib.dvo_b200_sharded_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, rc):
        if rc != 0:
            raise RuntimeError(f"dvo_b200 sharded status {rc}: {self.lib.dvo_b200_sharded_last_error(self.h).decode()}")

    def shard_range(self, total, shard):
        b, e = C.c_int64(), C.c_int64()
        self._check(self.lib.dvo_b200_shard_range(total, len(self.devices), shard, C.byref(b), C.byref(e)))
        return b.value, e.value

    def pyramid_batch(self, intensity, depth, intrinsics, levels):
        """intensity, depth: float32 arrays [n, h, w] on the host -> n pyramid handles (image i on its shard's device)."""
        I = np.ascontiguousarray(intensity, dtype=np.float32)
        Z = np.ascontiguousarray(depth, dtype=np.float32)
        n, h, w = I.shape
        out = (C.c_void_p * n)()
        fx, fy, ox, oy = [float(v) for v in intrinsics]
        self._check(self.lib.dvo_b200_sharded_pyramid_create_batch(self.h, n, I.ctypes.data, Z.ctypes.data, w, h, fx, fy, ox, oy, levels, out))
        return [C.c_void_p(v) for v in out]

    def release(self, handles):
        for p in handles:
            self.lib.dvo_b200_pyramid_release(p)

    def match_batch(self, refs, curs, cfg: Config, T_init=None):
        n = len(refs)
        rh = (C.c_void_p * n)(*[p.value for p in refs])
        ch = (C.c_void_p * n)(*[p.value for p in curs])
        T = None
        if T_init is not None:
            T = np.ascontiguousarray(np.asarray(T_init, dtype=np.float64).reshape(n, 16))
        res = (CResult * n)()
        self._check(self.lib.dvo_b200_match_batch_sharded(self.h, C.byref(cfg), n, rh, ch,
                                                          T.ctypes.data_as(C.POINTER(C.c_double)) if T is not None else None,
                                                          res, None, 0))
        return res
