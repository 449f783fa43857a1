"""The CPU oracle with reference point selections of any predicate and per-pixel masks (tests/native/selection_oracle.cpp).

Test infrastructure.  The library is the oracle's source (oracle/dvo_oracle.cpp, included unchanged) plus orc_select_ex /
orc_match_ex, compiled on first use in a temporary directory (removed once loaded) with the oracle's own compiler flags (oracle/Makefile), so
its plain functions compute what oracle/liboracle.so computes.  Pyramids of this module belong to its own library."""
from __future__ import annotations

import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

from oracle import oracle_py as orc

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SRC = os.path.join(ROOT, "tests", "native", "selection_oracle.cpp")
# oracle/Makefile CXXFLAGS
FLAGS = ["-std=c++17", "-O3", "-mavx2", "-mfma", "-msse3", "-ffp-contract=off", "-frounding-math", "-fPIC", "-shared"]

# = dvo_b200_predicate
PREDICATE_GRADIENT_THRESHOLD, PREDICATE_VALID_POINT, PREDICATE_MASK_ONLY = 0, 1, 2

_lib = None
_dir = None


def lib():
    global _lib, _dir
    if _lib is None:
        _dir = tempfile.mkdtemp(prefix="selection_oracle_")
        so = os.path.join(_dir, "libselection_oracle.so")
        cxx = os.environ.get("CXX") or shutil.which("g++") or "g++"
        subprocess.check_call([cxx] + FLAGS + ["-I", os.path.join(ROOT, "oracle"), "-o", so, SRC])
        L = C.CDLL(so)
        shutil.rmtree(_dir, ignore_errors=True)   # the loaded library stays mapped
        fp, dp, u8p = C.POINTER(C.c_float), C.POINTER(C.c_double), C.POINTER(C.c_uint8)
        L.orc_pyramid_create.restype = C.c_void_p
        L.orc_pyramid_create.argtypes = [fp, fp, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_float, C.c_int]
        L.orc_pyramid_destroy.argtypes = [C.c_void_p]
        L.orc_pyramid_level_info.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_int), C.POINTER(C.c_int), fp]
        L.orc_select.restype = C.c_int64
        L.orc_select.argtypes = [C.c_void_p, C.c_int, C.c_float, C.c_float, C.POINTER(orc.Mode), u8p]
        L.orc_select_ex.restype = C.c_int64
        L.orc_select_ex.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_float, C.c_float, u8p, C.POINTER(orc.Mode), u8p]
        L.orc_match.restype = C.c_int
        L.orc_match.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(orc.Config), dp, C.POINTER(orc.Mode), C.POINTER(orc.Result),
                                C.POINTER(orc.IterationStats), C.c_int, C.POINTER(C.c_int)]
        L.orc_match_ex.restype = C.c_int
        L.orc_match_ex.argtypes = [C.c_void_p, C.c_void_p, C.POINTER(orc.Config), C.c_int, C.c_float, C.c_float, C.POINTER(C.c_void_p), dp,
                                   C.POINTER(orc.Mode), C.POINTER(orc.Result), C.POINTER(orc.IterationStats), C.c_int, C.POINTER(C.c_int)]
        _lib = L
    return _lib


class Pyramid:
    def __init__(self, intensity, depth, intrinsics, levels):
        I = np.ascontiguousarray(np.asarray(intensity, dtype=np.float32))
        Z = np.ascontiguousarray(np.asarray(depth, dtype=np.float32))
        h, w = I.shape
        fx, fy, ox, oy = intrinsics
        fp = C.POINTER(C.c_float)
        self.h = lib().orc_pyramid_create(I.ctypes.data_as(fp), Z.ctypes.data_as(fp), w, h, fx, fy, ox, oy, levels)
        if not self.h:
            raise ValueError("orc_pyramid_create failed")
        self.levels = levels

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h and _lib is not None:
            try:
                _lib.orc_pyramid_destroy(h)
            except Exception:
                pass

    def level_info(self, level):
        w, h = C.c_int(), C.c_int()
        K = (C.c_float * 4)()
        lib().orc_pyramid_level_info(self.h, level, C.byref(w), C.byref(h), K)
        return w.value, h.value, tuple(K)


def _u8(a):
    return np.ascontiguousarray(np.asarray(a) != 0, dtype=np.uint8)


def _u8p(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint8)) if a is not None else None


def select(ref: Pyramid, level, ti=0.0, td=0.0, m=None):
    """oracle_py.select on this library"""
    w, h, _ = ref.level_info(level)
    mask = np.zeros((h, w), dtype=np.uint8)
    S = lib().orc_select(ref.h, level, ti, td, C.byref(m) if m is not None else None, _u8p(mask))
    return int(S), mask


def select_ex(ref: Pyramid, level, predicate=PREDICATE_GRADIENT_THRESHOLD, ti=0.0, td=0.0, level_mask=None, m=None):
    """(S, mask[h_l, w_l]) of a predicate ANDed with an optional mask of this level (nonzero = allowed)."""
    w, h, _ = ref.level_info(level)
    mask = np.zeros((h, w), dtype=np.uint8)
    lm = None if level_mask is None else _u8(level_mask)
    assert lm is None or lm.shape == (h, w)
    S = lib().orc_select_ex(ref.h, level, int(predicate), ti, td, _u8p(lm), C.byref(m) if m is not None else None, _u8p(mask))
    return int(S), mask


def _result(res, its, n_iters, max_iters):
    levels = [{"id": res.levels[i].id, "termination": res.levels[i].termination, "max_valid_pixels": res.levels[i].max_valid_pixels,
               "valid_pixels": res.levels[i].valid_pixels, "num_iterations": res.levels[i].num_iterations} for i in range(res.num_levels)]
    iters = [{"level": its[i].level, "id": its[i].id, "n": its[i].valid_constraints, "nll": its[i].tdist_log_likelihood}
             for i in range(min(n_iters, max_iters))]
    return {"T": np.array(res.transformation).reshape(4, 4), "information": np.array(res.information).reshape(6, 6),
            "log_likelihood": res.log_likelihood, "levels": levels, "iterations": iters}


def match(ref: Pyramid, cur: Pyramid, cfg, m, T_init=None, max_iters=1024):
    """oracle_py.match on this library"""
    T0 = np.ascontiguousarray(np.asarray(T_init if T_init is not None else np.eye(4), dtype=np.float64).reshape(16))
    res, its, n = orc.Result(), (orc.IterationStats * max_iters)(), C.c_int()
    assert lib().orc_match(ref.h, cur.h, C.byref(cfg), T0.ctypes.data_as(C.POINTER(C.c_double)), C.byref(m), C.byref(res), its,
                           max_iters, C.byref(n)) == 0
    return _result(res, its, n.value, max_iters)


def match_ex(ref: Pyramid, cur: Pyramid, cfg, m, predicate=PREDICATE_GRADIENT_THRESHOLD, ti=0.0, td=0.0, masks=None, T_init=None,
             max_iters=1024):
    """match() against the point lists of a predicate and optional per-level masks (one [h_l, w_l] array or None per level);
    cfg's derivative thresholds are not read."""
    T0 = np.ascontiguousarray(np.asarray(T_init if T_init is not None else np.eye(4), dtype=np.float64).reshape(16))
    res, its, n = orc.Result(), (orc.IterationStats * max_iters)(), C.c_int()
    keep, arr = [], None
    if masks is not None:
        assert len(masks) == ref.levels
        arr = (C.c_void_p * ref.levels)()
        for l, mk in enumerate(masks):
            if mk is not None:
                keep.append(_u8(mk))
                assert keep[-1].shape == ref.level_info(l)[1::-1]
                arr[l] = keep[-1].ctypes.data
    assert lib().orc_match_ex(ref.h, cur.h, C.byref(cfg), int(predicate), ti, td, arr, T0.ctypes.data_as(C.POINTER(C.c_double)),
                              C.byref(m), C.byref(res), its, max_iters, C.byref(n)) == 0
    return _result(res, its, n.value, max_iters)
