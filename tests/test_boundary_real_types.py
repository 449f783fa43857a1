"""The drop-in boundary with the REAL type spellings (SURVEY.md 8b): the adapter sources are compiled with
-DDVO_B200_WITH_EIGEN_OPENCV -- the branch a dvo_slam checkout uses -- against header-only Eigen / OpenCV / Boost
look-alikes that are spelled as the real include paths (oracle/ref_shim/, the same stand-ins that let the reference's own SSE
translation units compile for the pin).  Second test: a TUM frame loader that makes the dvo_core calls of dvo_benchmark's
loader (benchmark_slam.cpp:46-93: colour and raw depth images to an RgbdImagePyramid), together with the call sequence of
BenchmarkNode::run (benchmark_slam.cpp:384-392, 483-488), compiled against THIS repository's include/dvo headers: what
dvo_benchmark needs from dvo_core's tracking API exists with the reference's names, argument types and return types.
Nothing is executed (no GPU here)."""
import os
import shutil
import subprocess
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
STUBS = os.path.join(ROOT, "oracle", "ref_shim")
INC = os.path.join(ROOT, "include")
HOST = os.path.join(ROOT, "dvo_slam_b200", "host")
FLAGS = ["-std=c++17", "-O1", "-fPIC", "-DDVO_B200_WITH_EIGEN_OPENCV", "-I" + STUBS, "-I" + INC]


def _cxx():
    return os.environ.get("CXX") or shutil.which("g++") or "g++"


def _compile(src, obj):
    res = subprocess.run([_cxx()] + FLAGS + ["-c", src, "-o", obj], capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]


def test_adapter_compiles_with_real_type_spellings():
    lib = os.path.join(ROOT, "dvo_slam_b200", "libdvo_b200.so")
    with tempfile.TemporaryDirectory() as tmp:
        objs = {}
        for name in ("dvo_core_b200", "selftest", "tum_replay"):
            objs[name] = os.path.join(tmp, name + ".o")
            _compile(os.path.join(HOST, name + ".cpp"), objs[name])
        if os.path.exists(lib):   # the adapter + its self-test link against the C-ABI library (undefined symbols would show)
            for exe in ("selftest", "tum_replay"):
                res = subprocess.run([_cxx(), "-o", os.path.join(tmp, exe), objs[exe], objs["dvo_core_b200"], lib, "-lz", "-lpthread",
                                      "-Wl,-rpath," + os.path.dirname(lib), "-Wl,--allow-shlib-undefined"], capture_output=True, text=True)
                assert res.returncode == 0, res.stderr[-4000:]


def test_loader_and_call_site_compile_against_this_api():
    src = """
#include <string>
#include <dvo/dense_tracking.h>
#include <dvo/core/intrinsic_matrix.h>
#include <dvo/core/rgbd_image.h>
#include <dvo/core/surface_pyramid.h>

// a TUM RGB-D frame (8-bit BGR colour, 16-bit depth in 1/5000 m) through the dvo_core calls dvo_benchmark's loader makes
dvo::core::RgbdImagePyramidPtr load(dvo::core::RgbdCameraPyramid& camera, const std::string& rgb_path, const std::string& depth_path)
{
  cv::Mat bgr = cv::imread(rgb_path, 1), grey, intensity, depth;
  if(bgr.total() == 0) return dvo::core::RgbdImagePyramidPtr();
  cv::cvtColor(bgr, grey, CV_BGR2GRAY);
  grey.convertTo(intensity, CV_32F);
  dvo::core::SurfacePyramid::convertRawDepthImageSse(cv::imread(depth_path, -1), depth, 1.0f / 5000.0f);
  dvo::core::RgbdImagePyramidPtr pyramid = camera.create(intensity, depth);
  bgr.convertTo(pyramid->level(0).rgb, CV_32FC3);
  return pyramid;
}

// the calls BenchmarkNode::run makes (benchmark_slam.cpp:384-392: intrinsics and camera pyramid; :448-449: two frames;
// dvo::DenseTracker::match as LocalTracker::update reaches it, local_tracker.cpp:180-184; trajectory via Result)
int main(int argc, char** argv)
{
  dvo::core::IntrinsicMatrix intrinsics = dvo::core::IntrinsicMatrix::create(517.3, 516.5, 318.6, 255.3);
  dvo::core::RgbdCameraPyramid camera(640, 480, intrinsics);
  dvo::core::RgbdImagePyramidPtr reference = load(camera, argc > 1 ? argv[1] : "", argc > 2 ? argv[2] : "");
  dvo::core::RgbdImagePyramidPtr current = load(camera, argc > 3 ? argv[3] : "", argc > 4 ? argv[4] : "");
  if(!reference || !current) return 1;
  dvo::DenseTracker::Config cfg = dvo::DenseTracker::getDefaultConfig();
  cfg.FirstLevel = 3; cfg.LastLevel = 1; cfg.MaxIterationsPerLevel = 50; cfg.Precision = 1e-4; cfg.Mu = 0.05; cfg.UseInitialEstimate = true;
  dvo::DenseTracker tracker(cfg);
  dvo::DenseTracker::Result result;
  result.Transformation.setIdentity();
  bool ok = tracker.match(*reference, *current, result);
  dvo::core::AffineTransformd trajectory;
  trajectory.setIdentity();
  trajectory = trajectory * result.Transformation;
  Eigen::Vector3d t = trajectory.translation();
  return (ok && !result.isNaN() && t(0) == t(0) && result.Information(0, 0) >= 0 && result.LogLikelihood == result.LogLikelihood) ? 0 : 2;
}
"""
    with tempfile.TemporaryDirectory() as tmp:
        path = os.path.join(tmp, "loader.cpp")
        with open(path, "w") as f:
            f.write(src)
        _compile(path, os.path.join(tmp, "loader.o"))
