// selection_selftest.cpp -- DenseTracker::match(PointSelection&, current, result) with the selection's own predicate
// (dense_tracking.cpp:131-376), the way LocalTracker calls it (local_tracker.cpp:59-61,180-184).  Reads a raw float32 pair
// written by tests/test_gpu_selection.py and prints the poses of three alignments as JSON:
//   "own":    PointSelection with ValidPointAndGradientThresholdPredicate{0, 0} under a tracker configured with (5, 0.05)
//   "custom": PointSelection with a predicate of its own (valid point closer than 2 m), evaluated per pixel on the host
//   "plain":  match(pyramid, pyramid) of a tracker with the default configuration
// Exit 3 = no CUDA device.
#include <cstdio>
#include <cstdlib>
#include <fstream>
#include <stdexcept>
#include <string>

#include "dvo/dense_tracking.h"

namespace {
class NearPredicate : public dvo::core::PointSelectionPredicate {
 public:
  virtual bool isPointOk(const size_t&, const size_t&, const float& z, const float&, const float&, const float& zdx, const float& zdy) const {
    return z == z && zdx == zdx && zdy == zdy && z < 2.0f;
  }
};

cv::Mat load_plane(std::ifstream& f, int w, int h) {
  cv::Mat m(h, w, CV_32FC1);
  f.read(reinterpret_cast<char*>(m.ptr<float>()), sizeof(float) * size_t(w) * h);
  return m;
}

void print_pose(const char* name, const dvo::DenseTracker::Result& r, bool last) {
  std::printf("\"%s\": [", name);
  for (int i = 0; i < 16; ++i) std::printf("%.17g%s", r.Transformation.matrix()(i / 4, i % 4), i < 15 ? ", " : "");
  std::printf("]%s", last ? "" : ", ");
}
}  // namespace

int main(int argc, char** argv) {
  if (argc < 10) { std::fprintf(stderr, "usage: selection_selftest pair.bin w h fx fy ox oy first last\n"); return 2; }
  const int w = std::atoi(argv[2]), h = std::atoi(argv[3]);
  dvo::core::IntrinsicMatrix K = dvo::core::IntrinsicMatrix::create(float(std::atof(argv[4])), float(std::atof(argv[5])),
                                                                    float(std::atof(argv[6])), float(std::atof(argv[7])));
  std::ifstream f(argv[1], std::ios::binary);
  if (!f) { std::fprintf(stderr, "cannot open %s\n", argv[1]); return 2; }
  cv::Mat Ir = load_plane(f, w, h), Zr = load_plane(f, w, h), Ic = load_plane(f, w, h), Zc = load_plane(f, w, h);
  dvo::core::RgbdCameraPyramid camera(w, h, K);
  dvo::core::RgbdImagePyramidPtr reference = camera.create(Ir, Zr), current = camera.create(Ic, Zc);

  dvo::DenseTracker::Config cfg = dvo::DenseTracker::getDefaultConfig();
  cfg.FirstLevel = std::atoi(argv[8]);
  cfg.LastLevel = std::atoi(argv[9]);
  cfg.MaxIterationsPerLevel = 50;
  dvo::DenseTracker::Config thresholded = cfg;
  thresholded.IntensityDerivativeThreshold = 5.0f;
  thresholded.DepthDerivativeThreshold = 0.05f;
  try {
    dvo::DenseTracker tracker(thresholded), plain_tracker(cfg);
    dvo::core::ValidPointAndGradientThresholdPredicate zero;
    dvo::core::PointSelection own(*reference, zero);
    NearPredicate near;
    dvo::core::PointSelection custom(*reference, near);
    dvo::DenseTracker::Result r_own, r_custom, r_plain;
    tracker.match(own, *current, r_own);
    tracker.match(custom, *current, r_custom);
    tracker.match(custom, *current, r_custom);   // second call: the cached device selection
    plain_tracker.match(*reference, *current, r_plain);
    std::printf("{");
    print_pose("own", r_own, false);
    print_pose("custom", r_custom, false);
    print_pose("plain", r_plain, true);
    std::printf("}\n");
  } catch (const std::runtime_error& e) {
    std::fprintf(stderr, "%s\n", e.what());
    return 3;
  }
  return 0;
}
