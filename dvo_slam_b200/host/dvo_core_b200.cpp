// dvo_core_b200.cpp -- implementation of the adapter classes in include/dvo/ (the reference's
// libdvo_core.so surface for the hot path) on top of the C ABI of libdvo_b200.so.
#include <algorithm>
#include <cassert>
#include <cmath>
#include <cstring>
#include <cstdlib>
#include <stdexcept>

#include "dvo/dense_tracking.h"

namespace dvo {
namespace core {

// ---- cameras (rgbd_image.cpp:186-296) -------------------------------------------------------------
RgbdImagePtr RgbdCamera::create(const cv::Mat& intensity, const cv::Mat& depth) const {
  RgbdImagePtr r(new RgbdImage(*this));
  r->intensity = intensity;
  r->depth = depth;
  r->initialize();
  return r;
}
RgbdImagePtr RgbdCamera::create() const { return RgbdImagePtr(new RgbdImage(*this)); }

RgbdCameraPyramid::RgbdCameraPyramid(const RgbdCamera& base) { levels_.push_back(RgbdCameraPtr(new RgbdCamera(base))); }
RgbdCameraPyramid::RgbdCameraPyramid(size_t w, size_t h, const IntrinsicMatrix& k) { levels_.push_back(RgbdCameraPtr(new RgbdCamera(w, h, k))); }
RgbdImagePyramidPtr RgbdCameraPyramid::create(const cv::Mat& base_intensity, const cv::Mat& base_depth) {
  return RgbdImagePyramidPtr(new RgbdImagePyramid(*this, base_intensity, base_depth));
}
void RgbdCameraPyramid::build(size_t levels) {   // rgbd_image.cpp:283-296: whole K times 0.5 per level
  for (size_t idx = levels_.size(); idx < levels; ++idx) {
    const RgbdCamera& prev = *levels_[idx - 1];
    IntrinsicMatrix k(prev.intrinsics());
    k.scale(0.5f);
    levels_.push_back(RgbdCameraPtr(new RgbdCamera(prev.width() / 2, prev.height() / 2, k)));
  }
}
const RgbdCamera& RgbdCameraPyramid::level(size_t level) { build(level + 1); return *levels_[level]; }
const RgbdCamera& RgbdCameraPyramid::level(size_t level) const { return *levels_[level]; }

// ---- image pyramid ----------------------------------------------------------------------------------
RgbdImagePyramid::RgbdImagePyramid(RgbdCameraPyramid& camera, const cv::Mat& intensity, const cv::Mat& depth)
    : camera_(camera), device_(0), device_ctx_(0), device_levels_(0), requested_levels_(1) {
  levels_.push_back(camera_.level(0).create(intensity, depth));
}
RgbdImagePyramid::~RgbdImagePyramid() {
  if (device_) dvo_b200_pyramid_release(device_);
}
void RgbdImagePyramid::build(const size_t num_levels) {
  // Coarser levels are produced on the device together with their derivatives (rgbd_image.cpp:156-172);
  // here only the request is recorded, host copies of a level are fetched on demand by level().
  if (num_levels > requested_levels_) requested_levels_ = num_levels;
  camera_.build(num_levels);
}
double RgbdImagePyramid::timestamp() const { return !levels_.empty() ? levels_[0]->timestamp : 0.0; }

dvo_b200_pyramid* RgbdImagePyramid::device(dvo_b200_ctx* ctx, size_t levels) {
  std::lock_guard<std::mutex> lock(mutex_);
  if (levels < requested_levels_) levels = requested_levels_;
  if (device_ && device_levels_ >= levels) return device_;
  if (device_) { dvo_b200_pyramid_release(device_); device_ = 0; }
  RgbdImage& l0 = *levels_[0];
  if (l0.intensity.type() != CV_32FC1 || l0.depth.type() != CV_32FC1)
    throw std::runtime_error("RgbdImagePyramid: intensity and depth must be CV_32FC1 (benchmark_slam.cpp:60-77)");
  const IntrinsicMatrix& k = camera_.level(0).intrinsics();
  int rc = dvo_b200_pyramid_create(ctx, l0.intensity.ptr<float>(), l0.depth.ptr<float>(), l0.intensity.cols, l0.intensity.rows,
                                   k.fx(), k.fy(), k.ox(), k.oy(), int(levels), &device_);
  if (rc != 0) throw std::runtime_error(std::string("dvo_b200_pyramid_create: ") + dvo_b200_last_error(ctx));
  dvo_b200_synchronize(ctx);   // the host cv::Mat may be released by the caller
  device_ctx_ = ctx;
  device_levels_ = levels;
  return device_;
}

void RgbdImagePyramid::deviceBatch(dvo_b200_ctx* ctx, const std::vector<RgbdImagePyramid*>& pyramids, size_t levels,
                                   std::vector<dvo_b200_pyramid*>& out) {
  out.assign(pyramids.size(), static_cast<dvo_b200_pyramid*>(0));
  // distinct pyramids without a sufficient device mirror, of the geometry of the first such pyramid
  std::vector<RgbdImagePyramid*> todo;
  int w = 0, h = 0;
  for (size_t i = 0; i < pyramids.size(); ++i) {
    RgbdImagePyramid* p = pyramids[i];
    std::lock_guard<std::mutex> lock(p->mutex_);
    if (p->device_ && p->device_levels_ >= std::max(levels, p->requested_levels_)) continue;
    if (std::find(todo.begin(), todo.end(), p) != todo.end()) continue;
    const RgbdImage& l0 = *p->levels_[0];
    if (l0.intensity.type() != CV_32FC1 || l0.depth.type() != CV_32FC1) continue;
    if (todo.empty()) { w = l0.intensity.cols; h = l0.intensity.rows; }
    else if (l0.intensity.cols != w || l0.intensity.rows != h || &p->camera_ != &todo[0]->camera_) continue;
    todo.push_back(p);
  }
  if (todo.size() >= 2) {
    const size_t npx = size_t(w) * h, n = todo.size();
    size_t lv = levels;
    for (size_t i = 0; i < n; ++i) lv = std::max(lv, todo[i]->requested_levels_);
    std::vector<float> I(n * npx), Z(n * npx);
    for (size_t i = 0; i < n; ++i) {
      for (int y = 0; y < h; ++y) {   // row by row: a cv::Mat need not be continuous
        std::memcpy(&I[i * npx + size_t(y) * w], todo[i]->levels_[0]->intensity.ptr<float>(y), sizeof(float) * w);
        std::memcpy(&Z[i * npx + size_t(y) * w], todo[i]->levels_[0]->depth.ptr<float>(y), sizeof(float) * w);
      }
    }
    const IntrinsicMatrix& k = todo[0]->camera_.level(0).intrinsics();
    std::vector<dvo_b200_pyramid*> handles(n);
    int rc = dvo_b200_pyramid_create_batch(ctx, int(n), I.data(), Z.data(), w, h, k.fx(), k.fy(), k.ox(), k.oy(), int(lv), handles.data());
    if (rc != 0) throw std::runtime_error(std::string("dvo_b200_pyramid_create_batch: ") + dvo_b200_last_error(ctx));
    dvo_b200_synchronize(ctx);   // one synchronisation for the whole upload: the staging vectors go out of scope
    for (size_t i = 0; i < n; ++i) {
      std::lock_guard<std::mutex> lock(todo[i]->mutex_);
      if (todo[i]->device_) dvo_b200_pyramid_release(todo[i]->device_);
      todo[i]->device_ = handles[i];
      todo[i]->device_ctx_ = ctx;
      todo[i]->device_levels_ = lv;
    }
  }
  for (size_t i = 0; i < pyramids.size(); ++i) out[i] = pyramids[i]->device(ctx, levels);   // the rest one by one
}

RgbdImage& RgbdImagePyramid::level(size_t idx) {
  if (idx < levels_.size() && (idx == 0 || levels_[idx]->hasIntensity())) return *levels_[idx];
  if (!device_ || device_levels_ <= idx)
    throw std::runtime_error("RgbdImagePyramid::level: level not built (call build/compute and match first)");
  while (levels_.size() <= idx) levels_.push_back(camera_.level(levels_.size()).create());
  int w = 0, h = 0;
  float K[4];
  dvo_b200_pyramid_level_info(device_, int(idx), &w, &h, K);
  std::vector<float> planes(size_t(6) * w * h);
  // no context: the pyramid may be read after the tracker (and context) that uploaded it is gone
  if (dvo_b200_pyramid_download(nullptr, device_, int(idx), planes.data()) != 0)
    throw std::runtime_error("dvo_b200_pyramid_download failed");
  RgbdImage& img = *levels_[idx];
  cv::Mat* dst[6] = {&img.intensity, &img.depth, &img.intensity_dx, &img.intensity_dy, &img.depth_dx, &img.depth_dy};
  for (int c = 0; c < 6; ++c) {
    dst[c]->create(h, w, CV_32FC1);
    std::memcpy(dst[c]->ptr<float>(), planes.data() + size_t(c) * w * h, sizeof(float) * w * h);
  }
  return img;
}

}  // namespace core

// ---- DenseTracker -------------------------------------------------------------------------------------
DenseTracker::Config::Config()   // dense_tracking_config.cpp:27-42
    : FirstLevel(3), LastLevel(1), MaxIterationsPerLevel(100), Precision(5e-7), Mu(0), UseInitialEstimate(false),
      UseWeighting(true), UseParallel(false), InfluenceFuntionType(core::InfluenceFunctions::TDistribution),
      InfluenceFunctionParam(5.0f), ScaleEstimatorType(core::ScaleEstimators::TDistribution), ScaleEstimatorParam(5.0f),
      IntensityDerivativeThreshold(0.0f), DepthDerivativeThreshold(0.0f) {}

const DenseTracker::Config& DenseTracker::getDefaultConfig() {
  static Config c;
  return c;
}

DenseTracker::DenseTracker(const Config& config) : ctx_(0), collect_iterations_(false), reference_selection_(selection_predicate_) { configure(config); }
DenseTracker::DenseTracker(const DenseTracker& other) : ctx_(0), collect_iterations_(other.collect_iterations_), reference_selection_(selection_predicate_) {
  configure(other.configuration());
}
DenseTracker::~DenseTracker() {
  if (ctx_) dvo_b200_destroy(ctx_);
}

void DenseTracker::configure(const Config& config) {   // dense_tracking.cpp:72-97
  assert(config.IsSane());
  cfg = config;
  selection_predicate_.intensity_threshold = cfg.IntensityDerivativeThreshold;
  selection_predicate_.depth_threshold = cfg.DepthDerivativeThreshold;
}

dvo_b200_ctx* DenseTracker::context() {
  if (!ctx_) {
    const char* dev = std::getenv("DVO_B200_DEVICE");
    int rc = dvo_b200_create(dev ? std::atoi(dev) : 0, 0, &ctx_);
    if (rc != 0) throw std::runtime_error("dvo_b200_create failed: no usable CUDA device (the engine has no CPU fallback)");
  }
  return ctx_;
}

DenseTracker::Result::Result() : LogLikelihood(std::numeric_limits<double>::max()) {   // dense_tracking_config.cpp:101-108
  double nan = std::numeric_limits<double>::quiet_NaN();
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 4; ++j) Transformation.matrix()(i, j) = nan;
  Information.setIdentity();
}
bool DenseTracker::Result::isNaN() const {   // dense_tracking_config.cpp:96-99
  return !std::isfinite(Transformation.matrix().sum()) || !std::isfinite(Information.sum());
}
void DenseTracker::Result::setIdentity() {
  Transformation.setIdentity();
  Information.setIdentity();
  LogLikelihood = 0.0;
}

// dense_tracking_config.cpp:122-135.  EstimateInformation = A + mu*I is symmetric, so the real parts the reference takes from
// Eigen::EigenSolver are the eigenvalues of a symmetric matrix: cyclic Jacobi rotations on a copy, sorted ascending.
void DenseTracker::IterationStats::InformationEigenValues(core::Vector6d& eigenvalues) const {
  double a[6][6];
  for (int i = 0; i < 6; ++i) for (int j = 0; j < 6; ++j) a[i][j] = 0.5 * (EstimateInformation(i, j) + EstimateInformation(j, i));
  for (int sweep = 0; sweep < 64; ++sweep) {
    double off = 0.0, diag = 0.0;
    for (int i = 0; i < 6; ++i) { diag += a[i][i] * a[i][i]; for (int j = i + 1; j < 6; ++j) off += a[i][j] * a[i][j]; }
    if (!(off > 1e-32 * diag)) break;
    for (int p = 0; p < 5; ++p)
      for (int q = p + 1; q < 6; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = (theta >= 0 ? 1.0 : -1.0) / (std::fabs(theta) + std::sqrt(theta * theta + 1.0));
        const double cs = 1.0 / std::sqrt(t * t + 1.0), sn = t * cs;
        for (int k = 0; k < 6; ++k) { const double x = a[k][p], y = a[k][q]; a[k][p] = cs * x - sn * y; a[k][q] = sn * x + cs * y; }
        for (int k = 0; k < 6; ++k) { const double x = a[p][k], y = a[q][k]; a[p][k] = cs * x - sn * y; a[q][k] = sn * x + cs * y; }
      }
  }
  double ev[6];
  for (int i = 0; i < 6; ++i) ev[i] = a[i][i];
  std::sort(ev, ev + 6);
  for (int i = 0; i < 6; ++i) eigenvalues(i) = ev[i];
}

double DenseTracker::IterationStats::InformationConditionNumber() const {
  core::Vector6d ev;
  InformationEigenValues(ev);
  return std::abs(ev(5) / ev(0));
}

bool DenseTracker::LevelStats::HasIterationWithIncrement() const {   // dense_tracking_config.cpp:138-143
  int min = TerminationCriterion == TerminationCriteria::LogLikelihoodDecreased || TerminationCriterion == TerminationCriteria::TooFewConstraints ? 2 : 1;
  return int(Iterations.size()) >= min;
}
DenseTracker::IterationStats& DenseTracker::LevelStats::LastIterationWithIncrement() {
  assert(HasIterationWithIncrement());
  return TerminationCriterion == TerminationCriteria::LogLikelihoodDecreased ? Iterations[Iterations.size() - 2] : Iterations[Iterations.size() - 1];
}
const DenseTracker::IterationStats& DenseTracker::LevelStats::LastIterationWithIncrement() const {
  assert(HasIterationWithIncrement());
  return TerminationCriterion == TerminationCriteria::LogLikelihoodDecreased ? Iterations[Iterations.size() - 2] : Iterations[Iterations.size() - 1];
}

bool DenseTracker::match(core::RgbdImagePyramid& reference, core::RgbdImagePyramid& current, core::AffineTransformd& transformation) {
  Result result;
  result.Transformation = transformation;
  bool ok = match(reference, current, result);
  transformation = result.Transformation;
  return ok;
}
bool DenseTracker::match(core::PointSelection& reference, core::RgbdImagePyramid& current, core::AffineTransformd& transformation) {
  Result result;
  result.Transformation = transformation;
  bool ok = match(reference, current, result);
  transformation = result.Transformation;
  return ok;
}
bool DenseTracker::match(core::RgbdImagePyramid& reference, core::RgbdImagePyramid& current, Result& result) {   // dense_tracking.cpp:123-129
  reference.compute(cfg.getNumLevels());
  reference_selection_.setRgbdImagePyramid(reference);
  return match(reference_selection_, current, result);
}
bool DenseTracker::match(core::PointSelection& reference, core::RgbdImagePyramid& current, Result& result) {
  std::vector<core::PointSelection*> refs(1, &reference);
  std::vector<core::RgbdImagePyramid*> curs(1, &current);
  std::vector<Result> results(1, result);
  bool ok = matchBatch(refs, curs, results);
  result = results[0];
  return ok;
}

// The tracker's own selection, or a gradient-threshold predicate with the configured thresholds: the pyramid's built-in
// selection is exactly that (every call of dvo_slam).  Anything else gets a device selection of its own.
bool DenseTracker::usesOwnSelection(const core::PointSelection& reference) const {
  if (&reference == &reference_selection_) return true;
  const core::ValidPointAndGradientThresholdPredicate* g =
      dynamic_cast<const core::ValidPointAndGradientThresholdPredicate*>(&reference.predicate());
  return g && g->intensity_threshold == cfg.IntensityDerivativeThreshold && g->depth_threshold == cfg.DepthDerivativeThreshold;
}

// PointSelection::select with the selection's own predicate (point_selection.cpp:89-152), as a device selection cached in
// the PointSelection.  The two predicates of the reference map to their device forms; any other predicate is evaluated
// here on every level -- isPointOk(x, y, z, idx, idy, zdx, zdy) with z the true depth of the level (the level-0 depth
// subsampled) and the gradients of the device pyramid -- and handed over as MASK_ONLY masks.
dvo_b200_selection* DenseTracker::deviceSelection(dvo_b200_ctx* ctx, core::PointSelection& reference) {
  core::RgbdImagePyramid& pyr = reference.getRgbdImagePyramid();
  dvo_b200_pyramid* p = pyr.device(ctx, cfg.getNumLevels());
  if (dvo_b200_selection* s = reference.cachedDeviceSelection(p)) return s;
  const core::PointSelectionPredicate& pred = reference.predicate();
  const core::ValidPointAndGradientThresholdPredicate* g = dynamic_cast<const core::ValidPointAndGradientThresholdPredicate*>(&pred);
  dvo_b200_selection* s = 0;
  int rc;
  if (g)
    rc = dvo_b200_selection_create(ctx, p, DVO_B200_PREDICATE_GRADIENT_THRESHOLD, g->intensity_threshold, g->depth_threshold, 0, &s);
  else if (dynamic_cast<const core::ValidPointPredicate*>(&pred))
    rc = dvo_b200_selection_create(ctx, p, DVO_B200_PREDICATE_VALID_POINT, 0.f, 0.f, 0, &s);
  else {
    const int levels = dvo_b200_pyramid_num_levels(p);
    const cv::Mat& depth0 = pyr.level(0).depth;
    std::vector<std::vector<uint8_t> > masks(static_cast<size_t>(levels));
    std::vector<const uint8_t*> ptrs(static_cast<size_t>(levels));
    for (int l = 0; l < levels; ++l) {
      int w = 0, h = 0;
      float K[4];
      dvo_b200_pyramid_level_info(p, l, &w, &h, K);
      const size_t N = size_t(w) * h;
      std::vector<float> planes(6 * N);
      rc = dvo_b200_pyramid_download(ctx, p, l, planes.data());
      if (rc != 0) throw std::runtime_error(std::string("dvo_b200_pyramid_download: ") + dvo_b200_last_error(ctx));
      std::vector<uint8_t>& m = masks[size_t(l)];
      m.resize(N);
      for (int y = 0; y < h; ++y)
        for (int x = 0; x < w; ++x) {
          const size_t i = size_t(y) * w + x;
          const float z = depth0.at<float>(y << l, x << l);
          m[i] = pred.isPointOk(size_t(x), size_t(y), z, planes[2 * N + i], planes[3 * N + i], planes[4 * N + i], planes[5 * N + i]) ? 1 : 0;
        }
      ptrs[size_t(l)] = m.data();
    }
    rc = dvo_b200_selection_create(ctx, p, DVO_B200_PREDICATE_MASK_ONLY, 0.f, 0.f, ptrs.data(), &s);
  }
  if (rc != 0) throw std::runtime_error(std::string("dvo_b200_selection_create: ") + dvo_b200_last_error(ctx));
  reference.cacheDeviceSelection(p, s);
  return s;
}

bool DenseTracker::matchBatch(const std::vector<core::PointSelection*>& references, const std::vector<core::RgbdImagePyramid*>& currents,
                              std::vector<Result>& results) {
  std::vector<core::RgbdImagePyramid*> pyrs(references.size());
  bool own = true;
  for (size_t i = 0; i < references.size(); ++i) {
    pyrs[i] = &references[i]->getRgbdImagePyramid();
    own = own && usesOwnSelection(*references[i]);
  }
  return runBatch(pyrs, own ? 0 : &references, currents, results);
}

static void fill_result(const dvo_b200_result& r, const dvo_b200_iteration_stats* its, DenseTracker::Result& out) {
  for (int i = 0; i < 4; ++i)
    for (int j = 0; j < 4; ++j) out.Transformation.matrix()(i, j) = r.transformation[i * 4 + j];
  for (int i = 0; i < 6; ++i)
    for (int j = 0; j < 6; ++j) out.Information(i, j) = r.information[i * 6 + j];
  out.LogLikelihood = r.log_likelihood;
  int cursor = 0;
  for (int l = 0; l < r.num_levels; ++l) {   // match() appends to Statistics.Levels (dense_tracking.cpp:202)
    const dvo_b200_level_stats& ls = r.levels[l];
    DenseTracker::LevelStats s;
    s.Id = size_t(ls.id); s.MaxValidPixels = size_t(ls.max_valid_pixels); s.ValidPixels = size_t(ls.valid_pixels);
    s.TerminationCriterion = DenseTracker::TerminationCriteria::Enum(ls.termination);
    s.Iterations.resize(size_t(ls.num_iterations));
    for (int k = 0; k < ls.num_iterations; ++k) {
      DenseTracker::IterationStats& it = s.Iterations[size_t(k)];
      it.Id = size_t(k); it.ValidConstraints = 0; it.TDistributionLogLikelihood = 0; it.PriorLogLikelihood = 0;
      if (its) {
        const dvo_b200_iteration_stats& q = its[cursor + k];
        it.ValidConstraints = size_t(q.valid_constraints);
        it.TDistributionLogLikelihood = q.tdist_log_likelihood;
        it.PriorLogLikelihood = q.prior_log_likelihood;
        for (int a = 0; a < 2; ++a) for (int b = 0; b < 2; ++b) it.TDistributionPrecision(a, b) = q.tdist_precision[a * 2 + b];
        for (int a = 0; a < 6; ++a) it.EstimateIncrement(a) = q.increment[a];
        for (int a = 0; a < 6; ++a) for (int b = 0; b < 6; ++b) it.EstimateInformation(a, b) = q.information[a * 6 + b];
      }
    }
    // without the optional per-iteration log the fields the callers read are still filled
    // (keyframe_tracker.cpp:167, constraint_proposal_voter.cpp:128-129)
    if (!its && ls.num_iterations > 0) {
      s.Iterations.back().ValidConstraints = size_t(ls.last_valid_constraints);
      if (ls.has_iteration_with_increment) {
        DenseTracker::IterationStats& li = s.LastIterationWithIncrement();
        li.ValidConstraints = size_t(ls.last_increment_valid_constraints);
        li.TDistributionLogLikelihood = ls.last_increment_log_likelihood;
      }
    }
    cursor += ls.num_iterations;
    out.Statistics.Levels.push_back(s);
  }
}

bool DenseTracker::matchBatch(const std::vector<core::RgbdImagePyramid*>& references, const std::vector<core::RgbdImagePyramid*>& currents,
                              std::vector<Result>& results) {
  return runBatch(references, 0, currents, results);
}

// selections == 0: every pair against its reference pyramid's built-in selection (cfg's thresholds); else pair i against
// the device selection of (*selections)[i]
bool DenseTracker::runBatch(const std::vector<core::RgbdImagePyramid*>& references, const std::vector<core::PointSelection*>* selections,
                            const std::vector<core::RgbdImagePyramid*>& currents, std::vector<Result>& results) {
  const size_t n = references.size();
  if (n == 0 || currents.size() != n) return false;
  results.resize(n);
  dvo_b200_ctx* ctx = context();
  dvo_b200_config c;
  dvo_b200_config_default(&c);
  c.first_level = cfg.FirstLevel; c.last_level = cfg.LastLevel; c.max_iterations_per_level = cfg.MaxIterationsPerLevel;
  c.use_initial_estimate = cfg.UseInitialEstimate ? 1 : 0; c.precision = cfg.Precision; c.mu = cfg.Mu;
  c.intensity_derivative_threshold = cfg.IntensityDerivativeThreshold; c.depth_derivative_threshold = cfg.DepthDerivativeThreshold;
  std::vector<dvo_b200_pyramid*> r(n), q(n);
  std::vector<double> T(16 * n);
  {
    std::vector<core::RgbdImagePyramid*> all(references);
    all.insert(all.end(), currents.begin(), currents.end());
    for (size_t i = 0; i < all.size(); ++i) all[i]->compute(cfg.getNumLevels());   // dense_tracking.cpp:133
    std::vector<dvo_b200_pyramid*> dev;
    core::RgbdImagePyramid::deviceBatch(ctx, all, cfg.getNumLevels(), dev);        // one upload, one synchronisation
    for (size_t i = 0; i < n; ++i) { r[i] = dev[i]; q[i] = dev[n + i]; }
  }
  for (size_t i = 0; i < n; ++i) {
    if (cfg.UseInitialEstimate) assert(!results[i].isNaN() && "Provided initialization is NaN!");
    for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) T[16 * i + a * 4 + b] = results[i].Transformation.matrix()(a, b);
  }
  std::vector<dvo_b200_result> raw(n);
  const int max_log = collect_iterations_ ? (cfg.FirstLevel - cfg.LastLevel + 1) * (cfg.MaxIterationsPerLevel + 1) : 0;
  std::vector<dvo_b200_iteration_stats> log(size_t(max_log) * n);
  int rc;
  if (selections) {   // match(PointSelection&, ...): the selection's predicate decides, not cfg's thresholds
    std::vector<dvo_b200_selection*> sel(n);
    for (size_t i = 0; i < n; ++i) sel[i] = deviceSelection(ctx, *(*selections)[i]);
    rc = dvo_b200_match_batch_selected(ctx, &c, int(n), sel.data(), q.data(), cfg.UseInitialEstimate ? T.data() : 0, raw.data(),
                                       max_log ? log.data() : 0, max_log);
  } else {
    rc = dvo_b200_match_batch(ctx, &c, int(n), r.data(), q.data(), cfg.UseInitialEstimate ? T.data() : 0, raw.data(),
                              max_log ? log.data() : 0, max_log);
  }
  if (rc != 0) throw std::runtime_error(std::string("dvo_b200_match_batch: ") + dvo_b200_last_error(ctx));
  for (size_t i = 0; i < n; ++i) fill_result(raw[i], max_log ? &log[size_t(max_log) * i] : 0, results[i]);
  return true;   // the reference's match() always returns true (dense_tracking.cpp:135,375)
}

cv::Mat DenseTracker::computeIntensityErrorImage(core::RgbdImagePyramid& reference, core::RgbdImagePyramid& current,
                                                 const core::AffineTransformd& transformation, size_t level) {
  dvo_b200_ctx* ctx = context();
  reference.compute(level + 1);
  current.compute(level + 1);
  dvo_b200_pyramid* r = reference.device(ctx, level + 1);
  dvo_b200_pyramid* q = current.device(ctx, level + 1);
  int w = 0, h = 0;
  float K[4];
  dvo_b200_pyramid_level_info(r, int(level), &w, &h, K);
  double T[16];
  for (int a = 0; a < 4; ++a) for (int b = 0; b < 4; ++b) T[a * 4 + b] = transformation.matrix()(a, b);
  dvo_b200_config c;
  dvo_b200_config_default(&c);
  c.intensity_derivative_threshold = cfg.IntensityDerivativeThreshold; c.depth_derivative_threshold = cfg.DepthDerivativeThreshold;
  cv::Mat result = cv::Mat::zeros(h, w, CV_32FC1);
  if (dvo_b200_intensity_error_image(ctx, &c, r, q, int(level), T, result.ptr<float>(), nullptr) != 0)
    throw std::runtime_error(std::string("dvo_b200_intensity_error_image: ") + dvo_b200_last_error(ctx));
  return result;
}

}  // namespace dvo

std::ostream& operator<<(std::ostream& out, const dvo::DenseTracker::Config& c) {
  return out << "First Level = " << c.FirstLevel << ", Last Level = " << c.LastLevel << ", Max Iterations per Level = " << c.MaxIterationsPerLevel
             << ", Precision = " << c.Precision << ", Mu = " << c.Mu << ", Use Initial Estimate = " << (c.UseInitialEstimate ? "true" : "false")
             << ", Use Weighting = " << (c.UseWeighting ? "true" : "false") << ", Intensity Derivative Threshold = " << c.IntensityDerivativeThreshold
             << ", Depth Derivative Threshold = " << c.DepthDerivativeThreshold;
}
std::ostream& operator<<(std::ostream& o, const dvo::DenseTracker::IterationStats& s) {
  return o << "Iteration: " << s.Id << " ValidConstraints: " << s.ValidConstraints << " DataLogLikelihood: " << s.TDistributionLogLikelihood
           << " PriorLogLikelihood: " << s.PriorLogLikelihood << std::endl;
}
std::ostream& operator<<(std::ostream& o, const dvo::DenseTracker::LevelStats& s) {
  static const char* names[] = {"IterationsExceeded", "IncrementTooSmall", "LogLikelihoodDecreased", "TooFewConstraints"};
  int t = int(s.TerminationCriterion);
  o << "Level: " << s.Id << " Pixel: " << s.ValidPixels << "/" << s.MaxValidPixels << " Termination: " << (t >= 0 && t < 4 ? names[t] : "")
    << " Iterations: " << s.Iterations.size() << std::endl;
  for (size_t i = 0; i < s.Iterations.size(); ++i) o << s.Iterations[i];
  return o;
}
std::ostream& operator<<(std::ostream& o, const dvo::DenseTracker::Stats& s) {
  o << s.Levels.size() << " levels" << std::endl;
  for (size_t i = 0; i < s.Levels.size(); ++i) o << s.Levels[i];
  return o;
}
