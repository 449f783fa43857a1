// dvo/core/point_selection.h -- adapter counterpart of dvo_core/include/dvo/core/point_selection.h:39-124.
// The reference compacts selected reference pixels into a host point list; here selection is a
// per-level bit mask on the device: the pyramid's own for the tracker's predicate, or a device selection
// (dvo_b200_selection) that PointSelection caches for any other predicate.
#ifndef DVO_B200_ADAPTER_POINT_SELECTION_H_
#define DVO_B200_ADAPTER_POINT_SELECTION_H_
#include <cassert>
#include <cmath>
#include "rgbd_image.h"
namespace dvo { namespace core {

class PointSelectionPredicate {
 public:
  virtual ~PointSelectionPredicate() {}
  virtual bool isPointOk(const size_t& x, const size_t& y, const float& z, const float& idx, const float& idy, const float& zdx, const float& zdy) const = 0;
};

class ValidPointPredicate : public PointSelectionPredicate {   // point_selection.h:39-47
 public:
  virtual bool isPointOk(const size_t&, const size_t&, const float& z, const float&, const float&, const float& zdx, const float& zdy) const {
    return z == z && zdx == zdx && zdy == zdy;
  }
};

class ValidPointAndGradientThresholdPredicate : public PointSelectionPredicate {   // point_selection.h:52-67
 public:
  float intensity_threshold, depth_threshold;
  ValidPointAndGradientThresholdPredicate() : intensity_threshold(0.0f), depth_threshold(0.0f) {}
  virtual bool isPointOk(const size_t&, const size_t&, const float& z, const float& idx, const float& idy, const float& zdx, const float& zdy) const {
    return z == z && zdx == zdx && zdy == zdy && (std::abs(idx) > intensity_threshold || std::abs(idy) > intensity_threshold ||
                                                  std::abs(zdx) > depth_threshold || std::abs(zdy) > depth_threshold);
  }
};

class PointSelection {   // point_selection.h:69-122
 public:
  explicit PointSelection(const PointSelectionPredicate& predicate) : pyramid_(0), predicate_(predicate) {}
  PointSelection(RgbdImagePyramid& pyramid, const PointSelectionPredicate& predicate) : pyramid_(&pyramid), predicate_(predicate) {}
  PointSelection(const PointSelection& other) : pyramid_(other.pyramid_), predicate_(other.predicate_) {}   // the cache stays behind
  virtual ~PointSelection() { dropDeviceSelection(); }
  RgbdImagePyramid& getRgbdImagePyramid() { assert(pyramid_ != 0); return *pyramid_; }
  void setRgbdImagePyramid(RgbdImagePyramid& pyramid) { pyramid_ = &pyramid; dropDeviceSelection(); }
  void recycle(RgbdImagePyramid& pyramid) { setRgbdImagePyramid(pyramid); }
  size_t getMaximumNumberOfPoints(const size_t& level) {   // point_selection.cpp:68-71
    return size_t(double(pyramid_->level(0).intensity.total()) * std::pow(0.25, double(level)));
  }
  const PointSelectionPredicate& predicate() const { return predicate_; }

  // --- extension used by the adapter's DenseTracker: the device selection of this predicate on the device mirror
  // `device` of the pyramid, kept until the pyramid changes (the reference caches its point lists the same way,
  // Storage::is_cached, point_selection.cpp:51-59,100-113). ---
  dvo_b200_selection* cachedDeviceSelection(const dvo_b200_pyramid* device) const { return device_ == device ? selection_ : 0; }
  void cacheDeviceSelection(const dvo_b200_pyramid* device, dvo_b200_selection* selection) {
    dropDeviceSelection();
    device_ = device; selection_ = selection;
  }
  void dropDeviceSelection() {
    if (selection_) dvo_b200_selection_release(selection_);
    selection_ = 0; device_ = 0;
  }
 private:
  RgbdImagePyramid* pyramid_;
  const PointSelectionPredicate& predicate_;
  const dvo_b200_pyramid* device_ = 0;
  dvo_b200_selection* selection_ = 0;
};
} }
#endif
