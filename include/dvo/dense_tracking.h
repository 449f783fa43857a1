// dvo/dense_tracking.h -- adapter counterpart of dvo_core/include/dvo/dense_tracking.h:39-293.
// dvo::DenseTracker with the reference's nested types and member functions; match() forwards to the
// C ABI (include/dvo_b200.h).  Config fields that never influence match() in the reference
// (UseWeighting, InfluenceFuntionType/Param, ScaleEstimatorType/Param, UseParallel; SURVEY.md Q21/Q22)
// are kept so that callers' code compiles and behaves the same.
#ifndef DVO_B200_ADAPTER_DENSE_TRACKING_H_
#define DVO_B200_ADAPTER_DENSE_TRACKING_H_
#include <iostream>
#include <string>
#include <vector>
#include "../dvo_b200.h"
#include "core/datatypes.h"
#include "core/point_selection.h"
#include "core/rgbd_image.h"

namespace dvo {
namespace core {
struct InfluenceFunctions { typedef enum { Unit, Tukey, TDistribution, Huber, NumCalculators } enum_t; };   // weight_calculation.h
struct ScaleEstimators { typedef enum { Unit, NormalDistribution, TDistribution, MAD, NumEstimators } enum_t; };
}

class DenseTracker {
 public:
  struct Config {   // dense_tracking.h:42-69, defaults dense_tracking_config.cpp:27-42
    int FirstLevel, LastLevel;
    int MaxIterationsPerLevel;
    double Precision;
    double Mu;
    bool UseInitialEstimate;
    bool UseWeighting;
    bool UseParallel;
    core::InfluenceFunctions::enum_t InfluenceFuntionType;
    float InfluenceFunctionParam;
    core::ScaleEstimators::enum_t ScaleEstimatorType;
    float ScaleEstimatorParam;
    float IntensityDerivativeThreshold;
    float DepthDerivativeThreshold;
    Config();
    size_t getNumLevels() const { return size_t(FirstLevel + 1); }
    bool UseEstimateSmoothing() const { return Mu > 1e-6; }
    bool IsSane() const { return FirstLevel >= LastLevel; }
  };

  struct TerminationCriteria {
    enum Enum { IterationsExceeded, IncrementTooSmall, LogLikelihoodDecreased, TooFewConstraints, NumCriteria };
  };

  struct IterationStats {   // dense_tracking.h:83-101
    size_t Id, ValidConstraints;
    double TDistributionLogLikelihood;
    Eigen::Vector2d TDistributionMean;
    Eigen::Matrix2d TDistributionPrecision;
    double PriorLogLikelihood;
    core::Vector6d EstimateIncrement;
    core::Matrix6d EstimateInformation;
    void InformationEigenValues(core::Vector6d& eigenvalues) const;   // ascending (dense_tracking_config.cpp:122-127)
    double InformationConditionNumber() const;                        // |ev(5) / ev(0)| (dense_tracking_config.cpp:129-135)
  };
  typedef std::vector<IterationStats> IterationStatsVector;

  struct LevelStats {   // dense_tracking.h:104-117
    size_t Id, MaxValidPixels, ValidPixels;
    TerminationCriteria::Enum TerminationCriterion;
    IterationStatsVector Iterations;
    bool HasIterationWithIncrement() const;
    IterationStats& LastIterationWithIncrement();
    IterationStats& LastIteration() { return Iterations.back(); }
    const IterationStats& LastIterationWithIncrement() const;
    const IterationStats& LastIteration() const { return Iterations.back(); }
  };
  typedef std::vector<LevelStats> LevelStatsVector;
  struct Stats { LevelStatsVector Levels; };

  struct Result {   // dense_tracking.h:125-140
    core::AffineTransformd Transformation;
    core::Matrix6d Information;
    double LogLikelihood;
    Stats Statistics;
    Result();
    bool isNaN() const;
    void setIdentity();
    void clearStatistics() { Statistics.Levels.clear(); }
  };

  static const Config& getDefaultConfig();
  DenseTracker(const Config& cfg = getDefaultConfig());
  DenseTracker(const DenseTracker& other);
  ~DenseTracker();

  const Config& configuration() const { return cfg; }
  void configure(const Config& cfg);

  bool match(core::RgbdImagePyramid& reference, core::RgbdImagePyramid& current, core::AffineTransformd& transformation);
  bool match(core::PointSelection& reference, core::RgbdImagePyramid& current, core::AffineTransformd& transformation);
  bool match(core::RgbdImagePyramid& reference, core::RgbdImagePyramid& current, Result& result);
  bool match(core::PointSelection& reference, core::RgbdImagePyramid& current, Result& result);

  // |e.i| per reference pixel at the given transform (dense_tracking.cpp:378-444)
  cv::Mat computeIntensityErrorImage(core::RgbdImagePyramid& reference, core::RgbdImagePyramid& current,
                                     const core::AffineTransformd& transformation, size_t level = 0);

  // --- extension: n independent alignments in one call (the TBB fan-outs of local_tracker.cpp:180-184
  // and keyframe_graph.cpp:587-590).  results[i].Transformation is the initial guess on entry. ---
  bool matchBatch(const std::vector<core::RgbdImagePyramid*>& references, const std::vector<core::RgbdImagePyramid*>& currents,
                  std::vector<Result>& results);
  // the same against PointSelections, each with its own predicate (match(PointSelection&, ...) for n pairs)
  bool matchBatch(const std::vector<core::PointSelection*>& references, const std::vector<core::RgbdImagePyramid*>& currents,
                  std::vector<Result>& results);

  // per-iteration statistics are copied back only when requested (they are optional in the C ABI)
  void collectIterationStatistics(bool on) { collect_iterations_ = on; }

 private:
  dvo_b200_ctx* context();
  bool usesOwnSelection(const core::PointSelection& reference) const;
  dvo_b200_selection* deviceSelection(dvo_b200_ctx* ctx, core::PointSelection& reference);
  bool runBatch(const std::vector<core::RgbdImagePyramid*>& references, const std::vector<core::PointSelection*>* selections,
                const std::vector<core::RgbdImagePyramid*>& currents, std::vector<Result>& results);
  Config cfg;
  dvo_b200_ctx* ctx_;
  bool collect_iterations_;
  core::ValidPointAndGradientThresholdPredicate selection_predicate_;
  core::PointSelection reference_selection_;
};

}  // namespace dvo

std::ostream& operator<<(std::ostream& out, const dvo::DenseTracker::Config& config);
std::ostream& operator<<(std::ostream& o, const dvo::DenseTracker::IterationStats& s);
std::ostream& operator<<(std::ostream& o, const dvo::DenseTracker::LevelStats& s);
std::ostream& operator<<(std::ostream& o, const dvo::DenseTracker::Stats& s);

#endif
