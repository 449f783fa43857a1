// dvo_slam/batched_alignment.h -- the two places dvo_slam fans independent DenseTracker::match() calls out,
// restated as ONE batched call on the B200 engine (SURVEY.md 8f row N1):
//
//   * LocalTracker::update (dvo_slam/src/local_tracker.cpp:155-184): the new frame is aligned against the
//     keyframe and against the previous frame with tbb::parallel_invoke -- two alignments sharing `current`;
//   * ConstraintProposalValidator::validate (dvo_slam/src/constraints/constraint_proposal_validator.cpp:133-146):
//     a loop of tracker_.match() over loop-closure proposals, each keyframe appearing in several proposals.
//
// Both become DenseTracker::matchBatch: every pyramid is uploaded / built once (a keyframe that appears in four
// proposals is one device pyramid), and the alignments run as one batch.  Header-only; the callers keep their
// own types (the proposal type is a template parameter).
#ifndef DVO_SLAM_BATCHED_ALIGNMENT_H_
#define DVO_SLAM_BATCHED_ALIGNMENT_H_

#include <vector>

#include "dvo/dense_tracking.h"

namespace dvo_slam {

// The two alignments of LocalTracker::update.  r_keyframe.Transformation / r_odometry.Transformation carry the
// initial guesses on entry exactly as in local_tracker.cpp:165-167 (inverse of the last keyframe pose, identity).
// Both trackers of the reference are configured identically (LocalTracker::configure, local_tracker.cpp:100-104),
// so one tracker object serves both.
inline bool matchKeyframeAndOdometry(dvo::DenseTracker& tracker, dvo::core::RgbdImagePyramid& keyframe,
                                     dvo::core::RgbdImagePyramid& previous_frame, dvo::core::RgbdImagePyramid& current,
                                     dvo::DenseTracker::Result& r_keyframe, dvo::DenseTracker::Result& r_odometry) {
  std::vector<dvo::core::RgbdImagePyramid*> references, currents;
  references.push_back(&keyframe); references.push_back(&previous_frame);
  currents.push_back(&current); currents.push_back(&current);
  std::vector<dvo::DenseTracker::Result> results(2);
  results[0].Transformation = r_keyframe.Transformation;
  results[1].Transformation = r_odometry.Transformation;
  const bool ok = tracker.matchBatch(references, currents, results);
  r_keyframe = results[0];
  r_odometry = results[1];
  return ok;
}

// The same with the reference points of LocalTracker's own PointSelections (local_tracker.cpp:59-61,180-184: the keyframe's
// and the previous frame's selection, each with the tracker's predicate), so that their predicate reaches the device.
inline bool matchKeyframeAndOdometry(dvo::DenseTracker& tracker, dvo::core::PointSelection& keyframe,
                                     dvo::core::PointSelection& previous_frame, dvo::core::RgbdImagePyramid& current,
                                     dvo::DenseTracker::Result& r_keyframe, dvo::DenseTracker::Result& r_odometry) {
  std::vector<dvo::core::PointSelection*> references;
  std::vector<dvo::core::RgbdImagePyramid*> currents;
  references.push_back(&keyframe); references.push_back(&previous_frame);
  currents.push_back(&current); currents.push_back(&current);
  std::vector<dvo::DenseTracker::Result> results(2);
  results[0].Transformation = r_keyframe.Transformation;
  results[1].Transformation = r_odometry.Transformation;
  const bool ok = tracker.matchBatch(references, currents, results);
  r_keyframe = results[0];
  r_odometry = results[1];
  return ok;
}

// The tracking loop of ConstraintProposalValidator::validate.  ProposalPtrVector is any sequence of pointer-likes
// to objects with the members the reference's ConstraintProposal has: Reference->image(), Current->image()
// (RgbdImagePyramid::Ptr), InitialTransformation and TrackingResult (constraint_proposal.h).
template <typename ProposalPtrVector>
inline bool matchProposals(dvo::DenseTracker& tracker, ProposalPtrVector& proposals) {
  std::vector<dvo::core::RgbdImagePyramid*> references, currents;
  std::vector<dvo::DenseTracker::Result> results(proposals.size());
  size_t i = 0;
  for (typename ProposalPtrVector::iterator it = proposals.begin(); it != proposals.end(); ++it, ++i) {
    references.push_back(&*(*it)->Reference->image());
    currents.push_back(&*(*it)->Current->image());
    results[i].Transformation = (*it)->InitialTransformation;     // constraint_proposal_validator.cpp:144
  }
  if (proposals.empty()) return true;
  const bool ok = tracker.matchBatch(references, currents, results);
  i = 0;
  for (typename ProposalPtrVector::iterator it = proposals.begin(); it != proposals.end(); ++it, ++i) (*it)->TrackingResult = results[i];
  return ok;
}

}  // namespace dvo_slam

#endif
