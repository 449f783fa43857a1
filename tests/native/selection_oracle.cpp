// selection_oracle.cpp -- the CPU oracle (oracle/dvo_oracle.cpp, included unchanged) with reference point selections
// that carry their own predicate and an optional per-pixel mask: PointSelection(pyramid, predicate) +
// DenseTracker::match(PointSelection&, current, result) (point_selection.h:39-67, point_selection.cpp:89-152,
// dense_tracking.cpp:131-376).  Test infrastructure: compiled by tests/selection_oracle.py with the oracle's own flags, so
// its arithmetic is the oracle's, bit for bit.
//
// Predicates (= dvo_b200_predicate): 0 GRADIENT_THRESHOLD(ti, td) = ValidPointAndGradientThresholdPredicate, 1 VALID_POINT =
// ValidPointPredicate (z, zdx, zdy not NaN), 2 MASK_ONLY = every pixel the mask allows; a MASK_ONLY point whose six channels
// are not all valid counts in S and never projects (the reference's point list with a NaN-depth point).
#include "dvo_oracle.cpp"

namespace {

// PointSelection::selectPointsFromImage (point_selection.cpp:119-152) with any of the three predicates, ANDed with `mask`
// (h*w bytes, nonzero = allowed; NULL = no mask): sel[p] = 1 for the points of the list, in raster order as the reference
// lists them; returns S.
int64_t select_mask(const Level& L, int predicate, float ti, float td, const uint8_t* mask, std::vector<uint8_t>& sel) {
  const size_t N = size_t(L.w) * L.h;
  sel.assign(N, 0);
  int64_t S = 0;
  for (size_t p = 0; p < N; ++p) {
    const float z = L.ch[1][p], idx = L.ch[2][p], idy = L.ch[3][p], zdx = L.ch[4][p], zdy = L.ch[5][p];
    const bool valid = z == z && zdx == zdx && zdy == zdy;
    bool ok;
    if (predicate == 1) ok = valid;
    else if (predicate == 2) ok = true;
    else ok = valid && (std::fabs(idx) > ti || std::fabs(idy) > ti || std::fabs(zdx) > td || std::fabs(zdy) > td);
    if (mask && !mask[p]) ok = false;
    sel[p] = ok ? 1 : 0;
    S += ok ? 1 : 0;
  }
  return S;
}

}  // namespace

extern "C" {

// orc_select with a predicate and a mask of this level: S, and (optional) the h*w byte mask of the list (the odd last
// point dropped iff mode->drop_odd_point, as orc_select reports it).
int64_t orc_select_ex(const orc_pyramid* ref, int level, int predicate, float ti, float td, const uint8_t* level_mask,
                      const orc_mode* mode, uint8_t* mask) {
  const Level& L = ref->levels[level];
  std::vector<uint8_t> sel;
  const int64_t S = select_mask(L, predicate, ti, td, level_mask, sel);
  if (mask) {
    std::memcpy(mask, sel.data(), sel.size());
    if (mode && mode->drop_odd_point && (S % 2))
      for (size_t p = sel.size(); p-- > 0;)
        if (sel[p]) { mask[p] = 0; break; }
  }
  return S;
}

// orc_match against the point lists of a predicate and per-level masks (NULL, or one entry per level, each NULL or
// h_l*w_l bytes); cfg's derivative thresholds are not read.  orc_match runs unchanged on a copy of the reference pyramid
// whose planes encode the lists: with thresholds (-1, -1) its selection keeps exactly the pixels with valid z, zdx, zdy,
// so an unlisted pixel gets zdx = NaN, and a listed pixel without six valid channels (MASK_ONLY only) gets z = +inf and
// zero depth gradients -- it stays in the list, and its projection is NaN (inf / inf), so it fails the bounds test
// exactly like the reference's NaN-depth point.  Every other value of a listed point is the pyramid's own.
int orc_match_ex(orc_pyramid* ref, orc_pyramid* cur, const orc_config* cfg, int predicate, float ti, float td,
                 const uint8_t* const* level_masks, const double T_init[16], const orc_mode* mode, orc_result* result,
                 orc_iteration_stats* iters, int max_iters, int* num_iters) {
  orc_pyramid listed = *ref;
  for (size_t l = 0; l < listed.levels.size(); ++l) {
    Level& L = listed.levels[l];
    std::vector<uint8_t> sel;
    select_mask(ref->levels[l], predicate, ti, td, level_masks ? level_masks[l] : nullptr, sel);
    for (size_t p = 0; p < sel.size(); ++p) {
      bool all_valid = true;
      for (int c = 0; c < 6; ++c) all_valid = all_valid && L.ch[c][p] == L.ch[c][p];
      if (!sel[p]) L.ch[4][p] = kNaNf;
      else if (predicate == 2 && !all_valid) {
        L.ch[1][p] = std::numeric_limits<float>::infinity();
        L.ch[4][p] = 0.0f; L.ch[5][p] = 0.0f;
      }
    }
  }
  orc_config c = *cfg;
  c.intensity_derivative_threshold = -1.0f;
  c.depth_derivative_threshold = -1.0f;
  return orc_match(&listed, cur, &c, T_init, mode, result, iters, max_iters, num_iters);
}

}  // extern "C"
