// teaser/matcher.h -- teaser::Matcher with upstream TEASER++'s names (teaser/matcher.h there: FGR's
// AdvancedMatching over FLANN), computed on the GPU by psulvsb_match_host (include/psulvsb.h; DESIGN.md section 10).
// Differences, on purpose: the tuple test draws from a seeded Philox stream (setSeed) instead of rand() after
// srand(time); use_absolute_scale is accepted and has no effect, because FGR normalises both clouds by one global
// scale and the tuple test only compares length ratios.
#pragma once

#include <cstdint>
#include <utility>
#include <vector>

#include "../psulvsb.h"
#include "fpfh.h"
#include "geometry.h"

namespace teaser {

class Matcher {
public:
  Matcher() = default;

  void setSeed(uint64_t seed) { seed_ = seed; }

  /// (source index, target index) pairs; empty on failure (lastStatus() / psulvsb_last_error() say why).
  std::vector<std::pair<int, int>> calculateCorrespondences(PointCloud& source_points, PointCloud& target_points,
                                                            FPFHCloud& source_features, FPFHCloud& target_features,
                                                            bool use_absolute_scale = true, bool use_crosscheck = true,
                                                            bool use_tuple_test = true, float tuple_scale = 0) {
    (void)use_absolute_scale;
    std::vector<std::pair<int, int>> corres;
    const std::vector<double> s = coords(source_points), t = coords(target_points);
    const int ns = static_cast<int>(source_points.size()), nt = static_cast<int>(target_points.size());
    if (source_features.size() != source_points.size() || target_features.size() != target_points.size()) {
      status_ = PSULVSB_ERR_INVALID;
      return corres;
    }
    long long cap = use_tuple_test ? 3000 : (long long)ns + (use_crosscheck ? 0 : nt);
    std::vector<int> pairs(2 * static_cast<size_t>(cap > 0 ? cap : 1));
    long long n = 0;
    status_ = psulvsb_match_host(s.data(), ns, t.data(), nt, ns ? source_features[0].histogram : nullptr,
                                 nt ? target_features[0].histogram : nullptr, use_crosscheck, use_tuple_test,
                                 tuple_scale, seed_, pairs.data(), cap, &n);
    if (status_ != PSULVSB_OK) return corres;
    corres.reserve(static_cast<size_t>(n));
    for (long long k = 0; k < n; ++k) corres.emplace_back(pairs[2 * k], pairs[2 * k + 1]);
    return corres;
  }
  int lastStatus() const { return status_; }

private:
  static std::vector<double> coords(const PointCloud& c) {
    std::vector<double> v(3 * c.size());
    for (size_t i = 0; i < c.size(); ++i) {
      v[3 * i] = c[i].x;
      v[3 * i + 1] = c[i].y;
      v[3 * i + 2] = c[i].z;
    }
    return v;
  }
  uint64_t seed_ = 0;
  int status_ = PSULVSB_OK;
};

} // namespace teaser
