// teaser/fpfh.h -- teaser::FPFHEstimation with upstream TEASER++'s names and call sequence (teaser/fpfh.h there,
// over PCL), computed on the GPU by psulvsb_fpfh_host (include/psulvsb.h; DESIGN.md section 10).  No PCL types:
// FPFHSignature33 has the layout of pcl::FPFHSignature33, so FPFHCloud::points.data() is the n x 33 float buffer.
// Parity with PCL is unpinned (radius normals and descriptors follow PCL's definitions; summation order differs).
#pragma once

#include <cstddef>
#include <memory>
#include <vector>

#include "../psulvsb.h"
#include "geometry.h"

namespace teaser {

struct FPFHSignature33 {
  float histogram[33];
};

// the vector-like part of pcl::PointCloud<pcl::FPFHSignature33> that callers of the matcher use
class FPFHCloud {
public:
  std::vector<FPFHSignature33> points;
  std::size_t size() const { return points.size(); }
  bool empty() const { return points.empty(); }
  FPFHSignature33& operator[](std::size_t i) { return points[i]; }
  const FPFHSignature33& operator[](std::size_t i) const { return points[i]; }
  void push_back(const FPFHSignature33& f) { points.push_back(f); }
};

using FPFHCloudPtr = std::shared_ptr<FPFHCloud>;

class FPFHEstimation {
public:
  /// Radius normals (viewpoint: the origin) and 33-bin FPFH descriptors of every point.  On failure (no device,
  /// bad radii) the returned cloud is empty and lastStatus() / psulvsb_last_error() say why.
  FPFHCloudPtr computeFPFHFeatures(const PointCloud& input_cloud, double normal_search_radius = 0.03,
                                   double fpfh_search_radius = 0.05) {
    auto out = std::make_shared<FPFHCloud>();
    const std::size_t n = input_cloud.size();
    std::vector<double> pts(3 * n);
    for (std::size_t i = 0; i < n; ++i) {
      pts[3 * i] = input_cloud[i].x;
      pts[3 * i + 1] = input_cloud[i].y;
      pts[3 * i + 2] = input_cloud[i].z;
    }
    out->points.resize(n);
    status_ = psulvsb_fpfh_host(pts.data(), static_cast<int>(n), normal_search_radius, fpfh_search_radius, nullptr,
                                nullptr, n ? out->points[0].histogram : nullptr);
    if (status_ != PSULVSB_OK) out->points.clear();
    return out;
  }
  int lastStatus() const { return status_; }

private:
  int status_ = PSULVSB_OK;
};

} // namespace teaser
