// upstream TEASER++'s teaser_cpp_fpfh call sequence against include/teaser/{fpfh,matcher,registration}.h: FPFH of
// two clouds, crosscheck matching without the tuple test, solve(src_cloud, tgt_cloud, correspondences).
// Exit code: 0 = solved, otherwise the first PSULVSB status that failed.
#include <teaser/fpfh.h>
#include <teaser/matcher.h>
#include <teaser/registration.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>

int main(int argc, char** argv) {
  const int n = argc > 1 ? std::atoi(argv[1]) : 2000;
  teaser::PointCloud src, tgt;
  unsigned int s = 12345u;
  auto uni = [&s]() { s = s * 1664525u + 1013904223u; return (s >> 8) * (1.0 / 16777216.0); };
  for (int i = 0; i < n; ++i) {
    const double x = 2 * uni(), y = 2 * uni(), z = 0.3 * std::sin(2 * x) * std::cos(3 * y) + 0.1 * x * y;
    src.push_back({float(x), float(y), float(z)});
    tgt.push_back({float(-y + 0.5), float(x - 0.2), float(z + 0.1)});  // 90 degrees about z, then a shift
  }
  teaser::FPFHEstimation fpfh;
  auto fs = fpfh.computeFPFHFeatures(src, 0.06, 0.1);
  auto ft = fpfh.computeFPFHFeatures(tgt, 0.06, 0.1);
  if (fpfh.lastStatus() != PSULVSB_OK) {
    std::printf("fpfh status=%d %s\n", fpfh.lastStatus(), psulvsb_last_error());
    return fpfh.lastStatus();
  }
  teaser::Matcher matcher;
  auto corr = matcher.calculateCorrespondences(src, tgt, *fs, *ft, false, true, false, 0.95f);
  if (matcher.lastStatus() != PSULVSB_OK) {
    std::printf("match status=%d %s\n", matcher.lastStatus(), psulvsb_last_error());
    return matcher.lastStatus();
  }
  teaser::RobustRegistrationSolver::Params params;
  params.noise_bound = 0.01;
  params.estimate_scaling = false;
  teaser::RobustRegistrationSolver solver(params);
  auto sol = solver.solve(src, tgt, corr);
  std::printf("correspondences=%zu valid=%d R00=%.6f R10=%.6f t=(%.4f, %.4f, %.4f)\n", corr.size(), int(sol.valid),
              sol.rotation(0, 0), sol.rotation(1, 0), sol.translation(0), sol.translation(1), sol.translation(2));
  return sol.valid ? 0 : 1;
}
