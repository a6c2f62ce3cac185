// psulvsb_fpfh.cc -- upstream TEASER++'s teaser_cpp_fpfh flow against the B200 library: load a PLY, apply a rigid
// transform (and optional uniform noise), compute FPFH descriptors of both clouds, match them (crosscheck, no tuple
// test), solve(src_cloud, tgt_cloud, correspondences) and report the rotation and translation errors.  With
// icp_distance > 0 the solve's answer is then refined by point-to-point ICP on the two clouds (psulvsb_icp_host, the
// step upstream's Python example hands to Open3D) and a second line reports the refined errors.
//
//   psulvsb_fpfh <file.ply> [vertex_scale = 1] [normal_radius = 0.03] [feature_radius = 0.05] [noise = 0] [seed = 1]
//                [icp_distance = 0]
//
// Differences from the upstream example, on purpose: a seeded generator; the target is the transformed source itself
// (same points, same order) so that the true correspondences are known; normals and descriptors on the GPU.
#include <teaser/fpfh.h>
#include <teaser/matcher.h>
#include <teaser/ply_io.h>
#include <teaser/registration.h>

#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <random>
#include <vector>

int main(int argc, char** argv) {
  if (argc < 2) {
    std::fprintf(stderr, "usage: %s file.ply [vertex_scale] [normal_radius] [feature_radius] [noise] [seed] [icp_distance]\n",
                 argv[0]);
    return 64;
  }
  const double scale = argc > 2 ? std::atof(argv[2]) : 1.0;
  const double rn = argc > 3 ? std::atof(argv[3]) : 0.03, rf = argc > 4 ? std::atof(argv[4]) : 0.05;
  const double noise = argc > 5 ? std::atof(argv[5]) : 0.0;
  const unsigned long long seed = argc > 6 ? std::strtoull(argv[6], nullptr, 10) : 1ull;
  const double icp_distance = argc > 7 ? std::atof(argv[7]) : 0.0;

  teaser::PLYReader reader;
  teaser::PointCloud src;
  if (reader.read(argv[1], src) != 0) {
    std::fprintf(stderr, "cannot read %s: %s\n", argv[1], psulvsb_last_error());
    return 65;
  }
  for (auto& p : src) p = {float(p.x * scale), float(p.y * scale), float(p.z * scale)};

  // rotation: random axis, angle U[0, pi); translation |t| = U[0, 1) times the cloud's extent
  std::mt19937_64 rng(seed);
  std::normal_distribution<double> g(0.0, 1.0);
  std::uniform_real_distribution<double> u(0.0, 1.0);
  double ax[3] = {g(rng), g(rng), g(rng)};
  const double an = std::sqrt(ax[0] * ax[0] + ax[1] * ax[1] + ax[2] * ax[2]);
  for (double& a : ax) a /= an;
  const double ang = M_PI * u(rng), c = std::cos(ang), s = std::sin(ang);
  double R[3][3];  // Rodrigues: c I + (1 - c) a a^T + s [a]x
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) R[i][j] = c * (i == j) + (1 - c) * ax[i] * ax[j];
  R[0][1] -= s * ax[2];
  R[0][2] += s * ax[1];
  R[1][0] += s * ax[2];
  R[1][2] -= s * ax[0];
  R[2][0] -= s * ax[1];
  R[2][1] += s * ax[0];
  double lo[3] = {1e300, 1e300, 1e300}, hi[3] = {-1e300, -1e300, -1e300};
  for (const auto& p : src) {
    const double v[3] = {p.x, p.y, p.z};
    for (int r = 0; r < 3; ++r) lo[r] = std::fmin(lo[r], v[r]), hi[r] = std::fmax(hi[r], v[r]);
  }
  const double extent = std::sqrt((hi[0] - lo[0]) * (hi[0] - lo[0]) + (hi[1] - lo[1]) * (hi[1] - lo[1]) +
                                  (hi[2] - lo[2]) * (hi[2] - lo[2]));
  double t[3] = {g(rng), g(rng), g(rng)};
  const double tn = std::sqrt(t[0] * t[0] + t[1] * t[1] + t[2] * t[2]), tl = extent * u(rng);
  for (double& x : t) x *= tl / tn;
  std::uniform_real_distribution<double> nz(-noise, noise);
  teaser::PointCloud tgt;
  for (const auto& p : src) {
    const double v[3] = {p.x, p.y, p.z};
    float q[3];
    for (int r = 0; r < 3; ++r) q[r] = float(R[r][0] * v[0] + R[r][1] * v[1] + R[r][2] * v[2] + t[r] + (noise > 0 ? nz(rng) : 0.0));
    tgt.push_back({q[0], q[1], q[2]});
  }

  teaser::FPFHEstimation fpfh;
  auto fs = fpfh.computeFPFHFeatures(src, rn, rf);
  auto ft = fpfh.computeFPFHFeatures(tgt, rn, rf);
  if (fpfh.lastStatus() != PSULVSB_OK) {
    std::printf("fpfh failed (status %d): %s\n", fpfh.lastStatus(), psulvsb_last_error());
    return fpfh.lastStatus();
  }
  teaser::Matcher matcher;
  matcher.setSeed(seed);
  auto corr = matcher.calculateCorrespondences(src, tgt, *fs, *ft, false, true, false, 0.95f);
  if (matcher.lastStatus() != PSULVSB_OK) {
    std::printf("matcher failed (status %d): %s\n", matcher.lastStatus(), psulvsb_last_error());
    return matcher.lastStatus();
  }
  int true_pairs = 0;
  for (const auto& m : corr) true_pairs += m.first == m.second;

  teaser::RobustRegistrationSolver::Params params;
  params.noise_bound = noise > 0 ? 2 * noise : 0.01 * extent;
  params.estimate_scaling = false;
  teaser::RobustRegistrationSolver solver(params);
  auto sol = solver.solve(src, tgt, corr);
  double tr = 0.0, terr = 0.0;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) tr += sol.rotation(i, j) * R[i][j];
  for (int r = 0; r < 3; ++r) terr += (sol.translation(r) - t[r]) * (sol.translation(r) - t[r]);
  const double rot_err_deg = std::acos(std::fmax(-1.0, std::fmin(1.0, (tr - 1) / 2))) * 180.0 / M_PI;
  std::printf("points=%zu correspondences=%zu true=%d valid=%d rotation_error_deg=%.6f translation_error=%.6g "
              "extent=%.6g\n",
              src.size(), corr.size(), true_pairs, int(sol.valid), rot_err_deg, std::sqrt(terr), extent);
  if (!sol.valid || icp_distance <= 0) return sol.valid ? 0 : 1;

  std::vector<double> ps, pt;  // column-major 3 x n
  for (const auto& p : src) ps.insert(ps.end(), {p.x, p.y, p.z});
  for (const auto& p : tgt) pt.insert(pt.end(), {p.x, p.y, p.z});
  psulvsb_icp_params_t ip;
  psulvsb_icp_default_params(&ip);
  ip.max_correspondence_distance = icp_distance;
  double R0[9], t0[3];
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) R0[3 * j + i] = sol.rotation(i, j);
    t0[i] = sol.translation(i);
  }
  psulvsb_icp_result_t icp;
  const int rc = psulvsb_icp_host(ps.data(), int(src.size()), pt.data(), int(tgt.size()), nullptr, &ip, R0, t0, &icp,
                                  nullptr, nullptr);
  if (rc != PSULVSB_OK) {
    std::printf("icp failed (status %d): %s\n", rc, psulvsb_last_error());
    return rc;
  }
  double tr2 = 0.0, terr2 = 0.0;
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) tr2 += icp.rotation[3 * j + i] * R[i][j];
  for (int r = 0; r < 3; ++r) terr2 += (icp.translation[r] - t[r]) * (icp.translation[r] - t[r]);
  std::printf("icp: fitness=%.6f inlier_rmse=%.6g iterations=%d status=%d rotation_error_deg=%.6g "
              "translation_error=%.6g\n",
              icp.fitness, icp.inlier_rmse, icp.iterations, icp.status,
              std::acos(std::fmax(-1.0, std::fmin(1.0, (tr2 - 1) / 2))) * 180.0 / M_PI, std::sqrt(terr2));
  return 0;
}
