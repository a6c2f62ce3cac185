// eig3.cuh -- FP64 eigen-solver shared by the normal estimators (k6_normals.cu: k nearest neighbours,
// k8_features.cu: fixed radius).
#pragma once

namespace psulvsb {

// eigenvector of the smallest eigenvalue of a symmetric 3x3 matrix (cyclic Jacobi, FP64)
__device__ inline void smallest_eigenvector(double a[3][3], double out[3]) {
  double v[3][3] = {{1, 0, 0}, {0, 1, 0}, {0, 0, 1}};
  for (int sweep = 0; sweep < 24; ++sweep) {
    const double off = fabs(a[0][1]) + fabs(a[0][2]) + fabs(a[1][2]);
    const double diag = fabs(a[0][0]) + fabs(a[1][1]) + fabs(a[2][2]);
    if (off <= 1e-18 * diag || off == 0.0) break;
    for (int p = 0; p < 2; ++p)
      for (int q = p + 1; q < 3; ++q) {
        if (a[p][q] == 0.0) continue;
        const double theta = (a[q][q] - a[p][p]) / (2.0 * a[p][q]);
        const double t = copysign(1.0, theta) / (fabs(theta) + sqrt(theta * theta + 1.0));
        const double c = 1.0 / sqrt(t * t + 1.0), s = t * c;
        for (int k = 0; k < 3; ++k) {  // A <- A J
          const double akp = a[k][p], akq = a[k][q];
          a[k][p] = c * akp - s * akq;
          a[k][q] = s * akp + c * akq;
        }
        for (int k = 0; k < 3; ++k) {  // A <- J^T A
          const double apk = a[p][k], aqk = a[q][k];
          a[p][k] = c * apk - s * aqk;
          a[q][k] = s * apk + c * aqk;
        }
        for (int k = 0; k < 3; ++k) {
          const double vkp = v[k][p], vkq = v[k][q];
          v[k][p] = c * vkp - s * vkq;
          v[k][q] = s * vkp + c * vkq;
        }
      }
  }
  int m = 0;
  if (a[1][1] < a[m][m]) m = 1;
  if (a[2][2] < a[m][m]) m = 2;
  out[0] = v[0][m];
  out[1] = v[1][m];
  out[2] = v[2][m];
}

}  // namespace psulvsb
