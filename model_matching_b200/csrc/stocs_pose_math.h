// stocs_pose_math.h -- clustering::get_pose_diff (reference src/pose_clustering.cpp:5-72), the pose
// distance of the greedy clustering, as ONE statement shared by the host shim
// (host/pose_clustering.cpp) and the clustering kernels (csrc/cluster.cu).  Same rules as
// stocs_math.h: IEEE add/sub/mul/div/sqrt in a fixed order, no contraction, no libm -- so that g++
// (-ffp-contract=off) and nvcc (-fmad=false) return the same bits and the GPU keeps exactly the
// clusters the host loop keeps.  The 3-term sums are written out as a + (b + c) (Eigen's
// redux order) rather than through sum3, which the sensitivity switches of stocs_math.h redefine.
#pragma once
#include "stocs_math.h"

namespace stocsm {

// asin(x) for |x| < 1 (binary64): atan2(x, sqrt((1 - x)(1 + x))).  NaN in, NaN out.
STOCS_HD double asin_d(double x) { return atan2_d(x, sqrt((1.0 - x) * (1.0 + x))); }

// std::min / std::max as libstdc++ defines them (the NaN behaviour of the host loop follows from that)
STOCS_HD float min_std(float a, float b) { return (b < a) ? b : a; }
STOCS_HD float max_std(float a, float b) { return (a < b) ? b : a; }

// Inverse of the 3x3 rotation block by cofactors (the closed form of Eigen's Matrix3f::inverse()).
STOCS_HD void pose_inverse3(const float a[3][3], float inv[3][3]) {
  const float c00 = a[1][1] * a[2][2] - a[1][2] * a[2][1], c01 = a[1][2] * a[2][0] - a[1][0] * a[2][2],
              c02 = a[1][0] * a[2][1] - a[1][1] * a[2][0];
  const float det = a[0][0] * c00 + a[0][1] * c01 + a[0][2] * c02;
  const float id = 1.0f / det;
  inv[0][0] = c00 * id; inv[0][1] = (a[0][2] * a[2][1] - a[0][1] * a[2][2]) * id; inv[0][2] = (a[0][1] * a[1][2] - a[0][2] * a[1][1]) * id;
  inv[1][0] = c01 * id; inv[1][1] = (a[0][0] * a[2][2] - a[0][2] * a[2][0]) * id; inv[1][2] = (a[0][2] * a[1][0] - a[0][0] * a[1][2]) * id;
  inv[2][0] = c02 * id; inv[2][1] = (a[0][1] * a[2][0] - a[0][0] * a[2][1]) * id; inv[2][2] = (a[0][0] * a[1][1] - a[0][1] * a[1][0]) * id;
}

// The part of get_pose_diff that depends on the test pose only: inv(R_test), from a column-major 4x4.
STOCS_HD void pose_test_inverse(const float* T_test, float ti[3][3]) {
  float tr[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) tr[i][j] = T_test[j * 4 + i];
  pose_inverse3(tr, ti);
}

// Translation error: sqrt((dx^2 + dy^2) + dz^2) in binary64 from the binary32 differences base - test
// (dx^2 is exact there, so this is the reference's std::pow(d, 2) sum), rounded once to binary32.
STOCS_HD float pose_translation_error(const float* T_test, const float* T_base) {
  const double dx = (double)(T_base[12] - T_test[12]), dy = (double)(T_base[13] - T_test[13]),
               dz = (double)(T_base[14] - T_test[14]);
  return (float)sqrt((dx * dx + dy * dy) + dz * dz);
}

// Rotation error: max |Euler angle| in degrees of inv(R_test) * R_base after the symmetry folding.
// ti = pose_test_inverse(T_test); T_base column-major.
STOCS_HD float pose_rotation_error(const float ti[3][3], const float* T_base, const float sym[3]) {
  float rd[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j)
      rd[i][j] = ti[i][0] * T_base[j * 4 + 0] + (ti[i][1] * T_base[j * 4 + 1] + ti[i][2] * T_base[j * 4 + 2]);
  // Eigen::Quaternionf(Matrix3f): Shoemake's method
  float qw, qx, qy, qz;
  float t = rd[0][0] + rd[1][1] + rd[2][2];
  if (t > 0.0f) {
    t = sqrtf(t + 1.0f);
    qw = 0.5f * t;
    t = 0.5f / t;
    qx = (rd[2][1] - rd[1][2]) * t; qy = (rd[0][2] - rd[2][0]) * t; qz = (rd[1][0] - rd[0][1]) * t;
  } else {
    int i = 0;
    if (rd[1][1] > rd[0][0]) i = 1;
    if (rd[2][2] > rd[i][i]) i = 2;
    const int j = (i + 1) % 3, k = (j + 1) % 3;
    t = sqrtf(rd[i][i] - rd[j][j] - rd[k][k] + 1.0f);
    float q[3];
    q[i] = 0.5f * t;
    t = 0.5f / t;
    qw = (rd[k][j] - rd[j][k]) * t;
    q[j] = (rd[j][i] + rd[i][j]) * t;
    q[k] = (rd[k][i] + rd[i][k]) * t;
    qx = q[0]; qy = q[1]; qz = q[2];
  }
  // quaternion_to_euler (src/pose_clustering.cpp:5-26): float products and sums, widened to binary64
  float e[3];
  const double sinr = 2.0 * (double)(qw * qx + qy * qz), cosr = 1.0 - 2.0 * (double)(qx * qx + qy * qy);
  e[0] = (float)atan2_d(sinr, cosr);
  const double sinp = 2.0 * (double)(qw * qy - qz * qx);
  if ((sinp < 0.0 ? -sinp : sinp) >= 1.0) e[1] = (float)(sinp < 0.0 ? -kPiO2Hi : kPiO2Hi);   // copysign(M_PI / 2, sinp)
  else e[1] = (float)asin_d(sinp);
  const double siny = 2.0 * (double)(qw * qz + qx * qy), cosy = 1.0 - 2.0 * (double)(qy * qy + qz * qz);
  e[2] = (float)atan2_d(siny, cosy);
  for (int d = 0; d < 3; ++d) e[d] = (float)((double)e[d] * 180.0 / kPi);
  for (int d = 0; d < 3; ++d) {
    e[d] = fabsf(e[d]);
    if (sym[d] == 90.0f) {
      e[d] = fabsf(e[d] - 90.0f);
      e[d] = min_std(e[d], 90.0f - e[d]);
    } else if (sym[d] == 180.0f) {
      e[d] = min_std(e[d], 180.0f - e[d]);
    } else if (sym[d] == 360.0f) {
      e[d] = 0.0f;
    }
  }
  return max_std(max_std(e[0], e[1]), e[2]);
}

// get_pose_diff(test_pose, base_pose, sym_info, rot, trans); both poses column-major 4x4.
STOCS_HD void pose_diff(const float* T_test, const float* T_base, const float sym[3], float* rot, float* trans) {
  float ti[3][3];
  pose_test_inverse(T_test, ti);
  *rot = pose_rotation_error(ti, T_base, sym);
  *trans = pose_translation_error(T_test, T_base);
}

}  // namespace stocsm
