// pcl_eigen33.cuh — pcl::eigen33 restated for the device (float32), shared by preprocess.cu (normal estimation) and
// plane.cu (support-plane refinement). Include from a file compiled with -fmad=false: every float32 operation is
// rounded separately, like the oracle's.
#pragma once
#include <cfloat>

namespace {

// ---- pcl::eigen33 (common/impl/eigen.hpp), Scalar = float ------------------------------------------------
// The three libm calls of computeRoots (atan2f, cosf, sinf) are evaluated in float64 and rounded to float32:
// the correctly rounded float32 value (glibc's float functions are correctly rounded in all but rare cases).
__device__ void pcl_roots2(float b, float c, float *roots) {
  roots[0] = 0.0f;
  float d = (float)((double)(b * b) - 4.0 * (double)c);
  if (d < 0.0f) d = 0.0f;
  float sd = sqrtf(d);
  roots[2] = 0.5f * (b + sd);
  roots[1] = 0.5f * (b - sd);
}
__device__ void pcl_roots(const float m[3][3], float *roots) {
  float c0 = m[0][0] * m[1][1] * m[2][2] + 2.0f * m[0][1] * m[0][2] * m[1][2] - m[0][0] * m[1][2] * m[1][2] -
             m[1][1] * m[0][2] * m[0][2] - m[2][2] * m[0][1] * m[0][1];
  float c1 = m[0][0] * m[1][1] - m[0][1] * m[0][1] + m[0][0] * m[2][2] - m[0][2] * m[0][2] + m[1][1] * m[2][2] -
             m[1][2] * m[1][2];
  float c2 = m[0][0] + m[1][1] + m[2][2];
  if (fabsf(c0) < FLT_EPSILON) {
    pcl_roots2(c2, c1, roots);
    return;
  }
  const float s_inv3 = (float)(1.0 / 3.0);
  const float s_sqrt3 = sqrtf(3.0f);
  float c2_over_3 = c2 * s_inv3;
  float a_over_3 = (c1 - c2 * c2_over_3) * s_inv3;
  if (a_over_3 > 0.0f) a_over_3 = 0.0f;
  float half_b = 0.5f * (c0 + c2_over_3 * (2.0f * c2_over_3 * c2_over_3 - c1));
  float q = half_b * half_b + a_over_3 * a_over_3 * a_over_3;
  if (q > 0.0f) q = 0.0f;
  float rho = sqrtf(-a_over_3);
  float theta = (float)atan2((double)sqrtf(-q), (double)half_b) * s_inv3;
  float cos_theta = (float)cos((double)theta);
  float sin_theta = (float)sin((double)theta);
  roots[0] = c2_over_3 + 2.0f * rho * cos_theta;
  roots[1] = c2_over_3 - rho * (cos_theta + s_sqrt3 * sin_theta);
  roots[2] = c2_over_3 - rho * (cos_theta - s_sqrt3 * sin_theta);
  float t;
  if (roots[0] >= roots[1]) { t = roots[0]; roots[0] = roots[1]; roots[1] = t; }
  if (roots[1] >= roots[2]) {
    t = roots[1]; roots[1] = roots[2]; roots[2] = t;
    if (roots[0] >= roots[1]) { t = roots[0]; roots[0] = roots[1]; roots[1] = t; }
  }
  if (roots[0] <= 0.0f) pcl_roots2(c2, c1, roots);
}
__device__ void pcl_eigen33_smallest(const float cov[3][3], float *evec) {
  float scale = 0.0f;
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) scale = fmaxf(scale, fabsf(cov[r][c]));
  if (scale <= FLT_MIN) scale = 1.0f;
  float sm[3][3];
  for (int r = 0; r < 3; r++)
    for (int c = 0; c < 3; c++) sm[r][c] = cov[r][c] / scale;
  float ev[3];
  pcl_roots(sm, ev);
  for (int d = 0; d < 3; d++) sm[d][d] -= ev[0];
  float v[3][3];
  const int ra[3] = {0, 0, 1}, rb[3] = {1, 2, 2};
  float len[3];
  for (int k = 0; k < 3; k++) {
    const float *a = sm[ra[k]], *b = sm[rb[k]];
    v[k][0] = a[1] * b[2] - a[2] * b[1];
    v[k][1] = a[2] * b[0] - a[0] * b[2];
    v[k][2] = a[0] * b[1] - a[1] * b[0];
    len[k] = v[k][0] * v[k][0] + v[k][1] * v[k][1] + v[k][2] * v[k][2];
  }
  int best;
  if (len[0] >= len[1] && len[0] >= len[2]) best = 0;
  else if (len[1] >= len[0] && len[1] >= len[2]) best = 1;
  else best = 2;
  const float sl = sqrtf(len[best]);
  for (int k = 0; k < 3; k++) evec[k] = v[best][k] / sl;
}

}  // namespace
