/*
 * plane_oracle.cpp — CPU ORACLE of the support-plane fit behind gpdb_sample_above_plane (cfg key sample_above_plane;
 * the reference's Cloud::sampleAbovePlane, cloud.cpp:407-435), as specified by include/gpd_b200_plane.h.
 *
 * TEST INFRASTRUCTURE, NOT PRODUCT CODE: loaded by tests/ and tools/plane_bench.py through plane_oracle/__init__.py.
 * The product (libgpd_b200.so) never links or loads it. It is linked against the path's oracle (oracle/libgpd_oracle.so)
 * and takes pcl::eigen33 from there (gpdo_pcl_eigen33), the same restatement the normal estimation uses.
 * Compiled with -ffp-contract=off: every float32 operation is rounded separately, like the kernels' (-fmad=false).
 */
#include <cmath>
#include <cstdint>
#include <cstring>
#include <vector>
#ifdef _OPENMP
#include <omp.h>
#endif

#include "../include/gpd_b200.h"
#include "../include/gpd_b200_plane.h"

extern "C" {

// oracle/gpd_oracle.cpp: pcl::eigen33 (smallest eigenvalue + eigenvector) of a row-major 3x3 float32 matrix
void gpdo_pcl_eigen33(const float *cov9, float *eigenvalue, float *evec);

// RANSAC plane over fixed counter-based triples (OpenMP over hypotheses), PCL's optimizeModelCoefficients
// (computeMeanAndCovarianceMatrix in ascending inlier order + pcl::eigen33, PCL 1.9.1), selection with the final plane,
// off-plane indices. off_out has room for N; counts_out (may be NULL) receives the inlier count of every hypothesis, -1
// for an invalid one. Returns the number of off-plane indices, 0 when the fit fails, GPDB_ERR_INVALID for bad parameters.
int gpdo_sample_above_plane(const float *xyz, int32_t N, const gpdb_plane_params *pp, int32_t *off_out, gpdb_plane_info *info_out,
                            int32_t *counts_out, int32_t num_threads) {
  if (!pp || !off_out || !(pp->distance_threshold > 0.0) || !std::isfinite(pp->distance_threshold) || pp->num_hypotheses < 1 ||
      pp->num_hypotheses > GPDB_PLANE_MAX_HYPOTHESES)
    return GPDB_ERR_INVALID;
#ifdef _OPENMP
  if (num_threads > 0) omp_set_num_threads(num_threads);
#endif
  gpdb_plane_info info;
  std::memset(&info, 0, sizeof(info));
  info.hypothesis = -1;
  const int M = pp->num_hypotheses;
  if (counts_out)
    for (int h = 0; h < M; h++) counts_out[h] = -1;
  if (N < 3) {
    if (info_out) *info_out = info;
    return 0;
  }
  const float tf = gpdb_plane_float_threshold(pp->distance_threshold);
  std::vector<float> coef(4 * (size_t)M, 0.0f);
  std::vector<int> count(M, -1);
#pragma omp parallel for schedule(dynamic, 4)
  for (int h = 0; h < M; h++) {
    int id[3];
    for (int j = 0; j < 3; j++) id[j] = gpdb_plane_draw(pp->seed, h, j, N);
    if (id[0] == id[1] || id[0] == id[2] || id[1] == id[2]) continue;
    float *c = &coef[4 * (size_t)h];
    if (!gpdb_plane_of_triple(xyz + 3 * (size_t)id[0], xyz + 3 * (size_t)id[1], xyz + 3 * (size_t)id[2], c)) continue;
    int n = 0;
    for (int i = 0; i < N; i++) n += gpdb_plane_inlier(c, xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], tf);
    count[h] = n;
  }
  if (counts_out) std::memcpy(counts_out, count.data(), sizeof(int) * (size_t)M);
  int win = -1;
  for (int h = 0; h < M; h++)
    if (count[h] >= 0 && (win < 0 || count[h] > count[win])) win = h;
  if (win < 0) {
    if (info_out) *info_out = info;
    return 0;
  }
  float plane[4];
  for (int a = 0; a < 4; a++) info.hypothesis_coefficients[a] = plane[a] = coef[4 * (size_t)win + a];
  info.hypothesis = win;
  info.hypothesis_inliers = count[win];
  if (count[win] >= 4) {  // optimizeModelCoefficients: "inliers.size () <= sample_size_" keeps the model
    // computeMeanAndCovarianceMatrix (common/impl/centroid.hpp, PCL 1.9.1): float32 single pass in index order
    float accu[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
    for (int i = 0; i < N; i++) {
      const float x = xyz[3 * (size_t)i], y = xyz[3 * (size_t)i + 1], z = xyz[3 * (size_t)i + 2];
      if (!gpdb_plane_inlier(plane, x, y, z, tf)) continue;
      accu[0] += x * x;
      accu[1] += x * y;
      accu[2] += x * z;
      accu[3] += y * y;
      accu[4] += y * z;
      accu[5] += z * z;
      accu[6] += x;
      accu[7] += y;
      accu[8] += z;
    }
    const float cnt = (float)count[win];
    for (int k = 0; k < 9; k++) accu[k] /= cnt;
    float cov[9];
    cov[0] = accu[0] - accu[6] * accu[6];
    cov[1] = accu[1] - accu[6] * accu[7];
    cov[2] = accu[2] - accu[6] * accu[8];
    cov[4] = accu[3] - accu[7] * accu[7];
    cov[5] = accu[4] - accu[7] * accu[8];
    cov[8] = accu[5] - accu[8] * accu[8];
    cov[3] = cov[1];
    cov[6] = cov[2];
    cov[7] = cov[5];
    float ev, v[3];
    gpdo_pcl_eigen33(cov, &ev, v);
    plane[0] = v[0];
    plane[1] = v[1];
    plane[2] = v[2];
    plane[3] = -((v[0] * accu[6] + v[1] * accu[7]) + v[2] * accu[8]);
    info.refined = 1;
  }
  for (int a = 0; a < 4; a++) info.coefficients[a] = plane[a];
  int n_off = 0;
  for (int i = 0; i < N; i++)
    if (!gpdb_plane_inlier(plane, xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], tf)) off_out[n_off++] = i;
  info.inliers = N - n_off;
  if (info_out) *info_out = info;
  return (n_off == 0 || n_off == N) ? 0 : n_off;
}

}  // extern "C"
