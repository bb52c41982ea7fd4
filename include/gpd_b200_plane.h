/*
 * gpd_b200_plane.h — SPECIFICATION of the deterministic support-plane fit behind gpdb_sample_above_plane
 * (cfg key `sample_above_plane`; the reference's Cloud::sampleAbovePlane, cloud.cpp:407-435, called from
 * candidates_generator.cpp:32-34 and cem_detect_grasps.cpp:70-84).
 *
 * The reference fits the dominant plane with PCL's SACSegmentation (SACMODEL_PLANE, SAC_RANSAC,
 * setOptimizeCoefficients(true), distance threshold 0.01) and keeps the points OFF that plane as sample
 * indices. PCL's RANSAC cannot be reproduced: its draws come from boost::mt19937 + uniform_int and it stops
 * adaptively after at most 50 iterations. Both the CPU oracle (plane_oracle/plane_oracle.cpp) and the CUDA kernels
 * (gpd_b200/csrc/plane.cu) implement THIS definition over the installed cloud's float32 points p[0..N):
 *
 *  1. Hypotheses (THE VARIANT: the draw, a fixed budget, no adaptive stop). num_hypotheses triples; index j
 *     (0..2) of hypothesis h is gpdb_plane_draw(seed, h, j, N): splitmix64 of the counter 3h + j mixed with the
 *     seed, mapped to [0, N) by a multiply-high. A triple is invalid, and never redrawn, when two of its
 *     indices are equal, when it fails PCL's collinearity test (SampleConsensusModelPlane::isSampleGood:
 *     the element-wise ratios (p1-p0)/(p2-p0) all equal, float32), or when its cross product is zero (no
 *     plane to normalise; PCL would go on with a NaN model, which can never win).
 *  2. Plane of a triple (restates SampleConsensusModelPlane::computeModelCoefficients, float32): u = p1-p0,
 *     v = p2-p0, n = u x v, n /= sqrtf((n.x*n.x + n.y*n.y) + n.z*n.z), d = -((n.x*p0.x + n.y*p0.y) + n.z*p0.z).
 *  3. Distance predicate (restates countWithinDistance / selectWithinDistance): a point is an inlier of
 *     (a, b, c, d) when fabsf(((a*x + b*y) + c*z) + d) < threshold, every operation rounded to float32 (no FMA),
 *     the comparison in float64 as PCL's `float distance < double threshold_`. gpdb_plane_float_threshold
 *     gives the float32 bound that decides exactly the same comparison.
 *  4. Winner: the valid hypothesis with the most inliers; on a tie the lowest h.
 *  5. Refinement (restates optimizeModelCoefficients, PCL 1.9.1): with fewer than 4 inliers the winner's
 *     coefficients are kept. Otherwise computeMeanAndCovarianceMatrix in float32, ONE pass over the winner's
 *     inliers in ascending index order (accumulators xx xy xz yy yz zz x y z, each product rounded before it
 *     is added, then each divided by the count; cov = E[ab] - E[a]E[b]), the pcl::eigen33 eigenvector of the
 *     smallest eigenvalue as n, d = -((n.x*c.x + n.y*c.y) + n.z*c.z) with c the centroid. The inliers are then
 *     selected again with the refined plane (SACSegmentation::segment).
 *  6. Result: the indices of the points that are NOT inliers of the final plane, ascending (ExtractIndices
 *     with setNegative(true)). The fit FAILS (result: no indices, the caller keeps the whole cloud,
 *     cloud.cpp:420-433) when N < 3, when no hypothesis is valid, or when the final plane has no inlier or
 *     every point is an inlier.
 *
 * Parts 2, 3 and 5 restate PCL from its published algorithm (PCL 1.9.1, the minimum version the reference
 * names); they are not pinned against PCL binaries, and the float32 evaluation orders written above are this
 * specification's (PCL leaves them to Eigen's vectorised reductions). Parts 1 and 4 are the variant.
 */
#ifndef GPD_B200_PLANE_H_
#define GPD_B200_PLANE_H_

#include <math.h>
#include <stdint.h>

#ifndef GPDB_HD
#if defined(__CUDACC__)
#define GPDB_HD __host__ __device__ __forceinline__
#else
#define GPDB_HD static inline
#endif
#endif

#define GPDB_PLANE_THRESHOLD 0.01     /* cloud.cpp:418 */
#define GPDB_PLANE_HYPOTHESES 1024
#define GPDB_PLANE_MAX_HYPOTHESES (1 << 20)
#define GPDB_PLANE_SEED 1ull

GPDB_HD uint64_t gpdb_splitmix64(uint64_t z) {
  z += 0x9E3779B97F4A7C15ull;
  z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
  z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

/* index j (0..2) of hypothesis h over a cloud of n points */
GPDB_HD int32_t gpdb_plane_draw(uint64_t seed, int32_t h, int32_t j, int32_t n) {
  const uint64_t r = gpdb_splitmix64(gpdb_splitmix64(seed) + 3ull * (uint64_t)h + (uint64_t)j);
  return (int32_t)(((r >> 32) * (uint64_t)(uint32_t)n) >> 32);
}

/* plane of the triple p0, p1, p2 (each x, y, z); returns 0 for an invalid triple (collinear or zero normal) */
GPDB_HD int gpdb_plane_of_triple(const float *p0, const float *p1, const float *p2, float coef[4]) {
  const float u0 = p1[0] - p0[0], u1 = p1[1] - p0[1], u2 = p1[2] - p0[2];
  const float v0 = p2[0] - p0[0], v1 = p2[1] - p0[1], v2 = p2[2] - p0[2];
  const float r0 = u0 / v0, r1 = u1 / v1, r2 = u2 / v2;
  if (r0 == r1 && r2 == r1) return 0; /* isSampleGood: (dy1dy2[0] != dy1dy2[1]) || (dy1dy2[2] != dy1dy2[1]) */
  float a = u1 * v2 - u2 * v1;
  float b = u2 * v0 - u0 * v2;
  float c = u0 * v1 - u1 * v0;
  const float s = (a * a + b * b) + c * c;
  if (!(s > 0.0f)) return 0;
  const float nrm = sqrtf(s);
  a = a / nrm;
  b = b / nrm;
  c = c / nrm;
  coef[0] = a;
  coef[1] = b;
  coef[2] = c;
  coef[3] = -((a * p0[0] + b * p0[1]) + c * p0[2]);
  return 1;
}

/* the float32 value t such that, for every float x (NaN included), x < t  <=>  (double)x < threshold:
 * the smallest float32 that is >= threshold */
static inline float gpdb_plane_float_threshold(double threshold) {
  float t = (float)threshold;
  if ((double)t < threshold) t = nextafterf(t, INFINITY);
  return t;
}

/* point-to-plane predicate of part 3; tf = gpdb_plane_float_threshold(threshold) */
GPDB_HD int gpdb_plane_inlier(const float coef[4], float x, float y, float z, float tf) {
  const float v = ((coef[0] * x + coef[1] * y) + coef[2] * z) + coef[3];
  return fabsf(v) < tf;
}

#endif /* GPD_B200_PLANE_H_ */
