// plane.cu — the support-plane fit of Cloud::sampleAbovePlane (cloud.cpp:407-435) on the device, as specified by
// include/gpd_b200_plane.h (cfg key `sample_above_plane`):
//
//   k_plane_setup     one thread per hypothesis: draw the triple, validity, float32 plane
//   k_plane_count     hypotheses x points: a tile of the cloud in shared memory, PLANE_HPT hypotheses per thread with
//                     their inlier counts in registers, added into counts[h] with integer atomics (order-free, exact)
//   k_plane_argmax    one CTA: the largest (count, -h) key over the valid hypotheses
//   k_plane_flag      inlier / off-plane flag of every point against the winning or the refined plane
//     + cub scan + k_plane_compact   order-preserving compaction (the inliers' coordinates, or the off-plane indices)
//   k_plane_refine    one warp: the ordered float32 moments of the inliers (lanes 0..8 own one accumulator each, the
//                     whole warp stages the coordinates through shared memory), lane 0 runs pcl::eigen33
// Compiled with -fmad=false: every float32 operation is rounded separately, like the oracle's.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <cub/cub.cuh>

#include "../../include/gpd_b200_plane.h"
#include "common.cuh"
#include "pcl_eigen33.cuh"

namespace {

constexpr int PLANE_TB = 256;     // threads per CTA of the counting kernel
constexpr int PLANE_HPT = 4;      // hypotheses per thread (PLANE_TB * PLANE_HPT per CTA row)
constexpr int PLANE_TILE = 1024;  // cloud points per shared-memory tile
constexpr int MOM_TILE = 2048;    // inlier coordinates per tile of the moment pass
constexpr int MOM_STRIDE = MOM_TILE + 1;  // the three staged arrays start in different banks

// device-side state of one call
struct PlaneState {
  float hyp[4];      // winning hypothesis' plane
  float ref[4];      // final plane (refined, or the winner's when it has fewer than 4 inliers)
  int winner;        // -1: no valid hypothesis
  int win_count;
  int refined;
  int pad_;
};

__global__ void k_plane_setup(const float *xyz, int N, int M, unsigned long long seed, float4 *coef, int *ok, int *counts) {
  const int h = blockIdx.x * blockDim.x + threadIdx.x;
  if (h >= M) return;
  int id[3];
  for (int j = 0; j < 3; j++) id[j] = gpdb_plane_draw(seed, h, j, N);
  float c[4] = {0.f, 0.f, 0.f, 0.f};
  int good = id[0] != id[1] && id[0] != id[2] && id[1] != id[2];
  if (good) good = gpdb_plane_of_triple(xyz + 3 * (size_t)id[0], xyz + 3 * (size_t)id[1], xyz + 3 * (size_t)id[2], c);
  coef[h] = make_float4(c[0], c[1], c[2], c[3]);
  ok[h] = good;
  counts[h] = 0;
}

__global__ void __launch_bounds__(PLANE_TB) k_plane_count(const float *xyz, int N, int M, const float4 *coef, const int *ok,
                                                          float tf, int *counts) {
  __shared__ float sp[3][PLANE_TILE];
  float c[PLANE_HPT][4];
  int cnt[PLANE_HPT];
  bool use[PLANE_HPT];
#pragma unroll
  for (int q = 0; q < PLANE_HPT; q++) {
    const int h = blockIdx.y * PLANE_TB * PLANE_HPT + q * PLANE_TB + threadIdx.x;
    use[q] = h < M && ok[h];
    const float4 v = h < M ? coef[h] : make_float4(0.f, 0.f, 0.f, 0.f);
    c[q][0] = v.x;
    c[q][1] = v.y;
    c[q][2] = v.z;
    c[q][3] = v.w;
    cnt[q] = 0;
  }
  for (int t0 = blockIdx.x * PLANE_TILE; t0 < N; t0 += gridDim.x * PLANE_TILE) {
    const int m = min(PLANE_TILE, N - t0);
    __syncthreads();
    for (int e = threadIdx.x; e < 3 * m; e += PLANE_TB) sp[e % 3][e / 3] = xyz[3 * (size_t)t0 + e];
    __syncthreads();
    for (int k = 0; k < m; k++) {
      const float x = sp[0][k], y = sp[1][k], z = sp[2][k];
#pragma unroll
      for (int q = 0; q < PLANE_HPT; q++) cnt[q] += gpdb_plane_inlier(c[q], x, y, z, tf);
    }
  }
#pragma unroll
  for (int q = 0; q < PLANE_HPT; q++) {
    const int h = blockIdx.y * PLANE_TB * PLANE_HPT + q * PLANE_TB + threadIdx.x;
    if (use[q] && cnt[q]) atomicAdd(counts + h, cnt[q]);
  }
}

// key = count << 32 | (0xffffffff - h): the largest key has the most inliers, then the lowest h; 0 = invalid
__global__ void __launch_bounds__(1024) k_plane_argmax(int M, const float4 *coef, const int *ok, const int *counts,
                                                       PlaneState *st) {
  __shared__ unsigned long long s_best[32];
  unsigned long long best = 0;
  for (int h = threadIdx.x; h < M; h += blockDim.x)
    if (ok[h]) best = max(best, ((unsigned long long)(unsigned)counts[h] << 32) | (0xffffffffu - (unsigned)h));
  for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if ((threadIdx.x & 31) == 0) s_best[threadIdx.x >> 5] = best;
  __syncthreads();
  if (threadIdx.x >= 32) return;
  best = threadIdx.x < (blockDim.x >> 5) ? s_best[threadIdx.x] : 0ull;
  for (int o = 16; o > 0; o >>= 1) best = max(best, __shfl_xor_sync(0xffffffffu, best, o));
  if (threadIdx.x != 0) return;
  st->refined = 0;
  st->pad_ = 0;
  if (best == 0) {
    st->winner = -1;
    st->win_count = 0;
    for (int a = 0; a < 4; a++) st->hyp[a] = st->ref[a] = 0.f;
    return;
  }
  const int h = (int)(0xffffffffu - (unsigned)(best & 0xffffffffull));
  const float4 v = coef[h];
  st->winner = h;
  st->win_count = (int)(best >> 32);
  st->hyp[0] = st->ref[0] = v.x;
  st->hyp[1] = st->ref[1] = v.y;
  st->hyp[2] = st->ref[2] = v.z;
  st->hyp[3] = st->ref[3] = v.w;
}

// flag[i] = point i is an inlier of the plane (off = 0) or is not (off = 1)
__global__ void k_plane_flag(const float *xyz, int N, const float *plane, float tf, int off, int *flag) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  const float c[4] = {plane[0], plane[1], plane[2], plane[3]};
  flag[i] = gpdb_plane_inlier(c, xyz[3 * (size_t)i], xyz[3 * (size_t)i + 1], xyz[3 * (size_t)i + 2], tf) ^ off;
}

// flagged points in ascending index order: idx_out[k] = i, and (soa != nullptr) their coordinates soa[0|1|2][k]
__global__ void k_plane_compact(const float *xyz, int N, const int *flag, const int *pos, int *idx_out, float *soa) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N || !flag[i]) return;
  const int k = pos[i];
  if (idx_out) idx_out[k] = i;
  if (soa) {
    soa[k] = xyz[3 * (size_t)i];
    soa[(size_t)N + k] = xyz[3 * (size_t)i + 1];
    soa[2 * (size_t)N + k] = xyz[3 * (size_t)i + 2];
  }
}

// optimizeModelCoefficients over the n = pos[N-1] + flag[N-1] inliers whose coordinates soa holds in index order
__global__ void __launch_bounds__(32) k_plane_refine(const float *soa, int N, const int *flag, const int *pos, PlaneState *st) {
  __shared__ float s[3 * MOM_STRIDE];
  const int lane = threadIdx.x;
  const int n = pos[N - 1] + flag[N - 1];
  if (n < 4) return;  // the winner's coefficients stay (k_plane_argmax copied them to st->ref)
  // lanes 0..8 own accu[0..8] = xx xy xz yy yz zz x y z (lanes 6..8 multiply by 1.0f, which is exact)
  const int ia = (lane == 3 || lane == 4 || lane == 7) ? 1 : ((lane == 5 || lane == 8) ? 2 : 0);
  const int ib = (lane == 1 || lane == 3) ? 1 : ((lane == 2 || lane == 4 || lane == 5) ? 2 : (lane == 0 ? 0 : -1));
  const float *pa = s + ia * MOM_STRIDE;
  const float *pb = s + max(ib, 0) * MOM_STRIDE;
  const bool prod = ib >= 0;
  float acc = 0.0f;
  for (int b0 = 0; b0 < n; b0 += MOM_TILE) {
    const int m = min(MOM_TILE, n - b0);
    __syncwarp();
    for (int a = 0; a < 3; a++) {
      const float *g = soa + (size_t)a * N + b0;
#pragma unroll 4
      for (int k = lane; k < m; k += 32) s[a * MOM_STRIDE + k] = g[k];
    }
    __syncwarp();
    if (lane < 9) {
      // strictly ascending k; every product is rounded before it is added (-fmad=false)
#pragma unroll 8
      for (int k = 0; k < m; k++) acc += pa[k] * (prod ? pb[k] : 1.0f);
    }
  }
  acc = acc / (float)n;
  float a9[9];
#pragma unroll
  for (int k = 0; k < 9; k++) a9[k] = __shfl_sync(0xffffffffu, acc, k);
  if (lane != 0) return;
  float cov[3][3];
  cov[0][0] = a9[0] - a9[6] * a9[6];
  cov[0][1] = a9[1] - a9[6] * a9[7];
  cov[0][2] = a9[2] - a9[6] * a9[8];
  cov[1][1] = a9[3] - a9[7] * a9[7];
  cov[1][2] = a9[4] - a9[7] * a9[8];
  cov[2][2] = a9[5] - a9[8] * a9[8];
  cov[1][0] = cov[0][1];
  cov[2][0] = cov[0][2];
  cov[2][1] = cov[1][2];
  float v[3];
  pcl_eigen33_smallest(cov, v);
  st->ref[0] = v[0];
  st->ref[1] = v[1];
  st->ref[2] = v[2];
  st->ref[3] = -((v[0] * a9[6] + v[1] * a9[7]) + v[2] * a9[8]);
  st->refined = 1;
}

}  // namespace

#define LAUNCH_CHECK()                                   \
  do {                                                   \
    ctx->launches++;                                     \
    cudaError_t e__ = cudaGetLastError();                \
    if (e__ != cudaSuccess) {                            \
      gpdb_set_error(ctx, GPDB_ERR_CUDA, "%s:%d launch -> %s", __FILE__, __LINE__, cudaGetErrorString(e__)); \
      return GPDB_ERR_CUDA;                              \
    }                                                    \
  } while (0)

// flags against `plane` (a device pointer), exclusive scan, compaction. The number of flagged points is
// pos[N-1] + flag[N-1]: k_plane_refine reads it on the device, the host after the final selection.
static int plane_select(gpdb_ctx *ctx, const float *plane, float tf, int off, int *flag, int *pos, int *idx_out, float *soa) {
  const int N = ctx->N, tb = 256;
  k_plane_flag<<<(N + tb - 1) / tb, tb, 0, ctx->stream>>>(ctx->d_xyz, N, plane, tf, off, flag);
  LAUNCH_CHECK();
  size_t tmp_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, flag, pos, N, ctx->stream);
  void *tmp = gpdb_scratch(ctx, 1, tmp_bytes);
  if (!tmp) return GPDB_ERR_CUDA;
  CUDA_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flag, pos, N, ctx->stream));
  ctx->launches += 2;
  k_plane_compact<<<(N + tb - 1) / tb, tb, 0, ctx->stream>>>(ctx->d_xyz, N, flag, pos, idx_out, soa);
  LAUNCH_CHECK();
  return GPDB_OK;
}

extern "C" {

void gpdb_plane_params_default(gpdb_plane_params *pp) {
  pp->distance_threshold = GPDB_PLANE_THRESHOLD;
  pp->num_hypotheses = GPDB_PLANE_HYPOTHESES;
  pp->seed = GPDB_PLANE_SEED;
}

int gpdb_sample_above_plane(gpdb_ctx *ctx, const gpdb_plane_params *pp, int32_t *off_plane_idx_out, gpdb_plane_info *info_out) {
  if (!ctx) return GPDB_ERR_INVALID;
  if (!pp || !off_plane_idx_out || !(pp->distance_threshold > 0.0) || !std::isfinite(pp->distance_threshold) ||
      pp->num_hypotheses < 1 || pp->num_hypotheses > GPDB_PLANE_MAX_HYPOTHESES) {
    gpdb_set_error(ctx, GPDB_ERR_INVALID,
                   "gpdb_sample_above_plane: need params and an output array, 0 < distance_threshold < inf, "
                   "1 <= num_hypotheses <= %d", GPDB_PLANE_MAX_HYPOTHESES);
    return GPDB_ERR_INVALID;
  }
  if (!ctx->cloud_set) {
    gpdb_set_error(ctx, GPDB_ERR_STATE, "no point cloud: call gpdb_set_cloud / gpdb_preprocess first");
    return GPDB_ERR_STATE;
  }
  CUDA_TRY(cudaSetDevice(ctx->device));
  gpdb_plane_info info;
  memset(&info, 0, sizeof(info));
  info.hypothesis = -1;
  const int N = ctx->N, M = pp->num_hypotheses;
  if (N < 3) {  // no triple can be drawn: the fit fails
    if (info_out) *info_out = info;
    return 0;
  }
  const float tf = gpdb_plane_float_threshold(pp->distance_threshold);
  unsigned char *hb = (unsigned char *)gpdb_scratch(ctx, 19, sizeof(PlaneState) + (sizeof(float4) + 2 * sizeof(int)) * (size_t)M);
  if (!hb) return GPDB_ERR_CUDA;
  PlaneState *d_st = (PlaneState *)hb;
  float4 *coef = (float4 *)(hb + sizeof(PlaneState));
  int *ok = (int *)(coef + M), *counts = ok + M;
  int *flag = (int *)gpdb_scratch(ctx, 20, sizeof(int) * 6 * (size_t)N);
  if (!flag) return GPDB_ERR_CUDA;
  int *pos = flag + N, *idx = pos + N;
  float *soa = (float *)(idx + N);
  // ---- hypotheses, inlier counts, winner
  k_plane_setup<<<(M + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_xyz, N, M, (unsigned long long)pp->seed, coef, ok, counts);
  LAUNCH_CHECK();
  const int rows = (M + PLANE_TB * PLANE_HPT - 1) / (PLANE_TB * PLANE_HPT);
  const int tiles = (N + PLANE_TILE - 1) / PLANE_TILE;
  const int cols = std::max(1, std::min(tiles, (ctx->sm_count * 4 + rows - 1) / rows));
  k_plane_count<<<dim3(cols, rows), PLANE_TB, 0, ctx->stream>>>(ctx->d_xyz, N, M, coef, ok, tf, counts);
  LAUNCH_CHECK();
  k_plane_argmax<<<1, 1024, 0, ctx->stream>>>(M, coef, ok, counts, d_st);
  LAUNCH_CHECK();
  PlaneState st;
  CUDA_TRY(cudaMemcpyAsync(&st, d_st, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (st.winner < 0) {  // every triple degenerate
    if (info_out) *info_out = info;
    return 0;
  }
  // ---- optimizeModelCoefficients: the winner's inliers in index order, moments, eigen33; then the final selection
  int rc = plane_select(ctx, d_st->hyp, tf, 0, flag, pos, nullptr, soa);
  if (rc != GPDB_OK) return rc;
  k_plane_refine<<<1, 32, 0, ctx->stream>>>(soa, N, flag, pos, d_st);
  LAUNCH_CHECK();
  rc = plane_select(ctx, d_st->ref, tf, 1, flag, pos, idx, nullptr);
  if (rc != GPDB_OK) return rc;
  int last[2];
  CUDA_TRY(cudaMemcpyAsync(&st, d_st, sizeof(st), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(&last[0], flag + N - 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(&last[1], pos + N - 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  const int n_off = last[0] + last[1];
  for (int a = 0; a < 4; a++) {
    info.coefficients[a] = st.ref[a];
    info.hypothesis_coefficients[a] = st.hyp[a];
  }
  info.hypothesis = st.winner;
  info.hypothesis_inliers = st.win_count;
  info.inliers = N - n_off;
  info.refined = st.refined;
  if (info_out) *info_out = info;
  if (n_off == 0 || n_off == N) return 0;  // every point on the plane, or no point on it: the fit fails
  CUDA_TRY(cudaMemcpyAsync(off_plane_idx_out, idx, sizeof(int) * (size_t)n_off, cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  return n_off;
}

}  // extern "C"
