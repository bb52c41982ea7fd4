// preprocess.cu — cloud preprocessing on the device (SURVEY.md 8(f).1), the step immediately before the path:
//
//   CandidatesGenerator::preprocessPointCloud (candidates_generator.cpp:14-37)
//     removeNans          (cloud.cpp:154-164)   \  k_pre_flag + scan + k_pre_compact
//     filterWorkspace     (cloud.cpp:207-266)   /
//     voxelizeCloud       (cloud.cpp:286-348)      k_min3, k_vox_keys, radix sort, k_vox_heads, k_vox_emit
//     calculateNormalsOMP (cloud.cpp:497-535)   \  k_normals (one warp per point)
//     reverseNormals      (cloud.cpp:573-604)   /
//
// Design (not a translation of the std::set / kd-tree / OpenMP loops of the reference):
//   * voxelisation is a 63-bit key sort: points of one voxel become one run, the stable sort keeps them in index
//     order so the run head is the first-inserted point (whose camera source the reference keeps) and the normal
//     average is summed in the reference's order; the voxel set is an EXACT set (include/gpd_b200.h);
//   * normal estimation reuses the uniform grid of the hot path: one warp gathers the r-ball of its point with
//     FLANN's float32 predicate, sorts the (dist, index) keys in shared memory (bucketed rank sort) — PCL accumulates the
//     float32 covariance sums in the kd-tree's sorted order, and float32 addition does not commute — then
//     nine lanes walk the sorted list with one accumulator each (computeMeanAndCovarianceMatrix), lane 0 runs
//     pcl::eigen33's closed-form float32 solver, the viewpoint flip and reverseNormals.
// Compiled with -fmad=false: every float32 operation is rounded separately, like the oracle's.
#include <cfloat>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cub/cub.cuh>
#include <vector>

#include "common.cuh"
#include "grid.cuh"
#include "pcl_eigen33.cuh"

namespace {

constexpr int NRM_WARPS = 4;       // warps per CTA, tier 1
constexpr int NRM_CAP1 = 1024;     // neighbours per point, tier 1 (4 warps x 26 B x 1024 = 104 KB per CTA, 2 CTAs per SM)
constexpr int NRM_CAP2 = 8192;     // tier 2: one warp per CTA (208 KB)
constexpr int NRM_BYTES_PER = 26;  // key 8 + xyz 12 + bucket group 2 + pad 2 + rank 2 (keys / group / pad are reused: sorted xyz)
constexpr int NRM_NB1 = 32;        // distance buckets, tier 1
constexpr int NRM_NB2 = 256;       // tier 2

// monotone float <-> int encoding for atomicMin / atomicMax
__device__ __forceinline__ int f2ord(float f) {
  int i = __float_as_int(f);
  return i >= 0 ? i : i ^ 0x7fffffff;
}
__host__ __device__ __forceinline__ float ord2f(int i) {
  int j = i >= 0 ? i : i ^ 0x7fffffff;
#ifdef __CUDA_ARCH__
  return __int_as_float(j);
#else
  float f;
  memcpy(&f, &j, 4);
  return f;
#endif
}

// removeNans + filterWorkspace: strict inequalities of the float32 coordinates against the double bounds
__global__ void k_pre_flag(const float *xyz, int M, const double *ws, int *flag) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M) return;
  float x = xyz[3 * (size_t)i], y = xyz[3 * (size_t)i + 1], z = xyz[3 * (size_t)i + 2];
  bool ok = isfinite(x) && isfinite(y) && isfinite(z);
  ok = ok && (double)x > ws[0] && (double)x < ws[1] && (double)y > ws[2] && (double)y < ws[3] && (double)z > ws[4] &&
       (double)z < ws[5];
  flag[i] = ok ? 1 : 0;
}
__global__ void k_pre_compact(const float *xyz, const int *flag, const int *pos, int M, int *keep, float *xyz1) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= M || !flag[i]) return;
  int k = pos[i];
  keep[k] = i;
  xyz1[3 * (size_t)k] = xyz[3 * (size_t)i];
  xyz1[3 * (size_t)k + 1] = xyz[3 * (size_t)i + 1];
  xyz1[3 * (size_t)k + 2] = xyz[3 * (size_t)i + 2];
}
// pcl::getMinMax3D: per-axis minimum and maximum (ordered-int atomics), bounds[0..2] = min, [3..5] = max
__global__ void k_bounds(const float *xyz, int n, int *bounds) {
  int mn[3] = {INT_MAX, INT_MAX, INT_MAX}, mx[3] = {INT_MIN, INT_MIN, INT_MIN};
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x)
    for (int a = 0; a < 3; a++) {
      int o = f2ord(xyz[3 * (size_t)i + a]);
      mn[a] = min(mn[a], o);
      mx[a] = max(mx[a], o);
    }
  for (int a = 0; a < 3; a++) {
    mn[a] = __reduce_min_sync(0xffffffffu, mn[a]);
    mx[a] = __reduce_max_sync(0xffffffffu, mx[a]);
  }
  if ((threadIdx.x & 31) == 0)
    for (int a = 0; a < 3; a++) {
      atomicMin(bounds + a, mn[a]);
      atomicMax(bounds + 3 + a, mx[a]);
    }
}
// voxel index of a point: floorVector((pt - min_pt) / cell_size), float32 (cloud.cpp:299-301)
__device__ __forceinline__ int voxel_of(float v, float mn, float cell) { return (int)floorf((v - mn) / cell); }

__global__ void k_vox_keys(const float *xyz1, int n, const int *bounds, float cell, unsigned long long *keys, int *vals,
                           int *err) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n) return;
  unsigned long long key = 0;
  for (int a = 0; a < 3; a++) {
    int c = voxel_of(xyz1[3 * (size_t)k + a], ord2f(bounds[a]), cell);
    if (c < 0 || c >= (1 << 21)) {
      atomicAdd(err, 1);
      c = max(0, min(c, (1 << 21) - 1));
    }
    key = (key << 21) | (unsigned long long)c;
  }
  keys[k] = key;
  vals[k] = k;
}
__global__ void k_vox_heads(const unsigned long long *keys, int n, int *head) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n) return;
  head[s] = (s == 0 || keys[s] != keys[s - 1]) ? 1 : 0;
}
// one entry per voxel: first point (run head = smallest index: the sort is stable) and run start
__global__ void k_vox_groups(const int *head, const int *gid_incl, const int *vals, int n, int *gfirst, int *gbegin,
                             unsigned *gorder_key, int *gorder_val) {
  int s = blockIdx.x * blockDim.x + threadIdx.x;
  if (s >= n || !head[s]) return;
  int g = gid_incl[s] - 1;
  gfirst[g] = vals[s];
  gbegin[g] = s;
  gorder_key[g] = 0x7fffffffu - (unsigned)vals[s];  // ascending sort of this key = descending first index
  gorder_val[g] = g;
}
// voxel point = min_pt + cell_size * v.cast<float>() (cloud.cpp:322), camera source of the first point
// (cloud.cpp:325-327), normal = mean of the voxel's normals summed in index order (cloud.cpp:307-311,331-333)
__global__ void k_vox_emit(const int *gsorted, int U, int n1, const int *gfirst, const int *gbegin, const int *vals,
                           const unsigned long long *keys, const int *keep, const float *xyz1, const int *bounds,
                           float cell, const uint8_t *cam_in, const double *nrm_in, float *xyz_out, uint8_t *cam_out,
                           double *nrm_out, int *src_out) {
  int o = blockIdx.x * blockDim.x + threadIdx.x;
  if (o >= U) return;
  const int g = gsorted[o], k = gfirst[g], i = keep[k];
  for (int a = 0; a < 3; a++) {
    const float mn = ord2f(bounds[a]);
    const int c = voxel_of(xyz1[3 * (size_t)k + a], mn, cell);
    const float t = cell * (float)c;
    xyz_out[3 * (size_t)o + a] = mn + t;
  }
  cam_out[o] = cam_in[i];
  src_out[o] = i;
  if (nrm_in) {
    double acc[3] = {0.0, 0.0, 0.0};
    const unsigned long long key = keys[gbegin[g]];
    int s = gbegin[g];
    for (; s < n1 && keys[s] == key; s++) {
      const double *nn = nrm_in + 3 * (size_t)keep[vals[s]];
      acc[0] += nn[0];
      acc[1] += nn[1];
      acc[2] += nn[2];
    }
    const double cnt = (double)(s - gbegin[g]);
    nrm_out[3 * (size_t)o] = acc[0] / cnt;
    nrm_out[3 * (size_t)o + 1] = acc[1] / cnt;
    nrm_out[3 * (size_t)o + 2] = acc[2] / cnt;
  }
}
__global__ void k_gather_plain(const int *keep, int n1, const uint8_t *cam_in, const double *nrm_in, uint8_t *cam_out,
                               double *nrm_out, int *src_out) {
  int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= n1) return;
  const int i = keep[k];
  cam_out[k] = cam_in[i];
  src_out[k] = i;
  if (nrm_in)
    for (int a = 0; a < 3; a++) nrm_out[3 * (size_t)k + a] = nrm_in[3 * (size_t)i + a];
}

// ---- k_normals -------------------------------------------------------------------------------------------
// pcl::NormalEstimationOMP::computeFeature (radius search on the whole cloud, computePointNormal,
// flipNormalTowardsViewpoint) for the first camera that sees the point (convertCameraSourceMatrixToLists,
// cloud.cpp:606-621), then reverseNormals (cloud.cpp:573-604). One warp per point.
//   tier 0: point i = blockIdx.x * WARPS + warp, capacity cap; overflowing points are appended to `ovf`
//   tier 1: the points of `ovf` (one warp per CTA, large capacity); overflow -> err[4]
// Sorting the ball by (dist, index): the squared distance is quantised into NB monotone buckets (on a surface the
// neighbour count grows linearly in d^2, so the buckets fill evenly), the arrival positions are grouped by
// bucket with a counting pass, and each key is ranked inside its own bucket only: n^2 / NB comparisons, not n^2.
// Per-warp shared memory, 26 B per neighbour: keys u64[cap] + pc float[3][cap] (arrival order), grp u16[cap]
// (arrival positions grouped by bucket) + 2 B pad, rk u16[cap] (rank of each arrival position). Once the ranks are
// known, keys / grp / pad are dead and receive the coordinates IN SORTED ORDER (sx, sy over the keys, sz over grp + pad),
// so that the ordered accumulation reads three plain arrays sequentially (16-byte loads, no index chain).
template <int WARPS, int NB>
__global__ void __launch_bounds__(WARPS * 32) k_normals(const DevParams *Pp, DevCloud cl, int N, float r2, float rf,
                                                        int cap, double *nrm_out, int *ovf, int *ovf_count, int tier,
                                                        int *err) {
  const DevParams &P = *Pp;
  extern __shared__ __align__(16) unsigned char nrm_dyn[];
  __shared__ int s_hist[WARPS][2 * NB + 1];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  unsigned char *base = nrm_dyn + (size_t)warp * cap * NRM_BYTES_PER;
  unsigned long long *keys = reinterpret_cast<unsigned long long *>(base);
  float *pc = reinterpret_cast<float *>(keys + cap);  // [3][cap]
  unsigned short *grp = reinterpret_cast<unsigned short *>(pc + 3 * (size_t)cap);
  unsigned short *rk = grp + 2 * (size_t)cap;                       // after grp[cap] and the pad[cap]
  float *sxy = reinterpret_cast<float *>(keys);                     // sorted x [cap] | sorted y [cap] (over keys)
  float *sz = reinterpret_cast<float *>(grp);                       // sorted z [cap] (over grp + pad)
  int *hist = s_hist[warp];      // [0..NB]: bucket starts after the scan
  int *fill = hist + NB + 1;     // [0..NB): per-bucket cursor of the grouping pass
  int i;
  if (tier == 0) {
    i = blockIdx.x * WARPS + warp;
    if (i >= N) return;
  } else {
    if ((int)blockIdx.x >= *ovf_count) return;
    i = ovf[blockIdx.x];
  }
  const uint8_t camm = cl.cam[i];
  double *out = nrm_out + 3 * (size_t)i;
  if (camm == 0) {  // seen by no camera: the reference leaves the column uninitialised; specified as 0
    if (lane < 3) out[lane] = 0.0;
    return;
  }
  for (int b = lane; b < 2 * NB + 1; b += 32) hist[b] = 0;
  __syncwarp();
  const float q[3] = {cl.xyz[3 * (size_t)i], cl.xyz[3 * (size_t)i + 1], cl.xyz[3 * (size_t)i + 2]};
  const float bscale = (float)NB / r2;
  const SegRange sr = seg_range(P, q, rf);
  int cnt = 0;
  for (int j0 = 0; j0 < sr.nrows; j0 += 32) {
    int st = 0, len = 0;
    if (j0 + lane < sr.nrows) seg_row(P, cl.cell_start, sr, j0 + lane, st, len);
    unsigned nonempty = __ballot_sync(0xffffffffu, len > 0);
    while (nonempty) {
      const int j = __ffs(nonempty) - 1;
      nonempty &= nonempty - 1;
      const int rs = __shfl_sync(0xffffffffu, st, j), rl = __shfl_sync(0xffffffffu, len, j);
      // four 32-point chunks of the row in flight at once: the gather is bound by L2 latency, not bandwidth
      for (int k0 = 0; k0 < rl; k0 += 128) {
        float4 pv[4];
#pragma unroll
        for (int u = 0; u < 4; u++) {
          const int k = k0 + 32 * u + lane;
          pv[u] = (k < rl) ? __ldg(cl.pts4 + rs + k) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int u = 0; u < 4; u++) {
          if (k0 + 32 * u >= rl) break;
          const float4 p = pv[u];
          const float d = l2_simple(q, p.x, p.y, p.z);
          const bool hit = (k0 + 32 * u + lane < rl) && d < r2;
          const unsigned m = __ballot_sync(0xffffffffu, hit);
          const int pos = cnt + __popc(m & ((1u << lane) - 1));
          if (hit && pos < cap) {
            keys[pos] = ((unsigned long long)__float_as_uint(d) << 32) | (unsigned)__float_as_int(p.w);
            pc[pos] = p.x;
            pc[cap + pos] = p.y;
            pc[2 * cap + pos] = p.z;
            atomicAdd(hist + 1 + min((int)(d * bscale), NB - 1), 1);
          }
          cnt += __popc(m);
        }
      }
    }
  }
  if (cnt > cap) {
    if (lane == 0) {
      if (tier == 0) ovf[atomicAdd(ovf_count, 1)] = i;
      else atomicAdd(err + 4, 1);
    }
    if (tier == 0) return;
    cnt = cap;
  }
  __syncwarp();
  float n[3];
  if (cnt < 3) {  // computePointNormal: fewer than 3 neighbours -> NaN normal
    n[0] = n[1] = n[2] = __int_as_float(0x7fc00000);
  } else {
    // inclusive scan of the bucket counts in place: hist[1 + b] = end of bucket b, so hist[b] = start of bucket b
    int carry = 0;
    for (int b0 = 0; b0 < NB; b0 += 32) {
      const int b = b0 + lane;
      int incl = (b < NB) ? hist[1 + b] : 0;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
      }
      if (b < NB) hist[1 + b] = carry + incl;
      carry += __shfl_sync(0xffffffffu, incl, 31);
    }
    __syncwarp();
    // grouping pass: arrival positions grouped by bucket (unordered inside a bucket)
    for (int a = lane; a < cnt; a += 32) {
      const int b = min((int)(__uint_as_float((unsigned)(keys[a] >> 32)) * bscale), NB - 1);
      grp[hist[b] + atomicAdd(fill + b, 1)] = (unsigned short)a;
    }
    __syncwarp();
    // rank of every key inside its bucket -> rk[arrival position] = rank in ascending (dist, index) order
    for (int s = lane; s < cnt; s += 32) {
      const int a = grp[s];
      const unsigned long long ka = keys[a];
      const int b = min((int)(__uint_as_float((unsigned)(ka >> 32)) * bscale), NB - 1);
      const int lo = hist[b], hi = hist[b + 1];
      int rank = lo;
      for (int t = lo; t < hi; t++) rank += (keys[grp[t]] < ka);
      rk[a] = (unsigned short)rank;
    }
    __syncwarp();
    // keys / grp are dead: permute the coordinates into sorted order
    for (int a = lane; a < cnt; a += 32) {
      const int r = rk[a];
      sxy[r] = pc[a];
      sxy[cap + r] = pc[cap + a];
      sz[r] = pc[2 * cap + a];
    }
    __syncwarp();
    // computeMeanAndCovarianceMatrix (float32, single pass, sorted order): lanes 0..8 own accu[0..8]
    const int ia = (lane == 3 || lane == 4 || lane == 7) ? 1 : ((lane == 5 || lane == 8) ? 2 : 0);
    const int ib = (lane == 1 || lane == 3) ? 1 : ((lane == 2 || lane == 4 || lane == 5) ? 2 : (lane == 0 ? 0 : -1));
    float acc = 0.0f;
    if (lane < 9) {
      // one loop for all nine accumulators: lanes 6..8 (plain sums) multiply by 1.0f, which is exact. Strictly
      // ascending k; every product is rounded before it is added (-fmad=false): the reference's arithmetic.
      const float *pa = ia == 2 ? sz : sxy + (size_t)ia * cap;
      const float *pb = ib == 2 ? sz : sxy + (size_t)max(ib, 0) * cap;
      const bool prod = ib >= 0;
      int k = 0;
      for (; k + 4 <= cnt; k += 4) {
        const float4 a4 = *reinterpret_cast<const float4 *>(pa + k);
        float4 b4 = make_float4(1.0f, 1.0f, 1.0f, 1.0f);
        if (prod) b4 = *reinterpret_cast<const float4 *>(pb + k);
        acc += a4.x * b4.x;
        acc += a4.y * b4.y;
        acc += a4.z * b4.z;
        acc += a4.w * b4.w;
      }
      for (; k < cnt; k++) acc += pa[k] * (prod ? pb[k] : 1.0f);
    }
    const float fc = (float)cnt;
    acc = acc / fc;
    float a9[9];
#pragma unroll
    for (int k = 0; k < 9; k++) a9[k] = __shfl_sync(0xffffffffu, acc, k);
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
    if (lane != 0) return;
    pcl_eigen33_smallest(cov, n);
    // flipNormalTowardsViewpoint, float32, view point of the first camera that sees the point
    const int camera = __ffs((unsigned)camm) - 1;
    const float vx = (float)P.vp[camera][0] - q[0], vy = (float)P.vp[camera][1] - q[1], vz = (float)P.vp[camera][2] - q[2];
    const float cos_theta = vx * n[0] + vy * n[1] + vz * n[2];
    if (cos_theta < 0) {
      n[0] *= -1;
      n[1] *= -1;
      n[2] *= -1;
    }
  }
  if (lane != 0) return;
  double nd[3] = {(double)n[0], (double)n[1], (double)n[2]};
  bool needs_reverse = true;
  for (int j = 0; j < P.K; j++)
    if ((camm >> j) & 1) {
      const double d0 = (double)q[0] - P.vp[j][0], d1 = (double)q[1] - P.vp[j][1], d2 = (double)q[2] - P.vp[j][2];
      if (nd[0] * d0 + nd[1] * d1 + nd[2] * d2 < 0) {
        needs_reverse = false;
        break;
      }
    }
  if (needs_reverse) {
    nd[0] *= -1.0;
    nd[1] *= -1.0;
    nd[2] *= -1.0;
  }
  out[0] = nd[0];
  out[1] = nd[1];
  out[2] = nd[2];
}

__global__ void k_cam_expand(const uint8_t *cam, int N, int K, int *out) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N) return;
  for (int k = 0; k < K; k++) out[(size_t)i * K + k] = (cam[i] >> k) & 1;
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

// GPDB_TRACE=1: host wall-clock per sub-step (each followed by a stream sync) on stderr — development aid
struct PreTrace {
  bool on;
  cudaStream_t st;
  std::chrono::steady_clock::time_point t0;
  explicit PreTrace(cudaStream_t s) : on(getenv("GPDB_TRACE") != nullptr), st(s) { if (on) { cudaStreamSynchronize(st); t0 = std::chrono::steady_clock::now(); } }
  void mark(const char *what) {
    if (!on) return;
    cudaStreamSynchronize(st);
    auto t1 = std::chrono::steady_clock::now();
    fprintf(stderr, "[gpdb trace] %-28s %9.3f ms\n", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
    t0 = t1;
  }
};

// bounds of a device point array (used by the grid build when the cloud never existed on the host)
int pre_bounds(gpdb_ctx *ctx, const float *d_xyz, int n, int *d_bounds, float lo[3], float hi[3]) {
  const int init[6] = {INT_MAX, INT_MAX, INT_MAX, INT_MIN, INT_MIN, INT_MIN};
  CUDA_TRY(cudaMemcpyAsync(d_bounds, init, sizeof(init), cudaMemcpyHostToDevice, ctx->stream));
  k_bounds<<<std::min((n + 255) / 256, ctx->sm_count * 8), 256, 0, ctx->stream>>>(d_xyz, n, d_bounds);
  LAUNCH_CHECK();
  int b[6];
  CUDA_TRY(cudaMemcpyAsync(b, d_bounds, sizeof(b), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  for (int a = 0; a < 3; a++) {
    lo[a] = ord2f(b[a]);
    hi[a] = ord2f(b[3 + a]);
  }
  return GPDB_OK;
}

// Normal estimation over the installed cloud (ctx->cloud, grid built): writes ctx->d_nrm.
int pre_normals(gpdb_ctx *ctx, double radius) {
  const int N = ctx->N;
  const float r2 = (float)(radius * radius);
  const float rf = (float)radius * 1.0001f + 1e-6f;
  int *ovf = (int *)gpdb_scratch(ctx, 2, sizeof(int) * ((size_t)N + 1));
  if (!ovf) return GPDB_ERR_CUDA;
  int *ovf_count = ovf + N;
  CUDA_TRY(cudaMemsetAsync(ovf_count, 0, sizeof(int), ctx->stream));
  const size_t sm1 = (size_t)NRM_WARPS * NRM_CAP1 * NRM_BYTES_PER, sm2 = (size_t)NRM_CAP2 * NRM_BYTES_PER;
  CUDA_TRY(cudaFuncSetAttribute(k_normals<NRM_WARPS, NRM_NB1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm1));
  CUDA_TRY(cudaFuncSetAttribute(k_normals<1, NRM_NB2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)sm2));
  k_normals<NRM_WARPS, NRM_NB1><<<(N + NRM_WARPS - 1) / NRM_WARPS, NRM_WARPS * 32, sm1, ctx->stream>>>(
      ctx->dp, ctx->cloud, N, r2, rf, NRM_CAP1, ctx->d_nrm, ovf, ovf_count, 0, ctx->d_err);
  LAUNCH_CHECK();
  int h_ovf = 0;
  CUDA_TRY(cudaMemcpyAsync(&h_ovf, ovf_count, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  if (h_ovf > 0) {
    k_normals<1, NRM_NB2><<<h_ovf, 32, sm2, ctx->stream>>>(ctx->dp, ctx->cloud, N, r2, rf, NRM_CAP2, ctx->d_nrm, ovf, ovf_count, 1,
                                                  ctx->d_err);
    LAUNCH_CHECK();
    int e4 = 0;
    CUDA_TRY(cudaMemcpyAsync(&e4, ctx->d_err + 4, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (e4) {
      CUDA_TRY(cudaMemsetAsync(ctx->d_err + 4, 0, sizeof(int), ctx->stream));
      gpdb_set_error(ctx, GPDB_ERR_CAPACITY, "normal estimation: %d points have more than %d neighbours within normals_radius",
                     e4, NRM_CAP2);
      return GPDB_ERR_CAPACITY;
    }
  }
  return GPDB_OK;
}

// Filter + voxelise the raw device arrays into the context's cloud arrays (ctx->d_xyz / d_cam / d_nrm / d_src,
// reserved here once the output size is known). d_nrm_raw may be null.
int pre_filter_voxelize(gpdb_ctx *ctx, const float *d_xyz_raw, const uint8_t *d_cam_raw, const double *d_nrm_raw, int M,
                        const gpdb_preprocess_params &pp, int *n_out, cudaEvent_t ev_filter_done) {
  *n_out = 0;
  const int tb = 256;
  PreTrace tr(ctx->stream);
  // ---- removeNans + filterWorkspace
  double *d_ws = (double *)gpdb_scratch(ctx, 4, sizeof(double) * 6 + sizeof(int) * 8);
  if (!d_ws) return GPDB_ERR_CUDA;
  int *d_bounds = (int *)(d_ws + 6);
  int *d_verr = d_bounds + 6;
  CUDA_TRY(cudaMemcpyAsync(d_ws, pp.workspace, sizeof(double) * 6, cudaMemcpyHostToDevice, ctx->stream));
  CUDA_TRY(cudaMemsetAsync(d_verr, 0, sizeof(int), ctx->stream));
  int *flag = (int *)gpdb_scratch(ctx, 5, sizeof(int) * (size_t)M * 3 + sizeof(float) * 3 * (size_t)M);
  if (!flag) return GPDB_ERR_CUDA;
  int *pos = flag + M, *keep = pos + M;
  float *xyz1 = (float *)(keep + M);
  k_pre_flag<<<(M + tb - 1) / tb, tb, 0, ctx->stream>>>(d_xyz_raw, M, d_ws, flag);
  LAUNCH_CHECK();
  size_t tmp_bytes = 0;
  cub::DeviceScan::ExclusiveSum(nullptr, tmp_bytes, flag, pos, M, ctx->stream);
  void *tmp = gpdb_scratch(ctx, 1, tmp_bytes);
  if (!tmp) return GPDB_ERR_CUDA;
  CUDA_TRY(cub::DeviceScan::ExclusiveSum(tmp, tmp_bytes, flag, pos, M, ctx->stream));
  ctx->launches += 2;
  k_pre_compact<<<(M + tb - 1) / tb, tb, 0, ctx->stream>>>(d_xyz_raw, flag, pos, M, keep, xyz1);
  LAUNCH_CHECK();
  int last[2];
  CUDA_TRY(cudaMemcpyAsync(&last[0], flag + M - 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  CUDA_TRY(cudaMemcpyAsync(&last[1], pos + M - 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
  cudaEventRecord(ev_filter_done, ctx->stream);
  CUDA_TRY(cudaStreamSynchronize(ctx->stream));
  const int M1 = last[0] + last[1];
  tr.mark("filter + compact");
  if (M1 == 0) return GPDB_OK;

  int U = M1;
  if (!pp.voxelize) {
    int rc = gpdb_cloud_reserve(ctx, (size_t)U);
    if (rc != GPDB_OK) return rc;
    CUDA_TRY(cudaMemcpyAsync(ctx->d_xyz, xyz1, sizeof(float) * 3 * (size_t)U, cudaMemcpyDeviceToDevice, ctx->stream));
    k_gather_plain<<<(U + tb - 1) / tb, tb, 0, ctx->stream>>>(keep, U, d_cam_raw, d_nrm_raw, ctx->d_cam, ctx->d_nrm, ctx->d_src);
    LAUNCH_CHECK();
  } else {
    const float cell = (float)pp.voxel_size;  // voxelizeCloud(float cell_size)
    float lo[3], hi[3];
    int rc = pre_bounds(ctx, xyz1, M1, d_bounds, lo, hi);
    if (rc != GPDB_OK) return rc;
    tr.mark("bounds");
    // sort buffers: keys x2 (8 B), vals x2 (4 B), head + gid (4 B each)
    unsigned long long *keys = (unsigned long long *)gpdb_scratch(ctx, 6, (size_t)M1 * (16 + 8 + 8 + 24));
    if (!keys) return GPDB_ERR_CUDA;
    unsigned long long *keys2 = keys + M1;
    int *vals = (int *)(keys2 + M1), *vals2 = vals + M1, *head = vals2 + M1, *gid = head + M1;
    int *gfirst = gid + M1, *gbegin = gfirst + M1, *gord_v = gbegin + M1, *gord_v2 = gord_v + M1;
    unsigned *gord_k = (unsigned *)(gord_v2 + M1), *gord_k2 = gord_k + M1;
    k_vox_keys<<<(M1 + tb - 1) / tb, tb, 0, ctx->stream>>>(xyz1, M1, d_bounds, cell, keys, vals, d_verr);
    LAUNCH_CHECK();
    tr.mark("scratch + voxel keys");
    size_t t1 = 0, t2 = 0, t3 = 0;
    cub::DeviceRadixSort::SortPairs(nullptr, t1, keys, keys2, vals, vals2, M1, 0, 63, ctx->stream);
    cub::DeviceScan::InclusiveSum(nullptr, t2, head, gid, M1, ctx->stream);
    cub::DeviceRadixSort::SortPairs(nullptr, t3, gord_k, gord_k2, gord_v, gord_v2, M1, 0, 31, ctx->stream);
    tmp = gpdb_scratch(ctx, 1, std::max(t1, std::max(t2, t3)));
    if (!tmp) return GPDB_ERR_CUDA;
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(tmp, t1, keys, keys2, vals, vals2, M1, 0, 63, ctx->stream));
    ctx->launches += 9;
    tr.mark("radix sort 63 bit");
    k_vox_heads<<<(M1 + tb - 1) / tb, tb, 0, ctx->stream>>>(keys2, M1, head);
    LAUNCH_CHECK();
    CUDA_TRY(cub::DeviceScan::InclusiveSum(tmp, t2, head, gid, M1, ctx->stream));
    ctx->launches += 2;
    k_vox_groups<<<(M1 + tb - 1) / tb, tb, 0, ctx->stream>>>(head, gid, vals2, M1, gfirst, gbegin, gord_k, gord_v);
    LAUNCH_CHECK();
    int verr = 0;
    CUDA_TRY(cudaMemcpyAsync(&U, gid + M1 - 1, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaMemcpyAsync(&verr, d_verr, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    tr.mark("heads + scan + groups");
    if (verr) {
      gpdb_set_error(ctx, GPDB_ERR_INVALID, "voxelisation: %d points fall outside the 2^21-voxel range (voxel_size %g too small "
                     "for the cloud extent)", verr, (double)cell);
      return GPDB_ERR_INVALID;
    }
    CUDA_TRY(cub::DeviceRadixSort::SortPairs(tmp, t3, gord_k, gord_k2, gord_v, gord_v2, U, 0, 31, ctx->stream));
    ctx->launches += 5;
    tr.mark("group order sort");
    rc = gpdb_cloud_reserve(ctx, (size_t)U);
    if (rc != GPDB_OK) return rc;
    k_vox_emit<<<(U + tb - 1) / tb, tb, 0, ctx->stream>>>(gord_v2, U, M1, gfirst, gbegin, vals2, keys2, keep, xyz1, d_bounds, cell,
                                                          d_cam_raw, d_nrm_raw, ctx->d_xyz, ctx->d_cam, ctx->d_nrm, ctx->d_src);
    LAUNCH_CHECK();
    tr.mark("reserve + emit");
  }
  *n_out = U;
  return GPDB_OK;
}

int pre_cam_expand(gpdb_ctx *ctx, int *d_out) {
  k_cam_expand<<<(ctx->N + 255) / 256, 256, 0, ctx->stream>>>(ctx->d_cam, ctx->N, ctx->K, d_out);
  LAUNCH_CHECK();
  return GPDB_OK;
}
