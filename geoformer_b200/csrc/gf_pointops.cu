// pointnet2._ext operators other than FPS: gather / group (+grads), ball_query, three_nn,
// three_interpolate (+grad).  Reference: lib/pointnet2/_ext_src/src/{sampling,group_points,
// ball_query,interpolate}_gpu.cu.  The reference launches ONE block per batch element (so one SM
// of 148 does all the work when B == 1, which is how GeoFormer calls it); here every operator is
// flattened over all of its output elements so the grid fills the machine.
#include "gf_common.cuh"

namespace gf {

static inline int grid_for(long long total, int block) {
  long long g = (total + block - 1) / block;
  long long cap = (long long)num_sms() * 32;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

// ---- gather_points (sampling_gpu.cu:11-23): out[b,c,j] = points[b,c,idx[b,j]] ------------------
__global__ void gather_points_kernel(const float *__restrict__ points, const int *__restrict__ idx, int B, int C,
                                     int N, int m, float *__restrict__ out) {
  long long total = (long long)B * C * m;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    int j = (int)(e % m);
    long long bc = e / m;
    int b = (int)(bc / C);
    int a = idx[(long long)b * m + j];
    out[e] = points[bc * N + a];
  }
}

// ---- gather_points_grad (sampling_gpu.cu:37-50) -------------------------------------------------
__global__ void gather_points_grad_kernel(const float *__restrict__ grad_out, const int *__restrict__ idx, int B,
                                          int C, int N, int m, float *__restrict__ grad_points) {
  long long total = (long long)B * C * m;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    int j = (int)(e % m);
    long long bc = e / m;
    int b = (int)(bc / C);
    int a = idx[(long long)b * m + j];
    atomicAdd(grad_points + bc * N + a, grad_out[e]);
  }
}

// ---- group_points (group_points_gpu.cu:11-31): out[b,c,j,s] = points[b,c,idx[b,j,s]] ----------
// One thread per (b, j, s): the index is read once and reused for all C channels; for a fixed
// channel consecutive threads write consecutive addresses.
__global__ void group_points_kernel(const float *__restrict__ points, const int *__restrict__ idx, int B, int C,
                                    int N, long long M /* np*ns */, float *__restrict__ out) {
  long long total = (long long)B * M;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    long long b = e / M, r = e - b * M;
    int a = idx[e];
    const float *p = points + b * C * N + a;
    float *o = out + b * C * M + r;
    for (int c = 0; c < C; ++c) o[(long long)c * M] = __ldg(p + (long long)c * N);
  }
}

// ---- group_points_grad (group_points_gpu.cu:46-67) ----------------------------------------------
__global__ void group_points_grad_kernel(const float *__restrict__ grad_out, const int *__restrict__ idx, int B,
                                         int C, int N, long long M, float *__restrict__ grad_points) {
  long long total = (long long)B * M;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    long long b = e / M, r = e - b * M;
    int a = idx[e];
    float *g = grad_points + b * C * N + a;
    const float *o = grad_out + b * C * M + r;
    for (int c = 0; c < C; ++c) atomicAdd(g + (long long)c * N, o[(long long)c * M]);
  }
}

// ---- ball_query (ball_query_gpu.cu:12-47) -------------------------------------------------------
// The point cloud streams through shared memory in tiles shared by the 16 warps of a CTA.  FOUR warps work
// on one centre: each takes a quarter of the tile, votes its hits (ballot words kept in registers), the four
// hit counts meet in shared memory, and every warp then writes its hits behind those of the quarters before
// it -- so the row still holds the hits in ascending index order, truncated at nsample, the tail padded with
// the first hit, zeros if there is none (the reference's result).  One warp per centre left only ~14 warps
// per SM (2048 centres), each a long dependent chain of load -> distance -> vote steps.
constexpr int BQ_WPC = 4;        // warps per centre
constexpr int BQ_CENTRES = 4;    // centres per CTA (16 warps: two CTAs per SM at 64 registers)
constexpr int BQ_WARPS = BQ_WPC * BQ_CENTRES;
constexpr int BQ_TILE = 2048;
constexpr int BQ_PART = BQ_TILE / BQ_WPC;  // points of a tile per warp
constexpr int BQ_STEPS = BQ_PART / 32;

__global__ void __launch_bounds__(BQ_WARPS * 32)
    ball_query_kernel(const float *__restrict__ new_xyz, const float *__restrict__ xyz, int B, int N, int m,
                      float radius, int nsample, int *__restrict__ idx) {
#define GF_BQ_SCENE const float *P = xyz + (long long)b * N * 3;
#include "gf_ball_query_body.cuh"
#undef GF_BQ_SCENE
}

// A ragged batch: scene b is rows [off[b], off[b+1]) of the flat (sum N,3) array; one launch per 32 scenes.
constexpr int BQ_BATCH_MAX = 32;
struct BqOffsets {
  int off[BQ_BATCH_MAX + 1];
};

__global__ void __launch_bounds__(BQ_WARPS * 32)
    ball_query_batch_kernel(const float *__restrict__ new_xyz, const float *__restrict__ xyz,
                            const __grid_constant__ BqOffsets sc, int B, int m, float radius, int nsample,
                            int *__restrict__ idx) {
#define GF_BQ_SCENE                                   \
  const float *P = xyz + (long long)sc.off[b] * 3; \
  const int N = sc.off[b + 1] - sc.off[b];
#include "gf_ball_query_body.cuh"
#undef GF_BQ_SCENE
}

// ---- three_nn (interpolate_gpu.cu:12-62) --------------------------------------------------------
constexpr int TNN_TILE = 1024;
__global__ void __launch_bounds__(256)
    three_nn_kernel(const float *__restrict__ unknown, const float *__restrict__ known, int B, int n, int m,
                    float *__restrict__ dist2, int *__restrict__ idx) {
  __shared__ float sx[TNN_TILE], sy[TNN_TILE], sz[TNN_TILE];
  const int blocks_per_batch = (n + blockDim.x - 1) / blockDim.x;
  for (int g = blockIdx.x; g < B * blocks_per_batch; g += gridDim.x) {
    const int b = g / blocks_per_batch;
    const int j = (g - b * blocks_per_batch) * blockDim.x + threadIdx.x;
    const bool live = j < n;
    float ux = 0.f, uy = 0.f, uz = 0.f;
    if (live) {
      const float *u = unknown + ((long long)b * n + j) * 3;
      ux = u[0], uy = u[1], uz = u[2];
    }
    // the reference keeps doubles initialised to 1e40 and compares a float against them (:38-54);
    // that is the float comparison with +inf, and (float)1e40 == +inf on write-back (:56-58).
    float best1 = __int_as_float(0x7f800000), best2 = best1, best3 = best1;
    int b1 = 0, b2 = 0, b3 = 0;
    const float *K = known + (long long)b * m * 3;
    for (int base = 0; base < m; base += TNN_TILE) {
      const int tn = min(TNN_TILE, m - base);
      __syncthreads();
      for (int t = threadIdx.x; t < tn * 3; t += blockDim.x) {
        float v = __ldg(K + (long long)base * 3 + t);
        int pt = t / 3, ax = t - pt * 3;
        (ax == 0 ? sx : ax == 1 ? sy : sz)[pt] = v;
      }
      __syncthreads();
      if (live) {
        for (int t = 0; t < tn; ++t) {
          float d = sq3(ux - sx[t], uy - sy[t], uz - sz[t]);
          int k = base + t;
          if (d < best1) {
            best3 = best2; b3 = b2; best2 = best1; b2 = b1; best1 = d; b1 = k;
          } else if (d < best2) {
            best3 = best2; b3 = b2; best2 = d; b2 = k;
          } else if (d < best3) {
            best3 = d; b3 = k;
          }
        }
      }
    }
    if (live) {
      long long o = ((long long)b * n + j) * 3;
      dist2[o + 0] = best1; dist2[o + 1] = best2; dist2[o + 2] = best3;
      idx[o + 0] = b1; idx[o + 1] = b2; idx[o + 2] = b3;
    }
  }
}

// ---- three_interpolate (interpolate_gpu.cu:75-104) ----------------------------------------------
// nvcc contracts p1*w1 + p2*w2 + p3*w3 of the reference into FMUL(p2,w2); FFMA(p1,w1,.); FFMA(p3,w3,.)
__global__ void three_interpolate_kernel(const float *__restrict__ points, const int *__restrict__ idx,
                                         const float *__restrict__ weight, int B, int C, int m, int n,
                                         float *__restrict__ out) {
  long long total = (long long)B * C * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    int j = (int)(e % n);
    long long bc = e / n;
    long long b = bc / C;
    long long o = (b * n + j) * 3;
    const float *P = points + bc * m;
    float w1 = weight[o], w2 = weight[o + 1], w3 = weight[o + 2];
    out[e] = __fmaf_rn(__ldg(P + idx[o + 2]), w3, __fmaf_rn(__ldg(P + idx[o]), w1, __fmul_rn(__ldg(P + idx[o + 1]), w2)));
  }
}

// ---- three_interpolate_grad (interpolate_gpu.cu:119-146) ----------------------------------------
__global__ void three_interpolate_grad_kernel(const float *__restrict__ grad_out, const int *__restrict__ idx,
                                              const float *__restrict__ weight, int B, int C, int n, int m,
                                              float *__restrict__ grad_points) {
  long long total = (long long)B * C * n;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    int j = (int)(e % n);
    long long bc = e / n;
    long long b = bc / C;
    long long o = (b * n + j) * 3;
    float g = grad_out[e];
    float *G = grad_points + bc * m;
    atomicAdd(G + idx[o], __fmul_rn(g, weight[o]));
    atomicAdd(G + idx[o + 1], __fmul_rn(g, weight[o + 1]));
    atomicAdd(G + idx[o + 2], __fmul_rn(g, weight[o + 2]));
  }
}

}  // namespace gf

using namespace gf;

extern "C" int gf_gather_points(const float *points, const int *idx, int B, int C, int N, int m, float *out,
                                void *stream) {
  GF_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && m >= 0, "gather_points: negative size");
  long long total = (long long)B * C * m;
  if (total == 0) return GF_OK;
  GF_CHECK_ARG(points && idx && out, "gather_points: null pointer");
  gather_points_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(points, idx, B, C, N, m, out);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_gather_points_grad(const float *grad_out, const int *idx, int B, int C, int N, int m,
                                     float *grad_points, void *stream) {
  GF_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && m >= 0, "gather_points_grad: negative size");
  if ((long long)B * C * N == 0) return GF_OK;
  GF_CHECK_ARG(grad_points, "gather_points_grad: null pointer");
  GF_CUDA(cudaMemsetAsync(grad_points, 0, sizeof(float) * (size_t)B * C * N, (cudaStream_t)stream));
  long long total = (long long)B * C * m;
  if (total == 0) return GF_OK;
  GF_CHECK_ARG(grad_out && idx, "gather_points_grad: null pointer");
  gather_points_grad_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(grad_out, idx, B, C, N, m,
                                                                                   grad_points);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_group_points(const float *points, const int *idx, int B, int C, int N, int npoints, int nsample,
                               float *out, void *stream) {
  GF_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && npoints >= 0 && nsample >= 0, "group_points: negative size");
  long long M = (long long)npoints * nsample;
  if ((long long)B * M == 0 || C == 0) return GF_OK;
  GF_CHECK_ARG(points && idx && out, "group_points: null pointer");
  group_points_kernel<<<grid_for((long long)B * M, 256), 256, 0, (cudaStream_t)stream>>>(points, idx, B, C, N, M, out);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_group_points_grad(const float *grad_out, const int *idx, int B, int C, int N, int npoints,
                                    int nsample, float *grad_points, void *stream) {
  GF_CHECK_ARG(B >= 0 && C >= 0 && N >= 0 && npoints >= 0 && nsample >= 0, "group_points_grad: negative size");
  if ((long long)B * C * N == 0) return GF_OK;
  GF_CHECK_ARG(grad_points, "group_points_grad: null pointer");
  GF_CUDA(cudaMemsetAsync(grad_points, 0, sizeof(float) * (size_t)B * C * N, (cudaStream_t)stream));
  long long M = (long long)npoints * nsample;
  if ((long long)B * M == 0) return GF_OK;
  GF_CHECK_ARG(grad_out && idx, "group_points_grad: null pointer");
  group_points_grad_kernel<<<grid_for((long long)B * M, 256), 256, 0, (cudaStream_t)stream>>>(grad_out, idx, B, C, N,
                                                                                             M, grad_points);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_ball_query(const float *new_xyz, const float *xyz, int B, int N, int m, float radius, int nsample,
                             int *idx, void *stream) {
  GF_CHECK_ARG(B >= 0 && N >= 0 && m >= 0 && nsample >= 0, "ball_query: negative size");
  if ((long long)B * m * nsample == 0) return GF_OK;
  GF_CHECK_ARG(new_xyz && idx && (xyz || N == 0), "ball_query: null pointer");
  long long groups = (long long)B * ((m + BQ_CENTRES - 1) / BQ_CENTRES);
  int grid = (int)(groups < (long long)num_sms() * 8 ? groups : (long long)num_sms() * 8);
  ball_query_kernel<<<grid, BQ_WARPS * 32, 0, (cudaStream_t)stream>>>(new_xyz, xyz, B, N, m, radius, nsample, idx);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_ball_query_batch(const float *new_xyz, const float *xyz, const int *offsets, int B, int m,
                                   float radius, int nsample, int *idx, void *stream) {
  GF_CHECK_ARG(B >= 0 && m >= 0 && nsample >= 0, "ball_query_batch: negative size");
  if ((long long)B * m * nsample == 0) return GF_OK;
  GF_CHECK_ARG(offsets && new_xyz && idx, "ball_query_batch: null pointer");
  GF_CHECK_ARG(offsets[0] == 0, "ball_query_batch: offsets[0] = %d, not 0", offsets[0]);
  for (int b = 0; b < B; ++b)
    GF_CHECK_ARG(offsets[b + 1] >= offsets[b], "ball_query_batch: offsets fall at scene %d", b);
  GF_CHECK_ARG(xyz || offsets[B] == 0, "ball_query_batch: null xyz");
  for (int b0 = 0; b0 < B; b0 += BQ_BATCH_MAX) {  // one launch per 32 scenes: the offsets travel as a kernel parameter
    const int nb = B - b0 < BQ_BATCH_MAX ? B - b0 : BQ_BATCH_MAX;
    BqOffsets sc;
    for (int b = 0; b <= nb; ++b) sc.off[b] = offsets[b0 + b];
    long long groups = (long long)nb * ((m + BQ_CENTRES - 1) / BQ_CENTRES);
    int grid = (int)(groups < (long long)num_sms() * 8 ? groups : (long long)num_sms() * 8);
    ball_query_batch_kernel<<<grid, BQ_WARPS * 32, 0, (cudaStream_t)stream>>>(
        new_xyz + (size_t)b0 * m * 3, xyz, sc, nb, m, radius, nsample, idx + (size_t)b0 * m * nsample);
    GF_LAUNCHED();
  }
  return GF_OK;
}

extern "C" int gf_three_nn(const float *unknown, const float *known, int B, int n, int m, float *dist2, int *idx,
                           void *stream) {
  GF_CHECK_ARG(B >= 0 && n >= 0 && m >= 0, "three_nn: negative size");
  if ((long long)B * n == 0) return GF_OK;
  GF_CHECK_ARG(unknown && dist2 && idx && (known || m == 0), "three_nn: null pointer");
  long long blocks = (long long)B * ((n + 255) / 256);
  int grid = (int)(blocks < (long long)num_sms() * 8 ? blocks : (long long)num_sms() * 8);
  three_nn_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(unknown, known, B, n, m, dist2, idx);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_three_interpolate(const float *points, const int *idx, const float *weight, int B, int C, int m,
                                    int n, float *out, void *stream) {
  GF_CHECK_ARG(B >= 0 && C >= 0 && m >= 0 && n >= 0, "three_interpolate: negative size");
  long long total = (long long)B * C * n;
  if (total == 0) return GF_OK;
  GF_CHECK_ARG(points && idx && weight && out, "three_interpolate: null pointer");
  three_interpolate_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(points, idx, weight, B, C, m, n, out);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_three_interpolate_grad(const float *grad_out, const int *idx, const float *weight, int B, int C,
                                         int n, int m, float *grad_points, void *stream) {
  GF_CHECK_ARG(B >= 0 && C >= 0 && m >= 0 && n >= 0, "three_interpolate_grad: negative size");
  if ((long long)B * C * m == 0) return GF_OK;
  GF_CHECK_ARG(grad_points, "three_interpolate_grad: null pointer");
  GF_CUDA(cudaMemsetAsync(grad_points, 0, sizeof(float) * (size_t)B * C * m, (cudaStream_t)stream));
  long long total = (long long)B * C * n;
  if (total == 0) return GF_OK;
  GF_CHECK_ARG(grad_out && idx && weight, "three_interpolate_grad: null pointer");
  three_interpolate_grad_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)stream>>>(grad_out, idx, weight, B, C,
                                                                                       n, m, grad_points);
  GF_LAUNCHED();
  return GF_OK;
}
