// Training form of the fused set aggregator (gf_aggregate.cu): batch norm with batch statistics and the backward of
// group -> SharedMLP -> pool, for sm_100a.
//
// Layer l computes z_l = W_l h_{l-1} (h_{-1} = the grouped input), y_l = scale_l z_l + shift_l, h_l = relu(y_l), with
// the forward kernel's own expressions (agg_dot / agg_act below equal group_mlp_pool_kernel's loop body operation for
// operation), so every recomputed activation, ReLU mask and argmax is bit-identical to the forward's.  A layer is
// FIXED (scale and shift given: batch norm with running statistics folded, or no batch norm) or BATCH (batch norm
// with the statistics of this call's input).
//
// Forward with batch statistics: one statistics pass per BATCH layer l recomputes the layers below with their final
// scale and shift and accumulates sum z and sum z^2 per channel in fp64 (lane = channel); warps are combined into one
// partial row per CTA in warp order and a finishing kernel sums the rows in CTA order into mean, biased variance,
// invstd, scale and shift.  The output pass is gf_group_mlp_pool, unchanged, reading those device-resident constants.
//
// Backward: L + 1 passes p = L .. 0.  Pass p recomputes the forward of each sample, backpropagates from the pool down
// to layer p with the per-channel sums of the earlier passes, accumulates dW_p and dbias_p, collects sum dy and
// sum dy * xhat of layer p - 1 (dbeta, dgamma, and the batch-norm terms of pass p - 1), and pass 0 writes the input
// gradient of every (centre, sample, feature channel).  W^T dz is a fixed-order transposing warp reduction, so only
// the rows of W are held.  The feature gradient sums those input gradients per point in (b, j, s) order through a
// stable inverse of idx (count, scan, placement, per-point sort).  No float atomics: two calls give bitwise-equal
// results on the same device.
#include "gf_common.cuh"

namespace gf {

constexpr int AGT_MAX_LAYERS = 4;
constexpr int AGT_W = 32;
constexpr int AGT_THREADS = 256;
constexpr int AGT_WARPS = AGT_THREADS / 32;
constexpr int AGT_CONST = 5 * AGT_W;        // per layer: scale, shift, mean of z, invstd, biased variance
constexpr int AGT_WROW = AGT_W * AGT_W + AGT_W;  // per CTA: dW (32 x 32) and dbias of one layer
constexpr int AGT_SCAN_THREADS = 1024;

struct AgtArgs {
  const float *xyz, *new_xyz, *features;
  const int *idx;
  int B, N, m, ns, C;
  float radius;
  int normalize, use_xyz, n_layers, pool_avg;
  int width[AGT_MAX_LAYERS + 1];
  const float *w[AGT_MAX_LAYERS];
  int batch[AGT_MAX_LAYERS];  // 1: batch norm with batch statistics
  float *consts;              // (L, 5, 32)
  // statistics pass
  double *spart;              // (grid, 2, 32)
  // backward
  const float *dout;          // (B, width[L], m)
  int *arg;                   // (B*m, 32) first maximal sample of every output channel
  const double *S;            // (L, 2, 32) sum dy, sum dy * xhat
  float *wpart;               // (grid, AGT_WROW)
  double *Spart;              // (grid, 2, 32)
  float *gx;                  // (B*m*ns, C) input gradient of the feature channels, or null: not wanted
};

// lane i: input channel i of sample p -- group_mlp_pool_kernel's expressions
__device__ __forceinline__ float agg_in(const AgtArgs &a, int b, int p, unsigned lane, float centre) {
  const int xoff = a.use_xyz ? 3 : 0, c_in = a.width[0];
  float x = 0.f;
  if (a.use_xyz && lane < 3u) {
    x = __fsub_rn(__ldg(a.xyz + ((size_t)b * a.N + p) * 3 + lane), centre);
    if (a.normalize) x = __fdiv_rn(x, a.radius);
  } else if ((int)lane >= xoff && (int)lane < c_in) {
    x = __ldg(a.features + ((size_t)b * a.C + (lane - xoff)) * a.N + p);
  }
  return x;
}

__device__ __forceinline__ float agg_dot(const float (&w)[AGT_W], float x) {
  float accv = 0.f;
#pragma unroll
  for (int i = 0; i < AGT_W; ++i) accv = fmaf(w[i], __shfl_sync(0xffffffffu, x, i), accv);
  return accv;
}

__device__ __forceinline__ float agg_act(float z, float sc, float sh) { return fmaxf(fmaf(z, sc, sh), 0.f); }

__device__ __forceinline__ void agg_load_row(const AgtArgs &a, int l, unsigned lane, float (&w)[AGT_W]) {
  const bool live = (int)lane < a.width[l + 1];
#pragma unroll
  for (int i = 0; i < AGT_W; ++i) w[i] = live && i < a.width[l] ? __ldg(a.w[l] + lane * a.width[l] + i) : 0.f;
}

// sum of v[i] over the 32 lanes for all 32 i in 31 shuffles: lane l returns the sum of v[l].  Fixed order.
__device__ __forceinline__ float agg_warp_reduce32(float (&v)[AGT_W], unsigned lane) {
#pragma unroll
  for (int o = 16; o >= 1; o >>= 1) {
    const bool up = (lane & (unsigned)o) != 0;
#pragma unroll
    for (int i = 0; i < o; ++i) {
      const float send = up ? v[i] : v[i + o], keep = up ? v[i + o] : v[i];
      v[i] = __fadd_rn(keep, __shfl_xor_sync(0xffffffffu, send, o));
    }
  }
  return v[0];
}

// ---- forward: statistics of layer K --------------------------------------------------------------------------
template <int K>
__global__ void __launch_bounds__(AGT_THREADS) agg_stats_kernel(const AgtArgs a) {
  __shared__ double red[AGT_WARPS][2][AGT_W];
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const int warps_per_grid = (gridDim.x * blockDim.x) >> 5;
  float w[K + 1][AGT_W], sc[K + 1], sh[K + 1];
#pragma unroll
  for (int l = 0; l <= K; ++l) {
    agg_load_row(a, l, lane, w[l]);
    sc[l] = a.consts[l * AGT_CONST + lane];
    sh[l] = a.consts[l * AGT_CONST + AGT_W + lane];
  }
  double s1 = 0.0, s2 = 0.0;
  for (int cj = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; cj < a.B * a.m; cj += warps_per_grid) {
    const int b = cj / a.m;
    const int *idx = a.idx + (size_t)cj * a.ns;
    const float centre = lane < 3u ? __ldg(a.new_xyz + (size_t)cj * 3 + lane) : 0.f;
    for (int s = 0; s < a.ns; ++s) {
      float x = agg_in(a, b, __ldg(idx + s), lane, centre);
#pragma unroll
      for (int l = 0; l < K; ++l) x = agg_act(agg_dot(w[l], x), sc[l], sh[l]);
      const float z = agg_dot(w[K], x);
      s1 += (double)z;
      s2 = fma((double)z, (double)z, s2);
    }
  }
  red[warp][0][lane] = s1;
  red[warp][1][lane] = s2;
  __syncthreads();
  if (threadIdx.x < 2 * AGT_W) {
    const int k = threadIdx.x >> 5, c = threadIdx.x & 31;
    double t = 0.0;
    for (int q = 0; q < AGT_WARPS; ++q) t += red[q][k][c];
    a.spart[(size_t)blockIdx.x * 2 * AGT_W + threadIdx.x] = t;
  }
}

// mean, biased variance, invstd, scale and shift of layer l from the CTAs' partial sums, in CTA order
__global__ void agg_stats_finish_kernel(const double *__restrict__ spart, int nparts, double n, int width,
                                        const float *__restrict__ gamma, const float *__restrict__ beta, float eps,
                                        float *__restrict__ cst) {
  const int c = threadIdx.x;
  if (c >= AGT_W) return;
  if (c >= width) {
#pragma unroll
    for (int r = 0; r < 5; ++r) cst[r * AGT_W + c] = 0.f;
    return;
  }
  double t1 = 0.0, t2 = 0.0;
  for (int q = 0; q < nparts; ++q) {
    t1 += spart[(size_t)q * 2 * AGT_W + c];
    t2 += spart[(size_t)q * 2 * AGT_W + AGT_W + c];
  }
  const double mean = t1 / n;
  double var = t2 / n - mean * mean;
  if (var < 0.0) var = 0.0;
  const double invstd = 1.0 / sqrt(var + (double)eps);
  const double sc = (double)gamma[c] * invstd;
  cst[c] = (float)sc;
  cst[AGT_W + c] = (float)((double)beta[c] - mean * sc);
  cst[2 * AGT_W + c] = (float)mean;
  cst[3 * AGT_W + c] = (float)invstd;
  cst[4 * AGT_W + c] = (float)var;
}

// ---- backward pass p -----------------------------------------------------------------------------------------
template <int L>
__global__ void __launch_bounds__(AGT_THREADS) agg_backward_kernel(const AgtArgs a, const int p) {
  __shared__ float sw[AGT_WARPS][AGT_WROW];
  __shared__ double ss[AGT_WARPS][2][AGT_W];
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  const int warps_per_grid = (gridDim.x * blockDim.x) >> 5;
  const double n = (double)a.B * a.m * a.ns;
  float w[L][AGT_W], sc[L], sh[L], mu[L], is[L], m1[L], m2[L];
  bool dense = a.pool_avg != 0;  // every sample carries gradient (else only the argmax samples of max pooling)
#pragma unroll
  for (int l = 0; l < L; ++l) {
    agg_load_row(a, l, lane, w[l]);
    const float *cst = a.consts + l * AGT_CONST;
    sc[l] = cst[lane], sh[l] = cst[AGT_W + lane], mu[l] = cst[2 * AGT_W + lane], is[l] = cst[3 * AGT_W + lane];
    const bool have = a.batch[l] && l >= p;  // the sums of layer l come from pass l + 1
    m1[l] = have ? (float)(a.S[l * 2 * AGT_W + lane] / n) : 0.f;
    m2[l] = have ? (float)(a.S[l * 2 * AGT_W + AGT_W + lane] / n) : 0.f;
    if (have) dense = true;
  }
  const int c_out = a.width[L], xoff = a.use_xyz ? 3 : 0;
  float dw[AGT_W];
#pragma unroll
  for (int i = 0; i < AGT_W; ++i) dw[i] = 0.f;
  float db = 0.f;
  double s1 = 0.0, s2 = 0.0;
  for (int cj = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; cj < a.B * a.m; cj += warps_per_grid) {
    const int b = cj / a.m, j = cj - b * a.m;
    const int *idx = a.idx + (size_t)cj * a.ns;
    const float centre = lane < 3u ? __ldg(a.new_xyz + (size_t)cj * 3 + lane) : 0.f;
    const float g = (int)lane < c_out ? __ldg(a.dout + ((size_t)b * c_out + lane) * a.m + j) : 0.f;
    int arg = -1;
    if (!a.pool_avg) {
      if (p == L) {  // first maximal sample in s order (max_pool2d's backward), stored for the later passes
        float best = -INFINITY;
        for (int s = 0; s < a.ns; ++s) {
          float x = agg_in(a, b, __ldg(idx + s), lane, centre);
#pragma unroll
          for (int l = 0; l < L; ++l) x = agg_act(agg_dot(w[l], x), sc[l], sh[l]);
          if (x > best) best = x, arg = s;
        }
        a.arg[(size_t)cj * AGT_W + lane] = arg;
      } else {
        arg = a.arg[(size_t)cj * AGT_W + lane];
      }
    }
    for (int s = 0; s < a.ns; ++s) {
      const bool hit = a.pool_avg || arg == s;
      if (!dense && !__any_sync(0xffffffffu, hit)) continue;  // warp-uniform
      const float xin = agg_in(a, b, __ldg(idx + s), lane, centre);
      float z[L], h[L];
      {
        float x = xin;
#pragma unroll
        for (int l = 0; l < L; ++l) {
          z[l] = agg_dot(w[l], x);
          h[l] = agg_act(z[l], sc[l], sh[l]);
          x = h[l];
        }
      }
      float dh = hit ? (a.pool_avg ? __fdiv_rn(g, (float)a.ns) : g) : 0.f;
#pragma unroll
      for (int l = L - 1; l >= 0; --l) {
        if (l < p - 1) break;
        const float dy = h[l] > 0.f ? dh : 0.f;  // ReLU passes where its output is > 0
        const float xh = __fmul_rn(__fsub_rn(z[l], mu[l]), is[l]);
        if (l == p - 1) {
          s1 += (double)dy;
          s2 = fma((double)dy, (double)xh, s2);
          break;
        }
        const float dz = a.batch[l] ? __fmul_rn(sc[l], __fsub_rn(__fsub_rn(dy, m1[l]), __fmul_rn(xh, m2[l])))
                                    : __fmul_rn(sc[l], dy);
        if (l == p) {
          const float prev = l == 0 ? xin : h[l > 0 ? l - 1 : 0];
#pragma unroll
          for (int i = 0; i < AGT_W; ++i) dw[i] = fmaf(dz, __shfl_sync(0xffffffffu, prev, i), dw[i]);
          db = __fadd_rn(db, dz);
        }
        float v[AGT_W];
#pragma unroll
        for (int i = 0; i < AGT_W; ++i) v[i] = __fmul_rn(w[l][i], dz);
        dh = agg_warp_reduce32(v, lane);  // (W_l^T dz)[lane]
        if (l == 0 && a.gx && (int)lane >= xoff && (int)lane < a.width[0])
          a.gx[((size_t)cj * a.ns + s) * a.C + (lane - xoff)] = dh;
      }
    }
  }
  // warps -> one partial row per CTA, in warp order
#pragma unroll
  for (int i = 0; i < AGT_W; ++i) sw[warp][lane * AGT_W + i] = dw[i];
  sw[warp][AGT_W * AGT_W + lane] = db;
  ss[warp][0][lane] = s1;
  ss[warp][1][lane] = s2;
  __syncthreads();
  for (int e = threadIdx.x; e < AGT_WROW; e += AGT_THREADS) {
    float t = 0.f;
    for (int q = 0; q < AGT_WARPS; ++q) t = __fadd_rn(t, sw[q][e]);
    a.wpart[(size_t)blockIdx.x * AGT_WROW + e] = t;
  }
  if (threadIdx.x < 2 * AGT_W) {
    const int k = threadIdx.x >> 5, c = threadIdx.x & 31;
    double t = 0.0;
    for (int q = 0; q < AGT_WARPS; ++q) t += ss[q][k][c];
    a.Spart[(size_t)blockIdx.x * 2 * AGT_W + threadIdx.x] = t;
  }
}

// pass p's partial rows summed in CTA order: dW_p, dbias_p (p < L); the sums of layer p - 1 (p >= 1)
__global__ void agg_backward_finish_kernel(const float *__restrict__ wpart, const double *__restrict__ Spart,
                                           int nparts, int p, int L, int w_out, int w_in, float *__restrict__ dW,
                                           float *__restrict__ dvec, double *__restrict__ S, int w_prev) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e < AGT_WROW) {
    if (p >= L) return;
    const bool isw = e < AGT_W * AGT_W;
    const int c = isw ? e / AGT_W : e - AGT_W * AGT_W, i = isw ? e - c * AGT_W : 0;
    if (c >= w_out || i >= w_in) return;
    float t = 0.f;
    for (int q = 0; q < nparts; ++q) t = __fadd_rn(t, wpart[(size_t)q * AGT_WROW + e]);
    if (isw) dW[c * w_in + i] = t;
    else dvec[p * 3 * AGT_W + c] = t;  // dbias
  } else if (e < AGT_WROW + 2 * AGT_W) {
    if (p < 1) return;
    const int k = (e - AGT_WROW) >> 5, c = (e - AGT_WROW) & 31;
    double t = 0.0;
    for (int q = 0; q < nparts; ++q) t += Spart[(size_t)q * 2 * AGT_W + k * AGT_W + c];
    const int l = p - 1;
    S[l * 2 * AGT_W + k * AGT_W + c] = c < w_prev ? t : 0.0;
    dvec[(l * 3 + (k == 0 ? 2 : 1)) * AGT_W + c] = c < w_prev ? (float)t : 0.f;  // dbeta = sum dy, dgamma = sum dy xhat
  }
}

// ---- feature gradient: stable inverse of idx, then a segment sum per point ------------------------------------
__global__ void agg_count_kernel(const int *__restrict__ idx, long long n_ent, int mns, int N, int *__restrict__ cnt) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_ent; e += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(e / mns);
    atomicAdd(cnt + (size_t)b * N + idx[e], 1);
  }
}

// exclusive scan of cnt (n) into off (n + 1) in three steps: per-tile exclusive scans and tile totals, a scan of the
// tile totals (one CTA, carried over chunks of AGT_SCAN_THREADS tiles), the tile offsets added
__device__ __forceinline__ int agg_block_exclusive_scan(int v, int *warp_tot, int *total) {
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
  int x = v;
#pragma unroll
  for (int o = 1; o < 32; o <<= 1) {
    const int y = __shfl_up_sync(0xffffffffu, x, o);
    if ((int)lane >= o) x += y;
  }
  if (lane == 31u) warp_tot[warp] = x;
  __syncthreads();
  if (warp == 0) {
    int w = (int)lane < (int)(blockDim.x >> 5) ? warp_tot[lane] : 0;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int y = __shfl_up_sync(0xffffffffu, w, o);
      if ((int)lane >= o) w += y;
    }
    warp_tot[lane] = w;  // inclusive
  }
  __syncthreads();
  const int before = (warp ? warp_tot[warp - 1] : 0) + x - v;
  *total = warp_tot[(blockDim.x >> 5) - 1];
  __syncthreads();
  return before;
}

__global__ void __launch_bounds__(AGT_SCAN_THREADS) agg_scan_tiles_kernel(const int *__restrict__ cnt, long long n,
                                                                          int *__restrict__ off, int *__restrict__ tsum) {
  __shared__ int wt[32];
  const long long i = blockIdx.x * (long long)AGT_SCAN_THREADS + threadIdx.x;
  int total;
  const int ex = agg_block_exclusive_scan(i < n ? cnt[i] : 0, wt, &total);
  if (i < n) off[i] = ex;
  if (threadIdx.x == 0) tsum[blockIdx.x] = total;
}

__global__ void __launch_bounds__(AGT_SCAN_THREADS) agg_scan_totals_kernel(int *__restrict__ tsum, int tiles,
                                                                           int *__restrict__ off_end) {
  __shared__ int wt[32];
  int carry = 0;
  for (int base = 0; base < tiles; base += AGT_SCAN_THREADS) {
    const int t = base + (int)threadIdx.x;
    int total;
    const int ex = agg_block_exclusive_scan(t < tiles ? tsum[t] : 0, wt, &total);
    if (t < tiles) tsum[t] = carry + ex;
    carry += total;
  }
  if (threadIdx.x == 0) *off_end = carry;
}

__global__ void agg_scan_add_kernel(int *__restrict__ off, long long n, const int *__restrict__ tsum) {
  const long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (i < n) off[i] += tsum[i / AGT_SCAN_THREADS];
}

// places every entry in its point's segment (order within a segment fixed later); counts cnt back down to zero
__global__ void agg_place_kernel(const int *__restrict__ idx, long long n_ent, int mns, int N, const int *__restrict__ off,
                                 int *__restrict__ cnt, int *__restrict__ slot) {
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < n_ent; e += (long long)gridDim.x * blockDim.x) {
    const size_t key = (size_t)(e / mns) * N + idx[e];
    slot[off[key] + atomicSub(cnt + key, 1) - 1] = (int)e;
  }
}

// dfeatures[b, c, p] = sum over the point's entries in ascending (b, j, s) of gx[entry, c]
__global__ void agg_segment_sum_kernel(const int *__restrict__ off, int *__restrict__ slot, const float *__restrict__ gx,
                                       int B, int N, int C, float *__restrict__ dfeat) {
  const long long key = blockIdx.x * (long long)blockDim.x + threadIdx.x;
  if (key >= (long long)B * N) return;
  const int b = (int)(key / N), p = (int)(key - (long long)b * N);
  const int lo = off[key], hi = off[key + 1];
  for (int i = lo + 1; i < hi; ++i) {  // insertion sort: segments hold a handful of entries
    const int v = slot[i];
    int k = i - 1;
    while (k >= lo && slot[k] > v) {
      slot[k + 1] = slot[k];
      --k;
    }
    slot[k + 1] = v;
  }
  float t[AGT_W];
#pragma unroll
  for (int c = 0; c < AGT_W; ++c) t[c] = 0.f;
  for (int i = lo; i < hi; ++i) {
    const float *g = gx + (size_t)slot[i] * C;
#pragma unroll
    for (int c = 0; c < AGT_W; ++c)
      if (c < C) t[c] = __fadd_rn(t[c], g[c]);
  }
#pragma unroll
  for (int c = 0; c < AGT_W; ++c)
    if (c < C) dfeat[((size_t)b * C + c) * N + p] = t[c];
}

static int agt_grid(int B, int m, int per_sm) {
  const long long blocks = ((long long)B * m + AGT_WARPS - 1) / AGT_WARPS, cap = (long long)num_sms() * per_sm;
  return (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
}
constexpr int AGT_STATS_PER_SM = 8;
constexpr int AGT_BWD_PER_SM = 2;

static int agt_validate(const char *who, const float *xyz, const float *new_xyz, const float *features, const int *idx,
                        int B, int N, int m, int nsample, int C, int use_xyz, int n_layers, const int *widths,
                        const float *const *weights, const int *batch_stats, const float *consts) {
  GF_CHECK_ARG(B >= 0 && N >= 1 && m >= 0 && nsample >= 1 && C >= 0, "%s: bad sizes", who);
  GF_CHECK_ARG(n_layers >= 1 && n_layers <= AGT_MAX_LAYERS, "%s: %d layers, 1..%d supported", who, n_layers,
               AGT_MAX_LAYERS);
  GF_CHECK_ARG(xyz && new_xyz && idx && widths && weights && batch_stats && consts, "%s: null pointer", who);
  GF_CHECK_ARG(features || C == 0, "%s: null features", who);
  GF_CHECK_ARG(use_xyz || C > 0, "%s: neither coordinates nor features", who);
  GF_CHECK_ARG(widths[0] == (use_xyz ? 3 : 0) + C, "%s: first width %d != %d input channels", who, widths[0],
               (use_xyz ? 3 : 0) + C);
  for (int l = 0; l <= n_layers; ++l)
    GF_CHECK_ARG(widths[l] >= 1 && widths[l] <= AGT_W, "%s: width %d of layer %d outside [1,%d]", who, widths[l], l,
                 AGT_W);
  for (int l = 0; l < n_layers; ++l) GF_CHECK_ARG(weights[l], "%s: null weights of layer %d", who, l);
  return GF_OK;
}

static void agt_fill(AgtArgs &a, const float *xyz, const float *new_xyz, const float *features, const int *idx, int B,
                     int N, int m, int nsample, int C, float radius, int normalize_xyz, int use_xyz, int n_layers,
                     const int *widths, const float *const *weights, const int *batch_stats, float *consts,
                     int pool_avg) {
  a = AgtArgs{};
  a.xyz = xyz, a.new_xyz = new_xyz, a.features = features, a.idx = idx, a.B = B, a.N = N, a.m = m, a.ns = nsample;
  a.C = C, a.radius = radius, a.normalize = normalize_xyz ? 1 : 0, a.use_xyz = use_xyz ? 1 : 0;
  a.n_layers = n_layers, a.pool_avg = pool_avg ? 1 : 0;
  for (int l = 0; l <= n_layers; ++l) a.width[l] = widths[l];
  for (int l = 0; l < n_layers; ++l) a.w[l] = weights[l], a.batch[l] = batch_stats[l] ? 1 : 0;
  a.consts = consts;
}

}  // namespace gf

using namespace gf;

// the training forward's workspace: the per-CTA partial batch statistics
static Arena agt_train_carve(void *workspace, size_t workspace_bytes, int B, int m, double **spart) {
  Arena a(workspace, workspace_bytes);
  *spart = a.take<double>((size_t)agt_grid(B, m, AGT_STATS_PER_SM) * 2 * AGT_W);
  return a;
}

extern "C" size_t gf_group_mlp_pool_train_workspace_bytes(int B, int m) {
  if (B <= 0 || m <= 0) return 0;
  double *spart;
  return agt_train_carve(nullptr, 0, B, m, &spart).off;
}

extern "C" int gf_group_mlp_pool_train(const float *xyz, const float *new_xyz, const float *features, const int *idx,
                                       int B, int N, int m, int nsample, int C, float radius, int normalize_xyz,
                                       int use_xyz, int n_layers, const int *widths, const float *const *weights,
                                       const float *const *gammas, const float *const *betas, const float *eps,
                                       const int *batch_stats, float *consts, int pool_avg, float *out,
                                       void *workspace, size_t workspace_bytes, void *stream) {
  int rc = agt_validate("group_mlp_pool_train", xyz, new_xyz, features, idx, B, N, m, nsample, C, use_xyz, n_layers,
                        widths, weights, batch_stats, consts);
  if (rc) return rc;
  GF_CHECK_ARG(out && gammas && betas && eps, "group_mlp_pool_train: null pointer");
  for (int l = 0; l < n_layers; ++l)
    if (batch_stats[l])
      GF_CHECK_ARG(gammas[l] && betas[l] && eps[l] > 0.f, "group_mlp_pool_train: layer %d needs gamma, beta, eps > 0", l);
  if (B == 0 || m == 0) return GF_OK;
  const int grid = agt_grid(B, m, AGT_STATS_PER_SM);
  double *spart;
  const Arena ar = agt_train_carve(workspace, workspace_bytes, B, m, &spart);
  if (!ar.ok) return ar.fail("group_mlp_pool_train");
  AgtArgs a;
  agt_fill(a, xyz, new_xyz, features, idx, B, N, m, nsample, C, radius, normalize_xyz, use_xyz, n_layers, widths,
           weights, batch_stats, consts, pool_avg);
  a.spart = spart;
  cudaStream_t st = (cudaStream_t)stream;
  const double n = (double)B * m * nsample;
  for (int l = 0; l < n_layers; ++l) {
    if (!batch_stats[l]) continue;
    switch (l) {
      case 0: agg_stats_kernel<0><<<grid, AGT_THREADS, 0, st>>>(a); break;
      case 1: agg_stats_kernel<1><<<grid, AGT_THREADS, 0, st>>>(a); break;
      case 2: agg_stats_kernel<2><<<grid, AGT_THREADS, 0, st>>>(a); break;
      default: agg_stats_kernel<3><<<grid, AGT_THREADS, 0, st>>>(a); break;
    }
    GF_LAUNCHED();
    agg_stats_finish_kernel<<<1, AGT_W, 0, st>>>(spart, grid, n, widths[l + 1], gammas[l], betas[l], eps[l],
                                                 consts + l * AGT_CONST);
    GF_LAUNCHED();
  }
  const float *sc[AGT_MAX_LAYERS], *sh[AGT_MAX_LAYERS];
  for (int l = 0; l < n_layers; ++l) sc[l] = consts + l * AGT_CONST, sh[l] = consts + l * AGT_CONST + AGT_W;
  return gf_group_mlp_pool(xyz, new_xyz, features, idx, B, N, m, nsample, C, radius, normalize_xyz, use_xyz, n_layers,
                           widths, weights, sc, sh, pool_avg, out, stream);
}

// The backward's workspace: the pooling winners, the statistics and per-CTA partial sums of the layers, the
// gradient of every grouped sample, and the counting sort of the samples by source point that gathers dfeatures
struct AgtBwdLayout {
  int *arg;
  double *S;
  float *wpart;
  double *Spart;
  float *gx;
  int *cnt, *off, *slot, *tsum;
  int tiles;
};
static Arena agt_bwd_carve(void *workspace, size_t workspace_bytes, int B, int N, int m, int nsample, int C,
                           AgtBwdLayout *l) {
  Arena a(workspace, workspace_bytes);
  const size_t grid = (size_t)agt_grid(B, m, AGT_BWD_PER_SM), ent = (size_t)B * m * nsample, nkeys = (size_t)B * N;
  l->tiles = (int)((nkeys + AGT_SCAN_THREADS - 1) / AGT_SCAN_THREADS);
  l->arg = a.take<int>((size_t)B * m * AGT_W);
  l->S = a.take<double>(AGT_MAX_LAYERS * 2 * AGT_W);
  l->wpart = a.take<float>(grid * AGT_WROW);
  l->Spart = a.take<double>(grid * 2 * AGT_W);
  l->gx = a.take<float>(ent * (size_t)C);
  l->cnt = a.take<int>(nkeys);
  l->off = a.take<int>(nkeys + 1);
  l->slot = a.take<int>(ent);
  l->tsum = a.take<int>((size_t)l->tiles);
  return a;
}

extern "C" size_t gf_group_mlp_pool_backward_workspace_bytes(int B, int N, int m, int nsample, int C) {
  if (B <= 0 || m <= 0 || N <= 0 || nsample <= 0 || C < 0) return 0;
  AgtBwdLayout l;
  return agt_bwd_carve(nullptr, 0, B, N, m, nsample, C, &l).off;
}

extern "C" int gf_group_mlp_pool_backward(const float *xyz, const float *new_xyz, const float *features,
                                          const int *idx, int B, int N, int m, int nsample, int C, float radius,
                                          int normalize_xyz, int use_xyz, int n_layers, const int *widths,
                                          const float *const *weights, const int *batch_stats, const float *consts,
                                          int pool_avg, const float *dout, float *dfeatures,
                                          float *const *dweights, float *dvec, void *workspace,
                                          size_t workspace_bytes, void *stream) {
  int rc = agt_validate("group_mlp_pool_backward", xyz, new_xyz, features, idx, B, N, m, nsample, C, use_xyz, n_layers,
                        widths, weights, batch_stats, consts);
  if (rc) return rc;
  GF_CHECK_ARG(dout && dweights && dvec, "group_mlp_pool_backward: null pointer");
  for (int l = 0; l < n_layers; ++l) GF_CHECK_ARG(dweights[l], "group_mlp_pool_backward: null dweights of layer %d", l);
  cudaStream_t st = (cudaStream_t)stream;
  if (B == 0 || m == 0) {  // nothing pooled: every gradient is zero
    for (int l = 0; l < n_layers; ++l)
      GF_CUDA(cudaMemsetAsync(dweights[l], 0, sizeof(float) * widths[l] * widths[l + 1], st));
    GF_CUDA(cudaMemsetAsync(dvec, 0, sizeof(float) * n_layers * 3 * AGT_W, st));
    if (dfeatures && C > 0) GF_CUDA(cudaMemsetAsync(dfeatures, 0, sizeof(float) * (size_t)B * C * N, st));
    return GF_OK;
  }
  AgtBwdLayout l;
  const Arena ar = agt_bwd_carve(workspace, workspace_bytes, B, N, m, nsample, C, &l);
  if (!ar.ok) return ar.fail("group_mlp_pool_backward");
  const int grid = agt_grid(B, m, AGT_BWD_PER_SM);
  const size_t ent = (size_t)B * m * nsample;
  AgtArgs a;
  agt_fill(a, xyz, new_xyz, features, idx, B, N, m, nsample, C, radius, normalize_xyz, use_xyz, n_layers, widths,
           weights, batch_stats, const_cast<float *>(consts), pool_avg);
  a.dout = dout;
  a.arg = l.arg, a.S = l.S, a.wpart = l.wpart, a.Spart = l.Spart, a.gx = l.gx;
  const long long nkeys = (long long)B * N;
  const bool want_dfeat = dfeatures && C > 0;
  if (!want_dfeat) a.gx = nullptr;
  if (want_dfeat) GF_CUDA(cudaMemsetAsync(a.gx, 0, sizeof(float) * ent * C, st));  // samples without gradient
  GF_CUDA(cudaMemsetAsync(dvec, 0, sizeof(float) * n_layers * 3 * AGT_W, st));
  const int fin_blocks = (AGT_WROW + 2 * AGT_W + 127) / 128;
  for (int p = n_layers; p >= 0; --p) {
    switch (n_layers) {
      case 1: agg_backward_kernel<1><<<grid, AGT_THREADS, 0, st>>>(a, p); break;
      case 2: agg_backward_kernel<2><<<grid, AGT_THREADS, 0, st>>>(a, p); break;
      case 3: agg_backward_kernel<3><<<grid, AGT_THREADS, 0, st>>>(a, p); break;
      default: agg_backward_kernel<4><<<grid, AGT_THREADS, 0, st>>>(a, p); break;
    }
    GF_LAUNCHED();
    agg_backward_finish_kernel<<<fin_blocks, 128, 0, st>>>(a.wpart, a.Spart, grid, p, n_layers,
                                                          p < n_layers ? widths[p + 1] : 0, p < n_layers ? widths[p] : 0,
                                                          p < n_layers ? dweights[p] : nullptr, dvec, l.S,
                                                          p >= 1 ? widths[p] : 0);
    GF_LAUNCHED();
  }
  if (!want_dfeat) return GF_OK;
  const int mns = m * nsample;
  const int eb = (int)((ent + 255) / 256 < (size_t)num_sms() * 16 ? (ent + 255) / 256 : (size_t)num_sms() * 16);
  GF_CUDA(cudaMemsetAsync(l.cnt, 0, sizeof(int) * (size_t)B * N, st));
  agg_count_kernel<<<eb, 256, 0, st>>>(idx, (long long)ent, mns, N, l.cnt);
  GF_LAUNCHED();
  agg_scan_tiles_kernel<<<l.tiles, AGT_SCAN_THREADS, 0, st>>>(l.cnt, nkeys, l.off, l.tsum);
  GF_LAUNCHED();
  agg_scan_totals_kernel<<<1, AGT_SCAN_THREADS, 0, st>>>(l.tsum, l.tiles, l.off + nkeys);
  GF_LAUNCHED();
  agg_scan_add_kernel<<<(unsigned)((nkeys + 255) / 256), 256, 0, st>>>(l.off, nkeys, l.tsum);
  GF_LAUNCHED();
  agg_place_kernel<<<eb, 256, 0, st>>>(idx, (long long)ent, mns, N, l.off, l.cnt, l.slot);
  GF_LAUNCHED();
  agg_segment_sum_kernel<<<(unsigned)(((long long)B * N + 255) / 256), 256, 0, st>>>(l.off, l.slot, a.gx, B, N, C,
                                                                                      dfeatures);
  GF_LAUNCHED();
  return GF_OK;
}
