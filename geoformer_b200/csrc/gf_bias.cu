// The two "distance -> bias" epilogues that consume the geodesic maps.
//   decoder:   model/geoformer/geoformer_fs.py:680-702 (= geoformer.py:619-641)
//   mask head: model/geoformer/geoformer_fs.py:263-292 (= geoformer.py:286-313)
// Both need a per-seed row maximum and the maximum over all seeds before the element-wise part,
// so each is two kernels: a row-max reduction (with an ordered-int atomicMax for the global
// maximum) and a fused element-wise pass that writes the reference's output layout directly
// (no (Q,N,3) boolean-mask temporaries as in the reference).
#include "gf_bias.cuh"

namespace gf {

__device__ __forceinline__ float block_max(float v, float *sm) {
  for (int o = 16; o; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = v;
  __syncthreads();
  float r = sm[0];
  for (int w = 1; w < (int)(blockDim.x >> 5); ++w) r = fmaxf(r, sm[w]);
  __syncthreads();
  return r;
}

__global__ void bias_init_kernel(uint32_t *gmax) { *gmax = 0u; }
// ordered-int maxima: 0 is below every float, so zero is the identity of the atomicMax reductions
__global__ void bias_zero_kernel(uint32_t *p, int n) {
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) p[i] = 0u;
}

// ---- decoder epilogue -------------------------------------------------------------------------------
// rowmax[q] = max_c geo[q, ctx_idx[c]]      (geoformer_fs.py:685-691); several CTAs per row (a row is only
// C gathers: one CTA per row would be a chain of dependent L2 round trips), combined by an ordered atomicMax
__global__ void __launch_bounds__(256)
    bias_ctx_rowmax_kernel(const float *__restrict__ geo, int ld, const int *__restrict__ ctx_idx, int C,
                           uint32_t *__restrict__ rowmax_ord, uint32_t *__restrict__ gmax) {
  __shared__ float sm[8];
  const int q = blockIdx.y;
  float v = -__int_as_float(0x7f800000);
  for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < C; c += gridDim.x * blockDim.x)
    v = fmaxf(v, __ldg(geo + (size_t)q * ld + __ldg(ctx_idx + c)));
  float r = block_max(v, sm);
  if (threadIdx.x == 0 && r > -__int_as_float(0x7f800000)) {
    atomicMax(rowmax_ord + q, f2ord(r));
    atomicMax(gmax, f2ord(r));  // :692  max over every (batch, query)
  }
}

// out[q,c,:] = G >= 0 ? G : m_q + |query_xyz[q] - ctx_xyz[c]|      (:693-702)
__global__ void __launch_bounds__(256)
    bias_ctx_write_kernel(const float *__restrict__ geo, int ld, const int *__restrict__ ctx_idx,
                          const float *__restrict__ query_xyz, const float *__restrict__ ctx_xyz, int Q, int C,
                          const uint32_t *__restrict__ rowmax, const uint32_t *__restrict__ gmax, float *__restrict__ out) {
  const float M = ord2f(*gmax);
  for (int e = blockIdx.x * blockDim.x + threadIdx.x; e < Q * C; e += gridDim.x * blockDim.x) {
    const int q = e / C, c = e - q * C;
    float g = __ldg(geo + (size_t)q * ld + __ldg(ctx_idx + c));
    float m = ord2f(rowmax[q]);
    if (m < 0.f) m = M;  // :693
    float o0 = g, o1 = g, o2 = g;
    if (g < 0.f) {
      o0 = __fadd_rn(m, fabsf(__fsub_rn(query_xyz[q * 3 + 0], ctx_xyz[c * 3 + 0])));
      o1 = __fadd_rn(m, fabsf(__fsub_rn(query_xyz[q * 3 + 1], ctx_xyz[c * 3 + 1])));
      o2 = __fadd_rn(m, fabsf(__fsub_rn(query_xyz[q * 3 + 2], ctx_xyz[c * 3 + 2])));
    }
    float *o = out + (size_t)e * 3;
    o[0] = o0, o[1] = o1, o[2] = o2;
  }
}

// ---- decoder epilogue fused with the Fourier position embedding (SURVEY 8(f) rank 1) ------------------
// What the decoder consumes is not the (B,Q,C,3) tensor above but its embedding
// (geoformer_fs.py:704-712 -> pos_embedding.py:88-114, utils_pc.py:35-61):
//   v_a   = the value above, a = 0..2
//   n_a   = ((v_a - pc_min[b,a]) * 1 / (pc_max[b,a] - pc_min[b,a]) + 0) * 2pi     (shift_scale_points, then *= 2*np.pi)
//   p_j   = sum_a n_a * gauss_B[a,j]                                               (torch.mm, j < d_out)
//   out[b,q,c,j] = sin(p_j), out[b,q,c,d_out+j] = cos(p_j)
// i.e. the memory behind the reference's relative_pos view (Q,C,B,2*d_out).  One warp takes 32 contexts of one
// query: lane l prepares n_0..2 of context l (gather, fill, normalisation: done once, not once per
// frequency), then the warp walks the 32 contexts with lane = frequency, so every store is a full 128-byte line.
__global__ void __launch_bounds__(256)
    bias_ctx_fourier_kernel(const float *__restrict__ geo, int ld, const int *__restrict__ ctx_idx,
                            const float *__restrict__ query_xyz, const float *__restrict__ ctx_xyz, int Q, int C,
                            const uint32_t *__restrict__ rowmax, const uint32_t *__restrict__ gmax,
                            const float *__restrict__ gauss_B, int d_out, int ldb, const float *__restrict__ pc_min,
                            const float *__restrict__ pc_max, float *__restrict__ out) {
  const unsigned lane = threadIdx.x & 31u, warp = threadIdx.x >> 5, nwarp = blockDim.x >> 5;
  const int q = blockIdx.y;
  float m = ord2f(rowmax[q]);
  if (m < 0.f) m = ord2f(*gmax);  // :693
  const float qx = query_xyz[q * 3 + 0], qy = query_xyz[q * 3 + 1], qz = query_xyz[q * 3 + 2];
  const float mn0 = pc_min[0], mn1 = pc_min[1], mn2 = pc_min[2];
  const float df0 = __fsub_rn(pc_max[0], mn0), df1 = __fsub_rn(pc_max[1], mn1), df2 = __fsub_rn(pc_max[2], mn2);
  const float two_pi = 6.2831855f;  // float(2 * np.pi)
  const int d_pos = 2 * d_out;
  for (int c0 = (blockIdx.x * nwarp + warp) * 32; c0 < C; c0 += gridDim.x * nwarp * 32) {
    const int c = c0 + (int)lane;
    float n0 = 0.f, n1 = 0.f, n2 = 0.f;
    if (c < C) {
      const float g = __ldg(geo + (size_t)q * ld + __ldg(ctx_idx + c));
      float v0 = g, v1 = g, v2 = g;
      if (g < 0.f) {
        v0 = __fadd_rn(m, fabsf(__fsub_rn(qx, ctx_xyz[c * 3 + 0])));
        v1 = __fadd_rn(m, fabsf(__fsub_rn(qy, ctx_xyz[c * 3 + 1])));
        v2 = __fadd_rn(m, fabsf(__fsub_rn(qz, ctx_xyz[c * 3 + 2])));
      }
      n0 = __fmul_rn(__fdiv_rn(__fsub_rn(v0, mn0), df0), two_pi);
      n1 = __fmul_rn(__fdiv_rn(__fsub_rn(v1, mn1), df1), two_pi);
      n2 = __fmul_rn(__fdiv_rn(__fsub_rn(v2, mn2), df2), two_pi);
    }
    const int nc = min(32, C - c0);
    // warp-uniform trip count: every lane takes part in the shuffles of every round, lanes whose frequency
    // j is past d_out (d_out < 32 or not a multiple of 32) only skip the loads and the stores
    for (int jb = 0; jb < d_out; jb += 32) {
      const int j = jb + (int)lane;
      const bool live = j < d_out;
      const float b0 = live ? __ldg(gauss_B + j) : 0.f, b1 = live ? __ldg(gauss_B + ldb + j) : 0.f,
                  b2 = live ? __ldg(gauss_B + 2 * ldb + j) : 0.f;
      float *o = out + ((size_t)q * C + c0) * d_pos + j;
      for (int i = 0; i < nc; ++i) {
        const float x0 = __shfl_sync(0xffffffffu, n0, i), x1 = __shfl_sync(0xffffffffu, n1, i),
                    x2 = __shfl_sync(0xffffffffu, n2, i);
        if (live) {
          const float p = fmaf(x2, b2, fmaf(x1, b1, __fmul_rn(x0, b0)));
          float sn, cs;
          sincosf(p, &sn, &cs);
          __stcs(o + (size_t)i * d_pos, sn);
          __stcs(o + (size_t)i * d_pos + d_out, cs);
        }
      }
    }
  }
}

// ---- mask-head epilogue -----------------------------------------------------------------------------
// Pure streaming (read geo, write three times as much): 16-byte accesses, four points per thread.
// rowmax[q] = max_p geo[q,p]   (:274-275); several CTAs per row, combined with an ordered atomicMax
template <bool VEC>
__global__ void __launch_bounds__(256)
    bias_mask_rowmax_kernel(const float *__restrict__ geo, int N, int chunks, uint32_t *__restrict__ rowmax_ord,
                            uint32_t *__restrict__ gmax) {
  __shared__ float sm[8];
  const int q = blockIdx.x / chunks, ch = blockIdx.x - q * chunks;
  const float *row = geo + (size_t)q * N;
  float v = -__int_as_float(0x7f800000);
  if (VEC) {
    const int n4 = N >> 2, per = (n4 + chunks - 1) / chunks;
    const int p0 = ch * per, p1 = min(n4, p0 + per);
    const float4 *r4 = reinterpret_cast<const float4 *>(row);
    for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
      const float4 g = __ldg(r4 + p);
      v = fmaxf(fmaxf(v, fmaxf(g.x, g.y)), fmaxf(g.z, g.w));
    }
  } else {
    const int per = (N + chunks - 1) / chunks;
    const int p0 = ch * per, p1 = min(N, p0 + per);
    for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) v = fmaxf(v, __ldg(row + p));
  }
  float r = block_max(v, sm);
  if (threadIdx.x == 0 && r > -__int_as_float(0x7f800000)) {
    atomicMax(rowmax_ord + q, f2ord(r));
    atomicMax(gmax, f2ord(r));
  }
}

// row maxima handed over by the producer of the maps (gf_geodesic / gf_guidance `row_max`): no pass over geo.
// One block: it also initialises the global maximum, so nothing has to be zeroed beforehand.
__global__ void __launch_bounds__(1024)
    bias_rowmax_import_kernel(const float *__restrict__ row_max, int Q, uint32_t *__restrict__ rowmax_ord,
                              uint32_t *__restrict__ gmax) {
  __shared__ float sm[32];
  float v = -__int_as_float(0x7f800000);
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    const float r = row_max[q];
    rowmax_ord[q] = f2ord(r);
    v = fmaxf(v, r);
  }
  const float r = block_max(v, sm);
  if (threadIdx.x == 0) *gmax = r > -__int_as_float(0x7f800000) ? f2ord(r) : 0u;
}

// bias_mask_rowmax_kernel over the rows of a batch: block (row, chunk) with row = b*Q + q reduces its chunk of scene
// b's row q into rowmax[row] and scene b's own maximum gmax[b] (:276 takes the maximum over one scene's rows only)
__global__ void __launch_bounds__(256)
    bias_mask_rowmax_batch_kernel(const __grid_constant__ MaskMaps maps, uint32_t *__restrict__ rowmax_ord,
                                  uint32_t *__restrict__ gmax) {
  __shared__ float sm[8];
  const int row = blockIdx.x, b = row / maps.Q, q = row - b * maps.Q, N = maps.N[b], chunks = gridDim.y;
  const float *rp = maps.geo[b] + (size_t)q * N;
  float v = -__int_as_float(0x7f800000);
  if (N % 4 == 0 && ((uintptr_t)maps.geo[b] & 15) == 0) {
    const int n4 = N >> 2, per = (n4 + chunks - 1) / chunks;
    const int p0 = blockIdx.y * per, p1 = min(n4, p0 + per);
    const float4 *r4 = reinterpret_cast<const float4 *>(rp);
    for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) {
      const float4 g = __ldg(r4 + p);
      v = fmaxf(fmaxf(v, fmaxf(g.x, g.y)), fmaxf(g.z, g.w));
    }
  } else {
    const int per = (N + chunks - 1) / chunks;
    const int p0 = blockIdx.y * per, p1 = min(N, p0 + per);
    for (int p = p0 + threadIdx.x; p < p1; p += blockDim.x) v = fmaxf(v, __ldg(rp + p));
  }
  float r = block_max(v, sm);
  if (threadIdx.x == 0 && r > -__int_as_float(0x7f800000)) {
    atomicMax(rowmax_ord + row, f2ord(r));
    atomicMax(gmax + b, f2ord(r));
  }
}

// bias_rowmax_import_kernel per scene: block b imports row_max[b] (Q) and sets gmax[b]
__global__ void __launch_bounds__(1024)
    bias_rowmax_import_batch_kernel(const float *__restrict__ row_max, int Q, uint32_t *__restrict__ rowmax_ord,
                                    uint32_t *__restrict__ gmax) {
  __shared__ float sm[32];
  const size_t base = (size_t)blockIdx.x * Q;
  float v = -__int_as_float(0x7f800000);
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    const float r = row_max[base + q];
    rowmax_ord[base + q] = f2ord(r);
    v = fmaxf(v, r);
  }
  const float r = block_max(v, sm);
  if (threadIdx.x == 0) gmax[blockIdx.x] = r > -__int_as_float(0x7f800000) ? f2ord(r) : 0u;
}

// out[q,a,p] = d + (geo[q,p] < 0 ? sqrt(m_q) * sign(d) : 0),  d = seed_xyz[q,a] - coords[p,a]   (:271-289)
template <bool VEC>
__global__ void __launch_bounds__(256)
    bias_mask_write_kernel(const float *__restrict__ geo, const float *__restrict__ coords,
                           const float *__restrict__ seed_xyz, int Q, int N, const uint32_t *__restrict__ rowmax_ord,
                           const uint32_t *__restrict__ gmax, float *__restrict__ out) {
  const int q = blockIdx.y;
  float m = ord2f(rowmax_ord[q]);
  if (m < 0.f) m = ord2f(*gmax);  // :276
  const float s = sqrtf(m);       // :277
  const float sx = seed_xyz[q * 3 + 0], sy = seed_xyz[q * 3 + 1], sz = seed_xyz[q * 3 + 2];
  float *o = out + (size_t)q * 3 * N;
  const float *row = geo + (size_t)q * N;
  if (VEC) {
    const int n4 = N >> 2;
    const float4 *g4 = reinterpret_cast<const float4 *>(row);
    const float4 *c4 = reinterpret_cast<const float4 *>(coords);  // 4 points = 12 floats = 3 float4
    float4 *ox = reinterpret_cast<float4 *>(o), *oy = reinterpret_cast<float4 *>(o + N),
           *oz = reinterpret_cast<float4 *>(o + 2 * (size_t)N);
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < n4; p += gridDim.x * blockDim.x) {
      const float4 g = __ldg(g4 + p);
      const float4 a = __ldg(c4 + 3 * (size_t)p), b = __ldg(c4 + 3 * (size_t)p + 1), c = __ldg(c4 + 3 * (size_t)p + 2);
      // a = x0 y0 z0 x1 | b = y1 z1 x2 y2 | c = z2 x3 y3 z3
      float4 rx, ry, rz;
      rx.x = mask_push(__fsub_rn(sx, a.x), s, g.x < 0.f), ry.x = mask_push(__fsub_rn(sy, a.y), s, g.x < 0.f),
      rz.x = mask_push(__fsub_rn(sz, a.z), s, g.x < 0.f);
      rx.y = mask_push(__fsub_rn(sx, a.w), s, g.y < 0.f), ry.y = mask_push(__fsub_rn(sy, b.x), s, g.y < 0.f),
      rz.y = mask_push(__fsub_rn(sz, b.y), s, g.y < 0.f);
      rx.z = mask_push(__fsub_rn(sx, b.z), s, g.z < 0.f), ry.z = mask_push(__fsub_rn(sy, b.w), s, g.z < 0.f),
      rz.z = mask_push(__fsub_rn(sz, c.x), s, g.z < 0.f);
      rx.w = mask_push(__fsub_rn(sx, c.y), s, g.w < 0.f), ry.w = mask_push(__fsub_rn(sy, c.z), s, g.w < 0.f),
      rz.w = mask_push(__fsub_rn(sz, c.w), s, g.w < 0.f);
      __stcs(ox + p, rx);  // written once, never re-read by this kernel: streaming stores
      __stcs(oy + p, ry);
      __stcs(oz + p, rz);
    }
  } else {
    for (int p = blockIdx.x * blockDim.x + threadIdx.x; p < N; p += gridDim.x * blockDim.x) {
      const bool un = __ldg(row + p) < 0.f;
      o[p] = mask_push(__fsub_rn(sx, __ldg(coords + (size_t)p * 3 + 0)), s, un);
      o[(size_t)N + p] = mask_push(__fsub_rn(sy, __ldg(coords + (size_t)p * 3 + 1)), s, un);
      o[(size_t)2 * N + p] = mask_push(__fsub_rn(sz, __ldg(coords + (size_t)p * 3 + 2)), s, un);
    }
  }
}

// ordered-uint row maxima of the gathered maps and their global maximum (geoformer_fs.py:685-692); geo_ptrs / geo_ld
// are HOST arrays of B device pointers / row strides.  Shared with the fused cross-attention (gf_attention.cu).
int bias_ctx_rowmax(const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx, int B, int Q, int C,
                    const RowMax &rm, cudaStream_t st) {
  bias_zero_kernel<<<(B * Q + 256) / 256, 256, 0, st>>>(rm.rowmax, B * Q + 1);  // the row maxima and gmax after them
  GF_LAUNCHED();
  const int rchunks = C >= 1024 ? 4 : 1;
  for (int b = 0; b < B; ++b) {
    bias_ctx_rowmax_kernel<<<dim3(rchunks, Q), 256, 0, st>>>(geo_ptrs[b], geo_ld[b], ctx_idx + (size_t)b * C, C,
                                                           rm.rowmax + (size_t)b * Q, rm.gmax);
    GF_LAUNCHED();
  }
  return GF_OK;
}

// ordered-uint row maxima of the (Q,N) maps and their global maximum (geoformer_fs.py:274-276), or the producer's
// row_max imported; nothing has to be zeroed beforehand.  Shared with the fused mask head (gf_mask_head.cu).
int bias_mask_rowmax(const float *geo, int Q, int N, const float *row_max, bool vec, const RowMax &rm, cudaStream_t st) {
  uint32_t *rowmax = rm.rowmax, *gmax = rm.gmax;
  if (!row_max) {
    GF_CUDA(cudaMemsetAsync(rowmax, 0, sizeof(uint32_t) * (size_t)Q, st));
    bias_init_kernel<<<1, 1, 0, st>>>(gmax);
    GF_LAUNCHED();
  }
  const int work = vec ? N / 4 : N;
  int chunks = (num_sms() * 8 + Q - 1) / Q;
  if (chunks < 1) chunks = 1;
  if (chunks > (work + 1023) / 1024) chunks = (work + 1023) / 1024;
  if (chunks < 1) chunks = 1;
  if (row_max)
    bias_rowmax_import_kernel<<<1, 1024, 0, st>>>(row_max, Q, rowmax, gmax);
  else if (vec)
    bias_mask_rowmax_kernel<true><<<Q * chunks, 256, 0, st>>>(geo, N, chunks, rowmax, gmax);
  else
    bias_mask_rowmax_kernel<false><<<Q * chunks, 256, 0, st>>>(geo, N, chunks, rowmax, gmax);
  GF_LAUNCHED();
  return GF_OK;
}

// row maxima of a batch's maps, each scene's maximum its own; gmax must follow rowmax (B*Q) so that one fill clears both
int bias_mask_rowmax_batch(const MaskMaps &maps, const float *row_max, uint32_t *rowmax, uint32_t *gmax,
                           cudaStream_t st) {
  const int rows = maps.B * maps.Q;
  if (row_max) {
    bias_rowmax_import_batch_kernel<<<maps.B, 1024, 0, st>>>(row_max, maps.Q, rowmax, gmax);
    GF_LAUNCHED();
    return GF_OK;
  }
  bias_zero_kernel<<<(rows + maps.B + 255) / 256, 256, 0, st>>>(rowmax, rows + maps.B);
  GF_LAUNCHED();
  int nmax = 0;
  for (int b = 0; b < maps.B; ++b) nmax = maps.N[b] > nmax ? maps.N[b] : nmax;
  // as bias_mask_rowmax: about 8 blocks per SM, no chunk of the largest scene under 1024 loads
  int chunks = (num_sms() * 8 + rows - 1) / rows;
  if (chunks > (nmax / 4 + 1023) / 1024) chunks = (nmax / 4 + 1023) / 1024;
  if (chunks < 1) chunks = 1;
  bias_mask_rowmax_batch_kernel<<<dim3(rows, chunks), 256, 0, st>>>(maps, rowmax, gmax);
  GF_LAUNCHED();
  return GF_OK;
}

}  // namespace gf

using namespace gf;

// the workspace of the three epilogues: the row maxima of the `rows` maps
static Arena bias_carve(void *workspace, size_t workspace_bytes, size_t rows, RowMax *rm) {
  Arena a(workspace, workspace_bytes);
  *rm = take_rowmax(a, rows);
  return a;
}

extern "C" size_t gf_bias_workspace_bytes(int B, int Q) {
  if (B <= 0 || Q <= 0) return 0;
  RowMax rm;
  return bias_carve(nullptr, 0, (size_t)B * Q, &rm).off;
}

extern "C" int gf_bias_decoder(const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx,
                               const float *query_xyz, const float *ctx_xyz, int B, int Q, int C, float *out,
                               void *workspace, size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(B >= 0 && Q >= 0 && C >= 0, "bias_decoder: negative size");
  if ((long long)B * Q * C == 0) return GF_OK;
  GF_CHECK_ARG(geo_ptrs && geo_ld && ctx_idx && query_xyz && ctx_xyz && out, "bias_decoder: null pointer");
  RowMax rm;
  const Arena a = bias_carve(workspace, workspace_bytes, (size_t)B * Q, &rm);
  if (!a.ok) return a.fail("bias_decoder");
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = bias_ctx_rowmax(geo_ptrs, geo_ld, ctx_idx, B, Q, C, rm, st);
  if (rc) return rc;
  for (int b = 0; b < B; ++b) {
    int grid = (Q * C + 255) / 256;
    if (grid > num_sms() * 8) grid = num_sms() * 8;
    bias_ctx_write_kernel<<<grid, 256, 0, st>>>(geo_ptrs[b], geo_ld[b], ctx_idx + (size_t)b * C,
                                                query_xyz + (size_t)b * Q * 3, ctx_xyz + (size_t)b * C * 3, Q, C,
                                                rm.rowmax + (size_t)b * Q, rm.gmax, out + (size_t)b * Q * C * 3);
    GF_LAUNCHED();
  }
  return GF_OK;
}

extern "C" int gf_bias_decoder_fourier(const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx,
                                       const float *query_xyz, const float *ctx_xyz, int B, int Q, int C,
                                       const float *gauss_B, int d_out, int gauss_ld, const float *pc_min,
                                       const float *pc_max, float *out, void *workspace, size_t workspace_bytes,
                                       void *stream) {
  GF_CHECK_ARG(B >= 0 && Q >= 0 && C >= 0, "bias_decoder_fourier: negative size");
  GF_CHECK_ARG(d_out >= 1 && gauss_ld >= d_out, "bias_decoder_fourier: d_out=%d, gauss_ld=%d", d_out, gauss_ld);
  if ((long long)B * Q * C == 0) return GF_OK;
  GF_CHECK_ARG(geo_ptrs && geo_ld && ctx_idx && query_xyz && ctx_xyz && gauss_B && pc_min && pc_max && out,
               "bias_decoder_fourier: null pointer");
  RowMax rm;
  const Arena a = bias_carve(workspace, workspace_bytes, (size_t)B * Q, &rm);
  if (!a.ok) return a.fail("bias_decoder_fourier");
  cudaStream_t st = (cudaStream_t)stream;
  const int rc = bias_ctx_rowmax(geo_ptrs, geo_ld, ctx_idx, B, Q, C, rm, st);
  if (rc) return rc;
  for (int b = 0; b < B; ++b) {
    int gx = (C + 255) / 256;  // 8 warps x 32 contexts per block: one pass per warp, no ragged second round
    if (gx > 4096) gx = 4096;
    bias_ctx_fourier_kernel<<<dim3(gx, Q), 256, 0, st>>>(
        geo_ptrs[b], geo_ld[b], ctx_idx + (size_t)b * C, query_xyz + (size_t)b * Q * 3, ctx_xyz + (size_t)b * C * 3, Q, C,
        rm.rowmax + (size_t)b * Q, rm.gmax, gauss_B, d_out, gauss_ld, pc_min + (size_t)b * 3, pc_max + (size_t)b * 3,
        out + (size_t)b * Q * C * 2 * d_out);
    GF_LAUNCHED();
  }
  return GF_OK;
}

extern "C" int gf_bias_mask_head(const float *geo, const float *coords, const float *seed_xyz, int Q, int N,
                                 const float *row_max, float *out, void *workspace, size_t workspace_bytes,
                                 void *stream) {
  GF_CHECK_ARG(Q >= 0 && N >= 0, "bias_mask_head: negative size");
  if ((long long)Q * N == 0) return GF_OK;
  GF_CHECK_ARG(geo && coords && seed_xyz && out, "bias_mask_head: null pointer");
  RowMax rm;
  const Arena a = bias_carve(workspace, workspace_bytes, (size_t)Q, &rm);
  if (!a.ok) return a.fail("bias_mask_head");
  cudaStream_t st = (cudaStream_t)stream;
  // 16-byte path: N a multiple of 4 and all bases 16-byte aligned (torch allocations are)
  const bool vec = (N % 4 == 0) && ((((uintptr_t)geo | (uintptr_t)coords | (uintptr_t)out) & 15) == 0);
  const int work = vec ? N / 4 : N;
  const int rc = bias_mask_rowmax(geo, Q, N, row_max, vec, rm, st);
  if (rc != GF_OK) return rc;
  int gx = (work + 255) / 256;
  int cap = (num_sms() * 16 + Q - 1) / Q;
  if (cap < 1) cap = 1;
  if (gx > cap) gx = cap;
  if (vec)
    bias_mask_write_kernel<true><<<dim3(gx, Q), 256, 0, st>>>(geo, coords, seed_xyz, Q, N, rm.rowmax, rm.gmax, out);
  else
    bias_mask_write_kernel<false><<<dim3(gx, Q), 256, 0, st>>>(geo, coords, seed_xyz, Q, N, rm.rowmax, rm.gmax, out);
  GF_LAUNCHED();
  return GF_OK;
}
