// The mask head of GeoFormerFS fused into one pass over the geodesic maps, for sm_100a (tcgen05 / TMEM).
//
// Reference: model/geoformer/geoformer_fs.py:263-300 (mask_heads_forward), for one scene with m = 16:
//     rel[q,:,n]  = mask-head epilogue a11 (gf_bias.cu, bias_mask_write_kernel): seed - point, pushed out by
//                   sqrt(rowmax) * sign where the point is unreachable
//     x[q,:,n]    = [rel[q,0..2,n], feats[n,0..15]]                        (:291-293, torch.cat)
//     h[q,j,n]    = b0[q*16+j] + sum_c w0[q*16+j, c] x[q,c,n]               (:294-297, grouped conv1d, relu)
//     logit[q,n]  = b1[q] + sum_j w1[q,j] relu(h[q,j,n])
// The reference materialises (Q,16,N) and (Q,19,N) tensors (about 7 GB at Q = 256, N = 100k).  Here:
//   * Only the feature part W0f feats (K = 16) runs on the tensor cores: D (128 points x 256 columns) = feats tile
//     (128 x K) times the weights of a group of 16 queries (256 rows = 16 queries x 16 channels, K-major).  K is
//     padded to a 128-byte swizzled row so that the attention kernel's descriptors apply; only the two K = 8 steps
//     of the real channels are issued.
//   * The three coordinate channels stay fp32 on the CUDA cores in the epilogue, computed from rel exactly as a11
//     computes it (same mask_push, gf_bias.cuh), so every unreachable decision is bit-identical to a11.
//   * TMEM lane = point: one thread owns one point; its geo loads and logit stores are coalesced across the warp,
//     the sum over j is a per-thread loop over its TMEM columns, the per-(q,j) constants are warp-uniform
//     shared-memory reads.  16 warps: warp w reads TMEM lanes 32 (w & 3).. and the 4 queries 4 (w >> 2).. of a group.
//   * Two 256-column TMEM buffers: the product of query group g+1 is issued before the threads drain group g.
//   * Persistent CTAs own 128-point tiles and loop over all query groups; the (Q*16) x 16 weight operand stays in L2.
// The backward kernel is the same code with another epilogue: it recomputes h with the forward's products (so h and
// the ReLU masks are bit-identical to the forward's) and reduces in a fixed order without atomics.
#include "gf_bias.cuh"
#include "gf_umma.cuh"

namespace gf {

constexpr int MH_M = 16;         // mask feature channels (config/geoformer_fs_scannet.yaml: m = 16)
constexpr int MH_CIN = MH_M + 3; // input channels of the first dynamic conv
constexpr int MH_TILE = 128;     // points per tile = MMA M = TMEM lanes
constexpr int MH_QG = 16;        // queries per group
constexpr int MH_COLS = MH_QG * MH_M;  // MMA N = 256 TMEM columns per buffer
constexpr int MH_THREADS = 512;
constexpr int MH_A_BYTES = MH_TILE * 128;  // feats tile: 128 rows of one swizzled 128-byte row (32 fp32, 16 used)
constexpr int MH_B_BYTES = MH_COLS * 128;  // weights of one group: 256 rows
constexpr int MH_NPART = 384;              // per-query partial sums of the backward (see MhConst below)
constexpr uint32_t MH_IDESC = umma_idesc_tf32(128, MH_COLS);

// per-group constants, staged in shared memory next to the group's weight operand
struct MhConst {
  float4 wr[MH_COLS];  // (q,j): w0[., 0..2] (the coordinate channels), b0
  float w1[MH_COLS];   // (q,j)
  float4 seed[MH_QG];  // q: seed xyz, sqrt(rowmax)
  float b1[MH_QG];
};
constexpr int MH_C_BYTES = (sizeof(MhConst) + 1023) / 1024 * 1024;
constexpr int MH_PART_BYTES = 4 * MH_QG * MH_NPART * 4;  // backward: per lane quarter, query and partial sum
constexpr int MH_SMEM = MH_A_BYTES + 2 * MH_B_BYTES + 2 * MH_C_BYTES + 1024;
constexpr int MH_BWD_SMEM = MH_SMEM + MH_PART_BYTES;

struct MhArgs {
  const float *geo;               // (Q, N)
  const float *feats;             // (N, 16)
  const float *w0, *b0, *w1, *b1; // (Q*16, 19), (Q*16), (Q, 16), (Q)
  const float *coords, *seed_xyz; // (N, 3), (Q, 3)
  const uint32_t *rowmax, *gmax;  // ordered-uint row maxima and their maximum (bias_mask_rowmax)
  int Q, N;
  float *out;                     // (Q, N) logits
  // backward
  const float *dlogit;            // (Q, N)
  float *dfeats;                  // (N, 16)
  float *part;                    // (gridDim.x, Q, 384) per-CTA partial sums of the weight gradients
};

__device__ __forceinline__ void mh_sync_for_mma() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

// the group's weight operand (row ql*16 + j, column c = w0[q*16+j, 3+c]) and constants; queries past Q are zero
__device__ __forceinline__ void mh_stage_group(const MhArgs &a, int g, unsigned char *sB, MhConst *sc, unsigned tid) {
  {
    const int r = (int)(tid >> 1), c0 = (int)(tid & 1u) * 8;
    const int q = g * MH_QG + (r >> 4);
    float v[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = q < a.Q ? __ldg(a.w0 + ((size_t)g * MH_COLS + r) * MH_CIN + 3 + c0 + i) : 0.f;
    *reinterpret_cast<float4 *>(sB + sw128_off<MH_COLS>(r, c0)) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4 *>(sB + sw128_off<MH_COLS>(r, c0 + 4)) = make_float4(v[4], v[5], v[6], v[7]);
  }
  if (tid < MH_COLS) {
    const int q = g * MH_QG + (int)(tid >> 4);
    const size_t row = (size_t)g * MH_COLS + tid;
    float4 w = make_float4(0.f, 0.f, 0.f, 0.f);
    float w1 = 0.f;
    if (q < a.Q) {
      w = make_float4(__ldg(a.w0 + row * MH_CIN), __ldg(a.w0 + row * MH_CIN + 1), __ldg(a.w0 + row * MH_CIN + 2),
                      __ldg(a.b0 + row));
      w1 = __ldg(a.w1 + row);
    }
    sc->wr[tid] = w;
    sc->w1[tid] = w1;
  } else if (tid < MH_COLS + MH_QG) {
    const int ql = (int)tid - MH_COLS, q = g * MH_QG + ql;
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    float b1 = 0.f;
    if (q < a.Q) {
      float m = ord2f(a.rowmax[q]);
      if (m < 0.f) m = ord2f(*a.gmax);  // :276
      s = make_float4(a.seed_xyz[q * 3 + 0], a.seed_xyz[q * 3 + 1], a.seed_xyz[q * 3 + 2], sqrtf(m));  // :277
      b1 = __ldg(a.b1 + q);
    }
    sc->seed[ql] = s;
    sc->b1[ql] = b1;
  }
}

// h of one (query, channel): the product's feature part d, then b0 and the fp32 coordinate channels
__device__ __forceinline__ float mh_hidden(float d, float4 w, float r0, float r1, float r2) {
  return __fmaf_rn(w.z, r2, __fmaf_rn(w.y, r1, __fmaf_rn(w.x, r0, __fadd_rn(d, w.w))));
}

// torch.relu: NaN stays NaN (fmaxf would drop it)
__device__ __forceinline__ float mh_relu(float h) { return h < 0.f ? 0.f : h; }

// sum of v[i] over the 32 lanes for all 32 i in 31 shuffles: lane l returns the sum of v[l].  Fixed order.
__device__ __forceinline__ float mh_warp_reduce32(float (&v)[32], unsigned lane) {
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

// BWD = false: logits.  BWD = true: dfeats and the per-CTA partial sums of the weight gradients, per query
// [0, 256): dw0 feature part (j*16 + c), [256, 384): (j*8 + t), t = 0 dw1, 1 db0, 2..4 dw0 coordinate part, 5 db1 (j = 0)
template <bool BWD>
__global__ void __launch_bounds__(MH_THREADS, 1) mask_head_kernel(const MhArgs a) {
  extern __shared__ unsigned char mh_smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[2];
  __shared__ uint32_t s_tmem;
  const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  const unsigned lq = warp & 3u, qq = warp >> 2;  // TMEM lane quarter, query quarter of the group
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(mh_smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char *sA = smem, *sB = sA + MH_A_BYTES, *sCraw = sB + 2 * MH_B_BYTES;
  float *sPart = reinterpret_cast<float *>(sCraw + 2 * MH_C_BYTES);  // BWD only
  const uint32_t mbar0 = smem_u32(&s_mbar[0]), mbar1 = smem_u32(&s_mbar[1]);
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar0) : "memory");
    asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar1) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  mh_sync_for_mma();
  const uint32_t tmem = s_tmem;
  const uint32_t t_lane = tmem + ((lq * 32u) << 16) + qq * 64u;
  const uint32_t sA_s = smem_u32(sA), sB_s = smem_u32(sB);
  const int G = (a.Q + MH_QG - 1) / MH_QG, T = (a.N + MH_TILE - 1) / MH_TILE;
  float *part = BWD ? a.part + (size_t)blockIdx.x * a.Q * MH_NPART : nullptr;

  auto issue = [&](uint32_t k) {  // group k of this CTA (running count): TMEM buffer and mbarrier k & 1
    const uint32_t buf = k & 1u;
#pragma unroll
    for (int kk = 0; kk < 2; ++kk)
      umma_tf32<MH_IDESC>(tmem + buf * MH_COLS, umma_desc(sA_s + kk * 32), umma_desc(sB_s + buf * MH_B_BYTES + kk * 32),
                          kk > 0);
    umma_commit(buf ? mbar1 : mbar0);
  };

  uint32_t it = 0;
  bool first_tile = true;
  for (int tile = blockIdx.x; tile < T; tile += gridDim.x) {
    const int p = (int)(lq * 32u + lane), n = tile * MH_TILE + p;
    const bool valid = n < a.N;
    {  // feats tile: row = point (zero past N), 16 channels of the 32-float swizzled row
      const int r = (int)(tid >> 2), c0 = (int)(tid & 3u) * 4, nr = tile * MH_TILE + r;
      float4 f = make_float4(0.f, 0.f, 0.f, 0.f);
      if (nr < a.N) {
        const float *src = a.feats + (size_t)nr * MH_M + c0;
        f = make_float4(__ldg(src), __ldg(src + 1), __ldg(src + 2), __ldg(src + 3));
      }
      *reinterpret_cast<float4 *>(sA + sw128_off<MH_TILE>(r, c0)) = f;
    }
    const float px = valid ? __ldg(a.coords + (size_t)n * 3 + 0) : 0.f, py = valid ? __ldg(a.coords + (size_t)n * 3 + 1) : 0.f,
                pz = valid ? __ldg(a.coords + (size_t)n * 3 + 2) : 0.f;
    float fx[BWD ? MH_M : 1], dfa[BWD ? MH_M : 1];
    if (BWD) {
#pragma unroll
      for (int c = 0; c < MH_M; ++c) {
        fx[c] = valid ? __ldg(a.feats + (size_t)n * MH_M + c) : 0.f;
        dfa[c] = 0.f;
      }
    }
    mh_stage_group(a, 0, sB + (it & 1u) * MH_B_BYTES, reinterpret_cast<MhConst *>(sCraw + (it & 1u) * MH_C_BYTES), tid);
    mh_sync_for_mma();
    if (tid == 0) issue(it);

    for (int g = 0; g < G; ++g) {
      const uint32_t cur = it + (uint32_t)g, buf = cur & 1u;
      // map entries (and upstream gradients) of this warp's 4 queries, in flight while the product runs
      float gv[4], dl[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int q = g * MH_QG + (int)qq * 4 + i;
        const bool live = valid && q < a.Q;
        gv[i] = live ? __ldg(a.geo + (size_t)q * a.N + n) : 0.f;
        dl[i] = BWD && live ? __ldg(a.dlogit + (size_t)q * a.N + n) : 0.f;
      }
      if (g + 1 < G) {
        mh_stage_group(a, g + 1, sB + (buf ^ 1u) * MH_B_BYTES, reinterpret_cast<MhConst *>(sCraw + (buf ^ 1u) * MH_C_BYTES), tid);
        mh_sync_for_mma();
        if (tid == 0) issue(cur + 1);
      }
      mbar_wait(buf ? mbar1 : mbar0, (cur >> 1) & 1u);
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const MhConst *sc = reinterpret_cast<const MhConst *>(sCraw + buf * MH_C_BYTES);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int ql = (int)qq * 4 + i, q = g * MH_QG + ql;
        float d[16];
        tmem_ld16(t_lane + buf * MH_COLS + (uint32_t)i * 16u, d);  // every lane: .sync.aligned
        if (q >= a.Q) continue;  // warp-uniform
        const float4 sd = sc->seed[ql];
        const bool un = gv[i] < 0.f;
        const float r0 = mask_push(__fsub_rn(sd.x, px), sd.w, un), r1 = mask_push(__fsub_rn(sd.y, py), sd.w, un),
                    r2 = mask_push(__fsub_rn(sd.z, pz), sd.w, un);
        if (!BWD) {
          float o = sc->b1[ql];
#pragma unroll
          for (int j = 0; j < MH_M; ++j) {
            const int col = ql * MH_M + j;
            o = __fmaf_rn(sc->w1[col], mh_relu(mh_hidden(d[j], sc->wr[col], r0, r1, r2)), o);
          }
          if (valid) __stcs(a.out + (size_t)q * a.N + n, o);
        } else {
          const float gl = dl[i];
          float grh[MH_M], dh[MH_M];
#pragma unroll
          for (int j = 0; j < MH_M; ++j) {
            const int col = ql * MH_M + j;
            const float h = mh_hidden(d[j], sc->wr[col], r0, r1, r2);
            grh[j] = __fmul_rn(gl, mh_relu(h));
            dh[j] = h <= 0.f ? 0.f : __fmul_rn(gl, sc->w1[col]);  // torch's ReLU backward: a NaN h passes g
          }
          float *dst = sPart + ((size_t)lq * MH_QG + ql) * MH_NPART;
          // dw1, db0, dw0 coordinate part (and db1): four channels j per 32-value chunk
#pragma unroll
          for (int j4 = 0; j4 < MH_M; j4 += 4) {
            float v[32];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const float x = dh[j4 + jj];
              v[jj * 8 + 0] = grh[j4 + jj];
              v[jj * 8 + 1] = x;
              v[jj * 8 + 2] = __fmul_rn(x, r0);
              v[jj * 8 + 3] = __fmul_rn(x, r1);
              v[jj * 8 + 4] = __fmul_rn(x, r2);
              v[jj * 8 + 5] = (j4 + jj == 0) ? gl : 0.f;
              v[jj * 8 + 6] = 0.f;
              v[jj * 8 + 7] = 0.f;
            }
            dst[256 + j4 * 8 + lane] = mh_warp_reduce32(v, lane);
          }
          // dw0 feature part: two channels j per chunk; dfeats += dh w0f in fixed (q, j) order
#pragma unroll
          for (int jp = 0; jp < MH_M; jp += 2) {
            float v[32];
#pragma unroll
            for (int jj = 0; jj < 2; ++jj) {
              const int row = ql * MH_M + jp + jj;
#pragma unroll
              for (int c4 = 0; c4 < MH_M; c4 += 4) {
                const float4 w = *reinterpret_cast<const float4 *>(sB + buf * MH_B_BYTES + sw128_off<MH_COLS>(row, c4));
                dfa[c4 + 0] = __fmaf_rn(dh[jp + jj], w.x, dfa[c4 + 0]);
                dfa[c4 + 1] = __fmaf_rn(dh[jp + jj], w.y, dfa[c4 + 1]);
                dfa[c4 + 2] = __fmaf_rn(dh[jp + jj], w.z, dfa[c4 + 2]);
                dfa[c4 + 3] = __fmaf_rn(dh[jp + jj], w.w, dfa[c4 + 3]);
              }
#pragma unroll
              for (int c = 0; c < MH_M; ++c) v[jj * 16 + c] = __fmul_rn(dh[jp + jj], fx[c]);
            }
            dst[jp * 16 + lane] = mh_warp_reduce32(v, lane);
          }
        }
      }
      // TMEM buffer, constants (and partial sums) of this group are free once every thread is past this point
      asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
      __syncthreads();
      if (BWD) {  // the tile's sums over its four lane quarters, added to this CTA's partials in tile order
        for (int e = (int)tid; e < MH_QG * MH_NPART; e += MH_THREADS) {
          const int ql = e / MH_NPART, q = g * MH_QG + ql;
          if (q >= a.Q) continue;
          float s = sPart[e];
          s = __fadd_rn(s, sPart[MH_QG * MH_NPART + e]);
          s = __fadd_rn(s, sPart[2 * MH_QG * MH_NPART + e]);
          s = __fadd_rn(s, sPart[3 * MH_QG * MH_NPART + e]);
          float *pp = part + (size_t)g * MH_QG * MH_NPART + e;
          *pp = first_tile ? s : __fadd_rn(*pp, s);
        }
        __syncthreads();
      }
    }
    it += (uint32_t)G;
    if (BWD) {  // dfeats of the tile: the four query quarters summed in order
      float *sD = sPart;
#pragma unroll
      for (int c = 0; c < MH_M; ++c) sD[((size_t)qq * MH_TILE + p) * MH_M + c] = dfa[c];
      __syncthreads();
      for (int e = (int)tid; e < MH_TILE * MH_M; e += MH_THREADS) {
        const int pr = e / MH_M, nr = tile * MH_TILE + pr;
        if (nr >= a.N) continue;
        float s = sD[e];
        s = __fadd_rn(s, sD[MH_TILE * MH_M + e]);
        s = __fadd_rn(s, sD[2 * MH_TILE * MH_M + e]);
        s = __fadd_rn(s, sD[3 * MH_TILE * MH_M + e]);
        a.dfeats[(size_t)nr * MH_M + (e - pr * MH_M)] = s;
      }
      __syncthreads();
    }
    first_tile = false;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
  }
}

// the weight gradients: per (query, partial) the CTAs' partial sums in CTA order, scattered to the callers' layouts
__global__ void __launch_bounds__(256) mask_head_bwd_finish_kernel(const float *__restrict__ part, int nparts, int Q,
                                                                   float *__restrict__ dw0, float *__restrict__ db0,
                                                                   float *__restrict__ dw1, float *__restrict__ db1) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= Q * MH_NPART) return;
  float s = 0.f;
  for (int b = 0; b < nparts; ++b) s = __fadd_rn(s, part[(size_t)b * Q * MH_NPART + e]);
  const int q = e / MH_NPART, k = e - q * MH_NPART;
  if (k < 256) {
    const int j = k >> 4, c = k & 15;
    dw0[((size_t)q * MH_M + j) * MH_CIN + 3 + c] = s;
    return;
  }
  const int j = (k - 256) >> 3, t = (k - 256) & 7;
  const size_t row = (size_t)q * MH_M + j;
  if (t == 0) dw1[row] = s;
  else if (t == 1) db0[row] = s;
  else if (t <= 4) dw0[row * MH_CIN + (t - 2)] = s;
  else if (t == 5 && j == 0) db1[q] = s;
}

static int mh_set_smem() {
  static int done[64] = {0};
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (!__atomic_load_n(&done[dev], __ATOMIC_ACQUIRE)) {
    GF_CUDA(cudaFuncSetAttribute(mask_head_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MH_SMEM));
    GF_CUDA(cudaFuncSetAttribute(mask_head_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MH_BWD_SMEM));
    __atomic_store_n(&done[dev], 1, __ATOMIC_RELEASE);
  }
  return GF_OK;
}

static int mh_grid(int N) {
  const int T = (N + MH_TILE - 1) / MH_TILE;
  return T < num_sms() ? T : num_sms();
}

}  // namespace gf

using namespace gf;

extern "C" size_t gf_mask_head_workspace_bytes(int Q, int N) {
  if (Q <= 0 || N <= 0) return 0;
  return align256(sizeof(uint32_t) * (size_t)Q) + 256;
}

extern "C" size_t gf_mask_head_backward_workspace_bytes(int Q, int N) {
  if (Q <= 0 || N <= 0) return 0;
  return gf_mask_head_workspace_bytes(Q, N) + align256(sizeof(float) * (size_t)mh_grid(N) * Q * MH_NPART);
}

// arguments common to both entries; returns the workspace's row maxima
static int mh_prepare(MhArgs &a, const float *geo, const float *feats, const float *w0, const float *b0,
                      const float *w1, const float *b1, const float *coords, const float *seed_xyz,
                      const float *row_max, int Q, int N, Arena &ar, cudaStream_t st) {
  uint32_t *rowmax = ar.take<uint32_t>((size_t)Q);
  uint32_t *gmax = ar.take<uint32_t>(1);
  if (!ar.ok) {
    set_error("mask_head: workspace too small");
    return GF_ERR_WORKSPACE;
  }
  int rc = mh_set_smem();
  if (rc) return rc;
  const bool vec = (N % 4 == 0) && (((uintptr_t)geo & 15) == 0);
  if ((rc = bias_mask_rowmax(geo, Q, N, row_max, vec, rowmax, gmax, st))) return rc;
  a.geo = geo, a.feats = feats, a.w0 = w0, a.b0 = b0, a.w1 = w1, a.b1 = b1, a.coords = coords, a.seed_xyz = seed_xyz;
  a.rowmax = rowmax, a.gmax = gmax, a.Q = Q, a.N = N;
  a.out = nullptr, a.dlogit = nullptr, a.dfeats = nullptr;
  return GF_OK;
}

extern "C" int gf_mask_head_logits(const float *geo, const float *feats, const float *w0, const float *b0,
                                   const float *w1, const float *b1, const float *coords, const float *seed_xyz,
                                   const float *row_max, int Q, int N, int m, float *out, void *workspace,
                                   size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(Q >= 0 && N >= 0, "mask_head: negative size");
  GF_CHECK_ARG(m == MH_M, "mask_head: m=%d (only m = 16 is supported)", m);
  if ((long long)Q * N == 0) return GF_OK;
  GF_CHECK_ARG(geo && feats && w0 && b0 && w1 && b1 && coords && seed_xyz && out, "mask_head: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  Arena ar(workspace, workspace_bytes);
  MhArgs a;
  int rc = mh_prepare(a, geo, feats, w0, b0, w1, b1, coords, seed_xyz, row_max, Q, N, ar, st);
  if (rc) return rc;
  a.out = out;
  mask_head_kernel<false><<<mh_grid(N), MH_THREADS, MH_SMEM, st>>>(a);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_mask_head_logits_backward(const float *geo, const float *feats, const float *w0, const float *b0,
                                            const float *w1, const float *b1, const float *coords,
                                            const float *seed_xyz, const float *row_max, int Q, int N, int m,
                                            const float *dlogit, float *dfeats, float *dw0, float *db0, float *dw1,
                                            float *db1, void *workspace, size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(Q >= 0 && N >= 0, "mask_head_backward: negative size");
  GF_CHECK_ARG(m == MH_M, "mask_head_backward: m=%d (only m = 16 is supported)", m);
  if ((long long)Q * N != 0)
    GF_CHECK_ARG(geo && feats && w0 && b0 && w1 && b1 && coords && seed_xyz && dlogit && dfeats && dw0 && db0 && dw1 &&
                     db1,
                 "mask_head_backward: null pointer");
  cudaStream_t st = (cudaStream_t)stream;
  if ((long long)Q * N == 0) {  // no (query, point) pair: every gradient is zero
    if (N > 0 && dfeats) GF_CUDA(cudaMemsetAsync(dfeats, 0, sizeof(float) * (size_t)N * MH_M, st));
    if (Q > 0 && dw0) GF_CUDA(cudaMemsetAsync(dw0, 0, sizeof(float) * (size_t)Q * MH_M * MH_CIN, st));
    if (Q > 0 && db0) GF_CUDA(cudaMemsetAsync(db0, 0, sizeof(float) * (size_t)Q * MH_M, st));
    if (Q > 0 && dw1) GF_CUDA(cudaMemsetAsync(dw1, 0, sizeof(float) * (size_t)Q * MH_M, st));
    if (Q > 0 && db1) GF_CUDA(cudaMemsetAsync(db1, 0, sizeof(float) * (size_t)Q, st));
    return GF_OK;
  }
  Arena ar(workspace, workspace_bytes);
  MhArgs a;
  const int grid = mh_grid(N);
  int rc = mh_prepare(a, geo, feats, w0, b0, w1, b1, coords, seed_xyz, row_max, Q, N, ar, st);
  if (rc) return rc;
  a.part = ar.take<float>((size_t)grid * Q * MH_NPART);
  if (!ar.ok) {
    set_error("mask_head_backward: workspace too small");
    return GF_ERR_WORKSPACE;
  }
  a.dlogit = dlogit, a.dfeats = dfeats;
  mask_head_kernel<true><<<grid, MH_THREADS, MH_BWD_SMEM, st>>>(a);
  GF_LAUNCHED();
  mask_head_bwd_finish_kernel<<<(Q * MH_NPART + 255) / 256, 256, 0, st>>>(a.part, grid, Q, dw0, db0, dw1, db1);
  GF_LAUNCHED();
  return GF_OK;
}
