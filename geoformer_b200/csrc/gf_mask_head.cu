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
#include "gf_mask_head_tile.cuh"
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
  }
}

// partial sum k of query q (the layout of mask_head_kernel<true>'s partials) to the callers' gradient layouts
__device__ __forceinline__ void mh_scatter_grad(float s, int q, int k, float *__restrict__ dw0, float *__restrict__ db0,
                                                float *__restrict__ dw1, float *__restrict__ db1) {
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

// the weight gradients: per (query, partial) the CTAs' partial sums in CTA order, scattered to the callers' layouts
__global__ void __launch_bounds__(256) mask_head_bwd_finish_kernel(const float *__restrict__ part, int nparts, int Q,
                                                                   float *__restrict__ dw0, float *__restrict__ db0,
                                                                   float *__restrict__ dw1, float *__restrict__ db1) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= Q * MH_NPART) return;
  float s = 0.f;
  for (int b = 0; b < nparts; ++b) s = __fadd_rn(s, part[(size_t)b * Q * MH_NPART + e]);
  const int q = e / MH_NPART, k = e - q * MH_NPART;
  mh_scatter_grad(s, q, k, dw0, db0, dw1, db1);
}

// ---- ragged batches: up to MH_BATCH_MAX scenes in one launch ------------------------------------------------------
// The tiles of all scenes form one space: scene b owns the global tiles [tile0[b], tile0[b+1]), its tile i holding
// points 128 i.. of the scene (a tile never straddles two scenes).  CTA c takes the contiguous tiles
// [mh_range(c), mh_range(c + 1)).  The backward keeps one partial row per (CTA, scene) segment: the CTAs whose range
// meets scene b are cfirst[b].. in order, and their segments are seg0[b].. in the same order, at most
// grid + B - 1 segments in all.
struct MhBatchArgs {
  const float *geo[MH_BATCH_MAX];  // scene b's (Q, N_b) maps
  int off[MH_BATCH_MAX + 1];       // offsets: scene b is points off[b] .. off[b+1] of the flat arrays
  int tile0[MH_BATCH_MAX + 1];
  int seg0[MH_BATCH_MAX + 1];
  int cfirst[MH_BATCH_MAX];
  int B, Q;
  const float *feats, *coords;     // (sum N, 16), (sum N, 3)
  const float *w0, *b0, *w1, *b1;  // stacked: scene b's queries are rows b*Q ..
  const float *seed_xyz;           // (B, Q, 3)
  const uint32_t *rowmax, *gmax;   // (B, Q), (B): each scene's own maximum
  float *out;                      // scene b's (Q, N_b) block at Q * off[b]
  const float *dlogit;             // as out
  float *dfeats;                   // (sum N, 16)
  float *part;                     // (segments, Q, 384)
};

__host__ __device__ __forceinline__ int mh_range(int c, int T, int grid) { return (int)((long long)c * T / grid); }

// mask_head_kernel<BWD> over the tiles of a batch; each tile runs the single-scene kernel's tile body on its scene
template <bool BWD>
__global__ void __launch_bounds__(MH_THREADS, 1) mask_head_batch_kernel(const __grid_constant__ MhBatchArgs ba) {
  extern __shared__ unsigned char mh_smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[2];
  __shared__ uint32_t s_tmem;
  const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  const unsigned lq = warp & 3u, qq = warp >> 2;
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
  const int Q = ba.Q, G = (Q + MH_QG - 1) / MH_QG, T = ba.tile0[ba.B];

  auto issue = [&](uint32_t k) {
    const uint32_t buf = k & 1u;
#pragma unroll
    for (int kk = 0; kk < 2; ++kk)
      umma_tf32<MH_IDESC>(tmem + buf * MH_COLS, umma_desc(sA_s + kk * 32), umma_desc(sB_s + buf * MH_B_BYTES + kk * 32),
                          kk > 0);
    umma_commit(buf ? mbar1 : mbar0);
  };

  uint32_t it = 0;
  const int t0 = mh_range((int)blockIdx.x, T, (int)gridDim.x), t1 = mh_range((int)blockIdx.x + 1, T, (int)gridDim.x);
  int b = 0;
  for (int t = t0; t < t1; ++t) {
    while (t >= ba.tile0[b + 1]) ++b;
    const int tile = t - ba.tile0[b], n0 = ba.off[b];
    bool first_tile = t == t0 || tile == 0;  // a new (CTA, scene) segment
    const size_t qb = (size_t)b * Q;
    MhArgs a;
    a.geo = ba.geo[b], a.Q = Q, a.N = ba.off[b + 1] - n0;
    a.feats = ba.feats + (size_t)n0 * MH_M, a.coords = ba.coords + (size_t)n0 * 3;
    a.w0 = ba.w0 + qb * MH_M * MH_CIN, a.b0 = ba.b0 + qb * MH_M, a.w1 = ba.w1 + qb * MH_M, a.b1 = ba.b1 + qb;
    a.seed_xyz = ba.seed_xyz + qb * 3, a.rowmax = ba.rowmax + qb, a.gmax = ba.gmax + b;
    a.out = BWD ? nullptr : ba.out + (size_t)Q * n0;
    a.dlogit = BWD ? ba.dlogit + (size_t)Q * n0 : nullptr;
    a.dfeats = BWD ? ba.dfeats + (size_t)n0 * MH_M : nullptr;
    a.part = nullptr;
    float *part = BWD ? ba.part + (size_t)(ba.seg0[b] + (int)blockIdx.x - ba.cfirst[b]) * Q * MH_NPART : nullptr;
#include "gf_mask_head_tile.cuh"
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
  }
}

struct MhSegments {
  int seg0[MH_BATCH_MAX + 1];
};

// the weight gradients of a batch: per (scene, query, partial) the scene's segments summed in CTA order
__global__ void __launch_bounds__(256) mask_head_batch_bwd_finish_kernel(const float *__restrict__ part,
                                                                         const __grid_constant__ MhSegments sg, int B,
                                                                         int Q, float *__restrict__ dw0,
                                                                         float *__restrict__ db0,
                                                                         float *__restrict__ dw1,
                                                                         float *__restrict__ db1) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= B * Q * MH_NPART) return;
  const int qg = e / MH_NPART, k = e - qg * MH_NPART, b = qg / Q, q = qg - b * Q;
  float s = 0.f;
  for (int seg = sg.seg0[b]; seg < sg.seg0[b + 1]; ++seg) s = __fadd_rn(s, part[((size_t)seg * Q + q) * MH_NPART + k]);
  mh_scatter_grad(s, qg, k, dw0, db0, dw1, db1);
}

static int mh_set_smem() {
  static int done[64] = {0};
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (!__atomic_load_n(&done[dev], __ATOMIC_ACQUIRE)) {
    GF_CUDA(cudaFuncSetAttribute(mask_head_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MH_SMEM));
    GF_CUDA(cudaFuncSetAttribute(mask_head_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, MH_BWD_SMEM));
    GF_CUDA(cudaFuncSetAttribute(mask_head_batch_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, MH_SMEM));
    GF_CUDA(cudaFuncSetAttribute(mask_head_batch_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 MH_BWD_SMEM));
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

// the workspace: the row maxima of the maps, and for the backward the per-CTA partial sums of the weight gradients
struct MhLayout {
  RowMax rm;
  float *part;
};
static Arena mh_carve(void *workspace, size_t workspace_bytes, int Q, int N, bool backward, MhLayout *l) {
  Arena a(workspace, workspace_bytes);
  l->rm = take_rowmax(a, (size_t)Q);
  l->part = backward ? a.take<float>((size_t)mh_grid(N) * Q * MH_NPART) : nullptr;
  return a;
}

extern "C" size_t gf_mask_head_workspace_bytes(int Q, int N) {
  if (Q <= 0 || N <= 0) return 0;
  MhLayout l;
  return mh_carve(nullptr, 0, Q, N, false, &l).off;
}

extern "C" size_t gf_mask_head_backward_workspace_bytes(int Q, int N) {
  if (Q <= 0 || N <= 0) return 0;
  MhLayout l;
  return mh_carve(nullptr, 0, Q, N, true, &l).off;
}

// arguments common to both entries, and the row maxima into the carved workspace
static int mh_prepare(MhArgs &a, const float *geo, const float *feats, const float *w0, const float *b0,
                      const float *w1, const float *b1, const float *coords, const float *seed_xyz,
                      const float *row_max, int Q, int N, const MhLayout &l, cudaStream_t st) {
  int rc = mh_set_smem();
  if (rc) return rc;
  const bool vec = (N % 4 == 0) && (((uintptr_t)geo & 15) == 0);
  if ((rc = bias_mask_rowmax(geo, Q, N, row_max, vec, l.rm, st))) return rc;
  a.geo = geo, a.feats = feats, a.w0 = w0, a.b0 = b0, a.w1 = w1, a.b1 = b1, a.coords = coords, a.seed_xyz = seed_xyz;
  a.rowmax = l.rm.rowmax, a.gmax = l.rm.gmax, a.Q = Q, a.N = N;
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
  MhLayout l;
  const Arena ar = mh_carve(workspace, workspace_bytes, Q, N, false, &l);
  if (!ar.ok) return ar.fail("mask_head");
  MhArgs a;
  int rc = mh_prepare(a, geo, feats, w0, b0, w1, b1, coords, seed_xyz, row_max, Q, N, l, st);
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
  MhLayout l;
  const Arena ar = mh_carve(workspace, workspace_bytes, Q, N, true, &l);
  if (!ar.ok) return ar.fail("mask_head_backward");
  MhArgs a;
  const int grid = mh_grid(N);
  int rc = mh_prepare(a, geo, feats, w0, b0, w1, b1, coords, seed_xyz, row_max, Q, N, l, st);
  if (rc) return rc;
  a.part = l.part;
  a.dlogit = dlogit, a.dfeats = dfeats;
  mask_head_kernel<true><<<grid, MH_THREADS, MH_BWD_SMEM, st>>>(a);
  GF_LAUNCHED();
  mask_head_bwd_finish_kernel<<<(Q * MH_NPART + 255) / 256, 256, 0, st>>>(a.part, grid, Q, dw0, db0, dw1, db1);
  GF_LAUNCHED();
  return GF_OK;
}

// ---- ragged batches -------------------------------------------------------------------------------------------------
// the sizes of a batched call: 1..32 scenes, offsets from 0 rising strictly (no empty scene), Q >= 1
static int mh_batch_sizes(const int *offsets, int B, int Q, const char *who) {
  GF_CHECK_ARG(B >= 1 && B <= MH_BATCH_MAX, "%s: B=%d (1 to %d scenes per call)", who, B, MH_BATCH_MAX);
  GF_CHECK_ARG(Q >= 1, "%s: Q=%d (at least one query)", who, Q);
  GF_CHECK_ARG((long long)B * Q * MH_NPART < (1LL << 31), "%s: B*Q=%lld queries is too many", who, (long long)B * Q);
  GF_CHECK_ARG(offsets, "%s: null pointer (offsets)", who);
  GF_CHECK_ARG(offsets[0] == 0, "%s: offsets[0]=%d (must start at 0)", who, offsets[0]);
  for (int b = 0; b < B; ++b)
    GF_CHECK_ARG(offsets[b + 1] > offsets[b], "%s: scene %d is empty (offsets must rise strictly)", who, b);
  return GF_OK;
}

// the partition of a batched call's tiles over the CTAs (see MhBatchArgs) and its segment count
static void mh_batch_plan(const int *offsets, int B, int Q, MhBatchArgs *a, int *grid, int *nseg) {
  a->B = B, a->Q = Q;
  a->tile0[0] = 0;
  for (int b = 0; b <= B; ++b) a->off[b] = offsets[b];
  for (int b = 0; b < B; ++b) a->tile0[b + 1] = a->tile0[b] + (offsets[b + 1] - offsets[b] + MH_TILE - 1) / MH_TILE;
  const int T = a->tile0[B], g = T < num_sms() ? T : num_sms();
  auto owner = [&](int t) { return (int)(((long long)(t + 1) * g - 1) / T); };  // the c with t in [mh_range(c), ..)
  a->seg0[0] = 0;
  for (int b = 0; b < B; ++b) {
    a->cfirst[b] = owner(a->tile0[b]);
    a->seg0[b + 1] = a->seg0[b] + owner(a->tile0[b + 1] - 1) - a->cfirst[b] + 1;
  }
  *grid = g;
  *nseg = a->seg0[B];
}

// the workspace of a batched call: the row maxima (B, Q) with each scene's maximum (B) right after them (one zero
// fill clears both), and for the backward one partial row per segment
struct MhBatchLayout {
  uint32_t *rowmax, *gmax;
  float *part;
};
static Arena mh_batch_carve(void *workspace, size_t workspace_bytes, int B, int Q, int nseg, bool backward,
                            MhBatchLayout *l) {
  Arena a(workspace, workspace_bytes);
  uint32_t *r = a.take<uint32_t>((size_t)B * Q + B);
  l->rowmax = r, l->gmax = r ? r + (size_t)B * Q : nullptr;
  l->part = backward ? a.take<float>((size_t)nseg * Q * MH_NPART) : nullptr;
  return a;
}

static size_t mh_batch_workspace_bytes(const int *offsets, int B, int Q, bool backward) {
  if (mh_batch_sizes(offsets, B, Q, "mask_head_batch_workspace_bytes")) return 0;
  MhBatchArgs a;
  int grid, nseg;
  mh_batch_plan(offsets, B, Q, &a, &grid, &nseg);
  MhBatchLayout l;
  return mh_batch_carve(nullptr, 0, B, Q, nseg, backward, &l).off;
}

extern "C" size_t gf_mask_head_batch_workspace_bytes(const int *offsets, int B, int Q) {
  return mh_batch_workspace_bytes(offsets, B, Q, false);
}

extern "C" size_t gf_mask_head_batch_backward_workspace_bytes(const int *offsets, int B, int Q) {
  return mh_batch_workspace_bytes(offsets, B, Q, true);
}

// arguments common to both batched entries
static int mh_batch_check(const float *const *geo, const int *offsets, int B, int Q, int m, const float *feats,
                          const float *w0, const float *b0, const float *w1, const float *b1, const float *coords,
                          const float *seed_xyz, const char *who) {
  int rc = mh_batch_sizes(offsets, B, Q, who);
  if (rc) return rc;
  GF_CHECK_ARG(m == MH_M, "%s: m=%d (only m = 16 is supported)", who, m);
  GF_CHECK_ARG(geo && feats && w0 && b0 && w1 && b1 && coords && seed_xyz, "%s: null pointer", who);
  for (int b = 0; b < B; ++b) GF_CHECK_ARG(geo[b], "%s: null pointer (geo[%d])", who, b);
  return GF_OK;
}

// the plan, the carved workspace and the row maxima, once every argument has been checked
static int mh_batch_prepare(MhBatchArgs &a, int *grid, MhBatchLayout *l, const float *const *geo, const int *offsets,
                            int B, int Q, const float *feats, const float *w0, const float *b0, const float *w1,
                            const float *b1, const float *coords, const float *seed_xyz, const float *row_max,
                            void *workspace, size_t workspace_bytes, bool backward, cudaStream_t st, const char *who) {
  int nseg;
  mh_batch_plan(offsets, B, Q, &a, grid, &nseg);
  const Arena ar = mh_batch_carve(workspace, workspace_bytes, B, Q, nseg, backward, l);
  if (!ar.ok) return ar.fail(who);
  int rc = mh_set_smem();
  if (rc) return rc;
  MaskMaps maps;
  maps.B = B, maps.Q = Q;
  for (int b = 0; b < B; ++b) maps.geo[b] = geo[b], maps.N[b] = offsets[b + 1] - offsets[b], a.geo[b] = geo[b];
  if ((rc = bias_mask_rowmax_batch(maps, row_max, l->rowmax, l->gmax, st))) return rc;
  a.feats = feats, a.coords = coords, a.w0 = w0, a.b0 = b0, a.w1 = w1, a.b1 = b1, a.seed_xyz = seed_xyz;
  a.rowmax = l->rowmax, a.gmax = l->gmax;
  a.out = nullptr, a.dlogit = nullptr, a.dfeats = nullptr, a.part = l->part;
  return GF_OK;
}

extern "C" int gf_mask_head_logits_batch(const float *const *geo, const int *offsets, int B, int Q, int m,
                                         const float *feats, const float *w0, const float *b0, const float *w1,
                                         const float *b1, const float *coords, const float *seed_xyz,
                                         const float *row_max, float *out, void *workspace, size_t workspace_bytes,
                                         void *stream) {
  const char *who = "mask_head_batch";
  int rc = mh_batch_check(geo, offsets, B, Q, m, feats, w0, b0, w1, b1, coords, seed_xyz, who);
  if (rc) return rc;
  GF_CHECK_ARG(out, "%s: null pointer (out)", who);
  cudaStream_t st = (cudaStream_t)stream;
  MhBatchArgs a;
  MhBatchLayout l;
  int grid;
  if ((rc = mh_batch_prepare(a, &grid, &l, geo, offsets, B, Q, feats, w0, b0, w1, b1, coords, seed_xyz, row_max,
                             workspace, workspace_bytes, false, st, who)))
    return rc;
  a.out = out;
  mask_head_batch_kernel<false><<<grid, MH_THREADS, MH_SMEM, st>>>(a);
  GF_LAUNCHED();
  return GF_OK;
}

extern "C" int gf_mask_head_logits_batch_backward(const float *const *geo, const int *offsets, int B, int Q, int m,
                                                  const float *feats, const float *w0, const float *b0,
                                                  const float *w1, const float *b1, const float *coords,
                                                  const float *seed_xyz, const float *row_max, const float *dlogit,
                                                  float *dfeats, float *dw0, float *db0, float *dw1, float *db1,
                                                  void *workspace, size_t workspace_bytes, void *stream) {
  const char *who = "mask_head_batch_backward";
  int rc = mh_batch_check(geo, offsets, B, Q, m, feats, w0, b0, w1, b1, coords, seed_xyz, who);
  if (rc) return rc;
  GF_CHECK_ARG(dlogit && dfeats && dw0 && db0 && dw1 && db1, "%s: null pointer", who);
  cudaStream_t st = (cudaStream_t)stream;
  MhBatchArgs a;
  MhBatchLayout l;
  int grid;
  if ((rc = mh_batch_prepare(a, &grid, &l, geo, offsets, B, Q, feats, w0, b0, w1, b1, coords, seed_xyz, row_max,
                             workspace, workspace_bytes, true, st, who)))
    return rc;
  a.dlogit = dlogit, a.dfeats = dfeats;
  mask_head_batch_kernel<true><<<grid, MH_THREADS, MH_BWD_SMEM, st>>>(a);
  GF_LAUNCHED();
  MhSegments sg;
  for (int b = 0; b <= B; ++b) sg.seg0[b] = a.seg0[b];
  mask_head_batch_bwd_finish_kernel<<<(B * Q * MH_NPART + 255) / 256, 256, 0, st>>>(l.part, sg, B, Q, dw0, db0, dw1,
                                                                                    db1);
  GF_LAUNCHED();
  return GF_OK;
}
