// Decoder vector cross-attention over the geodesic relative-position embedding, for sm_100a (tcgen05 / TMEM).
//
// Reference: model/transformer_detr.py:443-454 (TransformerDecoderLayer.forward_pre_rel, MLPs defined at :384-396):
//     x    = tgt2[q] - memory[c] + relative_pos[q,c]                  (64)      for every (query q, context c)
//     sim  = W2 relu(W1 x + b1) + b2                                   attn_mlp
//     attn = softmax(sim / sqrt(64), over the CONTEXTS, per channel)   :449 (dim=1)
//     v2   = Wv (memory[c] + relative_pos[q,c]) + bv                   v_mlp
//     out  = relu(Wo (sum_c attn * v2) + bo)                           :452-453 (einsum, out_mlp)
// The reference materialises three (Q,C,B,64) tensors besides the embedding (134 MB each at Q=256, C=2048).
// Here one CTA owns one (query, batch element) and walks the contexts in tiles of 128:
//   * The (q,c)-dependent part of both first layers is ONE tensor-core product per tile: [Wv; W1] (128 x 64) times
//     the tile of the embedding (128 contexts x 64), M = 128, N = 128, K = 64 -> TMEM columns 0..127.  The query
//     part W1 tgt2[q] and the context parts W1 memory[c], Wv memory[c] are small matrices computed once per call
//     (aq, P1, Pv) and added in the epilogue: W1 x = W1 tgt2[q] - W1 memory[c] + W1 rel.
//   * Channel-major accumulators: TMEM lane = output channel, column = context.  Lanes 0..63 hold v2, lanes 64..127
//     the hidden layer; the second product [W2; 0] times the hidden tile lands in lanes 0..63 of columns 128..255,
//     i.e. in the SAME threads that hold v2 -- so the softmax over the contexts and the weighted sum are plain
//     per-thread loops over TMEM columns (online softmax, no shuffles, nothing written back).
//   * Operands are fp32 in shared memory, multiplied as TF32 (kind::tf32), accumulated in fp32; K-major tiles in
//     the 128-byte swizzle the UMMA descriptors describe, written by the threads themselves (the embedding is
//     either loaded from the (Q,C,B,64) tensor or -- fused with the decoder epilogue a10 -- computed on the fly
//     from the geodesic maps, so that it never exists in memory).
// tcgen05.mma is issued by one thread; completion is signalled through an mbarrier by tcgen05.commit.
#include "gf_common.cuh"

namespace gf {

constexpr int ATT_D = 64;        // channels (dec_dim of the model, geoformer_fs.py:116)
constexpr int ATT_TILE = 64;     // contexts per tile = MMA N
constexpr int ATT_THREADS = 256;
constexpr int ATT_MAX_B = 8;     // batch elements of the fused variant (map pointers travel in the kernel parameters)
constexpr int ATT_W_HALF = 128 * 128;           // one K-half (32 floats = 128 bytes per row) of a 128-row weight tile
constexpr int ATT_W_BYTES = 2 * ATT_W_HALF;     // [Wv; W1] and [W2; 0]: 128 x 64 fp32
constexpr int ATT_T_HALF = ATT_TILE * 128;      // one K-half of a 64-row operand tile (embedding / hidden)
constexpr int ATT_T_BYTES = 2 * ATT_T_HALF;
constexpr int ATT_SMEM = 2 * ATT_W_BYTES + 4 * ATT_T_BYTES + 1024;  // A1, A2, 2 embedding tiles, 2 hidden tiles
constexpr uint32_t ATT_D1_COL = 0, ATT_D2_COL = 3 * ATT_TILE;       // TMEM: three D1 buffers, two D2 buffers

struct AttArgs {
  const float *aq;   // (B, Q, 64)  W1 tgt2[q] + b1
  const float *p1;   // (B, C, 64)  W1 memory[c]
  const float *pv;   // (B, C, 64)  Wv memory[c] + bv
  const float *w1, *w2, *wv, *wo;  // (64, 64) row-major (out, in): nn.Linear.weight
  const float *b2, *bo;            // (64)
  int Q, C, B;
  // the embedding: either the tensor (Q, C, B, 64) ...
  const float *rel;
  // ... or its ingredients (decoder epilogue a10 + Fourier features, gf_bias.cu: bias_ctx_fourier_kernel)
  const float *geo[ATT_MAX_B];  // (Q, N_b) maps, one per batch element
  int geo_ld[ATT_MAX_B];        // their row strides
  const int *ctx_idx;            // (B, C)
  const float *query_xyz, *ctx_xyz;  // (B, Q, 3), (B, C, 3)
  const uint32_t *rowmax, *gmax;     // ordered-uint row maxima (B, Q) and the global maximum (bias_ctx_rowmax_kernel)
  const float *gauss_B;              // (3, ldb), 32 frequencies used
  int ldb;
  const float *pc_min, *pc_max;      // (B, 3)
  float *out;                        // (Q, B, 64)
  float *o_save, *lse_save;          // SAVE: (Q, B, 64) weighted sum before out_mlp and max + log(sum) of the scores
};

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// K-major tile with 128-byte swizzle, `rows` rows: row r, fp32 column k (0..63) -> byte offset inside the tile
template <int ROWS>
__device__ __forceinline__ uint32_t sw128_off(int r, int k) {
  const int half = k >> 5, kk = k & 31;
  return (uint32_t)(half * (ROWS * 128) + r * 128 + ((((kk >> 2) ^ (r & 7)) << 4) | ((kk & 3) << 2)));
}

// shared-memory matrix descriptor: K-major, SWIZZLE_128B, 8-row groups 1024 bytes apart (cute::UMMA::SmemDescriptor)
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr) {
  return (uint64_t)((saddr & 0x3FFFFu) >> 4) | (1ull << 16) | (64ull << 32) | (1ull << 46) | (2ull << 61);
}

// instruction descriptor (cute::UMMA::InstrDescriptor): D = F32, A = B = TF32, both K-major, M = 128, N = 64
constexpr uint32_t ATT_IDESC = (1u << 4) | (2u << 7) | (2u << 10) | ((ATT_TILE >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      :
      : "r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(ATT_IDESC), "r"(accumulate)
      : "memory");
}

// D (128 x 64, TMEM) (+)= A (128 x 64) * B^T (64 x 64): eight K = 8 steps, 32 bytes apart inside a swizzled row, the
// second half of K in the second half-tile (A_HALF bytes further for A: the A tile may be 128 rows of a taller region)
template <int A_HALF>
__device__ __forceinline__ void umma_k64(uint32_t d_tmem, uint32_t a_saddr, uint32_t b_saddr, bool accumulate) {
#pragma unroll
  for (int kk = 0; kk < 8; ++kk) {
    const uint32_t ka = (uint32_t)((kk >> 2) * A_HALF + (kk & 3) * 32), kb = (uint32_t)((kk >> 2) * ATT_T_HALF + (kk & 3) * 32);
    umma_tf32(d_tmem, umma_desc(a_saddr + ka), umma_desc(b_saddr + kb), accumulate || kk > 0);
  }
}

// the completion of every tcgen05.mma this thread issued so far arrives on `mbar`
__device__ __forceinline__ void umma_commit(uint32_t mbar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(mbar) : "memory");
}

__device__ __forceinline__ void umma_tile(uint32_t d_tmem, uint32_t a_saddr, uint32_t b_saddr, uint32_t mbar) {
  umma_k64<ATT_W_HALF>(d_tmem, a_saddr, b_saddr, false);
  umma_commit(mbar);
}

__device__ __forceinline__ void mbar_wait(uint32_t mbar, uint32_t parity) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "W: mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@!p bra W;\n\t}"
      :
      : "r"(mbar), "r"(parity)
      : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, float (&v)[32]) {
  uint32_t r[32];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < 32; ++i) v[i] = __uint_as_float(r[i]);
}

// The embedding tile of one (query, batch element), row = context, column = channel, in two steps, so that its global
// loads are in flight while the thread does its role's work: fetch(tile) issues them (a quarter of row tid / 4: 16
// floats, or for the fused variant the gathered map entry and the context's coordinates), stash writes the operand
// buffer (fused: after the sin / cos of its eight frequencies).  stash<true> also writes the transposed tile (row =
// channel, column = context) the backward's weight-gradient products take as K-major operand.
template <bool FUSED>
struct EmbTile {
  // ingredients of the fused embedding (gf_bias.cu: bias_ctx_fourier_kernel)
  float fm = 0.f, qx = 0.f, qy = 0.f, qz = 0.f, mn0 = 0.f, mn1 = 0.f, mn2 = 0.f, df0 = 1.f, df1 = 1.f, df2 = 1.f;
  const float *geo_row = nullptr;
  float4 pre[4];
  float n0 = 0.f, n1 = 0.f, n2 = 0.f;
  bool pre_live = false;
  int lr, qd;
  uint32_t st_off[4];  // this thread's four 16-byte chunks of row lr (unfused: columns 16 qd + 4 j; fused: see stash)

  __device__ __forceinline__ EmbTile(const AttArgs &a, int q, int b, unsigned tid) {
    if (FUSED) {
      fm = ord2f(a.rowmax[b * a.Q + q]);
      if (fm < 0.f) fm = ord2f(*a.gmax);  // geoformer_fs.py:693
      qx = a.query_xyz[((size_t)b * a.Q + q) * 3 + 0], qy = a.query_xyz[((size_t)b * a.Q + q) * 3 + 1],
      qz = a.query_xyz[((size_t)b * a.Q + q) * 3 + 2];
      mn0 = a.pc_min[b * 3 + 0], mn1 = a.pc_min[b * 3 + 1], mn2 = a.pc_min[b * 3 + 2];
      df0 = __fsub_rn(a.pc_max[b * 3 + 0], mn0), df1 = __fsub_rn(a.pc_max[b * 3 + 1], mn1),
      df2 = __fsub_rn(a.pc_max[b * 3 + 2], mn2);
      geo_row = a.geo[b] + (size_t)q * a.geo_ld[b];
    }
    lr = (int)(tid >> 2), qd = (int)(tid & 3u);
    // shared-space addresses with the swizzle folded into per-thread constants: no address arithmetic per store
#pragma unroll
    for (int j = 0; j < 4; ++j)
      st_off[j] = FUSED ? sw128_off<ATT_TILE>(lr, (j & 1) * 32 + 8 * qd + 4 * (j >> 1)) : sw128_off<ATT_TILE>(lr, 16 * qd + 4 * j);
  }

  static __device__ __forceinline__ void sts128(uint32_t addr, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
  }
  // the transpose of four consecutive channels k..k+3 of row lr
  __device__ __forceinline__ void sts_t(uint32_t dstT, int k, float4 v) const {
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(dstT + sw128_off<ATT_D>(k + 0, lr)), "f"(v.x) : "memory");
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(dstT + sw128_off<ATT_D>(k + 1, lr)), "f"(v.y) : "memory");
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(dstT + sw128_off<ATT_D>(k + 2, lr)), "f"(v.z) : "memory");
    asm volatile("st.shared.f32 [%0], %1;" ::"r"(dstT + sw128_off<ATT_D>(k + 3, lr)), "f"(v.w) : "memory");
  }

  __device__ __forceinline__ void fetch(const AttArgs &a, int q, int b, int tile) {
    const int c = tile * ATT_TILE + lr;
    pre_live = c < a.C;
    if (!FUSED) {
      const float4 *src = reinterpret_cast<const float4 *>(a.rel + (((size_t)q * a.C + (pre_live ? c : 0)) * a.B + b) * 64) + 4 * qd;
#pragma unroll
      for (int j = 0; j < 4; ++j) pre[j] = pre_live ? __ldg(src + j) : make_float4(0.f, 0.f, 0.f, 0.f);
    } else {
      n0 = n1 = n2 = 0.f;
      if (pre_live) {
        const float g = __ldg(geo_row + __ldg(a.ctx_idx + (size_t)b * a.C + c));
        float v0 = g, v1 = g, v2 = g;
        if (g < 0.f) {  // :699-702
          const float *cx = a.ctx_xyz + ((size_t)b * a.C + c) * 3;
          v0 = __fadd_rn(fm, fabsf(__fsub_rn(qx, cx[0])));
          v1 = __fadd_rn(fm, fabsf(__fsub_rn(qy, cx[1])));
          v2 = __fadd_rn(fm, fabsf(__fsub_rn(qz, cx[2])));
        }
        const float two_pi = 6.2831855f;
        n0 = __fmul_rn(__fdiv_rn(__fsub_rn(v0, mn0), df0), two_pi);
        n1 = __fmul_rn(__fdiv_rn(__fsub_rn(v1, mn1), df1), two_pi);
        n2 = __fmul_rn(__fdiv_rn(__fsub_rn(v2, mn2), df2), two_pi);
      }
    }
  }

  template <bool TRANSPOSED>
  __device__ __forceinline__ void stash(const AttArgs &a, uint32_t dst, uint32_t dstT) {
    if (!FUSED) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        sts128(dst + st_off[j], pre[j]);
        if (TRANSPOSED) sts_t(dstT, 16 * qd + 4 * j, pre[j]);
      }
    } else {
#pragma unroll
      for (int j4 = 0; j4 < 2; ++j4) {  // this thread's eight frequencies: sin -> columns j, cos -> columns 32 + j
        float sn[4], cs[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          const int j = 8 * qd + 4 * j4 + e;
          const float p = fmaf(n2, __ldg(a.gauss_B + 2 * a.ldb + j), fmaf(n1, __ldg(a.gauss_B + a.ldb + j), __fmul_rn(n0, __ldg(a.gauss_B + j))));
          sincosf(p, &sn[e], &cs[e]);
          if (!pre_live) sn[e] = cs[e] = 0.f;
        }
        sts128(dst + st_off[2 * j4], make_float4(sn[0], sn[1], sn[2], sn[3]));
        sts128(dst + st_off[2 * j4 + 1], make_float4(cs[0], cs[1], cs[2], cs[3]));
        if (TRANSPOSED) {
          sts_t(dstT, 8 * qd + 4 * j4, make_float4(sn[0], sn[1], sn[2], sn[3]));
          sts_t(dstT, 32 + 8 * qd + 4 * j4, make_float4(cs[0], cs[1], cs[2], cs[3]));
        }
      }
    }
  }
};

// Software pipeline over the tiles of one (query, batch element), one __syncthreads per tile.  In iteration i
//   every thread    loads tile i+2 of the embedding into the operand buffer tile i has just released
//   warps 2,3,6,7   (TMEM lanes 64..127) turn product 1 of tile i into the hidden tile  (two warps per lane
//                   quadrant, 32 contexts each)
//   warps 0,1,4,5   (TMEM lanes 0..63) run softmax + weighted sum of tile i-1 from product 2 and the v2 rows of product 1
//   thread 0        then issues product 2 of tile i and product 1 of tile i+2; both complete under the next iteration.
// Product 1 of a tile is issued two iterations before it is consumed, product 2 one iteration: three D1 and two D2
// accumulator buffers in TMEM, one mbarrier per buffer.
// SAVE: the merge also writes what the backward needs, o = sum_c a_c v_c and lse = max + log(sum) of the scores.
template <bool FUSED, bool SAVE>
__global__ void __launch_bounds__(ATT_THREADS, 1) rel_cross_attention_kernel(const AttArgs a) {
  extern __shared__ unsigned char att_smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[5];  // [0..2] product 1 into D1[b], [3..4] product 2 into D2[b]
  __shared__ uint32_t s_tmem;
  __shared__ float s_part[3][2][ATT_D];  // partial softmax states (max, sum, weighted sum) of the two column halves
  __shared__ float s_out[ATT_D];
  const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  const int q = blockIdx.x, b = blockIdx.y;
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(att_smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char *sA1 = smem, *sA2 = smem + ATT_W_BYTES, *sR = smem + 2 * ATT_W_BYTES, *sH = sR + 2 * ATT_T_BYTES;
  uint32_t mbar[5];
#pragma unroll
  for (int i = 0; i < 5; ++i) mbar[i] = smem_u32(&s_mbar[i]);

  // ---- one-time set-up: weights into swizzled K-major tiles, TMEM, barriers -----------------------------------
  // A1 rows 0..63 = Wv, rows 64..127 = W1;  A2 rows 0..63 = W2, rows 64..127 = 0
  for (int e = tid; e < 128 * ATT_D; e += ATT_THREADS) {
    const int r = e >> 6, k = e & 63;
    *reinterpret_cast<float *>(sA1 + sw128_off<128>(r, k)) = r < 64 ? __ldg(a.wv + r * 64 + k) : __ldg(a.w1 + (r - 64) * 64 + k);
    *reinterpret_cast<float *>(sA2 + sw128_off<128>(r, k)) = r < 64 ? __ldg(a.w2 + r * 64 + k) : 0.f;
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 512;" ::"r"(smem_u32(&s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 5; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar[i]) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }

  // roles and per-thread constants
  const bool hidden_role = (warp & 2u) != 0;     // warps 2,3,6,7: TMEM lanes 64..127
  const int ch = (int)(((warp & 1u) << 5) | lane);  // channel inside the role's 64 lanes
  const int colhalf = (int)(warp >> 2) * 32;      // which 32 of the tile's 64 contexts this warp handles
  const float aq = hidden_role ? __ldg(a.aq + ((size_t)b * a.Q + q) * 64 + ch) : 0.f;
  const float b2 = hidden_role ? 0.f : __ldg(a.b2 + ch);
  const float *p1 = a.p1 + (size_t)b * a.C * 64, *pv = a.pv + (size_t)b * a.C * 64;
  // hidden-tile store addresses: half-tile and word of column ch, plus the eight swizzled chunk offsets
  const uint32_t h_base = (uint32_t)((ch >> 5) * ATT_T_HALF + colhalf * 128 + ((ch & 3) << 2));
  uint32_t h_sw[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) h_sw[j] = (uint32_t)((((ch & 31) >> 2) ^ j) << 4);
  float m_run = -INFINITY, s_run = 0.f, acc = 0.f;  // online softmax over this warp's contexts, per channel

  EmbTile<FUSED> emb(a, q, b, tid);
  const uint32_t sR_s = smem_u32(sR), sH_s = smem_u32(sH);
  auto fetch = [&](int tile) { emb.fetch(a, q, b, tile); };
  auto stash = [&](int buf) { emb.template stash<false>(a, sR_s + (uint32_t)buf * ATT_T_BYTES, 0); };
  auto load_tile = [&](int tile, int buf) {
    fetch(tile);
    stash(buf);
  };

  const int T = (a.C + ATT_TILE - 1) / ATT_TILE;
  load_tile(0, 0);
  if (T > 1) load_tile(1, 1);
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // tiles were written through the generic proxy
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem = s_tmem;
  const uint32_t t_lane = tmem + (((warp & 3u) * 32u) << 16);  // this warp's 32 TMEM lanes
  if (tid == 0) {
    umma_tile(tmem + ATT_D1_COL, smem_u32(sA1), smem_u32(sR), mbar[0]);
    if (T > 1) umma_tile(tmem + ATT_D1_COL + ATT_TILE, smem_u32(sA1), smem_u32(sR + ATT_T_BYTES), mbar[1]);
  }

  for (int i = 0; i <= T; ++i) {
    // global loads first: tile i + 2 of the embedding and this thread's 32 table entries of the tile it works on
    const bool more = i + 2 < T;
    if (more) fetch(i + 2);
    float tab[32];
    {
      const int t = hidden_role ? i : i - 1;
      const float *src = (hidden_role ? p1 : pv) + ch;
      const int c0 = t * ATT_TILE + colhalf;
      if (t >= 0 && t < T) {
#pragma unroll
        for (int e = 0; e < 32; ++e) tab[e] = c0 + e < a.C ? __ldg(src + (size_t)(c0 + e) * 64) : 0.f;
      }
    }
    if (i < T) {  // product 1 of tile i has landed in D1[i % 3]; the operand buffer i % 2 is free again
      mbar_wait(mbar[i % 3], (uint32_t)((i / 3) & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    }
    if (hidden_role) {
      if (i < T) {  // h = relu(W1 rel + (W1 tgt2[q] + b1) - W1 memory[c]) -> hidden tile i % 2, row = context, column = ch
        float d[32];
        tmem_ld32(t_lane + ATT_D1_COL + (uint32_t)((i % 3) * ATT_TILE + colhalf), d);
        // row colhalf + e, column ch: (colhalf + e) & 7 == e & 7, so the swizzled chunk is one of eight per-thread
        // constants and the row is an immediate offset
        const uint32_t dst = sH_s + (uint32_t)(i & 1) * ATT_T_BYTES + h_base;
        const int c0 = i * ATT_TILE + colhalf;
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          const float h = c0 + e < a.C ? fmaxf(d[e] + aq - tab[e], 0.f) : 0.f;
          asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst + h_sw[e & 7] + (uint32_t)e * 128u), "f"(h) : "memory");
        }
      }
    } else if (i >= 1) {  // softmax over the contexts and weighted sum of tile i - 1
      const int t = i - 1;
      mbar_wait(mbar[3 + (t & 1)], (uint32_t)((t >> 1) & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      float sv[32], vv[32];
      tmem_ld32(t_lane + ATT_D2_COL + (uint32_t)((t & 1) * ATT_TILE + colhalf), sv);
      tmem_ld32(t_lane + ATT_D1_COL + (uint32_t)((t % 3) * ATT_TILE + colhalf), vv);
      const int c0 = t * ATT_TILE + colhalf;
      float mx = m_run;
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        sv[e] = c0 + e < a.C ? (sv[e] + b2) * 0.125f : -INFINITY;  // / sqrt(64), :449
        mx = fmaxf(mx, sv[e]);
      }
      if (mx > -INFINITY) {
        const float scale = __expf(m_run - mx);  // exp(-inf) = 0 for the first contexts
        s_run *= scale, acc *= scale;
#pragma unroll
        for (int e = 0; e < 32; ++e) {
          if (c0 + e < a.C) {
            const float w = __expf(sv[e] - mx);
            s_run += w;
            acc = fmaf(w, vv[e] + tab[e], acc);
          }
        }
        m_run = mx;
      }
    }
    if (more) stash(i & 1);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid == 0) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      if (i < T)  // product 2: lanes 0..63 <- W2 h
        umma_tile(tmem + ATT_D2_COL + (uint32_t)((i & 1) * ATT_TILE), smem_u32(sA2), smem_u32(sH + (i & 1) * ATT_T_BYTES), mbar[3 + (i & 1)]);
      if (i + 2 < T)  // product 1 of tile i + 2: lanes 0..63 <- Wv rel, lanes 64..127 <- W1 rel
        umma_tile(tmem + ATT_D1_COL + (uint32_t)(((i + 2) % 3) * ATT_TILE), smem_u32(sA1), smem_u32(sR + (i & 1) * ATT_T_BYTES), mbar[(i + 2) % 3]);
    }
  }
  // ---- merge the two column halves, then out_mlp: relu(Wo (acc / s) + bo) ----------------------------------------
  if (!hidden_role) {
    const int hh = (int)(warp >> 2);
    s_part[0][hh][ch] = m_run, s_part[1][hh][ch] = s_run, s_part[2][hh][ch] = acc;
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 64) {
    const float m0 = s_part[0][0][tid], m1 = s_part[0][1][tid];
    const float mx = fmaxf(m0, m1);
    float s = 0.f, av = 0.f;
    if (mx > -INFINITY) {
      const float e0 = __expf(m0 - mx), e1 = __expf(m1 - mx);
      s = s_part[1][0][tid] * e0 + s_part[1][1][tid] * e1;
      av = s_part[2][0][tid] * e0 + s_part[2][1][tid] * e1;
    }
    s_out[tid] = s > 0.f ? av / s : 0.f;
    if (SAVE) {
      a.o_save[((size_t)q * a.B + b) * 64 + tid] = s_out[tid];
      a.lse_save[((size_t)q * a.B + b) * 64 + tid] = mx + logf(s);
    }
  }
  __syncthreads();
  if (tid < 64) {
    float o = __ldg(a.bo + tid);
#pragma unroll 8
    for (int f = 0; f < 64; ++f) o = fmaf(__ldg(a.wo + tid * 64 + f), s_out[f], o);
    a.out[((size_t)q * a.B + b) * 64 + tid] = fmaxf(o, 0.f);
  }
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 512;" ::"r"(tmem) : "memory");
}


// ---- backward -------------------------------------------------------------------------------------------------
// Recompute-style, one CTA per (query, batch element) over the context tiles like the forward; nothing of size
// (Q, C, B, 64) was saved, only o and lse (Q, B, 64).  Per tile, one tcgen05 product after the other:
//   P1  D1 <- [Wv; W1] x R                 the forward's product 1 (same operands, same code: bit-identical)
//       hidden lanes: hp = W1 r + aq - p1, h = relu(hp) -> H (row = context) and H^T (row = channel); v lanes: v
//   P2  D2 <- [W2; 0] x H                  the forward's product 2: s = (W2 h + b2) / 8 bit-identical
//       v lanes: a = exp(s - lse), dv = a do, g = dv (v - o) / 8 -> G, and G^T, dV^T rows of the transposed tile T
//   P3  D2 <- [0; W2^T] x G                W2^T g in the hidden lanes
//   P4  DW2 += [G^T; dV^T] x H^T           lanes 0..63: sum_c g h^T            (lanes 64..127 unused)
//       hidden lanes: dh = W2^T g [hp > 0] -> dH^T rows of T; Hsum_q += dh in registers
//   P5  DW += [dV^T; dH^T] x R^T           lanes 0..63: sum_c dv r^T, lanes 64..127: sum_c dh r^T
// The weight tiles [W2; 0; W2^T] and the transposed tile [G^T; dV^T; dH^T] are 192-row regions of which a product
// takes 128 consecutive rows.  dh and dv of every pair go to the (Q, B, C, 128) buffer `pairs` the finishing kernels
// reduce over the queries in a fixed order (no atomics anywhere: two calls give bitwise-equal gradients).
constexpr int ATT_B_HALF = 192 * 128;  // one K-half of a 192-row region
constexpr int ATT_BWD_SMEM = ATT_W_BYTES + 2 * 2 * ATT_B_HALF + 5 * ATT_T_BYTES + 1024;
constexpr uint32_t ATT_BWD_D1 = 0, ATT_BWD_D2 = ATT_TILE, ATT_BWD_DW = 2 * ATT_TILE, ATT_BWD_DW2 = 3 * ATT_TILE;

struct AttBwdArgs {
  const float *o, *lse, *dout_o;  // (Q, B, 64): saved o and lse, do = Wo^T dz
  float *part;                    // (Q * B, 3, 64, 64) per-CTA sums over its contexts: dWv, dW1 (r terms), dW2
  float *hsum;                    // (Q, B, 64) Hsum_q
  float *pairs;                   // (Q, B, C, 128) [dh | dv] of every pair
};

// 32 consecutive K values (one K-half) of row r of a swizzled K-major region: eight 16-byte chunks
__device__ __forceinline__ void st_row32(uint32_t half_base, int r, const float (&v)[32]) {
#pragma unroll
  for (int j = 0; j < 8; ++j)
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(half_base + (uint32_t)(r * 128 + ((j ^ (r & 7)) << 4))),
                 "f"(v[4 * j]), "f"(v[4 * j + 1]), "f"(v[4 * j + 2]), "f"(v[4 * j + 3])
                 : "memory");
}

// generic-proxy shared stores and TMEM reads done, then thread 0 may issue the next products
__device__ __forceinline__ void att_sync_for_mma() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

__device__ __forceinline__ void att_wait_mma(uint32_t mbar, uint32_t parity) {
  mbar_wait(mbar, parity);
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}

template <bool FUSED>
__global__ void __launch_bounds__(ATT_THREADS, 1) rel_cross_attention_bwd_kernel(const AttArgs a, const AttBwdArgs g) {
  extern __shared__ unsigned char att_smem_raw[];
  __shared__ __align__(8) unsigned long long s_mbar[4];
  __shared__ uint32_t s_tmem;
  __shared__ float s_hsum[2][ATT_D];
  const unsigned tid = threadIdx.x, warp = tid >> 5, lane = tid & 31u;
  const int q = blockIdx.x, b = blockIdx.y;
  const size_t qb = (size_t)q * a.B + b;
  unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(att_smem_raw) + 1023) & ~(uintptr_t)1023);
  unsigned char *sA1 = smem, *sA2 = sA1 + ATT_W_BYTES, *sR = sA2 + 2 * ATT_B_HALF, *sRT = sR + ATT_T_BYTES,
                *sH = sRT + ATT_T_BYTES, *sHT = sH + ATT_T_BYTES, *sG = sHT + ATT_T_BYTES, *sT = sG + ATT_T_BYTES;
  uint32_t mbar[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) mbar[i] = smem_u32(&s_mbar[i]);

  // A1 = [Wv; W1] as in the forward; A2 = [W2; 0; W2^T] (row 128 + j, column i = W2[i][j])
  for (int e = tid; e < 128 * ATT_D; e += ATT_THREADS) {
    const int r = e >> 6, k = e & 63;
    *reinterpret_cast<float *>(sA1 + sw128_off<128>(r, k)) = r < 64 ? __ldg(a.wv + r * 64 + k) : __ldg(a.w1 + (r - 64) * 64 + k);
  }
  for (int e = tid; e < 192 * ATT_D; e += ATT_THREADS) {
    const int r = e >> 6, k = e & 63;
    *reinterpret_cast<float *>(sA2 + sw128_off<192>(r, k)) =
        r < 64 ? __ldg(a.w2 + r * 64 + k) : r < 128 ? 0.f : __ldg(a.w2 + k * 64 + (r - 128));
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], 256;" ::"r"(smem_u32(&s_tmem)) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < 4; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(mbar[i]) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }

  // roles as in the forward: warps 2,3,6,7 hold TMEM lanes 64..127 (hidden layer), the others lanes 0..63 (v / scores)
  const bool hidden_role = (warp & 2u) != 0;
  const int ch = (int)(((warp & 1u) << 5) | lane);
  const int colhalf = (int)(warp >> 2) * 32;
  const float aq = hidden_role ? __ldg(a.aq + ((size_t)b * a.Q + q) * 64 + ch) : 0.f;
  const float b2 = hidden_role ? 0.f : __ldg(a.b2 + ch);
  const float lse = hidden_role ? 0.f : __ldg(g.lse + qb * 64 + ch);
  const float o = hidden_role ? 0.f : __ldg(g.o + qb * 64 + ch);
  const float dout = hidden_role ? 0.f : __ldg(g.dout_o + qb * 64 + ch);
  const float *tab_src = (hidden_role ? a.p1 : a.pv) + (size_t)b * a.C * 64 + ch;
  float *pair_dst = g.pairs + qb * a.C * 128 + (hidden_role ? ch : 64 + ch);
  // row = context stores of H and G: the forward's hidden-tile addressing
  const uint32_t h_base = (uint32_t)((ch >> 5) * ATT_T_HALF + colhalf * 128 + ((ch & 3) << 2));
  uint32_t h_sw[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) h_sw[j] = (uint32_t)((((ch & 31) >> 2) ^ j) << 4);
  const uint32_t sA1_s = smem_u32(sA1), sA2_s = smem_u32(sA2), sR_s = smem_u32(sR), sRT_s = smem_u32(sRT),
                 sH_s = smem_u32(sH), sHT_s = smem_u32(sHT), sG_s = smem_u32(sG), sT_s = smem_u32(sT);
  // row = channel stores: the K-half of this warp's 32 contexts
  const uint32_t ht_half = sHT_s + (uint32_t)(colhalf >> 5) * ATT_T_HALF, t_half = sT_s + (uint32_t)(colhalf >> 5) * ATT_B_HALF;
  float hsum = 0.f;

  EmbTile<FUSED> emb(a, q, b, tid);
  emb.fetch(a, q, b, 0);
  att_sync_for_mma();
  const uint32_t tmem = s_tmem;
  const uint32_t t_lane = tmem + (((warp & 3u) * 32u) << 16);
  const int T = (a.C + ATT_TILE - 1) / ATT_TILE;
  for (int t = 0; t < T; ++t) {
    const uint32_t par = (uint32_t)(t & 1);
    const int c0 = t * ATT_TILE + colhalf;
    emb.template stash<true>(a, sR_s, sRT_s);
    float tab[32];
#pragma unroll
    for (int e = 0; e < 32; ++e) tab[e] = c0 + e < a.C ? __ldg(tab_src + (size_t)(c0 + e) * 64) : 0.f;
    att_sync_for_mma();
    if (tid == 0) {
      umma_k64<ATT_W_HALF>(tmem + ATT_BWD_D1, sA1_s, sR_s, false);
      umma_commit(mbar[0]);
    }
    if (t + 1 < T) emb.fetch(a, q, b, t + 1);
    att_wait_mma(mbar[0], par);

    float d[32];
    uint32_t mask = 0;  // hidden lanes: hp > 0 of this warp's 32 contexts
    tmem_ld32(t_lane + ATT_BWD_D1 + (uint32_t)colhalf, d);
    if (hidden_role) {
      const uint32_t dst = sH_s + h_base;
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const float hp = d[e] + aq - tab[e];
        const bool on = c0 + e < a.C && hp > 0.f;
        mask |= (uint32_t)on << e;
        d[e] = c0 + e < a.C ? fmaxf(hp, 0.f) : 0.f;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst + h_sw[e & 7] + (uint32_t)e * 128u), "f"(d[e]) : "memory");
      }
      st_row32(ht_half, ch, d);
    } else {
#pragma unroll
      for (int e = 0; e < 32; ++e) d[e] += tab[e];  // v = Wv (m + r) + bv
    }
    att_sync_for_mma();
    if (tid == 0) {
      umma_k64<ATT_B_HALF>(tmem + ATT_BWD_D2, sA2_s, sH_s, false);
      umma_commit(mbar[1]);
    }
    att_wait_mma(mbar[1], par);

    if (!hidden_role) {
      float sv[32], gv[32];
      tmem_ld32(t_lane + ATT_BWD_D2 + (uint32_t)colhalf, sv);
      const uint32_t dst = sG_s + h_base;
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        const bool live = c0 + e < a.C;
        const float w = live ? __expf((sv[e] + b2) * 0.125f - lse) : 0.f;  // the forward's s, :449
        const float dv = w * dout;
        gv[e] = dv * (d[e] - o) * 0.125f;
        d[e] = dv;
        if (live) pair_dst[(size_t)(c0 + e) * 128] = dv;
        asm volatile("st.shared.f32 [%0], %1;" ::"r"(dst + h_sw[e & 7] + (uint32_t)e * 128u), "f"(gv[e]) : "memory");
      }
      st_row32(t_half, ch, gv);
      st_row32(t_half, 64 + ch, d);
    }
    att_sync_for_mma();
    if (tid == 0) {
      umma_k64<ATT_B_HALF>(tmem + ATT_BWD_D2, sA2_s + 64 * 128, sG_s, false);
      umma_k64<ATT_B_HALF>(tmem + ATT_BWD_DW2, sT_s, sHT_s, t > 0);
      umma_commit(mbar[2]);
    }
    att_wait_mma(mbar[2], par);

    if (hidden_role) {
      tmem_ld32(t_lane + ATT_BWD_D2 + (uint32_t)colhalf, d);
#pragma unroll
      for (int e = 0; e < 32; ++e) {
        d[e] = (mask >> e) & 1u ? d[e] : 0.f;
        hsum += d[e];
        if (c0 + e < a.C) pair_dst[(size_t)(c0 + e) * 128] = d[e];
      }
      st_row32(t_half, 128 + ch, d);
    }
    att_sync_for_mma();
    if (tid == 0) {
      umma_k64<ATT_B_HALF>(tmem + ATT_BWD_DW, sT_s + 64 * 128, sRT_s, t > 0);
      umma_commit(mbar[3]);
    }
    att_wait_mma(mbar[3], par);  // every operand tile is free again
  }

  // per-CTA weight partials: DW lanes 0..127 = [dWv; dW1] rows, DW2 lanes 0..63 = dW2 rows; this warp's 32 columns
  {
    const int row = (int)((warp & 3u) * 32u + lane);
    float v[32];
    float *dst = g.part + qb * 3 * 4096 + (size_t)row * 64 + colhalf;
    tmem_ld32(t_lane + ATT_BWD_DW + (uint32_t)colhalf, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) reinterpret_cast<float4 *>(dst)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    if (row < 64) {
      tmem_ld32(t_lane + ATT_BWD_DW2 + (uint32_t)colhalf, v);
#pragma unroll
      for (int j = 0; j < 8; ++j)
        reinterpret_cast<float4 *>(dst + 2 * 4096)[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
    }
  }
  if (hidden_role) s_hsum[warp >> 2][ch] = hsum;
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (tid < 64) g.hsum[qb * 64 + tid] = s_hsum[0][tid] + s_hsum[1][tid];
  if (warp == 0) {
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, 256;" ::"r"(tmem) : "memory");
  }
}

}  // namespace gf

using namespace gf;

// tables of the query / context parts (three small matrix products, fp32 on the CUDA cores):
//   aq[b,q,:] = W1 tgt2[q,b,:] + b1,   p1[b,c,:] = W1 memory[c,b,:],   pv[b,c,:] = Wv memory[c,b,:] + bv
__global__ void att_tables_kernel(const float *__restrict__ tgt2, const float *__restrict__ memory, int Q, int C, int B,
                                  const float *__restrict__ w1, const float *__restrict__ b1,
                                  const float *__restrict__ wv, const float *__restrict__ bv, float *__restrict__ aq,
                                  float *__restrict__ p1, float *__restrict__ pv) {
  __shared__ float x[64];
  const int row = blockIdx.x, b = blockIdx.y, o = threadIdx.x;  // rows 0..Q-1: queries, Q..Q+C-1: contexts
  const bool is_q = row < Q;
  const float *src = is_q ? tgt2 + ((size_t)row * B + b) * 64 : memory + ((size_t)(row - Q) * B + b) * 64;
  x[o] = src[o];
  __syncthreads();
  float s1 = 0.f, sv = 0.f;
#pragma unroll 8
  for (int i = 0; i < 64; ++i) {
    s1 = fmaf(__ldg(w1 + o * 64 + i), x[i], s1);
    if (!is_q) sv = fmaf(__ldg(wv + o * 64 + i), x[i], sv);
  }
  if (is_q) {
    aq[((size_t)b * Q + row) * 64 + o] = s1 + b1[o];
  } else {
    p1[((size_t)b * C + (row - Q)) * 64 + o] = s1;
    pv[((size_t)b * C + (row - Q)) * 64 + o] = sv + bv[o];
  }
}

extern "C" size_t gf_rel_cross_attention_workspace_bytes(int Q, int C, int B) {
  if (Q <= 0 || C <= 0 || B <= 0) return 0;
  return align256(sizeof(float) * 64 * (size_t)B * Q) + 2 * align256(sizeof(float) * 64 * (size_t)B * C) +
         align256(sizeof(uint32_t) * ((size_t)B * Q + 1)) + 1024;
}

namespace gf {
// row maxima of the gathered maps, gf_bias.cu
int bias_ctx_rowmax(const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx, int B, int Q, int C,
                    uint32_t *rowmax, uint32_t *gmax, cudaStream_t st);
}  // namespace gf

// the tables (and for the fused variant the row maxima of the gathered maps) at the front of the workspace
static int att_prepare(AttArgs &a, const float *tgt2, const float *memory, const float *b1, const float *bv,
                       const float *const *geo_ptrs, const int *geo_ld, Arena &ar, const char *name, size_t needed,
                       cudaStream_t st) {
  float *aq = ar.take<float>(64 * (size_t)a.B * a.Q);
  float *p1 = ar.take<float>(64 * (size_t)a.B * a.C);
  float *pv = ar.take<float>(64 * (size_t)a.B * a.C);
  uint32_t *rm = ar.take<uint32_t>((size_t)a.B * a.Q + 1);
  if (!ar.ok) {
    set_error("%s: workspace too small (%zu bytes given, %zu needed)", name, ar.size, needed);
    return GF_ERR_WORKSPACE;
  }
  att_tables_kernel<<<dim3(a.Q + a.C, a.B), 64, 0, st>>>(tgt2, memory, a.Q, a.C, a.B, a.w1, b1, a.wv, bv, aq, p1, pv);
  GF_LAUNCHED();
  a.aq = aq, a.p1 = p1, a.pv = pv;
  if (geo_ptrs) {
    for (int b = 0; b < a.B; ++b) a.geo[b] = geo_ptrs[b], a.geo_ld[b] = geo_ld[b];
    int rc = bias_ctx_rowmax(geo_ptrs, geo_ld, a.ctx_idx, a.B, a.Q, a.C, rm, rm + (size_t)a.B * a.Q, st);
    if (rc) return rc;
    a.rowmax = rm, a.gmax = rm + (size_t)a.B * a.Q;
  }
  return GF_OK;
}

// the dynamic shared-memory opt-in of the attention kernels, once per device
static int att_set_smem() {
  static int done[64] = {0};
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (!__atomic_load_n(&done[dev], __ATOMIC_ACQUIRE)) {
    GF_CUDA(cudaFuncSetAttribute(rel_cross_attention_kernel<false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
    GF_CUDA(cudaFuncSetAttribute(rel_cross_attention_kernel<true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
    GF_CUDA(cudaFuncSetAttribute(rel_cross_attention_kernel<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
    GF_CUDA(cudaFuncSetAttribute(rel_cross_attention_kernel<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_SMEM));
    GF_CUDA(cudaFuncSetAttribute(rel_cross_attention_bwd_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_BWD_SMEM));
    GF_CUDA(cudaFuncSetAttribute(rel_cross_attention_bwd_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ATT_BWD_SMEM));
    __atomic_store_n(&done[dev], 1, __ATOMIC_RELEASE);
  }
  return GF_OK;
}

static int att_launch(AttArgs &a, const float *tgt2, const float *memory, const float *b1, const float *bv,
                      const float *const *geo_ptrs, const int *geo_ld, void *workspace, size_t workspace_bytes,
                      cudaStream_t st) {
  const bool fused = geo_ptrs != nullptr, save = a.o_save != nullptr;
  Arena ar(workspace, workspace_bytes);
  int rc = att_prepare(a, tgt2, memory, b1, bv, geo_ptrs, geo_ld, ar, "rel_cross_attention",
                       gf_rel_cross_attention_workspace_bytes(a.Q, a.C, a.B), st);
  if (rc) return rc;
  if ((rc = att_set_smem())) return rc;
  const dim3 grid(a.Q, a.B);
  if (fused)
    save ? rel_cross_attention_kernel<true, true><<<grid, ATT_THREADS, ATT_SMEM, st>>>(a)
         : rel_cross_attention_kernel<true, false><<<grid, ATT_THREADS, ATT_SMEM, st>>>(a);
  else
    save ? rel_cross_attention_kernel<false, true><<<grid, ATT_THREADS, ATT_SMEM, st>>>(a)
         : rel_cross_attention_kernel<false, false><<<grid, ATT_THREADS, ATT_SMEM, st>>>(a);
  GF_LAUNCHED();
  return GF_OK;
}

#define ATT_COMMON_CHECKS(name)                                                                            \
  GF_CHECK_ARG(Q >= 1 && C >= 1 && B >= 1, name ": need Q, C, B >= 1");                                      \
  GF_CHECK_ARG(tgt2 && memory && w1 && b1 && w2 && b2 && wv && bv && wo && bo && out, name ": null pointer")

extern "C" int gf_rel_cross_attention(const float *tgt2, const float *memory, const float *relative_pos, int Q, int C,
                                      int B, const float *w1, const float *b1, const float *w2, const float *b2,
                                      const float *wv, const float *bv, const float *wo, const float *bo, float *out,
                                      void *workspace, size_t workspace_bytes, void *stream) {
  ATT_COMMON_CHECKS("rel_cross_attention");
  GF_CHECK_ARG(relative_pos, "rel_cross_attention: null relative_pos");
  AttArgs a = {};
  a.w1 = w1, a.w2 = w2, a.wv = wv, a.wo = wo, a.b2 = b2, a.bo = bo, a.Q = Q, a.C = C, a.B = B, a.rel = relative_pos, a.out = out;
  return att_launch(a, tgt2, memory, b1, bv, nullptr, nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
}

#define ATT_FUSED_CHECKS(name)                                                                                     \
  GF_CHECK_ARG(geo_ptrs && geo_ld && ctx_idx && query_xyz && ctx_xyz && gauss_B && pc_min && pc_max,               \
               name ": null pointer");                                                                             \
  GF_CHECK_ARG(gauss_ld >= 32, name ": the embedding has 32 frequencies (gauss_B must be (3, >= 32))");            \
  GF_CHECK_ARG(B <= ATT_MAX_B, name ": B=%d, at most %d batch elements per call", B, ATT_MAX_B)

static void att_fused_args(AttArgs &a, const int *ctx_idx, const float *query_xyz, const float *ctx_xyz,
                           const float *gauss_B, int gauss_ld, const float *pc_min, const float *pc_max, int Q, int C,
                           int B, const float *w1, const float *w2, const float *b2, const float *wv, const float *wo,
                           const float *bo) {
  a.w1 = w1, a.w2 = w2, a.wv = wv, a.wo = wo, a.b2 = b2, a.bo = bo, a.Q = Q, a.C = C, a.B = B;
  a.ctx_idx = ctx_idx, a.query_xyz = query_xyz, a.ctx_xyz = ctx_xyz;
  a.gauss_B = gauss_B, a.ldb = gauss_ld, a.pc_min = pc_min, a.pc_max = pc_max;
}

extern "C" int gf_rel_cross_attention_fused(const float *tgt2, const float *memory, const float *const *geo_ptrs,
                                            const int *geo_ld, const int *ctx_idx, const float *query_xyz,
                                            const float *ctx_xyz, const float *gauss_B, int gauss_ld, const float *pc_min,
                                            const float *pc_max, int Q, int C, int B, const float *w1, const float *b1,
                                            const float *w2, const float *b2, const float *wv, const float *bv,
                                            const float *wo, const float *bo, float *out, void *workspace,
                                            size_t workspace_bytes, void *stream) {
  ATT_COMMON_CHECKS("rel_cross_attention_fused");
  ATT_FUSED_CHECKS("rel_cross_attention_fused");
  AttArgs a = {};
  att_fused_args(a, ctx_idx, query_xyz, ctx_xyz, gauss_B, gauss_ld, pc_min, pc_max, Q, C, B, w1, w2, b2, wv, wo, bo);
  a.out = out;
  return att_launch(a, tgt2, memory, b1, bv, geo_ptrs, geo_ld, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int gf_rel_cross_attention_save(const float *tgt2, const float *memory, const float *relative_pos, int Q,
                                           int C, int B, const float *w1, const float *b1, const float *w2,
                                           const float *b2, const float *wv, const float *bv, const float *wo,
                                           const float *bo, float *out, float *o, float *lse, void *workspace,
                                           size_t workspace_bytes, void *stream) {
  ATT_COMMON_CHECKS("rel_cross_attention_save");
  GF_CHECK_ARG(relative_pos && o && lse, "rel_cross_attention_save: null pointer");
  AttArgs a = {};
  a.w1 = w1, a.w2 = w2, a.wv = wv, a.wo = wo, a.b2 = b2, a.bo = bo, a.Q = Q, a.C = C, a.B = B, a.rel = relative_pos, a.out = out;
  a.o_save = o, a.lse_save = lse;
  return att_launch(a, tgt2, memory, b1, bv, nullptr, nullptr, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int gf_rel_cross_attention_fused_save(const float *tgt2, const float *memory, const float *const *geo_ptrs,
                                                 const int *geo_ld, const int *ctx_idx, const float *query_xyz,
                                                 const float *ctx_xyz, const float *gauss_B, int gauss_ld,
                                                 const float *pc_min, const float *pc_max, int Q, int C, int B,
                                                 const float *w1, const float *b1, const float *w2, const float *b2,
                                                 const float *wv, const float *bv, const float *wo, const float *bo,
                                                 float *out, float *o, float *lse, void *workspace,
                                                 size_t workspace_bytes, void *stream) {
  ATT_COMMON_CHECKS("rel_cross_attention_fused_save");
  ATT_FUSED_CHECKS("rel_cross_attention_fused_save");
  GF_CHECK_ARG(o && lse, "rel_cross_attention_fused_save: null pointer");
  AttArgs a = {};
  att_fused_args(a, ctx_idx, query_xyz, ctx_xyz, gauss_B, gauss_ld, pc_min, pc_max, Q, C, B, w1, w2, b2, wv, wo, bo);
  a.out = out, a.o_save = o, a.lse_save = lse;
  return att_launch(a, tgt2, memory, b1, bv, geo_ptrs, geo_ld, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- backward: prologue and finishing kernels (CUDA cores, fixed summation orders) ------------------------------

// dz = dy [out > 0], do = Wo^T dz, one block per (q, b)
__global__ void att_bwd_prologue_kernel(const float *__restrict__ out, const float *__restrict__ dy,
                                        const float *__restrict__ wo, float *__restrict__ dz, float *__restrict__ dout_o) {
  __shared__ float z[64];
  const size_t r = (size_t)blockIdx.x * 64;
  const int i = threadIdx.x;
  z[i] = out[r + i] > 0.f ? dy[r + i] : 0.f;
  dz[r + i] = z[i];
  __syncthreads();
  float s = 0.f;
#pragma unroll 8
  for (int k = 0; k < 64; ++k) s = fmaf(__ldg(wo + k * 64 + i), z[k], s);
  dout_o[r + i] = s;
}

// rows 0..Q-1: dtgt2[q,b] = W1^T Hsum[q,b];  rows Q..Q+C-1: [DH | DV][c,b] = sum over q of the pairs (in query order),
// dmemory[c,b] = Wv^T DV - W1^T DH
__global__ void att_bwd_rows_kernel(const float *__restrict__ hsum, const float *__restrict__ pairs, int Q, int C, int B,
                                    const float *__restrict__ w1, const float *__restrict__ wv,
                                    float *__restrict__ dtgt2, float *__restrict__ dhdv, float *__restrict__ dmemory) {
  __shared__ float x[128];
  const int row = blockIdx.x, b = blockIdx.y, i = threadIdx.x;
  if (row < Q) {
    const size_t r = (size_t)row * B + b;
    if (i < 64) x[i] = hsum[r * 64 + i];
    __syncthreads();
    if (i < 64) {
      float s = 0.f;
#pragma unroll 8
      for (int k = 0; k < 64; ++k) s = fmaf(__ldg(w1 + k * 64 + i), x[k], s);
      dtgt2[r * 64 + i] = s;
    }
    return;
  }
  const int c = row - Q;
  const size_t r = (size_t)c * B + b;
  float s = 0.f;
  for (int qq = 0; qq < Q; ++qq) s += pairs[(((size_t)qq * B + b) * C + c) * 128 + i];
  x[i] = s;
  dhdv[r * 128 + i] = s;
  __syncthreads();
  if (i < 64) {
    float sv = 0.f, s1 = 0.f;
#pragma unroll 8
    for (int k = 0; k < 64; ++k) {
      sv = fmaf(__ldg(wv + k * 64 + i), x[64 + k], sv);
      s1 = fmaf(__ldg(w1 + k * 64 + i), x[k], s1);
    }
    dmemory[r * 64 + i] = sv - s1;
  }
}

struct AttBwdWeights {
  const float *part, *hsum, *dhdv, *dz, *o, *dout_o, *tgt2, *memory;
  float *dw[4], *db[4];  // W1, Wv, W2, Wo
  int QB, CB;
};

// one block per (row i, weight): column j < 64 of the weight and, as column 64, the bias; the rows of each sum are
// split over ATT_WS_SLICES fixed slices whose partial sums are added in slice order
constexpr int ATT_WS_SLICES = 8;
__global__ void __launch_bounds__(65 * ATT_WS_SLICES) att_bwd_weights_kernel(const AttBwdWeights p) {
  __shared__ float acc_s[ATT_WS_SLICES][65];
  const int i = blockIdx.x, mat = blockIdx.y, j = threadIdx.x % 65, sl = threadIdx.x / 65;
  float acc = 0.f;
  if (j < 64) {
    if (mat != 3) {  // the per-CTA partials: part[cta][0] = dWv, [1] = dW1, [2] = dW2
      const int which = mat == 0 ? 1 : mat == 1 ? 0 : 2;
      for (int r = sl; r < p.QB; r += ATT_WS_SLICES) acc += p.part[((size_t)r * 3 + which) * 4096 + i * 64 + j];
    }
    if (mat == 0) {
      for (int r = sl; r < p.QB; r += ATT_WS_SLICES) acc = fmaf(p.hsum[(size_t)r * 64 + i], p.tgt2[(size_t)r * 64 + j], acc);
      for (int r = sl; r < p.CB; r += ATT_WS_SLICES) acc = fmaf(-p.dhdv[(size_t)r * 128 + i], p.memory[(size_t)r * 64 + j], acc);
    } else if (mat == 1) {
      for (int r = sl; r < p.CB; r += ATT_WS_SLICES) acc = fmaf(p.dhdv[(size_t)r * 128 + 64 + i], p.memory[(size_t)r * 64 + j], acc);
    } else if (mat == 3) {
      for (int r = sl; r < p.QB; r += ATT_WS_SLICES) acc = fmaf(p.dz[(size_t)r * 64 + i], p.o[(size_t)r * 64 + j], acc);
    }
  } else if (mat != 2) {  // db1 = sum Hsum, dbv = sum do, dbo = sum dz; db2 = 0 (the softmax is shift invariant)
    const float *v = mat == 0 ? p.hsum : mat == 1 ? p.dout_o : p.dz;
    for (int r = sl; r < p.QB; r += ATT_WS_SLICES) acc += v[(size_t)r * 64 + i];
  }
  acc_s[sl][j] = acc;
  __syncthreads();
  if (sl == 0) {
    float s = acc_s[0][j];
#pragma unroll
    for (int k = 1; k < ATT_WS_SLICES; ++k) s += acc_s[k][j];
    if (j < 64)
      p.dw[mat][i * 64 + j] = s;
    else
      p.db[mat][i] = s;
  }
}

// drel[q,c,b] = W1^T dh + Wv^T dv of every pair, 16 pairs per block
constexpr int ATT_DREL_PAIRS = 16;
__global__ void __launch_bounds__(256) att_bwd_drel_kernel(const float *__restrict__ pairs, int Q, int C, int B,
                                                           const float *__restrict__ w1, const float *__restrict__ wv,
                                                           float *__restrict__ drel) {
  __shared__ float sw1[64 * 64], swv[64 * 64], sp[ATT_DREL_PAIRS][128];
  const size_t n = (size_t)Q * B * C, base = (size_t)blockIdx.x * ATT_DREL_PAIRS;
  for (int e = threadIdx.x; e < 64 * 64; e += 256) sw1[e] = w1[e], swv[e] = wv[e];
  for (int e = threadIdx.x; e < ATT_DREL_PAIRS * 128; e += 256)
    sp[e >> 7][e & 127] = base + (e >> 7) < n ? pairs[base * 128 + e] : 0.f;
  __syncthreads();
  const int i = threadIdx.x & 63;
  for (int pp = threadIdx.x >> 6; pp < ATT_DREL_PAIRS; pp += 4) {
    const size_t row = base + pp;  // = (q * B + b) * C + c
    if (row >= n) break;
    float s1 = 0.f, sv = 0.f;
#pragma unroll 8
    for (int k = 0; k < 64; ++k) {
      s1 = fmaf(sw1[k * 64 + i], sp[pp][k], s1);
      sv = fmaf(swv[k * 64 + i], sp[pp][64 + k], sv);
    }
    const size_t qb = row / C, c = row % C, qq = qb / B, b = qb % B;
    drel[((qq * C + c) * B + b) * 64 + i] = s1 + sv;
  }
}

extern "C" size_t gf_rel_cross_attention_backward_workspace_bytes(int Q, int C, int B) {
  if (Q <= 0 || C <= 0 || B <= 0) return 0;
  const size_t QB = (size_t)Q * B, CB = (size_t)C * B;
  return gf_rel_cross_attention_workspace_bytes(Q, C, B) + 3 * align256(sizeof(float) * 64 * QB) +
         align256(sizeof(float) * 3 * 4096 * QB) + align256(sizeof(float) * 128 * QB * C) +
         align256(sizeof(float) * 128 * CB);
}

static int att_bwd_launch(AttArgs &a, const float *tgt2, const float *memory, const float *b1, const float *bv,
                          const float *const *geo_ptrs, const int *geo_ld, const float *o, const float *lse,
                          const float *dy, float *dtgt2, float *dmemory, float *drel, float *dw1, float *db1,
                          float *dw2, float *db2, float *dwv, float *dbv, float *dwo, float *dbo, void *workspace,
                          size_t workspace_bytes, cudaStream_t st) {
  const int Q = a.Q, C = a.C, B = a.B;
  const size_t QB = (size_t)Q * B;
  const size_t needed = gf_rel_cross_attention_backward_workspace_bytes(Q, C, B);
  Arena ar(workspace, workspace_bytes);
  int rc = att_prepare(a, tgt2, memory, b1, bv, geo_ptrs, geo_ld, ar, "rel_cross_attention_backward", needed, st);
  if (rc) return rc;
  AttBwdArgs g = {};
  float *dz = ar.take<float>(64 * QB), *dout_o = ar.take<float>(64 * QB);
  g.hsum = ar.take<float>(64 * QB);
  g.part = ar.take<float>(3 * 4096 * QB);
  g.pairs = ar.take<float>(128 * QB * C);
  float *dhdv = ar.take<float>(128 * (size_t)C * B);
  if (!ar.ok) {
    set_error("rel_cross_attention_backward: workspace too small (%zu bytes given, %zu needed)", workspace_bytes, needed);
    return GF_ERR_WORKSPACE;
  }
  g.o = o, g.lse = lse, g.dout_o = dout_o;
  if ((rc = att_set_smem())) return rc;
  att_bwd_prologue_kernel<<<(unsigned)QB, 64, 0, st>>>(a.out, dy, a.wo, dz, dout_o);
  GF_LAUNCHED();
  if (geo_ptrs)
    rel_cross_attention_bwd_kernel<true><<<dim3(Q, B), ATT_THREADS, ATT_BWD_SMEM, st>>>(a, g);
  else
    rel_cross_attention_bwd_kernel<false><<<dim3(Q, B), ATT_THREADS, ATT_BWD_SMEM, st>>>(a, g);
  GF_LAUNCHED();
  att_bwd_rows_kernel<<<dim3(Q + C, B), 128, 0, st>>>(g.hsum, g.pairs, Q, C, B, a.w1, a.wv, dtgt2, dhdv, dmemory);
  GF_LAUNCHED();
  AttBwdWeights p = {};
  p.part = g.part, p.hsum = g.hsum, p.dhdv = dhdv, p.dz = dz, p.o = o, p.dout_o = dout_o, p.tgt2 = tgt2, p.memory = memory;
  p.dw[0] = dw1, p.dw[1] = dwv, p.dw[2] = dw2, p.dw[3] = dwo;
  p.db[0] = db1, p.db[1] = dbv, p.db[2] = db2, p.db[3] = dbo;
  p.QB = (int)QB, p.CB = C * B;
  att_bwd_weights_kernel<<<dim3(64, 4), 65 * ATT_WS_SLICES, 0, st>>>(p);
  GF_LAUNCHED();
  GF_CUDA(cudaMemsetAsync(db2, 0, 64 * sizeof(float), st));
  if (drel) {
    att_bwd_drel_kernel<<<(unsigned)((QB * C + ATT_DREL_PAIRS - 1) / ATT_DREL_PAIRS), 256, 0, st>>>(g.pairs, Q, C, B, a.w1, a.wv, drel);
    GF_LAUNCHED();
  }
  return GF_OK;
}

#define ATT_BWD_CHECKS(name)                                                                                 \
  GF_CHECK_ARG(o && lse && dy && dtgt2 && dmemory && dw1 && db1 && dw2 && db2 && dwv && dbv && dwo && dbo, \
               name ": null pointer")

extern "C" int gf_rel_cross_attention_backward(const float *tgt2, const float *memory, const float *relative_pos, int Q,
                                               int C, int B, const float *w1, const float *b1, const float *w2,
                                               const float *b2, const float *wv, const float *bv, const float *wo,
                                               const float *bo, const float *out, const float *o, const float *lse,
                                               const float *dy, float *dtgt2, float *dmemory, float *drel, float *dw1,
                                               float *db1, float *dw2, float *db2, float *dwv, float *dbv, float *dwo,
                                               float *dbo, void *workspace, size_t workspace_bytes, void *stream) {
  ATT_COMMON_CHECKS("rel_cross_attention_backward");
  ATT_BWD_CHECKS("rel_cross_attention_backward");
  GF_CHECK_ARG(relative_pos, "rel_cross_attention_backward: null relative_pos");
  AttArgs a = {};
  a.w1 = w1, a.w2 = w2, a.wv = wv, a.wo = wo, a.b2 = b2, a.bo = bo, a.Q = Q, a.C = C, a.B = B, a.rel = relative_pos;
  a.out = const_cast<float *>(out);  // read by the prologue only
  return att_bwd_launch(a, tgt2, memory, b1, bv, nullptr, nullptr, o, lse, dy, dtgt2, dmemory, drel, dw1, db1, dw2,
                        db2, dwv, dbv, dwo, dbo, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int gf_rel_cross_attention_fused_backward(
    const float *tgt2, const float *memory, const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx,
    const float *query_xyz, const float *ctx_xyz, const float *gauss_B, int gauss_ld, const float *pc_min,
    const float *pc_max, int Q, int C, int B, const float *w1, const float *b1, const float *w2, const float *b2,
    const float *wv, const float *bv, const float *wo, const float *bo, const float *out, const float *o,
    const float *lse, const float *dy, float *dtgt2, float *dmemory, float *dw1, float *db1, float *dw2, float *db2,
    float *dwv, float *dbv, float *dwo, float *dbo, void *workspace, size_t workspace_bytes, void *stream) {
  ATT_COMMON_CHECKS("rel_cross_attention_fused_backward");
  ATT_BWD_CHECKS("rel_cross_attention_fused_backward");
  ATT_FUSED_CHECKS("rel_cross_attention_fused_backward");
  AttArgs a = {};
  att_fused_args(a, ctx_idx, query_xyz, ctx_xyz, gauss_B, gauss_ld, pc_min, pc_max, Q, C, B, w1, w2, b2, wv, wo, bo);
  a.out = const_cast<float *>(out);
  return att_bwd_launch(a, tgt2, memory, b1, bv, geo_ptrs, geo_ld, o, lse, dy, dtgt2, dmemory, nullptr, dw1, db1, dw2,
                        db2, dwv, dbv, dwo, dbo, workspace, workspace_bytes, (cudaStream_t)stream);
}
