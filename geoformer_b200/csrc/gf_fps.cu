// Furthest point sampling for sm_100a.
//
// Reference: lib/pointnet2/_ext_src/src/sampling_gpu.cu:72-232 -- ONE 512-thread block per scene,
// coordinates and the running min-distance re-read from global memory in each of the m-1 dependent
// rounds.  GeoFormer calls it with B == 1, so one SM of 148 does everything.
//
// Here a scene is owned by a thread-block CLUSTER (up to 16 CTAs x 1024 threads).  Every thread
// keeps its points AND their running min-distance in registers for the whole kernel (global memory
// is touched once), so a round is: P fused distance updates per thread -> two REDUX warp
// reductions -> one shared-memory hop -> the winning CTA-local candidate (key + coordinates) is
// pushed into every CTA of the cluster through distributed shared memory -> one cluster barrier.
//
// Index-exactness.  The reference's result depends on its reduction shape: thread `tid` scans
// k = tid, tid+bs, ... with a strict '>', then a shared-memory tree keeps the lower slot on ties
// (sampling_gpu.cu:62-68,111-171).  Among equal maxima the winner is therefore the k with the
// smallest (bitrev_L(k mod bs), k div bs), bs = 2^L = the reference's block size.  We reproduce it
// by giving each thread an ascending run of ONE residue class (so its own strict '>' scan keeps the
// right point) and reducing the 64-bit key (d2 bits, ~rank) with max.
#include <cooperative_groups.h>

#include "gf_common.cuh"

namespace cg = cooperative_groups;

namespace gf {

struct __align__(16) FpsSlot {
  uint32_t v, lo;  // key: distance bits, ~rank (0,0 = no eligible point in that CTA)
  float x, y;
  float z;
  float pad[3];
};
static_assert(sizeof(FpsSlot) == 32, "slot is two 16-byte vectors");

constexpr int FPS_MAX_CLUSTER = 16;

__device__ __forceinline__ uint32_t brev_bits(uint32_t c, int L) { return L ? (__brev(c) >> (32 - L)) : 0u; }

// ---- cluster-scope mbarrier signalling (replaces barrier.cluster in the round loop) -----------------
__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint32_t map_to_cta(uint32_t local_addr, uint32_t cta) {
  uint32_t r;
  asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(local_addr), "r"(cta));
  return r;
}
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_fence_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
// local arrival that also announces how many bytes of asynchronous stores this phase will receive
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
// 16-byte store into another CTA's shared memory that completes `16` transaction bytes on that CTA's
// mbarrier when it lands: data and signal travel together, no fence on either side (a cluster-scope
// acquire on the waiter would cost a CCTL.IVALL per round -- 46 % of the kernel in the first version).
__device__ __forceinline__ void st_async_v4(uint32_t remote_addr, uint32_t remote_bar, uint32_t a, uint32_t b,
                                            uint32_t c, uint32_t d) {
  asm volatile("st.async.weak.shared::cluster.mbarrier::complete_tx::bytes.v4.b32 [%0], {%1, %2, %3, %4}, [%5];" ::"r"(
                   remote_addr),
               "r"(a), "r"(b), "r"(c), "r"(d), "r"(remote_bar)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
  const uint32_t a = smem_u32(bar);
  uint32_t done;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(a), "r"(parity)
        : "memory");
  } while (!done);
}

// P > 0 : register-resident variant, thread owns points k = c + bs*(g*P + i), i < P
// P == 0: streaming variant for scenes that do not fit on chip: thread walks k = c + bs*(g + G*i)
//         and keeps the running min-distance in `temp` (global, L2 resident)
template <int T, int P>
__global__ void __launch_bounds__(T, 1)
    fps_cluster_kernel(const float *__restrict__ xyz_all, int N, int m, int L, float *__restrict__ temp_all,
                       int *__restrict__ idx_all) {
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned CS = cluster.num_blocks();
  const unsigned crank = cluster.block_rank();
  const int scene = blockIdx.x / CS;
  const float *__restrict__ xyz = xyz_all + (size_t)scene * N * 3;
  int *__restrict__ idx = idx_all + (size_t)scene * m;

#include "gf_fps_cluster_body.cuh"
}

// A ragged batch: cluster c samples scene c of the table, with that scene's own N and L.  T and P are those of the
// largest scene; a smaller one leaves slots padded with the -1 sentinel, which never wins a round.  The reference's
// tie order only needs CS * T >= 2^L (every residue class has a thread), which the largest scene's plan gives.
constexpr int FPS_BATCH_MAX = 32;
struct FpsScene {
  const float *xyz;  // (N,3) inside the flat array
  int *idx;          // (m) row of the output
  int N, L;
};
struct FpsBatchArgs {
  FpsScene s[FPS_BATCH_MAX];
};

template <int T, int P>
__global__ void __launch_bounds__(T, 1) fps_cluster_batch_kernel(const __grid_constant__ FpsBatchArgs a, int m) {
  static_assert(P > 0, "a ragged batch holds its scenes in registers");
  cg::cluster_group cluster = cg::this_cluster();
  const unsigned CS = cluster.num_blocks();
  const unsigned crank = cluster.block_rank();
  const int scene = blockIdx.x / CS;
  const float *__restrict__ xyz = a.s[scene].xyz;
  int *__restrict__ idx = a.s[scene].idx;
  const int N = a.s[scene].N, L = a.s[scene].L;
  float *__restrict__ temp_all = nullptr;  // register-resident instances only

#include "gf_fps_cluster_body.cuh"
}

// ---------------------------------------------------------------------------------------------------
// Whole-GPU variant for scenes beyond one cluster's register capacity (> 196k points, config c4).
// One 256-thread CTA per SM (cooperative launch => co-resident), the points again live in registers
// (148 x 256 x 32 = 1.2 M), and a round is exchanged through L2: every CTA publishes its candidate as
// five self-validating 8-byte words {payload, round tag} (8-byte accesses are single-copy atomic, so a
// reader can never pair a payload with the wrong round and no fence is needed), warp 0 of every CTA
// polls all slots, reduces them with REDUX and hands the winner to the CTA through shared memory.  ~2.5 us per round instead of ~25 us for
// the one-cluster streaming kernel at 1 M points.
constexpr int FPS_GRID_T = 256;
constexpr int FPS_MAX_GRID_CTAS = 160;  // >= the SM count of the device (148 on B200); checked at launch

constexpr int FPS_SLOT_WORDS = 8;  // 64-byte slots: {v,tag} {lo,tag} {x,tag} {y,tag} {z,tag} + padding
// strong (gpu-scope, relaxed) 64-bit accesses: single-copy atomic and coherent across both L2 partitions
__device__ __forceinline__ void st_cg_v2(uint2 *p, uint32_t payload, uint32_t tag) {
  const unsigned long long w = ((unsigned long long)tag << 32) | payload;
  asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(w) : "memory");
}
__device__ __forceinline__ unsigned long long ld_relaxed_u64(const uint2 *p) {
  unsigned long long w;
  asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
  return w;
}
__device__ __forceinline__ uint32_t poll_word(const uint2 *p, uint32_t tag) {
  unsigned long long w;
  do {
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(w) : "l"(p) : "memory");
  } while ((uint32_t)(w >> 32) != tag);
  return (uint32_t)w;
}

template <int P>
__global__ void __launch_bounds__(FPS_GRID_T, 1)
    fps_grid_kernel(const float *__restrict__ xyz_all, int B, int N, int m, int L, float *__restrict__ temp_all,
                    int *__restrict__ idx_all, uint2 *__restrict__ slots /* [2][gridDim.x][FPS_SLOT_WORDS] */) {
  constexpr int T = FPS_GRID_T;
  __shared__ uint32_t wkey_v[2][T / 32], wkey_lo[2][T / 32];
  __shared__ float s_center[2][4];
  __shared__ uint32_t s_win[2][2];
  const unsigned tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const unsigned nctas = gridDim.x;
  const unsigned u = blockIdx.x * T + tid;
  const unsigned bs = 1u << L;
  const unsigned c = u & (bs - 1), g = u >> L;
  const unsigned G = (nctas * T) >> L;
  const uint32_t rank_hi = L ? (brev_bits(c, L) << (32 - L)) : 0u;
  constexpr int PR = P > 0 ? P : 1;

  for (int b = 0; b < B; ++b) {
    const float *__restrict__ xyz = xyz_all + (size_t)b * N * 3;
    int *__restrict__ idx = idx_all + (size_t)b * m;
    float *__restrict__ temp = P == 0 ? temp_all + (size_t)b * N : nullptr;
    float px[PR], py[PR], pz[PR], tmp[PR];
    if (P > 0) {
#pragma unroll
      for (int i = 0; i < PR; ++i) {
        unsigned k = c + bs * (g * PR + i);
        px[i] = py[i] = pz[i] = 0.f;
        tmp[i] = -1.f;
        if (k < (unsigned)N) {
          px[i] = __ldg(xyz + (size_t)k * 3 + 0);
          py[i] = __ldg(xyz + (size_t)k * 3 + 1);
          pz[i] = __ldg(xyz + (size_t)k * 3 + 2);
          if (!((double)sq3(px[i], py[i], pz[i]) <= 1e-3)) tmp[i] = 1e10f;
        }
      }
    } else {
      for (unsigned k = c + bs * g; k < (unsigned)N; k += bs * G) temp[k] = 1e10f;  // own points only: no sync needed
    }
    float cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
    if (u == 0) idx[0] = 0;

    for (int j = 1; j < m; ++j) {
      // The rounds of the whole launch are numbered 1, 2, 3, ... without a gap, also from the last round of one
      // scene to the first of the next, so consecutive rounds use different buffers: a CTA writes buffer X again
      // only after every CTA has published the round in between, i.e. after every CTA has finished reading X.
      // Tag 0 (the zeroed slots) means "never written".
      const uint32_t tag = (uint32_t)b * (uint32_t)(m - 1) + (uint32_t)j;
      const int buf = tag & 1;
      float best = -1.f;
      uint32_t besti = 0;
      float bx = 0.f, by = 0.f, bz = 0.f;
      if (P > 0) {
#pragma unroll
        for (int i = 0; i < PR; ++i) {
          float d = sq3(px[i] - cx, py[i] - cy, pz[i] - cz);
          float t = fminf(d, tmp[i]);
          tmp[i] = t;
          if (t > best) {
            best = t;
            besti = i;
          }
        }
      } else {
        uint32_t i = 0;
        for (unsigned k = c + bs * g; k < (unsigned)N; k += bs * G, ++i) {
          float x = __ldg(xyz + (size_t)k * 3 + 0), y = __ldg(xyz + (size_t)k * 3 + 1), z = __ldg(xyz + (size_t)k * 3 + 2);
          if ((double)sq3(x, y, z) <= 1e-3) continue;
          float t = fminf(sq3(x - cx, y - cy, z - cz), temp[k]);
          temp[k] = t;
          if (t > best) {
            best = t;
            besti = g + G * i;
            bx = x, by = y, bz = z;
          }
        }
      }
      const bool has = best >= 0.f;
      const uint32_t vb = has ? __float_as_uint(best) : 0u;
      const uint32_t rank = rank_hi | (P > 0 ? (g * PR + besti) : besti);
      const uint32_t lo = has ? ~rank : 0u;
      uint32_t wv = __reduce_max_sync(0xffffffffu, vb);
      uint32_t wl = __reduce_max_sync(0xffffffffu, vb == wv ? lo : 0u);
      if (lane == 0) {
        wkey_v[buf][warp] = wv;
        wkey_lo[buf][warp] = wl;
      }
      __syncthreads();
      uint32_t tv = lane < T / 32 ? wkey_v[buf][lane] : 0u;
      uint32_t tl = lane < T / 32 ? wkey_lo[buf][lane] : 0u;
      const uint32_t cv = __reduce_max_sync(0xffffffffu, tv);
      const uint32_t cl = __reduce_max_sync(0xffffffffu, tv == cv ? tl : 0u);
      const bool owner = has && vb == cv && lo == cl;
      const bool nobody = (cv | cl) == 0u;
      if (owner || (nobody && tid == 0)) {
        if (P > 0 && owner) {
#pragma unroll
          for (int i = 0; i < PR; ++i)
            if (besti == (uint32_t)i) bx = px[i], by = py[i], bz = pz[i];
        }
        uint2 *dst = slots + ((size_t)buf * nctas + blockIdx.x) * FPS_SLOT_WORDS;
        st_cg_v2(dst + 0, cv, tag);
        st_cg_v2(dst + 1, cl, tag);
        st_cg_v2(dst + 2, __float_as_uint(bx), tag);
        st_cg_v2(dst + 3, __float_as_uint(by), tag);
        st_cg_v2(dst + 4, __float_as_uint(bz), tag);
      }
      if (warp == 0) {
        // Poll every CTA's slot of this round.  The key words of all of this lane's slots are requested
        // together (up to 5 slots x 2 words in flight) and only the slots whose tags are not there yet are
        // asked again; the coordinates are fetched from the winning slot alone.  Word-by-word spinning cost
        // one L2 round trip per word, and polling all five words of every slot made the 148 x 32 pollers
        // congest the few L2 lines that hold the slots.
        constexpr int MAXS = (FPS_MAX_GRID_CTAS + 31) / 32;
        uint32_t gv = 0, gl = 0, src = 0;
        unsigned pend = 0;
#pragma unroll
        for (int sI = 0; sI < MAXS; ++sI)
          if (lane + 32u * sI < nctas) pend |= 1u << sI;
        while (pend) {
          unsigned long long w[MAXS][2];
#pragma unroll
          for (int sI = 0; sI < MAXS; ++sI)
            if ((pend >> sI) & 1u) {
              const uint2 *sp = slots + ((size_t)buf * nctas + lane + 32u * sI) * FPS_SLOT_WORDS;
              // one 16-byte request for both key words; each carries its own tag, so a torn pair is detected
              asm volatile("ld.relaxed.gpu.global.v2.u64 {%0, %1}, [%2];"
                           : "=l"(w[sI][0]), "=l"(w[sI][1])
                           : "l"(sp)
                           : "memory");
            }
#pragma unroll
          for (int sI = 0; sI < MAXS; ++sI)
            if (((pend >> sI) & 1u) && (uint32_t)(w[sI][0] >> 32) == tag && (uint32_t)(w[sI][1] >> 32) == tag) {
              pend &= ~(1u << sI);
              const uint32_t sv = (uint32_t)w[sI][0], sl = (uint32_t)w[sI][1];
              if (sv > gv || (sv == gv && sl > gl)) gv = sv, gl = sl, src = lane + 32u * sI;
            }
        }
        const uint32_t mv = __reduce_max_sync(0xffffffffu, gv);
        const uint32_t ml = __reduce_max_sync(0xffffffffu, gv == mv ? gl : 0u);
        const unsigned wm = __ballot_sync(0xffffffffu, gv == mv && gl == ml);
        if (lane == (unsigned)(__ffs(wm) - 1)) {
          const uint2 *sp = slots + ((size_t)buf * nctas + src) * FPS_SLOT_WORDS;
          unsigned long long x, y, z;
          do {  // the three coordinate words of the winner, requested together
            x = ld_relaxed_u64(sp + 2), y = ld_relaxed_u64(sp + 3), z = ld_relaxed_u64(sp + 4);
          } while ((uint32_t)(x >> 32) != tag || (uint32_t)(y >> 32) != tag || (uint32_t)(z >> 32) != tag);
          s_center[buf][0] = __uint_as_float((uint32_t)x);
          s_center[buf][1] = __uint_as_float((uint32_t)y);
          s_center[buf][2] = __uint_as_float((uint32_t)z);
          s_win[buf][0] = mv;
          s_win[buf][1] = ml;
        }
      }
      __syncthreads();
      const uint32_t gv = s_win[buf][0], gl = s_win[buf][1];
      int old;
      if ((gv | gl) == 0u) {  // no eligible point anywhere: the reference's tree yields index 0
        old = 0;
        cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
      } else {
        const uint32_t rk = ~gl;
        old = L ? (int)(((rk & ((1u << (32 - L)) - 1u)) << L) | brev_bits(rk >> (32 - L), L)) : (int)rk;
        cx = s_center[buf][0], cy = s_center[buf][1], cz = s_center[buf][2];
      }
      if (u == 0) idx[j] = old;
    }
  }
}

// lib/pointnet2/_ext_src/include/cuda_utils.h:15-21 -- the block size the reference would use
static int ref_log2_block(int n) {
  int L = 0;
  while ((2 << L) <= n && L < 9) ++L;
  return L;
}

struct FpsPlan {
  int T, P, CS;  // CS == 0: whole-GPU (cooperative) variant, T = 256
};

// Few, fat warps: a round costs (points per SM) x ~10 instructions of arithmetic plus ~150 instructions
// of reduction / signalling PER WARP, so 8 warps with up to 32 register-resident points per thread beat
// 32 warps with 8 (measured: 1.87 us -> see profiles/).  Capacity = CS * T * P.
static const int kFpsP256[] = {1, 2, 4, 8, 12, 16, 20, 25, 32};

static FpsPlan plan_fps(int N, int max_cs) {
  if (N < 512) return {256, N <= 256 ? 1 : 2, 1};  // reference block size bs <= 256 <= T
  // smallest power-of-two cluster (>= 2 so that CS * 256 covers the 512 residue classes) whose
  // 256-thread CTAs hold the scene with P <= 32; prefer the largest cluster (least work per SM per round)
  int cs = max_cs;
  while (cs > 2 && (long long)(cs / 2) * 256 * 4 >= N) cs /= 2;  // tiny scenes: do not spread thinner than 4 pts/thread
  for (int pi = 0; pi < (int)(sizeof(kFpsP256) / sizeof(int)); ++pi)
    if ((long long)cs * 256 * kFpsP256[pi] >= N) return {256, kFpsP256[pi], cs};
  if ((long long)max_cs * 512 * 24 >= N) return {512, 24, max_cs};
  // beyond one cluster: one CTA per SM, registers if the scene fits (P <= 32), else streaming from L2
  int ctas = num_sms() & ~1;  // even, so that CTAs * 256 covers whole sets of 512 residue classes
  if (ctas > FPS_MAX_GRID_CTAS) ctas = FPS_MAX_GRID_CTAS;  // what launch_fps_grid launches
  const int p_opts[4] = {8, 16, 24, 32};
  for (int pi = 0; pi < 4; ++pi)
    if ((long long)ctas * FPS_GRID_T * p_opts[pi] >= N) return {FPS_GRID_T, p_opts[pi], 0};
  return {FPS_GRID_T, 0, 0};
}

template <int P>
static int launch_fps_grid(const float *xyz, int B, int N, int m, int L, float *temp, int *idx, uint2 *slots,
                           cudaStream_t st) {
  int ctas = num_sms() & ~1;
  if (ctas > FPS_MAX_GRID_CTAS) ctas = FPS_MAX_GRID_CTAS;
  GF_CUDA(cudaMemsetAsync(slots, 0, sizeof(uint2) * 2 * FPS_SLOT_WORDS * (size_t)ctas, st));  // tag 0 = never written
  void *args[] = {(void *)&xyz, &B, &N, &m, &L, &temp, &idx, &slots};
  GF_CUDA(cudaLaunchCooperativeKernel((const void *)fps_grid_kernel<P>, dim3(ctas), dim3(FPS_GRID_T), args, 0, st));
  count_launch();
  return GF_OK;
}

// B clusters of CS CTAs x T threads, one per scene
template <class... KArgs, class... Args>
static int launch_clusters(void (*kern)(KArgs...), int T, int B, int CS, cudaStream_t st, Args... args) {
  if (CS > 8) GF_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3((unsigned)B * CS, 1, 1);
  cfg.blockDim = dim3((unsigned)T, 1, 1);
  cfg.dynamicSmemBytes = 0;
  cfg.stream = st;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = CS;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  // FPS is the longest dependency chain of the hot path (m - 1 dependent rounds on <= 16 SMs): its cluster should be
  // placed ahead of queued bulk work.  As a launch attribute the priority also survives stream capture (a graph's
  // kernel nodes do not inherit the priority of the stream they were captured on).
  static const int prio_hi = [] {
    int lo = 0, hi = 0;
    return cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess ? hi : 0;
  }();
  attr[1].id = cudaLaunchAttributePriority;
  attr[1].val.priority = prio_hi;
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  GF_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
  count_launch();
  return GF_OK;
}

template <int T, int P>
static int launch_fps(const float *xyz, int B, int N, int m, int L, int CS, float *temp, int *idx, cudaStream_t st) {
  return launch_clusters(fps_cluster_kernel<T, P>, T, B, CS, st, xyz, N, m, L, temp, idx);
}

template <int T, int P>
static int launch_fps_batch(const FpsBatchArgs &a, int B, int m, int CS, cudaStream_t st) {
  return launch_clusters(fps_cluster_batch_kernel<T, P>, T, B, CS, st, a, m);
}

static int max_cluster_size() {
  // 16 (non-portable) when the device can co-schedule a 16-CTA x 1024-thread cluster, else 8
  static int cached = 0;
  if (cached) return cached;
  auto kern = fps_cluster_kernel<1024, 0>;
  int ok16 = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(16, 1, 1);
    cfg.blockDim = dim3(1024, 1, 1);
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 16;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, kern, &cfg) == cudaSuccess && n >= 1) ok16 = 1;
  }
  (void)cudaGetLastError();
  cached = ok16 ? 16 : 8;
  return cached;
}

}  // namespace gf

using namespace gf;

// workspace layout (only for scenes beyond the smallest cluster capacity): [slots: 4 x 256 uint4][temp: (B,N) f32]
static const size_t kFpsSlotBytes = sizeof(uint2) * 2 * FPS_SLOT_WORDS * 256;  // up to 256 CTAs

extern "C" size_t gf_fps_workspace_bytes(int B, int N, int m) {
  (void)m;
  if (B <= 0 || N <= 0) return 0;
  if ((long long)8 * 512 * 24 >= N) return 0;  // fits an 8-CTA cluster on every device: no scratch at all
  return align256(kFpsSlotBytes) + align256(sizeof(float) * (size_t)B * N);
}

extern "C" int gf_furthest_point_sampling(const float *xyz, int B, int N, int m, int *idx, void *workspace,
                                          size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(B >= 0 && N >= 0 && m >= 0, "furthest_point_sampling: negative size");
  if (B == 0 || m == 0) return GF_OK;
  GF_CHECK_ARG(idx, "furthest_point_sampling: null idx");
  cudaStream_t st = (cudaStream_t)stream;
  if (N == 0) {  // nothing to sample from: the zero-initialised output of sampling.cpp:71-73
    GF_CUDA(cudaMemsetAsync(idx, 0, sizeof(int) * (size_t)B * m, st));
    return GF_OK;
  }
  GF_CHECK_ARG(xyz, "furthest_point_sampling: null xyz");
  const int L = ref_log2_block(N);
  FpsPlan p = plan_fps(N, max_cluster_size());
  float *temp = nullptr;
  uint2 *slots = nullptr;
  if (p.P == 0 || p.CS == 0) {
    size_t need = align256(kFpsSlotBytes) + align256(sizeof(float) * (size_t)B * N);
    if (workspace == nullptr || workspace_bytes < need) {
      set_error("furthest_point_sampling: N=%d needs a %zu-byte workspace (gf_fps_workspace_bytes)", N, need);
      return GF_ERR_WORKSPACE;
    }
    slots = (uint2 *)workspace;
    temp = (float *)((char *)workspace + align256(kFpsSlotBytes));
  }
  if (p.CS == 0) {
    if (p.P == 8) return launch_fps_grid<8>(xyz, B, N, m, L, temp, idx, slots, st);
    if (p.P == 16) return launch_fps_grid<16>(xyz, B, N, m, L, temp, idx, slots, st);
    if (p.P == 24) return launch_fps_grid<24>(xyz, B, N, m, L, temp, idx, slots, st);
    if (p.P == 32) return launch_fps_grid<32>(xyz, B, N, m, L, temp, idx, slots, st);
    return launch_fps_grid<0>(xyz, B, N, m, L, temp, idx, slots, st);
  }
#define GF_FPS_CASE(TT, PP) \
  if (p.T == TT && p.P == PP) return launch_fps<TT, PP>(xyz, B, N, m, L, p.CS, temp, idx, st)
  GF_FPS_CASE(256, 1);
  GF_FPS_CASE(256, 2);
  GF_FPS_CASE(256, 4);
  GF_FPS_CASE(256, 8);
  GF_FPS_CASE(256, 12);
  GF_FPS_CASE(256, 16);
  GF_FPS_CASE(256, 20);
  GF_FPS_CASE(256, 25);
  GF_FPS_CASE(256, 32);
  GF_FPS_CASE(512, 24);
#undef GF_FPS_CASE
  set_error("furthest_point_sampling: no kernel variant for N=%d", N);
  return GF_ERR_INVALID;
}

// ---- a ragged batch: scenes b of the flat (offsets[B], 3) array --------------------------------------------------
// Scenes that fit one cluster (N <= max_cs * 512 * 24) go through ONE launch per 32 of them, planned for the largest;
// a larger scene runs the whole-GPU kernel of the single-scene call, after the cluster launches.  The largest scene
// sets the cluster size: at the model's sizes (60k-150k points) a smaller cluster cannot hold it (8 CTAs: 98,304
// points), so a batch with more scenes than co-resident clusters runs them in waves rather than on thinner clusters.
static int launch_fps_batch(const FpsPlan &p, const FpsBatchArgs &a, int B, int m, cudaStream_t st) {
#define GF_FPS_CASE(TT, PP) \
  if (p.T == TT && p.P == PP) return launch_fps_batch<TT, PP>(a, B, m, p.CS, st)
  GF_FPS_CASE(256, 1);
  GF_FPS_CASE(256, 2);
  GF_FPS_CASE(256, 4);
  GF_FPS_CASE(256, 8);
  GF_FPS_CASE(256, 12);
  GF_FPS_CASE(256, 16);
  GF_FPS_CASE(256, 20);
  GF_FPS_CASE(256, 25);
  GF_FPS_CASE(256, 32);
  GF_FPS_CASE(512, 24);
#undef GF_FPS_CASE
  set_error("furthest_point_sampling_batch: no cluster kernel variant for T=%d P=%d", p.T, p.P);
  return GF_ERR_INVALID;
}

static int fps_cluster_capacity() { return max_cluster_size() * 512 * 24; }

extern "C" size_t gf_fps_batch_workspace_bytes(const int *offsets, int B, int m) {
  if (!offsets || B <= 0) return 0;
  size_t need = 0;
  for (int b = 0; b < B; ++b) {
    const size_t w = gf_fps_workspace_bytes(1, offsets[b + 1] - offsets[b], m);
    if (w > need) need = w;
  }
  return need;
}

extern "C" int gf_furthest_point_sampling_batch(const float *xyz, const int *offsets, int B, int m, int *idx,
                                                void *workspace, size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(B >= 0 && m >= 0, "furthest_point_sampling_batch: negative size");
  if (B == 0 || m == 0) return GF_OK;
  GF_CHECK_ARG(offsets && idx, "furthest_point_sampling_batch: null offsets or idx");
  GF_CHECK_ARG(offsets[0] == 0, "furthest_point_sampling_batch: offsets[0] = %d, not 0", offsets[0]);
  for (int b = 0; b < B; ++b)
    GF_CHECK_ARG(offsets[b + 1] >= offsets[b], "furthest_point_sampling_batch: offsets fall at scene %d", b);
  GF_CHECK_ARG(xyz || offsets[B] == 0, "furthest_point_sampling_batch: null xyz");
  cudaStream_t st = (cudaStream_t)stream;
  const int cap = fps_cluster_capacity();
  int Nmax = 0;
  for (int b = 0; b < B; ++b) {
    const int N = offsets[b + 1] - offsets[b];
    if (N <= cap && N > Nmax) Nmax = N;
  }
  if (Nmax > 0) {
    const FpsPlan p = plan_fps(Nmax, max_cluster_size());
    FpsBatchArgs a;
    int n = 0;
    for (int b = 0; b <= B; ++b) {
      const int N = b < B ? offsets[b + 1] - offsets[b] : 0;
      if (b < B && N >= 1 && N <= cap) a.s[n++] = {xyz + (size_t)offsets[b] * 3, idx + (size_t)b * m, N, ref_log2_block(N)};
      if (n == FPS_BATCH_MAX || (b == B && n > 0)) {
        const int rc = launch_fps_batch(p, a, n, m, st);
        if (rc) return rc;
        n = 0;
      }
    }
  }
  for (int b = 0; b < B; ++b) {
    const int N = offsets[b + 1] - offsets[b];
    if (N >= 1 && N <= cap) continue;  // N == 0: the single-scene call writes the zero row
    const int rc = gf_furthest_point_sampling(xyz + (size_t)offsets[b] * 3, 1, N, m, idx + (size_t)b * m, workspace,
                                              workspace_bytes, stream);
    if (rc) return rc;
  }
  return GF_OK;
}
