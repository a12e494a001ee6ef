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

#include <algorithm>
#include <iterator>
#include <type_traits>

#include "gf_common.cuh"
#include "gf_fps.cuh"

namespace cg = cooperative_groups;

namespace gf {

// ---- the sampling rules of every FPS kernel ----------------------------------------------------------------------

// |p|^2 > 1e-3, compared in double (sampling_gpu.cu:103-104; sampling.cpp:74-76): only such a point can be a seed
__device__ __forceinline__ bool fps_eligible(float x, float y, float z) { return !((double)sq3(x, y, z) <= 1e-3); }

// The rank of original index i, (bitrev_L(i mod 2^L), i div 2^L) as one word: ascending rank is the reference's order
// among equal distances.  fps_rank_hi is the part of the residue c = i mod 2^L, bitrev_L(c) in the top L bits.
__device__ __forceinline__ uint32_t fps_rank_hi(uint32_t c, int L) { return L ? (__brev(c) >> (32 - L)) << (32 - L) : 0u; }
__device__ __forceinline__ uint32_t fps_rank(uint32_t i, int L) { return fps_rank_hi(i & ((1u << L) - 1u), L) | (i >> L); }
// the original index of the key word lo = ~rank
__device__ __forceinline__ int fps_index(uint32_t lo, int L) {
  const uint32_t rk = ~lo;
  return L ? (int)(((rk & ((1u << (32 - L)) - 1u)) << L) | (__brev(rk >> (32 - L)) >> (32 - L))) : (int)rk;
}

// A candidate's 64-bit key: the bits of its running minimum, then ~rank; the largest key wins a round, and {0, 0}
// stands for no eligible point.
struct FpsKey {
  uint32_t v, lo;
};
__device__ __forceinline__ bool operator==(FpsKey a, FpsKey b) { return a.v == b.v && a.lo == b.lo; }
__device__ __forceinline__ bool operator>(FpsKey a, FpsKey b) { return a.v > b.v || (a.v == b.v && a.lo > b.lo); }
// the largest key of the warp, by two REDUX
__device__ __forceinline__ FpsKey warp_max(FpsKey k) {
  const uint32_t v = __reduce_max_sync(0xffffffffu, k.v);
  return {v, __reduce_max_sync(0xffffffffu, k.v == v ? k.lo : 0u)};
}

// The end of a round won by key w at (x, y, z): returns the seed and moves the centre c there.  With no eligible
// point anywhere (w = {0, 0}) the reference's tree yields index 0, and the centre is point 0.
__device__ __forceinline__ int fps_round_end(FpsKey w, float x, float y, float z, const float *__restrict__ xyz, int L,
                                             float &cx, float &cy, float &cz) {
  if ((w.v | w.lo) == 0u) {
    cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
    return 0;
  }
  cx = x, cy = y, cz = z;
  return fps_index(w.lo, L);
}

// ---- the cluster kernels -----------------------------------------------------------------------------------------

struct __align__(16) FpsSlot {
  uint32_t v, lo;  // key (0,0 = no eligible point in that CTA)
  float x, y;
  float z;
  float pad[3];
};
static_assert(sizeof(FpsSlot) == 32, "slot is two 16-byte vectors");

constexpr int FPS_MAX_CLUSTER = 16;

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

// thread u = g * 2^L + c of the cluster owns points k = c + 2^L * (g*P + i), i < P, in registers
template <int T, int P>
__global__ void __launch_bounds__(T, 1)
    fps_cluster_kernel(const float *__restrict__ xyz_all, int N, int m, int L, int *__restrict__ idx_all) {
  static_assert(P > 0, "a scene of the cluster kernel is held in registers");
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
  const uint32_t rank_hi = fps_rank_hi(c, L);
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
          if (fps_eligible(px[i], py[i], pz[i])) tmp[i] = 1e10f;
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
          if (!fps_eligible(x, y, z)) continue;
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
      const FpsKey key = {has ? __float_as_uint(best) : 0u, has ? ~(rank_hi | (P > 0 ? (g * PR + besti) : besti)) : 0u};
      const FpsKey wk = warp_max(key);
      if (lane == 0) {
        wkey_v[buf][warp] = wk.v;
        wkey_lo[buf][warp] = wk.lo;
      }
      __syncthreads();
      const FpsKey ck = warp_max({lane < T / 32 ? wkey_v[buf][lane] : 0u, lane < T / 32 ? wkey_lo[buf][lane] : 0u});
      // field by field: `has && key == ck` allocates the kernel's registers differently
      const bool owner = has && key.v == ck.v && key.lo == ck.lo;
      const bool nobody = (ck.v | ck.lo) == 0u;
      if (owner || (nobody && tid == 0)) {
        if (P > 0 && owner) {
#pragma unroll
          for (int i = 0; i < PR; ++i)
            if (besti == (uint32_t)i) bx = px[i], by = py[i], bz = pz[i];
        }
        uint2 *dst = slots + ((size_t)buf * nctas + blockIdx.x) * FPS_SLOT_WORDS;
        st_cg_v2(dst + 0, ck.v, tag);
        st_cg_v2(dst + 1, ck.lo, tag);
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
        FpsKey gk = {0u, 0u};
        uint32_t src = 0;
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
              const FpsKey sk = {(uint32_t)w[sI][0], (uint32_t)w[sI][1]};
              if (sk > gk) gk = sk, src = lane + 32u * sI;
            }
        }
        const FpsKey mk = warp_max(gk);
        if (lane == (unsigned)(__ffs(__ballot_sync(0xffffffffu, gk == mk)) - 1)) {
          const uint2 *sp = slots + ((size_t)buf * nctas + src) * FPS_SLOT_WORDS;
          unsigned long long x, y, z;
          do {  // the three coordinate words of the winner, requested together
            x = ld_relaxed_u64(sp + 2), y = ld_relaxed_u64(sp + 3), z = ld_relaxed_u64(sp + 4);
          } while ((uint32_t)(x >> 32) != tag || (uint32_t)(y >> 32) != tag || (uint32_t)(z >> 32) != tag);
          s_center[buf][0] = __uint_as_float((uint32_t)x);
          s_center[buf][1] = __uint_as_float((uint32_t)y);
          s_center[buf][2] = __uint_as_float((uint32_t)z);
          s_win[buf][0] = mk.v;
          s_win[buf][1] = mk.lo;
        }
      }
      __syncthreads();
      const int old = fps_round_end({s_win[buf][0], s_win[buf][1]}, s_center[buf][0], s_center[buf][1],
                                    s_center[buf][2], xyz, L, cx, cy, cz);
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

// The cluster kernels' shapes, in the order plan_fps tries them; a cluster of CS CTAs holds CS * T * P points.  Few,
// fat warps: a round costs (points per SM) x ~10 instructions of arithmetic plus ~150 instructions of reduction /
// signalling PER WARP, so 8 warps with up to 32 register-resident points per thread beat 32 warps with 8 (measured:
// 1.87 us -> see profiles/).
struct FpsShape {
  int T, P;
};
constexpr FpsShape kFpsClusterShapes[] = {{256, 1},  {256, 2},  {256, 4},  {256, 8},  {256, 12},
                                          {256, 16}, {256, 20}, {256, 25}, {256, 32}, {512, 24}};
constexpr FpsShape kFpsLargestShape = kFpsClusterShapes[std::size(kFpsClusterShapes) - 1];
// the grid kernel's points per thread; the last, 0, streams them from L2 and takes any N
constexpr int kFpsGridP[] = {8, 16, 24, 32, 0};

static long long fps_cluster_capacity(int cs) { return (long long)cs * kFpsLargestShape.T * kFpsLargestShape.P; }

struct FpsPlan {
  bool grid;  // the whole-GPU cooperative kernel (T = FPS_GRID_T) instead of one cluster per scene
  int T, P;   // threads per CTA, points per thread
  int ctas;   // CTAs per cluster, or of the whole grid
};

static FpsPlan plan_fps(int N, int max_cs) {
  if (N < 512) return {false, 256, N <= 256 ? 1 : 2, 1};  // reference block size bs <= 256 <= T
  // smallest power-of-two cluster (>= 2 so that CS * 256 covers the 512 residue classes) whose
  // 256-thread CTAs hold the scene with P <= 32; prefer the largest cluster (least work per SM per round)
  int cs = max_cs;
  while (cs > 2 && (long long)(cs / 2) * 256 * 4 >= N) cs /= 2;  // tiny scenes: do not spread thinner than 4 pts/thread
  // a cluster smaller than max_cs holds the scene at P = 4, so the 512-thread shape only ever runs on max_cs CTAs
  for (const FpsShape &s : kFpsClusterShapes)
    if ((long long)cs * s.T * s.P >= N) return {false, s.T, s.P, cs};
  // beyond one cluster: one CTA per SM, registers if the scene fits (P <= 32), else streaming from L2
  const int ctas = std::min(num_sms() & ~1, FPS_MAX_GRID_CTAS);  // even: CTAs * 256 covers whole sets of 512 classes
  int P = 0;  // the streaming instance, unless the scene fits in registers
  for (int p : kFpsGridP)
    if (P == 0 && p && (long long)ctas * FPS_GRID_T * p >= N) P = p;
  return {true, FPS_GRID_T, P, ctas};
}

// launch(T, P) with the cluster shape (T, P) as compile-time constants (std::integral_constant)
template <int I = 0, typename F>
static int with_cluster_shape(int T, int P, F &&launch) {
  constexpr FpsShape s = kFpsClusterShapes[I];
  if (T == s.T && P == s.P) return launch(std::integral_constant<int, s.T>(), std::integral_constant<int, s.P>());
  if constexpr (I + 1 < (int)std::size(kFpsClusterShapes)) {
    return with_cluster_shape<I + 1>(T, P, launch);
  } else {
    set_error("furthest_point_sampling: no cluster kernel for T=%d P=%d", T, P);
    return GF_ERR_INVALID;
  }
}

// launch(P) with the grid kernel's P as a compile-time constant
template <int I = 0, typename F>
static int with_grid_p(int P, F &&launch) {
  if (P == kFpsGridP[I]) return launch(std::integral_constant<int, kFpsGridP[I]>());
  if constexpr (I + 1 < (int)std::size(kFpsGridP)) {
    return with_grid_p<I + 1>(P, launch);
  } else {
    set_error("furthest_point_sampling: no grid kernel for P=%d", P);
    return GF_ERR_INVALID;
  }
}

// FPS is the longest dependency chain of the hot path (m - 1 dependent rounds on a few SMs): its CTAs should be
// placed ahead of queued bulk work.  As a launch attribute the priority also survives stream capture (a graph's
// kernel nodes do not inherit the priority of the stream they were captured on).
static cudaLaunchAttribute fps_priority() {
  static const int prio_hi = [] {
    int lo = 0, hi = 0;
    return cudaDeviceGetStreamPriorityRange(&lo, &hi) == cudaSuccess ? hi : 0;
  }();
  cudaLaunchAttribute a;
  a.id = cudaLaunchAttributePriority;
  a.val.priority = prio_hi;
  return a;
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
  attr[1] = fps_priority();
  cfg.attrs = attr;
  cfg.numAttrs = 2;
  GF_CUDA(cudaLaunchKernelEx(&cfg, kern, args...));
  count_launch();
  return GF_OK;
}

static int max_cluster_size() {
  // 16 (non-portable) when the device can co-schedule a 16-CTA cluster of the largest shape, else 8
  static int cached = 0;
  if (cached) return cached;
  auto kern = fps_cluster_kernel<kFpsLargestShape.T, kFpsLargestShape.P>;
  int ok16 = 0;
  if (cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1) == cudaSuccess) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(16, 1, 1);
    cfg.blockDim = dim3(kFpsLargestShape.T, 1, 1);
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

// The workspace of the whole-GPU kernel, for sizing (over a null workspace the Arena only measures) and for the
// launch: exchange slots for up to 256 CTAs, then the (B, N) running minima of the streaming instance.
static Arena fps_carve(void *workspace, size_t workspace_bytes, int B, int N, uint2 **slots, float **temp) {
  Arena ar(workspace, workspace_bytes);
  *slots = ar.take<uint2>(2 * FPS_SLOT_WORDS * 256);
  *temp = ar.take<float>((size_t)B * N);
  return ar;
}

// ---------------------------------------------------------------------------------------------------
// Culled FPS on the cell order of the kNN grid: the seeds of a batched guidance call, one 1024-thread CTA per scene.
// A new seed c can only lower the running minimum t of a point closer to c than t, a neighbourhood of c that shrinks
// as seeds accumulate.  The points are taken in blocks of S consecutive cell-order positions (KnnGridBuffers::sorted),
// each with the tight box of its eligible points and the largest key of its points kept on chip; a round updates a
// block only if a lower bound of sq3(p - c) over its box is below the block's largest t, which skips 87-94 % of the
// point updates at c2 (tools/fps_cells_mirror.py).  Keys, tie order and the no-eligible-point rule are those of the
// sampling rules above, so the seeds are the reference's bit for bit.  The key order (FpsKey's operator>), the rank
// (fps_rank) and the end of a round (fps_round_end) are written out in place here: through those helpers the kernel
// compiled to other code and bench.py ran 0.1-0.3 % slower on a B200 (profiles/r13).
//
// Exactness of a skip: every point of a skipped block keeps t, because its computed d = sq3(px - cx, ...) >= lb >= t.
// Per axis fl(px - cx) is at least the box gap fl(lo - cx) (or fl(cx - hi)) in magnitude, since rounding is monotonic,
// and sq3 is monotonic in the magnitudes of its arguments: sq3 of the gaps never exceeds the computed d.  The bound is
// shrunk by 2^-20 all the same, which can only make a block update that did not need it.
//
// A round: every warp tests its own blocks (block b: warp b % NW, lane (b / NW) % 32, state at warp-major index so
// that a warp's lanes read consecutive words) and appends the ones to update to one list; after a barrier all warps
// take the list U blocks at a time (a warp per block, the U blocks' loads in flight together), so the round's
// dependent L2 round trips are shared by the whole CTA however the updated blocks are spread; after a second barrier
// every warp reduces its blocks' keys, and a third closes the round (candidates double-buffered by round parity).
constexpr int FPS_CELLS_T = 1024;
constexpr int FPS_CELLS_NW = FPS_CELLS_T / 32;
constexpr int FPS_CELLS_WORDS = 12;               // per block: box lo xyz, hi xyz, key (v, lo), key's point xyz, list
constexpr size_t FPS_CELLS_SMEM_MAX = 96 * 1024;  // the largest S (512 points) keeps every batchable scene under it
constexpr float FPS_CELLS_SHRINK = 1.f - 1.f / 1048576.f;

struct FpsCellsSlot {
  uint32_t v, lo;
  float x, y, z;
};

template <int SPL>  // S = 32 * SPL points per block, SPL per lane
__global__ void __launch_bounds__(FPS_CELLS_T, 1)
    fps_cells_kernel(const float4 *__restrict__ sorted, const float *__restrict__ xyz, int N, int m, int L,
                     float *__restrict__ tmin, int *__restrict__ idx) {
  // U blocks of a warp are updated together, QC points per lane and block loaded at a time: 4 loads in flight
  constexpr int S = 32 * SPL, U = SPL >= 4 ? 1 : 4 / SPL, QC = SPL > 4 ? 4 : SPL, NW = FPS_CELLS_NW;
  extern __shared__ uint32_t fc_smem[];
  __shared__ FpsCellsSlot slot[2][NW];
  __shared__ int list_n[2];
  const unsigned lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int nb = (N + S - 1) / S;
  const int nper = (nb + NW - 1) / NW;  // state of block warp + NW * n at [warp * nper + n]
  const int nown = (int)warp < nb ? (nb - 1 - (int)warp) / NW + 1 : 0;
  // FPS_CELLS_WORDS arrays of NW * nper words: box lo x y z, hi x y z, key v lo, key's point x y z, update list
  const int stride = NW * nper;
  float *const sf = (float *)fc_smem;
  uint32_t *const su = fc_smem;
  int *const list = (int *)fc_smem + 11 * stride;
  const uint32_t low = (1u << L) - 1u;

  float cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
  if (threadIdx.x == 0) idx[0] = 0, list_n[0] = list_n[1] = 0;

  // Updates blocks b[u] (b[u] < 0: none; warp-uniform) for the seed at c; lane 0 stores their states.  init: the
  // first round, which also sets the running minima (1e10 if eligible, else -1: gf_fps_cluster_body.cuh) and boxes.
  auto update = [&](const int (&b)[U], bool init) {
    uint32_t bv[U] = {}, bl[U] = {};
    float bx[U], by[U], bz[U];
    float lx[U], ly[U], lz[U], hx[U], hy[U], hz[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      bx[u] = by[u] = bz[u] = 0.f;
      lx[u] = ly[u] = lz[u] = __int_as_float(0x7f800000), hx[u] = hy[u] = hz[u] = -lx[u];
    }
#pragma unroll 1
    for (int q0 = 0; q0 < SPL; q0 += QC) {
      float4 p[U][QC];
      float t[U][QC];
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int q = 0; q < QC; ++q) {
          const int pos = b[u] * S + (q0 + q) * 32 + (int)lane;
          p[u][q] = make_float4(0.f, 0.f, 0.f, 0.f);
          t[u][q] = -1.f;
          if (b[u] >= 0 && pos < N) {
            p[u][q] = __ldg(sorted + pos);
            if (!init) t[u][q] = tmin[pos];
          }
        }
#pragma unroll
      for (int u = 0; u < U; ++u)
#pragma unroll
        for (int q = 0; q < QC; ++q) {
          const int pos = b[u] * S + (q0 + q) * 32 + (int)lane;
          const bool real = b[u] >= 0 && pos < N;  // b[u] < 0 gives a negative pos: no point, nothing stored
          const float4 a = p[u][q];
          float told = t[u][q];
          if (init && real && fps_eligible(a.x, a.y, a.z)) {
            told = 1e10f;
            lx[u] = fminf(lx[u], a.x), ly[u] = fminf(ly[u], a.y), lz[u] = fminf(lz[u], a.z);
            hx[u] = fmaxf(hx[u], a.x), hy[u] = fmaxf(hy[u], a.y), hz[u] = fmaxf(hz[u], a.z);
          }
          const float nt = fminf(sq3(a.x - cx, a.y - cy, a.z - cz), told);
          if (real && (init || nt != told)) tmin[pos] = nt;
          if (nt >= 0.f) {
            const uint32_t i = (uint32_t)__float_as_int(a.w);
            const uint32_t v = __float_as_uint(nt), lo = ~(__brev(i & low) | (i >> L));
            if (v > bv[u] || (v == bv[u] && lo > bl[u])) bv[u] = v, bl[u] = lo, bx[u] = a.x, by[u] = a.y, bz[u] = a.z;
          }
        }
    }
#pragma unroll
    for (int u = 0; u < U; ++u) {
      if (b[u] < 0) continue;
      const FpsKey wk = warp_max({bv[u], bl[u]});
      const uint32_t wv = wk.v, wl = wk.lo;
      const int src = __ffs(__ballot_sync(0xffffffffu, bv[u] == wv && bl[u] == wl)) - 1;
      const float x = __shfl_sync(0xffffffffu, bx[u], src), y = __shfl_sync(0xffffffffu, by[u], src),
                  z = __shfl_sync(0xffffffffu, bz[u], src);
      float box[6];
      if (init) {  // the box as order-preserving integers: six REDUX instead of thirty shuffles
        box[0] = ord2f(__reduce_min_sync(0xffffffffu, f2ord(lx[u])));
        box[1] = ord2f(__reduce_min_sync(0xffffffffu, f2ord(ly[u])));
        box[2] = ord2f(__reduce_min_sync(0xffffffffu, f2ord(lz[u])));
        box[3] = ord2f(__reduce_max_sync(0xffffffffu, f2ord(hx[u])));
        box[4] = ord2f(__reduce_max_sync(0xffffffffu, f2ord(hy[u])));
        box[5] = ord2f(__reduce_max_sync(0xffffffffu, f2ord(hz[u])));
      }
      if (lane == 0) {
        const int e = (b[u] % NW) * nper + b[u] / NW;
        su[6 * stride + e] = wv, su[7 * stride + e] = wl;
        sf[8 * stride + e] = x, sf[9 * stride + e] = y, sf[10 * stride + e] = z;
        if (init)
#pragma unroll
          for (int a = 0; a < 6; ++a) sf[a * stride + e] = box[a];
      }
    }
  };

  for (int n0 = 0; n0 < nown; n0 += U) {  // the first round: every block, each warp its own
    int b[U];
#pragma unroll
    for (int u = 0; u < U; ++u) b[u] = n0 + u < nown ? (int)warp + NW * (n0 + u) : -1;
    update(b, true);
  }
  __syncthreads();  // the states written by lane 0 of a warp, read by the block's lane below

  for (int j = 1; j < m; ++j) {
    const int buf = j & 1;
    if (j > 1) {
      // the blocks of this warp the seed at c can change, appended to the round's list
      for (int n0 = 0; n0 < nown; n0 += 32) {
        const int n = n0 + (int)lane;
        bool up = false;
        if (n < nown) {
          const int e = (int)warp * nper + n;
          const float gx = fmaxf(fmaxf(sf[e] - cx, cx - sf[3 * stride + e]), 0.f);
          const float gy = fmaxf(fmaxf(sf[stride + e] - cy, cy - sf[4 * stride + e]), 0.f);
          const float gz = fmaxf(fmaxf(sf[2 * stride + e] - cz, cz - sf[5 * stride + e]), 0.f);
          // a block without an eligible point has key v = 0 and is never updated
          up = __fmul_rn(sq3(gx, gy, gz), FPS_CELLS_SHRINK) < __uint_as_float(su[6 * stride + e]);
        }
        const unsigned mask = __ballot_sync(0xffffffffu, up);
        int base = 0;
        if (lane == 0 && mask) base = atomicAdd(&list_n[buf], __popc(mask));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (up) list[base + __popc(mask & ((1u << lane) - 1u))] = (int)warp + NW * n;
      }
      __syncthreads();
      const int cnt = list_n[buf];
      for (int i0 = (int)warp * U; i0 < cnt; i0 += NW * U) {
        int b[U];
#pragma unroll
        for (int u = 0; u < U; ++u) b[u] = i0 + u < cnt ? list[i0 + u] : -1;
        update(b, false);
      }
      __syncthreads();  // every updated state is visible to its owner
    }
    // this warp's largest block key, then the CTA's
    uint32_t bv = 0, bl = 0;
    int be = 0;
    for (int n = (int)lane; n < nown; n += 32) {
      const int e = (int)warp * nper + n;
      const uint32_t v = su[6 * stride + e], lo = su[7 * stride + e];
      if (v > bv || (v == bv && lo > bl)) bv = v, bl = lo, be = e;
    }
    const FpsKey wk = warp_max({bv, bl});
    const uint32_t wv = wk.v, wl = wk.lo;
    if ((unsigned)(__ffs(__ballot_sync(0xffffffffu, bv == wv && bl == wl)) - 1) == lane)
      slot[buf][warp] = (wv | wl) ? FpsCellsSlot{wv, wl, sf[8 * stride + be], sf[9 * stride + be], sf[10 * stride + be]}
                                  : FpsCellsSlot{0u, 0u, 0.f, 0.f, 0.f};
    if (threadIdx.x == 0) list_n[buf ^ 1] = 0;  // the next round's list (its last reader finished before this round)
    __syncthreads();
    const uint32_t sv = slot[buf][lane].v, sl = slot[buf][lane].lo;  // NW == 32: one candidate per lane
    const FpsKey gk = warp_max({sv, sl});
    const uint32_t gv = gk.v, gl = gk.lo;
    int old;
    if ((gv | gl) == 0u) {  // no eligible point anywhere: the reference's tree yields index 0
      old = 0;
      cx = __ldg(xyz + 0), cy = __ldg(xyz + 1), cz = __ldg(xyz + 2);
    } else {
      const int ws = __ffs(__ballot_sync(0xffffffffu, sv == gv && sl == gl)) - 1;
      old = fps_index(gl, L);
      cx = slot[buf][ws].x, cy = slot[buf][ws].y, cz = slot[buf][ws].z;
    }
    if (threadIdx.x == 0) idx[j] = old;
  }
}
static_assert(FPS_CELLS_NW == 32, "the final reduction takes one warp candidate per lane");

// points per lane of a block: the smallest whose block states fit FPS_CELLS_SMEM_MAX
static int fps_cells_spl(int N, size_t *smem) {
  for (int spl = 2; spl <= 16; spl *= 2) {
    const long long nb = ((long long)N + 32 * spl - 1) / (32 * spl);
    const size_t bytes = sizeof(uint32_t) * FPS_CELLS_WORDS * FPS_CELLS_NW * (size_t)((nb + FPS_CELLS_NW - 1) / FPS_CELLS_NW);
    if (bytes <= FPS_CELLS_SMEM_MAX) {
      *smem = bytes;
      return spl;
    }
  }
  return 0;
}

template <int SPL>
static int launch_fps_cells(const float4 *sorted, const float *xyz, int N, int m, float *tmin, int *idx, size_t smem,
                            cudaStream_t st) {
  static int ready[64];  // the opt-in to more than 48 KB of dynamic shared memory: once per device
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (!__atomic_load_n(&ready[dev], __ATOMIC_ACQUIRE)) {
    GF_CUDA(cudaFuncSetAttribute(fps_cells_kernel<SPL>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 (int)FPS_CELLS_SMEM_MAX));
    __atomic_store_n(&ready[dev], 1, __ATOMIC_RELEASE);
  }
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(1, 1, 1);
  cfg.blockDim = dim3(FPS_CELLS_T, 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = st;
  cudaLaunchAttribute attr[1] = {fps_priority()};
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  GF_CUDA(cudaLaunchKernelEx(&cfg, fps_cells_kernel<SPL>, sorted, xyz, N, m, ref_log2_block(N), tmin, idx));
  count_launch();
  return GF_OK;
}

// the running minima, in cell order
static Arena fps_cells_carve(void *workspace, size_t workspace_bytes, int N, float **tmin) {
  Arena ar(workspace, workspace_bytes);
  *tmin = ar.take<float>((size_t)N);
  return ar;
}

size_t fps_cells_workspace_bytes(int N) {
  float *tmin;
  return fps_cells_carve(nullptr, 0, N, &tmin).off;
}

int fps_cells(const float4 *sorted, const float *xyz, int N, int m, void *workspace, size_t workspace_bytes, int *idx,
              cudaStream_t st) {
  GF_CHECK_ARG(N >= 1 && m >= 1, "fps_cells: need N >= 1 and m >= 1 (N=%d m=%d)", N, m);
  float *tmin;
  const Arena ar = fps_cells_carve(workspace, workspace_bytes, N, &tmin);
  if (!ar.ok) return ar.fail("fps_cells");
  size_t smem = 0;
  switch (fps_cells_spl(N, &smem)) {
    case 2: return launch_fps_cells<2>(sorted, xyz, N, m, tmin, idx, smem, st);
    case 4: return launch_fps_cells<4>(sorted, xyz, N, m, tmin, idx, smem, st);
    case 8: return launch_fps_cells<8>(sorted, xyz, N, m, tmin, idx, smem, st);
    case 16: return launch_fps_cells<16>(sorted, xyz, N, m, tmin, idx, smem, st);
  }
  set_error("fps_cells: N=%d does not fit the on-chip block states", N);
  return GF_ERR_INVALID;
}

}  // namespace gf

using namespace gf;

extern "C" size_t gf_fps_workspace_bytes(int B, int N, int m) {
  (void)m;
  if (B <= 0 || N <= 0) return 0;
  if (fps_cluster_capacity(8) >= N) return 0;  // fits an 8-CTA cluster on every device: no scratch at all
  uint2 *slots;
  float *temp;
  return fps_carve(nullptr, 0, B, N, &slots, &temp).off;
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
  int L = ref_log2_block(N);
  const FpsPlan p = plan_fps(N, max_cluster_size());
  if (!p.grid)
    return with_cluster_shape(p.T, p.P, [&](auto T, auto P) {
      return launch_clusters(fps_cluster_kernel<T, P>, T, B, p.ctas, st, xyz, N, m, L, idx);
    });
  uint2 *slots;
  float *temp;
  const Arena ar = fps_carve(workspace, workspace_bytes, B, N, &slots, &temp);
  if (!ar.ok) return ar.fail("furthest_point_sampling");
  return with_grid_p(p.P, [&](auto P) {
    GF_CUDA(cudaMemsetAsync(slots, 0, sizeof(uint2) * 2 * FPS_SLOT_WORDS * (size_t)p.ctas, st));  // tag 0 = unwritten
    void *args[] = {(void *)&xyz, &B, &N, &m, &L, &temp, &idx, &slots};
    GF_CUDA(cudaLaunchCooperativeKernel((const void *)fps_grid_kernel<P>, dim3(p.ctas), dim3(FPS_GRID_T), args, 0, st));
    count_launch();
    return GF_OK;
  });
}

// ---- a ragged batch: scenes b of the flat (offsets[B], 3) array --------------------------------------------------
// Scenes that fit one cluster (N <= max_cs * 512 * 24) go through ONE launch per 32 of them, planned for the largest;
// a larger scene runs the whole-GPU kernel of the single-scene call, after the cluster launches.  The largest scene
// sets the cluster size: at the model's sizes (60k-150k points) a smaller cluster cannot hold it (8 CTAs: 98,304
// points), so a batch with more scenes than co-resident clusters runs them in waves rather than on thinner clusters.
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
  const long long cap = fps_cluster_capacity(max_cluster_size());
  int Nmax = 0, Nbig = 0;
  for (int b = 0; b < B; ++b) {
    const int N = offsets[b + 1] - offsets[b];
    if (N <= cap && N > Nmax) Nmax = N;
    if (N > cap && N > Nbig) Nbig = N;
  }
  if (Nbig > 0) {  // the scenes above the cluster capacity run the whole-GPU kernel, each on the whole workspace
    uint2 *slots;
    float *temp;
    const Arena ar = fps_carve(workspace, workspace_bytes, 1, Nbig, &slots, &temp);
    if (!ar.ok) return ar.fail("furthest_point_sampling_batch");
  }
  if (Nmax > 0) {
    const FpsPlan p = plan_fps(Nmax, max_cluster_size());
    FpsBatchArgs a;
    int n = 0;
    for (int b = 0; b <= B; ++b) {
      const int N = b < B ? offsets[b + 1] - offsets[b] : 0;
      if (b < B && N >= 1 && N <= cap) a.s[n++] = {xyz + (size_t)offsets[b] * 3, idx + (size_t)b * m, N, ref_log2_block(N)};
      if (n == FPS_BATCH_MAX || (b == B && n > 0)) {
        const int rc = with_cluster_shape(p.T, p.P, [&](auto T, auto P) {
          return launch_clusters(fps_cluster_batch_kernel<T, P>, T, n, p.ctas, st, a, m);
        });
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
