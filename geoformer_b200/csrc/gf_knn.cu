// Exact L2 k-nearest-neighbour graph for 3-D points on sm_100a.
//
// Replaces faiss.GpuIndexFlatL2.search as used by model/geoformer/geodesic_utils.py:11-24
// (call sites geoformer.py:172-177, geoformer_fs.py:170-175).  Result contract (SURVEY App. A.4):
// neighbours ordered by (d2, index), d2 = fmaf(dz,dz, fmaf(dx,dx, dy*dy)) in fp32, k-th missing
// neighbour = (-1, +inf).
//
// Two algorithms, identical results:
//   algo 0  uniform-grid search.  Points are counting-sorted into cells of edge h (chosen on the
//           device from the measured cell occupancy, no host round trip); each query walks the
//           cell shells around its own cell and stops as soon as the k-th best distance is
//           provably smaller than the distance to every unvisited cell.  Work per query is
//           O(k) instead of O(N); threads are laid out in cell order so a warp shares its cells.
//   algo 1  brute-force tiled scan (shared-memory tiles, register-resident sorted top-k).  This
//           is the formulation named in BASELINE.json; kept as an independent cross-check.
// 3-D coordinates make this a compare/select problem, not a contraction: no tensor cores.
#include <type_traits>

#include "gf_geodesic.cuh"
#include "gf_knn.cuh"

namespace gf {

constexpr int KNN_MAX_CELLS = 1 << 22;  // dense cell table (2 x 16 MB of int32)
constexpr int KNN_PASS0_CELLS = 1 << 18;
constexpr int KNN_SCAN_BLOCKS = 512;
constexpr int KNN_MAX_DIM = 1024;

// ---- device-side grid description --------------------------------------------------------------
// The control block (KnnCtl: KnnGrid + the scan states) is cleared by ONE cudaMemsetAsync per build; every field is
// laid out so that zero is its initial value.
struct KnnGrid {
  float ox, oy, oz;  // origin = bbox min
  float h, inv_h;
  float slack;  // safety margin of the termination test (absolute length)
  int dx, dy, dz, ncells;
  uint32_t mm[6];             // max over the points of ~ord(v) for x,y,z (= inverted minimum), then of ord(v)
  unsigned long long sum_sq;  // sum over cells of count^2 (occupancy estimate of the coarse pass)
  unsigned done[2];           // last-block-done counters of the two kernels that end with a planning tail
  unsigned pad_[2];
};
struct KnnCtl {
  KnnGrid g;
  unsigned long long scan_state[KNN_SCAN_BLOCKS];  // bit 63 = published, low bits = the block's cell-count sum
};

// pass 0: coarse guess from the bounding-box volume; pass 1: rescale h so that the occupancy seen
// by a point (sum c^2 / N, measured with the pass-0 grid) becomes the target tau.
// Runs in ONE thread, as the tail of the last block of the kernel that produced its inputs.
__device__ void knn_plan(KnnGrid *g, int N, int pass, float tau, int cap) {
  volatile KnnGrid *vg = g;  // the inputs were written by other blocks of the same launch
  float lo[3], ext[3], maxext = 0.f, maxabs = 0.f;
  for (int a = 0; a < 3; ++a) {
    const uint32_t mn = ~vg->mm[a], mx = vg->mm[3 + a];
    bool empty = mn == 0xffffffffu && mx == 0u;
    float l = empty ? 0.f : ord2f(mn), hgh = empty ? 0.f : ord2f(mx);
    lo[a] = l;
    ext[a] = hgh - l;
    maxext = fmaxf(maxext, ext[a]);
    maxabs = fmaxf(maxabs, fmaxf(fabsf(l), fabsf(hgh)));
  }
  if (!(maxext > 0.f)) maxext = 1.f;
  float h;
  if (pass == 0) {
    float vol = 1.f;
    for (int a = 0; a < 3; ++a) vol *= fmaxf(ext[a], 1e-3f * maxext);
    h = cbrtf(vol * tau / (float)(N > 0 ? N : 1));
  } else {
    float occ = (float)((double)vg->sum_sq / (double)(N > 0 ? N : 1));
    float f = sqrtf(tau / fmaxf(occ, 1e-3f));  // surface-like scaling (occupancy ~ h^2)
    f = fminf(fmaxf(f, 0.125f), 4.f);
    h = vg->h * f;
  }
  h = fmaxf(h, maxext * 1e-6f);
  h = fmaxf(h, maxext / (float)KNN_MAX_DIM);
  int d[3];
  for (int it = 0; it < 64; ++it) {
    long long cells = 1;
    for (int a = 0; a < 3; ++a) {
      d[a] = (int)fminf(floorf(ext[a] / h) + 1.f, (float)KNN_MAX_DIM);
      if (d[a] < 1) d[a] = 1;
      cells *= d[a];
    }
    if (cells <= cap) break;
    h *= 1.2599210f;
  }
  g->ox = lo[0], g->oy = lo[1], g->oz = lo[2];
  g->h = h;
  g->inv_h = 1.f / h;
  g->dx = d[0], g->dy = d[1], g->dz = d[2];
  g->ncells = d[0] * d[1] * d[2];
  // cell membership is decided in fp32: a point may sit one rounding error on the wrong side of
  // a face.  The slack below is orders of magnitude above that error and costs < 1 % extra rings.
  g->slack = 1e-3f * h + 4e-6f * maxabs;
}

// true in every thread of the block that finished last (its view of the other blocks' results is ordered
// by the fence / counter pair, as in the CUDA threadFenceReduction sample)
__device__ __forceinline__ bool last_block_done(unsigned *counter) {
  __shared__ bool s_last;
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const unsigned t = atomicAdd(counter, 1u);
    s_last = t == gridDim.x - 1;
    __threadfence();
  }
  __syncthreads();
  return s_last;
}

__device__ __forceinline__ int cell_coord(float v, float o, float inv_h, int dim) {
  float f = floorf((v - o) * inv_h);
  int c = (f >= 0.f) ? (f < (float)dim ? (int)f : dim - 1) : 0;  // NaN -> 0
  return c;
}
__device__ __forceinline__ int cell_of(const KnnGrid &g, float x, float y, float z) {
  int cx = cell_coord(x, g.ox, g.inv_h, g.dx), cy = cell_coord(y, g.oy, g.inv_h, g.dy),
      cz = cell_coord(z, g.oz, g.inv_h, g.dz);
  return (cz * g.dy + cy) * g.dx + cx;
}

// ---- batched build: blockIdx.y = scene, blockIdx.x = block of that scene ------------------------------------------
// Every kernel below reads its scene's descriptor from the parameter struct; gridDim.x blocks work on each scene, so the
// per-scene planning tails ("last block done") and the scan's chaining stay within one scene.
struct KnnBuildDesc {
  const float *xyz;
  KnnCtl *ctl;
  int *coarse_count, *cell_count, *cell_start, *cell_id, *slot, *order, *rank;
  float4 *sorted;
  int N, cap_coarse, cap_fine;
};
struct KnnBuildArgs {
  KnnBuildDesc s[KNN_BATCH_MAX];
  float tau;
};

// build kernel 1 of 5: bounding box (+ tail: coarse grid plan) and the zero fill of both cell tables
__global__ void __launch_bounds__(256) knn_bbox_kernel(const __grid_constant__ KnnBuildArgs ba) {
  const KnnBuildDesc &d = ba.s[blockIdx.y];
  const float *__restrict__ xyz = d.xyz;
  const int N = d.N;
  KnnGrid *g = &d.ctl->g;
  int4 *__restrict__ zero_a = (int4 *)d.coarse_count, *__restrict__ zero_b = (int4 *)d.cell_count;
  const int n4_a = (d.cap_coarse + 3) / 4, n4_b = (d.cap_fine + 4) / 4;
  const int gtid = blockIdx.x * blockDim.x + threadIdx.x, gsz = gridDim.x * blockDim.x;
  const int4 z4 = make_int4(0, 0, 0, 0);
  for (int i = gtid; i < n4_a; i += gsz) zero_a[i] = z4;
  for (int i = gtid; i < n4_b; i += gsz) zero_b[i] = z4;
  uint32_t lo[3] = {0u, 0u, 0u}, hi[3] = {0u, 0u, 0u};  // lo holds the maximum of ~ord = the inverted minimum
  for (int i = gtid; i < N; i += gsz) {
#pragma unroll
    for (int a = 0; a < 3; ++a) {
      float v = __ldg(xyz + (size_t)i * 3 + a);
      if (v == v && fabsf(v) <= 3.0e38f) {  // ignore NaN / inf for the box
        uint32_t o = f2ord(v);
        lo[a] = max(lo[a], ~o);
        hi[a] = max(hi[a], o);
      }
    }
  }
#pragma unroll
  for (int a = 0; a < 3; ++a) {
    uint32_t l = __reduce_max_sync(0xffffffffu, lo[a]);
    uint32_t h = __reduce_max_sync(0xffffffffu, hi[a]);
    if ((threadIdx.x & 31) == 0) {
      if (l) atomicMax(&g->mm[a], l);
      if (h) atomicMax(&g->mm[3 + a], h);
    }
  }
  if (last_block_done(&g->done[0]) && threadIdx.x == 0) knn_plan(g, N, 0, ba.tau, d.cap_coarse);
}

// build kernels 2 and 3: population of every cell.  The coarse pass (fine == 0) counts into the coarse table and also
// accumulates sum c^2 = sum over the points of (2 * slot + 1) from the slots its atomics return, and ends with the plan
// of the final grid; the final pass records every point's cell and slot for the scatter.
__global__ void __launch_bounds__(256) knn_count_kernel(const __grid_constant__ KnnBuildArgs ba, int fine) {
  const KnnBuildDesc &d = ba.s[blockIdx.y];
  const float *__restrict__ xyz = d.xyz;
  const int N = d.N;
  KnnGrid *gp = &d.ctl->g;
  int *__restrict__ cell_count = fine ? d.cell_count : d.coarse_count;
  int *__restrict__ cell_id = fine ? d.cell_id : nullptr;
  int *__restrict__ slot_in_cell = d.slot;
  const KnnGrid g = *gp;
  unsigned long long acc = 0;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < N; i += gridDim.x * blockDim.x) {
    float x = __ldg(xyz + (size_t)i * 3), y = __ldg(xyz + (size_t)i * 3 + 1), z = __ldg(xyz + (size_t)i * 3 + 2);
    int c = cell_of(g, x, y, z);
    int s = atomicAdd(cell_count + c, 1);
    if (cell_id) {
      cell_id[i] = c;
      slot_in_cell[i] = s;
    } else {
      acc += 2ull * (unsigned)s + 1ull;
    }
  }
  if (cell_id) return;
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if ((threadIdx.x & 31) == 0 && acc) atomicAdd(&gp->sum_sq, acc);
  if (last_block_done(&gp->done[1]) && threadIdx.x == 0) knn_plan(gp, N, 1, ba.tau, d.cap_fine);
}

// build kernel 4: exclusive scan of the cell populations in one launch.  Block b of a scene sums its chunk and
// publishes the sum; its carry-in is the sum of the published sums of the scene's blocks before it (blocks are issued
// x-fastest, so they were scheduled earlier and waiting for them cannot deadlock); then it rescans its chunk and
// writes the cell starts.  gridDim.x <= KNN_SCAN_BLOCKS.
__global__ void __launch_bounds__(256) knn_scan_kernel(const __grid_constant__ KnnBuildArgs ba) {
  const KnnBuildDesc &d = ba.s[blockIdx.y];
  KnnCtl *ctl = d.ctl;
  const int *__restrict__ cnt = d.cell_count;
  int *__restrict__ start = d.cell_start;
  const int N = d.N;
  const int n = ctl->g.ncells;
  const int chunk = (((n + (int)gridDim.x - 1) / (int)gridDim.x) + 3) & ~3;
  const int b0 = min(n, (int)blockIdx.x * chunk), b1 = min(n, b0 + chunk);
  __shared__ int ws[8];
  __shared__ int carry;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  int acc = 0;
  for (int i = b0 + threadIdx.x; i < b1; i += 256) acc += cnt[i];
  for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) ws[warp] = acc;
  __syncthreads();
  volatile unsigned long long *state = ctl->scan_state;
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < 8; ++w) t += ws[w];
    state[blockIdx.x] = (1ull << 63) | (unsigned long long)(unsigned)t;
  }
  int pre = 0;
  for (int j = threadIdx.x; j < (int)blockIdx.x; j += 256) {
    unsigned long long v;
    while (!((v = state[j]) >> 63)) __nanosleep(20);
    pre += (int)(unsigned)(v & 0xffffffffull);
  }
  for (int o = 16; o; o >>= 1) pre += __shfl_xor_sync(0xffffffffu, pre, o);
  __syncthreads();  // ws is reused
  if (lane == 0) ws[warp] = pre;
  __syncthreads();
  if (threadIdx.x == 0) {
    int t = 0;
    for (int w = 0; w < 8; ++w) t += ws[w];
    carry = t;
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) start[n] = N;
  __syncthreads();
  for (int t0 = b0; t0 < b1; t0 += 1024) {
    int i0 = t0 + threadIdx.x * 4;
    int c[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) c[e] = (i0 + e < b1) ? cnt[i0 + e] : 0;
    int tsum = c[0] + c[1] + c[2] + c[3];
    int inc = tsum;
    for (int o = 1; o < 32; o <<= 1) {
      int t = __shfl_up_sync(0xffffffffu, inc, o);
      if (lane >= o) inc += t;
    }
    if (lane == 31) ws[warp] = inc;
    __syncthreads();
    int woff = 0;
    for (int w = 0; w < warp; ++w) woff += ws[w];
    int excl = carry + woff + inc - tsum;
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      if (i0 + e < b1) start[i0 + e] = excl;
      excl += c[e];
    }
    __syncthreads();
    if (threadIdx.x == 255) carry = excl;
    __syncthreads();
  }
}

// build kernel 5: the points in cell order, each with its original index
__global__ void __launch_bounds__(256) knn_scatter_kernel(const __grid_constant__ KnnBuildArgs ba) {
  const KnnBuildDesc &d = ba.s[blockIdx.y];
  const float *__restrict__ xyz = d.xyz;
  const int *__restrict__ cell_id = d.cell_id, *__restrict__ slot_in_cell = d.slot, *__restrict__ start = d.cell_start;
  float4 *__restrict__ sorted = d.sorted;
  int *__restrict__ order = d.order, *__restrict__ rank = d.rank;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < d.N; i += gridDim.x * blockDim.x) {
    int pos = start[cell_id[i]] + slot_in_cell[i];
    float x = __ldg(xyz + (size_t)i * 3), y = __ldg(xyz + (size_t)i * 3 + 1), z = __ldg(xyz + (size_t)i * 3 + 2);
    sorted[pos] = make_float4(x, y, z, __int_as_float(i));
    order[pos] = i;  // order[cell-order position] = original index
    rank[i] = pos;   // rank[original index] = cell-order position
  }
}

// ---- register-resident sorted top-k -------------------------------------------------------------
// 64-bit keys (d2 bits << 32 | index): lexicographic (d2, index) order, all keys distinct.
// The list is kept ascending; slots [0, KT-k) are pinned to 0 so that the live part is always the
// last k entries and list[KT-1] is the current k-th best.
__device__ __forceinline__ unsigned long long knn_key(float d2, int index) {
  return ((unsigned long long)__float_as_uint(d2) << 32) | (unsigned)index;
}
template <int KT>
struct TopK {
  unsigned long long key[KT];
  __device__ __forceinline__ void init(int k) {
#pragma unroll
    for (int i = 0; i < KT; ++i) key[i] = (i < KT - k) ? 0ull : ~0ull;
  }
  __device__ __forceinline__ void offer(float d2, int index) { offer_key(knn_key(d2, index)); }
  __device__ __forceinline__ void offer_key(unsigned long long kk) {
    if (kk < key[KT - 1]) {
      // every slot decides for itself (no compare-exchange chain through the moving key): slot i takes its lower
      // neighbour if the new key sorts below that one, the new key if it sorts below the slot's own key, else it
      // keeps what it has; top down, so a slot's lower neighbour is still the old one when it is read
      bool below = true;  // kk < key[KT - 1]
#pragma unroll
      for (int i = KT - 1; i > 0; --i) {
        const bool below_prev = kk < key[i - 1];
        key[i] = below_prev ? key[i - 1] : (below ? kk : key[i]);
        below = below_prev;
      }
      if (below) key[0] = kk;
    }
  }
  __device__ __forceinline__ float kth_d2() const { return __uint_as_float((unsigned)(key[KT - 1] >> 32)); }
  // The row of the propagation's edge table (gf_geodesic.cu: geo_pack_edges_kernel, same rule): neighbour
  // 1 + e of the result as edge e if it may ever be used (sqrt(d2) <= radius, geodesic_utils.py:123,151),
  // else an edge to the sentinel point N; padded with such edges to KP = 1 << slot_bits entries.
  // rank != nullptr: the table lives in CELL ORDER (the caller passes the row of the query's cell-order position and
  // targets are translated through rank[]) with encoded targets (geo_edge_code); else original indices, plain.
  __device__ __forceinline__ void store_edges(int k, float radius, int N, int slot_bits, const int *__restrict__ rank,
                                              int *__restrict__ tgt, float *__restrict__ len) const {
    const int KP = 1 << slot_bits;
    auto code = [&](int t) { return rank ? geo_edge_code((unsigned)__ldg(rank + t)) : t; };
    const int none = geo_edge_none(N, rank != nullptr);
    if (k == KT && KP == KT) {  // the usual case (k a power of two): whole 16-byte stores
#pragma unroll
      for (int e0 = 0; e0 < KT; e0 += 4) {
        int t[4];
        float w[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = e0 + u;
          t[u] = none, w[u] = 0.f;
          if (e + 1 < KT) {
            const unsigned long long kk = key[e + 1];
            const float d = sqrtf(__uint_as_float((unsigned)(kk >> 32)));
            if (kk != ~0ull && d <= radius) t[u] = code((int)(unsigned)(kk & 0xffffffffu)), w[u] = d;
          }
        }
        reinterpret_cast<int4 *>(tgt)[e0 >> 2] = make_int4(t[0], t[1], t[2], t[3]);
        reinterpret_cast<float4 *>(len)[e0 >> 2] = make_float4(w[0], w[1], w[2], w[3]);
      }
      return;
    }
#pragma unroll
    for (int i = 0; i < KT; ++i) {
      const int e = i - (KT - k) - 1;
      if (e >= 0) {
        const unsigned long long kk = key[i];
        const float d = sqrtf(__uint_as_float((unsigned)(kk >> 32)));
        const bool ok = kk != ~0ull && d <= radius;
        tgt[e] = ok ? code((int)(unsigned)(kk & 0xffffffffu)) : none;
        len[e] = ok ? d : 0.f;
      }
    }
    for (int e = k - 1 > 0 ? k - 1 : 0; e < KP; ++e) tgt[e] = none, len[e] = 0.f;
  }
  __device__ __forceinline__ void store(int k, bool do_sqrt, float *__restrict__ dist, long long *__restrict__ i64,
                                        int *__restrict__ i32) const {
#pragma unroll
    for (int i = 0; i < KT; ++i) {
      int j = i - (KT - k);
      if (j >= 0) {
        unsigned long long kk = key[i];
        bool missing = kk == ~0ull;
        float d2 = missing ? __int_as_float(0x7f800000) : __uint_as_float((unsigned)(kk >> 32));
        int id = missing ? -1 : (int)(unsigned)(kk & 0xffffffffu);
        if (dist) dist[j] = do_sqrt ? sqrtf(d2) : d2;
        if (i64) i64[j] = (long long)id;
        if (i32) i32[j] = id;
      }
    }
  }
};

// ---- grid query ---------------------------------------------------------------------------------
// One launch covers the queries of up to KNN_BATCH_MAX scenes: scene i owns the 128-query blocks
// [block0, block0 + ceil(nq / 128)) of the grid, so a block belongs to exactly one scene.
struct KnnQueryDesc {
  const KnnGrid *grid;
  const float4 *sorted;
  const int *start;
  const float *queries;  // nullptr: the scene's own points, in cell order
  float *dist;
  long long *idx64;
  int *idx32;
  KnnEdgeOut eo;
  int nq, block0;
};
struct KnnQueryArgs {
  KnnQueryDesc s[KNN_BATCH_MAX];
  int B, k, do_sqrt;
};
// the block's scene (the last one whose first block is at or before this block) and its arguments under the names
// the query code uses.  PTR is how the pointers are held: `const &` reads them from the parameter space where they are
// used (copies held in registers from the start cost the k <= 16 kernels more spills than plain kernel parameters
// do); `__restrict__` copies them (the k = 64 kernel, 1 block per SM, is faster that way: 0.88 vs 0.91 ms per c2
// graph on a B200).
#define KNN_QUERY_SCENE(a, PTR)                                                                       \
  int sc_ = 0;                                                                                        \
  while (sc_ + 1 < (a).B && (int)blockIdx.x >= (a).s[sc_ + 1].block0) ++sc_;                          \
  const KnnQueryDesc &d = (a).s[sc_];                                                                 \
  const KnnGrid *PTR gp = d.grid;                                                                     \
  const float4 *PTR sorted = d.sorted;                                                                \
  const int *PTR start = d.start;                                                                     \
  const float *PTR queries = d.queries;                                                               \
  float *PTR dist = d.dist;                                                                           \
  long long *PTR idx64 = d.idx64;                                                                     \
  int *PTR idx32 = d.idx32;                                                                           \
  const KnnEdgeOut &eo = d.eo;                                                                        \
  const int nq = d.nq, k = (a).k, do_sqrt = (a).do_sqrt

// the sentinel row N of the edge table (written by the thread of query 0): only edges to N
__device__ __forceinline__ void knn_sentinel_row(const KnnEdgeOut &eo, int nq) {
  const int none = geo_edge_none(nq, eo.rank != nullptr);
  for (int e = 0; e < (1 << eo.slot_bits); ++e)
    eo.tgt[((size_t)nq << eo.slot_bits) + e] = none, eo.len[((size_t)nq << eo.slot_bits) + e] = 0.f;
}

// The bound of the termination test after shell R: the distance from the query to the nearest face of the visited
// block that still has cells behind it (+inf once the whole grid has been visited).  Every unvisited point is at
// least that far away, minus the fp32 slack g.slack.
__device__ __forceinline__ float knn_unvisited_bound(const KnnGrid &g, int cx, int cy, int cz, float qx, float qy,
                                                     float qz, int R) {
  float mfd = __int_as_float(0x7f800000);
  if (cx - R > 0) mfd = fminf(mfd, qx - (g.ox + (float)(cx - R) * g.h));
  if (cx + R + 1 < g.dx) mfd = fminf(mfd, (g.ox + (float)(cx + R + 1) * g.h) - qx);
  if (cy - R > 0) mfd = fminf(mfd, qy - (g.oy + (float)(cy - R) * g.h));
  if (cy + R + 1 < g.dy) mfd = fminf(mfd, (g.oy + (float)(cy + R + 1) * g.h) - qy);
  if (cz - R > 0) mfd = fminf(mfd, qz - (g.oz + (float)(cz - R) * g.h));
  if (cz + R + 1 < g.dz) mfd = fminf(mfd, (g.oz + (float)(cz + R + 1) * g.h) - qz);
  return mfd;
}

// The two macros below are the parts of both query kernels that read the pointers of KNN_QUERY_SCENE: macros, so
// that each kernel keeps holding them as it declares them (a function taking them changes the count-then-collect
// kernels' register allocation).
// query s and the row its results go to: a point of the scene in cell order (queries == nullptr), or queries[s]
#define KNN_QUERY_POINT()                                                                                        \
  do {                                                                                                           \
    if (queries == nullptr) {                                                                                    \
      float4 me = sorted[s];                                                                                     \
      qx = me.x, qy = me.y, qz = me.z;                                                                           \
      row = __float_as_int(me.w);                                                                                \
    } else {                                                                                                     \
      qx = __ldg(queries + (size_t)s * 3), qy = __ldg(queries + (size_t)s * 3 + 1);                              \
      qz = __ldg(queries + (size_t)s * 3 + 2);                                                                   \
      row = s;                                                                                                   \
    }                                                                                                            \
  } while (0)
// the epilogue: the (row, k) results that were asked for; for a self query (nq == N) the propagation's edge rows,
// written straight from the registers, in the cell-order row (= this thread's s) or the original row
#define KNN_QUERY_EPILOGUE(top)                                                                                  \
  do {                                                                                                           \
    if (dist || idx64 || idx32)                                                                                  \
      (top).store(k, do_sqrt != 0, dist ? dist + (size_t)row * k : nullptr,                                      \
                  idx64 ? idx64 + (size_t)row * k : nullptr, idx32 ? idx32 + (size_t)row * k : nullptr);         \
    if (eo.tgt) {                                                                                                \
      const size_t er = (size_t)(eo.rank ? s : row) << eo.slot_bits;                                             \
      (top).store_edges(k, eo.radius, nq, eo.slot_bits, eo.rank, eo.tgt + er, eo.len + er);                      \
    }                                                                                                            \
  } while (0)

// Thread per query, count then collect.  Offering every candidate to the sorted list as it is scanned makes the
// warp run the insertion at almost every candidate: a lane inserts at ~k (1 + ln(n/k)) of its n candidates, and the
// 32 lanes insert at different ones.  Here the first shell (R <= 1: the 27 cells around the query's cell, nine
// contiguous runs of `sorted`) is walked twice instead:
//   count    each candidate's d2 goes to one of KNN_NB bins (a function of d2 that never decreases) in a per-lane
//            histogram in shared memory; nothing is inserted;
//   collect  the second walk recomputes d2 with the same expression and lists the positions of the candidates whose
//            bin is at most b, the smallest bin with at least k candidates at or below it (every bin if the shell
//            has fewer than k);
//   insert   the listed candidates go through the unchanged TopK, ~k + 2 per lane, so most lanes insert together.
// At least k keys have bin <= b and a key of a higher bin is larger than all of them, so the k smallest (d2, index)
// keys of the shell are among the listed ones (keys tied at the threshold are all listed) and TopK orders them as
// before: the result is bit-identical to offering every candidate.  A lane whose list overflows (duplicates,
// lattices) offers every candidate of the shell instead.  Shells R >= 2 (after the unchanged termination test) offer
// every candidate to a top-k that is already exact for the first shell, so few of them insert.
constexpr int KNN_NB = 32;  // bins of d2 over [0, 4 h^2); the last one also takes everything beyond and NaN
constexpr int KNN_MIN_BLOCKS = 7;  // 72 registers for k <= 16, 24 KB of shared memory per block
template <int KT>
__global__ void __launch_bounds__(128, KT <= 16 ? KNN_MIN_BLOCKS : 1)
    knn_grid_query_kernel(const __grid_constant__ KnnQueryArgs a) {
  // counted on the c2 scene: a lane lists ~k + 2 candidates, at most k + 10 (k = 8, 16, 32)
  constexpr int LIST = KT + 16;
  __shared__ unsigned short hist[KNN_NB][128];  // per-lane counts (a shell of more than 65535 points is not binned)
  __shared__ int list[LIST][128];               // per-lane positions in `sorted` of the collected candidates
  KNN_QUERY_SCENE(a, const &);
  const KnnGrid g = *gp;
  const int tid = threadIdx.x;
  const int s = (blockIdx.x - d.block0) * blockDim.x + tid;
  if (s >= nq) return;
  if (eo.tgt && s == 0) knn_sentinel_row(eo, nq);
  float qx, qy, qz;
  int row;
  KNN_QUERY_POINT();
  const int cx = cell_coord(qx, g.ox, g.inv_h, g.dx), cy = cell_coord(qy, g.oy, g.inv_h, g.dy),
            cz = cell_coord(qz, g.oz, g.inv_h, g.dz);
  TopK<KT> top;
  top.init(k);
  auto offer_run = [&](int p, int p1) {
    for (; p + 4 <= p1; p += 4) {  // four candidates in flight: the loads and distances overlap the offers
      const float4 c0 = __ldg(sorted + p), c1 = __ldg(sorted + p + 1), c2 = __ldg(sorted + p + 2),
                   c3 = __ldg(sorted + p + 3);
      const float e0 = sq3(c0.x - qx, c0.y - qy, c0.z - qz), e1 = sq3(c1.x - qx, c1.y - qy, c1.z - qz),
                  e2 = sq3(c2.x - qx, c2.y - qy, c2.z - qz), e3 = sq3(c3.x - qx, c3.y - qy, c3.z - qz);
      top.offer(e0, __float_as_int(c0.w));
      top.offer(e1, __float_as_int(c1.w));
      top.offer(e2, __float_as_int(c2.w));
      top.offer(e3, __float_as_int(c3.w));
    }
    for (; p < p1; ++p) {
      const float4 c = __ldg(sorted + p);
      top.offer(sq3(c.x - qx, c.y - qy, c.z - qz), __float_as_int(c.w));
    }
  };
  // run r (0..8) of the first shell: row (dz, dy) = (r / 3 - 1, r % 3 - 1), cells cx - 1 .. cx + 1 of the row
  auto first_run = [&](int r, int &p0, int &p1) {
    const int z = cz + r / 3 - 1, y = cy + r % 3 - 1;
    p0 = p1 = 0;
    if (z < 0 || z >= g.dz || y < 0 || y >= g.dy) return;
    const int rowbase = (z * g.dy + y) * g.dx;
    p0 = __ldg(start + rowbase + max(cx - 1, 0)), p1 = __ldg(start + rowbase + min(cx + 1, g.dx - 1) + 1);
  };
  const float bin_scale = (float)KNN_NB * 0.25f * g.inv_h * g.inv_h;
  auto bin_of = [&](float d2) {
    const float t = d2 * bin_scale;
    return t < (float)(KNN_NB - 1) ? (int)t : KNN_NB - 1;  // NaN -> the last bin (NaN keys sort above +inf)
  };
  auto shells_done = [&](int R) {
    const float mfd = knn_unvisited_bound(g, cx, cy, cz, qx, qy, qz, R);
    if (mfd == __int_as_float(0x7f800000)) return true;  // the whole grid has been visited
    const float ms = mfd - g.slack;
    return ms > 0.f && top.kth_d2() < ms * ms;
  };

  // first shell, count
#pragma unroll
  for (int j = 0; j < KNN_NB; ++j) hist[j][tid] = 0;
  int ntot = 0;
  for (int r = 0; r < 9; ++r) {
    int p, p1;
    first_run(r, p, p1);
    ntot += p1 - p;
    for (; p + 4 <= p1; p += 4) {
      const float4 c0 = __ldg(sorted + p), c1 = __ldg(sorted + p + 1), c2 = __ldg(sorted + p + 2),
                   c3 = __ldg(sorted + p + 3);
      const int b0 = bin_of(sq3(c0.x - qx, c0.y - qy, c0.z - qz)), b1 = bin_of(sq3(c1.x - qx, c1.y - qy, c1.z - qz)),
                b2 = bin_of(sq3(c2.x - qx, c2.y - qy, c2.z - qz)), b3 = bin_of(sq3(c3.x - qx, c3.y - qy, c3.z - qz));
      ++hist[b0][tid], ++hist[b1][tid], ++hist[b2][tid], ++hist[b3][tid];
    }
    for (; p < p1; ++p) {
      const float4 c = __ldg(sorted + p);
      ++hist[bin_of(sq3(c.x - qx, c.y - qy, c.z - qz))][tid];
    }
  }
  bool listed = false;
  if (ntot <= 0xffff) {
    // threshold: b = the number of bins below KNN_NB - 1 whose cumulative count is still short of k
    int b = 0, cum = 0;
#pragma unroll
    for (int j = 0; j < KNN_NB - 1; ++j) {
      cum += hist[j][tid];
      b += cum < k;
    }
    // collect
    int n = 0;
    for (int r = 0; r < 9; ++r) {
      int p, p1;
      first_run(r, p, p1);
      for (; p < p1; ++p) {
        const float4 c = __ldg(sorted + p);
        if (bin_of(sq3(c.x - qx, c.y - qy, c.z - qz)) <= b) {
          if (n < LIST) list[n][tid] = p;
          ++n;
        }
      }
    }
    // insert
    if (n <= LIST) {
      listed = true;
      for (int i = 0; i < n; ++i) {
        const float4 c = __ldg(sorted + list[i][tid]);
        top.offer(sq3(c.x - qx, c.y - qy, c.z - qz), __float_as_int(c.w));
      }
    }
  }
  if (!listed) {
    for (int r = 0; r < 9; ++r) {
      int p, p1;
      first_run(r, p, p1);
      offer_run(p, p1);
    }
  }

  // shells R >= 2: every candidate is offered
  const int rmax = max(g.dx, max(g.dy, g.dz));
  if (!shells_done(1)) {
    for (int R = 2; R <= rmax; ++R) {
      const int xl = cx - R, xr = cx + R;
      const int side = 2 * R + 1, nrows = side * side;
      for (int ri = 0; ri < nrows; ++ri) {
        const int dz = ri / side - R, dy = ri % side - R;
        const int z = cz + dz, y = cy + dy;
        if (z < 0 || z >= g.dz || y < 0 || y >= g.dy) continue;
        const bool face = dz == -R || dz == R || dy == -R || dy == R;
        const int rowbase = (z * g.dy + y) * g.dx;
        // on a face of the shell the whole x-run belongs to it; otherwise only its two end cells
        const int nseg = face ? 1 : 2;
        for (int sgi = 0; sgi < nseg; ++sgi) {
          int xa, xb;
          if (nseg == 1) {
            xa = max(xl, 0), xb = min(xr, g.dx - 1);
          } else {
            xa = xb = sgi == 0 ? xl : xr;
            if (xa < 0 || xa >= g.dx) continue;
          }
          if (xa > xb) continue;
          offer_run(__ldg(start + rowbase + xa), __ldg(start + rowbase + xb + 1));
        }
      }
      if (shells_done(R)) break;
    }
  }
  KNN_QUERY_EPILOGUE(top);
}

// ---- grid query, warp-synchronous insertion (k = 64) ------------------------------------------------
// Offering every candidate as it is scanned, the 32 lanes of a warp insert at different candidates, so the warp
// executes the insertion network at nearly every candidate.  Here a candidate that beats the lane's current k-th key
// is only PUSHED onto a small per-lane stack in shared memory; the warp runs the insertion network when some lane's
// stack is nearly full, and then every lane with a pending key inserts one (LIFO: the order of insertions does not
// change the final set, keys are distinct; a key that no longer beats the k-th is dropped at the pop).
// Control flow is warp-uniform (votes), every lane walks its own sequence of candidate ranges and never idles
// before its shell is exhausted; the per-shell termination test is unchanged (after draining the stacks).
constexpr int KNN_PEND = 8;  // stack depth; a step pushes at most 4, the network runs while a stack holds > 4
template <int KT>
__global__ void __launch_bounds__(128, 1) knn_grid_query_sync_kernel(const __grid_constant__ KnnQueryArgs a) {
  __shared__ unsigned long long pend[KNN_PEND][128];
  constexpr unsigned FULL = 0xffffffffu;
  KNN_QUERY_SCENE(a, __restrict__);
  const KnnGrid g = *gp;
  const int tid = threadIdx.x;
  const int s = (blockIdx.x - d.block0) * blockDim.x + tid;
  const bool live = s < nq;
  if (eo.tgt && s == 0) knn_sentinel_row(eo, nq);
  float qx = 0.f, qy = 0.f, qz = 0.f;
  int row = 0;
  if (live) KNN_QUERY_POINT();
  const int cx = cell_coord(qx, g.ox, g.inv_h, g.dx), cy = cell_coord(qy, g.oy, g.inv_h, g.dy),
            cz = cell_coord(qz, g.oz, g.inv_h, g.dz);
  TopK<KT> top;
  top.init(k);
  int npend = 0;
  auto insert_round = [&]() {  // every lane with a pending key inserts its newest one
    if (npend > 0) top.offer_key(pend[--npend][tid]);
  };
  const int rmax = max(g.dx, max(g.dy, g.dz));
  bool active = live;
  for (int R = 0; R <= rmax; ++R) {
    if (!__any_sync(FULL, active)) break;
    const int z0 = max(cz - R, 0), z1 = min(cz + R, g.dz - 1);
    const int y0 = max(cy - R, 0), y1 = min(cy + R, g.dy - 1);
    const int xl = cx - R, xr = cx + R;
    // this lane's walk over the candidate ranges of shell R: rows (z, y) of the block; on a face of the shell the
    // whole x-run belongs to it (one range), otherwise only its two end cells (two ranges)
    int z = z0, y = y0, sg = 0, p = 0, p1 = 0;
    bool more = active;
    for (;;) {
      if (more && p >= p1) {
        for (;;) {
          if (z > z1) {
            more = false;
            break;
          }
          const bool face = R == 0 || z == cz - R || z == cz + R || y == cy - R || y == cy + R;
          const int rowbase = (z * g.dy + y) * g.dx;
          int xa, xb;
          bool last;
          if (face)
            xa = max(xl, 0), xb = min(xr, g.dx - 1), last = true;
          else
            xa = xb = sg == 0 ? xl : xr, last = sg == 1;
          if (last) {
            sg = 0;
            if (++y > y1) y = y0, ++z;
          } else {
            sg = 1;
          }
          if (xa < 0 || xb >= g.dx || xa > xb) continue;
          p = __ldg(start + rowbase + xa), p1 = __ldg(start + rowbase + xb + 1);
          if (p < p1) break;
        }
      }
      if (!__any_sync(FULL, more)) break;
      if (more) {  // up to four candidates of this lane's current range
        const int n = min(p1 - p, 4);
        float4 c[4];
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (u < n) c[u] = __ldg(sorted + p + u);
#pragma unroll
        for (int u = 0; u < 4; ++u)
          if (u < n) {
            const float d2 = sq3(c[u].x - qx, c[u].y - qy, c[u].z - qz);
            const unsigned long long kk = knn_key(d2, __float_as_int(c[u].w));
            if (kk < top.key[KT - 1]) pend[npend++][tid] = kk;
          }
        p += 4;
      }
      while (__any_sync(FULL, npend > KNN_PEND - 4)) insert_round();
    }
    while (__any_sync(FULL, npend > 0)) insert_round();
    if (active) {
      const float mfd = knn_unvisited_bound(g, cx, cy, cz, qx, qy, qz, R);
      if (mfd == __int_as_float(0x7f800000)) active = false;  // the whole grid has been visited
      const float ms = mfd - g.slack;
      if (ms > 0.f && top.kth_d2() < ms * ms) active = false;
    }
  }
  if (!live) return;
  KNN_QUERY_EPILOGUE(top);
}

// ---- brute force (algo 1) -----------------------------------------------------------------------
constexpr int BF_TILE = 1024;
template <int KT>
__global__ void __launch_bounds__(128)
    knn_brute_kernel(const float *__restrict__ xyz, int N, const float *__restrict__ queries, int nq, int k,
                     int do_sqrt, float *__restrict__ dist, long long *__restrict__ idx64, int *__restrict__ idx32) {
  __shared__ float sx[BF_TILE], sy[BF_TILE], sz[BF_TILE];
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = q < nq;
  float qx = 0.f, qy = 0.f, qz = 0.f;
  if (live) qx = __ldg(queries + (size_t)q * 3), qy = __ldg(queries + (size_t)q * 3 + 1), qz = __ldg(queries + (size_t)q * 3 + 2);
  TopK<KT> top;
  top.init(k);
  for (int base = 0; base < N; base += BF_TILE) {
    const int tn = min(BF_TILE, N - base);
    __syncthreads();
    for (int t = threadIdx.x; t < tn * 3; t += blockDim.x) {
      float v = __ldg(xyz + (size_t)base * 3 + t);
      int pt = t / 3, ax = t - pt * 3;
      (ax == 0 ? sx : ax == 1 ? sy : sz)[pt] = v;
    }
    __syncthreads();
    if (live) {
#pragma unroll 4
      for (int t = 0; t < tn; ++t) {
        float d2 = sq3(sx[t] - qx, sy[t] - qy, sz[t] - qz);
        top.offer(d2, base + t);
      }
    }
  }
  if (live)
    top.store(k, do_sqrt != 0, dist ? dist + (size_t)q * k : nullptr, idx64 ? idx64 + (size_t)q * k : nullptr,
              idx32 ? idx32 + (size_t)q * k : nullptr);
}

// ---- host orchestration -------------------------------------------------------------------------
// table sizes depend on N only (the workspace is sized before k is known)
static int knn_cap_fine(int N) {
  long long c = 8ll * N;
  if (c < (1 << 18)) c = 1 << 18;
  if (c > KNN_MAX_CELLS) c = KNN_MAX_CELLS;
  return (int)c;
}
static int knn_cap_coarse(int N) {
  int c = N < 4096 ? 4096 : N;
  return c > KNN_PASS0_CELLS ? KNN_PASS0_CELLS : c;
}

// The layout of one scene's grid workspace, for sizing (over a null workspace the Arena only measures) and for the
// build: the control block (a batch uses its ctl_block instead), both cell tables, the per-point arrays.
static Arena knn_carve(void *workspace, size_t workspace_bytes, int N, KnnBuildDesc *d) {
  Arena ar(workspace, workspace_bytes);
  d->N = N;
  d->cap_fine = knn_cap_fine(N), d->cap_coarse = knn_cap_coarse(N);
  d->ctl = ar.take<KnnCtl>(1);
  d->coarse_count = ar.take<int>(d->cap_coarse);
  d->cell_count = ar.take<int>(d->cap_fine + 4);
  d->cell_start = ar.take<int>(d->cap_fine + 4);
  d->cell_id = ar.take<int>(N);
  d->slot = ar.take<int>(N);
  d->order = ar.take<int>(N);
  d->rank = ar.take<int>(N);
  d->sorted = ar.take<float4>(N);
  return ar;
}

size_t knn_grid_workspace_bytes(int N) {
  KnnBuildDesc d;
  return knn_carve(nullptr, 0, N, &d).off + 1024;
}

// the register-resident top-k is sized KT = the power of two >= k (8 .. 64); launch(KT) is called with it as a
// compile-time constant (std::integral_constant)
template <typename F>
static void with_kt(int k, F &&launch) {
  if (k <= 8)
    launch(std::integral_constant<int, 8>());
  else if (k <= 16)
    launch(std::integral_constant<int, 16>());
  else if (k <= 32)
    launch(std::integral_constant<int, 32>());
  else
    launch(std::integral_constant<int, 64>());
}

size_t knn_ctl_block_bytes(int B) { return align256(sizeof(KnnCtl)) * (size_t)(B > 0 ? B : 0); }

// Five launches and one memset for the whole batch (round 1: thirteen launches per scene): bbox + coarse plan |
// coarse count + final plan | final count | scan | scatter.  Nothing returns to the host; grid dimensions are read
// from the device.  A scene gets nb / B blocks of each kernel (at least one, and for the count and scatter kernels no
// more than its points need): one scene keeps the single-scene grids, a batch stays about one wave wide.  How many
// blocks share a scene changes no result: the box and the occupancy are integer reductions, the scan is exact.
int knn_grid_build_batch(const KnnBuildScene *scenes, int B, int k, void *ctl_block, cudaStream_t st,
                         KnnGridBuffers *out) {
  if (B < 1 || B > KNN_BATCH_MAX || (ctl_block == nullptr && B != 1)) {
    set_error("knn: batched build of %d scenes (1..%d, control blocks %s)", B, KNN_BATCH_MAX,
              ctl_block ? "given" : "missing");
    return GF_ERR_INVALID;
  }
  KnnBuildArgs a;
  int maxN = 1;
  for (int b = 0; b < B; ++b) {
    const int N = scenes[b].N;
    KnnBuildDesc &d = a.s[b];
    d.xyz = scenes[b].xyz;
    const bool ok = knn_carve(scenes[b].workspace, scenes[b].workspace_bytes, N, &d).ok;
    if (ctl_block) d.ctl = (KnnCtl *)((char *)ctl_block + align256(sizeof(KnnCtl)) * b);
    if (!ok) {
      set_error("knn: workspace of scene %d too small (%zu bytes given, %zu needed)", b, scenes[b].workspace_bytes,
                knn_grid_workspace_bytes(N));
      return GF_ERR_WORKSPACE;
    }
    maxN = N > maxN ? N : maxN;
    out[b].grid = &d.ctl->g;
    out[b].cell_start = d.cell_start;
    out[b].sorted = d.sorted;
    out[b].order = d.order;
    out[b].rank = d.rank;
  }
  const int nb = num_sms() * 8;
  const int per_scene = nb / B > 1 ? nb / B : 1;
  const int npt = min(per_scene, (maxN + 255) / 256);
  const int nscan = min(per_scene, KNN_SCAN_BLOCKS);
  // target cell occupancy = tau_mul x k.  Measured (c2 / c1, B200): flat between 0.12 and 0.7 for k <= 32 (0.45 kept);
  // at k = 64 smaller cells win (0.2: 0.88 ms vs 1.03 ms per graph).
  const float tau_mul = k > 32 ? 0.2f : 0.45f;
  a.tau = fmaxf(2.f, tau_mul * (float)k);
  GF_CUDA(cudaMemsetAsync(a.s[0].ctl, 0, ctl_block ? knn_ctl_block_bytes(B) : sizeof(KnnCtl), st));
  knn_bbox_kernel<<<dim3(per_scene, B), 256, 0, st>>>(a);
  GF_LAUNCHED();
  knn_count_kernel<<<dim3(npt, B), 256, 0, st>>>(a, 0);
  GF_LAUNCHED();
  knn_count_kernel<<<dim3(npt, B), 256, 0, st>>>(a, 1);
  GF_LAUNCHED();
  knn_scan_kernel<<<dim3(nscan, B), 256, 0, st>>>(a);
  GF_LAUNCHED();
  knn_scatter_kernel<<<dim3(npt, B), 256, 0, st>>>(a);
  GF_LAUNCHED();
  return GF_OK;
}

int knn_grid_build(const float *xyz, int N, int k, void *workspace, size_t workspace_bytes, cudaStream_t st,
                   KnnGridBuffers *out) {
  const KnnBuildScene sc = {xyz, N, workspace, workspace_bytes};
  return knn_grid_build_batch(&sc, 1, k, nullptr, st, out);
}

int knn_grid_query_batch(const KnnQueryJob *jobs, int B, int k, int do_sqrt, cudaStream_t st) {
  if (B < 1 || B > KNN_BATCH_MAX) {
    set_error("knn: batched query of %d scenes (1..%d)", B, KNN_BATCH_MAX);
    return GF_ERR_INVALID;
  }
  KnnQueryArgs a;
  a.B = B, a.k = k, a.do_sqrt = do_sqrt;
  int blocks = 0;
  for (int b = 0; b < B; ++b) {
    const KnnQueryJob &j = jobs[b];
    KnnQueryDesc &d = a.s[b];
    d.grid = (const KnnGrid *)j.grid.grid;
    d.sorted = j.grid.sorted;
    d.start = j.grid.cell_start;
    d.queries = j.queries;
    d.dist = j.dist, d.idx64 = j.idx64, d.idx32 = j.idx32;
    d.eo = {nullptr, nullptr, 0.f, 0, nullptr};
    if (j.edges && j.queries == nullptr) {
      d.eo = *j.edges;
      if (d.eo.rank) d.eo.rank = j.grid.rank;  // any non-null value asks for the cell-order format
    }
    d.nq = j.nq;
    d.block0 = blocks;
    blocks += (j.nq + 127) / 128;
  }
  if (blocks == 0) return GF_OK;
  with_kt(k, [&](auto kt) {
    // Measured (c2, B200): at k <= 32 the count-then-collect kernel; at k = 64, where an insertion is 64
    // compare-exchanges, the warp-synchronous one (10-16 % faster than offering every candidate).
    constexpr int KT = decltype(kt)::value;
    if constexpr (KT > 32)
      knn_grid_query_sync_kernel<KT><<<blocks, 128, 0, st>>>(a);
    else
      knn_grid_query_kernel<KT><<<blocks, 128, 0, st>>>(a);
  });
  GF_LAUNCHED();
  return GF_OK;
}

int knn_grid_query(const KnnGridBuffers &b, const float *queries, int nq, int k, int do_sqrt, float *dist,
                   long long *idx64, int *idx32, cudaStream_t st, const KnnEdgeOut *edges) {
  const KnnQueryJob j = {b, queries, nq, dist, idx64, idx32, edges};
  return knn_grid_query_batch(&j, 1, k, do_sqrt, st);
}

}  // namespace gf

using namespace gf;

extern "C" size_t gf_knn_workspace_bytes(int N, int nq, int k, int algo) {
  (void)nq;
  (void)k;
  if (algo == 1 || N <= 0) return 0;
  return knn_grid_workspace_bytes(N);
}

extern "C" int gf_knn(const float *xyz, int N, const float *queries, int nq, int k, int sqrt_out, float *dist,
                      int64_t *idx64, int32_t *idx32, int algo, void *workspace, size_t workspace_bytes,
                      void *stream) {
  GF_CHECK_ARG(N >= 0 && nq >= 0, "knn: negative size");
  GF_CHECK_ARG(k >= 1 && k <= KNN_MAX_K, "knn: k=%d outside [1,%d]", k, KNN_MAX_K);
  GF_CHECK_ARG(algo == 0 || algo == 1, "knn: unknown algo %d", algo);
  cudaStream_t st = (cudaStream_t)stream;
  if (queries == nullptr) nq = N;
  if (nq == 0) return GF_OK;
  GF_CHECK_ARG(xyz || N == 0, "knn: null xyz");
  if (algo == 1 || N == 0) {
    const float *q = queries ? queries : xyz;
    with_kt(k, [&](auto kt) {
      knn_brute_kernel<decltype(kt)::value>
          <<<(nq + 127) / 128, 128, 0, st>>>(xyz, N, q, nq, k, sqrt_out, dist, (long long *)idx64, idx32);
    });
    GF_LAUNCHED();
    return GF_OK;
  }
  KnnGridBuffers b;
  int rc = knn_grid_build(xyz, N, k, workspace, workspace_bytes, st, &b);
  if (rc) return rc;
  return knn_grid_query(b, queries, nq, k, sqrt_out, dist, (long long *)idx64, idx32, st);
}

// ---- a batch of scenes, each against itself: one build and one query launch for all of them -------------------------
static size_t knn_batch_layout(const int *Ns, int B, size_t *off) {
  size_t o = align256(knn_ctl_block_bytes(B));
  for (int b = 0; b < B; ++b) {
    off[b] = o;
    o += align256(knn_grid_workspace_bytes(Ns[b]));
  }
  return o + 1024;
}

extern "C" size_t gf_knn_batch_workspace_bytes(const int *Ns, int B) {
  if (!Ns || B < 1 || B > KNN_BATCH_MAX) return 0;
  for (int b = 0; b < B; ++b)
    if (Ns[b] < 1) return 0;
  size_t off[KNN_BATCH_MAX];
  return knn_batch_layout(Ns, B, off);
}

extern "C" int gf_knn_batch(const float *const *xyz, const int *Ns, int B, int k, int sqrt_out, float *const *dist,
                            int32_t *const *idx32, void *workspace, size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(xyz && Ns && dist && idx32, "knn_batch: null pointer array");
  GF_CHECK_ARG(B >= 1 && B <= KNN_BATCH_MAX, "knn_batch: B=%d outside [1,%d]", B, KNN_BATCH_MAX);
  GF_CHECK_ARG(k >= 1 && k <= KNN_MAX_K, "knn_batch: k=%d outside [1,%d]", k, KNN_MAX_K);
  for (int b = 0; b < B; ++b) GF_CHECK_ARG(Ns[b] >= 1 && xyz[b], "knn_batch: scene %d: empty or null", b);
  size_t off[KNN_BATCH_MAX];
  const size_t need = knn_batch_layout(Ns, B, off);
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("knn_batch: workspace too small (%zu bytes given, %zu needed)", workspace_bytes, need);
    return GF_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char *w = (char *)workspace;
  KnnBuildScene sc[KNN_BATCH_MAX];
  KnnGridBuffers gb[KNN_BATCH_MAX];
  KnnQueryJob jobs[KNN_BATCH_MAX];
  for (int b = 0; b < B; ++b) sc[b] = {xyz[b], Ns[b], w + off[b], align256(knn_grid_workspace_bytes(Ns[b]))};
  int rc = knn_grid_build_batch(sc, B, k, w, st, gb);
  if (rc) return rc;
  for (int b = 0; b < B; ++b) jobs[b] = {gb[b], nullptr, Ns[b], dist[b], nullptr, idx32[b], nullptr};
  return knn_grid_query_batch(jobs, B, k, sqrt_out, st);
}
