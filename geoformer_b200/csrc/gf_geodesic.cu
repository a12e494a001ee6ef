// Multi-source geodesic propagation over the kNN graph for sm_100a.
//
// Reference: model/geoformer/geodesic_utils.py:91-164 (cal_geodesic_vectorize).  NOT a shortest
// path: it is a level-synchronous, first-visit-wins BFS.  A point receives its distance at the
// first hop level at which it is reached and is never relaxed again; among several parents at
// that level the winner is the first candidate in the reference's candidate order, i.e. the
// parent with the smallest point index, then the smallest neighbour slot (geodesic_utils.py:
// 131-136 keep the first occurrence of each (point, query) pair; the candidate list is built from
// the lexicographically sorted winner list of the previous level, :131-135, :154).
//
// Formulation.  The Q seeds are independent BFS runs over the same graph, so ONE CTA owns ONE seed
// from its first level to its last (persistent CTAs pull seeds from a counter).  Level
// synchronisation is a __syncthreads() -- no grid barrier, no host round trip (the reference
// synchronises the host >= 3 times per level).  Per seed, in shared memory: the visited bitmap, a
// "claimed at this level" bitmap and the compacted frontier queue (point ids).  The seed's own output
// row geo[q][:] doubles as the claim array.  One level:
//   claims   KP/4 lanes expand one frontier point p, each lane fetching four edge targets with one 16-byte
//            load.  An edge to an unvisited t claims it with a fire-and-forget
//            RED.MIN(bits(geo[q][t]), 0x80000000 | p << SB | j): smaller than "unvisited" (-1.0f =
//            0xBF800000), larger than any finished distance (a non-negative float), and ordered exactly
//            like the reference's tie rule (parent index, then slot); plus a fire-and-forget ATOMS.OR on
//            the claimed bitmap.  No atomic return value is ever waited for.
//   resolve  of the PREVIOUS level's winners, started before the claims and finished under them: the key
//            left in a point's row entry IS the reference's winner: decode (p, j), read the edge length and
//            p's finished distance, write geo[q][t] = D[p][j] + geo[q][p] (one fp32 add, as the reference).
//   commit   (after the CTA barrier) every thread owns whole 16-byte pieces of the bitmaps: claimed ->
//            visited, claimed cleared, set bits enumerated into the frontier queue of the next level.
// The claim loop has no bounds or validity branches: lanes past the end of the queue expand the sentinel
// point N, whose edge row holds only edges to N, and bit N of the visited bitmap is always set, so padding
// and filtered edges (radius / missing neighbour, :123 / :151, applied once when the graph is packed) look
// like edges to an already visited point.
// Levels whose frontier does not fit the on-chip queue read its tail from a global overflow area; scenes too
// large for the two bitmaps (N > ~860k) test / claim through the row with returning atomics (MODE 0; MODE 1
// keeps only the visited bitmap on chip).  Optional by-products: the maximum of every row (for the
// epilogues) and, for seed-sharded scenes, the finished row pushed into the peers' matrices over NVLink.
// History of the formulations that were measured and replaced: DESIGN.md section 4.3.
#include <string.h>

#include "gf_geodesic.cuh"
#include "gf_knn.cuh"

namespace gf {

constexpr int GEO_QCAP = 4096;  // frontier entries kept in shared memory (per buffer)
constexpr int GEO_THREADS = 1024;  // threads of the per-scene kernel: one CTA per seed, two per SM
constexpr int GEO_UNROLL = 2;  // frontier points in flight per lane group (x 4 edges per lane)
constexpr int GEO_MAX_PEERS = 15;
constexpr uint32_t GEO_UNVISITED = 0xBF800000u;  // bits of -1.0f
constexpr uint32_t GEO_KEYBIT = 0x80000000u;
constexpr uint32_t GEO_KEYMAX = 0x3F800000u;  // row-claim keys must stay below "unvisited"

struct GeoArgs {
  const int *tgt;   // (N + 1, KP) edge targets; unusable edges and the sentinel row N point to N
  const float *len;  // (N + 1, KP) edge lengths (read only when a winner is resolved)
  int N, Q, max_step;
  int slot_bits;  // KP = 1 << slot_bits
  const int *seeds;
  float *geo;                 // (Q,N)
  int *overflow;              // per CTA: N + 2 frontier entries beyond GEO_QCAP (two stacks, one per end)
  unsigned *seed_counter;     // work distribution
  unsigned long long *stats;  // [0] reached pairs, [1] deepest level (atomicMax)
  float *row_max;             // optional (Q): max of every finished row, a by-product for the mask-head epilogue
  int bitmap_words;           // shared-memory visited bitmap size (0 = test the output row instead)
  // seed-sharded scenes: finished rows are also stored into the other ranks' matrices (NVLink peer memory)
  int n_peers;
  float *peer_geo[GEO_MAX_PEERS];  // row q of this launch goes to peer_geo[r] + q * N
#ifdef GF_TRACE
  long long *trace;   // development only: per-seed start / end
  long long *trace2;  // development only: per-level, per-warp phase timestamps of CTAs 0..3 (streamlined kernel)
#endif
};

__device__ __forceinline__ uint32_t ld_cg_u32(const uint32_t *p) {
  uint32_t v;
  asm volatile("ld.global.cg.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}

// ---- edge packing ---------------------------------------------------------------------------------
// Edge j < k - 1 of point p is neighbour 1 + j of the kNN result if it may ever be used (D <= radius, 0 <= I < N;
// geodesic_utils.py:123,151); column 0 is dropped (:110-111).  Returns whether it is, with its target and length.
template <bool IS64>
__device__ __forceinline__ bool geo_edge_usable(const float *__restrict__ D, const void *__restrict__ I, int N, int k,
                                                float radius, int p, int j, int *t, float *w) {
  const size_t at = (size_t)p * k + 1 + j;
  const long long ti = IS64 ? ((const long long *)I)[at] : (long long)((const int *)I)[at];
  const float wi = __ldg(D + at);
  *t = (int)ti, *w = wi;
  return wi <= radius && ti >= 0 && ti < N;
}

// The table of one scene in the original numbering: tgt[p][j], len[p][j] = the usable edge, else N, 0.
// Row N (the sentinel point used to pad frontier queues) has only edges to N.  KP >= 4 so that a
// lane can fetch four targets with one 16-byte load.
template <bool IS64>
__global__ void geo_pack_edges_kernel(const float *__restrict__ D, const void *__restrict__ I, int N, int k,
                                      float radius, int slot_bits, int enc, int *__restrict__ tgt,
                                      float *__restrict__ len) {
  const int KP = 1 << slot_bits, K = k - 1;
  const long long total = ((long long)N + 1) << slot_bits;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const int p = (int)(e >> slot_bits), j = (int)(e & (KP - 1));
    int to = N, t;
    float wo = 0.f, w;
    if (j < K && p < N && geo_edge_usable<IS64>(D, I, N, k, radius, p, j, &t, &w)) to = t, wo = w;
    tgt[e] = enc ? geo_edge_code((unsigned)to) : to;
    len[e] = wo;
  }
}

// The tables of a batch of scenes in one launch (blockIdx.y = scene), each in the CELL ORDER of its kNN grid with
// encoded targets (the format of the batched kernel): row r holds the edges of point order[r], an edge to t is stored
// as geo_edge_code(rank[t]).  rank / order null: the original numbering (development builds, GF_GEO_ORIGINAL_ORDER).
struct GeoPackScene {
  const float *D;
  const void *I;
  const int *rank, *order;
  int *tgt;
  float *len;
  int N;
};
struct GeoPackArgs {
  GeoPackScene sc[GEO_BATCH_MAX];
  int k, slot_bits;
  float radius;
};
template <bool IS64>
__global__ void __launch_bounds__(256) geo_pack_edges_batch_kernel(const __grid_constant__ GeoPackArgs a) {
  const GeoPackScene &S = a.sc[blockIdx.y];
  const int N = S.N, sb = a.slot_bits, KP = 1 << sb, K = a.k - 1;
  const long long total = ((long long)N + 1) << sb;
  for (long long e = blockIdx.x * (long long)blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const int r = (int)(e >> sb), j = (int)(e & (KP - 1));
    int to = N, t;
    float wo = 0.f, w;
    if (j < K && r < N) {
      const int p = S.order ? __ldg(S.order + r) : r;
      if (geo_edge_usable<IS64>(S.D, S.I, N, a.k, a.radius, p, j, &t, &w)) to = S.rank ? __ldg(S.rank + t) : t, wo = w;
    }
    S.tgt[e] = geo_edge_code((unsigned)to);
    S.len[e] = wo;
  }
}

// ---- frontier storage -------------------------------------------------------------------------------
// Entry i of a frontier: the first qcap live in shared memory, the rest in the CTA's global overflow area
// (both propagation kernels).  Consecutive levels hold disjoint point sets (F_L + F_{L+1} <= N + 1), so ONE buffer
// of N + 2 entries serves both: odd levels grow up from index 0, even levels grow down from the top.
__device__ __forceinline__ size_t ovf_index(int i, int level_parity, int N, int qcap) {
  const size_t j = (size_t)(i - qcap);
  return level_parity ? j : (size_t)N + 1 - j;
}
__device__ __forceinline__ void frontier_put(int *sq, int *ovf, int i, int level_parity, int N, int t) {
  if (i < GEO_QCAP)
    sq[i] = t;
  else
    ovf[ovf_index(i, level_parity, N, GEO_QCAP)] = t;
}

// A row of N floats as 16-byte pieces: `head` floats before the first aligned address, `nvec` float4, then the
// floats from `tail0` on
struct RowSplit {
  size_t head, nvec;
  __device__ __forceinline__ size_t tail0() const { return head + nvec * 4; }
};
__device__ __forceinline__ RowSplit row_split(const float *row, int N) {
  const size_t head = ((16 - ((uintptr_t)row & 15)) & 15) / 4;
  const size_t h = head < (size_t)N ? head : (size_t)N;
  return {h, ((size_t)N - h) / 4};
}

// The maximum over the block of v (unsigned), valid in thread 0.  s_max: THREADS / 32 words of shared memory.
template <int THREADS>
__device__ __forceinline__ uint32_t block_max_u32(uint32_t v, uint32_t *s_max, unsigned tid) {
  const uint32_t wm = __reduce_max_sync(0xffffffffu, v);
  if ((tid & 31u) == 0) s_max[tid >> 5] = wm;
  __syncthreads();
  uint32_t m = 0u;
  if (tid < 32) m = __reduce_max_sync(0xffffffffu, tid < THREADS / 32 ? s_max[tid] : 0u);
  return m;
}

// one candidate edge p --(slot)--> t of the current level (t == N for padding / unusable edges)
// key = 0x80000000 | p << SB | slot, passed in pre-assembled (the shift is shared with the row address)
// MODE 2: visited + claimed bitmaps in shared memory (N <~ 800k); MODE 1: visited bitmap only, the first
// claimant is told by the returning atomic (N <~ 1.7 M); MODE 0: no on-chip state, the row is the visited set.
template <int MODE>
__device__ __forceinline__ void geo_claim(uint32_t key, int t, int N, int level, uint32_t *vis, uint32_t *clm,
                                          uint32_t *rowu, int *nq, int *ovf, int *s_next_n) {
  if (MODE >= 1) {
    const unsigned tw = (unsigned)t >> 5, tb = 1u << (t & 31);
    if (vis[tw] & tb) return;  // visited, padding, or filtered edge
    if (MODE == 2) {
      atomicMin(rowu + t, key);  // RED.MIN: fire and forget
      atomicOr(clm + tw, tb);    // fire and forget too: the next frontier is read off this bitmap after the level
      return;
    } else {
      if (atomicMin(rowu + t, key) != GEO_UNVISITED) return;
    }
  } else {
    if (t >= N || ld_cg_u32(rowu + t) < GEO_KEYBIT) return;
    if (atomicMin(rowu + t, key) != GEO_UNVISITED) return;
  }
  frontier_put(nq, ovf, atomicAdd(s_next_n, 1), level & 1, N, t);  // first claimant: t joins the next frontier
}

template <int MODE>
__device__ __forceinline__ void geo_claim4(uint32_t key, const int4 t, int N, int level, uint32_t *vis, uint32_t *clm,
                                           uint32_t *rowu, int *nq, int *ovf, int *s_next_n) {
  if (MODE == 0) {
    // Without on-chip state both the visited test and the claim are L2 round trips.  The four tests are
    // issued together, then the (returning) claims of the targets that passed, then the queue appends:
    // two round trips per lane and batch instead of up to eight in sequence.
    const int tt[4] = {t.x, t.y, t.z, t.w};
    uint32_t st[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) st[e] = tt[e] < N ? ld_cg_u32(rowu + tt[e]) : 0u;  // 0 = "visited": padding / filtered
    uint32_t old[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) old[e] = st[e] >= GEO_KEYBIT ? atomicMin(rowu + tt[e], key + e) : 0u;
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (old[e] == GEO_UNVISITED) frontier_put(nq, ovf, atomicAdd(s_next_n, 1), level & 1, N, tt[e]);
    return;
  }
  geo_claim<MODE>(key + 0, t.x, N, level, vis, clm, rowu, nq, ovf, s_next_n);
  geo_claim<MODE>(key + 1, t.y, N, level, vis, clm, rowu, nq, ovf, s_next_n);
  geo_claim<MODE>(key + 2, t.z, N, level, vis, clm, rowu, nq, ovf, s_next_n);
  geo_claim<MODE>(key + 3, t.w, N, level, vis, clm, rowu, nq, ovf, s_next_n);
}

template <int MODE>
__global__ void __launch_bounds__(GEO_THREADS, 2048 / GEO_THREADS) geo_seed_bfs_kernel(const GeoArgs a) {
  constexpr bool BITMAP = MODE >= 1;  // a visited bitmap lives in shared memory
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int *q0 = reinterpret_cast<int *>(smem_raw);
  // MODE 2 writes the next frontier only after the level's barrier, so one queue serves both
  int *q1 = MODE == 2 ? q0 : q0 + GEO_QCAP;
  uint32_t *vis = reinterpret_cast<uint32_t *>(q1 + GEO_QCAP);
  uint32_t *clm = vis + a.bitmap_words;
  __shared__ int s_next_n[2], s_seed_q;  // next-frontier counter, by level parity
  __shared__ uint32_t s_rmax[GEO_THREADS / 32];

  const int N = a.N;
  const unsigned sb = (unsigned)a.slot_bits, KP = 1u << sb;
  const unsigned tid = threadIdx.x;
  // a group of KP/4 lanes expands one frontier point: each lane fetches four targets with one 16-byte load
  const unsigned lsb = sb - 2, sub = tid & ((1u << lsb) - 1u);
  const unsigned group = tid >> lsb, ngroups = GEO_THREADS >> lsb;
  const int4 *__restrict__ trow = reinterpret_cast<const int4 *>(a.tgt) + sub;  // + (p << lsb)
  const uint32_t keybase = GEO_KEYBIT | (sub << 2);
  int *ovf = a.overflow + (size_t)blockIdx.x * ((size_t)N + 2);
  unsigned long long reached_total = 0;
  int deepest = 0;

  for (;;) {
    if (tid == 0) s_seed_q = (int)atomicAdd(a.seed_counter, 1u);
    __syncthreads();
    const int q = s_seed_q;
    if (q >= a.Q) break;
    float *row = a.geo + (size_t)q * N;
    uint32_t *rowu = reinterpret_cast<uint32_t *>(row);
#ifdef GF_TRACE
    long long tr_t0 = 0, tr_t1 = 0;
    const unsigned long long tr_r0 = reached_total;
    if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t0));
#endif
    {  // init: row = -1 (geodesic_utils.py:113), visited = claimed = {} (:114), sentinel bit N set
      const RowSplit rs = row_split(row, N);
      float4 *r4 = reinterpret_cast<float4 *>(row + rs.head);
      const float4 m1 = make_float4(-1.f, -1.f, -1.f, -1.f);
      for (size_t i = tid; i < rs.nvec; i += GEO_THREADS) r4[i] = m1;
      if ((size_t)tid < rs.head) row[tid] = -1.f;
      if ((size_t)tid < (size_t)N - rs.tail0()) row[rs.tail0() + tid] = -1.f;
      if (BITMAP)
        for (int i = tid; i < (MODE == 2 ? 2 : 1) * a.bitmap_words; i += GEO_THREADS) vis[i] = 0u;  // vis, clm contiguous
    }
    const int s = a.seeds[q];
    const bool seed_ok = s >= 0 && s < N;  // the reference would raise an index error; the row stays -1
    __syncthreads();
    if (tid == 0) {
      s_next_n[0] = s_next_n[1] = 0;
      if (BITMAP) vis[(unsigned)N >> 5] |= 1u << (N & 31);
    }
    if (tid == 0) q0[0] = s;  // frontier of level 1 = {seed}
    __syncthreads();
    int F = seed_ok ? 1 : 0;
    int *fq = q0, *nq = q1;
    // NOTE the seed is NOT marked visited before level 1: the reference's first expansion has no
    // visited filter (:123), so a seed that appears in its own neighbour row is re-won at level 1.
    int level = 0;
    // Distance of a point won at level `won`: the key left in its row entry is the reference's winner.
    // level 1: the distance is the edge itself (:127); later: edge + parent's distance (:144)
    float rmax = 0.f;  // largest distance this thread wrote into the row (all are >= 0)
    auto resolve_finish = [&](int t, uint32_t key, int won) {
      const unsigned p = (key & 0x7fffffffu) >> sb, j = key & (KP - 1);
      const float w = __ldg(a.len + ((size_t)p << sb) + j);
      const float d = won == 1 ? w : __fadd_rn(w, __uint_as_float(ld_cg_u32(rowu + p)));  // :139
      row[t] = d;
      rmax = fmaxf(rmax, d);
    };
    auto frontier_at = [&](const int *q, int i, int won) {
      return i < GEO_QCAP ? q[i] : ovf[ovf_index(i, won & 1, N, GEO_QCAP)];
    };
    while (F > 0 && level < a.max_step) {
      ++level;
      // The points of this frontier were won at level-1 and still hold their keys.  Their distances are
      // not needed to expand them, only to report them, so the resolve (two dependent L2 accesses) is
      // started here, runs under the claims of pass A, and is finished after it.  (Without the on-chip
      // bitmaps the visited test reads the row, so the row has to be resolved first.)
      int rt = -1;
      uint32_t rkey = 0;
      float rw = 0.f, rpd = 0.f;  // edge length and parent distance of this thread's point to resolve
      bool rissued = false;
      // second step of the resolve: needs the key (an L2 round trip after the level started), so it is issued
      // behind the first batch of edge-row loads and completes under the claims
      auto resolve_issue = [&]() {
        const unsigned p = (rkey & 0x7fffffffu) >> sb, j = rkey & (KP - 1);
        rw = __ldg(a.len + ((size_t)p << sb) + j);
        if (level > 2) rpd = __uint_as_float(ld_cg_u32(rowu + p));
        rissued = true;
      };
      if (level > 1) {
        if (BITMAP) {
          if ((int)tid < F) {
            rt = fq[tid];
            rkey = ld_cg_u32(rowu + rt);
          }
        } else {
          for (int i = tid; i < F; i += GEO_THREADS) {
            const int t = frontier_at(fq, i, level - 1);
            resolve_finish(t, ld_cg_u32(rowu + t), level - 1);
          }
          __syncthreads();
        }
      }
      // ---- pass A: claims ---------------------------------------------------------------------------
      const int Fs = F < GEO_QCAP ? F : GEO_QCAP;  // on-chip part; lanes past the end expand the sentinel point N
      for (int n0 = (int)group; n0 < Fs; n0 += (int)ngroups * GEO_UNROLL) {
        unsigned pl[GEO_UNROLL];  // p << lsb: 32-bit, (N + 1) << sb < 2^30 by the host-side key check
        int4 t[GEO_UNROLL];
#pragma unroll
        for (int u = 0; u < GEO_UNROLL; ++u) {
          const int at = n0 + u * (int)ngroups;
          pl[u] = (unsigned)(at < Fs ? fq[at] : N) << lsb;
        }
#pragma unroll
        for (int u = 0; u < GEO_UNROLL; ++u) t[u] = __ldg(trow + pl[u]);
        if (BITMAP && rt >= 0 && !rissued) resolve_issue();
#pragma unroll
        for (int u = 0; u < GEO_UNROLL; ++u) {
          // slots past the end hold the sentinel (every claim would be rejected): on small frontiers whole
          // warps skip them instead of running four rejected claims per lane
          if (u > 0 && n0 + u * (int)ngroups >= Fs) continue;
          const uint32_t key = keybase | (pl[u] << 2);
          geo_claim4<MODE>(key, t[u], N, level, vis, clm, rowu, nq, ovf, &s_next_n[level & 1]);
        }
      }
      for (int node = GEO_QCAP + (int)group; node < F; node += (int)ngroups) {  // spilled tail (rare)
        const unsigned pl = (unsigned)ovf[ovf_index(node, (level - 1) & 1, N, GEO_QCAP)] << lsb;
        const int4 t = __ldg(trow + pl);
        const uint32_t key = keybase | (pl << 2);
        geo_claim4<MODE>(key, t, N, level, vis, clm, rowu, nq, ovf, &s_next_n[level & 1]);
      }
      if (BITMAP && level > 1) {  // finish the resolve of the points won at level-1
        if (rt >= 0) {
          if (!rissued) resolve_issue();
          const float d = level == 2 ? rw : __fadd_rn(rw, rpd);  // :127 / :139,:144
          row[rt] = d;
          rmax = fmaxf(rmax, d);
        }
        for (int i = tid + GEO_THREADS; i < F; i += GEO_THREADS) {
          const int t = frontier_at(fq, i, level - 1);
          resolve_finish(t, ld_cg_u32(rowu + t), level - 1);
        }
      }
      __syncthreads();
      // ---- commit: the points claimed at this level become visited (:140) and form the next frontier ---
      if (tid == 0) s_next_n[(level + 1) & 1] = 0;  // idle since the previous level's reads; used again after the next barrier
      if (MODE == 2) {
        // Every thread owns whole 16-byte pieces of the bitmaps: claimed -> visited, claimed cleared, and the
        // set bits enumerated into the queue -- no atomics on the bitmaps, one counter atomic per piece.
        if (level == 1 && seed_ok && tid == (((unsigned)s >> 7) & (GEO_THREADS - 1))) {
          // the seed joins the visited set now; if no self edge re-won it, its distance stays 0
          // (a re-won seed holds its key until it is resolved with the other level-1 points)
          if (ld_cg_u32(rowu + s) == GEO_UNVISITED) row[s] = 0.f;
          vis[(unsigned)s >> 5] |= 1u << (s & 31);
        }
        uint4 *clm4 = reinterpret_cast<uint4 *>(clm), *vis4 = reinterpret_cast<uint4 *>(vis);
        const int n4 = a.bitmap_words >> 2;  // bitmap_words is a multiple of 4
        for (int i = tid; i < n4; i += GEO_THREADS) {
          const uint4 c = clm4[i];
          if ((c.x | c.y | c.z | c.w) == 0u) continue;
          clm4[i] = make_uint4(0u, 0u, 0u, 0u);
          uint4 v = vis4[i];
          v.x |= c.x, v.y |= c.y, v.z |= c.z, v.w |= c.w;
          vis4[i] = v;
          const int cnt = __popc(c.x) + __popc(c.y) + __popc(c.z) + __popc(c.w);
          int at = atomicAdd(&s_next_n[level & 1], cnt);
          const unsigned long long lo = ((unsigned long long)c.y << 32) | c.x, hi = ((unsigned long long)c.w << 32) | c.z;
          if (at + cnt <= GEO_QCAP) {  // the usual case: the whole piece lands in the on-chip queue
            for (unsigned long long m = lo; m; m &= m - 1) nq[at++] = i * 128 + __ffsll((long long)m) - 1;
            for (unsigned long long m = hi; m; m &= m - 1) nq[at++] = i * 128 + 64 + __ffsll((long long)m) - 1;
          } else {
            for (unsigned long long m = lo; m; m &= m - 1)
              frontier_put(nq, ovf, at++, level & 1, N, i * 128 + __ffsll((long long)m) - 1);
            for (unsigned long long m = hi; m; m &= m - 1)
              frontier_put(nq, ovf, at++, level & 1, N, i * 128 + 64 + __ffsll((long long)m) - 1);
          }
        }
        __syncthreads();
      }
      const int nextF = s_next_n[level & 1];
      if (MODE == 1) {
        for (int i = tid; i < nextF; i += GEO_THREADS) {
          const int t = frontier_at(nq, i, level);
          atomicOr(vis + ((unsigned)t >> 5), 1u << (t & 31));
        }
      }
      if (MODE != 2 && tid == 0 && level == 1) {
        if (ld_cg_u32(rowu + s) == GEO_UNVISITED) row[s] = 0.f;
        if (BITMAP) atomicOr(vis + ((unsigned)s >> 5), 1u << (s & 31));
      }
      if (nextF > 0) deepest = level > deepest ? level : deepest;
      reached_total += (unsigned long long)nextF;
      F = nextF;
      int *tq = fq;
      fq = nq;
      nq = tq;
      if (MODE != 2) __syncthreads();
    }
    // the points won at the last executed level still hold their keys
    if (level >= 1) {
      for (int i = tid; i < F; i += GEO_THREADS) {
        const int t = frontier_at(fq, i, level);
        resolve_finish(t, ld_cg_u32(rowu + t), level);
      }
    }
    if (level == 0 && seed_ok && tid == 0) row[s] = 0.f;  // max_step <= 0: only the seed entry (:118)
    if (a.row_max) {
      // max over the row = max over what was written (the seed's 0 included), or -1 for a row that stayed empty;
      // distances are non-negative, so their bit patterns order like unsigned integers
      const uint32_t m = block_max_u32<GEO_THREADS>(__float_as_uint(rmax), s_rmax, tid);
      if (tid == 0) a.row_max[q] = seed_ok ? __uint_as_float(m) : -1.f;
    }
    if (a.n_peers > 0) {
      // The row is final: push it into every peer's matrix now, while other CTAs are still propagating --
      // the exchange of a seed-sharded scene rides under the compute instead of following it as a
      // collective.  Same row index on every rank => same 16-byte alignment; stores over NVLink are posted.
      __syncthreads();
      const RowSplit rs = row_split(row, N);
      const float4 *s4 = reinterpret_cast<const float4 *>(row + rs.head);
      for (size_t i = tid; i < rs.nvec; i += GEO_THREADS) {
        const float4 v = __ldcg(s4 + i);
        for (int r = 0; r < a.n_peers; ++r)
          __stcs(reinterpret_cast<float4 *>(a.peer_geo[r] + (size_t)q * N + rs.head) + i, v);
      }
      if ((size_t)tid < rs.head)
        for (int r = 0; r < a.n_peers; ++r) a.peer_geo[r][(size_t)q * N + tid] = __ldcg(row + tid);
      if ((size_t)tid < (size_t)N - rs.tail0())
        for (int r = 0; r < a.n_peers; ++r) a.peer_geo[r][(size_t)q * N + rs.tail0() + tid] = __ldcg(row + rs.tail0() + tid);
    }
#ifdef GF_TRACE
    __syncthreads();
    if (tid == 0 && q < 1024 && a.trace) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t1));
      a.trace[q * 4 + 0] = tr_t0, a.trace[q * 4 + 1] = tr_t1;
      a.trace[q * 4 + 2] = (long long)(reached_total - tr_r0), a.trace[q * 4 + 3] = ((long long)blockIdx.x << 32) | level;
    }
#endif
  }
  if (tid == 0) {
    if (reached_total) atomicAdd(a.stats, reached_total);
    atomicMax(a.stats + 1, (unsigned long long)deepest);
  }
}

// ---- the batched kernel (scenes whose two bitmaps fit on chip: N <~ 860k) -------------------------------------
// Same algorithm as geo_seed_bfs_kernel<2> (level-synchronous first-visit BFS per seed, RED.MIN claim keys that
// reproduce the reference's tie rule, frontier read off a claimed bitmap), restated around what the round-2
// profiles showed: a per-seed run is a CHAIN OF DEPENDENT MEMORY LATENCIES (per level: queue -> edge row ->
// visited words -> barrier -> bitmap scan -> queue, plus the loads that turn a winning key into a distance), the
// SM issues at ~40 % with all its thread slots taken, 30 % of the warp time is spent at the barrier behind the
// slowest warp of a level, and that warp is slow because its loads miss L2: with the claims made in the seed's own
// output row, 296 concurrently live rows of 4N bytes (118 MB at N = 100k) are filled with -1 and then hit at random.
//  * CELL ORDER.  The propagation runs on the kNN grid's cell-order numbering of the points (rank / order of
//    gf_knn.cu: points of a cell are consecutive, cells of a row adjacent), so a frontier -- a shell in space --
//    touches a few dense runs of ids instead of N/8 random sectors.
//  * CLAIMS AND DISTANCES IN PER-CTA SCRATCH, not in the output row, and in ONE array indexed by cell-order id.
//    An entry is either a claim key of the running seed (< 2^31: order << slot_bits | slot, RED.MIN) or, with the
//    top bit set, a distance (the sign bit is spare, distances are >= 0) -- of the running seed if the point is
//    visited, else a leftover of an earlier seed of this CTA, which loses against every key.  So nothing is ever
//    reset: the array is cleared once per CTA, a resolve replaces the key by the distance, the final pass only
//    reads.  A seed touches ~13 % of the sectors (its reach) and they stay in L2.
//  * THE OUTPUT ROW IS WRITTEN ONCE, streaming, after the seed's last level: out[i] = visited(rank[i]) ?
//    distance(rank[i]) : -1 (geodesic_utils.py:113 fills with -1 first; same result).  No read-modify-write of the
//    402 MB/s-per-scene matrix, DRAM traffic = the matrix itself.
//  * The tie rule needs the ORIGINAL parent index (smallest parent index, then slot, wins): keys are
//    order[p] << slot_bits | slot; resolving maps the winner back through rank[].
//  * Work items are the (scene, seed) pairs of a whole BATCH of scenes (the reference's call is batched:
//    cal_geodesic_vectorize loops over the scenes of a batch, geodesic_utils.py:98), pulled from one counter by
//    persistent CTAs: one launch, one tail per batch instead of one per scene.
//  * Edge targets are stored ENCODED (geo_edge_code, gf_geodesic.cuh) so that the visited test is four instructions.
constexpr int GEO_MAXB = 32;  // scenes per launch (descriptors travel in the kernel parameters)
constexpr uint32_t GEO_UNCLAIMED = 0xFFFFFFFFu;
constexpr uint32_t GEO_DISTANCE = 0x80000000u;  // entries >= this are distances (or never touched), below: claim keys

struct GeoScene {
  const int *tgt;             // (N + 1, KP) encoded edge targets, rows and targets in cell order
  const float *len;           // (N + 1, KP) edge lengths
  const int *rank, *order;    // cell-order position of an original index and back; both null = identity
  const int *seeds;           // (Q) original indices
  float *geo;                 // (Q, N), original order
  float *row_max;             // optional (Q)
  unsigned long long *stats;  // optional: [0] reached pairs, [1] deepest level (device)
  int N, Q, item0, bitmap_words;
};
struct GeoBatchArgs {
  GeoScene sc[GEO_MAXB];
  int B, total_items, max_step, slot_bits, qcap;
  int *overflow;    // per CTA: ovf_stride frontier entries beyond the on-chip queue
  uint32_t *claim;  // per CTA: arr_stride entries: winning key (< 2^31) | 0x80000000 + distance bits
  size_t ovf_stride, arr_stride;
  unsigned *item_counter;
#ifdef GF_TRACE
  long long *trace, *trace2;
#endif
};

// The claims of four ENCODED edge targets (geo_edge_code, gf_geodesic.cuh).  The four visited words are fetched first
// (independent loads), then tested.
__device__ __forceinline__ void geo_claim4_enc(uint32_t key, const int4 t, uint32_t vis_s, uint32_t clm_s,
                                               unsigned char *claimb) {
  const unsigned tt[4] = {(unsigned)t.x, (unsigned)t.y, (unsigned)t.z, (unsigned)t.w};
  uint32_t w[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) asm("ld.shared.u32 %0, [%1];" : "=r"(w[e]) : "r"(vis_s + geo_edge_word_offset(tt[e])));
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    const uint32_t bit = __funnelshift_l(0u, 1u, tt[e]);  // 1 << (t & 31)
    if (!(w[e] & bit)) {
      // both fire and forget (RED.MIN, ATOMS.OR without a destination)
      asm volatile("red.relaxed.gpu.global.min.u32 [%0], %1;" ::"l"(claimb + geo_edge_entry_offset(tt[e])), "r"(key + e)
                   : "memory");
      asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(clm_s + geo_edge_word_offset(tt[e])), "r"(bit) : "memory");
    }
  }
}

template <int THREADS>
__global__ void __launch_bounds__(THREADS, 2048 / THREADS) geo_bfs_batch_kernel(const GeoBatchArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  int *fq = reinterpret_cast<int *>(smem_raw);  // the frontier queue (rebuilt by every commit), a.qcap entries
  uint32_t *vis = reinterpret_cast<uint32_t *>(fq + a.qcap);
  __shared__ int s_next_n[2], s_item;  // next-frontier counter, by level parity
  __shared__ uint32_t s_rmax[THREADS / 32];

  const int QC = a.qcap;
  const unsigned sb = (unsigned)a.slot_bits, KP = 1u << sb;
  const unsigned tid = threadIdx.x;
  const unsigned lsb = sb - 2, sub = tid & ((1u << lsb) - 1u);
  const unsigned group = tid >> lsb, ngroups = THREADS >> lsb;
  const uint32_t keysub = sub << 2;
  int *ovf = a.overflow + (size_t)blockIdx.x * a.ovf_stride;
  uint32_t *claim = a.claim + (size_t)blockIdx.x * a.arr_stride;
  {  // once per CTA: no entry may look like a claim key; afterwards every key is replaced by a distance when resolved
    uint4 *c4 = reinterpret_cast<uint4 *>(claim);
    const uint4 ff = make_uint4(GEO_UNCLAIMED, GEO_UNCLAIMED, GEO_UNCLAIMED, GEO_UNCLAIMED);
    for (size_t i = tid; i < a.arr_stride / 4; i += THREADS) c4[i] = ff;
  }
  // opaque copies: without them ptxas re-derives these addresses (S2R of the CTA's shared window, constant-bank
  // loads, 64-bit multiply-adds) inside every claim instead of spending a register on them
  uint32_t vis_s = (uint32_t)__cvta_generic_to_shared(vis), fq_s = (uint32_t)__cvta_generic_to_shared(fq);
  asm volatile("mov.u32 %0, %0;" : "+r"(vis_s));
  asm volatile("mov.u32 %0, %0;" : "+r"(fq_s));
  asm volatile("mov.u64 %0, %0;" : "+l"(claim));
  uint32_t cnt0_s = (uint32_t)__cvta_generic_to_shared(s_next_n);
  asm volatile("mov.u32 %0, %0;" : "+r"(cnt0_s));
  unsigned char *claimb = reinterpret_cast<unsigned char *>(claim);
  auto fq_at = [&](int i) {
    int v;
    asm volatile("ld.shared.s32 %0, [%1];" : "=r"(v) : "r"(fq_s + 4u * (unsigned)i) : "memory");
    return v;
  };

  for (;;) {
    if (tid == 0) s_item = (int)atomicAdd(a.item_counter, 1u);
    __syncthreads();
    const int item = s_item;
    if (item >= a.total_items) break;
    int b = 0;
    while (b + 1 < a.B && a.sc[b + 1].item0 <= item) ++b;
    const GeoScene &S = a.sc[b];
    const int q = item - S.item0, N = S.N, words = S.bitmap_words;
    const int *__restrict__ rank = S.rank, *__restrict__ order = S.order;
    auto frontier = [&](int i, int parity) { return i < QC ? fq_at(i) : ovf[ovf_index(i, parity, N, QC)]; };
    uint32_t clm_s = vis_s + 4u * (uint32_t)words;
    asm volatile("mov.u32 %0, %0;" : "+r"(clm_s));
    const int4 *__restrict__ trow = reinterpret_cast<const int4 *>(S.tgt) + sub;  // + (p << lsb)
#ifdef GF_TRACE
    long long tr_t0 = 0, tr_t1 = 0;
    if (tid == 0) asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t0));
#endif
    {  // visited = claimed = {} (geodesic_utils.py:114)
      uint4 *b4 = reinterpret_cast<uint4 *>(vis);
      for (int i = tid; i < words / 2; i += THREADS) b4[i] = make_uint4(0u, 0u, 0u, 0u);  // vis, clm contiguous
    }
    const int so = S.seeds[q];
    const bool seed_ok = so >= 0 && so < N;  // the reference would raise an index error; the row stays -1
    const int s = seed_ok ? (rank ? __ldg(rank + so) : so) : 0;
    __syncthreads();
    if (tid == 0) {
      s_next_n[0] = s_next_n[1] = 0;
      vis[(unsigned)N >> 5] |= 1u << (N & 31);  // the sentinel point N is "visited"
      fq[0] = s;                                // frontier of level 1 = {seed}
    }
    __syncthreads();
    int F = seed_ok ? 1 : 0;
    // NOTE the seed is NOT marked visited before level 1: the reference's first expansion has no
    // visited filter (:123), so a seed that appears in its own neighbour row is re-won at level 1.
    int level = 0;
    unsigned long long reached = 0;
    float rmax = 0.f;  // largest distance of this seed seen by this thread (all are >= 0)
    // distance of a point won at level `won`: the key left in its claim entry is the reference's winner.
    // level 1: the distance is the edge itself (:127); later: edge + parent's distance (:139,:144)
    auto resolve = [&](int t, int won) {
      const uint32_t key = ld_cg_u32(claim + t);
      const unsigned po = key >> sb, j = key & (KP - 1);
      const unsigned p = rank ? (unsigned)__ldg(rank + po) : po;
      const float w = __ldg(S.len + ((size_t)p << sb) + j);
      const float d = won == 1 ? w : __fadd_rn(w, __uint_as_float(ld_cg_u32(claim + p) & 0x7FFFFFFFu));
      claim[t] = __float_as_uint(d) | GEO_DISTANCE;
      rmax = fmaxf(rmax, d);
    };
#ifdef GF_TRACE
#define GF_TR(slot)                                                                                              \
  do {                                                                                                           \
    if (a.trace2 && blockIdx.x < 4 && item < 4096 && level <= 40 && (tid & 31u) == 0 && tid < 1024)              \
      a.trace2[((((size_t)blockIdx.x * 41 + level) * 32 + (tid >> 5)) * 8) + (slot)] = clock64();                 \
  } while (0)
#else
#define GF_TR(slot) \
  do {              \
  } while (0)
#endif
    while (F > 0 && level < a.max_step) {
      ++level;
      GF_TR(0);
      // first stage of this thread's own resolves: the keys of its first two frontier points (final since the barrier)
      int rt[2] = {-1, -1};
      uint32_t rkey[2] = {0u, 0u};
      if (level > 1) {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          const int i = (int)tid + u * THREADS;
          if (i < F) {
            rt[u] = frontier(i, (level - 1) & 1);
            rkey[u] = ld_cg_u32(claim + rt[u]);
          }
        }
      }
      // ---- claims: KP/4 lanes per frontier point ------------------------------------------------------------
      const int Fs = F < QC ? F : QC;
      for (int n0 = (int)group; n0 < Fs; n0 += (int)ngroups) {
        const int p = fq_at(n0);
        const unsigned po = order ? (unsigned)__ldg(order + p) : (unsigned)p;
        const int4 t = __ldg(trow + ((unsigned)p << lsb));
        geo_claim4_enc((po << sb) | keysub, t, vis_s, clm_s, claimb);
      }
      for (int node = QC + (int)group; node < F; node += (int)ngroups) {  // spilled tail (rare)
        const int p = ovf[ovf_index(node, (level - 1) & 1, N, QC)];
        const unsigned po = order ? (unsigned)__ldg(order + p) : (unsigned)p;
        geo_claim4_enc((po << sb) | keysub, __ldg(trow + ((unsigned)p << lsb)), vis_s, clm_s, claimb);
      }
      GF_TR(1);
      // ---- the frontier's own distances (its points were won at level-1 and still hold their keys) ----------
      if (level > 1) {
        // second stage: the two dependent round trips (rank of the winning parent, then its edge length and
        // distance) of both points are in flight together
        unsigned rp[2] = {0u, 0u};
        float rw[2] = {0.f, 0.f}, rpd[2] = {0.f, 0.f};
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if (rt[u] >= 0) {
            const unsigned po = rkey[u] >> sb;
            rp[u] = rank ? (unsigned)__ldg(rank + po) : po;
          }
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if (rt[u] >= 0) {
            rw[u] = __ldg(S.len + ((size_t)rp[u] << sb) + (rkey[u] & (KP - 1)));
            if (level > 2) rpd[u] = __uint_as_float(ld_cg_u32(claim + rp[u]) & 0x7FFFFFFFu);
          }
        for (int i = (int)tid + 2 * THREADS; i < F; i += THREADS) resolve(frontier(i, (level - 1) & 1), level - 1);
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if (rt[u] >= 0) {
            const float d = level == 2 ? rw[u] : __fadd_rn(rw[u], rpd[u]);
            claim[rt[u]] = __float_as_uint(d) | GEO_DISTANCE;
            rmax = fmaxf(rmax, d);
          }
      }
      GF_TR(2);
      __syncthreads();
      GF_TR(3);
      // ---- commit: the points claimed at this level become visited (:140) and form the next frontier -------
      if (tid == 0) s_next_n[(level + 1) & 1] = 0;  // idle since the previous level's reads; used after the next barrier
      if (level == 1 && seed_ok && tid == (((unsigned)s >> 5) & (THREADS - 1))) {  // the owner of the seed's word
        // the seed joins the visited set now; if no self edge re-won it, its distance stays 0
        // (a re-won seed holds its key until it is resolved with the other level-1 points)
        if (ld_cg_u32(claim + s) >= GEO_DISTANCE) claim[s] = GEO_DISTANCE;  // no key: distance 0
        vis[(unsigned)s >> 5] |= 1u << (s & 31);
      }
      {
        // Every thread owns single 32-bit words of the bitmaps, consecutive words to consecutive threads: claimed ->
        // visited, claimed cleared, one counter atomic per non-empty word, the set bits enumerated into the queue.
        // In cell order the claimed bits come in dense runs (a frontier is a shell in space: two short runs per row
        // of cells): with 16-byte pieces a run fell to one lane looping 50+ times while the CTA waited at the
        // barrier, and the rows of a shell to a few warps; word by word a run spreads over neighbouring lanes and the
        // shell over all warps.
        // All shared accesses go through the opaque 32-bit window addresses: left to itself ptxas re-derives the
        // generic addresses (S2R of the CTA's window, constant-bank loads) for every word, 18 instructions per test.
        const uint32_t cnt_s = cnt0_s + 4u * (uint32_t)(level & 1);
        const int par = level & 1;
        const uint32_t jend = clm_s + 4u * (uint32_t)words, v_off = 4u * (uint32_t)words;
        for (uint32_t ja = clm_s + 4u * tid; ja < jend; ja += 4u * THREADS) {
          uint32_t c;
          asm volatile("ld.shared.u32 %0, [%1];" : "=r"(c) : "r"(ja) : "memory");
          if (c == 0u) continue;
          asm volatile("st.shared.u32 [%0], %1;" ::"r"(ja), "r"(0u) : "memory");
          asm volatile("red.shared.or.b32 [%0], %1;" ::"r"(ja - v_off), "r"(c) : "memory");  // this thread owns the word
          const int n = __popc(c);
          int at;
          asm volatile("atom.shared.add.u32 %0, [%1], %2;" : "=r"(at) : "r"(cnt_s), "r"(n) : "memory");
          const int base = (int)((ja - clm_s) << 3);  // 32 * word index
          if (at + n <= QC) {  // the usual case: all of the word's points land in the on-chip queue
            uint32_t wa = fq_s + 4u * (uint32_t)at;
            do {  // highest bit first: one FLO per point (the order inside the frontier is immaterial)
              uint32_t bpos;
              asm("bfind.u32 %0, %1;" : "=r"(bpos) : "r"(c));
              asm volatile("st.shared.u32 [%0], %1;" ::"r"(wa), "r"(base + (int)bpos) : "memory");
              wa += 4u;
              c ^= 1u << bpos;
            } while (c);
          } else {
            for (uint32_t m = c; m; m &= m - 1) {
              const int t = base + __ffs((int)m) - 1;
              if (at < QC)
                fq[at] = t;
              else
                ovf[ovf_index(at, par, N, QC)] = t;
              ++at;
            }
          }
        }
      }
      GF_TR(4);
      __syncthreads();
      GF_TR(5);
      const int nextF = s_next_n[level & 1];
#ifdef GF_TRACE
      if (a.trace2 && blockIdx.x < 4 && item < 4096 && level <= 40 && tid == 0)
        a.trace2[((((size_t)blockIdx.x * 41 + level) * 32) * 8) + 6] = F, a.trace2[((((size_t)blockIdx.x * 41 + level) * 32) * 8) + 7] = nextF;
#endif
      reached += (unsigned long long)nextF;
      F = nextF;
    }
    // the points won at the last executed level still hold their keys
    if (level >= 1)
      for (int i = tid; i < F; i += THREADS) resolve(frontier(i, level & 1), level);
    if (level == 0 && seed_ok && tid == 0) {  // max_step <= 0: only the seed entry (:118)
      claim[s] = GEO_DISTANCE;  // distance 0
      vis[(unsigned)s >> 5] |= 1u << (s & 31);
    }
    __syncthreads();  // every reached point is in the visited bitmap and its entry holds its distance
    {  // ---- the output row, written once: out[i] = visited(rank[i]) ? distance(rank[i]) : -1 (:113) ------------
      float *row = S.geo + (size_t)q * N;
      auto value = [&](int r) {
        uint32_t w;
        asm("ld.shared.u32 %0, [%1];" : "=r"(w) : "r"(vis_s + geo_word_offset((unsigned)r)));
        return (w >> (r & 31)) & 1u ? __uint_as_float(__ldcg(claim + r) & 0x7FFFFFFFu) : -1.f;
      };
      if ((((uintptr_t)row) & 15) == 0) {
        const int nvec = N >> 2;
        const int4 *__restrict__ rank4 = reinterpret_cast<const int4 *>(rank);
        for (int i = tid; i < nvec; i += THREADS) {
          const int4 r = rank ? __ldg(rank4 + i) : make_int4(4 * i, 4 * i + 1, 4 * i + 2, 4 * i + 3);
          __stcs(reinterpret_cast<float4 *>(row) + i, make_float4(value(r.x), value(r.y), value(r.z), value(r.w)));
        }
        for (int i = nvec * 4 + (int)tid; i < N; i += THREADS) row[i] = value(rank ? __ldg(rank + i) : i);
      } else {
        for (int i = tid; i < N; i += THREADS) row[i] = value(rank ? __ldg(rank + i) : i);
      }
    }
    if (S.row_max) {
      // max over the row = max over what was written (the seed's 0 included), or -1 for a row that stayed empty;
      // distances are non-negative, so their bit patterns order like unsigned integers
      const uint32_t m = block_max_u32<THREADS>(__float_as_uint(rmax), s_rmax, tid);
      if (tid == 0) S.row_max[q] = seed_ok ? __uint_as_float(m) : -1.f;
    }
    if (tid == 0 && S.stats) {
      if (reached) atomicAdd(S.stats, reached);
      // the deepest level that won anything: the last level's frontier is empty exactly when the loop ended on F == 0
      const int deepest = (level > 0 && F == 0) ? level - 1 : level;
      atomicMax(S.stats + 1, (unsigned long long)(reached ? deepest : 0));
    }
#ifdef GF_TRACE
    __syncthreads();
    if (tid == 0 && item < 1024 && a.trace) {
      asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(tr_t1));
      a.trace[item * 4 + 0] = tr_t0, a.trace[item * 4 + 1] = tr_t1;
      a.trace[item * 4 + 2] = (long long)reached, a.trace[item * 4 + 3] = ((long long)blockIdx.x << 32) | level;
    }
#endif
  }
}

static int ceil_log2(int v) {
  int b = 0;
  while ((1 << b) < v) ++b;
  return b;
}
// edge rows are padded to KP = 2^slot_bits >= 4 entries (four targets per 16-byte load)
static int geo_slot_bits(int k) {
  const int sb = ceil_log2(k - 1 > 1 ? k - 1 : 1);
  return sb < 2 ? 2 : sb;
}

// ---- planning ---------------------------------------------------------------------------------------------
static int geo_bitmap_words(int N) { return ((N + 1 + 127) / 128) * 4; }  // + the sentinel point N; whole 16-byte pieces

// plan of the per-scene kernel (big scenes, seed-sharded scenes)
struct GeoPlan {
  int grid, bitmap_words, mode;
  size_t smem;
};

// identical for sizing and launching: 227 KB of shared memory usable per SM on sm_100 (1 KB reserved per CTA)
static void plan_geo(int N, int Q, GeoPlan *p) {
  const int words = geo_bitmap_words(N);
  auto bytes_of = [&](int mode) {
    return sizeof(int) * (size_t)(mode == 2 ? 1 : 2) * GEO_QCAP + sizeof(uint32_t) * (size_t)mode * words;
  };
  // both bitmaps must fit for mode 2; otherwise mode 0 (two CTAs per SM) measured slightly faster at 1 M
  // points and 512 seeds than mode 1 (157 KB of shared memory: one CTA per SM).  With no more seeds than SMs (a
  // rank's block of a seed-sharded scene) one CTA per SM loses nothing and the visited test stays on chip: mode 1.
  int m = 2;
  if (bytes_of(2) > (size_t)226 * 1024) m = Q <= num_sms() ? 1 : 0;
  if (m == 1 && bytes_of(1) > (size_t)226 * 1024) m = 0;
  const size_t bytes = bytes_of(m);
  int fit = (int)((size_t)(227 * 1024) / (bytes + 1024));
  if (fit < 1) fit = 1;
  const int cap = 2048 / GEO_THREADS;
  p->bitmap_words = m > 0 ? words : 0;
  p->smem = bytes;
  p->mode = m;
  int grid = num_sms() * (fit < cap ? fit : cap);
  if (grid > Q) grid = Q;
  p->grid = grid < 1 ? 1 : grid;
}

// plan of the batched kernel
struct GeoBatchPlan {
  int threads, per_sm, grid, qcap, words;
  size_t smem, ovf_stride, arr_stride;
};
// bytes of per-CTA scratch (frontier overflow + claim keys + distances: 12 bytes per point and CTA) a launch may
// reserve before the number of CTAs is cut below what the SMs could hold (never below one per SM)
constexpr size_t GEO_SCRATCH_BUDGET = (size_t)768 << 20;

// true when the scene can run in the batched kernel (both bitmaps + a queue fit one CTA's shared memory)
static bool geo_batchable(int maxN) {
  return sizeof(int) * 1024 + 2 * sizeof(uint32_t) * (size_t)geo_bitmap_words(maxN) <= (size_t)226 * 1024;
}

static void plan_batch(int maxN, long long items, GeoBatchPlan *p) {
  const int sms = num_sms();
  p->words = geo_bitmap_words(maxN);
  // One scene's worth of seeds cannot fill the thread slots anyway and a launch lasts as long as its slowest
  // seed: 1024 threads per seed.  A batch is throughput work: more, smaller CTAs per SM (see the kernel's header).
  const int threads = items <= 2ll * sms ? 1024 : 512;
  const int cap = 2048 / threads;
  int best_fit = 0, best_q = 0;
  for (int qcap = 4096; qcap >= 1024 && qcap >= threads; qcap >>= 1) {
    const size_t bytes = sizeof(int) * (size_t)qcap + 2 * sizeof(uint32_t) * (size_t)p->words;
    if (bytes > (size_t)226 * 1024) continue;
    int fit = (int)((size_t)(227 * 1024) / (bytes + 1024));
    if (fit > cap) fit = cap;
    if (fit > best_fit) best_fit = fit, best_q = qcap;  // the largest queue that reaches the most CTAs per SM
  }
  if (best_fit < 1) best_fit = 1, best_q = 1024;
  p->threads = threads;
  p->per_sm = best_fit;
  p->qcap = best_q;
  p->smem = sizeof(int) * (size_t)best_q + 2 * sizeof(uint32_t) * (size_t)p->words;
  p->ovf_stride = (size_t)maxN + 2;
  p->arr_stride = ((size_t)maxN + 1 + 3) & ~(size_t)3;  // claim keys / distances per CTA, whole 16-byte pieces
  long long grid = (long long)sms * best_fit;
  const long long ovf_cap = (long long)(GEO_SCRATCH_BUDGET / (sizeof(int) * (p->ovf_stride + p->arr_stride)));
  if (grid > ovf_cap) grid = ovf_cap > sms ? ovf_cap : sms;
  if (grid > items) grid = items;
  p->grid = (int)(grid < 1 ? 1 : grid);
}

// ---- workspace layouts, each stated once in a carve function that sizes it (over a null workspace) and hands it out
// Control block of a launch, cleared by one memset: the counter the CTAs pull seeds from, and the statistics
// (accumulated with atomics, a line apart from the counter)
struct GeoCtl {
  unsigned counter;
  alignas(128) unsigned long long stats[2];  // reached pairs, deepest level
};

// scratch of one batched launch: per CTA the frontier overflow and the claim array, then the control block
struct GeoBatchScratch {
  int *overflow;
  uint32_t *claim;
  GeoCtl *ctl;
};
static Arena geo_batch_carve(void *scratch, size_t scratch_bytes, const GeoBatchPlan &p, GeoBatchScratch *s) {
  Arena a(scratch, scratch_bytes);
  s->overflow = a.take<int>(p.ovf_stride * (size_t)p.grid);
  s->claim = a.take<uint32_t>(p.arr_stride * (size_t)p.grid);
  s->ctl = a.take<GeoCtl>(1);
  return a;
}
size_t geodesic_batch_scratch_bytes(int maxN, long long items) {
  GeoBatchPlan p;
  plan_batch(maxN, items, &p);
  GeoBatchScratch s;
  return geo_batch_carve(nullptr, 0, p, &s).off;
}

void geo_edges_carve(Arena &a, int N, int k, GeoEdges *e) {
  e->slot_bits = geo_slot_bits(k);
  e->tgt = a.take<int>(((size_t)N + 1) << e->slot_bits);
  e->len = a.take<float>(((size_t)N + 1) << e->slot_bits);
}

// workspace of the single-scene entry points: the packed edge table (+ sentinel row), then the scratch of the kernel
// that runs, sized for either: the per-scene kernel's (big scenes; seed-sharded scenes of any size) frontier overflow
// and control block, or for a batchable scene the scratch of a batched launch, if that is larger
struct GeoBuffers {
  GeoEdges e;
  int *overflow;  // the per-scene kernel's scratch ...
  GeoCtl *ctl;
  void *rest;  // ... or a batched launch's, at the same address
  size_t rest_bytes;
};
static Arena geo_carve(void *workspace, size_t workspace_bytes, int N, int k, int Q, GeoBuffers *b) {
  Arena a(workspace, workspace_bytes);
  geo_edges_carve(a, N, k, &b->e);
  b->rest = a.ok ? (void *)(a.base + a.off) : nullptr;
  b->rest_bytes = a.ok ? a.size - a.off : 0;
  GeoPlan pl;
  plan_geo(N, Q, &pl);
  Arena r(b->rest, b->rest_bytes);
  b->overflow = r.take<int>(((size_t)N + 2) * (size_t)pl.grid);
  b->ctl = r.take<GeoCtl>(1);
  const size_t batch = geo_batchable(N) ? geodesic_batch_scratch_bytes(N, Q) : 0;
  (void)a.take<char>(batch > r.off ? batch : r.off);
  return a;
}

size_t geodesic_workspace_bytes(int N, int k, int Q) {
  GeoBuffers b;
  return geo_carve(nullptr, 0, N, k, Q, &b).off;
}

int geodesic_edge_buffers(void *workspace, size_t workspace_bytes, int N, int k, int Q, GeoEdges *e, int *enc) {
  GeoBuffers b;
  const Arena a = geo_carve(workspace, workspace_bytes, N, k, Q, &b);
  if (!a.ok) return a.fail("geodesic");
  *e = b.e;
  *enc = geo_batchable(N) ? 1 : 0;
  return GF_OK;
}
int geodesic_edge_format(int N) { return geo_batchable(N) ? 1 : 0; }

// the opt-in to more than 48 KB of dynamic shared memory is a per-function, per-device attribute: set it once
// to the most any plan can ask for instead of before every launch (several host threads launch concurrently)
template <typename K>
static int geo_kernel_ready(K kernel, int *done) {
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) dev = 0;
  if (!__atomic_load_n(&done[dev], __ATOMIC_ACQUIRE)) {
    GF_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 226 * 1024));
    __atomic_store_n(&done[dev], 1, __ATOMIC_RELEASE);
  }
  return GF_OK;
}

#ifdef GF_TRACE
static long long *g_trace = nullptr, *g_trace2 = nullptr;
static const size_t kTrace2N = (size_t)4 * 41 * 32 * 8;
static void trace_dump(int items, cudaStream_t st) {
  static int calls = 0;
  if (++calls != 3) return;
  static long long h[4 * 1024];
  cudaStreamSynchronize(st);
  cudaMemcpy(h, g_trace, sizeof(h), cudaMemcpyDeviceToHost);
  long long t0 = h[0];
  for (int q = 0; q < items && q < 1024; ++q) t0 = h[q * 4] < t0 ? h[q * 4] : t0;
  for (int q = 0; q < items && q < 1024; ++q)
    fprintf(stderr, "TRACE seed %4d cta %3lld start_us=%8.2f dur_us=%8.2f reached=%7lld levels=%3lld\n", q,
            h[q * 4 + 3] >> 32, (h[q * 4] - t0) * 1e-3, (h[q * 4 + 1] - h[q * 4]) * 1e-3, h[q * 4 + 2],
            h[q * 4 + 3] & 0xffffffffll);
  // per level of CTAs 0..3 (their first seed): phase boundaries in cycles relative to the level's start, as
  // the minimum / maximum over the warps: claims done | resolve done | past barrier 1 | commit done | past barrier 2
  static long long h2[4 * 41 * 32 * 8];
  cudaMemcpy(h2, g_trace2, sizeof(h2), cudaMemcpyDeviceToHost);
  for (int c = 0; c < 4; ++c)
    for (int lv = 1; lv <= 40; ++lv) {
      const long long *b = h2 + (((size_t)c * 41 + lv) * 32) * 8;
      if (!b[0]) continue;
      long long t00 = b[0];
      for (int w = 0; w < 32; ++w)
        if (b[w * 8] && b[w * 8] < t00) t00 = b[w * 8];
      fprintf(stderr, "TRACE2 cta %d level %2d F=%5lld next=%5lld |", c, lv, b[6], b[7]);
      for (int sl = 0; sl < 6; ++sl) {
        long long mn = 1ll << 60, mx = 0;
        for (int w = 0; w < 32; ++w) {
          const long long v = b[w * 8 + sl] - t00;
          if (b[w * 8 + sl] == 0 || (sl >= 6)) continue;
          mn = v < mn ? v : mn, mx = v > mx ? v : mx;
        }
        fprintf(stderr, " %6lld..%-6lld", mn, mx);
      }
      fprintf(stderr, "\n");
    }
}
#endif

// One launch over the (scene, seed) items of up to GEO_MAXB scenes whose edge tables are already packed
// (encoded targets).  scratch: geodesic_batch_scratch_bytes(max N, total seeds).
int geodesic_batch_launch(const GeoSceneDesc *scenes, int B, int k, int max_step, void *scratch, size_t scratch_bytes,
                          cudaStream_t st) {
  if (B < 1 || B > GEO_MAXB) {
    set_error("geodesic: %d scenes in a batched launch, 1..%d supported", B, GEO_MAXB);
    return GF_ERR_INVALID;
  }
  GeoBatchArgs ga;
  memset(&ga, 0, sizeof(ga));
  int maxN = 0;
  long long items = 0;
  const int slot_bits = geo_slot_bits(k);
  for (int b = 0; b < B; ++b) {
    const GeoSceneDesc &d = scenes[b];
    if ((((unsigned long long)d.N + 1) << slot_bits) >= 0x80000000ull) {
      set_error("geodesic: N=%d with k=%d does not fit the 31-bit claim key", d.N, k);
      return GF_ERR_INVALID;
    }
    GeoScene &s = ga.sc[b];
    s.tgt = d.tgt, s.len = d.len, s.seeds = d.seeds, s.geo = d.geo, s.row_max = d.row_max;
    s.rank = d.rank, s.order = d.order;
    if ((d.rank == nullptr) != (d.order == nullptr)) {
      set_error("geodesic: scene %d: rank and order must be given together", b);
      return GF_ERR_INVALID;
    }
    s.stats = (unsigned long long *)d.stats;
    s.N = d.N, s.Q = d.Q, s.item0 = (int)items, s.bitmap_words = geo_bitmap_words(d.N);
    items += d.Q;
    maxN = d.N > maxN ? d.N : maxN;
  }
  if (items == 0) return GF_OK;
  if (!geo_batchable(maxN) || items > 0x7fffffffll) {
    set_error("geodesic: a scene of %d points does not fit the batched kernel", maxN);
    return GF_ERR_INVALID;
  }
  GeoBatchPlan p;
  plan_batch(maxN, items, &p);
  GeoBatchScratch sc;
  const Arena a = geo_batch_carve(scratch, scratch_bytes, p, &sc);
  if (!a.ok) return a.fail("geodesic: scratch");
  ga.overflow = sc.overflow, ga.claim = sc.claim, ga.item_counter = &sc.ctl->counter;
  ga.ovf_stride = p.ovf_stride, ga.arr_stride = p.arr_stride;
  ga.B = B, ga.total_items = (int)items, ga.max_step = max_step, ga.slot_bits = slot_bits, ga.qcap = p.qcap;
  GF_CUDA(cudaMemsetAsync(sc.ctl, 0, sizeof(GeoCtl), st));
#ifdef GF_TRACE
  if (!g_trace) cudaMalloc(&g_trace, 8 * 4 * 1024), cudaMalloc(&g_trace2, kTrace2N * 8);
  cudaMemsetAsync(g_trace, 0, 8 * 4 * 1024, st);
  cudaMemsetAsync(g_trace2, 0, kTrace2N * 8, st);
  ga.trace = g_trace, ga.trace2 = g_trace2;
#endif
  stage_mark(ST_GEO_READY, st);
  int rc = GF_OK;
#define GF_GEO_BATCH(T)                                            \
  do {                                                             \
    static int done[64] = {0};                                     \
    rc = geo_kernel_ready(geo_bfs_batch_kernel<T>, done);          \
    if (rc) return rc;                                             \
    geo_bfs_batch_kernel<T><<<p.grid, T, p.smem, st>>>(ga);        \
  } while (0)
  if (p.threads == 512)
    GF_GEO_BATCH(512);
  else
    GF_GEO_BATCH(1024);
#undef GF_GEO_BATCH
  GF_LAUNCHED();
#ifdef GF_TRACE
  trace_dump((int)items, st);
#endif
  stage_mark(ST_GEO_DONE, st);
  return GF_OK;
}

// One scene.  D == nullptr: the edge table in the workspace has already been written (by the kNN query kernel of
// the fused hot path, gf_knn.cu TopK::store_edges, in the format geodesic_edge_buffers reported) -- no packing pass.
int geodesic_run(const float *D, const void *I, int is64, int N, int k, const int *seeds, int Q, float radius,
                 int max_step, float *geo, int64_t *stats_out, void *workspace, size_t workspace_bytes,
                 cudaStream_t st, float *const *peer_rows, int n_peers, float *row_max, const int *rank,
                 const int *order) {
  if (n_peers < 0 || n_peers > GEO_MAX_PEERS || (n_peers > 0 && !peer_rows)) {
    set_error("geodesic: %d peers given, at most %d supported", n_peers, GEO_MAX_PEERS);
    return GF_ERR_INVALID;
  }
  const int slot_bits = geo_slot_bits(k);
  if ((((unsigned long long)N + 1) << slot_bits) >= GEO_KEYMAX) {
    set_error("geodesic: N=%d with k=%d does not fit the 30-bit claim key (N << %d must be < 2^30)", N, k, slot_bits);
    return GF_ERR_INVALID;
  }
  GeoBuffers b;
  const Arena a = geo_carve(workspace, workspace_bytes, N, k, Q, &b);
  if (!a.ok) return a.fail("geodesic");
  // also the format of an already packed edge table (seed-sharded scenes always run the per-scene kernel)
  const bool batched = geo_batchable(N) && n_peers == 0;
  if (D != nullptr) {
    const long long total = ((long long)N + 1) << slot_bits;
    long long blocks = (total + 255) / 256;
    const long long cap = (long long)num_sms() * 16;
    const int grid = (int)(blocks < cap ? (blocks > 0 ? blocks : 1) : cap);
    if (is64)
      geo_pack_edges_kernel<true><<<grid, 256, 0, st>>>(D, I, N, k, radius, slot_bits, batched ? 1 : 0, b.e.tgt, b.e.len);
    else
      geo_pack_edges_kernel<false><<<grid, 256, 0, st>>>(D, I, N, k, radius, slot_bits, batched ? 1 : 0, b.e.tgt, b.e.len);
    GF_LAUNCHED();
  }
  if (batched) {
    // the stats slot of the launch's control block (cleared by the launch's memset)
    GeoBatchPlan p;
    plan_batch(N, Q, &p);
    GeoBatchScratch sc;
    geo_batch_carve(b.rest, b.rest_bytes, p, &sc);
    unsigned long long *stats = sc.ctl->stats;
    GeoSceneDesc d;
    d.tgt = b.e.tgt, d.len = b.e.len, d.seeds = seeds, d.geo = geo, d.row_max = row_max;
    d.rank = D == nullptr ? rank : nullptr, d.order = D == nullptr ? order : nullptr;  // a packed foreign graph: identity
    d.stats = stats_out ? (int64_t *)stats : nullptr;
    d.N = N, d.Q = Q;
    int rc = geodesic_batch_launch(&d, 1, k, max_step, b.rest, b.rest_bytes, st);
    if (rc) return rc;
    if (stats_out) GF_CUDA(cudaMemcpyAsync(stats_out, stats, 16, cudaMemcpyDeviceToDevice, st));
    return GF_OK;
  }
  GeoPlan p;
  plan_geo(N, Q, &p);
  unsigned long long *stats = b.ctl->stats;
  GF_CUDA(cudaMemsetAsync(b.ctl, 0, sizeof(GeoCtl), st));
  stage_mark(ST_GEO_READY, st);
  GeoArgs ga;
  ga.tgt = b.e.tgt, ga.len = b.e.len, ga.N = N, ga.Q = Q, ga.max_step = max_step, ga.slot_bits = slot_bits;
  ga.seeds = seeds, ga.geo = geo, ga.overflow = b.overflow, ga.seed_counter = &b.ctl->counter, ga.stats = stats;
  ga.bitmap_words = p.bitmap_words;
  ga.row_max = row_max;
  ga.n_peers = n_peers;
  for (int r = 0; r < GEO_MAX_PEERS; ++r) ga.peer_geo[r] = r < n_peers ? peer_rows[r] : nullptr;
  for (int r = 0; r < n_peers; ++r)
    if (!peer_rows[r] || (((uintptr_t)peer_rows[r] ^ (uintptr_t)geo) & 15)) {
      set_error("geodesic: peer matrix %d is null or not aligned like the local one", r);
      return GF_ERR_INVALID;
    }
#ifdef GF_TRACE
  ga.trace = nullptr, ga.trace2 = nullptr;
#endif
  int rc = GF_OK;
#define GF_GEO_LAUNCH(M)                                                  \
  do {                                                                    \
    static int done[64] = {0};                                            \
    rc = geo_kernel_ready(geo_seed_bfs_kernel<M>, done);                  \
    if (rc) return rc;                                                    \
    geo_seed_bfs_kernel<M><<<p.grid, GEO_THREADS, p.smem, st>>>(ga);      \
  } while (0)
  if (p.mode == 2)
    GF_GEO_LAUNCH(2);
  else if (p.mode == 1)
    GF_GEO_LAUNCH(1);
  else
    GF_GEO_LAUNCH(0);
#undef GF_GEO_LAUNCH
  GF_LAUNCHED();
  stage_mark(ST_GEO_DONE, st);
  if (stats_out) GF_CUDA(cudaMemcpyAsync(stats_out, stats, 16, cudaMemcpyDeviceToDevice, st));
  return GF_OK;
}

}  // namespace gf

using namespace gf;

extern "C" size_t gf_geodesic_workspace_bytes(int N, int k, int Q) {
  if (N <= 0 || Q <= 0) return 0;
  return geodesic_workspace_bytes(N, k, Q);
}

extern "C" int gf_geodesic(const float *knn_dist, const void *knn_idx, int idx_is_i64, int N, int k, const int *seeds,
                           int Q, float radius, int max_step, float *geo, int64_t *stats, float *row_max,
                           void *workspace, size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(N >= 0 && Q >= 0, "geodesic: negative size");
  GF_CHECK_ARG(k >= 1 && k <= 256, "geodesic: k=%d outside [1,256]", k);
  if (N == 0 || Q == 0) return GF_OK;
  GF_CHECK_ARG(knn_dist && knn_idx && seeds && geo, "geodesic: null pointer");
  return geodesic_run(knn_dist, knn_idx, idx_is_i64, N, k, seeds, Q, radius, max_step, geo, stats, workspace,
                      workspace_bytes, (cudaStream_t)stream, nullptr, 0, row_max);
}

extern "C" int gf_geodesic_scatter(const float *knn_dist, const void *knn_idx, int idx_is_i64, int N, int k,
                                   const int *seeds, int Q, float radius, int max_step, float *geo,
                                   float *const *peer_geo, int n_peers, int64_t *stats, void *workspace,
                                   size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(N >= 0 && Q >= 0, "geodesic: negative size");
  GF_CHECK_ARG(k >= 1 && k <= 256, "geodesic: k=%d outside [1,256]", k);
  if (N == 0 || Q == 0) return GF_OK;
  GF_CHECK_ARG(knn_dist && knn_idx && seeds && geo, "geodesic: null pointer");
  return geodesic_run(knn_dist, knn_idx, idx_is_i64, N, k, seeds, Q, radius, max_step, geo, stats, workspace,
                      workspace_bytes, (cudaStream_t)stream, peer_geo, n_peers);
}

// ---- a batch of scenes over the caller's kNN graphs -----------------------------------------------------------------
namespace gf {
static_assert(KNN_BATCH_MAX == GEO_BATCH_MAX, "one batched call builds the grids of all its scenes at once");
// The workspace of a batch over given graphs: per scene the workspace of its kNN grid (only its cell-order numbering is
// used) and its edge table; then the control blocks of the batched build, the scratch of the batched propagation and
// the statistics of every scene
struct GraphBatchLayout {
  Span knn[GEO_BATCH_MAX];
  GeoEdges edges[GEO_BATCH_MAX];
  void *knn_ctl;
  Span scratch;
  int64_t *stats;
};
static Arena graph_batch_carve(void *workspace, size_t workspace_bytes, const int *Ns, int B, int Q, int k,
                               GraphBatchLayout *l) {
  Arena a(workspace, workspace_bytes);
  int maxN = 1;
  for (int b = 0; b < B; ++b) {
    l->knn[b] = a.span(knn_grid_workspace_bytes(Ns[b]));
    geo_edges_carve(a, Ns[b], k, &l->edges[b]);
    maxN = Ns[b] > maxN ? Ns[b] : maxN;
  }
  l->knn_ctl = a.take<char>(knn_ctl_block_bytes(B));
  l->scratch = a.span(geodesic_batch_scratch_bytes(maxN, (long long)Q * B));
  l->stats = a.take<int64_t>(2 * (size_t)B);
  return a;
}
}  // namespace gf

extern "C" size_t gf_geodesic_batch_workspace_bytes(const int *Ns, int B, int Q, int k) {
  if (!Ns || B <= 0 || B > GEO_BATCH_MAX || Q <= 0 || k <= 0 || k > 256) return 0;
  for (int b = 0; b < B; ++b)
    if (Ns[b] <= 0) return 0;
  GraphBatchLayout l;
  return graph_batch_carve(nullptr, 0, Ns, B, Q, k, &l).off;
}

extern "C" int gf_geodesic_batch(const float *const *xyz, const float *const *knn_dist, const void *const *knn_idx,
                                 int idx_is_i64, const int *Ns, int B, int k, const int *const *seeds, int Q,
                                 float radius, int max_step, float *const *geo, float *const *row_max, int64_t *stats,
                                 void *workspace, size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(xyz && knn_dist && knn_idx && Ns && seeds && geo, "geodesic_batch: null pointer array");
  GF_CHECK_ARG(B >= 1 && B <= GEO_BATCH_MAX, "geodesic_batch: B=%d outside [1,%d]", B, GEO_BATCH_MAX);
  GF_CHECK_ARG(Q >= 1 && (long long)Q * B <= 0x7fffffffll, "geodesic_batch: Q=%d outside [1, 2^31 / B]", Q);
  GF_CHECK_ARG(k >= 1 && k <= 256, "geodesic_batch: k=%d outside [1,256]", k);
  GF_CHECK_ARG(idx_is_i64 == 0 || idx_is_i64 == 1, "geodesic_batch: idx_is_i64=%d is not 0 or 1", idx_is_i64);
  for (int b = 0; b < B; ++b) {
    GF_CHECK_ARG(Ns[b] >= 1 && xyz[b] && knn_dist[b] && knn_idx[b] && seeds[b] && geo[b],
                 "geodesic_batch: scene %d: empty or null", b);
    GF_CHECK_ARG(geodesic_edge_format(Ns[b]) == 1,
                 "geodesic_batch: scene %d has %d points, beyond the on-chip bitmaps of the batched kernel "
                 "(use gf_geodesic per scene)", b, Ns[b]);
  }
  GraphBatchLayout w;
  const Arena ar = graph_batch_carve(workspace, workspace_bytes, Ns, B, Q, k, &w);
  if (!ar.ok) return ar.fail("geodesic_batch");
  cudaStream_t st = (cudaStream_t)stream;
  int64_t *d_stats = stats ? w.stats : nullptr;
  if (d_stats) GF_CUDA(cudaMemsetAsync(d_stats, 0, 16 * (size_t)B, st));
  // The cell-order numbering of every scene: the five build kernels, each launched once over all scenes.  The grid's
  // cell size depends on k only for the speed of a kNN query, which is not run here (it is tuned up to KNN_MAX_K).
  KnnBuildScene ks[GEO_BATCH_MAX];
  KnnGridBuffers gb[GEO_BATCH_MAX];
  for (int b = 0; b < B; ++b) ks[b] = {xyz[b], Ns[b], w.knn[b].ptr, w.knn[b].bytes};
#ifndef GF_GEO_ORIGINAL_ORDER
  int rc = knn_grid_build_batch(ks, B, k < KNN_MAX_K ? k : KNN_MAX_K, w.knn_ctl, st, gb);
  if (rc) return rc;
#else
  int rc = GF_OK;
  for (int b = 0; b < B; ++b) gb[b].rank = gb[b].order = nullptr;
#endif
  // every scene's edge table in its cell order: one launch
  GeoPackArgs pa;
  memset(&pa, 0, sizeof(pa));
  pa.k = k, pa.slot_bits = w.edges[0].slot_bits, pa.radius = radius;
  long long maxE = 0;
  GeoSceneDesc desc[GEO_BATCH_MAX];
  for (int b = 0; b < B; ++b) {
    pa.sc[b] = {knn_dist[b], knn_idx[b], gb[b].rank, gb[b].order, w.edges[b].tgt, w.edges[b].len, Ns[b]};
    const long long E = ((long long)Ns[b] + 1) << pa.slot_bits;
    maxE = E > maxE ? E : maxE;
    desc[b].tgt = w.edges[b].tgt, desc[b].len = w.edges[b].len, desc[b].seeds = seeds[b], desc[b].geo = geo[b];
    desc[b].rank = gb[b].rank, desc[b].order = gb[b].order;
    desc[b].row_max = row_max ? row_max[b] : nullptr;
    desc[b].stats = d_stats ? d_stats + 2 * b : nullptr;
    desc[b].N = Ns[b], desc[b].Q = Q;
  }
  const long long per_scene = (long long)num_sms() * 16 / B > 1 ? (long long)num_sms() * 16 / B : 1;
  const long long need = (maxE + 255) / 256;
  const dim3 grid((unsigned)(need < per_scene ? need : per_scene), (unsigned)B);
  if (idx_is_i64)
    geo_pack_edges_batch_kernel<true><<<grid, 256, 0, st>>>(pa);
  else
    geo_pack_edges_batch_kernel<false><<<grid, 256, 0, st>>>(pa);
  GF_LAUNCHED();
  rc = geodesic_batch_launch(desc, B, k, max_step, w.scratch.ptr, w.scratch.bytes, st);
  if (rc) return rc;
  if (stats) GF_CUDA(cudaMemcpyAsync(stats, d_stats, 16 * (size_t)B, cudaMemcpyDeviceToDevice, st));
  return GF_OK;
}
