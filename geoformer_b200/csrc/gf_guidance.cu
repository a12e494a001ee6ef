// The fused hot path of BASELINE.json's north_star: FPS seeds -> kNN graph -> geodesic maps for one
// scene (what GeoFormerFS.forward does at geoformer_fs.py:630-645 + :497-506 through three separate
// libraries and a Python loop).  FPS (a <= 16-SM cluster kernel, latency bound) runs on a forked
// stream concurrently with the kNN graph construction (which fills the other SMs); the geodesic
// waits for both.
#include <stdlib.h>

#include "gf_geodesic.cuh"
#include "gf_knn.cuh"

namespace gf {

// Auxiliary streams of the fused path, one set per (device, caller stream) of the calling thread: FPS (a <= 16-SM
// cluster, latency bound) runs next to the kNN kernels, and the scenes of a batch run side by side on LANES
// lanes.  Callers that keep several calls in flight on several streams get one set per stream, so their kernels
// do not queue on a single hidden stream.  FPS lanes have the highest priority: FPS is the longest dependency
// chain of a scene, its cluster should be placed as soon as SMs free up.
// Measured with the graphs of a 20-scene call built and queried in one launch each (c2 bench, B200 at 1000 W, two
// runs each): 4 lanes 1.090 / 1.091 M maps/s, 6 lanes 1.094 / 1.095, 8 lanes 1.053 / 1.053.  6 lanes are 0.4 %
// ahead, which does not pay for two more high-priority streams per caller stream; 8 lanes lose 3.5 % (DESIGN
// section 8).
constexpr int LANES = 4;
struct ForkJoin {
  cudaStream_t fps[LANES] = {}, knn[LANES] = {};  // knn[0] stays null: lane 0 builds its graph on the caller's stream
  cudaEvent_t fork = nullptr, join_fps[LANES] = {}, join_knn[LANES] = {};
};

static int get_fork_join(cudaStream_t user, ForkJoin **out, int lanes_needed = 1) {
  constexpr int SLOTS = 16;
  struct Entry {
    int dev;
    cudaStream_t user;
    ForkJoin fj;
    bool used;
  };
  static thread_local Entry pool[SLOTS];
  static thread_local int next_victim = 0;
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  Entry *e = nullptr;
  for (int i = 0; i < SLOTS; ++i)
    if (pool[i].used && pool[i].dev == dev && pool[i].user == user) e = &pool[i];
  if (!e) {
    for (int i = 0; i < SLOTS && !e; ++i)
      if (!pool[i].used) e = &pool[i];
    if (!e) {  // more caller streams than slots: share (correct, only less concurrent)
      e = &pool[next_victim];
      next_victim = (next_victim + 1) % SLOTS;
      if (e->dev != dev) e = nullptr;
    }
    if (e && !e->used) {
      e->fj = ForkJoin();
      GF_CUDA(cudaEventCreateWithFlags(&e->fj.fork, cudaEventDisableTiming));
      e->used = true;
      e->dev = dev;
    }
    if (e) e->user = user;
  }
  if (!e) {
    set_error("guidance: no auxiliary stream available on device %d", dev);
    return GF_ERR_CUDA;
  }
  // Lanes are created on first use: every stream beyond the device's hardware queues (CUDA_DEVICE_MAX_CONNECTIONS,
  // 8 by default) shares a queue with another one and inherits false dependencies -- a single-scene call needs
  // exactly one auxiliary stream, only a batch of four or more scenes all of them.
  ForkJoin &f = e->fj;
  for (int l = 0; l < lanes_needed && l < LANES; ++l) {
    if (f.fps[l]) continue;
    int lo = 0, hi = 0;
    GF_CUDA(cudaDeviceGetStreamPriorityRange(&lo, &hi));  // hi = numerically lowest = greatest priority
    GF_CUDA(cudaStreamCreateWithPriority(&f.fps[l], cudaStreamNonBlocking, hi));
    GF_CUDA(cudaEventCreateWithFlags(&f.join_fps[l], cudaEventDisableTiming));
    if (l > 0) GF_CUDA(cudaStreamCreateWithPriority(&f.knn[l], cudaStreamNonBlocking, lo));
    GF_CUDA(cudaEventCreateWithFlags(&f.join_knn[l], cudaEventDisableTiming));
  }
  *out = &e->fj;
  return GF_OK;
}

struct GuidancePlan {
  size_t fps, knn, geo, total;
};

static GuidancePlan plan_guidance(int N, int Q, int k) {
  GuidancePlan p;
  p.fps = align256(gf_fps_workspace_bytes(1, N, Q));
  p.knn = align256(knn_grid_workspace_bytes(N));
  p.geo = align256(geodesic_workspace_bytes(N, k, Q));
  p.total = p.fps + p.knn + p.geo + 1024;
  return p;
}

}  // namespace gf

using namespace gf;

extern "C" size_t gf_guidance_workspace_bytes(int N, int Q, int k) {
  if (N <= 0 || Q <= 0 || k <= 0) return 0;
  return plan_guidance(N, Q, k).total;
}

// seeds_given == 0: run FPS (forked stream) and write `seeds`; != 0: `seeds` is an input
static int guidance_impl(const float *xyz, int N, int Q, int k, float radius, int max_step, int *seeds,
                         int seeds_given, float *geo, float *knn_dist, int32_t *knn_idx32, int64_t *stats,
                         void *workspace, size_t workspace_bytes, void *stream, float *const *peer_geo = nullptr,
                         int n_peers = 0, float *row_max = nullptr, int q0 = 0, int q1 = -1) {
  // [q0, q1): the block of seeds that is propagated here (all of them by default); FPS always samples all Q
  if (q1 < 0) q1 = Q;
  GF_CHECK_ARG(N >= 1 && Q >= 1, "guidance: need N >= 1 and Q >= 1 (N=%d Q=%d)", N, Q);
  GF_CHECK_ARG(q0 >= 0 && q0 <= q1 && q1 <= Q, "guidance: seed block [%d, %d) outside [0, %d)", q0, q1, Q);
  GF_CHECK_ARG(k >= 1 && k <= KNN_MAX_K, "guidance: k=%d outside [1,%d]", k, KNN_MAX_K);
  GF_CHECK_ARG(xyz && seeds && geo, "guidance: null pointer");
  GuidancePlan p = plan_guidance(N, Q, k);
  if (workspace == nullptr || workspace_bytes < p.total) {
    set_error("guidance: workspace too small (%zu bytes given, %zu needed)", workspace_bytes, p.total);
    return GF_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char *w = (char *)workspace;
  void *ws_fps = w;
  w += p.fps;
  void *ws_knn = w;
  w += p.knn;
  void *ws_geo = w;

  ForkJoin *fj = nullptr;
  int rc = GF_OK;
  stage_mark(ST_BEGIN, st);
  if (!seeds_given) {
    rc = get_fork_join(st, &fj);
    if (rc) return rc;
    // fork: FPS on the auxiliary stream
    GF_CUDA(cudaEventRecord(fj->fork, st));
    GF_CUDA(cudaStreamWaitEvent(fj->fps[0], fj->fork, 0));
    rc = gf_furthest_point_sampling(xyz, 1, N, Q, seeds, ws_fps, p.fps, fj->fps[0]);
    if (rc) return rc;
    GF_CUDA(cudaEventRecord(fj->join_fps[0], fj->fps[0]));
  }
  // main stream: kNN graph
  KnnGridBuffers gb;
  rc = knn_grid_build(xyz, N, k, ws_knn, p.knn, st, &gb);
  if (rc) return rc;
  stage_mark(ST_KNN_BUILT, st);
  // the query kernel writes the propagation's edge table straight from its registers; the (N,k) distance / index
  // arrays are only written when the caller asked for them
  KnnEdgeOut eo;
  eo.radius = radius;
  int enc = 0;
  const int Qb = q1 - q0;  // the workspace was sized for Q >= Qb seeds: enough for any block
  rc = geodesic_edge_buffers(ws_geo, p.geo, N, k, Q, &eo.tgt, &eo.len, &eo.slot_bits, &enc);
  if (rc) return rc;
  if (n_peers > 0) enc = 0;  // seed-sharded scenes run the per-scene kernel: original numbering, plain targets
  eo.rank = enc ? gb.rank : nullptr;
  rc = knn_grid_query(gb, nullptr, N, k, /*sqrt=*/1, knn_dist, nullptr, knn_idx32, st, &eo);
  if (rc) return rc;
  // join, then propagate
  if (!seeds_given) GF_CUDA(cudaStreamWaitEvent(st, fj->join_fps[0], 0));
  stage_mark(ST_KNN_DONE, st);
  if (Qb == 0) return GF_OK;
  return geodesic_run(nullptr, nullptr, /*is64=*/0, N, k, seeds + q0, Qb, radius, max_step, geo, stats, ws_geo, p.geo,
                      st, peer_geo, n_peers, row_max, enc ? gb.rank : nullptr, enc ? gb.order : nullptr);
}

extern "C" int gf_guidance(const float *xyz, int N, int Q, int k, float radius, int max_step, int *seeds, float *geo,
                           float *knn_dist, int32_t *knn_idx32, int64_t *stats, float *row_max, void *workspace,
                           size_t workspace_bytes, void *stream) {
  return guidance_impl(xyz, N, Q, k, radius, max_step, seeds, 0, geo, knn_dist, knn_idx32, stats, workspace,
                       workspace_bytes, stream, nullptr, 0, row_max);
}

extern "C" int gf_guidance_seeded(const float *xyz, int N, const int *seeds, int Q, int k, float radius, int max_step,
                                  float *geo, float *knn_dist, int32_t *knn_idx32, int64_t *stats, float *row_max,
                                  void *workspace, size_t workspace_bytes, void *stream) {
  return guidance_impl(xyz, N, Q, k, radius, max_step, const_cast<int *>(seeds), 1, geo, knn_dist, knn_idx32, stats,
                       workspace, workspace_bytes, stream, nullptr, 0, row_max);
}

extern "C" int gf_guidance_shard(const float *xyz, int N, int Q, int q0, int q1, int k, float radius, int max_step,
                                 int *seeds, float *geo_block, int64_t *stats, float *row_max_block, void *workspace,
                                 size_t workspace_bytes, void *stream) {
  return guidance_impl(xyz, N, Q, k, radius, max_step, seeds, 0, geo_block, nullptr, nullptr, stats, workspace,
                       workspace_bytes, stream, nullptr, 0, row_max_block, q0, q1);
}

extern "C" int gf_guidance_seeded_scatter(const float *xyz, int N, const int *seeds, int Q, int k, float radius,
                                          int max_step, float *geo, float *const *peer_geo, int n_peers,
                                          int64_t *stats, void *workspace, size_t workspace_bytes, void *stream) {
  return guidance_impl(xyz, N, Q, k, radius, max_step, const_cast<int *>(seeds), 1, geo, nullptr, nullptr, stats,
                       workspace, workspace_bytes, stream, peer_geo, n_peers);
}

// ---- a batch of scenes (the reference's call is batched: geodesic_utils.py:98 loops over the scenes) -------------
namespace gf {
static_assert(KNN_BATCH_MAX == GEO_BATCH_MAX, "one batched call builds and queries all its scenes' graphs at once");
struct BatchPlan {
  size_t per_scene[GEO_BATCH_MAX * 4];  // offsets of (fps, knn, edges) per scene
  size_t knn_ctl, scratch, scratch_bytes, stats, total;
};
static int plan_batch_guidance(const int *Ns, int B, int Q, int k, BatchPlan *p, size_t *fps_b, size_t *knn_b,
                               size_t *edge_b) {
  size_t off = 0;
  int maxN = 1;
  for (int b = 0; b < B; ++b) {
    const int N = Ns[b];
    fps_b[b] = align256(gf_fps_workspace_bytes(1, N, Q));
    knn_b[b] = align256(knn_grid_workspace_bytes(N));
    // the edge tables are the head of a single-scene geodesic workspace; only that head is used here
    edge_b[b] = align256(geodesic_workspace_bytes(N, k, 1));
    p->per_scene[b * 3 + 0] = off, off += fps_b[b];
    p->per_scene[b * 3 + 1] = off, off += knn_b[b];
    p->per_scene[b * 3 + 2] = off, off += edge_b[b];
    maxN = N > maxN ? N : maxN;
  }
  p->knn_ctl = off;
  off += align256(knn_ctl_block_bytes(B));
  p->scratch = off;
  p->scratch_bytes = align256(geodesic_batch_scratch_bytes(maxN, (long long)Q * B));
  off += p->scratch_bytes;
  p->stats = off;
  off += align256(16 * (size_t)B);
  p->total = off + 1024;
  return maxN;
}
}  // namespace gf

extern "C" size_t gf_guidance_batch_workspace_bytes(const int *Ns, int B, int Q, int k) {
  if (!Ns || B <= 0 || B > GEO_BATCH_MAX || Q <= 0 || k <= 0) return 0;
  for (int b = 0; b < B; ++b)
    if (Ns[b] <= 0) return 0;
  BatchPlan p;
  size_t f[GEO_BATCH_MAX], n[GEO_BATCH_MAX], e[GEO_BATCH_MAX];
  plan_batch_guidance(Ns, B, Q, k, &p, f, n, e);
  return p.total;
}

extern "C" int gf_guidance_batch(const float *const *xyz, const int *Ns, int B, int Q, int k, float radius,
                                 int max_step, int *const *seeds, int seeds_given, float *const *geo,
                                 float *const *row_max, int64_t *stats, void *workspace, size_t workspace_bytes,
                                 void *stream) {
  GF_CHECK_ARG(xyz && Ns && seeds && geo, "guidance_batch: null pointer array");
  GF_CHECK_ARG(B >= 1 && B <= GEO_BATCH_MAX, "guidance_batch: B=%d outside [1,%d]", B, GEO_BATCH_MAX);
  GF_CHECK_ARG(Q >= 1, "guidance_batch: need Q >= 1");
  GF_CHECK_ARG(k >= 1 && k <= KNN_MAX_K, "guidance_batch: k=%d outside [1,%d]", k, KNN_MAX_K);
  for (int b = 0; b < B; ++b) {
    GF_CHECK_ARG(Ns[b] >= 1 && xyz[b] && seeds[b] && geo[b], "guidance_batch: scene %d: empty or null", b);
    GF_CHECK_ARG(geodesic_edge_format(Ns[b]) == 1,
                 "guidance_batch: scene %d has %d points, beyond the on-chip bitmaps of the batched kernel "
                 "(use gf_guidance per scene)", b, Ns[b]);
  }
  BatchPlan p;
  size_t fps_b[GEO_BATCH_MAX], knn_b[GEO_BATCH_MAX], edge_b[GEO_BATCH_MAX];
  plan_batch_guidance(Ns, B, Q, k, &p, fps_b, knn_b, edge_b);
  if (workspace == nullptr || workspace_bytes < p.total) {
    set_error("guidance_batch: workspace too small (%zu bytes given, %zu needed)", workspace_bytes, p.total);
    return GF_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char *w = (char *)workspace;
  ForkJoin *fj = nullptr;
  const int lanes = B < LANES ? B : LANES;
  int rc = get_fork_join(st, &fj, lanes);
  if (rc) return rc;
  stage_mark(ST_BEGIN, st);
  // The graphs.  Up to LANES scenes, every scene has a lane of its own (lane 0: the caller's stream) and its graph
  // is one short chain next to its FPS.  With more scenes a lane would run several graphs one after another, each a
  // chain of six launches ending in a single-wave tail; there the graphs of all scenes are built with one launch of
  // each build kernel and queried with one launch, on the caller's stream (DESIGN section 4.2).
  const bool batched = B > LANES;
  GF_CUDA(cudaEventRecord(fj->fork, st));
  for (int l = 0; l < lanes; ++l) {
    if (!seeds_given) GF_CUDA(cudaStreamWaitEvent(fj->fps[l], fj->fork, 0));
    if (l > 0 && !batched) GF_CUDA(cudaStreamWaitEvent(fj->knn[l], fj->fork, 0));
  }
  GeoSceneDesc desc[GEO_BATCH_MAX];
  int64_t *d_stats = stats ? (int64_t *)(w + p.stats) : nullptr;
  if (d_stats) GF_CUDA(cudaMemsetAsync(d_stats, 0, 16 * (size_t)B, st));
  // FPS first on every lane (the longest chains start first), then the graphs
  if (!seeds_given)
    for (int b = 0; b < B; ++b) {
      rc = gf_furthest_point_sampling(xyz[b], 1, Ns[b], Q, seeds[b], w + p.per_scene[b * 3 + 0], fps_b[b],
                                      fj->fps[b % lanes]);
      if (rc) return rc;
    }
  KnnBuildScene ks[GEO_BATCH_MAX];
  KnnGridBuffers gb[GEO_BATCH_MAX];
  KnnEdgeOut eo[GEO_BATCH_MAX];
  KnnQueryJob jobs[GEO_BATCH_MAX];
  for (int b = 0; b < B; ++b) ks[b] = {xyz[b], Ns[b], w + p.per_scene[b * 3 + 1], knn_b[b]};
  if (batched) {
    rc = knn_grid_build_batch(ks, B, k, w + p.knn_ctl, st, gb);
    if (rc) return rc;
  }
  for (int b = 0; b < B; ++b) {
    const int l = b % lanes;
    cudaStream_t kst = l == 0 ? st : fj->knn[l];
    if (!batched) {
      rc = knn_grid_build_batch(&ks[b], 1, k, nullptr, kst, &gb[b]);
      if (rc) return rc;
    }
    eo[b].radius = radius;
    int enc = 0;
    rc = geodesic_edge_buffers(w + p.per_scene[b * 3 + 2], edge_b[b], Ns[b], k, 1, &eo[b].tgt, &eo[b].len,
                               &eo[b].slot_bits, &enc);
    if (rc) return rc;
    eo[b].rank = gb[b].rank;  // cell-order table (every scene of a batched call is batchable: checked above)
    jobs[b] = {gb[b], nullptr, Ns[b], nullptr, nullptr, nullptr, &eo[b]};
    if (!batched) {
      rc = knn_grid_query_batch(&jobs[b], 1, k, /*sqrt=*/1, kst);
      if (rc) return rc;
    }
    desc[b].tgt = eo[b].tgt, desc[b].len = eo[b].len, desc[b].seeds = seeds[b], desc[b].geo = geo[b];
    desc[b].rank = gb[b].rank, desc[b].order = gb[b].order;
    desc[b].row_max = row_max ? row_max[b] : nullptr;
    desc[b].stats = d_stats ? d_stats + 2 * b : nullptr;
    desc[b].N = Ns[b], desc[b].Q = Q;
  }
  if (batched) {
    rc = knn_grid_query_batch(jobs, B, k, /*sqrt=*/1, st);
    if (rc) return rc;
  }
  for (int l = 0; l < lanes; ++l) {
    if (!seeds_given) {
      GF_CUDA(cudaEventRecord(fj->join_fps[l], fj->fps[l]));
      GF_CUDA(cudaStreamWaitEvent(st, fj->join_fps[l], 0));
    }
    if (l > 0 && !batched) {
      GF_CUDA(cudaEventRecord(fj->join_knn[l], fj->knn[l]));
      GF_CUDA(cudaStreamWaitEvent(st, fj->join_knn[l], 0));
    }
  }
  stage_mark(ST_KNN_DONE, st);
  rc = geodesic_batch_launch(desc, B, k, max_step, w + p.scratch, p.scratch_bytes, st);
  if (rc) return rc;
  if (stats) GF_CUDA(cudaMemcpyAsync(stats, d_stats, 16 * (size_t)B, cudaMemcpyDeviceToDevice, st));
  return GF_OK;
}

extern "C" size_t gf_guidance_host_workspace_bytes(int N, int Q, int k) {
  if (N <= 0 || Q <= 0 || k <= 0) return 0;
  return plan_guidance(N, Q, k).total + align256(sizeof(float) * (size_t)N * 3) + align256(sizeof(int) * (size_t)Q) +
         align256(sizeof(float) * (size_t)Q * N) + 1024;
}

extern "C" int gf_guidance_host(const float *xyz_host, int N, int Q, int k, float radius, int max_step,
                                int *seeds_host, float *geo_host, void *workspace, size_t workspace_bytes,
                                void *stream) {
  GF_CHECK_ARG(N >= 1 && Q >= 1, "guidance_host: need N >= 1 and Q >= 1");
  GF_CHECK_ARG(xyz_host && seeds_host && geo_host, "guidance_host: null host pointer");
  size_t need = gf_guidance_host_workspace_bytes(N, Q, k);
  if (workspace == nullptr || workspace_bytes < need) {
    set_error("guidance_host: workspace too small (%zu bytes given, %zu needed)", workspace_bytes, need);
    return GF_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char *w = (char *)workspace;
  float *d_xyz = (float *)w;
  w += align256(sizeof(float) * (size_t)N * 3);
  int *d_seeds = (int *)w;
  w += align256(sizeof(int) * (size_t)Q);
  float *d_geo = (float *)w;
  w += align256(sizeof(float) * (size_t)Q * N);
  size_t inner = plan_guidance(N, Q, k).total;
  GF_CUDA(cudaMemcpyAsync(d_xyz, xyz_host, sizeof(float) * (size_t)N * 3, cudaMemcpyHostToDevice, st));
  int rc = gf_guidance(d_xyz, N, Q, k, radius, max_step, d_seeds, d_geo, nullptr, nullptr, nullptr, nullptr, w, inner, st);
  if (rc) return rc;
  GF_CUDA(cudaMemcpyAsync(seeds_host, d_seeds, sizeof(int) * (size_t)Q, cudaMemcpyDeviceToHost, st));
  GF_CUDA(cudaMemcpyAsync(geo_host, d_geo, sizeof(float) * (size_t)Q * N, cudaMemcpyDeviceToHost, st));
  GF_CUDA(cudaStreamSynchronize(st));
  return GF_OK;
}

// ---- host-buffer variant of the batched call (what bench.py's `e2e` number times) ---------------------------------
// The maps are 4*Q*N bytes per scene: at PCIe speed their copy takes several times as long as computing them, so
// the call is organised around the LINK: the scenes go one by one over two internal lanes (copy in -> hot path ->
// copy out), lane l + 1 computes while lane l's maps travel, and the device -> host copies follow each other without
// a gap.  (The one-launch batched propagation would deliver all maps at once, after the last scene's compute.)
namespace gf {
constexpr int HOST_LANES = 2;
struct HostLanes {
  cudaStream_t lane[HOST_LANES] = {};
  cudaEvent_t fork = nullptr, join[HOST_LANES] = {};
};
static int get_host_lanes(HostLanes **out) {
  static thread_local HostLanes pool[8];
  static thread_local bool used[8] = {};
  int dev = 0;
  GF_CUDA(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 8) dev = 0;
  HostLanes &h = pool[dev];
  if (!used[dev]) {
    GF_CUDA(cudaEventCreateWithFlags(&h.fork, cudaEventDisableTiming));
    for (int l = 0; l < HOST_LANES; ++l) {
      GF_CUDA(cudaStreamCreateWithFlags(&h.lane[l], cudaStreamNonBlocking));
      GF_CUDA(cudaEventCreateWithFlags(&h.join[l], cudaEventDisableTiming));
    }
    used[dev] = true;
  }
  *out = &h;
  return GF_OK;
}

struct HostBatchPlan {
  size_t xyz[GEO_BATCH_MAX], seeds[GEO_BATCH_MAX], geo[GEO_BATCH_MAX], lane_ws[HOST_LANES], lane_bytes, total;
};
static void plan_host_batch(const int *Ns, int B, int Q, int k, HostBatchPlan *p) {
  size_t off = 0;
  int maxN = 1;
  for (int b = 0; b < B; ++b) {
    p->xyz[b] = off, off += align256(sizeof(float) * 3 * (size_t)Ns[b]);
    p->seeds[b] = off, off += align256(sizeof(int) * (size_t)Q);
    p->geo[b] = off, off += align256(sizeof(float) * (size_t)Q * Ns[b]);
    maxN = Ns[b] > maxN ? Ns[b] : maxN;
  }
  p->lane_bytes = align256(plan_guidance(maxN, Q, k).total);
  for (int l = 0; l < HOST_LANES; ++l) p->lane_ws[l] = off, off += p->lane_bytes;
  p->total = off + 1024;
}
}  // namespace gf

extern "C" size_t gf_guidance_batch_host_workspace_bytes(const int *Ns, int B, int Q, int k) {
  if (!Ns || B <= 0 || B > GEO_BATCH_MAX || Q <= 0 || k <= 0) return 0;
  for (int b = 0; b < B; ++b)
    if (Ns[b] <= 0) return 0;
  HostBatchPlan p;
  plan_host_batch(Ns, B, Q, k, &p);
  return p.total;
}

extern "C" int gf_guidance_batch_host(const float *const *xyz_host, const int *Ns, int B, int Q, int k, float radius,
                                      int max_step, int *const *seeds_host, float *const *geo_host, void *workspace,
                                      size_t workspace_bytes, void *stream) {
  GF_CHECK_ARG(xyz_host && Ns && seeds_host && geo_host, "guidance_batch_host: null pointer array");
  GF_CHECK_ARG(B >= 1 && B <= GEO_BATCH_MAX && Q >= 1, "guidance_batch_host: B=%d Q=%d", B, Q);
  GF_CHECK_ARG(k >= 1 && k <= KNN_MAX_K, "guidance_batch_host: k=%d outside [1,%d]", k, KNN_MAX_K);
  for (int b = 0; b < B; ++b)
    GF_CHECK_ARG(Ns[b] >= 1 && xyz_host[b] && seeds_host[b] && geo_host[b], "guidance_batch_host: scene %d: empty or null", b);
  HostBatchPlan p;
  plan_host_batch(Ns, B, Q, k, &p);
  if (workspace == nullptr || workspace_bytes < p.total) {
    set_error("guidance_batch_host: workspace too small (%zu bytes given, %zu needed)", workspace_bytes, p.total);
    return GF_ERR_WORKSPACE;
  }
  cudaStream_t st = (cudaStream_t)stream;
  char *w = (char *)workspace;
  HostLanes *hl = nullptr;
  int rc = get_host_lanes(&hl);
  if (rc) return rc;
  const int lanes = B < HOST_LANES ? B : HOST_LANES;
  GF_CUDA(cudaEventRecord(hl->fork, st));
  for (int l = 0; l < lanes; ++l) GF_CUDA(cudaStreamWaitEvent(hl->lane[l], hl->fork, 0));
  for (int b = 0; b < B; ++b) {
    const int l = b % lanes;
    cudaStream_t ls = hl->lane[l];
    float *d_xyz = (float *)(w + p.xyz[b]);
    int *d_seeds = (int *)(w + p.seeds[b]);
    float *d_geo = (float *)(w + p.geo[b]);
    GF_CUDA(cudaMemcpyAsync(d_xyz, xyz_host[b], sizeof(float) * 3 * (size_t)Ns[b], cudaMemcpyHostToDevice, ls));
    rc = gf_guidance(d_xyz, Ns[b], Q, k, radius, max_step, d_seeds, d_geo, nullptr, nullptr, nullptr, nullptr,
                     w + p.lane_ws[l], p.lane_bytes, ls);
    if (rc) return rc;
    GF_CUDA(cudaMemcpyAsync(seeds_host[b], d_seeds, sizeof(int) * (size_t)Q, cudaMemcpyDeviceToHost, ls));
    GF_CUDA(cudaMemcpyAsync(geo_host[b], d_geo, sizeof(float) * (size_t)Q * Ns[b], cudaMemcpyDeviceToHost, ls));
  }
  for (int l = 0; l < lanes; ++l) {
    GF_CUDA(cudaEventRecord(hl->join[l], hl->lane[l]));
    GF_CUDA(cudaStreamWaitEvent(st, hl->join[l], 0));
  }
  GF_CUDA(cudaStreamSynchronize(st));
  return GF_OK;
}
