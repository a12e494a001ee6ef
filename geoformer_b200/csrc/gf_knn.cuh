// Internal interface of the grid kNN (shared with the fused hot path in gf_guidance.cu).
#pragma once
#include "gf_common.cuh"

namespace gf {

constexpr int KNN_MAX_K = 64;  // register-resident top-k; GeoFormer uses neighbor <= 64 (geoformer_fs.py:503)

struct KnnGridBuffers {
  const void *grid;       // device KnnGrid
  const int *cell_start;  // (ncells+1) exclusive prefix of the cell populations
  const float4 *sorted;   // (N) points in cell order: x, y, z, bit-cast original index
  const int *order;       // (N) order[cell-order position] = original index
  const int *rank;        // (N) rank[original index] = cell-order position
};

// optional second output of the self query: the propagation's packed edge table (gf_geodesic.cuh)
struct KnnEdgeOut {
  int *tgt;    // (N + 1) << slot_bits
  float *len;  // (N + 1) << slot_bits
  float radius;
  int slot_bits;
  const int *rank;  // != nullptr: table in CELL ORDER (rows and targets are cell-order positions), targets stored
                    // encoded (geo_edge_code, gf_geodesic.cuh); nullptr: original indices, plain
};

// Scenes per batched build / query launch (the batched propagation's GEO_BATCH_MAX).  The kernels take one
// descriptor per scene as a kernel parameter.
constexpr int KNN_BATCH_MAX = 32;

size_t knn_grid_workspace_bytes(int N);
// the B <= KNN_BATCH_MAX control blocks of a batched build: one contiguous area, cleared by a single memset
size_t knn_ctl_block_bytes(int B);

// one scene of a batched build: its points and its own workspace of knn_grid_workspace_bytes(N) bytes
struct KnnBuildScene {
  const float *xyz;
  int N;
  void *workspace;
  size_t workspace_bytes;
};
// Builds the grids of B scenes with the five build kernels, each launched once over all scenes (blockIdx.y = scene).
// ctl_block: knn_ctl_block_bytes(B) bytes for the control blocks; nullptr only with B == 1, which uses the head of
// the scene's workspace.  out[b] receives scene b's buffers.
int knn_grid_build_batch(const KnnBuildScene *scenes, int B, int k, void *ctl_block, cudaStream_t st,
                         KnnGridBuffers *out);
int knn_grid_build(const float *xyz, int N, int k, void *workspace, size_t workspace_bytes, cudaStream_t st,
                   KnnGridBuffers *out);

// one scene of a batched query; queries == nullptr: the scene against itself (nq = N); edges only then
struct KnnQueryJob {
  KnnGridBuffers grid;
  const float *queries;
  int nq;
  float *dist;
  long long *idx64;
  int *idx32;
  const KnnEdgeOut *edges;
};
// One query launch over the queries of all B scenes (same k).
int knn_grid_query_batch(const KnnQueryJob *jobs, int B, int k, int do_sqrt, cudaStream_t st);
int knn_grid_query(const KnnGridBuffers &b, const float *queries, int nq, int k, int do_sqrt, float *dist,
                   long long *idx64, int *idx32, cudaStream_t st, const KnnEdgeOut *edges = nullptr);

}  // namespace gf
