// Internal interface of the geodesic propagation (shared with the fused hot path).
#pragma once
#include "gf_common.cuh"

namespace gf {

size_t geodesic_workspace_bytes(int N, int k, int Q);
int geodesic_run(const float *D, const void *I, int is64, int N, int k, const int *seeds, int Q, float radius,
                 int max_step, float *geo, int64_t *stats_out, void *workspace, size_t workspace_bytes,
                 cudaStream_t st, float *const *peer_rows = nullptr, int n_peers = 0, float *row_max = nullptr,
                 const int *rank = nullptr, const int *order = nullptr);

// ---- batched launch: the (scene, seed) pairs of several scenes in ONE kernel ----------------------------------
struct GeoSceneDesc {
  const int *tgt;    // packed edge table of the scene, in the format geodesic_edge_buffers reported (encoded)
  const float *len;
  const int *rank, *order;  // the numbering the table is written in (gf_knn.cuh: cell order); both null = original
  const int *seeds;  // (Q) device
  float *geo;        // (Q, N) device
  float *row_max;    // optional (Q)
  int64_t *stats;    // optional device [reached pairs, deepest level]; ACCUMULATED with atomics: clear before
  int N, Q;
};
size_t geodesic_batch_scratch_bytes(int maxN, long long items);
int geodesic_batch_launch(const GeoSceneDesc *scenes, int B, int k, int max_step, void *scratch, size_t scratch_bytes,
                          cudaStream_t st);
constexpr int GEO_BATCH_MAX = 32;

// the packed edge table of one scene, with its sentinel row N: (N + 1) << slot_bits targets and lengths
struct GeoEdges {
  int *tgt;
  float *len;
  int slot_bits;
};
// takes the edge table of a scene of N points with k neighbours from `a` (the head of the single-scene workspace; a
// batched call takes one per scene)
void geo_edges_carve(Arena &a, int N, int k, GeoEdges *e);

// where the packed edge table of a later geodesic_run(D = nullptr, ...) on the same workspace lives; the workspace
// must hold the whole layout that run uses, geodesic_workspace_bytes(N, k, Q) bytes
int geodesic_edge_buffers(void *workspace, size_t workspace_bytes, int N, int k, int Q, GeoEdges *e, int *enc);

int geodesic_edge_format(int N);  // 1 = encoded targets (the batched kernel takes the scene), 0 = plain

// ---- ENCODED edge targets (written by the kNN query and geo_pack_edges_kernel, read by the batched kernel) ------
// The edge table stores a target t as (t >> 5) << 7 | (t & 31), i.e. the byte offset of its bitmap word shifted left
// by 5 with the bit number in the low five bits.  The visited test of an edge -- 93 % of the edges of a kNN graph
// fail it -- is then four instructions (shift, LDS, funnel shift for the bit, LOP3 into a predicate) instead of
// eight; the byte offset into the claim array (4 * t) is only rebuilt on the rare hit.
__device__ __forceinline__ int geo_edge_code(unsigned t) { return (int)(((t >> 5) << 7) | (t & 31u)); }
// the target of an edge that is never taken: the sentinel point N
__device__ __forceinline__ int geo_edge_none(int N, bool encoded) { return encoded ? geo_edge_code((unsigned)N) : N; }
// byte offset of point t's word in a bitmap of the points, from t and from its code
__device__ __forceinline__ uint32_t geo_word_offset(unsigned t) { return (t >> 3) & ~3u; }
__device__ __forceinline__ uint32_t geo_edge_word_offset(unsigned code) { return code >> 5; }
// byte offset of the target's entry in an array of 4-byte entries per point: 4 * t
__device__ __forceinline__ uint32_t geo_edge_entry_offset(unsigned code) { return (code & ~127u) | ((code & 31u) << 2); }

}  // namespace gf
