/*
 * geoformer_b200.h -- C ABI of the B200 (sm_100a) geodesic-guidance library.
 *
 * Drop-in boundary for the hot path of VinAIResearch/GeoFormer:
 *   lib/pointnet2/_ext_src/src/bindings.cpp:9-22      (the nine pointnet2._ext operators)
 *   model/geoformer/geodesic_utils.py:11-24, 91-164   (find_knn, cal_geodesic_vectorize)
 *   model/geoformer/geoformer_fs.py:680-702, 263-292  (the two distance -> bias epilogues)
 *
 * Conventions
 *   - plain pointers and sizes only; no torch / ATen types.  `stream` is a cudaStream_t passed as
 *     void* (0 = legacy default stream).  All *device* entry points are asynchronous on `stream`
 *     and never synchronise the device; `*_host` entry points take HOST buffers, do their own
 *     H2D / D2H copies and return after the results are in host memory.
 *   - return value: 0 = ok, non-zero = error; gf_last_error() gives the message (thread-local).
 *     Nothing calls exit() (the reference does, cuda_utils.h:32-41).
 *   - layouts and dtypes are the reference's: float32 data, int32 indices for the pointnet2
 *     operators, batch-major (B,N,3) coordinates, channel-major (B,C,N) features, everything
 *     contiguous.  Outputs are fully written by the callee (the reference's zero-initialisation,
 *     e.g. ball_query rows without a hit, is reproduced by the callee, not assumed of the caller).
 *   - scratch memory is provided by the caller: gf_*_workspace_bytes() says how much.
 *   - there is no CPU fallback: every entry point needs a CUDA device.
 */
#ifndef GEOFORMER_B200_H
#define GEOFORMER_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define GF_OK 0
#define GF_ERR_INVALID 1 /* bad argument (the reference raises through AT_ASSERT, utils.h:8-28) */
#define GF_ERR_CUDA 2    /* CUDA runtime / launch failure */
#define GF_ERR_WORKSPACE 3

const char *gf_last_error(void);
int gf_version(void);
/* number of kernels launched by this library on the calling thread since the last reset */
int64_t gf_launch_count(void);
void gf_reset_launch_count(void);

/* Profiling hook: `events` = up to 5 cudaEvent_t (as void*) recorded, during the NEXT gf_guidance* /
 * gf_geodesic call of this thread only, on the launching stream at: [0] entry, [1] kNN grid built,
 * [2] kNN graph done (and FPS joined), [3] just before the propagation kernel, [4] propagation
 * kernel done.  NULL / 0 disarms.                                                                 */
int gf_set_stage_events(void **events, int n);
void *gf_event_create(void);                     /* cudaEventCreate, NULL on failure */
void gf_event_destroy(void *event);
float gf_event_elapsed_ms(void *start, void *stop); /* < 0 if either event has not completed */

/* ---- pointnet2._ext operators ------------------------------------------------------------- */

/* furthest_point_sampling  (sampling.cpp:67-88, sampling_gpu.cu:72-232; pointnet2_utils.py:59)
 * xyz (B,N,3) f32 -> idx (B,m) i32.  Start index 0, points with |p|^2 < 1e-3 are never selected,
 * ties resolved exactly like the reference's 512-wide shared-memory tree.                        */
size_t gf_fps_workspace_bytes(int B, int N, int m);
int gf_furthest_point_sampling(const float *xyz, int B, int N, int m, int *idx, void *workspace,
                               size_t workspace_bytes, void *stream);

/* The same over a RAGGED batch: xyz the flat (offsets[B],3) array, scene b its rows [offsets[b], offsets[b+1]);
 * offsets (B+1) is a HOST array, non-decreasing from 0.  idx (B,m) i32 with scene-local indices: row b is bit-identical
 * to gf_furthest_point_sampling on scene b alone.  The scenes that fit one thread-block cluster (N <= 196,608 with
 * 16-CTA clusters) run side by side, one launch per 32 of them, planned for the largest; each larger scene then runs
 * the single-scene whole-GPU kernel.  Workspace: gf_fps_batch_workspace_bytes (0 when every scene fits a cluster). */
size_t gf_fps_batch_workspace_bytes(const int *offsets, int B, int m);
int gf_furthest_point_sampling_batch(const float *xyz, const int *offsets, int B, int m, int *idx, void *workspace,
                                     size_t workspace_bytes, void *stream);

/* gather_points / gather_points_grad  (sampling.cpp:17-65, sampling_gpu.cu:11-60)
 * points (B,C,N), idx (B,m) -> out (B,C,m);   grad_out (B,C,m), idx -> grad_points (B,C,N)      */
int gf_gather_points(const float *points, const int *idx, int B, int C, int N, int m, float *out, void *stream);
int gf_gather_points_grad(const float *grad_out, const int *idx, int B, int C, int N, int m, float *grad_points,
                          void *stream);

/* ball_query  (ball_query.cpp:11-35, ball_query_gpu.cu:12-57).  Centres first, as in the binding.
 * new_xyz (B,m,3), xyz (B,N,3) -> idx (B,m,nsample) i32: first nsample indices (ascending) with
 * d2 < radius^2, padded with the first hit, all zero when there is none.                        */
int gf_ball_query(const float *new_xyz, const float *xyz, int B, int N, int m, float radius, int nsample, int *idx,
                  void *stream);

/* The same over a RAGGED batch: new_xyz (B,m,3), xyz the flat (offsets[B],3) array with offsets (B+1) a HOST array
 * as in gf_furthest_point_sampling_batch -> idx (B,m,nsample) i32, scene-local.  A centre of scene b searches only
 * the rows [offsets[b], offsets[b+1]); its row is bit-identical to gf_ball_query on scene b alone.  One launch per
 * 32 scenes.                                                                                                      */
int gf_ball_query_batch(const float *new_xyz, const float *xyz, const int *offsets, int B, int m, float radius,
                        int nsample, int *idx, void *stream);

/* group_points / group_points_grad  (group_points.cpp:15-62, group_points_gpu.cu:11-78)
 * points (B,C,N), idx (B,np,ns) -> out (B,C,np,ns);  grad_out (B,C,np,ns) -> grad_points (B,C,N) */
int gf_group_points(const float *points, const int *idx, int B, int C, int N, int npoints, int nsample, float *out,
                    void *stream);
int gf_group_points_grad(const float *grad_out, const int *idx, int B, int C, int N, int npoints, int nsample,
                         float *grad_points, void *stream);

/* three_nn / three_interpolate / three_interpolate_grad  (interpolate.cpp, interpolate_gpu.cu)
 * unknown (B,n,3), known (B,m,3) -> dist2 (B,n,3) f32 (squared), idx (B,n,3) i32                 */
int gf_three_nn(const float *unknown, const float *known, int B, int n, int m, float *dist2, int *idx, void *stream);
int gf_three_interpolate(const float *points, const int *idx, const float *weight, int B, int C, int m, int n,
                         float *out, void *stream);
int gf_three_interpolate_grad(const float *grad_out, const int *idx, const float *weight, int B, int C, int n, int m,
                              float *grad_points, void *stream);

/* ---- kNN graph (replaces faiss.GpuIndexFlatL2.search; geodesic_utils.py:18-22) ------------- */

/* Exact L2 kNN of `queries` (nq,3) against the database `xyz` (N,3), ordered by (d2, index) with
 * d2 = fmaf(dz,dz, fmaf(dx,dx, dy*dy)) in fp32 (the pointnet2 kernels' contraction).
 *   dist (nq,k) f32: squared distances, or their sqrt when sqrt_out != 0
 *   idx64 (nq,k) i64 and/or idx32 (nq,k) i32: either may be NULL.  Missing neighbours: -1 / +inf.
 *   queries == NULL means "the database against itself".
 *   algo: 0 = uniform-grid exact search (default), 1 = brute-force tiled scan (cross-check).     */
size_t gf_knn_workspace_bytes(int N, int nq, int k, int algo);
int gf_knn(const float *xyz, int N, const float *queries, int nq, int k, int sqrt_out, float *dist, int64_t *idx64,
           int32_t *idx32, int algo, void *workspace, size_t workspace_bytes, void *stream);

/* B <= 32 scenes, each against itself, through one launch of each grid-build kernel and one query launch:
 * scene b's dist[b] (Ns[b],k) f32 and idx32[b] (Ns[b],k) i32 (either may be NULL) equal what gf_knn with
 * queries == NULL and algo 0 writes for that scene alone.                                          */
size_t gf_knn_batch_workspace_bytes(const int *Ns, int B);
int gf_knn_batch(const float *const *xyz, const int *Ns, int B, int k, int sqrt_out, float *const *dist,
                 int32_t *const *idx32, void *workspace, size_t workspace_bytes, void *stream);

/* ---- geodesic propagation (cal_geodesic_vectorize, geodesic_utils.py:91-164) ---------------- */

/* One scene.  knn_dist (N,k) f32 (sqrt'ed), knn_idx (N,k) i64 or i32 (idx_is_i64), column 0 is
 * dropped like the reference (:110-111).  seeds (Q) i32.  geo (Q,N) f32, -1 = unreachable.
 * Level-synchronous first-visit BFS; within a level the parent with the smallest index, then the
 * smallest neighbour slot, wins.  Needs N << ceil(log2(k-1)) < 2^30.
 * stats (2) i64 device, optional: [0] = reached (q,p) pairs, [1] = deepest level reached.
 * row_max (Q) f32 device, optional: the maximum of every row of geo (a by-product of the propagation;
 * -1 for a row that stayed empty) -- what both epilogues start from (geoformer_fs.py:274-275).      */
size_t gf_geodesic_workspace_bytes(int N, int k, int Q);
int gf_geodesic(const float *knn_dist, const void *knn_idx, int idx_is_i64, int N, int k, const int *seeds, int Q,
                float radius, int max_step, float *geo, int64_t *stats, float *row_max, void *workspace,
                size_t workspace_bytes, void *stream);

/* ---- distance -> bias epilogues ------------------------------------------------------------- */

/* decoder relative-position bias (geoformer_fs.py:680-702):
 * geo[b] (Q,N_b) f32 given as an array of B device pointers, ctx_idx (B,C) i32, query_xyz (B,Q,3),
 * ctx_xyz (B,C,3) -> out (B,Q,C,3).                                                             */
size_t gf_bias_workspace_bytes(int B, int Q);
int gf_bias_decoder(const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx, const float *query_xyz,
                    const float *ctx_xyz, int B, int Q, int C, float *out, void *workspace, size_t workspace_bytes,
                    void *stream);
/* The same epilogue fused with the Fourier position embedding the decoder actually consumes
 * (geoformer_fs.py:704-712 -> PositionEmbeddingCoordsSine.get_fourier_embeddings, pos_embedding.py:88-114,
 * normalize=True -> shift_scale_points, utils_pc.py:35-61): gauss_B (3, >= d_out) f32 with row stride
 * gauss_ld, pc_min / pc_max (B,3) -> out (B,Q,C,2*d_out) f32 = [sin | cos]; the reference's
 * relative_embedding_pos is the (Q,C,B,2*d_out) permuted view of exactly this memory.  The (B,Q,C,3)
 * intermediate is never materialised.  Tolerance 2e-5 absolute (order of the 3-term dot product, sinf). */
int gf_bias_decoder_fourier(const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx,
                            const float *query_xyz, const float *ctx_xyz, int B, int Q, int C, const float *gauss_B,
                            int d_out, int gauss_ld, const float *pc_min, const float *pc_max, float *out,
                            void *workspace, size_t workspace_bytes, void *stream);
/* mask-head relative coordinates (geoformer_fs.py:263-292):
 * geo (Q,N), coords (N,3), seed_xyz (Q,3) -> out (Q,3,N).  row_max (Q) optional: the row maxima as
 * returned by gf_geodesic / gf_guidance; when given, geo is read once instead of twice.          */
int gf_bias_mask_head(const float *geo, const float *coords, const float *seed_xyz, int Q, int N,
                      const float *row_max, float *out, void *workspace, size_t workspace_bytes, void *stream);

/* ---- the consumer of the decoder bias: vector cross-attention (SURVEY 8(f) rank 2) -----------------------------
 * model/transformer_detr.py:443-454 (MLPs :384-396): for every query q and context c
 *     sim = W2 relu(W1 (tgt2[q] - memory[c] + rel[q,c]) + b1) + b2,   v2 = Wv (memory[c] + rel[q,c]) + bv
 *     out[q] = relu(Wo (sum_c softmax_c(sim / 8) * v2) + bo)          (softmax over the contexts, per channel)
 * tgt2 (Q,B,64) = norm2(tgt), memory (C,B,64), relative_pos (Q,C,B,64), weights (64,64) row-major (out,in) like
 * nn.Linear.weight -> out (Q,B,64), all f32 device.  One tcgen05 kernel (TF32 products, fp32 accumulation in
 * TMEM); the three (Q,C,B,64) temporaries of the reference are never materialised.  Tolerance vs fp32: 2e-3.
 * The _fused variant takes the arguments of gf_bias_decoder_fourier instead of relative_pos and builds the
 * embedding tile by tile in shared memory (32 frequencies: channels [sin | cos], B <= 8).                    */
size_t gf_rel_cross_attention_workspace_bytes(int Q, int C, int B);
int gf_rel_cross_attention(const float *tgt2, const float *memory, const float *relative_pos, int Q, int C, int B,
                           const float *w1, const float *b1, const float *w2, const float *b2, const float *wv,
                           const float *bv, const float *wo, const float *bo, float *out, void *workspace,
                           size_t workspace_bytes, void *stream);
int gf_rel_cross_attention_fused(const float *tgt2, const float *memory, const float *const *geo_ptrs,
                                 const int *geo_ld, const int *ctx_idx, const float *query_xyz, const float *ctx_xyz,
                                 const float *gauss_B, int gauss_ld, const float *pc_min, const float *pc_max, int Q,
                                 int C, int B, const float *w1, const float *b1, const float *w2, const float *b2,
                                 const float *wv, const float *bv, const float *wo, const float *bo, float *out,
                                 void *workspace, size_t workspace_bytes, void *stream);

/* Training.  The _save variants are the forwards above that also write what the backward needs: o (Q,B,64), the
 * softmax-weighted sum before out_mlp, and lse (Q,B,64) = max + log(sum) of the scores sim / 8; `out` is bitwise the
 * same as without saving.  The _backward entries take the forward's inputs, out, o, lse and the upstream gradient
 * dy (Q,B,64) and write the gradients of tgt2, memory, the eight weights and (unfused, when drel is not NULL)
 * relative_pos, all f32 device, same shapes as the inputs.  They recompute the scores tile by tile on the tensor
 * cores (TF32, like the forward) and reduce in a fixed order without atomics: two calls give bitwise-equal
 * gradients.  db2 is exactly zero (the softmax is shift invariant per channel).  The fused backward takes the
 * embedding ingredients as data: no gradient for the maps, locations or gauss_B.  The workspace holds a
 * (Q,B,C,128) buffer: gf_rel_cross_attention_backward_workspace_bytes.                                        */
int gf_rel_cross_attention_save(const float *tgt2, const float *memory, const float *relative_pos, int Q, int C,
                                int B, const float *w1, const float *b1, const float *w2, const float *b2,
                                const float *wv, const float *bv, const float *wo, const float *bo, float *out,
                                float *o, float *lse, void *workspace, size_t workspace_bytes, void *stream);
int gf_rel_cross_attention_fused_save(const float *tgt2, const float *memory, const float *const *geo_ptrs,
                                      const int *geo_ld, const int *ctx_idx, const float *query_xyz,
                                      const float *ctx_xyz, const float *gauss_B, int gauss_ld, const float *pc_min,
                                      const float *pc_max, int Q, int C, int B, const float *w1, const float *b1,
                                      const float *w2, const float *b2, const float *wv, const float *bv,
                                      const float *wo, const float *bo, float *out, float *o, float *lse,
                                      void *workspace, size_t workspace_bytes, void *stream);
size_t gf_rel_cross_attention_backward_workspace_bytes(int Q, int C, int B);
int gf_rel_cross_attention_backward(const float *tgt2, const float *memory, const float *relative_pos, int Q, int C,
                                    int B, const float *w1, const float *b1, const float *w2, const float *b2,
                                    const float *wv, const float *bv, const float *wo, const float *bo,
                                    const float *out, const float *o, const float *lse, const float *dy, float *dtgt2,
                                    float *dmemory, float *drel, float *dw1, float *db1, float *dw2, float *db2,
                                    float *dwv, float *dbv, float *dwo, float *dbo, void *workspace,
                                    size_t workspace_bytes, void *stream);
int gf_rel_cross_attention_fused_backward(const float *tgt2, const float *memory, const float *const *geo_ptrs,
                                          const int *geo_ld, const int *ctx_idx, const float *query_xyz,
                                          const float *ctx_xyz, const float *gauss_B, int gauss_ld,
                                          const float *pc_min, const float *pc_max, int Q, int C, int B,
                                          const float *w1, const float *b1, const float *w2, const float *b2,
                                          const float *wv, const float *bv, const float *wo, const float *bo,
                                          const float *out, const float *o, const float *lse, const float *dy,
                                          float *dtgt2, float *dmemory, float *dw1, float *db1, float *dw2,
                                          float *db2, float *dwv, float *dbv, float *dwo, float *dbo,
                                          void *workspace, size_t workspace_bytes, void *stream);

/* ---- mask head fused (geoformer_fs.py:263-300, mask_heads_forward) ---------------------------------------------
 * One scene: geo (Q,N) maps, feats (N,m) mask features, the dynamic weights w0 (Q*m, m+3), b0 (Q*m), w1 (Q, m),
 * b1 (Q) as the controller's parameter split gives them, coords (N,3), seed_xyz (Q,3) and optionally row_max (Q)
 * (the producer's row maxima, as gf_bias_mask_head takes them; NULL: computed from geo) -> out (Q,N) logits
 *     rel = gf_bias_mask_head's (Q,3,N) output, x = [rel | feats^T] (the order of the reference's cat),
 *     h = relu(w0 x + b0) per query, out = w1 h + b1.
 * Only m = 16.  The feature part of w0 x runs on the tensor cores (TF32, fp32 accumulation); the coordinate part,
 * the unreachable decisions and the second layer are fp32 on the CUDA cores.  Nothing of size (Q, >1, N) is
 * written.  Workspace: gf_mask_head_workspace_bytes.
 * The backward takes the same inputs and dlogit (Q,N) and writes the gradients of feats (N,m), w0 (Q*m, m+3),
 * b0 (Q*m), w1 (Q,m) and b1 (Q).  It recomputes h with the forward's products (bit-identical ReLU masks) and sums
 * in a fixed order without atomics: two calls give bitwise-equal gradients.  The maps and coordinates are data (no
 * gradient).  Workspace: gf_mask_head_backward_workspace_bytes.                                                  */
size_t gf_mask_head_workspace_bytes(int Q, int N);
int gf_mask_head_logits(const float *geo, const float *feats, const float *w0, const float *b0, const float *w1,
                        const float *b1, const float *coords, const float *seed_xyz, const float *row_max, int Q, int N,
                        int m, float *out, void *workspace, size_t workspace_bytes, void *stream);
size_t gf_mask_head_backward_workspace_bytes(int Q, int N);
int gf_mask_head_logits_backward(const float *geo, const float *feats, const float *w0, const float *b0,
                                 const float *w1, const float *b1, const float *coords, const float *seed_xyz,
                                 const float *row_max, int Q, int N, int m, const float *dlogit, float *dfeats,
                                 float *dw0, float *db0, float *dw1, float *db1, void *workspace,
                                 size_t workspace_bytes, void *stream);

/* ---- set_aggregator.mlp fused with its grouping (SURVEY 8(f) rank 3) --------------------------------------------
 * lib/pointnet2/pointnet2_modules.py:200-249 + QueryAndGroup.forward (pointnet2_utils.py:303-356) + SharedMLP
 * (pytorch_utils.py:9-32): per centre j and ball-query neighbour s the input [(xyz[idx] - new_xyz[j]) / radius |
 * features[:, idx]] goes through n_layers x (1x1 conv, batch norm in inference form, ReLU) and is max- or
 * mean-pooled over the nsample neighbours.  xyz (B,N,3), new_xyz (B,m,3), features (B,C,N) or NULL, idx (B,m,nsample)
 * i32 (gf_ball_query) -> out (B, widths[n_layers], m).  widths (n_layers+1, host): input channels (3 + C when use_xyz)
 * and every layer's output channels, each <= 32; weights[l] (widths[l+1], widths[l]) row-major, scales[l] / shifts[l]
 * (widths[l+1]): y = relu(scale * (W x) + shift), i.e. gamma / sqrt(var + eps) and beta - mean * that (host arrays of
 * device pointers).  The (B, 3+C, m, nsample) grouped tensors and per-layer activations are never materialised.   */
int gf_group_mlp_pool(const float *xyz, const float *new_xyz, const float *features, const int *idx, int B, int N, int m,
                      int nsample, int C, float radius, int normalize_xyz, int use_xyz, int n_layers, const int *widths,
                      const float *const *weights, const float *const *scales, const float *const *shifts, int pool_avg,
                      float *out, void *stream);

/* ---- set_aggregator in training form: batch statistics and the backward of gf_group_mlp_pool -------------------
 * Same inputs as gf_group_mlp_pool.  consts (n_layers, 5, 32) device floats per layer: scale, shift, mean of W h,
 * invstd, biased variance.  A layer with batch_stats[l] = 0 is FIXED: the caller fills its scale and shift (and, for
 * the backward, mean and invstd of its batch norm) with zeros past its width.  A layer with batch_stats[l] = 1 uses
 * the statistics of this call's input (torch's BatchNorm2d in training mode over all B * m * nsample elements): the
 * forward computes its five rows on the device from gammas[l], betas[l], eps[l] (host arrays of device pointers and
 * host floats), then runs gf_group_mlp_pool with them.  No host synchronisation.  Workspace:
 * gf_group_mlp_pool_train_workspace_bytes.
 * The backward takes the forward's consts and dout (B, widths[n_layers], m) and writes dweights[l] (widths[l+1],
 * widths[l]), dvec (n_layers, 3, 32): gradients of the conv bias, gamma and beta, and dfeatures (B, C, N) (NULL: not
 * computed).  It recomputes the forward with the forward's expressions (bit-identical ReLU masks and max-pool
 * argmax, first maximal sample) and sums in a fixed order without float atomics: two calls give bitwise-equal
 * gradients.  Workspace: gf_group_mlp_pool_backward_workspace_bytes.                                              */
size_t gf_group_mlp_pool_train_workspace_bytes(int B, int m);
int gf_group_mlp_pool_train(const float *xyz, const float *new_xyz, const float *features, const int *idx, int B,
                            int N, int m, int nsample, int C, float radius, int normalize_xyz, int use_xyz,
                            int n_layers, const int *widths, const float *const *weights, const float *const *gammas,
                            const float *const *betas, const float *eps, const int *batch_stats, float *consts,
                            int pool_avg, float *out, void *workspace, size_t workspace_bytes, void *stream);
size_t gf_group_mlp_pool_backward_workspace_bytes(int B, int N, int m, int nsample, int C);
int gf_group_mlp_pool_backward(const float *xyz, const float *new_xyz, const float *features, const int *idx, int B,
                               int N, int m, int nsample, int C, float radius, int normalize_xyz, int use_xyz,
                               int n_layers, const int *widths, const float *const *weights, const int *batch_stats,
                               const float *consts, int pool_avg, const float *dout, float *dfeatures,
                               float *const *dweights, float *dvec, void *workspace, size_t workspace_bytes,
                               void *stream);

/* ---- fused hot path: FPS -> kNN -> geodesic -------------------------------------------------- */

/* Device-resident scene: xyz (N,3) -> seeds (Q) i32, geo (Q,N) f32.  knn_dist / knn_idx32 (N,k)
 * may be NULL (kept in the workspace).                                                           */
size_t gf_guidance_workspace_bytes(int N, int Q, int k);
int gf_guidance(const float *xyz, int N, int Q, int k, float radius, int max_step, int *seeds, float *geo,
                float *knn_dist, int32_t *knn_idx32, int64_t *stats, float *row_max, void *workspace,
                size_t workspace_bytes, void *stream);

/* Same, with the seeds given (the body of cal_geodesic_vectorize for one scene, geodesic_utils.py:98-163:
 * kNN of the scene against itself, then the propagation from pre_enc_inds[b][:n_queries]).       */
int gf_guidance_seeded(const float *xyz, int N, const int *seeds, int Q, int k, float radius, int max_step,
                       float *geo, float *knn_dist, int32_t *knn_idx32, int64_t *stats, float *row_max,
                       void *workspace, size_t workspace_bytes, void *stream);

/* A BATCH of scenes in one call: what cal_geodesic_vectorize does for the scenes of a batch (geodesic_utils.py:98
 * loops over them one by one).  xyz[b] (Ns[b],3), seeds[b] (Q) i32 (written unless seeds_given), geo[b] (Q,Ns[b]),
 * optional row_max[b] (Q); the pointer ARRAYS live in host memory, what they point to in device memory.
 * stats: optional device (B,2) i64.  FPS and graph construction of the scenes run side by side on internal
 * streams; the propagation of ALL scenes is ONE launch whose work items are (scene, seed) pairs, so that the
 * GPU holds three to four times as many of these latency-bound runs as a scene alone offers.  B <= 32; every
 * scene must fit the on-chip bitmaps (N <~ 860k), larger scenes go through gf_guidance one by one.          */
size_t gf_guidance_batch_workspace_bytes(const int *Ns, int B, int Q, int k);
int gf_guidance_batch(const float *const *xyz, const int *Ns, int B, int Q, int k, float radius, int max_step,
                      int *const *seeds, int seeds_given, float *const *geo, float *const *row_max, int64_t *stats,
                      void *workspace, size_t workspace_bytes, void *stream);

/* ---- one scene over several GPUs, split by seed blocks (SURVEY 8(e), config c4) --------------------
 * New with this library (the reference is single-GPU, train.py:156-185).  Every rank holds the whole
 * (Q_total,N) matrix; rank r propagates the seeds [row0, row0+Q) and the propagation kernel itself stores
 * each finished row into the peers' matrices over NVLink while the other seeds are still running, so no
 * collective follows.  `geo` and every peer_geo[i] point at ROW row0 of the respective matrix (the
 * addresses of the peers' matrices in this process come from gf_peer_open).  n_peers <= 15.  The
 * caller separates consecutive calls by a barrier among the ranks (before: peers finished reading
 * the previous result; after: all rows have landed).                                              */
/* The same partition without any exchange: FPS samples all Q seeds (replicated: it is sequential and cheap next to
 * the propagation of a large scene), this rank propagates the seeds [q0, q1) into geo_block (q1 - q0, N); the
 * consumer of the maps is then sharded by query as well.  Workspace: gf_guidance_workspace_bytes(N, Q, k).       */
int gf_guidance_shard(const float *xyz, int N, int Q, int q0, int q1, int k, float radius, int max_step, int *seeds,
                      float *geo_block, int64_t *stats, float *row_max_block, void *workspace,
                      size_t workspace_bytes, void *stream);
int gf_geodesic_scatter(const float *knn_dist, const void *knn_idx, int idx_is_i64, int N, int k, const int *seeds,
                        int Q, float radius, int max_step, float *geo, float *const *peer_geo, int n_peers,
                        int64_t *stats, void *workspace, size_t workspace_bytes, void *stream);
int gf_guidance_seeded_scatter(const float *xyz, int N, const int *seeds, int Q, int k, float radius, int max_step,
                               float *geo, float *const *peer_geo, int n_peers, int64_t *stats, void *workspace,
                               size_t workspace_bytes, void *stream);
/* Peer-visible device memory: a plain cudaMalloc allocation (exportable as a whole), its 64-byte
 * CUDA IPC handle, and the mapping of another process's handle into this one.                   */
#define GF_PEER_HANDLE_BYTES 64
int gf_peer_alloc(void **dev_ptr, size_t bytes);
int gf_peer_free(void *dev_ptr);
int gf_peer_export(void *dev_ptr, void *handle_out);
int gf_peer_open(const void *handle, void **dev_ptr);
int gf_peer_close(void *dev_ptr);

/* Host-buffer variant (the reference-facing call timed as `e2e`): xyz_host (N,3) in, seeds_host (Q)
 * and geo_host (Q,N) out; copies are issued on `stream` and the call returns after they finish.
 * Device scratch of gf_guidance_host_workspace_bytes() is supplied by the caller.                */
size_t gf_guidance_host_workspace_bytes(int N, int Q, int k);
int gf_guidance_host(const float *xyz_host, int N, int Q, int k, float radius, int max_step, int *seeds_host,
                     float *geo_host, void *workspace, size_t workspace_bytes, void *stream);

/* The batched call with HOST buffers: xyz_host[b] (Ns[b],3) in, seeds_host[b] (Q) and geo_host[b] (Q,Ns[b]) out
 * (pinned memory for full copy speed); the pointer arrays live in host memory too.  Copies are issued on
 * `stream`, the call returns after the results are in host memory.  Two callers on two streams keep the link
 * busy: the device -> host copy of one batch (the maps are 4*Q*N bytes per scene) runs under the next batch.  */
size_t gf_guidance_batch_host_workspace_bytes(const int *Ns, int B, int Q, int k);
int gf_guidance_batch_host(const float *const *xyz_host, const int *Ns, int B, int Q, int k, float radius,
                           int max_step, int *const *seeds_host, float *const *geo_host, void *workspace,
                           size_t workspace_bytes, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* GEOFORMER_B200_H */
