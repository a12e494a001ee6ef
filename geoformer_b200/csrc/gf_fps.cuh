// Internal interface of the culled FPS on the kNN grid's cell order (shared with the batched hot path in gf_guidance.cu).
#pragma once
#include "gf_common.cuh"

namespace gf {

// the running minima of one scene: N floats in cell order
size_t fps_cells_workspace_bytes(int N);
// The m seeds of one scene (original indices, the reference's seeds bit for bit) from its points in cell order
// (KnnGridBuffers::sorted); xyz (N,3) gives seed 0.  One CTA, one launch.
int fps_cells(const float4 *sorted, const float *xyz, int N, int m, void *workspace, size_t workspace_bytes, int *idx,
              cudaStream_t st);

}  // namespace gf
