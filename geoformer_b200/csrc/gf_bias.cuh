// The mask-head epilogue's pieces shared by gf_bias.cu (a11, gf_bias_mask_head) and the fused mask head
// (gf_mask_head.cu), so that both make every "unreachable" decision with the same code.
#pragma once
#include "gf_common.cuh"

namespace gf {

__device__ __forceinline__ float mask_push(float d, float s, bool unreached) {
  // d + sqrt(rowmax) * sign(d) where the point is unreachable (:284-286); torch.sign: 0 -> 0, NaN -> NaN
  if (!unreached) return d;
  const float sg = d > 0.f ? 1.f : (d < 0.f ? -1.f : d);
  return __fadd_rn(d, __fmul_rn(s, sg));
}

// The workspace piece of the row maxima of `rows` maps, with their global maximum right after them so that one kernel
// can clear both.  Taken by the bias epilogues, the fused mask head and the fused cross-attention.
struct RowMax {
  uint32_t *rowmax, *gmax;
};
inline RowMax take_rowmax(Arena &a, size_t rows) {
  uint32_t *r = a.take<uint32_t>(rows + 1);
  return {r, r ? r + rows : nullptr};
}

// ordered-uint row maxima (B, Q) of the gathered maps and their global maximum (gf_bias.cu); geo_ptrs / geo_ld are
// HOST arrays
int bias_ctx_rowmax(const float *const *geo_ptrs, const int *geo_ld, const int *ctx_idx, int B, int Q, int C,
                    const RowMax &rm, cudaStream_t st);

// ordered-uint row maxima (Q) of the (Q,N) maps and their global maximum, or row_max (Q) imported (gf_bias.cu);
// vec: N % 4 == 0 and geo 16-byte aligned
int bias_mask_rowmax(const float *geo, int Q, int N, const float *row_max, bool vec, const RowMax &rm, cudaStream_t st);

// the (Q, N_b) maps of a batched mask head, up to 32 scenes (gf_mask_head.cu)
constexpr int MH_BATCH_MAX = 32;
struct MaskMaps {
  const float *geo[MH_BATCH_MAX];
  int N[MH_BATCH_MAX];
  int B, Q;
};

// ordered-uint row maxima (B, Q) of a batch's maps and each scene's own maximum of them, gmax (B), or row_max (B, Q)
// imported: one launch (after one zero fill when computed) for the whole batch (gf_bias.cu)
int bias_mask_rowmax_batch(const MaskMaps &maps, const float *row_max, uint32_t *rowmax, uint32_t *gmax,
                           cudaStream_t st);

}  // namespace gf
