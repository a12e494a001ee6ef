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

// ordered-uint row maxima (Q) of the (Q,N) maps and their global maximum, or row_max (Q) imported (gf_bias.cu);
// vec: N % 4 == 0 and geo 16-byte aligned
int bias_mask_rowmax(const float *geo, int Q, int N, const float *row_max, bool vec, uint32_t *rowmax, uint32_t *gmax,
                     cudaStream_t st);

}  // namespace gf
