// The exact fp32 arithmetic of the dense scores (score_dense_kernel / target_prob_kernel): one fmaf accumulator,
// k ascending, then 1 / (1 + expf(-z)).  Kernels that recheck a tensor-core classification (rank mode, top-k
// selection) recompute single probabilities with these so that they are bit-identical to rt_score_dense.
#pragma once
#include <stdint.h>

namespace rt {

__device__ __forceinline__ float exact_logit(const float* __restrict__ q, const float* __restrict__ o, int r2) {
  float z = 0.0f;                                   // same order as score_dense_kernel / target_prob_kernel
  int k = 0;
  if ((r2 & 3) == 0 && ((reinterpret_cast<uintptr_t>(q) | reinterpret_cast<uintptr_t>(o)) & 15u) == 0) {
    // 16-byte loads, eight in flight per operand: one thread walks one row, so the chain is bound by its own loads
    for (; k + 32 <= r2; k += 32) {
      float4 a[8], b[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) { a[u] = __ldg(reinterpret_cast<const float4*>(q + k) + u); b[u] = __ldg(reinterpret_cast<const float4*>(o + k) + u); }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        z = fmaf(a[u].x, b[u].x, z); z = fmaf(a[u].y, b[u].y, z); z = fmaf(a[u].z, b[u].z, z); z = fmaf(a[u].w, b[u].w, z);
      }
    }
    for (; k + 4 <= r2; k += 4) {
      const float4 a = __ldg(reinterpret_cast<const float4*>(q + k)), b = __ldg(reinterpret_cast<const float4*>(o + k));
      z = fmaf(a.x, b.x, z); z = fmaf(a.y, b.y, z); z = fmaf(a.z, b.z, z); z = fmaf(a.w, b.w, z);
    }
  }
  for (; k < r2; ++k) z = fmaf(__ldg(q + k), __ldg(o + k), z);
  return z;
}
__device__ __forceinline__ float sigmoid_ref(float z) { return 1.0f / (1.0f + expf(-z)); }

}  // namespace rt
