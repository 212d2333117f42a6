// The exact fp32 arithmetic of a score, defined once.
//
//   logit      z = q . o        one fmaf accumulator, k ascending (exact_logit; the 64 x 64 FFMA tile of score_bce.cu)
//   BCE        p = 1 / (1 + expf(-z)), log p and log(1 - p) clamped at -100 as nn.BCELoss does,
//              dL/dz = (p - t) / max(p (1 - p), 1e-12) * inv * p (1 - p)
//   softmax    2^((z - M) log2e - log2 S) with one ex2.approx, loss term t (log2 S ln 2 - (z - M))
//
// Ranks and top-k lists are counts of comparisons (p > p_t, p == p_t), so a difference in the last bit turns a tie
// into a win.  Every kernel below therefore agrees bit for bit with rt_score_dense / rt_score_dense_logits
// (score_dense_kernel) by using these functions and nothing else for the element arithmetic:
//   score_bce.cu  score_kernel (fp32 filtered ranking, variant-0 BCE / CE training), score_lse_kernel (logits of the
//                 CE log-sum-exp pass) and target_prob_kernel (p_target, the value ties are taken against);
//   apply_tc.cu   rank_candidates_kernel and rank_filter_fix_kernel, which recompute the entities the tensor-core
//                 ranking could not classify, and score_fix_positives_kernel / score_ce_fix_positives_kernel, which
//                 patch the positives of the tensor-core BCE and CE passes with score_kernel's values;
//   topk.cu       the exact pass of the top-k selection;  rank_logit.cu  the exact pass of the logit-space ranking.
// The tensor-core CE epilogue ce_chunk8 applies the same softmax element to its tensor-core logits.  The BCE epilogues
// rank_chunk8 / score_chunk8 reach 1e-5 parity through different, branch-free arithmetic and are not bound by this.
// None of these files may be built with fast-math: expf, logf and log1pf are the accurate ones.
#pragma once
#include <math.h>
#include <stdint.h>

namespace rt {

constexpr float kLog2e = 1.4426950408889634f, kLn2 = 0.6931471805599453f;

// the approximate special-function units (ftz): 2^x, log2 x, 1 / x; the softmax element and the branch-free BCE
// epilogues of apply_tc.cu and score_bce_v3.cu use these
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

__device__ __forceinline__ float exact_logit(const float* __restrict__ q, const float* __restrict__ o, int r2) {
  float z = 0.0f;
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

// log p and log(1 - p), clamped at -100
__device__ __forceinline__ float bce_log_p(float p) { return fmaxf(logf(p), -100.0f); }
__device__ __forceinline__ float bce_log_q(float p) { return fmaxf(log1pf(-p), -100.0f); }
// target t, inv = the loss's 1 / count; the guard keeps the gradient finite where p (1 - p) underflows
__device__ __forceinline__ float bce_grad(float p, float t, float inv) {
  const float pq = (1.0f - p) * p;
  return (p - t) / fmaxf(pq, 1e-12f) * inv * pq;
}

// d = z - M_b, log2S = log2 S_b of the row statistics (ce_row_stats)
__device__ __forceinline__ float ce_softmax(float d, float log2S) { return ex2_approx(fmaf(d, kLog2e, -log2S)); }
__device__ __forceinline__ float ce_loss_term(float t, float d, float log2S) { return t * fmaf(log2S, kLn2, -d); }

}  // namespace rt
