// Filtered ranking in logit space (rt_score_rank_logit) and the target's exact logit (rt_target_logit).
//
// For query b with target t and filter list F_b, z_bj the exact fp32 logit of exact.cuh (bit-identical to
// rt_score_dense_logits):
//   greater      = #{ j not in F_b + {t} : z_bj >  z_bt }
//   equal        = #{ j not in F_b + {t} : z_bj == z_bt },   equal_before = the same restricted to j < t
//   pos_sum      = sum_{j in F_b} z_bj  (double, for the cross-entropy evaluation loss)
// Filtered entities are REMOVED, not set to a score of 0 as in probability space (0 is an ordinary logit).
//
// Counting runs over every entity of the shard except the target, then the filter list is taken back out:
//   - tensor-core path (apply_tc.cu, rank_tc_logit): the rank mode of apply_tc_kernel with logit thresholds; the band's
//     candidates are recounted from their exact logits;
//   - exact path: logits over entity chunks staged in the workspace (score_dense_kernel<true>), counted by
//     rank_logit_count_kernel.  It is the whole path for thin ranks and short shards, and runs gated on a device flag
//     (no host synchronisation) when the tensor-core candidate list overflowed;
//   - removal: rank_logit_filter_kernel, kSlices CTAs per query, each a fixed interleaved share of the query's filter
//     entries (a 3000-entry hub query takes 3000 / (kSlices * 128) exact logits per thread instead of being the
//     critical path), with the positive logits summed in a fixed order (no float atomics).
#include "common.h"
#include "exact.cuh"
#include <algorithm>
#include <math.h>

namespace {

constexpr int kMaxB = 65535, kMaxR2 = 256;
constexpr int kSeg = 2048;                  // entities of one staged row counted by one CTA
constexpr int kSlices = 8;                  // CTAs per query of the filter removal
constexpr int kFltThreads = 128;
constexpr size_t kChunkFloats = 1u << 22;   // staged logits of the exact pass (16 MB)

__global__ void target_logit_kernel(const float* __restrict__ q, const float* __restrict__ O, int B, int r2, int n_begin,
                                    int n_local, const int32_t* __restrict__ target, float* __restrict__ z_target) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int t = __ldg(target + b) - n_begin;
  z_target[b] = (t >= 0 && t < n_local) ? rt::exact_logit(q + (int64_t)b * r2, O + (int64_t)t * r2, r2) : 0.0f;
}

__device__ __forceinline__ void block_add_counts(int g, int e, int eb, int b, int32_t* greater, int32_t* equal,
                                                 int32_t* equal_before) {
  __shared__ int sg[32], se[32], sb[32];
  g = rt::warp_sum(g); e = rt::warp_sum(e); eb = rt::warp_sum(eb);
  const int w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  if ((threadIdx.x & 31) == 0) { sg[w] = g; se[w] = e; sb[w] = eb; }
  __syncthreads();
  if (threadIdx.x == 0) {
    int tg = 0, te = 0, tb = 0;
    for (int i = 0; i < nw; ++i) { tg += sg[i]; te += se[i]; tb += sb[i]; }
    // integer atomics: order-independent, deterministic
    if (tg) atomicAdd(greater + b, tg);
    if (te) atomicAdd(equal + b, te);
    if (tb) atomicAdd(equal_before + b, tb);
  }
}

// exact path: counts of the staged logits Z[b][0, len) of entities id0 .. id0 + len - 1 against z_target[b], the
// target excluded.  gate == NULL: always; else a no-op unless *gate != 0.
__global__ void __launch_bounds__(256)
rank_logit_count_kernel(const float* __restrict__ Z, int64_t ldz, int len, int id0, const int32_t* __restrict__ target,
                        const float* __restrict__ z_target, const int* __restrict__ gate, int32_t* greater,
                        int32_t* equal, int32_t* equal_before) {
  if (gate && *gate == 0) return;
  const int b = blockIdx.y;
  const int j0 = blockIdx.x * kSeg, j1 = min(len, j0 + kSeg);
  const float* zb = Z + (int64_t)b * ldz;
  const float zt = __ldg(z_target + b);
  const int t = __ldg(target + b);
  int g = 0, e = 0, eb = 0;
  for (int i = j0 + threadIdx.x; i < j1; i += blockDim.x) {
    const int j = id0 + i;
    if (j == t) continue;
    const float z = __ldg(zb + i);
    const int eq = z == zt;
    g += z > zt;
    e += eq;
    eb += eq & (j < t);
  }
  block_add_counts(g, e, eb, b, greater, equal, equal_before);
}

// removal of the filter list from the counts, and the per-slice sums of the positive logits (part may be NULL)
__global__ void __launch_bounds__(kFltThreads)
rank_logit_filter_kernel(const float* __restrict__ q, const float* __restrict__ O, int r2, int n_begin, int n_local,
                         const int32_t* __restrict__ target, const float* __restrict__ z_target,
                         const int32_t* __restrict__ flt_off, const int32_t* __restrict__ flt_idx, int32_t* greater,
                         int32_t* equal, int32_t* equal_before, double* __restrict__ part) {
  const int b = blockIdx.y, slice = blockIdx.x;
  const int f0 = __ldg(flt_off + b), f1 = __ldg(flt_off + b + 1);
  const int t = __ldg(target + b);
  const float zt = __ldg(z_target + b);
  const float* qb = q + (int64_t)b * r2;
  int g = 0, e = 0, eb = 0;
  double pos = 0.0;
  for (int i = f0 + slice * kFltThreads + threadIdx.x; i < f1; i += kSlices * kFltThreads) {
    const int f = __ldg(flt_idx + i), fl = f - n_begin;
    if (fl < 0 || fl >= n_local) continue;
    const float z = rt::exact_logit(qb, O + (int64_t)fl * r2, r2);
    pos += (double)z;
    if (f == t) continue;
    const int eq = z == zt;
    g -= z > zt;
    e -= eq;
    eb -= eq & (f < t);
  }
  block_add_counts(g, e, eb, b, greater, equal, equal_before);   // (synchronises the block)
  if (!part) return;
  __shared__ double sp[kFltThreads / 32];
  pos = rt::warp_sum(pos);
  if ((threadIdx.x & 31) == 0) sp[threadIdx.x >> 5] = pos;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kFltThreads / 32; ++w) s += sp[w];
    part[(int64_t)b * kSlices + slice] = s;
  }
}

__global__ void pos_sum_finish_kernel(const double* __restrict__ part, int B, double* __restrict__ pos_sum) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  double s = 0.0;
#pragma unroll
  for (int i = 0; i < kSlices; ++i) s += part[(int64_t)b * kSlices + i];
  pos_sum[b] = s;
}

struct RankLogitLayout {
  size_t part, chunk, tc, total;
  int chunk_len, nchunks;
  bool use_tc;
};
RankLogitLayout rank_logit_layout(int B, int n_local, int r2) {
  RankLogitLayout L;
  B = std::max(B, 1); n_local = std::max(n_local, 0);
  L.use_tc = rt::rank_tc_supported(B, n_local, r2);
  L.chunk_len = (int)std::min<size_t>(std::max<size_t>(kChunkFloats / (size_t)B / 64 * 64, 64),
                                      (size_t)rt::align_up((size_t)std::max(n_local, 1), 64));
  L.nchunks = std::max(1, rt::cdiv(n_local, L.chunk_len));
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += rt::align_up(bytes, 256); return at; };
  L.part = take(sizeof(double) * (size_t)B * kSlices);
  L.chunk = take(sizeof(float) * (size_t)B * L.chunk_len);
  L.tc = L.use_tc ? take(rt::rank_tc_ws_bytes(B, n_local, r2)) : o;
  L.total = o;
  return L;
}

}  // namespace

extern "C" int rt_target_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                               const int32_t* target, float* z_target, void* stream) {
  RT_REQUIRE(B >= 0 && r2 > 0 && n_local >= 0, "rt_target_logit: bad shape B=%d r2=%d n_local=%d", B, r2, n_local);
  if (B == 0) return 0;
  target_logit_kernel<<<rt::cdiv(B, 128), 128, 0, (cudaStream_t)stream>>>(q, O, B, r2, n_begin, n_local, target,
                                                                          z_target);
  RT_LAUNCH_CHECK();
  return 0;
}

extern "C" size_t rt_score_rank_logit_ws_bytes(int B, int n_local, int r2) { return rank_logit_layout(B, n_local, r2).total; }

extern "C" int rt_score_rank_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                                   const int32_t* target, const float* z_target, const int32_t* flt_off,
                                   const int32_t* flt_idx, int32_t* greater, int32_t* equal, int32_t* equal_before,
                                   double* pos_sum, void* ws, void* stream) {
  RT_REQUIRE(B >= 1 && B <= kMaxB, "rt_score_rank_logit: B=%d outside 1..%d queries per call", B, kMaxB);
  RT_REQUIRE(r2 >= 1 && r2 <= kMaxR2, "rt_score_rank_logit: r2=%d outside 1..%d", r2, kMaxR2);
  RT_REQUIRE(n_local >= 0 && n_begin >= 0, "rt_score_rank_logit: bad shard n_begin=%d n_local=%d", n_begin, n_local);
  RT_REQUIRE((flt_off == nullptr) == (flt_idx == nullptr),
             "rt_score_rank_logit: flt_off and flt_idx must both be NULL or both set");
  RT_REQUIRE(q && (O || n_local == 0) && target && z_target && greater && equal && equal_before,
             "rt_score_rank_logit: NULL input or output");
  RT_REQUIRE(ws != nullptr, "rt_score_rank_logit: workspace is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  const RankLogitLayout L = rank_logit_layout(B, n_local, r2);
  char* base = (char*)ws;
  RT_CHECK_CUDA(cudaMemsetAsync(greater, 0, sizeof(int32_t) * B, s));
  RT_CHECK_CUDA(cudaMemsetAsync(equal, 0, sizeof(int32_t) * B, s));
  RT_CHECK_CUDA(cudaMemsetAsync(equal_before, 0, sizeof(int32_t) * B, s));
  const int* gate = nullptr;
  if (L.use_tc) {
    int rc = rt::rank_tc_logit(q, O, B, r2, n_begin, n_local, target, z_target, greater, equal, equal_before,
                               base + L.tc, s, &gate);
    if (rc) return rc;
  }
  float* Z = (float*)(base + L.chunk);
  for (int c = 0; c < L.nchunks && n_local > 0; ++c) {
    const int c0 = c * L.chunk_len, len = std::min(L.chunk_len, n_local - c0);
    int rc = rt::score_dense(q, O + (int64_t)c0 * r2, B, r2, len, Z, L.chunk_len, gate, s, true);
    if (rc) return rc;
    rank_logit_count_kernel<<<dim3(rt::cdiv(len, kSeg), B), 256, 0, s>>>(Z, L.chunk_len, len, n_begin + c0, target,
                                                                       z_target, gate, greater, equal, equal_before);
    RT_LAUNCH_CHECK();
  }
  double* part = (double*)(base + L.part);
  if (flt_off) {
    rank_logit_filter_kernel<<<dim3(kSlices, B), kFltThreads, 0, s>>>(q, O, r2, n_begin, n_local, target, z_target,
                                                                      flt_off, flt_idx, greater, equal, equal_before,
                                                                      pos_sum ? part : nullptr);
    RT_LAUNCH_CHECK();
  } else if (pos_sum) {
    RT_CHECK_CUDA(cudaMemsetAsync(part, 0, sizeof(double) * (size_t)B * kSlices, s));
  }
  if (pos_sum) {
    pos_sum_finish_kernel<<<rt::cdiv(B, 128), 128, 0, s>>>(part, B, pos_sum);
    RT_LAUNCH_CHECK();
  }
  return 0;
}
