// Filtered top-k link prediction without the B x N probability matrix: for each query (s, r, ?) the k entities of the
// shard with the highest p = sigmoid(q_b . O_j), known objects excluded, ordered by p descending then global id
// ascending (the order of the ranking metrics, rank = 1 + greater + equal_before).  Probabilities are the exact fp32
// values of rt_score_dense.
//
//   1. sample threshold: exact p of a strided sample of m entities per query; p_k[b] = the k-th best of the sample.
//      The k-th best of a subset never beats the k-th best of the whole shard, so every entity of the true top k has
//      p >= p_k: the sample size only moves the candidate count, never the result.  A query whose sample holds
//      fewer than k unfiltered entities is flagged for the exact pass.
//   2. candidates: the tensor-core logits of the ranking path (apply_tc.cu, top-k mode) classified against the band
//      of p_k; every entity that is not certainly below p_k lands in the query's segment (fixed capacity).
//   3. selection: one CTA per query recomputes the candidates' p exactly, drops filtered ids and keeps the best k.
//      A query whose segment overflowed is flagged.
//   4. exact pass: exact p over entity chunks staged in the workspace (score_dense_kernel), merged into a running top k
//      per flagged query.  Gated on a device flag "some query is flagged", so it is a no-op when nothing overflowed.
//      It is the whole path where the tensor-core pass is not supported (thin ranks, shards under 1024 rows).
// Steps 1, 3 and 4 share one block-level top-k routine over 64-bit (p, id) keys.
//
// Logit space (rt_score_topk_logit): the same four steps on the exact fp32 logit z instead of p, instantiated with
// LOGIT = true: the key maps z's bit pattern order-preservingly (negative z included), the sample gives a logit
// threshold z_k and the tensor-core band is the logit band of apply_tc.cu (logit_thresholds_kernel).
#include "common.h"
#include "exact.cuh"
#include <algorithm>
#include <math.h>

namespace {

typedef unsigned long long u64;

constexpr int kMaxK = 256, kMaxB = 1024, kMaxR2 = 256;
constexpr int kThreads = 256;
constexpr int kBuf = 2048;                 // keys of one selection CTA: the running best k, then a batch of new ones
constexpr int kCap = 16384;                // candidate slots per query on the tensor-core path
constexpr size_t kChunkFloats = 1u << 22;  // staged probabilities of the exact pass (16 MB)

// Key of (p, id): larger key = earlier in the order (p descending, then id ascending).  p >= 0, so its bit pattern
// orders like the value; 0 is the empty key (id -1, p -inf), below every real one.
__device__ __forceinline__ u64 make_key(float p, int id) {
  return ((u64)(__float_as_uint(p) + 1u) << 32) | (u64)(0xffffffffu - (uint32_t)id);
}
__device__ __forceinline__ float key_p(u64 key) { return key ? __uint_as_float((uint32_t)(key >> 32) - 1u) : -INFINITY; }
__device__ __forceinline__ int key_id(u64 key) { return key ? (int)(0xffffffffu - (uint32_t)key) : -1; }

// Key of (z, id) for a logit of either sign: the bit pattern with the sign bit set for z >= +0 and all bits inverted for
// z < 0 orders like the value (-inf lowest); 0 stays the empty key (only the pattern 0xffffffff, a negative NaN, maps
// there).  -0 orders just below +0.
__device__ __forceinline__ u64 make_key_z(float z, int id) {
  const uint32_t b = __float_as_uint(z);
  return ((u64)((b & 0x80000000u) ? ~b : (b | 0x80000000u)) << 32) | (u64)(0xffffffffu - (uint32_t)id);
}
__device__ __forceinline__ float key_z(u64 key) {
  const uint32_t h = (uint32_t)(key >> 32);
  return key ? __uint_as_float((h & 0x80000000u) ? (h & 0x7fffffffu) : ~h) : -INFINITY;
}

// the score of an exact logit and its key: p = sigmoid(z) (rt_score_topk) or z itself (rt_score_topk_logit)
template <bool LOGIT> __device__ __forceinline__ float score_of(float z) { return LOGIT ? z : rt::sigmoid_ref(z); }
template <bool LOGIT> __device__ __forceinline__ u64 key_of_score(float v, int id) {
  return LOGIT ? make_key_z(v, id) : make_key(v, id);
}
template <bool LOGIT> __device__ __forceinline__ float score_of_key(u64 key) { return LOGIT ? key_z(key) : key_p(key); }

// id in the ascending filter list flt_idx[f0, f1)?
__device__ __forceinline__ bool filtered(const int32_t* __restrict__ flt_idx, int f0, int f1, int id) {
  while (f0 < f1) {
    const int mid = (f0 + f1) >> 1;
    const int v = __ldg(flt_idx + mid);
    if (v == id) return true;
    if (v < id) f0 = mid + 1; else f1 = mid;
  }
  return false;
}

// descending bitonic sort of s[0, kBuf)
__device__ void sort_desc(u64* s) {
  for (int size = 2; size <= kBuf; size <<= 1)
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = threadIdx.x; i < kBuf / 2; i += blockDim.x) {
        const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
        const u64 x = s[lo], y = s[hi];
        if ((x < y) == ((lo & size) == 0)) { s[lo] = y; s[hi] = x; }
      }
      __syncthreads();
    }
}

// The block-level top-k routine.  s[0, kp) holds the running best keys, descending (set, and synchronised, by the
// caller); merges key_of(0 .. n-1) into it.  Keys are distinct (ids are), so the result does not depend on the
// order in which the keys arrive.  A batch in which no key beats the current k-th is not sorted.
template <class KeyOf>
__device__ void topk_merge(u64* s, int kp, int n, KeyOf key_of) {
  const int room = kBuf - kp;
  for (int base = 0; base < n; base += room) {
    const u64 kth = s[kp - 1];
    int any = 0;
    for (int i = threadIdx.x; i < room; i += blockDim.x) {
      u64 v = base + i < n ? key_of(base + i) : 0ull;
      if (v <= kth) v = 0ull;
      any |= v != 0ull;
      s[kp + i] = v;
    }
    if (__syncthreads_or(any)) sort_desc(s);
  }
}

__device__ __forceinline__ void clear_keys(u64* s, int kp) {
  for (int i = threadIdx.x; i < kp; i += blockDim.x) s[i] = 0ull;
  __syncthreads();
}

template <bool LOGIT>
__device__ __forceinline__ void write_out(const u64* s, int k, int b, int32_t* top_idx, float* top_p) {
  for (int i = threadIdx.x; i < k; i += blockDim.x) {
    top_idx[(int64_t)b * k + i] = key_id(s[i]);
    top_p[(int64_t)b * k + i] = score_of_key<LOGIT>(s[i]);
  }
}

// 1. per query: the k-th best exact p among the unfiltered entities 0, stride, 2 stride, ... (m of them)
template <bool LOGIT>
__global__ void __launch_bounds__(kThreads)
topk_sample_kernel(const float* __restrict__ q, const float* __restrict__ O, int r2, int n_begin, int stride, int m,
                   int k, const int32_t* __restrict__ flt_off, const int32_t* __restrict__ flt_idx,
                   float* __restrict__ p_k, int* __restrict__ flag) {
  __shared__ u64 s[kBuf];
  const int b = blockIdx.x;
  const float* qb = q + (int64_t)b * r2;
  const int f0 = flt_off ? __ldg(flt_off + b) : 0, f1 = flt_off ? __ldg(flt_off + b + 1) : 0;
  clear_keys(s, k);
  topk_merge(s, k, m, [&](int i) {
    const int e = i * stride, id = n_begin + e;
    if (filtered(flt_idx, f0, f1, id)) return 0ull;
    return key_of_score<LOGIT>(score_of<LOGIT>(rt::exact_logit(qb, O + (int64_t)e * r2, r2)), id);
  });
  if (threadIdx.x == 0) {
    const u64 kth = s[k - 1];
    flag[b] = kth == 0ull;
    p_k[b] = kth ? score_of_key<LOGIT>(kth) : (LOGIT ? INFINITY : 1.0f);
  }
}

// 3. per query: exact p of the candidates, best k; flags the query when its segment overflowed
template <bool LOGIT>
__global__ void __launch_bounds__(kThreads)
topk_select_kernel(const float* __restrict__ q, const float* __restrict__ O, int r2, int n_begin, int k,
                   const int32_t* __restrict__ flt_off, const int32_t* __restrict__ flt_idx,
                   const int* __restrict__ cnt, const int32_t* __restrict__ seg, int cap, int* __restrict__ flag,
                   int* __restrict__ any_flag, int32_t* __restrict__ top_idx, float* __restrict__ top_p,
                   int32_t* __restrict__ n_cand) {
  __shared__ u64 s[kBuf];
  const int b = blockIdx.x;
  const int c = cnt[b];
  if (flag[b] || c > cap) {
    if (threadIdx.x == 0) { flag[b] = 1; *any_flag = 1; }
    return;
  }
  const float* qb = q + (int64_t)b * r2;
  const int32_t* sb = seg + (int64_t)b * cap;
  const int f0 = flt_off ? __ldg(flt_off + b) : 0, f1 = flt_off ? __ldg(flt_off + b + 1) : 0;
  clear_keys(s, k);
  topk_merge(s, k, c, [&](int i) {
    const int e = __ldg(sb + i), id = n_begin + e;
    if (filtered(flt_idx, f0, f1, id)) return 0ull;
    return key_of_score<LOGIT>(score_of<LOGIT>(rt::exact_logit(qb, O + (int64_t)e * r2, r2)), id);
  });
  write_out<LOGIT>(s, k, b, top_idx, top_p);
  if (n_cand && threadIdx.x == 0) n_cand[b] = c;
}

// 4. per query: merge the staged exact probabilities P[b][0, len) of entities id0 .. id0 + len - 1 into the running
//    best k (run[b]); the last chunk writes the outputs.  flag == NULL: every query; gate == NULL: always.
template <bool LOGIT>
__global__ void __launch_bounds__(kThreads)
topk_exact_merge_kernel(const float* __restrict__ P, int64_t ldp, int len, int id0, int k,
                        const int32_t* __restrict__ flt_off, const int32_t* __restrict__ flt_idx,
                        const int* __restrict__ flag, const int* __restrict__ gate, u64* __restrict__ run, int first,
                        int last, int32_t* __restrict__ top_idx, float* __restrict__ top_p,
                        int32_t* __restrict__ n_cand) {
  __shared__ u64 s[kBuf];
  const int b = blockIdx.x;
  if ((gate && *gate == 0) || (flag && flag[b] == 0)) return;
  u64* rb = run + (int64_t)b * k;
  if (first) clear_keys(s, k);
  else {
    for (int i = threadIdx.x; i < k; i += blockDim.x) s[i] = rb[i];
    __syncthreads();
  }
  const float* pb = P + (int64_t)b * ldp;
  const int f0 = flt_off ? __ldg(flt_off + b) : 0, f1 = flt_off ? __ldg(flt_off + b + 1) : 0;
  topk_merge(s, k, len, [&](int i) {
    const int id = id0 + i;
    if (filtered(flt_idx, f0, f1, id)) return 0ull;
    return key_of_score<LOGIT>(__ldg(pb + i), id);
  });
  if (last) {
    write_out<LOGIT>(s, k, b, top_idx, top_p);
    if (n_cand && threadIdx.x == 0) n_cand[b] = -1;
  } else {
    for (int i = threadIdx.x; i < k; i += blockDim.x) rb[i] = s[i];
  }
}

struct TopkLayout {
  size_t scal, pk, flag, cnt, run, chunk, tc, seg, total;
  int chunk_len, nchunks;
  bool use_tc;
};
TopkLayout topk_layout(int B, int n_local, int r2, int k) {
  TopkLayout L;
  B = std::max(B, 1); n_local = std::max(n_local, 0); k = std::max(k, 1);
  L.use_tc = rt::rank_tc_supported(B, n_local, r2);
  L.chunk_len = (int)std::min<size_t>(std::max<size_t>(kChunkFloats / (size_t)B / 64 * 64, 64),
                                      (size_t)rt::align_up((size_t)std::max(n_local, 1), 64));
  L.nchunks = std::max(1, rt::cdiv(n_local, L.chunk_len));
  rt::WsArena ws;
  L.scal = ws.take(256);                                // [0] some query is flagged
  L.pk = ws.take(sizeof(float) * B);
  L.flag = ws.take(sizeof(int) * B);
  L.cnt = ws.take(sizeof(int) * B);
  L.run = ws.take(sizeof(u64) * (size_t)B * k);
  L.chunk = ws.take(sizeof(float) * (size_t)B * L.chunk_len);
  L.tc = L.use_tc ? ws.take(rt::topk_tc_ws_bytes(B, n_local, r2)) : ws.o;
  L.seg = L.use_tc ? ws.take(sizeof(int32_t) * (size_t)B * kCap) : ws.o;
  L.total = ws.o;
  return L;
}

template <bool LOGIT>
int score_topk(const char* fn, const float* q, const float* O, int B, int r2, int n_begin, int n_local, int k,
               const int32_t* flt_off, const int32_t* flt_idx, int32_t* top_idx, float* top_p, int32_t* n_cand, void* ws,
               void* stream) {
  RT_REQUIRE(k >= 1 && k <= kMaxK, "%s: k=%d outside 1..%d", fn, k, kMaxK);
  RT_REQUIRE(B >= 1 && B <= kMaxB, "%s: B=%d outside 1..%d queries per call", fn, B, kMaxB);
  RT_REQUIRE(r2 >= 1 && r2 <= kMaxR2, "%s: r2=%d outside 1..%d", fn, r2, kMaxR2);
  RT_REQUIRE(n_local >= 0 && n_begin >= 0, "%s: bad shard n_begin=%d n_local=%d", fn, n_begin, n_local);
  RT_REQUIRE((flt_off == nullptr) == (flt_idx == nullptr), "%s: flt_off and flt_idx must both be NULL or both set", fn);
  RT_REQUIRE(q && (O || n_local == 0) && top_idx && top_p, "%s: NULL input or output", fn);
  RT_REQUIRE(ws != nullptr, "%s: workspace is NULL", fn);
  cudaStream_t s = (cudaStream_t)stream;
  const TopkLayout L = topk_layout(B, n_local, r2, k);
  char* base = (char*)ws;
  int* any_flag = (int*)(base + L.scal);
  int* flag = (int*)(base + L.flag);
  const int* gate = nullptr;
  if (L.use_tc) {
    float* p_k = (float*)(base + L.pk);
    int* cnt = (int*)(base + L.cnt);
    RT_CHECK_CUDA(cudaMemsetAsync(any_flag, 0, sizeof(int), s));
    RT_CHECK_CUDA(cudaMemsetAsync(cnt, 0, sizeof(int) * B, s));
    // sample size: about sqrt(k n) balances the sample against the expected k n / m candidates; at least 4 k n / cap
    // keeps the expected candidates at a quarter of a segment
    const double kn = (double)k * n_local;
    const double m_target = std::max({2.0 * sqrt(kn), 4.0 * kn / kCap, (double)k});
    const int stride = std::max(1, (int)(n_local / m_target));
    const int m = rt::cdiv(n_local, stride);
    topk_sample_kernel<LOGIT><<<B, kThreads, 0, s>>>(q, O, r2, n_begin, stride, m, k, flt_off, flt_idx, p_k, flag);
    RT_LAUNCH_CHECK();
    int32_t* seg = (int32_t*)(base + L.seg);
    int rc = rt::topk_tc_pass(q, O, B, r2, n_local, p_k, flag, cnt, seg, kCap, base + L.tc, s, LOGIT);
    if (rc) return rc;
    topk_select_kernel<LOGIT><<<B, kThreads, 0, s>>>(q, O, r2, n_begin, k, flt_off, flt_idx, cnt, seg, kCap, flag, any_flag,
                                              top_idx, top_p, n_cand);
    RT_LAUNCH_CHECK();
    gate = any_flag;
  }
  float* P = (float*)(base + L.chunk);
  u64* run = (u64*)(base + L.run);
  for (int c = 0; c < L.nchunks; ++c) {
    const int c0 = c * L.chunk_len, len = std::min(L.chunk_len, n_local - c0);
    int rc = rt::score_dense(q, O + (int64_t)c0 * r2, B, r2, len, P, L.chunk_len, gate, s, LOGIT);
    if (rc) return rc;
    topk_exact_merge_kernel<LOGIT><<<B, kThreads, 0, s>>>(P, L.chunk_len, len, n_begin + c0, k, flt_off, flt_idx,
                                                   L.use_tc ? flag : nullptr, gate, run, c == 0, c == L.nchunks - 1,
                                                   top_idx, top_p, n_cand);
    RT_LAUNCH_CHECK();
  }
  return 0;
}

}  // namespace

extern "C" size_t rt_score_topk_ws_bytes(int B, int n_local, int r2, int k) { return topk_layout(B, n_local, r2, k).total; }

extern "C" int rt_score_topk(const float* q, const float* O, int B, int r2, int n_begin, int n_local, int k,
                             const int32_t* flt_off, const int32_t* flt_idx, int32_t* top_idx, float* top_p,
                             int32_t* n_cand, void* ws, void* stream) {
  return score_topk<false>("rt_score_topk", q, O, B, r2, n_begin, n_local, k, flt_off, flt_idx, top_idx, top_p, n_cand,
                           ws, stream);
}

extern "C" int rt_score_topk_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local, int k,
                                   const int32_t* flt_off, const int32_t* flt_idx, int32_t* top_idx, float* top_z,
                                   int32_t* n_cand, void* ws, void* stream) {
  return score_topk<true>("rt_score_topk_logit", q, O, B, r2, n_begin, n_local, k, flt_off, flt_idx, top_idx, top_z,
                          n_cand, ws, stream);
}
