// (a) Core contraction for a batch of (subject, relation) queries and its backward.
//
// Forward replaces reference src/model/asymmetric/R_TuckER.py:45-46 (and symmetric:42-43):
//   einsum("abc,da->dbc") materialises B x r1 x r2 (328 MB at rank 2r on WN18RR) and a bmm
//   reduces it; here q[b,:] = sum_{a,i} r[b,a] s[b,i] core[a,i,:] is ONE GEMM whose left operand
//   r[b,a]*s[b,i] is generated on the fly (never stored), K = r0*r1, split-K for occupancy.
// Backward is what autograd would compute for those two lines.
// Pair contraction (relation prediction, (s, ?, o)): t[b,a] = sum_{i,j} core[a,i,j] s[b,i] o[b,j], the same GEMM with
// K = r1*r2, the left operand s[b,i]*o[b,j] generated on the fly and the core read in place (no permuted copy); its
// backward (the relation-prediction training term) is the query backward's two kernels with the same folding.
//
// FP32 FFMA, deterministic (split partials reduced in a fixed order).
// Flops: fwd 2*B*r0*r1*r2, bwd 3x that.  Bytes: core once per pass (L2 resident) + rows.
#include "common.h"

namespace {

constexpr int T = 64;    // tile edge
constexpr int KC = 16;   // k chunk
using Smem = float[KC][T + 4];

// acc[4][4] += A[row, k] * B[k, col] for k in [kbeg, kend); la(row,k), lb(k,col) return 0 out of range.
template <bool A_LANES_ALONG_K, bool B_LANES_ALONG_N, class LA, class LB>
__device__ __forceinline__ void tile_mainloop(int kbeg, int kend, LA la, LB lb, float (&acc)[4][4],
                                              Smem& As, Smem& Bs) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  for (int k0 = kbeg; k0 < kend; k0 += KC) {
#pragma unroll
    for (int it = 0; it < (T * KC) / 256; ++it) {
      const int e = it * 256 + threadIdx.x;
      int rr, kk;
      if (A_LANES_ALONG_K) { rr = e / KC; kk = e % KC; } else { kk = e / T; rr = e % T; }
      As[kk][rr] = (k0 + kk < kend) ? la(rr, k0 + kk) : 0.0f;
      int cc, k2;
      if (B_LANES_ALONG_N) { k2 = e / T; cc = e % T; } else { cc = e / KC; k2 = e % KC; }
      Bs[k2][cc] = (k0 + k2 < kend) ? lb(k0 + k2, cc) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < KC; ++kk) {
      const float4 av = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[4] = {av.x, av.y, av.z, av.w};
      const float b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
}

__device__ __forceinline__ void zero_acc(float (&acc)[4][4]) {
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;
}

// ---- forward: partial[split][b][j] = sum_{k in split} r[b,a(k)] s[b,i(k)] core[k, j] ----------
__global__ void __launch_bounds__(256)
query_fwd_kernel(const float* __restrict__ core, const float* __restrict__ r_rows,
                 const float* __restrict__ s_rows, int B, int r0, int r1, int r2, int k_per_split,
                 float* __restrict__ partial) {
  __shared__ Smem As, Bs;
  const int b0 = blockIdx.x * T, j0 = blockIdx.y * T, split = blockIdx.z;
  const int K = r0 * r1;
  const int kbeg = split * k_per_split, kend = min(K, kbeg + k_per_split);
  float acc[4][4];
  zero_acc(acc);
  auto la = [&](int rr, int k) -> float {
    const int b = b0 + rr;
    if (b >= B) return 0.0f;
    const int a = k / r1, i = k - a * r1;
    return __ldg(r_rows + (int64_t)b * r0 + a) * __ldg(s_rows + (int64_t)b * r1 + i);
  };
  auto lb = [&](int k, int cc) -> float {
    const int j = j0 + cc;
    return (j < r2) ? __ldg(core + (int64_t)k * r2 + j) : 0.0f;
  };
  tile_mainloop<true, true>(kbeg, kend, la, lb, acc, As, Bs);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = b0 + ty * 4 + i;
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int jj = j0 + tx * 4 + j;
      if (jj < r2) partial[((int64_t)split * B + b) * r2 + jj] = acc[i][j];
    }
  }
}

// ---- pair contraction: partial[split][b][a] = sum_{k=(i,j) in split} s[b,i] o[b,j] core[a*K + k] ---------
// The relation-mode query of (s, ?, o).  Same loop as query_fwd_kernel run on the core permuted to (r1, r2, r0), with
// the permutation folded into the B operand's addressing (lanes along K: core[a, :, :] is contiguous in k), so the
// products and the order they are added in are those of rt_query_fwd on that permuted core.
__global__ void __launch_bounds__(256)
pair_fwd_kernel(const float* __restrict__ core, const float* __restrict__ s_rows,
                const float* __restrict__ o_rows, int B, int r0, int r1, int r2, int k_per_split,
                float* __restrict__ partial) {
  __shared__ Smem As, Bs;
  const int b0 = blockIdx.x * T, a0 = blockIdx.y * T, split = blockIdx.z;
  const int K = r1 * r2;
  const int kbeg = split * k_per_split, kend = min(K, kbeg + k_per_split);
  float acc[4][4];
  zero_acc(acc);
  auto la = [&](int rr, int k) -> float {
    const int b = b0 + rr;
    if (b >= B) return 0.0f;
    const int i = k / r2, j = k - i * r2;
    return __ldg(s_rows + (int64_t)b * r1 + i) * __ldg(o_rows + (int64_t)b * r2 + j);
  };
  auto lb = [&](int k, int cc) -> float {
    const int a = a0 + cc;
    return (a < r0) ? __ldg(core + (int64_t)a * K + k) : 0.0f;
  };
  tile_mainloop<true, false>(kbeg, kend, la, lb, acc, As, Bs);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = b0 + ty * 4 + i;
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int a = a0 + tx * 4 + j;
      if (a < r0) partial[((int64_t)split * B + b) * r0 + a] = acc[i][j];
    }
  }
}

__global__ void reduce_splits_kernel(const float* __restrict__ partial, int nsplit, int64_t count,
                                     float* __restrict__ out) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float s = 0.0f;
  for (int k = 0; k < nsplit; ++k) s += partial[(int64_t)k * count + i];
  out[i] = s;
}

// ---- backward (1): d_core[k=(a,i), j] = sum_b r[b,a] s[b,i] H[b,j] ----------------------------
// grid.z splits the batch (few k x j tiles at small ranks: 128 CTAs walked all 512 rows, 98 us); the partial sums are
// added in split order by reduce_splits_kernel
// PAIR: the backward of the pair contraction, run as this kernel on the core permuted to (r1, r2, r0) (so r0, r1, r2
// here are the permuted extents); only the store addressing differs: element (k, j) of the permuted core's gradient is
// written where the unpermuted core keeps it, d_core[j * K + k].
template <bool PAIR>
__global__ void __launch_bounds__(256)
query_bwd_core_kernel(const float* __restrict__ r_rows, const float* __restrict__ s_rows,
                      const float* __restrict__ H, int B, int r0, int r1, int r2, int b_per_split,
                      float* __restrict__ d_core) {
  __shared__ Smem As, Bs;
  const int k0 = blockIdx.x * T, j0 = blockIdx.y * T;
  const int K = r0 * r1;
  const int bbeg = blockIdx.z * b_per_split, bend = min(B, bbeg + b_per_split);
  d_core += (int64_t)blockIdx.z * K * r2;
  float acc[4][4];
  zero_acc(acc);
  auto la = [&](int rr, int b) -> float {  // A[row=k, kdim=b]
    const int k = k0 + rr;
    if (k >= K) return 0.0f;
    const int a = k / r1, i = k - a * r1;
    return __ldg(r_rows + (int64_t)b * r0 + a) * __ldg(s_rows + (int64_t)b * r1 + i);
  };
  auto lb = [&](int b, int cc) -> float {
    const int j = j0 + cc;
    return (j < r2) ? __ldg(H + (int64_t)b * r2 + j) : 0.0f;
  };
  tile_mainloop<false, true>(bbeg, bend, la, lb, acc, As, Bs);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int k = k0 + ty * 4 + i;
    if (k >= K) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int jj = j0 + tx * 4 + j;
      if (jj < r2) d_core[PAIR ? (int64_t)jj * K + k : (int64_t)k * r2 + jj] = acc[i][j];
    }
  }
}

// ---- backward (2): Y_a[b,i] = sum_j H[b,j] core[a,i,j];  ds[b,i] += r[b,a] Y_a;  dr[b,a] = sum_i s[b,i] Y_a
// grid (b tiles, i tiles, a splits).  ds partial per a-split, dr partial per i-tile.
// PAIR: as query_bwd_core_kernel<true>, the permuted core (r0, r1, r2 its extents) read in place: element (a, i, j) of
// the permuted core is core[(j * r0 + a) * r1 + i], contiguous along i, so the B operand's lanes run along i.
template <bool PAIR>
__global__ void __launch_bounds__(256)
query_bwd_rows_kernel(const float* __restrict__ core, const float* __restrict__ r_rows,
                      const float* __restrict__ s_rows, const float* __restrict__ H, int B, int r0,
                      int r1, int r2, int a_per_split, float* __restrict__ ds_partial,
                      float* __restrict__ dr_partial) {
  __shared__ Smem As, Bs;
  const int b0 = blockIdx.x * T, i0 = blockIdx.y * T, split = blockIdx.z;
  const int abeg = split * a_per_split, aend = min(r0, abeg + a_per_split);
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  float ds[4][4];
  zero_acc(ds);
  float sv[4][4];  // s[b,i] for this thread's micro-tile
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int b = b0 + ty * 4 + i, ii = i0 + tx * 4 + j;
      sv[i][j] = (b < B && ii < r1) ? __ldg(s_rows + (int64_t)b * r1 + ii) : 0.0f;
    }
  auto la = [&](int rr, int j) -> float {  // H[b, j]
    const int b = b0 + rr;
    return (b < B) ? __ldg(H + (int64_t)b * r2 + j) : 0.0f;
  };
  for (int a = abeg; a < aend; ++a) {
    float y[4][4];
    zero_acc(y);
    auto lb = [&](int j, int cc) -> float {  // core[a, i0+cc, j]
      const int ii = i0 + cc;
      if (ii >= r1) return 0.0f;
      return __ldg(core + (PAIR ? ((int64_t)j * r0 + a) * r1 + ii : ((int64_t)a * r1 + ii) * r2 + j));
    };
    tile_mainloop<true, PAIR>(0, r2, la, lb, y, As, Bs);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int b = b0 + ty * 4 + i;
      const float rv = (b < B) ? __ldg(r_rows + (int64_t)b * r0 + a) : 0.0f;
      float part = 0.0f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        ds[i][j] = fmaf(rv, y[i][j], ds[i][j]);
        part = fmaf(sv[i][j], y[i][j], part);
      }
      // reduce over the 16 tx lanes that share this row (lanes differ in the low 4 bits)
#pragma unroll
      for (int o = 8; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
      if (tx == 0 && b < B) dr_partial[((int64_t)blockIdx.y * B + b) * r0 + a] = part;
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = b0 + ty * 4 + i;
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int ii = i0 + tx * 4 + j;
      if (ii < r1) ds_partial[((int64_t)split * B + b) * r1 + ii] = ds[i][j];
    }
  }
}

struct QueryPlan {
  int ksplit, k_per_split;  // forward split-K
  int asplit, a_per_split;  // backward split over the relation rank
  int itiles;
  int bsplit, b_per_split;  // core-gradient split over the batch
};

QueryPlan query_plan(int B, int r0, int r1, int r2) {
  QueryPlan p;
  const int K = r0 * r1;
  const int tiles = rt::cdiv(B, T) * rt::cdiv(r2, T);
  int ks = rt::cdiv(2 * 148, tiles);
  const int max_ks = rt::cdiv(K, 4 * KC);
  if (ks > max_ks) ks = max_ks;
  if (ks < 1) ks = 1;
  p.k_per_split = rt::cdiv(rt::cdiv(K, ks), KC) * KC;
  p.ksplit = rt::cdiv(K, p.k_per_split);
  p.itiles = rt::cdiv(r1, T);
  const int tiles2 = rt::cdiv(B, T) * p.itiles;
  int as = rt::cdiv(2 * 148, tiles2);
  if (as > r0) as = r0;
  if (as < 1) as = 1;
  p.a_per_split = rt::cdiv(r0, as);
  p.asplit = rt::cdiv(r0, p.a_per_split);
  const int tiles3 = rt::cdiv(K, T) * rt::cdiv(r2, T);
  int bs = rt::cdiv(2 * 148, tiles3);
  if (bs > rt::cdiv(B, 4 * KC)) bs = rt::cdiv(B, 4 * KC);
  if (bs < 1) bs = 1;
  p.b_per_split = rt::cdiv(rt::cdiv(B, bs), KC) * KC;
  p.bsplit = rt::cdiv(B, p.b_per_split);
  return p;
}

// rt_query_bwd on (core, r_rows, s_rows, H) with extents (r0, r1, r2); PAIR: core is the unpermuted core of the pair
// contraction and (r0, r1, r2) the extents of its permutation (r1, r2, r0), d_core is written unpermuted.
template <bool PAIR>
int query_bwd(const float* core, const float* r_rows, const float* s_rows, const float* H, int B, int r0, int r1,
              int r2, float* d_core, float* ds_rows, float* dr_rows, void* ws, cudaStream_t s) {
  QueryPlan p = query_plan(B, r0, r1, r2);
  float* ds_partial = (float*)ws;
  float* dr_partial = ds_partial + (size_t)p.asplit * B * r1;
  {
    float* core_partial = dr_partial + (size_t)p.itiles * B * r0;
    dim3 grid(rt::cdiv(r0 * r1, T), rt::cdiv(r2, T), p.bsplit);
    query_bwd_core_kernel<PAIR><<<grid, 256, 0, s>>>(r_rows, s_rows, H, B, r0, r1, r2, p.b_per_split,
                                                     p.bsplit > 1 ? core_partial : d_core);
    RT_LAUNCH_CHECK();
    if (p.bsplit > 1) {
      const int64_t cc = (int64_t)r0 * r1 * r2;
      reduce_splits_kernel<<<(int)((cc + 255) / 256), 256, 0, s>>>(core_partial, p.bsplit, cc, d_core);
      RT_LAUNCH_CHECK();
    }
  }
  {
    dim3 grid(rt::cdiv(B, T), p.itiles, p.asplit);
    query_bwd_rows_kernel<PAIR><<<grid, 256, 0, s>>>(core, r_rows, s_rows, H, B, r0, r1, r2,
                                                     p.a_per_split, ds_partial, dr_partial);
    RT_LAUNCH_CHECK();
  }
  const int64_t c1 = (int64_t)B * r1, c0 = (int64_t)B * r0;
  reduce_splits_kernel<<<(int)((c1 + 255) / 256), 256, 0, s>>>(ds_partial, p.asplit, c1, ds_rows);
  RT_LAUNCH_CHECK();
  reduce_splits_kernel<<<(int)((c0 + 255) / 256), 256, 0, s>>>(dr_partial, p.itiles, c0, dr_rows);
  RT_LAUNCH_CHECK();
  return 0;
}

}  // namespace

extern "C" size_t rt_query_ws_bytes(int B, int r0, int r1, int r2) {
  if (B <= 0) return 16;
  QueryPlan p = query_plan(B, r0, r1, r2);
  size_t fwd = (size_t)p.ksplit * B * r2;
  size_t bwd = (size_t)p.asplit * B * r1 + (size_t)p.itiles * B * r0 + (p.bsplit > 1 ? (size_t)p.bsplit * r0 * r1 * r2 : 0);
  return sizeof(float) * (fwd > bwd ? fwd : bwd);
}

extern "C" int rt_query_fwd(const float* core, const float* r_rows, const float* s_rows, int B, int r0,
                            int r1, int r2, float* q, void* ws, void* stream) {
  RT_REQUIRE(B >= 0 && r0 > 0 && r1 > 0 && r2 > 0, "rt_query_fwd: bad shape");
  if (B == 0) return 0;
  RT_REQUIRE(ws != nullptr, "rt_query_fwd: workspace is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  QueryPlan p = query_plan(B, r0, r1, r2);
  dim3 grid(rt::cdiv(B, T), rt::cdiv(r2, T), p.ksplit);
  query_fwd_kernel<<<grid, 256, 0, s>>>(core, r_rows, s_rows, B, r0, r1, r2, p.k_per_split,
                                        (float*)ws);
  RT_LAUNCH_CHECK();
  const int64_t count = (int64_t)B * r2;
  reduce_splits_kernel<<<(int)((count + 255) / 256), 256, 0, s>>>((const float*)ws, p.ksplit, count, q);
  RT_LAUNCH_CHECK();
  return 0;
}

// The split plan of the permuted core (r1, r2, r0): the plan, and so the partial sums, of rt_query_fwd / rt_query_bwd
// there.  The workspace covers both passes.
extern "C" size_t rt_pair_ws_bytes(int B, int r0, int r1, int r2) { return rt_query_ws_bytes(B, r1, r2, r0); }

extern "C" int rt_pair_fwd(const float* core, const float* s_rows, const float* o_rows, int B, int r0, int r1,
                           int r2, float* t, void* ws, void* stream) {
  RT_REQUIRE(B >= 0 && r0 > 0 && r1 > 0 && r2 > 0, "rt_pair_fwd: bad shape");
  if (B == 0) return 0;
  RT_REQUIRE(ws != nullptr, "rt_pair_fwd: workspace is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  QueryPlan p = query_plan(B, r1, r2, r0);
  dim3 grid(rt::cdiv(B, T), rt::cdiv(r0, T), p.ksplit);
  pair_fwd_kernel<<<grid, 256, 0, s>>>(core, s_rows, o_rows, B, r0, r1, r2, p.k_per_split, (float*)ws);
  RT_LAUNCH_CHECK();
  const int64_t count = (int64_t)B * r0;
  reduce_splits_kernel<<<(int)((count + 255) / 256), 256, 0, s>>>((const float*)ws, p.ksplit, count, t);
  RT_LAUNCH_CHECK();
  return 0;
}

extern "C" int rt_query_bwd(const float* core, const float* r_rows, const float* s_rows,
                            const float* H, int B, int r0, int r1, int r2, float* d_core,
                            float* ds_rows, float* dr_rows, void* ws, void* stream) {
  RT_REQUIRE(B > 0 && r0 > 0 && r1 > 0 && r2 > 0, "rt_query_bwd: bad shape");
  RT_REQUIRE(ws != nullptr, "rt_query_bwd: workspace is NULL");
  return query_bwd<false>(core, r_rows, s_rows, H, B, r0, r1, r2, d_core, ds_rows, dr_rows, ws,
                          (cudaStream_t)stream);
}

// rt_query_bwd of the permuted core (r1, r2, r0) with (s_rows, o_rows) in place of (r_rows, s_rows): its ds is do, its
// dr is ds.
extern "C" int rt_pair_bwd(const float* core, const float* s_rows, const float* o_rows, const float* H_t, int B,
                           int r0, int r1, int r2, float* d_core, float* ds_rows, float* do_rows, void* ws,
                           void* stream) {
  RT_REQUIRE(B >= 0 && r0 > 0 && r1 > 0 && r2 > 0, "rt_pair_bwd: bad shape");
  if (B == 0) return 0;
  RT_REQUIRE(ws != nullptr, "rt_pair_bwd: workspace is NULL");
  return query_bwd<true>(core, s_rows, o_rows, H_t, B, r1, r2, r0, d_core, do_rows, ds_rows, ws,
                         (cudaStream_t)stream);
}
