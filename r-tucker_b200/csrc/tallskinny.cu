// Tall-skinny passes over the N x r factor matrices: Gram products, factor updates, row
// gather / scatter.  These carry every N-sized piece of the Riemannian projection, momentum
// transport and retraction (reference: tucker_riemopt grad / project / construct / round as
// called from src/model/asymmetric/optim.py:86-114 and src/model/symmetric/optim.py:80-107).
//
// Bound: HBM for thin ranks; at r ~ 200 the N x r x r products are FP32-FFMA bound
// (2*N*ra*rb flops per Gram, 2*N*rk*rc per update term).
#include "common.h"
#include <algorithm>

namespace {

// ------------------------------------------------------------------------------------------
// gather / scatter
// ------------------------------------------------------------------------------------------
__global__ void gather_rows_kernel(const float* __restrict__ table, int rows, int r, int row_begin,
                                   const int32_t* __restrict__ idx, float* __restrict__ out) {
  const int b = blockIdx.x;
  const int g = idx[b] - row_begin;
  const bool own = (g >= 0 && g < rows);
  for (int c = threadIdx.x; c < r; c += blockDim.x)
    out[(int64_t)b * r + c] = own ? __ldg(table + (int64_t)g * r + c) : 0.0f;
}

// One CTA per batch row; the first occurrence of an index is the leader and sums its
// duplicates in ascending batch order, so the result does not depend on scheduling.  The CTA scans the index list
// cooperatively (every thread walking all B indices twice cost 41 us per call at B = 512).
constexpr int kMaxDup = 64;
__global__ void scatter_rows_add_kernel(float* __restrict__ table, int rows, int r, int row_begin,
                                        const int32_t* __restrict__ idx, int B,
                                        const float* __restrict__ rows_in) {
  __shared__ int s_earlier, s_cnt, s_dup[kMaxDup];
  const int b = blockIdx.x;
  const int me = idx[b];
  const int g = me - row_begin;
  if (g < 0 || g >= rows) return;
  if (threadIdx.x == 0) { s_earlier = 0; s_cnt = 0; }
  __syncthreads();
  for (int bb = threadIdx.x; bb < B; bb += blockDim.x)
    if (__ldg(idx + bb) == me) {
      if (bb < b) s_earlier = 1;
      else { const int pos = atomicAdd(&s_cnt, 1); if (pos < kMaxDup) s_dup[pos] = bb; }
    }
  __syncthreads();
  if (s_earlier) return;          // not the leader (uniform across the CTA)
  const int n = s_cnt;
  if (n <= kMaxDup) {
    if (threadIdx.x == 0)         // ascending batch order (the list is short: insertion sort)
      for (int i = 1; i < n; ++i) {
        const int v = s_dup[i];
        int j = i - 1;
        while (j >= 0 && s_dup[j] > v) { s_dup[j + 1] = s_dup[j]; --j; }
        s_dup[j + 1] = v;
      }
    __syncthreads();
    for (int c = threadIdx.x; c < r; c += blockDim.x) {
      float acc = 0.0f;
      for (int i = 0; i < n; ++i) acc += rows_in[(int64_t)s_dup[i] * r + c];
      table[(int64_t)g * r + c] += acc;
    }
  } else {
    for (int c = threadIdx.x; c < r; c += blockDim.x) {
      float acc = 0.0f;
      for (int bb = b; bb < B; ++bb)
        if (idx[bb] == me) acc += rows_in[(int64_t)bb * r + c];
      table[(int64_t)g * r + c] += acc;
    }
  }
}

__global__ void core_axpby_kernel(const float* __restrict__ x, const double* __restrict__ alpha,
                                  const float* __restrict__ y, int count, float* __restrict__ out) {
  const float a = alpha ? (float)(*alpha) : 1.0f;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < count; i += gridDim.x * blockDim.x)
    out[i] = a * x[i] + (y ? y[i] : 0.0f);
}

// ------------------------------------------------------------------------------------------
// Gram:  out[ra, rb] = A^T B over n rows, fp32 products, fp64 accumulation across row blocks
// ------------------------------------------------------------------------------------------
constexpr int GT = 64;       // output tile edge
constexpr int GKC = 32;      // rows per smem chunk

// Exact Gram A^T B for A != B (A^T A takes gram_sym.cu): 64 x 64 tiles, two-stage fixed-order reduction; the products of two fp32
// values are exact in fp64 and accumulated in fp64 by mma.sync m8n8k4 (DMMA).  A CTA owns a 64 x 64 output tile over
// its row split; warp w owns the 8 x 64 strip of A-columns [8w, 8w + 8): eight 8 x 8 accumulator tiles.
// Row chunks are staged in shared memory as doubles (pitch 72: the four k-rows of a fragment load fall into
// different bank halves).
__device__ __forceinline__ void dmma884_g(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};\n"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}
constexpr int DG_LD = GT + 8;
__global__ void __launch_bounds__(256)
gram_dmma_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb,
                 int n, int ra, int rb, int tiles_b, int rows_per_split, double* __restrict__ partial) {
  __shared__ double As[GKC][DG_LD];
  __shared__ double Bs[GKC][DG_LD];
  const int tile = blockIdx.x, ta = tile / tiles_b, tb = tile - ta * tiles_b;
  const int a0 = ta * GT, b0 = tb * GT;
  const int split = blockIdx.y;
  const int row_beg = split * rows_per_split;
  const int row_end = min(n, row_beg + rows_per_split);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  const bool warp_ok = a0 + 8 * warp < ra;
  const int nbj = min(8, (rb - b0 + 7) / 8);
  const bool vec_a = (lda % 4 == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0);
  const bool vec_b = (ldb % 4 == 0) && ((reinterpret_cast<uintptr_t>(B) & 15) == 0);
  double c[8][2];
#pragma unroll
  for (int j = 0; j < 8; ++j) { c[j][0] = 0.0; c[j][1] = 0.0; }
  for (int r0 = row_beg; r0 < row_end; r0 += GKC) {
#pragma unroll
    for (int pass = 0; pass < 2; ++pass) {
      const int row = pass * 16 + (tid >> 4), c4 = (tid & 15) * 4;
      const int gr = r0 + row;
      float va[4] = {0.f, 0.f, 0.f, 0.f}, vb[4] = {0.f, 0.f, 0.f, 0.f};
      if (gr < row_end) {
        const float* pa = A + (int64_t)gr * lda + a0 + c4;
        const float* pb = B + (int64_t)gr * ldb + b0 + c4;
        if (vec_a && a0 + c4 + 4 <= ra) { const float4 x = __ldg(reinterpret_cast<const float4*>(pa)); va[0] = x.x; va[1] = x.y; va[2] = x.z; va[3] = x.w; }
        else {
#pragma unroll
          for (int u = 0; u < 4; ++u) if (a0 + c4 + u < ra) va[u] = __ldg(pa + u);
        }
        if (vec_b && b0 + c4 + 4 <= rb) { const float4 x = __ldg(reinterpret_cast<const float4*>(pb)); vb[0] = x.x; vb[1] = x.y; vb[2] = x.z; vb[3] = x.w; }
        else {
#pragma unroll
          for (int u = 0; u < 4; ++u) if (b0 + c4 + u < rb) vb[u] = __ldg(pb + u);
        }
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) { As[row][c4 + u] = (double)va[u]; Bs[row][c4 + u] = (double)vb[u]; }
    }
    __syncthreads();
    if (warp_ok) {
#pragma unroll
      for (int kk = 0; kk < GKC / 4; ++kk) {
        const double a = As[4 * kk + t][8 * warp + g];
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (j < nbj) dmma884_g(c[j][0], c[j][1], a, Bs[4 * kk + t][8 * j + g]);
      }
    }
    __syncthreads();
  }
  if (warp_ok) {
    const int i = a0 + 8 * warp + g;
    if (i < ra) {
      double* prow = partial + ((int64_t)split * ra + i) * rb;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const int col = b0 + 8 * j + 2 * t;
        if (j < nbj) {
          if (col < rb) prow[col] = c[j][0];
          if (col + 1 < rb) prow[col + 1] = c[j][1];
        }
      }
    }
  }
}

__global__ void gram_reduce_kernel(const double* __restrict__ partial, int nsplit, int count,
                                   double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double s = 0.0;
  for (int k = 0; k < nsplit; ++k) s += partial[(int64_t)k * count + i];  // fixed order
  out[i] = s;
}

struct GramPlan {
  int tiles_a, tiles_b, nsplit, rows_per_split;
};

GramPlan gram_plan(int n, int ra, int rb) {
  GramPlan p;
  p.tiles_a = rt::cdiv(ra, GT);
  p.tiles_b = rt::cdiv(rb, GT);
  const int tiles = p.tiles_a * p.tiles_b;
  const int target = 4 * 148;  // ~4 CTAs per SM in flight
  int nsplit = rt::cdiv(target, tiles);
  const int max_split = rt::cdiv(n, 4 * GKC);
  if (nsplit > max_split) nsplit = max_split;
  if (nsplit < 1) nsplit = 1;
  int rows = rt::cdiv(n, nsplit);
  rows = rt::cdiv(rows, GKC) * GKC;
  p.rows_per_split = rows;
  p.nsplit = rt::cdiv(n, rows);
  if (p.nsplit < 1) p.nsplit = 1;
  return p;
}

}  // namespace

extern "C" int rt_gather_rows(const float* table, int rows, int r, int row_begin, const int32_t* idx,
                              int B, float* out, void* stream) {
  RT_REQUIRE(B >= 0 && r > 0 && rows >= 0, "rt_gather_rows: bad shape");
  if (B == 0) return 0;
  gather_rows_kernel<<<B, 128, 0, (cudaStream_t)stream>>>(table, rows, r, row_begin, idx, out);
  RT_LAUNCH_CHECK();
  return 0;
}

extern "C" int rt_scatter_rows_add(float* table, int rows, int r, int row_begin, const int32_t* idx,
                                   int B, const float* rows_in, void* stream) {
  RT_REQUIRE(B >= 0 && r > 0 && rows >= 0, "rt_scatter_rows_add: bad shape");
  if (B == 0 || rows == 0) return 0;
  scatter_rows_add_kernel<<<B, 128, 0, (cudaStream_t)stream>>>(table, rows, r, row_begin, idx, B,
                                                               rows_in);
  RT_LAUNCH_CHECK();
  return 0;
}

extern "C" int rt_core_axpby(const float* dS_g, const double* alpha_dev, const float* pS_beta,
                             int count, float* dS_dir, void* stream) {
  RT_REQUIRE(count > 0, "rt_core_axpby: bad count");
  int blocks = rt::cdiv(count, 256);
  if (blocks > 148 * 8) blocks = 148 * 8;
  core_axpby_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(dS_g, alpha_dev, pS_beta, count,
                                                              dS_dir);
  RT_LAUNCH_CHECK();
  return 0;
}

// the register-tiled FP32 kernels of tallskinny_v2.cu are the default for the non-precise Gram and for apply
extern "C" size_t rt_gram_ws_bytes(int n, int ra, int rb) {
  if (n <= 0 || ra <= 0 || rb <= 0) return 0;
  GramPlan p = gram_plan(n, ra, rb);
  const size_t v1 = (size_t)p.nsplit * ra * rb * sizeof(double), v2 = rt::gram_v2_ws_bytes(n, ra, rb);
  const size_t v3 = (ra == rb && rt::gram_sym_supported(ra)) ? rt::gram_sym_ws_bytes(n, ra) : 0;
  return std::max(v1, std::max(v2, v3));
}

extern "C" int rt_gram(const float* A, int64_t lda, const float* B, int64_t ldb, int n, int ra,
                       int rb, double* out, int precise, void* ws, void* stream) {
  RT_REQUIRE(n >= 0 && ra > 0 && rb > 0 && lda >= ra && ldb >= rb, "rt_gram: bad shape n=%d ra=%d rb=%d",
             n, ra, rb);
  cudaStream_t s = (cudaStream_t)stream;
  if (n == 0) {
    RT_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * ra * rb, s));
    return 0;
  }
  RT_REQUIRE(ws != nullptr, "rt_gram: workspace is NULL");
  // A^T A (the norm and retraction Grams of a step): upper triangle on the fp64 tensor cores, exact accumulation
  if (A == B && lda == ldb && ra == rb && rt::gram_sym_supported(ra) && n >= 64)
    return rt::gram_sym(A, lda, n, ra, out, ws, s);
  if (!precise) return rt::gram_v2(A, lda, B, ldb, n, ra, rb, out, ws, stream);
  GramPlan p = gram_plan(n, ra, rb);
  dim3 grid(p.tiles_a * p.tiles_b, p.nsplit);
  gram_dmma_kernel<<<grid, 256, 0, s>>>(A, lda, B, ldb, n, ra, rb, p.tiles_b, p.rows_per_split, (double*)ws);
  RT_LAUNCH_CHECK();
  const int count = ra * rb;
  gram_reduce_kernel<<<rt::cdiv(count, 256), 256, 0, s>>>((const double*)ws, p.nsplit, count, out);
  RT_LAUNCH_CHECK();
  return 0;
}

extern "C" int rt_apply(float* Y, int64_t ldy, int n, int rc, const float* X0, int64_t ldx0,
                        const double* a0_dev, int nk, const float* const* X_host,
                        const int64_t* ldx_host, const int* rk_host, const double* const* K_host,
                        void* stream) {
  RT_REQUIRE(n >= 0 && rc > 0 && ldy >= rc, "rt_apply: bad shape n=%d rc=%d", n, rc);
  RT_REQUIRE(nk >= 0 && nk <= 4, "rt_apply: nk=%d out of range (max 4)", nk);
  RT_REQUIRE(X0 != nullptr || nk > 0, "rt_apply: nothing to compute");
  if (n == 0) return 0;
  return rt::apply_v2(Y, ldy, n, rc, X0, ldx0, a0_dev, nk, X_host, ldx_host, rk_host, K_host, stream);
}
