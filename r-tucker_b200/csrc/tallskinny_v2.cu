// Register-tiled FP32 kernels for the tall-skinny passes (the parity path: ~3e-7 relative error).
//   gram_v2 :  C[ra, rb] (+)= A[n, ra]^T B[n, rb]   104 x 104 output quadrants, 13 x 4 register tiles,
//              operand rows streamed with cp.async (row-major input IS the k-major smem layout)
//   apply_v2:  Y[n, rc] = a0 X0 + sum_t X_t K_t       128 x 104 tiles, 4 x 13 register tiles, double buffered
// r = 200 is exactly two 104-wide tiles (4 % padding).  FFMA-bound: 2*n*ra*rb and 2*n*rc*sum(rk) flop.
#include "common.h"

namespace {

__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n"
               :: "r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" :: "n"(N) : "memory"); }

// =====================================================================================================
// gram_v2
// =====================================================================================================
constexpr int GQ = 104;          // quadrant edge
constexpr int GLD = 108;         // smem row stride (floats): 16-byte aligned rows, conflict-light
constexpr int GKC = 16;          // operand rows per stage
constexpr int GST = 3;           // pipeline stages
constexpr int GTHREADS = 208;    // 8 (a) x 26 (b) threads, 13 x 4 accumulators each

__global__ void __launch_bounds__(GTHREADS)
gram_v2_kernel(const float* __restrict__ A, int64_t lda, const float* __restrict__ B, int64_t ldb, int n, int ra,
               int rb, int qb_count, int rows_per_split, float* __restrict__ partial, int vec_ok) {
  __shared__ __align__(16) float As[GST][GKC][GLD];
  __shared__ __align__(16) float Bs[GST][GKC][GLD];
  const int qa = blockIdx.x / qb_count, qb = blockIdx.x % qb_count;
  const int a0 = qa * GQ, b0 = qb * GQ;
  const int split = blockIdx.y;
  const int n0 = split * rows_per_split, n1 = min(n, n0 + rows_per_split);
  const int tid = threadIdx.x, ty = tid / 26, tx = tid % 26;
  const int nchunks = (n1 - n0 + GKC - 1) / GKC;

  auto issue = [&](int chunk, int stage) {
    const int row0 = n0 + chunk * GKC;
    // 16 rows x 26 float4 per operand
    for (int e = tid; e < GKC * 26; e += GTHREADS) {
      const int rr = e / 26, c4 = (e % 26) * 4;
      const int gr = row0 + rr;
      float* da = &As[stage][rr][c4];
      float* db = &Bs[stage][rr][c4];
      if (gr < n1 && vec_ok && a0 + c4 + 4 <= ra) cp_async16(da, A + (int64_t)gr * lda + a0 + c4);
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j) da[j] = (gr < n1 && a0 + c4 + j < ra) ? __ldg(A + (int64_t)gr * lda + a0 + c4 + j) : 0.0f;
      }
      if (gr < n1 && vec_ok && b0 + c4 + 4 <= rb) cp_async16(db, B + (int64_t)gr * ldb + b0 + c4);
      else {
#pragma unroll
        for (int j = 0; j < 4; ++j) db[j] = (gr < n1 && b0 + c4 + j < rb) ? __ldg(B + (int64_t)gr * ldb + b0 + c4 + j) : 0.0f;
      }
    }
    cp_async_commit();
  };

  float acc[13][4];
#pragma unroll
  for (int i = 0; i < 13; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.0f;

  for (int c = 0; c < GST - 1; ++c) { if (c < nchunks) issue(c, c); else cp_async_commit(); }
  for (int c = 0; c < nchunks; ++c) {
    cp_async_wait<GST - 2>();
    __syncthreads();
    if (c + GST - 1 < nchunks) issue(c + GST - 1, (c + GST - 1) % GST); else cp_async_commit();
    const int st = c % GST;
#pragma unroll 4
    for (int k = 0; k < GKC; ++k) {
      // a: columns {4*ty + 32*m + i, m<3} and {96 + ty}   b: columns 4*tx .. 4*tx+3
      float a[13];
#pragma unroll
      for (int m = 0; m < 3; ++m) {
        const float4 v = *reinterpret_cast<const float4*>(&As[st][k][4 * ty + 32 * m]);
        a[4 * m] = v.x; a[4 * m + 1] = v.y; a[4 * m + 2] = v.z; a[4 * m + 3] = v.w;
      }
      a[12] = As[st][k][96 + ty];
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[st][k][4 * tx]);
      const float b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 13; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
  }
  cp_async_wait<0>();
  // partial[split][ra][rb]
  float* out = partial + (int64_t)split * ra * rb;
#pragma unroll
  for (int i = 0; i < 13; ++i) {
    const int ai = a0 + ((i < 12) ? 4 * ty + 32 * (i >> 2) + (i & 3) : 96 + ty);
    if (ai >= ra) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int bj = b0 + 4 * tx + j;
      if (bj < rb) out[(int64_t)ai * rb + bj] = acc[i][j];
    }
  }
}

__global__ void gram_v2_reduce_kernel(const float* __restrict__ partial, int nsplit, int count, double* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  double s = 0.0;
  for (int k = 0; k < nsplit; ++k) s += (double)partial[(int64_t)k * count + i];
  out[i] = s;
}

struct GramV2Plan { int qa, qb, nsplit, rows_per_split; };
GramV2Plan gram_v2_plan(int n, int ra, int rb) {
  GramV2Plan p;
  p.qa = rt::cdiv(ra, GQ); p.qb = rt::cdiv(rb, GQ);
  const int quads = p.qa * p.qb;
  int nsplit = rt::cdiv(4 * 148, quads);           // ~4 CTAs per SM
  const int min_rows = 4 * GKC;
  if (nsplit > rt::cdiv(n, min_rows)) nsplit = rt::cdiv(n, min_rows);
  if (nsplit < 1) nsplit = 1;
  int rows = rt::cdiv(rt::cdiv(n, nsplit), GKC) * GKC;
  if (rows > 256) rows = 256;                       // fp32 accumulation is flushed at most every 256 rows
  p.rows_per_split = rows;
  p.nsplit = rt::cdiv(n, rows);
  return p;
}

// =====================================================================================================
// apply_v2
// =====================================================================================================
constexpr int AM = 128, AN = 104, AK = 16;
constexpr int ALDA = AM + 4;     // As[k][row]
constexpr int ALDB = 108;        // Bs[k][col]
constexpr int kMaxTerms = 4;

struct ApplyV2Args {
  const float* X[kMaxTerms]; int64_t ldx[kMaxTerms]; int rk[kMaxTerms]; const double* K[kMaxTerms];
  int nk;
};

__global__ void __launch_bounds__(256, 2)
apply_v2_kernel(float* __restrict__ Y, int64_t ldy, int n, int rc, const float* __restrict__ X0, int64_t ldx0,
                const double* __restrict__ a0_dev, ApplyV2Args args) {
  __shared__ __align__(16) float As[2][AK][ALDA];
  __shared__ __align__(16) float Bs[2][AK][ALDB];
  const int row0 = blockIdx.x * AM, col0 = blockIdx.y * AN;
  const int tid = threadIdx.x, tx = tid & 7, ty = tid >> 3;     // ty: rows 4*ty..+3 ; tx: cols {4*tx+32*m+i}, {96+tx}
  float acc[4][13];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 13; ++j) acc[i][j] = 0.0f;

  // flattened list of k-chunks over all terms
  int nchunks = 0;
  for (int t = 0; t < args.nk; ++t) nchunks += (args.rk[t] + AK - 1) / AK;
  float4 xa[2];        // prefetched X: 128 rows x 16 k = 512 float4, 2 per thread
  float kb[7];         // prefetched K: 16 x 104 = 1664 values, 6.5 per thread
  auto locate = [&](int chunk, int& t, int& k0) {
    t = 0;
    int c = chunk;
    while (true) {
      const int nt = (args.rk[t] + AK - 1) / AK;
      if (c < nt) break;
      c -= nt; ++t;
    }
    k0 = c * AK;
  };
  auto load = [&](int chunk) {
    int t, k0;
    locate(chunk, t, k0);
    const float* __restrict__ X = args.X[t];
    const int64_t ld = args.ldx[t];
    const int rk = args.rk[t];
    const bool vec = ((ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0);
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int e = it * 256 + tid;
      const int rr = e >> 2, kc = (e & 3) * 4;        // row, first of 4 consecutive k
      const int gr = row0 + rr, gk = k0 + kc;
      xa[it] = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gr < n && gk < rk) {
        const float* p = X + (int64_t)gr * ld + gk;
        if (vec && gk + 4 <= rk) xa[it] = __ldg(reinterpret_cast<const float4*>(p));
        else {
          xa[it].x = __ldg(p);
          if (gk + 1 < rk) xa[it].y = __ldg(p + 1);
          if (gk + 2 < rk) xa[it].z = __ldg(p + 2);
          if (gk + 3 < rk) xa[it].w = __ldg(p + 3);
        }
      }
    }
    const double* __restrict__ K = args.K[t];
#pragma unroll
    for (int it = 0; it < 7; ++it) {
      const int e = it * 256 + tid;
      kb[it] = 0.0f;
      if (e < AK * AN) {
        const int kk = e / AN, cc = e - kk * AN;
        const int gk = k0 + kk, gc = col0 + cc;
        if (gk < rk && gc < rc) kb[it] = (float)__ldg(K + (int64_t)gk * rc + gc);
      }
    }
  };
  auto store = [&](int stage) {
#pragma unroll
    for (int it = 0; it < 2; ++it) {
      const int e = it * 256 + tid;
      const int rr = e >> 2, kc = (e & 3) * 4;
      As[stage][kc + 0][rr] = xa[it].x; As[stage][kc + 1][rr] = xa[it].y;
      As[stage][kc + 2][rr] = xa[it].z; As[stage][kc + 3][rr] = xa[it].w;
    }
#pragma unroll
    for (int it = 0; it < 7; ++it) {
      const int e = it * 256 + tid;
      if (e < AK * AN) Bs[stage][e / AN][e % AN] = kb[it];
    }
  };

  if (nchunks > 0) { load(0); store(0); }
  __syncthreads();
  for (int c = 0; c < nchunks; ++c) {
    const int st = c & 1;
    if (c + 1 < nchunks) load(c + 1);
#pragma unroll
    for (int k = 0; k < AK; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[st][k][4 * ty]);
      const float a[4] = {av.x, av.y, av.z, av.w};
      float b[13];
#pragma unroll
      for (int m = 0; m < 3; ++m) {
        const float4 v = *reinterpret_cast<const float4*>(&Bs[st][k][4 * tx + 32 * m]);
        b[4 * m] = v.x; b[4 * m + 1] = v.y; b[4 * m + 2] = v.z; b[4 * m + 3] = v.w;
      }
      b[12] = Bs[st][k][96 + tx];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 13; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (c + 1 < nchunks) store(st ^ 1);
    __syncthreads();
  }
  const float a0 = a0_dev ? (float)(*a0_dev) : 1.0f;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int gr = row0 + 4 * ty + i;
    if (gr >= n) continue;
#pragma unroll
    for (int j = 0; j < 13; ++j) {
      const int gc = col0 + ((j < 12) ? 4 * tx + 32 * (j >> 2) + (j & 3) : 96 + tx);
      if (gc >= rc) continue;
      float v = acc[i][j];
      if (X0) v = fmaf(a0, X0[(int64_t)gr * ldx0 + gc], v);
      Y[(int64_t)gr * ldy + gc] = v;
    }
  }
}

}  // namespace

namespace rt {
size_t gram_v2_ws_bytes(int n, int ra, int rb) {
  if (n <= 0) return 16;
  GramV2Plan p = gram_v2_plan(n, ra, rb);
  return (size_t)p.nsplit * ra * rb * sizeof(float);
}

int gram_v2(const float* A, int64_t lda, const float* B, int64_t ldb, int n, int ra, int rb, double* out, void* ws,
            void* stream) {
  cudaStream_t s = (cudaStream_t)stream;
  if (n == 0) { RT_CHECK_CUDA(cudaMemsetAsync(out, 0, sizeof(double) * ra * rb, s)); return 0; }
  RT_REQUIRE(ws != nullptr, "rt_gram_v2: workspace is NULL");
  GramV2Plan p = gram_v2_plan(n, ra, rb);
  const int vec_ok = ((lda & 3) == 0) && ((ldb & 3) == 0) && ((reinterpret_cast<uintptr_t>(A) & 15) == 0) &&
                     ((reinterpret_cast<uintptr_t>(B) & 15) == 0);
  dim3 grid(p.qa * p.qb, p.nsplit);
  gram_v2_kernel<<<grid, GTHREADS, 0, s>>>(A, lda, B, ldb, n, ra, rb, p.qb, p.rows_per_split, (float*)ws, vec_ok);
  RT_LAUNCH_CHECK();
  const int count = ra * rb;
  gram_v2_reduce_kernel<<<rt::cdiv(count, 256), 256, 0, s>>>((const float*)ws, p.nsplit, count, out);
  RT_LAUNCH_CHECK();
  return 0;
}

int apply_v2(float* Y, int64_t ldy, int n, int rc, const float* X0, int64_t ldx0, const double* a0_dev, int nk,
             const float* const* X_host, const int64_t* ldx_host, const int* rk_host, const double* const* K_host,
             void* stream) {
  RT_REQUIRE(nk >= 0 && nk <= kMaxTerms, "rt_apply_v2: nk out of range");
  if (n == 0) return 0;
  ApplyV2Args a{};
  a.nk = nk;
  for (int k = 0; k < kMaxTerms; ++k) {
    a.X[k] = k < nk ? X_host[k] : nullptr; a.ldx[k] = k < nk ? ldx_host[k] : 0;
    a.rk[k] = k < nk ? rk_host[k] : 0; a.K[k] = k < nk ? K_host[k] : nullptr;
    if (k < nk) RT_REQUIRE(a.X[k] != Y, "rt_apply_v2: Y may alias X0 only");
  }
  dim3 grid(rt::cdiv(n, AM), rt::cdiv(rc, AN));
  apply_v2_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(Y, ldy, n, rc, X0, ldx0, a0_dev, a);
  RT_LAUNCH_CHECK();
  return 0;
}
}  // namespace rt
