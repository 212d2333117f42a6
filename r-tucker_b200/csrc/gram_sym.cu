// Symmetric Gram  G[r, r] = X[n, r]^T X[n, r]  with EXACT fp64 accumulation on the fp64 tensor cores (DMMA m8n8k4).
//
// Reference call sites: the Gram products inside tucker_riemopt's `TangentVector.norm` and the QR of [U | dV] in
// `round` (src/model/asymmetric/optim.py:90,108; symmetric/optim.py:84,102).  Both Grams of a step have A == B, so
// only the upper triangle of 32 x 32 tiles is computed (28 of 49 tiles at r = 200) and mirrored by the reduction.
// Products of fp32 inputs are exact in fp64, the accumulation is fp64: the result is the exactly-accumulated Gram
// the Cholesky of the retraction needs (and the norm gets it for free).
//
// One unit = (tile, row chunk).  The 8 warps of a CTA take the 4-row k-steps of the chunk round-robin; each warp
// keeps the whole 32 x 32 tile in 16 DMMA accumulators and feeds them with fragments loaded straight from global
// memory (8 lanes read 32 contiguous bytes: full sectors; fp32 -> fp64 in registers), three k-steps in flight.  Warp
// partials are summed through shared memory in a fixed order, chunk partials by a second kernel in a fixed order:
// bit-identical on every replica.
#include "prims.cuh"

namespace {

constexpr int GT = 32;
constexpr int GWARPS = 8, GTHREADS = 256;
constexpr int GLD = 34;                   // padded row stride of a warp partial in shared memory
constexpr int GMAX_T = 16;                // r <= 512

__global__ void __launch_bounds__(GTHREADS, 2)
gram_sym_kernel(const float* __restrict__ X, int64_t ld, int n, int r, int T, int ntiles, int rows_per_chunk,
                double* __restrict__ partial) {
  extern __shared__ __align__(16) double red[];          // [8][32][GLD]
  const int unit = blockIdx.x;
  const int chunk = unit / ntiles, tile = unit - chunk * ntiles;
  int ti, tj;
  rt::sym_tile(tile, T, ti, tj);
  const int i0 = ti * GT, j0 = tj * GT;
  const int row_beg = chunk * rows_per_chunk;
  const int row_end = min(n, row_beg + rows_per_chunk);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const bool diag = ti == tj;

  double c[4][4][2];
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b) { c[a][b][0] = 0.0; c[a][b][1] = 0.0; }

  // column validity of this lane's fragments (columns >= r read as zero)
  bool va[4], vb[4];
#pragma unroll
  for (int x = 0; x < 4; ++x) { va[x] = i0 + 8 * x + g < r; vb[x] = j0 + 8 * x + g < r; }
  const float* pa = X + i0 + g;
  const float* pb = X + j0 + g;
  const int steps_total = (row_end - row_beg + 3) / 4;          // k-steps of the chunk
  const int my_steps = steps_total > warp ? (steps_total - warp + GWARPS - 1) / GWARPS : 0;

  float fa[3][4], fb[3][4];
  auto load = [&](int s, float (&ra)[4], float (&rb)[4]) {
    const int row = row_beg + 4 * (warp + s * GWARPS) + t;
    const bool ok = row < row_end;
    const int64_t off = (int64_t)row * ld;
#pragma unroll
    for (int x = 0; x < 4; ++x) ra[x] = (ok && va[x]) ? __ldg(pa + off + 8 * x) : 0.0f;
    if (!diag) {
#pragma unroll
      for (int x = 0; x < 4; ++x) rb[x] = (ok && vb[x]) ? __ldg(pb + off + 8 * x) : 0.0f;
    }
  };
  auto mma = [&](const float (&ra)[4], const float (&rb)[4]) {
    double da[4], db[4];
#pragma unroll
    for (int x = 0; x < 4; ++x) { da[x] = (double)ra[x]; db[x] = diag ? da[x] : (double)rb[x]; }
#pragma unroll
    for (int a = 0; a < 4; ++a)
#pragma unroll
      for (int b = 0; b < 4; ++b) rt::dmma884(c[a][b][0], c[a][b][1], da[a], db[b]);
  };
  if (my_steps > 0) load(0, fa[0], fb[0]);
  if (my_steps > 1) load(1, fa[1], fb[1]);
  for (int s = 0; s < my_steps; s += 3) {
    if (s + 2 < my_steps) load(s + 2, fa[2], fb[2]);
    mma(fa[0], fb[0]);
    if (s + 1 >= my_steps) break;
    if (s + 3 < my_steps) load(s + 3, fa[0], fb[0]);
    mma(fa[1], fb[1]);
    if (s + 2 >= my_steps) break;
    if (s + 4 < my_steps) load(s + 4, fa[1], fb[1]);
    mma(fa[2], fb[2]);
  }
  // A fragment (row.col): a = A[g][t] -> element (i = 8a + g, k = t); B fragment: b = B[t][g] -> (k = t, j = 8b + g);
  // C fragment: c0, c1 = C[g][2t], C[g][2t + 1]
  double* mine = red + warp * (GT * GLD);
#pragma unroll
  for (int a = 0; a < 4; ++a)
#pragma unroll
    for (int b = 0; b < 4; ++b)
      *reinterpret_cast<double2*>(&mine[(8 * a + g) * GLD + 8 * b + 2 * t]) = make_double2(c[a][b][0], c[a][b][1]);
  __syncthreads();
  double* out = partial + ((int64_t)chunk * ntiles + tile) * (GT * GT);
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const int e = threadIdx.x + GTHREADS * m;
    const int row = e >> 5, col = e & 31;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < GWARPS; ++w) s += red[w * (GT * GLD) + row * GLD + col];
    out[e] = s;
  }
}

__global__ void gram_sym_reduce_kernel(const double* __restrict__ partial, int nchunks, int ntiles, int T, int r,
                                       double* __restrict__ out) {
  const int e = blockIdx.x * blockDim.x + threadIdx.x;
  if (e >= r * r) return;
  const int i = e / r, j = e - i * r;
  const int a = min(i, j), b = max(i, j);
  const int ti = a / GT, tj = b / GT;
  const int tile = ti * T - ti * (ti - 1) / 2 + (tj - ti);
  const int64_t at = (int64_t)tile * (GT * GT) + (a - ti * GT) * GT + (b - tj * GT);
  double s = 0.0;
  for (int k = 0; k < nchunks; ++k) s += partial[(int64_t)k * ntiles * (GT * GT) + at];   // fixed order
  out[e] = s;
}

struct SymPlan { int T, ntiles, nchunks, rows_per_chunk; };
SymPlan sym_plan(int n, int r) {
  SymPlan p;
  p.T = rt::cdiv(r, GT);
  p.ntiles = p.T * (p.T + 1) / 2;
  // two CTAs per SM resident; aim at whole waves of 2 * SMs units, chunks of at least 256 rows
  const int slots = 2 * rt::sm_count();
  int waves = 1;
  int nchunks = slots * waves / p.ntiles;
  while (nchunks < 1 || rt::cdiv(n, nchunks > 0 ? nchunks : 1) > 4096) { ++waves; nchunks = slots * waves / p.ntiles; }
  const int max_chunks = rt::cdiv(n, 256);
  if (nchunks > max_chunks) nchunks = max_chunks;
  if (nchunks < 1) nchunks = 1;
  p.rows_per_chunk = rt::cdiv(rt::cdiv(n, nchunks), 4) * 4;
  p.nchunks = rt::cdiv(n, p.rows_per_chunk);
  return p;
}

}  // namespace

namespace rt {
bool gram_sym_supported(int r) { return r >= 1 && r <= GT * GMAX_T; }
size_t gram_sym_ws_bytes(int n, int r) {
  const SymPlan p = sym_plan(n > 0 ? n : 1, r);
  return (size_t)p.nchunks * p.ntiles * GT * GT * sizeof(double);
}
int gram_sym(const float* X, int64_t ld, int n, int r, double* out, void* ws, cudaStream_t s) {
  const SymPlan p = sym_plan(n, r);
  const size_t smem = sizeof(double) * GWARPS * GT * GLD;
  RT_CHECK_CUDA(rt::ensure_dyn_smem((const void*)gram_sym_kernel, smem));
  gram_sym_kernel<<<p.nchunks * p.ntiles, GTHREADS, smem, s>>>(X, ld, n, r, p.T, p.ntiles, p.rows_per_chunk, (double*)ws);
  RT_LAUNCH_CHECK();
  gram_sym_reduce_kernel<<<rt::cdiv(r * r, 256), 256, 0, s>>>((const double*)ws, p.nchunks, p.ntiles, p.T, r, out);
  RT_LAUNCH_CHECK();
  return 0;
}
}  // namespace rt
