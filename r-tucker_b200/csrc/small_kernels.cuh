// Device kernels of the N-independent ("small") stage that small.cu launches directly, outside the recorded
// executor of small_exec.cuh: the SPD factorisation / inverse, and the rows-times-inverse product of
// rt_rows_times_ainv.  Internal to small.cu.
#pragma once
#include "prims.cuh"
#include <math.h>

namespace rt {
namespace small {

// C(f32)[m, r] = A(f32)[m, r] . K(f64)[r, r]
__global__ void __launch_bounds__(256)
rows_times_mat_kernel(const float* __restrict__ A, int m, int r, const double* __restrict__ K,
                      float* __restrict__ C) {
  extern __shared__ float rows[];  // [RPB][r]
  constexpr int RPB = 4;
  const int b0 = blockIdx.x * RPB;
  for (int e = threadIdx.x; e < RPB * r; e += 256) {
    const int rr = e / r, cc = e - rr * r;
    rows[e] = (b0 + rr < m) ? A[(int64_t)(b0 + rr) * r + cc] : 0.0f;
  }
  __syncthreads();
  for (int j = threadIdx.x; j < r; j += 256) {
    double acc[RPB];
#pragma unroll
    for (int i = 0; i < RPB; ++i) acc[i] = 0.0;
#pragma unroll 4
    for (int k = 0; k < r; ++k) {
      const double kv = K[(int64_t)k * r + j];
#pragma unroll
      for (int i = 0; i < RPB; ++i) acc[i] = fma((double)rows[i * r + k], kv, acc[i]);
    }
#pragma unroll
    for (int i = 0; i < RPB; ++i)
      if (b0 + i < m) C[(int64_t)(b0 + i) * r + j] = (float)acc[i];
  }
}

// ---- SPD factorisation: G = L L^T (packed in smem), Linv = L^-1, Ginv = Linv^T Linv ---------
struct SpdProblem {
  const double* G;   // [n][n]
  double* L;         // [n][n] lower (may be NULL)
  double* Linv;      // [n][n] lower (may be NULL)
  double* Ginv;      // [n][n] (may be NULL)
  int n;
};
struct SpdBatch { SpdProblem p[3]; int dmma; };   // dmma: O(n^3) phases on the fp64 tensor cores (needs 8 n more doubles of smem)

__device__ __forceinline__ int pk(int i, int j) { return i * (i + 1) / 2 + j; }
// sum of 8 interleaved partial accumulators in a fixed order
__device__ __forceinline__ double spd_sum8(const double (&c)[8][2], int e) {
  return ((c[0][e] + c[1][e]) + (c[2][e] + c[3][e])) + ((c[4][e] + c[5][e]) + (c[6][e] + c[7][e]));
}

// One CTA per problem of the batch.  It reads G, symmetrised as (G + G^T) / 2, and writes each of L, Linv and Ginv that
// is not NULL as a full n x n row-major matrix: the lower Cholesky factor with G = L L^T, its lower-triangular inverse
// L^-1, and G^-1 = Linv^T Linv.  A pivot <= 1e-12 x the largest diagonal entry of G counts as zero: that column of L
// and that row and column of Linv are zero, so Ginv inverts G on the other columns only.
//   Cholesky, left looking in blocks of 8 columns: (1) every row subtracts the contribution of all earlier
//   columns from its 8 block entries (the 8 "pivot rows" are broadcast reads), (2) warp 0 factors the 8x8
//   diagonal block, (3) every row below solves its 8 entries against that block.
//   Inverse, in blocks of 8 rows: the rows of L are staged, then thread group j produces column j of the 8 new rows
//   of L^-1 from its own (already inverted) column above.
constexpr int SPD_NB = 8;
// 512 threads, two per matrix row (n <= 256): 128 registers per thread, so that the 8 x 8 diagonal block really stays
// in the registers of the thread that factors it (at 1024 threads x 64 registers it spilled to local memory)
constexpr int SPD_THREADS = 512, SPD_TPR = 2;
__global__ void __launch_bounds__(SPD_THREADS, 1)
spd_blocked_kernel(SpdBatch batch) {
  // an executor program launched as this kernel's programmatic dependent (rt_small_prepare_project) starts on the SMs
  // the batch leaves idle; it must not touch the batch's matrices, and its end waits for this grid
  pdl_launch_dependents();
  extern __shared__ double sm[];
  const SpdProblem P = batch.p[blockIdx.x];
  const int n = P.n;
  if (n <= 0) return;
  double* Lp = sm;                              // packed lower n(n+1)/2
  double* stage = sm + n * (n + 1) / 2;         // [SPD_NB][n] staged rows of L
  __shared__ double D[SPD_NB][SPD_NB + 1], invd[SPD_NB];
  __shared__ double dinv_all[256];              // 1 / L[i][i] (0 for a zero pivot): the inverse never divides
  __shared__ double s_maxd, s_scale[4];
  const int tid = threadIdx.x, nt = blockDim.x;
  const int row = tid / SPD_TPR, sub = tid % SPD_TPR;
  for (int e = tid; e < n * (n + 1) / 2; e += nt) {
    int i = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
    while (i * (i + 1) / 2 > e) --i;
    while ((i + 1) * (i + 2) / 2 <= e) ++i;
    const int j = e - i * (i + 1) / 2;
    Lp[e] = 0.5 * (P.G[(int64_t)i * n + j] + P.G[(int64_t)j * n + i]);
  }
  __syncthreads();
  if (tid < 32) {
    double m = 0.0;
    for (int i = tid; i < n; i += 32) m = fmax(m, Lp[pk(i, i)]);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (tid == 0) {
      // the factorisation runs on G / 4^k with the largest diagonal entry in [0.25, 1): exact scaling (powers of two
      // in L, L^-1 and G^-1 as well), pivots inside the fp32 range for the reciprocal / rsqrt seeds, and no scaling
      // operations on the serial pivot chain
      int ex = 0;
      if (m > 0.0) { frexp(m, &ex); ex += ex & 1; }
      s_maxd = ldexp(m, -ex);
      s_scale[0] = ldexp(1.0, -ex);        // G      -> scaled
      s_scale[1] = ldexp(1.0, ex / 2);     // L      <- scaled
      s_scale[2] = ldexp(1.0, -(ex / 2));  // L^-1   <- scaled
      s_scale[3] = ldexp(1.0, -ex);        // G^-1   <- scaled
    }
  }
  __syncthreads();
  {
    const double sc = s_scale[0];
    for (int e = tid; e < n * (n + 1) / 2; e += nt) Lp[e] *= sc;
  }
  __syncthreads();
  const double tol = 1e-12 * s_maxd;
  double* Li = Lp + pk(row < n ? row : 0, 0);
#ifdef RT_SPD_PROF
  long long t_0 = clock64(), t_a = 0, t_b = 0, t_c = 0, t_x;
#define SPD_LAP(v) do { t_x = clock64(); v += t_x - t_0; t_0 = t_x; } while (0)
#else
#define SPD_LAP(v) do {} while (0)
#endif
  // ---------------- Cholesky ----------------
  // The plain fp64 pipe of this part runs at ~3 TFLOP/s per GPU (20 GFLOP/s per SM, tools/dmma_probe.cu) against 36 on the
  // fp64 tensor cores: the three n^3 / 3 phases (left-looking update, inverse, L^-T L^-1) took ~130 us each on the one SM
  // a problem owns.  With batch.dmma they run as 8 x 8 x 4 DMMAs on fragments read from the packed triangle; a tile's
  // contraction is spread over 8 interleaved accumulators (a dependent DMMA waits hundreds of cycles) summed in a
  // fixed order.
  const bool use_dmma = batch.dmma != 0;
  const int warp = tid >> 5, lane = tid & 31, fg = lane >> 2, ft = lane & 3;
  constexpr int NW = SPD_THREADS / 32;
  double* accS = stage + SPD_NB * n;              // [SPD_NB][n] tile results of the inverse (dmma only)
  for (int kb = 0; kb < n; kb += SPD_NB) {
    const int nbk = min(SPD_NB, n - kb);
    if (use_dmma) {
      // T[row][c] = sum_{k < kb} L[row][k] L[kb + c][k] for rows >= kb: A = L rows, B[k][c] = L[kb + c][k]
      if (kb > 0) {
        const int ntile = (n - kb + 7) >> 3, nsteps = kb >> 2;
        const int brow = kb + fg;
        const bool bv = brow < n;
        const double* Lb = Lp + pk(bv ? brow : 0, 0) + ft;
        for (int tile = warp; tile < ntile; tile += NW) {
          const int arow = kb + 8 * tile + fg;
          const bool av = arow < n;
          const double* La = Lp + pk(av ? arow : 0, 0) + ft;
          double c[8][2];
#pragma unroll
          for (int u = 0; u < 8; ++u) { c[u][0] = 0.0; c[u][1] = 0.0; }
          for (int s0 = 0; s0 < nsteps; s0 += 8) {
#pragma unroll
            for (int u = 0; u < 8; ++u)
              if (s0 + u < nsteps) dmma884(c[u][0], c[u][1], av ? La[4 * (s0 + u)] : 0.0, bv ? Lb[4 * (s0 + u)] : 0.0);
          }
          // result element: row 8 tile + fg (the SAME row this lane fetched), columns 2 ft, 2 ft + 1
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int col = 2 * ft + e;
            if (av && col < nbk && kb + col <= arow) Lp[pk(arow, kb + col)] -= spd_sum8(c, e);
          }
        }
      }
    } else {
      double acc[SPD_NB];
#pragma unroll
      for (int c = 0; c < SPD_NB; ++c) acc[c] = 0.0;
      if (row < n && row >= kb) {
        const double* Lc[SPD_NB];
#pragma unroll
        for (int c = 0; c < SPD_NB; ++c) Lc[c] = Lp + pk(kb + (c < nbk ? c : 0), 0);
        for (int k = sub; k < kb; k += SPD_TPR) {
          const double li = Li[k];
#pragma unroll
          for (int c = 0; c < SPD_NB; ++c) acc[c] = fma(li, Lc[c][k], acc[c]);
        }
      }
#pragma unroll
      for (int c = 0; c < SPD_NB; ++c) {
#pragma unroll
        for (int o = 1; o < SPD_TPR; o <<= 1) acc[c] += __shfl_xor_sync(0xffffffffu, acc[c], o);
      }
      if (row < n && row >= kb && sub == 0) {
#pragma unroll
        for (int c = 0; c < SPD_NB; ++c)
          if (c < nbk && kb + c <= row) Li[kb + c] -= acc[c];
      }
    }
    __syncthreads();
    SPD_LAP(t_a);
    if (tid < 32) {
      // The 8 x 8 diagonal block, by warp 0.  Every fp64 instruction occupies the fp64 pipe for a whole warp slot
      // whether one lane or 32 use it, and one thread doing all ~320 operations of a block was the longest phase of the
      // kernel: here each lane owns one (two for lanes 0-3) of the 36 entries, the block lives in shared memory, and
      // ALL lanes evaluate the pivot reciprocal redundantly (nothing to broadcast).  Rows past n are padded with the
      // identity.  Elimination in L D L^T form -- the next pivot needs 1 / d_cc (fp32 seed + two Newton steps) and one
      // fma -- then the square roots that turn it into the Cholesky factor, one column per lane.
      int er[2], ec[2];
#pragma unroll
      for (int u = 0; u < 2; ++u) {
        const int e = tid + 32 * u;                       // entry index in the packed 8 x 8 lower triangle
        int r = 0;
        while ((r + 1) * (r + 2) / 2 <= e) ++r;
        er[u] = r; ec[u] = e - r * (r + 1) / 2;
      }
      const bool has2 = tid + 32 < SPD_NB * (SPD_NB + 1) / 2;
      if (!has2) { er[1] = 0; ec[1] = 0; }                // unused second slot: keep its (ignored) reads inside D
#pragma unroll
      for (int u = 0; u < 2; ++u)
        if (u == 0 || has2)
          D[er[u]][ec[u]] = (er[u] < nbk) ? Lp[pk(kb + er[u], kb + ec[u])] : (er[u] == ec[u] ? 1.0 : 0.0);
      __syncwarp();
#pragma unroll
      for (int c = 0; c < SPD_NB - 1; ++c) {
        const double dc = D[c][c];
        double a_rc[2], a_cc[2];
#pragma unroll
        for (int u = 0; u < 2; ++u) { a_rc[u] = D[er[u]][c]; a_cc[u] = D[ec[u]][c]; }
        double ri = 0.0;                                  // 0 for a zero pivot: its column drops out of the updates
        if (dc > tol) {
          double y = (double)__frcp_rn((float)dc);
          y = fma(y, fma(-dc, y, 1.0), y);
          ri = fma(y, fma(-dc, y, 1.0), y);
        }
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if ((u == 0 || has2) && ec[u] > c) D[er[u]][ec[u]] = fma(-(a_rc[u] * a_cc[u]), ri, D[er[u]][ec[u]]);
        __syncwarp();
      }
      {
        // sqrt(d_cc) and its inverse for column c = lane & 7: fp32 seed, Newton steps (22 -> 44 -> 88 bits), one Heron
        // correction
        const int c = tid & (SPD_NB - 1);
        const double dc = D[c][c];
        double piv = 0.0, inv = 0.0;
        if (dc > tol) {
          double y = (double)rsqrtf((float)dc);
#pragma unroll
          for (int it = 0; it < 2; ++it) y = y * fma(-0.5 * dc, y * y, 1.5);
          piv = dc * y;
          piv = fma(0.5 * y, fma(-piv, piv, dc), piv);
          inv = fma(y, fma(-piv, y, 1.0), y);             // 1 / piv to the last bits
        }
        __syncwarp();
        if (tid < SPD_NB) {
          invd[c] = inv;
          if (c < nbk) dinv_all[kb + c] = inv;
        }
        __syncwarp();
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if ((u == 0 || has2) && er[u] != ec[u]) D[er[u]][ec[u]] *= invd[ec[u]];
        if (tid < SPD_NB) D[c][c] = piv;
        __syncwarp();
#pragma unroll
        for (int u = 0; u < 2; ++u)
          if ((u == 0 || has2) && er[u] < nbk) Lp[pk(kb + er[u], kb + ec[u])] = D[er[u]][ec[u]];
      }
    }
    __syncthreads();
    SPD_LAP(t_b);
    if (row < n && row >= kb + nbk && sub == 0) {
      double xs[SPD_NB];
#pragma unroll
      for (int c = 0; c < SPD_NB; ++c) {
        if (c < nbk) {
          double x = Li[kb + c];
#pragma unroll
          for (int c2 = 0; c2 < SPD_NB; ++c2)
            if (c2 < c) x = fma(-xs[c2], D[c][c2], x);
          x *= invd[c];
          xs[c] = x;
          Li[kb + c] = x;
        }
      }
    }
    __syncthreads();
    SPD_LAP(t_c);
  }
#ifdef RT_SPD_PROF
  if (tid == 0) printf("spd n=%d chol: update %lld diag %lld panel %lld\n", n, t_a, t_b, t_c);
  t_a = t_b = t_c = 0; t_0 = clock64();
#endif
  if (P.L) {
    for (int e = tid; e < n * n; e += nt) {
      const int i = e / n, j = e - i * n;
      P.L[e] = (j <= i) ? Lp[pk(i, j)] * s_scale[1] : 0.0;
    }
  }
  if (!P.Linv && !P.Ginv) return;
  __syncthreads();
  // ---------------- in-place inverse of the packed lower triangle, 8 rows at a time ----------------
  for (int ib = 0; ib < n; ib += SPD_NB) {
    const int nbi = min(SPD_NB, n - ib);
    for (int e = tid; e < nbi * n; e += nt) {
      const int r = e / n, k = e - r * n;
      stage[e] = (k <= ib + r) ? Lp[pk(ib + r, k)] : 0.0;
    }
    __syncthreads();
    const int j = row;                                   // column owned by this pair of threads
    double acc[SPD_NB];
#pragma unroll
    for (int r = 0; r < SPD_NB; ++r) acc[r] = 0.0;
    if (use_dmma) {
      // T[r][j] = sum_{k = j}^{ib - 1} L[ib + r][k] X[k][j]: A = the staged rows, B[k][j] = X[k][j] (0 above the diagonal);
      // a warp per tile of 8 columns, the contraction starts at the tile's first column
      const int ntile = ib >> 3;
      for (int tile = warp; tile < ntile; tile += NW) {
        const int j0 = 8 * tile, jc = j0 + fg;            // B column of this lane
        const int nsteps = (ib - j0) >> 2;
        double c[8][2];
#pragma unroll
        for (int u = 0; u < 8; ++u) { c[u][0] = 0.0; c[u][1] = 0.0; }
        for (int s0 = 0; s0 < nsteps; s0 += 8) {
#pragma unroll
          for (int u = 0; u < 8; ++u)
            if (s0 + u < nsteps) {
              const int k = j0 + 4 * (s0 + u) + ft;
              dmma884(c[u][0], c[u][1], stage[fg * n + k], k >= jc ? Lp[pk(k, jc)] : 0.0);
            }
        }
#pragma unroll
        for (int e = 0; e < 2; ++e) accS[fg * n + j0 + 2 * ft + e] = spd_sum8(c, e);
      }
      __syncthreads();
      if (j < n && j < ib) {
#pragma unroll
        for (int r = 0; r < SPD_NB; ++r) acc[r] = accS[r * n + j];
      }
    } else {
      if (j < n && j < ib) {
        for (int k = j + sub; k < ib; k += SPD_TPR) {
          const double xk = Lp[pk(k, j)];                  // X[k][j], rows above this block are already inverted
#pragma unroll
          for (int r = 0; r < SPD_NB; ++r) acc[r] = fma(stage[r * n + k], xk, acc[r]);   // rows r >= nbi are stale: unused
        }
      }
#pragma unroll
      for (int r = 0; r < SPD_NB; ++r) {
#pragma unroll
        for (int o = 1; o < SPD_TPR; o <<= 1) acc[r] += __shfl_xor_sync(0xffffffffu, acc[r], o);
      }
    }
    if (j < n && j < ib + nbi && sub == 0) {
      double xs[SPD_NB];
#pragma unroll
      for (int r = 0; r < SPD_NB; ++r) {
        xs[r] = 0.0;
        if (r < nbi) {
          const int i = ib + r;
          if (i >= j) {
            const double dinv = dinv_all[i];
            double x;
            if (i == j) {
              x = dinv;
            } else {
              double sacc = acc[r];
#pragma unroll
              for (int r2 = 0; r2 < SPD_NB; ++r2)
                if (r2 < r && ib + r2 >= j) sacc = fma(stage[r * n + ib + r2], xs[r2], sacc);
              x = -sacc * dinv;
            }
            xs[r] = x;
            Lp[pk(i, j)] = x;
          }
        }
      }
    }
    __syncthreads();
  }
  SPD_LAP(t_a);
  if (P.Linv) {
    for (int e = tid; e < n * n; e += nt) {
      const int i = e / n, j = e - i * n;
      P.Linv[e] = (j <= i) ? Lp[pk(i, j)] * s_scale[2] : 0.0;
    }
  }
  SPD_LAP(t_b);
  if (P.Ginv && use_dmma) {
    // Ginv = X^T X by 8 x 8 tiles of the lower half: G[i][j] = sum_{k >= i} X[k][i] X[k][j]; A[i][k] = X[k][i],
    // B[k][j] = X[k][j], both 0 above the diagonal of X (only the first k-steps of a tile need the mask)
    __syncthreads();
    const int T8 = (n + 7) >> 3;
    const double sc = s_scale[3];
    for (int u0 = warp; u0 < T8 * (T8 + 1) / 2; u0 += NW) {
      int it = (int)((sqrtf(8.0f * u0 + 1.0f) - 1.0f) * 0.5f);
      while (it * (it + 1) / 2 > u0) --it;
      while ((it + 1) * (it + 2) / 2 <= u0) ++it;
      const int jt = u0 - it * (it + 1) / 2;
      const int i0 = 8 * it, ic = i0 + fg, jc = 8 * jt + fg;
      const int nsteps = (n - i0 + 3) >> 2;
      double c[8][2];
#pragma unroll
      for (int u = 0; u < 8; ++u) { c[u][0] = 0.0; c[u][1] = 0.0; }
      for (int s0 = 0; s0 < nsteps; s0 += 8) {
#pragma unroll
        for (int u = 0; u < 8; ++u)
          if (s0 + u < nsteps) {
            const int k = i0 + 4 * (s0 + u) + ft;
            const bool kv = k < n;
            dmma884(c[u][0], c[u][1], (kv && ic < n && k >= ic) ? Lp[pk(k, ic)] : 0.0, (kv && jc < n && k >= jc) ? Lp[pk(k, jc)] : 0.0);
          }
      }
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const int i = i0 + fg, j = 8 * jt + 2 * ft + e;
        if (i < n && j <= i) {
          const double v = spd_sum8(c, e) * sc;
          P.Ginv[(int64_t)i * n + j] = v;
          P.Ginv[(int64_t)j * n + i] = v;
        }
      }
    }
  } else if (P.Ginv) {
    // Ginv = X^T X, lower half computed (four independent accumulators per element), mirrored on store
    for (int e = tid; e < n * (n + 1) / 2; e += nt) {
      int i = (int)((sqrt(8.0 * e + 1.0) - 1.0) * 0.5);
      while (i * (i + 1) / 2 > e) --i;
      while ((i + 1) * (i + 2) / 2 <= e) ++i;
      const int j = e - i * (i + 1) / 2;       // j <= i
      double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
      int k = i;
      for (; k + 3 < n; k += 4) {
        s0 = fma(Lp[pk(k, i)], Lp[pk(k, j)], s0);
        s1 = fma(Lp[pk(k + 1, i)], Lp[pk(k + 1, j)], s1);
        s2 = fma(Lp[pk(k + 2, i)], Lp[pk(k + 2, j)], s2);
        s3 = fma(Lp[pk(k + 3, i)], Lp[pk(k + 3, j)], s3);
      }
      for (; k < n; ++k) s0 = fma(Lp[pk(k, i)], Lp[pk(k, j)], s0);
      const double v = ((s0 + s1) + (s2 + s3)) * s_scale[3];
      P.Ginv[(int64_t)i * n + j] = v;
      P.Ginv[(int64_t)j * n + i] = v;
    }
  }
  SPD_LAP(t_c);
#ifdef RT_SPD_PROF
  if (tid == 0) printf("spd n=%d inverse %lld write Linv %lld Ginv %lld\n", n, t_a, t_b, t_c);
#endif
}

}  // namespace small
}  // namespace rt
