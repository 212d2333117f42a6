// Executor of the N-independent ("small") stage: ONE persistent cooperative launch runs a whole
// program of dependent small operations -- strided GEMMs on the fp64 tensor cores, split-K
// reductions, elementwise passes, dot products -- with a grid barrier between dependency levels,
// instead of one launch per operation (round 1: ~130 launches of 10-25 us per optimiser step for
// the projection / retraction arithmetic of tucker_riemopt, call sites
// src/model/asymmetric/optim.py:86-92,106-109).
//
// The host (small.cu) RECORDS operations in program order together with the byte ranges they read
// and write; levels are assigned from the read/write hazards, so independent operations (the three
// mode products of a retraction, the thirteen unfolding Grams, ...) share a level and fill the
// machine together.  Work units of a level (32 x 32 output tiles x K splits, 2048-element chunks)
// are dealt round-robin to the CTAs.
//
// GEMM unit: a CTA owns a 32 x 32 tile of C = alpha * sum_k A[m,k] B[k,n] (+ beta C) for arbitrary
// element strides and a two-level K index (mode products and unfolding Grams of r0 x r1 x r2
// tensors without permuting them); its 8 warps interleave the k-steps (4 deep, DMMA m8n8k4), each
// keeps a 32 x 32 fp64 accumulator in registers, operands are converted to fp64 on load (fp32 or
// fp64 storage), partial sums are combined in a fixed order through shared memory.  Long
// contractions with few tiles are split over CTAs; the partial tiles are summed by a REDUCE
// operation of the next level in split order -- deterministic, bit-identical on every replica.
#pragma once
#include "prims.cuh"
#include <math.h>

namespace rt {
namespace small {

enum OpKind : int { OP_GEMM = 0, OP_REDUCE = 1, OP_EW = 2, OP_DOT = 3, OP_DOTFIN = 4 };
enum DType : int { DT_F32 = 0, DT_F64 = 1 };
enum EwKind : int {
  EW_CVT = 0,          // z[i] (tz) = s * x[i] (tx),  s = s0 * (d0 ? (p0 ? *d0 * *d0 : *d0) : 1)
  EW_AXPBY64,          // z = a x + b y (fp64; y may be NULL), a = s0 * (d0 ? *d0 : 1), b = s1 * (d1 ? *d1 : 1)
  EW_CORE_MINUS_LR,    // z(f64) = x(f32) - *d0 * y(f32)
  EW_GRAD_CORE,        // z(f32) = x(f32) + 2 * d0[1] * y(f32)
  EW_CVT_2D,           // z[i, j] (ld p1, tz) = x[i, j] (ld p0, tx), rows p2, cols p3
  EW_TRANSPOSE_INTO,   // z[a, b] (ld p1) = x[b, a] (ld p0) for an n x n fp64 matrix, n = p2
  EW_SYMM_LOWER,       // z[i, j] = z[j, i] for j > i (n = p2, ld = p0), fp64 in place
  EW_ZERO64,           // z[i] = 0 (fp64)
  EW_ADAM_FINISH,      // SFTuckerAdam coefficients (symmetric/optim.py:133-145): x = ||g||^2, y = alpha out, z = norm out,
                       // d0 = hyper (hyper[2] <- momentum coefficient), d1 = adam state (updated in place)
  EW_NORM_FINISH,      // z[0] = sqrt(max(x[0], 0)); y[0] = d0[3] != 0 ? d0[3] / z[0] : 1   (z = norm, y = alpha: both outputs)
};

struct GemmPart {
  const void* A; const void* B; void* C;
  double* partial;
  const double* alpha_dev;
  int64_t a_m, a_k1, a_k2, b_k1, b_k2, b_n, c_m, c_n, a_b, b_b, c_b;
  double alpha, beta;
  int ta, tb, tc, m, n, K1, K2, batch, ksplit, steps_per_split, tiles_m, tiles_n;
  int thin, sym;    // sym: C = C^T (A = B, a Gram): only tiles with tn >= tm are computed, each is stored twice.  thin: m <= 16, K <= 32 (a mode product along a small rank): one output COLUMN per thread (thin_unit)
};
struct EwPart {
  const void* x; const void* y; void* z;
  const double* d0; const double* d1;
  int64_t count, p0, p1, p2, p3;
  double s0, s1;
  int tx, tz;
};
struct Op {
  int kind, level, units, ew;
  union { GemmPart g; EwPart e; };
};
// A program travels to the device as a kernel PARAMETER (by value: captured as is by CUDA graphs, no staging
// buffer to keep alive); CUDA >= 12.1 allows 32764 bytes of parameters.
constexpr int kMaxOps = 146;
struct Program {
  int nops;
  unsigned int* bar;
  Op ops[kMaxOps];
};
static_assert(sizeof(Program) <= 32000, "program must fit the kernel parameter space");

constexpr int XT = 32;            // tile edge
constexpr int XLD = 34;           // padded row stride of a warp partial
constexpr int kExecThreads = 256;
constexpr int kExecWarps = 8;
constexpr int kEwChunk = 2048;    // elements per elementwise unit
constexpr int kReduceChunk = 1024;

__device__ __forceinline__ double ld_as_f64(const void* p, int64_t i, int t) {
  return t == DT_F64 ? __ldcg(reinterpret_cast<const double*>(p) + i) : (double)__ldcg(reinterpret_cast<const float*>(p) + i);
}
__device__ __forceinline__ void st_from_f64(void* p, int64_t i, int t, double v) {
  if (t == DT_F64) reinterpret_cast<double*>(p)[i] = v; else reinterpret_cast<float*>(p)[i] = (float)v;
}

template <typename TA, typename TB>
__device__ __noinline__ void gemm_unit(const GemmPart& op, int unit, double* red) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  int rem = unit;
  const int z = rem % op.ksplit; rem /= op.ksplit;
  int tn, tm, b;
  if (op.sym) {                          // upper triangle of tiles, row by row: tm <= tn
    const int T = op.tiles_n, ntri = T * (T + 1) / 2;
    int tt = rem % ntri;
    b = rem / ntri;
    tm = 0;
    while (tt >= T - tm) { tt -= T - tm; ++tm; }
    tn = tm + tt;
  } else {
    tn = rem % op.tiles_n; rem /= op.tiles_n;
    tm = rem % op.tiles_m;
    b = rem / op.tiles_m;
  }
  const bool mirror = op.sym && tm != tn;
  const TA* A = reinterpret_cast<const TA*>(op.A) + (int64_t)b * op.a_b;
  const TB* B = reinterpret_cast<const TB*>(op.B) + (int64_t)b * op.b_b;
  const int i0 = tm * XT, j0 = tn * XT;
  const int nk2 = (op.K2 + 3) >> 2;
  const int S = op.K1 * nk2;
  const int s_beg = z * op.steps_per_split;
  const int s_end = min(S, s_beg + op.steps_per_split);
  const TA* pa[4]; const TB* pb[4];
  bool va[4], vb[4];
#pragma unroll
  for (int x = 0; x < 4; ++x) {
    const int row = i0 + 8 * x + g, col = j0 + 8 * x + g;
    va[x] = row < op.m; vb[x] = col < op.n;
    pa[x] = A + (int64_t)(va[x] ? row : 0) * op.a_m;
    pb[x] = B + (int64_t)(vb[x] ? col : 0) * op.b_n;
  }
  double c[4][4][2];
#pragma unroll
  for (int ti = 0; ti < 4; ++ti)
#pragma unroll
    for (int tj = 0; tj < 4; ++tj) { c[ti][tj][0] = 0.0; c[ti][tj][1] = 0.0; }
  double a0[4], b0[4], a1[4], b1[4], a2[4], b2[4];
  auto load = [&](int s, double (&ra)[4], double (&rb)[4]) {
    const int k1 = s / nk2;
    const int k2 = ((s - k1 * nk2) << 2) + t;
    const bool kv = k2 < op.K2;
    const int64_t oa = (int64_t)k1 * op.a_k1 + (int64_t)k2 * op.a_k2;
    const int64_t ob = (int64_t)k1 * op.b_k1 + (int64_t)k2 * op.b_k2;
#pragma unroll
    for (int x = 0; x < 4; ++x) {
      ra[x] = (va[x] && kv) ? (double)__ldcg(pa[x] + oa) : 0.0;
      rb[x] = (vb[x] && kv) ? (double)__ldcg(pb[x] + ob) : 0.0;
    }
  };
  auto mma = [&](const double (&ra)[4], const double (&rb)[4]) {
#pragma unroll
    for (int ti = 0; ti < 4; ++ti)
#pragma unroll
      for (int tj = 0; tj < 4; ++tj) dmma884(c[ti][tj][0], c[ti][tj][1], ra[ti], rb[tj]);
  };
  // three register buffers: the loads of two steps ahead are in flight while a step is multiplied
  constexpr int W = kExecWarps;
  int s = s_beg + warp;
  if (s < s_end) load(s, a0, b0);
  if (s + W < s_end) load(s + W, a1, b1);
  for (; s < s_end; s += 3 * W) {
    if (s + 2 * W < s_end) load(s + 2 * W, a2, b2);
    mma(a0, b0);
    if (s + W >= s_end) break;
    if (s + 3 * W < s_end) load(s + 3 * W, a0, b0);
    mma(a1, b1);
    if (s + 2 * W >= s_end) break;
    if (s + 4 * W < s_end) load(s + 4 * W, a1, b1);
    mma(a2, b2);
  }
  double* mine = red + warp * (XT * XLD);
#pragma unroll
  for (int ti = 0; ti < 4; ++ti)
#pragma unroll
    for (int tj = 0; tj < 4; ++tj)
      *reinterpret_cast<double2*>(&mine[(8 * ti + g) * XLD + 8 * tj + 2 * t]) = make_double2(c[ti][tj][0], c[ti][tj][1]);
  __syncthreads();
  const double alpha = op.alpha * (op.alpha_dev ? __ldcg(op.alpha_dev) : 1.0);
#pragma unroll
  for (int mI = 0; mI < 4; ++mI) {
    const int e = threadIdx.x + kExecThreads * mI;
    const int row = e >> 5, col = e & 31;
    double sum = 0.0;
#pragma unroll
    for (int w = 0; w < kExecWarps; ++w) sum += red[w * (XT * XLD) + row * XLD + col];
    const int mm = i0 + row, nn = j0 + col;
    if (mm < op.m && nn < op.n) {
      if (op.ksplit > 1) {
        op.partial[(((int64_t)z * op.batch + b) * op.m + mm) * op.n + nn] = sum;
        if (mirror) op.partial[(((int64_t)z * op.batch + b) * op.m + nn) * op.n + mm] = sum;
      } else {
        const int64_t ci = (int64_t)b * op.c_b + (int64_t)mm * op.c_m + (int64_t)nn * op.c_n;
        double v = alpha * sum;
        if (op.beta != 0.0) v += op.beta * ld_as_f64(op.C, ci, op.tc);
        st_from_f64(op.C, ci, op.tc, v);
        if (mirror) st_from_f64(op.C, (int64_t)b * op.c_b + (int64_t)nn * op.c_m + (int64_t)mm * op.c_n, op.tc, v);
      }
    }
  }
  __syncthreads();
}

// Thin GEMM unit: C[m, n] with m <= 16 rows and K <= 32 (the mode product along the relation rank, r0 = 10: out[a', x] =
// sum_a W[a', a] X[a, x] over 40 000 columns x).  As 32 x 32 DMMA tiles this was 1 250 units of three k-steps whose
// fixed cost (operand fetch, cross-warp reduction) is ~6 us each: 20-25 us per product, ten products per step.  Here a
// thread owns one column: K coalesced loads, m x K fp64 FMAs against the small matrix in shared memory, m coalesced stores.
constexpr int kThinM = 16, kThinK = 32, kThinCols = kExecThreads;
__device__ __forceinline__ void thin_unit(const GemmPart& op, int unit, double* As) {
  const int tid = threadIdx.x;
  const int K = op.K2;
  for (int e = tid; e < op.m * K; e += kExecThreads) {
    const int mm = e / K, k = e - mm * K;
    As[e] = ld_as_f64(op.A, (int64_t)mm * op.a_m + (int64_t)k * op.a_k2, op.ta);
  }
  __syncthreads();
  const int col = unit * kThinCols + tid;
  if (col < op.n) {
    double b[kThinK];
#pragma unroll
    for (int k = 0; k < kThinK; ++k) b[k] = k < K ? ld_as_f64(op.B, (int64_t)k * op.b_k2 + (int64_t)col * op.b_n, op.tb) : 0.0;
    const double alpha = op.alpha * (op.alpha_dev ? __ldcg(op.alpha_dev) : 1.0);
    for (int mm = 0; mm < op.m; ++mm) {
      double s0 = 0.0, s1 = 0.0;
#pragma unroll
      for (int k = 0; k < kThinK; k += 2) {
        if (k < K) s0 = fma(As[mm * K + k], b[k], s0);
        if (k + 1 < K) s1 = fma(As[mm * K + k + 1], b[k + 1], s1);
      }
      const int64_t ci = (int64_t)mm * op.c_m + (int64_t)col * op.c_n;
      double v = alpha * (s0 + s1);
      if (op.beta != 0.0) v += op.beta * ld_as_f64(op.C, ci, op.tc);
      st_from_f64(op.C, ci, op.tc, v);
    }
  }
  __syncthreads();
}

__device__ __forceinline__ void reduce_unit(const GemmPart& op, int unit) {
  const int64_t total = (int64_t)op.batch * op.m * op.n;
  const double alpha = op.alpha * (op.alpha_dev ? __ldcg(op.alpha_dev) : 1.0);
#pragma unroll
  for (int mI = 0; mI < kReduceChunk / kExecThreads; ++mI) {
    const int64_t e = (int64_t)unit * kReduceChunk + threadIdx.x + kExecThreads * mI;
    if (e >= total) continue;
    // 16 loads in flight per thread (a 63-way split summed 4 at a time was 16 dependent L2 round trips), fixed order
    double s0 = 0.0, s1 = 0.0, s2 = 0.0, s3 = 0.0;
    int zz = 0;
    for (; zz + 16 <= op.ksplit; zz += 16) {
      double v[16];
#pragma unroll
      for (int u = 0; u < 16; ++u) v[u] = __ldcg(op.partial + (int64_t)(zz + u) * total + e);
#pragma unroll
      for (int u = 0; u < 16; u += 4) { s0 += v[u]; s1 += v[u + 1]; s2 += v[u + 2]; s3 += v[u + 3]; }
    }
    for (; zz + 4 <= op.ksplit; zz += 4) {
      s0 += __ldcg(op.partial + (int64_t)zz * total + e);
      s1 += __ldcg(op.partial + (int64_t)(zz + 1) * total + e);
      s2 += __ldcg(op.partial + (int64_t)(zz + 2) * total + e);
      s3 += __ldcg(op.partial + (int64_t)(zz + 3) * total + e);
    }
    for (; zz < op.ksplit; ++zz) s0 += __ldcg(op.partial + (int64_t)zz * total + e);
    const double sum = (s0 + s1) + (s2 + s3);
    const int64_t mn = (int64_t)op.m * op.n;
    const int b = (int)(e / mn);
    const int64_t r = e - (int64_t)b * mn;
    const int mm = (int)(r / op.n), nn = (int)(r - (int64_t)mm * op.n);
    const int64_t ci = (int64_t)b * op.c_b + (int64_t)mm * op.c_m + (int64_t)nn * op.c_n;
    double v = alpha * sum;
    if (op.beta != 0.0) v += op.beta * ld_as_f64(op.C, ci, op.tc);
    st_from_f64(op.C, ci, op.tc, v);
  }
}

__device__ __forceinline__ void ew_unit(const EwPart& op, int ew, int unit) {
  const int64_t base = (int64_t)unit * kEwChunk;
  if (ew == EW_ADAM_FINISH) {
    if (threadIdx.x == 0) {
      double* st = const_cast<double*>(op.d1);          // [v, ratio_prev, t, beta1, beta2, eps, step_velocity, -]
      double* hyper = const_cast<double*>(op.d0);
      const double sq = fmax(__ldcg(reinterpret_cast<const double*>(op.x)), 0.0);
      const double nrm = sqrt(sq);
      const double v = __ldcg(st + 0), ratio_prev = __ldcg(st + 1), t = __ldcg(st + 2);
      const double b1 = __ldcg(st + 3), b2 = __ldcg(st + 4), eps = __ldcg(st + 5), vel = __ldcg(st + 6);
      const double vn = b2 * v + (1.0 - b2) * sq;
      const double e = floor(t / vel) + 1.0;            // step_t // step_velocity + 1
      const double vhat = vn / (1.0 - pow(b2, e));
      const double ratio = (1.0 - pow(b1, e)) * sqrt(vhat) + eps;
      reinterpret_cast<double*>(op.z)[0] = nrm;
      reinterpret_cast<double*>(const_cast<void*>(op.y))[0] = (1.0 - b1) / ratio;   // direction = momentum / ratio
      hyper[2] = b1 * ratio_prev / ratio;               // momentum_{k-1} = ratio_{k-1} * direction_{k-1}
      st[0] = vn; st[1] = ratio; st[2] = t + 1.0;
    }
    return;
  }
  if (ew == EW_NORM_FINISH) {
    if (threadIdx.x == 0) {
      const double nrm = sqrt(fmax(__ldcg(reinterpret_cast<const double*>(op.x)), 0.0));
      reinterpret_cast<double*>(op.z)[0] = nrm;
      const double ng = __ldcg(op.d0 + 3);
      reinterpret_cast<double*>(const_cast<void*>(op.y))[0] = (ng != 0.0) ? ng / nrm : 1.0;
    }
    return;
  }
  double sa = op.s0, sb = op.s1;
  if (ew == EW_CVT || ew == EW_AXPBY64) {
    if (op.d0) { const double d = __ldcg(op.d0); sa *= (ew == EW_CVT && op.p0) ? d * d : d; }
    if (op.d1) sb *= __ldcg(op.d1);
  } else if (ew == EW_CORE_MINUS_LR) {
    sa = __ldcg(op.d0);
  } else if (ew == EW_GRAD_CORE) {
    sa = 2.0 * __ldcg(op.d0 + 1);
  }
#pragma unroll
  for (int mI = 0; mI < kEwChunk / kExecThreads; ++mI) {
    const int64_t i = base + threadIdx.x + kExecThreads * mI;
    if (i >= op.count) continue;
    switch (ew) {
      case EW_CVT: st_from_f64(op.z, i, op.tz, sa * ld_as_f64(op.x, i, op.tx)); break;
      case EW_AXPBY64: {
        double v = sa * __ldcg(reinterpret_cast<const double*>(op.x) + i);
        if (op.y) v += sb * __ldcg(reinterpret_cast<const double*>(op.y) + i);
        reinterpret_cast<double*>(op.z)[i] = v;
        break;
      }
      case EW_CORE_MINUS_LR:
        reinterpret_cast<double*>(op.z)[i] = (double)__ldcg(reinterpret_cast<const float*>(op.x) + i) -
                                             sa * (double)__ldcg(reinterpret_cast<const float*>(op.y) + i);
        break;
      case EW_GRAD_CORE:
        reinterpret_cast<float*>(op.z)[i] = fmaf((float)sa, __ldcg(reinterpret_cast<const float*>(op.y) + i),
                                                 __ldcg(reinterpret_cast<const float*>(op.x) + i));
        break;
      case EW_CVT_2D: {
        const int64_t r = i / op.p3, cI = i - r * op.p3;
        st_from_f64(op.z, r * op.p1 + cI, op.tz, ld_as_f64(op.x, r * op.p0 + cI, op.tx));
        break;
      }
      case EW_TRANSPOSE_INTO: {
        const int64_t aI = i / op.p2, bI = i - aI * op.p2;
        reinterpret_cast<double*>(op.z)[aI * op.p1 + bI] = __ldcg(reinterpret_cast<const double*>(op.x) + bI * op.p0 + aI);
        break;
      }
      case EW_SYMM_LOWER: {
        const int64_t r = i / op.p2, cI = i - r * op.p2;
        if (cI > r) reinterpret_cast<double*>(op.z)[r * op.p0 + cI] = __ldcg(reinterpret_cast<const double*>(op.z) + cI * op.p0 + r);
        break;
      }
      case EW_ZERO64: reinterpret_cast<double*>(op.z)[i] = 0.0; break;
      default: break;
    }
  }
}

// DOT: z[unit] = sum over this unit's chunk of x[i] * y[i];  DOTFIN: z[0] = (p0 ? z[0] : 0) + s0 * sum_{i < count} x[i]
__device__ __forceinline__ void dot_unit(const EwPart& op, int unit, double* sh) {
  const int64_t base = (int64_t)unit * kEwChunk;
  double s = 0.0;
#pragma unroll
  for (int mI = 0; mI < kEwChunk / kExecThreads; ++mI) {
    const int64_t i = base + threadIdx.x + kExecThreads * mI;
    if (i < op.count) s = fma(ld_as_f64(op.x, i, op.tx), ld_as_f64(op.y, i, op.tz), s);
  }
  s = cta_sum<kExecWarps>(s, sh);
  if (threadIdx.x == 0) reinterpret_cast<double*>(op.z)[unit] = s;
}
__device__ __forceinline__ void dotfin_unit(const EwPart& op, double* sh) {
  const double* part = reinterpret_cast<const double*>(op.x);
  double s = 0.0;
  for (int64_t i = threadIdx.x; i < op.count; i += kExecThreads) s += __ldcg(part + i);
  s = cta_sum<kExecWarps>(s, sh);
  if (threadIdx.x == 0) {
    double* out = reinterpret_cast<double*>(op.z);
    out[0] = (op.p0 ? __ldcg(out) : 0.0) + op.s0 * s;
  }
}

// Two CTAs per SM: a unit is a chain of latency-bound phases (operand fetch from L2, 16 DMMAs per k-step, the
// cross-warp reduction), so a second resident CTA overlaps them (measured: -15 % on the whole small stage, with the
// 128-register cap costing a few hundred bytes of spills in the GEMM unit; tools/prof_one_step.py + RT_EXEC_PROF).
constexpr int kExecCtasPerSm = 2;
__global__ void __launch_bounds__(kExecThreads, kExecCtasPerSm)
small_exec_kernel(const __grid_constant__ Program prog) {
  extern __shared__ __align__(16) double xsm[];      // [8][32][XLD] warp partials
  __shared__ double sh_red[kExecWarps];
  __shared__ Op s_op;
  unsigned int bar_target = 0u;
  const int nops = prog.nops;
  int i = 0;
#ifdef RT_EXEC_PROF
  long long lv_t0 = clock64();
  __shared__ long long lv_cycles[64];
  __shared__ int lv_first[64], lv_last[64];
  int n_lv = 0;
#endif
  while (i < nops) {
    const int lv = prog.ops[i].level;
    int j = i, total = 0;
    while (j < nops && prog.ops[j].level == lv) { total += prog.ops[j].units; ++j; }
    int cached = -1;
    for (int u = blockIdx.x; u < total; u += gridDim.x) {
      int k = i, ub = 0;
      while (u >= ub + prog.ops[k].units) { ub += prog.ops[k].units; ++k; }
      if (k != cached) {
        __syncthreads();
        if (threadIdx.x == 0) s_op = prog.ops[k];   // the descriptor of this unit's operation, staged once per CTA
        __syncthreads();
        cached = k;
      }
      const Op& op = s_op;
      const int lu = u - ub;
      switch (op.kind) {
        case OP_GEMM:
          if (op.g.thin) thin_unit(op.g, lu, xsm);
          else if (op.g.ta == DT_F64 && op.g.tb == DT_F64) gemm_unit<double, double>(op.g, lu, xsm);
          else if (op.g.ta == DT_F32 && op.g.tb == DT_F32) gemm_unit<float, float>(op.g, lu, xsm);
          else if (op.g.ta == DT_F32) gemm_unit<float, double>(op.g, lu, xsm);
          else gemm_unit<double, float>(op.g, lu, xsm);
          break;
        case OP_REDUCE: reduce_unit(op.g, lu); break;
        case OP_EW: ew_unit(op.e, op.ew, lu); break;
        case OP_DOT: dot_unit(op.e, lu, sh_red); break;
        case OP_DOTFIN: dotfin_unit(op.e, sh_red); break;
        default: break;
      }
    }
#ifdef RT_EXEC_PROF
    const int i_first = i;
#endif
    i = j;
    if (i < nops) grid_barrier(prog.bar, bar_target);
#ifdef RT_EXEC_PROF
    if (blockIdx.x == 0 && threadIdx.x == 0) {
      const long long now = clock64();
      if (n_lv < 64) { lv_cycles[n_lv] = now - lv_t0; lv_first[n_lv] = i_first; lv_last[n_lv] = j; ++n_lv; }
      lv_t0 = clock64();
    }
#endif
  }
#ifdef RT_EXEC_PROF
  // per-level times of this program (CTA 0's clock, 1.9 GHz assumed); printed after the last level so that the
  // printf cost (~30 us each) does not perturb the measurement
  if (blockIdx.x == 0 && threadIdx.x == 0) {
    for (int l = 0; l < n_lv; ++l) {
      int ng = 0, ug = 0, K = 0, m = 0, n = 0, total = 0;
      for (int q = lv_first[l]; q < lv_last[l]; ++q) {
        total += prog.ops[q].units;
        if (prog.ops[q].kind == OP_GEMM) { ++ng; ug += prog.ops[q].units; K = prog.ops[q].g.K1 * prog.ops[q].g.K2; m = prog.ops[q].g.m; n = prog.ops[q].g.n; }
      }
      printf("  level %2d: %2d ops (%d gemm, %d gemm units, last m=%d n=%d K=%d) %4d units  %7.1f us\n", l, lv_last[l] - lv_first[l], ng, ug, m, n, K, total,
             (double)lv_cycles[l] / 1.9e3);
    }
    printf("program end (%d ops)\n", nops);
  }
#endif
  // A program launched as a programmatic dependent (Ctx::flush, Launch::kAfterPrimary) ends only after the kernel
  // before it has completed, so everything later on the stream sees that kernel's results.  Otherwise a no-op.
  pdl_wait();
}

}  // namespace small
}  // namespace rt
