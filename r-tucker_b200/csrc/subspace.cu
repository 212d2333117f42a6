// Dominant invariant subspace of symmetric PSD matrices WITHOUT an eigen-decomposition, in fp64 on
// the fp64 tensor cores (DMMA), one persistent cooperative launch for a batch of problems.
//
// Used by the HOSVD / SF-HOSVD inside the retraction (reference: Tucker.round / SFTucker.round of
// tucker_riemopt, called at src/model/asymmetric/optim.py:108 and symmetric/optim.py:55,102).  The
// retraction only needs an ORTHONORMAL BASIS of the dominant r_i-dimensional invariant subspace of each
// (2 r_i x 2 r_i) unfolding Gram: the new point X_new = T x_i (Y_i Y_i^T) does not depend on the basis.
// The reference gets it from cuSOLVER gesvd; round 1 of this library from a block-Jacobi eigensolver
// (eig.cu: ~3.5 ms per 400 x 400 problem, latency-bound on serial rotation chains).  Here:
//
//   1. trace-correcting purification (Niklasson's TC2): X_0 = N / ||N||_F has its spectrum in [0, 1];
//        X_{k+1} = X_k^2          if tr X_k >  r     (pushes eigenvalues towards 0)
//                  2 X_k - X_k^2  otherwise           (pushes eigenvalues towards 1)
//      converges to the spectral projector P onto the r dominant eigenvectors with NO knowledge of the
//      eigenvalue that separates them; one symmetric n^3 product per iteration, ~log2(||N|| / gap) + 10
//      iterations (30-60 for the graded spectra of a training run).  tr X_k^2 comes out of the product's
//      epilogue; the idempotency defect tr X_k - tr X_k^2 is the stopping test.
//   2. orthonormal basis of range(P): Newton-Schulz polar iteration Z <- Z (1.5 I - 0.5 Z^T Z) started
//      from the first r columns of P (singular values = cosines of the principal angles to the old
//      subspace, in (0, 1]); 3-20 iterations, quadratically convergent at the end.
//
// Everything is a GEMM with k-contiguous operand rows ("NT"), so ONE tile routine serves all phases:
// a CTA owns a 32 x 32 output tile, its 8 warps split K, each warp keeps a 32 x 32 fp64 accumulator
// in registers (16 DMMA m8n8k4 per k-step, fragments loaded straight from L2 with ld.global.cg: the
// operands are rewritten by other CTAs every iteration, L1 must not keep them), partials are summed
// in a fixed order through shared memory.  All reductions (traces, defects) go through per-tile
// slots that every CTA sums in the same order: the result is bit-identical on every replica of an
// entity-sharded run, which keeps the replicated cores identical.
#include "prims.cuh"
#include <math.h>
#include <stdlib.h>

namespace rt {

constexpr int ST = 32;                 // tile edge
constexpr int SLD = 34;                // padded row stride of a warp partial in shared memory
constexpr int kSubThreads = 256;
constexpr int kSubWarps = 8;
constexpr int kSubMaxProblems = 4;
constexpr int kSlotsPerProblem = 160;  // >= tiles with a reduction contribution per round (T (T+1) / 2, T <= 16)
constexpr int kTc2MaxIter = 120;
constexpr int kNsMaxIter = 60;

struct SubProblem {
  const double* N_in;   // [n][n]
  double* Y_out;        // [n][ldy], first r columns are written
  double* X[2];         // [np][np] ping-pong
  double* Z[2];         // [np][rp]
  double* Zt[2];        // [rp][np]
  double* G;            // [rp][rp]
  double* slots;        // [2][kSlotsPerProblem]
  int* info;            // [4]: tc2 iterations, ns iterations, flags
  int n, r, np, rp, ldy;
};

struct SubBatch {
  SubProblem p[kSubMaxProblems];
  int count;
  unsigned int* bar;    // grid barrier counter (zeroed by the host before the launch)
  double* scratch;      // [gridDim][2 * kSubMaxProblems] per-CTA partials of phase 0
  int debug;            // RT_SUB_PRINT=1: print the iteration counts of every problem
};

enum SubState { S_TC2 = 0, S_COPY = 1, S_NSG = 2, S_NSZ = 3, S_DONE = 4 };

// C(32 x 32) = A[i0.., :K] * B[j0.., :K]^T with rows of A and B contiguous in k.  The 8 warps split K
// (K is a multiple of 32); the sum of their partials lands in red[0] (fixed order).  `out[m]` of thread t
// is element e = t + 256 m, (row, col) = (e / 32, e % 32).
__device__ __forceinline__ void tile_nt(const double* __restrict__ A, int lda, int i0, const double* __restrict__ B,
                                        int ldb, int j0, int K, double* red, double (&out)[4]) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int kw = K / kSubWarps;              // multiple of 4
  const int k0 = warp * kw;
  double c[4][4][2];
#pragma unroll
  for (int ti = 0; ti < 4; ++ti)
#pragma unroll
    for (int tj = 0; tj < 4; ++tj) { c[ti][tj][0] = 0.0; c[ti][tj][1] = 0.0; }
  const double* pa = A + (int64_t)(i0 + g) * lda + k0 + t;
  const double* pb = B + (int64_t)(j0 + g) * ldb + k0 + t;
  const int64_t sa = (int64_t)8 * lda, sb = (int64_t)8 * ldb;
  // three register buffers: the loads of step s + 2 are in flight while step s is multiplied (an L2 round trip is
  // longer than the 16 DMMAs of one step)
  double a0[4], b0[4], a1[4], b1[4], a2[4], b2[4];
  const int steps = kw / 4;
  auto load = [&](int st, double (&ra)[4], double (&rb)[4]) {
#pragma unroll
    for (int x = 0; x < 4; ++x) { ra[x] = __ldcg(pa + x * sa + 4 * st); rb[x] = __ldcg(pb + x * sb + 4 * st); }
  };
  auto mma = [&](const double (&ra)[4], const double (&rb)[4]) {
#pragma unroll
    for (int ti = 0; ti < 4; ++ti)
#pragma unroll
      for (int tj = 0; tj < 4; ++tj) dmma884(c[ti][tj][0], c[ti][tj][1], ra[ti], rb[tj]);
  };
  load(0, a0, b0);
  if (steps > 1) load(1, a1, b1);
  for (int st = 0; st < steps; st += 3) {
    if (st + 2 < steps) load(st + 2, a2, b2);
    mma(a0, b0);
    if (st + 1 >= steps) break;
    if (st + 3 < steps) load(st + 3, a0, b0);
    mma(a1, b1);
    if (st + 2 >= steps) break;
    if (st + 4 < steps) load(st + 4, a1, b1);
    mma(a2, b2);
  }
  double* mine = red + warp * (ST * SLD);
#pragma unroll
  for (int ti = 0; ti < 4; ++ti)
#pragma unroll
    for (int tj = 0; tj < 4; ++tj)
      *reinterpret_cast<double2*>(&mine[(8 * ti + g) * SLD + 8 * tj + 2 * t]) = make_double2(c[ti][tj][0], c[ti][tj][1]);
  __syncthreads();
#pragma unroll
  for (int m = 0; m < 4; ++m) {
    const int e = threadIdx.x + kSubThreads * m;
    const int row = e >> 5, col = e & 31;
    double s = 0.0;
#pragma unroll
    for (int w = 0; w < kSubWarps; ++w) s += red[w * (ST * SLD) + row * SLD + col];
    out[m] = s;
  }
  __syncthreads();
}

// sum of `count` (<= 160) slots in a fixed order, by one warp; every warp of every CTA gets the same bits
__device__ __forceinline__ double slot_sum(const double* slots, int count) {
  const int lane = threadIdx.x & 31;
  double v = 0.0;
  for (int i = lane; i < count; i += 32) v += __ldcg(slots + i);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// One CTA per SM: with two (296 CTAs, 128 registers) a round costs 18 us instead of 9 (spills in the tile routine and a
// grid barrier twice as wide outweigh the second wave), tools/subspace_bench.py.
constexpr int kSubCtasPerSm = 1;
__global__ void __launch_bounds__(kSubThreads, kSubCtasPerSm)
subspace_kernel(SubBatch batch) {
  extern __shared__ __align__(16) double ssm[];          // [8][32][SLD] warp partials
  __shared__ double sh_red[kSubWarps];
  const int tid = threadIdx.x;
  const int gtid = blockIdx.x * kSubThreads + tid;
  const int nthreads = gridDim.x * kSubThreads;
  unsigned int bar_target = 0u;
  const int count = batch.count;

  // ---- phase 0: ||N||_F^2 and tr N (deterministic two-stage sums) ----
  for (int pi = 0; pi < count; ++pi) {
    const SubProblem& P = batch.p[pi];
    double f2 = 0.0, tr = 0.0;
    const int nn = P.n * P.n;
    for (int e = gtid; e < nn; e += nthreads) {
      const double v = P.N_in[e];
      f2 = fma(v, v, f2);
      const int i = e / P.n;
      if (e - i * P.n == i) tr += v;
    }
    f2 = cta_sum<kSubWarps>(f2, sh_red);
    tr = cta_sum<kSubWarps>(tr, sh_red);
    if (tid == 0) {
      batch.scratch[(int64_t)blockIdx.x * (2 * kSubMaxProblems) + 2 * pi] = f2;
      batch.scratch[(int64_t)blockIdx.x * (2 * kSubMaxProblems) + 2 * pi + 1] = tr;
    }
  }
  grid_barrier(batch.bar, bar_target);
  // per-problem state: identical in every CTA (same inputs, same order of operations), kept in shared memory
  __shared__ double trace[kSubMaxProblems];
  __shared__ int state[kSubMaxProblems], iters[kSubMaxProblems], ns_iters[kSubMaxProblems], cur[kSubMaxProblems],
      zcur[kSubMaxProblems], ns_last[kSubMaxProblems];
  for (int pi = 0; pi < count; ++pi) {
    const SubProblem& P = batch.p[pi];
    double f2 = 0.0, tr = 0.0;
    for (int b = tid & 31; b < (int)gridDim.x; b += 32) {
      f2 += __ldcg(&batch.scratch[(int64_t)b * (2 * kSubMaxProblems) + 2 * pi]);
      tr += __ldcg(&batch.scratch[(int64_t)b * (2 * kSubMaxProblems) + 2 * pi + 1]);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      f2 += __shfl_xor_sync(0xffffffffu, f2, o);
      tr += __shfl_xor_sync(0xffffffffu, tr, o);
    }
    const double fro = sqrt(f2);
    const double inv = fro > 0.0 ? 1.0 / fro : 0.0;
    if (tid == 0) {
      trace[pi] = tr * inv;
      state[pi] = S_TC2; iters[pi] = 0; ns_iters[pi] = 0; cur[pi] = 0; zcur[pi] = 0; ns_last[pi] = 0;
    }
    // X_0 = N / ||N||_F, zero padded
    const int np = P.np;
    for (int e = gtid; e < np * np; e += nthreads) {
      const int i = e / np, j = e - i * np;
      P.X[0][e] = (i < P.n && j < P.n) ? P.N_in[(int64_t)i * P.n + j] * inv : 0.0;
    }
  }
  grid_barrier(batch.bar, bar_target);

  int round = 0;
  for (;;) {
    // ---- unit list of this round ----
    int ubeg[kSubMaxProblems + 1];
    ubeg[0] = 0;
    bool any = false;
    for (int pi = 0; pi < count; ++pi) {
      const SubProblem& P = batch.p[pi];
      const int T = P.np / ST, Tr = P.rp / ST;
      int nu = 0;
      switch (state[pi]) {
        case S_TC2: nu = T * (T + 1) / 2; break;
        case S_COPY: nu = T * Tr; break;
        case S_NSG: nu = Tr * (Tr + 1) / 2; break;
        case S_NSZ: nu = T * Tr; break;
        default: nu = 0;
      }
      any |= state[pi] != S_DONE;
      ubeg[pi + 1] = ubeg[pi] + nu;
    }
    if (!any) break;
    const int par = round & 1;
    for (int u = blockIdx.x; u < ubeg[count]; u += gridDim.x) {
      int pi = 0;
      while (u >= ubeg[pi + 1]) ++pi;
      const int lu = u - ubeg[pi];
      const SubProblem& P = batch.p[pi];
      const int np = P.np, rp = P.rp, T = np / ST, Tr = rp / ST;
      double* slots = P.slots + par * kSlotsPerProblem;
      double acc[4];
      if (state[pi] == S_TC2) {
        int ti, tj;
        sym_tile(lu, T, ti, tj);
        const double* X = P.X[cur[pi]];
        double* Xn = P.X[cur[pi] ^ 1];
        double xo[4];                      // this thread's entries of X_k (for 2 X - X^2), fetched behind the product
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int e = tid + kSubThreads * m;
          xo[m] = __ldcg(&X[(int64_t)(ti * ST + (e >> 5)) * np + tj * ST + (e & 31)]);
        }
        tile_nt(X, np, ti * ST, X, np, tj * ST, np, ssm, acc);
        const bool square = trace[pi] > (double)P.r;
        double trc = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int e = tid + kSubThreads * m;
          const int i = ti * ST + (e >> 5), j = tj * ST + (e & 31);
          const double c = acc[m];
          if (ti == tj && i == j) trc += c;
          const double v = square ? c : 2.0 * xo[m] - c;
          Xn[(int64_t)i * np + j] = v;
          if (ti != tj) Xn[(int64_t)j * np + i] = v;
        }
        if (ti == tj) {                      // slot ti: trace of X^2 over this diagonal tile
          trc = cta_sum<kSubWarps>(trc, sh_red);
          if (tid == 0) slots[ti] = trc;
        }
      } else if (state[pi] == S_COPY) {
        // Z = P[:, :r] (zero padded), Zt = its transpose: P is symmetric, so Zt rows are P rows
        const int ti = lu / Tr, tj = lu - ti * Tr;
        const double* X = P.X[cur[pi]];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int e = tid + kSubThreads * m;
          const int i = ti * ST + (e >> 5), j = tj * ST + (e & 31);
          const double v = (j < P.r) ? __ldcg(&X[(int64_t)i * np + j]) : 0.0;
          P.Z[0][(int64_t)i * rp + j] = v;
          P.Zt[0][(int64_t)j * np + i] = v;
        }
      } else if (state[pi] == S_NSG) {
        int ti, tj;
        sym_tile(lu, Tr, ti, tj);
        const double* Zt = P.Zt[zcur[pi]];
        tile_nt(Zt, np, ti * ST, Zt, np, tj * ST, np, ssm, acc);
        double err2 = 0.0;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int e = tid + kSubThreads * m;
          const int i = ti * ST + (e >> 5), j = tj * ST + (e & 31);
          const double gij = acc[m];
          P.G[(int64_t)i * rp + j] = gij;
          if (ti != tj) P.G[(int64_t)j * rp + i] = gij;
          if (i < P.r && j < P.r) {
            const double d = (i == j ? 1.0 : 0.0) - gij;
            err2 = fma(d, d, err2);
          }
        }
        err2 = cta_sum<kSubWarps>(err2, sh_red);
        if (tid == 0) slots[lu] = (ti == tj) ? err2 : 2.0 * err2;
      } else if (state[pi] == S_NSZ) {
        const int ti = lu / Tr, tj = lu - ti * Tr;
        const double* Z = P.Z[zcur[pi]];
        double zo[4];
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int e = tid + kSubThreads * m;
          zo[m] = __ldcg(&Z[(int64_t)(ti * ST + (e >> 5)) * rp + tj * ST + (e & 31)]);
        }
        tile_nt(Z, rp, ti * ST, P.G, rp, tj * ST, rp, ssm, acc);
        const bool last = ns_last[pi] != 0;
#pragma unroll
        for (int m = 0; m < 4; ++m) {
          const int e = tid + kSubThreads * m;
          const int i = ti * ST + (e >> 5), j = tj * ST + (e & 31);
          const double v = 1.5 * zo[m] - 0.5 * acc[m];
          if (last) {
            if (i < P.n && j < P.r) P.Y_out[(int64_t)i * P.ldy + j] = v;
          } else {
            P.Z[zcur[pi] ^ 1][(int64_t)i * rp + j] = v;
            P.Zt[zcur[pi] ^ 1][(int64_t)j * np + i] = v;
          }
        }
      }
    }
    grid_barrier(batch.bar, bar_target);
    // ---- state update: every CTA reads the same slots and takes the same decisions (warp 0, then broadcast
    //      through shared memory) ----
    if (tid < 32) {
      for (int pi = 0; pi < count; ++pi) {
        const SubProblem& P = batch.p[pi];
        const int T = P.np / ST, Tr = P.rp / ST;
        const double* slots = P.slots + par * kSlotsPerProblem;
        const int st = state[pi];
        if (st == S_TC2) {
          const double trc = slot_sum(slots, T);
          const double tr = trace[pi];
          const double idem = tr - trc;                       // tr X_k - tr X_k^2 = sum lambda (1 - lambda) >= 0
          const bool conv = idem < 1e-11 && fabs(tr - (double)P.r) < 0.25;
          __syncwarp();
          if (tid == 0) {
            trace[pi] = (tr > (double)P.r) ? trc : 2.0 * tr - trc;
            cur[pi] ^= 1;
            ++iters[pi];
            if (conv || iters[pi] >= kTc2MaxIter) state[pi] = S_COPY;
          }
        } else if (st == S_COPY) {
          if (tid == 0) state[pi] = S_NSG;
        } else if (st == S_NSG) {
          const double err2 = slot_sum(slots, Tr * (Tr + 1) / 2);
          if (tid == 0) {
            ++ns_iters[pi];
            // quadratic convergence: a defect below 1e-6 becomes ~1e-12 (rounding level) after one more update
            ns_last[pi] = ((err2 < 1e-12) || ns_iters[pi] >= kNsMaxIter) ? 1 : 0;
            state[pi] = S_NSZ;
          }
        } else if (st == S_NSZ) {
          if (tid == 0) {
            if (ns_last[pi]) {
              state[pi] = S_DONE;
              if (blockIdx.x == 0 && P.info) { P.info[0] = iters[pi]; P.info[1] = ns_iters[pi]; }
              if (blockIdx.x == 0 && batch.debug) printf("subspace problem %d (n=%d r=%d): purification %d rounds, Newton-Schulz %d x 2 rounds\n", pi, P.n, P.r, iters[pi], ns_iters[pi]);
            } else {
              zcur[pi] ^= 1;
              state[pi] = S_NSG;
            }
          }
        }
        __syncwarp();
      }
    }
    __syncthreads();
    ++round;
  }
}

struct SubLayout {
  int np, rp;
  size_t X[2], Z[2], Zt[2], G, slots, info, total;
};

static SubLayout sub_layout(int n, int r) {
  SubLayout L;
  L.np = cdiv(n, ST) * ST;
  L.rp = cdiv(r, ST) * ST;
  WsArena ws;
  for (int k = 0; k < 2; ++k) L.X[k] = ws.take(sizeof(double) * L.np * L.np);
  for (int k = 0; k < 2; ++k) L.Z[k] = ws.take(sizeof(double) * L.np * L.rp);
  for (int k = 0; k < 2; ++k) L.Zt[k] = ws.take(sizeof(double) * L.np * L.rp);
  L.G = ws.take(sizeof(double) * L.rp * L.rp);
  L.slots = ws.take(sizeof(double) * 2 * kSlotsPerProblem);
  L.info = ws.take(sizeof(int) * 4);
  L.total = ws.o;
  return L;
}

size_t subspace_ws_bytes(int n, int r) { return sub_layout(n, r).total; }
// shared by the whole batch: barrier counter + per-CTA phase-0 partials
size_t subspace_shared_ws_bytes() { return 256 + sizeof(double) * 2 * kSubMaxProblems * 1024; }

// Orthonormal bases Y_i (n_i x r_i, row stride ldy_i) of the dominant r_i-dimensional invariant subspaces of
// `count` (<= 4) symmetric PSD matrices, one cooperative launch.  ws[i]: subspace_ws_bytes(n_i, r_i) bytes;
// shared_ws: subspace_shared_ws_bytes() bytes.  info[i] (optional, device int[4]): TC2 / Newton-Schulz iterations.
int subspace_batch(int count, const double* const* N, const int* n, const int* r, double* const* Y, const int* ldy,
                   void* const* ws, void* shared_ws, int* const* info, cudaStream_t s) {
  RT_REQUIRE(count >= 1 && count <= kSubMaxProblems, "subspace_batch: count=%d out of range", count);
  SubBatch b{};
  b.count = count;
  b.bar = (unsigned int*)shared_ws;
  b.scratch = (double*)((char*)shared_ws + 256);
  { static const int dbg = getenv("RT_SUB_PRINT") ? atoi(getenv("RT_SUB_PRINT")) : 0; b.debug = dbg; }
  for (int i = 0; i < count; ++i) {
    RT_REQUIRE(n[i] >= 1 && n[i] <= 512 && r[i] >= 1 && r[i] <= n[i], "subspace_batch: n=%d r=%d out of range", n[i], r[i]);
    SubLayout L = sub_layout(n[i], r[i]);
    char* base = (char*)ws[i];
    SubProblem& P = b.p[i];
    P.N_in = N[i]; P.Y_out = Y[i]; P.ldy = ldy[i];
    for (int k = 0; k < 2; ++k) {
      P.X[k] = (double*)(base + L.X[k]); P.Z[k] = (double*)(base + L.Z[k]); P.Zt[k] = (double*)(base + L.Zt[k]);
    }
    P.G = (double*)(base + L.G);
    P.slots = (double*)(base + L.slots);
    P.info = info ? info[i] : nullptr;
    P.n = n[i]; P.r = r[i]; P.np = L.np; P.rp = L.rp;
  }
  RT_CHECK_CUDA(cudaMemsetAsync(b.bar, 0, 256, s));
  const size_t smem = sizeof(double) * kSubWarps * ST * SLD;
  RT_CHECK_CUDA(cudaFuncSetAttribute(subspace_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid = kSubCtasPerSm * sm_count();
  if (grid > 1024) grid = 1024;
  void* args[] = {(void*)&b};
  RT_CHECK_CUDA(cudaLaunchCooperativeKernel((const void*)subspace_kernel, dim3(grid), dim3(kSubThreads), args, smem, s));
  ++g_launches;
  return 0;
}

}  // namespace rt

extern "C" size_t rt_dominant_subspace_ws_bytes(int n, int r) {
  if (n <= 0 || r <= 0) return 0;
  return rt::align_up(rt::subspace_ws_bytes(n, r), 256) + rt::subspace_shared_ws_bytes();
}

extern "C" int rt_dominant_subspace(const double* A, int n, int r, double* Y, int* info, void* ws, void* stream) {
  RT_REQUIRE(ws != nullptr && A != nullptr && Y != nullptr, "rt_dominant_subspace: NULL argument");
  const double* Ain[1] = {A};
  double* Yo[1] = {Y};
  void* wss[1] = {ws};
  int* inf[1] = {info};
  void* shared = (char*)ws + rt::align_up(rt::subspace_ws_bytes(n, r), 256);
  return rt::subspace_batch(1, Ain, &n, &r, Yo, &r, wss, shared, inf, (cudaStream_t)stream);
}
