// Batched symmetric eigen-decomposition by two-sided BLOCK JACOBI (fp64), one cooperative launch.
//
// Used for the HOSVD / SF-HOSVD inside the retraction (reference: Tucker.round / SFTucker.round
// of tucker_riemopt, called at src/model/asymmetric/optim.py:108 and symmetric/optim.py:55,102),
// where the left singular vectors of each unfolding of the rank-2r core are the eigenvectors of
// its (2r_i x 2r_i) Gram matrix.  The reference calls cuSOLVER gesvd on the unfoldings.
//
// Scheme: blocks of 16 indices; a round-robin tournament pairs the blocks; per round
//   phase A: one warp per block pair rotates every cross index pair of its 32x32 tile once (and, in
//            the first round of a sweep, every pair inside the two blocks) and publishes the product Q;
//   phase B: every 32x32 tile (pair k rows, pair l cols) becomes Q_k^T A_kl Q_l, and V <- V Q.
// grid.sync() separates the phases.  N-independent, latency-bound: reported separately from the
// HBM / tensor rooflines (SURVEY.md section 8d "N-independent serial part").
#include "common.h"
#include "tc.cuh"
#include <cooperative_groups.h>
#include <math.h>

namespace cg = cooperative_groups;

namespace rt {

constexpr int EB = 16;         // block size
constexpr int EP = 2 * EB;     // pair tile edge (32)
constexpr int ELD = EP + 2;    // padded smem leading dim (even: 16-byte aligned rows for LDS.128)
constexpr int kMaxProblems = 4;
constexpr int kEigThreads = 256;
constexpr int kEigWarps = kEigThreads / 32;
constexpr int kMaxSweeps = 20;
constexpr int kScaleSlot = 1 + kMaxSweeps;   // scal[kScaleSlot] = max |a_ij| (positive doubles order like uint64)
constexpr int kPermSlot = 2 + kMaxSweeps;    // scal[kPermSlot + i] = rank of eigenvalue i
static_assert(EP == 32, "phase B register blocking (4 rows x 8 cols per lane) assumes 32x32 tiles");

struct EigProblem {
  const double* A_in;  // [n][n] dense symmetric
  double* w;           // [n] descending
  double* V_out;       // [n][n] columns = eigenvectors
  double* Ap;          // [np][np] padded work copy
  double* Vp;          // [np][np]
  double* J;           // [npairs][EP*EP]
  int* skip;           // [npairs]
  double* scal;        // [0]=norm2, [1+sweep]=off2 of that sweep, scale, permutation
  int n, np, nb, npairs;
};

struct EigBatch {
  EigProblem p[kMaxProblems];
  int count;
  double stop;       // a problem is done once the off-diagonal mass SEEN in a sweep is <= stop * ||A||_F^2
  long long* prof;   // optional [gridDim][4] cycle counters: phase A, sync, phase B, sync
};

// round-robin tournament (circle method) on nb (even) players: pair k of round t
__device__ __forceinline__ void rr_pair(int nb, int t, int k, int& bi, int& bj) {
  const int m = nb - 1;
  if (k == 0) { bi = m; bj = t % m; }
  else { bi = (t + k) % m; bj = (t - k + m) % m; }
  if (bi > bj) { const int x = bi; bi = bj; bj = x; }
}

__device__ __forceinline__ int pair_index(int bi, int bj, int i) {  // i in [0, EP)
  return (i < EB) ? bi * EB + i : bj * EB + (i - EB);
}

// Rotation for the pivot with diagonal difference d = a_qq - a_pp and off-diagonal a = a_pq (fp32).  The ANGLE
// is evaluated in fp32 (MUFU + FFMA, a short dependent chain) and steers the fp32 tile at once; a second warp
// re-normalises (c, s) in fp64 one round later (a dependent fp64 operation costs ~80 cycles here), so the rotation
// that is accumulated into Q is orthogonal to ~1e-15.  An fp32-accurate angle leaves a residual of ~1e-7 |a_pq|
// instead of an exact zero, which only replaces the last quadratic step of the Jacobi iteration by one more sweep.
__device__ __forceinline__ void rotation(float d, float a, float& c, float& s) {
  c = 1.0f;
  s = 0.0f;
  if (a * a > 1e-34f) {   // entries are scaled to <= 1: keeps the fp32 chain inside float range
    // tan(2 theta) = 2 a / d:  cos(2 theta) = |d| / h,  h = sqrt(d^2 + 4 a^2)
    const float x = fmaf(d, d, 4.0f * a * a);
    const float rh = rsqrtf(x);
    const float y = fmaf(0.5f * fabsf(d), rh, 0.5f);       // cos^2(theta) in [0.5, 1]
    const float ry = rsqrtf(y);
    c = y * ry;
    s = (d >= 0.0f ? a : -a) * rh * ry;                     // sin(theta) = sin(2 theta) / (2 cos(theta))
  }
}
// (c0, s0) in fp32 -> the same rotation with c^2 + s^2 = 1 to ~1e-15 (fp64), off the critical path of the visit
__device__ __forceinline__ void renormalise(float c0f, float s0f, double& c, double& s) {
  const double c0 = (double)c0f, s0 = (double)s0f;
  const double e = fma(c0, c0, fma(s0, s0, -1.0));       // c0^2 + s0^2 - 1 ~ 1e-7
  const double f = fma(e, fma(e, 0.375, -0.5), 1.0);     // (1 + e)^(-1/2) to O(e^3)
  c = c0 * f;
  s = s0 * f;
}

__device__ __forceinline__ void cp_async16_d(double* dst_smem, const double* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n"
               :: "r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all_d() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// fp64 tensor-core MMA: D(8x8) += A(8x4) B(4x8); lane l holds A[l>>2][l&3], B[l&3][l>>2], C[l>>2][2*(l&3)+{0,1}]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};\n"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// C(32x32) = op(A) * B for one warp on the fp64 tensor cores.  A element (i, m) is read from
// As[i * ELD + m] (a_trans = false) or As[m * ELD + i] (a_trans = true); B element (m, j) = Bs[m * ELD + j].
template <bool A_TRANS>
__device__ __forceinline__ void warp_mm32(const double* As, const double* Bs, double (&c)[4][4][2], int lane) {
  const int g = lane >> 2, t = lane & 3;
#pragma unroll
  for (int ti = 0; ti < 4; ++ti)
#pragma unroll
    for (int tj = 0; tj < 4; ++tj) { c[ti][tj][0] = 0.0; c[ti][tj][1] = 0.0; }
#pragma unroll 2
  for (int kk = 0; kk < EP / 4; ++kk) {
    double a[4], b[4];
#pragma unroll
    for (int ti = 0; ti < 4; ++ti)
      a[ti] = A_TRANS ? As[(4 * kk + t) * ELD + 8 * ti + g] : As[(8 * ti + g) * ELD + 4 * kk + t];
#pragma unroll
    for (int tj = 0; tj < 4; ++tj) b[tj] = Bs[(4 * kk + t) * ELD + 8 * tj + g];
#pragma unroll
    for (int ti = 0; ti < 4; ++ti)
#pragma unroll
      for (int tj = 0; tj < 4; ++tj) dmma884(c[ti][tj][0], c[ti][tj][1], a[ti], b[tj]);
  }
}

// The tile that STEERS the rotations lives in fp32 (shifted by the mean diagonal so that diagonal
// differences keep their accuracy); only the accumulated rotation Q and the (c, s) pairs are fp64.
// Phase B re-derives every tile, including the pair's own, as Q_k^T A_kl Q_l in fp64, so the
// transformation applied to the matrix is an exact orthogonal similarity whatever the angles are.
constexpr int ELDF = 48;   // row stride = 16 banks: the 2 x 16 blocks a warp touches per access are conflict free
// Rotation tables live in THREE slots (round r uses slot r % 3): round r + 1 is being written by warp 0 while
// round r steers the tile and round r - 1 is still being accumulated into Q.  WHICH indices pair k of a round
// rotates is never stored: pair_of / slot_of derive it from the round number with a few integer operations
// (a table in shared memory costs more load bandwidth than the rotations themselves).
constexpr int kSlots = 3;
// Shared-memory map of a visit (inside the phase-B tile regions, idle during phase A):
//   Q fp64 [EP][ELD] | cs fp64 [3][EB][2] | S fp32 2 x [EP][ELDF] (round r reads S[r&1], writes S[(r+1)&1]) | csf fp32 [3][EB][2]
// The accessors name the dynamic shared array directly: a pointer that travels through a struct or a call loses its
// address space, and every access becomes a generic load with 64-bit address arithmetic.
__device__ __forceinline__ double* vis_Q() { extern __shared__ __align__(16) double esm[]; return esm; }
__device__ __forceinline__ double2* vis_cs() { return reinterpret_cast<double2*>(vis_Q() + EP * ELD); }
__device__ __forceinline__ float* vis_S(int buf) { return reinterpret_cast<float*>(vis_cs() + kSlots * EB) + buf * (EP * ELDF); }
__device__ __forceinline__ float2* vis_csf() { return reinterpret_cast<float2*>(vis_S(0) + 2 * EP * ELDF); }

// Pairing of an inner round t.  INTRA: round-robin tournament inside each of the two blocks (EB - 1 rounds, pairs
// 0..EB/2-1 in the first block, the rest in the second); otherwise round t pairs index k with EB + (k + t) % EB.
// The kind of round is a template parameter: 24 of 25 visits only have the second kind, whose index arithmetic is two
// integer instructions, and the visit is bound by the instruction count of its slowest warp.
template <bool INTRA>
__device__ __forceinline__ void pair_of(int t, int k, int& p, int& q) {
  if (INTRA) {
    rr_pair(EB, t, k % (EB / 2), p, q);
    const int o = (k < EB / 2) ? 0 : EB;
    p += o; q += o;
  } else {
    p = k;
    q = EB + ((k + t) & (EB - 1));
  }
}
// the pair of round t that contains tile index x (inverse of pair_of)
template <bool INTRA>
__device__ __forceinline__ int slot_of(int t, int x) {
  if (INTRA) {
    constexpr int m = EB - 1;
    const int y = x & (EB - 1), o = (x >= EB) ? EB / 2 : 0;
    if (y == m) return o;
    const int d = (y - t % m + m) % m;     // y = (t + k) % m  ->  k = d;   y = (t - k) % m  ->  k = m - d
    return o + (d <= EB / 2 - 1 ? d : m - d);
  }
  return x < EB ? x : ((x - t) & (EB - 1));
}

// rotations of the FIRST inner round, from the tile itself
template <bool INTRA>
__device__ __forceinline__ void first_pairs() {
  const int tid = threadIdx.x;
  if (tid < EB) {
    int p, q;
    pair_of<INTRA>(0, tid, p, q);
    const float* S = vis_S(0);
    float c, s;
    rotation(S[q * ELDF + q] - S[p * ELDF + p], S[p * ELDF + q], c, s);
    vis_csf()[tid] = make_float2(c, s);
  }
}

// Rotations of round r+1 (round tn of kind INTRA_N), computed by lanes 0..EB-1 of warp 0 WHILE the other warps apply
// round r (round t of kind INTRA): the pivot entries of S_{r+1} = J_r^T S_r J_r are closed-form in S_r (read-only this
// round) and the rotations of round r:  S'[i,j] = sum_{a in pair(i)} sum_{b in pair(j)} J[a,i] J[b,j] S[a,b].
template <bool INTRA, bool INTRA_N>
__device__ __forceinline__ void next_pairs(int buf, int slot, int slot_next, int t, int tn) {
  const int tid = threadIdx.x;
  if (tid < EB) {
    int p, q, a1, a2, b1, b2;
    pair_of<INTRA_N>(tn, tid, p, q);
    const int kp = slot_of<INTRA>(t, p), kq = slot_of<INTRA>(t, q);
    pair_of<INTRA>(t, kp, a1, a2);
    pair_of<INTRA>(t, kq, b1, b2);
    const float* S = vis_S(buf);
    const float2 rp = vis_csf()[slot * EB + kp], rq = vis_csf()[slot * EB + kq];
    const float saa1 = S[a1 * ELDF + a1], saa2 = S[a1 * ELDF + a2], saa3 = S[a2 * ELDF + a1], saa4 = S[a2 * ELDF + a2];
    const float sbb1 = S[b1 * ELDF + b1], sbb2 = S[b1 * ELDF + b2], sbb3 = S[b2 * ELDF + b1], sbb4 = S[b2 * ELDF + b2];
    const float sab1 = S[a1 * ELDF + b1], sab2 = S[a1 * ELDF + b2], sab3 = S[a2 * ELDF + b1], sab4 = S[a2 * ELDF + b2];
    // column p of J_r is wa1 e_a1 + wa2 e_a2, column q is wb1 e_b1 + wb2 e_b2
    const float wa1 = (p == a1) ? rp.x : rp.y, wa2 = (p == a1) ? -rp.y : rp.x;
    const float wb1 = (q == b1) ? rq.x : rq.y, wb2 = (q == b1) ? -rq.y : rq.x;
    const float saa = wa1 * (wa1 * saa1 + wa2 * saa2) + wa2 * (wa1 * saa3 + wa2 * saa4);
    const float sbb = wb1 * (wb1 * sbb1 + wb2 * sbb2) + wb2 * (wb1 * sbb3 + wb2 * sbb4);
    const float sab = wa1 * (wb1 * sab1 + wb2 * sab2) + wa2 * (wb1 * sab3 + wb2 * sab4);
    float c, s;
    rotation(sbb - saa, sab, c, s);
    vis_csf()[slot_next * EB + tid] = make_float2(c, s);
  }
}

// warp 1: fp64 re-normalisation of the rotations of `slot` (they steer the tile in fp32 meanwhile)
__device__ __forceinline__ void renorm_round(int slot) {
  const int l = threadIdx.x - 32;
  if (l >= 0 && l < EB) {
    const float2 r = vis_csf()[slot * EB + l];
    double c, s;
    renormalise(r.x, r.y, c, s);
    vis_cs()[slot * EB + l] = make_double2(c, s);
  }
}

// Threads kApplyFirst .. kEigThreads-1:  S[buf^1] <- R^T S[buf] R in fp32 for the EB disjoint rotations of round ts
// (kind INTRA_S, tables in slot_s; DO_S = false: nothing), and Q <- Q R in fp64 for the rotations of round tq (kind
// INTRA_Q, slot_q), which are one round older and already re-normalised (DO_Q = false: nothing).  Every thread first
// LOADS all of its work, then computes, then stores, so the independent chains overlap.
constexpr int kApplyFirst = 64;
template <bool DO_S, bool INTRA_S, bool DO_Q, bool INTRA_Q>
__device__ __forceinline__ void apply_round(int buf, int slot_s, int ts, int slot_q, int tq) {
  const float* __restrict__ Si = vis_S(buf);
  float* __restrict__ So = vis_S(buf ^ 1);
  double* __restrict__ Q = vis_Q();
  constexpr int nthr = kEigThreads - kApplyFirst;
  const int t0 = threadIdx.x - kApplyFirst;
  if (t0 < 0) return;
  constexpr int NB = DO_S ? (EB * EB + nthr - 1) / nthr : 0, NQ = DO_Q ? (EP * EB + nthr - 1) / nthr : 0;
  const float2* __restrict__ csf = vis_csf() + slot_s * EB;
  const double2* __restrict__ cs = vis_cs() + slot_q * EB;
  int p[NB + 1], q[NB + 1], u[NB + 1], v[NB + 1];
  float2 rk[NB + 1], rl[NB + 1];
  float m00[NB + 1], m01[NB + 1], m10[NB + 1], m11[NB + 1];
  bool okb[NB + 1];
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    const int blk = t0 + i * nthr;
    okb[i] = blk < EB * EB;
    const int k = okb[i] ? blk / EB : 0, l = okb[i] ? blk % EB : 0;
    pair_of<INTRA_S>(ts, k, p[i], q[i]);
    pair_of<INTRA_S>(ts, l, u[i], v[i]);
    rk[i] = csf[k]; rl[i] = csf[l];
    m00[i] = Si[p[i] * ELDF + u[i]]; m01[i] = Si[p[i] * ELDF + v[i]];
    m10[i] = Si[q[i] * ELDF + u[i]]; m11[i] = Si[q[i] * ELDF + v[i]];
  }
  int qr[NQ + 1], qu_i[NQ + 1], qv_i[NQ + 1];
  double2 qcs[NQ + 1];
  double qu[NQ + 1], qv[NQ + 1];
  bool okq[NQ + 1];
#pragma unroll
  for (int i = 0; i < NQ; ++i) {
    const int it = t0 + i * nthr;
    okq[i] = it < EP * EB;
    qr[i] = okq[i] ? it / EB : 0;
    const int l = okq[i] ? it % EB : 0;
    pair_of<INTRA_Q>(tq, l, qu_i[i], qv_i[i]);
    qcs[i] = cs[l];
    qu[i] = Q[qr[i] * ELD + qu_i[i]]; qv[i] = Q[qr[i] * ELD + qv_i[i]];
  }
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    const float ck = rk[i].x, sk = rk[i].y, cl = rl[i].x, sl = rl[i].y;
    const float t00 = ck * m00[i] - sk * m10[i], t01 = ck * m01[i] - sk * m11[i];
    const float t10 = sk * m00[i] + ck * m10[i], t11 = sk * m01[i] + ck * m11[i];
    m00[i] = cl * t00 - sl * t01; m01[i] = sl * t00 + cl * t01;
    m10[i] = cl * t10 - sl * t11; m11[i] = sl * t10 + cl * t11;
  }
#pragma unroll
  for (int i = 0; i < NQ; ++i) {
    const double a = qcs[i].x * qu[i] - qcs[i].y * qv[i], bb = qcs[i].y * qu[i] + qcs[i].x * qv[i];
    qu[i] = a; qv[i] = bb;
  }
#pragma unroll
  for (int i = 0; i < NB; ++i) {
    if (okb[i]) {
      So[p[i] * ELDF + u[i]] = m00[i]; So[p[i] * ELDF + v[i]] = m01[i];
      So[q[i] * ELDF + u[i]] = m10[i]; So[q[i] * ELDF + v[i]] = m11[i];
    }
  }
#pragma unroll
  for (int i = 0; i < NQ; ++i) {
    if (okq[i]) { Q[qr[i] * ELD + qu_i[i]] = qu[i]; Q[qr[i] * ELD + qv_i[i]] = qv[i]; }
  }
}

// One visit of a block pair by the whole CTA: (first round of a sweep only) one cyclic pass over the
// pairs INSIDE each of the two blocks, then one pass over the EB*EB cross pairs, as rounds of EB
// disjoint rotations.  Over a sweep every index pair of the matrix is rotated exactly once: this is
// cyclic Jacobi whose rotations are applied to the matrix tile-wise in phase B.
#ifdef RT_EIG_PROF
__device__ long long g_vprof[8];
#endif
// Pipeline, ONE barrier per inner round r:
//   warp 0  derives the fp32 rotations of round r+1 from S_r and the rotations of round r (slot (r+1) % 3),
//   warp 1  re-normalises the rotations of round r in fp64 (slot r % 3),
//   warps 2.. apply round r to the steering tile (S_r -> S_{r+1}, fp32) and round r-1 to Q (fp64).
// One more Q-only step after the last round.
// one inner round: the three roles, then the barrier
template <bool INTRA, bool INTRA_N, bool HAS_NEXT, bool DO_Q, bool INTRA_Q>
__device__ __forceinline__ void visit_round(int r, int& slot, int t, int tn, int tq) {
  const int tid = threadIdx.x;
  const int slot_next = slot == kSlots - 1 ? 0 : slot + 1;
  const int slot_prev = slot == 0 ? kSlots - 1 : slot - 1;
#ifdef RT_EIG_PROF
  const long long c0 = clock64();
#endif
  if (tid < 32) {
    if (HAS_NEXT) next_pairs<INTRA, INTRA_N>(r & 1, slot, slot_next, t, tn);
  } else if (tid < kApplyFirst) {
    renorm_round(slot);
  } else {
    apply_round<true, INTRA, DO_Q, INTRA_Q>(r & 1, slot, t, slot_prev, tq);
  }
#ifdef RT_EIG_PROF
  const long long c1 = clock64();
#endif
  __syncthreads();
#ifdef RT_EIG_PROF
  if (blockIdx.x == 5 && (tid == 0 || tid == 32 || tid == 64)) {
    const long long c2 = clock64();
    atomicAdd((unsigned long long*)&g_vprof[(tid >> 5) * 2], (unsigned long long)(c1 - c0));
    atomicAdd((unsigned long long*)&g_vprof[(tid >> 5) * 2 + 1], (unsigned long long)(c2 - c1));
    if (tid == 0) atomicAdd((unsigned long long*)&g_vprof[6], 1ull);
  }
#endif
  slot = slot_next;
}

__device__ __forceinline__ void cta_visit(bool intra) {
  const int tid = threadIdx.x;
  for (int e = tid; e < EP * EP; e += kEigThreads) vis_Q()[(e / EP) * ELD + (e % EP)] = (e / EP == e % EP) ? 1.0 : 0.0;
  int slot = 0;                                      // r % 3
  int r = 0;
  if (intra) {
    // EB - 1 tournament rounds inside the two blocks, then the EB cross rounds
    first_pairs<true>();
    __syncthreads();
    visit_round<true, true, true, false, true>(r, slot, 0, 1, 0); ++r;
    for (; r < EB - 2; ++r) visit_round<true, true, true, true, true>(r, slot, r, r + 1, r - 1);
    visit_round<true, false, true, true, true>(r, slot, r, 0, r - 1); ++r;          // r = EB - 2: next is cross round 0
    visit_round<false, false, true, true, true>(r, slot, 0, 1, r - 1); ++r;         // cross round 0, Q still has an intra round
    for (int t = 1; t < EB - 1; ++t, ++r) visit_round<false, false, true, true, false>(r, slot, t, t + 1, t - 1);
  } else {
    first_pairs<false>();
    __syncthreads();
    visit_round<false, false, true, false, false>(r, slot, 0, 1, 0); ++r;
    for (int t = 1; t < EB - 1; ++t, ++r) visit_round<false, false, true, true, false>(r, slot, t, t + 1, t - 1);
  }
  visit_round<false, false, false, true, false>(r, slot, EB - 1, 0, EB - 2);
  // the rotations of the last round are re-normalised by now: accumulate them
  apply_round<false, false, true, false>(0, 0, 0, slot == 0 ? kSlots - 1 : slot - 1, EB - 1);
  __syncthreads();
}

// Grid barrier of the round loop (two per round, ~230 rounds per problem: a fifth of the kernel's time went into
// cooperative-groups grid.sync).  Arrival is a fire-and-forget reduction, the wait polls the same word in L2: one L2
// round trip less than an atomic with a return value followed by the poll.  The launch is cooperative (all CTAs are
// resident); the counter only grows during a launch and is reset by CTA 0 before the kernel's first grid.sync.
__device__ unsigned int g_eig_barrier;
__device__ __forceinline__ void round_barrier(unsigned int& target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += gridDim.x;
    // release: this CTA's writes (ordered before thread 0 by the barrier above) become visible with the arrival
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;\n" :: "l"(&g_eig_barrier) : "memory");
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];\n" : "=r"(seen) : "l"(&g_eig_barrier) : "memory");
    } while (seen < target);
  }
  __syncthreads();
}

__global__ void __launch_bounds__(kEigThreads, 1)
eig_block_jacobi_kernel(EigBatch batch) {
  extern __shared__ __align__(16) double esm[];
  cg::grid_group grid = cg::this_grid();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int gwarp = blockIdx.x * kEigWarps + warp;
  const int nwarps = gridDim.x * kEigWarps;
  const int gtid = blockIdx.x * kEigThreads + threadIdx.x;
  const int nthreads = gridDim.x * kEigThreads;
  double* T = esm + warp * (3 * EP * ELD + 4 * EB);  // per-warp: T, Qk, Ql, cs
  double* Qk = T + EP * ELD;
  double* Ql = Qk + EP * ELD;
  __shared__ double red[kEigWarps], red2[kEigWarps];
  __shared__ uint64_t jbar[kEigWarps];      // per warp: completion of the bulk copies of Q_l / Q_k in phase B
  uint32_t jph = 0u;
  if (threadIdx.x == 0) {
    for (int wq = 0; wq < kEigWarps; ++wq) tc::mbar_init(&jbar[wq], 1);
    tc::fence_mbar_init();
  }
  __syncthreads();

  unsigned int bar_target = 0u;
  if (blockIdx.x == 0 && threadIdx.x == 0) g_eig_barrier = 0u;      // visible to all after the grid.sync below
  // ---- phase 0: scale factor, padded copies, V = I, norms ----
  for (int pi = 0; pi < batch.count; ++pi) {
    const EigProblem& P = batch.p[pi];
    double m = 0.0;
    for (int e = gtid; e < P.n * P.n; e += nthreads) m = fmax(m, fabs(P.A_in[e]));
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_xor_sync(0xffffffffu, m, o));
    if (lane == 0 && m > 0.0)
      atomicMax(reinterpret_cast<unsigned long long*>(&P.scal[kScaleSlot]),
                (unsigned long long)__double_as_longlong(m));
  }
  grid.sync();
  for (int pi = 0; pi < batch.count; ++pi) {
    const EigProblem& P = batch.p[pi];
    const double amax = P.scal[kScaleSlot];
    const double inv_scale = amax > 0.0 ? 1.0 / amax : 1.0;
    double loc = 0.0;
    for (int e = gtid; e < P.np * P.np; e += nthreads) {
      const int i = e / P.np, j = e - i * P.np;
      double v = 0.0;
      if (i < P.n && j < P.n) v = 0.5 * inv_scale * (P.A_in[(int64_t)i * P.n + j] + P.A_in[(int64_t)j * P.n + i]);
      P.Ap[e] = v;
      P.Vp[e] = (i == j) ? 1.0 : 0.0;
      loc += v * v;
    }
    loc = rt::warp_sum(loc);
    if (lane == 0 && loc != 0.0) atomicAdd(&P.scal[0], loc);
  }
  grid.sync();

  int max_rounds = 0;
  for (int pi = 0; pi < batch.count; ++pi) max_rounds = max(max_rounds, batch.p[pi].nb - 1);
  bool done[kMaxProblems];
  for (int pi = 0; pi < kMaxProblems; ++pi) done[pi] = (pi >= batch.count);

  double norm2[kMaxProblems];                 // ||A||_F^2 of every problem: fixed after the set-up phase
  for (int pi = 0; pi < kMaxProblems; ++pi) norm2[pi] = (pi < batch.count) ? batch.p[pi].scal[0] : 0.0;
  long long tA = 0, tS1 = 0, tB = 0, tS2 = 0, t0 = 0, t1 = 0;
#ifdef RT_EIG_PROF
  long long pLoad = 0, pVisit = 0, pStore = 0, pN = 0;
#endif
  for (int sweep = 0; sweep < kMaxSweeps; ++sweep) {
    bool all_done = true;
    for (int pi = 0; pi < batch.count; ++pi) all_done = all_done && done[pi];
    if (all_done) break;
    for (int round = 0; round < max_rounds; ++round) {
      // ---- phase A: rotations of this round's block pairs ----
      t0 = clock64();
      int base = 0;
      for (int pi = 0; pi < batch.count; ++pi) {
        const EigProblem& P = batch.p[pi];
        if (done[pi] || round >= P.nb - 1) continue;
        // one pair per CTA (the whole CTA works on the visit; esm[0..] = warp 0's tile region)
        for (int item = (int)((blockIdx.x + gridDim.x - base) % gridDim.x); item < P.npairs;
             item += gridDim.x) {
          int bi, bj;
          rr_pair(P.nb, round, item, bi, bj);
          double off = 0.0;
          const bool intra = (round == 0);
          float* Sf0 = vis_S(0);
          double* Qm = vis_Q();
          double dsum = 0.0;
#ifdef RT_EIG_PROF
          long long q0 = clock64(), q1;
#endif
          // the tile is read from global memory ONCE (all loads in flight together) and kept in registers for the
          // steering copy below: the visit is on the critical path of the round, every L2 round trip counts
          constexpr int kTileRegs = (EP * EP) / kEigThreads;
          static_assert(kTileRegs * kEigThreads == EP * EP, "tile elements per thread");
          double tv[kTileRegs];
#pragma unroll
          for (int u = 0; u < kTileRegs; ++u) {
            const int e = threadIdx.x + u * kEigThreads;
            const int i = e / EP, j = e % EP;
            tv[u] = P.Ap[(int64_t)pair_index(bi, bj, i) * P.np + pair_index(bi, bj, j)];
          }
#pragma unroll
          for (int u = 0; u < kTileRegs; ++u) {
            const int e = threadIdx.x + u * kEigThreads;
            const int i = e / EP, j = e % EP;
            const double v = tv[u];
            const bool cross = (i < EB) != (j < EB);
            if (cross || (intra && i != j)) off += v * v;
            if (i == j) dsum += v;
          }
          off = rt::warp_sum(off);
          dsum = rt::warp_sum(dsum);
          if (lane == 0) { red[warp] = off; red2[warp] = dsum; }
          __syncthreads();
          off = 0.0; dsum = 0.0;
          for (int wq = 0; wq < kEigWarps; ++wq) { off += red[wq]; dsum += red2[wq]; }
          const bool skip = (off <= 1e-30 * norm2[pi]);
          if (!skip) {
            const double mu = dsum / EP;       // the steering tile holds A - mu I (rotations do not see the shift)
#pragma unroll
            for (int u = 0; u < kTileRegs; ++u) {
              const int e = threadIdx.x + u * kEigThreads;
              const int i = e / EP, j = e % EP;
              Sf0[i * ELDF + j] = (float)(i == j ? tv[u] - mu : tv[u]);
            }
            __syncthreads();
#ifdef RT_EIG_PROF
            q1 = clock64(); pLoad += q1 - q0; q0 = q1;
#endif
            cta_visit(intra);
#ifdef RT_EIG_PROF
            q1 = clock64(); pVisit += q1 - q0; q0 = q1; ++pN;
#endif
            // J keeps the padded shared-memory layout [EP][ELD], so that phase B fetches it with ONE bulk copy
            for (int e = threadIdx.x; e < EP * ELD; e += kEigThreads)
              P.J[(int64_t)item * EP * ELD + e] = Qm[e];
#ifdef RT_EIG_PROF
            q1 = clock64(); pStore += q1 - q0; q0 = q1;
#endif
          }
          if (threadIdx.x == 0) {
            P.skip[item] = skip ? 1 : 0;
            if (off != 0.0) atomicAdd(&P.scal[1 + sweep], off);
          }
          __syncthreads();
        }
        base = (base + P.npairs) % gridDim.x;
      }
      t1 = clock64(); tA += t1 - t0;
      round_barrier(bar_target);
      t0 = clock64(); tS1 += t0 - t1;
      // ---- phase B: A_kl <- Q_k^T A_kl Q_l (k != l),  V[:, l] <- V[:, l] Q_l ----
      base = 0;
      for (int pi = 0; pi < batch.count; ++pi) {
        const EigProblem& P = batch.p[pi];
        if (done[pi] || round >= P.nb - 1) continue;
        const int nA = P.npairs * P.npairs;
        const int nV = (P.np / EP) * P.npairs;
        for (int item = (int)((blockIdx.x + gridDim.x * warp + nwarps - base) % nwarps); item < nA + nV;
             item += nwarps) {
          const bool isV = item >= nA;
          int k, l;
          if (isV) { k = (item - nA) / P.npairs; l = (item - nA) % P.npairs; }
          else { k = item / P.npairs; l = item % P.npairs; }
          int bik = 0, bjk = 0, bil, bjl;
          if (!isV) rr_pair(P.nb, round, k, bik, bjk);
          rr_pair(P.nb, round, l, bil, bjl);
          double* M = isV ? P.Vp : P.Ap;
          // ---- tiles -> shared memory.  The gathered tile goes first (16-byte cp.async, all in flight together, issued
          //      before the skip flags are even read: their L2 round trip hides behind it); the rotation products
          //      Q_l, Q_k arrive by bulk copies (one instruction each: a warp's cp.async stream was the slowest part) ----
          __syncwarp();                                   // earlier reads of T / Ql / Qk by this warp are done
          for (int cidx = lane; cidx < EP * (EP / 2); cidx += 32) {
            const int i = cidx >> 4, jc = (cidx & 15) * 2;            // row, first of two columns
            const int gi = isV ? k * EP + i : pair_index(bik, bjk, i);
            cp_async16_d(&T[i * ELD + jc], M + (int64_t)gi * P.np + pair_index(bil, bjl, jc));
          }
          const bool sk = isV ? true : (P.skip[k] != 0);
          const bool sl = P.skip[l] != 0;
          if (sk && sl) { cp_async_wait_all_d(); __syncwarp(); continue; }
          const bool need_l = !sl, need_k = !isV && !sk;
          if (lane == 0 && (need_l || need_k)) {
            asm volatile("fence.proxy.async;\n" ::: "memory");     // generic accesses (smem reads, J written by other CTAs) before the async proxy
            tc::mbar_expect_tx(&jbar[warp], (uint32_t)((need_l ? 1 : 0) + (need_k ? 1 : 0)) * (uint32_t)(EP * ELD * sizeof(double)));
            if (need_l) tc::bulk_g2s(Ql, P.J + (int64_t)l * EP * ELD, (uint32_t)(EP * ELD * sizeof(double)), &jbar[warp]);
            if (need_k) tc::bulk_g2s(Qk, P.J + (int64_t)k * EP * ELD, (uint32_t)(EP * ELD * sizeof(double)), &jbar[warp]);
          }
          if (sl || (!isV && sk)) {
            for (int cidx = lane; cidx < EP * (EP / 2); cidx += 32) {
              const int i = cidx >> 4, jc = (cidx & 15) * 2;
              if (sl) { Ql[i * ELD + jc] = (i == jc) ? 1.0 : 0.0; Ql[i * ELD + jc + 1] = (i == jc + 1) ? 1.0 : 0.0; }
              if (!isV && sk) { Qk[i * ELD + jc] = (i == jc) ? 1.0 : 0.0; Qk[i * ELD + jc + 1] = (i == jc + 1) ? 1.0 : 0.0; }
            }
          }
          cp_async_wait_all_d();
          if (need_l || need_k) { tc::mbar_wait(&jbar[warp], jph); jph ^= 1u; }
          __syncwarp();
          // ---- X = T Ql ;  Y = Qk^T X  on the fp64 tensor cores ----
          const int g = lane >> 2, t = lane & 3;
          double c[4][4][2];
          warp_mm32<false>(T, Ql, c, lane);
          if (!isV) {
            __syncwarp();
#pragma unroll
            for (int ti = 0; ti < 4; ++ti)
#pragma unroll
              for (int tj = 0; tj < 4; ++tj)
                *reinterpret_cast<double2*>(&T[(8 * ti + g) * ELD + 8 * tj + 2 * t]) = make_double2(c[ti][tj][0], c[ti][tj][1]);
            __syncwarp();
            warp_mm32<true>(Qk, T, c, lane);
          }
#pragma unroll
          for (int ti = 0; ti < 4; ++ti) {
            const int i = 8 * ti + g;
            const int gi = isV ? k * EP + i : pair_index(bik, bjk, i);
#pragma unroll
            for (int tj = 0; tj < 4; ++tj)
              *reinterpret_cast<double2*>(&M[(int64_t)gi * P.np + pair_index(bil, bjl, 8 * tj + 2 * t)]) =
                  make_double2(c[ti][tj][0], c[ti][tj][1]);
          }
          __syncwarp();
        }
        base = (base + nA + nV) % nwarps;
      }
      t1 = clock64(); tB += t1 - t0;
      round_barrier(bar_target);
      t0 = clock64(); tS2 += t0 - t1;
    }
    // convergence: off-diagonal mass seen during this sweep (uniform decision: same memory, after sync)
    for (int pi = 0; pi < batch.count; ++pi) {
      if (done[pi]) continue;
      const EigProblem& P = batch.p[pi];
      const double off2 = P.scal[1 + sweep], n2 = P.scal[0];
      // default 1e-14: mass seen (before annihilation) below 1e-7 ||A||, the rotations of this sweep leave ~1e-14.
      // The HOSVD passes 1e-10: the convergence is quadratic, what is left is ~1e-9 ||A|| -- far below the fp32
      // rounding of the factors the eigenvectors are multiplied into (V stays orthogonal to 1e-15 regardless: it
      // is a product of renormalised rotations).
#ifdef RT_EIG_PROF
      if (gtid == 0) printf("eig problem %d (n=%d) sweep %d: off-diagonal mass seen / ||A||^2 = %.3e\n", pi, P.n, sweep, off2 / n2);
#endif
      if (off2 <= batch.stop * n2) done[pi] = true;
    }
  }

#ifdef RT_EIG_PROF
  if (threadIdx.x == 0 && blockIdx.x == 5)
    printf("visit rounds %lld: warp0 next_pairs %lld wait %lld | warp1 renorm %lld wait %lld | apply %lld wait %lld (cycles per round)\n",
           g_vprof[6], g_vprof[0] / max(1ll, g_vprof[6]), g_vprof[1] / max(1ll, g_vprof[6]), g_vprof[2] / max(1ll, g_vprof[6]),
           g_vprof[3] / max(1ll, g_vprof[6]), g_vprof[4] / max(1ll, g_vprof[6]), g_vprof[5] / max(1ll, g_vprof[6]));
  if (threadIdx.x == 0 && blockIdx.x == 5)
    printf("eig cta %d: phaseA %lld = load %lld visit %lld store %lld (visits %lld) sync1 %lld phaseB %lld sync2 %lld\n",
           blockIdx.x, tA, pLoad, pVisit, pStore, pN, tS1, tB, tS2);
#endif
  if (batch.prof && threadIdx.x == 0) {
    batch.prof[blockIdx.x * 4 + 0] = tA; batch.prof[blockIdx.x * 4 + 1] = tS1;
    batch.prof[blockIdx.x * 4 + 2] = tB; batch.prof[blockIdx.x * 4 + 3] = tS2;
  }
  // ---- final: sort eigenvalues descending, emit w and V ----
  for (int pi = 0; pi < batch.count; ++pi) {
    const EigProblem& P = batch.p[pi];
    for (int i = gtid; i < P.n; i += nthreads) {
      const double di = P.Ap[(int64_t)i * P.np + i];
      int rank = 0;
      for (int j = 0; j < P.n; ++j) {
        const double dj = P.Ap[(int64_t)j * P.np + j];
        rank += (dj > di) || (dj == di && j < i);
      }
      P.w[rank] = di * P.scal[kScaleSlot];
      P.scal[kPermSlot + i] = (double)rank;
    }
  }
  grid.sync();
  for (int pi = 0; pi < batch.count; ++pi) {
    const EigProblem& P = batch.p[pi];
    for (int e = gtid; e < P.n * P.n; e += nthreads) {
      const int i = e / P.n, j = e - i * P.n;
      const int rank = (int)P.scal[kPermSlot + j];
      P.V_out[(int64_t)i * P.n + rank] = P.Vp[(int64_t)i * P.np + j];
    }
  }
}

struct EigLayout {
  int np, nb, npairs;
  size_t off_Ap, off_Vp, off_J, off_skip, off_scal, total;
};

EigLayout eig_layout(int n) {
  EigLayout L;
  L.nb = cdiv(n, EB);
  if (L.nb & 1) L.nb += 1;
  if (L.nb < 2) L.nb = 2;
  L.np = L.nb * EB;
  L.npairs = L.nb / 2;
  size_t o = 0;
  L.off_Ap = o; o += align_up(sizeof(double) * L.np * L.np, 256);
  L.off_Vp = o; o += align_up(sizeof(double) * L.np * L.np, 256);
  L.off_J = o; o += align_up(sizeof(double) * L.npairs * EP * ELD, 256);
  L.off_skip = o; o += align_up(sizeof(int) * L.npairs, 256);
  L.off_scal = o; o += align_up(sizeof(double) * (kPermSlot + L.np), 256);
  L.total = o;
  return L;
}

static size_t eig_ws_bytes(int n) { return eig_layout(n).total; }

// Solve `count` (<= 4) independent problems in one cooperative launch.
long long* g_eig_prof = nullptr;   // set through rt_eigh_set_profile (debug)

static int eig_batch(int count, const double* const* A, const int* n, double* const* w, double* const* V,
                     void* const* ws, cudaStream_t s, double stop) {
  RT_REQUIRE(count >= 1 && count <= kMaxProblems, "eig_batch: count=%d out of range", count);
  EigBatch b{};
  b.count = count;
  b.stop = stop > 0.0 ? stop : 1e-14;
  b.prof = g_eig_prof;
  int total_items = 0;
  for (int i = 0; i < count; ++i) {
    RT_REQUIRE(n[i] >= 1 && n[i] <= 1024, "eig_batch: n=%d out of range", n[i]);
    EigLayout L = eig_layout(n[i]);
    char* base = (char*)ws[i];
    EigProblem& P = b.p[i];
    P.A_in = A[i]; P.w = w[i]; P.V_out = V[i];
    P.Ap = (double*)(base + L.off_Ap);
    P.Vp = (double*)(base + L.off_Vp);
    P.J = (double*)(base + L.off_J);
    P.skip = (int*)(base + L.off_skip);
    P.scal = (double*)(base + L.off_scal);
    P.n = n[i]; P.np = L.np; P.nb = L.nb; P.npairs = L.npairs;
    RT_CHECK_CUDA(cudaMemsetAsync(P.scal, 0, sizeof(double) * (kPermSlot + L.np), s));
    total_items += L.npairs * L.npairs + (L.np / EP) * L.npairs;
  }
  const size_t smem = (size_t)kEigWarps * (3 * EP * ELD + 4 * EB) * sizeof(double);
  RT_CHECK_CUDA(ensure_dyn_smem((const void*)eig_block_jacobi_kernel, smem));   // cached per (kernel, device)
  // one warp per phase-B tile if possible (latency matters more than occupancy), capped at 1 CTA / SM
  // (launch bounds) so the cooperative grid is co-resident
  int grid = total_items;
  const int max_grid = sm_count();
  if (grid > max_grid) grid = max_grid;
  if (grid < 1) grid = 1;
  void* args[] = {(void*)&b};
  RT_CHECK_CUDA(cudaLaunchCooperativeKernel((const void*)eig_block_jacobi_kernel, dim3(grid),
                                            dim3(kEigThreads), args, smem, s));
  ++g_launches;
  return 0;
}

}  // namespace rt

extern "C" size_t rt_eigh_ws_bytes(int n) { return n > 0 ? rt::eig_ws_bytes(n) : 0; }

extern "C" int rt_eigh(double* A, int n, double* w, double* V, void* ws, void* stream) {
  RT_REQUIRE(ws != nullptr, "rt_eigh: workspace is NULL");
  const double* Ain[1] = {A};
  double* wo[1] = {w};
  double* Vo[1] = {V};
  void* wss[1] = {ws};
  return rt::eig_batch(1, Ain, &n, wo, Vo, wss, (cudaStream_t)stream, 1e-14);
}

// Debug: cycle counters per CTA ([grid][4] int64: phase A, sync, phase B, sync), NULL to disable.
extern "C" int rt_eigh_set_profile(long long* dev_buf) { rt::g_eig_prof = dev_buf; return 0; }
