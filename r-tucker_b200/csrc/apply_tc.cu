// Tall-skinny factor updates on the tensor cores (tcgen05, TF32 with a 3-product hi/lo split) at fp32 accuracy.
//
//   Y[n, rc] = a0 * X0 + sum_t X_t[n, rk_t] . K_t[rk_t, rc]          (K_t fp64, r x r)
//
// = the N-sized factor updates of the Riemannian gradient / momentum transport / retraction
// (reference call sites src/model/asymmetric/optim.py:86-92,106-114, symmetric/optim.py:80-86,100-107).
// Several independent updates ("jobs": the subject and the object factor) run in ONE persistent launch.
//
// Accuracy.  x = x_hi + x_lo (both TF32, round-to-nearest) and x.y ~ x_lo.y_hi + x_hi.y_lo + x_hi.y_hi loses 2^-24
// per product, but the tensor core's fp32 accumulator TRUNCATES: measured bias -0.4 ulp per MMA instruction, i.e.
// -1.8e-6 / -4e-6 / -6e-6 relative for 1 / 2 / 3 terms of K = 200 (tools/tc_acc.py).  So an accumulator in tensor
// memory only ever holds the sum over GB*KB = 32 contraction elements (started from zero); two such accumulators
// alternate, and the epilogue warps add each finished partial sum to an fp32 running sum in registers with
// round-to-nearest.  Result: the accuracy of the FFMA kernel (a few 1e-7 norm-wise).
//
// Roles (one persistent CTA per SM, 16 warps, register file re-partitioned with setmaxnreg).  Warps 0-7, epilogue:
// drain finished partial sums (tcgen05.ld) into 104 fp32 registers per thread, at the end of a row tile add
// a0 * X0 and store Y.  Warps 8-11, producers: load the X blocks from global memory (coalesced float4, PF blocks in
// flight in registers), split them into the hi / lo operand images in shared memory, optionally write the raw block
// to a second destination (the "old point" / "kept direction" copies of the optimiser, which would otherwise be
// separate passes).  Warp 12 (one lane) issues the MMAs; warp 13 (one lane) streams the pre-split K images with
// bulk async copies (TMA, mbarrier complete_tx).
#include "common.h"
#include "tc.cuh"
#include "exact.cuh"
#include <algorithm>
#include <limits.h>
#include <math.h>

namespace {
using namespace rt::tc;

constexpr int kEpiWarps = 8, kProdWarps = 4, kMmaWarp = 12, kLoadWarp = 13;
constexpr int kThreads = 512;       // 16 warps = 4 warpgroups: epilogue (2), producers (1), MMA + loader + 2 idle (1)
constexpr int kRegsEpi = 168, kRegsOther = 88;                  // setmaxnreg: 256 * 168 + 256 * 88 = 64 K registers
constexpr int kRegsEpiLogits = 176, kRegsOtherLogits = 80;      // rank / score mode: 128 logits + counters per thread
                                                                // (top-k mode: 128 logits and no counters, the factor-update split)
constexpr int TM = 128;             // rows per tile
constexpr int KB = 16;              // contraction elements per staged block (2 MMA k-steps)
constexpr int GB = 2;               // blocks per partial sum held in tensor memory (factor updates)
constexpr int GB_LOGITS = 7;        // rank / score mode: a 200-wide contraction is two partial sums, so that a whole tile can
                                    // sit in the two accumulators while the (long) epilogue of the previous tile runs; the
                                    // truncation bias of 112-element partial sums is ~6e-7, inside the logit margins
constexpr int PF = 3;               // X blocks in flight per producer thread (registers)
constexpr int XPT = TM * (KB / 4) / (kProdWarps * 32);          // float4 per producer thread and block
constexpr int MAX_STAGES = 6;
constexpr uint32_t RS = 128;
constexpr uint32_t CS_X = TM * 16 + 32;                 // chunk stride of the X images: (CS_X / 16) % 8 == 2 keeps the
                                                        // 16-byte stores of a quarter warp on distinct banks
constexpr uint32_t X_HALF = (KB / 4) * CS_X;            // one image (hi or lo) of a block: 8320 bytes
constexpr int RCP_MAX = 256;
constexpr int MAX_JOBS = 4, MAX_TERMS = 4;
constexpr size_t SMEM_LIMIT = 226 * 1024;
// epilogue modes of apply_tc_kernel (its MODE parameter): the factor update Y = a0 X0 + sum X_t K_t, and the logits
// passes (rows = entities, 256 queries per job) of the filtered ranking, the BCE score, the top-k candidates, the
// log-sum-exp parts and the cross-entropy score
constexpr int kModeApply = 0, kModeRank = 1, kModeScore = 2, kModeTopk = 3, kModeLse = 4, kModeCe = 5;

struct Job {
  float* Y; int64_t ldy;
  const float* X0; int64_t ldx0; const double* a0;
  const float* X[MAX_TERMS]; int64_t ldx[MAX_TERMS];
  float* copy[MAX_TERMS]; int64_t ldc[MAX_TERMS];
  int rk[MAX_TERMS]; int blk_end[MAX_TERMS];        // blk_end[t]: first block index after term t
  int xt[MAX_TERMS];                                // term given transposed: element (row, k) at X + k * ldx + row
  int n, nk, nblk, kblk0, tile0, ntiles;
  // replication: the job is run `reps` times on shifted operands (row chunks of a long contraction whose partial
  // results are summed afterwards): rep r uses X_t + r * x_rep[t], Y + r * y_rep, K blocks kblk0 + r * nblk
  int reps, tiles_per_rep;
  int64_t x_rep[MAX_TERMS], y_rep;
};
struct Args {
  Job job[MAX_JOBS];
  int njobs, ntiles, rc, rcp, nstages, gb;
  const unsigned char* Kimg;          // [total blocks][hi | lo][KB/4 chunks][cs_k bytes]
  uint32_t cs_k, kimg_bytes, stage_bytes;
  int debug;                          // profiling build only (RT_APPLY_DEBUG): 1 no X loads, 2 no K loads, 4 no MMAs, 8 ld.cg
  // ---- rank mode (kModeRank): rows = entities of the shard, columns of job j = queries [256 j, 256 j + 256) ----
  const float* thr;                   // [4][Bp]: lo0, hi0, eqlo0, slope per query (Bp = 256 * njobs), see rank_thresholds_kernel
  const float* onorms;                // [n_local] upper bounds of the entity row norms
  const int32_t* target;              // [B] global id of the target entity
  int B, n_begin;
  int32_t* greater; int32_t* equal; int32_t* equal_before;
  int2* cand; int* cand_count; int cand_cap;   // (local entity, query) pairs whose probability must be recomputed exactly
  double* loss_sum;                   // sum of softplus(z) over every valid (entity, query)
  // ---- score mode (kModeScore): the same logits; the epilogue writes G[e][b] = dBCE/dz for all-negative targets ----
  float* G; int64_t ldg;              // [n_local][ldg] (ldg = 256 * njobs)
  float t_neg, inv_count;
  double* loss_partial;               // [grid]
  // ---- top-k mode (kModeTopk): the rank-mode logits; entities not certainly below the query's threshold are
  //      appended to its segment seg[b][0, cand_cap) (overflow: cnt[b] > cand_cap; thr and onorms as in rank mode) ----
  int32_t* topk_seg; int* topk_cnt;
};
struct PackArgs {
  const void* K[MAX_JOBS * MAX_TERMS]; int rk[MAX_JOBS * MAX_TERMS]; int blk0[MAX_JOBS * MAX_TERMS + 1];
  int f32[MAX_JOBS * MAX_TERMS];            // source type of the term: fp64 (0) or fp32 (1), row-major [rows][rc]
  int rep_blocks[MAX_JOBS * MAX_TERMS];     // blocks per repetition (0: not replicated); rep r reads rows r * rk + k
  int rows_total[MAX_JOBS * MAX_TERMS];     // rows that exist in the source (beyond: zeros)
  int nterms, rc, rcp; unsigned char* img; uint32_t cs_k, kimg_bytes;
};

__device__ __forceinline__ void split_tf32(float x, uint32_t& hi, uint32_t& lo) {
  hi = to_tf32(x);
  lo = to_tf32(x - __uint_as_float(hi));
}

// same split with the round-to-nearest (ties away) done on the bit pattern: add half an ulp of TF32, clear 13 bits
// (Inf / NaN inputs are not special-cased: they poison the row either way)
__device__ __forceinline__ void split_tf32_fast(float x, uint32_t& hi, uint32_t& lo) {
  hi = (__float_as_uint(x) + 0x1000u) & 0xffffe000u;
  lo = (__float_as_uint(x - __uint_as_float(hi)) + 0x1000u) & 0xffffe000u;
}

// image of block `blk`: element (c, kk) = K_t[kb*KB + kk][c], K-major B operand (rows = c), hi then lo
__global__ void pack_K_kernel(PackArgs a) {
  const int blk = blockIdx.x;
  int t = 0;
  while (t + 1 < a.nterms && blk >= a.blk0[t + 1]) ++t;
  int kb = blk - a.blk0[t], rep = 0;
  if (a.rep_blocks[t] > 0) { rep = kb / a.rep_blocks[t]; kb -= rep * a.rep_blocks[t]; }
  const int rk = a.rk[t];
  const int64_t row_base = (int64_t)rep * rk;
  unsigned char* img = a.img + (size_t)blk * a.kimg_bytes;
  const uint32_t half = (KB / 4) * a.cs_k;
  for (int e = threadIdx.x; e < KB * a.rcp; e += blockDim.x) {
    const int kk = e / a.rcp, c = e - kk * a.rcp;
    const int k = kb * KB + kk;
    float v = 0.0f;
    if (k < rk && c < a.rc && row_base + k < a.rows_total[t]) {
      const int64_t at = (row_base + k) * a.rc + c;
      v = a.f32[t] ? __ldg(reinterpret_cast<const float*>(a.K[t]) + at) : (float)reinterpret_cast<const double*>(a.K[t])[at];
    }
    uint32_t hi, lo;
    split_tf32(v, hi, lo);
    const uint32_t off = (uint32_t)(kk >> 2) * a.cs_k + (uint32_t)(c >> 3) * RS + (uint32_t)(c & 7) * 16u + (uint32_t)(kk & 3) * 4u;
    *reinterpret_cast<uint32_t*>(img + off) = hi;
    *reinterpret_cast<uint32_t*>(img + half + off) = lo;
  }
}

#ifdef RT_APPLY_PROF
#include <stdlib.h>
#define DBG(bit) ((a.debug >> (bit)) & 1)
#else
#define DBG(bit) 0
#endif
#ifdef RT_APPLY_PROF
#define PROF_DECL long long pt0 = clock64(), pw0 = 0, pw1 = 0, pw2 = 0, ptmp = 0
#define PROF_BEGIN ptmp = clock64()
#define PROF_END(x) x += clock64() - ptmp
#define PROF_PRINT(role) if (blockIdx.x == 0 || blockIdx.x == 100) printf("cta %d %s: total %lld wait0 %lld wait1 %lld wait2 %lld\n", blockIdx.x, role, clock64() - pt0, pw0, pw1, pw2)
#else
#define PROF_DECL
#define PROF_BEGIN
#define PROF_END(x)
#define PROF_PRINT(role)
#endif

__device__ __forceinline__ float lg2_fast(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
// ---- filtered-ranking epilogue of 8 columns (queries) of one thread's row (entity) --------------------------------
// NOT inlined: the epilogue of a tile is 128 columns per thread, and as one unrolled block it was ~30 000 instructions
// (0.5 MB) executed once per tile -- ncu showed the epilogue warps stalled on instruction fetch (stall_no_inst at every
// reconvergence point), 110 k cycles per tile against 10 k of tensor work.  As a function called 16 times the code
// stays resident.
struct RankChunkCtx {
  const float* lo; const float* hi; const float* eq; const float* slope;   // thresholds of query 0 of this warp's columns
  float onorm;                                            // upper bound of ||O_j|| of this thread's entity
  const int32_t* target; int32_t* equal; int32_t* equal_before;
  int2* cand; int* cand_count;
  int cand_cap, B, q0, e_loc, e_glob;
  bool rv, any_eq;
};
struct RankChunkOut { uint32_t counts; float lsum; };
__device__ __noinline__ RankChunkOut rank_chunk8(const RankChunkCtx& cx, int c0, float z0, float z1, float z2, float z3, float z4,
                                                 float z5, float z6, float z7) {
  const int lane = threadIdx.x & 31;
  // hot fields of the context in registers; the rare paths (saturated targets, candidates) read theirs from memory
  const int cB = cx.B, q0 = cx.q0;
  const bool rv = cx.rv, any_eq = cx.any_eq;
  const float zs[8] = {z0, z1, z2, z3, z4, z5, z6, z7};
  const float* lop = cx.lo + c0;
  const float* hip = cx.hi + c0;
  const float* slp = cx.slope + c0;
  const float onorm = cx.onorm;
  RankChunkOut out;
  out.counts = 0u; out.lsum = 0.0f;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    // thresholds of 4 columns at a time (all 8 at once spilled 340 bytes in this function)
    float4 lo4, hi4, sl4;
    if ((u & 3) == 0) {
      lo4 = __ldg(reinterpret_cast<const float4*>(lop + u)); hi4 = __ldg(reinterpret_cast<const float4*>(hip + u));
      sl4 = __ldg(reinterpret_cast<const float4*>(slp + u));
    }
    const float lo0 = (u & 3) == 0 ? lo4.x : (u & 3) == 1 ? lo4.y : (u & 3) == 2 ? lo4.z : lo4.w;
    const float hi0 = (u & 3) == 0 ? hi4.x : (u & 3) == 1 ? hi4.y : (u & 3) == 2 ? hi4.z : hi4.w;
    const float sl0 = (u & 3) == 0 ? sl4.x : (u & 3) == 1 ? sl4.y : (u & 3) == 2 ? sl4.z : sl4.w;
    const float m = sl0 * onorm, lo_u = lo0 - m, hi_u = hi0 + m;
    const int c = c0 + u;
    const int b = q0 + c;
    const float z = zs[u];
    const bool on = rv && b < cB;
    bool eqd = false;
    if (any_eq) {                                                   // certainly p == 1 == p_target (rare, warp-uniform)
      eqd = on && z > __ldg(cx.eq + c) + m;
      const unsigned em = __ballot_sync(0xffffffffu, eqd);
      if (em) {
        const int t = __ldg(cx.target + b);
        const unsigned em2 = __ballot_sync(0xffffffffu, eqd && cx.e_glob != t);
        const unsigned bm = __ballot_sync(0xffffffffu, eqd && cx.e_glob < t);
        if (lane == 0) {
          if (em2) atomicAdd(cx.equal + b, __popc(em2));
          if (bm) atomicAdd(cx.equal_before + b, __popc(bm));
        }
      }
    }
    // "greater" as a 4-bit counter per column in this thread's registers: no warp collective in the hot loop;
    // the cross-lane sums happen once per job (or every 15 tiles), see flush_counts
    const bool gt = on && z > hi_u;
    const bool cd = on && !eqd && z >= lo_u && z <= hi_u;
    out.counts += (gt ? 1u : 0u) << (u * 4);
    if (cd) {                                                          // rare: recomputed exactly afterwards
      const int pos = atomicAdd(cx.cand_count, 1);
      if (pos < cx.cand_cap) cx.cand[pos] = make_int2(cx.e_loc, b);
    }
    if (on) {
      // -log(1 - p) with the reference's fp32 semantics: for z >= 0 through the fp32 probability itself (1 - p
      // is quantised to multiples of 2^-24 there: up to 0.35 per element near saturation, 2e-4 of a batch's
      // BCE), p == 1 from z = 24 ln 2 on (BCELoss clamps log(1 - p) at -100); for z < 0 log(1 + e^z)
      const float en = rt::ex2_approx(-rt::kLog2e * fabsf(z));
      const float sden = 1.0f + en;
      const bool pos = z >= 0.0f;                                      // branch-free: both signs share every warp
      const float lg = rt::kLn2 * lg2_fast(pos ? 1.0f - __frcp_rn(sden) : sden);
      float sp = pos ? -lg : lg;
      sp = (!pos && en < 1e-3f) ? en * (1.0f - 0.5f * en) : sp;
      sp = (pos && z >= 16.635532f) ? 100.0f : sp;
      out.lsum += sp;
    }
  }
  return out;
}

// ---- score epilogue of 8 columns (queries) of one thread's row (entity): G[e][b] = dBCE/dz and the BCE itself for
//      ALL-NEGATIVE targets (t = t_neg), with the reference's fp32 semantics (exact.cuh: p = 1 / (1 + expf(-z)), log
//      terms clamped at -100, gradient scaled by p (1 - p) / max(p (1 - p), 1e-12)); the sparse positives are fixed up
//      afterwards.  Not inlined for the same reason as rank_chunk8 (instruction footprint of 128 unrolled columns). ----
__device__ __noinline__ float score_chunk8(float* __restrict__ gdst, bool rv, int ncols, float tn, float inv, float z0, float z1,
                                           float z2, float z3, float z4, float z5, float z6, float z7) {
  const float zs[8] = {z0, z1, z2, z3, z4, z5, z6, z7};
  float gv[8];
  float lsum = 0.0f;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const float z = zs[u];
    // three special-function operations per element (ex2, rcp, lg2), BRANCH-FREE (the two signs of z share every warp:
    // as if / else both sides ran for every element)
    const float en = rt::ex2_approx(-rt::kLog2e * fabsf(z));                                 // e^-|z|
    const float sden = 1.0f + en;
    const float rq = __frcp_rn(sden);                                                 // 1 / (1 + e^-|z|)
    const bool pos = z >= 0.0f;
    // z >= 0: p in [0.5, 1] is the fp32 quotient, 1 - p is exact, log(1 - p) from it (p == 1 from z = 24 ln 2 on);
    // z <  0: p = e^z / (1 + e^z), log(1 - p) = -log(1 + e^z) (series for tiny e^z)
    const float p = pos ? rq : en * rq;
    const float lg = rt::kLn2 * lg2_fast(pos ? 1.0f - rq : sden);
    float lq = pos ? lg : -lg;
    lq = (!pos && en < 1e-3f) ? -(en * (1.0f - 0.5f * en)) : lq;
    lq = (pos && z >= 16.635532f) ? -100.0f : lq;
    // log p = log(1 - p) + z (exact identity; its term carries the weight t_neg = ls / N ~ 1e-6 of the loss)
    const float lp = fmaxf(lq + z, -100.0f);
    const float pq = (1.0f - p) * p;
    float g = (p - tn) * inv;
    if (pq < 1e-12f) g *= pq * 1e12f;
    const bool on = rv && u < ncols;
    if (on) lsum -= tn * lp + (1.0f - tn) * lq;
    gv[u] = on ? g : 0.0f;
  }
  if (rv) {
    *reinterpret_cast<float4*>(gdst) = make_float4(gv[0], gv[1], gv[2], gv[3]);
    *reinterpret_cast<float4*>(gdst + 4) = make_float4(gv[4], gv[5], gv[6], gv[7]);
  }
  return lsum;
}

// ---- top-k candidate epilogue of 8 columns (queries) of one thread's row (entity): append the entity to the segment of
//      every query whose band it reaches (z >= lo_b - slope_b ||O_j||: not certainly below the sample threshold).
//      Inlined: one compare per column; with the factor-update register split it does not spill. ----
__device__ __forceinline__ void topk_chunk8(const float* __restrict__ lop, const float* __restrict__ slp, float onorm, bool rv,
                                         int ncols, int b0, int e_loc, int* cnt, int32_t* seg, int cap, float z0, float z1,
                                         float z2, float z3, float z4, float z5, float z6, float z7) {
  const float zs[8] = {z0, z1, z2, z3, z4, z5, z6, z7};
  if (!rv) return;
#pragma unroll
  for (int u = 0; u < 8; u += 4) {
    const float4 lo4 = __ldg(reinterpret_cast<const float4*>(lop + u)), sl4 = __ldg(reinterpret_cast<const float4*>(slp + u));
    const float lo[4] = {lo4.x, lo4.y, lo4.z, lo4.w}, sl[4] = {sl4.x, sl4.y, sl4.z, sl4.w};
#pragma unroll
    for (int v = 0; v < 4; ++v) {
      if (u + v < ncols && zs[u + v] >= lo[v] - sl[v] * onorm) {       // rare: a few hundred entities per query
        const int b = b0 + u + v;
        const int pos = atomicAdd(cnt + b, 1);
        if (pos < cap) seg[(int64_t)b * cap + pos] = e_loc;
      }
    }
  }
}

// ---- 1-N softmax cross-entropy, log-sum-exp epilogue of 8 columns (queries) over the warp's 32 rows (entities): per
//      column m = the largest valid logit (integer warp max on an order-preserving key), s = sum exp(z - m); the 8 sums
//      by a reduce-scatter butterfly (4 + 2 + 1 shuffles leave lane group j = (lane >> 2) & 7 holding column j, 2 more
//      finish it) instead of 8 full warp sums.  Lane 4j writes dst[j] = (m_j, s_j).  Rows / columns that do not exist
//      count as -inf. ----
__device__ __noinline__ void lse_chunk8(float2* __restrict__ dst, bool rv, int ncols, float z0, float z1, float z2, float z3,
                                        float z4, float z5, float z6, float z7) {
  const int lane = threadIdx.x & 31;
  const float zs[8] = {z0, z1, z2, z3, z4, z5, z6, z7};
  float m[8], e[8];
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const bool on = rv && u < ncols;
    const int bits = __float_as_int(zs[u]);
    const int key = on ? (bits >= 0 ? bits : bits ^ 0x7fffffff) : INT_MIN;
    const int mk = __reduce_max_sync(0xffffffffu, key);
    m[u] = mk == INT_MIN ? -INFINITY : __int_as_float(mk >= 0 ? mk : mk ^ 0x7fffffff);
    e[u] = on ? rt::ex2_approx((zs[u] - m[u]) * rt::kLog2e) : 0.0f;
  }
  const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
  float v[4], w[2];
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = (b4 ? e[i + 4] : e[i]) + __shfl_xor_sync(0xffffffffu, b4 ? e[i] : e[i + 4], 16);
#pragma unroll
  for (int i = 0; i < 2; ++i) w[i] = (b3 ? v[i + 2] : v[i]) + __shfl_xor_sync(0xffffffffu, b3 ? v[i] : v[i + 2], 8);
  float x = (b2 ? w[1] : w[0]) + __shfl_xor_sync(0xffffffffu, b2 ? w[0] : w[1], 4);
  x += __shfl_xor_sync(0xffffffffu, x, 2);
  x += __shfl_xor_sync(0xffffffffu, x, 1);
  const float mlo = b3 ? (b2 ? m[3] : m[2]) : (b2 ? m[1] : m[0]);
  const float mhi = b3 ? (b2 ? m[7] : m[6]) : (b2 ? m[5] : m[4]);
  if ((lane & 3) == 0) dst[(lane >> 2) & 7] = make_float2(b4 ? mhi : mlo, x);
}

// ---- 1-N softmax cross-entropy, gradient epilogue of 8 columns of one thread's row: G[e][b] = (softmax - ls/N) / B for
//      ALL-NEGATIVE targets, softmax = 2^((z - M_b) log2e - log2 S_b) (one ex2), loss += (ls/N) (lse_b - z); the sparse
//      positives are fixed up afterwards (score_ce_fix_positives_kernel).  Not inlined, like score_chunk8. ----
__device__ __noinline__ float ce_chunk8(float* __restrict__ gdst, const float* __restrict__ mp, const float* __restrict__ lp,
                                        bool rv, int ncols, float tn, float inv, float z0, float z1, float z2, float z3, float z4,
                                        float z5, float z6, float z7) {
  const float zs[8] = {z0, z1, z2, z3, z4, z5, z6, z7};
  const float4 m0 = __ldg(reinterpret_cast<const float4*>(mp)), m1 = __ldg(reinterpret_cast<const float4*>(mp + 4));
  const float4 l0 = __ldg(reinterpret_cast<const float4*>(lp)), l1 = __ldg(reinterpret_cast<const float4*>(lp + 4));
  const float M[8] = {m0.x, m0.y, m0.z, m0.w, m1.x, m1.y, m1.z, m1.w};
  const float L[8] = {l0.x, l0.y, l0.z, l0.w, l1.x, l1.y, l1.z, l1.w};
  float gv[8];
  float lsum = 0.0f;
#pragma unroll
  for (int u = 0; u < 8; ++u) {
    const float d = zs[u] - M[u];
    const float p = rt::ce_softmax(d, L[u]);
    const bool on = rv && u < ncols;
    if (on) lsum += rt::ce_loss_term(tn, d, L[u]);
    gv[u] = on ? (p - tn) * inv : 0.0f;
  }
  if (rv) {
    *reinterpret_cast<float4*>(gdst) = make_float4(gv[0], gv[1], gv[2], gv[3]);
    *reinterpret_cast<float4*>(gdst + 4) = make_float4(gv[4], gv[5], gv[6], gv[7]);
  }
  return lsum;
}

// position in this CTA's flattened sequence of (tile, block) pairs
struct Cursor {
  int tile, job, blk, nblk, kblk0;
  __device__ __forceinline__ bool valid(const Args& a) const { return tile < a.ntiles; }
  __device__ __forceinline__ void set_job(const Args& a) {
    if (tile < a.ntiles) {
      job = 0;
      while (job + 1 < a.njobs && tile >= a.job[job + 1].tile0) ++job;
      nblk = a.job[job].nblk;
      kblk0 = a.job[job].kblk0 + ((tile - a.job[job].tile0) / a.job[job].tiles_per_rep) * nblk;
    }
  }
  __device__ __forceinline__ void init(const Args& a) { tile = blockIdx.x; blk = 0; job = 0; nblk = 1; kblk0 = 0; set_job(a); }
  __device__ __forceinline__ void next(const Args& a) {
    if (++blk == nblk) { blk = 0; tile += gridDim.x; set_job(a); }
  }
};

__device__ __forceinline__ void tmem_ld8(uint32_t taddr, uint32_t (&v)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
               : "r"(taddr) : "memory");
}

// HC8 = 8-column groups of the accumulator owned by one epilogue warp (rcp / 16): 13 for r = 200, 16 = any rcp <= 256
template <int HC8, int MODE = kModeApply>
__global__ void __launch_bounds__(kThreads, 1)
apply_tc_kernel(const __grid_constant__ Args a) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t bar_full[MAX_STAGES], bar_empty[MAX_STAGES], bar_acc_full[2], bar_acc_empty[2];
  __shared__ uint32_t tmem_slot;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int NS = a.nstages;
  // register split: the factor update's, or the logits passes' (top-k, with 128 logits and no counters, takes the former)
  constexpr bool kUpdateRegs = MODE == kModeApply || MODE == kModeTopk;
  if (tid == 0) {
    for (int s = 0; s < NS; ++s) { mbar_init(&bar_full[s], kProdWarps + 1); mbar_init(&bar_empty[s], 1); }
    for (int i = 0; i < 2; ++i) { mbar_init(&bar_acc_full[i], 1); mbar_init(&bar_acc_empty[i], kEpiWarps); }
    fence_mbar_init();
  }
  if (warp == kMmaWarp) tmem_alloc<512>(&tmem_slot);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const int halfcols = a.rcp >> 1;                 // columns of the accumulator owned by one epilogue warp
  // the launch gives every thread 128 registers; the epilogue warps need 104 accumulators + a 32-register drain batch

  if (warp < kEpiWarps) {
    // ================= epilogue: partial sums -> fp32 running sum (round to nearest) -> Y =================
    if (kUpdateRegs) asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" :: "n"(kRegsEpi));
    else asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;\n" :: "n"(kRegsEpiLogits));
    const int quarter = warp & 3, half = warp >> 2;
    constexpr int NACC = HC8 * 8;
    float acc[NACC];
#pragma unroll
    for (int j = 0; j < NACC; ++j) acc[j] = 0.0f;
    PROF_DECL;
    // rank mode: "greater" counts of this thread's row(s), one 4-bit counter per column (16 columns per word)
    uint32_t cntw[HC8];
    int cnt_job = -1, cnt_tiles = 0;
    double lacc = 0.0;
#pragma unroll
    for (int u = 0; u < HC8; ++u) cntw[u] = 0u;
    // sum the counters over the lanes and add them to greater[] (job = query block the counters belong to)
    auto flush_counts = [&](int job_of) {
      if (MODE != kModeRank || job_of < 0) return;
      const int q0 = job_of * 256 + (warp >> 2) * halfcols;
#pragma unroll
      for (int c = 0; c < HC8 * 8; ++c) {
        const int v = (int)((cntw[c >> 3] >> ((c & 7) * 4)) & 15u);
        const int tot = __reduce_add_sync(0xffffffffu, v);
        if (lane == (c & 31) && tot && c < halfcols && q0 + c < a.B) atomicAdd(a.greater + q0 + c, tot);
      }
#pragma unroll
      for (int u = 0; u < HC8; ++u) cntw[u] = 0u;
    };
    int g = 0;                                       // finished partial sums so far (accumulator = g & 1)
    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
      int job = 0;
      while (job + 1 < a.njobs && tile >= a.job[job + 1].tile0) ++job;
      const Job& J = a.job[job];
      const int ngroups = (J.nblk + a.gb - 1) / a.gb;
      for (int grp = 0; grp < ngroups; ++grp, ++g) {
        const int ab = g & 1;
        PROF_BEGIN;
        mbar_wait(&bar_acc_full[ab], (uint32_t)(g >> 1) & 1u);
        PROF_END(pw0);
        fence_after_sync();
        const bool first = grp == 0;                 // first partial sum of the tile: set, do not add
        const uint32_t tbase = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(ab * 256 + half * halfcols);
#pragma unroll
        for (int cb = 0; cb < HC8 / 4; ++cb) {
          if (cb * 32 < halfcols) {
            uint32_t v[32];
            tmem_ld32(tbase + (uint32_t)(cb * 32), v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j)
              acc[cb * 32 + j] = first ? __uint_as_float(v[j]) : acc[cb * 32 + j] + __uint_as_float(v[j]);
          }
        }
#pragma unroll
        for (int c8 = (HC8 / 4) * 4; c8 < HC8; ++c8) {
          if (c8 * 8 < halfcols) {
            uint32_t v[8];
            tmem_ld8(tbase + (uint32_t)(c8 * 8), v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 8; ++j)
              acc[c8 * 8 + j] = first ? __uint_as_float(v[j]) : acc[c8 * 8 + j] + __uint_as_float(v[j]);
          }
        }
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&bar_acc_empty[ab]);
      }
      PROF_BEGIN;
      if (MODE == kModeRank) {
        // ---- filtered-ranking epilogue: acc[c] = logit of (entity row, query column) ----
        if (job != cnt_job || cnt_tiles == 15) { flush_counts(cnt_job); cnt_job = job; cnt_tiles = 0; }
        ++cnt_tiles;
        const int e_loc = (tile - J.tile0) * TM + quarter * 32 + lane;       // entity (row) of this thread (reps == 1)
        const bool rv = e_loc < J.n;
        const int e_glob = a.n_begin + e_loc;
        const int q0 = job * 256 + half * halfcols;                          // first query of this warp's columns
        const int Bp = 256 * a.njobs;
        const float* lo_p = a.thr + q0;
        const float* hi_p = a.thr + Bp + q0;
        const float* eq_p = a.thr + 2 * Bp + q0;
        float lsum = 0.0f;
        // does any query of these columns have a saturated target (p_t == 1)?  (eqlo finite: rare, warp-uniform)
        bool any_eq = false;
#pragma unroll
        for (int c4 = 0; c4 < NACC; c4 += 4) {
          const float4 e4 = __ldg(reinterpret_cast<const float4*>(eq_p + c4));
          any_eq |= (e4.x < INFINITY) | (e4.y < INFINITY) | (e4.z < INFINITY) | (e4.w < INFINITY);
        }
        RankChunkCtx cx;
        cx.lo = lo_p; cx.hi = hi_p; cx.eq = eq_p; cx.slope = a.thr + 3 * Bp + q0; cx.onorm = rv ? __ldg(a.onorms + e_loc) : 0.0f;
        cx.target = a.target; cx.equal = a.equal; cx.equal_before = a.equal_before;
        cx.cand = a.cand; cx.cand_count = a.cand_count; cx.cand_cap = a.cand_cap; cx.B = a.B; cx.q0 = q0; cx.e_loc = e_loc;
        cx.e_glob = e_glob; cx.rv = rv; cx.any_eq = any_eq;
#pragma unroll
        for (int c8 = 0; c8 < HC8; ++c8) {
          const RankChunkOut o = rank_chunk8(cx, c8 * 8, acc[c8 * 8], acc[c8 * 8 + 1], acc[c8 * 8 + 2], acc[c8 * 8 + 3],
                                             acc[c8 * 8 + 4], acc[c8 * 8 + 5], acc[c8 * 8 + 6], acc[c8 * 8 + 7]);
          cntw[c8] += o.counts;
          lsum += o.lsum;
        }
        lacc += (double)lsum;
      } else if (MODE == kModeScore) {
        // ---- score epilogue: G[e][b] = dBCE/dz and the BCE itself for ALL-NEGATIVE targets (t = t_neg), with the
        //      reference's fp32 semantics (exact.cuh: p = 1 / (1 + expf(-z)), log terms clamped at -100, gradient
        //      scaled by p (1 - p) / max(p (1 - p), 1e-12)); the sparse positives are fixed up afterwards ----
        const int e_loc = (tile - J.tile0) * TM + quarter * 32 + lane;
        const bool rv = e_loc < J.n;
        const int q0 = job * 256 + half * halfcols;
        float* grow = a.G + (int64_t)e_loc * a.ldg + q0;
        const float tn = a.t_neg, inv = a.inv_count;
        float lsum = 0.0f;
#pragma unroll
        for (int c8 = 0; c8 < HC8; ++c8)
          lsum += score_chunk8(grow + c8 * 8, rv, a.B - (q0 + c8 * 8), tn, inv, acc[c8 * 8], acc[c8 * 8 + 1], acc[c8 * 8 + 2],
                               acc[c8 * 8 + 3], acc[c8 * 8 + 4], acc[c8 * 8 + 5], acc[c8 * 8 + 6], acc[c8 * 8 + 7]);
        lacc += (double)lsum;
      } else if (MODE == kModeTopk) {
        // ---- top-k candidate epilogue: acc[c] = logit of (entity row, query column) ----
        const int e_loc = (tile - J.tile0) * TM + quarter * 32 + lane;
        const bool rv = e_loc < J.n;
        const int q0 = job * 256 + half * halfcols;
        const int Bp = 256 * a.njobs;
        const float onorm = rv ? __ldg(a.onorms + e_loc) : 0.0f;
#pragma unroll
        for (int c8 = 0; c8 < HC8; ++c8)
          topk_chunk8(a.thr + q0 + c8 * 8, a.thr + 3 * Bp + q0 + c8 * 8, onorm, rv, a.B - (q0 + c8 * 8), q0 + c8 * 8, e_loc,
                      a.topk_cnt, a.topk_seg, a.cand_cap, acc[c8 * 8], acc[c8 * 8 + 1], acc[c8 * 8 + 2], acc[c8 * 8 + 3],
                      acc[c8 * 8 + 4], acc[c8 * 8 + 5], acc[c8 * 8 + 6], acc[c8 * 8 + 7]);
      } else if (MODE == kModeLse) {
        // ---- CE log-sum-exp epilogue: (m, s) of this warp's 32 rows per query column -> part[row group][column]
        //      (G reinterpreted as float2 [4 * tiles per job][ldg]) ----
        const int e_loc = (tile - J.tile0) * TM + quarter * 32 + lane;
        const bool rv = e_loc < J.n;
        const int q0 = job * 256 + half * halfcols;
        float2* dst = reinterpret_cast<float2*>(a.G) + (int64_t)((tile - J.tile0) * 4 + quarter) * a.ldg + q0;
#pragma unroll
        for (int c8 = 0; c8 < HC8; ++c8)
          lse_chunk8(dst + c8 * 8, rv, a.B - (q0 + c8 * 8), acc[c8 * 8], acc[c8 * 8 + 1], acc[c8 * 8 + 2], acc[c8 * 8 + 3],
                     acc[c8 * 8 + 4], acc[c8 * 8 + 5], acc[c8 * 8 + 6], acc[c8 * 8 + 7]);
      } else if (MODE == kModeCe) {
        // ---- CE gradient epilogue: thr = row statistics [M_b | log2 S_b] with stride ldg (ce_row_stats) ----
        const int e_loc = (tile - J.tile0) * TM + quarter * 32 + lane;
        const bool rv = e_loc < J.n;
        const int q0 = job * 256 + half * halfcols;
        float* grow = a.G + (int64_t)e_loc * a.ldg + q0;
        const float tn = a.t_neg, inv = a.inv_count;
        float lsum = 0.0f;
#pragma unroll
        for (int c8 = 0; c8 < HC8; ++c8)
          lsum += ce_chunk8(grow + c8 * 8, a.thr + q0 + c8 * 8, a.thr + a.ldg + q0 + c8 * 8, rv, a.B - (q0 + c8 * 8), tn, inv,
                            acc[c8 * 8], acc[c8 * 8 + 1], acc[c8 * 8 + 2], acc[c8 * 8 + 3], acc[c8 * 8 + 4], acc[c8 * 8 + 5],
                            acc[c8 * 8 + 6], acc[c8 * 8 + 7]);
        lacc += (double)lsum;
      } else {
      const int lt = tile - J.tile0, rep = lt / J.tiles_per_rep;
      const int row0 = (lt - rep * J.tiles_per_rep) * TM;
      const int row = quarter * 32 + lane;
      if (row0 + row < J.n) {
        const float a0 = J.a0 ? (float)(*J.a0) : 1.0f;
        float* y = J.Y + (int64_t)rep * J.y_rep + (int64_t)(row0 + row) * J.ldy + half * halfcols;
        const float* x0 = J.X0 ? J.X0 + (int64_t)(row0 + row) * J.ldx0 + half * halfcols : nullptr;
        const int cmax = min(halfcols, a.rc - half * halfcols);     // valid columns of this half
        const bool vec = ((J.ldy & 3) == 0) && ((reinterpret_cast<uintptr_t>(J.Y) & 15) == 0) &&
                         (!x0 || (((J.ldx0 & 3) == 0) && ((reinterpret_cast<uintptr_t>(J.X0) & 15) == 0)));
#pragma unroll
        for (int j = 0; j < NACC; j += 4) {
          if (j < cmax) {
            if (vec && j + 4 <= cmax) {
              float4 r = make_float4(acc[j], acc[j + 1], acc[j + 2], acc[j + 3]);
              if (x0) {
                const float4 x = *reinterpret_cast<const float4*>(x0 + j);
                r.x = fmaf(a0, x.x, r.x); r.y = fmaf(a0, x.y, r.y); r.z = fmaf(a0, x.z, r.z); r.w = fmaf(a0, x.w, r.w);
              }
              *reinterpret_cast<float4*>(y + j) = r;
            } else {
#pragma unroll
              for (int u = 0; u < 4; ++u)
                if (j + u < cmax) y[j + u] = x0 ? fmaf(a0, x0[j + u], acc[j + u]) : acc[j + u];
            }
          }
        }
      }
      }
      PROF_END(pw1);
    }
    if (MODE == kModeRank) {
      flush_counts(cnt_job);
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) lacc += __shfl_xor_sync(0xffffffffu, lacc, o);
      if (lane == 0 && lacc != 0.0) atomicAdd(a.loss_sum, lacc);
    }
    if (MODE == kModeScore || MODE == kModeCe) {   // one slot per epilogue warp: summed later in a fixed order
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) lacc += __shfl_xor_sync(0xffffffffu, lacc, o);
      if (lane == 0) a.loss_partial[blockIdx.x * kEpiWarps + warp] = lacc;
    }
    if (tid == 0) { PROF_PRINT("epilogue (acc_full, store)"); }
  } else if (warp < kEpiWarps + kProdWarps) {
    // ================= producers: X block -> hi / lo operand images (+ optional raw copy) =================
    if (kUpdateRegs) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOther));
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOtherLogits));
    const int ptid = tid - kEpiWarps * 32;             // 0 .. kProdWarps*32-1
    // thread -> (16-byte chunk ch of the block's 4, rows r0, r0 + rstep, ...).  Row-major terms: 4 lanes cover the 64
    // contiguous bytes of a row; transposed terms (element (row, k) at X + k * ld + row): a warp per chunk, lanes along
    // the rows, so that the loads coalesce either way
    constexpr int RSTEP_N = kProdWarps * 8, RSTEP_T = 32;
    // blocks this CTA will produce
    int todo = 0;
    for (int tile = blockIdx.x; tile < a.ntiles; tile += gridDim.x) {
      int job = 0;
      while (job + 1 < a.njobs && tile >= a.job[job + 1].tile0) ++job;
      todo += a.job[job].nblk;
    }
    // ---- load side: a (tile, term, k-block) walk whose per-term state lives in registers ----
    int l_tile = blockIdx.x - gridDim.x, l_job = 0, l_t = 0, l_nk = 0, l_kb = 0, l_nkb = 0;
    int l_k = 0, l_rk = 0, l_nitems = 0, l_left = todo, l_rep = 0, l_trow = 0, l_rows = 0;
    bool l_fast = false, l_xt = false;
    const float* l_p = nullptr; float* l_q = nullptr;
    int64_t l_pstep = 0, l_qstep = 0, l_kstep = 0, l_ld = 0;
    uint32_t l_smoff = 0, l_smstep = 0;
    float4 xf[PF][XPT];
    float* cq[PF]; int64_t cqstep[PF]; int cni[PF];    // raw-copy destination of the block held in slot u (cni < 0: slow path)
    uint32_t csm[PF], csmstep[PF];                     // shared-memory offset of the thread's first item and item stride
    auto load_next = [&](float4 (&x)[XPT], float*& q, int64_t& qstep, int& ni_copy, uint32_t& smo, uint32_t& sms) {
      if (l_kb == l_nkb) {                             // next term, or next tile
        if (++l_t >= l_nk) {
          l_tile += gridDim.x;
          l_job = 0;
          while (l_job + 1 < a.njobs && l_tile >= a.job[l_job + 1].tile0) ++l_job;
          const Job& J = a.job[l_job];
          l_nk = J.nk; l_t = 0;
          const int lt = l_tile - J.tile0;
          l_rep = lt / J.tiles_per_rep;
          l_trow = (lt - l_rep * J.tiles_per_rep) * TM;
          l_rows = min(TM, J.n - l_trow);
        }
        const Job& J = a.job[l_job];
        l_xt = J.xt[l_t] != 0;
        const int ch = l_xt ? (ptid >> 5) : (ptid & 3), r0 = l_xt ? (ptid & 31) : (ptid >> 2);
        const int rstep = l_xt ? RSTEP_T : RSTEP_N;
        l_smoff = (uint32_t)ch * CS_X + (uint32_t)(r0 >> 3) * RS + (uint32_t)(r0 & 7) * 16u;
        l_smstep = (uint32_t)(rstep / 8) * RS;
        const int left = l_rows - r0;
        l_nitems = left <= 0 ? 0 : (left + rstep - 1) / rstep;
        const float* X = J.X[l_t] + (int64_t)l_rep * J.x_rep[l_t];
        l_ld = J.ldx[l_t];
        l_rk = J.rk[l_t];
        l_kb = 0; l_nkb = J.blk_end[l_t] - (l_t ? J.blk_end[l_t - 1] : 0);
        l_k = 4 * ch;
        const int row = l_trow + r0;
        if (l_xt) {
          l_p = X + (int64_t)l_k * l_ld + row;
          l_pstep = rstep; l_kstep = (int64_t)KB * l_ld;
          l_fast = false;
        } else {
          l_p = X + (int64_t)row * l_ld + l_k;
          l_pstep = (int64_t)rstep * l_ld; l_kstep = KB;
          l_fast = ((l_ld & 3) == 0) && ((reinterpret_cast<uintptr_t>(X) & 15) == 0) && ((l_rk & 3) == 0);
        }
        l_q = nullptr; l_qstep = 0;
        if (J.copy[l_t] && !l_xt) {
          l_q = J.copy[l_t] + (int64_t)row * J.ldc[l_t] + l_k;
          l_qstep = (int64_t)rstep * J.ldc[l_t];
          l_fast = l_fast && ((J.ldc[l_t] & 3) == 0) && ((reinterpret_cast<uintptr_t>(J.copy[l_t]) & 15) == 0);
        }
      }
      q = l_q; qstep = l_qstep; smo = l_smoff; sms = l_smstep;
      if (l_fast) {
        const int ni = (l_k < l_rk) ? l_nitems : 0;
        ni_copy = ni;
        const int nl = DBG(0) ? 0 : ni;
#pragma unroll
        for (int i = 0; i < XPT; ++i)
          x[i] = i < nl ? __ldg(reinterpret_cast<const float4*>(l_p + i * l_pstep)) : make_float4(0.f, 0.f, 0.f, 0.f);
      } else {
        ni_copy = -1 - (l_nitems + 16 * max(0, min(4, l_rk - l_k)));
        const int64_t ks = l_xt ? l_ld : 1;            // distance between consecutive k of one row
#pragma unroll
        for (int i = 0; i < XPT; ++i) {
          const float* p = l_p + i * l_pstep;
          const bool on = i < l_nitems && !DBG(0);
          x[i].x = (on && l_k + 0 < l_rk) ? __ldg(p) : 0.f;
          x[i].y = (on && l_k + 1 < l_rk) ? __ldg(p + ks) : 0.f;
          x[i].z = (on && l_k + 2 < l_rk) ? __ldg(p + 2 * ks) : 0.f;
          x[i].w = (on && l_k + 3 < l_rk) ? __ldg(p + 3 * ks) : 0.f;
        }
      }
      ++l_kb; l_k += KB; l_p += l_kstep; if (l_q) l_q += KB;
      --l_left;
    };
    PROF_DECL;
    int ps = 0; uint32_t pphase = 0;                   // stage / parity of the produce side
    bool wrapped = false;
    auto produce = [&](const float4 (&x)[XPT], float* q, int64_t qstep, int ni_copy, uint32_t smo, uint32_t sms) {
      PROF_BEGIN;
      if (wrapped) mbar_wait(&bar_empty[ps], pphase ^ 1u);
      PROF_END(pw0);
      PROF_BEGIN;
      unsigned char* st = smem + (size_t)ps * a.stage_bytes + smo;
#pragma unroll
      for (int i = 0; i < XPT; ++i) {
        const float4 v = x[i];
        uint4 h, l;
        if (DBG(5)) { h = make_uint4(__float_as_uint(v.x), __float_as_uint(v.y), __float_as_uint(v.z), __float_as_uint(v.w)); l = h; }
        else {
        split_tf32_fast(v.x, h.x, l.x); split_tf32_fast(v.y, h.y, l.y);
        split_tf32_fast(v.z, h.z, l.z); split_tf32_fast(v.w, h.w, l.w);
        }
        *reinterpret_cast<uint4*>(st + i * sms) = h;
        *reinterpret_cast<uint4*>(st + X_HALF + i * sms) = l;
      }
      if (q) {                                         // raw copy of the block (the data is in registers by now)
        if (ni_copy >= 0) {
#pragma unroll
          for (int i = 0; i < XPT; ++i)
            if (i < ni_copy) *reinterpret_cast<float4*>(q + i * qstep) = x[i];
        } else {                                       // unaligned / ragged: ni_copy = -1 - (nitems + 16 * valid k)
          const int code = -1 - ni_copy, nitems = code & 15, kleft = code >> 4;
#pragma unroll
          for (int i = 0; i < XPT; ++i) {
            float* qq = q + i * qstep;
            const bool on = i < nitems;
            if (on && 0 < kleft) qq[0] = x[i].x;
            if (on && 1 < kleft) qq[1] = x[i].y;
            if (on && 2 < kleft) qq[2] = x[i].z;
            if (on && 3 < kleft) qq[3] = x[i].w;
          }
        }
      }
      if (!DBG(4)) fence_async_smem();
      __syncwarp();
      if (lane == 0) mbar_arrive(&bar_full[ps]);
      PROF_END(pw1);
      if (++ps == NS) { ps = 0; pphase ^= 1u; wrapped = true; }
    };
#pragma unroll
    for (int u = 0; u < PF; ++u)
      if (l_left > 0) load_next(xf[u], cq[u], cqstep[u], cni[u], csm[u], csmstep[u]);
    while (todo > 0) {
#pragma unroll
      for (int u = 0; u < PF; ++u) {
        if (todo > 0) {
          produce(xf[u], cq[u], cqstep[u], cni[u], csm[u], csmstep[u]);
          --todo;
          if (l_left > 0) load_next(xf[u], cq[u], cqstep[u], cni[u], csm[u], csmstep[u]);
        }
      }
    }
    if (ptid == 0) { PROF_PRINT("producer (empty, produce)"); }
  } else if (warp == kMmaWarp) {
    // ================= MMA issuer =================
    if (kUpdateRegs) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOther));
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOtherLogits));
    if (lane == 0) {
      const uint32_t idesc = make_idesc_tf32(TM, a.rcp, false, false);
      Cursor c;
      c.init(a);
      int g = 0;
      PROF_DECL;
      int s = 0; uint32_t phase = 0;
      for (; c.valid(a); c.next(a)) {
        const bool group_start = (c.blk % a.gb) == 0;
        const bool group_end = c.blk == c.nblk - 1 || ((c.blk + 1) % a.gb) == 0;
        const int ab = g & 1;
        PROF_BEGIN;
        if (group_start && g >= 2) mbar_wait(&bar_acc_empty[ab], (uint32_t)((g >> 1) - 1) & 1u);
        PROF_END(pw1);
        PROF_BEGIN;
        mbar_wait(&bar_full[s], phase);
        PROF_END(pw0);
        fence_after_sync();
        const uint32_t aXh = smem_u32(smem + (size_t)s * a.stage_bytes), aXl = aXh + X_HALF;
        const uint32_t aKh = aXh + 2 * X_HALF, aKl = aKh + (KB / 4) * a.cs_k;
        const uint32_t d = tmem + (uint32_t)(ab * 256);
#pragma unroll
        for (int ks = 0; ks < KB / 8; ++ks) {
          if (DBG(2) && !(group_start && ks == 0)) continue;
          const uint64_t dXh = make_desc(aXh + ks * 2 * CS_X, CS_X, RS), dXl = make_desc(aXl + ks * 2 * CS_X, CS_X, RS);
          const uint64_t dKh = make_desc(aKh + ks * 2 * a.cs_k, a.cs_k, RS), dKl = make_desc(aKl + ks * 2 * a.cs_k, a.cs_k, RS);
          mma_tf32(d, dXl, dKh, idesc, !(group_start && ks == 0));     // small terms first
          mma_tf32(d, dXh, dKl, idesc, true);
          mma_tf32(d, dXh, dKh, idesc, true);
        }
        mma_commit(&bar_empty[s]);
        if (group_end) { mma_commit(&bar_acc_full[ab]); ++g; }
        if (++s == NS) { s = 0; phase ^= 1u; }
      }
      PROF_PRINT("mma (full, acc_empty)");
    }
    __syncwarp();
  } else if (warp == kLoadWarp) {
    // ================= K image loader =================
    if (kUpdateRegs) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOther));
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOtherLogits));
    if (lane == 0) {
      Cursor c;
      c.init(a);
      PROF_DECL;
      int s = 0; uint32_t phase = 0; bool wrapped = false;
      for (; c.valid(a); c.next(a)) {
        PROF_BEGIN;
        if (wrapped) mbar_wait(&bar_empty[s], phase ^ 1u);
        PROF_END(pw0);
        if (DBG(1) && wrapped) mbar_arrive(&bar_full[s]);
        else {
          mbar_expect_tx(&bar_full[s], a.kimg_bytes);
          bulk_g2s(smem + (size_t)s * a.stage_bytes + 2 * X_HALF,
                   a.Kimg + (size_t)(c.kblk0 + c.blk) * a.kimg_bytes, a.kimg_bytes, &bar_full[s]);
        }
        if (++s == NS) { s = 0; phase ^= 1u; wrapped = true; }
      }
      PROF_PRINT("loader (empty)");
    }
    __syncwarp();
  } else {
    if (kUpdateRegs) asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOther));
    else asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;\n" :: "n"(kRegsOtherLogits));     // idle warps of the last warpgroup
  }
  fence_before_sync();
  __syncthreads();
  if (warp == kMmaWarp) tmem_dealloc<512>(tmem);
}

struct Plan { int rcp, nstages; uint32_t cs_k, kimg_bytes, stage_bytes; size_t smem; };
Plan make_plan(int rc) {
  Plan p;
  p.rcp = (rc + 15) / 16 * 16;
  p.cs_k = (uint32_t)p.rcp * 16u + 16u;
  p.kimg_bytes = 2u * (KB / 4) * p.cs_k;
  p.stage_bytes = 2 * X_HALF + p.kimg_bytes;
  int ns = (int)(SMEM_LIMIT / p.stage_bytes);
  p.nstages = ns > MAX_STAGES ? MAX_STAGES : ns;
  p.smem = (size_t)p.nstages * p.stage_bytes;
  return p;
}


// ---------------------------------------------------------------------------------------------------------------
// Rank mode: filtered ranking without the B x N probability matrix (reference: filter_predictions + metrics,
// src/utils/utils.py:15-22, src/utils/metrics.py:4-22, on the scores of R_TuckER.py:47-48).
//
// The reference ranks fp32 probabilities p = sigmoid(z) with z an fp32 dot product.  The tensor-core pass computes
// every logit to ~4e-7 relative (3xTF32 + round-to-nearest partial sums) and classifies it against per-query logit
// thresholds derived from the target's probability: above `hi` the entity certainly has p > p_t, below `lo`
// certainly p < p_t, above `eqlo` (only when p_t == 1) certainly p == 1 == p_t.  Everything in between -- a few
// entities per query -- goes to a candidate list and is recomputed by rank_candidates_kernel with the EXACT fp32
// arithmetic of the dense path (exact.cuh), so the counts equal the ones the fp32 kernel produces.  Filtered entities
// are corrected from their exact probabilities afterwards.
// ---------------------------------------------------------------------------------------------------------------

// max_j ||O_j||^2 over the shard (bounds the error of a logit); out is a float bit pattern updated with atomicMax
__global__ void rank_rownorm_kernel(const float* __restrict__ O, int n_local, int r2, unsigned int* out,
                                    float* __restrict__ norms) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int nwarps = (gridDim.x * blockDim.x) >> 5;
  float best = 0.0f;
  for (int j = warp; j < n_local; j += nwarps) {
    float s = 0.0f;
    for (int k = lane; k < r2; k += 32) { const float v = __ldg(O + (int64_t)j * r2 + k); s = fmaf(v, v, s); }
    s = rt::warp_sum(s);
    best = fmaxf(best, s);
    // an UPPER bound of ||O_j|| (the fp32 sum of squares is off by at most r2 * 2^-24 relative)
    if (lane == 0) norms[j] = sqrtf(s) * (1.0f + 1e-4f) + 1e-30f;
  }
  if (lane == 0) atomicMax(out, __float_as_uint(best));
}

// thresholds thr[4][Bp] of every query from p_target: (lo0, hi0, eqlo0, slope).  The band of entity j is
// [lo0 - slope * ||O_j||, hi0 + slope * ||O_j||] (eqlo0 + slope * ||O_j|| for the saturated-target test): the error
// bound of a logit is proportional to ||q_b|| ||O_j|| with the entity's OWN norm -- with the shard maximum the band
// of every entity was as wide as the heaviest row needs (rows 8x heavier than average after a few hundred steps: the
// candidate list filled up and the evaluation batch went from 0.9 to 4 ms).  Queries >= B get an empty band.
// slope of query b's band (one warp): |z_fp32 - z_tensor| <= (r2 * 2^-24 + 1e-6) * ||q|| ||o||  (fp32 recurrence +
// 3xTF32); factor 2 of safety, and 1e-3 relative for the fp32 evaluation of lo0 - slope * norm in the epilogue
__device__ __forceinline__ float rank_band_slope(const float* __restrict__ q, int b, int r2, int lane) {
  float s = 0.0f;
  for (int k = lane; k < r2; k += 32) { const float v = __ldg(q + (int64_t)b * r2 + k); s = fmaf(v, v, s); }
  s = rt::warp_sum(s);
  return (float)(2.0 * ((double)r2 * 5.96e-8 + 1e-6) * sqrt((double)s) * 1.001) + 1e-30f;
}

__global__ void rank_thresholds_kernel(const float* __restrict__ q, const float* __restrict__ p_target, int B, int Bp,
                                       int r2, float* __restrict__ thr) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= Bp) return;
  float lo = INFINITY, hi = INFINITY, eqlo = INFINITY, slope = 0.0f;
  if (b < B) {
    slope = rank_band_slope(q, b, r2, lane);
    const double margin = 2e-6;                      // absolute part of the old margin (+ the conversions to fp32)
    const float pt = __ldg(p_target + b);
    if (pt >= 1.0f) {                 // saturated target: nothing is greater; z > 18 certainly gives p == 1
      lo = 15.0f; hi = INFINITY; eqlo = (float)(18.5 + margin);
    } else if (pt <= 0.0f) {          // p_t == 0: ties only with other underflowed probabilities
      lo = -INFINITY; hi = (float)(-80.0 + margin);
    } else {
      const double u = (double)nextafterf(pt, 2.0f) - (double)pt;
      const double plo = (double)pt - 2.0 * u, phi = (double)pt + 2.0 * u;
      lo = plo > 0.0 ? (float)(log(plo / (1.0 - plo)) - margin - 1e-6) : -INFINITY;
      hi = phi < 1.0 ? (float)(log(phi / (1.0 - phi)) + margin + 1e-6) : 19.0f;
      lo = nextafterf(lo, -INFINITY); hi = nextafterf(hi, INFINITY);
      lo -= 4e-7f * fabsf(lo); hi += 4e-7f * fabsf(hi);        // rounding of lo0 - m, hi0 + m in the epilogue
    }
  }
  if (lane == 0) { thr[b] = lo; thr[Bp + b] = hi; thr[2 * Bp + b] = eqlo; thr[3 * Bp + b] = slope; }
}

// Logit space (rt_score_rank_logit, rt_score_topk_logit): thresholds of a per-query reference LOGIT z_ref (the target's
// exact fp32 logit, or the top-k sample threshold z_k).  lo0 = hi0 = z_ref widened by 4e-7 |z_ref| and one ulp, eqlo0 =
// +inf (no saturated-target test: logits do not saturate), slope as above.  The bound: the epilogue classifies the
// tensor-core logit z' of entity j against lo_u = fl(lo0 - m), hi_u = fl(hi0 + m), m = fl(slope ||O_j||) >= 2 E_j,
// E_j = the error bound above, so |z - z'| <= E_j for the exact fp32 logit z.  Round to nearest moves hi0 + m by at
// most 2^-24 |hi0 + m| <= 6e-8 (|hi0| + m): the widening of hi0 covers the |hi0| part, the factor 2 of m its m part,
// so hi_u >= z_ref + E_j and z' > hi_u gives z > z_ref (certainly greater); symmetrically z' < lo_u gives z < z_ref.
// Everything in [lo_u, hi_u] is a candidate and is recounted from its exact logit.  Queries >= B: empty band.
__global__ void logit_thresholds_kernel(const float* __restrict__ q, const float* __restrict__ z_ref, int B, int Bp,
                                        int r2, float* __restrict__ thr) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= Bp) return;
  float lo = INFINITY, hi = INFINITY, slope = 0.0f;
  if (b < B) {
    slope = rank_band_slope(q, b, r2, lane);
    const double z = (double)__ldg(z_ref + b);
    lo = nextafterf((float)(z - 4e-7 * fabs(z)), -INFINITY);
    hi = nextafterf((float)(z + 4e-7 * fabs(z)), INFINITY);
  }
  if (lane == 0) { thr[b] = lo; thr[Bp + b] = hi; thr[2 * Bp + b] = INFINITY; thr[3 * Bp + b] = slope; }
}

// K images of the query chunks: job j, block kb: element (c, kk) = q[256 j + c][kb * KB + kk]
__global__ void rank_pack_q_kernel(const float* __restrict__ q, int B, int r2, int nblk, int rcp, unsigned char* img,
                                   uint32_t cs_k, uint32_t kimg_bytes) {
  const int blk = blockIdx.x, job = blk / nblk, kb = blk - job * nblk;
  unsigned char* out = img + (size_t)blk * kimg_bytes;
  const uint32_t half = (KB / 4) * cs_k;
  for (int e = threadIdx.x; e < KB * rcp; e += blockDim.x) {
    const int c = e / KB, kk = e - c * KB;
    const int b = job * 256 + c, k = kb * KB + kk;
    const float v = (b < B && k < r2) ? __ldg(q + (int64_t)b * r2 + k) : 0.0f;
    uint32_t hi, lo;
    split_tf32(v, hi, lo);
    const uint32_t off = (uint32_t)(kk >> 2) * cs_k + (uint32_t)(c >> 3) * RS + (uint32_t)(c & 7) * 16u + (uint32_t)(kk & 3) * 4u;
    *reinterpret_cast<uint32_t*>(out + off) = hi;
    *reinterpret_cast<uint32_t*>(out + half + off) = lo;
  }
}

// LOGIT: compare exact logits with the target's logit (p_target then holds z_target)
template <bool LOGIT>
__global__ void rank_candidates_kernel(const float* __restrict__ q, const float* __restrict__ O, int r2, int n_begin,
                                       const int32_t* __restrict__ target, const float* __restrict__ p_target,
                                       const int2* __restrict__ cand, const int* __restrict__ cand_count, int cap,
                                       int32_t* greater, int32_t* equal, int32_t* equal_before, int* overflow) {
  const int n = *cand_count;
  if (n > cap) { if (blockIdx.x == 0 && threadIdx.x == 0) *overflow = 1; return; }
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
    const int2 c = cand[i];
    const int j = n_begin + c.x, b = c.y, t = __ldg(target + b);
    if (j == t) continue;
    const float z = rt::exact_logit(q + (int64_t)b * r2, O + (int64_t)c.x * r2, r2);
    const float p = LOGIT ? z : rt::sigmoid_ref(z);
    const float pt = __ldg(p_target + b);
    if (p > pt) atomicAdd(greater + b, 1);
    else if (p == pt) { atomicAdd(equal + b, 1); if (j < t) atomicAdd(equal_before + b, 1); }
  }
}

// one THREAD per filter entry (a warp per query made the hub queries -- thousands of known objects -- the critical path:
// 245 us per batch of 512 on WN18RR): entities of the filter list count as p' = 0 (utils.py:19) and as positives of the BCE
__global__ void rank_filter_fix_kernel(const float* __restrict__ q, const float* __restrict__ O, int B, int r2,
                                       int n_begin, int n_local, const int32_t* __restrict__ target,
                                       const float* __restrict__ p_target, const int32_t* __restrict__ flt_off,
                                       const int32_t* __restrict__ flt_idx, int32_t* greater, int32_t* equal,
                                       int32_t* equal_before, double* loss_sum, const int* __restrict__ overflow) {
  if (*overflow) return;                              // the fp32 kernel redoes the batch
  const int nnz = __ldg(flt_off + B);
  double dl = 0.0;
  for (int i = __ldg(flt_off) + blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += gridDim.x * blockDim.x) {
    int lo = 0, hi = B;                               // query of entry i: flt_off[b] <= i < flt_off[b + 1]
    while (hi - lo > 1) { const int mid = (lo + hi) >> 1; if (__ldg(flt_off + mid) <= i) lo = mid; else hi = mid; }
    const int b = lo;
    const int f = __ldg(flt_idx + i), fl = f - n_begin;
    if (fl < 0 || fl >= n_local) continue;
    const int t = __ldg(target + b);
    const float pt = __ldg(p_target + b);
    const float z = rt::exact_logit(q + (int64_t)b * r2, O + (int64_t)fl * r2, r2);
    const float p = rt::sigmoid_ref(z);
    const float lp = rt::bce_log_p(p), lq = rt::bce_log_q(p);
    dl += (double)(-lp) - (double)(-lq);              // the pass over all entities charged -log(1 - p)
    if (f != t) {
      const int was_eq = (p == pt), is_eq = (0.0f == pt);
      if (p > pt) atomicAdd(greater + b, -1);
      if (is_eq != was_eq) {
        atomicAdd(equal + b, is_eq - was_eq);
        if (f < t) atomicAdd(equal_before + b, is_eq - was_eq);
      }
    }
  }
  dl = rt::warp_sum(dl);
  if ((threadIdx.x & 31) == 0 && dl != 0.0) atomicAdd(loss_sum, dl);
}

__global__ void rank_finish_kernel(const double* loss_sum, double* bce_sum, const int* overflow) {
  if (threadIdx.x == 0 && blockIdx.x == 0 && !*overflow && bce_sum) *bce_sum = *loss_sum;
}
__global__ void rank_reset_if_overflow_kernel(int B, int32_t* greater, int32_t* equal, int32_t* equal_before,
                                              const int* overflow) {
  if (!*overflow) return;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < B; i += gridDim.x * blockDim.x) {
    greater[i] = 0; equal[i] = 0; equal_before[i] = 0;
  }
}

// ---------------------------------------------------------------------------------------------------------------
// The logits passes (rank, top-k, BCE score, log-sum-exp, CE score): Z = O q^T on apply_tc_kernel, rows = the n_local
// entities of the shard, the B queries in jobs of 256 columns, contraction over r2; the epilogue mode decides what
// becomes of the logits.  Their shapes: rt::rank_tc_supported.
// ---------------------------------------------------------------------------------------------------------------
struct LogitGeom { int njobs, Bp, nblk, tiles_per_job; size_t kimg_bytes; };   // kimg_bytes: all query images
LogitGeom logit_geom(int B, int n_local, int r2) {
  LogitGeom g;
  g.njobs = rt::cdiv(B, 256); g.Bp = 256 * g.njobs; g.nblk = rt::cdiv(r2, KB); g.tiles_per_job = rt::cdiv(n_local, TM);
  g.kimg_bytes = (size_t)g.njobs * g.nblk * make_plan(256).kimg_bytes;
  return g;
}

// Packs q into the query images at kimg and runs the logits pass with epilogue MODE on min(tiles, SMs) persistent
// CTAs.  `a` carries the mode's own fields (thresholds and counters, G and loss slots, top-k segments); the modes with
// loss slots get them zeroed before the launch.
template <int MODE>
int launch_logits(Args a, const float* q, const float* O, int B, int r2, int n_local, unsigned char* kimg,
                  cudaStream_t s) {
  const Plan p = make_plan(256);
  const LogitGeom g = logit_geom(B, n_local, r2);
  rank_pack_q_kernel<<<g.njobs * g.nblk, 256, 0, s>>>(q, B, r2, g.nblk, p.rcp, kimg, p.cs_k, p.kimg_bytes);
  RT_LAUNCH_CHECK();
  a.rc = 256; a.rcp = p.rcp; a.nstages = p.nstages; a.cs_k = p.cs_k; a.kimg_bytes = p.kimg_bytes; a.gb = GB_LOGITS;
  a.stage_bytes = p.stage_bytes; a.Kimg = kimg;
  a.njobs = g.njobs; a.ntiles = g.njobs * g.tiles_per_job; a.B = B;
  for (int j = 0; j < g.njobs; ++j) {
    Job& J = a.job[j];
    J.n = n_local; J.nk = 1; J.X[0] = O; J.ldx[0] = r2; J.rk[0] = r2;
    for (int t = 0; t < MAX_TERMS; ++t) J.blk_end[t] = g.nblk;
    J.nblk = g.nblk; J.kblk0 = j * g.nblk; J.tile0 = j * g.tiles_per_job; J.ntiles = g.tiles_per_job;
    J.reps = 1; J.tiles_per_rep = g.tiles_per_job;
  }
#ifdef RT_APPLY_PROF
  a.debug = getenv("RT_APPLY_DEBUG") ? atoi(getenv("RT_APPLY_DEBUG")) : 0;
#endif
  if (MODE == kModeScore || MODE == kModeCe)
    RT_CHECK_CUDA(cudaMemsetAsync(a.loss_partial, 0, sizeof(double) * (size_t)rt::sm_count() * kEpiWarps, s));
  const int grid = std::min(a.ntiles, rt::sm_count());
  RT_CHECK_CUDA(rt::ensure_dyn_smem((const void*)apply_tc_kernel<16, MODE>, SMEM_LIMIT));
  apply_tc_kernel<16, MODE><<<grid, kThreads, p.smem, s>>>(a);
  RT_LAUNCH_CHECK();
  return 0;
}

// Workspace of the rank and top-k passes: scalars, per-query band thresholds [4][Bp], entity norms, query images, and
// a candidate list of `cap` (local entity, query) pairs (the rank pass; top-k keeps its candidates in the per-query
// segments of its caller and passes cap = 0)
struct BandLayout { LogitGeom g; size_t scal, thr, norms, kimg, cand, total; int cap; };
BandLayout band_layout(int B, int n_local, int r2, int cap) {
  BandLayout L;
  L.g = logit_geom(B, n_local, r2);
  L.cap = cap;
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += rt::align_up(bytes, 256); return at; };
  L.scal = take(256);                                 // [0] cand_count, [1] overflow, [2] max ||O_j||^2, [4..5] loss (double)
  L.thr = take(sizeof(float) * 4 * L.g.Bp);
  L.norms = take(sizeof(float) * (size_t)(n_local > 0 ? n_local : 1));
  L.kimg = take(L.g.kimg_bytes);
  L.cand = take(sizeof(int2) * (size_t)cap);
  L.total = o;
  return L;
}
BandLayout rank_layout(int B, int n_local, int r2) {
  const long long all = (long long)B * n_local;
  return band_layout(B, n_local, r2, (int)std::min<long long>(std::max<long long>(all / 8, 1 << 16), 1 << 22));
}

}  // namespace

namespace rt {
// the shapes of every logits pass: at most MAX_JOBS jobs of 256 queries, a contraction of 64 .. 1024, shards of at
// least 1024 rows, three pipeline stages at width 256
bool rank_tc_supported(int B, int n_local, int r2) {
  return B >= 1 && B <= 256 * MAX_JOBS && r2 >= 64 && r2 <= 1024 && n_local >= 1024 && make_plan(256).nstages >= 3;
}
size_t rank_tc_ws_bytes(int B, int n_local, int r2) { return rank_layout(B, n_local, r2).total; }
static int rank_tc_impl(bool logit, const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                        const int32_t* target, const float* p_target, const int32_t* flt_off, const int32_t* flt_idx,
                        int32_t* greater, int32_t* equal, int32_t* equal_before, double* bce_sum, void* ws, cudaStream_t s,
                        const int** overflow_flag);
// Counts and BCE of one evaluation batch on the tensor cores; *overflow_flag (device int inside ws, returned) is set
// when the candidate list did not fit: the caller then runs the fp32 kernel gated on that flag.
int rank_tc(const float* q, const float* O, int B, int r2, int n_begin, int n_local, const int32_t* target,
            const float* p_target, const int32_t* flt_off, const int32_t* flt_idx, int32_t* greater, int32_t* equal,
            int32_t* equal_before, double* bce_sum, void* ws, cudaStream_t s, const int** overflow_flag) {
  return rank_tc_impl(false, q, O, B, r2, n_begin, n_local, target, p_target, flt_off, flt_idx, greater, equal,
                      equal_before, bce_sum, ws, s, overflow_flag);
}
// Logit space (rank_logit.cu): counts of every entity of the shard against z_target, the target itself excluded and
// the filter list NOT applied (the caller removes it); counts are zeroed when the candidate list overflowed, with
// *overflow_flag set as above.  The epilogue's BCE sum goes to a scratch slot of ws.
int rank_tc_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local, const int32_t* target,
                  const float* z_target, int32_t* greater, int32_t* equal, int32_t* equal_before, void* ws,
                  cudaStream_t s, const int** overflow_flag) {
  return rank_tc_impl(true, q, O, B, r2, n_begin, n_local, target, z_target, nullptr, nullptr, greater, equal,
                      equal_before, nullptr, ws, s, overflow_flag);
}
static int rank_tc_impl(bool logit, const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                        const int32_t* target, const float* p_target, const int32_t* flt_off, const int32_t* flt_idx,
                        int32_t* greater, int32_t* equal, int32_t* equal_before, double* bce_sum, void* ws, cudaStream_t s,
                        const int** overflow_flag) {
  const BandLayout L = rank_layout(B, n_local, r2);
  char* base = (char*)ws;
  int* scal = (int*)(base + L.scal);
  double* loss = (double*)(base + L.scal + 16);
  float* thr = (float*)(base + L.thr);
  RT_CHECK_CUDA(cudaMemsetAsync(scal, 0, 256, s));
  float* onorms = (float*)(base + L.norms);
  rank_rownorm_kernel<<<rt::sm_count() * 4, 256, 0, s>>>(O, n_local, r2, (unsigned int*)(scal + 2), onorms);
  RT_LAUNCH_CHECK();
  if (logit) logit_thresholds_kernel<<<rt::cdiv(L.g.Bp, 8), 256, 0, s>>>(q, p_target, B, L.g.Bp, r2, thr);
  else rank_thresholds_kernel<<<rt::cdiv(L.g.Bp, 8), 256, 0, s>>>(q, p_target, B, L.g.Bp, r2, thr);
  RT_LAUNCH_CHECK();
  Args a{};
  a.thr = thr; a.onorms = onorms; a.target = target; a.n_begin = n_begin;
  a.greater = greater; a.equal = equal; a.equal_before = equal_before;
  a.cand = (int2*)(base + L.cand); a.cand_count = scal; a.cand_cap = L.cap; a.loss_sum = loss;
  if (int rc = launch_logits<kModeRank>(a, q, O, B, r2, n_local, (unsigned char*)(base + L.kimg), s)) return rc;
  if (logit) {
    rank_candidates_kernel<true><<<rt::sm_count() * 2, 256, 0, s>>>(q, O, r2, n_begin, target, p_target, a.cand, scal,
                                                                    L.cap, greater, equal, equal_before, scal + 1);
    RT_LAUNCH_CHECK();
    rank_reset_if_overflow_kernel<<<rt::cdiv(B, 256), 256, 0, s>>>(B, greater, equal, equal_before, scal + 1);
    RT_LAUNCH_CHECK();
    *overflow_flag = scal + 1;
    return 0;
  }
  rank_candidates_kernel<false><<<rt::sm_count() * 2, 256, 0, s>>>(q, O, r2, n_begin, target, p_target, a.cand, scal,
                                                                   L.cap, greater, equal, equal_before, scal + 1);
  RT_LAUNCH_CHECK();
  rank_filter_fix_kernel<<<rt::sm_count() * 2, 128, 0, s>>>(q, O, B, r2, n_begin, n_local, target, p_target, flt_off, flt_idx,
                                                        greater, equal, equal_before, loss, scal + 1);
  RT_LAUNCH_CHECK();
  rank_finish_kernel<<<1, 32, 0, s>>>(loss, bce_sum, scal + 1);
  RT_LAUNCH_CHECK();
  rank_reset_if_overflow_kernel<<<rt::cdiv(B, 256), 256, 0, s>>>(B, greater, equal, equal_before, scal + 1);
  RT_LAUNCH_CHECK();
  *overflow_flag = scal + 1;
  return 0;
}

// ---- top-k mode: the rank-mode pass with the per-query sample threshold p_k in place of p_target (topk.cu) ----
size_t topk_tc_ws_bytes(int B, int n_local, int r2) { return band_layout(B, n_local, r2, 0).total; }
}  // namespace rt

namespace {
// queries the sample already sent to the exact pass get an empty band
__global__ void topk_empty_band_kernel(float* __restrict__ thr, int B, const int* __restrict__ flag) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b < B && flag[b]) thr[b] = INFINITY;
}
}  // namespace

namespace rt {
// Appends to seg[b][0, cap) every entity j of the shard whose tensor-core logit is not certainly below the logit of
// p_k[b] (the band of rank_thresholds_kernel for p_target = p_k); cnt[b] (zeroed by the caller) ends as the number of
// such entities, > cap when the segment overflowed.  Queries with flag[b] != 0 are skipped.
// logit: p_k holds the sample's logit threshold z_k and the band is logit_thresholds_kernel's.
int topk_tc_pass(const float* q, const float* O, int B, int r2, int n_local, const float* p_k, const int* flag, int* cnt,
                 int32_t* seg, int cap, void* ws, cudaStream_t s, bool logit) {
  const BandLayout L = band_layout(B, n_local, r2, 0);
  char* base = (char*)ws;
  unsigned int* maxnorm = (unsigned int*)(base + L.scal + 8);
  float* thr = (float*)(base + L.thr);
  float* onorms = (float*)(base + L.norms);
  RT_CHECK_CUDA(cudaMemsetAsync(maxnorm, 0, sizeof(unsigned int), s));
  rank_rownorm_kernel<<<rt::sm_count() * 4, 256, 0, s>>>(O, n_local, r2, maxnorm, onorms);
  RT_LAUNCH_CHECK();
  if (logit) logit_thresholds_kernel<<<rt::cdiv(L.g.Bp, 8), 256, 0, s>>>(q, p_k, B, L.g.Bp, r2, thr);
  else rank_thresholds_kernel<<<rt::cdiv(L.g.Bp, 8), 256, 0, s>>>(q, p_k, B, L.g.Bp, r2, thr);
  RT_LAUNCH_CHECK();
  topk_empty_band_kernel<<<rt::cdiv(B, 256), 256, 0, s>>>(thr, B, flag);
  RT_LAUNCH_CHECK();
  Args a{};
  a.thr = thr; a.onorms = onorms;
  a.topk_seg = seg; a.topk_cnt = cnt; a.cand_cap = cap;
  return launch_logits<kModeTopk>(a, q, O, B, r2, n_local, (unsigned char*)(base + L.kimg), s);
}
}  // namespace rt

// ---- C ABI -------------------------------------------------------------------------------------------
extern "C" int rt_apply_tc_supported(int rc, int nk, const int* rk_host) {
  if (rc < 1 || rc > RCP_MAX || nk < 1 || nk > MAX_TERMS) return 0;
  for (int t = 0; t < nk; ++t)
    if (rk_host[t] < 1) return 0;
  return make_plan(rc).nstages >= 3 ? 1 : 0;
}

extern "C" size_t rt_apply_tc_ws_bytes(int rc, int nk, const int* rk_host) {
  const Plan p = make_plan(rc);
  size_t blocks = 0;
  for (int t = 0; t < nk; ++t) blocks += rt::cdiv(rk_host[t], KB);
  return blocks * p.kimg_bytes + 256;
}

extern "C" size_t rt_apply_multi_ws_bytes(int njobs, const rt_apply_job* jobs, int rc) {
  const Plan p = make_plan(rc);
  size_t blocks = 0;
  for (int j = 0; j < njobs; ++j)
    for (int t = 0; t < jobs[j].nk; ++t) blocks += rt::cdiv(jobs[j].rk[t], KB);
  return blocks * p.kimg_bytes + 256;
}

namespace {
// internal job description: rt_apply_job plus what the score kernel needs (fp32 right factors, transposed and
// replicated terms)
struct TermSpec { const float* X; int64_t ldx; int rk; const void* K; int k_f32; int xt; float* copy; int64_t ldc;
                  int64_t x_rep; int rows_total; };
struct JobSpec { float* Y; int64_t ldy; int n; const float* X0; int64_t ldx0; const double* a0; int nk; TermSpec t[MAX_TERMS];
                 int reps; int64_t y_rep; };

size_t run_apply_ws_bytes(int njobs, const JobSpec* jobs, int rc) {
  const Plan p = make_plan(rc);
  size_t blocks = 0;
  for (int j = 0; j < njobs; ++j)
    for (int t = 0; t < jobs[j].nk; ++t) blocks += (size_t)std::max(jobs[j].reps, 1) * rt::cdiv(jobs[j].t[t].rk, KB);
  return blocks * p.kimg_bytes + 256;
}

int run_apply(int njobs, const JobSpec* jobs, int rc, void* ws, cudaStream_t s) {
  const Plan p = make_plan(rc);
  Args a{};
  PackArgs pk{};
  a.rc = rc; a.rcp = p.rcp; a.nstages = p.nstages; a.cs_k = p.cs_k; a.kimg_bytes = p.kimg_bytes; a.gb = GB;
  a.stage_bytes = p.stage_bytes; a.Kimg = (const unsigned char*)ws;
  int tiles = 0, blocks = 0, nj = 0, nterms = 0;
  for (int j = 0; j < njobs; ++j) {
    const JobSpec& in = jobs[j];
    if (in.n == 0) continue;
    const int reps = std::max(in.reps, 1);
    RT_REQUIRE(reps == 1 || in.nk == 1, "run_apply: replicated jobs have one term");
    Job& J = a.job[nj++];
    J.Y = in.Y; J.ldy = in.ldy; J.X0 = in.X0; J.ldx0 = in.ldx0; J.a0 = in.a0; J.n = in.n; J.nk = in.nk;
    J.reps = reps; J.tiles_per_rep = rt::cdiv(in.n, TM); J.y_rep = in.y_rep;
    J.kblk0 = blocks; J.tile0 = tiles; J.ntiles = reps * J.tiles_per_rep;
    int b = 0;
    for (int t = 0; t < MAX_TERMS; ++t) {
      const bool on = t < in.nk;
      const TermSpec& T = in.t[t];
      J.X[t] = on ? T.X : nullptr; J.ldx[t] = on ? T.ldx : 0; J.rk[t] = on ? T.rk : 0;
      J.copy[t] = on ? T.copy : nullptr; J.ldc[t] = on ? T.ldc : 0;
      J.xt[t] = on ? T.xt : 0; J.x_rep[t] = on ? T.x_rep : 0;
      if (on) {
        RT_REQUIRE(T.copy != in.Y || T.copy == nullptr, "rt_apply_multi: copy_out may not alias Y");
        const int nb = rt::cdiv(T.rk, KB);
        pk.K[nterms] = T.K; pk.rk[nterms] = T.rk; pk.blk0[nterms] = blocks + b; pk.f32[nterms] = T.k_f32;
        pk.rep_blocks[nterms] = reps > 1 ? nb : 0;
        pk.rows_total[nterms] = T.rows_total > 0 ? T.rows_total : T.rk * reps;
        ++nterms;
        b += nb;
      }
      J.blk_end[t] = b;
    }
    J.nblk = b;
    blocks += b * reps;
    tiles += J.ntiles;
  }
  if (nj == 0) return 0;
  a.njobs = nj; a.ntiles = tiles;
#ifdef RT_APPLY_PROF
  a.debug = getenv("RT_APPLY_DEBUG") ? atoi(getenv("RT_APPLY_DEBUG")) : 0;
#endif
  pk.blk0[nterms] = blocks; pk.nterms = nterms; pk.rc = rc; pk.rcp = p.rcp; pk.img = (unsigned char*)ws;
  pk.cs_k = p.cs_k; pk.kimg_bytes = p.kimg_bytes;
  pack_K_kernel<<<blocks, 256, 0, s>>>(pk);
  RT_LAUNCH_CHECK();
  const int grid = tiles < rt::sm_count() ? tiles : rt::sm_count();
  if (p.rcp == 208) {
    RT_CHECK_CUDA(rt::ensure_dyn_smem((const void*)apply_tc_kernel<13>, SMEM_LIMIT));
    apply_tc_kernel<13><<<grid, kThreads, p.smem, s>>>(a);
  } else {
    RT_CHECK_CUDA(rt::ensure_dyn_smem((const void*)apply_tc_kernel<16>, SMEM_LIMIT));
    apply_tc_kernel<16><<<grid, kThreads, p.smem, s>>>(a);
  }
  RT_LAUNCH_CHECK();
  return 0;
}

// ---------------------------------------------------------------------------------------------------------------
// Score mode: fused 1-N score + BCE + backward at fp32 accuracy on the tensor cores (variant 3).
//   1. logits Z = O Q^T by the 3xTF32 kernel (rows = entities, 256 queries per job); its epilogue turns them into
//      the BCE and G = dBCE/dZ for all-negative targets with the reference's fp32 semantics and stores G[e][b];
//   2. the few positives (CSR targets) are recomputed exactly and patched into G and the loss;
//   3. dO = G Q        -- the same kernel as a plain factor update (X = G, right factor = the query rows);
//   4. H  = G^T O      -- the same kernel on transposed operand blocks, the contraction over the entities cut into
//                          chunks (replicated job) whose partial results are summed in a fixed order.
// The logit / probability matrices never exist; G (B x N fp32, 84 MB at WN18RR size) is staged between the three
// launches and stays resident in the 126 MB L2.
//
// 1-N softmax cross-entropy on the tensor cores (variant 3 of rt_score_lse / rt_score_ce_fwd_bwd, rtucker.h).
//   log-sum-exp pass: the score mode's logits (same query images, job layout and 3xTF32 accumulation), epilogue
//     kModeLse writes (m, s) per (32-row group, query); lse_combine (score_bce.cu) merges the groups in a fixed order;
//   gradient pass: ce_row_stats turns the parts of all shards into (M_b, log2 S_b), then the four steps above with
//     epilogue kModeCe (G = (softmax - ls/N) / B and the ls/N part of the loss) and score_ce_fix_positives_kernel.
// ---------------------------------------------------------------------------------------------------------------
__global__ void score_fix_positives_kernel(const float* __restrict__ q, const float* __restrict__ O, int B, int r2,
                                           int n_begin, int n_local, const int32_t* __restrict__ off,
                                           const int32_t* __restrict__ idx, float t_pos, float t_neg, float inv_count,
                                           float* __restrict__ G, int64_t ldg, double* __restrict__ delta) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  double dl = 0.0;
  for (int i = __ldg(off + b) + lane; i < __ldg(off + b + 1); i += 32) {
    const int fl = __ldg(idx + i) - n_begin;
    if (fl < 0 || fl >= n_local) continue;
    const float z = rt::exact_logit(q + (int64_t)b * r2, O + (int64_t)fl * r2, r2);
    const float p = rt::sigmoid_ref(z);
    const float lp = rt::bce_log_p(p), lq = rt::bce_log_q(p);
    G[(int64_t)fl * ldg + b] = rt::bce_grad(p, t_pos, inv_count);
    dl += -(double)(t_pos - t_neg) * ((double)lp - (double)lq);     // the kernel charged the negative-target term
  }
  dl = rt::warp_sum(dl);
  if (lane == 0) delta[b] = dl;
}

__global__ void score_ce_fix_positives_kernel(const float* __restrict__ q, const float* __restrict__ O, int B, int r2,
                                              int n_begin, int n_local, const int32_t* __restrict__ off,
                                              const int32_t* __restrict__ idx, float one_minus_ls, float t_neg,
                                              float inv_count, const float* __restrict__ stats, int ldst,
                                              float* __restrict__ G, int64_t ldg, double* __restrict__ delta) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  const int e0 = __ldg(off + b), e1 = __ldg(off + b + 1);
  const float tp = e1 > e0 ? one_minus_ls / (float)(e1 - e0) : 0.0f;    // (1 - ls) / |y_b| from the FULL target list
  const float M = __ldg(stats + b), L2 = __ldg(stats + ldst + b);
  double dl = 0.0;
  for (int i = e0 + lane; i < e1; i += 32) {
    const int fl = __ldg(idx + i) - n_begin;
    if (fl < 0 || fl >= n_local) continue;
    const float d = rt::exact_logit(q + (int64_t)b * r2, O + (int64_t)fl * r2, r2) - M;
    const float p = rt::ce_softmax(d, L2);
    G[(int64_t)fl * ldg + b] = (p - (tp + t_neg)) * inv_count;
    dl += (double)tp * ((double)L2 * 0.6931471805599453 - (double)d);   // the epilogue charged the ls/N part
  }
  // a query without targets: loss_b = lse_b - (ls/N) sum_j z_bj, i.e. (1 - ls) lse_b beyond the ls/N part, charged
  // once, to the shard that starts at entity 0
  if (lane == 0 && e1 == e0 && n_begin == 0 && L2 < INFINITY) dl += (double)one_minus_ls * ((double)M + (double)L2 * 0.6931471805599453);
  dl = rt::warp_sum(dl);
  if (lane == 0) delta[b] = dl;
}

__global__ void score_finish_kernel(const float* __restrict__ Hpart, int reps, int count, float* __restrict__ H,
                                    const double* __restrict__ loss_slots, int nslots, const double* __restrict__ delta,
                                    int B, double* __restrict__ loss_out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < count) {
    float s = 0.0f;
    for (int r = 0; r < reps; ++r) s += Hpart[(size_t)r * count + i];      // fixed order
    H[i] = s;
  }
  if (blockIdx.x == 0 && threadIdx.x < 32) {       // lane-strided partial sums + butterfly: the same association every run
    double t = 0.0;
    for (int k = threadIdx.x; k < nslots; k += 32) t += loss_slots[k];
    for (int b = threadIdx.x; b < B; b += 32) t += delta[b];
    t = rt::warp_sum(t);
    if (threadIdx.x == 0) loss_out[0] = t;
  }
}

struct ScoreLayout { LogitGeom g; size_t G, kq, kws, hpart, slots, delta, total; int chunk, reps; };
ScoreLayout score_layout(int B, int n_local, int r2) {
  ScoreLayout L;
  L.g = logit_geom(B, n_local, r2);
  // H = G^T O: chunks of the entity range so that (query tiles) x (chunks) fills the SMs about once
  const int qtiles = rt::cdiv(B, TM);
  int reps = std::max(1, rt::sm_count() / qtiles);
  int chunk = rt::cdiv(rt::cdiv(n_local, reps), KB) * KB;
  if (chunk < 256) chunk = 256;
  L.chunk = chunk; L.reps = rt::cdiv(n_local, chunk);
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += rt::align_up(bytes, 256); return at; };
  L.G = take(sizeof(float) * (size_t)L.reps * L.chunk * L.g.Bp);
  L.kq = take(L.g.kimg_bytes);
  JobSpec j2{}; j2.n = n_local; j2.nk = 1; j2.t[0].rk = B; j2.reps = 1;
  JobSpec j3{}; j3.n = B; j3.nk = 1; j3.t[0].rk = L.chunk; j3.reps = L.reps;
  L.kws = take(std::max(run_apply_ws_bytes(1, &j2, r2), run_apply_ws_bytes(1, &j3, r2)));
  L.hpart = take(sizeof(float) * (size_t)L.reps * B * r2);
  L.slots = take(sizeof(double) * (size_t)rt::sm_count() * kEpiWarps);
  L.delta = take(sizeof(double) * (size_t)B);
  L.total = o;
  return L;
}

// The four steps with epilogue MODE: kModeScore (label-smoothed BCE) or kModeCe (softmax cross-entropy; stats = the
// row statistics [M_b | log2 S_b] of ce_row_stats, stride Bp).
template <int MODE>
int score_tc3(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local, int n_total,
              int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing, const float* stats,
              double* loss_sum, float* H, float* dO, void* ws, cudaStream_t s) {
  const ScoreLayout L = score_layout(B, n_local, r2);
  const int Bp = L.g.Bp;
  char* base = (char*)ws;
  float* G = (float*)(base + L.G);
  double* delta = (double*)(base + L.delta);
  const float t_neg = label_smoothing / (float)n_total;
  const float inv_count = MODE == kModeCe ? (float)(1.0 / (double)b_total)
                                          : (float)(1.0 / ((double)b_total * (double)n_total));
  // rows [n_local, reps * chunk) of G are contraction padding of step 4
  const size_t pad_rows = (size_t)L.reps * L.chunk - n_local;
  if (pad_rows) RT_CHECK_CUDA(cudaMemsetAsync(G + (size_t)n_local * Bp, 0, pad_rows * Bp * sizeof(float), s));
  // ---- 1. logits -> loss, G for all-negative targets ----
  Args a{};
  a.n_begin = n_begin; a.G = G; a.ldg = Bp; a.t_neg = t_neg; a.inv_count = inv_count; a.thr = stats;
  a.loss_partial = (double*)(base + L.slots);
  if (int rc = launch_logits<MODE>(a, q, O, B, r2, n_local, (unsigned char*)(base + L.kq), s)) return rc;
  // ---- 2. positives ----
  if (MODE == kModeCe)
    score_ce_fix_positives_kernel<<<rt::cdiv(B, 8), 256, 0, s>>>(q, O, B, r2, n_begin, n_local, tgt_off, tgt_idx,
                                                                 1.0f - label_smoothing, t_neg, inv_count, stats, Bp, G,
                                                                 Bp, delta);
  else
    score_fix_positives_kernel<<<rt::cdiv(B, 8), 256, 0, s>>>(q, O, B, r2, n_begin, n_local, tgt_off, tgt_idx,
                                                              (1.0f - label_smoothing) + t_neg, t_neg, inv_count, G, Bp,
                                                              delta);
  RT_LAUNCH_CHECK();
  // ---- 3. dO = G Q'  (Q' = qp = q A_O when the caller folds the right factor of the projection in, else q) ----
  {
    JobSpec j{};
    j.Y = dO; j.ldy = r2; j.n = n_local; j.nk = 1; j.reps = 1;
    j.t[0].X = G; j.t[0].ldx = Bp; j.t[0].rk = B; j.t[0].K = qp ? qp : q; j.t[0].k_f32 = 1; j.t[0].rows_total = B;
    int rc = run_apply(1, &j, r2, base + L.kws, s);
    if (rc) return rc;
  }
  // ---- 4. H = G^T O in entity chunks ----
  {
    JobSpec j{};
    float* Hpart = (float*)(base + L.hpart);
    j.Y = Hpart; j.ldy = r2; j.n = B; j.nk = 1; j.reps = L.reps; j.y_rep = (int64_t)B * r2;
    j.t[0].X = G; j.t[0].ldx = Bp; j.t[0].xt = 1; j.t[0].rk = L.chunk; j.t[0].x_rep = (int64_t)L.chunk * Bp;
    j.t[0].K = O; j.t[0].k_f32 = 1; j.t[0].rows_total = n_local;
    int rc = run_apply(1, &j, r2, base + L.kws, s);
    if (rc) return rc;
    score_finish_kernel<<<rt::cdiv(B * r2, 256), 256, 0, s>>>(Hpart, L.reps, B * r2, H, (const double*)(base + L.slots),
                                                              rt::sm_count() * kEpiWarps, delta, B, loss_sum);
    RT_LAUNCH_CHECK();
  }
  return 0;
}

struct LseLayout { LogitGeom g; size_t kq, part, total; int groups; };
LseLayout lse_layout(int B, int n_local, int r2) {
  LseLayout L;
  L.g = logit_geom(B, n_local, r2);
  L.groups = 4 * L.g.tiles_per_job;                          // 32-row groups of one job's tiles
  size_t o = 0;
  auto take = [&](size_t bytes) { size_t at = o; o += rt::align_up(bytes, 256); return at; };
  L.kq = take(L.g.kimg_bytes);
  L.part = take(sizeof(float2) * (size_t)L.groups * L.g.Bp);
  L.total = o;
  return L;
}
}  // namespace

extern "C" int rt_score_bce_tc3_supported(int B, int n_local, int r2) {
  return (rt::rank_tc_supported(B, n_local, r2) && r2 <= RCP_MAX && make_plan(r2).nstages >= 3) ? 1 : 0;
}
extern "C" size_t rt_score_bce_tc3_ws_bytes(int B, int n_local, int r2) { return score_layout(B, n_local, r2).total; }

extern "C" int rt_score_bce_tc3(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local,
                                int n_total, int b_total, const int32_t* tgt_off, const int32_t* tgt_idx,
                                float label_smoothing, double* loss_sum, float* H, float* dO, void* ws, void* stream) {
  RT_REQUIRE(rt_score_bce_tc3_supported(B, n_local, r2), "rt_score_bce_tc3: unsupported shape B=%d n_local=%d r2=%d", B, n_local, r2);
  RT_REQUIRE(ws != nullptr, "rt_score_bce_tc3: workspace is NULL");
  return score_tc3<kModeScore>(q, qp, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx, label_smoothing,
                               nullptr, loss_sum, H, dO, ws, (cudaStream_t)stream);
}

namespace rt {
size_t score_lse_tc3_ws_bytes(int B, int n_local, int r2) { return lse_layout(B, n_local, r2).total; }

int score_lse_tc3(const float* q, const float* O, int B, int r2, int n_local, float* parts, void* ws, cudaStream_t s) {
  const LseLayout L = lse_layout(B, n_local, r2);
  char* base = (char*)ws;
  Args a{};
  a.G = (float*)(base + L.part); a.ldg = L.g.Bp;
  if (int rc = launch_logits<kModeLse>(a, q, O, B, r2, n_local, (unsigned char*)(base + L.kq), s)) return rc;
  return lse_combine((const float2*)(base + L.part), L.groups, L.g.Bp, B, parts, s);
}

size_t score_ce_tc3_ws_bytes(int B, int n_local, int r2) {
  const ScoreLayout L = score_layout(B, n_local, r2);
  return L.total + rt::align_up(sizeof(float) * 2 * (size_t)L.g.Bp, 256);
}

int score_ce_tc3(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local, int n_total,
                 int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing, const float* parts,
                 int nparts, double* loss_sum, float* H, float* dO, void* ws, cudaStream_t s) {
  const ScoreLayout L = score_layout(B, n_local, r2);
  float* stats = (float*)((char*)ws + L.total);              // [M_b | log2 S_b], stride Bp
  if (int rc = ce_row_stats(parts, nparts, B, L.g.Bp, stats, s)) return rc;
  return score_tc3<kModeCe>(q, qp, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx, label_smoothing,
                            stats, loss_sum, H, dO, ws, s);
}
}  // namespace rt

extern "C" int rt_apply_multi(int njobs, const rt_apply_job* jobs, int rc, void* ws, void* stream) {
  RT_REQUIRE(njobs >= 1 && njobs <= MAX_JOBS, "rt_apply_multi: 1..%d jobs per launch, got %d", MAX_JOBS, njobs);
  RT_REQUIRE(ws != nullptr, "rt_apply_multi: workspace is NULL");
  JobSpec js[MAX_JOBS] = {};
  for (int j = 0; j < njobs; ++j) {
    const rt_apply_job& in = jobs[j];
    RT_REQUIRE(rt_apply_tc_supported(rc, in.nk, in.rk), "rt_apply_multi: unsupported shape rc=%d nk=%d", rc, in.nk);
    JobSpec& o = js[j];
    o.Y = in.Y; o.ldy = in.ldy; o.n = in.n; o.X0 = in.X0; o.ldx0 = in.ldx0; o.a0 = in.a0_dev; o.nk = in.nk; o.reps = 1;
    for (int t = 0; t < in.nk; ++t) {
      o.t[t].X = in.X[t]; o.t[t].ldx = in.ldx[t]; o.t[t].rk = in.rk[t]; o.t[t].K = in.K[t]; o.t[t].k_f32 = 0;
      o.t[t].copy = in.copy_out[t]; o.t[t].ldc = in.ldcopy[t]; o.t[t].rows_total = in.rk[t];
    }
  }
  return run_apply(njobs, js, rc, ws, (cudaStream_t)stream);
}

extern "C" int rt_apply_tc(float* Y, int64_t ldy, int n, int rc, const float* X0, int64_t ldx0, const double* a0_dev,
                           int nk, const float* const* X_host, const int64_t* ldx_host, const int* rk_host,
                           const double* const* K_host, void* ws, void* stream) {
  RT_REQUIRE(rt_apply_tc_supported(rc, nk, rk_host), "rt_apply_tc: unsupported shape rc=%d nk=%d", rc, nk);
  rt_apply_job j{};
  j.Y = Y; j.ldy = ldy; j.n = n; j.X0 = X0; j.ldx0 = ldx0; j.a0_dev = a0_dev; j.nk = nk;
  for (int t = 0; t < nk; ++t) { j.X[t] = X_host[t]; j.ldx[t] = ldx_host[t]; j.rk[t] = rk_host[t]; j.K[t] = K_host[t]; }
  return rt_apply_multi(1, &j, rc, ws, stream);
}
