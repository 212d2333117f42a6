// (b) Fused 1-N scoring: logits, sigmoid, label-smoothed BCE against SPARSE multi-hot targets and
// both backward contractions in one pass over the entity matrix; (d) fused filtered ranking.
//
// Replaces, for training: reference src/model/asymmetric/R_TuckER.py:47-48 (q @ O^T, sigmoid),
// nn.BCELoss(mean) (train.py:79,136) on the dense targets of src/data/Dataset.py:43-52, and the
// autograd backward of those ops (dL/dq and dL/dO).  For evaluation: train.py:112-117
// (predictions, BCE, filter_predictions, metrics) without materialising B x N.
//
// This file is the FP32-FFMA variant (parity path, and the thin-rank path r2 ~ 20).
// Work per launch: 6*B*N*r2 flops (three B x N x r2 contractions), algorithmic bytes 8*N*r2
// (read O once, write dO once).  The tcgen05 variant lives in score_bce_tc.cu.
//
// Decomposition: persistent CTAs; a CTA owns entity tiles of 64 rows; per tile it loops over the
// batch in chunks of 64 queries:  Z = Q_chunk O_tile^T  ->  elementwise (p, loss, G)  ->
// H_chunk += G O_tile (accumulated in this CTA's private workspace slice, summed over CTAs in a
// fixed order afterwards)  and  dO_tile += G^T QP_chunk (registers, across the chunk loop).
#include "common.h"
#include "exact.cuh"
#include <math.h>

namespace {

constexpr int BT = 64;      // queries per chunk
constexpr int NT = 64;      // entities per tile
constexpr int GLD = NT + 4; // leading dim of the G / G^T tiles

// Row stride (floats) of the staged Q / QP / O tiles: wide enough for r2 and for the 16*CPT
// columns the k-major GEMMs touch, with stride/4 odd so float4 row reads are conflict-free.
__host__ __device__ inline int row_ld(int r2, int cpt) {
  int w = r2 > 16 * cpt ? r2 : 16 * cpt;
  w = (w + 3) / 4 * 4;
  return ((w / 4) & 1) ? w : w + 4;
}

// Dynamic shared memory of one staged 64-entity + 64-query tile (stage_logit_tile).
size_t logit_tile_smem(int r2) { return (size_t)(NT + BT) * row_ld(r2, 1) * sizeof(float); }

// The logits of the staged tiles (pitch ldw, zero padded beyond r2): z[i][j] = q_b . O_n for query row ty + 16 i and
// entity row tx + 16 j, one fmaf accumulator, k ascending -- the order of exact_logit, the padding adds exact zeros.
// k_end = r2 rounded up to a multiple of 4, computed by the caller outside its tile loops.
struct LogitTile { float z[4][4]; };
__device__ __forceinline__ LogitTile logit_tile(const float* Qs, const float* Os, int ldw, int k_end) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  LogitTile t;
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) t.z[i][j] = 0.0f;
  for (int k = 0; k < k_end; k += 4) {
    float4 qv[4], ov[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) qv[i] = *reinterpret_cast<const float4*>(Qs + (ty + 16 * i) * ldw + k);
#pragma unroll
    for (int j = 0; j < 4; ++j) ov[j] = *reinterpret_cast<const float4*>(Os + (tx + 16 * j) * ldw + k);
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        t.z[i][j] = fmaf(qv[i].x, ov[j].x, t.z[i][j]);
        t.z[i][j] = fmaf(qv[i].y, ov[j].y, t.z[i][j]);
        t.z[i][j] = fmaf(qv[i].z, ov[j].z, t.z[i][j]);
        t.z[i][j] = fmaf(qv[i].w, ov[j].w, t.z[i][j]);
      }
  }
  return t;
}

// Stages entities [n0, n0 + 64) and queries [b0, b0 + 64) in smem (logit_tile_smem bytes) and returns their logits.
__device__ __forceinline__ LogitTile stage_logit_tile(const float* __restrict__ q, const float* __restrict__ O, int B,
                                                      int r2, int n_local, int n0, int b0, unsigned char* smem) {
  const int ldw = row_ld(r2, 1);
  float* Os = reinterpret_cast<float*>(smem);
  float* Qs = Os + NT * ldw;
  for (int e = threadIdx.x; e < NT * ldw; e += 256) {
    const int rr = e / ldw, cc = e - rr * ldw;
    Os[e] = (n0 + rr < n_local && cc < r2) ? __ldg(O + (int64_t)(n0 + rr) * r2 + cc) : 0.0f;
    Qs[e] = (b0 + rr < B && cc < r2) ? __ldg(q + (int64_t)(b0 + rr) * r2 + cc) : 0.0f;
  }
  __syncthreads();
  return logit_tile(Qs, Os, ldw, (r2 + 3) / 4 * 4);
}

struct ScoreArgs {
  const float* q;
  const float* qp;
  const float* O;
  int B, r2, n_begin, n_local, n_total;
  const int32_t* off;   // CSR row offsets (targets for train, filter lists for eval)
  const int32_t* idx;   // global entity ids
  float t_pos, t_neg;   // smoothed target values
  float inv_count;      // 1 / (B_total * n_total)
  // train outputs
  double* loss_partial; // [grid]
  float* H_ws;          // [grid][B][r2]
  float* dO;            // [n_local][r2]
  // eval
  const int32_t* target;
  const float* p_target;
  int32_t* greater;
  int32_t* equal;
  int32_t* equal_before;
  int n_tiles;
  const int* gate;      // eval only: when not NULL the launch is a no-op unless *gate != 0 (fallback of the tcgen05 ranking)
};

// acc[i][jj] += sum_k Gk[k][ty*4+i] * Mk[k][tx+16*jj],  k < 64
template <int CPT>
__device__ __forceinline__ void gemm_k64(const float* __restrict__ Gk, const float* __restrict__ Mk,
                                         int ld, float (&acc)[4][CPT]) {
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
#pragma unroll 4
  for (int k = 0; k < 64; ++k) {
    const float4 g = *reinterpret_cast<const float4*>(Gk + k * GLD + ty * 4);
    const float gv[4] = {g.x, g.y, g.z, g.w};
    const float* m = Mk + k * ld + tx;
#pragma unroll
    for (int jj = 0; jj < CPT; ++jj) {
      const float mv = m[16 * jj];
#pragma unroll
      for (int i = 0; i < 4; ++i) acc[i][jj] = fmaf(gv[i], mv, acc[i][jj]);
    }
  }
}

// CE (1-N softmax cross-entropy) reuses ScoreArgs: p_target = row statistics [2][B] (max logit M_b, log2 S_b of the
// whole batch row, see ce_row_stats_kernel), t_pos = 1 - ls, t_neg = ls / n_total, inv_count = 1 / B_total.
template <int CPT, bool EVAL, bool CE = false>
__global__ void __launch_bounds__(256, 1)
score_kernel(ScoreArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  if (EVAL && a.gate && *a.gate == 0) return;
  const int r2 = a.r2;
  const int ldw = row_ld(r2, CPT);
  const int k_end = (r2 + 3) / 4 * 4;
  float* Os = reinterpret_cast<float*>(smem_raw);   // [NT][ldw]
  float* Qs = Os + NT * ldw;                        // [BT][ldw]
  float* QPs = Qs + BT * ldw;                       // [BT][ldw]   (train only)
  float* Gz = EVAL ? Qs + BT * ldw : QPs + BT * ldw; // [BT][GLD]  G[b][n]
  float* GzT = Gz + BT * GLD;                       // [NT][GLD]  G^T[n][b]
  unsigned long long* mask = reinterpret_cast<unsigned long long*>(GzT + NT * GLD);  // [BT]
  __shared__ double red[8];

  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  double loss_acc = 0.0;
  const int n_chunks = (a.B + BT - 1) / BT;
  bool first_tile = true;

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int n0 = tile * NT;
    __syncthreads();
    // ---- stage the entity tile (zero padded) ----
    for (int e = threadIdx.x; e < NT * ldw; e += 256) {
      const int rr = e / ldw, cc = e - rr * ldw;
      const int n = n0 + rr;
      Os[e] = (n < a.n_local && cc < r2) ? __ldg(a.O + (int64_t)n * r2 + cc) : 0.0f;
    }
    float acc3[4][CPT];  // dO tile accumulators (train)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int jj = 0; jj < CPT; ++jj) acc3[i][jj] = 0.0f;

    for (int chunk = 0; chunk < n_chunks; ++chunk) {
      const int b0 = chunk * BT;
      __syncthreads();  // previous chunk's consumers of Qs/QPs/Gz are done
      for (int e = threadIdx.x; e < BT * ldw; e += 256) {
        const int rr = e / ldw, cc = e - rr * ldw;
        const int b = b0 + rr;
        const bool ok = (b < a.B && cc < r2);
        Qs[e] = ok ? __ldg(a.q + (int64_t)b * r2 + cc) : 0.0f;
        if (!EVAL) QPs[e] = ok ? __ldg(a.qp + (int64_t)b * r2 + cc) : 0.0f;
      }
      if (threadIdx.x < BT) mask[threadIdx.x] = 0ull;
      __syncthreads();
      {  // positives (train) / filter list (eval) falling into this (chunk, tile)
        const int rr = threadIdx.x >> 2, part = threadIdx.x & 3;
        const int b = b0 + rr;
        if (b < a.B) {
          const int e1 = a.off[b + 1];
          unsigned long long m = 0ull;
          for (int e = a.off[b] + part; e < e1; e += 4) {
            const int o = a.idx[e] - a.n_begin - n0;
            if (o >= 0 && o < NT) m |= (1ull << o);
          }
          if (m) atomicOr(&mask[rr], m);
        }
      }
      // ---- GEMM1: Z[b][n], b = ty + 16 i, n = tx + 16 j ----
      const LogitTile lt = logit_tile(Qs, Os, ldw, k_end);
      __syncthreads();  // mask complete
      // ---- elementwise ----
      float loss_t = 0.0f;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int rr = ty + 16 * i;
        const int b = b0 + rr;
        const unsigned long long m = mask[rr];
        int cg = 0, ce = 0, cb = 0;
        float pt = 0.0f;
        int tcol = -1;
        if (EVAL && b < a.B) { pt = a.p_target[b]; tcol = a.target[b] - a.n_begin - n0; }
        float rowM = 0.0f, rowL = 0.0f, tpos = 0.0f;
        if (CE && b < a.B) {
          rowM = a.p_target[b]; rowL = a.p_target[a.B + b];
          const int cnt = a.off[b + 1] - a.off[b];
          tpos = (cnt > 0 ? a.t_pos / (float)cnt : 0.0f) + a.t_neg;
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int cc = tx + 16 * j;
          const bool valid = (b < a.B) && (n0 + cc < a.n_local);
          const bool pos = (m >> cc) & 1ull;
          const float zz = lt.z[i][j];
          if (CE) {
            // G = (softmax - t) / B_total with softmax = 2^((z - M) log2e - log2 S); loss += t (lse - z)
            const float t = pos ? tpos : a.t_neg;
            float g = 0.0f;
            if (valid) {
              const float d = zz - rowM;
              g = (rt::ce_softmax(d, rowL) - t) * a.inv_count;
              loss_t += rt::ce_loss_term(t, d, rowL);
            }
            Gz[rr * GLD + cc] = g;
            GzT[cc * GLD + rr] = g;
            continue;
          }
          const float p = rt::sigmoid_ref(zz);
          const float lp = rt::bce_log_p(p), lq = rt::bce_log_q(p);
          if (EVAL) {
            const float t = pos ? 1.0f : 0.0f;
            if (valid) {
              loss_t -= t * lp + (1.0f - t) * lq;
              if (cc != tcol) {
                const float v = pos ? 0.0f : p;
                cg += (v > pt);
                const int eq = (v == pt);
                ce += eq;
                cb += eq & (cc < tcol);
              }
            }
          } else {
            const float t = pos ? a.t_pos : a.t_neg;
            float g = 0.0f;
            if (valid) {
              loss_t -= t * lp + (1.0f - t) * lq;
              g = rt::bce_grad(p, t, a.inv_count);
            }
            Gz[rr * GLD + cc] = g;
            GzT[cc * GLD + rr] = g;
          }
        }
        if (EVAL) {
#pragma unroll
          for (int o = 8; o > 0; o >>= 1) {
            cg += __shfl_xor_sync(0xffffffffu, cg, o);
            ce += __shfl_xor_sync(0xffffffffu, ce, o);
            cb += __shfl_xor_sync(0xffffffffu, cb, o);
          }
          if (tx == 0 && b < a.B) {
            if (cg) atomicAdd(a.greater + b, cg);
            if (ce) atomicAdd(a.equal + b, ce);
            if (cb) atomicAdd(a.equal_before + b, cb);
          }
        }
      }
      loss_acc += (double)loss_t;
      if (!EVAL) {
        __syncthreads();  // Gz / GzT visible
        // ---- GEMM2: Hc[b][c] = sum_n G[b][n] O[n][c]   (k-major operand: GzT) ----
        float acc2[4][CPT];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int jj = 0; jj < CPT; ++jj) acc2[i][jj] = 0.0f;
        gemm_k64<CPT>(GzT, Os, ldw, acc2);
        float* Hc = a.H_ws + ((int64_t)blockIdx.x * a.B + b0) * r2;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int rr = ty * 4 + i;
          if (b0 + rr >= a.B) continue;
#pragma unroll
          for (int jj = 0; jj < CPT; ++jj) {
            const int c = tx + 16 * jj;
            if (c >= r2) continue;
            float* p = Hc + (int64_t)rr * r2 + c;
            *p = first_tile ? acc2[i][jj] : (*p + acc2[i][jj]);
          }
        }
        // ---- GEMM3: dO[n][c] += sum_b G[b][n] QP[b][c]   (k-major operand: Gz) ----
        gemm_k64<CPT>(Gz, QPs, ldw, acc3);
      }
    }
    if (!EVAL) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int n = n0 + ty * 4 + i;
        if (n >= a.n_local) continue;
#pragma unroll
        for (int jj = 0; jj < CPT; ++jj) {
          const int c = tx + 16 * jj;
          if (c < r2) a.dO[(int64_t)n * r2 + c] = acc3[i][jj];
        }
      }
    }
    first_tile = false;
  }
  // CTAs that own no tile still have to define their H slice
  if (!EVAL && first_tile) {
    float* Hc = a.H_ws + (int64_t)blockIdx.x * a.B * r2;
    for (int64_t e = threadIdx.x; e < (int64_t)a.B * r2; e += 256) Hc[e] = 0.0f;
  }
  // ---- loss: block reduce in a fixed order ----
  double v = rt::warp_sum(loss_acc);
  if (lane == 0) red[warp] = v;
  __syncthreads();
  if (threadIdx.x == 0) {
    double s = 0.0;
    for (int w = 0; w < 8; ++w) s += red[w];
    a.loss_partial[blockIdx.x] = s;
  }
}

__global__ void reduce_H_kernel(const float* __restrict__ H_ws, int nparts, int64_t count,
                                float* __restrict__ H) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float s = 0.0f;
  for (int k = 0; k < nparts; ++k) s += H_ws[(int64_t)k * count + i];
  H[i] = s;
}

__global__ void reduce_loss_kernel(const double* __restrict__ partial, int n, double* __restrict__ out,
                                   int accumulate) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += partial[i];
    out[0] = accumulate ? out[0] + s : s;
  }
}

__global__ void target_prob_kernel(const float* __restrict__ q, const float* __restrict__ O, int B,
                                   int r2, int n_begin, int n_local, const int32_t* __restrict__ target,
                                   float* __restrict__ p_target) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const int t = target[b] - n_begin;
  const bool local = t >= 0 && t < n_local;
  p_target[b] = local ? rt::sigmoid_ref(rt::exact_logit(q + (int64_t)b * r2, O + (int64_t)t * r2, r2)) : 0.0f;
}

// Dense compatibility path: P[b, j] = sigmoid(q_b . O_j) written out (what score_fn(T) returns in
// the reference, R_TuckER.py:47-48).  gate (may be NULL): the launch is a no-op unless *gate != 0 (the exact
// passes of the top-k selection, topk.cu, and of the logit-space ranking, rank_logit.cu).
// LOGIT: the logits z themselves (rt_score_dense_logits).
template <bool LOGIT = false>
__global__ void __launch_bounds__(256)
score_dense_kernel(const float* __restrict__ q, const float* __restrict__ O, int B, int r2, int n_local,
                   float* __restrict__ P, int64_t ldp, const int* __restrict__ gate) {
  if (gate && *gate == 0) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n0 = blockIdx.x * NT, b0 = blockIdx.y * BT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const LogitTile lt = stage_logit_tile(q, O, B, r2, n_local, n0, b0, smem_raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = b0 + ty + 16 * i;
    if (b >= B) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx + 16 * j;
      if (n < n_local) P[(int64_t)b * ldp + n] = LOGIT ? lt.z[i][j] : rt::sigmoid_ref(lt.z[i][j]);
    }
  }
}

struct Plan {
  int cpt, grid, n_tiles;
  size_t smem;
};

Plan make_plan(int n_local, int r2, bool eval) {
  Plan p;
  p.cpt = (r2 <= 32) ? 2 : (r2 <= 64) ? 4 : (r2 <= 112) ? 7 : (r2 <= 208) ? 13 : 16;
  p.n_tiles = rt::cdiv(n_local, NT);
  const int sms = rt::sm_count();
  const int waves = rt::cdiv(p.n_tiles, sms);
  p.grid = waves > 0 ? rt::cdiv(p.n_tiles, waves) : 1;
  if (p.grid < 1) p.grid = 1;
  const int ldw = row_ld(r2, p.cpt);
  size_t fl = (size_t)NT * ldw + (size_t)BT * ldw * (eval ? 1 : 2) + 2 * (size_t)BT * GLD;
  p.smem = fl * sizeof(float) + BT * sizeof(unsigned long long);
  return p;
}

template <int CPT, bool EVAL, bool CE = false>
int launch(const ScoreArgs& a, const Plan& p, cudaStream_t s) {
  RT_CHECK_CUDA(cudaFuncSetAttribute(score_kernel<CPT, EVAL, CE>,
                                     cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  score_kernel<CPT, EVAL, CE><<<p.grid, 256, p.smem, s>>>(a);
  RT_LAUNCH_CHECK();
  return 0;
}

template <bool EVAL, bool CE = false>
int dispatch(const ScoreArgs& a, const Plan& p, cudaStream_t s) {
  switch (p.cpt) {
    case 2: return launch<2, EVAL, CE>(a, p, s);
    case 4: return launch<4, EVAL, CE>(a, p, s);
    case 7: return launch<7, EVAL, CE>(a, p, s);
    case 13: return launch<13, EVAL, CE>(a, p, s);
    default: return launch<16, EVAL, CE>(a, p, s);
  }
}

// Variant 0 of the training passes, BCE (CE = false) or softmax cross-entropy (CE = true, stats = the row statistics
// of ce_row_stats): score_kernel over the shard, then H and the loss summed over the CTAs in a fixed order.
// ws: [grid][B][r2] partial H, then [grid] partial losses (rt_score_bce_ws_bytes).
template <bool CE>
int score_train_ffma(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local,
                     int n_total, int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing,
                     const float* stats, double* loss_sum, float* H, float* dO, void* ws, cudaStream_t s) {
  const Plan p = make_plan(n_local, r2, false);
  ScoreArgs a{};
  a.q = q; a.qp = qp ? qp : q; a.O = O;
  a.B = B; a.r2 = r2; a.n_begin = n_begin; a.n_local = n_local; a.n_total = n_total;
  a.off = tgt_off; a.idx = tgt_idx;
  a.t_neg = label_smoothing / (float)n_total;
  a.t_pos = CE ? 1.0f - label_smoothing : (1.0f - label_smoothing) + a.t_neg;
  a.inv_count = CE ? (float)(1.0 / (double)b_total) : (float)(1.0 / ((double)b_total * (double)n_total));
  a.p_target = stats;
  a.H_ws = (float*)ws;
  a.loss_partial = (double*)((char*)ws + rt::align_up((size_t)p.grid * B * r2 * sizeof(float), 256));
  a.dO = dO;
  a.n_tiles = p.n_tiles;
  if (int rc = dispatch<false, CE>(a, p, s)) return rc;
  const int64_t count = (int64_t)B * r2;
  reduce_H_kernel<<<(int)((count + 255) / 256), 256, 0, s>>>(a.H_ws, p.grid, count, H);
  RT_LAUNCH_CHECK();
  reduce_loss_kernel<<<1, 32, 0, s>>>(a.loss_partial, p.grid, loss_sum, 0);
  RT_LAUNCH_CHECK();
  return 0;
}

// ---- 1-N softmax cross-entropy, FFMA path: the log-sum-exp pass --------------------------------------------------
// Tile of 64 queries x 64 entities per CTA, the logits of score_dense_kernel.  Per query row and tile: m = the largest
// logit, s = sum exp(z - m) (online max: no fixed shift can keep every term of a trained query from underflowing),
// written to part[tile][b].
__device__ __forceinline__ void lse_merge(float& m, float& s, float m2, float s2) {
  if (m2 == -INFINITY) return;
  if (m == -INFINITY) { m = m2; s = s2; return; }
  const float mn = fmaxf(m, m2);
  s = s * rt::ex2_approx((m - mn) * rt::kLog2e) + s2 * rt::ex2_approx((m2 - mn) * rt::kLog2e);
  m = mn;
}

__global__ void __launch_bounds__(256)
score_lse_kernel(const float* __restrict__ q, const float* __restrict__ O, int B, int r2, int n_local,
                 float2* __restrict__ part) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const int n0 = blockIdx.x * NT, b0 = blockIdx.y * BT;
  const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;
  const LogitTile lt = stage_logit_tile(q, O, B, r2, n_local, n0, b0, smem_raw);
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int b = b0 + ty + 16 * i;
    float m = -INFINITY, s = 0.0f;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (n0 + tx + 16 * j < n_local) m = fmaxf(m, lt.z[i][j]);
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (n0 + tx + 16 * j < n_local) s += rt::ex2_approx((lt.z[i][j] - m) * rt::kLog2e);
    // the 16 lanes of this row: butterfly (merge is commutative, so every lane ends with the same bits)
#pragma unroll
    for (int o = 8; o > 0; o >>= 1) {
      const float m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
      lse_merge(m, s, m2, s2);
    }
    if (tx == 0 && b < B) part[(int64_t)blockIdx.x * B + b] = make_float2(m, s);
  }
}

// out[b] = (m, s) of query b merged over part[g][b], g < ngroups (row stride ld), in a fixed order: one warp per query,
// lane-strided groups, then a butterfly.  fp64 inside.  ngroups == 0 gives the empty part (-inf, 0).
__global__ void lse_combine_kernel(const float2* __restrict__ part, int ngroups, int64_t ld, int B,
                                   float* __restrict__ out) {
  const int b = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= B) return;
  double m = -INFINITY, s = 0.0;
  for (int g = lane; g < ngroups; g += 32) {
    const float2 p = __ldg(part + (int64_t)g * ld + b);
    if (p.x == -INFINITY) continue;
    const double pm = p.x;
    if (pm > m) { s = s * exp(m - pm) + (double)p.y; m = pm; }
    else s += (double)p.y * exp(pm - m);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const double m2 = __shfl_xor_sync(0xffffffffu, m, o), s2 = __shfl_xor_sync(0xffffffffu, s, o);
    if (m2 != -INFINITY) {
      if (m == -INFINITY) { m = m2; s = s2; }
      else { const double mn = fmax(m, m2); s = s * exp(m - mn) + s2 * exp(m2 - mn); m = mn; }
    }
  }
  if (lane == 0) { out[2 * b] = (float)m; out[2 * b + 1] = (float)s; }
}

// Row statistics of the whole batch from the shard parts [nparts][B][2] (fixed order over the parts):
// stats[b] = M_b (largest logit over all shards), stats[ld + b] = log2 S_b with S_b = sum_p s_p 2^((m_p - M_b) log2e),
// so that lse_b = M_b + ln 2 * log2 S_b.  Columns b in [B, ld) get (0, +inf): softmax 0.
__global__ void ce_row_stats_kernel(const float* __restrict__ parts, int nparts, int B, int ld, float* __restrict__ stats) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= ld) return;
  double M = -INFINITY, S = 0.0;
  if (b < B) {
    for (int p = 0; p < nparts; ++p) M = fmax(M, (double)parts[((int64_t)p * B + b) * 2]);
    if (M != -INFINITY)
      for (int p = 0; p < nparts; ++p) {
        const double m = parts[((int64_t)p * B + b) * 2], s = parts[((int64_t)p * B + b) * 2 + 1];
        if (m != -INFINITY) S += s * exp(m - M);
      }
  }
  const bool ok = S > 0.0;
  stats[b] = ok ? (float)M : 0.0f;
  stats[ld + b] = ok ? (float)log2(S) : INFINITY;
}

// loss_sum += sum over the queries WITHOUT targets of (1 - ls) lse_b: their loss is lse_b - (ls/N) sum_j z_bj and the
// elementwise pass charged the ls/N part.  One warp, fixed order.  Called for the shard that starts at entity 0.
__global__ void ce_empty_rows_kernel(const int32_t* __restrict__ off, int B, const float* __restrict__ stats, int ld,
                                     float one_minus_ls, double* __restrict__ loss_sum) {
  double v = 0.0;
  for (int b = threadIdx.x; b < B; b += 32)
    if (off[b + 1] == off[b] && stats[ld + b] < INFINITY)
      v += (double)one_minus_ls * ((double)stats[b] + (double)stats[ld + b] * 0.6931471805599453);
  v = rt::warp_sum(v);
  if (threadIdx.x == 0) loss_sum[0] += v;
}

}  // namespace

// variant 1: tcgen05 TF32 (score_bce_tc.cu); variant 2: warp-specialised fp16 tcgen05 (score_bce_v3.cu)
extern "C" size_t rt_score_bce_ws_bytes(int B, int n_local, int r2, int variant) {
  if (variant == 1) return rt::score_bce_tc_ws_bytes(B, n_local, r2);
  if (variant == 2) return rt_score_bce_v3_ws_bytes(B, n_local, r2);
  Plan p = make_plan(n_local, r2, false);
  return rt::align_up((size_t)p.grid * B * r2 * sizeof(float), 256) + (size_t)p.grid * sizeof(double);
}

extern "C" int rt_score_bce_fwd_bwd(const float* q, const float* qp, const float* O, int B, int r2,
                                    int n_begin, int n_local, int n_total, int b_total,
                                    const int32_t* tgt_off, const int32_t* tgt_idx,
                                    float label_smoothing, double* loss_sum, float* H, float* dO,
                                    int variant, void* ws, void* stream) {
  RT_REQUIRE(B > 0 && r2 > 0 && r2 <= 256 && n_local >= 0 && n_total > 0 && b_total > 0,
             "rt_score_bce_fwd_bwd: bad shape B=%d r2=%d n_local=%d", B, r2, n_local);
  RT_REQUIRE(ws != nullptr, "rt_score_bce_fwd_bwd: workspace is NULL");
  if (variant == 1)
    return rt::score_bce_tc(q, qp, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx,
                            label_smoothing, loss_sum, H, dO, ws, stream);
  if (variant == 2) {
    RT_REQUIRE(qp == nullptr || qp == q, "rt_score_bce_fwd_bwd: variant 2 computes dO = G^T q only (pass qp = NULL and "
               "fold the right factor into the following rt_apply)");
    return rt_score_bce_v3(q, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx, label_smoothing, 0.0f,
                           loss_sum, H, dO, nullptr, ws, stream);
  }
  RT_REQUIRE(variant == 0, "rt_score_bce_fwd_bwd: unknown variant %d", variant);
  return score_train_ffma<false>(q, qp, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx, label_smoothing,
                                 nullptr, loss_sum, H, dO, ws, (cudaStream_t)stream);
}

extern "C" int rt_target_prob(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                              const int32_t* target, float* p_target, void* stream) {
  RT_REQUIRE(B >= 0 && r2 > 0, "rt_target_prob: bad shape");
  if (B == 0) return 0;
  target_prob_kernel<<<rt::cdiv(B, 128), 128, 0, (cudaStream_t)stream>>>(q, O, B, r2, n_begin, n_local,
                                                                        target, p_target);
  RT_LAUNCH_CHECK();
  return 0;
}

__global__ void gated_reduce_loss_kernel(const double* __restrict__ partial, int n, double* __restrict__ out,
                                         const int* __restrict__ gate) {
  if (*gate == 0 || threadIdx.x != 0 || blockIdx.x != 0) return;
  double s = 0.0;
  for (int i = 0; i < n; ++i) s += partial[i];
  out[0] = s;
}

extern "C" size_t rt_score_rank_ws_bytes(int B, int n_local, int r2) {
  Plan p = make_plan(n_local, r2, true);
  size_t bytes = (size_t)p.grid * sizeof(double) + 256;
  if (rt::rank_tc_supported(B, n_local, r2)) bytes += rt::rank_tc_ws_bytes(B, n_local, r2);
  return bytes;
}

extern "C" int rt_score_rank_fused(const float* q, const float* O, int B, int r2, int n_begin,
                                   int n_local, const int32_t* target, const float* p_target,
                                   const int32_t* flt_off, const int32_t* flt_idx, int32_t* greater,
                                   int32_t* equal, int32_t* equal_before, double* bce_sum, void* ws,
                                   void* stream) {
  RT_REQUIRE(B > 0 && r2 > 0 && r2 <= 256 && n_local >= 0, "rt_score_rank_fused: bad shape");
  RT_REQUIRE(ws != nullptr, "rt_score_rank_fused: workspace is NULL");
  cudaStream_t s = (cudaStream_t)stream;
  RT_CHECK_CUDA(cudaMemsetAsync(greater, 0, sizeof(int32_t) * B, s));
  RT_CHECK_CUDA(cudaMemsetAsync(equal, 0, sizeof(int32_t) * B, s));
  RT_CHECK_CUDA(cudaMemsetAsync(equal_before, 0, sizeof(int32_t) * B, s));
  Plan p = make_plan(n_local, r2, true);
  // wide ranks, long shards: logits on the tensor cores (3xTF32), exact fp32 recomputation of the few entities whose
  // probability could tie with or cross the target's (apply_tc.cu, rank mode); the fp32 kernel below then only
  // runs -- gated on a device flag, no host synchronisation -- when that candidate list overflowed
  const int* gate = nullptr;
  if (rt::rank_tc_supported(B, n_local, r2)) {
    char* tc_ws = (char*)ws + rt::align_up((size_t)p.grid * sizeof(double) + 256, 256);
    int rc = rt::rank_tc(q, O, B, r2, n_begin, n_local, target, p_target, flt_off, flt_idx, greater, equal,
                         equal_before, bce_sum, tc_ws, s, &gate);
    if (rc) return rc;
  }
  ScoreArgs a{};
  a.q = q; a.qp = q; a.O = O;
  a.B = B; a.r2 = r2; a.n_begin = n_begin; a.n_local = n_local; a.n_total = n_local;
  a.off = flt_off; a.idx = flt_idx;
  a.t_pos = 1.0f; a.t_neg = 0.0f; a.inv_count = 1.0f;
  a.loss_partial = (double*)ws;
  a.target = target; a.p_target = p_target;
  a.greater = greater; a.equal = equal; a.equal_before = equal_before;
  a.n_tiles = p.n_tiles;
  a.gate = gate;
  int rc = dispatch<true>(a, p, s);
  if (rc) return rc;
  if (bce_sum) {
    if (gate) gated_reduce_loss_kernel<<<1, 32, 0, s>>>(a.loss_partial, p.grid, bce_sum, gate);
    else reduce_loss_kernel<<<1, 32, 0, s>>>(a.loss_partial, p.grid, bce_sum, 0);
    RT_LAUNCH_CHECK();
  }
  return 0;
}

namespace rt {
int score_dense(const float* q, const float* O, int B, int r2, int n_local, float* P, int64_t ldp, const int* gate,
                cudaStream_t s, bool logits) {
  if (B == 0 || n_local == 0) return 0;
  const size_t smem = logit_tile_smem(r2);
  dim3 grid(rt::cdiv(n_local, NT), rt::cdiv(B, BT));
  if (logits) {
    RT_CHECK_CUDA(cudaFuncSetAttribute(score_dense_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    score_dense_kernel<true><<<grid, 256, smem, s>>>(q, O, B, r2, n_local, P, ldp, gate);
  } else {
    RT_CHECK_CUDA(cudaFuncSetAttribute(score_dense_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)smem));
    score_dense_kernel<false><<<grid, 256, smem, s>>>(q, O, B, r2, n_local, P, ldp, gate);
  }
  RT_LAUNCH_CHECK();
  return 0;
}
}  // namespace rt

extern "C" int rt_score_dense(const float* q, const float* O, int B, int r2, int n_local, float* P,
                              int64_t ldp, void* stream) {
  RT_REQUIRE(B >= 0 && r2 > 0 && r2 <= 1024 && n_local >= 0 && ldp >= n_local, "rt_score_dense: bad shape");
  return rt::score_dense(q, O, B, r2, n_local, P, ldp, nullptr, (cudaStream_t)stream, false);
}

extern "C" int rt_score_dense_logits(const float* q, const float* O, int B, int r2, int n_local, float* Z, int64_t ldz,
                                     void* stream) {
  RT_REQUIRE(B >= 0 && r2 > 0 && r2 <= 1024 && n_local >= 0 && ldz >= n_local, "rt_score_dense_logits: bad shape");
  return rt::score_dense(q, O, B, r2, n_local, Z, ldz, nullptr, (cudaStream_t)stream, true);
}

// ---- 1-N softmax cross-entropy (rtucker.h: rt_score_lse / rt_score_ce_fwd_bwd) ------------------------------------
// Variant 3 lives in apply_tc.cu (log-sum-exp and CE epilogue modes of apply_tc_kernel); variant 0 is the FFMA path:
// score_lse_kernel + lse_combine_kernel, then ce_row_stats_kernel + score_kernel<., false, true>.
namespace rt {
int lse_combine(const float2* part, int ngroups, int64_t ld, int B, float* out, cudaStream_t s) {
  lse_combine_kernel<<<rt::cdiv(B, 8), 256, 0, s>>>(part, ngroups, ld, B, out);
  RT_LAUNCH_CHECK();
  return 0;
}
int ce_row_stats(const float* parts, int nparts, int B, int ld, float* stats, cudaStream_t s) {
  ce_row_stats_kernel<<<rt::cdiv(ld, 256), 256, 0, s>>>(parts, nparts, B, ld, stats);
  RT_LAUNCH_CHECK();
  return 0;
}
}  // namespace rt

static int ce_check_variant(const char* fn, int variant, int B, int n_local, int r2) {
  RT_REQUIRE(variant == 0 || variant == 3, "%s: variant %d has no cross-entropy path (0 = FFMA, 3 = tensor cores)", fn,
             variant);
  RT_REQUIRE(variant == 0 || rt_score_bce_tc3_supported(B, n_local, r2),
             "%s: variant 3 needs r2 >= 64, n_local >= 1024 and B <= 1024 (got B=%d n_local=%d r2=%d); use variant 0", fn,
             B, n_local, r2);
  return 0;
}

extern "C" size_t rt_score_lse_ws_bytes(int B, int n_local, int r2, int variant) {
  if (variant == 3) return rt::score_lse_tc3_ws_bytes(B, n_local, r2);
  return (size_t)rt::cdiv(n_local, NT) * (size_t)B * sizeof(float2) + 256;
}

extern "C" int rt_score_lse(const float* q, const float* O, int B, int r2, int n_local, int variant, float* parts,
                            void* ws, void* stream) {
  RT_REQUIRE(B > 0 && r2 > 0 && r2 <= 256 && n_local >= 0, "rt_score_lse: bad shape B=%d r2=%d n_local=%d", B, r2,
             n_local);
  RT_REQUIRE(ws != nullptr && parts != nullptr, "rt_score_lse: workspace or parts is NULL");
  if (int rc = ce_check_variant("rt_score_lse", variant, B, n_local, r2)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (variant == 3) return rt::score_lse_tc3(q, O, B, r2, n_local, parts, ws, s);
  const int n_tiles = rt::cdiv(n_local, NT);
  float2* part = (float2*)ws;
  if (n_tiles > 0) {
    const size_t smem = logit_tile_smem(r2);
    RT_CHECK_CUDA(rt::ensure_dyn_smem((const void*)score_lse_kernel, smem));
    score_lse_kernel<<<dim3(n_tiles, rt::cdiv(B, BT)), 256, smem, s>>>(q, O, B, r2, n_local, part);
    RT_LAUNCH_CHECK();
  }
  return rt::lse_combine(part, n_tiles, B, B, parts, s);
}

extern "C" size_t rt_score_ce_ws_bytes(int B, int n_local, int r2, int variant) {
  if (variant == 3) return rt::score_ce_tc3_ws_bytes(B, n_local, r2);
  return rt::align_up(rt_score_bce_ws_bytes(B, n_local, r2, 0), 256) + 2 * (size_t)B * sizeof(float);
}

extern "C" int rt_score_ce_fwd_bwd(const float* q, const float* qp, const float* O, int B, int r2, int n_begin,
                                   int n_local, int n_total, int b_total, const int32_t* tgt_off, const int32_t* tgt_idx,
                                   float label_smoothing, const float* parts, int nparts, double* loss_sum, float* H,
                                   float* dO, int variant, void* ws, void* stream) {
  RT_REQUIRE(B > 0 && r2 > 0 && r2 <= 256 && n_local >= 0 && n_total > 0 && b_total > 0,
             "rt_score_ce_fwd_bwd: bad shape B=%d r2=%d n_local=%d", B, r2, n_local);
  RT_REQUIRE(nparts >= 1, "rt_score_ce_fwd_bwd: nparts must be >= 1 (got %d)", nparts);
  RT_REQUIRE(ws != nullptr && parts != nullptr, "rt_score_ce_fwd_bwd: workspace or parts is NULL");
  if (int rc = ce_check_variant("rt_score_ce_fwd_bwd", variant, B, n_local, r2)) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (variant == 3)
    return rt::score_ce_tc3(q, qp, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx, label_smoothing,
                            parts, nparts, loss_sum, H, dO, ws, s);
  const size_t bce_bytes = rt::align_up(rt_score_bce_ws_bytes(B, n_local, r2, 0), 256);
  float* stats = (float*)((char*)ws + bce_bytes);
  if (int rc = rt::ce_row_stats(parts, nparts, B, B, stats, s)) return rc;
  if (int rc = score_train_ffma<true>(q, qp, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx,
                                      label_smoothing, stats, loss_sum, H, dO, ws, s))
    return rc;
  if (n_begin == 0) {
    ce_empty_rows_kernel<<<1, 32, 0, s>>>(tgt_off, B, stats, B, 1.0f - label_smoothing, loss_sum);
    RT_LAUNCH_CHECK();
  }
  return 0;
}
