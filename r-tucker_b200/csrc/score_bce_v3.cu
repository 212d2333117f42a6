// (b) Warp-specialised tcgen05 / TMEM kernel for the fused 1-N score + sigmoid + label-smoothed BCE + backward.
//
// Reference semantics: src/model/asymmetric/R_TuckER.py:47-48 (scores), nn.BCELoss at train.py:79,136 on the
// multi-hot targets of src/data/Dataset.py:43-52, and their backward w.r.t. the query rows and the entity factor:
//      Z[b,n]  = sum_k Q[b,k] O[n,k]          p = sigmoid(Z),  G = dBCE/dZ = (p - t) / (B N)
//      H[b,c]  = sum_n G[b,n] O[n,c]          (gradient w.r.t. the query rows)
//      dO[n,c] = sum_b G[b,n] Q[b,c]          (Euclidean gradient w.r.t. the entity factor)
// The B x N logit / probability / target matrices never exist in HBM.
//
// Design (one persistent CTA per SM, 14 warps):
//   warp 0     TMA producer: bulk copies of pre-packed fp16 operand images (O tile ring x2, Q chunk ring x2)
//   warp 1     MMA issuer: tcgen05.mma kind::f16, fp32 accumulation in tensor memory
//                 GEMM1  Z  = Q  O^T    (A, B K-major)             -> TMEM Z   [128 x TN]
//                 GEMM2  D2 = G  O      (A K-major, B MN-major)    -> TMEM D2  [128 x r2p]   per (tile, chunk)
//                 GEMM3  D3 += G^T Q    (A, B MN-major)            -> TMEM D3  [TN  x r2p]   accumulates over the chunks
//              GEMM1 of pair p+1 is issued before GEMM2/3 of pair p, so the tensor pipe works while the
//              epilogue warps turn Z(p) into G(p).
//   warps 2-9  epilogue: Z -> registers (Z is released at once), sigmoid / BCE / gradient in fp32 with the
//              reference's saturation semantics, G -> shared memory as fp16 in the interleaved core-matrix
//              format that is simultaneously a K-major operand (GEMM2) and an MN-major operand (GEMM3)
//   warps 10-13 flush: D2 -> per-CTA H partial straight from registers (st.global on the first visit of a chunk,
//              red.global.add.v4.f32 afterwards; a staging + cp.reduce.async.bulk variant measured slower),
//              D3 -> dO rows once per tile (32-byte stores)
//   Query chunks are visited in boustrophedon order over the tiles, so the chunk at a tile boundary repeats: its Q
//   image stays in shared memory and its H accumulator stays in TMEM (one flush and one reload less per tile).
// Operands are fp16 scaled by powers of two (exact) chosen from the arrays' absolute maxima: 11 significant
// bits like TF32 at twice the tensor rate and half the shared-memory footprint.  Stated tolerance: 2e-3 (same as
// the TF32 kernel of score_bce_tc.cu); the fp32-FFMA kernel of score_bce.cu is the 1e-5 path.
//
// Work per launch 6*B*N*r2 flop; algorithmic bytes 8*N*r2.
#include "common.h"
#include "tc.cuh"
#include <cuda_fp16.h>
#include <math.h>

namespace {
using namespace rt::tc;

constexpr int TB = 128;                 // queries per chunk
constexpr int kEpiWarps = 8, kFlushWarps = 4;
constexpr int kWarps = 2 + kEpiWarps + kFlushWarps;
constexpr int kThreads = kWarps * 32;   // 448
constexpr int kMaxCachedChunks = 4;     // query chunks whose target lists an epilogue thread keeps in registers
constexpr uint32_t QCS = TB * 16;       // byte stride between 8-column blocks of a Q chunk image (and of G)
constexpr float G_SCALE = 1024.0f;      // G is stored as (p - t) * 2^10 in fp16; 1/(B N) is applied at the flush
constexpr int R2P_MAX = 208;

struct V3Args {
  const unsigned char* Opk;   // [n_tiles][OB]   fp16 image of O rows of the tile, scaled by scal[1]
  const unsigned char* Qpk;   // [n_chunks][QB]  fp16 image of the query chunk, scaled by scal[0]
  const float* scal;          // [0] = sQ, [1] = sO (powers of two)
  int B, r2, r2p, n_begin, n_local, n_tiles, n_chunks;
  const int32_t* off; const int32_t* idx;
  float t_pos, t_neg, inv_count;
  float* H_ws;                // [grid][n_chunks][r2p * 128] partial H in flush layout
  double* loss_partial;       // [grid]
  double* gsum_partial;       // [grid] sum of (p - t) over the valid elements (next launch's centre)
  const float* cq;            // [r2p] centre * inv_count * sum_b q[b, :]: what the centring removed from every dO row
  float* dO;                  // [n_local][r2]
  uint32_t OB, QB;
  long long* prof;            // optional [grid][4 roles][10] cycle counters (debug, rt_score_v3_set_profile)
};

template <bool ENABLED>
struct ProfT {
  long long t0, acc[10];
  bool on;
  __device__ __forceinline__ void start(bool o) {
    on = o;
#pragma unroll
    for (int i = 0; i < 10; ++i) acc[i] = 0;
    if (on) t0 = clock64();
  }
  __device__ __forceinline__ void lap(int i) {
    if (on) { const long long t = clock64(); acc[i] += t - t0; t0 = t; }
  }
  __device__ __forceinline__ void dump(long long* dst) {
    if (on) {
#pragma unroll
      for (int i = 0; i < 10; ++i) dst[i] = acc[i];
    }
  }
};
template <>
struct ProfT<false> {
  static constexpr bool on = false;
  __device__ __forceinline__ void start(bool) {}
  __device__ __forceinline__ void lap(int) {}
  __device__ __forceinline__ void dump(long long*) {}
};

__device__ __forceinline__ void bulk_g2s_split(unsigned char* dst, const unsigned char* src, uint32_t bytes, uint64_t* bar) {
  for (uint32_t o = 0; o < bytes; o += 32768u) bulk_g2s(dst + o, src + o, min(32768u, bytes - o), bar);
}
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float lg2_approx(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ void red_add_v4(float* p, float x, float y, float z, float w) {
  asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};\n" :: "l"(p), "f"(x), "f"(y), "f"(z), "f"(w) : "memory");
}
__device__ __forceinline__ void st_v8(float* p, float a, float b, float c, float d, float e, float f, float g, float h) {
  asm volatile("st.global.v8.f32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};\n"
               :: "l"(p), "f"(a), "f"(b), "f"(c), "f"(d), "f"(e), "f"(f), "f"(g), "f"(h) : "memory");
}
__device__ __forceinline__ uint32_t pack_half2(float lo, float hi) {
  const __half2 h = __floats2half2_rn(lo, hi);
  return *reinterpret_cast<const uint32_t*>(&h);
}
template <int TN>
struct Cfg {
  static constexpr int CH = TN / 2;                       // entity columns per epilogue warp
  static constexpr int D3_COL = 0;
  static constexpr int D2_COL = (TN == 96) ? 208 : 176;   // r2p <= D2_COL
  static constexpr int Z_COL = 2 * D2_COL;
  static constexpr uint32_t OCS = TN * 16;                // byte stride between 8-column blocks of an O tile image
  static constexpr uint32_t GB = (TN / 8) * QCS;          // G bytes
  static_assert(Z_COL + TN <= 512, "TMEM budget");
};

template <int TN, bool PROF>
__global__ void __launch_bounds__(kThreads, 1)
score_v3_kernel(V3Args a) {
  using C = Cfg<TN>;
  using Prof = ProfT<PROF>;
  constexpr int CH = C::CH;
  extern __shared__ __align__(1024) unsigned char smem[];
  __shared__ uint64_t ofull[2], oempty[2], qfull[2], qempty[2], zfull, zfree, gfull, gfree, d2full, d2free, d3full, d3free;
  __shared__ uint32_t tmem_slot;
  __shared__ double red[kEpiWarps], redg[kEpiWarps];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  unsigned char* sO[2] = {smem, smem + a.OB};
  unsigned char* sQ[2] = {smem + 2 * a.OB, smem + 2 * a.OB + a.QB};
  unsigned char* sG = smem + 2 * a.OB + 2 * a.QB;

  if (tid == 0) {
    for (int s = 0; s < 2; ++s) { mbar_init(&ofull[s], 1); mbar_init(&oempty[s], 1); mbar_init(&qfull[s], 1); mbar_init(&qempty[s], 1); }
    mbar_init(&zfull, 1); mbar_init(&zfree, kEpiWarps);
    mbar_init(&gfull, kEpiWarps); mbar_init(&gfree, 1);
    mbar_init(&d2full, 1); mbar_init(&d2free, kFlushWarps);
    mbar_init(&d3full, 1); mbar_init(&d3free, kFlushWarps);
    fence_mbar_init();
  }
  if (warp == 1) tmem_alloc<512>(&tmem_slot);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_slot;
  const int r2p = a.r2p, n_chunks = a.n_chunks;
  const int first_tile = blockIdx.x, tile_step = gridDim.x;

  if (warp == 0) {
    // ============================== TMA producer ==============================
    if (lane == 0) {
      Prof pf; pf.start(a.prof != nullptr);
      auto load_O = [&](int lt, int tile) {
        const int s = lt & 1;
        pf.lap(2);
        if (lt >= 2) mbar_wait(&oempty[s], ((lt >> 1) + 1) & 1);
        pf.lap(0);
        mbar_expect_tx(&ofull[s], a.OB);
        bulk_g2s_split(sO[s], a.Opk + (size_t)tile * a.OB, a.OB, &ofull[s]);
      };
      if (first_tile < a.n_tiles) load_O(0, first_tile);
      int lt = 0, rho = -1;
      for (int tile = first_tile; tile < a.n_tiles; tile += tile_step, ++lt) {
        for (int i = 0; i < n_chunks; ++i) {
          const int c = (lt & 1) ? n_chunks - 1 - i : i;     // boustrophedon: the chunk at a tile boundary repeats
          if (i > 0 || lt == 0) {                             // a new run of pairs sharing one query chunk
            ++rho;
            const int s = rho & 1;
            pf.lap(2);
            if (rho >= 2) mbar_wait(&qempty[s], ((rho >> 1) + 1) & 1);
            pf.lap(1);
            mbar_expect_tx(&qfull[s], a.QB);
            bulk_g2s_split(sQ[s], a.Qpk + (size_t)c * a.QB, a.QB, &qfull[s]);
          }
          if (i == 0 && tile + tile_step < a.n_tiles) load_O(lt + 1, tile + tile_step);
        }
      }
      pf.lap(2);
      if (PROF && a.prof) pf.dump(a.prof + ((size_t)blockIdx.x * 4 + 0) * 10);
    }
  } else if (warp == 1) {
    // ============================== MMA issuer ==============================
    if (lane == 0) {
      const uint32_t idesc1 = make_idesc_f16(TB, TN, false, false);
      const uint32_t idesc2 = make_idesc_f16(TB, r2p, false, true);
      const uint32_t idesc3 = make_idesc_f16(128, r2p, true, true);
      const uint32_t aG = smem_u32(sG);
      const int ks1 = r2p / 16;
      const uint64_t dQk0 = make_desc(smem_u32(sQ[0]), QCS, 128), dQk1 = make_desc(smem_u32(sQ[1]), QCS, 128);      // K-major
      const uint64_t dQm0 = make_desc(smem_u32(sQ[0]), 128, QCS), dQm1 = make_desc(smem_u32(sQ[1]), 128, QCS);      // MN-major
      const uint64_t dOk0 = make_desc(smem_u32(sO[0]), C::OCS, 128), dOk1 = make_desc(smem_u32(sO[1]), C::OCS, 128);
      const uint64_t dOm0 = make_desc(smem_u32(sO[0]), 128, C::OCS), dOm1 = make_desc(smem_u32(sO[1]), 128, C::OCS);
      const uint64_t dGk = make_desc(aG, QCS, 128), dGm = make_desc(aG, 128, QCS);
      Prof pf; pf.start(a.prof != nullptr);
      // GEMM2 + GEMM3 of pair pp = (tile lt, chunk c) whose operands sit in stages (os, qs)
      // GEMM3 + GEMM2 of pair pp = (tile lt, position i) whose operands sit in stages (os, qs); run = maximal
      // sequence of consecutive pairs with the same query chunk (D2 keeps accumulating inside a run)
      auto g23 = [&](int pp, int lt, int i, int os, int qs, int rho, bool new_run, bool end_run) {
        mbar_wait(&gfull, pp & 1);
        pf.lap(4);
        if (i == 0 && lt > 0) mbar_wait(&d3free, (lt - 1) & 1);
        pf.lap(7);
        fence_after_sync();
        // descriptors are built once per stage; a k-step only adds to the 14-bit address field (the uniform datapath
        // that feeds tcgen05.mma has a long latency per dependent operation: rebuilding descriptors per MMA made the
        // issue loop the bottleneck)
        const uint64_t dQm = qs ? dQm1 : dQm0, dOm = os ? dOm1 : dOm0;
#pragma unroll
        for (int ks = 0; ks < TB / 16; ++ks)        // D3[n, c] += sum_b G[b, n] Q[b, c]
          mma_f16(tmem + C::D3_COL, dGm + (uint64_t)(ks * 16), dQm + (uint64_t)(ks * 16), idesc3, (i | ks) != 0);
        if (end_run) mma_commit(&qempty[qs]);        // the Q stage is free as early as possible: its refill is the
        if (i == n_chunks - 1) mma_commit(&d3full);  // longest latency of the pipeline
        pf.lap(8);
        if (new_run && rho > 0) { mbar_wait(&d2free, (rho - 1) & 1); fence_after_sync(); }
        pf.lap(5);
#pragma unroll
        for (int ks = 0; ks < TN / 16; ++ks)        // D2[b, c] (+)= sum_n G[b, n] O[n, c]
          mma_f16(tmem + C::D2_COL, dGk + (uint64_t)(ks * (2 * QCS >> 4)), dOm + (uint64_t)(ks * 16), idesc2,
                  !new_run || ks != 0);
        if (end_run) mma_commit(&d2full);
        mma_commit(&gfree);
        if (i == n_chunks - 1) mma_commit(&oempty[os]);
        pf.lap(6);
      };
      int pair = 0, lt = 0, rho = -1;
      int pv = 0, pv_lt = 0, pv_i = 0, pv_os = 0, pv_qs = 0, pv_rho = 0;
      bool pv_new = false, pv_end = false;
      for (int tile = first_tile; tile < a.n_tiles; tile += tile_step, ++lt) {
        const int os = lt & 1;
        const bool last_tile = tile + tile_step >= a.n_tiles;
        mbar_wait(&ofull[os], (lt >> 1) & 1);
        pf.lap(0);
        for (int i = 0; i < n_chunks; ++i, ++pair) {
          const bool new_run = (i > 0 || lt == 0), end_run = (i < n_chunks - 1 || last_tile);
          if (new_run) { ++rho; mbar_wait(&qfull[rho & 1], (rho >> 1) & 1); }
          const int qs = rho & 1;
          pf.lap(1);
          if (pair > 0) mbar_wait(&zfree, (pair - 1) & 1);
          pf.lap(2);
          fence_after_sync();
          const uint64_t dQk = qs ? dQk1 : dQk0, dOk = os ? dOk1 : dOk0;
#pragma unroll
          for (int ks = 0; ks < R2P_MAX / 16; ++ks)  // Z[b, n] = sum_k Q[b, k] O[n, k]
            if (ks < ks1)
              mma_f16(tmem + C::Z_COL, dQk + (uint64_t)(ks * (2 * QCS >> 4)), dOk + (uint64_t)(ks * (2 * C::OCS >> 4)),
                      idesc1, ks != 0);
          mma_commit(&zfull);
          pf.lap(3);
          if (pv) g23(pair - 1, pv_lt, pv_i, pv_os, pv_qs, pv_rho, pv_new, pv_end);
          pv = 1; pv_lt = lt; pv_i = i; pv_os = os; pv_qs = qs; pv_rho = rho; pv_new = new_run; pv_end = end_run;
        }
      }
      if (pv) g23(pair - 1, pv_lt, pv_i, pv_os, pv_qs, pv_rho, pv_new, pv_end);
      if (PROF && a.prof) pf.dump(a.prof + ((size_t)blockIdx.x * 4 + 1) * 10);
    }
  } else if (warp < 2 + kEpiWarps) {
    // ============================== epilogue: Z -> loss, G ==============================
    const int quarter = warp & 3;                 // TMEM lanes [32 * quarter, +32) are the ones this warp may touch
    const int half = (warp - 2) >> 2;             // which half of the tile's entity columns
    const int r = quarter * 32 + lane;            // query row within the chunk
    const float sQ = a.scal[0], sO = a.scal[1];
    const float zs = 1.0f / (sQ * sO);            // Z = raw * zs (exact: powers of two)
    const float nk = -zs * 1.4426950408889634f;   // e^{-z} = 2^x, x = raw * nk
    // fast path window: y = x - 8 with |y| < 32, i.e. z in (-27.7, 16.6): p != 1 and p (1 - p) > 1e-12, so none of
    // the reference's saturation branches is taken (the generic path below handles everything else)
    // G is stored CENTRED: (p - t) - centre, centre = scal[2] = last launch's mean of p - t.  fp16 keeps 11 bits: at
    // the start of training every p is 0.5 +- 1e-4 and the information is in the deviations, which fp16 (spacing
    // 2.4e-4 at 0.5) would round away; the rank-one part  centre * (column sums of O, sum of the query rows)  is added
    // back exactly in fp32 (reduce_H_v3_kernel, the dO stores of the flush warps)
    const float centre = a.scal[2];
    const float gneg = -(a.t_neg + centre) * G_SCALE;
    float gsum = 0.0f;
    // target lists of this thread's rows (one per chunk) stay in registers: bounds + the first two entries
    int ce0[kMaxCachedChunks], ce1[kMaxCachedChunks], ci0[kMaxCachedChunks], ci1[kMaxCachedChunks];
#pragma unroll
    for (int c = 0; c < kMaxCachedChunks; ++c) {
      const int b = c * TB + r;
      ce0[c] = ce1[c] = 0; ci0[c] = ci1[c] = -1;
      if (c < n_chunks && b < a.B) {
        ce0[c] = a.off[b]; ce1[c] = a.off[b + 1];
        if (ce1[c] > ce0[c]) ci0[c] = a.idx[ce0[c]];
        if (ce1[c] > ce0[c] + 1) ci1[c] = a.idx[ce0[c] + 1];
      }
    }
    double loss_acc = 0.0, g_acc = 0.0;
    int pair = 0;
    Prof pf; pf.start(PROF && a.prof != nullptr && warp == 2 && lane == 0);
    int lt_e = 0;
    for (int tile = first_tile; tile < a.n_tiles; tile += tile_step, ++lt_e) {
      const int n0 = tile * TN;
      const int cols_valid = min(CH, a.n_local - n0 - half * CH);     // may be <= 0 on the last tile
      const int nbase = a.n_begin + n0 + half * CH;
#pragma unroll 1
      for (int i = 0; i < n_chunks; ++i, ++pair) {
        const int c = (lt_e & 1) ? n_chunks - 1 - i : i;
        const int b = c * TB + r;
        const bool row_ok = b < a.B;
        // sparse positives of (row, this warp's columns) as a bit mask
        unsigned long long mask = 0ull;
        {
          int e0 = 0, e1 = 0, i0 = -1, i1 = -1;
          if (c < kMaxCachedChunks) {
#pragma unroll
            for (int cc = 0; cc < kMaxCachedChunks; ++cc)
              if (cc == c) { e0 = ce0[cc]; e1 = ce1[cc]; i0 = ci0[cc]; i1 = ci1[cc]; }
          } else if (row_ok) {
            e0 = a.off[b]; e1 = a.off[b + 1];
            if (e1 > e0) i0 = a.idx[e0];
            if (e1 > e0 + 1) i1 = a.idx[e0 + 1];
          }
          unsigned o = (unsigned)(i0 - nbase);
          if (i0 >= 0 && o < (unsigned)CH) mask |= 1ull << o;
          o = (unsigned)(i1 - nbase);
          if (i1 >= 0 && o < (unsigned)CH) mask |= 1ull << o;
          for (int e = e0 + 2; e < e1; ++e) {        // long lists (hub queries): the rest comes from memory
            o = (unsigned)(a.idx[e] - nbase);
            if (o < (unsigned)CH) mask |= 1ull << o;
          }
        }
        pf.lap(0);
        mbar_wait(&zfull, pair & 1);
        __syncwarp();
        pf.lap(1);
        fence_after_sync();
        uint32_t v[CH];
        const uint32_t taddr = tmem + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(C::Z_COL + half * CH);
#pragma unroll
        for (int g = 0; g < CH / 16; ++g) tmem_ld16(taddr + 16 * g, *reinterpret_cast<uint32_t(*)[16]>(&v[16 * g]));
        tmem_ld_wait();
        fence_before_sync();
        __syncwarp();
        if (lane == 0) mbar_arrive(&zfree);        // Z may be overwritten by GEMM1 of the next pair
        pf.lap(2);
        uint32_t gp[CH / 2];
        float A1 = 0.0f, Y2 = 0.0f, Ls = 0.0f;
        int nfast = 0;
#pragma unroll
        for (int g = 0; g < CH / 16; ++g) {
          float y[16];
          float ym = 0.0f;
#pragma unroll
          for (int j = 0; j < 16; ++j) {
            y[j] = fmaf(__uint_as_float(v[16 * g + j]), nk, -8.0f);
            ym = fmaxf(ym, fabsf(y[j]));
          }
          const unsigned mg = (unsigned)(mask >> (16 * g)) & 0xffffu;
          const bool fast = row_ok && mg == 0u && ym < 32.0f && (16 * g + 16 <= cols_valid);
          if (fast) {
            nfast += 16;
            // sum of log2(1 + e^{-z}) as log2 of products of three (each factor < 2^40 + 1 inside the window): one
            // MUFU.LG2 per three logits instead of one each -- the epilogue is bound by the MUFU / MIO pipe
            float prod = 1.0f;
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              float gq[2];
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                const float s = fmaf(ex2_approx(y[j + u]), 256.0f, 1.0f);    // 1 + e^{-z}
                const float p = rcp_approx(s);
                gsum += p;
                prod *= s;
                if ((j + u) % 3 == 2 || j + u == 15) { A1 += lg2_approx(prod); prod = 1.0f; }
                Y2 += y[j + u];
                gq[u] = fmaf(p, G_SCALE, gneg);
              }
              gp[(16 * g + j) >> 1] = pack_half2(gq[0], gq[1]);
            }
          } else {
#pragma unroll
            for (int j = 0; j < 16; j += 2) {
              float gq[2];
#pragma unroll
              for (int u = 0; u < 2; ++u) {
                const int col = 16 * g + j + u;
                const float z = __uint_as_float(v[col]) * zs;
                const bool valid = row_ok && col < cols_valid;
                const bool pos = (mg >> (j + u)) & 1u;
                // p = sigmoid(z) in fp32 with the reference's saturation semantics (BCELoss on probabilities):
                // p == 1 -> log(1-p) clamps at -100 and the gradient vanishes; p tiny -> log p clamps at -100.
                const float e = __expf(-z);
                const float sden = 1.0f + e;
                const float p = __fdividef(1.0f, sden);
                const float lp = fmaxf(-__logf(sden), -100.0f);
                const float lq = (p == 1.0f) ? -100.0f : fmaxf(lp - z, -100.0f);
                const float t = pos ? a.t_pos : a.t_neg;
                const float pq = (1.0f - p) * p;
                float gv = p - t;
                if (pq < 1e-12f) gv *= pq * 1e12f;
                if (valid) { Ls -= t * lp + (1.0f - t) * lq; gsum += gv + a.t_neg; gv -= centre; } else gv = 0.0f;
                gq[u] = gv * G_SCALE;
              }
              gp[(16 * g + j) >> 1] = pack_half2(gq[0], gq[1]);
            }
          }
        }
        // loss of the fast groups: sum ln(1 + e^{-z}) + (1 - t_neg) z  with  z = -(y + 8) ln 2
        {
          const float zsum = -0.6931471805599453f * (Y2 + 8.0f * (float)nfast);
          loss_acc += (double)(0.6931471805599453f * A1 + (1.0f - a.t_neg) * zsum + Ls);
          g_acc += (double)gsum;
          gsum = 0.0f;
        }
        pf.lap(3);
        if (pair > 0) mbar_wait(&gfree, (pair - 1) & 1);     // GEMM2/3 of the previous pair no longer read G
        pf.lap(4);
        {
          unsigned char* gdst = sG + (uint32_t)((half * CH) >> 3) * QCS + (uint32_t)(r >> 3) * 128u + (uint32_t)(r & 7) * 16u;
#pragma unroll
          for (int k = 0; k < CH / 8; ++k)
            *reinterpret_cast<uint4*>(gdst + k * QCS) = make_uint4(gp[4 * k], gp[4 * k + 1], gp[4 * k + 2], gp[4 * k + 3]);
        }
        fence_async_smem();
        __syncwarp();
        if (lane == 0) mbar_arrive(&gfull);
        pf.lap(5);
      }
    }
    if (PROF && pf.on) pf.dump(a.prof + ((size_t)blockIdx.x * 4 + 2) * 10);
    const double wsum = rt::warp_sum(loss_acc);
    const double gws = rt::warp_sum(g_acc);
    if (lane == 0) { red[warp - 2] = wsum; redg[warp - 2] = gws; }
  } else {
    // ============================== flush: D2 -> H partial of this CTA, D3 -> dO ==============================
    // H partial: thread (row r) owns H_ws[cta][chunk][quad][r][0..3]; the first visit of a chunk stores, later ones add
    // with red.global.add.v4.f32 (same thread, same address, program order: deterministic).  TMEM loads of the
    // next 32 columns are in flight while the current ones are written.
    const int quarter = warp & 3;
    const int r = quarter * 32 + lane;
    const float sQ = a.scal[0], sO = a.scal[1];
    const float hscale = a.inv_count / (G_SCALE * sO);
    const float dscale = a.inv_count / (G_SCALE * sQ);
    const uint32_t lanebits = (uint32_t)(quarter * 32) << 16;
    const int np = (r2p + 31) / 32;               // 32-column pieces (the last one may hold 16 columns)
    const bool vec_ok = (a.r2 % 4 == 0);
    const bool vec8_ok = (a.r2 % 8 == 0) && ((reinterpret_cast<uintptr_t>(a.dO) & 31) == 0);
    int lt = 0, rho = -1;
    unsigned long long touched = 0ull;            // chunks whose H slice this CTA has already written once
    Prof pf; pf.start(PROF && a.prof != nullptr && warp == 2 + kEpiWarps && lane == 0);
    auto ld_piece = [&](uint32_t col0, int h, uint32_t (&v)[32]) {
      if (32 * h + 32 <= r2p) tmem_ld32(tmem + lanebits + col0 + 32u * h, v);
      else tmem_ld16(tmem + lanebits + col0 + 32u * h, *reinterpret_cast<uint32_t(*)[16]>(&v[0]));
    };
    for (int tile = first_tile; tile < a.n_tiles; tile += tile_step, ++lt) {
      const int n0 = tile * TN;
      const int n_valid = min(TN, a.n_local - n0);
      const bool last_tile = tile + tile_step >= a.n_tiles;
      for (int i = 0; i < n_chunks; ++i) {
        const int c = (lt & 1) ? n_chunks - 1 - i : i;
        if (i > 0 || lt == 0) ++rho;
        if (!(i < n_chunks - 1 || last_tile)) continue;      // the run continues into the next tile: D2 keeps accumulating
        const bool first_touch = !((touched >> c) & 1ull);
        touched |= 1ull << c;
        float* hrow = a.H_ws + ((size_t)blockIdx.x * n_chunks + c) * ((size_t)r2p * TB) + (size_t)r * 4;
        auto st_piece = [&](int h, const uint32_t (&v)[32]) {
          const int nq = (32 * h + 32 <= r2p) ? 8 : 4;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            if (j < nq) {
              // a warp instruction covers 32 rows x 16 B = 512 contiguous bytes: whole 32-byte sectors for the
              // L2 atomic units (a 32-byte-per-thread layout halves their throughput: measured)
              float* dst = hrow + (size_t)(8 * h + j) * (TB * 4);
              const float x0 = __uint_as_float(v[4 * j]) * hscale, x1 = __uint_as_float(v[4 * j + 1]) * hscale;
              const float x2 = __uint_as_float(v[4 * j + 2]) * hscale, x3 = __uint_as_float(v[4 * j + 3]) * hscale;
              if (first_touch) *reinterpret_cast<float4*>(dst) = make_float4(x0, x1, x2, x3);
              else red_add_v4(dst, x0, x1, x2, x3);
            }
          }
        };
        mbar_wait(&d2full, rho & 1);
        __syncwarp();
        pf.lap(0);
        fence_after_sync();
        uint32_t va[32], vb[32];
        ld_piece(C::D2_COL, 0, va);
        for (int h = 0; h < np; h += 2) {
          tmem_ld_wait();
          pf.lap(2);
          if (h + 1 < np) ld_piece(C::D2_COL, h + 1, vb);
          else { fence_before_sync(); __syncwarp(); if (lane == 0) mbar_arrive(&d2free); }
          st_piece(h, va);
          pf.lap(first_touch ? 3 : 1);
          if (h + 1 >= np) break;
          tmem_ld_wait();
          pf.lap(2);
          if (h + 2 < np) ld_piece(C::D2_COL, h + 2, va);
          else { fence_before_sync(); __syncwarp(); if (lane == 0) mbar_arrive(&d2free); }
          st_piece(h + 1, vb);
          pf.lap(first_touch ? 3 : 1);
        }
      }
      // ---- tile epilogue: D3 -> dO rows of this tile (transposed through shared memory: 128-byte row segments) ----
      mbar_wait(&d3full, lt & 1);
      __syncwarp();
      pf.lap(7);
      fence_after_sync();
      {
        // straight from registers: every memory instruction of these warps queues behind the epilogue's MUFU stream
        // (same MIO path), so the fewest, widest instructions win: 32-byte stores where the row pitch allows
        uint32_t v[32];
        ld_piece(C::D3_COL, 0, v);
        for (int h = 0; h < np; ++h) {
          const int ncol = min(min(32, r2p - 32 * h), a.r2 - 32 * h);
          tmem_ld_wait();
          pf.lap(9);
          if (r < n_valid) {
            float* drow = a.dO + (size_t)(n0 + r) * a.r2 + 32 * h;
            const float* cq = a.cq + 32 * h;           // the rank-one part removed by the centring (same for every row)
            auto val = [&](int j) { return fmaf(__uint_as_float(v[j]), dscale, __ldg(cq + j)); };
            if (vec8_ok) {
#pragma unroll
              for (int j = 0; j < 4; ++j)
                if (8 * j < ncol)
                  st_v8(drow + 8 * j, val(8 * j), val(8 * j + 1), val(8 * j + 2), val(8 * j + 3), val(8 * j + 4),
                        val(8 * j + 5), val(8 * j + 6), val(8 * j + 7));
            } else if (vec_ok) {
#pragma unroll
              for (int j = 0; j < 8; ++j)
                if (4 * j < ncol)
                  *reinterpret_cast<float4*>(drow + 4 * j) = make_float4(val(4 * j), val(4 * j + 1), val(4 * j + 2), val(4 * j + 3));
            } else {
#pragma unroll
              for (int j = 0; j < 32; ++j)
                if (j < ncol) drow[j] = val(j);
            }
          }
          if (h + 1 < np) ld_piece(C::D3_COL, h + 1, v);
          else { fence_before_sync(); __syncwarp(); if (lane == 0) mbar_arrive(&d3free); }
          pf.lap(8);
        }
      }
      pf.lap(8);
    }
    if (PROF && pf.on) pf.dump(a.prof + ((size_t)blockIdx.x * 4 + 3) * 10);
  }
  fence_before_sync();
  __syncthreads();
  if (tid == 0) {
    double s = 0.0, sg = 0.0;
    for (int w = 0; w < kEpiWarps; ++w) { s += red[w]; sg += redg[w]; }
    a.loss_partial[blockIdx.x] = s;
    a.gsum_partial[blockIdx.x] = sg;
  }
  if (warp == 1) tmem_dealloc<512>(tmem);
}

// ---- operand scaling: absolute maxima -> power-of-two scales that map them into [2^12, 2^13) ----
__global__ void absmax_kernel(const float* __restrict__ x, size_t n, unsigned* __restrict__ out) {
  float m = 0.0f;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    m = fmaxf(m, fabsf(x[i]));
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.0f) atomicMax(out, __float_as_uint(m));   // non-negative floats order like uints
}
__device__ __forceinline__ float scale_for(float amax) {
  if (!(amax > 0.0f) || !isfinite(amax)) return 1.0f;
  int e;
  frexpf(amax, &e);                    // amax = m 2^e, m in [0.5, 1)
  e = 13 - e;
  e = max(-100, min(100, e));
  return ldexpf(1.0f, e);
}
// Scale of q from its absolute maximum (every CTA measures it redundantly: q is a few hundred KB and L2 resident,
// so no second launch or atomic is needed), scale of O from the hint or from absbits[0] (absmax_kernel), then the
// fp16 images of the query chunks (CTA i packs the image elements i, i + gridDim, ...).
__global__ void __launch_bounds__(512)
prep_q_kernel(const float* __restrict__ q, int B, int r2, int ncb, int n_chunks, const unsigned* __restrict__ absbits,
              float o_hint, float* __restrict__ scal, unsigned char* __restrict__ Qpk, uint32_t QB,
              const float* __restrict__ centre_state, float inv_count, float* __restrict__ cq) {
  __shared__ float wmax[16];
  if (blockIdx.x == 0) {
    // centre of this launch (the mean of p - t the previous launch measured) and the rank-one term it removes from
    // every dO row: centre * inv_count * sum_b q[b, :]   (fixed summation order: deterministic)
    const float c = centre_state ? centre_state[1] : 0.0f;
    for (int col = threadIdx.x; col < 8 * ncb; col += 512) {
      float sacc = 0.0f;
      if (col < r2)
        for (int b = 0; b < B; ++b) sacc += __ldg(q + (size_t)b * r2 + col);
      cq[col] = c * inv_count * sacc;
    }
    if (threadIdx.x == 0) scal[2] = c;
  }
  __shared__ float s_scale;
  float m = 0.0f;
  const size_t n = (size_t)B * r2;
  if ((n & 3) == 0 && (reinterpret_cast<uintptr_t>(q) & 15) == 0) {
    const float4* q4 = reinterpret_cast<const float4*>(q);
    const size_t n4 = n >> 2;
#pragma unroll 8
    for (size_t i = threadIdx.x; i < n4; i += 512) {
      const float4 v = __ldg(q4 + i);
      m = fmaxf(fmaxf(m, fmaxf(fabsf(v.x), fabsf(v.y))), fmaxf(fabsf(v.z), fabsf(v.w)));
    }
  } else {
#pragma unroll 8
    for (size_t i = threadIdx.x; i < n; i += 512) m = fmaxf(m, fabsf(__ldg(q + i)));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0) wmax[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x == 0) {
    float mm = 0.0f;
    for (int w = 0; w < 16; ++w) mm = fmaxf(mm, wmax[w]);
    s_scale = scale_for(mm);
    if (blockIdx.x == 0) {
      scal[0] = s_scale;
      scal[1] = scale_for(o_hint > 0.0f ? o_hint : __uint_as_float(absbits[0]));
    }
  }
  __syncthreads();
  const float sc = s_scale;
  const bool vec_ok = (r2 % 4 == 0);
  const int per = TB * ncb;
  for (int e = blockIdx.x * 512 + threadIdx.x; e < n_chunks * per; e += gridDim.x * 512) {
    const int chunk = e / per, w = e - chunk * per;
    const int row = w / ncb, cb = w - row * ncb;
    const int b = chunk * TB + row;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = 0.0f;
    if (b < B) {
      const float* p = q + (size_t)b * r2 + 8 * cb;
      if (vec_ok && 8 * cb + 8 <= r2) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(p)), y = __ldg(reinterpret_cast<const float4*>(p + 4));
        f[0] = x.x; f[1] = x.y; f[2] = x.z; f[3] = x.w; f[4] = y.x; f[5] = y.y; f[6] = y.z; f[7] = y.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (8 * cb + j < r2) f[j] = __ldg(p + j);
      }
    }
    uint4 o;
    o.x = pack_half2(f[0] * sc, f[1] * sc); o.y = pack_half2(f[2] * sc, f[3] * sc);
    o.z = pack_half2(f[4] * sc, f[5] * sc); o.w = pack_half2(f[6] * sc, f[7] * sc);
    *reinterpret_cast<uint4*>(Qpk + (size_t)chunk * QB + (uint32_t)cb * QCS + (uint32_t)(row >> 3) * 128u +
                              (uint32_t)(row & 7) * 16u) = o;
  }
}

// fp16 image of rows [blk*rows_per, +rows_per) of src[n_rows][r2]: element (row, col) at il16_offset(row, col, rows_per*16),
// ncb 8-column blocks, zero padded, scaled by scal[which]
__global__ void __launch_bounds__(256)
pack16_kernel(const float* __restrict__ src, int n_rows, int r2, int rows_per, int ncb, const float* __restrict__ scal,
              int which, unsigned char* __restrict__ dst, uint32_t img_bytes, float* __restrict__ tile_colsum) {
  const float s = scal[which];
  const int row0 = blockIdx.x * rows_per;
  if (tile_colsum) {                       // column sums of this tile's rows in row order (deterministic)
    for (int col = threadIdx.x; col < 8 * ncb; col += 256) {
      float acc = 0.0f;
      if (col < r2)
        for (int row = 0; row < rows_per && row0 + row < n_rows; ++row) acc += __ldg(src + (size_t)(row0 + row) * r2 + col);
      tile_colsum[(size_t)blockIdx.x * (8 * ncb) + col] = acc;
    }
  }
  unsigned char* img = dst + (size_t)blockIdx.x * img_bytes;
  const uint32_t CS = (uint32_t)rows_per * 16u;
  const bool vec_ok = (r2 % 4 == 0);
  for (int e = threadIdx.x; e < rows_per * ncb; e += 256) {
    const int row = e / ncb, cb = e - row * ncb;
    float f[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) f[j] = 0.0f;
    if (row0 + row < n_rows) {
      const float* p = src + (size_t)(row0 + row) * r2 + 8 * cb;
      if (vec_ok && 8 * cb + 8 <= r2) {
        const float4 x = __ldg(reinterpret_cast<const float4*>(p)), y = __ldg(reinterpret_cast<const float4*>(p + 4));
        f[0] = x.x; f[1] = x.y; f[2] = x.z; f[3] = x.w; f[4] = y.x; f[5] = y.y; f[6] = y.z; f[7] = y.w;
      } else {
#pragma unroll
        for (int j = 0; j < 8; ++j)
          if (8 * cb + j < r2) f[j] = __ldg(p + j);
      }
    }
    uint4 o;
    o.x = pack_half2(f[0] * s, f[1] * s); o.y = pack_half2(f[2] * s, f[3] * s);
    o.z = pack_half2(f[4] * s, f[5] * s); o.w = pack_half2(f[6] * s, f[7] * s);
    *reinterpret_cast<uint4*>(img + (uint32_t)cb * CS + (uint32_t)(row >> 3) * 128u + (uint32_t)(row & 7) * 16u) = o;
  }
}

// hc[col] = centre * inv_count * sum over the tiles of their column sums (fixed order)
__global__ void colsum_reduce_kernel(const float* __restrict__ tile_colsum, int n_tiles, int r2p, const float* __restrict__ scal,
                                     float inv_count, float* __restrict__ hc) {
  const int col = blockIdx.x * blockDim.x + threadIdx.x;
  if (col >= r2p) return;
  float acc = 0.0f;
  for (int t = 0; t < n_tiles; ++t) acc += tile_colsum[(size_t)t * r2p + col];
  hc[col] = scal[2] * inv_count * acc;
}

// H[b][c] = sum over the CTAs' partial slices, loss = sum of the CTAs' partial sums; both in a fixed order
// (deterministic).  Block = 32 positions (b, column quad) x 8 slices of the part index; block 0 also sums the loss.
__global__ void __launch_bounds__(256)
reduce_H_v3_kernel(const float* __restrict__ H_ws, int nparts, int n_chunks, int r2p, int B, int r2,
                   float* __restrict__ H, const double* __restrict__ loss_partial, double* __restrict__ loss_out,
                   const float* __restrict__ hc, const double* __restrict__ gsum_partial, double valid_count, float t_neg,
                   float* __restrict__ centre_state) {
  __shared__ float4 part[8][32];
  const int px = threadIdx.x & 31, ks = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + px;
  const int nq = r2p / 4;
  const bool in = i < n_chunks * nq * TB;
  const int bl = i % TB, q = (i / TB) % nq, c = i / (TB * nq);
  const size_t slice = (size_t)r2p * TB;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (in) {
    const float* p = H_ws + (size_t)c * slice + ((size_t)q * TB + bl) * 4;
#pragma unroll 4
    for (int k = ks; k < nparts; k += 8) {
      const float4 v = *reinterpret_cast<const float4*>(p + (size_t)k * n_chunks * slice);
      s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w;
    }
  }
  part[ks][px] = s;
  __syncthreads();
  if (ks == 0 && in) {
#pragma unroll
    for (int k = 1; k < 8; ++k) { const float4 v = part[k][px]; s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w; }
    const int b = c * TB + bl;
    if (b < B) {
      float* o = H + (size_t)b * r2 + 4 * q;              // + the rank-one part removed by the centring of G
      if (4 * q + 0 < r2) o[0] = s.x + hc[4 * q + 0];
      if (4 * q + 1 < r2) o[1] = s.y + hc[4 * q + 1];
      if (4 * q + 2 < r2) o[2] = s.z + hc[4 * q + 2];
      if (4 * q + 3 < r2) o[3] = s.w + hc[4 * q + 3];
    }
  }
  if (blockIdx.x == 0 && threadIdx.x < 32) {
    double t = 0.0, gs = 0.0;
    for (int k = threadIdx.x; k < nparts; k += 32) { t += loss_partial[k]; gs += gsum_partial[k]; }
    t = rt::warp_sum(t);            // xor-butterfly: the same association on every lane and every run
    gs = rt::warp_sum(gs);
    if (threadIdx.x == 0) {
      loss_out[0] = t;
      if (centre_state) centre_state[1] = (float)(gs / valid_count - (double)t_neg);   // mean of p - t: the next centre
    }
  }
}

long long* g_v3_prof = nullptr;

struct V3Layout {
  int TN, r2p, ncb, n_tiles, n_chunks, grid;
  uint32_t OB, QB, smem;
  size_t off_loss, off_gsum, off_cq, off_hc, off_tcs, off_scal, off_abs, off_Opk, off_Qpk, total;
};
V3Layout v3_layout(int B, int n_local, int r2) {
  V3Layout L;
  L.r2p = (r2 + 15) / 16 * 16;
  L.TN = (L.r2p <= 176) ? 128 : 96;
  L.ncb = L.r2p / 8;
  L.n_tiles = rt::cdiv(n_local, L.TN);
  L.n_chunks = rt::cdiv(B, TB);
  L.grid = L.n_tiles < rt::sm_count() ? L.n_tiles : rt::sm_count();
  if (L.grid < 1) L.grid = 1;
  L.OB = (uint32_t)L.ncb * L.TN * 16u;
  L.QB = (uint32_t)L.ncb * QCS;
  // G3 reads 16 n-blocks of G whatever TN is: keep 32 KB addressable behind sG
  const uint32_t tail = (uint32_t)(L.TN / 8) * QCS;
  L.smem = 2 * L.OB + 2 * L.QB + (tail < 16 * QCS ? 16 * QCS : tail);
  size_t o = rt::align_up((size_t)L.grid * L.n_chunks * L.r2p * TB * sizeof(float), 256);
  L.off_loss = o; o += rt::align_up((size_t)L.grid * sizeof(double), 256);
  L.off_gsum = o; o += rt::align_up((size_t)L.grid * sizeof(double), 256);
  L.off_cq = o; o += rt::align_up((size_t)L.r2p * sizeof(float), 256);
  L.off_hc = o; o += rt::align_up((size_t)L.r2p * sizeof(float), 256);
  L.off_tcs = o; o += rt::align_up((size_t)(L.n_tiles > 0 ? L.n_tiles : 1) * L.r2p * sizeof(float), 256);
  L.off_scal = o; o += 256;
  L.off_abs = o; o += 256;
  L.off_Opk = o; o += rt::align_up((size_t)(L.n_tiles > 0 ? L.n_tiles : 1) * L.OB, 256);
  L.off_Qpk = o; o += rt::align_up((size_t)L.n_chunks * L.QB, 256);
  L.total = o;
  return L;
}

}  // namespace

extern "C" int rt_score_bce_v3_supported(int r2) { return r2 >= 1 && r2 <= R2P_MAX; }

extern "C" size_t rt_score_bce_v3_ws_bytes(int B, int n_local, int r2) { return v3_layout(B, n_local, r2).total; }

extern "C" int rt_score_bce_v3(const float* q, const float* O, int B, int r2, int n_begin, int n_local, int n_total,
                               int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing,
                               float o_absmax_hint, double* loss_sum, float* H, float* dO, float* centre_state, void* ws,
                               void* stream) {
  return rt_score_bce_v3_phases(q, O, B, r2, n_begin, n_local, n_total, b_total, tgt_off, tgt_idx, label_smoothing,
                                o_absmax_hint, loss_sum, H, dO, centre_state, ws, stream, 7);
}

// phases: bit 0 = operand scaling + packing, bit 1 = the fused kernel, bit 2 = H / loss reduction.  Running a
// single phase needs a workspace already prepared by the earlier phases on the same inputs (bench.py times the
// fused kernel alone this way).
extern "C" int rt_score_bce_v3_phases(const float* q, const float* O, int B, int r2, int n_begin, int n_local,
                                      int n_total, int b_total, const int32_t* tgt_off, const int32_t* tgt_idx,
                                      float label_smoothing, float o_absmax_hint, double* loss_sum, float* H, float* dO,
                                      float* centre_state, void* ws, void* stream, int phases) {
  RT_REQUIRE(rt_score_bce_v3_supported(r2), "rt_score_bce_v3: r2=%d out of range (1..%d)", r2, R2P_MAX);
  RT_REQUIRE(B >= 1 && B <= 64 * TB && n_local >= 0, "rt_score_bce_v3: bad sizes B=%d (1..%d) n_local=%d", B, 64 * TB, n_local);
  cudaStream_t s = (cudaStream_t)stream;
  const V3Layout L = v3_layout(B, n_local, r2);
  char* base = (char*)ws;
  if (n_local == 0) {
    RT_CHECK_CUDA(cudaMemsetAsync(H, 0, (size_t)B * r2 * sizeof(float), s));
    RT_CHECK_CUDA(cudaMemsetAsync(loss_sum, 0, sizeof(double), s));
    return 0;
  }
  V3Args a{};
  a.Opk = (unsigned char*)(base + L.off_Opk);
  a.Qpk = (unsigned char*)(base + L.off_Qpk);
  a.scal = (float*)(base + L.off_scal);
  unsigned* absbits = (unsigned*)(base + L.off_abs);
  a.B = B; a.r2 = r2; a.r2p = L.r2p; a.n_begin = n_begin; a.n_local = n_local;
  a.n_tiles = L.n_tiles; a.n_chunks = L.n_chunks;
  a.off = tgt_off; a.idx = tgt_idx;
  a.t_neg = label_smoothing / (float)n_total;
  a.t_pos = (1.0f - label_smoothing) + a.t_neg;
  a.inv_count = (float)(1.0 / ((double)b_total * (double)n_total));
  a.H_ws = (float*)ws;
  a.loss_partial = (double*)(base + L.off_loss);
  a.gsum_partial = (double*)(base + L.off_gsum);
  a.cq = (const float*)(base + L.off_cq);
  float* hc = (float*)(base + L.off_hc);
  float* tile_colsum = (float*)(base + L.off_tcs);
  a.dO = dO;
  a.OB = L.OB; a.QB = L.QB;
  a.prof = g_v3_prof;

  if (phases & 1) {
  if (!(o_absmax_hint > 0.0f)) {
    RT_CHECK_CUDA(cudaMemsetAsync(absbits, 0, sizeof(unsigned), s));
    absmax_kernel<<<4 * rt::sm_count(), 256, 0, s>>>(O, (size_t)n_local * r2, absbits);
    RT_LAUNCH_CHECK();
  }
  prep_q_kernel<<<8 * L.n_chunks, 512, 0, s>>>(q, B, r2, L.ncb, L.n_chunks, absbits, o_absmax_hint, (float*)a.scal,
                                   (unsigned char*)a.Qpk, L.QB, centre_state, a.inv_count, (float*)a.cq);
  RT_LAUNCH_CHECK();
  pack16_kernel<<<L.n_tiles, 256, 0, s>>>(O, n_local, r2, L.TN, L.ncb, a.scal, 1, (unsigned char*)a.Opk, L.OB,
                                          centre_state ? tile_colsum : nullptr);
  RT_LAUNCH_CHECK();
  if (centre_state) {
    colsum_reduce_kernel<<<rt::cdiv(L.r2p, 128), 128, 0, s>>>(tile_colsum, L.n_tiles, L.r2p, a.scal, a.inv_count, hc);
    RT_LAUNCH_CHECK();
  } else {
    RT_CHECK_CUDA(cudaMemsetAsync(hc, 0, (size_t)L.r2p * sizeof(float), s));
  }
  }
  if (phases & 2) {
#define RT_V3_LAUNCH(TN_, PROF_)                                                                                   \
  do {                                                                                                            \
    RT_CHECK_CUDA(cudaFuncSetAttribute(score_v3_kernel<TN_, PROF_>, cudaFuncAttributeMaxDynamicSharedMemorySize, \
                                       (int)L.smem));                                                             \
    score_v3_kernel<TN_, PROF_><<<L.grid, kThreads, L.smem, s>>>(a);                                              \
  } while (0)
  if (L.TN == 96) { if (a.prof) RT_V3_LAUNCH(96, true); else RT_V3_LAUNCH(96, false); }
  else            { if (a.prof) RT_V3_LAUNCH(128, true); else RT_V3_LAUNCH(128, false); }
#undef RT_V3_LAUNCH
  RT_LAUNCH_CHECK();
  }
  if (phases & 4) {
  const int cnt = L.n_chunks * (L.r2p / 4) * TB;
  reduce_H_v3_kernel<<<(cnt + 31) / 32, 256, 0, s>>>(a.H_ws, L.grid, L.n_chunks, L.r2p, B, r2, H, a.loss_partial, loss_sum,
                                                     hc, a.gsum_partial, (double)B * (double)n_local, a.t_neg, centre_state);
  RT_LAUNCH_CHECK();
  }
  return 0;
}

// Debug: per-CTA, per-role cycle counters of score_v3_kernel ([grid][4][10] int64), NULL to disable.
extern "C" int rt_score_v3_set_profile(long long* dev_buf) { g_v3_prof = dev_buf; return 0; }
