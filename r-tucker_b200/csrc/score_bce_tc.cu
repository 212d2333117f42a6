// (b) tcgen05 / TMEM variant of the fused 1-N score + sigmoid + label-smoothed BCE + backward kernel.
//
// Same contract as the FFMA kernel in score_bce.cu (reference: src/model/asymmetric/R_TuckER.py:47-48,
// nn.BCELoss at train.py:79,136 on the targets of src/data/Dataset.py:43-52, and their backward), but the
// three B x N x r2 contractions run on the 5th-generation tensor cores in TF32 with fp32 accumulation
// in tensor memory:
//      GEMM1  Z[b,n]   = sum_k Q[b,k]  O[n,k]        D in TMEM cols [256,384)
//      GEMM2  H[b,c]  += sum_n G[b,n]  O[n,c]        D in TMEM cols [256,256+R2P)  (re-uses Z's columns)
//      GEMM3  dO[n,c] += sum_b G[b,n]  Q'[b,c]       D in TMEM cols [0,R2P), accumulates over the batch chunks
// TF32 tcgen05.mma only accepts K-major shared-memory operands (MN-major returns zeros: measured,
// tools/tc_probe2.py), so the operands whose contraction index is not their contiguous index are
// staged TRANSPOSED (O^T, G^T, Q'^T); all staging uses the interleaved core-matrix format of tc.cuh.
// Looser tolerance than the FFMA path: TF32 inputs (10-bit mantissa, round-to-nearest at staging).
//
// Work per launch 6*B*N*r2 flop; algorithmic bytes 8*N*r2.
#include "common.h"
#include "tc.cuh"
#include <math.h>

namespace {
using namespace rt::tc;

constexpr int TB = 128;            // queries per chunk   (MMA M of GEMM1/GEMM2, K of GEMM3)
constexpr int TN = 128;            // entities per tile   (MMA N of GEMM1, K of GEMM2, M of GEMM3)
constexpr int KB = 32;             // r2-columns per staged block (GEMM1 k-block, GEMM2/3 n-block)
constexpr int kThreads = 256;
constexpr uint32_t RS = 128;       // 8 rows x 16 B
constexpr uint32_t CS_G = TB * 16;            // G[b][n]:  column-chunk stride (conflict-free: 32 lanes = 32 rows)
constexpr uint32_t CS_GT = TN * 16 + 16;      // G^T[n][b]: padded so 4-byte transposed stores spread over banks
constexpr uint32_t CS_ROW = TB * 16 + 16;     // staged [128 rows][32 cols] blocks (Q, O), padded
constexpr uint32_t CS_T = KB * 16;            // staged transposed [32 rows][128 cols] blocks (O^T, Q'^T)
constexpr uint32_t G_BYTES = (TN / 4) * CS_G;          // 65536
constexpr uint32_t GT_BYTES = (TB / 4) * CS_GT;        // 66048
constexpr uint32_t HALF_BYTES = (KB / 4) * CS_ROW;     // 16512  (>= (TN/4)*CS_T = 16384)
constexpr uint32_t STAGE_BYTES = 2 * HALF_BYTES;       // 33024
constexpr uint32_t OFF_G = 0, OFF_GT = OFF_G + G_BYTES, OFF_STAGE = OFF_GT + GT_BYTES;
// GEMM1 phase: the whole Q chunk and O tile (all of K) are resident at once, over the G / G^T / stage
// areas that are idle then: [0, FULL) = Q, [FULL, 2*FULL) = O, FULL = 64 chunks * CS_ROW (r2 <= 256)
constexpr uint32_t FULL_BYTES = 50 * CS_ROW;             // r2 <= 200 on this path (103,200 B); wider ranks fall back
constexpr uint32_t OFF_MASK = (OFF_STAGE + 2 * STAGE_BYTES > 2 * FULL_BYTES) ? OFF_STAGE + 2 * STAGE_BYTES : 2 * FULL_BYTES;
constexpr uint32_t SMEM_BYTES = OFF_MASK + TB * 2 * 8;   // 208,448
constexpr int HB_LD = 132;                                // epilogue transpose buffer [128][132] floats (16-byte aligned rows) in the stage area
static_assert(OFF_STAGE + 128 * HB_LD * 4 <= OFF_MASK, "transpose buffer must fit between the stage area start and the masks");
constexpr uint32_t TM_D3 = 0, TM_Z = 256, TM_D2 = 256;

struct TcArgs {
  const float* q; const float* qp; const float* O;
  int B, r2, n_begin, n_local;
  const int32_t* off; const int32_t* idx;
  float t_pos, t_neg, inv_count;
  double* loss_partial; float* H_ws; float* dO;
  int n_tiles, r2p;
  long long* prof;   // optional [grid][12] cycle counters per phase (debug)
  // packed operand images (pre-rounded to TF32, already in the shared-memory layout), see pack_*_kernel
  const unsigned char* Opk1; const unsigned char* Qpk1;   // [tile | chunk][full_bytes]        K-major, all of K
  const unsigned char* Opk2; const unsigned char* Qpk2;   // [tile | chunk][ncb][TBLK_BYTES]   transposed blocks
  uint32_t full_bytes;
  int packed, ncb;
};

// [rows0, rows0+128) x [col0, col0+32) of src (row-major, ld) -> K-major block, zero padded.
// All global loads of a thread are issued before the first shared-memory store (latency paid once).
__device__ __forceinline__ void stage_rows(unsigned char* dst, const float* __restrict__ src, int ld, int row0,
                                           int rows_valid, int col0, int cols_valid, bool vec_ok) {
  constexpr int IT = TB * (KB / 4) / kThreads;   // 4
  float4 f[IT];
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int e = it * kThreads + threadIdx.x;
    const int row = e >> 3, ch = e & 7;
    const int gc = col0 + 4 * ch;
    f[it] = make_float4(0.f, 0.f, 0.f, 0.f);
    if (row < rows_valid) {
      const float* p = src + (int64_t)(row0 + row) * ld + gc;
      if (vec_ok && gc + 4 <= col0 + cols_valid) {
        f[it] = __ldg(reinterpret_cast<const float4*>(p));
      } else {
        if (gc + 0 < col0 + cols_valid) f[it].x = __ldg(p + 0);
        if (gc + 1 < col0 + cols_valid) f[it].y = __ldg(p + 1);
        if (gc + 2 < col0 + cols_valid) f[it].z = __ldg(p + 2);
        if (gc + 3 < col0 + cols_valid) f[it].w = __ldg(p + 3);
      }
    }
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int e = it * kThreads + threadIdx.x;
    const int row = e >> 3, ch = e & 7;
    *reinterpret_cast<uint4*>(dst + (uint32_t)ch * CS_ROW + (uint32_t)(row >> 3) * RS + (uint32_t)(row & 7) * 16u) =
        make_uint4(to_tf32(f[it].x), to_tf32(f[it].y), to_tf32(f[it].z), to_tf32(f[it].w));
  }
}

__device__ __forceinline__ void cp_async16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" :: "r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// Whole [128 rows][r2 cols] operand (all of K) -> K-major interleaved block: every 16-byte chunk is one
// cp.async (all in flight at once), then rounded to TF32 in place by the thread that copied it.
// Requires r2 % 4 == 0 (16-byte aligned rows).  Invalid rows are zero filled.
__device__ __forceinline__ void stage_full_async(unsigned char* dst, const float* __restrict__ src, int r2, int row0,
                                                 int rows_valid) {
  const int nch = r2 >> 2;
  const int nchp = nch + (nch & 1);       // an MMA k-step consumes two chunks: pad odd chunk counts with zeros
  const uint32_t d0 = smem_u32(dst);
  for (int e = threadIdx.x; e < TB * nchp; e += kThreads) {
    const int row = e / nchp, ch = e - row * nchp;
    const uint32_t off = (uint32_t)ch * CS_ROW + (uint32_t)(row >> 3) * RS + (uint32_t)(row & 7) * 16u;
    if (row < rows_valid && ch < nch) cp_async16(d0 + off, src + (int64_t)(row0 + row) * r2 + 4 * ch);
    else *reinterpret_cast<uint4*>(dst + off) = make_uint4(0u, 0u, 0u, 0u);
  }
}
__device__ __forceinline__ void round_full_inplace(unsigned char* dst, int r2, int rows_valid) {
  // same (row, chunk) -> thread mapping as stage_full_async: a thread only touches its own cp.async data
  const int nch = r2 >> 2;
  const int nchp = nch + (nch & 1);
  for (int e = threadIdx.x; e < TB * nchp; e += kThreads) {
    const int row = e / nchp, ch = e - row * nchp;
    if (row >= rows_valid || ch >= nch) continue;
    uint4* p = reinterpret_cast<uint4*>(dst + (uint32_t)ch * CS_ROW + (uint32_t)(row >> 3) * RS + (uint32_t)(row & 7) * 16u);
    uint4 v = *p;
    v.x = to_tf32(__uint_as_float(v.x)); v.y = to_tf32(__uint_as_float(v.y));
    v.z = to_tf32(__uint_as_float(v.z)); v.w = to_tf32(__uint_as_float(v.w));
    *p = v;
  }
}

// transposed: dst[c][r] for c in [col0, col0+32), r in [row0, row0+128): K-major along r
__device__ __forceinline__ void stage_cols_T(unsigned char* dst, const float* __restrict__ src, int ld, int row0,
                                             int rows_valid, int col0, int cols_valid) {
  constexpr int IT = KB * (TN / 4) / kThreads;   // 4
  float t[IT][4];
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int e = it * kThreads + threadIdx.x;
    const int c = e & 31, rch = e >> 5;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = 4 * rch + j;
      t[it][j] = (r < rows_valid && c < cols_valid) ? __ldg(src + (int64_t)(row0 + r) * ld + col0 + c) : 0.0f;
    }
  }
#pragma unroll
  for (int it = 0; it < IT; ++it) {
    const int e = it * kThreads + threadIdx.x;
    const int c = e & 31, rch = e >> 5;
    *reinterpret_cast<uint4*>(dst + (uint32_t)rch * CS_T + (uint32_t)c * 16u) =
        make_uint4(to_tf32(t[it][0]), to_tf32(t[it][1]), to_tf32(t[it][2]), to_tf32(t[it][3]));
  }
}

constexpr uint32_t TBLK_BYTES = (TN / 4) * CS_T;    // one transposed 32-column block image (16,384 B)

// ---- operand pre-packing (once per launch): global fp32 -> TF32-rounded shared-memory images ----
// K-major full-K image of rows [128*blk, +128) of src[n_rows][r2]
__global__ void __launch_bounds__(256)
pack_rows_kernel(const float* __restrict__ src, int n_rows, int r2, unsigned char* __restrict__ dst, uint32_t full_bytes) {
  const int row0 = blockIdx.x * TB;
  const int nch = r2 >> 2, nchp = nch + (nch & 1);
  unsigned char* img = dst + (size_t)blockIdx.x * full_bytes;
  for (int e = threadIdx.x; e < TB * nchp; e += 256) {
    const int row = e / nchp, ch = e - row * nchp;
    uint4 v = make_uint4(0u, 0u, 0u, 0u);
    if (row0 + row < n_rows && ch < nch) {
      const float4 f = __ldg(reinterpret_cast<const float4*>(src + (int64_t)(row0 + row) * r2 + 4 * ch));
      v = make_uint4(to_tf32(f.x), to_tf32(f.y), to_tf32(f.z), to_tf32(f.w));
    }
    *reinterpret_cast<uint4*>(img + (uint32_t)ch * CS_ROW + (uint32_t)(row >> 3) * RS + (uint32_t)(row & 7) * 16u) = v;
  }
}
// transposed 32-column block images: dst[blk][cb][c][r] = src[128*blk + r][32*cb + c]
__global__ void __launch_bounds__(256)
pack_cols_kernel(const float* __restrict__ src, int n_rows, int r2, int ncb, unsigned char* __restrict__ dst) {
  const int row0 = blockIdx.x * TN, cb = blockIdx.y;
  unsigned char* img = dst + ((size_t)blockIdx.x * ncb + cb) * TBLK_BYTES;
  for (int e = threadIdx.x; e < KB * (TN / 4); e += 256) {
    const int c = e & 31, rch = e >> 5;
    uint32_t t[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int r = row0 + 4 * rch + j, col = cb * KB + c;
      t[j] = (r < n_rows && col < r2) ? to_tf32(__ldg(src + (int64_t)r * r2 + col)) : 0u;
    }
    *reinterpret_cast<uint4*>(img + (uint32_t)rch * CS_T + (uint32_t)c * 16u) = make_uint4(t[0], t[1], t[2], t[3]);
  }
}

// ---- TMA bulk copy (global -> shared), completion counted in bytes on an mbarrier ----
__device__ __forceinline__ void bulk_g2s_split(unsigned char* dst, const unsigned char* src, uint32_t bytes, uint64_t* bar) {
  for (uint32_t o = 0; o < bytes; o += 32768u) bulk_g2s(dst + o, src + o, min(32768u, bytes - o), bar);
}

__global__ void __launch_bounds__(kThreads, 1)
score_tc_kernel(TcArgs a) {
  extern __shared__ __align__(128) unsigned char smem[];
  __shared__ uint64_t bar_stage[2], bar_z, bar_d, bar_ld, bar_full[2];
  __shared__ uint32_t tmem_slot;
  __shared__ double red[kThreads / 32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int quarter = warp & 3, half = warp >> 2;       // TMEM lane quarter / column half of this warp
  unsigned char* sG = smem + OFF_G;
  unsigned char* sGT = smem + OFF_GT;
  unsigned char* sStage[2] = {smem + OFF_STAGE, smem + OFF_STAGE + STAGE_BYTES};
  unsigned long long* mask = reinterpret_cast<unsigned long long*>(smem + OFF_MASK);   // [TB][2]
  float* hbuf = reinterpret_cast<float*>(smem + OFF_STAGE);

  if (tid == 0) {
    mbar_init(&bar_stage[0], 1); mbar_init(&bar_stage[1], 1); mbar_init(&bar_z, 1); mbar_init(&bar_d, 1);
    mbar_init(&bar_ld, 1); mbar_init(&bar_full[0], 1); mbar_init(&bar_full[1], 1);
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc<512>(&tmem_slot);
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = tmem_slot;

  const int r2 = a.r2, r2p = a.r2p;
  const bool vec_ok = (r2 % 4 == 0);
  const bool full_k = vec_ok && r2 <= 200;   // whole-K staging fits in the idle G / G^T / stage areas
  const int nkb = (r2 + KB - 1) / KB;          // GEMM1 k-blocks
  const int ncb = r2p / KB + ((r2p % KB) ? 1 : 0);   // GEMM2/3 column blocks (last one may be 16 wide)
  const int n_chunks = (a.B + TB - 1) / TB;
  const uint32_t idesc1 = make_idesc_tf32(TB, TN, false, false);
  uint32_t ph_stage[2] = {0u, 0u}, ph_z = 0u, ph_d = 0u, ph_ld = 0u, ph_full[2] = {0u, 0u};
  int used[2] = {0, 0};                          // number of un-waited commits per stage (0 or 1)
  double loss_acc = 0.0;
  bool first_tile = true;
  long long tp[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0}, tc0 = clock64(), tc1;
#define RT_TC_PROF(i) do { tc1 = clock64(); tp[i] += tc1 - tc0; tc0 = tc1; } while (0)

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int n0 = tile * TN;
    const int n_valid = min(TN, a.n_local - n0);
    for (int chunk = 0; chunk < n_chunks; ++chunk) {
      const int b0 = chunk * TB;
      const int b_valid = min(TB, a.B - b0);
      // ================= GEMM1: Z = Q O^T =================
      if (a.packed) {
        // both operands (all of K) arrive as two TMA bulk copies of ready-made images; one thread drives it
        unsigned char* sQ = smem;
        unsigned char* sO = smem + FULL_BYTES;
        if (tid == 0) {
          fence_async_smem();      // earlier generic-proxy accesses of this memory (G, G^T, hbuf) are ordered first
          mbar_expect_tx(&bar_ld, 2u * a.full_bytes);
          bulk_g2s_split(sQ, a.Qpk1 + (size_t)chunk * a.full_bytes, a.full_bytes, &bar_ld);
          bulk_g2s_split(sO, a.Opk1 + (size_t)tile * a.full_bytes, a.full_bytes, &bar_ld);
          mbar_wait(&bar_ld, ph_ld);
          fence_after_sync();
          const uint32_t aA = smem_u32(sQ), aB = smem_u32(sO);
          const int ksteps = (r2 + 7) / 8;
          for (int ks = 0; ks < ksteps; ++ks)
            mma_tf32(tmem + TM_Z, make_desc(aA + ks * 2 * CS_ROW, CS_ROW, RS), make_desc(aB + ks * 2 * CS_ROW, CS_ROW, RS),
                     idesc1, ks != 0);
          mma_commit(&bar_z);
        }
        ph_ld ^= 1u;
      } else if (full_k) {
        // whole K resident: one asynchronous staging wave, then all MMAs back to back
        unsigned char* sQ = smem;
        unsigned char* sO = smem + FULL_BYTES;
        stage_full_async(sQ, a.q, r2, b0, b_valid);
        stage_full_async(sO, a.O, r2, n0, n_valid);
        RT_TC_PROF(8);    // cp.async issue
        cp_async_wait_all();
        RT_TC_PROF(9);    // cp.async wait
        round_full_inplace(sQ, r2, b_valid);
        round_full_inplace(sO, r2, n_valid);
        fence_async_smem();
        RT_TC_PROF(10);   // in-place TF32 rounding
        __syncthreads();
        RT_TC_PROF(11);   // barrier
        if (tid == 0) {
          fence_after_sync();
          const uint32_t aA = smem_u32(sQ), aB = smem_u32(sO);
          const int ksteps = (r2 + 7) / 8;      // r2 % 8 == 4: the last step's second chunk is the zero pad
          for (int ks = 0; ks < ksteps; ++ks)
            mma_tf32(tmem + TM_Z, make_desc(aA + ks * 2 * CS_ROW, CS_ROW, RS), make_desc(aB + ks * 2 * CS_ROW, CS_ROW, RS),
                     idesc1, ks != 0);
          mma_commit(&bar_z);
        }
      } else {
      // k-blocked, 2-stage ring (any r2)
      for (int kb = 0; kb < nkb; ++kb) {
        const int s = kb & 1;
        if (used[s]) { mbar_wait(&bar_stage[s], ph_stage[s]); ph_stage[s] ^= 1u; used[s] = 0; }
        const int kw = min(KB, r2 - kb * KB);
        stage_rows(sStage[s], a.q, r2, b0, b_valid, kb * KB, kw, vec_ok);
        stage_rows(sStage[s] + HALF_BYTES, a.O, r2, n0, n_valid, kb * KB, kw, vec_ok);
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
          fence_after_sync();
          const uint32_t aA = smem_u32(sStage[s]), aB = aA + HALF_BYTES;
          const int ksteps = (kw + 7) / 8;
          for (int ks = 0; ks < ksteps; ++ks)
            mma_tf32(tmem + TM_Z, make_desc(aA + ks * 2 * CS_ROW, CS_ROW, RS), make_desc(aB + ks * 2 * CS_ROW, CS_ROW, RS),
                     idesc1, (kb | ks) != 0);
          mma_commit(&bar_stage[s]);
          if (kb == nkb - 1) mma_commit(&bar_z);
        }
        used[s] = 1;
      }
      }
      RT_TC_PROF(0);   // GEMM1 staging + issue
      // ---- sparse positives of this (chunk, tile) as 128-bit row masks ----
      mask[tid] = 0ull;                                   // kThreads == 2 * TB
      __syncthreads();
      {
        const int rr = tid >> 1, part = tid & 1;
        const int b = b0 + rr;
        if (b < a.B) {
          unsigned long long m0 = 0ull, m1 = 0ull;
          const int e1 = a.off[b + 1];
          for (int e = a.off[b] + part; e < e1; e += 2) {
            const int o = a.idx[e] - a.n_begin - n0;
            if (o >= 0 && o < 64) m0 |= 1ull << o;
            else if (o >= 64 && o < TN) m1 |= 1ull << (o - 64);
          }
          if (m0) atomicOr(&mask[rr * 2 + 0], m0);
          if (m1) atomicOr(&mask[rr * 2 + 1], m1);
        }
      }
      __syncthreads();
      // ================= epilogue 1: Z -> p, loss, G ; G and G^T staged as TF32 =================
      RT_TC_PROF(1);   // mask
      mbar_wait(&bar_z, ph_z); ph_z ^= 1u;
      fence_after_sync();
      RT_TC_PROF(2);   // wait for GEMM1
      {
        const int rr = quarter * 32 + lane;              // query row of this thread (TMEM lane)
        const int b = b0 + rr;
        const unsigned long long mrow = mask[rr * 2 + half];
        float loss_t = 0.0f;
#pragma unroll 1
        for (int cgp = 0; cgp < 2; ++cgp) {
          const int cbase = half * 64 + cgp * 32;          // entity column within the tile
          uint32_t v[32];
          tmem_ld32(tmem + TM_Z + ((uint32_t)(quarter * 32) << 16) + (uint32_t)cbase, v);
          tmem_ld_wait();
          // store bases: G^T[n][b] element (cc, rr) sits at gt_base + 16*cc; G[b][n] chunk at g_base + (cc/4)*CS_G
          unsigned char* gt_base = sGT + (uint32_t)(rr >> 2) * CS_GT + (uint32_t)(rr & 3) * 4u + (uint32_t)cbase * 16u;
          unsigned char* g_base = sG + (uint32_t)(cbase >> 2) * CS_G + (uint32_t)(rr >> 3) * RS + (uint32_t)(rr & 7) * 16u;
          const bool row_ok = (b < a.B);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            uint32_t gq[4];
#pragma unroll
            for (int jj = 0; jj < 4; ++jj) {
              const int j = j4 * 4 + jj;
              const bool valid = row_ok && (cbase + j < n_valid);
              const bool pos = (mrow >> (cgp * 32 + j)) & 1ull;
              const float z = __uint_as_float(v[j]);
              // p = sigmoid(z) in fp32 with the reference's saturation semantics (BCELoss on probabilities):
              // p == 1 -> log(1-p) clamps at -100 and the gradient vanishes; p tiny -> log p clamps at -100.
              const float e = __expf(-z);
              const float sden = 1.0f + e;
              const float p = __fdividef(1.0f, sden);
              const float lp = fmaxf(-__logf(sden), -100.0f);
              const float lq = (p == 1.0f) ? -100.0f : fmaxf(lp - z, -100.0f);
              const float t = pos ? a.t_pos : a.t_neg;
              const float pq = (1.0f - p) * p;
              float g = (p - t) * a.inv_count;
              if (pq < 1e-12f) g *= pq * 1e12f;
              if (valid) loss_t -= t * lp + (1.0f - t) * lq; else g = 0.0f;
              gq[jj] = to_tf32(g);
              *reinterpret_cast<uint32_t*>(gt_base + j * 16) = gq[jj];
            }
            *reinterpret_cast<uint4*>(g_base + j4 * CS_G) = make_uint4(gq[0], gq[1], gq[2], gq[3]);
          }
        }
        loss_acc += (double)loss_t;
      }
      fence_before_sync();
      fence_async_smem();
      __syncthreads();
      RT_TC_PROF(3);   // epilogue 1
      // ================= GEMM2 (H chunk) and GEMM3 (dO tile), column-blocked =================
      if (a.packed) {
        // one thread runs a 2-stage TMA ring over the transposed 32-column blocks of O^T and Q'^T
        if (tid == 0) {
          fence_after_sync();
          auto fill = [&](int cb) {
            const int s = cb & 1;
            mbar_expect_tx(&bar_full[s], 2u * TBLK_BYTES);
            bulk_g2s(sStage[s], a.Opk2 + ((size_t)tile * ncb + cb) * TBLK_BYTES, TBLK_BYTES, &bar_full[s]);
            bulk_g2s(sStage[s] + HALF_BYTES, a.Qpk2 + ((size_t)chunk * ncb + cb) * TBLK_BYTES, TBLK_BYTES, &bar_full[s]);
          };
          fence_async_smem();
          fill(0);
          if (ncb > 1) fill(1);
          const uint32_t aG = smem_u32(sG), aGT = smem_u32(sGT);
          for (int cb = 0; cb < ncb; ++cb) {
            const int s = cb & 1;
            mbar_wait(&bar_full[s], ph_full[s]); ph_full[s] ^= 1u;
            fence_after_sync();
            const int cw = min(KB, r2p - cb * KB);
            const uint32_t idn = make_idesc_tf32(128, cw, false, false);
            const uint32_t aOT = smem_u32(sStage[s]), aQT = aOT + HALF_BYTES;
            for (int ks = 0; ks < TN / 8; ++ks)
              mma_tf32(tmem + TM_D2 + cb * KB, make_desc(aG + ks * 2 * CS_G, CS_G, RS),
                       make_desc(aOT + ks * 2 * CS_T, CS_T, RS), idn, ks != 0);
            for (int ks = 0; ks < TB / 8; ++ks)
              mma_tf32(tmem + TM_D3 + cb * KB, make_desc(aGT + ks * 2 * CS_GT, CS_GT, RS),
                       make_desc(aQT + ks * 2 * CS_T, CS_T, RS), idn, (chunk | ks) != 0);
            mma_commit(&bar_stage[s]);
            if (cb + 2 < ncb) {            // refill this stage once its MMAs have consumed it
              mbar_wait(&bar_stage[s], ph_stage[s]); ph_stage[s] ^= 1u;
              fill(cb + 2);
            } else {
              used[s] = 1;                  // drained below together with bar_d
            }
          }
          mma_commit(&bar_d);
        } else {
          // keep the phase bookkeeping of the other threads in step with thread 0
          for (int cb = 0; cb < ncb; ++cb) {
            const int s = cb & 1;
            ph_full[s] ^= 1u;
            if (cb + 2 < ncb) ph_stage[s] ^= 1u; else used[s] = 1;
          }
        }
      } else
      for (int cb = 0; cb < ncb; ++cb) {
        const int s = cb & 1;
        if (used[s]) { mbar_wait(&bar_stage[s], ph_stage[s]); ph_stage[s] ^= 1u; used[s] = 0; }
        const int cw = min(KB, r2p - cb * KB);             // 32 or 16
        const int cvalid = max(0, min(cw, r2 - cb * KB));
        stage_cols_T(sStage[s], a.O, r2, n0, n_valid, cb * KB, cvalid);                 // O^T [c][n]
        stage_cols_T(sStage[s] + HALF_BYTES, a.qp, r2, b0, b_valid, cb * KB, cvalid);   // Q'^T [c][b]
        fence_async_smem();
        __syncthreads();
        if (tid == 0) {
          fence_after_sync();
          const uint32_t idn = make_idesc_tf32(128, cw, false, false);
          const uint32_t aOT = smem_u32(sStage[s]), aQT = aOT + HALF_BYTES;
          const uint32_t aG = smem_u32(sG), aGT = smem_u32(sGT);
          for (int ks = 0; ks < TN / 8; ++ks)      // H[b, c-block] = sum_n G[b,n] O^T[c,n]
            mma_tf32(tmem + TM_D2 + cb * KB, make_desc(aG + ks * 2 * CS_G, CS_G, RS),
                     make_desc(aOT + ks * 2 * CS_T, CS_T, RS), idn, ks != 0);
          for (int ks = 0; ks < TB / 8; ++ks)      // dO[n, c-block] += sum_b G^T[n,b] Q'^T[c,b]
            mma_tf32(tmem + TM_D3 + cb * KB, make_desc(aGT + ks * 2 * CS_GT, CS_GT, RS),
                     make_desc(aQT + ks * 2 * CS_T, CS_T, RS), idn, (chunk | ks) != 0);
          mma_commit(&bar_stage[s]);
          if (cb == ncb - 1) mma_commit(&bar_d);
        }
        used[s] = 1;
      }
      RT_TC_PROF(4);   // GEMM2/3 staging + issue
      // all MMAs of this chunk done: operands (G, G^T, stages) and D2 are free / ready
      mbar_wait(&bar_d, ph_d); ph_d ^= 1u;
      fence_after_sync();
      for (int s = 0; s < 2; ++s)
        if (used[s]) { mbar_wait(&bar_stage[s], ph_stage[s]); ph_stage[s] ^= 1u; used[s] = 0; }
      RT_TC_PROF(5);   // wait for GEMM2/3
      // ================= epilogue 2: D2 -> H_ws slice of this CTA (through smem for coalescing) =================
      for (int pass = 0; pass * 128 < r2p; ++pass) {
        const int c0 = pass * 128;
        const int cw = min(128, r2p - c0);
        for (int cblk = half; cblk * 32 < cw; cblk += 2) {
          const int rr = quarter * 32 + lane;
          if (cw - cblk * 32 >= 32) {
            uint32_t v[32];
            tmem_ld32(tmem + TM_D2 + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c0 + cblk * 32), v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 32; ++j) hbuf[rr * HB_LD + cblk * 32 + j] = __uint_as_float(v[j]);
          } else {
            uint32_t v[16];
            tmem_ld16(tmem + TM_D2 + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c0 + cblk * 32), v);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) hbuf[rr * HB_LD + cblk * 32 + j] = __uint_as_float(v[j]);
          }
        }
        fence_before_sync();
        __syncthreads();
        const int cols = min(cw, r2 - c0);
        float* Hc = a.H_ws + ((int64_t)blockIdx.x * a.B + b0) * r2 + c0;
        // warp w owns rows w, w+8, ...; lanes run along the columns (coalesced); 4 rows in flight
        if (vec_ok) {
          const int c4n = cols >> 2;                 // float4 per row (r2 % 4 == 0 => cols % 4 == 0)
          for (int rr0 = warp; rr0 < b_valid; rr0 += 4 * (kThreads / 32)) {
            for (int c4 = lane; c4 < c4n; c4 += 32) {
              float4 old[4];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int rr = rr0 + u * (kThreads / 32);
                old[u] = (!first_tile && rr < b_valid) ? *reinterpret_cast<const float4*>(Hc + (int64_t)rr * r2 + 4 * c4)
                                                       : make_float4(0.f, 0.f, 0.f, 0.f);
              }
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int rr = rr0 + u * (kThreads / 32);
                if (rr < b_valid) {
                  const float4 hv = *reinterpret_cast<const float4*>(&hbuf[rr * HB_LD + 4 * c4]);
                  *reinterpret_cast<float4*>(Hc + (int64_t)rr * r2 + 4 * c4) =
                      make_float4(old[u].x + hv.x, old[u].y + hv.y, old[u].z + hv.z, old[u].w + hv.w);
                }
              }
            }
          }
        } else
        for (int rr0 = warp; rr0 < b_valid; rr0 += 4 * (kThreads / 32)) {
          for (int c = lane; c < cols; c += 32) {
            float old[4];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int rr = rr0 + u * (kThreads / 32);
              old[u] = (!first_tile && rr < b_valid) ? Hc[(int64_t)rr * r2 + c] : 0.0f;
            }
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int rr = rr0 + u * (kThreads / 32);
              if (rr < b_valid) Hc[(int64_t)rr * r2 + c] = old[u] + hbuf[rr * HB_LD + c];
            }
          }
        }
        __syncthreads();
      }
      fence_after_sync();
      RT_TC_PROF(6);   // epilogue 2
    }
    // ================= tile epilogue: D3 -> dO rows of this tile =================
    for (int pass = 0; pass * 128 < r2p; ++pass) {
      const int c0 = pass * 128;
      const int cw = min(128, r2p - c0);
      for (int cblk = half; cblk * 32 < cw; cblk += 2) {
        const int rr = quarter * 32 + lane;
        if (cw - cblk * 32 >= 32) {
          uint32_t v[32];
          tmem_ld32(tmem + TM_D3 + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c0 + cblk * 32), v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 32; ++j) hbuf[rr * HB_LD + cblk * 32 + j] = __uint_as_float(v[j]);
        } else {
          uint32_t v[16];
          tmem_ld16(tmem + TM_D3 + ((uint32_t)(quarter * 32) << 16) + (uint32_t)(c0 + cblk * 32), v);
          tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 16; ++j) hbuf[rr * HB_LD + cblk * 32 + j] = __uint_as_float(v[j]);
        }
      }
      fence_before_sync();
      __syncthreads();
      const int cols = min(cw, r2 - c0);
      if (vec_ok) {
        const int c4n = cols >> 2;
        for (int e = tid; e < n_valid * c4n; e += kThreads) {
          const int rr = e / c4n, c4 = e - rr * c4n;
          *reinterpret_cast<float4*>(a.dO + (int64_t)(n0 + rr) * r2 + c0 + 4 * c4) =
              *reinterpret_cast<const float4*>(&hbuf[rr * HB_LD + 4 * c4]);
        }
      } else
      for (int e = tid; e < n_valid * cols; e += kThreads) {
        const int rr = e / cols, c = e - rr * cols;
        a.dO[(int64_t)(n0 + rr) * r2 + c0 + c] = hbuf[rr * HB_LD + c];
      }
      __syncthreads();
    }
    fence_after_sync();
    first_tile = false;
    RT_TC_PROF(7);   // tile epilogue
  }
  if (a.prof && tid == 0)
    for (int i = 0; i < 12; ++i) a.prof[blockIdx.x * 12 + i] = tp[i];
  if (first_tile) {   // CTA without a tile: its H slice must still be defined
    float* Hc = a.H_ws + (int64_t)blockIdx.x * a.B * r2;
    for (int64_t e = tid; e < (int64_t)a.B * r2; e += kThreads) Hc[e] = 0.0f;
  }
  double v = rt::warp_sum(loss_acc);
  if (lane == 0) red[warp] = v;
  fence_before_sync();
  __syncthreads();
  if (tid == 0) {
    double s = 0.0;
    for (int w = 0; w < kThreads / 32; ++w) s += red[w];
    a.loss_partial[blockIdx.x] = s;
  }
  if (warp == 0) tmem_dealloc<512>(tmem);
}

__global__ void reduce_H_tc_kernel(const float* __restrict__ H_ws, int nparts, int64_t count, float* __restrict__ H) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  float s = 0.0f;
  for (int k = 0; k < nparts; ++k) s += H_ws[(int64_t)k * count + i];
  H[i] = s;
}
__global__ void reduce_loss_tc_kernel(const double* __restrict__ partial, int n, double* __restrict__ out) {
  if (threadIdx.x == 0 && blockIdx.x == 0) {
    double s = 0.0;
    for (int i = 0; i < n; ++i) s += partial[i];
    out[0] = s;
  }
}

long long* g_tc_prof = nullptr;

int tc_grid(int n_local) {
  const int n_tiles = rt::cdiv(n_local, TN);
  const int sms = rt::sm_count();
  const int waves = rt::cdiv(n_tiles, sms);
  int grid = waves > 0 ? rt::cdiv(n_tiles, waves) : 1;
  return grid < 1 ? 1 : grid;
}

}  // namespace

struct TcLayout {
  int grid, n_tiles, n_chunks, ncb, packed;
  uint32_t full_bytes;
  size_t off_loss, off_Opk1, off_Qpk1, off_Opk2, off_Qpk2, total;
};
static TcLayout tc_layout(int B, int n_local, int r2) {
  TcLayout L;
  L.grid = tc_grid(n_local);
  L.n_tiles = rt::cdiv(n_local, TN);
  L.n_chunks = rt::cdiv(B, TB);
  const int r2p = (r2 + 15) / 16 * 16;
  L.ncb = r2p / KB + ((r2p % KB) ? 1 : 0);
  L.packed = (r2 % 4 == 0 && r2 <= 200) ? 1 : 0;
  const int nch = r2 >> 2, nchp = nch + (nch & 1);
  L.full_bytes = (uint32_t)nchp * CS_ROW;
  size_t o = rt::align_up((size_t)L.grid * B * r2 * sizeof(float), 256);
  L.off_loss = o; o += rt::align_up((size_t)L.grid * sizeof(double), 256);
  L.off_Opk1 = o; if (L.packed) o += rt::align_up((size_t)L.n_tiles * L.full_bytes, 256);
  L.off_Qpk1 = o; if (L.packed) o += rt::align_up((size_t)L.n_chunks * L.full_bytes, 256);
  L.off_Opk2 = o; if (L.packed) o += rt::align_up((size_t)L.n_tiles * L.ncb * TBLK_BYTES, 256);
  L.off_Qpk2 = o; if (L.packed) o += rt::align_up((size_t)L.n_chunks * L.ncb * TBLK_BYTES, 256);
  L.total = o;
  return L;
}

namespace rt {
size_t score_bce_tc_ws_bytes(int B, int n_local, int r2) { return tc_layout(B, n_local, r2).total; }

int score_bce_tc(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local, int n_total,
                 int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing, double* loss_sum,
                 float* H, float* dO, void* ws, void* stream) {
  RT_REQUIRE(r2 >= 1 && r2 <= 256, "rt_score_bce_tc: r2=%d out of range (1..256)", r2);
  cudaStream_t s = (cudaStream_t)stream;
  const TcLayout L = tc_layout(B, n_local, r2);
  const int grid = L.grid;
  char* base = (char*)ws;
  TcArgs a{};
  a.q = q; a.qp = qp ? qp : q; a.O = O;
  a.B = B; a.r2 = r2; a.n_begin = n_begin; a.n_local = n_local;
  a.off = tgt_off; a.idx = tgt_idx;
  a.t_neg = label_smoothing / (float)n_total;
  a.t_pos = (1.0f - label_smoothing) + a.t_neg;
  a.inv_count = (float)(1.0 / ((double)b_total * (double)n_total));
  a.H_ws = (float*)ws;
  a.loss_partial = (double*)(base + L.off_loss);
  a.dO = dO;
  a.n_tiles = L.n_tiles;
  a.r2p = (r2 + 15) / 16 * 16;
  a.prof = g_tc_prof;
  a.packed = L.packed; a.ncb = L.ncb; a.full_bytes = L.full_bytes;
  if (L.packed && n_local > 0) {
    a.Opk1 = (unsigned char*)(base + L.off_Opk1); a.Qpk1 = (unsigned char*)(base + L.off_Qpk1);
    a.Opk2 = (unsigned char*)(base + L.off_Opk2); a.Qpk2 = (unsigned char*)(base + L.off_Qpk2);
    pack_rows_kernel<<<L.n_tiles, 256, 0, s>>>(O, n_local, r2, (unsigned char*)a.Opk1, L.full_bytes);
    RT_LAUNCH_CHECK();
    pack_rows_kernel<<<L.n_chunks, 256, 0, s>>>(q, B, r2, (unsigned char*)a.Qpk1, L.full_bytes);
    RT_LAUNCH_CHECK();
    pack_cols_kernel<<<dim3(L.n_tiles, L.ncb), 256, 0, s>>>(O, n_local, r2, L.ncb, (unsigned char*)a.Opk2);
    RT_LAUNCH_CHECK();
    pack_cols_kernel<<<dim3(L.n_chunks, L.ncb), 256, 0, s>>>(a.qp, B, r2, L.ncb, (unsigned char*)a.Qpk2);
    RT_LAUNCH_CHECK();
  }
  RT_CHECK_CUDA(cudaFuncSetAttribute(score_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SMEM_BYTES));
  score_tc_kernel<<<grid, kThreads, SMEM_BYTES, s>>>(a);
  RT_LAUNCH_CHECK();
  const int64_t count = (int64_t)B * r2;
  reduce_H_tc_kernel<<<(int)((count + 255) / 256), 256, 0, s>>>(a.H_ws, grid, count, H);
  RT_LAUNCH_CHECK();
  reduce_loss_tc_kernel<<<1, 32, 0, s>>>(a.loss_partial, grid, loss_sum);
  RT_LAUNCH_CHECK();
  return 0;
}
}  // namespace rt

// Debug: per-CTA, per-phase cycle counters of score_tc_kernel ([grid][12] int64), NULL to disable.
extern "C" int rt_score_tc_set_profile(long long* dev_buf) { g_tc_prof = dev_buf; return 0; }
