/* Debug, self-test and profiling entry points of librtucker_b200.so -- NOT part of the drop-in boundary
 * (include/rtucker.h).  Used by tests/ (known-answer tests of the tcgen05 building blocks), tools/ and bench.py
 * (timing the fused kernel alone). */
#ifndef RTUCKER_DEBUG_H
#define RTUCKER_DEBUG_H
#include "rtucker.h"
#ifdef __cplusplus
extern "C" {
#endif

/* Same call restricted to some of its phases (bit 0: operand scaling + packing, bit 1: the fused kernel,
 * bit 2: H / loss reduction); a single phase needs a workspace prepared by the earlier ones on the same inputs.
 * bench.py times the fused kernel alone this way. */
int rt_score_bce_v3_phases(const float* q, const float* O, int B, int r2, int n_begin, int n_local, int n_total,
                           int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing,
                           float o_absmax_hint, double* loss_sum, float* H, float* dO, float* centre_state, void* ws,
                           void* stream, int phases);

/* Debug: per-CTA, per-role (producer, MMA issuer, epilogue, flush) cycle counters [grid][4][10] int64; NULL = off. */
int rt_score_v3_set_profile(long long* dev_buf);
/* Debug: per-CTA, per-phase cycle counters of the variant-1 score kernel ([grid][12] int64); NULL = off. */
int rt_score_tc_set_profile(long long* dev_buf);
/* Debug: per-CTA cycle counters of rt_eigh's block Jacobi kernel ([grid][4] int64: phase A, sync, phase B, sync);
 * NULL = off. */
int rt_eigh_set_profile(long long* dev_buf);

/* Known-answer self test of the tcgen05 building blocks: D[128,N] = op(A) op(B)^T in TF32
 * (a_mn/b_mn select MN-major operands given as [K][M] / [K][N]); used by tests/test_gpu_tc.py. */
int rt_tc_selftest(const float* A, const float* B, float* D, int N, int K, int a_mn, int b_mn, int flags,
                   void* stream);
/* Same with fp16 operands (kind::f16), the building block of variant 2; and a known-answer test of the
 * shared->global bulk copies: out[0:n] = a (bulk store) then out += b (bulk fp32 add-reduction at the L2). */
int rt_tc_selftest16(const float* A, const float* B, float* D, int N, int K, int a_mn, int b_mn, int flags,
                     void* stream);
int rt_bulk_reduce_selftest(const float* a, const float* b, float* out, int n, void* stream);
/* Debug: issue `reps` back-to-back kind::f16 MMAs (M = 128, N, K = 16) on shared-memory operands in the K-major
 * (0) or MN-major (1) view; out_dev[0] = cycles to issue, out_dev[1] = cycles until all have completed. */
int rt_mma_probe(int N, int ksteps, int a_mn, int b_mn, int reps, long long* out_dev, void* stream);

/* fp64 flops (2 m n K per product, half for a symmetric Gram) of all GEMM operations the small stage has recorded in
 * this process -- host-side count at record time, so it advances on eager launches only (not on CUDA-graph replays).
 * bench.py divides its increase over the eagerly launched profile steps by the stage time. */
double rt_small_flop_count(void);

#ifdef __cplusplus
}
#endif
#endif
