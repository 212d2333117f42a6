// Shared helpers for librtucker_b200 (sm_100a only).  Not part of the public ABI.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include "../../include/rtucker.h"
#include "../../include/rtucker_debug.h"

namespace rt {

void set_error(const char* fmt, ...);
extern unsigned long long g_launches;  // kernels launched by this library in this process
extern double g_small_flops;           // fp64 flops of the GEMM operations RECORDED by the small stage (host side, eager launches)

#define RT_CHECK_CUDA(expr)                                                            \
  do {                                                                                 \
    cudaError_t _e = (expr);                                                           \
    if (_e != cudaSuccess) {                                                           \
      rt::set_error("%s:%d: %s failed: %s", __FILE__, __LINE__, #expr,                 \
                    cudaGetErrorString(_e));                                           \
      return 1;                                                                        \
    }                                                                                  \
  } while (0)

#define RT_REQUIRE(cond, ...)                                                          \
  do {                                                                                 \
    if (!(cond)) {                                                                     \
      rt::set_error(__VA_ARGS__);                                                      \
      return 2;                                                                        \
    }                                                                                  \
  } while (0)

#define RT_LAUNCH_CHECK()                 \
  do {                                    \
    ++rt::g_launches;                     \
    RT_CHECK_CUDA(cudaGetLastError());    \
  } while (0)

inline int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    if (n <= 0) n = 148;
  }
  return n;
}

// cudaFuncAttributeMaxDynamicSharedMemorySize, set once per (kernel, device) instead of on every launch
inline cudaError_t ensure_dyn_smem(const void* func, size_t bytes) {
  constexpr int kSlots = 64, kDevs = 16;
  static const void* funcs[kSlots];
  static size_t done[kSlots][kDevs];
  int dev = 0;
  cudaGetDevice(&dev);
  int slot = 0;
  while (slot < kSlots && funcs[slot] && funcs[slot] != func) ++slot;
  if (slot < kSlots && dev < kDevs) {
    if (funcs[slot] == func && done[slot][dev] >= bytes) return cudaSuccess;
    funcs[slot] = func;
  }
  cudaError_t e = cudaFuncSetAttribute(func, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e == cudaSuccess && slot < kSlots && dev < kDevs) done[slot][dev] = bytes;
  return e;
}

static inline int cdiv(int a, int b) { return (a + b - 1) / b; }
static inline size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

// Carves a workspace into regions in call order: take() returns the next region's byte offset and advances by its size
// rounded up to 256 bytes; o is then the total.
struct WsArena {
  size_t o = 0;
  size_t take(size_t bytes) { const size_t at = o; o += align_up(bytes, 256); return at; }
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ int warp_sum(int v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ---- functions shared between translation units ---------------------------------------------------------------------
// Each is defined in the file named above its group and called from at least one other.  They return 0 or an error
// code with rt_last_error() set, like the C ABI, unless they return a size or a flag.

// apply_tc.cu: the logits passes of apply_tc_kernel (3xTF32 tensor cores)
bool rank_tc_supported(int B, int n_local, int r2);
size_t rank_tc_ws_bytes(int B, int n_local, int r2);
int rank_tc(const float* q, const float* O, int B, int r2, int n_begin, int n_local, const int32_t* target,
            const float* p_target, const int32_t* flt_off, const int32_t* flt_idx, int32_t* greater, int32_t* equal,
            int32_t* equal_before, double* bce_sum, void* ws, cudaStream_t s, const int** overflow_flag);
int rank_tc_logit(const float* q, const float* O, int B, int r2, int n_begin, int n_local, const int32_t* target,
                  const float* z_target, int32_t* greater, int32_t* equal, int32_t* equal_before, void* ws,
                  cudaStream_t s, const int** overflow_flag);
size_t topk_tc_ws_bytes(int B, int n_local, int r2);
int topk_tc_pass(const float* q, const float* O, int B, int r2, int n_local, const float* p_k, const int* flag, int* cnt,
                 int32_t* seg, int cap, void* ws, cudaStream_t s, bool logit);
size_t score_lse_tc3_ws_bytes(int B, int n_local, int r2);
int score_lse_tc3(const float* q, const float* O, int B, int r2, int n_local, float* parts, void* ws, cudaStream_t s);
size_t score_ce_tc3_ws_bytes(int B, int n_local, int r2);
int score_ce_tc3(const float* q, const float* qp, const float* O, int B, int r2, int n_begin, int n_local, int n_total,
                 int b_total, const int32_t* tgt_off, const int32_t* tgt_idx, float label_smoothing, const float* parts,
                 int nparts, double* loss_sum, float* H, float* dO, void* ws, cudaStream_t s);

// score_bce.cu: exact fp32 probabilities or logits, and the log-sum-exp reductions of the cross-entropy
int score_dense(const float* q, const float* O, int B, int r2, int n_local, float* P, int64_t ldp, const int* gate,
                cudaStream_t s, bool logits);
int lse_combine(const float2* part, int ngroups, int64_t ld, int B, float* out, cudaStream_t s);
int ce_row_stats(const float* parts, int nparts, int B, int ld, float* stats, cudaStream_t s);

// gram_sym.cu: X^T X on the fp64 tensor cores
bool gram_sym_supported(int r);
size_t gram_sym_ws_bytes(int n, int r);
int gram_sym(const float* X, int64_t ld, int n, int r, double* out, void* ws, cudaStream_t s);

// tallskinny_v2.cu: register-tiled FP32 Gram and factor update
size_t gram_v2_ws_bytes(int n, int ra, int rb);
int gram_v2(const float* A, int64_t lda, const float* B, int64_t ldb, int n, int ra, int rb, double* out, void* ws,
            void* stream);
int apply_v2(float* Y, int64_t ldy, int n, int rc, const float* X0, int64_t ldx0, const double* a0_dev, int nk,
             const float* const* X_host, const int64_t* ldx_host, const int* rk_host, const double* const* K_host,
             void* stream);

// subspace.cu: batched dominant invariant subspaces
int subspace_batch(int count, const double* const* N, const int* n, const int* r, double* const* Y, const int* ldy,
                   void* const* ws, void* shared_ws, int* const* info, cudaStream_t s);
size_t subspace_ws_bytes(int n, int r);
size_t subspace_shared_ws_bytes();

}  // namespace rt
