// Device building blocks shared by the fp64 and staging kernels (inline PTX and fixed-order sums), defined once.  The
// tcgen05 / TMEM / mbarrier / bulk-copy helpers are in tc.cuh, the score's special functions in exact.cuh.
#pragma once
#include "common.h"

namespace rt {

// fp64 tensor-core MMA: D(8x8) += A(8x4) B(4x8); lane l holds A[l>>2][l&3], B[l&3][l>>2], C[l>>2][2*(l&3)+{0,1}]
__device__ __forceinline__ void dmma884(double& c0, double& c1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0, %1}, {%2}, {%3}, {%0, %1};\n"
               : "+d"(c0), "+d"(c1) : "d"(a), "d"(b));
}

// Grid barrier on the counter *bar.  It holds only if the kernel runs under a cooperative launch (every CTA is
// resident), *bar is zero before the first CTA's first call, and every CTA calls it equally often with its own
// `target`, starting at 0.  Thread 0 arrives with a release reduction: the CTA's writes, ordered before it by the first
// __syncthreads, are visible to any thread that observes the arrival.  It then polls with acquire loads until all
// gridDim.x arrivals of this round are seen, which orders every other CTA's writes before this CTA's reads after the
// second __syncthreads.  The fire-and-forget arrival saves one L2 round trip over an atomic with a return value.
__device__ __forceinline__ void grid_barrier(unsigned int* bar, unsigned int& target) {
  __syncthreads();
  if (threadIdx.x == 0) {
    target += gridDim.x;
    asm volatile("red.release.gpu.global.add.u32 [%0], 1;\n" :: "l"(bar) : "memory");
    unsigned int seen;
    do {
      asm volatile("ld.acquire.gpu.global.u32 %0, [%1];\n" : "=r"(seen) : "l"(bar) : "memory");
    } while (seen < target);
  }
  __syncthreads();
}

// Programmatic dependent launch.  launch_dependents lets the next kernel of the stream, if it was launched with
// programmatic stream serialization, start once every CTA of this grid has signalled (or exited).  wait blocks until
// the grids this one depends on programmatically have completed and their writes are visible; without such a
// dependency it returns at once.
__device__ __forceinline__ void pdl_launch_dependents() { asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;\n" ::: "memory"); }

// 16-byte asynchronous global -> shared copy (L2 only), to a shared-memory address or a generic pointer into shared
// memory; completion through commit / wait_group or wait_all
__device__ __forceinline__ void cp_async16(uint32_t dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" :: "r"(dst_smem), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst_smem, const void* src) {
  cp_async16((uint32_t)__cvta_generic_to_shared(dst_smem), src);
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;\n" :: "n"(N) : "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// deterministic CTA-wide sum of a kWarps-warp CTA (fixed shuffle tree, fixed warp order); result valid in every thread
template <int kWarps>
__device__ __forceinline__ double cta_sum(double v, double* sh) {
  v = warp_sum(v);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = v;
  __syncthreads();
  double s = 0.0;
#pragma unroll
  for (int w = 0; w < kWarps; ++w) s += sh[w];
  return s;
}

// u-th tile (ti, tj) with ti <= tj of a T x T tile grid, row by row
__device__ __forceinline__ void sym_tile(int u, int T, int& ti, int& tj) {
  ti = 0;
  while (u >= T - ti) { u -= T - ti; ++ti; }
  tj = ti + u;
}

// out[i] = sum over k < nsplit of part[k * count + i], k ascending, accumulated in Acc: the second stage of a split
// reduction, bit-identical on every replica.  Idx (int or int64_t) is the index type of the call site's count.  Each
// source file gets its own copy (internal linkage): the library exports no kernel of this header.
namespace {
template <typename Acc, typename P, typename Out, typename Idx>
__global__ void split_sum_kernel(const P* __restrict__ part, int nsplit, Idx count, Out* __restrict__ out) {
  const Idx i = (Idx)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  Acc s = 0;
  for (int k = 0; k < nsplit; ++k) s += (Acc)part[(int64_t)k * count + i];
  out[i] = (Out)s;
}
}  // namespace

}  // namespace rt
