// Counter-based standard normal fill (rt_fill_normal, include/rtucker.h): the seeded Gaussian directions and core
// entries that set_rank (rank.py) adds when a rank grows.  Every value is a pure function of (seed, stream_id,
// global row, column): Philox4x32-10 on the counter (column / 4, row lo, row hi, stream_id) under the key (seed lo,
// seed hi), two Box-Muller pairs per counter.  An entity shard that passes its first global row as row_begin
// therefore draws exactly the rows of the unsharded draw, and replicated objects draw the same bits on every rank,
// with no generator state to keep in step across ranks.
#include "common.h"

namespace {

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
  constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int i = 0; i < 10; ++i) {
    const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
    const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
    c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
    k.x += W0;
    k.y += W1;
  }
  return c;
}

// Box-Muller on two 24-bit uniforms: u1 in (0, 1] (so the log is finite), the angle 2 pi u2 with u2 in [0, 1)
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  const float u1 = (float)((a >> 8) + 1u) * 0x1p-24f;
  const float r = sqrtf(-2.0f * logf(u1));
  float s, c;
  sincospif((float)(b >> 8) * 0x1p-23f, &s, &c);
  return make_float2(r * c, r * s);
}

__global__ void __launch_bounds__(256)
fill_normal_kernel(float* __restrict__ out, int rows, int cols, int64_t row_begin, uint2 key, uint32_t stream_id) {
  const int quads = (cols + 3) >> 2;
  const int64_t items = (int64_t)rows * quads;
  for (int64_t it = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; it < items; it += (int64_t)gridDim.x * blockDim.x) {
    const int row = (int)(it / quads), q = (int)(it - (int64_t)row * quads);
    const uint64_t g = (uint64_t)(row_begin + row);
    const uint4 x = philox4x32_10(make_uint4((uint32_t)q, (uint32_t)g, (uint32_t)(g >> 32), stream_id), key);
    const float2 z01 = box_muller(x.x, x.y), z23 = box_muller(x.z, x.w);
    const float z[4] = {z01.x, z01.y, z23.x, z23.y};
    float* dst = out + (int64_t)row * cols;
    const int c0 = 4 * q;
#pragma unroll
    for (int j = 0; j < 4; ++j)
      if (c0 + j < cols) dst[c0 + j] = z[j];
  }
}

}  // namespace

extern "C" int rt_fill_normal(float* out, int rows, int cols, int64_t row_begin, uint64_t seed, uint32_t stream_id,
                              void* stream) {
  RT_REQUIRE(rows >= 0 && cols >= 0 && row_begin >= 0, "rt_fill_normal: bad shape rows=%d cols=%d row_begin=%lld",
             rows, cols, (long long)row_begin);
  if (rows == 0 || cols == 0) return 0;
  RT_REQUIRE(out != nullptr, "rt_fill_normal: out is NULL");
  const int64_t items = (int64_t)rows * ((cols + 3) / 4);
  const int64_t want = (items + 255) / 256, cap = (int64_t)rt::sm_count() * 8;
  const int grid = (int)(want < cap ? want : cap);
  fill_normal_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, rows, cols, row_begin,
                                                             make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)),
                                                             stream_id);
  RT_LAUNCH_CHECK();
  return 0;
}
