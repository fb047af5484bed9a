// Device / host helpers shared by the row kernels (rowops.cu) and the single-token decode kernels (decode.cu).
#pragma once
#include "host_common.h"
#include "ptx.cuh"

namespace vl2 {

// ---------------------------------------------------------------------------------------------------------
// helpers
// ---------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void unpack8(const uint4& u, float (&f)[8]) {
  f[0] = bf16_lo(u.x); f[1] = bf16_hi(u.x); f[2] = bf16_lo(u.y); f[3] = bf16_hi(u.y);
  f[4] = bf16_lo(u.z); f[5] = bf16_hi(u.z); f[6] = bf16_lo(u.w); f[7] = bf16_hi(u.w);
}
__device__ __forceinline__ uint4 pack8(const float (&f)[8]) {
  return make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]), pack_bf16(f[6], f[7]));
}
__device__ __forceinline__ float silu(float x) { return x / (1.f + __expf(-x)); }

// Block-wide sum of two floats (blockDim.x multiple of 32, <= 1024).  `red` is 64 floats of shared memory.
__device__ __forceinline__ float2 block_sum2(float a, float b, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();  // protect `red` against the previous use
  if (lane == 0) { red[warp] = a; red[32 + warp] = b; }
  __syncthreads();
  float ra = (lane < nw) ? red[lane] : 0.f;
  float rb = (lane < nw) ? red[32 + lane] : 0.f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ra += __shfl_xor_sync(0xffffffffu, ra, o);
    rb += __shfl_xor_sync(0xffffffffu, rb, o);
  }
  return make_float2(ra, rb);
}

// Block-wide sum of four floats in one round (blockDim.x multiple of 32, <= 1024).  `red` is 128 floats of shared memory.
__device__ __forceinline__ float4 block_sum4(float a, float b, float c, float d, float* red) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
    c += __shfl_xor_sync(0xffffffffu, c, o);
    d += __shfl_xor_sync(0xffffffffu, d, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nw = blockDim.x >> 5;
  __syncthreads();  // protect `red` against the previous use
  if (lane == 0) { red[warp] = a; red[32 + warp] = b; red[64 + warp] = c; red[96 + warp] = d; }
  __syncthreads();
  float ra = (lane < nw) ? red[lane] : 0.f, rb = (lane < nw) ? red[32 + lane] : 0.f;
  float rc = (lane < nw) ? red[64 + lane] : 0.f, rd = (lane < nw) ? red[96 + lane] : 0.f;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ra += __shfl_xor_sync(0xffffffffu, ra, o);
    rb += __shfl_xor_sync(0xffffffffu, rb, o);
    rc += __shfl_xor_sync(0xffffffffu, rc, o);
    rd += __shfl_xor_sync(0xffffffffu, rd, o);
  }
  return make_float4(ra, rb, rc, rd);
}

static inline int row_threads(int C) {
  int t = (C / 8 + 31) / 32 * 32;
  if (t > 512) t = 512;
  if (t < 32) t = 32;
  return t;
}
static constexpr int kMaxVec = 4;  // vectors of 8 channels held per thread => C <= 512*8*4 = 16384

__device__ __forceinline__ float warp_sum(float a) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) a += __shfl_xor_sync(0xffffffffu, a, o);
  return a;
}

static inline int grid_for(int64_t work_items, int threads, int max_blocks = 148 * 16) {
  int64_t b = (work_items + threads - 1) / threads;
  if (b > max_blocks) b = max_blocks;
  if (b < 1) b = 1;
  return (int)b;
}

// M = 1 GEMV launcher (decode.cu); vl2_gemm_skinny routes single-row calls to it.  w_scale != nullptr: W is fp8 E4M3
// with one fp32 scale per row (vl2_gemv_fp8).
int launch_gemv(const void* x, const void* W, const float* bias, const void* residual, void* y, int out_f32, int N, int K,
                int act, float rms_eps, cudaStream_t stream, const float* w_scale = nullptr);

}  // namespace vl2
