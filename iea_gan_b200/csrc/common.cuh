// common.cuh -- shared helpers for libiea_sm100.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <stdint.h>
#include <stdio.h>
#include "../../include/iea_b200.h"

namespace iea {

void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define IEA_CHECK_ARG(cond, ...)                 \
  do {                                           \
    if (!(cond)) {                               \
      iea::set_error(__VA_ARGS__);               \
      return -2;                                 \
    }                                            \
  } while (0)

#define IEA_CUDA(call)                                                        \
  do {                                                                        \
    cudaError_t e_ = (call);                                                  \
    if (e_ != cudaSuccess) {                                                  \
      iea::set_error("%s failed: %s", #call, cudaGetErrorString(e_));         \
      return -3;                                                              \
    }                                                                         \
  } while (0)

typedef __nv_bfloat16 bf16;

__device__ __forceinline__ float ld_act(const void* p, int dtype, int64_t i) {
  return dtype == IEA_BF16 ? __bfloat162float(((const bf16*)p)[i]) : ((const float*)p)[i];
}
__device__ __forceinline__ void st_act(void* p, int dtype, int64_t i, float v) {
  if (dtype == IEA_BF16) ((bf16*)p)[i] = __float2bfloat16_rn(v);
  else ((float*)p)[i] = v;
}
// value as the consumer will read it back (rounded through the storage type)
__device__ __forceinline__ float round_act(int dtype, float v) {
  return dtype == IEA_BF16 ? __bfloat162float(__float2bfloat16_rn(v)) : v;
}
static inline size_t dtype_size(int dtype) { return dtype == IEA_BF16 ? 2 : 4; }

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}
// block-wide sum, result valid in every thread; blockDim.x multiple of 32, <= 1024.
// `red` is shared scratch of >= 33 floats.  Deterministic (fixed tree).
__device__ __forceinline__ float block_sum(float v, float* red) {
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float t = lane < nw ? red[lane] : 0.f;
    t = warp_sum(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}
__device__ __forceinline__ float block_max(float v, float* red) {
  int lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
  v = warp_max(v);
  __syncthreads();
  if (lane == 0) red[wid] = v;
  __syncthreads();
  if (wid == 0) {
    float t = lane < nw ? red[lane] : -3.4e38f;
    t = warp_max(t);
    if (lane == 0) red[32] = t;
  }
  __syncthreads();
  return red[32];
}

// packed fp32 pairs (Blackwell FFMA2 / FADD2): half the issue slots of scalar fp32
__device__ __forceinline__ float2 ffma2(float2 a, float2 b, float2 c) {
  float2 r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(reinterpret_cast<unsigned long long&>(r))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)),
        "l"(reinterpret_cast<unsigned long long&>(c)));
  return r;
}
__device__ __forceinline__ float2 fadd2(float2 a, float2 b) {
  float2 r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(reinterpret_cast<unsigned long long&>(r))
      : "l"(reinterpret_cast<unsigned long long&>(a)), "l"(reinterpret_cast<unsigned long long&>(b)));
  return r;
}

// bf16 <-> fp32: two channels in a 32-bit word, eight in a 16-byte chunk
__device__ __forceinline__ float2 bf2_to_f2(uint32_t w) { return make_float2(__uint_as_float(w << 16), __uint_as_float(w & 0xFFFF0000u)); }
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  __nv_bfloat162 t = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&t);
}
__device__ __forceinline__ void unpack8(const uint4& q, float* f) {
  const uint32_t w[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    f[2 * i] = __uint_as_float(w[i] << 16);
    f[2 * i + 1] = __uint_as_float(w[i] & 0xFFFF0000u);
  }
}
__device__ __forceinline__ uint4 pack8(const float* f) {
  return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
}

// 16-byte global -> shared copy (cp.async.cg) and its commit / wait groups
__device__ __forceinline__ void cp16(uint32_t dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"(dst), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>  // wait until at most N committed groups are still in flight
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

inline int cdiv(int64_t a, int64_t b) { return (int)((a + b - 1) / b); }

// SMs of the current device (persistent-kernel grids); 148 (B200) when the query fails
inline int sm_count() {
  int dev = 0, sms = 148;
  cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
  return sms;
}
// stored size of the input along a conv-resolution extent v: half behind nearest-up2, twice behind the 2x2 pool
__host__ __device__ inline int stored_res(const iea_conv_desc& d, int v) {
  return d.in_mode == IEA_IN_UP2 ? v / 2 : (d.in_mode == IEA_IN_POOL2 ? v * 2 : v);
}
// tensor-memory columns to allocate for `need` accumulator columns: a power of two, at least 32
inline uint32_t tmem_cols_for(uint32_t need) {
  uint32_t cols = 32;
  while (cols < need) cols <<= 1;
  return cols;
}

}  // namespace iea
