// common.cuh -- shared helpers for libhrb200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>

#include "../../include/hrb200.h"

#define HRB_API extern "C" __attribute__((visibility("default")))

namespace hrb {

// thread-local detail message behind hrb_last_error()
char* err_buf();
int fail(int status, const char* fmt, ...);

#define HRB_REQUIRE(cond, ...)                              \
  do {                                                      \
    if (!(cond)) return ::hrb::fail(HRB_BAD_ARG, __VA_ARGS__); \
  } while (0)

#define HRB_CUDA(call)                                                                          \
  do {                                                                                          \
    cudaError_t e_ = (call);                                                                    \
    if (e_ != cudaSuccess)                                                                      \
      return ::hrb::fail(HRB_CUDA_ERROR, "%s:%d %s -> %s", __FILE__, __LINE__, #call,           \
                         cudaGetErrorString(e_));                                               \
  } while (0)

// every kernel launch of this library goes through this macro: it counts the launch
// (hrb_launch_count) and surfaces launch-configuration errors
#define HRB_LAUNCH_CHECK()             \
  do {                                 \
    ::hrb::count_launches(1);          \
    HRB_CUDA(cudaGetLastError());      \
  } while (0)

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

void count_launches(int n);
int sm_count();  // cached cudaDevAttrMultiProcessorCount of the current device

// ---------------------------------------------------------------------------------------------
// device helpers
// ---------------------------------------------------------------------------------------------
// 128-bit read-only gather load that does not allocate in L1 (rows are touched once per CTA).
__device__ __forceinline__ float4 ldg_nc_na(const float4* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0,%1,%2,%3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
// streaming 128-bit store (output is consumed by a later kernel, not by this CTA)
__device__ __forceinline__ void stg_na(float4* p, const float4& v) {
  asm volatile("st.global.L1::no_allocate.v4.f32 [%0], {%1,%2,%3,%4};" ::"l"(p), "f"(v.x), "f"(v.y),
               "f"(v.z), "f"(v.w)
               : "memory");
}

__host__ __device__ __forceinline__ uint32_t hash_u32(uint32_t x) {  // lowbias32, mirrored in oracle
  x ^= x >> 16;
  x *= 0x7FEB352Du;
  x ^= x >> 15;
  x *= 0x846CA68Bu;
  x ^= x >> 16;
  return x;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// true in every thread of the last CTA to finish (the partials of every CTA are then visible to it).  The barrier first: every
// thread of this CTA has stored its partials before thread 0 publishes the CTA as done.
__device__ __forceinline__ bool last_block(unsigned int* counter) {
  __shared__ bool last;
  __syncthreads();
  __threadfence();
  if (threadIdx.x == 0) last = atomicAdd(counter, 1u) == gridDim.x - 1;
  __syncthreads();
  if (last) __threadfence();
  return last;
}

// Keras Ftrl (TF ApplyFtrl / ApplyFtrlV2 functors) on one element; acc and lin are its accumulator and linear slots, g already
// holds the l2 regulariser term, l2 has beta / (2*lr) added.  Returns the new weight.  The row update (plan.cuh), the dense step
// and the multi-tensor step (misc.cu) all call this: every operation is rounded explicitly (no contraction left to the
// compiler), so a step from the same slots gives the same bits on every path.  The final select (not a multiply) keeps a
// y of 0 (acc = 0, l2 = 0) from turning the 0 of a small |linear| into NaN.
__device__ __forceinline__ float ftrl_pow(float a, float lr_power) { return lr_power == -0.5f ? __fsqrt_rn(a) : powf(a, -lr_power); }
__device__ __forceinline__ float ftrl_elem(float w, float& acc, float& lin, float g, float lr, float l1, float l2, float lr_power,
                                           float l2_shrinkage) {
  const float gs = __fadd_rn(g, __fmul_rn(__fmul_rn(2.f, l2_shrinkage), w));
  const float acc_new = __fadd_rn(acc, __fmul_rn(g, g));
  const float p_new = ftrl_pow(acc_new, lr_power);
  const float sigma = __fdiv_rn(__fsub_rn(p_new, ftrl_pow(acc, lr_power)), lr);
  lin = __fadd_rn(lin, __fsub_rn(gs, __fmul_rn(sigma, w)));
  acc = acc_new;
  const float y = __fadd_rn(__fdiv_rn(p_new, lr), __fmul_rn(2.f, l2));
  return fabsf(lin) > l1 ? __fdiv_rn(__fsub_rn(copysignf(l1, lin), lin), y) : 0.f;
}

__device__ __forceinline__ float sigmoidf_(float x) { return 1.0f / (1.0f + expf(-x)); }

__device__ __forceinline__ float act_apply(int act, float x) {
  switch (act) {
    case HRB_ACT_RELU: return fmaxf(x, 0.0f);
    case HRB_ACT_SIGMOID: return sigmoidf_(x);
    case HRB_ACT_TANH: return tanhf(x);
    default: return x;
  }
}
// derivative expressed with the activation OUTPUT y
__device__ __forceinline__ float act_grad_from_out(int act, float y) {
  switch (act) {
    case HRB_ACT_RELU: return y > 0.0f ? 1.0f : 0.0f;
    case HRB_ACT_SIGMOID: return y * (1.0f - y);
    case HRB_ACT_TANH: return 1.0f - y * y;
    default: return 1.0f;
  }
}

}  // namespace hrb
