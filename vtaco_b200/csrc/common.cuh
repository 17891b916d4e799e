// Shared device/host helpers of the vtaco_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "../../include/vtaco_b200.h"

namespace vtaco {

void set_last_cuda_error(cudaError_t e);

#define VTACO_CUDA_CHECK(expr)                                   \
  do {                                                           \
    cudaError_t _e = (expr);                                     \
    if (_e != cudaSuccess) {                                     \
      ::vtaco::set_last_cuda_error(_e);                          \
      return VTACO_ERR_CUDA;                                     \
    }                                                            \
  } while (0)

#define VTACO_LAUNCH_CHECK() VTACO_CUDA_CHECK(cudaPeekAtLastError())

int num_sms();  // SM count of the current device (cached)
// Lets `kernel` use `bytes` of dynamic shared memory on the current device.  The attribute is set once per
// (kernel, device), and again only for a larger size; safe to call from several host threads.
cudaError_t smem_opt_in(const void* kernel, size_t bytes);

// Constants of src/common.py:283,288,302,306 formed like Python does: in double,
// rounded to fp32 where they meet an fp32 tensor.
struct NormConst {
  float d2, inv2, hi2;  // normalize_coordinate:    / (1+padding+10e-6), clamp 1-10e-6
  float d3, inv3, hi3;  // normalize_3d_coordinate: / (1+padding+10e-4), clamp 1-10e-4
  int div_true;
};

inline NormConst make_norm_const(double padding, int div_mode) {
  NormConst c;
  const double d2 = (1.0 + padding) + 10e-6, d3 = (1.0 + padding) + 10e-4;
  c.d2 = (float)d2;
  c.d3 = (float)d3;
  // ATen CUDA div_true_kernel_cuda multiplies by the reciprocal of the python scalar;
  // measured on B200 / torch 2.11 (tests/test_coords_gpu.py): the reciprocal is formed
  // in double from the double scalar and then rounded to fp32 — fp32(1/1.10001) differs
  // from 1.0f/fp32(1.10001) in the last bit.
  c.inv2 = (float)(1.0 / d2);
  c.inv3 = (float)(1.0 / d3);
  c.hi2 = (float)(1.0 - 10e-6);
  c.hi3 = (float)(1.0 - 10e-4);
  c.div_true = (div_mode == VTACO_DIV_TRUE);
  return c;
}

// src/common.py:283-290 (per element; NaN passes through like the masked writes do)
__device__ __forceinline__ float norm2d(float v, const NormConst& c) {
  float u = c.div_true ? __fdiv_rn(v, c.d2) : __fmul_rn(v, c.inv2);
  u = __fadd_rn(u, 0.5f);
  if (u >= 1.0f) u = c.hi2;
  if (u < 0.0f) u = 0.0f;
  return u;
}
// src/common.py:302-308
__device__ __forceinline__ float norm3d(float v, const NormConst& c) {
  float u = c.div_true ? __fdiv_rn(v, c.d3) : __fmul_rn(v, c.inv3);
  u = __fadd_rn(u, 0.5f);
  if (u >= 1.0f) u = c.hi3;
  if (u < 0.0f) u = 0.0f;
  return u;
}
// src/common.py:342 — (x * reso).long(): fp32 multiply, truncation
__device__ __forceinline__ int cell_of(float u, int reso) {
  return (int)__fmul_rn(u, (float)reso);
}

// Monotone float <-> int32 key: signed-int order == float order (for atomicMin/Max).
__host__ __device__ __forceinline__ int32_t float_to_key(float f) {
#ifdef __CUDA_ARCH__
  int32_t b = __float_as_int(f);
#else
  union { float f; int32_t i; } u; u.f = f; int32_t b = u.i;
#endif
  return b >= 0 ? b : (b ^ 0x7fffffff);
}
__host__ __device__ __forceinline__ float key_to_float(int32_t k) {
  int32_t b = k >= 0 ? k : (k ^ 0x7fffffff);
#ifdef __CUDA_ARCH__
  return __int_as_float(b);
#else
  union { float f; int32_t i; } u; u.i = b; return u.f;
#endif
}

}  // namespace vtaco
