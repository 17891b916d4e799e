// Library plumbing (status strings, device query), point->cell indexing and the
// self-measured FP32 FMA peak used as the decoder's roofline denominator.
#include "common.cuh"
#include <map>
#include <mutex>

namespace vtaco {

static thread_local cudaError_t g_last_err = cudaSuccess;
void set_last_cuda_error(cudaError_t e) { g_last_err = e; }

int num_sms() {
  static std::atomic<int> cached[64];
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 148;
  int c = cached[dev & 63].load(std::memory_order_relaxed);
  if (c == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    c = n;
    cached[dev & 63].store(n, std::memory_order_relaxed);
  }
  return c;
}

cudaError_t smem_opt_in(const void* kernel, size_t bytes) {
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  static std::mutex mu;
  static std::map<std::pair<const void*, int>, size_t> done;   // largest size set, per (kernel, device)
  std::lock_guard<std::mutex> lock(mu);
  size_t& set = done[{kernel, dev}];
  if (set < bytes) {
    e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    if (e == cudaSuccess) set = bytes;
  }
  return e;
}

// ---------------------------------------------------------------------------------------
// (1) point -> cell.  src/common.py:268-309 (normalise + clamp) and :333-348 (index).
// One thread per point; 12 B in, 4/8 B out per point — pure streaming.
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) point_to_cell_kernel(const float* __restrict__ p, long long n, NormConst nc,
                                                            int reso, int kind, int32_t* __restrict__ idx32,
                                                            int64_t* __restrict__ idx64, float* __restrict__ coord) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float x = p[i * 3 + 0], y = p[i * 3 + 1], z = p[i * 3 + 2];
    int idx;
    if (kind == VTACO_GRID) {
      const float ux = norm3d(x, nc), uy = norm3d(y, nc), uz = norm3d(z, nc);
      idx = cell_of(ux, reso) + reso * (cell_of(uy, reso) + reso * cell_of(uz, reso));
      if (coord) { coord[i * 3 + 0] = ux; coord[i * 3 + 1] = uy; coord[i * 3 + 2] = uz; }
    } else {
      const float a = (kind == VTACO_PLANE_YZ) ? y : x;
      const float b = (kind == VTACO_PLANE_XY) ? y : z;
      const float ua = norm2d(a, nc), ub = norm2d(b, nc);
      idx = cell_of(ua, reso) + reso * cell_of(ub, reso);
      if (coord) { coord[i * 2 + 0] = ua; coord[i * 2 + 1] = ub; }
    }
    if (idx32) idx32[i] = idx;
    if (idx64) idx64[i] = idx;
  }
}

// ---------------------------------------------------------------------------------------
// (4) FP32 FMA peak: 64 independent accumulators per thread, weights in registers.
// ---------------------------------------------------------------------------------------
template <bool F2>
__global__ void __launch_bounds__(256) fp32_peak_kernel(float* out, int iters, float seed) {
  float2 acc[32];
  float2 w[8];
#pragma unroll
  for (int j = 0; j < 32; ++j) acc[j] = make_float2(seed * j, seed * (j + 1));
#pragma unroll
  for (int j = 0; j < 8; ++j) w[j] = make_float2(1.0f + seed * j, 1.0f - seed * j);
  float x = seed + threadIdx.x * 1e-9f;
  for (int it = 0; it < iters; ++it) {
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      if (F2) {
        const float2 xx = make_float2(x, x);
#pragma unroll
        for (int j = 0; j < 32; ++j) acc[j] = __ffma2_rn(w[j & 7], xx, acc[j]);
      } else {
#pragma unroll
        for (int j = 0; j < 32; ++j) {
          acc[j].x = fmaf(w[j & 7].x, x, acc[j].x);
          acc[j].y = fmaf(w[j & 7].y, x, acc[j].y);
        }
      }
      x = x * 0.999f;
    }
  }
  float s = 0.f;
#pragma unroll
  for (int j = 0; j < 32; ++j) s += acc[j].x + acc[j].y;
  if (s == 12345.678f) out[0] = s;  // keep the loop alive
}

}  // namespace vtaco

using namespace vtaco;

extern "C" int vtaco_abi_version(void) { return VTACO_ABI_VERSION; }

extern "C" const char* vtaco_status_string(int status) {
  switch (status) {
    case VTACO_OK: return "ok";
    case VTACO_ERR_INVALID_ARG: return "invalid argument";
    case VTACO_ERR_UNSUPPORTED: return "unsupported shape or configuration";
    case VTACO_ERR_CUDA: return "CUDA runtime error";
    case VTACO_ERR_CAPACITY: return "output capacity too small";
    default: return "unknown status";
  }
}

extern "C" const char* vtaco_last_cuda_error(void) { return cudaGetErrorString(g_last_err); }

extern "C" int vtaco_point_to_cell(const float* p, int64_t n_points, double padding, int reso, int kind, int div_mode,
                                   int32_t* idx32, int64_t* idx64, float* coord, void* stream) {
  if (n_points == 0) return VTACO_OK;
  if (!p || n_points < 0 || reso < 1 || kind < 0 || kind > 3) return VTACO_ERR_INVALID_ARG;
  if (div_mode != VTACO_DIV_RECIPROCAL && div_mode != VTACO_DIV_TRUE) return VTACO_ERR_INVALID_ARG;
  if (kind == VTACO_GRID ? reso > 1290 : reso > 46340) return VTACO_ERR_UNSUPPORTED;  // int32 flat index
  const NormConst nc = make_norm_const(padding, div_mode);
  long long blocks = (n_points + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  point_to_cell_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p, n_points, nc, reso, kind, idx32, idx64,
                                                                         coord);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_fp32_peak(int variant, int iters, double* flops_per_s_host, void* stream) {
  if (!flops_per_s_host || iters <= 0) return VTACO_ERR_INVALID_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  float* d = nullptr;
  VTACO_CUDA_CHECK(cudaMalloc(&d, sizeof(float)));
  cudaEvent_t e0, e1;
  VTACO_CUDA_CHECK(cudaEventCreate(&e0));
  VTACO_CUDA_CHECK(cudaEventCreate(&e1));
  const int blocks = num_sms() * 4;
  double best = 0.0;
  for (int rep = 0; rep < 4; ++rep) {
    VTACO_CUDA_CHECK(cudaEventRecord(e0, st));
    if (variant == 1) fp32_peak_kernel<true><<<blocks, 256, 0, st>>>(d, iters, 1e-3f);
    else fp32_peak_kernel<false><<<blocks, 256, 0, st>>>(d, iters, 1e-3f);
    VTACO_CUDA_CHECK(cudaEventRecord(e1, st));
    VTACO_CUDA_CHECK(cudaEventSynchronize(e1));
    float ms = 0.f;
    VTACO_CUDA_CHECK(cudaEventElapsedTime(&ms, e0, e1));
    const double flops = 2.0 * 64.0 * 4.0 * (double)iters * 256.0 * blocks;
    const double rate = flops / (ms * 1e-3);
    if (rep > 0 && rate > best) best = rate;
  }
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  cudaFree(d);
  VTACO_LAUNCH_CHECK();
  *flops_per_s_host = best;
  return VTACO_OK;
}
