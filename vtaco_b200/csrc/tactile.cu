// Compact tactile conditioning (SURVEY 8f-1): which tactile sensor's feature a query point takes,
// as ONE byte per query instead of the reference's dense c_img_all tensor (nx^3 x 32 floats =
// 2.1 GB at 256^3, built on the host with scipy.cdist).  The decoder kernels read the byte map
// (vtaco_decoder_args.tip_map) and add fc_p_img.weight[:, 3:] @ feature[id - 1].
//   * fingertip form  — generation.py:190-200, training.py:560-575: nearest fingertip (float64
//     cdist), within `radius`, and that finger touched;
//   * point-cloud form — generation.py:222-255 (encode_t2d): every query within `radius` of ANY
//     back-projected tactile point of sensor t takes sensor t's feature, sensors in increasing
//     order, later ones overwrite (the reference's hard-coded `64**3 x 8` split, which only works
//     for nx = 128, is not needed).
#include "decoder_common.cuh"
#include <math_constants.h>

namespace vtaco {

struct TipSet {
  double pos[VTACO_MAX_TIPS][3];
  int touch[VTACO_MAX_TIPS];
  int n;
  double radius;
};

__device__ __forceinline__ double dist3(double ax, double ay, double az, double bx, double by, double bz) {
  const double dx = ax - bx, dy = ay - by, dz = az - bz;
  return sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
}

// ids[i] = f + 1 if f = argmin_f |p_i - tip_f| (first minimum, like np.argmin), that distance
// < radius and touch[f]; else 0
__global__ void __launch_bounds__(256) fingertip_ids_kernel(const float* __restrict__ p, long long n, TipSet T,
                                                            uint8_t* __restrict__ ids) {
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double x = (double)p[3 * i], y = (double)p[3 * i + 1], z = (double)p[3 * i + 2];
    double best = CUDART_INF;
    int bi = -1;
    for (int f = 0; f < T.n; ++f) {
      const double d = dist3(x, y, z, T.pos[f][0], T.pos[f][1], T.pos[f][2]);
      if (d < best) { best = d; bi = f; }
    }
    ids[i] = (bi >= 0 && best < T.radius && T.touch[bi]) ? (uint8_t)(bi + 1) : (uint8_t)0;
  }
}

// per-scene fingertips on B dense lattices (blockIdx.y = scene): the decoder's own assignment (tip_assign), so the
// ids equal what a single-scene decode with these fingertips assigns in the kernel
__global__ void __launch_bounds__(256) fingertip_lattice_ids_kernel(const float* __restrict__ axis, int nx,
                                                                    const double* __restrict__ tips,
                                                                    const int32_t* __restrict__ touch, int n_tips,
                                                                    double radius, uint8_t* __restrict__ ids) {
  __shared__ DecParams sP;   // only the fingertip fields, which are all tip_assign reads
  const int b = blockIdx.y;
  if (threadIdx.x == 0) {
    sP.n_tips = n_tips;
    sP.tip_radius = radius;
    sP.tip_r2_hi = tip_prefilter_r2(radius);
    for (int f = 0; f < n_tips; ++f) {
      for (int d = 0; d < 3; ++d) {
        sP.tips[f][d] = tips[((size_t)b * n_tips + f) * 3 + d];
        sP.tipsf[f][d] = (float)sP.tips[f][d];
      }
      sP.tip_touch[f] = touch[(size_t)b * n_tips + f];
    }
  }
  __syncthreads();
  const long long n = (long long)nx * nx * nx;
  uint8_t* out = ids + (size_t)b * n;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < n; q += (long long)gridDim.x * blockDim.x) {
    const int iz = (int)(q % nx), iy = (int)((q / nx) % nx), ix = (int)(q / ((long long)nx * nx));
    const int f = tip_assign(sP, __ldg(axis + ix), __ldg(axis + iy), __ldg(axis + iz));
    out[q] = (uint8_t)(f + 1);
  }
}

// flat queries: map[i] = value where any of the n_pts points is closer than radius
__global__ void __launch_bounds__(256) point_map_flat_kernel(const float* __restrict__ p, long long n,
                                                             const double* __restrict__ pts, int n_pts, double radius,
                                                             uint8_t value, uint8_t* __restrict__ map) {
  extern __shared__ double spts[];
  for (int i = threadIdx.x; i < n_pts * 3; i += blockDim.x) spts[i] = pts[i];
  __syncthreads();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const double x = (double)p[3 * i], y = (double)p[3 * i + 1], z = (double)p[3 * i + 2];
    bool hit = false;
    for (int k = 0; k < n_pts && !hit; ++k) hit = dist3(spts[3 * k], spts[3 * k + 1], spts[3 * k + 2], x, y, z) < radius;
    if (hit) map[i] = value;
  }
}

// dense lattice: one block per tactile point walks the lattice cells of its bounding cube
__global__ void __launch_bounds__(128) point_map_dense_kernel(const float* __restrict__ axis, int nx,
                                                              const double* __restrict__ pts, double radius,
                                                              uint8_t value, uint8_t* __restrict__ map) {
  const double px = pts[3 * blockIdx.x], py = pts[3 * blockIdx.x + 1], pz = pts[3 * blockIdx.x + 2];
  __shared__ int lo[3], hi[3];
  if (threadIdx.x < 3) {
    // axis is increasing: first index with axis >= c - radius - slack, last with axis <= c + radius + slack
    const double c = threadIdx.x == 0 ? px : (threadIdx.x == 1 ? py : pz);
    const double slack = 1e-6;
    int a = 0, b = nx;                       // lower bound
    while (a < b) { const int m = (a + b) >> 1; if ((double)axis[m] < c - radius - slack) a = m + 1; else b = m; }
    lo[threadIdx.x] = a;
    a = 0; b = nx;                           // upper bound
    while (a < b) { const int m = (a + b) >> 1; if ((double)axis[m] <= c + radius + slack) a = m + 1; else b = m; }
    hi[threadIdx.x] = a;                     // exclusive
  }
  __syncthreads();
  const int ex = hi[0] - lo[0], ey = hi[1] - lo[1], ez = hi[2] - lo[2];
  if (ex <= 0 || ey <= 0 || ez <= 0) return;
  const int total = ex * ey * ez;
  for (int t = threadIdx.x; t < total; t += blockDim.x) {
    const int iz = lo[2] + t % ez, iy = lo[1] + (t / ez) % ey, ix = lo[0] + t / (ez * ey);
    if (dist3(px, py, pz, (double)axis[ix], (double)axis[iy], (double)axis[iz]) < radius)
      map[((size_t)ix * nx + iy) * nx + iz] = value;     // all writers of one launch store the same value
  }
}

}  // namespace vtaco

using namespace vtaco;

extern "C" int vtaco_fingertip_ids(const float* p, int64_t n, const double* tips_host, const int32_t* touch_host,
                                   int32_t n_tips, double radius, uint8_t* ids, void* stream) {
  if (n == 0) return VTACO_OK;
  if (!p || !ids || n < 0 || !tips_host || !touch_host || n_tips < 1 || n_tips > VTACO_MAX_TIPS) return VTACO_ERR_INVALID_ARG;
  TipSet T = {};
  T.n = n_tips;
  T.radius = radius;
  for (int f = 0; f < n_tips; ++f) {
    for (int d = 0; d < 3; ++d) T.pos[f][d] = tips_host[3 * f + d];
    T.touch[f] = touch_host[f];
  }
  long long blocks = (n + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  fingertip_ids_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(p, n, T, ids);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_tactile_point_map(const float* p, int64_t n, const float* axis, int32_t nx, const double* pts,
                                       int32_t n_pts, double radius, int32_t value, uint8_t* map, void* stream) {
  if (n_pts == 0) return VTACO_OK;
  if (!pts || !map || n_pts < 0 || value < 1 || value > 255 || radius < 0) return VTACO_ERR_INVALID_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  if (p) {
    if (n <= 0) return n == 0 ? VTACO_OK : VTACO_ERR_INVALID_ARG;
    if (n_pts > 2048) return VTACO_ERR_UNSUPPORTED;
    long long blocks = (n + 255) / 256;
    const long long cap = (long long)num_sms() * 8;
    if (blocks > cap) blocks = cap;
    point_map_flat_kernel<<<(unsigned)blocks, 256, (size_t)n_pts * 3 * sizeof(double), st>>>(p, n, pts, n_pts, radius,
                                                                                         (uint8_t)value, map);
  } else {
    if (!axis || nx < 1) return VTACO_ERR_INVALID_ARG;
    point_map_dense_kernel<<<n_pts, 128, 0, st>>>(axis, nx, pts, radius, (uint8_t)value, map);
  }
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_fingertip_lattice_ids(const float* axis, int32_t nx, int32_t B, const double* tips,
                                           const int32_t* touch, int32_t n_tips, double radius, uint8_t* ids,
                                           void* stream) {
  if (!axis || !tips || !touch || !ids || nx < 1 || B < 1 || B > 65535 || n_tips < 1 || n_tips > VTACO_MAX_TIPS)
    return VTACO_ERR_INVALID_ARG;
  const long long n = (long long)nx * nx * nx;
  long long blocks = (n + 255) / 256;
  long long cap = (long long)num_sms() * 8 / B;
  if (cap < 1) cap = 1;
  if (blocks > cap) blocks = cap;
  fingertip_lattice_ids_kernel<<<dim3((unsigned)blocks, (unsigned)B), 256, 0, (cudaStream_t)stream>>>(
      axis, nx, tips, touch, n_tips, radius, ids);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}
