// Shared pieces of the SIMT and tcgen05 decoder kernels: launch parameters, ATen
// grid_sampler arithmetic (reference decoder.py:55-68) and the fingertip assignment
// (reference generation.py:190-200).
#pragma once
#include "common.cuh"
#include <math_constants.h>

namespace vtaco {

constexpr int kThreads = 256;
constexpr int kTileQ = 512;
constexpr int kSC = kTileQ + 1;  // column stride (floats): conflict-free for both phases
constexpr unsigned kFull = 0xffffffffu;

struct DecParams {
  const float* p;
  const float* axis;
  const float* grid;
  const float* plane[3];
  const float* weights;
  const float* c_img;
  const float* tip_feat;
  const uint8_t* tip_map;   // optional: per-query tactile id (0 = none), replaces the in-kernel fingertip test
  float* logits;
  float* contact;
  int32_t* minmax_key;
  long long N;       // queries per sample (flat) / nx^3 (dense)
  long long total;   // flat: B*N
  long long n_tiles;
  int B, nx, x0, x1, nbx, nby;  // dense: bricks along x (slab) and along y/z
  int Rg, Rp, n_blocks, leaky, use_img, nearest, n_tips, wfloats, has_c;
  float* peers[8];   // dense multi-GPU: logit grids of all ranks (fused all-gather)
  float* mcast;      // NVLS multicast alias of those grids (one multimem.st reaches every rank) or NULL
  int n_peers;
  int tc_products;   // 3 = 3xTF32 (fp32 fidelity); 2 = TF32 main + BF16 corrections; 1 = single TF32 product (variant 3: timing experiments, ~1e-3 accuracy)
  int tc_split;      // tcgen05 kernels: threads per query (1 | 2)
  int t_nbx, t_nby, t_nbz, t_xend;  // tcgen05 kernel, dense mode: 2x2x32 bricks and slab end row
  NormConst nc;
  double tips[VTACO_MAX_TIPS][3];
  float tipsf[VTACO_MAX_TIPS][3];   // fp32 copies for the prefilter
  int tip_touch[VTACO_MAX_TIPS];
  double tip_radius;
  float tip_r2_hi;  // fp32 prefilter threshold (squared, padded)
  int tip_ps;       // tip_feat is [B][n_tips][32]: one table per sample (byte-map form, tcgen05 kernels)
};

__device__ __forceinline__ void store_logit(const DecParams& P, long long idx, float v) {
  if (P.mcast) {
    asm volatile("multimem.st.relaxed.sys.global.f32 [%0], %1;" ::"l"(P.mcast + idx), "f"(v) : "memory");
  } else if (P.n_peers > 0) {
#pragma unroll 1
    for (int r = 0; r < P.n_peers; ++r) P.peers[r][idx] = v;
  } else {
    P.logits[idx] = v;
  }
}

// ---- ATen grid_sampler arithmetic (align_corners=True, padding_mode='border') ----
// decoder.py:58 `vgrid = 2.0 * xy - 1.0`, then grid_sampler_unnormalize:
// ((g + 1) / 2) * (size - 1), clip to [0, size-1].
__device__ __forceinline__ float unnormalize(float u, int R) {
  float g = __fsub_rn(__fmul_rn(2.0f, u), 1.0f);
  float t = __fmul_rn(__fmul_rn(__fadd_rn(g, 1.0f), 0.5f), (float)(R - 1));
  return fminf((float)(R - 1), fmaxf(t, 0.0f));
}

__device__ __forceinline__ float4 f4_fma(float w, float4 v, float4 a) {
  a.x = fmaf(v.x, w, a.x); a.y = fmaf(v.y, w, a.y); a.z = fmaf(v.z, w, a.z); a.w = fmaf(v.w, w, a.w);
  return a;
}
__device__ __forceinline__ float4 f4_add(float4 a, float4 b) {
  return make_float4(a.x + b.x, a.y + b.y, a.z + b.z, a.w + b.w);
}

// Trilinear sample of a channels-last volume [Rz][Ry][Rx][32]; `vol` already points
// at this lane's 4 channels of the sample.  Corner order and weights follow
// ATen's grid_sampler_3d (tnw,tne,tsw,tse,bnw,bne,bsw,bse).
__device__ __forceinline__ float4 sample_volume(const float4* __restrict__ vol, int R, float ux, float uy,
                                                float uz, bool nearest) {
  const float tx = unnormalize(ux, R), ty = unnormalize(uy, R), tz = unnormalize(uz, R);
  if (nearest) {
    const int x = (int)nearbyintf(tx), y = (int)nearbyintf(ty), z = (int)nearbyintf(tz);
    return __ldg(vol + ((size_t)(z * R + y) * R + x) * 8);
  }
  const float flx = floorf(tx), fly = floorf(ty), flz = floorf(tz);
  const int x0 = (int)flx, y0 = (int)fly, z0 = (int)flz;
  const float fx1 = tx - flx, fx0 = (flx + 1.0f) - tx;
  const float fy1 = ty - fly, fy0 = (fly + 1.0f) - ty;
  const float fz1 = tz - flz, fz0 = (flz + 1.0f) - tz;
  // out-of-range corners (index == R) carry weight 0 and are skipped by ATen; read a
  // clamped address instead and keep the (zero) weight.
  const int x1 = min(x0 + 1, R - 1), y1 = min(y0 + 1, R - 1), z1 = min(z0 + 1, R - 1);
  const bool vx = (x0 + 1 < R), vy = (y0 + 1 < R), vz = (z0 + 1 < R);
  const size_t r00 = (size_t)(z0 * R + y0) * R, r01 = (size_t)(z0 * R + y1) * R;
  const size_t r10 = (size_t)(z1 * R + y0) * R, r11 = (size_t)(z1 * R + y1) * R;
  const float4 v000 = __ldg(vol + (r00 + x0) * 8), v001 = __ldg(vol + (r00 + x1) * 8);
  const float4 v010 = __ldg(vol + (r01 + x0) * 8), v011 = __ldg(vol + (r01 + x1) * 8);
  const float4 v100 = __ldg(vol + (r10 + x0) * 8), v101 = __ldg(vol + (r10 + x1) * 8);
  const float4 v110 = __ldg(vol + (r11 + x0) * 8), v111 = __ldg(vol + (r11 + x1) * 8);
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  a = f4_fma(fx0 * fy0 * fz0, v000, a);
  a = f4_fma(vx ? fx1 * fy0 * fz0 : 0.f, v001, a);
  a = f4_fma(vy ? fx0 * fy1 * fz0 : 0.f, v010, a);
  a = f4_fma((vx && vy) ? fx1 * fy1 * fz0 : 0.f, v011, a);
  a = f4_fma(vz ? fx0 * fy0 * fz1 : 0.f, v100, a);
  a = f4_fma((vx && vz) ? fx1 * fy0 * fz1 : 0.f, v101, a);
  a = f4_fma((vy && vz) ? fx0 * fy1 * fz1 : 0.f, v110, a);
  a = f4_fma((vx && vy && vz) ? fx1 * fy1 * fz1 : 0.f, v111, a);
  return a;
}

// Bilinear sample of a channels-last plane [R_i1][R_i0][32] (ua -> W/i0, ub -> H/i1);
// corner order nw, ne, sw, se as in ATen's grid_sampler_2d.
__device__ __forceinline__ float4 sample_plane(const float4* __restrict__ pl, int R, float ua, float ub,
                                               bool nearest) {
  const float tx = unnormalize(ua, R), ty = unnormalize(ub, R);
  if (nearest) {
    const int x = (int)nearbyintf(tx), y = (int)nearbyintf(ty);
    return __ldg(pl + ((size_t)y * R + x) * 8);
  }
  const float flx = floorf(tx), fly = floorf(ty);
  const int x0 = (int)flx, y0 = (int)fly;
  const float fx1 = tx - flx, fx0 = (flx + 1.0f) - tx;
  const float fy1 = ty - fly, fy0 = (fly + 1.0f) - ty;
  const int x1 = min(x0 + 1, R - 1), y1 = min(y0 + 1, R - 1);
  const bool vx = (x0 + 1 < R), vy = (y0 + 1 < R);
  const float4 v00 = __ldg(pl + ((size_t)y0 * R + x0) * 8), v01 = __ldg(pl + ((size_t)y0 * R + x1) * 8);
  const float4 v10 = __ldg(pl + ((size_t)y1 * R + x0) * 8), v11 = __ldg(pl + ((size_t)y1 * R + x1) * 8);
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  a = f4_fma(fx0 * fy0, v00, a);
  a = f4_fma(vx ? fx1 * fy0 : 0.f, v01, a);
  a = f4_fma(vy ? fx0 * fy1 : 0.f, v10, a);
  a = f4_fma((vx && vy) ? fx1 * fy1 : 0.f, v11, a);
  return a;
}

// c of one query (decoder.py:55-68): the sum of its samples of the grid and the planes, channels
// [4*sub, 4*sub + 4) of sample b
__device__ __forceinline__ float4 sample_feature_sum(const DecParams& P, int b, int sub, float x, float y, float z) {
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (P.grid) {
    const int R = P.Rg;
    const float4* vol = reinterpret_cast<const float4*>(P.grid) + (size_t)b * R * R * R * 8 + sub;
    c = sample_volume(vol, R, norm3d(x, P.nc), norm3d(y, P.nc), norm3d(z, P.nc), P.nearest);
  }
  if (P.plane[0] || P.plane[1] || P.plane[2]) {
    const int R = P.Rp;
    const float ux = norm2d(x, P.nc), uy = norm2d(y, P.nc), uz = norm2d(z, P.nc);
    const size_t boff = (size_t)b * R * R * 8 + sub;
    if (P.plane[0]) c = f4_add(c, sample_plane(reinterpret_cast<const float4*>(P.plane[0]) + boff, R, ux, uz, P.nearest));
    if (P.plane[1]) c = f4_add(c, sample_plane(reinterpret_cast<const float4*>(P.plane[1]) + boff, R, ux, uy, P.nearest));
    if (P.plane[2]) c = f4_add(c, sample_plane(reinterpret_cast<const float4*>(P.plane[2]) + boff, R, uy, uz, P.nearest));
  }
  return c;
}

// Warp-reduce the running logit min / max and merge them into P.minmax_key (ordered-int keys)
__device__ __forceinline__ void flush_minmax(const DecParams& P, float vmin, float vmax, int lane) {
  if (P.minmax_key) {
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) {
      vmin = fminf(vmin, __shfl_xor_sync(kFull, vmin, d));
      vmax = fmaxf(vmax, __shfl_xor_sync(kFull, vmax, d));
    }
    if (lane == 0 && vmin <= vmax) {
      atomicMin(P.minmax_key, float_to_key(vmin));
      atomicMax(P.minmax_key + 1, float_to_key(vmax));
    }
  }
}

// fp32 prefilter threshold of tip_assign (squared, padded so that it never rejects a query within `radius`)
__host__ __device__ __forceinline__ float tip_prefilter_r2(double radius) {
  const double r = radius * 1.01 + 1e-4;
  return (float)(r * r);
}
// generation.py:190-200: nearest fingertip in float64 (scipy cdist), within radius, touched.
__device__ __forceinline__ int tip_assign(const DecParams& P, float x, float y, float z);
// tactile feature row of a query: from the byte map when given, else the in-kernel fingertip test
__device__ __forceinline__ int tip_of_query(const DecParams& P, long long qidx, float x, float y, float z) {
  if (P.tip_map) {
    const int f = (int)__ldg(P.tip_map + qidx) - 1;
    return f < P.n_tips ? f : -1;
  }
  return tip_assign(P, x, y, z);
}
__device__ __forceinline__ int tip_assign(const DecParams& P, float x, float y, float z) {
  bool near = false;
  for (int f = 0; f < P.n_tips; ++f) {
    const float dx = x - P.tipsf[f][0], dy = y - P.tipsf[f][1], dz = z - P.tipsf[f][2];
    near |= (dx * dx + dy * dy + dz * dz) < P.tip_r2_hi;
  }
  if (!near) return -1;
  double best = CUDART_INF;
  int bi = -1;
  for (int f = 0; f < P.n_tips; ++f) {
    const double dx = (double)x - P.tips[f][0], dy = (double)y - P.tips[f][1], dz = (double)z - P.tips[f][2];
    const double d = sqrt(__dadd_rn(__dadd_rn(__dmul_rn(dx, dx), __dmul_rn(dy, dy)), __dmul_rn(dz, dz)));
    if (d < best) { best = d; bi = f; }
  }
  return (bi >= 0 && best < P.tip_radius && P.tip_touch[bi]) ? bi : -1;
}

// Variant 1 (exact fp32 SIMT kernel, decoder.cu), which a tcgen05 launcher runs instead when its shared-memory
// layout does not fit at P.n_blocks.  P must still carry the SIMT tiling vtaco_decoder_forward set, so the
// launchers call it before set_tc_tiles.  VTACO_ERR_UNSUPPORTED for a call with a tip byte map.
int launch_decoder_simt(const DecParams& P, bool dense, cudaStream_t stream);

}  // namespace vtaco
