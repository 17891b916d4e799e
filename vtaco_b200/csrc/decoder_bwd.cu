// Backward of the fused LocalDecoder for sm_100a (SURVEY §8f-2).
//
// Gradients of LocalDecoder.forward / forward_img / forward_contact (reference
// src/conv_onet/models/decoder.py:71-161; trained through autograd by
// src/conv_onet/training.py:79,617) with respect to every decoder parameter, the
// feature tensors of c_plane (grid and/or planes) and the per-query c_img.
//
//   forward:   n_0 = fc_p(p) [+ W_img c_img]
//              m_i = n_i + fc_c[i](c);  h_i = fc_0(relu(m_i));  n_{i+1} = m_i + fc_1(relu(h_i))
//              out = fc_out(act(n_5))
//   backward:  g_5 = dout * w_out * act'(n_5)
//              gh_i = (W1_i^T g_{i+1}) * [h_i > 0];   g_i = g_{i+1} + (W0_i^T gh_i) * [m_i > 0]
//              dc  += Wc_i^T g_i;   dW1_i = g_{i+1} (x) relu(h_i);  dW0_i = gh_i (x) relu(m_i);  dWc_i = g_i (x) c
//
// Kernel 1 (decoder_bwd_query_kernel): one thread per query, persistent CTAs, all weights in
// shared memory (the K-major forward packing serves both W x — broadcast LDS.128 against a
// private shared-memory column — and W^T g — row dot products against registers).  The forward
// pass is recomputed in fp32 (nothing is saved by the forward kernels); ReLU masks are kept
// as 32-bit masks.  Per-layer activations A and output gradients G are written as
// [slot][query][32] rows (128-byte rows, STG.128) for kernel 2; dc is scattered into the
// channels-last feature gradients with 16-byte vector atomics (red.global.add.v4.f32).
// Kernel 2 (linear_wgrad_kernel, wgrad.cuh): dW = G^T A, one CTA per (matrix, query chunk),
// 128-query tiles staged in shared memory, 32x32 outer-product accumulators spread over 256
// threads (4 per thread), one atomicAdd per element and CTA; db = column sums of G.
#include "decoder_common.cuh"
#include "wgrad.cuh"
#include <algorithm>

namespace vtaco {

constexpr int kBT = 256;       // threads per CTA == queries per tile (352 threads — what registers and shared memory allow — measured slower: 400 vs 307 us at 65 536 queries)
constexpr int kBS = kBT + 1;   // column stride (floats)
constexpr int kMaxBlocks = 8;

// workspace slots (rows of 32 floats per query)
constexpr int kSlotC = 0;                      // sampled features c
__host__ __device__ constexpr int slot_rm(int i) { return 1 + i; }                       // relu(m_i)
__host__ __device__ constexpr int slot_rh(int nb, int i) { return 1 + nb + i; }          // relu(h_i)
__host__ __device__ constexpr int slot_aout(int nb) { return 1 + 2 * nb; }               // act(n_last)
__host__ __device__ constexpr int slot_gm(int nb, int i) { return 2 + 2 * nb + i; }      // dL/dn_i, i = 0..nb
__host__ __device__ constexpr int slot_gh(int nb, int i) { return 3 + 3 * nb + i; }      // dL/dh_i (masked)
__host__ __device__ constexpr int n_slots(int nb) { return 3 + 4 * nb; }

struct BwdParams {
  const float* p;
  const float* c_img;
  const float* grid;
  const float* plane[3];
  const float* weights;
  const float* dlogits;
  const float* dcontact;
  float* ws;
  float* d_grid;
  float* d_plane[3];
  float* d_c_img;
  long long Q, N;
  int Rg, Rp, n_blocks, leaky, use_img, nearest, has_c, wfloats;
  NormConst nc;
};

// ---- interpolation taps (same arithmetic as sample_volume / sample_plane) ----
__device__ __forceinline__ void volume_taps(int R, float ux, float uy, float uz, bool nearest, int (&off)[8],
                                            float (&w)[8]) {
  const float tx = unnormalize(ux, R), ty = unnormalize(uy, R), tz = unnormalize(uz, R);
  if (nearest) {
    const int x = (int)nearbyintf(tx), y = (int)nearbyintf(ty), z = (int)nearbyintf(tz);
#pragma unroll
    for (int t = 0; t < 8; ++t) { off[t] = (z * R + y) * R + x; w[t] = 0.f; }
    w[0] = 1.f;
    return;
  }
  const float flx = floorf(tx), fly = floorf(ty), flz = floorf(tz);
  const int x0 = (int)flx, y0 = (int)fly, z0 = (int)flz;
  const float fx1 = tx - flx, fx0 = (flx + 1.0f) - tx;
  const float fy1 = ty - fly, fy0 = (fly + 1.0f) - ty;
  const float fz1 = tz - flz, fz0 = (flz + 1.0f) - tz;
  const int x1 = min(x0 + 1, R - 1), y1 = min(y0 + 1, R - 1), z1 = min(z0 + 1, R - 1);
  const bool vx = (x0 + 1 < R), vy = (y0 + 1 < R), vz = (z0 + 1 < R);
  off[0] = (z0 * R + y0) * R + x0; w[0] = fx0 * fy0 * fz0;
  off[1] = (z0 * R + y0) * R + x1; w[1] = vx ? fx1 * fy0 * fz0 : 0.f;
  off[2] = (z0 * R + y1) * R + x0; w[2] = vy ? fx0 * fy1 * fz0 : 0.f;
  off[3] = (z0 * R + y1) * R + x1; w[3] = (vx && vy) ? fx1 * fy1 * fz0 : 0.f;
  off[4] = (z1 * R + y0) * R + x0; w[4] = vz ? fx0 * fy0 * fz1 : 0.f;
  off[5] = (z1 * R + y0) * R + x1; w[5] = (vx && vz) ? fx1 * fy0 * fz1 : 0.f;
  off[6] = (z1 * R + y1) * R + x0; w[6] = (vy && vz) ? fx0 * fy1 * fz1 : 0.f;
  off[7] = (z1 * R + y1) * R + x1; w[7] = (vx && vy && vz) ? fx1 * fy1 * fz1 : 0.f;
}

__device__ __forceinline__ void plane_taps(int R, float ua, float ub, bool nearest, int (&off)[4], float (&w)[4]) {
  const float tx = unnormalize(ua, R), ty = unnormalize(ub, R);
  if (nearest) {
    const int x = (int)nearbyintf(tx), y = (int)nearbyintf(ty);
#pragma unroll
    for (int t = 0; t < 4; ++t) { off[t] = y * R + x; w[t] = 0.f; }
    w[0] = 1.f;
    return;
  }
  const float flx = floorf(tx), fly = floorf(ty);
  const int x0 = (int)flx, y0 = (int)fly;
  const float fx1 = tx - flx, fx0 = (flx + 1.0f) - tx;
  const float fy1 = ty - fly, fy0 = (fly + 1.0f) - ty;
  const int x1 = min(x0 + 1, R - 1), y1 = min(y0 + 1, R - 1);
  const bool vx = (x0 + 1 < R), vy = (y0 + 1 < R);
  off[0] = y0 * R + x0; w[0] = fx0 * fy0;
  off[1] = y0 * R + x1; w[1] = vx ? fx1 * fy0 : 0.f;
  off[2] = y1 * R + x0; w[2] = vy ? fx0 * fy1 : 0.f;
  off[3] = y1 * R + x1; w[3] = (vx && vy) ? fx1 * fy1 : 0.f;
}

template <int T>
__device__ __forceinline__ void gather_taps(float (&c)[32], const float* __restrict__ base, const int (&off)[T],
                                            const float (&w)[T]) {
#pragma unroll
  for (int t = 0; t < T; ++t) {
    if (w[t] != 0.f) {
      const float4* src = reinterpret_cast<const float4*>(base + (size_t)off[t] * 32);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 v = __ldg(src + j);
        c[4 * j + 0] = fmaf(w[t], v.x, c[4 * j + 0]);
        c[4 * j + 1] = fmaf(w[t], v.y, c[4 * j + 1]);
        c[4 * j + 2] = fmaf(w[t], v.z, c[4 * j + 2]);
        c[4 * j + 3] = fmaf(w[t], v.w, c[4 * j + 3]);
      }
    }
  }
}

// d_feat[tap] += w[tap] * dc, dc read from the thread's shared-memory column
template <int T>
__device__ __forceinline__ void scatter_taps(float* __restrict__ base, const int (&off)[T], const float (&w)[T],
                                             const float* __restrict__ dcol) {
#pragma unroll
  for (int t = 0; t < T; ++t) {
    if (w[t] != 0.f) {
      float4* dst = reinterpret_cast<float4*>(base + (size_t)off[t] * 32);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 v = make_float4(w[t] * dcol[(4 * j + 0) * kBS], w[t] * dcol[(4 * j + 1) * kBS],
                                     w[t] * dcol[(4 * j + 2) * kBS], w[t] * dcol[(4 * j + 3) * kBS]);
        atomicAdd(dst + j, v);
      }
    }
  }
}

// acc[j] += sum_k W[k][j] * xcol[k]          (W K-major in shared memory: W[k][j] = weight[j][k])
__device__ __forceinline__ void mv_fwd(float (&acc)[32], const float* __restrict__ W, const float* __restrict__ xcol) {
#pragma unroll 4
  for (int k = 0; k < 32; ++k) {
    const float x = xcol[k * kBS];
    const float4* w4 = reinterpret_cast<const float4*>(W + k * 32);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 w = w4[j];
      acc[4 * j + 0] = fmaf(w.x, x, acc[4 * j + 0]);
      acc[4 * j + 1] = fmaf(w.y, x, acc[4 * j + 1]);
      acc[4 * j + 2] = fmaf(w.z, x, acc[4 * j + 2]);
      acc[4 * j + 3] = fmaf(w.w, x, acc[4 * j + 3]);
    }
  }
}

// ocol[k] (+)= sum_j W[k][j] * g[j]          (= (weight^T g)[k])
template <bool ACC>
__device__ __forceinline__ void mv_bwd(float* __restrict__ ocol, const float* __restrict__ W, const float (&g)[32]) {
#pragma unroll 4
  for (int k = 0; k < 32; ++k) {
    const float4* w4 = reinterpret_cast<const float4*>(W + k * 32);
    float s0 = 0.f, s1 = 0.f, s2 = 0.f, s3 = 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 w = w4[j];
      s0 = fmaf(w.x, g[4 * j + 0], s0);
      s1 = fmaf(w.y, g[4 * j + 1], s1);
      s2 = fmaf(w.z, g[4 * j + 2], s2);
      s3 = fmaf(w.w, g[4 * j + 3], s3);
    }
    const float s = (s0 + s1) + (s2 + s3);
    if (ACC) ocol[k * kBS] += s; else ocol[k * kBS] = s;
  }
}

__device__ __forceinline__ void store_row(float* __restrict__ row, const float (&v)[32]) {
  float4* r4 = reinterpret_cast<float4*>(row);
#pragma unroll
  for (int j = 0; j < 8; ++j) r4[j] = make_float4(v[4 * j], v[4 * j + 1], v[4 * j + 2], v[4 * j + 3]);
}

__global__ void __launch_bounds__(kBT, 1) decoder_bwd_query_kernel(const __grid_constant__ BwdParams P) {
  extern __shared__ __align__(16) float smem[];
  float* sW = smem;
  float* sC = sW + P.wfloats;
  float* sX = sC + 32 * kBS;
  float* sD = sX + 32 * kBS;
  uint32_t* sM = reinterpret_cast<uint32_t*>(sD + 32 * kBS);  // [2*n_blocks][kBT] ReLU masks

  for (int i = threadIdx.x; i < P.wfloats / 4; i += kBT)
    reinterpret_cast<float4*>(sW)[i] = __ldg(reinterpret_cast<const float4*>(P.weights) + i);
  __syncthreads();

  const int nb = P.n_blocks;
  const size_t slot_stride = (size_t)P.Q * 32;
  float* ccol = sC + threadIdx.x;
  float* xcol = sX + threadIdx.x;
  float* dcol = sD + threadIdx.x;
  uint32_t* mcol = sM + threadIdx.x;
  const float* Wo = sW + VTACO_DEC_OFF_BLOCKS + nb * VTACO_DEC_BLOCK_STRIDE;
  const float slope = P.leaky ? 0.2f : 0.0f;

  // every column is private to its thread: no block-level barrier inside the tile loop
  for (long long q = (long long)blockIdx.x * kBT + threadIdx.x; q < P.Q; q += (long long)gridDim.x * kBT) {
    const float px = __ldg(P.p + q * 3), py = __ldg(P.p + q * 3 + 1), pz = __ldg(P.p + q * 3 + 2);
    const int b = (int)(q / P.N);
    float* wsq = P.ws + (size_t)q * 32;
    float n[32], h[32];

    // ---------------- features c = sum over grid / planes (decoder.py:72-83) ----------------
    if (P.has_c) {
#pragma unroll
      for (int k = 0; k < 32; ++k) h[k] = 0.f;
      if (P.grid) {
        int off[8]; float w[8];
        volume_taps(P.Rg, norm3d(px, P.nc), norm3d(py, P.nc), norm3d(pz, P.nc), P.nearest, off, w);
        gather_taps<8>(h, P.grid + (size_t)b * P.Rg * P.Rg * P.Rg * 32, off, w);
      }
      if (P.plane[0] || P.plane[1] || P.plane[2]) {
        const float ux = norm2d(px, P.nc), uy = norm2d(py, P.nc), uz = norm2d(pz, P.nc);
        const size_t boff = (size_t)b * P.Rp * P.Rp * 32;
        int off[4]; float w[4];
        if (P.plane[0]) { plane_taps(P.Rp, ux, uz, P.nearest, off, w); gather_taps<4>(h, P.plane[0] + boff, off, w); }
        if (P.plane[1]) { plane_taps(P.Rp, ux, uy, P.nearest, off, w); gather_taps<4>(h, P.plane[1] + boff, off, w); }
        if (P.plane[2]) { plane_taps(P.Rp, uy, uz, P.nearest, off, w); gather_taps<4>(h, P.plane[2] + boff, off, w); }
      }
#pragma unroll
      for (int k = 0; k < 32; ++k) { ccol[k * kBS] = h[k]; dcol[k * kBS] = 0.f; }
      store_row(wsq + kSlotC * slot_stride, h);
    }

    // ---------------- forward recompute ----------------
    {
      const float* Wp = sW + (P.use_img ? VTACO_DEC_OFF_WPI : VTACO_DEC_OFF_WP);
#pragma unroll
      for (int j = 0; j < 32; ++j)
        n[j] = fmaf(Wp[64 + j], pz, fmaf(Wp[32 + j], py, fmaf(Wp[j], px, Wp[VTACO_DEC_OFF_BP - VTACO_DEC_OFF_WP + j])));  // = BPI - WPI
      if (P.use_img && P.c_img) {
        const float4* ci = reinterpret_cast<const float4*>(P.c_img) + q * 8;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 v = __ldg(ci + j);
          xcol[(4 * j) * kBS] = v.x; xcol[(4 * j + 1) * kBS] = v.y;
          xcol[(4 * j + 2) * kBS] = v.z; xcol[(4 * j + 3) * kBS] = v.w;
        }
        mv_fwd(n, sW + VTACO_DEC_OFF_WIMG, xcol);
      }
    }
#pragma unroll 1
    for (int i = 0; i < nb; ++i) {
      const float* Wb = sW + VTACO_DEC_OFF_BLOCKS + i * VTACO_DEC_BLOCK_STRIDE;
      if (P.has_c) {
        mv_fwd(n, Wb + VTACO_DEC_BLK_WC, ccol);
#pragma unroll
        for (int k = 0; k < 32; ++k) n[k] += Wb[VTACO_DEC_BLK_BC + k];
      }
      uint32_t mm = 0, mh = 0;
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        mm |= (n[k] > 0.f ? 1u : 0u) << k;
        h[k] = fmaxf(n[k], 0.f);
        xcol[k * kBS] = h[k];
      }
      store_row(wsq + slot_rm(i) * slot_stride, h);
#pragma unroll
      for (int k = 0; k < 32; ++k) h[k] = Wb[VTACO_DEC_BLK_B0 + k];
      mv_fwd(h, Wb + VTACO_DEC_BLK_W0, xcol);
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        mh |= (h[k] > 0.f ? 1u : 0u) << k;
        h[k] = fmaxf(h[k], 0.f);
        xcol[k * kBS] = h[k];
      }
      store_row(wsq + slot_rh(nb, i) * slot_stride, h);
      mv_fwd(n, Wb + VTACO_DEC_BLK_W1, xcol);
#pragma unroll
      for (int k = 0; k < 32; ++k) n[k] += Wb[VTACO_DEC_BLK_B1 + k];
      mcol[(2 * i) * kBT] = mm;
      mcol[(2 * i + 1) * kBT] = mh;
    }

    // ---------------- output layer: g = dL/dn_last ----------------
    {
      const float dout = P.dlogits ? __ldg(P.dlogits + q) : 0.f;
      const float dcon = P.dcontact ? __ldg(P.dcontact + q) : 0.f;
#pragma unroll
      for (int k = 0; k < 32; ++k) {
        const bool pos = n[k] > 0.f;
        h[k] = pos ? n[k] : n[k] * slope;
        n[k] = fmaf(dcon, Wo[VTACO_DEC_TAIL_WCON + k], dout * Wo[VTACO_DEC_TAIL_WOUT + k]) * (pos ? 1.f : slope);
      }
      store_row(wsq + slot_aout(nb) * slot_stride, h);
      store_row(wsq + slot_gm(nb, nb) * slot_stride, n);
    }

    // ---------------- backward sweep ----------------
#pragma unroll 1
    for (int i = nb - 1; i >= 0; --i) {
      const float* Wb = sW + VTACO_DEC_OFF_BLOCKS + i * VTACO_DEC_BLOCK_STRIDE;
      const uint32_t mm = mcol[(2 * i) * kBT], mh = mcol[(2 * i + 1) * kBT];
      mv_bwd<false>(xcol, Wb + VTACO_DEC_BLK_W1, n);       // W1^T g
#pragma unroll
      for (int k = 0; k < 32; ++k) h[k] = ((mh >> k) & 1u) ? xcol[k * kBS] : 0.f;
      store_row(wsq + slot_gh(nb, i) * slot_stride, h);
      mv_bwd<false>(xcol, Wb + VTACO_DEC_BLK_W0, h);       // W0^T gh
#pragma unroll
      for (int k = 0; k < 32; ++k) n[k] += ((mm >> k) & 1u) ? xcol[k * kBS] : 0.f;
      store_row(wsq + slot_gm(nb, i) * slot_stride, n);
      if (P.has_c) mv_bwd<true>(dcol, Wb + VTACO_DEC_BLK_WC, n);  // dc += Wc^T g
    }

    // ---------------- d c_img = W_img^T g_0 ----------------
    if (P.use_img && P.c_img && P.d_c_img) {
      mv_bwd<false>(xcol, sW + VTACO_DEC_OFF_WIMG, n);
#pragma unroll
      for (int k = 0; k < 32; ++k) h[k] = xcol[k * kBS];
      store_row(P.d_c_img + (size_t)q * 32, h);
    }

    // ---------------- scatter dc into the feature gradients ----------------
    if (P.has_c) {
      if (P.grid && P.d_grid) {
        int off[8]; float w[8];
        volume_taps(P.Rg, norm3d(px, P.nc), norm3d(py, P.nc), norm3d(pz, P.nc), P.nearest, off, w);
        scatter_taps<8>(P.d_grid + (size_t)b * P.Rg * P.Rg * P.Rg * 32, off, w, dcol);
      }
      const float ux = norm2d(px, P.nc), uy = norm2d(py, P.nc), uz = norm2d(pz, P.nc);
      const size_t boff = (size_t)b * P.Rp * P.Rp * 32;
      int off[4]; float w[4];
      if (P.plane[0] && P.d_plane[0]) { plane_taps(P.Rp, ux, uz, P.nearest, off, w); scatter_taps<4>(P.d_plane[0] + boff, off, w, dcol); }
      if (P.plane[1] && P.d_plane[1]) { plane_taps(P.Rp, ux, uy, P.nearest, off, w); scatter_taps<4>(P.d_plane[1] + boff, off, w, dcol); }
      if (P.plane[2] && P.d_plane[2]) { plane_taps(P.Rp, uy, uz, P.nearest, off, w); scatter_taps<4>(P.d_plane[2] + boff, off, w, dcol); }
    }
  }
}

}  // namespace vtaco

using namespace vtaco;

extern "C" size_t vtaco_decoder_backward_workspace_bytes(int64_t total_queries, int32_t n_blocks) {
  if (total_queries <= 0 || n_blocks <= 0) return 0;
  return (size_t)n_slots(n_blocks) * (size_t)total_queries * 32 * sizeof(float);
}

extern "C" int vtaco_decoder_backward(const vtaco_decoder_bwd_args* a, void* stream_) {
  cudaStream_t stream = (cudaStream_t)stream_;
  if (!a || !a->p || !a->weights || !a->d_params || !a->workspace) return VTACO_ERR_INVALID_ARG;
  if (a->B <= 0 || a->N <= 0) return VTACO_OK;
  if (a->n_blocks < 1 || a->n_blocks > kMaxBlocks) return VTACO_ERR_UNSUPPORTED;
  if (!a->dlogits && !a->dcontact) return VTACO_ERR_INVALID_ARG;
  const bool has_planes = a->plane[0] || a->plane[1] || a->plane[2];
  const bool has_c = a->grid || has_planes;
  if (a->grid && a->reso_grid < 1) return VTACO_ERR_INVALID_ARG;
  if (has_planes && a->reso_plane < 1) return VTACO_ERR_INVALID_ARG;
  const long long Q = (long long)a->B * a->N;
  if (a->workspace_bytes < vtaco_decoder_backward_workspace_bytes(Q, a->n_blocks)) return VTACO_ERR_CAPACITY;
  const int nb = a->n_blocks;

  BwdParams P{};
  P.p = a->p; P.c_img = a->use_img ? a->c_img : nullptr;
  P.grid = a->grid;
  for (int i = 0; i < 3; ++i) { P.plane[i] = a->plane[i]; P.d_plane[i] = a->d_plane[i]; }
  P.weights = a->weights;
  P.dlogits = a->dlogits; P.dcontact = a->dcontact;
  P.ws = static_cast<float*>(a->workspace);
  P.d_grid = a->d_grid; P.d_c_img = a->d_c_img;
  P.Q = Q; P.N = a->N;
  P.Rg = a->reso_grid; P.Rp = a->reso_plane;
  P.n_blocks = nb; P.leaky = a->leaky; P.use_img = a->use_img;
  P.nearest = (a->sample_mode == VTACO_SAMPLE_NEAREST);
  P.has_c = has_c;
  P.wfloats = VTACO_DEC_PACKED_FLOATS(nb);
  P.nc = make_norm_const(a->padding, a->div_mode);

  const size_t smem = ((size_t)P.wfloats + 3 * 32 * kBS) * sizeof(float) + (size_t)2 * nb * kBT * sizeof(uint32_t);
  VTACO_CUDA_CHECK(smem_opt_in((const void*)decoder_bwd_query_kernel, 227 * 1024));
  if (smem > 227 * 1024) return VTACO_ERR_UNSUPPORTED;
  const long long tiles = (Q + kBT - 1) / kBT;
  const int grid = (int)std::min<long long>(tiles, num_sms());
  decoder_bwd_query_kernel<<<grid, kBT, smem, stream>>>(P);
  VTACO_LAUNCH_CHECK();

  // ---- weight / bias gradients (native nn.Linear layout [out][in] at the packed offsets) ----
  WParams W{};
  W.Q = Q;
  int np = 0;
  float* ws = P.ws;
  float* dp = a->d_params;
  const size_t ss = (size_t)Q * 32;
  auto slot = [&](int s) { return ws + (size_t)s * ss; };
  auto add = [&](const float* G, int g_ld, int n_out, const float* A, int a_ld, int n_in, float* dW, int w_ld,
                 float* db) {
    WProd& r = W.prod[np++];
    r.G = G; r.g_ld = g_ld; r.n_out = n_out; r.A = A; r.a_ld = a_ld; r.n_in = n_in; r.dW = dW; r.w_ld = w_ld; r.db = db;
    r.a_relu = 0;
  };
  const float* g0 = slot(slot_gm(nb, 0));
  if (a->use_img) {
    add(g0, 32, 32, a->p, 3, 3, dp + VTACO_DEC_OFF_WPI, 3, dp + VTACO_DEC_OFF_BPI);
    if (P.c_img) add(g0, 32, 32, P.c_img, 32, 32, dp + VTACO_DEC_OFF_WIMG, 32, nullptr);
  } else {
    add(g0, 32, 32, a->p, 3, 3, dp + VTACO_DEC_OFF_WP, 3, dp + VTACO_DEC_OFF_BP);
  }
  for (int i = 0; i < nb; ++i) {
    float* d = dp + VTACO_DEC_OFF_BLOCKS + i * VTACO_DEC_BLOCK_STRIDE;
    if (has_c) add(slot(slot_gm(nb, i)), 32, 32, slot(kSlotC), 32, 32, d + VTACO_DEC_BLK_WC, 32, d + VTACO_DEC_BLK_BC);
    add(slot(slot_gh(nb, i)), 32, 32, slot(slot_rm(i)), 32, 32, d + VTACO_DEC_BLK_W0, 32, d + VTACO_DEC_BLK_B0);
    add(slot(slot_gm(nb, i + 1)), 32, 32, slot(slot_rh(nb, i)), 32, 32, d + VTACO_DEC_BLK_W1, 32, d + VTACO_DEC_BLK_B1);
  }
  float* dt = dp + VTACO_DEC_OFF_BLOCKS + nb * VTACO_DEC_BLOCK_STRIDE;
  if (a->dlogits) add(a->dlogits, 1, 1, slot(slot_aout(nb)), 32, 32, dt + VTACO_DEC_TAIL_WOUT, 32, dt + VTACO_DEC_TAIL_BOUT);
  if (a->dcontact) add(a->dcontact, 1, 1, slot(slot_aout(nb)), 32, 32, dt + VTACO_DEC_TAIL_WCON, 32, dt + VTACO_DEC_TAIL_BCON);
  return launch_wgrad(W, np, stream);
}
