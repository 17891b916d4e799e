// Weight / bias gradients of the per-query (decoder) and per-point (encoder) linear layers:
//   dW[o][k] += sum_q G[q][o] * A[q][k];   db[o] += sum_q G[q][o]
// G = gradients at the layer outputs, A = layer inputs, both stored as rows per query.
// One CTA per (product, query chunk): 128-row tiles staged in shared memory, the 32x32
// outer-product accumulators spread over 256 threads (4 per thread), one atomicAdd per
// element and CTA.  Matrices wider than 32 are split into several products by the caller
// (pointer offsets + leading dimensions).
#pragma once
#include "common.cuh"
#include <algorithm>

namespace vtaco {

constexpr int kMaxProd = 32;
constexpr int kWTile = 128;

struct WProd {
  const float* G;   // rows of g_ld floats, n_out (<= 32) used
  const float* A;   // rows of a_ld floats, n_in (<= 32) used
  float* dW;        // [n_out][w_ld], accumulated into
  float* db;        // [n_out] or NULL
  int g_ld, n_out, a_ld, n_in, w_ld;
  int a_relu;       // use max(A, 0) (layer input was relu(A))
};
struct WParams {
  WProd prod[kMaxProd];
  long long Q;
  int q_per_cta;
  int list[kMaxProd];   // product indices a launch covers (blockIdx.y -> product): the 32x32 ones go to the fast kernel
};

static __global__ void __launch_bounds__(256) linear_wgrad_kernel(const __grid_constant__ WParams P) {
  __shared__ __align__(16) float sG[kWTile][32];
  __shared__ __align__(16) float sA[kWTile][32];
  const WProd& pr = P.prod[P.list[blockIdx.y]];
  const long long q_begin = (long long)blockIdx.x * P.q_per_cta;
  const long long q_end = min(P.Q, q_begin + P.q_per_cta);
  const int o = threadIdx.x >> 3, k4 = threadIdx.x & 7;
  float acc[4] = {0.f, 0.f, 0.f, 0.f};
  float bsum = 0.f;
  for (long long q0 = q_begin; q0 < q_end; q0 += kWTile) {
    const int nq = (int)min((long long)kWTile, q_end - q0);
    __syncthreads();
#pragma unroll 4
    for (int idx = threadIdx.x; idx < kWTile * 32; idx += 256) {
      const int r = idx >> 5, c = idx & 31;
      float g = 0.f, a = 0.f;
      if (r < nq) {
        if (c < pr.n_out) g = __ldg(pr.G + (size_t)(q0 + r) * pr.g_ld + c);
        if (c < pr.n_in) a = __ldg(pr.A + (size_t)(q0 + r) * pr.a_ld + c);
        if (pr.a_relu) a = fmaxf(a, 0.f);
      }
      sG[r][c] = g;
      sA[r][c] = a;
    }
    __syncthreads();
#pragma unroll 8
    for (int r = 0; r < kWTile; ++r) {   // rows beyond nq are zero
      const float g = sG[r][o];
      const float4 a = *reinterpret_cast<const float4*>(&sA[r][4 * k4]);
      acc[0] = fmaf(g, a.x, acc[0]);
      acc[1] = fmaf(g, a.y, acc[1]);
      acc[2] = fmaf(g, a.z, acc[2]);
      acc[3] = fmaf(g, a.w, acc[3]);
      bsum += g;
    }
  }
  if (o < pr.n_out) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int k = 4 * k4 + e;
      if (k < pr.n_in) atomicAdd(pr.dW + (size_t)o * pr.w_ld + k, acc[e]);
    }
    if (pr.db && k4 == 0) atomicAdd(pr.db + o, bsum);
  }
}

// ---- fast path: full 32 x 32 products with 16-byte aligned rows (every hidden layer) ----
// The generic kernel above loads a tile with scalar loads, waits, computes, and repeats: ncu at the training shape
// (18 products x 65 536 queries) shows long-scoreboard stalls of 7.4 warps per issue and 276 us for 2.4 GFLOP.
// Here the next tile arrives by cp.async (16-byte chunks, zero-filled past the end) while the current one is
// reduced, a thread owns a 4 x 4 block of the outer product (two 16-byte shared loads per 16 FMAs, issued as
// packed FFMA2) over a quarter of the tile's rows, and the four row groups meet in shared memory before one
// atomicAdd per element and CTA.
constexpr int kW32Stage = kWTile * 32 * 2;     // floats per stage: G tile | A tile

__device__ __forceinline__ void wgrad_cp16(float* dst_smem, const float* src, bool valid) {
  const unsigned d = (unsigned)__cvta_generic_to_shared(dst_smem);
  const int bytes = valid ? 16 : 0;              // src-size 0: the 16 destination bytes are zero-filled
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(bytes) : "memory");
}

static __global__ void __launch_bounds__(256) linear_wgrad32_kernel(const __grid_constant__ WParams P) {
  extern __shared__ __align__(16) float wsm[];   // 2 stages
  const WProd& pr = P.prod[P.list[blockIdx.y]];
  const long long q_begin = (long long)blockIdx.x * P.q_per_cta;
  const long long q_end = min(P.Q, q_begin + P.q_per_cta);
  const int tid = threadIdx.x;
  const int og = tid & 7, kg = (tid >> 3) & 7, rg = tid >> 6;
  const int n_tiles = (int)((q_end - q_begin + kWTile - 1) / kWTile);
  auto load_tile = [&](int t, int stage) {
    float* sG = wsm + stage * kW32Stage;
    float* sA = sG + kWTile * 32;
    const long long q0 = q_begin + (long long)t * kWTile;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int idx = tid + j * 256, r = idx >> 3, c4 = idx & 7;
      const bool ok = q0 + r < q_end;
      const long long row = ok ? q0 + r : q_begin;
      wgrad_cp16(sG + r * 32 + 4 * c4, pr.G + (size_t)row * pr.g_ld + 4 * c4, ok);
      wgrad_cp16(sA + r * 32 + 4 * c4, pr.A + (size_t)row * pr.a_ld + 4 * c4, ok);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  float2 acc[4][2];
  float bsum[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int i = 0; i < 4; ++i) acc[i][0] = acc[i][1] = make_float2(0.f, 0.f);
  if (n_tiles > 0) load_tile(0, 0);
  for (int t = 0; t < n_tiles; ++t) {
    const int stage = t & 1;
    if (t + 1 < n_tiles) {
      load_tile(t + 1, stage ^ 1);
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const float* sG = wsm + stage * kW32Stage + rg * 32 * 32;
    const float* sA = wsm + stage * kW32Stage + kWTile * 32 + rg * 32 * 32;
#pragma unroll 8
    for (int r = 0; r < 32; ++r) {   // rows beyond the end are zero
      const float4 g = *reinterpret_cast<const float4*>(sG + r * 32 + 4 * og);
      float4 a = *reinterpret_cast<const float4*>(sA + r * 32 + 4 * kg);
      if (pr.a_relu) { a.x = fmaxf(a.x, 0.f); a.y = fmaxf(a.y, 0.f); a.z = fmaxf(a.z, 0.f); a.w = fmaxf(a.w, 0.f); }
      const float2 a01 = make_float2(a.x, a.y), a23 = make_float2(a.z, a.w);
      const float gs[4] = {g.x, g.y, g.z, g.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 gg = make_float2(gs[i], gs[i]);
        acc[i][0] = __ffma2_rn(a01, gg, acc[i][0]);
        acc[i][1] = __ffma2_rn(a23, gg, acc[i][1]);
        bsum[i] += gs[i];
      }
    }
    __syncthreads();   // the stage is refilled by the next iteration's prefetch
  }
  // ---- the four row groups meet in shared memory: [rg][o][k] and [rg][o] ----
  float* red = wsm;                       // 4 x 1024 floats
  float* redb = wsm + 4 * 1024;           // 4 x 32 floats
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float* d = red + rg * 1024 + (4 * og + i) * 32 + 4 * kg;
    *reinterpret_cast<float4*>(d) = make_float4(acc[i][0].x, acc[i][0].y, acc[i][1].x, acc[i][1].y);
    if (kg == 0) redb[rg * 32 + 4 * og + i] = bsum[i];
  }
  __syncthreads();
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int e = tid + j * 256, o = e >> 5, k = e & 31;
    const float v = (red[e] + red[1024 + e]) + (red[2048 + e] + red[3072 + e]);
    atomicAdd(pr.dW + (size_t)o * pr.w_ld + k, v);
  }
  if (pr.db && tid < 32) atomicAdd(pr.db + tid, (redb[tid] + redb[32 + tid]) + (redb[64 + tid] + redb[96 + tid]));
}

static inline void wgrad_add(WParams& W, int& np, const float* G, int g_ld, int n_out, const float* A, int a_ld,
                             int n_in, float* dW, int w_ld, float* db, int a_relu = 0) {
  WProd& r = W.prod[np++];
  r.G = G; r.g_ld = g_ld; r.n_out = n_out; r.A = A; r.a_ld = a_ld; r.n_in = n_in;
  r.dW = dW; r.w_ld = w_ld; r.db = db; r.a_relu = a_relu;
}

// launch `np` products over W.Q rows, ~8 CTAs per SM over all products; full 32 x 32 products with aligned rows
// take the fast kernel
static inline int launch_wgrad(WParams& W, int np, cudaStream_t stream) {
  if (np <= 0 || W.Q <= 0) return VTACO_OK;
  if (np > kMaxProd) return VTACO_ERR_UNSUPPORTED;
  const long long Q = W.Q;
  const long long want = (long long)num_sms() * 8 / np + 1;
  long long chunks = std::min<long long>((Q + kWTile - 1) / kWTile, want);
  if (chunks < 1) chunks = 1;
  long long per = (Q + chunks - 1) / chunks;
  per = (per + kWTile - 1) / kWTile * kWTile;
  W.q_per_cta = (int)per;
  chunks = (Q + per - 1) / per;
  int fast[kMaxProd], slow[kMaxProd], nf = 0, ns = 0;
  for (int i = 0; i < np; ++i) {
    const WProd& r = W.prod[i];
    const bool f = r.n_out == 32 && r.n_in == 32 && (r.g_ld & 3) == 0 && (r.a_ld & 3) == 0 &&
                   (reinterpret_cast<uintptr_t>(r.G) & 15) == 0 && (reinterpret_cast<uintptr_t>(r.A) & 15) == 0;
    if (f) fast[nf++] = i; else slow[ns++] = i;
  }
  if (nf > 0) {
    constexpr int smem = 2 * kW32Stage * (int)sizeof(float);
    VTACO_CUDA_CHECK(smem_opt_in((const void*)linear_wgrad32_kernel, smem));
    for (int i = 0; i < nf; ++i) W.list[i] = fast[i];
    linear_wgrad32_kernel<<<dim3((unsigned)chunks, (unsigned)nf), 256, smem, stream>>>(W);
    VTACO_LAUNCH_CHECK();
  }
  if (ns > 0) {
    // the few narrow products (3-wide input layer, 1-wide heads): their own chunking, ~8 CTAs per SM over them, so that
    // a CTA walks one or two tiles instead of eight (the generic kernel is latency-bound per tile: 99 -> ~20 us)
    const long long want_s = (long long)num_sms() * 8 / ns + 1;
    long long chunks_s = std::min<long long>((Q + kWTile - 1) / kWTile, want_s);
    if (chunks_s < 1) chunks_s = 1;
    long long per_s = (Q + chunks_s - 1) / chunks_s;
    per_s = (per_s + kWTile - 1) / kWTile * kWTile;
    W.q_per_cta = (int)per_s;
    chunks_s = (Q + per_s - 1) / per_s;
    for (int i = 0; i < ns; ++i) W.list[i] = slow[i];
    linear_wgrad_kernel<<<dim3((unsigned)chunks_s, (unsigned)ns), 256, 0, stream>>>(W);
    VTACO_LAUNCH_CHECK();
  }
  return VTACO_OK;
}

}  // namespace vtaco
