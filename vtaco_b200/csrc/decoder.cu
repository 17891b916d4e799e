// Fused LocalDecoder kernel for sm_100a.
//
// Replaces LocalDecoder.forward / forward_img / forward_contact
// (reference src/conv_onet/models/decoder.py:71-161) and, in dense mode, the
// lattice construction + chunk loop of Generator3D.eval_points
// (src/conv_onet/generation.py:155-157,338-383).
//
// One persistent CTA per SM (256 threads, ~201 KB of shared memory):
//   * all MLP weights (68.7 KB, K-major) are staged in shared memory once;
//   * a tile is 512 queries (dense mode: an 8x8x8 brick of the lattice, so the
//     interpolation taps of neighbouring queries hit the same L1 lines);
//   * gather phase: 8 lanes x float4 cover the 32 channels of one tap (one 128 B
//     line of the channels-last feature tensor); 4 queries per warp instruction;
//     results go to the per-query column sC[k][q];
//   * MLP phase: each thread owns 2 queries; the residual stream and the layer
//     accumulators stay in registers (2 x 32 + 2 x 32 floats), layer inputs are
//     read from the thread's private shared-memory column, weights arrive as
//     broadcast LDS.128 — 64 FMAs per 10 shared loads; no block-level barrier in
//     the loop (warps drift so gathers overlap the FMA-bound MLP of other warps).
// HBM traffic per query: 12 B in (flat mode) or 0 (dense), 4 B out.
#include "decoder_common.cuh"

namespace vtaco {

int launch_decoder_tc(DecParams P, bool dense, const float* wtc, cudaStream_t stream);  // decoder_tc.cu
int launch_decoder_tc4(DecParams P, bool dense, const float* wtc, cudaStream_t stream);  // decoder_tc4.cu

// acc[s][j] += sum_k W[k][j] * X[k][q_s]  for the thread's two queries.
// W: shared, K-major [32][32] (broadcast LDS.128); X: shared column base.
template <bool F2>
__device__ __forceinline__ void matvec(float2 (&a)[2][16], const float* __restrict__ W,
                                       const float* __restrict__ xcol) {
#pragma unroll 4
  for (int k = 0; k < 32; ++k) {
    const float x0 = xcol[k * kSC];
    const float x1 = xcol[k * kSC + kThreads];
    const float4* w4 = reinterpret_cast<const float4*>(W + k * 32);
    if (F2) {
      const float2 xx0 = make_float2(x0, x0), xx1 = make_float2(x1, x1);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 w = w4[j];
        const float2 wl = make_float2(w.x, w.y), wh = make_float2(w.z, w.w);
        a[0][2 * j] = __ffma2_rn(wl, xx0, a[0][2 * j]);
        a[0][2 * j + 1] = __ffma2_rn(wh, xx0, a[0][2 * j + 1]);
        a[1][2 * j] = __ffma2_rn(wl, xx1, a[1][2 * j]);
        a[1][2 * j + 1] = __ffma2_rn(wh, xx1, a[1][2 * j + 1]);
      }
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 w = w4[j];
        a[0][2 * j].x = fmaf(w.x, x0, a[0][2 * j].x);
        a[0][2 * j].y = fmaf(w.y, x0, a[0][2 * j].y);
        a[0][2 * j + 1].x = fmaf(w.z, x0, a[0][2 * j + 1].x);
        a[0][2 * j + 1].y = fmaf(w.w, x0, a[0][2 * j + 1].y);
        a[1][2 * j].x = fmaf(w.x, x1, a[1][2 * j].x);
        a[1][2 * j].y = fmaf(w.y, x1, a[1][2 * j].y);
        a[1][2 * j + 1].x = fmaf(w.z, x1, a[1][2 * j + 1].x);
        a[1][2 * j + 1].y = fmaf(w.w, x1, a[1][2 * j + 1].y);
      }
    }
  }
}

__device__ __forceinline__ void add_bias(float2 (&a)[2][16], const float* __restrict__ b) {
  const float2* b2 = reinterpret_cast<const float2*>(b);
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float2 v = b2[j];
    a[0][j].x += v.x; a[0][j].y += v.y;
    a[1][j].x += v.x; a[1][j].y += v.y;
  }
}
__device__ __forceinline__ void set_bias(float2 (&a)[2][16], const float* __restrict__ b) {
  const float2* b2 = reinterpret_cast<const float2*>(b);
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    const float2 v = b2[j];
    a[0][j] = v; a[1][j] = v;
  }
}
// X[k][q_s] = relu(a[s][k])
__device__ __forceinline__ void store_relu(const float2 (&a)[2][16], float* __restrict__ xcol) {
#pragma unroll
  for (int j = 0; j < 16; ++j) {
    xcol[(2 * j) * kSC] = fmaxf(a[0][j].x, 0.f);
    xcol[(2 * j + 1) * kSC] = fmaxf(a[0][j].y, 0.f);
    xcol[(2 * j) * kSC + kThreads] = fmaxf(a[1][j].x, 0.f);
    xcol[(2 * j + 1) * kSC + kThreads] = fmaxf(a[1][j].y, 0.f);
  }
}

template <bool DENSE, bool F2>
__global__ void __launch_bounds__(kThreads, 1) decoder_kernel(const __grid_constant__ DecParams P) {
  extern __shared__ __align__(16) float smem[];
  float* sW = smem;
  float* sC = sW + P.wfloats;
  float* sX = sC + 32 * kSC;
  float* sTip = sX + 32 * kSC;

  for (int i = threadIdx.x; i < P.wfloats / 4; i += kThreads)
    reinterpret_cast<float4*>(sW)[i] = __ldg(reinterpret_cast<const float4*>(P.weights) + i);
  __syncthreads();
  if (P.n_tips > 0) {  // fc_p_img.weight[:, 3:] @ tip_feat[f]
    for (int o = threadIdx.x; o < P.n_tips * 32; o += kThreads) {
      const int f = o >> 5, j = o & 31;
      float a = 0.f;
      for (int k = 0; k < 32; ++k) a = fmaf(sW[VTACO_DEC_OFF_WIMG + k * 32 + j], __ldg(P.tip_feat + f * 32 + k), a);
      sTip[o] = a;
    }
    __syncthreads();
  }

  const int lane = threadIdx.x & 31, wbase = threadIdx.x & ~31;
  const int grp = lane >> 3, sub = lane & 7;
  const int nx = P.nx;
  float vmin = CUDART_INF_F, vmax = -CUDART_INF_F;

  for (long long tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x) {
    // ---------------- coordinates of the two queries this thread owns ----------------
    float px[2], py[2], pz[2];
    long long oidx[2];
    int qb[2];
    bool valid[2];
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const int q = s * kThreads + threadIdx.x;
      if (DENSE) {
        long long t = tile;
        const int bz = (int)(t % P.nby); t /= P.nby;
        const int by = (int)(t % P.nby); t /= P.nby;
        const int bx = (int)(t % P.nbx);
        const int b = (int)(t / P.nbx);
        const int ix = P.x0 + bx * 8 + (q >> 6), iy = by * 8 + ((q >> 3) & 7), iz = bz * 8 + (q & 7);
        valid[s] = (ix < P.x1) && (iy < nx) && (iz < nx);
        px[s] = __ldg(P.axis + min(ix, nx - 1));
        py[s] = __ldg(P.axis + min(iy, nx - 1));
        pz[s] = __ldg(P.axis + min(iz, nx - 1));
        qb[s] = b;
        oidx[s] = (((long long)b * nx + ix) * nx + iy) * nx + iz;
      } else {
        const long long n = tile * kTileQ + q;
        valid[s] = n < P.total;
        const long long nn = valid[s] ? n : 0;
        px[s] = __ldg(P.p + nn * 3 + 0);
        py[s] = __ldg(P.p + nn * 3 + 1);
        pz[s] = __ldg(P.p + nn * 3 + 2);
        qb[s] = (int)(nn / P.N);
        oidx[s] = nn;
      }
      if (!valid[s]) oidx[s] = 0;
    }

    // ---------------- gather phase: 8 lanes per query, 4 queries per step ----------------
    if (P.has_c || (P.use_img && P.c_img)) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
#pragma unroll 2
        for (int it = 0; it < 8; ++it) {
          const int src = it * 4 + grp;
          const float x = __shfl_sync(kFull, px[s], src);
          const float y = __shfl_sync(kFull, py[s], src);
          const float z = __shfl_sync(kFull, pz[s], src);
          const int b = __shfl_sync(kFull, qb[s], src);
          const int q = s * kThreads + wbase + src;
          if (P.has_c) {
            const float4 c = sample_feature_sum(P, b, sub, x, y, z);
            float* dst = sC + (4 * sub) * kSC + q;
            dst[0] = c.x; dst[kSC] = c.y; dst[2 * kSC] = c.z; dst[3 * kSC] = c.w;
          }
          if (P.use_img && P.c_img) {
            const unsigned lo = __shfl_sync(kFull, (unsigned)(oidx[s] & 0xffffffffll), src);
            const unsigned hi = __shfl_sync(kFull, (unsigned)(oidx[s] >> 32), src);
            const long long row = ((long long)hi << 32) | lo;
            const float4 ci = __ldg(reinterpret_cast<const float4*>(P.c_img) + row * 8 + sub);
            float* dst = sX + (4 * sub) * kSC + q;
            dst[0] = ci.x; dst[kSC] = ci.y; dst[2 * kSC] = ci.z; dst[3 * kSC] = ci.w;
          }
        }
      }
    }
    __syncwarp();

    // ---------------- MLP phase: 2 queries per thread ----------------
    float2 net[2][16], acc[2][16];
    const float* ccol = sC + threadIdx.x;
    float* xcol = sX + threadIdx.x;
    {
      const float* Wp = sW + (P.use_img ? VTACO_DEC_OFF_WPI : VTACO_DEC_OFF_WP);
      const float2* w0 = reinterpret_cast<const float2*>(Wp);
      const float2* w1 = reinterpret_cast<const float2*>(Wp + 32);
      const float2* w2 = reinterpret_cast<const float2*>(Wp + 64);
      const float2* bp = reinterpret_cast<const float2*>(Wp + (VTACO_DEC_OFF_BP - VTACO_DEC_OFF_WP));  // = BPI - WPI
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float2 a0 = w0[j], a1 = w1[j], a2 = w2[j], bb = bp[j];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          net[s][j].x = fmaf(a2.x, pz[s], fmaf(a1.x, py[s], fmaf(a0.x, px[s], bb.x)));
          net[s][j].y = fmaf(a2.y, pz[s], fmaf(a1.y, py[s], fmaf(a0.y, px[s], bb.y)));
        }
      }
    }
    if (P.use_img && P.c_img) matvec<F2>(net, sW + VTACO_DEC_OFF_WIMG, xcol);
    if (P.use_img && P.n_tips > 0) {
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        const int f = tip_assign(P, px[s], py[s], pz[s]);
        if (f >= 0) {
          const float2* t2 = reinterpret_cast<const float2*>(sTip + f * 32);
#pragma unroll
          for (int j = 0; j < 16; ++j) { const float2 v = t2[j]; net[s][j].x += v.x; net[s][j].y += v.y; }
        }
      }
    }
    for (int i = 0; i < P.n_blocks; ++i) {
      const float* Wb = sW + VTACO_DEC_OFF_BLOCKS + i * VTACO_DEC_BLOCK_STRIDE;
      if (P.has_c) {  // net = net + fc_c[i](c)                       decoder.py:92-94
        matvec<F2>(net, Wb + VTACO_DEC_BLK_WC, ccol);
        add_bias(net, Wb + VTACO_DEC_BLK_BC);
      }
      store_relu(net, xcol);            // ResnetBlockFC: fc_0(relu(x))     layers.py:42
      set_bias(acc, Wb + VTACO_DEC_BLK_B0);
      matvec<F2>(acc, Wb + VTACO_DEC_BLK_W0, xcol);
      store_relu(acc, xcol);            // fc_1(relu(net))                  layers.py:43
      matvec<F2>(net, Wb + VTACO_DEC_BLK_W1, xcol);
      add_bias(net, Wb + VTACO_DEC_BLK_B1);  // x_s + dx (identity shortcut)     layers.py:45-50
    }
    {
      const float* Wo = sW + VTACO_DEC_OFF_BLOCKS + P.n_blocks * VTACO_DEC_BLOCK_STRIDE;
      const float slope = P.leaky ? 0.2f : 0.0f;
      float o[2] = {Wo[VTACO_DEC_TAIL_BOUT], Wo[VTACO_DEC_TAIL_BOUT]};
      float oc[2] = {Wo[VTACO_DEC_TAIL_BCON], Wo[VTACO_DEC_TAIL_BCON]};
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        const float2 w = reinterpret_cast<const float2*>(Wo + VTACO_DEC_TAIL_WOUT)[j];
        const float2 wc = reinterpret_cast<const float2*>(Wo + VTACO_DEC_TAIL_WCON)[j];
#pragma unroll
        for (int s = 0; s < 2; ++s) {
          const float ax = net[s][j].x > 0.f ? net[s][j].x : net[s][j].x * slope;
          const float ay = net[s][j].y > 0.f ? net[s][j].y : net[s][j].y * slope;
          o[s] = fmaf(w.y, ay, fmaf(w.x, ax, o[s]));
          oc[s] = fmaf(wc.y, ay, fmaf(wc.x, ax, oc[s]));
        }
      }
#pragma unroll
      for (int s = 0; s < 2; ++s) {
        if (valid[s]) {
          store_logit(P, oidx[s], o[s]);
          if (P.contact) P.contact[oidx[s]] = oc[s];
          vmin = fminf(vmin, o[s]);
          vmax = fmaxf(vmax, o[s]);
        }
      }
    }
    __syncwarp();
  }

  flush_minmax(P, vmin, vmax, lane);
}

// Gather-only kernel behind LocalDecoder.sample_plane_feature / sample_grid_feature
// (reference decoder.py:55-68): out [B][32][N], 8 lanes per query.
__global__ void __launch_bounds__(256) sample_features_kernel(const __grid_constant__ DecParams P,
                                                              float* __restrict__ out) {
  const int sub = threadIdx.x & 7;
  const long long stride = ((long long)gridDim.x * blockDim.x) >> 3;
  for (long long n = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 3; n < P.total; n += stride) {
    const float x = __ldg(P.p + n * 3), y = __ldg(P.p + n * 3 + 1), z = __ldg(P.p + n * 3 + 2);
    const int b = (int)(n / P.N);
    const long long i = n - (long long)b * P.N;
    const float4 c = sample_feature_sum(P, b, sub, x, y, z);
    float* o = out + ((size_t)b * 32 + 4 * sub) * P.N + i;
    o[0] = c.x; o[P.N] = c.y; o[2 * P.N] = c.z; o[3 * P.N] = c.w;
  }
}

// ---------------------------------------------------------------------------------------
// channels-first <-> channels-last relayout: [B][C][S] <-> [B][S][C], 32x32 tiles via smem
// ---------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) transpose_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                        int rows, long long cols) {
  // src [rows][cols] -> dst [cols][rows] per batch (blockIdx.z)
  __shared__ float tile[32][33];
  const size_t boff = (size_t)blockIdx.z * rows * cols;
  const long long c0 = (long long)blockIdx.x * 32;
  const int r0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int r = r0 + ty + i;
    const long long c = c0 + tx;
    if (r < rows && c < cols) tile[ty + i][tx] = src[boff + (size_t)r * cols + c];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const long long c = c0 + ty + i;
    const int r = r0 + tx;
    if (r < rows && c < cols) dst[boff + (size_t)c * rows + r] = tile[tx][ty + i];
  }
}

static int launch_transpose(const float* src, float* dst, int B, long long rows, long long cols, void* stream) {
  if (!src || !dst || B <= 0 || rows <= 0 || cols <= 0) return VTACO_ERR_INVALID_ARG;
  // grid.x carries the long dimension
  if (cols >= rows) {
    dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((rows + 31) / 32), (unsigned)B);
    if (grid.y > 65535 || grid.z > 65535) return VTACO_ERR_UNSUPPORTED;
    transpose_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, (int)rows, cols);
  } else {
    return VTACO_ERR_UNSUPPORTED;
  }
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

// [S][C] -> [C][S]: rows = S is the long dimension; dedicated kernel with grid.x over rows
__global__ void __launch_bounds__(256) transpose_tall_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                             long long rows, int cols) {
  __shared__ float tile[32][33];
  const size_t boff = (size_t)blockIdx.z * rows * cols;
  const long long r0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const long long r = r0 + ty + i;
    const int c = c0 + tx;
    if (r < rows && c < cols) tile[ty + i][tx] = src[boff + (size_t)r * cols + c];
  }
  __syncthreads();
#pragma unroll
  for (int i = 0; i < 32; i += 8) {
    const int c = c0 + ty + i;
    const long long r = r0 + tx;
    if (r < rows && c < cols) dst[boff + (size_t)c * rows + r] = tile[tx][ty + i];
  }
}

}  // namespace vtaco

using namespace vtaco;

extern "C" int vtaco_relayout_cl(const float* src, float* dst, int B, int C, int64_t S, void* stream) {
  if (C <= 0 || S <= 0) return VTACO_ERR_INVALID_ARG;
  if (S >= C) return launch_transpose(src, dst, B, C, S, stream);
  // degenerate tiny spatial extent
  if (!src || !dst || B <= 0) return VTACO_ERR_INVALID_ARG;
  dim3 grid((unsigned)((C + 31) / 32), (unsigned)((S + 31) / 32), (unsigned)B);
  transpose_tall_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, C, (int)S);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_relayout_cf(const float* src, float* dst, int B, int C, int64_t S, void* stream) {
  if (!src || !dst || B <= 0 || C <= 0 || S <= 0) return VTACO_ERR_INVALID_ARG;
  dim3 grid((unsigned)((S + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B);
  if (grid.y > 65535 || grid.z > 65535) return VTACO_ERR_UNSUPPORTED;
  transpose_tall_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(src, dst, (long long)S, C);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

// the SIMT kernel's shared memory: packed weights, the two per-query column blocks, the fingertip table
static size_t simt_smem_bytes(int n_blocks) {
  return ((size_t)VTACO_DEC_PACKED_FLOATS(n_blocks) + 2 * 32 * kSC + VTACO_MAX_TIPS * 32) * sizeof(float);
}

template <bool DENSE, bool F2>
static int launch_decoder(const DecParams& P, cudaStream_t stream) {
  const size_t smem_bytes = simt_smem_bytes(P.n_blocks);
  VTACO_CUDA_CHECK(smem_opt_in((const void*)decoder_kernel<DENSE, F2>, smem_bytes));
  const long long grid = P.n_tiles < (long long)num_sms() ? P.n_tiles : (long long)num_sms();
  decoder_kernel<DENSE, F2><<<(unsigned)grid, kThreads, smem_bytes, stream>>>(P);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

int vtaco::launch_decoder_simt(const DecParams& P, bool dense, cudaStream_t stream) {
  if (P.tip_map) return VTACO_ERR_UNSUPPORTED;   // the byte map is read by the tcgen05 kernels only
  return dense ? launch_decoder<true, true>(P, stream) : launch_decoder<false, true>(P, stream);
}

extern "C" int vtaco_decoder_forward(const vtaco_decoder_args* a, void* stream) {
  if (!a || !a->weights || !a->logits) return VTACO_ERR_INVALID_ARG;
  if (a->B <= 0 || a->n_blocks < 0) return VTACO_ERR_INVALID_ARG;
  if (a->sample_mode != VTACO_SAMPLE_BILINEAR && a->sample_mode != VTACO_SAMPLE_NEAREST) return VTACO_ERR_INVALID_ARG;
  if (a->div_mode != VTACO_DIV_RECIPROCAL && a->div_mode != VTACO_DIV_TRUE) return VTACO_ERR_INVALID_ARG;
  if (a->n_tips < 0 || a->n_tips > VTACO_MAX_TIPS) return VTACO_ERR_INVALID_ARG;
  const bool dense = (a->p == nullptr);
  DecParams P;
  P.p = a->p; P.axis = a->axis; P.grid = a->grid;
  for (int i = 0; i < 3; ++i) P.plane[i] = a->plane[i];
  P.weights = a->weights; P.c_img = a->c_img; P.tip_feat = a->tip_feat; P.tip_map = a->tip_map;
  if (a->tip_map && !(a->variant >= 2 && a->variant <= 7)) return VTACO_ERR_UNSUPPORTED;   // byte map: tcgen05 kernels only
  P.logits = a->logits; P.contact = a->contact; P.minmax_key = a->minmax_key;
  P.B = a->B; P.Rg = a->reso_grid; P.Rp = a->reso_plane;
  P.n_blocks = a->n_blocks; P.leaky = a->leaky ? 1 : 0; P.use_img = a->use_img ? 1 : 0;
  P.nearest = (a->sample_mode == VTACO_SAMPLE_NEAREST);
  // features enter the network only through the blocks' fc_c (decoder.py:92-94): none without blocks
  P.has_c = (a->n_blocks > 0 && (a->grid || a->plane[0] || a->plane[1] || a->plane[2])) ? 1 : 0;
  if (a->grid && a->reso_grid < 1) return VTACO_ERR_INVALID_ARG;
  if ((a->plane[0] || a->plane[1] || a->plane[2]) && a->reso_plane < 1) return VTACO_ERR_INVALID_ARG;
  P.n_tips = P.use_img ? a->n_tips : 0;
  if (P.n_tips > 0 && !a->tip_feat) return VTACO_ERR_INVALID_ARG;
  if (P.use_img && !a->c_img && P.n_tips == 0) { /* c_img == 0 everywhere */ }
  for (int f = 0; f < VTACO_MAX_TIPS; ++f) {
    for (int d = 0; d < 3; ++d) {
      P.tips[f][d] = f < P.n_tips ? a->tips[f][d] : 0.0;
      P.tipsf[f][d] = (float)P.tips[f][d];
    }
    P.tip_touch[f] = f < P.n_tips ? a->tip_touch[f] : 0;
  }
  P.tip_radius = a->tip_radius;
  // per-sample tip tables: byte-map form only (the ids select the row), tcgen05 kernels only (the SIMT launcher
  // refuses a byte map)
  if (a->tip_feat_per_sample && (!a->tip_map || !(a->variant >= 2 && a->variant <= 7))) return VTACO_ERR_UNSUPPORTED;
  P.tip_ps = (a->tip_feat_per_sample && P.n_tips > 0) ? 1 : 0;
  P.tip_r2_hi = tip_prefilter_r2(a->tip_radius);
  P.nc = make_norm_const(a->padding, a->div_mode);
  P.wfloats = VTACO_DEC_PACKED_FLOATS(a->n_blocks);
  if (P.wfloats % 4) return VTACO_ERR_UNSUPPORTED;
  if (simt_smem_bytes(a->n_blocks) > 227 * 1024) return VTACO_ERR_UNSUPPORTED;  // n_blocks too large for one SM
  if (dense) {
    if (!a->axis || a->nx < 1 || a->x0 < 0 || a->x1 > a->nx || a->x0 >= a->x1) return VTACO_ERR_INVALID_ARG;
    P.nx = a->nx; P.x0 = a->x0; P.x1 = a->x1;
    P.nbx = (a->x1 - a->x0 + 7) / 8;
    P.nby = (a->nx + 7) / 8;
    P.N = (long long)a->nx * a->nx * a->nx;
    P.total = P.N * a->B;
    P.n_tiles = (long long)a->B * P.nbx * P.nby * P.nby;
  } else {
    if (a->N <= 0) return VTACO_ERR_INVALID_ARG;
    P.nx = 0; P.x0 = P.x1 = 0; P.nbx = P.nby = 1;
    P.N = a->N;
    P.total = (long long)a->B * a->N;
    P.n_tiles = (P.total + kTileQ - 1) / kTileQ;
  }
  cudaStream_t st = (cudaStream_t)stream;
  P.t_nbx = P.t_nby = P.t_nbz = P.t_xend = 0;
  P.n_peers = 0;
  P.mcast = nullptr;
  if (a->n_peers < 0 || a->n_peers > 8) return VTACO_ERR_INVALID_ARG;
  if (a->n_peers > 0) {
    if (!dense) return VTACO_ERR_UNSUPPORTED;
    P.n_peers = a->n_peers;
    for (int r = 0; r < a->n_peers; ++r) {
      if (!a->logits_peers[r]) return VTACO_ERR_INVALID_ARG;
      P.peers[r] = a->logits_peers[r];
    }
    P.mcast = a->logits_multicast;
  }
  P.tc_products = (a->variant == 3) ? 1 : (VTACO_DEC_TC_MODE(a->variant) == VTACO_DEC_TC_MODE_BF16) ? 2 : 3;
  P.tc_split = (a->variant == 5 || a->variant == 6) ? 2 : 1;
  if (a->variant == 7) return launch_decoder_tc4(P, dense, a->weights_tc, st);
  if (a->variant >= 2 && a->variant <= 6) return launch_decoder_tc(P, dense, a->weights_tc, st);
  const bool f2 = (a->variant == 1);
  if (dense) return f2 ? launch_decoder<true, true>(P, st) : launch_decoder<true, false>(P, st);
  return f2 ? launch_decoder<false, true>(P, st) : launch_decoder<false, false>(P, st);
}

extern "C" float vtaco_key_to_float_host(int32_t key) { return key_to_float(key); }

extern "C" int vtaco_sample_features(const vtaco_decoder_args* a, const float* p, int64_t N, float* out, void* stream) {
  if (!a || !p || !out || a->B <= 0 || N <= 0) return VTACO_ERR_INVALID_ARG;
  if (!(a->grid || a->plane[0] || a->plane[1] || a->plane[2])) return VTACO_ERR_INVALID_ARG;
  DecParams P = {};
  P.p = p; P.grid = a->grid;
  for (int i = 0; i < 3; ++i) P.plane[i] = a->plane[i];
  P.B = a->B; P.N = N; P.total = (long long)a->B * N;
  P.Rg = a->reso_grid; P.Rp = a->reso_plane;
  P.nearest = (a->sample_mode == VTACO_SAMPLE_NEAREST);
  P.nc = make_norm_const(a->padding, a->div_mode);
  long long blocks = (P.total * 8 + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  sample_features_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(P, out);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}
