// LocalPoolPointnet (PointNet part) for sm_100a.
//
// Replaces reference src/encoder/pointnet.py:135-172 (forward), :116-132 (pool_local),
// :85-114 (generate_plane_features / generate_grid_features before the UNets) and the
// torch_scatter scatter_max / scatter_mean kernels they call.
//
// Design
//  * point -> cell once per key (int32), then cell -> SLOT compaction: the lowest point
//    id that falls into a cell (atomicMin on a dense int32 map) represents the cell, so
//    every pooling buffer is [points][32] instead of [R^3][32] (33.5 MB/sample at 64^3)
//    and nothing of size R^3 x 32 is filled or read while pooling.
//  * per-point MLP: one thread per point, layer inputs in a private shared-memory column,
//    accumulators in registers, K-major weights broadcast from shared memory.
//  * scatter: rows are transposed through shared memory so that lane == channel; a warp
//    walks its 32 points, folds runs of equal slot in registers and issues ONE 128-byte
//    row atomic per run (warp-aggregated; only the final reduction is atomic).
//  * max pooling uses atomicMax/atomicMin on the int view of the floats: order
//    independent, hence bit-exact.  The final scatter_mean is an fp32 atomicAdd sum
//    (order not fixed -> tolerance), divided by the cell count, written once per occupied
//    cell into a zero-filled channels-last tensor.
#include "common.cuh"
#include "wgrad.cuh"
#include <math_constants.h>
#include <cmath>

namespace vtaco {

constexpr int kET = 128;        // threads per block
constexpr int kES = kET + 1;    // shared column stride
constexpr unsigned kFullMask = 0xffffffffu;

struct EncParams {
  const float* p;
  long long n, T;
  int B;
  NormConst nc;
  int nkeys;
  int kind[4];
  int reso[4];
  long long cells[4];
  int pool_mean;
  int n_blocks;
  const float* W;
  int32_t* idx[4];
  int32_t* slot[4];
  int32_t* map[4];
  int32_t* count[4];
  float* net[2];
  float* pool[3][4];
  float* sum[4];
  float* out_cl[4];
  float* c_out;
};

__device__ __forceinline__ void atomic_max_float(float* addr, float v) {
  v += 0.0f;  // -0 -> +0
  if (v >= 0.0f) atomicMax(reinterpret_cast<int*>(addr), __float_as_int(v));
  else atomicMin(reinterpret_cast<unsigned int*>(addr), __float_as_uint(v));
}

__device__ __forceinline__ int cell_index(const float x, const float y, const float z, int kind, int reso,
                                          const NormConst& nc) {
  if (kind == VTACO_GRID)
    return cell_of(norm3d(x, nc), reso) + reso * (cell_of(norm3d(y, nc), reso) + reso * cell_of(norm3d(z, nc), reso));
  const float a = (kind == VTACO_PLANE_YZ) ? y : x;
  const float b = (kind == VTACO_PLANE_XY) ? y : z;
  return cell_of(norm2d(a, nc), reso) + reso * cell_of(norm2d(b, nc), reso);
}

// pointnet.py:139-152 for every enabled key + election of the cell representative.
__global__ void __launch_bounds__(256) enc_index_kernel(const __grid_constant__ EncParams P) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= P.n) return;
  const float x = P.p[n * 3], y = P.p[n * 3 + 1], z = P.p[n * 3 + 2];
  const long long b = n / P.T;
  for (int k = 0; k < P.nkeys; ++k) {
    const int c = cell_index(x, y, z, P.kind[k], P.reso[k], P.nc);
    P.idx[k][n] = c;
    atomicMin(P.map[k] + b * P.cells[k] + c, (int)n);
  }
}

// generic: representative election from precomputed indices
__global__ void __launch_bounds__(256) map_min_kernel(const int32_t* __restrict__ idx, int32_t* __restrict__ map,
                                                      long long n, long long T, long long cells) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  atomicMin(map + (i / T) * cells + idx[i], (int)i);
}

__device__ __forceinline__ void fill_row(float* row, float v) {
  const float4 f = make_float4(v, v, v, v);
#pragma unroll
  for (int j = 0; j < 8; ++j) reinterpret_cast<float4*>(row)[j] = f;
}

// slot[n] = representative of n's cell; count[rep] += 1; first pooling buffer initialised.
__global__ void __launch_bounds__(256) enc_slot_kernel(const __grid_constant__ EncParams P, int init_pool) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= P.n) return;
  const long long b = n / P.T;
  const float init = P.pool_mean ? 0.0f : -CUDART_INF_F;
  for (int k = 0; k < P.nkeys; ++k) {
    const int s = P.map[k][b * P.cells[k] + P.idx[k][n]];
    P.slot[k][n] = s;
    atomicAdd(P.count[k] + s, 1);
    if (init_pool) fill_row(P.pool[0][k] + n * 32, init);
  }
}

// y[j] += sum_k W[k][j] * x  helpers (W K-major in shared memory, broadcast float4 loads)
__device__ __forceinline__ void axpy32(float (&acc)[32], const float* __restrict__ Wk, float x) {
  const float4* w4 = reinterpret_cast<const float4*>(Wk);
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const float4 w = w4[j];
    acc[4 * j] = fmaf(w.x, x, acc[4 * j]);
    acc[4 * j + 1] = fmaf(w.y, x, acc[4 * j + 1]);
    acc[4 * j + 2] = fmaf(w.z, x, acc[4 * j + 2]);
    acc[4 * j + 3] = fmaf(w.w, x, acc[4 * j + 3]);
  }
}

// One ResnetBlockFC(64 -> 32) per launch (layers.py:41-50) with its input assembly:
//   FIRST : x = fc_pos(p)                                   pointnet.py:154,156
//   else  : x = cat[net, pool_local(net)]                   pointnet.py:157-160
// and the scatter of its output into the next pooling buffer.
//
// FOUR warps per group of 32 points: warp q computes output channels [8q, 8q+8) of every layer for the 32
// points (lane == point), the inputs / hidden activations are shared through shared-memory columns.  The first
// version gave a point to one thread: 5 120 dependent-ish FMAs per thread and, at the shipped T = 3 640, 29 CTAs of
// one warp per scheduler — 40 us per block, latency-bound (ncu: issue slots 15 %, the rest waiting).  Per output
// channel the accumulation order over k is unchanged, so the results are bit-identical to that version.
constexpr int kEG = 32;          // points per group
constexpr int kEGS = kEG + 1;    // shared column stride (conflict-free for lane == point and lane == channel)
constexpr size_t kEncBlockSmem = (VTACO_ENC_BLOCK_STRIDE + VTACO_ENC_OFF_BLOCKS + 96 * kEGS) * sizeof(float);

__device__ __forceinline__ void axpy8(float (&acc)[8], const float* __restrict__ Wk, float x) {
  const float4 w0 = reinterpret_cast<const float4*>(Wk)[0], w1 = reinterpret_cast<const float4*>(Wk)[1];
  acc[0] = fmaf(w0.x, x, acc[0]); acc[1] = fmaf(w0.y, x, acc[1]); acc[2] = fmaf(w0.z, x, acc[2]); acc[3] = fmaf(w0.w, x, acc[3]);
  acc[4] = fmaf(w1.x, x, acc[4]); acc[5] = fmaf(w1.y, x, acc[5]); acc[6] = fmaf(w1.z, x, acc[6]); acc[7] = fmaf(w1.w, x, acc[7]);
}

// Points [i0, i1) of a 32-point group whose columns start at sX with stride `cs`, lane == channel: store the row,
// fold runs of equal slot, one row-wide atomic per run (warp-aggregated).
template <bool MEAN>
__device__ __forceinline__ void scatter_rows_range(const float* __restrict__ sX, int cs, int i0, int i1, long long n0,
                                                   long long nmax, int lane, int nkeys, const int (&myslot)[4],
                                                   float* const (&dst)[4], float* __restrict__ row_out) {
  int cur[4] = {-1, -1, -1, -1};
  float val[4] = {0.f, 0.f, 0.f, 0.f};
  for (int i = i0; i < i1; ++i) {
    const long long ni = n0 + i;
    if (ni >= nmax) break;  // uniform
    const float v = sX[lane * cs + i];
    if (row_out) row_out[ni * 32 + lane] = v;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      if (k < nkeys && dst[k]) {
        const int s = __shfl_sync(kFullMask, myslot[k], i);
        if (s != cur[k]) {
          if (cur[k] >= 0) {
            if (MEAN) atomicAdd(dst[k] + (long long)cur[k] * 32 + lane, val[k]);
            else atomic_max_float(dst[k] + (long long)cur[k] * 32 + lane, val[k]);
          }
          cur[k] = s;
          val[k] = v;
        } else {
          val[k] = MEAN ? (val[k] + v) : fmaxf(val[k], v);
        }
      }
    }
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k < nkeys && dst[k] && cur[k] >= 0) {
      if (MEAN) atomicAdd(dst[k] + (long long)cur[k] * 32 + lane, val[k]);
      else atomic_max_float(dst[k] + (long long)cur[k] * 32 + lane, val[k]);
    }
  }
}

template <bool FIRST>
__global__ void __launch_bounds__(128) enc_block_kernel(const __grid_constant__ EncParams P, int blk, int r_read,
                                                        int r_write, int r_init, int net_in, int net_out,
                                                        long long n_groups) {
  extern __shared__ __align__(16) float esm[];
  float* sW = esm;                                                // block weights [+ fc_pos]
  float* sX = sW + VTACO_ENC_BLOCK_STRIDE + VTACO_ENC_OFF_BLOCKS;  // [64][kEGS] inputs, later [32][kEGS] outputs
  float* sH = sX + 64 * kEGS;               // [32][kEGS] hidden activations
  const float* Wg = P.W + VTACO_ENC_OFF_BLOCKS + (long long)blk * VTACO_ENC_BLOCK_STRIDE;
  for (int i = threadIdx.x; i < VTACO_ENC_BLOCK_STRIDE / 4; i += 128)
    reinterpret_cast<float4*>(sW)[i] = __ldg(reinterpret_cast<const float4*>(Wg) + i);
  if (FIRST) {
    for (int i = threadIdx.x; i < VTACO_ENC_OFF_BLOCKS / 4; i += 128)
      reinterpret_cast<float4*>(sW + VTACO_ENC_BLOCK_STRIDE)[i] = __ldg(reinterpret_cast<const float4*>(P.W) + i);
    __syncthreads();   // fc_pos is read right away; otherwise the weight fill overlaps the first input gather
  }
  const int tid = threadIdx.x, lane = tid & 31, q = tid >> 5;
  float* dst[4] = {nullptr, nullptr, nullptr, nullptr};
  if (r_write >= 0)
    for (int k = 0; k < P.nkeys; ++k) dst[k] = P.pool[r_write][k];

  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const long long n0 = grp * kEG;
    const long long n = n0 + lane;
    const bool valid = n < P.n;
    int myslot[4] = {0, 0, 0, 0};
    for (int k = 0; k < P.nkeys; ++k) myslot[k] = valid ? P.slot[k][n] : 0;

    if (FIRST) {   // lane == point: channels [16q, 16q+16) of fc_pos(p)
      const float* Wp = sW + VTACO_ENC_BLOCK_STRIDE;
      const float px = valid ? P.p[n * 3] : 0.f, py = valid ? P.p[n * 3 + 1] : 0.f, pz = valid ? P.p[n * 3 + 2] : 0.f;
#pragma unroll 8
      for (int jj = 0; jj < 16; ++jj) {
        const int j = 16 * q + jj;
        sX[j * kEGS + lane] = fmaf(Wp[128 + j], pz, fmaf(Wp[64 + j], py, fmaf(Wp[j], px, Wp[VTACO_ENC_OFF_BPOS + j])));
      }
    } else {       // lane == channel: warp q assembles points 8q .. 8q+7, all their global loads in flight together
      const float* netin = P.net[net_in];
      float a[8], s[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = 8 * q + u;
        const long long ni = n0 + i;
        const bool ok = ni < P.n;                       // warp-uniform
        a[u] = ok ? netin[ni * 32 + lane] : 0.f;
        s[u] = 0.f;  // c_out = 0; c_out += fea  (key order xz, xy, yz, grid)
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          if (k < P.nkeys) {
            const int sl = __shfl_sync(kFullMask, myslot[k], i);
            float v = ok ? P.pool[r_read][k][(long long)sl * 32 + lane] : 0.f;
            if (P.pool_mean && ok) v = v / (float)P.count[k][sl];
            s[u] += v;
          }
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = 8 * q + u;
        sX[lane * kEGS + i] = a[u];
        sX[(32 + lane) * kEGS + i] = s[u];
      }
    }
    __syncthreads();   // inputs of the group (and, the first time, the weights) are in shared memory

    float h[8], o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) { h[j] = sW[VTACO_ENC_BLK_B0 + 8 * q + j]; o[j] = sW[VTACO_ENC_BLK_B1 + 8 * q + j]; }
#pragma unroll 4
    for (int k = 0; k < 64; ++k) {
      const float x = sX[k * kEGS + lane];
      axpy8(h, sW + VTACO_ENC_BLK_W0 + k * 32 + 8 * q, fmaxf(x, 0.f));  // fc_0(relu(x))
      axpy8(o, sW + VTACO_ENC_BLK_WS + k * 32 + 8 * q, x);              // shortcut(x), no bias
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) sH[(8 * q + j) * kEGS + lane] = fmaxf(h[j], 0.f);
    __syncthreads();   // hidden activations complete; nobody reads the input columns any more
#pragma unroll 4
    for (int k = 0; k < 32; ++k) axpy8(o, sW + VTACO_ENC_BLK_W1 + k * 32 + 8 * q, sH[k * kEGS + lane]);  // fc_1(relu(net))
#pragma unroll
    for (int j = 0; j < 8; ++j) sX[(8 * q + j) * kEGS + lane] = o[j];
    __syncthreads();

    // lane == channel again: warp q stores / scatters points 8q .. 8q+7
    if (P.pool_mean) scatter_rows_range<true>(sX, kEGS, 8 * q, 8 * q + 8, n0, P.n, lane, P.nkeys, myslot, dst, P.net[net_out]);
    else scatter_rows_range<false>(sX, kEGS, 8 * q, 8 * q + 8, n0, P.n, lane, P.nkeys, myslot, dst, P.net[net_out]);

    if (r_init >= 0 && valid) {   // re-initialise the buffer after next: two float4 of the point's row per warp
      const float init = P.pool_mean ? 0.0f : -CUDART_INF_F;
      const float4 f = make_float4(init, init, init, init);
      for (int k = 0; k < P.nkeys; ++k) {
        float4* row = reinterpret_cast<float4*>(P.pool[r_init][k] + n * 32);
        row[2 * q] = f;
        row[2 * q + 1] = f;
      }
    }
    __syncthreads();   // the columns are reused by the next group
  }
}

static unsigned enc_block_grid(long long n_groups) {
  const long long cap = (long long)num_sms() * 6;
  return (unsigned)(n_groups < cap ? n_groups : cap);
}

// c = fc_c(net) (pointnet.py:162) and the atomicAdd half of scatter_mean (:93,108).  Same shape as the block
// kernel: four warps per group of 32 points, warp q computes channels [8q, 8q+8).
constexpr size_t kEncFinalSmem = (VTACO_ENC_TAIL + 64 * kEGS) * sizeof(float);
__global__ void __launch_bounds__(128) enc_final_kernel(const __grid_constant__ EncParams P, int net_in, long long n_groups) {
  extern __shared__ __align__(16) float esm[];
  float* sW = esm;                   // fc_c section
  float* sX = sW + VTACO_ENC_TAIL;   // [32][kEGS] inputs
  float* sO = sX + 32 * kEGS;        // [32][kEGS] outputs
  const float* Wg = P.W + VTACO_ENC_OFF_BLOCKS + (long long)P.n_blocks * VTACO_ENC_BLOCK_STRIDE;
  for (int i = threadIdx.x; i < VTACO_ENC_TAIL / 4; i += 128)
    reinterpret_cast<float4*>(sW)[i] = __ldg(reinterpret_cast<const float4*>(Wg) + i);
  const int tid = threadIdx.x, lane = tid & 31, q = tid >> 5;
  float* dst[4] = {nullptr, nullptr, nullptr, nullptr};
  for (int k = 0; k < P.nkeys; ++k) dst[k] = P.sum[k];
  const float* netin = P.net[net_in];
  for (long long grp = blockIdx.x; grp < n_groups; grp += gridDim.x) {
    const long long n0 = grp * kEG;
    const long long n = n0 + lane;
    int myslot[4] = {0, 0, 0, 0};
    for (int k = 0; k < P.nkeys; ++k) myslot[k] = n < P.n ? P.slot[k][n] : 0;
#pragma unroll
    for (int u = 0; u < 8; ++u) {      // lane == channel: warp q loads points 8q .. 8q+7
      const int i = 8 * q + u;
      sX[lane * kEGS + i] = (n0 + i < P.n) ? netin[(n0 + i) * 32 + lane] : 0.f;
    }
    __syncthreads();
    float c[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) c[j] = sW[VTACO_ENC_FCC_B + 8 * q + j];
#pragma unroll 4
    for (int k = 0; k < 32; ++k) axpy8(c, sW + VTACO_ENC_FCC_W + k * 32 + 8 * q, sX[k * kEGS + lane]);
#pragma unroll
    for (int j = 0; j < 8; ++j) sO[(8 * q + j) * kEGS + lane] = c[j];
    __syncthreads();
    scatter_rows_range<true>(sO, kEGS, 8 * q, 8 * q + 8, n0, P.n, lane, P.nkeys, myslot, dst, P.c_out);
    // next group: sX is rewritten right away (its readers all passed the second barrier), sO only after the next
    // group's first barrier, which every warp reaches after this scatter
  }
}

// mean = sum / count, written once per occupied cell (the representative's thread) into the
// zero-filled channels-last output [B][cells][32].
__global__ void __launch_bounds__(256) enc_finalize_kernel(const __grid_constant__ EncParams P) {
  const long long n = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= P.n) return;
  const long long b = n / P.T;
  for (int k = 0; k < P.nkeys; ++k) {
    if (P.slot[k][n] != (int)n || !P.out_cl[k]) continue;
    const float cnt = (float)P.count[k][n];
    const float4* s4 = reinterpret_cast<const float4*>(P.sum[k] + n * 32);
    float4* o4 = reinterpret_cast<float4*>(P.out_cl[k] + (b * P.cells[k] + P.idx[k][n]) * 32);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float4 s = s4[j];
      o4[j] = make_float4(s.x / cnt, s.y / cnt, s.z / cnt, s.w / cnt);
    }
  }
}

// ---- row kernels of the stand-alone pooling (vtaco_pool_local / vtaco_scatter_mean) and of the backward ----
// Both pool into the cell rows P.pool[0] ([slot][32]) by P.slot.

// src rows [n][32] -> their cell rows: sum (MEAN) or maximum
template <bool MEAN>
__global__ void __launch_bounds__(kET) rows_scatter_kernel(const __grid_constant__ EncParams P,
                                                           const float* __restrict__ src) {
  __shared__ float sX[32 * kES];
  const int tid = threadIdx.x, lane = tid & 31, col0 = tid & ~31;
  const long long nb0 = (long long)blockIdx.x * kET;
  const long long me = nb0 + tid;
  int myslot[4] = {0, 0, 0, 0};
  for (int k = 0; k < P.nkeys; ++k) myslot[k] = me < P.n ? P.slot[k][me] : 0;
  for (int i = 0; i < 32; ++i) {
    const long long ni = nb0 + col0 + i;
    if (ni >= P.n) break;
    sX[lane * kES + col0 + i] = src[ni * 32 + lane];
  }
  __syncwarp();
  scatter_rows_range<MEAN>(sX + col0, kES, 0, 32, nb0 + col0, P.n, lane, P.nkeys, myslot, P.pool[0], nullptr);
}

// out[n] = sum over keys of the cell row of n (divided by the cell count for mean pooling)
__global__ void __launch_bounds__(256) rows_gather_kernel(const __grid_constant__ EncParams P, float* __restrict__ out) {
  const long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long ni = t >> 5;
  const int lane = threadIdx.x & 31;
  if (ni >= P.n) return;
  float s = 0.f;
  for (int k = 0; k < P.nkeys; ++k) {
    const int r = P.slot[k][ni];
    float v = P.pool[0][k][(long long)r * 32 + lane];
    if (P.pool_mean) v = v / (float)P.count[k][r];
    s += v;
  }
  out[ni * 32 + lane] = s;
}

static inline long long align_up(long long v, long long a) { return (v + a - 1) / a * a; }

struct Carver {
  char* base;
  long long off;
  template <typename T>
  T* take(long long count) {
    T* r = reinterpret_cast<T*>(base + off);
    off = align_up(off + count * (long long)sizeof(T), 256);
    return r;
  }
};

static long long cells_of(int kind, int reso) {
  return kind == VTACO_GRID ? (long long)reso * reso * reso : (long long)reso * reso;
}

// Workspace of the inference forward: per key idx, slot, count, map, three pooling buffers and the scatter_mean
// sums, then two net buffers.  Points P at it and returns its bytes; a null base only sizes it.
static long long carve_enc_fwd(char* base, int B, long long T, int nkeys, const int32_t* kind, const int32_t* reso,
                               EncParams& P) {
  const long long n = (long long)B * T;
  Carver c{base, 0};
  for (int k = 0; k < nkeys; ++k) {
    P.idx[k] = c.take<int32_t>(n); P.slot[k] = c.take<int32_t>(n); P.count[k] = c.take<int32_t>(n);
    P.map[k] = c.take<int32_t>((long long)B * cells_of(kind[k], reso[k]));
    for (int r = 0; r < 3; ++r) P.pool[r][k] = c.take<float>(n * 32);
    P.sum[k] = c.take<float>(n * 32);
  }
  P.net[0] = c.take<float>(n * 32);
  P.net[1] = c.take<float>(n * 32);
  return c.off;
}

// Workspace of the stand-alone pooling: per key slot, count, map and the cell rows P.pool[0].  Points P at it and
// returns its bytes; a null base only sizes it.
static long long carve_pool(char* base, int B, long long T, int nkeys, const int64_t* cells, EncParams& P) {
  const long long n = (long long)B * T;
  Carver c{base, 0};
  for (int k = 0; k < nkeys; ++k) {
    P.slot[k] = c.take<int32_t>(n); P.count[k] = c.take<int32_t>(n);
    P.map[k] = c.take<int32_t>((long long)B * cells[k]);
    P.pool[0][k] = c.take<float>(n * 32);
  }
  return c.off;
}

// Keys and point count of the forward and the backward: 1..4 keys of a known kind with reso >= 1 (else
// INVALID_ARG); fewer than n_max points and flat cell indices in int32 range (else UNSUPPORTED).
static int check_keys(int n_keys, const int32_t* kind, const int32_t* reso, long long n, long long n_max) {
  if (n_keys < 1 || n_keys > 4) return VTACO_ERR_INVALID_ARG;
  if (n >= n_max) return VTACO_ERR_UNSUPPORTED;
  for (int k = 0; k < n_keys; ++k) {
    if (kind[k] < 0 || kind[k] > 3 || reso[k] < 1) return VTACO_ERR_INVALID_ARG;
    if (!cell_index_fits(kind[k], reso[k])) return VTACO_ERR_UNSUPPORTED;
  }
  return VTACO_OK;
}

// Points, keys and weights of the forward and the backward (vtaco_encoder_args / vtaco_encoder_bwd_args).
template <class Args>
static EncParams enc_params(const Args* a) {
  EncParams P = {};
  P.p = a->p; P.n = (long long)a->B * a->T; P.T = a->T; P.B = a->B;
  P.nc = make_norm_const(a->padding, a->div_mode);
  P.nkeys = a->n_keys; P.pool_mean = a->pool_mean ? 1 : 0; P.n_blocks = a->n_blocks; P.W = a->weights;
  for (int k = 0; k < a->n_keys; ++k) {
    P.kind[k] = a->kind[k]; P.reso[k] = a->reso[k]; P.cells[k] = cells_of(a->kind[k], a->reso[k]);
  }
  return P;
}

// Per-key reset before the cell election: map = 0x7f7f7f7f, so that atomicMin elects a cell's lowest point; count = 0.
static int reset_cells(const EncParams& P, cudaStream_t st) {
  for (int k = 0; k < P.nkeys; ++k) {
    VTACO_CUDA_CHECK(cudaMemsetAsync(P.map[k], 0x7f, sizeof(int32_t) * P.B * P.cells[k], st));
    VTACO_CUDA_CHECK(cudaMemsetAsync(P.count[k], 0, sizeof(int32_t) * P.n, st));
  }
  return VTACO_OK;
}

// Cell election, slots and the ResnetBlockFC stack (pointnet.py:139-160), for the inference forward and for the
// backward's recompute.  Block i reads pool level i, scatters into level i + 1 and initialises level i + 2, each only
// if it is below nb (there is no level 0; enc_slot_kernel initialises level 1); it reads net level i - 1 and writes
// net level i.  pool(l, k) and net(l) are the buffers of a level.  Each launch gets its window [level i, i + 1, i + 2]
// in P.pool[0..2] and its net levels [i - 1, i] in P.net[0..1].
template <class PoolLevel, class NetLevel>
static int launch_block_stack(EncParams P, const PoolLevel& pool, const NetLevel& net, cudaStream_t st) {
  const int nb = P.n_blocks;
  const auto window = [&](int l) {
    for (int w = 0; w < 3; ++w)
      for (int k = 0; k < P.nkeys; ++k) P.pool[w][k] = (l + w >= 1 && l + w < nb) ? pool(l + w, k) : nullptr;
  };
  const int r = reset_cells(P, st);
  if (r != VTACO_OK) return r;
  const unsigned g256 = (unsigned)((P.n + 255) / 256);
  enc_index_kernel<<<g256, 256, 0, st>>>(P);
  window(1);
  enc_slot_kernel<<<g256, 256, 0, st>>>(P, nb > 1);
  const long long n_groups = (P.n + kEG - 1) / kEG;
  const unsigned gB = enc_block_grid(n_groups);
  for (int i = 0; i < nb; ++i) {
    window(i);
    P.net[0] = i > 0 ? net(i - 1) : nullptr;
    P.net[1] = net(i);
    const int r_write = i + 1 < nb ? 1 : -1, r_init = i + 2 < nb ? 2 : -1;
    if (i == 0) enc_block_kernel<true><<<gB, 128, kEncBlockSmem, st>>>(P, 0, -1, r_write, r_init, 0, 1, n_groups);
    else enc_block_kernel<false><<<gB, 128, kEncBlockSmem, st>>>(P, i, 0, r_write, r_init, 0, 1, n_groups);
  }
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

// Stand-alone pooling of src rows [n][32] into the cell rows P.pool[0] by the caller's cell indices P.idx.
static int pool_rows(const EncParams& P, const float* src, cudaStream_t st) {
  const int r = reset_cells(P, st);
  if (r != VTACO_OK) return r;
  const unsigned g256 = (unsigned)((P.n + 255) / 256), gE = (unsigned)((P.n + kET - 1) / kET);
  for (int k = 0; k < P.nkeys; ++k) map_min_kernel<<<g256, 256, 0, st>>>(P.idx[k], P.map[k], P.n, P.T, P.cells[k]);
  enc_slot_kernel<<<g256, 256, 0, st>>>(P, 1);
  if (P.pool_mean) rows_scatter_kernel<true><<<gE, kET, 0, st>>>(P, src);
  else rows_scatter_kernel<false><<<gE, kET, 0, st>>>(P, src);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

// EncParams of the stand-alone pooling: n = B * T points, the caller's cell indices and cell counts per key.
static EncParams pool_params(int B, long long T, int nkeys, const int32_t* const* idx, const int64_t* cells, int mean) {
  EncParams P = {};
  P.n = (long long)B * T; P.T = T; P.B = B;
  P.nkeys = nkeys; P.pool_mean = mean ? 1 : 0;
  for (int k = 0; k < nkeys; ++k) {
    P.idx[k] = const_cast<int32_t*>(idx[k]);   // enc_slot_kernel and enc_finalize_kernel only read idx
    P.cells[k] = cells[k];
  }
  return P;
}

}  // namespace vtaco

using namespace vtaco;

extern "C" int64_t vtaco_encoder_workspace_bytes(int32_t B, int64_t T, int32_t n_keys, const int32_t* kind,
                                                 const int32_t* reso) {
  if (B <= 0 || T <= 0 || n_keys <= 0 || n_keys > 4 || !kind || !reso) return VTACO_ERR_INVALID_ARG;
  EncParams P = {};
  return carve_enc_fwd(nullptr, B, T, n_keys, kind, reso, P);
}

extern "C" int vtaco_encoder_pointnet(const vtaco_encoder_args* a, void* stream) {
  if (!a || !a->p || !a->weights || !a->workspace) return VTACO_ERR_INVALID_ARG;
  if (a->B <= 0 || a->T <= 0 || a->n_blocks < 1) return VTACO_ERR_INVALID_ARG;
  const long long n = (long long)a->B * a->T;
  int r = check_keys(a->n_keys, a->kind, a->reso, n, 1ll << 31);
  if (r != VTACO_OK) return r;
  EncParams P = enc_params(a);
  if (carve_enc_fwd(reinterpret_cast<char*>(a->workspace), a->B, a->T, a->n_keys, a->kind, a->reso, P) >
      a->workspace_bytes)
    return VTACO_ERR_CAPACITY;
  cudaStream_t st = (cudaStream_t)stream;
  P.c_out = a->c_out;
  for (int k = 0; k < a->n_keys; ++k) {
    P.out_cl[k] = a->out_cl[k];
    VTACO_CUDA_CHECK(cudaMemsetAsync(P.sum[k], 0, sizeof(float) * n * 32, st));
    if (P.out_cl[k])
      VTACO_CUDA_CHECK(cudaMemsetAsync(P.out_cl[k], 0, sizeof(float) * a->B * P.cells[k] * 32, st));
  }
  const int nb = a->n_blocks;
  const auto pool_level = [&](int l, int k) { return P.pool[(l - 1) % 3][k]; };   // three buffers in turn
  const auto net_level = [&](int l) { return P.net[l & 1]; };                      // two buffers in turn
  r = launch_block_stack(P, pool_level, net_level, st);
  if (r != VTACO_OK) return r;
  EncParams F = P;   // fc_c reads the output of the last block
  F.net[0] = net_level(nb - 1);
  const long long n_groups = (n + kEG - 1) / kEG;
  enc_final_kernel<<<enc_block_grid(n_groups), 128, kEncFinalSmem, st>>>(F, 0, n_groups);
  enc_finalize_kernel<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(P);
  VTACO_LAUNCH_CHECK();
  for (int k = 0; k < a->n_keys; ++k)
    if (a->index_out[k])
      VTACO_CUDA_CHECK(cudaMemcpyAsync(a->index_out[k], P.idx[k], sizeof(int32_t) * n, cudaMemcpyDeviceToDevice, st));
  return VTACO_OK;
}

extern "C" int64_t vtaco_pool_workspace_bytes(int32_t B, int64_t T, int32_t n_keys, const int64_t* cells) {
  if (B <= 0 || T <= 0 || n_keys <= 0 || n_keys > 4 || !cells) return VTACO_ERR_INVALID_ARG;
  EncParams P = {};
  return carve_pool(nullptr, B, T, n_keys, cells, P);
}

extern "C" int vtaco_pool_local(const float* feat, int32_t B, int64_t T, int32_t n_keys, const int32_t* const* idx32,
                                const int64_t* cells, int32_t mean, void* workspace, int64_t workspace_bytes,
                                float* out, void* stream) {
  if (!feat || !idx32 || !cells || !workspace || !out) return VTACO_ERR_INVALID_ARG;
  if (B <= 0 || T <= 0 || n_keys <= 0 || n_keys > 4) return VTACO_ERR_INVALID_ARG;
  EncParams P = pool_params(B, T, n_keys, idx32, cells, mean);
  if (carve_pool(reinterpret_cast<char*>(workspace), B, T, n_keys, cells, P) > workspace_bytes)
    return VTACO_ERR_CAPACITY;
  if (P.n >= (1ll << 31)) return VTACO_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  const int r = pool_rows(P, feat, st);
  if (r != VTACO_OK) return r;
  rows_gather_kernel<<<(unsigned)((P.n * 32 + 255) / 256), 256, 0, st>>>(P, out);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_scatter_mean(const float* c, const int32_t* idx32, int32_t B, int64_t T, int64_t cells,
                                  void* workspace, int64_t workspace_bytes, float* out_cl, void* stream) {
  if (!c || !idx32 || !workspace || !out_cl || B <= 0 || T <= 0 || cells <= 0) return VTACO_ERR_INVALID_ARG;
  EncParams P = pool_params(B, T, 1, &idx32, &cells, 1);
  if (carve_pool(reinterpret_cast<char*>(workspace), B, T, 1, &cells, P) > workspace_bytes) return VTACO_ERR_CAPACITY;
  if (P.n >= (1ll << 31)) return VTACO_ERR_UNSUPPORTED;
  cudaStream_t st = (cudaStream_t)stream;
  P.sum[0] = P.pool[0][0];
  P.out_cl[0] = out_cl;
  VTACO_CUDA_CHECK(cudaMemsetAsync(out_cl, 0, sizeof(float) * B * cells * 32, st));
  const int r = pool_rows(P, c, st);
  if (r != VTACO_OK) return r;
  enc_finalize_kernel<<<(unsigned)((P.n + 255) / 256), 256, 0, st>>>(P);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

#include "encoder_bwd.inl"

// ---------------------------------------------------------------------------------------
// GroupNorm over contiguous NC[D]HW fp32 tensors (the 'g' of UNet3D's 'gcr' layers, reference
// src/encoder/unet3d.py:create_conv).  ATen launches one block per (sample, group) — 8 blocks
// for the 64^3 x 32 grid, ~0.5 ms each; here the reduction is spread over the whole chip:
//   stats : grid (chunks, N*G); per-block fp32 partial sums -> fp64 atomics (sum, sum of squares)
//   apply : y = (x - mean) * rstd * gamma[c] + beta[c], float4 vectorised
// HBM-bound: 4 B read (stats) + 8 B read/write (apply) per element.
// ---------------------------------------------------------------------------------------
namespace vtaco {

__global__ void __launch_bounds__(256) gn_stats_kernel(const float* __restrict__ x, long long L, double* __restrict__ acc) {
  const long long ng = blockIdx.y;
  const float* base = x + ng * L;
  float s = 0.f, ss = 0.f;
  const long long per = (L + gridDim.x - 1) / gridDim.x;
  const long long lo = (long long)blockIdx.x * per, hi = min(L, lo + per);
  if (((L | per) & 3) == 0) {
    for (long long i = lo + 4 * threadIdx.x; i < hi; i += 4 * 256) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(base + i));
      s += (v.x + v.y) + (v.z + v.w);
      ss += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
    }
  } else {
    for (long long i = lo + threadIdx.x; i < hi; i += 256) {
      const float v = base[i];
      s += v;
      ss += v * v;
    }
  }
  double ds = (double)s, dss = (double)ss;
#pragma unroll
  for (int d = 16; d > 0; d >>= 1) {
    ds += __shfl_xor_sync(0xffffffffu, ds, d);
    dss += __shfl_xor_sync(0xffffffffu, dss, d);
  }
  __shared__ double sh[2][8];
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (lane == 0) { sh[0][w] = ds; sh[1][w] = dss; }
  __syncthreads();
  if (threadIdx.x == 0) {
    double a = 0, b = 0;
    for (int i = 0; i < 8; ++i) { a += sh[0][i]; b += sh[1][i]; }
    atomicAdd(acc + 2 * ng, a);
    atomicAdd(acc + 2 * ng + 1, b);
  }
}

__global__ void __launch_bounds__(256) gn_apply_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       const double* __restrict__ acc, int C, int G, long long S,
                                                       long long total, double eps) {
  const int cpg = C / G;
  const long long L = (long long)cpg * S;
  const bool vec = (S & 3) == 0;
  const long long step = (long long)gridDim.x * blockDim.x * (vec ? 4 : 1);
  for (long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * (vec ? 4 : 1); i < total; i += step) {
    const long long nc = i / S;            // n*C + c   (4 consecutive elements share it when S % 4 == 0)
    const int c = (int)(nc % C);
    const long long ng = (nc / C) * G + c / cpg;
    const double mean = acc[2 * ng] / (double)L;
    const double var = fmax(acc[2 * ng + 1] / (double)L - mean * mean, 0.0);
    const float rstd = (float)(1.0 / sqrt(var + eps));
    const float g = gamma ? gamma[c] : 1.f, b = beta ? beta[c] : 0.f;
    const float sc = rstd * g, sh = b - (float)mean * sc;
    if (vec) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(x + i));
      *reinterpret_cast<float4*>(y + i) = make_float4(fmaf(v.x, sc, sh), fmaf(v.y, sc, sh), fmaf(v.z, sc, sh), fmaf(v.w, sc, sh));
    } else {
      y[i] = fmaf(x[i], sc, sh);
    }
  }
}

}  // namespace vtaco

extern "C" int vtaco_group_norm(const float* x, float* y, const float* gamma, const float* beta, int32_t N, int32_t C,
                                int32_t G, int64_t S, double eps, double* stats_ws, void* stream) {
  if (!x || !y || !stats_ws || N <= 0 || C <= 0 || G <= 0 || S <= 0 || C % G) return VTACO_ERR_INVALID_ARG;
  cudaStream_t st = (cudaStream_t)stream;
  const long long L = (long long)(C / G) * S, total = (long long)N * C * S;
  VTACO_CUDA_CHECK(cudaMemsetAsync(stats_ws, 0, sizeof(double) * 2 * N * G, st));
  long long chunks = (L + 16383) / 16384;
  const long long cap = (long long)vtaco::num_sms() * 8 / ((long long)N * G) + 1;
  if (chunks > cap) chunks = cap;
  if (chunks < 1) chunks = 1;
  vtaco::gn_stats_kernel<<<dim3((unsigned)chunks, (unsigned)(N * G)), 256, 0, st>>>(x, L, stats_ws);
  long long blocks = (total / 4 + 255) / 256 + 1;
  const long long bcap = (long long)vtaco::num_sms() * 16;
  if (blocks > bcap) blocks = bcap;
  vtaco::gn_apply_kernel<<<(unsigned)blocks, 256, 0, st>>>(x, y, gamma, beta, stats_ws, C, G, S, total, eps);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

// ---------------------------------------------------------------------------------------
// GroupNorm, channels-last: x, y [N][S][C] (torch channels_last / channels_last_3d storage).
// Keeping UNet3D in channels-last end to end removes cuDNN's NCDHW<->NDHWC conversion kernels
// around every convolution (about half of the UNet3D time at 64^3 x 32).  A thread owns one
// float4 channel quad (C/4 divides the block size, so the quad — and its group — is fixed per
// thread); per-block fp32 partials -> shared fp64 -> one global fp64 atomic per group and block.
// ---------------------------------------------------------------------------------------
namespace vtaco {

__global__ void __launch_bounds__(256) gn_cl_stats_kernel(const float4* __restrict__ x, long long S, int C, int G,
                                                          double* __restrict__ acc) {
  __shared__ double sh[64][2];
  const int n = blockIdx.y, q = C >> 2, cpg = C / G;
  for (int i = threadIdx.x; i < G; i += 256) { sh[i][0] = 0.0; sh[i][1] = 0.0; }
  __syncthreads();
  const long long total = S * q;                       // float4 elements of this sample
  const long long per = (total + gridDim.x - 1) / gridDim.x / 256 * 256 + 256;
  const long long lo = (long long)blockIdx.x * per, hi = min(total, lo + per);
  const float4* base = x + (long long)n * total;
  float s = 0.f, ss = 0.f;
  for (long long e = lo + threadIdx.x; e < hi; e += 256) {
    const float4 v = __ldg(base + e);
    s += (v.x + v.y) + (v.z + v.w);
    ss += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
  }
  const int g = ((threadIdx.x % q) * 4) / cpg;         // lo is a multiple of 256 and q | 256
  atomicAdd(&sh[g][0], (double)s);
  atomicAdd(&sh[g][1], (double)ss);
  __syncthreads();
  for (int i = threadIdx.x; i < G; i += 256) {
    atomicAdd(acc + 2 * ((long long)n * G + i), sh[i][0]);
    atomicAdd(acc + 2 * ((long long)n * G + i) + 1, sh[i][1]);
  }
}

__global__ void __launch_bounds__(256) gn_cl_apply_kernel(const float4* __restrict__ x, float4* __restrict__ y,
                                                          const float* __restrict__ gamma, const float* __restrict__ beta,
                                                          const double* __restrict__ acc, long long S, int C, int G,
                                                          double eps) {
  const int n = blockIdx.y, q = C >> 2, cpg = C / G;
  const long long total = S * q;
  const int cq = threadIdx.x % q, c0 = cq * 4, g = c0 / cpg;
  const double L = (double)cpg * (double)S;
  const double mean = acc[2 * ((long long)n * G + g)] / L;
  const double var = fmax(acc[2 * ((long long)n * G + g) + 1] / L - mean * mean, 0.0);
  const float rstd = (float)(1.0 / sqrt(var + eps));
  float sc[4], sf[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    sc[j] = rstd * (gamma ? gamma[c0 + j] : 1.f);
    sf[j] = (beta ? beta[c0 + j] : 0.f) - (float)mean * sc[j];
  }
  const float4* xb = x + (long long)n * total;
  float4* yb = y + (long long)n * total;
  for (long long e = (long long)blockIdx.x * 256 + threadIdx.x; e < total; e += (long long)gridDim.x * 256) {
    const float4 v = __ldg(xb + e);
    yb[e] = make_float4(fmaf(v.x, sc[0], sf[0]), fmaf(v.y, sc[1], sf[1]), fmaf(v.z, sc[2], sf[2]), fmaf(v.w, sc[3], sf[3]));
  }
}

}  // namespace vtaco

extern "C" int vtaco_group_norm_cl(const float* x, float* y, const float* gamma, const float* beta, int32_t N,
                                   int32_t C, int32_t G, int64_t S, double eps, double* stats_ws, void* stream) {
  if (!x || !y || !stats_ws || N <= 0 || C <= 0 || G <= 0 || G > 64 || S <= 0 || C % G) return VTACO_ERR_INVALID_ARG;
  const int q = C / 4, cpg = C / G;
  if (C % 4 || cpg % 4 || 256 % q) return VTACO_ERR_UNSUPPORTED;   // caller falls back to the contiguous kernel
  cudaStream_t st = (cudaStream_t)stream;
  VTACO_CUDA_CHECK(cudaMemsetAsync(stats_ws, 0, sizeof(double) * 2 * N * G, st));
  const long long total = S * q;
  long long chunks = (total + 256 * 64 - 1) / (256 * 64);
  const long long cap = (long long)vtaco::num_sms() * 8 / N + 1;
  if (chunks > cap) chunks = cap;
  if (chunks < 1) chunks = 1;
  vtaco::gn_cl_stats_kernel<<<dim3((unsigned)chunks, (unsigned)N), 256, 0, st>>>(reinterpret_cast<const float4*>(x), S, C, G, stats_ws);
  long long blocks = (total + 255) / 256;
  const long long bcap = (long long)vtaco::num_sms() * 16 / N + 1;
  if (blocks > bcap) blocks = bcap;
  vtaco::gn_cl_apply_kernel<<<dim3((unsigned)blocks, (unsigned)N), 256, 0, st>>>(
      reinterpret_cast<const float4*>(x), reinterpret_cast<float4*>(y), gamma, beta, stats_ws, S, C, G, eps);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

// ---------------------------------------------------------------------------------------
// UNet3D decoder input (reference src/encoder/unet3d.py Decoder.forward / _joining):
//   out = cat(skip, interpolate(x, size = skip.shape[2:], mode='nearest'), dim=1)
// in one pass over the output instead of ATen's upsample (writes C2 x S) + cat (reads and
// writes (C1 + C2) x S).  Contiguous NCDHW fp32; source index as ATen's
// nearest_neighbor_compute_source_index: min(floor(dst * (float)in / out), in - 1).
// ---------------------------------------------------------------------------------------
namespace vtaco {

__global__ void __launch_bounds__(256) upsample_concat3d_kernel(const float* __restrict__ skip, const float* __restrict__ x,
                                                                float* __restrict__ out, int C1, int C2, int Do, int Ho,
                                                                int Wo, int Di, int Hi, int Wi, float sd, float sh,
                                                                float sw, long long quads) {
  const long long So = (long long)Do * Ho * Wo, Si = (long long)Di * Hi * Wi;
  const int Wq = Wo >> 2;
  for (long long q = (long long)blockIdx.x * 256 + threadIdx.x; q < quads; q += (long long)gridDim.x * 256) {
    long long t = q;
    const int xq = (int)(t % Wq); t /= Wq;
    const int y = (int)(t % Ho); t /= Ho;
    const int z = (int)(t % Do); t /= Do;
    const int c = (int)(t % (C1 + C2));
    const long long n = t / (C1 + C2);
    const long long o = ((n * (C1 + C2) + c) * So + ((long long)z * Ho + y) * Wo) + 4 * xq;
    float4 v;
    if (c < C1) {
      v = __ldg(reinterpret_cast<const float4*>(skip + (n * C1 + c) * So + ((long long)z * Ho + y) * Wo + 4 * xq));
    } else {
      const int zi = min((int)floorf(z * sd), Di - 1), yi = min((int)floorf(y * sh), Hi - 1);
      const float* row = x + (n * C2 + (c - C1)) * Si + ((long long)zi * Hi + yi) * Wi;
      const int x0 = 4 * xq;
      v.x = __ldg(row + min((int)floorf(x0 * sw), Wi - 1));
      v.y = __ldg(row + min((int)floorf((x0 + 1) * sw), Wi - 1));
      v.z = __ldg(row + min((int)floorf((x0 + 2) * sw), Wi - 1));
      v.w = __ldg(row + min((int)floorf((x0 + 3) * sw), Wi - 1));
    }
    *reinterpret_cast<float4*>(out + o) = v;
  }
}

}  // namespace vtaco

extern "C" int vtaco_upsample_concat3d(const float* skip, const float* x, float* out, int32_t N, int32_t C1, int32_t C2,
                                       int32_t Do, int32_t Ho, int32_t Wo, int32_t Di, int32_t Hi, int32_t Wi,
                                       void* stream) {
  if (!skip || !x || !out || N <= 0 || C1 <= 0 || C2 <= 0 || Do <= 0 || Ho <= 0 || Wo <= 0 || Di <= 0 || Hi <= 0 || Wi <= 0)
    return VTACO_ERR_INVALID_ARG;
  if (Wo % 4) return VTACO_ERR_UNSUPPORTED;   // float4 rows; callers fall back to two ATen ops
  const long long quads = (long long)N * (C1 + C2) * Do * Ho * (Wo / 4);
  long long blocks = (quads + 255) / 256;
  const long long cap = (long long)vtaco::num_sms() * 16;
  if (blocks > cap) blocks = cap;
  vtaco::upsample_concat3d_kernel<<<(unsigned)blocks, 256, 0, (cudaStream_t)stream>>>(
      skip, x, out, C1, C2, Do, Ho, Wo, Di, Hi, Wi, (float)Di / (float)Do, (float)Hi / (float)Ho, (float)Wi / (float)Wo,
      quads);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}
