// UNet3D building blocks on our own kernels (SURVEY 8f-3; reference src/encoder/unet3d.py:
// SingleConv 'gcr' = GroupNorm -> Conv3d(3x3x3, pad 1, no bias) -> ReLU, Encoder = MaxPool3d(2) +
// DoubleConv, Decoder = nearest-upsample + concat + DoubleConv, final 1x1x1 Conv3d with bias).
//
// One 'gcr' layer = ONE kernel: implicit-GEMM convolution on the 5th-gen tensor cores
// (tcgen05.mma kind::tf32, A and B from shared memory, accumulator in TMEM) over channels-last
// activations, with
//   * GroupNorm-apply fused into the operand loader (per-channel scale / shift derived in the
//     prologue from per-channel (sum, sumsq) that the PRODUCER of the input accumulated),
//   * nearest-upsample + concat fused into the loader (channels >= C1 are read from the
//     half-resolution tensor), so the concatenated tensor is never materialised,
//   * ReLU + per-channel (sum, sumsq) of the output (the next layer's GroupNorm statistics) fused
//     into the epilogue.
// Tiling: a CTA owns 1 x 16 x 8 (z,y,x) output voxels = the 128 rows of an M128 N32 MMA and 32
// output channels.  Per 16 input channels the loader builds the halo brick (3 x 18 x 10 voxels) in
// shared memory as 4 planes [channel quad][voxel][4], the UMMA canonical K-major no-swizzle
// layout with the voxel as the row: a filter tap is then just a different START ADDRESS of the
// same brick (row-group stride = one brick row), so im2col costs no data movement at all —
// 27 taps x 2 MMAs (K = 8) per chunk.
// Arithmetic: single-pass TF32 (operands rounded to nearest TF32, fp32 accumulation) — what the
// reference runs on a GPU (cuDNN with torch.backends.cudnn.allow_tf32 = True, torch's default).
#include "common.cuh"
#include <math_constants.h>
#include <cstdio>
#include <cstdlib>

namespace vtaco {

constexpr int kCvThreads = 544;            // one persistent CTA per SM: 16 worker warps (bricks, epilogue) + 1 MMA-issuer warp
constexpr int kCvKC = 16;                 // input channels per chunk (4 planes of 4)
constexpr int kCvTileY = 16, kCvTileX = 8;
constexpr int kCvMaxCin = 512;
constexpr int kCvLoaders = 512;            // warps 0..15 fill the bricks and run the epilogue; warp 16 only issues the MMAs
constexpr uint32_t kCvIdesc = (1u << 4) | (2u << 7) | (2u << 10) | (4u << 17) | (8u << 24);  // F32 acc, TF32 x TF32, K-major, N=32, M=128

struct ConvParams {
  const float* x;      // [N][D][H][W][C1]
  const float* x2;     // [N][D2][H2][W2][C2] or NULL
  const float* w;      // packed: [Cout/32][Cin/16][taps][4][32][4]
  const float* bias;   // [Cout] or NULL
  const double* in_stats;   // [N][Cin][2] or NULL (no GroupNorm)
  const float* gamma;  // [Cin]
  const float* beta;
  float* y;            // [N][D][H][W][Cout]
  double* out_stats;   // [N][Cout][2] or NULL
  int N, D, H, W, C1, C2, D2, H2, W2, Cout, ksize, groups, relu;   // (the filter's z extent is a template parameter)
  int tiles_x, tiles_y, n_tiles;
  double eps;
  long long* trace;    // debug (VTACO_CV_TRACE=1): clock64 stamps of thread 0 of block 0
};
#define CV_STAMP(slot)                                                                        \
  do {                                                                                        \
    if (P.trace && blockIdx.x == 0 && blockIdx.y == 0 && tid == 0 && trace_n < 2048)          \
      P.trace[trace_n++] = ((long long)(slot) << 56) | (clock64() & 0x00ffffffffffffffll);    \
  } while (0)

__device__ __forceinline__ uint32_t cv_smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ uint64_t cv_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fff);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3fff) << 16;   // between core matrices adjacent in K
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3fff) << 32;   // between 8-row groups
  d |= (uint64_t)1 << 46;                             // descriptor version (Blackwell)
  return d;
}
__device__ __forceinline__ void cv_mma_ss(uint32_t d, uint64_t adesc, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n" ::"r"(d), "l"(adesc), "l"(bdesc), "r"(kCvIdesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ float cv_tf32(float v) {   // round to nearest (ties away), like cvt.rna.tf32
  return __uint_as_float((__float_as_uint(v) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ void cv_mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n.reg .pred p;\nCV_WAIT:\nmbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n@p bra CV_DONE;\nbra CV_WAIT;\nCV_DONE:\n}\n" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void cv_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}

// shared memory: 2 brick buffers | 2 weight-chunk slots | GroupNorm tables | statistics | barriers
struct CvSmem { int brick, w, scale, shift, stat, bar, tmem, total, plane_stride, brick_bytes, row_pitch, bvox, wslot; };
__host__ __device__ inline CvSmem cv_layout(int ksize, int kz, int cin) {
  CvSmem s;
  const int h = ksize / 2, hz = kz / 2;
  const int bz = 1 + 2 * hz, by = kCvTileY + 2 * h, bx = kCvTileX + 2 * h;
  s.bvox = bz * by * bx;
  s.row_pitch = bx * 16;                                   // bytes between brick rows (= 8-row groups of the MMA)
  s.plane_stride = (s.bvox * 16 + 80 + 127) / 128 * 128 + 16;   // odd multiple of 16 B: spreads the planes over the banks
  s.brick_bytes = (4 * s.plane_stride + 127) / 128 * 128;
  s.brick = 0;
  s.w = 2 * s.brick_bytes;
  const int taps = ksize * ksize * kz;
  s.wslot = taps * 2048;
  s.scale = s.w + 2 * s.wslot;
  s.shift = s.scale + cin * 4;
  s.stat = s.shift + cin * 4;
  // [0,1] MMAs that read brick / weight slot b done, [2,3] weights of slot b landed, [4,5] accumulator a done,
  // [6,7] brick buffer b filled (one arrival per worker warp)
  s.bar = (s.stat + 64 * 4 + 15) / 16 * 16;
  s.tmem = s.bar + 64;
  s.total = s.tmem + 16;
  return s;
}

// KZ = extent of the filter along z: KSIZE (3-D convolution) or 1 (a 2-D convolution on every z-slice — the
// feature planes of the 2-D U-Net are volumes of depth 1: a third of the taps and of the halo brick)
template <int KSIZE, int KZ>
__global__ void __launch_bounds__(kCvThreads, 1) conv3d_tc_kernel(const __grid_constant__ ConvParams P) {
  extern __shared__ __align__(128) unsigned char sm[];
  const int Cin = P.C1 + P.C2;
  const CvSmem L = cv_layout(KSIZE, KZ, Cin);
  float* sScale = reinterpret_cast<float*>(sm + L.scale);
  float* sShift = reinterpret_cast<float*>(sm + L.shift);
  float* sStat = reinterpret_cast<float*>(sm + L.stat);
  uint64_t* sBar = reinterpret_cast<uint64_t*>(sm + L.bar);
  uint32_t* sTmem = reinterpret_cast<uint32_t*>(sm + L.tmem);
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  constexpr int h = KSIZE / 2, hz = KZ / 2, taps = KSIZE * KSIZE * KZ;
  constexpr int bx_ext = kCvTileX + 2 * h, by_ext = kCvTileY + 2 * h, bz_ext = 1 + 2 * hz;
  constexpr int kBvox = bz_ext * by_ext * bx_ext;
  constexpr int kCvItems = (kBvox * 4 + kCvLoaders - 1) / kCvLoaders;   // brick float4s per loader thread
  constexpr int kPlane = (kBvox * 16 + 80 + 127) / 128 * 128 + 16;      // == cv_layout().plane_stride
  constexpr int kRowPitch = bx_ext * 16;
  const int ntile = blockIdx.y, n = blockIdx.z;
  const int ltid = tid;                      // worker index (warps 0..15); warp 16 is the MMA issuer
  const bool issuer = warp == 16;
  const int n_chunks = Cin / kCvKC;
  int trace_n = 0;

  // ---- prologue: GroupNorm scale / shift per input channel, barriers, TMEM (two accumulators) ----
  if (P.in_stats) {
    const int cpg = Cin / P.groups;
    const double cnt = (double)P.D * P.H * P.W * cpg;
    for (int c = tid; c < Cin; c += kCvThreads) {
      const int g = c / cpg;
      double s = 0.0, ss = 0.0;
      for (int j = 0; j < cpg; ++j) {
        s += P.in_stats[((size_t)n * Cin + g * cpg + j) * 2];
        ss += P.in_stats[((size_t)n * Cin + g * cpg + j) * 2 + 1];
      }
      const double mean = s / cnt;
      double var = ss / cnt - mean * mean;
      if (var < 0.0) var = 0.0;
      const double rstd = 1.0 / sqrt(var + P.eps);
      const double ga = P.gamma ? (double)P.gamma[c] : 1.0, be = P.beta ? (double)P.beta[c] : 0.0;
      sScale[c] = (float)(rstd * ga);
      sShift[c] = (float)(be - mean * rstd * ga);
    }
  } else {
    for (int c = tid; c < Cin; c += kCvThreads) { sScale[c] = 1.0f; sShift[c] = 0.0f; }
  }
  if (tid < 64) sStat[tid] = 0.0f;
  if (tid == 0) {
    for (int i = 0; i < 6; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(cv_smem_u32(sBar + i)) : "memory");
    for (int i = 6; i < 8; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 16;" ::"r"(cv_smem_u32(sBar + i)) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(cv_smem_u32(sTmem)), "r"(64)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tmem_base = *sTmem;
  const uint32_t bar0 = cv_smem_u32(sBar);
  const uint32_t brick_sm = cv_smem_u32(sm + L.brick), w_sm = cv_smem_u32(sm + L.w);
  const float4* wsrc = reinterpret_cast<const float4*>(P.w) + (size_t)ntile * n_chunks * taps * 128;
  const bool resident = n_chunks == 2;       // the two weight slots hold the whole filter: loaded once per CTA
  constexpr int total_items = kBvox * 4;
  const int q = tid & 3;
  // epilogue mapping: warp w reads TMEM lane quarter w % 4, column group w / 4 (8 of the 32 output channels)
  const int lq = warp & 3, cg = warp >> 2;
  const int m = lq * 32 + lane;
  const int co0 = ntile * 32 + 8 * cg;
  float acc_s[8], acc_q[8];                  // this thread's running (sum, sumsq) of its 8 channels over the CTA's tiles
#pragma unroll
  for (int j = 0; j < 8; ++j) { acc_s[j] = 0.f; acc_q[j] = 0.f; }

  auto epilogue = [&](int tile, int acc) {
    int t = tile;
    const int tx = t % P.tiles_x; t /= P.tiles_x;
    const int ty = t % P.tiles_y;
    const int z = t / P.tiles_y;
    const int gy = ty * kCvTileY + (m >> 3), gx = tx * kCvTileX + (m & 7);
    const bool valid = gy < P.H && gx < P.W;
    uint32_t r[8];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(tmem_base + ((uint32_t)(32 * lq) << 16) + (uint32_t)(32 * acc + 8 * cg))
                 : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
    float o[8];
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float v = __uint_as_float(r[j]);
      if (P.bias) v += __ldg(P.bias + co0 + j);
      if (P.relu) v = fmaxf(v, 0.0f);
      o[j] = valid ? v : 0.0f;
    }
    if (valid) {
      float4* dst = reinterpret_cast<float4*>(P.y + ((((size_t)n * P.D + z) * P.H + gy) * P.W + gx) * P.Cout + co0);
      dst[0] = make_float4(o[0], o[1], o[2], o[3]);
      dst[1] = make_float4(o[4], o[5], o[6], o[7]);
    }
    if (P.out_stats) {
#pragma unroll
      for (int j = 0; j < 8; ++j) { acc_s[j] += o[j]; acc_q[j] = fmaf(o[j], o[j], acc_q[j]); }
    }
  };

  // brick-relative coordinates of this thread's items (the same for every tile): z | y << 8 | x << 16, or -1
  int rel[kCvItems];
#pragma unroll
  for (int u = 0; u < kCvItems; ++u) {
    const int i = ltid + u * kCvLoaders;
    const int v = i >> 2;
    const int bxv = v % bx_ext, r = v / bx_ext;
    rel[u] = (i < total_items && !issuer) ? ((r / by_ext) | ((r % by_ext) << 8) | (bxv << 16)) : -1;
  }

  // ---- persistent loop over this CTA's tiles; g counts chunk steps (brick buffer / weight slot = g & 1) ----
  if (issuer) {
    // ===== MMA issuer warp: weights (TMA bulk copies) + tcgen05.mma; never touches the bricks =====
    uint32_t elected;
    asm volatile("{\n.reg .b32 rx;\n.reg .pred px;\nelect.sync rx|px, 0xffffffff;\nselp.u32 %0, 1, 0, px;\n}\n" : "=r"(elected));
    if (elected) {
      int g = 0, it = 0;
      for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
        const int acc = it & 1;
        for (int ch = 0; ch < n_chunks; ++ch, ++g) {
          const int b = g & 1;
          const bool load_w = resident ? (g < n_chunks) : true;    // resident: slot b == chunk b, filled during the first tile
          if (load_w) {
            if (g >= 2) cv_mbar_wait(bar0 + 8 * b, (uint32_t)(((g >> 1) - 1) & 1));   // MMAs that read weight slot b are done
            const uint32_t bytes = (uint32_t)taps * 2048u;
            const float4* src = wsrc + (size_t)ch * taps * 128;
            const uint32_t wb = bar0 + 8 * (2 + b);
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(wb), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                             w_sm + (uint32_t)(b * L.wslot)),
                         "l"(src), "r"(bytes), "r"(wb)
                         : "memory");
          }
          cv_mbar_wait(bar0 + 8 * (6 + b), (uint32_t)((g >> 1) & 1));                  // brick buffer b filled by the workers
          cv_mbar_wait(bar0 + 8 * (2 + b), (uint32_t)((resident ? 0 : (g >> 1)) & 1)); // weights of slot b landed
          asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
          const uint32_t abase = brick_sm + (uint32_t)(b * L.brick_bytes), wbase = w_sm + (uint32_t)(b * L.wslot);
          const uint32_t d = tmem_base + (uint32_t)(32 * acc);
          // descriptors differ from one MMA to the next only in the start-address field (16-byte units, bits 0-13;
          // shared memory is < 256 KB so the field never carries): one 64-bit add of a compile-time constant each
          const uint64_t adesc0 = cv_desc(abase, kPlane, kRowPitch), bdesc0 = cv_desc(wbase, 512, 128);
#pragma unroll
          for (int tap = 0; tap < taps; ++tap) {
            constexpr int kk = KSIZE;
            const int dx = tap % kk, dy = (tap / kk) % kk, dz = tap / (kk * kk);
#pragma unroll
            for (int ks = 0; ks < 2; ++ks) {
              const uint64_t aoff = (uint64_t)((((dz * by_ext + dy) * bx_ext + dx) * 16 + ks * 2 * kPlane) >> 4);
              const uint64_t boff = (uint64_t)((tap * 2048 + ks * 1024) >> 4);
              cv_mma_ss(d, adesc0 + aoff, bdesc0 + boff, (tap | ks) ? 1u : (ch ? 1u : 0u));
            }
          }
          cv_commit(bar0 + 8 * b);                                  // brick buffer / weight slot b free again
          if (ch == n_chunks - 1) cv_commit(bar0 + 8 * (4 + acc));  // accumulator `acc` complete
        }
      }
    }
    __syncwarp();
  } else {
    // ===== worker warps: fill the bricks, run the epilogues =====
    int g = 0, it = 0, prev_tile = -1;
    for (int tile = blockIdx.x; tile < P.n_tiles; tile += gridDim.x, ++it) {
      int t = tile;
      const int tx = t % P.tiles_x; t /= P.tiles_x;
      const int ty = t % P.tiles_y;
      const int z = t / P.tiles_y;
      const int y0 = ty * kCvTileY, x0 = tx * kCvTileX;
      const int acc = it & 1;
      // this thread's brick items (i = tid + u * 512 -> voxel i / 4, channel quad i % 4 == tid % 4): voxel index in
      // the full-resolution source and in the half-resolution one, or -1 outside the volume
      int voxA[kCvItems], voxB[kCvItems];
#pragma unroll
      for (int u = 0; u < kCvItems; ++u) {
        const int gz = z + (rel[u] & 0xff) - hz, gy = y0 + ((rel[u] >> 8) & 0xff) - h, gx = x0 + ((rel[u] >> 16) & 0xff) - h;
        const bool inb = rel[u] >= 0 && gz >= 0 && gz < P.D && gy >= 0 && gy < P.H && gx >= 0 && gx < P.W;
        voxA[u] = inb ? (int)((((size_t)n * P.D + gz) * P.H + gy) * P.W + gx) : -1;
        voxB[u] = -1;
        if (inb && P.C2 > 0) {   // ATen nearest: src = min(floor(dst * in / out), in - 1)
          const int sz = min(gz * P.D2 / P.D, P.D2 - 1), sy = min(gy * P.H2 / P.H, P.H2 - 1), sx = min(gx * P.W2 / P.W, P.W2 - 1);
          voxB[u] = (int)((((size_t)n * P.D2 + sz) * P.H2 + sy) * P.W2 + sx);
        }
      }
      for (int ch = 0; ch < n_chunks; ++ch, ++g) {
        const int b = g & 1;
        CV_STAMP(1);   // chunk start
        // the MMAs of chunk step g-2 read brick buffer b: they must be done before it is refilled
        if (g >= 2) cv_mbar_wait(bar0 + 8 * b, (uint32_t)(((g >> 1) - 1) & 1));
        CV_STAMP(2);   // buffer free
        // ---- halo brick of 16 input channels: GroupNorm-apply, TF32 rounding, zero padding ----
        {
          const int c0 = ch * kCvKC;
          const bool second = c0 >= P.C1;                       // channels from the half-resolution tensor (upsample + concat)
          const float* src = second ? P.x2 : P.x;
          const int Cs = second ? P.C2 : P.C1, cs0 = second ? c0 - P.C1 : c0;
          const float4 sc = *reinterpret_cast<const float4*>(sScale + c0 + 4 * q);
          const float4 sh = *reinterpret_cast<const float4*>(sShift + c0 + 4 * q);
          unsigned char* bdst = sm + L.brick + b * L.brick_bytes + q * kPlane;
          float4 val[kCvItems];
#pragma unroll
          for (int u = 0; u < kCvItems; ++u) {
            const int vox = second ? voxB[u] : voxA[u];
            val[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (vox >= 0) val[u] = __ldg(reinterpret_cast<const float4*>(src + (size_t)vox * Cs + cs0) + q);
          }
#pragma unroll
          for (int u = 0; u < kCvItems; ++u) {
            const int i = ltid + u * kCvLoaders;
            if (i < total_items) {
              float4 o = val[u];
              if ((second ? voxB[u] : voxA[u]) >= 0) {
                o.x = cv_tf32(fmaf(o.x, sc.x, sh.x));
                o.y = cv_tf32(fmaf(o.y, sc.y, sh.y));
                o.z = cv_tf32(fmaf(o.z, sc.z, sh.z));
                o.w = cv_tf32(fmaf(o.w, sc.w, sh.w));
              }
              *reinterpret_cast<float4*>(bdst + (i >> 2) * 16) = o;
            }
          }
        }
        CV_STAMP(3);   // brick stored
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");    // generic-proxy stores -> visible to the tensor core
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncwarp();
        if (lane == 0) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar0 + 8 * (6 + b)) : "memory");
        CV_STAMP(4);   // signalled
      }
      // while this tile's MMAs run: epilogue of the previous tile (other accumulator)
      if (prev_tile >= 0) {
        cv_mbar_wait(bar0 + 8 * (4 + (acc ^ 1)), (uint32_t)(((it - 1) >> 1) & 1));
        CV_STAMP(6);   // previous accumulator complete
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        epilogue(prev_tile, acc ^ 1);
        CV_STAMP(7);   // epilogue done
      }
      prev_tile = tile;
    }
    if (prev_tile >= 0) {
      const int last = it - 1;
      cv_mbar_wait(bar0 + 8 * (4 + (last & 1)), (uint32_t)((last >> 1) & 1));
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      epilogue(prev_tile, last & 1);
    }
  }
  if (P.out_stats) {
    if (!issuer) {
      // per-channel sums over the warp's 32 voxel rows: all-reduce over lane bits 4 and 3, reduce-scatter over bits 2..0
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float a = acc_s[j], b = acc_q[j];
        a += __shfl_xor_sync(0xffffffffu, a, 16); b += __shfl_xor_sync(0xffffffffu, b, 16);
        a += __shfl_xor_sync(0xffffffffu, a, 8);  b += __shfl_xor_sync(0xffffffffu, b, 8);
        acc_s[j] = a; acc_q[j] = b;
      }
#pragma unroll
      for (int w = 4; w >= 1; w >>= 1) {      // after the step with width w a lane keeps w values
        const bool upper = (lane & w) != 0;
#pragma unroll
        for (int j = 0; j < w; ++j) {
          const float send_s = upper ? acc_s[j] : acc_s[j + w], keep_s = upper ? acc_s[j + w] : acc_s[j];
          const float send_q = upper ? acc_q[j] : acc_q[j + w], keep_q = upper ? acc_q[j + w] : acc_q[j];
          acc_s[j] = keep_s + __shfl_xor_sync(0xffffffffu, send_s, w);
          acc_q[j] = keep_q + __shfl_xor_sync(0xffffffffu, send_q, w);
        }
      }
      if (lane < 8) {                         // lane l holds channel l & 7
        atomicAdd(sStat + 8 * cg + lane, acc_s[0]);
        atomicAdd(sStat + 32 + 8 * cg + lane, acc_q[0]);
      }
    }
    __syncthreads();
    if (tid < 64) {
      const int c = tid & 31, which = tid >> 5;
      atomicAdd(P.out_stats + ((size_t)n * P.Cout + ntile * 32 + c) * 2 + which, (double)sStat[tid]);
    }
  }
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(64) : "memory");
}

// MaxPool3d(2) over channels-last activations + per-channel (sum, sumsq) of the result.
// One thread per (output voxel, channel quad).
__global__ void __launch_bounds__(256) maxpool2_cl_kernel(const float* __restrict__ x, float* __restrict__ y, int N, int D,
                                                          int H, int W, int C, double* __restrict__ stats) {
  const int C4 = C >> 2, Do = D >> 1, Ho = H >> 1, Wo = W >> 1;
  const long long total = (long long)N * Do * Ho * Wo * C4;
  extern __shared__ float pool_sm[];      // [2][C]
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) pool_sm[i] = 0.f;
  __syncthreads();
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (long long)gridDim.x * blockDim.x) {
    const int q = (int)(t % C4);
    long long v = t / C4;
    const int xo = (int)(v % Wo); v /= Wo;
    const int yo = (int)(v % Ho); v /= Ho;
    const int zo = (int)(v % Do);
    const int n = (int)(v / Do);
    float4 m = make_float4(-CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F, -CUDART_INF_F);
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int zi = 2 * zo + (k >> 2), yi = 2 * yo + ((k >> 1) & 1), xi = 2 * xo + (k & 1);
      const float4 a = __ldg(reinterpret_cast<const float4*>(x + ((((size_t)n * D + zi) * H + yi) * W + xi) * C) + q);
      m.x = fmaxf(m.x, a.x); m.y = fmaxf(m.y, a.y); m.z = fmaxf(m.z, a.z); m.w = fmaxf(m.w, a.w);
    }
    reinterpret_cast<float4*>(y + ((((size_t)n * Do + zo) * Ho + yo) * Wo + xo) * C)[q] = m;
    if (stats) {   // N == 1 per launch when statistics are wanted (the host loops over samples)
      atomicAdd(pool_sm + 4 * q, m.x); atomicAdd(pool_sm + 4 * q + 1, m.y);
      atomicAdd(pool_sm + 4 * q + 2, m.z); atomicAdd(pool_sm + 4 * q + 3, m.w);
      atomicAdd(pool_sm + C + 4 * q, m.x * m.x); atomicAdd(pool_sm + C + 4 * q + 1, m.y * m.y);
      atomicAdd(pool_sm + C + 4 * q + 2, m.z * m.z); atomicAdd(pool_sm + C + 4 * q + 3, m.w * m.w);
    }
  }
  if (stats) {
    __syncthreads();
    for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
      const int c = i % C, which = i / C;
      atomicAdd(stats + (size_t)c * 2 + which, (double)pool_sm[i]);
    }
  }
}

// per-channel (sum, sumsq) of a channels-last tensor [S][C] (one sample)
__global__ void __launch_bounds__(256) channel_stats_cl_kernel(const float* __restrict__ x, long long S, int C,
                                                               double* __restrict__ stats) {
  extern __shared__ float st_sm[];        // [2][C]
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) st_sm[i] = 0.f;
  __syncthreads();
  const int C4 = C >> 2;
  // a thread keeps one channel quad (blockDim.x is a multiple of C4) and strides over the voxels
  const int q = threadIdx.x % C4, lanes = blockDim.x / C4;
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f), ss = s;
  for (long long v = (long long)blockIdx.x * lanes + threadIdx.x / C4; v < S; v += (long long)gridDim.x * lanes) {
    const float4 a = __ldg(reinterpret_cast<const float4*>(x + (size_t)v * C) + q);
    s.x += a.x; s.y += a.y; s.z += a.z; s.w += a.w;
    ss.x = fmaf(a.x, a.x, ss.x); ss.y = fmaf(a.y, a.y, ss.y); ss.z = fmaf(a.z, a.z, ss.z); ss.w = fmaf(a.w, a.w, ss.w);
  }
  atomicAdd(st_sm + 4 * q, s.x); atomicAdd(st_sm + 4 * q + 1, s.y); atomicAdd(st_sm + 4 * q + 2, s.z); atomicAdd(st_sm + 4 * q + 3, s.w);
  atomicAdd(st_sm + C + 4 * q, ss.x); atomicAdd(st_sm + C + 4 * q + 1, ss.y); atomicAdd(st_sm + C + 4 * q + 2, ss.z);
  atomicAdd(st_sm + C + 4 * q + 3, ss.w);
  __syncthreads();
  for (int i = threadIdx.x; i < 2 * C; i += blockDim.x) {
    const int c = i % C, which = i / C;
    atomicAdd(stats + (size_t)c * 2 + which, (double)st_sm[i]);
  }
}

}  // namespace vtaco

using namespace vtaco;

extern "C" int vtaco_conv3d_cl(const vtaco_conv3d_args* a, void* stream) {
  if (!a || !a->x || !a->w_packed || !a->y) return VTACO_ERR_INVALID_ARG;
  if (a->N < 1 || a->D < 1 || a->H < 1 || a->W < 1 || a->C1 < 1 || a->C2 < 0 || a->Cout < 1) return VTACO_ERR_INVALID_ARG;
  if (a->ksize != 1 && a->ksize != 3) return VTACO_ERR_UNSUPPORTED;
  const int kz = a->ksize_z ? a->ksize_z : a->ksize;
  if (kz != 1 && kz != a->ksize) return VTACO_ERR_UNSUPPORTED;
  const int Cin = a->C1 + a->C2;
  if (a->C1 % kCvKC || a->C2 % kCvKC || a->Cout % 32 || Cin > kCvMaxCin) return VTACO_ERR_UNSUPPORTED;
  if (a->C2 > 0 && (!a->x2 || a->D2 < 1 || a->H2 < 1 || a->W2 < 1)) return VTACO_ERR_INVALID_ARG;
  if (a->in_stats && (a->groups < 1 || Cin % a->groups)) return VTACO_ERR_INVALID_ARG;
  ConvParams P = {};
  P.x = a->x; P.x2 = a->x2; P.w = a->w_packed; P.bias = a->bias; P.in_stats = a->in_stats; P.gamma = a->gamma; P.beta = a->beta;
  P.y = a->y; P.out_stats = a->out_stats;
  P.N = a->N; P.D = a->D; P.H = a->H; P.W = a->W; P.C1 = a->C1; P.C2 = a->C2; P.D2 = a->D2; P.H2 = a->H2; P.W2 = a->W2;
  P.Cout = a->Cout; P.ksize = a->ksize; P.groups = a->groups; P.relu = a->relu ? 1 : 0; P.eps = a->eps;
  P.tiles_x = (a->W + kCvTileX - 1) / kCvTileX;
  P.tiles_y = (a->H + kCvTileY - 1) / kCvTileY;
  const long long tiles = (long long)P.tiles_x * P.tiles_y * a->D;
  if (tiles > 0x7fffffffll || a->Cout / 32 > 65535 || a->N > 65535) return VTACO_ERR_UNSUPPORTED;
  // the kernel keeps voxel indices (n, z, y, x flattened) of both inputs in 32-bit integers
  if ((long long)a->N * a->D * a->H * a->W > 0x7fffffffll) return VTACO_ERR_UNSUPPORTED;
  if (a->C2 > 0 && (long long)a->N * a->D2 * a->H2 * a->W2 > 0x7fffffffll) return VTACO_ERR_UNSUPPORTED;
  P.n_tiles = (int)tiles;
  const CvSmem L = cv_layout(a->ksize, kz, Cin);
  if (L.total > 227 * 1024) return VTACO_ERR_UNSUPPORTED;
  VTACO_CUDA_CHECK(smem_opt_in((const void*)conv3d_tc_kernel<3, 3>, 227 * 1024));
  VTACO_CUDA_CHECK(smem_opt_in((const void*)conv3d_tc_kernel<3, 1>, 227 * 1024));
  VTACO_CUDA_CHECK(smem_opt_in((const void*)conv3d_tc_kernel<1, 1>, 227 * 1024));
  // persistent CTAs: one per SM in total, split over the (out-channel tile, sample) pairs
  long long gx = num_sms() / ((long long)(a->Cout / 32) * a->N);
  if (gx < 1) gx = 1;
  if (gx > tiles) gx = tiles;
  dim3 grid((unsigned)gx, (unsigned)(a->Cout / 32), (unsigned)a->N);
  static const bool want_trace = getenv("VTACO_CV_TRACE") != nullptr;
  if (want_trace) {
    VTACO_CUDA_CHECK(cudaMalloc(&P.trace, 2048 * sizeof(long long)));
    VTACO_CUDA_CHECK(cudaMemsetAsync(P.trace, 0, 2048 * sizeof(long long), (cudaStream_t)stream));
  }
  if (a->ksize == 3 && kz == 3) conv3d_tc_kernel<3, 3><<<grid, kCvThreads, L.total, (cudaStream_t)stream>>>(P);
  else if (a->ksize == 3) conv3d_tc_kernel<3, 1><<<grid, kCvThreads, L.total, (cudaStream_t)stream>>>(P);
  else conv3d_tc_kernel<1, 1><<<grid, kCvThreads, L.total, (cudaStream_t)stream>>>(P);
  VTACO_LAUNCH_CHECK();
  if (P.trace) {   // debug: average cycles between consecutive stamps, per (from -> to) slot pair
    static long long hbuf[2048];
    VTACO_CUDA_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
    VTACO_CUDA_CHECK(cudaMemcpy(hbuf, P.trace, sizeof(hbuf), cudaMemcpyDeviceToHost));
    cudaFree(P.trace);
    double sum[8][8] = {{0}};
    long long cnt[8][8] = {{0}};
    for (int i = 1; i < 2048 && hbuf[i]; ++i) {
      const int f = (int)(hbuf[i - 1] >> 56) & 7, t = (int)(hbuf[i] >> 56) & 7;
      const long long d = (hbuf[i] & 0x00ffffffffffffffll) - (hbuf[i - 1] & 0x00ffffffffffffffll);
      if (d >= 0 && d < 10000000) { sum[f][t] += (double)d; cnt[f][t]++; }
    }
    fprintf(stderr, "[vtaco conv trace] Cin=%d Cout=%d %dx%dx%d k=%d grid=(%u,%u)\n", Cin, a->Cout, a->D, a->H, a->W, a->ksize, grid.x, grid.y);
    for (int f = 0; f < 8; ++f)
      for (int t = 0; t < 8; ++t)
        if (cnt[f][t]) fprintf(stderr, "[vtaco conv trace]   %d -> %d : %8.0f cycles (n=%lld)\n", f, t, sum[f][t] / cnt[f][t], cnt[f][t]);
  }
  return VTACO_OK;
}

extern "C" int vtaco_maxpool2_cl(const float* x, float* y, int32_t N, int32_t D, int32_t H, int32_t W, int32_t C,
                                 double* stats, void* stream) {
  if (!x || !y || N < 1 || D < 2 || H < 2 || W < 2 || C < 4 || (C & 3)) return VTACO_ERR_INVALID_ARG;
  if ((D | H | W) & 1) return VTACO_ERR_UNSUPPORTED;
  if (stats && N != 1) return VTACO_ERR_UNSUPPORTED;
  const long long total = (long long)N * (D / 2) * (H / 2) * (W / 2) * (C / 4);
  long long blocks = (total + 255) / 256;
  const long long cap = (long long)num_sms() * 8;
  if (blocks > cap) blocks = cap;
  maxpool2_cl_kernel<<<(unsigned)blocks, 256, 2 * C * sizeof(float), (cudaStream_t)stream>>>(x, y, N, D, H, W, C, stats);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int vtaco_channel_stats_cl(const float* x, int64_t S, int32_t C, double* stats, void* stream) {
  if (!x || !stats || S < 1 || C < 4 || (C & 3) || 256 % (C / 4)) return VTACO_ERR_INVALID_ARG;
  long long blocks = (S * (C / 4) + 255) / 256;
  const long long cap = (long long)num_sms() * 4;
  if (blocks > cap) blocks = cap;
  channel_stats_cl_kernel<<<(unsigned)blocks, 256, 2 * C * sizeof(float), (cudaStream_t)stream>>>(x, S, C, stats);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}
