// tcgen05 / TMEM PTX wrappers and the gather, set-up and tracing helpers shared by the tensor-core decoder kernels
// (decoder_tc.cu: 3 tiles per SM, 3xTF32; decoder_tc4.cu: 4 tiles per SM, TF32 + BF16 residual).
#pragma once
#include "decoder_common.cuh"
#include <cuda_bf16.h>

namespace vtaco {

constexpr int kTcThreads = 384;
constexpr int kTcGroups = 3;
constexpr int kTcTile = 128;
constexpr int kColsPerGroup = 168;   // C_hi 0, C_lo 32, X_hi 64, X_lo 96, ones 128 (8), D 136 (32)
constexpr int kStageStride = 36;     // floats per staged query row (conflict-free LDS.128)
constexpr uint32_t kIdescTf32 = (1u << 4) | (2u << 7) | (2u << 10) | (4u << 17) | (8u << 24);  // F32 acc, TF32 x TF32, K-major, N=32, M=128
constexpr uint32_t kIdescBf16 = (1u << 4) | (1u << 7) | (1u << 10) | (4u << 17) | (8u << 24);  // F32 acc, BF16 x BF16 (kind::f16, K=16)

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "LAB_WAIT:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE;\n"
      "bra LAB_WAIT;\n"
      "DONE:\n"
      "}\n" ::"r"(bar), "r"(parity)
      : "memory");
}
// exactly one lane of a converged warp; unlike `lane == 0` the compiler knows a single lane is
// active, so tcgen05.mma sequences compile to back-to-back UTCHMMA without per-instruction
// ELECT / retry loops (measured: ~45 -> ~16 cycles of issue per MMA)
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .b32 rx;\n"
      ".reg .pred px;\n"
      "elect.sync rx|px, 0xffffffff;\n"
      "selp.u32 %0, 1, 0, px;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tc_wait_st() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void group_sync(int g) { asm volatile("bar.sync %0, 128;" ::"r"(g + 1) : "memory"); }

__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar) : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem desc]
__device__ __forceinline__ void tc_mma_ts(uint32_t d, uint32_t a, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d), "r"(a), "l"(bdesc), "r"(kIdescTf32), "r"(accumulate)
      : "memory");
}
// same with BF16 operands (two per 32-bit TMEM column, K = 16 per instruction)
__device__ __forceinline__ void tc_mma_ts_bf16(uint32_t d, uint32_t a, uint64_t bdesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n"
      "}\n" ::"r"(d), "r"(a), "l"(bdesc), "r"(kIdescBf16), "r"(accumulate)
      : "memory");
}
// K-major, no swizzle: 8 rows x 16 B core matrices; K-chunk stride 512 B, 8-row-group stride 128 B
__device__ __forceinline__ uint64_t make_bdesc(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fff);
  d |= (uint64_t)(512 >> 4) << 16;   // leading (K) byte offset
  d |= (uint64_t)(128 >> 4) << 32;   // stride (N) byte offset
  d |= (uint64_t)1 << 46;            // descriptor version (Blackwell)
  return d;
}

#define TC_R32(r) r[0], r[1], r[2], r[3], r[4], r[5], r[6], r[7], r[8], r[9], r[10], r[11], r[12], r[13], r[14], r[15], \
                  r[16], r[17], r[18], r[19], r[20], r[21], r[22], r[23], r[24], r[25], r[26], r[27], r[28], r[29], r[30], r[31]
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%32], "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31};"
      ::"r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]),
        "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]),
        "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31]), "r"(taddr)
      : "memory");
}

// Activation split: hi = x with the 13 low mantissa bits cleared (exactly what the tensor core
// keeps of an fp32 container), lo = x - hi (exact).  cvt.rna.tf32 would cost 4 SASS ops per
// element (it is emulated); truncation is 1 LOP3 and leaves |lo| <= 2^-10 |x|, whose own
// truncation to TF32 is a 2^-21 relative error — far inside the 1e-4 parity bar.
__device__ __forceinline__ uint32_t trunc_tf32(float x) { return __float_as_uint(x) & 0xffffe000u; }

__device__ __forceinline__ uint32_t pack_bf16(float k_even, float k_odd) {   // element 2c in the low half
  const __nv_bfloat162 v = __floats2bfloat162_rn(k_even, k_odd);
  return *reinterpret_cast<const uint32_t*>(&v);
}

// x[32] (fp32) -> operands stored to TMEM columns [col, col+32) and [col+32, col+64):
//   3xTF32 : hi | lo (both TF32 in fp32 containers)
//   mixed  : hi (TF32) | correction operand in BF16, K = 64: bf16(lo[0..31]) then bf16(hi[0..31]),
//            two elements per column.  The main product hi*W_hi stays TF32; lo*W and hi*W_lo are
//            ~2^-11 of it, so BF16's 2^-9 relative rounding leaves a ~2^-19 relative error.
__device__ __forceinline__ void split_store(uint32_t taddr, const float (&x)[32], bool mixed) {
  uint32_t hi[32], lo[32];
#pragma unroll
  for (int j = 0; j < 32; ++j) hi[j] = trunc_tf32(x[j]);
  if (mixed) {
#pragma unroll
    for (int c = 0; c < 16; ++c) {
      lo[c] = pack_bf16(x[2 * c] - __uint_as_float(hi[2 * c]), x[2 * c + 1] - __uint_as_float(hi[2 * c + 1]));
      lo[16 + c] = pack_bf16(__uint_as_float(hi[2 * c]), __uint_as_float(hi[2 * c + 1]));
    }
  } else {
#pragma unroll
    for (int j = 0; j < 32; ++j) lo[j] = __float_as_uint(x[j] - __uint_as_float(hi[j]));
  }
  tmem_st32(taddr, hi);
  tmem_st32(taddr + 32, lo);
}

// ---------------------------------------------------------------------------------------
// Interpolation set-up computed ONCE per query by its owner thread and broadcast to the 8
// lanes that fetch the taps (the SIMT kernel recomputes it in every lane).
// ---------------------------------------------------------------------------------------
struct TapInfo {
  int base;       // index (in taps) of corner (x0,y0[,z0])
  int step;       // bit0: x0+1 < R, bit1: y0+1 < R, bit2: z0+1 < R   (else the weight is 0 and the address is clamped)
  float fx, fy, fz;
};
__device__ __forceinline__ TapInfo tap_volume(float ux, float uy, float uz, int R, bool nearest) {
  const float tx = unnormalize(ux, R), ty = unnormalize(uy, R), tz = unnormalize(uz, R);
  TapInfo t;
  if (nearest) {
    const int x = (int)nearbyintf(tx), y = (int)nearbyintf(ty), z = (int)nearbyintf(tz);
    t.base = (z * R + y) * R + x; t.step = 0; t.fx = t.fy = t.fz = 0.f;
    return t;
  }
  const float flx = floorf(tx), fly = floorf(ty), flz = floorf(tz);
  const int x0 = (int)flx, y0 = (int)fly, z0 = (int)flz;
  t.base = (z0 * R + y0) * R + x0;
  t.step = (int)(x0 + 1 < R) | ((int)(y0 + 1 < R) << 1) | ((int)(z0 + 1 < R) << 2);
  t.fx = tx - flx; t.fy = ty - fly; t.fz = tz - flz;
  return t;
}
__device__ __forceinline__ TapInfo tap_plane(float ua, float ub, int R, bool nearest) {
  const float tx = unnormalize(ua, R), ty = unnormalize(ub, R);
  TapInfo t;
  t.fz = 0.f;
  if (nearest) {
    const int x = (int)nearbyintf(tx), y = (int)nearbyintf(ty);
    t.base = y * R + x; t.step = 0; t.fx = t.fy = 0.f;
    return t;
  }
  const float flx = floorf(tx), fly = floorf(ty);
  const int x0 = (int)flx, y0 = (int)fly;
  t.base = y0 * R + x0;
  t.step = (int)(x0 + 1 < R) | ((int)(y0 + 1 < R) << 1);
  t.fx = tx - flx; t.fy = ty - fly;
  return t;
}
__device__ __forceinline__ TapInfo tap_bcast(const TapInfo& t, int src) {
  TapInfo r;
  r.base = __shfl_sync(kFull, t.base, src);
  r.step = __shfl_sync(kFull, t.step, src);
  r.fx = __shfl_sync(kFull, t.fx, src);
  r.fy = __shfl_sync(kFull, t.fy, src);
  r.fz = __shfl_sync(kFull, t.fz, src);
  return r;
}
// ATen corner order / weights (see sample_volume in decoder_common.cuh); the weight of a
// clamped corner is exactly 0 because its fraction is 0.
__device__ __forceinline__ float4 fetch_volume(const float4* __restrict__ vol, int R, const TapInfo& t, bool nearest) {
  if (nearest) return __ldg(vol + (size_t)t.base * 8);
  const int dx = (t.step & 1) ? 8 : 0, dy = (t.step & 2) ? R * 8 : 0, dz = (t.step & 4) ? R * R * 8 : 0;
  const float4* p = vol + (size_t)t.base * 8;
  const float4 v000 = __ldg(p), v001 = __ldg(p + dx), v010 = __ldg(p + dy), v011 = __ldg(p + dy + dx);
  const float4 v100 = __ldg(p + dz), v101 = __ldg(p + dz + dx), v110 = __ldg(p + dz + dy), v111 = __ldg(p + dz + dy + dx);
  const float fx1 = (t.step & 1) ? t.fx : 0.f, fy1 = (t.step & 2) ? t.fy : 0.f, fz1 = (t.step & 4) ? t.fz : 0.f;
  const float fx0 = 1.0f - t.fx, fy0 = 1.0f - t.fy, fz0 = 1.0f - t.fz;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  a = f4_fma(fx0 * fy0 * fz0, v000, a);
  a = f4_fma(fx1 * fy0 * fz0, v001, a);
  a = f4_fma(fx0 * fy1 * fz0, v010, a);
  a = f4_fma(fx1 * fy1 * fz0, v011, a);
  a = f4_fma(fx0 * fy0 * fz1, v100, a);
  a = f4_fma(fx1 * fy0 * fz1, v101, a);
  a = f4_fma(fx0 * fy1 * fz1, v110, a);
  a = f4_fma(fx1 * fy1 * fz1, v111, a);
  return a;
}
__device__ __forceinline__ float4 fetch_plane(const float4* __restrict__ pl, int R, const TapInfo& t, bool nearest) {
  if (nearest) return __ldg(pl + (size_t)t.base * 8);
  const int dx = (t.step & 1) ? 8 : 0, dy = (t.step & 2) ? R * 8 : 0;
  const float4* p = pl + (size_t)t.base * 8;
  const float4 v00 = __ldg(p), v01 = __ldg(p + dx), v10 = __ldg(p + dy), v11 = __ldg(p + dy + dx);
  const float fx1 = (t.step & 1) ? t.fx : 0.f, fy1 = (t.step & 2) ? t.fy : 0.f;
  const float fx0 = 1.0f - t.fx, fy0 = 1.0f - t.fy;
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
  a = f4_fma(fx0 * fy0, v00, a);
  a = f4_fma(fx1 * fy0, v01, a);
  a = f4_fma(fx0 * fy1, v10, a);
  a = f4_fma(fx1 * fy1, v11, a);
  return a;
}

__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%16], {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15};"
      ::"r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]),
        "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_st8(uint32_t taddr, const uint32_t (&r)[8]) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%8], {%0,%1,%2,%3,%4,%5,%6,%7};" ::"r"(r[0]), "r"(r[1]),
               "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(taddr)
               : "memory");
}

// ---------------------------------------------------------------------------------------
// Per-query helpers of the tcgen05 kernels
// ---------------------------------------------------------------------------------------
// Taps of one query in every feature tensor, computed by the thread that owns the query
struct QueryTaps { TapInfo v, p0, p1, p2; bool planes; };
__device__ __forceinline__ QueryTaps query_taps(const DecParams& P, float px, float py, float pz) {
  QueryTaps t;
  if (P.grid) t.v = tap_volume(norm3d(px, P.nc), norm3d(py, P.nc), norm3d(pz, P.nc), P.Rg, P.nearest);
  t.planes = P.plane[0] || P.plane[1] || P.plane[2];
  if (t.planes) {
    const float ux = norm2d(px, P.nc), uy = norm2d(py, P.nc), uz = norm2d(pz, P.nc);
    if (P.plane[0]) t.p0 = tap_plane(ux, uz, P.Rp, P.nearest);
    if (P.plane[1]) t.p1 = tap_plane(ux, uy, P.Rp, P.nearest);
    if (P.plane[2]) t.p2 = tap_plane(uy, uz, P.Rp, P.nearest);
  }
  return t;
}
// c of the query whose taps lane `src` holds, summed over the grid and the planes: float4 `ch` (channels
// 4*ch .. 4*ch+3) of sample b
__device__ __forceinline__ float4 gather_taps(const DecParams& P, QueryTaps t, int src, int b, int ch) {
  float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
  if (P.grid) {
    const int R = P.Rg;
    const float4* vol = reinterpret_cast<const float4*>(P.grid) + (size_t)b * R * R * R * 8 + ch;
    c = fetch_volume(vol, R, tap_bcast(t.v, src), P.nearest);
  }
  if (t.planes) {
    const int R = P.Rp;
    const size_t boff = (size_t)b * R * R * 8 + ch;
    if (P.plane[0]) c = f4_add(c, fetch_plane(reinterpret_cast<const float4*>(P.plane[0]) + boff, R, tap_bcast(t.p0, src), P.nearest));
    if (P.plane[1]) c = f4_add(c, fetch_plane(reinterpret_cast<const float4*>(P.plane[1]) + boff, R, tap_bcast(t.p1, src), P.nearest));
    if (P.plane[2]) c = f4_add(c, fetch_plane(reinterpret_cast<const float4*>(P.plane[2]) + boff, R, tap_bcast(t.p2, src), P.nearest));
  }
  return c;
}

// Separable dense gather (grid only, bilinear): a warp is one z-run of lattice points at fixed (x, y), so the
// (x,y)-bilinear part of the trilinear sample is shared by the run.  The kernels reduce the 4 (x,y) corners once
// per needed z-row into shared memory, then every thread lerps its two z-rows.
struct SepGather {
  int z0, zmin, nz;        // the query's lower z-row; the run needs rows [zmin, zmin + nz)
  int dx, dy;              // float4 offsets of the x+1 / y+1 corners (0 where clamped: their weight is 0)
  float w00, w01, w10, w11, fz0, fz1;
  const float4* col;       // corner (x0, y0) at z = 0: float4 `ch` of the query's sample
};
__device__ __forceinline__ SepGather sep_gather_setup(const DecParams& P, float px, float py, float pz, int qb, int ch) {
  const int R = P.Rg;
  const float tx = unnormalize(norm3d(px, P.nc), R), ty = unnormalize(norm3d(py, P.nc), R);
  const float tz = unnormalize(norm3d(pz, P.nc), R);
  const float flx = floorf(tx), fly = floorf(ty), flz = floorf(tz);
  const int x0 = (int)flx, y0 = (int)fly, z0 = (int)flz;
  const float fx1 = tx - flx, fx0 = (flx + 1.0f) - tx, fy1 = ty - fly, fy0 = (fly + 1.0f) - ty;
  SepGather s;
  s.z0 = z0;
  s.fz1 = tz - flz; s.fz0 = (flz + 1.0f) - tz;
  s.zmin = __shfl_sync(kFull, z0, 0);
  const int zmax = min(__shfl_sync(kFull, z0, 31) + 1, R - 1);
  s.nz = zmax - s.zmin + 1;
  s.dx = (x0 + 1 < R) ? 8 : 0; s.dy = (y0 + 1 < R) ? R * 8 : 0;
  s.w00 = fx0 * fy0; s.w01 = fx1 * fy0; s.w10 = fx0 * fy1; s.w11 = fx1 * fy1;
  s.col = reinterpret_cast<const float4*>(P.grid) + (size_t)qb * R * R * R * 8 + ((size_t)y0 * R + x0) * 8 + ch;
  return s;
}

// Query tq of a tile.  Dense: 2 (x) x 2 (y) x 32 (z) bricks, so a warp is one z-run and its 32 logits are one
// 128-byte store; the axis is read from sAxis where the kernel caches it (axis_sm).  Flat: 128 consecutive queries.
// A padding query (valid = false) reads clamped coordinates and has oidx 0.
struct TileQuery { float px, py, pz; long long oidx; int qb; bool valid; };
__device__ __forceinline__ TileQuery tile_query(const DecParams& P, bool dense, long long tile, int tq,
                                                const float* sAxis, bool axis_sm, int nx) {
  TileQuery q;
  if (dense) {
    unsigned t = (unsigned)tile;                        // n_tiles < 2^31 (checked at launch)
    const int bz = (int)(t % (unsigned)P.t_nbz); t /= (unsigned)P.t_nbz;
    const int by = (int)(t % (unsigned)P.t_nby); t /= (unsigned)P.t_nby;
    const int bx = (int)(t % (unsigned)P.t_nbx);
    q.qb = (int)(t / (unsigned)P.t_nbx);
    const int ix = P.x0 + bx * 2 + (tq >> 6), iy = by * 2 + ((tq >> 5) & 1), iz = bz * 32 + (tq & 31);
    q.valid = (ix < P.t_xend) && (iy < nx) && (iz < nx);
    const int cx = min(ix, nx - 1), cy = min(iy, nx - 1), cz = min(iz, nx - 1);
    q.px = axis_sm ? sAxis[cx] : __ldg(P.axis + cx);
    q.py = axis_sm ? sAxis[cy] : __ldg(P.axis + cy);
    q.pz = axis_sm ? sAxis[cz] : __ldg(P.axis + cz);
    q.oidx = (((long long)q.qb * nx + ix) * nx + iy) * nx + iz;
  } else {
    const long long n = tile * kTcTile + tq;
    q.valid = n < P.total;
    const long long nn = q.valid ? n : 0;
    q.px = __ldg(P.p + nn * 3 + 0);
    q.py = __ldg(P.p + nn * 3 + 1);
    q.pz = __ldg(P.p + nn * 3 + 2);
    q.qb = (int)(nn / P.N);
    q.oidx = nn;
  }
  if (!q.valid) q.oidx = 0;
  return q;
}

// ---------------------------------------------------------------------------------------
// CTA set-up and teardown of the tcgen05 kernels (nthreads: the CTA's thread count)
// ---------------------------------------------------------------------------------------
// sSmall[0, 128): fc_p (or fc_p_img[:, :3]) as Wp[3][32], bp[32]; sSmall[128, ...): the packed tail (fc_out, fc_contact)
__device__ __forceinline__ void load_small(float* sSmall, const DecParams& P, int nb, int tid, int nthreads) {
  for (int i = tid; i < 128; i += nthreads) sSmall[i] = P.weights[(P.use_img ? VTACO_DEC_OFF_WPI : VTACO_DEC_OFF_WP) + i];
  for (int i = tid; i < VTACO_DEC_TAIL; i += nthreads)
    sSmall[128 + i] = P.weights[VTACO_DEC_OFF_BLOCKS + nb * VTACO_DEC_BLOCK_STRIDE + i];
}
// sTip[f][j]: fc_p_img.weight[:, 3:] @ tip_feat[f]
__device__ __forceinline__ void load_tips(float* sTip, const DecParams& P, int tid, int nthreads) {
  if (P.n_tips > 0) {
    for (int o = tid; o < P.n_tips * 32; o += nthreads) {
      const int f = o >> 5, j = o & 31;
      float a = 0.f;
      for (int k = 0; k < 32; ++k)
        a = fmaf(__ldg(P.weights + VTACO_DEC_OFF_WIMG + k * 32 + j), __ldg(P.tip_feat + f * 32 + k), a);
      sTip[o] = a;
    }
  }
}
// one MMA-completion mbarrier per group
__device__ __forceinline__ void init_group_bars(uint64_t* sBars, int n_groups, int tid) {
  if (tid == 0) {
    for (int i = 0; i < n_groups; ++i) mbar_init(smem_u32(sBars + i), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
}
// All 512 TMEM columns (one CTA per SM), allocated by warp 0; ends with a CTA barrier and returns the base address.
__device__ __forceinline__ uint32_t tmem_alloc_all(uint32_t* sTmem, int warp) {
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(sTmem)), "r"(512)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  return __shfl_sync(kFull, *sTmem, 0);
}
__device__ __forceinline__ void tmem_free_all(uint32_t tmem_base, int warp) {
  tc_fence_before();
  __syncthreads();
  if (warp == 0) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(512) : "memory");
  }
}

// ---------------------------------------------------------------------------------------
// Debug-only phase tracing (VTACO_TC_TRACE=1): clock64 stamps of warp 0 of block 0, the slot number in the top
// byte.  `on` enables a stamp; the kernel provides trace, trace_n, warp and lane.
// ---------------------------------------------------------------------------------------
constexpr int kTraceSlots = 4096;
#define TC_STAMP(on, slot)                                                             \
  do {                                                                                 \
    if ((on) && blockIdx.x == 0 && warp == 0 && lane == 0 && trace_n < kTraceSlots)    \
      trace[trace_n++] = ((long long)(slot) << 56) | (clock64() & 0x00ffffffffffffffll); \
  } while (0)
// *trace = a zeroed stamp buffer when VTACO_TC_TRACE is set, else nullptr
int tc_trace_begin(long long** trace, cudaStream_t stream);
// nothing without a buffer; else waits for the kernel, prints the average cycles between consecutive stamps per
// (from -> to) slot pair as "[vtaco <tag> trace]" lines on stderr, and frees the buffer
int tc_trace_end(long long* trace, const char* tag, cudaStream_t stream);

// Tiles of the tcgen05 kernels (see tile_query); the kernels count tiles in 32 bits.
inline int set_tc_tiles(DecParams& P, bool dense) {
  if (dense) {
    P.t_xend = P.x1;
    P.t_nbz = (P.nx + 31) / 32;
    P.t_nby = (P.nx + 1) / 2;
    P.t_nbx = (P.x1 - P.x0 + 1) / 2;
    P.n_tiles = (long long)P.B * P.t_nbx * P.t_nby * P.t_nbz;
  } else {
    P.n_tiles = (P.total + kTcTile - 1) / kTcTile;
  }
  return P.n_tiles < (1ll << 31) ? VTACO_OK : VTACO_ERR_UNSUPPORTED;
}

}  // namespace vtaco
