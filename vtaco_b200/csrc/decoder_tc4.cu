// Fused LocalDecoder on tcgen05, FOUR 128-query tiles in flight per SM (variant 7, the default).
//
// Same contract as decoder.cu / decoder_tc.cu (reference src/conv_onet/models/decoder.py:71-161).
// Why a third tensor-core kernel: ncu on decoder_tc2_kernel (profiles/decoder_tc_ncu_summary.json)
// shows the tensor pipe 52 % busy and 40 % of all warp samples waiting on the MMA mbarrier — the
// kernel is bound by the per-step dependency chain (st -> fence -> barrier -> MMA -> commit ->
// mbarrier -> ld, ~1 750 cycles of which ~280 are tensor work) with only 3 tiles per SM to overlap,
// and 3 is what TMEM allows at 168 columns per tile.  This kernel makes a tile fit 128 columns, so
// that 4 tiles (32 warps, 1 024 threads) share an SM:
//   * operands are split x = hi + lo with hi = tf32_trunc(x) in an fp32 container (32 columns) and
//     lo = x - hi (exact, |lo| <= 2^-10 |x|) rounded to BF16, two per column (16 columns);
//   * a 32x32 product is  hi*W_hi + hi*W_lo  (kind::tf32, 4 + 4 MMAs of K = 8)  +  lo*bf16(W)
//     (kind::f16, 2 MMAs of K = 16): 10 MMAs instead of 12, error terms ~2^-19 relative
//     (bf16 rounding of lo and of W under a 2^-10 factor; the dropped lo*W_lo is 2^-21);
//   * biases need no ones-block (8 columns in the 3-tile kernel): a thread writes the NEXT step's bias into its own
//     accumulator columns right after reading them (one tcgen05.st.x16), and every MMA of a step accumulates;
//   * columns per tile: C_hi 0 | C_lo 32 | X_hi 48 | X_lo 80 | D 96..127;
//   * the 3-wide input layer is two K = 8 MMAs as well (A = (p, 1, p_lo, 0) in the X columns of step 0);
//   * the 165 KB of operand blocks arrive by TMA bulk copies that overlap TMEM allocation and the first gather;
//   * with 8 warps per scheduler, time follows the instruction count: packed FADD2 / FFMA2 arithmetic,
//     2*relu(x) = x + |x| (half-scaled fc_0 / fc_1), 16-wide tcgen05.st, descriptors as base + immediate, the
//     network depth 5 as a compile-time constant, one polling warp per tile (DESIGN.md 4.1 has the measurements).
// Two threads per query, the separable dense gather, the step structure and the elected issuer rotating over
// the warps of a group are decoder_tc2_kernel's.
#include "decoder_tc_common.cuh"

namespace vtaco {

constexpr int kT4Threads = 1024;
constexpr int kT4Groups = 4;
constexpr int kT4Cols = 128;
constexpr int kT4StageRows = 24;          // staged z-rows per warp (separable gather) / 16 queries per pass (generic)
constexpr int kT4Mode = VTACO_DEC_TC_MODE_TILE4;   // weights_tc is copied to shared memory as it is
constexpr int kT4MaxAxis = 2048;

struct Tc4Smem { int w, bias, pw, small, tips, stage, head, axis, mm, bars, tmem_ptr, total; };
__host__ __device__ inline Tc4Smem tc4_smem_layout(int n_blocks) {
  Tc4Smem s;
  s.w = 0;                                                   // 3*nb matrices, then fc_p_img.weight[:, 3:]
  s.bias = s.w + 4 * VTACO_DEC_TC_BIAS(kT4Mode, n_blocks, 0);   // (2*nb+1) fp32 bias vectors
  s.pw = (s.bias + (2 * n_blocks + 1) * 4 * VTACO_DEC_TC_BVEC_FLOATS + 127) / 128 * 128;   // fc_p or fc_p_img[:, :3]: two K-blocks
  s.small = s.pw + 2 * 4 * VTACO_DEC_TC_KBLK_FLOATS;
  s.tips = s.small + (128 + VTACO_DEC_TAIL) * 4;
  s.stage = s.tips + VTACO_MAX_TIPS * 32 * 4;
  s.stage = (s.stage + 15) / 16 * 16;
  s.head = s.stage + (kT4Threads / 32) * kT4StageRows * 16 * 4;
  s.axis = s.head + kT4Groups * 128 * 2 * 4;
  s.mm = s.axis + kT4MaxAxis * 4;                            // per warp: ordered-int keys of min / max logit
  s.bars = s.mm + (kT4Threads / 32) * 2 * 4;
  s.tmem_ptr = s.bars + 64;
  s.total = s.tmem_ptr + 16;
  return s;
}

// staged row r, float4 slot j (0..3) of a warp's stage buffer: rows are 64 bytes, the slot is
// XOR-swizzled with the row pair so that lanes reading rows r and r+2 hit different banks
__device__ __forceinline__ int stage_idx(int r, int j) { return r * 16 + ((j ^ (r >> 1)) & 3) * 4; }

// 2 * relu(x) = x + |x| (exact): one FADD on the FMA pipe instead of an FMNMX on the ALU pipe, which the
// truncation (LOP3) and the BF16 pack (F2FP) already load (ncu: ALU pipe 47 %, FMA pipe 16 %).  The factor 2
// is undone by the weights: fc_0 / fc_1 are packed times 0.5 (a power of two: every product is unchanged).
__device__ __forceinline__ float2 relu2(float2 x) {   // FADD2 with an |.| operand modifier: two channels per instruction
  return __fadd2_rn(x, make_float2(fabsf(x.x), fabsf(x.y)));
}

// Channels [16*hv, 16*hv + 16) of x (already activated) -> operand columns of the block at `tblk`: hi (tf32
// container: x with the 13 low mantissa bits cleared) at tblk + 16*hv, lo = bf16(x - hi), two per column, at
// tblk + 32 + 8*hv.  x - hi is formed as fma(hi, -1, x) on register pairs (FFMA2: one instruction per two channels).
__device__ __forceinline__ void split_store_t4(uint32_t tblk, int hv, const float (&x)[16]) {
  uint32_t hi[16], lo[8];
#pragma unroll
  for (int j = 0; j < 16; ++j) hi[j] = trunc_tf32(x[j]);
#pragma unroll
  for (int c = 0; c < 8; ++c) {
    const float2 d = __ffma2_rn(make_float2(__uint_as_float(hi[2 * c]), __uint_as_float(hi[2 * c + 1])),
                                make_float2(-1.0f, -1.0f), make_float2(x[2 * c], x[2 * c + 1]));
    lo[c] = pack_bf16(d.x, d.y);
  }
  tmem_st16(tblk + 16 * hv, hi);
  tmem_st8(tblk + 32 + 8 * hv, lo);
}

// The bias of the NEXT accumulation step goes into the accumulator columns as soon as this thread has read them
// (its own lane, its own 16 columns): the step's MMAs then all accumulate, and neither the bias add after the
// tcgen05.ld nor its operand loads are needed — one tcgen05.st.x16 replaces eight packed adds.
__device__ __forceinline__ void store_bias16(uint32_t taddr, const float* __restrict__ b) {
  uint32_t v[16];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float4 bb = reinterpret_cast<const float4*>(b)[j];
    v[4 * j] = __float_as_uint(bb.x); v[4 * j + 1] = __float_as_uint(bb.y);
    v[4 * j + 2] = __float_as_uint(bb.z); v[4 * j + 3] = __float_as_uint(bb.w);
  }
  tmem_st16(taddr, v);
}

// Shared-memory descriptor of a B block `units` 16-byte units after the block described by `lo`:
// K-major, no swizzle, K-chunk stride 512 B, 8-row-group stride 128 B (see make_bdesc).  The start
// address field is (addr >> 4) in bits 0-13; all operand blocks sit below 256 KB, so adding the
// offset to the low word never carries out of the field — one uniform add per MMA instead of the
// shift / mask / or sequence.
__device__ __forceinline__ uint64_t bdesc_at(uint32_t lo, uint32_t units) {
  return ((uint64_t)0x4008u << 32) | (uint64_t)(lo + units);
}

// descriptor units (16 bytes) of `floats` floats
__host__ __device__ constexpr uint32_t desc_units(int floats) { return (uint32_t)floats / 4u; }
constexpr uint32_t kKBlkUnits = desc_units(VTACO_DEC_TC_KBLK_FLOATS);   // a K = 8 TF32 block, or a K = 16 BF16 block

// D (+)= A * W for one 32x32 matrix: A = (a_hi: 32 tf32 columns, a_lo = a_hi + 32: 16 bf16x2 columns),
// W = the matrix whose descriptor low word is `wlo`
__device__ __forceinline__ void issue_product_t4(uint32_t d, uint32_t a_hi, uint32_t wlo, uint32_t accumulate_first) {
#pragma unroll
  for (int kk = 0; kk < 4; ++kk)   // hi * W_lo
    tc_mma_ts(d, a_hi + 8 * kk, bdesc_at(wlo, desc_units(VTACO_DEC_TC_SUB_LO) + kk * kKBlkUnits), kk > 0 ? 1u : accumulate_first);
#pragma unroll
  for (int kk = 0; kk < 2; ++kk)   // lo * bf16(W)
    tc_mma_ts_bf16(d, a_hi + 32 + 8 * kk, bdesc_at(wlo, desc_units(VTACO_DEC_TC_SUB_BF16) + kk * kKBlkUnits), 1);
#pragma unroll
  for (int kk = 0; kk < 4; ++kk)   // hi * W_hi
    tc_mma_ts(d, a_hi + 8 * kk, bdesc_at(wlo, desc_units(VTACO_DEC_TC_SUB_HI) + kk * kKBlkUnits), 1);
}

// NB > 0: the network depth as a compile-time constant (the shipped 5): the block loop is unrolled and the operand
// descriptors of every step are base + immediate.  TIP_PS: per-sample fingertip tables (P.tip_ps), an instantiation
// of its own so that the other instantiations keep their register allocation.
template <bool DENSE, bool TRACE, int NB, bool TIP_PS = false>
__global__ void __launch_bounds__(kT4Threads, 1) decoder_tc4_kernel(const __grid_constant__ DecParams P,
                                                                    const float* __restrict__ wtc,
                                                                    long long* __restrict__ trace) {
  int trace_n = 0;
  extern __shared__ __align__(1024) unsigned char tsm[];
  const Tc4Smem L = tc4_smem_layout(P.n_blocks);
  float* sWtc = reinterpret_cast<float*>(tsm + L.w);
  float* sBias = reinterpret_cast<float*>(tsm + L.bias);
  float* sSmall = reinterpret_cast<float*>(tsm + L.small);
  float* sPw = reinterpret_cast<float*>(tsm + L.pw);
  float* sTip = reinterpret_cast<float*>(tsm + L.tips);
  float* sStage = reinterpret_cast<float*>(tsm + L.stage);
  float* sHead = reinterpret_cast<float*>(tsm + L.head);
  float* sAxis = reinterpret_cast<float*>(tsm + L.axis);
  int32_t* sMM = reinterpret_cast<int32_t*>(tsm + L.mm);
  uint64_t* sBars = reinterpret_cast<uint64_t*>(tsm + L.bars);
  uint32_t* sTmem = reinterpret_cast<uint32_t*>(tsm + L.tmem_ptr);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(kFull, tid >> 5, 0);
  const int g = warp >> 3, wq = warp & 7;   // group (tile slot), warp within the group
  const int lq = wq & 3, hv = wq >> 2;      // TMEM lane quarter (== warp % 4), channel half
  const int tq = lq * 32 + lane;            // query within the tile == TMEM lane
  const int nb = NB > 0 ? NB : P.n_blocks;
  const int nx = P.nx;

  const bool cimg = P.use_img && P.c_img;   // per-query tactile feature tensor (decoder.py:83-85)
  // ---- one-time setup: operand blocks + bias vectors (contiguous in wtc), small vectors, barriers, TMEM ----
  // The 165 KB of operand blocks + bias vectors arrive by TMA bulk copies (cp.async.bulk ... mbarrier::complete_tx)
  // issued by one thread; they land while the CTA allocates TMEM and gathers its first tile, and every thread waits
  // for them once, just before the first MMA issue (the plain load / store loop stood in front of everything: a few
  // microseconds per launch, 10 % of a training-shape call and 1 % of an 8-GPU slab).
  const int wtc_floats = VTACO_DEC_TC_INPUT(nb, 0);   // matrices and bias vectors
  const uint32_t wbar = smem_u32(sBars + kT4Groups);
  const bool w_tma = (reinterpret_cast<uintptr_t>(wtc) & 15) == 0;
  if (w_tma) {
    if (tid == 0) {
      mbar_init(wbar, 1);
      asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
      const uint32_t total = (uint32_t)wtc_floats * 4u;
      asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(wbar), "r"(total) : "memory");
      for (uint32_t off = 0; off < total; off += 32768u) {
        const uint32_t bytes = min(32768u, total - off);
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                         smem_u32(sWtc) + off),
                     "l"(reinterpret_cast<const char*>(wtc) + off), "r"(bytes), "r"(wbar)
                     : "memory");
      }
    }
  } else {
    for (int i = tid; i < wtc_floats / 4; i += kT4Threads)
      reinterpret_cast<float4*>(sWtc)[i] = __ldg(reinterpret_cast<const float4*>(wtc) + i);
  }
  // the two input-layer K-blocks of fc_p or fc_p_img[:, :3]
  for (int i = tid; i < 2 * VTACO_DEC_TC_KBLK_FLOATS; i += kT4Threads)
    sPw[i] = __ldg(wtc + wtc_floats + (P.use_img ? 2 * VTACO_DEC_TC_KBLK_FLOATS : 0) + i);
  for (int i = tid; i < 128; i += kT4Threads) {
    float v = P.weights[(P.use_img ? VTACO_DEC_OFF_WPI : VTACO_DEC_OFF_WP) + i];
    // bc_0 joins the fc_p bias: net = (W p + (bp + bc_0)) + Wc_0 c
    if (i >= 96 && P.has_c) v += __ldg(wtc + VTACO_DEC_TC_BIAS(kT4Mode, nb, 0) + (i - 96));
    sSmall[i] = v;
  }
  for (int i = tid; i < VTACO_DEC_TAIL; i += kT4Threads)
    sSmall[128 + i] = P.weights[VTACO_DEC_OFF_BLOCKS + nb * VTACO_DEC_BLOCK_STRIDE + i];
  const bool axis_sm = DENSE && nx <= kT4MaxAxis;
  if (axis_sm)
    for (int i = tid; i < nx; i += kT4Threads) sAxis[i] = __ldg(P.axis + i);
  load_tips(sTip, P, tid, kT4Threads);
  if (tid < (kT4Threads / 32) * 2) sMM[tid] = (tid & 1) ? INT32_MIN : INT32_MAX;
  init_group_bars(sBars, kT4Groups, tid);
  const uint32_t tmem_base = tmem_alloc_all(sTmem, warp);
  const uint32_t tbase = tmem_base + ((uint32_t)(32 * lq) << 16) + (uint32_t)(g * kT4Cols);
  const uint32_t tC = tbase, tX = tbase + 48, tD = tbase + 96;
  const uint32_t mbase = tmem_base + (uint32_t)(g * kT4Cols);
  const uint32_t mC = mbase, mX = mbase + 48, mD = mbase + 96;
  const uint32_t bar = smem_u32(sBars + g);
  // descriptor low word of matrix 0 (start address >> 4 | K-chunk stride 512 B); matrix m is m * kMatUnits further
  const uint32_t wlo0 = ((smem_u32(sWtc) >> 4) & 0x3fffu) | ((512u >> 4) << 16);
  constexpr uint32_t kMatUnits = desc_units(VTACO_DEC_TC_MAT_FLOATS(kT4Mode));
  const uint32_t pwlo = ((smem_u32(sPw) >> 4) & 0x3fffu) | ((512u >> 4) << 16);
  const int gsync_id = g + 1;
  int step = 0;   // accumulation steps issued so far by this group: rotates the issuing warp, its parity is the mbarrier phase
  auto group_sync = [&]() { asm volatile("bar.sync %0, 256;" ::"r"(gsync_id) : "memory"); };
  // Wait for the MMAs of the step issued last (step counts them; its parity is the mbarrier phase).  Only the
  // warp that issued them polls the mbarrier; the other seven sleep in the group's hardware barrier, which
  // costs no issue slots (ncu: with all eight warps polling, a quarter of all issued instructions were the
  // try_wait loop, taken from the warps that had work).
  auto mma_wait = [&]() {
    if (wq == ((step - 1) & 7)) {
      mbar_wait(bar, (uint32_t)(step - 1) & 1u);
      tc_fence_after();
      tc_fence_before();
    }
    asm volatile("bar.sync %0, 256;" ::"r"(gsync_id) : "memory");
  };
  float* stage = sStage + warp * kT4StageRows * 16;
  float* head = sHead + g * 256;
  const int sub = lane & 3;          // float4 within the 16-channel half
  const int zr = lane >> 2;          // 8 rows / queries per load step
  const int ch0 = 16 * hv;           // first channel of this thread
  const bool sep_cfg = DENSE && P.has_c && P.grid && !P.nearest && !(P.plane[0] || P.plane[1] || P.plane[2]);

  const int n_tiles = (int)P.n_tiles;   // < 2^31 (checked at launch)
  // dense mode: brick coordinates of the group's tile, advanced by the (decomposed) grid stride with carries
  // instead of three integer divisions per tile
  int bz = 0, by = 0, bx = 0, bq = 0, sz = 0, sy = 0, sx = 0, sq = 0;
  if (DENSE) {
    unsigned t = (unsigned)(blockIdx.x * kT4Groups + g);
    bz = (int)(t % (unsigned)P.t_nbz); t /= (unsigned)P.t_nbz;
    by = (int)(t % (unsigned)P.t_nby); t /= (unsigned)P.t_nby;
    bx = (int)(t % (unsigned)P.t_nbx);
    bq = (int)(t / (unsigned)P.t_nbx);
    unsigned u = (unsigned)(gridDim.x * kT4Groups);
    sz = (int)(u % (unsigned)P.t_nbz); u /= (unsigned)P.t_nbz;
    sy = (int)(u % (unsigned)P.t_nby); u /= (unsigned)P.t_nby;
    sx = (int)(u % (unsigned)P.t_nbx);
    sq = (int)(u / (unsigned)P.t_nbx);
  }
  for (int tile = blockIdx.x * kT4Groups + g; tile < n_tiles; tile += gridDim.x * kT4Groups) {
    float px, py, pz;
    int oidx;      // output index, < 2^31 (checked at launch); -1 = padding query
    int qb;
    if (DENSE) {
      qb = bq;
      const int ix = P.x0 + bx * 2 + (tq >> 6), iy = by * 2 + ((tq >> 5) & 1), iz = bz * 32 + (tq & 31);
      const bool valid = (ix < P.t_xend) && (iy < nx) && (iz < nx);
      const int cx = min(ix, nx - 1), cy = min(iy, nx - 1), cz = min(iz, nx - 1);
      px = axis_sm ? sAxis[cx] : __ldg(P.axis + cx);
      py = axis_sm ? sAxis[cy] : __ldg(P.axis + cy);
      pz = axis_sm ? sAxis[cz] : __ldg(P.axis + cz);
      oidx = valid ? ((qb * nx + ix) * nx + iy) * nx + iz : -1;
      bz += sz; if (bz >= P.t_nbz) { bz -= P.t_nbz; ++by; }     // next tile of this group
      by += sy; if (by >= P.t_nby) { by -= P.t_nby; ++bx; }
      bx += sx; if (bx >= P.t_nbx) { bx -= P.t_nbx; ++bq; }
      bq += sq;
    } else {
      const int n = tile * kTcTile + tq;
      const bool valid = n < (int)P.total;
      const int nn = valid ? n : 0;
      px = __ldg(P.p + (size_t)nn * 3 + 0);
      py = __ldg(P.p + (size_t)nn * 3 + 1);
      pz = __ldg(P.p + (size_t)nn * 3 + 2);
      qb = (int)(nn / (int)P.N);
      oidx = valid ? n : -1;
    }
    TC_STAMP(TRACE, 13);  // tile start: coordinates loaded

    // ---------------- gather: this thread's 16 channels of its query (+ of its c_img row): operands of step 0 ----------------
    {
      if (P.has_c) {
        bool sep_done = false;
        if (sep_cfg) {
          // separable dense gather (see SepGather): the warp is one z-run at fixed (x, y); the 4
          // (x,y) corners are reduced once per needed z-row into shared memory, then each thread
          // lerps its two z-rows
          const int R = P.Rg;
          const float tx = unnormalize(norm3d(px, P.nc), R), ty = unnormalize(norm3d(py, P.nc), R);
          const float tz = unnormalize(norm3d(pz, P.nc), R);
          const float flx = floorf(tx), fly = floorf(ty), flz = floorf(tz);
          const int x0 = (int)flx, y0 = (int)fly, z0 = (int)flz;
          const float fx1 = tx - flx, fx0 = (flx + 1.0f) - tx, fy1 = ty - fly, fy0 = (fly + 1.0f) - ty;
          const float fz1 = tz - flz, fz0 = (flz + 1.0f) - tz;
          const int zmin = __shfl_sync(kFull, z0, 0);
          const int zmax = min(__shfl_sync(kFull, z0, 31) + 1, R - 1);
          const int nz = zmax - zmin + 1;
          if (nz <= kT4StageRows) {   // warp-uniform
            const int dx = (x0 + 1 < R) ? 8 : 0, dy = (y0 + 1 < R) ? R * 8 : 0;   // clamped corners carry weight 0
            const float w00 = fx0 * fy0, w01 = fx1 * fy0, w10 = fx0 * fy1, w11 = fx1 * fy1;
            const float4* col = reinterpret_cast<const float4*>(P.grid) + (size_t)qb * R * R * R * 8 +
                                ((size_t)y0 * R + x0) * 8 + 4 * hv + sub;
#pragma unroll 2
            for (int zb = 0; zb < nz; zb += 8) {
              const int zrow = zb + zr;
              if (zrow < nz) {
                const float4* p = col + (size_t)(zmin + zrow) * R * R * 8;
                const float4 v00 = __ldg(p), v01 = __ldg(p + dx), v10 = __ldg(p + dy), v11 = __ldg(p + dy + dx);
                // (same operation order as f4_fma from 0: fma(v00, w00, 0) == v00 * w00, then three FMAs; two lanes per FFMA2)
                float2 lo2 = __fmul2_rn(make_float2(v00.x, v00.y), make_float2(w00, w00));
                float2 hi2 = __fmul2_rn(make_float2(v00.z, v00.w), make_float2(w00, w00));
                lo2 = __ffma2_rn(make_float2(v01.x, v01.y), make_float2(w01, w01), lo2);
                hi2 = __ffma2_rn(make_float2(v01.z, v01.w), make_float2(w01, w01), hi2);
                lo2 = __ffma2_rn(make_float2(v10.x, v10.y), make_float2(w10, w10), lo2);
                hi2 = __ffma2_rn(make_float2(v10.z, v10.w), make_float2(w10, w10), hi2);
                lo2 = __ffma2_rn(make_float2(v11.x, v11.y), make_float2(w11, w11), lo2);
                hi2 = __ffma2_rn(make_float2(v11.z, v11.w), make_float2(w11, w11), hi2);
                *reinterpret_cast<float4*>(stage + stage_idx(zrow, sub)) = make_float4(lo2.x, lo2.y, hi2.x, hi2.y);
              }
            }
            __syncwarp();
            const int ra = z0 - zmin, rb = min(z0 + 1, R - 1) - zmin;
            float cv[16];   // (its own array: the generic path's cv lives in local memory)
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const float4 a = *reinterpret_cast<const float4*>(stage + stage_idx(ra, j));
              const float4 b = *reinterpret_cast<const float4*>(stage + stage_idx(rb, j));
              const float2 f0 = make_float2(fz0, fz0), f1 = make_float2(fz1, fz1);
              const float2 c0 = __ffma2_rn(make_float2(b.x, b.y), f1, __fmul2_rn(make_float2(a.x, a.y), f0));
              const float2 c1 = __ffma2_rn(make_float2(b.z, b.w), f1, __fmul2_rn(make_float2(a.z, a.w), f0));
              cv[4 * j + 0] = c0.x; cv[4 * j + 1] = c0.y; cv[4 * j + 2] = c1.x; cv[4 * j + 3] = c1.y;
            }
            __syncwarp();
            TC_STAMP(TRACE, 15);  // features of the thread's query in registers
            split_store_t4(tC, hv, cv);
            sep_done = true;
          }
        }
        if (!sep_done) {   // generic gather: the owner computes the taps, 4 lanes fetch a query's 16 channels
          float cv[16];
          TapInfo tv, tp0, tp1, tp2;
          if (P.grid) tv = tap_volume(norm3d(px, P.nc), norm3d(py, P.nc), norm3d(pz, P.nc), P.Rg, P.nearest);
          const bool planes = P.plane[0] || P.plane[1] || P.plane[2];
          if (planes) {
            const float ux = norm2d(px, P.nc), uy = norm2d(py, P.nc), uz = norm2d(pz, P.nc);
            if (P.plane[0]) tp0 = tap_plane(ux, uz, P.Rp, P.nearest);
            if (P.plane[1]) tp1 = tap_plane(ux, uy, P.Rp, P.nearest);
            if (P.plane[2]) tp2 = tap_plane(uy, uz, P.Rp, P.nearest);
          }
#pragma unroll 1
          for (int half = 0; half < 2; ++half) {   // 16 queries per pass (the stage buffer holds 24 rows)
#pragma unroll 1
            for (int it = 0; it < 2; ++it) {
              const int row = it * 8 + zr;
              const int src = half * 16 + row;
              const int b = __shfl_sync(kFull, qb, src);
              float4 c = make_float4(0.f, 0.f, 0.f, 0.f);
              if (P.grid) {
                const int R = P.Rg;
                const float4* vol = reinterpret_cast<const float4*>(P.grid) + (size_t)b * R * R * R * 8 + 4 * hv + sub;
                c = fetch_volume(vol, R, tap_bcast(tv, src), P.nearest);
              }
              if (planes) {
                const int R = P.Rp;
                const size_t boff = (size_t)b * R * R * 8 + 4 * hv + sub;
                if (P.plane[0]) c = f4_add(c, fetch_plane(reinterpret_cast<const float4*>(P.plane[0]) + boff, R, tap_bcast(tp0, src), P.nearest));
                if (P.plane[1]) c = f4_add(c, fetch_plane(reinterpret_cast<const float4*>(P.plane[1]) + boff, R, tap_bcast(tp1, src), P.nearest));
                if (P.plane[2]) c = f4_add(c, fetch_plane(reinterpret_cast<const float4*>(P.plane[2]) + boff, R, tap_bcast(tp2, src), P.nearest));
              }
              *reinterpret_cast<float4*>(stage + stage_idx(row, sub)) = c;
            }
            __syncwarp();
            if ((lane >> 4) == half) {   // (cv of the other half-warp waits in local memory: 16 words per tile)
#pragma unroll
              for (int j = 0; j < 4; ++j) {
                const float4 v = *reinterpret_cast<const float4*>(stage + stage_idx(lane & 15, j));
                cv[4 * j] = v.x; cv[4 * j + 1] = v.y; cv[4 * j + 2] = v.z; cv[4 * j + 3] = v.w;
              }
            }
            __syncwarp();
          }
          split_store_t4(tC, hv, cv);
        }
      }
      if (cimg) {   // fc_p_img(cat[p, c_img]) = fc_p_img[:, :3] p + b + W_img c_img: the last term rides in step 0
        float xv[16];
        const float4* row = reinterpret_cast<const float4*>(P.c_img + (size_t)max(oidx, 0) * 32 + ch0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 v = __ldg(row + j);
          xv[4 * j] = v.x; xv[4 * j + 1] = v.y; xv[4 * j + 2] = v.z; xv[4 * j + 3] = v.w;
        }
        split_store_t4(tX, hv, xv);
      } else if (hv == 0) {
        // fc_p on the tensor core as well: A = (px, py, pz, 1, px_lo, py_lo, pz_lo, 0) in the first 8 X columns
        // (the tensor core reads the top 19 bits of px, i.e. px_hi), B1 = rows (Wp_hi x3, b_hi, Wp_hi x3, 0),
        // B2 = rows (Wp_lo x3, b_lo, 0...) — 3xTF32 for the 3-wide layer with two K = 8 MMAs
        uint32_t a[8];
        a[0] = __float_as_uint(px); a[1] = __float_as_uint(py); a[2] = __float_as_uint(pz);
        a[3] = __float_as_uint(1.0f);
        a[4] = __float_as_uint(px - __uint_as_float(trunc_tf32(px)));
        a[5] = __float_as_uint(py - __uint_as_float(trunc_tf32(py)));
        a[6] = __float_as_uint(pz - __uint_as_float(trunc_tf32(pz)));
        a[7] = 0u;
        tmem_st8(tX, a);
      }
      if (w_tma && step == 0) mbar_wait(wbar, 0);   // the operand blocks have landed (first tile of the group only)
      tc_wait_st();
      tc_fence_before();
      group_sync();
      if (wq == (step & 7) && elect_one()) {     // step 0: D = C*Wc_0 + (c_img*W_img | fc_p(p) + bc_0)
        tc_fence_after();
        uint32_t acc = 0;
        if (P.has_c) {
          issue_product_t4(mD, mC, wlo0, 0);
          acc = 1;
        }
        if (cimg) {
          issue_product_t4(mD, mX, wlo0 + (uint32_t)(3 * nb) * kMatUnits, acc);
        } else {
          tc_mma_ts(mD, mX, bdesc_at(pwlo, kKBlkUnits), acc);
          tc_mma_ts(mD, mX, bdesc_at(pwlo, 0), 1);
        }
        tc_commit(bar);
      }
      ++step;
    }

    // ---------------- net = fc_p(p) | fc_p_img(p, tip feature): this thread's 16 channels ----------------
    // (the fingertip test runs in float64: evaluate it before the residual stream occupies registers)
    int tipf = -1;
    if (P.use_img && P.n_tips > 0) {
      bool any_near = true;
      if (DENSE && !P.tip_map) {
        // the warp is one z-run at fixed (x, y): lane f tests fingertip f against the whole segment (fp32,
        // padded threshold); almost every run is far from every fingertip and skips the per-query test
        const float z_lo = __shfl_sync(kFull, pz, 0), z_hi = __shfl_sync(kFull, pz, 31);
        bool near = false;
        if (lane < P.n_tips) {
          const float dx = px - P.tipsf[lane][0], dy = py - P.tipsf[lane][1];
          const float tz = P.tipsf[lane][2];
          const float dz = fmaxf(fmaxf(z_lo - tz, tz - z_hi), 0.f);
          near = dx * dx + dy * dy + dz * dz < P.tip_r2_hi;
        }
        any_near = __any_sync(kFull, near);
      }
      if (any_near) tipf = tip_of_query(P, max(oidx, 0), px, py, pz);
    }
    float net[16];
    {  // net = fc_c[0](c) + (W_img c_img | fc_p(p) + bc_0)
      uint32_t r[16];
      mma_wait();
      tc_fence_after();
      tmem_ld16(tD + ch0, r);
      tc_wait_ld();
#pragma unroll
      for (int j = 0; j < 16; ++j) net[j] = __uint_as_float(r[j]);
      if (nb > 0) store_bias16(tD + ch0, sBias + 1 * VTACO_DEC_TC_BVEC_FLOATS + ch0);      // b0_0 for the first W0 step
    }
    if (cimg) {   // c_img occupies the X columns: the 3-wide layer runs on the CUDA cores
      const float4* w0 = reinterpret_cast<const float4*>(sSmall + ch0);
      const float4* w1 = reinterpret_cast<const float4*>(sSmall + 32 + ch0);
      const float4* w2 = reinterpret_cast<const float4*>(sSmall + 64 + ch0);
      const float4* bp = reinterpret_cast<const float4*>(sSmall + 96 + ch0);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 a0 = w0[j], a1 = w1[j], a2 = w2[j], bb = bp[j];
        net[4 * j + 0] += fmaf(a2.x, pz, fmaf(a1.x, py, fmaf(a0.x, px, bb.x)));
        net[4 * j + 1] += fmaf(a2.y, pz, fmaf(a1.y, py, fmaf(a0.y, px, bb.y)));
        net[4 * j + 2] += fmaf(a2.z, pz, fmaf(a1.z, py, fmaf(a0.z, px, bb.z)));
        net[4 * j + 3] += fmaf(a2.w, pz, fmaf(a1.w, py, fmaf(a0.w, px, bb.w)));
      }
    }
    if (tipf >= 0) {
      if (TIP_PS) {
        add_tip_row<16>(net, P, sTip, tipf, max(oidx, 0), ch0);
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) net[j] += sTip[tipf * 32 + ch0 + j];
      }
    }

    // ---------------- residual blocks: 2 accumulation steps each ----------------
    uint32_t r[16];
#pragma unroll
    for (int i = 0; i < (NB > 0 ? NB : nb); ++i) {
      TC_STAMP(TRACE, 1);   // ALU phase starts (accumulator already read)
      {
        float y[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float2 v = relu2(make_float2(net[2 * j], net[2 * j + 1]));
          y[2 * j] = v.x; y[2 * j + 1] = v.y;
        }
        split_store_t4(tX, hv, y);
      }
      TC_STAMP(TRACE, 2);   // operands computed, tcgen05.st issued
      tc_wait_st();
      tc_fence_before();
      TC_STAMP(TRACE, 3);   // stores complete
      group_sync();
      TC_STAMP(TRACE, 4);   // group barrier passed
      if (wq == (step & 7) && elect_one()) {     // D = relu(net)*W0_i
        tc_fence_after();
        issue_product_t4(mD, mX, wlo0 + (uint32_t)(3 * i + 1) * kMatUnits, 1);   // D already holds b0_i
        tc_commit(bar);
        TC_STAMP(TRACE, 20);  // issuer only: MMAs + commit issued
      }
      ++step;
      TC_STAMP(TRACE, 5);
      mma_wait();
      TC_STAMP(TRACE, 6);   // MMAs complete
      tc_fence_after();
      tmem_ld16(tD + ch0, r);
      tc_wait_ld();
      TC_STAMP(TRACE, 7);   // accumulator in registers
      {                                           // h = relu(D)   (D = b0_i + relu(net) W0_i)
        float y[16];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float2 v = relu2(make_float2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])));
          y[2 * j] = v.x; y[2 * j + 1] = v.y;
        }
        split_store_t4(tX, hv, y);
      }
      store_bias16(tD + ch0, sBias + (2 * i + 2) * VTACO_DEC_TC_BVEC_FLOATS + ch0);       // b1_i + bc_{i+1} for the W1 step
      tc_wait_st();
      tc_fence_before();
      group_sync();
      if (wq == (step & 7) && elect_one()) {     // D = relu(h)*W1_i [+ C*Wc_{i+1}]
        tc_fence_after();
        issue_product_t4(mD, mX, wlo0 + (uint32_t)(3 * i + 2) * kMatUnits, 1);   // D already holds b1_i + bc_{i+1}
        if (P.has_c && i + 1 < nb) issue_product_t4(mD, mC, wlo0 + (uint32_t)(3 * i + 3) * kMatUnits, 1);
        tc_commit(bar);
      }
      ++step;
      mma_wait();
      tc_fence_after();
      tmem_ld16(tD + ch0, r);
      tc_wait_ld();
#pragma unroll
      for (int j = 0; j < 8; ++j) {               // net += D   (D = b1_i + bc_{i+1} + relu(h) W1_i + c Wc_{i+1}), packed adds
        const float2 n0 = __fadd2_rn(make_float2(net[2 * j], net[2 * j + 1]),
                                     make_float2(__uint_as_float(r[2 * j]), __uint_as_float(r[2 * j + 1])));
        net[2 * j] = n0.x; net[2 * j + 1] = n0.y;
      }
      if (i + 1 < nb) store_bias16(tD + ch0, sBias + (2 * i + 3) * VTACO_DEC_TC_BVEC_FLOATS + ch0);   // b0_{i+1} for the next W0 step
    }

    TC_STAMP(TRACE, 19);    // blocks done
    // ---------------- heads: partial dot products of the two halves, combined through shared memory ----------------
    {
      const float* Wo = sSmall + 128;
      float o = 0.f, oc = 0.f;
      if (P.leaky) {
#pragma unroll
        for (int j = 0; j < 16; ++j) net[j] = net[j] > 0.f ? net[j] : net[j] * 0.2f;
      } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) net[j] = fmaxf(net[j], 0.f);
      }
      {   // 16-term dot product as two 8-term chains on register pairs
        float2 acc = make_float2(0.f, 0.f);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          acc = __ffma2_rn(make_float2(Wo[VTACO_DEC_TAIL_WOUT + ch0 + 2 * j], Wo[VTACO_DEC_TAIL_WOUT + ch0 + 2 * j + 1]),
                           make_float2(net[2 * j], net[2 * j + 1]), acc);
        o = acc.x + acc.y;
      }
      if (P.contact) {
#pragma unroll
        for (int j = 0; j < 16; ++j) oc = fmaf(Wo[VTACO_DEC_TAIL_WCON + ch0 + j], net[j], oc);
      }
      if (hv == 1) { head[tq] = o; head[128 + tq] = oc; }
      group_sync();
      if (hv == 0) {   // warp-uniform
        const bool valid = oidx >= 0;
        o = (Wo[VTACO_DEC_TAIL_BOUT] + o) + head[tq];
        if (valid) {
          store_logit(P, oidx, o);
          if (P.contact) P.contact[oidx] = (Wo[VTACO_DEC_TAIL_BCON] + oc) + head[128 + tq];
        }
        if (P.minmax_key) {   // running min / max as ordered-int keys, one pair per warp in shared memory
          const int key = float_to_key(o);
          const int kmin = __reduce_min_sync(kFull, valid ? key : INT32_MAX);
          const int kmax = __reduce_max_sync(kFull, valid ? key : INT32_MIN);
          if (lane == 0) {
            sMM[2 * warp] = min(sMM[2 * warp], kmin);
            sMM[2 * warp + 1] = max(sMM[2 * warp + 1], kmax);
          }
        }
      }
    }
  }

  if (P.minmax_key && lane == 0 && hv == 0 && sMM[2 * warp] <= sMM[2 * warp + 1]) {
    atomicMin(P.minmax_key, sMM[2 * warp]);
    atomicMax(P.minmax_key + 1, sMM[2 * warp + 1]);
  }
  if (w_tma && tid == 0) mbar_wait(wbar, 0);        // a group without tiles never waited: no bulk copy may outlive the CTA
  tmem_free_all(tmem_base, warp);
}

int launch_decoder_tc4(DecParams P, bool dense, const float* wtc, cudaStream_t stream) {
  if (!wtc) return VTACO_ERR_INVALID_ARG;
  const Tc4Smem L = tc4_smem_layout(P.n_blocks);
  if (L.total > 227 * 1024) return launch_decoder_simt(P, dense, stream);
  if (const int e = set_tc_tiles(P, dense)) return e;
  if ((dense ? (long long)P.B * P.nx * P.nx * P.nx : P.total) >= (1ll << 31)) return VTACO_ERR_UNSUPPORTED;   // 32-bit output index
  long long* trace;
  if (const int e = tc_trace_begin(&trace, stream)) return e;
  using Kernel = void (*)(DecParams, const float*, long long*);
  const Kernel k = P.tip_ps ? (P.n_blocks == 5 ? (dense ? decoder_tc4_kernel<true, false, 5, true>
                                                         : decoder_tc4_kernel<false, false, 5, true>)
                                               : (dense ? decoder_tc4_kernel<true, false, 0, true>
                                                        : decoder_tc4_kernel<false, false, 0, true>))
                   : trace ? (dense ? decoder_tc4_kernel<true, true, 0> : decoder_tc4_kernel<false, true, 0>)
                   : P.n_blocks == 5 ? (dense ? decoder_tc4_kernel<true, false, 5> : decoder_tc4_kernel<false, false, 5>)
                                     : (dense ? decoder_tc4_kernel<true, false, 0> : decoder_tc4_kernel<false, false, 0>);
  VTACO_CUDA_CHECK(smem_opt_in((const void*)k, L.total));
  long long grid = (P.n_tiles + kT4Groups - 1) / kT4Groups;
  if (grid > num_sms()) grid = num_sms();
  k<<<(unsigned)grid, kT4Threads, L.total, stream>>>(P, wtc, trace);
  VTACO_LAUNCH_CHECK();
  return tc_trace_end(trace, "tc4", stream);
}

}  // namespace vtaco
