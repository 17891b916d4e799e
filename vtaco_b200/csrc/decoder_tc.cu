// Fused LocalDecoder on the 5th-gen tensor cores (tcgen05 + TMEM), sm_100a.
//
// Same contract as decoder.cu (reference src/conv_onet/models/decoder.py:71-161); selected
// with vtaco_decoder_args.variant == 2.  Why: ncu on the SIMT kernel shows the 32-wide
// contraction is pipe-bound (shared-memory wavefronts 71 %, FMA pipe 62 %), not latency
// bound (profiles/decoder_ncu_summary.json) — the condition the design brief sets for moving
// it to the tensor pipe.
//
// fp32 fidelity on a TF32 pipe: every operand is split x = hi + lo with hi = tf32(x) and the
// product is evaluated as hi*hi + lo*hi + hi*lo (3xTF32, fp32 accumulation in TMEM); the
// dropped lo*lo term and the truncation of lo are ~2^-22 relative.
//
// Structure (one persistent CTA per SM, 384 threads = 3 independent groups of 4 warps):
//   * a group owns a tile of 128 queries = the 128 TMEM lanes; thread t <-> query t <-> lane t;
//   * all 3*n_blocks weight matrices (hi and lo, UMMA canonical K-major, no swizzle) stay in
//     shared memory for the life of the CTA (120 KB); they are the B operands;
//   * activations are the A operands and live in TMEM (tcgen05.st from registers), so a layer
//     costs per thread: tcgen05.ld of 32 accumulator columns, bias/residual/ReLU/split
//     (~4 ALU ops per element), tcgen05.st of hi and lo — no shared-memory traffic at all;
//   * biases ride along as one more K-block: a constant (1,1,0,..) A block times a B block
//     whose rows 0/1 hold the bias hi/lo; fc_c[i+1](c) accumulates into the same TMEM
//     accumulator as fc_1 of block i, so a block costs 2 accumulator reads, not 3;
//   * one elected thread per group (the role rotates over the 4 warps) issues the tcgen05.mma
//     (M128 N32 K8, kind::tf32) of a step and commits to the group's mbarrier; the groups
//     interleave on the tensor pipe, so one group's ALU phase overlaps the others' MMA phases;
//   * the residual stream stays in registers; feature gather, fc_p, tips and fc_out run on the
//     CUDA cores exactly as in the SIMT kernel.
#include "decoder_tc_common.cuh"
#include <cstdio>
#include <cstdlib>

namespace vtaco {


// weights_tc is copied to shared memory as it is.  Pack modes 0 and 1 place every block alike (they differ only
// inside a matrix's lo sub-block), so the offsets are mode 0's; byte sizes of the pieces an MMA reads:
constexpr int kTcMode = VTACO_DEC_TC_MODE_3XTF32;
constexpr int kMatBytes = 4 * VTACO_DEC_TC_MAT_FLOATS(kTcMode);
constexpr int kKBlkBytes = 4 * VTACO_DEC_TC_KBLK_FLOATS;   // a K = 8 TF32 block (also a bias step), or a K = 16 BF16 block
constexpr int kLoBytes = 4 * VTACO_DEC_TC_SUB_LO;
// the layouts below and wimg_sm find fc_p_img.weight[:, 3:] right after the 2*nb+1 bias K-blocks
static_assert(VTACO_DEC_TC_WIMG(kTcMode, VTACO_MAX_BLOCKS) ==
                  VTACO_DEC_TC_BIAS(kTcMode, VTACO_MAX_BLOCKS, 0) + (2 * VTACO_MAX_BLOCKS + 1) * VTACO_DEC_TC_KBLK_FLOATS,
              "W_img block must follow the bias K-blocks");

struct TcSmem {
  // byte offsets into dynamic shared memory
  int w, bias, small, tips, stage, bars, tmem_ptr, total;
};
__host__ __device__ inline TcSmem tc_smem_layout(int n_blocks) {
  TcSmem s;
  s.w = 0;                                                      // weights_tc: 3*nb matrices,
  s.bias = s.w + 4 * VTACO_DEC_TC_BIAS(kTcMode, n_blocks, 0);   // the bias K-blocks, then fc_p_img.weight[:, 3:]
  s.small = s.bias + (2 * n_blocks + 1) * kKBlkBytes + kMatBytes;   // Wp[3][32], bp[32], Wout[64], bout[2]+pad
  s.tips = s.small + (128 + VTACO_DEC_TAIL) * 4;
  s.stage = s.tips + VTACO_MAX_TIPS * 32 * 4;
  s.stage = (s.stage + 15) / 16 * 16;
  s.bars = s.stage + (kTcThreads / 32) * 32 * kStageStride * 4;
  s.tmem_ptr = s.bars + 64;
  s.total = s.tmem_ptr + 16;
  return s;
}

// MMAs of one accumulation step, issued by one thread.  D = [A_x * W] + ones * Bias [+ C * Wc]
__device__ __forceinline__ void issue_product(uint32_t d, uint32_t a_hi, uint32_t w_smem, uint32_t accumulate_first,
                                              int n_products = 3) {
  const uint32_t a_lo = a_hi + 32;
  if (n_products == 2) {   // mixed: BF16 correction (K = 64) then the TF32 main product
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) tc_mma_ts_bf16(d, a_lo + 8 * kk, make_bdesc(w_smem + kLoBytes + kk * kKBlkBytes), kk > 0 ? 1u : accumulate_first);
    accumulate_first = 1;
  }
  if (n_products >= 3) {
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) tc_mma_ts(d, a_lo + 8 * kk, make_bdesc(w_smem + kk * kKBlkBytes), kk > 0 ? 1u : accumulate_first);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) tc_mma_ts(d, a_hi + 8 * kk, make_bdesc(w_smem + kLoBytes + kk * kKBlkBytes), 1);
    accumulate_first = 1;
  }
#pragma unroll
  for (int kk = 0; kk < 4; ++kk) tc_mma_ts(d, a_hi + 8 * kk, make_bdesc(w_smem + kk * kKBlkBytes), kk > 0 ? 1u : accumulate_first);
}

template <bool DENSE, bool MIXED>
__global__ void __launch_bounds__(kTcThreads, 1) decoder_tc_kernel(const __grid_constant__ DecParams P,
                                                                   const float* __restrict__ wtc,
                                                                   long long* __restrict__ trace) {
  int trace_n = 0;
  extern __shared__ __align__(1024) unsigned char tsm[];
  const TcSmem L = tc_smem_layout(P.n_blocks);
  float* sWtc = reinterpret_cast<float*>(tsm + L.w);
  float* sSmall = reinterpret_cast<float*>(tsm + L.small);
  float* sTip = reinterpret_cast<float*>(tsm + L.tips);
  float* sStage = reinterpret_cast<float*>(tsm + L.stage);
  uint64_t* sBars = reinterpret_cast<uint64_t*>(tsm + L.bars);
  uint32_t* sTmem = reinterpret_cast<uint32_t*>(tsm + L.tmem_ptr);

  // warp index through a shuffle: the compiler can then prove g / wg and everything derived
  // from them warp-uniform (uniform registers for the MMA descriptors, uniform branches)
  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(kFull, tid >> 5, 0);
  const int g = warp >> 2, wg = warp & 3, tg = tid & 127;
  const int nb = P.n_blocks;

  // ---- one-time setup: weights + bias blocks (contiguous in wtc), small vectors, barriers, TMEM ----
  const bool cimg = P.use_img && P.c_img;   // per-query tactile feature tensor (decoder.py:83-85)
  const int wtc_floats = VTACO_DEC_TC_WIMG(kTcMode, nb) + (cimg ? VTACO_DEC_TC_MAT_FLOATS(kTcMode) : 0);
  for (int i = tid; i < wtc_floats / 4; i += kTcThreads)
    reinterpret_cast<float4*>(sWtc)[i] = __ldg(reinterpret_cast<const float4*>(wtc) + i);
  load_small(sSmall, P, nb, tid, kTcThreads);
  load_tips(sTip, P, tid, kTcThreads);
  init_group_bars(sBars, kTcGroups, tid);
  const uint32_t tmem_base = tmem_alloc_all(sTmem, warp);
  // group columns: C_hi 0, C_lo 32, X_hi 64, X_lo 96, ones 128 (8), D 136 (32)
  const uint32_t tbase = tmem_base + ((uint32_t)(32 * wg) << 16) + (uint32_t)(g * kColsPerGroup);
  const uint32_t tC = tbase, tX = tbase + 64, tOnes = tbase + 128, tD = tbase + 136;
  const uint32_t mbase = tmem_base + (uint32_t)(g * kColsPerGroup);
  const uint32_t mC = mbase, mX = mbase + 64, mOnes = mbase + 128, mD = mbase + 136;
  const uint32_t bar = smem_u32(sBars + g);
  const uint32_t wsm = smem_u32(sWtc), bsm = smem_u32(tsm + L.bias);
  const uint32_t wimg_sm = bsm + (uint32_t)(2 * nb + 1) * (uint32_t)kKBlkBytes;   // after the bias steps
  uint32_t ph = 0;
  {  // the constant A block that multiplies the bias rows: columns (1, 1, 0, 0, 0, 0, 0, 0)
    const uint32_t one = __float_as_uint(1.0f);
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(tOnes), "r"(one),
                 "r"(one), "r"(0u), "r"(0u), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
                 : "memory");
    tc_wait_st();
  }
  float* stage = sStage + warp * 32 * kStageStride;
  const int grp = lane >> 3, sub = lane & 7;
  const int nx = P.nx;
  float vmin = CUDART_INF_F, vmax = -CUDART_INF_F;
  int step = 0;  // accumulation steps issued so far by this group (rotates the issuing warp)
  constexpr bool mixed = MIXED;   // compile-time: the 3xTF32 kernel keeps its register budget

  for (long long tile = (long long)blockIdx.x * kTcGroups + g; tile < P.n_tiles;
       tile += (long long)gridDim.x * kTcGroups) {
    const auto [px, py, pz, oidx, qb, valid] = tile_query(P, DENSE, tile, tg, nullptr, false, nx);   // this thread's query
    TC_STAMP(trace, 13);  // tile start: coordinates loaded

    // ---------------- gather (+ the query's c_img row): operands of step 0 ----------------
    if (P.has_c || cimg) {
     if (P.has_c) {
      float cv[32];
      bool sep_done = false;
      if (DENSE && P.grid && !P.nearest && !(P.plane[0] || P.plane[1] || P.plane[2])) {
        // Separable dense gather (4 z-rows x 8 channel quads per load step): ~40 tap loads per run instead of 256
        const int R = P.Rg;
        const SepGather sg = sep_gather_setup(P, px, py, pz, qb, sub);
        if (sg.nz <= 32) {   // warp-uniform
          const int zr = lane >> 3;
#pragma unroll 2
          for (int zb = 0; zb < sg.nz; zb += 4) {
            const int zrow = zb + zr;
            if (zrow < sg.nz) {
              const float4* p = sg.col + (size_t)(sg.zmin + zrow) * R * R * 8;
              const float4 v00 = __ldg(p), v01 = __ldg(p + sg.dx), v10 = __ldg(p + sg.dy), v11 = __ldg(p + sg.dy + sg.dx);
              float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
              a = f4_fma(sg.w00, v00, a);
              a = f4_fma(sg.w01, v01, a);
              a = f4_fma(sg.w10, v10, a);
              a = f4_fma(sg.w11, v11, a);
              *reinterpret_cast<float4*>(stage + zrow * kStageStride + 4 * sub) = a;
            }
          }
          __syncwarp();
          const float* r0 = stage + (sg.z0 - sg.zmin) * kStageStride;
          const float* r1 = stage + (min(sg.z0 + 1, R - 1) - sg.zmin) * kStageStride;
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 a = *reinterpret_cast<const float4*>(r0 + 4 * j);
            const float4 b = *reinterpret_cast<const float4*>(r1 + 4 * j);
            cv[4 * j + 0] = fmaf(b.x, sg.fz1, a.x * sg.fz0);
            cv[4 * j + 1] = fmaf(b.y, sg.fz1, a.y * sg.fz0);
            cv[4 * j + 2] = fmaf(b.z, sg.fz1, a.z * sg.fz0);
            cv[4 * j + 3] = fmaf(b.w, sg.fz1, a.w * sg.fz0);
          }
          __syncwarp();
          sep_done = true;
        }
      }
      if (!sep_done) {
      // generic gather: the owner computes the taps, 8 lanes fetch them
      const QueryTaps taps = query_taps(P, px, py, pz);
      TC_STAMP(trace, 14);  // taps computed
#pragma unroll 2
      for (int it = 0; it < 8; ++it) {
        const int src = it * 4 + grp;
        const int b = __shfl_sync(kFull, qb, src);
        *reinterpret_cast<float4*>(stage + src * kStageStride + 4 * sub) = gather_taps(P, taps, src, b, sub);
      }
      __syncwarp();
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 v = *reinterpret_cast<const float4*>(stage + lane * kStageStride + 4 * j);
        cv[4 * j] = v.x; cv[4 * j + 1] = v.y; cv[4 * j + 2] = v.z; cv[4 * j + 3] = v.w;
      }
      __syncwarp();
      }  // generic gather
      TC_STAMP(trace, 15);  // features of the thread's query in registers
      split_store(tC, cv, mixed);
     }
      if (cimg) {   // fc_p_img(cat[p, c_img]) = fc_p_img[:, :3] p + b + W_img c_img: the last term rides in step 0
        float xv[32];
        const float4* row = reinterpret_cast<const float4*>(P.c_img + (size_t)oidx * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 v = __ldg(row + j);
          xv[4 * j] = v.x; xv[4 * j + 1] = v.y; xv[4 * j + 2] = v.z; xv[4 * j + 3] = v.w;
        }
        split_store(tX, xv, mixed);
      }
      tc_wait_st();
      tc_fence_before();
      group_sync(g);
      TC_STAMP(trace, 16);  // C in TMEM, group synced
      if (wg == (step & 3) && elect_one()) {     // step 0: D = C*Wc_0 + ones*bc_0 [+ c_img*W_img]
        tc_fence_after();
        uint32_t acc = 0;
        if (P.has_c) {
          issue_product(mD, mC, wsm, 0, P.tc_products);
          tc_mma_ts(mD, mOnes, make_bdesc(bsm), 1);
          acc = 1;
        }
        if (cimg) issue_product(mD, mX, wimg_sm, acc, P.tc_products);
        tc_commit(bar);
      }
      ++step;
    }

    // ---------------- net = fc_p(p) | fc_p_img(p, tip feature) on the CUDA cores ----------------
    float net[32];
    {
      const float4* w0 = reinterpret_cast<const float4*>(sSmall);
      const float4* w1 = reinterpret_cast<const float4*>(sSmall + 32);
      const float4* w2 = reinterpret_cast<const float4*>(sSmall + 64);
      const float4* bp = reinterpret_cast<const float4*>(sSmall + 96);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float4 a0 = w0[j], a1 = w1[j], a2 = w2[j], bb = bp[j];
        net[4 * j + 0] = fmaf(a2.x, pz, fmaf(a1.x, py, fmaf(a0.x, px, bb.x)));
        net[4 * j + 1] = fmaf(a2.y, pz, fmaf(a1.y, py, fmaf(a0.y, px, bb.y)));
        net[4 * j + 2] = fmaf(a2.z, pz, fmaf(a1.z, py, fmaf(a0.z, px, bb.z)));
        net[4 * j + 3] = fmaf(a2.w, pz, fmaf(a1.w, py, fmaf(a0.w, px, bb.w)));
      }
    }
    if (P.use_img && P.n_tips > 0) {
      const int f = tip_of_query(P, oidx, px, py, pz);
      if (f >= 0) add_tip_row<32>(net, P, sTip, f, oidx, 0);
    }
    TC_STAMP(trace, 17);    // fc_p / tips done
    uint32_t r[32];
    float x[32];
    if (P.has_c || cimg) {  // net += fc_c[0](c) [+ W_img c_img]
      mbar_wait(bar, ph); ph ^= 1;
      tc_fence_after();
      tmem_ld32(tD, r);
      tc_wait_ld();
#pragma unroll
      for (int j = 0; j < 32; ++j) net[j] += __uint_as_float(r[j]);
    }

    TC_STAMP(trace, 18);    // step 0 consumed
    // ---------------- residual blocks: 2 accumulation steps each ----------------
    for (int i = 0; i < nb; ++i) {
      TC_STAMP(trace, 1);   // ALU phase starts (accumulator already read)
#pragma unroll
      for (int j = 0; j < 32; ++j) x[j] = fmaxf(net[j], 0.f);
      split_store(tX, x, mixed);
      TC_STAMP(trace, 2);   // operands computed, tcgen05.st issued
      tc_wait_st();
      tc_fence_before();
      TC_STAMP(trace, 3);   // stores complete
      group_sync(g);
      TC_STAMP(trace, 4);   // group barrier passed
      if (wg == (step & 3) && elect_one()) {     // D = relu(net)*W0_i + ones*b0_i
        tc_fence_after();
        issue_product(mD, mX, wsm + 4 * VTACO_DEC_TC_MAT(kTcMode, 3 * i + 1), 0, P.tc_products);
        tc_mma_ts(mD, mOnes, make_bdesc(bsm + (2 * i + 1) * kKBlkBytes), 1);
        tc_commit(bar);
      }
      ++step;
      TC_STAMP(trace, 5);   // (issuing warp: MMAs issued)
      mbar_wait(bar, ph); ph ^= 1;
      TC_STAMP(trace, 6);   // MMAs complete
      tc_fence_after();
      tmem_ld32(tD, r);
      tc_wait_ld();
      TC_STAMP(trace, 7);   // accumulator in registers
#pragma unroll
      for (int j = 0; j < 32; ++j) x[j] = fmaxf(__uint_as_float(r[j]), 0.f);
      split_store(tX, x, mixed);
      TC_STAMP(trace, 8 + 16 * (i & 1));    // W1 step: operands computed (+16: warp 0 is this step's issuer)
      tc_wait_st();
      tc_fence_before();
      group_sync(g);
      TC_STAMP(trace, 9 + 16 * (i & 1));
      if (wg == (step & 3) && elect_one()) {     // D = relu(h)*W1_i + ones*(b1_i + bc_{i+1}) [+ C*Wc_{i+1}]
        tc_fence_after();
        issue_product(mD, mX, wsm + 4 * VTACO_DEC_TC_MAT(kTcMode, 3 * i + 2), 0, P.tc_products);
        tc_mma_ts(mD, mOnes, make_bdesc(bsm + (2 * i + 2) * kKBlkBytes), 1);
        if (P.has_c && i + 1 < nb) issue_product(mD, mC, wsm + 4 * VTACO_DEC_TC_MAT(kTcMode, 3 * (i + 1)), 1, P.tc_products);
        tc_commit(bar);
      }
      ++step;
      TC_STAMP(trace, 10 + 16 * (i & 1));
      mbar_wait(bar, ph); ph ^= 1;
      TC_STAMP(trace, 11 + 16 * (i & 1));
      tc_fence_after();
      tmem_ld32(tD, r);
      tc_wait_ld();
      TC_STAMP(trace, 12 + 16 * (i & 1));
#pragma unroll
      for (int j = 0; j < 32; ++j) net[j] += __uint_as_float(r[j]);
    }

    TC_STAMP(trace, 19);    // blocks done
    // ---------------- heads ----------------
    {
      const float* Wo = sSmall + 128;
      const float slope = P.leaky ? 0.2f : 0.0f;
      float o = Wo[VTACO_DEC_TAIL_BOUT], oc = Wo[VTACO_DEC_TAIL_BCON];
#pragma unroll
      for (int j = 0; j < 32; ++j) {
        net[j] = net[j] > 0.f ? net[j] : net[j] * slope;
        o = fmaf(Wo[VTACO_DEC_TAIL_WOUT + j], net[j], o);
      }
      if (P.contact) {
#pragma unroll
        for (int j = 0; j < 32; ++j) oc = fmaf(Wo[VTACO_DEC_TAIL_WCON + j], net[j], oc);
      }
      if (valid) {
        store_logit(P, oidx, o);
        if (P.contact) P.contact[oidx] = oc;
        vmin = fminf(vmin, o);
        vmax = fmaxf(vmax, o);
      }
    }
  }

  flush_minmax(P, vmin, vmax, lane);
  tmem_free_all(tmem_base, warp);
}


// =======================================================================================
// Two threads per query (variants 5 / 6): the same algorithm with 8 warps per 128-query tile.
// Warps w and w+4 of a group share a TMEM lane quarter and split the 32 channels 16 / 16, so
// every per-step phase (TMEM load, bias/residual/ReLU/split, TMEM store) is half as long per
// warp and each scheduler has 6 warps instead of 3 to interleave.  TMEM capacity (3 tiles per SM)
// is what rules out simply adding tiles.  768 threads -> 85 registers per thread.
// =======================================================================================
constexpr int kTc2Threads = 768;
constexpr int kTcMaxAxis = 2048;  // dense mode: lattice axes up to this length are kept in shared memory
constexpr int kTc2Stage = 20;   // floats per staged row (16 channels + pad)

// channels [16*hv, 16*hv+16) of x -> operand columns of the block at `tblk` (hi at +0, lo / correction at +32)
template <bool MIXED>
__device__ __forceinline__ void split_store16(uint32_t tblk, int hv, const float (&x)[16]) {
  uint32_t hi[16];
#pragma unroll
  for (int j = 0; j < 16; ++j) hi[j] = trunc_tf32(x[j]);
  tmem_st16(tblk + 16 * hv, hi);
  if (MIXED) {
    uint32_t lo8[8], hi8[8];
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      lo8[c] = pack_bf16(x[2 * c] - __uint_as_float(hi[2 * c]), x[2 * c + 1] - __uint_as_float(hi[2 * c + 1]));
      hi8[c] = pack_bf16(__uint_as_float(hi[2 * c]), __uint_as_float(hi[2 * c + 1]));
    }
    tmem_st8(tblk + 32 + 8 * hv, lo8);        // bf16 lo, k = 16*hv .. +15
    tmem_st8(tblk + 48 + 8 * hv, hi8);        // bf16 hi, k = 32 + 16*hv .. +15
  } else {
    uint32_t lo[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) lo[j] = __float_as_uint(x[j] - __uint_as_float(hi[j]));
    tmem_st16(tblk + 32 + 16 * hv, lo);
  }
}

struct Tc2Smem { int w, bias, small, tips, stage, head, axis, bars, tmem_ptr, total; };
__host__ __device__ inline Tc2Smem tc2_smem_layout(int n_blocks) {
  Tc2Smem s;
  s.w = 0;
  s.bias = s.w + 4 * VTACO_DEC_TC_BIAS(kTcMode, n_blocks, 0);
  s.small = s.bias + (2 * n_blocks + 1) * kKBlkBytes + kMatBytes;   // bias K-blocks, then fc_p_img.weight[:, 3:]
  s.tips = s.small + (128 + VTACO_DEC_TAIL) * 4;
  s.stage = s.tips + VTACO_MAX_TIPS * 32 * 4;
  s.stage = (s.stage + 15) / 16 * 16;
  s.head = s.stage + (kTc2Threads / 32) * 32 * kTc2Stage * 4;   // per warp: 32 rows x 16 channels
  s.axis = s.head + kTcGroups * 128 * 2 * 4;                     // partial head sums of the upper halves
  s.bars = s.axis + kTcMaxAxis * 4;
  s.tmem_ptr = s.bars + 64;
  s.total = s.tmem_ptr + 16;
  return s;
}

template <bool DENSE, bool MIXED>
__global__ void __launch_bounds__(kTc2Threads, 1) decoder_tc2_kernel(const __grid_constant__ DecParams P,
                                                                     const float* __restrict__ wtc,
                                                                     long long* __restrict__ trace) {
  int trace_n = 0;
  extern __shared__ __align__(1024) unsigned char tsm[];
  const Tc2Smem L = tc2_smem_layout(P.n_blocks);
  float* sWtc = reinterpret_cast<float*>(tsm + L.w);
  float* sSmall = reinterpret_cast<float*>(tsm + L.small);
  float* sTip = reinterpret_cast<float*>(tsm + L.tips);
  float* sStage = reinterpret_cast<float*>(tsm + L.stage);
  float* sHead = reinterpret_cast<float*>(tsm + L.head);
  float* sAxis = reinterpret_cast<float*>(tsm + L.axis);
  uint64_t* sBars = reinterpret_cast<uint64_t*>(tsm + L.bars);
  uint32_t* sTmem = reinterpret_cast<uint32_t*>(tsm + L.tmem_ptr);

  const int tid = threadIdx.x, lane = tid & 31;
  const int warp = __shfl_sync(kFull, tid >> 5, 0);
  const int g = warp >> 3, wq = warp & 7;   // group, warp within the group
  const int lq = wq & 3, hv = wq >> 2;      // TMEM lane quarter (== warp % 4), channel half
  const int tq = lq * 32 + lane;            // query within the tile == TMEM lane
  const int nb = P.n_blocks;
  const int nx = P.nx;

  const bool cimg = P.use_img && P.c_img;   // per-query tactile feature tensor (decoder.py:83-85)
  const int wtc_floats = VTACO_DEC_TC_WIMG(kTcMode, nb) + (cimg ? VTACO_DEC_TC_MAT_FLOATS(kTcMode) : 0);
  for (int i = tid; i < wtc_floats / 4; i += kTc2Threads)
    reinterpret_cast<float4*>(sWtc)[i] = __ldg(reinterpret_cast<const float4*>(wtc) + i);
  load_small(sSmall, P, nb, tid, kTc2Threads);
  const bool axis_sm = DENSE && nx <= kTcMaxAxis;
  if (axis_sm)
    for (int i = tid; i < nx; i += kTc2Threads) sAxis[i] = __ldg(P.axis + i);
  load_tips(sTip, P, tid, kTc2Threads);
  init_group_bars(sBars, kTcGroups, tid);
  const uint32_t tmem_base = tmem_alloc_all(sTmem, warp);
  const uint32_t tbase = tmem_base + ((uint32_t)(32 * lq) << 16) + (uint32_t)(g * kColsPerGroup);
  const uint32_t tC = tbase, tX = tbase + 64, tOnes = tbase + 128, tD = tbase + 136;
  const uint32_t mbase = tmem_base + (uint32_t)(g * kColsPerGroup);
  const uint32_t mC = mbase, mX = mbase + 64, mOnes = mbase + 128, mD = mbase + 136;
  const uint32_t bar = smem_u32(sBars + g);
  const uint32_t wsm = smem_u32(sWtc), bsm = smem_u32(tsm + L.bias);
  const uint32_t wimg_sm = bsm + (uint32_t)(2 * nb + 1) * (uint32_t)kKBlkBytes;   // after the bias steps
  const int gsync_id = g + 1;
  auto group_sync2 = [&]() { asm volatile("bar.sync %0, 256;" ::"r"(gsync_id) : "memory"); };
  uint32_t ph = 0;
  if (hv == 0) {
    const uint32_t one = __float_as_uint(1.0f);
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};" ::"r"(tOnes), "r"(one),
                 "r"(one), "r"(0u), "r"(0u), "r"(0u), "r"(0u), "r"(0u), "r"(0u)
                 : "memory");
    tc_wait_st();
  }
  float* stage = sStage + warp * 32 * kTc2Stage;
  float* head = sHead + g * 256;
  const int sub = lane & 3;          // float4 within the 16-channel half
  const int zr = lane >> 2;          // 8 rows / queries per load step
  const int ch0 = 16 * hv;           // first channel of this thread
  float vmin = CUDART_INF_F, vmax = -CUDART_INF_F;
  int step = 0;
  const bool sep_cfg = DENSE && P.has_c && P.grid && !P.nearest && !(P.plane[0] || P.plane[1] || P.plane[2]);
  const int n_prod = MIXED ? 2 : 3;

  for (long long tile = (long long)blockIdx.x * kTcGroups + g; tile < P.n_tiles;
       tile += (long long)gridDim.x * kTcGroups) {
    const auto [px, py, pz, oidx, qb, valid] = tile_query(P, DENSE, tile, tq, sAxis, axis_sm, nx);
    TC_STAMP(trace, 13);  // tile start: coordinates loaded

    // ---------------- gather: this thread's 16 channels of its query (+ of its c_img row): operands of step 0 ----------------
    if (P.has_c || cimg) {
     if (P.has_c) {
      float cv[16];
      bool sep_done = false;
      if (sep_cfg) {
        const int R = P.Rg;
        const SepGather sg = sep_gather_setup(P, px, py, pz, qb, 4 * hv + sub);
        if (sg.nz <= 32) {
#pragma unroll 2
          for (int zb = 0; zb < sg.nz; zb += 8) {
            const int zrow = zb + zr;
            if (zrow < sg.nz) {
              const float4* p = sg.col + (size_t)(sg.zmin + zrow) * R * R * 8;
              const float4 v00 = __ldg(p), v01 = __ldg(p + sg.dx), v10 = __ldg(p + sg.dy), v11 = __ldg(p + sg.dy + sg.dx);
              float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
              a = f4_fma(sg.w00, v00, a);
              a = f4_fma(sg.w01, v01, a);
              a = f4_fma(sg.w10, v10, a);
              a = f4_fma(sg.w11, v11, a);
              *reinterpret_cast<float4*>(stage + zrow * kTc2Stage + 4 * sub) = a;
            }
          }
          __syncwarp();
          const float* r0 = stage + (sg.z0 - sg.zmin) * kTc2Stage;
          const float* r1 = stage + (min(sg.z0 + 1, R - 1) - sg.zmin) * kTc2Stage;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            const float4 a = *reinterpret_cast<const float4*>(r0 + 4 * j);
            const float4 b = *reinterpret_cast<const float4*>(r1 + 4 * j);
            cv[4 * j + 0] = fmaf(b.x, sg.fz1, a.x * sg.fz0);
            cv[4 * j + 1] = fmaf(b.y, sg.fz1, a.y * sg.fz0);
            cv[4 * j + 2] = fmaf(b.z, sg.fz1, a.z * sg.fz0);
            cv[4 * j + 3] = fmaf(b.w, sg.fz1, a.w * sg.fz0);
          }
          __syncwarp();
          sep_done = true;
        }
      }
      if (!sep_done) {   // generic gather: the owner computes the taps, 4 lanes fetch a query's 16 channels
        const QueryTaps taps = query_taps(P, px, py, pz);
#pragma unroll 2
        for (int it = 0; it < 4; ++it) {
          const int src = it * 8 + zr;
          const int b = __shfl_sync(kFull, qb, src);
          *reinterpret_cast<float4*>(stage + src * kTc2Stage + 4 * sub) = gather_taps(P, taps, src, b, 4 * hv + sub);
        }
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 v = *reinterpret_cast<const float4*>(stage + lane * kTc2Stage + 4 * j);
          cv[4 * j] = v.x; cv[4 * j + 1] = v.y; cv[4 * j + 2] = v.z; cv[4 * j + 3] = v.w;
        }
        __syncwarp();
      }
      TC_STAMP(trace, 15);  // features of the thread's query in registers
      split_store16<MIXED>(tC, hv, cv);
     }
      if (cimg) {   // fc_p_img(cat[p, c_img]) = fc_p_img[:, :3] p + b + W_img c_img: the last term rides in step 0
        float xv[16];
        const float4* row = reinterpret_cast<const float4*>(P.c_img + (size_t)oidx * 32 + ch0);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float4 v = __ldg(row + j);
          xv[4 * j] = v.x; xv[4 * j + 1] = v.y; xv[4 * j + 2] = v.z; xv[4 * j + 3] = v.w;
        }
        split_store16<MIXED>(tX, hv, xv);
      }
      tc_wait_st();
      tc_fence_before();
      group_sync2();
      if (wq == (step & 7) && elect_one()) {     // step 0: D = C*Wc_0 + ones*bc_0 [+ c_img*W_img]
        tc_fence_after();
        uint32_t acc = 0;
        if (P.has_c) {
          issue_product(mD, mC, wsm, 0, n_prod);
          tc_mma_ts(mD, mOnes, make_bdesc(bsm), 1);
          acc = 1;
        }
        if (cimg) issue_product(mD, mX, wimg_sm, acc, n_prod);
        tc_commit(bar);
      }
      ++step;
    }

    // ---------------- net = fc_p(p) | fc_p_img(p, tip feature): this thread's 16 channels ----------------
    float net[16];
    {
      const float4* w0 = reinterpret_cast<const float4*>(sSmall + ch0);
      const float4* w1 = reinterpret_cast<const float4*>(sSmall + 32 + ch0);
      const float4* w2 = reinterpret_cast<const float4*>(sSmall + 64 + ch0);
      const float4* bp = reinterpret_cast<const float4*>(sSmall + 96 + ch0);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float4 a0 = w0[j], a1 = w1[j], a2 = w2[j], bb = bp[j];
        net[4 * j + 0] = fmaf(a2.x, pz, fmaf(a1.x, py, fmaf(a0.x, px, bb.x)));
        net[4 * j + 1] = fmaf(a2.y, pz, fmaf(a1.y, py, fmaf(a0.y, px, bb.y)));
        net[4 * j + 2] = fmaf(a2.z, pz, fmaf(a1.z, py, fmaf(a0.z, px, bb.z)));
        net[4 * j + 3] = fmaf(a2.w, pz, fmaf(a1.w, py, fmaf(a0.w, px, bb.w)));
      }
    }
    if (P.use_img && P.n_tips > 0) {
      const int f = tip_of_query(P, oidx, px, py, pz);
      if (f >= 0) add_tip_row<16>(net, P, sTip, f, oidx, ch0);
    }
    uint32_t r[16];
    float x[16];
    if (P.has_c || cimg) {  // net += fc_c[0](c) [+ W_img c_img]
      mbar_wait(bar, ph); ph ^= 1;
      tc_fence_after();
      tmem_ld16(tD + ch0, r);
      tc_wait_ld();
#pragma unroll
      for (int j = 0; j < 16; ++j) net[j] += __uint_as_float(r[j]);
    }

    // ---------------- residual blocks ----------------
    for (int i = 0; i < nb; ++i) {
      TC_STAMP(trace, 1);   // ALU phase starts (accumulator already read)
#pragma unroll
      for (int j = 0; j < 16; ++j) x[j] = fmaxf(net[j], 0.f);
      split_store16<MIXED>(tX, hv, x);
      TC_STAMP(trace, 2);   // operands computed, tcgen05.st issued
      tc_wait_st();
      tc_fence_before();
      TC_STAMP(trace, 3);   // stores complete
      group_sync2();
      TC_STAMP(trace, 4);   // group barrier passed
      if (wq == (step & 7) && elect_one()) {     // D = relu(net)*W0_i + ones*b0_i
        tc_fence_after();
        issue_product(mD, mX, wsm + 4 * VTACO_DEC_TC_MAT(kTcMode, 3 * i + 1), 0, n_prod);
        tc_mma_ts(mD, mOnes, make_bdesc(bsm + (2 * i + 1) * kKBlkBytes), 1);
        tc_commit(bar);
        TC_STAMP(trace, 20);  // issuer only: 13 MMAs + commit issued
      }
      ++step;
      TC_STAMP(trace, 5);   // (issuing warp: MMAs issued)
      mbar_wait(bar, ph); ph ^= 1;
      TC_STAMP(trace, 6);   // MMAs complete
      tc_fence_after();
      tmem_ld16(tD + ch0, r);
      tc_wait_ld();
      TC_STAMP(trace, 7);   // accumulator in registers
#pragma unroll
      for (int j = 0; j < 16; ++j) x[j] = fmaxf(__uint_as_float(r[j]), 0.f);
      split_store16<MIXED>(tX, hv, x);
      tc_wait_st();
      tc_fence_before();
      group_sync2();
      if (wq == (step & 7) && elect_one()) {     // D = relu(h)*W1_i + ones*(b1_i + bc_{i+1}) [+ C*Wc_{i+1}]
        tc_fence_after();
        issue_product(mD, mX, wsm + 4 * VTACO_DEC_TC_MAT(kTcMode, 3 * i + 2), 0, n_prod);
        tc_mma_ts(mD, mOnes, make_bdesc(bsm + (2 * i + 2) * kKBlkBytes), 1);
        if (P.has_c && i + 1 < nb) issue_product(mD, mC, wsm + 4 * VTACO_DEC_TC_MAT(kTcMode, 3 * (i + 1)), 1, n_prod);
        tc_commit(bar);
      }
      ++step;
      mbar_wait(bar, ph); ph ^= 1;
      tc_fence_after();
      tmem_ld16(tD + ch0, r);
      tc_wait_ld();
#pragma unroll
      for (int j = 0; j < 16; ++j) net[j] += __uint_as_float(r[j]);
    }

    TC_STAMP(trace, 19);    // blocks done
    // ---------------- heads: partial dot products of the two halves, combined through shared memory ----------------
    {
      const float* Wo = sSmall + 128;
      const float slope = P.leaky ? 0.2f : 0.0f;
      float o = 0.f, oc = 0.f;
#pragma unroll
      for (int j = 0; j < 16; ++j) {
        net[j] = net[j] > 0.f ? net[j] : net[j] * slope;
        o = fmaf(Wo[VTACO_DEC_TAIL_WOUT + ch0 + j], net[j], o);
      }
      if (P.contact) {
#pragma unroll
        for (int j = 0; j < 16; ++j) oc = fmaf(Wo[VTACO_DEC_TAIL_WCON + ch0 + j], net[j], oc);
      }
      if (hv == 1) { head[tq] = o; head[128 + tq] = oc; }
      group_sync2();
      if (hv == 0 && valid) {
        o = (Wo[VTACO_DEC_TAIL_BOUT] + o) + head[tq];
        store_logit(P, oidx, o);
        if (P.contact) P.contact[oidx] = (Wo[VTACO_DEC_TAIL_BCON] + oc) + head[128 + tq];
        vmin = fminf(vmin, o);
        vmax = fmaxf(vmax, o);
      }
    }
  }

  flush_minmax(P, vmin, vmax, lane);
  tmem_free_all(tmem_base, warp);
}

int tc_trace_begin(long long** trace, cudaStream_t stream) {
  static const bool want = getenv("VTACO_TC_TRACE") != nullptr;
  *trace = nullptr;
  if (want) {
    VTACO_CUDA_CHECK(cudaMalloc(trace, kTraceSlots * sizeof(long long)));
    VTACO_CUDA_CHECK(cudaMemsetAsync(*trace, 0, kTraceSlots * sizeof(long long), stream));
  }
  return VTACO_OK;
}

int tc_trace_end(long long* trace, const char* tag, cudaStream_t stream) {
  if (!trace) return VTACO_OK;
  long long h[kTraceSlots];
  VTACO_CUDA_CHECK(cudaStreamSynchronize(stream));
  VTACO_CUDA_CHECK(cudaMemcpy(h, trace, sizeof(h), cudaMemcpyDeviceToHost));
  cudaFree(trace);
  double sum[32][32] = {};
  long long cnt[32][32] = {};
  for (int i = 1; i < kTraceSlots && h[i]; ++i) {
    const int a = (int)(h[i - 1] >> 56) & 31, b = (int)(h[i] >> 56) & 31;
    const long long d = (h[i] & 0x00ffffffffffffffll) - (h[i - 1] & 0x00ffffffffffffffll);
    if (d >= 0 && d < 1000000) { sum[a][b] += (double)d; cnt[a][b]++; }
  }
  for (int a = 0; a < 32; ++a)
    for (int b = 0; b < 32; ++b)
      if (cnt[a][b]) fprintf(stderr, "[vtaco %s trace] %d -> %d : %8.0f cycles (n=%lld)\n", tag, a, b, sum[a][b] / cnt[a][b], cnt[a][b]);
  return VTACO_OK;
}

int launch_decoder_tc(DecParams P, bool dense, const float* wtc, cudaStream_t stream) {
  if (!wtc) return VTACO_ERR_INVALID_ARG;
  const bool mixed = (P.tc_products == 2);
  using Kernel = void (*)(DecParams, const float*, long long*);
  Kernel k;
  int threads, smem;
  const char* tag;
  if (P.tc_split == 2) {   // two threads per query
    k = dense ? (mixed ? decoder_tc2_kernel<true, true> : decoder_tc2_kernel<true, false>)
              : (mixed ? decoder_tc2_kernel<false, true> : decoder_tc2_kernel<false, false>);
    threads = kTc2Threads;
    smem = tc2_smem_layout(P.n_blocks).total;
    tag = "tc2";
  } else {
    k = dense ? (mixed ? decoder_tc_kernel<true, true> : decoder_tc_kernel<true, false>)
              : (mixed ? decoder_tc_kernel<false, true> : decoder_tc_kernel<false, false>);
    threads = kTcThreads;
    smem = tc_smem_layout(P.n_blocks).total;
    tag = "tc";
  }
  if (smem > 227 * 1024) return launch_decoder_simt(P, dense, stream);
  if (const int e = set_tc_tiles(P, dense)) return e;
  VTACO_CUDA_CHECK(smem_opt_in((const void*)k, smem));
  long long grid = (P.n_tiles + kTcGroups - 1) / kTcGroups;
  if (grid > num_sms()) grid = num_sms();
  long long* trace;
  if (const int e = tc_trace_begin(&trace, stream)) return e;
  k<<<(unsigned)grid, threads, smem, stream>>>(P, wtc, trace);
  VTACO_LAUNCH_CHECK();
  return tc_trace_end(trace, tag, stream);
}

}  // namespace vtaco
