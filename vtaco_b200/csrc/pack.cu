// Weight packing in ONE launch each (instead of ~100 torch slice-assign launches per parameter
// version): nn.Linear parameters -> the K-major fp32 buffers the encoder / decoder kernels read
// (layouts in include/vtaco_b200.h), and that buffer -> the UMMA canonical TF32 hi/lo (or
// TF32 + BF16-correction) operand blocks of the tcgen05 decoder.  Training re-packs after every
// optimizer step (reference training.py:79,617 trains through these modules), so the pack is on
// the training hot path.
#include "common.cuh"
#include <cuda_bf16.h>

namespace vtaco {

struct PackDescs {
  vtaco_pack_desc d[VTACO_PACK_MAX_DESCS];
};

// one block per descriptor; element (n = out, k = in) of the parameter goes to
// dst[dst_off + k * out_dim + n]  (K-major: "[in][out]")
__global__ void __launch_bounds__(256) pack_linear_kernel(const __grid_constant__ PackDescs D, float* __restrict__ dst) {
  const vtaco_pack_desc& e = D.d[blockIdx.x];
  const int count = e.out_dim * e.in_dim;
  for (int i = threadIdx.x; i < count; i += blockDim.x) {
    const int k = i / e.out_dim, n = i - k * e.out_dim;   // consecutive threads -> consecutive dst
    dst[e.dst_off + i] = __ldg(e.src + (size_t)n * e.src_stride + e.src_col0 + k);
  }
}

__device__ __forceinline__ float tf32_rn(float w) {   // round to nearest, ties away (magnitude)
  return __uint_as_float((__float_as_uint(w) + 0x1000u) & 0xffffe000u);
}
__device__ __forceinline__ float tf32_trunc(float w) { return __uint_as_float(__float_as_uint(w) & 0xffffe000u); }

// blocks [0, n_mats): 32x32 matrices (K-major source at packed[src_off[m] + k*32 + n]);
// blocks [n_mats, n_mats + n_bias): bias K-blocks (sum of up to two 32-vectors).
struct TcPackPlan {
  int n_mats, n_bias, mixed;
  int mat_src[3 * VTACO_MAX_BLOCKS + 1];    // float offsets into `packed`
  int mat_dst[3 * VTACO_MAX_BLOCKS + 1];    // float offsets into the tc buffer
  int bias_src0[2 * VTACO_MAX_BLOCKS + 1];  // -1 = zero
  int bias_src1[2 * VTACO_MAX_BLOCKS + 1];
  int bias_dst;
  int pw_dst;
};

__global__ void __launch_bounds__(256) pack_tc_kernel(const __grid_constant__ TcPackPlan Pn,
                                                      const float* __restrict__ packed, float* __restrict__ dst) {
  const int b = blockIdx.x;
  if (b < Pn.n_mats) {
    const float* src = packed + Pn.mat_src[b];
    float* out = dst + Pn.mat_dst[b];
    for (int i = threadIdx.x; i < VTACO_DEC_HIDDEN * VTACO_DEC_HIDDEN; i += blockDim.x) {
      const int k = i >> 5, n = i & 31;
      float w = __ldg(src + i);                            // W[n][k] (nn.Linear weight[out=n][in=k])
      if (Pn.mixed == 2 && b < 3 * ((Pn.n_mats - 1) / 3) && (b % 3) != 0) w *= 0.5f;   // variant 7: fc_0 / fc_1 take 2*relu(x)
      const float hi = tf32_rn(w);
      const int idx = (k >> 2) * 128 + (n >> 3) * 32 + (n & 7) * 4 + (k & 3);
      out[VTACO_DEC_TC_SUB_HI + idx] = hi;
      if (Pn.mixed == 2) {   // TF32 hi | TF32 lo | bf16(W) (K = 32)
        out[VTACO_DEC_TC_SUB_LO + idx] = tf32_trunc(w - hi);
        __nv_bfloat16* o16 = reinterpret_cast<__nv_bfloat16*>(out + VTACO_DEC_TC_SUB_BF16);
        o16[(k >> 3) * 256 + (n >> 3) * 64 + (n & 7) * 8 + (k & 7)] = __float2bfloat16_rn(w);
      } else if (Pn.mixed) {   // K = 64 BF16 correction operand: rows k < 32 bf16(W), rows k >= 32 bf16(W - hi)
        __nv_bfloat16* o16 = reinterpret_cast<__nv_bfloat16*>(out + VTACO_DEC_TC_SUB_LO);
        const int k1 = k + 32;
        o16[(k >> 3) * 256 + (n >> 3) * 64 + (n & 7) * 8 + (k & 7)] = __float2bfloat16_rn(w);
        o16[(k1 >> 3) * 256 + (n >> 3) * 64 + (n & 7) * 8 + (k1 & 7)] = __float2bfloat16_rn(w - hi);
      } else {
        out[VTACO_DEC_TC_SUB_LO + idx] = tf32_trunc(w - hi);
      }
    }
  } else if (b >= Pn.n_mats + Pn.n_bias) {
    // variant 7: fc_p / fc_p_img[:, :3] (+ their bias + bc_0) as K = 8 operand blocks for the 3xTF32 product
    // with A = (px, py, pz, 1, px_lo, py_lo, pz_lo, 0):  B1 rows (W_hi x3, b_hi, W_hi x3, 0), B2 rows (W_lo x3, b_lo, 0 x4)
    const int q = b - Pn.n_mats - Pn.n_bias;          // 0: fc_p B1, 1: fc_p B2, 2: fc_p_img B1, 3: fc_p_img B2
    const int wsrc = (q >> 1) ? VTACO_DEC_OFF_WPI : VTACO_DEC_OFF_WP;
    const int bsrc = (q >> 1) ? VTACO_DEC_OFF_BPI : VTACO_DEC_OFF_BP;
    float* out = dst + Pn.pw_dst + q * VTACO_DEC_TC_KBLK_FLOATS;
    const int i = threadIdx.x;                        // 256 threads == one K-block
    const int k = (i >> 7) * 4 + (i & 3), n = ((i >> 5) & 3) * 8 + ((i >> 2) & 7);
    const int kk = k & 3;
    float v;
    if (kk < 3) {
      v = __ldg(packed + wsrc + kk * 32 + n);
    } else {
      v = __ldg(packed + bsrc + n);
      if (Pn.bias_src0[0] >= 0) v = v + __ldg(packed + Pn.bias_src0[0] + n);   // + bc_0
    }
    const float hi = tf32_rn(v);
    float o;
    if ((q & 1) == 0) o = (k == 7) ? 0.f : hi;                          // B1
    else o = (k < 4) ? tf32_trunc(v - hi) : 0.f;                       // B2
    out[i] = o;
  } else {
    const int s = b - Pn.n_mats;
    if (Pn.mixed == 2) {   // the four-tile kernel adds the biases on the CUDA cores: plain fp32 vectors
      if (threadIdx.x < VTACO_DEC_TC_BVEC_FLOATS) {
        float bsum = 0.f;
        if (Pn.bias_src0[s] >= 0) bsum = __ldg(packed + Pn.bias_src0[s] + threadIdx.x);
        if (Pn.bias_src1[s] >= 0) bsum = bsum + __ldg(packed + Pn.bias_src1[s] + threadIdx.x);
        dst[Pn.bias_dst + s * VTACO_DEC_TC_BVEC_FLOATS + threadIdx.x] = bsum;
      }
      return;
    }
    float* out = dst + Pn.bias_dst + s * VTACO_DEC_TC_KBLK_FLOATS;
    for (int i = threadIdx.x; i < VTACO_DEC_TC_KBLK_FLOATS; i += blockDim.x) {
      // layout (k/4)*128 + (n/8)*32 + (n%8)*4 + (k%4) with k in [0,8): i -> (k, n)
      const int k = (i >> 7) * 4 + (i & 3), n = ((i >> 5) & 3) * 8 + ((i >> 2) & 7);
      float v = 0.f;
      if (k < 2) {
        float bsum = 0.f;
        if (Pn.bias_src0[s] >= 0) bsum = __ldg(packed + Pn.bias_src0[s] + n);
        if (Pn.bias_src1[s] >= 0) bsum = bsum + __ldg(packed + Pn.bias_src1[s] + n);
        const float hi = tf32_rn(bsum);
        v = (k == 0) ? hi : tf32_trunc(bsum - hi);
      }
      out[i] = v;
    }
  }
}

}  // namespace vtaco

using namespace vtaco;

extern "C" int vtaco_pack_linear(const vtaco_pack_desc* descs_host, int32_t n_descs, float* dst, int64_t dst_floats,
                                 void* stream) {
  if (!descs_host || !dst || n_descs < 1 || n_descs > VTACO_PACK_MAX_DESCS) return VTACO_ERR_INVALID_ARG;
  PackDescs D = {};
  for (int i = 0; i < n_descs; ++i) {
    const vtaco_pack_desc& e = descs_host[i];
    if (!e.src || e.out_dim < 1 || e.in_dim < 1 || e.src_stride < 1 || e.src_col0 < 0 || e.dst_off < 0)
      return VTACO_ERR_INVALID_ARG;
    if ((int64_t)e.dst_off + (int64_t)e.out_dim * e.in_dim > dst_floats) return VTACO_ERR_CAPACITY;
    D.d[i] = e;
  }
  pack_linear_kernel<<<n_descs, 256, 0, (cudaStream_t)stream>>>(D, dst);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}

extern "C" int64_t vtaco_decoder_tc_floats(int32_t n_blocks) {
  if (n_blocks < 0 || n_blocks > VTACO_MAX_BLOCKS) return VTACO_ERR_INVALID_ARG;
  return VTACO_DEC_TC_FLOATS(n_blocks);
}

extern "C" int vtaco_decoder_pack_tc(const float* packed, int32_t n_blocks, int32_t mixed, float* dst, void* stream) {
  if (!packed || !dst || n_blocks < 0 || n_blocks > VTACO_MAX_BLOCKS) return VTACO_ERR_INVALID_ARG;
  if (mixed < 0 || mixed > 2) return VTACO_ERR_INVALID_ARG;
  TcPackPlan Pn = {};
  Pn.mixed = mixed;
  const int nb = n_blocks;
  for (int i = 0; i < nb; ++i) {
    const int o = VTACO_DEC_OFF_BLOCKS + i * VTACO_DEC_BLOCK_STRIDE;
    const int srcs[3] = {o + VTACO_DEC_BLK_WC, o + VTACO_DEC_BLK_W0, o + VTACO_DEC_BLK_W1};   // fc_c[i], fc_0, fc_1
    for (int j = 0; j < 3; ++j) {
      Pn.mat_src[3 * i + j] = srcs[j];
      Pn.mat_dst[3 * i + j] = VTACO_DEC_TC_MAT(mixed, 3 * i + j);
    }
  }
  Pn.mat_src[3 * nb] = VTACO_DEC_OFF_WIMG;                       // fc_p_img.weight[:, 3:]
  Pn.mat_dst[3 * nb] = VTACO_DEC_TC_WIMG(mixed, nb);
  Pn.n_mats = 3 * nb + 1;
  // bias steps: bc_0 | b0_i, b1_i + bc_{i+1}
  Pn.bias_dst = VTACO_DEC_TC_BIAS(mixed, nb, 0);
  Pn.n_bias = 2 * nb + 1;
  Pn.bias_src0[0] = nb > 0 ? VTACO_DEC_OFF_BLOCKS + VTACO_DEC_BLK_BC : -1;
  Pn.bias_src1[0] = -1;
  for (int i = 0; i < nb; ++i) {
    const int o = VTACO_DEC_OFF_BLOCKS + i * VTACO_DEC_BLOCK_STRIDE;
    Pn.bias_src0[2 * i + 1] = o + VTACO_DEC_BLK_B0;
    Pn.bias_src1[2 * i + 1] = -1;
    Pn.bias_src0[2 * i + 2] = o + VTACO_DEC_BLK_B1;
    Pn.bias_src1[2 * i + 2] = (i + 1 < nb) ? o + VTACO_DEC_BLOCK_STRIDE + VTACO_DEC_BLK_BC : -1;
  }
  Pn.pw_dst = VTACO_DEC_TC_INPUT(nb, 0);     // mode 2 only
  pack_tc_kernel<<<Pn.n_mats + Pn.n_bias + (mixed == 2 ? 4 : 0), 256, 0, (cudaStream_t)stream>>>(Pn, packed, dst);
  VTACO_LAUNCH_CHECK();
  return VTACO_OK;
}
