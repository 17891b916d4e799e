/*
 * vtaco_b200.h — C ABI of the B200-native convolutional-occupancy hot path.
 *
 * Drop-in boundary for jeffsonyu/VTacO's conv-occupancy path.  The reference has
 * no FFI layer of its own (it is pure Python/PyTorch): its "operator API" is the
 * nn.Module interface of src/encoder/pointnet.py and
 * src/conv_onet/models/decoder.py, which vtaco_b200/ mirrors in Python.  Below
 * those modules every arithmetic step goes through the entry points declared
 * here; each one cites the reference code it replaces.
 *
 * Conventions
 *  - plain pointers + sizes only; every pointer is a DEVICE pointer unless the
 *    name ends in _host.  No torch types, no allocation.  Process-wide state is limited to
 *    idempotent caches held in atomics (SM count per device, the one-time opt-in of each
 *    kernel to its dynamic shared-memory size per device) and a THREAD-LOCAL copy of the last
 *    CUDA error for vtaco_last_cuda_error(): entry points may be called from several host
 *    threads; calls that share a stream are ordered by that stream as usual.
 *  - `stream` is a cudaStream_t passed as void*; all work is enqueued on it and
 *    the call returns without synchronising.
 *  - return value: 0 on success, negative vtaco_status on error (never throws).
 *  - all feature tensors are fp32; "channels-last" (CL) means the channel index
 *    is the fastest one: grid [B][Rz][Ry][Rx][C], plane [B][R_i1][R_i0][C].
 */
#ifndef VTACO_B200_H
#define VTACO_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VTACO_ABI_VERSION 1

typedef enum {
  VTACO_OK = 0,
  VTACO_ERR_INVALID_ARG = -1,   /* null pointer, bad size, bad enum */
  VTACO_ERR_UNSUPPORTED = -2,   /* shape outside what the kernels implement */
  VTACO_ERR_CUDA = -3,          /* a CUDA runtime call failed (see vtaco_last_cuda_error) */
  VTACO_ERR_CAPACITY = -4       /* caller-supplied output capacity too small */
} vtaco_status;

/* plane / volume kinds, in the reference's key vocabulary */
enum { VTACO_PLANE_XZ = 0, VTACO_PLANE_XY = 1, VTACO_PLANE_YZ = 2, VTACO_GRID = 3 };

/* `tensor / python_scalar`: CUDA ATen multiplies by fp32(1/d), CPU ATen divides (SURVEY §7.2-1) */
enum { VTACO_DIV_RECIPROCAL = 0, VTACO_DIV_TRUE = 1 };

enum { VTACO_SAMPLE_BILINEAR = 0, VTACO_SAMPLE_NEAREST = 1 };

int vtaco_abi_version(void);
const char* vtaco_status_string(int status);
/* cudaGetErrorString of the last CUDA error seen by this library on this thread */
const char* vtaco_last_cuda_error(void);

/* ------------------------------------------------------------------------- *
 * (1) point -> cell index.
 * Replaces normalize_coordinate (src/common.py:268-291) or
 * normalize_3d_coordinate (:293-309) followed by coordinate2index (:333-348).
 * p: [n_points][3].  kind: VTACO_PLANE_* or VTACO_GRID.  Writes int32 and/or
 * int64 flat cell indices (either pointer may be NULL) and, if non-NULL, the
 * normalised coordinates ([n_points][2] for planes, [n_points][3] for the grid).
 * ------------------------------------------------------------------------- */
int vtaco_point_to_cell(const float* p, int64_t n_points, double padding, int reso, int kind,
                        int div_mode, int32_t* idx32, int64_t* idx64, float* coord, void* stream);

/* ------------------------------------------------------------------------- *
 * (2) channels-first -> channels-last relayout of a feature tensor.
 * src [B][C][S] -> dst [B][S][C]  (S = R*R or R*R*R).  The decoder kernel
 * gathers from CL so one interpolation tap is one 128-byte line (C = 32).
 * ------------------------------------------------------------------------- */
int vtaco_relayout_cl(const float* src, float* dst, int B, int C, int64_t S, void* stream);
/* inverse: [B][S][C] -> [B][C][S] (API-facing tensors are channels-first) */
int vtaco_relayout_cf(const float* src, float* dst, int B, int C, int64_t S, void* stream);

/* ------------------------------------------------------------------------- *
 * (3) fused LocalDecoder forward.
 * Replaces LocalDecoder.forward / forward_img / forward_contact
 * (src/conv_onet/models/decoder.py:71-161): normalise + clamp, bi/trilinear
 * grid_sample (border, align_corners=True) of every present feature tensor,
 * sum, fc_p | fc_p_img, n_blocks x {fc_c[i], ResnetBlockFC}, fc_out
 * [, fc_out_contact] — one kernel, activations never leave the SM.
 * In dense mode it also replaces make_3d_grid (src/common.py:178-197) and the
 * chunk loop of Generator3D.eval_points (src/conv_onet/generation.py:338-383).
 *
 * Packed weight buffer (fp32, device), hidden = c_dim = 32: every weight K-major ("[in][out]", the
 * transpose of nn.Linear's), fc_p_img.weight split by columns into the 3 point inputs (OFF_WPI) and the
 * 32 c_img inputs (OFF_WIMG).  n_blocks blocks of BLOCK_STRIDE floats start at OFF_BLOCKS (offsets
 * VTACO_DEC_BLK_* inside a block), then the tail (offsets VTACO_DEC_TAIL_*; 2 floats of padding).
 * ------------------------------------------------------------------------- */
#define VTACO_DEC_HIDDEN 32
#define VTACO_DEC_OFF_WP 0        /* fc_p.weight^T [3][32] */
#define VTACO_DEC_OFF_BP 96       /* fc_p.bias [32] */
#define VTACO_DEC_OFF_WPI 128     /* fc_p_img.weight[:, :3]^T [3][32] */
#define VTACO_DEC_OFF_BPI 224     /* fc_p_img.bias [32] */
#define VTACO_DEC_OFF_WIMG 256    /* fc_p_img.weight[:, 3:]^T [32][32] */
#define VTACO_DEC_OFF_BLOCKS 1280
#define VTACO_DEC_BLOCK_STRIDE 3168
#define VTACO_DEC_BLK_WC 0        /* fc_c[i].weight^T [32][32] */
#define VTACO_DEC_BLK_BC 1024     /* fc_c[i].bias [32] */
#define VTACO_DEC_BLK_W0 1056     /* blocks[i].fc_0.weight^T [32][32] */
#define VTACO_DEC_BLK_B0 2080     /* blocks[i].fc_0.bias [32] */
#define VTACO_DEC_BLK_W1 2112     /* blocks[i].fc_1.weight^T [32][32] */
#define VTACO_DEC_BLK_B1 3136     /* blocks[i].fc_1.bias [32] */
#define VTACO_DEC_TAIL_WOUT 0     /* fc_out.weight [32] */
#define VTACO_DEC_TAIL_WCON 32    /* fc_out_contact.weight [32] */
#define VTACO_DEC_TAIL_BOUT 64    /* fc_out.bias */
#define VTACO_DEC_TAIL_BCON 65    /* fc_out_contact.bias */
#define VTACO_DEC_TAIL 68
#define VTACO_DEC_PACKED_FLOATS(n_blocks) (VTACO_DEC_OFF_BLOCKS + VTACO_DEC_BLOCK_STRIDE * (n_blocks) + VTACO_DEC_TAIL)
#define VTACO_MAX_TIPS 8
#define VTACO_MAX_BLOCKS 8   /* n_blocks the shared-memory-resident kernels can hold */

/* tcgen05 operand buffer `weights_tc` (fp32, device), built from `weights` by vtaco_decoder_pack_tc in one of
 * three pack modes.  Offsets in floats.  A K-block is a 32 (n = out) x 8 (k = in) operand slice in the UMMA
 * canonical K-major no-swizzle layout: float index of (n, k) = (k/4)*128 + (n/8)*32 + (n%8)*4 + (k%4).
 * A matrix holds one 32x32 weight: sub-block hi = rn_tf32(W) (4 K-blocks, the same index formula with k in
 * [0,32)), then lo = tf32(W - hi) (modes 0, 2) or, mode 1, the K = 64 BF16 correction operand
 * [bf16(W) ; bf16(W - hi)] with bf16 index of (n, k) = (k/8)*256 + (n/8)*64 + (n%8)*8 + (k%8); mode 2 adds
 * bf16(W) (K = 32, same bf16 index) and stores fc_0 / fc_1 times 0.5 (the kernel feeds them 2*relu(x) = x + |x|).
 * A bias step is a K-block with row k=0 = bias hi, k=1 = bias lo, other rows 0 (modes 0, 1), or the plain fp32
 * vector (mode 2).  Mode 2's input-layer K-blocks q = 0, 1 (fc_p) and 2, 3 (fc_p_img[:, :3]) are B1 = rows
 * (W_hi[:,0..2], (b + bc_0)_hi, W_hi[:,0..2], 0) and B2 = rows (W_lo[:,0..2], (b + bc_0)_lo, 0, 0, 0, 0), the
 * B operands of A = (px, py, pz, 1, px_lo, py_lo, pz_lo, 0). */
#define VTACO_DEC_TC_MODE_3XTF32 0   /* TF32 hi | TF32 lo: variants 2, 3, 5 */
#define VTACO_DEC_TC_MODE_BF16 1     /* TF32 hi | K = 64 BF16 correction: variants 4, 6 */
#define VTACO_DEC_TC_MODE_TILE4 2    /* TF32 hi | TF32 lo | bf16(W), fp32 bias vectors, K-block input layer: variant 7 */
#define VTACO_DEC_TC_MODE(variant) ((variant) == 7 ? 2 : ((variant) == 4 || (variant) == 6) ? 1 : 0)
#define VTACO_DEC_TC_KBLK_FLOATS 256
#define VTACO_DEC_TC_BVEC_FLOATS 32  /* a mode-2 bias step */
#define VTACO_DEC_TC_SUB_HI 0        /* sub-blocks of a matrix */
#define VTACO_DEC_TC_SUB_LO 1024
#define VTACO_DEC_TC_SUB_BF16 2048   /* mode 2 only */
#define VTACO_DEC_TC_MAT_FLOATS(mode) ((mode) == 2 ? 2560 : 2048)
/* matrix m = 3*i + {0, 1, 2}: fc_c[i].weight, blocks[i].fc_0.weight, blocks[i].fc_1.weight; in mode 2 also
 * m = 3*n_blocks: fc_p_img.weight[:, 3:] */
#define VTACO_DEC_TC_MAT(mode, m) ((m) * VTACO_DEC_TC_MAT_FLOATS(mode))
/* bias step s = 0 .. 2*n_blocks: bc_0 | b0_i, b1_i + bc_{i+1} (i = 0..n_blocks-1); after the matrices */
#define VTACO_DEC_TC_BIAS_STEP_FLOATS(mode) ((mode) == 2 ? VTACO_DEC_TC_BVEC_FLOATS : VTACO_DEC_TC_KBLK_FLOATS)
#define VTACO_DEC_TC_BIAS(mode, n_blocks, s) \
  (VTACO_DEC_TC_MAT(mode, 3 * (n_blocks) + ((mode) == 2)) + (s) * VTACO_DEC_TC_BIAS_STEP_FLOATS(mode))
/* fc_p_img.weight[:, 3:] (the product with a per-query c_img tensor): after the bias steps in modes 0 and 1 */
#define VTACO_DEC_TC_WIMG(mode, n_blocks) \
  ((mode) == 2 ? VTACO_DEC_TC_MAT(mode, 3 * (n_blocks)) : VTACO_DEC_TC_BIAS(mode, n_blocks, 2 * (n_blocks) + 1))
/* mode 2: input-layer K-block q = 0..3 */
#define VTACO_DEC_TC_INPUT(n_blocks, q) (VTACO_DEC_TC_BIAS(2, n_blocks, 2 * (n_blocks) + 1) + (q) * VTACO_DEC_TC_KBLK_FLOATS)
#define VTACO_DEC_TC_USED_FLOATS(mode, n_blocks) \
  ((mode) == 2 ? VTACO_DEC_TC_INPUT(n_blocks, 4) : VTACO_DEC_TC_WIMG(mode, n_blocks) + VTACO_DEC_TC_MAT_FLOATS(mode))
/* floats reserved for `weights_tc` in any mode: the widest matrices, a K-block per bias step, mode 2's input layer */
#define VTACO_DEC_TC_FLOATS(n_blocks) \
  ((3 * (n_blocks) + 1) * VTACO_DEC_TC_MAT_FLOATS(2) + (2 * (n_blocks) + 1 + 4) * VTACO_DEC_TC_KBLK_FLOATS)

typedef struct vtaco_decoder_args {
  /* ---- queries ---- */
  const float* p;          /* flat mode: [B][N][3]; NULL selects dense mode            */
  int32_t B;               /* batch (samples; each has its own feature tensors)          */
  int64_t N;               /* flat mode: queries per sample                              */
  /* dense mode: the lattice (1+padding)*make_3d_grid(nx^3); query (ix,iy,iz) has
   * p = (axis[ix], axis[iy], axis[iz]); rows ix in [x0, x1) are evaluated (slab).  */
  const float* axis;       /* [nx] exact axis values (host computes them like the reference) */
  int32_t nx, x0, x1;
  /* ---- features, channels-last; NULL = key absent.  Order of summation is
   * grid, xz, xy, yz as in decoder.py:75-82 ---- */
  const float* grid;       /* [B][Rg][Rg][Rg][32] */
  const float* plane[3];   /* xz, xy, yz: [B][Rp][Rp][32] */
  int32_t reso_grid, reso_plane;
  double padding;          /* python float of the reference (0.1); constants are formed in double */
  int32_t div_mode;        /* VTACO_DIV_* */
  int32_t sample_mode;     /* VTACO_SAMPLE_* */
  /* ---- network ---- */
  const float* weights;    /* packed, see above */
  int32_t n_blocks;
  int32_t leaky;           /* activation before fc_out: 0 ReLU, 1 LeakyReLU(0.2)         */
  int32_t use_img;         /* 0: net = fc_p(p); 1: net = fc_p_img(cat[p, c_img])         */
  const float* c_img;      /* use_img, dense tensor: [B][N][32] (dense mode: [nx^3][32]); may be NULL if tips used */
  /* compact tactile conditioning (dense mode; generation.py:190-200): a query takes
   * tip_feat[f] iff f = argmin_f |p - tip_f| (float64), that distance < tip_radius and
   * tip_touch[f] != 0.  Ignored when n_tips == 0. */
  int32_t n_tips;
  double tips[VTACO_MAX_TIPS][3];
  int32_t tip_touch[VTACO_MAX_TIPS];
  double tip_radius;
  const float* tip_feat;   /* [n_tips][32] device */
  /* ---- outputs ---- */
  float* logits;           /* flat: [B][N]; dense: [nx][nx][nx] (full grid base pointer) */
  float* contact;          /* optional second head (forward_contact), same shape, or NULL */
  int32_t* minmax_key;     /* optional [2]: ordered-int keys of min / max logit, updated with
                              atomicMin/atomicMax (caller initialises to INT32_MAX, INT32_MIN) */
  int32_t variant;         /* 0 = scalar-FFMA SIMT kernel; 1 = packed-FFMA2 SIMT kernel; 2 = tcgen05 3xTF32 kernel;
                            * 3 = single TF32 product (debug, ~1e-3); 4 = tcgen05 TF32 main product + BF16 corrections;
                            * 5 / 6 = 2 / 4 with two threads per query (768-thread CTAs, 3 tiles per SM);
                            * 7 = four tiles per SM (1024-thread CTAs): TF32 hi products + BF16 residual product, biases
                            *     on the CUDA cores (fastest; needs fewer than 2^31 outputs per call, else 5 is used) */
  /* variants 2-7: VTACO_DEC_TC_FLOATS(n_blocks) floats in pack mode VTACO_DEC_TC_MODE(variant) (layout
   * VTACO_DEC_TC_*, above), built by vtaco_decoder_pack_tc */
  const float* weights_tc;
  /* dense mode, multi-GPU: when n_peers > 0 every logit of the slab is stored to
   * logits_peers[0..n_peers) instead of `logits` — the (nx,nx,nx) grids of all ranks (own one
   * included), peer-mapped over NVLink (torch symmetric memory / CUDA IPC).  This fuses the
   * all-gather of the logit slabs into the decoder epilogue: no separate collective. */
  float* logits_peers[8];
  int32_t n_peers;
  /* optional NVLS multicast address of the same grids (all ranks bound to one multicast object):
   * when non-NULL (and n_peers > 0) each logit is written ONCE with multimem.st and the NVSwitch
   * replicates it to every rank, instead of n_peers unicast stores. */
  float* logits_multicast;
  /* compact tactile conditioning, third form (use_img): one byte per query (flat: [B*N]; dense:
   * [nx^3] in lattice order) — 0 = no tactile feature, k = tip_feat[k-1] (n_tips rows, tips[] /
   * tip_touch[] / tip_radius unused).  Built by vtaco_fingertip_ids / vtaco_tactile_point_map.
   * tcgen05 variants only. */
  const uint8_t* tip_map;
} vtaco_decoder_args;

int vtaco_decoder_forward(const vtaco_decoder_args* args, void* stream);
/* Interpolation only — LocalDecoder.sample_plane_feature / sample_grid_feature
 * (decoder.py:55-68).  Uses the feature / padding / div_mode / sample_mode fields of
 * `args`; p: [B][N][3]; out: [B][32][N] (sum over the present keys). */
int vtaco_sample_features(const vtaco_decoder_args* args, const float* p, int64_t N, float* out, void* stream);
/* ------------------------------------------------------------------------- *
 * (4b) Backward of LocalDecoder.forward / forward_img / forward_contact — what autograd
 * computes when src/conv_onet/training.py:79,617 trains through decoder.py:71-161
 * (SURVEY §8f-2).  Flat queries only.  The forward pass is recomputed in fp32 inside the
 * kernel (the forward kernels save nothing).  Gradient w.r.t. the query points p is not
 * produced (the reference never asks for it).
 *
 * d_params: flat fp32 buffer of VTACO_DEC_PACKED_FLOATS(n_blocks) floats, ACCUMULATED into
 * (zero it first): the fields of the packed forward weights (VTACO_DEC_OFF_*, _BLK_*, _TAIL_*), but
 * each matrix in nn.Linear's native [out][in] orientation (fc_p_img.weight[:, :3] [32][3] at OFF_WPI,
 * fc_p_img.weight[:, 3:] [32][32] at OFF_WIMG).
 * d_grid / d_plane[k]: channels-last gradients [B][R..][32], ACCUMULATED into with vector
 * atomics (NULL = not wanted).  d_c_img: [B][N][32], overwritten (NULL = not wanted).
 * workspace: vtaco_decoder_backward_workspace_bytes(B*N, n_blocks) bytes of device memory. */
typedef struct vtaco_decoder_bwd_args {
  const float* p;          /* [B][N][3] */
  int32_t B;
  int64_t N;
  const float* grid;       /* channels-last features as in vtaco_decoder_args, or NULL */
  const float* plane[3];   /* xz, xy, yz */
  int32_t reso_grid, reso_plane;
  double padding;
  int32_t div_mode, sample_mode;
  const float* weights;    /* packed forward weights (VTACO_DEC_* layout) */
  int32_t n_blocks, leaky;
  int32_t use_img;         /* 1: net0 = fc_p_img(cat(p, c_img)) */
  const float* c_img;      /* [B][N][32] or NULL */
  const float* dlogits;    /* [B][N] dL/dlogits, or NULL (then dcontact must be given) */
  const float* dcontact;   /* [B][N] dL/dcontact (forward_contact) or NULL */
  void* workspace;
  size_t workspace_bytes;
  float* d_params;
  float* d_grid;
  float* d_plane[3];
  float* d_c_img;
} vtaco_decoder_bwd_args;
size_t vtaco_decoder_backward_workspace_bytes(int64_t total_queries, int32_t n_blocks);
int vtaco_decoder_backward(const vtaco_decoder_bwd_args* args, void* stream);

/* ------------------------------------------------------------------------- *
 * (3b) Tactile conditioning maps (SURVEY 8f-1) — replace the reference's host-side construction
 * of c_img_all (scipy.cdist over all query points + a dense (N, c_dim) tensor).
 * vtaco_fingertip_ids: generation.py:190-200 / training.py:560-575.  ids[i] = f+1 where f is the
 *   NEAREST fingertip of query p[i] (float64 distances, first minimum), if that distance < radius
 *   and touch_host[f] != 0; else 0.  p: [n][3] device; tips_host: [n_tips][3] host doubles.
 * vtaco_tactile_point_map: generation.py:222-255 (encode_t2d).  map[i] = value for every query
 *   closer than `radius` (float64) to any of the n_pts points (device doubles [n_pts][3]); other
 *   entries are left untouched: zero the map, then call once per touched sensor t in increasing
 *   order with value = t+1 (later sensors overwrite, like the reference's loop).  Queries: flat
 *   p [n][3], or (p == NULL) the dense lattice axis[nx]^3 in lattice order.
 * ------------------------------------------------------------------------- */
int vtaco_fingertip_ids(const float* p, int64_t n, const double* tips_host, const int32_t* touch_host,
                        int32_t n_tips, double radius, uint8_t* ids, void* stream);
int vtaco_tactile_point_map(const float* p, int64_t n, const float* axis, int32_t nx, const double* pts,
                            int32_t n_pts, double radius, int32_t value, uint8_t* map, void* stream);

/* ------------------------------------------------------------------------- *
 * (4c) Weight packing, one launch each.  nn.Linear stores weight[out][in]; the kernels read
 * K-major "[in][out]" blocks (layouts above / below).  A descriptor copies one parameter:
 * element (n = out, k = in) = src[n*src_stride + src_col0 + k] -> dst[dst_off + k*out_dim + n]
 * (bias vectors: in_dim = 1).  At most VTACO_PACK_MAX_DESCS descriptors per call; `dst` must be
 * zero-initialised where no descriptor writes (padding, absent fc_c when c_dim = 0).
 * vtaco_decoder_pack_tc derives the tcgen05 operand buffer (`weights_tc`, VTACO_DEC_TC_FLOATS
 * floats) from the packed decoder buffer; `mixed` is the pack mode, VTACO_DEC_TC_MODE(variant).  It writes
 * every float of the mode's VTACO_DEC_TC_USED_FLOATS.
 * ------------------------------------------------------------------------- */
#define VTACO_PACK_MAX_DESCS 64
typedef struct vtaco_pack_desc {
  const float* src;
  int32_t out_dim, in_dim;
  int32_t src_stride;
  int32_t src_col0;
  int32_t dst_off;
} vtaco_pack_desc;
int vtaco_pack_linear(const vtaco_pack_desc* descs_host, int32_t n_descs, float* dst, int64_t dst_floats, void* stream);
int64_t vtaco_decoder_tc_floats(int32_t n_blocks);
int vtaco_decoder_pack_tc(const float* packed, int32_t n_blocks, int32_t mixed, float* dst, void* stream);

/* decode an ordered-int key written by the decoder / encoder kernels back to float (host helper) */
float vtaco_key_to_float_host(int32_t key);

/* ------------------------------------------------------------------------- *
 * (5) LocalPoolPointnet, PointNet part.
 * Replaces LocalPoolPointnet.forward up to (not including) the UNet/UNet3D
 * (src/encoder/pointnet.py:135-172): point->cell per key, fc_pos, n_blocks x
 * ResnetBlockFC(2H->H) with pool_local (:116-132; torch_scatter scatter_max or
 * scatter_mean + gather) between blocks, fc_c, and scatter_mean of the per-point
 * code into zero-filled feature planes / grid (:85-114).
 *
 * Keys are listed in the reference's insertion order (xz, xy, yz, grid; only the
 * enabled ones).  Outputs are CHANNELS-LAST dense tensors [B][cells][32]; the
 * Python module exposes them as (B,32,R,R[,R]) views in torch's channels_last
 * memory format, so values/shapes are the reference's and the decoder reads them
 * without a copy.
 *
 * Packed weights (hidden_dim = 32, c_dim = 32), every weight K-major ("[in][out]"): fc_pos, then
 * n_blocks blocks of BLOCK_STRIDE floats from OFF_BLOCKS (offsets VTACO_ENC_BLK_* inside a block),
 * then the fc_c section of VTACO_ENC_TAIL floats (offsets VTACO_ENC_FCC_*).
 * ------------------------------------------------------------------------- */
#define VTACO_ENC_OFF_WPOS 0      /* fc_pos.weight^T [3][64] */
#define VTACO_ENC_OFF_BPOS 192    /* fc_pos.bias [64] */
#define VTACO_ENC_OFF_BLOCKS 256
#define VTACO_ENC_BLOCK_STRIDE 5184
#define VTACO_ENC_BLK_W0 0        /* blocks[i].fc_0.weight^T [64][32] */
#define VTACO_ENC_BLK_B0 2048     /* blocks[i].fc_0.bias [32] */
#define VTACO_ENC_BLK_W1 2080     /* blocks[i].fc_1.weight^T [32][32] */
#define VTACO_ENC_BLK_B1 3104     /* blocks[i].fc_1.bias [32] */
#define VTACO_ENC_BLK_WS 3136     /* blocks[i].shortcut.weight^T [64][32] */
#define VTACO_ENC_FCC_W 0         /* fc_c.weight^T [32][32] */
#define VTACO_ENC_FCC_B 1024      /* fc_c.bias [32] */
#define VTACO_ENC_TAIL 1056
#define VTACO_ENC_PACKED_FLOATS(n_blocks) (VTACO_ENC_OFF_BLOCKS + VTACO_ENC_BLOCK_STRIDE * (n_blocks) + VTACO_ENC_TAIL)

typedef struct vtaco_encoder_args {
  const float* p;          /* [B][T][3] */
  int32_t B;
  int64_t T;
  double padding;
  int32_t div_mode;        /* VTACO_DIV_* */
  int32_t n_keys;          /* 1..4 */
  int32_t kind[4];         /* VTACO_PLANE_* / VTACO_GRID per key */
  int32_t reso[4];
  int32_t pool_mean;       /* scatter_type: 0 'max' (default), 1 'mean' */
  int32_t n_blocks;
  const float* weights;    /* packed, see above */
  void* workspace;         /* >= vtaco_encoder_workspace_bytes(...) */
  int64_t workspace_bytes;
  float* out_cl[4];        /* per key [B][cells][32], zero-filled by the call; NULL skips the key's output */
  float* c_out;            /* optional [B][T][32]: per-point code c = fc_c(net) */
  int32_t* index_out[4];   /* optional per key [B*T] int32 cell indices */
} vtaco_encoder_args;

int64_t vtaco_encoder_workspace_bytes(int32_t B, int64_t T, int32_t n_keys, const int32_t* kind, const int32_t* reso);
int vtaco_encoder_pointnet(const vtaco_encoder_args* args, void* stream);

/* (5b) Backward of the PointNet part (SURVEY §8f-2): what autograd computes through
 * src/encoder/pointnet.py:135-172 when training.py trains the encoder.  Given the gradients of
 * the scatter_mean feature tensors (channels-last, [B][cells][32] per key, NULL = no gradient
 * for that key; same key order as vtaco_encoder_args) it ACCUMULATES parameter gradients into
 * d_params (zero it first): the fields of the packed forward weights (VTACO_ENC_OFF_*, _BLK_*,
 * _FCC_*) with every matrix in nn.Linear's native [out][in] orientation (fc_pos.weight [64][3],
 * fc_0.weight [32][64]).  The forward is recomputed inside (nothing is saved
 * by vtaco_encoder_pointnet).  scatter_max routes a cell's gradient to the lowest-index point
 * among exact ties (torch_scatter: one arg-max point, unspecified which). */
typedef struct vtaco_encoder_bwd_args {
  const float* p;          /* [B][T][3] */
  int32_t B;
  int64_t T;
  double padding;
  int32_t div_mode;
  int32_t n_keys;
  int32_t kind[4];
  int32_t reso[4];
  int32_t pool_mean;
  int32_t n_blocks;
  const float* weights;    /* packed forward weights */
  void* workspace;
  int64_t workspace_bytes; /* >= vtaco_encoder_backward_workspace_bytes(...) */
  const float* d_out_cl[4];
  float* d_params;
} vtaco_encoder_bwd_args;
int64_t vtaco_encoder_backward_workspace_bytes(int32_t B, int64_t T, int32_t n_keys, const int32_t* kind,
                                               const int32_t* reso, int32_t n_blocks);
int vtaco_encoder_backward(const vtaco_encoder_bwd_args* args, void* stream);

/* pool_local stand-alone (src/encoder/pointnet.py:116-132): feat [B][T][32] row-major,
 * idx32_host_array[k] = device pointer to key k's [B*T] int32 cell indices, cells[k] = R^2 | R^3;
 * out [B][T][32] = sum over keys of (per-cell max | mean gathered back to the points). */
int64_t vtaco_pool_workspace_bytes(int32_t B, int64_t T, int32_t n_keys, const int64_t* cells_host);
int vtaco_pool_local(const float* feat, int32_t B, int64_t T, int32_t n_keys, const int32_t* const* idx32_host_array,
                     const int64_t* cells_host, int32_t mean, void* workspace, int64_t workspace_bytes, float* out,
                     void* stream);
/* scatter_mean stand-alone (pointnet.py:91-93,106-108): c [B][T][32] -> out_cl [B][cells][32] (zero-filled here).
 * workspace >= vtaco_pool_workspace_bytes(B, T, 1, &cells). */
int vtaco_scatter_mean(const float* c, const int32_t* idx32, int32_t B, int64_t T, int64_t cells, void* workspace,
                       int64_t workspace_bytes, float* out_cl, void* stream);

/* ------------------------------------------------------------------------- *
 * (6) marching cubes over the decoded grid.
 * Replaces skimage.measure.marching_cubes(value_grid, gradient_direction='ascent')
 * and the vertex rescale of Generator3D.generate_obj_mesh_wnf
 * (src/conv_onet/generation.py:268-272).  grid: [nx][ny][nz] fp32 (axis0 = x).
 * level = `level`, or 0.5f*(min+max) decoded from `level_keys` (the ordered-int keys
 * the decoder kernel / vtaco_grid_minmax maintain) — skimage's level=None.
 * A corner is above iff value > level; one vertex per cut grid edge (id order =
 * lattice order of the owning point, then axis); faces in lattice order of the
 * cell, then table order (oracle/mc_tables.py); vertices are
 * (index_coordinate - voffset) * vscale  (0,1 -> array-index coordinates).
 * counts (device int64[4]) always receives {V, F, V_numbered, -}; vertices / faces beyond the
 * given capacities are counted but not written (V > vertex_capacity or F > face_capacity: the
 * caller re-runs phase 2 with larger buffers).  phase: 1 = count, 2 = emit (after a count on the
 * same scratch), 3 = both.
 * Slab mode, for extraction sharded over GPUs by x-rows (SURVEY 8e, "gather of mesh pieces"):
 * `grid` holds the slab's rows followed by up to two halo rows and x_emit = number of owned rows.
 * Vertex ids are numbered over the whole sub-volume, but only vertices owned by rows < x_emit and
 * faces of cells in rows < x_emit are emitted / counted (V_numbered also counts the halo rows'),
 * so that a face may name a vertex id >= V: it is the (id - V)-th vertex of the NEXT slab.
 * Concatenating the pieces of consecutive slabs (ids + sum of the previous slabs' V) gives
 * exactly the mesh of the whole volume.  x_emit = 0 or nx: whole volume.  The halo rows may be read in place from
 * another buffer (halo_grid / halo_rows) instead of being part of `grid`.
 * ------------------------------------------------------------------------- */
typedef struct vtaco_mc_args {
  const float* grid;
  int32_t nx, ny, nz;
  float level;
  const int32_t* level_keys;   /* optional device int32[2 * n_level_keys]: (min,max) key pairs, reduced over the pairs */
  int32_t n_level_keys;        /* number of pairs (0 or 1 = one pair); >1: one pair per rank (fused exchange) */
  void* scratch;               /* >= vtaco_mc_scratch_bytes(nx,ny,nz) */
  int64_t scratch_bytes;
  float* vertices;             /* [vertex_capacity][3] */
  int64_t vertex_capacity;
  int32_t* faces;              /* [face_capacity][3] */
  int64_t face_capacity;
  int64_t* counts;             /* device int64[4] */
  float voffset, vscale;
  int32_t phase;
  int32_t x_emit;              /* slab mode: rows [0, x_emit) are owned; 0 = all */
  int32_t x_origin;            /* slab mode: lattice row of grid row 0 (vertex x = local row + x_origin) */
  const float* level_ptr;      /* optional device float: the level (takes precedence; written by vtaco_exchange_level) */
  /* slab mode, optional: the halo rows live somewhere else — rows [nx - halo_rows, nx) of the sub-volume are read
   * from halo_grid ([halo_rows][ny][nz]; e.g. the NEXT rank's first owned rows, peer-mapped over NVLink) and `grid`
   * holds only the first nx - halo_rows rows.  A rank then decodes its own rows only. */
  const float* halo_grid;
  int32_t halo_rows;
} vtaco_mc_args;

int64_t vtaco_mc_scratch_bytes(int32_t nx, int32_t ny, int32_t nz);
int vtaco_marching_cubes(const vtaco_mc_args* args, void* stream);
/* keys[0..1] <- ordered-int keys of min / max of grid[0..n) (initialised by the call) */
int vtaco_grid_minmax(const float* grid, int64_t n, int32_t* keys, void* stream);
/* multi-GPU iso-level exchange without a collective: copy this rank's (min,max) key pair into
 * slot `rank` (0..7) of each of the `n_peers` int32[world][2] tables given (peer-mapped pointers:
 * all ranks' tables for an all-gather, only the root's for a gather), then reset `keys` to
 * (INT32_MAX, INT32_MIN) for the next step. */
int vtaco_publish_keys(int32_t* keys, int32_t* const* tables_host_array, int32_t n_peers, int32_t rank, void* stream);

/* ------------------------------------------------------------------------- *
 * (6b) Multi-GPU exchange of the sharded extraction (SURVEY 8e; call site of the pieces:
 * generation.py:268-272 on x-slabs).  Device-side signalling over peer-mapped memory — no host
 * synchronisation, capturable in a CUDA graph.  Every rank owns a zero-initialised control block
 * of VTACO_EXCHANGE_CTRL_BYTES in memory that all ranks can address (torch symmetric memory /
 * CUDA IPC); ctrl[r] is rank r's block as mapped into THIS process.  All ranks must make the same
 * sequence of calls.  A wait that sees no peer for ~2 s gives up and sets the int32 at
 * VTACO_EXCHANGE_ERR_OFFSET of the local block to 1 (results are then undefined).
 *
 * vtaco_exchange_level: all-gather of the ranks' (min,max) ordered-int key pairs (`keys`, as the
 *   decoder maintains them; reset to (INT32_MAX, INT32_MIN) by the call); writes
 *   0.5f*(min+max) — skimage's level=None over the WHOLE lattice — to the float at
 *   VTACO_EXCHANGE_LEVEL_OFFSET of the local block (pass that address as vtaco_mc_args.level_ptr).
 * vtaco_exchange_mesh: all-gather of the pieces' (V,F) counts (the slab-mode counts of
 *   vtaco_marching_cubes), exclusive scan, then every rank copies its vertices to
 *   dst_vertices[r] + 3*vbase and its faces (+vbase) to dst_faces[r] + 3*fbase for every r with
 *   non-NULL destinations (peer-mapped buffers of rank r: all ranks for an all-gather, one for a
 *   gather).  A destination rank returns (in stream order) only after all pieces have landed;
 *   total_counts (local device int64[2], optional) receives the mesh totals {V, F}.  Pieces that
 *   exceed the capacities are truncated — compare the totals with the capacities.
 *   Re-use of the destination buffers by the next step is safe when the destination rank
 *   consumes them in stream order before its next vtaco_exchange_mesh.
 * ------------------------------------------------------------------------- */
#define VTACO_EXCHANGE_CTRL_BYTES 1024
#define VTACO_EXCHANGE_ERR_OFFSET 556
#define VTACO_EXCHANGE_LEVEL_OFFSET 560
#define VTACO_EXCHANGE_BASE_OFFSET 568   /* int64[4]: this rank's vertex base, face base, total V, total F */
typedef struct vtaco_exchange {
  void* ctrl[8];
  int32_t world, rank;
} vtaco_exchange;
typedef struct vtaco_mesh_piece {
  const int64_t* counts;       /* device int64[>=2]: {V, F} of this rank's piece */
  const float* vertices;       /* [V][3] */
  const int32_t* faces;        /* [F][3], vertex ids local to the piece (may exceed V: next piece) */
  float* dst_vertices[8];
  int32_t* dst_faces[8];
  int64_t vertex_capacity, face_capacity;   /* of every destination buffer, in vertices / faces */
  int64_t* total_counts;
} vtaco_mesh_piece;
int vtaco_exchange_level(const vtaco_exchange* ex, int32_t* keys, void* stream);
int vtaco_exchange_mesh(const vtaco_exchange* ex, const vtaco_mesh_piece* piece, void* stream);

/* ------------------------------------------------------------------------- *
 * (7) GroupNorm of the UNet3D that post-processes the feature grid
 * (reference src/encoder/unet3d.py, layer order 'gcr': nn.GroupNorm before every Conv3d).
 * x, y: contiguous [N][C][S] fp32 (y may alias x); gamma/beta [C] or NULL;
 * stats_ws: device double[2*N*G] scratch.  Same result as torch.nn.functional.group_norm
 * to fp32 rounding (biased variance, eps inside the sqrt).
 * ------------------------------------------------------------------------- */
int vtaco_group_norm(const float* x, float* y, const float* gamma, const float* beta, int32_t N, int32_t C,
                     int32_t G, int64_t S, double eps, double* stats_ws, void* stream);
/* same for channels-last storage [N][S][C] (torch channels_last_3d); returns VTACO_ERR_UNSUPPORTED
 * unless C % 4 == 0, (C/G) % 4 == 0 and (C/4) divides 256 — callers then use vtaco_group_norm. */
int vtaco_group_norm_cl(const float* x, float* y, const float* gamma, const float* beta, int32_t N, int32_t C,
                        int32_t G, int64_t S, double eps, double* stats_ws, void* stream);

/* ------------------------------------------------------------------------- *
 * (7b) UNet3D layers on the tensor cores (SURVEY 8f-3; reference src/encoder/unet3d.py:
 * SingleConv order 'gcr' = GroupNorm -> Conv3d(3x3x3, padding 1, no bias) -> ReLU; Encoder =
 * MaxPool3d(2) + DoubleConv; Decoder = nearest-upsample + concat + DoubleConv; final 1x1x1 conv).
 * Activations are CHANNELS-LAST [N][D][H][W][C] fp32.  vtaco_conv3d_cl is one fused layer:
 *   y = [relu]( conv_k( GN(x_cat) ) [+ bias] ),  x_cat = cat(x, nearest_upsample(x2)) along C
 * where GN is applied per element from per-channel statistics: in_stats[n][c] = (sum, sum of
 * squares) of x_cat's channel c over the sample's D*H*W voxels, accumulated by the PRODUCER of
 * the tensor (this call's out_stats, vtaco_maxpool2_cl, vtaco_channel_stats_cl; for the upsampled
 * half multiply the half-resolution sums by 8).  in_stats = NULL: no GroupNorm.  x2 = NULL (C2 =
 * 0): no concat.  out_stats (optional, ZEROED by the caller) receives the per-channel sums of y.
 * Arithmetic: implicit GEMM on tcgen05 in single-pass TF32 (operands rounded to nearest TF32,
 * fp32 accumulation) — the arithmetic of the reference on a GPU (cuDNN, allow_tf32 default).
 * Packed weights: float index of W[co][ci][dz][dy][dx] =
 *   ((((co/32) * (Cin/16) + ci/16) * k^3 + (dz*k+dy)*k+dx) * 4 + (ci%16)/4) * 128 + (co%32)*4 + ci%4,
 * values pre-rounded to TF32.  Requires C1 % 16 == C2 % 16 == 0, Cout % 32 == 0, Cin <= 512, k in {1,3}.
 * ------------------------------------------------------------------------- */
typedef struct vtaco_conv3d_args {
  const float* x;          /* [N][D][H][W][C1] */
  const float* x2;         /* optional [N][D2][H2][W2][C2], read at nearest-upsampled positions */
  int32_t N, D, H, W, C1, C2, D2, H2, W2;
  const float* w_packed;
  const float* bias;       /* optional [Cout] */
  int32_t Cout, ksize;
  const double* in_stats;  /* optional [N][C1+C2][2] */
  const float* gamma;      /* GroupNorm weight [C1+C2] (NULL: 1) */
  const float* beta;       /* GroupNorm bias (NULL: 0) */
  int32_t groups;
  double eps;
  int32_t relu;
  float* y;                /* [N][D][H][W][Cout] */
  double* out_stats;       /* optional [N][Cout][2], accumulated */
  int32_t ksize_z;         /* extent of the filter along z: 0 = ksize (3-D convolution), 1 = a 2-D k x k convolution on
                              every z-slice (packed weights then hold k*k taps: W[co][ci][dy][dx]) */
} vtaco_conv3d_args;
int vtaco_conv3d_cl(const vtaco_conv3d_args* args, void* stream);
/* MaxPool3d(kernel 2, stride 2), channels-last; stats (optional, zeroed by the caller, N must be 1):
 * per-channel (sum, sumsq) of y.  D, H, W even; C % 4 == 0. */
int vtaco_maxpool2_cl(const float* x, float* y, int32_t N, int32_t D, int32_t H, int32_t W, int32_t C,
                      double* stats, void* stream);
/* per-channel (sum, sumsq) of one channels-last sample x [S][C] accumulated into stats [C][2]
 * (zeroed by the caller); C % 4 == 0 and C/4 divides 256. */
int vtaco_channel_stats_cl(const float* x, int64_t S, int32_t C, double* stats, void* stream);
/* (7c) 2-D U-Net on the feature planes (reference src/encoder/unet.py:45-239): its 3x3 / 1x1 convolutions run on
 * vtaco_conv3d_cl with D = 1 (a 2-D filter is the middle z-slice of a 3x3x3 one; bias + ReLU in the epilogue, no
 * GroupNorm; the skip connection is the second input at the same resolution).  The two other layers:
 * vtaco_maxpool2d_cl: MaxPool2d(2) on x [N][H][W][C] -> y [N][H/2][W/2][C] (H, W even, C % 4 == 0);
 * vtaco_depth_to_space2_cl: x [N][H][W][4*C], channel (a*2+b)*C + c -> y [N][2H][2W][C] at (2i+a, 2j+b) — the
 *   interleave of ConvTranspose2d(kernel 2, stride 2), whose arithmetic is a 1x1 convolution to 4*C channels. */
int vtaco_maxpool2d_cl(const float* x, float* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);
int vtaco_depth_to_space2_cl(const float* x, float* y, int32_t N, int32_t H, int32_t W, int32_t C, void* stream);

/* UNet3D decoder input in one pass (src/encoder/unet3d.py Decoder.forward):
 * out [N][C1+C2][Do][Ho][Wo] = cat(skip [N][C1][Do][Ho][Wo], nearest-upsample(x [N][C2][Di][Hi][Wi]), dim=1),
 * contiguous NCDHW fp32, ATen's nearest source index min(floor(dst * in/out), in-1).
 * Wo % 4 != 0 -> VTACO_ERR_UNSUPPORTED. */
int vtaco_upsample_concat3d(const float* skip, const float* x, float* out, int32_t N, int32_t C1, int32_t C2,
                            int32_t Do, int32_t Ho, int32_t Wo, int32_t Di, int32_t Hi, int32_t Wi, void* stream);

/* ------------------------------------------------------------------------- *
 * (4) self-measured FP32 FMA peak (roofline denominator of the decoder; SURVEY §8d).
 * Runs a register-resident FMA loop on every SM and returns achieved FLOP/s in
 * *flops_per_s_host.  variant 0: scalar FFMA, 1: packed FFMA2 (fma.rn.f32x2).
 * Synchronises the stream (measurement helper, not a data-path call).
 * ------------------------------------------------------------------------- */
int vtaco_fp32_peak(int variant, int iters, double* flops_per_s_host, void* stream);

/* ------------------------------------------------------------------------- *
 * (9) Chamfer distance — the metric computed right after mesh extraction
 * (src/common.py:54-137 chamfer_distance{,_naive,_kdtree}, called by
 * generation.py:281 on 2048 mesh vertices vs 2048 ground-truth points).
 * p1 [B][T1][3], p2 [B][T2][3].  dist12[b][i] = min_j |p1_i - p2_j|^2 (fp32, (dx^2+dy^2)+dz^2),
 * idx12 = the arg-min (first minimum), dist21 / idx21 the other direction; idx* optional.
 * chamfer1[b] = mean_i dist12, chamfer2[b] = mean_j dist21 (optional).  The reference's
 * value is chamfer1 + chamfer2. */
int vtaco_chamfer(const float* p1, const float* p2, int32_t B, int64_t T1, int64_t T2, float* dist12, int32_t* idx12,
                  float* dist21, int32_t* idx21, float* chamfer1, float* chamfer2, void* stream);

/* ------------------------------------------------------------------------- *
 * (10) Earth-Mover distance — the other metric of generate_obj_mesh_wnf
 * (src/common.py:45-51, called at generation.py:282): cost of the minimum-cost matching
 * between p1 [n1][3] and p2 [n2][3] under the float64 Euclidean distance, divided by n1
 * (scipy cdist + linear_sum_assignment in the reference).  Float64 auction algorithm with
 * epsilon-scaling on the device; the result is within eps_final (<= 0: 1e-9) of the optimum.
 * n1 != n2: min(n1,n2) pairs are matched, like linear_sum_assignment.  assignment (optional,
 * device int32[n1]): matched row of p2 or -1.  Synchronises the stream (the auction's
 * termination test and the result are host reads). max(n1,n2) <= 8192.
 * ------------------------------------------------------------------------- */
int64_t vtaco_emd_workspace_bytes(int64_t n1, int64_t n2);
int vtaco_emd(const float* p1, int64_t n1, const float* p2, int64_t n2, void* workspace, int64_t workspace_bytes,
              double eps_final, double* emd_host, int32_t* assignment, int64_t* iterations_host, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* VTACO_B200_H */
