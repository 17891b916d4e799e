"""ctypes binding of the C ABI declared in include/vtaco_b200.h.

The shared library (vtaco_b200/lib/libvtaco_b200.so) is built in-tree by
`python -m vtaco_b200.build`.  There is NO fallback: if the library is missing
or a call fails, a RuntimeError is raised.
"""
import ctypes as C
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, 'lib', 'libvtaco_b200.so')

MAX_TIPS = 8
MAX_BLOCKS = 8
PLANE_XZ, PLANE_XY, PLANE_YZ, GRID = 0, 1, 2, 3
KIND = {'xz': PLANE_XZ, 'xy': PLANE_XY, 'yz': PLANE_YZ, 'grid': GRID}
DIV_RECIPROCAL, DIV_TRUE = 0, 1
SAMPLE = {'bilinear': 0, 'nearest': 1}

# packed parameter layouts (VTACO_DEC_* / VTACO_ENC_* of include/vtaco_b200.h)
DEC_HIDDEN = 32
DEC_OFF_WP, DEC_OFF_BP, DEC_OFF_WPI, DEC_OFF_BPI, DEC_OFF_WIMG = 0, 96, 128, 224, 256
DEC_OFF_BLOCKS, DEC_BLOCK_STRIDE, DEC_TAIL = 1280, 3168, 68
DEC_BLK_WC, DEC_BLK_BC, DEC_BLK_W0, DEC_BLK_B0, DEC_BLK_W1, DEC_BLK_B1 = 0, 1024, 1056, 2080, 2112, 3136
DEC_TAIL_WOUT, DEC_TAIL_WCON, DEC_TAIL_BOUT, DEC_TAIL_BCON = 0, 32, 64, 65
ENC_OFF_WPOS, ENC_OFF_BPOS, ENC_OFF_BLOCKS, ENC_BLOCK_STRIDE = 0, 192, 256, 5184
ENC_BLK_W0, ENC_BLK_B0, ENC_BLK_W1, ENC_BLK_B1, ENC_BLK_WS = 0, 2048, 2080, 3104, 3136
ENC_FCC_W, ENC_FCC_B, ENC_TAIL = 0, 1024, 1056


def dec_packed_floats(n_blocks):
    return DEC_OFF_BLOCKS + DEC_BLOCK_STRIDE * n_blocks + DEC_TAIL


def enc_packed_floats(n_blocks):
    return ENC_OFF_BLOCKS + ENC_BLOCK_STRIDE * n_blocks + ENC_TAIL


class DecoderArgs(C.Structure):
    _fields_ = [
        ('p', C.c_void_p), ('B', C.c_int32), ('N', C.c_int64),
        ('axis', C.c_void_p), ('nx', C.c_int32), ('x0', C.c_int32), ('x1', C.c_int32),
        ('grid', C.c_void_p), ('plane', C.c_void_p * 3),
        ('reso_grid', C.c_int32), ('reso_plane', C.c_int32),
        ('padding', C.c_double), ('div_mode', C.c_int32), ('sample_mode', C.c_int32),
        ('weights', C.c_void_p), ('n_blocks', C.c_int32), ('leaky', C.c_int32), ('use_img', C.c_int32),
        ('c_img', C.c_void_p),
        ('n_tips', C.c_int32), ('tips', (C.c_double * 3) * MAX_TIPS), ('tip_touch', C.c_int32 * MAX_TIPS),
        ('tip_radius', C.c_double), ('tip_feat', C.c_void_p),
        ('logits', C.c_void_p), ('contact', C.c_void_p), ('minmax_key', C.c_void_p),
        ('variant', C.c_int32), ('weights_tc', C.c_void_p),
        ('logits_peers', C.c_void_p * 8), ('n_peers', C.c_int32), ('logits_multicast', C.c_void_p),
        ('tip_map', C.c_void_p),
    ]


class DecoderBwdArgs(C.Structure):
    _fields_ = [
        ('p', C.c_void_p), ('B', C.c_int32), ('N', C.c_int64),
        ('grid', C.c_void_p), ('plane', C.c_void_p * 3),
        ('reso_grid', C.c_int32), ('reso_plane', C.c_int32),
        ('padding', C.c_double), ('div_mode', C.c_int32), ('sample_mode', C.c_int32),
        ('weights', C.c_void_p), ('n_blocks', C.c_int32), ('leaky', C.c_int32), ('use_img', C.c_int32),
        ('c_img', C.c_void_p), ('dlogits', C.c_void_p), ('dcontact', C.c_void_p),
        ('workspace', C.c_void_p), ('workspace_bytes', C.c_size_t),
        ('d_params', C.c_void_p), ('d_grid', C.c_void_p), ('d_plane', C.c_void_p * 3), ('d_c_img', C.c_void_p),
    ]


class EncoderArgs(C.Structure):
    _fields_ = [
        ('p', C.c_void_p), ('B', C.c_int32), ('T', C.c_int64),
        ('padding', C.c_double), ('div_mode', C.c_int32),
        ('n_keys', C.c_int32), ('kind', C.c_int32 * 4), ('reso', C.c_int32 * 4),
        ('pool_mean', C.c_int32), ('n_blocks', C.c_int32),
        ('weights', C.c_void_p), ('workspace', C.c_void_p), ('workspace_bytes', C.c_int64),
        ('out_cl', C.c_void_p * 4), ('c_out', C.c_void_p), ('index_out', C.c_void_p * 4),
    ]


class EncoderBwdArgs(C.Structure):
    _fields_ = [
        ('p', C.c_void_p), ('B', C.c_int32), ('T', C.c_int64),
        ('padding', C.c_double), ('div_mode', C.c_int32),
        ('n_keys', C.c_int32), ('kind', C.c_int32 * 4), ('reso', C.c_int32 * 4),
        ('pool_mean', C.c_int32), ('n_blocks', C.c_int32),
        ('weights', C.c_void_p), ('workspace', C.c_void_p), ('workspace_bytes', C.c_int64),
        ('d_out_cl', C.c_void_p * 4), ('d_params', C.c_void_p),
    ]


class McArgs(C.Structure):
    _fields_ = [
        ('grid', C.c_void_p), ('nx', C.c_int32), ('ny', C.c_int32), ('nz', C.c_int32),
        ('level', C.c_float), ('level_keys', C.c_void_p), ('n_level_keys', C.c_int32),
        ('scratch', C.c_void_p), ('scratch_bytes', C.c_int64),
        ('vertices', C.c_void_p), ('vertex_capacity', C.c_int64),
        ('faces', C.c_void_p), ('face_capacity', C.c_int64),
        ('counts', C.c_void_p),
        ('voffset', C.c_float), ('vscale', C.c_float), ('phase', C.c_int32),
        ('x_emit', C.c_int32), ('x_origin', C.c_int32), ('level_ptr', C.c_void_p),
        ('halo_grid', C.c_void_p), ('halo_rows', C.c_int32),
    ]


class Exchange(C.Structure):
    _fields_ = [('ctrl', C.c_void_p * 8), ('world', C.c_int32), ('rank', C.c_int32)]


class MeshPiece(C.Structure):
    _fields_ = [('counts', C.c_void_p), ('vertices', C.c_void_p), ('faces', C.c_void_p),
                ('dst_vertices', C.c_void_p * 8), ('dst_faces', C.c_void_p * 8),
                ('vertex_capacity', C.c_int64), ('face_capacity', C.c_int64), ('total_counts', C.c_void_p)]


EXCHANGE_CTRL_BYTES, EXCHANGE_ERR_OFFSET, EXCHANGE_LEVEL_OFFSET, EXCHANGE_BASE_OFFSET = 1024, 556, 560, 568


class Conv3dArgs(C.Structure):
    _fields_ = [('x', C.c_void_p), ('x2', C.c_void_p),
                ('N', C.c_int32), ('D', C.c_int32), ('H', C.c_int32), ('W', C.c_int32), ('C1', C.c_int32),
                ('C2', C.c_int32), ('D2', C.c_int32), ('H2', C.c_int32), ('W2', C.c_int32),
                ('w_packed', C.c_void_p), ('bias', C.c_void_p), ('Cout', C.c_int32), ('ksize', C.c_int32),
                ('in_stats', C.c_void_p), ('gamma', C.c_void_p), ('beta', C.c_void_p), ('groups', C.c_int32),
                ('eps', C.c_double), ('relu', C.c_int32), ('y', C.c_void_p), ('out_stats', C.c_void_p),
                ('ksize_z', C.c_int32)]


class PackDesc(C.Structure):
    _fields_ = [('src', C.c_void_p), ('out_dim', C.c_int32), ('in_dim', C.c_int32), ('src_stride', C.c_int32),
                ('src_col0', C.c_int32), ('dst_off', C.c_int32)]


PACK_MAX_DESCS = 64


# tcgen05 operand buffer `weights_tc` (VTACO_DEC_TC_* of include/vtaco_b200.h): pack modes, sizes and offsets
DEC_TC_MODE_3XTF32, DEC_TC_MODE_BF16, DEC_TC_MODE_TILE4 = 0, 1, 2
DEC_TC_KBLK_FLOATS, DEC_TC_BVEC_FLOATS = 256, 32
DEC_TC_SUB_HI, DEC_TC_SUB_LO, DEC_TC_SUB_BF16 = 0, 1024, 2048


def dec_tc_mode(variant):
    return 2 if variant == 7 else 1 if variant in (4, 6) else 0


def dec_tc_mat_floats(mode):
    return 2560 if mode == 2 else 2048


def dec_tc_mat(mode, m):
    return m * dec_tc_mat_floats(mode)


def dec_tc_bias_step_floats(mode):
    return DEC_TC_BVEC_FLOATS if mode == 2 else DEC_TC_KBLK_FLOATS


def dec_tc_bias(mode, n_blocks, s):
    return dec_tc_mat(mode, 3 * n_blocks + int(mode == 2)) + s * dec_tc_bias_step_floats(mode)


def dec_tc_wimg(mode, n_blocks):
    return dec_tc_mat(mode, 3 * n_blocks) if mode == 2 else dec_tc_bias(mode, n_blocks, 2 * n_blocks + 1)


def dec_tc_input(n_blocks, q):
    return dec_tc_bias(2, n_blocks, 2 * n_blocks + 1) + q * DEC_TC_KBLK_FLOATS


def dec_tc_used_floats(mode, n_blocks):
    return dec_tc_input(n_blocks, 4) if mode == 2 else dec_tc_wimg(mode, n_blocks) + dec_tc_mat_floats(mode)


def dec_tc_floats(n_blocks):
    """VTACO_DEC_TC_FLOATS: floats reserved for `weights_tc` in any pack mode."""
    return (3 * n_blocks + 1) * dec_tc_mat_floats(2) + (2 * n_blocks + 1 + 4) * DEC_TC_KBLK_FLOATS


def pack_linear(entries, dst, cache=None):
    """One launch of vtaco_pack_linear.  entries: (tensor, dst_off[, col0, n_cols]) — an nn.Linear
    weight (out,in) / bias (out,) goes K-major to dst[dst_off + k*out + n].
    `cache` (a dict owned by the module): the descriptor table is rebuilt only when a parameter's storage
    moved — training re-packs after every optimizer step and building 40 ctypes descriptors was ~0.15 ms."""
    key = None
    if cache is not None:
        key = tuple(e[0].data_ptr() for e in entries)
        hit = cache.get('descs')
        if hit is not None and hit[0] == key:
            with torch.cuda.device(dst.device):
                st = lib().vtaco_pack_linear(hit[1], len(entries), ptr(dst), dst.numel(), stream_ptr(dst.device))
            check(st, 'pack_linear')
            return
    descs = (PackDesc * len(entries))()
    keep = []
    for d, e in zip(descs, entries):
        t, off = e[0], e[1]
        col0 = e[2] if len(e) > 2 else 0
        t = t.detach()
        if t.dtype != torch.float32 or not t.is_cuda:
            raise TypeError('vtaco_b200: parameters must be float32 CUDA tensors')
        if t.dim() == 1:
            t = t.contiguous()
            d.out_dim, d.in_dim, d.src_stride = t.shape[0], 1, 1
        else:
            if t.stride(1) != 1:
                t = t.contiguous()
            d.out_dim, d.src_stride = t.shape[0], t.stride(0)
            d.in_dim = (e[3] if len(e) > 3 else t.shape[1] - col0)
        keep.append(t)
        d.src, d.src_col0, d.dst_off = t.data_ptr(), col0, off
    with torch.cuda.device(dst.device):
        st = lib().vtaco_pack_linear(descs, len(entries), ptr(dst), dst.numel(), stream_ptr(dst.device))
    check(st, 'pack_linear')
    # cacheable only if no temporary copy was made (a descriptor must not outlive the tensor it points into)
    if cache is not None and all(k.data_ptr() == e[0].data_ptr() for k, e in zip(keep, entries)):
        cache['descs'] = (key, descs)


def layout_entries(layout, params, n_blocks):
    """pack_linear entries of every field of a packed parameter buffer, in layout order.
    layout = (offset of the blocks, block stride, head, block, tail): head entries (parameter name, offset[, first
    column, columns]), block entries (name with %d for the block index, offset inside the block) for each of the
    n_blocks blocks, tail entries (name, offset from the end of the blocks).  params: name -> parameter."""
    off, stride, head, block, tail = layout
    end = off + n_blocks * stride
    return ([(params[e[0]],) + e[1:] for e in head] +
            [(params[name % i], off + i * stride + o) for i in range(n_blocks) for name, o in block] +
            [(params[name], end + o) for name, o in tail])


def layout_grads(layout, params, flat, n_blocks):
    """name -> gradient of every parameter of `layout` (see layout_entries) from `flat`, a buffer in that layout with
    every matrix in nn.Linear's [out][in] orientation: views of `flat`, except for a weight packed as column ranges,
    whose gradient is their concatenation."""
    off, stride, head, block, tail = layout
    base, end = flat.storage_offset(), off + n_blocks * stride
    g, ranges = {}, {}
    for name, o, *cols in list(head) + [(name, end + o) for name, o in tail]:
        shape = tuple(params[name].shape)
        if cols:    # columns [first, first + count) of an [out][in] weight, stored as [out][count]
            ranges.setdefault(name, []).append(flat.as_strided((shape[0], cols[1]), (cols[1], 1), base + o))
        else:       # [out][in] or [out], contiguous
            g[name] = flat.as_strided(shape, shape[1:] + (1,), base + o)
    for name, parts in ranges.items():
        g[name] = torch.cat(parts, 1)
    # a block field is the same view every `stride` floats: one strided view and one unbind per field
    for name, o in block if n_blocks else ():
        shape = tuple(params[name % 0].shape)
        fields = flat.as_strided((n_blocks,) + shape, (stride,) + shape[1:] + (1,), base + off + o).unbind(0)
        for i, t in enumerate(fields):
            g[name % i] = t
    return g


_lib = None


def lib():
    """Load the shared library (once).  Fails loudly when it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(os.environ.get('VTACO_B200_LIB', LIB_PATH)):
        raise RuntimeError(
            'vtaco_b200: %s not found. Build it with `python -m vtaco_b200.build` '
            '(nvcc, sm_100a). There is no CPU / PyTorch fallback.' % LIB_PATH)
    L = C.CDLL(os.environ.get('VTACO_B200_LIB', LIB_PATH))   # (override: A/B runs of two builds in one process tree)
    L.vtaco_abi_version.restype = C.c_int
    L.vtaco_status_string.restype = C.c_char_p
    L.vtaco_status_string.argtypes = [C.c_int]
    L.vtaco_last_cuda_error.restype = C.c_char_p
    L.vtaco_point_to_cell.argtypes = [C.c_void_p, C.c_int64, C.c_double, C.c_int, C.c_int, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.vtaco_relayout_cl.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p]
    L.vtaco_relayout_cf.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int64, C.c_void_p]
    L.vtaco_decoder_forward.argtypes = [C.POINTER(DecoderArgs), C.c_void_p]
    L.vtaco_sample_features.argtypes = [C.POINTER(DecoderArgs), C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.vtaco_decoder_backward.argtypes = [C.POINTER(DecoderBwdArgs), C.c_void_p]
    L.vtaco_decoder_backward_workspace_bytes.restype = C.c_size_t
    L.vtaco_decoder_backward_workspace_bytes.argtypes = [C.c_int64, C.c_int32]
    L.vtaco_key_to_float_host.restype = C.c_float
    L.vtaco_key_to_float_host.argtypes = [C.c_int32]
    L.vtaco_fp32_peak.argtypes = [C.c_int, C.c_int, C.POINTER(C.c_double), C.c_void_p]
    L.vtaco_pack_linear.argtypes = [C.POINTER(PackDesc), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p]
    L.vtaco_decoder_tc_floats.restype = C.c_int64
    L.vtaco_decoder_tc_floats.argtypes = [C.c_int32]
    L.vtaco_decoder_pack_tc.argtypes = [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p]
    L.vtaco_encoder_workspace_bytes.restype = C.c_int64
    L.vtaco_encoder_workspace_bytes.argtypes = [C.c_int32, C.c_int64, C.c_int32, C.POINTER(C.c_int32),
                                                C.POINTER(C.c_int32)]
    L.vtaco_encoder_pointnet.argtypes = [C.POINTER(EncoderArgs), C.c_void_p]
    L.vtaco_encoder_backward_workspace_bytes.restype = C.c_int64
    L.vtaco_encoder_backward_workspace_bytes.argtypes = [C.c_int32, C.c_int64, C.c_int32, C.POINTER(C.c_int32),
                                                         C.POINTER(C.c_int32), C.c_int32]
    L.vtaco_encoder_backward.argtypes = [C.POINTER(EncoderBwdArgs), C.c_void_p]
    L.vtaco_pool_workspace_bytes.restype = C.c_int64
    L.vtaco_pool_workspace_bytes.argtypes = [C.c_int32, C.c_int64, C.c_int32, C.POINTER(C.c_int64)]
    L.vtaco_pool_local.argtypes = [C.c_void_p, C.c_int32, C.c_int64, C.c_int32, C.POINTER(C.c_void_p),
                                   C.POINTER(C.c_int64), C.c_int32, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]
    L.vtaco_scatter_mean.argtypes = [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_int64,
                                     C.c_void_p, C.c_void_p]
    for name, argtypes in _OPTIONAL.items():
        getattr(L, name).argtypes = argtypes
    L.vtaco_mc_scratch_bytes.restype = C.c_int64
    if L.vtaco_abi_version() != 1:
        raise RuntimeError('vtaco_b200: ABI version mismatch')
    _lib = L
    return L


_OPTIONAL = {
    'vtaco_marching_cubes': [C.POINTER(McArgs), C.c_void_p],
    'vtaco_mc_scratch_bytes': [C.c_int32, C.c_int32, C.c_int32],
    'vtaco_grid_minmax': [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p],
    'vtaco_publish_keys': [C.c_void_p, C.POINTER(C.c_void_p), C.c_int32, C.c_int32, C.c_void_p],
    'vtaco_conv3d_cl': [C.POINTER(Conv3dArgs), C.c_void_p],
    'vtaco_maxpool2_cl': [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                          C.c_void_p],
    'vtaco_channel_stats_cl': [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_void_p],
    'vtaco_maxpool2d_cl': [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p],
    'vtaco_depth_to_space2_cl': [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_void_p],
    'vtaco_fingertip_ids': [C.c_void_p, C.c_int64, C.POINTER(C.c_double), C.POINTER(C.c_int32), C.c_int32, C.c_double,
                            C.c_void_p, C.c_void_p],
    'vtaco_tactile_point_map': [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_double,
                                C.c_int32, C.c_void_p, C.c_void_p],
    'vtaco_exchange_level': [C.POINTER(Exchange), C.c_void_p, C.c_void_p],
    'vtaco_exchange_mesh': [C.POINTER(Exchange), C.POINTER(MeshPiece), C.c_void_p],
    'vtaco_group_norm_cl': [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                            C.c_double, C.c_void_p, C.c_void_p],
    'vtaco_group_norm': [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int64,
                         C.c_double, C.c_void_p, C.c_void_p],
    'vtaco_upsample_concat3d': [C.c_void_p] * 3 + [C.c_int32] * 9 + [C.c_void_p],
    'vtaco_chamfer': [C.c_void_p, C.c_void_p, C.c_int32, C.c_int64, C.c_int64] + [C.c_void_p] * 7,
}


def check(status, what):
    if status != 0:
        L = lib()
        msg = L.vtaco_status_string(status).decode()
        if status == -3:
            msg += ': ' + L.vtaco_last_cuda_error().decode()
        raise RuntimeError('vtaco_b200.%s failed: %s' % (what, msg))


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def ptr(t):
    return C.c_void_p(t.data_ptr()) if t is not None else C.c_void_p(0)


def require_cuda(t, name):
    if not t.is_cuda:
        raise RuntimeError('vtaco_b200: %s must be a CUDA tensor (CUDA-only build, no CPU fallback)' % name)
    if t.dtype != torch.float32:
        raise TypeError('vtaco_b200: %s must be float32, got %s' % (name, t.dtype))


def wants_grad(*tensors):
    return torch.is_grad_enabled() and any(torch.is_tensor(t) and t.requires_grad for t in tensors)


def forbid_autograd(*tensors):
    """For the entry points that have no backward kernel (SURVEY §8f-2 covers the decoder)."""
    if wants_grad(*tensors):
        raise NotImplementedError(
            'vtaco_b200: this kernel is forward-only: call it under torch.no_grad() '
            '(backward kernels exist for LocalDecoder.forward / forward_img / forward_contact)')
