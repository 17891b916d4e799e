"""TEST INFRASTRUCTURE ONLY — CPU restatement (torch CPU ops, fp32) of the
reference's encoder / decoder / dense-evaluation arithmetic; decoder_forward also
runs in float64 (dtype=torch.float64), the high-precision reference of the kernel tests.

Every function cites the reference lines it follows (paths relative to the
jeffsonyu/VTacO tree).  Weights are passed as a plain ``dict`` keyed exactly
like the reference modules' ``state_dict()`` so the same dict can be loaded
into the reference (tests/golden/make_golden.py) and into the CUDA modules.

PINNED: tests/test_oracle_golden.py replays tests/golden/*.npz, which were
produced by the reference's own modules (see tests/golden/make_golden.py).

Third-party arithmetic that is NOT under the reference tree and is restated
here from published semantics:
  * torch_scatter==2.0.9 (requirements.txt:30) scatter_mean / scatter_max —
    call sites src/encoder/pointnet.py:93,108,124-128.
  * torch F.grid_sample / F.linear are used as they are (torch is present).
"""
import numpy as np
import torch
import torch.nn.functional as F

PLANE_AXES = {'xz': (0, 2), 'xy': (0, 1), 'yz': (1, 2)}


# --------------------------------------------------------------------------- #
# src/common.py
# --------------------------------------------------------------------------- #
def _divide(x, d, cuda_division):
    """`tensor / python_scalar`.

    CPU ATen performs an IEEE fp32 division by fp32(d); CUDA ATen
    (div_true_kernel_cuda) multiplies by fp32(1/d).  The two differ in the
    last bit for ~half of the inputs (SURVEY.md §7.2-1).
    """
    if not cuda_division:
        return x / d
    inv = np.float32(1.0 / d)  # reciprocal formed in double, then rounded (measured, see common.cuh)
    return x * float(inv)  # fp32 tensor * python scalar -> fp32 multiply by fp32(inv)


def normalize_coordinate(p, padding=0.1, plane='xz', cuda_division=False):
    """src/common.py:268-291."""
    a, b = PLANE_AXES[plane] if plane in PLANE_AXES else (1, 2)
    xy = p[:, :, [a, b]]
    xy_new = _divide(xy, (1 + padding + 10e-6), cuda_division)
    xy_new = xy_new + 0.5
    # `if xy_new.max() >= 1: xy_new[xy_new >= 1] = 1 - 10e-6` is a per-element
    # clamp (NaNs pass through both masks).
    hi = torch.tensor(1 - 10e-6, dtype=xy_new.dtype)
    xy_new = torch.where(xy_new >= 1, hi, xy_new)
    xy_new = torch.where(xy_new < 0, torch.zeros((), dtype=xy_new.dtype), xy_new)
    return xy_new


def normalize_3d_coordinate(p, padding=0.1, cuda_division=False):
    """src/common.py:293-309."""
    p_nor = _divide(p, (1 + padding + 10e-4), cuda_division)
    p_nor = p_nor + 0.5
    hi = torch.tensor(1 - 10e-4, dtype=p_nor.dtype)
    p_nor = torch.where(p_nor >= 1, hi, p_nor)
    p_nor = torch.where(p_nor < 0, torch.zeros((), dtype=p_nor.dtype), p_nor)
    return p_nor


def coordinate2index(x, reso, coord_type='2d'):
    """src/common.py:333-348."""
    x = (x * reso).long()
    if coord_type == '2d':
        index = x[:, :, 0] + reso * x[:, :, 1]
    else:
        index = x[:, :, 0] + reso * (x[:, :, 1] + reso * x[:, :, 2])
    return index[:, None, :]


def make_3d_grid(bb_min, bb_max, shape):
    """src/common.py:178-197 — x slowest, z fastest."""
    size = shape[0] * shape[1] * shape[2]
    pxs = torch.linspace(bb_min[0], bb_max[0], shape[0])
    pys = torch.linspace(bb_min[1], bb_max[1], shape[1])
    pzs = torch.linspace(bb_min[2], bb_max[2], shape[2])
    pxs = pxs.view(-1, 1, 1).expand(*shape).contiguous().view(size)
    pys = pys.view(1, -1, 1).expand(*shape).contiguous().view(size)
    pzs = pzs.view(1, 1, -1).expand(*shape).contiguous().view(size)
    return torch.stack([pxs, pys, pzs], dim=1)


# --------------------------------------------------------------------------- #
# torch_scatter 2.0.9 (published semantics; un-vendored dependency)
# --------------------------------------------------------------------------- #
def scatter_mean(src, index, dim_size=None, out=None):
    """torch_scatter.scatter_mean(src, index, dim=-1, out=..., dim_size=...):
    scatter_add of src, scatter_add of ones, count.clamp_(min=1), true_divide_.
    `index` (B,1,T) broadcasts over the channel dim of `src` (B,C,T)."""
    idx = index.expand_as(src)
    if out is None:
        out = src.new_zeros(src.shape[0], src.shape[1], dim_size)
    out.scatter_add_(2, idx, src)
    count = src.new_zeros(index.shape[0], index.shape[1], out.shape[2])
    count.scatter_add_(2, index, torch.ones_like(index, dtype=src.dtype))
    count.clamp_(min=1)
    out.true_divide_(count)
    return out


def scatter_max(src, index, dim_size):
    """torch_scatter.scatter_max(...)[0]: per-cell maximum, 0 for cells that
    received no element (the arg output is never used by the reference,
    src/encoder/pointnet.py:127-128)."""
    idx = index.expand_as(src)
    out = src.new_zeros(src.shape[0], src.shape[1], dim_size)
    out.scatter_reduce_(2, idx, src, 'amax', include_self=False)
    return out


# --------------------------------------------------------------------------- #
# src/layers.py
# --------------------------------------------------------------------------- #
def resnet_block_fc(x, W, prefix):
    """src/layers.py:41-50 — x_s + fc_1(relu(fc_0(relu(x))))."""
    net = F.linear(F.relu(x), W[prefix + 'fc_0.weight'], W[prefix + 'fc_0.bias'])
    dx = F.linear(F.relu(net), W[prefix + 'fc_1.weight'], W[prefix + 'fc_1.bias'])
    if (prefix + 'shortcut.weight') in W:
        x_s = F.linear(x, W[prefix + 'shortcut.weight'])
    else:
        x_s = x
    return x_s + dx


# --------------------------------------------------------------------------- #
# src/encoder/pointnet.py (LocalPoolPointnet, PointNet part; UNets are torch.nn)
# --------------------------------------------------------------------------- #
def _plane_list(plane_type):
    # membership is tested with `in` on a str or a list (pointnet.py:141-150)
    return [k for k in ('xz', 'xy', 'yz', 'grid') if k in plane_type]


def encoder_indices(p, plane_type, reso_plane, reso_grid, padding=0.1, cuda_division=False):
    """src/encoder/pointnet.py:139-152."""
    coord, index = {}, {}
    for key in _plane_list(plane_type):
        if key == 'grid':
            coord[key] = normalize_3d_coordinate(p.clone(), padding, cuda_division)
            index[key] = coordinate2index(coord[key], reso_grid, '3d')
        else:
            coord[key] = normalize_coordinate(p.clone(), padding, key, cuda_division)
            index[key] = coordinate2index(coord[key], reso_plane)
    return coord, index


def pool_local(index, net, reso_plane, reso_grid, scatter_type='max'):
    """src/encoder/pointnet.py:116-132."""
    c_out = 0
    for key in index:
        dim_size = reso_grid ** 3 if key == 'grid' else reso_plane ** 2
        src = net.permute(0, 2, 1)
        if scatter_type == 'max':
            fea = scatter_max(src, index[key], dim_size)
        else:
            fea = scatter_mean(src, index[key], dim_size)
        fea = fea.gather(dim=2, index=index[key].expand(-1, net.size(2), -1))
        c_out = c_out + fea
    return c_out.permute(0, 2, 1)


def encoder_pointnet(p, W, plane_type, reso_plane=None, reso_grid=None, padding=0.1,
                     n_blocks=5, scatter_type='max', cuda_division=False,
                     return_intermediates=False):
    """src/encoder/pointnet.py:135-172 without the UNet post-processing:
    returns dict key -> scatter_mean features, keys in the order grid,xz,xy,yz."""
    coord, index = encoder_indices(p, plane_type, reso_plane, reso_grid, padding, cuda_division)
    inter = {}
    net = F.linear(p, W['fc_pos.weight'], W['fc_pos.bias'])
    net = resnet_block_fc(net, W, 'blocks.0.')
    inter['net0'] = net
    for i in range(1, n_blocks):
        pooled = pool_local(index, net, reso_plane, reso_grid, scatter_type)
        inter['pooled%d' % i] = pooled
        net = torch.cat([net, pooled], dim=2)
        net = resnet_block_fc(net, W, 'blocks.%d.' % i)
        inter['net%d' % i] = net
    c = F.linear(net, W['fc_c.weight'], W['fc_c.bias'])
    inter['c'] = c
    c_dim = c.shape[2]
    fea = {}
    order = [k for k in ('grid', 'xz', 'xy', 'yz') if k in plane_type]
    for key in order:
        if key == 'grid':  # generate_grid_features, pointnet.py:102-114
            out = c.new_zeros(p.size(0), c_dim, reso_grid ** 3)
            out = scatter_mean(c.permute(0, 2, 1), index[key], out=out)
            fea[key] = out.reshape(p.size(0), c_dim, reso_grid, reso_grid, reso_grid)
        else:  # generate_plane_features, pointnet.py:85-100
            out = c.new_zeros(p.size(0), c_dim, reso_plane ** 2)
            out = scatter_mean(c.permute(0, 2, 1), index[key], out=out)
            fea[key] = out.reshape(p.size(0), c_dim, reso_plane, reso_plane)
    if return_intermediates:
        return fea, index, inter
    return fea


# --------------------------------------------------------------------------- #
# src/conv_onet/models/decoder.py (LocalDecoder)
# --------------------------------------------------------------------------- #
def _grid_sample(c, vgrid, sample_mode, dtype):
    """F.grid_sample of the reference's call sites; with dtype != fp32 the interpolation runs in `dtype` on
    the fp32 grid coordinates (the coordinates themselves stay what the fp32 reference computes)."""
    if dtype != torch.float32:
        c, vgrid = c.to(dtype), vgrid.to(dtype)
    return F.grid_sample(c, vgrid, padding_mode='border', align_corners=True, mode=sample_mode)


def sample_plane_feature(p, c, plane, padding=0.1, sample_mode='bilinear', cuda_division=False,
                         dtype=torch.float32):
    """src/conv_onet/models/decoder.py:55-60."""
    xy = normalize_coordinate(p.clone(), padding, plane, cuda_division)
    xy = xy[:, :, None].float()
    vgrid = 2.0 * xy - 1.0
    return _grid_sample(c, vgrid, sample_mode, dtype).squeeze(-1)


def sample_grid_feature(p, c, padding=0.1, sample_mode='bilinear', cuda_division=False, dtype=torch.float32):
    """src/conv_onet/models/decoder.py:62-68."""
    p_nor = normalize_3d_coordinate(p.clone(), padding, cuda_division)
    p_nor = p_nor[:, :, None, None].float()
    vgrid = 2.0 * p_nor - 1.0
    return _grid_sample(c, vgrid, sample_mode, dtype).squeeze(-1).squeeze(-1)


def sample_features(p, c_plane, padding=0.1, sample_mode='bilinear', cuda_division=False, dtype=torch.float32):
    """Sum over present keys in the order grid,xz,xy,yz (decoder.py:72-83)."""
    c = 0
    keys = list(c_plane.keys())
    if 'grid' in keys:
        c = c + sample_grid_feature(p, c_plane['grid'], padding, sample_mode, cuda_division, dtype)
    for k in ('xz', 'xy', 'yz'):
        if k in keys:
            c = c + sample_plane_feature(p, c_plane[k], k, padding, sample_mode, cuda_division, dtype)
    return c.transpose(1, 2)


def decoder_forward(p, c_plane, W, mode='forward', c_img=None, n_blocks=5, leaky=False,
                    sample_mode='bilinear', padding=0.1, c_dim=32, cuda_division=False,
                    dtype=torch.float32, return_preacts=False):
    """LocalDecoder.forward (decoder.py:135-161), .forward_img (:71-103),
    .forward_contact (:105-133) selected by `mode` in {forward, img, contact}.

    dtype=torch.float64: the query normalisation, clamp and grid coordinates are computed in fp32 exactly as
    the reference does (they decide which cells are read); interpolation, feature sums, every layer and the
    heads run in float64 on float64 copies of the features, weights, points and c_img.  This is the
    high-precision reference the fp32 kernels are measured against.
    return_preacts: also return {'m': [m_i], 'h': [h_i], 'n_last': n} — the inputs of every ReLU (m_i = block
    input after fc_c, h_i = fc_0 output) and of the head activation, to locate queries near a kink."""
    if c_dim != 0:
        c = sample_features(p, c_plane, padding, sample_mode, cuda_division, dtype)
    if dtype == torch.float32:
        p = p.float()
        lin = F.linear
    else:
        p = p.to(dtype)
        if c_img is not None:
            c_img = c_img.to(dtype)
        lin = lambda x, w, b=None: F.linear(x, w.to(dtype), None if b is None else b.to(dtype))  # noqa: E731
    if mode == 'img':
        net = lin(torch.cat((p, c_img), 2), W['fc_p_img.weight'], W['fc_p_img.bias'])
    else:
        net = lin(p, W['fc_p.weight'], W['fc_p.bias'])
    pre = {'m': [], 'h': []}
    for i in range(n_blocks):
        if c_dim != 0:
            net = net + lin(c, W['fc_c.%d.weight' % i], W['fc_c.%d.bias' % i])
        if return_preacts or dtype != torch.float32:
            # resnet_block_fc, spelled out (src/layers.py:41-50, identity shortcut)
            pfx = 'blocks.%d.' % i
            h = lin(F.relu(net), W[pfx + 'fc_0.weight'], W[pfx + 'fc_0.bias'])
            pre['m'].append(net)
            pre['h'].append(h)
            net = net + lin(F.relu(h), W[pfx + 'fc_1.weight'], W[pfx + 'fc_1.bias'])
        else:
            net = resnet_block_fc(net, W, 'blocks.%d.' % i)
    pre['n_last'] = net
    act = (lambda x: F.leaky_relu(x, 0.2)) if leaky else F.relu
    out = lin(act(net), W['fc_out.weight'], W['fc_out.bias']).squeeze(-1)
    if mode == 'contact':
        oc = lin(act(net), W['fc_out_contact.weight'], W['fc_out_contact.bias']).squeeze(-1)
        out = (out, oc)
    return (out, pre) if return_preacts else out


# --------------------------------------------------------------------------- #
# src/conv_onet/generation.py
# --------------------------------------------------------------------------- #
def dense_grid_points(nx, padding=0.1):
    """generation.py:119-120,155-157: (1+padding) * make_3d_grid((-.5,)*3,(.5,)*3,(nx,)*3)."""
    return (1 + padding) * make_3d_grid((-0.5,) * 3, (0.5,) * 3, (nx,) * 3)


def eval_points(p, c_plane, W, c_img_all=None, points_batch_size=100000, **dec_kw):
    """Generator3D.eval_points, generation.py:338-383 (non-crop branch):
    split into chunks, decode[_img] each, concatenate on the host."""
    p_split = torch.split(p, points_batch_size)
    if c_img_all is not None:
        c_img = torch.split(c_img_all.squeeze(0) if c_img_all.dim() == 3 else c_img_all,
                            points_batch_size)
    occ = []
    with torch.no_grad():
        for idx, pi in enumerate(p_split):
            pi = pi.unsqueeze(0)
            if c_img_all is not None:
                o = decoder_forward(pi, c_plane, W, mode='img', c_img=c_img[idx].unsqueeze(0), **dec_kw)
            else:
                o = decoder_forward(pi, c_plane, W, mode='forward', **dec_kw)
            occ.append(o.squeeze(0))
    return torch.cat(occ, dim=0)


def fingertip_c_img(p, tips, tip_feat, touch, radius=0.05):
    """generation.py:190-200: rows of c_img_all within `radius` of the NEAREST
    fingertip (float64 cdist) take that fingertip's feature if it touched."""
    pn = p.detach().cpu().numpy().astype(np.float64)
    tp = np.asarray(tips, dtype=np.float64)
    d = np.sqrt(((pn[:, None, :] - tp[None, :, :]) ** 2).sum(-1))
    dmin, amin = d.min(1), d.argmin(1)
    out = torch.zeros(p.shape[0], tip_feat.shape[1], dtype=torch.float32)
    for f in range(tp.shape[0]):
        if touch[f]:
            sel = np.where((dmin < radius) & (amin == f))[0]
            out[sel] = tip_feat[f]
    return out


# --------------------------------------------------------------------------- #
# src/common.py:54-137 — Chamfer distance (the metric after mesh extraction)
# --------------------------------------------------------------------------- #
def chamfer_distance_naive(points1, points2):
    """src/common.py:69-91."""
    if points2.size()[1] < 2048:
        points1 = points1[:, :points2.size()[1], :]
    assert points1.size() == points2.size()
    B, T, _ = points1.size()
    d = (points1.view(B, T, 1, 3) - points2.view(B, 1, T, 3)).pow(2).sum(-1)
    return d.min(dim=1)[0].mean(dim=1) + d.min(dim=2)[0].mean(dim=1)


def chamfer_distance_kdtree(points1, points2, give_id=False):
    """src/common.py:94-137 with the kd-tree query (pykdtree, un-vendored) restated as an exact
    nearest-neighbour search in float64."""
    d = torch.cdist(points1.double(), points2.double())
    i12, i21 = d.argmin(2), d.argmin(1)
    p12 = torch.gather(points2, 1, i12[:, :, None].expand_as(points1))
    p21 = torch.gather(points1, 1, i21[:, :, None].expand_as(points2))
    c1 = (points1 - p12).pow(2).sum(2).mean(1)
    c2 = (points2 - p21).pow(2).sum(2).mean(1)
    if give_id:
        return c1, c2, i12, i21
    return c1 + c2


def tactile_points_c_img(p, points_per_sensor, sensor_feat, touch, radius=0.015):
    """generation.py:222-255 (encode_t2d branch), the part after the depth back-projection:
    for t in 0..4, if the sensor touched, every query within `radius` (float64 cdist) of ANY of
    sensor t's world points takes c_img[t]; later sensors overwrite.  (The reference walks the
    lattice in 8 hard-coded chunks of 64**3 — only valid for nx = 128; the chunking does not
    change the result and is not restated.)"""
    pn = p.detach().cpu().numpy().astype(np.float64)
    out = torch.zeros(p.shape[0], sensor_feat.shape[1], dtype=torch.float32)
    for t, pts in enumerate(points_per_sensor):
        if pts is None or not touch[t]:
            continue
        q = np.asarray(pts, dtype=np.float64).reshape(-1, 3)
        if q.shape[0] == 0:
            continue
        hit = np.zeros(pn.shape[0], dtype=bool)
        for s in range(0, pn.shape[0], 65536):
            d = np.sqrt(((q[:, None, :] - pn[None, s:s + 65536, :]) ** 2).sum(-1))
            hit[s:s + 65536] = (d < radius).any(0)
        out[np.where(hit)[0]] = sensor_feat[t]
    return out


def earth_mover_distance(points1, points2):
    """src/common.py:45-51 (scipy is the reference's own dependency: requirements.txt)."""
    from scipy.optimize import linear_sum_assignment
    from scipy.spatial import distance
    d = distance.cdist(points1, points2)
    assignment = linear_sum_assignment(d)
    return d[assignment].sum() / len(d)
