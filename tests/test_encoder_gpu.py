"""GPU parity of the LocalPoolPointnet kernels (through the C ABI).
 * cell indices: bit-exact; local max-pooling op: bit-exact;
 * per-point code / scatter_mean features: |a-b| <= 1e-4*max(1,|b|) (fp32 atomics order)."""
import numpy as np
import pytest
import torch

from util import load, weights, close, rs_randn, synthetic_cloud

pytestmark = pytest.mark.gpu
TOL = 1e-4

ENC_CTOR = {'grid': dict(plane_type='grid', grid_resolution=32),
            'tri': dict(plane_type=['xz', 'xy', 'yz'], plane_resolution=32),
            'all_mean': dict(plane_type=['xz', 'xy', 'yz', 'grid'], plane_resolution=16, grid_resolution=16,
                             scatter_type='mean')}
ENC_ORACLE = {'grid': dict(plane_type='grid', reso_grid=32),
              'tri': dict(plane_type=['xz', 'xy', 'yz'], reso_plane=32),
              'all_mean': dict(plane_type=['xz', 'xy', 'yz', 'grid'], reso_plane=16, reso_grid=16,
                               scatter_type='mean')}


def make_encoder(W, division='true', **kw):
    from vtaco_b200.encoder import encoder_dict
    enc = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, **kw)
    enc.load_state_dict(W, strict=True)
    enc = enc.cuda().eval()
    enc.division = division
    return enc


@pytest.mark.parametrize('tag', ['grid', 'tri', 'all_mean'])
def test_encoder_golden(tag):
    g = load('encoder_%s.npz' % tag)
    enc = make_encoder(weights(g), **ENC_CTOR[tag])
    with torch.no_grad():
        fea = enc(torch.from_numpy(g['p']).cuda())
    assert list(fea.keys()) == [str(k) for k in g['key_order']]
    for k, v in fea.items():
        assert tuple(v.shape) == tuple(g['fea_%s_shape' % k])
        flat = v.contiguous().cpu().numpy().reshape(v.shape[0], v.shape[1], -1)
        occ = np.abs(flat).sum(1) != 0
        b_idx, cell = np.nonzero(occ)
        assert np.array_equal(b_idx, g['fea_%s_b' % k]) and np.array_equal(cell, g['fea_%s_cell' % k]), k
        assert close(flat[b_idx, :, cell], g['fea_%s_val' % k]) < TOL, k


@pytest.mark.parametrize('tag,B,T', [('grid', 4, 3640), ('tri', 3, 3640), ('all_mean', 2, 1000),
                                     ('grid', 1, 1), ('tri', 1, 33), ('grid', 2, 129)])
def test_encoder_vs_oracle(tag, B, T):
    from oracle import convonet as oc
    g = load('encoder_%s.npz' % tag)
    W = weights(g)
    enc = make_encoder(W, **ENC_CTOR[tag])
    if T >= 640:
        p = np.stack([synthetic_cloud(100 + b, T - 640)[0] for b in range(B)])
    else:
        p = np.random.RandomState(7).uniform(-0.6, 0.6, size=(B, T, 3)).astype(np.float32)
    p = torch.from_numpy(p)
    with torch.no_grad():
        ref, ref_idx, inter = oc.encoder_pointnet(p, W, return_intermediates=True, **ENC_ORACLE[tag])
        fea, code, idx = enc.pointnet_features(p.cuda(), return_code=True, return_index=True)
    for k in ref_idx:  # bit-exact cell indices
        assert torch.equal(idx[k].cpu().long(), ref_idx[k]), k
    assert close(code.cpu().numpy(), inter['c'].numpy()) < TOL
    for k in ref:
        assert close(fea[k].contiguous().cpu().numpy(), ref[k].numpy()) < TOL, k


def test_all_points_one_cell_and_outliers():
    """collisions: every point in one cell; outliers beyond the padded cube are clamped."""
    from oracle import convonet as oc
    g = load('encoder_grid.npz')
    W = weights(g)
    enc = make_encoder(W, **ENC_CTOR['grid'])
    p = np.zeros((2, 300, 3), dtype=np.float32)
    p[0] = 0.1 + np.random.RandomState(1).uniform(0, 1e-3, size=(300, 3))
    p[1] = np.random.RandomState(2).uniform(-2, 2, size=(300, 3))
    p = torch.from_numpy(p)
    with torch.no_grad():
        ref = oc.encoder_pointnet(p, W, **ENC_ORACLE['grid'])
        fea = enc.pointnet_features(p.cuda())
    assert close(fea['grid'].contiguous().cpu().numpy(), ref['grid'].numpy()) < TOL


ALL_KEYS = ['xz', 'xy', 'yz', 'grid']


@pytest.mark.parametrize('scatter_type,keys', [
    pytest.param('max', ALL_KEYS, id='max'), pytest.param('mean', ALL_KEYS, id='mean'),
    pytest.param('max', ['grid'], id='max-grid'), pytest.param('mean', ['grid'], id='mean-grid'),
    pytest.param('max', ['xz', 'yz'], id='max-xz-yz'), pytest.param('mean', ['xz', 'yz'], id='mean-xz-yz')])
def test_pool_local_op(scatter_type, keys):
    """pool_local (pointnet.py:116-132) on given inputs: max is order independent -> bit-exact.  Fewer than four
    keys leave key slots of the kernels empty."""
    from oracle import convonet as oc
    g = load('encoder_all_mean.npz')
    enc = make_encoder(weights(g), plane_type=ALL_KEYS, plane_resolution=16, grid_resolution=16,
                       scatter_type=scatter_type)
    B, T = 3, 2000
    p = torch.from_numpy(np.stack([synthetic_cloud(200 + b, T - 640)[0] for b in range(B)]))
    net = torch.from_numpy(rs_randn(5, B, T, 32))
    coord, index = oc.encoder_indices(p, keys, 16, 16)
    ref = oc.pool_local(index, net, 16, 16, scatter_type)
    with torch.no_grad():
        got = enc.pool_local(coord, {k: v.cuda() for k, v in index.items()}, net.cuda())
    if scatter_type == 'max':
        # per-key maxima are exact; the sum over the keys is evaluated in the same order
        assert torch.equal(got.cpu(), ref)
    else:
        assert close(got.cpu().numpy(), ref.numpy()) < TOL


def test_generate_features_ops():
    from oracle import convonet as oc
    g = load('encoder_tri.npz')
    enc = make_encoder(weights(g), plane_type=['xz', 'xy', 'yz', 'grid'], plane_resolution=32, grid_resolution=24)
    B, T = 2, 1500
    p = torch.from_numpy(np.stack([synthetic_cloud(300 + b, T - 640)[0] for b in range(B)]))
    c = torch.from_numpy(rs_randn(6, B, T, 32))
    with torch.no_grad():
        for key in ('xz', 'xy', 'yz'):
            idx = oc.coordinate2index(oc.normalize_coordinate(p.clone(), 0.1, key), 32)
            ref = oc.scatter_mean(c.permute(0, 2, 1), idx, dim_size=32 * 32).reshape(B, 32, 32, 32)
            got = enc.generate_plane_features(p.cuda(), c.cuda(), plane=key)
            assert got.shape == ref.shape
            assert close(got.contiguous().cpu().numpy(), ref.numpy()) < TOL
        idx = oc.coordinate2index(oc.normalize_3d_coordinate(p.clone(), 0.1), 24, '3d')
        ref = oc.scatter_mean(c.permute(0, 2, 1), idx, dim_size=24 ** 3).reshape(B, 32, 24, 24, 24)
        got = enc.generate_grid_features(p.cuda(), c.cuda())
        assert close(got.contiguous().cpu().numpy(), ref.numpy()) < TOL


def test_encoder_decoder_end_to_end_with_unet3d():
    """shipped VTacO_YCB shapes (grid-64 + UNet3D, decoder simple_local) against the oracle +
    the same torch UNet3D fed with the oracle's features."""
    from oracle import convonet as oc
    from vtaco_b200.encoder import encoder_dict
    from vtaco_b200.conv_onet.models import decoder_dict, ConvolutionalOccupancyNetwork
    torch.manual_seed(0)
    enc = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, plane_type='grid',
                                              grid_resolution=64, unet3d=True,
                                              unet3d_kwargs=dict(num_levels=4, f_maps=32, in_channels=32,
                                                                 out_channels=32))
    dec = decoder_dict['simple_local'](dim=3, c_dim=32, padding=0.1, with_contact=False, sample_mode='bilinear',
                                       hidden_size=32)
    with torch.no_grad():
        for m in (enc, dec):
            for b in m.blocks:
                b.fc_1.weight.normal_(0, 0.1)
    net = ConvolutionalOccupancyNetwork(dec, enc, device='cuda').eval()
    enc.division = dec.division = 'true'
    enc.unet3d.fused = False      # fp32 torch.nn / cuDNN modules here; the fused TF32 kernels: tests/test_unet3d_gpu.py
    p = torch.from_numpy(synthetic_cloud(9, 3000)[0])[None]
    q = torch.from_numpy(np.random.RandomState(4).uniform(-0.55, 0.55, size=(1, 5000, 3)).astype(np.float32))
    c_img = torch.from_numpy(rs_randn(10, 1, 5000, 32))
    prev = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        with torch.no_grad():
            c = net.encode_inputs(p.cuda())
            assert c['grid'].shape == (1, 32, 64, 64, 64)
            logits = net.decode_img(q.cuda(), c, c_img.cuda()).logits
            We = {k: v.cpu() for k, v in enc.state_dict().items() if not k.startswith('unet')}
            Wd = {k: v.cpu() for k, v in dec.state_dict().items()}
            ref_fea = oc.encoder_pointnet(p, We, plane_type='grid', reso_grid=64)
            ref_c = {'grid': enc.unet3d(ref_fea['grid'].cuda())}
            assert close(c['grid'].contiguous().cpu().numpy(), ref_c['grid'].cpu().numpy()) < 1e-3
            ref_logits = oc.decoder_forward(q, {'grid': c['grid'].contiguous().cpu()}, Wd, 'img', c_img=c_img)
    finally:
        torch.backends.cudnn.allow_tf32 = prev
    assert close(logits.cpu().numpy(), ref_logits.numpy()) < TOL


@pytest.mark.parametrize('shape,groups', [((1, 32, 64, 64, 64), 8), ((2, 64, 16, 16, 16), 8), ((3, 8, 5, 7, 3), 1),
                                          ((1, 256, 8, 8, 8), 8)])
def test_group_norm_kernel(shape, groups):
    """vtaco_group_norm == torch.nn.functional.group_norm (UNet3D 'g' layers)."""
    from vtaco_b200.encoder.unet3d import GroupNorm
    torch.manual_seed(0)
    gn = GroupNorm(groups, shape[1]).cuda()
    with torch.no_grad():
        gn.weight.normal_()
        gn.bias.normal_()
        x = torch.randn(*shape, device='cuda') * 3 + 1.5
        ref = torch.nn.functional.group_norm(x, groups, gn.weight, gn.bias, gn.eps)
        got = gn(x)
        xcl = x.contiguous(memory_format=torch.channels_last_3d)
        gn.prefer_channels_last = True
        got_cl = gn(xcl)                      # channels-last kernel where the shape allows it
    assert close(got.cpu().numpy(), ref.cpu().numpy()) < 1e-5
    assert got_cl.shape == ref.shape and close(got_cl.contiguous().cpu().numpy(), ref.cpu().numpy()) < 1e-5


@pytest.mark.parametrize('shape', [((2, 8, 16, 16, 16), (2, 16, 8, 8, 8)), ((1, 3, 12, 8, 16), (1, 5, 5, 3, 7)),
                                   ((1, 32, 64, 64, 64), (1, 64, 32, 32, 32))])
def test_upsample_concat_bit_exact(shape):
    """fused UNet3D decoder input == cat(skip, F.interpolate(x, size, 'nearest')) bit for bit."""
    import torch.nn.functional as F
    from vtaco_b200.encoder.unet3d import _upsample_concat
    s_shape, x_shape = shape
    skip = torch.from_numpy(rs_randn(1, *s_shape)).cuda()
    x = torch.from_numpy(rs_randn(2, *x_shape)).cuda()
    ref = torch.cat((skip, F.interpolate(x, size=skip.shape[2:], mode='nearest')), dim=1)
    with torch.no_grad():
        got = _upsample_concat(skip, x)
    assert got.shape == ref.shape and torch.equal(got, ref)
    xs = x.clone().requires_grad_(True)          # autograd path: the two ATen ops
    out = _upsample_concat(skip, xs)
    assert out.requires_grad and torch.equal(out.detach(), ref)
