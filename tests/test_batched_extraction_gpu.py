"""Batched mesh extraction: B lattices per decoder launch, per-scene iso-levels, B meshes per marching-cubes
pass.  Every scene of a batch must be bit-identical to the single-scene path on the same features / volume."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu


def _decoder(variant, seed=0):
    from vtaco_b200.conv_onet.models import decoder_dict
    torch.manual_seed(seed)
    dec = decoder_dict['simple_local'](dim=3, c_dim=32, hidden_size=32).cuda().eval()
    with torch.no_grad():
        for b in dec.blocks:
            b.fc_1.weight.normal_(0, 0.1)
    dec.kernel_variant = variant
    return dec


def _features(B, R=16, seed=1):
    g = torch.Generator().manual_seed(seed)
    return {'grid': torch.randn(B, 32, R, R, R, generator=g).cuda()}


def _single(dec, c, b, nx):
    from vtaco_b200.mcubes import new_minmax_key
    keys = new_minmax_key('cuda')
    out = dec.forward_dense({k: t[b:b + 1] for k, t in c.items()}, nx, minmax_key=keys)
    return out, keys


@pytest.mark.parametrize('variant', [7, 5, 1])
@pytest.mark.parametrize('nx', [37, 64, 128])
@pytest.mark.parametrize('B', [1, 3, 8])
def test_decoder_batch_matches_single_scene(B, nx, variant):
    from vtaco_b200.mcubes import new_minmax_key
    dec = _decoder(variant)
    c = _features(B, seed=10 * B + nx)
    keys = new_minmax_key('cuda', B)
    with torch.no_grad():
        out = dec.forward_dense(c, nx, out=torch.empty((B, nx, nx, nx), device='cuda'), minmax_key=keys)
        assert out.shape == (B, nx, nx, nx)
        for b in range(B):
            ref, rkeys = _single(dec, c, b, nx)
            assert torch.equal(out[b], ref), 'scene %d logits' % b
            assert torch.equal(keys[b], rkeys), 'scene %d keys' % b


def _tip_batch(seed=3):
    """three scenes of five fingertips: scene 0 touches nothing, scene 1 has two overlapping tip balls (the
    nearest-tip rule decides), scene 2 has a tip outside the box"""
    rs = np.random.RandomState(seed)
    pos = rs.uniform(-0.35, 0.35, size=(3, 5, 3))
    pos[1, 1] = pos[1, 0] + np.array([0.03, 0.01, -0.02])
    pos[2, 4] = np.array([0.8, 0.1, -0.2])
    touch = np.array([[0, 0, 0, 0, 0], [1, 1, 0, 1, 1], [1, 0, 1, 1, 1]], dtype=np.int32)
    feat = torch.from_numpy(rs.randn(3, 5, 32).astype(np.float32)).cuda()
    return (torch.from_numpy(pos).cuda(), feat, torch.from_numpy(touch).cuda(), 0.05), pos, touch


@pytest.mark.parametrize('nx', [37, 64])
def test_fingertip_lattice_ids_match_oracle(nx):
    from oracle import convonet as oc
    from vtaco_b200.common import dense_axis
    from vtaco_b200.conv_onet import tactile
    (dpos, feat, dtouch, radius), pos, touch = _tip_batch()
    ids = tactile.fingertip_lattice_ids(dense_axis(nx, 0.1, 'cuda'), dpos, dtouch, radius)
    assert ids.shape == (3, nx ** 3)
    dense = tactile.c_img_from_ids(ids, feat).cpu()
    lattice = oc.dense_grid_points(nx)
    for b in range(3):
        ref = oc.fingertip_c_img(lattice, pos[b], feat[b].cpu(), touch[b].astype(bool), radius)
        assert torch.equal(dense[b], ref), 'scene %d' % b
    assert int((ids[0] > 0).sum()) == 0
    assert int((ids[1] == 1).sum()) > 0 and int((ids[1] == 2).sum()) > 0    # both overlapping balls win somewhere


@pytest.mark.parametrize('variant', [7, 5])
@pytest.mark.parametrize('nx', [37, 64])
def test_decoder_batch_fingertips_match_single_scene(nx, variant):
    from vtaco_b200.mcubes import new_minmax_key
    dec = _decoder(variant)
    c = _features(3, seed=nx)
    tips, pos, touch = _tip_batch()
    keys = new_minmax_key('cuda', 3)
    with torch.no_grad():
        out = dec.forward_dense(c, nx, use_img=True, tips=tips, minmax_key=keys)
        plain = dec.forward_dense(c, nx, use_img=True)
        for b in range(3):
            rkeys = new_minmax_key('cuda')
            ref = dec.forward_dense({k: t[b:b + 1] for k, t in c.items()}, nx, use_img=True, minmax_key=rkeys,
                                    tips=(pos[b], tips[1][b], touch[b].astype(bool), tips[3]))
            assert torch.equal(out[b], ref), 'scene %d logits' % b
            assert torch.equal(keys[b], rkeys), 'scene %d keys' % b
    assert torch.equal(out[0], plain[0]) and not torch.equal(out[1], plain[1])   # no touch / touched


def _volumes():
    """decoded lattices of three scenes, with a constant scene between two real ones"""
    from vtaco_b200.mcubes import new_minmax_key
    dec = _decoder(7)
    c = _features(2, seed=5)
    keys = new_minmax_key('cuda', 2)
    with torch.no_grad():
        out = dec.forward_dense(c, 48, minmax_key=keys)
    vols = torch.stack([out[0], torch.full_like(out[0], 0.25), out[1]]).contiguous()
    return vols


def _assert_batch_equals_single(vols, v, f, sc, level=None):
    from vtaco_b200.mcubes import MarchingCubes, split_meshes
    single = MarchingCubes('cuda')
    parts = split_meshes(v, f, sc.cpu())
    assert len(parts) == vols.shape[0]
    for b, (vb, fb) in enumerate(parts):
        rv, rf = single(vols[b], level=level, voffset=np.float32(24), vscale=np.float32(1.1 / 48))
        assert torch.equal(vb, rv) and torch.equal(fb, rf), 'scene %d' % b


def test_mc_batch_matches_single_volume_with_empty_scene():
    from vtaco_b200.mcubes import MarchingCubes
    vols = _volumes()
    ex = MarchingCubes('cuda')
    v, f, sc = ex.batch(vols, voffset=np.float32(24), vscale=np.float32(1.1 / 48))
    sc = sc.cpu()
    assert sc[1].tolist() == [0, 0] and sc[0, 1] > 0 and sc[2, 1] > 0
    assert int(sc[:, 0].sum()) == v.shape[0] and int(sc[:, 1].sum()) == f.shape[0]
    _assert_batch_equals_single(vols, v, f, sc)
    # explicit per-scene keys (as forward_dense of a batch writes them) give the same meshes
    from vtaco_b200.mcubes import new_minmax_key, volume_keys
    keys = volume_keys(vols, new_minmax_key('cuda', 3))
    v2, f2, sc2 = ex.batch(vols, level_keys=keys, voffset=np.float32(24), vscale=np.float32(1.1 / 48))
    assert torch.equal(v2, v) and torch.equal(f2, f) and torch.equal(sc2.cpu(), sc)


def test_mc_batch_ragged_volumes_one_level():
    """extents that are not powers of two (scene boundaries inside a look-back block), one level for all"""
    from vtaco_b200.mcubes import MarchingCubes, split_meshes
    rs = np.random.RandomState(7)
    vols = torch.from_numpy(rs.randn(5, 9, 13, 33).astype(np.float32)).cuda()
    v, f, sc = MarchingCubes('cuda').batch(vols, level=0.0)
    single = MarchingCubes('cuda')
    for b, (vb, fb) in enumerate(split_meshes(v, f, sc.cpu())):
        rv, rf = single(vols[b], level=0.0)
        assert torch.equal(vb, rv) and torch.equal(fb, rf), 'scene %d' % b


def test_mc_batch_of_one_equals_single_call():
    from vtaco_b200.mcubes import MarchingCubes
    vols = _volumes()[:1].contiguous()
    v, f, sc = MarchingCubes('cuda').batch(vols)
    rv, rf = MarchingCubes('cuda')(vols[0])
    assert torch.equal(v, rv) and torch.equal(f, rf)
    assert sc.cpu().tolist() == [[rv.shape[0], rf.shape[0]]]


def test_mc_batch_capacity_overflow_and_rerun():
    from vtaco_b200.mcubes import MarchingCubes
    vols = _volumes()
    ex = MarchingCubes('cuda')
    ex._ensure(0, 8, 8)
    ex._verts, ex._faces = ex._verts[:8].clone(), ex._faces[:8].clone()
    vb, fb, counts, sc = ex.batch(vols, sync=False)
    V, F = [int(x) for x in counts[:2].cpu()]
    assert V > 8 and F > 8 and int(sc[:, 0].sum()) == V and int(sc[:, 1].sum()) == F   # counted, not written
    ex._verts, ex._faces = ex._verts[:8].clone(), ex._faces[:8].clone()
    v, f, sc = ex.batch(vols, voffset=np.float32(24), vscale=np.float32(1.1 / 48))   # grows, re-runs phase 2
    assert v.shape[0] == V and f.shape[0] == F
    _assert_batch_equals_single(vols, v, f, sc)


def _generator(with_img=False):
    from vtaco_b200.encoder import encoder_dict
    from vtaco_b200.conv_onet.models import decoder_dict, ConvolutionalOccupancyNetwork
    from vtaco_b200.conv_onet.generation import Generator3D
    torch.manual_seed(0)
    enc = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, plane_type='grid',
                                              grid_resolution=32)
    dec = decoder_dict['simple_local'](dim=3, c_dim=32, hidden_size=32)
    with torch.no_grad():
        for m in (enc, dec):
            for b in m.blocks:
                b.fc_1.weight.normal_(0, 0.1)
    net = ConvolutionalOccupancyNetwork(dec, enc, device='cuda').eval()
    return Generator3D(net, device='cuda', resolution0=16, padding=0.1, input_type='pointcloud', with_img=with_img)


def test_generate_meshes_equals_generate_mesh_loop():
    gen = _generator()
    rs = np.random.RandomState(4)
    clouds = torch.from_numpy(rs.uniform(-0.45, 0.45, size=(4, 1500, 3)).astype(np.float32)).cuda()
    with torch.no_grad():
        c = gen.model.encode_inputs(clouds)
    meshes = gen.generate_meshes(c=c)
    assert len(meshes) == 4
    for b, (v, f) in enumerate(meshes):
        rv, rf = gen.generate_mesh(c={k: t[b:b + 1] for k, t in c.items()})
        assert np.array_equal(v, rv) and np.array_equal(f, rf), 'scene %d' % b
        assert len(f) > 0
    dv = gen.generate_meshes(c=c, to_host=False)
    assert all(torch.equal(d[0].cpu(), torch.from_numpy(m[0])) and torch.equal(d[1].cpu(), torch.from_numpy(m[1]))
               for d, m in zip(dv, meshes))


def test_generate_meshes_fingertips_equal_generate_mesh_loop():
    gen = _generator(with_img=True)
    rs = np.random.RandomState(8)
    clouds = torch.from_numpy(rs.uniform(-0.45, 0.45, size=(3, 1500, 3)).astype(np.float32)).cuda()
    (dpos, feat, dtouch, radius), pos, touch = _tip_batch()
    with torch.no_grad():
        c = gen.model.encode_inputs(clouds)
    meshes = gen.generate_meshes(c=c, tips=(pos, feat, touch), radius=radius)
    plain = gen.generate_meshes(c=c)
    for b, (v, f) in enumerate(meshes):
        rv, rf = gen.generate_mesh(c={k: t[b:b + 1] for k, t in c.items()},
                                   tips=(pos[b], feat[b], touch[b].astype(bool), radius))
        assert np.array_equal(v, rv) and np.array_equal(f, rf), 'scene %d' % b
    assert np.array_equal(meshes[0][1], plain[0][1])


def test_capture_generate_batch_rereads_fingertips():
    gen = _generator(with_img=True)
    rs = np.random.RandomState(9)
    clouds = torch.from_numpy(rs.uniform(-0.45, 0.45, size=(3, 1500, 3)).astype(np.float32)).pin_memory()
    (dpos, feat, dtouch, radius), _, _ = _tip_batch()
    tips = (dpos, feat, dtouch)

    def similar(ma, mb):
        return len(ma) == len(mb) and all(abs(len(a[1]) - len(b[1])) <= max(4, 0.01 * len(b[1])) for a, b in zip(ma, mb))

    run = gen.capture_generate_batch(clouds, tips=tips, radius=radius)
    assert similar(run(), gen.generate_meshes(inputs=clouds, tips=tips, radius=radius))
    # new fingertips written into the same tensors: the replay decodes with them
    dpos.copy_(torch.from_numpy(rs.uniform(-0.3, 0.3, size=(3, 5, 3))))
    dtouch.fill_(1)
    feat.mul_(3.0)
    replay = run()
    eager = gen.generate_meshes(inputs=clouds, tips=tips, radius=radius)
    assert similar(replay, eager)
    with pytest.raises(ValueError):   # host fingertips cannot be re-read by a graph
        gen.capture_generate_batch(clouds, tips=(dpos.cpu().numpy(), feat, dtouch))


def test_capture_generate_batch_matches_eager():
    gen = _generator()
    rs = np.random.RandomState(5)
    clouds = torch.from_numpy(rs.uniform(-0.45, 0.45, size=(3, 1500, 3)).astype(np.float32)).pin_memory()

    # the encoder's scatter_mean sums in arrival order: separate runs may differ in the last bits, so meshes
    # of separate encodes are compared by size (the decode / extraction of given features is bit-exact above)
    def similar(ma, mb):
        return len(ma) == len(mb) and all(abs(len(a[1]) - len(b[1])) <= max(4, 0.01 * len(b[1])) for a, b in zip(ma, mb))

    eager = gen.generate_meshes(inputs=clouds)
    run = gen.capture_generate_batch(clouds)
    assert similar(run(), eager)
    clouds.copy_(torch.from_numpy(rs.uniform(-0.35, 0.35, size=(3, 1500, 3)).astype(np.float32)))   # new batch
    replay = run()
    eager = gen.generate_meshes(inputs=clouds)
    assert similar(replay, eager)
    for v, f in replay:
        assert len(f) == 0 or (f.min() >= 0 and f.max() < len(v))


def test_argument_errors(monkeypatch):
    from vtaco_b200 import dist as vdist
    from vtaco_b200.mcubes import MarchingCubes, new_minmax_key
    dec = _decoder(7)
    c = _features(3)
    with torch.no_grad():
        with pytest.raises(ValueError):    # features of 3 scenes, out of 2
            dec.forward_dense(c, 16, out=torch.empty((2, 16, 16, 16), device='cuda'))
        with pytest.raises(ValueError):    # a single lattice for 3 scenes
            dec.forward_dense(c, 16, out=torch.empty((16, 16, 16), device='cuda'))
        with pytest.raises(ValueError):    # keys of 2 scenes
            dec.forward_dense(c, 16, minmax_key=new_minmax_key('cuda', 2))
        with pytest.raises(ValueError):    # keys of the wrong dtype
            dec.forward_dense(c, 16, minmax_key=torch.zeros((3, 2), dtype=torch.int64, device='cuda'))
        with pytest.raises(ValueError):    # out of the wrong dtype
            dec.forward_dense(c, 16, out=torch.empty((3, 16, 16, 16), dtype=torch.float64, device='cuda'))
        with pytest.raises(NotImplementedError):
            dec.forward_dense(c, 16, use_img=True, c_img=torch.zeros((3 * 16 ** 3, 32), device='cuda'))
        with pytest.raises(NotImplementedError):
            dec.forward_dense(c, 16, x0=0, x1=8)
    ex = MarchingCubes('cuda')
    vols = torch.zeros((3, 8, 8, 8), device='cuda')
    with pytest.raises(ValueError):
        ex.batch(vols, level_keys=new_minmax_key('cuda', 2))
    with pytest.raises(ValueError):
        ex.batch(vols, level_keys=torch.zeros((3, 2), dtype=torch.int64, device='cuda'))
    with pytest.raises(TypeError):
        ex.batch(vols.double())
    with pytest.raises(ValueError):
        ex.batch(vols[0])
    tips = _tip_batch()[0]
    with torch.no_grad():
        with pytest.raises(ValueError):    # fingertips of 2 scenes for 3
            dec.forward_dense(c, 16, use_img=True, tips=(tips[0][:2], tips[1][:2], tips[2][:2], 0.05))
        with pytest.raises(ValueError):    # float32 positions
            dec.forward_dense(c, 16, use_img=True, tips=(tips[0].float(), tips[1], tips[2], 0.05))
        with pytest.raises(ValueError):    # bool touch mask
            dec.forward_dense(c, 16, use_img=True, tips=(tips[0], tips[1], tips[2].bool(), 0.05))
        with pytest.raises(ValueError):    # float64 features
            dec.forward_dense(c, 16, use_img=True, tips=(tips[0], tips[1].double(), tips[2], 0.05))
        dec.kernel_variant = 1
        with pytest.raises(NotImplementedError):   # the byte map is read by the tcgen05 kernels only
            dec.forward_dense(c, 16, use_img=True, tips=tips)
    gen = _generator()
    cl = torch.zeros((2, 100, 3)).pin_memory()
    monkeypatch.setattr(vdist, 'rank_world', lambda group=None: (0, 2))
    with pytest.raises(NotImplementedError):
        gen.generate_meshes(c=c)
    with pytest.raises(NotImplementedError):
        gen.capture_generate_batch(cl)
