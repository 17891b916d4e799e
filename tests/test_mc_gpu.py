"""GPU marching cubes (through the C ABI) against the oracle, bit for bit: counts, faces and vertices.

The kernel places a vertex at e0 / (e0 + e1) with e = FLT_EPSILON + |value - level|; the oracle uses Lewiner's
w1 / (w0 + w1) with w = 1 / e (an infinite sample has weight 0 in both).  Both are float64 rounded to float32, so
they can differ only by the double rounding of the two formulas.  assert_matches_oracle therefore recomputes the kernel's formula in numpy and demands it bit for
bit, and demands that this formula is within one float32 ulp of the oracle's vertex."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle import marching_cubes as omc

pytestmark = pytest.mark.gpu

INF = float('inf')


def _np(t):
    return t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)


def same_bits(a, b):
    """float32 arrays equal bit for bit (signed zeros included); any NaN matches any NaN"""
    a, b = np.asarray(a, dtype=np.float32), np.asarray(b, dtype=np.float32)
    return a.shape == b.shape and bool(((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))).all())


def kernel_vertices(vol, level):
    """the kernel's vertex formula (csrc/mcubes.cu, mc_emit_kernel) in numpy, in the oracle's vertex order"""
    vol = np.ascontiguousarray(vol, dtype=np.float32)
    with np.errstate(invalid='ignore'):   # -inf + inf: a NaN level
        level = omc.iso_level(vol) if level is None else np.float32(level)
    above = vol > level
    flags = np.zeros(vol.shape + (3,), dtype=bool)
    flags[:-1, :, :, 0] = above[:-1] != above[1:]
    flags[:, :-1, :, 1] = above[:, :-1] != above[:, 1:]
    flags[:, :, :-1, 2] = above[:, :, :-1] != above[:, :, 1:]
    i, j, k, a = np.argwhere(flags).T
    step = np.eye(3, dtype=np.int64)[a]
    with np.errstate(invalid='ignore'):   # inf - inf at an infinite level: a NaN vertex on both sides
        e0 = omc.FLT_EPSILON + np.abs(vol[i, j, k].astype(np.float64) - float(level))
        e1 = omc.FLT_EPSILON + np.abs(vol[i + step[:, 0], j + step[:, 1], k + step[:, 2]].astype(np.float64) -
                                      float(level))
        t = np.where((e0 == np.inf) & (e1 < np.inf), 1.0, e0 / (e0 + e1))
        verts = np.stack([i, j, k], 1).astype(np.float64)
        verts[np.arange(len(a)), a] += t
    return verts.astype(np.float32)


def assert_matches_oracle(vol, level, v, f, rescale_nx=None):
    """GPU mesh (v, f) of `vol` at `level` == oracle: faces bit for bit, vertices bit for bit equal to the kernel's
    formula, which is within 1 ulp of the oracle's; with rescale_nx, the vertices are rescale_vertices of those.
    Returns the oracle's (vertices, faces)."""
    vol = np.ascontiguousarray(vol, dtype=np.float32)
    with np.errstate(invalid='ignore'):
        rv, rf, _ = omc.marching_cubes(vol, level)
    v, f = _np(v), _np(f)
    assert v.shape == rv.shape and f.shape == rf.shape, (v.shape, rv.shape, f.shape, rf.shape)
    assert np.array_equal(f, rf)
    kv = kernel_vertices(vol, level)
    assert kv.shape == rv.shape
    fin = ~np.isnan(rv)
    assert np.array_equal(np.isnan(kv), ~fin)
    # index coordinates are >= 0, so adjacent floats have adjacent bit patterns
    assert np.abs(kv[fin].view(np.int32).astype(np.int64) - rv[fin].view(np.int32)).max(initial=0) <= 1
    want = kv if rescale_nx is None else omc.rescale_vertices(kv, rescale_nx)
    assert same_bits(v, want), 'vertices differ from the kernel formula at %d places' % int(
        (v.view(np.uint32) != want.view(np.uint32)).sum())
    return rv, rf


def smooth(shape, seed=0):
    """closed surfaces: a union of balls inside the box, in index units of the largest extent"""
    rs = np.random.RandomState(seed)
    n = max(shape)
    x, y, z = np.meshgrid(*[np.arange(s, dtype=np.float32) / n for s in shape], indexing='ij')
    out = np.full(shape, -1.0, dtype=np.float32)
    for _ in range(4):
        c = rs.uniform(0.2, 0.8, 3) * np.array(shape) / n
        r = rs.uniform(0.08, 0.25) * min(shape) / n
        out = np.maximum(out, (r - np.sqrt((x - c[0]) ** 2 + (y - c[1]) ** 2 + (z - c[2]) ** 2)).astype(np.float32))
    return out


def fields():
    rs = np.random.RandomState(0)
    ax = np.linspace(-1, 1, 48, dtype=np.float32)
    x, y, z = np.meshgrid(ax, ax, ax, indexing='ij')
    out = {'sphere': (0.7 - np.sqrt(x * x + y * y + z * z)).astype(np.float32),
           'noise': np.pad(rs.randn(20, 21, 22).astype(np.float32), 1, constant_values=-10.0),
           'ragged': rs.randn(5, 9, 33).astype(np.float32),
           'flat': np.zeros((6, 6, 6), dtype=np.float32),
           'tiny': np.arange(8, dtype=np.float32).reshape(2, 2, 2),
           # integers: ties with levels 0 and 1 everywhere
           'ties': rs.randint(-2, 3, size=(19, 20, 24)).astype(np.float32)}
    # -0.0 and +0.0 side by side (level -0.0 and +0.0 must select the same corners), float4 and scalar row loads
    zeros = np.array([-1.0, -0.0, 0.0, 1.0], dtype=np.float32)
    out['signed_zeros'] = zeros[rs.randint(0, 4, size=(17, 18, 24))]
    out['signed_zeros_ragged'] = zeros[rs.randint(0, 4, size=(17, 18, 21))]
    inf = rs.randn(16, 17, 32).astype(np.float32)
    inf[rs.rand(*inf.shape) < 0.1] = np.inf
    inf[rs.rand(*inf.shape) < 0.1] = -np.inf
    out['inf'] = inf
    nan = rs.randn(16, 17, 19).astype(np.float32)
    nan[rs.rand(*nan.shape) < 0.1] = np.nan
    nan[rs.rand(*nan.shape) < 0.05] = -np.nan
    out['nan'] = nan
    nan8 = rs.randn(16, 17, 24).astype(np.float32)
    nan8[rs.rand(*nan8.shape) < 0.1] = np.nan
    out['nan_rows8'] = nan8
    return out


def _level_of_keys(keys):
    from vtaco_b200.mcubes import keys_to_level
    return np.float32(keys_to_level(keys))


@pytest.mark.parametrize('name', list(fields()))
@pytest.mark.parametrize('level', [None, 0.0, -0.0, 1.0, INF, -INF])
def test_mc_matches_oracle(name, level):
    """every field at every level; level=None: the level itself equals the oracle's iso_level bit for bit (NaN
    when the volume holds a NaN, or both infinities)"""
    from vtaco_b200.mcubes import MarchingCubes
    vol = fields()[name]
    ex = MarchingCubes('cuda')
    v, f = ex(torch.from_numpy(vol).cuda(), level)
    if level is None:
        with np.errstate(invalid='ignore'):
            assert same_bits(_level_of_keys(ex._keys), omc.iso_level(vol))
    assert_matches_oracle(vol, level, v, f)


def _shape_cases():
    cases = [(9, 10, nz) for nz in list(range(8, 17)) + [1, 2, 7]]     # every nz % 8, both row paths
    cases += [(1, 12, 13), (12, 1, 13), (1, 1, 16)]                      # vertices and no faces
    cases += [(33, 64, 128), (33, 63, 120)]                              # shift / division run coordinates
    cases += [(16, 8, 64), (41, 25, 8), (64, 128, 64), (65, 128, 64)]    # 1 024, 1 025, 65 536, 66 560 runs
    cases += [(128, 128, 128), (300, 97, 130)]
    out = []
    for s in cases:
        for field in ('noise', 'smooth'):
            if field == 'noise' and np.prod(s) > 128 ** 3:
                continue
            out.append(pytest.param(s, field, id='%dx%dx%d-%s' % (s + (field,))))
    return out


@pytest.mark.parametrize('shape,field', _shape_cases())
def test_mc_shapes_match_oracle(shape, field):
    """Extents at the edges of the row loads (nz % 8, nz < 8), of the run coordinates (power-of-two ny / nzc or
    not) and of the look-back blocks of 1 024 runs: one block, one more run, 64 blocks (what one look-back round
    reads), one more block, and up to 484 blocks.  The 256^3 lattice tests below have 2 048 blocks, more than the
    CTAs resident at once (6 per SM), so CTAs draw several tickets there.  These sizes make a second look-back
    round, polling on unpublished predecessors and CTAs that draw several tickets possible; which of them happen
    depends on timing, and a test cannot force them."""
    from vtaco_b200.mcubes import marching_cubes
    rs = np.random.RandomState(sum(shape))
    vol = rs.randn(*shape).astype(np.float32) if field == 'noise' else smooth(shape)
    level = 0.0 if field == 'noise' else None
    v, f = marching_cubes(torch.from_numpy(vol).cuda(), level)
    assert_matches_oracle(vol, level, v, f)


def test_mc_level_sources_match_oracle():
    """level=None taken from given keys, from a device float (level_ptr) and from three key pairs merged in
    the kernel (the per-rank pairs of the fused exchange) == the oracle at iso_level"""
    from vtaco_b200 import _abi
    from vtaco_b200.mcubes import MarchingCubes, new_minmax_key, volume_keys
    vol = smooth((40, 44, 48), seed=3)
    vol[5:9] += 0.5          # the maximum lies in the first of the three parts below, the minimum in the last
    vol[35] -= 1.0
    vt = torch.from_numpy(vol).cuda()
    ex = MarchingCubes('cuda')
    keys = volume_keys(vt[None], new_minmax_key('cuda', 1))[0]
    assert same_bits(_level_of_keys(keys), omc.iso_level(vol))
    v, f = ex(vt, level_keys=keys)
    assert_matches_oracle(vol, None, v, f)
    lv = torch.tensor([omc.iso_level(vol)], dtype=torch.float32, device='cuda')
    v, f = ex(vt, level=123.0, level_ptr=lv.data_ptr())        # the device level takes precedence
    assert_matches_oracle(vol, None, v, f)
    L = _abi.lib()
    pairs = torch.zeros((3, 2), dtype=torch.int32, device='cuda')
    for r, (x0, x1) in enumerate([(0, 10), (10, 30), (30, 40)]):
        part = vt[x0:x1].contiguous()
        _abi.check(L.vtaco_grid_minmax(_abi.ptr(part), part.numel(), _abi.ptr(pairs[r]), _abi.stream_ptr()), 'minmax')
    assert not torch.equal(pairs[0], pairs[1])
    v, f = ex(vt, level_keys=pairs)
    assert_matches_oracle(vol, None, v, f)


def test_mc_nan_level_rule_single_equals_batch():
    """level=None on a volume with a NaN: NaN, so the mesh is empty, in the single-volume and the batched path"""
    from vtaco_b200.mcubes import MarchingCubes
    vol = fields()['nan_rows8']
    vt = torch.from_numpy(vol).cuda()
    ex = MarchingCubes('cuda')
    v, f = ex(vt)
    assert np.isnan(_level_of_keys(ex._keys)) and v.shape[0] == 0 and f.shape[0] == 0
    vb, fb, sc = ex.batch(vt[None].contiguous())
    assert vb.shape[0] == 0 and fb.shape[0] == 0 and sc.cpu().tolist() == [[0, 0]]


def test_mc_misaligned_view_matches_oracle():
    """a contiguous view that starts one float into its buffer (not 16-byte aligned), with nz % 8 == 0, and a
    separate halo buffer at an odd address"""
    from vtaco_b200.mcubes import marching_cubes
    vol = smooth((24, 20, 32), seed=5)
    for off in (1, 2, 3):
        buf = torch.empty(vol.size + off, dtype=torch.float32, device='cuda')
        t = buf[off:].view(vol.shape)
        t.copy_(torch.from_numpy(vol))
        assert t.data_ptr() % 16 != 0
        v, f = marching_cubes(t, None)
        assert_matches_oracle(vol, None, v, f)
        pv, pf = _mc_pieces(t, 0.0, [(0, 7), (7, 24)], separate_halo=True, halo_offset=off)
        assert_matches_oracle(vol, 0.0, pv, pf)


def test_mc_capacity_regrow_and_rescale():
    from vtaco_b200.mcubes import MarchingCubes
    ex = MarchingCubes('cuda')
    vol = fields()['noise']
    small = torch.from_numpy(fields()['tiny']).cuda()
    ex(small)  # allocates small buffers
    ex._verts = ex._verts[:4].clone()
    ex._faces = ex._faces[:4].clone()
    nx = vol.shape[0]
    v, f = ex(torch.from_numpy(vol).cuda(), 0.0, voffset=np.float32(nx / 2), vscale=np.float32(1.1 / nx))
    assert_matches_oracle(vol, 0.0, v, f, rescale_nx=nx)


def test_mc_overflow_writes_nothing_past_the_capacity():
    """capacities one short of the mesh, and tiny ones: the counts are right, what fits is the oracle's prefix,
    a guard region past each capacity keeps its sentinel, and the re-run with grown buffers is the oracle's mesh"""
    from vtaco_b200.mcubes import MarchingCubes
    vol = fields()['noise']
    rv, rf, _ = omc.marching_cubes(vol, 0.0)
    V, F = len(rv), len(rf)
    vt = torch.from_numpy(vol).cuda()
    guard = 64
    for vcap, fcap in [(V - 1, F - 1), (V, F - 1), (V - 1, F), (1, 1)]:
        ex = MarchingCubes('cuda')
        vbuf = torch.full((vcap + guard, 3), -7.0, device='cuda')
        fbuf = torch.full((fcap + guard, 3), -7, dtype=torch.int32, device='cuda')
        ex._verts, ex._faces = vbuf[:vcap], fbuf[:fcap]
        _, _, counts = ex(vt, 0.0, sync=False)
        assert counts[:3].cpu().tolist() == [V, F, V]
        vb, fb = vbuf.cpu().numpy(), fbuf.cpu().numpy()
        assert same_bits(vb[:vcap], kernel_vertices(vol, 0.0)[:vcap]) and np.array_equal(fb[:fcap], rf[:fcap])
        assert (vb[vcap:] == -7.0).all() and (fb[fcap:] == -7).all()
        v, f = ex(vt, 0.0)
        assert_matches_oracle(vol, 0.0, v, f)


def _mc_args(vol_t, level, scratch, counts, verts, faces, phase):
    from vtaco_b200 import _abi
    a = _abi.McArgs()
    a.grid = vol_t.data_ptr()
    a.nx, a.ny, a.nz = vol_t.shape[-3:]
    a.level = level
    a.scratch, a.scratch_bytes = scratch.data_ptr(), scratch.numel()
    a.counts = counts.data_ptr()
    a.vertices, a.vertex_capacity = verts.data_ptr(), verts.shape[0]
    a.faces, a.face_capacity = faces.data_ptr(), faces.shape[0]
    a.vscale, a.phase = 1.0, phase
    return a


@pytest.mark.parametrize('batch', [False, True])
def test_mc_count_only_writes_nothing(batch):
    """phase 1: the counts (and per-scene counts) of the oracle; vertex and face buffers keep their sentinel"""
    from vtaco_b200 import _abi
    L = _abi.lib()
    vols = np.stack([fields()['noise'], smooth((22, 23, 24), seed=1), np.zeros((22, 23, 24), np.float32)])
    if not batch:
        vols = vols[:1]
    vt = torch.from_numpy(vols).cuda()
    B = vols.shape[0]
    nbytes = L.vtaco_mc_batch_scratch_bytes(B, *vols.shape[1:]) if batch else L.vtaco_mc_scratch_bytes(*vols.shape[1:])
    scratch = torch.full((nbytes,), 0x5a, dtype=torch.uint8, device='cuda')
    counts = torch.full((4,), -1, dtype=torch.int64, device='cuda')
    verts = torch.full((1 << 16, 3), -7.0, device='cuda')
    faces = torch.full((1 << 16, 3), -7, dtype=torch.int32, device='cuda')
    a = _mc_args(vt if batch else vt[0], 0.0, scratch, counts, verts, faces, 1)
    sc = torch.full((B, 2), -1, dtype=torch.int64, device='cuda')
    if batch:
        a.n_volumes, a.scene_counts = B, sc.data_ptr()
    _abi.check(L.vtaco_marching_cubes(C.byref(a), _abi.stream_ptr()), 'marching_cubes')
    ref = [omc.marching_cubes(vols[b], 0.0)[:2] for b in range(B)]
    V, F = sum(len(r[0]) for r in ref), sum(len(r[1]) for r in ref)
    assert counts[:3].cpu().tolist() == [V, F, V]
    if batch:
        assert sc.cpu().tolist() == [[len(rv), len(rf)] for rv, rf in ref]
    assert (verts == -7.0).all().item() and (faces == -7).all().item()


def _key(x):
    """float -> the ordered-int key of csrc/common.cuh (float_to_key)"""
    b = int(np.float32(x).view(np.int32))
    return b if b >= 0 else b ^ 0x7fffffff


def test_mc_batch_matches_oracle_per_scene():
    """B = 8 volumes of (37, 50, 41) at per-scene levels from keys: an empty (constant) scene, a scene whose keys
    put every sample above its level, and a scene whose surface reaches its last row, the row it shares with the
    next scene.  Each scene and its counts == the oracle on that volume alone."""
    from vtaco_b200.mcubes import MarchingCubes, new_minmax_key, split_meshes, volume_keys
    shape = (37, 50, 41)
    rs = np.random.RandomState(11)
    vols = [smooth(shape, seed=20 + b) for b in range(8)]
    vols[1] = np.full(shape, 0.25, np.float32)                               # empty
    vols[3] = rs.randn(*shape).astype(np.float32)
    vols[5] = np.broadcast_to((np.arange(37, dtype=np.float32) - 35.5)[:, None, None], shape).copy()   # last row above
    vols[5] += 0.01 * rs.rand(*shape).astype(np.float32)
    vols[7] = rs.randint(-1, 2, size=shape).astype(np.float32)
    vt = torch.from_numpy(np.stack(vols)).cuda()
    keys = volume_keys(vt, new_minmax_key('cuda', 8))
    keys[2] = torch.tensor([_key(-5.0), _key(-3.0)], dtype=torch.int32)    # level -4: every sample is above
    keys[5] = torch.tensor([_key(-1.0), _key(1.0)], dtype=torch.int32)     # level 0: only the last row is above
    levels = [_level_of_keys(keys[b]) for b in range(8)]
    for b in (0, 1, 3, 4, 6, 7):
        assert same_bits(levels[b], omc.iso_level(vols[b]))
    v, f, sc = MarchingCubes('cuda').batch(vt, level_keys=keys)
    sc = sc.cpu()
    parts = split_meshes(v, f, sc)
    for b, (vb, fb) in enumerate(parts):
        rv, rf = assert_matches_oracle(vols[b], levels[b], vb, fb)
        assert sc[b].tolist() == [len(rv), len(rf)], 'scene %d' % b
    assert sc[1].tolist() == [0, 0] and sc[2].tolist() == [0, 0]
    assert float(parts[5][0][:, 0].max()) > 35.0      # scene 5 has vertices between its last two rows


# ------------------------------------------------------------------------------------------------
# the decoded 256^3 lattice of the benchmarked size
# ------------------------------------------------------------------------------------------------
@pytest.fixture(scope='module')
def lattice_256():
    """decoded 256^3 lattice, its keys, and the oracle's mesh of it"""
    from vtaco_b200.conv_onet.models import decoder_dict, ConvolutionalOccupancyNetwork
    from vtaco_b200.conv_onet.generation import Generator3D
    torch.manual_seed(0)
    dec = decoder_dict['simple_local'](dim=3, c_dim=32, hidden_size=32)
    with torch.no_grad():
        for b in dec.blocks:
            b.fc_1.weight.normal_(0, 0.1)
    net = ConvolutionalOccupancyNetwork(dec, None, device='cuda')
    gen = Generator3D(net, device='cuda', resolution0=64, with_img=False, padding=0.1, input_type='pointcloud')
    grid, keys = gen.eval_lattice({'grid': torch.randn(1, 32, 64, 64, 64, device='cuda')})
    return gen, grid.clone(), keys.clone(), grid.cpu().numpy()


def test_generator_mesh_pipeline_256_properties(lattice_256):
    """full size: 256^3 lattice decode + MC: the level from the decoder's keys is the oracle's iso_level bit for
    bit, the mesh is the oracle's, and a second extraction repeats it"""
    from vtaco_b200.mcubes import keys_to_level
    gen, grid, keys, host = lattice_256
    assert grid.shape == (256, 256, 256)
    level = keys_to_level(keys)
    assert same_bits(np.float32(level), omc.iso_level(host))
    v, f = gen.extract_mesh(grid, keys)
    v2, f2 = [t.clone() for t in (v, f)]
    v, f = gen.extract_mesh(grid, keys)
    assert torch.equal(v, v2) and torch.equal(f, f2)
    assert f.numel() > 0 and float(v.abs().max()) <= 0.55 + 1e-6
    assert_matches_oracle(host, None, v, f, rescale_nx=256)


def test_mc_scratch_reuse_between_sizes(lattice_256):
    """one extractor: 256^3, then (9, 13, 33), then 256^3 again; both large meshes == the oracle"""
    from vtaco_b200.mcubes import MarchingCubes
    _, grid, keys, host = lattice_256
    ex = MarchingCubes('cuda')
    v, f = ex(grid, level_keys=keys)
    assert_matches_oracle(host, None, v, f)
    small = np.random.RandomState(2).randn(9, 13, 33).astype(np.float32)
    v, f = ex(torch.from_numpy(small).cuda(), 0.0)
    assert_matches_oracle(small, 0.0, v, f)
    v, f = ex(grid, level_keys=keys)
    assert_matches_oracle(host, None, v, f)


def test_bench_lattice_with_fingertips_matches_oracle():
    """the benchmark's configuration (bench.build_models / synthetic_scene): encoder + UNet3D features, the 256^3
    lattice decoded with fingertip conditioning, extracted and rescaled as Generator3D does == the oracle"""
    from bench import build_models, synthetic_scene
    from vtaco_b200.conv_onet.generation import Generator3D
    dev = torch.device('cuda')
    net = build_models(dev)
    cloud, tips, tf, touch = synthetic_scene(0)
    gen = Generator3D(net, device=dev, resolution0=64, with_img=True, padding=0.1, input_type='pointcloud')
    with torch.no_grad():
        c = net.encode_inputs(torch.from_numpy(cloud)[None].to(dev))
        grid, keys = gen.eval_lattice(c, tips=(tips, torch.from_numpy(tf).to(dev), touch, 0.05))
        v, f = gen.extract_mesh(grid, keys)
    host = grid.cpu().numpy()
    assert f.shape[0] > 1000
    assert_matches_oracle(host, None, v, f, rescale_nx=256)


def test_cuda_graph_paths_match_eager():
    """capture_step / capture_generate replay == eager launches (same grid, same mesh)."""
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
    gen = Generator3D(net, device='cuda', resolution0=16, with_img=True, padding=0.1, input_type='pointcloud')
    rs = np.random.RandomState(3)
    cloud = torch.from_numpy(rs.uniform(-0.5, 0.5, size=(1, 1500, 3)).astype(np.float32)).pin_memory()
    tips = (rs.uniform(-0.3, 0.3, size=(3, 3)), torch.randn(3, 32, device='cuda'), [True, False, True], 0.05)
    v0, f0 = gen.generate_mesh(inputs=cloud, tips=tips)
    v0, f0 = v0.copy(), f0.copy()
    with torch.no_grad():
        c = net.encode_inputs(cloud.cuda())
    graph, out = gen.capture_step(c, tips=tips)
    graph.replay()
    V, F = [int(x) for x in out[2][:2].cpu()]
    assert F == f0.shape[0] and np.array_equal(out[1][:F].cpu().numpy(), f0)
    assert np.abs(out[0][:V].cpu().numpy() - v0).max() <= 1e-6
    # the encoder's scatter_mean uses fp32 atomics (order not fixed), so two encoder runs may differ
    # in the last bits: compare meshes of separate runs by size, not bit-for-bit
    def similar(fa, fb):
        return abs(len(fa) - len(fb)) <= max(4, 0.01 * len(fb))
    run = gen.capture_generate(cloud, tips=tips)
    v1, f1 = run()
    assert similar(f1, f0) and np.abs(v1).max() <= 0.55 + 1e-6
    cloud.copy_(torch.from_numpy(rs.uniform(-0.4, 0.4, size=(1, 1500, 3)).astype(np.float32)))   # new scene, same graph
    v2, f2 = run()
    v3, f3 = gen.generate_mesh(inputs=cloud, tips=tips)
    assert similar(f2, f3)


def _mc_pieces(vol_t, level, slabs, separate_halo=False, halo_offset=0):
    """slab-mode marching cubes on each x-slab (+ 2 halo rows), pieces concatenated with their bases —
    the single-GPU emulation of the sharded extraction (csrc/mcubes.cu slab mode + exchange.cu's rebase).
    separate_halo: the halo rows are a copy in another buffer, passed by address (vtaco_mc_args.halo_grid) —
    what a rank does with the next rank's peer-mapped grid; halo_offset floats into that buffer."""
    from vtaco_b200.mcubes import MarchingCubes
    ex = MarchingCubes('cuda')
    nx = vol_t.shape[0]
    vs, fs, base = [], [], 0
    for x0, x1 in slabs:
        xh = min(x1 + 2, nx)
        kw = {}
        vol = vol_t[x0:xh]
        if separate_halo and xh > x1:
            rows = vol_t[x1:xh]
            other = torch.empty(rows.numel() + halo_offset, device=rows.device)[halo_offset:].view(rows.shape)
            other.copy_(rows)
            vol = vol_t[x0:x1].clone()          # nothing behind the slab's own rows
            kw = {'halo': (other.data_ptr(), xh - x1)}
        v, f, counts = ex(vol, level, x_emit=x1 - x0, x_origin=x0, sync=False, **kw)
        V, F, Vnum = [int(x) for x in counts[:3].cpu()]
        if V > v.shape[0] or F > f.shape[0]:
            ex._ensure(0, V + 16, F + 16)
            v, f, counts = ex(vol, level, x_emit=x1 - x0, x_origin=x0, sync=False, **kw)
        assert Vnum >= V
        vs.append(v[:V].clone())
        fs.append(f[:F].clone() + base)
        base += V
    return torch.cat(vs), torch.cat(fs)


@pytest.mark.parametrize('name,slabs', [
    ('sphere', [(0, 12), (12, 24), (24, 36), (36, 48)]),
    ('sphere', [(0, 1), (1, 2), (2, 47), (47, 48)]),
    ('noise', [(0, 7), (7, 8), (8, 20), (20, 22)]),
    ('ragged', [(0, 2), (2, 5)]),
    ('tiny', [(0, 1), (1, 2)]),
])
def test_slab_pieces_concatenate_to_the_whole_mesh(name, slabs):
    """vertex / face ids and order of the concatenated slab pieces == marching cubes of the whole
    volume, bit-for-bit (what makes the N-GPU mesh identical to the 1-GPU mesh), == the oracle."""
    from vtaco_b200.mcubes import marching_cubes
    vol = torch.from_numpy(fields()[name]).cuda()
    level = 0.0 if name != 'tiny' else 3.5
    v, f = marching_cubes(vol, level)
    for separate_halo in (False, True):
        pv, pf = _mc_pieces(vol, level, slabs, separate_halo)
        assert pv.shape == v.shape and pf.shape == f.shape
        assert torch.equal(pf, f) and torch.equal(pv, v)
    assert_matches_oracle(fields()[name], level, pv, pf)


def test_slab_pieces_256_lattice(lattice_256):
    """the benchmarked size: 8 slabs of a decoded 256^3 lattice reproduce the whole mesh and the oracle's."""
    from vtaco_b200.mcubes import keys_to_level, marching_cubes
    _, grid, keys, host = lattice_256
    level = keys_to_level(keys)
    v, f = marching_cubes(grid, level)
    for separate_halo in (False, True):
        pv, pf = _mc_pieces(grid, level, [(32 * r, 32 * r + 32) for r in range(8)], separate_halo)
        assert f.shape[0] > 1000 and torch.equal(pf, f) and torch.equal(pv, v)
    assert_matches_oracle(host, level, pv, pf)


def test_exchange_kernels_world_1():
    """vtaco_exchange_level / vtaco_exchange_mesh with a single rank (plain device memory as the
    control block): level == 0.5*(min+max) of the published keys, the piece lands rebased at base 0,
    totals and sequence numbers advance; three steps in a row (double-buffer parity)."""
    from vtaco_b200 import _abi
    L = _abi.lib()
    dev = torch.device('cuda')
    ctrl = torch.zeros(_abi.EXCHANGE_CTRL_BYTES // 4, dtype=torch.int32, device=dev)
    ex = _abi.Exchange()
    ex.ctrl[0], ex.world, ex.rank = ctrl.data_ptr(), 1, 0
    st = _abi.stream_ptr(dev)
    for step in range(3):
        g = torch.randn(1000, device=dev) * (step + 1)
        keys = torch.zeros(2, dtype=torch.int32, device=dev)
        _abi.check(L.vtaco_grid_minmax(_abi.ptr(g), g.numel(), _abi.ptr(keys), st), 'minmax')
        _abi.check(L.vtaco_exchange_level(C.byref(ex), _abi.ptr(keys), st), 'level')
        level = ctrl[_abi.EXCHANGE_LEVEL_OFFSET // 4:_abi.EXCHANGE_LEVEL_OFFSET // 4 + 1].view(torch.float32).item()
        want = (torch.tensor(0.5) * (g.min().cpu() + g.max().cpu())).item()
        assert level == want
        assert keys.tolist() == [2 ** 31 - 1, -2 ** 31]          # reset for the next step
        V, F = 50 + step, 80 + step
        verts = torch.randn(V, 3, device=dev)
        faces = torch.randint(0, V, (F, 3), dtype=torch.int32, device=dev)
        counts = torch.tensor([V, F, V, 0], dtype=torch.int64, device=dev)
        dv = torch.zeros(100, 3, device=dev)
        df = torch.zeros(100, 3, dtype=torch.int32, device=dev)
        tot = torch.zeros(2, dtype=torch.int64, device=dev)
        m = _abi.MeshPiece()
        m.counts, m.vertices, m.faces = counts.data_ptr(), verts.data_ptr(), faces.data_ptr()
        m.dst_vertices[0], m.dst_faces[0] = dv.data_ptr(), df.data_ptr()
        m.vertex_capacity, m.face_capacity, m.total_counts = 100, 100, tot.data_ptr()
        _abi.check(L.vtaco_exchange_mesh(C.byref(ex), C.byref(m), st), 'mesh')
        assert tot.tolist() == [V, F]
        assert torch.equal(dv[:V], verts) and torch.equal(df[:F], faces)
        assert ctrl[_abi.EXCHANGE_ERR_OFFSET // 4].item() == 0
