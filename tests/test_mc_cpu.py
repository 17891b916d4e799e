"""CPU: invariants that pin the marching-cubes restatement (skimage is absent — PARITY UNPINNED):
watertightness, Euler characteristic, outward orientation, vertices on the analytic
surface, and that the generated CUDA header matches the rule."""
import os

import numpy as np
import pytest

from oracle import marching_cubes as mc, mc_tables as T


def lattice(n):
    ax = np.linspace(-1, 1, n, dtype=np.float32)
    return np.meshgrid(ax, ax, ax, indexing='ij')


def test_header_in_sync(tmp_path):
    p = tmp_path / 'mc_tables.h'
    T.write_header(str(p))
    assert open(p).read() == open(T.header_path()).read(), 'run `python oracle/mc_tables.py`'


def test_table_basic_properties():
    assert T.MAX_TRIS == 5
    assert T.TRI_COUNT[0] == 0 and T.TRI_COUNT[255] == 0
    for c in range(256):
        cut = 0
        for e in range(12):
            a, off = T.edge_owner(e)
            c0 = off[0] | off[1] << 1 | off[2] << 2
            c1 = c0 | (1 << a)
            if ((c >> c0) & 1) != ((c >> c1) & 1):
                cut |= 1 << e
        assert int(T.EDGE_MASK[c]) == cut, 'case %d must use exactly its cut edges' % c
        loops = T.case_loops(c)
        assert sum(len(l) for l in loops) == bin(cut).count('1')
        assert int(T.TRI_COUNT[c]) == sum(len(l) - 2 for l in loops)


@pytest.mark.parametrize('n', [16, 33])
def test_sphere_is_closed_oriented_manifold(n):
    x, y, z = lattice(n)
    vol = (0.7 - np.sqrt(x * x + y * y + z * z)).astype(np.float32)  # inside higher ("ascent")
    v, f, case = mc.marching_cubes(vol, level=0.0)
    s = mc.mesh_stats(v, f)
    assert s['closed'] and s['oriented'] and s['all_vertices_used']
    assert s['euler'] == 2
    h = 2.0 / (n - 1)
    true_vol = 4 / 3 * np.pi * 0.7 ** 3 / h ** 3
    assert s['signed_volume'] > 0, 'normals must point out of the high-valued region'
    assert abs(s['signed_volume'] - true_vol) / true_vol < 0.05
    r = np.linalg.norm(v * h - 1.0, axis=1)
    assert np.abs(r - 0.7).max() < 0.6 * h * h + 1e-3


def test_torus_and_two_blobs_topology():
    x, y, z = lattice(40)
    tor = (0.25 - np.sqrt((np.sqrt(x * x + y * y) - 0.6) ** 2 + z * z)).astype(np.float32)
    v, f, _ = mc.marching_cubes(tor, level=0.0)
    s = mc.mesh_stats(v, f)
    assert s['closed'] and s['oriented'] and s['euler'] == 0
    two = np.maximum(0.3 - np.sqrt((x - 0.5) ** 2 + y * y + z * z), 0.3 - np.sqrt((x + 0.5) ** 2 + y * y + z * z))
    v, f, _ = mc.marching_cubes(two.astype(np.float32), level=0.0)
    s = mc.mesh_stats(v, f)
    assert s['closed'] and s['oriented'] and s['euler'] == 4


def test_random_field_is_watertight_inside():
    """ambiguous faces everywhere: every edge not on the volume boundary is shared by exactly 2 faces."""
    rs = np.random.RandomState(0)
    vol = rs.randn(14, 15, 16).astype(np.float32)
    vol = np.pad(vol, 1, constant_values=-10.0)  # close the surface
    v, f, case = mc.marching_cubes(vol, level=0.0)
    s = mc.mesh_stats(v, f)
    assert s['closed'] and s['oriented'] and s['all_vertices_used']
    assert len(np.unique(case)) > 200


def test_level_default_and_vertex_interpolation():
    vol = np.zeros((3, 3, 3), dtype=np.float32)
    vol[1, 1, 1] = 4.0
    assert mc.iso_level(vol) == np.float32(2.0)
    v, f, _ = mc.marching_cubes(vol)
    s = mc.mesh_stats(v, f)
    assert s['V'] == 6 and s['F'] == 8 and s['closed'] and s['euler'] == 2 and s['signed_volume'] > 0
    assert np.allclose(np.sort(np.abs(v - 1.0).max(1)), 0.5, atol=1e-6)
    # plane z = 0.25 between samples: exact linear interpolation
    vol = np.broadcast_to(np.array([1.0, 0.5, -1.5, -2.0], dtype=np.float32), (4, 4, 4)).copy()
    v, f, _ = mc.marching_cubes(vol, level=0.0)
    assert np.allclose(v[:, 2], 1.25, atol=1e-6) and len(v) == 16 and len(f) == 18


def test_empty_and_degenerate():
    v, f, _ = mc.marching_cubes(np.zeros((5, 5, 5), dtype=np.float32))
    assert v.shape == (0, 3) and f.shape == (0, 3)
    v, f, _ = mc.marching_cubes(np.arange(8, dtype=np.float32).reshape(2, 2, 2))
    assert len(f) >= 1


def _edge_value_fields():
    """ties (integers at levels 0 and 1), -0.0 / +0.0 at levels +0.0 and -0.0, and +-inf samples at level 0; each
    padded with a value below every level so that the surface is closed"""
    rs = np.random.RandomState(1)
    zeros = np.array([-1.0, -0.0, 0.0, 1.0], dtype=np.float32)
    inf = rs.randn(12, 13, 14).astype(np.float32)
    inf[rs.rand(*inf.shape) < 0.15] = np.inf
    inf[rs.rand(*inf.shape) < 0.15] = -np.inf
    ties = rs.randint(-2, 3, size=(12, 13, 14)).astype(np.float32)
    signed = zeros[rs.randint(0, 4, size=(12, 13, 14))]
    out = [(ties, 0.0), (ties, 1.0), (signed, 0.0), (signed, -0.0), (inf, 0.0)]
    return [(np.pad(v, 1, constant_values=-10.0), lv) for v, lv in out]


@pytest.mark.parametrize('case', range(5))
def test_edge_values_give_closed_oriented_manifold(case):
    vol, level = _edge_value_fields()[case]
    v, f, _ = mc.marching_cubes(vol, level=level)
    s = mc.mesh_stats(v, f)
    assert s['F'] > 100 and s['closed'] and s['oriented'] and s['all_vertices_used']
    if case in (2, 3):                   # levels +0.0 and -0.0 select the same corners
        v2, f2, _ = mc.marching_cubes(vol, level=-level)
        assert np.array_equal(f, f2) and np.array_equal(v, v2)


def test_unit_extent_has_vertices_and_no_faces():
    rs = np.random.RandomState(2)
    for shape in [(1, 12, 13), (12, 1, 13), (12, 13, 1), (1, 1, 16)]:
        v, f, case = mc.marching_cubes(rs.randn(*shape).astype(np.float32), level=0.0)
        assert len(v) > 0 and f.shape == (0, 3) and case.size == 0


def test_rescale_matches_reference_formula():
    v = np.array([[0, 64, 128]], dtype=np.float32)
    out = mc.rescale_vertices(v, 128)
    assert np.allclose(out, [[-0.55, 0.0, 0.55]])


# ------------------------------------------------------------------------------------------------
# Cross-check against scikit-image where it is importable (SURVEY §8c: "if skimage turns out to be
# importable, add a cross-check there; do not assume it").  It is NOT installed in the build
# container nor on the GPU image, so this is skipped there and Lewiner parity stays UNPINNED; on a
# machine that has it, this is the test that pins (or refutes) it.
# ------------------------------------------------------------------------------------------------
import importlib.util

_HAS_SKIMAGE = importlib.util.find_spec('skimage') is not None


def _canonical(verts, faces, decimals=4):
    """order-independent form: vertices rounded and sorted; faces as sorted rows of rotation-normalised
    triples of the vertices' sorted ranks."""
    v = np.round(np.asarray(verts, dtype=np.float64), decimals)
    order = np.lexsort((v[:, 2], v[:, 1], v[:, 0]))
    rank = np.empty(len(v), dtype=np.int64)
    rank[order] = np.arange(len(v))
    f = rank[np.asarray(faces, dtype=np.int64)]
    r = np.argmin(f, axis=1)
    f = np.stack([f[np.arange(len(f)), (r + s) % 3] for s in range(3)], 1)   # rotate the smallest id first (keeps winding)
    return v[order], f[np.lexsort((f[:, 2], f[:, 1], f[:, 0]))]


@pytest.mark.skipif(not _HAS_SKIMAGE, reason='scikit-image not installed: Lewiner parity stays unpinned')
@pytest.mark.parametrize('name', ['sphere', 'two_blobs', 'noise'])
def test_cross_check_against_skimage(name):
    from skimage import measure
    x, y, z = lattice(40)
    if name == 'sphere':
        vol = (0.7 - np.sqrt(x * x + y * y + z * z)).astype(np.float32)
    elif name == 'two_blobs':
        vol = np.maximum(0.35 - np.sqrt((x - 0.45) ** 2 + y * y + z * z),
                         0.35 - np.sqrt((x + 0.45) ** 2 + y * y + z * z)).astype(np.float32)
    else:
        vol = np.random.RandomState(0).randn(18, 19, 20).astype(np.float32)
    sv, sf, _, _ = measure.marching_cubes(vol, gradient_direction='ascent')   # the reference's call, generation.py:270
    v, f, _ = mc.marching_cubes(vol, None)
    cv, cf = _canonical(v, f)
    csv, csf = _canonical(sv, sf)
    # table-independent parts must agree exactly: one vertex per cut edge at the same place
    # (Lewiner may add interior vertices on ambiguous cells of the noise field only)
    if name != 'noise':
        assert cv.shape == csv.shape and np.abs(cv - csv).max() <= 1e-4
        assert np.array_equal(cf, csf), 'triangulation differs from skimage on an unambiguous surface'
    else:
        assert len(csv) >= len(cv)
        same = len(csf) == len(cf) and np.array_equal(cf, csf)
        if not same:
            pytest.xfail('ambiguous cases (3,4,6,7,10,12,13) are triangulated differently from skimage Lewiner: '
                         '%d vs %d faces' % (len(cf), len(csf)))
