"""Shared helpers for the tests (fixtures, stable random streams)."""
import os
import numpy as np
import torch

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')


def rs_randn(seed, *shape, scale=1.0):
    return (np.random.RandomState(seed).randn(*shape) * scale).astype(np.float32)


def rs_uniform(seed, lo, hi, *shape):
    return np.random.RandomState(seed).uniform(lo, hi, size=shape).astype(np.float32)


def load(name):
    return dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))


def weights(g, device='cpu'):
    return {k[2:]: torch.from_numpy(v).to(device) for k, v in g.items() if k.startswith('w.')}


def decoder_feats(g, device='cpu'):
    s = g['feat_seeds']
    Rg, Rp = [int(x) for x in g['feat_shapes']]
    B = g['p'].shape[0]
    f = {'grid': rs_randn(int(s[0]), B, 32, Rg, Rg, Rg), 'xz': rs_randn(int(s[1]), B, 32, Rp, Rp),
         'xy': rs_randn(int(s[2]), B, 32, Rp, Rp), 'yz': rs_randn(int(s[3]), B, 32, Rp, Rp)}
    return {k: torch.from_numpy(v).to(device) for k, v in f.items()}


COMBOS = {'grid': ['grid'], 'tri': ['xz', 'xy', 'yz'], 'all': ['grid', 'xz', 'xy', 'yz'], 'xz': ['xz']}


def close(a, b, rtol=1e-4):
    """north_star tolerance: |a-b| <= rtol * max(1, |b|)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    err = np.abs(a - b) / np.maximum(1.0, np.abs(b))
    return float(err.max()) if err.size else 0.0


def synthetic_cloud(seed, n_visual, n_tactile_per_tip=128, n_tips=5):
    rs = np.random.RandomState(seed)
    vis = rs.uniform(-0.5, 0.5, size=(n_visual, 3))
    tips = rs.uniform(-0.35, 0.35, size=(n_tips, 3))
    tac = (tips[:, None, :] + rs.randn(n_tips, n_tactile_per_tip, 3) * 0.01).reshape(-1, 3)
    pts = np.concatenate([vis, tac], 0) + rs.randn(n_visual + n_tips * n_tactile_per_tip, 3) * 0.005
    return pts.astype(np.float32), tips.astype(np.float32)


def randomise(module, seed):
    """the parameter stream of tests/golden/make_golden.py: every parameter (sorted by name) re-drawn from
    RandomState(seed); ResnetBlockFC.fc_1.weight ~ N(0, 0.1^2), the rest uniform(+-1/sqrt(fan_in))."""
    rs = np.random.RandomState(seed)
    with torch.no_grad():
        for name, prm in sorted(module.named_parameters()):
            fan_in = prm.shape[1] if prm.dim() > 1 else prm.shape[0]
            bound = 1.0 / np.sqrt(max(fan_in, 1))
            if name.endswith('fc_1.weight'):
                val = rs.randn(*prm.shape) * 0.1
            else:
                val = rs.uniform(-bound, bound, size=tuple(prm.shape))
            prm.copy_(torch.from_numpy(val.astype(np.float32)))


# --------------------------------------------------------------------------- #
# fp32 query -> voxel coordinate, as the reference (normalize_* then grid_sample's unnormalize) and the
# decoder kernels (common.cuh norm2d / norm3d, decoder_common.cuh unnormalize) compute it
# --------------------------------------------------------------------------- #
def _norm_u(v, three_d, division, padding=0.1):
    v = np.asarray(v, dtype=np.float32)
    d = (1.0 + padding) + (10e-4 if three_d else 10e-6)
    if division == 'cuda':
        u = v * np.float32(1.0 / d)
    else:
        u = v / np.float32(d)
    u = (u + np.float32(0.5)).astype(np.float32)
    u = np.where(u >= 1, np.float32(1 - (10e-4 if three_d else 10e-6)), u)
    return np.where(u < 0, np.float32(0), u).astype(np.float32)


def voxel_coord(v, R, three_d, division):
    """Continuous voxel coordinate in [0, R-1] of fp32 coordinate(s) v along one axis."""
    g = (np.float32(2) * _norm_u(v, three_d, division) - np.float32(1)).astype(np.float32)
    return ((g + np.float32(1)) * np.float32(0.5) * np.float32(R - 1)).astype(np.float32)


def lattice_node(k, R, three_d, division):
    """An fp32 coordinate whose voxel coordinate is exactly the lattice node k (tap weights exactly 0 and 1),
    or the closest one within 64 ulps of the exact preimage."""
    d = (1.0 + 0.1) + (10e-4 if three_d else 10e-6)
    v = np.float32((k / (R - 1) - 0.5) * d)
    best, best_err = v, np.inf
    for s in range(-64, 65):
        c = np.float32(v)
        step = np.float32(np.inf) if s > 0 else np.float32(-np.inf)
        for _ in range(abs(s)):
            c = np.nextafter(c, step)
        err = abs(float(voxel_coord(c, R, three_d, division)) - k)
        if err < best_err:
            best, best_err = c, err
            if err == 0:
                break
    return np.float32(best)


# --------------------------------------------------------------------------- #
# gradient checks
# --------------------------------------------------------------------------- #
def grad_excess(got, ref, a, r):
    """max over elements of |got - ref| / (a * max|ref| + r * |ref|): <= 1 passes the element-wise bound.
    Unlike a relative Frobenius norm, it sees one query's contribution missing from a tensor of thousands."""
    got = np.asarray(got, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    if ref.size == 0:
        return 0.0
    bound = a * np.abs(ref).max() + r * np.abs(ref)
    err = np.abs(got - ref)
    with np.errstate(divide='ignore', invalid='ignore'):
        q = np.where(bound > 0, err / bound, np.where(err > 0, np.inf, 0.0))
    return float(q.max())


def kink_mask(preacts, rel=1e-5):
    """(B, N) bool: queries with any ReLU / LeakyReLU input within rel * (that layer's max |input|) of 0 —
    rounding may put them on either side of the kink, so they are given zero incoming gradient."""
    layers = list(preacts['m']) + list(preacts['h']) + [preacts['n_last']]
    near = None
    for t in layers:
        t = t.detach()
        m = (t.abs() <= rel * t.abs().max()).any(-1)
        near = m if near is None else (near | m)
    return near
