"""GPU: the fused decoder (every kernel variant, forward and backward) and the PointNet encoder at every depth and
configuration their modules accept, against the float64 reference (oracle.convonet.decoder_forward(dtype=
torch.float64), pinned by tests/test_reference64_cpu.py).

Forward: err = |got - ref| / max(1, |ref|) per output.  Per case and variant class its max is bounded, and so is
its mean where the case has at least MEAN_MIN_OUTPUTS outputs (the mean of one output is its max).  A bound is
the class figure below or FLOOR x the fp32 oracle's own deviation from float64 on the same case, whichever is
larger: exact fp32 arithmetic cannot be closer to float64 than fp32 rounding allows, and through 5-7 blocks of
32-wide layers the fp32 oracle itself is up to 7.5e-7 (mean 1.1e-7) away.
  class                                   bound max / mean    measured on a B200 (1000 W), max / mean
  variants 0, 1 (exact fp32 SIMT)         1e-6 / 1e-7         1.8e-6 / 2.4e-7  (7 blocks; fp32 oracle 7.5e-7 / 1.1e-7)
  variants 2, 5 (tcgen05 3xTF32)          4e-6 / 4e-7         1.8e-6 / 2.6e-7  (6-7 blocks run variant 1)
  variants 4, 6, 7 (TF32 + BF16 terms)    1e-5 / 1e-6         4.9e-6 / 7.7e-7
  variant 3 (single TF32 product, debug)  5e-3 / 5e-4         1.9e-3 / 3.8e-4
With one block matrix's lo / BF16 correction zeroed (test_accuracy_check_sees_one_matrix_losing_its_correction)
variants 5, 7 measure 1.2e-4 / 1.5e-5 and variant 6 2.5e-4 / 3.4e-5.

Backward: per gradient tensor, element-wise |got - ref| <= a * max|ref| + r * |ref| with a = 1e-5, r = 1e-4;
queries with a ReLU input within 1e-5 of its layer's scale get zero incoming gradient on both sides.  Largest
share of that bound used on a B200: parameter gradients 0.09, feature gradients 0.021, c_img 0.0095."""
import numpy as np
import pytest
import torch

from util import rs_randn, close, randomise, synthetic_cloud, voxel_coord, lattice_node, grad_excess, kink_mask

pytestmark = pytest.mark.gpu
F64 = torch.float64

# variant class -> (max bound, mean bound) on |got - ref| / max(1, |ref|)
BOUNDS = {0: (1e-6, 1e-7), 1: (1e-6, 1e-7), 2: (4e-6, 4e-7), 5: (4e-6, 4e-7),
          4: (1e-5, 1e-6), 6: (1e-5, 1e-6), 7: (1e-5, 1e-6), 3: (5e-3, 5e-4)}
FLOOR = 4                 # x the fp32 oracle's deviation from float64 (see the module docstring)
MEAN_MIN_OUTPUTS = 1000
GRAD_A, GRAD_R = 1e-5, 1e-4
KEYS = {'grid': ('grid',), 'xz': ('xz',), 'xy+yz': ('xy', 'yz'), 'all': ('grid', 'xz', 'xy', 'yz')}


class Case:
    def __init__(self, nb, c_dim, keys='grid', Rg=17, Rp=9, smode='bilinear', div='cuda', mode='forward',
                 leaky=False, B=3, N=1237):
        self.nb, self.c_dim, self.keys, self.Rg, self.Rp = nb, c_dim, keys, Rg, Rp
        self.smode, self.div, self.mode, self.leaky, self.B, self.N = smode, div, mode, leaky, B, N

    def __repr__(self):
        return 'nb%d_c%d_%s_g%dp%d_%s_%s_%s%s_B%dN%d' % (self.nb, self.c_dim, self.keys, self.Rg, self.Rp,
                                                       self.smode[:4], self.div, self.mode,
                                                       '_leaky' if self.leaky else '', self.B, self.N)


C = Case
# every n_blocks 0-7 with both c_dim; keys grid / xz / xy+yz / all; Rg != Rp and R = 2; both sample modes, both
# divisions, the three heads, leaky on and off, B = 1 and 3, N = 1 and ragged
FWD_CASES = [
    C(0, 0), C(0, 32, 'all', mode='img'), C(0, 32, 'grid', mode='contact', B=1, N=1),
    C(1, 0, mode='img', leaky=True), C(1, 32, 'xz', div='true'), C(1, 32, 'all', 2, 2, mode='contact'),
    C(2, 0, smode='nearest', mode='contact'), C(2, 32, 'xy+yz', smode='nearest', mode='img'),
    C(2, 32, 'grid', 2, 2, leaky=True, B=1),
    C(3, 0, div='true', B=1, N=1), C(3, 32, 'all', smode='nearest', div='true', leaky=True),
    C(3, 32, 'xz', Rp=2, mode='img'),
    C(4, 0, mode='img'), C(4, 32, 'grid', mode='contact', leaky=True), C(4, 32, 'xy+yz', Rp=17, B=1),
    C(5, 0, leaky=True), C(5, 32, 'all', mode='img', div='true'), C(5, 32, 'grid', smode='nearest', mode='contact'),
    C(5, 32, 'xz', B=1, N=1, mode='img'),
    C(6, 0, mode='contact', B=1), C(6, 32, 'all'), C(6, 32, 'grid', mode='img', leaky=True),
    C(6, 32, 'xy+yz', smode='nearest', div='true', mode='contact'),
    C(7, 0, smode='nearest', mode='img'), C(7, 32, 'all', mode='contact'), C(7, 32, 'grid', div='true', leaky=True),
    C(7, 32, 'xz', 2, 2, mode='img', B=1), C(7, 32, 'xy+yz', smode='nearest', B=1, N=1),
]
DENSE_CASES = [C(5, 32, 'grid', B=1), C(7, 32, 'all', B=1, leaky=True), C(2, 32, 'xz', smode='nearest', B=1)]


# --------------------------------------------------------------------------- inputs
def make_decoder(case, seed=0):
    from vtaco_b200.conv_onet.models import decoder_dict
    dec = decoder_dict['simple_local'](dim=3, c_dim=case.c_dim, hidden_size=32, n_blocks=case.nb, leaky=case.leaky,
                                       sample_mode=case.smode, padding=0.1, with_contact=True)
    randomise(dec, 100 + seed)
    dec.division = case.div
    return dec.cuda()


def make_feats(case, seed=0):
    f = {}
    for i, k in enumerate(KEYS[case.keys]):
        R = case.Rg if k == 'grid' else case.Rp
        shape = (case.B, 32) + (R,) * (3 if k == 'grid' else 2)
        f[k] = torch.from_numpy(rs_randn(200 + 10 * seed + i, *shape))
    return f


def tie_free(p, case):
    """nearest mode: False where any voxel coordinate lies within 1e-4 of a .5 tie (rounding decides the cell)."""
    ok = np.ones(p.shape[:-1], dtype=bool)
    if case.smode != 'nearest':
        return ok
    for R, three_d in ((case.Rg, True), (case.Rp, False)):
        t = voxel_coord(p, R, three_d, case.div)
        ok &= (np.abs(t - np.floor(t) - 0.5) > 1e-4).all(-1)
    return ok


def make_queries(case, seed=0):
    """(B, N, 3) fp32: points on the clamp boundary +-0.55 and outside it (+-0.6), points on the fp32 lattice nodes
    of the grid and of the planes (tap weights exactly 0 / 1; the top node R-1 as close as the clamp allows),
    then uniform +-0.6."""
    rs = np.random.RandomState(300 + seed)
    v = np.array([-0.6, -0.55, 0.0, 0.55, 0.6], dtype=np.float32)
    special = [np.stack(np.meshgrid(v, v, v, indexing='ij'), -1).reshape(-1, 3)]
    for R, three_d in ((case.Rg, True), (case.Rp, False)):
        nodes = np.array([lattice_node(k, R, three_d, case.div) for k in range(R)], dtype=np.float32)
        idx = rs.randint(0, R, size=(3 * R, 3))
        idx[:R, 0] = np.arange(R)            # every node on some axis, the last cell's edge included
        idx[:3, :] = R - 1
        special.append(nodes[idx])
    special = np.concatenate(special).astype(np.float32)
    out = np.empty((case.B, case.N, 3), dtype=np.float32)
    for b in range(case.B):
        pool = np.concatenate([special[rs.permutation(len(special))],
                               rs.uniform(-0.6, 0.6, size=(case.N + 64, 3)).astype(np.float32)])
        out[b] = pool[tie_free(pool, case)][:case.N]
    return torch.from_numpy(out)


def reference(case, dec, p, feats, c_img, **kw):
    from oracle import convonet as oc
    W = {k: v.detach().cpu().double() for k, v in dec.state_dict().items()}
    return oc.decoder_forward(p, feats, W, case.mode, c_img=c_img, n_blocks=case.nb, leaky=case.leaky,
                              sample_mode=case.smode, c_dim=case.c_dim, cuda_division=(case.div == 'cuda'),
                              dtype=F64, **kw)


def run(dec, case, p, feats, c_img):
    with torch.no_grad():
        if case.mode == 'img':
            return (dec.forward_img(p, feats, c_img),)
        if case.mode == 'contact':
            return dec.forward_contact(p, feats)
        return (dec(p, feats),)


def errs(got, ref):
    got = torch.cat([g.reshape(-1).double().cpu() for g in got])
    ref = torch.cat([r.reshape(-1) for r in ref])
    e = ((got - ref).abs() / ref.abs().clamp(min=1.0)).numpy()
    return float(e.max()), float(e.mean())


def fp32_floor(case, dec, p, feats, c_img):
    """(max, mean) error of the fp32 oracle against the float64 reference on this case."""
    from oracle import convonet as oc
    W = {k: v.detach().cpu() for k, v in dec.state_dict().items()}
    ref = reference(case, dec, p, feats, c_img)
    r32 = oc.decoder_forward(p, feats, W, case.mode, c_img=c_img, n_blocks=case.nb, leaky=case.leaky,
                             sample_mode=case.smode, c_dim=case.c_dim, cuda_division=(case.div == 'cuda'))
    as_t = lambda x: x if isinstance(x, tuple) else (x,)  # noqa: E731
    return errs(as_t(r32), as_t(ref))


def within(v, mx, mean, n_out, floor):
    ok = mx <= max(BOUNDS[v][0], FLOOR * floor[0])
    if n_out >= MEAN_MIN_OUTPUTS:
        ok = ok and mean <= max(BOUNDS[v][1], FLOOR * floor[1])
    return ok


def inputs(case):
    dec = make_decoder(case)
    feats = make_feats(case)
    p = make_queries(case)
    c_img = torch.from_numpy(rs_randn(400, case.B, case.N, case.c_dim)) if case.mode == 'img' else None
    ref = reference(case, dec, p, feats, c_img)
    ref = ref if isinstance(ref, tuple) else (ref,)
    ref = (ref, fp32_floor(case, dec, p, feats, c_img))
    fc = {k: v.cuda() for k, v in feats.items()}
    return dec, p.cuda(), fc, (c_img.cuda() if c_img is not None else None), ref


def check_variants(dec, case, p, fc, ci, ref, variants=range(8)):
    ref, floor = ref
    n_out = sum(r.numel() for r in ref)
    failed = []
    for v in variants:
        dec.kernel_variant = v
        mx, mean = errs(run(dec, case, p, fc, ci), ref)
        print('fwd %-50s variant %d  max %.3e  mean %.3e  (fp32 oracle %.1e / %.1e)' % (case, v, mx, mean, *floor))
        if not within(v, mx, mean, n_out, floor):
            failed.append((v, mx, mean))
    return failed


# --------------------------------------------------------------------------- forward sweep
@pytest.mark.parametrize('case', FWD_CASES, ids=repr)
def test_forward_every_variant_vs_float64(case):
    dec, p, fc, ci, ref = inputs(case)
    assert check_variants(dec, case, p, fc, ci, ref) == []


@pytest.mark.parametrize('case', DENSE_CASES, ids=repr)
def test_forward_dense_odd_lattice_vs_float64(case):
    """forward_dense at nx = 37 (partial bricks on every axis) against the reference at dense_grid_points(37)."""
    from oracle import convonet as oc
    dec = make_decoder(case)
    feats = make_feats(case)
    nx = 37
    pts = oc.dense_grid_points(nx)[None]
    ref = reference(case, dec, pts, feats, None)
    floor = fp32_floor(case, dec, pts, feats, None)
    fc = {k: v.cuda() for k, v in feats.items()}
    failed = []
    for v in range(8):
        dec.kernel_variant = v
        with torch.no_grad():
            got = dec.forward_dense(fc, nx)
        mx, mean = errs((got,), (ref,))
        print('dense %-48s variant %d  max %.3e  mean %.3e' % (case, v, mx, mean))
        if not within(v, mx, mean, ref.numel(), floor):
            failed.append((v, mx, mean))
    assert failed == []


@pytest.mark.parametrize('variant', [7, 5, 6])
def test_accuracy_check_sees_one_matrix_losing_its_correction(variant):
    """Zeroing the lo (pack modes 0, 2) or BF16 correction (mode 1) sub-block of ONE block matrix of the cached
    tcgen05 operand buffer — one layer computed with the TF32 hi product only — must fail the bounds above."""
    from vtaco_b200 import _abi
    case = C(5, 32, 'all', mode='img')
    dec, p, fc, ci, ref = inputs(case)
    dec.eval()
    assert check_variants(dec, case, p, fc, ci, ref, [variant]) == []
    mode = _abi.dec_tc_mode(variant)
    wtc = dec._packed_weights_tc(mode)
    m = 3 * 2 + 1                                 # blocks[2].fc_0
    off = _abi.dec_tc_mat(mode, m) + _abi.DEC_TC_SUB_LO
    with torch.no_grad():
        wtc[off:off + 1024].zero_()
    assert dec._packed_weights_tc(mode) is wtc    # the launch reads the altered buffer
    assert check_variants(dec, case, p, fc, ci, ref, [variant]) != []
    dec.invalidate()
    assert check_variants(dec, case, p, fc, ci, ref, [variant]) == []


def test_eight_blocks_is_not_supported():
    """No forward kernel holds 8 blocks in shared memory (VTACO_MAX_BLOCKS = 7): the module says so."""
    case = C(8, 32, B=1, N=5)
    dec = make_decoder(case)
    p = make_queries(case).cuda()
    fc = {k: v.cuda() for k, v in make_feats(case).items()}
    with pytest.raises(NotImplementedError):
        with torch.no_grad():
            dec(p, fc)


# --------------------------------------------------------------------------- backward sweep
BWD_CASES = [
    C(0, 0, mode='img'), C(0, 32, 'all', mode='contact', N=700), C(0, 32, 'grid', smode='nearest'),
    C(1, 32, 'xy+yz', mode='img', N=701), C(1, 0, mode='contact', leaky=True),
    C(2, 32, 'grid', smode='nearest', mode='img'), C(2, 32, 'xz', Rp=2),
    C(3, 32, 'all', mode='contact', leaky=True), C(3, 0, smode='nearest', N=301),
    C(7, 32, 'xy+yz', mode='img'), C(7, 32, 'grid', smode='nearest', mode='contact', N=515),
]
CONTACT_ONLY = {repr(C(0, 32, 'all', mode='contact', N=700)), repr(C(7, 32, 'grid', smode='nearest',
                                                                       mode='contact', N=515))}


@pytest.mark.parametrize('case', BWD_CASES, ids=repr)
def test_backward_vs_float64_autograd(case):
    assert case.div == 'cuda'
    contact_only = repr(case) in CONTACT_ONLY
    dec = make_decoder(case).train()
    feats = make_feats(case)
    p = make_queries(case)
    c_img = torch.from_numpy(rs_randn(400, case.B, case.N, case.c_dim)) if case.mode == 'img' else None
    # float64 reference: parameters, features and c_img as float64 leaves
    W = {k: v.detach().cpu().double().requires_grad_(True) for k, v in dec.state_dict().items()}
    f64 = {k: v.double().requires_grad_(True) for k, v in feats.items()}
    ci64 = c_img.double().requires_grad_(True) if c_img is not None else None
    from oracle import convonet as oc
    out, pre = oc.decoder_forward(p, f64, W, case.mode, c_img=ci64, n_blocks=case.nb, leaky=case.leaky,
                                  sample_mode=case.smode, c_dim=case.c_dim, cuda_division=True, dtype=F64,
                                  return_preacts=True)
    keep = ~kink_mask(pre)
    r = torch.from_numpy(rs_randn(500, case.B, case.N)).double() * keep
    r2 = torch.from_numpy(rs_randn(501, case.B, case.N)).double() * keep

    def loss_of(o):
        if case.mode != 'contact':
            return (o * r.to(o)).sum()
        if contact_only:
            return (o[1] * r2.to(o[1])).sum()
        return (o[0] * r.to(o[0])).sum() + (o[1] * r2.to(o[1])).sum()

    loss_of(out).backward()
    cp = {k: v.cuda().requires_grad_(True) for k, v in feats.items()}
    ci = c_img.cuda().requires_grad_(True) if c_img is not None else None
    pc = p.cuda()
    if case.mode == 'img':
        o = dec.forward_img(pc, cp, ci)
    elif case.mode == 'contact':
        o = dec.forward_contact(pc, cp)
    else:
        o = dec(pc, cp)
    loss_of(o).backward()
    pairs = []
    for n, prm in dec.named_parameters():
        ref = W[n].grad
        if ref is None:       # unused by this loss: the kernel writes nothing or zeros
            assert prm.grad is None or not prm.grad.any(), n
            continue
        assert prm.grad is not None, n
        pairs.append(('dw.' + n, prm.grad, ref))
    for k in feats:
        ref = f64[k].grad if f64[k].grad is not None else torch.zeros_like(f64[k])
        got = cp[k].grad if cp[k].grad is not None else torch.zeros_like(cp[k])
        pairs.append(('dfeat.' + k, got, ref))
    if ci is not None and case.c_dim:
        pairs.append(('dc_img', ci.grad, ci64.grad))
    worst = {}
    for name, got, ref in pairs:
        assert tuple(got.shape) == tuple(ref.shape), name
        x = grad_excess(got.detach().cpu().numpy(), ref.numpy(), GRAD_A, GRAD_R)
        cls = name.split('.')[0]
        worst[cls] = max(worst.get(cls, 0.0), x)
        print('bwd %-50s %-28s excess %.3f' % (case, name, x))
        assert x <= 1, (name, x)
    print('bwd %-50s masked %d / %d queries, worst %s' % (case, int((~keep).sum()), keep.numel(), worst))


# --------------------------------------------------------------------------- encoder depth sweep
ENC_TYPES = {'grid': (dict(plane_type='grid', grid_resolution=16), dict(plane_type='grid', reso_grid=16)),
             'tri': (dict(plane_type=['xz', 'xy', 'yz'], plane_resolution=16),
                     dict(plane_type=['xz', 'xy', 'yz'], reso_plane=16)),
             'all': (dict(plane_type=['xz', 'xy', 'yz', 'grid'], plane_resolution=8, grid_resolution=8),
                     dict(plane_type=['xz', 'xy', 'yz', 'grid'], reso_plane=8, reso_grid=8))}


def make_encoder(nb, tag, pool, seed=0):
    from vtaco_b200.encoder import encoder_dict
    ctor, okw = ENC_TYPES[tag]
    enc = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, n_blocks=nb,
                                              scatter_type=pool, **ctor)
    randomise(enc, 600 + seed)
    enc.division = 'true'
    return enc.cuda(), dict(okw, scatter_type=pool, n_blocks=nb)


@pytest.mark.parametrize('pool', ['max', 'mean'])
@pytest.mark.parametrize('tag', ['grid', 'tri', 'all'])
@pytest.mark.parametrize('nb', [1, 2, 3, 4, 6, 7])
def test_encoder_depth_forward(nb, tag, pool):
    """Depths that put every phase of the encoder's pool-level (% 3) and net-buffer (& 1) rotation last."""
    from oracle import convonet as oc
    enc, okw = make_encoder(nb, tag, pool)
    p = torch.from_numpy(np.stack([synthetic_cloud(700 + b, 1500)[0] for b in range(2)]))
    W = {k: v.cpu() for k, v in enc.state_dict().items()}
    with torch.no_grad():
        ref, ref_idx, inter = oc.encoder_pointnet(p, W, return_intermediates=True, **okw)
        fea, code, idx = enc.eval().pointnet_features(p.cuda(), return_code=True, return_index=True)
    for k in ref_idx:
        assert torch.equal(idx[k].cpu().long(), ref_idx[k]), k
    assert close(code.cpu().numpy(), inter['c'].numpy()) < 1e-4
    for k in ref:
        assert close(fea[k].contiguous().cpu().numpy(), ref[k].numpy()) < 1e-4, k


@pytest.mark.parametrize('tag,pool', [('all', 'max'), ('tri', 'mean')])
@pytest.mark.parametrize('nb', [1, 2, 3, 8])
def test_encoder_depth_backward(nb, tag, pool):
    """One pool level per block in the backward: against the oracle's autograd in fp32 and float64, with the
    fp32-vs-float64 disagreement of the oracle itself as the floor (test_encoder_backward_vs_oracle_shipped_cloud)."""
    from oracle import convonet as oc
    from test_oracle_golden import rel_fro
    enc, okw = make_encoder(nb, tag, pool, seed=1)
    p = torch.from_numpy(np.stack([synthetic_cloud(800 + b, 1500)[0] for b in range(2)]))
    ref = {}
    for dt in (torch.float32, torch.float64):
        W = {k: v.detach().cpu().to(dt).requires_grad_(True) for k, v in enc.state_dict().items()}
        fea = oc.encoder_pointnet(p.to(dt), W, **okw)
        rs = {k: torch.from_numpy(rs_randn(900 + i, *v.shape)) for i, (k, v) in enumerate(fea.items())}
        sum((v * rs[k].to(dt)).sum() for k, v in fea.items()).backward()
        ref[dt] = {k: v.grad.double().numpy() for k, v in W.items()}
    out = enc.train()(p.cuda())
    assert list(out.keys()) == list(fea.keys())
    sum((v * rs[k].cuda()).sum() for k, v in out.items()).backward()
    for n, prm in enc.named_parameters():
        floor = rel_fro(ref[torch.float32][n], ref[torch.float64][n])
        err = min(rel_fro(prm.grad.cpu().numpy(), ref[dt][n]) for dt in ref)
        assert err < max(1e-4, 3 * floor), (n, err, floor)
