"""CPU: the float64 decoder reference (oracle.convonet.decoder_forward(dtype=torch.float64)) that the GPU
configuration sweep (tests/test_configs_gpu.py) measures the kernels against, and the power of the
element-wise gradient check that sweep uses.

The float64 path keeps the reference's fp32 query normalisation and grid coordinates (they decide which cells
are read) and runs everything after them in float64, so it must agree with the fp32 oracle — which
test_oracle_golden.py pins to the reference's own outputs — to fp32 rounding."""
import pytest
import torch

from oracle import convonet as oc
from util import load, weights, decoder_feats, COMBOS, close, rs_randn, grad_excess, kink_mask
from test_oracle_golden import GRAD_CASES, rel_fro

F64 = torch.float64


@pytest.mark.parametrize('tag', ['relu', 'leaky'])
def test_float64_forward_matches_fp32_oracle(tag):
    g = load('decoder_%s.npz' % tag)
    W = weights(g)
    W64 = {k: v.double() for k, v in W.items()}
    feats = decoder_feats(g)
    p, c_img = torch.from_numpy(g['p']), torch.from_numpy(g['c_img'])
    leaky = tag == 'leaky'
    worst = 0.0
    with torch.no_grad():
        for keys in COMBOS.values():
            cp = {k: feats[k] for k in keys}
            for smode in ('bilinear', 'nearest'):
                for mode in ('forward', 'img') + (() if leaky else ('contact',)):
                    kw = dict(c_img=c_img if mode == 'img' else None, leaky=leaky, sample_mode=smode)
                    a = oc.decoder_forward(p, cp, W, mode, **kw)
                    b = oc.decoder_forward(p, cp, W64, mode, dtype=F64, **kw)
                    a, b = (a, b) if mode != 'contact' else (torch.stack(a), torch.stack(b))
                    assert b.dtype == F64
                    worst = max(worst, close(a.numpy(), b.numpy()))
    assert 0 < worst < 1e-5, worst     # fp32 rounding, and no more


def test_preacts_are_the_relu_inputs():
    """return_preacts hands back what the activations see: recomputing the head from n_last gives the output,
    and one entry per block for m_i and h_i."""
    g = load('decoder_relu.npz')
    W64 = {k: v.double() for k, v in weights(g).items()}
    feats = decoder_feats(g)
    p = torch.from_numpy(g['p'])
    out, pre = oc.decoder_forward(p, {'grid': feats['grid']}, W64, 'forward', dtype=F64, return_preacts=True)
    assert len(pre['m']) == len(pre['h']) == 5
    head = torch.nn.functional.linear(torch.relu(pre['n_last']), W64['fc_out.weight'], W64['fc_out.bias'])
    assert torch.equal(head.squeeze(-1), out)
    out32 = oc.decoder_forward(p, {'grid': feats['grid']}, weights(g), 'forward')
    out32p, _ = oc.decoder_forward(p, {'grid': feats['grid']}, weights(g), 'forward', return_preacts=True)
    assert torch.equal(out32, out32p)    # spelling the blocks out does not change fp32 results


def float64_grads(g, tag, leaky, keys, mode, smode, r=None, r2=None):
    """autograd through the float64 reference on the decoder_grads.npz case `tag`."""
    W = {k[len(tag) + 3:]: torch.from_numpy(v).double().requires_grad_(True)
         for k, v in g.items() if k.startswith(tag + '.w.')}
    feats = decoder_feats(g)
    cp = {k: feats[k].double().requires_grad_(True) for k in keys}
    p = torch.from_numpy(g['p'])
    c_img = torch.from_numpy(g['c_img']).double().requires_grad_(True)
    r = torch.from_numpy(g['r']).double() if r is None else r
    r2 = torch.from_numpy(g['r2']).double() if r2 is None else r2
    if mode == 'contact':
        (o, c_), pre = oc.decoder_forward(p, cp, W, 'contact', leaky=leaky, sample_mode=smode, dtype=F64,
                                          return_preacts=True)
        loss = (o * r).sum() + (c_ * r2).sum()
    else:
        o, pre = oc.decoder_forward(p, cp, W, mode, c_img=c_img if mode == 'img' else None, leaky=leaky,
                                    sample_mode=smode, dtype=F64, return_preacts=True)
        loss = (o * r).sum()
    loss.backward()
    out = {'dw.' + k: v.grad for k, v in W.items() if v.grad is not None}
    out.update({'dfeat.' + k: v.grad for k, v in cp.items()})
    if mode == 'img':
        out['dc_img'] = c_img.grad
    return loss.item(), out, pre


@pytest.mark.parametrize('case', GRAD_CASES, ids=[c[0] for c in GRAD_CASES])
def test_float64_gradients_match_reference(case):
    """autograd through the float64 reference == the reference modules' fp32 autograd (decoder_grads.npz)."""
    tag, leaky, keys, mode, smode = case
    g = load('decoder_grads.npz')
    loss, grads, _ = float64_grads(g, tag, leaky, keys, mode, smode)
    assert abs(loss - float(g[tag + '.loss'])) <= 1e-5 * max(1.0, abs(float(g[tag + '.loss'])))
    assert sorted(grads) == sorted(k[len(tag) + 1:] for k in g if k.startswith(tag + '.d'))
    for k, v in grads.items():
        assert rel_fro(v.numpy(), g['%s.%s' % (tag, k)]) < 1e-5, k


def test_elementwise_check_sees_one_missing_query():
    """The bound the GPU backward sweep applies, |got - ref| <= 1e-5 max|ref| + 1e-4 |ref| per element, rejects a
    gradient that lacks the contribution of ONE query (here one with a small incoming gradient) out of 3072, which
    the relative Frobenius error <= 1e-4 of the older tests accepts."""
    g = load('decoder_relu.npz')
    W0 = {k: v.double() for k, v in weights(g).items()}
    feats = decoder_feats(g)
    p, c_img = torch.from_numpy(g['p']), torch.from_numpy(g['c_img']).double()
    B, N = p.shape[:2]
    assert B * N == 3072
    q = (1, 777)
    r = torch.from_numpy(rs_randn(40, B, N)).double()
    r[q] = 1e-3 * r.abs().mean()

    def grads(r):
        W = {k: v.clone().requires_grad_(True) for k, v in W0.items()}
        cp = {'grid': feats['grid'].double().requires_grad_(True)}
        ci = c_img.clone().requires_grad_(True)
        o, pre = oc.decoder_forward(p, cp, W, 'img', c_img=ci, dtype=F64, return_preacts=True)
        (o * r).sum().backward()
        out = {k: v.grad.numpy() for k, v in W.items() if v.grad is not None}
        out.update({'dfeat.grid': cp['grid'].grad.numpy(), 'dc_img': ci.grad.numpy()})
        return out, pre

    ref, pre = grads(r)
    assert not kink_mask(pre)[q]                             # an ordinary query, not one near a ReLU kink
    r_drop = r.clone()
    r_drop[q] = 0
    got, _ = grads(r_drop)
    assert all(rel_fro(got[k], ref[k]) < 1e-4 for k in ref)
    assert max(grad_excess(got[k], ref[k], 1e-5, 1e-4) for k in ref) > 1
    for k in ref:                                            # and it accepts the reference itself
        assert grad_excess(ref[k].copy(), ref[k], 1e-5, 1e-4) == 0


def test_kink_mask_marks_only_near_zero_inputs():
    t = torch.tensor([[[1.0, -2.0, 3e-6], [1.0, -2.0, 4.0]]], dtype=F64)
    m = kink_mask({'m': [t], 'h': [], 'n_last': torch.ones(1, 2, 3, dtype=F64)})
    assert m.tolist() == [[True, False]]
