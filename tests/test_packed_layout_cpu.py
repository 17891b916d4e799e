"""CPU: the packed parameter layouts of the fused decoder and the PointNet encoder.

Both models read their weights from one flat fp32 buffer and their backward kernels write the parameter
gradients into a flat buffer with the same offsets.  The expected offsets below are written out from the
layouts include/vtaco_b200.h documents, independently of the constants the package derives them from: the
header macros must equal their Python mirror, the pack descriptors the modules hand to vtaco_pack_linear must
land each parameter where the header says, and the gradient views must be cut from the same places.  The same
goes for the tcgen05 operand buffer the decoder derives from its packed buffer (`weights_tc`)."""
import itertools
import os
import re
import shutil
import subprocess

import pytest
import torch

from vtaco_b200 import _abi
from vtaco_b200.conv_onet.models.decoder import LocalDecoder
from vtaco_b200.encoder.pointnet import LocalPoolPointnet

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
N_BLOCKS = (1, 3, 5)
# (with_contact head, contact output requested)
CONTACT = ((False, False), (True, False), (True, True))


def _decoder_fields(nb, c_dim, contact_head):
    """(name, offset, pack columns (first, count) or (), gradient shape) of every packed decoder field,
    in the order the descriptors are built."""
    f = [('fc_p.weight', 0, (), (32, 3)), ('fc_p.bias', 96, (), (32,)),
         ('fc_p_img.weight', 128, (0, 3), (32, 3)), ('fc_p_img.bias', 224, (), (32,))]
    if c_dim:
        f.append(('fc_p_img.weight', 256, (3, 32), (32, 32)))
    for i in range(nb):
        o = 1280 + 3168 * i
        if c_dim:
            f += [('fc_c.%d.weight' % i, o, (), (32, 32)), ('fc_c.%d.bias' % i, o + 1024, (), (32,))]
        f += [('blocks.%d.fc_0.weight' % i, o + 1056, (), (32, 32)), ('blocks.%d.fc_0.bias' % i, o + 2080, (), (32,)),
              ('blocks.%d.fc_1.weight' % i, o + 2112, (), (32, 32)), ('blocks.%d.fc_1.bias' % i, o + 3136, (), (32,))]
    t = 1280 + 3168 * nb
    f += [('fc_out.weight', t, (), (1, 32)), ('fc_out.bias', t + 64, (), (1,))]
    if contact_head:
        f += [('fc_out_contact.weight', t + 32, (), (1, 32)), ('fc_out_contact.bias', t + 65, (), (1,))]
    return f, t + 68


def _encoder_fields(nb):
    f = [('fc_pos.weight', 0, (), (64, 3)), ('fc_pos.bias', 192, (), (64,))]
    for i in range(nb):
        o = 256 + 5184 * i
        f += [('blocks.%d.fc_0.weight' % i, o, (), (32, 64)), ('blocks.%d.fc_0.bias' % i, o + 2048, (), (32,)),
              ('blocks.%d.fc_1.weight' % i, o + 2080, (), (32, 32)), ('blocks.%d.fc_1.bias' % i, o + 3104, (), (32,)),
              ('blocks.%d.shortcut.weight' % i, o + 3136, (), (32, 64))]
    t = 256 + 5184 * nb
    f += [('fc_c.weight', t, (), (32, 32)), ('fc_c.bias', t + 1024, (), (32,))]
    return f, t + 1056


def _decoder(nb, c_dim, contact_head):
    return LocalDecoder(dim=3, c_dim=c_dim, hidden_size=32, n_blocks=nb, with_contact=contact_head)


def _encoder(nb):
    return LocalPoolPointnet(c_dim=32, dim=3, hidden_dim=32, n_blocks=nb, plane_type='grid', grid_resolution=8)


def _captured_pack(module, monkeypatch):
    """The descriptor entries and destination buffers _packed_weights() passes to pack_linear."""
    calls = []
    monkeypatch.setattr(_abi, 'pack_linear', lambda entries, dst, cache=None: calls.append((list(entries), dst)))
    buf = module._packed_weights()
    assert calls and all(dst is buf for _, dst in calls)
    names = {id(p): n for n, p in module.named_parameters()}
    return [(names[id(e[0])], e[1], tuple(e[2:])) for entries, _ in calls for e in entries], buf


def _is_view_of(t, flat):
    return t.untyped_storage().data_ptr() == flat.untyped_storage().data_ptr()


def _flat(size):
    """arange values in a buffer that does not start at the beginning of its storage"""
    return torch.arange(size + 7, dtype=torch.float32)[7:]


def _check_views(grads, fields, flat):
    for name, off, _, shape in fields:
        t = grads[name]
        assert tuple(t.shape) == shape, name
        assert _is_view_of(t, flat) and t.storage_offset() == flat.storage_offset() + off, name
        n = t.numel()
        assert torch.equal(t, flat[off:off + n].view(shape)), name


# ---------------------------------------------------------------------------------------------------------------
# arguments every function-like layout macro is evaluated at: pack modes 0-2, 0-8 blocks, every decoder variant,
# every matrix index m (3*n_blocks + 1 of them), bias step s (2*n_blocks + 1) and input-layer K-block q (4, + the end)
MACRO_ARGS = {'n_blocks': range(9), 'mode': range(3), 'variant': range(8), 'm': range(3 * 8 + 1), 's': range(2 * 8 + 1),
              'q': range(5)}


def test_layout_macros_match_the_python_mirror(tmp_path):
    """VTACO_MAX_BLOCKS and every VTACO_DEC_* / VTACO_ENC_* layout and size macro of the header, as a C compiler evaluates it, equals
    its mirror in vtaco_b200._abi (VTACO_X -> _abi.X; VTACO_X(args) -> _abi.x(args) at every combination of
    MACRO_ARGS)."""
    if shutil.which('gcc') is None:
        pytest.skip('no C compiler')
    hdr = open(os.path.join(ROOT, 'include', 'vtaco_b200.h')).read()
    consts = re.findall(r'^#define (VTACO_(?:DEC|ENC)_[A-Z0-9_]+|VTACO_MAX_BLOCKS)[ \t]', hdr, flags=re.M)
    funcs = {m: tuple(a.strip() for a in args.split(','))
             for m, args in re.findall(r'^#define (VTACO_(?:DEC|ENC)_[A-Z0-9_]+)\(([^)]*)\)', hdr, flags=re.M)}
    assert {'VTACO_DEC_BLK_W1', 'VTACO_DEC_TAIL_BCON', 'VTACO_ENC_BLK_WS', 'VTACO_ENC_FCC_B', 'VTACO_MAX_BLOCKS'} <= set(consts)
    assert {'VTACO_DEC_PACKED_FLOATS', 'VTACO_ENC_PACKED_FLOATS'} <= set(funcs)
    assert {'VTACO_DEC_TC_SUB_BF16', 'VTACO_DEC_TC_KBLK_FLOATS', 'VTACO_DEC_TC_MODE_TILE4'} <= set(consts)
    assert {'VTACO_DEC_TC_MODE', 'VTACO_DEC_TC_MAT', 'VTACO_DEC_TC_BIAS', 'VTACO_DEC_TC_WIMG', 'VTACO_DEC_TC_INPUT',
            'VTACO_DEC_TC_USED_FLOATS', 'VTACO_DEC_TC_FLOATS'} <= set(funcs)
    calls = [(m, args) for m, names in funcs.items() for args in itertools.product(*(MACRO_ARGS[n] for n in names))]
    lines = ['#include <stdio.h>', '#include "vtaco_b200.h"', 'int main(void) {']
    lines += ['  printf("%s %%ld\\n", (long)(%s));' % (m, m) for m in consts]
    lines += ['  printf("%s %%ld\\n", (long)(%s(%s)));' % (m, m, ', '.join(map(str, a))) for m, a in calls]
    lines += ['  return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = str(tmp_path / 'layout')
    subprocess.run(['gcc', '-std=c99', '-I', os.path.join(ROOT, 'include'), str(src), '-o', exe], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split('\n')[:-1]
    assert len(out) == len(consts) + len(calls)
    for line, (macro, args) in zip(out, [(m, None) for m in consts] + calls):
        name, val = line.split()
        assert name == macro
        name = macro[len('VTACO_'):]
        want = getattr(_abi, name) if args is None else getattr(_abi, name.lower())(*args)
        assert int(val) == want, (macro, args, int(val), want)


# weights_tc section offsets as vtaco_decoder_pack_tc placed them before they were named, per pack mode:
# n_blocks -> (floats per matrix, W_img block, first bias step, floats per bias step, first input-layer K-block or
# None, floats used); and the floats reserved, VTACO_DEC_TC_FLOATS
TC_LAYOUT = {
    0: {1: (2048, 6912, 6144, 256, None, 8960), 3: (2048, 20224, 18432, 256, None, 22272),
        5: (2048, 33536, 30720, 256, None, 35584)},
    2: {1: (2560, 7680, 10240, 32, 10336, 11360), 3: (2560, 23040, 25600, 32, 25824, 26848),
        5: (2560, 38400, 40960, 32, 41312, 42336)},
}
TC_LAYOUT[1] = TC_LAYOUT[0]     # mode 1 differs from mode 0 only inside a matrix's lo sub-block
TC_FLOATS = {1: 12032, 3: 28416, 5: 44800}


@pytest.mark.parametrize('nb', N_BLOCKS)
@pytest.mark.parametrize('mode', (0, 1, 2))
def test_tc_section_offsets_match_the_documented_layout(mode, nb):
    mat, wimg, bias0, step, input0, used = TC_LAYOUT[mode][nb]
    assert [_abi.dec_tc_mat(mode, m) for m in range(3 * nb)] == [m * mat for m in range(3 * nb)]
    assert _abi.dec_tc_mat_floats(mode) == mat
    assert _abi.dec_tc_wimg(mode, nb) == wimg
    if mode == 2:
        assert _abi.dec_tc_mat(mode, 3 * nb) == wimg
        assert [_abi.dec_tc_input(nb, q) for q in range(4)] == [input0 + 256 * q for q in range(4)]
    assert [_abi.dec_tc_bias(mode, nb, s) for s in range(2 * nb + 1)] == [bias0 + step * s for s in range(2 * nb + 1)]
    assert _abi.dec_tc_used_floats(mode, nb) == used
    assert _abi.dec_tc_floats(nb) == TC_FLOATS[nb]


@pytest.mark.parametrize('mode', (0, 1, 2))
def test_tc_sections_tile_the_used_floats(mode):
    """For 0-8 blocks the matrices, the W_img block, the bias steps and (mode 2) the input-layer K-blocks do not
    overlap, leave no gap (vtaco_decoder_pack_tc writes every float in front of VTACO_DEC_TC_USED_FLOATS) and fit
    the VTACO_DEC_TC_FLOATS reserved for the buffer; the sub-blocks fit their matrix."""
    mat = _abi.dec_tc_mat_floats(mode)
    subs = [(_abi.DEC_TC_SUB_HI, 1024), (_abi.DEC_TC_SUB_LO, 1024)] + ([(_abi.DEC_TC_SUB_BF16, 512)] if mode == 2 else [])
    assert sorted(subs) == subs and all(a + n == b for (a, n), (b, _) in zip(subs, subs[1:] + [(mat, 0)]))
    for nb in range(9):
        sec = [(_abi.dec_tc_mat(mode, m), mat) for m in range(3 * nb)] + [(_abi.dec_tc_wimg(mode, nb), mat)]
        sec += [(_abi.dec_tc_bias(mode, nb, s), _abi.dec_tc_bias_step_floats(mode)) for s in range(2 * nb + 1)]
        if mode == 2:
            sec += [(_abi.dec_tc_input(nb, q), _abi.DEC_TC_KBLK_FLOATS) for q in range(4)]
        sec.sort()
        assert sec[0][0] == 0, nb
        assert all(a + n == b for (a, n), (b, _) in zip(sec, sec[1:])), nb
        assert sec[-1][0] + sec[-1][1] == _abi.dec_tc_used_floats(mode, nb) <= _abi.dec_tc_floats(nb), nb


def test_tc_pack_mode_of_each_variant():
    assert {v: _abi.dec_tc_mode(v) for v in range(2, 8)} == {2: 0, 3: 0, 4: 1, 5: 0, 6: 1, 7: 2}


@pytest.mark.parametrize('nb', N_BLOCKS)
def test_packed_sizes_match_the_documented_layout(nb):
    assert _abi.dec_packed_floats(nb) == _decoder_fields(nb, 32, True)[1]
    assert _abi.enc_packed_floats(nb) == _encoder_fields(nb)[1]


@pytest.mark.parametrize('nb', N_BLOCKS)
@pytest.mark.parametrize('c_dim', (0, 32))
@pytest.mark.parametrize('contact_head', (False, True))
def test_decoder_pack_descriptors(nb, c_dim, contact_head, monkeypatch):
    dec = _decoder(nb, c_dim, contact_head)
    got, buf = _captured_pack(dec, monkeypatch)
    fields, size = _decoder_fields(nb, c_dim, contact_head)
    assert got == [(n, off, cols) for n, off, cols, _ in fields]
    assert buf.numel() == size and buf.dtype == torch.float32 and not buf.any()


@pytest.mark.parametrize('nb', N_BLOCKS)
def test_encoder_pack_descriptors(nb, monkeypatch):
    enc = _encoder(nb)
    got, buf = _captured_pack(enc, monkeypatch)
    fields, size = _encoder_fields(nb)
    assert got == [(n, off, cols) for n, off, cols, _ in fields]
    assert buf.numel() == size and buf.dtype == torch.float32 and not buf.any()


@pytest.mark.parametrize('nb', N_BLOCKS)
@pytest.mark.parametrize('c_dim', (0, 32))
@pytest.mark.parametrize('use_img', (False, True))
@pytest.mark.parametrize('contact_head,contact', CONTACT)
def test_decoder_gradient_views(nb, c_dim, use_img, contact_head, contact):
    """Only what the backward writes is returned (fc_p.* or fc_p_img.*, fc_c.* with c_dim, fc_out_contact.* with
    the contact output), every gradient a view of the flat buffer except fc_p_img.weight, which concatenates
    its two fields."""
    dec = _decoder(nb, c_dim, contact_head)
    fields, size = _decoder_fields(nb, c_dim, contact_head)
    flat = _flat(size)
    g = dec._unpack_param_grads(flat, use_img, contact)
    skip = ('fc_p.' if use_img else 'fc_p_img.',) + (() if contact else ('fc_out_contact.',))
    views = [f for f in fields if not f[0].startswith(skip) and f[0] != 'fc_p_img.weight']
    want = {f[0] for f in views} | ({'fc_p_img.weight'} if use_img else set())
    assert set(g) == want
    _check_views(g, views, flat)
    if use_img:
        w = g['fc_p_img.weight']
        parts = [flat[off:off + 32 * cols[1]].view(shape) for n, off, cols, shape in fields if n == 'fc_p_img.weight']
        assert tuple(w.shape) == (32, 3 + c_dim) and not _is_view_of(w, flat)
        assert torch.equal(w, torch.cat(parts, 1))


@pytest.mark.parametrize('nb', N_BLOCKS)
def test_encoder_gradient_views(nb):
    enc = _encoder(nb)
    fields, size = _encoder_fields(nb)
    flat = _flat(size)
    g = enc._unpack_param_grads(flat)
    assert set(g) == {f[0] for f in fields}
    assert set(g) == {n for n, _ in enc._pointnet_params()}
    _check_views(g, fields, flat)
