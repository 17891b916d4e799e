"""CPU: drop-in contract of the modules — constructor kwargs, state_dict keys/shapes
identical to the reference's (tests/golden/state_dict_contract.json, dumped from the
reference), UNet/UNet3D re-implementations equal to the reference's outputs, and the
no-fallback rule (CPU tensors are refused, missing library fails loudly)."""
import json
import os

import numpy as np
import pytest
import torch

from util import GOLDEN, load, close


def _contract():
    with open(os.path.join(GOLDEN, 'state_dict_contract.json')) as f:
        return json.load(f)


def test_state_dict_contract():
    from vtaco_b200.encoder import encoder_dict
    from vtaco_b200.conv_onet.models import decoder_dict
    c = _contract()
    enc_g = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, plane_type='grid',
                                                grid_resolution=64, unet3d=True,
                                                unet3d_kwargs=dict(num_levels=4, f_maps=32, in_channels=32,
                                                                   out_channels=32))
    enc_t = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32,
                                                plane_type=['xz', 'xy', 'yz'], plane_resolution=32, unet=True,
                                                unet_kwargs=dict(depth=4, merge_mode='concat', start_filts=32))
    dec = decoder_dict['simple_local'](dim=3, c_dim=32, padding=0.1, with_contact=True, sample_mode='bilinear',
                                       hidden_size=32)
    for name, m in (('encoder_grid_unet3d', enc_g), ('encoder_tri_unet', enc_t), ('decoder_contact', dec)):
        mine = {k: list(v.shape) for k, v in m.state_dict().items()}
        assert mine == c[name], name
        assert list(mine.keys()) == sorted(c[name].keys(), key=list(mine.keys()).index)


def test_shipped_yaml_kwargs_accepted():
    """the factories pass **encoder_kwargs straight through (conv_onet/config.py:82-93);
    unknown UNet keys such as the YAML typo `start_flits` are swallowed."""
    from vtaco_b200.encoder import encoder_dict
    e = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, plane_type=['xz', 'xy', 'yz'],
                                            plane_resolution=64, unet=True,
                                            unet_kwargs=dict(depth=4, merge_mode='concat', start_flits=32))
    assert e.unet.start_filts == 32
    with pytest.raises(ValueError, match='incorrect scatter type'):
        encoder_dict['pointnet_local_pool'](c_dim=32, hidden_dim=32, scatter_type='sum')
    with pytest.raises(NotImplementedError):
        encoder_dict['pointnet_local_pool'](c_dim=32, hidden_dim=32, out_mano=True, out_dim=51)


def test_invalidate_reaches_every_packed_weight_cache():
    """ADVICE r1 (medium): the packed-operand caches are keyed on (data_ptr, _version), which `param.data`
    updates do not change — `invalidate()` is the documented way out and has to reach the UNets' caches too."""
    from vtaco_b200.encoder import encoder_dict
    e = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, plane_type=['grid', 'xz'],
                                            grid_resolution=16, plane_resolution=16, unet=True,
                                            unet_kwargs=dict(depth=2, start_filts=32), unet3d=True,
                                            unet3d_kwargs=dict(num_levels=2, f_maps=32, in_channels=32, out_channels=32))
    e.unet.__dict__['_wcache'] = {'stale': 1}
    e.unet3d._wcache = {'stale': 1}
    e._pack_cache = ('stale', None)
    e.invalidate()
    assert e.unet.__dict__['_wcache'] == {} and e.unet3d._wcache == {} and e._pack_cache is None
    e.unet3d._wcache = {'stale': 1}
    e.load_state_dict(e.state_dict())          # load_state_dict / .to() invalidate on their own
    assert e.unet3d._wcache == {}


def test_fc1_zero_init_like_reference():
    from vtaco_b200.layers import ResnetBlockFC
    b = ResnetBlockFC(64, 32)
    assert float(b.fc_1.weight.abs().sum()) == 0.0 and b.shortcut.bias is None
    assert ResnetBlockFC(32).shortcut is None


def test_unets_match_reference():
    from vtaco_b200.encoder.unet import UNet
    from vtaco_b200.encoder.unet3d import UNet3D
    from util import rs_randn
    g = load('unets.npz')
    u2 = UNet(8, in_channels=8, depth=3, merge_mode='concat', start_filts=8)
    u2.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith('u2.')}, strict=True)
    u3 = UNet3D(in_channels=8, out_channels=8, num_levels=3, f_maps=8)
    u3.load_state_dict({k[3:]: torch.from_numpy(v) for k, v in g.items() if k.startswith('u3.')}, strict=True)
    with torch.no_grad():
        o2 = u2.eval()(torch.from_numpy(rs_randn(83, 2, 8, 16, 16)))
        o3 = u3.eval()(torch.from_numpy(rs_randn(84, 1, 8, 8, 8, 8)))
    assert close(o2.numpy(), g['unet_out']) < 1e-5
    assert close(o3.numpy(), g['unet3d_out']) < 1e-5


def test_no_cpu_fallback():
    from vtaco_b200.conv_onet.models import decoder_dict
    from vtaco_b200 import common as vc
    dec = decoder_dict['simple_local'](dim=3, c_dim=32, hidden_size=32)
    with torch.no_grad():
        with pytest.raises(RuntimeError, match='CUDA'):
            dec(torch.zeros(1, 4, 3), {'grid': torch.zeros(1, 32, 8, 8, 8)})
        with pytest.raises(RuntimeError, match='CUDA'):
            vc.normalize_coordinate(torch.zeros(1, 4, 3))


def test_unsupported_width_raises():
    from vtaco_b200.conv_onet.models import decoder_dict
    dec = decoder_dict['simple_local'](dim=3, c_dim=128, hidden_size=256)  # constructible (state_dict), not runnable
    assert dec.fc_p.weight.shape == (256, 3)
    with pytest.raises(NotImplementedError):
        dec._check_supported()


def test_library_exports_every_declared_symbol():
    """the C-ABI library loads and exports every function include/vtaco_b200.h declares."""
    import ctypes
    import re
    from vtaco_b200 import _abi
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    hdr = open(os.path.join(root, 'include', 'vtaco_b200.h')).read()
    hdr = re.sub(r'/\*.*?\*/', '', hdr, flags=re.S)
    names = set(re.findall(r'\b(vtaco_[a-z0-9_]+)\s*\(', hdr))
    assert len(names) >= 10
    L = ctypes.CDLL(_abi.LIB_PATH)
    for n in sorted(names):
        assert hasattr(L, n), 'missing export %s' % n
    assert L.vtaco_abi_version() == 1
    # host-only size helpers: the Python mirror of the header macros must agree with the library
    L.vtaco_decoder_tc_floats.restype = ctypes.c_int64
    for nb in range(0, 9):
        assert L.vtaco_decoder_tc_floats(nb) == _abi.dec_tc_floats(nb), nb


def test_make_3d_grid_matches_reference():
    from vtaco_b200.common import make_3d_grid, dense_axis
    g = load('coords.npz')
    assert np.array_equal(make_3d_grid((-0.5,) * 3, (0.5,) * 3, (4, 3, 2)).numpy(), g['grid3_4'])
    for nx in (8, 32, 128, 256):
        assert np.array_equal(dense_axis(nx).numpy(), g['axis_%d' % nx])


def test_off_roundtrip(tmp_path):
    """export_off writes what read_off (reference src/utils/io.py:27-80 semantics) reads back."""
    import numpy as np
    from vtaco_b200.io import export_off, read_off
    rs = np.random.RandomState(0)
    v = rs.uniform(-0.55, 0.55, size=(50, 3)).astype(np.float32)
    f = rs.randint(0, 50, size=(80, 3)).astype(np.int32)
    path = str(tmp_path / 'm.off')
    export_off(path, torch.from_numpy(v), torch.from_numpy(f))
    v2, f2 = read_off(path)
    assert np.array_equal(f2, f) and np.allclose(v2, v, rtol=0, atol=1e-7)
    with open(path) as fp:
        assert fp.readline().strip() == 'OFF' and fp.readline().split() == ['50', '80', '0']
    with open(path, 'w') as fp:          # ModelNet variant: counts on the OFF line
        fp.write('OFF3 1 0\n0 0 0\n1 0 0\n0 1 0\n3 0 1 2\n')
    v3, f3 = read_off(path)
    assert v3.shape == (3, 3) and f3.tolist() == [[0, 1, 2]]
    with pytest.raises(ValueError):
        export_off(path, v, np.array([[0, 1, 50]]))


def test_ctypes_structs_match_the_c_header(tmp_path):
    """sizeof / offsetof of every argument struct of include/vtaco_b200.h as a C compiler lays it
    out == the ctypes mirror the Python side passes through the ABI."""
    import ctypes as C
    import os
    import shutil
    import subprocess
    from vtaco_b200 import _abi
    from vtaco_b200._abi import EncoderArgs, EncoderBwdArgs
    if shutil.which('gcc') is None:
        pytest.skip('no C compiler')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    structs = {'vtaco_decoder_args': _abi.DecoderArgs, 'vtaco_decoder_bwd_args': _abi.DecoderBwdArgs,
               'vtaco_encoder_args': EncoderArgs, 'vtaco_encoder_bwd_args': EncoderBwdArgs,
               'vtaco_mc_args': _abi.McArgs, 'vtaco_conv3d_args': _abi.Conv3dArgs, 'vtaco_exchange': _abi.Exchange,
               'vtaco_mesh_piece': _abi.MeshPiece, 'vtaco_pack_desc': _abi.PackDesc}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vtaco_b200.h"', 'int main(void) {']
    for cname, cls in structs.items():
        lines.append('  printf("%s sizeof %%zu\\n", sizeof(%s));' % (cname, cname))
        for fname, _ in cls._fields_:
            lines.append('  printf("%s %s %%zu\\n", offsetof(%s, %s));' % (cname, fname, cname, fname))
    lines += ['  return 0;', '}']
    src = tmp_path / 'layout.c'
    src.write_text('\n'.join(lines))
    exe = str(tmp_path / 'layout')
    subprocess.run(['gcc', '-std=c99', '-I', os.path.join(root, 'include'), str(src), '-o', exe], check=True)
    out = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.split('\n')
    seen = 0
    for ln in out:
        if not ln:
            continue
        cname, field, val = ln.split()
        cls = structs[cname]
        want = C.sizeof(cls) if field == 'sizeof' else getattr(cls, field).offset
        assert int(val) == want, (cname, field, int(val), want)
        seen += 1
    assert seen == sum(len(c._fields_) + 1 for c in structs.values())


def test_c_example_compiles_and_links(tmp_path):
    """examples/dense_extract.c (the ABI used from plain C) builds against the header and the library."""
    import os
    import shutil
    import subprocess
    from vtaco_b200 import _abi
    if shutil.which('gcc') is None or not os.path.exists(_abi.LIB_PATH):
        pytest.skip('needs gcc and the built library')
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    cuda_lib = '/usr/local/cuda/lib64'
    if not os.path.exists(os.path.join(cuda_lib, 'libcudart.so')):
        pytest.skip('no libcudart to link against')
    exe = str(tmp_path / 'dense_extract')
    r = subprocess.run(['gcc', '-std=c99', '-Wall', '-Werror', '-I', os.path.join(root, 'include'),
                        os.path.join(root, 'examples', 'dense_extract.c'), '-L', os.path.dirname(_abi.LIB_PATH),
                        '-lvtaco_b200', '-L', cuda_lib, '-lcudart', '-lm', '-o', exe], capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


def test_generation_helpers_match_reference_golden():
    """R_from_PYR / norm_pc_1 / the fingertip transform of generation.py:177-188 against values computed
    by the reference's own functions (tests/golden/make_golden.py helpers)."""
    import numpy as np
    from util import load
    from vtaco_b200.conv_onet.generation import R_from_PYR, norm_pc_1, fingertips_from_mano, Mesh
    g = load('helpers.npz')
    for a, R in zip(g['angles'], g['R']):
        assert np.allclose(R_from_PYR(a), R, rtol=0, atol=1e-15)
    assert np.allclose(norm_pc_1(g['pc'], g['pc_obj']), g['norm'], rtol=0, atol=1e-14)
    tips = fingertips_from_mano(g['joints'], g['wrist_rot'], g['wrist_pos'], g['pc_obj'])
    assert np.allclose(tips, g['tips'], rtol=0, atol=1e-13)
    m = Mesh(np.zeros((3, 3), np.float32), np.array([[0, 1, 2]], np.int32))
    assert m.vertices.shape == (3, 3) and m.faces.shape == (1, 3)
