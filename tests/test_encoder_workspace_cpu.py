"""CPU: the workspace sizes of the PointNet encoder entries.  The forward, the backward and the stand-alone pooling
carve their workspaces with the same layout functions the size helpers call; these byte counts pin that layout."""
import ctypes as C

import pytest

XZ, XY, YZ, GRID = 0, 1, 2, 3

# (B, T, kinds, resos, encoder_workspace_bytes, encoder_backward_workspace_bytes at n_blocks 1 / 5 / 8,
#  pool_workspace_bytes with cells = reso^2 | reso^3 per key)
CASES = [
    (1, 3640, [GRID], [64], 3887872, (7149312, 10876672, 13672192), 1543680),
    (2, 1000, [XZ, XY, YZ], [32, 32, 32], 3682304, (4450304, 8546304, 11618304), 841728),
    (3, 777, [XZ, XY, YZ, GRID], [16, 16, 16, 8], 5501952, (5799936, 11769856, 16247296), 1285120),
]


@pytest.fixture(scope='module')
def lib():
    from vtaco_b200 import _abi
    L = C.CDLL(_abi.LIB_PATH)
    for f in ('vtaco_encoder_workspace_bytes', 'vtaco_encoder_backward_workspace_bytes', 'vtaco_pool_workspace_bytes'):
        getattr(L, f).restype = C.c_int64
    return L


def _i32(v):
    return (C.c_int32 * 4)(*v)


def _cells(kinds, resos):
    return (C.c_int64 * 4)(*[r ** (3 if k == GRID else 2) for k, r in zip(kinds, resos)])


@pytest.mark.parametrize('B,T,kinds,resos,fwd,bwd,pool', CASES)
def test_workspace_bytes(lib, B, T, kinds, resos, fwd, bwd, pool):
    nk = len(kinds)
    assert lib.vtaco_encoder_workspace_bytes(B, C.c_int64(T), nk, _i32(kinds), _i32(resos)) == fwd
    for nb, want in zip((1, 5, 8), bwd):
        assert lib.vtaco_encoder_backward_workspace_bytes(B, C.c_int64(T), nk, _i32(kinds), _i32(resos), nb) == want
    assert lib.vtaco_pool_workspace_bytes(B, C.c_int64(T), nk, _cells(kinds, resos)) == pool


@pytest.mark.parametrize('n_keys', [0, 5])
def test_workspace_bytes_reject_key_count(lib, n_keys):
    kinds, resos = [GRID] * 4, [64] * 4
    assert lib.vtaco_encoder_workspace_bytes(1, C.c_int64(3640), n_keys, _i32(kinds), _i32(resos)) == -1
    assert lib.vtaco_encoder_backward_workspace_bytes(1, C.c_int64(3640), n_keys, _i32(kinds), _i32(resos), 5) == -1
    assert lib.vtaco_pool_workspace_bytes(1, C.c_int64(3640), n_keys, _cells(kinds, resos)) == -1


@pytest.mark.parametrize('n_blocks', [0, 9])
def test_backward_workspace_bytes_reject_block_count(lib, n_blocks):
    assert lib.vtaco_encoder_backward_workspace_bytes(1, C.c_int64(3640), 1, _i32([GRID]), _i32([64]), n_blocks) == -1


def test_workspace_bytes_do_not_check_reso(lib):
    """the size helper sizes any reso; the forward itself refuses a grid above 1290^3 cells."""
    assert lib.vtaco_encoder_workspace_bytes(1, C.c_int64(3640), 1, _i32([GRID]), _i32([2000])) == 32002839296
