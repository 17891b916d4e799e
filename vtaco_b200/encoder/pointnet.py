"""LocalPoolPointnet — drop-in for reference src/encoder/pointnet.py:12-210.

Same constructor arguments, parameter names / shapes and return convention
(dict key -> (B,c_dim,R,R[,R]), keys in the order grid, xz, xy, yz).  The PointNet
part (indexing, fc_pos, ResnetBlockFC stack with local pooling, fc_c,
scatter_mean) runs in the CUDA kernels of vtaco_b200/csrc/encoder.cu through the
C ABI; the optional UNet / UNet3D post-processing stays torch.nn (cuDNN).

The returned tensors are in torch's channels_last / channels_last_3d memory
format: same shape and values as the reference's, and the layout the fused
decoder gathers from without a copy.

With grad enabled the PointNet part is an autograd node whose backward is
vtaco_encoder_backward (csrc/encoder_bwd.inl); the UNets train through torch autograd.

Out of scope (raises): the MANO hand head (`out_mano=True`), reference
pointnet.py:175-198 — a different model (SURVEY §2 row 13).
"""
import ctypes as C

import torch
import torch.nn as nn

from .. import _abi
from .._abi import EncoderArgs, EncoderBwdArgs
from ..common import _div_mode
from ..layers import ResnetBlockFC
from .unet import UNet
from .unet3d import UNet3D

_KEY_ORDER_IN = ('xz', 'xy', 'yz', 'grid')    # insertion order of coord/index dicts (pointnet.py:141-152)
_KEY_ORDER_OUT = ('grid', 'xz', 'xy', 'yz')   # insertion order of the returned dict (pointnet.py:165-172)


# The fields of the packed buffer (include/vtaco_b200.h), as _abi.layout_entries takes them
_LAYOUT = (_abi.ENC_OFF_BLOCKS, _abi.ENC_BLOCK_STRIDE,
           [('fc_pos.weight', _abi.ENC_OFF_WPOS), ('fc_pos.bias', _abi.ENC_OFF_BPOS)],
           [('blocks.%d.fc_0.weight', _abi.ENC_BLK_W0), ('blocks.%d.fc_0.bias', _abi.ENC_BLK_B0),
            ('blocks.%d.fc_1.weight', _abi.ENC_BLK_W1), ('blocks.%d.fc_1.bias', _abi.ENC_BLK_B1),
            ('blocks.%d.shortcut.weight', _abi.ENC_BLK_WS)],
           [('fc_c.weight', _abi.ENC_FCC_W), ('fc_c.bias', _abi.ENC_FCC_B)])


class _PointnetFn(torch.autograd.Function):
    """autograd bridge of the PointNet part: forward = vtaco_encoder_pointnet, backward =
    vtaco_encoder_backward (what torch autograd does for the reference when training.py trains
    the encoder through pointnet.py:135-172)."""

    @staticmethod
    def forward(ctx, mod, p, names, *params):
        fea = mod._pointnet_impl(p)
        ctx.mod, ctx.names, ctx.keys = mod, names, tuple(fea.keys())
        ctx.w = mod._packed_weights()   # the weights this forward saw
        ctx.save_for_backward(p)
        return tuple(fea[k] for k in ctx.keys)

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *grads):
        (p,) = ctx.saved_tensors
        mod = ctx.mod
        if all(g is None for g in grads) or p.numel() == 0:
            return (None, None, None) + (None,) * len(ctx.names)
        flat = mod._pointnet_backward(p, ctx.w, dict(zip(ctx.keys, grads)))
        pg = mod._unpack_param_grads(flat)
        need = ctx.needs_input_grad
        return (None, None, None) + tuple(pg.get(n) if need[3 + i] else None for i, n in enumerate(ctx.names))


class LocalPoolPointnet(nn.Module):
    ''' PointNet-based encoder network with ResNet blocks for each point.

    Args:
        c_dim (int): dimension of latent code c
        dim (int): input points dimension
        hidden_dim (int): hidden dimension of the network
        scatter_type (str): feature aggregation when doing local pooling ('max' | 'mean')
        unet (bool): whether to use U-Net
        unet_kwargs (str): U-Net parameters
        unet3d (bool): whether to use 3D U-Net
        unet3d_kwargs (str): 3D U-Net parameters
        plane_resolution (int): defined resolution for plane feature
        grid_resolution (int): defined resolution for grid feature
        plane_type (str): feature type, 'xz' - 1-plane, ['xz', 'xy', 'yz'] - 3-plane, ['grid'] - 3D grid volume
        padding (float): conventional padding paramter of ONet for unit cube
        n_blocks (int): number of blocks ResNetBlockFC layers
    '''

    def __init__(self, c_dim=128, dim=3, hidden_dim=128, scatter_type='max',
                 unet=False, unet_kwargs=None, unet3d=False, unet3d_kwargs=None,
                 plane_resolution=None, grid_resolution=None, plane_type='xz', padding=0.1, n_blocks=5,
                 out_mano=False, out_dim=None, manolayer_kwargs=None):
        super().__init__()
        self.c_dim = c_dim
        self.dim = dim
        self.fc_pos = nn.Linear(dim, 2 * hidden_dim)
        self.blocks = nn.ModuleList([ResnetBlockFC(2 * hidden_dim, hidden_dim) for _ in range(n_blocks)])
        self.fc_c = nn.Linear(hidden_dim, c_dim)
        self.actvn = nn.ReLU()
        self.hidden_dim = hidden_dim
        self.n_blocks = n_blocks
        self.unet = UNet(c_dim, in_channels=c_dim, **unet_kwargs) if unet else None
        self.unet3d = UNet3D(**unet3d_kwargs) if unet3d else None
        self.reso_plane = plane_resolution
        self.reso_grid = grid_resolution
        self.plane_type = plane_type
        self.padding = padding
        if scatter_type not in ('max', 'mean'):
            raise ValueError('incorrect scatter type')
        self.scatter_type = scatter_type
        self.out_mano = out_mano
        self.out_dim = out_dim
        if out_mano or manolayer_kwargs is not None:
            raise NotImplementedError(
                'vtaco_b200: the MANO hand head of LocalPoolPointnet (out_mano / manolayer_kwargs) is outside the '
                'conv-occupancy hot path and is not built (SURVEY.md §2 row 13)')
        self.division = 'cuda'
        self._pack_cache = None
        self._pack_params = None
        self._ws = None

    # ------------------------------------------------------------------ helpers
    def _keys_in(self):
        return [k for k in _KEY_ORDER_IN if k in self.plane_type]

    def _reso(self, key):
        r = self.reso_grid if key == 'grid' else self.reso_plane
        if r is None:
            raise ValueError('%s_resolution is required for plane_type %r'
                             % ('grid' if key == 'grid' else 'plane', self.plane_type))
        return int(r)

    def _check_supported(self):
        if self.dim != 3 or self.hidden_dim != 32 or self.c_dim != 32:
            raise NotImplementedError(
                'vtaco_b200 encoder kernels implement dim=3, hidden_dim=32, c_dim=32 (every shipped VTacO '
                'conv-occupancy config); got dim=%d hidden_dim=%d c_dim=%d' % (self.dim, self.hidden_dim, self.c_dim))

    def invalidate(self):
        """Drop the packed-weight cache (keyed on (data_ptr, _version) of the parameters; updates made
        through `param.data` do not bump `_version` — call this after one when running under no_grad;
        with grad enabled every call re-packs, and `.to()` / `load_state_dict` invalidate on their own)."""
        self._pack_cache = None
        self._pack_params = None
        self.__dict__['_desc_cache'] = {}
        for name in ('unet', 'unet3d'):      # their packed convolution weights follow the same keying
            m = getattr(self, name, None)
            if m is not None and hasattr(m, 'invalidate'):
                m.invalidate()

    def _apply(self, fn, *args, **kwargs):
        self.invalidate()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):
        self.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def _packed_weights(self):
        """K-major fp32 buffer (layout in include/vtaco_b200.h), one vtaco_pack_linear launch."""
        params = self._params_by_name()
        key = tuple((p.data_ptr(), p._version) for p in params.values())
        if self._pack_cache is not None and self._pack_cache[0] == key:
            return self._pack_cache[1]
        buf = torch.zeros(_abi.enc_packed_floats(self.n_blocks), dtype=torch.float32, device=self.fc_pos.weight.device)
        ent = _abi.layout_entries(_LAYOUT, params, self.n_blocks)
        for j in range(0, len(ent), _abi.PACK_MAX_DESCS):
            _abi.pack_linear(ent[j:j + _abi.PACK_MAX_DESCS], buf,
                             cache=self.__dict__.setdefault('_desc_cache', {}).setdefault(j, {}))
        self._pack_cache = (key, buf)
        return buf

    def _workspace(self, nbytes, device):
        if self._ws is None or self._ws.numel() < nbytes or self._ws.device != device:
            self._ws = torch.empty(int(nbytes), dtype=torch.uint8, device=device)
        return self._ws

    # ------------------------------------------------------------------ fused PointNet part
    def pointnet_features(self, p, return_code=False, return_index=False):
        """Everything of forward() before the UNets: dict key -> channels-last-format feature
        tensor (B,32,R,R[,R]) in the OUTPUT key order; optionally the per-point code c (B,T,32)
        and the int32 cell indices per key."""
        self._check_supported()
        _abi.require_cuda(p, 'p')
        if p.dim() != 3 or p.size(2) != 3:
            raise ValueError('p must have shape (B, T, 3)')
        own = self._pointnet_params() if torch.is_grad_enabled() else ()   # (walks the module tree: not under no_grad)
        if own and _abi.wants_grad(p, *[t for _, t in own]):
            # no gradient w.r.t. the input cloud is produced (backward returns None for p), like the
            # decoder: the reference never reads it
            if return_code or return_index:
                raise NotImplementedError('vtaco_b200: return_code / return_index are inference-only outputs; '
                                          'call under torch.no_grad()')
            self._pack_cache = None    # training: re-pack every step (one launch), immune to `.data` updates
            names, params = zip(*own)
            outs = _PointnetFn.apply(self, p, names, *params)
            return dict(zip([k for k in _KEY_ORDER_OUT if k in self._keys_in()], outs))
        return self._pointnet_impl(p, return_code, return_index)

    def _pointnet_params(self):
        return [(n, t) for n, t in self.named_parameters() if not n.startswith(('unet.', 'unet3d.'))]

    def _params_by_name(self):
        """name -> parameter of the PointNet part (cached: walking the module tree costs more than the check it
        feeds)."""
        if self._pack_params is None:
            self._pack_params = dict(self._pointnet_params())
        return self._pack_params

    def _pointnet_impl(self, p, return_code=False, return_index=False):
        L = _abi.lib()
        B, T = p.shape[0], p.shape[1]
        keys = self._keys_in()
        if not keys:
            raise ValueError('plane_type %r selects no feature' % (self.plane_type,))
        dev = p.device
        pc = p.contiguous()
        a = EncoderArgs()
        a.p, a.B, a.T = pc.data_ptr(), B, T
        a.padding, a.div_mode = float(self.padding), _div_mode(self.division)
        a.n_keys = len(keys)
        outs, idxs = {}, {}
        for i, k in enumerate(keys):
            a.kind[i], a.reso[i] = _abi.KIND[k], self._reso(k)
            R = self._reso(k)
            shape = (B, R, R, R, 32) if k == 'grid' else (B, R, R, 32)
            outs[k] = torch.empty(shape, dtype=torch.float32, device=dev)
            a.out_cl[i] = outs[k].data_ptr()
            if return_index:
                idxs[k] = torch.empty((B, 1, T), dtype=torch.int32, device=dev)
                a.index_out[i] = idxs[k].data_ptr()
        a.pool_mean = int(self.scatter_type == 'mean')
        a.n_blocks = self.n_blocks
        w = self._packed_weights()
        a.weights = w.data_ptr()
        code = None
        if return_code:
            code = torch.empty((B, T, 32), dtype=torch.float32, device=dev)
            a.c_out = code.data_ptr()
        if B * T > 0:
            nbytes = L.vtaco_encoder_workspace_bytes(B, T, a.n_keys, a.kind, a.reso)
            if nbytes < 0:
                _abi.check(int(nbytes), 'encoder_workspace_bytes')
            ws = self._workspace(nbytes, dev)
            a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
            with torch.cuda.device(dev):
                st = L.vtaco_encoder_pointnet(C.byref(a), _abi.stream_ptr(dev))
            _abi.check(st, 'encoder_pointnet')
        else:
            for t in outs.values():
                t.zero_()
        fea = {}
        for k in _KEY_ORDER_OUT:
            if k in outs:
                t = outs[k]
                fea[k] = t.permute(0, 4, 1, 2, 3) if k == 'grid' else t.permute(0, 3, 1, 2)
        res = (fea,)
        if return_code:
            res += (code,)
        if return_index:
            res += (idxs,)
        return res if len(res) > 1 else fea

    # ------------------------------------------------------------------ backward (SURVEY §8f-2)
    def _pointnet_backward(self, p, w, grads):
        """vtaco_encoder_backward: `grads` maps key -> gradient of the (B,32,R,R[,R]) feature tensor
        (or None); returns the flat parameter-gradient buffer (native layout, include/vtaco_b200.h)."""
        L = _abi.lib()
        B, T = p.shape[0], p.shape[1]
        dev = p.device
        keys = self._keys_in()
        pc = p.contiguous()
        a = EncoderBwdArgs()
        a.p, a.B, a.T = pc.data_ptr(), B, T
        a.padding, a.div_mode = float(self.padding), _div_mode(self.division)
        a.n_keys = len(keys)
        keep = []
        for i, k in enumerate(keys):
            a.kind[i], a.reso[i] = _abi.KIND[k], self._reso(k)
            g = grads.get(k)
            if g is not None:
                gcl = (g.permute(0, 2, 3, 4, 1) if k == 'grid' else g.permute(0, 2, 3, 1)).contiguous().float()
                keep.append(gcl)
                a.d_out_cl[i] = gcl.data_ptr()
        a.pool_mean = int(self.scatter_type == 'mean')
        a.n_blocks = self.n_blocks
        a.weights = w.data_ptr()
        flat = torch.zeros(_abi.enc_packed_floats(self.n_blocks), dtype=torch.float32, device=dev)
        a.d_params = flat.data_ptr()
        nbytes = L.vtaco_encoder_backward_workspace_bytes(B, T, a.n_keys, a.kind, a.reso, self.n_blocks)
        if nbytes < 0:
            _abi.check(int(nbytes), 'encoder_backward_workspace_bytes')
        ws = torch.empty(int(nbytes), dtype=torch.uint8, device=dev)
        a.workspace, a.workspace_bytes = ws.data_ptr(), ws.numel()
        with torch.cuda.device(dev):
            st = L.vtaco_encoder_backward(C.byref(a), _abi.stream_ptr(dev))
        _abi.check(st, 'encoder_backward')
        return flat

    def _unpack_param_grads(self, flat):
        """name -> gradient of every parameter of the PointNet part, from the buffer vtaco_encoder_backward wrote."""
        return _abi.layout_grads(_LAYOUT, self._params_by_name(), flat, self.n_blocks)

    # ------------------------------------------------------------------ reference API
    def forward(self, p):
        """reference pointnet.py:135-172 (MANO head excluded)."""
        fea = self.pointnet_features(p)
        out = {}
        for k, t in fea.items():
            if k == 'grid':
                out[k] = self.unet3d(t) if self.unet3d is not None else t
            else:
                out[k] = self.unet(t) if self.unet is not None else t
        return out

    def _index32(self, index, B, T):
        if index.dim() == 3:
            index = index[:, 0, :]
        return index.reshape(B * T).to(torch.int32).contiguous()

    def pool_local(self, xy, index, c):
        """reference pointnet.py:116-132.  `index`: dict key -> (B,1,T) integer cell indices;
        c (B,T,32) -> (B,T,32).  (`xy` is only used for its keys, as in the reference.)"""
        _abi.require_cuda(c, 'c')
        _abi.forbid_autograd(c)
        L = _abi.lib()
        B, T, Cc = c.shape
        if Cc != 32:
            raise NotImplementedError('pool_local kernel implements 32 channels')
        keys = list(xy.keys())
        if not 1 <= len(keys) <= 4:
            raise ValueError('1..4 keys expected')
        idx = [self._index32(index[k], B, T) for k in keys]
        cells = (C.c_int64 * len(keys))(*[self._reso(k) ** (3 if k == 'grid' else 2) for k in keys])
        ptrs = (C.c_void_p * len(keys))(*[t.data_ptr() for t in idx])
        cc = c.contiguous()
        out = torch.empty_like(cc)
        nbytes = L.vtaco_pool_workspace_bytes(B, T, len(keys), cells)
        ws = self._workspace(nbytes, c.device)
        with torch.cuda.device(c.device):
            st = L.vtaco_pool_local(_abi.ptr(cc), B, T, len(keys), ptrs, cells, int(self.scatter_type == 'mean'),
                                    _abi.ptr(ws), ws.numel(), _abi.ptr(out), _abi.stream_ptr(c.device))
        _abi.check(st, 'pool_local')
        return out

    def _scatter_mean(self, p, c, key):
        from ..common import point_to_cell
        _abi.require_cuda(c, 'c')
        _abi.forbid_autograd(p, c)
        L = _abi.lib()
        B, T = p.shape[0], p.shape[1]
        R = self._reso(key)
        idx = point_to_cell(p, R, key, self.padding, self.division, index_dtype=torch.int32).reshape(-1)
        cells = R ** (3 if key == 'grid' else 2)
        cc = c.contiguous()
        shape = (B, R, R, R, 32) if key == 'grid' else (B, R, R, 32)
        out = torch.empty(shape, dtype=torch.float32, device=c.device)
        nbytes = L.vtaco_pool_workspace_bytes(B, T, 1, (C.c_int64 * 1)(cells))
        ws = self._workspace(nbytes, c.device)
        with torch.cuda.device(c.device):
            st = L.vtaco_scatter_mean(_abi.ptr(cc), _abi.ptr(idx), B, T, cells, _abi.ptr(ws), ws.numel(),
                                      _abi.ptr(out), _abi.stream_ptr(c.device))
        _abi.check(st, 'scatter_mean')
        return out.permute(0, 4, 1, 2, 3) if key == 'grid' else out.permute(0, 3, 1, 2)

    def generate_plane_features(self, p, c, plane='xz'):
        """reference pointnet.py:85-100."""
        fea = self._scatter_mean(p, c, plane if plane in ('xz', 'xy') else 'yz')
        return self.unet(fea) if self.unet is not None else fea

    def generate_grid_features(self, p, c):
        """reference pointnet.py:102-114."""
        fea = self._scatter_mean(p, c, 'grid')
        return self.unet3d(fea) if self.unet3d is not None else fea
