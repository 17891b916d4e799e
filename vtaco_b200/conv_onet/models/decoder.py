"""LocalDecoder — drop-in for reference src/conv_onet/models/decoder.py:9-161.

Same constructor arguments, parameter names / shapes (state_dict compatible) and
method names.  All arithmetic runs in ONE fused CUDA kernel
(vtaco_decoder_forward, vtaco_b200/csrc/decoder.cu); there is no PyTorch or CPU
fallback.  With grad enabled, forward / forward_img / forward_contact are autograd
nodes whose backward is vtaco_decoder_backward (csrc/decoder_bwd.cu): gradients for
all parameters, the c_plane feature tensors and c_img.  Extra, non-reference entry point: `forward_dense` evaluates the
extraction lattice of Generator3D without materialising the query tensor.
"""
import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F

from ... import _abi
from ...common import _div_mode, dense_axis
from ...layers import ResnetBlockFC

_PLANES = ('xz', 'xy', 'yz')


def _as_channels_last(t):
    """Return a contiguous tensor laid out [B][spatial...][C] holding the values of the
    channels-first tensor `t` (B,C,*spatial); zero-copy when `t` already is in torch's
    channels_last(_3d) memory format."""
    nd = t.dim()
    perm = (0,) + tuple(range(2, nd)) + (1,)
    v = t.permute(*perm)
    if v.is_contiguous():
        return v
    B, Cc = t.shape[0], t.shape[1]
    S = t[0, 0].numel()
    src = t.contiguous()
    dst = torch.empty(v.shape, dtype=t.dtype, device=t.device)
    with torch.cuda.device(t.device):
        st = _abi.lib().vtaco_relayout_cl(_abi.ptr(src), _abi.ptr(dst), B, Cc, S, _abi.stream_ptr(t.device))
    _abi.check(st, 'relayout_cl')
    return dst


class _DecodeFn(torch.autograd.Function):
    """autograd bridge: forward = vtaco_decoder_forward, backward = vtaco_decoder_backward
    (the role torch autograd plays for the reference decoder in training.py:79,617)."""

    @staticmethod
    def forward(ctx, mod, use_img, contact, keys, names, p, c_img, *tensors):
        nk = len(keys)
        feats = tensors[:nk]
        out, out_c, keep = mod._decode_impl(p, dict(zip(keys, feats)), use_img, c_img, contact)
        ctx.mod, ctx.use_img, ctx.contact, ctx.keys, ctx.names = mod, use_img, contact, keys, names
        ctx.keep = keep  # channels-last feature copies and packed weights as the forward launch saw them
        ctx.save_for_backward(p, c_img)
        return (out, out_c) if contact else out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, *grads):
        mod, keys, names = ctx.mod, ctx.keys, ctx.names
        p, c_img = ctx.saved_tensors
        nk = len(keys)
        none_head = (None,) * 6   # mod, use_img, contact, keys, names, p
        if ctx.keep is None:      # empty batch
            return none_head + (None,) * (1 + nk + len(names))
        cl, w = ctx.keep[0], ctx.keep[1]
        dlogits = grads[0]
        dcontact = grads[1] if ctx.contact and len(grads) > 1 else None
        if dlogits is None and dcontact is None:
            return none_head + (None,) * (1 + nk + len(names))
        need = ctx.needs_input_grad
        need_feat = {k: need[7 + i] for i, k in enumerate(keys)}
        flat, d_feat, d_cimg = mod._decode_backward(p, c_img, cl, w, ctx.use_img, dlogits, dcontact,
                                                    need_feat, need[6])
        pg = mod._unpack_param_grads(flat, ctx.use_img, ctx.contact)
        gfeat = []
        for k in keys:
            t = d_feat.get(k)
            if t is None:
                gfeat.append(None)
            else:  # channels-last storage, channels-first shape
                gfeat.append(t.permute(0, 4, 1, 2, 3) if k == 'grid' else t.permute(0, 3, 1, 2))
        gpar = [pg.get(n) if need[7 + nk + i] else None for i, n in enumerate(names)]
        return none_head + (d_cimg,) + tuple(gfeat) + tuple(gpar)


class LocalDecoder(nn.Module):
    ''' Decoder conditioned on plane / volume local features (reference decoder.py:9-52).

    Args:
        dim (int): input dimension
        c_dim (int): dimension of latent conditioned code c
        hidden_size (int): hidden size of Decoder network
        n_blocks (int): number of blocks ResNetBlockFC layers
        leaky (bool): whether to use leaky ReLUs
        sample_mode (str): sampling feature strategy, bilinear|nearest
        padding (float): conventional padding paramter of ONet for unit cube
        with_contact (bool): add the fc_out_contact head
    '''

    def __init__(self, dim=3, c_dim=128, hidden_size=256, n_blocks=5, leaky=False,
                 sample_mode='bilinear', padding=0.1, with_contact=False):
        super().__init__()
        self.c_dim = c_dim
        self.n_blocks = n_blocks
        self.dim = dim
        self.hidden_size = hidden_size
        if c_dim != 0:
            self.fc_c = nn.ModuleList([nn.Linear(c_dim, hidden_size) for _ in range(n_blocks)])
        self.fc_p = nn.Linear(dim, hidden_size)
        self.fc_p_img = nn.Linear(dim + c_dim, hidden_size)
        self.blocks = nn.ModuleList([ResnetBlockFC(hidden_size) for _ in range(n_blocks)])
        self.fc_out = nn.Linear(hidden_size, 1)
        if with_contact:
            self.fc_out_contact = nn.Linear(hidden_size, 1)
        self.leaky = bool(leaky)
        self.actvn = F.relu if not leaky else (lambda x: F.leaky_relu(x, 0.2))
        self.sample_mode = sample_mode
        self.padding = padding
        # how `tensor / python_scalar` of normalize_* is evaluated ('cuda' | 'true'), SURVEY §7.2-1
        self.division = 'cuda'
        # 0 scalar-FFMA SIMT, 1 packed-FFMA2 SIMT (exact fp32; per-query c_img tensors are routed here),
        # 2 tcgen05 3xTF32 (fp32-accurate to ~1.5e-6), 4 tcgen05 TF32 main product + BF16 corrections (3.6e-6),
        # 5 / 6 = 2 / 4 with two threads per query (8 warps per 128-query tile, 3 tiles per SM),
        # 7 = four tiles per SM (TF32 hi products + BF16 residual product; fastest, default; calls with
        #     >= 2^31 outputs run variant 5), 3 single TF32 product (debug, ~1e-3).  Where a tcgen05 kernel's
        #     shared memory cannot hold n_blocks (tc2 / tc4 at 6-7 blocks, tc at 7) the call runs variant 1.
        self.kernel_variant = 7
        self._pack_cache = None
        self._pack_tc_cache = None
        self._cl_cache = {}
        self._params = None

    def _named_param_tuples(self):
        """(names, parameters) of the module, cached like `_param_tuple` (the training path hands them to autograd)."""
        if self.__dict__.get('_named_params') is None:
            names, params = zip(*self.named_parameters())
            self.__dict__['_named_params'] = (tuple(names), tuple(params))
        return self.__dict__['_named_params']

    def _params_by_name(self):
        """name -> parameter, cached like `_param_tuple` (the packed layout names its fields by parameter)."""
        if self.__dict__.get('_by_name') is None:
            self.__dict__['_by_name'] = dict(zip(*self._named_param_tuples()))
        return self.__dict__['_by_name']

    def _param_tuple(self):
        """The module's parameters as a cached tuple: `self.parameters()` walks the module tree (37 modules,
        ~25 us) and the hot path needs the list three times per call — it was most of the 0.13 ms a flat call
        cost on the host.  Dropped by `invalidate()` / `.to()` / `load_state_dict`; call `invalidate()` after
        adding or replacing a Parameter object by hand."""
        if self._params is None:
            self._params = tuple(self.parameters())
        return self._params

    # ------------------------------------------------------------------ packing
    def _check_supported(self):
        if self.dim != 3 or self.hidden_size != 32 or self.c_dim not in (0, 32):
            raise NotImplementedError(
                'vtaco_b200 fused decoder kernel implements dim=3, hidden_size=32, c_dim in {0,32} '
                '(every shipped VTacO config); got dim=%d hidden_size=%d c_dim=%d'
                % (self.dim, self.hidden_size, self.c_dim))
        if self.sample_mode not in _abi.SAMPLE:
            raise ValueError('sample_mode must be bilinear|nearest, got %r' % (self.sample_mode,))

    def invalidate(self):
        """Drop the packed-weight and channels-last caches.  They are keyed on each tensor's
        (data_ptr, _version); an in-place update made through `param.data` (EMA / clipping code,
        `w.data.normal_()`) does not bump `_version`, so call this after such an update when running
        under torch.no_grad().  Not needed for training: with grad enabled every call re-packs (one
        launch), and `.to()` / `load_state_dict` invalidate on their own."""
        self._pack_cache = None
        self._pack_tc_cache = None
        self._cl_cache = {}
        self._params = None
        self.__dict__['_desc_cache'] = {}
        self.__dict__['_named_params'] = None
        self.__dict__['_by_name'] = None

    def _apply(self, fn, *args, **kwargs):
        self.invalidate()
        return super()._apply(fn, *args, **kwargs)

    def _load_from_state_dict(self, *args, **kwargs):
        self.invalidate()
        return super()._load_from_state_dict(*args, **kwargs)

    def _layout(self):
        """The fields of the packed buffer (include/vtaco_b200.h) this module has, as _abi.layout_entries takes them."""
        head = [('fc_p.weight', _abi.DEC_OFF_WP), ('fc_p.bias', _abi.DEC_OFF_BP),
                ('fc_p_img.weight', _abi.DEC_OFF_WPI, 0, self.dim), ('fc_p_img.bias', _abi.DEC_OFF_BPI)]
        block = [('blocks.%d.fc_0.weight', _abi.DEC_BLK_W0), ('blocks.%d.fc_0.bias', _abi.DEC_BLK_B0),
                 ('blocks.%d.fc_1.weight', _abi.DEC_BLK_W1), ('blocks.%d.fc_1.bias', _abi.DEC_BLK_B1)]
        tail = [('fc_out.weight', _abi.DEC_TAIL_WOUT), ('fc_out.bias', _abi.DEC_TAIL_BOUT)]
        if self.c_dim:
            head.append(('fc_p_img.weight', _abi.DEC_OFF_WIMG, self.dim, self.c_dim))
            block[:0] = [('fc_c.%d.weight', _abi.DEC_BLK_WC), ('fc_c.%d.bias', _abi.DEC_BLK_BC)]
        if hasattr(self, 'fc_out_contact'):
            tail += [('fc_out_contact.weight', _abi.DEC_TAIL_WCON), ('fc_out_contact.bias', _abi.DEC_TAIL_BCON)]
        return _abi.DEC_OFF_BLOCKS, _abi.DEC_BLOCK_STRIDE, head, block, tail

    def _packed_weights(self):
        """Flat fp32 buffer in the layout documented in include/vtaco_b200.h — one launch of
        vtaco_pack_linear into a fresh buffer (an earlier forward's autograd node may still hold
        the previous one)."""
        params = self._param_tuple()
        key = tuple((p.data_ptr(), p._version) for p in params)
        if self._pack_cache is not None and self._pack_cache[0] == key:
            return self._pack_cache[1]
        dev = self.fc_p.weight.device
        nb = self.n_blocks
        if nb > _abi.MAX_BLOCKS:
            raise NotImplementedError('vtaco_b200 decoder kernels hold at most %d blocks in shared memory' % _abi.MAX_BLOCKS)
        buf = torch.zeros(_abi.dec_packed_floats(nb), dtype=torch.float32, device=dev)
        ent = _abi.layout_entries(self._layout(), self._params_by_name(), nb)
        _abi.pack_linear(ent, buf, cache=self.__dict__.setdefault('_desc_cache', {}))
        self._pack_cache = (key, buf)
        self._pack_tc_cache = None
        return buf

    def _packed_weights_tc(self, mixed=False):
        """The tcgen05 operand buffer `weights_tc` in pack mode `mixed` (False / True / 2 = modes 0 / 1 / 2; the
        layout is VTACO_DEC_TC_* in include/vtaco_b200.h, mirrored by _abi.dec_tc_*).  One launch
        (vtaco_decoder_pack_tc) from the packed fp32 buffer."""
        w = self._packed_weights()
        if self._pack_tc_cache is None:
            self._pack_tc_cache = {}
        mixed = int(mixed)
        if mixed in self._pack_tc_cache:
            return self._pack_tc_cache[mixed]
        out = torch.empty(_abi.dec_tc_floats(self.n_blocks), dtype=torch.float32, device=w.device)
        with torch.cuda.device(w.device):
            st = _abi.lib().vtaco_decoder_pack_tc(_abi.ptr(w), self.n_blocks, int(mixed), _abi.ptr(out),
                                                  _abi.stream_ptr(w.device))
        _abi.check(st, 'decoder_pack_tc')
        self._pack_tc_cache[mixed] = out
        return out

    def _features_cl(self, c_plane):
        """Channels-last views/copies of the feature tensors (cached per tensor version)."""
        out = {}
        live = set()
        for k, t in c_plane.items():
            if k not in ('grid',) + _PLANES:
                continue
            _abi.require_cuda(t, "c_plane['%s']" % k)
            want_dim = 5 if k == 'grid' else 4
            if t.dim() != want_dim or t.size(1) != 32:
                raise ValueError("c_plane['%s'] must be (B,32,%s), got %s"
                                 % (k, 'R,R,R' if k == 'grid' else 'R,R', tuple(t.shape)))
            if len(set(t.shape[2:])) != 1:
                raise NotImplementedError('feature tensors must be cubic/square')
            # The entry keeps the SOURCE tensor: `src is t` makes a recycled allocation (same address,
            # version and shape after the caller dropped the previous features) a miss instead of a
            # stale hit, and holding it keeps the address from being reused while the entry lives.
            hit = self._cl_cache.get(k)
            if hit is None or hit[0] is not t or hit[1] != t._version:
                hit = (t, t._version, _as_channels_last(t))
                self._cl_cache[k] = hit
            live.add(k)
            out[k] = hit[2]
        for k in list(self._cl_cache):
            if k not in live:
                del self._cl_cache[k]
        return out

    # ------------------------------------------------------------------ kernel call
    def _run(self, args, device):
        with torch.cuda.device(device):
            st = _abi.lib().vtaco_decoder_forward(C.byref(args), _abi.stream_ptr(device))
        _abi.check(st, 'decoder_forward')

    def _base_args(self, c_plane, B, n_outputs=0):
        self._check_supported()
        a = _abi.DecoderArgs()
        cl = self._features_cl(c_plane) if self.c_dim != 0 else {}
        if self.c_dim != 0 and not cl:
            raise ValueError('c_plane holds none of grid/xz/xy/yz')
        for k, t in cl.items():
            if t.size(0) != B:
                raise ValueError("c_plane['%s'] batch %d != %d" % (k, t.size(0), B))
        a.B = B
        if 'grid' in cl:
            a.grid = cl['grid'].data_ptr()
            a.reso_grid = cl['grid'].size(1)
        rp = None
        for i, k in enumerate(_PLANES):
            if k in cl:
                a.plane[i] = cl[k].data_ptr()
                if rp is not None and rp != cl[k].size(1):
                    raise NotImplementedError('all planes must share one resolution')
                rp = cl[k].size(1)
        a.reso_plane = rp or 0
        a.padding = float(self.padding)
        a.div_mode = _div_mode(self.division)
        a.sample_mode = _abi.SAMPLE[self.sample_mode]
        w = self._packed_weights()
        a.weights = w.data_ptr()
        a.n_blocks = self.n_blocks
        a.leaky = int(self.leaky)
        a.variant = int(self.kernel_variant)
        if a.variant == 7 and n_outputs >= 2 ** 31:
            a.variant = 5      # the four-tile kernel indexes its outputs with 32 bits
        keep = [cl, w]
        if a.variant in (2, 3, 4, 5, 6, 7):
            wtc = self._packed_weights_tc(mixed=_abi.dec_tc_mode(a.variant))
            a.weights_tc = wtc.data_ptr()
            keep.append(wtc)
        return a, keep

    def _decode(self, p, c_plane, use_img=False, c_img=None, contact=False, tip_ids=None):
        """tip_ids = (ids (B,N) uint8, features (F,c_dim) or (1,F,c_dim)): compact per-query tactile
        conditioning instead of a dense c_img tensor (inference only; vtaco_b200.conv_onet.tactile)."""
        _abi.require_cuda(p, 'p')
        if p.dim() != 3 or p.size(2) != 3:
            raise ValueError('p must have shape (B, N, 3)')
        feats = {k: t for k, t in c_plane.items() if k in ('grid',) + _PLANES and torch.is_tensor(t)}
        if torch.is_grad_enabled() and _abi.wants_grad(p, c_img, *self._param_tuple(), *feats.values()):
            # The reference training loop builds its query points with requires_grad=True
            # (training.py:310,362,614,729,868) but never reads p.grad: no gradient w.r.t. p is
            # produced (backward returns None for it), everything else is differentiated.
            self._pack_cache = None     # training: re-pack every step (one launch), immune to `.data` updates
            if tip_ids is not None:
                raise NotImplementedError('vtaco_b200: tip_ids is an inference-only form; pass '
                                          'tactile.c_img_from_ids(ids, c_img) as c_img when training')
            names, params = self._named_param_tuples()
            return _DecodeFn.apply(self, bool(use_img), bool(contact), tuple(feats.keys()), names, p, c_img,
                                   *feats.values(), *params)
        out, out_c, _ = self._decode_impl(p, c_plane, use_img, c_img, contact, tip_ids)
        return (out, out_c) if contact else out

    def _tip_map_args(self, a, keep, ids, feat, n_queries):
        ids = ids.reshape(-1)
        if ids.dtype != torch.uint8 or not ids.is_cuda or ids.numel() != n_queries:
            raise ValueError('tip ids must be a CUDA uint8 tensor with one entry per query')
        feat = feat.reshape(-1, feat.shape[-1]).contiguous()
        _abi.require_cuda(feat, 'tip features')
        if feat.shape[0] > _abi.MAX_TIPS or feat.shape[1] != 32:
            raise ValueError('tip features must be (F <= %d, 32)' % _abi.MAX_TIPS)
        if a.variant not in (2, 4, 5, 6, 7):
            raise NotImplementedError('the per-query tactile id map needs a tcgen05 kernel variant (2, 4, 5, 6, 7)')
        ids = ids.contiguous()
        a.tip_map, a.tip_feat, a.n_tips = ids.data_ptr(), feat.data_ptr(), feat.shape[0]
        keep += [ids, feat]

    def _decode_impl(self, p, c_plane, use_img=False, c_img=None, contact=False, tip_ids=None):
        """Launch the forward kernel; returns (logits, contact|None, tensors the launch reads)."""
        B, N = p.shape[0], p.shape[1]
        pc = p.contiguous()
        out = torch.empty((B, N), dtype=torch.float32, device=p.device)
        out_c = torch.empty((B, N), dtype=torch.float32, device=p.device) if contact else None
        if N == 0 or B == 0:
            return out, out_c, None
        a, keep = self._base_args(c_plane, B, B * N)
        a.p = pc.data_ptr()
        a.N = N
        a.use_img = int(use_img)
        if use_img and tip_ids is not None:
            if B != 1 and tip_ids[1].dim() == 3 and tip_ids[1].shape[0] != 1:
                raise NotImplementedError('tip_ids: one feature table per call (B = 1, or features shared by the batch)')
            self._tip_map_args(a, keep, tip_ids[0], tip_ids[1], B * N)
        elif use_img:
            if c_img is None:
                raise ValueError('forward_img needs c_img')
            _abi.require_cuda(c_img, 'c_img')
            if tuple(c_img.shape) != (B, N, self.c_dim):
                raise ValueError('c_img must have shape (B, N, c_dim)')
            cic = c_img.contiguous()
            a.c_img = cic.data_ptr() if self.c_dim else None
            keep.append(cic)
        a.logits = out.data_ptr()
        if contact:
            if not hasattr(self, 'fc_out_contact'):
                raise AttributeError("'LocalDecoder' object has no attribute 'fc_out_contact'")
            a.contact = out_c.data_ptr()
        self._run(a, p.device)
        return out, out_c, keep

    # ------------------------------------------------------------------ backward (SURVEY §8f-2)
    _BWD_MAX_QUERIES = 1 << 19   # per launch: 23 workspace rows of 128 B per query (1.5 GB)

    def _decode_backward(self, p, c_img, cl, w, use_img, dlogits, dcontact, need_feat, need_cimg):
        """vtaco_decoder_backward: returns (flat parameter gradients in the packed native layout,
        dict of channels-last feature gradients, d_c_img | None)."""
        dev = p.device
        B, N = p.shape[0], p.shape[1]
        nb = self.n_blocks
        L = _abi.lib()
        d_params = torch.zeros(_abi.dec_packed_floats(nb), dtype=torch.float32, device=dev)
        d_feat = {k: torch.zeros_like(t) for k, t in cl.items() if need_feat.get(k)}
        has_cimg = bool(use_img and self.c_dim and c_img is not None)
        d_cimg = torch.empty((B, N, 32), dtype=torch.float32, device=dev) if (need_cimg and has_cimg) else None
        pc = p.contiguous()
        cic = c_img.contiguous() if has_cimg else None
        dl = dlogits.contiguous() if dlogits is not None else None
        dc = dcontact.contiguous() if dcontact is not None else None
        if B * N <= self._BWD_MAX_QUERIES:
            pieces = [(0, B, 0, N)]
        else:
            pieces = [(b, 1, n0, min(self._BWD_MAX_QUERIES, N - n0))
                      for b in range(B) for n0 in range(0, N, self._BWD_MAX_QUERIES)]
        qmax = max(nbatch * n for _, nbatch, _, n in pieces)
        ws_bytes = L.vtaco_decoder_backward_workspace_bytes(qmax, nb)
        ws = torch.empty(ws_bytes // 4, dtype=torch.float32, device=dev)
        for b0, nbatch, n0, n in pieces:
            a = _abi.DecoderBwdArgs()
            whole = (nbatch == B and n == N)
            # a piece inside one sample is passed as B=1 with every per-sample pointer advanced
            psl = pc if whole else pc[b0, n0:n0 + n]
            a.p = psl.data_ptr()
            a.B, a.N = nbatch, n
            if 'grid' in cl:
                a.grid = cl['grid'][b0].data_ptr()
                a.reso_grid = cl['grid'].size(1)
                if 'grid' in d_feat:
                    a.d_grid = d_feat['grid'][b0].data_ptr()
            for i, k in enumerate(_PLANES):
                if k in cl:
                    a.plane[i] = cl[k][b0].data_ptr()
                    a.reso_plane = cl[k].size(1)
                    if k in d_feat:
                        a.d_plane[i] = d_feat[k][b0].data_ptr()
            a.padding = float(self.padding)
            a.div_mode = _div_mode(self.division)
            a.sample_mode = _abi.SAMPLE[self.sample_mode]
            a.weights = w.data_ptr()
            a.n_blocks, a.leaky, a.use_img = nb, int(self.leaky), int(use_img)
            if has_cimg:
                a.c_img = (cic if whole else cic[b0, n0:n0 + n]).data_ptr()
                if d_cimg is not None:
                    a.d_c_img = (d_cimg if whole else d_cimg[b0, n0:n0 + n]).data_ptr()
            if dl is not None:
                a.dlogits = (dl if whole else dl[b0, n0:n0 + n]).data_ptr()
            if dc is not None:
                a.dcontact = (dc if whole else dc[b0, n0:n0 + n]).data_ptr()
            a.workspace, a.workspace_bytes = ws.data_ptr(), ws_bytes
            a.d_params = d_params.data_ptr()
            with torch.cuda.device(dev):
                st = L.vtaco_decoder_backward(C.byref(a), _abi.stream_ptr(dev))
            _abi.check(st, 'decoder_backward')
        return d_params, d_feat, d_cimg

    def _unpack_param_grads(self, flat, use_img, contact):
        """name -> gradient of every parameter vtaco_decoder_backward wrote into `flat`: the input layer used
        (fc_p or fc_p_img), fc_c with c_dim, fc_out_contact with `contact`."""
        off, stride, head, block, tail = self._layout()
        unwritten = ('fc_p.' if use_img else 'fc_p_img.',) + (() if contact else ('fc_out_contact.',))
        head = [e for e in head if not e[0].startswith(unwritten)]
        tail = [e for e in tail if not e[0].startswith(unwritten)]
        return _abi.layout_grads((off, stride, head, block, tail), self._params_by_name(), flat, self.n_blocks)

    # ------------------------------------------------------------------ reference API
    def forward(self, p, c_plane, **kwargs):
        """reference decoder.py:135-161 -> logits (B,N)."""
        return self._decode(p, c_plane)

    def forward_img(self, p, c_plane, c_img=None, tip_ids=None, **kwargs):
        """reference decoder.py:71-103 -> logits (B,N).  Extra: `tip_ids=(ids, features)` instead of
        the dense c_img tensor (see _decode)."""
        return self._decode(p, c_plane, use_img=True, c_img=c_img, tip_ids=tip_ids)

    def forward_contact(self, p, c_plane, **kwargs):
        """reference decoder.py:105-133 -> (logits, contact) each (B,N)."""
        return self._decode(p, c_plane, contact=True)

    def sample_plane_feature(self, p, c, plane='xz'):
        """reference decoder.py:55-60 -> (B, c_dim, N)."""
        return self._sample(p, {plane if plane in ('xz', 'xy') else 'yz': c})

    def sample_grid_feature(self, p, c):
        """reference decoder.py:62-68 -> (B, c_dim, N)."""
        return self._sample(p, {'grid': c})

    def _sample(self, p, c_plane):
        _abi.require_cuda(p, 'p')
        _abi.forbid_autograd(p, *c_plane.values())
        B, N = p.shape[0], p.shape[1]
        a, keep = self._base_args(c_plane, B)
        pc = p.contiguous()
        out = torch.empty((B, 32, N), dtype=torch.float32, device=p.device)
        L = _abi.lib()
        with torch.cuda.device(p.device):
            st = L.vtaco_sample_features(C.byref(a), _abi.ptr(pc), N, _abi.ptr(out), _abi.stream_ptr(p.device))
        _abi.check(st, 'sample_features')
        return out

    # ------------------------------------------------------------------ dense lattice (Generator3D fast path)
    def forward_dense(self, c_plane, nx, x0=0, x1=None, use_img=False, c_img=None, tips=None,
                      out=None, minmax_key=None, axis=None, peers=None, multicast=None, tip_map=None):
        """Evaluate the extraction lattice (1+padding)*make_3d_grid(nx^3) (reference
        generation.py:155-157) for rows x in [x0,x1) directly into `out` (nx,nx,nx).

        use_img + c_img (nx^3, 32): dense tactile tensor as in eval_points;
        use_img + tips=(pos (F,3) float64, feat (F,32) cuda tensor, touch (F,) bool, radius):
        compact form of generation.py:190-200.  `minmax_key` (int32[2], init
        [INT32_MAX, INT32_MIN]) receives ordered-int keys of min/max logit.

        A feature batch of B > 1 scenes decodes all B lattices in one launch: `out` (B,nx,nx,nx) and
        `minmax_key` (B,2) (init [INT32_MAX, INT32_MIN] per row) receive each scene's logits and keys, bit for
        bit those of a B = 1 call on that scene's features (and fingertips).  Per-scene fingertips: use_img +
        tips=(pos (B,F,3) float64, feat (B,F,32) float32, touch (B,F) int32 — CUDA tensors, read at launch
        time — , radius); they go through the per-query byte map (tcgen05 variants).  Whole lattices only,
        without a dense c_img tensor or multi-GPU outputs."""
        dev = self.fc_out.weight.device
        if torch.is_grad_enabled():
            _abi.forbid_autograd(*self._param_tuple())
        feats = [t for k, t in c_plane.items() if k in ('grid',) + _PLANES and torch.is_tensor(t)]
        B = feats[0].size(0) if feats and self.c_dim != 0 else (out.size(0) if out is not None and out.dim() == 4 else 1)
        if B != 1 or (out is not None and out.dim() == 4):
            if x0 != 0 or (x1 is not None and x1 != nx) or peers or multicast:
                raise NotImplementedError('a batch of lattices is decoded whole, on one GPU (x0 = 0, x1 = nx, no peers)')
            if use_img and (c_img is not None or tip_map is not None):
                raise NotImplementedError('a batch of lattices takes tactile features as per-scene fingertips (tips)')
            return self._forward_dense_batch(c_plane, nx, B, out, minmax_key, axis, dev, use_img, tips)
        x1 = nx if x1 is None else x1
        if out is None:
            out = torch.empty((nx, nx, nx), dtype=torch.float32, device=dev)
        if tuple(out.shape) != (nx, nx, nx) or not out.is_contiguous():
            raise ValueError('out must be a contiguous (nx,nx,nx) tensor')
        a, keep = self._base_args(c_plane, 1, nx ** 3)
        if axis is None:
            axis = dense_axis(nx, self.padding, dev)
        a.axis = axis.data_ptr()
        a.nx, a.x0, a.x1 = nx, x0, x1
        a.use_img = int(use_img)
        if use_img and c_img is not None:
            _abi.require_cuda(c_img, 'c_img')
            cic = c_img.reshape(-1, 32).contiguous()
            if cic.size(0) != nx ** 3:
                raise ValueError('dense c_img must have nx^3 rows')
            a.c_img = cic.data_ptr()
        if use_img and tip_map is not None:       # (uint8 map (nx^3,), features (F,32)): tactile.tactile_point_map
            self._tip_map_args(a, keep, tip_map[0], tip_map[1], nx ** 3)
        elif use_img and tips is not None:
            pos, feat, touch, radius = tips
            F_ = len(pos)
            if F_ > _abi.MAX_TIPS:
                raise ValueError('at most %d tips' % _abi.MAX_TIPS)
            a.n_tips = F_
            for f in range(F_):
                for d in range(3):
                    a.tips[f][d] = float(pos[f][d])
                a.tip_touch[f] = int(bool(touch[f]))
            a.tip_radius = float(radius)
            _abi.require_cuda(feat, 'tip features')
            featc = feat.contiguous()
            a.tip_feat = featc.data_ptr()
        a.logits = out.data_ptr()
        if peers:  # fused all-gather: device pointers of every rank's (nx,nx,nx) grid (vtaco_b200.dist.FusedExchange)
            if len(peers) > 8:
                raise ValueError('at most 8 peers')
            a.n_peers = len(peers)
            for r, ptr_ in enumerate(peers):
                a.logits_peers[r] = int(ptr_)
            if multicast:
                a.logits_multicast = int(multicast)
        if minmax_key is not None:
            a.minmax_key = minmax_key.data_ptr()
        self._run(a, dev)
        return out

    def _forward_dense_batch(self, c_plane, nx, B, out, minmax_key, axis, dev, use_img=False, tips=None):
        """forward_dense of B scenes: one decoder launch over the B lattices, then the per-scene (min,max) keys
        in one reduction launch over the stored logits (vtaco_volume_keys: the reduction the decoder applies to
        a single scene)."""
        from ...mcubes import volume_keys
        if out is None:
            out = torch.empty((B, nx, nx, nx), dtype=torch.float32, device=dev)
        if tuple(out.shape) != (B, nx, nx, nx) or not out.is_contiguous() or out.dtype != torch.float32 \
                or out.device != dev:
            raise ValueError('out must be a contiguous float32 (%d,%d,%d,%d) tensor on %s' % (B, nx, nx, nx, dev))
        if minmax_key is not None and (minmax_key.dtype != torch.int32 or minmax_key.device != dev or
                                       tuple(minmax_key.shape) != (B, 2) or not minmax_key.is_contiguous()):
            raise ValueError('minmax_key must be a contiguous int32 (%d,2) tensor on %s' % (B, dev))
        a, keep = self._base_args(c_plane, B, B * nx ** 3)
        if axis is None:
            axis = dense_axis(nx, self.padding, dev)
        a.axis = axis.data_ptr()
        a.nx, a.x0, a.x1 = nx, 0, nx
        a.use_img = int(use_img)
        if use_img and tips is not None:
            from ..tactile import fingertip_lattice_ids
            pos, feat, touch, radius = tips
            if not (torch.is_tensor(feat) and feat.is_cuda and feat.dtype == torch.float32 and feat.dim() == 3
                    and tuple(feat.shape) == (B, pos.shape[1], 32)):
                raise ValueError('tip features must be a float32 CUDA tensor (%d,F,32)' % B)
            if pos.dim() != 3 or pos.shape[0] != B:
                raise ValueError('tips must hold the fingertips of %d scenes' % B)
            if a.variant not in (2, 4, 5, 6, 7):
                raise NotImplementedError('per-scene fingertips need a tcgen05 kernel variant (2, 4, 5, 6, 7)')
            ids = fingertip_lattice_ids(axis, pos, touch, radius)
            featc = feat.contiguous()
            a.tip_map, a.tip_feat, a.n_tips, a.tip_feat_per_sample = ids.data_ptr(), featc.data_ptr(), feat.shape[1], 1
            keep += [ids, featc]
        a.logits = out.data_ptr()
        self._run(a, dev)
        if minmax_key is not None:
            volume_keys(out, minmax_key)
        return out
