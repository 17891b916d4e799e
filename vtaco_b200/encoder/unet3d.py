"""3-D U-Net applied to the feature grid — state_dict-compatible with reference
src/encoder/unet3d.py:361-491 (encoders.N.basic_module.SingleConv{1,2}.{groupnorm,conv,...},
decoders.N.basic_module..., final_conv).

Inference on CUDA runs on our own kernels (SURVEY §8f-3, csrc/conv3d.cu): every 'gcr' layer is one
tcgen05 implicit-GEMM kernel over channels-last activations with GroupNorm-apply, nearest-upsample +
concat, ReLU and the next layer's GroupNorm statistics fused in; the output is written in the
decoder's channels-last layout.  Arithmetic: single-pass TF32 with fp32 accumulation, i.e. what the
reference computes on a GPU (cuDNN, torch.backends.cudnn.allow_tf32 = True by default); set
`UNet3D.fused = False` for the torch.nn / cuDNN modules (used for training: autograd)."""
from collections import OrderedDict

import torch
import torch.nn as nn
import torch.nn.functional as F


class GroupNorm(nn.GroupNorm):
    """nn.GroupNorm with the same parameters / state_dict; on CUDA fp32 inference it runs
    vtaco_group_norm (chip-wide reduction) instead of ATen's one-block-per-group kernel."""
    prefer_channels_last = False

    def forward(self, x):
        if (x.is_cuda and x.dtype == torch.float32 and x.dim() >= 3
                and not (torch.is_grad_enabled() and (x.requires_grad or self.weight.requires_grad))):
            from .. import _abi
            N, Cc = x.shape[0], x.shape[1]
            S = x[0, 0].numel()
            ws = torch.empty(2 * N * self.num_groups, dtype=torch.float64, device=x.device)
            perm = (0,) + tuple(range(2, x.dim())) + (1,)
            cpg = Cc // self.num_groups
            # channels-last kernel only on request: measured on B200, cuDNN's fp32 Conv3d is not faster in
            # channels_last_3d at these sizes (UNet3D 64^3 x 32: e2e 5.27 ms contiguous vs 5.48 ms channels-last)
            if (self.prefer_channels_last and x.dim() in (4, 5) and x.permute(*perm).is_contiguous() and Cc % 4 == 0 and cpg % 4 == 0
                    and 256 % (Cc // 4) == 0 and self.num_groups <= 64):
                y = torch.empty_like(x)          # keeps the channels-last strides
                with torch.cuda.device(x.device):
                    st = _abi.lib().vtaco_group_norm_cl(_abi.ptr(x), _abi.ptr(y), _abi.ptr(self.weight),
                                                        _abi.ptr(self.bias), N, Cc, self.num_groups, S, float(self.eps),
                                                        _abi.ptr(ws), _abi.stream_ptr(x.device))
                _abi.check(st, 'group_norm_cl')
                return y
            xc = x.contiguous()
            y = torch.empty_like(xc)
            with torch.cuda.device(x.device):
                st = _abi.lib().vtaco_group_norm(_abi.ptr(xc), _abi.ptr(y), _abi.ptr(self.weight), _abi.ptr(self.bias),
                                                 N, Cc, self.num_groups, S, float(self.eps), _abi.ptr(ws),
                                                 _abi.stream_ptr(x.device))
            _abi.check(st, 'group_norm')
            return y
        return super().forward(x)


def _upsample_concat(skip, x):
    """cat(skip, interpolate(x, size=skip.shape[2:], mode='nearest'), dim=1) (reference unet3d.py
    Decoder.forward); one fused kernel on CUDA fp32 inference, the two ATen ops otherwise."""
    if (skip.is_cuda and x.is_cuda and skip.dtype == torch.float32 and x.dtype == torch.float32 and skip.dim() == 5
            and skip.size(4) % 4 == 0 and skip.is_contiguous() and x.is_contiguous()
            and not (torch.is_grad_enabled() and (skip.requires_grad or x.requires_grad))):
        from .. import _abi
        N, C1, Do, Ho, Wo = skip.shape
        C2, Di, Hi, Wi = x.shape[1:]
        out = torch.empty((N, C1 + C2, Do, Ho, Wo), dtype=torch.float32, device=skip.device)
        L = _abi.lib()
        with torch.cuda.device(skip.device):
            st = L.vtaco_upsample_concat3d(_abi.ptr(skip), _abi.ptr(x), _abi.ptr(out), N, C1, C2, Do, Ho, Wo, Di, Hi, Wi,
                                           _abi.stream_ptr(skip.device))
        _abi.check(st, 'upsample_concat3d')
        return out
    x = F.interpolate(x, size=skip.size()[2:], mode='nearest')
    return torch.cat((skip, x), dim=1)


def _single_conv(cin, cout, order, num_groups, kernel_size=3, padding=1):
    assert 'c' in order, 'Conv layer MUST be present'
    assert order[0] not in 'rle', 'Non-linearity cannot be the first operation in the layer'
    mods = OrderedDict()
    for i, ch in enumerate(order):
        if ch == 'r':
            mods['ReLU'] = nn.ReLU(inplace=True)
        elif ch == 'l':
            mods['LeakyReLU'] = nn.LeakyReLU(negative_slope=0.1, inplace=True)
        elif ch == 'e':
            mods['ELU'] = nn.ELU(inplace=True)
        elif ch == 'c':
            mods['conv'] = nn.Conv3d(cin, cout, kernel_size, padding=padding, bias=not ('g' in order or 'b' in order))
        elif ch == 'g':
            nch = cin if i < order.index('c') else cout
            groups = 1 if nch < num_groups else num_groups
            assert nch % groups == 0
            mods['groupnorm'] = GroupNorm(num_groups=groups, num_channels=nch)
        elif ch == 'b':
            mods['batchnorm'] = nn.BatchNorm3d(cin if i < order.index('c') else cout)
        else:
            raise ValueError("Unsupported layer type '%s'. MUST be one of ['b', 'g', 'r', 'l', 'e', 'c']" % ch)
    return nn.Sequential(mods)


def _double_conv(cin, cout, encoder, order, num_groups):
    if encoder:
        c1 = max(cout // 2, cin)
        shapes = ((cin, c1), (c1, cout))
    else:
        shapes = ((cin, cout), (cout, cout))
    return nn.Sequential(OrderedDict([
        ('SingleConv1', _single_conv(shapes[0][0], shapes[0][1], order, num_groups)),
        ('SingleConv2', _single_conv(shapes[1][0], shapes[1][1], order, num_groups))]))


class _Encoder(nn.Module):
    def __init__(self, cin, cout, apply_pooling, order, num_groups):
        super().__init__()
        self.pooling = nn.MaxPool3d(kernel_size=(2, 2, 2)) if apply_pooling else None
        self.basic_module = _double_conv(cin, cout, True, order, num_groups)

    def forward(self, x):
        if self.pooling is not None:
            x = self.pooling(x)
        return self.basic_module(x)


class _Decoder(nn.Module):
    def __init__(self, cin, cout, order, num_groups):
        super().__init__()
        self.basic_module = _double_conv(cin, cout, False, order, num_groups)

    def forward(self, skip, x):
        return self.basic_module(_upsample_concat(skip, x))


def _pack_conv_weight(w):
    """(Cout, Cin, kD, kH, kW) -> the tcgen05 operand layout of vtaco_conv3d_cl (include/vtaco_b200.h),
    values rounded to nearest TF32."""
    Cout, Cin = w.shape[0], w.shape[1]
    taps = w.shape[2] * w.shape[3] * w.shape[4]
    wt = w.detach().float().reshape(Cout // 32, 32, Cin // 16, 4, 4, taps)       # [nt][n][ch][kc][kk][tap]
    wt = wt.permute(0, 2, 5, 3, 1, 4).contiguous()                               # [nt][ch][tap][kc][n][kk]
    wt = ((wt.view(torch.int32) + 0x1000) & ~0x1fff).view(torch.float32)
    return wt.reshape(-1)


class UNet3D(nn.Module):
    fused = True     # CUDA inference through vtaco_conv3d_cl (class-wide switch; per-instance override allowed)

    def __init__(self, in_channels, out_channels, final_sigmoid=True, f_maps=64, layer_order='gcr',
                 num_groups=8, num_levels=4, is_segmentation=True, testing=False, **kwargs):
        super().__init__()
        self.testing = testing
        self.layer_order = layer_order
        self._wcache = {}
        if isinstance(f_maps, int):
            f_maps = [f_maps * 2 ** k for k in range(num_levels)]
        self.encoders = nn.ModuleList([
            _Encoder(in_channels if i == 0 else f_maps[i - 1], f, i > 0, layer_order, num_groups)
            for i, f in enumerate(f_maps)])
        rev = list(reversed(f_maps))
        self.decoders = nn.ModuleList([
            _Decoder(rev[i] + rev[i + 1], rev[i + 1], layer_order, num_groups) for i in range(len(rev) - 1)])
        self.final_conv = nn.Conv3d(f_maps[0], out_channels, 1)
        if is_segmentation:
            self.final_activation = nn.Sigmoid() if final_sigmoid else nn.Softmax(dim=1)
        else:
            self.final_activation = None

    # ------------------------------------------------------------------ fused CUDA inference path
    def _fusable(self, x):
        if not (self.fused and x.is_cuda and x.dtype == torch.float32 and x.dim() == 5 and self.layer_order == 'gcr'):
            return False
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            return False
        if self.testing and self.final_activation is not None:
            return False
        if getattr(self, '_fusable_static', None) is None:   # the module tree does not change after construction
            convs = [m for m in self.modules() if isinstance(m, nn.Conv3d)]
            ok = all(c.in_channels % 16 == 0 and c.out_channels % 32 == 0 and c.in_channels <= 512 and
                     c.kernel_size[0] in (1, 3) and c.kernel_size[0] == c.kernel_size[1] == c.kernel_size[2] for c in convs)
            self._fusable_static = (ok, sum(1 for e in self.encoders if e.pooling is not None))
        ok, n_pool = self._fusable_static
        D, H, W = x.shape[2:]
        return ok and all(d % (2 ** n_pool) == 0 for d in (D, H, W))

    def invalidate(self):
        """Drop the packed-weight cache (keyed on (data_ptr, _version) of each weight: an update made through
        `param.data` does not bump `_version` — call this after one; LocalPoolPointnet.invalidate() does)."""
        self._wcache = {}
        self._fusable_static = None

    def _packed(self, conv):
        key = (id(conv), conv.weight.data_ptr(), conv.weight._version)
        hit = self._wcache.get(id(conv))
        if hit is None or hit[0] != key:
            hit = (key, _pack_conv_weight(conv.weight))
            self._wcache[id(conv)] = hit
        return hit[1]

    def _conv(self, x, x2, gn, conv, in_stats, relu, want_stats):
        """one fused layer on channels-last tensors (N,D,H,W,C); returns (y, y_stats | None)."""
        from .. import _abi
        import ctypes as C
        N, D, H, W, C1 = x.shape
        a = _abi.Conv3dArgs()
        a.x, a.N, a.D, a.H, a.W, a.C1 = x.data_ptr(), N, D, H, W, C1
        if x2 is not None:
            a.x2, a.C2, a.D2, a.H2, a.W2 = x2.data_ptr(), x2.shape[4], x2.shape[1], x2.shape[2], x2.shape[3]
        wp = self._packed(conv)
        a.w_packed = wp.data_ptr()
        if conv.bias is not None:
            a.bias = conv.bias.data_ptr()
        a.Cout, a.ksize = conv.out_channels, conv.kernel_size[0]
        if gn is not None:
            a.in_stats = in_stats.data_ptr()
            a.gamma, a.beta = gn.weight.data_ptr(), gn.bias.data_ptr()
            a.groups, a.eps = gn.num_groups, float(gn.eps)
        a.relu = int(relu)
        y = torch.empty((N, D, H, W, conv.out_channels), dtype=torch.float32, device=x.device)
        a.y = y.data_ptr()
        ys = None
        if want_stats:
            ys = self._take_stats(N, conv.out_channels)
            a.out_stats = ys.data_ptr()
        with torch.cuda.device(x.device):
            st = _abi.lib().vtaco_conv3d_cl(C.byref(a), _abi.stream_ptr(x.device))
        _abi.check(st, 'conv3d_cl')
        return y, ys

    def _take_stats(self, N, C):
        """(N, C, 2) float64 slice of the forward's statistics arena (zeroed once per forward)."""
        n = N * C * 2
        out = self._arena[self._arena_pos:self._arena_pos + n].view(N, C, 2)
        self._arena_pos += n
        return out

    def _forward_fused(self, x):
        from .. import _abi
        L = _abi.lib()
        dev = x.device
        cur = x.permute(0, 2, 3, 4, 1)
        if not cur.is_contiguous():
            cur = cur.contiguous()
        N = cur.shape[0]
        stream = _abi.stream_ptr(dev)
        convs = [m for m in self.modules() if isinstance(m, nn.Conv3d)]
        total = cur.shape[4] + sum(c.out_channels for c in convs) + sum(c.in_channels for c in convs)   # generous bound
        self._arena = torch.zeros(N * 2 * total, dtype=torch.float64, device=dev)     # one fill instead of one per layer
        self._arena_pos = 0
        with torch.cuda.device(dev):
            stats = self._take_stats(N, cur.shape[4])
            for n in range(N):
                _abi.check(L.vtaco_channel_stats_cl(_abi.ptr(cur[n]), cur[n].numel() // cur.shape[4], cur.shape[4],
                                                    _abi.ptr(stats[n]), stream), 'channel_stats_cl')
            feats = []
            for enc in self.encoders:
                if enc.pooling is not None:
                    _, D, H, W, Cc = cur.shape
                    nxt = torch.empty((N, D // 2, H // 2, W // 2, Cc), dtype=torch.float32, device=dev)
                    stats = self._take_stats(N, Cc)
                    for n in range(N):
                        _abi.check(L.vtaco_maxpool2_cl(_abi.ptr(cur[n]), _abi.ptr(nxt[n]), 1, D, H, W, Cc,
                                                       _abi.ptr(stats[n]), stream), 'maxpool2_cl')
                    cur = nxt
                for sc in (enc.basic_module.SingleConv1, enc.basic_module.SingleConv2):
                    cur, stats = self._conv(cur, None, sc.groupnorm, sc.conv, stats, True, True)
                feats.insert(0, (cur, stats))
            for dec, (skip, skip_stats) in zip(self.decoders, feats[1:]):
                # cat(skip, nearest-upsample(cur)) is never materialised: its per-channel sums are the skip's
                # and 8x the half-resolution tensor's (every voxel is replicated 2x2x2 times)
                if tuple(skip.shape[1:4]) != tuple(2 * d for d in cur.shape[1:4]):
                    raise NotImplementedError('fused UNet3D needs exact 2x upsampling')
                cat_stats = torch.cat([skip_stats, 8.0 * stats], 1).contiguous()
                sc1, sc2 = dec.basic_module.SingleConv1, dec.basic_module.SingleConv2
                cur, stats = self._conv(skip, cur, sc1.groupnorm, sc1.conv, cat_stats, True, True)
                cur, stats = self._conv(cur, None, sc2.groupnorm, sc2.conv, stats, True, True)
            cur, _ = self._conv(cur, None, None, self.final_conv, None, False, False)
        return cur.permute(0, 4, 1, 2, 3)       # (N,C,D,H,W) in channels_last_3d memory format

    def forward(self, x):
        if self._fusable(x):
            return self._forward_fused(x)
        feats = []
        for enc in self.encoders:
            x = enc(x)
            feats.insert(0, x)
        for dec, skip in zip(self.decoders, feats[1:]):
            x = dec(skip, x)
        x = self.final_conv(x)
        if self.testing and self.final_activation is not None:
            x = self.final_activation(x)
        return x
