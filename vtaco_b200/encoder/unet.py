"""2-D U-Net applied to the feature planes — state_dict-compatible with reference
src/encoder/unet.py:117-239 (down_convs.N.conv{1,2}, up_convs.N.{upconv,conv1,conv2},
conv_final).

CUDA inference (no grad, up_mode='transpose', merge_mode='concat' — the shipped kwargs) runs on our own
kernels (SURVEY §8f-3): every 3x3 / 1x1 convolution, with its bias and ReLU, is one launch of the tcgen05
implicit-GEMM kernel vtaco_conv3d_cl on the plane as a depth-1 channels-last volume (filter z-extent 1;
the skip connection is the kernel's second input, the concatenation is never
materialised); ConvTranspose2d(2, stride 2) is a 1x1 convolution to 4*Cout channels + vtaco_depth_to_space2_cl;
MaxPool2d(2) is vtaco_maxpool2d_cl.  Arithmetic: single-pass TF32 with fp32 accumulation, what the reference
runs on a GPU (cuDNN, allow_tf32).  Training / other modes use the torch.nn modules below (`fused = False`
forces them)."""
import ctypes as C

import torch
import torch.nn as nn
import torch.nn.functional as F

from .unet3d import _pack_conv_weight


class _Down(nn.Module):
    def __init__(self, cin, cout, pooling):
        super().__init__()
        self.conv1 = nn.Conv2d(cin, cout, 3, padding=1)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)
        self.pooling = pooling
        if pooling:
            self.pool = nn.MaxPool2d(2, 2)

    def forward(self, x):
        x = F.relu(self.conv2(F.relu(self.conv1(x))))
        return (self.pool(x) if self.pooling else x), x


class _Up(nn.Module):
    def __init__(self, cin, cout, merge_mode, up_mode):
        super().__init__()
        self.merge_mode = merge_mode
        if up_mode == 'transpose':
            self.upconv = nn.ConvTranspose2d(cin, cout, 2, stride=2)
        else:
            self.upconv = nn.Sequential(nn.Upsample(mode='bilinear', scale_factor=2), nn.Conv2d(cin, cout, 1))
        self.conv1 = nn.Conv2d(2 * cout if merge_mode == 'concat' else cout, cout, 3, padding=1)
        self.conv2 = nn.Conv2d(cout, cout, 3, padding=1)

    def forward(self, skip, x):
        x = self.upconv(x)
        x = torch.cat((x, skip), 1) if self.merge_mode == 'concat' else x + skip
        return F.relu(self.conv2(F.relu(self.conv1(x))))


class UNet(nn.Module):
    fused = True     # CUDA inference through our kernels (class-wide switch; per-instance override allowed)

    def __init__(self, num_classes, in_channels=3, depth=4, start_filts=32, up_mode='transpose',
                 merge_mode='concat', **kwargs):  # unknown keys (e.g. the YAML typo `start_flits`) are swallowed
        super().__init__()
        if up_mode not in ('transpose', 'upsample'):
            raise ValueError('"{}" is not a valid mode for upsampling. Only "transpose" and '
                             '"upsample" are allowed.'.format(up_mode))
        if merge_mode not in ('concat', 'add'):
            raise ValueError('"{}" is not a valid mode for merging up and down paths. '
                             'Only "concat" and "add" are allowed.'.format(up_mode))
        if up_mode == 'upsample' and merge_mode == 'add':
            raise ValueError('up_mode "upsample" is incompatible with merge_mode "add"')
        self.num_classes, self.in_channels, self.start_filts, self.depth = num_classes, in_channels, start_filts, depth
        self.up_mode, self.merge_mode = up_mode, merge_mode
        downs, ups = [], []
        outs = in_channels
        for i in range(depth):
            ins, outs = outs, start_filts * (2 ** i)
            downs.append(_Down(ins, outs, pooling=i < depth - 1))
        for i in range(depth - 1):
            ins, outs = outs, outs // 2
            ups.append(_Up(ins, outs, merge_mode, up_mode))
        self.down_convs = nn.ModuleList(downs)
        self.up_convs = nn.ModuleList(ups)
        self.conv_final = nn.Conv2d(outs, num_classes, 1)
        for m in self.modules():
            if isinstance(m, nn.Conv2d):  # reference weight_init (ConvTranspose2d keeps its default)
                nn.init.xavier_normal_(m.weight)
                nn.init.constant_(m.bias, 0)

    # ------------------------------------------------------------------ fused CUDA inference path
    def _fusable(self, x):
        if not (self.fused and x.is_cuda and x.dtype == torch.float32 and x.dim() == 4):
            return False
        if self.up_mode != 'transpose' or self.merge_mode != 'concat':
            return False
        if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for p in self.parameters())):
            return False
        chans = [self.in_channels] + [self.start_filts * 2 ** i for i in range(self.depth)]
        if any(c % 16 for c in chans) or any(c % 32 for c in chans[1:]) or self.num_classes % 32 or 2 * chans[-1] > 512:
            return False
        H, W = x.shape[2:]
        return H % (2 ** (self.depth - 1)) == 0 and W % (2 ** (self.depth - 1)) == 0

    def invalidate(self):
        """Drop the packed-weight cache (keyed on (data_ptr, _version) of each weight / bias: an update made through
        `param.data` does not bump `_version` — call this after one; LocalPoolPointnet.invalidate() does)."""
        self.__dict__['_wcache'] = {}

    def _packed(self, key, conv, kind):
        """operand buffers of a layer, cached per parameter version: (packed weights, bias)."""
        ver = (conv.weight.data_ptr(), conv.weight._version, conv.bias.data_ptr(), conv.bias._version)
        cache = self.__dict__.setdefault('_wcache', {})
        hit = cache.get(key)
        if hit is None or hit[0] != ver:
            w = conv.weight.detach().float()
            if kind == 'conv3':        # (Cout, Cin, 3, 3): a filter of z-extent 1 (vtaco_conv3d_args.ksize_z = 1)
                w5 = w.reshape(w.shape[0], w.shape[1], 1, 3, 3)
                b = conv.bias.detach().float().contiguous()
            elif kind == 'conv1':      # (Cout, Cin, 1, 1)
                w5 = w.reshape(w.shape[0], w.shape[1], 1, 1, 1)
                b = conv.bias.detach().float().contiguous()
            else:                      # ConvTranspose2d (Cin, Cout, 2, 2) -> 1x1 conv to (a*2+b)*Cout + co
                w5 = w.permute(2, 3, 1, 0).reshape(4 * w.shape[1], w.shape[0], 1, 1, 1)
                b = conv.bias.detach().float().repeat(4).contiguous()
            hit = (ver, _pack_conv_weight(w5), b)
            cache[key] = hit
        return hit[1], hit[2]

    def _conv(self, x, x2, wp, bias, cout, ksize, relu):
        """one fused layer on channels-last planes (N,H,W,C) [+ second input (N,H,W,C2)]."""
        from .. import _abi
        N, H, W, C1 = x.shape
        a = _abi.Conv3dArgs()
        a.x, a.N, a.D, a.H, a.W, a.C1 = x.data_ptr(), N, 1, H, W, C1
        if x2 is not None:
            a.x2, a.C2, a.D2, a.H2, a.W2 = x2.data_ptr(), x2.shape[3], 1, x2.shape[1], x2.shape[2]
        a.w_packed, a.bias = wp.data_ptr(), bias.data_ptr()
        a.Cout, a.ksize, a.ksize_z, a.relu = cout, ksize, 1, int(relu)
        y = torch.empty((N, H, W, cout), dtype=torch.float32, device=x.device)
        a.y = y.data_ptr()
        with torch.cuda.device(x.device):
            st = _abi.lib().vtaco_conv3d_cl(C.byref(a), _abi.stream_ptr(x.device))
        _abi.check(st, 'conv3d_cl')
        return y

    def _forward_fused(self, x):
        from .. import _abi
        L = _abi.lib()
        dev = x.device
        cur = x.permute(0, 2, 3, 1)
        if not cur.is_contiguous():
            cur = cur.contiguous()
        stream = _abi.stream_ptr(dev)
        skips = []
        for i, d in enumerate(self.down_convs):
            cur = self._conv(cur, None, *self._packed(('d1', i), d.conv1, 'conv3'), d.conv1.out_channels, 3, True)
            cur = self._conv(cur, None, *self._packed(('d2', i), d.conv2, 'conv3'), d.conv2.out_channels, 3, True)
            skips.append(cur)
            if d.pooling:
                N, H, W, Cc = cur.shape
                y = torch.empty((N, H // 2, W // 2, Cc), dtype=torch.float32, device=dev)
                with torch.cuda.device(dev):
                    _abi.check(L.vtaco_maxpool2d_cl(_abi.ptr(cur), _abi.ptr(y), N, H, W, Cc, stream), 'maxpool2d_cl')
                cur = y
        for i, u in enumerate(self.up_convs):
            skip = skips[-(i + 2)]
            cout = u.upconv.out_channels
            t = self._conv(cur, None, *self._packed(('up', i), u.upconv, 'convT'), 4 * cout, 1, False)
            N, H, W, _ = t.shape
            up = torch.empty((N, 2 * H, 2 * W, cout), dtype=torch.float32, device=dev)
            with torch.cuda.device(dev):
                _abi.check(L.vtaco_depth_to_space2_cl(_abi.ptr(t), _abi.ptr(up), N, H, W, cout, stream), 'depth_to_space2_cl')
            # torch.cat((from_up, from_down), 1): the up-sampled tensor first, then the skip
            cur = self._conv(up, skip, *self._packed(('u1', i), u.conv1, 'conv3'), u.conv1.out_channels, 3, True)
            cur = self._conv(cur, None, *self._packed(('u2', i), u.conv2, 'conv3'), u.conv2.out_channels, 3, True)
        out = self._conv(cur, None, *self._packed(('fin', 0), self.conv_final, 'conv1'), self.num_classes, 1, False)
        return out.permute(0, 3, 1, 2)     # (N, C, H, W) in channels_last memory format: the decoder reads it as is

    def forward(self, x):
        if self._fusable(x):
            return self._forward_fused(x)
        skips = []
        for d in self.down_convs:
            x, before = d(x)
            skips.append(before)
        for i, u in enumerate(self.up_convs):
            x = u(skips[-(i + 2)], x)
        return self.conv_final(x)
