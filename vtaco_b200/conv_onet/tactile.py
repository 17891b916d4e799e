"""Compact tactile conditioning (SURVEY §8f-1) — device-side replacements for the host code that
builds `c_img_all` in the reference: generation.py:172-200 (fingertip form), generation.py:202-255
(encode_t2d: back-projected tactile point clouds) and training.py:537-612 (training samples).

The reference materialises a dense (B, N, c_dim) tensor whose rows are either zero or one of <= 5
sensor features (2.1 GB at 256^3) after a scipy.cdist over all query points on the host.  Here the
same assignment is ONE byte per query, computed on the device (csrc/tactile.cu) and consumed by the
fused decoder (`tip_map`); `c_img_from_ids` expands it to the reference's dense tensor where a caller
wants that (it is what `LocalDecoder.forward_img` takes, and what autograd differentiates)."""
import ctypes as C

import numpy as np
import torch

from .. import _abi
from ..common import dense_axis


def fingertip_ids(p, tips, touch, radius=0.05):
    """ids (B,N) uint8: f+1 where f is the NEAREST fingertip of p[b,n] (float64, first minimum) if it is
    closer than `radius` and touch[b][f]; else 0  (generation.py:190-200, training.py:560-575).
    p (B,N,3) float32 CUDA; tips (B,F,3) or (F,3) array-like (float64 on the host); touch (B,F) or (F,)."""
    _abi.require_cuda(p, 'p')
    B, N = p.shape[0], p.shape[1]
    tips = np.asarray(tips, dtype=np.float64)
    touch = np.asarray(torch.as_tensor(touch).cpu() if torch.is_tensor(touch) else touch).astype(bool)
    if tips.ndim == 2:
        tips = np.broadcast_to(tips, (B,) + tips.shape)
    if touch.ndim == 1:
        touch = np.broadcast_to(touch, (B,) + touch.shape)
    F_ = tips.shape[1]
    if F_ > _abi.MAX_TIPS:
        raise ValueError('at most %d fingertips' % _abi.MAX_TIPS)
    pc = p.contiguous()
    ids = torch.empty((B, N), dtype=torch.uint8, device=p.device)
    L = _abi.lib()
    with torch.cuda.device(p.device):
        for b in range(B):
            tp = (C.c_double * (3 * F_))(*np.ascontiguousarray(tips[b]).reshape(-1))
            tc = (C.c_int32 * F_)(*[int(x) for x in touch[b]])
            st = L.vtaco_fingertip_ids(_abi.ptr(pc[b]), N, tp, tc, F_, float(radius), _abi.ptr(ids[b]),
                                       _abi.stream_ptr(p.device))
            _abi.check(st, 'fingertip_ids')
    return ids


def fingertip_lattice_ids(axis, tips, touch, radius=0.05, out=None):
    """ids (B,nx^3) uint8 of B dense lattices axis[nx]^3 with per-scene fingertips: ids[b, q] = f+1 where f is the
    nearest fingertip of scene b (float64, first minimum) if it is closer than `radius` and touch[b, f]; else 0 —
    the decoder's own in-kernel assignment.  axis (nx,) float32 CUDA; tips (B,F,3) float64 and touch (B,F) int32
    CUDA tensors, read by the launch (a captured graph re-reads them at replay)."""
    _abi.require_cuda(axis, 'axis')
    if not (torch.is_tensor(tips) and tips.is_cuda and tips.dtype == torch.float64 and tips.dim() == 3
            and tips.shape[2] == 3 and tips.is_contiguous()):
        raise ValueError('tips must be a contiguous float64 CUDA tensor (B,F,3)')
    B, F_ = tips.shape[0], tips.shape[1]
    if not (torch.is_tensor(touch) and touch.is_cuda and touch.dtype == torch.int32 and tuple(touch.shape) == (B, F_)
            and touch.is_contiguous()):
        raise ValueError('touch must be a contiguous int32 CUDA tensor (%d,%d)' % (B, F_))
    if not 1 <= F_ <= _abi.MAX_TIPS:
        raise ValueError('1 to %d fingertips per scene' % _abi.MAX_TIPS)
    nx = axis.numel()
    if out is None:
        out = torch.empty((B, nx ** 3), dtype=torch.uint8, device=axis.device)
    with torch.cuda.device(axis.device):
        _abi.check(_abi.lib().vtaco_fingertip_lattice_ids(_abi.ptr(axis), nx, B, _abi.ptr(tips), _abi.ptr(touch), F_,
                                                          float(radius), _abi.ptr(out), _abi.stream_ptr(axis.device)),
                   'fingertip_lattice_ids')
    return out


def tactile_point_map(points_per_sensor, touch, radius=0.015, p=None, nx=None, padding=0.1, device=None):
    """generation.py:222-255 (encode_t2d branch): map (N,) / (nx^3,) uint8 — t+1 for every query closer than
    `radius` to any point of sensor t's back-projected tactile cloud, sensors in increasing order (later ones
    overwrite), touched sensors only; 0 elsewhere.  points_per_sensor: list of (n_t, 3) float64 arrays (or None /
    empty); queries: `p` (N,3) float32 CUDA tensor, or the dense lattice (1+padding)*make_3d_grid(nx^3)."""
    dev = p.device if p is not None else torch.device(device)
    L = _abi.lib()
    if p is not None:
        _abi.require_cuda(p, 'p')
        pc = p.reshape(-1, 3).contiguous()
        n = pc.shape[0]
        out = torch.zeros(n, dtype=torch.uint8, device=dev)
        axis = None
    else:
        n = 0
        out = torch.zeros(nx ** 3, dtype=torch.uint8, device=dev)
        axis = dense_axis(nx, padding, dev)
    with torch.cuda.device(dev):
        for t, pts in enumerate(points_per_sensor):
            if pts is None or not bool(touch[t]):
                continue
            pts = torch.as_tensor(np.asarray(pts, dtype=np.float64).reshape(-1, 3), device=dev).contiguous()
            if pts.shape[0] == 0:
                continue
            st = L.vtaco_tactile_point_map(_abi.ptr(pc) if p is not None else None, n,
                                           _abi.ptr(axis) if axis is not None else None, nx or 0, _abi.ptr(pts),
                                           pts.shape[0], float(radius), t + 1, _abi.ptr(out), _abi.stream_ptr(dev))
            _abi.check(st, 'tactile_point_map')
    return out


def c_img_from_ids(ids, c_img):
    """The reference's dense tensor: c_img_all[b, n] = c_img[b, ids[b,n]-1] (zeros where ids == 0).
    ids (B,N) uint8, c_img (B,F,c_dim) -> (B,N,c_dim); differentiable w.r.t. c_img (an index op)."""
    B, Fn, Cd = c_img.shape
    table = torch.cat([c_img.new_zeros(B, 1, Cd), c_img], 1)
    return torch.gather(table, 1, ids.long().unsqueeze(-1).expand(-1, -1, Cd))


def build_training_samples(p, occ, c_img, tips, touch, num_sample, max_per_finger=512, radius=0.05, generator=None):
    """training.py:560-612 on the device: the query points near a touching fingertip (at most
    `max_per_finger` per finger, drawn WITH replacement like np.random.choice) come first in the
    sample, carrying that finger's feature; the rest of the `num_sample` points are drawn uniformly
    (with replacement) from the other points and carry zeros.  Returns (p_sample (B,S,3), occ_new (B,S),
    c_img_all (B,S,c_dim)).  The draws use torch's generator, not numpy's global state."""
    B, N, _ = p.shape
    dev = p.device
    ids = fingertip_ids(p, tips, touch, radius)
    p_out = torch.empty((B, num_sample, 3), dtype=p.dtype, device=dev)
    occ_out = torch.empty((B, num_sample), dtype=occ.dtype, device=dev)
    idc = torch.zeros((B, num_sample), dtype=torch.uint8, device=dev)
    for b in range(B):
        chosen, fid = [], []
        for f in range(c_img.shape[1]):
            sel = torch.nonzero(ids[b] == f + 1).flatten()
            if sel.numel() > max_per_finger:
                sel = sel[torch.randint(sel.numel(), (max_per_finger,), device=dev, generator=generator)]
            chosen.append(sel)
            fid.append(torch.full((sel.numel(),), f + 1, dtype=torch.uint8, device=dev))
        tip_idx = torch.cat(chosen)[:num_sample]
        k = tip_idx.numel()
        rest_mask = torch.ones(N, dtype=torch.bool, device=dev)
        rest_mask[tip_idx] = False
        rest = torch.nonzero(rest_mask).flatten()
        # the reference indexes p_new with positions drawn from range(len(sample_rest)) (training.py:603-606),
        # i.e. it draws from the FIRST len(sample_rest) points, not from sample_rest itself; kept as written
        draw = torch.randint(max(int(rest.numel()), 1), (num_sample - k,), device=dev, generator=generator)
        idx = torch.cat([tip_idx, draw])
        p_out[b] = p[b, idx]
        occ_out[b] = occ[b, idx]
        idc[b, :k] = torch.cat(fid)[:num_sample]
    return p_out, occ_out, c_img_from_ids(idc, c_img)
