"""Time vtaco_encoder_backward alone at the shipped training shape: batches of 3 and 6 clouds of 3 640 points
(3 000 visual + 640 tactile), grid-64 features, max pooling, 5 blocks.  Prints ms per call (CUDA events, median of
7 windows of 20 calls) as one JSON line.  VTACO_B200_LIB selects the library, so two builds can be timed in turn."""
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from vtaco_b200.encoder import encoder_dict

T, R = 3640, 64


def cloud(rs, B):
    """points near a sphere, as a scanned surface gives: many points share a cell"""
    d = rs.randn(B, T, 3)
    p = 0.35 * d / np.linalg.norm(d, axis=2, keepdims=True) + 0.005 * rs.randn(B, T, 3)
    return torch.from_numpy(p.astype(np.float32)).cuda()


def main():
    torch.manual_seed(0)
    rs = np.random.RandomState(0)
    res = {'gpu': torch.cuda.get_device_name()}
    for B in (3, 6):
        enc = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, plane_type='grid',
                                                  grid_resolution=R).cuda().train()
        with torch.no_grad():
            for b in enc.blocks:
                b.fc_1.weight.normal_(0, 0.1)
        p = cloud(rs, B)
        w = enc._packed_weights()
        # channels-last storage, as the kernel reads it: no copy inside the timed call
        g = {'grid': torch.randn(B, R, R, R, 32, device='cuda').permute(0, 4, 1, 2, 3)}
        for _ in range(5):
            enc._pointnet_backward(p, w, g)
        ts = []
        for _ in range(7):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            a.record()
            for _ in range(20):
                enc._pointnet_backward(p, w, g)
            b.record()
            torch.cuda.synchronize()
            ts.append(a.elapsed_time(b) / 20)
        res['B%d_T%d_grid%d' % (B, T, R)] = {'ms_median': float(np.median(ts)), 'ms_min': float(min(ts))}
    print(json.dumps(res))


if __name__ == '__main__':
    main()
