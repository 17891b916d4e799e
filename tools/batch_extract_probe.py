"""Scenes per second of batched mesh extraction against a loop of single-scene extractions.

For B in {1, 4, 16} scenes and lattices of nx in {64, 128, 256} points per axis, both paths run from a pinned
host point cloud to meshes in device memory (H2D copy, encoder with UNet3D, lattice decode, iso-level, marching
cubes), each captured as a CUDA graph:
  * batched: one graph of Generator3D.lattices_and_meshes over the B clouds;
  * loop: the single-scene graph (Generator3D.lattice_and_mesh) replayed B times back to back, with no host
    synchronisation between the scenes (a lower bound for a loop that reads each scene's mesh counters).
A timed step is one batch of B scenes between CUDA events; a 256 MiB write flushes the L2 between steps, as in
bench.py.  Every captured graph has its own model instance: module workspaces (the PointNet encoder's grows with
the batch) are baked into a graph, so a graph must not share them with one captured for another batch size.  The
decoder and the marching-cubes pass of the batched path are also timed on their own (eager
launches, L2 flushed before each).  Both paths decode with five fingertips per scene (the bench.py configuration,
with_img): the single-scene graph with the in-kernel fingertip test, the batched one with the per-scene byte map
(vtaco_fingertip_lattice_ids) and per-scene tip tables.  The card name and power limit are read in the same run.

    python tools/batch_extract_probe.py [--out profiles/batch_extract_probe.json] [--steps 10]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from bench import build_models  # noqa: E402
from vtaco_b200.conv_onet.generation import Generator3D  # noqa: E402
from vtaco_b200.mcubes import new_minmax_key, volume_keys  # noqa: E402


def card():
    info = {'name': torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(['nvidia-smi', '--query-gpu=power.limit,clocks.max.sm', '--format=csv,noheader'],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        info['power_limit'], info['sm_max_clock'] = [x.strip() for x in q.split(',')]
    except Exception as e:   # the numbers are still recorded, marked without a power limit
        info['power_limit'] = 'unavailable (%s)' % type(e).__name__
    return info


def timed(fn, flush, steps, warmup=2):
    """median / min milliseconds of fn() between CUDA events, L2 flushed before each step"""
    for _ in range(warmup):
        fn()
    ts = []
    for s in range(steps):
        flush.fill_(float(s))
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return float(np.median(ts)), float(np.min(ts))


def clouds(B, seed=0):
    rs = np.random.RandomState(seed)
    return torch.from_numpy(rs.uniform(-0.5, 0.5, size=(B, 3000, 3)).astype(np.float32)).pin_memory()


def fingertips(B, seed=0):
    """five fingertips per scene, four of them touching (bench.py's synthetic scene, one draw per scene)"""
    rs = np.random.RandomState(seed)
    pos = rs.uniform(-0.35, 0.35, size=(B, 5, 3))
    feat = rs.randn(B, 5, 32).astype(np.float32)
    touch = np.tile(np.array([1, 1, 0, 1, 1], dtype=np.int32), (B, 1))
    return pos, feat, touch


def capture(fn):
    with torch.no_grad():
        for _ in range(2):
            out = fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fn()
    return g, out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(ROOT, 'profiles', 'batch_extract_probe.json'))
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--nx', type=int, nargs='+', default=[64, 128, 256])
    ap.add_argument('--batch', type=int, nargs='+', default=[1, 4, 16])
    args = ap.parse_args()
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)
    rows = []
    for nx in args.nx:
        net1 = build_models(dev)
        single = Generator3D(net1, device=dev, resolution0=nx // 4, padding=0.1, input_type='pointcloud',
                             with_img=True)
        one = clouds(1)
        p1, f1, t1 = fingertips(1)
        tips1 = (p1[0], torch.from_numpy(f1[0]).to(dev), t1[0].astype(bool), 0.05)
        one_dev = torch.empty(one.shape, device=dev)

        def single_body():
            one_dev.copy_(one, non_blocking=True)
            return single.lattice_and_mesh(net1.encode_inputs(one_dev), tips=tips1)

        with torch.no_grad():   # mesh buffers sized before the capture (as capture_generate does)
            out = single_body()
            V, F = [int(x) for x in out[2][:2].cpu()]
            single.mc._ensure(0, int(V * 1.5) + 16, int(F * 1.5) + 16)
        g1, _ = capture(single_body)
        for B in args.batch:
            net = build_models(dev)
            gen = Generator3D(net, device=dev, resolution0=nx // 4, padding=0.1, input_type='pointcloud',
                              with_img=True)
            host = clouds(B)
            pB, fB, tB = fingertips(B)
            tipsB = (torch.from_numpy(pB).to(dev), torch.from_numpy(fB).to(dev), torch.from_numpy(tB).to(dev), 0.05)
            host_dev = torch.empty(host.shape, device=dev)

            def batch_body():
                host_dev.copy_(host, non_blocking=True)
                return gen.lattices_and_meshes(net.encode_inputs(host_dev), tipsB)

            with torch.no_grad():
                out = batch_body()
                V, F = [int(x) for x in out[2][:2].cpu()]
                gen._batch_mc._ensure(0, int(V * 1.5) + 16, int(F * 1.5) + 16)
            gB, outB = capture(batch_body)
            t_batch = timed(gB.replay, flush, args.steps)

            def loop():
                for _ in range(B):
                    g1.replay()
            t_loop = timed(loop, flush, args.steps)
            # kernels of the batched path on their own (eager), from the captured graph's features
            with torch.no_grad():
                c = net.encode_inputs(host_dev)
                grid = torch.empty((B, nx, nx, nx), device=dev)
                keys0 = new_minmax_key(dev, B)
                keys = keys0.clone()
                axis = gen._batch[3]

                def dec():
                    keys.copy_(keys0)
                    net.decoder.forward_dense(c, nx, use_img=True, tips=tipsB, out=grid, minmax_key=keys, axis=axis)
                t_dec = timed(dec, flush, args.steps)
                t_keys = timed(lambda: volume_keys(grid, keys), flush, args.steps)
                t_mc = timed(lambda: gen._batch_mc.batch(grid, level_keys=keys, sync=False), flush, args.steps)
                dec_one = timed(lambda: net.decoder.forward_dense({k: v[:1] for k, v in c.items()}, nx, use_img=True,
                                                                  tips=tips1, out=grid[0], axis=axis),
                                flush, args.steps)
                mc_one = timed(lambda: gen._batch_mc(grid[0], level_keys=keys[0], sync=False), flush, args.steps)
            sc = outB[3].cpu()
            row = {'nx': nx, 'B': B,
                   'batched_graph_ms': t_batch[0], 'batched_graph_min_ms': t_batch[1],
                   'loop_of_single_graphs_ms': t_loop[0], 'loop_of_single_graphs_min_ms': t_loop[1],
                   'batched_scenes_per_s': 1e3 * B / t_batch[0], 'loop_scenes_per_s': 1e3 * B / t_loop[0],
                   'speedup': t_loop[0] / t_batch[0],
                   'batched_decoder_ms': t_dec[0], 'batched_volume_keys_ms': t_keys[0], 'batched_mc_ms': t_mc[0],
                   'single_decoder_ms': dec_one[0], 'single_mc_ms': mc_one[0],
                   'faces_per_scene': [int(x) for x in sc[:, 1]]}
            print(json.dumps(row), flush=True)
            rows.append(row)
            del gB, outB, gen, grid, c, net
            torch.cuda.empty_cache()
        del g1, single, net1
        torch.cuda.empty_cache()
    res = {'card': card(), 'steps': args.steps,
           'workload': 'bench.py models (PointNet + UNet3D grid-64 encoder, 5-block decoder, variant 7), 3000-point '
                       'uniform clouds, five fingertips per scene (four touching); L2 flushed (256 MiB write) before every timed step',
           'rows': rows}
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, 'w') as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res['card']))


if __name__ == '__main__':
    main()
