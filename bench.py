#!/usr/bin/env python
"""bench.py — occupancy query-points/sec of the conv-occupancy hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json configs[3], the one the metric's target is quoted on: "decodes a
256^3 occupancy grid"): VTacOH_YCB shapes — LocalPoolPointnet(grid 64^3, hidden 32) +
UNet3D features, LocalDecoder(simple_local, hidden 32, 5 blocks, forward_img with
fingertip conditioning), dense 256^3 lattice (resolution_0 = 64), marching cubes at
level 0.5*(min+max).  Synthetic cloud (3000 visual + 5x128 tactile points), random-init
weights (fc_1 re-randomised, it is zero-initialised in the reference).

A step = one pass over the whole lattice: fused decode of nx^3 queries + marching cubes.  N>1:
x-slabs over the ranks, every rank extracts the mesh piece of its slab and the pieces are gathered
on rank 0 (device-side signalling over NVLink peer memory; --exchange selects the older schemes).
`value`  : nx^3 / step time, features already resident in HBM (device timed, CUDA events); they are computed
           once on the host (host_grid_features), so that every run decodes the same bits.
`e2e`    : the same through Generator3D.capture_generate with HOST buffers: pinned point
           cloud -> H2D -> encoder (PointNet kernels + UNet3D) [-> broadcast] -> decode -> MC -> mesh D2H.
`--impl reference`: the reference's CPU implementation of the path (the oracle port: same
           torch CPU ops as the reference's modules + the numpy marching-cubes restatement; the
           reference is Python and is not present on the GPU box) on a bounded sample of the lattice.
`identity_ok` (N>1): the mesh assembled from the ranks' pieces equals, bit for bit, the mesh rank 0
           computes alone from the same features (checked before the timed region).
`--dump-outputs DIR` (N=1): after the timed steps, what the last step computed as DIR/<name>.npy, so that
           two builds can be compared output for output (see dump_outputs).
"""
import argparse
import json
import os
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = 'occupancy query-points/sec (dense lattice decode + marching cubes)'
UNIT = 'query-points/s'
FLOP_PER_QUERY = 30976          # algorithmic MLP FLOPs/query (LocalDecoder.forward; SURVEY §8a a12)
FLOP_PER_QUERY_IMG = 33024      # forward_img with a dense c_img tensor
DUMP_BYTES = 64 << 20           # --dump-outputs: upper bound of all files together
DUMP_LOGITS = 1 << 20           # --dump-outputs: lattice points in the logit sample


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# --------------------------------------------------------------------------------------
# synthetic scene (SURVEY §8d)
# --------------------------------------------------------------------------------------
def synthetic_scene(seed=0):
    rs = np.random.RandomState(seed)
    vis = rs.uniform(-0.5, 0.5, size=(3000, 3))
    tips = rs.uniform(-0.35, 0.35, size=(5, 3))
    tac = (tips[:, None, :] + rs.randn(5, 128, 3) * 0.01).reshape(-1, 3)
    cloud = (np.concatenate([vis, tac], 0) + rs.randn(3640, 3) * 0.005).astype(np.float32)
    tip_feat = rs.randn(5, 32).astype(np.float32)
    touch = np.array([True, True, False, True, True])
    return cloud, tips.astype(np.float64), tip_feat, touch


def build_models(device, seed=0):
    from vtaco_b200.encoder import encoder_dict
    from vtaco_b200.conv_onet.models import decoder_dict, ConvolutionalOccupancyNetwork
    torch.manual_seed(seed)
    enc = encoder_dict['pointnet_local_pool'](dim=3, c_dim=32, padding=0.1, hidden_dim=32, plane_type='grid',
                                              grid_resolution=64, unet3d=True,
                                              unet3d_kwargs=dict(num_levels=4, f_maps=32, in_channels=32,
                                                                 out_channels=32))
    dec = decoder_dict['simple_local'](dim=3, c_dim=32, padding=0.1, with_contact=False, sample_mode='bilinear',
                                       hidden_size=32)
    with torch.no_grad():
        for m in (enc, dec):
            for b in m.blocks:
                b.fc_1.weight.normal_(0, 0.1)
    return ConvolutionalOccupancyNetwork(dec, enc, device=device).eval()


def host_grid_features(net, cloud):
    """The encoder's grid features of `cloud` (numpy (T, 3)) computed on the host by the reference computation
    (the oracle's PointNet and the UNet3D modules' torch.nn path, fp32): (1, 32, 64, 64, 64) float32.
    The timed step decodes these so that its input is the same bits on every run; the GPU encoder sums the
    grid's scatter-mean and its GroupNorm statistics with atomics, whose order varies from run to run.  One host
    thread: the summation order of the host convolution depends on the thread count."""
    import copy
    from oracle import convonet as oc
    enc = net.encoder
    W = {k: v.detach().cpu() for k, v in enc.state_dict().items()}
    threads = torch.get_num_threads()
    torch.set_num_threads(1)
    try:
        with torch.no_grad():
            fea = oc.encoder_pointnet(torch.from_numpy(cloud)[None], W, plane_type='grid', reso_grid=64)['grid']
            return copy.deepcopy(enc.unet3d).cpu()(fea)
    finally:
        torch.set_num_threads(threads)


# --------------------------------------------------------------------------------------
# clocks during the timed region
# --------------------------------------------------------------------------------------
class ClockSampler(object):
    REASONS = {0x1: 'gpu_idle', 0x2: 'applications_clocks_setting', 0x4: 'sw_power_cap', 0x8: 'hw_slowdown',
               0x10: 'sync_boost', 0x20: 'sw_thermal_slowdown', 0x40: 'hw_thermal_slowdown',
               0x80: 'hw_power_brake_slowdown', 0x100: 'display_clock_setting'}

    def __init__(self, index):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._h = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self._nv = pynvml
            self._h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        nv = self._nv
        while not self._stop.is_set():
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                for bit, name in self.REASONS.items():
                    if r & bit and name != 'gpu_idle':
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.001)   # the timed region is ~10-60 ms: sample every millisecond

    def __enter__(self):
        if self._h is not None:
            self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._h is not None:
            self._t.join(timeout=1.0)

    def summary(self):
        if not self.samples:
            return {'sm_mhz': None, 'sm_max_mhz': self.max_mhz, 'reasons': [], 'note': 'NVML unavailable'}
        return {'sm_mhz': float(np.median(self.samples)), 'sm_max_mhz': self.max_mhz,
                'reasons': sorted(self.reasons), 'samples': len(self.samples)}


# --------------------------------------------------------------------------------------
# CPU reference (oracle port) on a bounded sample of the lattice
# --------------------------------------------------------------------------------------
class CpuReference(object):
    """The reference CPU path on a bounded sample: Generator3D.eval_points chunking (100k)
    through LocalDecoder.forward_img with a dense c_img_all (generation.py:338-383) on
    `n_sample` consecutive lattice points (whole x-rows from the middle of the nx^3
    lattice, so fingertip rows are hit), grid-64 features; all host threads."""

    def __init__(self, nx, n_sample, seed=0):
        from oracle import convonet as oc
        from vtaco_b200.conv_onet.models import decoder_dict
        self.oc = oc
        torch.set_num_threads(os.cpu_count() or 1)
        g = torch.Generator().manual_seed(seed)
        self.feats = {'grid': torch.randn(1, 32, 64, 64, 64, generator=g)}
        torch.manual_seed(seed)
        dec = decoder_dict['simple_local'](dim=3, c_dim=32, hidden_size=32)
        with torch.no_grad():
            for b in dec.blocks:
                b.fc_1.weight.normal_(0, 0.1)
        self.W = {k: v.detach() for k, v in dec.state_dict().items()}
        cloud, tips, tip_feat, touch = synthetic_scene(seed)
        ax = 1.1 * torch.linspace(-0.5, 0.5, nx)
        rows = max(1, -(-n_sample // (nx * nx)))
        x0 = max(0, nx // 2 - rows // 2)
        gx, gy, gz = torch.meshgrid(ax[x0:x0 + rows], ax, ax, indexing='ij')
        self.p = torch.stack([gx, gy, gz], -1).reshape(-1, 3)[:n_sample].contiguous()
        self.c_img = oc.fingertip_c_img(self.p, tips, torch.from_numpy(tip_feat), touch, 0.05)
        self.n = self.p.shape[0]
        self.rows, self.nx = rows, nx
        self.cores = torch.get_num_threads()

    def run(self):
        """decode the sample rows (eval_points chunking) + marching cubes on them (generation.py:268-272)."""
        from oracle import marching_cubes as omc
        t0 = time.perf_counter()
        occ = self.oc.eval_points(self.p, self.feats, self.W, self.c_img, points_batch_size=100000)
        if self.rows >= 2 and occ.numel() == self.rows * self.nx * self.nx:
            vol = occ.reshape(self.rows, self.nx, self.nx).numpy()
            v, f, _ = omc.marching_cubes(vol, None)
            omc.rescale_vertices(v, self.nx)
        return time.perf_counter() - t0

    def run_torch_eager_gpu(self):
        """The same algorithm the way the reference runs it on a GPU (generation.py:352-383): host chunk ->
        .to(device) -> decode_img through torch eager ATen kernels -> .cpu().  SURVEY §8d's "GPU bar"."""
        dev = torch.device('cuda', torch.cuda.current_device())
        if not hasattr(self, 'feats_g'):
            self.feats_g = {k: v.to(dev) for k, v in self.feats.items()}
            self.W_g = {k: v.to(dev) for k, v in self.W.items()}
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        occ = []
        with torch.no_grad():
            for pi, ci in zip(torch.split(self.p, 100000), torch.split(self.c_img, 100000)):
                o = self.oc.decoder_forward(pi.unsqueeze(0).to(dev), self.feats_g, self.W_g, mode='img',
                                            c_img=ci.unsqueeze(0).to(dev))
                occ.append(o.squeeze(0).cpu())
        torch.cat(occ, dim=0)
        return time.perf_counter() - t0


def run_reference(args, rank, world):
    if rank != 0:
        return
    nx = args.nx
    t_all = time.perf_counter()
    ref = CpuReference(nx, args.cpu_sample)
    for _ in range(args.warmup):
        ref.run()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ref.run()
    dt = time.perf_counter() - t0
    n, cores = ref.n, ref.cores
    value = float(n * args.steps / dt)
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': dt / args.steps * 1e3,
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(nx, args),
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                         'sample': '%d consecutive lattice points (x-rows from the middle of the %d^3 lattice) per '
                                   'step through the oracle port of Generator3D.eval_points + '
                                   'LocalDecoder.forward_img (torch CPU ops, 100k chunks) + the numpy marching-cubes '
                                   'restatement on those rows; a rate, not a whole-lattice time' % (n, nx)},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0, 'wall_s': time.perf_counter() - t_all,
    }
    print(json.dumps(line))


def measure_tensor_peaks(dev, n=8192, reps=10):
    """cuBLAS burst peaks (TFLOP/s) of a TF32 and a BF16 GEMM n^3 on this GPU — roofline denominators, measured
    after the timed regions (plain library GEMMs, not part of the product path)."""
    out = []
    prev = torch.backends.cuda.matmul.allow_tf32
    try:
        for dt, tf32 in ((torch.float32, True), (torch.bfloat16, False)):
            torch.backends.cuda.matmul.allow_tf32 = tf32
            a = torch.randn(n, n, device=dev, dtype=dt)
            b = torch.randn(n, n, device=dev, dtype=dt)
            for _ in range(3):
                a @ b
            best = float('inf')
            for _ in range(reps):
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda.synchronize(dev)
                e0.record()
                a @ b
                e1.record()
                torch.cuda.synchronize(dev)
                best = min(best, e0.elapsed_time(e1))
            out.append(2.0 * n ** 3 / (best * 1e-3) / 1e12)
            del a, b
    finally:
        torch.backends.cuda.matmul.allow_tf32 = prev
    return out[0], out[1]


def workload_config(nx, args):
    return {'workload': 'VTacOH_YCB dense %d^3 occupancy-lattice decode (LocalDecoder.forward_img, grid-64 '
                        'features, fingertip conditioning) + marching cubes' % nx,
            'nx': nx, 'queries_per_step': nx ** 3, 'encoder': 'LocalPoolPointnet grid64 hidden32 + UNet3D(4 levels)',
            'decoder': 'LocalDecoder simple_local hidden32 c_dim32 n_blocks5 bilinear', 'input_points': 3640,
            'parallelism': 'x-slabs of the lattice over %d GPU(s), features replicated, logit slabs %s' % (
                args.gpus, {'fused': 'stored into every rank over NVLink peer memory by the decoder kernel (fused '
                                     'all-gather)',
                            'root': 'pushed into rank 0 by one bulk NVLink peer copy per rank (double-buffered; marching '
                                    'cubes on rank 0 overlaps the peers\' next decode)',
                            'nccl': 'all-gathered with NCCL',
                            'mesh': 'never leave their rank: marching cubes runs per slab (+2 halo rows) and only mesh '
                                    'pieces are gathered on rank 0 (device-side signalling over NVLink peer memory)'}[
                                getattr(args, 'exchange', 'mesh')]),
            'l2': 'flushed between timed steps (256 MiB write outside the step events; N>1: followed by an untimed '
                  'device-side rendezvous so that every rank\'s step event starts aligned)',
            'kernel_variant': args.variant,
            'features': 'timed step: the grid features of the synthetic cloud computed once on the host (host_grid_features: '
                        'fp32 reference computation of the same encoder weights); e2e: the GPU encoder',
            'unet3d_conv_math': 'e2e only: UNet3D runs on our tcgen05 implicit-GEMM kernels (csrc/conv3d.cu) in single-pass TF32 '
                                'with fp32 accumulation - the arithmetic of the reference on a GPU (cuDNN, '
                                'torch.backends.cudnn.allow_tf32 = True by default; tests/test_unet3d_gpu.py: same deviation '
                                'from fp32 as cuDNN TF32, 4.4e-3 mean); PointNet, decoder and marching cubes are fp32-accurate '
                                '(3xTF32 on the tensor pipe)'}


def dump_outputs(path, mesh, grid):
    """Write what one step computed as float32 / float64 .npy files under `path`:
    vertices.npy (V, 3) float32 and faces.npy (F, 3) float64 (the int32 vertex ids, exact): the mesh the step
        returns; if the two together exceed DUMP_BYTES less the logit sample, both keep the same fraction of
        their rows, drawn with RandomState(0) and kept in order;
    logits_sample.npy (DUMP_LOGITS,) float32: the step's lattice logits at DUMP_LOGITS distinct flat (x, y, z)
        indices of the nx^3 grid, drawn with RandomState(0) and sorted.
    Vertex and face order are those of the extractor, so equal meshes give equal files."""
    v, f, counts = mesh
    V, F = [int(x) for x in counts[:2].cpu()]
    out = {'vertices': v[:V].cpu().numpy().astype(np.float32), 'faces': f[:F].cpu().numpy().astype(np.float64)}
    flat = grid.reshape(-1)
    idx = np.sort(np.random.RandomState(0).choice(flat.numel(), min(DUMP_LOGITS, flat.numel()), replace=False))
    out['logits_sample'] = flat[torch.from_numpy(idx).to(flat.device)].cpu().numpy().astype(np.float32)
    mesh_bytes = out['vertices'].nbytes + out['faces'].nbytes
    budget = DUMP_BYTES - out['logits_sample'].nbytes - 3 * 1024      # (and the three .npy headers)
    if mesh_bytes > budget:
        for k in ('vertices', 'faces'):
            a = out[k]
            keep = int(len(a) * budget // mesh_bytes)
            out[k] = a[np.sort(np.random.RandomState(0).choice(len(a), keep, replace=False))]
    os.makedirs(path, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(path, k + '.npy'), a)


# --------------------------------------------------------------------------------------
# ours
# --------------------------------------------------------------------------------------
def run_ours(args, rank, local_rank, world):
    import torch.distributed as dist
    from vtaco_b200 import _abi
    from vtaco_b200.conv_onet.generation import Generator3D
    import ctypes as C

    dev = torch.device('cuda', local_rank)
    torch.cuda.set_device(dev)
    group = None
    if world > 1:
        dist.init_process_group('nccl', device_id=dev)
        group = dist.group.WORLD
    nx = args.nx
    net = build_models(dev)
    net.decoder.kernel_variant = args.variant
    gen = Generator3D(net, device=dev, resolution0=nx // 4, with_img=True, padding=0.1, input_type='pointcloud')
    gen.use_multicast = not args.no_multicast
    cloud_np, tips, tip_feat_np, touch = synthetic_scene(0)
    cloud_host = torch.from_numpy(cloud_np)[None].pin_memory()
    tip_feat_host = torch.from_numpy(tip_feat_np).pin_memory()
    tip_feat = tip_feat_host.to(dev)

    def encode_features(host_grid=None):
        with torch.no_grad():
            if rank == 0 and host_grid is not None:
                g = host_grid.to(dev).contiguous(memory_format=torch.channels_last_3d)   # the encoder's layout
            elif rank == 0:
                c = net.encode_inputs(cloud_host.to(dev, non_blocking=True))
                g = c['grid']
            else:
                g = torch.empty((1, 64, 64, 64, 32), dtype=torch.float32, device=dev).permute(0, 4, 1, 2, 3)
            if world > 1:
                # broadcast the channels-last storage so every rank decodes from identical bits
                flat = g.permute(0, 2, 3, 4, 1)
                flat = flat if flat.is_contiguous() else flat.contiguous()
                dist.broadcast(flat, 0, group=group)
                g = flat.permute(0, 4, 1, 2, 3)
            return {'grid': g}

    def encode_features_local():
        with torch.no_grad():
            return net.encode_inputs(cloud_host.to(dev, non_blocking=True))

    c = encode_features(host_grid_features(net, cloud_np) if rank == 0 else None)
    tips_arg = (tips, tip_feat, touch, 0.05)
    exchange_note = None
    if world > 1 and args.exchange == 'root':
        # balance: rank 0 decodes fewer rows so that decode_0 + marching cubes == a peer's decode
        rr = torch.zeros(1, device=dev)
        if rank == 0:
            with torch.no_grad():
                g0, k0 = gen.eval_lattice(c_probe := encode_features_local(), tips=None, group=False)
                gen.mc(g0, level_keys=k0, sync=False)
                torch.cuda.synchronize(dev)
                ea, eb, ec = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
                ea.record()
                g0, k0 = gen.eval_lattice(c_probe, tips=None, group=False)
                eb.record()
                gen.mc(g0, level_keys=k0, sync=False)
                ec.record()
                torch.cuda.synchronize(dev)
            row_ms = ea.elapsed_time(eb) / nx
            mc_rows = 0.85 * eb.elapsed_time(ec) / row_ms   # eager MC timing includes launch gaps the graph does not have
            per = (nx + mc_rows) / world
            rr.fill_(max(2.0, per - mc_rows))
        dist.broadcast(rr, 0, group=group)
        gen.root_rows = int(rr.item()) // 2 * 2
    if world > 1 and args.exchange in ('fused', 'root', 'mesh'):
        # symmetric-memory rendezvous must succeed on EVERY rank, else all ranks use NCCL
        ok = torch.ones(1, device=dev)
        try:
            for _ in range(2):
                if args.exchange == 'mesh':
                    gen.sharded_mesh(c, tips=tips_arg, group=group)
                else:
                    gen.eval_lattice(c, tips=tips_arg, group=group, exchange=args.exchange)
        except Exception as e:  # noqa: BLE001 - report and fall back to the NCCL plumbing
            ok.zero_()
            exchange_note = 'peer-memory exchange unavailable (%s: %s); NCCL all-gather used' % (type(e).__name__, str(e)[:120])
        dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if ok.item() == 0:
            args.exchange = 'nccl'
            gen._fused = None
            gen._root_ex = None
            gen._mesh_ex = None
            exchange_note = exchange_note or 'peer-memory exchange unavailable on a peer; NCCL all-gather used' 
    flush = torch.empty(256 * 1024 * 1024 // 4, dtype=torch.float32, device=dev)

    def device_step():
        return gen.lattice_and_mesh(c, tips=tips_arg, group=group, exchange=args.exchange)

    def barrier():
        if world > 1:
            dist.barrier(group=group)
        torch.cuda.synchronize(dev)

    # ---- FP32 FMA peak (roofline denominator, self-measured) ----
    peaks = {}
    for v in (0, 1):
        r = C.c_double(0)
        _abi.check(_abi.lib().vtaco_fp32_peak(v, 4096, C.byref(r), _abi.stream_ptr(dev)), 'fp32_peak')
        peaks[v] = r.value
    fp32_peak = max(peaks.values())

    # ---- warm-up ----
    for _ in range(max(args.warmup, 1)):
        device_step()
    if world > 1 and args.exchange == 'mesh':
        gen._settle_sharded(device_step, group)      # piece / destination buffers large enough on every rank
    # make sure the MC buffers are large enough, then no more host reads inside the steps
    if world > 1 and args.exchange == 'root' and max(args.warmup, 1) % 2 == 0:
        device_step()                      # keep the buffer parity even before the next pair of steps
    out_ = device_step()
    V = F = 0
    grow = torch.zeros(1, device=dev)
    if out_ is not None:
        v_, f_, counts = out_
        V, F = [int(x) for x in counts[:2].cpu()]
        if args.exchange != 'mesh' and (V > v_.shape[0] or F > f_.shape[0]):
            gen.mc._ensure(0, int(V * 1.25) + 16, int(F * 1.25) + 16)
            grow.fill_(1)
    if world > 1:
        dist.all_reduce(grow, group=group)
    if grow.item() > 0:
        device_step()
        device_step()

    # ---- N>1: the exchanged result == what rank 0 computes alone from the same features ----
    identity = None
    if world > 1:
        import hashlib
        ok_id = torch.ones(1, device=dev)
        out_x = device_step()
        torch.cuda.synchronize(dev)
        if rank == 0:
            with torch.no_grad():
                vx, fx = out_x[0][:V].clone(), out_x[1][:F].clone()
                g1, k1 = gen.eval_lattice(c, tips=tips_arg, group=False)          # whole lattice, this rank alone
                v1, f1, c1 = gen.mc(g1, level_keys=k1, voffset=np.float32(nx / 2), vscale=np.float32(1.1 / nx), sync=False)
                V1, F1 = [int(x) for x in c1[:2].cpu()]
                same = (V1, F1) == (V, F) and torch.equal(v1[:V1], vx) and torch.equal(f1[:F1], fx)
                ok_id.fill_(1.0 if same else 0.0)
                h = hashlib.sha1(vx.cpu().numpy().tobytes())
                h.update(fx.cpu().numpy().tobytes())
                identity = {'ok': bool(same), 'mesh_sha1': h.hexdigest()[:16], 'single_rank_mesh': [V1, F1]}
        dist.all_reduce(ok_id, op=dist.ReduceOp.MIN, group=group)
        if world > 1 and args.exchange == 'root' and gen._root_ex is not None and gen._root_ex.parity:
            device_step()                  # keep the double-buffer parity even

    # ---- CUDA graph of the step (decode [+ exchange] + marching cubes) ----
    graph, graph_note = None, 'eager launches'
    step_out = None         # (vertex buffer, face buffer, counts) the timed step writes, for --dump-outputs
    if not args.no_graph and (world == 1 or args.exchange in ('fused', 'root', 'mesh')):
        ok = torch.ones(1, device=dev)
        try:
            graph, step_out = gen.capture_step(c, tips=tips_arg, group=group, exchange=args.exchange)
            graph.replay()
            torch.cuda.synchronize(dev)
        except Exception as e:  # noqa: BLE001
            ok.zero_()
            graph_note = 'eager launches (graph capture failed: %s)' % type(e).__name__
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
        if ok.item() == 0:
            graph = None
        else:
            graph_note = 'CUDA graph replay'
    elif not args.no_graph:
        graph_note = 'eager launches (NCCL exchange is not captured)'

    # ---- timed region: K steps, per-step CUDA events, L2 flushed in between ----
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True),
           torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    barrier()
    if world > 1 and graph is not None:
        graph.replay()          # untimed: the step's own device-side waits align the ranks after the host barrier
    # N>1, mesh exchange: the L2 flush between the steps (a measurement artefact, outside the step events) takes a
    # different time on every GPU, and the first rendezvous of the next step would charge the difference to the
    # ranks that flushed faster.  An untimed device-side rendezvous (the 16-byte level exchange with neutral
    # keys) after the flush starts every rank's step event aligned, like the barrier before the timed region.
    align_keys = None
    if world > 1 and graph is not None and args.exchange == 'mesh' and gen._mesh_ex is not None:
        from vtaco_b200.conv_onet.generation import new_minmax_key
        align_keys = new_minmax_key(dev)
    wall0 = time.perf_counter()
    with ClockSampler(local_rank) as clocks:
        for s in range(args.steps):
            flush.fill_(float(s))
            if align_keys is not None:
                gen._mesh_ex.level(align_keys)
            e0, e_dec, e1 = ev[s]
            e0.record()
            if graph is not None:
                graph.replay()
                e_dec.record()
            else:
                grid, keys = gen.eval_lattice(c, tips=tips_arg, group=None if world == 1 else group,
                                              exchange=args.exchange)
                e_dec.record()
                step_out = gen.mc(grid, level_keys=keys, voffset=np.float32(nx / 2), vscale=np.float32(1.1 / nx),
                                  sync=False)
            e1.record()
        barrier()
    wall = time.perf_counter() - wall0
    if args.dump_outputs:   # before the decoder-alone and e2e runs below re-use the generator's buffers
        dump_outputs(args.dump_outputs, step_out, gen._grid)
    step_ms = [e0.elapsed_time(e1) for e0, _, e1 in ev]
    dec_ms = [e0.elapsed_time(ed) for e0, ed, _ in ev]
    if graph is not None:   # stages are inside one graph launch: split by the separately timed decoder kernel below
        dec_ms = None
    total_ms = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    per_rank_steps = None
    if world > 1:
        dist.all_reduce(total_ms, op=dist.ReduceOp.MAX, group=group)
        allsteps = [torch.zeros(args.steps, dtype=torch.float64, device=dev) for _ in range(world)]
        dist.all_gather(allsteps, torch.tensor(step_ms, dtype=torch.float64, device=dev), group=group)
        per_rank_steps = [[round(float(x), 4) for x in t.cpu()] for t in allsteps]
    total_ms = float(total_ms.item())
    value = nx ** 3 * args.steps / (total_ms * 1e-3)

    # ---- decoder kernel alone (dominant kernel) for the roofline: events around the launch ----
    _vd = __import__('vtaco_b200.dist', fromlist=['slab'])
    x0, x1 = (_vd.slab_root(nx, rank, world, gen.root_rows) if (world > 1 and args.exchange == 'root')
              else _vd.slab(nx, rank, world))
    if world > 1 and args.exchange == 'mesh' and not (gen.halo_from_peer and rank + 1 < world):
        x1 = min(x1 + 2, nx)              # the two halo rows a rank decodes in addition when it does not read them from its neighbour
    if x1 <= x0:
        x0, x1 = 0, 2
    kq = (x1 - x0) * nx * nx
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    out_grid = gen._grid
    with torch.no_grad():
        for a, b in kev:
            flush.fill_(1.0)
            a.record()
            net.decoder.forward_dense(c, nx, x0=x0, x1=x1, use_img=True, tips=tips_arg, out=out_grid, axis=gen._axis)
            b.record()
    torch.cuda.synchronize(dev)
    k_ms = float(np.mean([a.elapsed_time(b) for a, b in kev]))
    achieved = kq * FLOP_PER_QUERY / (k_ms * 1e-3)

    # ---- end-to-end through Generator3D with host buffers ----
    e2e_times, h2d, d2h = [], 0, 0
    e2e_run, e2e_mode = None, 'Generator3D.generate_mesh (eager launches)'
    if not args.no_graph and (world == 1 or args.exchange == 'mesh'):
        ok = torch.ones(1, device=dev)
        try:
            e2e_run = gen.capture_generate(cloud_host, tips=(tips, tip_feat, touch, 0.05), group=group)
            e2e_mode = ('Generator3D.capture_generate (CUDA graph: H2D + encoder + decode + MC)' if world == 1 else
                        'Generator3D.capture_generate (one CUDA graph per rank: rank 0 H2D + encoder, NCCL broadcast of the '
                        'feature grid, slab decode, per-slab marching cubes, gather of mesh pieces on rank 0)')
        except Exception as e:  # noqa: BLE001
            ok.zero_()
            e2e_run, e2e_mode = None, 'Generator3D.generate_mesh (eager; graph capture failed: %s)' % type(e).__name__
        if world > 1:
            dist.all_reduce(ok, op=dist.ReduceOp.MIN, group=group)
            if ok.item() == 0:
                e2e_run = None
                if e2e_mode.startswith('Generator3D.capture'):
                    e2e_mode = 'Generator3D.generate_mesh (eager; graph capture failed on a peer)'
    for s in range(max(args.warmup, 1) + args.steps):
        if e2e_run is not None:
            barrier()
            t0 = time.perf_counter()
            tip_feat.copy_(tip_feat_host, non_blocking=True)     # H2D of the fingertip features
            res = e2e_run()                                      # H2D cloud + encode [+ broadcast] + decode + MC, mesh D2H
            barrier()
            if s >= max(args.warmup, 1):
                e2e_times.append(time.perf_counter() - t0)
                if res is not None:
                    vh, fh = res
                    h2d = cloud_host.numel() * 4 + tip_feat_host.numel() * 4
                    d2h = vh.size * 4 + fh.size * 4 + 16
            continue
        barrier()
        t0 = time.perf_counter()
        with torch.no_grad():
            cc = encode_features()                               # H2D of the pinned cloud + encoder (+ broadcast)
            tf = tip_feat_host.to(dev, non_blocking=True)        # H2D of the fingertip features
            if world > 1 and args.exchange == 'mesh':
                res = gen.generate_mesh(c=cc, tips=(tips, tf, touch, 0.05), group=group, exchange='mesh')
                if res is not None:
                    vh, fh = res
            else:
                grid, keys = gen.eval_lattice(cc, tips=(tips, tf, touch, 0.05), group=group, exchange=args.exchange)
                if grid is not None:
                    vv, ff = gen.extract_mesh(grid, keys)            # reads the two counters (D2H)
                    if rank == 0:
                        vh, fh = gen._to_host(vv, ff)                # mesh D2H into pinned buffers
        barrier()
        if s >= max(args.warmup, 1):
            e2e_times.append(time.perf_counter() - t0)
            if rank == 0:
                h2d = cloud_host.numel() * 4 + tip_feat_host.numel() * 4
                d2h = vh.size * 4 + fh.size * 4 + 16
    e2e_t = torch.tensor([sum(e2e_times)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(e2e_t, op=dist.ReduceOp.MAX, group=group)
    e2e_value = nx ** 3 * args.steps / float(e2e_t.item())

    if rank == 0:
        peaks_file = os.path.join(ROOT, 'MEASURED_PEAKS.json')
        measured = json.load(open(peaks_file)) if os.path.exists(peaks_file) else {}
        bf16_peak = measured.get('bf16_tflops', 1590.0)        # burst figure: the kernel is timed alone
        peak_tag = 'of measured' if 'bf16_tflops' in measured else 'of fallback'
        traffic = None
        prof = os.path.join(ROOT, 'profiles', 'decoder_ncu_summary.json' if args.variant < 2
                            else 'r02_decoder_tc4_ncu_summary.json' if args.variant == 7
                            else 'decoder_tc_ncu_summary.json')
        if os.path.exists(prof):
            try:
                traffic = json.load(open(prof)).get('dram_bytes_per_launch')
            except Exception:
                traffic = None
        hbm_gbs = kq * 4 / (k_ms * 1e-3) / 1e9
        common = {'flop_per_query_algorithmic': FLOP_PER_QUERY, 'queries_per_launch': kq, 'kernel_ms': k_ms,
                  'fp32_equivalent_tflops': achieved / 1e12,
                  'fp32_ffma_peak_self_measured_tflops': fp32_peak / 1e12,
                  'frac_of_self_measured_ffma_peak': achieved / fp32_peak,
                  'hbm_algorithmic_gbs': hbm_gbs,
                  'hbm_frac_of_measured': hbm_gbs / measured['hbm_gbs'] if 'hbm_gbs' in measured else None,
                  'traffic': traffic}
        if args.variant >= 2:
            # Denominator: the TF32 tensor peak MEASURED in this run (cuBLAS TF32 GEMM 8192^3, best of 10 — the
            # method MEASURED_PEAKS.json uses for bf16).  fp32 fidelity on the TF32 pipe takes 3 passes (3xTF32:
            # hi*hi + lo*hi + hi*lo), so the ceiling for ALGORITHMIC fp32 FLOPs is peak / 3 (SURVEY 8d: "measured
            # tensor peak of the precision used x passes"); the mixed mode (TF32 + BF16 corrections) needs
            # 1 TF32 pass + 1 BF16 pass over K = 64, i.e. 1 + 2/2 = 2 TF32-pass equivalents.
            tf32_peak, bf16_now = measure_tensor_peaks(dev)
            nb_ = 5
            mixed = args.variant in (4, 6)
            four = args.variant == 7
            split = 2 if args.variant in (5, 6, 7) else 1
            # variant 7: hi*W_hi + hi*W_lo in TF32 (2 passes) + lo*bf16(W) in BF16 (1 pass at the BF16 rate): the
            # ceiling time per algorithmic FLOP is 2 / tf32_peak + 1 / bf16_peak, i.e. 2 + tf32/bf16 TF32-pass equivalents
            passes = (2.0 + tf32_peak / bf16_now) if four else 2.0 if mixed else 3.0
            alg_tflops = achieved / 1e12
            ceiling = tf32_peak / passes
            # executed tensor work (every MMA issued: split products, bias K-blocks / K padding of the older variants),
            # reported separately, NOT the fraction:
            tf32_mmas = 8 * (3 * nb_) + 2 if four else (4 if mixed else 12) * (3 * nb_) + (2 * nb_ + 1)
            bf16_mmas = 2 * (3 * nb_) if four else 4 * (3 * nb_) if mixed else 0
            tf32_fpq = tf32_mmas * 128 * 32 * 8 * 2 / 128.0
            bf16_fpq = bf16_mmas * 128 * 32 * 16 * 2 / 128.0
            exec_frac = kq * (tf32_fpq / (tf32_peak * 1e12) + bf16_fpq / (bf16_now * 1e12)) / (k_ms * 1e-3)
            kname = '%s<dense> (tcgen05 %s, %d thread%s per query)' % (
                'decoder_tc4_kernel' if four else 'decoder_tc2_kernel' if split == 2 else 'decoder_tc_kernel',
                'kind::tf32 hi*W_hi + hi*W_lo, kind::f16 bf16(lo)*bf16(W); 4 tiles per SM' if four else
                'kind::tf32 main + kind::f16 BF16 corrections' if mixed else 'kind::tf32, 3xTF32',
                split, 's' if split > 1 else '')
            roofline = dict(common, bound='tensor', kernel=kname,
                            achieved=alg_tflops, peak=ceiling, unit='TFLOP/s', frac=alg_tflops / ceiling,
                            peak_source='measured in this run: cuBLAS TF32 GEMM 8192^3 burst = %.1f TFLOP/s (bf16 %.1f; '
                                        'MEASURED_PEAKS.json bf16 %.1f), divided by %g passes (%s)'
                                        % (tf32_peak, bf16_now, bf16_peak, passes,
                                           '2 TF32 passes + 1 BF16 pass counted as tf32_peak / bf16_peak of a TF32 pass' if four
                                           else 'TF32 main product + BF16 K=64 correction product' if mixed else '3xTF32'),
                            tf32_peak_measured_tflops=tf32_peak, passes=passes,
                            executed_tensor_flop_per_query=tf32_fpq + bf16_fpq,
                            executed_tensor_tflops=kq * (tf32_fpq + bf16_fpq) / (k_ms * 1e-3) / 1e12,
                            executed_frac_of_tensor_peak=exec_frac,
                            traffic_source='dram__bytes_read+write of one `ncu --set full` capture of this kernel at '
                                           'this shape, read from profiles/%s (not re-measured in this run)'
                                           % os.path.basename(prof),
                            frac_if_counted_as_3_tf32_passes=alg_tflops / (tf32_peak / 3.0),
                            note='frac = algorithmic FLOPs (30 976 per query) x passes / kernel time / measured TF32 peak; '
                                 + ('executed_* counts every MMA the kernel issues: three products per 32x32 matrix '
                                    '(hi*W_hi, hi*W_lo, lo*bf16(W)) and the two K = 8 blocks of the input layer'
                                    if four else
                                    'executed_* also counts the bias K-blocks and K padding the kernel issues'))
        else:
            roofline = dict(common, bound='fp32', kernel='decoder_kernel<dense> (SIMT)', achieved=achieved / 1e12,
                            peak=fp32_peak / 1e12, unit='TFLOP/s', frac=achieved / fp32_peak,
                            peak_source='self-measured register-resident FMA loop (vtaco_fp32_peak: scalar %.1f, '
                                        'packed FFMA2 %.1f TFLOP/s); MEASURED_PEAKS.json has no FP32 figure'
                                        % (peaks[0] / 1e12, peaks[1] / 1e12),
                            frac_of_measured_bf16_tensor_peak=(achieved / 1e12) / bf16_peak)
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': world, 'steps': args.steps,
            'warmup': args.warmup, 'ms_per_step': total_ms / args.steps, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': workload_config(nx, args),
            'roofline': roofline,
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h,
                    'ms_per_step': float(e2e_t.item()) / args.steps * 1e3,
                    'path': e2e_mode + ': pinned cloud -> H2D -> LocalPoolPointnet+UNet3D -> decode -> marching '
                            'cubes -> mesh D2H (pinned)'},
            # our kernels per step: fused decoder, marching-cubes classification + emit [+ level exchange and the
            # mesh-exchange kernel when N>1, mesh exchange]; the look-back state memset is not a kernel
            'gpu_launches': args.steps * (3 + (2 if (world > 1 and args.exchange == 'mesh') else 0)),
            'stage_ms': ({'decode_plus_exchange': float(np.mean(dec_ms)), 'marching_cubes':
                          float(np.mean(step_ms)) - float(np.mean(dec_ms))} if dec_ms is not None else
                         {'decoder_kernel_alone': k_ms, 'rest_of_step(exchange+marching_cubes)':
                          float(np.mean(step_ms)) - k_ms}),
            'launch_mode': graph_note,
            'mesh': {'vertices': V, 'faces': F},
            'clocks': clocks.summary(), 'wall_s_timed_region': wall,
        }
        if world > 1:
            line['step_ms_per_rank'] = per_rank_steps
            line['identity_ok'] = bool(identity and identity['ok'])
            line['identity'] = identity
            line['exchange'] = args.exchange if exchange_note is None else exchange_note
            if gen._mesh_ex is not None:
                line['exchange'] += (' (per-slab marching cubes, mesh pieces gathered on rank 0 by device-side signalling; '
                                     'timed out: %s)' % gen._mesh_ex.timed_out())
            if gen._fused is not None:
                line['exchange'] += ' (NVLS multicast stores)' if gen._fused.grid_multicast else ' (unicast peer stores)'
            if gen._root_ex is not None:
                line['exchange'] += ' (gather to rank 0, double-buffered, 1 barrier/step, rank 0 decodes %d of %d rows)' % (gen.root_rows, nx)
        if world == 1 and not args.no_cpu_baseline:
            ref = CpuReference(nx, args.cpu_sample)
            ref.run()
            sec = min(ref.run() for _ in range(3))
            line['cpu_baseline'] = {
                'value': ref.n / sec, 'unit': UNIT, 'cores': ref.cores, 'kind': 'port',
                'sample': '%d consecutive lattice points of the %d^3 lattice, best of 3 after 1 warm-up, oracle port '
                          'of Generator3D.eval_points + LocalDecoder.forward_img (torch CPU ops, 100k chunks) + numpy '
                          'marching cubes on those rows; a rate' % (ref.n, nx)}
            refg = CpuReference(nx, 16 * args.cpu_sample)
            refg.run_torch_eager_gpu()
            secg = min(refg.run_torch_eager_gpu() for _ in range(3))
            line['torch_eager_gpu_baseline'] = {
                'value': refg.n / secg, 'unit': UNIT, 'kind': 'port',
                'sample': '%d lattice points, best of 3 after 1 warm-up: the oracle port (the same ATen ops the '
                          'reference executes) on this GPU under torch %s eager, with the chunking and host<->device '
                          'copies of Generator3D.eval_points (generation.py:352-383) - compare with e2e, not value'
                          % (refg.n, torch.__version__)}
        print(json.dumps(line), flush=True)
    if world > 1:
        # Tear down in a fixed order: graphs that captured NCCL / symmetric-memory work first, then a last
        # barrier, then leave without the process-group destructor (ncclCommDestroy with captured graphs alive
        # can block; the line above is already flushed).
        del e2e_run, graph
        torch.cuda.synchronize(dev)
        dist.barrier(group=group)
        torch.cuda.synchronize(dev)
        sys.stdout.flush()
        sys.stderr.flush()
        os._exit(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=10)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--nx', type=int, default=256)
    ap.add_argument('--variant', type=int, default=7,
                    help='decoder kernel: 0 scalar-FFMA SIMT, 1 packed-FFMA2 SIMT, 2 tcgen05 3xTF32, 4 tcgen05 TF32 + BF16 '
                         'corrections, 5 / 6 = 2 / 4 with two threads per query, 7 (default) four tiles per SM')
    ap.add_argument('--cpu-sample', type=int, default=4 * 256 * 256)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-multicast', action='store_true', help='fused exchange with unicast peer stores only')
    ap.add_argument('--no-graph', action='store_true', help='launch the step eagerly instead of replaying a CUDA graph')
    ap.add_argument('--exchange', default='auto', choices=['auto', 'mesh', 'root', 'fused', 'nccl'],
                    help='N>1: auto = mesh (logits stay on their rank, marching cubes per slab, mesh pieces gathered on rank 0); '
                         'root = slabs pushed into rank 0 only by bulk peer copies (double-buffered, 1 barrier/step, MC on '
                         'rank 0, rank 0 decodes fewer rows); fused = decoder stores slabs into every rank (NVLS multicast); '
                         'nccl = all_gather_into_tensor')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='one GPU: after the timed steps write the mesh and a fixed sample of the lattice logits of '
                         'the last step as DIR/<name>.npy (float32 / float64, at most 64 MB)')
    args = ap.parse_args()
    rank, local_rank, world = env_int('RANK', 0), env_int('LOCAL_RANK', 0), env_int('WORLD_SIZE', 1)
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and (args.impl != 'ours' or world > 1):
        ap.error('--dump-outputs applies to --impl ours on one GPU')
    if args.exchange == 'auto':
        args.exchange = 'mesh'
    os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device — the product path has no CPU fallback '
                         '(use --impl reference for the CPU arm)')
    run_ours(args, rank, local_rank, world)


if __name__ == '__main__':
    main()
