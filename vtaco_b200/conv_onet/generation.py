"""Generator3D — dense occupancy-grid evaluation + mesh extraction, drop-in for the
hot-path part of reference src/conv_onet/generation.py:21-72,115-284,338-383.

`eval_points` keeps the reference's signature and semantics (host tensor in, host
tensor out) but evaluates the whole point set in one fused-decoder launch instead of
100k-point chunks with per-chunk H2D/D2H.  `generate_mesh` is the fast path of
`generate_obj_mesh_wnf`'s tail: lattice -> logits -> iso-level 0.5*(min+max) ->
marching cubes -> vertex rescale, all on the device, optionally sharded over the ranks of
a torch.distributed process group by x-slabs of the lattice.

Out of scope (SURVEY §2 row 5): hand mesh, tactile point clouds, CD/EMD metrics, trimesh.
"""
import numpy as np
import torch

from ..common import make_3d_grid, dense_axis
from ..mcubes import MarchingCubes, new_minmax_key, split_meshes
from .. import dist as vdist


class Mesh(object):
    """Minimal stand-in for trimesh.Trimesh(vertices, faces) — what generate_obj_mesh_wnf returns when
    trimesh is not installed: `.vertices` (V,3) float32, `.faces` (F,3) int32, `.export(path)` (.off)."""

    def __init__(self, vertices, faces):
        self.vertices = np.asarray(vertices)
        self.faces = np.asarray(faces)

    def export(self, path):
        from ..io import export_off
        export_off(path, self.vertices, self.faces)
        return path


def _make_mesh(vertices, faces):
    try:
        import trimesh
        return trimesh.Trimesh(vertices, faces, process=False)
    except ImportError:
        return Mesh(vertices, faces)


def R_from_PYR(wrist_rot):
    """reference src/common.py:591-604 (roll about z, pitch about x, yaw about y; R_pitch @ R_yaw @ R_roll)."""
    roll, pitch, yaw = wrist_rot
    cr, sr, cp, sp, cy, sy = np.cos(roll), np.sin(roll), np.cos(pitch), np.sin(pitch), np.cos(yaw), np.sin(yaw)
    R_roll = np.array([[cr, -sr, 0], [sr, cr, 0], [0, 0, 1]])
    R_pitch = np.array([[1, 0, 0], [0, cp, sp], [0, -sp, cp]])
    R_yaw = np.array([[cy, 0, -sy], [0, 1, 0], [sy, 0, cy]])
    return R_pitch @ R_yaw @ R_roll


def norm_pc_1(pc, pc_obj):
    """reference src/common.py:606-612: centre on pc_obj's centroid, scale by twice its radius."""
    centroid = np.mean(pc_obj, axis=0)
    m = np.max(np.sqrt(np.sum((pc_obj - centroid) ** 2, axis=1)))
    return (pc - centroid) / (2 * m)


def fingertips_from_mano(mano_joints, wrist_rot_euler, wrist_pos, pc_ply):
    """generation.py:177-188: MANO joints (21,3) -> the five fingertip positions in the normalised
    object frame the query points live in."""
    tips = np.asarray(mano_joints)[[4, 8, 12, 16, 20]]
    tips = tips - np.array([0.11, 0.005, 0], dtype=np.float32)
    tips = np.linalg.inv(R_from_PYR(np.array([-np.pi / 2, np.pi / 2, 0]))) @ tips.T
    tips = np.linalg.inv(R_from_PYR(np.array(wrist_rot_euler))) @ tips
    return norm_pc_1(tips.T + wrist_pos, pc_ply)


class Generator3D(object):
    '''  Generator class for Occupancy Networks (reference generation.py:21-72).

    Args:
        model (nn.Module): trained Occupancy Network model
        points_batch_size (int): batch size for points evaluation (kept for API parity; the fused
            kernel needs no chunking)
        threshold (float): threshold value
        device (device): pytorch device
        resolution0 (int): the dense lattice has nx = 4 * resolution0 points per axis
        padding (float): how much padding should be used
        with_img (bool): decode with the tactile feature (decode_img)
    '''

    def __init__(self, model, points_batch_size=100000, threshold=0.5, refinement_step=0, device=None,
                 resolution0=16, upsampling_steps=3, with_normals=False, padding=0.1, sample=False,
                 input_type=None, vol_info=None, vol_bound=None, simplify_nfaces=None, alpha=0.2,
                 with_img=False, encode_t2d=False):
        self.model = model.to(device)
        self.points_batch_size = points_batch_size
        self.refinement_step = refinement_step
        self.threshold = threshold
        self.device = device
        self.resolution0 = resolution0
        self.upsampling_steps = upsampling_steps
        self.with_normals = with_normals
        self.input_type = input_type
        self.padding = padding
        self.sample = sample
        self.simplify_nfaces = simplify_nfaces
        self.alpha = alpha
        self.with_img = with_img
        self.encode_t2d = encode_t2d
        self.vol_bound = vol_bound
        if input_type == 'pointcloud_crop':
            raise NotImplementedError('vtaco_b200: the sliding-window (pointcloud_crop) path is out of scope '
                                      '(SURVEY.md §2 row 9)')
        self._mc = None
        self._grid = None
        self._shared_grid = None
        self.halo_from_peer = True    # sharded extraction: read the two halo rows from the next rank instead of decoding them
        self._keys = None
        self._keys_init = None
        self._batch = None          # (grid (B,nx,nx,nx), keys (B,2), initial keys, axis) of the batched path
        self._batch_mc = None       # the batched path's extractor (its buffers are not the single-scene path's)
        self._pin = None
        self._fused = None
        self._root_ex = None
        self._mesh_ex = None
        self.mesh_gather = 'root'   # exchange='mesh': 'root' = the mesh is assembled on rank 0, 'all' = on every rank
        self.root_rows = None       # exchange='root': lattice rows decoded by rank 0 (None: nx / world)
        self.use_multicast = True   # NVLS multimem.st for the fused exchange when the fabric supports it

    @property
    def mc(self):
        if self._mc is None:
            self._mc = MarchingCubes(self.device)
        return self._mc

    # ------------------------------------------------------------------ reference API
    def eval_points(self, p, c=None, c_img_all=None, vol_bound=None, **kwargs):
        ''' Evaluates the occupancy values for the points (reference generation.py:338-383).

        Args:
            p (tensor): points (N,3), host or device
            c (dict): encoded feature volumes
            c_img_all (tensor): (1,N,c_dim) tactile feature per point (with_img)
        Returns a host tensor (N,) like the reference.
        '''
        dev = self.device
        with torch.no_grad():
            pi = p.to(dev, non_blocking=True).unsqueeze(0)
            if self.with_img:
                ci = c_img_all.to(dev, non_blocking=True).reshape(1, p.shape[0], -1)
                occ = self.model.decode_img(pi, c, ci, **kwargs).logits
            else:
                occ = self.model.decode(pi, c, **kwargs).logits
        return occ.squeeze(0).detach().cpu()

    def generate_obj_mesh_wnf(self, data):
        ''' Object mesh + metrics for one scene — reference generation.py:115-284, same signature and
        return triple `(mesh, emd, cd)`; called by train.py:246.

        Everything from the feature grid on runs on the device: fused lattice decode with the compact
        tactile conditioning, marching cubes, Chamfer distance and Earth-Mover distance of 2048
        shuffled mesh vertices against `points.points_obj` (generation.py:275-282).

        Inputs read from `data` (the reference's keys): 'inputs' (1,T,3), 'points.points_obj' (1,2048,3),
        and with `with_img`: 'inputs.touch_success' (1,5) plus
          * the tactile features: 'tactile.features' (1,5,c_dim), else `model.encode_img_inputs(
            data['inputs.img'])` when an image encoder is attached to the model;
          * fingertip branch (encode_t2d False): 'tactile.tips' (5,3) fingertip positions, else computed
            like generation.py:172-188 from the attached hand encoder's 'mano_joints' and
            'points.wrist', 'points.mano', 'inputs.pc_ply';
          * encode_t2d branch: 'tactile.points' — list of 5 (n,3) arrays, the back-projected tactile
            point clouds in the normalised object frame (generation.py:222-246 computes them with the
            RFUniverse camera model, which is outside the hot path; SURVEY §2).
        The hand / tactile-image networks themselves are out of scope (SURVEY §2 rows 13-15): attach
        your own modules as `encoder_hand` / `encoder_img`, or pass the 'tactile.*' entries.

        The vertex rescale uses the reference's hard-coded 1.1/nx (generation.py:272), which equals
        (1+padding)/nx for the shipped padding 0.1.  Triangulation of ambiguous cells follows
        oracle/mc_tables.py, not skimage's Lewiner tables (parity unpinned, DESIGN.md §2).'''
        from ..common import chamfer_distance, EarthMoverDistance
        from . import tactile
        self.model.eval()
        dev = self.device
        nx = self.resolution0 * 4
        inputs = data.get('inputs', torch.empty(1, 0)).to(dev)
        points_obj = data.get('points.points_obj')
        tips = tip_map = None
        with torch.no_grad():
            c = self.model.encode_inputs(inputs)
            if self.with_img:
                touch = torch.as_tensor(data.get('inputs.touch_success')).reshape(-1).cpu().numpy().astype(bool)
                c_img = data.get('tactile.features')
                if c_img is None:
                    c_img = self.model.encode_img_inputs(data.get('inputs.img').to(dev))
                c_img = torch.as_tensor(c_img, dtype=torch.float32).to(dev).reshape(1, touch.shape[0], -1)
                if not self.encode_t2d:
                    tp = data.get('tactile.tips')
                    if tp is None:
                        c_hand = self.model.encode_hand_inputs(inputs)
                        tp = fingertips_from_mano(
                            c_hand['mano_joints'].detach().cpu().numpy()[0],
                            data.get('points.wrist').squeeze().detach().cpu().numpy(),
                            data.get('points.mano').squeeze().detach().cpu().numpy()[:3],
                            data.get('inputs.pc_ply').detach().cpu().numpy().squeeze())
                    tips = (np.asarray(torch.as_tensor(tp).cpu(), dtype=np.float64).reshape(-1, 3), c_img[0], touch, 0.05)
                else:
                    pts = data.get('tactile.points')
                    if pts is None:
                        raise KeyError("generate_obj_mesh_wnf(encode_t2d=True) needs data['tactile.points'] (the "
                                       'back-projected tactile point clouds, generation.py:222-246)')
                    tip_map = (tactile.tactile_point_map(pts, touch, 0.015, nx=nx, padding=self.padding, device=dev),
                               c_img[0])
            grid, keys = self.eval_lattice(c, tips=tips, tip_map=tip_map, group=False)
            v, f = self.mc(grid, level_keys=keys, voffset=np.float32(nx / 2), vscale=np.float32(1.1 / nx))
            vertices, faces = self._to_host(v, f)
        vertices, faces = vertices.copy(), faces.copy()
        mesh = _make_mesh(vertices.copy(), faces)
        np.random.shuffle(vertices)                      # numpy's global RNG, like the reference
        vertices = np.ascontiguousarray(vertices[:2048], dtype=np.float32)
        vt = torch.from_numpy(vertices)[None].to(dev)
        cd = chamfer_distance(torch.as_tensor(points_obj).to(dev), vt, use_kdtree=False)
        emd = EarthMoverDistance(torch.as_tensor(points_obj)[0].to(dev), vt[0])
        return mesh, emd, cd.item()

    # ------------------------------------------------------------------ device-resident fast path
    def lattice_points(self):
        """(1+padding) * make_3d_grid(nx^3) of reference generation.py:155-157 (host tensor)."""
        nx = self.resolution0 * 4
        return (1 + self.padding) * make_3d_grid((-0.5,) * 3, (0.5,) * 3, (nx,) * 3)

    def eval_lattice(self, c, tips=None, c_img_all=None, group=None, exchange=None, tip_map=None):
        """Logits on the dense lattice, device tensor (nx,nx,nx), + int32 min/max keys.
        With a process group the x-slabs are decoded by different ranks; `exchange`:
          'fused' (default): the decoder kernel stores its slab into every rank's grid over
                   NVLink peer memory (torch symmetric memory) — no collective on the data path;
          'nccl' : all_gather_into_tensor of the slabs + MAX all-reduce of the keys.
        Returns (grid, keys); with the fused exchange `keys` holds one (min,max) pair per rank."""
        nx = self.resolution0 * 4
        dev = self.device
        dec = self.model.decoder
        if self._grid is None or self._grid.shape[0] != nx:
            self._grid = torch.empty((nx, nx, nx), dtype=torch.float32, device=dev)
            self._axis = dense_axis(nx, self.padding, dev)
        if self._keys is None:
            self._keys_init = new_minmax_key(dev)
            self._keys = self._keys_init.clone()
        keys = self._keys
        keys.copy_(self._keys_init)
        rank, world = vdist.rank_world(group)
        x0, x1 = vdist.slab(nx, rank, world)
        if world > 1 and exchange == 'root':
            # gather-to-root, double-buffered, one barrier per step (vdist.RootExchange)
            if self._root_ex is None or self._root_ex.grids[0].shape[0] != nx:
                self._root_ex = vdist.RootExchange(nx, dev, group)
            ex = self._root_ex
            b = ex.parity
            ex.parity ^= 1
            x0, x1 = vdist.slab_root(nx, rank, world, self.root_rows if self.root_rows is not None else nx // world)
            with torch.no_grad():
                if x1 > x0:
                    # rank 0 decodes straight into buffer b; a peer decodes into its local grid and
                    # pushes the slab with one bulk P2P copy (same stream: ordered before the barrier)
                    local = ex.grids[b] if rank == 0 else self._grid
                    dec.forward_dense(c, nx, x0=x0, x1=x1, use_img=self.with_img, c_img=c_img_all, tips=tips,
                                      out=local, minmax_key=keys, axis=self._axis)
                    if rank != 0:
                        ex.root_view[b][x0:x1].copy_(local[x0:x1], non_blocking=True)
                ex.publish(keys, b)
                ex.barrier()
            if rank == 0:
                return ex.grids[b], ex.tables[b][:2 * world]
            return None, None
        if world > 1 and (exchange or 'fused') == 'fused':
            if self._fused is None or self._fused.grid.shape[0] != nx:
                self._fused = vdist.FusedExchange(nx, dev, group, use_multicast=self.use_multicast)
            ex = self._fused
            with torch.no_grad():
                ex.barrier()                       # every rank is done reading the previous grid
                if x1 > x0:
                    dec.forward_dense(c, nx, x0=x0, x1=x1, use_img=self.with_img, c_img=c_img_all, tips=tips,
                                      out=ex.grid, minmax_key=keys, axis=self._axis, peers=ex.grid_ptrs,
                                      multicast=ex.grid_multicast)
                ex.publish(keys)                   # (min,max) -> slot `rank` of every table; resets keys
                ex.barrier()                       # all slabs and key pairs have landed
            return ex.grid, ex.table
        with torch.no_grad():
            if x1 > x0:
                dec.forward_dense(c, nx, x0=x0, x1=x1, use_img=self.with_img, c_img=c_img_all, tips=tips,
                                  out=self._grid, minmax_key=keys, axis=self._axis, tip_map=tip_map)
            if world > 1:
                vdist.all_gather_slabs(self._grid, nx, group)
                vdist.all_reduce_minmax(keys, group)
        return self._grid, keys

    def extract_mesh(self, grid, keys=None, level=None, rescale=True, sync=True):
        """marching cubes at level 0.5*(min+max) + `(v - nx/2) * (1+padding)/nx`
        (reference generation.py:268-272).  Returns device tensors (vertices, faces)."""
        nx = grid.shape[0]
        box = 1 + self.padding
        if rescale:
            return self.mc(grid, level=level, level_keys=keys, voffset=np.float32(nx / 2), vscale=np.float32(box / nx),
                           sync=sync)
        return self.mc(grid, level=level, level_keys=keys, sync=sync)

    def sharded_mesh(self, c, tips=None, c_img_all=None, group=None):
        """exchange='mesh' (SURVEY 8e, "gather of mesh pieces"): every rank decodes its x-slab into its
        grid (symmetric memory), the ranks agree on the iso-level (16 B each), every rank runs marching
        cubes on its slab — the two halo rows it needs are read in place from the next rank's grid
        (`halo_from_peer`; False: decoded locally as well) — and the pieces are concatenated into the
        destination rank(s): vertex / face order and ids identical to the single-GPU mesh.  Hazards: the
        level rendezvous orders every rank's decode before any peer read; the count rendezvous inside
        `ex.push` keeps a rank from starting its next decode while a neighbour still reads its rows.
        No host synchronisation;
        returns (vertex buffer, face buffer, int64[2] totals) of vdist.MeshExchange (valid on the
        destination ranks)."""
        nx = self.resolution0 * 4
        dev = self.device
        dec = self.model.decoder
        rank, world = vdist.rank_world(group)
        if self._mesh_ex is None or self._mesh_ex.gather != self.mesh_gather:
            cap = max(1024, 12 * nx * nx)
            self._mesh_ex = vdist.MeshExchange(dev, group, cap, 2 * cap, gather=self.mesh_gather)
        ex = self._mesh_ex
        if self._shared_grid is None or self._shared_grid[0].shape[0] != nx:
            # the lattice grid lives in symmetric memory: the halo rows of a slab are the next rank's first rows and
            # are read in place over NVLink by marching cubes instead of being decoded a second time
            self._shared_grid = ex.shared_grid(nx)
            self._axis = dense_axis(nx, self.padding, dev)
        grid, grid_ptrs = self._shared_grid
        self._grid = grid
        if self._keys is None:
            self._keys_init = new_minmax_key(dev)
            self._keys = self._keys_init.clone()
        x0, x1 = vdist.slab(nx, rank, world)
        xh = min(x1 + 2, nx)          # two halo rows: the next slab's first row and the row that numbers its vertices
        # ... which the next rank decodes anyway, if it owns them both (always, unless there are about as many ranks as rows)
        peer_halo = self.halo_from_peer and rank + 1 < world and xh > x1 and vdist.slab(nx, rank + 1, world)[1] >= xh
        x_dec = x1 if peer_halo else xh
        with torch.no_grad():
            if x1 > x0:
                dec.forward_dense(c, nx, x0=x0, x1=x_dec, use_img=self.with_img, c_img=c_img_all, tips=tips,
                                  out=grid, minmax_key=self._keys, axis=self._axis)
            # publishes (min,max), waits for every rank's — i.e. for every rank's decode of this step — and resets the keys
            ex.level(self._keys)
            if x1 > x0:
                halo = (grid_ptrs[rank + 1] + x1 * nx * nx * 4, xh - x1) if peer_halo else None
                v, f, counts = self.mc(grid[x0:x_dec], level_ptr=ex.level_ptr, x_emit=x1 - x0, x_origin=x0, halo=halo,
                                       voffset=np.float32(nx / 2), vscale=np.float32((1 + self.padding) / nx), sync=False)
            else:                         # more ranks than row pairs: an empty piece
                self.mc._ensure(0, 16, 16)
                v, f, counts = self.mc._verts, self.mc._faces, self.mc._counts
                counts.zero_()
            ex.push(counts, v, f)
        return ex.verts, ex.faces, ex.totals

    def lattice_and_mesh(self, c, tips=None, c_img_all=None, group=None, exchange=None):
        """One device-resident pass: lattice logits (+ exchange) and marching cubes, no host
        synchronisation.  Returns the extractor's (vertex buffer, face buffer, int64[2] counts)."""
        nx = self.resolution0 * 4
        if exchange == 'mesh' and vdist.rank_world(group)[1] > 1:
            return self.sharded_mesh(c, tips=tips, c_img_all=c_img_all, group=group)
        grid, keys = self.eval_lattice(c, tips=tips, c_img_all=c_img_all, group=group, exchange=exchange)
        if grid is None:      # exchange='root' on a non-root rank: the mesh is extracted by rank 0 only
            return None
        return self.mc(grid, level_keys=keys, voffset=np.float32(nx / 2), vscale=np.float32((1 + self.padding) / nx),
                       sync=False)

    def capture_step(self, c, tips=None, c_img_all=None, group=None, exchange=None, warmup=2):
        """Capture `lattice_and_mesh` into a CUDA graph (launch latency and Python overhead off
        the critical path — it matters once a slab decodes in well under a millisecond).
        Returns (graph, outputs); call graph.replay() per step.  The feature tensors, tips and
        all buffers are baked into the graph: re-capture when they change."""
        if exchange == 'root' and vdist.rank_world(group)[1] > 1:
            return self._capture_root_steps(c, tips, c_img_all, group, warmup)
        if exchange == 'mesh' and vdist.rank_world(group)[1] > 1:
            for _ in range(max(1, warmup)):
                self.sharded_mesh(c, tips, c_img_all, group)
            self._settle_sharded(lambda: self.sharded_mesh(c, tips, c_img_all, group), group)
            torch.cuda.synchronize(self.device)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = self.sharded_mesh(c, tips, c_img_all, group)
            return graph, out
        for _ in range(max(1, warmup)):          # allocations, attribute set-up, rendezvous
            out = self.lattice_and_mesh(c, tips, c_img_all, group, exchange)
        V, F = [int(x) for x in out[2][:2].cpu()]
        if V > out[0].shape[0] or F > out[1].shape[0]:
            self.mc._ensure(0, int(V * 1.5) + 16, int(F * 1.5) + 16)
            self.lattice_and_mesh(c, tips, c_img_all, group, exchange)
        torch.cuda.synchronize(self.device)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            out = self.lattice_and_mesh(c, tips, c_img_all, group, exchange)
        return graph, out

    def _settle_sharded(self, step, group):
        """After a sharded step ran: grow this rank's piece buffers and (collectively) the destination
        buffers until the mesh fits, re-running `step` on every rank while any rank had to grow.
        Host-synchronising — warm-up / eager path only."""
        import torch.distributed as dist
        ex = self._mesh_ex
        for _ in range(4):
            V, F = [int(x) for x in self.mc._counts[:2].cpu()]
            tv, tf = [int(x) for x in ex.totals.cpu()]
            grew = torch.zeros(1, device=self.device)
            if V > self.mc._verts.shape[0] or F > self.mc._faces.shape[0]:
                self.mc._ensure(0, int(V * 1.5) + 16, int(F * 1.5) + 16)
                grew.fill_(1)
            if ex.ensure_capacity(tv, tf):        # same decision on every rank
                grew.fill_(1)
            dist.all_reduce(grew, op=dist.ReduceOp.MAX, group=group)
            if grew.item() == 0:
                break
            step()
        if ex.timed_out():
            raise RuntimeError('vtaco_b200: a rank did not arrive at the mesh exchange within 2 s')
        return ex.verts, ex.faces, ex.totals

    def _capture_root_steps(self, c, tips, c_img_all, group, warmup):
        """exchange='root': the step alternates between two symmetric buffers, so two graphs are
        captured (one per buffer parity) and replayed in turn."""
        import torch.distributed as dist
        rank = dist.get_rank(group)
        for _ in range(2 * max(1, warmup)):      # even count: parity returns to 0
            out = self.lattice_and_mesh(c, tips, c_img_all, group, 'root')
        need = torch.zeros(1, device=self.device)
        if rank == 0:
            V, F = [int(x) for x in out[2][:2].cpu()]
            if V > out[0].shape[0] or F > out[1].shape[0]:
                self.mc._ensure(0, int(V * 1.5) + 16, int(F * 1.5) + 16)
                need.fill_(1)
        dist.all_reduce(need, group=group)
        if need.item() > 0:
            for _ in range(2):
                self.lattice_and_mesh(c, tips, c_img_all, group, 'root')
        torch.cuda.synchronize(self.device)
        graphs, outs = [], []
        for _ in range(2):
            gph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gph):
                o = self.lattice_and_mesh(c, tips, c_img_all, group, 'root')
            graphs.append(gph)
            outs.append(o)

        class _Alternating(object):
            def __init__(self):
                self.i = 0

            def replay(self):
                graphs[self.i].replay()
                self.i ^= 1

        return _Alternating(), outs[1]

    def capture_generate(self, inputs_host, tips=None, warmup=2, group=None):
        """CUDA graph of the whole extraction for a fixed input shape:
        H2D copy of the (pinned) host cloud -> encoder (PointNet kernels + UNet/UNet3D) ->
        lattice decode -> marching cubes.  Usage:
            run = gen.capture_generate(pinned_cloud, tips)      # once per shape
            pinned_cloud.copy_(new_cloud); v, f = run()         # per scene (host arrays)
        The tip positions / touch mask are baked in; tip features are read from the tensor
        passed in `tips` at replay time (update it in place).
        With a process group (one process per GPU): rank 0 copies and encodes, the channels-last
        feature grid is broadcast (NCCL, captured in the graph) so that every rank decodes from
        identical bits, then the sharded step (exchange='mesh') runs; `run()` returns the mesh on
        the destination rank(s) and None elsewhere.  Every rank must call `run()` per scene."""
        rank, world = vdist.rank_world(group)
        if rank == 0 and not inputs_host.is_pinned():
            raise ValueError('inputs_host must be a pinned host tensor (it is re-read at every replay)')
        dev = self.device
        static_in = torch.empty(inputs_host.shape, dtype=torch.float32, device=dev)
        self.model.eval()
        feat = None
        if world > 1:
            import torch.distributed as dist
            R = self.model.encoder.reso_grid
            feat = torch.empty((1, R, R, R, self.model.encoder.c_dim), dtype=torch.float32, device=dev)

        def body():
            if world == 1:
                static_in.copy_(inputs_host, non_blocking=True)
                c = self.model.encode_inputs(static_in)
                return self.lattice_and_mesh(c, tips=tips)
            if rank == 0:
                static_in.copy_(inputs_host, non_blocking=True)
                g = self.model.encode_inputs(static_in)['grid'].permute(0, 2, 3, 4, 1)
                if g.is_contiguous():
                    feat_r = g
                else:
                    feat.copy_(g)
                    feat_r = feat
            else:
                feat_r = feat
            dist.broadcast(feat_r, 0, group=group)
            return self.sharded_mesh({'grid': feat_r.permute(0, 4, 1, 2, 3)}, tips=tips, group=group)

        with torch.no_grad():
            for _ in range(max(1, warmup)):
                out = body()
            if world > 1:
                self._settle_sharded(body, group)
            else:
                V, F = [int(x) for x in out[2][:2].cpu()]
                if V > out[0].shape[0] or F > out[1].shape[0]:
                    self.mc._ensure(0, int(V * 1.5) + 16, int(F * 1.5) + 16)
                    body()
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            # thread_local: NCCL's watchdog thread polls CUDA events while we capture
            with torch.cuda.graph(graph, capture_error_mode='thread_local' if world > 1 else 'global'):
                out = body()
        has_result = world == 1 or self._mesh_ex.has_result()

        def run():
            graph.replay()
            if not has_result:
                return None
            V, F = [int(x) for x in out[2][:2].cpu()]           # D2H of the two counters (synchronises)
            if V > out[0].shape[0] or F > out[1].shape[0]:
                raise RuntimeError('mesh larger than the captured buffers (%d vertices, %d faces): re-capture' % (V, F))
            return self._to_host(out[0][:V], out[1][:F])

        run.graph = graph
        return run

    def generate_mesh(self, inputs=None, c=None, tips=None, c_img_all=None, group=None, to_host=True, exchange=None):
        """inputs (1,T,3) point cloud -> encoder -> lattice logits -> mesh.
        tips = (positions (F,3) float64, features (F,c_dim) device tensor, touch (F,), radius)."""
        self.model.eval()
        dev = self.device
        with torch.no_grad():
            if c is None:
                c = self.model.encode_inputs(inputs.to(dev, non_blocking=True))
            if exchange == 'mesh' and vdist.rank_world(group)[1] > 1:
                # sharded marching cubes; with gather='root' only rank 0 gets the mesh (others: None)
                step = lambda: self.sharded_mesh(c, tips=tips, c_img_all=c_img_all, group=group)   # noqa: E731
                step()
                vb, fb, tot = self._settle_sharded(step, group)
                if not self._mesh_ex.has_result():
                    return None
                V, F = [int(x) for x in tot.cpu()]
                v, f = vb[:V], fb[:F]
                return self._to_host(v, f) if to_host else (v, f)
            grid, keys = self.eval_lattice(c, tips=tips, c_img_all=c_img_all, group=group, exchange=exchange)
            v, f = self.extract_mesh(grid, keys)
        if to_host:
            return self._to_host(v, f)
        return v, f

    # ------------------------------------------------------------------ batched extraction (single GPU)
    def _batch_check(self, group):
        if vdist.rank_world(group)[1] > 1:
            raise NotImplementedError('batched mesh extraction runs on one GPU: call generate_mesh per scene with a '
                                      'process group')

    def _batch_tips(self, tips, radius):
        """(pos (B,F,3), feat (B,F,c_dim), touch (B,F)) -> the CUDA tensors the batched decode reads: float64
        positions, float32 features, int32 touch mask (tensors of that kind on the device are used as they are,
        so a captured graph re-reads them at replay)."""
        if tips is None or not self.with_img:
            return None
        pos, feat, touch = tips
        dev = self.device
        pos = torch.as_tensor(pos).to(device=dev, dtype=torch.float64).contiguous()
        touch = torch.as_tensor(touch).to(device=dev).to(torch.int32).contiguous()
        feat = torch.as_tensor(feat).to(device=dev, dtype=torch.float32)
        return pos, feat, touch, float(radius)

    def lattices_and_meshes(self, c, tips=None):
        """Batched `lattice_and_mesh`: the B lattices of the feature batch `c` in one decoder launch (with
        `with_img`: per-scene fingertips tips = (pos (B,F,3) float64, feat (B,F,32), touch (B,F) int32, radius)
        as CUDA tensors), the per-scene iso-levels, and the B meshes in one marching-cubes pass; no host
        synchronisation.  The batched path has its own lattice axis and extractor, so graphs of the single-scene
        path on this generator keep their buffers.  Returns the batch extractor's (vertex buffer, face buffer,
        int64[4] totals, (B,2) per-scene (V,F) counts)."""
        nx = self.resolution0 * 4
        dev = self.device
        B = next(t.size(0) for k, t in c.items() if torch.is_tensor(t))
        if self._batch is None or tuple(self._batch[0].shape) != (B, nx, nx, nx):
            init = new_minmax_key(dev, B)
            self._batch = (torch.empty((B, nx, nx, nx), dtype=torch.float32, device=dev), init.clone(), init,
                           dense_axis(nx, self.padding, dev))
        if self._batch_mc is None:
            self._batch_mc = MarchingCubes(dev)
        grid, keys, init, axis = self._batch
        keys.copy_(init)
        self.model.decoder.forward_dense(c, nx, use_img=self.with_img, tips=tips, out=grid, minmax_key=keys, axis=axis)
        return self._batch_mc.batch(grid, level_keys=keys, voffset=np.float32(nx / 2),
                                    vscale=np.float32((1 + self.padding) / nx), sync=False)

    def generate_meshes(self, inputs=None, c=None, tips=None, radius=0.05, to_host=True, group=None):
        """Batched `generate_mesh`: inputs (B,T,3) point clouds (or their features `c`) -> encoder -> B lattices
        decoded in one launch -> per-scene iso-level 0.5*(min+max) -> B meshes in one marching-cubes pass.
        tips = (pos (B,F,3), feat (B,F,c_dim), touch (B,F)): every scene's own fingertips (with_img), within
        `radius`.  Returns a list of B (vertices, faces), each equal to `generate_mesh` of that scene's features
        and fingertips (faces index the scene's own vertices); host arrays with to_host, else device tensors.
        One GPU."""
        self._batch_check(group)
        self.model.eval()
        with torch.no_grad():
            if c is None:
                c = self.model.encode_inputs(inputs.to(self.device, non_blocking=True))
            vb, fb, counts, scene_counts = self.lattices_and_meshes(c, self._batch_tips(tips, radius))
            V, F = [int(x) for x in counts[:2].cpu()]
            if V > vb.shape[0] or F > fb.shape[0]:   # re-run phase 2 with larger buffers
                grid, keys, _, _ = self._batch
                vb, fb, scene_counts = self._batch_mc.batch(grid, level_keys=keys,
                                                            voffset=np.float32(grid.shape[1] / 2),
                                                            vscale=np.float32((1 + self.padding) / grid.shape[1]))
            sc = scene_counts.cpu()
            v, f = vb[:V], fb[:F]
            if to_host:
                v, f = self._to_host(v, f)
                v, f = v.copy(), f.copy()
        return split_meshes(v, f, sc)

    def capture_generate_batch(self, inputs_host, tips=None, radius=0.05, warmup=2, group=None):
        """CUDA graph of the batched extraction for a fixed batch shape: H2D copy of the (pinned) host clouds
        (B,T,3) -> encoder -> B lattices in one decoder launch -> B meshes in one marching-cubes pass.  Usage:
            run = gen.capture_generate_batch(pinned_clouds, tips)   # once per shape
            pinned_clouds.copy_(new_clouds); meshes = run()         # per batch: list of B host (vertices, faces)
        tips = (pos (B,F,3) float64, feat (B,F,c_dim) float32, touch (B,F) int32) as CUDA tensors are read at
        every replay: write new fingertips into them in place.  run() reads all counters with one host
        synchronisation per batch; the copy of the meshes, sized by those counters, waits once more.  The graph
        uses the model's and this generator's batch buffers as they are at capture; a later call with a larger
        batch or lattice on the same model / generator may grow (re-allocate) them: capture each shape on its
        own generator and model, or capture again."""
        self._batch_check(group)
        if not inputs_host.is_pinned():
            raise ValueError('inputs_host must be a pinned host tensor (it is re-read at every replay)')
        dev = self.device
        dtips = self._batch_tips(tips, radius)
        if dtips is not None and not (tips[0] is dtips[0] and tips[1] is dtips[1] and tips[2] is dtips[2]):
            raise ValueError('capture_generate_batch re-reads the fingertips at replay: pass them as CUDA tensors '
                             '(pos float64, feat float32, touch int32)')
        static_in = torch.empty(inputs_host.shape, dtype=torch.float32, device=dev)
        self.model.eval()

        def body():
            static_in.copy_(inputs_host, non_blocking=True)
            return self.lattices_and_meshes(self.model.encode_inputs(static_in), dtips)

        with torch.no_grad():
            for _ in range(max(1, warmup)):
                out = body()
            V, F = [int(x) for x in out[2][:2].cpu()]
            if V > out[0].shape[0] or F > out[1].shape[0]:
                self._batch_mc._ensure(0, int(V * 1.5) + 16, int(F * 1.5) + 16)
                body()
            torch.cuda.synchronize(dev)
            graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(graph):
                out = body()

        def run():
            graph.replay()
            counts = torch.cat([out[2][:2], out[3].reshape(-1)]).cpu()     # one D2H of all counters
            V, F = int(counts[0]), int(counts[1])
            if V > out[0].shape[0] or F > out[1].shape[0]:
                raise RuntimeError('meshes larger than the captured buffers (%d vertices, %d faces): re-capture' % (V, F))
            v, f = self._to_host(out[0][:V], out[1][:F])
            return split_meshes(v.copy(), f.copy(), counts[2:].reshape(-1, 2))

        run.graph = graph
        return run

    def mesh_chamfer(self, vertices, points_obj, n_sample=2048, generator=None):
        """The Chamfer metric of generate_obj_mesh_wnf (reference generation.py:275-281): shuffle the
        mesh vertices, keep `n_sample`, chamfer_distance(points_obj, vertices, use_kdtree=False).
        vertices (V,3) device tensor (extract_mesh output), points_obj (1,T,3).  Stays on the device;
        the shuffle uses torch's generator instead of numpy's global one.  (The reference also reports
        an Earth-Mover distance through scipy's Hungarian solver — not built, SURVEY §8f-4.)"""
        from ..common import chamfer_distance
        v = torch.as_tensor(vertices, device=self.device, dtype=torch.float32)
        perm = torch.randperm(v.shape[0], device=self.device, generator=generator)[:n_sample]
        return chamfer_distance(points_obj.to(self.device), v[perm][None].contiguous(), use_kdtree=False)

    def _to_host(self, v, f):
        """mesh D2H through cached pinned staging buffers (one synchronisation)."""
        if self._pin is None or self._pin[0].shape[0] < v.shape[0] or self._pin[1].shape[0] < f.shape[0]:
            self._pin = (torch.empty((int(v.shape[0] * 1.25) + 16, 3), dtype=torch.float32, pin_memory=True),
                         torch.empty((int(f.shape[0] * 1.25) + 16, 3), dtype=torch.int32, pin_memory=True))
        hv, hf = self._pin[0][:v.shape[0]], self._pin[1][:f.shape[0]]
        hv.copy_(v, non_blocking=True)
        hf.copy_(f, non_blocking=True)
        torch.cuda.current_stream(self.device).synchronize()
        return hv.numpy(), hf.numpy()
