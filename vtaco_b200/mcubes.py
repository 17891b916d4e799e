"""GPU marching cubes — replaces `skimage.measure.marching_cubes(value_grid,
gradient_direction='ascent')` as called by the reference
(src/conv_onet/generation.py:270); conventions in oracle/mc_tables.py."""
import ctypes as C

import torch

from . import _abi

INT32_MAX, INT32_MIN = 2 ** 31 - 1, -2 ** 31


def new_minmax_key(device, n=None):
    """int32[2] accumulator for the decoder's min/max tracking; with `n`, (n,2): one pair per volume."""
    if n is None:
        return torch.tensor([INT32_MAX, INT32_MIN], dtype=torch.int32, device=device)
    return torch.tensor([[INT32_MAX, INT32_MIN]] * n, dtype=torch.int32, device=device)


def volume_keys(volumes, keys):
    """Merge the ordered-int (min,max) keys of each volume of `volumes` (B,...) float32 into `keys` (B,2) int32
    (initialise with new_minmax_key(device, B)): per volume the keys the decoder tracks when it decodes it alone."""
    _abi.require_cuda(volumes, 'volumes')
    if not volumes.is_contiguous() or volumes.dim() < 2:
        raise ValueError('volumes must be a contiguous (B,...) tensor')
    B = volumes.shape[0]
    if keys.dtype != torch.int32 or keys.device != volumes.device or tuple(keys.shape) != (B, 2) \
            or not keys.is_contiguous():
        raise ValueError('keys must be a contiguous int32 (%d,2) tensor on %s' % (B, volumes.device))
    with torch.cuda.device(volumes.device):
        _abi.check(_abi.lib().vtaco_volume_keys(_abi.ptr(volumes), B, volumes[0].numel(), _abi.ptr(keys),
                                                _abi.stream_ptr(volumes.device)), 'volume_keys')
    return keys


def keys_to_level(keys):
    """level=None of skimage: 0.5*(min+max) in fp32 (host helper; syncs)."""
    L = _abi.lib()
    k = keys.cpu().reshape(-1, 2)
    lo, hi = L.vtaco_key_to_float_host(int(k[:, 0].min())), L.vtaco_key_to_float_host(int(k[:, 1].max()))
    return float(torch.tensor(0.5, dtype=torch.float32) * (torch.tensor(lo, dtype=torch.float32) +
                                                            torch.tensor(hi, dtype=torch.float32)))


class MarchingCubes(object):
    """Re-usable extractor: keeps scratch and output buffers between calls so a steady
    stream of grids of one size runs without allocation or host synchronisation other
    than the final read of the two counters."""

    def __init__(self, device):
        self.device = torch.device(device)
        self._scratch = None
        self._verts = None
        self._faces = None
        self._counts = torch.zeros(4, dtype=torch.int64, device=self.device)
        self._keys = torch.zeros(2, dtype=torch.int32, device=self.device)
        self._scene_counts = None
        self._batch_keys = None

    def _ensure(self, nbytes, vcap, fcap):
        if self._scratch is None or self._scratch.numel() < nbytes:
            self._scratch = torch.empty(int(nbytes), dtype=torch.uint8, device=self.device)
        if self._verts is None or self._verts.size(0) < vcap:
            self._verts = torch.empty((int(vcap), 3), dtype=torch.float32, device=self.device)
        if self._faces is None or self._faces.size(0) < fcap:
            self._faces = torch.empty((int(fcap), 3), dtype=torch.int32, device=self.device)

    def __call__(self, volume, level=None, level_keys=None, voffset=0.0, vscale=1.0, sync=True,
                 x_emit=None, x_origin=0, level_ptr=None, halo=None):
        """volume: (nx,ny,nz) float32 CUDA tensor (axis0 = x), any alignment.  level: float, or None ->
        0.5*(min+max) (from `level_keys` if the decoder tracked them, else computed here; NaN, and so an empty
        mesh, when the volume holds a NaN, as in .batch);
        `level_ptr`: address of a device float holding the level (multi-GPU exchange).
        Returns (vertices (V,3) float32, faces (F,3) int32) views of internal buffers
        (valid until the next call) — or, with sync=False, the un-trimmed buffers and the
        device counter tensor (int64[4]: V, F, numbered vertices, -).
        Slab mode (`x_emit` rows owned, the rest of the volume are halo rows, `x_origin` = lattice
        row of volume[0]): include/vtaco_b200.h, vtaco_marching_cubes.  `halo=(device address, rows)`:
        the halo rows are not part of `volume` but are read in place from another (ny,nz)-row buffer —
        the next rank's grid, peer-mapped (vtaco_mc_args.halo_grid)."""
        _abi.require_cuda(volume, 'volume')
        if volume.dim() != 3 or not volume.is_contiguous():
            raise ValueError('volume must be a contiguous (nx,ny,nz) tensor')
        L = _abi.lib()
        nx, ny, nz = volume.shape
        halo_ptr, halo_rows = (int(halo[0]), int(halo[1])) if halo is not None else (0, 0)
        if halo_rows:
            if level_ptr is None and level is None and level_keys is None:
                raise ValueError('a separate halo needs an explicit level (the min/max scan covers `volume` only)')
            nx += halo_rows
        n = volume.numel()
        nbytes = L.vtaco_mc_scratch_bytes(nx, ny, nz)
        vcap = self._verts.size(0) if self._verts is not None else max(1024, 12 * max(nx * ny, ny * nz, nx * nz))
        fcap = self._faces.size(0) if self._faces is not None else 2 * vcap
        self._ensure(nbytes, vcap, fcap)
        a = _abi.McArgs()
        a.grid, a.nx, a.ny, a.nz = volume.data_ptr(), nx, ny, nz
        if halo_rows:
            a.halo_grid, a.halo_rows = halo_ptr, halo_rows
        st = _abi.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            if level_ptr is not None:
                a.level_ptr = int(level_ptr)
            elif level is None:
                if level_keys is None:
                    _abi.check(L.vtaco_grid_minmax(_abi.ptr(volume), n, _abi.ptr(self._keys), st), 'grid_minmax')
                    level_keys = self._keys
                a.level_keys = level_keys.data_ptr()
                a.n_level_keys = max(1, level_keys.numel() // 2)
            else:
                a.level = float(level)
            a.scratch, a.scratch_bytes = self._scratch.data_ptr(), self._scratch.numel()
            a.counts = self._counts.data_ptr()
            a.voffset, a.vscale = float(voffset), float(vscale)
            a.vertices, a.vertex_capacity = self._verts.data_ptr(), self._verts.size(0)
            a.faces, a.face_capacity = self._faces.data_ptr(), self._faces.size(0)
            a.phase = 3
            if x_emit is not None:
                a.x_emit, a.x_origin = int(x_emit), int(x_origin)
            _abi.check(L.vtaco_marching_cubes(C.byref(a), st), 'marching_cubes')
            if not sync:
                return self._verts, self._faces, self._counts
            V, F = [int(v) for v in self._counts[:2].cpu()]
            if V > self._verts.size(0) or F > self._faces.size(0):
                self._ensure(nbytes, int(V * 1.25) + 16, int(F * 1.25) + 16)
                a.vertices, a.vertex_capacity = self._verts.data_ptr(), self._verts.size(0)
                a.faces, a.face_capacity = self._faces.data_ptr(), self._faces.size(0)
                a.phase = 2
                _abi.check(L.vtaco_marching_cubes(C.byref(a), st), 'marching_cubes')
        return self._verts[:V], self._faces[:F]

    def batch(self, volumes, level=None, level_keys=None, voffset=0.0, vscale=1.0, sync=True):
        """Meshes of B volumes in one classification and one emit launch.  volumes: contiguous (B,nx,ny,nz)
        float32 CUDA tensor.  Each volume is extracted at its own level: 0.5*(min+max) from its row of
        `level_keys` (B,2) int32 (LocalDecoder.forward_dense of a batch fills them), else `level` for every
        volume, else 0.5*(min+max) computed here per volume.
        Returns (vertices (V,3) float32, faces (F,3) int32, scene_counts (B,2) int64 device tensor): the meshes
        concatenated in volume order, each volume's faces indexing its own vertex block; scene b's mesh is
        vertices[sum V_<b : +V_b], faces[sum F_<b : +F_b] and equals `self(volumes[b])` bit for bit.  Views of
        internal buffers, valid until the next call.  sync=False: the un-trimmed buffers, the int64[4] totals
        and the per-volume counts, without host synchronisation (outputs beyond the buffers are counted, not
        written: compare the totals with the buffer sizes)."""
        _abi.require_cuda(volumes, 'volumes')
        if volumes.dim() != 4 or not volumes.is_contiguous():
            raise ValueError('volumes must be a contiguous (B,nx,ny,nz) tensor')
        L = _abi.lib()
        B, nx, ny, nz = volumes.shape
        if level_keys is not None and (level_keys.dtype != torch.int32 or level_keys.device != volumes.device or
                                       tuple(level_keys.shape) != (B, 2) or not level_keys.is_contiguous()):
            raise ValueError('level_keys must be a contiguous int32 (%d,2) tensor on %s' % (B, volumes.device))
        nbytes = L.vtaco_mc_batch_scratch_bytes(B, nx, ny, nz)
        _abi.check(min(int(nbytes), 0), 'mc_batch_scratch_bytes')
        vcap = self._verts.size(0) if self._verts is not None else B * max(1024, 12 * max(nx * ny, ny * nz, nx * nz))
        fcap = self._faces.size(0) if self._faces is not None else 2 * vcap
        self._ensure(nbytes, vcap, fcap)
        if self._scene_counts is None or self._scene_counts.size(0) < B:
            self._scene_counts = torch.zeros((B, 2), dtype=torch.int64, device=self.device)
        scene_counts = self._scene_counts[:B]
        a = _abi.McArgs()
        a.grid, a.nx, a.ny, a.nz = volumes.data_ptr(), nx, ny, nz
        a.n_volumes, a.scene_counts = B, scene_counts.data_ptr()
        st = _abi.stream_ptr(self.device)
        with torch.cuda.device(self.device):
            if level is None:
                if level_keys is None:
                    if self._batch_keys is None or self._batch_keys[0].size(0) != B:
                        init = new_minmax_key(self.device, B)
                        self._batch_keys = (init, init.clone())
                    level_keys = self._batch_keys[1]
                    level_keys.copy_(self._batch_keys[0])
                    volume_keys(volumes, level_keys)
                a.level_keys = level_keys.data_ptr()
            else:
                a.level = float(level)
            a.scratch, a.scratch_bytes = self._scratch.data_ptr(), self._scratch.numel()
            a.counts = self._counts.data_ptr()
            a.voffset, a.vscale = float(voffset), float(vscale)
            a.vertices, a.vertex_capacity = self._verts.data_ptr(), self._verts.size(0)
            a.faces, a.face_capacity = self._faces.data_ptr(), self._faces.size(0)
            a.phase = 3
            _abi.check(L.vtaco_marching_cubes(C.byref(a), st), 'marching_cubes')
            if not sync:
                return self._verts, self._faces, self._counts, scene_counts
            V, F = [int(v) for v in self._counts[:2].cpu()]
            if V > self._verts.size(0) or F > self._faces.size(0):
                self._ensure(nbytes, int(V * 1.25) + 16, int(F * 1.25) + 16)
                a.vertices, a.vertex_capacity = self._verts.data_ptr(), self._verts.size(0)
                a.faces, a.face_capacity = self._faces.data_ptr(), self._faces.size(0)
                a.phase = 2
                _abi.check(L.vtaco_marching_cubes(C.byref(a), st), 'marching_cubes')
        return self._verts[:V], self._faces[:F], scene_counts


def split_meshes(vertices, faces, scene_counts):
    """(vertices, faces, per-scene (V,F) counts) of MarchingCubes.batch -> list of per-scene (vertices, faces)
    (views; torch tensors or numpy arrays)."""
    out, v0, f0 = [], 0, 0
    for nv, nf in [(int(a), int(b)) for a, b in scene_counts]:
        out.append((vertices[v0:v0 + nv], faces[f0:f0 + nf]))
        v0, f0 = v0 + nv, f0 + nf
    return out


_extractors = {}


def marching_cubes(volume, level=None, **kw):
    """Functional form (one cached extractor per device); returns fresh tensors."""
    dev = volume.device
    ex = _extractors.get(dev)
    if ex is None:
        ex = _extractors[dev] = MarchingCubes(dev)
    v, f = ex(volume, level, **kw)
    return v.clone(), f.clone()
