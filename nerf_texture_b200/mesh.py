"""Mesh front end of the texture field (SURVEY §8 f3): nearest-hit ray casts, K nearest mesh vertices and the fused
`MeshProjector.project` over libntx's mesh handle (include/ntx.h, csrc/mesh.cu).

    m = Mesh(vertices, faces)                                   # builds both search trees once, like RayTracer(...) + frnn's grid
    positions, face_normals, depth, face_idx = m.trace(o, d)    # external/RayTracer RayTracer.trace
    dists, idxs = m.knn(xyz, K=8, r=100.)                       # frnn.frnn_grid_points (squared distances)
    p_sur, sdf, normal, face_idx = m.project(xyz, vertex_normals, K=8)      # tools/map.py:414-433 in one launch

The drop-in packages `RayTracer` and `frnn` under compat/ keep the reference's names and signatures on top of this class.
There is no CPU fallback: without libntx.so these raise RuntimeError.
"""
import ctypes as C

import numpy as np
import torch

from . import _lib as L

_F32, _I64 = torch.float32, torch.int64
SORT_MIN = 1 << 19      # batches at least this large are visited in Morton order of their positions (see spatial_order)
_SPREAD = {}            # device -> int32 [1024] table: 10 bits -> every third bit


def _spread_table(device):
    t = _SPREAD.get(device)
    if t is None:
        v = torch.arange(1024, dtype=torch.int32)
        v = (v | (v << 16)) & 0x030000FF
        v = (v | (v << 8)) & 0x0300F00F
        v = (v | (v << 4)) & 0x030C30C3
        v = (v | (v << 2)) & 0x09249249
        t = _SPREAD[device] = v.to(device)
    return t


def spatial_order(x, lo=None, hi=None):
    """Permutation that visits the points x [N,3] along a 30-bit Morton curve of the box [lo, hi] (default: their own bounding box).

    The mesh kernels run one thread per query and a warp costs what its slowest lane costs; queries that are neighbours in SPACE walk the
    same tree nodes (lanes stay together, the nodes are in L1).  Samples arrive ordered by ray and step — neighbours in a warp are
    then 10..100 leaf diameters apart.  Results do not depend on the order (every query is independent), only the time does: measured
    on B200, 2^20 projections 4.37 -> 3.66 ms including the 0.5 ms this ordering cost in its first form (profiles/r02_mesh_morton_order.txt);
    below ~2^19 queries the ordering costs more than it saves, hence SORT_MIN."""
    if lo is None or hi is None:
        lo, hi = x.min(dim=0)[0], x.max(dim=0)[0]
    g = ((x - lo) * (1023.0 / (hi - lo).clamp_min(1e-30))).to(torch.int64).clamp_(0, 1023)   # clamped AFTER the conversion: NaN / inf land in range
    t = _spread_table(x.device)
    code = t[g[:, 0]] | (t[g[:, 1]] << 1) | (t[g[:, 2]] << 2)
    return torch.sort(code)[1]


class Mesh:
    def __init__(self, vertices, triangles=None, device=None):
        """vertices [n,3], triangles [m,3] (numpy or tensors, any float / integer dtype; triangles may be None or empty: neighbour
        queries only).  The trees are built on the host and live on `device` (default: the current CUDA device)."""
        if torch.is_tensor(vertices):
            vertices = vertices.detach().cpu().numpy()
        if torch.is_tensor(triangles):
            triangles = triangles.detach().cpu().numpy()
        v = np.ascontiguousarray(vertices, dtype=np.float32).reshape(-1, 3)
        t = np.zeros((0, 3), np.int32) if triangles is None else np.asarray(triangles).reshape(-1, 3)
        if t.size and (t.min() < 0 or t.max() >= v.shape[0]):
            raise RuntimeError("Mesh: triangle index out of range")
        t = np.ascontiguousarray(t, dtype=np.int32)
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.n_vertices, self.n_triangles = int(v.shape[0]), int(t.shape[0])
        self._h = C.c_void_p()
        with torch.cuda.device(self.device):
            L.call("ntx_mesh_create", v.ctypes.data_as(C.c_void_p), self.n_vertices, t.ctypes.data_as(C.c_void_p), self.n_triangles, C.byref(self._h))

    def __del__(self):
        h, self._h = getattr(self, "_h", None), None
        if h:
            try:
                L.lib().ntx_mesh_destroy(h)
            except Exception:
                pass

    def info(self):
        out = (C.c_uint32 * 6)()
        L.call("ntx_mesh_info", self._h, out)
        return dict(zip(("n_vertices", "n_triangles", "triangle_nodes", "triangle_depth", "vertex_nodes", "vertex_depth"), list(out)))

    def _dev(self, t):
        t = t.to(device=self.device, dtype=_F32)
        return t.contiguous()

    def trace(self, rays_o, rays_d, inplace=False):
        """external/RayTracer/RayTracer/raytracer.py:31-68: positions, face_normals, depth, face_idx (i64, -1 = no hit within 10)."""
        rays_o, rays_d = self._dev(rays_o), self._dev(rays_d)
        prefix = rays_o.shape[:-1]
        o, d = rays_o.view(-1, 3), rays_d.view(-1, 3)
        N = o.shape[0]
        face_idx = torch.full((N,), -1, dtype=_I64, device=self.device)
        positions, normals = (o, d) if inplace else (torch.empty_like(o), torch.empty_like(d))
        depth = torch.empty(N, dtype=_F32, device=self.device)
        with torch.cuda.device(self.device):
            L.call("ntx_mesh_trace", self._h, L.ptr(o, _F32), L.ptr(d, _F32), L.ptr(positions, _F32), L.ptr(normals, _F32), L.ptr(depth, _F32),
                   L.ptr(face_idx, _I64), N, L.stream())
        return positions.view(*prefix, 3), normals.view(*prefix, 3), depth.view(*prefix), face_idx

    def knn(self, queries, K=8, r=100.0, sort=None):
        """K nearest mesh vertices within r: squared dists [..., K] f32 ascending, idxs [..., K] i64; -1 padding.
        sort: visit the queries in Morton order (None = for batches of SORT_MIN or more); the results are the same either way."""
        q = self._dev(queries)
        prefix = q.shape[:-1]
        q = q.view(-1, 3)
        N = q.shape[0]
        order = spatial_order(q) if (N >= SORT_MIN if sort is None else (sort and N > 1)) else None
        if order is not None:
            q = q[order]
        dists = torch.empty(N, K, dtype=_F32, device=self.device)
        idxs = torch.empty(N, K, dtype=_I64, device=self.device)
        with torch.cuda.device(self.device):
            L.call("ntx_mesh_knn", self._h, L.ptr(q, _F32), N, int(K), float(r), L.ptr(dists, _F32), L.ptr(idxs, _I64), L.stream())
        if order is not None:
            dists, idxs = torch.empty_like(dists).index_copy_(0, order, dists), torch.empty_like(idxs).index_copy_(0, order, idxs)
        return dists.view(*prefix, K), idxs.view(*prefix, K)

    def project(self, xyz, vertex_normals, K=8, r=100.0, dir_vec_wdist=0.05, sort=None):
        """MeshProjector.project (tools/map.py:414-433) without its tbn gather / h_mask: p_sur [...,3], sdf [...,1], normal [...,3], face_idx [...].
        sort: as in knn()."""
        x = self._dev(xyz)
        vn = self._dev(vertex_normals)
        if vn.shape != (self.n_vertices, 3):
            raise RuntimeError("project: vertex_normals must be [%d, 3]" % self.n_vertices)
        prefix = x.shape[:-1]
        x = x.view(-1, 3)
        N = x.shape[0]
        order = spatial_order(x) if (N >= SORT_MIN if sort is None else (sort and N > 1)) else None
        if order is not None:
            x = x[order]
        p_sur, normal = torch.empty_like(x), torch.empty_like(x)
        sdf = torch.empty(N, dtype=_F32, device=self.device)
        face_idx = torch.empty(N, dtype=_I64, device=self.device)
        with torch.cuda.device(self.device):
            L.call("ntx_mesh_project", self._h, L.ptr(vn, _F32), L.ptr(x, _F32), N, int(K), float(r), float(dir_vec_wdist), L.ptr(p_sur, _F32),
                   L.ptr(sdf, _F32), L.ptr(normal, _F32), L.ptr(face_idx, _I64), L.stream())
        if order is not None:
            p_sur, normal = torch.empty_like(p_sur).index_copy_(0, order, p_sur), torch.empty_like(normal).index_copy_(0, order, normal)
            sdf, face_idx = torch.empty_like(sdf).index_copy_(0, order, sdf), torch.empty_like(face_idx).index_copy_(0, order, face_idx)
        return p_sur.view(*prefix, 3), sdf.view(*prefix, 1), normal.view(*prefix, 3), face_idx.view(*prefix)


def projector_mesh(projector):
    """The Mesh of the reference's `MeshProjector` (`.mesh_vertices` and `.faces` or `.mesh.faces`), built on first use and cached on it."""
    m = getattr(projector, "_ntx_mesh", None)
    if m is None:
        faces = projector.faces if getattr(projector, "faces", None) is not None else projector.mesh.faces
        m = projector._ntx_mesh = Mesh(projector.mesh_vertices, faces, device=projector.mesh_vertices.device)
    return m


def project(projector, xyz, K=8, h_threshold=None):
    """Drop-in body for `MeshProjector.project(xyz, K, h_threshold)` (tools/map.py:414): `projector` is the reference's object (it needs
    `.mesh_vertices`, `.vertex_normals`, `.tbn`, `.depth_threshold`, `.radius` and a mesh with faces); the handle is cached on it.
    Returns p_sur, sdf, h_mask, normal, tbn like the reference."""
    m = projector_mesh(projector)
    p_sur, sdf, normal, face_idx = m.project(xyz, projector.vertex_normals, K=min(K, m.n_vertices), r=projector.radius)
    tbn = projector.tbn[face_idx] if getattr(projector, "tbn", None) is not None else None
    thr = projector.depth_threshold if h_threshold is None else min(projector.depth_threshold, h_threshold)
    h_mask = (sdf.abs() < thr).squeeze(-1)
    return p_sur, sdf, h_mask, normal, tbn
