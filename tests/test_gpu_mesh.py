"""GPU parity tests of the mesh front end (SURVEY §8 f3) through the C ABI / the drop-in `RayTracer` and `frnn` packages:
bit-exact against the oracle's exhaustive scans for the ray casts and the neighbour search, and to tolerance for the fused projection
(its reference is a chain of torch reductions)."""
import numpy as np
import pytest
import torch

import _util as U

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _bits(a):
    return np.ascontiguousarray(a, np.float32).view(np.int32)


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


@pytest.fixture(scope="module")
def sphere():
    v, f, vn = U.bumpy_sphere(80, 120)
    from nerf_texture_b200.mesh import Mesh
    U.ntx()
    return v, f, vn, Mesh(v, f)


def _check_trace(mesh, v, f, o, d):
    O = U.oracle()
    pos, nrm, depth, face = O.mesh_trace(v, f, o, d)
    gp, gn, gd, gf = mesh.trace(_t(o), _t(d))
    torch.cuda.synchronize()
    assert np.array_equal(_bits(gd.cpu().numpy()), _bits(depth))
    assert np.array_equal(gf.cpu().numpy(), face)
    assert np.array_equal(_bits(gp.cpu().numpy()), _bits(pos))
    assert np.array_equal(_bits(gn.cpu().numpy()), _bits(nrm))
    return face


def test_trace_bit_exact_against_exhaustive_scan(sphere):
    v, f, _, mesh = sphere
    info = mesh.info()
    assert info["n_triangles"] == len(f) and info["triangle_depth"] < 64
    o, d = U.random_rays(np.random.default_rng(0), 100000)
    face = _check_trace(mesh, v, f, o, d)
    assert 0.2 < (face >= 0).mean() < 0.9


def test_trace_ties_degenerates_and_in_plane_rays():
    from nerf_texture_b200.mesh import Mesh
    v, f, _ = U.bumpy_sphere(20, 30, bump=0.0)
    f2 = np.concatenate([f, f[:50], np.array([[0, 0, 1], [2, 2, 2]], np.int32)]).astype(np.int32)
    o, d = U.adversarial_rays(np.random.default_rng(1), v, f)
    _check_trace(Mesh(v, f2), v, f2, o, d)


@pytest.mark.parametrize("n_tri", [1, 2, 5, 9])
def test_trace_tiny_meshes_need_no_padding(n_tri):
    """the reference pads meshes of <= 8 triangles with dummies (raytracer.py:17-24); here any size works and gives the same hits"""
    from RayTracer import RayTracer
    rng = np.random.default_rng(n_tri)
    v = rng.uniform(-1, 1, (3 * n_tri, 3)).astype(np.float32)
    f = np.arange(3 * n_tri, dtype=np.int32).reshape(-1, 3)
    o, d = U.random_rays(rng, 20000)
    O = U.oracle()
    _, _, depth, face = O.mesh_trace(v, f, o, d)
    rt = RayTracer(v.astype(np.float64), f.astype(np.int64))           # the reference passes trimesh's float64 / int64 arrays
    pos, nrm, gd, gf = rt.trace(_t(o), _t(d))
    assert np.array_equal(_bits(gd.cpu().numpy()), _bits(depth)) and np.array_equal(gf.cpu().numpy(), face)
    assert (face >= 0).any()


def test_raytracer_dropin_signature_shapes_inplace_and_cpu_inputs(sphere):
    v, f, _, _ = sphere
    from RayTracer import RayTracer
    rt = RayTracer(torch.from_numpy(v), torch.from_numpy(f))            # tensors are accepted too (raytracer.py:13-14)
    o, d = U.random_rays(np.random.default_rng(2), 6 * 50)
    o3, d3 = torch.from_numpy(o).view(6, 50, 3), torch.from_numpy(d).view(6, 50, 3)    # CPU inputs are moved to the GPU (raytracer.py:39-41)
    pos, nrm, depth, face = rt.trace(o3.double(), d3)                   # and cast to float (raytracer.py:35-36)
    assert pos.shape == (6, 50, 3) and nrm.shape == (6, 50, 3) and depth.shape == (6, 50) and face.shape == (300,)
    assert pos.is_cuda and face.dtype == torch.int64 and depth.dtype == torch.float32
    oc, dc = _t(o), _t(d)
    keep_o, keep_d = oc.clone(), dc.clone()
    p2, n2, depth2, face2 = rt.trace(oc, dc, inplace=True)              # positions land in rays_o, normals in rays_d
    assert p2.data_ptr() == oc.data_ptr() and n2.data_ptr() == dc.data_ptr()
    assert torch.equal(p2.view(6, 50, 3), pos) and torch.equal(n2.view(6, 50, 3), nrm) and torch.equal(face2, face)
    hit = face >= 0
    assert torch.equal(p2[~hit], keep_o[~hit] + 10.0 * keep_d[~hit])    # a miss: depth 10, zero normal, face -1 (bvh.cu:705-717)
    assert (depth2[~hit] == 10).all() and (n2[~hit] == 0).all()
    e = rt.trace(oc[:0], dc[:0])
    assert e[0].shape == (0, 3) and e[3].shape == (0,)


@pytest.mark.parametrize("K,r", [(8, 100.0), (5, 100.0), (8, 0.3), (1, 100.0), (16, 100.0), (32, 0.5)])
def test_knn_bit_exact_against_exhaustive_scan(sphere, K, r):
    v, _, _, mesh = sphere
    O = U.oracle()
    q = np.random.default_rng(K).uniform(-1, 1, (60000, 3)).astype(np.float32)
    od, oi = O.points_knn(v, q, K, r)
    gd, gi = mesh.knn(_t(q), K=K, r=r)
    assert np.array_equal(_bits(gd.cpu().numpy()), _bits(od)) and np.array_equal(gi.cpu().numpy(), oi)


def test_knn_ties_and_duplicates():
    from nerf_texture_b200.mesh import Mesh
    O = U.oracle()
    rng = np.random.default_rng(2)
    pts = np.round(rng.uniform(-1, 1, (3000, 3)) * 8) / 8
    pts = np.concatenate([pts, pts[:500]]).astype(np.float32)
    q = (np.round(rng.uniform(-1, 1, (20000, 3)) * 16) / 16).astype(np.float32)
    for cloud in (pts, pts[:1], pts[:9]):
        od, oi = O.points_knn(cloud, q, 8, 100.0)
        gd, gi = Mesh(cloud).knn(_t(q), K=8, r=100.0)
        assert np.array_equal(_bits(gd.cpu().numpy()), _bits(od)) and np.array_equal(gi.cpu().numpy(), oi)


def test_frnn_dropin_contract(sphere):
    """the two call shapes of the reference: tools/map.py:396 (build the grid on the vertices themselves) and :456 (query with it)"""
    v, _, _, _ = sphere
    import frnn
    O = U.oracle()
    verts = _t(v)
    _, _, _, grid = frnn.frnn_grid_points(verts.unsqueeze(0), verts.unsqueeze(0), None, None, K=8, r=100., grid=None, return_nn=False, return_sorted=True)
    q = np.random.default_rng(5).uniform(-1, 1, (5000, 3)).astype(np.float32)
    dis, idx, nn, grid2 = frnn.frnn_grid_points(_t(q).unsqueeze(0), verts.unsqueeze(0), None, None, K=8, r=100., grid=grid, return_nn=True, return_sorted=True)
    assert grid2 is grid and dis.shape == (1, 5000, 8) and idx.shape == (1, 5000, 8) and idx.dtype == torch.int64 and nn.shape == (1, 5000, 8, 3)
    od, oi = O.points_knn(v, q, 8, 100.0)
    assert np.array_equal(_bits(dis[0].cpu().numpy()), _bits(od)) and np.array_equal(idx[0].cpu().numpy(), oi)
    assert torch.equal(nn[0], verts[idx[0]])
    # a query of the cloud against itself finds itself first, at distance 0
    dis, idx, _, _ = frnn.frnn_grid_points(verts.unsqueeze(0), verts.unsqueeze(0), None, None, K=1, r=100., grid=grid)
    assert (dis == 0).all()
    with pytest.raises(TypeError):
        frnn.frnn_grid_points(torch.zeros(1, 4, 3), torch.zeros(1, 4, 3), K=2, r=1.0)


def _project_tolerances(got, want, x, label):
    """p_sur / sdf / normal / face from two implementations of the projection whose normals differ in the last bits: the casts are
    continuous in the normal except across triangle edges and at the silhouette, so a small fraction of samples may land on a
    neighbouring face (or flip hit/miss) — those are counted, everything else must agree to 1e-4."""
    gp, gs, gn, gf = [np.asarray(a) for a in got]
    wp, ws, wn, wf = [np.asarray(a) for a in want]
    nerr = np.abs(gn - wn).max(1)
    assert (nerr < 2e-5).mean() > 0.9998, label                          # (the sign choice of map.py:478 can flip when its dot product is ~0)
    same = gf == wf
    assert same.mean() > 0.998, "%s: %.4f%% of the samples changed face" % (label, 100 * (1 - same.mean()))
    assert np.abs(gs.reshape(-1) - ws.reshape(-1))[same].max() < 1e-4 and np.abs(gp - wp)[same].max() < 1e-4, label
    close = np.abs(gs.reshape(-1) - ws.reshape(-1)) < 1e-3
    assert (same | close).mean() > 0.9995, label                         # a changed face is still the same surface almost everywhere


def test_project_against_oracle(sphere):
    v, f, vn, mesh = sphere
    O = U.oracle()
    rng = np.random.default_rng(7)
    x = rng.normal(size=(40000, 3))
    x = (x / np.linalg.norm(x, axis=1, keepdims=True) * rng.uniform(0.4, 1.0, (40000, 1))).astype(np.float32)
    want = O.mesh_project(v, vn, f, x)
    p, s, n, fi = mesh.project(_t(x), _t(vn), K=8)
    assert s.shape == (40000, 1) and fi.dtype == torch.int64
    _project_tolerances((p.cpu().numpy(), s.cpu().numpy(), n.cpu().numpy(), fi.cpu().numpy()), want, x, "fused kernel vs oracle")
    assert (fi >= 0).float().mean() > 0.95


def _shell_samples(n, seed):
    rng = np.random.default_rng(seed)
    x = rng.normal(size=(n, 3))
    return _t((x / np.linalg.norm(x, axis=1, keepdims=True) * rng.uniform(0.4, 1.0, (n, 1))).astype(np.float32))


def test_morton_visit_order_changes_nothing(sphere):
    """large batches are visited in Morton order of their positions (mesh.spatial_order): same bits out, in the caller's order"""
    v, f, vn, mesh = sphere
    x = _shell_samples(150000, 31)
    a = mesh.knn(x, K=8, sort=False)
    b = mesh.knn(x, K=8, sort=True)
    c = mesh.knn(x, K=8)                                     # default: sorted from mesh.SORT_MIN queries on
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(a[0], c[0]) and torch.equal(a[1], c[1])
    pa = mesh.project(x, _t(vn), K=8, sort=False)
    pb = mesh.project(x, _t(vn), K=8, sort=True)
    for u, w in zip(pa, pb):
        assert torch.equal(u, w)
    few = mesh.project(x[:1], _t(vn), K=8, sort=True)        # a single sample cannot be ordered
    assert torch.equal(few[1], pa[1][:1])


def test_full_size_properties():
    """BASELINE-size batch (2^22 samples, 230 K triangles): properties that need no exhaustive scan"""
    from nerf_texture_b200.mesh import Mesh
    v, f, vn = U.bumpy_sphere(340, 340)
    mesh = Mesh(v, f)
    N = 1 << 22
    g = torch.Generator(device=DEV).manual_seed(0)
    o = torch.rand(N, 3, device=DEV, generator=g) * 2 - 1
    d = torch.nn.functional.normalize(torch.randn(N, 3, device=DEV, generator=g), dim=-1)
    pos, nrm, depth, face = mesh.trace(o, d)
    hit = face >= 0
    assert 0.2 < hit.float().mean().item() < 0.9
    assert torch.equal(pos, o + depth[:, None] * d)                    # position = o + depth * d, unfused, hit or miss
    assert (depth[~hit] == 10).all() and (nrm[~hit] == 0).all() and (depth[hit] < 10).all() and (depth >= 0).all()
    tri = _t(v)[_t(f.astype(np.int64))[face[hit]]]                       # [n,3,3]
    n_true = torch.nn.functional.normalize(torch.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0], dim=-1), dim=-1)
    assert (nrm[hit] - n_true).abs().max() < 1e-5
    off_plane = ((pos[hit] - tri[:, 0]) * n_true).sum(-1).abs()
    assert off_plane.max() < 1e-4                                       # the hit point lies in the reported face's plane
    # nothing is nearer: a second cast from just before the hit, backwards, must not find a surface before the origin
    back = mesh.trace(pos[hit] - 1e-3 * d[hit], -d[hit])[2]
    assert (back >= depth[hit] - 2e-3).float().mean() > 0.9999
    # neighbour search: ascending, and the first neighbour of a vertex is itself
    dis, idx = mesh.knn(o[: 1 << 20], K=8)
    assert (dis[:, 1:] >= dis[:, :-1]).all() and (idx >= 0).all()
    dv, iv = mesh.knn(_t(v), K=1)
    assert (dv == 0).all()
