"""Shared helpers of the test-suite: loaders for the checker libraries and synthetic scene builders."""
import importlib.util
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")


def oracle():
    sys.path.insert(0, ROOT) if ROOT not in sys.path else None
    from oracle import oracle as O
    O.lib()
    return O


def ref(name):
    """the reference's own CUDA extension rebuilt for sm_100a (oracle/_ref, see oracle/build_ref.py); skip if absent"""
    import torch  # noqa: F401  (libtorch must be loaded first)
    path = os.path.join(ROOT, "oracle", "_ref", "_ref_%s.so" % name)
    if not os.path.exists(path):
        pytest.skip("reference extension %s not built (oracle/_ref)" % name)
    modname = "_ref_%s" % name
    if modname in sys.modules:
        return sys.modules[modname]
    spec = importlib.util.spec_from_file_location(modname, path)
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    sys.modules[modname] = mod
    return mod


# ------------------------------------------------------------------------------------------------ stored reference outputs
REFERENCE_OUTPUTS = os.path.join(GOLDEN, "reference_outputs.npz")
_RECORD_TO = os.environ.get("NTX_RECORD_REFERENCE")      # path: run the reference live (oracle/_ref) and store what it returned
_stored = None
_recorded = {}
FULL_BYTES = 512             # arrays up to this size are stored whole; larger ones as a sample of elements plus a digest of the whole
SAMPLE = 128                 # elements kept of an array compared to a tolerance (of one compared exactly: EXACT_SAMPLE, for the message)
EXACT_SAMPLE = 16


def _canonical(a):
    a = np.ascontiguousarray(a)
    if a.dtype.kind == "f":      # value equality like assert_array_equal: -0 == +0, any NaN == any NaN
        a = np.where(np.isnan(a), np.array(np.nan, a.dtype), a + a.dtype.type(0))
    return a


def _digest(a):
    import hashlib
    a = _canonical(a)
    return np.frombuffer(hashlib.sha256(str((a.dtype.str, a.shape)).encode() + a.tobytes()).digest(), np.uint8)


def _sample_index(key, size, n):
    import zlib
    return np.sort(np.random.default_rng(zlib.crc32(key.encode())).choice(size, min(n, size), replace=False))


class Recorded:
    """An output of the reference: whole (`index` is None) or the elements `index` of the flattened array, with its SHA-256 `digest`."""

    def __init__(self, sample, index=None, digest=None, shape=None):
        self.sample, self.index, self.digest, self.shape = sample, index, digest, shape

    def take(self, a):
        """the same elements of one of our arrays"""
        a = np.asarray(a)
        if self.shape is not None:
            assert a.shape == tuple(self.shape), (a.shape, tuple(self.shape))
        return a if self.index is None else a.reshape(-1)[self.index]

    def assert_equal(self, a, msg=""):
        """our array equals the reference's, element for element (the whole array, not only the stored sample)"""
        np.testing.assert_array_equal(self.take(a), self.sample, err_msg=msg)
        if self.digest is not None:
            assert np.array_equal(_digest(a), self.digest), "%s: equal on the %d stored elements, different elsewhere" % (msg, len(self.index))


def save_packed(path, arrays):
    """many small arrays as one .npz of five (an .npz entry costs a few hundred bytes of zip headers)"""
    keys = sorted(arrays)
    vals = [np.asarray(arrays[k]) for k in keys]
    np.savez_compressed(path, keys=np.array(keys), dtypes=np.array([v.dtype.str for v in vals]), ndims=np.array([v.ndim for v in vals], np.int64),
                        dims=np.array([d for v in vals for d in v.shape], np.int64), blob=np.frombuffer(b"".join(v.tobytes() for v in vals), np.uint8))


def load_packed(path):
    z = np.load(path)
    out, at, d = {}, 0, 0
    dims = z["dims"]
    for k, dt, nd in zip(z["keys"], z["dtypes"], z["ndims"]):
        shape = tuple(int(x) for x in dims[d:d + nd])
        n = int(np.prod(shape)) * np.dtype(dt).itemsize
        out[str(k)] = np.frombuffer(z["blob"][at:at + n].tobytes(), dt).reshape(shape)
        at, d = at + n, d + nd
    return out


def _record(key, v):
    if not _recorded:
        import atexit
        atexit.register(lambda: save_packed(_RECORD_TO, _recorded))
        if os.path.exists(_RECORD_TO):
            _recorded.update(load_packed(_RECORD_TO))
    _recorded[key] = v


def reference_output(key, compute, exact=False):
    """What the reference's own CUDA kernels (oracle/_ref) computed for `key` on the test's seeded inputs.

    The reference is not part of this repository: its outputs are stored in tests/golden/reference_outputs.npz, written by running
    the GPU tests with NTX_RECORD_REFERENCE=<that file> on a B200 where oracle/build_ref.py has built oracle/_ref.  Only then is
    `compute` called.  A scalar comes back as a float, an array as a Recorded: whole when it is small, else a fixed sample of its
    elements (chosen from `key`) and the digest of the whole array.  `exact`: the array is only ever compared for equality, so the
    digest decides and a few elements suffice."""
    global _stored
    n = EXACT_SAMPLE if exact else SAMPLE
    if _RECORD_TO:
        v = compute()
        if np.ndim(v) == 0:
            _record(key, np.float64(v))
            return float(v)
        v = np.ascontiguousarray(v)
        if v.nbytes <= FULL_BYTES:
            _record(key, v)
            return Recorded(v)
        index = _sample_index(key, v.size, n)
        rec = Recorded(v.reshape(-1)[index], index, _digest(v), v.shape)
        _record(key + ":sample", rec.sample)
        _record(key + ":digest", rec.digest)
        _record(key + ":shape", np.array(v.shape, np.int64))
        return rec
    if _stored is None:
        _stored = load_packed(REFERENCE_OUTPUTS)
    if key in _stored:
        v = _stored[key]
        return float(v) if v.ndim == 0 else Recorded(v)
    assert key + ":sample" in _stored, "no stored reference output %r in %s" % (key, REFERENCE_OUTPUTS)
    shape = _stored[key + ":shape"]
    return Recorded(_stored[key + ":sample"], _sample_index(key, int(np.prod(shape)), n), _stored[key + ":digest"], shape)


def ntx():
    import nerf_texture_b200
    nerf_texture_b200.install()
    from nerf_texture_b200 import _lib
    _lib.lib()
    return _lib


# ------------------------------------------------------------------------------------------------ encoder configs
def cfgA():
    """network_ff's encoder: get_encoder('hashgrid', desired_resolution=2048) (tools/encoding.py:48,61-63)"""
    return dict(input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=19, desired_resolution=2048, align_corners=True)


def cfgB():
    """BASELINE config 1: L=4, T=2^14, F=2, constructor defaults otherwise"""
    return dict(input_dim=3, num_levels=4, level_dim=2, per_level_scale=2, base_resolution=16, log2_hashmap_size=14, align_corners=False)


def cfgT():
    """NeRF-Texture's texture grid (tools/map.py:563)"""
    return dict(input_dim=3, num_levels=8, level_dim=2, base_resolution=512, log2_hashmap_size=19, desired_resolution=1024, align_corners=True)


# ------------------------------------------------------------------------------------------------ synthetic scene
def _expand_bits(v):
    v = v.astype(np.uint32)
    v = (v * np.uint32(0x00010001)) & np.uint32(0xFF0000FF)
    v = (v * np.uint32(0x00000101)) & np.uint32(0x0F00F00F)
    v = (v * np.uint32(0x00000011)) & np.uint32(0xC30C30C3)
    v = (v * np.uint32(0x00000005)) & np.uint32(0x49249249)
    return v


def morton3D_np(x, y, z):
    return _expand_bits(x) | (_expand_bits(y) << np.uint32(1)) | (_expand_bits(z) << np.uint32(2))


def ball_density_grid(cascade, H, bound, radius=0.5, center=(0.0, 0.0, 0.0)):
    """density_grid [cascade, H^3] (Morton order, like renderer.py:585-600): 1 inside the ball, 0 outside"""
    g = np.arange(H, dtype=np.uint32)
    X, Y, Z = np.meshgrid(g, g, g, indexing="ij")
    idx = morton3D_np(X.ravel(), Y.ravel(), Z.ravel()).astype(np.int64)
    grid = np.zeros((cascade, H ** 3), np.float32)
    for c in range(cascade):
        b = min(2.0 ** c, bound)
        xyz = (np.stack([X.ravel(), Y.ravel(), Z.ravel()], 1).astype(np.float32) + 0.5) / H * 2 - 1
        xyz = xyz * b - np.asarray(center, np.float32)
        grid[c, idx] = (np.linalg.norm(xyz, axis=1) < radius).astype(np.float32)
    return grid


def pinhole_rays(H, W, fovy_deg=50.0, radius=2.5, azim_deg=30.0, elev_deg=20.0, dtype=np.float32):
    """rays of a camera on a sphere looking at the origin (OpenGL convention: camera looks down -z)"""
    az, el = np.deg2rad(azim_deg), np.deg2rad(elev_deg)
    eye = np.array([radius * np.cos(el) * np.sin(az), radius * np.sin(el), radius * np.cos(el) * np.cos(az)], np.float64)
    fwd = -eye / np.linalg.norm(eye)
    right = np.cross(fwd, np.array([0.0, 1.0, 0.0])); right /= np.linalg.norm(right)
    up = np.cross(right, fwd)
    focal = 0.5 * H / np.tan(0.5 * np.deg2rad(fovy_deg))
    i, j = np.meshgrid(np.arange(W) + 0.5, np.arange(H) + 0.5, indexing="xy")
    d = ((i - W / 2) / focal)[..., None] * right + (-(j - H / 2) / focal)[..., None] * up + fwd
    d = d / np.linalg.norm(d, axis=-1, keepdims=True)
    o = np.broadcast_to(eye, d.shape)
    return np.ascontiguousarray(o.reshape(-1, 3).astype(dtype)), np.ascontiguousarray(d.reshape(-1, 3).astype(dtype))


def ulp16(x):
    """fp16 unit in the last place at |x| (as float32)"""
    x = np.abs(np.asarray(x, np.float32))
    e = np.floor(np.log2(np.maximum(x, 2.0 ** -14)))
    return (2.0 ** (e - 10)).astype(np.float32)


# ------------------------------------------------------------------------------------------------ synthetic meshes (SURVEY §8 f3)
def bumpy_sphere(n_lat, n_lon, bump=0.1, radius=0.7):
    """closed-ish lat/lon sphere with a smooth bump pattern: vertices [n,3] f32, faces [m,3] i32, outward vertex normals [n,3] f32"""
    th = np.linspace(0.05, np.pi - 0.05, n_lat)
    ph = np.linspace(0, 2 * np.pi, n_lon, endpoint=False)
    T, P = np.meshgrid(th, ph, indexing="ij")
    r = radius + bump * np.sin(5 * T) * np.cos(3 * P)
    v = np.stack([r * np.sin(T) * np.cos(P), r * np.sin(T) * np.sin(P), r * np.cos(T)], -1).reshape(-1, 3).astype(np.float32)
    i, j = np.meshgrid(np.arange(n_lat - 1), np.arange(n_lon), indexing="ij")
    a, b = i * n_lon + j, i * n_lon + (j + 1) % n_lon
    c, d = (i + 1) * n_lon + j, (i + 1) * n_lon + (j + 1) % n_lon
    f = np.stack([np.stack([a, c, b], -1), np.stack([b, c, d], -1)], 2).reshape(-1, 3).astype(np.int32)
    return v, f, vertex_normals(v, f)


def vertex_normals(v, f):
    """area-weighted vertex normals (what open3d's compute_vertex_normals gives the reference, tools/map.py:369,394)"""
    fn = np.cross(v[f[:, 1]] - v[f[:, 0]], v[f[:, 2]] - v[f[:, 0]])
    vn = np.zeros_like(v)
    for k in range(3):
        np.add.at(vn, f[:, k], fn)
    return (vn / (np.linalg.norm(vn, axis=1, keepdims=True) + 1e-12)).astype(np.float32)


def random_rays(rng, n, extent=1.0):
    o = rng.uniform(-extent, extent, (n, 3)).astype(np.float32)
    d = rng.normal(size=(n, 3)).astype(np.float32)
    return o, (d / np.linalg.norm(d, axis=1, keepdims=True)).astype(np.float32)


def adversarial_rays(rng, v, f):
    """rays aimed exactly at vertices, edge midpoints and centroids (ties between the triangles that share them), from inside and from
    outside; axis-parallel rays from lattice origins (rays that run IN box faces); rays that start on vertices"""
    tgt = np.concatenate([v, 0.5 * (v[f[:, 0]] + v[f[:, 1]]), (v[f[:, 0]] + v[f[:, 1]] + v[f[:, 2]]) / 3]).astype(np.float32)
    d = (tgt / np.linalg.norm(tgt, axis=1, keepdims=True)).astype(np.float32)
    ax = np.eye(3, dtype=np.float32)[rng.integers(0, 3, 4000)] * rng.choice([-1.0, 1.0], (4000, 1)).astype(np.float32)
    oa = rng.uniform(-1, 1, (4000, 3)).astype(np.float32)
    oa[:2000] = np.round(oa[:2000] * 4) / 4
    ov = v[rng.integers(0, len(v), 4000)]
    dv = rng.normal(size=(4000, 3)).astype(np.float32)
    o = np.concatenate([np.zeros_like(tgt), 2 * tgt, oa, ov]).astype(np.float32)
    return o, np.concatenate([d, -d, ax, dv]).astype(np.float32)


def build_mesh_host_check():
    """g++ build of tests/native/mesh_host_check.cpp (the product's tree builder + traversals compiled for the host); returns a CDLL"""
    import ctypes
    import subprocess
    src = os.path.join(ROOT, "tests", "native", "mesh_host_check.cpp")
    out_dir = os.path.join(ROOT, "tests", "native", "_build")
    so = os.path.join(out_dir, "libmesh_host_check.so")
    deps = [src] + [os.path.join(ROOT, "nerf_texture_b200", "csrc", f) for f in ("mesh_bvh.cuh", "mesh_build.h")]
    if not os.path.exists(so) or any(os.path.getmtime(d) > os.path.getmtime(so) for d in deps):
        os.makedirs(out_dir, exist_ok=True)
        cmd = ["g++", "-O2", "-ffp-contract=off", "-fopenmp", "-fPIC", "-shared", "-std=c++17", "-Wno-unknown-pragmas", "-o", so, src]
        r = subprocess.run(cmd, capture_output=True, text=True)
        if r.returncode != 0:
            raise RuntimeError("mesh_host_check build failed:\n" + r.stderr[-4000:])
    return ctypes.CDLL(so)
