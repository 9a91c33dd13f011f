"""Fused texture-field density (ntx_texture_field_density, nerf_texture_b200.texture.density): NeRFNetwork.density of the product's model
(nerf/network_curvedfield.py:412-433) in one kernel, against the same computation composed from the in-tree drop-in operators under fp16
autocast — Mesh.project -> GridEncoder -> frequency encoding -> tinycudann.Network -> exp / mask — and against the C oracle."""
import ctypes
import functools

import numpy as np
import pytest
import torch
import torch.nn as nn

import _util as U

DEV = "cuda:0"
TF_ARGS = "ntx_texture_field_density"


def _t(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


class FreqEncoder(nn.Module):
    """tools/encoding.py:5-43 as get_encoder('frequency', input_dim=1, multires=12) builds it (max_freq_log2 = 11, 12 bands, log sampling,
    include_input): [x, sin(2^0 x), cos(2^0 x), ..., sin(2^11 x), cos(2^11 x)], each product and function in the input's dtype."""

    def __init__(self, input_dim=1, multires=12):
        super().__init__()
        self.freq_bands = (2.0 ** torch.linspace(0.0, multires - 1, multires)).numpy().tolist()
        self.output_dim = input_dim + input_dim * multires * 2

    def forward(self, x):
        out = [x]
        for f in self.freq_bands:
            out += [torch.sin(x * f), torch.cos(x * f)]
        return torch.cat(out, dim=-1)


class Projector:
    """what MeshProjector.project reads of the reference's object (tools/map.py:340-433)"""

    def __init__(self, v, f, vn):
        self.mesh_vertices, self.faces, self.vertex_normals = _t(v), _t(f.astype(np.int64)), _t(vn)
        self.radius, self.depth_threshold, self.tbn = 100.0, 9.5, None


class Field(nn.Module):
    """MeshFeatureField's attributes in main.py's configuration (tools/map.py:546-618): hash grid cfgT, no prob_model, no import"""

    def __init__(self, projector, K=8, h_threshold=0.1, seed=0):
        super().__init__()
        from nerf_texture_b200.operators import GridEncoder
        self.meshprojector = projector
        self.encoder = GridEncoder(**U.cfgT()).to(DEV)
        g = torch.Generator().manual_seed(seed)
        with torch.no_grad():
            self.encoder.embeddings.copy_(torch.rand(self.encoder.embeddings.shape, generator=g) * 2 - 1)
        self.encoder_z = FreqEncoder()
        self.K, self.h_threshold, self.bound = K, h_threshold, 1
        self.hash, self.prob_model, self.imported, self.imported_type = True, False, False, None


class Model(nn.Module):
    """NeRFNetwork's density path on the drop-in packages (network_curvedfield.py:412-433 over MeshFeatureField.forward, map.py:620-719);
    `calls` counts how often it ran"""

    def __init__(self, field, hidden=32, hidden_layers=1, seed=3):
        super().__init__()
        import tinycudann as tcnn
        self.meshfea_field = field
        n_in = 2 * field.encoder.num_levels + field.encoder_z.output_dim
        self.sigma_net = tcnn.Network(n_in, 16, {"otype": "FullyFusedMLP", "activation": "ReLU", "output_activation": "None", "n_neurons": hidden,
                                                 "n_hidden_layers": hidden_layers}, seed=seed).to(DEV)
        self.calls = 0

    def density(self, x):
        from nerf_texture_b200 import mesh
        self.calls += 1
        mf = self.meshfea_field
        p_sur, sdf, h_mask, _, _ = mesh.project(mf.meshprojector, x, K=mf.K, h_threshold=mf.h_threshold)
        embed = torch.cat([mf.encoder(p_sur, bound=mf.bound), mf.encoder_z(sdf)], dim=-1)
        h = self.sigma_net(embed)
        sigma = torch.exp(h[..., 0].float())                      # trunc_exp: custom_fwd(cast_inputs=float32), tools/activation.py:5-10
        return {"sigma": torch.where(h_mask, sigma, torch.zeros_like(sigma)), "geo_feat": h[..., 1:]}


@pytest.fixture(scope="module")
def scene():
    U.ntx()
    v, f, vn = U.bumpy_sphere(40, 50)                             # 3 900 triangles
    return v, f, vn, Projector(v, f, vn)


def _samples(n, seed):
    """a mix: near the surface (inside and outside the h_threshold shell), well beyond the shell, far enough that neither cast hits,
    and anywhere in the box"""
    rng = np.random.default_rng(seed)
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    u = rng.random(n)
    r = np.where(u < 0.45, rng.uniform(0.55, 0.85, n), np.where(u < 0.7, rng.uniform(0.2, 0.45, n), rng.uniform(12.0, 20.0, n)))
    x = d * r[:, None]
    box = rng.random(n) < 0.15
    x[box] = rng.uniform(-1, 1, (box.sum(), 3))
    return _t(x.astype(np.float32))


def _both(model, x):
    from nerf_texture_b200 import texture
    with torch.no_grad(), torch.autocast("cuda", torch.float16):
        want = model.density(x)
        calls = model.calls
        got = texture.density(model, x)
        assert model.calls == calls, "the fused path fell back to the model's own density"
    torch.cuda.synchronize()
    return got, want


def _assert_same_bits(got, want):
    for k in ("sigma", "geo_feat"):
        assert got[k].dtype == want[k].dtype and got[k].shape == want[k].shape, k
    assert torch.equal(got["sigma"].view(torch.int32), want["sigma"].view(torch.int32))
    assert torch.equal(got["geo_feat"].view(torch.int16), want["geo_feat"].view(torch.int16))


@pytest.mark.gpu
def test_bit_for_bit_against_the_composed_dropins_and_close_to_the_oracle(scene):
    """sigma and h bit for bit like the drop-in composition, in and beyond the shell and where neither cast hits; the same inputs
    within a few fp16 ulp of the C oracle's grid -> frequency encoding -> MLP -> exp (fed the same projection, which the oracle
    reproduces only to tolerance: test_gpu_mesh.py).  sinf / cosf are the functions torch's sin / cos call for fp32 on CUDA, so the
    frequency encoding, and everything after it, is expected to be bit-identical; this test is what checks that."""
    from nerf_texture_b200 import mesh
    v, f, vn, proj = scene
    model = Model(Field(proj))
    N = 128 * 40 + 17
    x = _samples(N, 1)
    got, want = _both(model, x)
    _assert_same_bits(got, want)
    assert got["sigma"].shape == (N,) and got["geo_feat"].shape == (N, 15) and got["geo_feat"]._is_view()
    p_sur, sdf, h_mask, _, _ = mesh.project(proj, x, K=8, h_threshold=0.1)
    _, _, _, face = mesh.projector_mesh(proj).project(x, proj.vertex_normals, K=8)
    inside = h_mask.cpu().numpy()
    assert 0.1 < inside.mean() < 0.6 and (face == -1).float().mean().item() > 0.05      # all three kinds of sample are there
    assert (got["sigma"][~h_mask] == 0).all() and (got["sigma"][h_mask] > 0).all()
    assert torch.isfinite(got["geo_feat"][~h_mask].float()).all() and (got["geo_feat"][~h_mask] != 0).any()   # h computed everywhere

    # C oracle: grid_encode -> FreqEncoder (float64 sin / cos, rounded) -> ffmlp_forward -> trunc_exp
    L_, O = U.ntx(), U.oracle()
    enc, net = model.meshfea_field.encoder, model.sigma_net
    scales = torch.empty(8, device=DEV)
    S = float(np.log2(enc.per_level_scale))
    L_.call("ntx_grid_level_scales", S, 512, 8, L_.ptr(scales), L_.stream())
    x01 = ((p_sur + 1) / 2).cpu().numpy()
    feats = O.grid_encode(x01, enc.embeddings.detach().half().cpu().numpy(), enc.offsets.cpu().numpy(), enc.per_level_scale, 512, gridtype=0,
                          align_corners=True, level_scales=scales.cpu().numpy())
    s = sdf.cpu().numpy().astype(np.float32)
    z = [s] + [fn((s * np.float32(2.0 ** i)).astype(np.float64)).astype(np.float32) for i in range(12) for fn in (np.sin, np.cos)]
    inp = np.concatenate([feats.astype(np.float32)] + z + [np.zeros((N, 7), np.float32)], axis=1).astype(np.float16)
    h = O.ffmlp_forward(inp, net.params.detach().half().cpu().numpy(), 48, 16, 32, 1).astype(np.float32)
    scale = np.abs(h).max()
    assert np.abs(got["geo_feat"].float().cpu().numpy() - h[:, 1:]).max() <= 4 * U.ulp16(scale)
    sig = got["sigma"].cpu().numpy()
    assert np.abs(np.log(sig[inside]) - h[inside, 0]).max() <= 4 * U.ulp16(scale) + 1e-6      # sigma = exp(h0) in the shell


@pytest.mark.gpu
@pytest.mark.parametrize("K", [1, 8, 16])
@pytest.mark.parametrize("N", [0, 1, 127, 128, 129])
def test_sizes_and_neighbour_counts(scene, N, K):
    """N = 0 is checked for shapes and dtypes only: the composition cannot run on an empty batch (the drop-in grid encoder refuses
    the null data pointer of an empty tensor)"""
    from nerf_texture_b200 import texture
    v, f, vn, proj = scene
    model = Model(Field(proj, K=K, seed=K))
    x = _samples(max(N, 1), 10 + N)[:N]
    if N == 0:
        with torch.no_grad(), torch.autocast("cuda", torch.float16):
            got = texture.density(model, x)
        assert model.calls == 0 and got["sigma"].dtype == torch.float32 and got["geo_feat"].dtype == torch.float16
    else:
        got, want = _both(model, x)
        _assert_same_bits(got, want)
    assert got["sigma"].shape == (N,) and got["geo_feat"].shape == (N, 15)


@pytest.mark.gpu
def test_morton_ordered_batch_equals_small_chunks_and_repeats(scene):
    """2^19 + 5 samples take the Morton-ordered path (mesh.SORT_MIN); the same samples in chunks below it give the same bits, and so
    does a second launch"""
    from nerf_texture_b200 import mesh, texture
    v, f, vn, proj = scene
    model = Model(Field(proj))
    N = (1 << 19) + 5
    assert N >= mesh.SORT_MIN
    x = _samples(N, 2)
    with torch.no_grad(), torch.autocast("cuda", torch.float16):
        a = texture.density(model, x)
        b = texture.density(model, x)
        parts = [texture.density(model, x[i:i + (1 << 17)]) for i in range(0, N, 1 << 17)]
    assert model.calls == 0
    _assert_same_bits(a, b)
    _assert_same_bits(a, {k: torch.cat([p[k] for p in parts]) for k in ("sigma", "geo_feat")})


@pytest.mark.gpu
def test_out_of_scope_models_call_their_own_density(scene):
    from nerf_texture_b200 import texture
    v, f, vn, proj = scene
    x = _samples(300, 3)

    def fused(model, autocast=True, grad=False):
        model.calls = 0
        with torch.set_grad_enabled(grad), torch.autocast("cuda", torch.float16, enabled=autocast):
            out = texture.density(model, x)
        return model.calls, out

    model = Model(Field(proj))
    assert fused(model)[0] == 0                                    # in scope: never the model's own density
    bound = functools.partial(texture.density, model)              # the binding INTEGRATION.md documents
    with torch.no_grad(), torch.autocast("cuda", torch.float16):
        bound(x)
    assert model.calls == 0
    assert fused(model, autocast=False)[0] == 1                    # fp32 table
    assert fused(model, grad=True)[0] == 1                         # the parameters require grad
    for attr, value in (("prob_model", True), ("hash", False)):
        m = Model(Field(proj))
        setattr(m.meshfea_field, attr, value)
        assert fused(m)[0] == 1, attr
    m = Model(Field(proj))
    m.meshfea_field.imported, m.meshfea_field.imported_type = True, "field"
    assert fused(m)[0] == 1
    assert fused(Model(Field(proj), hidden=64))[0] == 1           # not the 32-neuron, 1-hidden-layer network
    assert fused(Model(Field(proj), hidden_layers=2))[0] == 1
    m = Model(Field(proj))
    m.meshfea_field.encoder_z = FreqEncoder(multires=10)           # output_dim 21
    m.sigma_net = Model(m.meshfea_field).sigma_net
    assert fused(m)[0] == 1


@pytest.mark.gpu
def test_triangle_less_mesh_is_refused(scene):
    from nerf_texture_b200.mesh import Mesh
    L_ = U.ntx()
    v, _, vn, _ = scene
    m = Mesh(v)                                                    # vertices only
    x = torch.zeros(4, 3, device=DEV)
    with pytest.raises(RuntimeError, match="no triangles"):
        L_.call(TF_ARGS, m._h, L_.ptr(_t(vn)), L_.ptr(x), 4, 8, 100.0, 0.05, 0.1, 1.0, 16, 16, 8, 1.0, 512, 1, 16, 16, 16, L_.stream())


def test_argument_validation_needs_no_gpu():
    """a null mesh, K outside 1..16 and L outside 1..32 return NTX_ERR_INVALID_ARGUMENT before any CUDA call"""
    from nerf_texture_b200 import _lib as L_
    lib = L_.lib()

    def rc(mesh, K, L):
        return lib.ntx_texture_field_density(mesh, 8, 8, 4, K, 100.0, 0.05, 0.1, 1.0, 16, 16, L, 1.0, 512, 1, 16, 16, 16, None)

    fake = ctypes.create_string_buffer(64)                        # zeroed memory: not a mesh handle
    for K, L, msg in ((0, 8, "K must be in 1..16"), (17, 8, "K must be in 1..16"), (8, 0, "L must be in 1..32"), (8, 33, "L must be in 1..32")):
        assert rc(ctypes.addressof(fake), K, L) == -1
        assert msg in lib.ntx_last_error().decode()
    assert rc(None, 8, 8) == -1 and "not a mesh handle" in lib.ntx_last_error().decode()
    assert rc(ctypes.addressof(fake), 8, 8) == -1 and "not a mesh handle" in lib.ntx_last_error().decode()
