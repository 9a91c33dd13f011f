"""Fused texture field of the product's model (nerf/network_curvedfield.py) on libntx.

    model.density = functools.partial(texture.density, model)      # NeRFNetwork.density (network_curvedfield.py:412-433)

`density(model, x)` evaluates MeshProjector.project -> texture grid -> frequency encoding of the sdf -> sigma_net -> exp / mask as ONE
kernel (`ntx_texture_field_density`, include/ntx.h) for the configuration main.py trains, under fp16 autocast and without gradients:
that is how the reference's `update_extra_state` calls it, 50 times in `initialize_states` and then every 16 training steps.  Outside
that scope it calls the model's own `density` (the composed path on the drop-in packages), so binding it never changes a result.
"""
import numpy as np
import torch

from . import _lib as L
from .mesh import SORT_MIN, projector_mesh, spatial_order
from .operators import _half_table

_F32, _HALF = torch.float32, torch.half
MAX_LEVELS = 32            # kFieldMaxLevels of the kernel


def _freq_dim_ok(enc):
    return getattr(enc, "output_dim", None) == 25


def _sigma_net_ok(net, in_dim):
    """the tinycudann shim's FullyFusedMLP (compat/tinycudann): 32 neurons, one hidden layer, ReLU, no output activation"""
    return (hasattr(net, "params") and getattr(net, "hidden", None) == 32 and getattr(net, "n_hidden_layers", None) == 1
            and getattr(net, "activation", None) == 0 and getattr(net, "output_activation", None) == 6
            and getattr(net, "n_input_dims", None) == in_dim and getattr(net, "padded_in", None) == (in_dim + 15) // 16 * 16
            and 1 <= getattr(net, "n_output_dims", 0) <= 16)


def _grid_ok(enc):
    """a hash grid the kernel gathers: 3-D, 2 features per level, every level's index computed like gridtype 'hash'"""
    return (hasattr(enc, "embeddings") and hasattr(enc, "offsets") and getattr(enc, "input_dim", None) == 3
            and getattr(enc, "level_dim", None) == 2 and getattr(enc, "gridtype", None) == "hash"
            and 1 <= getattr(enc, "num_levels", 0) <= MAX_LEVELS)


def in_scope(model, x):
    """True when `density(model, x)` runs the fused kernel rather than the model's own `density`."""
    mf = getattr(model, "meshfea_field", None)
    net = getattr(model, "sigma_net", None)
    if mf is None or net is None or not torch.is_tensor(x) or not x.is_cuda or x.shape[-1] != 3:
        return False
    if not (torch.is_autocast_enabled("cuda") and torch.get_autocast_dtype("cuda") == _HALF):
        return False                                      # autocast off: the composed path gathers the fp32 table
    enc, enc_z = getattr(mf, "encoder", None), getattr(mf, "encoder_z", None)
    if getattr(mf, "prob_model", True) or not getattr(mf, "hash", False):
        return False
    if getattr(mf, "imported", False) and getattr(mf, "imported_type", None) is not None:
        return False                                      # imported textures take other branches of MeshFeatureField.forward (map.py:646-710)
    if not (_grid_ok(enc) and _freq_dim_ok(enc_z) and _sigma_net_ok(net, 2 * enc.num_levels + 25)):
        return False
    if torch.is_grad_enabled() and (x.requires_grad or any(p.requires_grad for m in (net, mf) for p in m.parameters())):
        return False                                      # training: the kernel has no backward
    return True


def density(model, x):
    """Drop-in body for `NeRFNetwork.density(x)` (network_curvedfield.py:412-433): {'sigma': [...] f32, 'geo_feat': [..., n_out - 1] f16},
    geo_feat a view of the sigma net's output h.  x: [..., 3] in [-bound, bound]."""
    if not in_scope(model, x):
        return type(model).density(model, x)
    mf, net = model.meshfea_field, model.sigma_net
    proj, enc = mf.meshprojector, mf.encoder
    m = projector_mesh(proj)
    prefix = x.shape[:-1]
    xs = m._dev(x).view(-1, 3)
    N = xs.shape[0]
    order = spatial_order(xs) if N >= SORT_MIN else None          # the rule of Mesh.project
    if order is not None:
        xs = xs[order]
    vn = m._dev(proj.vertex_normals)
    if vn.shape != (m.n_vertices, 3):
        raise RuntimeError("density: vertex_normals must be [%d, 3]" % m.n_vertices)
    thr = proj.depth_threshold if mf.h_threshold is None else min(proj.depth_threshold, mf.h_threshold)
    table = _half_table(enc.embeddings).contiguous()
    w = net.params.detach().to(_HALF).contiguous()
    sigma = torch.empty(N, dtype=_F32, device=m.device)
    h = torch.empty(N, 16, dtype=_HALF, device=m.device)
    with torch.cuda.device(m.device):
        L.call("ntx_texture_field_density", m._h, L.ptr(vn, _F32), L.ptr(xs, _F32), N, int(min(mf.K, m.n_vertices)), float(proj.radius), 0.05,
               float(thr), float(mf.bound), L.ptr(table, _HALF), L.ptr(enc.offsets), enc.num_levels, float(np.log2(enc.per_level_scale)),
               int(enc.base_resolution), int(enc.align_corners), L.ptr(w, _HALF), L.ptr(sigma, _F32), L.ptr(h, _HALF), L.stream())
    if order is not None:
        sigma, h = torch.empty_like(sigma).index_copy_(0, order, sigma), torch.empty_like(h).index_copy_(0, order, h)
    h = h[:, :net.n_output_dims].view(*prefix, net.n_output_dims)
    return {"sigma": sigma.view(prefix), "geo_feat": h[..., 1:]}
