"""CPU tests of the host-side logic: drop-in package surface, level tables, state layout, ray sharding, and the N>1 gather
path on a world_size-2 gloo group."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from _util import ROOT, oracle


def _compat():
    import nerf_texture_b200
    nerf_texture_b200.install()


def test_dropin_package_surface():
    _compat()
    import ffmlp
    import gridencoder
    import raymarching
    import shencoder
    from gridencoder.grid_clustering import ClusteringLayer, GridEncoder_clustering   # tools/map.py:22 imports it like this
    for n in ("near_far_from_aabb", "polar_from_ray", "morton3D", "morton3D_invert", "packbits", "march_rays_train", "march_rays_train_differentiable",
              "composite_rays_train", "march_rays", "composite_rays", "compact_rays"):
        assert callable(getattr(raymarching, n)), n
    assert callable(gridencoder.grid_encode) and callable(ffmlp.ffmlp_forward) and callable(shencoder.sh_encode)
    assert ClusteringLayer and GridEncoder_clustering


def test_grid_encoder_state_matches_reference_layout():
    _compat()
    from gridencoder import GridEncoder, GridEncoder_clustering
    O = oracle()
    e = GridEncoder(input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=19, desired_resolution=2048, gridtype="hash", align_corners=True)
    offs, pls = O.grid_offsets(3, 16, 2, base_resolution=16, log2_hashmap_size=19, desired_resolution=2048, align_corners=True)
    np.testing.assert_array_equal(e.offsets.numpy(), offs)
    assert e.offsets.dtype == torch.int32 and tuple(e.embeddings.shape) == (6098120, 2) and e.embeddings.dtype == torch.float32
    assert e.output_dim == 32 and abs(e.per_level_scale - pls) < 1e-12 and e.gridtype_id == 0
    assert float(e.embeddings.abs().max()) <= 1e-4                       # U(-1e-4, 1e-4) init (grid.py:133-134)
    assert set(e.state_dict()) == {"embeddings", "offsets"}              # checkpoint-compatible names
    t = GridEncoder(num_levels=4, log2_hashmap_size=14, gridtype="tiled")
    assert t.gridtype_id == 1 and np.diff(t.offsets.numpy()).tolist() == [4920, 16384, 16384, 16384]
    c = GridEncoder_clustering(num_levels=4, log2_hashmap_size=12)
    c = c.to(c.cluster_layers[0].cluster_centers.device)                  # the centres start on the GPU when there is one, like the reference's
    assert len(c.cluster_layers) == 4 and float(c.clustering_loss(pick_level=False)) == pytest.approx(float(c.clustering_loss(pick_level=False)))


def test_ffmlp_module_state():
    _compat()
    from ffmlp import FFMLP
    m = FFMLP(32, 3, 64, 3)
    assert m.padded_output_dim == 16 and m.weights.numel() == 64 * (32 + 64 * 2 + 16) and m.weights.dtype == torch.float32
    assert float(m.weights.abs().max()) <= np.sqrt(3 / 64) + 1e-6
    m2 = FFMLP(32, 3, 64, 3)
    assert torch.equal(m.weights, m2.weights)                           # reset_parameters reseeds with 42 (ffmlp.py:142)
    for bad in (dict(input_dim=20, output_dim=3, hidden_dim=64, num_layers=2), dict(input_dim=32, output_dim=17, hidden_dim=64, num_layers=2),
                dict(input_dim=32, output_dim=3, hidden_dim=48, num_layers=2), dict(input_dim=32, output_dim=3, hidden_dim=64, num_layers=1)):
        with pytest.raises(AssertionError):
            FFMLP(**bad)


def test_no_cpu_fallback():
    _compat()
    from gridencoder import GridEncoder
    e = GridEncoder(num_levels=4, log2_hashmap_size=12)
    with pytest.raises(RuntimeError, match="CUDA"):
        e(torch.rand(8, 3))


def test_shard_plan_is_a_partition_and_inverts():
    from nerf_texture_b200 import render
    N = 1024 * 1024 + 777
    for world in (2, 3, 8):
        parts = [render.shard_indices(N, world, r) for r in range(world)]
        allidx = torch.cat(parts)
        assert allidx.numel() == N and torch.equal(torch.sort(allidx).values, torch.arange(N))
        sizes = [p.numel() for p in parts]
        assert max(sizes) - min(sizes) <= 1024
        idxs, n_max, inv = render._shard_plan(N, world, 1024, torch.device("cpu"))
        gathered = torch.full((world * n_max,), -1, dtype=torch.long)
        for r, i in enumerate(idxs):
            gathered[r * n_max: r * n_max + i.numel()] = i
        assert torch.equal(gathered[inv], torch.arange(N))


WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from nerf_texture_b200 import render
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=2)
rank = dist.get_rank()
N = 5000
g = torch.Generator().manual_seed(0)
full = torch.rand(N, 5, generator=g)
idx = render.shard_indices(N, 2, rank)
out = dict(image=full[idx, 0:3].clone(), depth=full[idx, 3].clone(), weights_sum=full[idx, 4].clone(), iterations=1)
res = render.gather_frame(out, N)
ok = torch.equal(res["image"], full[:, 0:3]) and torch.equal(res["depth"], full[:, 3]) and torch.equal(res["weights_sum"], full[:, 4])
print("RANK%%d %%s" %% (rank, "OK" if ok else "MISMATCH"))
dist.destroy_process_group()
""" % ROOT


def test_two_rank_gather_frame_gloo(tmp_path):
    """the N>1 path of bench.py / render_image_sharded: shard -> per-rank result -> ONE all_gather -> un-permute"""
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29517", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, "-c", WORKER], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120) for p in procs]
    for r, (so, se) in enumerate(outs):
        assert "RANK%d OK" % r in so, (so, se[-2000:])


def test_sample_schedules():
    """schedule helpers of the device-driven frame (render.py): the reference's rule is (N, 8); auto never asks for fewer samples
    per iteration than the reference and stays within the marcher's chunking"""
    from nerf_texture_b200 import render
    assert render.SCHEDULES["reference"] == (1, 8)
    for n in (1, 100, 1 << 17, 1 << 20, 1 << 22):
        mult, cap = render.auto_schedule(n)
        assert mult >= 1 and 8 <= cap <= 1024
    assert render.WALK_BUDGET > 0


def test_level_offsets_match_the_oracle_and_the_reference_rule():
    """operators.hashgrid_level_offsets (what GridEncoder allocates) == the oracle's table sizing for every encoder config the
    reference builds (gridencoder/grid.py:113-124: min(2^T, R^D) entries per level, rounded up to a multiple of 8)"""
    import numpy as np
    from _util import cfgA, cfgB, cfgT, oracle
    from nerf_texture_b200.operators import GridEncoder, hashgrid_level_offsets
    O = oracle()
    for cfg in (cfgA(), cfgB(), cfgT(), dict(input_dim=2, num_levels=6, level_dim=4, per_level_scale=1.5, base_resolution=8, log2_hashmap_size=10, align_corners=False)):
        want, pls = O.grid_offsets(**{k: v for k, v in cfg.items() if k != "level_dim"})
        enc = GridEncoder(**cfg)
        assert enc.offsets.dtype == torch.int32 and enc.offsets.tolist() == [int(v) for v in want]
        assert abs(float(enc.per_level_scale) - float(pls)) < 1e-12
        got = hashgrid_level_offsets(cfg["input_dim"], cfg["num_levels"], enc.per_level_scale, cfg["base_resolution"], cfg["log2_hashmap_size"], cfg["align_corners"])
        assert got == enc.offsets.tolist() and all(n % 8 == 0 for n in np.diff(got))
        assert enc.embeddings.shape == (got[-1], cfg["level_dim"]) and enc.output_dim == cfg["num_levels"] * cfg["level_dim"]


DP_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, %r)
from nerf_texture_b200 import parallel
dist.init_process_group("gloo", rank=int(os.environ["RANK"]), world_size=2)
rank = dist.get_rank()
g = torch.Generator().manual_seed(7)
shapes = [(1000, 2), (64 * 112,), (64 * 176,)]          # table slice, sigma-net weights, colour-net weights
full = [[torch.randn(*s, generator=g) for s in shapes] for _ in range(2)]     # the gradients of rank 0 and rank 1
params = [torch.nn.Parameter(torch.zeros(*s)) for s in shapes]
for p, gr in zip(params, full[rank]):
    p.grad = gr.clone()
params[1].grad = None if rank == 1 else params[1].grad               # a rank without a gradient for one parameter contributes zeros
parallel.allreduce_gradients(params, average=True)
want = [(full[0][i] + (full[1][i] if i != 1 else 0)) / 2 for i in range(3)]
ok = all(torch.allclose(p.grad, w, rtol=0, atol=1e-6) for p, w in zip(params, want))
print("RANK%%d %%s" %% (rank, "OK" if ok else "MISMATCH"))
dist.destroy_process_group()
""" % ROOT


def test_two_rank_gradient_allreduce_gloo():
    """SURVEY 8 f4: the data-parallel step's one collective — all gradients packed into one buffer, summed over the ranks, averaged"""
    env = dict(os.environ, MASTER_ADDR="127.0.0.1", MASTER_PORT="29519", WORLD_SIZE="2")
    procs = [subprocess.Popen([sys.executable, "-c", DP_WORKER], env=dict(env, RANK=str(r)), stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True) for r in range(2)]
    outs = [p.communicate(timeout=120) for p in procs]
    for r, (so, se) in enumerate(outs):
        assert "RANK%d OK" % r in so, (so, se[-2000:])


def test_checkpoint_round_trip_cpu(tmp_path):
    """the state a reference Trainer checkpoint holds for the hot path (nerf/utils.py:1490-1521: {'model': state_dict, ...}) survives
    torch.save / torch.load / load_state_dict(strict=True) on the drop-in modules, with the reference's parameter names and shapes"""
    _compat()
    from ffmlp import FFMLP
    from gridencoder import GridEncoder

    class Field(torch.nn.Module):           # the attribute names of nerf/network_ff.py:29-49
        def __init__(self):
            super().__init__()
            self.encoder = GridEncoder(input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=15, desired_resolution=512, align_corners=True)
            self.sigma_net = FFMLP(input_dim=32, output_dim=16, hidden_dim=64, num_layers=2)
            self.color_net = FFMLP(input_dim=32, output_dim=3, hidden_dim=64, num_layers=3)

    a, b = Field(), Field()
    with torch.no_grad():
        a.encoder.embeddings.uniform_(-1, 1)
        a.sigma_net.weights.uniform_(-1, 1)
    sd = a.state_dict()
    assert set(sd) == {"encoder.embeddings", "encoder.offsets", "sigma_net.weights", "color_net.weights"}      # grid.py:125-131, ffmlp.py:136
    assert sd["encoder.offsets"].dtype == torch.int32 and sd["sigma_net.weights"].shape == (64 * (32 + 64 + 16),) and sd["color_net.weights"].shape == (64 * (32 + 128 + 16),)
    path = str(tmp_path / "ckpt.pth")
    torch.save({"epoch": 3, "global_step": 100, "stats": {}, "model": sd}, path)
    ck = torch.load(path, map_location="cpu")
    missing, unexpected = b.load_state_dict(ck["model"], strict=True)
    assert not missing and not unexpected
    for k, v in b.state_dict().items():
        assert torch.equal(v, sd[k]), k


def test_spatial_order_is_a_permutation_whatever_the_input():
    """mesh.spatial_order only decides the order queries are visited in; it must return a permutation even for NaN / inf / identical points"""
    import torch
    from nerf_texture_b200.mesh import spatial_order
    g = torch.Generator().manual_seed(0)
    x = torch.rand(5000, 3, generator=g) * 2 - 1
    x[5] = float("nan"); x[7, 1] = float("inf"); x[9, 2] = -float("inf")
    for pts in (x, torch.zeros(17, 3), x[:1]):
        o = spatial_order(pts)
        assert sorted(o.tolist()) == list(range(len(pts)))
    xs = x[10:][spatial_order(x[10:])]
    assert (xs[1:] - xs[:-1]).norm(dim=1).mean() < 0.3 * (x[11:] - x[10:-1]).norm(dim=1).mean()      # neighbours in the order are neighbours in space
