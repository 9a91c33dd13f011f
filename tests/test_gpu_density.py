"""Density-grid maintenance (SURVEY 8 f2): ntx_update_density_grid / nerf_texture_b200.density.update_extra_state against the CPU
oracle (positions as renderer.py:590-598 computes them -> oracle field -> EMA-max -> packbits) on a small grid."""
import numpy as np
import pytest
import torch

from _util import ntx, oracle

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda", 0) if torch.cuda.is_available() else None


def test_density_update_vs_oracle_small_grid():
    """H = 32, 2 cascades, explicit jitter and a partial cell list, against numpy + the C oracle's field"""
    L_ = ntx()
    O = oracle()
    from nerf_texture_b200 import density, render
    from nerf_texture_b200.operators import FFMLP, GridEncoder
    H, C, bound = 32, 2, 2.0
    enc = GridEncoder(input_dim=3, num_levels=16, level_dim=2, base_resolution=16, log2_hashmap_size=15, desired_resolution=512, align_corners=True).to(DEV)
    net = FFMLP(32, 16, 64, 2).to(DEV)
    g = torch.Generator().manual_seed(5)
    with torch.no_grad():
        enc.embeddings.copy_((torch.rand(enc.embeddings.shape, generator=g) * 2 - 1) * 0.5)
    H3 = H ** 3
    grid0 = (torch.rand(C, H3, generator=g) * 2 - 0.5)            # some cells negative (= never trained: must stay untouched)
    grid0[grid0 < 0] = -1.0
    noise = torch.rand(C, H3, 3, generator=g)
    scales = torch.empty(16, device=DEV)
    S = float(np.log2(enc.per_level_scale))
    L_.call("ntx_grid_level_scales", S, 16, 16, L_.ptr(scales), L_.stream())

    def oracle_update(grid, cells, nz):
        grid = grid.copy()
        tmp = -np.ones_like(grid)
        emb = enc.embeddings.detach().half().cpu().numpy()
        for cas in range(C):
            cb = min(2.0 ** cas, bound)
            hgs = cb / H
            idx = np.arange(H3, dtype=np.int64) if cells is None else cells[cas].astype(np.int64)
            coords = O.morton3D_invert(idx.astype(np.int32)).astype(np.float32)
            xyz = (np.float32(2) * coords * np.float32(1.0 / np.float32(H - 1)) - np.float32(1)) * np.float32(cb - hgs)
            if nz is not None:
                rows = np.arange(len(idx)) if cells is not None else (coords[:, 0].astype(np.int64) * H + coords[:, 1].astype(np.int64)) * H + coords[:, 2].astype(np.int64)
                xyz = xyz + (nz[cas][rows] * np.float32(2) - np.float32(1)) * np.float32(hgs)
            dirs = np.zeros_like(xyz); dirs[:, 2] = 1
            sig, _ = O.ngp_field(xyz.astype(np.float32), dirs.astype(np.float32), bound, emb, enc.offsets.cpu().numpy(), float(enc.per_level_scale), 16,
                                 net.weights.detach().half().cpu().numpy(), np.zeros(64 * (32 + 128 + 16), np.float16), align_corners=True,
                                 level_scales=scales.cpu().numpy())
            tmp[cas, idx] = sig
        valid = (grid >= 0) & (tmp >= 0)
        grid[valid] = np.maximum(grid[valid] * np.float32(0.95), tmp[valid])
        return grid, tmp

    for cells in (None, torch.randint(0, H3, (C, 5000), generator=g).to(torch.int32)):
        nz = noise if cells is None else noise[:, :5000].contiguous()
        dgrid = grid0.clone().to(DEV)
        bits = torch.zeros(C * H3 // 8, dtype=torch.uint8, device=DEV)
        stats = density.update_density_grid(dgrid, bits, bound, 1.0, 0.01, enc, net, decay=0.95, cells=cells, noise=nz)
        torch.cuda.synchronize()
        want, tmp = oracle_update(grid0.numpy(), None if cells is None else cells.numpy(), nz.numpy())
        got = dgrid.cpu().numpy()
        if cells is not None:      # duplicate cells in the list: either writer may win — compare where the list names a cell once
            flat = cells.numpy().astype(np.int64) + (np.arange(C)[:, None] * H3)
            uniq, cnt = np.unique(flat, return_counts=True)
            keep = np.ones(C * H3, bool); keep[uniq[cnt > 1]] = False
            got, want = got.reshape(-1)[keep], want.reshape(-1)[keep]
        # sigma = exp(fp16 h): the oracle's MLP differs from tcgen05 by a few fp16 ulp of h -> relative 4 * 2^-10 on sigma
        np.testing.assert_allclose(got, want, rtol=8e-3, atol=1e-6)
        mean = float(np.clip(dgrid.cpu().numpy(), 0, None).mean())
        assert abs(float(stats[0]) - mean) <= 1e-5 * max(1.0, mean)
        thr = float(stats[1])
        assert thr == pytest.approx(min(mean, 0.01), rel=1e-5)
        np.testing.assert_array_equal(bits.cpu().numpy(), O.packbits(dgrid.cpu().numpy(), thr))
