"""GPU parity of the fused field kernel (hash-grid -> sigma MLP -> SH -> colour MLP in one launch).

Checked against
  * the same pipeline assembled from the stand-alone libntx ops + torch glue exactly like nerf/network_ff.py:85-101 does
    under fp16 autocast (must agree to the last bit: same kernels' arithmetic, only the data movement differs);
  * the CPU oracle composition (fp32 accumulation order may differ -> a few fp16 ulp);
  * the reference's own CUDA ops assembled the same way (fp16 accumulation in its MLP -> its own error bar; its outputs on these seeded
    inputs are stored in tests/golden/reference_outputs.npz).
"""
import numpy as np
import pytest
import torch

from _util import cfgA, cfgT, ntx, oracle, ref, reference_output, ulp16

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _make(cfg, M, seed=0, bound=1.0, coherent=False):
    O = oracle()
    offsets, pls = O.grid_offsets(**{k: v for k, v in cfg.items() if k != "level_dim"})
    rng = np.random.default_rng(seed)
    if coherent:
        o = rng.random((M // 64 + 1, 3), dtype=np.float32) * 0.2 - 0.1
        d = rng.standard_normal((M // 64 + 1, 3)).astype(np.float32)
        d /= np.linalg.norm(d, axis=1, keepdims=True)
        t = (np.arange(64, dtype=np.float32) * 0.0034)[None, :, None]
        xyz = (o[:, None, :] + t * d[:, None, :]).reshape(-1, 3)[:M]
        dirs = np.repeat(d, 64, axis=0)[:M]
    else:
        xyz = (rng.random((M, 3), dtype=np.float32) * 2 - 1) * bound
        dirs = rng.standard_normal((M, 3)).astype(np.float32)
        dirs /= np.linalg.norm(dirs, axis=1, keepdims=True)
    xyz = np.ascontiguousarray(xyz.astype(np.float32))
    dirs = np.ascontiguousarray(dirs.astype(np.float32))
    emb = (rng.random((int(offsets[-1]), 2), dtype=np.float32) * 2 - 1).astype(np.float16)
    nfeat = 2 * cfg["num_levels"]
    ws = ((rng.random(64 * (nfeat + 64 + 16), dtype=np.float32) * 2 - 1) * np.sqrt(3 / 64)).astype(np.float16)
    wc = ((rng.random(64 * (32 + 64 * 2 + 16), dtype=np.float32) * 2 - 1) * np.sqrt(3 / 64)).astype(np.float16)
    return O, xyz, dirs, emb, offsets, pls, ws, wc


def _fused(L_, xyz, dirs, emb, offsets, pls, H, align, ws, wc, bound, density_scale=1.0, deltas=None):
    M = xyz.shape[0]
    xt, dt, et, ot, wst, wct = (torch.from_numpy(a).to(DEV) for a in (xyz, dirs, emb, offsets, ws, wc))
    dl = None if deltas is None else torch.from_numpy(deltas).to(DEV)
    sig = torch.full((M,), float("nan"), device=DEV)
    rgb = torch.full((M, 3), float("nan"), device=DEV)
    L_.call("ntx_ngp_field_forward", xt.data_ptr(), dt.data_ptr(), None if dl is None else dl.data_ptr(), M, float(bound), et.data_ptr(), ot.data_ptr(),
            offsets.shape[0] - 1, float(np.log2(pls)), int(H), int(align), wst.data_ptr(), wct.data_ptr(), float(density_scale), sig.data_ptr(),
            rgb.data_ptr(), L_.stream())
    torch.cuda.synchronize()
    return sig.cpu().numpy(), rgb.cpu().numpy()


def _composed_ntx(L_, xyz, dirs, emb, offsets, pls, H, align, ws, wc, bound):
    """network_ff.forward with the stand-alone ops"""
    M = xyz.shape[0]
    nlev = offsets.shape[0] - 1
    xt, dt, et, ot, wst, wct = (torch.from_numpy(a).to(DEV) for a in (xyz, dirs, emb, offsets, ws, wc))
    x01 = ((xt + bound) / (2 * bound)).contiguous()
    feat = torch.empty(M, nlev * 2, dtype=torch.half, device=DEV)
    L_.call("ntx_grid_encode_forward", x01.data_ptr(), et.data_ptr(), ot.data_ptr(), feat.data_ptr(), M, 3, 2, nlev, float(np.log2(pls)), int(H), 0, None, 0,
            int(align), L_.F16, L_.LAYOUT_BLC, L_.stream())
    h = torch.empty(M, 16, dtype=torch.half, device=DEV)
    L_.call("ntx_ffmlp_inference", feat.data_ptr(), wst.data_ptr(), M, nlev * 2, 16, 64, 2, 0, 6, None, h.data_ptr(), L_.stream())
    sigma = torch.exp(h[:, 0].float())
    sh = torch.empty(M, 16, device=DEV)
    L_.call("ntx_sh_encode_forward", dt.data_ptr(), sh.data_ptr(), M, 3, 4, 0, None, L_.stream())
    cin = torch.cat([sh, h[:, 1:].float(), torch.zeros(M, 1, device=DEV)], dim=-1).half().contiguous()
    hc = torch.empty(M, 16, dtype=torch.half, device=DEV)
    L_.call("ntx_ffmlp_inference", cin.data_ptr(), wct.data_ptr(), M, 32, 16, 64, 3, 0, 6, None, hc.data_ptr(), L_.stream())
    rgb = torch.sigmoid(hc[:, :3]).float()
    torch.cuda.synchronize()
    return sigma.cpu().numpy(), rgb.cpu().numpy(), h.cpu().numpy()


def _composed_ref(xyz, dirs, emb, offsets, pls, H, align, ws, wc, bound):
    g, f, s = ref("gridencoder"), ref("ffmlp"), ref("shencoder")
    f.allocate_splitk(4)
    M = xyz.shape[0]
    nlev = offsets.shape[0] - 1
    xt, dt, et, ot, wst, wct = (torch.from_numpy(a).to(DEV) for a in (xyz, dirs, emb, offsets, ws, wc))
    x01 = ((xt + bound) / (2 * bound)).contiguous()
    out = torch.empty(nlev, M, 2, dtype=torch.half, device=DEV)
    dy = torch.empty(1, dtype=torch.half, device=DEV)
    g.grid_encode_forward(x01, et, ot, out, M, 3, 2, nlev, float(np.log2(pls)), int(H), False, dy, 0, align)
    feat = out.permute(1, 0, 2).reshape(M, nlev * 2).contiguous()
    h = torch.empty(M, 16, dtype=torch.half, device=DEV)
    buf = torch.empty(M, 64, dtype=torch.half, device=DEV)
    f.ffmlp_inference(feat, wst, M, nlev * 2, 16, 64, 2, 0, 6, buf, h)
    sigma = torch.exp(h[:, 0].float())
    sh = torch.empty(M, 16, device=DEV)
    s.sh_encode_forward(dt, sh, M, 3, 4, False, torch.empty(1, device=DEV))
    cin = torch.cat([sh, h[:, 1:].float(), torch.zeros(M, 1, device=DEV)], dim=-1).half().contiguous()
    hc = torch.empty(M, 16, dtype=torch.half, device=DEV)
    f.ffmlp_inference(cin, wct, M, 32, 16, 64, 3, 0, 6, buf, hc)
    rgb = torch.sigmoid(hc[:, :3]).float()
    torch.cuda.synchronize()
    return sigma.cpu().numpy(), rgb.cpu().numpy()


@pytest.mark.parametrize("cfg,M,bound,coherent", [(cfgA(), 128 * 40, 1.0, False), (cfgA(), 128 * 33 + 17, 1.0, True), (cfgT(), 128 * 16, 2.0, False)],
                         ids=["cfgA-random", "cfgA-coherent-ragged", "cfgT-bound2"])
def test_fused_field_matches_composition_oracle_and_reference(cfg, M, bound, coherent):
    L_ = ntx()
    O, xyz, dirs, emb, offsets, pls, ws, wc = _make(cfg, M, bound=bound, coherent=coherent)
    H, align = cfg["base_resolution"], cfg["align_corners"]
    sig, rgb = _fused(L_, xyz, dirs, emb, offsets, pls, H, align, ws, wc, bound)
    assert np.isfinite(sig).all() and np.isfinite(rgb).all()
    csig, crgb, ch = _composed_ntx(L_, xyz, dirs, emb, offsets, pls, H, align, ws, wc, bound)
    np.testing.assert_array_equal(sig, csig)
    np.testing.assert_array_equal(rgb, crgb)

    scales = torch.empty(cfg["num_levels"], device=DEV)
    L_.call("ntx_grid_level_scales", float(np.log2(pls)), int(H), cfg["num_levels"], scales.data_ptr(), L_.stream())
    osig, orgb = O.ngp_field(xyz, dirs, bound, emb, offsets, pls, H, ws, wc, align_corners=align, level_scales=scales.cpu().numpy())
    # sigma = exp(h0): a 1-ulp(fp16) flip of h0 changes sigma by up to ulp16(h0) relative
    h0 = ch[:, 0].astype(np.float32)
    rel = np.abs(sig - osig) / np.maximum(np.abs(osig), 1e-30)
    assert (rel <= 4 * ulp16(np.maximum(np.abs(h0), 1.0)) + 1e-6).all(), rel.max()
    assert np.abs(rgb - orgb).max() <= 4 * 2.0 ** -11 + 1e-6   # rgb in (0,1): a few fp16 ulps

    if M % 128 == 0:
        live = {}

        def ref_run(i):
            if not live:
                live["r"] = _composed_ref(xyz, dirs, emb, offsets, pls, H, align, ws, wc, bound)
            return live["r"][i]
        key = "field_L%d_H%d_M%d_%s" % (cfg["num_levels"], H, M, "coherent" if coherent else "random")
        # the reference MLP accumulates in fp16: compare both to the oracle; ours must be at least as close
        err_ref_rgb = reference_output(key + "_rgb_max_error", lambda: np.abs(ref_run(1) - orgb).max())
        err_our_rgb = np.abs(rgb - orgb).max()
        assert err_our_rgb <= err_ref_rgb + 2.0 ** -11
        rrgb = reference_output(key + "_rgb", lambda: ref_run(1))
        assert np.abs(rrgb.take(rgb) - rrgb.sample).max() <= 2 * err_ref_rgb + 4 * 2.0 ** -11
        rrel_median = reference_output(key + "_sigma_median_rel_error", lambda: np.median(np.abs(ref_run(0) - osig) / np.maximum(np.abs(osig), 1e-30)))
        assert np.median(rel) <= rrel_median + 1e-6


def test_fused_field_skips_sentinel_rows_and_scales_density():
    L_ = ntx()
    cfg = cfgA()
    O, xyz, dirs, emb, offsets, pls, ws, wc = _make(cfg, 1024, seed=3)
    deltas = np.full((1024, 2), 0.0034, np.float32)
    deltas[::3] = 0
    sig, rgb = _fused(L_, xyz, dirs, emb, offsets, pls, 16, True, ws, wc, 1.0, density_scale=2.5, deltas=deltas)
    sig1, rgb1 = _fused(L_, xyz, dirs, emb, offsets, pls, 16, True, ws, wc, 1.0)
    assert (sig[::3] == 0).all() and (rgb[::3] == 0).all()
    keep = np.ones(1024, bool); keep[::3] = False
    np.testing.assert_array_equal(sig[keep], (np.float32(2.5) * sig1[keep]).astype(np.float32))
    np.testing.assert_array_equal(rgb[keep], rgb1[keep])


def test_fused_field_many_launches_of_every_size_are_deterministic():
    """The kernel is a producer/consumer pipeline over mbarriers: a protocol slip shows up as a hang (the waits trap) or as
    run-to-run differences.  Launch it a few hundred times over ragged sizes — fewer tiles than CTAs, one row, many tiles per
    CTA — back to back without synchronising, and compare every size against its first result."""
    L_ = ntx()
    cfg = cfgA()
    Mmax = 128 * 1200 + 77
    O, xyz, dirs, emb, offsets, pls, ws, wc = _make(cfg, Mmax, seed=11, coherent=True)
    xt, dt, et, ot, wst, wct = (torch.from_numpy(a).to(DEV) for a in (xyz, dirs, emb, offsets, ws, wc))
    rng = np.random.default_rng(5)
    sizes = [1, 127, 128, 129, 128 * 296, 128 * 297 + 5, Mmax] + [int(s) for s in rng.integers(1, Mmax, size=40)]
    first = {}
    for rep in range(6):
        outs = []
        for M in sizes:
            sig = torch.full((M,), float("nan"), device=DEV)
            rgb = torch.full((M, 3), float("nan"), device=DEV)
            L_.call("ntx_ngp_field_forward", xt.data_ptr(), dt.data_ptr(), None, M, 1.0, et.data_ptr(), ot.data_ptr(), offsets.shape[0] - 1,
                    float(np.log2(pls)), 16, 0, wst.data_ptr(), wct.data_ptr(), 1.0, sig.data_ptr(), rgb.data_ptr(), L_.stream())
            outs.append((M, sig, rgb))
        torch.cuda.synchronize()
        for M, sig, rgb in outs:
            assert torch.isfinite(sig).all() and torch.isfinite(rgb).all()
            if M not in first:
                first[M] = (sig, rgb)
            else:
                assert torch.equal(first[M][0], sig) and torch.equal(first[M][1], rgb)
    # prefix property: rows are independent, so a shorter launch equals the head of the longest one
    big_sig, big_rgb = first[Mmax]
    for M, (sig, rgb) in first.items():
        assert torch.equal(big_sig[:M], sig) and torch.equal(big_rgb[:M], rgb)
