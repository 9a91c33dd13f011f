"""GPU parity of the hash-grid encoder: libntx (through the C ABI) vs the CPU oracle and vs the reference's own CUDA (its outputs
on the same seeded inputs, stored in tests/golden/reference_outputs.npz).

Bars (SURVEY.md F6 / section 8c):
  * integer corner-index streams: bit-exact vs the oracle (fed the device's per-level scales);
  * fp32 and fp16 tables, forward: bit-exact vs the reference CUDA kernels (same operations, same rounding points);
    vs the oracle: bit-exact for fp16 and fp32 when the oracle is given the device scales;
  * backward (atomic order is arbitrary): fp32 rtol 1e-4 / fp16 within a few fp16 ulp of the fp64 result.
"""
import numpy as np
import pytest
import torch

from _util import cfgA, cfgB, cfgT, ntx, oracle, ref, reference_output

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _setup(cfg, B, dtype, seed=0, table_range=1.0, oob_frac=0.0):
    O = oracle()
    kw = dict(cfg)
    D = kw["input_dim"]
    offsets, pls = O.grid_offsets(**{k: v for k, v in kw.items() if k != "level_dim"})
    rng = np.random.default_rng(seed)
    x = rng.random((B, D), dtype=np.float32)
    if oob_frac > 0:
        n = int(B * oob_frac)
        x[:n, 0] = 1.0 + rng.random(n, dtype=np.float32)
        x[n:2 * n, D - 1] = -rng.random(n, dtype=np.float32) - 1e-3
    # exact boundary values are in range
    x[-1] = 1.0
    x[-2] = 0.0
    emb = ((rng.random((int(offsets[-1]), kw["level_dim"]), dtype=np.float32) * 2 - 1) * table_range).astype(dtype)
    return O, x, emb, offsets, pls, kw


def _device_scales(L_, S, H, nlev):
    out = torch.empty(nlev, dtype=torch.float32, device=DEV)
    L_.call("ntx_grid_level_scales", float(S), int(H), int(nlev), out.data_ptr(), L_.stream())
    return out.cpu().numpy()


def _ntx_forward(L_, x, emb, offsets, pls, H, gridtype, align, calc=False, layout=1):
    xt = torch.from_numpy(x).to(DEV)
    et = torch.from_numpy(emb).to(DEV)
    ot = torch.from_numpy(offsets).to(DEV)
    B, D = x.shape
    nlev = offsets.shape[0] - 1
    C = emb.shape[1]
    out = torch.empty((B, nlev * C) if layout == 1 else (nlev, B, C), dtype=et.dtype, device=DEV)
    dy = torch.empty(B, nlev * D * C, dtype=et.dtype, device=DEV) if calc else torch.empty(1, dtype=et.dtype, device=DEV)
    L_.call("ntx_grid_encode_forward", xt.data_ptr(), et.data_ptr(), ot.data_ptr(), out.data_ptr(), B, D, C, nlev, float(np.log2(pls)), int(H),
            int(calc), dy.data_ptr(), int(gridtype), int(align), L_.dtype_id(et.dtype), layout, L_.stream())
    torch.cuda.synchronize()
    return out.cpu().numpy(), (dy.cpu().numpy() if calc else None)


def _ref_forward(x, emb, offsets, pls, H, gridtype, align, calc=False):
    m = ref("gridencoder")
    xt = torch.from_numpy(x).to(DEV)
    et = torch.from_numpy(emb).to(DEV)
    ot = torch.from_numpy(offsets).to(DEV)
    B, D = x.shape
    nlev = offsets.shape[0] - 1
    C = emb.shape[1]
    out = torch.empty(nlev, B, C, dtype=et.dtype, device=DEV)
    dy = torch.empty(B, nlev * D * C, dtype=et.dtype, device=DEV) if calc else torch.empty(1, dtype=et.dtype, device=DEV)
    m.grid_encode_forward(xt, et, ot, out, B, D, C, nlev, float(np.log2(pls)), int(H), calc, dy, gridtype, align)
    torch.cuda.synchronize()
    return out.permute(1, 0, 2).reshape(B, nlev * C).cpu().numpy(), (dy.cpu().numpy() if calc else None)


def test_level_scales_close_to_host():
    L_ = ntx()
    O = oracle()
    for cfg in (cfgA(), cfgB(), cfgT()):
        offsets, pls = O.grid_offsets(**{k: v for k, v in cfg.items() if k != "level_dim"})
        S = np.float32(np.log2(pls))
        dev = _device_scales(L_, S, cfg["base_resolution"], cfg["num_levels"])
        host = O.grid_level_scales(S, cfg["base_resolution"], cfg["num_levels"])
        np.testing.assert_allclose(dev, host, rtol=3e-7)
        # the resolutions (ceil(scale)+1) that size the dense levels must agree exactly
        np.testing.assert_array_equal(np.ceil(dev), np.ceil(host))


@pytest.mark.parametrize("cfg,gridtype", [(cfgA(), 0), (cfgB(), 0), (cfgT(), 0), (cfgA(), 1), (dict(cfgB(), input_dim=2), 0)])
def test_index_stream_bit_exact(cfg, gridtype):
    L_ = ntx()
    O, x, emb, offsets, pls, kw = _setup(cfg, 8192, np.float32, oob_frac=0.05)
    S = np.float32(np.log2(pls))
    scales = _device_scales(L_, S, kw["base_resolution"], kw["num_levels"])
    xt = torch.from_numpy(x).to(DEV)
    ot = torch.from_numpy(offsets).to(DEV)
    D = kw["input_dim"]
    for level in range(kw["num_levels"]):
        out = torch.empty(x.shape[0], 1 << D, dtype=torch.int32, device=DEV)
        L_.call("ntx_grid_debug_indices", xt.data_ptr(), ot.data_ptr(), x.shape[0], D, level, float(S), kw["base_resolution"], gridtype,
                int(kw["align_corners"]), out.data_ptr(), L_.stream())
        got = out.cpu().numpy().view(np.uint32)
        want = O.grid_indices(x, offsets, level, scales[level], gridtype, kw["align_corners"])
        np.testing.assert_array_equal(got, want, err_msg="level %d" % level)


@pytest.mark.parametrize("cfg", [cfgA(), cfgB(), cfgT()], ids=["cfgA", "cfgB", "cfgT"])
@pytest.mark.parametrize("dtype", [np.float32, np.float16], ids=["f32", "f16"])
def test_forward_pair_kernel_bit_exact(cfg, dtype):
    L_ = ntx()
    O, x, emb, offsets, pls, kw = _setup(cfg, 4096 + 37, dtype, oob_frac=0.03)
    H, align = kw["base_resolution"], kw["align_corners"]
    got, _ = _ntx_forward(L_, x, emb, offsets, pls, H, 0, align)
    scales = _device_scales(L_, np.float32(np.log2(pls)), H, kw["num_levels"])
    want = O.grid_encode(x, emb, offsets, pls, H, gridtype=0, align_corners=align, level_scales=scales)
    np.testing.assert_array_equal(got.view(np.uint16 if dtype == np.float16 else np.uint32),
                                  want.view(np.uint16 if dtype == np.float16 else np.uint32))
    bits = np.uint16 if dtype == np.float16 else np.uint32
    rgot = reference_output("grid_pair_L%d_H%d_%s" % (kw["num_levels"], H, np.dtype(dtype).name),
                            lambda: _ref_forward(x, emb, offsets, pls, H, 0, align)[0].view(bits), exact=True)
    rgot.assert_equal(got.view(bits))
    # [L,B,C] layout of the same kernel
    got_lbc, _ = _ntx_forward(L_, x, emb, offsets, pls, H, 0, align, layout=0)
    nlev, C = kw["num_levels"], kw["level_dim"]
    np.testing.assert_array_equal(got_lbc.transpose(1, 0, 2).reshape(x.shape[0], nlev * C), got)


@pytest.mark.parametrize("D,C,gridtype,align,dtype", [
    (3, 1, 0, False, np.float32), (3, 4, 0, True, np.float16), (3, 8, 0, False, np.float32), (2, 2, 0, False, np.float16),
    (2, 4, 1, True, np.float32), (3, 2, 1, False, np.float16), (3, 2, 0, True, np.float64), (3, 1, 0, True, np.float16),
])
def test_forward_generic_and_dydx(D, C, gridtype, align, dtype):
    L_ = ntx()
    cfg = dict(input_dim=D, num_levels=6, level_dim=C, per_level_scale=1.7, base_resolution=8, log2_hashmap_size=12, align_corners=align)
    O, x, emb, offsets, pls, kw = _setup(cfg, 2048 + 5, dtype, oob_frac=0.03)
    H = kw["base_resolution"]
    got, gdy = _ntx_forward(L_, x, emb, offsets, pls, H, gridtype, align, calc=True)
    scales = _device_scales(L_, np.float32(np.log2(pls)), H, kw["num_levels"])
    want_lbc, wdy = O.grid_encode_forward(x, emb, offsets, pls, H, calc_grad_inputs=True, gridtype=gridtype, align_corners=align, level_scales=scales)
    want = want_lbc.transpose(1, 0, 2).reshape(got.shape)
    if dtype == np.float64:
        np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(gdy, wdy, rtol=1e-12, atol=1e-12)
    else:
        np.testing.assert_array_equal(got, want)
        np.testing.assert_array_equal(gdy, wdy)
    key = "grid_generic_D%d_C%d_t%d_a%d_%s" % (D, C, gridtype, align, np.dtype(dtype).name)
    live = {}

    def ref_run(i):
        if not live:
            live["r"] = _ref_forward(x, emb, offsets, pls, H, gridtype, align, calc=True)
        return live["r"][i]
    reference_output(key + "_out", lambda: ref_run(0), exact=True).assert_equal(got)
    reference_output(key + "_dydx", lambda: ref_run(1), exact=True).assert_equal(gdy)


def test_out_of_range_rows_are_zero():
    L_ = ntx()
    O, x, emb, offsets, pls, kw = _setup(cfgA(), 1024, np.float16, oob_frac=0.25)
    got, _ = _ntx_forward(L_, x, emb, offsets, pls, 16, 0, True)
    oob = ((x < 0) | (x > 1)).any(1)
    assert oob.sum() > 100
    assert np.all(got[oob] == 0)
    assert np.all(np.abs(got[~oob]).sum(1) > 0)


def test_unsupported_shapes_raise_runtime_error():
    L_ = ntx()
    a = torch.zeros(8, 3, device=DEV)
    e = torch.zeros(64, 3, device=DEV)
    o = torch.tensor([0, 64], dtype=torch.int32, device=DEV)
    out = torch.zeros(8, 3, device=DEV)
    with pytest.raises(RuntimeError, match="C must be 1, 2, 4, or 8"):
        L_.call("ntx_grid_encode_forward", a.data_ptr(), e.data_ptr(), o.data_ptr(), out.data_ptr(), 8, 3, 3, 1, 1.0, 16, 0, None, 0, 0, 0, 1, L_.stream())
    with pytest.raises(RuntimeError):
        L_.call("ntx_grid_encode_forward", a.data_ptr(), e.data_ptr(), o.data_ptr(), out.data_ptr(), 8, 4, 2, 1, 1.0, 16, 0, None, 0, 0, 0, 1, L_.stream())


@pytest.mark.parametrize("dtype", [np.float32, np.float16], ids=["f32", "f16"])
@pytest.mark.parametrize("cfg", [cfgB(), cfgA()], ids=["cfgB", "cfgA"])
def test_backward_table_and_input_grads(cfg, dtype):
    L_ = ntx()
    B = 4096
    O, x, emb, offsets, pls, kw = _setup(cfg, B, dtype, oob_frac=0.02, seed=3)
    H, align, nlev, C, D = kw["base_resolution"], kw["align_corners"], kw["num_levels"], kw["level_dim"], kw["input_dim"]
    rng = np.random.default_rng(5)
    grad = rng.standard_normal((B, nlev * C)).astype(dtype)
    scales = _device_scales(L_, np.float32(np.log2(pls)), H, nlev)
    # forward with dy_dx to feed the input gradient
    _, gdy = _ntx_forward(L_, x, emb, offsets, pls, H, 0, align, calc=True)
    xt, et, ot = torch.from_numpy(x).to(DEV), torch.from_numpy(emb).to(DEV), torch.from_numpy(offsets).to(DEV)
    gt = torch.from_numpy(grad).to(DEV)
    dyt = torch.from_numpy(gdy).to(DEV)
    ge = torch.zeros_like(et)
    gi = torch.zeros(B, D, dtype=et.dtype, device=DEV)
    L_.call("ntx_grid_encode_backward", gt.data_ptr(), xt.data_ptr(), et.data_ptr(), ot.data_ptr(), ge.data_ptr(), B, D, C, nlev, float(np.log2(pls)), H, 1,
            dyt.data_ptr(), gi.data_ptr(), 0, int(align), L_.dtype_id(et.dtype), 1, L_.stream())
    torch.cuda.synchronize()
    # fp64 truth from the oracle
    grad_lbc = np.ascontiguousarray(grad.reshape(B, nlev, C).transpose(1, 0, 2)).astype(np.float64)
    ge64, gi64 = O.grid_encode_backward(grad_lbc, x, emb.astype(np.float64), offsets, pls, H, dy_dx=gdy.astype(np.float64), align_corners=align,
                                        level_scales=scales)
    got_ge, got_gi = ge.cpu().numpy().astype(np.float64), gi.cpu().numpy().astype(np.float64)
    scale = np.abs(ge64).max()
    if dtype == np.float32:
        np.testing.assert_allclose(got_ge, ge64, rtol=1e-4, atol=1e-5 * scale)
        np.testing.assert_allclose(got_gi, gi64, rtol=1e-3, atol=1e-3 * np.abs(gi64).max())
    else:
        # fp16 atomics round after every add: error grows with the number of contributions per entry
        err = np.abs(got_ge - ge64)
        assert err.max() <= 0.02 * scale + 1e-3, (err.max(), scale)
        assert np.abs(got_gi - gi64).max() <= 0.05 * np.abs(gi64).max()
    # the reference's own backward on the same inputs has the same kind of error; ours must not be worse by much
    def ref_error():
        m = ref("gridencoder")
        rge = torch.zeros_like(et)
        rgi = torch.zeros(B, D, dtype=et.dtype, device=DEV)
        glbc = gt.view(B, nlev, C).permute(1, 0, 2).contiguous()
        m.grid_encode_backward(glbc, xt, et, ot, rge, B, D, C, nlev, float(np.log2(pls)), H, True, dyt, rgi, 0, align)
        torch.cuda.synchronize()
        return np.abs(rge.cpu().numpy().astype(np.float64) - ge64).max()
    ref_err = reference_output("grid_backward_L%d_%s_max_error" % (nlev, np.dtype(dtype).name), ref_error)
    our_err = np.abs(got_ge - ge64).max()
    assert our_err <= 2.0 * ref_err + 1e-6 * scale, (our_err, ref_err)
