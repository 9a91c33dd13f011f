"""GPU parity of the tcgen05 fully-fused MLP (C ABI: ntx_ffmlp_inference / ntx_ffmlp_forward).

The reference accumulates in fp16 inside wmma fragments (ffmlp.cu:68), the B200 kernel in fp32 (TMEM); both round the
activations to fp16 once per layer.  So (SURVEY.md F6):
  * vs the oracle with the same rounding points (acc_mode 0): equal up to fp32 summation order, i.e. <= 1 fp16 ulp flips
    that can propagate through the layers -> a few fp16 ulp of the output scale;
  * vs the reference CUDA: our error w.r.t. an fp64 evaluation must not exceed the reference's own error (its outputs on the
    same seeded inputs are stored in tests/golden/reference_outputs.npz).
"""
import numpy as np
import pytest
import torch

from _util import ntx, oracle, ref, reference_output, ulp16

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _weights(rng, in_dim, hidden, layers, scale=None):
    n = hidden * (in_dim + hidden * (layers - 1) + 16)
    s = np.sqrt(3.0 / hidden) if scale is None else scale
    return ((rng.random(n, dtype=np.float32) * 2 - 1) * s).astype(np.float16)


def _fp64_mlp(x, w, in_dim, hidden, layers, act="relu"):
    x = x.astype(np.float64)
    o = 0
    W0 = w[o:o + hidden * in_dim].astype(np.float64).reshape(hidden, in_dim); o += hidden * in_dim
    h = np.maximum(x @ W0.T, 0)
    for _ in range(layers - 1):
        Wk = w[o:o + hidden * hidden].astype(np.float64).reshape(hidden, hidden); o += hidden * hidden
        h = np.maximum(h @ Wk.T, 0)
    Wl = w[o:o + 16 * hidden].astype(np.float64).reshape(16, hidden)
    return h @ Wl.T


def _run(L_, x, w, in_dim, hidden, layers, act=0, out_act=6, train=False):
    xt = torch.from_numpy(x).to(DEV)
    wt = torch.from_numpy(w).to(DEV)
    B = x.shape[0]
    out = torch.full((B, 16), float("nan"), dtype=torch.half, device=DEV)
    if train:
        fb = torch.full((layers, B, hidden), float("nan"), dtype=torch.half, device=DEV)
        L_.call("ntx_ffmlp_forward", xt.data_ptr(), wt.data_ptr(), B, in_dim, 16, hidden, layers, act, out_act, fb.data_ptr(), out.data_ptr(), L_.stream())
        torch.cuda.synchronize()
        return out.cpu().numpy(), fb.cpu().numpy()
    L_.call("ntx_ffmlp_inference", xt.data_ptr(), wt.data_ptr(), B, in_dim, 16, hidden, layers, act, out_act, None, out.data_ptr(), L_.stream())
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("in_dim,hidden,layers,B", [
    (32, 64, 2, 4096),      # sigma net of network_ff
    (32, 64, 3, 4096),      # colour net
    (16, 16, 2, 1024), (32, 32, 2, 1024 + 300), (64, 64, 4, 640), (48, 128, 2, 2048), (32, 128, 3, 257), (32, 256, 2, 512), (16, 64, 2, 1),
])
def test_inference_matches_oracle_and_beats_reference_error(in_dim, hidden, layers, B):
    L_ = ntx()
    O = oracle()
    rng = np.random.default_rng(in_dim + hidden + layers)
    x = (rng.standard_normal((B, in_dim)) * 0.5).astype(np.float16)
    w = _weights(rng, in_dim, hidden, layers)
    got = _run(L_, x, w, in_dim, hidden, layers).astype(np.float32)
    assert np.isfinite(got).all()
    want = O.ffmlp_forward(x, w, in_dim, 16, hidden, layers, acc_mode=0).astype(np.float32)
    truth = _fp64_mlp(x, w, in_dim, hidden, layers)
    scale = np.abs(truth).max()
    # same rounding points: a handful of fp16 ulps of the output scale at most
    assert np.abs(got - want).max() <= 4 * ulp16(scale), (np.abs(got - want).max(), ulp16(scale))
    err_ours = np.abs(got - truth).max()
    if B % 128 == 0 and hidden <= 128:
        live = {}

        def ref_out():
            if not live:
                m = ref("ffmlp")
                m.allocate_splitk(layers + 1)
                xt, wt = torch.from_numpy(x).to(DEV), torch.from_numpy(w).to(DEV)
                rout = torch.empty(B, 16, dtype=torch.half, device=DEV)
                rbuf = torch.empty(B, hidden, dtype=torch.half, device=DEV)
                m.ffmlp_inference(xt, wt, B, in_dim, 16, hidden, layers, 0, 6, rbuf, rout)
                torch.cuda.synchronize()
                live["out"] = rout.cpu().numpy().astype(np.float32)
            return live["out"]
        key = "ffmlp_inference_%d_%d_%d_%d" % (in_dim, hidden, layers, B)
        err_ref = reference_output(key + "_max_error", lambda: np.abs(ref_out() - truth).max())
        assert err_ours <= err_ref * 1.05 + ulp16(scale), (err_ours, err_ref)
        # and the two implementations agree to the reference's own accuracy
        rgot = reference_output(key, ref_out)
        assert np.abs(rgot.take(got) - rgot.sample).max() <= 2 * err_ref + 2 * ulp16(scale)


def test_forward_buffer_and_ragged_tiles():
    L_ = ntx()
    O = oracle()
    rng = np.random.default_rng(11)
    for B in (128, 1000):
        x = (rng.standard_normal((B, 32)) * 0.5).astype(np.float16)
        w = _weights(rng, 32, 64, 2)
        out, fb = _run(L_, x, w, 32, 64, 2, train=True)
        want, wfb = O.ffmlp_forward(x, w, 32, 16, 64, 2, want_forward_buffer=True)
        assert np.isfinite(fb.astype(np.float32)).all() and np.isfinite(out.astype(np.float32)).all()
        assert (fb >= 0).all()
        d = np.abs(fb.astype(np.float32) - wfb.astype(np.float32))
        assert d.max() <= 4 * ulp16(np.abs(wfb.astype(np.float32)).max())
        assert np.abs(out.astype(np.float32) - want.astype(np.float32)).max() <= 4 * ulp16(np.abs(want.astype(np.float32)).max())
        inf = _run(L_, x, w, 32, 64, 2)
        np.testing.assert_array_equal(inf, out)   # training and inference variants compute the same thing


@pytest.mark.parametrize("act", [1, 2, 3, 4, 5, 6])
def test_other_activations(act):
    L_ = ntx()
    O = oracle()
    rng = np.random.default_rng(act)
    x = (rng.standard_normal((512, 32)) * 0.3).astype(np.float16)
    w = _weights(rng, 32, 32, 2, scale=0.2)
    got = _run(L_, x, w, 32, 32, 2, act=act, out_act=act if act in (3, 6) else 6).astype(np.float32)
    want = O.ffmlp_forward(x, w, 32, 16, 32, 2, activation=act, output_activation=act if act in (3, 6) else 6).astype(np.float32)
    assert np.isfinite(got).all()
    assert np.abs(got - want).max() <= 8 * ulp16(np.abs(want).max())


def test_argument_errors():
    L_ = ntx()
    a = torch.zeros(128, 32, dtype=torch.half, device=DEV)
    w = torch.zeros(64 * (32 + 64 + 16), dtype=torch.half, device=DEV)
    o = torch.zeros(128, 16, dtype=torch.half, device=DEV)
    with pytest.raises(RuntimeError, match="hidden_dim"):
        L_.call("ntx_ffmlp_inference", a.data_ptr(), w.data_ptr(), 128, 32, 16, 48, 2, 0, 6, None, o.data_ptr(), L_.stream())
    with pytest.raises(RuntimeError, match="input_dim"):
        L_.call("ntx_ffmlp_inference", a.data_ptr(), w.data_ptr(), 128, 20, 16, 64, 2, 0, 6, None, o.data_ptr(), L_.stream())
