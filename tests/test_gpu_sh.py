"""GPU parity of the SH direction encoder vs the oracle (fp64 evaluation of the same polynomials) and the reference CUDA (its outputs on
the same inputs, stored in tests/golden/reference_outputs.npz)."""
import numpy as np
import pytest
import torch

from _util import ntx, oracle, ref, reference_output

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _dirs(B, seed, unit=True):
    rng = np.random.default_rng(seed)
    d = rng.standard_normal((B, 3)).astype(np.float32)
    if unit:
        d /= np.linalg.norm(d, axis=1, keepdims=True)
    else:
        d *= 0.7   # the reference does not normalise its input: parity must hold off the sphere too
    return d


@pytest.mark.parametrize("degree", range(1, 9))
@pytest.mark.parametrize("unit", [True, False])
def test_forward_and_dydx(degree, unit):
    L_ = ntx()
    O = oracle()
    B = 3000 + degree
    d = _dirs(B, degree, unit)
    dt = torch.from_numpy(d).to(DEV)
    out = torch.empty(B, degree * degree, device=DEV)
    dy = torch.empty(B, 3 * degree * degree, device=DEV)
    L_.call("ntx_sh_encode_forward", dt.data_ptr(), out.data_ptr(), B, 3, degree, 1, dy.data_ptr(), L_.stream())
    out2 = torch.empty_like(out)
    L_.call("ntx_sh_encode_forward", dt.data_ptr(), out2.data_ptr(), B, 3, degree, 0, None, L_.stream())
    torch.cuda.synchronize()
    want, wdy = O.sh_encode_forward(d, degree, calc_grad_inputs=True)
    got, gdy = out.cpu().numpy(), dy.cpu().numpy()
    np.testing.assert_array_equal(got, out2.cpu().numpy())
    # fp32 polynomial evaluation vs fp64: absolute error relative to the coefficient scale of the band
    tol = 8e-6 * max(1.0, np.abs(want).max())
    assert np.abs(got - want).max() <= tol
    assert np.abs(gdy - wdy).max() <= 2e-5 * max(1.0, np.abs(wdy).max())
    live = {}

    def ref_run(i):
        if not live:
            m = ref("shencoder")
            rout = torch.empty_like(out)
            rdy = torch.empty_like(dy)
            m.sh_encode_forward(dt, rout, B, 3, degree, True, rdy)
            torch.cuda.synchronize()
            live["r"] = rout.cpu().numpy(), rdy.cpu().numpy()
        return live["r"][i]
    key = "sh_deg%d_%s" % (degree, "unit" if unit else "offsphere")
    rerr = reference_output(key + "_max_error", lambda: np.abs(ref_run(0) - want).max())
    rout, rdy = reference_output(key + "_out", lambda: ref_run(0)), reference_output(key + "_dydx", lambda: ref_run(1))
    assert np.abs(rout.take(got) - rout.sample).max() <= tol + rerr
    assert np.abs(got - want).max() <= max(2 * rerr, tol)
    assert np.abs(rdy.take(gdy) - rdy.sample).max() <= 4e-5 * max(1.0, np.abs(wdy).max())


def test_backward_accumulates():
    L_ = ntx()
    O = oracle()
    B, degree = 2048, 4
    d = _dirs(B, 1)
    rng = np.random.default_rng(2)
    g = rng.standard_normal((B, 16)).astype(np.float32)
    dt, gt = torch.from_numpy(d).to(DEV), torch.from_numpy(g).to(DEV)
    out = torch.empty(B, 16, device=DEV)
    dy = torch.empty(B, 48, device=DEV)
    L_.call("ntx_sh_encode_forward", dt.data_ptr(), out.data_ptr(), B, 3, degree, 1, dy.data_ptr(), L_.stream())
    gi = torch.zeros(B, 3, device=DEV)
    L_.call("ntx_sh_encode_backward", gt.data_ptr(), dt.data_ptr(), B, 3, degree, dy.data_ptr(), gi.data_ptr(), L_.stream())
    torch.cuda.synchronize()
    want = O.sh_encode_backward(g, degree, dy.cpu().numpy())
    np.testing.assert_allclose(gi.cpu().numpy(), want, rtol=1e-5, atol=1e-5)


def test_errors():
    L_ = ntx()
    a = torch.zeros(8, 3, device=DEV)
    o = torch.zeros(8, 100, device=DEV)
    with pytest.raises(RuntimeError, match="degree"):
        L_.call("ntx_sh_encode_forward", a.data_ptr(), o.data_ptr(), 8, 3, 9, 0, None, L_.stream())
    with pytest.raises(RuntimeError, match="input dim"):
        L_.call("ntx_sh_encode_forward", a.data_ptr(), o.data_ptr(), 8, 2, 4, 0, None, L_.stream())
