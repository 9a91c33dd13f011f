"""GPU parity of the ray-marching family vs the CPU oracle and the reference's own CUDA kernels.

Integer outputs (Morton codes, bit-fields, ray ids, sample offsets/counts, compacted ray ids) must be bit-exact; the
reference allocates output slots with global atomics (arbitrary order, SURVEY.md F7), so against it they are compared
as sets keyed by ray id, while against the oracle (ascending order, like libntx) they are compared directly.  The reference's
outputs on these seeded inputs are stored in tests/golden/reference_outputs.npz.
"""
import numpy as np
import pytest
import torch

from _util import ball_density_grid, ntx, oracle, pinhole_rays, ref, reference_output

pytestmark = pytest.mark.gpu
DEV = "cuda"


def T(a):
    return torch.from_numpy(np.ascontiguousarray(a)).to(DEV)


def _scene(Himg=48, Wimg=64, cascade=1, Hg=128, bound=1.0, radius=0.5, center=(0, 0, 0)):
    O = oracle()
    o, d = pinhole_rays(Himg, Wimg)
    grid = ball_density_grid(cascade, Hg, bound, radius, center)
    bits = O.packbits(grid, 0.5)
    aabb = np.array([-bound] * 3 + [bound] * 3, np.float32)
    nears, fars = O.near_far_from_aabb(o, d, aabb, 0.2)
    return O, o, d, grid, bits, aabb, nears, fars


def test_near_far_polar_morton_packbits():
    L_ = ntx()
    O, o, d, grid, bits, aabb, nears, fars = _scene(cascade=2, Hg=64, bound=2.0)
    N = o.shape[0]
    # make a few rays miss the box and a few axis-parallel
    o[:7] += 50.0
    d[7:11] = np.array([0.0, 0.0, -1.0], np.float32)
    nears, fars = O.near_far_from_aabb(o, d, aabb, 0.2)
    ot, dt, at = T(o), T(d), T(aabb)
    n_, f_ = torch.empty(N, device=DEV), torch.empty(N, device=DEV)
    L_.call("ntx_near_far_from_aabb", ot.data_ptr(), dt.data_ptr(), at.data_ptr(), N, 0.2, n_.data_ptr(), f_.data_ptr(), L_.stream())
    live = {}

    def ref_near_far(i):
        if not live:
            m = ref("raymarching")
            rn, rf = torch.empty(N, device=DEV), torch.empty(N, device=DEV)
            m.near_far_from_aabb(ot, dt, at, N, 0.2, rn, rf)
            torch.cuda.synchronize()
            live["r"] = rn.cpu().numpy(), rf.cpu().numpy()
        return live["r"][i]
    torch.cuda.synchronize()
    reference_output("near_far_nears", lambda: ref_near_far(0), exact=True).assert_equal(n_.cpu().numpy())
    reference_output("near_far_fars", lambda: ref_near_far(1), exact=True).assert_equal(f_.cpu().numpy())
    np.testing.assert_array_equal(n_.cpu().numpy(), nears)
    np.testing.assert_array_equal(f_.cpu().numpy(), fars)
    assert (nears[:7] > 1e38).all()

    o2, d2 = pinhole_rays(16, 16, radius=0.3)
    c_ = torch.empty(256, 2, device=DEV)
    o2t, d2t = T(o2), T(d2)   # keep alive: a temporary's storage is recycled as soon as data_ptr() returns
    L_.call("ntx_polar_from_ray", o2t.data_ptr(), d2t.data_ptr(), 4.0, 256, c_.data_ptr(), L_.stream())

    def ref_polar():
        rc = torch.empty(256, 2, device=DEV)
        ref("raymarching").polar_from_ray(o2t, d2t, 4.0, 256, rc)
        torch.cuda.synchronize()
        return rc.cpu().numpy()
    rc = reference_output("polar_from_ray", ref_polar)
    torch.cuda.synchronize()
    np.testing.assert_allclose(rc.take(c_.cpu().numpy()), rc.sample, rtol=0, atol=2e-7)
    np.testing.assert_allclose(c_.cpu().numpy(), O.polar_from_ray(o2, d2, 4.0), rtol=0, atol=2e-6)

    rng = np.random.default_rng(0)
    coords = rng.integers(0, 1024, (5000, 3)).astype(np.int32)
    ct = T(coords)
    idx = torch.empty(5000, dtype=torch.int32, device=DEV)
    L_.call("ntx_morton3D", ct.data_ptr(), 5000, idx.data_ptr(), L_.stream())
    back = torch.empty(5000, 3, dtype=torch.int32, device=DEV)
    L_.call("ntx_morton3D_invert", idx.data_ptr(), 5000, back.data_ptr(), L_.stream())
    torch.cuda.synchronize()
    np.testing.assert_array_equal(idx.cpu().numpy(), O.morton3D(coords))
    np.testing.assert_array_equal(back.cpu().numpy(), coords)

    dens = rng.random((2, 64 ** 3)).astype(np.float32)
    for n_bytes in (2 * 64 ** 3 // 8, 1001):
        bf = torch.zeros(n_bytes, dtype=torch.uint8, device=DEV)
        dens_t = T(dens)
        L_.call("ntx_packbits", dens_t.data_ptr(), n_bytes, 0.37, bf.data_ptr(), L_.stream())
        torch.cuda.synchronize()
        np.testing.assert_array_equal(bf.cpu().numpy(), O.packbits(dens.ravel()[:n_bytes * 8], 0.37))


def _ntx_march_train(L_, o, d, bits, bound, C, Hg, nears, fars, M, perturb, dt_gamma, max_steps, want_ts=False):
    N = o.shape[0]
    xyzs, dirs, deltas = torch.zeros(M, 3, device=DEV), torch.zeros(M, 3, device=DEV), torch.zeros(M, 2, device=DEV)
    ts = torch.zeros(M, 1, device=DEV) if want_ts else None
    rays = torch.full((N, 3), -1, dtype=torch.int32, device=DEV)
    counter = torch.zeros(2, dtype=torch.int32, device=DEV)
    ws = L_.workspace("march_train", L_.lib().ntx_march_rays_train_workspace_bytes(N), torch.device(DEV, 0))
    ot, dt, bt, nt, ft = T(o), T(d), T(bits), T(nears), T(fars)
    L_.call("ntx_march_rays_train", ot.data_ptr(), dt.data_ptr(), bt.data_ptr(), bound, dt_gamma, max_steps, N, C, Hg, M, nt.data_ptr(),
            ft.data_ptr(), xyzs.data_ptr(), dirs.data_ptr(), deltas.data_ptr(), None if ts is None else ts.data_ptr(), rays.data_ptr(),
            counter.data_ptr(), int(perturb), ws.data_ptr(), L_.stream())
    torch.cuda.synchronize()
    assert int(ws.sum()) == 0, "scan workspace must be left zeroed"
    return xyzs.cpu().numpy(), dirs.cpu().numpy(), deltas.cpu().numpy(), rays.cpu().numpy(), counter.cpu().numpy(), (None if ts is None else ts.cpu().numpy())


@pytest.mark.parametrize("cascade,Hg,bound,dt_gamma,perturb", [(1, 128, 1.0, 0.0, 0), (1, 128, 1.0, 0.0, 1), (2, 64, 2.0, 1.0 / 128, 1), (3, 32, 3.0, 0.0, 0)])
def test_march_rays_train(cascade, Hg, bound, dt_gamma, perturb):
    L_ = ntx()
    O, o, d, grid, bits, aabb, nears, fars = _scene(cascade=cascade, Hg=Hg, bound=bound, radius=0.45, center=(0.1, -0.05, 0.0))
    N = o.shape[0]
    max_steps = 256
    M = N * max_steps
    gx, gd, gl, grays, gcnt, gts = _ntx_march_train(L_, o, d, bits, bound, cascade, Hg, nears, fars, M, perturb, dt_gamma, max_steps, want_ts=True)
    wx, wd, wl, wrays, wcnt, wts = O.march_rays_train(o, d, bound, bits, cascade, Hg, nears, fars, M, perturb=perturb, dt_gamma=dt_gamma, max_steps=max_steps,
                                                       want_ts=True)
    assert wcnt[0] > 1000
    np.testing.assert_array_equal(gcnt, wcnt)
    np.testing.assert_array_equal(grays, wrays)
    m_used = int(wcnt[0])
    np.testing.assert_array_equal(gx[:m_used], wx[:m_used])
    np.testing.assert_array_equal(gd[:m_used], wd[:m_used])
    np.testing.assert_array_equal(gl[:m_used], wl[:m_used])
    np.testing.assert_array_equal(gts[:m_used], wts[:m_used])
    assert not gx[m_used:].any()
    # reference CUDA: same multiset of (ray -> count) and the same samples per ray
    live = {}

    def ref_march(name):
        if not live:
            m = ref("raymarching")
            rx, rd, rl = torch.zeros(M, 3, device=DEV), torch.zeros(M, 3, device=DEV), torch.zeros(M, 2, device=DEV)
            rrays = torch.empty(N, 3, dtype=torch.int32, device=DEV)
            rcnt = torch.zeros(2, dtype=torch.int32, device=DEV)
            m.march_rays_train(T(o), T(d), T(bits), bound, dt_gamma, max_steps, N, cascade, Hg, M, T(nears), T(fars), rx, rd, rl, rrays, rcnt, perturb)
            torch.cuda.synchronize()
            rrays = rrays.cpu().numpy()
            rrays = rrays[np.argsort(rrays[:, 0])]
            live.update(counter=rcnt.cpu().numpy(), ray_ids=rrays[:, 0], ray_counts=rrays[:, 2],
                        xyzs=_samples_by_ray(rx.cpu().numpy(), rrays), deltas=_samples_by_ray(rl.cpu().numpy(), rrays))
        return live[name]
    key = "march_train_c%d_H%d_b%g_g%g_p%d_" % (cascade, Hg, bound, dt_gamma, perturb)
    reference_output(key + "counter", lambda: ref_march("counter"), exact=True).assert_equal(gcnt)
    reference_output(key + "ray_ids", lambda: ref_march("ray_ids"), exact=True).assert_equal(grays[:, 0])
    reference_output(key + "ray_counts", lambda: ref_march("ray_counts"), exact=True).assert_equal(grays[:, 2])
    # the samples of every ray, rays in ascending id order (the reference places each ray's block of samples with an atomic)
    reference_output(key + "xyzs", lambda: ref_march("xyzs"), exact=True).assert_equal(_samples_by_ray(gx, grays))
    reference_output(key + "deltas", lambda: ref_march("deltas"), exact=True).assert_equal(_samples_by_ray(gl, grays))


def _samples_by_ray(x, rays):
    """the rows of x that rays [id, offset, count] (in id order) point at, concatenated"""
    return np.concatenate([x[a:a + c] for a, c in zip(rays[:, 1], rays[:, 2])] + [x[:0]])


def test_march_rays_train_overflow_budget_skips_rays():
    L_ = ntx()
    O, o, d, grid, bits, aabb, nears, fars = _scene()
    M = 4096  # far too small: rays whose segment would cross M are skipped (raymarching.cu:419)
    gx, gd, gl, grays, gcnt, _ = _ntx_march_train(L_, o, d, bits, 1.0, 1, 128, nears, fars, M, 0, 0.0, 256)
    wx, wd, wl, wrays, wcnt, _ = O.march_rays_train(o, d, 1.0, bits, 1, 128, nears, fars, M, max_steps=256)
    np.testing.assert_array_equal(gcnt, wcnt)
    np.testing.assert_array_equal(grays, wrays)
    np.testing.assert_array_equal(gx, wx)
    np.testing.assert_array_equal(gl, wl)


def test_composite_rays_train_forward_backward():
    L_ = ntx()
    O, o, d, grid, bits, aabb, nears, fars = _scene()
    N = o.shape[0]
    M = N * 256
    xyzs, dirs, deltas, rays, cnt, _ = O.march_rays_train(o, d, 1.0, bits, 1, 128, nears, fars, M, max_steps=256)
    m_used = int(cnt[0]) + 128
    rng = np.random.default_rng(0)
    sig = (rng.random(m_used).astype(np.float32) * 20)
    rgb = rng.random((m_used, 3)).astype(np.float32)
    dl = deltas[:m_used]
    ws, dp, im = torch.empty(N, device=DEV), torch.empty(N, device=DEV), torch.empty(N, 3, device=DEV)
    st, rt, dlt, rayt = T(sig), T(rgb), T(dl), T(rays)
    L_.call("ntx_composite_rays_train_forward", st.data_ptr(), rt.data_ptr(), dlt.data_ptr(), rayt.data_ptr(), m_used, N, ws.data_ptr(), dp.data_ptr(), im.data_ptr(), L_.stream())
    wws, wdp, wim = O.composite_rays_train_forward(sig, rgb, dl, rays)
    torch.cuda.synchronize()
    live = {}

    def ref_forward(i):
        if not live:
            rws, rdp, rim = torch.empty(N, device=DEV), torch.empty(N, device=DEV), torch.empty(N, 3, device=DEV)
            ref("raymarching").composite_rays_train_forward(st, rt, dlt, rayt, m_used, N, rws, rdp, rim)
            torch.cuda.synchronize()
            live["r"] = rws.cpu().numpy(), rdp.cpu().numpy(), rim.cpu().numpy()
        return live["r"][i]
    for i, (name, a, b) in enumerate((("weights_sum", ws, wws), ("depth", dp, wdp), ("image", im, wim))):
        c = reference_output("composite_train_forward_" + name, lambda: ref_forward(i))
        np.testing.assert_allclose(c.take(a.cpu().numpy()), c.sample, rtol=1e-6, atol=1e-7)   # same __expf, same order
        np.testing.assert_allclose(a.cpu().numpy(), b, rtol=2e-5, atol=2e-6)                 # expf vs __expf
    gws, gim = T(rng.standard_normal(N).astype(np.float32)), T(rng.standard_normal((N, 3)).astype(np.float32))
    gs, gc = torch.zeros(m_used, device=DEV), torch.zeros(m_used, 3, device=DEV)
    L_.call("ntx_composite_rays_train_backward", gws.data_ptr(), gim.data_ptr(), st.data_ptr(), rt.data_ptr(), dlt.data_ptr(), rayt.data_ptr(), ws.data_ptr(),
            im.data_ptr(), m_used, N, gs.data_ptr(), gc.data_ptr(), L_.stream())
    torch.cuda.synchronize()
    live_b = {}

    def ref_backward(i):
        if not live_b:
            rgs, rgc = torch.zeros(m_used, device=DEV), torch.zeros(m_used, 3, device=DEV)
            ref("raymarching").composite_rays_train_backward(gws, gim, st, rt, dlt, rayt, ws, im, m_used, N, rgs, rgc)
            torch.cuda.synchronize()
            live_b["r"] = rgs.cpu().numpy(), rgc.cpu().numpy()
        return live_b["r"][i]
    rgs, rgc = reference_output("composite_train_backward_grad_sigmas", lambda: ref_backward(0)), reference_output("composite_train_backward_grad_rgbs", lambda: ref_backward(1))
    np.testing.assert_allclose(rgs.take(gs.cpu().numpy()), rgs.sample, rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(rgc.take(gc.cpu().numpy()), rgc.sample, rtol=1e-6, atol=1e-7)
    ogs, ogc = O.composite_rays_train_backward(gws.cpu().numpy(), gim.cpu().numpy(), sig, rgb, dl, rays, ws.cpu().numpy(), im.cpu().numpy())
    np.testing.assert_allclose(gs.cpu().numpy(), ogs, rtol=1e-3, atol=1e-4)
    np.testing.assert_allclose(gc.cpu().numpy(), ogc, rtol=2e-5, atol=2e-6)


@pytest.mark.parametrize("perturb,use_mip", [(0, False), (3, False), (0, True), (3, True)])
def test_inference_loop_march_composite_compact(perturb, use_mip):
    """the body of renderer.py:459-485 for a few iterations, libntx vs oracle (exact) and vs reference CUDA (as sets)"""
    L_ = ntx()
    O, o, d, grid, bits, aabb, nears, fars = _scene(Himg=40, Wimg=40)
    N = o.shape[0]
    rng = np.random.default_rng(1)
    ot, dt, bt, nt, ft = T(o), T(d), T(bits), T(nears), T(fars)
    dev0 = torch.device(DEV, 0)

    # state: ours (g), oracle (w, numpy), reference (r: only run when its outputs are being recorded)
    g_alive = torch.zeros(2, N, dtype=torch.int32, device=DEV); g_alive[0] = torch.arange(N, device=DEV)
    g_t = torch.zeros(2, N, device=DEV); g_t[0] = nt
    g_ws, g_dp, g_im = torch.zeros(N, device=DEV), torch.zeros(N, device=DEV), torch.zeros(N, 3, device=DEV)
    r_alive, r_t = g_alive.clone(), g_t.clone()
    r_ws, r_dp, r_im = g_ws.clone(), g_dp.clone(), g_im.clone()
    w_alive, w_t = np.arange(N, dtype=np.int32), nears.copy()
    w_ws, w_dp, w_im = np.zeros(N, np.float32), np.zeros(N, np.float32), np.zeros((N, 3), np.float32)

    mip = torch.empty(L_.lib().ntx_occupancy_mip_bytes(1, 128), dtype=torch.uint8, device=DEV)
    L_.call("ntx_build_occupancy_mip", bt.data_ptr(), 1, 128, mip.data_ptr(), L_.stream())
    mip_ptr = mip.data_ptr() if use_mip else None
    n_alive, i, step = N, 0, 0
    while step < 64:
        key = "inference_loop_p%d_mip%d_it%d_" % (perturb, use_mip, i)
        if step > 0:
            cnt = torch.zeros(1, dtype=torch.int32, device=DEV)
            ws = L_.workspace("compact", L_.lib().ntx_compact_rays_workspace_bytes(n_alive), dev0)
            L_.call("ntx_compact_rays", n_alive, g_alive[i % 2].data_ptr(), g_alive[(i + 1) % 2].data_ptr(), g_t[i % 2].data_ptr(), g_t[(i + 1) % 2].data_ptr(),
                    cnt.data_ptr(), ws.data_ptr(), L_.stream())
            w_alive, w_t, wn = O.compact_rays(n_alive, w_alive, w_t)
            torch.cuda.synchronize()
            assert int(ws.sum()) == 0
            n_new = int(cnt.item())
            np.testing.assert_array_equal(g_alive[i % 2][:n_new].cpu().numpy(), w_alive[:n_new])
            np.testing.assert_array_equal(g_t[i % 2][:n_new].cpu().numpy(), w_t[:n_new])
            live = {}

            def ref_compact(name):
                if not live:
                    rcnt = torch.zeros(1, dtype=torch.int32, device=DEV)
                    ref("raymarching").compact_rays(n_alive, r_alive[i % 2], r_alive[(i + 1) % 2], r_t[i % 2], r_t[(i + 1) % 2], rcnt)
                    torch.cuda.synchronize()
                    rn = int(rcnt.item())
                    # same set of (ray id, t); re-order the reference state to ascending ids so the loop stays in lock-step
                    ra, rt_ = r_alive[i % 2][:rn].cpu().numpy(), r_t[i % 2][:rn].cpu().numpy()
                    order = np.argsort(ra, kind="stable")
                    r_alive[i % 2][:rn] = T(ra[order]); r_t[i % 2][:rn] = T(rt_[order])
                    live.update(count=rn, ids=ra[order], t=rt_[order])
                return live[name]
            assert n_new == wn == int(reference_output(key + "compact_count", lambda: ref_compact("count")))
            reference_output(key + "compact_ids", lambda: ref_compact("ids"), exact=True).assert_equal(w_alive[:n_new])
            reference_output(key + "compact_t", lambda: ref_compact("t"), exact=True).assert_equal(w_t[:n_new])
            n_alive = n_new
        if n_alive <= 0:
            break
        n_step = max(min(N // n_alive, 8), 1)
        Mp = n_alive * n_step; Mp += 128 - (Mp % 128)
        gx = torch.full((Mp, 3), float("nan"), device=DEV); gd = torch.full((Mp, 3), float("nan"), device=DEV); gl = torch.full((Mp, 2), float("nan"), device=DEV)
        L_.call("ntx_march_rays", n_alive, n_step, g_alive[i % 2].data_ptr(), g_t[i % 2].data_ptr(), ot.data_ptr(), dt.data_ptr(), 1.0, 0.0, 1024, 1, 128,
                bt.data_ptr(), nt.data_ptr(), ft.data_ptr(), gx.data_ptr(), gd.data_ptr(), gl.data_ptr(), perturb, 1, Mp, mip_ptr, L_.stream())
        wx, wd, wl = O.march_rays(n_alive, n_step, w_alive, w_t, o, d, 1.0, bits, 1, 128, nears, fars, align=128, perturb=perturb, max_steps=1024)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(gx.cpu().numpy(), wx)
        np.testing.assert_array_equal(gd.cpu().numpy(), wd)
        np.testing.assert_array_equal(gl.cpu().numpy(), wl)
        rl = torch.zeros(Mp, 2, device=DEV)
        live = {}

        def ref_march(name):
            if not live:
                rx, rd = torch.zeros(Mp, 3, device=DEV), torch.zeros(Mp, 3, device=DEV)
                ref("raymarching").march_rays(n_alive, n_step, r_alive[i % 2], r_t[i % 2], ot, dt, 1.0, 0.0, 1024, 1, 128, bt, nt, ft, rx, rd, rl, perturb)
                torch.cuda.synchronize()
                live.update(xyzs=rx.cpu().numpy(), deltas=rl.cpu().numpy())
            return live[name]
        reference_output(key + "march_xyzs", lambda: ref_march("xyzs"), exact=True).assert_equal(gx.cpu().numpy())
        reference_output(key + "march_deltas", lambda: ref_march("deltas"), exact=True).assert_equal(gl.cpu().numpy())
        sig = (rng.random(Mp).astype(np.float32) * 30)
        rgb = rng.random((Mp, 3)).astype(np.float32)
        st, ct = T(sig), T(rgb)
        L_.call("ntx_composite_rays", n_alive, n_step, g_alive[i % 2].data_ptr(), g_t[i % 2].data_ptr(), st.data_ptr(), ct.data_ptr(), gl.data_ptr(),
                g_ws.data_ptr(), g_dp.data_ptr(), g_im.data_ptr(), L_.stream())
        wt_view = w_t[:n_alive].copy()
        O.composite_rays(n_alive, n_step, w_alive, wt_view, sig, rgb, wl, w_ws, w_dp, w_im)
        w_t = wt_view
        torch.cuda.synchronize()
        live = {}

        def ref_composite(name):
            if not live:
                ref("raymarching").composite_rays(n_alive, n_step, r_alive[i % 2], r_t[i % 2], st, ct, rl, r_ws, r_dp, r_im)
                torch.cuda.synchronize()
                live.update(t=r_t[i % 2][:n_alive].cpu().numpy(), weights_sum=r_ws.cpu().numpy(), image=r_im.cpu().numpy(), depth=r_dp.cpu().numpy())
            return live[name]
        reference_output(key + "composite_t", lambda: ref_composite("t"), exact=True).assert_equal(g_t[i % 2][:n_alive].cpu().numpy())
        for name, a in (("weights_sum", g_ws), ("image", g_im), ("depth", g_dp)):
            r = reference_output(key + "composite_" + name, lambda: ref_composite(name))
            np.testing.assert_allclose(r.take(a.cpu().numpy()), r.sample, rtol=1e-6, atol=1e-7)
        # oracle uses expf: the early-termination decision (T < 1e-4) may differ in the last ulp only in degenerate cases
        np.testing.assert_allclose(g_ws.cpu().numpy(), w_ws, rtol=3e-5, atol=3e-6)
        np.testing.assert_allclose(g_im.cpu().numpy(), w_im, rtol=3e-5, atol=3e-6)
        np.testing.assert_array_equal(g_t[i % 2][:n_alive].cpu().numpy() < 0, w_t < 0)
        # keep the oracle's state identical to the GPU's for the next iteration
        w_t = g_t[i % 2][:n_alive].cpu().numpy().copy()
        w_ws, w_dp, w_im = g_ws.cpu().numpy().copy(), g_dp.cpu().numpy().copy(), g_im.cpu().numpy().copy()
        w_alive = w_alive[:n_alive]
        step += n_step
        i += 1
    assert i >= 5


def test_compact_rays_large_and_counter_accumulates():
    L_ = ntx()
    O = oracle()
    rng = np.random.default_rng(0)
    for n in (1, 31, 1024, 1025, 300_000, 1 << 20):
        ids = rng.permutation(n).astype(np.int32)
        t = np.where(rng.random(n) < 0.6, rng.random(n).astype(np.float32) * 3, -1.0).astype(np.float32)
        out_id, out_t = torch.full((n + 8,), -7, dtype=torch.int32, device=DEV), torch.full((n + 8,), -7.0, device=DEV)
        cnt = torch.tensor([5], dtype=torch.int32, device=DEV)   # pre-loaded: the kernel ADDS like the reference's atomicAdd
        ws = L_.workspace("compact", L_.lib().ntx_compact_rays_workspace_bytes(n), torch.device(DEV, 0))
        ids_t, t_t = T(ids), T(t)
        L_.call("ntx_compact_rays", n, out_id.data_ptr(), ids_t.data_ptr(), out_t.data_ptr(), t_t.data_ptr(),
                cnt.data_ptr(), ws.data_ptr(), L_.stream())
        torch.cuda.synchronize()
        assert int(ws.sum()) == 0
        keep = t >= 0
        k = int(keep.sum())
        assert int(cnt.item()) == 5 + k
        np.testing.assert_array_equal(out_id.cpu().numpy()[5:5 + k], ids[keep])
        np.testing.assert_array_equal(out_t.cpu().numpy()[5:5 + k], t[keep])
